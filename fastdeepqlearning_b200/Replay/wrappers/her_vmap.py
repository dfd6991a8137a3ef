"""Mirror of franQ/Replay/wrappers/her_vmap.py:10-123 (her_mode="vmap"): every stored row carries `num_virtual_goals`
virtual goals plus its real goal, and the rewards / dones it would have had under each; the read head picks ONE column
for the whole batch.

Write head: the episode in flight is held on the host; at `episode_done` its rows go to the ring in one batch and the
virtual columns are produced on the device by fdql_vmap_flush_episodes (the reference runs a jax.vmap over goals on the host
and then pushes rows one by one through Python).  The goal picks use `np.random.randint(0, L, V)` like her_vmap.py:75.
Read head: fdql_vmap_select_column reads only the chosen column.  `compute_reward` is a device functor (RewardOp) or a TorchReward,
which the ring evaluates once per flush over the [L, V+1] grid of (row, goal) pairs for fdql_vmap_flush_episodes_given."""
import random

import numpy as np
import torch

from .wrapper_base_class import ReplayMemoryWrapper
from .nstep_return import stack_rows
from ...reward_ops import RewardOp


class HindsightVmapWrite(ReplayMemoryWrapper):
    def __init__(self, replay_buffer, compute_reward, ignore_keys=("info",), num_virtual_goals=32):
        ReplayMemoryWrapper.__init__(self, replay_buffer)
        self.compute_reward = RewardOp.coerce(compute_reward)
        self._ignored_keys = tuple(ignore_keys)
        self.num_virtual_goals = int(num_virtual_goals)
        self.set_reward_op(self.compute_reward)  # reaches the ring through the wrapper chain
        self._reset()

    def _reset(self):
        self.rows = []

    def _pick_virtual_goals(self, L):
        """Chronological indices of the rows whose achieved_goal become the virtual goals.  her_vmap.py:75 indexes the
        newest-first deque with np.random.randint(0, L, V): deque index i is chronological index L-1-i."""
        return L - 1 - np.random.randint(0, L, size=self.num_virtual_goals)

    def add(self, experience):
        self.rows.append({k: v for k, v in experience.items() if k not in self._ignored_keys})
        if experience["episode_done"]:
            rows = self.rows
            self._reset()
            self._hindsight_flush(rows)

    def _hindsight_flush(self, rows):
        L, V = len(rows), self.num_virtual_goals
        cols = stack_rows(rows)
        G = cols["desired_goal"].shape[1]
        dev = self.device
        # the virtual columns are produced on the device; their slots are appended as device zeros (no host traffic)
        cols["virtual_goals"] = torch.zeros((L, (V + 1) * G), device=dev)
        cols["virtual_rewards"] = torch.zeros((L, V + 1), device=dev)
        cols["virtual_dones"] = torch.zeros((L, V + 1), device=dev)
        picks = self._pick_virtual_goals(L)
        self.replay_buffer.add_vmap_rows(cols, L, picks)


class HindsightVmapRead(ReplayMemoryWrapper):
    """Reader head (her_vmap.py:93-123): one virtual-goal column, drawn with random.randint(0, V) (inclusive: column V is
    the real goal), replaces desired_goal / reward / task_done / mc_return of the whole batch; the virtual keys are dropped."""

    def __init__(self, replay_buffer, aux=False):
        ReplayMemoryWrapper.__init__(self, replay_buffer)
        self.aux = aux

    def temporal_sample(self, column=None, **kwargs):
        if kwargs.pop("prioritized", False):
            raise NotImplementedError("prioritized replay is not supported with the vmap hindsight variant")
        ring = self.replay_buffer
        while hasattr(ring, "replay_buffer") or hasattr(ring, "replay"):
            ring = getattr(ring, "replay_buffer", None) or ring.replay
        if len(ring) < 2 * ring._temporal_len or len(ring) < ring._batch_size:
            from ..replay_memory import OversampleError
            raise OversampleError("Trying to sample more memories than available!")
        ring.flush()
        num_virtual_goals = ring._widths[ring._keys.index("virtual_rewards")]
        idx = random.randint(0, num_virtual_goals - 1) if column is None else int(column)
        kwargs.setdefault("aux", self.aux)
        return ring.vmap_temporal_sample(idx, **kwargs)
