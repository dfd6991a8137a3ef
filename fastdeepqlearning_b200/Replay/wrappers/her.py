"""Mirror of franQ/Replay/wrappers/her.py:8-95 (write-time hindsight, modes "final" / "random") plus the sample-time
form used by the B200 path (mode "future", relabel probability k/(k+1)).

Write-time: the episode in flight is held on the host; at `episode_done` the real rows go to the ring in one batch and
the hindsight copy (goal substitution, reward recompute, synthetic-episode splitting of task_done / episode_step, and
the inner NStepReturn's return over the relabelled rewards) is produced on the device by fdql_her_flush_episodes.
`compute_reward` is a device functor (RewardOp) or a TorchReward; with the latter the ring evaluates it once per flush on the
gathered goals and fdql_her_flush_episodes_given consumes the results.  The goal pick uses Python's `random` like her.py:51-53."""
import random

from .wrapper_base_class import ReplayMemoryWrapper
from .nstep_return import stack_rows
from ...reward_ops import RewardOp, require_device_functor


class HindsightNStepReplay(ReplayMemoryWrapper):
    def __init__(self, replay_buffer, compute_reward, ignore_keys=("info",), mode="random"):
        ReplayMemoryWrapper.__init__(self, replay_buffer)
        self.compute_reward = RewardOp.coerce(compute_reward)
        if mode not in ("final", "random"):
            raise ValueError("mode must be 'final' or 'random' (her.py:48-53)")
        self._ignored_keys = tuple(ignore_keys)
        self._mode = mode
        self.set_reward_op(self.compute_reward)  # reaches the ring through the wrapper chain
        self._reset()

    def _reset(self):
        self.rows = []

    def _select_virtual_goal(self, L):
        """Chronological index of the row whose achieved_goal becomes the goal (her.py:48-53; the reference's deque is
        newest-first, so deque index i is chronological index L-1-i)."""
        if self._mode == "final":
            return L - 1
        return L - 1 - random.choice(range(L))

    def add(self, experience):
        if "info" not in experience and "info" in self._ignored_keys:
            pass  # the reference needs the key only to zip over it (quirk Q6); nothing is read from it
        self.rows.append({k: v for k, v in experience.items() if k not in self._ignored_keys})
        if experience["episode_done"]:
            rows = self.rows
            self._reset()
            L = len(rows)
            begin = self.replay_buffer.add_rows(stack_rows(rows), episode_lengths=[L])       # her.py:36-46
            goal = (begin + self._select_virtual_goal(L)) % self._maxlen
            self.replay_buffer.add_hindsight_rows([begin], [L], [goal])                      # her.py:55-95


class IgnoreKeys(ReplayMemoryWrapper):
    """Write head of the sample-time hindsight mode: drops the keys the reference's HER wrappers ignore (`info`, her.py:13), which the
    Runner keeps in every row whenever use_HER is on (runner.py:185-186); rows are stored once, nothing else happens at write time."""

    def __init__(self, replay_buffer, ignore_keys=("info",)):
        ReplayMemoryWrapper.__init__(self, replay_buffer)
        self._ignored_keys = tuple(ignore_keys)

    def add(self, experience):
        self.replay_buffer.add({k: v for k, v in experience.items() if k not in self._ignored_keys})


class SampleTimeHindsight(ReplayMemoryWrapper):
    """Read head that relabels at sample time: each sampled window is relabelled with probability `relabel_prob`
    towards the achieved goal of a later row of its episode ("future" strategy, k = p/(1-p)), with reward, task_done,
    episode_step and the return-to-go recomputed by the fused gather kernel.  Rows are stored once."""

    def __init__(self, replay_buffer, relabel_prob=0.8, goal_mode=None, aux=True):
        ReplayMemoryWrapper.__init__(self, replay_buffer)
        require_device_functor(getattr(replay_buffer, "reward_op", None), "SampleTimeHindsight")
        self.relabel_prob, self.goal_mode, self.aux = relabel_prob, goal_mode, aux

    def temporal_sample(self, *args, **kwargs):
        kwargs.setdefault("relabel_prob", self.relabel_prob)
        kwargs.setdefault("goal_mode", self.goal_mode)
        kwargs.setdefault("aux", self.aux)
        return self.replay_buffer.temporal_sample(*args, **kwargs)
