"""Device-resident ring replay: mirror of franQ/Replay/replay_memory.py:9-73 over the HBM arena of libfdql.so.

Same constructor, same duck type (`add`, `sample`, `temporal_sample`, `__getitem__`, `__len__`), same cursor
arithmetic (quirk Q1: the length saturates at maxlen-1) and the same `OversampleError`.  Differences, all on purpose:
  * storage is fp32 structure-of-arrays slabs in HBM (the dtype franQ's TorchDataLoader casts every key to,
    torch_dataloader.py:36); values must be fp32-representable;
  * samples are CUDA tensors `[T, B, w]`, not numpy arrays, so TorchDataLoader becomes a pass-through;
  * `add` stages rows in pinned host memory and moves them in batches; any read flushes first;
  * rows of finished episodes carry their episode extents so that sampled windows can be hindsight-relabelled
    and their returns recomputed at sample time (`temporal_sample(flags=..., goal_rows=...)`).
"""
from __future__ import annotations

import ctypes as C
import functools
import threading
import typing as T

import numpy as np
import torch

from .. import _lib as L
from .._lib import OversampleError, check
from ..reward_ops import RewardOp, TorchReward, require_device_functor


def _locked(fn):
    """One writer thread (Runner._replay_handler) and the learner's reader thread share a ring in the reference without a lock
    (async_replay_memory.py:55-70: the two sides live in different threads of the child process).  Here both sides touch the host
    staging block and the arena cursor, so the public entry points serialise on a re-entrant lock; the device work they enqueue is
    ordered by the stream."""
    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        with self._lock:
            return fn(self, *a, **k)
    return wrapper


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _DevView:
    """__cuda_array_interface__ carrier for zero-copy torch views of arena slabs."""

    def __init__(self, ptr, shape, strides_bytes):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False), "version": 3,
                                         "strides": tuple(strides_bytes)}


class ReplayMemory:
    def __init__(self, maxlen, batch_size, temporal_len, device="cuda:0", stage_rows=1024, roles=None, **kwargs):
        self._batch_size, self._temporal_len, self._maxlen = batch_size, temporal_len, int(maxlen)
        self.batch_size = batch_size
        self._top, self._curr_len = 0, 0
        self._lock = threading.RLock()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.FdqlError("ReplayMemory lives in HBM: device must be a CUDA device (no CPU path)")
        self._lib = L.lib()
        self._h = None
        self._keys: T.List[str] = []
        self._widths: T.List[int] = []
        self._shapes: T.Dict[str, tuple] = {}
        self._role_override = dict(roles or {})
        self._stage_rows = max(1, min(int(stage_rows), self._maxlen))  # a flush never carries more rows than the ring holds
        self._stage = None       # two pinned host blocks [stage_rows, row_floats]: add() packs rows into one while the other drains
        self._stage_np = None    # per block: key -> numpy view [stage_rows, width] into the block
        self._stage_ev = [None, None]
        self._stage_cur = 0
        self._n_staged = 0
        self.squash_rewards = False  # Pohlen transform of the reward column inside the append kernel (wrappers.SquashRewards)
        self._pending_eps: T.List[T.Tuple[int, int]] = []  # (first row, length) of finished, uncommitted episodes
        self._open_ep_first, self._open_ep_len = 0, 0
        self.reward_op: T.Union[RewardOp, TorchReward, None] = None
        self.gamma = 0.99
        self._rng_seed = int(kwargs.get("seed", 0x5EED))
        self._rng_counter = 0
        self._rng_counter_dev = None
        self.device_counter = False  # True: the draw counter lives in device memory (CUDA-graph capture of the learner step)
        self._published_len = -1     # ring length last stored next to the device-side draw counter (see publish_len)
        self._out_cache: T.Dict[tuple, dict] = {}
        self._per_conf = None  # (alpha, eps, eta) of the priority store once enable_priorities() was called
        self._per = None       # fdql_per handle (created with the arena)
        self._per_beta = None  # device float32 [1]: the importance-sampling exponent the PER sampler reads at kernel time

    # ------------------------------------------------------------------ allocation (replay_memory.py:23-35)
    def _jit_initialize(self, widths: T.Dict[str, int], shapes=None):
        assert self._h is None
        self._keys = list(widths)
        if len(self._keys) > L.MAX_KEYS:
            raise ValueError(f"at most {L.MAX_KEYS} keys per row")
        self._widths = [int(widths[k]) for k in self._keys]
        self._shapes = dict(shapes or {k: (w,) for k, w in widths.items()})
        roles = [self._role_override.get(k, L.ROLE_BY_NAME.get(k, L.ROLE_NONE)) for k in self._keys]
        n = len(self._keys)
        h = C.c_void_p()
        check(self._lib.fdql_arena_create(self._maxlen, n, (C.c_int32 * n)(*self._widths), (C.c_int32 * n)(*roles),
                                          self.device.index or 0, C.byref(h)))
        self._h = h
        # packed staging: every key of a row side by side, offsets and row size multiples of 4 floats (128-bit path of the append kernel)
        self._key_off, off = [], 0
        for w in self._widths:
            self._key_off.append(off)
            off += (w + 3) // 4 * 4
        self._row_floats = off
        self._key_off_c = (C.c_int32 * n)(*self._key_off)
        self._stage = [torch.zeros((self._stage_rows, self._row_floats), dtype=torch.float32).pin_memory() for _ in range(2)]
        self._stage_np = [{k: blk.numpy()[:, o:o + w] for k, o, w in zip(self._keys, self._key_off, self._widths)} for blk in self._stage]
        self._scalar_key = {k: (w == 1) for k, w in zip(self._keys, self._widths)}
        if self._per_conf is not None:
            self._create_per()

    def enable_squash_rewards(self, on=True):
        """wrappers.SquashRewards: Pohlen transform (squash_rewards.py:5-7) of the reward column of every row appended from now on."""
        self.flush()
        self.squash_rewards = bool(on)

    def set_reward_op(self, op, gamma=None):
        """The reward of hindsight relabelling: a RewardOp (every mode) or a TorchReward (write-time flushes only)."""
        self.reward_op = RewardOp.coerce(op)
        if gamma is not None:
            self.gamma = float(gamma)

    # ------------------------------------------------------------------ write side (replay_memory.py:38-46)
    def _advance(self, n):
        for _ in range(n) if n < 8 else ():
            self._top = (self._top + 1) % self._maxlen
            self._curr_len = max(self._top, self._curr_len)
        if n >= 8:  # closed form of n single steps
            cap, top = self._maxlen, self._top
            if n >= cap:
                mx = cap - 1
            elif top + n < cap:
                mx = top + n
            else:
                mx = cap - 1 if top <= cap - 2 else top + n - cap
            self._top = (top + n) % cap
            self._curr_len = max(self._curr_len, mx)

    @_locked
    def add(self, experience_dict: dict):
        if self._h is None:
            widths, shapes = {}, {}
            for k, v in experience_dict.items():
                if isinstance(v, np.ndarray):
                    widths[k], shapes[k] = int(v.size), tuple(v.shape)
                else:
                    assert np.isclose(np.float32(v), v), \
                        "Anything thats not a numpy array must be representable as a float32 for numeric stability"
                    widths[k], shapes[k] = 1, (1,)
            self._jit_initialize(widths, shapes)
        i = self._n_staged
        views = self._stage_np[self._stage_cur]
        for k, v in experience_dict.items():
            if getattr(v, "ndim", 0) > 1:
                v = v.reshape(-1)
            views[k][i] = v  # numpy casts to fp32 on assignment
        self._track_episode(bool(experience_dict.get("episode_done", False)) if "episode_done" in experience_dict else None)
        self._n_staged += 1
        self._advance(1)
        if self._n_staged == self._stage_rows:
            self.flush()

    def _track_episode(self, done):
        if done is None:
            return
        if self._open_ep_len == 0:
            self._open_ep_first = self._top
        self._open_ep_len += 1
        if done:
            if self._open_ep_len <= self._maxlen:
                self._pending_eps.append((self._open_ep_first, self._open_ep_len))
            self._open_ep_len = 0

    @_locked
    def flush(self):
        """Move staged rows to the arena and commit the extents of the episodes that finished."""
        if self._h is None:
            return
        if self._n_staged:
            cur = self._stage_cur
            stream = torch.cuda.current_stream(self.device)
            check(self._lib.fdql_arena_append_packed_host(self._h, self._n_staged, C.c_void_p(self._stage[cur].data_ptr()), self._row_floats,
                                                          self._key_off_c, L.APPEND_SQUASH_REWARDS if self.squash_rewards else 0,
                                                          C.c_void_p(stream.cuda_stream)))
            ev = torch.cuda.Event()
            ev.record(stream)
            self._stage_ev[cur] = ev
            # the other block takes the next rows; its own copy was enqueued a whole flush ago (no stream sync in steady state)
            self._stage_cur = cur ^ 1
            if self._stage_ev[cur ^ 1] is not None:
                self._stage_ev[cur ^ 1].synchronize()
            self._n_staged = 0
        if self._pending_eps:
            eps, self._pending_eps = self._pending_eps, []
            self._commit(eps, with_returns=False)

    def _commit(self, eps, with_returns, gamma=None):
        begins = torch.tensor([e[0] for e in eps], dtype=torch.int64, device=self.device)
        lens = torch.tensor([e[1] for e in eps], dtype=torch.int32, device=self.device)
        self.commit_episodes(begins, lens, with_returns=with_returns, gamma=gamma)

    @_locked
    def commit_episodes(self, begins: torch.Tensor, lens: torch.Tensor, with_returns=False, gamma=None):
        """Record episode extents (and optionally return-to-go, nstep_return.py:60-72) for episodes already in the ring.  With a
        TorchReward the scan records carry no goal-agnostic reward: those serve sample-time relabelling, which needs a RewardOp."""
        op = self.reward_op if isinstance(self.reward_op, RewardOp) else RewardOp(L.REWARD_NONE)
        params, n_params = op.c_params()
        check(self._lib.fdql_commit_episodes(self._h, int(begins.numel()), C.c_void_p(begins.data_ptr()),
                                             C.c_void_p(lens.data_ptr()), float(self.gamma if gamma is None else gamma),
                                             int(bool(with_returns)), op.op, params, n_params, _stream_ptr(self.device)))

    @_locked
    def add_rows(self, cols: T.Dict[str, T.Any], episode_lengths=None, with_returns=False, gamma=None):
        """Batched `add`: cols[k] is [n, w] (numpy or torch, host or device).  When `episode_lengths` is given the rows
        are whole episodes laid end to end and are committed (extents, optional returns) in the same call."""
        first = next(iter(cols.values()))
        n = int(first.shape[0])
        self.ensure_schema(cols)
        self.flush()
        dev = []
        for k, w in zip(self._keys, self._widths):
            t = torch.as_tensor(cols[k])
            t = t.to(device=self.device, dtype=torch.float32, non_blocking=True).reshape(n, w).contiguous()
            if self.squash_rewards and k == "reward":  # squash_rewards.py:5-7 in fp64 like numpy on the Python float, fp32 store
                x = t.double()
                t = (torch.sign(x) * (torch.sqrt(x.abs() + 1) - 1) + 1e-2 * x).float()
            dev.append(t)
        begin = self._top
        check(self._lib.fdql_arena_append(self._h, n, L.ptr_array([t.data_ptr() for t in dev]), _stream_ptr(self.device)))
        self._advance(n)
        if episode_lengths is not None:
            lens = torch.as_tensor(episode_lengths, dtype=torch.int64)
            begins = (begin + torch.cumsum(lens, 0) - lens) % self._maxlen
            self.commit_episodes(begins.to(self.device), lens.to(device=self.device, dtype=torch.int32),
                                 with_returns=with_returns, gamma=gamma)
        return begin

    @_locked
    def add_vmap_rows(self, cols, L, picks):
        """HindsightVmapWrite without an NStepReturnVmap underneath (use_nStep_lowerbounds=False): no virtual_mc_return key."""
        begin = self.add_rows(cols, episode_lengths=[L])
        rows = (begin + np.asarray(picks, dtype=np.int64)) % self._maxlen
        self.vmap_flush([begin], [L], pick_rows=rows, fill=True, returns=False)
        return begin

    @_locked
    def add_hindsight_rows(self, src_begins, lens, goal_rows, with_returns=True, gamma=None):
        """Write-time hindsight copy of whole episodes (her.py:55-95): reserves sum(lens) rows at the cursor and fills
        them on the device.  Returns the first destination row of each copy."""
        self.flush()
        if self.reward_op is None:
            raise ValueError("set_reward_op first")
        lens_t = torch.as_tensor(lens, dtype=torch.int64)
        dst = (self._top + torch.cumsum(lens_t, 0) - lens_t) % self._maxlen
        total = int(lens_t.sum())
        first = C.c_int64()
        check(self._lib.fdql_arena_reserve(self._h, total, C.byref(first)))
        self._advance(total)
        src = torch.as_tensor(src_begins, dtype=torch.int64).to(self.device)
        goal = torch.as_tensor(goal_rows, dtype=torch.int64).to(self.device)
        dst_d = dst.to(self.device)
        lens_d = lens_t.to(device=self.device, dtype=torch.int32)
        gam = float(self.gamma if gamma is None else gamma)
        if isinstance(self.reward_op, TorchReward):
            # R(ag_j, g*) and R(ag_j, dg_j) of every source row, packed episode after episode, from ONE call of the user's function
            rows = self._episode_rows(src_begins, lens_t)
            n = rows.numel()
            ag, dg = self._gather_goals(torch.cat([rows, goal]))
            gstar = ag[n:].repeat_interleave(lens_t.to(self.device), dim=0, output_size=n)
            r, d = self.reward_op(torch.cat([ag[:n], ag[:n]]), torch.cat([gstar, dg[:n]]))
            check(self._lib.fdql_her_flush_episodes_given(self._h, int(lens_t.numel()), C.c_void_p(src.data_ptr()),
                                                          C.c_void_p(lens_d.data_ptr()), C.c_void_p(dst_d.data_ptr()),
                                                          C.c_void_p(goal.data_ptr()), n, C.c_void_p(r.data_ptr()),
                                                          C.c_void_p(d.data_ptr()), C.c_void_p(r[n:].data_ptr()), gam,
                                                          int(bool(with_returns)), _stream_ptr(self.device)))
            return dst
        params, n_params = self.reward_op.c_params()
        check(self._lib.fdql_her_flush_episodes(self._h, int(lens_t.numel()), C.c_void_p(src.data_ptr()),
                                                C.c_void_p(lens_d.data_ptr()), C.c_void_p(dst_d.data_ptr()),
                                                C.c_void_p(goal.data_ptr()), self.reward_op.op, params, n_params, gam,
                                                int(bool(with_returns)), _stream_ptr(self.device)))
        return dst

    def _episode_rows(self, begins, lens):
        """Ring rows of whole episodes, episode after episode, each oldest row first (the packed order of the *_given entry points)."""
        lens = np.asarray(lens, dtype=np.int64)
        first = np.repeat(np.asarray(begins, dtype=np.int64) - np.cumsum(lens) + lens, lens)
        return torch.from_numpy((first + np.arange(int(lens.sum()))) % self._maxlen).to(self.device)

    def _gather_goals(self, rows):
        """(achieved_goal, desired_goal) [n, G] of ring rows `rows` (device int64 [n]), gathered by fdql_gather_rows."""
        n = rows.numel()
        roles = [self._role_override.get(k, L.ROLE_BY_NAME.get(k, L.ROLE_NONE)) for k in self._keys]
        if L.ROLE_ACHIEVED_GOAL not in roles or L.ROLE_DESIRED_GOAL not in roles:
            raise ValueError("hindsight relabelling needs achieved_goal and desired_goal keys")
        ka, kd = roles.index(L.ROLE_ACHIEVED_GOAL), roles.index(L.ROLE_DESIRED_GOAL)
        ag = torch.empty((n, self._widths[ka]), dtype=torch.float32, device=self.device)
        dg = torch.empty((n, self._widths[kd]), dtype=torch.float32, device=self.device)
        out = [0] * len(self._keys)
        out[ka], out[kd] = ag.data_ptr(), dg.data_ptr()
        check(self._lib.fdql_gather_rows(self._h, n, C.c_void_p(rows.data_ptr()), L.ptr_array(out), _stream_ptr(self.device)))
        return ag, dg

    # ------------------------------------------------------------------ "vmap" hindsight variant (her_vmap.py, nstep_return_vmap.py)
    VMAP_KEYS = ("virtual_goals", "virtual_rewards", "virtual_dones", "virtual_mc_return")

    def _vmap_key_ids(self):
        ids = [self._keys.index(k) if k in self._keys else -1 for k in self.VMAP_KEYS]
        if min(ids[:3]) < 0:
            raise KeyError("the ring has no virtual_goals / virtual_rewards / virtual_dones keys (write with HindsightVmapWrite)")
        return ids

    @_locked
    def vmap_flush(self, begins, lens, pick_rows=None, fill=True, returns=False, gamma=None, done_quirk=False):
        """Fill the virtual columns of whole episodes already in the ring: goals / rewards / dones from `pick_rows`
        ([n_eps, V] ring rows whose achieved_goal become the virtual goals; her_vmap.py:66-88) and / or the per-column
        return-to-go (nstep_return_vmap.py:37-48,61-74; `done_quirk` reproduces the reference's `* dones[i]`, quirk Q7)."""
        self.flush()
        kg, kr, kd, kret = self._vmap_key_ids()
        b = torch.as_tensor(begins, dtype=torch.int64).to(self.device).contiguous()
        l = torch.as_tensor(lens).to(device=self.device, dtype=torch.int32).contiguous()
        picks = None
        if fill:
            if self.reward_op is None:
                raise ValueError("set_reward_op first")
            picks = torch.as_tensor(np.asarray(pick_rows, dtype=np.int64)).to(self.device).contiguous()
            V = self._widths[kr] - 1
            if picks.numel() != b.numel() * V:
                raise ValueError(f"pick_rows must hold {V} rows per episode")
        gam = float(self.gamma if gamma is None else gamma)
        mode = (1 if fill else 0) | (2 if returns else 0)
        if fill and isinstance(self.reward_op, TorchReward):
            # the [n_rows, V+1] grid: R(ag, virtual goal v) in columns v < V, R(ag, dg) in column V, from ONE call of the user's function
            lens_np = np.asarray(lens, dtype=np.int64)
            rows = self._episode_rows(begins, lens_np)
            n = rows.numel()
            ag, dg = self._gather_goals(torch.cat([rows, picks.reshape(-1)]))
            G = ag.shape[1]
            vg = ag[n:].reshape(b.numel(), V, G).repeat_interleave(l.long(), dim=0, output_size=n)
            goals = torch.cat([vg, dg[:n, None]], dim=1).reshape(n * (V + 1), G)
            r, d = self.reward_op(ag[:n, None].expand(n, V + 1, G).reshape(n * (V + 1), G), goals)
            check(self._lib.fdql_vmap_flush_episodes_given(self._h, int(b.numel()), C.c_void_p(b.data_ptr()), C.c_void_p(l.data_ptr()),
                                                           C.c_void_p(picks.data_ptr()), kg, kr, kd, kret if returns else -1, n,
                                                           C.c_void_p(r.data_ptr()), C.c_void_p(d.data_ptr()), gam, mode,
                                                           int(bool(done_quirk)), _stream_ptr(self.device)))
            return
        op = self.reward_op if isinstance(self.reward_op, RewardOp) else RewardOp(L.REWARD_NONE)
        params, n_params = op.c_params()
        check(self._lib.fdql_vmap_flush_episodes(self._h, int(b.numel()), C.c_void_p(b.data_ptr()), C.c_void_p(l.data_ptr()),
                                                 C.c_void_p(picks.data_ptr()) if picks is not None else None, kg, kr, kd,
                                                 kret if returns else -1, op.op, params, n_params, gam, mode,
                                                 int(bool(done_quirk)), _stream_ptr(self.device)))

    @_locked
    def vmap_temporal_sample(self, column, starts=None, aux=False, n=None, length=None):
        """HindsightVmapRead.temporal_sample (her_vmap.py:104-123): the window batch with desired_goal / reward / task_done /
        mc_return taken from virtual column `column` and the virtual keys removed.  Only that column is read from HBM."""
        _len = len(self) if length is None else int(length)
        Tn = self._temporal_len
        if starts is None:
            starts, _, _ = self.draw_streams(self._batch_size if n is None else int(n), Tn)
        starts = self._to_dev_i64(starts)
        res = self.temporal_sample(starts=starts, length=_len, exclude_keys=self.VMAP_KEYS)
        kg, kr, kd, kret = self._vmap_key_ids()
        nw = starts.numel()
        if kret >= 0 and "mc_return" not in res:
            res["mc_return"] = torch.empty((Tn, nw, 1), dtype=torch.float32, device=self.device)
        aux_t = [None, None, None]
        if aux:
            aux_t = [torch.empty((Tn, nw, 1), dtype=torch.float32, device=self.device),
                     torch.empty((Tn - 1, nw, 1), dtype=torch.float32, device=self.device),
                     torch.empty((Tn - 1, nw, 1), dtype=torch.float32, device=self.device)]
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self._lib.fdql_vmap_select_column(self._h, nw, Tn, _len, C.c_void_p(starts.data_ptr()), int(column), kg, kr, kd, kret, nw,
                                                ptr(res.get("desired_goal")), ptr(res.get("reward")), ptr(res.get("task_done")),
                                                ptr(res.get("mc_return")) if kret >= 0 else None, *[ptr(t) for t in aux_t],
                                                _stream_ptr(self.device)))
        if aux:
            res["mask"], res["is_contiguous"], res["loss_weight"] = aux_t
        return res

    def ensure_schema(self, cols):
        """Allocate the arena from a column dict if no row has been added yet (replay_memory.py:23-35)."""
        if self._h is None:
            self._jit_initialize({k: int(np.prod(v.shape[1:])) if len(v.shape) > 1 else 1 for k, v in cols.items()},
                                 {k: tuple(v.shape[1:]) or (1,) for k, v in cols.items()})

    @_locked
    def reserve_rows(self, n):
        """Advance the cursor by n rows whose content a device kernel will produce; returns the first reserved row."""
        self.flush()
        first = C.c_int64()
        check(self._lib.fdql_arena_reserve(self._h, int(n), C.byref(first)))
        self._advance(int(n))
        return first.value

    @_locked
    def q3_duplicate(self, src_row, n_step, dst_row, gamma):
        """quirk Q3: the oldest row of an episode longer than n_step, stored once more with the n-step-truncated return."""
        check(self._lib.fdql_q3_duplicate(self._h, int(src_row), int(n_step), int(dst_row), float(gamma), _stream_ptr(self.device)))

    # ------------------------------------------------------------------ prioritized replay (fdql_per_*, include/fdql.h): proportional PER
    # (Schaul et al. 2016) over the window starts.  Not a reference mode: franQ samples uniformly (replay_memory.py:59).
    def enable_priorities(self, alpha=0.6, eps=1e-6, eta=0.9):
        """Keep a priority per window start: `temporal_sample(prioritized=True)` draws starts with probability q / sum(q),
        q = (delta + eps)^alpha, and `update_priorities` sets delta from the critic's per-transition loss (eta max + (1 - eta) mean
        over the window, R2D2's mix).  New rows enter with the largest priority written so far.  The store is created with the arena."""
        alpha, eps, eta = float(alpha), float(eps), float(eta)
        if not (alpha >= 0 and eps > 0 and 0 <= eta <= 1):
            raise ValueError(f"need alpha >= 0, eps > 0, eta in [0, 1]; got alpha={alpha} eps={eps} eta={eta}")
        if self._per is not None:
            raise RuntimeError("priorities are already enabled")
        self._per_conf = (alpha, eps, eta)
        if self._h is not None:
            self._create_per()

    def _create_per(self):
        h = C.c_void_p()
        check(self._lib.fdql_per_create(self._h, self._temporal_len, *self._per_conf, C.byref(h)))
        self._per = h
        self._per_beta = torch.full((1,), 0.4, dtype=torch.float32, device=self.device)

    def _require_per(self):
        if self._per is None:
            raise RuntimeError("prioritized sampling needs enable_priorities() and at least one stored row")

    @_locked
    def set_priority_beta(self, beta):
        """Store the importance-sampling exponent in the device scalar the sampler reads (stream-ordered: a captured step picks it up
        at its next replay)."""
        self._require_per()
        self._per_beta.fill_(float(beta))

    @_locked
    def draw_prioritized(self, n=None, beta=None, goal_mode=None, relabel_prob=0.0, xi=None):
        """(starts, flags, goal_rows, is_weight) of n windows drawn by priority.  `xi` (device float64 [n] in [0, 1)) injects the
        stratum offsets instead of drawing them; `beta` (None: the stored one) sets the importance-sampling exponent first."""
        self._require_per()
        self.flush()
        n = self._batch_size if n is None else int(n)
        if beta is not None:
            self._per_beta.fill_(float(beta))
        starts = torch.empty(n, dtype=torch.int64, device=self.device)
        weight = torch.empty(n, dtype=torch.float32, device=self.device)
        flags = goals = None
        if relabel_prob > 0:
            flags = torch.empty(n, dtype=torch.uint8, device=self.device)
            goals = torch.empty(n, dtype=torch.int64, device=self.device)
        if xi is not None:
            xi = torch.as_tensor(xi, dtype=torch.float64).to(self.device).contiguous()
            if xi.numel() != n:
                raise ValueError(f"xi must hold {n} values")
        if self._rng_counter_dev is None:
            self._rng_counter_dev = torch.zeros(4, dtype=torch.int64, device=self.device)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self._lib.fdql_per_sample(self._per, n, L.GOAL_FUTURE if goal_mode is None else int(goal_mode), float(relabel_prob),
                                        self._rng_seed, self._rng_counter, ptr(self._rng_counter_dev) if self.device_counter else None,
                                        ptr(xi), ptr(self._per_beta), ptr(starts), ptr(flags), ptr(goals), ptr(weight),
                                        _stream_ptr(self.device)))
        if not self.device_counter:
            self._rng_counter += 1
        return starts, flags, goals, weight

    @_locked
    def update_priorities(self, starts, loss, contig=None):
        """New priorities of the windows `starts` [B] from the per-transition loss [T-1, B(, 1)] of their transitions and the gather's
        is_contiguous [T-1, B(, 1)] (None: all count).  Stream-ordered; duplicate starts: the last window of the batch wins."""
        self._require_per()
        starts = self._to_dev_i64(starts)
        n = starts.numel()
        loss = loss.detach().to(device=self.device, dtype=torch.float32).reshape(-1, n).contiguous()
        if loss.shape[0] != self._temporal_len - 1:
            raise ValueError(f"loss must be [T-1={self._temporal_len - 1}, {n}], got {tuple(loss.shape)}")
        if contig is not None:
            contig = contig.detach().to(device=self.device, dtype=torch.float32).reshape(loss.shape).contiguous()
        check(self._lib.fdql_per_update(self._per, n, C.c_void_p(starts.data_ptr()), C.c_void_p(loss.data_ptr()),
                                        C.c_void_p(contig.data_ptr()) if contig is not None else None, _stream_ptr(self.device)))

    @_locked
    def apply_pending_priorities(self):
        """Give the rows written since the last PER call their priority (q_max, or 0 past the start range) on the current stream."""
        if self._per is None:
            return
        self.flush()
        check(self._lib.fdql_per_apply_pending(self._per, _stream_ptr(self.device)))

    def priority_views(self):
        """(leaves [maxlen], q_max [1]): zero-copy float32 views of the priority store (write leaves, then rebuild_priorities())."""
        self._require_per()
        leaves, qmax = C.c_void_p(), C.c_void_p()
        check(self._lib.fdql_per_view(self._per, C.byref(leaves), C.byref(qmax)))
        return (torch.as_tensor(_DevView(leaves.value, (self._maxlen,), (4,)), device=self.device),
                torch.as_tensor(_DevView(qmax.value, (2,), (4,)), device=self.device)[:1])

    def priority_tree(self):
        """[(sums float64 [n_l], mins float32 [n_l]) for l = 1 .. L]: zero-copy views of the tree levels above the leaves (root last)."""
        self._require_per()
        out, level = [], 1
        while True:
            sums, mins, n = C.c_void_p(), C.c_void_p(), C.c_int64()
            if self._lib.fdql_per_level_view(self._per, level, C.byref(sums), C.byref(mins), C.byref(n)) != L.FDQL_OK:
                return out
            s = torch.as_tensor(_DevView(sums.value, (n.value, 2), (8, 4)), device=self.device).view(torch.float64).reshape(-1)
            out.append((s, torch.as_tensor(_DevView(mins.value, (n.value,), (4,)), device=self.device)))
            level += 1

    @_locked
    def rebuild_priorities(self):
        self._require_per()
        check(self._lib.fdql_per_rebuild(self._per, _stream_ptr(self.device)))

    # ------------------------------------------------------------------ snapshot / restore (the reference never persists its replay;
    # its dormant analogue is memmap_replay_memory.py).  Every slab is saved raw -- user keys, episode extents, scan and link
    # records -- so the restored ring answers any call bit for bit, stale (partly overwritten) episodes included.
    def _meta_rows(self, which):
        base, stride, col = C.c_void_p(), C.c_int64(), C.c_int32()
        check(self._lib.fdql_arena_meta_view(self._h, which, C.byref(base), C.byref(stride), C.byref(col)))
        return torch.as_tensor(_DevView(base.value, (self._maxlen, 4), (4 * stride.value, 4)), device=self.device)

    @_locked
    def state_dict(self):
        self.flush()
        es, ee = self.episode_extents()
        gam, st = C.c_double(), C.c_int32()
        check(self._lib.fdql_arena_link_state(self._h, 0, C.byref(gam), C.byref(st)))
        return {"maxlen": self._maxlen, "keys": list(self._keys), "widths": list(self._widths), "shapes": dict(self._shapes),
                "top": self._top, "len": self._curr_len, "gamma": self.gamma, "link": (gam.value, st.value),
                "reward_op": self._reward_op_state(),
                "memory": {k: v.cpu().clone() for k, v in self.memory.items()}, "ep_start": es.cpu().clone(), "ep_end": ee.cpu().clone(),
                "scan": self._meta_rows(2).view(torch.int32).cpu().clone(), "links": self._meta_rows(3).view(torch.int32).cpu().clone(),
                "per": self._per_state()}

    def _reward_op_state(self):
        """(op, params) of a RewardOp; "torch" for a TorchReward, whose function is not pickled (set it again before restoring)."""
        if self.reward_op is None:
            return None
        if isinstance(self.reward_op, TorchReward):
            return "torch"
        return (self.reward_op.op, list(self.reward_op.params or []))

    def _per_state(self):
        if self._per is None:
            return None
        self.apply_pending_priorities()
        leaves, qmax = self.priority_views()
        return {"conf": list(self._per_conf), "leaves": leaves.cpu().clone(), "q_max": qmax.cpu().clone()}

    @_locked
    def load_state_dict(self, sd):
        if self._h is not None:
            raise RuntimeError("load_state_dict needs a fresh ReplayMemory")
        if int(sd["maxlen"]) != self._maxlen:
            raise ValueError(f"snapshot of a ring of {sd['maxlen']} rows, this one has {self._maxlen}")
        if sd["reward_op"] == "torch" and not isinstance(self.reward_op, TorchReward):
            raise ValueError("the snapshot's reward is a TorchReward, whose function a snapshot does not carry: call "
                             "set_reward_op(TorchReward(fn)) (or build the ring through its hindsight wrapper) before load_state_dict")
        self._jit_initialize(dict(zip(sd["keys"], sd["widths"])), sd["shapes"])
        self.gamma = float(sd["gamma"])
        if sd["reward_op"] is not None and sd["reward_op"] != "torch":
            self.reward_op = RewardOp(sd["reward_op"][0], sd["reward_op"][1] or ())
        dev = [sd["memory"][k].to(self.device, dtype=torch.float32).reshape(self._maxlen, w).contiguous()
               for k, w in zip(self._keys, self._widths)]
        check(self._lib.fdql_arena_append(self._h, self._maxlen, L.ptr_array([t.data_ptr() for t in dev]), _stream_ptr(self.device)))
        check(self._lib.fdql_arena_set_cursor(self._h, int(sd["top"]), int(sd["len"])))
        self._top, self._curr_len = int(sd["top"]), int(sd["len"])
        es, ee = self.episode_extents()
        es.copy_(sd["ep_start"].to(self.device))
        ee.copy_(sd["ep_end"].to(self.device))
        self._meta_rows(2).view(torch.int32).copy_(sd["scan"].to(self.device))
        self._meta_rows(3).view(torch.int32).copy_(sd["links"].to(self.device))
        gam, st = C.c_double(float(sd["link"][0])), C.c_int32(int(sd["link"][1]))
        check(self._lib.fdql_arena_link_state(self._h, 1, C.byref(gam), C.byref(st)))
        per = sd.get("per")
        if per is not None and self._per is None:
            self._per_conf = tuple(float(x) for x in per["conf"])
            self._create_per()
        if self._per is not None:
            self.apply_pending_priorities()  # the restored rows were recorded as written: settle that first, then overwrite the leaves
            if per is not None:
                leaves, qmax = self.priority_views()
                leaves.copy_(per["leaves"].to(self.device))
                qmax.copy_(per["q_max"].to(self.device))
                self.rebuild_priorities()
        torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ read side (replay_memory.py:48-70)
    def __len__(self):
        return self._curr_len

    @property
    def keys(self):
        return list(self._keys)

    @property
    def memory(self) -> T.Dict[str, torch.Tensor]:
        """Zero-copy strided views of the arena slabs, `memory[k]` is [maxlen, w] like the reference's numpy dict."""
        self.flush()
        out = {}
        for i, (k, w) in enumerate(zip(self._keys, self._widths)):
            base, stride, col = C.c_void_p(), C.c_int64(), C.c_int32()
            check(self._lib.fdql_arena_key_view(self._h, i, C.byref(base), C.byref(stride), C.byref(col)))
            out[k] = torch.as_tensor(_DevView(base.value + 4 * col.value, (self._maxlen, w), (4 * stride.value, 4)),
                                     device=self.device)
        return out

    def _meta(self, which):
        base, stride, col = C.c_void_p(), C.c_int64(), C.c_int32()
        check(self._lib.fdql_arena_meta_view(self._h, which, C.byref(base), C.byref(stride), C.byref(col)))
        return torch.as_tensor(_DevView(base.value + 4 * col.value, (self._maxlen, 1), (4 * stride.value, 4)), device=self.device)

    def episode_extents(self):
        """(ep_start, ep_end) int32 [maxlen] views; -1 where the row's episode has not been committed."""
        self.flush()
        return self._meta(0).view(torch.int32).reshape(-1), self._meta(1).view(torch.int32).reshape(-1)

    def _outputs(self, lead: tuple, reuse: bool, exclude: tuple = ()):
        key = lead + exclude
        if reuse and key in self._out_cache:
            return self._out_cache[key]
        out = {k: torch.empty(lead + (w,), dtype=torch.float32, device=self.device) for k, w in zip(self._keys, self._widths)
               if k not in exclude}
        if reuse:
            self._out_cache[key] = out
        return out

    def _to_dev_i64(self, x):
        if isinstance(x, torch.Tensor) and x.device == self.device and x.dtype == torch.int64:
            return x.contiguous()
        return torch.as_tensor(np.asarray(x, dtype=np.int64) if not isinstance(x, torch.Tensor) else x,
                               dtype=torch.int64).to(self.device).contiguous()

    @_locked
    def __getitem__(self, idxes) -> T.Dict[str, torch.Tensor]:
        self.flush()
        idx = self._to_dev_i64(idxes)
        shape = tuple(idx.shape)
        flat = idx.reshape(-1)
        if bool(((flat < 0) | (flat >= self._maxlen)).any()):
            raise IndexError("row index out of range")
        out = self._outputs((flat.numel(),), reuse=False)
        check(self._lib.fdql_gather_rows(self._h, flat.numel(), C.c_void_p(flat.data_ptr()),
                                         L.ptr_array([out[k].data_ptr() for k in self._keys]), _stream_ptr(self.device)))
        return {k: v.reshape(shape + (v.shape[-1],)) for k, v in out.items()}

    @_locked
    def draw_streams(self, n=None, temporal_len=None, goal_mode=None, relabel_prob=0.0):
        """Device-side np.random.randint(0, len-T, B) (+ hindsight flag / goal row per window when relabel_prob > 0)."""
        self.flush()
        n = self._batch_size if n is None else int(n)
        Tn = self._temporal_len if temporal_len is None else int(temporal_len)
        starts = torch.empty(n, dtype=torch.int64, device=self.device)
        flags = goals = None
        if relabel_prob > 0:
            flags = torch.empty(n, dtype=torch.uint8, device=self.device)
            goals = torch.empty(n, dtype=torch.int64, device=self.device)
        self._sync_cursor()
        if self._rng_counter_dev is None:  # {draw counter, block ticket}: lets a captured graph draw fresh streams per replay
            self._rng_counter_dev = torch.zeros(4, dtype=torch.int64, device=self.device)
        check(self._lib.fdql_sample_streams(self._h, n, Tn, L.GOAL_FUTURE if goal_mode is None else int(goal_mode),
                                            float(relabel_prob), self._rng_seed, self._rng_counter,
                                            C.c_void_p(self._rng_counter_dev.data_ptr()) if self.device_counter else None,
                                            C.c_void_p(starts.data_ptr()),
                                            C.c_void_p(flags.data_ptr()) if flags is not None else None,
                                            C.c_void_p(goals.data_ptr()) if goals is not None else None,
                                            _stream_ptr(self.device)))
        if not self.device_counter:
            self._rng_counter += 1
        return starts, flags, goals

    @_locked
    def publish_len(self):
        """Store the ring's length next to the device-side draw counter ({counter, ticket, length, 0}): a captured sample / gather
        launch reads its start range from there, so one captured learner step keeps sampling the whole ring while it fills."""
        if self._rng_counter_dev is None:
            self._rng_counter_dev = torch.zeros(4, dtype=torch.int64, device=self.device)
        if self._published_len != self._curr_len:
            self._rng_counter_dev[2:3].fill_(self._curr_len)
            self._published_len = self._curr_len

    def _sync_cursor(self):
        top, ln = C.c_int64(), C.c_int64()
        check(self._lib.fdql_arena_info(self._h, None, C.byref(top), C.byref(ln), None))
        assert (top.value, ln.value) == (self._top, self._curr_len), "host and arena cursors diverged"

    @_locked
    def sample(self, idx=None, prioritized=False) -> T.Dict[str, torch.Tensor]:
        if prioritized:
            raise NotImplementedError("prioritized replay draws window starts: use temporal_sample(prioritized=True)")
        if len(self) < self._batch_size:
            raise OversampleError("Trying to sample more memories than available!")
        if idx is None:
            idx, _, _ = self.draw_streams(self._batch_size, 0)
        return self[idx]

    @_locked
    def temporal_sample(self, starts=None, flags=None, goal_rows=None, exact_episode_step=False, aux=False,
                        reuse_outputs=False, n=None, relabel_prob=0.0, goal_mode=None, length=None, exclude_keys=(),
                        prioritized=False, beta=None, xi=None):
        """[T, B, w] window gather (replay_memory.py:54-66).  `starts` (and for hindsight relabelling `flags`,
        `goal_rows`) inject the index streams; when absent they are drawn on the device.  With `aux=True` the dict
        also carries `mask`, `is_contiguous` and `loss_weight` (deepQlearning.py:201-203,222-225).
        `prioritized=True` (after enable_priorities) draws the starts by priority (draw_prioritized: `beta`, `xi`) and gathers them
        with the same kernel as injected starts; the dict then also carries `is_weight` [B] and the `starts` [B] drawn."""
        if relabel_prob > 0:
            require_device_functor(self.reward_op, "sample-time relabelling (relabel_prob > 0)")
        if prioritized:
            if starts is not None or length is not None:
                raise ValueError("prioritized sampling draws its own starts")
            if len(self) < self._temporal_len * 2 or len(self) < self._batch_size:
                raise OversampleError("Trying to sample more memories than available!")
            starts, flags, goal_rows, weight = self.draw_prioritized(n, beta, goal_mode, relabel_prob, xi)
            # every drawn start is < len - T, so its window never wraps: the capacity as modulus gives the rows len would, and stays
            # right inside a captured step while the ring grows
            res = self.temporal_sample(starts=starts, flags=flags, goal_rows=goal_rows, exact_episode_step=exact_episode_step, aux=aux,
                                       reuse_outputs=reuse_outputs, length=self._maxlen, exclude_keys=exclude_keys)
            self.last_streams = (starts, flags, goal_rows)
            res["is_weight"], res["starts"] = weight, starts
            return res
        _len = len(self) if length is None else int(length)
        Tn = self._temporal_len
        n = self._batch_size if n is None else int(n)
        if (_len < (Tn * 2)) or (_len < self._batch_size):
            raise OversampleError("Trying to sample more memories than available!")
        self.flush()
        fused = starts is None and length is None  # streams drawn inside the gather kernel (fdql_sample_gather_draw)
        if fused:
            self._sync_cursor()
            starts = torch.empty(n, dtype=torch.int64, device=self.device)
            if relabel_prob > 0:
                flags = torch.empty(n, dtype=torch.uint8, device=self.device)
                goal_rows = torch.empty(n, dtype=torch.int64, device=self.device)
            if self._rng_counter_dev is None:
                self._rng_counter_dev = torch.zeros(4, dtype=torch.int64, device=self.device)
        elif starts is None:
            starts, flags, goal_rows = self.draw_streams(n, Tn, goal_mode, relabel_prob)
        starts = self._to_dev_i64(starts)
        n = starts.numel()
        if flags is not None:
            flags = torch.as_tensor(flags).to(device=self.device, dtype=torch.uint8).contiguous()
            goal_rows = self._to_dev_i64(goal_rows)
            if self.reward_op is None:
                raise ValueError("relabelling needs set_reward_op(...)")
            require_device_functor(self.reward_op, "sample-time relabelling")
        out = self._outputs((Tn, n), reuse=reuse_outputs, exclude=tuple(exclude_keys))
        opts = (L.OPT_EXACT_EPISODE_STEP if exact_episode_step else 0) | (L.OPT_EMIT_LEARNER_AUX if aux else 0)
        aux_t = [None, None, None]
        if aux:
            ck = ("aux", Tn, n)
            if reuse_outputs and ck in self._out_cache:
                aux_t = self._out_cache[ck]
            else:
                aux_t = [torch.empty((Tn, n, 1), dtype=torch.float32, device=self.device),
                         torch.empty((Tn - 1, n, 1), dtype=torch.float32, device=self.device),
                         torch.empty((Tn - 1, n, 1), dtype=torch.float32, device=self.device)]
                if reuse_outputs:
                    self._out_cache[ck] = aux_t
        op = self.reward_op if isinstance(self.reward_op, RewardOp) else RewardOp(L.REWARD_NONE)
        params, n_params = op.c_params()
        if fused:
            check(self._lib.fdql_sample_gather_draw(
                self._h, n, Tn, L.GOAL_FUTURE if goal_mode is None else int(goal_mode), float(relabel_prob), self._rng_seed,
                self._rng_counter, C.c_void_p(self._rng_counter_dev.data_ptr()) if self.device_counter else None,
                C.c_void_p(starts.data_ptr()), C.c_void_p(flags.data_ptr()) if flags is not None else None,
                C.c_void_p(goal_rows.data_ptr()) if flags is not None else None,
                op.op if flags is not None else L.REWARD_NONE, params, n_params, float(self.gamma), opts, n,
                L.ptr_array([out[k].data_ptr() if k in out else 0 for k in self._keys]),
                *[C.c_void_p(t.data_ptr()) if t is not None else None for t in aux_t], _stream_ptr(self.device)))
            if not self.device_counter:
                self._rng_counter += 1
            self.last_streams = (starts, flags, goal_rows)
            res = dict(out)
            if aux:
                res["mask"], res["is_contiguous"], res["loss_weight"] = aux_t
            return res
        check(self._lib.fdql_sample_gather(
            self._h, n, Tn, _len, C.c_void_p(starts.data_ptr()),
            C.c_void_p(flags.data_ptr()) if flags is not None else None,
            C.c_void_p(goal_rows.data_ptr()) if flags is not None else None,
            op.op if flags is not None else L.REWARD_NONE, params, n_params, float(self.gamma), opts, n,
            L.ptr_array([out[k].data_ptr() if k in out else 0 for k in self._keys]),
            *[C.c_void_p(t.data_ptr()) if t is not None else None for t in aux_t], _stream_ptr(self.device)))
        res = dict(out)
        if aux:
            res["mask"], res["is_contiguous"], res["loss_weight"] = aux_t
        return res

    def _temporal_sample_idxes(self, batch, _len):
        return self.temporal_sample(starts=batch, length=_len)

    def __del__(self):
        per, self._per = getattr(self, "_per", None), None
        if per is not None:
            try:
                self._lib.fdql_per_destroy(per)  # before its arena
            except Exception:
                pass
        h, self._h = getattr(self, "_h", None), None
        if h is not None:
            try:
                self._lib.fdql_arena_destroy(h)
            except Exception:
                pass
