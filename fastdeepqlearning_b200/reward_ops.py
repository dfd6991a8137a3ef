"""Reward functions R(achieved_goal, goal) -> (reward, done) for hindsight relabelling.

franQ's HER wrapper receives an arbitrary Python callable (franQ/Replay/wrappers/her.py:13,62,67).  Here the `compute_reward` slot
of the mirror wrappers accepts two kinds of value:
  * `RewardOp`: an enum-dispatched device functor (include/fdql.h FDQL_REWARD_*), evaluated inside the CUDA kernels.  It serves
    every mode, sample-time relabelling included.
  * `TorchReward`: a batched PyTorch function on CUDA tensors, for rewards the functors cannot express.  It serves write-time
    relabelling only (her_mode "final", "random" and "vmap"), where the reward is evaluated once per stored row when an episode
    is flushed: one call per flush, whose results the flush kernels consume.
A plain Python callable is refused: there is no host relabelling path."""
from __future__ import annotations

from . import _lib as L


class TorchReward:
    """A reward function written in PyTorch: `fn(achieved_goal, goal) -> (reward, done)`.

    `achieved_goal` and `goal` are CUDA float32 tensors [N, G] on the ring's device, N being every (row, goal) pair of one flush.
    `reward` must be float32 [N] or [N, 1]; `done` bool (or any numeric dtype, non-zero = done) [N] or [N, 1], on the same device.
    `fn` must be row-wise: output row i may depend on input row i only, because the rows of one call come from many episodes and
    goals.  It runs on the current CUDA stream of the writing thread, under torch.no_grad().

    Sample-time relabelling (her_mode "future", `temporal_sample(relabel_prob > 0)`) evaluates the reward per window row inside the
    gather kernels and so needs a `RewardOp`; with a TorchReward it raises a ConfigurationError.  Ring snapshots record that the
    reward was a TorchReward but not `fn` itself: set it again before `load_state_dict`."""

    def __init__(self, fn):
        if not callable(fn):
            raise TypeError(f"TorchReward needs a callable fn(achieved_goal, goal) -> (reward, done), got {type(fn).__name__}")
        self.fn = fn

    def __call__(self, achieved_goal, goal):
        """Evaluate fn and check what it returned: (reward float32 [N], done uint8 [N]), both contiguous."""
        import torch  # the package imports without torch; its callers already hold CUDA tensors
        n = achieved_goal.shape[0]
        with torch.no_grad():
            out = self.fn(achieved_goal, goal)
        if not (isinstance(out, (tuple, list)) and len(out) == 2):
            raise TypeError("TorchReward fn must return a pair (reward, done)")
        reward, done = out
        for name, t in (("reward", reward), ("done", done)):
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"TorchReward fn returned a {type(t).__name__} as {name}, expected a torch.Tensor")
            if t.device != achieved_goal.device:
                raise ValueError(f"TorchReward fn returned {name} on {t.device}, expected {achieved_goal.device}")
            if tuple(t.shape) not in ((n,), (n, 1)):
                raise ValueError(f"TorchReward fn returned {name} of shape {tuple(t.shape)}, expected ({n},) or ({n}, 1)")
        if reward.dtype != torch.float32:
            raise TypeError(f"TorchReward fn returned reward of dtype {reward.dtype}, expected torch.float32")
        if done.dtype.is_complex:
            raise TypeError(f"TorchReward fn returned done of dtype {done.dtype}, expected torch.bool or 0/1 values")
        if done.dtype != torch.bool:
            done = done != 0
        return reward.reshape(n).contiguous(), done.reshape(n).to(torch.uint8).contiguous()


class RewardOp:
    def __init__(self, op: int, params=()):
        self.op = int(op)
        self.params = [float(p) for p in params]

    @classmethod
    def bitflip(cls):
        """franQ/Env/bitflip.py:143-152: all(ag==dg) ? 0 : -1, done = reward==0"""
        return cls(L.REWARD_BITFLIP)

    @classmethod
    def all_geq(cls):
        """franQ/Env/classic_control_goal/classic_goal.py:88-93"""
        return cls(L.REWARD_ALL_GEQ)

    @classmethod
    def first_geq(cls):
        """franQ/Env/classic_control_goal/classic_goal.py:306-311"""
        return cls(L.REWARD_FIRST_GEQ)

    @classmethod
    def weighted_pnorm(cls, weights, success_threshold, p=0.5):
        """franQ/Env/eleurent_parking.py:42-55: -(sum |ag-dg|*w)^p, done = reward > -threshold"""
        return cls(L.REWARD_WEIGHTED_PNORM, [p, success_threshold, *list(weights)])

    @classmethod
    def coerce(cls, obj):
        """A RewardOp or TorchReward unchanged; "bitflip" / "all_geq" / "first_geq"; an object carrying `fdql_reward_op`."""
        if isinstance(obj, (cls, TorchReward)):
            return obj
        if isinstance(obj, str):
            return {"bitflip": cls.bitflip, "all_geq": cls.all_geq, "first_geq": cls.first_geq}[obj]()
        op = getattr(obj, "fdql_reward_op", None)
        if isinstance(op, cls):
            return op
        raise TypeError("compute_reward must be a fastdeepqlearning_b200.RewardOp (device functor); arbitrary Python "
                        "callables cannot run inside the CUDA relabel kernels and there is no host fallback.  For write-time "
                        "relabelling (her_mode 'final', 'random' or 'vmap') wrap a batched PyTorch function as "
                        "fastdeepqlearning_b200.TorchReward(fn)")

    def c_params(self):
        return L.f32_array(self.params)


def require_device_functor(op, what):
    """Raise the ConfigurationError of a sample-time path handed a TorchReward."""
    if isinstance(op, TorchReward):
        from .Replay.wrappers.torch_dataloader import ConfigurationError
        raise ConfigurationError(f"{what} evaluates the reward inside the CUDA gather kernels and needs a device functor "
                                 "(fastdeepqlearning_b200.RewardOp); a TorchReward serves write-time relabelling only "
                                 "(her_mode 'final', 'random' or 'vmap')")
