"""fastdeepqlearning_b200 -- B200 (sm_100a) learner hot path of franQ / FastDeepQLearning.

Host-side mirror of the reference's `franQ.Replay` and `franQ.Agent.components` interfaces over libfdql.so
(hand-written CUDA behind the C ABI in include/fdql.h).  No CPU fallback: importing is cheap, but every
operation needs the built library and a CUDA device and fails loudly otherwise."""
from ._lib import lib, FdqlError, OversampleError, LIB_PATH, EXPORTS  # noqa: F401
from .reward_ops import RewardOp, TorchReward  # noqa: F401

__all__ = ["lib", "FdqlError", "OversampleError", "RewardOp", "TorchReward", "Replay", "Agent", "Runner"]


def __getattr__(name):  # lazy: the sub-packages import torch
    if name in ("Replay", "Agent", "Runner"):
        import importlib
        return importlib.import_module(f"{__name__}.{name}")
    raise AttributeError(name)
