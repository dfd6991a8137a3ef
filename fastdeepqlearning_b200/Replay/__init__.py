"""Mirror of franQ/Replay/__init__.py: `make(conf, **kwargs) -> (read_heads, write_heads)`, one pair per
`conf.num_instances` (one shard per actor stream; with torch.distributed the shards of this rank only)."""
from .async_replay_memory import AsyncReplayMemory
from .replay_memory import ReplayMemory, OversampleError
from . import wrappers
from ..reward_ops import RewardOp, require_device_functor


def make(conf, **kwargs):
    """Replay/__init__.py:8-38.  Composition order is the reference's: NStepReturn (inner) -> SquashRewards -> HER (outer).
    `kwargs["compute_reward"]` is a device reward functor (fastdeepqlearning_b200.RewardOp) or, for the write-time modes
    ("final", "random", "vmap"), a fastdeepqlearning_b200.TorchReward."""
    device = getattr(conf, "training_device", "cuda:0")
    # conf.replay_key_dtypes (optional): {key: uint8 / int8} keys stored at one byte per element, sampled as fp32 (ReplayMemory)
    shards = [AsyncReplayMemory(int(conf.replay_size), conf.batch_size, conf.temporal_len, device=device,
                                key_dtypes=getattr(conf, "replay_key_dtypes", None))
              for _ in range(conf.num_instances)]
    write_heads = read_heads = shards
    her_mode = getattr(conf, "her_mode", "final")
    if getattr(conf, "use_prioritized_replay", False):  # prioritized replay (not a reference mode): a priority per window start
        if conf.use_HER and her_mode == "vmap":
            raise NotImplementedError("use_prioritized_replay is not supported with her_mode='vmap'")
        for r in shards:
            r.enable_priorities(alpha=getattr(conf, "per_alpha", 0.6), eps=getattr(conf, "per_eps", 1e-6), eta=getattr(conf, "per_eta", 0.9))
    if conf.use_nStep_lowerbounds:
        if her_mode == "vmap":  # Replay/__init__.py:21-23; quirk Q7 is opt-in (conf.vmap_reference_done_quirk)
            write_heads = [wrappers.NStepReturnVmap(r, conf.nStep_return_steps, conf.gamma,
                                                    reference_done_quirk=getattr(conf, "vmap_reference_done_quirk", False))
                           for r in write_heads]
        else:
            write_heads = [wrappers.NStepReturn(r, conf.nStep_return_steps, conf.gamma) for r in write_heads]
    if getattr(conf, "use_squashed_rewards", False) and not conf.use_HER:
        write_heads = [wrappers.SquashRewards(r) for r in write_heads]
    if conf.use_HER:
        if her_mode == "vmap":  # Replay/__init__.py:30-32
            write_heads = [wrappers.HindsightVmapWrite(r, kwargs["compute_reward"]) for r in write_heads]
            read_heads = [wrappers.HindsightVmapRead(r) for r in read_heads]
        elif her_mode == "future":  # sample-time relabelling (BASELINE.json configs[2]); rows are stored once
            require_device_functor(RewardOp.coerce(kwargs["compute_reward"]), "her_mode='future' (sample-time relabelling)")
            for r in shards:
                r.replay.set_reward_op(kwargs["compute_reward"], conf.gamma)
            read_heads = [wrappers.SampleTimeHindsight(r, relabel_prob=getattr(conf, "her_relabel_prob", 0.8)) for r in read_heads]
            write_heads = [wrappers.IgnoreKeys(r) for r in write_heads]
        else:
            write_heads = [wrappers.HindsightNStepReplay(r, kwargs["compute_reward"], mode=her_mode) for r in write_heads]
    return read_heads, write_heads
