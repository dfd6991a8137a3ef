"""CPU checks of write-time relabelling with a TorchReward: the argument validation of fdql_her_flush_episodes_given and
fdql_vmap_flush_episodes_given (NULL or inconsistent arguments give FDQL_EINVAL and a message before the arena or any device array
is read), the checks TorchReward applies to what the user's function returns, and the configuration errors of the sample-time
paths, which need a device functor."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import fastdeepqlearning_b200 as pkg
    return pkg


def her_given(L, a=ctypes.c_void_p(8), n_eps=2, n_rows=5, table=True, reward=True, done=True, reward_dg=True):
    d = ctypes.c_void_p(16)  # never dereferenced: every check below fails before any pointer is read
    t = d if table else None
    return L.fdql_her_flush_episodes_given(a, n_eps, t, t, t, t, n_rows, d if reward else None, d if done else None,
                                           d if reward_dg else None, 0.99, 1, None)


def vmap_given(L, a=ctypes.c_void_p(8), n_eps=2, n_rows=5, mode=1, table=True, picks=True, grid=True):
    d = ctypes.c_void_p(16)
    t = d if table else None
    g = d if grid else None
    return L.fdql_vmap_flush_episodes_given(a, n_eps, t, t, d if picks else None, 0, 1, 2, -1, n_rows, g, g, 0.99, mode, 0, None)


def test_given_flush_argument_validation_needs_no_gpu(built):
    from fastdeepqlearning_b200 import _lib as Lm
    L = built.lib()
    her_cases = [
        (dict(a=None), b"bad argument"),
        (dict(n_eps=-1), b"bad argument"),
        (dict(n_rows=-1), b"bad argument"),
        (dict(n_eps=0, n_rows=3), b"no episodes"),
        (dict(table=False), b"null episode table"),
        (dict(reward=False), b"null reward"),
        (dict(done=False), b"null reward"),
        (dict(reward_dg=False), b"reward_dg"),
    ]
    for kw, word in her_cases:
        assert her_given(L, **kw) == Lm.FDQL_EINVAL, kw
        assert word in L.fdql_last_error(), (kw, L.fdql_last_error())
    assert her_given(L, n_eps=0, n_rows=0) == Lm.FDQL_OK
    vmap_cases = [
        (dict(a=None), b"bad argument"),
        (dict(n_rows=-1), b"bad argument"),
        (dict(mode=2), b"mode"),
        (dict(mode=0), b"mode"),
        (dict(mode=5), b"mode"),
        (dict(n_eps=0, n_rows=3), b"no episodes"),
        (dict(table=False), b"null episode table"),
        (dict(picks=False), b"virtual goals"),
        (dict(grid=False), b"null reward or done grid"),
    ]
    for kw, word in vmap_cases:
        assert vmap_given(L, **kw) == Lm.FDQL_EINVAL, kw
        assert word in L.fdql_last_error(), (kw, L.fdql_last_error())
    assert vmap_given(L, n_eps=0, n_rows=0, mode=3) == Lm.FDQL_OK


def _robotics(ag, g):
    d = (ag - g).norm(dim=-1)
    return -(d > 0.05).float(), d <= 0.05


def test_torch_reward_checks_what_fn_returns(built):
    import torch
    TR = built.TorchReward
    ag, g = torch.zeros(6, 3), torch.ones(6, 3)
    r, d = TR(_robotics)(ag, g)
    assert r.dtype == torch.float32 and tuple(r.shape) == (6,) and d.dtype == torch.uint8 and d.tolist() == [0] * 6
    # [N, 1] outputs and numeric dones (non-zero = done) are accepted
    r, d = TR(lambda a, b: (torch.zeros(6, 1), torch.ones(6, 1)))(ag, g)
    assert tuple(r.shape) == (6,) and d.tolist() == [1] * 6
    bad = [
        (lambda a, b: (torch.zeros(5), torch.zeros(5, dtype=torch.bool)), ValueError, "shape"),
        (lambda a, b: (torch.zeros(6, 2), torch.zeros(6, dtype=torch.bool)), ValueError, "shape"),
        (lambda a, b: (torch.zeros(6), torch.zeros(3, 2, dtype=torch.bool)), ValueError, "shape"),
        (lambda a, b: (torch.zeros(6, dtype=torch.float64), torch.zeros(6, dtype=torch.bool)), TypeError, "dtype"),
        (lambda a, b: (torch.zeros(6, dtype=torch.float16), torch.zeros(6, dtype=torch.bool)), TypeError, "dtype"),
        (lambda a, b: (torch.zeros(6), torch.zeros(6, dtype=torch.complex64)), TypeError, "dtype"),
        (lambda a, b: (torch.zeros(6, device="meta"), torch.zeros(6, dtype=torch.bool)), ValueError, "meta"),
        (lambda a, b: (torch.zeros(6), torch.zeros(6, dtype=torch.bool, device="meta")), ValueError, "meta"),
        (lambda a, b: (torch.zeros(6), [False] * 6), TypeError, "torch.Tensor"),
        (lambda a, b: torch.zeros(6), TypeError, "pair"),
    ]
    for fn, exc, word in bad:
        with pytest.raises(exc, match=word):
            TR(fn)(ag, g)
    with pytest.raises(TypeError):
        TR(3)


def test_coerce_keeps_torch_reward_and_refuses_plain_callables(built):
    tr = built.TorchReward(_robotics)
    assert built.RewardOp.coerce(tr) is tr
    with pytest.raises(TypeError, match="TorchReward"):
        built.RewardOp.coerce(_robotics)


def _conf(**kw):
    import types
    d = dict(replay_size=4096, batch_size=8, temporal_len=2, num_instances=1, use_nStep_lowerbounds=True, nStep_return_steps=1000,
             gamma=0.99, use_squashed_rewards=False, use_HER=True, her_mode="future", training_device="cuda:0")
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_sample_time_paths_refuse_a_torch_reward_at_configuration(built):
    from fastdeepqlearning_b200 import Replay
    from fastdeepqlearning_b200.Replay.wrappers import ConfigurationError
    tr = built.TorchReward(_robotics)
    with pytest.raises(ConfigurationError, match="device functor"):
        Replay.make(_conf(her_mode="future"), compute_reward=tr)
    ring = Replay.ReplayMemory(64, 8, 2)
    ring.set_reward_op(tr)
    with pytest.raises(ConfigurationError, match="device functor"):
        Replay.wrappers.SampleTimeHindsight(ring)
    with pytest.raises(ConfigurationError, match="device functor"):
        ring.temporal_sample(relabel_prob=0.8)
    # the write-time modes take it
    for mode in ("final", "random", "vmap"):
        Replay.make(_conf(her_mode=mode), compute_reward=tr)


def test_snapshot_of_a_torch_reward_ring_needs_the_reward_set_again(built):
    from fastdeepqlearning_b200 import Replay
    sd = {"maxlen": 64, "reward_op": "torch"}
    with pytest.raises(ValueError, match="TorchReward"):
        Replay.ReplayMemory(64, 8, 2).load_state_dict(sd)
    ring = Replay.ReplayMemory(64, 8, 2)
    ring.set_reward_op(built.RewardOp.bitflip())
    with pytest.raises(ValueError, match="TorchReward"):
        ring.load_state_dict(sd)
