"""CPU checks of prioritized replay: the numpy restatement (oracle/per.py) against a naive searchsorted(cumsum) and hand-built update
cases, and the argument validation of the fdql_per_* ABI and its Python mirror without a GPU."""
import ctypes

import numpy as np
import pytest

from oracle import per as P


def dyadic_leaves(rng, n, n_elig):
    q = np.zeros(n, np.float32)
    q[:n_elig] = np.ldexp(1.0, rng.integers(-12, 4, n_elig)).astype(np.float32)
    return q


@pytest.mark.parametrize("n,n_elig", [(2, 1), (31, 20), (33, 33), (1025, 1000), (40000, 39990)])
def test_descent_equals_searchsorted_of_the_cumsum(n, n_elig):
    rng = np.random.default_rng(n)
    q = dyadic_leaves(rng, n, n_elig)
    tree = P.build(q)
    assert len(tree[-1][0]) == 1 and tree[-1][0][0] == q.astype(np.float64).sum()  # dyadic: exact in any order
    assert tree[-1][1][0] == q[q > 0].min()
    xi = rng.random(512)
    t = P.targets(tree, xi)
    want = np.searchsorted(np.cumsum(q.astype(np.float64)), t, side="right")
    np.testing.assert_array_equal(P.descend(q, tree, t), want)
    starts, w = P.sample(q, xi, 0.4)
    assert (q[starts] > 0).all() and (starts < n_elig).all()
    np.testing.assert_allclose(w, (q[q > 0].min() / q[starts].astype(np.float64)) ** np.float64(np.float32(0.4)), rtol=1e-7)
    assert w.max() <= 1.0


def test_rounding_past_the_last_positive_leaf_is_clamped():
    q = np.zeros(100, np.float32)
    q[:70] = 1.0
    tree = P.build(q)
    assert P.descend(q, tree, [70.0, 1e9])[0] == 69 and P.descend(q, tree, [1e9])[0] == 69


def test_levels_of_a_1e7_ring():
    assert P._levels_of(10_000_000) == [10_000_000, 312500, 9766, 306, 10, 1]


def test_update_rule_hand_built():
    q = np.ones(10, np.float32)
    q[8:] = 0  # not eligible
    starts = np.array([1, 2, 1, 8, 3, 4, 5])
    # T = 3: two transitions per window, time-major [T-1, B]
    loss = np.array([[1.0, 4.0, 2.0, 5.0, 1.0, np.nan, 3.0],
                     [3.0, 0.0, 6.0, 5.0, 2.0, 1.0, 9.0]], np.float32)
    contig = np.array([[1, 1, 1, 1, 0, 1, 0],
                       [1, 0, 1, 1, 0, 1, 1]], np.float32)
    new, qmax = P.update(q, 1.0, starts, loss, contig, alpha=1.0, eps=0.5, eta=0.5)
    assert new[1] == np.float32(0.5 * 6 + 0.5 * 4 + 0.5)      # window 2 (the later duplicate) wins over window 0
    assert new[2] == np.float32(0.5 * 4 + 0.5 * 4 + 0.5)      # one contiguous transition
    assert new[8] == 0                                      # ineligible leaf stays 0
    assert new[3] == np.float32(0.5)                        # no contiguous transition: delta = 0
    assert new[4] == np.float32(1.0)                        # NaN loss: the q_max of before the update
    assert new[5] == np.float32(0.5 * 9 + 0.5 * 9 + 0.5)
    assert qmax == np.float32(9.5)
    # T = 2 with eta = 0.9: delta is the loss itself
    new, _ = P.update(np.ones(4, np.float32), 1.0, [0, 3], np.array([[2.0, np.inf]], np.float32), None, alpha=0.5, eps=1e-6, eta=0.9)
    assert new[0] == np.float32((2.0 + np.float64(np.float32(1e-6))) ** 0.5) and new[3] == 1.0


def test_update_floor_keeps_eligible_leaves_positive():
    new, _ = P.update(np.ones(2, np.float32), 1.0, [0], np.zeros((1, 1), np.float32), None, alpha=40.0, eps=1e-6, eta=0.9)
    assert new[0] == np.finfo(np.float32).tiny


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import fastdeepqlearning_b200 as pkg
    return pkg


def test_per_argument_validation_needs_no_gpu(built):
    L = built.lib()
    out = ctypes.c_void_p()
    fake = ctypes.c_void_p(8)  # never dereferenced: every check below fails before the arena is read
    assert L.fdql_per_create(None, 2, 0.6, 1e-6, 0.9, ctypes.byref(out)) == -1
    for T, alpha, eps, eta, word in [(1, 0.6, 1e-6, 0.9, b"T must"), (2, -0.1, 1e-6, 0.9, b"alpha"), (2, 0.6, 0.0, 0.9, b"eps"),
                                     (2, 0.6, -1.0, 0.9, b"eps"), (2, 0.6, 1e-6, 1.5, b"eta"), (2, 0.6, 1e-6, -0.1, b"eta"),
                                     (2, float("nan"), 1e-6, 0.9, b"alpha")]:
        assert L.fdql_per_create(fake, T, alpha, eps, eta, ctypes.byref(out)) == -1
        assert word in L.fdql_last_error()
    assert L.fdql_per_sample(None, 4, 2, 0.0, 0, 0, None, None, None, None, None, None, None, None) == -1
    assert L.fdql_per_update(None, 4, None, None, None, None) == -1
    assert L.fdql_per_apply_pending(None, None) == -1
    assert L.fdql_per_rebuild(None, None) == -1
    assert L.fdql_per_view(None, None, None) == -1
    assert L.fdql_per_level_view(None, 1, None, None, None) == -1
    assert L.fdql_per_destroy(None) == 0


def test_python_mirror_validates_and_refuses_out_of_scope_modes(built):
    from fastdeepqlearning_b200 import Agent, Replay
    rm = Replay.ReplayMemory(100, 4, 2, device="cuda:0")
    for kw in (dict(alpha=-1), dict(eps=0), dict(eta=2)):
        with pytest.raises(ValueError):
            rm.enable_priorities(**kw)
    with pytest.raises(NotImplementedError):
        rm.sample(prioritized=True)
    with pytest.raises(NotImplementedError):
        Replay.wrappers.HindsightVmapRead(rm).temporal_sample(prioritized=True)
    conf = Agent.LearnerConf()
    assert conf.use_prioritized_replay is False and conf.per_alpha == 0.6 and conf.per_beta0 == 0.4 and conf.per_eta == 0.9
