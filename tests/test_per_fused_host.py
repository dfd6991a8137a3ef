"""CPU checks of fdql_fused_pass_per's argument validation: NULL or inconsistent arguments give FDQL_EINVAL and a message before any
device work (and before the store is read)."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import fastdeepqlearning_b200 as pkg
    return pkg


def call(L, per=None, n_windows=4, flags=None, goal_rows=None, beta=None, is_weight=None, critic_weight=None, opts=0, M=0,
         loss=None, loss_starts=None):
    d = ctypes.c_void_p(16)  # never dereferenced: every check below fails before any pointer is read
    out = (ctypes.c_void_p * 1)(16)
    params = (ctypes.c_float * 1)(0.0)
    return L.fdql_fused_pass_per(per, n_windows, 2, 0.8, 1, 0, None, None, beta, d, flags, goal_rows, is_weight, critic_weight, 1, params, 0,
                                 0.99, opts, 0, out, d, d, d, M, 125, 10, d, d, d, d, d, d, None, 0.2, 0.99, loss, d, None, loss_starts,
                                 None, None)


def test_fused_per_argument_validation_needs_no_gpu(built):
    from fastdeepqlearning_b200 import _lib as Lm
    L = built.lib()
    fake = ctypes.c_void_p(8)
    d = ctypes.c_void_p(16)
    cases = [
        (dict(per=None), b"null priority store"),
        (dict(per=fake, n_windows=-1), b"bad sizes"),
        (dict(per=fake, flags=d), b"flags and goal_rows"),
        (dict(per=fake, is_weight=d), b"beta_dev"),
        (dict(per=fake, critic_weight=d, is_weight=d, beta=d), b"FDQL_OPT_EMIT_LEARNER_AUX"),
        (dict(per=fake, critic_weight=d, opts=Lm.OPT_EMIT_LEARNER_AUX, beta=d), b"is_weight"),
        (dict(per=fake, M=4, loss=d), b"loss_starts"),
        (dict(per=fake, M=4, loss_starts=d), b"loss_starts"),
        (dict(per=fake, n_windows=0, M=4), b"loss_starts"),
    ]
    for kw, word in cases:
        assert call(L, **kw) == Lm.FDQL_EINVAL, kw
        assert word in L.fdql_last_error(), (kw, L.fdql_last_error())
