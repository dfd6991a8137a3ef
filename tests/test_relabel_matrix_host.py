"""CPU checks of what the relabelling parity matrix (test_gpu_relabel_matrix.py) rests on: the fp32-reward form of the oracle
functors, the p-norm functor at every p the matrix uses, and the adversarial goal data reaching each of its deciding cases at every
(functor, goal width)."""
import numpy as np
import pytest

from oracle import cpu_restatement as O
from test_gpu_relabel_matrix import FUNCTORS, WIDTHS, assert_cases_reached, functor, matrix_data, pnorm_weights


def test_fp32_reward_rounds_the_reward_and_keeps_the_fp64_done():
    def fn(ag, dg):
        r = np.array([-(1 + 2.0 ** -30), -1.0, -(1 - 2.0 ** -30)])
        return r, r > -1.0
    r, d = O.fp32_reward(fn)(None, None)
    assert r.dtype == np.float64
    np.testing.assert_array_equal(r, [-1.0, -1.0, -1.0])
    np.testing.assert_array_equal(d, [False, False, True])  # the third reward rounds onto the threshold but is done


@pytest.mark.parametrize("p", [0.5, 1.0, 2.0])
def test_weighted_pnorm_at_each_p(p):
    rng = np.random.default_rng(3)
    w = np.array([1.0, 0.0, 2.0, 0.25])
    ag = rng.standard_normal((50, 4))
    dg = ag + rng.standard_normal((50, 4)) * 0.3
    r, d = O.make_reward_weighted_pnorm(w, 0.7, p)(ag, dg)
    want = -np.array([sum(abs(a - g) * wi for a, g, wi in zip(ra, rg, w)) ** p for ra, rg in zip(ag, dg)])
    np.testing.assert_allclose(r, want, rtol=1e-14)
    np.testing.assert_array_equal(d, want > -0.7)
    assert 0 < d.sum() < len(d)


@pytest.mark.parametrize("name", FUNCTORS)
@pytest.mark.parametrize("G", WIDTHS)
def test_matrix_data_reaches_every_deciding_case(name, G):
    for seed in (0, 1, 2):
        cols = matrix_data(name, G, seed)[0]
        assert_cases_reached(name, G, cols)
        if name.startswith("pnorm"):
            # dyadic goals and weights: the fp64 norm is exact, so no summation order can change a reward or a done
            ag, dg = cols["achieved_goal"].astype(np.float64), cols["desired_goal"].astype(np.float64)
            ok = np.isfinite(ag).all(1)
            terms = np.abs(ag[ok] - dg[ok]) * pnorm_weights(G)
            np.testing.assert_array_equal(terms.sum(1), terms[:, ::-1].sum(1))
            np.testing.assert_array_equal(terms @ np.ones(G), np.sort(terms, 1).sum(1))
            assert functor(name, G)[1][0] == "weighted_pnorm"
