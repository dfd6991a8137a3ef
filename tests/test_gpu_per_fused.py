"""GPU checks of fdql_fused_pass_per (prioritized draw in the gather role of the fused pass, priority update after the loss): bit for
bit against the separate launches over several passes (streams, weights, batch, loss, gradient and every tree level), draws that follow
the priorities, injected offsets against oracle/per.py, a captured sequence against the eager one while the ring fills, and alpha = 0."""
import ctypes as C

import numpy as np
import pytest

from oracle import per as P

pytestmark = pytest.mark.gpu
G = 16


def npy(t):
    return t.detach().cpu().numpy()


class Pass:
    """One ring with a priority store and the buffers of a sequence of passes; `fused(k)` is call k of fdql_fused_pass_per (gather of
    batch k, loss and update of batch k - 1), `separate(k)` the same work as fdql_per_sample -> co-resident fdql_sample_gather ->
    critic weight -> fdql_tqc_loss -> fdql_per_update."""

    def __init__(self, fdql, n, T, n_atoms, n_drop, ep_len=64, permute=False, with_lb=True, with_stats=True, alpha=0.6, cap=None,
                 n_eps=None, seed=0, device_counter=False, weights=True):
        import torch
        from fastdeepqlearning_b200 import Replay, _lib as L
        from test_gpu_replay import _synthetic
        self.torch, self.L, self.lib = torch, L, fdql.lib()
        rng = np.random.default_rng(5 + seed)
        n_eps = n_eps or 600 * 64 // ep_len + 1
        cols, lengths, _, _, _ = _synthetic(rng, n_eps, 0, G, obs=64, act=8, fixed_len=ep_len)
        if permute:
            order = ["obs_1d", "episode_step", "action", "mc_return", "achieved_goal", "task_done", "desired_goal", "reward", "episode_done"]
            cols = {k: cols[k] for k in order}
        self.cols, self.lengths = cols, lengths
        N = int(lengths.sum())
        self.ring = Replay.ReplayMemory(cap or N + 1, 4096, T)
        self.ring.set_reward_op(fdql.RewardOp.bitflip(), 0.99)
        self.ring.enable_priorities(alpha=alpha, eps=1e-3, eta=0.9)
        self.ring.add_rows(cols, episode_lengths=lengths, with_returns=True)
        self.ring.set_priority_beta(0.7)
        self.counter_dev = None
        if device_counter:
            self.counter_dev = torch.zeros(4, dtype=torch.int64, device="cuda")
        self.n, self.T, self.n_atoms, self.n_drop, self.with_lb, self.with_stats = n, T, n_atoms, n_drop, with_lb, with_stats
        M = (T - 1) * n
        gen = torch.Generator(device="cuda").manual_seed(n)
        self.z = torch.randn(M, n_atoms, device="cuda", generator=gen) * 3
        self.q = torch.randn(M, n_atoms, device="cuda", generator=gen) * 3
        self.lp = torch.randn(M, device="cuda", generator=gen)
        self.bufs, self.losses = {}, {}
        self.opts = L.OPT_EMIT_LEARNER_AUX | L.OPT_EXACT_EPISODE_STEP
        self.xi = None
        self.weights = weights  # False: no is_weight / critic_weight and no beta_dev (the loss takes aux_weight)

    def p(self, t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def sp(self):
        return C.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def buf(self, k):
        torch, n, T = self.torch, self.n, self.T
        if k not in self.bufs:
            out = {key: torch.full((T, n, w), -7.0, device="cuda") for key, w in zip(self.ring._keys, self.ring._widths)}
            self.bufs[k] = {"out": out, "outp": self.L.ptr_array([out[key].data_ptr() for key in self.ring._keys]),
                            "mask": torch.empty(T, n, device="cuda"), "contig": torch.empty(T - 1, n, device="cuda"),
                            "weight": torch.empty(T - 1, n, device="cuda"), "critic": torch.full((T - 1, n), -7.0, device="cuda"),
                            "isw": torch.full((n,), -7.0, device="cuda"), "st": torch.empty(n, dtype=torch.int64, device="cuda"),
                            "fl": torch.empty(n, dtype=torch.uint8, device="cuda"), "go": torch.empty(n, dtype=torch.int64, device="cuda")}
            M = (T - 1) * n
            self.losses[k] = (torch.empty(M, device="cuda"), torch.empty(M, self.n_atoms, device="cuda"),
                              torch.zeros(4, dtype=torch.float64, device="cuda"))
        return self.bufs[k]

    def loss_args(self, k):
        b = self.buf(k)
        loss, grad, stats = self.losses[k]
        return ((self.T - 1) * self.n, self.n_atoms, self.n_drop, self.p(self.z), self.p(self.q), self.p(self.lp),
                self.p(b["out"]["reward"][1:]), self.p(b["mask"][1:]), self.p(b["out"]["mc_return"][1:]) if self.with_lb else None,
                self.p(b["critic"] if self.weights else b["weight"]), 0.2, 0.99, self.p(loss), self.p(grad), self.p(stats) if self.with_stats else None)

    def draw_args(self, k):
        return (self.L.GOAL_FUTURE, 0.8, 11, k, self.p(self.counter_dev), self.p(self.xi))

    def weight_ptrs(self, g):
        if not self.weights:
            return None, None, None
        return self.p(self.ring._per_beta), self.p(g["isw"]), self.p(g["critic"])

    def fused(self, k, n_windows=None):
        L, r = self.L, self.ring
        g = self.buf(k)
        beta, isw, critic = self.weight_ptrs(g)
        params, n_params = r.reward_op.c_params()
        if k == 0:
            lo = (0, self.n_atoms, self.n_drop) + (None,) * 7 + (0.2, 0.99) + (None,) * 3
            ls, lc = None, None
        else:
            lo = self.loss_args(k - 1)
            ls, lc = self.p(self.buf(k - 1)["st"]), self.p(self.buf(k - 1)["contig"])
        nw = self.n if n_windows is None else n_windows
        L.check(self.lib.fdql_fused_pass_per(r._per, nw, *self.draw_args(k), beta, self.p(g["st"]), self.p(g["fl"]),
                                             self.p(g["go"]), isw, critic, r.reward_op.op, params, n_params, 0.99,
                                             self.opts, 4096, g["outp"], self.p(g["mask"]), self.p(g["contig"]), self.p(g["weight"]), *lo,
                                             ls, lc, self.sp()))

    def separate(self, k):
        L, r, n = self.L, self.ring, self.n
        g = self.buf(k)
        params, n_params = r.reward_op.c_params()
        beta, isw, _ = self.weight_ptrs(g)
        L.check(self.lib.fdql_per_sample(r._per, n, *self.draw_args(k), beta, self.p(g["st"]), self.p(g["fl"]),
                                         self.p(g["go"]), isw, self.sp()))
        # (window modulus: the capacity -- a drawn start is < len - T, so no window wraps)
        L.check(self.lib.fdql_sample_gather(r._h, n, self.T, r._maxlen, self.p(g["st"]), self.p(g["fl"]), self.p(g["go"]), r.reward_op.op,
                                            params, n_params, 0.99, self.opts | L.OPT_CORESIDENT, 4096, g["outp"], self.p(g["mask"]),
                                            self.p(g["contig"]), self.p(g["weight"]), self.sp()))
        if self.weights:
            g["critic"].copy_(g["weight"] * g["isw"][None])
        if k > 0:
            a = self.loss_args(k - 1)
            L.check(self.lib.fdql_tqc_loss(*a[:14], None, a[14], self.sp()))
            prev = self.buf(k - 1)
            L.check(self.lib.fdql_per_update(r._per, n, self.p(prev["st"]), a[12], self.p(prev["contig"]), self.sp()))

    def tree(self):
        leaves, qmax = self.ring.priority_views()
        return [leaves.clone(), qmax.clone()] + [t.clone() for lv in self.ring.priority_tree() for t in lv]

    def set_leaves(self, q):
        leaves, _ = self.ring.priority_views()
        leaves.copy_(self.torch.as_tensor(q, device="cuda"))
        self.ring.rebuild_priorities()


def same_bits(a, b):
    import torch
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    if a.dtype == torch.float64:
        return torch.equal(a.view(torch.int64), b.view(torch.int64))
    return torch.equal(a, b)


# the shapes of test_gpu_r2.py::test_fused_pass_equals_the_two_launches, plus a non-finite q_pred row and forced duplicate starts
@pytest.mark.parametrize("n,T,n_atoms,n_drop,with_lb,with_stats,ep_len,permute,case", [
    (24576, 2, 125, 10, True, True, 64, False, ""),            # the fused kernel, headline shape (T = 2 build, compiled copy plan)
    (20000, 2, 125, 10, False, False, 64, False, ""),          # ragged last group and chunk, no lower bound / summaries
    (6001, 5, 125, 10, True, True, 64, False, ""),             # five-row windows: general build
    (24576, 2, 100, 8, True, False, 64, False, ""),            # 100 atoms
    (24576, 2, 125, 10, True, True, 40000, False, ""),         # episodes without a chain of equal goals: out-of-line tail scan
    (24576, 2, 125, 10, True, True, 64, True, ""),             # scalar keys in another order: general build
    (3000, 2, 125, 10, True, True, 64, False, ""),             # batch too small for the fused kernel: separate launches
    (24576, 2, 50, 4, True, True, 64, False, ""),              # 64-entry loss tables: separate launches
    (24576, 2, 125, 10, True, True, 64, False, "nonfinite"),   # a NaN q_pred row: its window's priority becomes q_max
    (24576, 2, 125, 10, True, True, 64, False, "duplicates"),  # a few heavy leaves: many windows share a start
    (24576, 2, 125, 10, True, True, 64, False, "noweights"),   # no is_weight / critic_weight / beta_dev: nothing reads beta
    (3000, 2, 125, 10, True, True, 64, False, "noweights"),    # ... and the same through the separate launches
])
def test_fused_per_pass_equals_the_separate_launches(fdql, n, T, n_atoms, n_drop, with_lb, with_stats, ep_len, permute, case):
    import torch
    passes = 4  # batch 3 draws from a tree that batch 1's update changed
    sides = [Pass(fdql, n, T, n_atoms, n_drop, ep_len, permute, with_lb, with_stats, weights=case != "noweights") for _ in range(2)]
    for s in sides:
        if case == "nonfinite":
            s.q[7] = float("nan")
        if case == "duplicates":
            s.ring.apply_pending_priorities()
            leaves, _ = s.ring.priority_views()
            q = npy(leaves).copy()
            q[np.flatnonzero(q > 0)[::4099]] = 1e4
            s.set_leaves(q)
    fu, se = sides
    for k in range(passes):
        fu.fused(k)
        se.separate(k)
        torch.cuda.synchronize()
        for a, b in zip(fu.tree(), se.tree()):
            assert same_bits(a, b), k
    if case == "duplicates":
        st = npy(fu.buf(1)["st"])
        assert len(np.unique(st)) < len(st) // 2
    if case == "nonfinite":
        assert not np.isfinite(npy(fu.losses[0][0])[7])
    for k in range(passes):
        a, b = fu.buf(k), se.buf(k)
        for key in ("st", "fl", "go", "isw", "critic", "mask", "contig", "weight"):
            assert same_bits(a[key], b[key]), (k, key)
        for key in a["out"]:
            assert same_bits(a["out"][key], b["out"][key]), (k, key)
        if case == "noweights":  # never written
            assert bool((a["isw"] == -7).all()) and bool((a["critic"] == -7).all())
        else:
            assert (npy(a["isw"]) <= 1).all() and (npy(a["isw"]) > 0).all()
    for k in range(passes - 1):
        (l1, g1, s1), (l2, g2, s2) = fu.losses[k], se.losses[k]
        assert same_bits(l1, l2) and same_bits(g1, g2), k
        if with_stats:
            np.testing.assert_allclose(npy(s1), npy(s2), rtol=1e-12)
    # the loss and the update alone (n_windows = 0) and the gather alone (M = 0: call 0 above) through the same entry point
    before = fu.tree()
    fu.fused(passes, n_windows=0)
    torch.cuda.synchronize()
    assert any(not same_bits(x, y) for x, y in zip(before, fu.tree()))


def test_fused_draws_follow_the_priorities_chi_square(fdql):
    import torch
    from scipy import stats
    n = 24576
    s = Pass(fdql, n, 2, 125, 10, ep_len=32, cap=400, n_eps=8)  # 256 rows
    s.ring.apply_pending_priorities()
    n_elig = len(s.ring) - 2
    rng = np.random.default_rng(2)
    q = np.zeros(400, np.float32)
    q[:n_elig] = rng.uniform(0.1, 4.0, n_elig).astype(np.float32)
    counts = np.zeros(400, np.int64)
    s.fused(0)
    for k in range(1, 41):
        s.set_leaves(q)  # the call's draw reads the tree before its update writes it
        s.fused(k)
        counts += np.bincount(npy(s.buf(k)["st"]), minlength=400)
        torch.cuda.synchronize()
        del s.bufs[k - 1], s.losses[k - 1]
    expected = q[:n_elig].astype(np.float64) / q[:n_elig].astype(np.float64).sum() * counts.sum()
    assert counts[n_elig:].sum() == 0
    _, pv = stats.chisquare(counts[:n_elig], expected)
    assert pv > 1e-4, pv


def test_fused_injected_xi_on_dyadic_priorities_matches_the_oracle(fdql):
    import torch
    n = 24576
    s = Pass(fdql, n, 2, 125, 10, cap=50000, n_eps=700)
    s.ring.apply_pending_priorities()
    cap, n_elig = 50000, len(s.ring) - 2
    rng = np.random.default_rng(1)
    q = np.zeros(cap, np.float32)
    q[:n_elig] = np.ldexp(1.0, rng.integers(-10, 6, n_elig)).astype(np.float32)  # every fp64 sum exact in any order
    s.set_leaves(q)
    xi = rng.random(n)
    s.xi = torch.as_tensor(xi, device="cuda")
    s.fused(0)  # the gather alone: separate launches
    s.set_leaves(q)
    s.fused(1)  # the fused kernel draws batch 1 before the update of batch 0
    torch.cuda.synchronize()
    want_s, want_w = P.sample(q, xi, np.float32(0.7))
    for k in (0, 1):
        np.testing.assert_array_equal(npy(s.buf(k)["st"]), want_s)
        np.testing.assert_allclose(npy(s.buf(k)["isw"]), want_w, rtol=1e-6)


def test_captured_fused_passes_keep_to_the_eligible_range_and_equal_the_eager_ones(fdql):
    import torch
    n, T = 24576, 2
    kw = dict(ep_len=64, cap=80000, n_eps=200, device_counter=True)
    eager, graph = Pass(fdql, n, T, 125, 10, **kw), Pass(fdql, n, T, 125, 10, **kw)
    for s in (eager, graph):  # warm-up: the gather alone, one fused pass
        s.fused(0)
        s.fused(1)
    torch.cuda.synchronize()
    # three passes over buffers 2, 3, 4 (call 2 reads batch 1's buffers), captured once; the eager side runs the same calls
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    for k in (2, 3, 4):
        graph.buf(k)
    with torch.cuda.graph(g):
        for k in (2, 3, 4):
            graph.fused(k)
    for k in (2, 3, 4):
        eager.fused(k)
    g.replay()
    torch.cuda.synchronize()
    for k in (2, 3, 4):
        for key in ("st", "fl", "go", "isw", "critic", "weight"):
            assert same_bits(eager.buf(k)[key], graph.buf(k)[key]), (k, key)
        for key in eager.buf(k)["out"]:
            assert same_bits(eager.buf(k)["out"][key], graph.buf(k)["out"][key]), (k, key)
    for a, b in zip(eager.tree(), graph.tree()):
        assert same_bits(a, b)
    # replays while the ring fills: no start outside [0, len - T), and the gathered rows are the ring's rows at the drawn starts (the
    # length at capture time is not the window modulus).  The ring does not wrap: row r holds the r-th row added.
    rng = np.random.default_rng(3)
    from test_gpu_replay import _synthetic
    rows = {key: [graph.cols[key]] for key in ("obs_1d", "action")}
    seen = 0
    for step in range(12):
        cols, lengths, _, _, _ = _synthetic(rng, 40, 0, G, obs=64, act=8, fixed_len=64)
        graph.ring.add_rows(cols, episode_lengths=lengths, with_returns=True)
        for key in rows:
            rows[key].append(cols[key])
        graph.ring.apply_pending_priorities()
        g.replay()
        torch.cuda.synchronize()
        ring_rows = {key: np.concatenate(v) for key, v in rows.items()}
        for k in (2, 3, 4):
            st = npy(graph.buf(k)["st"])
            assert (st >= 0).all() and (st < len(graph.ring) - T).all(), step
            seen = max(seen, int(st.max()))
            for key, v in ring_rows.items():
                np.testing.assert_array_equal(npy(graph.buf(k)["out"][key]), v[st[None, :] + np.arange(T)[:, None]], err_msg=f"{step} {k} {key}")
    assert seen > 12800 + 20000
    assert int(graph.counter_dev[0]) == 2 + 3 * 13  # one draw per call: two eager calls, three per replay


def test_alpha_zero_gives_unit_weights_and_the_uniform_critic_weight(fdql):
    import torch
    s = Pass(fdql, 24576, 2, 125, 10, alpha=0.0)
    for k in range(3):
        s.fused(k)
    torch.cuda.synchronize()
    for k in range(3):
        b = s.buf(k)
        assert bool((b["isw"] == 1).all())
        assert same_bits(b["critic"], b["weight"])


@pytest.mark.parametrize("n,n_atoms,n_drop,fused", [(24576, 125, 10, True), (3000, 125, 10, False), (24576, 50, 4, False)])
def test_the_fused_kernel_serves_the_fused_shapes(fdql, n, n_atoms, n_drop, fused):
    """The bit-for-bit test above cannot tell the fused kernel from the separate launches: the kernels a call runs, from the profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    s = Pass(fdql, n, 2, n_atoms, n_drop)
    s.fused(0)
    s.fused(1)  # (first launches of each kernel outside the profiled call)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.fused(2)
        torch.cuda.synchronize()
    names = " ".join(e.key for e in prof.key_averages())
    assert ("fused_pass_per_kernel" in names) == fused, names
    assert ("per_sample_kernel" in names) == (not fused), names
    assert "per_claim_kernel" in names  # the update of batch 1
