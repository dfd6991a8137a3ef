"""Relabelling parity matrix: every reward functor at every goal width, episode length and relabel route, against the fp64 oracle.

The functors (bitflip, all_geq, first_geq, weighted p-norm with p in {0.5, 1, 2}) are evaluated warp-cooperatively by eval_chunk
with LPR = 1 .. 32 lanes per goal row, chosen from the goal width, and row by row by the vmap fill.  Each relabel site is pinned to
oracle/cpu_restatement.py over the goal widths below (every LPR, each with a full and a partial last float4), over episodes of 1 to
200 rows (one and several 32-row chunks) laid into a ring so that some wrap its physical end, and over adversarial goal data whose
deciding cases the generator counts and requires.

Sites: the episode commit (goal-agnostic term and returns) with sample-time relabelling on every route the debug switch can force,
the write-time hindsight flush, the vmap fill and column select, the TorchReward given path, the drawing entry points that fall back
for non-bitflip functors, and the refusal of goals wider than 128 floats.

Tolerances: goals, dones, episode steps, masks and flag-functor rewards bit-exact.  p-norm rewards within 1 fp32 ulp of the oracle
(whose functor rounds its reward to fp32 as it reaches the ring, O.fp32_reward); the p-norm data lie on a dyadic grid with dyadic
weights, so the fp64 norm is exact in any summation order and its dones must match everywhere.  Sample-time returns within 1e-5
relative; write-time and vmap returns bit-exact wherever the rewards are (they run the reference's sequential recurrence)."""
import ctypes as C
import re

import numpy as np
import pytest

from oracle import cpu_restatement as O

pytestmark = pytest.mark.gpu

WIDTHS = [1, 2, 3, 4, 5, 8, 9, 16, 17, 31, 32, 33, 64, 100, 127, 128]
LENGTHS = [1, 2, 31, 32, 33, 63, 64, 65, 200]
WINDOWS = [1, 2, 5, 33, 50]
FUNCTORS = ["bitflip", "all_geq", "first_geq", "pnorm0.5", "pnorm1", "pnorm2"]
GAMMA = 0.98
CAP, FILL = 512, 300  # ring rows; rows of a first episode, so that the matrix episodes start at row 300 and wrap the ring's end
THR = 1.0
V = 8


def lpr_of(G):
    vecs, lpr = (G + 3) // 4, 1
    while lpr < vecs:
        lpr <<= 1
    return lpr


def pnorm_weights(G):
    """Non-uniform dyadic weights with zeros; the last component and the one the highest lane group reads weigh non-zero."""
    w = np.resize(np.array([1.0, 0.0, 2.0, 0.5, 0.25, 0.0, 1.5, 3.0]), G)
    w[G - 1] = 1.0
    w[hi_component(G)] = 2.0
    return w


def hi_component(G):
    """A component read by a lane of the upper half of the row's lane group (0 when the row has one lane)."""
    lpr = lpr_of(G)
    return min(G - 1, 4 * (lpr // 2)) if lpr > 1 else G - 1


def functor(name, G):
    """(oracle reward_fn in fp64, RewardOp factory args) of one functor at width G."""
    if name.startswith("pnorm"):
        p = float(name[5:])
        return O.make_reward_weighted_pnorm(pnorm_weights(G), THR, p), ("weighted_pnorm", (list(pnorm_weights(G)), THR, p))
    return O.REWARD_OPS[name], (name, ())


def reward_op(fdql, name, G):
    kind, args = functor(name, G)[1]
    return fdql.RewardOp.coerce(kind) if not args else fdql.RewardOp.weighted_pnorm(*args)


def torch_reward(fdql, name, G):
    """The functor restated in torch: the enum path's arithmetic (fp64 norm, fp32 reward)."""
    import torch
    if name.startswith("pnorm"):
        w32, p = np.asarray(pnorm_weights(G), np.float32), float(name[5:])

        def f(ag, g):
            w = torch.as_tensor(w32, device=ag.device).double()
            r = -torch.pow(((ag.double() - g.double()).abs() * w).sum(-1), torch.tensor(p, dtype=torch.float64, device=ag.device))
            return r.float(), r > -THR
    else:
        def f(ag, g):
            hit = {"bitflip": lambda: (ag == g).all(-1), "all_geq": lambda: (ag >= g).all(-1), "first_geq": lambda: ag[:, 0] >= g[:, 0]}[name]()
            return hit.float() - 1.0, hit
    return fdql.TorchReward(f)


# ---------------------------------------------------------------------------------------------- adversarial goal data
def episode_goals(rng, name, L, G):
    """(achieved_goal [L, G], desired_goal [G]) of one episode.  Goals on a small grid (ties common); the last row achieves the
    desired goal exactly (the pivot: hindsight goals drawn there compare every row with dg); other rows are near copies of it that
    differ in the last component, in a component of the upper lane group, by the sign of a zero, by one NaN or inf, in component 0
    only against all the others (first_geq), or revisit an earlier row."""
    pn = name.startswith("pnorm")
    grid = (lambda n: rng.integers(-4, 5, n) / 4) if pn else (lambda n: rng.integers(0, 2, n).astype(float)) if name == "bitflip" \
        else (lambda n: rng.integers(-1, 2, n).astype(float))
    dg = grid(G)
    dg[rng.random(G) < 0.3] = 0.0
    dg[rng.integers(0, G)] = 0.0
    ag = np.empty((L, G))
    step = 0.25 if pn else 1.0
    hc = hi_component(G)
    for t in range(L):
        a = dg.copy()
        kind = rng.integers(0, 11) if t < L - 1 else -1
        if kind == 0:
            a = grid(G)
        elif kind == 1:
            a[G - 1] += step * rng.choice([-1, 1])
        elif kind == 2:
            a[hc] += step * rng.choice([-1, 1])
        elif kind == 3:
            a[a == 0] = -0.0
        elif kind == 4:
            a[rng.integers(0, G)] = np.nan
        elif kind == 5:
            a[rng.integers(0, G)] = rng.choice([np.inf, -np.inf])
        elif kind == 6 and G > 1:  # component 0 says yes, every other component says no (and the reverse)
            if rng.random() < 0.5:
                a[0] += step
                a[1:] -= step
            else:
                a[0] -= step
                a[1:] += step
        elif kind in (7, 8) and t > 0:
            a = ag[rng.integers(0, t)].copy()
        elif kind == 9:
            a[rng.integers(0, G)] += step * rng.choice([-4, -2, -1, 1, 2, 4])
        elif kind == 10 and pn:  # the last component weighs 1: a norm of exactly 1, on the threshold
            a[G - 1] += rng.choice([-1.0, 1.0])
        ag[t] = a
    dgz = dg.copy()
    dgz[dgz == 0] = np.where(rng.random(int((dgz == 0).sum())) < 0.5, -0.0, 0.0)
    ag[L - 1] = dgz if rng.random() < 0.5 else dg
    return ag.astype(np.float32), dg.astype(np.float32)


def case_counts(name, ag, g):
    """Rows of `ag` (against goals `g`, same shape) where each adversarial case is the deciding one."""
    G = ag.shape[1]
    fin = np.isfinite(ag).all(1)
    eq = ag == g
    hc = hi_component(G)
    last_only = (eq[:, :-1].all(1) & ~eq[:, -1]) & fin
    m = np.ones(G, bool)
    m[hc] = False
    hi_only = eq[:, m].all(1) & ~eq[:, hc] & fin
    negzero = (eq.all(1) & (np.signbit(ag) != np.signbit(g)).any(1))
    out = {"tie": int(eq.all(1).sum()), "negzero": int(negzero.sum()), "last_only": int(last_only.sum()),
           "hi_only": int(hi_only.sum()), "nan": int(np.isnan(ag).any(1).sum()), "inf": int(np.isinf(ag).any(1).sum())}
    if name == "first_geq" and G > 1:
        out["first_decides"] = int(((ag[:, 0] >= g[:, 0]) != (ag[:, 1:] >= g[:, 1:]).all(1)).sum())
    if name.startswith("pnorm"):  # the threshold: rows on both sides of it and rows exactly on it (done is reward > -thr)
        r, _ = functor(name, G)[0](ag, g)
        out.update(done=int((r > -THR).sum()), not_done=int((r < -THR).sum()), on_threshold=int((r == -THR).sum()))
    return out


def revisits(ag, dg, episode_done):
    """Rows whose achieved_goal equals (==) an earlier row's of the same episode and differs from its desired_goal: the hits of the
    bitflip functor's chain of equal achieved goals that the desired goal does not also give."""
    ends = np.flatnonzero(episode_done.reshape(-1)) + 1
    n = 0
    for s, e in zip(np.concatenate([[0], ends[:-1]]), ends):
        a = ag[s:e]
        same = (a[:, None] == a[None]).all(-1)
        earlier = np.tril(same, -1).any(1)
        n += int((earlier & ~(a == dg[s:e]).all(1)).sum())
    return n


MIN_CASES = {"tie": 20, "negzero": 5, "last_only": 5, "hi_only": 5, "nan": 5, "inf": 5, "first_decides": 5, "done": 20,
             "not_done": 20, "on_threshold": 1, "revisit": 10, "goal_agnostic_offset": 20}


def assert_cases_reached(name, G, cols):
    """The generator must keep producing every adversarial case: a minimum count of rows where the case decides, per (functor, width)."""
    counts = case_counts(name, cols["achieved_goal"], cols["desired_goal"])
    counts["revisit"] = revisits(cols["achieved_goal"], cols["desired_goal"], cols["episode_done"])
    if name.startswith("pnorm"):  # rows whose stored reward is not R(ag, dg) itself: a relabel that drops r - R(ag, dg) shows
        Rd, _ = O.fp32_reward(functor(name, G)[0])(cols["achieved_goal"], cols["desired_goal"])
        counts["goal_agnostic_offset"] = int((cols["reward"].reshape(-1) != Rd).sum())
    low = {k: v for k, v in counts.items() if v < MIN_CASES[k]}
    assert not low, f"{name} G={G}: too few rows of the cases {low} (need {MIN_CASES})"
    return counts


def matrix_data(name, G, seed=0):
    """Columns (chronological) of the LENGTHS episodes, their extents, and a filler episode of FILL rows."""
    rng = np.random.default_rng(seed * 1000 + G * 10 + FUNCTORS.index(name))
    fn = functor(name, G)[0]
    ags, dgs = [], []
    for L in LENGTHS:
        a, d = episode_goals(rng, name, L, G)
        ags.append(a)
        dgs.append(np.repeat(d[None], L, 0))
    ag, dg = np.concatenate(ags), np.concatenate(dgs)
    N = len(ag)
    lengths = np.array(LENGTHS)
    ends = np.cumsum(lengths) - 1
    first = ends - lengths + 1
    ep_of = np.repeat(np.arange(len(lengths)), lengths)
    r, d = O.fp32_reward(fn)(ag, dg)
    if name.startswith("pnorm"):
        # the env's reward R(ag, dg) plus a goal-agnostic term k in {0, -1, -2}, where R + k is exact in fp32 (else k = 0): then every
        # relabelled reward k + R(ag, g*) has one rounding, on the device as in the oracle, and no cancellation (R <= 0, k <= 0)
        k = rng.integers(-2, 1, N).astype(np.float64)
        with np.errstate(invalid="ignore"):
            exact = np.float32(r + k).astype(np.float64) - r == k
        reward = np.where(exact, r + k, r).astype(np.float32)
    else:
        reward = rng.integers(-1, 1, N).astype(np.float32)  # goal-agnostic terms of -1, 0 and +1
    step = (np.arange(N) - first[ep_of]).astype(np.float32)
    cols = {"obs_1d": rng.standard_normal((N, 4)).astype(np.float32), "action": rng.uniform(-1, 1, (N, 4)).astype(np.float32),
            "achieved_goal": ag, "desired_goal": dg, "reward": reward.reshape(-1, 1),
            "task_done": np.asarray(d, np.float32).reshape(-1, 1),
            "episode_done": np.isin(np.arange(N), ends).astype(np.float32).reshape(-1, 1), "episode_step": step.reshape(-1, 1)}
    cols["mc_return"] = O.segmented_returns(cols["reward"], cols["episode_done"], GAMMA).reshape(-1, 1)
    fa, fd = episode_goals(rng, name, FILL, G)
    filler = {k: np.resize(v[:1], (FILL,) + v.shape[1:]).copy() for k, v in cols.items()}
    filler["achieved_goal"], filler["desired_goal"] = fa, np.repeat(fd[None], FILL, 0)
    filler["episode_done"][:] = 0
    filler["episode_done"][-1] = 1
    return cols, filler, first[ep_of], ends[ep_of], first, ends


def sentinel_returns(cols):
    return {k: (np.full_like(v, -1234.5) if k == "mc_return" else v) for k, v in cols.items()}


# ---------------------------------------------------------------------------------------------- comparisons
def npy(t):
    return t.detach().cpu().numpy()


def same_bits(got, want, what):
    """Bit for bit; any NaN equals any NaN."""
    a, b = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(want, np.float32)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    na, nb = np.isnan(a), np.isnan(b)
    np.testing.assert_array_equal(na, nb, err_msg=f"{what}: NaN positions")
    np.testing.assert_array_equal(np.where(na, 0, a.view(np.int32)), np.where(nb, 0, b.view(np.int32)), err_msg=what)


def same_values(got, want, what):
    """Equal values (+0 == -0); NaN equals NaN."""
    a, b = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    np.testing.assert_array_equal(a, b, err_msg=what)


def ulps(got, want):
    """fp32 ulp distance (+0 and -0 coincide; NaN against NaN is 0, NaN against a number is huge)."""
    def ordered(x):
        i = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    a, b = np.asarray(got, np.float32), np.asarray(want, np.float32)
    d = np.abs(ordered(a) - ordered(b))
    both = np.isnan(a) & np.isnan(b)
    one = np.isnan(a) ^ np.isnan(b)
    return np.where(both, 0, np.where(one, 1 << 40, d))


def check_reward(name, got, want, what):
    if name.startswith("pnorm"):
        d = ulps(got, want)
        assert d.max(initial=0) <= 1, f"{what}: {int((d > 1).sum())} rewards more than 1 ulp from the oracle (max {d.max()})"
    else:
        same_values(got, want, what)


def check_goal_agnostic(name, z, cols, fn32, what):
    """The scan record's r - R(ag, dg): exact for the flag functors; for the p-norm within one fp32 ulp of the R(ag, dg) it is formed
    from (the term is a small integer k, or 0, while R may be large: an ulp of R is the device's freedom, an ulp of k is not)."""
    Rd, _ = fn32(cols["achieved_goal"], cols["desired_goal"])
    with np.errstate(invalid="ignore"):
        ga = (cols["reward"].reshape(-1).astype(np.float64) - Rd).astype(np.float32)
    if not name.startswith("pnorm"):
        same_values(z, ga, what)
        return
    same_values(np.isnan(z), np.isnan(ga), f"{what}: NaN positions")
    fin = ~np.isnan(ga)
    with np.errstate(invalid="ignore"):
        err = np.abs(z[fin].astype(np.float64) - ga[fin])
    bound = np.spacing(np.abs(Rd[fin]).astype(np.float32)).astype(np.float64)
    assert (err <= bound).all(), f"{what}: {int((err > bound).sum())} terms further than 1 ulp of R(ag, dg) from the oracle"


def check_returns(got, want, exact, what):
    if exact:
        same_values(got, want, what)
    else:
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6, err_msg=what)


# ---------------------------------------------------------------------------------------------- route check
def launched_kernels(fn):
    """Names of the CUDA kernels `fn` launches (torch.profiler, CUDA activity); None when the profiler reports no kernel at all."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    names = [n for n in names if not n.startswith(("Memcpy", "Memset", "cudaMemcpy", "cudaMemset"))]
    return names or None


def assert_route(fn, pattern, what):
    names = launched_kernels(fn)
    if names is None:
        pytest.skip(f"{what}: the profiler reported no CUDA kernel, so the route cannot be asserted (the parity checks ran)")
    assert any(re.search(pattern, n) for n in names), f"{what}: expected a kernel matching {pattern!r}, launched {names}"


# ---------------------------------------------------------------------------------------------- the ring of one (functor, width)
class MatrixRing:
    def __init__(self, fdql, name, G):
        from fastdeepqlearning_b200 import Replay
        self.name, self.G = name, G
        self.fn = functor(name, G)[0]
        self.cols, filler, self.ep_start, self.ep_end, self.first, self.ends = matrix_data(name, G)
        self.N = len(self.cols["reward"])
        assert_cases_reached(name, G, self.cols)
        ring = Replay.ReplayMemory(CAP, 8, 2)
        ring.set_reward_op(reward_op(fdql, name, G), GAMMA)
        # mc_return is appended as a sentinel: the commit must write every return
        ring.add_rows(sentinel_returns(filler), episode_lengths=[FILL], with_returns=True)
        ring.add_rows(sentinel_returns(self.cols), episode_lengths=LENGTHS, with_returns=True)
        self.ring = ring
        assert len(ring) == CAP - 1 and ring._top == (FILL + self.N) % CAP
        phys = self.phys(np.arange(self.N))
        assert (np.diff(phys) < 0).any(), "no episode wraps the end of the ring"

    def phys(self, logical):
        return (FILL + np.asarray(logical)) % CAP


_RINGS = {}


@pytest.fixture(scope="module")
def rings(fdql):
    def get(name, G):
        if (name, G) not in _RINGS:
            _RINGS.clear()  # one ring at a time: tests run in grid order
            _RINGS[(name, G)] = MatrixRing(fdql, name, G)
        return _RINGS[(name, G)]
    yield get
    _RINGS.clear()


GRID = [(n, G) for n in FUNCTORS for G in WIDTHS]


# ---------------------------------------------------------------------------------------------- 1. commit + sample-time relabelling
def routes(name, G):
    """(debug switch, kernel name pattern) of every route the switch can force for this functor and width, at the small batches of
    the matrix.  There bit 3 (warp-per-window instead of the tile kernel) and the default route launch the same kernel: the tile kernel
    is only chosen unforced from 1024 windows with link records (or 49152 without); test_bitflip_routes_at_a_tile_sized_batch forces
    bits 3 and 4 where it would be."""
    lpr = lpr_of(G)
    generic = (1, rf"sample_gather_kernel<{lpr}, true>")
    if name != "bitflip":
        fast = rf"sample_gather_fast_kernel<\d, {lpr}, 1>"
        return [(0, fast), generic, (8, fast)]
    out = [(0, r"sample_gather_fast_kernel<\d, 1, [23]>"), generic, (8, r"sample_gather_fast_kernel<\d, 1, [23]>"),
           (2, rf"sample_gather_fast_kernel<\d, {lpr}, 1>"), (32 << 8, r"sample_gather_tile_kernel"),
           (256 << 8, r"sample_gather_tile_kernel"), ((256 << 8) | 16, r"sample_gather_tile_kernel")]
    if G % 4 == 0 and 2 * G // 4 + 2 <= 32:
        out.append((32, r"sample_gather_lean_kernel"))
    return out


def windows(mr, T, rng, B=160):
    """Logical window starts: across episode ends, at episode starts, across the ring's physical end, and at random."""
    N = mr.N
    wrap = CAP - FILL  # the logical row stored at physical row 0
    s = list(rng.integers(0, N - T + 1, B // 2))
    s += [int(e) - int(k) for e in mr.ends for k in rng.integers(0, T, 2)]
    s += [int(f) for f in mr.first]
    s += [wrap - int(k) for k in rng.integers(1, T + 1, 8)]
    s = np.clip(np.array(s), 0, N - T)
    return s


@pytest.mark.parametrize("name,G", GRID)
def test_sample_time_relabel_every_route(fdql, rings, name, G):
    mr = rings(name, G)
    lib = fdql.lib()
    fn32 = O.fp32_reward(mr.fn)
    # the goal-agnostic term r - R(ag, dg) of every committed row (scan record .z)
    z = npy(mr.ring._meta(2)).reshape(-1)[mr.phys(np.arange(mr.N))]
    check_goal_agnostic(name, z, mr.cols, fn32, "goal-agnostic term")
    stored = mr.ring.memory
    same_values(npy(stored["mc_return"])[mr.phys(np.arange(mr.N))], mr.cols["mc_return"], "committed mc_return")
    rng = np.random.default_rng(G)
    route_list = routes(name, G)
    for T in WINDOWS:
        mr.ring._temporal_len = T
        starts = windows(mr, T, rng)
        B = len(starts)
        flags = rng.random(B) < 0.8
        pick_last = rng.random(B) < 0.5
        goal_rows = np.where(pick_last, mr.ep_end[starts],
                             [rng.integers(s, mr.ep_end[s] + 1) for s in starts])
        check_relabel_windows(lib, mr, T, starts, flags, goal_rows, [switch for switch, _ in route_list])
    mr.ring._temporal_len = 2


def relabel_call(mr, T, starts, flags, goal_rows):
    return lambda: mr.ring.temporal_sample(starts=mr.phys(starts), flags=flags.astype(np.uint8), goal_rows=mr.phys(goal_rows),
                                           exact_episode_step=True, aux=T > 1, length=CAP)


def check_relabel_windows(lib, mr, T, starts, flags, goal_rows, switches, patterns=None):
    """Relabelled windows (logical starts / goal rows) against O.sample_time_relabel under each forced route; with `patterns`, each
    route must also have launched a kernel of its family."""
    name, G = mr.name, mr.G
    want = O.sample_time_relabel(mr.cols, starts, T, flags, goal_rows, mr.ep_start, mr.ep_end, O.fp32_reward(mr.fn), GAMMA)
    mask, contig = O.learner_preprocess(want["task_done"], want["episode_step"])
    for i, switch in enumerate(switches):
        what = f"{name} G={G} T={T} windows={len(starts)} switch={switch}"
        old = lib.fdql_debug_force_generic_gather(switch)
        try:
            got = {k: npy(v) for k, v in relabel_call(mr, T, starts, flags, goal_rows)().items()}
            if patterns is not None:
                assert_route(relabel_call(mr, T, starts, flags, goal_rows), patterns[i], what)
        finally:
            lib.fdql_debug_force_generic_gather(old)
        for k in mr.cols:
            if k == "reward":
                check_reward(name, got[k], want[k], f"{what}: {k}")
            elif k == "mc_return":
                np.testing.assert_allclose(got[k], want[k], rtol=1e-5, atol=1e-6, err_msg=f"{what}: {k}")
            else:
                same_bits(got[k], want[k], f"{what}: {k}")
        if T > 1:
            same_bits(got["mask"], mask.astype(np.float32), f"{what}: mask")
            same_bits(got["is_contiguous"], contig.astype(np.float32), f"{what}: is_contiguous")
            np.testing.assert_allclose(got["loss_weight"], O.upstream_weight(contig, T), rtol=1e-6, atol=1e-12,
                                       err_msg=f"{what}: loss_weight")


@pytest.mark.parametrize("G", [4, 33, 128])
def test_bitflip_routes_at_a_tile_sized_batch(fdql, rings, G):
    """From 1024 windows with link records (T <= 32) the unforced bitflip gather takes the tile kernel.  There bit 3 must take the
    warp-per-window kernel instead and bit 4 (no link records: the tile kernel only from 49152 windows) the warp-per-window kernel as
    well, each with the oracle's results."""
    mr = rings("bitflip", G)
    lib = fdql.lib()
    rng = np.random.default_rng(G + 3)
    fast = r"sample_gather_fast_kernel<\d, 1, [23]>"
    try:
        for T in (2, 5):
            mr.ring._temporal_len = T
            starts = windows(mr, T, rng, B=2400)
            assert len(starts) >= 1024
            flags = rng.random(len(starts)) < 0.8
            goal_rows = np.array([rng.integers(s, mr.ep_end[s] + 1) for s in starts])
            check_relabel_windows(lib, mr, T, starts, flags, goal_rows, [0, 8, 16], [r"sample_gather_tile_kernel", fast, fast])
    finally:
        mr.ring._temporal_len = 2


@pytest.mark.parametrize("name", FUNCTORS)
@pytest.mark.parametrize("G", [1, 5, 9, 17, 33, 128])  # LPR 1, 2, 4, 8, 16, 32
def test_forced_routes_launch_their_kernel(fdql, rings, name, G):
    """A forced route that fell through to another kernel would make its parity run worthless: each launches its own family."""
    mr = rings(name, G)
    lib = fdql.lib()
    T = 5
    mr.ring._temporal_len = T
    starts = np.arange(0, 320, 2)
    try:
        for switch, pattern in routes(name, G):
            old = lib.fdql_debug_force_generic_gather(switch)
            try:
                assert_route(lambda: mr.ring.temporal_sample(starts=mr.phys(starts), flags=np.ones(len(starts), np.uint8),
                                                             goal_rows=mr.phys(mr.ep_end[starts]), exact_episode_step=True, aux=True,
                                                             length=CAP), pattern, f"{name} G={G} switch={switch}")
            finally:
                lib.fdql_debug_force_generic_gather(old)
    finally:
        mr.ring._temporal_len = 2


# ---------------------------------------------------------------------------------------------- 2. write-time hindsight flush (+ 4. TorchReward)
def her_ring(fdql, name, G, reward, cols, filler, goal_rows_rel, first):
    from fastdeepqlearning_b200 import Replay
    ring = Replay.ReplayMemory(1024, 8, 2)
    ring.set_reward_op(reward, GAMMA)
    ring.add_rows(sentinel_returns({k: np.resize(v, (800,) + v.shape[1:]) for k, v in filler.items()}), episode_lengths=[800],
                  with_returns=True)
    begin = ring.add_rows(sentinel_returns(cols), episode_lengths=LENGTHS, with_returns=True)
    src = (begin + first) % 1024
    dst = npy(ring.add_hindsight_rows(src, LENGTHS, (src + goal_rows_rel) % 1024, with_returns=True))
    return ring, src, dst


@pytest.mark.parametrize("mode", ["final", "random"])
@pytest.mark.parametrize("name,G", GRID)
def test_write_time_flush_vs_oracle(fdql, name, G, mode):
    fn = functor(name, G)[0]
    fn32 = O.fp32_reward(fn)
    cols, filler, _, _, first, _ = matrix_data(name, G, seed=1)
    rng = np.random.default_rng(G + 7)
    rel = np.array([L - 1 if mode == "final" else rng.integers(0, L) for L in LENGTHS])
    filler["achieved_goal"] = np.resize(filler["achieved_goal"], (800, G))
    filler["desired_goal"] = np.resize(filler["desired_goal"], (800, G))
    ring, src, dst = her_ring(fdql, name, G, reward_op(fdql, name, G), cols, filler, rel, first)
    tring, _, tdst = her_ring(fdql, name, G, torch_reward(fdql, name, G), cols, filler, rel, first)
    assert (src[1:] < src[:-1]).any() or ((src + np.array(LENGTHS) - 1) >= 1024).any(), "no source episode wraps the ring's end"
    mem = {k: npy(v) for k, v in ring.memory.items()}
    tmem = {k: npy(v) for k, v in tring.memory.items()}
    np.testing.assert_array_equal(dst, tdst)
    ga_z = npy(ring._meta(2)).reshape(-1)
    all_exact = True
    for e, L in enumerate(LENGTHS):
        sl = slice(first[e], first[e] + L)
        rows_d = (dst[e] + np.arange(L)) % 1024
        goal = cols["achieved_goal"][first[e] + rel[e]]
        nr, nd, ns = O.her_relabel_episode(cols["achieved_goal"][sl], cols["desired_goal"][sl], cols["reward"][sl].reshape(-1),
                                           cols["episode_step"][sl].reshape(-1), goal, fn32)
        what = f"{name} G={G} {mode} episode of {L}"
        for k in ("obs_1d", "action", "achieved_goal", "episode_done"):
            same_bits(mem[k][rows_d], cols[k][sl], f"{what}: {k}")
        same_bits(mem["desired_goal"][rows_d], np.repeat(goal[None], L, 0), f"{what}: desired_goal")
        same_values(mem["task_done"][rows_d].reshape(-1), nd.astype(np.float32), f"{what}: task_done")
        same_values(mem["episode_step"][rows_d].reshape(-1), ns, f"{what}: episode_step")
        got_r = mem["reward"][rows_d].reshape(-1)
        check_reward(name, got_r, nr, f"{what}: reward")
        exact = np.array_equal(got_r, nr, equal_nan=True)
        all_exact &= exact
        check_returns(mem["mc_return"][rows_d].reshape(-1), O.mc_return_chrono(got_r if exact else nr, GAMMA), exact, f"{what}: mc_return")
        check_goal_agnostic(name, ga_z[rows_d], {k: v[sl] for k, v in cols.items()}, fn32, f"{what}: goal-agnostic term")
    # the TorchReward path stores the rows the enum path stores
    for k in mem:
        same_bits(tmem[k], mem[k], f"{name} G={G} {mode} TorchReward: {k}")
    if not name.startswith("pnorm"):
        assert all_exact


# ---------------------------------------------------------------------------------------------- 3. vmap fill and select (+ 4. TorchReward)
def vmap_ring(fdql, reward, cols, filler, first, picks_rel, with_ret, quirk, G):
    from fastdeepqlearning_b200 import Replay
    ring = Replay.ReplayMemory(CAP, 8, 5)
    ring.set_reward_op(reward, GAMMA)

    def with_virtual(c):
        n = len(c["reward"])
        d = {k: v for k, v in c.items() if k != "mc_return"}
        d["virtual_goals"] = np.zeros((n, (V + 1) * G), np.float32)
        d["virtual_rewards"] = np.zeros((n, V + 1), np.float32)
        d["virtual_dones"] = np.zeros((n, V + 1), np.float32)
        if with_ret:
            d["virtual_mc_return"] = np.zeros((n, V + 1), np.float32)
        return d
    ring.add_rows(with_virtual(filler), episode_lengths=[FILL])
    begin = ring.add_rows(with_virtual(cols), episode_lengths=LENGTHS)
    src = (begin + first) % CAP
    picks = ((src[:, None] + picks_rel) % CAP).reshape(-1)
    ring.vmap_flush(src, LENGTHS, pick_rows=picks, fill=True, returns=with_ret, done_quirk=quirk)
    return ring, begin


@pytest.mark.parametrize("returns", ["none", "quirk", "sane"])
@pytest.mark.parametrize("name,G", GRID)
def test_vmap_fill_and_select_vs_oracle(fdql, name, G, returns):
    fn = functor(name, G)[0]
    with_ret, quirk = returns != "none", returns == "quirk"
    cols, filler, _, _, first, ends = matrix_data(name, G, seed=2)
    rng = np.random.default_rng(G + 11)
    picks_rel = np.stack([np.concatenate([[L - 1], rng.integers(0, L, V - 1)]) for L in LENGTHS])
    ring, begin = vmap_ring(fdql, reward_op(fdql, name, G), cols, filler, first, picks_rel, with_ret, quirk, G)
    tring, _ = vmap_ring(fdql, torch_reward(fdql, name, G), cols, filler, first, picks_rel, with_ret, quirk, G)
    N = len(cols["reward"])
    phys = (begin + np.arange(N)) % CAP
    assert (np.diff(phys) < 0).any()
    mem = {k: npy(v) for k, v in ring.memory.items()}
    want = {k: [] for k in ("virtual_goals", "virtual_rewards", "virtual_dones", "virtual_mc_return")}
    for e, L in enumerate(LENGTHS):
        sl = slice(first[e], first[e] + L)
        o = O.vmap_write_episode({k: v[sl] for k, v in cols.items()}, picks_rel[e], fn, GAMMA if with_ret else None, quirk)
        for k in want:
            if k in o:
                want[k].append(o[k])
    what = f"{name} G={G} returns={returns}"
    same_bits(mem["virtual_goals"][phys], np.concatenate(want["virtual_goals"]).reshape(N, -1), f"{what}: virtual_goals")
    same_values(mem["virtual_dones"][phys], np.concatenate(want["virtual_dones"]).astype(np.float32), f"{what}: virtual_dones")
    vr = np.concatenate(want["virtual_rewards"])
    check_reward(name, mem["virtual_rewards"][phys], vr, f"{what}: virtual_rewards")
    exact = np.array_equal(mem["virtual_rewards"][phys], vr, equal_nan=True)
    if not name.startswith("pnorm"):
        assert exact
    if with_ret:
        got_ret = mem["virtual_mc_return"][phys]
        if exact:
            same_values(got_ret, np.concatenate(want["virtual_mc_return"]), f"{what}: virtual_mc_return")
        else:
            np.testing.assert_allclose(got_ret, np.concatenate(want["virtual_mc_return"]), rtol=1e-5, atol=1e-6)
    for k, v in tring.memory.items():
        same_bits(npy(v), mem[k], f"{what} TorchReward: {k}")
    # the read head: one column of the stored virtual keys per window
    T = 5
    starts = np.clip(np.concatenate([rng.integers(0, N - T + 1, 40), ends - 2, [CAP - FILL - 2]]), 0, N - T)
    stored = {k: v[phys] for k, v in mem.items()}
    idx = np.arange(T)[:, None] + starts[None]
    batch = {k: v[idx] for k, v in stored.items()}
    batch["virtual_goals"] = batch["virtual_goals"].reshape(T, len(starts), V + 1, G)
    for column in (0, V - 1, V):
        got = {k: npy(x) for k, x in ring.vmap_temporal_sample(column, starts=phys[starts], aux=True, length=CAP).items()}
        sel = O.vmap_read_select(batch, column)
        for k in ("desired_goal", "reward", "task_done", "episode_step", "achieved_goal"):
            same_bits(got[k], sel[k], f"{what} column {column}: {k}")
        if with_ret:
            same_bits(got["mc_return"], sel["mc_return"], f"{what} column {column}: mc_return")
        mask, contig = O.learner_preprocess(sel["task_done"], sel["episode_step"])
        same_bits(got["mask"], mask.astype(np.float32), f"{what} column {column}: mask")
        same_bits(got["is_contiguous"], contig.astype(np.float32), f"{what} column {column}: is_contiguous")


# ---------------------------------------------------------------------------------------------- 5. drawing entry points, non-bitflip functors
@pytest.mark.parametrize("name", ["all_geq", "pnorm0.5"])
@pytest.mark.parametrize("G", [5, 33, 128])
def test_drawing_gather_falls_back_to_the_same_batch(fdql, rings, name, G):
    """fdql_sample_gather_draw serves the bitflip functor only; with another functor it falls back to fdql_sample_streams +
    fdql_sample_gather, which must give the batch and streams of those two calls made explicitly with the same seed and counter."""
    mr = rings(name, G)
    ring = mr.ring
    for T, n in ((2, 4096), (5, 300)):
        ring._temporal_len = T
        try:
            c0 = ring._rng_counter
            got = {k: npy(v) for k, v in ring.temporal_sample(n=n, relabel_prob=0.8, exact_episode_step=True, aux=True).items()}
            streams = [npy(s) for s in ring.last_streams]
            ring._rng_counter = c0
            st, fl, go = ring.draw_streams(n, T, relabel_prob=0.8)
            for a, b in zip(streams, (st, fl, go)):
                np.testing.assert_array_equal(a, npy(b))
            want = {k: npy(v) for k, v in ring.temporal_sample(starts=st, flags=fl, goal_rows=go, exact_episode_step=True, aux=True).items()}
            assert set(got) == set(want)
            for k in want:
                same_bits(got[k], want[k], f"{name} G={G} T={T}: {k}")
            assert streams[1].any()
        finally:
            ring._temporal_len = 2


def _streams_batch_buffers(ring, T, n):
    import torch
    from fastdeepqlearning_b200 import _lib as L
    out = {k: torch.full((T, n, w), -7.0, device="cuda") for k, w in zip(ring._keys, ring._widths)}
    return {"out": out, "outp": L.ptr_array([out[k].data_ptr() for k in ring._keys]), "mask": torch.empty(T, n, device="cuda"),
            "contig": torch.empty(T - 1, n, device="cuda"), "weight": torch.empty(T - 1, n, device="cuda"),
            "st": torch.empty(n, dtype=torch.int64, device="cuda"), "fl": torch.empty(n, dtype=torch.uint8, device="cuda"),
            "go": torch.empty(n, dtype=torch.int64, device="cuda")}


@pytest.mark.parametrize("name", ["all_geq", "pnorm0.5"])
@pytest.mark.parametrize("G", [5, 128])
def test_fused_pass_falls_back_to_the_same_launches(fdql, rings, name, G):
    """fdql_fused_pass fuses the loss with the gather role only for the bitflip functor; with another functor it runs streams, gather
    and loss as launches of their own.  Two calls (the gather of batch 0 alone, then the loss of batch 0 with the gather of batch 1)
    against explicit fdql_sample_streams + fdql_sample_gather + fdql_tqc_loss on the same seed and counters: the same streams, batches,
    loss and gradient, bit for bit."""
    import torch
    from fastdeepqlearning_b200 import _lib as L
    ring = rings(name, G).ring
    lib = fdql.lib()
    T, n, n_atoms, n_drop = 2, 4096, 125, 10
    M = (T - 1) * n
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    params, n_params = ring.reward_op.c_params()
    opts = L.OPT_EMIT_LEARNER_AUX | L.OPT_EXACT_EPISODE_STEP
    gen = torch.Generator(device="cuda").manual_seed(G)
    z, q = torch.randn(M, n_atoms, device="cuda", generator=gen) * 3, torch.randn(M, n_atoms, device="cuda", generator=gen) * 3
    lp = torch.randn(M, device="cuda", generator=gen)

    def loss_bufs():
        return torch.empty(M, device="cuda"), torch.empty(M, n_atoms, device="cuda"), torch.zeros(4, dtype=torch.float64, device="cuda")

    def g_half(b, ctr):
        return (ring._h, n, T, L.GOAL_FUTURE, 0.8, 11, ctr, None, p(b["st"]), p(b["fl"]), p(b["go"]), ring.reward_op.op, params, n_params,
                GAMMA, opts, 4096, b["outp"], p(b["mask"]), p(b["contig"]), p(b["weight"]))

    def t_half(b, m, loss, grad, stats):
        return (m, n_atoms, n_drop, p(z), p(q), p(lp), p(b["out"]["reward"][1:]), p(b["mask"][1:]), p(b["out"]["mc_return"][1:]),
                p(b["weight"]), 0.2, 0.99, p(loss), p(grad), p(stats))
    ref = [_streams_batch_buffers(ring, T, n) for _ in range(2)]
    for k, b in enumerate(ref):
        L.check(lib.fdql_sample_streams(ring._h, n, T, L.GOAL_FUTURE, 0.8, 11, k, None, p(b["st"]), p(b["fl"]), p(b["go"]), sp))
        L.check(lib.fdql_sample_gather(ring._h, n, T, len(ring), p(b["st"]), p(b["fl"]), p(b["go"]), ring.reward_op.op, params, n_params,
                                       GAMMA, opts, 4096, b["outp"], p(b["mask"]), p(b["contig"]), p(b["weight"]), sp))
    rl, rg, rs = loss_bufs()
    a = t_half(ref[0], M, rl, rg, rs)
    L.check(lib.fdql_tqc_loss(*a[:14], None, a[14], sp))
    got = [_streams_batch_buffers(ring, T, n) for _ in range(2)]
    fl_, fg, fs = loss_bufs()
    dummy = torch.empty(1, device="cuda")
    L.check(lib.fdql_fused_pass(*g_half(got[0], 0), *t_half(got[0], 0, dummy, dummy, None), sp))
    L.check(lib.fdql_fused_pass(*g_half(got[1], 1), *t_half(got[0], M, fl_, fg, fs), sp))
    torch.cuda.synchronize()
    for k, (a_, b_) in enumerate(zip(ref, got)):
        for key in ("st", "fl", "go"):
            np.testing.assert_array_equal(npy(b_[key]), npy(a_[key]), err_msg=f"{name} G={G} batch {k}: {key}")
        for key in ("mask", "contig", "weight"):
            same_bits(npy(b_[key]), npy(a_[key]), f"{name} G={G} batch {k}: {key}")
        for key in a_["out"]:
            same_bits(npy(b_["out"][key]), npy(a_["out"][key]), f"{name} G={G} batch {k}: {key}")
        assert npy(a_["fl"]).any() and not npy(a_["fl"]).all()
    same_bits(npy(fl_), npy(rl), f"{name} G={G}: loss")
    same_bits(npy(fg), npy(rg), f"{name} G={G}: grad")
    np.testing.assert_allclose(npy(fs), npy(rs), rtol=1e-12)
    assert np.isfinite(npy(rl)).any()


@pytest.mark.parametrize("name", ["all_geq", "pnorm1"])
def test_fused_per_pass_falls_back_to_the_same_launches(fdql, name):
    """fdql_fused_pass_per draws from the priority tree inside the fused kernel only for the bitflip functor; with another functor it
    runs fdql_per_sample, the gather, the critic weights, the loss and the priority update as launches of their own.  Three calls
    against that chain made explicitly: streams, importance weights, batches, loss, gradient and every tree level, bit for bit."""
    import torch
    from fastdeepqlearning_b200 import Replay, _lib as L
    from test_gpu_per_fused import Pass, same_bits as same_tensor_bits
    G = 33

    class MatrixPass(Pass):
        def __init__(self):  # Pass's buffers and launch sequences on a ring of the matrix data, committed with this functor
            self.torch, self.L, self.lib = torch, L, fdql.lib()
            cols, filler = matrix_data(name, G)[:2]
            self.ring = Replay.ReplayMemory(CAP, 8, 2)
            self.ring.set_reward_op(reward_op(fdql, name, G), GAMMA)
            self.ring.enable_priorities(alpha=0.6, eps=1e-3, eta=0.9)
            self.ring.add_rows(sentinel_returns(filler), episode_lengths=[FILL], with_returns=True)
            self.ring.add_rows(sentinel_returns(cols), episode_lengths=LENGTHS, with_returns=True)
            self.ring.set_priority_beta(0.7)
            self.counter_dev, self.xi, self.weights = None, None, True
            self.n, self.T, self.n_atoms, self.n_drop, self.with_lb, self.with_stats = 4096, 2, 125, 10, True, True
            gen = torch.Generator(device="cuda").manual_seed(3)
            self.z = torch.randn(self.n, 125, device="cuda", generator=gen) * 3
            self.q = torch.randn(self.n, 125, device="cuda", generator=gen) * 3
            self.lp = torch.randn(self.n, device="cuda", generator=gen)
            self.bufs, self.losses = {}, {}
            self.opts = L.OPT_EMIT_LEARNER_AUX | L.OPT_EXACT_EPISODE_STEP
    fu, se = MatrixPass(), MatrixPass()
    passes = 3  # batch 2 draws from the tree batch 0's update changed
    for k in range(passes):
        fu.fused(k)
        se.separate(k)
        torch.cuda.synchronize()
        for a, b in zip(fu.tree(), se.tree()):
            assert same_tensor_bits(a, b), k
    for k in range(passes):
        a, b = fu.buf(k), se.buf(k)
        for key in ("st", "fl", "go", "isw", "critic", "mask", "contig", "weight"):
            assert same_tensor_bits(a[key], b[key]), (k, key)
        for key in a["out"]:
            assert same_tensor_bits(a["out"][key], b["out"][key]), (k, key)
        assert npy(a["fl"]).any() and (npy(a["isw"]) > 0).all()
    for k in range(passes - 1):
        (l1, g1, s1), (l2, g2, s2) = fu.losses[k], se.losses[k]
        assert same_tensor_bits(l1, l2) and same_tensor_bits(g1, g2), k
        np.testing.assert_allclose(npy(s1), npy(s2), rtol=1e-12)


# ---------------------------------------------------------------------------------------------- 6. refusals
def _raw_arena(lib, G, with_reward=True):
    import torch
    from fastdeepqlearning_b200 import _lib as L
    widths = [G, G, 1, 1, 1]
    roles = [L.ROLE_ACHIEVED_GOAL, L.ROLE_DESIRED_GOAL, L.ROLE_REWARD, L.ROLE_TASK_DONE, L.ROLE_EPISODE_STEP]
    h = C.c_void_p()
    L.check(lib.fdql_arena_create(64, 5, (C.c_int32 * 5)(*widths), (C.c_int32 * 5)(*roles), 0, C.byref(h)))
    src = [torch.zeros((8, w), device="cuda") for w in widths]
    L.check(lib.fdql_arena_append(h, 8, L.ptr_array([t.data_ptr() for t in src]), None))
    return h, src


def test_goals_wider_than_128_floats_are_refused(fdql):
    import torch
    from fastdeepqlearning_b200 import Replay, _lib as L
    lib = fdql.lib()
    msg = b"goal wider than 128 floats is not supported"
    h, keep = _raw_arena(lib, 129)
    try:
        dev = lambda v, dt: torch.tensor(v, dtype=dt, device="cuda")
        p = lambda t: C.c_void_p(t.data_ptr())
        begin, lens, dst, goal = dev([0], torch.int64), dev([8], torch.int32), dev([8], torch.int64), dev([3], torch.int64)
        pn, n_pn = L.f32_array([0.5, 1.0] + [1.0] * 129)
        for op, params, n_params in ((L.REWARD_NONE, None, 0), (L.REWARD_ALL_GEQ, None, 0), (L.REWARD_WEIGHTED_PNORM, pn, n_pn)):
            assert lib.fdql_commit_episodes(h, 1, p(begin), p(lens), GAMMA, 1, op, params, n_params, None) == L.FDQL_EINVAL
            assert msg in lib.fdql_last_error(), lib.fdql_last_error()
        for op, params, n_params in ((L.REWARD_BITFLIP, None, 0), (L.REWARD_WEIGHTED_PNORM, pn, n_pn)):
            assert lib.fdql_her_flush_episodes(h, 1, p(begin), p(lens), p(dst), p(goal), op, params, n_params, GAMMA, 1, None) \
                == L.FDQL_EINVAL
            assert msg in lib.fdql_last_error()
        r, d = torch.zeros(8, device="cuda"), torch.zeros(8, dtype=torch.uint8, device="cuda")
        assert lib.fdql_her_flush_episodes_given(h, 1, p(begin), p(lens), p(dst), p(goal), 8, p(r), p(d), p(r), GAMMA, 1, None) \
            == L.FDQL_EINVAL
        assert msg in lib.fdql_last_error()
        T, n = 2, 4
        outs = [torch.empty((T, n, w), device="cuda") for w in (129, 129, 1, 1, 1)]
        st, fl, go = dev([0, 1, 2, 3], torch.int64), dev([1, 1, 0, 1], torch.uint8), dev([5, 5, 5, 5], torch.int64)
        for op, params, n_params in ((L.REWARD_FIRST_GEQ, None, 0), (L.REWARD_WEIGHTED_PNORM, pn, n_pn)):
            assert lib.fdql_sample_gather(h, n, T, 8, p(st), p(fl), p(go), op, params, n_params, GAMMA, 0, n,
                                          L.ptr_array([t.data_ptr() for t in outs]), None, None, None, None) == L.FDQL_EINVAL
            assert msg in lib.fdql_last_error()
        torch.cuda.synchronize()
    finally:
        lib.fdql_arena_destroy(h)
    # the Python layer refuses at the first write and stores nothing
    for write in ("add_rows", "add"):
        ring = Replay.ReplayMemory(64, 8, 2)
        ring.set_reward_op(fdql.RewardOp.all_geq())
        cols = {"achieved_goal": np.zeros((4, 129), np.float32), "desired_goal": np.zeros((4, 129), np.float32),
                "reward": np.zeros((4, 1), np.float32), "episode_done": np.array([[0], [0], [0], [1]], np.float32)}
        with pytest.raises(ValueError, match="goal wider than 128 floats is not supported"):
            if write == "add_rows":
                ring.add_rows(cols, episode_lengths=[4])
            else:
                ring.add({k: v[0] if v.shape[1] > 1 else float(v[0, 0]) for k, v in cols.items()})
        assert len(ring) == 0 and ring._h is None
    # a desired_goal that no achieved_goal is compared with is stored and committed at any width
    ring = Replay.ReplayMemory(64, 8, 2)
    ring.add_rows({"desired_goal": np.ones((4, 200), np.float32), "reward": np.zeros((4, 1), np.float32)}, episode_lengths=[4])
    assert len(ring) == 4 and float(ring.memory["desired_goal"][3, 199]) == 1.0


def test_pnorm_parameter_count_must_match_the_goal_width(fdql):
    from fastdeepqlearning_b200 import Replay
    for n_w in (7, 9):
        ring = Replay.ReplayMemory(64, 8, 2)
        ring.set_reward_op(fdql.RewardOp.weighted_pnorm([1.0] * n_w, 0.5, 1.0))
        cols = {"achieved_goal": np.zeros((4, 8), np.float32), "desired_goal": np.zeros((4, 8), np.float32),
                "reward": np.zeros((4, 1), np.float32)}
        with pytest.raises(ValueError, match=f"needs 10 params .* got {n_w + 2}"):
            ring.add_rows(cols, episode_lengths=[4])
