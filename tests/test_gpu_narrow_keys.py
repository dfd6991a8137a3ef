"""GPU checks of narrow (uint8 / int8) keys.  Twin arenas: the same rows go into an all-fp32 ring and into a ring whose obs (and in
some cases action) key is stored narrow, with values spanning the whole type; every entry point must then give bit-identical outputs
from both -- every key, the aux, the drawn streams, the loss and the gradient -- and the narrow ring must hold the exact integers."""
import ctypes as C
import random
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
G = 16


def npy(t):
    return t.detach().cpu().numpy()


def _ints(rng, shape, dt):
    lo, hi = (0, 255) if dt == "uint8" else (-128, 127)
    x = rng.integers(lo, hi + 1, shape)
    x.reshape(-1)[:2] = (lo, hi)  # both ends of the type
    return x


class Twin:
    """Ring `f` stores every key as fp32, ring `n` stores `narrow` ({key: "uint8" | "int8"}) at one byte per element."""

    def __init__(self, fdql, narrow, obs=64, act=8, n_eps=120, ep_len=None, max_len=90, cap=None, T=2, batch=16, seed=0, per=False,
                 device_rows=False):
        import torch
        from fastdeepqlearning_b200 import Replay
        from test_gpu_replay import _synthetic
        self.torch, self.fdql = torch, fdql
        rng = np.random.default_rng(seed)
        cols, lengths, starts_ep, ends, ep_of = _synthetic(rng, n_eps, max_len, G, obs=obs, act=act, fixed_len=ep_len)
        for k, dt in narrow.items():
            cols[k] = _ints(rng, cols[k].shape, dt).astype(np.float32)
        self.cols, self.lengths, self.starts_ep, self.ends, self.ep_of = cols, lengths, starts_ep, ends, ep_of
        self.N = int(lengths.sum())
        self.narrow = narrow
        cap = cap or self.N + 1
        self.f = Replay.ReplayMemory(cap, batch, T)
        self.n = Replay.ReplayMemory(cap, batch, T, key_dtypes={k: getattr(torch, dt) for k, dt in narrow.items()})
        for r in (self.f, self.n):
            r.set_reward_op(fdql.RewardOp.bitflip(), 0.98)
            if per:
                r.enable_priorities(alpha=0.6, eps=1e-3, eta=0.9)
        self.f.add_rows(cols, episode_lengths=lengths, with_returns=True)
        # the narrow ring gets the storage type: numpy on the host, or device tensors
        ncols = {k: (v.astype(narrow[k]) if k in narrow else v) for k, v in cols.items()}
        if device_rows:
            ncols = {k: torch.as_tensor(v).cuda() for k, v in ncols.items()}
        self.n.add_rows(ncols, episode_lengths=lengths, with_returns=True)

    def assert_same(self, a, b, keys=None):
        torch = self.torch
        for k in keys or a:
            assert a[k].dtype == torch.float32 and b[k].dtype == torch.float32, k
            assert torch.equal(a[k], b[k]), k

    def assert_memory(self):
        """the narrow slabs hold the exact integers, and read back as the fp32 ring's values"""
        torch = self.torch
        mf, mn = self.f.memory, self.n.memory
        for k in mf:
            if k in self.narrow:
                assert mn[k].dtype == getattr(torch, self.narrow[k])
                assert torch.equal(mn[k].float(), mf[k]), k
            else:
                assert torch.equal(mn[k], mf[k]), k


NARROW_CASES = [({"obs_1d": "uint8"}, 3), ({"obs_1d": "int8"}, 16), ({"obs_1d": "uint8", "action": "int8"}, 17),
                ({"obs_1d": "int8", "action": "uint8"}, 64), ({"obs_1d": "uint8"}, 28224)]


@pytest.mark.parametrize("narrow,obs", NARROW_CASES)
@pytest.mark.parametrize("T", [1, 2, 5])
def test_sample_gather_injected_streams(fdql, narrow, obs, T):
    """fdql_sample_gather with injected streams (starts over the whole ring, so windows wrap at len), relabel flags and aux;
    and fdql_gather_rows through memory[idx]"""
    tw = Twin(fdql, narrow, obs=obs, n_eps=40 if obs > 1000 else 120, T=T)
    tw.assert_memory()
    rng = np.random.default_rng(obs + T)
    N, B = tw.N, 600
    starts = rng.integers(0, N, B)
    flags = (rng.random(B) < 0.7).astype(np.uint8)
    goal_rows = np.array([rng.integers(s, tw.ends[tw.ep_of[s]] + 1) for s in starts])
    for kw in (dict(), dict(flags=flags, goal_rows=goal_rows, exact_episode_step=True)):
        a = tw.f.temporal_sample(starts=starts, length=N, aux=T > 1, **kw)
        b = tw.n.temporal_sample(starts=starts, length=N, aux=T > 1, **kw)
        tw.assert_same(a, b)
        for k, dt in narrow.items():  # window row t of window b is ring row (s_b + t) mod len, as the reference's
            rows = (starts[None, :] + np.arange(T)[:, None]) % N
            np.testing.assert_array_equal(npy(b[k]), tw.cols[k][rows].astype(np.float32))
    idx = rng.integers(0, tw.N, 333)
    tw.assert_same(tw.f[idx], tw.n[idx])


@pytest.mark.parametrize("narrow,obs", NARROW_CASES[:4])
def test_sample_gather_draw(fdql, narrow, obs):
    """fdql_sample_gather_draw: fused-draw shapes (tile kernel) and the two-launch fallback; same streams, same batch.  The narrow ring
    is filled by add_rows from device tensors."""
    tw = Twin(fdql, narrow, obs=obs, n_eps=600, ep_len=64, T=2, device_rows=True)
    for n, T in ((300, 2), (60000, 2), (500, 50)):
        tw.f._temporal_len = tw.n._temporal_len = T
        for r in (tw.f, tw.n):
            r._rng_counter = 3
        a = tw.f.temporal_sample(n=n, relabel_prob=0.8, aux=True)
        sa = [x.clone() if x is not None else None for x in tw.f.last_streams]
        b = tw.n.temporal_sample(n=n, relabel_prob=0.8, aux=True)
        for x, y in zip(sa, tw.n.last_streams):
            assert (x is None) == (y is None) and (x is None or torch_equal(x, y))
        tw.assert_same(a, b)


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class Batches:
    """The buffers of a sequence of fused passes on one ring (see tests/test_gpu_r2.py::test_fused_pass_equals_the_two_launches)."""

    def __init__(self, ring, n, T, n_atoms):
        import torch
        from fastdeepqlearning_b200 import _lib as L
        self.torch, self.L, self.ring, self.n, self.T, self.n_atoms = torch, L, ring, n, T, n_atoms
        M = max(T - 1, 1) * n
        gen = torch.Generator(device="cuda").manual_seed(n)
        self.z = torch.randn(M, n_atoms, device="cuda", generator=gen) * 3
        self.q = torch.randn(M, n_atoms, device="cuda", generator=gen) * 3
        self.lp = torch.randn(M, device="cuda", generator=gen)
        self.bufs = []

    def buf(self):
        torch, n, T = self.torch, self.n, self.T
        out = {k: torch.full((T, n, w), -7.0, device="cuda") for k, w in zip(self.ring._keys, self.ring._widths)}
        b = {"out": out, "outp": self.L.ptr_array([out[k].data_ptr() for k in self.ring._keys]), "mask": torch.full((T, n), -7.0, device="cuda"),
             "contig": torch.full((max(T - 1, 1), n), -7.0, device="cuda"), "weight": torch.full((max(T - 1, 1), n), -7.0, device="cuda"),
             "st": torch.empty(n, dtype=torch.int64, device="cuda"), "fl": torch.empty(n, dtype=torch.uint8, device="cuda"),
             "go": torch.empty(n, dtype=torch.int64, device="cuda"), "isw": torch.full((n,), -7.0, device="cuda"),
             "critic": torch.full((max(T - 1, 1), n), -7.0, device="cuda")}
        self.bufs.append(b)
        return b

    def g_half(self, b, ctr):
        params, n_params = self.ring.reward_op.c_params()
        return (self.n, self.T, self.L.GOAL_FUTURE, 0.8, 11, ctr, None, _ptr(b["st"]), _ptr(b["fl"]), _ptr(b["go"]), self.ring.reward_op.op,
                params, n_params, 0.99, self.L.OPT_EMIT_LEARNER_AUX | self.L.OPT_EXACT_EPISODE_STEP, 4096, b["outp"], _ptr(b["mask"]),
                _ptr(b["contig"]), _ptr(b["weight"]))

    def t_half(self, b, m, loss, grad, stats):
        return (m, self.n_atoms, 10, _ptr(self.z), _ptr(self.q), _ptr(self.lp), _ptr(b["out"]["reward"][1:]), _ptr(b["mask"][1:]),
                _ptr(b["out"]["mc_return"][1:]), _ptr(b["weight"]), 0.2, 0.99, _ptr(loss), _ptr(grad), _ptr(stats))

    def loss_bufs(self):
        torch, M = self.torch, (self.T - 1) * self.n
        return (torch.full((max(M, 1),), -7.0, device="cuda"), torch.full((max(M, 1), self.n_atoms), -7.0, device="cuda"),
                torch.zeros(4, dtype=torch.float64, device="cuda"))


def _same_batches(xa, xb):
    import torch
    for a, b in zip(xa.bufs, xb.bufs):
        for k in ("st", "fl", "go", "mask", "contig", "weight", "isw", "critic"):
            assert torch.equal(a[k], b[k]), k
        for k in a["out"]:
            assert torch.equal(a["out"][k], b["out"][k]), k


@pytest.mark.parametrize("n,T", [(24576, 2), (3000, 2), (6001, 5), (1024, 50), (4096, 1)])
@pytest.mark.parametrize("narrow", [{"obs_1d": "uint8"}, {"obs_1d": "int8", "action": "int8"}])
def test_fused_pass(fdql, n, T, narrow):
    """fdql_fused_pass over three passes (the fused kernel at 24576 x 2, 6001 x 5 and 1024 x 50; the separate launches at 3000 windows;
    the gather alone at T = 1): streams, batches, loss and gradient bit-identical to the fp32 twin's"""
    import torch
    tw = Twin(fdql, narrow, obs=64, n_eps=600, ep_len=64, T=T)
    lib = fdql.lib()
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    for ring in (tw.f, tw.n):
        x = Batches(ring, n, T, 125)
        losses = []
        dummy = torch.empty(1, device="cuda")
        b = x.buf()
        fdql._lib.check(lib.fdql_fused_pass(ring._h, *x.g_half(b, 0), *x.t_half(b, 0, dummy, dummy, None), sp))
        for k in range(2):
            prev, b = b, x.buf()
            loss, grad, stats = x.loss_bufs()
            M = (T - 1) * n
            fdql._lib.check(lib.fdql_fused_pass(ring._h, *x.g_half(b, k + 1), *x.t_half(prev, M, loss, grad, stats), sp))
            losses.append((loss, grad, stats))
        torch.cuda.synchronize()
        res.append((x, losses))
    _same_batches(res[0][0], res[1][0])
    for (la, ga, sa), (lb, gb, sb) in zip(res[0][1], res[1][1]):
        assert torch.equal(la, lb) and torch.equal(ga, gb)
        np.testing.assert_allclose(npy(sa), npy(sb), rtol=1e-12)  # (summaries: fp64 sums in atomic order)


@pytest.mark.parametrize("n", [24576, 3000])
def test_fused_pass_per(fdql, n):
    """fdql_fused_pass_per over four passes (fused at 24576 windows, the separate prioritized chain at 3000): streams, importance and
    critic weights, batches, loss, gradient and every tree level bit-identical to the fp32 twin's"""
    import torch
    T = 2
    tw = Twin(fdql, {"obs_1d": "uint8", "action": "int8"}, obs=64, n_eps=600, ep_len=64, T=T, per=True)
    lib = fdql.lib()
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    for ring in (tw.f, tw.n):
        ring.set_priority_beta(0.7)
        x = Batches(ring, n, T, 125)
        losses = []
        prev = None
        for k in range(4):
            b = x.buf()
            loss, grad, stats = x.loss_bufs()
            M = (T - 1) * n if prev is not None else 0
            g = x.g_half(b, k)
            t = x.t_half(prev if prev is not None else b, M, loss, grad, stats)
            fdql._lib.check(lib.fdql_fused_pass_per(
                ring._per, n, g[2], g[3], g[4], g[5], None, None, _ptr(ring._per_beta), g[7], g[8], g[9], _ptr(b["isw"]),
                _ptr(b["critic"]), *g[10:], *t[:9], _ptr(prev["critic"]) if prev is not None else None, *t[10:],
                _ptr(prev["st"]) if prev is not None else None, _ptr(prev["contig"]) if prev is not None else None, sp))
            if M:
                losses.append((loss, grad, stats))
            prev = b
        torch.cuda.synchronize()
        res.append((x, losses, [(s.clone(), m.clone()) for s, m in ring.priority_tree()], ring.priority_views()[0].clone()))
    _same_batches(res[0][0], res[1][0])
    for (la, ga, sa), (lb, gb, sb) in zip(res[0][1], res[1][1]):
        assert torch.equal(la, lb) and torch.equal(ga, gb)
        np.testing.assert_allclose(npy(sa), npy(sb), rtol=1e-12)  # (summaries: fp64 sums in atomic order)
    assert torch.equal(res[0][3], res[1][3])
    for (sa, ma), (sb, mb) in zip(res[0][2], res[1][2]):
        assert torch.equal(sa, sb) and torch.equal(ma, mb)


@pytest.mark.parametrize("n", [3000, 20000])
def test_hotpath_step_host(fdql, n):
    """fdql_hotpath_step_host (host streams and critic outputs, sliced above 4096 windows): batch, loss and gradient"""
    import torch
    T, n_atoms = 2, 125
    tw = Twin(fdql, {"obs_1d": "uint8"}, obs=64, n_eps=600, ep_len=64, T=T)
    rng = np.random.default_rng(n)
    starts = rng.integers(0, tw.N - T, n).astype(np.int64)
    flags = (rng.random(n) < 0.8).astype(np.uint8)
    goals = np.array([rng.integers(s, tw.ends[tw.ep_of[s]] + 1) for s in starts], dtype=np.int64)
    M = (T - 1) * n
    z = rng.standard_normal((M, n_atoms)).astype(np.float32)
    q = rng.standard_normal((M, n_atoms)).astype(np.float32)
    lp = rng.standard_normal(M).astype(np.float32)
    hp = lambda a: a.ctypes.data_as(C.c_void_p)
    res = []
    for ring in (tw.f, tw.n):
        out = {k: torch.full((T, n, w), -7.0, device="cuda") for k, w in zip(ring._keys, ring._widths)}
        loss, grad = np.zeros(M, np.float32), np.zeros((M, n_atoms), np.float32)
        params, n_params = ring.reward_op.c_params()
        fdql._lib.check(fdql.lib().fdql_hotpath_step_host(
            ring._h, n, T, tw.N, hp(starts), hp(flags), hp(goals), ring.reward_op.op, params, n_params, 0.98, 0,
            fdql._lib.ptr_array([out[k].data_ptr() for k in ring._keys]), n_atoms, 10, hp(z), hp(q), hp(lp), 0.2, hp(loss), hp(grad),
            C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        res.append((out, loss, grad))
    tw.assert_same(res[0][0], res[1][0])
    np.testing.assert_array_equal(res[0][1], res[1][1])
    np.testing.assert_array_equal(res[0][2], res[1][2])


def _ring(head):
    while hasattr(head, "replay_buffer"):
        head = head.replay_buffer
    return head.replay


def _bitflip_torch(ag, g):
    import torch
    done = (ag == g).all(dim=-1)
    return done.to(torch.float32) - 1.0, done


@pytest.mark.parametrize("mode", ["final", "random"])
@pytest.mark.parametrize("torch_reward", [False, True])
@pytest.mark.parametrize("narrow,obs", [({"obs_1d": "uint8"}, 17), ({"obs_1d": "int8", "action": "uint8"}, 64)])
def test_write_time_her_and_q3_through_make_heads(fdql, mode, torch_reward, narrow, obs):
    """rows added one dict at a time through Replay.make write heads (NStepReturn -> HER final / random, n_step 3 so that quirk Q3
    duplicates rows): the hindsight copies and the duplicates carry the narrow keys; a wrapping ring; then a sample of every row"""
    import torch
    from fastdeepqlearning_b200 import Replay
    rng = np.random.default_rng(obs)
    heads = []
    for dts in ({}, narrow):
        conf = types.SimpleNamespace(replay_size=600, batch_size=8, temporal_len=2, num_instances=1, use_nStep_lowerbounds=True,
                                     nStep_return_steps=3, gamma=0.98, use_squashed_rewards=False, use_HER=True, her_mode=mode,
                                     training_device="cuda:0", replay_key_dtypes={k: getattr(np, dt) for k, dt in dts.items()} or None)
        op = fdql.TorchReward(_bitflip_torch) if torch_reward else fdql.RewardOp.bitflip()
        heads.append(Replay.make(conf, compute_reward=op)[1][0])
    random.seed(7)  # the "random" mode's goal picks come from Python's generator (her.py): the same picks for both heads
    state = random.getstate()
    rows = []
    for ep in range(40):
        L = int(rng.integers(1, 30))
        dg = rng.integers(0, 2, G).astype(np.float32)
        for t in range(L):
            ag = rng.integers(0, 2, G).astype(np.float32)
            r = 0.0 if (ag == dg).all() else -1.0
            xp = {"obs_1d": _ints(rng, (obs,), narrow["obs_1d"]), "action": _ints(rng, (3,), narrow.get("action", "uint8")),
                  "achieved_goal": ag, "desired_goal": dg, "reward": r, "task_done": r == 0.0, "episode_done": t == L - 1,
                  "episode_step": t}
            rows.append(xp)
    for h in heads:
        random.setstate(state)
        for xp in rows:
            h.add({k: (v.astype(np.float32) if k in narrow and h is heads[0] else v) for k, v in xp.items()})
        _ring(h).flush()
    f, nr = [_ring(h) for h in heads]
    assert len(f) == len(nr) and f._top == nr._top and len(f) == f._maxlen - 1  # the ring wrapped
    torch.cuda.synchronize()
    mf, mn = f.memory, nr.memory
    for k in mf:
        assert torch.equal(mn[k].float() if k in narrow else mn[k], mf[k]), k
    starts = np.arange(0, len(f) - 2)
    a = f.temporal_sample(starts=starts, length=len(f), aux=True)
    b = nr.temporal_sample(starts=starts, length=len(f), aux=True)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_q3_duplicate_and_state_dict_round_trip(fdql):
    """fdql_q3_duplicate copies the narrow row; a snapshot carries the storage types and restores the ring bit for bit (a snapshot of
    an all-fp32 ring carries none and restores as fp32)"""
    import torch
    from fastdeepqlearning_b200 import Replay
    tw = Twin(fdql, {"obs_1d": "uint8", "action": "int8"}, obs=28224, n_eps=12, max_len=30, cap=400)
    for r in (tw.f, tw.n):
        dst = r.reserve_rows(1)
        r.q3_duplicate(5, 3, dst, 0.98)
    tw.assert_memory()
    assert torch.equal(tw.n.memory["obs_1d"][dst], tw.n.memory["obs_1d"][5])
    sd, sdf = tw.n.state_dict(), tw.f.state_dict()
    assert sd["dtypes"] == {"obs_1d": "uint8", "action": "int8"} and "dtypes" not in sdf
    assert sd["memory"]["obs_1d"].dtype == torch.uint8
    r2 = Replay.ReplayMemory(400, 16, 2)
    r2.load_state_dict(sd)
    assert r2.key_dtypes["obs_1d"] == torch.uint8 and r2.key_dtypes["action"] == torch.int8
    for k, v in tw.n.memory.items():
        assert torch.equal(r2.memory[k], v), k
    rf = Replay.ReplayMemory(400, 16, 2)
    rf.load_state_dict(sdf)
    assert all(dt == torch.float32 for dt in rf.key_dtypes.values())
    starts = np.arange(0, len(tw.n) - 2)
    a, b = tw.f.temporal_sample(starts=starts, aux=True), r2.temporal_sample(starts=starts, aux=True)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_info_bytes_and_narrow_view(fdql):
    import torch
    tw = Twin(fdql, {"obs_1d": "uint8"}, obs=28224, n_eps=10, max_len=20, cap=256)
    lib = fdql.lib()
    info = []
    for r in (tw.f, tw.n):
        b = C.c_int64()
        fdql._lib.check(lib.fdql_arena_info(r._h, None, None, None, C.byref(b)))
        info.append(b.value)
    assert info[0] - info[1] == 256 * (28224 * 4 - 28224)
    base, stride, dt = C.c_void_p(), C.c_int64(), C.c_int32()
    fdql._lib.check(lib.fdql_arena_narrow_view(tw.n._h, tw.n._keys.index("obs_1d"), C.byref(base), C.byref(stride), C.byref(dt)))
    assert stride.value == 28224 and dt.value == fdql._lib.DTYPE_U8
    assert torch.equal(tw.n.memory["obs_1d"][:tw.N].float(), torch.as_tensor(tw.cols["obs_1d"]).cuda())


def test_add_rows_from_device_and_out_of_range_values(fdql):
    """add_rows from device tensors (float and integer) and one-dict add; values the type does not hold raise and stage nothing"""
    import torch
    from fastdeepqlearning_b200 import Replay
    r = Replay.ReplayMemory(64, 4, 2, key_dtypes={"obs": torch.uint8, "s": np.int8})
    x = torch.tensor([[0.0, 255.0, 7.0]], device="cuda")
    r.add_rows({"obs": x, "s": torch.tensor([[-128, 127]], device="cuda"), "reward": torch.zeros(1, 1, device="cuda")})
    for bad in (256.0, -1.0, 0.5, float("nan")):
        with pytest.raises(ValueError):
            r.add_rows({"obs": torch.tensor([[bad, 0.0, 0.0]], device="cuda"), "s": torch.zeros(1, 2, device="cuda"),
                        "reward": torch.zeros(1, 1, device="cuda")})
        with pytest.raises(ValueError):
            r.add({"obs": np.array([bad, 0.0, 0.0]), "s": np.zeros(2), "reward": 0.0})
    with pytest.raises(ValueError):
        r.add({"obs": np.zeros(3), "s": np.array([-129, 0]), "reward": 0.0})
    r.add({"obs": np.array([1, 2, 3], np.uint8), "s": np.array([-5, 5]), "reward": 1.0})
    assert len(r) == 2
    m = r.memory
    assert m["obs"][:2].tolist() == [[0, 255, 7], [1, 2, 3]] and m["s"][:2].tolist() == [[-128, 127], [-5, 5]]
    assert m["s"].dtype == torch.int8
    got = r[np.array([0, 1])]
    assert got["obs"].dtype == torch.float32 and got["obs"].tolist() == [[0.0, 255.0, 7.0], [1.0, 2.0, 3.0]]
    assert got["s"].tolist() == [[-128.0, 127.0], [-5.0, 5.0]]


def test_refusals(fdql):
    """each refusal of the C ABI and of the Python mirror raises its documented error"""
    import torch
    from fastdeepqlearning_b200 import Replay, _lib as L
    lib = fdql.lib()
    h = C.c_void_p()
    arr = lambda *v: (C.c_int32 * len(v))(*v)
    # a narrow dtype on a width-1 key, on a key with a role; an unknown dtype
    for widths, roles, dtypes, msg in (((1, 4), (0, 0), (1, 0), b"width"), ((4, 4), (L.ROLE_ACHIEVED_GOAL, L.ROLE_DESIRED_GOAL), (1, 0), b"role"),
                                       ((4, 4), (0, 0), (3, 0), b"unknown dtype")):
        assert lib.fdql_arena_create_typed(16, 2, arr(*widths), arr(*roles), arr(*dtypes), 0, C.byref(h)) == L.FDQL_EINVAL
        assert msg in lib.fdql_last_error()
    r = Replay.ReplayMemory(64, 4, 2, key_dtypes={"obs": torch.uint8})
    r.add_rows({"obs": np.zeros((3, 5), np.uint8), "act": np.zeros((3, 2), np.float32), "reward": np.zeros((3, 1), np.float32)})
    base, stride, col = C.c_void_p(), C.c_int64(), C.c_int32()
    assert lib.fdql_arena_key_view(r._h, 0, C.byref(base), C.byref(stride), C.byref(col)) == L.FDQL_EINVAL
    assert b"fdql_arena_narrow_view" in lib.fdql_last_error()
    dt = C.c_int32()
    assert lib.fdql_arena_narrow_view(r._h, 1, C.byref(base), C.byref(stride), C.byref(dt)) == L.FDQL_EINVAL
    # the vmap entry points refuse a narrow virtual key
    hv = C.c_void_p()
    widths, roles = arr(2, 2, 2, 2, 1, 1), arr(L.ROLE_ACHIEVED_GOAL, L.ROLE_DESIRED_GOAL, 0, 0, L.ROLE_REWARD, L.ROLE_TASK_DONE)
    L.check(lib.fdql_arena_create_typed(16, 6, widths, roles, arr(0, 0, 0, 1, 0, 0), 0, C.byref(hv)))
    try:
        starts = torch.zeros(1, dtype=torch.int64, device="cuda")
        assert lib.fdql_vmap_select_column(hv, 1, 1, 4, C.c_void_p(starts.data_ptr()), 0, 0, 2, 3, -1, 1, None, None, None, None, None,
                                           None, None, None) == L.FDQL_EINVAL
        assert b"uint8 / int8" in lib.fdql_last_error()
        assert lib.fdql_vmap_flush_episodes(hv, 1, C.c_void_p(starts.data_ptr()), C.c_void_p(starts.data_ptr()), None, 0, 2, 3, -1, 1,
                                            None, 0, 0.9, 2, 0, None) == L.FDQL_EINVAL
        assert b"uint8 / int8" in lib.fdql_last_error()
        assert lib.fdql_vmap_flush_episodes_given(hv, 1, C.c_void_p(starts.data_ptr()), C.c_void_p(starts.data_ptr()),
                                                  C.c_void_p(starts.data_ptr()), 0, 2, 3, -1, 1, C.c_void_p(starts.data_ptr()),
                                                  C.c_void_p(starts.data_ptr()), 0.9, 1, 0, None) == L.FDQL_EINVAL
        assert b"uint8 / int8" in lib.fdql_last_error()
    finally:
        lib.fdql_arena_destroy(hv)
    # the mirror: unknown key, role / scalar key, vmap virtual key, other dtypes -- before any row is stored
    for kd, cols in (({"nope": torch.uint8}, None), ({"reward": torch.uint8}, None), ({"achieved_goal": torch.uint8}, None),
                     ({"virtual_rewards": torch.uint8}, {"virtual_rewards": np.zeros((2, 3), np.float32)}),
                     ({"obs": torch.float16}, None), ({"obs": np.int16}, None)):
        r = Replay.ReplayMemory(64, 4, 2, key_dtypes=kd)
        base_cols = {"obs": np.zeros((2, 5), np.float32), "achieved_goal": np.zeros((2, 4), np.float32),
                     "desired_goal": np.zeros((2, 4), np.float32), "reward": np.zeros((2, 1), np.float32)}
        with pytest.raises(ValueError):
            r.add_rows({**base_cols, **(cols or {})})
        assert r._h is None


def test_captured_learner_step_equals_eager_on_a_narrow_ring(fdql):
    """A graphed learner over a ring whose obs is uint8: the captured step is the eager step (as for an fp32 ring), and the eager
    narrow learner takes the same update as the eager fp32 twin"""
    import torch
    from fastdeepqlearning_b200 import Agent, Replay
    from test_gpu_agent import make_conf
    rng = np.random.default_rng(0)
    Lep, n_eps = 32, 400
    N = Lep * n_eps
    ag = rng.integers(0, 2, (N, 16)).astype(np.float32)
    dg = np.repeat(rng.integers(0, 2, (n_eps, 16)).astype(np.float32), Lep, 0)
    hit = (ag == dg).all(-1, keepdims=True).astype(np.float32)
    step = (np.arange(N) % Lep).astype(np.float32).reshape(-1, 1)
    cols = {"obs_1d": rng.integers(0, 256, (N, 64)).astype(np.float32), "action": rng.uniform(-1, 1, (N, 8)).astype(np.float32),
            "achieved_goal": ag, "desired_goal": dg, "reward": hit - 1, "task_done": hit,
            "episode_done": (step == Lep - 1).astype(np.float32), "episode_step": step}

    def build(graph, narrow):
        torch.manual_seed(0)
        conf = make_conf(Agent, replay_size=N + 1, use_HER=True, her_mode="future", num_instances=1, temporal_len=2, batch_size=512,
                         use_cuda_graph=graph, replay_key_dtypes={"obs_1d": torch.uint8} if narrow else None)
        read, write = Replay.make(conf, compute_reward=fdql.RewardOp.bitflip())
        write[0].add_rows(cols, episode_lengths=[Lep] * n_eps)
        assert write[0].replay.key_dtypes["obs_1d"] == (torch.uint8 if narrow else torch.float32)
        return Agent.Learner(conf, read)

    lg = build(True, True)
    lg.train_step()  # three eager warm-up updates and one replay
    le = build(False, True)
    for _ in range(4):
        le.train_step()
    lf = build(False, False)
    for _ in range(4):
        lf.train_step()
    for (n1, p1), (n2, p2), (n3, p3) in zip(lg.actor_critic.state_dict().items(), le.actor_critic.state_dict().items(),
                                            lf.actor_critic.state_dict().items()):
        assert n1 == n2 == n3
        torch.testing.assert_close(p1, p2, rtol=1e-5, atol=1e-6, msg=lambda m, n1=n1: f"{n1}: {m}")
        torch.testing.assert_close(p2, p3, rtol=1e-5, atol=1e-6, msg=lambda m, n1=n1: f"{n1}: {m}")
