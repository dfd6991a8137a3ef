"""GPU checks of prioritized replay (fdql_per_*): the eligibility invariant through every writer, the incremental tree against a full
rebuild bit for bit, descent and importance weights against oracle/per.py, Philox-drawn frequencies, the update rule, hindsight streams
of prioritized starts, and the learner (alpha = 0 equals the uniform update; captured step equals eager step)."""
import types

import numpy as np
import pytest

from oracle import per as P

pytestmark = pytest.mark.gpu
G = 8


def episodes(rng, n_eps, Lep):
    N = n_eps * Lep
    ag = rng.integers(0, 2, (N, G)).astype(np.float32)
    dg = np.repeat(rng.integers(0, 2, (n_eps, G)).astype(np.float32), Lep, 0)
    hit = (ag == dg).all(-1, keepdims=True).astype(np.float32)
    step = (np.arange(N) % Lep).astype(np.float32).reshape(-1, 1)
    return {"obs_1d": rng.standard_normal((N, 12)).astype(np.float32), "action": rng.uniform(-1, 1, (N, 4)).astype(np.float32),
            "achieved_goal": ag, "desired_goal": dg, "reward": hit - 1, "task_done": hit,
            "episode_done": (step == Lep - 1).astype(np.float32), "episode_step": step}


def make_ring(fdql, cap, B, T, **per):
    from fastdeepqlearning_b200 import Replay
    ring = Replay.ReplayMemory(cap, B, T, device="cuda:0")
    ring.set_reward_op(fdql.RewardOp.bitflip(), 0.98)
    ring.enable_priorities(**per)
    return ring


def tree_snapshot(ring):
    leaves, qmax = ring.priority_views()
    return [leaves.clone(), qmax.clone()] + [t.clone() for lv in ring.priority_tree() for t in lv]


def assert_invariant_and_rebuild_equal(torch, ring):
    ring.apply_pending_priorities()
    leaves, _ = ring.priority_views()
    T = ring._temporal_len
    elig = torch.as_tensor(P.eligible(ring._maxlen, len(ring), T), device="cuda:0")
    assert torch.equal(leaves > 0, elig), "q[r] > 0 iff r < len - T"
    before = tree_snapshot(ring)
    ring.rebuild_priorities()
    after = tree_snapshot(ring)
    for a, b in zip(before, after):
        assert torch.equal(a.view(torch.int32 if a.dtype == torch.float32 else torch.int64),
                           b.view(torch.int32 if b.dtype == torch.float32 else torch.int64))
    # and the levels equal the numpy restatement of the same layout
    want = P.build(leaves.cpu().numpy())
    for (s, m), (ws, wm) in zip(ring.priority_tree(), want):
        np.testing.assert_array_equal(s.cpu().numpy(), ws)
        np.testing.assert_array_equal(m.cpu().numpy(), wm)


def random_update(torch, ring, rng, n):
    T = ring._temporal_len
    starts, _, _, _ = ring.draw_prioritized(n)
    loss = torch.as_tensor(rng.exponential(1.0, (T - 1, n)).astype(np.float32), device="cuda:0")
    ring.update_priorities(starts, loss)


def test_invariant_through_every_writer_and_tree_equals_rebuild(fdql):
    import torch
    rng = np.random.default_rng(0)
    T, cap = 5, 3000
    ring = make_ring(fdql, cap, 64, T)
    for _ in range(3):  # fills in several flushes, with updates in between
        ring.add_rows(episodes(rng, 10, 32), episode_lengths=[32] * 10)
        random_update(torch, ring, rng, 64)
        assert_invariant_and_rebuild_equal(torch, ring)
    for _ in range(5):  # staged single-row adds
        for r in [{k: v[i] for k, v in episodes(rng, 1, 4).items()} for i in range(4)]:
            ring.add({k: (v if v.size > 1 else float(v[0])) for k, v in r.items()})
    assert_invariant_and_rebuild_equal(torch, ring)
    src = ring.add_rows(episodes(rng, 20, 32), episode_lengths=[32] * 20)
    ring.add_hindsight_rows([src, src + 32], [32, 32], [src + 31, src + 63])  # reserve + write-time hindsight copy
    random_update(torch, ring, rng, 128)
    assert_invariant_and_rebuild_equal(torch, ring)
    for _ in range(4):  # wrap the ring more than once
        ring.add_rows(episodes(rng, 30, 32), episode_lengths=[32] * 30)
        random_update(torch, ring, rng, 256)
    assert len(ring) == cap - 1
    assert_invariant_and_rebuild_equal(torch, ring)
    # restore: the priorities come back bit for bit, the tree equals a rebuild, sampling with the same xi gives the same windows
    sd = ring.state_dict()
    from fastdeepqlearning_b200 import Replay
    ring2 = Replay.ReplayMemory(cap, 64, T, device="cuda:0")
    ring2.load_state_dict(sd)
    for a, b in zip(tree_snapshot(ring), tree_snapshot(ring2)):
        assert torch.equal(a, b)
    assert_invariant_and_rebuild_equal(torch, ring2)
    xi = torch.rand(64, dtype=torch.float64, device="cuda:0")
    s1 = ring.draw_prioritized(64, beta=0.7, xi=xi)
    s2 = ring2.draw_prioritized(64, beta=0.7, xi=xi)
    assert torch.equal(s1[0], s2[0]) and torch.equal(s1[3], s2[3])
    # set_cursor (the restore path) shrinking the ring moves the eligible range down
    ring2._lib.fdql_arena_set_cursor(ring2._h, 100, 1000)
    ring2._top, ring2._curr_len = 100, 1000
    assert_invariant_and_rebuild_equal(torch, ring2)


def set_leaves(torch, ring, q):
    leaves, _ = ring.priority_views()
    leaves.copy_(torch.as_tensor(q, device="cuda:0"))
    ring.rebuild_priorities()


def test_starts_and_weights_from_injected_xi_match_the_oracle(fdql):
    import torch
    rng = np.random.default_rng(1)
    T, cap, n = 2, 50000, 4096
    ring = make_ring(fdql, cap, n, T)
    ring.add_rows(episodes(rng, 1400, 32), episode_lengths=[32] * 1400)
    ring.apply_pending_priorities()
    n_elig = len(ring) - T
    q = np.zeros(cap, np.float32)
    q[:n_elig] = np.ldexp(1.0, rng.integers(-10, 6, n_elig)).astype(np.float32)  # dyadic: every fp64 sum exact in any order
    q[0] = np.float32(2.0 ** -11)                                                 # the unique minimum, drawn by xi_0 = 0
    set_leaves(torch, ring, q)
    xi = rng.random(n)
    xi[0] = 0.0
    starts, _, _, w = ring.draw_prioritized(n, beta=0.6, xi=torch.as_tensor(xi, device="cuda:0"))
    want_s, want_w = P.sample(q, xi, 0.6)
    np.testing.assert_array_equal(starts.cpu().numpy(), want_s)
    np.testing.assert_allclose(w.cpu().numpy(), want_w, rtol=1e-6)
    assert int(starts[0]) == 0 and float(w[0]) == 1.0 and float(w.max()) == 1.0
    # random fp32 priorities: a mismatch only where the target lies within 1e-9 S of a boundary
    q[:n_elig] = rng.uniform(0.01, 10, n_elig).astype(np.float32)
    set_leaves(torch, ring, q)
    starts, _, _, w = ring.draw_prioritized(n, beta=0.6, xi=torch.as_tensor(xi, device="cuda:0"))
    got = starts.cpu().numpy()
    cum = np.cumsum(q.astype(np.float64))
    t = P.targets(P.build(q), xi)
    want = np.searchsorted(cum, t, side="right")
    bad = np.nonzero(got != want)[0]
    S = cum[-1]
    for b in bad:
        edge = cum[min(got[b], want[b])]
        assert abs(t[b] - edge) <= 1e-9 * S, (b, got[b], want[b])
    assert (q[got] > 0).all()
    np.testing.assert_allclose(w.cpu().numpy(), (q[q > 0].min() / q[got].astype(np.float64)) ** np.float64(np.float32(0.6)), rtol=1e-6)


def test_philox_draws_follow_the_priorities_chi_square(fdql):
    import torch
    from scipy import stats
    rng = np.random.default_rng(2)
    T, cap, n = 2, 400, 1024
    ring = make_ring(fdql, cap, n, T)
    ring.add_rows(episodes(rng, 8, 32), episode_lengths=[32] * 8)  # 256 rows
    ring.apply_pending_priorities()
    n_elig = len(ring) - T
    q = np.zeros(cap, np.float32)
    q[:n_elig] = rng.uniform(0.1, 4.0, n_elig).astype(np.float32)
    set_leaves(torch, ring, q)
    counts = np.zeros(cap, np.int64)
    for _ in range(200):
        s, _, _, _ = ring.draw_prioritized(n)
        counts += np.bincount(s.cpu().numpy(), minlength=cap)
    q64 = q[:n_elig].astype(np.float64)
    expected = q64 / q64.sum() * counts.sum()
    assert counts[n_elig:].sum() == 0
    _, p = stats.chisquare(counts[:n_elig], expected)
    assert p > 1e-4, p


def test_no_ineligible_start_while_the_ring_fills_under_a_captured_graph(fdql):
    import torch
    rng = np.random.default_rng(3)
    T, cap, n = 5, 20000, 2048
    ring = make_ring(fdql, cap, n, T)
    ring.add_rows(episodes(rng, 70, 32), episode_lengths=[32] * 70)
    ring.device_counter = True
    ring.apply_pending_priorities()
    out = {}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out["w"] = ring.draw_prioritized(n)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out["g"] = ring.draw_prioritized(n)
    seen = 0
    for step in range(40):
        ring.add_rows(episodes(rng, 10, 32), episode_lengths=[32] * 10)  # 12.8 k rows more over the loop
        ring.apply_pending_priorities()
        g.replay()
        st = out["g"][0].cpu().numpy()
        assert (st < len(ring) - T).all() and (st >= 0).all(), step
        seen = max(seen, int(st.max()))
    assert seen > 10000
    assert int(ring._rng_counter_dev[0]) >= 41


@pytest.mark.parametrize("T", [2, 5])
def test_update_rule_matches_the_oracle(fdql, T):
    import torch
    rng = np.random.default_rng(4)
    cap, n = 5000, 3000
    ring = make_ring(fdql, cap, n, T, alpha=0.7, eps=1e-3, eta=0.9)
    ring.add_rows(episodes(rng, 100, 32), episode_lengths=[32] * 100)
    ring.apply_pending_priorities()
    leaves, qmax = ring.priority_views()
    n_elig = len(ring) - T
    starts = rng.integers(0, n_elig + 40, n)          # duplicates, and a few starts past the eligible range
    loss = rng.exponential(2.0, (T - 1, n)).astype(np.float32)
    loss[:, 5] = np.nan
    loss[0, 7] = np.inf
    contig = (rng.random((T - 1, n)) < 0.8).astype(np.float32)
    contig[:, 9] = 0
    before = leaves.cpu().numpy()
    want, want_max = P.update(before, float(qmax), starts, loss, contig, 0.7, 1e-3, 0.9)
    ring.update_priorities(torch.as_tensor(starts, device="cuda:0"), torch.as_tensor(loss, device="cuda:0"),
                           torch.as_tensor(contig, device="cuda:0"))
    np.testing.assert_array_equal(leaves.cpu().numpy(), want)
    assert float(qmax) == want_max
    assert_invariant_and_rebuild_equal(torch, ring)
    # a non-finite loss after q_max grew writes the new q_max; contig=None counts every transition
    loss2 = np.full((T - 1, 2), 50.0, np.float32)
    loss2[0, 1] = np.nan
    want, want_max = P.update(leaves.cpu().numpy(), float(qmax), [3, 4], loss2, None, 0.7, 1e-3, 0.9)
    ring.update_priorities(torch.as_tensor([3, 4], device="cuda:0"), torch.as_tensor(loss2, device="cuda:0"))
    np.testing.assert_array_equal(leaves.cpu().numpy(), want)
    assert float(qmax) == want_max


def test_hindsight_streams_of_prioritized_starts_follow_the_uniform_rules(fdql):
    import torch
    rng = np.random.default_rng(5)
    T, cap, n, Lep = 2, 10000, 4096, 32
    ring = make_ring(fdql, cap, n, T)
    ring.add_rows(episodes(rng, 200, Lep), episode_lengths=[Lep] * 200)
    ring.add_rows({k: v[:50] for k, v in episodes(rng, 2, Lep).items()})  # an open (uncommitted) episode at the head
    es, ee = [t.cpu().numpy() for t in ring.episode_extents()]
    for mode in (0, 1, 2):
        s, f, g, _ = ring.draw_prioritized(n, goal_mode=mode, relabel_prob=0.8)
        s, f, g = s.cpu().numpy(), f.cpu().numpy().astype(bool), g.cpu().numpy()
        committed = es[s] >= 0
        assert not f[~committed].any() and (g[~f] == s[~f]).all()
        assert abs(f[committed].mean() - 0.8) < 0.03
        e0, e1 = es[s[f]], ee[s[f]]
        if mode == 0:
            assert (g[f] == e1).all()
        elif mode == 1:
            assert ((g[f] >= e0) & (g[f] <= e1)).all()
        else:
            assert (((g[f] > s[f]) & (g[f] <= e1)) | ((s[f] == e1) & (g[f] == e1))).all()
    # the flag comes from the same Philox word as the uniform sampler's: with the same counter both give the same flag wherever both
    # starts are committed rows
    ring._rng_counter = 77
    s1, f1, _, _ = ring.draw_prioritized(n, relabel_prob=0.5)
    ring._rng_counter = 77
    s2, f2, _ = ring.draw_streams(n, relabel_prob=0.5)
    s1, s2, f1, f2 = s1.cpu().numpy(), s2.cpu().numpy(), f1.cpu().numpy(), f2.cpu().numpy()
    both = (es[s1] >= 0) & (es[s2] >= 0)
    assert both.mean() > 0.9 and (f1[both] == f2[both]).all()


def learner_conf(Agent, **kw):
    d = dict(training_device="cuda:0", obs_space={"obs_1d": 12, "achieved_goal": G, "desired_goal": G},
             action_space=types.SimpleNamespace(shape=(4,)), num_critics=3, num_q_predictions=25, top_quantiles_to_drop=0.08,
             batch_size=512, temporal_len=2, pi_hidden_dims=(32,), critic_hidden_dims=(32, 32), replay_size=20000, use_HER=True,
             her_mode="future", num_instances=1)
    d.update(kw)
    return Agent.LearnerConf(**d)


def test_learner_alpha_zero_equals_the_uniform_update_bit_for_bit(fdql):
    import torch
    from fastdeepqlearning_b200 import Agent, Replay
    rng = np.random.default_rng(6)
    conf_p = learner_conf(Agent, use_prioritized_replay=True, per_alpha=0.0)
    read, write = Replay.make(conf_p, compute_reward=fdql.RewardOp.bitflip())
    write[0].add_rows(episodes(rng, 300, 32), episode_lengths=[32] * 300)
    torch.manual_seed(0)
    lp = Agent.Learner(conf_p, read)
    torch.manual_seed(0)
    lu = Agent.Learner(learner_conf(Agent), read)
    ring = lp._ring_of(read[0])
    ring.set_priority_beta(lp.per_beta())
    xi = torch.rand(512, dtype=torch.float64, device="cuda:0")
    torch.manual_seed(1)
    lp.optimizer.zero_grad(set_to_none=False)
    loss_p = lp._one_update(read[0], xi=xi)
    starts, flags, goals = ring.last_streams
    leaves, _ = ring.priority_views()
    assert bool((leaves[leaves > 0] == 1).all())  # alpha = 0: every written leaf is 1, so every weight is exactly 1
    torch.manual_seed(1)
    lu.optimizer.zero_grad(set_to_none=False)
    loss_u = lu._one_update(read[0], starts=starts.clone(), flags=flags.clone(), goal_rows=goals.clone())
    assert torch.equal(loss_p, loss_u)
    for a, b in zip(lp.params, lu.params):
        assert torch.equal(a, b)


def test_captured_prioritized_step_equals_the_eager_step(fdql):
    import torch
    from fastdeepqlearning_b200 import Agent, Replay
    rng = np.random.default_rng(7)
    cols = episodes(rng, 300, 32)

    def build(graph):
        torch.manual_seed(0)
        conf = learner_conf(Agent, use_prioritized_replay=True, per_beta0=1.0, use_cuda_graph=graph)
        read, write = Replay.make(conf, compute_reward=fdql.RewardOp.bitflip())
        write[0].add_rows(cols, episode_lengths=[32] * 300)
        return Agent.Learner(conf, read), read[0]

    lg, hg = build(True)
    lg.train_step()  # three eager warm-up updates and one replay of the captured step
    le, he = build(False)
    for _ in range(4):
        le.train_step()
    for (n1, p1), (n2, p2) in zip(lg.actor_critic.state_dict().items(), le.actor_critic.state_dict().items()):
        torch.testing.assert_close(p1, p2, rtol=1e-5, atol=1e-6, msg=lambda m, n1=n1: f"{n1}: {m}")
    rg, re_ = lg._ring_of(hg), le._ring_of(he)
    torch.testing.assert_close(rg.priority_views()[0], re_.priority_views()[0], rtol=1e-4, atol=1e-6)
    losses = [float(lg.train_step()) for _ in range(4)]
    assert all(np.isfinite(losses)) and len(set(losses)) > 1
