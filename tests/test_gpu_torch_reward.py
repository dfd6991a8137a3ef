"""Write-time hindsight relabelling with a TorchReward (a user reward function evaluated in PyTorch on the device once per flush,
consumed by fdql_her_flush_episodes_given / fdql_vmap_flush_episodes_given).

Each enum functor restated in torch must store exactly the rows the enum path stores; the reference goldens must come out of the
callable path as they come out of the enum path; a reward no functor expresses (the gym-robotics form) must match the CPU
restatement; the errors are the documented ones; and a graphed learner keeps training while TorchReward flushes run between its
replays."""
import random
import types

import numpy as np
import pytest

from conftest import load_golden
from oracle import cpu_restatement as O

pytestmark = pytest.mark.gpu


def npy(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------- the enum functors restated in torch
def t_bitflip(ag, g):
    hit = (ag == g).all(-1)
    return hit.float() - 1.0, hit


def t_all_geq(ag, g):
    hit = (ag >= g).all(-1)
    return hit.float() - 1.0, hit


def t_first_geq(ag, g):
    hit = ag[:, 0] >= g[:, 0]
    return hit.float() - 1.0, hit


def t_pnorm(weights, threshold, p):
    """FDQL_REWARD_WEIGHTED_PNORM in torch: the functor reads its parameters as float32 and evaluates in fp64."""
    import torch
    w32, thr, p32 = np.asarray(weights, np.float32), float(np.float32(threshold)), float(np.float32(p))

    def f(ag, g):
        w = torch.as_tensor(w32, device=ag.device).double()
        acc = ((ag.double() - g.double()).abs() * w).sum(-1)
        r = -torch.pow(acc, torch.tensor(p32, dtype=torch.float64, device=ag.device))
        return r.float(), r > -thr
    return f


PNORM = dict(weights=[1.0, 0.5, 0.25, 2.0, 1.0, 0.5], threshold=0.3, p=0.5)


def reward_pair(fdql, name, G=None):
    """(RewardOp, TorchReward) of one functor."""
    if name == "pnorm":
        w = (PNORM["weights"] * 8)[:G]
        return fdql.RewardOp.weighted_pnorm(w, PNORM["threshold"], PNORM["p"]), fdql.TorchReward(t_pnorm(w, PNORM["threshold"], PNORM["p"]))
    fn = {"bitflip": t_bitflip, "all_geq": t_all_geq, "first_geq": t_first_geq}[name]
    return fdql.RewardOp.coerce(name), fdql.TorchReward(fn)


def goals(rng, name, n, G, nan=True):
    """Goal rows where the functors hit often, with NaN and -0 mixed in.  pnorm uses multiples of 1/8 and power-of-two weights:
    every product and sum of its fp64 norm is exact, so the result does not depend on the order of summation."""
    if name == "bitflip":
        x = rng.integers(0, 2, (n, G)).astype(np.float32)
    elif name == "pnorm":
        x = (rng.integers(-4, 5, (n, G)) / 8).astype(np.float32)
    else:
        x = rng.integers(-1, 2, (n, G)).astype(np.float32)
    x[(x == 0) & (rng.random((n, G)) < 0.5)] = -0.0
    if nan:
        x[rng.random((n, G)) < 0.01] = np.nan
    return x


def episode_rows(rng, name, lengths, G, obs=5, nan=True):
    """Per-row dicts of whole episodes, as a runner hands them to a write head."""
    rows = []
    for L in lengths:
        ag = goals(rng, name, L, G, nan)
        dg = np.repeat(goals(rng, name, 1, G, nan), L, 0)
        for t in range(L):
            r = {"obs_1d": rng.standard_normal(obs).astype(np.float32), "action": rng.uniform(-1, 1, 2).astype(np.float32),
                 "achieved_goal": ag[t], "desired_goal": dg[t], "reward": float(rng.integers(-1, 1)),
                 "task_done": bool(rng.random() < 0.1), "episode_done": t == L - 1, "episode_step": t, "info": {}}
            rows.append(r)
    return rows


def same_bits(a, b, what):
    """Equal bit for bit, except that any NaN equals any NaN (the payload of a NaN the reward function makes is its own)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, what
    na, nb = np.isnan(a), np.isnan(b)
    np.testing.assert_array_equal(na, nb, err_msg=f"{what}: NaN positions")
    np.testing.assert_array_equal(np.where(na, 0, a.view(np.int32)), np.where(nb, 0, b.view(np.int32)), err_msg=what)


def ring_of(head):
    while hasattr(head, "replay_buffer"):
        head = head.replay_buffer
    return getattr(head, "replay", head)


def assert_same_ring(r1, r2):
    assert (r1._top, r1._curr_len) == (r2._top, r2._curr_len)
    m1, m2 = r1.memory, r2.memory
    assert list(m1) == list(m2)
    for k in m1:
        same_bits(npy(m1[k]), npy(m2[k]), k)
    for a, b in zip(r1.episode_extents(), r2.episode_extents()):
        np.testing.assert_array_equal(npy(a), npy(b), err_msg="episode extents")


def make(mode, op, n_step, gamma=0.98, replay_size=4096):
    from fastdeepqlearning_b200 import Replay
    conf = types.SimpleNamespace(replay_size=replay_size, batch_size=8, temporal_len=2, num_instances=1, use_nStep_lowerbounds=True,
                                 nStep_return_steps=n_step, gamma=gamma, use_squashed_rewards=False, use_HER=True, her_mode=mode,
                                 training_device="cuda:0")
    return Replay.make(conf, compute_reward=op)


def feed(head, rows, seed):
    random.seed(seed)
    np.random.seed(seed)
    for r in rows:
        head.add(r)


# ---------------------------------------------------------------------------------------------- 1. same rows as the enum path
@pytest.mark.parametrize("name", ["bitflip", "all_geq", "first_geq", "pnorm"])
@pytest.mark.parametrize("mode", ["final", "random"])
@pytest.mark.parametrize("n_step", [1000, 4])
def test_write_time_rows_equal_the_enum_path(fdql, name, mode, n_step):
    """Episodes of 1, 7, 128 and 1000 rows through HindsightNStepReplay(NStepReturn) twice -- the ring wraps, and with n_step = 4
    every longer episode gets its Q3 duplicates -- once with the RewardOp and once with the same functor as a TorchReward."""
    G = 6
    op, tr = reward_pair(fdql, name, G)
    rows = episode_rows(np.random.default_rng(7), name, [1, 7, 128, 1000, 7, 128, 1000, 1], G)
    rings = []
    for reward in (op, tr):
        _, write = make(mode, reward, n_step, replay_size=3001)
        feed(write[0], rows, 11)
        rings.append(ring_of(write[0]))
    assert rings[0]._curr_len == 3000  # wrapped
    mem = npy(rings[1].memory["task_done"])
    assert 0 < mem.sum() < mem.size
    assert_same_ring(*rings)


# ---------------------------------------------------------------------------------------------- 2. vmap write
@pytest.mark.parametrize("name", ["bitflip", "pnorm"])
@pytest.mark.parametrize("returns", ["none", "quirk", "sane"])
def test_vmap_write_equals_the_enum_path(fdql, name, returns):
    """HindsightVmapWrite with V = 32, G = 16 (over NStepReturnVmap with n_step = 4 < most episodes, in both done modes, or alone)
    through fdql_vmap_flush_episodes_given against the enum path; the ring wraps."""
    from fastdeepqlearning_b200 import Replay
    from fastdeepqlearning_b200.Replay import wrappers as W
    G, V = 16, 32
    op, tr = reward_pair(fdql, name, G)
    rows = episode_rows(np.random.default_rng(3), name, [1, 7, 128, 300, 7, 128], G)
    rings = []
    for reward in (op, tr):
        shard = Replay.AsyncReplayMemory(500, 8, 2)
        inner = shard if returns == "none" else W.NStepReturnVmap(shard, 4, 0.97, reference_done_quirk=returns == "quirk")
        feed(W.HindsightVmapWrite(inner, reward, num_virtual_goals=V), rows, 5)
        rings.append(shard.replay)
    assert rings[0]._curr_len == 499
    assert ("virtual_mc_return" in rings[0].keys) == (returns != "none")
    vd = npy(rings[1].memory["virtual_dones"])
    assert 0 < vd.sum() < vd.size
    assert_same_ring(*rings)


# ---------------------------------------------------------------------------------------------- 3. reference goldens
def _feed_golden(head, g, name, gdt):
    off = 0
    for L in g[f"{name}_lengths"]:
        for t in range(L):
            i = off + t
            head.add({"obs_1d": g[f"{name}_in_obs"][i], "action": g[f"{name}_in_action"][i],
                      "achieved_goal": g[f"{name}_in_ag"][i].astype(gdt), "desired_goal": g[f"{name}_in_dg"][i].astype(gdt),
                      "reward": float(g[f"{name}_in_reward"][i]), "task_done": bool(g[f"{name}_in_task_done"][i]),
                      "episode_done": t == L - 1, "episode_step": t, "info": {}})
        off += L


@pytest.mark.parametrize("name", ["bitflip", "all_geq", "first_geq"])
@pytest.mark.parametrize("mode", ["final", "random"])
def test_her_golden_through_the_callable_path(fdql, name, mode, monkeypatch):
    g = load_golden("her")
    read, write = make(mode, reward_pair(fdql, name)[1], 1000, float(g["gamma"]))
    it = iter(list(g[f"{name}_picks"]))
    monkeypatch.setattr(random, "choice", lambda seq: seq[len(seq) - 1 - next(it)])
    _feed_golden(write[0], g, name, np.int64 if name == "bitflip" else np.float64)
    ring = read[0]
    n = len(ring)
    assert n == 2 * g[f"{name}_lengths"].sum()
    mem = {k: npy(v)[:n] for k, v in ring.memory.items()}
    for k in ("obs_1d", "action", "achieved_goal", "desired_goal", "task_done", "episode_done", "episode_step", "reward", "mc_return"):
        np.testing.assert_array_equal(mem[k], g[f"{name}_{mode}_{k}"].astype(np.float32), err_msg=k)


def _parking(fdql, g):
    return fdql.TorchReward(t_pnorm(list(g["weights"]), float(g["success"]), float(g["p"])))


@pytest.mark.parametrize("mode", ["final", "random"])
def test_parking_golden_through_the_callable_path(fdql, mode, monkeypatch):
    g = load_golden("pnorm")
    read, write = make(mode, _parking(fdql, g), 1000, float(g["gamma"]))
    it = iter(list(g["parking_picks"]))
    monkeypatch.setattr(random, "choice", lambda seq: seq[len(seq) - 1 - next(it)])
    _feed_golden(write[0], g, "parking", np.float64)
    ring = read[0]
    n = len(ring)
    assert n == 2 * g["parking_lengths"].sum()
    mem = {k: npy(v)[:n] for k, v in ring.memory.items()}
    for k in ("obs_1d", "action", "achieved_goal", "desired_goal", "task_done", "episode_done", "episode_step"):
        np.testing.assert_array_equal(mem[k], g[f"parking_{mode}_{k}"].astype(np.float32), err_msg=k)
    assert mem["task_done"].sum() > 0
    np.testing.assert_allclose(mem["reward"], g[f"parking_{mode}_reward"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(mem["mc_return"], g[f"parking_{mode}_mc_return"], rtol=1e-5, atol=1e-6)


def test_parking_vmap_golden_through_the_callable_path(fdql, monkeypatch):
    from fastdeepqlearning_b200 import Replay
    from fastdeepqlearning_b200.Replay import wrappers as W
    g = load_golden("pnorm")
    V = int(g["V"])
    lengths = g["vmap_lengths"]
    picks = iter(g["vmap_picks_deque"].reshape(len(lengths), V))
    shard = Replay.AsyncReplayMemory(4096, 8, 2)
    her = W.HindsightVmapWrite(W.NStepReturnVmap(shard, 1000, float(g["gamma"]), reference_done_quirk=True), _parking(fdql, g),
                               num_virtual_goals=V)
    monkeypatch.setattr(np.random, "randint", lambda low, high=None, size=None: np.asarray(next(picks)))
    _feed_golden(her, g, "vmap", np.float32)
    monkeypatch.undo()
    n = int(lengths.sum())
    mem = {k: npy(v)[:n] for k, v in shard.replay.memory.items()}
    np.testing.assert_array_equal(mem["virtual_goals"].reshape(n, -1), g["vmap_virtual_goals"].reshape(n, -1).astype(np.float32))
    np.testing.assert_array_equal(mem["virtual_dones"], g["vmap_virtual_dones"].astype(np.float32))
    np.testing.assert_allclose(mem["virtual_rewards"], g["vmap_virtual_rewards"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(mem["virtual_mc_return"], g["vmap_virtual_mc_return"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", ["bitflip", "all_geq"])
@pytest.mark.parametrize("with_returns", [True, False])
def test_her_vmap_golden_through_the_callable_path(fdql, name, with_returns, monkeypatch):
    from fastdeepqlearning_b200 import Replay
    from fastdeepqlearning_b200.Replay import wrappers as W
    g = load_golden("her_vmap")
    V = int(g["V"])
    lengths = g[f"{name}_lengths"]
    picks = iter(g[f"{name}_picks_deque"].reshape(len(lengths), V))
    shard = Replay.AsyncReplayMemory(4096, 8, 2)
    inner = W.NStepReturnVmap(shard, 1000, float(g["gamma"]), reference_done_quirk=True) if with_returns else shard
    her = W.HindsightVmapWrite(inner, reward_pair(fdql, name)[1], num_virtual_goals=V)
    monkeypatch.setattr(np.random, "randint", lambda low, high=None, size=None: np.asarray(next(picks)))
    _feed_golden(her, g, name, np.float32)
    monkeypatch.undo()
    tag = "ret" if with_returns else "noret"
    n = int(lengths.sum())
    mem = shard.replay.memory
    want_keys = [k[len(f"{name}_{tag}_"):] for k in g.files if k.startswith(f"{name}_{tag}_")]
    assert set(want_keys) == set(mem)
    for k in want_keys:
        want = g[f"{name}_{tag}_{k}"]
        np.testing.assert_array_equal(npy(mem[k])[:n].reshape(n, -1), want.reshape(n, -1).astype(np.float32), err_msg=k)


# ---------------------------------------------------------------------------------------------- 4. a reward no functor expresses
EPS = 0.05


def robotics_torch(ag, g):
    """gym-robotics / panda-gym sparse reward: -(||ag - g||_2 > eps), done = ||ag - g||_2 <= eps."""
    d = (ag - g).norm(dim=-1)
    return -(d > EPS).float(), d <= EPS


def robotics_numpy(ag, g):
    d = np.linalg.norm(np.asarray(ag, np.float64) - np.asarray(g, np.float64), axis=-1)
    return -(d > EPS).astype(np.float64), d <= EPS


@pytest.mark.parametrize("mode", ["final", "random"])
def test_robotics_reward_vs_cpu_restatement(fdql, mode):
    """The goals lie on a lattice of pitch 0.25 with a jitter of at most 1e-3 per component: two goals are either within 3.5e-3 of
    each other or at least 0.245 apart, never near eps = 0.05, so the fp32 torch norm and the fp64 numpy norm cannot disagree on
    which side of the threshold a pair lies."""
    rng = np.random.default_rng(5)
    G, lengths, gamma = 3, [5, 50, 200, 1, 37], 0.97

    def lattice(n):
        return (rng.integers(0, 3, (n, G)) * 0.25 + rng.uniform(-1e-3, 1e-3, (n, G))).astype(np.float32)
    rows = []
    for L in lengths:
        ag, dg = lattice(L), np.repeat(lattice(1), L, 0)
        r, d = robotics_numpy(ag, dg)
        for t in range(L):
            rows.append({"obs_1d": rng.standard_normal(4).astype(np.float32), "action": rng.uniform(-1, 1, 2).astype(np.float32),
                         "achieved_goal": ag[t], "desired_goal": dg[t], "reward": float(r[t]), "task_done": bool(d[t]),
                         "episode_done": t == L - 1, "episode_step": t})
    read, write = make(mode, fdql.TorchReward(robotics_torch), 1000, gamma)
    feed(write[0], rows, 9)
    random.seed(9)
    oracle = O.RingOracle(4096, 8, 2)
    her = O.HindsightOracle(O.NStepOracle(oracle, 1000, gamma), robotics_numpy, mode=mode,
                          goal_picker=lambda L: L - 1 - random.choice(range(L)))
    for r in rows:
        her.add(r)
    n = len(read[0])
    assert n == len(oracle) == 2 * sum(lengths)
    mem = {k: npy(v)[:n] for k, v in read[0].memory.items()}
    want = {k: np.asarray(v[:n], np.float32).reshape(n, -1) for k, v in oracle.memory.items()}
    for k in ("obs_1d", "action", "achieved_goal", "desired_goal", "task_done", "episode_done", "episode_step", "reward"):
        np.testing.assert_array_equal(mem[k].reshape(n, -1), want[k], err_msg=k)
    assert 0 < mem["task_done"].sum() < n
    np.testing.assert_allclose(mem["mc_return"].reshape(n, -1), want["mc_return"], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------- 5. errors
def _filled_ring(fdql, reward):
    from fastdeepqlearning_b200 import Replay
    ring = Replay.ReplayMemory(256, 8, 2)
    ring.set_reward_op(reward, 0.99)
    rng = np.random.default_rng(0)
    L = 10
    ag = rng.integers(0, 2, (L, 4)).astype(np.float32)
    cols = {"obs_1d": rng.standard_normal((L, 3)).astype(np.float32), "achieved_goal": ag, "desired_goal": ag[::-1].copy(),
            "reward": -np.ones((L, 1), np.float32), "task_done": np.zeros((L, 1), np.float32),
            "episode_done": (np.arange(L) == L - 1).astype(np.float32).reshape(-1, 1),
            "episode_step": np.arange(L, dtype=np.float32).reshape(-1, 1), "mc_return": np.zeros((L, 1), np.float32)}
    begin = ring.add_rows(cols, episode_lengths=[L], with_returns=True)
    return ring, begin, L


def test_wrong_outputs_of_fn_raise_on_the_flush(fdql):
    import torch
    bad = [
        (lambda a, g: (torch.zeros(a.shape[0] + 1, device=a.device), torch.zeros(a.shape[0] + 1, dtype=torch.bool, device=a.device)),
         ValueError, "shape"),
        (lambda a, g: (torch.zeros(a.shape[0], dtype=torch.float64, device=a.device), (a == g).all(-1)), TypeError, "dtype"),
        (lambda a, g: (torch.zeros(a.shape[0]), torch.zeros(a.shape[0], dtype=torch.bool)), ValueError, "cpu"),
    ]
    for fn, exc, word in bad:
        ring, begin, L = _filled_ring(fdql, fdql.TorchReward(fn))
        with pytest.raises(exc, match=word):
            ring.add_hindsight_rows([begin], [L], [begin + L - 1])
    with pytest.raises(TypeError, match="TorchReward"):
        _filled_ring(fdql, t_bitflip)


def test_sample_time_relabelling_refuses_a_torch_reward(fdql):
    from fastdeepqlearning_b200 import Replay
    from fastdeepqlearning_b200.Replay.wrappers import ConfigurationError
    ring, begin, L = _filled_ring(fdql, fdql.TorchReward(t_bitflip))
    with pytest.raises(ConfigurationError, match="device functor"):
        ring.temporal_sample(relabel_prob=0.8)
    starts, flags, goals_ = ring.draw_streams(8, relabel_prob=0.8)
    with pytest.raises(ConfigurationError, match="device functor"):
        ring.temporal_sample(starts=starts, flags=flags, goal_rows=goals_)
    with pytest.raises(ConfigurationError, match="device functor"):
        Replay.wrappers.SampleTimeHindsight(ring)
    with pytest.raises(ConfigurationError, match="device functor"):
        make("future", fdql.TorchReward(t_bitflip), 1000)
    ring.temporal_sample()  # plain windows are served


def test_snapshot_records_a_torch_reward_and_needs_it_set_again(fdql):
    from fastdeepqlearning_b200 import Replay
    tr = fdql.TorchReward(t_bitflip)
    ring, begin, L = _filled_ring(fdql, tr)
    ring.add_hindsight_rows([begin], [L], [begin + 3])
    sd = ring.state_dict()
    assert sd["reward_op"] == "torch"
    with pytest.raises(ValueError, match="TorchReward"):
        Replay.ReplayMemory(256, 8, 2).load_state_dict(sd)
    restored = Replay.ReplayMemory(256, 8, 2)
    restored.set_reward_op(tr)
    restored.load_state_dict(sd)
    assert restored.reward_op is tr
    assert_same_ring(ring, restored)
    dst = int(restored.add_hindsight_rows([begin], [L], [begin + 5])[0])  # the restored ring flushes with the reward it was given
    ring.add_hindsight_rows([begin], [L], [begin + 5])
    for k, v in ring.memory.items():
        same_bits(npy(v), npy(restored.memory[k]), k)
    for a, b in zip(ring.episode_extents(), restored.episode_extents()):
        np.testing.assert_array_equal(npy(a)[dst:dst + L], npy(b)[dst:dst + L], err_msg="extents of the flushed copy")


def test_given_entry_points_check_rows_and_goal_roles_on_the_host(fdql):
    import ctypes as C
    import torch
    from fastdeepqlearning_b200 import Replay, _lib as Lm
    lib = fdql.lib()
    ring, begin, L = _filled_ring(fdql, fdql.TorchReward(t_bitflip))
    dev = lambda v, dt: torch.tensor(v, dtype=dt, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    src, lens, dst, goal = dev([begin], torch.int64), dev([L], torch.int32), dev([100], torch.int64), dev([begin], torch.int64)
    r, d = torch.zeros(L + 1, device="cuda"), torch.zeros(L + 1, dtype=torch.uint8, device="cuda")
    assert lib.fdql_her_flush_episodes_given(ring._h, 1, p(src), p(lens), p(dst), p(goal), L + 1, p(r), p(d), p(r), 0.99, 1, None) \
        == Lm.FDQL_EINVAL
    assert b"episodes hold 10 rows" in lib.fdql_last_error()
    bad_len = dev([0], torch.int32)
    assert lib.fdql_her_flush_episodes_given(ring._h, 1, p(src), p(bad_len), p(dst), p(goal), 0, p(r), p(d), p(r), 0.99, 1, None) \
        == Lm.FDQL_EINVAL
    assert b"ep_len[0]" in lib.fdql_last_error()
    picks = dev([begin] * 4, torch.int64)
    assert lib.fdql_vmap_flush_episodes_given(ring._h, 1, p(src), p(lens), p(picks), 0, 1, 2, -1, L, p(r), p(d), 0.99, 1, 0, None) \
        == Lm.FDQL_EINVAL  # no virtual keys in this ring
    plain = Replay.ReplayMemory(64, 8, 2)
    plain.add_rows({"obs_1d": np.zeros((L, 3), np.float32), "reward": np.zeros((L, 1), np.float32)}, episode_lengths=[L])
    assert lib.fdql_her_flush_episodes_given(plain._h, 1, p(src), p(lens), p(dst), p(goal), L, p(r), p(d), p(r), 0.99, 1, None) \
        == Lm.FDQL_EINVAL
    assert b"achieved_goal and desired_goal" in lib.fdql_last_error()
    vm = Replay.ReplayMemory(64, 8, 2)
    vm.add_rows({"virtual_goals": np.zeros((L, 10), np.float32), "virtual_rewards": np.zeros((L, 5), np.float32),
                 "virtual_dones": np.zeros((L, 5), np.float32), "reward": np.zeros((L, 1), np.float32)}, episode_lengths=[L])
    assert lib.fdql_vmap_flush_episodes_given(vm._h, 1, p(src), p(lens), p(picks), 0, 1, 2, -1, L, p(r), p(d), 0.99, 1, 0, None) \
        == Lm.FDQL_EINVAL
    assert b"achieved_goal, desired_goal" in lib.fdql_last_error()
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- 6. end to end
def test_graphed_learner_trains_while_torch_reward_flushes_run(fdql):
    """Replay.make(her_mode="random") with a TorchReward feeding a learner whose whole step is a CUDA graph: episodes are flushed
    (gather, torch call, given-reward kernel, on the writer's stream) between the replays of the captured step, for 300 steps."""
    import torch
    from fastdeepqlearning_b200 import Agent, Replay
    torch.manual_seed(0)
    conf = Agent.LearnerConf(training_device="cuda:0", obs_space={"obs_1d": 8, "achieved_goal": 8, "desired_goal": 8},
                             action_space=types.SimpleNamespace(shape=(2,)), num_critics=2, num_q_predictions=5, top_quantiles_to_drop=0.2,
                             batch_size=128, temporal_len=2, replay_size=20000, use_HER=True, her_mode="random", num_instances=1,
                             gamma=0.98, pi_hidden_dims=(32,), critic_hidden_dims=(32, 32), use_cuda_graph=True)
    read, write = Replay.make(conf, compute_reward=fdql.TorchReward(t_bitflip))
    rows = episode_rows(np.random.default_rng(2), "bitflip", [16] * 400, 8, obs=8, nan=False)
    for r in rows[:16 * 40]:
        write[0].add(r)
    learner = Agent.Learner(conf, read)
    ring = ring_of(read[0])
    it = iter(rows[16 * 40:])
    losses = []
    for step in range(300):
        for _ in range(12):  # three quarters of an episode per step: a flush every other step or so
            r = next(it, None)
            if r is not None:
                write[0].add(r)
        losses.append(float(learner.train_step()))
        for out in ring._out_cache.values():
            for t in (out.values() if isinstance(out, dict) else out):
                assert bool(torch.isfinite(t).all()), step
    assert np.isfinite(losses).all() and len(set(losses)) > 1
    assert len(learner._graphs) == 1
    assert len(read[0]) == 2 * (16 * 40 + 12 * 300)  # every episode stored twice: its real rows and the relabelled copy
