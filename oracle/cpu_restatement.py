"""CPU restatement of the franQ learner hot path -- TEST INFRASTRUCTURE (see oracle/__init__.py).

Every function cites the reference lines (relative to /root/reference) whose behaviour it
restates.  Storage is fp32 like the reference's numpy ring / torch tensors; where the
reference computes a step in Python floats (fp64) and rounds on store, so does this file.
Nothing here is imported by the product package.
"""
from __future__ import annotations

import numpy as np

try:  # torch is only needed for the *_torch helpers (CPU tensors)
    import torch
except Exception:  # pragma: no cover
    torch = None


class OversampleError(Exception):
    """franQ/Replay/replay_memory.py:6"""


# ----------------------------------------------------------------------------------------------
# Ring replay  (franQ/Replay/replay_memory.py:9-73)
# ----------------------------------------------------------------------------------------------
class RingOracle:
    """SoA ring with the reference's exact cursor arithmetic.

    * lazy allocation on first add: ndarray values keep shape+dtype, anything else becomes a
      ``(maxlen, 1) float32`` column and must be float32-representable (replay_memory.py:23-35);
    * ``_top = (_top+1) % maxlen``; ``_curr_len = max(_top, _curr_len)`` so the length saturates at
      ``maxlen-1`` (quirk Q1, replay_memory.py:45-46);
    * ``temporal_sample`` draws starts in ``[0, len-T)`` and indexes ``(arange(T)[:,None]+start) % len``
      (replay_memory.py:54-66); ``sample`` draws in ``[0, len)`` (replay_memory.py:48-52).
    """

    def __init__(self, maxlen, batch_size, temporal_len, **_):
        self._maxlen, self._batch_size, self._temporal_len = int(maxlen), batch_size, temporal_len
        self._top = 0
        self._curr_len = 0
        self.memory = {}

    def _allocate(self, row):
        for k, v in row.items():
            if isinstance(v, np.ndarray):
                self.memory[k] = np.zeros((self._maxlen,) + tuple(v.shape), v.dtype)
            else:
                assert np.isclose(np.float32(v), v), "scalar fields must be float32-representable"
                self.memory[k] = np.zeros((self._maxlen, 1), np.float32)

    def add(self, row):
        if not self.memory:
            self._allocate(row)
        for k, v in row.items():
            self.memory[k][self._top] = v
        self._top = (self._top + 1) % self._maxlen
        self._curr_len = max(self._top, self._curr_len)

    def __len__(self):
        return self._curr_len

    def __getitem__(self, idx):
        idx = np.asarray(idx)
        return {k: v[idx] for k, v in self.memory.items()}

    def window_indices(self, starts, length=None):
        length = len(self) if length is None else length
        t = np.arange(self._temporal_len).reshape(-1, 1)
        return (t + np.asarray(starts).reshape(1, -1)) % length

    def check_temporal(self):
        n = len(self)
        if n < 2 * self._temporal_len or n < self._batch_size:
            raise OversampleError("not enough rows")

    def temporal_sample(self, starts=None, rng=None):
        self.check_temporal()
        n = len(self)
        if starts is None:
            rng = np.random if rng is None else rng
            starts = rng.randint(0, n - self._temporal_len, self._batch_size)
        return self[self.window_indices(starts, n)]

    def sample(self, idx=None, rng=None):
        if len(self) < self._batch_size:
            raise OversampleError("not enough rows")
        if idx is None:
            rng = np.random if rng is None else rng
            idx = rng.randint(0, self._curr_len, self._batch_size)
        return self[idx]


def to_learner_dtype(batch):
    """TorchDataLoader casts every key to conf.dtype=float32 (torch_dataloader.py:36)."""
    return {k: np.asarray(v).astype(np.float32) for k, v in batch.items()}


# ----------------------------------------------------------------------------------------------
# n-step / Monte-Carlo return  (franQ/Replay/wrappers/nstep_return.py:23-72)
# ----------------------------------------------------------------------------------------------
def mc_return_newest_first(rewards, gamma):
    """nstep_return.py:60-72.  ``rewards[0]`` is the newest step.  Each step is evaluated in
    fp64 (gamma is a Python float) and rounded to fp32 on store, exactly like the numba loop."""
    r = np.asarray(rewards, dtype=np.float32).squeeze()
    if r.ndim == 0:
        return r.reshape(1)
    r = r.copy()
    for i in range(1, r.shape[0]):
        r[i] = np.float32(np.float64(r[i]) + np.float64(r[i - 1]) * gamma)
    return r


def mc_return_chrono(rewards, gamma):
    """Chronological view of the same recurrence: G_t = r_t + gamma*G_{t+1}, G_last = r_last."""
    r = np.asarray(rewards, dtype=np.float32).reshape(-1)
    return mc_return_newest_first(r[::-1], gamma)[::-1].copy()


def mc_return_chrono_f64(rewards, gamma):
    r = np.asarray(rewards, dtype=np.float64).reshape(-1)
    g = np.zeros_like(r)
    acc = 0.0
    for i in range(len(r) - 1, -1, -1):
        acc = r[i] + gamma * acc
        g[i] = acc
    return g


def segmented_returns(rewards, episode_done, gamma):
    """Return-to-go for a chronological stream of complete episodes delimited by ``episode_done``
    (what NStepReturn stores when n_step >= episode length, nstep_return.py:31,36-48)."""
    r = np.asarray(rewards, np.float32).reshape(-1)
    d = np.asarray(episode_done).reshape(-1).astype(bool)
    out = np.zeros_like(r)
    acc = np.float32(0)
    for i in range(len(r) - 1, -1, -1):
        if d[i]:
            acc = r[i]
        else:
            acc = np.float32(np.float64(r[i]) + np.float64(acc) * gamma)
        out[i] = acc
    return out


class NStepOracle:
    """Row-level behaviour of NStepReturn (nstep_return.py:23-57), incl. quirk Q3: when the
    buffer length reaches n_step the oldest row is emitted with the truncated return and is
    NOT removed, so it is emitted again at the episode flush."""

    def __init__(self, sink, n_step, discount, reward_name="reward", return_name="mc_return",
                 done_name="episode_done"):
        self.sink, self.n_step, self.discount = sink, n_step, discount
        self.reward_name, self.return_name, self.done_name = reward_name, return_name, done_name
        self.rows = []

    def add(self, row):
        self.rows.append(dict(row))
        if row[self.done_name]:
            g = mc_return_chrono([r[self.reward_name] for r in self.rows], self.discount)
            for r, gi in zip(self.rows, g):
                out = dict(r)
                out[self.return_name] = gi
                self.sink.add(out)
            self.rows = []
        elif len(self.rows) == self.n_step:
            g = mc_return_chrono([r[self.reward_name] for r in self.rows], self.discount)
            out = dict(self.rows[0])
            out[self.return_name] = g[0]
            self.sink.add(out)


# ----------------------------------------------------------------------------------------------
# Reward functors  R(achieved_goal, desired_goal) -> (reward, done), vectorised over leading dims
# ----------------------------------------------------------------------------------------------
def reward_bitflip(ag, dg):
    """franQ/Env/bitflip.py:143-152: 0 when every component matches else -1; done = reward==0."""
    m = (np.asarray(ag) == np.asarray(dg)).all(-1)
    r = np.where(m, 0.0, -1.0)
    return r, m


def reward_all_geq(ag, dg):
    """franQ/Env/classic_control_goal/classic_goal.py:88-93 (acrobot goal env)."""
    m = (np.asarray(ag) >= np.asarray(dg)).all(-1)
    return np.where(m, 0.0, -1.0), m


def reward_first_geq(ag, dg):
    """classic_goal.py:306-311 (mountain-car goal env): done = ag[0] >= dg[0]; reward = done-1."""
    m = np.asarray(ag)[..., 0] >= np.asarray(dg)[..., 0]
    return m.astype(np.float64) - 1.0, m


def make_reward_weighted_pnorm(weights, success_threshold, p=0.5):
    """franQ/Env/eleurent_parking.py:42-55: -(|ag-dg| . w)^p ; done = reward > -threshold."""
    w = np.asarray(weights, np.float64)

    def f(ag, dg):
        r = -np.power(np.abs(np.asarray(ag, np.float64) - np.asarray(dg, np.float64)) @ w, p)
        return r, r > -success_threshold

    return f


def fp32_reward(reward_fn):
    """``reward_fn`` with its reward rounded to fp32 and its done left as the fp64 evaluation decided it: the form in which a
    reward value reaches a float32 ring (the device functors evaluate in fp64 and store fp32, as the env's reward column is)."""

    def f(ag, dg):
        r, d = reward_fn(ag, dg)
        return np.asarray(r, np.float64).astype(np.float32).astype(np.float64), d

    return f


REWARD_OPS = {"bitflip": reward_bitflip, "all_geq": reward_all_geq, "first_geq": reward_first_geq}


# ----------------------------------------------------------------------------------------------
# Hindsight relabelling  (franQ/Replay/wrappers/her.py:24-95)
# ----------------------------------------------------------------------------------------------
def her_relabel_episode(achieved_goal, desired_goal, reward, episode_step, goal, reward_fn):
    """Chronological restatement of ``_hindsight_flush`` (her.py:55-95) for one real episode.

    reward'_t       = (reward_t - R(ag_t, dg_t)) + R(ag_t, g*)            (her.py:62-69)
    task_done'_t    = done(R(ag_t, g*))                                    (her.py:62,93)
    episode_step'_t = step_t - step_(oldest row of the synthetic segment)  (her.py:72-83)
       where a synthetic segment ends (chronologically) at every row with task_done' true.
    """
    ag = np.asarray(achieved_goal)
    L = ag.shape[0]
    gr, d = reward_fn(ag, np.broadcast_to(np.asarray(goal), ag.shape))
    orig, _ = reward_fn(ag, np.asarray(desired_goal))
    r = np.asarray(reward, np.float64).reshape(L)
    new_r = (r - orig) + gr
    d = np.asarray(d).astype(bool).reshape(L)
    step = np.asarray(episode_step, np.float64).reshape(L)
    new_step = np.zeros(L, np.float64)
    seg_first = 0
    for t in range(L):
        new_step[t] = step[t] - step[seg_first]
        if d[t]:
            seg_first = t + 1
    return new_r.astype(np.float32), d, new_step.astype(np.float32)


class HindsightOracle:
    """Row-level behaviour of HindsightNStepReplay (her.py:24-95): buffer an episode, on
    ``episode_done`` push the real rows oldest->newest, then one relabelled copy.

    ``goal_picker(L) -> chronological index`` injects the goal choice for mode="random"
    (the reference calls ``random.choice`` on the newest-first deque, her.py:51-53)."""

    def __init__(self, sink, reward_fn, ignore_keys=("info",), mode="random", goal_picker=None):
        self.sink, self.reward_fn, self.ignore, self.mode = sink, reward_fn, tuple(ignore_keys), mode
        self.goal_picker = goal_picker
        self.rows = []

    def add(self, row):
        self.rows.append(dict(row))
        if not row["episode_done"]:
            return
        rows, self.rows = self.rows, []
        keep = [{k: v for k, v in r.items() if k not in self.ignore} for r in rows]
        for r in keep:
            self.sink.add(dict(r))
        L = len(rows)
        if self.mode == "final":
            gi = L - 1
        else:
            gi = int(self.goal_picker(L))
        goal = rows[gi]["achieved_goal"]
        ag = np.stack([np.asarray(r["achieved_goal"]) for r in rows])
        dg = np.stack([np.asarray(r["desired_goal"]) for r in rows])
        rew = np.array([float(np.asarray(r["reward"]).reshape(-1)[0]) for r in rows])
        step = np.array([float(np.asarray(r["episode_step"]).reshape(-1)[0]) for r in rows])
        nr, nd, ns = her_relabel_episode(ag, dg, rew, step, goal, self.reward_fn)
        for t, r in enumerate(keep):
            out = dict(r)
            out["desired_goal"] = goal
            out["task_done"] = bool(nd[t])
            out["episode_step"] = ns[t]
            out["reward"] = nr[t]
            self.sink.add(out)


# ----------------------------------------------------------------------------------------------
# "vmap" hindsight variant  (franQ/Replay/wrappers/her_vmap.py, nstep_return_vmap.py)
# ----------------------------------------------------------------------------------------------
def vmap_virtual_columns(achieved_goal, desired_goal, reward, task_done, virtual_goals, reward_fn):
    """``_virtual_episode_calc`` (her_vmap.py:30-43) for one episode, chronological rows.

    virtual_reward[t, v] = fl32(fl32(reward_t - R(ag_t, dg_t)) + R(ag_t, vg_v))                          (:34,39)
    virtual_done[t, v]   = (task_done_t and not done(R(ag_t, dg_t))) or done(R(ag_t, vg_v))              (:37,40)
    Returns ([L, V+1] float32, [L, V+1] bool, [L, V+1, G]) with the real goal / reward / done appended as column V (:85-87)."""
    ag, dg = np.asarray(achieved_goal), np.asarray(desired_goal)
    vg = np.asarray(virtual_goals)
    L, V = ag.shape[0], vg.shape[0]
    r = np.asarray(reward, np.float32).reshape(L)
    d = np.asarray(task_done).astype(bool).reshape(L)
    Rd, dd = reward_fn(ag, dg)
    ga_r = (r - np.asarray(Rd, np.float32)).astype(np.float32)
    ga_d = d & ~np.asarray(dd).astype(bool)
    vr = np.zeros((L, V + 1), np.float32)
    vd = np.zeros((L, V + 1), bool)
    goals = np.zeros((L, V + 1) + ag.shape[1:], np.float64)
    for v in range(V):
        Rv, dv = reward_fn(ag, np.broadcast_to(vg[v], ag.shape))
        vr[:, v] = (ga_r + np.asarray(Rv, np.float32)).astype(np.float32)
        vd[:, v] = ga_d | np.asarray(dv).astype(bool)
        goals[:, v] = vg[v]
    vr[:, V], vd[:, V], goals[:, V] = r, d, dg
    return vr, vd, goals


def vmap_returns(virtual_rewards, virtual_dones, gamma, reference_done_quirk=True):
    """``calculate_montecarlo_return`` / ``_inner`` of nstep_return_vmap.py:61-74 for one episode, chronological [L, V+1]:
    G_t = fl32(r_t + G_{t+1} * gamma * m_t) evaluated in fp64, m_t = dones[t] as the reference has it (quirk Q7) or
    1 - dones[t] (``reference_done_quirk=False``: the return stops at a virtual terminal)."""
    r = np.asarray(virtual_rewards, np.float32).copy()
    d = np.asarray(virtual_dones).astype(bool)
    m = d if reference_done_quirk else ~d
    for t in range(r.shape[0] - 2, -1, -1):
        r[t] = (r[t].astype(np.float64) + r[t + 1].astype(np.float64) * float(gamma) * m[t]).astype(np.float32)
    return r


def vmap_write_episode(cols, picks_chrono, reward_fn, gamma=None, reference_done_quirk=True):
    """HindsightVmapWrite._hindsight_flush (+ NStepReturnVmap._flush when gamma is given) for one episode given as
    chronological columns; ``picks_chrono`` are the rows whose achieved_goal become the virtual goals (her_vmap.py:75)."""
    vg = np.asarray(cols["achieved_goal"])[np.asarray(picks_chrono)]
    vr, vd, goals = vmap_virtual_columns(cols["achieved_goal"], cols["desired_goal"], cols["reward"], cols["task_done"], vg, reward_fn)
    out = {k: np.asarray(v) for k, v in cols.items()}
    out["virtual_goals"], out["virtual_rewards"], out["virtual_dones"] = goals, vr, vd
    if gamma is not None:
        out["virtual_mc_return"] = vmap_returns(vr, vd, gamma, reference_done_quirk)
    return out


def vmap_pop_returns(virtual_rewards, virtual_dones, n_step, gamma, reference_done_quirk=True):
    """NStepReturnVmap._pop (nstep_return_vmap.py:50-57): when the episode buffer reaches n_step rows the oldest row is emitted with
    the recurrence evaluated over those n_step rows only -- and is not removed (quirk Q3), so it is stored again at the flush.
    Returns the [V+1] truncated returns of the oldest row (chronological inputs [L, V+1], L > n_step)."""
    return vmap_returns(np.asarray(virtual_rewards)[:n_step], np.asarray(virtual_dones)[:n_step], gamma, reference_done_quirk)[0]


def vmap_read_select(batch, column):
    """HindsightVmapRead.temporal_sample + cleanup (her_vmap.py:104-123) on a gathered [T, B, ...] batch."""
    out = {k: v for k, v in batch.items() if not k.startswith("virtual_")}
    out["desired_goal"] = batch["virtual_goals"][:, :, column]
    out["reward"] = batch["virtual_rewards"][:, :, column, None]
    out["task_done"] = batch["virtual_dones"][:, :, column, None]
    if "virtual_mc_return" in batch:
        out["mc_return"] = batch["virtual_mc_return"][:, :, column, None]
    return out


def pohlen_transform(x, epsilon=1e-2, power=0.5):
    """franQ/Replay/wrappers/squash_rewards.py:5-7."""
    x = np.asarray(x, np.float64)
    return np.sign(x) * (np.power(np.abs(x) + 1, power) - 1) + epsilon * x


def sample_time_relabel(cols, starts, T, flags, goal_rows, ep_start, ep_end, reward_fn, gamma):
    """What the device's sample-time relabelling must return, defined through the write-time
    reference semantics: for a window whose start row lies in real episode [s, e] and whose
    flag is set, every window row inside that episode equals the hindsight row the reference
    would have stored for it with goal ``achieved_goal[goal_row]`` (her.py:55-95), and its
    mc_return is the recurrence nstep_return.py:69-72 over the relabelled rewards of the WHOLE
    real episode (quirk Q5).  Rows of the window that fall outside that episode, and windows
    whose flag is clear, are returned as stored.

    cols: dict of [N, w] arrays with keys achieved_goal, desired_goal, reward, task_done,
    episode_step, mc_return (+ any others, gathered verbatim).  Returns {k: [T, B, w]} fp32."""
    starts = np.asarray(starts)
    B = len(starts)
    idx = np.arange(T).reshape(-1, 1) + starts.reshape(1, -1)
    out = {k: np.asarray(v)[idx].astype(np.float32) for k, v in cols.items()}
    for b in range(B):
        if not flags[b]:
            continue
        s, e = int(ep_start[starts[b]]), int(ep_end[starts[b]])
        rows = np.arange(s, e + 1)
        goal = np.asarray(cols["achieved_goal"])[int(goal_rows[b])]
        nr, nd, ns = her_relabel_episode(cols["achieved_goal"][rows], cols["desired_goal"][rows],
                                         cols["reward"][rows].reshape(-1), cols["episode_step"][rows].reshape(-1),
                                         goal, reward_fn)
        g = mc_return_chrono(nr, gamma)
        for t in range(T):
            row = int(starts[b]) + t
            if row > e:
                break
            j = row - s
            out["desired_goal"][t, b] = goal
            out["reward"][t, b, 0] = nr[j]
            out["task_done"][t, b, 0] = float(nd[j])
            out["episode_step"][t, b, 0] = ns[j]
            out["mc_return"][t, b, 0] = g[j]
    return out


# ----------------------------------------------------------------------------------------------
# Learner pre/post-processing  (franQ/Agent/deepQlearning.py:198-258)
# ----------------------------------------------------------------------------------------------
def learner_preprocess(task_done, episode_step):
    """deepQlearning.py:201-203.  Inputs [T,B,1] fp32 -> mask [T,B,1] bool, is_contiguous [T-1,B,1] bool."""
    mask = np.logical_not(np.asarray(task_done))
    step = np.asarray(episode_step)
    contig = (step[1:] == step[:-1] + 1) & mask[:-1]
    return mask, contig


def action_onehot(action, n):
    """deepQlearning.py:206-210."""
    a = np.asarray(action)
    return np.eye(n, dtype=a.dtype)[a.reshape(a.shape[:-1]).astype(np.int64)]


def loss_reduce(per_step_loss, is_contiguous, temporal_len):
    """deepQlearning.py:222-225,249: sum_t(loss*contig) / (sum_t contig + 1e-4), mean over batch, / T."""
    c = np.asarray(is_contiguous, np.float32)
    num = (np.asarray(per_step_loss, np.float32) * c).sum(0)
    return np.float32((num / (c.sum(0) + np.float32(1e-4))).mean() / temporal_len)


def upstream_weight(is_contiguous, temporal_len):
    """d(loss_reduce)/d(per_step_loss[t,b]) = contig / ((sum_t contig + 1e-4) * B * T)."""
    c = np.asarray(is_contiguous, np.float32)
    B = c.shape[1]
    return (c / (c.sum(0, keepdims=True) + np.float32(1e-4)) / np.float32(B) / np.float32(temporal_len)).astype(np.float32)


# ----------------------------------------------------------------------------------------------
# TQC target + quantile-Huber loss  (franQ/Agent/components/distributional_soft_actor_critic.py:40-103)
# ----------------------------------------------------------------------------------------------
def n_atoms_dropped(top_quantiles_to_drop, n_atoms):
    """distributional_soft_actor_critic.py:51-53: ``int(p * CQ)`` atoms are removed from the top."""
    return int(top_quantiles_to_drop * n_atoms)


def tqc_td_target(next_z, next_log_pi, reward, mask, alpha, gamma, n_drop, use_max_entropy_q=True,
                  dtype=np.float32):
    """distributional_soft_actor_critic.py:50-58.  next_z [...,CQ]; the others [...,1].
    n_drop == 0 would make the reference slice ``[:-0]`` (empty target, quirk Q8) -> rejected."""
    if n_drop <= 0:
        raise ValueError("top_quantiles_to_drop*CQ must be >= 1 (reference yields an empty target)")
    z = np.sort(np.asarray(next_z, dtype), axis=-1)[..., :-n_drop]
    if use_max_entropy_q:
        z = z + dtype(alpha) * (-np.asarray(next_log_pi, dtype))
    return (np.asarray(reward, dtype) + np.asarray(mask, dtype) * dtype(gamma) * z).astype(dtype)


def quantile_huber(quantiles, samples, dtype=np.float64):
    """distributional_soft_actor_critic.py:90-103, brute force over the [..., N, K] pair tensor.
    tau_j = j/N + 1/(2N) over the N concatenated atoms (quirk Q9)."""
    q = np.asarray(quantiles, dtype)
    s = np.asarray(samples, dtype)
    delta = s[..., None, :] - q[..., :, None]
    a = np.abs(delta)
    huber = np.where(a > 1, a - dtype(0.5), delta * delta * dtype(0.5))
    n = q.shape[-1]
    tau = (np.arange(n, dtype=np.float32) / np.float32(n) + np.float32(1 / 2 / n)).astype(dtype)
    w = np.abs(tau[:, None] - (delta < 0).astype(dtype))
    return (w * huber).mean((-1, -2))


def quantile_huber_grad(quantiles, samples, dtype=np.float64):
    """d quantile_huber / d quantiles  (SURVEY Appendix B5)."""
    q = np.asarray(quantiles, dtype)
    s = np.asarray(samples, dtype)
    delta = s[..., None, :] - q[..., :, None]
    n, k = q.shape[-1], s.shape[-1]
    tau = (np.arange(n, dtype=np.float32) / np.float32(n) + np.float32(1 / 2 / n)).astype(dtype)
    w = np.abs(tau[:, None] - (delta < 0).astype(dtype))
    return -(w * np.clip(delta, -1, 1)).sum(-1) / (n * k)


def tqc_q_loss(q_pred, next_z, next_log_pi, reward, mask, mc_return, alpha, gamma, n_drop,
               use_max_entropy_q=True, use_lower_bound=True, dtype=np.float64):
    """Critic loss half of DistributionalSoftActorCritic.q_loss given the MLP outputs
    (distributional_soft_actor_critic.py:50-87).  Returns (q_loss [...,1], dloss/dq_pred [...,CQ], summaries)."""
    td = tqc_td_target(next_z, next_log_pi, reward, mask, alpha, gamma, n_drop, use_max_entropy_q, dtype)
    q = np.asarray(q_pred, dtype)
    loss = quantile_huber(q, td, dtype)[..., None]
    grad = quantile_huber_grad(q, td, dtype)
    summaries = {"q_pred_mu": q.mean(), "q_pred_var": q.var(-1, ddof=1).mean()}
    if use_lower_bound:
        lb = np.maximum(np.asarray(mc_return, dtype) - q, 0)
        loss = loss + lb.mean(-1, keepdims=True)
        grad = grad - (lb > 0).astype(dtype) / q.shape[-1]
        summaries["mc_constraint_violations"] = float((lb > 0).sum()) / lb.size
    return loss, grad, summaries


def sac_min_target_loss(q_pred, target_z, next_log_pi, reward, mask, mc_return, alpha, gamma,
                        use_max_entropy_q=True, use_lower_bound=True, dtype=np.float64):
    """Non-distributional variant, franQ/Agent/components/soft_actor_critic.py:63-134 (without the
    optional minibatch bootstrap bound): min over atoms (after adding the entropy term),
    smooth-L1 against every predicted atom, lower bound replaces the TD term where it is active."""
    z = np.asarray(target_z, dtype)
    if use_max_entropy_q:
        z = z + dtype(alpha) * (-np.asarray(next_log_pi, dtype))
    tgt = z.min(-1, keepdims=True)
    td = np.asarray(reward, dtype) + np.asarray(mask, dtype) * dtype(gamma) * tgt
    q = np.asarray(q_pred, dtype)
    d = q - td
    a = np.abs(d)
    l1 = np.where(a < 1, 0.5 * d * d, a - 0.5)
    g = np.clip(d, -1, 1)
    summaries = {"q_pred_mu": q.mean(), "q_pred_var": q.var(-1, ddof=1).mean()}
    if use_lower_bound:
        lb = np.maximum(np.asarray(mc_return, dtype) - q, 0)
        inactive = (lb == 0)
        l1 = l1 * inactive + lb
        g = g * inactive - (lb > 0)
        summaries["mc_constraint_violations"] = float((~inactive).sum()) / lb.size
    n = q.shape[-1]
    return l1.mean(-1, keepdims=True), g / n, summaries


def sac_bootstrap_bound(q_pred, target_z, next_log_pi, reward, mask, alpha, gamma, use_max_entropy_q=True, dtype=np.float64):
    """soft_actor_critic.py:102-132: minibatch n-step bootstrap bound.  Inputs [T-1, B, .]; returns ([B, CQ] bound, d sum(bound*w)/d q_pred
    is -w where the bound is active, on q_pred[0] only).  bound = prod_t mask * relu(sum_t gamma^t r_t + gamma^(T-1) td_target[-1] - q_pred[0])."""
    z = np.asarray(target_z, dtype)
    if use_max_entropy_q:
        z = z + dtype(alpha) * (-np.asarray(next_log_pi, dtype))
    td = np.asarray(reward, dtype) + np.asarray(mask, dtype) * dtype(gamma) * z.min(-1, keepdims=True)
    Tm1 = z.shape[0]
    g = (dtype(gamma) ** np.arange(Tm1)).reshape(-1, 1, 1)
    ret = (np.asarray(reward, dtype) * g).sum(0)
    valid = np.asarray(mask, dtype).prod(0)
    return valid * np.maximum((ret + dtype(gamma) ** Tm1 * td[-1]) - np.asarray(q_pred, dtype)[0], 0)


# torch-CPU forms used as the timed CPU baseline (same operator sequence as the reference) -------
def tqc_q_loss_torch(q_pred, next_z, next_log_pi, reward, mask, mc_return, alpha, gamma, n_drop,
                     use_max_entropy_q=True, use_lower_bound=True):
    """Operator-for-operator torch restatement of distributional_soft_actor_critic.py:50-79,90-103
    (sort, slice, entropy term, td target, [.., N, K] pairwise Huber tensor, mean, relu bound)."""
    with torch.no_grad():
        z, _ = torch.sort(next_z, dim=-1)
        z = z[..., :-n_drop]
        if use_max_entropy_q:
            z = z + alpha * (-next_log_pi)
        td = reward + mask * gamma * z
    delta = td[..., None, :] - q_pred[..., None]
    a = delta.abs()
    huber = torch.where(a > 1, a - 0.5, delta ** 2 * 0.5)
    n = q_pred.shape[-1]
    tau = (torch.arange(n, dtype=q_pred.dtype) / n + 1 / 2 / n).view(*([1] * (q_pred.dim() - 1)), n, 1)
    loss = ((tau - (delta < 0).float()).abs() * huber).mean((-1, -2)).unsqueeze(-1)
    if use_lower_bound:
        lb = (mc_return - q_pred).relu()
        loss = loss + lb.mean(-1, keepdim=True)
    return loss
