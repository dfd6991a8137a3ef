"""Mirror of franQ/Agent/components/soft_actor_critic.py: SoftActorCritic with the same members (critic, critic_target,
critic_frozen, actor, actor_target, log_alpha, curr_alpha), `q_loss`, `actor_loss`, `update_target`.

`q_loss(curr_xp, next_xp) -> (q_loss [T-1,B,1], None, summaries)` keeps the reference signature; everything after the
critics' forward passes (entropy term, min over atoms, TD target, smooth-L1, lower bound, summaries and the gradient
w.r.t. q_pred) is ONE launch of fdql_sac_min_target_loss instead of a dozen torch ops."""
import math

import torch
from torch import nn

from . import models
from ... import ops


def make_actor(conf, input_dim):
    if getattr(conf, "discrete", False):  # soft_actor_critic.py:12-14
        return models.GumbelPolicy(input_dim, conf.action_space.n, conf.pi_hidden_dims)
    return models.GaussianPolicy(input_dim, conf.action_space.shape[0], conf.pi_hidden_dims)


def make_critic(conf, input_dim):
    act = conf.action_space.n if getattr(conf, "discrete", False) else conf.action_space.shape[-1]
    cls = models.BatchedMLPEnsemble if getattr(conf, "batched_critics", True) else models.MLPEnsemble
    return cls(input_dim + act, conf.num_q_predictions, conf.critic_hidden_dims, ensemble_size=conf.num_critics)


def _summaries_from_stats(stats, n_atoms, with_violations):
    """q_pred mean, mean unbiased row variance, constraint violations (soft_actor_critic.py:86-87,95-97) from the
    kernel's 4 accumulators {sum q, sum row-var, #violations, M}; stays on the device (no sync)."""
    m = stats[3].clamp(min=1)
    out = {"q_pred_mu": (stats[0] / (m * n_atoms)).float(), "q_pred_var": (stats[1] / m).float()}
    if with_violations:
        out["mc_constraint_violations"] = (stats[2] / (m * n_atoms)).float()
    return out


class _LossWithStats(torch.autograd.Function):
    """Differentiable wrapper: forward launches the fused kernel once (loss, d loss/d q_pred, stats), backward scales."""

    @staticmethod
    def forward(ctx, q_pred, fn):
        r = fn(q_pred)
        ctx.save_for_backward(r["grad"])
        ctx.mark_non_differentiable(r["stats"])
        return r["loss"], r["stats"]

    @staticmethod
    def backward(ctx, g_loss, _g_stats):
        (grad,) = ctx.saved_tensors
        return grad * g_loss, None


class _ReducedLossWithStats(torch.autograd.Function):
    """sum_m weight[m] * loss[m] as one scalar; the kernel applied `weight` to d loss / d q_pred itself (grad_scale).  The unweighted
    per-transition loss comes out as a third, non-differentiable output (the priority signal of prioritized replay)."""

    @staticmethod
    def forward(ctx, q_pred, fn, weight):
        r = fn(q_pred)
        ctx.save_for_backward(r["grad"])
        ctx.mark_non_differentiable(r["stats"], r["loss"])
        return (r["loss"] * weight).sum(), r["stats"], r["loss"]

    @staticmethod
    def backward(ctx, g_total, _g_stats, _g_loss):
        (grad,) = ctx.saved_tensors
        return grad * g_total, None, None


class SoftActorCritic(nn.Module):
    def __init__(self, conf, input_dim, actor_factory=make_actor, critic_factory=make_critic):
        super().__init__()
        self.conf = conf
        self.critic = critic_factory(conf, input_dim)
        self.critic_target = critic_factory(conf, input_dim)
        self.critic_frozen = critic_factory(conf, input_dim)  # used for updating the actor (soft_actor_critic.py:33)
        self.critic_target.load_state_dict(self.critic.state_dict())
        self.actor = actor_factory(conf, input_dim)
        self.actor_target = actor_factory(conf, input_dim)
        self.actor_target.load_state_dict(self.actor.state_dict())
        self.log_alpha = nn.Parameter(torch.tensor(float(conf.init_log_alpha), dtype=torch.float32))
        # curr_alpha = exp(log_alpha) (soft_actor_critic.py:40,151), kept as a 1-element device tensor: the loss kernel reads it
        # from device memory, so no step of the learner needs a host sync (and the step can be captured in a CUDA graph)
        self.register_buffer("curr_alpha", torch.tensor([math.exp(float(conf.init_log_alpha))], dtype=torch.float32))
        self.target_entropy = -float(conf.action_space.n if getattr(conf, "discrete", False)
                                     else math.prod(conf.action_space.shape))
        for p in list(self.critic_target.parameters()) + list(self.critic_frozen.parameters()) + list(self.actor_target.parameters()):
            p.requires_grad_(False)
        self.param_dict = {"actor": list(self.actor.parameters()), "critic": list(self.critic.parameters()),
                           "log_alpha": [self.log_alpha]}
        self._fast_params = sum(self.param_dict.values(), start=[])

    def parameters(self, *args, **kwargs):  # trainable parameters only, like the reference (:50-51)
        return self._fast_params

    @torch.no_grad()
    def update_target(self):
        pairs = [(self.actor_target, self.actor), (self.critic_target, self.critic)]
        for tgt, src in pairs:
            t, s = list(tgt.parameters()), list(src.parameters())
            if getattr(self.conf, "use_hard_updates", False):
                torch._foreach_copy_(t, s)
            else:
                torch._foreach_lerp_(t, s, float(self.conf.tau))  # t*(1-tau) + s*tau (utils/common.py:10-13)

    # ---- shared front half of q_loss: the MLP forward passes (ordinary torch) --------------------------------------
    def _critic_io(self, curr_xp, next_xp):
        with torch.no_grad():
            next_action, next_log_pi, _ = self.actor_target(next_xp["state"])
            next_z = self.critic_target(torch.cat((next_xp["state"], next_action), dim=-1))
        action = curr_xp["action_onehot"] if getattr(self.conf, "discrete", False) else curr_xp["action"]
        q_pred = self.critic(torch.cat((curr_xp["state"], action), dim=-1))
        return q_pred, next_z, next_log_pi

    def _bootstrap_bound(self, q_pred, next_z, next_log_pi, next_xp):
        """soft_actor_critic.py:102-132: the n-step return over the whole sampled window, bootstrapped from the target network at its
        last row, as a lower bound on the prediction at t = 0; zero for windows that cross a terminal.  [B, CQ] like the reference
        (plain torch: off in every reference preset, a handful of [B]-sized ops)."""
        conf = self.conf
        Tm1 = q_pred.shape[0]
        with torch.no_grad():
            tz = next_z[-1]
            if next_log_pi is not None:
                tz = tz + self.curr_alpha * (-next_log_pi[-1])
            td_last = next_xp["reward"][-1] + next_xp["mask"][-1] * conf.gamma * tz.min(-1, keepdim=True)[0]
            g = conf.gamma ** torch.arange(Tm1, device=q_pred.device, dtype=q_pred.dtype).view(-1, *[1] * (next_xp["reward"].dim() - 1))
            ret = (next_xp["reward"] * g).sum(0)
            valid = next_xp["mask"].to(q_pred.dtype).prod(0)
        return valid * ((ret + (conf.gamma ** Tm1) * td_last) - q_pred[0]).relu()

    def q_loss(self, curr_xp, next_xp, grad_scale=None):
        conf = self.conf
        q_pred, next_z, next_log_pi = self._critic_io(curr_xp, next_xp)
        lb = next_xp["mc_return"] if conf.use_nStep_lowerbounds else None
        lp = next_log_pi if conf.use_max_entropy_q else None
        loss, stats = _LossWithStats.apply(q_pred, lambda q: self._q_loss_fused(q, next_z, lp, next_xp, lb, grad_scale))
        summ = _summaries_from_stats(stats, q_pred.shape[-1], lb is not None)
        bound = None
        if conf.use_nStep_lowerbounds and getattr(conf, "use_bootstrap_minibatch_nstep", False):
            bound = self._bootstrap_bound(q_pred, next_z, lp, next_xp)
            summ["bootstrap_minibatch_nstep_violations"] = (bound.detach() != 0).float().mean()
        return loss, bound, summ

    def _q_loss_fused(self, q_pred, next_z, lp, next_xp, lb, grad_scale):
        return ops.sac_min_target_loss(q_pred, next_z, lp, next_xp["reward"], next_xp["mask"], lb, self.curr_alpha, self.conf.gamma,
                                       grad_scale=grad_scale, want_stats=True)

    def q_loss_reduced(self, curr_xp, next_xp, weight, with_loss=False):
        """(sum over the [T-1, B] transitions of weight * q_loss, summaries): q_loss followed by the learner's loss reduce
        (deepQlearning.py:222-225,249) with the reduce weights folded into the kernel's backward pass.  `with_loss=True` appends the
        unweighted per-transition loss [T-1, B, 1] (detached) to the pair."""
        conf = self.conf
        q_pred, next_z, next_log_pi = self._critic_io(curr_xp, next_xp)
        lb = next_xp["mc_return"] if conf.use_nStep_lowerbounds else None
        lp = next_log_pi if conf.use_max_entropy_q else None
        total, stats, loss = _ReducedLossWithStats.apply(q_pred, lambda q: self._q_loss_fused(q, next_z, lp, next_xp, lb, weight), weight)
        summ = _summaries_from_stats(stats, q_pred.shape[-1], lb is not None)
        return (total, summ, loss) if with_loss else (total, summ)

    def _alias_frozen_critic(self):
        """soft_actor_critic.py:142 copies critic -> critic_frozen before every actor update so that the policy gradient flows through
        the critic's function but not into its weights.  Here critic_frozen's parameters (requires_grad False) SHARE the critic's
        storage: always equal, nothing to copy per step, and the optimizer's in-place updates are seen at once."""
        for pf, p in zip(self.critic_frozen.parameters(), self.critic.parameters()):
            if pf.data_ptr() != p.data_ptr():
                pf.data = p.data

    def actor_loss(self, xp):
        """soft_actor_critic.py:136-154 (ordinary torch: it differentiates through the critic MLP)."""
        pi, log_pi, _ = self.actor(xp["state"])
        entropy = -log_pi
        self._alias_frozen_critic()
        qpi = self.critic_frozen(torch.cat((xp["state"].detach(), pi), dim=-1)).mean(-1, keepdim=True)
        alpha_now = self.curr_alpha.detach().clone()  # the buffer is refreshed in place below
        policy_loss = -(alpha_now * entropy) - qpi
        alpha_loss = -(self.log_alpha * (self.target_entropy - entropy).detach())
        with torch.no_grad():
            self.curr_alpha.copy_(torch.exp(self.log_alpha).reshape(1))
        return policy_loss.mean(-1, keepdim=True), alpha_loss, {"curr_alpha": self.curr_alpha}
