"""Learner: mirror of the training half of franQ/Agent/deepQlearning.py (`get_losses` :198-249, `train_step` :105-127,
`_temporal_difference_shift` :251-258) over the device replay and the fused loss kernels.

One `train_step()` consumes one batch from every local replay shard (the reference's loop over `self.replays`).  Under
torch.distributed each rank owns its shards and only gradients cross GPUs: one flat bucket, one NCCL all-reduce per
optimizer step (SURVEY.md section 8e).  The encoder is the reference's default for 1-D observations -- concatenation of
the obs keys -- so `state` is a view-free torch.cat; MLP encoders stay user torch modules (`encoder=` argument)."""
import types

import torch
from torch import nn

from .components.distributional_soft_actor_critic import DistributionalSoftActorCritic
from .components.soft_actor_critic import SoftActorCritic


class LearnerConf(types.SimpleNamespace):
    """The hot-path knobs of franQ/Agent/conf.py:8-76 with the reference's names and defaults."""

    def __init__(self, **kw):
        d = dict(batch_size=256, replay_size=int(5e4), temporal_len=50, use_nStep_lowerbounds=True, nStep_return_steps=1000,
                 gamma=0.99, tau=5e-3, use_hard_updates=False, use_HER=False, her_mode="final", num_critics=5,
                 num_q_predictions=10, top_quantiles_to_drop=0.2, use_max_entropy_q=True, use_distributional_sac=True,
                 use_squashed_rewards=False, num_instances=1, training_device="cuda:0", dtype=torch.float32,
                 init_log_alpha=0.0, learning_rate=3e-4, pi_hidden_dims=(256,), critic_hidden_dims=(256, 256), discrete=False,
                 obs_keys=("obs_1d", "achieved_goal", "desired_goal"), use_bootstrap_minibatch_nstep=False, clip_grad_norm=None,
                 # prioritized replay (Schaul et al. 2016; not a reference mode): priority exponent, importance-sampling exponent annealed
                 # linearly from per_beta0 to 1 over per_beta_steps updates, priority floor, max / mean mix over a window (R2D2)
                 use_prioritized_replay=False, per_alpha=0.6, per_beta0=0.4, per_beta_steps=100_000, per_eps=1e-6, per_eta=0.9,
                 # {key: uint8 / int8} keys the ring stores at one byte per element (image frames, bit-flip states); batches stay fp32
                 replay_key_dtypes=None)
        d.update(kw)
        super().__init__(**d)


class ConcatEncoder(nn.Module):
    """encoder.py:52-58 for 1-D observation spaces without a joiner: state = cat(obs keys)."""

    def __init__(self, keys):
        super().__init__()
        self.keys = tuple(keys)

    def forward_train(self, xp):
        return torch.cat([xp[k] for k in self.keys if k in xp], dim=-1)


class Learner:
    def __init__(self, conf, replays=None, encoder=None, state_dim=None):
        self.conf = conf
        self.device = torch.device(conf.training_device)
        self.encoder = encoder or ConcatEncoder(conf.obs_keys)
        if state_dim is None:
            state_dim = sum(conf.obs_space[k] for k in conf.obs_keys if k in conf.obs_space)
        ac_cls = DistributionalSoftActorCritic if conf.use_distributional_sac else SoftActorCritic
        self.actor_critic = ac_cls(conf, state_dim).to(self.device)
        params = list(self.actor_critic.parameters()) + [p for p in self.encoder.parameters() if p.requires_grad]
        self.params = params
        on_gpu = self.device.type == "cuda"
        self.optimizer = torch.optim.Adam(params, lr=conf.learning_rate, fused=on_gpu, capturable=on_gpu)
        self._graphs = {}  # replay index -> (CUDAGraph, static loss, ring length at capture)
        self.replays = list(replays or [])
        self.train_steps = 0
        self._flat = None
        self._side = None
        self._buckets = None  # (critic parameters, all the others): the two gradient buckets of the split backward
        self._prefetched = {}  # replay -> batch sampled during the previous step's gradient all-reduce
        self.last_summaries = {}
        self._per = bool(getattr(conf, "use_prioritized_replay", False))
        self._priority_signal = None  # (starts, per-transition critic loss, is_contiguous) of the batch get_losses last saw

    def close(self):
        """Drop the captured step graphs.  Call before torch.distributed.destroy_process_group(): a CUDA graph that captured the
        gradient all-reduce keeps NCCL work alive and can block the communicator's teardown."""
        self._graphs.clear()
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def enable_training(self, replays):
        """deepQlearning.py:64-71,96-103: register the read heads (already device loaders)."""
        self.replays = list(replays)

    @staticmethod
    def _temporal_difference_shift(xp):
        curr, nxt = {}, {}
        for k, v in xp.items():
            curr[k], nxt[k] = v[:-1], v[1:]
        return curr, nxt

    def get_losses(self, xp, parts=False):
        """deepQlearning.py:198-249.  `xp` is a sampled [T, B, .] dict; it is mutated like in the reference (mask,
        is_contiguous, state).  When the gather kernel already emitted mask / is_contiguous (aux=True) they are used as is.
        `parts=True` (folded reduce only) returns (critic part, actor + temperature part) of the same scalar: their backward passes
        touch disjoint parameters, which `_one_update` uses to overlap the critic gradients' all-reduce with the actor's backward.
        A prioritized batch (`is_weight` [B] and `starts` [B] in xp) weights the CRITIC loss of window b by is_weight[b], in the folded
        path (grad_scale of the loss kernel) and the unfolded one alike; the actor and temperature losses keep the uniform reduce
        weights.  The critic's per-transition loss is kept for update_priorities."""
        conf = self.conf
        is_w, starts = xp.pop("is_weight", None), xp.pop("starts", None)
        if "mask" not in xp:
            xp["mask"] = torch.logical_not(xp["task_done"] != 0).to(xp["task_done"].dtype)
        if "is_contiguous" not in xp:
            step = xp["episode_step"]
            xp["is_contiguous"] = ((step[1:] == step[:-1] + 1) & (xp["mask"][:-1] != 0)).to(step.dtype)
        is_contiguous = xp.pop("is_contiguous")
        weight = xp.pop("loss_weight", None)
        if getattr(conf, "discrete", False):  # :206-210 one-hot of the stored action index (fdql_action_onehot)
            from .. import ops
            xp["action_onehot"] = ops.action_onehot(xp["action"], conf.action_space.n)
        xp["state"] = self.encoder.forward_train(xp)
        curr, nxt = self._temporal_difference_shift(xp)
        bootstrap = getattr(conf, "use_bootstrap_minibatch_nstep", False) and conf.use_nStep_lowerbounds
        if weight is not None and not bootstrap and getattr(conf, "fold_loss_reduce", True):
            # :222-225,249 folded into the loss kernel: the gather kernel's aux weight contig / ((sum_t contig + 1e-4) B T) goes in as
            # grad_scale, so d loss / d q_pred leaves the kernel already reduced and the scalar is sum(weight * per-transition loss)
            if is_w is None:
                q_sum, summ = self.actor_critic.q_loss_reduced(curr, nxt, weight)
            else:
                q_sum, summ, q_each = self.actor_critic.q_loss_reduced(curr, nxt, weight * is_w.view(1, -1, 1), with_loss=True)
                self._priority_signal = (starts, q_each, is_contiguous)
            pi_loss, alpha_loss, asumm = self.actor_critic.actor_loss(curr)
            self.last_summaries = {**summ, **asumm, "Valid_Portion": is_contiguous.mean()}
            if parts:
                return q_sum, ((pi_loss + alpha_loss) * weight).sum()
            return q_sum + ((pi_loss + alpha_loss) * weight).sum()
        if parts:
            if is_w is not None:
                xp["is_weight"], xp["starts"] = is_w, starts  # for the unsplit call that follows
            return None
        q_loss, bound, summ = self.actor_critic.q_loss(curr, nxt)
        pi_loss, alpha_loss, asumm = self.actor_critic.actor_loss(curr)
        if is_w is not None:
            self._priority_signal = (starts, q_loss.detach(), is_contiguous)
            q_loss = q_loss * is_w.view(1, -1, 1)
        loss = ((q_loss + pi_loss + alpha_loss) * is_contiguous).sum(0) / (is_contiguous.sum(0) + 1e-4)   # :222-225
        loss = loss.mean()
        if bootstrap:                                                                                   # :226-228
            loss = loss + (bound * is_contiguous.prod(0)).mean()
        self.last_summaries = {**summ, **asumm, "Valid_Portion": is_contiguous.mean()}
        return loss / conf.temporal_len                                                                # :249

    def _allreduce_grads(self, params=None, bucket=0):
        """Mean of the gradients over the ranks: one flat bucket, one all-reduce (`params`: a subset with its own bucket)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        grads = [p.grad for p in (self.params if params is None else params) if p.grad is not None]
        if not grads:
            return
        n = sum(g.numel() for g in grads)
        if not isinstance(self._flat, dict):
            self._flat = {}
        if bucket not in self._flat or self._flat[bucket].numel() != n:
            self._flat[bucket] = torch.empty(n, dtype=grads[0].dtype, device=grads[0].device)
        flat = self._flat[bucket]
        torch._foreach_copy_(list(flat.split([g.numel() for g in grads])), [g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.div_(dist.get_world_size())
        torch._foreach_copy_([g.reshape(-1) for g in grads], list(flat.split([g.numel() for g in grads])))

    def _one_update(self, replay, **sample_kw):
        """sample -> loss -> backward -> gradient all-reduce -> Adam -> targets.  Under torch.distributed the all-reduce runs on a
        side stream while the main stream already samples and relabels the NEXT step's batch (SURVEY.md section 5: the only
        collective of the path hides behind work that does not depend on it); the prefetched batch is consumed by the next call."""
        key = id(replay)
        if self._per:
            sample_kw.setdefault("prioritized", True)
        xp = self._prefetched.pop(key, None)
        if xp is None:
            xp = replay.temporal_sample(**sample_kw)
        overlap = self._world_size() > 1 and getattr(self.conf, "overlap_allreduce", True)
        split = None
        sb = getattr(self.conf, "split_backward", True)  # True: with the overlapped all-reduce; "force": always (tests); False: never
        if ((overlap and sb) or sb == "force") and self.device.type == "cuda" and not any(p.requires_grad for p in self.encoder.parameters()):
            split = self.get_losses(xp, parts=True)  # None when the reduce is not folded (then: one backward, one bucket)
            if split is not None:
                self._feed_priorities(replay)
        if split is not None:
            # critic gradients first; their all-reduce (most of the bytes) runs on the side stream under the actor's backward
            q_part, pi_part = split
            cur = torch.cuda.current_stream(self.device)
            if self._side is None:
                self._side = torch.cuda.Stream(self.device)
            if self._buckets is None:
                crit = [p for p in self.actor_critic.critic.parameters() if p.requires_grad]
                ids = {id(p) for p in crit}
                self._buckets = (crit, [p for p in self.params if id(p) not in ids and p.requires_grad])
            crit, rest = self._buckets
            torch.autograd.backward(q_part, inputs=crit)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self._allreduce_grads(crit, bucket=1)
            torch.autograd.backward(pi_part, inputs=rest)
            loss = q_part.detach() + pi_part.detach()
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self._allreduce_grads(rest, bucket=2)
            self._prefetched[key] = replay.temporal_sample(**sample_kw)
            cur.wait_stream(self._side)
            if self.conf.clip_grad_norm:
                torch.nn.utils.clip_grad_norm_(self.params, self.conf.clip_grad_norm)
            self.optimizer.step()
            self.actor_critic.update_target()
            return loss
        loss = self.get_losses(xp)
        self._feed_priorities(replay)
        loss.backward()
        if overlap:
            cur = torch.cuda.current_stream(self.device)
            if self._side is None:
                self._side = torch.cuda.Stream(self.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self._allreduce_grads()
            # backward has consumed the current batch (stream order), so the same output buffers can take the next one
            self._prefetched[key] = replay.temporal_sample(**sample_kw)
            cur.wait_stream(self._side)
        else:
            self._allreduce_grads()
        if self.conf.clip_grad_norm:
            torch.nn.utils.clip_grad_norm_(self.params, self.conf.clip_grad_norm)
        self.optimizer.step()
        self.actor_critic.update_target()
        return loss.detach()

    def _feed_priorities(self, replay):
        """update_priorities from the critic loss of the batch just consumed, enqueued before the next batch (or the prefetch) is drawn."""
        if self._priority_signal is None:
            return
        starts, q_each, contig = self._priority_signal
        self._priority_signal = None
        replay.update_priorities(starts, q_each, contig)

    def per_beta(self):
        """Importance-sampling exponent of the current update: per_beta0 annealed linearly to 1 over per_beta_steps updates."""
        c = self.conf
        frac = min(1.0, self.train_steps / max(1, int(c.per_beta_steps)))
        return float(c.per_beta0) + (1.0 - float(c.per_beta0)) * frac

    @staticmethod
    def _ring_of(replay):
        """The ReplayMemory under a read head's wrappers."""
        ring = replay
        while hasattr(ring, "replay_buffer") or (hasattr(ring, "replay") and not hasattr(ring, "flush")):
            ring = getattr(ring, "replay_buffer", None) or ring.replay
        return getattr(ring, "replay", ring)

    @staticmethod
    def _world_size():
        import torch.distributed as dist
        return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1

    def train_step(self):
        """deepQlearning.py:105-127: for each local shard: sample -> loss -> backward -> (all-reduce) -> Adam -> targets."""
        last = None
        for i, replay in enumerate(self.replays):
            if self._per:
                self._ring_of(replay).set_priority_beta(self.per_beta())  # device scalar: read by the sampler, eager or replayed
            if getattr(self.conf, "use_cuda_graph", False):
                last = self._graphed_update(i, replay)
            else:
                self.optimizer.zero_grad(set_to_none=False)
                last = self._one_update(replay)
            self.train_steps += 1
        return last

    # ---- whole-step CUDA graph (SURVEY.md section 8f rank 2): sample/relabel kernel, MLP forward/backward, fused loss, Adam and
    #      the target update are captured once and replayed; the draw counter and the temperature live in device memory.
    def _graphed_update(self, i, replay):
        ring = self._ring_of(replay)
        ring.flush()
        n_now = len(ring)
        entry = self._graphs.get(i)
        if entry is None:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and not getattr(self.conf, "graph_allreduce", False):
                raise RuntimeError("use_cuda_graph with world_size > 1 needs conf.graph_allreduce=True (NCCL capture)")
            if self.conf.clip_grad_norm:
                raise RuntimeError("clip_grad_norm is not capturable")
            ring.device_counter = True  # draw counter AND ring length are read from device memory: one capture serves a filling ring
            ring.publish_len()
            ring.apply_pending_priorities()  # rows recorded since the last PER call: applied outside the graph, never captured
            cur = torch.cuda.current_stream(self.device)
            side = torch.cuda.Stream(self.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(3):  # warm-up on a side stream (allocator, autograd buffers, Adam state)
                    self.optimizer.zero_grad(set_to_none=True)
                    self._one_update(replay, reuse_outputs=True)
            cur.wait_stream(side)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            self.optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(graph):
                static_loss = self._one_update(replay, reuse_outputs=True)
            entry = (graph, static_loss, n_now)
            self._graphs[i] = entry
        ring.publish_len()  # (a no-op unless rows were added since the last step)
        ring.apply_pending_priorities()
        entry[0].replay()
        return entry[1]
