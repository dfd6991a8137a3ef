#!/usr/bin/env python
"""End-to-end use of the drop-in path on the reference's HER showcase task (franQ/Env/bitflip.py: flip one bit per step until the
state equals the goal; reward -1 until then): vectorised numpy bit-flip envs -> `Replay.make` write heads (device ring, episode
commit, link records) -> `Learner.train_step` (sample-time "future" hindsight relabelling, fused TQC loss, discrete Gumbel-softmax
actor with the one-hot kernel, whole step as a CUDA graph).  Prints the greedy success rate as it trains.

With --torch-reward the reward is the bit-flip function written in PyTorch (a TorchReward) instead of the device functor, and
hindsight relabelling moves to write time (her_mode "random": one relabelled copy of every episode, made when it is flushed),
because sample-time relabelling evaluates the reward inside the gather kernels.

    python examples/train_bitflip_her.py --bits 10 --updates 4000 [--per] [--torch-reward]
"""
import argparse
import os
import sys
import time
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastdeepqlearning_b200 as fdql  # noqa: E402
from fastdeepqlearning_b200 import Agent, Replay  # noqa: E402


def rollout(actor, n_envs, bits, horizon, device, greedy, rng, eps=0.0):
    """Batch of bit-flip episodes; returns the per-row dicts of every env (time-major) and the success flags."""
    state = rng.integers(0, 2, (n_envs, bits)).astype(np.float32)
    goal = rng.integers(0, 2, (n_envs, bits)).astype(np.float32)
    rows = [[] for _ in range(n_envs)]
    alive = np.ones(n_envs, bool)
    success = np.zeros(n_envs, bool)
    solved = (state == goal).all(-1)
    reward = np.zeros(n_envs, np.float32)  # env_handler.py:38: the reset row carries reward 0
    for t in range(horizon + 1):
        obs = torch.as_tensor(np.concatenate([state, state, goal], -1), device=device)
        with torch.no_grad():
            a_onehot, _, logits = actor(obs)
        act = (logits.argmax(-1) if greedy else a_onehot.argmax(-1)).cpu().numpy()
        if eps > 0:  # a little uniform exploration on top of the policy's own sampling
            rnd = rng.random(n_envs) < eps
            act = np.where(rnd, rng.integers(0, bits, n_envs), act)
        done = solved | (t == horizon)
        for e in np.nonzero(alive)[0]:
            rows[e].append({"obs_1d": state[e].copy(), "achieved_goal": state[e].copy(), "desired_goal": goal[e].copy(),
                            "action": float(act[e]), "reward": float(reward[e]), "task_done": bool(solved[e] and t > 0),
                            "episode_done": bool(done[e]), "episode_step": t})
        success |= alive & solved
        alive &= ~done
        if not alive.any():
            break
        idx = np.nonzero(alive)[0]  # finished envs stay where they ended
        state[idx, act[idx]] = 1 - state[idx, act[idx]]
        solved = (state == goal).all(-1)
        reward = np.where(solved, 0.0, -1.0).astype(np.float32)
    return rows, success


def bitflip_reward(achieved_goal, goal):
    """franQ/Env/bitflip.py:143-152 in PyTorch, batched over rows: reward 0 when every bit matches, else -1; done on a match."""
    hit = (achieved_goal == goal).all(-1)
    return hit.float() - 1.0, hit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bits", type=int, default=10)
    ap.add_argument("--updates", type=int, default=4000)
    ap.add_argument("--envs", type=int, default=64)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--eps", type=float, default=0.2)
    ap.add_argument("--per", action="store_true", help="prioritized replay (use_prioritized_replay=True)")
    ap.add_argument("--torch-reward", action="store_true", help="reward as a TorchReward, write-time hindsight (her_mode='random')")
    args = ap.parse_args()
    device = torch.device("cuda:0")
    rng = np.random.default_rng(0)
    torch.manual_seed(0)
    bits, horizon = args.bits, 2 * args.bits
    conf = Agent.LearnerConf(training_device="cuda:0", obs_space={"obs_1d": bits, "achieved_goal": bits, "desired_goal": bits},
                             action_space=types.SimpleNamespace(n=bits, shape=()), discrete=True, num_critics=5, num_q_predictions=10,
                             top_quantiles_to_drop=0.2, batch_size=args.batch, temporal_len=2, replay_size=200_000, use_HER=True,
                             her_mode="random" if args.torch_reward else "future", num_instances=1, gamma=0.98, learning_rate=1e-3, use_cuda_graph=True,
                             use_prioritized_replay=args.per, per_beta_steps=args.updates)
    reward = fdql.TorchReward(bitflip_reward) if args.torch_reward else fdql.RewardOp.bitflip()
    read, write = Replay.make(conf, compute_reward=reward)
    learner = Agent.Learner(conf, read)
    actor = learner.actor_critic.actor
    t0, updates = time.time(), 0
    while updates < args.updates:
        rows, _ = rollout(actor, args.envs, bits, horizon, device, greedy=False, rng=rng, eps=args.eps)
        for ep in rows:
            for r in ep:
                write[0].add(r)
        if len(read[0]) < 4 * args.batch:
            continue
        for _ in range(40):
            learner.train_step()
        updates += 40
        if updates % 400 == 0:
            _, ok = rollout(actor, 256, bits, horizon, device, greedy=True, rng=np.random.default_rng(1))
            print(f"updates {updates:5d}  ring {len(read[0]):6d} rows  greedy success {ok.mean():.2f}  ({time.time() - t0:.0f} s)", flush=True)
    return float(ok.mean())


if __name__ == "__main__":
    main()
