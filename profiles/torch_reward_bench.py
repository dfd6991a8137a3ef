"""Write-time hindsight flush rate: the bit-flip reward as the device functor (RewardOp.bitflip) against the same function written in
PyTorch (TorchReward), which adds a goal gather and one torch call per flush and loads the results in the flush kernel.

Two numbers per variant, 128-step episodes with 64-bit goals:
  * flush: `ReplayMemory.add_hindsight_rows` over episodes already in the ring, 1 or 64 episodes per call, relabelled rows per
    second of wall time with a device synchronise at the end of each timed batch of calls;
  * write path: rows per second through `Replay.make(her_mode="random")` write heads fed one row dict at a time (what a runner does),
    stored rows (real + relabelled) per second.
The variants alternate within each round; the script prints the median and spread of the rounds and the card's name and power limit,
read in the same run.

    python profiles/torch_reward_bench.py [--rounds 5] [--out torch_reward_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastdeepqlearning_b200 as fdql  # noqa: E402
from fastdeepqlearning_b200 import Replay  # noqa: E402

L_EP, G, OBS, ACT, GAMMA = 128, 64, 64, 8, 0.98


def bitflip_torch(ag, g):
    hit = (ag == g).all(-1)
    return hit.float() - 1.0, hit


def rewards():
    return {"enum": fdql.RewardOp.bitflip(), "torch": fdql.TorchReward(bitflip_torch)}


def episode_cols(rng, n_eps):
    N = n_eps * L_EP
    ag = rng.integers(0, 2, (N, G)).astype(np.float32)
    dg = np.repeat(rng.integers(0, 2, (n_eps, G)).astype(np.float32), L_EP, 0)
    hit = (ag == dg).all(-1, keepdims=True).astype(np.float32)
    step = (np.arange(N) % L_EP).astype(np.float32).reshape(-1, 1)
    return {"obs_1d": rng.standard_normal((N, OBS)).astype(np.float32), "action": rng.uniform(-1, 1, (N, ACT)).astype(np.float32),
            "achieved_goal": ag, "desired_goal": dg, "reward": hit - 1, "task_done": hit,
            "episode_done": (step == L_EP - 1).astype(np.float32), "episode_step": step, "mc_return": np.zeros((N, 1), np.float32)}


def flush_rate(reward, eps_per_call, calls, src_eps=64):
    """Relabelled rows per second of add_hindsight_rows; the hindsight copies go to the ring after the source episodes."""
    cap = src_eps * L_EP + (calls + 3) * eps_per_call * L_EP + 1
    ring = Replay.ReplayMemory(cap, 256, 2)
    ring.set_reward_op(reward, GAMMA)
    begin = ring.add_rows(episode_cols(np.random.default_rng(0), src_eps), episode_lengths=[L_EP] * src_eps, with_returns=True)
    rng = np.random.default_rng(1)

    def call():
        e = rng.integers(0, src_eps, eps_per_call)
        src = [(begin + int(i) * L_EP) % cap for i in e]
        goal = [(s + int(rng.integers(0, L_EP))) % cap for s in src]
        ring.add_hindsight_rows(src, [L_EP] * eps_per_call, goal, with_returns=True)
    for _ in range(3):  # warm-up: module load, allocator, torch kernels
        call()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        call()
    torch.cuda.synchronize()
    return calls * eps_per_call * L_EP / (time.perf_counter() - t0)


def write_path_rate(reward, n_eps):
    conf = types.SimpleNamespace(replay_size=4 * n_eps * L_EP, batch_size=256, temporal_len=2, num_instances=1, use_nStep_lowerbounds=True,
                                 nStep_return_steps=1000, gamma=GAMMA, use_squashed_rewards=False, use_HER=True, her_mode="random",
                                 training_device="cuda:0")
    _, write = Replay.make(conf, compute_reward=reward)
    cols = episode_cols(np.random.default_rng(2), n_eps + 2)
    keys = [k for k in cols if k != "mc_return"]
    rows = [{k: (cols[k][i] if cols[k].shape[1] > 1 else float(cols[k][i, 0])) for k in keys} for i in range((n_eps + 2) * L_EP)]
    for r in rows[:2 * L_EP]:  # warm-up: two episodes
        write[0].add(r)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r in rows[2 * L_EP:]:
        write[0].add(r)
    torch.cuda.synchronize()
    return 2 * n_eps * L_EP / (time.perf_counter() - t0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--write-eps", type=int, default=64, help="episodes per write-path measurement")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("torch_reward_bench.py measures on a CUDA device; none is visible")
    fdql.lib()
    cases = [("flush_1ep", lambda r: flush_rate(r, 1, 200)), ("flush_64ep", lambda r: flush_rate(r, 64, 20)),
             ("write_path", lambda r: write_path_rate(r, args.write_eps))]
    res = {c: {v: [] for v in ("enum", "torch")} for c, _ in cases}
    for i in range(args.rounds):
        for c, fn in cases:
            order = ("enum", "torch") if i % 2 == 0 else ("torch", "enum")
            for v in order:
                res[c][v].append(fn(rewards()[v]))
    out = {"card": card(), "episode_len": L_EP, "goal_bits": G, "rounds": args.rounds, "unit": "rows/s"}
    for c in res:
        out[c] = {v: {"median": statistics.median(x), "min": min(x), "max": max(x)} for v, x in res[c].items()}
        out[c]["torch_over_enum"] = out[c]["torch"]["median"] / out[c]["enum"]["median"]
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
