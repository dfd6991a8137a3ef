#!/usr/bin/env python
"""Prioritized replay on the bench.py workload (1e7-row ring, obs 64, act 8, goal 16+16, T = 2, B = 4096): one JSON line with

  per_sample_ms / per_update_ms   one fdql_per_sample (4096 windows, hindsight streams, IS weights) and one fdql_per_update (4096
                                  windows), CUDA events over 20 replays of a graph holding 50 launches (launch gaps excluded);
  updates_per_s                   whole learner steps (bench.py's second metric, the step captured in one CUDA graph) with PER off and
                                  on, in the same process, alternated;
  pass                            64 x 4096 windows: the uniform fused pass (fdql_fused_pass, bench.py's headline) beside a PER pass
                                  as four launches (fdql_per_sample + injected fdql_sample_gather + fdql_tqc_loss + fdql_per_update),
                                  graphed, and the four launches timed one by one (`split_ms`);
  fused_per                       the same 64 x 4096 windows through fdql_fused_pass_per (prioritized draw in the gather role, update
                                  after the launch) against the uniform fused pass, alternated in one run: median and spread over repeats.

The card name, its power limit and the SM clock are read in the same run: the numbers belong to that card at that limit.
    python profiles/per_bench.py [--ring-rows 10000000] [--split-only]   (--split-only: the four-launch split alone, which every
                                                                          build with fdql_per_* can run)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload constants and the synthetic ring)


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"], out["sm_mhz_now"] = float(q[0]), float(q[1]), float(q[2])
    except Exception as e:  # the numbers stand without it, but say so
        out["power_limit_w"] = f"unavailable: {e}"
    return out


def graph_ms(torch, fn, per_graph=50, reps=20):
    """ms per fn() call: fn captured per_graph times in one graph, replayed reps times between CUDA events."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (per_graph * reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ring-rows", type=int, default=10_000_000)
    ap.add_argument("--passes", type=int, default=64, help="batches of 4096 windows per pass")
    ap.add_argument("--updates", type=int, default=60)
    ap.add_argument("--split-only", action="store_true", help="only the per-launch split of the four-launch PER pass")
    ap.add_argument("--repeats", type=int, default=7, help="alternations of the uniform and the prioritized fused pass")
    args = ap.parse_args()
    import torch
    import fastdeepqlearning_b200 as pkg
    from fastdeepqlearning_b200 import Agent, Replay, _lib as L
    from fastdeepqlearning_b200.Replay.wrappers import SampleTimeHindsight
    if not torch.cuda.is_available():
        raise SystemExit("per_bench.py needs a CUDA device")
    lib = pkg.lib()
    dev = torch.device("cuda:0")
    B, T, CQ = bench.B, bench.T, bench.CQ
    ring = bench.build_ring(torch, pkg, Replay, args.ring_rows, dev, seed=1234)
    ring.enable_priorities(alpha=0.6, eps=1e-6, eta=0.9)
    ring.device_counter = True
    ring.publish_len()
    ring.apply_pending_priorities()
    res = {"metric": "prioritized replay overhead", "card": card(), "ring_rows": len(ring), "batch": B, "T": T}
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None

    # ---- sample / update kernels alone
    st = torch.empty(B, dtype=torch.int64, device=dev)
    fl = torch.empty(B, dtype=torch.uint8, device=dev)
    go = torch.empty(B, dtype=torch.int64, device=dev)
    w = torch.empty(B, device=dev)
    loss = torch.rand(T - 1, B, device=dev) * 3

    def sample():
        L.check(lib.fdql_per_sample(ring._per, B, L.GOAL_FUTURE, bench.P_RELABEL, 7, 0, p(ring._rng_counter_dev), None, p(ring._per_beta),
                                    p(st), p(fl), p(go), p(w), C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    def update():
        L.check(lib.fdql_per_update(ring._per, B, p(st), p(loss), None, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    if not args.split_only:
        res["per_sample_ms"] = graph_ms(torch, sample)
        res["per_update_ms"] = graph_ms(torch, update)
        learner_rates(torch, Agent, SampleTimeHindsight, ring, args, res)
    pass_rates(torch, lib, L, ring, args, res, p)
    res["card_after"] = card()
    print(json.dumps(res))


def learner_rates(torch, Agent, SampleTimeHindsight, ring, args, res):
    B, T, CQ = bench.B, bench.T, bench.CQ

    # ---- learner updates/s, PER off and on, alternated
    def learner(per):
        torch.manual_seed(0)
        conf = Agent.LearnerConf(training_device="cuda:0", obs_space={"obs_1d": bench.OBS, "achieved_goal": bench.GOAL, "desired_goal": bench.GOAL},
                                 action_space=types.SimpleNamespace(shape=(bench.ACT,)), num_critics=bench.C_CRIT,
                                 num_q_predictions=bench.Q_ATOMS, top_quantiles_to_drop=bench.N_DROP / CQ + 1e-9, batch_size=B, temporal_len=T,
                                 gamma=bench.GAMMA, use_cuda_graph=True, use_prioritized_replay=per)
        lr = Agent.Learner(conf, [SampleTimeHindsight(ring, relabel_prob=bench.P_RELABEL)])
        for _ in range(5):
            lr.train_step()
        return lr
    learners = {False: learner(False), True: learner(True)}
    ms = {False: [], True: []}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(6):
        for per in (False, True):
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.updates // 6):
                learners[per].train_step()
            e1.record()
            torch.cuda.synchronize()
            ms[per].append(e0.elapsed_time(e1) / (args.updates // 6))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    res["learner"] = {"uniform_ms_per_update": med[False], "per_ms_per_update": med[True], "uniform_updates_per_s": 1e3 / med[False],
                      "per_updates_per_s": 1e3 / med[True], "per_overhead_pct": 100 * (med[True] / med[False] - 1),
                      "spread_ms": {"uniform": [min(ms[False]), max(ms[False])], "per": [min(ms[True]), max(ms[True])]}}
    del learners


def pass_rates(torch, lib, L, ring, args, res, p):
    B, T, CQ = bench.B, bench.T, bench.CQ
    dev = torch.device("cuda:0")
    # ---- a pass of 64 x 4096 windows: uniform fused pass vs PER pass
    n = args.passes * B
    M = (T - 1) * n
    keys = ring.keys
    gen = torch.Generator(device=dev).manual_seed(99)
    z = torch.randn(M, CQ, device=dev, generator=gen) * 3
    q = torch.randn(M, CQ, device=dev, generator=gen) * 3
    lp = torch.randn(M, device=dev, generator=gen)
    out = {k: torch.empty((T, n, wd), device=dev) for k, wd in zip(keys, ring._widths)}
    outp = L.ptr_array([out[k].data_ptr() for k in keys])
    mask, contig, weight = torch.empty(T, n, device=dev), torch.empty(T - 1, n, device=dev), torch.empty(T - 1, n, device=dev)
    sts, fls, gos = torch.empty(n, dtype=torch.int64, device=dev), torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.int64, device=dev)
    isw = torch.empty(n, device=dev)
    ploss, grad = torch.empty(M, device=dev), torch.empty(M, CQ, device=dev)
    stats = torch.zeros(4, dtype=torch.float64, device=dev)
    params, n_params = ring.reward_op.c_params()
    opts = L.OPT_EMIT_LEARNER_AUX | L.OPT_EXACT_EPISODE_STEP
    sp = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ctr = torch.zeros(4, dtype=torch.int64, device=dev)

    # the fused kernel's halves must not alias: its gather writes a second buffer set while its loss reads the first
    out2 = {k: torch.empty_like(v) for k, v in out.items()}
    outp2 = L.ptr_array([out2[k].data_ptr() for k in keys])
    mask2, contig2, weight2 = torch.empty_like(mask), torch.empty_like(contig), torch.empty_like(weight)

    def fused():  # loss of one batch + gather of the next in one launch: the steady state of bench.py's schedule
        L.check(lib.fdql_fused_pass(ring._h, n, T, L.GOAL_FUTURE, bench.P_RELABEL, 7, 0, p(ctr), p(sts), p(fls), p(gos), ring.reward_op.op,
                                    params, n_params, bench.GAMMA, opts, B, outp2, p(mask2), p(contig2), p(weight2), M, CQ, bench.N_DROP, p(z),
                                    p(q), p(lp), p(out["reward"][1:]), p(mask[1:]), p(out["mc_return"][1:]), p(weight), bench.ALPHA,
                                    bench.GAMMA, p(ploss), p(grad), p(stats), sp()))

    def per_pass():
        L.check(lib.fdql_per_sample(ring._per, n, L.GOAL_FUTURE, bench.P_RELABEL, 7, 0, p(ctr), None, p(ring._per_beta), p(sts), p(fls), p(gos),
                                    p(isw), sp()))
        L.check(lib.fdql_sample_gather(ring._h, n, T, ring._maxlen, p(sts), p(fls), p(gos), ring.reward_op.op, params, n_params, bench.GAMMA,
                                       opts, B, outp, p(mask), p(contig), p(weight), sp()))
        L.check(lib.fdql_tqc_loss(M, CQ, bench.N_DROP, p(z), p(q), p(lp), p(out["reward"][1:]), p(mask[1:]), p(out["mc_return"][1:]),
                                  p(weight), bench.ALPHA, bench.GAMMA, p(ploss), p(grad), None, p(stats), sp()))
        L.check(lib.fdql_per_update(ring._per, n, p(sts), p(ploss), p(contig), sp()))
    t_per = graph_ms(torch, per_pass, per_graph=10, reps=10)  # (also leaves a gathered batch in the first set for the fused loss)
    t_fused = graph_ms(torch, fused, per_graph=10, reps=10)
    # the four launches of the PER pass one by one (each graphed alone; the inputs are those the pass above left)

    def l_sample():
        L.check(lib.fdql_per_sample(ring._per, n, L.GOAL_FUTURE, bench.P_RELABEL, 7, 0, p(ctr), None, p(ring._per_beta), p(sts), p(fls), p(gos),
                                    p(isw), sp()))

    def l_gather():
        L.check(lib.fdql_sample_gather(ring._h, n, T, ring._maxlen, p(sts), p(fls), p(gos), ring.reward_op.op, params, n_params, bench.GAMMA,
                                       opts, B, outp, p(mask), p(contig), p(weight), sp()))

    def l_loss():
        L.check(lib.fdql_tqc_loss(M, CQ, bench.N_DROP, p(z), p(q), p(lp), p(out["reward"][1:]), p(mask[1:]), p(out["mc_return"][1:]),
                                  p(weight), bench.ALPHA, bench.GAMMA, p(ploss), p(grad), None, p(stats), sp()))

    def l_update():
        L.check(lib.fdql_per_update(ring._per, n, p(sts), p(ploss), p(contig), sp()))
    split = {name: graph_ms(torch, fn, per_graph=10, reps=10) for name, fn in
             (("per_sample", l_sample), ("sample_gather", l_gather), ("tqc_loss", l_loss), ("per_update", l_update))}
    res["pass"] = {"windows": n, "uniform_fused_ms": t_fused, "per_ms": t_per, "uniform_fused_transitions_per_s": M / t_fused * 1e3,
                   "per_transitions_per_s": M / t_per * 1e3, "split_ms": split,
                   "note": "the uniform pass fuses loss k with gather k+1 in one launch; the PER pass is four launches in stream order, "
                           "the gather as the injected-stream kernel"}
    if args.split_only or not hasattr(lib, "fdql_fused_pass_per"):
        return

    # ---- fdql_fused_pass_per: loss + update of one batch, prioritized gather of the next, against the uniform fused pass, alternated.
    # Call k reads batch k's set (critic weight as grad_scale, starts and is_contiguous for the update) and writes batch k+1's set.
    isw2, crit, crit2 = torch.empty_like(isw), torch.empty_like(weight), torch.empty_like(weight)
    sts2 = torch.empty_like(sts)
    crit.copy_(weight)

    def fused_per():
        L.check(lib.fdql_fused_pass_per(ring._per, n, L.GOAL_FUTURE, bench.P_RELABEL, 7, 0, p(ctr), None, p(ring._per_beta), p(sts2), p(fls),
                                        p(gos), p(isw2), p(crit2), ring.reward_op.op, params, n_params, bench.GAMMA, opts, B, outp2, p(mask2),
                                        p(contig2), p(weight2), M, CQ, bench.N_DROP, p(z), p(q), p(lp), p(out["reward"][1:]), p(mask[1:]),
                                        p(out["mc_return"][1:]), p(crit), bench.ALPHA, bench.GAMMA, p(ploss), p(grad), p(stats), p(sts),
                                        p(contig), sp()))
    ms = {"uniform": [], "per": []}
    for _ in range(args.repeats):
        ms["uniform"].append(graph_ms(torch, fused, per_graph=10, reps=10))
        ms["per"].append(graph_ms(torch, fused_per, per_graph=10, reps=10))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    res["fused_per"] = {"windows": n, "uniform_fused_ms": med["uniform"], "per_fused_ms": med["per"], "ratio": med["per"] / med["uniform"],
                        "per_fused_transitions_per_s": M / med["per"] * 1e3,
                        "spread_ms": {k: [min(v), max(v)] for k, v in ms.items()}, "repeats": args.repeats,
                        "note": "per_fused_ms = the fused launch (loss k + prioritized gather k+1) plus the priority update of batch k"}


if __name__ == "__main__":
    main()
