#!/usr/bin/env python
"""bench.py -- sampled+relabelled+targeted transitions/s of the B200 learner hot path (BASELINE.json metric).

One pass of the hot path = `batches_per_step` batches of 4096 sampled windows (T=2, one TD pair per window):
  fdql_sample_gather_draw  (uniform starts, hindsight flag p=0.8 = "future, k=4", goal row drawn in the kernel   [sampled]
                            + window gather + sample-time HER relabel + reward and return recompute;            [relabelled]
                            --separate-streams: fdql_sample_streams + fdql_sample_gather, two launches)
  fdql_tqc_loss        (pool 5x25 target atoms, sort, drop 10, soft target, quantile-Huber fwd+bwd,
                        n-step lower bound) on synthetic critic outputs resident in HBM             [targeted]
on a 1e7-row ring (obs 64, act 8, goal 16+16, 5 scalars; fp32).  One step = `passes_per_step` such passes, so that the timed
region of a 20-step run is about half a second.  By default the passes are pipelined the way the reference pipelines sampling
and training (torch_dataloader.py:22-39: a prefetch thread keeps one sampled batch ahead of the learner): ONE launch per pass,
fdql_fused_pass, whose loss role (16 warps per SM) works on pass k while its gather role (8 warps per SM) samples, relabels and
gathers pass k+1 into the other batch buffer; every pass is complete inside the timed region (K gathers and K losses: the first
launch of a step is a gather alone, the last one a loss alone).  --two-streams is the round-2a schedule (the gather of pass k+1 on
a second stream, two small co-resident blocks per SM, under the loss kernel of pass k); --serial runs the two kernels back to back.
`value` is device-timed with everything resident in HBM; `e2e` is the same pass through the host-buffer C-ABI call
fdql_hotpath_step_host (index streams and critic outputs from pinned host memory, loss and dloss/dq back to host memory).
`--impl reference` times the CPU restatement of the reference path (oracle/, numpy + torch-CPU, all host cores) on a bounded
sample of the same workload.

Launch: python bench.py [--gpus N --steps K --warmup W]; for N>1 under torchrun (one rank per GPU, no data-path
collective: the replay shards by actor stream, scaling = weak)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OBS, ACT, GOAL, LEP = 64, 8, 16, 128
B, T, C_CRIT, Q_ATOMS, N_DROP = 4096, 2, 5, 25, 10
CQ = C_CRIT * Q_ATOMS
GAMMA, ALPHA, P_RELABEL = 0.99, 1.0, 0.8
ROW_BYTES = 4 * (OBS + ACT + 2 * GOAL) + 4 * 5  # 436 B, SURVEY.md section 8(d)

# algorithmic bytes per transition (T=2), SURVEY.md section 8(d) / DESIGN.md:
#   A gather: read 2 rows + 8 B start, write 2 rows                         = 4*436 + 8       = 1752
#   B relabel: goal source row 4*G + its scan record 16 + goal_row(8) + flag(1) = 64 + 25      =   89   (x p)
#   C return under relabel: n tail rows x one 16-byte scan record (64-bit goal hash, goal-agnostic reward, NaN flag);
#     mean tail of a uniform start in a 128-row episode = 64.5 rows         = 16 * 64.5       = 1032   (x p)
#     (SURVEY.md 8(d) counts 72*n B for this term, reading the goal vectors themselves: 4644 B.  The hash-assisted scan
#      is exact -- hash matches are verified on the full vectors -- and moves 4.5x fewer bytes; the roofline below uses
#      the bytes THIS algorithm needs, and `survey_bytes_per_transition` reports the SURVEY figure beside it.)
#   D TQC: next_z + q_pred + grad_q (3 x 4*125) + 4 scalars in + loss out   = 1500 + 20       = 1520
BYTES_GATHER = 4 * ROW_BYTES + 8
BYTES_RELABEL_SCAN = P_RELABEL * ((4 * GOAL + 25) + 16 * (LEP + 1) / 2)  # --tail-scan: 16 B scan record per tail row
BYTES_RELABEL = P_RELABEL * ((4 * GOAL + 25) + 16 * T)  # goal row + its link record + streams + one link record per window row
BYTES_RELABEL_SURVEY = P_RELABEL * ((4 * GOAL + 5) + 72 * (LEP + 1) / 2)
BYTES_TQC = 3 * 4 * CQ + 20
BYTES_STREAMS = 32 + 17  # read the start row's record sector, write start/flag/goal


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ring-rows", type=int, default=10_000_000)
    ap.add_argument("--batches-per-step", type=int, default=64)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-batches", type=int, default=0, help="bounded CPU-baseline sample, 0 = auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-small", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the T=50 figure (reference default temporal_len, SURVEY 8)")
    ap.add_argument("--no-updates", action="store_true")
    ap.add_argument("--fast-episode-step", action="store_true",
                    help="episode_step of relabelled rows re-based inside the window only (mask / is_contiguous stay exact); default: "
                         "the reference's value (her.py:72-83), bit for bit")
    ap.add_argument("--serial", action="store_true", help="gather and loss back to back on one stream instead of pipelined on two")
    ap.add_argument("--buffers", type=int, default=3, help="batch buffers of the pipelined schedule (gathers run up to buffers-1 passes ahead)")
    ap.add_argument("--two-streams", action="store_true",
                    help="gather of pass k+1 on a second stream under the loss kernel of pass k (two launches per pass) instead of the "
                         "default one warp-specialised launch per pass (fdql_fused_pass: loss of pass k + gather of pass k+1)")
    ap.add_argument("--fused", action="store_true", help="(default; kept for older command lines)")
    ap.add_argument("--no-step-graph", action="store_true",
                    help="pipelined schedule launched from Python every step instead of one captured CUDA graph per step")
    ap.add_argument("--passes-per-step", type=int, default=0, help="passes of batches_per_step batches per step, 0 = auto (128 fused, 64 otherwise)")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the BASELINE.json configs[0..2] sections (Pendulum / CartPole / 64-bit HER shapes)")
    ap.add_argument("--no-graph", action="store_true", help="learner step launched eagerly instead of as one CUDA graph")
    ap.add_argument("--separate-streams", action="store_true", help="draw the index / goal streams in their own launch (fdql_sample_streams)")
    ap.add_argument("--tail-scan", action="store_true", help="relabelled returns by scanning the episode tail instead of the link records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the batch, loss and d loss / d q_pred of the last timed pass as DIR/<name>.npy "
                         "(a fixed, seeded sample of its windows); inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    return args


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", os.environ.get("FDQL_BENCH_CLOCK_MS", "200"),
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: fall back to every sample seen
            sm = [float(x.split(",")[1]) for _, x in self.lines if x.count(",") >= 8] or [0.0]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------------------
def build_ring(torch, pkg, Replay, n_rows, device, seed):
    """Synthetic bitflip-like replay: fixed-length episodes, goals in {0,1}^16, reward/done from R(ag, dg)."""
    n_eps = n_rows // LEP
    ring = Replay.ReplayMemory(n_eps * LEP + 1, B, T, device=device, seed=seed)
    ring.set_reward_op(pkg.RewardOp.bitflip(), GAMMA)
    gen = torch.Generator(device=device).manual_seed(seed)
    chunk_eps = 8192
    for e0 in range(0, n_eps, chunk_eps):
        ne = min(chunk_eps, n_eps - e0)
        n = ne * LEP
        ag = (torch.rand(n, GOAL, device=device, generator=gen) < 0.5).float()
        dg = (torch.rand(ne, GOAL, device=device, generator=gen) < 0.5).float().repeat_interleave(LEP, 0)
        hit = (ag == dg).all(-1, keepdim=True).float()
        step = torch.arange(n, device=device).remainder(LEP).float().unsqueeze(-1)
        cols = {"obs_1d": torch.randn(n, OBS, device=device, generator=gen),
                "action": torch.rand(n, ACT, device=device, generator=gen) * 2 - 1,
                "achieved_goal": ag, "desired_goal": dg, "reward": hit - 1, "task_done": hit,
                "episode_done": (step == LEP - 1).float(), "episode_step": step, "mc_return": torch.zeros(n, 1, device=device)}
        ring.add_rows(cols, episode_lengths=torch.full((ne,), LEP), with_returns=True)
    torch.cuda.synchronize(device)
    return ring


def run_ours(args):
    import torch
    import fastdeepqlearning_b200 as pkg
    from fastdeepqlearning_b200 import Replay, _lib as L

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    if os.environ.get("FDQL_LIB"):  # A/B runs of kernel variants (profiles/variants/): another build of the same C ABI
        L.LIB_PATH = os.environ["FDQL_LIB"]
    pkg.lib()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    from fastdeepqlearning_b200 import parallel
    numa_cpus = parallel.bind_to_gpu_numa_node(local) if world > 1 else None  # host buffers next to this rank's GPU
    dist = None
    if world > 1:
        import torch.distributed as dist
        # keep stdout to the one JSON line: NCCL's version / debug lines go to a file unless the caller chose one
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/fdql_nccl.%h.%p.log")
        dist.init_process_group("nccl", device_id=device)
    lib = pkg.lib()
    if os.environ.get("FDQL_PROBE_DBG"):  # profiles/: probe switches of the gather role (GatherArgs.dbg); results are then NOT valid batches
        lib.fdql_debug_force_generic_gather(int(os.environ["FDQL_PROBE_DBG"]) << 6)
    D = args.batches_per_step
    n = D * B
    M = (T - 1) * n
    ring = build_ring(torch, pkg, Replay, args.ring_rows, device, seed=1234 + rank)
    keys = ring.keys
    h = ring._h
    gen = torch.Generator(device=device).manual_seed(99 + rank)
    z = torch.randn(M, CQ, device=device, generator=gen) * 3
    q = torch.randn(M, CQ, device=device, generator=gen) * 3
    lp = torch.randn(M, device=device, generator=gen)
    def make_buf():
        o = {k: torch.empty((T, n, w), device=device) for k, w in zip(keys, ring._widths)}
        return {"out": o, "outp": L.ptr_array([o[k].data_ptr() for k in keys]), "mask": torch.empty(T, n, device=device),
                "contig": torch.empty(T - 1, n, device=device), "weight": torch.empty(T - 1, n, device=device),
                "starts": torch.empty(n, dtype=torch.int64, device=device), "flags": torch.empty(n, dtype=torch.uint8, device=device),
                "goals": torch.empty(n, dtype=torch.int64, device=device)}
    NB = max(2, args.buffers)
    bufs = [make_buf() for _ in range(NB)]  # the pipelined schedule samples passes k+1 .. k+NB-1 into the others while pass k's loss reads one
    out, outp, aux_mask, aux_contig, aux_weight = (bufs[0][k] for k in ("out", "outp", "mask", "contig", "weight"))
    starts, flags, goals = bufs[0]["starts"], bufs[0]["flags"], bufs[0]["goals"]
    loss = torch.empty(M, device=device)
    grad = torch.empty(M, CQ, device=device)
    stats = torch.zeros(4, dtype=torch.float64, device=device)
    params, n_params = ring.reward_op.c_params()
    exact = not args.fast_episode_step
    opts = L.OPT_EMIT_LEARNER_AUX | (L.OPT_EXACT_EPISODE_STEP if exact else 0)
    if args.tail_scan:
        lib.fdql_debug_force_generic_gather(16)  # tile kernel without the link records
    bytes_relabel = BYTES_RELABEL_SCAN if args.tail_scan else BYTES_RELABEL
    stream = torch.cuda.current_stream(device)
    side = torch.cuda.Stream(device)
    sp = C.c_void_p(stream.cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())
    rlen = len(ring)
    counter = [0]
    ctr_dev = torch.zeros(4, dtype=torch.int64, device=device)  # device-side draw counter of the captured step
    use_ctr_dev = [False]
    pipelined = not args.serial and not args.separate_streams
    fused = pipelined and not args.two_streams
    step_graph = pipelined and not args.no_step_graph
    P = args.passes_per_step or (128 if fused else 64)  # the fused schedule pays one unfused gather and one unfused loss per step

    # argument tuples are built once per (buffer, stream): the pipelined schedule needs ~6000 launches per second from this loop
    _args = {}

    def gather(b, st, extra=0):
        key = ("g", id(b), st.cuda_stream, extra)
        a = _args.get(key)
        if a is None:
            spx = C.c_void_p(st.cuda_stream)
            a = _args[key] = {
                "draw_head": (h, n, T, L.GOAL_FUTURE, P_RELABEL, 7 + rank),
                "draw_tail": (None, p(b["starts"]), p(b["flags"]), p(b["goals"]), ring.reward_op.op, params, n_params, GAMMA, opts | extra, B,
                              b["outp"], p(b["mask"]), p(b["contig"]), p(b["weight"]), spx),
                "streams_tail": (None, p(b["starts"]), p(b["flags"]), p(b["goals"]), spx),
                "gather": (h, n, T, rlen, p(b["starts"]), p(b["flags"]), p(b["goals"]), ring.reward_op.op, params, n_params, GAMMA,
                           opts | extra, B, b["outp"], p(b["mask"]), p(b["contig"]), p(b["weight"]), spx)}
        if args.separate_streams:
            L.check(lib.fdql_sample_streams(*a["draw_head"], counter[0], *a["streams_tail"]))
            L.check(lib.fdql_sample_gather(*a["gather"]))
        elif use_ctr_dev[0]:  # captured launches: the draw counter lives in device memory and every launch advances it
            L.check(lib.fdql_sample_gather_draw(*a["draw_head"], 1 << 40, p(ctr_dev), *a["draw_tail"][1:]))
        else:  # streams drawn inside the gather kernel: one launch
            L.check(lib.fdql_sample_gather_draw(*a["draw_head"], counter[0], *a["draw_tail"]))
        counter[0] += 1

    def tqc(b, st):
        key = ("t", id(b), st.cuda_stream)
        a = _args.get(key)
        if a is None:
            # the target reads reward / mask / mc_return of the NEXT row (t=1), quirk Q10
            a = _args[key] = (M, CQ, N_DROP, p(z), p(q), p(lp), p(b["out"]["reward"][1:]), p(b["mask"][1:]), p(b["out"]["mc_return"][1:]),
                              p(b["weight"]), ALPHA, GAMMA, p(loss), p(grad), None, p(stats), C.c_void_p(st.cuda_stream))
        L.check(lib.fdql_tqc_loss(*a))

    def run_serial(n_pass, evs=None):
        for i in range(n_pass):
            e = evs[i] if evs is not None and i < len(evs) else None
            if e:
                e[0].record(stream)
            gather(bufs[0], stream)
            if e:
                e[1].record(stream)
            tqc(bufs[0], stream)
            if e:
                e[2].record(stream)

    last_buf = [0]

    loss_stream = torch.cuda.Stream(device)

    def run_pipelined(n_pass, evs=None, every=16):
        """loss stream: loss(k); side stream: gathers up to NB - 1 passes ahead.  loss(k) waits for gather(k); gather(k + NB) waits
        for loss(k), whose inputs it overwrites (NB batch buffers: with three, the gather of pass k+2 fills the SMs while loss(k)
        drains and loss(k+1) ramps up).  Starts and ends with nothing in flight: n_pass gathers and n_pass losses, all inside the
        call (both streams fork from and join back into the caller's stream, so the call can be captured into a CUDA graph).
        Timing events (evs) only take timestamps; the dependencies ride on their own events."""
        cur_stream = torch.cuda.current_stream(device)
        t0 = torch.cuda.Event()
        t0.record(cur_stream)
        side.wait_event(t0)
        loss_stream.wait_event(t0)
        done_g, done_t = [None] * NB, [None] * NB

        def issue_gather(k):
            e = evs[k // every] if evs is not None and k % every == every // 2 and k // every < len(evs) else None
            slot = k % NB
            if done_t[slot] is not None:
                side.wait_event(done_t[slot])
            if e:
                e[0].record(side)
            gather(bufs[slot], side, L.OPT_CORESIDENT)
            if e:
                e[1].record(side)
            done_g[slot] = torch.cuda.Event()
            done_g[slot].record(side)

        for k in range(min(NB - 1, n_pass)):
            issue_gather(k)
        for k in range(n_pass):
            cur = k % NB
            e = evs[k // every] if evs is not None and k % every == every // 2 and k // every < len(evs) else None
            if k + NB - 1 < n_pass:
                issue_gather(k + NB - 1)
            loss_stream.wait_event(done_g[cur])
            if e:
                e[2].record(loss_stream)
            tqc(bufs[cur], loss_stream)
            if e:
                e[3].record(loss_stream)
            done_t[cur] = torch.cuda.Event()
            done_t[cur].record(loss_stream)
        cur_stream.wait_event(done_t[(n_pass - 1) % NB])
        cur_stream.wait_event(side_join(side))
        last_buf[0] = (n_pass - 1) % NB

    def run_fused(n_pass, evs=None, every=16):
        """one stream, one launch per pass: fdql_fused_pass = loss role on pass k's batch + gather role filling the other buffer with
        pass k+1's batch.  The first launch is a gather alone, the last one a loss alone: n_pass gathers and n_pass losses per call."""
        cur_stream = torch.cuda.current_stream(device)
        spx = C.c_void_p(cur_stream.cuda_stream)

        def half_g(b):
            return (h, n, T, L.GOAL_FUTURE, P_RELABEL, 7 + rank, (1 << 40) if use_ctr_dev[0] else counter[0],
                    p(ctr_dev) if use_ctr_dev[0] else None, p(b["starts"]), p(b["flags"]), p(b["goals"]), ring.reward_op.op, params, n_params,
                    GAMMA, opts, B, b["outp"], p(b["mask"]), p(b["contig"]), p(b["weight"]))

        def half_t(b, m):
            return (m, CQ, N_DROP, p(z), p(q), p(lp), p(b["out"]["reward"][1:]), p(b["mask"][1:]), p(b["out"]["mc_return"][1:]),
                    p(b["weight"]), ALPHA, GAMMA, p(loss), p(grad), p(stats), spx)
        for k in range(n_pass + 1):
            gb, tb = bufs[k % 2], bufs[(k + 1) % 2]
            g_half = half_g(gb)
            if k == n_pass:  # no gather: n_windows = 0
                g_half = (h, 0) + g_half[2:]
            e = evs[k // every] if evs is not None and k % every == every // 2 and k // every < len(evs) else None
            if e:
                e[0].record(cur_stream)
                e[2].record(cur_stream)
            L.check(lib.fdql_fused_pass(*g_half, *half_t(tb, M if k > 0 else 0)))
            if e:
                e[1].record(cur_stream)
                e[3].record(cur_stream)
            counter[0] += 1
        last_buf[0] = (n_pass - 1) % 2

    def side_join(st):
        e = torch.cuda.Event()
        e.record(st)
        return e

    # ---- the two kernels alone, back to back on one stream (kernel-level figures; also the --serial headline) ----
    lib.fdql_set_coresident(0)
    run_serial(3)
    torch.cuda.synchronize(device)
    sev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(20)]
    run_serial(20, sev)
    torch.cuda.synchronize(device)
    alone_ms = np.array([[e[j].elapsed_time(e[j + 1]) for j in range(2)] for e in sev]).mean(0)  # gather, tqc

    if pipelined:
        lib.fdql_set_coresident(1)  # the loss kernel leaves room on every SM for the co-resident gather blocks
    run = run_fused if fused else run_pipelined if pipelined else run_serial
    if fused:
        lib.fdql_set_coresident(0)
    for _ in range(max(args.warmup, 3)):
        run(P)
    torch.cuda.synchronize(device)
    K = args.steps
    n_ev = 8
    cg_step = None
    if step_graph:
        # one step = P passes of the pipelined schedule captured ONCE (both streams, every cross-stream dependency, device-side draw
        # counter); the timed region replays it K times.  Eight passes of the step carry external timing events around their two
        # kernels (event-record nodes: they take real timestamps at every replay).
        use_ctr_dev[0] = True
        run(2)  # the counter-from-device variant of the launch, once outside the capture
        torch.cuda.synchronize(device)
        gev = [[torch.cuda.Event(enable_timing=True, external=True) for _ in range(4)] for _ in range(n_ev)]
        cg_step = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg_step):
            run(P, gev, every=max(P // n_ev, 1))
        for _ in range(2):
            cg_step.replay()
        torch.cuda.synchronize(device)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K * n_ev)]
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.25)
    if dist:
        dist.barrier()
    torch.cuda.synchronize(device)
    t0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    g_acc = np.zeros((0, 3))
    for i in range(K):
        if cg_step is not None:
            cg_step.replay()
            if i % 25 == 24 or i == K - 1:  # read the in-graph timestamps of this replay (a sync every 25 steps; the GPU queue is 25 deep)
                torch.cuda.current_stream(device).synchronize()
                g_acc = np.concatenate([g_acc, [[float("nan"), e[0].elapsed_time(e[1]), e[2].elapsed_time(e[3])] for e in gev]])
        elif pipelined:
            run(P, evs[i * n_ev:(i + 1) * n_ev], every=max(P // n_ev, 1))
        else:
            run_serial(P, [[a, b_, c] for a, b_, c, _ in evs[i * n_ev:(i + 1) * n_ev]])
    e1.record(stream)
    torch.cuda.synchronize(device)
    t1 = time.time()
    if dist:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    clk = clocks.stop(t0, t1)

    def _el(a, b_):
        try:
            return a.elapsed_time(b_)
        except Exception:  # an event that was never recorded (P < 8 passes per step)
            return float("nan")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)  # (a column of this schedule's unused slots is all NaN)
        if cg_step is not None:
            k_ms = np.nanmean(g_acc, 0)
        elif pipelined:
            k_ms = np.nanmean(np.array([[float("nan"), _el(e[0], e[1]), _el(e[2], e[3])] for e in evs]), 0)  # -, gather, tqc (overlapped)
        else:
            k_ms = np.nanmean(np.array([[float("nan"), _el(e[0], e[1]), _el(e[1], e[2])] for e in evs]), 0)
    lib.fdql_set_coresident(0)
    if dist:
        tmax = torch.tensor([ms_total], device=device)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms_total = float(tmax.item())
    ms_step = ms_total / K
    ms_pass = ms_step / P
    value = world * M * P / (ms_step * 1e-3)
    chk = bufs[last_buf[0]] if pipelined else bufs[0]  # the batch of the last timed pass: spot-checked against the oracle below

    # ---- spot check of the last timed pass against the oracle (outside the timed region; oracle/ is the checker only).  It runs here,
    #      before the sections below reuse the batch buffers and loss / grad for their own launches ------------------------------------
    parity = None
    if not args.no_parity_check and rank == 0:
        parity = oracle_spot_check(torch, ring, chk, z, q, lp, loss, grad, n, exact)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, chk, loss, grad, n)
    loss_mean_timed, relabel_frac_timed = float(loss.mean()), float(chk["flags"].float().mean())
    if dist:
        dist.barrier()

    # ---- single-batch launches (B=4096 windows per launch): latency-bound figure, reported beside the headline ----
    def small_step(i):
        o = (i % D) * B
        outs = L.ptr_array([out[k].data_ptr() for k in keys])
        # outputs of a B-window launch are laid out [T, B, w] inside the first T*B rows of the big buffers
        L.check(lib.fdql_sample_gather_draw(h, B, T, L.GOAL_FUTURE, P_RELABEL, 7 + rank, 10_000 + i, None, p(starts[o:]), p(flags[o:]),
                                            p(goals[o:]), ring.reward_op.op, params, n_params, GAMMA, opts, B, outs, p(aux_mask),
                                            p(aux_contig), p(aux_weight), sp))
        L.check(lib.fdql_tqc_loss(B, CQ, N_DROP, p(z[o:]), p(q[o:]), p(lp[o:]), p(out["reward"].view(-1)[B:]),
                                  p(aux_mask.view(-1)[B:]), p(out["mc_return"].view(-1)[B:]), p(aux_weight), ALPHA, GAMMA,
                                  p(loss[o:]), p(grad[o:]), None, None, sp))
    small_ms = float("nan")
    if not args.no_small:
        for i in range(10):
            small_step(i)
        torch.cuda.synchronize(device)
        e0.record(stream)
        n_small = 200
        for i in range(n_small):
            small_step(i)
        e1.record(stream)
        torch.cuda.synchronize(device)
        small_ms = e0.elapsed_time(e1) / n_small

    # ---- the same per-batch launches as a CUDA graph of G batches round-robin over four streams (the learner's prefetch
    #      pattern: later batches are sampled/relabelled while earlier ones are targeted).  Draw counters live in device memory.
    graph_ms = float("nan")
    if not args.no_small:
        G = 16
        slots = []
        for i in range(G):
            so = {k: torch.empty((T, B, w), device=device) for k, w in zip(keys, ring._widths)}
            slots.append({"out": so, "outp": L.ptr_array([so[k].data_ptr() for k in keys]), "mask": torch.empty(T, B, device=device),
                          "contig": torch.empty(T - 1, B, device=device), "weight": torch.empty(T - 1, B, device=device),
                          "ctr": torch.zeros(4, dtype=torch.int64, device=device)})

        def graph_batch(i, st):
            sl, o, spx = slots[i], i * B, C.c_void_p(st.cuda_stream)
            L.check(lib.fdql_sample_gather_draw(h, B, T, L.GOAL_FUTURE, P_RELABEL, 1000 + 97 * rank + i, 0, p(sl["ctr"]), p(starts[o:]),
                                                p(flags[o:]), p(goals[o:]), ring.reward_op.op, params, n_params, GAMMA, opts, B,
                                                sl["outp"], p(sl["mask"]), p(sl["contig"]), p(sl["weight"]), spx))
            L.check(lib.fdql_tqc_loss(B, CQ, N_DROP, p(z[o:]), p(q[o:]), p(lp[o:]), p(sl["out"]["reward"][1:]), p(sl["mask"][1:]),
                                      p(sl["out"]["mc_return"][1:]), p(sl["weight"]), ALPHA, GAMMA, p(loss[o:]), p(grad[o:]), None,
                                      None, spx))
        NS = 4
        side = [torch.cuda.Stream(device) for _ in range(NS)]
        for i in range(G):  # warm-up outside capture
            graph_batch(i, stream)
        torch.cuda.synchronize(device)
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            cs = torch.cuda.current_stream(device)
            for st_ in side:
                st_.wait_stream(cs)
            for i in range(G):
                graph_batch(i, side[i % NS])
            for st_ in side:
                cs.wait_stream(st_)
        for _ in range(3):
            cg.replay()
        torch.cuda.synchronize(device)
        reps = 20
        first = starts[:B].clone()
        e0.record(stream)
        for _ in range(reps):
            cg.replay()
        e1.record(stream)
        torch.cuda.synchronize(device)
        assert not torch.equal(first, starts[:B]), "graph replays must draw fresh windows"
        graph_ms = e0.elapsed_time(e1) / (reps * G)

    # ---- secondary figure: the reference's default temporal_len = 50 (conf.py:38): 49 TD pairs per sampled window ------
    secondary = None
    if not args.no_secondary:
        T2, n2 = 50, 4 * B
        M2 = (T2 - 1) * n2
        out2 = {k: torch.empty((T2, n2, w), device=device) for k, w in zip(keys, ring._widths)}
        outp2 = L.ptr_array([out2[k].data_ptr() for k in keys])
        mask2, contig2, weight2 = (torch.empty(T2, n2, device=device), torch.empty(T2 - 1, n2, device=device),
                                   torch.empty(T2 - 1, n2, device=device))
        st2, fl2, go2 = (torch.empty(n2, dtype=torch.int64, device=device), torch.empty(n2, dtype=torch.uint8, device=device),
                         torch.empty(n2, dtype=torch.int64, device=device))
        z2 = torch.randn(M2, CQ, device=device, generator=gen) * 3
        q2 = torch.randn(M2, CQ, device=device, generator=gen) * 3
        lp2 = torch.randn(M2, device=device, generator=gen)
        loss2, grad2 = torch.empty(M2, device=device), torch.empty(M2, CQ, device=device)
        ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

        def step50(i, ev=None):
            if ev:
                ev[0].record(stream)
            L.check(lib.fdql_sample_streams(h, n2, T2, L.GOAL_FUTURE, P_RELABEL, 31 + rank, 50_000 + i, None, p(st2), p(fl2), p(go2), sp))
            L.check(lib.fdql_sample_gather(h, n2, T2, rlen, p(st2), p(fl2), p(go2), ring.reward_op.op, params, n_params, GAMMA,
                                           opts, B, outp2, p(mask2), p(contig2), p(weight2), sp))
            if ev:
                ev[1].record(stream)
            L.check(lib.fdql_tqc_loss(M2, CQ, N_DROP, p(z2), p(q2), p(lp2), p(out2["reward"][1:]), p(mask2[1:]),
                                      p(out2["mc_return"][1:]), p(weight2), ALPHA, GAMMA, p(loss2), p(grad2), None, None, sp))
            if ev:
                ev[2].record(stream)
        for i in range(3):
            step50(i)
        torch.cuda.synchronize(device)
        reps2, acc2 = 10, np.zeros(2)
        for i in range(reps2):
            step50(3 + i, ev2)
            torch.cuda.synchronize(device)
            acc2 += [ev2[0].elapsed_time(ev2[1]), ev2[1].elapsed_time(ev2[2])]
        ms2 = float(acc2.sum() / reps2)
        if dist:
            tm = torch.tensor([ms2], device=device)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms2 = float(tm.item())
        peak2, _ = peaks()
        # bytes per TD pair at T = 50: every window row is read and written once (436 B each way) per 49/50 pairs, relabelled windows
        # scan their episode tail's 16-byte records once per WINDOW; the loss moves 1520 B per pair
        gb2 = (2 * ROW_BYTES * T2 + 8 + P_RELABEL * (4 * GOAL + 25 + 16 * (LEP + 1) / 2)) / (T2 - 1)
        roof2 = {"bound": "hbm", "peak": peak2, "unit": "GB/s",
                 "gather": {"bytes_per_transition": gb2, "achieved": gb2 * M2 / (acc2[0] / reps2 * 1e-3) / 1e9,
                            "frac": gb2 * M2 / (acc2[0] / reps2 * 1e-3) / 1e9 / peak2},
                 "tqc": {"bytes_per_transition": BYTES_TQC, "achieved": BYTES_TQC * M2 / (acc2[1] / reps2 * 1e-3) / 1e9,
                         "frac": BYTES_TQC * M2 / (acc2[1] / reps2 * 1e-3) / 1e9 / peak2},
                 "whole_step": {"bytes_per_transition": gb2 + BYTES_TQC, "frac": (gb2 + BYTES_TQC) * M2 / (ms2 * 1e-3) / 1e9 / peak2}}
        # the same pass through the fused schedule of the headline: loss role on pass k + gather role on pass k+1, one launch per pass
        # (two batch buffers; first launch = gather alone, last = loss alone: R gathers and R losses inside the timed region)
        fused50 = None
        if fused:
            b50 = [{"out": out2, "outp": outp2, "mask": mask2, "contig": contig2, "weight": weight2, "st": st2, "fl": fl2, "go": go2}]
            o3 = {k: torch.empty((T2, n2, w), device=device) for k, w in zip(keys, ring._widths)}
            b50.append({"out": o3, "outp": L.ptr_array([o3[k].data_ptr() for k in keys]), "mask": torch.empty(T2, n2, device=device),
                        "contig": torch.empty(T2 - 1, n2, device=device), "weight": torch.empty(T2 - 1, n2, device=device),
                        "st": torch.empty(n2, dtype=torch.int64, device=device), "fl": torch.empty(n2, dtype=torch.uint8, device=device),
                        "go": torch.empty(n2, dtype=torch.int64, device=device)})

            def pass50(k, n_w, m):
                gb, tb = b50[k % 2], b50[(k + 1) % 2]
                L.check(lib.fdql_fused_pass(h, n_w, T2, L.GOAL_FUTURE, P_RELABEL, 31 + rank, 60_000 + k, None, p(gb["st"]), p(gb["fl"]),
                                            p(gb["go"]), ring.reward_op.op, params, n_params, GAMMA, opts, B, gb["outp"], p(gb["mask"]),
                                            p(gb["contig"]), p(gb["weight"]), m, CQ, N_DROP, p(z2), p(q2), p(lp2), p(tb["out"]["reward"][1:]),
                                            p(tb["mask"][1:]), p(tb["out"]["mc_return"][1:]), p(tb["weight"]), ALPHA, GAMMA, p(loss2),
                                            p(grad2), None, sp))

            def run50(R):
                pass50(0, n2, 0)
                for k in range(1, R):
                    pass50(k, n2, M2)
                pass50(R, 0, M2)
            run50(3)
            torch.cuda.synchronize(device)
            R50 = 20
            e0.record(stream)
            run50(R50)
            e1.record(stream)
            torch.cuda.synchronize(device)
            ms50 = e0.elapsed_time(e1) / R50
            if dist:
                tm = torch.tensor([ms50], device=device)
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                ms50 = float(tm.item())
            fused50 = {"ms_per_pass": ms50, "transitions_per_s": world * M2 / (ms50 * 1e-3), "passes": R50,
                       "frac": (gb2 + BYTES_TQC) * M2 / (ms50 * 1e-3) / 1e9 / peak2,
                       "schedule": "fdql_fused_pass, one launch per pass (loss of pass k + draw / gather / relabel of pass k+1), launched from "
                                   "Python; first launch = gather alone, last = loss alone"}
            del o3, b50
        secondary = {"temporal_len": T2, "windows_per_step": n2, "transitions_per_step_per_gpu": M2, "ms_per_step": ms2, "roofline": roof2,
                     "fused": fused50,
                     "transitions_per_s": world * M2 / (ms2 * 1e-3), "rows_gathered_per_s": world * T2 * n2 / (acc2[0] / reps2 * 1e-3),
                     "gather_ms": float(acc2[0] / reps2), "tqc_ms": float(acc2[1] / reps2), "loss_mean": float(loss2.mean()),
                     "note": "reference default temporal_len (conf.py:38): one window gives 49 TD pairs, so the gather is amortised and "
                             "the loss kernel is the step; transitions_per_s / gather_ms / tqc_ms: one serial pass (streams drawn by "
                             "fdql_sample_streams, relabelled returns by the tail scan: link records serve T <= 32); fused: the headline's "
                             "schedule at this temporal_len"}
        del out2, z2, q2, grad2, loss2, lp2

    # ---- e2e: the host-buffer C-ABI call, pinned host inputs, host outputs ---------------------------------------------
    e2e = None
    if not args.no_e2e:
        rng = np.random.default_rng(5 + rank)
        s_np = rng.integers(0, rlen - T, n)
        tail = (LEP - 1) - (s_np % LEP)  # rows after the start row inside its episode
        g_np = np.minimum(s_np + np.where(tail > 0, 1 + (rng.random(n) * tail).astype(np.int64), 0), s_np - s_np % LEP + LEP - 1)
        hs, hg = torch.from_numpy(s_np).pin_memory(), torch.from_numpy(g_np).pin_memory()
        hf = torch.from_numpy((rng.random(n) < P_RELABEL).astype(np.uint8)).pin_memory()
        hz, hq, hlp = z.cpu().pin_memory(), q.cpu().pin_memory(), lp.cpu().pin_memory()
        hloss = torch.empty(M).pin_memory()
        hgrad = torch.empty(M, CQ).pin_memory()
        ph = lambda t: C.c_void_p(t.data_ptr())

        def host_step():
            L.check(lib.fdql_hotpath_step_host(h, n, T, rlen, ph(hs), ph(hf), ph(hg), ring.reward_op.op, params, n_params, GAMMA,
                                               opts & ~L.OPT_EMIT_LEARNER_AUX, outp, CQ, N_DROP, ph(hz), ph(hq), ph(hlp), ALPHA,
                                               ph(hloss), ph(hgrad), sp))
            stream.synchronize()  # the caller reads loss / grad from host memory after every step
        for _ in range(2):
            host_step()
        if dist:
            dist.barrier()
        torch.cuda.synchronize(device)
        tw0 = time.perf_counter()
        e0.record(stream)
        for _ in range(args.e2e_steps):
            host_step()
        e1.record(stream)
        torch.cuda.synchronize(device)
        tw1 = time.perf_counter()
        ms_e2e = max(e0.elapsed_time(e1), (tw1 - tw0) * 1e3) / args.e2e_steps  # host sync is part of the call
        if dist:
            tm = torch.tensor([ms_e2e], device=device)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms_e2e = float(tm.item())
        e2e = {"value": world * M / (ms_e2e * 1e-3), "unit": "transitions/s",
               "h2d_bytes_per_step": int(n * 17 + M * CQ * 8 + M * 4), "d2h_bytes_per_step": int(M * 4 + M * CQ * 4),
               "ms_per_step": ms_e2e, "api": "fdql_hotpath_step_host (pinned host streams + critic outputs in, loss + dloss/dq out)",
               "loss_mean": float(hloss.mean())}

    # ---- second metric of BASELINE.json: TQC updates/s = full learner steps (sample+relabel on this ring, PyTorch MLP
    #      forward/backward for 5x25 critics + actor, fused TQC loss, Adam, soft target update; gradient all-reduce if N>1)
    updates = None
    if not args.no_updates:
        import types
        from fastdeepqlearning_b200 import Agent
        from fastdeepqlearning_b200.Replay.wrappers import SampleTimeHindsight
        torch.manual_seed(0)
        lconf = Agent.LearnerConf(training_device=str(device), obs_space={"obs_1d": OBS, "achieved_goal": GOAL, "desired_goal": GOAL},
                                  action_space=types.SimpleNamespace(shape=(ACT,)), num_critics=C_CRIT, num_q_predictions=Q_ATOMS,
                                  top_quantiles_to_drop=N_DROP / CQ + 1e-9, batch_size=B, temporal_len=T, gamma=GAMMA,
                                  use_cuda_graph=not args.no_graph, graph_allreduce=True)
        learner = Agent.Learner(lconf, [SampleTimeHindsight(ring, relabel_prob=P_RELABEL)])
        for _ in range(5):
            learner.train_step()
        if dist:
            dist.barrier()
        torch.cuda.synchronize(device)
        n_upd = 30
        e0.record(stream)
        for _ in range(n_upd):
            last = learner.train_step()
        e1.record(stream)
        torch.cuda.synchronize(device)
        ms_upd = e0.elapsed_time(e1) / n_upd
        if dist:
            tm = torch.tensor([ms_upd], device=device)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms_upd = float(tm.item())
        updates = {"value": 1e3 / ms_upd, "unit": "updates/s (each rank steps on its own 4096-window batch, gradients averaged)",
                   "ms_per_update": ms_upd, "transitions_per_s": world * B * (T - 1) * 1e3 / ms_upd,
                   "params": int(sum(p.numel() for p in learner.params)), "loss": float(last),
                   "cuda_graph": bool(lconf.use_cuda_graph),
                   "note": "policy/critic MLPs are ordinary PyTorch fp32 modules; sample/relabel/target/loss are this repo's CUDA kernels; "
                           "the whole step (kernels + MLP fwd/bwd + gradient all-reduce + Adam + target update) is one captured CUDA graph"}

    # ---- roofline of the dominant kernel (by measured time) ------------------------------------------------------------
    peak, peak_src = peaks()
    gname = "sample_gather_lean_kernel" if pipelined else "sample_gather_tile_kernel"
    kernels = {
        "sample_gather_kernel": {"ms": float(k_ms[1]), "ms_alone": float(alone_ms[0]),
                                 "bytes_per_transition": BYTES_GATHER + bytes_relabel + (0 if args.separate_streams else 17),
                                 "symbol": f"fdql::{gname}" + ("" if args.separate_streams else " (draws its own index / goal streams)"),
                                 "limiter": ("co-resident: two 4-warp blocks per SM under the loss kernel, wide keys through cp.async staging + "
                                             "bulk shared->global write-back (LDGSTS / UBLKCP), lane = (window, part) so one copy instruction "
                                             "serves eight windows; alone it is HBM-latency bound (long-scoreboard stalls), next to the loss kernel "
                                             "its duration is set by the issue slots that kernel leaves" if pipelined else
                                             "HBM latency on random 32-256 B segments (ncu: long-scoreboard stalls dominate)"),
                                 "relabelled_returns": "tail scan (16 B per tail row)" if args.tail_scan else
                                 "link records: chain of equal achieved goals + goal-agnostic return, O(hits) per window"},
        "tqc_loss_kernel": {"ms": float(k_ms[2]), "ms_alone": float(alone_ms[1]), "bytes_per_transition": BYTES_TQC,
                            "symbol": "fdql::tqc_loss_group_kernel<128, 7>",
                            "limiter": "instruction issue (82% active alone, ALU pipe 63%) and the LSU data pipe (shared-memory wavefronts 81% of "
                                       "peak): 128-value sort network + 375 seven-level searches per transition; not HBM (ncu, profiles/r2_*)"},
    }
    for kd in kernels.values():
        kd["note"] = ("ms = average launch duration inside the timed region, where the two kernels share every SM; ms_alone = the same "
                      "launch with the GPU to itself") if pipelined else "ms = average launch duration inside the timed region"
    alone = None
    if fused:
        # one launch per pass: the two stand-alone kernels only appear as the first / last launch of a step; their figures alone stay
        # in the line as `alone`, the kernel of the timed region is the fused one with both roles' algorithmic bytes
        alone = {k: {"ms_alone": kd["ms_alone"], "bytes_per_transition": kd["bytes_per_transition"], "symbol": kd["symbol"],
                     "frac_alone": kd["bytes_per_transition"] * M / (kd["ms_alone"] * 1e-3) / 1e9 / peak} for k, kd in kernels.items()}
        alone["sample_gather_kernel"]["symbol"] = "fdql::sample_gather_tile_kernel (draws its own index / goal streams)"
        kernels = {"fused_pass_kernel": {
            "ms": float(k_ms[2]), "bytes_per_transition": sum(kd["bytes_per_transition"] for kd in kernels.values()),
            "symbol": "fdql::fused_pass_kernel<7, true, true, 2, 0x44111> (T = 2 build: window length, record columns and copy plan "
                      "at compile time; the launcher falls back to the general build when any of them does not hold)",
            "roles": {"loss": "16 warps per SM: tqc_group_body on pass k (pool, sort, drop, soft target, quantile-Huber fwd+bwd, lower bound): %d B"
                              % BYTES_TQC,
                      "gather": "8 warps per SM: gather_lean_body on pass k+1 (draw, window gather through cp.async staging + bulk "
                                "shared->global write-back, HER relabel, reward / return recompute, learner aux): %.1f B"
                                % (BYTES_GATHER + bytes_relabel + 17)},
            "limiter": "instruction issue: 224 M warp instructions per launch (loss 209 M + gather 15 M), issue slots 76-78 % active (ncu, "
                       "profiles/r2_fused_*); LSU data pipe 78 %; DRAM 46 %.  Launch duration = instructions / issue rate with the gather "
                       "role's phases switched off one at a time (DESIGN 4.1f)",
            "note": "ms = average launch duration inside the timed region (CUDA-event nodes around 8 of the 64 launches of a step; a "
                    "launch between event nodes cannot overlap its neighbours' ramps, so this is a little above ms_per_pass)"}}
    if args.separate_streams:
        kernels["sample_streams_kernel"] = {"ms": float(k_ms[0]), "bytes_per_transition": BYTES_STREAMS, "symbol": "fdql::sample_streams_kernel"}
    for kd in kernels.values():
        kd["achieved_gbs"] = kd["bytes_per_transition"] * M / (kd["ms"] * 1e-3) / 1e9
        kd["frac"] = kd["achieved_gbs"] / peak
        if "ms_alone" in kd:
            kd["frac_alone"] = kd["bytes_per_transition"] * M / (kd["ms_alone"] * 1e-3) / 1e9 / peak
    dom = max(kernels, key=lambda k: kernels[k].get("ms_alone", kernels[k]["ms"]))
    total_bytes = sum(kd["bytes_per_transition"] for kd in kernels.values())
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "frac_alone": kernels[dom].get("frac_alone"), "traffic": None, "peak_source": peak_src,
                "note": ("one launch per pass (loss role on pass k + gather role on pass k+1): achieved = both roles' algorithmic bytes over "
                         "the launch duration; `alone` = the two stand-alone kernels with the GPU to themselves") if fused else
                        ("launch_ms / achieved / frac: this kernel's average duration inside the timed region, where it shares every SM with "
                         "the co-resident gather of the next pass (so they are lower than the kernel's own figures); frac_alone: the same "
                         "launch with the GPU to itself; whole_step: both kernels' bytes over the pass time") if pipelined else None,
                "algorithmic_bytes_per_launch": kernels[dom]["bytes_per_transition"] * M, "launch_ms": kernels[dom]["ms"],
                "survey_bytes_per_transition": {"sample_gather_kernel": BYTES_GATHER + BYTES_RELABEL_SURVEY, "tqc_loss_kernel": BYTES_TQC},
                "kernels": kernels, "alone": alone,
                "whole_step": {"bytes_per_transition": total_bytes, "achieved_gbs": total_bytes * M / (ms_pass * 1e-3) / 1e9,
                               "frac": total_bytes * M / (ms_pass * 1e-3) / 1e9 / peak, "ms_per_pass": ms_pass,
                               "note": "both kernels' algorithmic bytes over the time of one pass of the pipelined schedule"},
                "traffic_source": "dram__bytes per launch from the ncu --set full capture summarised in profiles/ (constant, not measured in-run)"}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            roofline["traffic"] = pj.get(dom)
            # second view for kernels that are not HBM-bound: warp instructions per launch (ncu, profiles/) against the SM issue rate
            # (148 SMs x 4 schedulers x 1 instruction per clock at the sampled SM clock), with this run's launch time
            sm_clk = (clk.get("sm_mhz") or 1965.0) * 1e6
            for name, kd in kernels.items():
                wi = pj.get("warp_instructions", {}).get(name)
                if wi and not args.tail_scan and not args.separate_streams:
                    kd["issue"] = {"warp_instructions_per_launch": wi, "achieved_ginst_s": wi / (kd["ms"] * 1e-3) / 1e9,
                                   "peak_ginst_s": 148 * 4 * sm_clk / 1e9, "frac": wi / (kd["ms"] * 1e-3) / (148 * 4 * sm_clk)}
        except Exception:
            pass

    line = {"metric": "sampled+relabelled+targeted transitions/s", "value": value, "unit": "transitions/s", "n_gpus": world,
            "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "ours",
            "config": {"workload": "HER(future,k=4: relabel p=0.8, return-to-go recomputed over the whole episode tail) + TQC 5x25 drop 10 + "
                                   "n-step lower bound; obs64/act8/goal16; ring %d rows/GPU (L=128 episodes); batch 4096, T=2"
                                   % (len(ring) + 1),
                       "batch": B, "temporal_len": T, "batches_per_step": D, "passes_per_step": P, "transitions_per_step_per_gpu": M * P,
                       "transitions_per_pass_per_gpu": M,
                       "schedule": ("one launch per pass (fdql_fused_pass, one persistent 24-warp block per SM): the loss role (16 warps) works on pass k "
                                    "while the gather role (8 warps) draws, gathers and relabels pass k+1 into the other batch buffer, as the "
                                    "reference's prefetch thread does (torch_dataloader.py:22-39); every pass complete inside the timed region "
                                    "(first launch of a step = gather alone, last = loss alone)" +
                                    ("; one step = one captured CUDA graph, replayed" if step_graph else "; launched from Python")) if fused else
                                   ("pipelined on two streams over %d batch buffers: gather of pass k+1 (FDQL_OPT_CORESIDENT, two 4-warp blocks per SM) "
                                    "under the loss of pass k, as the reference's prefetch thread does (torch_dataloader.py:22-39); every pass complete "
                                    "inside the timed region" + ("; one step = one captured CUDA graph, replayed" if step_graph else
                                                                  "; launched from Python")) % NB if pipelined
                       else "gather and loss back to back on one stream",
                       "ring_rows_per_gpu": len(ring) + 1,
                       "l2": "inputs larger than L2 (random rows of a %.1f GB arena; %d MB of critic outputs per step)"
                             % ((len(ring) + 1) * (ROW_BYTES + 16) / 1e9, M * CQ * 8 // 2 ** 20),
                       "exact_episode_step": bool(exact), "parallelism": f"replay shards x{world}, no data-path collective",
                       "numa_bound_cpus": len(numa_cpus) if numa_cpus else None},
            "roofline": roofline, "gpu_launches": (P + 1) * K if fused else (3 if args.separate_streams else 2) * K * P, "clocks": clk,
            "ms_per_pass": ms_pass,
            "single_batch_launches": {"windows_per_launch": B, "ms_per_batch": small_ms, "transitions_per_s": world * B / (small_ms * 1e-3),
                                      "note": "2 launches per 4096-window batch from Python (gather with fused draw, loss), launch-latency bound",
                                      "cuda_graph_4_streams": {"ms_per_batch": graph_ms, "transitions_per_s": world * B / (graph_ms * 1e-3),
                                                               "note": "16 batches x 2 launches captured once, round-robin over four streams"}},
            "checks": {"loss_mean": loss_mean_timed, "relabel_frac": relabel_frac_timed,
                       "violations": float(stats[2] / max(float(stats[3]), 1) / CQ), "parity_vs_oracle": parity}}
    if secondary:
        line["secondary_T50"] = secondary
    if not args.no_extra and rank == 0:
        line["extra"] = extra_configs(torch, pkg, Replay, L, lib, device)
    if e2e:
        line["e2e"] = e2e
    if updates:
        line["tqc_updates"] = updates
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference(args, steps=3, warmup=1, quiet=True)["cpu_baseline"]
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist:
        # NCCL kernels captured in the learner's CUDA graph must go before the communicator does; a watchdog ends the process
        # if the teardown still blocks (the JSON line is out by then)
        import gc
        import threading
        threading.Timer(20.0, lambda: os._exit(0)).start()
        if not args.no_updates:
            learner.close()
        learner = None  # noqa: F841
        gc.collect()
        torch.cuda.synchronize(device)
        dist.barrier()
        dist.destroy_process_group()
        os._exit(0)


# ---------------------------------------------------------------------------------------------------------------------
EXTRA_SPECS = {
    # BASELINE.json configs[0]: SAC on Pendulum with uniform replay + n-step lower bound (obs 3, act 1, no goals; the non-distributional
    # head: 5 critics x 1 value, min over the ensemble, smooth-L1, lower bound replaces the TD term -- soft_actor_critic.py:63-99)
    "config0_pendulum_sac": dict(obs=3, act=1, goal=0, discrete_n=0, critics=5, atoms=1, n_drop=0, her=False, loss="sac"),
    # configs[1]: discrete Gumbel-softmax SAC on CartPole with n-step replay, batch 4096 (obs 4, 2 actions stored as an index and
    # one-hot encoded by get_losses, deepQlearning.py:206-210; reference default head 5 x 10 atoms, drop int(0.2 * 50) = 10)
    "config1_cartpole_discrete": dict(obs=4, act=1, goal=0, discrete_n=2, critics=5, atoms=10, n_drop=10, her=False, loss="tqc"),
    # configs[2]: HER on the 64-bit bit-flipping env (bitflip.py: obs 64, achieved / desired goal 64, 64 discrete actions), future k=4
    "config2_her_bitflip64": dict(obs=64, act=1, goal=64, discrete_n=64, critics=5, atoms=25, n_drop=10, her=True, loss="tqc"),
}


def extra_configs(torch, pkg, Replay, L, lib, device, rows=2_000_000, D=64, reps=10):
    """One serial pass (gather [+ relabel] [+ one-hot] + loss) at the other BASELINE.json shapes: D batches of 4096 windows, T = 2, on a
    ring of `rows` rows; per-kernel CUDA-event times, algorithmic bytes (SURVEY.md section 8d applied to the shape) and roofline
    fractions.  Parity on the same shapes: tests/test_gpu_r2.py::test_baseline_config_shapes_vs_oracle."""
    from fastdeepqlearning_b200 import ops
    peak, _ = peaks()
    out = {}
    n = D * B
    for name, sp in EXTRA_SPECS.items():
        gen = torch.Generator(device=device).manual_seed(5)
        n_eps = rows // LEP
        N = n_eps * LEP
        ring = Replay.ReplayMemory(N + 1, B, T, device=device, seed=11)
        step = torch.arange(N, device=device).remainder(LEP).float().unsqueeze(-1)
        cols = {"obs_1d": torch.randn(N, sp["obs"], device=device, generator=gen)}
        if sp["discrete_n"]:
            cols["action"] = torch.randint(0, sp["discrete_n"], (N, 1), device=device, generator=gen).float()
        else:
            cols["action"] = torch.rand(N, sp["act"], device=device, generator=gen) * 2 - 1
        if sp["goal"]:
            ag = (torch.rand(N, sp["goal"], device=device, generator=gen) < 0.5).float()
            dg = (torch.rand(n_eps, sp["goal"], device=device, generator=gen) < 0.5).float().repeat_interleave(LEP, 0)
            hit = (ag == dg).all(-1, keepdim=True).float()
            cols.update(achieved_goal=ag, desired_goal=dg, reward=hit - 1, task_done=hit)
            ring.set_reward_op(pkg.RewardOp.bitflip(), GAMMA)
        else:
            cols.update(reward=-torch.rand(N, 1, device=device, generator=gen), task_done=(step == LEP - 1).float())
        cols.update(episode_done=(step == LEP - 1).float(), episode_step=step, mc_return=torch.zeros(N, 1, device=device))
        ring.add_rows(cols, episode_lengths=torch.full((n_eps,), LEP), with_returns=True)
        del cols
        CQx = sp["critics"] * sp["atoms"]
        z = torch.randn(T - 1, n, CQx, device=device, generator=gen) * 3
        q = torch.randn(T - 1, n, CQx, device=device, generator=gen) * 3
        lp = torch.randn(T - 1, n, 1, device=device, generator=gen)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        acc = np.zeros(3)
        for i in range(3 + reps):
            ev[0].record()
            xp = ring.temporal_sample(n=n, relabel_prob=P_RELABEL if sp["her"] else 0.0, aux=True, exact_episode_step=True, reuse_outputs=True)
            ev[1].record()
            if sp["discrete_n"]:
                onehot = ops.action_onehot(xp["action"], sp["discrete_n"])
            ev[2].record()
            if sp["loss"] == "sac":
                r = ops.sac_min_target_loss(q, z, lp, xp["reward"][1:], xp["mask"][1:], xp["mc_return"][1:], ALPHA, GAMMA,
                                            grad_scale=xp["loss_weight"], want_stats=True)
            else:
                r = ops.tqc_loss(q, z, lp, xp["reward"][1:], xp["mask"][1:], xp["mc_return"][1:], ALPHA, GAMMA, sp["n_drop"],
                                 grad_scale=xp["loss_weight"], want_stats=True)
            ev[3].record()
            torch.cuda.synchronize(device)
            if i >= 3:
                acc += [ev[j].elapsed_time(ev[j + 1]) for j in range(3)]
        ms = acc / reps
        row_b = 4 * (sp["obs"] + sp["act"] + 2 * sp["goal"]) + 4 * 5
        b_gather = 4 * row_b + 8 + (P_RELABEL * (4 * sp["goal"] + 25 + 16 * T) + 17 if sp["her"] else 8)
        b_onehot = (4 + 4 * sp["discrete_n"]) * T if sp["discrete_n"] else 0
        b_loss = 3 * 4 * CQx + 20
        tot = float(ms.sum())
        gf = lambda b_, m_: b_ * n / (m_ * 1e-3) / 1e9 if m_ > 0 else 0.0
        out[name] = {"shape": sp, "ring_rows": N, "windows_per_pass": n, "ms": {"gather": float(ms[0]), "onehot": float(ms[1]), "loss": float(ms[2])},
                     "transitions_per_s": n / (tot * 1e-3), "loss_mean": float(r["loss"].mean()),
                     "bytes_per_transition": {"gather": b_gather, "onehot": b_onehot, "loss": b_loss},
                     "roofline": {"bound": "hbm", "peak": peak, "unit": "GB/s",
                                  "gather": {"achieved": gf(b_gather, ms[0]), "frac": gf(b_gather, ms[0]) / peak},
                                  "loss": {"achieved": gf(b_loss, ms[2]), "frac": gf(b_loss, ms[2]) / peak},
                                  "whole_pass": {"achieved": gf(b_gather + b_onehot + b_loss, tot), "frac": gf(b_gather + b_onehot + b_loss, tot) / peak}},
                     "kernels": ("sample_gather_tile_kernel (fused draw)" + (" + onehot_kernel" if sp["discrete_n"] else "") +
                                 (" + sac_min_target_kernel" if sp["loss"] == "sac" else " + tqc_loss_group_kernel"))}
        del ring, z, q, lp, xp, r
        torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------------------------
def oracle_spot_check(torch, ring, b, z, q, lp, loss, grad, n, exact, n_check=1024):
    """The first `n_check` windows of the last timed pass against the CPU oracle (outside the timed region): the sampled and
    relabelled batch vs oracle.sample_time_relabel on the same drawn streams, then loss and d loss / d q_pred of those transitions vs
    oracle.tqc_q_loss.  Returns mismatch counts for the bit-exact outputs and maximum relative errors for the fp32 ones."""
    from oracle import cpu_restatement as O
    w = min(n_check, n)
    s_np = b["starts"][:w].cpu().numpy()
    f_np = b["flags"][:w].cpu().numpy().astype(bool)
    g_np = b["goals"][:w].cpu().numpy()
    eps = np.unique(np.concatenate([s_np // LEP, (s_np + T - 1) // LEP]))  # fixed-length episodes laid end to end from row 0
    rows = (eps[:, None] * LEP + np.arange(LEP)[None]).reshape(-1)
    pos = {int(e): i * LEP for i, e in enumerate(eps)}
    rows_t = torch.as_tensor(rows, device=b["starts"].device)
    mem = ring.memory
    cols = {k: mem[k][rows_t].cpu().numpy() for k in ring.keys}
    remap = lambda r: np.array([pos[int(x) // LEP] + int(x) % LEP for x in r])
    cs, cg = remap(s_np), remap(g_np)
    es = (np.arange(len(rows)) // LEP) * LEP
    want = O.sample_time_relabel(cols, cs, T, f_np, cg, es, es + LEP - 1, O.reward_bitflip, GAMMA)
    got = {k: v[:, :w].cpu().numpy() for k, v in b["out"].items()}
    exact_keys = [k for k in cols if k not in ("reward", "mc_return") and (exact or k != "episode_step")]
    mism = {k: int((got[k] != want[k]).sum()) for k in exact_keys}
    rel = lambda a, c: float(np.max(np.abs(a - c) / np.maximum(np.abs(c), 1.0)))
    mask, contig = O.learner_preprocess(want["task_done"], want["episode_step"])
    mism["mask"] = int((b["mask"][:, :w].cpu().numpy() != mask[..., 0]).sum())
    mism["is_contiguous"] = int((b["contig"][:, :w].cpu().numpy() != contig[..., 0]).sum())
    wgt = O.upstream_weight(contig, T)[..., 0] * (w / B)  # the kernel normalises by the configured batch size B
    zq = lambda t: t[:w].cpu().numpy().astype(np.float64)
    ol, og, _ = O.tqc_q_loss(zq(q), zq(z), zq(lp).reshape(-1, 1), want["reward"][1].astype(np.float64), mask[1].astype(np.float64),
                             want["mc_return"][1].astype(np.float64), ALPHA, GAMMA, N_DROP)
    og = og * wgt[0][:, None]
    gl, gg = loss[:w].cpu().numpy(), grad[:w].cpu().numpy()
    return {"windows": int(w), "exact_mismatches": mism, "relabelled": int(f_np.sum()),
            "max_rel_err": {"reward": rel(got["reward"], want["reward"]), "mc_return": rel(got["mc_return"], want["mc_return"]),
                            "loss": rel(gl, ol[:, 0]), "grad_q_over_its_scale": float(np.max(np.abs(gg - og)) / max(np.abs(og).max(), 1e-30))},
            "tolerance": "bit-exact for indices, goals, done masks, steps; 1e-5 relative for returns, targets and losses",
            "ok": bool(sum(mism.values()) == 0 and rel(got["mc_return"], want["mc_return"]) < 1e-5 and rel(gl, ol[:, 0]) < 1e-5)}


def dump_outputs(torch, d, b, loss, grad, n, n_sample=16384, seed=0):
    """What the caller of the timed path receives for its last pass, as d/<name>.npy: the drawn streams (start row, hindsight
    flag, goal row), the relabelled batch [T, windows, width] with its learner aux (mask, is_contiguous, loss_weight), and the
    per-transition loss and d loss / d q_pred [T - 1, windows(, CQ)].  The whole pass is ~360 MB, so the same fixed, seeded
    sample of `n_sample` windows (window_index) is taken from every array: ~23 MB.  Row indices are stored as float64 (exact)."""
    os.makedirs(d, exist_ok=True)
    idx = np.sort(np.random.default_rng(seed).choice(n, min(n_sample, n), replace=False))
    it = torch.as_tensor(idx, device=loss.device)
    arrays = {"window_index": torch.as_tensor(idx), "starts": b["starts"][it], "hindsight_flags": b["flags"][it],
              "goal_rows": b["goals"][it]}
    arrays.update((k, v[:, it]) for k, v in b["out"].items())
    arrays.update(mask=b["mask"][:, it], is_contiguous=b["contig"][:, it], loss_weight=b["weight"][:, it],
                  loss=loss.view(T - 1, n)[:, it], grad_q=grad.view(T - 1, n, CQ)[:, it])
    for name, a in arrays.items():
        a = a.cpu().numpy()
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float64 if a.dtype == np.int64 else np.float32))


# ---------------------------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_window_chunk(job):
    """One worker: window gather (numpy fancy index, replay_memory.py:62-70) + hindsight relabel + return recompute for a
    slice of the batch, by the oracle's restatement of her.py:55-95 / nstep_return.py:60-72.  The ring is inherited from the parent
    (copy-on-write); the slice of the index / goal streams travels in the job."""
    from oracle import cpu_restatement as O
    t, s, f, g = job
    c = _CPU
    return O.sample_time_relabel(c["cols"], s, t, f, g, c["ep_start"], c["ep_end"], O.reward_bitflip, GAMMA)


def _cpu_gather_only(job):
    """ReplayMemory.temporal_sample (replay_memory.py:54-70) of one independent shard process: randint + fancy index of every key."""
    t, seed, reps = job
    rng = np.random.default_rng(seed)
    cols = _CPU["cols"]
    n_rows = len(cols["reward"])
    t0 = time.perf_counter()
    for _ in range(reps):
        idx = (np.arange(t)[:, None] + rng.integers(0, n_rows - t, B)[None, :]) % n_rows
        out = {k: v[idx] for k, v in cols.items()}
    return time.perf_counter() - t0, out["reward"].shape


def _cpu_write_path(job):
    """HindsightNStepReplay(random) -> NStepReturn(1000) -> ReplayMemory row by row (her.py:24-95, nstep_return.py:23-72), one core."""
    from oracle import cpu_restatement as O
    n_eps, seed = job
    rng = np.random.default_rng(seed)
    sink = O.RingOracle(4 * n_eps * LEP, B, T)
    picks = iter(rng.integers(0, LEP, n_eps).tolist())
    her = O.HindsightOracle(O.NStepOracle(sink, 1000, GAMMA), O.reward_bitflip, mode="random", goal_picker=lambda L_: next(picks))
    ag = (rng.random((n_eps * LEP, GOAL)) < 0.5).astype(np.float32)
    dg = np.repeat((rng.random((n_eps, GOAL)) < 0.5).astype(np.float32), LEP, 0)
    obs = rng.standard_normal((n_eps * LEP, OBS)).astype(np.float32)
    act = rng.standard_normal((n_eps * LEP, ACT)).astype(np.float32)
    t0 = time.perf_counter()
    for i in range(n_eps * LEP):
        hit = bool((ag[i] == dg[i]).all())
        her.add({"obs_1d": obs[i], "action": act[i], "achieved_goal": ag[i], "desired_goal": dg[i], "reward": 0.0 if hit else -1.0,
                 "task_done": hit, "episode_done": i % LEP == LEP - 1, "episode_step": i % LEP, "info": {}})
    return time.perf_counter() - t0, len(sink)


class _LazyExtent:
    """ep_start / ep_end of a row for fixed-length episodes without materialising 1e7-entry tables per worker."""

    def __init__(self, last):
        self.last = last

    def __getitem__(self, row):
        base = (int(row) // LEP) * LEP
        return base + LEP - 1 if self.last else base


def cpu_reference(args, steps, warmup, quiet=False, stages=True):
    """The reference's CPU replay-and-target path (oracle port) on the host cores, same workload, bounded sample."""
    import multiprocessing as mp
    import torch
    from oracle import cpu_restatement as O

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rng = np.random.default_rng(0)
    n_rows = (args.ring_rows // LEP) * LEP
    ep_of_n = n_rows // LEP
    ag = (rng.random((n_rows, GOAL), dtype=np.float32) < 0.5).astype(np.float32)
    dg = np.repeat((rng.random((ep_of_n, GOAL), dtype=np.float32) < 0.5).astype(np.float32), LEP, axis=0)
    hit = (ag == dg).all(-1, keepdims=True)
    step = (np.arange(n_rows) % LEP).astype(np.float32).reshape(-1, 1)
    cols = {"obs_1d": rng.standard_normal((n_rows, OBS), dtype=np.float32),
            "action": rng.random((n_rows, ACT), dtype=np.float32) * 2 - 1, "achieved_goal": ag, "desired_goal": dg,
            "reward": hit.astype(np.float32) - 1, "task_done": hit.astype(np.float32),
            "episode_done": (step == LEP - 1).astype(np.float32), "episode_step": step}
    cols["mc_return"] = O.segmented_returns(cols["reward"][:LEP * 64], cols["episode_done"][:LEP * 64], GAMMA).reshape(-1, 1)
    cols["mc_return"] = np.resize(cols["mc_return"], (n_rows, 1))  # values only feed the lower bound; timing-equivalent
    nb = args.cpu_batches or 1
    n = nb * B
    _CPU.update(cols=cols, ep_start=_LazyExtent(False), ep_end=_LazyExtent(True))
    z = torch.randn(n, CQ) * 3
    q = torch.randn(n, CQ) * 3
    lp = torch.randn(n, 1)
    workers = min(cores, 64)
    # ONE pool for the whole run, forked after the ring exists (shared copy-on-write); each step's streams travel in the jobs
    pool = mp.get_context("fork").Pool(workers) if workers > 1 else None
    stage_t = {"gather_relabel": 0.0, "tqc": 0.0}

    def tqc_stage(xp, n_):
        mask = 1.0 - xp["task_done"]
        qp = q[:n_].clone().requires_grad_(True)
        loss = O.tqc_q_loss_torch(qp.view(T - 1, n_, CQ), z[:n_].view(T - 1, n_, CQ), lp[:n_].view(T - 1, n_, 1), xp["reward"][1:], mask[1:],
                                  xp["mc_return"][1:], ALPHA, GAMMA, N_DROP)
        loss.mean().backward()
        return float(loss.mean())

    def one_step():
        t0 = time.perf_counter()
        s = rng.integers(0, n_rows - T, n)
        tail = (LEP - 1) - (s % LEP)
        g = s + np.where(tail > 0, 1 + (rng.random(n) * tail).astype(np.int64), 0)
        g = np.minimum(g, s - s % LEP + LEP - 1)
        f = rng.random(n) < P_RELABEL
        per = (n + workers - 1) // workers
        jobs = [(T, s[i:i + per], f[i:i + per], g[i:i + per]) for i in range(0, n, per)]
        parts = pool.map(_cpu_window_chunk, jobs) if pool else [_cpu_window_chunk(j) for j in jobs]
        batch = {k: np.concatenate([p_[k] for p_ in parts], axis=1) for k in parts[0]}
        xp = {k: torch.from_numpy(v) for k, v in batch.items()}  # TorchDataLoader cast (already fp32)
        t1 = time.perf_counter()
        out = tqc_stage(xp, n)
        t2 = time.perf_counter()
        stage_t["gather_relabel"] += t1 - t0
        stage_t["tqc"] += t2 - t1
        return out

    for _ in range(warmup):
        one_step()
    stage_t.update(gather_relabel=0.0, tqc=0.0)
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    tt = time.perf_counter() - t0
    ms_step = tt / steps * 1e3
    value = (T - 1) * n / (ms_step * 1e-3)
    base = {"value": value, "unit": "transitions/s", "cores": cores, "kind": "port",
            "sample": f"{steps} step(s) of {nb} batch(es) x {B} windows (T={T}) on a {n_rows}-row numpy ring: fancy-index gather + "
                      f"oracle HER relabel/return recompute over one persistent pool of {workers} forked workers, then the reference's "
                      f"torch-CPU TQC sort/target/[CQ x K] pairwise quantile-Huber fwd+bwd on {cores} threads",
            "stage_ms_per_step": {"gather_relabel_return": stage_t["gather_relabel"] / steps * 1e3, "tqc_target_loss_fwd_bwd": stage_t["tqc"] / steps * 1e3}}
    if stages:  # BASELINE.md section 3: per-stage figures of record, each a bounded sample on these host cores
        st = {}
        for t_len, reps in ((2, 20), (50, 4)):
            el, _ = _cpu_gather_only((t_len, 1, reps))
            st[f"temporal_sample_T{t_len}_1proc"] = {"ms_per_call": el / reps * 1e3, "rows_per_s": reps * t_len * B / el}
            if pool:
                res = pool.map(_cpu_gather_only, [(t_len, 10 + i, reps) for i in range(workers)])
                el_max = max(r[0] for r in res)
                st[f"temporal_sample_T{t_len}_{workers}proc"] = {"ms_per_call": el_max / reps * 1e3, "rows_per_s": workers * reps * t_len * B / el_max,
                                                                  "note": "independent shard processes, the reference's own scaling model"}
        el, stored = _cpu_write_path((6, 3))
        st["write_path_her_random_nstep_1core"] = {"env_rows_per_s": 6 * LEP / el, "stored_rows_per_s": stored / el,
                                                   "note": "HindsightNStepReplay(random) -> NStepReturn(1000) -> ring, 128-step episodes, row by row"}
        xp1 = {k: torch.from_numpy(cols[k][:2 * B].reshape(T, B, -1)) for k in ("reward", "task_done", "mc_return")}
        tqc_stage(xp1, B)
        t0 = time.perf_counter()
        for _ in range(3):
            tqc_stage(xp1, B)
        el = (time.perf_counter() - t0) / 3
        st["tqc_target_loss_fwd_bwd"] = {"ms_per_batch": el * 1e3, "transitions_per_s": B / el, "threads": torch.get_num_threads()}
        try:
            st["full_update"] = _cpu_full_update(torch)
        except Exception as e:  # the learner mirror needs the CUDA library even for its plain-torch modules' import
            st["full_update"] = {"unavailable": repr(e)[:200]}
        base["stages"] = st
    if pool:
        pool.close()
        pool.join()
    line = {"metric": "sampled+relabelled+targeted transitions/s", "value": value, "unit": "transitions/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "HER(future,k=4: relabel p=0.8, return-to-go recomputed over the whole episode tail) + TQC 5x25 drop 10 + "
                                   "n-step lower bound; obs64/act8/goal16; ring %d rows/GPU (L=128 episodes); batch 4096, T=2" % (n_rows + 1),
                       "batch": B, "temporal_len": T, "batches_per_step": nb},
            "cpu_baseline": base, "e2e": {"value": value, "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    return line


def _cpu_full_update(torch):
    """get_losses + backward + Adam step + update_targets on CPU torch with the reference's network shapes (deepQlearning.py:105-127,
    198-249: encoder MLPs 96 -> 256 -> 256, actor [256], 5 critics [256, 256] x 25 atoms), B = 4096, T = 2: updates/s."""
    from torch import nn

    def mlp(i, o, hs):  # models/mlp.py:62-90: the head sees the input and every hidden layer
        class M(nn.Module):
            def __init__(self):
                super().__init__()
                d = [i] + list(hs)
                self.h = nn.ModuleList([nn.Linear(a, b) for a, b in zip(d[:-1], d[1:])])
                self.o = nn.Linear(sum(d), o)

            def forward(self, x):
                f = [x]
                for l_ in self.h:
                    x = nn.functional.leaky_relu(l_(x))
                    f.append(x)
                return self.o(torch.cat(f, -1))
        return M()
    from oracle import cpu_restatement as O
    S = 256
    enc = nn.Sequential(mlp(OBS + 2 * GOAL, 256, (256,)), mlp(256, S, (256,)))
    actor, actor_t = mlp(S, 2 * ACT, (256,)), mlp(S, 2 * ACT, (256,))
    crit = nn.ModuleList([mlp(S + ACT, Q_ATOMS, (256, 256)) for _ in range(C_CRIT)])
    crit_t = nn.ModuleList([mlp(S + ACT, Q_ATOMS, (256, 256)) for _ in range(C_CRIT)])
    params = list(enc.parameters()) + list(actor.parameters()) + list(crit.parameters())
    opt = torch.optim.Adam(params, lr=3e-4)
    xp = {"obs": torch.randn(T, B, OBS + 2 * GOAL), "action": torch.rand(T, B, ACT) * 2 - 1, "reward": -torch.ones(T, B, 1),
          "mask": torch.ones(T, B, 1), "mc_return": -torch.ones(T, B, 1) * 5}

    def pi(net, st):
        mu, ls = net(st).chunk(2, -1)
        ls = ls.clamp(-20, 2)
        eps = torch.randn_like(mu)
        a = torch.tanh(mu + ls.exp() * eps)
        return a, (-0.5 * eps ** 2 - ls - 0.9189385 - torch.log(1 - a ** 2 + 1e-4)).sum(-1, keepdim=True)

    def update():
        st = enc(xp["obs"])
        cur, nxt = st[:-1], st[1:]
        with torch.no_grad():
            na, nlp = pi(actor_t, nxt)
            nz = torch.cat([c(torch.cat((nxt, na), -1)) for c in crit_t], -1)
        qp = torch.cat([c(torch.cat((cur, xp["action"][:-1]), -1)) for c in crit], -1)
        ql = O.tqc_q_loss_torch(qp, nz, nlp, xp["reward"][1:], xp["mask"][1:], xp["mc_return"][1:], ALPHA, GAMMA, N_DROP)
        a, lpi = pi(actor, cur)
        qpi = torch.cat([c(torch.cat((cur.detach(), a), -1)) for c in crit], -1).mean(-1, keepdim=True)
        loss = (ql + (lpi - qpi)).mean() / T
        opt.zero_grad()
        loss.backward()
        opt.step()
        with torch.no_grad():
            for t_, s_ in zip(list(crit_t.parameters()) + list(actor_t.parameters()), list(crit.parameters()) + list(actor.parameters())):
                t_.lerp_(s_, 5e-3)
    update()
    t0 = time.perf_counter()
    for _ in range(2):
        update()
    el = (time.perf_counter() - t0) / 2
    return {"ms_per_update": el * 1e3, "updates_per_s": 1 / el, "transitions_per_s": B / el, "threads": torch.get_num_threads(),
            "params": int(sum(p_.numel() for p_ in params))}


def main():
    args = parse()
    if args.impl == "reference":
        if int(os.environ.get("RANK", 0)) != 0:
            return
        print(json.dumps(cpu_reference(args, steps=max(args.steps, 1), warmup=args.warmup)))
        return
    run_ours(args)


if __name__ == "__main__":
    main()
