"""Narrow (uint8) observation keys: the narrow gather alone, a whole sample against the fp32 twin, the arena bytes of both, and the
write path.

Ring: 2e5 rows of 84x84x4 uint8 frames (28,224 B a row, 5.6 GB: far larger than the 126 MB L2, and the windows start at random rows,
so every frame is read from HBM) next to the headline's other keys (action 8, achieved / desired goal 16, reward, task_done,
episode_done, episode_step, mc_return).  The fp32 twin holds the same rows as fp32 (22.6 GB).
  * narrow_gather_kernel alone, at B = 4096, T = 2 and at B = 256, T = 50 (franQ's defaults): kernel time from torch.profiler (CUDA
    activity, the kernels named narrow_gather_kernel), and bytes / s for the bytes the gather must move: w read + 4 w written per row,
    8 B of start per window;
  * a whole sample (fdql_sample_gather, injected starts) of the narrow ring against the fp32 twin: CUDA events over 50 calls;
  * fdql_arena_info bytes of both rings;
  * write path: rows / s through add_rows (device uint8 frames, 2048 rows a call) and through one-dict add (host numpy frames).
The card's name, power limit and SM clock are read in the same run.

    python profiles/narrow_gather_bench.py [--rows 200000] [--out narrow_gather_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fastdeepqlearning_b200 as fdql  # noqa: E402
from fastdeepqlearning_b200 import Replay  # noqa: E402

FRAME = (84, 84, 4)
W = 84 * 84 * 4
LEP = 100


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.splitlines()[0].split(",")])) if out else {}


def copy_bandwidth():
    """MEASURED_PEAKS.json's copy bandwidth when the machine has one, else a device-to-device copy of 4 GiB measured here (bytes read +
    written over the time of the copy)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth)"
    src = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    del src, dst
    torch.cuda.empty_cache()
    return 2 * (1 << 32) / ms / 1e6, "measured here: torch device-to-device copy of 4 GiB, (read + written) / time"


def fill(ring, rows, narrow, chunk=2000):
    g = torch.Generator(device="cuda").manual_seed(1)
    for b in range(0, rows, chunk):
        n = min(chunk, rows - b)
        step = (torch.arange(b, b + n, device="cuda") % LEP).float().view(n, 1)
        obs = torch.randint(0, 256, (n, W), device="cuda", generator=g, dtype=torch.uint8)
        cols = {"obs": obs if narrow else obs.float(), "action": torch.rand(n, 8, device="cuda", generator=g),
                "achieved_goal": torch.randint(0, 2, (n, 16), device="cuda", generator=g).float(),
                "desired_goal": torch.randint(0, 2, (n, 16), device="cuda", generator=g).float(),
                "reward": -torch.ones(n, 1, device="cuda"), "task_done": torch.zeros(n, 1, device="cuda"),
                "episode_done": (step == LEP - 1).float(), "episode_step": step, "mc_return": torch.zeros(n, 1, device="cuda")}
        ring.add_rows(cols, episode_lengths=[LEP] * (n // LEP))
    torch.cuda.synchronize()


def gather_args(ring, starts, T, keys):
    from fastdeepqlearning_b200 import _lib as L
    n = starts.numel()
    out = {k: torch.empty((T, n, w), device="cuda") for k, w in zip(ring._keys, ring._widths) if k in keys}
    ptrs = L.ptr_array([out[k].data_ptr() if k in out else 0 for k in ring._keys])
    return out, (ring._h, n, T, len(ring), C.c_void_p(starts.data_ptr()), None, None, 0, None, 0, 0.99, 0, n, ptrs, None, None, None)


def sample(lib, args):
    fdql._lib.check(lib.fdql_sample_gather(*args, C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def narrow_kernel_ms(lib, ring, B, T, reps=30):
    starts = torch.randint(0, len(ring) - T, (B,), device="cuda")
    _, args = gather_args(ring, starts, T, ("obs",))
    for _ in range(5):
        sample(lib, args)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            sample(lib, args)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "narrow_gather_kernel" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
    if not ev:
        raise RuntimeError("the profile holds no narrow_gather_kernel launch")
    ms = sum(e.device_time_total for e in ev) / len(ev) / 1e3
    bytes_ = B * T * (W + 4 * W) + 8 * B
    return {"B": B, "T": T, "kernel_ms": ms, "bytes": bytes_, "gb_per_s": bytes_ / ms / 1e6, "launches": len(ev)}


def whole_sample_ms(lib, ring, B, T, reps=50):
    starts = torch.randint(0, len(ring) - T, (B,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
    _, args = gather_args(ring, starts, T, tuple(ring._keys))
    for _ in range(5):
        sample(lib, args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        sample(lib, args)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def info_bytes(lib, ring):
    b = C.c_int64()
    fdql._lib.check(lib.fdql_arena_info(ring._h, None, None, None, C.byref(b)))
    return b.value


def write_rates(narrow):
    kd = {"obs": torch.uint8} if narrow else None
    ring = Replay.ReplayMemory(20000, 256, 2, key_dtypes=kd)
    n = 2048
    g = torch.Generator(device="cuda").manual_seed(2)
    obs = torch.randint(0, 256, (n, W), device="cuda", generator=g, dtype=torch.uint8)
    cols = {"obs": obs if narrow else obs.float(), "action": torch.rand(n, 8, device="cuda"), "reward": torch.zeros(n, 1, device="cuda")}
    ring.add_rows(cols)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        ring.add_rows(cols)
    torch.cuda.synchronize()
    rows_s = 10 * n / (time.perf_counter() - t0)
    rng = np.random.default_rng(0)
    frames = rng.integers(0, 256, (64,) + FRAME, dtype=np.uint8)
    xps = [{"obs": frames[i % 64], "action": np.zeros(8, np.float32), "reward": 0.0} for i in range(3000)]
    if not narrow:
        xps = [dict(x, obs=x["obs"].astype(np.float32)) for x in xps]
    for x in xps[:1024]:
        ring.add(x)
    ring.flush()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for x in xps:
        ring.add(x)
    ring.flush()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    # the same rows split into host staging (add below the staging block's 1024 rows) and the flushes
    stage = flush = 0.0
    for b in range(0, len(xps), 1000):
        ta = time.perf_counter()
        for x in xps[b:b + 1000]:
            ring.add(x)
        tb = time.perf_counter()
        ring.flush()
        torch.cuda.synchronize()
        stage, flush = stage + tb - ta, flush + time.perf_counter() - tb
    return {"add_rows_rows_per_s": rows_s, "add_one_dict_rows_per_s": len(xps) / (t1 - t0),
            "add_one_dict_staging_us_per_row": stage / len(xps) * 1e6, "add_one_dict_flush_us_per_row": flush / len(xps) * 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=200_000)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    lib = fdql.lib()
    res = {"card": card(), "rows": a.rows, "frame": list(FRAME)}
    bw, src = copy_bandwidth()
    res["copy_gb_per_s"], res["copy_bw_source"] = bw, src
    n = Replay.ReplayMemory(a.rows + 1, 256, 2, key_dtypes={"obs": torch.uint8})
    fill(n, a.rows, True)
    res["narrow_kernel"] = [narrow_kernel_ms(lib, n, 4096, 2), narrow_kernel_ms(lib, n, 256, 50)]
    if bw:
        for r in res["narrow_kernel"]:
            r["share_of_copy_bw"] = r["gb_per_s"] / bw
    f = Replay.ReplayMemory(a.rows + 1, 256, 2)
    fill(f, a.rows, False)
    res["arena_bytes"] = {"uint8": info_bytes(lib, n), "fp32": info_bytes(lib, f)}
    res["whole_sample_ms"] = []
    for B, T in ((4096, 2), (256, 50)):
        for _ in range(2):  # alternate the twins
            res["whole_sample_ms"].append({"B": B, "T": T, "uint8": whole_sample_ms(lib, n, B, T), "fp32": whole_sample_ms(lib, f, B, T)})
    del n, f
    torch.cuda.empty_cache()
    res["write_path"] = {"uint8": write_rates(True), "fp32": write_rates(False)}
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
