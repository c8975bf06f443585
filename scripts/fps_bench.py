"""Farthest-point sampling timing (csrc/fps.cu): median CUDA-event time per vcr_fps call and per sampling step, over
B in {1, 16, 148} clouds, N in {14 336, 16 384, 65 536, 229 376} points and npoint in {32, 1024}.  N = 14 336 is the
largest cloud of the one-CTA kernel; the other sizes run on clusters of 2, 8 and 16 CTAs.  The device name and power
limit are read in the same run.  The B = 1 results are checked against oracle/canon.c.

    python scripts/fps_bench.py --out DIR [--warmup 2] [--min-ms 200]    -> DIR/fps_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from vcr_net_b200 import ops
from oracle import canon

BS = (1, 16, 148)
NS = (14336, 16384, 65536, 229376)
NPOINTS = (32, 1024)
MAX_SLICE = 14336               # points per CTA (16 bytes each in 224 KB of shared memory)


def route(N):
    if N <= MAX_SLICE:
        return "one CTA"
    C = 2
    while C * MAX_SLICE < N:
        C *= 2
    return f"cluster of {C}"


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() if r.returncode == 0 else None
    except (OSError, subprocess.TimeoutExpired):
        return None


def time_calls(x, npoint, warmup, min_ms):
    for _ in range(warmup):
        ops.fps(x, npoint, want64=False)
    torch.cuda.synchronize()
    times, total = [], 0.0
    while len(times) < 5 or (total < min_ms and len(times) < 200):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = ops.fps(x, npoint, want64=False)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        times.append(ms)
        total += ms
    return out, times


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for fps_bench.json")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--min-ms", type=float, default=200.0, help="timed window per size (at least 5 calls)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fps_bench: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = "cuda:0"
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_index_power_limit_max_sm_clock": power_limit(),
           "timing": "CUDA events around each vcr_fps call after warm-up; median over the calls",
           "cluster_barrier_us_per_step": "not measured", "runs": []}
    rs = np.random.RandomState(0)
    for N in NS:
        for B in BS:
            p = rs.randn(B, 3, N).astype(np.float32)
            x = torch.from_numpy(p).to(dev)
            for npoint in NPOINTS:
                out, times = time_calls(x, npoint, a.warmup, a.min_ms)
                med = float(np.median(times))
                row = {"B": B, "N": N, "npoint": npoint, "route": route(N), "calls": len(times),
                       "median_ms_per_call": med, "min_ms_per_call": float(np.min(times)),
                       "max_ms_per_call": float(np.max(times)), "median_us_per_step": med * 1e3 / npoint}
                if B == 1:
                    row["equals_canon"] = bool(np.array_equal(out.cpu().numpy(), canon.fps(p, npoint)))
                res["runs"].append(row)
                print(f"B={B:3d} N={N:6d} npoint={npoint:4d} {row['route']:>13s}: {med:9.3f} ms/call "
                      f"{row['median_us_per_step']:8.2f} us/step  ({len(times)} calls)"
                      + (f"  canon={row['equals_canon']}" if B == 1 else ""), flush=True)
    path = os.path.join(a.out, "fps_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(res["device"], res["nvidia_smi_index_power_limit_max_sm_clock"], "->", path)


if __name__ == "__main__":
    main()
