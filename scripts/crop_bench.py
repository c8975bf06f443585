"""Timing of the data step's nearest-to-anchor crop (csrc/datastep.cu): `ops.crop_nearest` over N in {1 024, 8 192, 25 600,
25 601, 87 303, 305 558} points and P in {1, 24, 148} clouds, keep = int(N * 0.750681278) (the reserve of --overlap 0.575).
Up to 25 600 points both kernels run on the same inputs: the one-CTA rank count (`vcr_crop_nearest`, what
`ops.crop_nearest` routes to there) and the segmented radix sort (`vcr_crop_nearest_sort`); above that only the sort runs.

Two times per call, medians over the calls after warm-up: `graph` replays one captured call between CUDA events (device
time of the launches, as a captured data step sees it); `eager` is a CUDA-event pair around one `ops` call from Python
(what an eager caller waits for, host enqueue of the sort's 26 launches and its workspace allocation included).  Inputs are
uniform in [-0.5, 0.5)^3, generated on the device from a fixed seed; at P = 1 the output is checked against
oracle/synth.crop_nearest_to_last and at N <= 25 600 the two kernels against each other.  The device name and power limit
are read in the same run.

    python scripts/crop_bench.py --out DIR [--warmup 2] [--min-ms 200]    -> DIR/crop_bench.json
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
from vcr_net_b200._lib import lib
from oracle import synth

NS = (1024, 8192, 25600, 25601, 87303, 305558)
PS = (1, 24, 148)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() if r.returncode == 0 else None
    except (OSError, subprocess.TimeoutExpired):
        return None


def timed(fn, warmup, min_ms):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times, total = [], 0.0
    while len(times) < 5 or (total < min_ms and len(times) < 500):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
        total += times[-1]
    return times


def measure(crop, x, keep, warmup, min_ms):
    eager = timed(lambda: crop(x, keep), warmup, min_ms)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = crop(x, keep)
    graph = timed(g.replay, warmup, min_ms)
    res = {"graph_median_ms": float(np.median(graph)), "graph_min_ms": float(np.min(graph)), "graph_calls": len(graph),
           "eager_median_ms": float(np.median(eager)), "eager_calls": len(eager)}
    return out.clone(), res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for crop_bench.json")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--min-ms", type=float, default=200.0, help="timed window per size, route and timing (>= 5 calls)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("crop_bench: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = "cuda:0"
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_index_power_limit_max_sm_clock": power_limit(),
           "reserve": synth.RESERVE_0575, "one_cta_max_points": ops.CROP_ONE_CTA_MAX_POINTS,
           "timing": "CUDA events; graph = replay of one captured call, eager = one ops call from Python; medians",
           "runs": [], "sort_faster_from_points": {}}
    gen = torch.Generator(device=dev).manual_seed(0)
    L = lib()
    for P in PS:
        for N in NS:
            keep = int(N * synth.RESERVE_0575)
            x = torch.rand((P, 3, N), dtype=torch.float64, device=dev, generator=gen) - 0.5
            routes = [("sort", ops.crop_nearest_sort)]
            if N <= ops.CROP_ONE_CTA_MAX_POINTS:
                routes.insert(0, ("one_cta", ops.crop_nearest))
            outs = {}
            for name, crop in routes:
                outs[name], row = measure(crop, x, keep, a.warmup, a.min_ms)
                row.update({"P": P, "N": N, "keep": keep, "route": name,
                            "workspace_bytes": int(L.vcr_crop_nearest_workspace_bytes(P, N)) if name == "sort" else 0,
                            "gpoints_per_s_graph": P * N / row["graph_median_ms"] / 1e6})
                if P == 1:
                    want = synth.crop_nearest_to_last(x[0].cpu().numpy(), synth.RESERVE_0575).astype(np.float32)
                    row["equals_oracle"] = bool(np.array_equal(outs[name][0].cpu().numpy(), want))
                res["runs"].append(row)
                print(f"P={P:3d} N={N:6d} {name:>7s}: graph {row['graph_median_ms']:9.4f} ms  eager "
                      f"{row['eager_median_ms']:9.4f} ms" + (f"  oracle={row['equals_oracle']}" if P == 1 else ""),
                      flush=True)
            if len(outs) == 2:
                same = bool(torch.equal(outs["one_cta"], outs["sort"]))
                res["runs"][-1]["equals_one_cta"] = same
                print(f"           sort == one_cta: {same}", flush=True)
            del x, outs
            torch.cuda.empty_cache()
        both = {}
        for r in res["runs"]:
            if r["P"] == P and r["N"] <= ops.CROP_ONE_CTA_MAX_POINTS:
                both.setdefault(r["N"], {})[r["route"]] = r["graph_median_ms"]
        faster = [n for n in sorted(both) if both[n]["sort"] < both[n]["one_cta"]]
        res["sort_faster_from_points"][str(P)] = faster[0] if faster else None
    path = os.path.join(a.out, "crop_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(res["device"], res["nvidia_smi_index_power_limit_max_sm_clock"], "sort faster from (graph time):",
          res["sort_faster_from_points"], "->", path)


if __name__ == "__main__":
    main()
