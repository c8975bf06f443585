"""Partial-to-partial registration above 16 384 points: VCRNet(partial=True), h3, vcrnetIter at iter 1 and 3 for clouds
of N in {16 384, 20 480, 32 768, 65 536, 131 072, 229 376} points, B = 1 and B = 4 pairs (B = 4 up to 131 072 points).

Per size it records the CUDA-event time of a vcrnetIter call (eager launch sequence: the captured-graph replay saves
launch overhead that is negligible at these sizes), torch.cuda.max_memory_allocated over that call, the selectCom
statistics call (four launches of the fused tensor-core kernel; each launch also timed once under torch.profiler, in
a separate pass) and the top-K calls of the partial path.  At 16 384 points, where the score matrix still fits,
select_stats_tc is timed against the materialised path (the [Ns, Nt] fp32 dot + negdist + softmax passes) on the same
operands, with the peak memory of each.  The device name and power limit are read in the same run.

    python scripts/partial_large_bench.py --out DIR [--sizes 16384,20480,...] [--min-ms 500]   -> DIR/partial_large_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("VCR_CUDA_GRAPH", "0")
import numpy as np
import torch

SIZES = (16384, 20480, 32768, 65536, 131072, 229376)
B4_MAX = 131072
D = 512


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() if r.returncode == 0 else None
    except (OSError, subprocess.TimeoutExpired):
        return None


def time_ms(fn, warmup, min_ms, min_calls=3, max_calls=50):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    while len(times) < min_calls or (sum(times) < min_ms and len(times) < max_calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return {"median_ms": float(np.median(times)), "min_ms": float(np.min(times)), "max_ms": float(np.max(times)),
            "calls": len(times)}


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return int(torch.cuda.max_memory_allocated()), int(torch.cuda.max_memory_allocated() - base)


def partial_pairs(synth, B, N, first_item):
    num = int(np.ceil(N / synth.RESERVE_0575))
    while int(num * synth.RESERVE_0575) > N:
        num -= 1
    while int(num * synth.RESERVE_0575) < N:
        num += 1
    p = synth.make_pairs(B, num, partial=True, base_points=num, first_item=first_item)
    assert p["src"].shape[2] == N
    return p


def layernormed(ops, Fn, B, N, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, N, D, device=dev, generator=g)
    _, op, sq = ops.layernorm_head(x, torch.ones(D, device=dev), torch.zeros(D, device=dev), want_out=False)
    return Fn.HeadPre(op, sq)


def stats_kernel_ms(ops, ps, pt, B, N):
    """Each of the four launches of one select_stats_tc call under torch.profiler (a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile
    ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, N, N, D)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, N, N, D)
        torch.cuda.synchronize()
    out = []
    for ev in prof.events():
        if "softcorr_tc_kernel" in ev.name:
            dt = getattr(ev, "device_time", None)
            if dt is None:
                dt = ev.cuda_time
            out.append({"kernel": ev.name, "ms": float(dt) / 1e3})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for partial_large_bench.json")
    ap.add_argument("--sizes", default=",".join(str(n) for n in SIZES))
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--min-ms", type=float, default=500.0, help="timed window per measurement (at least 3 calls)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("partial_large_bench: no CUDA device")
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops
    from vcr_net_b200 import functional as Fn
    from vcr_net_b200.synthetic import default_args
    from oracle import synth
    config.set_precision("h3")
    config.cuda_graph = False
    os.makedirs(a.out, exist_ok=True)
    dev = "cuda:0"
    lpd = dict(np.load(os.path.join(ROOT, "tests", "golden", "lpd_pretrained_weights.npz")))
    net = V.VCRNet(default_args(partial=True, overlap2=synth.OVERLAP2_0575)).to(dev).eval()
    net.load_state_dict(synth.checkpoint_to_torch(synth.make_checkpoint(1234, emb_weights=lpd)), strict=True)
    ov2 = synth.OVERLAP2_0575
    L = ops.lib()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_index_power_limit_max_sm_clock": power_limit(),
           "precision": "h3", "overlap2": ov2,
           "timing": "CUDA events around each call after warm-up, median; vcrnetIter on the eager launch sequence; L2 not "
                     "flushed (every working set here is larger than the 126 MB L2 except the top-K rows)",
           "select_stats_flop_per_pair": "4 launches x 3 fp16 products x 2*N*N*512",
           "cluster_barrier_cost": "not measured", "runs": [], "stats_vs_materialised": None}
    for N in (int(s) for s in a.sizes.split(",")):
        for B in ((1, 4) if N <= B4_MAX else (1,)):
            row = {"N": N, "B": B}
            try:
                p = partial_pairs(synth, B, N, 11)
                src, tgt = torch.from_numpy(p["src"]).to(dev), torch.from_numpy(p["tgt"]).to(dev)
                for it in (1, 3):
                    t = time_ms(lambda: V.vcrnetIter(net, src, tgt, iter=it), a.warmup, a.min_ms)
                    t["ms_per_pair"] = t["median_ms"] / B
                    t["peak_bytes"], _ = peak_bytes(lambda: V.vcrnetIter(net, src, tgt, iter=it))
                    row[f"iter{it}"] = t
                del src, tgt
                ps = layernormed(ops, Fn, B, N, 1, dev)
                pt = layernormed(ops, Fn, B, N, 2, dev)
                st = time_ms(lambda: ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, N, N, D), 1, a.min_ms)
                st["tflops"] = 4 * 3 * 2.0 * N * N * D * B / (st["median_ms"] * 1e-3) / 1e12
                st["kernels_profiled"] = stats_kernel_ms(ops, ps, pt, B, N)
                row["select_stats_tc"] = st
                K_sel, K_pair = int(N * 0.84 * ov2), int(int(N * 0.84 * ov2) * 0.52 * ov2)
                both = torch.rand(2 * B, N, device=dev)
                conf = torch.rand(B, int(N * 0.84 * ov2), device=dev)
                row["topk_selectcom_ms"] = time_ms(lambda: ops.topk_select(both, K_sel), 1, a.min_ms)
                row["topk_copair_ms"] = time_ms(lambda: ops.topk_select(conf, K_pair), 1, a.min_ms)
                row["topk_keymask_ms"] = time_ms(
                    lambda: ops.topk_select(both[:B], int(N * ov2), want_idx=False, want_mask=True), 1, a.min_ms)
                row["attn_colsum_workspace_bytes"] = int(L.vcr_attn_colsum_workspace_bytes(B, 4, N, N))
                if N == 16384 and B == 1:
                    mat = time_ms(lambda: Fn._select_stats_materialised(None, None, (ps, pt), B, N, N), 1, a.min_ms)
                    _, mat["peak_extra_bytes"] = peak_bytes(lambda: Fn._select_stats_materialised(None, None, (ps, pt), B, N, N))
                    fus = dict(st)
                    _, fus["peak_extra_bytes"] = peak_bytes(lambda: ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, N, N, D))
                    r1, c1 = ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, N, N, D)
                    r2, c2 = Fn._select_stats_materialised(None, None, (ps, pt), B, N, N)
                    res["stats_vs_materialised"] = {
                        "N": N, "B": B, "select_stats_tc": fus, "materialised": mat,
                        "max_rel_diff_row": float(((r1 - r2).abs().max() / r2.abs().max()).item()),
                        "max_rel_diff_col": float(((c1 - c2).abs().max() / c2.abs().max()).item())}
                del ps, pt, both, conf
            except torch.cuda.OutOfMemoryError as e:
                row["error"] = f"out of memory: {str(e).splitlines()[0]}"
            torch.cuda.empty_cache()
            res["runs"].append(row)
            msg = {k: (v["median_ms"] if isinstance(v, dict) and "median_ms" in v else v) for k, v in row.items()}
            print(json.dumps(msg), flush=True)
    path = os.path.join(a.out, "partial_large_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(res["device"], res["nvidia_smi_index_power_limit_max_sm_clock"], "->", path)


if __name__ == "__main__":
    main()
