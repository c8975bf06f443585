"""Throughput of ragged batches (vcrnetIterRagged) against one vcrnetIter call per pair and a uniform batch.

24 whole-to-whole pairs with seeded sizes in [512, 1024] (source and target sizes drawn separately), h3, iter 1 and 3:
  (a) ragged   one vcrnetIterRagged call on the padded batch (eager, and replayed from a captured CUDA graph)
  (b) per pair one vcrnetIter call per pair (product default: the graph cache holds 4 shapes)
  (c) uniform  one vcrnetIter call on 24 pairs of 1024 points (product default: graph replay), the cost ceiling
Rates are pairs per second from CUDA events around `--reps` calls after a warm-up.  Per-kernel device times compare each
ragged entry point with the same entry point's uniform launch at N_max = 1024 (CUDA events per C-ABI call, summed per
name over one call).  Usage: python scripts/ragged_bench.py [--out profiles/ragged_bench.json]

--partial: the same for partial-to-partial pairs (vcrnetIterRaggedPartial, VCRNet(partial=True)): pair b comes from
synth.make_pairs(partial=True) at a seeded num_points in [512, 1024] (its clouds keep the default reserve, 3/4 of them), and
(c) is the benchmark's shape, 24 pairs of 768 points cropped from 1024.  Per-kernel sums cover every C-ABI entry point,
each ragged one filed under its uniform name.  Writes profiles/ragged_partial_bench.json by default.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vcr_net_b200 as V  # noqa: E402
from vcr_net_b200 import config, ragged  # noqa: E402
from vcr_net_b200._lib import lib  # noqa: E402
from oracle import synth  # noqa: E402
from oracle.ref_harness import default_args  # noqa: E402

DEV = "cuda:0"


def timed(fn, reps):
    for _ in range(3):          # vcrnetIter's graph cache runs a shape eagerly, captures it on the second call, replays after
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def per_kernel(fn):
    L = lib()
    L.profile_begin()
    fn()
    out = {}
    for name, ms, _ in L.profile_end():
        out[name] = out.get(name, 0.0) + ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--partial", action="store_true")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--pairs", type=int, default=24)
    a = ap.parse_args()
    out_path = a.out or ("profiles/ragged_partial_bench.json" if a.partial else "profiles/ragged_bench.json")
    config.set_precision("h3")
    config.cuda_graph = True
    rng = np.random.RandomState(2026)
    P = a.pairs
    if a.partial:
        npts = rng.randint(512, 1025, P)
        ps = [synth.make_pairs(1, int(n), partial=True, seed=5, first_item=b) for b, n in enumerate(npts)]
        src_l = [torch.from_numpy(q["src"][0]).to(DEV) for q in ps]
        tgt_l = [torch.from_numpy(q["tgt"][0]).to(DEV) for q in ps]
        ns, nt = np.array([c.shape[1] for c in src_l]), np.array([c.shape[1] for c in tgt_l])
        p = synth.make_pairs(P, 1024, partial=True, reserve=0.75, seed=5)
        uniform = "uniform_768"
        run_ragged = V.vcrnetIterRaggedPartial
    else:
        ns, nt = rng.randint(512, 1025, P), rng.randint(512, 1025, P)
        p = synth.make_pairs(P, 1024, seed=5)
        src_l = [torch.from_numpy(p["src"][b, :, :ns[b]]).to(DEV) for b in range(P)]
        tgt_l = [torch.from_numpy(p["tgt"][b, :, :nt[b]]).to(DEV) for b in range(P)]
        uniform = "uniform_1024"
        run_ragged = V.vcrnetIterRagged
    src_u, tgt_u = torch.from_numpy(p["src"]).to(DEV), torch.from_numpy(p["tgt"]).to(DEV)
    src, sl = ragged.pad_clouds(src_l)
    tgt, tl = ragged.pad_clouds(tgt_l)
    ckpt = synth.make_checkpoint(1234)
    net = V.VCRNet(default_args(partial=a.partial)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=False)
    res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                 capture_output=True, text=True).stdout.strip(),
           "pairs": P, "partial": a.partial, "src_sizes": ns.tolist(), "tgt_sizes": nt.tolist(), "precision": "h3",
           "reps": a.reps, "iter": {}}
    for it in (1, 3):
        r = {}
        r["ragged_eager_ms"] = timed(lambda: run_ragged(net, src, tgt, sl, tl, iter=it), a.reps)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            run_ragged(net, src, tgt, sl, tl, iter=it)
        torch.cuda.current_stream().wait_stream(s)
        with torch.cuda.graph(g):
            run_ragged(net, src, tgt, sl, tl, iter=it)
        r["ragged_graph_ms"] = timed(g.replay, a.reps)

        def per_pair():
            for b in range(P):
                V.vcrnetIter(net, src_l[b][None], tgt_l[b][None], iter=it)
        r["per_pair_ms"] = timed(per_pair, max(2, a.reps // 4))
        r[uniform + "_ms"] = timed(lambda: V.vcrnetIter(net, src_u, tgt_u, iter=it), a.reps)
        for k in ("ragged_eager", "ragged_graph", "per_pair", uniform):
            r[k + "_pairs_per_s"] = P / (r[k + "_ms"] * 1e-3)
        saved = config.cuda_graph
        config.cuda_graph = False
        try:
            kr = per_kernel(lambda: run_ragged(net, src, tgt, sl, tl, iter=it))
            ku = per_kernel(lambda: V.vcrnetIter(net, src_u, tgt_u, iter=it))
        finally:
            config.cuda_graph = saved
        if a.partial:                                   # every entry point, the ragged ones under their uniform name
            base = lambda n: n.replace("_ragged_keep", "").replace("_ragged", "")
            r["kernel_ms"] = {}
            for n, ms in kr.items():
                r["kernel_ms"].setdefault(base(n), {"ragged": 0.0, uniform: 0.0})["ragged"] += ms
            for n, ms in ku.items():
                r["kernel_ms"].setdefault(n, {"ragged": 0.0, uniform: 0.0})[uniform] += ms
        else:
            r["kernel_ms"] = {n: {"ragged": kr.get(n + "_ragged", 0.0), uniform: ku.get(n, 0.0)}
                              for n in ("vcr_knn_topk", "vcr_knn_topk_tc", "vcr_flash_attn_tc", "vcr_softcorr_tc",
                                        "vcr_svd_head")}
            r["kernel_ms"]["vcr_zero_padding"] = {"ragged": kr.get("vcr_zero_padding", 0.0), uniform: 0.0}
        r["total_c_abi_ms"] = {"ragged": sum(kr.values()), uniform: sum(ku.values())}
        res["iter"][str(it)] = r
        print(json.dumps({it: {k: v for k, v in r.items() if k.endswith("pairs_per_s")}}), flush=True)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
