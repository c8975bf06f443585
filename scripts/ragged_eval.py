"""A device-resident ragged evaluation against the same evaluation run one pair at a time.

24 pairs with seeded num_points in [512, 1024], whole and partial (synth.RESERVE_0575 / OVERLAP2_0575), h3, iter 1 and 3:
  (a) ragged    PairSource.batch_ragged (n_max 1024) -> vcrnetIterRagged / vcrnetIterRaggedPartial replayed from a graph
                captured once -> EvalAccumulator.update_ragged
  (b) per pair  PairGenerator(num_points=N_i).batch([item]) -> vcrnetIter (product default: the graph cache holds 4 shapes)
                -> EvalAccumulator.update, once per pair
Reported: pairs/s of both loops (CUDA events around `--reps` steps after a warm-up, host draws included); the device time of
the data step, one ragged call against the 24 per-item calls (CUDA events per C-ABI call, summed); the largest relative
difference between the two accumulators' metrics after one step.
Usage: python scripts/ragged_eval.py [--out profiles/ragged_eval.json]
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
from vcr_net_b200.data import EvalAccumulator, PairGenerator  # noqa: E402
from vcr_net_b200.synthetic import PairSource  # noqa: E402
from oracle import synth  # noqa: E402
from oracle.ref_harness import default_args  # noqa: E402

DEV = "cuda:0"


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def device_ms(fn):
    L = lib()
    L.profile_begin()
    fn()
    return sum(ms for _, ms, _ in L.profile_end())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/ragged_eval.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--pairs", type=int, default=24)
    a = ap.parse_args()
    config.set_precision("h3")
    config.cuda_graph = True
    P, n_max = a.pairs, 1024
    Ns = np.random.RandomState(2026).randint(512, n_max + 1, P).tolist()
    ckpt = synth.make_checkpoint(1234)
    res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                 capture_output=True, text=True).stdout.strip(),
           "pairs": P, "num_points": Ns, "n_max": n_max, "precision": "h3", "reps": a.reps, "runs": {}}
    for partial in (False, True):
        reserve, ov = (synth.RESERVE_0575, synth.OVERLAP2_0575) if partial else (1.0, 0.75)
        kind = "partial" if partial else "whole"
        net = V.VCRNet(default_args(partial=partial, overlap2=ov)).to(DEV).eval()
        net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=False)
        ps = PairSource(P, DEV, num_points=n_max, partial=partial, reserve=reserve)
        gens = [PairGenerator(ps.gen.base, num_points=n, partial=partial, reserve=reserve) for n in Ns]
        reg = V.vcrnetIterRaggedPartial if partial else V.vcrnetIterRagged
        d = ps.batch_ragged(0, P, Ns, n_max)
        src, tgt, lengths = d["src"].clone(), d["tgt"].clone(), d["lengths"].clone()
        corr = ragged.corr_lengths(lengths, ov) if partial else lengths
        data_ms = {"ragged": device_ms(lambda: ps.batch_ragged(0, P, Ns, n_max)),
                   "per_item": device_ms(lambda: [g.batch([b]) for b, g in enumerate(gens)])}
        for it in (1, 3):
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                reg(net, src, tgt, lengths, lengths, iter=it)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = reg(net, src, tgt, lengths, lengths, iter=it)

            def ragged_step(acc):
                q = ps.batch_ragged(0, P, Ns, n_max)
                src.copy_(q["src"]); tgt.copy_(q["tgt"]); lengths.copy_(q["lengths"])
                graph.replay()
                acc.update_ragged(src, tgt, lengths, out[0], out[1], corr, q["R_ab"], q["t_ab"], *out[2:])

            def per_pair_step(acc):
                for b, g in enumerate(gens):
                    q = g.batch([b])
                    o = V.vcrnetIter(net, q["src"], q["tgt"], iter=it)
                    acc.update(q["src"], q["tgt"], o[0], o[1], q["R_ab"], q["t_ab"], *o[2:])

            acc_r, acc_p = EvalAccumulator(DEV), EvalAccumulator(DEV)
            ragged_step(acc_r)
            per_pair_step(acc_p)
            rr, rp = acc_r.result(), acc_p.result()
            scratch = EvalAccumulator(DEV)
            r = {"ragged_ms": timed(lambda: ragged_step(scratch), a.reps),
                 "per_pair_ms": timed(lambda: per_pair_step(scratch), max(2, a.reps // 2))}
            r["ragged_pairs_per_s"] = P / (r["ragged_ms"] * 1e-3)
            r["per_pair_pairs_per_s"] = P / (r["per_pair_ms"] * 1e-3)
            r["metrics_ragged"], r["metrics_per_pair"] = rr, rp
            r["max_rel_diff"] = max(abs(rr[k] - rp[k]) / max(abs(rp[k]), 1e-300) for k in EvalAccumulator.KEYS)
            r["data_step_device_ms"] = data_ms
            res["runs"][f"{kind}_iter{it}"] = r
            print(json.dumps({f"{kind}_iter{it}": {k: v for k, v in r.items() if not k.startswith("metrics")}}),
                  flush=True)
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
