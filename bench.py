#!/usr/bin/env python
"""bench.py -- registration pairs/sec of the B200-native VCR-Net inference path.

Contract (task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.  A "step" = one
pass of the hot path (vcrnetIter: LPDNet embedding of both clouds -> Transformer pointer -> VCP head -> SVD head, all --iter
iterations) over one batch of synthetic ModelNet40-shaped pairs.  Headline workload at every N: BASELINE.json configs[1]
"partial-to-partial eval, overlap 0.575 crops (768 of 1024 pts), --iter 3, batch 24" per GPU (weak scaling: each rank
registers its own batch, no collective on the data path).

  value      pairs/s, inputs resident in HBM, CUDA events per step on the launching stream, L2 flushed between steps; the
             product's default path (module API `vcrnetIter`: loop invariants hoisted, repeated shapes replayed from a CUDA
             graph -- both bit-identical to the plain loop, which is reported as `variant_eager` / `variant_no_hoisting`)
  e2e        same metric from pinned HOST buffers: H2D of src/tgt + vcrnetIter + D2H of R_ab, t_ab, R_ba, t_ba (what the
             reference's test loop pulls back, model/vcrnet_model.py:570-580) inside the timed region
  roofline   dominant C-ABI entry point: algorithmic FLOP or bytes per launch / CUDA-event launch time vs
             MEASURED_PEAKS.json; `rooflines` lists the same for the kNN, attention, key-statistic, soft-correspondence and
             LayerNorm kernels (north_star asks for kNN and attention explicitly)
  cpu_baseline   the reference's own `vcrnetIter` on this box's host cores (oracle/_ref, kind "reference") when the
             staged reference travelled with the snapshot, else the torch-CPU port (oracle/vcr_oracle_torch.py, kind "port");
             `--impl reference` makes that the measured arm, at the GPU arm's batch size
  other_workloads   configs[0] (whole-to-whole, 1024 pts, batch 16, iter 1) with its own cpu_baseline; configs[3]
             (4096 pts, 256 pairs split over the N ranks = strong scaling, in micro-batches of 32); configs[2] (LPD
             pre-training forward + loss + hand-written backward, batch 16; e2e copies the loss back)
  variants   single-pass fp16 / bf16 tensor modes with the tolerance tests/test_gpu_parity.py asserts for them; batch-1
             latency
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

LPD_WEIGHTS = os.path.join(ROOT, "tests", "golden", "lpd_pretrained_weights.npz")   # the reference's shipped emb_nn tensors


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="partial", choices=["whole", "partial", "lpd-train", "cfg4"])
    ap.add_argument("--batch", type=int, default=0, help="pairs per GPU per step (default: config's)")
    ap.add_argument("--num-points", type=int, default=0)
    ap.add_argument("--precision", default=os.environ.get("VCR_PRECISION", "h3"),
                    choices=["fp32", "h3", "fp16", "bf16"],
                    help="matrix engine: fp32 SIMT | h3 = tcgen05 3-term fp16 split (fp32 parity) | fp16 | bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--cpu-sample-pairs", type=int, default=0, help="pairs in the cpu_baseline sample (default: one batch)")
    ap.add_argument("--cpu-kind", default="auto", choices=["auto", "reference", "port"])
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference: where the reference's own code runs (cpu = the contract's reference arm; cuda = the "
                         "stock PyTorch path of the unmodified reference on this GPU, context only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what rank 0's last timed step returned as DIR/<name>.npy (float32 / "
                         "float64; a training step adds the parameter gradients as grad.<parameter>); above 64 MB in all, "
                         "the per-pair outputs are cut to a fixed seeded sample of pairs, listed in pair_index.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return a


def workload_cfg(a, name=None, world=1):
    from vcr_net_b200 import synthetic
    name = name or a.workload
    reserve, overlap2 = synthetic.reserve_overlap2(0.575)
    if name == "lpd-train":
        return dict(key=name, name="LPDNet pre-train forward+backward (LPD loss), index-aligned pairs, 1024 pts",
                    partial=False, iters=1, batch=a.batch or 16, overlap2=0.75, reserve=1.0, train=True,
                    num_points=a.num_points or 1024, micro=0)
    if name == "whole":
        return dict(key=name, name="VCR-Net whole-to-whole eval, synthetic ModelNet40-shaped pairs, 1024 pts, iter=1",
                    partial=False, iters=1, batch=a.batch or 16, overlap2=0.75, reserve=1.0,
                    num_points=a.num_points or 1024, micro=0)
    if name == "cfg4":       # BASELINE.json configs[3]: 4096 pts/cloud, batch 256 sharded over the ranks (strong scaling)
        total = a.batch or 256
        return dict(key=name, name="Scaled inference: whole-to-whole, 4096 pts/cloud, 256 pairs per step split across the "
                                   "ranks, iter=1", partial=False, iters=1, batch=max(1, total // world), overlap2=0.75,
                    reserve=1.0, num_points=a.num_points or 4096, micro=32, strong=True, total=total)
    return dict(key="partial", name="VCR-Net partial-to-partial eval, overlap=0.575 crops (768 of 1024 pts), iter=3",
                partial=True, iters=3, batch=a.batch or 24, overlap2=overlap2, reserve=reserve,
                num_points=a.num_points or 1024, micro=0)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path on the host cores (bounded sample)
# ------------------------------------------------------------------------------------------------

PORT_DESC = ("oracle/vcr_oracle_torch.py: the reference's registration loop restated on torch CPU operators (same ATen "
             "kernels, fp32, all host threads); parity-checked against the live-reference golden vectors")
REF_DESC = ("the reference's own model/vcrnet_model.py vcrnetIter(VCRNet(args).eval(), src, tgt, iter) imported unmodified "
            "from oracle/_ref (staged copy of qiaozhijian/VCR-Net), torch CPU, fp32, all host threads")


def cpu_kind(a):
    from oracle import build_ref
    if a.cpu_kind == "port":
        return "port"
    if build_ref.staged():
        return "reference"
    if a.cpu_kind == "reference":
        raise SystemExit("bench.py: --cpu-kind reference needs the staged reference (python -m oracle.build_ref)")
    return "port"


class CpuArm:
    """Runs in a process where CUDA is hidden (the reference picks 'cuda' whenever torch.cuda.is_available(),
    model/vcrnet_model.py:216)."""

    def __init__(self, cfg, kind, device="cpu"):
        import torch
        from oracle import synth
        torch.set_num_threads(os.cpu_count())
        self.cfg, self.kind, self.torch, self.device = cfg, kind, torch, device
        lpd = dict(np.load(LPD_WEIGHTS))
        self.ckpt = synth.make_checkpoint(1234, emb_weights=lpd)
        if kind == "reference":
            from oracle import ref_harness
            ref = ref_harness.import_reference()
            self.VM = ref.vcrnet_model
            args = ref_harness.default_args(partial=cfg["partial"], overlap2=cfg["overlap2"], iter=cfg["iters"],
                                            num_points=cfg["num_points"])
            self.net = self.VM.VCRNet(args).eval()
            self.net.load_state_dict(synth.checkpoint_to_torch(self.ckpt), strict=True)
            self.net = self.net.to(device)

    def pairs(self, n, first=0):
        from oracle import synth
        c = self.cfg
        return synth.make_pairs(n, c["num_points"], partial=c["partial"], reserve=c["reserve"] if c["partial"] else 1.0,
                                first_item=first, base_points=max(2048, c["num_points"]))

    def run(self, p):
        """-> seconds for one pass over the pairs in p."""
        torch, c = self.torch, self.cfg
        t0 = time.perf_counter()
        if self.kind == "reference":
            with torch.no_grad():
                out = self.VM.vcrnetIter(self.net, torch.from_numpy(p["src"]).to(self.device),
                                         torch.from_numpy(p["tgt"]).to(self.device), iter=c["iters"])
                if self.device != "cpu":
                    out[2].cpu()                                    # the loop pulls the poses back (:570-580): includes the sync
        else:
            from oracle import vcr_oracle_torch as OT
            OT.vcrnet_iter(self.ckpt, p["src"], p["tgt"], c["iters"], partial=c["partial"], overlap2=c["overlap2"])
        return time.perf_counter() - t0


def run_reference_arm(a, cfg, rank, world):
    """`--impl reference`: the reference's CPU implementation on rank 0's host cores, same config as the GPU arm.  Each step
    is one batch of the GPU arm's size unless that would push K + W steps past ~4 minutes, in which case the batch is cut
    (and the line says so)."""
    if rank != 0:
        return
    kind = cpu_kind(a)
    on_gpu = a.ref_device == "cuda"
    if on_gpu and kind != "reference":
        raise SystemExit("bench.py: --ref-device cuda needs the staged reference (python -m oracle.build_ref)")
    arm = CpuArm(cfg, kind, device="cuda" if on_gpu else "cpu")
    n = a.cpu_sample_pairs or cfg["batch"]
    budget_s = 240.0
    times = []
    p = arm.pairs(n)
    total_steps = a.warmup + a.steps
    if total_steps > 1:
        dt0 = arm.run(p)                                      # untimed: first touch of weights / thread pool
        if dt0 * total_steps > budget_s and not a.cpu_sample_pairs:
            n = max(2, int(n * budget_s / (dt0 * total_steps)))
            p = arm.pairs(n)
    for i in range(total_steps):
        dt = arm.run(p)
        if i >= a.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = n / (ms / 1e3)
    cores = os.cpu_count()
    M = int(p["src"].shape[2])
    line = {
        "impl": "reference" if not on_gpu else "reference-on-gpu (stock PyTorch, context only)",
        "metric": "pairs/sec @1024 pts", "value": value, "unit": "pairs/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "batch_per_gpu": n, "num_points": cfg["num_points"], "points_in_net": M,
                   "iter": cfg["iters"], "precision": "fp32 (torch CPU)" if not on_gpu else "fp32 (stock torch CUDA kernels, TF32 off for matmul)",
                   "parallelism": "host cores of rank 0 only" if not on_gpu else "one GPU, the reference's own nn.Module path",
                   "weights": "synthetic 59-key checkpoint"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind,
                         "sample": f"{n} pairs per step ({'the GPU arm batch' if n == cfg['batch'] else 'a bounded sample'}) "
                                   f"through {REF_DESC if kind == 'reference' else PORT_DESC}"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def cpu_baseline_subprocess(a, cfg, pairs, device="cpu", steps=1, warmup=0):
    """cpu_baseline leg of the GPU arm: one pass in a child process with CUDA hidden; returns the child's cpu_baseline dict.
    device="cuda": the same child runs the reference's stock PyTorch path on this GPU instead (context only)."""
    env = dict(os.environ)
    if device == "cpu":
        env["CUDA_VISIBLE_DEVICES"] = ""
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "LOCAL_WORLD_SIZE", "GROUP_RANK",
              "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", cfg["key"], "--steps", str(steps),
           "--warmup", str(warmup), "--cpu-sample-pairs", str(pairs), "--cpu-kind", a.cpu_kind, "--ref-device", device,
           "--num-points", str(cfg["num_points"]), "--batch", str(cfg["batch"])]
    try:
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
        line = json.loads(r.stdout.strip().splitlines()[-1])
        cb = line["cpu_baseline"]
        if device != "cpu":
            return {"value": line["value"], "unit": "pairs/s", "ms_per_step": line["ms_per_step"], "batch": pairs,
                    "what": "the unmodified reference's own vcrnetIter on THIS GPU through stock PyTorch CUDA kernels "
                            "(oracle/_ref; fp32, cuDNN/cuBLAS defaults), device-resident inputs, poses pulled back per step; "
                            "context only -- the contract's reference arm is the CPU path"}
        cb["sample"] = (f"{pairs} pairs of the same workload, one pass ({line['ms_per_step'] / 1e3:.1f} s) through "
                        + cb["sample"].split("through ", 1)[1])
        return cb
    except Exception as e:                                   # reporting leg: never lose the GPU measurement over it
        return {"value": None, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": f"failed: {e!r}"}


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------

class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def build_net(cfg, dev):
    import torch
    import vcr_net_b200 as V
    from vcr_net_b200 import synthetic
    lpd = dict(np.load(LPD_WEIGHTS))
    if cfg.get("train"):   # BASELINE config 3: LPD(args) forward + loss + backward (model/lpdnet_model.py:140-229)
        net = V.LPD(synthetic.default_args(model="lpd", num_points=cfg["num_points"])).to(dev).train()
        net.load_state_dict({k: torch.from_numpy(v) for k, v in lpd.items()}, strict=True)
        return net
    net = V.VCRNet(synthetic.default_args(partial=cfg["partial"], overlap2=cfg["overlap2"])).to(dev).eval()
    net.load_state_dict(synthetic.state_dict(1234, emb_weights=lpd), strict=True)
    return net


def measure(cfg, rank, world, dev, local_rank, steps, warmup, profile=False, clocks=False, e2e=True, dump=False):
    """Time `steps` steps of one workload on this rank's GPU through the module API.  -> per-rank sums (ms) etc.
    dump: res["outputs"] = (per-pair arrays, other arrays) of the last timed step, as host float32 / float64."""
    import torch
    import torch.distributed as dist
    import vcr_net_b200 as V
    from vcr_net_b200 import config as vcfg
    from vcr_net_b200 import graph as vgraph
    from vcr_net_b200 import synthetic
    from vcr_net_b200._lib import lib
    L = lib()
    train = bool(cfg.get("train"))
    net = build_net(cfg, dev)
    B = cfg["batch"]
    micro = min(cfg.get("micro") or B, B)               # cfg4: a step = B pairs registered in micro-batches
    nbatches = 2
    # each rank registers its own pairs: items (rank*nbatches + j)*B .. +B-1, generated on the device by the data step
    source = synthetic.PairSource((world * nbatches) * B, dev, num_points=cfg["num_points"], partial=cfg["partial"],
                                  reserve=cfg["reserve"] if cfg["partial"] else 1.0,
                                  base_points=max(2048, cfg["num_points"]), aligned=train)
    devb = []
    for j in range(nbatches):
        b = source.batch((rank * nbatches + j) * B, B)
        devb.append((b["src"], b["tgt"]))
    host = [(s.cpu().pin_memory(), t.cpu().pin_memory()) for s, t in devb]
    del source
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
    stream = torch.cuda.current_stream()

    def run(s, t):
        if train:
            net.zero_grad(set_to_none=True)
            out = net(s, t)
            out[2].backward()
            return out
        if micro >= B:
            return V.vcrnetIter(net, s, t, iter=cfg["iters"])
        outs = [V.vcrnetIter(net, s[i:i + micro], t[i:i + micro], iter=cfg["iters"]) for i in range(0, B, micro)]
        return tuple(torch.cat([o[k] for o in outs]) for k in range(6))

    def step(i):
        return run(*devb[i % nbatches])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def launches():
        return L.vcr_launch_count() + vgraph.replayed_launches

    res = {"B": B, "M": int(devb[0][0].shape[2])}
    with (torch.enable_grad() if train else torch.no_grad()):
        for i in range(max(warmup, 3)):                 # >= 3: eager call, graph capture, first replay
            step(i)
        barrier()
        clk = Clocks(local_rank) if clocks else None
        if clk:
            clk.start()
        # ---- device-resident timing -------------------------------------------------------------
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = launches()
        barrier()
        t_wall0 = time.perf_counter()
        for i in range(steps):
            flush.fill_(float(i))                     # L2 flush, outside the per-step event bracket
            ev[i][0].record(stream)
            out = step(i)
            ev[i][1].record(stream)
            if i < steps - 1:
                del out                               # only the last step's outputs outlive the step
        barrier()
        res["wall_s"] = time.perf_counter() - t_wall0
        res["launches"] = launches() - l0
        res["ms_total"] = sum(e0.elapsed_time(e1) for e0, e1 in ev)
        if dump:                                      # before the e2e steps recompute the gradients
            to_host = lambda t: t.detach().to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()
            names = (("src_embedding", "tgt_embedding", "loss", "mse_ab", "mae_ab") if train else
                     ("srcK", "src_corrK", "R_ab", "t_ab", "R_ba", "t_ba"))
            outs = {n: to_host(o) for n, o in zip(names, out)}
            per_pair = {n: v for n, v in outs.items() if v.ndim and v.shape[0] == B}
            other = {n: v for n, v in outs.items() if n not in per_pair}
            if train:
                other.update(("grad." + n, to_host(p.grad)) for n, p in net.named_parameters() if p.grad is not None)
            res["outputs"] = (per_pair, other)
        del out
        res["ms_e2e"], res["h2d"], res["d2h"] = float("nan"), 0, 0
        if e2e:
            # ---- end-to-end: pinned host -> device -> vcrnetIter -> host --------------------------------
            pose_host = [torch.empty(sh, dtype=torch.float32).pin_memory() for sh in ((B, 3, 3), (B, 3), (B, 3, 3), (B, 3))]
            sbuf, tbuf = torch.empty_like(devb[0][0]), torch.empty_like(devb[0][1])

            def e2e_step(i):
                hs, ht = host[i % nbatches]
                sbuf.copy_(hs, non_blocking=True)
                tbuf.copy_(ht, non_blocking=True)
                out = run(sbuf, tbuf)
                if train:
                    pose_host[1][0, :1].copy_(out[2].detach().reshape(1), non_blocking=True)       # the loss
                else:
                    for h, o in zip(pose_host, out[2:6]):                                          # R_ab, t_ab, R_ba, t_ba
                        h.copy_(o, non_blocking=True)

            for i in range(2):
                e2e_step(i)
            barrier()
            ee = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for i in range(steps):
                flush.fill_(float(i))
                ee[i][0].record(stream)
                e2e_step(i)
                ee[i][1].record(stream)
            barrier()
            res["ms_e2e"] = sum(e0.elapsed_time(e1) for e0, e1 in ee)
            res["h2d"] = 2 * B * 3 * res["M"] * 4
            res["d2h"] = 4 if train else B * (9 + 3 + 9 + 3) * 4
        res["clocks"] = clk.stop() if clk else None
        # ---- per-kernel CUDA-event profile of the same step (roofline leg): eager launches, one event pair per C-ABI call
        res["prof"], res["nprof"] = [], 3
        if profile:
            old = vcfg.cuda_graph
            vcfg.cuda_graph = False
            try:
                step(0)
                L.profile_begin()
                for i in range(res["nprof"]):
                    flush.fill_(1.0)
                    # park the stream for ~10 ms so the host enqueues the whole step before the GPU starts it: each event
                    # pair then brackets pure kernel time, not the Python -> ctypes launch gap of a starved GPU
                    torch.cuda._sleep(20_000_000)
                    step(i)
                res["prof"] = L.profile_end()
            finally:
                vcfg.cuda_graph = old
    net.__dict__.pop("_vcr_graph_cache", None)
    del net, devb, flush
    torch.cuda.empty_cache()
    return res


DUMP_BYTES = 64 * 10**6


def dump_outputs(path, per_pair, other):
    """--dump-outputs: write every array as path/<name>.npy.  When they would pass DUMP_BYTES, the arrays indexed by pair
    keep the same seeded sample of pairs (pair_index.npy), so that two runs with the same arguments write the same files."""
    os.makedirs(path, exist_ok=True)
    header = 4096                                             # bound on one .npy header, with room to spare
    pairs = next(iter(per_pair.values())).shape[0] if per_pair else 0
    room = DUMP_BYTES - sum(v.nbytes for v in other.values()) - header * (len(per_pair) + len(other) + 1)
    pair_bytes = sum(v.nbytes for v in per_pair.values()) // max(pairs, 1)
    if pair_bytes * pairs > room:
        keep = np.sort(np.random.RandomState(0).choice(pairs, max(room, 0) // (pair_bytes + 8), replace=False))
        per_pair = {n: v[keep] for n, v in per_pair.items()}
        other = dict(other, pair_index=keep.astype(np.float64))
    for n, v in {**per_pair, **other}.items():
        np.save(os.path.join(path, n + ".npy"), v)


def reduce_max(world, dev, *vals):
    if world == 1:
        return vals
    import torch
    import torch.distributed as dist
    tt = torch.tensor(list(vals), dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return tuple(float(x) for x in tt)


def reduce_sum_int(world, dev, v):
    if world == 1:
        return int(v)
    import torch
    import torch.distributed as dist
    t = torch.tensor([int(v)], dtype=torch.int64, device=dev)
    dist.all_reduce(t)
    return int(t[0])


def ncu_evidence(kernel):
    """DRAM traffic / pipe activity of `kernel` from the committed `ncu --set full` capture (profiles/*_ncu_traffic.json)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json")))
    if not files:
        return None
    try:
        d = json.load(open(files[-1])).get(kernel)
        if d:
            d = dict(d, file=os.path.relpath(files[-1], ROOT))
        return d
    except Exception:
        return None


def algorithmic_work(name, kw):
    """(flops, bytes) of one C-ABI call from its arguments -- SURVEY.md section 8(d)'s per-unit figures."""
    g = kw.get
    try:
        if name in ("vcr_gemm_f32", "vcr_gemm_tc"):
            return 2.0 * g("M") * g("N") * g("K") * g("nb_outer") * g("nb_inner"), 0.0
        if name == "vcr_flash_attn_tc":                  # QK^T + PV: 4 Nq Nk dk per (batch, head)
            return 4.0 * g("Nq") * g("Nk") * g("dk") * g("B") * g("H"), 0.0
        if name == "vcr_attn_colsum_tc":                 # two QK^T sweeps
            return 2.0 * 2.0 * g("Nq") * g("Nk") * g("dk") * g("B") * g("H"), 0.0
        if name in ("vcr_softcorr_tc", "vcr_softcorr_best_tc"):
            return (2.0 * g("D") + 6.0) * g("Ns") * g("Nt") * g("B"), 0.0
        if name in ("vcr_knn_topk", "vcr_knn_topk_tc"):  # 2 D N^2 flop per cloud; 4 D N in + 4 k N out bytes
            B, D, N, k = g("B"), g("D"), g("N"), g("k")
            return 2.0 * D * N * N * B, (4.0 * D * N + 4.0 * k * N) * B
        if name == "vcr_layernorm_operand":              # fp32 [M, D] in, `planes` 16-bit planes out
            return 0.0, (4.0 + 2.0 * g("planes")) * g("M") * g("D")
        if name in ("vcr_layernorm", "vcr_layernorm_head"):
            return 0.0, 2.0 * 4.0 * g("M") * g("D")
        if name == "vcr_to_operand":
            return 0.0, (4.0 + 2.0 * g("planes")) * g("rows") * g("cols")
        if name == "vcr_wgrad_f32":
            return 2.0 * g("M") * g("N") * g("K"), 4.0 * g("M") * (g("N") + g("K")) + 4.0 * g("N") * g("K")
        if name == "vcr_gather_max":                     # 4 k C bytes gathered + 4 C read + 4 C written per point
            return 0.0, (4.0 * g("k") * g("C") + 2 * 4.0 * g("C")) * g("total_pts")
    except TypeError:
        pass
    return 0.0, 0.0


def rooflines_from_profile(prof, nprof, precision, peaks, protos):
    agg = {}
    for name, ms, args in prof:
        names = [n for _, n in protos[name][1]]
        kw = dict(zip(names, args))
        key = name
        if name == "vcr_knn_topk":
            key = "vcr_knn_topk[D=%d]" % kw.get("D", 0)
        d = agg.setdefault(key, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0, "entry": name})
        fl, by = algorithmic_work(name, kw)
        d["ms"] += ms; d["n"] += 1; d["flops"] += fl; d["bytes"] += by
    step_ms = sum(d["ms"] for d in agg.values()) / max(nprof, 1)
    tpeak = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm = peaks.get("hbm_gbs", 6650.0)
    src = "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 1.4 PFLOP/s / 6650 GB/s (of fallback)"
    tensor_entries = ("vcr_gemm_tc", "vcr_flash_attn_tc", "vcr_attn_colsum_tc", "vcr_softcorr_tc", "vcr_softcorr_best_tc",
                      "vcr_knn_topk_tc")
    out = {}
    for key, d in agg.items():
        entry = d["entry"]
        r = {"kernel": key, "launches_per_step": d["n"] / nprof, "avg_launch_ms": d["ms"] / d["n"],
             "share_of_step": d["ms"] / nprof / step_ms if step_ms else None}
        tensor_bound = entry in tensor_entries or entry == "vcr_gemm_f32" or (entry == "vcr_knn_topk" and "D=3" not in key)
        if tensor_bound and d["flops"] > 0:
            ach = d["flops"] / (d["ms"] / 1e3) / 1e12
            passes = 3 if (precision == "h3" and entry in tensor_entries) else 1
            r.update(bound="tensor", achieved=ach, peak=tpeak, unit="TFLOP/s", frac=ach / tpeak, peak_source=src,
                     tensor_passes_per_product=passes, tensor_work_frac=passes * ach / tpeak)
            if entry in ("vcr_gemm_f32", "vcr_knn_topk"):
                r["note"] = "FP32 SIMT kernel (exact fp32 chain) measured against the dense bf16 tensor peak"
            elif entry == "vcr_knn_topk_tc":
                r["note"] = ("tcgen05 distance tiles as a certified prefilter (3 fp16 passes) + exact fp32 re-rank; the "
                             "selection, not the distance flops, is the cost")
            elif passes == 3:
                r["note"] = ("achieved = algorithmic flops / CUDA-event launch time; the h3 parity mode issues 3 fp16 tensor "
                             "passes per product, so the tensor pipe does tensor_work_frac of the measured bf16 peak")
        elif d["bytes"] > 0:
            ach = d["bytes"] / (d["ms"] / 1e3) / 1e9
            r.update(bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm, peak_source=src,
                     note="achieved = algorithmic bytes (operands streamed once) / CUDA-event launch time"
                          + ("; moves ~12 bytes per point: ALU/selection-bound, not bandwidth-bound (SURVEY 8d caveat)"
                             if "knn" in key else ""))
            if d["flops"] > 0:
                r["fp32_tflops"] = d["flops"] / (d["ms"] / 1e3) / 1e12
        else:
            continue
        ev = ncu_evidence(key) or (ncu_evidence(entry) if key == entry else None)
        r["traffic"] = ev["mean_dram_bytes_per_launch"] if ev else None
        if ev:
            r["ncu"] = ev
        out[key] = r
    breakdown = {k: round(v["ms"] / nprof, 4) for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}
    top = max(agg.items(), key=lambda kv: kv[1]["ms"])[0] if agg else None
    return out, top, breakdown


def run_gpu_arm(a, cfg, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=b200) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from vcr_net_b200 import config as vcfg
    from vcr_net_b200._lib import lib
    vcfg.set_precision(a.precision)
    train = bool(cfg.get("train"))
    extras = not a.no_other_workloads and not train and a.workload == "partial"

    def pairs_per_s(r, steps, key="ms_total"):
        (m,) = reduce_max(world, dev, r[key])
        return r["B"] * steps * world / (m / 1e3), m / steps

    r = measure(cfg, rank, world, dev, local_rank, a.steps, a.warmup, profile=True, clocks=True,
                dump=bool(a.dump_outputs) and rank == 0)
    if "outputs" in r:
        dump_outputs(a.dump_outputs, *r.pop("outputs"))
    ms_total, ms_e2e = reduce_max(world, dev, r["ms_total"], r["ms_e2e"])
    launches = reduce_sum_int(world, dev, r["launches"])

    short = max(5, a.steps // 2)
    variants, other = {}, {}
    if extras:
        def variant(label, note, **switch):
            old = {k: getattr(vcfg, k) for k in switch}
            for k, v in switch.items():
                setattr(vcfg, k, v)
            try:
                rv = measure(cfg, rank, world, dev, local_rank, short, 3)
            finally:
                for k, v in old.items():
                    setattr(vcfg, k, v)
            v, ms = pairs_per_s(rv, short)
            e, _ = pairs_per_s(rv, short, "ms_e2e")
            variants[label] = {"value": v, "e2e": e, "unit": "pairs/s", "ms_per_step": ms, "steps": short, "note": note}

        variant("variant_eager", "VCR_CUDA_GRAPH=0: every call through the eager Python -> ctypes launch sequence "
                "(bit-identical outputs to the headline)", cuda_graph=False)
        variant("variant_no_hoisting", "VCR_HOIST=none: emb_nn(tgt), encoder(tgt) and the decoder's first self-attention "
                "sublayer on tgt recomputed in every --iter iteration, i.e. exactly the work the reference does per iteration "
                "(bit-identical outputs to the headline)", hoist="none")
        for prec, tol in (("fp16", "3e-3"), ("bf16", "3e-2")):
            variant("variant_" + prec, f"single-pass {prec} tensor GEMMs / attention (VCP logits keep the 3-term split); "
                    f"NOT fp32 parity: Transformer output within {tol} relative of the reference, asserted by "
                    "tests/test_gpu_parity.py::test_throughput_modes_reported_tolerance", precision=prec)
        # batch-1 latency (one pair per call), graph replay vs eager
        lat = {}
        for label, g in (("cuda_graph", True), ("eager", False)):
            old = vcfg.cuda_graph
            vcfg.cuda_graph = g
            try:
                rl = measure(dict(cfg, batch=1), rank, world, dev, local_rank, 10, 3, e2e=False)
            finally:
                vcfg.cuda_graph = old
            (m,) = reduce_max(world, dev, rl["ms_total"])
            lat[label + "_ms_per_pair"] = m / 10
        variants["latency_batch1"] = dict(lat, note="one pair per vcrnetIter call (all --iter iterations), device-resident inputs")
        # the other BASELINE configs, short, same timing rules
        a1 = argparse.Namespace(**vars(a)); a1.batch = 0; a1.num_points = 0
        for wl in ("whole", "cfg4", "lpd-train"):
            c2 = workload_cfg(a1, wl, world)
            st2 = 3 if wl == "cfg4" else short
            r2 = measure(c2, rank, world, dev, local_rank, st2, 3)
            v2, ms2 = pairs_per_s(r2, st2)
            e2, _ = pairs_per_s(r2, st2, "ms_e2e")
            other[wl] = {"workload": c2["name"], "value": v2, "unit": "pairs/s", "e2e": e2, "batch_per_gpu": r2["B"],
                         "micro_batch": min(c2.get("micro") or r2["B"], r2["B"]), "ms_per_step": ms2, "steps": st2,
                         "scaling": "strong" if c2.get("strong") else "weak"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    B, M, clk, t_wall = r["B"], r["M"], r["clocks"], r["wall_s"]
    pairs_total = B * a.steps * world
    value = pairs_total / (ms_total / 1e3)
    e2e_value = pairs_total / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    roofs, top, breakdown = rooflines_from_profile(r["prof"], r["nprof"], a.precision, peaks, lib().protos)
    roof = roofs.get(top) if top else None
    if roof is None and top:
        roof = {"kernel": top, "bound": None, "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None}

    line = {
        "metric": "pairs/sec @1024 pts", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
        "scaling": "strong" if cfg.get("strong") else "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "h3": "f16x3-split+f32acc (fp32-equivalent)", "fp16": "f16", "bf16": "bf16"}[a.precision],
        "data": "synthetic",
        "config": {"workload": cfg["name"], "batch_per_gpu": B, "num_points": cfg["num_points"], "points_in_net": M,
                   "iter": cfg["iters"], "precision": a.precision, "parallelism": f"batch-shard x{world}, no collective",
                   "l2": "flushed between timed steps (256 MB fill)", "weights": "synthetic 59-key checkpoint",
                   "path": f"module API vcrnetIter; hoist={vcfg.hoist}; cuda_graph={'on' if vcfg.cuda_graph and not train else 'off'}"},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": int(launches),
        "roofline": roof,
        "rooflines": [v for k, v in roofs.items() if k != top and ("knn" in k or "flash" in k or "colsum" in k
                                                                   or "softcorr" in k or "layernorm_operand" in k
                                                                   or "gemm_tc" in k)],
        "kernel_ms_per_step": breakdown,
        "wall_s_timed_region": t_wall,
    }
    if other:
        line["other_workloads"] = other
    line.update(variants)
    if not a.no_cpu_baseline and not train and world == 1:      # rank 0 at N=1 only (task contract)
        line["cpu_baseline"] = cpu_baseline_subprocess(a, cfg, a.cpu_sample_pairs or min(cfg["batch"], 24))
        if "whole" in other:
            a1 = argparse.Namespace(**vars(a)); a1.batch = 0; a1.num_points = 0
            other["whole"]["cpu_baseline"] = cpu_baseline_subprocess(a, workload_cfg(a1, "whole", world), 16)
        if cpu_kind(a) == "reference" and not a.no_other_workloads:
            line["reference_on_this_gpu"] = cpu_baseline_subprocess(a, cfg, cfg["batch"], device="cuda", steps=5, warmup=2)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_STDOUT_FD = None


def emit(line):
    """Print the result line on the real stdout."""
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)
    if _STDOUT_FD is not None:
        os.dup2(2, 1)                                  # anything printed during teardown goes to stderr again


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference" and a.ref_device == "cpu":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""        # before torch is imported: the reference must stay on the host cores
    if a.gpus > 1 and "WORLD_SIZE" not in os.environ and a.impl != "reference":
        # launched as plain `python bench.py --gpus N`: re-exec one rank per GPU
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                  f"--nproc-per-node={a.gpus}", "--master-addr", "127.0.0.1", "--master-port",
                                  str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:])
    # stdout carries exactly ONE line (the JSON result): everything else a library prints there (e.g. NCCL's version banner
    # at communicator creation) is sent to stderr by pointing fd 1 at fd 2 until the result is emitted
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    cfg = workload_cfg(a, world=world)
    if a.impl == "reference":
        run_reference_arm(a, cfg, rank, world)
    else:
        run_gpu_arm(a, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
