"""bench.py contract checks.  Without a GPU: the reference arm (`--impl reference`, the reference's loop on the host
cores) prints exactly ONE JSON line on stdout with the keys the driver reads, and the GPU arm refuses to run without a
device instead of falling back to the CPU.  On the GPU: `--dump-outputs` writes what the last timed step returned."""
import argparse
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*flags):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                          env=env, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pairs/sec @1024 pts" and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("VCR-Net partial-to-partial")          # BASELINE.json configs[1]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                          # the GPU arm itself is exercised by the driver / gpu_round.sh
    r = _run("--steps", "1", "--warmup", "0")
    assert r.returncode != 0 and r.stdout.strip() == "" and "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["partial", "lpd-train"])
def test_dump_outputs_are_the_last_timed_step(tmp_path, workload):
    """Two timed steps alternate between the bench's two batches, so the dump must hold the second batch's outputs.  The
    lpd-train step returns more than the 64 MB the dump may take: its per-pair embeddings are cut to a seeded sample."""
    import torch
    import bench
    import vcr_net_b200 as V
    from conftest import rel_err
    from vcr_net_b200 import synthetic
    d = tmp_path / "dump"
    r = _run("--steps", "2", "--warmup", "1", "--workload", workload, "--no-cpu-baseline", "--no-other-workloads",
             "--dump-outputs", str(d))
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([l for l in r.stdout.splitlines() if l.strip()]) == 1, r.stdout
    files = {os.path.basename(f)[:-4]: f for f in glob.glob(str(d / "*.npy"))}
    assert sum(os.path.getsize(f) for f in files.values()) <= bench.DUMP_BYTES
    got = {n: np.load(f) for n, f in files.items()}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())

    cfg = bench.workload_cfg(argparse.Namespace(batch=0, num_points=0, workload=workload))
    B, dev = cfg["batch"], "cuda:0"
    train = bool(cfg.get("train"))
    source = synthetic.PairSource(2 * B, dev, num_points=cfg["num_points"], partial=cfg["partial"],
                                  reserve=cfg["reserve"] if cfg["partial"] else 1.0, base_points=max(2048, cfg["num_points"]),
                                  aligned=train)
    b = source.batch(B, B)                                    # batch 1: the one the second (last) timed step registers
    net = bench.build_net(cfg, dev)
    if train:
        assert set(got) == {"src_embedding", "tgt_embedding", "loss", "mse_ab", "mae_ab", "pair_index"} | {
            "grad." + n for n, _ in net.named_parameters()}
        keep = got["pair_index"].astype(np.int64)
        assert 0 < len(keep) < B and np.array_equal(keep, np.unique(keep))
        out = net(b["src"], b["tgt"])
        out[2].backward()
        for n, o in zip(("src_embedding", "tgt_embedding"), out):
            assert rel_err(got[n], o.detach().cpu().numpy()[keep]) < 1e-5, n
        assert rel_err(got["loss"], out[2].item()) < 1e-5
        for n, p in net.named_parameters():
            assert rel_err(got["grad." + n], p.grad.cpu().numpy()) < 1e-5, n
    else:
        with torch.no_grad():
            out = V.vcrnetIter(net, b["src"], b["tgt"], iter=cfg["iters"])
        names = ("srcK", "src_corrK", "R_ab", "t_ab", "R_ba", "t_ba")
        assert set(got) == set(names)
        for n, o in zip(names, out):
            assert np.array_equal(got[n], o.cpu().numpy()), n
