"""Synthetic inputs and weights for benchmarks and demos of the B200 path (product-side; no test infrastructure).

The reference's trained checkpoints are not distributed (``.MISSING_LARGE_BLOBS``: pretrained/vcrnet-{whole,part}.t7) and
its dataset is a download (util/data.py:16-26), so a benchmark needs stand-ins of the right shape:

  * ``default_args``      the fields the module constructors read, with the reference's argparse defaults
                          (util/initPara.py:127-205)
  * ``state_dict``        the 59-key VCRNet state_dict (reference key order and shapes) drawn from nn.Linear / nn.Conv's
                          default distribution with a portable numpy RandomState; the embedding can be overridden by the
                          12 tensors of the one checkpoint the reference does ship (pretrained/lpd-pretrained.t7)
  * ``PairSource``        ModelNet40-shaped pairs generated ON THE DEVICE by the data step (vcr_net_b200/data.py, reference
                          util/data.py:247-329) from uniform base clouds (model/icp_model.py:124's distribution)
  * ``reserve_overlap2``  util/initPara.py:109-124's cubic for --overlap, by bisection (no sympy)
"""
from __future__ import annotations

import math
from argparse import Namespace
from collections import OrderedDict

import numpy as np


def default_args(partial=False, overlap2=0.75, **kw):
    a = dict(emb_dims=512, cycle=False, emb_nn="lpdnet", pointer="transformer", vcp_nn="topK", t3d=False, tfea=False,
             n_blocks=1, dropout=0.0, ff_dims=1024, n_heads=4, overlap2=overlap2, partial=partial, num_points=1024,
             iter=1, model="vcrnet", loss="point", max_iterations=50)
    a.update(kw)
    return Namespace(**a)


def reserve_overlap2(overlap: float):
    """-> (reserve, overlap2) as util/initPara.py:109-124 derives them from --overlap."""

    def f(n):
        a = (n - 1.5 * n * n) * (1.0 - 2.0 * n)
        b = 0.5 * (n - 1.0) ** 2 * n - (1.0 - n) ** 3 / 6.0 + (1.0 - 2.0 * n) ** 3 / 6.0
        return ((a + b) * 2.0 + (1.0 - 2.0 * n) ** 3) / (1.0 - n) ** 2 - overlap

    lo, hi = 0.0, 0.5
    flo = f(lo)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if (f(mid) > 0) == (flo > 0):
            lo = mid
        else:
            hi = mid
    reserve = 1.0 - 0.5 * (lo + hi)
    return reserve, overlap / reserve


def state_dict(seed: int = 1234, emb_dims: int = 512, ff_dims: int = 1024, emb_weights=None):
    """59-key VCRNet(lpdnet, transformer, topK) state_dict as torch tensors, reference key order."""
    import torch
    rs = np.random.RandomState(seed)
    sd = OrderedDict()

    def dense(name, o, i, extra=()):
        bound = 1.0 / math.sqrt(i)
        sd[f"{name}.weight"] = rs.uniform(-bound, bound, size=(o, i)).astype(np.float32).reshape((o, i) + extra)
        sd[f"{name}.bias"] = rs.uniform(-bound, bound, size=(o,)).astype(np.float32)

    def norm(name):
        sd[f"{name}.a_2"] = np.ones(emb_dims, np.float32)
        sd[f"{name}.b_2"] = np.zeros(emb_dims, np.float32)

    dense("emb_nn.convDG1.0", 128, 128, (1, 1))
    dense("emb_nn.convDG2.0", 128, 128, (1, 1))
    dense("emb_nn.convSN1.0", 256, 256, (1, 1))
    dense("emb_nn.conv1_lpd", 64, 3, (1,))
    dense("emb_nn.conv2_lpd", 64, 64, (1,))
    dense("emb_nn.conv3_lpd", emb_dims, 512, (1,))
    for side, attns, nsub in (("encoder", ("self_attn",), 2), ("decoder", ("self_attn", "src_attn"), 3)):
        pre = f"pointer.model.{side}"
        for att in attns:
            for i in range(4):
                dense(f"{pre}.layers.0.{att}.linears.{i}", emb_dims, emb_dims)
        dense(f"{pre}.layers.0.feed_forward.w_1", ff_dims, emb_dims)
        dense(f"{pre}.layers.0.feed_forward.w_2", emb_dims, ff_dims)
        for i in range(nsub):
            norm(f"{pre}.layers.0.sublayer.{i}.norm")
        norm(f"{pre}.norm")
    sd["svd.reflect"] = np.diag([1.0, 1.0, -1.0]).astype(np.float32)
    if emb_weights is not None:
        for k, v in emb_weights.items():
            assert k in sd and sd[k].shape == tuple(v.shape), (k, tuple(v.shape))
            sd[k] = np.asarray(v, dtype=np.float32)
    return OrderedDict((k, torch.from_numpy(np.ascontiguousarray(v)).clone()) for k, v in sd.items())


class PairSource:
    """Device-resident synthetic dataset: ``n_items`` base clouds of ``base_points`` uniform points in [-0.5, 0.5)^3 (seeded)
    and the reference's per-item pair construction run by the CUDA data step.  ``batch(first, count)`` -> dict of device
    tensors (src, tgt, R_ab, t_ab, R_ba, t_ba, euler_ab, euler_ba) for items first .. first+count-1."""

    def __init__(self, n_items, device, num_points=1024, partial=False, reserve=1.0, base_points=2048, seed=1234,
                 aligned=False):
        import torch
        from .data import PairGenerator
        base_points = max(base_points, num_points)
        base = np.random.RandomState(seed).rand(n_items, base_points, 3).astype(np.float32) - 0.5
        self.n_items = n_items
        self.gen = PairGenerator(torch.from_numpy(base).to(device), num_points=num_points, partial=partial,
                                 reserve=reserve, aligned=aligned)

    def batch(self, first, count):
        assert first + count <= self.n_items
        return self.gen.batch(range(first, first + count))

    def batch_ragged(self, first, count, num_points, n_max=None):
        """batch() as a ragged batch, item first + i at num_points[i] points (PairGenerator.batch_ragged)."""
        assert first + count <= self.n_items
        return self.gen.batch_ragged(range(first, first + count), num_points, n_max)
