"""Device-side data step (SURVEY.md section 8f row 2; reference util/data.py:247-309, 320-329).

The reference builds every pair on the host inside ``ModelNet40.__getitem__`` (numpy + scipy + sklearn) and ships
the clouds through a DataLoader.  Here the host only DRAWS what is random -- Euler angles, translation and the
permutations, from ``np.random.RandomState(item)`` in the reference's call order, a few KB per item -- and the
device gathers, applies the float64 rigid transform, crops the ``reserve`` fraction nearest to the last point and
casts to fp32 (csrc/datastep.cu).  The base clouds stay resident in HBM.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import ops, ragged
from ._lib import lib


def euler_to_R(ax, ay, az):
    """Rx.Ry.Rz exactly as util/data.py:262-278 builds R_ab."""
    cx, cy, cz, sx, sy, sz = math.cos(ax), math.cos(ay), math.cos(az), math.sin(ax), math.sin(ay), math.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]], dtype=np.float64)
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]], dtype=np.float64)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]], dtype=np.float64)
    return Rx @ Ry @ Rz


class PairGenerator:
    """base: device tensor [items, Nb, 3] fp32 (the dataset's point clouds, util/data.py:30-47 layout).

    ``batch(items)`` -> dict(src [P,3,M], tgt [P,3,M], R_ab, t_ab, R_ba, t_ba, euler_ab, euler_ba) on the device, the
    same values ``ModelNet40.__getitem__`` returns for test-partition items (np.random.seed(item), :255-256).
    ``batch_ragged(items, num_points)`` builds a ragged batch, one point count per item."""

    def __init__(self, base: torch.Tensor, num_points=1024, partial=False, reserve=1.0, factor=4.0, aligned=False):
        if not base.is_cuda:
            raise RuntimeError("PairGenerator: base clouds must live on a CUDA device (there is no CPU path)")
        assert base.dim() == 3 and base.shape[2] == 3 and base.dtype == torch.float32
        self.base = base.contiguous()
        self.num_points, self.partial, self.reserve, self.factor, self.aligned = num_points, partial, reserve, factor, aligned

    def draw(self, items, num_points=None, width=None):
        """Host draws, in the reference's RandomState call order, item r at num_points[r] points (default: every item at
        self.num_points).  -> idx_src, idx_tgt [P,width] int32 (width defaults to the largest count; columns past an
        item's count are 0), pose [P,12] f64, euler [P,3]."""
        Ns = [self.num_points] * len(items) if num_points is None else [int(n) for n in num_points]
        Nb = self.base.shape[1]
        width = max(Ns, default=0) if width is None else width
        idx_s = np.zeros((len(items), width), dtype=np.int32)
        idx_t = np.zeros((len(items), width), dtype=np.int32)
        pose = np.empty((len(items), 12), dtype=np.float64)
        euler = np.empty((len(items), 3), dtype=np.float64)
        for r, (item, N) in enumerate(zip(items, Ns)):
            rs = np.random.RandomState(item)
            ax = rs.uniform() * math.pi / self.factor
            ay = rs.uniform() * math.pi / self.factor
            az = rs.uniform() * math.pi / self.factor
            R = euler_to_R(ax, ay, az)
            t = np.array([rs.uniform(-0.5, 0.5), rs.uniform(-0.5, 0.5), rs.uniform(-0.5, 0.5)])
            first = rs.permutation(Nb)[:N]                       # np.random.permutation(pointcloud)[:num_points] (:288)
            if self.aligned:                                     # --model=lpd: one shared permutation (:304-309)
                perm = rs.permutation(N)
                idx_s[r, :N] = first[perm]
                idx_t[r, :N] = first[perm]
            else:
                idx_s[r, :N] = first[rs.permutation(N)]          # :298
                idx_t[r, :N] = first[rs.permutation(N)]          # :301
            pose[r, :9] = R.reshape(-1)
            pose[r, 9:] = t
            euler[r] = (az, ay, ax)                              # euler_ab, zyx order (:293)
        return idx_s, idx_t, pose, euler

    def _base(self, items):
        sel = torch.as_tensor(items, device=self.base.device)
        return self.base.index_select(0, sel) if items != list(range(self.base.shape[0])) else self.base

    def batch(self, items):
        items = list(items)
        dev = self.base.device
        idx_s, idx_t, pose, euler = self.draw(items)
        P, N, Nb = len(items), self.num_points, self.base.shape[1]
        base = self._base(items)
        d_is, d_it = torch.from_numpy(idx_s).to(dev), torch.from_numpy(idx_t).to(dev)
        d_pose = torch.from_numpy(pose).to(dev)
        L = lib()
        st = torch.cuda.current_stream(dev).cuda_stream
        if self.partial and not self.aligned:
            keep = int(N * self.reserve)                         # int(max(shape) * reserve) (:322-323)
            s64 = torch.empty((P, 3, N), dtype=torch.float64, device=dev)
            t64 = torch.empty((P, 3, N), dtype=torch.float64, device=dev)
            L.check(L.vcr_make_pairs(base.data_ptr(), P, Nb, d_is.data_ptr(), d_it.data_ptr(), d_pose.data_ptr(), N,
                                     s64.data_ptr(), t64.data_ptr(), None, None, st), "vcr_make_pairs")
            src = ops.crop_nearest(s64, keep)
            tgt = ops.crop_nearest(t64, keep)
        else:
            src = torch.empty((P, 3, N), dtype=torch.float32, device=dev)
            tgt = torch.empty((P, 3, N), dtype=torch.float32, device=dev)
            L.check(L.vcr_make_pairs(base.data_ptr(), P, Nb, d_is.data_ptr(), d_it.data_ptr(), d_pose.data_ptr(), N,
                                     None, None, src.data_ptr(), tgt.data_ptr(), st), "vcr_make_pairs")
        return {"src": src, "tgt": tgt} | _poses(pose, euler, dev)

    def batch_ragged(self, items, num_points, n_max=None):
        """A ragged batch: item i built exactly as PairGenerator(base, num_points[i], partial, reserve).batch([item i])
        builds it, in one set of launches.  -> batch()'s dict with src / tgt [P,3,L] zero-padded and ``lengths`` int32 [P]
        on the device, the points of pair i's source and target: num_points[i] for whole pairs, int(num_points[i] *
        reserve) for partial ones.  L is n_max (default max(num_points)), or int(n_max * reserve) for partial pairs;
        keeping n_max fixed keeps the shapes of successive batches, so a graph captured on one serves the next."""
        if self.aligned:
            raise NotImplementedError("PairGenerator.batch_ragged: aligned (LPD pre-training) pairs have no ragged "
                                      "consumer; use batch() per size")
        items, Ns = list(items), [int(n) for n in num_points]
        if len(Ns) != len(items):
            raise ValueError(f"PairGenerator.batch_ragged: {len(Ns)} point counts for {len(items)} items")
        if not items:
            raise ValueError("PairGenerator.batch_ragged: no items")
        Nb = self.base.shape[1]
        n_max = max(Ns) if n_max is None else int(n_max)
        bad = [n for n in Ns if n > min(Nb, n_max)]
        if bad:
            raise ValueError(f"PairGenerator.batch_ragged: point counts above the base cloud size {Nb} or n_max {n_max}: "
                             f"{bad}")
        crop = self.partial
        keeps = [int(n * self.reserve) for n in Ns] if crop else Ns  # int(max(shape) * reserve) (:322-323)
        L = int(n_max * self.reserve) if crop else n_max              # int(N * reserve) is non-decreasing in N
        ragged.check_lengths(keeps, L)
        dev = self.base.device
        idx_s, idx_t, pose, euler = self.draw(items, Ns, n_max)
        d_is, d_it = torch.from_numpy(idx_s).to(dev), torch.from_numpy(idx_t).to(dev)
        d_pose = torch.from_numpy(pose).to(dev)
        n = torch.tensor(Ns, dtype=torch.int32, device=dev)
        lengths = torch.tensor(keeps, dtype=torch.int32, device=dev)
        src, tgt = ops.make_pairs_ragged(self._base(items), d_is, d_it, d_pose, n, fp64=crop)
        if crop:
            src = ops.crop_nearest_ragged(src, n, lengths, L)
            tgt = ops.crop_nearest_ragged(tgt, n, lengths, L)
        return {"src": src, "tgt": tgt, "lengths": lengths} | _poses(pose, euler, dev)


def _poses(pose, euler, dev):
    """Host draws -> the pose entries of a batch (util/data.py:282-293) as fp32 device tensors."""
    P = pose.shape[0]
    R = pose[:, :9].reshape(P, 3, 3)
    t = pose[:, 9:]
    R_ba = R.transpose(0, 2, 1)
    t_ba = -np.einsum("pij,pj->pi", R_ba, t)                     # translation_ba = -R_ba.dot(translation_ab) (:286)
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    return {"R_ab": f32(R), "t_ab": f32(t), "R_ba": f32(R_ba), "t_ba": f32(t_ba), "euler_ab": f32(euler),
            "euler_ba": f32(-euler[:, ::-1])}


class EvalAccumulator:
    """Device-resident accumulation of test_one_epoch's running metrics (model/vcrnet_model.py:583-630, 645-650): one
    kernel per batch, no host synchronisation until ``result()``."""

    KEYS = ("loss", "cycle_loss", "mse_ab", "mae_ab", "mse_ba", "mae_ba")

    def __init__(self, device):
        self.acc = torch.zeros(8, dtype=torch.float64, device=device)

    def update(self, src, tgt, srcK, corrK, R_gt, t_gt, R_ab, t_ab, R_ba, t_ba):
        B, _, N = src.shape
        M = srcK.shape[2]
        assert tgt.shape == src.shape, "transformed_target - src needs equally sized clouds (:626)"
        ts = [x.contiguous() for x in (src, tgt, srcK, corrK, R_gt, t_gt, R_ab, t_ab, R_ba, t_ba)]
        L = lib()
        L.check(L.vcr_eval_metrics(ts[0].data_ptr(), ts[1].data_ptr(), N, ts[2].data_ptr(), ts[3].data_ptr(), M,
                                   ts[4].data_ptr(), ts[5].data_ptr(), ts[6].data_ptr(), ts[7].data_ptr(),
                                   ts[8].data_ptr(), ts[9].data_ptr(), B, self.acc.data_ptr(),
                                   torch.cuda.current_stream(src.device).cuda_stream), "vcr_eval_metrics")

    def update_ragged(self, src, tgt, lengths, srcK, corrK, corr_lengths, R_gt, t_gt, R_ab, t_ab, R_ba, t_ba):
        """update() for a ragged batch: src / tgt [B,3,N_max] with lengths[b] points in pair b, srcK / corrK [B,3,M_max]
        with corr_lengths[b] columns (int32 [B] on the device; lengths for whole pairs, ragged.corr_lengths(lengths,
        overlap2) for partial ones).  Pair b adds what update() adds for it alone; padded columns are never read."""
        B, _, N = src.shape
        M = srcK.shape[2]
        shapes = {"tgt": (tgt, (B, 3, N)), "srcK": (srcK, (B, 3, M)), "corrK": (corrK, (B, 3, M)),
                  "R_gt": (R_gt, (B, 3, 3)), "t_gt": (t_gt, (B, 3)), "R_ab": (R_ab, (B, 3, 3)), "t_ab": (t_ab, (B, 3)),
                  "R_ba": (R_ba, (B, 3, 3)), "t_ba": (t_ba, (B, 3))}
        for name, (x, want) in shapes.items():
            if tuple(x.shape) != want:
                raise ValueError(f"EvalAccumulator.update_ragged: `{name}` must be {want}, got {tuple(x.shape)}")
        ops.eval_metrics_ragged(self.acc, src, tgt, lengths, srcK, corrK, corr_lengths, R_gt, t_gt, R_ab, t_ab, R_ba,
                                t_ba)

    def result(self):
        a = self.acc.cpu().numpy()
        n = max(a[6], 1.0)
        return {k: float(a[i] / n) for i, k in enumerate(self.KEYS)} | {"num_examples": int(a[6])}
