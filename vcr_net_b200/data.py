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

from . import ops
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
    same values ``ModelNet40.__getitem__`` returns for test-partition items (np.random.seed(item), :255-256)."""

    def __init__(self, base: torch.Tensor, num_points=1024, partial=False, reserve=1.0, factor=4.0, aligned=False):
        if not base.is_cuda:
            raise RuntimeError("PairGenerator: base clouds must live on a CUDA device (there is no CPU path)")
        assert base.dim() == 3 and base.shape[2] == 3 and base.dtype == torch.float32
        self.base = base.contiguous()
        self.num_points, self.partial, self.reserve, self.factor, self.aligned = num_points, partial, reserve, factor, aligned

    def draw(self, items):
        """Host draws, in the reference's RandomState call order.  -> idx_src, idx_tgt [P,N] int32, pose [P,12] f64, euler [P,3]."""
        N, Nb = self.num_points, self.base.shape[1]
        idx_s = np.empty((len(items), N), dtype=np.int32)
        idx_t = np.empty((len(items), N), dtype=np.int32)
        pose = np.empty((len(items), 12), dtype=np.float64)
        euler = np.empty((len(items), 3), dtype=np.float64)
        for r, item in enumerate(items):
            rs = np.random.RandomState(item)
            ax = rs.uniform() * math.pi / self.factor
            ay = rs.uniform() * math.pi / self.factor
            az = rs.uniform() * math.pi / self.factor
            R = euler_to_R(ax, ay, az)
            t = np.array([rs.uniform(-0.5, 0.5), rs.uniform(-0.5, 0.5), rs.uniform(-0.5, 0.5)])
            first = rs.permutation(Nb)[:N]                       # np.random.permutation(pointcloud)[:num_points] (:288)
            if self.aligned:                                     # --model=lpd: one shared permutation (:304-309)
                perm = rs.permutation(N)
                idx_s[r] = first[perm]
                idx_t[r] = first[perm]
            else:
                idx_s[r] = first[rs.permutation(N)]              # :298
                idx_t[r] = first[rs.permutation(N)]              # :301
            pose[r, :9] = R.reshape(-1)
            pose[r, 9:] = t
            euler[r] = (az, ay, ax)                              # euler_ab, zyx order (:293)
        return idx_s, idx_t, pose, euler

    def batch(self, items):
        items = list(items)
        dev = self.base.device
        idx_s, idx_t, pose, euler = self.draw(items)
        P, N, Nb = len(items), self.num_points, self.base.shape[1]
        sel = torch.as_tensor(items, device=dev)
        base = self.base.index_select(0, sel) if items != list(range(self.base.shape[0])) else self.base
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
        R = pose[:, :9].reshape(P, 3, 3)
        t = pose[:, 9:]
        R_ba = R.transpose(0, 2, 1)
        t_ba = -np.einsum("pij,pj->pi", R_ba, t)                 # translation_ba = -R_ba.dot(translation_ab) (:286)
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        return {"src": src, "tgt": tgt, "R_ab": f32(R), "t_ab": f32(t), "R_ba": f32(R_ba), "t_ba": f32(t_ba),
                "euler_ab": f32(euler), "euler_ba": f32(-euler[:, ::-1])}


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

    def result(self):
        a = self.acc.cpu().numpy()
        n = max(a[6], 1.0)
        return {k: float(a[i] / n) for i, k in enumerate(self.KEYS)} | {"num_examples": int(a[6])}
