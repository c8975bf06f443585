"""Farthest-point sampling above 14 336 points per cloud (csrc/fps.cu fps_cluster_kernel: one thread-block cluster of
2, 4, 8 or 16 CTAs per cloud).  Every index comparison is exact equality with the canonical C oracle."""
import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import ops
from oracle import canon, synth
from oracle import vcr_oracle as O
from oracle.ref_harness import default_args

DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def nump(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("npoint", [32, 256])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("N", [14337, 16384, 20000, 50000, 100000, 229376])   # C = 2, 2, 2, 4, 8, 16
def test_fps_cluster_sizes(N, B, npoint):
    p = np.random.RandomState(N + B).randn(B, 3, N).astype(np.float32)
    want = canon.fps(p, npoint)
    x = cu(p)
    got64 = nump(V.farthest_point_sample(x, npoint))
    assert got64.dtype == np.int64 and np.array_equal(got64, want)
    got32 = nump(ops.fps(x, npoint, want64=False))
    assert got32.dtype == np.int32 and np.array_equal(got32, want)


def test_fps_boundary_between_kernels():
    """14 336 points run on the one-CTA kernel, 14 337 on a cluster of two: prefixes of one cloud, both canonical."""
    p = np.random.RandomState(14336).randn(2, 3, 14337).astype(np.float32)
    for n in (14336, 14337):
        q = np.ascontiguousarray(p[:, :, :n])
        assert np.array_equal(nump(V.farthest_point_sample(cu(q), 64)), canon.fps(q, 64)), n


def test_fps_ties_across_ctas():
    """A dyadic grid cloud tiled ten times (60 000 points, 8 CTAs of 7 500): every maximum has equal copies in other CTAs,
    and the lower global index must win."""
    base = synth.grid_cloud(np.random.RandomState(9), (2, 3, 6000), 4, -1.0, 1.0)
    p = np.ascontiguousarray(np.tile(base, (1, 1, 10)))
    want = canon.fps(p, 256)
    assert np.array_equal(nump(V.farthest_point_sample(cu(p), 256)), want)


def test_fps_cluster_waves_on_side_stream():
    """40 clusters of 8 CTAs (one CTA per SM) do not fit at once; launched on a non-default stream."""
    p = np.random.RandomState(40).randn(40, 3, 100000).astype(np.float32)
    want = canon.fps(p, 32)
    x = cu(p)
    s = torch.cuda.Stream(device=DEV)
    s.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(s):
        out = V.farthest_point_sample(x, 32)
    s.synchronize()
    got = nump(out)
    for b in range(40):
        assert np.array_equal(got[b], want[b]), b


def test_fps_limit_is_named():
    x = torch.zeros(1, 3, 229377, device=DEV)
    with pytest.raises(RuntimeError, match="229376"):
        V.farthest_point_sample(x, 32)


def test_lpd_pretraining_at_16384_points(monkeypatch):
    """LPD pre-training loss (model/lpdnet_model.py getLoss: FPS of 32 anchors over the whole cloud) forward and backward
    at 16 384 points."""
    from vcr_net_b200.util import util as U
    lpd_w = load_golden("lpd_pretrained_weights")
    net = V.LPD(default_args(model="lpd", num_points=16384)).to(DEV).train()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in lpd_w.items()}, strict=True)
    pa = synth.make_pairs(2, 16384, aligned=True, first_item=21)
    anchors = []
    fps = U.farthest_point_sample

    def recording_fps(xyz, npoint):
        idx = fps(xyz, npoint)
        anchors.append(idx)
        return idx

    monkeypatch.setattr(U, "farthest_point_sample", recording_fps)
    se, te, loss, _, _ = net(cu(pa["src"]), cu(pa["tgt"]))
    loss.backward()
    torch.cuda.synchronize()
    assert len(anchors) == 1 and np.array_equal(nump(anchors[0]), canon.fps(pa["src"], 32))
    want = float(O.lpd_loss(pa["src"], nump(se), nump(te)))
    assert abs(float(loss.detach()) - want) <= 1e-4 * abs(want), (float(loss.detach()), want)
    for name, prm in net.emb_nn.named_parameters():
        assert prm.grad is not None and bool(torch.isfinite(prm.grad).all()), name
