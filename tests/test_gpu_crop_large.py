"""The data step's nearest-to-anchor crop at any cloud size (csrc/datastep.cu, vcr_crop_nearest_sort).

* The segmented radix sort against oracle/synth.crop_nearest_to_last (a stable numpy argsort of the same fp64 distances),
  exact equality of the fp32 output, from 25 601 to 305 558 points.
* Bit-identity with the one-CTA rank-count kernel (vcr_crop_nearest) wherever both run.
* Ties, duplicates, copies of the anchor, NaN, graph capture and streams, the limits.
* PairGenerator / PairSource(partial=True) above 25 600 points, and the data flow of test_one_epoch on them.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops
    from vcr_net_b200._lib import lib
    from vcr_net_b200.data import EvalAccumulator, PairGenerator
    from vcr_net_b200.synthetic import PairSource
from oracle import synth
from oracle import vcr_oracle as O
from oracle.ref_harness import default_args

DEV = "cuda:0"
RES = synth.RESERVE_0575


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def nump(t):
    return t.detach().cpu().numpy()


def oracle_crop(pc, keep):
    """pc fp64 [P,3,N] -> fp32 [P,3,keep] by oracle/synth.crop_nearest_to_last (its full order, first `keep` columns)."""
    return np.stack([synth.crop_nearest_to_last(c, 1.0)[:, :keep] for c in pc]).astype(np.float32)


def cloud(P, N, seed):
    return np.random.RandomState(seed).rand(P, 3, N) - 0.5


def assert_same(got, want):
    g = nump(got)
    assert g.shape == want.shape and g.dtype == np.float32
    assert np.array_equal(g, want, equal_nan=True), int((g != want).sum())


# ---------------------------------------------------------------- sizes ----------------------------------------------
@pytest.mark.parametrize("P", [1, 3])
@pytest.mark.parametrize("N", [25601, 27282, 87303, 305558])          # keep at the reserve: 19 218, 20 480, 65 536, 229 376
def test_crop_sort_sizes(N, P):
    pc = cloud(P, N, N + P)
    x = cu(pc)
    full = oracle_crop(pc, N)
    for keep in (int(N * RES), 1, N):
        assert_same(ops.crop_nearest(x, keep), full[:, :, :keep])
    for p in range(P):                                                 # the oracle of the data step itself
        assert np.array_equal(full[p, :, :int(N * RES)], synth.crop_nearest_to_last(pc[p], RES).astype(np.float32))


def test_crop_sort_more_clouds_than_sms():
    P, N = 160, 27282
    pc = cloud(P, N, 160)
    assert_same(ops.crop_nearest(cu(pc), int(N * RES)), oracle_crop(pc, int(N * RES)))


# ---------------------------------------------------------------- agreement with the one-CTA kernel -------------------
@pytest.mark.parametrize("N", [1, 2, 333, 1024, 25600])
def test_crop_sort_equals_one_cta_kernel(N):
    pc = cloud(3, N, 7 + N)
    x = cu(pc)
    full = oracle_crop(pc, N)
    for keep in sorted({1, max(1, int(N * RES)), N}):
        one = ops.crop_nearest(x, keep)                                # N <= 25 600: the rank-count kernel
        srt = ops.crop_nearest_sort(x, keep)
        assert torch.equal(one, srt)
        assert_same(srt, full[:, :, :keep])


# ---------------------------------------------------------------- ties --------------------------------------------------
def tie_clouds(N, seed):
    """Four clouds with few distinct distances: a dyadic grid, the grid with duplicated points and several exact copies of
    the anchor (d2 = 0), a cloud whose points are all equal, and a two-valued cloud."""
    rs = np.random.RandomState(seed)
    grid = synth.grid_cloud(rs, (3, N), 2, -1.0, 1.0).astype(np.float64)       # 8 values per axis
    dup = grid.copy()
    src = rs.randint(0, N, size=N // 3)
    dup[:, rs.randint(0, N, size=N // 3)] = dup[:, src]
    dup[:, rs.randint(0, N - 1, size=17)] = dup[:, N - 1:N]                      # copies of the anchor
    const = np.full((3, N), 0.125)
    two = np.where(rs.rand(3, N) < 0.5, 0.25, -0.25)
    return np.stack([grid, dup, const, two])


@pytest.mark.parametrize("N", [5000, 30011])
def test_crop_sort_ties_go_to_the_lower_index(N):
    pc = tie_clouds(N, N)
    x = cu(pc)
    full = oracle_crop(pc, N)
    for keep in (1, int(N * RES), N):
        srt = ops.crop_nearest_sort(x, keep)
        assert_same(srt, full[:, :, :keep])
        if N <= ops.CROP_ONE_CTA_MAX_POINTS:
            assert torch.equal(srt, ops.crop_nearest(x, keep))


def sort_into(x, keep, fill):
    """vcr_crop_nearest_sort straight into an output prefilled with `fill` (to see that every column is written)."""
    P, _, N = x.shape
    L = lib()
    out = torch.full((P, 3, keep), fill, dtype=torch.float32, device=DEV)
    wsb = L.vcr_crop_nearest_workspace_bytes(P, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.check(L.vcr_crop_nearest_sort(x.data_ptr(), P, N, keep, out.data_ptr(), ws.data_ptr(), wsb,
                                    torch.cuda.current_stream(DEV).cuda_stream), "vcr_crop_nearest_sort")
    return out


@pytest.mark.parametrize("N", [777, 26000])
def test_crop_sort_nan_goes_last_and_every_column_is_written(N):
    """NaN coordinates give NaN distances: they sort after +inf in index order; a NaN anchor makes every distance NaN."""
    pc = cloud(3, N, 11)
    rs = np.random.RandomState(12)
    pc[0, rs.randint(0, 3, size=N // 10), rs.randint(0, N - 1, size=N // 10)] = np.nan
    pc[1, 0, rs.randint(0, N - 1, size=5)] = np.inf
    pc[2, 1, N - 1] = np.nan
    full = oracle_crop(pc, N)
    for keep in (1, int(N * RES), N):
        assert_same(sort_into(cu(pc), keep, 1234.5), full[:, :, :keep])


# ---------------------------------------------------------------- capture and streams ---------------------------------
def test_crop_sort_graph_capture_and_streams():
    N, keep = 87303, int(87303 * RES)
    pc = cloud(2, N, 3)
    x = cu(pc)
    eager = ops.crop_nearest(x, keep)
    again = ops.crop_nearest(x, keep)
    assert torch.equal(eager, again)
    assert_same(eager, oracle_crop(pc, keep))

    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        on_side = ops.crop_nearest(x, keep)
    side.synchronize()
    assert torch.equal(on_side, eager)

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = ops.crop_nearest(x, keep)
    x.copy_(cu(cloud(2, N, 4)))                         # replay reads the inputs as they are at replay time
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, ops.crop_nearest(x, keep))
    x.copy_(cu(pc))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)


# ---------------------------------------------------------------- limits ----------------------------------------------
def test_crop_limits():
    big = torch.zeros(1, 3, 1, dtype=torch.float64, device=DEV).expand(83887, 3, 25601)    # P * N = 2^31 + 107 439
    with pytest.raises(RuntimeError, match=str(2**31 - 1)):
        ops.crop_nearest(big, 10)

    L = lib()
    st = torch.cuda.current_stream(DEV).cuda_stream
    P, N = 2, 30000
    x = cu(cloud(P, N, 5))
    out = torch.empty((P, 3, N), dtype=torch.float32, device=DEV)
    wsb = L.vcr_crop_nearest_workspace_bytes(P, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    torch.cuda.synchronize()
    launches = L.vcr_launch_count()
    assert L.vcr_crop_nearest_sort(x.data_ptr(), 65536, 32768, 1, out.data_ptr(), ws.data_ptr(), wsb, st) == -2
    assert L.vcr_crop_nearest_workspace_bytes(65536, 32768) == 0
    assert L.vcr_crop_nearest_sort(x.data_ptr(), P, N, 0, out.data_ptr(), ws.data_ptr(), wsb, st) == -2
    assert L.vcr_crop_nearest_sort(x.data_ptr(), P, N, N + 1, out.data_ptr(), ws.data_ptr(), wsb, st) == -2
    assert L.vcr_crop_nearest_sort(x.data_ptr(), P, N, N, out.data_ptr(), ws.data_ptr(), wsb - 1, st) == -4
    assert L.vcr_launch_count() == launches
    assert L.vcr_crop_nearest_sort(x.data_ptr(), P, N, N, out.data_ptr(), ws.data_ptr(), wsb, st) == 0
    assert L.vcr_launch_count() > launches
    assert_same(out, oracle_crop(nump(x), N))


# ---------------------------------------------------------------- data step ---------------------------------------------
@pytest.mark.parametrize("N", [25600, 25601, 27282, 87303])
def test_partial_pair_generator_above_one_cta_cap(N):
    """PairGenerator(partial=True) against synth.make_pairs within the bars of test_device_data_step_matches_host_generator:
    the device's fp64 transform differs from numpy's by at most one ulp, which can move a point by one fp32 ulp."""
    n_items, first = 2, 3
    Nb = max(2048, N)
    base = np.random.RandomState(1234).rand(first + n_items, Nb, 3).astype(np.float32) - 0.5   # synth.make_pairs' base
    gen = PairGenerator(cu(base), num_points=N, partial=True, reserve=RES)
    got = gen.batch(range(first, first + n_items))
    want = synth.make_pairs(n_items, N, partial=True, reserve=RES, first_item=first)
    assert tuple(got["src"].shape) == want["src"].shape == (n_items, 3, int(N * RES))
    for k in ("src", "tgt"):
        d = np.abs(nump(got[k]) - want[k])
        assert d.max() <= 6e-8, (k, d.max())
        assert (d > 0).mean() < 1e-3


@pytest.fixture
def h3():
    old = config.precision
    config.set_precision("h3")
    yield
    config.set_precision(old)


def test_partial_pair_source_to_eval_accumulator(ckpt, h3):
    """test_one_epoch's data flow at 27 282 points (20 480 after the crop): device pairs -> vcrnetIter -> EvalAccumulator."""
    B, N = 2, 27282
    net = V.VCRNet(default_args(partial=True, overlap2=synth.OVERLAP2_0575)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=True)
    data = PairSource(B, DEV, num_points=N, partial=True, reserve=RES).batch(0, B)
    src, tgt = data["src"], data["tgt"]
    assert tuple(src.shape) == tuple(tgt.shape) == (B, 3, 20480)
    for it in (1, 3):
        out = V.vcrnetIter(net, src, tgt, iter=it)
        acc = EvalAccumulator(DEV)
        acc.update(src, tgt, out[0], out[1], data["R_ab"], data["t_ab"], out[2], out[3], out[4], out[5])
        res = acc.result()
        assert all(np.isfinite(nump(o)).all() for o in out)
        want = O.eval_metrics_batch(nump(src), nump(tgt), nump(out[0]), nump(out[1]), nump(data["R_ab"]),
                                    nump(data["t_ab"]), nump(out[2]), nump(out[3]), nump(out[4]), nump(out[5]))
        assert res["num_examples"] == B
        for i, k in enumerate(acc.KEYS):
            w = want[i] / B
            assert np.isfinite(res[k]) and abs(res[k] - w) <= 1e-5 * max(abs(w), 1e-6), (it, k, res[k], w)
        print(f"[pair source 27282 iter {it}] " + " ".join(f"{k} {res[k]:.4g}" for k in acc.KEYS))
