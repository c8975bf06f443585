"""Ragged batches from the device data step: PairGenerator / PairSource.batch_ragged and EvalAccumulator.update_ragged.

Each item of a ragged batch must get the bits it gets from batch([item]) at its own size, whichever crop route the
batch takes, and each pair must add to the accumulator what update() adds for it alone.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops, ragged
    from vcr_net_b200._lib import lib
    from vcr_net_b200.data import EvalAccumulator, PairGenerator
    from vcr_net_b200.synthetic import PairSource
from oracle import synth
from oracle import vcr_oracle as O
from oracle.ref_harness import default_args

DEV = "cuda:0"
RES = synth.RESERVE_0575
WHOLE_N = [21, 300, 767, 1024, 2049, 8200]
PARTIAL_N = [28, 512, 1024, 4097]                      # keep int(N * RES): 21, 384, 768, 3 075
NB = 9000


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def nump(t):
    return t.detach().cpu().numpy()


def lens(x):
    return torch.tensor([int(v) for v in x], dtype=torch.int32, device=DEV)


@pytest.fixture(scope="module")
def base():
    """synth.make_pairs' base clouds at NB points: row i is item i's cloud for any first_item."""
    return cu(np.random.RandomState(1234).rand(12, NB, 3).astype(np.float32) - 0.5)


@pytest.fixture
def h3():
    old = config.precision
    config.set_precision("h3")
    yield
    config.set_precision(old)


def check_items(got, gen, items, Ns):
    """got = batch_ragged(items, Ns): item b against batch([item b]) at Ns[b], bit for bit, zeros past its length."""
    L = got["src"].shape[2]
    assert got["lengths"].dtype == torch.int32 and got["lengths"].device.type == "cuda"
    for b, (item, n) in enumerate(zip(items, Ns)):
        want = PairGenerator(gen.base, num_points=n, partial=gen.partial, reserve=gen.reserve).batch([item])
        k = want["src"].shape[2]
        assert int(got["lengths"][b]) == k
        for key in ("src", "tgt"):
            assert torch.equal(got[key][b, :, :k], want[key][0]), (b, n, key)
            assert not got[key][b, :, k:].any(), (b, n, key)
            assert got[key].shape == (len(items), 3, L)
        for key in ("R_ab", "t_ab", "R_ba", "t_ba", "euler_ab", "euler_ba"):
            assert torch.equal(got[key][b], want[key][0]), (b, key)


# ---------------------------------------------------------------- 1, 2: per-item identity and the oracle ---------------
@pytest.mark.parametrize("partial", [False, True])
@pytest.mark.parametrize("extra", [0, 777])
def test_batch_ragged_equals_each_item_alone(base, partial, extra):
    Ns = PARTIAL_N if partial else WHOLE_N
    items = [7, 2, 9, 0, 5, 11][:len(Ns)]
    gen = PairGenerator(base, num_points=1024, partial=partial, reserve=RES if partial else 1.0)
    n_max = max(Ns) + extra if extra else None
    got = gen.batch_ragged(items, Ns, n_max=n_max)
    L = max(Ns) + extra
    assert got["src"].shape[2] == (int(L * RES) if partial else L)
    check_items(got, gen, items, Ns)


@pytest.mark.parametrize("partial", [False, True])
def test_batch_ragged_against_the_oracle(base, partial):
    """Within the bars of test_device_data_step_matches_host_generator: the device's fp64 transform differs from numpy's by
    at most one ulp, which can move a point by one fp32 ulp."""
    Ns = PARTIAL_N if partial else WHOLE_N
    items = [3, 8, 1, 10, 4, 6][:len(Ns)]
    got = PairGenerator(base, partial=partial, reserve=RES if partial else 1.0).batch_ragged(items, Ns)
    for b, (item, n) in enumerate(zip(items, Ns)):
        want = synth.make_pairs(1, n, partial=partial, reserve=RES, first_item=item, base_points=NB)
        k = want["src"].shape[2]
        assert int(got["lengths"][b]) == k
        for key in ("src", "tgt"):
            d = np.abs(nump(got[key][b, :, :k]) - want[key][0])
            assert d.max() <= 6e-8, (b, key, d.max())
            assert (d > 0).mean() < 1e-3
        for key in ("R_ab", "t_ab", "euler_ab"):
            assert np.allclose(nump(got[key][b]), want[key][0], atol=1e-7), (b, key)


# ---------------------------------------------------------------- 3: crop routes --------------------------------------
CROP_N = [28, 1024, 3001, 25600, 26000, 27282]


def oracle_crop(pc, n, keep, width):
    out = np.zeros((len(n), 3, width), dtype=np.float32)
    for p, (nb, kb) in enumerate(zip(n, keep)):
        out[p, :, :kb] = synth.crop_nearest_to_last(pc[p, :, :nb], 1.0)[:, :kb].astype(np.float32)
    return out


def padded(clouds, width, fill=0.0):
    pc = np.full((len(clouds), 3, width), fill)
    for p, c in enumerate(clouds):
        pc[p, :, :c.shape[1]] = c
    return pc


def assert_same(got, want):
    g = nump(got)
    assert g.shape == want.shape and g.dtype == np.float32
    assert np.array_equal(g, want, equal_nan=True), int((g != want).sum())


def test_crop_ragged_routes():
    """N_max above 25 600 sends every cloud, small ones included, through the sort; below, the one-CTA kernel.  Both equal
    the per-cloud crop and the oracle exactly; padding (here NaN) is never read."""
    rs = np.random.RandomState(5)
    clouds = [rs.rand(3, n) - 0.5 for n in CROP_N]
    keep = [int(n * RES) for n in CROP_N]
    km = int(max(CROP_N) * RES)
    x = cu(padded(clouds, max(CROP_N), np.nan))
    got = ops.crop_nearest_ragged(x, lens(CROP_N), lens(keep), km)
    assert_same(got, oracle_crop(padded(clouds, max(CROP_N)), CROP_N, keep, km))
    for p, n in enumerate(CROP_N):
        alone = ops.crop_nearest(cu(clouds[p][None]), keep[p])
        assert torch.equal(got[p:p + 1, :, :keep[p]], alone), n
    small = [p for p, n in enumerate(CROP_N) if n <= ops.CROP_ONE_CTA_MAX_POINTS]
    xs = cu(padded([clouds[p] for p in small], ops.CROP_ONE_CTA_MAX_POINTS, np.nan))
    one_cta = ops.crop_nearest_ragged(xs, lens([CROP_N[p] for p in small]), lens([keep[p] for p in small]), km)
    assert torch.equal(one_cta, got[small])


def tie_clouds(N, rs):
    grid = synth.grid_cloud(rs, (3, N), 2, -1.0, 1.0).astype(np.float64)        # 8 values per axis
    dup = grid.copy()
    dup[:, rs.randint(0, N, size=N // 3)] = dup[:, rs.randint(0, N, size=N // 3)]
    dup[:, rs.randint(0, N - 1, size=17)] = dup[:, N - 1:N]                       # copies of the anchor
    return [grid, dup]


def crop_into(x, n, keep, keep_max, fill):
    """Both ragged C entry points (by N_max) straight into an output prefilled with `fill`."""
    P, _, N = x.shape
    L = lib()
    st = torch.cuda.current_stream(DEV).cuda_stream
    out = torch.full((P, 3, keep_max), fill, dtype=torch.float32, device=DEV)
    if N <= ops.CROP_ONE_CTA_MAX_POINTS:
        L.check(L.vcr_crop_nearest_ragged(x.data_ptr(), n.data_ptr(), keep.data_ptr(), P, N, keep_max, out.data_ptr(),
                                          st), "vcr_crop_nearest_ragged")
    else:
        wsb = L.vcr_crop_nearest_workspace_bytes(P, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        L.check(L.vcr_crop_nearest_sort_ragged(x.data_ptr(), n.data_ptr(), keep.data_ptr(), P, N, keep_max,
                                               out.data_ptr(), ws.data_ptr(), wsb, st), "vcr_crop_nearest_sort_ragged")
    return out


@pytest.mark.parametrize("N_max", [25600, 26001])
def test_crop_ragged_ties_and_every_column_written(N_max):
    rs = np.random.RandomState(N_max)
    n = [5000, 333, 21000, 4096]
    clouds = [tie_clouds(v, rs)[p % 2] for p, v in enumerate(n)]
    x = cu(padded(clouds, N_max, 7.0))
    for keep in ([1] * 4, [int(v * RES) for v in n], n):
        km = max(keep) + 3
        got = crop_into(x, lens(n), lens(keep), km, np.nan)
        assert_same(got, oracle_crop(padded(clouds, N_max), n, keep, km))


def test_crop_ragged_nan_goes_last():
    """NaN distances sort after +inf in index order and before the padding; a NaN anchor makes every distance NaN."""
    rs = np.random.RandomState(12)
    n = [777, 26000, 300]
    clouds = [rs.rand(3, v) - 0.5 for v in n]
    c0 = clouds[0]
    c0[rs.randint(0, 3, size=77), rs.randint(0, 776, size=77)] = np.nan
    clouds[1][0, rs.randint(0, 25999, size=5)] = np.inf
    clouds[2][1, 299] = np.nan
    keep = [int(v * RES) for v in n]
    N_max = 26011
    for full in (False, True):
        k = n if full else keep
        got = crop_into(cu(padded(clouds, N_max, np.nan)), lens(n), lens(k), max(k), 1234.5)
        assert_same(got, oracle_crop(padded(clouds, N_max), n, k, max(k)))


# ---------------------------------------------------------------- 4: graph capture and streams ----------------------
def test_three_ops_graph_capture_and_side_stream(base):
    gen = PairGenerator(base, partial=True, reserve=RES)
    n_max = 1100
    L = int(n_max * RES)

    def host(items, Ns):
        idx_s, idx_t, pose, _ = gen.draw(items, Ns, n_max)
        d = gen.batch_ragged(items, Ns, n_max)
        keep = [int(v * RES) for v in Ns]
        return [base[items], cu(idx_s), cu(idx_t), cu(pose), lens(Ns), lens(keep),
                d["R_ab"], d["t_ab"], d["R_ba"], d["t_ba"]]

    def run(acc, b, i_s, i_t, pose, n, keep, R, t, Rb, tb):
        s64, t64 = ops.make_pairs_ragged(b, i_s, i_t, pose, n, fp64=True)
        s, tg = ops.crop_nearest_ragged(s64, n, keep, L), ops.crop_nearest_ragged(t64, n, keep, L)
        ops.eval_metrics_ragged(acc, s, tg, keep, s, tg, keep, R, t, Rb, tb, Rb, tb)
        return s, tg

    first = host([0, 1, 2, 3], [600, 1100, 28, 900])
    second = host([4, 5, 6, 7], [1024, 100, 700, 333])
    acc_e = [torch.zeros(8, dtype=torch.float64, device=DEV) for _ in range(2)]
    eager = [run(acc_e[i], *a) for i, a in enumerate((first, second))]
    d = gen.batch_ragged([4, 5, 6, 7], [1024, 100, 700, 333], n_max)
    assert torch.equal(eager[1][0], d["src"]) and torch.equal(eager[1][1], d["tgt"])

    static = [a.clone() for a in first]
    acc = torch.zeros(8, dtype=torch.float64, device=DEV)
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        on_side = run(acc, *static)
    side.synchronize()
    assert all(torch.equal(a, c) for a, c in zip(on_side, eager[0]))
    assert torch.allclose(acc, acc_e[0], rtol=1e-12, atol=0)          # fp64 atomics: the order of the sums may differ

    g = torch.cuda.CUDAGraph()
    acc.zero_()
    with torch.cuda.graph(g):
        captured = run(acc, *static)
    for k, a in enumerate((second, first)):
        for s_, v in zip(static, a):
            s_.copy_(v)
        acc.zero_()
        g.replay()
        torch.cuda.synchronize()
        want = eager[1 - k]
        assert all(torch.equal(x, y) for x, y in zip(captured, want)), k
        assert torch.allclose(acc, acc_e[1 - k], rtol=1e-12, atol=0), k


# ---------------------------------------------------------------- 5: metrics ------------------------------------------
def test_update_ragged_equals_update_per_pair():
    g = torch.Generator(device=DEV).manual_seed(4)
    n, m = [21, 300, 1024, 77, 500], [5, 300, 600, 1, 77]
    B, N, M = len(n), max(n) + 9, max(m) + 4
    src, tgt = torch.randn(B, 3, N, generator=g, device=DEV), torch.randn(B, 3, N, generator=g, device=DEV)
    srcK, corrK = torch.randn(B, 3, M, generator=g, device=DEV), torch.randn(B, 3, M, generator=g, device=DEV)
    for b in range(B):                                               # padding is never read
        for x, k in ((src, n[b]), (tgt, n[b]), (srcK, m[b]), (corrK, m[b])):
            x[b, :, k:] = float("nan")
    R = [torch.linalg.qr(torch.randn(B, 3, 3, generator=g, device=DEV, dtype=torch.float64))[0].float() for _ in range(3)]
    t = [torch.randn(B, 3, generator=g, device=DEV) for _ in range(3)]
    acc = EvalAccumulator(DEV)
    acc.update_ragged(src, tgt, lens(n), srcK, corrK, lens(m), R[0], t[0], R[1], t[1], R[2], t[2])
    per = EvalAccumulator(DEV)
    want = np.zeros(7)
    for b in range(B):
        args = (src[b:b + 1, :, :n[b]], tgt[b:b + 1, :, :n[b]], srcK[b:b + 1, :, :m[b]], corrK[b:b + 1, :, :m[b]],
                R[0][b:b + 1], t[0][b:b + 1], R[1][b:b + 1], t[1][b:b + 1], R[2][b:b + 1], t[2][b:b + 1])
        per.update(*args)
        want += np.array(O.eval_metrics_batch(*[nump(a) for a in args]), dtype=np.float64)
    res, res_p = acc.result(), per.result()
    assert res["num_examples"] == res_p["num_examples"] == B
    for i, k in enumerate(acc.KEYS):
        assert np.isfinite(res[k]) and abs(res[k] - res_p[k]) <= 1e-12 * abs(res_p[k]), (k, res[k], res_p[k])
        w = want[i] / B
        assert abs(res[k] - w) <= 1e-5 * max(abs(w), 1e-6), (k, res[k], w)


# ---------------------------------------------------------------- 6: end to end ---------------------------------------
E2E_N = [512, 1024, 300, 767, 900, 640]


@pytest.mark.parametrize("partial", [False, True])
def test_pair_source_ragged_end_to_end(ckpt, h3, partial):
    """PairSource.batch_ragged -> vcrnetIterRagged(Partial) -> update_ragged against batch([item]) -> vcrnetIter ->
    update, pair by pair."""
    Ns = [28] + E2E_N[1:] if partial else [21] + E2E_N[1:]
    ov = synth.OVERLAP2_0575
    net = V.VCRNet(default_args(partial=partial, overlap2=ov)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=False)
    ps = PairSource(len(Ns) + 2, DEV, num_points=1024, partial=partial, reserve=RES if partial else 1.0)
    first = 2
    d = ps.batch_ragged(first, len(Ns), Ns, n_max=1024)
    reg = V.vcrnetIterRaggedPartial if partial else V.vcrnetIterRagged
    for it in (1, 3):
        out = reg(net, d["src"], d["tgt"], d["lengths"], d["lengths"], iter=it)
        corr = ragged.corr_lengths(d["lengths"], ov) if partial else d["lengths"]
        acc = EvalAccumulator(DEV)
        acc.update_ragged(d["src"], d["tgt"], d["lengths"], out[0], out[1], corr, d["R_ab"], d["t_ab"], *out[2:])
        per = EvalAccumulator(DEV)
        kb = corr.tolist()
        for b, n in enumerate(Ns):
            q = PairGenerator(ps.gen.base, num_points=n, partial=partial, reserve=ps.gen.reserve).batch([first + b])
            want = V.vcrnetIter(net, q["src"], q["tgt"], iter=it)
            per.update(q["src"], q["tgt"], want[0], want[1], q["R_ab"], q["t_ab"], *want[2:])
            assert want[0].shape[2] == kb[b]
            for i, (o, w) in enumerate(zip(out, want)):
                o_b = o[b:b + 1, :, :kb[b]] if i < 2 else o[b:b + 1]
                assert torch.equal(o_b, w), (it, b, i)
        res, res_p = acc.result(), per.result()
        assert res["num_examples"] == res_p["num_examples"] == len(Ns)
        for k in acc.KEYS:
            assert np.isfinite(res[k]) and abs(res[k] - res_p[k]) <= 1e-12 * abs(res_p[k]), (it, k, res[k], res_p[k])


# ---------------------------------------------------------------- 7: errors -------------------------------------------
def test_batch_ragged_errors(base):
    whole = PairGenerator(base)
    part = PairGenerator(base, partial=True, reserve=RES)
    with pytest.raises(ValueError, match="2 point counts for 3 items"):
        whole.batch_ragged([0, 1, 2], [100, 200])
    with pytest.raises(ValueError, match="base cloud size"):
        whole.batch_ragged([0, 1], [100, NB + 1])
    with pytest.raises(ValueError, match="n_max"):
        whole.batch_ragged([0, 1], [100, 600], n_max=500)
    with pytest.raises(ValueError, match=r"\[21, 600\]"):
        whole.batch_ragged([0, 1], [20, 600])
    with pytest.raises(ValueError, match=r"\[21, 450\]"):
        part.batch_ragged([0, 1], [27, 600])                    # int(27 * RES) = 20
    with pytest.raises(NotImplementedError, match="aligned"):
        PairGenerator(base, aligned=True).batch_ragged([0], [100])
    with pytest.raises(NotImplementedError, match="aligned"):
        PairSource(2, DEV, aligned=True).batch_ragged(0, 1, [100])
    d = whole.batch_ragged([0, 1], [100, 200])
    acc = EvalAccumulator(DEV)
    with pytest.raises(ValueError, match="corrK"):
        acc.update_ragged(d["src"], d["tgt"], d["lengths"], d["src"], d["tgt"][:, :, :5], d["lengths"],
                          d["R_ab"], d["t_ab"], d["R_ab"], d["t_ab"], d["R_ba"], d["t_ba"])
    with pytest.raises(RuntimeError, match="lengths|shape"):
        acc.update_ragged(d["src"], d["tgt"], d["lengths"][:1], d["src"], d["tgt"], d["lengths"],
                          d["R_ab"], d["t_ab"], d["R_ab"], d["t_ab"], d["R_ba"], d["t_ba"])


def test_ragged_entry_points_reject_before_any_launch():
    L = lib()
    st = torch.cuda.current_stream(DEV).cuda_stream
    P, N = 2, 30000
    x = torch.zeros((P, 3, N), dtype=torch.float64, device=DEV)
    n, keep = lens([N, 100]), lens([10, 10])
    out = torch.empty((P, 3, N), dtype=torch.float32, device=DEV)
    wsb = L.vcr_crop_nearest_workspace_bytes(P, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    idx = torch.zeros((P, N), dtype=torch.int32, device=DEV)
    pose = torch.zeros((P, 12), dtype=torch.float64, device=DEV)
    base = torch.zeros((P, 10, 3), dtype=torch.float32, device=DEV)
    f = torch.zeros(64, dtype=torch.float32, device=DEV)
    acc = torch.zeros(8, dtype=torch.float64, device=DEV)
    torch.cuda.synchronize()
    launches = L.vcr_launch_count()
    sort = lambda P_, N_, k_, b_: L.vcr_crop_nearest_sort_ragged(x.data_ptr(), n.data_ptr(), keep.data_ptr(), P_, N_, k_,
                                                                 out.data_ptr(), ws.data_ptr(), b_, st)
    one = lambda P_, N_, k_: L.vcr_crop_nearest_ragged(x.data_ptr(), n.data_ptr(), keep.data_ptr(), P_, N_, k_,
                                                       out.data_ptr(), st)
    assert sort(65536, 32768, 1, wsb) == -2
    assert sort(P, N, 0, wsb) == -2
    assert sort(P, N, N + 1, wsb) == -2
    assert sort(P, N, N, wsb - 1) == -4
    assert one(P, 25601, 10) == -2
    assert one(P, 1000, 0) == -2
    assert one(P, 1000, 1001) == -2
    assert one(0, 1000, 10) == -2
    mp = lambda P_, N_: L.vcr_make_pairs_ragged(base.data_ptr(), P_, 10, idx.data_ptr(), idx.data_ptr(),
                                                pose.data_ptr(), n.data_ptr(), N_, None, None, out.data_ptr(),
                                                out.data_ptr(), st)
    assert mp(0, 100) == -2 and mp(65536, 100) == -2 and mp(P, 0) == -2
    em = lambda B_, N_, M_: L.vcr_eval_metrics_ragged(f.data_ptr(), f.data_ptr(), n.data_ptr(), N_, f.data_ptr(),
                                                      f.data_ptr(), n.data_ptr(), M_, f.data_ptr(), f.data_ptr(),
                                                      f.data_ptr(), f.data_ptr(), f.data_ptr(), f.data_ptr(), B_,
                                                      acc.data_ptr(), st)
    assert em(0, 4, 4) == -2 and em(65536, 4, 4) == -2 and em(1, 0, 4) == -2 and em(1, 4, 0) == -2
    assert L.vcr_launch_count() == launches
    assert sort(P, N, N, wsb) == 0
    assert L.vcr_launch_count() > launches
