"""Partial-to-partial registration above 16 384 points per cloud.

* Top-K selection on one thread-block cluster per row (csrc/select.cu topk_sort_cluster_kernel, 16 384 < n <= 262 144):
  exact equality with the canonical order of oracle.vcr_oracle.topk_desc.
* selectCom's statistics on tensor cores without the [Ns, Nt] score matrix (csrc/softcorr_tc.cu, vcr_select_stats_tc)
  against float64 and against the materialised path on the same operands.
* VCRNet(partial=True) end to end at 20 480 and 65 536 points.
"""
import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops
    from vcr_net_b200 import functional as Fn
from oracle import synth
from oracle import vcr_oracle as O
from oracle.ref_harness import default_args

DEV = "cuda:0"
OV2 = synth.OVERLAP2_0575


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def nump(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------- top-K ------------------------------------------------
def tie_heavy_rows(B, n, seed):
    """Values rounded to 0.1 (about 60 distinct values per row), +0 and -0 both present, row 1 constant."""
    rs = np.random.RandomState(seed)
    v = np.round(rs.randn(B, n), 1).astype(np.float32)
    z = rs.rand(B, n)
    v[z < 0.05] = 0.0
    v[(z >= 0.05) & (z < 0.1)] = -0.0
    if B > 1:
        v[1] = 0.5
    return v


def check_topk(v, K, stream=None):
    x = cu(v)
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream(DEV))
        with torch.cuda.stream(stream):
            idx, mask = ops.topk_select(x, K, want_idx=True, want_mask=True)
        stream.synchronize()
    else:
        idx, mask = ops.topk_select(x, K, want_idx=True, want_mask=True)
    want = O.topk_desc(v, K, axis=-1)
    got = nump(idx)
    assert got.dtype == np.int32 and np.array_equal(got, want), (got != want).sum()
    want_mask = np.zeros(v.shape, dtype=np.uint8)
    np.put_along_axis(want_mask, want, 1, axis=-1)
    assert np.array_equal(nump(mask), want_mask)


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("kind", ["one", "select", "all"])
@pytest.mark.parametrize("n", [16385, 40000, 100000, 229376, 262144])     # C = 2, 4, 8, 16, 16
def test_topk_cluster_sizes(n, kind, B):
    K = {"one": 1, "select": int(0.84 * 0.575 * n), "all": n}[kind]
    check_topk(tie_heavy_rows(B, n, n + B), K)


def test_topk_boundary_between_kernels():
    """16 384 values run on the one-CTA kernel, 16 385 on a cluster of two: prefixes of one row, both canonical."""
    v = tie_heavy_rows(1, 16385, 7)
    for n in (16384, 16385):
        for K in (1, int(0.84 * 0.575 * n), n):
            check_topk(np.ascontiguousarray(v[:, :n]), K)


def test_topk_cluster_waves_on_side_stream():
    """64 rows on clusters of 8 CTAs (one CTA per SM) run in several waves; launched on a non-default stream."""
    v = tie_heavy_rows(64, 100000, 64)
    check_topk(v, int(0.84 * 0.575 * 100000), stream=torch.cuda.Stream(device=DEV))


def test_topk_limit_is_named():
    x = torch.zeros(1, 262145, device=DEV)
    with pytest.raises(RuntimeError, match="262144"):
        ops.topk_select(x, 10)


# ---------------------------------------------------------------- selectCom statistics --------------------------------
def layernormed(B, N, seed):
    """LayerNorm-ed random rows (|f|^2 ~ 512, so the logits cancel as they do in the model): fp32 tokens + head operands."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(B, N, 512, device=DEV, generator=g)
    one, zero = torch.ones(512, device=DEV), torch.zeros(512, device=DEV)
    out, op, sq = ops.layernorm_head(x, one, zero)
    return out, Fn.HeadPre(op, sq)


def stats64(s, t):
    """selectCom's statistics (oracle.select_com) in float64: (row_stat [B,Ns], col_stat [B,Nt])."""
    s, t = s.double(), t.double()
    xx, yy = (s * s).sum(-1), (t * t).sum(-1)
    pd = (-xx[:, :, None] + 2.0 * torch.bmm(s, t.transpose(1, 2))) - yy[:, None, :]
    col = torch.softmax(pd, dim=2).sum(dim=1)
    row = torch.softmax(pd, dim=1).sum(dim=2)
    return row, col


def jaccard_near_ties(got, want64, K, tol):
    """Jaccard index of the top-K sets; every element in one set only must sit within tol of the float64 K-th value."""
    a, b = set(O.topk_desc(got, K).tolist()), set(O.topk_desc(want64, K).tolist())
    kth = np.sort(want64)[::-1][K - 1]
    for e in a ^ b:
        assert abs(want64[e] - kth) <= tol * np.abs(want64).max(), (e, want64[e], kth)
    return len(a & b) / len(a | b)


@pytest.mark.parametrize("B,Ns,Nt", [(2, 768, 768), (3, 257, 331), (1, 40, 1024), (1, 16385, 20000)])
def test_select_stats_tc(B, Ns, Nt):
    s_tok, ps = layernormed(B, Ns, 1000 + Ns)
    t_tok, pt = layernormed(B, Nt, 2000 + Nt)
    row, col = ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, Ns, Nt, 512)
    row2, col2 = ops.select_stats_tc(ps.op, pt.op, ps.sq, pt.sq, B, Ns, Nt, 512)
    assert torch.equal(row, row2) and torch.equal(col, col2)
    row64, col64 = (nump(a) for a in stats64(s_tok, t_tok))
    mrow, mcol = (nump(a) for a in Fn._select_stats_materialised(None, None, (ps, pt), B, Ns, Nt))
    row, col = nump(row), nump(col)
    e64 = (rel_err(row, row64), rel_err(col, col64))
    emat = (rel_err(row, mrow), rel_err(col, mcol))
    jac = []
    for b in range(B):
        jac.append(jaccard_near_ties(col[b], col64[b], int(Nt * 0.84 * OV2), 1e-4))
        jac.append(jaccard_near_ties(row[b], row64[b], int(Ns * 0.84 * OV2), 1e-4))
    print(f"[select_stats_tc] B={B} Ns={Ns} Nt={Nt}: rel_err vs fp64 row {e64[0]:.3g} col {e64[1]:.3g}; "
          f"vs materialised row {emat[0]:.3g} col {emat[1]:.3g}; top-K Jaccard min {min(jac):.4f}")
    assert max(e64) < 1e-4 and max(emat) < 1e-5
    assert min(jac) >= 0.99


# ---------------------------------------------------------------- end to end ------------------------------------------
@pytest.fixture(scope="module")
def net_partial(ckpt):
    net = V.VCRNet(default_args(partial=True, overlap2=OV2)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=True)
    return net


@pytest.fixture
def precision_mode(request):
    old = config.precision
    config.set_precision(request.param)
    yield request.param
    config.set_precision(old)


def partial_pairs(B, N, first_item):
    """B partial pairs whose clouds hold exactly N points after the crop (oracle.synth: int(num_points * reserve))."""
    num = int(np.ceil(N / synth.RESERVE_0575))
    while int(num * synth.RESERVE_0575) > N:
        num -= 1
    while int(num * synth.RESERVE_0575) < N:
        num += 1
    p = synth.make_pairs(B, num, partial=True, base_points=num, first_item=first_item)
    assert p["src"].shape[2] == N and p["tgt"].shape[2] == N
    return p


def check_properties(out, B, N):
    M = int(int(N * 0.84 * OV2) * 0.52 * OV2)
    assert tuple(out[0].shape) == (B, 3, M) and tuple(out[1].shape) == (B, 3, M)
    R, t = nump(out[2]).astype(np.float64), nump(out[3]).astype(np.float64)
    assert np.isfinite(R).all() and np.isfinite(t).all()
    assert np.allclose(np.einsum("bij,bkj->bik", R, R), np.eye(3), atol=1e-5)
    assert np.allclose(np.linalg.det(R), 1.0, atol=1e-5)
    Rb, tb = nump(out[4]).astype(np.float64), nump(out[5]).astype(np.float64)
    assert np.allclose(np.einsum("bij,bjk->bik", Rb, R), np.eye(3), atol=1e-5)
    assert np.allclose(np.einsum("bij,bj->bi", Rb, t) + tb, 0, atol=1e-5)
    return M


def check_selected_are_inputs(out1, p, B, M):
    """Iteration 1: every selected source point is an input point (distinct), every correspondence a target point."""
    for b in range(B):
        src_set = {tuple(c) for c in p["src"][b].T.tolist()}
        tgt_set = {tuple(c) for c in p["tgt"][b].T.tolist()}
        sel = nump(out1[0])[b].T.tolist()
        assert all(tuple(c) in src_set for c in sel) and len({tuple(c) for c in sel}) == M
        assert all(tuple(c) in tgt_set for c in nump(out1[1])[b].T.tolist())


@pytest.mark.parametrize("precision_mode", ["h3"], indirect=True)
def test_partial_20480_points_h3(net_partial, precision_mode, product_defaults, monkeypatch):
    N, B = 20480, 2
    p = partial_pairs(B, N, 3)
    src, tgt = cu(p["src"]), cu(p["tgt"])
    for it in (1, 3):
        calls = [V.vcrnetIter(net_partial, src, tgt, iter=it) for _ in range(3)]   # eager, capture, replay
        torch.cuda.synchronize()
        M = check_properties(calls[0], B, N)
        for other in calls[1:]:
            for a, b in zip(calls[0], other):
                assert torch.equal(a, b)
        one = V.vcrnetIter(net_partial, src[1:2], tgt[1:2], iter=it)
        for k in (2, 3):                                                  # R_ab, t_ab
            assert np.abs(nump(one[k]) - nump(calls[0][k])[1:2]).max() < 1e-5
        if it == 1:
            check_selected_are_inputs(calls[0], p, B, M)
    print(f"[partial 20480 h3] peak memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")

    # selectCom's selection inside the network against a float64 selectCom on the network's own head embeddings
    seen = []
    select = Fn.vcp_select

    def recording_select(*a, **kw):
        r = select(*a, **kw)
        seen.append((r[4], r[5]))
        return r

    monkeypatch.setattr(Fn, "vcp_select", recording_select)
    st = {}
    net_partial(src, tgt, stages=st)
    assert seen                                                           # seen[0]: src -> tgt
    row64, col64 = stats64(st["src_emb"], st["tgt_emb"])
    K = int(N * 0.84 * OV2)
    for b in range(B):
        for got, want in ((seen[0][0][b], row64[b]), (seen[0][1][b], col64[b])):
            a, w = set(nump(got).tolist()), set(O.topk_desc(nump(want), K).tolist())
            jac = len(a & w) / len(a | w)
            print(f"[partial 20480 h3] selectCom Jaccard vs fp64, pair {b}: {jac:.4f}")
            assert jac >= 0.98


@pytest.mark.parametrize("precision_mode", ["fp32"], indirect=True)
def test_partial_20480_points_fp32(net_partial, precision_mode):
    N = 20480
    p = partial_pairs(1, N, 5)
    src, tgt = cu(p["src"]), cu(p["tgt"])
    out1 = V.vcrnetIter(net_partial, src, tgt, iter=1)
    M = check_properties(out1, 1, N)
    check_selected_are_inputs(out1, p, 1, M)
    check_properties(V.vcrnetIter(net_partial, src, tgt, iter=3), 1, N)


@pytest.mark.parametrize("precision_mode", ["h3"], indirect=True)
def test_partial_65536_points(net_partial, precision_mode):
    N = 65536
    p = partial_pairs(1, N, 7)
    src, tgt = cu(p["src"]), cu(p["tgt"])
    torch.cuda.reset_peak_memory_stats()
    out = V.vcrnetIter(net_partial, src, tgt, iter=1)
    torch.cuda.synchronize()
    M = check_properties(out, 1, N)
    check_selected_are_inputs(out, p, 1, M)
    print(f"[partial 65536 h3] peak memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")
