"""Value range of the LPD pre-training backward.

The "h3" GEMM carries every fp32 operand as hi = fp16(x), lo = fp16((x - hi) * 2^11); it is fp32-exact only while the
operands sit inside fp16's normal range.  The LPD loss is a mean over B*32 anchors, so its gradients shrink with the
batch and the cloud size.  These tests pin the operand window of the h3 GEMM, the loss-scale invariance of the LPDNet
backward, the backward at the bench's pre-training size (16 pairs x 1024 points) with the real loss, the csrc/train.cu
kernels against fp64, and that the backward routes every max over k to the edge whose value the forward kept."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden, rel_err

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops
    from vcr_net_b200 import functional as Fn
from oracle.ref_harness import default_args

DEV = "cuda:0"


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def nump(t):
    return t.detach().cpu().numpy()


def f64(t):
    return t.detach().cpu().double().numpy()


class _precision:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        self.old = config.precision
        config.set_precision(self.mode)

    def __exit__(self, *exc):
        config.set_precision(self.old)


@pytest.fixture(params=[0, 1], ids=["single-cta", "cta-pair"])
def gemm_pair(request):
    old = ops.set_gemm_pair(request.param)
    yield request.param
    ops.set_gemm_pair(old)


def _lpd(num_points):
    lpd_w = load_golden("lpd_pretrained_weights")
    net = V.LPD(default_args(model="lpd", num_points=num_points)).to(DEV).train()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in lpd_w.items()}, strict=True)
    return net


# ---------------------------------------------------------------- 1. operand range of the h3 GEMM --------------------
# Window of max|operand| over which the h3 GEMM stays at the fp32 level (3e-6 max-norm against fp64).
H3_WINDOW = (-17, 15)
SWEEP = range(-30, 16)


def _h3_split_f64(op):
    """hi, lo planes of an "h3" Operand as float64 (exact)."""
    b = op.buf[:, :, :op.cols].cpu().double().numpy()
    return b[0], b[1]


def test_to_operand_reconstructs_inside_the_window():
    """hi + lo / 2048 == x to 2^-22 relative (max-norm) for max|x| in [2^-14, 2^15]: hi keeps 11 significant bits, and
    lo, when subnormal, still resolves 2^-36 absolute.  Below 2^-14 hi itself is subnormal and the error doubles per
    binade (split model: 4.8e-7 at 2^-15, 1.5e-5 at 2^-20, 1.6e-2 at 2^-30).  x = uniform(-1, 1) * 2^e has
    max|x| just below 2^e, so the sweep starts at e = -13."""
    rs = np.random.RandomState(3)
    x0 = rs.uniform(-1.0, 1.0, (257, 516)).astype(np.float32)
    x0[0, :4] = [1.0, -1.0, 0.0, 2.0 ** -12]
    for e in range(-13, 16):
        x = x0 * np.float32(2.0 ** e)
        hi, lo = _h3_split_f64(ops.to_operand(cu(x), "h3"))
        assert np.isfinite(hi).all() and np.isfinite(lo).all(), e
        assert np.array_equal(hi, x.astype(np.float16).astype(np.float64)), e        # round to nearest even
        assert rel_err(hi + lo / 2048.0, x) <= 2.0 ** -22, (e, rel_err(hi + lo / 2048.0, x))


@pytest.mark.parametrize("M,N,K", [(256, 256, 512), (300, 200, 520)])
def test_gemm_h3_operand_range(M, N, K, gemm_pair):
    """A and B uniform in +-2^e, swept separately over e = -30 .. 15 (the other operand uniform in +-1), against fp64.

    Measured on a B200 (max-norm relative error over both shapes and both sides; the single-CTA and CTA-pair kernels
    give the same bits):
      2^-14 .. 2^15    6.9e-7 .. 1.0e-6 (fp32 level)
      2^-16 1.0e-6 .. 1.3e-6    2^-17 1.9e-6 .. 2.4e-6    2^-18 3.6e-6 .. 4.3e-6
      2^-20 1.4e-5 .. 1.7e-5    2^-24 2.3e-4 .. 2.9e-4    2^-27 1.8e-3 .. 2.4e-3    2^-30 1.3e-2 .. 1.6e-2
    (hi turns subnormal below 2^-14 and the error doubles per binade).  Above 65504, hi is inf and the product NaN."""
    rs = np.random.RandomState(M + N + K)
    a0 = rs.uniform(-1.0, 1.0, (M, K)).astype(np.float32)
    b0 = rs.uniform(-1.0, 1.0, (N, K)).astype(np.float32)
    errs = {}
    c = torch.empty(M, N, device=DEV)
    for side in ("A", "B"):
        for e in SWEEP:
            s = np.float32(2.0 ** e)
            a, b = (a0 * s, b0) if side == "A" else (a0, b0 * s)
            ref = a.astype(np.float64) @ b.astype(np.float64).T
            c.fill_(float("nan"))
            ops.gemm_tc(ops.to_operand(cu(a), "h3"), ops.to_operand(cu(b), "h3"), M, N, K, c=c)
            errs[(side, e)] = rel_err(nump(c), ref)
    print({f"{s}2^{e}": f"{v:.1e}" for (s, e), v in errs.items()})
    inside = {k: v for k, v in errs.items() if H3_WINDOW[0] <= k[1] <= H3_WINDOW[1]}
    assert max(inside.values()) < 3e-6, inside
    # outside the window the error is set by fp16's subnormal spacing (~2^(-36-e)), not by a fault
    for (side, e), v in errs.items():
        assert v < max(3e-6, 8 * 2.0 ** (-36 - e)), (side, e, v)


# ---------------------------------------------------------------- 2. loss-scale invariance of the LPDNet backward -----
def _golden_setup():
    g = load_golden("lpd_train")
    x = cu(np.concatenate([g["src"], g["tgt"]], axis=0))
    keep = np.unpackbits(g["Rw_keep_bits"])[:4 * 512 * 256].reshape(4, 512, 256).astype(np.float32)
    Rw = cu(np.random.RandomState(7).standard_normal((4, 512, 256)).astype(np.float32) * keep)   # see make_golden.py
    return g, x, Rw, cu(g["idx_feat"], torch.int32), cu(g["idx_xyz"], torch.int32)


@pytest.mark.parametrize("mode", ["fp32", "h3"])
def test_lpdnet_backward_is_loss_scale_invariant(mode):
    """Backpropagate s * sum(emb * Rw) for s = 1, 2^-10, 2^-20, 2^-30: the exact gradient is s * (the s = 1 gradient),
    and power-of-two scaling is exact in fp32.  fp32: grad / s equals the s = 1 run up to the order of the fp32 atomics
    (wgrad, edge_bwd_scatter).  h3: grad / s matches the reference autograd gradient at every s.  Without the
    power-of-two rescaling of g_emb in LPDNetTrainFn.backward, h3 measured 9.0e-5 at s = 2^-20 and 7.6e-2 at 2^-30."""
    g, x, Rw, idx_f, idx_x = _golden_setup()
    net = _lpd(256)
    emb = net.emb_nn
    grads = {}
    with _precision(mode):
        for e in (0, -10, -20, -30):
            s = 2.0 ** e
            emb.zero_grad(set_to_none=True)
            out = emb(x, idx_feat=idx_f, idx_xyz=idx_x)
            (s * (out * Rw).sum()).backward()
            grads[e] = {n: f64(p.grad) / s for n, p in emb.named_parameters()}
    errs = {}
    for e, gr in grads.items():
        for n, v in gr.items():
            want = grads[0][n] if mode == "fp32" else g["ga." + n]
            errs[(e, n)] = rel_err(v, want)
    worst = {e: max(v for (ee, _), v in errs.items() if ee == e) for e in grads}
    print(mode, {f"2^{e}": f"{v:.2e}" for e, v in worst.items()})
    # fp32: the reordered atomics alone measured up to 1.2e-6 (conv1_lpd.bias, a sum over all points with cancellation)
    assert max(errs.values()) < (4e-6 if mode == "fp32" else 1e-4), {k: v for k, v in errs.items() if v >= 1e-6}


# ---------------------------------------------------------------- 3. the real loss at the bench's size ----------------
def _lpd_loss_grads(net, src, tgt, idx_f, idx_x):
    """LPD.forward + getLoss with injected neighbour sets; -> (per-parameter gradients, g_emb [2B, 512, N])."""
    B = src.shape[0]
    net.zero_grad(set_to_none=True)
    both = net.emb_nn(torch.cat([src, tgt], dim=0), idx_feat=idx_f, idx_xyz=idx_x)
    seen = {}
    both.register_hook(lambda gr: seen.setdefault("g", gr.detach().clone()))
    loss = net.getLoss(src, both[:B], both[B:])
    loss.backward()
    return {n: f64(p.grad) for n, p in net.emb_nn.named_parameters()}, seen["g"], float(loss.detach())


def test_lpd_loss_grads_at_bench_size_h3_vs_fp32():
    """16 pairs x 1024 points (the bench's lpd-train batch), the real LPD loss.  The fp32 run's neighbour sets are
    injected into the h3 run so both route through the same neighbours.

    Measured on a B200: max|g_emb| = 1.0e-5 (2^-16.6, at the edge of the h3 window), median of the nonzero entries
    1e-10, smallest 2e-18.  The gradients of the two modes differ by at most 1.2e-3 (conv1_lpd.bias; conv3_lpd 1.7e-5),
    the same with and without the rescaling of g_emb: the triplet term's gradient sits on 32 anchors per cloud, and the
    1e-7 differences of the two forwards move a few arg-max routes and LeakyReLU kinks among them.  The bound is set
    above that."""
    from oracle import synth
    pa = synth.make_pairs(16, 1024, aligned=True, first_item=900)
    src, tgt = cu(pa["src"]), cu(pa["tgt"])
    net = _lpd(1024)
    st = {}
    with _precision("fp32"), torch.no_grad():
        net.emb_nn.forward_tokens(torch.cat([src, tgt], dim=0), stages=st)
    idx_f, idx_x = st["idx_feat"].clone(), st["idx_xyz"].clone()
    with _precision("fp32"):
        g32, ge32, l32 = _lpd_loss_grads(net, src, tgt, idx_f, idx_x)
    with _precision("h3"):
        gh3, geh3, lh3 = _lpd_loss_grads(net, src, tgt, idx_f, idx_x)
    a = ge32.abs()
    nz = a[a > 0]
    print(f"|g_emb| at 16 x 1024: max {float(a.max()):.3e}, median nonzero {float(nz.median()):.3e}, "
          f"min nonzero {float(nz.min()):.3e}; loss fp32 {l32:.6f} h3 {lh3:.6f}")
    errs = {n: rel_err(gh3[n], g32[n]) for n in g32}
    print({k: f"{v:.2e}" for k, v in errs.items()})
    assert abs(lh3 - l32) < 1e-4 * max(1.0, abs(l32))
    assert max(errs.values()) < 2e-3, errs


# ---------------------------------------------------------------- 4. csrc/train.cu kernels against fp64 --------------
def _leaky(v, slope):
    return np.where(v >= 0, v, v * np.asarray(slope, dtype=v.dtype))


def _cloud_with_ties(rs, B, N, C, step=0.125):
    """[B, N, C] rows of a cloud with duplicated points (rows 2i+1 copy rows 2i in a third of the pairs) and values on a
    coarse grid, so that maxima over neighbours tie exactly, across and within rows."""
    x = np.round(rs.randn(B, N, C) / step) * step
    dup = rs.rand(N // 2) < 0.33
    rows = np.nonzero(dup)[0] * 2
    x[:, rows + 1] = x[:, rows]
    return x.astype(np.float32)


def _neighbours(rs, B, N, k):
    return np.stack([np.stack([rs.choice(N, k, replace=False) for _ in range(N)]) for _ in range(B)]).astype(np.int32)


def _first_argmax(v, axis):
    return np.argmax(v, axis=axis)             # numpy returns the first of equal maxima, like torch.max(dim)


KERNEL_CASES = [(k, C, slope) for k in (1, 20) for C in (128, 256) for slope in (0.0, 0.2)]


@pytest.mark.parametrize("k,C,slope", KERNEL_CASES)
def test_gather_max_bwd_vs_fp64(k, C, slope):
    """x3 = act(max_k P[nbr] + Q): gQ = g * act'(s), gP[arg-max neighbour] += the same, on the strided [P3 | Q3] column
    views the product passes (ld 2C), 3 clouds, exact ties going to the lowest k."""
    rs = np.random.RandomState(k * 1000 + C + int(slope * 10))
    B, N = 3, 97
    pq = np.concatenate([_cloud_with_ties(rs, B, N, C), _cloud_with_ties(rs, B, N, C)], axis=2)
    idx = _neighbours(rs, B, N, k)
    gout = rs.randn(B, N, 2 * C).astype(np.float32)
    P, Q = pq[:, :, :C], pq[:, :, C:]
    pq_d, gout_d = cu(pq), cu(gout)
    gpq = torch.zeros(B, N, 2 * C, device=DEV)
    ops.gather_max_bwd(pq_d[:, :, 0:C], pq_d[:, :, C:], cu(idx), slope, gout_d[:, :, C:], gpq[:, :, 0:C], gpq[:, :, C:])
    vals = P[np.arange(B)[:, None, None], idx]                                         # [B, N, k, C]
    kk = _first_argmax(vals, axis=2)                                                     # [B, N, C]
    best = np.take_along_axis(vals, kk[:, :, None, :], axis=2)[:, :, 0, :]
    s = best.astype(np.float64) + Q
    g = gout[:, :, C:] * np.where(s > 0, np.float32(1.0), np.float32(slope))
    assert np.array_equal(nump(gpq[:, :, C:]), g)
    j = idx[np.arange(B)[:, None, None], np.arange(N)[None, :, None], kk]              # [B, N, C] neighbour row
    gP = np.zeros((B, N, C))
    np.add.at(gP, (np.arange(B)[:, None, None], j, np.arange(C)[None, None, :]), g.astype(np.float64))
    assert rel_err(nump(gpq[:, :, 0:C]), gP) < 1e-6


@pytest.mark.parametrize("k,C,slope", KERNEL_CASES)
def test_edge_gather_act_and_edge_max_bwd_vs_fp64(k, C, slope):
    """e1 = act(P[nbr] + Q) from a strided [P | Q] view; edge_max_bwd_ routes g_x (strided) through act' at the max to
    the first arg-max edge of z and zeroes the others."""
    rs = np.random.RandomState(7 * k + C + int(slope * 10))
    B, N = 3, 83
    buf = np.concatenate([_cloud_with_ties(rs, B, N, 2 * C), rs.randn(B, N, 64).astype(np.float32)], axis=2)
    idx = _neighbours(rs, B, N, k)
    E = nump(ops.edge_gather_act(cu(buf)[:, :, :2 * C], cu(idx), slope))
    P, Q = buf[:, :, :C], buf[:, :, C:2 * C]
    want = _leaky(P[np.arange(B)[:, None, None], idx] + Q[:, :, None, :], slope)       # float32, same rounding
    assert np.array_equal(E, want.reshape(B * N * k, C))
    T = B * N
    z = _cloud_with_ties(rs, 1, T * k, C)[0]
    gbuf = rs.randn(T, 2 * C).astype(np.float32)
    zd = cu(z)
    ops.edge_max_bwd_(zd, cu(gbuf)[:, C:], k, slope)
    zk = z.reshape(T, k, C)
    kk = _first_argmax(zk, axis=1)
    best = np.take_along_axis(zk, kk[:, None, :], axis=1)[:, 0, :]
    g = gbuf[:, C:] * np.where(best > 0, np.float32(1.0), np.float32(slope))
    want = np.zeros((T, k, C), dtype=np.float32)
    np.put_along_axis(want, kk[:, None, :], g[:, None, :], axis=1)
    assert np.array_equal(nump(zd).reshape(T, k, C), want)


@pytest.mark.parametrize("k,C,slope", KERNEL_CASES)
def test_edge_bwd_scatter_vs_fp64(k, C, slope):
    """g_e1 (+ g_x1 at the first arg-max edge of e1) through act' -> gQ = sum over edges, gP scattered to the neighbour
    rows, on 3 clouds with exact ties in e1 and a strided g_x1."""
    rs = np.random.RandomState(11 * k + C + int(slope * 10))
    B, N = 3, 89
    T = B * N
    idx = _neighbours(rs, B, N, k)
    e = _cloud_with_ties(rs, 1, T * k, C)[0]
    ge = rs.randn(T * k, C).astype(np.float32)
    gx = rs.randn(T, 3 * C).astype(np.float32)
    gpq = ops.edge_bwd_scatter(cu(e), cu(ge), cu(gx)[:, C:2 * C], cu(idx), slope)
    ek, gek = e.reshape(T, k, C).astype(np.float64), ge.reshape(T, k, C).astype(np.float64)
    kk = _first_argmax(ek, axis=1)
    gek = gek.copy()
    np.put_along_axis(gek, kk[:, None, :], np.take_along_axis(gek, kk[:, None, :], axis=1) + gx[:, None, C:2 * C], axis=1)
    gs = gek * np.where(ek > 0, 1.0, slope)
    gQ = gs.sum(axis=1).reshape(B, N, C)
    gP = np.zeros((B, N, C))
    bi = np.repeat(np.arange(B), N * k * C).reshape(B, N, k, C)
    np.add.at(gP, (bi, np.broadcast_to(idx[:, :, :, None], (B, N, k, C)), np.broadcast_to(np.arange(C), (B, N, k, C))),
              gs.reshape(B, N, k, C))
    assert rel_err(nump(gpq[:, :, C:]), gQ) < 1e-6
    assert rel_err(nump(gpq[:, :, :C]), gP) < 1e-6


@pytest.mark.parametrize("M,N,K", [(1000, 256, 128), (4099, 128, 256), (77, 100, 60)])
def test_wgrad_strided_views_vs_fp64(M, N, K):
    """dW = G^T X, db = column sums of G, with G and X column views of wider rows (ldg = 2N, ldx = K + 64)."""
    rs = np.random.RandomState(M + N + K)
    gbuf = rs.randn(M, 2 * N).astype(np.float32)
    xbuf = rs.randn(M, K + 64).astype(np.float32)
    dW, db = ops.wgrad(cu(gbuf)[:, N:], cu(xbuf)[:, 64:])
    G, X = gbuf[:, N:].astype(np.float64), xbuf[:, 64:].astype(np.float64)
    assert rel_err(nump(dW), G.T @ X) < 1e-5
    assert rel_err(nump(db), G.sum(0)) < 1e-5


# ---------------------------------------------------------------- 5. routing consistency -----------------------------
@pytest.mark.parametrize("mode", ["fp32", "h3", "fp16"])
def test_backward_recomputes_the_forward_maxima(mode):
    """For every max over k of LPDNet (x1, x2, x3), what the backward recomputes must give act(max_k z) == the forward's
    slice of cat bit for bit; otherwise a near-tie sends the gradient to an edge the forward did not keep."""
    from oracle import synth
    net = _lpd(1024)
    m = net.emb_nn
    pa = synth.make_pairs(2, 1024, aligned=True, first_item=41)
    x = torch.cat([cu(pa["src"]), cu(pa["tgt"])], dim=0)
    slope = float(m.negative_slope)
    st = {}
    with _precision(mode), torch.no_grad():
        m.forward_tokens(x, stages=st)
        cat, pq1, pq3, idx_f, idx_x = st["cat"], st["pq1"], st["pq3"], st["idx_feat"], st["idx_xyz"]
        B, N, _ = cat.shape
        k = idx_f.shape[2]
        e1, z2 = Fn.lpdnet_dg2_edges(m, pq1, idx_f)
        x1 = e1.view(B, N, k, 128).amax(dim=2)
        x2 = F.leaky_relu(z2.view(B, N, k, 128).amax(dim=2), slope)
        p3 = pq3[:, :, 0:256]
        nbr = torch.stack([p3[b][idx_x[b].long()] for b in range(B)])                  # [B, N, k, 256]
        x3 = F.leaky_relu(nbr.amax(dim=2) + pq3[:, :, 256:512], slope)
    bad = {name: int((got != cat[:, :, c0:c0 + got.shape[2]]).sum())
           for name, got, c0 in (("x1", x1, 0), ("x2", x2, 128), ("x3", x3, 256))}
    print(mode, "elements that differ from the forward:", bad)
    assert not any(bad.values()), bad
