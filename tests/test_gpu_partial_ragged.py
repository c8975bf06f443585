"""Ragged batches for partial-to-partial registration: every kernel with per-item lengths and counts, and
vcrnetIterRaggedPartial, must give each pair exactly the bits it gets when computed alone."""
import pytest
import torch

import vcr_net_b200.ragged as ragged

DEV = "cuda:0"
OVERLAPS = (0.5, 0.75, 0.9, 1.0)


# ------------------------------------------------------------------ counts (host-checkable arithmetic, run on the device)

@pytest.mark.gpu
@pytest.mark.parametrize("ov", OVERLAPS)
def test_counts_match_python_int_chain(ov):
    n = torch.arange(1, 300001, dtype=torch.int32, device=DEV)
    key, sel, corr = ragged.key_counts(n, ov), ragged.select_counts(n, ov), ragged.corr_lengths(n, ov)
    want_key = torch.tensor([int(i * ov) for i in range(1, 300001)], dtype=torch.int32)
    want_sel = [int(i * 0.84 * ov) for i in range(1, 300001)]
    want_corr = torch.tensor([int(s * 0.52 * ov) for s in want_sel], dtype=torch.int32)
    assert torch.equal(key.cpu(), want_key)
    assert torch.equal(sel.cpu(), torch.tensor(want_sel, dtype=torch.int32))
    assert torch.equal(corr.cpu(), want_corr)


if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops
    from vcr_net_b200 import functional as Fn

from oracle import synth
from oracle.ref_harness import default_args

pytestmark = pytest.mark.gpu


def _lens(x):
    return torch.tensor(x, dtype=torch.int32, device=DEV)


# ------------------------------------------------------------------ top-K

TOPK_N = [1, 2, 21, 31, 32, 33, 1024, 1025, 4097, 16384]


@pytest.mark.parametrize("kind", ["random", "ties"])
def test_topk_ragged_equals_each_row_alone(kind):
    g = torch.Generator().manual_seed(3)
    N = max(TOPK_N)
    rows = []
    for n in TOPK_N:
        v = torch.randn(n, generator=g) if kind == "random" else torch.randint(-3, 4, (n,), generator=g).float()
        if kind == "ties":
            v[v == 0] = torch.where(torch.rand(int((v == 0).sum()), generator=g) < 0.5, -0.0, 0.0)
        rows.append(v)
    for which in ("one", "all"):
        ks = [1 if which == "one" else n for n in TOPK_N]
        vals = torch.full((len(TOPK_N), N), 1e4)
        for b, v in enumerate(rows):
            vals[b, :len(v)] = v
            vals[b, len(v):] = 1e4 if b % 2 else -1e4                   # padding must never be picked
        vals = vals.to(DEV)
        K = max(ks)
        idx, mask = ops.topk_select_ragged(vals, _lens(TOPK_N), _lens(ks), K, want_idx=True, want_mask=True)
        for b, (n, k) in enumerate(zip(TOPK_N, ks)):
            wi, wm = ops.topk_select(rows[b][None].to(DEV), k, want_idx=True, want_mask=True)
            assert torch.equal(idx[b, :k], wi[0]), (b, n, k)
            assert torch.equal(mask[b, :n], wm[0]), (b, n, k)
            assert not idx[b, k:].any() and not mask[b, n:].any(), (b, n, k)


# ------------------------------------------------------------------ key statistic and flash attention with keep

# (nq, nk): 128-tile crossings and both sides of the rows-per-CTA bend at 436 keys
STAT_LENGTHS = [(21, 300), (128, 436), (129, 437), (700, 768), (300, 2100), (1000, 129)]
H, DK, D = 4, 128, 512


def _qkv(mode, seed=2):
    B = len(STAT_LENGTHS)
    Nq, Nk = max(a for a, _ in STAT_LENGTHS), max(b for _, b in STAT_LENGTHS)
    g = torch.Generator().manual_seed(seed)
    q = torch.randn((B, Nq, D), generator=g)
    k = torch.randn((B, Nk, D), generator=g)
    vt = torch.randn((B, D, Nk), generator=g)
    for b, (mq, mk) in enumerate(STAT_LENGTHS):                        # garbage padding
        q[b, mq:] = 1e4
        k[b, mk:] = -1e4
        vt[b, :, mk:] = 3.0
    q_op = ops.to_operand(q.view(B * Nq, D).to(DEV), mode)
    k_op = ops.to_operand(k.view(B * Nk, D).to(DEV), mode)
    vt_op = ops.to_operand(vt.view(B * D, Nk).to(DEV), mode)
    return B, Nq, Nk, q_op, k_op, vt_op


def _scores(q_op, k_op, nb, Nq, Nk):
    ldS = (Nk + 3) // 4 * 4
    S = torch.empty((nb, H, Nq, ldS), dtype=torch.float32, device=DEV)
    ops.gemm_tc(q_op, k_op, Nq, Nk, DK, nbo=nb, nbi=H, a_off=(Nq, 0, 0, DK), b_off=(Nk, 0, 0, DK), alpha=DK ** -0.5, c=S,
                c_strides=(H * Nq * ldS, Nq * ldS))
    return S


@pytest.mark.parametrize("route", ["tc_h3", "softmax_h3", "softmax_fp16", "softmax_bf16"])
def test_key_statistic_ragged_equals_each_item_alone(route):
    mode = route.split("_")[1]
    B, Nq, Nk, q_op, k_op, _ = _qkv(mode)
    nq, nk = _lens([a for a, _ in STAT_LENGTHS]), _lens([b for _, b in STAT_LENGTHS])
    if route == "tc_h3":
        got = ops.attn_colsum_tc_ragged(q_op, k_op, B, H, Nq, Nk, DK, DK ** -0.5, nq, nk)
    else:
        got = ops.softmax_colsum_ragged(_scores(q_op, k_op, B, Nq, Nk), H, Nq, Nk, nq, nk)
    for b, (mq, mk) in enumerate(STAT_LENGTHS):
        qb, kb = q_op.rows_view(b * Nq, mq), k_op.rows_view(b * Nk, mk)
        if route == "tc_h3":
            want = ops.attn_colsum_tc(qb, kb, 1, H, mq, mk, DK, DK ** -0.5)
        else:
            S = _scores(qb, kb, 1, mq, mk)
            want = ops.colsum_softmax(S.view(H * mq, S.shape[-1]), mk, 1)
        assert torch.equal(got[b:b + 1, :mk], want), (b, mq, mk)
        assert not got[b, mk:].any(), b


@pytest.mark.parametrize("mode", ["h3", "fp16", "bf16"])
def test_flash_keep_ragged_equals_each_item_alone(mode):
    B, Nq, Nk, q_op, k_op, vt_op = _qkv(mode, seed=5)
    nq, nk = _lens([a for a, _ in STAT_LENGTHS]), _lens([b for _, b in STAT_LENGTHS])
    g = torch.Generator().manual_seed(8)
    keep = (torch.rand((B, Nk), generator=g) < 0.6).to(torch.uint8).to(DEV)
    out = ops.Operand.empty(B * Nq, D, mode, DEV)
    out.buf.fill_(float("nan"))
    ops.flash_attn_tc_ragged_keep(q_op, k_op, vt_op, out, B, H, Nq, Nk, DK, DK ** -0.5, nq, nk, keep)
    for b, (mq, mk) in enumerate(STAT_LENGTHS):
        vt_b = ops.Operand.empty(D, mk, mode, DEV)
        vt_b.buf[:, :, :mk] = vt_op.buf[:, b * D:(b + 1) * D, :mk]
        o_b = ops.Operand.empty(mq, D, mode, DEV)
        ops.flash_attn_tc(q_op.rows_view(b * Nq, mq), k_op.rows_view(b * Nk, mk), vt_b, o_b, 1, H, mq, mk, DK, DK ** -0.5,
                          keep=keep[b:b + 1, :mk].contiguous())
        assert torch.equal(out.buf[:, b * Nq:b * Nq + mq, :D], o_b.buf[:, :, :D]), (b, mq, mk)


# ------------------------------------------------------------------ selectCom statistics and getCopair

SEL_NT = [21, 700, 1024, 1025, 3000]
SEL_NS = [300, 21, 1500, 64, 900]


def _tokens(lengths, seed, fill):
    g = torch.Generator().manual_seed(seed)
    N = max(lengths)
    x = torch.full((len(lengths), N, 128), fill)
    for b, n in enumerate(lengths):
        x[b, :n] = torch.randn((n, 128), generator=g) * 0.3
    return x.to(DEV)


def test_select_stats_ragged_equals_each_pair_alone():
    s_tok, t_tok = _tokens(SEL_NS, 1, 50.0), _tokens(SEL_NT, 2, -50.0)
    B, Ns, Nt = len(SEL_NS), max(SEL_NS), max(SEL_NT)
    row, col = Fn._select_stats_ragged(s_tok, t_tok, None, B, Ns, Nt, _lens(SEL_NS), _lens(SEL_NT))
    for b, (ms, mt) in enumerate(zip(SEL_NS, SEL_NT)):
        want = Fn._select_stats_materialised(s_tok[b:b + 1, :ms], t_tok[b:b + 1, :mt], None, 1, ms, mt)
        assert torch.equal(row[b:b + 1, :ms], want[0]), (b, ms, mt)
        assert torch.equal(col[b:b + 1, :mt], want[1]), (b, ms, mt)
        assert not row[b, ms:].any() and not col[b, mt:].any(), b


def test_softcorr_best_ragged_equals_each_pair_alone():
    s_tok, t_tok = _tokens(SEL_NS, 3, 9.0), _tokens(SEL_NT, 4, -9.0)
    B, Ns, Nt = len(SEL_NS), max(SEL_NS), max(SEL_NT)
    xx, yy = ops.sqnorm_rows(s_tok), ops.sqnorm_rows(t_tok)
    s_op, t_op = ops.to_operand(s_tok.view(B * Ns, 128), "h3"), ops.to_operand(t_tok.view(B * Nt, 128), "h3")
    bi, bv = ops.softcorr_best_tc_ragged(s_op, t_op, xx, yy, B, Ns, Nt, 128, _lens(SEL_NS), _lens(SEL_NT))
    for b, (ms, mt) in enumerate(zip(SEL_NS, SEL_NT)):
        wi, wv = ops.softcorr_best_tc(s_op.rows_view(b * Ns, ms), t_op.rows_view(b * Nt, mt), xx[b:b + 1, :ms].contiguous(),
                                      yy[b:b + 1, :mt].contiguous(), 1, ms, mt, 128)
        assert torch.equal(bi[b:b + 1, :ms], wi) and torch.equal(bv[b:b + 1, :ms], wv), b
        assert not bi[b, ms:].any() and not bv[b, ms:].any(), b


# ------------------------------------------------------------------ end to end

SRC_LENGTHS = [21, 300, 768, 1000, 1100, 640]
TGT_LENGTHS = [64, 1300, 21, 1024, 700, 1025]


def _net(ckpt, **kw):
    net = V.VCRNet(default_args(partial=True, **kw)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=False)
    return net


def _pairs(src_n, tgt_n, seed=77):
    # a partial cloud keeps int(num_points * reserve) points, reserve < 1
    p = synth.make_pairs(len(src_n), 2 * max(max(src_n), max(tgt_n)), partial=True, seed=seed)
    src = [torch.from_numpy(p["src"][b, :, :n]).to(DEV) for b, n in enumerate(src_n)]
    tgt = [torch.from_numpy(p["tgt"][b, :, :n]).to(DEV) for b, n in enumerate(tgt_n)]
    return src, tgt


@pytest.fixture(scope="module")
def pairs():
    return _pairs(SRC_LENGTHS, TGT_LENGTHS)


def _check_against_alone(net, src_l, tgt_l, it):
    src, sl = ragged.pad_clouds(src_l)
    tgt, tl = ragged.pad_clouds(tgt_l)
    out = V.vcrnetIterRaggedPartial(net, src, tgt, sl, tl, iter=it)
    kb = ragged.corr_lengths(sl, net.head.overlap2).tolist()
    assert out[0].shape[2] == int(int(src.shape[2] * 0.84 * net.head.overlap2) * 0.52 * net.head.overlap2)
    for b in range(len(src_l)):
        want = V.vcrnetIter(net, src_l[b][None], tgt_l[b][None], iter=it)
        assert want[0].shape[2] == kb[b]
        for i, (o, w) in enumerate(zip(out, want)):
            o_b = o[b:b + 1, :, :kb[b]] if i < 2 else o[b:b + 1]
            assert torch.equal(o_b, w), (b, i)
        for i in (0, 1):
            assert not out[i][b, :, kb[b]:].any(), (b, i)
    return out


@pytest.mark.parametrize("mode,it,cycle", [("h3", 1, False), ("h3", 3, True), ("fp16", 1, True), ("fp16", 3, False),
                                           ("bf16", 1, False), ("bf16", 3, True)])
def test_partial_ragged_equals_each_pair_alone(ckpt, pairs, mode, it, cycle):
    old = config.precision
    config.set_precision(mode)
    try:
        _check_against_alone(_net(ckpt, cycle=cycle), *pairs, it)
    finally:
        config.set_precision(old)


@pytest.mark.parametrize("ov", [0.75, 0.6])
def test_partial_ragged_identity_pointer_and_overlap(ckpt, pairs, ov):
    _check_against_alone(_net(ckpt, pointer="identity", overlap2=ov), *pairs, 2)
    _check_against_alone(_net(ckpt, overlap2=ov), pairs[0][:3], pairs[1][:3], 1)


def test_partial_ragged_up_to_16384_points(ckpt):
    src_l, tgt_l = _pairs([16384, 2100], [5000, 16384], seed=5)
    _check_against_alone(_net(ckpt), src_l, tgt_l, 1)


def test_partial_ragged_padding_neighbour_graph_and_stream(ckpt, pairs):
    net = _net(ckpt)
    src_l, tgt_l = pairs
    src, sl = ragged.pad_clouds(src_l)
    tgt, tl = ragged.pad_clouds(tgt_l)
    base = V.vcrnetIterRaggedPartial(net, src, tgt, sl, tl, iter=2)
    g = torch.Generator(device=DEV).manual_seed(9)
    s2, t2 = src.clone(), tgt.clone()
    for b in range(src.shape[0]):
        s2[b, :, SRC_LENGTHS[b]:] = (torch.rand(s2[b, :, SRC_LENGTHS[b]:].shape, generator=g, device=DEV) - 0.5) * 2e4
        t2[b, :, TGT_LENGTHS[b]:] = (torch.rand(t2[b, :, TGT_LENGTHS[b]:].shape, generator=g, device=DEV) - 0.5) * 2e4
    for a, c in zip(base, V.vcrnetIterRaggedPartial(net, s2, t2, sl, tl, iter=2)):
        assert torch.equal(a, c)
    s3, sl3 = src.clone(), sl.clone()
    s3[0] = src[2]
    sl3[0] = SRC_LENGTHS[2]
    for a, c in zip(base, V.vcrnetIterRaggedPartial(net, s3, tgt, sl3, tl, iter=2)):
        assert torch.equal(a[1:], c[1:])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = V.vcrnetIterRaggedPartial(net, src, tgt, sl, tl, iter=2)
    torch.cuda.current_stream().wait_stream(s)
    for a, c in zip(side, base):
        assert torch.equal(a, c)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = V.vcrnetIterRaggedPartial(net, src, tgt, sl, tl, iter=2)
    order = [3, 0, 5, 1, 2, 4]
    ps, nsl = ragged.pad_clouds([src_l[i] for i in order], n_max=src.shape[2])
    pt, ntl = ragged.pad_clouds([tgt_l[i] for i in order[::-1]], n_max=tgt.shape[2])
    src.copy_(ps); tgt.copy_(pt); sl.copy_(nsl); tl.copy_(ntl)
    graph.replay()
    for a, c in zip(static_out, V.vcrnetIterRaggedPartial(net, ps, pt, nsl, ntl, iter=2)):
        assert torch.equal(a, c)


def test_partial_ragged_errors(ckpt, pairs):
    src_l, tgt_l = pairs
    src, sl = ragged.pad_clouds(src_l[:2])
    tgt, tl = ragged.pad_clouds(tgt_l[:2])
    net = _net(ckpt)
    big, bl = ragged.pad_clouds(src_l[:2], n_max=16385)
    with pytest.raises(NotImplementedError, match="16384"):
        V.vcrnetIterRaggedPartial(net, big, tgt, bl, tl)
    with pytest.raises(NotImplementedError, match="DataParallel"):
        V.vcrnetIterRaggedPartial(torch.nn.DataParallel(net, device_ids=[0]), src, tgt, sl, tl)
    for kw, msg in ((dict(emb_nn="dgcnn"), "DGCNN"), (dict(vcp_nn="att"), "VcpAtt")):
        with pytest.raises(NotImplementedError, match=msg):
            V.vcrnetIterRaggedPartial(V.VCRNet(default_args(partial=True, **kw)).to(DEV).eval(), src, tgt, sl, tl)
    with pytest.raises(NotImplementedError, match="partial"):
        V.vcrnetIterRaggedPartial(V.VCRNet(default_args()).to(DEV).eval(), src, tgt, sl, tl)
    with pytest.raises(ValueError, match="overlap2"):
        V.vcrnetIterRaggedPartial(_net(ckpt, overlap2=0.05), src, tgt, sl, tl)
    old = config.precision
    config.set_precision("fp32")
    try:
        with pytest.raises(NotImplementedError, match="fp32"):
            V.vcrnetIterRaggedPartial(net, src, tgt, sl, tl)
    finally:
        config.set_precision(old)
