"""Ragged batches (pairs of different sizes in one call): every kernel with per-item lengths and vcrnetIterRagged must
give each pair exactly the bits it gets when computed alone."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import vcr_net_b200 as V
    from vcr_net_b200 import config, ops, ragged
    from vcr_net_b200 import functional as Fn

from oracle import synth
from oracle.ref_harness import default_args

DEV = "cuda:0"
K = 20


def _ragged_tokens(lengths, D, seed, token_major=True, fill=7.0):
    """Padded batch of random clouds + int32 lengths; padding is `fill` (results must not depend on it)."""
    g = torch.Generator().manual_seed(seed)
    B, N = len(lengths), max(lengths)
    x = torch.full((B, N, D), fill, dtype=torch.float32)
    alone = []
    for b, n in enumerate(lengths):
        c = torch.rand((n, D), generator=g) - 0.5
        x[b, :n] = c
        alone.append(c)
    x = x.to(DEV)
    alone = [(a if token_major else a.t()).contiguous().unsqueeze(0).to(DEV) for a in alone]
    if not token_major:
        x = x.transpose(1, 2).contiguous()
    return x, torch.tensor(lengths, dtype=torch.int32, device=DEV), alone


KNN_LENGTHS = [21, 64, 257, 700, 768, 1024, 2100, 8200]


@pytest.mark.parametrize("D,token_major", [(3, False), (3, True), (64, True), (64, False)])
@pytest.mark.parametrize("direct", [1, 0])
def test_knn_ragged_equals_each_cloud_alone(D, token_major, direct):
    x, n, alone = _ragged_tokens(KNN_LENGTHS, D, 11 + D, token_major)
    old = V.ops.lib().vcr_set_knn3_direct(direct)
    try:
        idx = ops.knn_topk_ragged(x, n, K, token_major=token_major)
        for b, a in enumerate(alone):
            m = KNN_LENGTHS[b]
            assert torch.equal(idx[b, :m], ops.knn_topk(a, K, token_major=token_major)[0]), (b, m)
            pad = torch.arange(m, x.shape[1] if token_major else x.shape[2], device=DEV, dtype=torch.int32)
            assert torch.equal(idx[b, m:], pad[:, None].expand(-1, K)), b
    finally:
        V.ops.lib().vcr_set_knn3_direct(old)


@pytest.mark.parametrize("tpq", [0, 1, 2])
def test_knn_tc_ragged_equals_each_cloud_alone(tpq):
    x, n, alone = _ragged_tokens(KNN_LENGTHS, 64, 5)
    old = ops.lib().vcr_set_knn_tc_tpq(tpq)
    try:
        idx = ops.knn_topk_tc_ragged(x, None, n, K)
        for b, a in enumerate(alone):
            m = KNN_LENGTHS[b]
            assert torch.equal(idx[b, :m], ops.knn_topk(a, K, token_major=True)[0]), (b, m)
            pad = torch.arange(m, x.shape[1], device=DEV, dtype=torch.int32)
            assert torch.equal(idx[b, m:], pad[:, None].expand(-1, K)), b
    finally:
        ops.lib().vcr_set_knn_tc_tpq(old)


def test_knn_ragged_padding_values_do_not_matter():
    x, n, _ = _ragged_tokens(KNN_LENGTHS, 64, 3)
    y = x.clone()
    for b, m in enumerate(KNN_LENGTHS):
        y[b, m:] = float("nan") if b % 2 else -1e4
    for fn in (lambda t: ops.knn_topk_ragged(t, n, K, token_major=True), lambda t: ops.knn_topk_tc_ragged(t, None, n, K)):
        assert torch.equal(fn(x), fn(y))


# (query length, key length) per item: multiples of 128 and not, Nq != Nk, a query tile wholly past an item's queries
ATTN_LENGTHS = [(128, 300), (21, 21), (700, 129), (1000, 1000), (257, 64), (64, 1024), (1024, 700)]


@pytest.mark.parametrize("mode", ["h3", "fp16", "bf16"])
def test_flash_attention_ragged_equals_each_item_alone(mode):
    H, dk, D = 4, 128, 512
    B = len(ATTN_LENGTHS)
    Nq, Nk = max(a for a, _ in ATTN_LENGTHS), max(b for _, b in ATTN_LENGTHS)
    g = torch.Generator().manual_seed(2)
    q = torch.randn((B * Nq, D), generator=g).to(DEV)
    k = torch.randn((B * Nk, D), generator=g).to(DEV)
    vt = torch.randn((B * D, Nk), generator=g).to(DEV)
    q_op, k_op, vt_op = ops.to_operand(q, mode), ops.to_operand(k, mode), ops.to_operand(vt, mode)
    nq = torch.tensor([a for a, _ in ATTN_LENGTHS], dtype=torch.int32, device=DEV)
    nk = torch.tensor([b for _, b in ATTN_LENGTHS], dtype=torch.int32, device=DEV)
    out = ops.Operand.empty(B * Nq, D, mode, DEV)
    out.buf.fill_(float("nan"))                                  # several items per CTA, into a dirty buffer
    scale = 1.0 / dk ** 0.5
    ops.flash_attn_tc_ragged(q_op, k_op, vt_op, out, B, H, Nq, Nk, dk, scale, nq, nk)
    for b, (mq, mk) in enumerate(ATTN_LENGTHS):
        vt_b = ops.Operand.empty(D, mk, mode, DEV)                # the item's V^T with exactly mk key columns
        vt_b.buf[:, :, :mk] = vt_op.buf[:, b * D:(b + 1) * D, :mk]
        o_b = ops.Operand.empty(mq, D, mode, DEV)
        ops.flash_attn_tc(q_op.rows_view(b * Nq, mq), k_op.rows_view(b * Nk, mk), vt_b, o_b, 1, H, mq, mk, dk, scale)
        got = out.buf[:, b * Nq:b * Nq + mq, :D]
        assert torch.equal(got, o_b.buf[:, :, :D]), (b, mq, mk)
        dead = (mq + 127) // 128 * 128                           # rows of query tiles past the item: zeros
        assert torch.equal(out.buf[:, b * Nq + dead:(b + 1) * Nq, :D],
                           torch.zeros_like(out.buf[:, b * Nq + dead:(b + 1) * Nq, :D])), b
        assert not torch.isnan(out.buf[:, b * Nq:(b + 1) * Nq, :D].float()).any(), b


def test_softcorr_and_svd_ragged_equal_each_pair_alone():
    lengths = [(128, 300), (21, 21), (700, 129), (1000, 1000), (257, 64), (64, 1024), (1024, 700)]
    B, D = len(lengths), 512
    Ns, Nt = max(a for a, _ in lengths), max(b for _, b in lengths)
    g = torch.Generator().manual_seed(4)
    s_tok = (torch.randn((B, Ns, D), generator=g) * 0.3).to(DEV)
    t_tok = (torch.randn((B, Nt, D), generator=g) * 0.3).to(DEV)
    tgt = torch.randn((B, 3, Nt), generator=g).to(DEV)
    src = torch.randn((B, 3, Ns), generator=g).to(DEV)
    ns = torch.tensor([a for a, _ in lengths], dtype=torch.int32, device=DEV)
    nt = torch.tensor([b for _, b in lengths], dtype=torch.int32, device=DEV)
    xx, yy = ops.sqnorm_rows(s_tok), ops.sqnorm_rows(t_tok)
    s_op, t_op = ops.to_operand(s_tok.view(B * Ns, D), "h3"), ops.to_operand(t_tok.view(B * Nt, D), "h3")
    corr = ops.softcorr_tc_ragged(s_op, t_op, xx, yy, tgt, B, Ns, Nt, D, ns, nt)
    R, t, Rb, tb = ops.svd_head_ragged(src, corr, ns)
    for b, (ms, mt) in enumerate(lengths):
        c_b = ops.softcorr_tc(s_op.rows_view(b * Ns, ms), t_op.rows_view(b * Nt, mt), xx[b:b + 1, :ms].contiguous(),
                              yy[b:b + 1, :mt].contiguous(), tgt[b:b + 1, :, :mt], 1, ms, mt, D)
        assert torch.equal(corr[b:b + 1, :, :ms], c_b), b
        assert torch.equal(corr[b, :, ms:], torch.zeros_like(corr[b, :, ms:])), b
        want = ops.svd_head(src[b:b + 1, :, :ms].contiguous(), c_b)
        for got, w in zip((R, t, Rb, tb), want):
            assert torch.equal(got[b:b + 1], w), b


# ------------------------------------------------------------------ end to end

SRC_LENGTHS = [21, 300, 768, 1000, 2100, 4097, 8200]
TGT_LENGTHS = [64, 300, 769, 1500, 2048, 3000, 8200]


@pytest.fixture(scope="module")
def pairs():
    p = synth.make_pairs(len(SRC_LENGTHS), max(SRC_LENGTHS), seed=77)
    src = [torch.from_numpy(p["src"][b, :, :n]).to(DEV) for b, n in enumerate(SRC_LENGTHS)]
    tgt = [torch.from_numpy(p["tgt"][b, :, :n]).to(DEV) for b, n in enumerate(TGT_LENGTHS)]
    return src, tgt


def _net(ckpt, **kw):
    net = V.VCRNet(default_args(**kw)).to(DEV).eval()
    net.load_state_dict(synth.checkpoint_to_torch(ckpt), strict=False)
    return net


def _check_against_alone(net, src_l, tgt_l, it):
    src, sl = ragged.pad_clouds(src_l)
    tgt, tl = ragged.pad_clouds(tgt_l)
    out = V.vcrnetIterRagged(net, src, tgt, sl, tl, iter=it)
    for b in range(len(src_l)):
        ms = src_l[b].shape[1]
        want = V.vcrnetIter(net, src_l[b][None], tgt_l[b][None], iter=it)
        for i, (o, w) in enumerate(zip(out, want)):
            o_b = o[b:b + 1, :, :ms] if i < 2 else o[b:b + 1]
            assert torch.equal(o_b, w), (b, i)
        assert torch.equal(out[1][b, :, ms:], torch.zeros_like(out[1][b, :, ms:]))
        assert torch.equal(out[0][b, :, ms:], torch.zeros_like(out[0][b, :, ms:]))
    return out


@pytest.mark.parametrize("mode,it,cycle", [("h3", 1, False), ("h3", 3, False), ("h3", 1, True), ("h3", 3, True),
                                           ("fp16", 1, True), ("fp16", 3, False), ("bf16", 1, False), ("bf16", 3, True)])
def test_vcrnet_iter_ragged_equals_each_pair_alone(ckpt, pairs, mode, it, cycle):
    old = config.precision
    config.set_precision(mode)
    try:
        _check_against_alone(_net(ckpt, cycle=cycle), *pairs, it)
    finally:
        config.set_precision(old)


def test_vcrnet_iter_ragged_identity_pointer(ckpt, pairs):
    src_l, tgt_l = pairs
    _check_against_alone(_net(ckpt, pointer="identity"), src_l[:4], tgt_l[:4], 2)


def test_vcrnet_iter_ragged_padding_independence(ckpt, pairs):
    net = _net(ckpt)
    src_l, tgt_l = pairs
    src, sl = ragged.pad_clouds(src_l)
    tgt, tl = ragged.pad_clouds(tgt_l)
    base = V.vcrnetIterRagged(net, src, tgt, sl, tl, iter=2)
    g = torch.Generator(device=DEV).manual_seed(9)
    s2, t2 = src.clone(), tgt.clone()
    for b in range(src.shape[0]):
        s2[b, :, SRC_LENGTHS[b]:] = (torch.rand(s2[b, :, SRC_LENGTHS[b]:].shape, generator=g, device=DEV) - 0.5) * 2e4
        t2[b, :, TGT_LENGTHS[b]:] = (torch.rand(t2[b, :, TGT_LENGTHS[b]:].shape, generator=g, device=DEV) - 0.5) * 2e4
    garbage = V.vcrnetIterRagged(net, s2, t2, sl, tl, iter=2)
    for a, c in zip(base, garbage):
        assert torch.equal(a, c)
    # another neighbour: pair 0 replaced by a different cloud, the other pairs keep their bits
    s3, t3 = src.clone(), tgt.clone()
    s3[0], t3[0] = tgt[1, :, :src.shape[2]] if tgt.shape[2] >= src.shape[2] else src[1], tgt[2]
    sl3 = sl.clone()
    sl3[0] = SRC_LENGTHS[1]
    other = V.vcrnetIterRagged(net, s3, t3, sl3, tl, iter=2)
    for a, c in zip(base, other):
        assert torch.equal(a[1:], c[1:])


def test_vcrnet_iter_ragged_graph_capture_and_side_stream(ckpt, pairs):
    net = _net(ckpt)
    src_l, tgt_l = pairs
    B, Ns, Nt = 5, 2200, 3100
    src, sl = ragged.pad_clouds(src_l[:5], n_max=Ns)
    tgt, tl = ragged.pad_clouds(tgt_l[:5], n_max=Nt)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = V.vcrnetIterRagged(net, src, tgt, sl, tl, iter=2)
    torch.cuda.current_stream().wait_stream(s)
    eager = V.vcrnetIterRagged(net, src, tgt, sl, tl, iter=2)
    for a, c in zip(side, eager):
        assert torch.equal(a, c)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = V.vcrnetIterRagged(net, src, tgt, sl, tl, iter=2)
    # new clouds and lengths written into the captured buffers
    new_s, new_t = [src_l[i] for i in (2, 0, 1, 3, 2)], [tgt_l[i] for i in (4, 1, 0, 2, 3)]
    ps, nsl = ragged.pad_clouds(new_s, n_max=Ns)
    pt, ntl = ragged.pad_clouds(new_t, n_max=Nt)
    src.copy_(ps); tgt.copy_(pt); sl.copy_(nsl); tl.copy_(ntl)
    graph.replay()
    want = V.vcrnetIterRagged(net, ps, pt, nsl, ntl, iter=2)
    for a, c in zip(static_out, want):
        assert torch.equal(a, c)


def test_ragged_errors(ckpt, pairs):
    src_l, tgt_l = pairs
    short = src_l[0][:, :20]
    with pytest.raises(ValueError):
        ragged.pad_clouds([src_l[1], short])
    with pytest.raises(ValueError):
        ragged.pad_clouds([src_l[1], src_l[2]], n_max=400)
    src, sl = ragged.pad_clouds(src_l[:3])
    tgt, tl = ragged.pad_clouds(tgt_l[:3])
    nets = {"partial": dict(partial=True), "dgcnn": dict(emb_nn="dgcnn"), "att": dict(vcp_nn="att")}
    for name, kw in nets.items():
        net = V.VCRNet(default_args(**kw)).to(DEV).eval()
        with pytest.raises(NotImplementedError, match={"partial": "partial", "dgcnn": "DGCNN", "att": "VcpAtt"}[name]):
            V.vcrnetIterRagged(net, src, tgt, sl, tl)
    net = _net(ckpt)
    with pytest.raises(NotImplementedError, match="DataParallel"):
        V.vcrnetIterRagged(torch.nn.DataParallel(net, device_ids=[0]), src, tgt, sl, tl)
    old = config.precision
    config.set_precision("fp32")
    try:
        with pytest.raises(NotImplementedError, match="fp32"):
            V.vcrnetIterRagged(net, src, tgt, sl, tl)
    finally:
        config.set_precision(old)
