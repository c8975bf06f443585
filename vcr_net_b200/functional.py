"""Host-side orchestration of the registration path over the CUDA ops (token-major internally).

Each function restates one reference function as a short sequence of kernel launches:
  lpdnet_tokens        model/lpdnet_model.py:103-137  (LPDNet.forward)
  encoder_decoder_tok  model/transformer.py:72-82,108-185 (EncoderDecoder/Encoder/Decoder layers)
  mha_tok              model/transformer.py:202-224
  vcp_whole/partial    model/vcrnet_model.py:173-347
All activations are [B, N, C] row-major ("tokens"); the reference's [B, C, N] appears only at the
module boundary (one transpose kernel in, one out).
"""
from __future__ import annotations

import math

import torch

from . import config, ops

_F32 = torch.float32


# --------------------------------------------------------------------------------------------------
# weight packing (cached on the module, invalidated by parameter version counters)
# --------------------------------------------------------------------------------------------------

def _versions(params):
    return tuple((p.data_ptr(), p._version) for p in params)


def packed(module, key, params, build):
    """Packed-weight cache on the module, keyed by (data_ptr, _version) of the source tensors.

    nn.DataParallel: ``replicate()`` shallow-copies ``__dict__`` on every forward, so the original's cache dict would be
    SHARED by the per-device replica threads and keyed by freshly broadcast weight copies whose addresses are recycled from
    call to call (a stale hit after an optimizer step).  Replicas therefore use a dict of their own, created on the replica
    (its ``__dict__`` is a private copy), which lives exactly as long as the replica: one forward."""
    d = module.__dict__
    cache = d.setdefault("_vcr_packed_replica", {}) if d.get("_is_replica", False) else d.setdefault("_vcr_packed", {})
    ver = _versions(params)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    with torch.no_grad():
        val = build()
    cache[key] = (ver, val)
    return val


def _split_edge_weight(conv):
    """Conv2d(2C -> Co, 1x1) acting on [f_j ; x_i] (util/util.py:197)  ->  stacked [2Co, C] weight
    producing [P | Q] with P = W_a f (no bias), Q = W_b f + bias."""
    w = conv.weight.detach().reshape(conv.weight.shape[0], -1)
    co, c2 = w.shape
    c = c2 // 2
    wa, wb = w[:, :c], w[:, c:]
    stacked = torch.cat([wa, wb], dim=0).contiguous()
    bias = torch.cat([torch.zeros_like(conv.bias.detach()), conv.bias.detach()]).contiguous()
    return stacked, bias


def lpdnet_weights(m):
    convs = [m.conv1_lpd, m.conv2_lpd, m.conv3_lpd, m.convDG1[0], m.convDG2[0], m.convSN1[0]]
    params = [p for c in convs for p in (c.weight, c.bias)]

    def build():
        dg1_w, dg1_b = _split_edge_weight(m.convDG1[0])
        sn1_w, sn1_b = _split_edge_weight(m.convSN1[0])
        return {
            "w1": m.conv1_lpd.weight.detach().reshape(m.conv1_lpd.weight.shape[0], 3).contiguous(),
            "b1": m.conv1_lpd.bias.detach().contiguous(),
            "w2": m.conv2_lpd.weight.detach().reshape(64, 64).contiguous(),
            "b2": m.conv2_lpd.bias.detach().contiguous(),
            "dg1_w": dg1_w, "dg1_b": dg1_b,
            "dg2_w": m.convDG2[0].weight.detach().reshape(128, 128).contiguous(),
            "dg2_b": m.convDG2[0].bias.detach().contiguous(),
            "sn1_w": sn1_w, "sn1_b": sn1_b,
            "w3": m.conv3_lpd.weight.detach().reshape(m.conv3_lpd.weight.shape[0], 512).contiguous(),
            "b3": m.conv3_lpd.bias.detach().contiguous(),
        }

    return packed(m, "lpdnet", params, build)


def lpdnet_tokens(m, xyz: torch.Tensor, idx_feat=None, idx_xyz=None, stages=None, out=None):
    """xyz [B,3,N] -> embedding tokens [B,N,emb_dims]  (model/lpdnet_model.py:103-137, incl. the optional t3d / tfea
    TranformNets, eval mode).

    idx_feat / idx_xyz (int32 [B,N,20]) inject neighbour sets, as get_graph_feature(x, idx=...) allows."""
    W = lpdnet_weights(m)
    slope = float(m.negative_slope)
    k = m.k
    B, _, N = xyz.shape
    xyz = xyz.contiguous()
    xyz_in = xyz
    if m.t3d:                                                                # :107-109  x <- (x^T trans)^T = trans^T x
        trans = transform_net_matrix(m.t_net3d, xyz)
        xyz_in = ops.rigid_apply(xyz, trans.transpose(1, 2).contiguous(),
                                 torch.zeros((B, 3), dtype=_F32, device=xyz.device))
    tc = config.precision != "fp32"
    fused_ops = tc and not m.tfea            # producers write the "h3" operand copies their consumers read (no to_operand passes)
    if fused_ops and W["w1"].shape[0] == 64:
        h1, h2, h2_op = ops.lpd_point_mlp(xyz_in, W["w1"], W["b1"], W["w2"], W["b2"], slope,
                                          want_h1=stages is not None, want_operand=True)      # :111-112
    else:
        h1 = ops.conv3_act(xyz_in, W["w1"], W["b1"], slope)                  # :111
        h2 = ops.gemm(h1, W["w2"], W["b2"], act=1, slope=slope)              # :112  [B,N,64]
        if m.tfea:                                                           # :114-118  per-cloud [N,64] x [64,64]
            trans_feat = transform_net_matrix(m.t_net_fea, h2)
            h2t = torch.empty_like(h2)
            ops.bgemm(h2, 64, N * 64, 0, trans_feat, 64, 64 * 64, 0, 1, h2t, 64, N * 64, 0, N, 64, 64, B, 1)
            h2 = h2t
        h2_op = ops.to_operand(h2.view(B * N, 64), "h3") if tc else None     # shared by the kNN prefilter and the DG1 GEMM
    if idx_feat is None:                                                     # :122 (feature-space kNN)
        if config.use_knn_tc(N) and ops.knn_tc_supported(64, k):
            idx_feat = ops.knn_topk_tc(h2, h2_op, k)
        else:
            idx_feat = ops.knn_topk(h2, k, token_major=True)
    if tc:     # K = 64 / 128 products are output-bandwidth bound: 3-term split on tensor cores in every TC mode
        wpq = packed(m, "pq_h3", [m.convDG1[0].weight, m.convSN1[0].weight],
                     lambda: (ops.to_operand(W["dg1_w"], "h3"), ops.to_operand(W["sn1_w"], "h3")))
        pq1 = torch.empty((B, N, 256), dtype=_F32, device=xyz.device)
        ops.gemm_tc(h2_op, wpq[0], B * N, 256, 64, bias=W["dg1_b"], c=pq1)
    else:
        pq1 = ops.gemm(h2, W["dg1_w"], W["dg1_b"])                           # [B,N,256] = [P|Q]
    cat = torch.empty((B, N, 512), dtype=_F32, device=xyz.device)
    mode = config.precision
    # the conv3 GEMM's A operand [x1 | x2 | x3]: in the parity mode each producer writes its slice in operand format
    cat_op = ops.Operand.empty(B * N, 512, "h3", xyz.device) if mode == "h3" else None
    if config.precision == "fp32":
        ops.edgeconv_dg(pq1, idx_feat, W["dg2_w"], W["dg2_b"], slope, cat[:, :, 0:128], cat[:, :, 128:256])  # :123-126
    else:
        ops.edgeconv_dg_tc(pq1, idx_feat, W["dg2_w"], W["dg2_b"], slope, cat[:, :, 0:128], cat[:, :, 128:256],
                           config.precision, op1=cat_op.cols_view(0, 128) if cat_op is not None else None,
                           op2=cat_op.cols_view(128, 128) if cat_op is not None else None)
    if idx_xyz is None:
        idx_xyz = ops.knn_topk(xyz, k, token_major=False)                    # :129 (3-d kNN)
    if tc:
        pq3 = torch.empty((B, N, 512), dtype=_F32, device=xyz.device)
        x2_op = cat_op.cols_view(128, 128) if cat_op is not None else ops.to_operand(cat[:, :, 128:256], "h3")
        ops.gemm_tc(x2_op, wpq[1], B * N, 512, 128, bias=W["sn1_b"], c=pq3)
    else:
        pq3 = ops.gemm(cat[:, :, 128:256], W["sn1_w"], W["sn1_b"])           # [B,N,512] = [P3|Q3]
    ops.gather_max(pq3[:, :, 0:256], pq3[:, :, 256:512], idx_xyz, slope, cat[:, :, 256:512],
                   op=cat_op.cols_view(256, 256) if cat_op is not None else None)               # :130-132
    if mode == "fp32":
        emb = ops.gemm(cat, W["w3"], W["b3"], act=1, slope=slope, out=out)   # :134-135
    else:
        w3 = packed(m, "w3_" + mode, [m.conv3_lpd.weight], lambda: ops.to_operand(W["w3"], mode))
        emb = out if out is not None else torch.empty((B, N, W["w3"].shape[0]), dtype=_F32, device=xyz.device)
        ops.gemm_tc(cat_op if cat_op is not None else ops.to_operand(cat, mode), w3, B * N, W["w3"].shape[0], 512,
                    bias=W["b3"], act=1, slope=slope, c=emb)
    if stages is not None:
        stages.update(f64=h2, idx_feat=idx_feat, idx_xyz=idx_xyz, cat=cat, h1=h1, pq1=pq1, pq3=pq3)
        if m.t3d:
            stages.update(trans=trans)
        if m.tfea:
            stages.update(trans_feat=trans_feat)
    return emb


# --------------------------------------------------------------------------------------------------
# TranformNet (model/lpdnet_model.py:19-70): the --t3d / --tfea input / feature alignment matrices
# --------------------------------------------------------------------------------------------------

def _fold_bn_bias(layer, bn):
    """Eval-mode BatchNorm1d folded into the biased conv / linear in front of it."""
    w = layer.weight.detach().reshape(layer.weight.shape[0], -1)
    s = bn.weight.detach() / torch.sqrt(bn.running_var.detach() + bn.eps)
    return (w * s[:, None]).contiguous(), ((layer.bias.detach() - bn.running_mean.detach()) * s + bn.bias.detach()).contiguous()


def cloud_max(h: torch.Tensor, B: int, N: int):
    """h [B*N, C] -> [B, C]: max over the points of each cloud (torch.max(x, 2), :57), as a tree of vcr_edge_max passes
    (<= 32 rows per thread and pass) so a 1024-point cloud is not reduced by one serial loop."""
    C = h.shape[1]
    n = N
    while n > 1:
        k = next((d for d in range(min(32, n), 1, -1) if n % d == 0), n)
        out = torch.empty((B * (n // k), C), dtype=_F32, device=h.device)
        ops.edge_max(h, k, out)
        h, n = out, n // k
    return h


def transform_net_matrix(tn, x: torch.Tensor):
    """TranformNet.forward.  x = xyz [B,3,N] (k = 3) or feature tokens [B,N,64] (k = 64)  ->  [B,k,k].
    conv1-3 + BN + ReLU per point (GEMMs), max over the cloud, fc1-2 + BN + ReLU, fc3 + identity."""
    _require_eval(tn)
    mode = config.precision
    k = tn.k
    layers = [(tn.conv1, tn.bn1), (tn.conv2, tn.bn2), (tn.conv3, tn.bn3), (tn.fc1, tn.bn4), (tn.fc2, tn.bn5)]
    params = [p for l, bn in layers for p in (l.weight, l.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var)]
    W = packed(tn, "tnet", params, lambda: [_fold_bn_bias(l, bn) for l, bn in layers])
    if k == 3:
        B, _, N = x.shape
        h = ops.conv3_act(x.contiguous(), W[0][0], W[0][1], 0.0).view(B * N, 64)          # :54
    else:
        B, N, _ = x.shape
        h = ops.gemm(x.reshape(B * N, k), W[0][0], W[0][1], act=1, slope=0.0)
    h, hop = _edge_mlp(h, *W[1], mode, True)                                              # :55  [B*N,128]
    h, _ = _edge_mlp(hop if hop is not None else h, *W[2], mode, False)                   # :56  [B*N,1024]
    g = cloud_max(h, B, N)                                                                # :57-58 [B,1024]
    g = ops.gemm(g, W[3][0], W[3][1], act=1, slope=0.0)                                   # :60
    g = ops.gemm(g, W[4][0], W[4][1], act=1, slope=0.0)                                   # :61
    iden = torch.eye(k, dtype=_F32, device=g.device).reshape(1, k * k).repeat(B, 1)      # :64-66
    w3 = tn.fc3.weight.detach().contiguous()
    out = ops.gemm(g, w3, tn.fc3.bias.detach().contiguous(), residual=iden)               # :62, :68
    return out.view(B, k, k)


def lpdnet_dg2_edges(m, pq1, idx_feat):
    """What LPDNetTrainFn.backward recomputes for convDG1 / convDG2 (:123-126): e1 = act(P1[nbr] + Q1) and the
    convDG2 pre-activations z2 = e1 W2^T + b2, both [B*N*k, 128].  The backward routes the gradient of
    x2 = act(max_k z2) to the arg-max edge of these z2, so they come from the forward's own arithmetic: the SIMT GEMM
    sums in the order of vcr_edgeconv_dg, and in the tensor-core modes vcr_edgeconv_dg_tc writes them itself."""
    W = lpdnet_weights(m)
    slope = float(m.negative_slope)
    e1 = ops.edge_gather_act(pq1, idx_feat, slope)
    if config.precision == "fp32":
        return e1, ops.gemm(e1, W["dg2_w"], W["dg2_b"])
    B, N, _ = pq1.shape
    z2 = torch.empty_like(e1)
    x12 = torch.empty((B, N, 256), dtype=_F32, device=pq1.device)             # x1, x2 again: not needed here
    ops.edgeconv_dg_tc(pq1, idx_feat, W["dg2_w"], W["dg2_b"], slope, x12[:, :, 0:128], x12[:, :, 128:256],
                       config.precision, z=z2)
    return e1, z2


class LPDNetTrainFn(torch.autograd.Function):
    """LPDNet.forward with a hand-written backward (BASELINE config 3; the reference differentiates
    model/lpdnet_model.py:103-137 with autograd).  Forward = lpdnet_tokens; backward = csrc/train.cu kernels +
    data-gradient products (vcr_gemm_f32, or the 3-term tcgen05 GEMM on a power-of-two scaled g_emb in TC modes).
    Gradients flow to the 12 parameters only (the input cloud and the kNN indices carry none, as in the reference)."""

    @staticmethod
    def forward(ctx, m, xyz, idx_feat, idx_xyz, *params):
        st = {}
        with torch.no_grad():
            emb = lpdnet_tokens(m, xyz, idx_feat=idx_feat, idx_xyz=idx_xyz, stages=st)
            xyz_t = ops.transpose_batched(xyz.contiguous())                  # [B,N,3]
        ctx.m = m
        ctx.st = st
        ctx.save_for_backward(xyz_t, emb)          # outputs are allowed here; no output -> grad_fn -> ctx -> output cycle
        return emb

    @staticmethod
    def backward(ctx, g_emb):
        m, st = ctx.m, ctx.st
        xyz_t, emb = ctx.saved_tensors
        W = lpdnet_weights(m)
        slope = float(m.negative_slope)
        k = m.k
        h1, h2, pq1, cat, pq3 = st["h1"], st["f64"], st["pq1"], st["cat"], st["pq3"]
        idx_f, idx_x = st["idx_feat"], st["idx_xyz"]
        B, N, _ = emb.shape
        T = B * N
        g_emb = g_emb.contiguous()
        tc = config.precision != "fp32"

        def dgrad(g, w):
            """g [M,Nout] @ w[Nout,Nin]: data gradient of y = x w^T.  SIMT fp32, or the 3-term tcgen05 GEMM
            (fp32-equivalent inside fp16's normal range) in TC modes."""
            if not tc:
                return ops.gemm(g, w, b_layout=1)
            wt = w.t().contiguous()
            if g.shape[-1] % 8 or wt.shape[0] % 4:
                return ops.gemm(g, wt)
            M, K = g.shape
            out = torch.empty((M, wt.shape[0]), dtype=_F32, device=g.device)
            ops.gemm_tc(ops.to_operand(g, "h3"), ops.to_operand(wt, "h3"), M, wt.shape[0], K, c=out)
            return out

        # The LPD loss is a mean over B*32 anchors and B*N points: at 16 x 1024 points its gradients are ~1e-7, where
        # the "h3" split's hi = fp16(x) is subnormal (tests/test_gpu_train_range.py).  The tensor-core modes therefore
        # run the backward on g_emb * 2^-floor(log2 max|g_emb|), a power of two picked on the device (no host sync).
        # Every step from g_emb to the parameter gradients is linear in g_emb (the activation derivatives and arg-max
        # routes come from forward values), so multiplying the results by the inverse power of two is exact.
        bits = ops.absmax_bits(g_emb) if tc else None

        # conv3_lpd (:134-135)
        g_z3 = ops.act_bwd(g_emb.view(T, -1), emb.view(T, -1), slope, scale_bits=bits)
        gW3, gb3 = ops.wgrad(g_z3, cat.view(T, 512))
        g_cat = dgrad(g_z3, W["w3"]).view(B, N, 512)
        # convSN1 + max (:130-132)
        g_pq3 = torch.zeros((B, N, 512), dtype=_F32, device=emb.device)
        ops.gather_max_bwd(pq3[:, :, 0:256], pq3[:, :, 256:512], idx_x, slope, g_cat[:, :, 256:512],
                           g_pq3[:, :, 0:256], g_pq3[:, :, 256:512])
        gWsn, gbsn = ops.wgrad(g_pq3.view(T, 512), cat[:, :, 128:256])
        g_x2 = (dgrad(g_pq3.view(T, 512), W["sn1_w"]) + g_cat[:, :, 128:256].reshape(T, 128)).view(B, N, 128)
        # convDG2 + max (:125-126), convDG1 + max (:123-124)
        e1, z2 = lpdnet_dg2_edges(m, pq1, idx_f)                               # [T*k,128] each
        ops.edge_max_bwd_(z2, g_x2, k, slope)                                  # z2 <- g_z2
        gWdg2, gbdg2 = ops.wgrad(z2, e1)
        g_e1 = dgrad(z2, W["dg2_w"])
        g_pq1 = ops.edge_bwd_scatter(e1, g_e1, g_cat[:, :, 0:128], idx_f, slope)
        del e1, z2, g_e1
        gWdg1, gbdg1 = ops.wgrad(g_pq1.view(T, 256), h2.view(T, 64))
        g_h2 = dgrad(g_pq1.view(T, 256), W["dg1_w"])
        # conv2_lpd, conv1_lpd (:111-112)
        g_z2 = ops.act_bwd(g_h2, h2.view(T, 64), slope)
        gW2, gb2 = ops.wgrad(g_z2, h1.view(T, 64))
        g_h1 = dgrad(g_z2, W["w2"])
        g_z1 = ops.act_bwd(g_h1, h1.view(T, 64), slope)
        gW1, gb1 = ops.wgrad(g_z1, xyz_t.view(T, 3))

        def unsplit(gw, gb, conv):
            co = conv.weight.shape[0]
            return (torch.cat([gw[:co], gw[co:]], dim=1).reshape(conv.weight.shape), gb[co:].clone())

        gdg1_w, gdg1_b = unsplit(gWdg1, gbdg1, m.convDG1[0])
        gsn_w, gsn_b = unsplit(gWsn, gbsn, m.convSN1[0])
        grads = {
            "conv1_lpd.weight": gW1.reshape(m.conv1_lpd.weight.shape), "conv1_lpd.bias": gb1,
            "conv2_lpd.weight": gW2.reshape(m.conv2_lpd.weight.shape), "conv2_lpd.bias": gb2,
            "conv3_lpd.weight": gW3.reshape(m.conv3_lpd.weight.shape), "conv3_lpd.bias": gb3,
            "convDG1.0.weight": gdg1_w, "convDG1.0.bias": gdg1_b,
            "convDG2.0.weight": gWdg2.reshape(m.convDG2[0].weight.shape), "convDG2.0.bias": gbdg2,
            "convSN1.0.weight": gsn_w, "convSN1.0.bias": gsn_b,
        }
        if tc:
            inv = ops.pow2_inverse(bits)
            for g in grads.values():
                g.mul_(inv)
        ctx.st = None
        return (None, None, None, None) + tuple(grads[n] for n in LPDNET_PARAM_ORDER)


LPDNET_PARAM_ORDER = ("conv1_lpd.weight", "conv1_lpd.bias", "conv2_lpd.weight", "conv2_lpd.bias",
                      "conv3_lpd.weight", "conv3_lpd.bias", "convDG1.0.weight", "convDG1.0.bias",
                      "convDG2.0.weight", "convDG2.0.bias", "convSN1.0.weight", "convSN1.0.bias")


def lpdnet_param_tensors(m):
    """The 12 trainable tensors in LPDNET_PARAM_ORDER, read from the conv ATTRIBUTES: inside an nn.DataParallel replica
    ``parameters()`` / ``named_parameters()`` are empty (the broadcast copies are plain attributes, torch replicate())."""
    out = []
    for name in LPDNET_PARAM_ORDER:
        obj = m
        for part in name.split("."):
            obj = obj[int(part)] if part.isdigit() else getattr(obj, part)
        out.append(obj)
    return out


def lpdnet_tokens_train(m, xyz, idx_feat=None, idx_xyz=None):
    """Differentiable lpdnet_tokens (w.r.t. the module's parameters)."""
    return LPDNetTrainFn.apply(m, xyz, idx_feat, idx_xyz, *lpdnet_param_tensors(m))


# --------------------------------------------------------------------------------------------------
# DGCNN / PointNet embeddings (--emb_nn dgcnn | pointnet; model/vcrnet_model.py:66-123)
# --------------------------------------------------------------------------------------------------

def _fold_bn(conv, bn):
    """Eval-mode BatchNorm folded into the bias-free 1x1 conv in front of it: y = (W x - mean) * g / sqrt(var + eps) + b."""
    w = conv.weight.detach().reshape(conv.weight.shape[0], -1)
    s = bn.weight.detach() / torch.sqrt(bn.running_var.detach() + bn.eps)
    return (w * s[:, None]).contiguous(), (bn.bias.detach() - bn.running_mean.detach() * s).contiguous()


def _bn_params(m, n):
    ps = []
    for i in range(1, n + 1):
        bn = getattr(m, f"bn{i}")
        ps += [getattr(m, f"conv{i}").weight, bn.weight, bn.bias, bn.running_mean, bn.running_var]
    return ps


def _require_eval(m):
    if m.training:
        raise RuntimeError(f"{type(m).__name__}: only eval() mode (running BatchNorm statistics folded into the convs) is "
                           "implemented on the B200 path; call .eval() as the reference's test loop does")


def _edge_mlp(e_prev, w, b, mode, want_operand):
    """One per-edge 1x1 conv + folded BN + ReLU over a materialised [T*k, Cin] edge tensor."""
    if mode == "fp32":
        return ops.gemm(e_prev, w, b, act=1, slope=0.0), None
    rows = e_prev.rows if isinstance(e_prev, ops.Operand) else e_prev.shape[0]
    a = e_prev if isinstance(e_prev, ops.Operand) else ops.to_operand(e_prev, mode)
    co, ci = w.shape
    out = torch.empty((rows, co), dtype=_F32, device=w.device)
    h = ops.Operand.empty(rows, co, mode, w.device) if want_operand else None
    ops.gemm_tc(a, ops.to_operand(w, mode), rows, co, ci, bias=b, act=1, slope=0.0, c=out,
                **({"h": h, "h_split": co} if want_operand else {}))
    return out, h


def dgcnn_tokens(m, xyz: torch.Tensor, idx=None, stages=None):
    """DGCNN.forward (model/vcrnet_model.py:105-123): xyz [B,3,N] -> tokens [B,N,emb_dims].
    conv1 acts on the raw concat [x_j ; x_i] (util/util.py:197) so it splits into per-point products P + Q like the
    LPDNet EdgeConvs; conv2..4 are per-edge GEMMs over [T*k, C]; every max over k is vcr_edge_max."""
    _require_eval(m)
    mode = config.precision
    k = 20
    B, _, N = xyz.shape
    xyz = xyz.contiguous()

    def build():
        w1, b1 = _fold_bn(m.conv1, m.bn1)                                   # [64,6]
        stacked = torch.cat([w1[:, :3], w1[:, 3:]], dim=0).contiguous()     # [P | Q] rows
        bias = torch.cat([torch.zeros_like(b1), b1]).contiguous()
        return {"w1": stacked, "b1": bias, **{f"w{i}": _fold_bn(getattr(m, f"conv{i}"), getattr(m, f"bn{i}"))
                                              for i in (2, 3, 4, 5)}}

    W = packed(m, "dgcnn", _bn_params(m, 5), build)
    if idx is None:
        idx = ops.knn_topk(xyz, k, token_major=False)                       # get_graph_feature(x) -> knn(x, 20)
    pq1 = ops.conv3_act(xyz, W["w1"], W["b1"], 1.0)                          # slope 1 = identity: [B,N,128] = [P|Q]
    cat = torch.empty((B, N, 512), dtype=_F32, device=xyz.device)
    e = ops.edge_gather_act(pq1, idx, 0.0)                                   # relu(bn1(conv1(edge)))  [T*k,64]
    ops.edge_max(e, k, cat[:, :, 0:64])                                      # x1
    e, eop = _edge_mlp(e, *W["w2"], mode, True)
    ops.edge_max(e, k, cat[:, :, 64:128])                                    # x2
    e, eop = _edge_mlp(eop if eop is not None else e, *W["w3"], mode, True)
    ops.edge_max(e, k, cat[:, :, 128:256])                                   # x3
    e, _ = _edge_mlp(eop if eop is not None else e, *W["w4"], mode, False)
    ops.edge_max(e, k, cat[:, :, 256:512])                                   # x4
    emb, _ = _edge_mlp(cat.view(B * N, 512), *W["w5"], mode, False)          # relu(bn5(conv5(cat)))
    if stages is not None:
        stages.update(idx=idx, cat=cat)
    return emb.view(B, N, -1)


def pointnet_tokens(m, xyz: torch.Tensor):
    """PointNet.forward (model/vcrnet_model.py:82-88): five per-point conv + BN + ReLU layers."""
    _require_eval(m)
    mode = config.precision
    B, _, N = xyz.shape
    W = packed(m, "pointnet", _bn_params(m, 5),
               lambda: {f"w{i}": _fold_bn(getattr(m, f"conv{i}"), getattr(m, f"bn{i}")) for i in range(1, 6)})
    h = ops.conv3_act(xyz.contiguous(), W["w1"][0], W["w1"][1], 0.0).view(B * N, -1)
    hop = None
    for i in (2, 3, 4, 5):
        h, hop = _edge_mlp(hop if hop is not None else h, *W[f"w{i}"], mode, i < 5)
    return h.view(B, N, -1)


# --------------------------------------------------------------------------------------------------
# Transformer
# --------------------------------------------------------------------------------------------------

def mha_weights(m):
    params = [p for l in m.linears for p in (l.weight, l.bias)]

    def build():
        w = [l.weight.detach() for l in m.linears]
        b = [l.bias.detach() for l in m.linears]
        return {
            "wqkv": torch.cat(w[0:3], dim=0).contiguous(), "bqkv": torch.cat(b[0:3]).contiguous(),
            "wq": w[0].contiguous(), "bq": b[0].contiguous(),
            "wkv": torch.cat(w[1:3], dim=0).contiguous(), "bkv": torch.cat(b[1:3]).contiguous(),
            "wo": w[3].contiguous(), "bo": b[3].contiguous(),
        }

    return packed(m, "mha", params, build)


def mha_tok(m, xq: torch.Tensor, xkv: torch.Tensor | None, residual=None, want_attn=False):
    """MultiHeadedAttention.forward on tokens (model/transformer.py:202-224).

    xq [B,Nq,D]; xkv None => self-attention (query=key=value=xq, one fused QKV GEMM), else
    key=value=xkv.  Returns linears[3](attn) (+ residual fused into the GEMM epilogue)."""
    W = mha_weights(m)
    B, Nq, D = xq.shape
    h, dk = m.h, m.d_k
    dev = xq.device
    if xkv is None:
        qkv = ops.gemm(xq, W["wqkv"], W["bqkv"])                  # [B,Nq,3D]
        Nk = Nq
        q = (qkv, 3 * D, Nq * 3 * D, dk)
        kk = (qkv[:, :, D:], 3 * D, Nq * 3 * D, dk)
        vv = (qkv[:, :, 2 * D:], 3 * D, Nq * 3 * D, dk)
    else:
        Nk = xkv.shape[1]
        qb = ops.gemm(xq, W["wq"], W["bq"])                       # [B,Nq,D]
        kvb = ops.gemm(xkv, W["wkv"], W["bkv"])                   # [B,Nk,2D]
        q = (qb, D, Nq * D, dk)
        kk = (kvb, 2 * D, Nk * 2 * D, dk)
        vv = (kvb[:, :, D:], 2 * D, Nk * 2 * D, dk)
    att = torch.empty((B, Nq, D), dtype=_F32, device=dev)
    out = (att, D, Nq * D, dk)
    scale = 1.0 / math.sqrt(dk)
    if m.is_src:
        # partial overlap: pass 1 gets the column sums, top-int(Nk*overlap2) keys survive (:35-53)
        csum = ops.attention_f32(q, kk, vv, B, h, Nq, Nk, dk, scale, out, keep=None, colsum_out=True)
        keep_n = int(Nk * m.overlap2)
        _, keep = ops.topk_select(csum, keep_n, want_idx=False, want_mask=True)
        ops.attention_f32(q, kk, vv, B, h, Nq, Nk, dk, scale, out, keep=keep)
    else:
        ops.attention_f32(q, kk, vv, B, h, Nq, Nk, dk, scale, out)
    return ops.gemm(att, W["wo"], W["bo"], residual=residual)


def ffn_tok(m, x: torch.Tensor, residual=None):
    """PositionwiseFeedForward.forward (model/transformer.py:237-238): w_2(relu(w_1 x))."""
    hdn = ops.gemm(x, m.w_1.weight, m.w_1.bias, act=1, slope=0.0)
    return ops.gemm(hdn, m.w_2.weight, m.w_2.bias, residual=residual)


def _ln(norm, x, residual=None):
    return ops.layernorm(x, norm.a_2, norm.b_2, norm.eps, residual=residual)


def encoder_decoder_tok(model, src: torch.Tensor, tgt: torch.Tensor, final_residual=None):
    """decode(encode(src), tgt) on tokens (model/transformer.py:72-82).  Pre-LN residual blocks:
    x + sublayer(norm(x)) (:147-153); the residual add rides in the epilogue of the last GEMM of
    each sublayer.  ``final_residual`` is added to the decoder's final LayerNorm output (the
    `emb + emb_p` of model/vcrnet_model.py:504-505)."""
    if config.precision != "fp32":
        return encoder_decoder_tc(model, src.contiguous(), tgt.contiguous(), final_residual, config.precision)
    x = src
    for layer in model.encoder.layers:
        n = _ln(layer.sublayer[0].norm, x)
        x = mha_tok(layer.self_attn, n, None, residual=x)
        n = _ln(layer.sublayer[1].norm, x)
        x = ffn_tok(layer.feed_forward, n, residual=x)
    mem = _ln(model.encoder.norm, x)
    y = tgt
    for layer in model.decoder.layers:
        n = _ln(layer.sublayer[0].norm, y)
        y = mha_tok(layer.self_attn, n, None, residual=y)
        n = _ln(layer.sublayer[1].norm, y)
        y = mha_tok(layer.src_attn, n, mem, residual=y)
        n = _ln(layer.sublayer[2].norm, y)
        y = ffn_tok(layer.feed_forward, n, residual=y)
    return _ln(model.decoder.norm, y, residual=final_residual)


# --------------------------------------------------------------------------------------------------
# Transformer on tensor cores (operand-format chaining, see csrc/gemm_tc.cu)
# --------------------------------------------------------------------------------------------------

def mha_weights_tc(m, mode):
    W = mha_weights(m)
    params = [p for l in m.linears for p in (l.weight, l.bias)]
    return packed(m, "mha_" + mode, params, lambda: {
        "wqkv": ops.to_operand(W["wqkv"], mode), "wq": ops.to_operand(W["wq"], mode),
        "wkv": ops.to_operand(W["wkv"], mode), "wo": ops.to_operand(W["wo"], mode)})


def mha_project_self(m, x_op, B, N, mode, dev, qk=None, vt=None):
    """Self-attention projections: one fused QKV GEMM writing Q | K row-major and V TRANSPOSED per head, all in operand
    format, straight from the epilogue.  qk / vt: optional destination views (rows of a larger buffer)."""
    W, Wt = mha_weights(m), mha_weights_tc(m, mode)
    D = m.h * m.d_k
    if qk is None:
        qk = ops.Operand.empty(B * N, 2 * D, mode, dev)
    if vt is None:
        vt = ops.Operand.empty(B * D, N, mode, dev)                      # rows (b, head*dk + d), cols = keys
    ops.gemm_tc(x_op, Wt["wqkv"], N, 3 * D, D, nbo=B, a_off=(N, 0, 0, 0), bias=W["bqkv"],
                h=qk, h_strides=(N * qk.ld, 0), h_split=2 * D, ht=vt, ht_strides=(D * vt.ld, 0))
    return qk.cols_view(0, D), qk.cols_view(D, D), vt


def mha_project_q(m, xq_op, rows, mode, dev, out=None):
    W, Wt = mha_weights(m), mha_weights_tc(m, mode)
    D = m.h * m.d_k
    q_v = out if out is not None else ops.Operand.empty(rows, D, mode, dev)
    ops.gemm_tc(xq_op, Wt["wq"], rows, D, D, bias=W["bq"], h=q_v, h_split=D)
    return q_v


def mha_project_kv(m, xkv_op, B, Nk, mode, dev, k_out=None, vt_out=None):
    W, Wt = mha_weights(m), mha_weights_tc(m, mode)
    D = m.h * m.d_k
    k_v = k_out if k_out is not None else ops.Operand.empty(B * Nk, D, mode, dev)
    vt = vt_out if vt_out is not None else ops.Operand.empty(B * D, Nk, mode, dev)
    ops.gemm_tc(xkv_op, Wt["wkv"], Nk, 2 * D, D, nbo=B, a_off=(Nk, 0, 0, 0), bias=W["bkv"],
                h=k_v, h_strides=(Nk * k_v.ld, 0), h_split=D, ht=vt, ht_strides=(D * vt.ld, 0))
    return k_v, vt


def mha_attention(m, q_v, k_v, vt, B, Nq, Nk, mode, dev, max_ws_bytes=3 << 30):
    """softmax(QK^T/sqrt(d_k)) V (+ the partial-overlap key selection, model/transformer.py:29-55) with the heads merged:
    -> operand-format [B*Nq, D].  q_v / k_v / vt: operand-format projections of B batch items."""
    D, h, dk = m.h * m.d_k, m.h, m.d_k
    scale = 1.0 / math.sqrt(dk)
    att = ops.Operand.empty(B * Nq, D, mode, dev)
    keep = None
    if m.is_src:
        # partial overlap (:35-53): column sums of the unmasked probabilities pick the surviving keys.
        if dk == 128 and mode == "h3" and config.fused_key_stat:
            # two tcgen05 sweeps per (batch, head, query tile): no score matrix in HBM (csrc/attn_colsum_tc.cu)
            csum = ops.attn_colsum_tc(q_v, k_v, B, h, Nq, Nk, dk, scale)
        else:
            ldS = (Nk + 3) // 4 * 4
            cb = max(1, min(B, min(max_ws_bytes, config.stat_chunk_bytes) // (h * Nq * ldS * 4)))
            S = torch.empty((cb, h, Nq, ldS), dtype=_F32, device=dev)
            csum = torch.empty((B, Nk), dtype=_F32, device=dev)
            for b0 in range(0, B, cb):
                nb = min(cb, B - b0)
                ops.gemm_tc(q_v.rows_view(b0 * Nq, nb * Nq), k_v.rows_view(b0 * Nk, nb * Nk), Nq, Nk, dk, nbo=nb, nbi=h,
                            a_off=(Nq, 0, 0, dk), b_off=(Nk, 0, 0, dk), alpha=scale, c=S,
                            c_strides=(h * Nq * ldS, Nq * ldS))
                csum[b0:b0 + nb] = ops.colsum_softmax(S[:nb].view(nb * h * Nq, ldS), Nk, nb)
        _, keep = ops.topk_select(csum, int(Nk * m.overlap2), want_idx=False, want_mask=True)
    if dk == 128 and config.flash_attention:
        ops.flash_attn_tc(q_v, k_v, vt, att, B, h, Nq, Nk, dk, scale, keep=keep)
    else:
        ldS = (Nk + 3) // 4 * 4
        cb = max(1, min(B, max_ws_bytes // (h * Nq * ldS * 4 * 2)))
        S = torch.empty((cb, h, Nq, ldS), dtype=_F32, device=dev)
        for b0 in range(0, B, cb):
            nb = min(cb, B - b0)
            ops.gemm_tc(q_v.rows_view(b0 * Nq, nb * Nq), k_v.rows_view(b0 * Nk, nb * Nk), Nq, Nk, dk, nbo=nb, nbi=h,
                        a_off=(Nq, 0, 0, dk), b_off=(Nk, 0, 0, dk), alpha=scale, c=S,
                        c_strides=(h * Nq * ldS, Nq * ldS))
            P = ops.softmax_operand(S[:nb].view(nb * h * Nq, ldS), Nk, mode,
                                    keep=keep[b0:b0 + nb] if keep is not None else None, rows_per_batch=h * Nq)
            ops.gemm_tc(P, vt.rows_view(b0 * D, nb * D), Nq, dk, Nk, nbo=nb, nbi=h, a_off=(h * Nq, Nq, 0, 0),
                        b_off=(D, dk, 0, 0), h=att.rows_view(b0 * Nq, nb * Nq), h_strides=(Nq * att.ld, dk), h_split=dk)
    if m.__dict__.get("record_attn", False):
        m.attn = attn_probs_head_sum(q_v, k_v, B, h, Nq, Nk, dk, scale, keep)
    return att


def mha_output(m, att, B, Nq, residual, mode, out=None):
    """linears[3] of the merged heads + the sublayer's residual (model/transformer.py:220-224, :147-153)."""
    W, Wt = mha_weights(m), mha_weights_tc(m, mode)
    D = m.h * m.d_k
    if out is None:
        out = torch.empty((B, Nq, D), dtype=_F32, device=residual.device)
    ops.gemm_tc(att, Wt["wo"], B * Nq, D, D, bias=W["bo"], c=out, residual=residual)
    return out


def mha_attend(m, q_v, k_v, vt, B, Nq, Nk, residual, mode, out=None, max_ws_bytes=3 << 30):
    att = mha_attention(m, q_v, k_v, vt, B, Nq, Nk, mode, residual.device, max_ws_bytes=max_ws_bytes)
    return mha_output(m, att, B, Nq, residual, mode, out=out)


def first_self_attention_pair(enc_layer, dec_layer, tok, B, N, mode, dec_out):
    """Encoder layer 0's and decoder layer 0's self-attention sublayers of the hoisted loop read the SAME tokens (the cloud's
    embedding): their QKV projections write the halves of one [2B]-item Q|K / V^T buffer and the attention itself runs as ONE
    flash launch over 2B items instead of two over B (each (batch, head) item is independent, so the bits do not change).
    Returns the encoder's sublayer output; the decoder's goes to ``dec_out``."""
    ea, da = enc_layer.self_attn, dec_layer.self_attn
    D = ea.h * ea.d_k
    dev = tok.device
    if (ea.h, ea.d_k, ea.is_src, da.is_src) != (da.h, da.d_k, False, False) or ea.__dict__.get("record_attn") or \
            da.__dict__.get("record_attn"):
        x = mha_tc(ea, _ln_op(enc_layer.sublayer[0].norm, tok, mode), None, B, N, N, tok, mode)
        mha_tc(da, _ln_op(dec_layer.sublayer[0].norm, tok, mode), None, B, N, N, tok, mode, out=dec_out)
        return x
    qk2 = ops.Operand.empty(2 * B * N, 2 * D, mode, dev)
    vt2 = ops.Operand.empty(2 * B * D, N, mode, dev)
    mha_project_self(ea, _ln_op(enc_layer.sublayer[0].norm, tok, mode), B, N, mode, dev, qk=qk2.rows_view(0, B * N),
                     vt=vt2.rows_view(0, B * D))
    mha_project_self(da, _ln_op(dec_layer.sublayer[0].norm, tok, mode), B, N, mode, dev, qk=qk2.rows_view(B * N, B * N),
                     vt=vt2.rows_view(B * D, B * D))
    att = mha_attention(ea, qk2.cols_view(0, D), qk2.cols_view(D, D), vt2, 2 * B, N, N, mode, dev)
    x = mha_output(ea, att.rows_view(0, B * N), B, N, tok, mode)
    mha_output(da, att.rows_view(B * N, B * N), B, N, tok, mode, out=dec_out)
    return x


def attn_probs_head_sum(q_v, k_v, B, h, Nq, Nk, dk, scale, keep):
    """``MultiHeadedAttention.attn`` (model/transformer.py:216-219): the probabilities summed over the heads, [B, Nq, Nk],
    what util/util.py:31-44 plots.  OPT-IN (``module.record_attn = True``): it is the one O(N^2) tensor of the path that
    the flash kernel exists to avoid, so it is materialised through the score GEMM + softmax only on request."""
    dev = q_v.buf.device
    ldS = (Nk + 3) // 4 * 4
    S = torch.empty((B, h, Nq, ldS), dtype=_F32, device=dev)
    ops.gemm_tc(q_v, k_v, Nq, Nk, dk, nbo=B, nbi=h, a_off=(Nq, 0, 0, dk), b_off=(Nk, 0, 0, dk), alpha=scale, c=S,
                c_strides=(h * Nq * ldS, Nq * ldS))
    ops.softmax_rows_(S.view(B * h * Nq, ldS)[:, :Nk], keep, h * Nq)
    return S[..., :Nk].sum(dim=1)


def mha_tc(m, xq_op, xkv_op, B, Nq, Nk, residual, mode, max_ws_bytes=3 << 30, out=None):
    """MultiHeadedAttention.forward (model/transformer.py:202-224) on tensor cores.

    xq_op / xkv_op: operand-format LayerNorm outputs [B*N, D] (xkv_op None => self-attention).
    Projections write Q, K row-major and V TRANSPOSED per head in operand format straight from the
    GEMM epilogue; attention is the flash kernel over (batch, head) addressed by row/column offsets."""
    dev = residual.device
    if xkv_op is None:
        q_v, k_v, vt = mha_project_self(m, xq_op, B, Nq, mode, dev)
    else:
        q_v = mha_project_q(m, xq_op, B * Nq, mode, dev)
        k_v, vt = mha_project_kv(m, xkv_op, B, Nk, mode, dev)
    return mha_attend(m, q_v, k_v, vt, B, Nq, Nk, residual, mode, out=out, max_ws_bytes=max_ws_bytes)


def ffn_tc(m, n_op, rows, residual, mode):
    """PositionwiseFeedForward (model/transformer.py:237-238); the hidden activation never exists in fp32."""
    w = packed(m, "ffn_" + mode, [m.w_1.weight, m.w_2.weight],
               lambda: (ops.to_operand(m.w_1.weight.detach(), mode), ops.to_operand(m.w_2.weight.detach(), mode)))
    F_, D = m.w_1.weight.shape
    hid = ops.Operand.empty(rows, F_, mode, residual.device)
    ops.gemm_tc(n_op, w[0], rows, F_, D, bias=m.w_1.bias, act=1, slope=0.0, h=hid, h_split=F_)
    out = torch.empty_like(residual)
    ops.gemm_tc(hid, w[1], rows, D, F_, bias=m.w_2.bias, c=out, residual=residual)
    return out


def _ln_op(norm, x, mode):
    return ops.layernorm_operand(x, norm.a_2, norm.b_2, norm.eps, mode)


class HeadPre:
    """What the VCP head derives from a Transformer output: its "h3" operand copy and squared row norms, written by the
    final LayerNorm kernel (vcr_layernorm_head) instead of separate to_operand / sqnorm_rows passes."""

    def __init__(self, op, sq):
        self.op, self.sq = op, sq


def encoder_decoder_tc(model, src, tgt, final_residual, mode, swap_mem=False, want_head=False, want_out=True):
    """swap_mem: decoder batch item b attends to the encoder output of item (b + B/2) mod B -- the two directions of
    Transformer.forward run as one batch [src; tgt] without building the swapped copy [tgt; src]: only the encoder's
    final LayerNorm writes its two halves exchanged."""
    B, Ns, D = src.shape
    Nt = tgt.shape[1]
    x = src
    for layer in model.encoder.layers:
        x = mha_tc(layer.self_attn, _ln_op(layer.sublayer[0].norm, x, mode), None, B, Ns, Ns, x, mode)
        x = ffn_tc(layer.feed_forward, _ln_op(layer.sublayer[1].norm, x, mode), B * Ns, x, mode)
    if swap_mem:
        half, nrm = B // 2, model.encoder.norm
        mem = ops.Operand.empty(B * Ns, D, mode, src.device)
        ops.layernorm_operand(x[:half], nrm.a_2, nrm.b_2, nrm.eps, mode, out=mem.rows_view(half * Ns, half * Ns))
        ops.layernorm_operand(x[half:], nrm.a_2, nrm.b_2, nrm.eps, mode, out=mem.rows_view(0, half * Ns))
    else:
        mem = _ln_op(model.encoder.norm, x, mode)
    y = tgt
    for layer in model.decoder.layers:
        y = mha_tc(layer.self_attn, _ln_op(layer.sublayer[0].norm, y, mode), None, B, Nt, Nt, y, mode)
        y = mha_tc(layer.src_attn, _ln_op(layer.sublayer[1].norm, y, mode), mem, B, Nt, Ns, y, mode)
        y = ffn_tc(layer.feed_forward, _ln_op(layer.sublayer[2].norm, y, mode), B * Nt, y, mode)
    if want_head:
        nrm = model.decoder.norm
        return ops.layernorm_head(y, nrm.a_2, nrm.b_2, nrm.eps, residual=final_residual, want_out=want_out)
    return _ln(model.decoder.norm, y, residual=final_residual)


class TargetInvariants:
    """Everything of one ``vcrnetIter`` call that depends on the TARGET cloud only (model/vcrnet_model.py:24-28: the loop
    transforms ``src`` and re-runs the network, ``tgt`` never changes), computed once per call instead of once per
    iteration as the reference does:

      * ``emb_nn(tgt)``                                                   (model/vcrnet_model.py:500)
      * ``encoder(tgt_emb)`` -- the memory of the ``src_p = model(tgt, src)`` direction (model/transformer.py:270) --
        and its K / V^T projections in every decoder layer's ``src_attn``
      * decoder layer 0's self-attention sublayer on ``tgt`` and the Q projection of the next sublayer
        (the ``tgt_p = model(src, tgt)`` direction, model/transformer.py:180-183)

    The per-iteration kernels read these through COMBINED 2B-item buffers ([src half | tgt half]) whose invariant half is
    written once here and whose other half is rewritten each iteration in place, so nothing is copied.  Every kernel on
    the path computes a batch item independently of its neighbours, hence outputs are bit-identical to the non-hoisted
    path (tests/test_gpu_parity.py::test_vcrnet_iter_hoisting_is_bit_identical)."""

    def __init__(self, net, tgt: torch.Tensor):
        tr = net.pointer
        model = tr.model
        mode = config.precision
        B, _, N = tgt.shape
        dev = tgt.device
        D = tr.emb_dims
        self.B, self.N, self.D, self.mode = B, N, D, mode
        self.emb2 = torch.empty((2 * B, N, D), dtype=_F32, device=dev)         # [emb(src) | emb(tgt)]
        emb_tokens(net.emb_nn, tgt, out=self.emb2[B:])
        tgt_tok = self.emb2[B:]
        # encoder(tgt): memory of the decoder items that hold src
        l0 = model.decoder.layers[0]
        self.y1 = torch.empty((2 * B, N, D), dtype=_F32, device=dev)           # [y1(src) | y1(tgt)]
        x = tgt_tok
        for li, layer in enumerate(model.encoder.layers):
            if li == 0:      # + decoder layer 0's self-attention sublayer on tgt (same input), one flash launch for both
                x = first_self_attention_pair(layer, l0, tgt_tok, B, N, mode, self.y1[B:])
            else:
                x = mha_tc(layer.self_attn, _ln_op(layer.sublayer[0].norm, x, mode), None, B, N, N, x, mode)
            x = ffn_tc(layer.feed_forward, _ln_op(layer.sublayer[1].norm, x, mode), B * N, x, mode)
        mem_t = _ln_op(model.encoder.norm, x, mode)
        self.k2, self.vt2 = [], []                                             # per decoder layer: [from enc(tgt) | from enc(src)]
        for layer in model.decoder.layers:
            k2 = ops.Operand.empty(2 * B * N, D, mode, dev)
            vt2 = ops.Operand.empty(2 * B * D, N, mode, dev)
            mha_project_kv(layer.src_attn, mem_t, B, N, mode, dev, k_out=k2.rows_view(0, B * N), vt_out=vt2.rows_view(0, B * D))
            self.k2.append(k2); self.vt2.append(vt2)
        # decoder layer 0: the query projection of sublayer 1 on tgt (sublayer 0 ran with the encoder's above)
        self.q2 = ops.Operand.empty(2 * B * N, D, mode, dev)                   # [Q(src) | Q(tgt)]
        mha_project_q(l0.src_attn, _ln_op(l0.sublayer[1].norm, self.y1[B:], mode), B * N, mode, dev,
                      out=self.q2.rows_view(B * N, B * N))

    @staticmethod
    def supported(net, src, tgt) -> bool:
        from .model.transformer import Transformer
        return (config.precision != "fp32" and isinstance(net.pointer, Transformer) and src.shape == tgt.shape
                and len(net.pointer.model.decoder.layers) >= 1 and len(net.pointer.model.encoder.layers) >= 1)


def emb_tokens(emb_nn, xyz, out=None):
    """emb_nn.forward_tokens, written into ``out`` when given (LPDNet writes there directly, the other embeddings copy)."""
    from .model.lpdnet_model import LPDNet
    if out is None:
        return emb_nn.forward_tokens(xyz)
    if isinstance(emb_nn, LPDNet) and not torch.is_grad_enabled():
        return lpdnet_tokens(emb_nn, xyz, out=out)
    out.copy_(emb_nn.forward_tokens(xyz))
    return out


def transformer_tokens_hoisted(tr, inv: TargetInvariants, want_head=False, want_out=True):
    """One refinement iteration of Transformer.forward + the VCRNet residual (model/transformer.py:264-272,
    model/vcrnet_model.py:504-505) given the target-side invariants; ``inv.emb2[:B]`` holds this iteration's emb(src).
    Returns what transformer_tokens(add_input=True) returns."""
    model, mode = tr.model, inv.mode
    B, N, D = inv.B, inv.N, inv.D
    dev = inv.emb2.device
    src_tok = inv.emb2[:B]
    # encoder(src): memory of the decoder items that hold tgt
    x = src_tok
    for li, layer in enumerate(model.encoder.layers):
        if li == 0:          # + decoder layer 0's self-attention sublayer on src (same input), one flash launch for both
            x = first_self_attention_pair(layer, model.decoder.layers[0], src_tok, B, N, mode, inv.y1[:B])
        else:
            x = mha_tc(layer.self_attn, _ln_op(layer.sublayer[0].norm, x, mode), None, B, N, N, x, mode)
        x = ffn_tc(layer.feed_forward, _ln_op(layer.sublayer[1].norm, x, mode), B * N, x, mode)
    mem_s = _ln_op(model.encoder.norm, x, mode)
    y = None
    for li, layer in enumerate(model.decoder.layers):
        k2, vt2 = inv.k2[li], inv.vt2[li]
        mha_project_kv(layer.src_attn, mem_s, B, N, mode, dev, k_out=k2.rows_view(B * N, B * N), vt_out=vt2.rows_view(B * D, B * D))
        if li == 0:
            y = inv.y1                           # sublayer 0 on src ran with the encoder's first layer above
            mha_project_q(layer.src_attn, _ln_op(layer.sublayer[1].norm, y[:B], mode), B * N, mode, dev,
                          out=inv.q2.rows_view(0, B * N))
            q2 = inv.q2
        else:
            y = mha_tc(layer.self_attn, _ln_op(layer.sublayer[0].norm, y, mode), None, 2 * B, N, N, y, mode)
            q2 = mha_project_q(layer.src_attn, _ln_op(layer.sublayer[1].norm, y, mode), 2 * B * N, mode, dev)
        y = mha_attend(layer.src_attn, q2, k2, vt2, 2 * B, N, N, y, mode)
        y = ffn_tc(layer.feed_forward, _ln_op(layer.sublayer[2].norm, y, mode), 2 * B * N, y, mode)
    nrm = model.decoder.norm
    if want_head:
        out, op, sq = ops.layernorm_head(y, nrm.a_2, nrm.b_2, nrm.eps, residual=inv.emb2, want_out=want_out)
        pre = (HeadPre(op.rows_view(0, B * N), sq[:B]), HeadPre(op.rows_view(B * N, B * N), sq[B:]))
        return (out[:B], out[B:], pre) if out is not None else (None, None, pre)
    out = _ln(nrm, y, residual=inv.emb2)
    return out[:B], out[B:]


def transformer_tokens(tr, src_tok: torch.Tensor, tgt_tok: torch.Tensor, add_input=False, want_head=False, want_out=True):
    """Transformer.forward on tokens (model/transformer.py:264-272).  The two directions
    (model(src,tgt) -> tgt_p and model(tgt,src) -> src_p) share weights and are independent, so
    they run as ONE batch of 2B.  Returns (src_p, tgt_p) tokens; with ``add_input`` the
    VCRNet residual (vcrnet_model.py:504-505) is fused: (src+src_p, tgt+tgt_p)."""
    B = src_tok.shape[0]
    if src_tok.shape[1] == tgt_tok.shape[1]:
        if (src_tok.is_contiguous() and tgt_tok.is_contiguous() and src_tok.untyped_storage().data_ptr() ==
                tgt_tok.untyped_storage().data_ptr() and
                tgt_tok.storage_offset() == src_tok.storage_offset() + src_tok.numel()):
            # the two halves of one embedding batch (VCRNet.forward): [src; tgt] already exists, no copy
            enc_in = src_tok.as_strided((2 * B,) + tuple(src_tok.shape[1:]), src_tok.stride(), src_tok.storage_offset())
        else:
            enc_in = torch.cat([src_tok, tgt_tok], dim=0)
        if config.precision != "fp32":
            enc_in = enc_in.contiguous()
            out = encoder_decoder_tc(tr.model, enc_in, enc_in, enc_in if add_input else None, config.precision, swap_mem=True,
                                     want_head=want_head, want_out=want_out)
            if want_head:
                out, op, sq = out
                n = enc_in.shape[1]
                pre = (HeadPre(op.rows_view(0, B * n), sq[:B]), HeadPre(op.rows_view(B * n, B * n), sq[B:]))
                return (out[:B], out[B:], pre) if out is not None else (None, None, pre)
            return out[:B], out[B:]
        dec_in = torch.cat([tgt_tok, src_tok], dim=0)
        out = encoder_decoder_tok(tr.model, enc_in, dec_in, final_residual=dec_in if add_input else None)
        return (out[B:], out[:B], None) if want_head else (out[B:], out[:B])
    tgt_p = encoder_decoder_tok(tr.model, src_tok, tgt_tok, final_residual=tgt_tok if add_input else None)
    src_p = encoder_decoder_tok(tr.model, tgt_tok, src_tok, final_residual=src_tok if add_input else None)
    return (src_p, tgt_p, None) if want_head else (src_p, tgt_p)


# --------------------------------------------------------------------------------------------------
# VCP head
# --------------------------------------------------------------------------------------------------

def pair_dots(src_tok, tgt_tok, alpha=1.0, pre=None):
    """dot[b,i,j] = alpha * s_i . t_j (the matmul of model/vcrnet_model.py:337): fp32 SIMT or 3-term tensor cores.
    The throughput modes keep the 3-term split here: these logits cancel catastrophically
    (|f|^2 ~ 500 against gaps < 1), SURVEY.md section 7 hard part 2."""
    if config.precision == "fp32":
        dot, ld = ops.pair_dots(src_tok, tgt_tok)
        if alpha != 1.0:
            dot.mul_(alpha)
        return dot, ld
    B, Ns, D = src_tok.shape
    Nt = tgt_tok.shape[1]
    ld = (Nt + 3) // 4 * 4
    dot = torch.empty((B, Ns, ld), dtype=_F32, device=src_tok.device)
    s_op = pre[0].op if pre is not None else ops.to_operand(src_tok, "h3")
    t_op = pre[1].op if pre is not None else ops.to_operand(tgt_tok, "h3")
    ops.gemm_tc(s_op, t_op, Ns, Nt, D, nbo=B,
                a_off=(Ns, 0, 0, 0), b_off=(Nt, 0, 0, 0), alpha=alpha, c=dot, c_strides=(Ns * ld, 0))
    return dot, ld


def vcp_whole(src_tok, tgt_tok, tgt_xyz, pre=None):
    """getCopairALL (model/vcrnet_model.py:334-347): src_corr [B,3,N].  pre: (HeadPre src, HeadPre tgt) from the final
    LayerNorm of the Transformer (operand copies + squared norms already in HBM)."""
    if pre is not None and config.precision == "fp32":
        pre = None
    if pre is not None:
        B, Ns, Nt, D = pre[0].sq.shape[0], pre[0].sq.shape[1], pre[1].sq.shape[1], pre[0].op.cols
    else:
        B, Ns, D = src_tok.shape
        Nt = tgt_tok.shape[1]
    xx, yy = (pre[0].sq, pre[1].sq) if pre is not None else (ops.sqnorm_rows(src_tok), ops.sqnorm_rows(tgt_tok))
    if config.precision != "fp32" and config.fused_softcorr:
        # one kernel: 3-term tcgen05 products + online softmax + weighted sum of the target points in the epilogue
        s_op = pre[0].op if pre is not None else ops.to_operand(src_tok.reshape(B * Ns, D), "h3")
        t_op = pre[1].op if pre is not None else ops.to_operand(tgt_tok.reshape(B * Nt, D), "h3")
        return ops.softcorr_tc(s_op, t_op, xx, yy, tgt_xyz, B, Ns, Nt, D)
    dot, ld = pair_dots(src_tok, tgt_tok, pre=pre)
    corr, _, _ = ops.softcorr_rows(dot, ld, Ns, Nt, xx, yy, tgt=tgt_xyz.contiguous(), mode=0)
    return corr


def vcp_by_dis(src_tok, tgt_tok, tgt_xyz):
    """VcpByDis.forward (model/vcrnet_model.py:402-421): softmax_j(s_i . t_j / sqrt(d_k)), src_corr = tgt P^T.
    Runs through the same fused row pass as getCopairALL with logits 2*(dot/(2 sqrt d_k)) - 0 - 0."""
    B, Ns, D = src_tok.shape
    Nt = tgt_tok.shape[1]
    dot, ld = pair_dots(src_tok, tgt_tok, alpha=0.5 / math.sqrt(D))
    zs = torch.zeros((B, Ns), dtype=_F32, device=src_tok.device)
    zt = torch.zeros((B, Nt), dtype=_F32, device=src_tok.device)
    corr, _, _ = ops.softcorr_rows(dot, ld, Ns, Nt, zs, zt, tgt=tgt_xyz.contiguous(), mode=0)
    return corr


def vcp_att(m, src_tok, tgt_tok, tgt_xyz):
    """VcpAtt.forward (model/vcrnet_model.py:424-460): two Linear(emb, emb) projections, then the getCopairALL arithmetic
    (linears_3d exist in the state_dict but are unused by the reference forward)."""
    q = ops.gemm(src_tok.contiguous(), m.linears_emb[0].weight, m.linears_emb[0].bias)
    k = ops.gemm(tgt_tok.contiguous(), m.linears_emb[1].weight, m.linears_emb[1].bias)
    return vcp_whole(q, k, tgt_xyz)


class Selected:
    """selectCom's output on the tensor-core path: the kept points' embeddings as "h3" operand rows + squared norms
    (gathered from the copies the Transformer's final LayerNorm wrote), never going back through fp32."""

    def __init__(self, op, sq):
        self.op, self.sq = op, sq


# vcp_select materialises the [B, Ns, Nt] fp32 score products up to this many points per cloud (in every precision
# mode); past it the tensor-core modes take the statistics from select_stats_tc and fp32 keeps materialising.
SELECT_STATS_MATERIALISED_MAX = 16384


def _select_stats_materialised(src_tok, tgt_tok, pre, B, Ns, Nt):
    """selectCom's (row_stat, col_stat) over the score products dot [B, Ns, ld] written to HBM."""
    if pre is None:
        src_tok, tgt_tok = src_tok.contiguous(), tgt_tok.contiguous()
        dot, ld = pair_dots(src_tok, tgt_tok)
        xx, yy = ops.sqnorm_rows(src_tok), ops.sqnorm_rows(tgt_tok)
    else:
        D = pre[0].op.cols
        ld = (Nt + 3) // 4 * 4
        dot = torch.empty((B, Ns, ld), dtype=_F32, device=pre[0].sq.device)
        ops.gemm_tc(pre[0].op, pre[1].op, Ns, Nt, D, nbo=B, a_off=(Ns, 0, 0, 0), b_off=(Nt, 0, 0, 0), c=dot,
                    c_strides=(Ns * ld, 0))
        xx, yy = pre[0].sq, pre[1].sq
    if Nt <= 1024:
        # scores (:213-214), both softmaxes and their sums (:221-222, :243-244) in one fused two-read pass
        row_stat, col_stat = ops.select_stats(dot, ld, Ns, Nt, xx, yy)
    else:                                                              # materialised passes for long clouds
        pd = ops.negdist_(dot, ld, Ns, Nt, xx, yy)
        row_stat = ops.rowsum_colsoftmax(pd, ld, Ns, Nt)
        col_stat = ops.colsum(ops.softmax_rows_(pd.view(B * Ns, ld)[:, :Nt]), B)
    return row_stat, col_stat


def vcp_select(src_xyz, src_tok, tgt_xyz, tgt_tok, overlap2, pre=None, want_tokens=True):
    """selectCom (model/vcrnet_model.py:190-262) without the unused *_remain host round trips.

    The two selection statistics come from one fused two-read pass over the score products (vcr_select_stats), or, in
    the tensor-core modes past 16 384 points, from the operands without the score products (vcr_select_stats_tc).  With
    ``pre`` (operand copies + squared norms of both embeddings) and ``want_tokens=False`` the selected embeddings are
    returned as ``Selected`` operand rows for vcp_copair instead of fp32 tokens (src_tok / tgt_tok may then be None)."""
    if pre is not None and config.precision == "fp32":
        pre = None
    ref = pre[0].sq if pre is not None else src_tok
    B, Ns = ref.shape[0], ref.shape[1]
    Nt = pre[1].sq.shape[1] if pre is not None else tgt_tok.shape[1]
    srcK = int(Ns * 0.84 * overlap2)
    tgtK = int(Nt * 0.84 * overlap2)
    if pre is not None and max(Ns, Nt) > SELECT_STATS_MATERIALISED_MAX:
        # past 16 384 points the [Ns, Nt] score matrix is 1 GB per pair and up: statistics from the operands instead
        row_stat, col_stat = ops.select_stats_tc(pre[0].op, pre[1].op, pre[0].sq, pre[1].sq, B, Ns, Nt, pre[0].op.cols)
    else:
        row_stat, col_stat = _select_stats_materialised(src_tok, tgt_tok, pre, B, Ns, Nt)
    both = row_stat._base
    if srcK == tgtK and both is not None and both is col_stat._base and tuple(both.shape) == (2, B, Ns):
        idx = ops.topk_select(both.view(2 * B, Ns), srcK)[0]           # both rankings (:222, :244) in one launch
        idx_s, idx_t = idx[:B], idx[B:]
    else:
        idx_t, _ = ops.topk_select(col_stat, tgtK)
        idx_s, _ = ops.topk_select(row_stat, srcK)
    so, to = ops.gather_cols(src_xyz, idx_s), ops.gather_cols(tgt_xyz, idx_t)
    if pre is not None and not want_tokens:
        s_sel = Selected(*ops.gather_operand_rows(pre[0].op, pre[0].sq, idx_s, B, Ns))
        t_sel = Selected(*ops.gather_operand_rows(pre[1].op, pre[1].sq, idx_t, B, Nt))
        return so, s_sel, to, t_sel, idx_s, idx_t
    return so, ops.gather_rows(src_tok, idx_s), to, ops.gather_rows(tgt_tok, idx_t), idx_s, idx_t


def vcp_copair(src_xyz, src_tok, tgt_xyz, tgt_tok, overlap2):
    """getCopair (model/vcrnet_model.py:264-332): hard arg-max correspondences for the
    int(Ns*0.52*overlap2) most confident sources (tgtK == 1 makes val/val_sum == 1).
    src_tok / tgt_tok: fp32 tokens [B,N,D], or ``Selected`` operand rows from vcp_select."""
    B, _, Ns = src_xyz.shape
    Nt = tgt_xyz.shape[2]
    srcK = int(Ns * 0.52 * overlap2)
    if isinstance(src_tok, Selected):
        best_i, best_v = ops.softcorr_best_tc(src_tok.op, tgt_tok.op, src_tok.sq, tgt_tok.sq, B, Ns, Nt, src_tok.op.cols)
    else:
        D = src_tok.shape[2]
        xx, yy = ops.sqnorm_rows(src_tok), ops.sqnorm_rows(tgt_tok)
        if config.precision != "fp32" and config.fused_softcorr:
            best_i, best_v = ops.softcorr_best_tc(ops.to_operand(src_tok.reshape(B * Ns, D), "h3"),
                                                  ops.to_operand(tgt_tok.reshape(B * Nt, D), "h3"), xx, yy, B, Ns, Nt, D)
        else:
            dot, ld = pair_dots(src_tok, tgt_tok)
            _, best_i, best_v = ops.softcorr_rows(dot, ld, Ns, Nt, xx, yy, mode=2)
    keep, _ = ops.topk_select(best_v, srcK)                            # [B,srcK] sorted by confidence
    src_k, corr_k = ops.copair_gather(src_xyz, tgt_xyz, keep, best_i)
    return src_k, corr_k, keep, best_i
