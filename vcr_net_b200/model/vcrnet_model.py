"""VCRNet assembly, VCP head, SVD head and the --iter loop with the reference's API
(reference model/vcrnet_model.py:21-43, 162-399, 463-518).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .lpdnet_model import LPDNet
from .transformer import Transformer


def vcrnetIter(net, src, tgt, iter=1):
    """model/vcrnet_model.py:21-43 with the reference's signature.

    ``net`` may be the bare VCRNet or the ``nn.DataParallel`` wrapper the reference's bootstrap always applies
    (util/initPara.py:260) and its loops pass in (model/vcrnet_model.py:561-563):
      * one device: the wrapper would call ``net.module`` directly (torch DataParallel.forward), so it is unwrapped here and
        the loop runs on the module -- with the loop-invariant hoisting and, when enabled, CUDA-graph replay;
      * several devices: the batch is scattered ONCE and every replica runs the whole ``iter`` loop on its shard
        (one replicate / scatter / gather per call instead of one per iteration); pairs are independent, so the gathered
        result has the bits of the single-device loop.
    With ``config.cuda_graph`` repeated calls with the same network, shapes and ``iter`` are served by a captured CUDA graph
    (vcr_net_b200/graph.py): the first call of a shape runs eagerly, the second captures, later ones replay; results are
    fresh tensors and bit-identical to the eager loop; any change of a parameter or buffer drops the cache."""
    from .. import config
    if isinstance(net, nn.DataParallel) and isinstance(net.module, VCRNet) and src.is_cuda:
        if len(net.device_ids) == 1 and src.device.index == net.device_ids[0]:
            net = net.module
        elif len(net.device_ids) > 1 and not (net.module.training and torch.is_grad_enabled()):
            loop = nn.DataParallel(_IterLoop(net.module, int(iter)), device_ids=net.device_ids,
                                   output_device=net.output_device, dim=net.dim)
            return loop(src, tgt)
    if (config.cuda_graph and isinstance(net, VCRNet) and not net.training and src.is_cuda
            and not torch.cuda.is_current_stream_capturing() and not net.__dict__.get("_is_replica", False)
            and not any(m.__dict__.get("record_attn", False) for m in net.modules())):
        return _vcrnet_iter_cached(net, src, tgt, int(iter))
    return _vcrnet_iter_eager(net, src, tgt, iter)


def vcrnetIterRagged(net, src, tgt, src_len, tgt_len, iter=1):
    """vcrnetIter over a ragged batch: pairs of different sizes in one call.

    src [B,3,Ns_max], tgt [B,3,Nt_max] fp32 CUDA, padded; src_len / tgt_len int32 [B] on the same device: pair b is
    (src[b, :, :src_len[b]], tgt[b, :, :tgt_len[b]]) -- vcr_net_b200.ragged.pad_clouds builds such a batch and checks the
    lengths (21 <= len <= N_max).  Padded columns may hold any finite values; nothing depends on them.
    Returns (srcK, src_corrK, R_ab, t_ab, R_ba, t_ba) as vcrnetIter does; restricted to a pair's lengths, each output equals
    vcrnetIter(net, src_b, tgt_b, iter) on the pair alone bit for bit.  Padded columns of srcK and src_corrK are 0.

    The lengths are read on the device only: no host sync and no length-dependent allocation, so the call can be captured
    in a CUDA graph once per (B, Ns_max, Nt_max) and replayed with new clouds and lengths written into the same tensors.
    Supported: eval-mode VCRNet on one device, whole-to-whole (partial=False), LPDNet embedding without t3d / tfea,
    Transformer or Identity pointer, topK head, the tensor-core precision modes; anything else raises
    NotImplementedError.  The network's cycle estimate (R_ba, t_ba of VCRNet.forward) is never computed: vcrnetIter
    returns the inverse of the composed pose instead, so ``cycle`` does not change the outputs."""
    _check_ragged_support(net, "vcrnetIterRagged", partial=False)
    return _iter_ragged(net, src, tgt, src_len, tgt_len, iter, "vcrnetIterRagged")


# the ragged partial path runs the one-CTA top-K selection and the materialised selectCom statistics (DESIGN section 8)
RAGGED_PARTIAL_MAX_POINTS = 16384


def vcrnetIterRaggedPartial(net, src, tgt, src_len, tgt_len, iter=1):
    """vcrnetIterRagged for partial-to-partial registration (VCRNet(partial=True)): pairs of different sizes in one call.

    Same arguments, padding contract and graph-capture property as vcrnetIterRagged, up to 16 384 points per cloud.
    Returns (srcK, src_corrK, R_ab, t_ab, R_ba, t_ba) as vcrnetIter does, srcK / src_corrK [B,3,K_max] with
    K_max = count(Ns_max): pair b has K_b = ragged.corr_lengths(src_len, net.head.overlap2)[b] valid columns, the rest are
    0.  Restricted to K_b columns, every output equals vcrnetIter(net, src_b, tgt_b, iter) on the pair alone bit for bit.
    Supported: as vcrnetIterRagged, with partial=True; the cycle estimate is not computed.  An overlap2 that leaves a
    cloud of 21 points with no key, selected point or correspondence raises ValueError."""
    from .. import ragged
    _check_ragged_support(net, "vcrnetIterRaggedPartial", partial=True)
    for name, x in (("src", src), ("tgt", tgt)):
        if x.dim() == 3 and x.shape[2] > RAGGED_PARTIAL_MAX_POINTS:
            raise NotImplementedError(f"vcrnetIterRaggedPartial: {x.shape[2]} points in `{name}` (at most "
                                      f"{RAGGED_PARTIAL_MAX_POINTS} per cloud; call vcrnetIter per pair beyond)")
    n0 = ragged.MIN_POINTS
    counts = [int(n0 * a.overlap2) for a in _partial_attentions(net)]
    ov = net.head.overlap2
    sel = int(n0 * 0.84 * ov)
    counts += [sel, int(sel * 0.52 * ov)]
    if min(counts) <= 0:
        raise ValueError(f"vcrnetIterRaggedPartial: overlap2 = {ov} keeps nothing of a {n0}-point cloud")
    return _iter_ragged(net, src, tgt, src_len, tgt_len, iter, "vcrnetIterRaggedPartial")


def _partial_attentions(net):
    if isinstance(net.pointer, Transformer):
        return [m for m in net.pointer.modules() if getattr(m, "is_src", False)]
    return []


def _iter_ragged(net, src, tgt, src_len, tgt_len, iter, fn):
    from .. import config
    if config.precision == "fp32":
        raise NotImplementedError(f"{fn}: precision 'fp32' (the tensor-core modes h3 / fp16 / bf16 are supported)")
    B = src.shape[0]
    for name, x in (("src", src), ("tgt", tgt)):
        ops._chk(x, name)
        if x.dim() != 3 or x.shape[0] != B or x.shape[1] != 3:
            raise ValueError(f"{fn}: `{name}` must be [B,3,N], got {tuple(x.shape)}")
    for name, n in (("src_len", src_len), ("tgt_len", tgt_len)):
        ops._lengths(n, B, name)
        if n.device != src.device:
            raise ValueError(f"{fn}: `{name}` must be on {src.device}")
    k = net.emb_nn.k
    with torch.no_grad():
        # the padding is replaced by zeros once: every padded row the network computes is then finite (flash attention
        # multiplies padded V columns by probabilities of exactly 0), whatever the caller left there
        transformed_src = ops.zero_padding(src, src_len, k + 1)
        tgt_z = ops.zero_padding(tgt, tgt_len, k + 1)
        R_f = t_f = None
        srcK = src_corrK = None
        for _ in range(iter):
            srcK, src_corrK, R, t = _forward_ragged(net, transformed_src, tgt_z, src_len, tgt_len)
            transformed_src = ops.rigid_apply(transformed_src, R, t)
            if R_f is None:
                R_f, t_f = R, t
            else:
                ops.pose_compose_(R, t, R_f, t_f)
        R_ba, t_ba = ops.pose_inverse(R_f, t_f)
        if not net.head.partial:
            srcK = ops.zero_padding(srcK, src_len, k + 1)
        return srcK, src_corrK, R_f, t_f, R_ba, t_ba


def _check_ragged_support(net, fn, partial):
    if isinstance(net, nn.DataParallel):
        raise NotImplementedError(f"{fn}: nn.DataParallel (pass the module on one device)")
    if not isinstance(net, VCRNet):
        raise NotImplementedError(f"{fn}: {type(net).__name__} (a VCRNet is required)")
    if net.training:
        raise NotImplementedError(f"{fn}: training mode (call .eval())")
    if not isinstance(net.emb_nn, LPDNet):
        raise NotImplementedError(f"{fn}: emb_nn {type(net.emb_nn).__name__} (only lpdnet)")
    if net.emb_nn.t3d or net.emb_nn.tfea:
        raise NotImplementedError(f"{fn}: LPDNet with t3d / tfea")
    if not isinstance(net.pointer, (Transformer, Identity)):
        raise NotImplementedError(f"{fn}: pointer {type(net.pointer).__name__} (transformer or identity)")
    if not isinstance(net.head, VcpTopK):
        raise NotImplementedError(f"{fn}: vcp_nn {type(net.head).__name__} (only topK)")
    if net.head.partial and not partial:
        raise NotImplementedError(f"{fn}: partial=True (only whole-to-whole registration; vcrnetIterRaggedPartial "
                                  "registers partial pairs)")
    if partial and not net.head.partial:
        raise NotImplementedError(f"{fn}: partial=False (vcrnetIterRagged registers whole-to-whole pairs)")


def _forward_ragged(net, src, tgt, src_len, tgt_len):
    """VCRNet.forward's (srcK, src_corrK, R_ab, t_ab) for a ragged batch (model/vcrnet_model.py:495-516)."""
    from .. import config, ragged
    src_tok = Fn.lpdnet_tokens(net.emb_nn, src, lengths=src_len)
    tgt_tok = Fn.lpdnet_tokens(net.emb_nn, tgt, lengths=tgt_len)
    pre = None
    if isinstance(net.pointer, Identity):
        src_tok, tgt_tok = src_tok * 2.0, tgt_tok * 2.0                                   # :502-505 with Identity
    else:
        # Transformer.forward (model/transformer.py:264-272) + emb: tgt_p = model(src, tgt), src_p = model(tgt, src), each
        # attention restricted to the pair's own tokens; the final LayerNorm writes what the head reads
        model, mode = net.pointer.model, config.precision
        _, op_t, sq_t = Fn.encoder_decoder_tc(model, src_tok, tgt_tok, tgt_tok, mode, want_head=True, want_out=False,
                                              lens=(src_len, tgt_len))
        _, op_s, sq_s = Fn.encoder_decoder_tc(model, tgt_tok, src_tok, src_tok, mode, want_head=True, want_out=False,
                                              lens=(tgt_len, src_len))
        pre = (Fn.HeadPre(op_s, sq_s), Fn.HeadPre(op_t, sq_t))
        src_tok = tgt_tok = None
    if net.head.partial:                                                                       # :507 (selectCom, getCopair)
        ov = net.head.overlap2
        so, seo, to, teo, _, _ = Fn.vcp_select(src, src_tok, tgt, tgt_tok, ov, pre=pre, want_tokens=False,
                                               lengths=(src_len, tgt_len))
        sel = (ragged.select_counts(src_len, ov), ragged.select_counts(tgt_len, ov))
        srcK, corr, _, _ = Fn.vcp_copair(so, seo, to, teo, ov, lengths=sel)
        m = ragged.copair_counts(sel[0], ov)
    else:
        srcK, corr = src, Fn.vcp_whole(src_tok, tgt_tok, tgt, pre=pre, lengths=(src_len, tgt_len))
        m = src_len
    R, t, _, _ = ops.svd_head_ragged(srcK, corr, m)                                            # :509-516
    return srcK, corr, R, t


class _IterLoop(nn.Module):
    """The refinement loop as a module, so that nn.DataParallel replicates / scatters once per vcrnetIter call."""

    def __init__(self, net, iters):
        super().__init__()
        self.net, self.iters = net, iters

    def forward(self, src, tgt):
        return _vcrnet_iter_eager(self.net, src, tgt, self.iters)


_GRAPH_CACHE_MAX = 4


def _vcrnet_iter_cached(net, src, tgt, iter):
    from .. import config
    from ..graph import GraphedRegistration
    # every parameter AND buffer by (address, version): catches in-place updates, replaced tensors (.to() / .half() /
    # load_state_dict(assign=True) / p.data = ...) and BatchNorm statistics
    stamp = tuple((t.data_ptr(), t._version) for t in list(net.parameters()) + list(net.buffers()))
    cache = net.__dict__.setdefault("_vcr_graph_cache", {"stamp": stamp, "entries": {}})
    if cache["stamp"] != stamp:                       # weights were updated in place: captured pointers may be stale
        cache["stamp"], cache["entries"] = stamp, {}
    key = (tuple(src.shape), tuple(tgt.shape), iter, str(src.device)) + config.graph_key()
    ent = cache["entries"].get(key)
    if ent is None:
        if len(cache["entries"]) >= _GRAPH_CACHE_MAX:
            cache["entries"].pop(next(k0 for k0 in cache["entries"]))      # oldest shape first
        cache["entries"][key] = "seen"               # capture on the second call of this shape, not for one-off shapes
        return _vcrnet_iter_eager(net, src, tgt, iter)
    if ent == "seen":
        ent = cache["entries"][key] = GraphedRegistration(net, batch=src.shape[0], num_points=src.shape[2], iter=iter,
                                                          num_points_tgt=tgt.shape[2])
    return tuple(o.clone() for o in ent(src, tgt))


def _vcrnet_iter_eager(net, src, tgt, iter=1):
    """model/vcrnet_model.py:21-43: refine `iter` times, composing R_f <- R_i R_f, t_f <- R_i t_f + t_i.

    The target cloud never changes inside the loop, so with iter > 1 everything that depends on it alone
    (functional.TargetInvariants: emb_nn(tgt), encoder(tgt_emb), the decoder's first self-attention sublayer on tgt and
    the projections that read them) is computed once per call instead of ``iter`` times as the reference does (:27).
    ``config.hoist`` = "all" (default) | "emb" | "none"; outputs are bit-identical at every level."""
    from .. import config
    transformed_src = src
    R_f = t_f = None
    srcK = src_corrK = None
    kw = {}
    if iter > 1 and config.hoist != "none" and isinstance(net, VCRNet) and not (net.training and torch.is_grad_enabled()):
        with torch.no_grad():
            tgt_c = tgt.contiguous()
            if config.hoist == "all" and Fn.TargetInvariants.supported(net, src, tgt_c):
                kw = {"invariants": Fn.TargetInvariants(net, tgt_c)}
            else:
                kw = {"tgt_tokens": net.emb_nn.forward_tokens(tgt_c)}
    for _ in range(iter):
        srcK, src_corrK, R, t, _, _ = net(transformed_src, tgt, **kw)
        transformed_src = ops.rigid_apply(transformed_src, R, t)
        if R_f is None:
            R_f, t_f = R.detach().clone(), t.detach().clone()
        else:
            ops.pose_compose_(R.detach(), t.detach(), R_f, t_f)
    R_ba, t_ba = ops.pose_inverse(R_f, t_f)
    return srcK, src_corrK, R_f, t_f, R_ba, t_ba


def vcrnetIcpNet(args, net, src, tgt):
    """model/vcrnet_model.py:46-62 (--iter=0): one network pass, then ICP refinement of the transformed source."""
    from .icp_model import ICP
    icp = ICP(max_iterations=args.max_iterations).to(src.device)
    _, _, R, t, _, _ = net(src, tgt)
    transformed_src = ops.rigid_apply(src, R, t)
    _, _, R_icp, t_icp, _, _ = icp(transformed_src, tgt)
    R_f, t_f = R.clone(), t.clone()
    ops.pose_compose_(R_icp, t_icp, R_f, t_f)                              # R <- R_icp R, t <- R_icp t + t_icp
    R_ba, t_ba = ops.pose_inverse(R_f, t_f)
    return transformed_src, tgt, R_f, t_f, R_ba, t_ba


class Identity(nn.Module):
    def forward(self, *input):
        return input


class PointNet(nn.Module):
    """model/vcrnet_model.py:66-88 (--emb_nn pointnet).  Same parameter / buffer names as the reference
    (conv1..5 bias-free Conv1d, bn1..5 BatchNorm1d); eval-mode forward on the CUDA path."""

    def __init__(self, emb_dims=512):
        super().__init__()
        dims = [3, 64, 64, 64, 128, emb_dims]
        for i in range(5):
            setattr(self, f"conv{i + 1}", nn.Conv1d(dims[i], dims[i + 1], kernel_size=1, bias=False))
        for i in range(5):
            setattr(self, f"bn{i + 1}", nn.BatchNorm1d(dims[i + 1]))

    def forward_tokens(self, x):
        return Fn.pointnet_tokens(self, x)

    def forward(self, x):
        return ops.transpose_batched(self.forward_tokens(x))


class DGCNN(nn.Module):
    """model/vcrnet_model.py:90-123 (--emb_nn dgcnn).  Same parameter / buffer names as the reference
    (conv1..5 bias-free Conv2d, bn1..5 BatchNorm2d); eval-mode forward on the CUDA path."""

    def __init__(self, emb_dims=512):
        super().__init__()
        dims = [(6, 64), (64, 64), (64, 128), (128, 256), (512, emb_dims)]
        for i, (ci, co) in enumerate(dims):
            setattr(self, f"conv{i + 1}", nn.Conv2d(ci, co, kernel_size=1, bias=False))
        for i, (ci, co) in enumerate(dims):
            setattr(self, f"bn{i + 1}", nn.BatchNorm2d(co))

    def forward_tokens(self, x, idx=None, stages=None):
        return Fn.dgcnn_tokens(self, x, idx=idx, stages=stages)

    def forward(self, x, idx=None):
        return ops.transpose_batched(self.forward_tokens(x, idx=idx))


class VcpTopK(nn.Module):
    """model/vcrnet_model.py:162-347.  forward(src_emb, tgt_emb [B,D,N], src, tgt [B,3,N]) -> (src, src_corr)."""

    def __init__(self, args):
        super().__init__()
        self.emb_nn = args.emb_nn
        self.partial = args.partial
        self.overlap2 = float(args.overlap2)

    def forward_tokens(self, src_tok, tgt_tok, src, tgt, pre=None):
        """pre: (HeadPre src, HeadPre tgt) from the Transformer's final LayerNorm; the tokens may then be None."""
        if self.partial:
            so, seo, to, teo, _, _ = Fn.vcp_select(src, src_tok, tgt, tgt_tok, self.overlap2, pre=pre, want_tokens=False)
            s, c, _, _ = Fn.vcp_copair(so, seo, to, teo, self.overlap2)
            return s, c
        if src_tok is not None:
            src_tok, tgt_tok = src_tok.contiguous(), tgt_tok.contiguous()
        return src, Fn.vcp_whole(src_tok, tgt_tok, tgt, pre=pre)

    def forward(self, *input):
        src_tok = ops.transpose_batched(input[0])
        tgt_tok = ops.transpose_batched(input[1])
        return self.forward_tokens(src_tok, tgt_tok, input[2], input[3])

    # reference method names, channel-major signatures
    def getCopairALL(self, src, src_emb, tgt, tgt_emb):
        return src, Fn.vcp_whole(ops.transpose_batched(src_emb), ops.transpose_batched(tgt_emb), tgt)

    def selectCom(self, src, src_emb, tgt, tgt_emb, overlap2=0.75):
        so, seo, to, teo, _, _ = Fn.vcp_select(src, ops.transpose_batched(src_emb), tgt,
                                               ops.transpose_batched(tgt_emb), float(overlap2))
        return so, ops.transpose_batched(seo), to, ops.transpose_batched(teo), None, None

    def getCopair(self, src, src_emb, tgt, tgt_emb, overlap2):
        s, c, _, _ = Fn.vcp_copair(src, ops.transpose_batched(src_emb), tgt, ops.transpose_batched(tgt_emb),
                                   float(overlap2))
        return s, c


class VcpByDis(nn.Module):
    """model/vcrnet_model.py:402-421 (--vcp_nn dist): scaled-dot softmax correspondences."""

    def __init__(self, args):
        super().__init__()
        self.emb_nn = args.emb_nn

    def forward_tokens(self, src_tok, tgt_tok, src, tgt):
        return src, Fn.vcp_by_dis(src_tok.contiguous(), tgt_tok.contiguous(), tgt)

    def forward(self, *input):
        return self.forward_tokens(ops.transpose_batched(input[0]), ops.transpose_batched(input[1]), input[2], input[3])


class VcpAtt(nn.Module):
    """model/vcrnet_model.py:424-460 (--vcp_nn att).  Same parameters as the reference: linears_emb.{0,1} (used) and
    linears_3d.{0,1} (present in the checkpoint, unused by the reference forward)."""

    def __init__(self, args):
        super().__init__()
        from .transformer import clones
        self.emb_dims = args.emb_dims
        self.linears_emb = clones(nn.Linear(self.emb_dims, self.emb_dims), 2)
        self.linears_3d = clones(nn.Linear(3, 3), 2)
        self.attn = None
        self.dropout = None
        self.mask = None

    def forward_tokens(self, src_tok, tgt_tok, src, tgt):
        return src, Fn.vcp_att(self, src_tok, tgt_tok, tgt)

    def forward(self, *input):
        return self.forward_tokens(ops.transpose_batched(input[0]), ops.transpose_batched(input[1]), input[2], input[3])


class SVDHead(nn.Module):
    """model/vcrnet_model.py:350-399.  forward(src, src_corr [B,3,M]) -> (R [B,3,3], t [B,3])."""

    def __init__(self, args):
        super().__init__()
        self.reflect = nn.Parameter(torch.eye(3), requires_grad=False)
        self.reflect[2, 2] = -1

    def forward(self, src, src_corr):
        R, t, _, _ = ops.svd_head(src, src_corr)
        return R, t


class VCRNet(nn.Module):
    """model/vcrnet_model.py:463-518.  forward(src, tgt [B,3,N]) ->
    (srcK, src_corrK, R_ab, t_ab, R_ba, t_ba)."""

    def __init__(self, args):
        super().__init__()
        self.emb_dims = args.emb_dims
        self.cycle = args.cycle
        if args.emb_nn == 'pointnet':                      # :468-475
            self.emb_nn = PointNet(emb_dims=self.emb_dims)
        elif args.emb_nn == 'dgcnn':
            self.emb_nn = DGCNN(emb_dims=self.emb_dims)
        elif args.emb_nn == 'lpdnet':
            self.emb_nn = LPDNet(args)
        else:
            raise Exception('Not implemented')
        if args.pointer == 'identity':
            self.pointer = Identity()
        elif args.pointer == 'transformer':
            self.pointer = Transformer(args=args)
        else:
            self.pointer = None
        if args.vcp_nn == 'topK':                          # :484-491
            self.head = VcpTopK(args=args)
        elif args.vcp_nn == 'att':
            self.head = VcpAtt(args=args)
        elif args.vcp_nn == 'dist':
            self.head = VcpByDis(args=args)
        else:
            raise Exception("Not implemented")
        self.svd = SVDHead(args=args)

    def forward(self, *input, stages=None, tgt_tokens=None, invariants=None):
        # registration INFERENCE path: only the LPD pre-training path (LPD / LPDNet) has a backward
        if self.training and torch.is_grad_enabled():
            raise NotImplementedError(
                "VCRNet training is not implemented on the B200 path (inference only: model/vcrnet_model.py:495-518 under "
                "eval() / torch.no_grad(), as test_one_epoch runs it); LPD pre-training (--model=lpd) has a backward")
        with torch.no_grad():
            return self._forward(*input, stages=stages, tgt_tokens=tgt_tokens, invariants=invariants)

    def _forward(self, *input, stages=None, tgt_tokens=None, invariants=None):
        src, tgt = input[0].contiguous(), input[1].contiguous()
        B = src.shape[0]
        same = src.shape == tgt.shape
        if invariants is not None:                         # loop-invariant target-side state supplied by vcrnetIter
            Fn.emb_tokens(self.emb_nn, src, out=invariants.emb2[:B])
            src_tok, tgt_tok = invariants.emb2[:B], invariants.emb2[B:]
        elif tgt_tokens is not None:                       # loop-invariant target embedding supplied by vcrnetIter
            src_tok, tgt_tok = self.emb_nn.forward_tokens(src), tgt_tokens
        elif same:                                         # both clouds through ONE batch of 2B
            emb = self.emb_nn.forward_tokens(torch.cat([src, tgt], dim=0))
            src_tok, tgt_tok = emb[:B], emb[B:]
        else:
            src_tok, tgt_tok = self.emb_nn.forward_tokens(src), self.emb_nn.forward_tokens(tgt)
        if stages is not None:
            stages.update(src_emb0=src_tok, tgt_emb0=tgt_tok)
        pre = None
        if isinstance(self.pointer, Identity):
            # :502-505 with Identity: emb_p = emb, so emb + emb_p = 2 * emb for both clouds (head logits scale by 4)
            src_tok, tgt_tok = src_tok * 2.0, tgt_tok * 2.0
        elif isinstance(self.pointer, Transformer) and invariants is not None:
            want_head = isinstance(self.head, VcpTopK)
            res = Fn.transformer_tokens_hoisted(self.pointer, invariants, want_head=want_head, want_out=stages is not None)
            src_tok, tgt_tok = res[0], res[1]
            pre = res[2] if want_head else None
        elif isinstance(self.pointer, Transformer):
            if isinstance(self.head, VcpTopK):     # the final LayerNorm also writes what the head derives from its output
                # (operand copy + squared norms); the fp32 copy is only stored when a caller asks for the stages
                src_tok, tgt_tok, pre = self.pointer.forward_tokens(src_tok, tgt_tok, add_input=True, want_head=True,
                                                                    want_out=stages is not None)
            else:
                src_tok, tgt_tok = self.pointer.forward_tokens(src_tok, tgt_tok, add_input=True)   # :503-505
        if stages is not None:
            stages.update(src_emb=src_tok, tgt_emb=tgt_tok)
        hk = {"pre": pre} if pre is not None else {}
        srcK, src_corrK = self.head.forward_tokens(src_tok, tgt_tok, src, tgt, **hk)            # :507
        R_ab, t_ab, R_ba, t_ba = ops.svd_head(srcK, src_corrK)                                  # :509-516
        if self.cycle:
            hk = {"pre": (pre[1], pre[0])} if pre is not None else {}
            srcK_ba, corrK_ba = self.head.forward_tokens(tgt_tok, src_tok, tgt, src, **hk)
            R_ba, t_ba, _, _ = ops.svd_head(srcK_ba, corrK_ba)
        return srcK, src_corrK, R_ab, t_ab, R_ba, t_ba
