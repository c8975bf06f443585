"""Thin torch-tensor front-end over the C ABI (include/vcr_b200.h).

PyTorch is plumbing here: device memory (torch.empty), the current CUDA stream and nothing
else.  Every function launches hand-written sm_100a kernels from libvcr_b200.so on
``torch.cuda.current_stream()`` of the tensor's device; CPU tensors are rejected (no fallback).
"""
from __future__ import annotations

import math

import torch

from ._lib import lib

_F32 = torch.float32


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _chk(t: torch.Tensor, name: str, dtype=_F32):
    if not t.is_cuda:
        raise RuntimeError(f"vcr_net_b200: `{name}` must be a CUDA tensor (no CPU fallback exists)")
    if t.dtype != dtype:
        raise RuntimeError(f"vcr_net_b200: `{name}` must be {dtype}, got {t.dtype}")
    return t


def _rows(t: torch.Tensor):
    """2-D row-major view info of a tensor whose last dim is contiguous and whose leading dims
    collapse to a single row stride: (rows, cols, ld)."""
    assert t.stride(-1) == 1, "last dim must be contiguous"
    cols = t.shape[-1]
    ld = t.stride(-2) if t.dim() >= 2 else cols
    rows = 1
    for d in range(t.dim() - 1):
        rows *= t.shape[d]
    exp = ld
    for d in range(t.dim() - 2, -1, -1):       # leading dims must be dense over ld
        assert t.shape[d] == 1 or t.stride(d) == exp, "tensor rows are not uniformly strided"
        exp *= t.shape[d]
    return rows, cols, ld


# --------------------------------------------------------------------------------------------------
# kNN / graph / FPS
# --------------------------------------------------------------------------------------------------

def knn_topk(x: torch.Tensor, k: int, token_major: bool = False, want64: bool = False):
    """x [B,D,N] (or [B,N,D] when token_major) -> idx int32 [B,N,k] (and int64 when want64)."""
    _chk(x, "x")
    x = x.contiguous()
    if token_major:
        B, N, D = x.shape
    else:
        B, D, N = x.shape
    L = lib()
    idx32 = torch.empty((B, N, k), dtype=torch.int32, device=x.device)
    idx64 = torch.empty((B, N, k), dtype=torch.int64, device=x.device) if want64 else None
    ws_bytes = L.vcr_knn_workspace_bytes(B, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    L.check(L.vcr_knn_topk(x.data_ptr(), B, D, N, k, int(token_major), idx32.data_ptr(),
                           idx64.data_ptr() if want64 else None, ws.data_ptr(), ws_bytes, _stream(x)),
            "vcr_knn_topk")
    return (idx32, idx64) if want64 else idx32


def set_knn3_direct(on: bool) -> bool:
    """D == 3 route of knn_topk: on-the-fly distances (default) or the generic distance-tile kernel; same indices."""
    return bool(lib().vcr_set_knn3_direct(int(bool(on))))


def knn_topk_tc(x: torch.Tensor, xop, k: int, want64: bool = False, want_flagged: bool = False):
    """Feature-space kNN with the tcgen05 prefilter (csrc/knn.cu): x fp32 token-major [B,N,D], xop its "h3" Operand
    (None: converted here).  Same (bit-identical) result as knn_topk(x, k, token_major=True).
    want_flagged: also return the device counter of queries that were recomputed by the exact kernel."""
    _chk(x, "x")
    x = x.contiguous()
    B, N, D = x.shape
    if xop is None:
        xop = to_operand(x.view(B * N, D), "h3")
    assert xop.mode == "h3" and xop.rows == B * N and xop.cols == D
    L = lib()
    idx32 = torch.empty((B, N, k), dtype=torch.int32, device=x.device)
    idx64 = torch.empty((B, N, k), dtype=torch.int64, device=x.device) if want64 else None
    ws_bytes = L.vcr_knn_tc_workspace_bytes(B, N)
    ws = torch.empty(ws_bytes // 4, dtype=torch.int32, device=x.device)
    L.check(L.vcr_knn_topk_tc(x.data_ptr(), xop.ptr, xop.ld, xop.plane_stride, B, D, N, k, idx32.data_ptr(),
                              idx64.data_ptr() if want64 else None, ws.data_ptr(), ws_bytes, _stream(x)),
            "vcr_knn_topk_tc")
    out = (idx32, idx64) if want64 else (idx32,)
    if want_flagged:
        out = out + (ws[-1:],)
    return out if len(out) > 1 else out[0]


def knn_tc_supported(D: int, k: int) -> bool:
    return 16 <= D <= 128 and D % 4 == 0 and 1 <= k <= 30


def graph_feature(xt: torch.Tensor, idx: torch.Tensor):
    """xt token-major [B,N,D], idx int32 [B,N,k] -> [B,2D,N,k] (reference layout)."""
    _chk(xt, "xt"); _chk(idx, "idx", torch.int32)
    xt, idx = xt.contiguous(), idx.contiguous()
    B, N, D = xt.shape
    k = idx.shape[2]
    out = torch.empty((B, 2 * D, N, k), dtype=_F32, device=xt.device)
    L = lib()
    L.check(L.vcr_graph_feature(xt.data_ptr(), B, D, N, k, idx.data_ptr(), out.data_ptr(), _stream(xt)),
            "vcr_graph_feature")
    return out


# vcr_fps: one CTA per cloud up to 14 336 points, one cluster of up to 16 such CTAs beyond
FPS_MAX_POINTS = 16 * 14336


def fps(xyz: torch.Tensor, npoint: int, want64: bool = True):
    _chk(xyz, "xyz")
    xyz = xyz.contiguous()
    B, C, N = xyz.shape
    assert C == 3
    dt = torch.int64 if want64 else torch.int32
    out = torch.empty((B, npoint), dtype=dt, device=xyz.device)
    L = lib()
    rc = L.vcr_fps(xyz.data_ptr(), B, N, npoint, None if want64 else out.data_ptr(),
                   out.data_ptr() if want64 else None, _stream(xyz))
    if rc != 0 and N > FPS_MAX_POINTS:
        raise RuntimeError(f"vcr_fps failed: {rc}: farthest-point sampling takes at most {FPS_MAX_POINTS} points "
                           f"per cloud, got {N}")
    L.check(rc, "vcr_fps")
    return out


# --------------------------------------------------------------------------------------------------
# nearest-to-anchor crop of the data step
# --------------------------------------------------------------------------------------------------

# vcr_crop_nearest: one CTA per cloud (its fp64 distances in shared memory) up to 25 600 points; vcr_crop_nearest_sort:
# a segmented radix sort in a workspace, any cloud size while the batch holds at most 2^31 - 1 points
CROP_ONE_CTA_MAX_POINTS = 25600
CROP_MAX_TOTAL_POINTS = 2**31 - 1


def crop_nearest(pc64: torch.Tensor, keep: int):
    """pc64 fp64 [P,3,N] -> fp32 [P,3,keep]: the keep points nearest to point N-1, nearest first, ties to the lower index
    (util/data.py:320-329).  Up to 25 600 points the one-CTA rank-count kernel, above that the radix sort."""
    _chk(pc64, "pc64", torch.float64)
    P, C, N = pc64.shape
    assert C == 3
    if N > CROP_ONE_CTA_MAX_POINTS:
        return crop_nearest_sort(pc64, keep)
    pc64 = pc64.contiguous()
    out = torch.empty((P, 3, keep), dtype=_F32, device=pc64.device)
    L = lib()
    L.check(L.vcr_crop_nearest(pc64.data_ptr(), P, N, keep, out.data_ptr(), _stream(pc64)), "vcr_crop_nearest")
    return out


def crop_nearest_sort(pc64: torch.Tensor, keep: int):
    """crop_nearest by the segmented radix sort (vcr_crop_nearest_sort) at any N; P * N <= 2^31 - 1."""
    _chk(pc64, "pc64", torch.float64)
    P, C, N = pc64.shape
    assert C == 3
    if P * N > CROP_MAX_TOTAL_POINTS:
        raise RuntimeError(f"vcr_crop_nearest_sort: the crop takes at most {CROP_MAX_TOTAL_POINTS} points per call "
                           f"(clouds x points), got {P} x {N}")
    pc64 = pc64.contiguous()
    out = torch.empty((P, 3, keep), dtype=_F32, device=pc64.device)
    L = lib()
    wsb = L.vcr_crop_nearest_workspace_bytes(P, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=pc64.device)
    L.check(L.vcr_crop_nearest_sort(pc64.data_ptr(), P, N, keep, out.data_ptr(), ws.data_ptr(), wsb, _stream(pc64)),
            "vcr_crop_nearest_sort")
    return out


# --------------------------------------------------------------------------------------------------
# GEMM
# --------------------------------------------------------------------------------------------------

def gemm(a: torch.Tensor, w: torch.Tensor, bias=None, *, out=None, residual=None, act: int = 0,
         slope: float = 0.0, alpha: float = 1.0, b_layout: int = 0):
    """out[M,N] = act(alpha * a[M,K] @ w[N,K]^T + bias) + residual.  a/out/residual may be strided
    row views (last dim contiguous).  b_layout=1: w is stored [K,N] (out = a @ w, the data-gradient product)."""
    _chk(a, "a"); _chk(w, "w")
    M, K, lda = _rows(a)
    if b_layout == 0:
        N, K2, ldb = _rows(w)
    else:
        K2, N, ldb = _rows(w)
    assert K == K2, (K, K2)
    if out is None:
        out = torch.empty(a.shape[:-1] + (N,), dtype=_F32, device=a.device)
    Mo, No, ldc = _rows(out)
    assert (Mo, No) == (M, N)
    ldr = 0
    if residual is not None:
        Mr, Nr, ldr = _rows(residual)
        assert (Mr, Nr) == (M, N)
    L = lib()
    L.check(L.vcr_gemm_f32(a.data_ptr(), lda, 0, 0, w.data_ptr(), ldb, 0, 0, int(b_layout),
                           out.data_ptr(), ldc, 0, 0,
                           bias.data_ptr() if bias is not None else None,
                           residual.data_ptr() if residual is not None else None, ldr, 0, 0,
                           M, N, K, 1, 1, float(alpha), int(act), float(slope), _stream(a)), "vcr_gemm_f32")
    return out


def bgemm(a, a_ld, a_so, a_si, b, b_ld, b_so, b_si, b_layout, c, c_ld, c_so, c_si, M, N, K, nbo, nbi,
          alpha=1.0):
    """Raw batched GEMM over base tensors + element strides (attention heads, per-pair scores)."""
    L = lib()
    L.check(L.vcr_gemm_f32(a.data_ptr(), a_ld, a_so, a_si, b.data_ptr(), b_ld, b_so, b_si, b_layout,
                           c.data_ptr(), c_ld, c_so, c_si, None, None, 0, 0, 0,
                           M, N, K, nbo, nbi, float(alpha), 0, 0.0, _stream(c)), "vcr_gemm_f32")
    return c


# --------------------------------------------------------------------------------------------------
# tensor-core GEMM on operand-format buffers
# --------------------------------------------------------------------------------------------------

TC_MODES = {"h3": 0, "fp16": 1, "bf16": 2}


class Operand:
    """16-bit K-major operand buffer [planes, rows, ld] for vcr_gemm_tc: plane 0 = hi = fp16(x),
    plane 1 = lo = fp16((x - hi) * 2^11) in the 3-term "h3" mode; one plane in fp16 / bf16 modes.
    Views (column / row sub-ranges) share the storage and only move the base pointer."""

    def __init__(self, buf, rows, cols, ld, planes, plane_stride, ptr, mode):
        self.buf, self.rows, self.cols, self.ld = buf, rows, cols, ld
        self.planes, self.plane_stride, self.ptr, self.mode = planes, plane_stride, ptr, mode

    @staticmethod
    def empty(rows, cols, mode="h3", device="cuda"):
        planes = 2 if mode == "h3" else 1
        dt = torch.bfloat16 if mode == "bf16" else torch.float16
        ld = (cols + 7) // 8 * 8
        buf = torch.empty((planes, rows, ld), dtype=dt, device=device)
        return Operand(buf, rows, cols, ld, planes, rows * ld, buf.data_ptr(), mode)

    def cols_view(self, c0, ncols):
        assert c0 % 8 == 0
        return Operand(self.buf, self.rows, ncols, self.ld, self.planes, self.plane_stride, self.ptr + 2 * c0, self.mode)

    def rows_view(self, r0, nrows):
        return Operand(self.buf, nrows, self.cols, self.ld, self.planes, self.plane_stride,
                       self.ptr + 2 * r0 * self.ld, self.mode)

    def to_float(self):
        x = self.buf[0, :, :self.cols].float()
        if self.planes == 2:
            x = x + self.buf[1, :, :self.cols].float() / 2048.0
        return x


def to_operand(x: torch.Tensor, mode="h3") -> Operand:
    """fp32 rows [.., cols] -> operand format."""
    _chk(x, "x")
    rows, cols, ld = _rows(x)
    out = Operand.empty(rows, cols, mode, x.device)
    L = lib()
    L.check(L.vcr_to_operand(x.data_ptr(), ld, rows, cols, out.ptr, out.ld, out.plane_stride,
                             out.planes, int(mode == "bf16"), _stream(x)), "vcr_to_operand")
    return out


def gemm_tc(a: Operand, b: Operand, M, N, K, *, nbo=1, nbi=1,
            a_off=(0, 0, 0, 0), b_off=(0, 0, 0, 0), alpha=1.0, bias=None, act=0, slope=0.0,
            c=None, c_strides=(0, 0), residual=None, r_strides=(0, 0),
            h: Operand | None = None, h_strides=(0, 0), h_split=0,
            ht: Operand | None = None, ht_strides=(0, 0)):
    """C[z] = act(alpha*A[z] B[z]^T + bias) + residual on tensor cores; see include/vcr_b200.h."""
    L = lib()
    ldc = c.stride(-2) if c is not None else 0
    ldr = residual.stride(-2) if residual is not None else 0
    outp = h if h is not None else ht
    L.check(L.vcr_gemm_tc(
        a.ptr, a.ld, a.rows, a.cols, a.plane_stride, *a_off,
        b.ptr, b.ld, b.rows, b.cols, b.plane_stride, *b_off,
        M, N, K, nbo, nbi, TC_MODES[a.mode], float(alpha), bias.data_ptr() if bias is not None else None,
        int(act), float(slope),
        c.data_ptr() if c is not None else None, ldc, *c_strides,
        residual.data_ptr() if residual is not None else None, ldr, *r_strides,
        h.ptr if h is not None else None, h.ld if h is not None else 0,
        h.plane_stride if h is not None else 0, *h_strides, h_split,
        ht.ptr if ht is not None else None, ht.ld if ht is not None else 0,
        ht.plane_stride if ht is not None else 0, *ht_strides,
        outp.planes if outp is not None else 1, _stream(a.buf)), "vcr_gemm_tc")


def set_gemm_pair(policy):
    """CTA-pair (tcgen05 cta_group::2) policy of the h3 GEMMs: False / 0 never, True / 1 always, "auto" / 2 (default).
    Returns the previous policy code.  Results are bit-identical under every setting."""
    code = 2 if policy == "auto" else int(policy)
    return lib().vcr_set_gemm_pair(code)


def set_flash_warps(nwq: int) -> int:
    """Softmax warps per TMEM lane quarter of the flash attention kernel (2 or 4); returns the previous setting."""
    return lib().vcr_set_flash_warps(int(nwq))


def flash_attn_tc(q: Operand, k: Operand, vt: Operand, out: Operand, B, H, Nq, Nk, dk, scale, keep=None, lse=None):
    """softmax(Q K^T * scale) V per (batch, head) on tensor cores, nothing of size Nq x Nk touches HBM."""
    L = lib()
    L.check(L.vcr_flash_attn_tc(q.ptr, q.ld, q.plane_stride, k.ptr, k.ld, k.plane_stride, vt.ptr, vt.ld,
                                vt.plane_stride, B, H, Nq, Nk, dk, TC_MODES[q.mode], float(scale),
                                keep.data_ptr() if keep is not None else None, out.ptr, out.ld, out.plane_stride,
                                lse.data_ptr() if lse is not None else None, _stream(q.buf)), "vcr_flash_attn_tc")
    return out


def attn_colsum_tc(q: Operand, k: Operand, B, H, Nq, Nk, dk, scale):
    """Column sums over heads and queries of softmax(Q K^T * scale) -> [B, Nk]; scores never reach HBM."""
    assert q.mode == "h3" and k.mode == "h3"
    dev = q.buf.device
    L = lib()
    wsb = L.vcr_attn_colsum_workspace_bytes(B, H, Nq, Nk)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    out = torch.empty((B, Nk), dtype=_F32, device=dev)
    L.check(L.vcr_attn_colsum_tc(q.ptr, q.ld, q.plane_stride, k.ptr, k.ld, k.plane_stride, B, H, Nq, Nk, dk,
                                 float(scale), out.data_ptr(), ws.data_ptr(), wsb, _stream(q.buf)), "vcr_attn_colsum_tc")
    return out


def layernorm_operand(x: torch.Tensor, a, b, eps, mode, out: Operand | None = None) -> Operand:
    _chk(x, "x")
    M, D, ldx = _rows(x)
    if out is None:
        out = Operand.empty(M, D, mode, x.device)
    assert out.rows == M and out.cols == D and out.mode == mode
    L = lib()
    L.check(L.vcr_layernorm_operand(x.data_ptr(), ldx, a.data_ptr(), b.data_ptr(), float(eps), M, D, out.ptr,
                                    out.ld, out.plane_stride, out.planes, int(mode == "bf16"), _stream(x)),
            "vcr_layernorm_operand")
    return out


def softmax_operand(S: torch.Tensor, n: int, mode, keep=None, rows_per_batch=0) -> Operand:
    """S fp32 [rows, ld] (first n columns valid) -> probabilities in operand format [rows, n]."""
    rows, _, ld = _rows(S)
    out = Operand.empty(rows, n, mode, S.device)
    L = lib()
    L.check(L.vcr_softmax_operand(S.data_ptr(), ld, rows, n, keep.data_ptr() if keep is not None else None,
                                  rows_per_batch, out.ptr, out.ld, out.plane_stride, out.planes,
                                  int(mode == "bf16"), _stream(S)), "vcr_softmax_operand")
    return out


def colsum_softmax(S: torch.Tensor, n: int, B: int, fused: bool = True):
    """column sums per batch of softmax(S) over rows, S fp32 [B*rows_per_batch, ld] left untouched.
    fused: one kernel that reads S from HBM once (rows staged in shared memory); else row_lse + colsum_softmax."""
    rows, _, ld = _rows(S)
    dev = S.device
    if fused:
        L = lib()
        wsb = L.vcr_softmax_colsum_workspace_bytes(B, rows // B, ld, n)
        if wsb > 0:
            out = torch.empty((B, n), dtype=_F32, device=dev)
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            L.check(L.vcr_softmax_colsum(S.data_ptr(), ld, B, rows // B, n, out.data_ptr(), ws.data_ptr(), wsb,
                                         _stream(S)), "vcr_softmax_colsum")
            return out
    rmax = torch.empty(rows, dtype=_F32, device=dev)
    rsum = torch.empty(rows, dtype=_F32, device=dev)
    out = torch.empty((B, n), dtype=_F32, device=dev)
    L = lib()
    st = _stream(S)
    L.check(L.vcr_row_lse(S.data_ptr(), ld, rows, n, None, 0, rmax.data_ptr(), rsum.data_ptr(), st), "vcr_row_lse")
    wsb = L.vcr_colsum_workspace_bytes(B, n)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    L.check(L.vcr_colsum_softmax(S.data_ptr(), ld, B, rows // B, n, rmax.data_ptr(), rsum.data_ptr(), out.data_ptr(),
                                 ws.data_ptr(), wsb, st), "vcr_colsum_softmax")
    return out


# --------------------------------------------------------------------------------------------------
# LPDNet pieces
# --------------------------------------------------------------------------------------------------

def conv3_act(xyz: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, slope: float):
    """xyz [B,3,N] -> token-major [B,N,Cout]."""
    _chk(xyz, "xyz")
    xyz = xyz.contiguous()
    B, _, N = xyz.shape
    Cout = w.shape[0]
    out = torch.empty((B, N, Cout), dtype=_F32, device=xyz.device)
    L = lib()
    L.check(L.vcr_conv3_act(xyz.data_ptr(), w.data_ptr(), bias.data_ptr(), B, N, Cout, float(slope),
                            out.data_ptr(), Cout, _stream(xyz)), "vcr_conv3_act")
    return out


def edgeconv_dg(pq: torch.Tensor, idx: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, slope: float,
                x1: torch.Tensor, x2: torch.Tensor):
    """pq [B,N,256], idx int32 [B,N,20]; writes x1, x2 (row views [B,N,128])."""
    B, N, _ = pq.shape
    _, _, ldpq = _rows(pq)
    _, _, ld1 = _rows(x1)
    _, _, ld2 = _rows(x2)
    L = lib()
    L.check(L.vcr_edgeconv_dg(pq.data_ptr(), ldpq, idx.data_ptr(), idx.shape[2], N, B * N, w2.data_ptr(),
                              b2.data_ptr(), float(slope), x1.data_ptr(), ld1, x2.data_ptr(), ld2, _stream(pq)),
            "vcr_edgeconv_dg")


def edgeconv_dg_tc(pq: torch.Tensor, idx: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, slope: float,
                   x1: torch.Tensor, x2: torch.Tensor, mode: str, op1: "Operand | None" = None, op2: "Operand | None" = None,
                   z: torch.Tensor | None = None):
    """edgeconv_dg on tcgen05 tensor cores (csrc/edgeconv_tc.cu); mode in TC_MODES.
    op1 / op2: optional "h3" Operand views (same buffer) that also receive x1 / x2 in operand format.
    z: optional contiguous [B*N*20, 128] that receives the per-edge convDG2 pre-activations x2 is the max of."""
    B, N, _ = pq.shape
    _, _, ldpq = _rows(pq)
    _, _, ld1 = _rows(x1)
    _, _, ld2 = _rows(x2)
    if op1 is not None:
        assert op1.mode == "h3" and op2.mode == "h3" and op1.ld == op2.ld and op1.plane_stride == op2.plane_stride
    if z is not None:
        _chk(z, "z")
        assert z.is_contiguous() and tuple(z.shape) == (B * N * idx.shape[2], 128)
    L = lib()
    L.check(L.vcr_edgeconv_dg_tc(pq.data_ptr(), ldpq, idx.data_ptr(), idx.shape[2], N, B * N, w2.data_ptr(),
                                 b2.data_ptr(), float(slope), TC_MODES[mode], x1.data_ptr(), ld1, x2.data_ptr(), ld2,
                                 op1.ptr if op1 is not None else None, op2.ptr if op2 is not None else None,
                                 op1.ld if op1 is not None else 0, op1.plane_stride if op1 is not None else 0,
                                 z.data_ptr() if z is not None else None, _stream(pq)), "vcr_edgeconv_dg_tc")


def gather_max(p: torch.Tensor, q: torch.Tensor, idx: torch.Tensor, slope: float, out: torch.Tensor,
               op: "Operand | None" = None):
    """out[b,n,:] = act(max_k p[b, idx[b,n,k], :] + q[b,n,:]); p, q, out are [B,N,C] row views.
    op: optional "h3" Operand view that also receives the rows in operand format."""
    B, N, C = p.shape
    _, _, ldp = _rows(p)
    _, _, ldq = _rows(q)
    _, _, ldo = _rows(out)
    L = lib()
    L.check(L.vcr_gather_max(p.data_ptr(), ldp, q.data_ptr(), ldq, idx.data_ptr(), idx.shape[2], N, B * N, C,
                             float(slope), out.data_ptr(), ldo, op.ptr if op is not None else None,
                             op.ld if op is not None else 0, op.plane_stride if op is not None else 0, _stream(p)),
            "vcr_gather_max")


def lpd_point_mlp(xyz: torch.Tensor, w1, b1, w2, b2, slope: float, want_h1: bool = True, want_operand: bool = False):
    """conv1_lpd + conv2_lpd (model/lpdnet_model.py:111-112) in one kernel: xyz [B,3,N] -> (h1 [B,N,64] or None, h2 [B,N,64],
    "h3" Operand of h2 or None); bit-identical to conv3_act + gemm."""
    _chk(xyz, "xyz")
    xyz = xyz.contiguous()
    B, _, N = xyz.shape
    assert tuple(w1.shape) == (64, 3) and tuple(w2.shape) == (64, 64)
    dev = xyz.device
    h1 = torch.empty((B, N, 64), dtype=_F32, device=dev) if want_h1 else None
    h2 = torch.empty((B, N, 64), dtype=_F32, device=dev)
    op = Operand.empty(B * N, 64, "h3", dev) if want_operand else None
    L = lib()
    L.check(L.vcr_lpd_point_mlp(xyz.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), B, N, float(slope),
                                h1.data_ptr() if want_h1 else None, h2.data_ptr(), op.ptr if op is not None else None,
                                op.ld if op is not None else 0, op.plane_stride if op is not None else 0, _stream(xyz)),
            "vcr_lpd_point_mlp")
    return h1, h2, op


def edge_max(e: torch.Tensor, k: int, out: torch.Tensor):
    """e [T*k, C] contiguous -> out [T, C] row view: max over the k edges of each point."""
    _chk(e, "e")
    T, C, ldo = _rows(out)
    assert e.is_contiguous() and e.shape == (T * k, C)
    L = lib()
    L.check(L.vcr_edge_max(e.data_ptr(), k, T, C, out.data_ptr(), ldo, _stream(e)), "vcr_edge_max")
    return out


# --------------------------------------------------------------------------------------------------
# LPDNet backward pieces (csrc/train.cu)
# --------------------------------------------------------------------------------------------------

def wgrad(g: torch.Tensor, x: torch.Tensor, want_bias: bool = True):
    """g [M,N], x [M,K] row views -> (dW [N,K] = g^T x, db [N] = column sums of g)."""
    _chk(g, "g"); _chk(x, "x")
    M, N, ldg = _rows(g)
    M2, K, ldx = _rows(x)
    assert M == M2, (M, M2)
    dW = torch.zeros((N, K), dtype=_F32, device=g.device)
    db = torch.zeros((N,), dtype=_F32, device=g.device) if want_bias else None
    L = lib()
    L.check(L.vcr_wgrad_f32(g.data_ptr(), ldg, x.data_ptr(), ldx, M, N, K, dW.data_ptr(), K,
                            db.data_ptr() if want_bias else None, _stream(g)), "vcr_wgrad_f32")
    return dW, db


def act_bwd(gy: torch.Tensor, y: torch.Tensor, slope: float, scale_bits: torch.Tensor | None = None):
    """gz = gy * LeakyReLU'(z), y = the saved post-activation output (row views).
    scale_bits: absmax_bits(gy); gz is then also scaled by 2^-floor(log2 max|gy|)."""
    _chk(gy, "gy"); _chk(y, "y")
    M, N, ldg = _rows(gy)
    M2, N2, ldy = _rows(y)
    assert (M, N) == (M2, N2)
    if scale_bits is not None:
        _chk(scale_bits, "scale_bits", torch.int32)
    gz = torch.empty(gy.shape, dtype=_F32, device=gy.device)
    L = lib()
    L.check(L.vcr_act_bwd(gy.data_ptr(), ldg, y.data_ptr(), ldy, M, N, float(slope),
                          scale_bits.data_ptr() if scale_bits is not None else None, gz.data_ptr(), N, _stream(gy)),
            "vcr_act_bwd")
    return gz


def absmax_bits(x: torch.Tensor):
    """x contiguous fp32 -> int32 [1]: the bit pattern of max|x| (on the device, no host synchronisation)."""
    _chk(x, "x")
    assert x.is_contiguous()
    bits = torch.zeros(1, dtype=torch.int32, device=x.device)
    L = lib()
    L.check(L.vcr_absmax_bits(x.data_ptr(), x.numel(), bits.data_ptr(), _stream(x)), "vcr_absmax_bits")
    return bits


def pow2_inverse(bits: torch.Tensor):
    """absmax_bits output -> fp32 [1]: the inverse of the scale act_bwd applies for it."""
    _chk(bits, "bits", torch.int32)
    out = torch.empty(1, dtype=_F32, device=bits.device)
    L = lib()
    L.check(L.vcr_pow2_inverse(bits.data_ptr(), out.data_ptr(), _stream(bits)), "vcr_pow2_inverse")
    return out


def gather_max_bwd(p: torch.Tensor, q: torch.Tensor, idx: torch.Tensor, slope: float, gout: torch.Tensor,
                   gp: torch.Tensor, gq: torch.Tensor):
    """backward of gather_max: gq written, gp (pre-zeroed) accumulated; all [B,N,C] row views."""
    B, N, C = p.shape
    _, _, ldp = _rows(p); _, _, ldq = _rows(q); _, _, ldo = _rows(gout)
    _, _, ldgp = _rows(gp); _, _, ldgq = _rows(gq)
    L = lib()
    L.check(L.vcr_gather_max_bwd(p.data_ptr(), ldp, q.data_ptr(), ldq, idx.data_ptr(), idx.shape[2], N, B * N, C,
                                 float(slope), gout.data_ptr(), ldo, gp.data_ptr(), ldgp, gq.data_ptr(), ldgq,
                                 _stream(p)), "vcr_gather_max_bwd")


def edge_gather_act(pq: torch.Tensor, idx: torch.Tensor, slope: float):
    """pq [B,N,2C] = [P|Q], idx int32 [B,N,k] -> e1 [B*N*k, C] = act(P[nbr] + Q[centre])."""
    _chk(pq, "pq")
    B, N, C2 = pq.shape
    C = C2 // 2
    k = idx.shape[2]
    _, _, ldpq = _rows(pq)
    E = torch.empty((B * N * k, C), dtype=_F32, device=pq.device)
    L = lib()
    L.check(L.vcr_edge_gather_act(pq.data_ptr(), ldpq, idx.data_ptr(), k, N, B * N, C, float(slope), E.data_ptr(),
                                  _stream(pq)), "vcr_edge_gather_act")
    return E


def edge_max_bwd_(z: torch.Tensor, gx: torch.Tensor, k: int, slope: float):
    """z [T*k, C] (convDG2 pre-activations) -> in place g_z; gx [T, C] row view."""
    _chk(z, "z"); _chk(gx, "gx")
    T, C, ldg = _rows(gx)
    assert z.is_contiguous() and z.shape == (T * k, C)
    L = lib()
    L.check(L.vcr_edge_max_bwd(z.data_ptr(), gx.data_ptr(), ldg, k, T, C, float(slope), _stream(z)), "vcr_edge_max_bwd")
    return z


def edge_bwd_scatter(e: torch.Tensor, ge: torch.Tensor, gx1: torch.Tensor, idx: torch.Tensor, slope: float):
    """e, ge [T*k, C]; gx1 [T, C] row view; idx int32 [B,N,k] -> gPQ [B,N,2C] = [gP | gQ]."""
    B, N, k = idx.shape
    T, C, ldg = _rows(gx1)
    assert T == B * N and e.is_contiguous() and ge.is_contiguous()
    gpq = torch.zeros((B, N, 2 * C), dtype=_F32, device=e.device)
    L = lib()
    L.check(L.vcr_edge_bwd_scatter(e.data_ptr(), ge.data_ptr(), gx1.data_ptr(), ldg, idx.data_ptr(), k, N, T, C,
                                   float(slope), gpq.data_ptr(), 2 * C, _stream(e)), "vcr_edge_bwd_scatter")
    return gpq


# --------------------------------------------------------------------------------------------------
# Transformer pieces
# --------------------------------------------------------------------------------------------------

def layernorm(x: torch.Tensor, a: torch.Tensor, b: torch.Tensor, eps: float = 1e-6, residual=None, out=None):
    _chk(x, "x")
    M, D, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, dtype=_F32, device=x.device)
    _, _, ldo = _rows(out)
    ldr = 0
    if residual is not None:
        _, _, ldr = _rows(residual)
    L = lib()
    L.check(L.vcr_layernorm(x.data_ptr(), ldx, a.data_ptr(), b.data_ptr(), float(eps), M, D,
                            residual.data_ptr() if residual is not None else None, ldr,
                            out.data_ptr(), ldo, _stream(x)), "vcr_layernorm")
    return out


def layernorm_head(x: torch.Tensor, a: torch.Tensor, b: torch.Tensor, eps: float = 1e-6, residual=None, want_out=True):
    """layernorm(x) (+ residual) -> (out fp32 or None, its "h3" Operand copy, its squared row norms), one kernel.
    want_out=False skips the fp32 store: the VCP head only reads the operand copy and the norms."""
    _chk(x, "x")
    M, D, ldx = _rows(x)
    out = torch.empty(x.shape, dtype=_F32, device=x.device) if want_out else None
    op = Operand.empty(M, D, "h3", x.device)
    sq = torch.empty(x.shape[:-1], dtype=_F32, device=x.device)
    ldr = 0
    if residual is not None:
        _, _, ldr = _rows(residual)
    L = lib()
    L.check(L.vcr_layernorm_head(x.data_ptr(), ldx, a.data_ptr(), b.data_ptr(), float(eps), M, D,
                                 residual.data_ptr() if residual is not None else None, ldr,
                                 out.data_ptr() if out is not None else None, D,
                                 op.ptr, op.ld, op.plane_stride, sq.data_ptr(), _stream(x)), "vcr_layernorm_head")
    return out, op, sq


def softmax_rows_(S: torch.Tensor, keep: torch.Tensor | None = None, rows_per_batch: int = 0):
    rows, n, ld = _rows(S)
    L = lib()
    L.check(L.vcr_softmax_rows(S.data_ptr(), ld, rows, n, keep.data_ptr() if keep is not None else None,
                               rows_per_batch, _stream(S)), "vcr_softmax_rows")
    return S


def colsum(P: torch.Tensor, B: int, out=None):
    """P [B*rows_per_batch, n] -> [B, n] column sums per batch."""
    rows, n, ld = _rows(P)
    if out is None:
        out = torch.empty((B, n), dtype=_F32, device=P.device)
    L = lib()
    wsb = L.vcr_colsum_workspace_bytes(B, n)
    ws = torch.empty(wsb, dtype=torch.uint8, device=P.device)
    L.check(L.vcr_colsum(P.data_ptr(), ld, B, rows // B, n, out.data_ptr(), ws.data_ptr(), wsb, _stream(P)),
            "vcr_colsum")
    return out


# vcr_topk_select: one CTA per row up to 16 384 values, one cluster of up to 16 such CTAs beyond
TOPK_MAX_N = 16 * 16384


def topk_select(vals: torch.Tensor, K: int, want_idx=True, want_mask=False):
    _chk(vals, "vals")
    vals = vals.contiguous()
    B, n = vals.shape
    idx = torch.empty((B, K), dtype=torch.int32, device=vals.device) if want_idx else None
    mask = torch.empty((B, n), dtype=torch.uint8, device=vals.device) if want_mask else None
    L = lib()
    rc = L.vcr_topk_select(vals.data_ptr(), B, n, K, idx.data_ptr() if want_idx else None,
                           mask.data_ptr() if want_mask else None, _stream(vals))
    if rc != 0 and n > TOPK_MAX_N:
        raise RuntimeError(f"vcr_topk_select failed: {rc}: top-K selection takes at most {TOPK_MAX_N} values per row, "
                           f"got {n}")
    L.check(rc, "vcr_topk_select")
    return idx, mask


def attention_f32(q, k, v, B, h, Nq, Nk, dk, scale, out, keep=None, colsum_out=False, max_ws_bytes=1 << 31):
    """softmax(q k^T * scale) v per (batch, head) in fp32 (model/transformer.py:13-55).

    q/k/v: (tensor, ld, batch_stride, head_stride) tuples addressing [B, h, N, dk] inside fused
    projection buffers; out likewise.  Scores are materialised per chunk of batches (fp32 mode);
    the tensor-core modes use the flash kernel instead.  ``keep`` uint8 [B,Nk] masks keys.
    Returns the per-batch column sums of the probabilities when ``colsum_out``."""
    qt, qld, qsb, qsh = q
    kt, kld, ksb, ksh = k
    vt, vld, vsb, vsh = v
    ot, old, osb, osh = out
    dev = qt.device
    ldS = (Nk + 3) // 4 * 4                  # rows padded to 16 bytes: float4 row starts for any key count
    per_b = h * Nq * ldS * 4
    cb = max(1, min(B, max_ws_bytes // per_b))
    S = torch.empty((cb, h, Nq, ldS), dtype=_F32, device=dev)
    csum = torch.empty((B, Nk), dtype=_F32, device=dev) if colsum_out else None
    esz = 4
    for b0 in range(0, B, cb):
        nb = min(cb, B - b0)
        off = lambda t, sb: t.data_ptr() + b0 * sb * esz
        L = lib()
        st = _stream(qt)
        L.check(L.vcr_gemm_f32(off(qt, qsb), qld, qsb, qsh, off(kt, ksb), kld, ksb, ksh, 0,
                               S.data_ptr(), ldS, h * Nq * ldS, Nq * ldS, None, None, 0, 0, 0,
                               Nq, Nk, dk, nb, h, float(scale), 0, 0.0, st), "vcr_gemm_f32(QK)")
        Sv = S[:nb].view(nb * h * Nq, ldS)[:, :Nk]
        kp = keep[b0:b0 + nb] if keep is not None else None
        softmax_rows_(Sv, kp, h * Nq)
        if colsum_out:
            colsum(Sv, nb, out=csum[b0:b0 + nb])
        L.check(L.vcr_gemm_f32(S.data_ptr(), ldS, h * Nq * ldS, Nq * ldS, off(vt, vsb), vld, vsb, vsh, 1,
                               off(ot, osb), old, osb, osh, None, None, 0, 0, 0,
                               Nq, dk, Nk, nb, h, 1.0, 0, 0.0, st), "vcr_gemm_f32(PV)")
    return csum


# --------------------------------------------------------------------------------------------------
# VCP head
# --------------------------------------------------------------------------------------------------

def sqnorm_rows(x: torch.Tensor):
    rows, D, ld = _rows(x)
    out = torch.empty(x.shape[:-1], dtype=_F32, device=x.device)
    L = lib()
    L.check(L.vcr_sqnorm_rows(x.data_ptr(), ld, rows, D, out.data_ptr(), _stream(x)), "vcr_sqnorm_rows")
    return out


def pair_dots(s_tok: torch.Tensor, t_tok: torch.Tensor):
    """s_tok [B,Ns,D], t_tok [B,Nt,D] (contiguous) -> dot [B,Ns,ld] with ld = Nt rounded up to 4."""
    B, Ns, D = s_tok.shape
    Nt = t_tok.shape[1]
    ld = (Nt + 3) // 4 * 4
    dot = torch.empty((B, Ns, ld), dtype=_F32, device=s_tok.device)
    bgemm(s_tok, D, Ns * D, 0, t_tok, D, Nt * D, 0, 0, dot, ld, Ns * ld, 0, Ns, Nt, D, B, 1)
    return dot, ld


def softcorr_rows(dot, ld, Ns, Nt, xx, yy, tgt=None, mode=0):
    B = dot.shape[0]
    dev = dot.device
    L = lib()
    corr = best_i = best_v = None
    if mode == 0:
        corr = torch.empty((B, 3, Ns), dtype=_F32, device=dev)
    elif mode == 2:
        best_i = torch.empty((B, Ns), dtype=torch.int32, device=dev)
        best_v = torch.empty((B, Ns), dtype=_F32, device=dev)
    L.check(L.vcr_softcorr_rows(dot.data_ptr(), ld, B, Ns, Nt, xx.data_ptr(), yy.data_ptr(),
                                tgt.data_ptr() if tgt is not None else None, mode,
                                corr.data_ptr() if corr is not None else None,
                                best_i.data_ptr() if best_i is not None else None,
                                best_v.data_ptr() if best_v is not None else None, _stream(dot)),
            "vcr_softcorr_rows")
    return corr, best_i, best_v


def softcorr_tc(s_op: "Operand", t_op: "Operand", xx, yy, tgt_xyz: torch.Tensor, B: int, Ns: int, Nt: int, D: int):
    """Fused getCopairALL on tensor cores (csrc/softcorr_tc.cu): corr [B,3,Ns]; no [Ns,Nt] matrix in HBM."""
    assert s_op.mode == "h3" and t_op.mode == "h3" and s_op.rows == B * Ns and t_op.rows == B * Nt
    tgt_xyz = tgt_xyz.contiguous()
    _chk(tgt_xyz, "tgt")
    corr = torch.empty((B, 3, Ns), dtype=_F32, device=tgt_xyz.device)
    L = lib()
    L.check(L.vcr_softcorr_tc(s_op.ptr, s_op.ld, s_op.plane_stride, t_op.ptr, t_op.ld, t_op.plane_stride,
                              xx.data_ptr(), yy.data_ptr(), tgt_xyz.data_ptr(), B, Ns, Nt, D, corr.data_ptr(),
                              _stream(tgt_xyz)), "vcr_softcorr_tc")
    return corr


def softcorr_best_tc(s_op: "Operand", t_op: "Operand", xx, yy, B: int, Ns: int, Nt: int, D: int):
    """Fused getCopair statistics on tensor cores: (argmax_j pd_ij int32 [B,Ns], max_j softmax_j(pd_ij) [B,Ns])."""
    assert s_op.mode == "h3" and t_op.mode == "h3" and s_op.rows == B * Ns and t_op.rows == B * Nt
    dev = xx.device
    best_i = torch.empty((B, Ns), dtype=torch.int32, device=dev)
    best_v = torch.empty((B, Ns), dtype=_F32, device=dev)
    L = lib()
    L.check(L.vcr_softcorr_best_tc(s_op.ptr, s_op.ld, s_op.plane_stride, t_op.ptr, t_op.ld, t_op.plane_stride,
                                   xx.data_ptr(), yy.data_ptr(), B, Ns, Nt, D, best_i.data_ptr(), best_v.data_ptr(),
                                   _stream(xx)), "vcr_softcorr_best_tc")
    return best_i, best_v


def negdist_(dot, ld, Ns, Nt, xx, yy):
    B = dot.shape[0]
    L = lib()
    L.check(L.vcr_negdist(dot.data_ptr(), ld, B, Ns, Nt, xx.data_ptr(), yy.data_ptr(), _stream(dot)), "vcr_negdist")
    return dot


def rowsum_colsoftmax(pd, ld, Ns, Nt):
    B = pd.shape[0]
    out = torch.empty((B, Ns), dtype=_F32, device=pd.device)
    L = lib()
    ws = torch.empty(L.vcr_rowsum_colsoftmax_workspace_bytes(B, Nt) // 4, dtype=_F32, device=pd.device)
    L.check(L.vcr_rowsum_colsoftmax(pd.data_ptr(), ld, B, Ns, Nt, out.data_ptr(), ws.data_ptr(), ws.numel() * 4,
                                    _stream(pd)), "vcr_rowsum_colsoftmax")
    return out


def select_stats(dot: torch.Tensor, ld: int, Ns: int, Nt: int, xx: torch.Tensor, yy: torch.Tensor):
    """selectCom's two statistics from the score products dot [B,Ns,ld] (untouched): (row_stat [B,Ns], col_stat [B,Nt])."""
    B = dot.shape[0]
    dev = dot.device
    L = lib()
    if Ns == Nt:                              # one [2, B, N] buffer: the caller can rank both statistics in one launch
        both = torch.empty((2, B, Ns), dtype=_F32, device=dev)
        row_stat, col_stat = both[0], both[1]
    else:
        row_stat = torch.empty((B, Ns), dtype=_F32, device=dev)
        col_stat = torch.empty((B, Nt), dtype=_F32, device=dev)
    wsb = L.vcr_select_stats_workspace_bytes(B, Ns, Nt)
    ws = torch.empty(wsb // 4, dtype=_F32, device=dev)
    L.check(L.vcr_select_stats(dot.data_ptr(), ld, B, Ns, Nt, xx.data_ptr(), yy.data_ptr(), row_stat.data_ptr(),
                               col_stat.data_ptr(), ws.data_ptr(), wsb, _stream(dot)), "vcr_select_stats")
    return row_stat, col_stat


def select_stats_tc(s_op: "Operand", t_op: "Operand", xx, yy, B: int, Ns: int, Nt: int, D: int):
    """selectCom's two statistics on tensor cores from "h3" operands (csrc/softcorr_tc.cu), no [Ns,Nt] matrix in HBM:
    (row_stat [B,Ns], col_stat [B,Nt]), laid out as select_stats lays them out."""
    assert s_op.mode == "h3" and t_op.mode == "h3" and s_op.rows == B * Ns and t_op.rows == B * Nt
    dev = xx.device
    if Ns == Nt:                              # one [2, B, N] buffer: the caller can rank both statistics in one launch
        both = torch.empty((2, B, Ns), dtype=_F32, device=dev)
        row_stat, col_stat = both[0], both[1]
    else:
        row_stat = torch.empty((B, Ns), dtype=_F32, device=dev)
        col_stat = torch.empty((B, Nt), dtype=_F32, device=dev)
    L = lib()
    wsb = L.vcr_select_stats_tc_workspace_bytes(B, Ns, Nt)
    ws = torch.empty(wsb // 4, dtype=_F32, device=dev)
    L.check(L.vcr_select_stats_tc(s_op.ptr, s_op.ld, s_op.plane_stride, t_op.ptr, t_op.ld, t_op.plane_stride,
                                  xx.data_ptr(), yy.data_ptr(), B, Ns, Nt, D, row_stat.data_ptr(), col_stat.data_ptr(),
                                  ws.data_ptr(), wsb, _stream(xx)), "vcr_select_stats_tc")
    return row_stat, col_stat


def gather_operand_rows(op: "Operand", sq: torch.Tensor, idx: torch.Tensor, B: int, Nin: int):
    """Rows idx [B,K] of an "h3" Operand [B*Nin, C] and of its squared norms sq [B,Nin] -> (Operand [B*K, C], sq [B,K])."""
    assert op.mode == "h3" and op.rows == B * Nin
    K = idx.shape[1]
    out = Operand.empty(B * K, op.cols, "h3", sq.device)
    sq_out = torch.empty((B, K), dtype=_F32, device=sq.device)
    L = lib()
    L.check(L.vcr_gather_operand_rows(op.ptr, op.ld, op.plane_stride, B, Nin, idx.data_ptr(), K, op.cols, out.ptr, out.ld,
                                      out.plane_stride, sq.data_ptr(), sq_out.data_ptr(), _stream(sq)),
            "vcr_gather_operand_rows")
    return out, sq_out


def gather_rows(x_tok: torch.Tensor, idx: torch.Tensor):
    """x_tok [B,N,C] -> [B,K,C] rows idx[b,:]."""
    B, N, C = x_tok.shape
    _, _, ld = _rows(x_tok)
    K = idx.shape[1]
    out = torch.empty((B, K, C), dtype=_F32, device=x_tok.device)
    L = lib()
    L.check(L.vcr_gather_rows(x_tok.data_ptr(), ld, B, N, idx.data_ptr(), K, C, out.data_ptr(), C, _stream(x_tok)),
            "vcr_gather_rows")
    return out


def gather_cols(x: torch.Tensor, idx: torch.Tensor):
    """x [B,C,N] channel-major -> [B,C,K]."""
    x = x.contiguous()
    B, C, N = x.shape
    K = idx.shape[1]
    out = torch.empty((B, C, K), dtype=_F32, device=x.device)
    L = lib()
    L.check(L.vcr_gather_cols(x.data_ptr(), B, C, N, idx.data_ptr(), K, out.data_ptr(), _stream(x)), "vcr_gather_cols")
    return out


def copair_gather(src_xyz, tgt_xyz, keep, best_i):
    """src_k[b,:,r] = src[b,:,keep[b,r]];  corr_k[b,:,r] = tgt[b,:,best_i[b,keep[b,r]]]
    (model/vcrnet_model.py:300-331 with tgtK == 1)."""
    src_xyz, tgt_xyz = src_xyz.contiguous(), tgt_xyz.contiguous()
    B, _, Ns = src_xyz.shape
    Nt = tgt_xyz.shape[2]
    K = keep.shape[1]
    so = torch.empty((B, 3, K), dtype=_F32, device=src_xyz.device)
    co = torch.empty((B, 3, K), dtype=_F32, device=src_xyz.device)
    L = lib()
    L.check(L.vcr_copair_gather(src_xyz.data_ptr(), tgt_xyz.data_ptr(), B, Ns, Nt, keep.data_ptr(),
                                best_i.data_ptr(), K, so.data_ptr(), co.data_ptr(), _stream(src_xyz)),
            "vcr_copair_gather")
    return so, co


# --------------------------------------------------------------------------------------------------
# SVD head / pose algebra / layout
# --------------------------------------------------------------------------------------------------

def svd_head(src: torch.Tensor, corr: torch.Tensor, want_H=False):
    _chk(src, "src"); _chk(corr, "src_corr")
    src, corr = src.contiguous(), corr.contiguous()
    B, _, M = src.shape
    dev = src.device
    R = torch.empty((B, 3, 3), dtype=_F32, device=dev)
    t = torch.empty((B, 3), dtype=_F32, device=dev)
    Rb = torch.empty((B, 3, 3), dtype=_F32, device=dev)
    tb = torch.empty((B, 3), dtype=_F32, device=dev)
    H = torch.empty((B, 3, 3), dtype=_F32, device=dev) if want_H else None
    L = lib()
    L.check(L.vcr_svd_head(src.data_ptr(), corr.data_ptr(), B, M, R.data_ptr(), t.data_ptr(), Rb.data_ptr(),
                           tb.data_ptr(), H.data_ptr() if want_H else None, _stream(src)), "vcr_svd_head")
    return (R, t, Rb, tb, H) if want_H else (R, t, Rb, tb)


def rigid_apply(pc: torch.Tensor, R: torch.Tensor, t: torch.Tensor):
    _chk(pc, "point_cloud")
    pc, R, t = pc.contiguous(), R.contiguous(), t.contiguous()
    B, _, N = pc.shape
    out = torch.empty_like(pc)
    L = lib()
    L.check(L.vcr_rigid_apply(pc.data_ptr(), R.data_ptr(), t.data_ptr(), B, N, out.data_ptr(), _stream(pc)),
            "vcr_rigid_apply")
    return out


def pose_compose_(R_i, t_i, R_f, t_f):
    L = lib()
    L.check(L.vcr_pose_compose(R_i.data_ptr(), t_i.data_ptr(), R_f.data_ptr(), t_f.data_ptr(), R_f.shape[0],
                               _stream(R_f)), "vcr_pose_compose")


def pose_inverse(R, t):
    Ri, ti = torch.empty_like(R), torch.empty_like(t)
    L = lib()
    L.check(L.vcr_pose_inverse(R.data_ptr(), t.data_ptr(), Ri.data_ptr(), ti.data_ptr(), R.shape[0], _stream(R)),
            "vcr_pose_inverse")
    return Ri, ti


def icp_nearest(src: torch.Tensor, dst: torch.Tensor, err_slot: torch.Tensor, want_idx=False):
    """src [B,3,Ns], dst [B,3,Nt] -> corr [B,3,Ns]; err_slot (float64, 1 element, zero) accumulates sum(best pd)."""
    _chk(src, "src"); _chk(dst, "dst")
    src, dst = src.contiguous(), dst.contiguous()
    B, _, Ns = src.shape
    Nt = dst.shape[2]
    assert err_slot.dtype == torch.float64 and err_slot.is_cuda
    corr = torch.empty_like(src)
    idx = torch.empty((B, Ns), dtype=torch.int32, device=src.device) if want_idx else None
    L = lib()
    L.check(L.vcr_icp_nearest(src.data_ptr(), dst.data_ptr(), B, Ns, Nt, corr.data_ptr(),
                              idx.data_ptr() if want_idx else None, err_slot.data_ptr(), _stream(src)), "vcr_icp_nearest")
    return (corr, idx) if want_idx else corr


def icp_state(device):
    n = lib().vcr_icp_state_bytes()
    return torch.zeros((n + 7) // 8, dtype=torch.int64, device=device)


def icp_advance_(src: torch.Tensor, R: torch.Tensor, t: torch.Tensor, err_slot: torch.Tensor, tolerance: float,
                 state: torch.Tensor):
    """In place: src <- R src + t unless the device-side state says the loop has converged; updates the state."""
    assert src.is_contiguous()
    B, _, Ns = src.shape
    L = lib()
    L.check(L.vcr_icp_advance(src.data_ptr(), R.data_ptr(), t.data_ptr(), B, Ns, err_slot.data_ptr(), float(tolerance),
                              state.data_ptr(), _stream(src)), "vcr_icp_advance")


def transpose_batched(x: torch.Tensor):
    """[nb,R,C] contiguous -> [nb,C,R] contiguous (module-boundary layout change)."""
    _chk(x, "x")
    x = x.contiguous()
    nb, R, C = x.shape
    out = torch.empty((nb, C, R), dtype=_F32, device=x.device)
    L = lib()
    L.check(L.vcr_transpose(x.data_ptr(), out.data_ptr(), nb, R, C, C, R, R * C, R * C, _stream(x)), "vcr_transpose")
    return out
