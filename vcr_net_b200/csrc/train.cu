// Backward kernels of the LPDNet embedding (BASELINE config 3: LPD pre-training forward + backward,
// reference model/lpdnet_model.py:103-137 differentiated by autograd, driven by :149-229).
//
// The forward pass factors every EdgeConv as per-point GEMMs + gathers (DESIGN.md section 4); the backward
// pass mirrors that factoring, all in fp32:
//   vcr_wgrad_f32          dW[n,k] += sum_m G[m,n] X[m,k], db[n] += sum_m G[m,n]   (weight / bias gradients of
//                          every 1x1 conv: a tall-skinny A^T B product, split over M across CTAs)
//   vcr_act_bwd            gz = gy * LeakyReLU'(z), from the saved post-activation output (y > 0 <=> z > 0), optionally
//                          times the power of two vcr_absmax_bits picked for gy (see LPDNetTrainFn.backward)
//   vcr_gather_max_bwd     backward of x3 = act(max_k P3[nbr] + Q3)  (convSN1 + max, :130-132)
//   vcr_edge_gather_act    e1 = act(P1[nbr] + Q1), materialised [T*k, C]   (convDG1 output, :123)
//   vcr_edge_max_bwd       route g_x2 to the arg-max edge of z2 = convDG2(e1) per (point, channel)   (:125-126)
//   vcr_edge_bwd_scatter   g_e1 (+ the x1 = max_k e1 route, :124) through LeakyReLU' to gQ1 (sum over edges) and
//                          gP1 (atomic scatter to the neighbour rows)
// The dense products between them (data gradients g.W, z2 = e1.W2^T) reuse vcr_gemm_f32.
// Roofline: all of these stream [T*k, C] fp32 edge tensors once: HBM bound (4*k*C bytes per point and tensor).
#include "common.cuh"

namespace {

constexpr int WG_T = 64;      // dW tile edge
constexpr int WG_MC = 32;     // rows of G / X per smem step

__global__ void __launch_bounds__(256)
wgrad_kernel(const float* __restrict__ G, int ldg, const float* __restrict__ X, int ldx, long long M, int N, int K,
             long long rows_per_split, float* __restrict__ dW, int lddw, float* __restrict__ db) {
    __shared__ __align__(16) float Gs[WG_MC][WG_T + 4];
    __shared__ __align__(16) float Xs[WG_MC][WG_T + 4];
    const int tid = threadIdx.x, tn = tid >> 4, tk = tid & 15;
    const int n0 = blockIdx.y * WG_T, k0 = blockIdx.x * WG_T;
    const long long m_begin = (long long)blockIdx.z * rows_per_split;
    const long long m_end = min(M, m_begin + rows_per_split);
    float acc[4][4];
    float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (long long m0 = m_begin; m0 < m_end; m0 += WG_MC) {
        __syncthreads();
        for (int e = tid; e < WG_MC * WG_T; e += 256) {
            const int r = e >> 6, c = e & 63;
            const long long m = m0 + r;
            Gs[r][c] = (m < m_end && n0 + c < N) ? G[m * ldg + n0 + c] : 0.f;
            Xs[r][c] = (m < m_end && k0 + c < K) ? X[m * ldx + k0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < WG_MC; ++r) {
            const float4 g = *reinterpret_cast<const float4*>(&Gs[r][tn * 4]);
            const float4 x = *reinterpret_cast<const float4*>(&Xs[r][tk * 4]);
            const float gv[4] = {g.x, g.y, g.z, g.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                bsum[i] += gv[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(gv[i], xv[j], acc[i][j]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + tn * 4 + i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tk * 4 + j;
            if (k < K) atomicAdd(dW + (size_t)n * lddw + k, acc[i][j]);
        }
        if (db && blockIdx.x == 0 && tk == 0) atomicAdd(db + n, bsum[i]);
    }
}

// 2^-floor(log2 m) (inverse = false) or 2^floor(log2 m) (inverse = true) for the bit pattern of m = max|g| >= 0, with
// floor(log2 m) clamped to [-126, 126] so that both are normal floats (m = 0 gives 2^126 / 2^-126)
__device__ __forceinline__ float pow2_scale(int mbits, bool inverse) {
    const int e = min(max((mbits >> 23) & 255, 1), 253);
    return __int_as_float((inverse ? e : 254 - e) << 23);
}

__global__ void absmax_kernel(const float* __restrict__ x, long long n, int* __restrict__ mbits) {
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(x[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(mbits, __float_as_int(m));     // non-negative floats order like their bits
}

__global__ void act_bwd_kernel(const float* __restrict__ gy, int ldg, const float* __restrict__ y, int ldy,
                               long long rows, int cols, float slope, const int* __restrict__ mbits,
                               float* __restrict__ gz, int ldz) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * cols) return;
    const long long r = e / cols;
    const int c = (int)(e - r * cols);
    const float g = mbits ? gy[r * ldg + c] * pow2_scale(*mbits, false) : gy[r * ldg + c];
    gz[r * ldz + c] = g * (y[r * ldy + c] > 0.f ? 1.f : slope);
}

__global__ void pow2_inverse_kernel(const int* __restrict__ mbits, float* __restrict__ out) {
    *out = pow2_scale(*mbits, true);
}

// x3[pt,c] = act(max_k P[nbr_k,c] + Q[pt,c]):  gQ[pt,c] = g * act'(s),  gP[argmax nbr, c] += the same
__global__ void gather_max_bwd_kernel(const float* __restrict__ P, int ldp, const float* __restrict__ Q, int ldq,
                                      const int* __restrict__ idx, int k, int N, long long total_pts, int C, float slope,
                                      const float* __restrict__ gout, int ldgo, float* __restrict__ gP, int ldgp,
                                      float* __restrict__ gQ, int ldgq) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total_pts * C) return;
    const long long pt = e / C;
    const int c = (int)(e - pt * C);
    const long long cloud0 = (pt / N) * N;
    const int* ip = idx + pt * k;
    float best = -INFINITY;
    int bj = 0;
    for (int kk = 0; kk < k; ++kk) {
        const int j = ip[kk];
        const float v = P[(cloud0 + j) * ldp + c];
        if (v > best) { best = v; bj = j; }
    }
    const float s = best + Q[pt * ldq + c];
    const float g = gout[pt * ldgo + c] * (s > 0.f ? 1.f : slope);
    gQ[pt * ldgq + c] = g;
    atomicAdd(gP + (cloud0 + bj) * ldgp + c, g);
}

__global__ void edge_gather_act_kernel(const float* __restrict__ PQ, int ldpq, const int* __restrict__ idx, int k, int N,
                                       long long total_pts, int C, float slope, float* __restrict__ E) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int C4 = C >> 2;
    if (e >= total_pts * k * C4) return;
    const long long edge = e / C4;
    const int c4 = (int)(e - edge * C4);
    const long long pt = edge / k;
    const long long cloud0 = (pt / N) * N;
    const int j = idx[edge];
    const float4 a = *reinterpret_cast<const float4*>(PQ + (cloud0 + j) * ldpq + c4 * 4);
    const float4 q = *reinterpret_cast<const float4*>(PQ + pt * ldpq + C + c4 * 4);
    float4 v;
    v.x = leaky(a.x + q.x, slope); v.y = leaky(a.y + q.y, slope);
    v.z = leaky(a.z + q.z, slope); v.w = leaky(a.w + q.w, slope);
    *reinterpret_cast<float4*>(E + edge * C + c4 * 4) = v;
}

// Z [T,k,C] holds z2 = convDG2(e1) (bias included) on entry and g_z2 on exit
__global__ void edge_max_bwd_kernel(float* __restrict__ Z, const float* __restrict__ gx, int ldgx, int k,
                                    long long total_pts, int C, float slope) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total_pts * C) return;
    const long long pt = e / C;
    const int c = (int)(e - pt * C);
    float* z = Z + pt * k * C + c;
    float best = -INFINITY;
    int bk = 0;
    for (int kk = 0; kk < k; ++kk) {
        const float v = z[(size_t)kk * C];
        if (v > best) { best = v; bk = kk; }
    }
    const float g = gx[pt * ldgx + c] * (best > 0.f ? 1.f : slope);
    for (int kk = 0; kk < k; ++kk) z[(size_t)kk * C] = kk == bk ? g : 0.f;
}

__global__ void edge_bwd_scatter_kernel(const float* __restrict__ E, const float* __restrict__ gE,
                                        const float* __restrict__ gx1, int ldgx, const int* __restrict__ idx, int k, int N,
                                        long long total_pts, int C, float slope, float* __restrict__ gPQ, int ldg) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total_pts * C) return;
    const long long pt = e / C;
    const int c = (int)(e - pt * C);
    const long long cloud0 = (pt / N) * N;
    const float* er = E + pt * k * C + c;
    const float* gr = gE + pt * k * C + c;
    float best = -INFINITY;
    int bk = 0;
    for (int kk = 0; kk < k; ++kk) {
        const float v = er[(size_t)kk * C];
        if (v > best) { best = v; bk = kk; }
    }
    const float g1 = gx1[pt * ldgx + c];
    float sumq = 0.f;
    for (int kk = 0; kk < k; ++kk) {
        const float ge = gr[(size_t)kk * C] + (kk == bk ? g1 : 0.f);
        const float gs = ge * (er[(size_t)kk * C] > 0.f ? 1.f : slope);
        sumq += gs;
        atomicAdd(gPQ + (cloud0 + idx[pt * k + kk]) * ldg + c, gs);
    }
    gPQ[pt * ldg + C + c] = sumq;
}

inline unsigned blocks_for(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

// dW [N, K] (row stride lddw) += G[M,N]^T X[M,K];  db [N] += column sums of G (db may be NULL).  Accumulates with
// fp32 atomics: the caller zero-initialises dW / db.
VCR_API int vcr_wgrad_f32(const float* G, int ldg, const float* X, int ldx, long long M, int N, int K, float* dW,
                          int lddw, float* db, cudaStream_t stream) {
    VCR_REQUIRE(G && X && dW && M > 0 && N > 0 && K > 0);
    const int tiles = vcr_cdiv(N, WG_T) * vcr_cdiv(K, WG_T);
    long long splits = (4LL * 148 + tiles - 1) / tiles;
    const long long max_splits = (M + 4 * WG_MC - 1) / (4 * WG_MC);
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    if (splits > 65535) splits = 65535;
    long long rps = (M + splits - 1) / splits;
    rps = (rps + WG_MC - 1) / WG_MC * WG_MC;
    splits = (M + rps - 1) / rps;
    dim3 grid(vcr_cdiv(K, WG_T), vcr_cdiv(N, WG_T), (unsigned)splits);
    wgrad_kernel<<<grid, 256, 0, stream>>>(G, ldg, X, ldx, M, N, K, rps, dW, lddw, db);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_act_bwd(const float* gy, int ldg, const float* y, int ldy, long long rows, int cols, float slope,
                        const int* scale_bits, float* gz, int ldz, cudaStream_t stream) {
    VCR_REQUIRE(gy && y && gz && rows > 0 && cols > 0);
    act_bwd_kernel<<<blocks_for(rows * cols, 256), 256, 0, stream>>>(gy, ldg, y, ldy, rows, cols, slope, scale_bits, gz,
                                                                    ldz);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_absmax_bits(const float* x, long long n, int* bits, cudaStream_t stream) {
    VCR_REQUIRE(x && bits && n > 0);
    const long long want = (n + 255) / 256;
    absmax_kernel<<<(unsigned)(want < 4 * 148 ? want : 4 * 148), 256, 0, stream>>>(x, n, bits);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_pow2_inverse(const int* bits, float* out, cudaStream_t stream) {
    VCR_REQUIRE(bits && out);
    pow2_inverse_kernel<<<1, 1, 0, stream>>>(bits, out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_gather_max_bwd(const float* P, int ldp, const float* Q, int ldq, const int* idx, int k, int N,
                               long long total_pts, int C, float slope, const float* gout, int ldgo, float* gP,
                               int ldgp, float* gQ, int ldgq, cudaStream_t stream) {
    VCR_REQUIRE(P && Q && idx && gout && gP && gQ && k >= 1 && N > 0 && total_pts > 0 && C > 0);
    gather_max_bwd_kernel<<<blocks_for(total_pts * C, 256), 256, 0, stream>>>(P, ldp, Q, ldq, idx, k, N, total_pts, C,
                                                                             slope, gout, ldgo, gP, ldgp, gQ, ldgq);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_edge_gather_act(const float* PQ, int ldpq, const int* idx, int k, int N, long long total_pts, int C,
                                float slope, float* E, cudaStream_t stream) {
    VCR_REQUIRE(PQ && idx && E && k >= 1 && N > 0 && total_pts > 0 && C > 0 && C % 4 == 0 && ldpq % 4 == 0);
    edge_gather_act_kernel<<<blocks_for(total_pts * k * (C / 4), 256), 256, 0, stream>>>(PQ, ldpq, idx, k, N, total_pts,
                                                                                        C, slope, E);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_edge_max_bwd(float* Z, const float* gx, int ldgx, int k, long long total_pts, int C, float slope,
                             cudaStream_t stream) {
    VCR_REQUIRE(Z && gx && k >= 1 && total_pts > 0 && C > 0);
    edge_max_bwd_kernel<<<blocks_for(total_pts * C, 256), 256, 0, stream>>>(Z, gx, ldgx, k, total_pts, C, slope);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_edge_bwd_scatter(const float* E, const float* gE, const float* gx1, int ldgx, const int* idx, int k,
                                 int N, long long total_pts, int C, float slope, float* gPQ, int ldg,
                                 cudaStream_t stream) {
    VCR_REQUIRE(E && gE && gx1 && idx && gPQ && k >= 1 && N > 0 && total_pts > 0 && C > 0);
    edge_bwd_scatter_kernel<<<blocks_for(total_pts * C, 256), 256, 0, stream>>>(E, gE, gx1, ldgx, idx, k, N, total_pts, C,
                                                                               slope, gPQ, ldg);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
