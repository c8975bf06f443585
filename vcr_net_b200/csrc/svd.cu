// SVD (Procrustes) head and rigid-pose helpers.
//   vcr_svd_head      : reference model/vcrnet_model.py:356-399 (SVDHead.forward) + the inverse pose of
//                       VCRNet.forward (:515-516), one warp per pair, no host round trip (the
//                       reference loops torch.svd/torch.det in Python with B+1 host syncs).
//   vcr_rigid_apply   : util/util.py:91-96 transform_point_cloud (rotation-matrix branch)
//   vcr_pose_compose  : model/vcrnet_model.py:35-38  R_f <- R_i R_f ; t_f <- R_i t_f + t_i
//   vcr_pose_inverse  : model/vcrnet_model.py:40-41
// Means, the 3x3 covariance and the SVD are carried in FP64 (the inputs are FP32; this only removes
// our own rounding, it is 9 numbers per pair).  The SVD is a one-sided (Hestenes) Jacobi iteration
// kept in registers: rotate column pairs of H until orthogonal; singular values = column norms,
// sorted descending so that the reflection fix flips the SMALLEST one (vcrnet_model.py:353-354,383-386).
// HBM roofline: 2*4*3*M bytes per pair, latency-bound at B <= a few thousand (report us/pair).
#include "common.cuh"

namespace {

struct M3 { double m[3][3]; };

__host__ __device__ __forceinline__ void jacobi_svd3(const M3& H, M3& U, double S[3], M3& V) {
    double a[3][3], v[3][3];   // a[c] = column c of the working matrix, v[c] = column c of V
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r) { a[c][r] = H.m[r][c]; v[c][r] = (r == c) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            const double alpha = a[p][0] * a[p][0] + a[p][1] * a[p][1] + a[p][2] * a[p][2];
            const double beta = a[q][0] * a[q][0] + a[q][1] * a[q][1] + a[q][2] * a[q][2];
            const double gamma = a[p][0] * a[q][0] + a[p][1] * a[q][1] + a[p][2] * a[q][2];
            const double lim = 1e-15 * sqrt(alpha * beta);
            if (fabs(gamma) > lim && gamma != 0.0) {
                off = fmax(off, fabs(gamma) / fmax(sqrt(alpha * beta), 1e-300));
                const double zeta = (beta - alpha) / (2.0 * gamma);
                const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const double ap = a[p][r], aq = a[q][r];
                    a[p][r] = c * ap - s * aq; a[q][r] = s * ap + c * aq;
                    const double vp = v[p][r], vq = v[q][r];
                    v[p][r] = c * vp - s * vq; v[q][r] = s * vp + c * vq;
                }
            }
        }
        if (off < 1e-14) break;
    }
    double sv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) sv[c] = sqrt(a[c][0] * a[c][0] + a[c][1] * a[c][1] + a[c][2] * a[c][2]);
    // sort columns by singular value, descending (3-element network)
    auto swp = [&](int i, int j) {
        if (sv[i] < sv[j]) {
            double t = sv[i]; sv[i] = sv[j]; sv[j] = t;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                t = a[i][r]; a[i][r] = a[j][r]; a[j][r] = t;
                t = v[i][r]; v[i][r] = v[j][r]; v[j][r] = t;
            }
        }
    };
    swp(0, 1); swp(0, 2); swp(1, 2);
    double u[3][3];
    // u0
    const double tiny = 1e-300;
    {
        const double inv = 1.0 / fmax(sv[0], tiny);
        u[0][0] = a[0][0] * inv; u[0][1] = a[0][1] * inv; u[0][2] = a[0][2] * inv;
        if (sv[0] < tiny) { u[0][0] = 1.0; u[0][1] = 0.0; u[0][2] = 0.0; }
    }
    // u1: a1 made orthogonal to u0 (it already is up to rounding), or any unit vector orthogonal to u0
    {
        double w0 = a[1][0], w1 = a[1][1], w2 = a[1][2];
        const double d = w0 * u[0][0] + w1 * u[0][1] + w2 * u[0][2];
        w0 -= d * u[0][0]; w1 -= d * u[0][1]; w2 -= d * u[0][2];
        double n = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
        if (n <= 1e-14 * fmax(sv[0], tiny)) {
            // rank <= 1: pick the coordinate axis least aligned with u0
            const double ax = fabs(u[0][0]), ay = fabs(u[0][1]), az = fabs(u[0][2]);
            double e0 = 0, e1 = 0, e2 = 0;
            if (ax <= ay && ax <= az) e0 = 1; else if (ay <= az) e1 = 1; else e2 = 1;
            const double dd = e0 * u[0][0] + e1 * u[0][1] + e2 * u[0][2];
            w0 = e0 - dd * u[0][0]; w1 = e1 - dd * u[0][1]; w2 = e2 - dd * u[0][2];
            n = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
        }
        u[1][0] = w0 / n; u[1][1] = w1 / n; u[1][2] = w2 / n;
    }
    // u2 = +-(u0 x u1), sign following a2 when it carries information
    {
        double c0 = u[0][1] * u[1][2] - u[0][2] * u[1][1];
        double c1 = u[0][2] * u[1][0] - u[0][0] * u[1][2];
        double c2 = u[0][0] * u[1][1] - u[0][1] * u[1][0];
        const double d = c0 * a[2][0] + c1 * a[2][1] + c2 * a[2][2];
        const double sgn = d < 0.0 ? -1.0 : 1.0;
        u[2][0] = sgn * c0; u[2][1] = sgn * c1; u[2][2] = sgn * c2;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        S[c] = sv[c];
#pragma unroll
        for (int r = 0; r < 3; ++r) { U.m[r][c] = u[c][r]; V.m[r][c] = v[c][r]; }
    }
}

__host__ __device__ __forceinline__ double det3(const M3& A) {
    return A.m[0][0] * (A.m[1][1] * A.m[2][2] - A.m[1][2] * A.m[2][1]) -
           A.m[0][1] * (A.m[1][0] * A.m[2][2] - A.m[1][2] * A.m[2][0]) +
           A.m[0][2] * (A.m[1][0] * A.m[2][1] - A.m[1][1] * A.m[2][0]);
}

__global__ void svd_head_kernel(const float* __restrict__ src, const float* __restrict__ corr, int B, int M,
                                float* __restrict__ R_ab, float* __restrict__ t_ab,
                                float* __restrict__ R_ba, float* __restrict__ t_ba,
                                float* __restrict__ H_out, const int* __restrict__ mlen) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    const float* s = src + (size_t)b * 3 * M;
    const float* c = corr + (size_t)b * 3 * M;
    const int ld = M;                                  // row stride of the pair's three coordinate rows
    M = vcr_item_len(mlen, b, ld, 1);                  // points of the pair: all of them, or its length in a ragged batch
    double ms[3] = {0, 0, 0}, mc[3] = {0, 0, 0};
    for (int n = lane; n < M; n += 32) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { ms[a] += s[a * ld + n]; mc[a] += c[a * ld + n]; }
    }
    float fs[3], fc[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        ms[a] = warp_sum(ms[a]) / M; mc[a] = warp_sum(mc[a]) / M;
        fs[a] = (float)ms[a]; fc[a] = (float)mc[a];           // the reference's means are fp32
    }
    double h[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int n = lane; n < M; n += 32) {
        float sv[3], cv[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) { sv[a] = s[a * ld + n] - fs[a]; cv[a] = c[a * ld + n] - fc[a]; }
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) h[i][j] += (double)sv[i] * (double)cv[j];
    }
    M3 H;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) H.m[i][j] = warp_sum(h[i][j]);
    // every lane now holds the same H; all lanes run the (tiny) SVD redundantly, lane 0 writes
    M3 U, V;
    double S[3];
    jacobi_svd3(H, U, S, V);
    M3 R;
    auto vut = [&]() {
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j)
                R.m[i][j] = V.m[i][0] * U.m[j][0] + V.m[i][1] * U.m[j][1] + V.m[i][2] * U.m[j][2];
    };
    vut();
    if (det3(R) < 0.0) {
        V.m[0][2] = -V.m[0][2]; V.m[1][2] = -V.m[1][2]; V.m[2][2] = -V.m[2][2];
        vut();
    }
    if (lane == 0) {
        float Rf[3][3], tf[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) Rf[i][j] = (float)R.m[i][j];
            tf[i] = (float)(-(R.m[i][0] * fs[0] + R.m[i][1] * fs[1] + R.m[i][2] * fs[2]) + fc[i]);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                R_ab[b * 9 + i * 3 + j] = Rf[i][j];
                if (R_ba) R_ba[b * 9 + i * 3 + j] = Rf[j][i];
                if (H_out) H_out[b * 9 + i * 3 + j] = (float)H.m[i][j];
            }
            t_ab[b * 3 + i] = tf[i];
        }
        if (t_ba) {
#pragma unroll
            for (int i = 0; i < 3; ++i)
                t_ba[b * 3 + i] = -(Rf[0][i] * tf[0] + Rf[1][i] * tf[1] + Rf[2][i] * tf[2]);
        }
    }
}

__global__ void rigid_apply_kernel(const float* __restrict__ pc, const float* __restrict__ R,
                                   const float* __restrict__ t, int N, float* __restrict__ out) {
    const int b = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float* p = pc + (size_t)b * 3 * N;
    const float* r = R + b * 9;
    const float x = p[n], y = p[N + n], z = p[2 * N + n];
    float* o = out + (size_t)b * 3 * N;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float acc = r[i * 3 + 0] * x;
        acc = fmaf(r[i * 3 + 1], y, acc);
        acc = fmaf(r[i * 3 + 2], z, acc);
        o[i * N + n] = acc + t[b * 3 + i];
    }
}

__global__ void pose_compose_kernel(const float* __restrict__ Ri, const float* __restrict__ ti,
                                    float* __restrict__ Rf, float* __restrict__ tf, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float r[9], f[9], tt[3];
    for (int i = 0; i < 9; ++i) { r[i] = Ri[b * 9 + i]; f[i] = Rf[b * 9 + i]; }
    for (int i = 0; i < 3; ++i) tt[i] = tf[b * 3 + i];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            float acc = r[i * 3 + 0] * f[0 * 3 + j];
            acc = fmaf(r[i * 3 + 1], f[1 * 3 + j], acc);
            acc = fmaf(r[i * 3 + 2], f[2 * 3 + j], acc);
            Rf[b * 9 + i * 3 + j] = acc;
        }
        float acc = r[i * 3 + 0] * tt[0];
        acc = fmaf(r[i * 3 + 1], tt[1], acc);
        acc = fmaf(r[i * 3 + 2], tt[2], acc);
        tf[b * 3 + i] = acc + ti[b * 3 + i];
    }
}

__global__ void pose_inverse_kernel(const float* __restrict__ R, const float* __restrict__ t,
                                    float* __restrict__ Rinv, float* __restrict__ tinv, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float r[9], tt[3];
    for (int i = 0; i < 9; ++i) r[i] = R[b * 9 + i];
    for (int i = 0; i < 3; ++i) tt[i] = t[b * 3 + i];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) Rinv[b * 9 + i * 3 + j] = r[j * 3 + i];
        float acc = r[0 * 3 + i] * tt[0];
        acc = fmaf(r[1 * 3 + i], tt[1], acc);
        acc = fmaf(r[2 * 3 + i], tt[2], acc);
        tinv[b * 3 + i] = -acc;
    }
}

}  // namespace

// Host-side entry to the SAME Jacobi routine the kernel runs (CPU unit tests of the device math).
// H, U, V: row-major 3x3 doubles; S: 3 doubles (descending).  H = U diag(S) V^T.
VCR_API int vcr_host_svd3(const double* H, double* U, double* S, double* V) {
    M3 h, u, v;
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) h.m[i][j] = H[i * 3 + j];
    jacobi_svd3(h, u, S, v);
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { U[i * 3 + j] = u.m[i][j]; V[i * 3 + j] = v.m[i][j]; }
    return VCR_OK;
}

// src, corr: [B,3,M].  R_ab [B,3,3], t_ab [B,3] required; R_ba, t_ba, H_out optional (may be NULL).
VCR_API int vcr_svd_head(const float* src, const float* corr, int B, int M, float* R_ab, float* t_ab,
                         float* R_ba, float* t_ba, float* H_out, cudaStream_t stream) {
    VCR_REQUIRE(src && corr && R_ab && t_ab && B > 0 && M > 0);
    const int wpb = 4;
    svd_head_kernel<<<vcr_cdiv(B, wpb), wpb * 32, 0, stream>>>(src, corr, B, M, R_ab, t_ab, R_ba, t_ba, H_out, nullptr);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

// Ragged batch: pair b has m[b] points (clamped to [1, M]) in its M columns; the result equals vcr_svd_head on the pair's
// first m[b] columns alone (the fp64 sums run over the same points in the same order).
VCR_API int vcr_svd_head_ragged(const float* src, const float* corr, const int* m, int B, int M, float* R_ab, float* t_ab,
                                float* R_ba, float* t_ba, float* H_out, cudaStream_t stream) {
    VCR_REQUIRE(src && corr && m && R_ab && t_ab && B > 0 && M > 0);
    const int wpb = 4;
    svd_head_kernel<<<vcr_cdiv(B, wpb), wpb * 32, 0, stream>>>(src, corr, B, M, R_ab, t_ab, R_ba, t_ba, H_out, m);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

__global__ void zero_padding_kernel(const float* x, const int* __restrict__ len, int C, int N, int lo,
                                    float* out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (n >= N) return;
    const bool real = n < vcr_item_len(len, b, N, lo);
    for (int c = 0; c < C; ++c) {
        const size_t o = ((size_t)b * C + c) * N + n;
        out[o] = real ? x[o] : 0.f;
    }
}

// out[b,c,n] = x[b,c,n] for n < len[b] (clamped to [lo, N]), 0 past it: a ragged batch [B,C,N] with its padding zeroed.
VCR_API int vcr_zero_padding(const float* x, const int* len, int B, int C, int N, int lo, float* out, cudaStream_t stream) {
    VCR_REQUIRE(x && len && out && B > 0 && C > 0 && N > 0 && B <= 65535 && lo >= 1);
    zero_padding_kernel<<<dim3(vcr_cdiv(N, 256), B), 256, 0, stream>>>(x, len, C, N, lo, out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_rigid_apply(const float* pc, const float* R, const float* t, int B, int N, float* out,
                            cudaStream_t stream) {
    VCR_REQUIRE(pc && R && t && out && B > 0 && N > 0 && B <= 65535);
    dim3 g(vcr_cdiv(N, 256), B);
    rigid_apply_kernel<<<g, 256, 0, stream>>>(pc, R, t, N, out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_pose_compose(const float* R_i, const float* t_i, float* R_f, float* t_f, int B, cudaStream_t stream) {
    VCR_REQUIRE(R_i && t_i && R_f && t_f && B > 0);
    pose_compose_kernel<<<vcr_cdiv(B, 128), 128, 0, stream>>>(R_i, t_i, R_f, t_f, B);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_pose_inverse(const float* R, const float* t, float* R_inv, float* t_inv, int B, cudaStream_t stream) {
    VCR_REQUIRE(R && t && R_inv && t_inv && B > 0);
    pose_inverse_kernel<<<vcr_cdiv(B, 128), 128, 0, stream>>>(R, t, R_inv, t_inv, B);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
