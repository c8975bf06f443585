// k-nearest-neighbour graph kernel (SURVEY.md K1a/K1b; reference util/util.py:143-160).
//
// Canonical arithmetic (identical, op for op, to oracle/canon.c so indices are bit-exact):
//   xx_i   = fma chain over d = 0..D-1 of x_i[d]*x_i[d], start 0
//   dot_ij = fma chain over d = 0..D-1 of x_i[d]*x_j[d], start 0
//   pd_ij  = (-xx_j - (-2*dot_ij)) - xx_i           (reference op order, util/util.py:157-158)
//   neighbours(i) = ranks 1..k of pd_i* sorted descending, ties -> lower j
// The N x N matrix is never materialised.  A CTA owns 32 query rows and walks the cloud in chunks of
// 512 candidates:
//   compute  an SGEMM-style 32 x 512 tile, 8 x 8 register block per thread, the d-chain of every
//            (i, j) pair kept in ONE accumulator in d order (bit-exact by construction), operands
//            staged through shared memory 16 dims at a time (cp.async when rows are 16-byte aligned);
//   select   the 32 x 512 distance tile goes through shared memory to a warp-per-query selection:
//            a lane holds 16 distances in registers, a threshold tau (first chunk: the (k+1)-th largest
//            of the 32 lane maxima, found by a shuffle bitonic sort; later chunks: the running
//            (k+1)-th best) filters the chunk down to ~30 survivors with ballot/popc compaction, the
//            survivors are sorted 32 at a time as 64-bit (ordered-float, ~index) keys by shuffle
//            bitonic networks and bitonic-merged into the running top-32 list (one entry per lane).
//            Nothing is dropped unless k+1 seen elements are strictly better, so ranks 0..k are exact.
//
// Roofline: bytes = 4*D*N in + 4*k*N out per cloud (candidate chunks are re-read from L2 by the N/32
// CTAs of a cloud), flops = 2*D*N^2 (+ ~N^2 select steps): FP32-FMA bound at D = 64, selection
// (issue) bound at D = 3 -- DESIGN.md section 4.
#include <atomic>
#include "tc_common.cuh"

namespace {

constexpr int TQ = 32;        // queries per CTA
constexpr int TC = 512;       // candidates per chunk
constexpr int NT = 256;       // threads per CTA: 8 warps = 4 query groups x 2 candidate groups, 8 x 8 per thread
constexpr int RPL = TC / 32;  // distances per lane in the selection phase

// xx[b*N + i] = fma chain.  One thread per point.
template <bool TOKEN_MAJOR>
__global__ void knn_sqnorm_kernel(const float* __restrict__ x, int D, int N, float* __restrict__ xx) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float* xb = x + (size_t)b * D * N;
    float acc = 0.f;
    for (int d = 0; d < D; ++d) {
        const float v = TOKEN_MAJOR ? xb[(size_t)i * D + d] : xb[(size_t)d * N + i];
        acc = fmaf(v, v, acc);
    }
    xx[(size_t)b * N + i] = acc;
}

// order-preserving float -> uint32 (-0.0 canonicalised to +0.0 first: the two compare equal)
__device__ __forceinline__ uint32_t okey(float v) {
    const uint32_t b = __float_as_uint(v + 0.f);
    return b ^ (uint32_t)(((int32_t)b >> 31) | 0x80000000);
}
__device__ __forceinline__ float okey_inv(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}
// 64-bit key (ordered value, ~index) kept as two 32-bit registers; keys of real entries are distinct
struct Key { uint32_t hi, lo; };
__device__ __forceinline__ Key key_xchg(Key v, int j, bool take_max) {
    Key o;
    o.hi = __shfl_xor_sync(0xffffffffu, v.hi, j);
    o.lo = __shfl_xor_sync(0xffffffffu, v.lo, j);
    const bool gt = v.hi > o.hi || (v.hi == o.hi && v.lo > o.lo);
    return gt == take_max ? v : o;
}
__device__ __forceinline__ Key key_max(Key a, Key b) {
    return (a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo)) ? a : b;
}

// W independent 32-lane bitonic sorts (descending), one element per lane each
template <int W>
__device__ __forceinline__ void sort32_desc(Key (&v)[W], int lane) {
#pragma unroll
    for (int ks = 2; ks <= 32; ks <<= 1) {
#pragma unroll
        for (int j = ks >> 1; j > 0; j >>= 1) {
            const bool take_max = ((lane & j) == 0) == ((lane & ks) == 0);
#pragma unroll
            for (int w = 0; w < W; ++w) v[w] = key_xchg(v[w], j, take_max);
        }
    }
}
template <int W>
__device__ __forceinline__ void sort32_desc_f(float (&v)[W], int lane) {
#pragma unroll
    for (int ks = 2; ks <= 32; ks <<= 1) {
#pragma unroll
        for (int j = ks >> 1; j > 0; j >>= 1) {
            const bool take_max = ((lane & j) == 0) == ((lane & ks) == 0);
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const float o = __shfl_xor_sync(0xffffffffu, v[w], j);
                v[w] = take_max ? fmaxf(v[w], o) : fminf(v[w], o);
            }
        }
    }
}
// run, add: descending-sorted 32-lists -> run = top 32 of the union, descending
template <int W>
__device__ __forceinline__ void merge32_desc(Key (&run)[W], const Key (&add)[W], int lane) {
#pragma unroll
    for (int w = 0; w < W; ++w) {
        Key o;
        o.hi = __shfl_sync(0xffffffffu, add[w].hi, 31 - lane);
        o.lo = __shfl_sync(0xffffffffu, add[w].lo, 31 - lane);
        run[w] = key_max(run[w], o);
    }
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const bool take_max = (lane & j) == 0;
#pragma unroll
        for (int w = 0; w < W; ++w) run[w] = key_xchg(run[w], j, take_max);
    }
}

// Filter W queries' chunk rows (TCN candidates each, row stride LDD floats) by their thresholds into buf (capacity
// CAP keys), then sort the survivors 32 at a time and merge them into the running lists.  Returns false, leaving
// `run` untouched, if buf would overflow (impossible for W == 1 when CAP >= TCN).
template <int W, int TCN, int LDD, int CAP>
__device__ __forceinline__ bool filter_merge_t(const float* drows, const float (&tau)[W], Key (&run)[W], uint2* buf,
                                               int j0, int lane) {
    constexpr int RP = TCN / 32;
    const uint32_t lt = (1u << lane) - 1u;
    int cnt[W], off[W];
    int base = 0;
    __syncwarp();
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const float* dr = drows + w * LDD + lane;
        float v[RP];
#pragma unroll
        for (int r = 0; r < RP; ++r) v[r] = dr[r * 32];
        off[w] = base;
        int n = base;
        // branch-free: the ballots are independent, only the running offset chains
#pragma unroll
        for (int r = 0; r < RP; ++r) {
            const bool p = v[r] >= tau[w];
            const uint32_t bal = __ballot_sync(0xffffffffu, p);
            const int pos = n + __popc(bal & lt);
            if (p && pos < CAP) buf[pos] = make_uint2(~(uint32_t)(j0 + r * 32 + lane), okey(v[r]));
            n += __popc(bal);
        }
        cnt[w] = n - base;
        base = n;
    }
    __syncwarp();
    if (base > CAP) return false;
    int rounds = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) rounds = max(rounds, (cnt[w] + 31) >> 5);
    for (int r = 0; r < rounds; ++r) {
        Key e[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int p = r * 32 + lane;
            const uint2 t = p < cnt[w] ? buf[off[w] + p] : make_uint2(0u, 0u);
            e[w].lo = t.x; e[w].hi = t.y;
        }
        sort32_desc<W>(e, lane);
        merge32_desc<W>(run, e, lane);
    }
    return true;
}
template <int W>
__device__ __forceinline__ bool filter_merge(const float* drows, const float (&tau)[W], Key (&run)[W], uint2* buf,
                                             int j0, int lane) {
    return filter_merge_t<W, TC, TC, TC>(drows, tau, run, buf, j0, lane);
}

// Selection of one 32-query x 512-candidate distance tile: warp w owns queries QW*w .. QW*w+QW-1, `run` holds their
// running top-32 lists (one entry per lane), rank `kk` (0-based) is the threshold rank: nothing is dropped unless kk+1
// seen elements are at least as good, so ranks 0..kk of the final lists are exact.
__device__ __forceinline__ void select_chunk(const float* dist, uint2* surv, Key (&run)[TQ / (NT / 32)], int j0, int kk,
                                             int warp, int lane, bool first) {
    constexpr int QWn = TQ / (NT / 32);
    uint2* buf = surv + (size_t)warp * TC;
    const float* drows = dist + (size_t)(warp * QWn) * TC;
    float tau[QWn];
    if (first) {
        float m[QWn];
#pragma unroll
        for (int w = 0; w < QWn; ++w) {
            const float* dr = drows + w * TC + lane;
            float mm = dr[0];
#pragma unroll
            for (int r = 1; r < RPL; ++r) mm = fmaxf(mm, dr[r * 32]);
            m[w] = mm;
        }
        sort32_desc_f<QWn>(m, lane);
#pragma unroll
        for (int w = 0; w < QWn; ++w) tau[w] = __shfl_sync(0xffffffffu, m[w], kk);
    } else {
#pragma unroll
        for (int w = 0; w < QWn; ++w) tau[w] = okey_inv(__shfl_sync(0xffffffffu, run[w].hi, kk));
    }
    // common case: the survivors of all QW queries fit the warp's buffer and are sorted / merged together
    if (!filter_merge<QWn>(drows, tau, run, buf, j0, lane)) {
        // heavy ties (or an adversarial candidate order): one query at a time, any survivor count fits
#pragma unroll
        for (int w = 0; w < QWn; ++w) {
            float t1[1] = {tau[w]};
            Key r1[1] = {run[w]};
            filter_merge<1>(drows + w * TC, t1, r1, buf, j0, lane);
            run[w] = r1[0];
        }
    }
}

__device__ __forceinline__ void cp_async16(float* dst, const float* src, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int NPEND>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(NPEND) : "memory"); }

// one DCH-dim slab of the chunk's TC candidates (rows j0..) and the CTA's TQ queries (rows q0..) of a token-major cloud
// into Cb [TC][DCP] / Qb [TQ][DCP], as one cp.async group (16-byte pieces; rows / dims past N / D are zero-filled)
template <int DCH, int DCP>
__device__ __forceinline__ void issue_slab(const float* __restrict__ xb, int D, int N, int j0, int q0, int d0,
                                           float* Cb, float* Qb, int tid) {
    constexpr int PPR = DCH / 4;       // 16-byte pieces per row
    constexpr int RPP = 256 / PPR;     // rows covered per pass (NT threads)
    const int part = tid % PPR, r0 = tid / PPR;
    const bool dok = d0 + 4 * part < D;
    const float* src = xb + (size_t)(j0 + r0) * D + d0 + 4 * part;
    float* dst = Cb + r0 * DCP + 4 * part;
#pragma unroll
    for (int n = 0; n < 512 / RPP; ++n) {
        const bool ok = dok && j0 + r0 + n * RPP < N;
        cp_async16(dst + n * RPP * DCP, ok ? src + (size_t)n * RPP * D : xb, ok);
    }
    if (r0 < 32) {
        const bool ok = dok && q0 + r0 < N;
        cp_async16(Qb + r0 * DCP + 4 * part, ok ? xb + (size_t)(q0 + r0) * D + d0 + 4 * part : xb, ok);
    }
    cp_async_commit();
}

constexpr int QW = TQ / (NT / 32);   // queries per warp in the selection phase (4)
constexpr size_t SURV_BYTES = (size_t)(NT / 32) * TC * sizeof(uint2);   // per-warp survivor buffers (alias the operand stage)

template <int DCH>
struct Smem {
    static constexpr int DCP = DCH == 4 ? 12 : DCH + 4;   // row stride (floats): conflict-free LDS.128 across 8 lanes
    static constexpr size_t stage_bytes = (size_t)(TC + TQ) * DCP * sizeof(float);
    static constexpr size_t region0 = stage_bytes > SURV_BYTES ? stage_bytes : SURV_BYTES;
    static constexpr size_t total = region0 + (size_t)TC * sizeof(float) + (size_t)TQ * TC * sizeof(float);
};

// Ragged batches (nlen != null): item b holds nlen[b] real points in its N rows.  Candidates past it are never ranked, and
// a padded query (nlen[b] <= q < N) gets its own index in all k slots, so consumers of the graph stay inside the cloud.
__device__ __forceinline__ void knn_write_self(int32_t* idx32, int64_t* idx64, int b, int N, int k, int q0, int nq, int tid,
                                               int nthreads) {
    for (int e = tid; e < nq * k; e += nthreads) {
        const int q = q0 + e / k;
        const size_t o = ((size_t)b * N + q) * k + e % k;
        if (idx32) idx32[o] = q;
        if (idx64) idx64[o] = (int64_t)q;
    }
}

template <int DCH, bool TOKEN_MAJOR>
__global__ void __launch_bounds__(NT, 2)
knn_select_kernel(const float* __restrict__ x, const float* __restrict__ xx, int D, int N, int k,
                  int32_t* __restrict__ idx32, int64_t* __restrict__ idx64, const int* __restrict__ redo,
                  const int* __restrict__ nlen) {
    // redo != null: this launch only repairs the 32-query groups the tensor-core kernel could not certify
    if (redo != nullptr && redo[blockIdx.y * gridDim.x + blockIdx.x] == 0) return;
    const int Nb = vcr_item_len(nlen, blockIdx.y, N, k + 1);
    if ((int)blockIdx.x * TQ >= Nb) {                     // every query of the CTA is padding
        knn_write_self(idx32, idx64, blockIdx.y, N, k, blockIdx.x * TQ, min(TQ, N - (int)blockIdx.x * TQ), threadIdx.x, NT);
        return;
    }
    using S = Smem<DCH>;
    constexpr int DCP = S::DCP;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Cs = reinterpret_cast<float*>(smem_raw);                       // [TC][DCP]
    float* Qs = Cs + TC * DCP;                                            // [TQ][DCP]
    uint2* surv = reinterpret_cast<uint2*>(smem_raw);                     // [8][TC], aliases Cs/Qs during selection
    float* xxc = reinterpret_cast<float*>(smem_raw + S::region0);         // [TC]
    float* dist = xxc + TC;                                               // [TQ][TC]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int qg = warp & 3, cg = warp >> 2;
    const int b = blockIdx.y, q0 = blockIdx.x * TQ;
    const float* xb = x + (size_t)b * D * N;
    const float* xxb = xx + (size_t)b * N;
    const bool vec = TOKEN_MAJOR && (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);

    Key run[QW];
#pragma unroll
    for (int w = 0; w < QW; ++w) run[w].hi = run[w].lo = 0u;

    for (int j0 = 0; j0 < Nb; j0 += TC) {
        float acc[8][8];
#pragma unroll
        for (int qi = 0; qi < 8; ++qi)
#pragma unroll
            for (int ci = 0; ci < 8; ++ci) acc[qi][ci] = 0.f;

        // Operand slabs (DCH dims of the chunk's candidates + the CTA's queries).  The token-major vector path double-buffers
        // them with cp.async: slab s + 1 streams in while slab s is multiplied; the second buffer aliases the distance tile,
        // which is only live between the end of this loop and the end of the selection (ncu had 29 % of the warp samples
        // in the load-and-wait phase of the single-buffered loop).
        const int nslab = (D + DCH - 1) / DCH;
        __syncthreads();                           // the previous chunk's selection no longer reads region 0 / dist
        if (vec) issue_slab<DCH, DCP>(xb, D, N, j0, q0, 0, Cs, Qs, tid);
        for (int c = tid; c < TC; c += NT) xxc[c] = (j0 + c < N) ? xxb[j0 + c] : 0.f;
        for (int si = 0; si < nslab; ++si) {
            const int d0 = si * DCH;
            const float* Cb = (vec && (si & 1)) ? dist : Cs;
            const float* Qb = Cb + TC * DCP;
            if (vec) {
                if (si + 1 < nslab) {
                    float* Cn = (si & 1) ? Cs : dist;      // last read by slab si - 1, ordered by the trailing barrier
                    issue_slab<DCH, DCP>(xb, D, N, j0, q0, d0 + DCH, Cn, Cn + TC * DCP, tid);
                    cp_async_wait_group<1>();
                } else {
                    cp_async_wait_group<0>();
                }
            } else {
                for (int e = tid; e < (TC + TQ) * DCH; e += NT) {
                    int row, d;
                    if (TOKEN_MAJOR) { row = e / DCH; d = e - row * DCH; }
                    else if (e < TC * DCH) { d = e / TC; row = e - d * TC; }
                    else { const int e2 = e - TC * DCH; d = e2 / TQ; row = TC + e2 - d * TQ; }
                    const int g = row < TC ? j0 + row : q0 + (row - TC);
                    float v = 0.f;
                    if (g < N && d0 + d < D)
                        v = TOKEN_MAJOR ? xb[(size_t)g * D + d0 + d] : xb[(size_t)(d0 + d) * N + g];
                    Cs[row * DCP + d] = v;
                }
            }
            __syncthreads();

            const float* qrow = Qb + (qg * 8) * DCP;
            const float* crow = Cb + (cg * 256 + lane) * DCP;
            if (j0 + cg * 256 < Nb) {              // else this warp's 256 candidates are all past N (e.g. N = 768): warp-uniform
#pragma unroll 1   // (a fully unrolled body makes ptxas rotate the 64 accumulators: +20% MOVs and spills at 128 regs)
            for (int d4 = 0; d4 < DCH / 4; ++d4) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float4 cv[4];
#pragma unroll
                    for (int ci = 0; ci < 4; ++ci)
                        cv[ci] = *reinterpret_cast<const float4*>(crow + ((h * 4 + ci) * 32) * DCP + d4 * 4);
#pragma unroll
                    for (int qi = 0; qi < 8; ++qi) {
                        const float4 qv = *reinterpret_cast<const float4*>(qrow + qi * DCP + d4 * 4);
                        // chain order d = 0,1,2,... per accumulator, exactly as oracle/canon.c; padded dims add 0*0
#pragma unroll
                        for (int ci = 0; ci < 4; ++ci) acc[qi][h * 4 + ci] = fmaf(qv.x, cv[ci].x, acc[qi][h * 4 + ci]);
#pragma unroll
                        for (int ci = 0; ci < 4; ++ci) acc[qi][h * 4 + ci] = fmaf(qv.y, cv[ci].y, acc[qi][h * 4 + ci]);
#pragma unroll
                        for (int ci = 0; ci < 4; ++ci) acc[qi][h * 4 + ci] = fmaf(qv.z, cv[ci].z, acc[qi][h * 4 + ci]);
#pragma unroll
                        for (int ci = 0; ci < 4; ++ci) acc[qi][h * 4 + ci] = fmaf(qv.w, cv[ci].w, acc[qi][h * 4 + ci]);
                    }
                }
            }
            }
            __syncthreads();                       // this slab's buffer may be refilled; the last one also orders the dist stores
        }

        // distances of this chunk -> dist[q][c]; candidates past N become -inf
        float xxq[8];
#pragma unroll
        for (int qi = 0; qi < 8; ++qi) {
            const int q = q0 + qg * 8 + qi;
            xxq[qi] = q < N ? xxb[q] : 0.f;
        }
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) {
            const int c = cg * 256 + ci * 32 + lane;
            const float nxc = -xxc[c];
            const bool cvalid = j0 + c < Nb;
#pragma unroll
            for (int qi = 0; qi < 8; ++qi) {
                const float pd = __fsub_rn(__fsub_rn(nxc, -2.f * acc[qi][ci]), xxq[qi]);
                dist[(qg * 8 + qi) * TC + c] = cvalid ? pd : -INFINITY;
            }
        }
        __syncthreads();

        // ---- selection: warp w owns queries QW*w .. QW*w+QW-1 ------------------------------------------
        select_chunk(dist, surv, run, j0, k, warp, lane, j0 == 0);
        // the loop-top __syncthreads orders these smem reads before the next chunk's stores
    }

#pragma unroll
    for (int w = 0; w < QW; ++w) {
        const int q = q0 + warp * QW + w;
        if (q < N && lane >= 1 && lane <= k) {
            const int j = q < Nb ? (int)(~run[w].lo) : q;
            const size_t o = ((size_t)b * N + q) * k + lane - 1;
            if (idx32) idx32[o] = j;
            if (idx64) idx64[o] = (int64_t)j;
        }
    }
}

template <int DCH, bool TM>
int launch_knn(const float* x, const float* xx, int B, int D, int N, int k, int32_t* i32, int64_t* i64,
               cudaStream_t st, const int* redo = nullptr, const int* nlen = nullptr) {
    auto kern = knn_select_kernel<DCH, TM>;
    const size_t smem = Smem<DCH>::total;
    // set on every launch: the attribute is per device, and one process may drive several (nn.DataParallel)
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return VCR_ERR_LAUNCH;
    dim3 grid(vcr_cdiv(N, TQ), B);
    kern<<<grid, NT, smem, st>>>(x, xx, D, N, k, i32, i64, redo, nlen);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

// =====================================================================================================
// 3-d kNN (the xyz graphs of LPDNet's SN1 / DGCNN): distances on the fly.  With D = 3 a distance is three FMAs, so the
// generic kernel's 32 x 512 distance tile in shared memory (64 KB, two CTAs per SM) only buys smem traffic and low
// occupancy for a selection whose shuffle networks are latency-bound.  Here a CTA keeps one 512-candidate chunk of the
// cloud as x | y | z | xx rows (8 KB) plus the survivor buffers (32 KB); every lane evaluates its 16 candidates of a query
// straight from those rows -- twice in the first chunk (lane maxima for the threshold, then the filter), once afterwards --
// with the canonical chain  acc = fma(qz, cz, fma(qy, cy, fma(qx, cx, 0)));  pd = (-xx_j - (-2 acc)) - xx_i,  and the
// same threshold / ballot-compaction / shuffle-bitonic selection as knn_select_kernel.  4 CTAs per SM.
// =====================================================================================================
template <int W, class F>
__device__ __forceinline__ bool filter_merge_fn(F&& get, const float (&tau)[W], Key (&run)[W], uint2* buf, int j0, int lane) {
    constexpr int RP = TC / 32;
    const uint32_t lt = (1u << lane) - 1u;
    int cnt[W], off[W];
    int base = 0;
    __syncwarp();
#pragma unroll
    for (int w = 0; w < W; ++w) {
        off[w] = base;
        int n = base;
#pragma unroll
        for (int r = 0; r < RP; ++r) {
            const float v = get(w, r);
            const bool p = v >= tau[w];
            const uint32_t bal = __ballot_sync(0xffffffffu, p);
            const int pos = n + __popc(bal & lt);
            if (p && pos < TC) buf[pos] = make_uint2(~(uint32_t)(j0 + r * 32 + lane), okey(v));
            n += __popc(bal);
        }
        cnt[w] = n - base;
        base = n;
    }
    __syncwarp();
    if (base > TC) return false;
    int rounds = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) rounds = max(rounds, (cnt[w] + 31) >> 5);
    for (int r = 0; r < rounds; ++r) {
        Key e[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int p = r * 32 + lane;
            const uint2 t = p < cnt[w] ? buf[off[w] + p] : make_uint2(0u, 0u);
            e[w].lo = t.x; e[w].hi = t.y;
        }
        sort32_desc<W>(e, lane);
        merge32_desc<W>(run, e, lane);
    }
    return true;
}

constexpr int QW3 = 2;                   // queries per warp (register budget: 64 / thread at 4 CTAs per SM)
constexpr int TQ3 = QW3 * (NT / 32);     // queries per CTA
template <bool TOKEN_MAJOR>
__global__ void __launch_bounds__(NT, 4)
knn3_kernel(const float* __restrict__ x, const float* __restrict__ xx, int N, int k,
            int32_t* __restrict__ idx32, int64_t* __restrict__ idx64, const int* __restrict__ nlen) {
    __shared__ float cs[4][TC];                       // x | y | z | xx of the chunk's candidates
    __shared__ uint2 surv[NT / 32][TC];               // per-warp survivor buffers
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y, q0 = blockIdx.x * TQ3;
    const float* xb = x + (size_t)b * 3 * N;
    const float* xxb = xx + (size_t)b * N;
    const int Nb = vcr_item_len(nlen, b, N, k + 1);
    if (q0 >= Nb) {                                   // every query of the CTA is padding
        knn_write_self(idx32, idx64, b, N, k, q0, min(TQ3, N - q0), tid, NT);
        return;
    }

    float qx[QW3], qy[QW3], qz[QW3], xxq[QW3];
#pragma unroll
    for (int w = 0; w < QW3; ++w) {
        const int q = min(q0 + warp * QW3 + w, Nb - 1); // queries past the cloud are computed and not written
        qx[w] = TOKEN_MAJOR ? xb[(size_t)q * 3 + 0] : xb[q];
        qy[w] = TOKEN_MAJOR ? xb[(size_t)q * 3 + 1] : xb[(size_t)N + q];
        qz[w] = TOKEN_MAJOR ? xb[(size_t)q * 3 + 2] : xb[2 * (size_t)N + q];
        xxq[w] = xxb[q];
    }
    Key run[QW3];
#pragma unroll
    for (int w = 0; w < QW3; ++w) run[w].hi = run[w].lo = 0u;
    uint2* buf = surv[warp];

    for (int j0 = 0; j0 < Nb; j0 += TC) {
        __syncthreads();                               // the previous chunk's rows are no longer read
        for (int c = tid; c < TC; c += NT) {
            const int g = j0 + c;
            const bool ok = g < N;
            cs[0][c] = ok ? (TOKEN_MAJOR ? xb[(size_t)g * 3 + 0] : xb[g]) : 0.f;
            cs[1][c] = ok ? (TOKEN_MAJOR ? xb[(size_t)g * 3 + 1] : xb[(size_t)N + g]) : 0.f;
            cs[2][c] = ok ? (TOKEN_MAJOR ? xb[(size_t)g * 3 + 2] : xb[2 * (size_t)N + g]) : 0.f;
            cs[3][c] = ok ? xxb[g] : 0.f;
        }
        __syncthreads();
        auto pd = [&](int w, int r) -> float {
            const int c = r * 32 + lane;
            const float acc = fmaf(qz[w], cs[2][c], fmaf(qy[w], cs[1][c], fmaf(qx[w], cs[0][c], 0.f)));
            const float v = __fsub_rn(__fsub_rn(-cs[3][c], -2.f * acc), xxq[w]);
            return j0 + c < Nb ? v : -INFINITY;
        };
        float tau[QW3];
        if (j0 == 0) {
            float m[QW3];
#pragma unroll
            for (int w = 0; w < QW3; ++w) {
                float mm = pd(w, 0);
#pragma unroll
                for (int r = 1; r < RPL; ++r) mm = fmaxf(mm, pd(w, r));
                m[w] = mm;
            }
            sort32_desc_f<QW3>(m, lane);
#pragma unroll
            for (int w = 0; w < QW3; ++w) tau[w] = __shfl_sync(0xffffffffu, m[w], k);
        } else {
#pragma unroll
            for (int w = 0; w < QW3; ++w) tau[w] = okey_inv(__shfl_sync(0xffffffffu, run[w].hi, k));
        }
        if (!filter_merge_fn<QW3>(pd, tau, run, buf, j0, lane)) {
            // heavy ties: one query at a time, any survivor count fits the buffer
#pragma unroll
            for (int w = 0; w < QW3; ++w) {
                float t1[1] = {tau[w]};
                Key r1[1] = {run[w]};
                filter_merge_fn<1>([&](int, int r) { return pd(w, r); }, t1, r1, buf, j0, lane);
                run[w] = r1[0];
            }
        }
    }
#pragma unroll
    for (int w = 0; w < QW3; ++w) {
        const int q = q0 + warp * QW3 + w;
        if (q < N && lane >= 1 && lane <= k) {
            const int j = q < Nb ? (int)(~run[w].lo) : q;
            const size_t o = ((size_t)b * N + q) * k + lane - 1;
            if (idx32) idx32[o] = j;
            if (idx64) idx64[o] = (int64_t)j;
        }
    }
}

// =====================================================================================================
// Tensor-core variant for feature-space kNN (16 <= D <= 128, token-major): the exact kernel's geometry (a CTA owns 32
// queries, 512-candidate chunks, the same warp-per-query selection) with the FP32 FMA phase replaced by tcgen05
// distance tiles used as a PREFILTER, then an exact canonical re-rank with a per-query certificate.
//
//   approx  per chunk 4 MMA tiles D[128 candidates x 32 queries] (candidates on the M side so that a TMEM lane is a
//           candidate and a thread's 32 columns are the 32 queries: the epilogue's smem stores dist[q][c] are
//           lane-contiguous).  dot~ from the 3-term fp16 split of the operand-format copy of x (hi*hi' in one TMEM
//           accumulator, hi*lo' + lo*hi' in a second, combined in fp32); pd~ = (-xx_j - (-2 dot~)) - xx_i with the
//           CANONICAL xx.  One producer warp (TMA candidate tiles through one smem stage, MMA issue), 8 consumer warps
//           (TMEM -> pd~ tile -> selection keeping ranks 0..ksel, ksel = k + 8).  The survivor buffers alias the
//           candidate stage, two CTAs per SM overlap one CTA's TMA/MMA phase with the other's selection.
//   exact   the 32 list entries of a query are re-evaluated with the canonical fp32 fma chain (one entry per lane)
//           and sorted by (pd, lower index): ranks 1..k are the answer IF no candidate outside the certified part
//           of the list can reach rank k:   pd_exact(rank k) > pd~(rank ksel) + eps,   eps >= |pd~ - pd| for this
//           query against any candidate (bound below).  Otherwise the query's 32-group (= this CTA) is flagged and
//           recomputed by the exact kernel (same launch sequence, no host sync).  The result is therefore
//           bit-identical to vcr_knn_topk on every input; only the speed depends on the data.
//   eps     |dot~ - dot_canon| <= (split 3*2^-22 + fp32 chain D*2^-24 + TMEM accumulation D*2^-24) |x_i||x_j|
//           < 2^-15 |x_i||x_j| for D <= 128; pd doubles it and adds <= 2 ulp of (xx_i + xx_j + 2|dot|):
//           eps_i = 2^-14 sqrt(xx_i * xxmax) + 2^-20 xxmax, xxmax = max_j xx_j of the cloud.
//           Clouds with xxmax outside [2^-20, 2^30] (fp16 range of the split) go to the exact kernel entirely.
// =====================================================================================================
constexpr int T2M = 128;                  // candidates per MMA tile (UMMA M)
constexpr int T2TILES = TC / T2M;         // MMA tiles per chunk (4)
constexpr int T2NT = NT + 32;             // 8 consumer warps + 1 producer warp
constexpr int T2CTILE = T2M * 128;        // bytes of one [128 candidates][64 x fp16] swizzled tile
constexpr int T2QTILE = TQ * 128;         // bytes of one [32 queries][64 x fp16] swizzled tile

struct KnnTcParams {
    const float* x;          // [B, N, D] fp32 token-major
    const float* xx;         // [B*N] canonical squared norms
    const uint32_t* xxmax;   // [B] bit pattern of max_j xx_j
    int* redo;               // [B * ceil(N/32)] flags for the exact kernel (one per CTA)
    int* nflag;              // [1] number of uncertified queries (telemetry)
    const int* nlen;         // [B] points per item of a ragged batch, or null
    int D, N, k, ksel, KB;
    int32_t* idx32;
    int64_t* idx64;
};

// smem: Q tiles | candidate stage (aliased by the survivor buffers during selection) | pd~ tile | xx of the queries | barriers
__host__ __device__ constexpr size_t knn_tc_stage_bytes(int KB) {
    return (size_t)KB * 2 * T2CTILE > SURV_BYTES ? (size_t)KB * 2 * T2CTILE : SURV_BYTES;
}
__host__ __device__ constexpr size_t knn_tc_smem_bytes(int KB) {
    return (size_t)KB * 2 * T2QTILE + knn_tc_stage_bytes(KB) + (size_t)TQ * TC * 4 + TQ * 4 + 64 + 1024;
}

__global__ void knn_sqnorm_max_kernel(const float* __restrict__ x, int D, int N, float* __restrict__ xx,
                                      uint32_t* __restrict__ xxmax, const int* __restrict__ nlen, int k) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t bits = 0u;
    if (i < N) {
        const float* r = x + ((size_t)b * N + i) * D;
        float acc = 0.f;
        for (int d = 0; d < D; ++d) acc = fmaf(r[d], r[d], acc);      // canonical chain (oracle/canon.c)
        xx[(size_t)b * N + i] = acc;
        // acc >= 0 (or NaN, which sorts above +inf); the maximum is taken over the real points only
        if (i < vcr_item_len(nlen, b, N, k + 1)) bits = __float_as_uint(acc);
    }
    bits = __reduce_max_sync(0xffffffffu, bits);
    if ((threadIdx.x & 31) == 0 && bits) atomicMax(xxmax + b, bits);
}

__global__ void __launch_bounds__(T2NT, 2)
knn_tc_kernel(const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmQ, const KnnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const int KB = p.KB, N = p.N, D = p.D, k = p.k, ksel = p.ksel;
    const int qbytes = KB * 2 * T2QTILE, cbytes = KB * 2 * T2CTILE;
    uint8_t* q_s = smem;
    uint8_t* c_s = smem + qbytes;
    uint2* surv = reinterpret_cast<uint2*>(c_s);                              // [8][512], valid during selection only
    float* dist = reinterpret_cast<float*>(c_s + knn_tc_stage_bytes(KB));     // [32][512]
    float* xxq_s = dist + TQ * TC;                                            // [32]
    uint64_t* bars = reinterpret_cast<uint64_t*>(xxq_s + TQ);
    uint64_t* q_full = bars + 0;
    uint64_t* c_full = bars + 1;          // candidate tile landed                  (4 phases per chunk)
    uint64_t* mma_bar = bars + 2;         // MMAs of a tile retired: stage reusable (4 phases per chunk)
    uint64_t* chunk_ready = bars + 3;     // all 4 tiles of the chunk are in TMEM   (1 phase per chunk)
    uint64_t* stage_free = bars + 4;      // 8 consumer warps finished the chunk's selection (TMEM + stage + dist free)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, q0 = blockIdx.x * TQ;
    const float* xxb = p.xx + (size_t)b * N;
    const int Nb = vcr_item_len(p.nlen, b, N, k + 1);
    if (q0 >= Nb) {                                   // every query of the CTA is padding
        knn_write_self(p.idx32, p.idx64, b, N, k, q0, min(TQ, N - q0), tid, T2NT);
        return;
    }
    const int nch = (Nb + TC - 1) / TC;

    if (warp == NT / 32 && lane == 0) {
        tc::tma_prefetch_desc(&tmC); tc::tma_prefetch_desc(&tmQ);
        tc::mbar_init(q_full, 1); tc::mbar_init(c_full, 1); tc::mbar_init(mma_bar, 1);
        tc::mbar_init(chunk_ready, 1); tc::mbar_init(stage_free, NT / 32);
        tc::fence_barrier_init();
    }
    if (warp == 0) { tc::tmem_alloc(tmem_slot, 256); tc::tmem_relinquish(); }
    if (tid < TQ) xxq_s[tid] = q0 + tid < N ? xxb[q0 + tid] : 0.f;
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const float xm = __uint_as_float(p.xxmax[b]);
    const bool cloud_ok = xm >= 9.5367431640625e-07f && xm <= 1073741824.f;     // [2^-20, 2^30]; false for NaN
    if (!cloud_ok) {
        // outside the fp16 range of the split: the exact kernel computes this 32-group
        if (tid == 0) {
            p.redo[b * gridDim.x + blockIdx.x] = 1;
            atomicAdd(p.nflag, min(TQ, N - q0));
        }
    } else if (warp == NT / 32) {
        // ============================== TMA producer + MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::umma_idesc(T2M, TQ, 0);
            const int row0 = b * N;
            tc::mbar_expect_tx(q_full, qbytes);
            for (int kb = 0; kb < KB; ++kb)
                for (int pl = 0; pl < 2; ++pl)
                    tc::tma_load_3d(q_s + (kb * 2 + pl) * T2QTILE, &tmQ, q_full, kb * 64, row0 + q0, pl);
            tc::mbar_wait(q_full, 0);
            const uint32_t q_addr = tc::smem_u32(q_s), c_addr = tc::smem_u32(c_s);
            uint32_t g = 0;                                              // tile counter: parity of c_full / mma_bar
            for (int c = 0; c < nch; ++c) {
                if (c > 0) { tc::mbar_wait(stage_free, (c - 1) & 1); tc::tc_fence_after(); }
                for (int t = 0; t < T2TILES; ++t, ++g) {
                    const int cand0 = c * TC + t * T2M;
                    if (cand0 < Nb) {
                        tc::mbar_expect_tx(c_full, cbytes);
                        for (int kb = 0; kb < KB; ++kb)
                            for (int pl = 0; pl < 2; ++pl)
                                tc::tma_load_3d(c_s + (kb * 2 + pl) * T2CTILE, &tmC, c_full, kb * 64, row0 + cand0, pl);
                        tc::mbar_wait(c_full, g & 1);
                        tc::tc_fence_after();
                        const uint32_t d0 = tmem_base + t * TQ, d1 = tmem_base + T2TILES * TQ + t * TQ;
                        for (int kb = 0; kb < KB; ++kb) {
                            const uint64_t c_hi = tc::umma_desc_k_sw128(c_addr + (kb * 2) * T2CTILE);
                            const uint64_t c_lo = tc::umma_desc_k_sw128(c_addr + (kb * 2 + 1) * T2CTILE);
                            const uint64_t q_hi = tc::umma_desc_k_sw128(q_addr + (kb * 2) * T2QTILE);
                            const uint64_t q_lo = tc::umma_desc_k_sw128(q_addr + (kb * 2 + 1) * T2QTILE);
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                const uint32_t acc = (kb | kk) != 0;
                                const uint64_t adv = (uint64_t)(kk * 2);
                                tc::umma_f16(d0, c_hi + adv, q_hi + adv, idesc, acc);
                                tc::umma_f16(d1, c_hi + adv, q_lo + adv, idesc, acc);
                                tc::umma_f16(d1, c_lo + adv, q_hi + adv, idesc, 1);
                            }
                        }
                        tc::umma_commit(mma_bar);
                        tc::mbar_wait(mma_bar, g & 1);                   // tile consumed: the stage may be refilled
                    } else {
                        // tile entirely past N: nothing to load; keep the barrier phases in step
                        tc::mbar_arrive(c_full);
                        tc::mbar_arrive(mma_bar);
                    }
                }
                tc::umma_commit(chunk_ready);                            // arrives once every MMA of the chunk has retired
            }
        }
    } else {
        // ============================== consumers: TMEM -> pd~ tile -> selection ==============================
        const int qq = warp & 3, th = warp >> 2;                         // TMEM lane quarter, tile half
        Key run[QW];
#pragma unroll
        for (int w = 0; w < QW; ++w) run[w].hi = run[w].lo = 0u;

        for (int c = 0; c < nch; ++c) {
            const int j0 = c * TC;
            tc::mbar_wait(chunk_ready, c & 1);
            tc::tc_fence_after();
#pragma unroll
            for (int tt = 0; tt < T2TILES / 2; ++tt) {
                const int t = th * (T2TILES / 2) + tt;
                const int cl = t * T2M + qq * 32 + lane;                 // candidate of this thread within the chunk
                const int j = j0 + cl;
                float* dcol = dist + cl;
                if (j0 + t * T2M < Nb) {                                 // warp-uniform: the tile holds data
                    const uint32_t ta = tmem_base + ((uint32_t)(qq * 32) << 16) + t * TQ;
                    const bool cvalid = j < Nb;
                    const float nxc = cvalid ? -xxb[j] : 0.f;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint32_t r0[16], r1[16];
                        tc::tmem_ld_32x16(ta + h * 16, r0);
                        tc::tmem_ld_32x16(ta + T2TILES * TQ + h * 16, r1);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            const float dot = fmaf(__uint_as_float(r1[q]), 1.f / 2048.f, __uint_as_float(r0[q]));
                            const float pd = __fsub_rn(__fsub_rn(nxc, -2.f * dot), xxq_s[h * 16 + q]);
                            dcol[(h * 16 + q) * TC] = cvalid ? pd : -INFINITY;
                        }
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < TQ; ++q) dcol[q * TC] = -INFINITY;
                }
            }
            tc::tc_fence_before();
            asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");       // pd~ tile complete (consumer warps only)
            select_chunk(dist, surv, run, j0, ksel, warp, lane, c == 0);
            tc::fence_proxy_async();                                     // survivor stores (generic proxy) before the next TMA fill
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(stage_free);
        }

        // ---- exact re-rank + certificate, one query at a time, one list entry per lane ----
        const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.x) & 15) == 0);
        bool all_safe = true;
#pragma unroll
        for (int qi = 0; qi < QW; ++qi) {
            const int q = q0 + warp * QW + qi;
            if (q >= N) continue;                                        // warp-uniform
            if (q >= Nb) {                                               // padded query: its own index
                if (lane < k) knn_write_self(p.idx32, p.idx64, b, N, k, q, 1, lane, k);
                continue;
            }
            const Key a = run[qi];
            const uint32_t thr_hi = __shfl_sync(0xffffffffu, a.hi, ksel);
            const int j = (int)(~a.lo);
            const bool valid = j >= 0 && j < Nb;
            const float xxq = xxq_s[warp * QW + qi];
            Key e[1];
            e[0].hi = 0u; e[0].lo = 0u;
            if (valid) {
                const float* xq = p.x + ((size_t)b * N + q) * D;
                const float* xj = p.x + ((size_t)b * N + j) * D;
                float acc = 0.f;
                if (vec) {
                    for (int d = 0; d < D; d += 4) {
                        const float4 qv = __ldg(reinterpret_cast<const float4*>(xq + d));
                        const float4 cv = __ldg(reinterpret_cast<const float4*>(xj + d));
                        acc = fmaf(qv.x, cv.x, acc); acc = fmaf(qv.y, cv.y, acc);
                        acc = fmaf(qv.z, cv.z, acc); acc = fmaf(qv.w, cv.w, acc);
                    }
                } else {
                    for (int d = 0; d < D; ++d) acc = fmaf(__ldg(xq + d), __ldg(xj + d), acc);
                }
                const float pd = __fsub_rn(__fsub_rn(-xxb[j], -2.f * acc), xxq);
                e[0].hi = okey(pd); e[0].lo = a.lo;
            }
            sort32_desc<1>(e, lane);
            const uint32_t ek_hi = __shfl_sync(0xffffffffu, e[0].hi, k);
            const float eps = 6.103515625e-05f * sqrtf(xxq * xm) + 9.5367431640625e-07f * xm;
            const bool safe = ek_hi != 0u && (thr_hi == 0u || okey_inv(ek_hi) > okey_inv(thr_hi) + eps);
            if (safe) {
                if (lane >= 1 && lane <= k) {
                    const int jn = (int)(~e[0].lo);
                    const size_t o = ((size_t)b * N + q) * k + lane - 1;
                    if (p.idx32) p.idx32[o] = jn;
                    if (p.idx64) p.idx64[o] = (int64_t)jn;
                }
            } else {
                all_safe = false;
                if (lane == 0) atomicAdd(p.nflag, 1);
            }
        }
        if (!all_safe && lane == 0) p.redo[b * gridDim.x + blockIdx.x] = 1;
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem_base, 256);
}

#include "knn_tpq.cuh"      // thread-per-query selection: knn3_tpq_kernel (D = 3, exact), knn_tc2_kernel (tcgen05 prefilter)

}  // namespace

VCR_API size_t vcr_knn_workspace_bytes(int B, int N) { return (size_t)B * N * sizeof(float); }

// x: [B,D,N] (token_major=0, the reference layout) or [B,N,D] (token_major=1); idx: [B,N,k].
// Either idx32 or idx64 (or both) may be given.  Requires 1 <= k <= 31, N >= k+1; any D >= 1 (D <= 4 is staged
// 4 dims at a time, wider features 16 dims at a time).
static std::atomic<int> g_vcr_knn3_direct{1};      // tuning knob (see vcr_set_knn3_direct)
static std::atomic<int> g_vcr_knn_tc_tpq{2};       // tuning knob (see vcr_set_knn_tc_tpq)

// D == 3: distances on the fly (knn3_kernel, default) or the generic tile kernel.  Same indices; returns the previous setting.
VCR_API int vcr_set_knn3_direct(int on) {
    return g_vcr_knn3_direct.exchange(on ? 1 : 0);
}

// Feature-space tensor-core route: 1 = always the thread-per-query selection from TMEM (knn_tc2_kernel), 0 = always the
// warp-per-query selection from a shared-memory distance tile (knn_tc_kernel), 2 (default) = thread-per-query from
// N >= 8192, where it measured faster.  Same indices; returns the previous setting.
VCR_API int vcr_set_knn_tc_tpq(int on) {
    return g_vcr_knn_tc_tpq.exchange(on < 0 ? 0 : (on > 2 ? 2 : on));
}

static int knn_topk_impl(const float* x, const int* nlen, int B, int D, int N, int k, int token_major, int32_t* idx32,
                         int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    if (N < k + 1) return VCR_ERR_INVALID;
    if (!workspace || workspace_bytes < vcr_knn_workspace_bytes(B, N)) return VCR_ERR_WORKSPACE;
    float* xx = reinterpret_cast<float*>(workspace);
    dim3 g(vcr_cdiv(N, 256), B);
    if (token_major) knn_sqnorm_kernel<true><<<g, 256, 0, stream>>>(x, D, N, xx);
    else knn_sqnorm_kernel<false><<<g, 256, 0, stream>>>(x, D, N, xx);
    VCR_CHECK_LAUNCH();
    if (k > 31) return VCR_ERR_UNSUPPORTED;
    const int route3 = g_vcr_knn3_direct.load(std::memory_order_relaxed);
    if (D == 3 && route3 != 0) {
        dim3 grid(vcr_cdiv(N, TQ3), B);
        if (token_major) knn3_kernel<true><<<grid, NT, 0, stream>>>(x, xx, N, k, idx32, idx64, nlen);
        else knn3_kernel<false><<<grid, NT, 0, stream>>>(x, xx, N, k, idx32, idx64, nlen);
        VCR_CHECK_LAUNCH();
        return VCR_OK;
    }
    if (D <= 4)
        return token_major ? launch_knn<4, true>(x, xx, B, D, N, k, idx32, idx64, stream, nullptr, nlen)
                           : launch_knn<4, false>(x, xx, B, D, N, k, idx32, idx64, stream, nullptr, nlen);
    return token_major ? launch_knn<16, true>(x, xx, B, D, N, k, idx32, idx64, stream, nullptr, nlen)
                       : launch_knn<16, false>(x, xx, B, D, N, k, idx32, idx64, stream, nullptr, nlen);
}

VCR_API int vcr_knn_topk(const float* x, int B, int D, int N, int k, int token_major, int32_t* idx32,
                         int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(x && (idx32 || idx64) && B > 0 && N > 0 && k >= 1);
    return knn_topk_impl(x, nullptr, B, D, N, k, token_major, idx32, idx64, workspace, workspace_bytes, stream);
}

// Ragged batch: item b has n[b] real points (clamped to [k+1, N]) in its N rows.  Indices of real queries equal
// vcr_knn_topk's on the item alone; padded queries get their own index in all k slots.
VCR_API int vcr_knn_topk_ragged(const float* x, const int* n, int B, int D, int N, int k, int token_major, int32_t* idx32,
                                int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(x && n && (idx32 || idx64) && B > 0 && N > 0 && k >= 1);
    return knn_topk_impl(x, n, B, D, N, k, token_major, idx32, idx64, workspace, workspace_bytes, stream);
}

// ---- tensor-core prefilter + exact re-rank (16 <= D <= 128, token-major) --------------------------------------
// workspace layout (4-byte words): xx [B*N] | xxmax [B] | redo [B*ceil(N/32)] | nflag [1]
VCR_API size_t vcr_knn_tc_workspace_bytes(int B, int N) {
    return ((size_t)B * N + (size_t)B + (size_t)B * ((N + 31) / 32) + 1) * 4;
}

static int knn_topk_tc_impl(const float* x, const void* xop, int ld, long long plane_stride, const int* nlen, int B, int D,
                            int N, int k, int32_t* idx32, int64_t* idx64, void* workspace, size_t workspace_bytes,
                            cudaStream_t stream) {
    if (N < k + 1) return VCR_ERR_INVALID;
    if (D < 16 || D > 128 || k > 30 || (long long)B * N > 0x7fffffffLL || B > 65535) return VCR_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vcr_knn_tc_workspace_bytes(B, N)) return VCR_ERR_WORKSPACE;
    const int nq32 = (N + 31) / 32;
    float* xx = reinterpret_cast<float*>(workspace);
    uint32_t* xxmax = reinterpret_cast<uint32_t*>(xx + (size_t)B * N);
    int* redo = reinterpret_cast<int*>(xxmax + B);
    int* nflag = redo + (size_t)B * nq32;
    if (cudaMemsetAsync(xxmax, 0, ((size_t)B + (size_t)B * nq32 + 1) * 4, stream) != cudaSuccess) return VCR_ERR_LAUNCH;
    dim3 g(vcr_cdiv(N, 256), B);
    knn_sqnorm_max_kernel<<<g, 256, 0, stream>>>(x, D, N, xx, xxmax, nlen, k);
    VCR_CHECK_LAUNCH();
    CUtensorMap tmC, tmQ;
    const int tpq = g_vcr_knn_tc_tpq.load(std::memory_order_relaxed);
    if (tpq == 1 || (tpq == 2 && N >= 8192)) {
        int rc = vcr_make_operand_tmap(&tmC, xop, D, (long long)B * N, ld, plane_stride, 2, TC2);
        if (rc != VCR_OK) return rc;
        rc = vcr_make_operand_tmap(&tmQ, xop, D, (long long)B * N, ld, plane_stride, 2, TQ2);
        if (rc != VCR_OK) return rc;
        KnnTcParams p;
        p.x = x; p.xx = xx; p.xxmax = xxmax; p.redo = redo; p.nflag = nflag; p.nlen = nlen;
        p.D = D; p.N = N; p.k = k; p.ksel = k + 8 < 31 ? k + 8 : 31; p.KB = (D + 63) / 64;
        p.idx32 = idx32; p.idx64 = idx64;
        const size_t smem = knn_tc2_smem_bytes(p.KB);
        if (cudaFuncSetAttribute(knn_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return VCR_ERR_LAUNCH;
        knn_tc2_kernel<<<dim3(vcr_cdiv(N, TQ2), B), T2_THREADS, smem, stream>>>(tmC, tmQ, p);
        VCR_CHECK_LAUNCH();
        return launch_knn<16, true>(x, xx, B, D, N, k, idx32, idx64, stream, redo, nlen);   // repairs flagged groups only
    }
    int rc = vcr_make_operand_tmap(&tmC, xop, D, (long long)B * N, ld, plane_stride, 2, T2M);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tmQ, xop, D, (long long)B * N, ld, plane_stride, 2, TQ);
    if (rc != VCR_OK) return rc;
    KnnTcParams p;
    p.x = x; p.xx = xx; p.xxmax = xxmax; p.redo = redo; p.nflag = nflag; p.nlen = nlen;
    p.D = D; p.N = N; p.k = k; p.ksel = k + 8 < 31 ? k + 8 : 31; p.KB = (D + 63) / 64;
    p.idx32 = idx32; p.idx64 = idx64;
    const size_t smem = knn_tc_smem_bytes(p.KB);
    if (cudaFuncSetAttribute(knn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return VCR_ERR_LAUNCH;
    knn_tc_kernel<<<dim3(nq32, B), T2NT, smem, stream>>>(tmC, tmQ, p);
    VCR_CHECK_LAUNCH();
    return launch_knn<16, true>(x, xx, B, D, N, k, idx32, idx64, stream, redo, nlen);       // repairs flagged groups only
}

// x: fp32 [B,N,D] token-major; xop: its operand-format copy [2 planes][B*N][ld] (fp16 hi, lo*2^11; vcr_to_operand).
// Writes exactly what vcr_knn_topk writes (bit-identical indices) -- see the kernel comment for the certificate.
// After the call, the last word of the workspace holds the number of queries that went through the exact kernel.
VCR_API int vcr_knn_topk_tc(const float* x, const void* xop, int ld, long long plane_stride, int B, int D, int N, int k,
                            int32_t* idx32, int64_t* idx64, void* workspace, size_t workspace_bytes,
                            cudaStream_t stream) {
    VCR_REQUIRE(x && xop && (idx32 || idx64) && B > 0 && N > 0 && k >= 1);
    return knn_topk_tc_impl(x, xop, ld, plane_stride, nullptr, B, D, N, k, idx32, idx64, workspace, workspace_bytes, stream);
}

// Ragged batch, as vcr_knn_topk_ragged: the maximum squared norm of the certificate is taken over item b's n[b] points.
VCR_API int vcr_knn_topk_tc_ragged(const float* x, const void* xop, int ld, long long plane_stride, const int* n, int B,
                                   int D, int N, int k, int32_t* idx32, int64_t* idx64, void* workspace,
                                   size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(x && xop && n && (idx32 || idx64) && B > 0 && N > 0 && k >= 1);
    return knn_topk_tc_impl(x, xop, ld, plane_stride, n, B, D, N, k, idx32, idx64, workspace, workspace_bytes, stream);
}
