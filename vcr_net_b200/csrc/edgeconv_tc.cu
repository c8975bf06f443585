// EdgeConv DG block on tcgen05 / TMEM (sm_100a): convDG1 + max + convDG2 + max of the LPDNet embedding
// (reference model/lpdnet_model.py:122-126 on top of util/util.py:176-199) in ONE kernel, the
// [N*k, 128] edge tensors (335 MB per 32 clouds in the reference) never leave the SM.
//
// Algebra as in edgeconv.cu: e1[edge] = act(P[j] + Q[i]) with PQ = [P | Q] from the per-point GEMM,
// x1 = max_k e1, e2 = W2 e1 + b2, x2 = act(max_k e2) (LeakyReLU slope >= 0 is monotone).
//
// The DG2 GEMM is issued TRANSPOSED:  D[o][edge] = sum_c W2[o][c] * e1[edge][c]
//   A = W2   [128 out-channels (M)][128 c (K)]  K-major, converted once per CTA, resident in smem
//   B = e1   [80 edges (N) = 4 points x 20][128 c (K)]  K-major, built by the producer warps
//   D in TMEM: lane = output channel, column = edge  ->  max over a point's 20 edges is an in-thread
//   reduction over 20 consecutive columns after tcgen05.ld, and the x2 store of a warp is 32 consecutive
//   channels of one point (coalesced); no cross-lane traffic, no padding of the MMA tile.
//
// Warp roles (512 threads, persistent CTA per SM, tile = 8 points = two 80-edge MMA groups):
//   warps 8-15  producers: warp w owns point w of the tile: gathers the 20 neighbour rows of P (L2),
//               adds Q, LeakyReLU, running max -> x1, writes fp16 (hi, lo*2^11) rows into the swizzled B stage
//   warp 1      one elected thread issues tcgen05.mma (128 x 80 x 16), 3 terms in the fp32-parity mode
//   warps 4-7   epilogue: tcgen05.ld 80 columns, max per 20, + b2, LeakyReLU, store x2
//   warp 2      TMEM allocation
// Roofline: tensor work 2*128*128*20 flop per point (x3 terms); HBM bytes 4*(256 in + 256 out) + 4*20 per
// point; the neighbour gather (20 x 512 B per point) is served by L2.
#include "tc_common.cuh"

namespace {

constexpr int C = 128;            // channels in / out of convDG2
constexpr int KN = 20;            // neighbours
constexpr int PTS_SUB = 4;        // points per MMA group
constexpr int NSUB = 2;           // MMA groups per stage
constexpr int PTS_TILE = PTS_SUB * NSUB;
constexpr int EN = PTS_SUB * KN;  // 80 edges = MMA N
constexpr int W_TILE = 128 * 128; // [128 rows][128 B]
constexpr int B_TILE = EN * 128;  // [80 rows][128 B]
constexpr int NPROD = 8;          // producer warps
constexpr int NTHREADS = 512;
constexpr int ACC_STRIDE = 256;   // TMEM columns per accumulator buffer: D0 at +0, D1 at +128

template <int NTERMS>
struct ECfg {
    static constexpr int PL = NTERMS == 3 ? 2 : 1;
    static constexpr int W_BYTES = PL * 2 * W_TILE;               // [plane][kb]
    static constexpr int SUB_BYTES = PL * 2 * B_TILE;             // [plane][kb]
    static constexpr int STAGE_BYTES = NSUB * SUB_BYTES;
    static constexpr int NSTAGE = 2;
    static constexpr int OFF_B = W_BYTES;
    static constexpr int OFF_BAR = OFF_B + NSTAGE * STAGE_BYTES;
    static constexpr int SMEM = OFF_BAR + 256 + 1024;
    static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
};

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

// byte offset of 4 consecutive K elements (c4*4 .. c4*4+3) of row r inside a [plane][kb][rows][128 B]
// K-major SWIZZLE_128B operand (the 8-byte piece a lane owns); tile_bytes = rows * 128
__device__ __forceinline__ uint32_t sw_off(int r, int c4, int tile_bytes) {
    const int kb = c4 >> 4, chunk = (c4 & 15) >> 1;
    return (uint32_t)(kb * tile_bytes + r * 128 + ((chunk ^ (r & 7)) << 4) + ((c4 & 1) << 3));
}

// ZOUT: also write the per-edge pre-activations z (a separate instantiation keeps the forward's machine code unchanged)
template <int NTERMS, int FMT, bool ZOUT>
__global__ void __launch_bounds__(NTHREADS, 1)
edgeconv_dg_tc_kernel(const float* __restrict__ PQ, int ldpq, const int* __restrict__ idx, int N, long long total_pts,
                      const float* __restrict__ W2, const float* __restrict__ b2, float slope,
                      float* __restrict__ x1, int ld1, float* __restrict__ x2, int ld2,
                      __half* __restrict__ op1, __half* __restrict__ op2, int ldop, long long op_plane,
                      float* __restrict__ z) {
    using C_ = ECfg<NTERMS>;
    constexpr int PL = C_::PL;
    constexpr int obf = FMT;      // 1: bf16 operands
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C_::OFF_BAR);
    uint64_t* full = bars;            // [2]  producers -> MMA
    uint64_t* empty = bars + 2;       // [2]  MMA -> producers
    uint64_t* tfull = bars + 4;       // [2]  MMA -> epilogue (per accumulator buffer = MMA group)
    uint64_t* tempty = bars + 6;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long ntiles = (total_pts + PTS_TILE - 1) / PTS_TILE;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&full[s], NPROD * 32); tc::mbar_init(&empty[s], 1);
            tc::mbar_init(&tfull[s], 1);         tc::mbar_init(&tempty[s], 128);
        }
        tc::fence_barrier_init();
    }
    if (warp == 2) { tc::tmem_alloc(tmem_slot, C_::TMEM_COLS); tc::tmem_relinquish(); }
    // W2 -> A operand (hi / lo planes), every thread converts 8 float4
    for (int e = threadIdx.x; e < C * C / 4; e += NTHREADS) {
        const int o = e >> 5, c4 = e & 31;
        const float4 w = __ldg(reinterpret_cast<const float4*>(W2) + e);
        const uint32_t off = sw_off(o, c4, W_TILE);
        *reinterpret_cast<uint2*>(smem + off) = make_uint2(tc::pack_h2(w.x, w.y, obf), tc::pack_h2(w.z, w.w, obf));
        if (PL == 2)
            *reinterpret_cast<uint2*>(smem + 2 * W_TILE + off) =
                make_uint2(tc::pack_h2(tc::lo_part(w.x, obf), tc::lo_part(w.y, obf), obf),
                           tc::pack_h2(tc::lo_part(w.z, obf), tc::lo_part(w.w, obf), obf));
    }
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= 8) {
        // ============================== producers: one point per warp ==============================
        const int pw = warp - 8;
        const int sub = pw >> 2, prow0 = (pw & 3) * KN;
        int it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = it & 1;
            const long long pt = tile * PTS_TILE + pw;
            // gather requests first: they do not depend on the stage being free
            float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f);
            int myidx = 0;
            long long cloud0 = 0;
            const bool ok = pt < total_pts;
            if (ok) {
                cloud0 = (pt / N) * N;
                if (lane < KN) myidx = __ldg(idx + pt * KN + lane);
                q4 = __ldg(reinterpret_cast<const float4*>(PQ + pt * ldpq + C) + lane);
            }
            tc::mbar_wait(&empty[s], ((it >> 1) & 1) ^ 1);
            if (ok) {
                uint8_t* st = smem + C_::OFF_B + s * C_::STAGE_BYTES + sub * C_::SUB_BYTES;
                float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll
                for (int k0 = 0; k0 < KN; k0 += 10) {
                    float4 a[10];
#pragma unroll
                    for (int u = 0; u < 10; ++u) {
                        const int j = __shfl_sync(0xffffffffu, myidx, k0 + u);
                        a[u] = __ldg(reinterpret_cast<const float4*>(PQ + (cloud0 + j) * ldpq) + lane);
                    }
#pragma unroll
                    for (int u = 0; u < 10; ++u) {
                        float4 v;
                        v.x = leaky(a[u].x + q4.x, slope); v.y = leaky(a[u].y + q4.y, slope);
                        v.z = leaky(a[u].z + q4.z, slope); v.w = leaky(a[u].w + q4.w, slope);
                        mx.x = fmaxf(mx.x, v.x); mx.y = fmaxf(mx.y, v.y); mx.z = fmaxf(mx.z, v.z); mx.w = fmaxf(mx.w, v.w);
                        const uint32_t off = sw_off(prow0 + k0 + u, lane, B_TILE);
                        *reinterpret_cast<uint2*>(st + off) = make_uint2(tc::pack_h2(v.x, v.y, obf), tc::pack_h2(v.z, v.w, obf));
                        if (PL == 2)
                            *reinterpret_cast<uint2*>(st + 2 * B_TILE + off) =
                                make_uint2(tc::pack_h2(tc::lo_part(v.x, obf), tc::lo_part(v.y, obf), obf),
                                           tc::pack_h2(tc::lo_part(v.z, obf), tc::lo_part(v.w, obf), obf));
                    }
                }
                *reinterpret_cast<float4*>(x1 + pt * ld1 + lane * 4) = mx;
                if (op1 != nullptr) {     // the same row in "h3" operand format (fp16 hi / lo * 2^11) for the next GEMM
                    __half* orow = op1 + pt * ldop + lane * 4;
                    *reinterpret_cast<uint2*>(orow) = make_uint2(tc::pack_h2(mx.x, mx.y, 0), tc::pack_h2(mx.z, mx.w, 0));
                    *reinterpret_cast<uint2*>(orow + op_plane) =
                        make_uint2(tc::pack_h2(tc::lo_part(mx.x, 0), tc::lo_part(mx.y, 0), 0),
                                   tc::pack_h2(tc::lo_part(mx.z, 0), tc::lo_part(mx.w, 0), 0));
                }
            }
            tc::fence_proxy_async();                      // generic-proxy smem writes -> visible to the tensor core
            tc::mbar_arrive(&full[s]);
        }
    } else if (warp == 1) {
        // ============================== MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::umma_idesc(128, EN, FMT);
            const uint32_t w_addr = tc::smem_u32(smem);
            int it = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
                const int s = it & 1;
                tc::mbar_wait(&full[s], (it >> 1) & 1);
                tc::tc_fence_after();
#pragma unroll
                for (int sub = 0; sub < NSUB; ++sub) {
                    tc::mbar_wait(&tempty[sub], (it & 1) ^ 1);
                    tc::tc_fence_after();
                    const uint32_t b_addr = tc::smem_u32(smem + C_::OFF_B + s * C_::STAGE_BYTES + sub * C_::SUB_BYTES);
                    const uint32_t d0 = tmem_base + sub * ACC_STRIDE, d1 = d0 + 128;
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t a_hi = tc::umma_desc_k_sw128(w_addr + kb * W_TILE);
                        const uint64_t b_hi = tc::umma_desc_k_sw128(b_addr + kb * B_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint32_t acc = (kb | kk) != 0;
                            const uint64_t adv = (uint64_t)(kk * 2);
                            tc::umma_f16(d0, a_hi + adv, b_hi + adv, idesc, acc);
                            if (NTERMS == 3) {
                                const uint64_t a_lo = tc::umma_desc_k_sw128(w_addr + (2 + kb) * W_TILE);
                                const uint64_t b_lo = tc::umma_desc_k_sw128(b_addr + (2 + kb) * B_TILE);
                                tc::umma_f16(d1, a_hi + adv, b_lo + adv, idesc, acc);
                                tc::umma_f16(d1, a_lo + adv, b_hi + adv, idesc, 1);
                            }
                        }
                    }
                    tc::umma_commit(&tfull[sub]);
                }
                tc::umma_commit(&empty[s]);
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // ============================== epilogue: thread = output channel ==============================
        const int ew = warp - 4;
        const int o = ew * 32 + lane;
        const float bias = __ldg(b2 + o);
        const uint32_t lane_adr = (uint32_t)(ew * 32) << 16;
        int it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
#pragma unroll 1
            for (int sub = 0; sub < NSUB; ++sub) {
                tc::mbar_wait(&tfull[sub], it & 1);
                tc::tc_fence_after();
                const uint32_t ta = tmem_base + sub * ACC_STRIDE + lane_adr;
                float v[EN];
#pragma unroll
                for (int c0 = 0; c0 < EN; c0 += 16) {
                    uint32_t r0[16];
                    tmem_ld_32x16(ta + c0, r0);
                    if (NTERMS == 3) {
                        uint32_t r1[16];
                        tmem_ld_32x16(ta + 128 + c0, r1);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[c0 + i] = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i]));
                    } else {
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[c0 + i] = __uint_as_float(r0[i]);
                    }
                }
                tc::tc_fence_before();
                tc::mbar_arrive(&tempty[sub]);
#pragma unroll
                for (int g = 0; g < PTS_SUB; ++g) {
                    float m = v[g * KN];
#pragma unroll
                    for (int i = 1; i < KN; ++i) m = fmaxf(m, v[g * KN + i]);
                    const long long pt = tile * PTS_TILE + sub * PTS_SUB + g;
                    if (pt < total_pts) {
                        if (ZOUT) {              // per-edge pre-activations; max_k z == m + bias (rounding is monotone)
#pragma unroll
                            for (int i = 0; i < KN; ++i) z[(pt * KN + i) * C + o] = v[g * KN + i] + bias;
                        }
                        const float val = leaky(m + bias, slope);
                        x2[pt * ld2 + o] = val;
                        if (op2 != nullptr) {
                            const __half hi = __float2half_rn(val);
                            op2[pt * ldop + o] = hi;
                            op2[pt * ldop + op_plane + o] = __float2half_rn((val - __half2float(hi)) * 2048.f);
                        }
                    }
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem_base, C_::TMEM_COLS);
}

template <int NTERMS, int FMT>
int launch_dg_tc(const float* PQ, int ldpq, const int* idx, int N, long long total_pts, const float* W2, const float* b2,
                 float slope, float* x1, int ld1, float* x2, int ld2, __half* op1, __half* op2, int ldop, long long op_plane,
                 float* z, cudaStream_t stream) {
    using C_ = ECfg<NTERMS>;
    auto kern = z != nullptr ? edgeconv_dg_tc_kernel<NTERMS, FMT, true> : edgeconv_dg_tc_kernel<NTERMS, FMT, false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C_::SMEM) != cudaSuccess) return VCR_ERR_LAUNCH;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long ntiles = (total_pts + PTS_TILE - 1) / PTS_TILE;
    const int grid = (int)(ntiles < sms ? ntiles : sms);
    kern<<<grid, NTHREADS, C_::SMEM, stream>>>(PQ, ldpq, idx, N, total_pts, W2, b2, slope, x1, ld1, x2, ld2, op1, op2, ldop, op_plane,
                                               z);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

}  // namespace

// Tensor-core flavour of vcr_edgeconv_dg (same contract).  mode: 0 = fp16 3-term split ("h3", fp32 parity),
// 1 = fp16, 2 = bf16 single pass.  k must be 20; ldpq, ld1 multiples of 4; PQ, x1 16-byte aligned.
// z (optional): the convDG2 pre-activations of every edge, [total_pts * 20][128], the values x2 is the max of.
VCR_API int vcr_edgeconv_dg_tc(const float* PQ, int ldpq, const int* idx, int k, int N, long long total_pts,
                               const float* W2, const float* b2, float slope, int mode, float* x1, int ld1,
                               float* x2, int ld2, void* op1, void* op2, int ldop, long long op_plane, float* z,
                               cudaStream_t stream) {
    VCR_REQUIRE(PQ && idx && W2 && b2 && x1 && x2 && N > 0 && total_pts > 0);
    if (k != KN || mode < 0 || mode > 2 || slope < 0.f) return VCR_ERR_UNSUPPORTED;
    if ((ldpq & 3) || (ld1 & 3) || (reinterpret_cast<uintptr_t>(PQ) & 15) || (reinterpret_cast<uintptr_t>(x1) & 15) ||
        (reinterpret_cast<uintptr_t>(W2) & 15))
        return VCR_ERR_INVALID;
    // optional "h3" operand-format copies of x1 / x2 (fp16 hi, lo * 2^11 planes; both or neither)
    if ((op1 == nullptr) != (op2 == nullptr)) return VCR_ERR_INVALID;
    if (op1 && ((ldop & 3) || (op_plane & 3) || (reinterpret_cast<uintptr_t>(op1) & 7))) return VCR_ERR_INVALID;
    __half* o1 = reinterpret_cast<__half*>(op1);
    __half* o2 = reinterpret_cast<__half*>(op2);
    if (mode == 0) return launch_dg_tc<3, 0>(PQ, ldpq, idx, N, total_pts, W2, b2, slope, x1, ld1, x2, ld2, o1, o2, ldop, op_plane, z, stream);
    if (mode == 1) return launch_dg_tc<1, 0>(PQ, ldpq, idx, N, total_pts, W2, b2, slope, x1, ld1, x2, ld2, o1, o2, ldop, op_plane, z, stream);
    return launch_dg_tc<1, 1>(PQ, ldpq, idx, N, total_pts, W2, b2, slope, x1, ld1, x2, ld2, o1, o2, ldop, op_plane, z, stream);
}
