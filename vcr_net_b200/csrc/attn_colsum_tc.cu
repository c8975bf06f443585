// Partial-overlap key statistic on tcgen05 / TMEM / TMA (sm_100a): reference model/transformer.py:33-39
//     colsum[b, j] = sum over heads h and queries i of softmax_j(q_i . k_j / sqrt(d_k))
// (the column sums of the UNMASKED attention probabilities; their top int(Nk * overlap2) keys survive).
// The reference takes them from the materialised [B,h,Nq,Nk] probability tensor; the previous CUDA path wrote the
// scaled scores with the GEMM kernel (453 MB per 48 x 4 x 768 x 768 call) and read them back once.  Here nothing of
// size Nq x Nk touches HBM: a work item is (batch, head, 128-query tile) and makes TWO sweeps over the key tiles with
// the Q tile resident in shared memory --
//   sweep 0   S = Q K_j^T (tcgen05, 3-term fp16 split, S double-buffered in TMEM)  ->  running row max / row sum
//   sweep 1   S recomputed                                                          ->  p = exp2(s - M) / L, summed over
//             the 128 query rows of the tile (in-register butterfly transpose-reduce per warp, fixed order)
// and writes one partial column-sum vector per (item, lane quarter); a second tiny kernel reduces the partials in a
// fixed order (deterministic: the statistic feeds a top-K selection).
// The Q tile is copied smem -> TMEM once per item by the statistics warps (double-buffered, one item ahead) and the products
// take their A operand from tensor memory: with Q in shared memory a 128x128x16 instruction reads 8 KB per 64 cycles, the
// whole shared-memory port, and the K tiles arriving by TMA (64 KB per tile) stretched the tile from 1536 to ~2500 cycles.
// Warp roles as in attn_tc.cu: warp 0 TMA (Q once per item, K tiles through a 2-stage ring), warp 1 MMA issuer,
// warp 2 TMEM allocator, warps 4-19 statistics (thread = query row, four warps split the 128 key columns of a tile: the
// per-tile work of a warp is one dependent chain -- TMEM load, maximum, exp2, sum / transpose-reduce -- and with two warps
// per scheduler its latency, 2x the tile's tensor time, set the pace; four warps with half the chain each hide it).
#include "tc_common.cuh"

namespace {

constexpr int DK = 128;
constexpr int BQ = 128;
constexpr int BKV = 128;
constexpr int TILE = 128 * 128;                     // bytes of a [128 rows][64 x fp16] swizzled tile
constexpr int Q_BYTES = 4 * TILE;                   // 2 k-blocks x (hi, lo)
constexpr int K_STAGE = 4 * TILE;
constexpr int OFF_K = Q_BYTES;
constexpr int OFF_BAR = OFF_K + 2 * K_STAGE;
constexpr int OFF_XCH = OFF_BAR + 128;              // [4 column quarters][128 rows][2] (m, l)
constexpr int SMEM = OFF_XCH + 4 * 128 * 2 * 4 + 1024;
constexpr int NSTAT = 512;                          // statistics threads
constexpr int S_COLS = BKV;                         // one accumulator per S buffer (scale-input-d, see below)
constexpr int Q_COL0 = 2 * S_COLS;                  // Q buffer qb, plane pl, k-block kb at Q_COL0 + qb * 128 + pl * 64 + kb * 32
constexpr int TMEM_COLS = 512;
constexpr float kLog2e = 1.4426950408889634f;

struct ColsumParams {
    int B, H, Nq, Nk;
    float scale_log2;
    float* part;          // [B][H * nqt * 4][Nk]
    const int* nq_len;    // ragged batch: queries / keys of item b (clamped to [0, Nq] / [0, Nk]); null in a uniform batch
    const int* nk_len;
};

// Ragged batch: the items a CTA walks are those whose query tile holds a query of its batch item; every role walks the same
// list.  Item b's partial slabs are laid out as the item alone lays them out, (hh * nqt_b + qt) * 4 + ew with
// nqt_b = ceil(nq_b / 128), so colsum_reduce_kernel adds them in the pair-alone order.
struct ItemLens {
    int nq, nk, nqt, nkt;
};
template <bool RAGGED>
__device__ __forceinline__ ItemLens colsum_item(const ColsumParams& p, int b) {
    ItemLens r;
    r.nq = RAGGED ? min(max(__ldg(p.nq_len + b), 0), p.Nq) : p.Nq;
    r.nk = RAGGED ? min(max(__ldg(p.nk_len + b), 0), p.Nk) : p.Nk;
    r.nqt = (r.nq + BQ - 1) / BQ;
    r.nkt = (r.nk + BKV - 1) / BKV;
    return r;
}

__device__ __forceinline__ float ex2_approx(float x) { return tc::ex2_mufu(x); }

template <bool RAGGED>
__global__ void __launch_bounds__(128 + NSTAT, 1)
attn_colsum_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK, const ColsumParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* q_full = bars + 0;  uint64_t* q_empty = bars + 1;  uint64_t* qt_full = bars + 11;
    uint64_t* k_full = bars + 2;  uint64_t* k_empty = bars + 4;      // [2] each
    uint64_t* s_full = bars + 6;  uint64_t* s_empty = bars + 8;      // [2] each
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nqt = (p.Nq + BQ - 1) / BQ;
    const int nkt_u = (p.Nk + BKV - 1) / BKV;                // a uniform batch: every item's key tiles
    const long long items = (long long)p.B * p.H * nqt;
    // first item at or after `it` (stride gridDim.x) with a live query tile; every item in a uniform batch
    auto next_item = [&](long long it) -> long long {
        if (RAGGED)
            for (; it < items; it += gridDim.x)
                if ((int)(it % nqt) < colsum_item<true>(p, (int)(it / nqt) / p.H).nqt) break;
        return it;
    };

    if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tmQ); tc::tma_prefetch_desc(&tmK); }
    if (warp == 1 && lane == 0) {
        tc::mbar_init(q_full, 1); tc::mbar_init(q_empty, NSTAT); tc::mbar_init(qt_full, NSTAT);
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&k_full[s], 1); tc::mbar_init(&k_empty[s], 1);
            tc::mbar_init(&s_full[s], 1); tc::mbar_init(&s_empty[s], NSTAT);
        }
        tc::fence_barrier_init();
    }
    if (warp == 2) { tc::tmem_alloc(tmem_slot, TMEM_COLS); tc::tmem_relinquish(); }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ============================== TMA producer ==============================
        if (tc::elect_one()) {
            uint32_t g = 0, w = 0;
            auto load_q = [&](long long it) {                   // Q of the item into the staging tile
                const int qt = (int)(it % nqt);
                const int bh = (int)(it / nqt);
                const int hh = bh % p.H, b = bh / p.H;
                tc::mbar_expect_tx(q_full, Q_BYTES);
#pragma unroll
                for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                    for (int pl = 0; pl < 2; ++pl)
                        tc::tma_load_3d(smem + (kb * 2 + pl) * TILE, &tmQ, q_full, hh * DK + kb * 64, b * p.Nq + qt * BQ, pl);
            };
            const long long first = next_item(blockIdx.x);
            if (first < items) load_q(first);
            for (long long it = first; it < items; it = next_item(it + gridDim.x), ++w) {
                const int bh = (int)(it / nqt);
                const int hh = bh % p.H, b = bh / p.H;
                const int nkt = RAGGED ? colsum_item<true>(p, b).nkt : nkt_u;
                const long long nx = next_item(it + gridDim.x);
                if (nx < items) {                               // next item's Q: staging is free once this item's Q is in TMEM
                    tc::mbar_wait(q_empty, w & 1);
                    load_q(nx);
                }
                for (int sw = 0; sw < 2; ++sw)
                    for (int j = 0; j < nkt; ++j, ++g) {
                        const int s = g & 1;
                        uint8_t* st = smem + OFF_K + s * K_STAGE;
                        tc::mbar_wait(&k_empty[s], ((g >> 1) & 1) ^ 1);
                        tc::mbar_expect_tx(&k_full[s], K_STAGE);
#pragma unroll
                        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                            for (int pl = 0; pl < 2; ++pl)
                                tc::tma_load_3d(st + (kb * 2 + pl) * TILE, &tmK, &k_full[s], hh * DK + kb * 64,
                                                b * p.Nk + j * BKV, pl);
                    }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::umma_idesc(BQ, BKV, 0);
            uint32_t g = 0, w = 0;
            for (long long it = next_item(blockIdx.x); it < items; it = next_item(it + gridDim.x), ++w) {
                const int nkt = RAGGED ? colsum_item<true>(p, (int)(it / nqt) / p.H).nkt : nkt_u;
                tc::mbar_wait(qt_full, w & 1);
                tc::tc_fence_after();
                const uint32_t q_tm = tmem_base + Q_COL0 + (w & 1) * 128;
                for (int t = 0; t < 2 * nkt; ++t, ++g) {
                    const int s = g & 1;
                    const uint32_t ph = (g >> 1) & 1;
                    tc::mbar_wait(&k_full[s], ph);
                    tc::mbar_wait(&s_empty[s], ph ^ 1);
                    tc::tc_fence_after();
                    const uint32_t k_addr = tc::smem_u32(smem + OFF_K + s * K_STAGE);
                    // one accumulator: every correction product (hi*lo' + lo*hi', carrying 2^11) first, then the main products,
                    // the first of them with tcgen05.mma's scale-input-d = 11 (Q and the key tile are resident for the whole
                    // d_k = 128 product) -- half the TMEM read per tile in both sweeps
                    const uint32_t d0 = tmem_base + s * S_COLS;
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * 2) * TILE);
                        const uint64_t k_lo = tc::umma_desc_k_sw128(k_addr + (kb * 2 + 1) * TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            tc::umma_f16_ts(d0, q_tm + kb * 32 + kk * 8, k_lo + adv, idesc, (kb | kk) != 0);
                            tc::umma_f16_ts(d0, q_tm + 64 + kb * 32 + kk * 8, k_hi + adv, idesc, 1);
                        }
                    }
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * 2) * TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            if ((kb | kk) == 0) tc::umma_f16_ts_scale_d11(d0, q_tm, k_hi + adv, idesc);
                            else tc::umma_f16_ts(d0, q_tm + kb * 32 + kk * 8, k_hi + adv, idesc, 1);
                        }
                    }
                    tc::umma_commit(&s_full[s]);
                    tc::umma_commit(&k_empty[s]);
                }
            }
        }
    } else if (warp >= 4) {
        // ============================== statistics ==============================
        const int ew = warp & 3, cq = (warp - 4) >> 2;          // TMEM lane quarter, column quarter of the tile
        const int rloc = ew * 32 + lane;
        const uint32_t lane_adr = (uint32_t)(ew * 32) << 16;
        float* xch = reinterpret_cast<float*>(smem + OFF_XCH);  // [4][128][2]
        const float sc = p.scale_log2;
        // Q of item number w: staging tile cq = kb * 2 + pl (row rloc) -> TMEM buffer w & 1
        auto copy_q = [&](uint32_t w) {
            tc::mbar_wait(q_full, w & 1);
            const uint8_t* row = smem + cq * TILE + rloc * 128;
            uint32_t r[32];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint4 x = *reinterpret_cast<const uint4*>(row + ((c ^ (rloc & 7)) * 16));
                r[4 * c] = x.x; r[4 * c + 1] = x.y; r[4 * c + 2] = x.z; r[4 * c + 3] = x.w;
            }
            tc::tmem_st_32x32(tmem_base + Q_COL0 + (w & 1) * 128 + lane_adr + (cq & 1) * 64 + (cq >> 1) * 32, r);
            tc::tmem_st_wait();
            tc::tc_fence_before();
            tc::mbar_arrive(qt_full);
            tc::mbar_arrive(q_empty);
        };
        uint32_t g = 0, w = 0;
        const long long first = next_item(blockIdx.x);
        if (first < items) copy_q(0);
        for (long long it = first; it < items; it = next_item(it + gridDim.x), ++w) {
            const int qt = (int)(it % nqt);
            const int bh = (int)(it / nqt);
            const int hh = bh % p.H, b = bh / p.H;
            const ItemLens li = RAGGED ? colsum_item<true>(p, b) : ItemLens{p.Nq, p.Nk, nqt, nkt_u};
            const int nkt = li.nkt, nk = li.nk;
            const bool row_ok = qt * BQ + rloc < li.nq;
            float m = -INFINITY, l = 0.f;        // sweep 0: running max / sum;  sweep 1: -M and 1/L
            for (int sw = 0; sw < 2; ++sw) {
                for (int j = 0; j < nkt; ++j, ++g) {
                    const int sb = g & 1;
                    tc::mbar_wait(&s_full[sb], (g >> 1) & 1);
                    tc::tc_fence_after();
                    const int key0 = j * BKV + cq * 32;         // first key of this warp's 32 columns
                    if (key0 < nk) {                            // warp-uniform
                        float x[32];
                        {
                            const uint32_t sa = tmem_base + sb * S_COLS + lane_adr + cq * 32;
                            uint32_t r0[32];
                            tc::tmem_ld_32x32(sa, r0);
                            tc::tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(r0[i]);   // raw scores: sc > 0 is applied in the fma below
                        }
                        if (key0 + 32 > nk) {
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (key0 + i >= nk) x[i] = -INFINITY;
                        }
                        if (sw == 0) {
                            float c4[4] = {x[0], x[1], x[2], x[3]};             // four independent chains
#pragma unroll
                            for (int i = 4; i < 32; ++i) c4[i & 3] = fmaxf(c4[i & 3], x[i]);
                            const float cm = fmaxf(fmaxf(c4[0], c4[1]), fmaxf(c4[2], c4[3])) * sc;
                            if (cm > m) { l *= ex2_approx(m - cm); m = cm; }     // m = -inf on the first chunk: l = 0 * 0
                            const float nm = -m;
                            float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                            for (int i = 0; i < 32; ++i) a4[i & 3] += ex2_approx(fmaf(x[i], sc, nm));
                            l += (a4[0] + a4[1]) + (a4[2] + a4[3]);
                        } else {
                            const float w = row_ok ? l : 0.f;   // rows past Nq (next batch / padding) contribute nothing
#pragma unroll
                            for (int i = 0; i < 32; ++i) x[i] = ex2_approx(fmaf(x[i], sc, m)) * w;
                            // transpose-reduce: afterwards x[0] of lane c is the sum over the warp's 32 rows of column c
#pragma unroll
                            for (int off = 16; off >= 1; off >>= 1) {
                                const bool up = (lane & off) != 0;
#pragma unroll
                                for (int i = 0; i < off; ++i) {
                                    const float send = up ? x[i] : x[i + off];
                                    const float keep = up ? x[i + off] : x[i];
                                    x[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                                }
                            }
                            const int key = key0 + lane;
                            if (key < nk)
                                p.part[((size_t)b * (p.H * nqt * 4) + ((size_t)(hh * li.nqt + qt) * 4 + ew)) * p.Nk + key] = x[0];
                        }
                    }
                    tc::tc_fence_before();
                    tc::mbar_arrive(&s_empty[sb]);
                }
                if (sw == 0) {
                    // combine the row statistics of the four column quarters in a fixed order (quarter barrier, 128 threads)
                    xch[(cq * 128 + rloc) * 2 + 0] = m;
                    xch[(cq * 128 + rloc) * 2 + 1] = l;
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + ew) : "memory");
                    float mm[4], ll[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) { mm[u] = xch[(u * 128 + rloc) * 2 + 0]; ll[u] = xch[(u * 128 + rloc) * 2 + 1]; }
                    const float M = fmaxf(fmaxf(mm[0], mm[1]), fmaxf(mm[2], mm[3]));
                    float L = 0.f;                               // a quarter without keys: m = -inf, l = 0
#pragma unroll
                    for (int u = 0; u < 4; ++u) L += ll[u] * ex2_approx(mm[u] - M);
                    m = -M;
                    l = 1.f / L;
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + ew) : "memory");         // xch reusable
                    // next item's Q into the other TMEM buffer (its previous user's products retired an item ago)
                    if (next_item(it + gridDim.x) < items) copy_q(w + 1);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

// out[b, j] = sum_s part[b, s, j] in slab order.  Ragged batch (RAGGED): item b adds its first H * nqt_b * 4 slabs and
// writes 0 past its keys.
template <bool RAGGED>
__global__ void colsum_reduce_kernel(const float* __restrict__ part, int slabs, int n, float* __restrict__ out,
                                     ColsumParams p) {
    const int b = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int ns = slabs;
    if (RAGGED) {
        const ItemLens li = colsum_item<true>(p, b);
        if (j >= li.nk) { out[(size_t)b * n + j] = 0.f; return; }
        ns = p.H * li.nqt * 4;
    }
    const float* pb = part + (size_t)b * slabs * n + j;
    float acc = 0.f;
    for (int s = 0; s < ns; ++s) acc += pb[(size_t)s * n];
    out[(size_t)b * n + j] = acc;
}

static int attn_colsum_launch(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                              const int* nq, const int* nk, int B, int H, int Nq, int Nk, int dk, float scale, float* out,
                              void* workspace, size_t workspace_bytes, cudaStream_t stream);

}  // namespace

VCR_API size_t vcr_attn_colsum_workspace_bytes(int B, int H, int Nq, int Nk) {
    return (size_t)B * H * ((Nq + BQ - 1) / BQ) * 4 * Nk * sizeof(float);
}

namespace {
int attn_colsum_launch(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                       const int* nq, const int* nk, int B, int H, int Nq, int Nk, int dk, float scale, float* out,
                       void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    if (dk != DK) return VCR_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < vcr_attn_colsum_workspace_bytes(B, H, Nq, Nk)) return VCR_ERR_WORKSPACE;
    CUtensorMap tq, tk;
    int rc = vcr_make_operand_tmap(&tq, Q, H * DK, (long long)B * Nq, ldq, q_plane, 2, BQ);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tk, K, H * DK, (long long)B * Nk, ldk, k_plane, 2, BKV);
    if (rc != VCR_OK) return rc;
    ColsumParams p;
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.scale_log2 = scale * kLog2e;
    p.part = reinterpret_cast<float*>(workspace);
    p.nq_len = nq; p.nk_len = nk;
    const bool ragged = nq != nullptr;
    auto kern = ragged ? attn_colsum_tc_kernel<true> : attn_colsum_tc_kernel<false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess)
        return VCR_ERR_LAUNCH;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int nqt = (Nq + BQ - 1) / BQ;
    const long long items = (long long)B * H * nqt;
    const int grid = (int)(items < sms ? items : sms);
    kern<<<grid, 128 + NSTAT, SMEM, stream>>>(tq, tk, p);
    VCR_CHECK_LAUNCH();
    if (ragged) colsum_reduce_kernel<true><<<dim3(vcr_cdiv(Nk, 128), B), 128, 0, stream>>>(p.part, H * nqt * 4, Nk, out, p);
    else colsum_reduce_kernel<false><<<dim3(vcr_cdiv(Nk, 128), B), 128, 0, stream>>>(p.part, H * nqt * 4, Nk, out, p);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
}  // namespace

// Q: operand buffer [2 planes][B*Nq][ldq] ("h3": fp16 hi, lo * 2^11), head hh in columns [hh*128, hh*128+128);
// K: [2][B*Nk][ldk] likewise.  out [B, Nk] = column sums over heads and queries of softmax_j(q.k * scale).
VCR_API int vcr_attn_colsum_tc(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                               int B, int H, int Nq, int Nk, int dk, float scale, float* out, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(Q && K && out && B > 0 && H > 0 && Nq > 0 && Nk > 0 && B <= 65535);
    return attn_colsum_launch(Q, ldq, q_plane, K, ldk, k_plane, nullptr, nullptr, B, H, Nq, Nk, dk, scale, out, workspace,
                              workspace_bytes, stream);
}

// Ragged batch: item b has nq[b] queries and nk[b] keys (clamped to [0, Nq] / [0, Nk]) in its Nq / Nk rows.  Keys past nk[b]
// are -inf in the row maxima and sums, key tiles past them are not loaded, query tiles past nq[b] are skipped.  out [B, Nk]:
// columns < nk[b] equal vcr_attn_colsum_tc on the item alone, bit for bit; the rest are 0.  Workspace as vcr_attn_colsum_tc.
VCR_API int vcr_attn_colsum_tc_ragged(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                                      const int* nq, const int* nk, int B, int H, int Nq, int Nk, int dk, float scale,
                                      float* out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(Q && K && nq && nk && out && B > 0 && H > 0 && Nq > 0 && Nk > 0 && B <= 65535);
    return attn_colsum_launch(Q, ldq, q_plane, K, ldk, k_plane, nq, nk, B, H, Nq, Nk, dk, scale, out, workspace,
                              workspace_bytes, stream);
}
