// Flash-style multi-head attention on tcgen05 / TMEM / TMA (sm_100a): softmax(Q K^T * scale) V for
// d_k = 128 without ever writing the [B,h,Nq,Nk] score or probability tensors (reference
// model/transformer.py:13-55 materialises both in fp32: 2 x 268 MB per call at B=16, N=1024).
//
// Two kernels share this file: flash_attn_ts_kernel (the default, further down: Q and P are tcgen05.mma A operands held in
// TENSOR memory) and flash_attn_tc_kernel (every operand in shared memory, three softmax organisations; kept selectable).
// Work item = (batch, head, 128-query tile); persistent CTAs walk the items.  Per 64-key tile:
//   warp 1 (one elected thread)  S = Q K_j^T          tcgen05.mma 128x64x16, S in TMEM (double-buffered)
//   warps 4-11 (2 threads per query row, 32 keys each) online softmax: tcgen05.ld S -> exp2 -> P (fp16 hi/lo) -> smem / TMEM
//   warp 1                        O += P V_j           tcgen05.mma 128x128x16, O stays in TMEM
//   warp 0 (one elected thread)  TMA: Q once per item, {K_j, V^T_j} through a 2-stage ring
// QK^T of tile j+1 is issued before P V of tile j, so the tensor core works while the softmax warps
// are busy.  O is rescaled LAZILY: the running maximum used for exp2 only moves when a row's new maximum
// exceeds it by more than 2^8 (exact after the final 1/l normalisation, no overflow in fp16 P), so the
// TMEM read-modify-write of O is rare.
//
// Precision: NTERMS = 3 is the fp32-parity mode -- Q, K, V and P are carried as fp16 (hi, lo*2^11) pairs,
// each product is hi*hi + 2^-11 (hi*lo + lo*hi).  O keeps main and correction terms in separate TMEM
// accumulators (see gemm_tc.cu) because it accumulates across key tiles; S = Q K_j^T is complete within one
// tile, so its correction products are issued first and the first main product rescales the accumulator with
// tcgen05.mma's scale-input-d = 11: one accumulator, half the per-tile TMEM read.  NTERMS = 1: single fp16 / bf16 pass.
// Optional key mask keep[B,Nk] (partial overlap, model/transformer.py:48-52): masked keys get -1e9.
#include <atomic>
#include "tc_common.cuh"

namespace {

constexpr int DK = 128;           // head dim
constexpr int BQ = 128;           // queries per work item
constexpr int BKV = 64;           // keys per inner tile
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kRescaleThreshold = 8.0f;   // log2 units

struct AttnParams {
    int B, H, Nq, Nk;
    float scale_log2;             // softmax scale * log2(e)
    const uint8_t* keep;          // [B, Nk] or null
    const int* nq_len;            // ragged batch (flash_attn_ts_kernel only): queries of item b, or null
    const int* nk_len;            // keys of item b, or null (a uniform batch)
    __half* O; int ldo; long long o_plane;
    float* lse;                   // [B, H, Nq] log2-domain log-sum-exp, or null
    int out_bf16;
};

template <int NTERMS>
struct ACfg {
    static constexpr int PL = NTERMS == 3 ? 2 : 1;
    static constexpr int Q_TILE = BQ * 128;                     // [128 rows][64 elems] 16 KB
    static constexpr int K_TILE = BKV * 128;                    // [64 keys][64 elems]   8 KB
    static constexpr int V_TILE = DK * 128;                     // [128 d][64 keys]     16 KB
    static constexpr int P_TILE = BQ * 128;                     // [128 rows][64 keys]  16 KB
    static constexpr int Q_BYTES = 2 * PL * Q_TILE;             // 2 k-blocks of d_k
    static constexpr int KV_STAGE = 2 * PL * K_TILE + PL * V_TILE;
    static constexpr int P_BYTES = 2 * P_TILE;                  // P (hi | lo); also the write-out staging area of the 8 softmax warps (8 x 4 KB)
    static constexpr int NSTAGE = 2;
    static constexpr int OFF_KV = Q_BYTES;
    static constexpr int OFF_P = OFF_KV + NSTAGE * KV_STAGE;
    static constexpr int OFF_BAR = OFF_P + P_BYTES;
    static constexpr int OFF_XCH = OFF_BAR + 256;               // row max / sum exchange between the warp pair
    static constexpr int SLACK = 768;                           // alignment slack (the dynamic smem base is 1 KB aligned in practice; checked)
    static constexpr int SMEM = OFF_XCH + 2048 + SLACK;
    static constexpr int S_COLS = PL * BKV;                     // per S buffer: D0 | D1
    static constexpr int O_COL0 = 2 * S_COLS;
    static constexpr int TMEM_COLS = NTERMS == 3 ? 512 : 256;
};

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// NWQ = softmax warps per TMEM lane quarter (2: a warp owns 32 key columns of its 32 rows, 384 threads; 4: 16 columns,
// 640 threads).  The softmax is a chain of dependent phases (TMEM load, max, exchange, exp2, split, store) per tile, and
// with two warps per scheduler the chain's latency, not its ~380 instructions, set the tile period (ncu: tensor pipe
// 50 % active, stalls on scoreboards and the pair barrier); four warps per scheduler with half the chain each hide it.
// Key tiles item (b, query tile qt) walks: all of them in a uniform batch; in a ragged batch those up to item b's key count,
// and a single tile for a query tile wholly past the item's queries (its output rows are written as zeros).
__device__ __forceinline__ int attn_item_kv_tiles(const AttnParams& p, int b, int qt) {
    if (p.nk_len == nullptr) return (p.Nk + BKV - 1) / BKV;
    if (qt * BQ >= vcr_item_len(p.nq_len, b, p.Nq, 1)) return 1;
    return (vcr_item_len(p.nk_len, b, p.Nk, 1) + BKV - 1) / BKV;
}

__device__ __forceinline__ int ordered_key(float f) { const int b = __float_as_int(f); return b >= 0 ? b : b ^ 0x7fffffff; }
__device__ __forceinline__ float ordered_val(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }
constexpr int kNegInfKey = (int)0x807fffffu;         // ordered_key(-inf)

template <int NTERMS, int FMT, int NWQ, bool PING>
__global__ void __launch_bounds__(128 + 128 * NWQ, 1)
flash_attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
    using C_ = ACfg<NTERMS>;
    constexpr int PL = C_::PL;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    if ((int)(smem - smem_raw) > C_::SLACK) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C_::OFF_BAR);
    uint64_t* q_full = bars + 0;  uint64_t* q_empty = bars + 1;
    uint64_t* k_full = bars + 2;              // [2]  K and V^T tiles share a smem stage but are released
    uint64_t* k_empty = bars + 4;             // [2]  separately: K_j is free right after Q K_j^T (one tile ahead of
    uint64_t* v_full = bars + 14;             // [2]  the softmax), V_j only after P V_j, so the K load of tile j+2
    uint64_t* v_empty = bars + 16;            // [2]  never waits for the P V chain.
    uint64_t* s_full = bars + 6;              // [2]
    uint64_t* s_empty = bars + 8;             // [2]
    uint64_t* p_full = bars + 10; uint64_t* p_empty = bars + 11;
    uint64_t* o_full = bars + 12; uint64_t* o_empty = bars + 13;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nqt = (p.Nq + BQ - 1) / BQ;
    const int nkv = (p.Nk + BKV - 1) / BKV;
    const long long items = (long long)p.B * p.H * nqt;

    if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tmQ); tc::tma_prefetch_desc(&tmK); tc::tma_prefetch_desc(&tmV); }
    if (warp == 1 && lane == 0) {
        tc::mbar_init(q_full, 1); tc::mbar_init(q_empty, 1);
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&k_full[s], 1); tc::mbar_init(&k_empty[s], 1);
            tc::mbar_init(&v_full[s], 1); tc::mbar_init(&v_empty[s], 1);
            tc::mbar_init(&s_full[s], 1);  tc::mbar_init(&s_empty[s], PING ? 128 : 128 * NWQ);
        }
        tc::mbar_init(p_full, PING ? 128 : 128 * NWQ); tc::mbar_init(p_empty, 1);
        tc::mbar_init(o_full, 1);   tc::mbar_init(o_empty, 128 * NWQ);
        tc::fence_barrier_init();
    }
    if (warp == 2) { tc::tmem_alloc(tmem_slot, C_::TMEM_COLS); tc::tmem_relinquish(); }
    if (NWQ == 4 && warp == 3) {                      // row-maximum slots (3 x 128 ordered-int keys) start at -inf
        int* mx = reinterpret_cast<int*>(smem + C_::OFF_XCH);
        for (int i = lane; i < 3 * 128; i += 32) mx[i] = kNegInfKey;
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ============================== TMA producer ==============================
        if (tc::elect_one()) {
            uint32_t g = 0, w = 0;
            for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
                const int qt = (int)(it % nqt);
                const int bh = (int)(it / nqt);
                const int hh = bh % p.H, b = bh / p.H;
                tc::mbar_wait(q_empty, (w & 1) ^ 1);
                tc::mbar_expect_tx(q_full, C_::Q_BYTES);
#pragma unroll
                for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl)
                        tc::tma_load_3d(smem + (kb * PL + pl) * C_::Q_TILE, &tmQ, q_full, hh * DK + kb * 64,
                                        b * p.Nq + qt * BQ, pl);
                for (int j = 0; j < nkv; ++j, ++g) {
                    const int s = g & 1;
                    uint8_t* st = smem + C_::OFF_KV + s * C_::KV_STAGE;
                    tc::mbar_wait(&k_empty[s], ((g >> 1) & 1) ^ 1);
                    tc::mbar_expect_tx(&k_full[s], 2 * PL * C_::K_TILE);
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                        for (int pl = 0; pl < PL; ++pl)
                            tc::tma_load_3d(st + (kb * PL + pl) * C_::K_TILE, &tmK, &k_full[s], hh * DK + kb * 64,
                                            b * p.Nk + j * BKV, pl);
                    tc::mbar_wait(&v_empty[s], ((g >> 1) & 1) ^ 1);
                    tc::mbar_expect_tx(&v_full[s], PL * C_::V_TILE);
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl)
                        tc::tma_load_3d(st + 2 * PL * C_::K_TILE + pl * C_::V_TILE, &tmV, &v_full[s], j * BKV,
                                        (b * p.H + hh) * DK, pl);
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc_qk = tc::umma_idesc(BQ, BKV, FMT);
            constexpr uint32_t idesc_pv = tc::umma_idesc(BQ, DK, FMT);
            const uint32_t q_addr = tc::smem_u32(smem);
            const uint32_t p_addr = tc::smem_u32(smem + C_::OFF_P);
            uint32_t g_qk = 0, g_pv = 0, w = 0;
            auto issue_qk = [&]() {
                const int s = g_qk & 1;
                const uint32_t ph = (g_qk >> 1) & 1;
                tc::mbar_wait(&k_full[s], ph);
                tc::mbar_wait(&s_empty[s], ph ^ 1);
                tc::tc_fence_after();
                const uint32_t k_addr = tc::smem_u32(smem + C_::OFF_KV + s * C_::KV_STAGE);
                const uint32_t d0 = tmem_base + s * C_::S_COLS;
                if (NTERMS == 3) {
                    // Q and K_j are both resident for the whole product (d_k = 128 = two k-blocks), so every correction term
                    // (hi*lo' + lo*hi', carrying 2^11) goes first and the main terms follow into the SAME accumulator, the
                    // first of them with scale-input-d = 11: S = sum hi*hi' + 2^-11 sum corr, one 64-column tile to read.
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t q_hi = tc::umma_desc_k_sw128(q_addr + (kb * PL) * C_::Q_TILE);
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
                        const uint64_t q_lo = tc::umma_desc_k_sw128(q_addr + (kb * PL + 1) * C_::Q_TILE);
                        const uint64_t k_lo = tc::umma_desc_k_sw128(k_addr + (kb * PL + 1) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            tc::umma_f16(d0, q_hi + adv, k_lo + adv, idesc_qk, (kb | kk) != 0);
                            tc::umma_f16(d0, q_lo + adv, k_hi + adv, idesc_qk, 1);
                        }
                    }
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t q_hi = tc::umma_desc_k_sw128(q_addr + (kb * PL) * C_::Q_TILE);
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            if ((kb | kk) == 0) tc::umma_f16_scale_d11(d0, q_hi + adv, k_hi + adv, idesc_qk);
                            else tc::umma_f16(d0, q_hi + adv, k_hi + adv, idesc_qk, 1);
                        }
                    }
                } else {
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t q_hi = tc::umma_desc_k_sw128(q_addr + (kb * PL) * C_::Q_TILE);
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            tc::umma_f16(d0, q_hi + (uint64_t)(kk * 2), k_hi + (uint64_t)(kk * 2), idesc_qk, (kb | kk) != 0);
                    }
                }
                tc::umma_commit(&s_full[s]);
                tc::umma_commit(&k_empty[s]);                    // K_j consumed
                ++g_qk;
            };
            for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
                tc::mbar_wait(q_full, w & 1);
                tc::tc_fence_after();
                issue_qk();
                for (int j = 0; j < nkv; ++j) {
                    if (j + 1 < nkv) issue_qk();
                    else tc::umma_commit(q_empty);               // Q tile free once every QK^T of the item retired
                    const int s = g_pv & 1;
                    tc::mbar_wait(p_full, g_pv & 1);
                    tc::mbar_wait(&v_full[s], (g_pv >> 1) & 1);
                    if (j == 0) tc::mbar_wait(o_empty, (w & 1) ^ 1);
                    tc::tc_fence_after();
                    const uint32_t v_addr = tc::smem_u32(smem + C_::OFF_KV + s * C_::KV_STAGE + 2 * PL * C_::K_TILE);
                    const uint32_t o0 = tmem_base + C_::O_COL0, o1 = o0 + DK;
                    const uint64_t p_hi = tc::umma_desc_k_sw128(p_addr);
                    const uint64_t v_hi = tc::umma_desc_k_sw128(v_addr);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (j | kk) != 0;
                        const uint64_t adv = (uint64_t)(kk * 2);
                        tc::umma_f16(o0, p_hi + adv, v_hi + adv, idesc_pv, acc);
                        if (NTERMS == 3) {
                            const uint64_t p_lo = tc::umma_desc_k_sw128(p_addr + C_::P_TILE);
                            const uint64_t v_lo = tc::umma_desc_k_sw128(v_addr + C_::V_TILE);
                            tc::umma_f16(o1, p_hi + adv, v_lo + adv, idesc_pv, acc);
                            tc::umma_f16(o1, p_lo + adv, v_hi + adv, idesc_pv, 1);
                        }
                    }
                    tc::umma_commit(&v_empty[s]);                // V_j consumed
                    tc::umma_commit(p_empty);                    // P buffer free / O safe to rescale
                    ++g_pv;
                }
                tc::umma_commit(o_full);
            }
        }
    } else if (PING && warp >= 4) {
        // ============================== softmax + output, two groups alternating key tiles ==============================
        // The per-tile softmax is a chain of dependent hand-offs (S ready -> TMEM load -> max -> exp2 -> P store -> fence ->
        // mbarrier -> MMA issue -> commit -> P buffer free ...), and with every softmax warp on the SAME tile that chain,
        // ~2x the tile's tensor time, set the tile period (ncu: tensor pipe 42-49 % active, issue slots 32 %).  Here the 8
        // warps form two groups of 4 (one warp per TMEM lane quarter, a thread owns a whole 64-key row of the tile: no
        // column split, no per-tile exchange barrier); group g takes tiles j = g, g+2, ...  The only per-tile dependence
        // between consecutive tiles is the running reference maximum: the owner of tile j publishes it right after its row
        // maximum is known (named barrier arrive), the owner of tile j+1 picks it up (named barrier sync) -- so tile j+1's
        // TMEM load and maximum overlap tile j's exp2 / split / P store, and its P store only waits for P V_j.
        // Each group keeps its own partial row sum l relative to the maximum it last saw; the partials are brought to the
        // final maximum and added once per item.
        constexpr int OW = DK / 2;                    // O columns per warp at write-out
        const int qq = warp & 3, grp = (warp - 4) >> 2;
        const int rloc = qq * 32 + lane;
        const uint32_t lane_adr = (uint32_t)(qq * 32) << 16;
        constexpr int obf = FMT;              // output / P format is the operand format: compile-time, no per-element branches
        uint8_t* p_smem = smem + C_::OFF_P + rloc * 128;
        float* xch = reinterpret_cast<float*>(smem + C_::OFF_XCH);      // [0,128): reference maximum, [128,384): l exchange
        auto quarter_bar = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + qq) : "memory"); };
        // turn hand-off between the two warps of a lane quarter: ids 5.. (group 0 -> 1), 9.. (group 1 -> 0)
        auto turn_arrive = [&]() { asm volatile("bar.arrive %0, 64;" ::"r"(5 + 4 * grp + qq) : "memory"); };
        auto turn_wait = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(5 + 4 * (grp ^ 1) + qq) : "memory"); };
        uint32_t w = 0, gbase = 0;
        for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w, gbase += (uint32_t)nkv) {
            const int qt = (int)(it % nqt);
            const int bh = (int)(it / nqt);
            const int hh = bh % p.H, b = bh / p.H;
            const uint8_t* keep = p.keep ? p.keep + (size_t)b * p.Nk : nullptr;
            float m_seen = 0.f, l = 0.f;
            bool seen = false;
            for (int j = grp; j < nkv; j += 2) {
                const uint32_t g = gbase + (uint32_t)j;
                const int sb = g & 1;
                uint32_t km0 = 0xffffffffu, km1 = 0xffffffffu;
                if (keep != nullptr) {
                    const int key = j * BKV + lane;
                    km0 = __ballot_sync(0xffffffffu, key < p.Nk && __ldg(keep + key) != 0);
                    km1 = __ballot_sync(0xffffffffu, key + 32 < p.Nk && __ldg(keep + key + 32) != 0);
                }
                tc::mbar_wait(&s_full[sb], (g >> 1) & 1);
                tc::tc_fence_after();
                float s[BKV];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t sa = tmem_base + sb * C_::S_COLS + lane_adr + h * 32;
                    uint32_t r0[32];
                    tc::tmem_ld_32x32(sa, r0);                   // one accumulator in every mode (scale-input-d, see issue_qk)
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) s[h * 32 + i] = __uint_as_float(r0[i]);
                }
                tc::tc_fence_before();
                tc::mbar_arrive(&s_empty[sb]);                   // S buffer may be overwritten by QK^T of tile j+2
                // ---- (mask,) row maximum of the tile ----
                float sc = p.scale_log2;
                if (keep != nullptr || j * BKV + BKV > p.Nk) {    // warp-uniform: ragged or masked tile
#pragma unroll
                    for (int i = 0; i < BKV; ++i) {
                        float x = s[i] * sc;
                        const int key = j * BKV + i;
                        const uint32_t km = i < 32 ? km0 : km1;
                        if (key >= p.Nk) x = -INFINITY;
                        else if (!((km >> (i & 31)) & 1u)) x = -1e9f * kLog2e;
                        s[i] = x;
                    }
                    sc = 1.f;
                }
                float mt = s[0];
#pragma unroll
                for (int i = 1; i < BKV; ++i) mt = fmaxf(mt, s[i]);
                mt *= sc;                                         // sc > 0
                // ---- my turn: reference maximum (lazy: it only moves when exceeded by more than 2^8) ----
                float m_ref = mt, o_factor = 1.f;
                bool need = false;
                if (j > 0) {
                    turn_wait();
                    const float m_prev = xch[rloc];
                    if (mt > m_prev + kRescaleThreshold) { o_factor = ex2_approx(m_prev - mt); need = true; }
                    else m_ref = m_prev;
                }
                if (j + 1 < nkv) { xch[rloc] = m_ref; turn_arrive(); }
                if (seen && m_seen != m_ref) l *= ex2_approx(m_seen - m_ref);     // my partial sum follows the reference
                m_seen = m_ref; seen = true;
                const float neg_m = -m_ref;
                float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
                for (int i = 0; i < BKV; i += 2) {
                    s[i] = ex2_approx(fmaf(s[i], sc, neg_m));         rs0 += s[i];
                    s[i + 1] = ex2_approx(fmaf(s[i + 1], sc, neg_m)); rs1 += s[i + 1];
                }
                l += rs0 + rs1;
                // ---- P buffer free (P V of the previous tile retired), also the point where O may be touched ----
                tc::mbar_wait(p_empty, (g & 1) ^ 1);
                if (__any_sync(0xffffffffu, need)) {
                    tc::tc_fence_after();
#pragma unroll 1
                    for (int c = 0; c < PL * DK; c += 32) {       // all of this lane quarter's O columns (D0, and D1)
                        const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + c;
                        uint32_t r[32];
                        tc::tmem_ld_32x32(oa, r);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * o_factor);
                        tc::tmem_st_32x32(oa, r);
                    }
                    tc::tmem_st_wait();
                    tc::tc_fence_before();
                }
                // ---- P (fp16 hi / lo*2^11) into the swizzled K-major A-operand tile: 8 16-byte chunks per plane ----
#pragma unroll
                for (int c = 0; c < BKV / 8; ++c) {
                    const int pos = (c ^ (rloc & 7)) * 16;
                    uint32_t wv[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) wv[q] = tc::pack_h2(s[c * 8 + 2 * q], s[c * 8 + 2 * q + 1], obf);
                    *reinterpret_cast<uint4*>(p_smem + pos) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                    if (NTERMS == 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            wv[q] = tc::pack_h2(tc::lo_part(s[c * 8 + 2 * q], obf), tc::lo_part(s[c * 8 + 2 * q + 1], obf), obf);
                        *reinterpret_cast<uint4*>(p_smem + C_::P_TILE + pos) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                    }
                }
                tc::fence_proxy_async();                          // generic-proxy smem writes -> visible to the tensor core
                tc::mbar_arrive(p_full);
            }
            // ---- item done: bring both partial sums to the final reference maximum (the last tile's), add them ----
            if (((nkv - 1) & 1) == grp) xch[rloc] = m_seen;       // owner of the last tile
            quarter_bar();
            const float m_fin = xch[rloc];
            if (seen && m_seen != m_fin) l *= ex2_approx(m_seen - m_fin);
            xch[128 + grp * 128 + rloc] = l;
            quarter_bar();
            l = xch[128 + rloc] + xch[256 + rloc];
            quarter_bar();                                        // the exchange area is reused by the next item
            tc::mbar_wait(o_full, w & 1);
            tc::tc_fence_after();
            const int q = qt * BQ + rloc;
            const bool q_ok = q < p.Nq;
            const float inv_l = 1.f / l;
            const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + grp * OW;
            __half* orow = p.O + ((size_t)b * p.Nq + q) * p.ldo + hh * DK + grp * OW;
#pragma unroll 1
            for (int c = 0; c < OW; c += 32) {
                uint32_t r0[32];
                float v[32];
                tc::tmem_ld_32x32(oa + c, r0);
                if (NTERMS == 3) {
                    uint32_t r1[32];
                    tc::tmem_ld_32x32(oa + DK + c, r1);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i])) * inv_l;
                } else {
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r0[i]) * inv_l;
                }
                if (q_ok) {
#pragma unroll
                    for (int i = 0; i < 32; i += 8) {
                        uint32_t wv[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) wv[t] = tc::pack_h2(v[i + 2 * t], v[i + 2 * t + 1], obf);
                        *reinterpret_cast<uint4*>(orow + c + i) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                        if (NTERMS == 3) {
#pragma unroll
                            for (int t = 0; t < 4; ++t)
                                wv[t] = tc::pack_h2(tc::lo_part(v[i + 2 * t], obf), tc::lo_part(v[i + 2 * t + 1], obf), obf);
                            *reinterpret_cast<uint4*>(orow + p.o_plane + c + i) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                        }
                    }
                }
            }
            if (p.lse && q_ok && grp == 0) p.lse[((size_t)b * p.H + hh) * p.Nq + q] = m_fin + log2f(l);
            tc::tc_fence_before();
            tc::mbar_arrive(o_empty);
        }
    } else if (warp >= 4) {
        // ============================== softmax + output ==============================
        // 4 * NWQ warps: warp w owns query rows (TMEM lanes) 32*(w%4)..+32 and key columns CW*hf..+CW of the tile
        // (hf = (w-4)/4, CW = 64 / NWQ).  The warps of a row quarter agree on the running maximum through smem (quarter
        // barrier): NWQ = 2 exchanges fp32 values in two alternating slots, NWQ = 4 takes an atomic max of order-preserving
        // integer keys in three rotating slots (the 2 KB exchange area cannot hold 2 x 4 x 128 floats; the slot of tile
        // g + 2 is reset after the barrier of tile g, when every reader of tile g - 1 has passed).  The partial sums l
        // are combined once per item in a fixed order.  Each warp rescales / writes out its DK / NWQ columns of O.
        constexpr int CW = BKV / NWQ;                 // key columns per warp
        constexpr int OW = DK / NWQ;                  // O columns per warp
        constexpr int OC = NWQ == 4 ? 16 : 32;        // O write-out chunk (register budget: 96 / thread at 640 threads)
        const int qq = warp & 3, hf = (warp - 4) >> 2;
        const int rloc = qq * 32 + lane;
        const uint32_t lane_adr = (uint32_t)(qq * 32) << 16;
        constexpr int obf = FMT;              // output / P format is the operand format: compile-time, no per-element branches
        uint8_t* p_smem = smem + C_::OFF_P + rloc * 128;
        float* xch = reinterpret_cast<float*>(smem + C_::OFF_XCH);      // NWQ = 2: [2 slots][2][128]; l exchange: [NWQ][128]
        int* mxk = reinterpret_cast<int*>(smem + C_::OFF_XCH);          // NWQ = 4: [3 slots][128] ordered keys
        auto pair_bar = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + qq), "r"(32 * NWQ) : "memory"); };
        uint32_t g = 0, w = 0;
        int g3 = 0;                                                       // g % 3
        for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
            const int qt = (int)(it % nqt);
            const int bh = (int)(it / nqt);
            const int hh = bh % p.H, b = bh / p.H;
            const uint8_t* keep = p.keep ? p.keep + (size_t)b * p.Nk : nullptr;
            float m_used = -INFINITY, l = 0.f;
            for (int j = 0; j < nkv; ++j, ++g) {
                const int sb = g & 1;
                // kept keys of this warp's columns as a bit mask: one byte per lane, requested before the wait on S
                uint32_t km = 0xffffffffu;
                if (keep != nullptr) {
                    const int key = j * BKV + hf * CW + (lane & (CW - 1));
                    km = __ballot_sync(0xffffffffu, key < p.Nk && __ldg(keep + key) != 0);
                }
                tc::mbar_wait(&s_full[sb], (g >> 1) & 1);
                tc::tc_fence_after();
                float s[CW];
                {
                    const uint32_t sa = tmem_base + sb * C_::S_COLS + lane_adr + hf * CW;
                    uint32_t r0[CW];
                    if (CW == 32) tc::tmem_ld_32x32(sa, reinterpret_cast<uint32_t(&)[32]>(r0));
                    else tc::tmem_ld_32x16(sa, reinterpret_cast<uint32_t(&)[16]>(r0));
                    tc::tmem_ld_wait();                          // one accumulator in every mode (scale-input-d, see issue_qk)
#pragma unroll
                    for (int i = 0; i < CW; ++i) s[i] = __uint_as_float(r0[i]);
                }
                tc::tc_fence_before();
                tc::mbar_arrive(&s_empty[sb]);                   // S buffer may be overwritten by QK^T of tile j+2
                // ---- (mask,) partial row maximum ----
                const int key0 = j * BKV + hf * CW;
                float sc = p.scale_log2;                          // exp2(s*sc - m) below
                if (keep != nullptr || j * BKV + BKV > p.Nk) {    // warp-uniform: ragged or masked tile
#pragma unroll
                    for (int i = 0; i < CW; ++i) {
                        float x = s[i] * sc;
                        const int key = key0 + i;
                        if (key >= p.Nk) x = -INFINITY;
                        else if (!((km >> i) & 1u)) x = -1e9f * kLog2e;
                        s[i] = x;
                    }
                    sc = 1.f;
                }
                float mt = s[0];
#pragma unroll
                for (int i = 1; i < CW; ++i) mt = fmaxf(mt, s[i]);
                mt *= sc;                                         // sc > 0
                if (NWQ == 2) {
                    float* slot = xch + (g & 1) * 256;
                    slot[hf * 128 + rloc] = mt;
                    pair_bar();
                    mt = fmaxf(mt, slot[(hf ^ 1) * 128 + rloc]);
                } else {
                    atomicMax(mxk + g3 * 128 + rloc, ordered_key(mt));
                    pair_bar();
                    mt = ordered_val(mxk[g3 * 128 + rloc]);
                    const int g3n = g3 == 0 ? 2 : g3 - 1;         // (g + 2) % 3: last read at tile g - 1
                    if (hf == 0) mxk[g3n * 128 + rloc] = kNegInfKey;
                    g3 = g3 == 2 ? 0 : g3 + 1;
                }
                float factor = 1.f;
                bool need = false;
                if (j == 0) {
                    m_used = mt;
                } else if (mt > m_used + kRescaleThreshold) {
                    factor = ex2_approx(m_used - mt);
                    m_used = mt;
                    need = true;
                }
                const float neg_m = -m_used;
                float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
                for (int i = 0; i < CW; i += 2) {
                    s[i] = ex2_approx(fmaf(s[i], sc, neg_m));         rs0 += s[i];
                    s[i + 1] = ex2_approx(fmaf(s[i + 1], sc, neg_m)); rs1 += s[i + 1];
                }
                l = l * factor + (rs0 + rs1);
                // ---- P buffer free (P V of the previous tile retired), also the point where O may be touched ----
                tc::mbar_wait(p_empty, (g & 1) ^ 1);
                if (__any_sync(0xffffffffu, need)) {
                    tc::tc_fence_after();
#pragma unroll 1
                    for (int c = 0; c < PL * OW; c += 32) {       // this warp's OW columns of D0 (and of D1)
                        const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + (c >= OW ? DK - OW : 0) + hf * OW + c;
                        uint32_t r[32];
                        tc::tmem_ld_32x32(oa, r);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * factor);
                        tc::tmem_st_32x32(oa, r);
                    }
                    tc::tmem_st_wait();
                    tc::tc_fence_before();
                }
                // ---- P (fp16 hi / lo*2^11) into the swizzled K-major A-operand tile: CW / 8 16-byte chunks per plane ----
#pragma unroll
                for (int c = 0; c < CW / 8; ++c) {
                    const int pos = ((hf * (CW / 8) + c) ^ (rloc & 7)) * 16;
                    uint32_t wv[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) wv[q] = tc::pack_h2(s[c * 8 + 2 * q], s[c * 8 + 2 * q + 1], obf);
                    *reinterpret_cast<uint4*>(p_smem + pos) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                    if (NTERMS == 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            wv[q] = tc::pack_h2(tc::lo_part(s[c * 8 + 2 * q], obf), tc::lo_part(s[c * 8 + 2 * q + 1], obf), obf);
                        *reinterpret_cast<uint4*>(p_smem + C_::P_TILE + pos) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                    }
                }
                tc::fence_proxy_async();                          // generic-proxy smem writes -> visible to the tensor core
                tc::mbar_arrive(p_full);
            }
            // ---- item done: combine the partial sums (fixed order), O / l -> operand-format output (this warp's OW columns) ----
            pair_bar();
            xch[hf * 128 + rloc] = l;
            pair_bar();
            if (NWQ == 2) {
                l += xch[(hf ^ 1) * 128 + rloc];
            } else {
                l = (xch[rloc] + xch[128 + rloc]) + (xch[256 + rloc] + xch[384 + rloc]);
            }
            pair_bar();
            if (NWQ == 4) {                                       // the l exchange overwrote the maximum slots
                if (hf == 0) { mxk[rloc] = kNegInfKey; mxk[128 + rloc] = kNegInfKey; mxk[256 + rloc] = kNegInfKey; }
                pair_bar();
                g3 = 0;
            }
            tc::mbar_wait(o_full, w & 1);
            tc::tc_fence_after();
            const int q = qt * BQ + rloc;
            const bool q_ok = q < p.Nq;
            const float inv_l = 1.f / l;
            const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + hf * OW;
            if constexpr (NWQ == 2) {
                // A thread owns 64 columns of one query row: written straight from registers, every 16-byte store of a warp
                // lands in a different 128-byte line (32 L1 wavefronts per instruction, ~6 us per item: the whole per-item
                // bubble of the kernel).  Staged through this warp's 4 KB of the (idle) P buffer instead, swizzled like the P
                // tile, and read back so that a store instruction covers 4 complete rows of 128 bytes.
                float v[OW];
#pragma unroll
                for (int c = 0; c < OW; c += 32) {
                    uint32_t r0[32];
                    tc::tmem_ld_32x32(oa + c, r0);
                    if (NTERMS == 3) {
                        uint32_t r1[32];
                        tc::tmem_ld_32x32(oa + DK + c, r1);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            v[c + i] = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i])) * inv_l;
                    } else {
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[c + i] = __uint_as_float(r0[i]) * inv_l;
                    }
                }
                tc::tc_fence_before();
                tc::mbar_arrive(o_empty);                         // O is in registers: P V_0 of the next item may overwrite it
                uint8_t* stg = smem + C_::OFF_P + (hf * 4 + qq) * 4096;          // [32 rows][128 B]
                const int q0 = qt * BQ + qq * 32;
                __half* obase = p.O + ((size_t)b * p.Nq + q0) * p.ldo + hh * DK + hf * OW + (lane & 7) * 8;
#pragma unroll
                for (int pl = 0; pl < PL; ++pl) {
#pragma unroll
                    for (int c = 0; c < OW / 8; ++c) {
                        uint32_t wv[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const float a0 = v[c * 8 + 2 * t], a1 = v[c * 8 + 2 * t + 1];
                            wv[t] = pl == 0 ? tc::pack_h2(a0, a1, obf) : tc::pack_h2(tc::lo_part(a0, obf), tc::lo_part(a1, obf), obf);
                        }
                        *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) * 16)) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                    }
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int row = i * 4 + (lane >> 3);
                        const uint4 x = *reinterpret_cast<const uint4*>(stg + row * 128 + (((lane & 7) ^ (row & 7)) * 16));
                        if (q0 + row < p.Nq) *reinterpret_cast<uint4*>(obase + (size_t)row * p.ldo + pl * p.o_plane) = x;
                    }
                    __syncwarp();
                }
                if (p.lse && q_ok && hf == 0) p.lse[((size_t)b * p.H + hh) * p.Nq + q] = m_used + log2f(l);
                continue;                                         // (the next P store of this row quarter follows a pair barrier)
            }
            __half* orow = p.O + ((size_t)b * p.Nq + q) * p.ldo + hh * DK + hf * OW;
#pragma unroll 1
            for (int c = 0; c < OW; c += OC) {
                uint32_t r0[OC];
                float v[OC];
                if (OC == 32) tc::tmem_ld_32x32(oa + c, reinterpret_cast<uint32_t(&)[32]>(r0));
                else tc::tmem_ld_32x16(oa + c, reinterpret_cast<uint32_t(&)[16]>(r0));
                if (NTERMS == 3) {
                    uint32_t r1[OC];
                    if (OC == 32) tc::tmem_ld_32x32(oa + DK + c, reinterpret_cast<uint32_t(&)[32]>(r1));
                    else tc::tmem_ld_32x16(oa + DK + c, reinterpret_cast<uint32_t(&)[16]>(r1));
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < OC; ++i) v[i] = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i])) * inv_l;
                } else {
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < OC; ++i) v[i] = __uint_as_float(r0[i]) * inv_l;
                }
                if (q_ok) {
#pragma unroll
                    for (int i = 0; i < OC; i += 8) {
                        uint32_t wv[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) wv[t] = tc::pack_h2(v[i + 2 * t], v[i + 2 * t + 1], obf);
                        *reinterpret_cast<uint4*>(orow + c + i) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                        if (NTERMS == 3) {
#pragma unroll
                            for (int t = 0; t < 4; ++t)
                                wv[t] = tc::pack_h2(tc::lo_part(v[i + 2 * t], obf), tc::lo_part(v[i + 2 * t + 1], obf), obf);
                            *reinterpret_cast<uint4*>(orow + p.o_plane + c + i) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                        }
                    }
                }
            }
            if (p.lse && q_ok && hf == 0) p.lse[((size_t)b * p.H + hh) * p.Nq + q] = m_used + log2f(l);
            tc::tc_fence_before();
            tc::mbar_arrive(o_empty);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem_base, C_::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------------------------------
// Organisation 3 ("operands in TMEM"): the A side of BOTH products lives in tensor memory.
// tcgen05.mma reads a shared-memory A operand once per instruction, and the 3-term split issues 24 QK^T instructions of
// 128x64x16 per key tile: 6 KB of operand reads per 32-cycle instruction against a ~128 B/cycle shared-memory port, so the
// all-smem tile costs 2054 cycles of tensor issue against a 1536-cycle floor (scripts/mma_rate.cu, profiles/r02_mma_rate.txt:
// QK 128x64x16 from smem 1.76x its floor, P V 1.12x; with A in TMEM both run at 1.00x).  Here
//   Q (hi | lo, 128 TMEM columns) is copied smem -> TMEM once per item by the softmax warps (tcgen05.st), and
//   P is written by tcgen05.st straight over the S tile it was computed from (fp16 pairs: hi 32 | lo 32 columns),
// so only K_j and V_j are read from shared memory by the tensor core, the P tile no longer crosses shared memory at all, and
// the Q staging buffer is free for the NEXT item's Q as soon as the copy is done.  TMEM: S/P 2 x 64 | O 2 x 128 | Q 128 = 512.
// An S buffer is reused by Q K_{j+2}^T, which is issued after P V_j (same thread, the tensor pipe runs in issue order), so no
// "S empty" barrier is needed; P V_j completion is only waited for in the rare O rescale.
// ---------------------------------------------------------------------------------------------------------------------
template <int NTERMS>
struct TCfg {
    static constexpr int PL = NTERMS == 3 ? 2 : 1;
    static constexpr int Q_TILE = BQ * 128, K_TILE = BKV * 128, V_TILE = DK * 128;
    static constexpr int Q_BYTES = 2 * PL * Q_TILE;
    static constexpr int KV_STAGE = 2 * PL * K_TILE + PL * V_TILE;
    static constexpr int OFF_KV = Q_BYTES;
    static constexpr int OFF_STG = OFF_KV + 2 * KV_STAGE;       // write-out staging: 8 warps x 4 KB
    static constexpr int OFF_BAR = OFF_STG + 8 * 4096;
    static constexpr int OFF_XCH = OFF_BAR + 256;
    static constexpr int SLACK = 768;
    static constexpr int SMEM = OFF_XCH + 2048 + SLACK;
    static constexpr int O_COL0 = 128;
    static constexpr int Q_COL0 = O_COL0 + PL * DK;             // plane pl, k-block kb at Q_COL0 + pl * 64 + kb * 32
};

template <int NTERMS, int FMT>
__global__ void __launch_bounds__(384, 1)
flash_attn_ts_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
    using C_ = TCfg<NTERMS>;
    constexpr int PL = C_::PL;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    if ((int)(smem - smem_raw) > C_::SLACK) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C_::OFF_BAR);
    uint64_t* q_full = bars + 0;  uint64_t* q_empty = bars + 1;  uint64_t* qt_full = bars + 2;
    uint64_t* k_full = bars + 4;  uint64_t* k_empty = bars + 6;
    uint64_t* v_full = bars + 8;  uint64_t* v_empty = bars + 10;
    uint64_t* s_full = bars + 12;
    uint64_t* p_full = bars + 14; uint64_t* pv_done = bars + 15;
    uint64_t* o_full = bars + 16; uint64_t* o_empty = bars + 17;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nqt = (p.Nq + BQ - 1) / BQ;
    const long long items = (long long)p.B * p.H * nqt;

    if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tmQ); tc::tma_prefetch_desc(&tmK); tc::tma_prefetch_desc(&tmV); }
    if (warp == 1 && lane == 0) {
        tc::mbar_init(q_full, 1); tc::mbar_init(q_empty, 256); tc::mbar_init(qt_full, 256);
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&k_full[s], 1); tc::mbar_init(&k_empty[s], 1);
            tc::mbar_init(&v_full[s], 1); tc::mbar_init(&v_empty[s], 1);
            tc::mbar_init(&s_full[s], 1);
        }
        tc::mbar_init(p_full, 256); tc::mbar_init(pv_done, 1);
        tc::mbar_init(o_full, 1);   tc::mbar_init(o_empty, 256);
        tc::fence_barrier_init();
    }
    if (warp == 2) { tc::tmem_alloc(tmem_slot, 512); tc::tmem_relinquish(); }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ============================== TMA producer ==============================
        if (tc::elect_one()) {
            uint32_t g = 0, w = 0;
            for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
                const int qt = (int)(it % nqt);
                const int bh = (int)(it / nqt);
                const int hh = bh % p.H, b = bh / p.H;
                tc::mbar_wait(q_empty, (w & 1) ^ 1);
                tc::mbar_expect_tx(q_full, C_::Q_BYTES);
#pragma unroll
                for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl)
                        tc::tma_load_3d(smem + (kb * PL + pl) * C_::Q_TILE, &tmQ, q_full, hh * DK + kb * 64,
                                        b * p.Nq + qt * BQ, pl);
                const int nkv = attn_item_kv_tiles(p, b, qt);
                for (int j = 0; j < nkv; ++j, ++g) {
                    const int s = g & 1;
                    uint8_t* st = smem + C_::OFF_KV + s * C_::KV_STAGE;
                    tc::mbar_wait(&k_empty[s], ((g >> 1) & 1) ^ 1);
                    tc::mbar_expect_tx(&k_full[s], 2 * PL * C_::K_TILE);
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                        for (int pl = 0; pl < PL; ++pl)
                            tc::tma_load_3d(st + (kb * PL + pl) * C_::K_TILE, &tmK, &k_full[s], hh * DK + kb * 64,
                                            b * p.Nk + j * BKV, pl);
                    tc::mbar_wait(&v_empty[s], ((g >> 1) & 1) ^ 1);
                    tc::mbar_expect_tx(&v_full[s], PL * C_::V_TILE);
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl)
                        tc::tma_load_3d(st + 2 * PL * C_::K_TILE + pl * C_::V_TILE, &tmV, &v_full[s], j * BKV,
                                        (b * p.H + hh) * DK, pl);
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc_qk = tc::umma_idesc(BQ, BKV, FMT);
            constexpr uint32_t idesc_pv = tc::umma_idesc(BQ, DK, FMT);
            const uint32_t q_tm = tmem_base + C_::Q_COL0;
            uint32_t g_qk = 0, g_pv = 0, w = 0;
            auto issue_qk = [&]() {
                const int s = g_qk & 1;
                tc::mbar_wait(&k_full[s], (g_qk >> 1) & 1);
                tc::tc_fence_after();
                const uint32_t k_addr = tc::smem_u32(smem + C_::OFF_KV + s * C_::KV_STAGE);
                const uint32_t d0 = tmem_base + s * BKV;
                if (NTERMS == 3) {
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
                        const uint64_t k_lo = tc::umma_desc_k_sw128(k_addr + (kb * PL + 1) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            tc::umma_f16_ts(d0, q_tm + kb * 32 + kk * 8, k_lo + adv, idesc_qk, (kb | kk) != 0);
                            tc::umma_f16_ts(d0, q_tm + 64 + kb * 32 + kk * 8, k_hi + adv, idesc_qk, 1);
                        }
                    }
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            if ((kb | kk) == 0) tc::umma_f16_ts_scale_d11(d0, q_tm, k_hi + adv, idesc_qk);
                            else tc::umma_f16_ts(d0, q_tm + kb * 32 + kk * 8, k_hi + adv, idesc_qk, 1);
                        }
                    }
                } else {
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const uint64_t k_hi = tc::umma_desc_k_sw128(k_addr + (kb * PL) * C_::K_TILE);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            tc::umma_f16_ts(d0, q_tm + kb * 32 + kk * 8, k_hi + (uint64_t)(kk * 2), idesc_qk, (kb | kk) != 0);
                    }
                }
                tc::umma_commit(&s_full[s]);
                tc::umma_commit(&k_empty[s]);
                ++g_qk;
            };
            for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
                const int nkv = attn_item_kv_tiles(p, (int)(it / nqt) / p.H, (int)(it % nqt));
                tc::mbar_wait(qt_full, w & 1);
                tc::tc_fence_after();
                issue_qk();
                for (int j = 0; j < nkv; ++j) {
                    if (j + 1 < nkv) issue_qk();
                    const int s = g_pv & 1;
                    tc::mbar_wait(p_full, g_pv & 1);
                    tc::mbar_wait(&v_full[s], (g_pv >> 1) & 1);
                    if (j == 0) tc::mbar_wait(o_empty, (w & 1) ^ 1);
                    tc::tc_fence_after();
                    const uint32_t v_addr = tc::smem_u32(smem + C_::OFF_KV + s * C_::KV_STAGE + 2 * PL * C_::K_TILE);
                    const uint32_t o0 = tmem_base + C_::O_COL0, o1 = o0 + DK;
                    const uint32_t p_tm = tmem_base + s * BKV;                    // P over S: hi 32 columns | lo 32 columns
                    const uint64_t v_hi = tc::umma_desc_k_sw128(v_addr);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (j | kk) != 0;
                        const uint64_t adv = (uint64_t)(kk * 2);
                        tc::umma_f16_ts(o0, p_tm + kk * 8, v_hi + adv, idesc_pv, acc);
                        if (NTERMS == 3) {
                            const uint64_t v_lo = tc::umma_desc_k_sw128(v_addr + C_::V_TILE);
                            tc::umma_f16_ts(o1, p_tm + kk * 8, v_lo + adv, idesc_pv, acc);
                            tc::umma_f16_ts(o1, p_tm + 32 + kk * 8, v_hi + adv, idesc_pv, 1);
                        }
                    }
                    tc::umma_commit(&v_empty[s]);
                    tc::umma_commit(pv_done);
                    ++g_pv;
                }
                tc::umma_commit(o_full);
            }
        }
    } else if (warp >= 4) {
        // ============================== softmax + output (8 warps, two per TMEM lane quarter) ==============================
        // warp w owns query rows (TMEM lanes) 32*(w%4)..+32 and key columns 32*hf..+32 of the tile, hf = (w-4)/4.  (Four warps
        // per quarter with 16 columns each measured 0.95x: the tile is not paced by the length of a warp's chain.)
        constexpr int CW = BKV / 2, OW = DK / 2;
        const int qq = warp & 3, hf = (warp - 4) >> 2;
        const int rloc = qq * 32 + lane;
        const uint32_t lane_adr = (uint32_t)(qq * 32) << 16;
        constexpr int obf = FMT;
        float* xch = reinterpret_cast<float*>(smem + C_::OFF_XCH);      // [2 slots][2][128] maxima; l exchange [2][128]
        auto pair_bar = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + qq) : "memory"); };
        // Q of item number w: smem staging (row rloc, k-block hf, every plane) -> TMEM
        auto copy_q = [&](uint32_t w) {
            tc::mbar_wait(q_full, w & 1);
#pragma unroll
            for (int pl = 0; pl < PL; ++pl) {
                const int kb = hf;
                const uint8_t* row = smem + (kb * PL + pl) * C_::Q_TILE + rloc * 128;
                uint32_t r[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint4 x = *reinterpret_cast<const uint4*>(row + ((c ^ (rloc & 7)) * 16));
                    r[4 * c] = x.x; r[4 * c + 1] = x.y; r[4 * c + 2] = x.z; r[4 * c + 3] = x.w;
                }
                tc::tmem_st_32x32(tmem_base + C_::Q_COL0 + lane_adr + pl * 64 + kb * 32, r);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            tc::mbar_arrive(qt_full);
            tc::mbar_arrive(q_empty);
        };
        uint32_t g = 0, w = 0;
        if ((long long)blockIdx.x < items) copy_q(0);
        for (long long it = blockIdx.x; it < items; it += gridDim.x, ++w) {
            const int qt = (int)(it % nqt);
            const int bh = (int)(it / nqt);
            const int hh = bh % p.H, b = bh / p.H;
            const uint8_t* keep = p.keep ? p.keep + (size_t)b * p.Nk : nullptr;
            const int nkv = attn_item_kv_tiles(p, b, qt);
            const int nk_b = vcr_item_len(p.nk_len, b, p.Nk, 1);
            const bool q_live = qt * BQ < vcr_item_len(p.nq_len, b, p.Nq, 1);
            float m_used = -INFINITY, l = 0.f;
            for (int j = 0; j < nkv; ++j, ++g) {
                const int sb = g & 1;
                // additive score bias of key (this warp's column `lane`): 0 = kept, -1e9 (log2 domain) = masked, -inf = past
                // the item's keys; requested before the wait on S, broadcast column by column with shuffles below
                const bool biased = keep != nullptr || j * BKV + BKV > nk_b;      // warp-uniform
                float bias_l = 0.f;
                if (biased) {
                    const int key = j * BKV + hf * CW + lane;
                    if (key >= nk_b) bias_l = -INFINITY;
                    else if (keep != nullptr && __ldg(keep + key) == 0) bias_l = -1e9f * kLog2e;
                }
                tc::mbar_wait(&s_full[sb], (g >> 1) & 1);
                tc::tc_fence_after();
                const uint32_t s_tm = tmem_base + sb * BKV + lane_adr;
                float s[CW];
                {
                    uint32_t r0[CW];
                    tc::tmem_ld_32x32(s_tm + hf * CW, r0);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < CW; ++i) s[i] = __uint_as_float(r0[i]);
                }
                float sc = p.scale_log2;
                if (biased) {                                     // one shuffle + one fma per score (the bias is the same for every row)
#pragma unroll
                    for (int i = 0; i < CW; ++i) {
                        const float bi = __shfl_sync(0xffffffffu, bias_l, i);
                        // a key past the item is -inf whatever its score (the padding of a ragged batch may hold anything)
                        s[i] = bi == -INFINITY ? -INFINITY : fmaf(s[i], sc, bi);
                    }
                    sc = 1.f;
                }
                float mt;
                {
                    float m4[4] = {s[0], s[1], s[2], s[3]};       // four independent chains
#pragma unroll
                    for (int i = 4; i < CW; ++i) m4[i & 3] = fmaxf(m4[i & 3], s[i]);
                    mt = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * sc;
                }
                {
                    float* slot = xch + (g & 1) * 256;
                    slot[hf * 128 + rloc] = mt;
                    pair_bar();                                   // also: both warps of the quarter have read their S columns
                    mt = fmaxf(mt, slot[(hf ^ 1) * 128 + rloc]);
                }
                float factor = 1.f;
                bool need = false;
                if (j == 0) {
                    m_used = mt;
                } else if (mt > m_used + kRescaleThreshold) {
                    factor = ex2_approx(m_used - mt);
                    m_used = mt;
                    need = true;
                }
                const float neg_m = -m_used;
                float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
                for (int i = 0; i < CW; i += 2) {
                    s[i] = ex2_approx(fmaf(s[i], sc, neg_m));         rs0 += s[i];
                    s[i + 1] = ex2_approx(fmaf(s[i + 1], sc, neg_m)); rs1 += s[i + 1];
                }
                l = l * factor + (rs0 + rs1);
                if (__any_sync(0xffffffffu, need)) {              // rare: O may only be touched once P V of the previous tile retired
                    tc::mbar_wait(pv_done, (g & 1) ^ 1);
                    tc::tc_fence_after();
#pragma unroll 1
                    for (int c = 0; c < PL * OW; c += 32) {
                        const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + (c >= OW ? DK - OW : 0) + hf * OW + c;
                        uint32_t r[32];
                        tc::tmem_ld_32x32(oa, r);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * factor);
                        tc::tmem_st_32x32(oa, r);
                    }
                }
                // ---- P (fp16 hi / lo * 2^11 pairs) over this warp's share of the S tile ----
                {
                    uint32_t ph[CW / 2];
#pragma unroll
                    for (int i = 0; i < CW / 2; ++i) ph[i] = tc::pack_h2(s[2 * i], s[2 * i + 1], obf);
                    tc::tmem_st_32x16(s_tm + hf * (CW / 2), ph);
                    if (NTERMS == 3) {
#pragma unroll
                        for (int i = 0; i < CW / 2; ++i) ph[i] = tc::pack_h2(tc::lo_part(s[2 * i], obf), tc::lo_part(s[2 * i + 1], obf), obf);
                        tc::tmem_st_32x16(s_tm + 32 + hf * (CW / 2), ph);
                    }
                }
                tc::tmem_st_wait();
                tc::tc_fence_before();
                tc::mbar_arrive(p_full);
            }
            // ---- item done: combine the partial sums, prefetch-copy the next Q, O / l -> operand-format output ----
            pair_bar();
            xch[hf * 128 + rloc] = l;
            pair_bar();
            l += xch[(hf ^ 1) * 128 + rloc];
            pair_bar();
            if (it + gridDim.x < items) copy_q(w + 1);            // every Q K^T of this item has retired (s_full of its last tile)
            tc::mbar_wait(o_full, w & 1);
            tc::tc_fence_after();
            const int q = qt * BQ + rloc;
            const bool q_ok = q < p.Nq;
            const float inv_l = 1.f / l;
            const uint32_t oa = tmem_base + C_::O_COL0 + lane_adr + hf * OW;
            float v[OW];
#pragma unroll
            for (int c = 0; c < OW; c += 32) {
                uint32_t r0[32];
                tc::tmem_ld_32x32(oa + c, r0);
                if (NTERMS == 3) {
                    uint32_t r1[32];
                    tc::tmem_ld_32x32(oa + DK + c, r1);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        v[c + i] = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i])) * inv_l;
                } else {
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[c + i] = __uint_as_float(r0[i]) * inv_l;
                }
            }
            if (!q_live) {                                        // query tile past the item's queries: rows written as 0
#pragma unroll
                for (int i = 0; i < OW; ++i) v[i] = 0.f;
            }
            tc::tc_fence_before();
            tc::mbar_arrive(o_empty);
            uint8_t* stg = smem + C_::OFF_STG + (hf * 4 + qq) * 4096;            // [32 rows][128 B], this warp's
            const int q0 = qt * BQ + qq * 32;
            __half* obase = p.O + ((size_t)b * p.Nq + q0) * p.ldo + hh * DK + hf * OW + (lane & 7) * 8;
#pragma unroll
            for (int pl = 0; pl < PL; ++pl) {
#pragma unroll
                for (int c = 0; c < OW / 8; ++c) {
                    uint32_t wv[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const float a0 = v[c * 8 + 2 * t], a1 = v[c * 8 + 2 * t + 1];
                        wv[t] = pl == 0 ? tc::pack_h2(a0, a1, obf) : tc::pack_h2(tc::lo_part(a0, obf), tc::lo_part(a1, obf), obf);
                    }
                    *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) * 16)) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                }
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int row = i * 4 + (lane >> 3);
                    const uint4 x = *reinterpret_cast<const uint4*>(stg + row * 128 + (((lane & 7) ^ (row & 7)) * 16));
                    if (q0 + row < p.Nq) *reinterpret_cast<uint4*>(obase + (size_t)row * p.ldo + pl * p.o_plane) = x;
                }
                __syncwarp();
            }
            if (p.lse && q_ok && hf == 0) p.lse[((size_t)b * p.H + hh) * p.Nq + q] = m_used + log2f(l);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem_base, 512);
}

template <int NTERMS, int FMT>
int launch_attn_ts(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnParams& p, cudaStream_t st) {
    using C_ = TCfg<NTERMS>;
    auto kern = flash_attn_ts_kernel<NTERMS, FMT>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C_::SMEM) != cudaSuccess) return VCR_ERR_LAUNCH;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long items = (long long)p.B * p.H * ((p.Nq + BQ - 1) / BQ);
    const int grid = (int)(items < sms ? items : sms);
    kern<<<grid, 384, C_::SMEM, st>>>(tq, tk, tv, p);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

template <int NTERMS, int FMT, int NWQ, bool PING = false>
int launch_attn(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnParams& p, cudaStream_t st) {
    using C_ = ACfg<NTERMS>;
    auto kern = flash_attn_tc_kernel<NTERMS, FMT, NWQ, PING>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C_::SMEM) != cudaSuccess) return VCR_ERR_LAUNCH;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long items = (long long)p.B * p.H * ((p.Nq + BQ - 1) / BQ);
    const int grid = (int)(items < sms ? items : sms);
    kern<<<grid, 128 + 128 * NWQ, C_::SMEM, st>>>(tq, tk, tv, p);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

}  // namespace

static std::atomic<int> g_vcr_flash_warps{3};      // tuning knob (see vcr_set_flash_warps)

// Organisation of the flash attention kernel: 3 (default) = Q and P in tensor memory, 8 softmax warps (flash_attn_ts_kernel);
// 2 = every operand in shared memory, 8 warps on every tile, two per TMEM lane quarter splitting the key columns; 4 = 16
// warps, four per quarter; 1 = two groups of 4 warps alternating key tiles.  Measured at 48 x 4 x 768 x 768 in the parity
// mode (profiles/r02_flash_organisations.txt): 139.5 / 155.1 / 176.3 / 176.0 us.  Process-wide; returns the previous setting.
// 2 and 3 are bit-identical; the others agree to fp32 rounding of the row sums.
VCR_API int vcr_set_flash_warps(int nwq) {
    return g_vcr_flash_warps.exchange(nwq >= 1 && nwq <= 4 ? nwq : 3);
}

// Q: operand buffer [planes][B*Nq][ldq], head hh in columns [hh*128, hh*128+128) of the given base;
// K: [planes][B*Nk][ldk] likewise; VT: [planes][B*H*128][ldv] with row (b*H + hh)*128 + d and Nk key columns;
// O: [planes][B*Nq][ldo] operand-format output (same head layout as Q).  d_k must be 128.
// mode: 0 = fp16 3-term split ("h3"), 1 = fp16, 2 = bf16.  keep: optional uint8 [B,Nk] key mask.
// lse: optional [B,H,Nq] log2-domain log-sum-exp of the scaled scores.
VCR_API int vcr_flash_attn_tc(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                              const void* VT, int ldv, long long v_plane, int B, int H, int Nq, int Nk, int dk,
                              int mode, float scale, const uint8_t* keep, void* O, int ldo, long long o_plane,
                              float* lse, cudaStream_t stream) {
    VCR_REQUIRE(Q && K && VT && O && B > 0 && H > 0 && Nq > 0 && Nk > 0);
    if (dk != DK || mode < 0 || mode > 2) return VCR_ERR_UNSUPPORTED;
    if ((ldo & 7) || (o_plane & 7)) return VCR_ERR_INVALID;
    const int planes = mode == 0 ? 2 : 1;
    CUtensorMap tq, tk, tv;
    int rc = vcr_make_operand_tmap(&tq, Q, H * DK, (long long)B * Nq, ldq, q_plane, planes, BQ);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tk, K, H * DK, (long long)B * Nk, ldk, k_plane, planes, BKV);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tv, VT, Nk, (long long)B * H * DK, ldv, v_plane, planes, DK);
    if (rc != VCR_OK) return rc;
    AttnParams p;
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk;
    p.scale_log2 = scale * kLog2e; p.keep = keep; p.nq_len = nullptr; p.nk_len = nullptr;
    p.O = reinterpret_cast<__half*>(O); p.ldo = ldo; p.o_plane = o_plane; p.lse = lse; p.out_bf16 = mode == 2;
    const int org = g_vcr_flash_warps.load(std::memory_order_relaxed);
    if (org == 3) {
        if (mode == 0) return launch_attn_ts<3, 0>(tq, tk, tv, p, stream);
        if (mode == 1) return launch_attn_ts<1, 0>(tq, tk, tv, p, stream);
        return launch_attn_ts<1, 1>(tq, tk, tv, p, stream);
    }
    if (org == 1) {
        if (mode == 0) return launch_attn<3, 0, 2, true>(tq, tk, tv, p, stream);
        if (mode == 1) return launch_attn<1, 0, 2, true>(tq, tk, tv, p, stream);
        return launch_attn<1, 1, 2, true>(tq, tk, tv, p, stream);
    }
    if (org == 4) {
        if (mode == 0) return launch_attn<3, 0, 4>(tq, tk, tv, p, stream);
        if (mode == 1) return launch_attn<1, 0, 4>(tq, tk, tv, p, stream);
        return launch_attn<1, 1, 4>(tq, tk, tv, p, stream);
    }
    if (mode == 0) return launch_attn<3, 0, 2>(tq, tk, tv, p, stream);
    if (mode == 1) return launch_attn<1, 0, 2>(tq, tk, tv, p, stream);
    return launch_attn<1, 1, 2>(tq, tk, tv, p, stream);
}

static int flash_ragged_launch(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                               const void* VT, int ldv, long long v_plane, const int* nq, const int* nk, int B, int H,
                               int Nq, int Nk, int dk, int mode, float scale, const uint8_t* keep, void* O, int ldo,
                               long long o_plane, cudaStream_t stream) {
    if (dk != DK || mode < 0 || mode > 2) return VCR_ERR_UNSUPPORTED;
    if ((ldo & 7) || (o_plane & 7)) return VCR_ERR_INVALID;
    const int planes = mode == 0 ? 2 : 1;
    CUtensorMap tq, tk, tv;
    int rc = vcr_make_operand_tmap(&tq, Q, H * DK, (long long)B * Nq, ldq, q_plane, planes, BQ);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tk, K, H * DK, (long long)B * Nk, ldk, k_plane, planes, BKV);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tv, VT, Nk, (long long)B * H * DK, ldv, v_plane, planes, DK);
    if (rc != VCR_OK) return rc;
    AttnParams p;
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk;
    p.scale_log2 = scale * kLog2e; p.keep = keep; p.nq_len = nq; p.nk_len = nk;
    p.O = reinterpret_cast<__half*>(O); p.ldo = ldo; p.o_plane = o_plane; p.lse = nullptr; p.out_bf16 = mode == 2;
    if (mode == 0) return launch_attn_ts<3, 0>(tq, tk, tv, p, stream);
    if (mode == 1) return launch_attn_ts<1, 0>(tq, tk, tv, p, stream);
    return launch_attn_ts<1, 1>(tq, tk, tv, p, stream);
}

// Ragged batch: item b has nq[b] queries and nk[b] keys (each clamped to [1, Nq] / [1, Nk]) in its Nq / Nk rows.  Key tiles
// past nk[b] are not loaded, the last one is masked as the tail of a call with Nk = nk[b], and a query tile wholly past
// nq[b] is written as zeros after one key tile.  Rows of a real query equal vcr_flash_attn_tc on the item alone, bit for
// bit, provided the padded V columns of the last key tile are finite (their probability is exactly 0).  Always the default
// organisation (Q and P in tensor memory); no key mask, no lse.
VCR_API int vcr_flash_attn_tc_ragged(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                                     const void* VT, int ldv, long long v_plane, const int* nq, const int* nk, int B, int H,
                                     int Nq, int Nk, int dk, int mode, float scale, void* O, int ldo, long long o_plane,
                                     cudaStream_t stream) {
    VCR_REQUIRE(Q && K && VT && O && nq && nk && B > 0 && H > 0 && Nq > 0 && Nk > 0);
    return flash_ragged_launch(Q, ldq, q_plane, K, ldk, k_plane, VT, ldv, v_plane, nq, nk, B, H, Nq, Nk, dk, mode, scale,
                               nullptr, O, ldo, o_plane, stream);
}

// vcr_flash_attn_tc_ragged with the partial-overlap key mask keep [B, Nk] (uint8, row stride Nk): a key of item b with
// keep == 0 gets -1e9 as in vcr_flash_attn_tc, a key past nk[b] gets -inf whatever keep holds.  Rows of a real query equal
// vcr_flash_attn_tc(keep = the item's first nk[b] mask bytes) on the item alone, bit for bit.
VCR_API int vcr_flash_attn_tc_ragged_keep(const void* Q, int ldq, long long q_plane, const void* K, int ldk,
                                          long long k_plane, const void* VT, int ldv, long long v_plane, const int* nq,
                                          const int* nk, const uint8_t* keep, int B, int H, int Nq, int Nk, int dk, int mode,
                                          float scale, void* O, int ldo, long long o_plane, cudaStream_t stream) {
    VCR_REQUIRE(Q && K && VT && O && nq && nk && keep && B > 0 && H > 0 && Nq > 0 && Nk > 0);
    return flash_ragged_launch(Q, ldq, q_plane, K, ldk, k_plane, VT, ldv, v_plane, nq, nk, B, H, Nq, Nk, dk, mode, scale,
                               keep, O, ldo, o_plane, stream);
}
