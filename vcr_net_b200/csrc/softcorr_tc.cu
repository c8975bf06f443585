// Fused virtual-correspondence generation on tcgen05 / TMEM / TMA (sm_100a): getCopairALL of the reference
// (model/vcrnet_model.py:334-347)
//     pd_ij   = (-|s_i|^2 - (-2 s_i . t_j)) - |t_j|^2
//     corr_i  = sum_j softmax_j(pd_ij) * tgt_xyz_j
// in ONE kernel: the [Ns, Nt] score / probability matrices (67 MB per 16 pairs at N = 1024, 2.1 GB per 32 pairs at
// N = 4096) never reach HBM.  A work item is (pair, 128-query tile); a persistent CTA walks its items and, per item,
// all 128-target tiles: the main loop is the 3-term fp16-split GEMM of gemm_tc.cu (warp 0 TMA producer, warp 1 MMA
// issuer, accumulators double-buffered in TMEM so the softmax of tile n overlaps the products of tile n+1), the
// epilogue (8 warps, thread = query row, two warps share a row and split the 128 columns) turns each accumulator
// row into pd with the reference's operation order, keeps a running (max, sum, sum * xyz) per row (online softmax)
// and writes corr[B,3,Ns] at the end of the item.  The logits cancel catastrophically (|f|^2 ~ 500 against gaps
// < 1, SURVEY.md section 7), so this kernel exists in the 3-term mode only, in every precision mode.
// The same main loop gives selectCom's two statistics (vcr_select_stats_tc): MODE 3 keeps only the row's running
// (max, sum) and writes (max, 1/sum); MODE 4 sums exp(pd_ij - M_j) * invL_j with per-column (M, 1/L) staged in shared
// memory.  SWAP runs a launch with the targets as rows: pd keeps the reference order with the source norm first.
#include "tc_common.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int TILE_BYTES = 128 * 128;
constexpr int NSTAGES = 3;
constexpr int STAGE_BYTES = 4 * TILE_BYTES;          // A hi, A lo, B hi, B lo
constexpr int EPI_WARPS = 8;
constexpr int NTHREADS = 128 + EPI_WARPS * 32;
constexpr int ACC_COLS = 2 * BN;                     // D0 | D1
constexpr int TMEM_COLS = 2 * ACC_COLS;
constexpr int OFF_BAR = NSTAGES * STAGE_BYTES;
constexpr int OFF_COLS = OFF_BAR + 256;              // per epilogue warp: yy | x | y | z of its 64 columns
constexpr int OFF_XCH = OFF_COLS + EPI_WARPS * 4 * 64 * 4;   // [128 rows][5] partial state of the upper column half
constexpr int SMEM_BYTES = OFF_XCH + 128 * 5 * 4 + 1024;

struct SoftcorrParams {
    int B, Ns, Nt, D;
    const float* xx;      // [B*Ns]  |s_i|^2
    const float* yy;      // [B*Nt]  |t_j|^2
    const float* tgt;     // [B,3,Nt]           (mode 0)
    float* corr;          // [B,3,Ns]           (mode 0)
    int* best_idx;        // [B,Ns] argmax_j     (mode 2: hard correspondences, model/vcrnet_model.py:295-299)
    float* best_val;      // [B,Ns] max_j P_ij   (mode 2)
    float* row_m;         // [B,Ns] max_j pd_ij          (mode 3)
    float* row_il;        // [B,Ns] 1 / sum_j exp(pd_ij - max)   (mode 3)
    const float* col_m;   // [B,Nt] per-column max        (mode 4)
    const float* col_il;  // [B,Nt] per-column 1 / sum    (mode 4)
    float* row_stat;      // [B,Ns] sum_j exp(pd_ij - col_m_j) * col_il_j   (mode 4)
};

// SWAP: the rows (A, xx) are targets and the columns (B, yy) sources.
template <int MODE, bool SWAP = false>
__global__ void __launch_bounds__(NTHREADS, 1)
softcorr_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SoftcorrParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* full = bars;                         // [NSTAGES]
    uint64_t* empty = bars + NSTAGES;              // [NSTAGES]
    uint64_t* tfull = bars + 2 * NSTAGES;          // [2]
    uint64_t* tempty = tfull + 2;                  // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_m = (p.Ns + BM - 1) / BM, tiles_n = (p.Nt + BN - 1) / BN;
    const int items = p.B * tiles_m;
    const int nkb = (p.D + BK - 1) / BK;

    if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tmA); tc::tma_prefetch_desc(&tmB); }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < NSTAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { tc::mbar_init(&tfull[a], 1); tc::mbar_init(&tempty[a], EPI_WARPS * 32); }
        tc::fence_barrier_init();
    }
    if (warp == 2) { tc::tmem_alloc(tmem_slot, TMEM_COLS); tc::tmem_relinquish(); }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (tc::elect_one()) {
            int s = 0; uint32_t ph = 0;
            for (int it = blockIdx.x; it < items; it += gridDim.x) {
                const int b = it / tiles_m, m_blk = it - b * tiles_m;
                const int a_row = b * p.Ns + m_blk * BM;
                for (int n_blk = 0; n_blk < tiles_n; ++n_blk) {
                    const int b_row = b * p.Nt + n_blk * BN;
                    for (int kb = 0; kb < nkb; ++kb) {
                        tc::mbar_wait(&empty[s], ph ^ 1);
                        tc::mbar_expect_tx(&full[s], STAGE_BYTES);
                        uint8_t* st = smem + s * STAGE_BYTES;
#pragma unroll
                        for (int pl = 0; pl < 2; ++pl) {
                            tc::tma_load_3d(st + pl * TILE_BYTES, &tmA, &full[s], kb * BK, a_row, pl);
                            tc::tma_load_3d(st + (2 + pl) * TILE_BYTES, &tmB, &full[s], kb * BK, b_row, pl);
                        }
                        if (++s == NSTAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::umma_idesc(BM, BN, 0);
            int s = 0; uint32_t ph = 0;
            int tl = 0;                                               // running tile counter of this CTA
            for (int it = blockIdx.x; it < items; it += gridDim.x) {
                for (int n_blk = 0; n_blk < tiles_n; ++n_blk, ++tl) {
                    const int a = tl & 1;
                    const uint32_t aph = (tl >> 1) & 1;
                    tc::mbar_wait(&tempty[a], aph ^ 1);
                    tc::tc_fence_after();
                    const uint32_t d0 = tmem_base + a * ACC_COLS;
                    const uint32_t d1 = d0 + BN;
                    for (int kb = 0; kb < nkb; ++kb) {
                        tc::mbar_wait(&full[s], ph);
                        tc::tc_fence_after();
                        const uint32_t st = tc::smem_u32(smem + s * STAGE_BYTES);
                        const uint64_t a_hi = tc::umma_desc_k_sw128(st);
                        const uint64_t a_lo = tc::umma_desc_k_sw128(st + TILE_BYTES);
                        const uint64_t b_hi = tc::umma_desc_k_sw128(st + 2 * TILE_BYTES);
                        const uint64_t b_lo = tc::umma_desc_k_sw128(st + 3 * TILE_BYTES);
#pragma unroll
                        for (int kk = 0; kk < BK / 16; ++kk) {
                            const uint32_t acc = (kb | kk) != 0;
                            const uint64_t adv = (uint64_t)(kk * 2);  // 16 elements = 32 B along K
                            tc::umma_f16(d0, a_hi + adv, b_hi + adv, idesc, acc);
                            if (SWAP) {                               // per element: s_hi t_lo, then s_lo t_hi, as unswapped
                                tc::umma_f16(d1, a_lo + adv, b_hi + adv, idesc, acc);
                                tc::umma_f16(d1, a_hi + adv, b_lo + adv, idesc, 1);
                            } else {
                                tc::umma_f16(d1, a_hi + adv, b_lo + adv, idesc, acc);
                                tc::umma_f16(d1, a_lo + adv, b_hi + adv, idesc, 1);
                            }
                        }
                        tc::umma_commit(&empty[s]);
                        if (++s == NSTAGES) { s = 0; ph ^= 1; }
                    }
                    tc::umma_commit(&tfull[a]);
                }
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: online softmax + weighted sum of the target points =====================
        const int ew = warp & 3;                               // TMEM lane quarter
        const int chalf = (warp - 4) >> 2;                     // column half of the tile
        float* cols = reinterpret_cast<float*>(smem + OFF_COLS) + (warp - 4) * (4 * 64);   // yy | x | y | z
        float* xch = reinterpret_cast<float*>(smem + OFF_XCH);
        const int rloc = ew * 32 + lane;
        int tl = 0;
        for (int it = blockIdx.x; it < items; it += gridDim.x) {
            const int b = it / tiles_m, m_blk = it - b * tiles_m;
            const int row = m_blk * BM + rloc;
            const bool row_ok = row < p.Ns;
            const float nx = row_ok ? -p.xx[(size_t)b * p.Ns + row] : 0.f;
            const float* yb = p.yy + (size_t)b * p.Nt;
            const float* tb = MODE == 0 ? p.tgt + (size_t)b * 3 * p.Nt : nullptr;
            float m = -INFINITY, s = 0.f, cx = 0.f, cy = 0.f, cz = 0.f;
            int mj = 0x7fffffff;                               // MODE 2: arg-max, ties -> lower index
            for (int n_blk = 0; n_blk < tiles_n; ++n_blk, ++tl) {
                const int a = tl & 1;
                const uint32_t aph = (tl >> 1) & 1;
                const int col_h = n_blk * BN + chalf * 64;     // first column of this warp's half
                // stage |t_j|^2 and the target points of the warp's 64 columns (previous tile's reads are done: the
                // __syncwarp at the end of the tile)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int cj = col_h + q * 32 + lane;
                    const bool ok = cj < p.Nt;
                    cols[q * 32 + lane] = ok ? yb[cj] : 0.f;
                    if (MODE == 0) {
                        cols[64 + q * 32 + lane] = ok ? tb[cj] : 0.f;
                        cols[128 + q * 32 + lane] = ok ? tb[p.Nt + cj] : 0.f;
                        cols[192 + q * 32 + lane] = ok ? tb[2 * p.Nt + cj] : 0.f;
                    }
                    if (MODE == 4) {
                        cols[64 + q * 32 + lane] = ok ? p.col_m[(size_t)b * p.Nt + cj] : 0.f;
                        cols[128 + q * 32 + lane] = ok ? p.col_il[(size_t)b * p.Nt + cj] : 0.f;
                    }
                }
                __syncwarp();
                tc::mbar_wait(&tfull[a], aph);
                tc::tc_fence_after();
                const uint32_t tadr = tmem_base + a * ACC_COLS + ((uint32_t)(ew * 32) << 16) + chalf * 64;
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    const int col0 = col_h + cc * 32;
                    if (col0 >= p.Nt) break;                   // warp-uniform
                    float pd[32];
                    {
                        uint32_t r0[32], r1[32];
                        tc::tmem_ld_32x32(tadr + cc * 32, r0);
                        tc::tmem_ld_32x32(tadr + BN + cc * 32, r1);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float dot = fmaf(__uint_as_float(r1[j]), 1.f / 2048.f, __uint_as_float(r0[j]));
                            // reference op order (:341-342): (-xx - (-2 dot)) - yy
                            if (SWAP) pd[j] = __fsub_rn(__fsub_rn(-cols[cc * 32 + j], -2.f * dot), -nx);
                            else pd[j] = __fsub_rn(__fsub_rn(nx, -2.f * dot), cols[cc * 32 + j]);
                        }
                    }
                    if (col0 + 32 > p.Nt) {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (col0 + j >= p.Nt) pd[j] = -INFINITY;
                    }
                    if (MODE == 4) {                           // columns past Nt: exp(-inf) * 0
#pragma unroll
                        for (int j = 0; j < 32; ++j) s = fmaf(__expf(pd[j] - cols[64 + cc * 32 + j]), cols[128 + cc * 32 + j], s);
                        continue;
                    }
                    float cm = pd[0];
                    int cj = 0;
#pragma unroll
                    for (int j = 1; j < 32; ++j) {
                        if (MODE == 2) { if (pd[j] > cm) { cm = pd[j]; cj = j; } }      // first (lowest) index of the maximum
                        else cm = fmaxf(cm, pd[j]);
                    }
                    if (cm > m) {                              // rescale the running sums to the new maximum
                        const float f = __expf(m - cm);        // m = -inf on the first chunk: f = 0
                        s *= f; cx *= f; cy *= f; cz *= f;
                        m = cm;
                        mj = col0 + cj;                        // columns are visited in increasing order: strict > keeps the lower index
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float e = __expf(pd[j] - m);
                        s += e;
                        if (MODE == 0) {
                            cx = fmaf(e, cols[64 + cc * 32 + j], cx);
                            cy = fmaf(e, cols[128 + cc * 32 + j], cy);
                            cz = fmaf(e, cols[192 + cc * 32 + j], cz);
                        }
                    }
                }
                tc::tc_fence_before();
                tc::mbar_arrive(&tempty[a]);                   // accumulator free for tile n+2
                __syncwarp();
            }
            // ---- combine the two column halves of a row (pair barrier, 64 threads), write corr ----
            if (chalf == 1) {
                float* x5 = xch + rloc * 5;
                x5[0] = m; x5[1] = s;
                if (MODE == 0) { x5[2] = cx; x5[3] = cy; x5[4] = cz; }
                else x5[2] = __int_as_float(mj);
            }
            asm volatile("bar.sync %0, 64;" ::"r"(1 + ew) : "memory");
            if (chalf == 0) {
                const float* x5 = xch + rloc * 5;
                const float m1 = x5[0];
                const float mt = fmaxf(m, m1);
                const float f0 = __expf(m - mt), f1 = __expf(m1 - mt);     // a half without columns has m = -inf: f = 0
                const float st = s * f0 + x5[1] * f1;
                if (row_ok) {
                    if (MODE == 0) {
                        float* cb = p.corr + (size_t)b * 3 * p.Ns;
                        cb[row] = (cx * f0 + x5[2] * f1) / st;
                        cb[p.Ns + row] = (cy * f0 + x5[3] * f1) / st;
                        cb[2 * p.Ns + row] = (cz * f0 + x5[4] * f1) / st;
                    } else if (MODE == 2) {
                        // equal maxima in the two halves: the lower index wins (the halves interleave 64-column blocks)
                        const int mj1 = __float_as_int(x5[2]);
                        const int best = (m1 > m || (m1 == m && mj1 < mj)) ? mj1 : mj;
                        p.best_idx[(size_t)b * p.Ns + row] = best;
                        p.best_val[(size_t)b * p.Ns + row] = 1.0f / st;     // exp(0) / sum: the maximum probability
                    } else if (MODE == 3) {
                        p.row_m[(size_t)b * p.Ns + row] = mt;
                        p.row_il[(size_t)b * p.Ns + row] = 1.0f / st;
                    } else {
                        p.row_stat[(size_t)b * p.Ns + row] = s + x5[1];           // no running max: plain sum
                    }
                }
            }
            asm volatile("bar.sync %0, 64;" ::"r"(1 + ew) : "memory");      // xch reusable for the next item
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

template <int MODE, bool SWAP>
static int softcorr_run(const CUtensorMap& tmA, const CUtensorMap& tmB, const SoftcorrParams& p, cudaStream_t stream) {
    auto kern = softcorr_tc_kernel<MODE, SWAP>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess)
        return VCR_ERR_LAUNCH;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long items = (long long)p.B * vcr_cdiv(p.Ns, BM);
    const int grid = (int)(items < sms ? items : sms);
    kern<<<grid, NTHREADS, SMEM_BYTES, stream>>>(tmA, tmB, p);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

// S / T: operand-format ("h3": 2 planes, fp16 hi and lo * 2^11) embeddings [2][B*Ns][lds] / [2][B*Nt][ldt];
// xx / yy: their fp32 squared row norms (vcr_sqnorm_rows); tgt [B,3,Nt]; corr [B,3,Ns].
// Replaces the matmul + softmax + matmul of model/vcrnet_model.py:337-345 without materialising the score matrix.
static int softcorr_launch(int mode, const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                           const float* xx, const float* yy, const float* tgt, int B, int Ns, int Nt, int D,
                           float* corr, int* best_idx, float* best_val, cudaStream_t stream) {
    if ((long long)B * (Ns > Nt ? Ns : Nt) > 0x7fffffffLL) return VCR_ERR_UNSUPPORTED;
    CUtensorMap tmA, tmB;
    int rc = vcr_make_operand_tmap(&tmA, S, D, (long long)B * Ns, lds, s_plane, 2, BM);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tmB, T, D, (long long)B * Nt, ldt, t_plane, 2, BN);
    if (rc != VCR_OK) return rc;
    SoftcorrParams p = {};
    p.B = B; p.Ns = Ns; p.Nt = Nt; p.D = D; p.xx = xx; p.yy = yy; p.tgt = tgt; p.corr = corr;
    p.best_idx = best_idx; p.best_val = best_val;
    return mode == 0 ? softcorr_run<0, false>(tmA, tmB, p, stream) : softcorr_run<2, false>(tmA, tmB, p, stream);
}

VCR_API int vcr_softcorr_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                            const float* xx, const float* yy, const float* tgt, int B, int Ns, int Nt, int D,
                            float* corr, cudaStream_t stream) {
    VCR_REQUIRE(S && T && xx && yy && tgt && corr && B > 0 && Ns > 0 && Nt > 0 && D > 0);
    return softcorr_launch(0, S, lds, s_plane, T, ldt, t_plane, xx, yy, tgt, B, Ns, Nt, D, corr, nullptr, nullptr, stream);
}

// getCopair (model/vcrnet_model.py:264-332), same fused kernel: best_idx[B,Ns] = argmax_j pd_ij (ties -> lower j),
// best_val[B,Ns] = max_j softmax_j(pd_ij).
VCR_API int vcr_softcorr_best_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                                 const float* xx, const float* yy, int B, int Ns, int Nt, int D,
                                 int* best_idx, float* best_val, cudaStream_t stream) {
    VCR_REQUIRE(S && T && xx && yy && best_idx && best_val && B > 0 && Ns > 0 && Nt > 0 && D > 0);
    return softcorr_launch(2, S, lds, s_plane, T, ldt, t_plane, xx, yy, nullptr, B, Ns, Nt, D, nullptr, best_idx, best_val, stream);
}

VCR_API size_t vcr_select_stats_tc_workspace_bytes(int B, int Ns, int Nt) {
    return (size_t)2 * ((size_t)B * Ns + (size_t)B * Nt) * sizeof(float);
}

// selectCom's two statistics (model/vcrnet_model.py:213-222, 243-244) from the operands, without the [Ns, Nt] matrix:
//   row_stat[i] = sum_j exp(pd_ij - Mc_j) / Lc_j      col_stat[j] = sum_i exp(pd_ij - Mr_i) / Lr_i
// Four launches of the fused kernel, each owning its rows: (a) sources x targets -> (Mr, 1/Lr); (b) targets x sources ->
// (Mc, 1/Lc); (c) sources x targets -> row_stat; (d) targets x sources -> col_stat.  Every sum runs inside one thread (two
// column halves added once) in tile order, so the result is deterministic.  workspace: Mr | 1/Lr | Mc | 1/Lc.
VCR_API int vcr_select_stats_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                                const float* xx, const float* yy, int B, int Ns, int Nt, int D, float* row_stat,
                                float* col_stat, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(S && T && xx && yy && row_stat && col_stat && B > 0 && Ns > 0 && Nt > 0 && D > 0);
    if (!workspace || workspace_bytes < vcr_select_stats_tc_workspace_bytes(B, Ns, Nt)) return VCR_ERR_WORKSPACE;
    if ((long long)B * (Ns > Nt ? Ns : Nt) > 0x7fffffffLL) return VCR_ERR_UNSUPPORTED;
    CUtensorMap tmS, tmT;                                  // BM == BN: one map per operand serves both roles
    int rc = vcr_make_operand_tmap(&tmS, S, D, (long long)B * Ns, lds, s_plane, 2, BM);
    if (rc != VCR_OK) return rc;
    rc = vcr_make_operand_tmap(&tmT, T, D, (long long)B * Nt, ldt, t_plane, 2, BN);
    if (rc != VCR_OK) return rc;
    float* mr = reinterpret_cast<float*>(workspace);
    float* ilr = mr + (size_t)B * Ns;
    float* mc = ilr + (size_t)B * Ns;
    float* ilc = mc + (size_t)B * Nt;
    SoftcorrParams ps = {}, pt = {};                       // rows = sources / rows = targets
    ps.B = B; ps.Ns = Ns; ps.Nt = Nt; ps.D = D; ps.xx = xx; ps.yy = yy;
    pt.B = B; pt.Ns = Nt; pt.Nt = Ns; pt.D = D; pt.xx = yy; pt.yy = xx;
    ps.row_m = mr; ps.row_il = ilr;
    pt.row_m = mc; pt.row_il = ilc;
    if ((rc = softcorr_run<3, false>(tmS, tmT, ps, stream)) != VCR_OK) return rc;
    if ((rc = softcorr_run<3, true>(tmT, tmS, pt, stream)) != VCR_OK) return rc;
    ps.col_m = mc; ps.col_il = ilc; ps.row_stat = row_stat;
    pt.col_m = mr; pt.col_il = ilr; pt.row_stat = col_stat;
    if ((rc = softcorr_run<4, false>(tmS, tmT, ps, stream)) != VCR_OK) return rc;
    return softcorr_run<4, true>(tmT, tmS, pt, stream);
}
