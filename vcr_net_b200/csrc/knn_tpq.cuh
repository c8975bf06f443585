// Thread-per-query k-nearest-neighbour selection for the tensor-core prefilter (included by knn.cu inside its anonymous
// namespace).
//
// The warp-per-query kernels of knn.cu spend their issue slots on 32-lane shuffle networks (ncu r1: 32 % of the D = 64
// kernel's and 66 % of the D = 3 kernel's instructions are selection).  Here a THREAD owns a query:
//
//   * candidates arrive 32 at a time as one tcgen05.ld of the thread's TMEM lane -- queries sit on the M side of the MMA,
//     so a lane IS a query and no distance tile goes through shared memory;
//   * a candidate that beats the thread's current threshold (the running rank-kk key) is appended to the thread's survivor
//     column in shared memory: compare + predicated store, no ballots, no shuffles;
//   * when any lane of the warp is about to run out of survivor slots, all lanes REFRESH: the survivors are sorted by a
//     bitonic network held entirely in registers (240 compare-exchanges, every index a compile-time constant, 32 queries
//     per warp-instruction) and merged into the thread's sorted top-32 list, which tightens the threshold.
//
// MEASURED (B200, round 2, profiles/r02_knn_tpq_diag.txt, profiles/r02_ncu_knn_tpq.txt): bit-identical to the exact kernel
// on every test input, 2.6x fewer instructions per query than the warp-per-query selection when one thread scans a whole
// cloud -- but a query per THREAD leaves 18 k queries (24 clouds x 768 points, the benchmark's call) as 576 warps on 592
// schedulers, each issuing once per 8.8 cycles (dependent ISETP -> SEL chains, 150-212 registers cap the occupancy at 3-5
// warps per scheduler): 145 us vs 131 us for the warp-per-query tensor-core kernel and 116 us for the FP32 SIMT kernel at
// 24 x 768 x 64-d.  It wins only where there is a long candidate stream per query: 1.25x at N = 16384.  So it is routed for
// N >= 8192 only (vcr_set_knn_tc_tpq); a D = 3 variant of the same selection (2-3x slower than the warp-per-query kernel at
// every size tried, for the same reason) was measured and dropped.

struct KP { uint32_t k, p; };            // k: order-preserving key of the value (0 = empty slot), p: ~index (larger = lower index)

template <bool EXACT>
__device__ __forceinline__ bool kp_before(const KP& a, const KP& b) {      // a ranks strictly before b (branch-free)
    if (EXACT) {
        const unsigned long long A = ((unsigned long long)a.k << 32) | a.p, B = ((unsigned long long)b.k << 32) | b.p;
        return A > B;                                                       // one carry-chained 64-bit compare
    }
    return a.k > b.k;
}
template <bool EXACT>
__device__ __forceinline__ void kp_ce(KP& hi, KP& lo) {                    // afterwards hi ranks before (or ties) lo
    const bool sw = kp_before<EXACT>(lo, hi);
    const uint32_t hk = hi.k, hp = hi.p;
    hi.k = sw ? lo.k : hk; hi.p = sw ? lo.p : hp;
    lo.k = sw ? hk : lo.k; lo.p = sw ? hp : lo.p;
}
// bitonic sort, descending, N a power of two, everything in registers
template <bool EXACT, int N>
__device__ __forceinline__ void kp_sort_desc(KP (&v)[N]) {
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const int l = i ^ j;
                if (l > i) {
                    if ((i & k) == 0) kp_ce<EXACT>(v[i], v[l]);
                    else kp_ce<EXACT>(v[l], v[i]);
                }
            }
        }
    }
}
// run, add: descending-sorted N-lists -> run = the best N of the union, descending
template <bool EXACT, int N>
__device__ __forceinline__ void kp_merge_desc(KP (&run)[N], const KP (&add)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const bool t = kp_before<EXACT>(add[N - 1 - i], run[i]);
        run[i].k = t ? add[N - 1 - i].k : run[i].k;
        run[i].p = t ? add[N - 1 - i].p : run[i].p;
    }
#pragma unroll
    for (int j = N >> 1; j > 0; j >>= 1) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int l = i ^ j;
            if (l > i) kp_ce<EXACT>(run[i], run[l]);
        }
    }
}

constexpr int TPQ_L = 32;            // list length (ranks 0..31), also the candidates per step
constexpr int TPQ_CAP = 48;          // survivor slots per thread: a step may add 32, so refresh when a lane holds > 16
constexpr int TPQ_TRIG = TPQ_CAP - TPQ_L;

// Survivor columns: slot-major [TPQ_CAP][T] so that the lanes of a warp hit distinct banks whatever their fill levels.
template <int T>
struct TpqBuf {
    uint32_t* k; uint32_t* p;
    __device__ __forceinline__ TpqBuf(void* base) : k(reinterpret_cast<uint32_t*>(base)), p(k + TPQ_CAP * T) {}
    static constexpr size_t bytes = (size_t)2 * TPQ_CAP * T * sizeof(uint32_t);
};

// merge the thread's cnt buffered survivors into its list (one or two rounds of 32), tighten the threshold
template <bool EXACT, int T>
__device__ __forceinline__ void tpq_refresh(KP (&run)[TPQ_L], const TpqBuf<T>& buf, int tid, int& cnt, int kk, uint32_t& tau,
                                            bool two_rounds) {
#pragma unroll 1
    for (int r = 0; r < 2; ++r) {
        if (r == 1 && !two_rounds) break;
        KP add[TPQ_L];
#pragma unroll
        for (int s = 0; s < TPQ_L; ++s) {
            const int slot = r * TPQ_L + s;
            const bool ok = slot < cnt && slot < TPQ_CAP;
            add[s].k = ok ? buf.k[(slot < TPQ_CAP ? slot : 0) * T + tid] : 0u;
            add[s].p = ok ? buf.p[(slot < TPQ_CAP ? slot : 0) * T + tid] : 0u;
        }
        kp_sort_desc<EXACT, TPQ_L>(add);
        kp_merge_desc<EXACT, TPQ_L>(run, add);
    }
    cnt = 0;
    // threshold = key of rank kk (kk is warp-uniform but not a compile-time constant)
    uint32_t t = 0u;
#pragma unroll
    for (int i = 0; i < TPQ_L; ++i) t = (i == kk) ? run[i].k : t;
    tau = t;
}

// =====================================================================================================
// Feature space (16 <= D <= 128, token-major): tcgen05 distance tiles as a certified PREFILTER, thread-per-query
// selection straight from TMEM, exact canonical re-rank of the list + certificate (same contract as knn_tc_kernel:
// bit-identical to the exact kernel on every input; uncertified 32-query groups are flagged for it).
//
//   CTA = 128 queries (UMMA M = 128: a TMEM lane is a query) + one producer warp.  Candidates stream through a ring of
//   64-row TMA stages; per tile S~ = Q C^T with the 3-term fp16 split (hi*hi' in D0, hi*lo' + lo*hi' in D1), D0 | D1
//   double-buffered in TMEM (256 columns: two CTAs per SM), so the MMAs of tile t+1 run under the selection of tile t.
//   A consumer thread reads its lane 32 candidates at a time, forms pd~ = (-xx_j - (-2 dot~)) - xx_i and filters against
//   its own threshold.  No distance tile in shared memory, no cross-lane traffic.
// =====================================================================================================
constexpr int TQ2 = 128;                 // queries per CTA
constexpr int TC2 = 64;                  // candidates per tile
constexpr int T2_THREADS = TQ2 + 32;     // 4 consumer warps + 1 producer warp
constexpr int T2_QTILE = TQ2 * 128;      // bytes of one [128 queries][64 x fp16] swizzled tile
constexpr int T2_CTILE = TC2 * 128;      // bytes of one [64 candidates][64 x fp16] swizzled tile

__host__ __device__ constexpr int knn_tc2_stages(int KB) { return KB == 1 ? 2 : 2; }
__host__ __device__ constexpr size_t knn_tc2_smem_bytes(int KB) {
    return (size_t)KB * 2 * T2_QTILE + (size_t)knn_tc2_stages(KB) * KB * 2 * T2_CTILE + TpqBuf<TQ2>::bytes + 128 + 1024;
}

__global__ void __launch_bounds__(T2_THREADS, 1)
knn_tc2_kernel(const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmQ, const KnnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const int KB = p.KB, N = p.N, D = p.D, k = p.k, ksel = p.ksel;
    const int NSTG = knn_tc2_stages(KB);
    const int qbytes = KB * 2 * T2_QTILE, cbytes = KB * 2 * T2_CTILE;
    uint8_t* q_s = smem;
    uint8_t* c_s = smem + qbytes;
    uint8_t* b_s = c_s + (size_t)NSTG * cbytes;
    TpqBuf<TQ2> buf(b_s);
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_s + TpqBuf<TQ2>::bytes);
    uint64_t* q_full = bars + 0;
    uint64_t* c_full = bars + 1;          // [2] candidate stage landed
    uint64_t* c_empty = bars + 3;         // [2] MMAs that read the stage retired
    uint64_t* a_full = bars + 5;          // [2] accumulator pair of a tile complete
    uint64_t* a_empty = bars + 7;         // [2] all 128 consumer threads have read it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, q0 = blockIdx.x * TQ2;
    const float* xxb = p.xx + (size_t)b * N;
    const int Nb = vcr_item_len(p.nlen, b, N, k + 1);      // ragged batch: candidates and queries past Nb are padding
    if (q0 >= Nb) {
        knn_write_self(p.idx32, p.idx64, b, N, k, q0, min(TQ2, N - q0), tid, T2_THREADS);
        return;
    }
    const int ntiles = (Nb + TC2 - 1) / TC2;

    if (warp == 4 && lane == 0) {
        tc::tma_prefetch_desc(&tmC); tc::tma_prefetch_desc(&tmQ);
        tc::mbar_init(q_full, 1);
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&c_full[s], 1); tc::mbar_init(&c_empty[s], 1);
            tc::mbar_init(&a_full[s], 1); tc::mbar_init(&a_empty[s], TQ2);
        }
        tc::fence_barrier_init();
    }
    if (warp == 0) { tc::tmem_alloc(tmem_slot, 256); tc::tmem_relinquish(); }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const float xm = __uint_as_float(p.xxmax[b]);
    const bool cloud_ok = xm >= 9.5367431640625e-07f && xm <= 1073741824.f;     // [2^-20, 2^30]; false for NaN
    const int nq32 = (N + 31) / 32;
    if (!cloud_ok) {
        // outside the fp16 range of the split: the exact kernel computes these queries
        if (warp < 4 && lane == 0 && q0 + warp * 32 < N) {
            p.redo[b * nq32 + (q0 >> 5) + warp] = 1;
            atomicAdd(p.nflag, min(32, N - (q0 + warp * 32)));
        }
    } else if (warp == 4) {
        // ============================== TMA producer + MMA issuer ==============================
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::umma_idesc(TQ2, TC2, 0);
            const int row0 = b * N;
            tc::mbar_expect_tx(q_full, qbytes);
            for (int kb = 0; kb < KB; ++kb)
                for (int pl = 0; pl < 2; ++pl)
                    tc::tma_load_3d(q_s + (kb * 2 + pl) * T2_QTILE, &tmQ, q_full, kb * 64, row0 + q0, pl);
            auto load_tile = [&](int t) {
                const int s = t % NSTG;
                if (t >= NSTG) tc::mbar_wait(&c_empty[s], ((t / NSTG) - 1) & 1);
                tc::mbar_expect_tx(&c_full[s], cbytes);
                for (int kb = 0; kb < KB; ++kb)
                    for (int pl = 0; pl < 2; ++pl)
                        tc::tma_load_3d(c_s + (size_t)s * cbytes + (kb * 2 + pl) * T2_CTILE, &tmC, &c_full[s], kb * 64,
                                        row0 + t * TC2, pl);
            };
            for (int t = 0; t < NSTG - 1 && t < ntiles; ++t) load_tile(t);
            tc::mbar_wait(q_full, 0);
            const uint32_t q_addr = tc::smem_u32(q_s);
            for (int t = 0; t < ntiles; ++t) {
                if (t + NSTG - 1 < ntiles) load_tile(t + NSTG - 1);
                const int s = t % NSTG, a = t & 1;
                tc::mbar_wait(&c_full[s], (t / NSTG) & 1);
                if (t >= 2) tc::mbar_wait(&a_empty[a], ((t >> 1) - 1) & 1);
                tc::tc_fence_after();
                const uint32_t c_addr = tc::smem_u32(c_s + (size_t)s * cbytes);
                const uint32_t d0 = tmem_base + a * (2 * TC2), d1 = d0 + TC2;
                for (int kb = 0; kb < KB; ++kb) {
                    const uint64_t q_hi = tc::umma_desc_k_sw128(q_addr + (kb * 2) * T2_QTILE);
                    const uint64_t q_lo = tc::umma_desc_k_sw128(q_addr + (kb * 2 + 1) * T2_QTILE);
                    const uint64_t c_hi = tc::umma_desc_k_sw128(c_addr + (kb * 2) * T2_CTILE);
                    const uint64_t c_lo = tc::umma_desc_k_sw128(c_addr + (kb * 2 + 1) * T2_CTILE);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (kb | kk) != 0;
                        const uint64_t adv = (uint64_t)(kk * 2);
                        tc::umma_f16(d0, q_hi + adv, c_hi + adv, idesc, acc);
                        tc::umma_f16(d1, q_hi + adv, c_lo + adv, idesc, acc);
                        tc::umma_f16(d1, q_lo + adv, c_hi + adv, idesc, 1);
                    }
                }
                tc::umma_commit(&a_full[a]);
                tc::umma_commit(&c_empty[s]);
            }
        }
    } else {
        // ============================== consumers: thread = query ==============================
        const int q = q0 + tid;
        const bool qok = q < Nb;
        const float xxq = qok ? xxb[q] : 0.f;
        const uint32_t lane_adr = (uint32_t)(warp * 32) << 16;
        KP run[TPQ_L];
#pragma unroll
        for (int i = 0; i < TPQ_L; ++i) run[i].k = run[i].p = 0u;
        uint32_t tau = 0u;
        int cnt = 0;
#pragma unroll 1
        for (int st = 0; st < 2 * ntiles; ++st) {
            const int t = st >> 1, h = st & 1, a = t & 1;
            {
                const int mx = __reduce_max_sync(0xffffffffu, cnt);
                if (mx > TPQ_TRIG) tpq_refresh<false, TQ2>(run, buf, tid, cnt, ksel, tau, mx > TPQ_L);
            }
            if (h == 0) { tc::mbar_wait(&a_full[a], (t >> 1) & 1); tc::tc_fence_after(); }
            uint32_t r0[32], r1[32];
            const uint32_t ta = tmem_base + lane_adr + a * (2 * TC2) + h * 32;
            tc::tmem_ld_32x32(ta, r0);
            tc::tmem_ld_32x32(ta + TC2, r1);
            tc::tmem_ld_wait();
            if (h == 1) { tc::tc_fence_before(); tc::mbar_arrive(&a_empty[a]); }
            const int j0 = t * TC2 + h * 32;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int j = j0 + i;
                const float dot = fmaf(__uint_as_float(r1[i]), 1.f / 2048.f, __uint_as_float(r0[i]));
                const float nxc = -__ldg(xxb + min(j, N - 1));                  // warp-uniform address: one broadcast load
                const float pd = __fsub_rn(__fsub_rn(nxc, -2.f * dot), xxq);
                const uint32_t key = okey(pd);
                if (qok && j < Nb && key > tau) {
                    buf.k[cnt * TQ2 + tid] = key;
                    buf.p[cnt * TQ2 + tid] = ~(uint32_t)j;
                    ++cnt;
                }
            }
        }
        {
            const int mx = __reduce_max_sync(0xffffffffu, cnt);
            if (mx > 0) tpq_refresh<false, TQ2>(run, buf, tid, cnt, ksel, tau, mx > TPQ_L);
        }

        // ---- exact re-rank (canonical fp32 chain) of ranks 0..ksel + certificate, thread = query ----
        const uint32_t thr_k = tau;                                              // pd~ key of rank ksel (0: fewer entries)
        const float* xq = p.x + ((size_t)b * N + (qok ? q : 0)) * D;
        const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.x) & 15) == 0);
        KP e[TPQ_L];
#pragma unroll
        for (int g = 0; g < TPQ_L; g += 4) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            const float* xj[4];
            bool valid[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = (int)(~run[g + u].p);
                valid[u] = qok && g + u <= ksel && run[g + u].k != 0u && j >= 0 && j < Nb;
                xj[u] = p.x + ((size_t)b * N + (valid[u] ? j : 0)) * D;
            }
            if (g <= ksel) {                                                     // warp-uniform
                if (vec) {
                    for (int d = 0; d < D; d += 4) {
                        const float4 qv = __ldg(reinterpret_cast<const float4*>(xq + d));
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 cv = __ldg(reinterpret_cast<const float4*>(xj[u] + d));
                            acc[u] = fmaf(qv.x, cv.x, acc[u]); acc[u] = fmaf(qv.y, cv.y, acc[u]);
                            acc[u] = fmaf(qv.z, cv.z, acc[u]); acc[u] = fmaf(qv.w, cv.w, acc[u]);
                        }
                    }
                } else {
                    for (int d = 0; d < D; ++d) {
                        const float qv = __ldg(xq + d);
#pragma unroll
                        for (int u = 0; u < 4; ++u) acc[u] = fmaf(qv, __ldg(xj[u] + d), acc[u]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = (int)(~run[g + u].p);
                const float pd = __fsub_rn(__fsub_rn(-xxb[valid[u] ? j : 0], -2.f * acc[u]), xxq);
                e[g + u].k = valid[u] ? okey(pd) : 0u;
                e[g + u].p = valid[u] ? run[g + u].p : 0u;
            }
        }
        kp_sort_desc<true, TPQ_L>(e);
        uint32_t ek = 0u;
#pragma unroll
        for (int i = 0; i < TPQ_L; ++i) ek = (i == k) ? e[i].k : ek;
        const float eps = 6.103515625e-05f * sqrtf(xxq * xm) + 9.5367431640625e-07f * xm;
        const bool safe = !qok || (ek != 0u && (thr_k == 0u || okey_inv(ek) > okey_inv(thr_k) + eps));
        if (qok && safe) {
            const size_t o = ((size_t)b * N + q) * k;
#pragma unroll
            for (int i = 1; i < TPQ_L; ++i) {
                if (i <= k) {
                    const int jn = (int)(~e[i].p);
                    if (p.idx32) p.idx32[o + i - 1] = jn;
                    if (p.idx64) p.idx64[o + i - 1] = (int64_t)jn;
                }
            }
        } else if (!qok && q < N) {
            knn_write_self(p.idx32, p.idx64, b, N, k, q, 1, 0, 1);     // padded query of a ragged batch
        }
        const uint32_t bad = __ballot_sync(0xffffffffu, !safe);
        if (bad != 0u && lane == 0) {
            p.redo[b * nq32 + (q0 >> 5) + warp] = 1;
            atomicAdd(p.nflag, __popc(bad));
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem_base, 256);
}
