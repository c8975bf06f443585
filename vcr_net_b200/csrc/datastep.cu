// On-device data step and evaluation metrics either side of the registration path (SURVEY.md section 8f row 2).
//
//   vcr_make_pairs     util/data.py:247-309 (ModelNet40.__getitem__) minus the random draws: the host draws the per-item
//                      pose and permutations exactly as the reference does (they are data, drawn from numpy's
//                      RandomState(item)), the device gathers, applies the float64 rigid transform
//                      (Rotation.from_euler('zyx').apply + t, :289-291) and casts to fp32 -- the clouds never exist
//                      on the host.
//   vcr_crop_nearest   util/data.py:320-329 nearest_neighbor(): keep the int(N*reserve) points nearest to the LAST point,
//                      nearest first (float64 squared distances, ties -> lower index), by rank counting in shared memory
//                      (one CTA per cloud, N <= 25 600).
//   vcr_crop_nearest_sort  the same crop for any N: a segmented stable radix sort of the distances' bit patterns in a
//                      caller-provided workspace (8 passes of 8-bit digits), then a gather of the first `keep`.
//   vcr_eval_metrics   model/vcrnet_model.py:583-630: pose loss, cycle loss, mse/mae of the a->b and b->a transformed
//                      clouds, accumulated into a device-resident double[8] (the reference does 6+ .item() host
//                      syncs per batch).
// Roofline: HBM / latency bound helpers (a few bytes per point); they exist to keep the 8 GPUs fed without host work.
#include "common.cuh"

namespace {

// base [P, Nb, 3] fp32; idx_src / idx_tgt [P, N] int32 (indices into the item's base cloud, permutations composed on
// the host); pose [P, 12] fp64 = row-major R (9) then t (3).  src[p,:,n] = base[idx_src[n]], tgt[p,:,n] = R base[idx_tgt[n]] + t.
__global__ void make_pairs_kernel(const float* __restrict__ base, int Nb, const int* __restrict__ idx_src,
                                  const int* __restrict__ idx_tgt, const double* __restrict__ pose, int N,
                                  double* __restrict__ src64, double* __restrict__ tgt64,
                                  float* __restrict__ src, float* __restrict__ tgt) {
    const int p = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float* bp = base + (size_t)p * Nb * 3;
    const double* ps = pose + (size_t)p * 12;
    const int is = idx_src[(size_t)p * N + n], it = idx_tgt[(size_t)p * N + n];
    const double sx = bp[is * 3 + 0], sy = bp[is * 3 + 1], sz = bp[is * 3 + 2];
    const double x = bp[it * 3 + 0], y = bp[it * 3 + 1], z = bp[it * 3 + 2];
    double o[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
        o[i] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(ps[i * 3 + 0], x), __dmul_rn(ps[i * 3 + 1], y)),
                                   __dmul_rn(ps[i * 3 + 2], z)), ps[9 + i]);
    const size_t o0 = (size_t)p * 3 * N + n;
    if (src64) { src64[o0] = sx; src64[o0 + N] = sy; src64[o0 + 2 * N] = sz; }
    if (tgt64) { tgt64[o0] = o[0]; tgt64[o0 + N] = o[1]; tgt64[o0 + 2 * N] = o[2]; }
    if (src) { src[o0] = (float)sx; src[o0 + N] = (float)sy; src[o0 + 2 * N] = (float)sz; }
    if (tgt) { tgt[o0] = (float)o[0]; tgt[o0 + N] = (float)o[1]; tgt[o0 + 2 * N] = (float)o[2]; }
}

// Squared distance of (x, y, z) to the anchor (lx, ly, lz) in fp64, in the order of ((x-l)**2).sum(axis=1); both crops
// rank by exactly this value.
__device__ __forceinline__ double sqdist_to_anchor(double x, double y, double z, double lx, double ly, double lz) {
    const double dx = x - lx, dy = y - ly, dz = z - lz;
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// pc64 [P,3,N] fp64 -> out [P,3,keep] fp32: the keep points nearest to point N-1, nearest first
__global__ void crop_nearest_kernel(const double* __restrict__ pc64, int N, int keep, float* __restrict__ out) {
    extern __shared__ double d2[];
    const int p = blockIdx.x;
    const double* pc = pc64 + (size_t)p * 3 * N;
    const double lx = pc[N - 1], ly = pc[2 * N - 1], lz = pc[3 * N - 1];
    for (int i = threadIdx.x; i < N; i += blockDim.x)
        d2[i] = sqdist_to_anchor(pc[i], pc[N + i], pc[2 * N + i], lx, ly, lz);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const double di = d2[i];
        int rank = 0;
        for (int j = 0; j < N; ++j) {
            const double dj = d2[j];
            rank += (dj < di) || (dj == di && j < i);
        }
        if (rank < keep) {
            float* o = out + (size_t)p * 3 * keep;
            o[rank] = (float)pc[i]; o[keep + rank] = (float)pc[N + i]; o[2 * keep + rank] = (float)pc[2 * N + i];
        }
    }
}

// ---- the same crop for any N: a stable LSD radix sort of (d2 bits, index) pairs, segmented per cloud ------------------
// A pass over one 8-bit digit is three launches: per-tile digit histograms, an exclusive scan per cloud over the
// histograms laid out digit-major across tiles (so the scan yields, for every (digit, tile), where that tile's keys of
// that digit start in the cloud's output), and a stable scatter inside each tile.  Keys start in index order and every
// pass is stable, so equal distances stay in index order without a comparison.
constexpr int kSortThreads = 256;
constexpr int kSortRounds = 8;                              // keys per thread and tile
constexpr int kSortTile = kSortThreads * kSortRounds;       // 2048 keys per tile
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kScanThreads = 1024;

// d2 is +0, positive or NaN (a sum of squares is never -0 or negative): for such doubles the bit pattern read as uint64
// orders like the value.  Every NaN gets the one key above +inf, so NaNs go last in index order, where numpy's stable
// argsort puts them.
__device__ __forceinline__ unsigned long long crop_key(double d2) {
    return d2 != d2 ? 0x7ff8000000000000ull : (unsigned long long)__double_as_longlong(d2);
}

template <int THREADS>
__device__ __forceinline__ unsigned block_exclusive_scan(unsigned v, unsigned* warp_tot) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    if (w == 0) {
        unsigned s = lane < THREADS / 32 ? warp_tot[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < THREADS / 32) warp_tot[lane] = s;
    }
    __syncthreads();
    return x - v + (w ? warp_tot[w - 1] : 0u);
}

// keys[p*N + i] = crop_key(d2 of point i of cloud p to its point N-1), idx[p*N + i] = i
__global__ void crop_keys_kernel(const double* __restrict__ pc64, int N, size_t total,
                                 unsigned long long* __restrict__ keys, unsigned* __restrict__ idx) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const size_t p = g / N, i = g - p * N;
    const double* pc = pc64 + p * 3 * N;
    keys[g] = crop_key(sqdist_to_anchor(pc[i], pc[N + i], pc[2 * (size_t)N + i], pc[N - 1], pc[2 * (size_t)N - 1],
                                        pc[3 * (size_t)N - 1]));
    idx[g] = (unsigned)i;
}

// counts[(p*256 + digit)*tiles + t] = keys of tile t of cloud p whose digit at `shift` is `digit`; one CTA per tile
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const unsigned long long* __restrict__ keys, int N,
                                                                  int tiles, int shift, unsigned* __restrict__ counts) {
    __shared__ unsigned h[256];
    const int p = blockIdx.x / tiles, t = blockIdx.x - p * tiles;
    const unsigned long long* k = keys + (size_t)p * N + (size_t)t * kSortTile;
    const int n = (int)min((long long)kSortTile, (long long)N - (long long)t * kSortTile);
    h[threadIdx.x] = 0;
    __syncthreads();
    // one shared atomic per distinct digit in a warp: in the passes over the exponent bytes nearly all keys of a tile
    // share one digit, and per-key atomics on that counter would serialise
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int s = r * kSortThreads + threadIdx.x;
        const unsigned d = s < n ? (unsigned)(k[s] >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (d < 256u && (peers & ((1u << lane) - 1u)) == 0u) atomicAdd(&h[d], (unsigned)__popc(peers));
    }
    __syncthreads();
    counts[((size_t)p * 256 + threadIdx.x) * tiles + t] = h[threadIdx.x];
}

// In place exclusive scan of each cloud's len = 256*tiles counts; one CTA per cloud.  The counts go through shared memory
// in chunks of 8192 (coalesced loads and stores); each thread scans 8 consecutive counts of a chunk, a block scan joins
// the threads, and a carry joins the chunks.
constexpr int kScanPer = 8, kScanChunk = kScanThreads * kScanPer;
__device__ __forceinline__ int scan_slot(int e) { return e + (e >> 5); }       // one pad word per 32: no bank conflicts
__global__ void __launch_bounds__(kScanThreads) radix_scan_kernel(unsigned* __restrict__ counts, int len) {
    __shared__ unsigned buf[kScanChunk + kScanChunk / 32];
    __shared__ unsigned warp_tot[kScanThreads / 32];
    unsigned* c = counts + (size_t)blockIdx.x * len;
    unsigned carry = 0;
    for (int c0 = 0; c0 < len; c0 += kScanChunk) {
        const int n = min(kScanChunk, len - c0);
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            const int e = j * kScanThreads + threadIdx.x;
            buf[scan_slot(e)] = e < n ? c[c0 + e] : 0u;
        }
        __syncthreads();
        unsigned v[kScanPer], sum = 0;
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            v[j] = buf[scan_slot(threadIdx.x * kScanPer + j)];
            sum += v[j];
        }
        unsigned run = carry + block_exclusive_scan<kScanThreads>(sum, warp_tot);   // ends with a barrier
        carry += warp_tot[kScanThreads / 32 - 1];                                   // the chunk's total
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            buf[scan_slot(threadIdx.x * kScanPer + j)] = run;
            run += v[j];
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            const int e = j * kScanThreads + threadIdx.x;
            if (e < n) c[c0 + e] = buf[scan_slot(e)];
        }
        __syncthreads();                              // buf and warp_tot are rewritten by the next chunk
    }
}

// One tile of 2048 (key, index) pairs goes to its place in the cloud's output, stable by digit.  The tile is read in
// 8 rounds of 256 consecutive keys; in a round each key's rank among the earlier keys of its digit in its warp comes from
// __match_any_sync, the warps' per-digit counts are scanned by the thread that owns the digit, and a running count carries
// the rounds.  A block scan of the tile's digit counts then places every pair in shared memory in digit order, and the
// sorted tile is written out so that neighbouring threads store neighbouring addresses within a digit's run.
__global__ void __launch_bounds__(kSortThreads, 4) radix_scatter_kernel(
    const unsigned long long* __restrict__ keys_in, const unsigned* __restrict__ idx_in, int N, int tiles, int shift,
    const unsigned* __restrict__ offsets, unsigned long long* __restrict__ keys_out, unsigned* __restrict__ idx_out) {
    __shared__ unsigned cnt[kSortWarps][256];        // this round: keys of each digit in each warp
    __shared__ unsigned pre[kSortWarps][256];        // the tile's keys of that digit before that warp's in this round
    __shared__ unsigned long long skey[kSortTile];
    __shared__ unsigned sidx[kSortTile];
    __shared__ unsigned start[256], goff[256], warp_tot[kSortWarps];

    const int p = blockIdx.x / tiles, t = blockIdx.x - p * tiles;
    const size_t base = (size_t)p * N, t0 = (size_t)t * kSortTile;
    const int n = (int)min((long long)kSortTile, (long long)N - (long long)t0);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < kSortWarps * 256; i += kSortThreads) (&cnt[0][0])[i] = 0u;
    goff[threadIdx.x] = offsets[((size_t)p * 256 + threadIdx.x) * tiles + t];
    __syncthreads();

    unsigned long long key[kSortRounds];
    unsigned id[kSortRounds], rank[kSortRounds];
    unsigned run = 0;                                 // keys of digit threadIdx.x in the rounds so far
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int s = r * kSortThreads + threadIdx.x;
        const bool valid = s < n;
        key[r] = valid ? keys_in[base + t0 + s] : 0ull;
        id[r] = valid ? idx_in[base + t0 + s] : 0u;
        const unsigned d = valid ? (unsigned)(key[r] >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const unsigned before = __popc(peers & ((1u << lane) - 1u));
        if (valid && before == 0) cnt[w][d] = __popc(peers);
        __syncthreads();
#pragma unroll
        for (int ww = 0; ww < kSortWarps; ++ww) {
            const unsigned c = cnt[ww][threadIdx.x];
            pre[ww][threadIdx.x] = run;
            cnt[ww][threadIdx.x] = 0u;
            run += c;
        }
        __syncthreads();
        rank[r] = valid ? pre[w][d] + before : 0u;
    }
    const unsigned st = block_exclusive_scan<kSortThreads>(run, warp_tot);
    start[threadIdx.x] = st;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        if (r * kSortThreads + threadIdx.x < n) {
            const unsigned pos = start[(unsigned)(key[r] >> shift) & 255u] + rank[r];
            skey[pos] = key[r];
            sidx[pos] = id[r];
        }
    }
    __syncthreads();
    for (int s = threadIdx.x; s < n; s += kSortThreads) {
        const unsigned long long k = skey[s];
        const unsigned d = (unsigned)(k >> shift) & 255u;
        const size_t g = base + goff[d] + (s - start[d]);
        keys_out[g] = k;
        idx_out[g] = sidx[s];
    }
}

// out[p, :, j] = (float)pc64[p, :, order[p*N + j]] for j < keep
__global__ void crop_gather_kernel(const double* __restrict__ pc64, int N, int keep, size_t total,
                                   const unsigned* __restrict__ order, float* __restrict__ out) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const size_t p = g / keep, j = g - p * keep;
    const double* pc = pc64 + p * 3 * N;
    const size_t i = order[p * N + j];
    float* o = out + p * 3 * keep;
    o[j] = (float)pc[i];
    o[keep + j] = (float)pc[N + i];
    o[2 * (size_t)keep + j] = (float)pc[2 * (size_t)N + i];
}

__device__ __forceinline__ void rigid(const float* R, const float* t, float x, float y, float z, float* o) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float acc = R[i * 3 + 0] * x;
        acc = fmaf(R[i * 3 + 1], y, acc);
        acc = fmaf(R[i * 3 + 2], z, acc);
        o[i] = acc + t[i];
    }
}

// acc[0] pose loss, [1] cycle loss, [2] mse_ab, [3] mae_ab, [4] mse_ba, [5] mae_ba, [6] number of examples (each already
// multiplied by the batch size as the reference accumulates `.item() * batch_size`)
__global__ void eval_metrics_kernel(const float* __restrict__ src, const float* __restrict__ tgt, int N,
                                    const float* __restrict__ srcK, const float* __restrict__ corrK, int M,
                                    const float* __restrict__ R_gt, const float* __restrict__ t_gt,
                                    const float* __restrict__ R_ab, const float* __restrict__ t_ab,
                                    const float* __restrict__ R_ba, const float* __restrict__ t_ba, int B,
                                    double* __restrict__ acc) {
    __shared__ double red[4][8];
    double s_ab2 = 0.0, s_ab1 = 0.0, s_ba2 = 0.0, s_ba1 = 0.0;
    const int stride = gridDim.x * blockDim.x, g = blockIdx.x * blockDim.x + threadIdx.x;
    for (long long e = g; e < (long long)B * M; e += stride) {             // transformed_srcK vs src_corrK (:591,623-624)
        const int b = (int)(e / M), m = (int)(e - (long long)b * M);
        const float* s = srcK + (size_t)b * 3 * M;
        const float* c = corrK + (size_t)b * 3 * M;
        float o[3];
        rigid(R_gt + b * 9, t_gt + b * 3, s[m], s[M + m], s[2 * M + m], o);
#pragma unroll
        for (int i = 0; i < 3; ++i) { const double d = (double)(o[i] - c[i * M + m]); s_ab2 += d * d; s_ab1 += fabs(d); }
    }
    for (long long e = g; e < (long long)B * N; e += stride) {             // transformed_target vs src (:589,626-627)
        const int b = (int)(e / N), n = (int)(e - (long long)b * N);
        const float* t = tgt + (size_t)b * 3 * N;
        const float* s = src + (size_t)b * 3 * N;
        float o[3];
        rigid(R_ba + b * 9, t_ba + b * 3, t[n], t[N + n], t[2 * N + n], o);
#pragma unroll
        for (int i = 0; i < 3; ++i) { const double d = (double)(o[i] - s[i * N + n]); s_ba2 += d * d; s_ba1 += fabs(d); }
    }
    double v[4] = {s_ab2, s_ab1, s_ba2, s_ba1};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        v[q] = warp_sum(v[q]);
        if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v[q];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[threadIdx.x][w];
        const double denom = threadIdx.x < 2 ? 3.0 * M : 3.0 * N;          // mean over [B,3,*] times batch size
        atomicAdd(acc + 2 + threadIdx.x, s / denom);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {                              // pose / cycle losses (:598-617), tiny
        double lr = 0.0, lt = 0.0, cr = 0.0, ct = 0.0;
        for (int b = 0; b < B; ++b) {
            const float* Rp = R_ab + b * 9; const float* Rg = R_gt + b * 9; const float* Rb = R_ba + b * 9;
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) {
                    float m1 = 0.f, m2 = 0.f;                                 // (R_pred^T R_gt)_ij and (R_ba R_ab)_ij
                    for (int k = 0; k < 3; ++k) { m1 = fmaf(Rp[k * 3 + i], Rg[k * 3 + j], m1); m2 = fmaf(Rb[i * 3 + k], Rp[k * 3 + j], m2); }
                    const double d1 = (double)m1 - (i == j), d2 = (double)m2 - (i == j);
                    lr += d1 * d1; cr += d2 * d2;
                }
            for (int i = 0; i < 3; ++i) {
                const double d = (double)t_ab[b * 3 + i] - (double)t_gt[b * 3 + i];
                lt += d * d;
                float m = 0.f;                                               // (R_ba^T t_ab + t_ba)_i
                for (int k = 0; k < 3; ++k) m = fmaf(Rb[k * 3 + i], t_ab[b * 3 + k], m);
                const double c = (double)m + (double)t_ba[b * 3 + i];
                ct += c * c;
            }
        }
        const double pose = lr / (9.0 * B) + lt / (3.0 * B);
        const double cyc = cr / (9.0 * B) + ct / (3.0 * B);
        atomicAdd(acc + 0, pose * B);
        atomicAdd(acc + 1, cyc * B);
        atomicAdd(acc + 6, (double)B);
    }
}

}  // namespace

VCR_API int vcr_make_pairs(const float* base, int P, int Nb, const int* idx_src, const int* idx_tgt, const double* pose,
                           int N, double* src64, double* tgt64, float* src, float* tgt, cudaStream_t stream) {
    VCR_REQUIRE(base && idx_src && idx_tgt && pose && P > 0 && Nb > 0 && N > 0 && P <= 65535 && (src64 || src) && (tgt64 || tgt));
    dim3 g(vcr_cdiv(N, 256), P);
    make_pairs_kernel<<<g, 256, 0, stream>>>(base, Nb, idx_src, idx_tgt, pose, N, src64, tgt64, src, tgt);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

VCR_API int vcr_crop_nearest(const double* pc64, int P, int N, int keep, float* out, cudaStream_t stream) {
    VCR_REQUIRE(pc64 && out && P > 0 && N > 0 && keep > 0 && keep <= N);
    if ((size_t)N * sizeof(double) > 200 * 1024) return VCR_ERR_UNSUPPORTED;
    const size_t smem = (size_t)N * sizeof(double);
    // set on every launch: the attribute is per device, and one process may drive several (nn.DataParallel)
    if (cudaFuncSetAttribute(crop_nearest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) return VCR_ERR_LAUNCH;
    crop_nearest_kernel<<<P, 256, smem, stream>>>(pc64, N, keep, out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

namespace {
// Workspace of vcr_crop_nearest_sort: two (key, index) buffers the passes alternate between, then the per-tile counts.
struct CropSortLayout {
    size_t keys0, keys1, idx0, idx1, counts, bytes;
    int tiles;
};
size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
bool crop_sort_shape_ok(int P, int N) { return P >= 1 && N >= 1 && (long long)P * N <= 2147483647ll; }
CropSortLayout crop_sort_layout(int P, int N) {
    CropSortLayout l;
    const size_t n = (size_t)P * N;
    l.tiles = vcr_cdiv(N, kSortTile);
    l.keys0 = 0;
    l.keys1 = l.keys0 + align256(n * 8);
    l.idx0 = l.keys1 + align256(n * 8);
    l.idx1 = l.idx0 + align256(n * 4);
    l.counts = l.idx1 + align256(n * 4);
    l.bytes = l.counts + align256((size_t)P * 256 * l.tiles * 4);
    return l;
}
}  // namespace

VCR_API size_t vcr_crop_nearest_workspace_bytes(int P, int N) {
    return crop_sort_shape_ok(P, N) ? crop_sort_layout(P, N).bytes : 0;
}

VCR_API int vcr_crop_nearest_sort(const double* pc64, int P, int N, int keep, float* out, void* workspace,
                                  size_t workspace_bytes, cudaStream_t stream) {
    VCR_REQUIRE(pc64 && out && workspace && ((uintptr_t)workspace & 7) == 0);
    if (!crop_sort_shape_ok(P, N) || keep < 1 || keep > N) return VCR_ERR_UNSUPPORTED;
    const CropSortLayout l = crop_sort_layout(P, N);
    if (workspace_bytes < l.bytes) return VCR_ERR_WORKSPACE;
    char* ws = static_cast<char*>(workspace);
    unsigned long long* keys[2] = {reinterpret_cast<unsigned long long*>(ws + l.keys0),
                                   reinterpret_cast<unsigned long long*>(ws + l.keys1)};
    unsigned* idx[2] = {reinterpret_cast<unsigned*>(ws + l.idx0), reinterpret_cast<unsigned*>(ws + l.idx1)};
    unsigned* counts = reinterpret_cast<unsigned*>(ws + l.counts);
    const size_t n = (size_t)P * N;
    crop_keys_kernel<<<vcr_cdiv(n, 256), 256, 0, stream>>>(pc64, N, n, keys[0], idx[0]);
    VCR_CHECK_LAUNCH();
    const int tiles_total = P * l.tiles;                  // <= P * N
    for (int pass = 0; pass < 8; ++pass) {                // even, so the sorted pairs end in buffer 0
        const int src = pass & 1, shift = 8 * pass;
        radix_hist_kernel<<<tiles_total, kSortThreads, 0, stream>>>(keys[src], N, l.tiles, shift, counts);
        VCR_CHECK_LAUNCH();
        radix_scan_kernel<<<P, kScanThreads, 0, stream>>>(counts, 256 * l.tiles);
        VCR_CHECK_LAUNCH();
        radix_scatter_kernel<<<tiles_total, kSortThreads, 0, stream>>>(keys[src], idx[src], N, l.tiles, shift, counts,
                                                                       keys[src ^ 1], idx[src ^ 1]);
        VCR_CHECK_LAUNCH();
    }
    const size_t total = (size_t)P * keep;
    crop_gather_kernel<<<vcr_cdiv(total, 256), 256, 0, stream>>>(pc64, N, keep, total, idx[0], out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

// acc: device double[8], zero-initialised once per evaluation run; src/tgt [B,3,N], srcK/corrK [B,3,M].
VCR_API int vcr_eval_metrics(const float* src, const float* tgt, int N, const float* srcK, const float* corrK, int M,
                             const float* R_gt, const float* t_gt, const float* R_ab, const float* t_ab,
                             const float* R_ba, const float* t_ba, int B, double* acc, cudaStream_t stream) {
    VCR_REQUIRE(src && tgt && srcK && corrK && R_gt && t_gt && R_ab && t_ab && R_ba && t_ba && acc && B > 0 && N > 0 && M > 0);
    const long long work = (long long)B * (N > M ? N : M);
    int blocks = vcr_cdiv(work, 256);
    if (blocks > 592) blocks = 592;
    eval_metrics_kernel<<<blocks, 256, 0, stream>>>(src, tgt, N, srcK, corrK, M, R_gt, t_gt, R_ab, t_ab, R_ba, t_ba, B, acc);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
