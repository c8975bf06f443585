// Top-K selection with the canonical order (value descending, ties -> lower index) used by the
// partial-overlap path: key subset of the cross attention (reference model/transformer.py:39-47),
// selectCom (model/vcrnet_model.py:222-223, 244-245) and getCopair (:309).  torch.topk leaves tie
// order unspecified; the oracle (oracle/vcr_oracle.py topk_desc) fixes the same rule.
// n <= 16 384: one CTA per batch row, bitonic sort of 64-bit (order-preserving float key, index) in shared memory.
// 16 384 < n <= 262 144: one thread-block cluster of C in {2, 4, 8, 16} CTAs per row (topk_sort_cluster_kernel), the same
// network over C slices of 16 384 keys; stages whose partner key is in another CTA read it over distributed shared memory.
#include <atomic>
#include "tc_common.cuh"      // cluster_ctarank / cluster_nctarank / cluster_addr / cluster_sync_all

namespace {

__device__ __forceinline__ unsigned int float_desc_key(float v) {
    if (v == 0.f) v = 0.f;                               // -0.0 and +0.0 compare equal: one key
    unsigned int u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);      // ascending order-preserving
    return ~u;                                           // descending
}

__global__ void topk_sort_kernel(const float* __restrict__ vals, int n, int npad, int K,
                                 int* __restrict__ idx_out, uint8_t* __restrict__ mask_out) {
    extern __shared__ unsigned long long keys[];
    const int b = blockIdx.x;
    const float* v = vals + (size_t)b * n;
    for (int i = threadIdx.x; i < npad; i += blockDim.x)
        keys[i] = i < n ? (((unsigned long long)float_desc_key(v[i]) << 32) | (unsigned int)i) : ~0ull;
    __syncthreads();
    for (int size = 2; size <= npad; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < npad / 2; t += blockDim.x) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long a = keys[lo], c = keys[hi];
                if ((a > c) == up) { keys[lo] = c; keys[hi] = a; }
            }
            __syncthreads();
        }
    }
    if (mask_out)
        for (int i = threadIdx.x; i < n; i += blockDim.x) mask_out[(size_t)b * n + i] = 0;
    __syncthreads();
    for (int r = threadIdx.x; r < K; r += blockDim.x) {
        const int i = (int)(keys[r] & 0xffffffffu);
        if (idx_out) idx_out[(size_t)b * K + r] = i;
        if (mask_out) mask_out[(size_t)b * n + i] = 1;
    }
}

// npad <= 1024: one key per thread.  Compare-exchange partners closer than a warp are reached with shuffles, the 15 stages
// with stride >= 32 go through double-buffered shared memory (one barrier each): 15 barriers instead of 55.  Same network,
// same result as topk_sort_kernel.
__global__ void __launch_bounds__(1024)
topk_sort_warp_kernel(const float* __restrict__ vals, int n, int npad, int K, int* __restrict__ idx_out,
                      uint8_t* __restrict__ mask_out) {
    __shared__ unsigned long long xch[2][1024];
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* v = vals + (size_t)b * n;
    unsigned long long key = tid < n ? (((unsigned long long)float_desc_key(v[tid]) << 32) | (unsigned int)tid) : ~0ull;
    int buf = 0;
    for (int size = 2; size <= npad; size <<= 1) {
        const bool up = (tid & size) == 0;
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            unsigned long long other;
            if (stride >= 32) {
                xch[buf][tid] = key;
                __syncthreads();
                other = xch[buf][tid ^ stride];
                buf ^= 1;                                  // the next smem stage writes the other buffer: no second barrier
            } else {
                other = __shfl_xor_sync(0xffffffffu, key, stride);
            }
            const bool lower = (tid & stride) == 0;
            const bool take_min = lower == up;
            key = take_min ? (key < other ? key : other) : (key > other ? key : other);
        }
    }
    if (mask_out)
        for (int i = tid; i < n; i += blockDim.x) mask_out[(size_t)b * n + i] = 0;
    __syncthreads();
    if (tid < K) {
        const int i = (int)(key & 0xffffffffu);
        if (idx_out) idx_out[(size_t)b * K + tid] = i;
        if (mask_out) mask_out[(size_t)b * n + i] = 1;
    }
}

constexpr int TOPK_SLICE = 16384;                    // keys per CTA of a cluster: 128 KB of 64-bit keys
constexpr int TOPK_MAX_CLUSTER = 16;                 // non-portable cluster size; n <= 16 * 16 384 = 262 144
constexpr int TOPK_CL_THREADS = 1024;
constexpr int TOPK_CL_KEYS = TOPK_SLICE / TOPK_CL_THREADS;   // keys per thread in a cross-CTA stage
constexpr int TOPK_CL_SMEM = TOPK_SLICE * (int)sizeof(unsigned long long);

__device__ __forceinline__ unsigned long long ld_cluster_u64(uint32_t a) {
    unsigned long long v;
    asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
    return v;
}

// One cluster of C CTAs per row (blocks [b*C, (b+1)*C) of a 1-D grid); CTA r holds the keys of global positions
// [r*16384, (r+1)*16384) of the padded row.  The network, directions included, is topk_sort_kernel's on npad = C*16384
// keys.  A stage with stride >= 16384 pairs position g with g ^ stride in CTA r ^ (stride / 16384), at the same local
// offset: every thread reads its 16 partner keys into registers, a cluster barrier, then it writes its own 16 results.
// Compare-exchanging in place would race with the partner reading the same keys.  The keys are unique (the index is in the
// low word), so the result is the same total order as the one-CTA kernels, for every C.
__global__ void __launch_bounds__(TOPK_CL_THREADS)
topk_sort_cluster_kernel(const float* __restrict__ vals, int n, int K, int* __restrict__ idx_out,
                         uint8_t* __restrict__ mask_out) {
    extern __shared__ unsigned long long keys[];
    const int tid = threadIdx.x;
    const int C = tc::cluster_nctarank(), rank = (int)tc::cluster_ctarank();
    const int b = blockIdx.x / C, base = rank * TOPK_SLICE, npad = C * TOPK_SLICE;
    const float* v = vals + (size_t)b * n;
    for (int l = tid; l < TOPK_SLICE; l += TOPK_CL_THREADS) {
        const int g = base + l;
        keys[l] = g < n ? (((unsigned long long)float_desc_key(v[g]) << 32) | (unsigned int)g) : ~0ull;
        if (mask_out && g < n) mask_out[(size_t)b * n + g] = 0;   // ordered before any CTA's ones by the cluster barriers
    }
    __syncthreads();
    for (int size = 2; size <= npad; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride >= TOPK_SLICE) {
                const int step = stride / TOPK_SLICE;
                tc::cluster_sync_all();                        // peers started, their previous stages' keys written
                const uint32_t pa = tc::cluster_addr(keys, rank ^ step);
                unsigned long long other[TOPK_CL_KEYS];
#pragma unroll
                for (int q = 0; q < TOPK_CL_KEYS; ++q)
                    other[q] = ld_cluster_u64(pa + 8u * (uint32_t)(tid + q * TOPK_CL_THREADS));
                tc::cluster_sync_all();                        // every read of this stage is done before any write
                const bool up = (base & size) == 0;            // size > 16384: the same for the whole slice
                const bool take_min = ((rank & step) == 0) == up;
#pragma unroll
                for (int q = 0; q < TOPK_CL_KEYS; ++q) {
                    const int l = tid + q * TOPK_CL_THREADS;
                    const unsigned long long a = keys[l], o = other[q];
                    keys[l] = take_min ? (a < o ? a : o) : (a > o ? a : o);
                }
            } else {
                for (int t = tid; t < TOPK_SLICE / 2; t += TOPK_CL_THREADS) {
                    const int lo = 2 * t - (t & (stride - 1));
                    const int hi = lo + stride;
                    const bool up = ((base + lo) & size) == 0;
                    const unsigned long long a = keys[lo], c = keys[hi];
                    if ((a > c) == up) { keys[lo] = c; keys[hi] = a; }
                }
            }
            __syncthreads();
        }
    }
    // Sorted position base + l.  No CTA reads a peer's keys after the last cross-CTA stage's second barrier, so CTAs
    // may exit independently.
    for (int l = tid; l < TOPK_SLICE && base + l < K; l += TOPK_CL_THREADS) {
        const int i = (int)(keys[l] & 0xffffffffu);
        if (idx_out) idx_out[(size_t)b * K + base + l] = i;
        if (mask_out) mask_out[(size_t)b * n + i] = 1;
    }
}

// Clusters of C CTAs the device co-schedules, per device and C (0 = unknown, n + 1 = n clusters; -1 when the function
// attributes cannot be set).  Same probe as fps_cluster_capacity.
int topk_cluster_capacity(int C) {
    static std::atomic<int> max_clusters_dev[64][4];
    int dev = 0;
    cudaGetDevice(&dev);
    std::atomic<int>& slot = max_clusters_dev[dev & 63][__builtin_ctz(C) - 1];
    if (slot.load(std::memory_order_acquire) == 0) {
        if (cudaFuncSetAttribute(topk_sort_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_CL_SMEM) != cudaSuccess ||
            cudaFuncSetAttribute(topk_sort_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
            cudaGetLastError();
            return -1;
        }
        cudaLaunchConfig_t q = {};
        q.gridDim = dim3(C, 1, 1); q.blockDim = dim3(TOPK_CL_THREADS, 1, 1); q.dynamicSmemBytes = TOPK_CL_SMEM;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        q.attrs = at; q.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, topk_sort_cluster_kernel, &q) != cudaSuccess) { cudaGetLastError(); nc = 0; }
        slot.store(nc + 1, std::memory_order_release);
    }
    return slot.load(std::memory_order_acquire) - 1;
}

int topk_cluster_launch(const float* vals, int B, int n, int npad, int K, int* idx_out, uint8_t* mask_out,
                        cudaStream_t stream) {
    if (npad > TOPK_MAX_CLUSTER * TOPK_SLICE) return VCR_ERR_UNSUPPORTED;
    const int C = npad / TOPK_SLICE;
    VCR_REQUIRE((long long)B * C <= 0x7fffffffLL);
    const int cap = topk_cluster_capacity(C);
    if (cap < 0) return VCR_ERR_LAUNCH;
    if (cap < 1) return VCR_ERR_UNSUPPORTED;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * C, 1, 1); cfg.blockDim = dim3(TOPK_CL_THREADS, 1, 1);
    cfg.dynamicSmemBytes = TOPK_CL_SMEM; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, topk_sort_cluster_kernel, vals, n, K, idx_out, mask_out) != cudaSuccess) {
        cudaGetLastError();
        return VCR_ERR_LAUNCH;
    }
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}

}  // namespace

// vals [B,n] -> idx_out [B,K] (sorted, optional) and/or mask_out [B,n] uint8 (1 = selected, optional).
// n <= 16 384: one CTA per row; n <= 262 144: one cluster of 2, 4, 8 or 16 CTAs per row.  Larger n, or a device that cannot
// co-schedule the cluster, returns VCR_ERR_UNSUPPORTED.  No workspace, no host synchronisation (graph-capturable).
VCR_API int vcr_topk_select(const float* vals, int B, int n, int K, int* idx_out, uint8_t* mask_out,
                            cudaStream_t stream) {
    VCR_REQUIRE(vals && (idx_out || mask_out) && B > 0 && n > 0 && K > 0 && K <= n);
    int npad = 2;
    while (npad < n) npad <<= 1;
    if (npad >= 32 && npad <= 1024) {
        topk_sort_warp_kernel<<<B, npad, 0, stream>>>(vals, n, npad, K, idx_out, mask_out);
        VCR_CHECK_LAUNCH();
        return VCR_OK;
    }
    if (npad > TOPK_SLICE) return topk_cluster_launch(vals, B, n, npad, K, idx_out, mask_out, stream);
    const size_t smem = (size_t)npad * sizeof(unsigned long long);
    if (smem > 224 * 1024) return VCR_ERR_UNSUPPORTED;
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(topk_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return VCR_ERR_LAUNCH;
    const int threads = npad / 2 < 1024 ? (npad / 2 < 32 ? 32 : npad / 2) : 1024;
    topk_sort_kernel<<<B, threads, smem, stream>>>(vals, n, npad, K, idx_out, mask_out);
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
