// Farthest-point sampling (SURVEY.md K12; reference util/util.py:107-140 == util/fps.py:10-49).
// N <= 14 336: one CTA per cloud (fps_kernel); coordinates and running min-distances live in shared memory; each of the
// npoint sequential steps is one fused pass (distance, running min, arg-max) + a block arg-max.
// 14 336 < N <= 229 376: one thread-block cluster of C in {2, 4, 8, 16} CTAs per cloud (fps_cluster_kernel); CTA r keeps
// the slice [r*S, min(N, (r+1)*S)), S = ceil(N/C), in its shared memory and the CTAs exchange their per-step arg-max
// records through distributed shared memory, one cluster barrier per step.
//
// Canonical arithmetic, identical to oracle/canon.c so indices are bit-exact:
//   barycentre = float(double-sum) / float(N)           (IEEE fp32 division)
//   d = (dx*dx + dy*dy) + dz*dz with separately rounded multiplies and adds (no FMA contraction)
//   arg-max returns the FIRST maximal index.
// Roofline: 12*N bytes read per cloud once; the loop is latency/ALU bound (npoint*N*~9 flops).
#include <atomic>
#include "tc_common.cuh"      // cluster_ctarank / cluster_sync_all / smem_u32

namespace {

constexpr int FPS_THREADS = 512;
constexpr int FPS_MAX_SLICE = 14336;                  // points per CTA: 16 bytes each in 224 KB of shared memory
constexpr int FPS_MAX_CLUSTER = 16;                   // non-portable cluster size; N <= 16 * 14 336 = 229 376
constexpr int FPS_SMEM_MAX = 4 * FPS_MAX_SLICE * (int)sizeof(float);

__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// (value, index) arg-max with ties -> lower index
__device__ __forceinline__ void argmax_combine(float& v, int& i, float ov, int oi) {
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
}

__device__ __forceinline__ int block_argmax(float v, int i, float* sv, int* si) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        argmax_combine(v, i, ov, oi);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();                       // protect sv/si from the previous round's readers
    if (lane == 0) { sv[warp] = v; si[warp] = i; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        v = lane < nw ? sv[lane] : -INFINITY;
        i = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, i, o);
            argmax_combine(v, i, ov, oi);
        }
        if (lane == 0) si[32] = i;
    }
    __syncthreads();
    return si[32];
}

__global__ void __launch_bounds__(FPS_THREADS)
fps_kernel(const float* __restrict__ xyz, int N, int npoint, int32_t* __restrict__ out32,
           int64_t* __restrict__ out64) {
    extern __shared__ __align__(16) float sm[];
    float* X = sm; float* Y = X + N; float* Z = Y + N; float* Dm = Z + N;
    __shared__ float sv[32];
    __shared__ int si[33];
    __shared__ double sd[3][FPS_THREADS / 32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* p = xyz + (size_t)b * 3 * N;
    double sx = 0, sy = 0, sz = 0;
    for (int n = tid; n < N; n += FPS_THREADS) {
        const float x = p[n], y = p[N + n], z = p[2 * N + n];
        X[n] = x; Y[n] = y; Z[n] = z; Dm[n] = 1e10f;
        sx += x; sy += y; sz += z;
    }
    sx = warp_sum(sx); sy = warp_sum(sy); sz = warp_sum(sz);
    if ((tid & 31) == 0) { sd[0][tid >> 5] = sx; sd[1][tid >> 5] = sy; sd[2][tid >> 5] = sz; }
    __syncthreads();
    sx = sy = sz = 0;
    for (int w = 0; w < FPS_THREADS / 32; ++w) { sx += sd[0][w]; sy += sd[1][w]; sz += sd[2][w]; }
    const float bx = __fdiv_rn((float)sx, (float)N), by = __fdiv_rn((float)sy, (float)N),
                bz = __fdiv_rn((float)sz, (float)N);
    float bv = -INFINITY; int bi = 0x7fffffff;
    for (int n = tid; n < N; n += FPS_THREADS) {
        const float d = sqdist3(X[n], Y[n], Z[n], bx, by, bz);
        if (d > bv) { bv = d; bi = n; }
    }
    int far = block_argmax(bv, bi, sv, si);
    for (int s = 0; s < npoint; ++s) {
        if (tid == 0) {
            if (out32) out32[(size_t)b * npoint + s] = far;
            if (out64) out64[(size_t)b * npoint + s] = far;
        }
        const float cx = X[far], cy = Y[far], cz = Z[far];
        bv = -INFINITY; bi = 0x7fffffff;
        for (int n = tid; n < N; n += FPS_THREADS) {
            const float d = sqdist3(X[n], Y[n], Z[n], cx, cy, cz);
            float cur = Dm[n];
            if (d < cur) { cur = d; Dm[n] = d; }
            if (cur > bv) { bv = cur; bi = n; }
        }
        far = block_argmax(bv, bi, sv, si);
    }
}

// ---------------------------------------------------------------- cluster variant ------------------------
using tc::cluster_nctarank;
using tc::cluster_addr;
__device__ __forceinline__ float4 ld_cluster_f4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float ld_cluster_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ double ld_cluster_f64(uint32_t a) {
    double v;
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}

// A CTA's arg-max of one step, {value, global index (bits), x, y, z}: the winner's coordinates travel with it.
__device__ __forceinline__ void put_record(float* rec, float v, int i, float x, float y, float z) {
    rec[0] = v; rec[1] = __int_as_float(i); rec[2] = x; rec[3] = y; rec[4] = z;
}

// After the cluster barrier: lane r < C of every warp reads rank r's record over DSMEM and the warp reduces them.  The
// order (value descending, index ascending) is total, so every warp of every CTA gets the same winner, whatever C.
__device__ __forceinline__ int cluster_argmax(const float* rec, int C, float& cx, float& cy, float& cz) {
    const int lane = threadIdx.x & 31;
    float4 q = make_float4(-INFINITY, __int_as_float(0x7fffffff), 0.f, 0.f);
    float qz = 0.f;
    if (lane < C) {
        const uint32_t a = cluster_addr(rec, lane);
        q = ld_cluster_f4(a);
        qz = ld_cluster_f32(a + 16);
    }
    float v = q.x; int i = __float_as_int(q.y);
    for (int o = C >> 1; o > 0; o >>= 1) {          // C is a power of two: lanes < C only meet lanes < C
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        argmax_combine(v, i, ov, oi);
    }
    i = __shfl_sync(0xffffffffu, i, 0);
    const int src = __ffs(__ballot_sync(0xffffffffu, lane < C && __float_as_int(q.y) == i)) - 1;
    cx = __shfl_sync(0xffffffffu, q.z, src);
    cy = __shfl_sync(0xffffffffu, q.w, src);
    cz = __shfl_sync(0xffffffffu, qz, src);
    return i;
}

// One cluster of C CTAs per cloud (blocks [b*C, (b+1)*C) of a 1-D grid); S points per CTA.  Same arithmetic, tie rule and
// output as fps_kernel.  Record slots alternate by step parity: a CTA rewrites slot k & 1 at step k + 2 only after every
// peer has arrived at barrier k + 1, which each does after its reads of step k.
__global__ void __launch_bounds__(FPS_THREADS)
fps_cluster_kernel(const float* __restrict__ xyz, int N, int S, int npoint, int32_t* __restrict__ out32,
                   int64_t* __restrict__ out64) {
    extern __shared__ __align__(16) float sm[];
    float* X = sm; float* Y = X + S; float* Z = Y + S; float* Dm = Z + S;
    __shared__ float sv[32];
    __shared__ int si[33];
    __shared__ double sd[3][FPS_THREADS / 32];
    __shared__ double part[3];                      // this CTA's coordinate sums, read by every CTA of the cluster
    __shared__ float bary[3];
    __shared__ __align__(16) float rec[2][8];
    const int tid = threadIdx.x;
    const int C = cluster_nctarank(), rank = (int)tc::cluster_ctarank();
    const int b = blockIdx.x / C, lo = rank * S;
    const int cnt = max(0, min(N - lo, S));
    const float* p = xyz + (size_t)b * 3 * N + lo;
    double sx = 0, sy = 0, sz = 0;
    for (int n = tid; n < cnt; n += FPS_THREADS) {
        const float x = p[n], y = p[N + n], z = p[2 * N + n];
        X[n] = x; Y[n] = y; Z[n] = z; Dm[n] = 1e10f;
        sx += x; sy += y; sz += z;
    }
    sx = warp_sum(sx); sy = warp_sum(sy); sz = warp_sum(sz);
    if ((tid & 31) == 0) { sd[0][tid >> 5] = sx; sd[1][tid >> 5] = sy; sd[2][tid >> 5] = sz; }
    __syncthreads();
    if (tid == 0) {
        sx = sy = sz = 0;
        for (int w = 0; w < FPS_THREADS / 32; ++w) { sx += sd[0][w]; sy += sd[1][w]; sz += sd[2][w]; }
        part[0] = sx; part[1] = sy; part[2] = sz;
    }
    tc::cluster_sync_all();
    if (tid == 0) {
        sx = sy = sz = 0;
        for (int r = 0; r < C; ++r) {               // rank order: every CTA forms the same sums
            const uint32_t a = cluster_addr(part, r);
            sx += ld_cluster_f64(a); sy += ld_cluster_f64(a + 8); sz += ld_cluster_f64(a + 16);
        }
        bary[0] = __fdiv_rn((float)sx, (float)N);
        bary[1] = __fdiv_rn((float)sy, (float)N);
        bary[2] = __fdiv_rn((float)sz, (float)N);
    }
    __syncthreads();
    const float bx = bary[0], by = bary[1], bz = bary[2];
    float bv = -INFINITY; int bi = 0x7fffffff;
    for (int n = tid; n < cnt; n += FPS_THREADS) {
        const float d = sqdist3(X[n], Y[n], Z[n], bx, by, bz);
        if (d > bv) { bv = d; bi = lo + n; }
    }
    int w = block_argmax(bv, bi, sv, si);
    if (tid == 0) {
        const int n = w - lo;
        if (cnt > 0) put_record(rec[0], sqdist3(X[n], Y[n], Z[n], bx, by, bz), w, X[n], Y[n], Z[n]);
        else put_record(rec[0], -INFINITY, 0x7fffffff, 0.f, 0.f, 0.f);
    }
    tc::cluster_sync_all();
    float cx, cy, cz;
    int far = cluster_argmax(rec[0], C, cx, cy, cz);
    for (int s = 0;; ++s) {
        if (rank == 0 && tid == 0) {
            if (out32) out32[(size_t)b * npoint + s] = far;
            if (out64) out64[(size_t)b * npoint + s] = far;
        }
        if (s + 1 == npoint) break;
        bv = -INFINITY; bi = 0x7fffffff;
        for (int n = tid; n < cnt; n += FPS_THREADS) {
            const float d = sqdist3(X[n], Y[n], Z[n], cx, cy, cz);
            float cur = Dm[n];
            if (d < cur) { cur = d; Dm[n] = d; }
            if (cur > bv) { bv = cur; bi = lo + n; }
        }
        w = block_argmax(bv, bi, sv, si);
        float* slot = rec[(s + 1) & 1];
        if (tid == 0) {
            const int n = w - lo;
            if (cnt > 0) put_record(slot, Dm[n], w, X[n], Y[n], Z[n]);
            else put_record(slot, -INFINITY, 0x7fffffff, 0.f, 0.f, 0.f);
        }
        tc::cluster_sync_all();
        far = cluster_argmax(slot, C, cx, cy, cz);
    }
    tc::cluster_sync_all();                         // no CTA exits while a peer may still read its shared memory
}

// Clusters of C CTAs with the largest slice the device co-schedules, per device and C (0 = unknown, n + 1 = n clusters;
// -1 when the function attributes cannot be set).  Published with release/acquire like launch_tc_pair's probe.
int fps_cluster_capacity(int C) {
    static std::atomic<int> max_clusters_dev[64][4];
    int dev = 0;
    cudaGetDevice(&dev);
    std::atomic<int>& slot = max_clusters_dev[dev & 63][__builtin_ctz(C) - 1];
    if (slot.load(std::memory_order_acquire) == 0) {
        if (cudaFuncSetAttribute(fps_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FPS_SMEM_MAX) != cudaSuccess ||
            cudaFuncSetAttribute(fps_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
            cudaGetLastError();
            return -1;
        }
        cudaLaunchConfig_t q = {};
        q.gridDim = dim3(C, 1, 1); q.blockDim = dim3(FPS_THREADS, 1, 1); q.dynamicSmemBytes = FPS_SMEM_MAX;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        q.attrs = at; q.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, fps_cluster_kernel, &q) != cudaSuccess) { cudaGetLastError(); n = 0; }
        slot.store(n + 1, std::memory_order_release);
    }
    return slot.load(std::memory_order_acquire) - 1;
}

}  // namespace

// xyz [B,3,N] -> idx [B,npoint] (int32 and/or int64).  N <= 14 336: one CTA per cloud (16*N bytes of shared memory);
// N <= 229 376: one cluster of 2, 4, 8 or 16 CTAs per cloud.  Larger N, or a device that cannot co-schedule the
// cluster, returns VCR_ERR_UNSUPPORTED.
VCR_API int vcr_fps(const float* xyz, int B, int N, int npoint, int32_t* idx32, int64_t* idx64, cudaStream_t stream) {
    VCR_REQUIRE(xyz && (idx32 || idx64) && B > 0 && N > 0 && npoint > 0);
    if (N <= FPS_MAX_SLICE) {
        const size_t smem = (size_t)4 * N * sizeof(float);
        if (smem > 48 * 1024 &&
            cudaFuncSetAttribute(fps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return VCR_ERR_LAUNCH;
        fps_kernel<<<B, FPS_THREADS, smem, stream>>>(xyz, N, npoint, idx32, idx64);
        VCR_CHECK_LAUNCH();
        return VCR_OK;
    }
    if (N > FPS_MAX_CLUSTER * FPS_MAX_SLICE) return VCR_ERR_UNSUPPORTED;
    int C = 2;
    while (C * FPS_MAX_SLICE < N) C *= 2;
    VCR_REQUIRE((long long)B * C <= 0x7fffffffLL);
    const int cap = fps_cluster_capacity(C);
    if (cap < 0) return VCR_ERR_LAUNCH;
    if (cap < 1) return VCR_ERR_UNSUPPORTED;
    const int S = vcr_cdiv(N, C);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * C, 1, 1); cfg.blockDim = dim3(FPS_THREADS, 1, 1);
    cfg.dynamicSmemBytes = (size_t)4 * S * sizeof(float); cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, fps_cluster_kernel, xyz, N, S, npoint, idx32, idx64) != cudaSuccess) {
        cudaGetLastError();
        return VCR_ERR_LAUNCH;
    }
    VCR_CHECK_LAUNCH();
    return VCR_OK;
}
