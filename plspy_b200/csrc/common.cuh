// Shared host/device helpers for libplsb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>

#include "../../include/plsb200.h"

namespace plsb {

// ---------------------------------------------------------------- host side
char* err_buf();
void set_err(const char* fmt, ...);
void count_launch(int n = 1);

#define PLSB_CHECK_ARG(cond, ...)                      \
    do {                                               \
        if (!(cond)) {                                 \
            plsb::set_err(__VA_ARGS__);                \
            return PLSB200_EINVAL;                     \
        }                                              \
    } while (0)

#define PLSB_CUDA(call)                                                                     \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            plsb::set_err("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return PLSB200_ECUDA;                                                           \
        }                                                                                   \
    } while (0)

#define PLSB_LAUNCH_CHECK(name)                                                             \
    do {                                                                                    \
        cudaError_t e__ = cudaGetLastError();                                               \
        if (e__ != cudaSuccess) {                                                           \
            plsb::set_err("launch of %s failed: %s", name, cudaGetErrorString(e__));        \
            return PLSB200_ECUDA;                                                           \
        }                                                                                   \
        plsb::count_launch();                                                               \
    } while (0)

inline int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// output-stationary bootstrap-moments path for N > 320 (boot_os.cu), reached through the plsb200_boot_* entry points
size_t boot_os_coef_bytes(int N, int K, int R);
size_t boot_os_workspace(int N, int64_t p, int K, int R);
int boot_os_pack(const double* E, int N, int K, const int32_t* idx, int R, double* coef, cudaStream_t st);
// the factored collapsed bootstrap's J pseudo-resamples in the same layout (boot_os_coef_bytes(N, K, J) bytes)
int boot_os_factor_pack(const double* E, int N, int K, const double* L, int J, const int32_t* sid, double* coef,
                        cudaStream_t st);
int boot_os_moments(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R,
                    const double* pivot, double* sum, double* sumsq, void* workspace, size_t workspace_bytes,
                    cudaStream_t st, const char* what);
// the same with X stored as float32 (widened as the tile-major FP64 image is built); `what` names the entry point in
// error messages
int boot_os_moments(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R,
                    const double* pivot, double* sum, double* sumsq, void* workspace, size_t workspace_bytes,
                    cudaStream_t st, const char* what);

// ---------------------------------------------------------------- device side
#ifdef __CUDACC__

// The split partials of the bootstrap GEMMs, whose period or column range is divided over the grid: out1[i] = sum of
// part1[s*n + i] over s = 0 .. nsplit-1 in that order (deterministic), and out2 likewise from part2 unless out2 is
// null.  Defined in boot.cu.
__global__ void split_sum_kernel(const double* __restrict__ part1, const double* __restrict__ part2, int nsplit,
                                 long long n, double* __restrict__ out1, double* __restrict__ out2);

// D(8x8) += A(8x4, row) * B(4x8, col), FP64 tensor core (SASS: DMMA.8x8x4 -- the only native f64
// MMA shape on sm_100a; the m16n8k{4,8,16} PTX shapes lower to sequences of it).
//   a : A[row = lane/4][k = lane%4]      b : B[k = lane%4][col = lane/4]
//   d0,d1 : D[row = lane/4][col = 2*(lane%4) + {0,1}]
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// non-blocking probe of a phase (mbarrier.test_wait never suspends the thread)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// global -> shared, completion signalled on an mbarrier (bytes multiple of 16, both 16-B aligned)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- thread-block clusters: rank, cluster barrier, remote mbarrier arrive ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
// Remote arrive with the default (release.cta) semantics, as CUTLASS's ClusterBarrier::arrive(cta_id) does: what the
// barriers of these kernels order across CTAs is asynchronous-proxy traffic (bulk copies into shared memory and
// reads of it that have completed when the arrive is issued), so no cluster-scope fence is needed --
// .release.cluster / .acquire.cluster compile to MEMBAR.ALL.GPU + CCTL.IVALL per pipeline stage.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];\n" ::"r"(cluster_addr) : "memory");
}

// ---- ordered source lists of one resample (coefficient packs) ----
// C_r = scatter(E, idx_r): target row i receives the rows E[src] of all sources with idx_r[src] == i, summed in increasing
// src (the order fixes the rounding: deterministic and identical in every pack kernel).  The first packs let every
// target thread scan all N sources -- O(N^2) dependent shared-memory reads per resample, the whole cost of a pack
// (0.42-0.57 ms for 5000 resamples of 300 rows).  Here the block builds, per resample, a stable counting sort of the
// sources by target: histogram (shared-memory atomics: counts are order-independent), exclusive prefix sum (warp 0),
// stable fill (warp 0, 32 sources at a time in order: __match_any_sync ranks the lanes that share a target).
// Afterwards list[start[i] .. start[i+1]) are the sources of target i in increasing order.
// Shared memory: ids[N], start[N + 1], cur[N], list[N] ints.  All threads of the block must call it.
__device__ __forceinline__ void build_source_lists(const int32_t* __restrict__ idx_row, int N, int* ids, int* start,
                                                   int* cur, int* list) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    for (int i = tid; i < N; i += nt) { ids[i] = idx_row[i]; cur[i] = 0; }
    __syncthreads();
    for (int i = tid; i < N; i += nt) atomicAdd(cur + ids[i], 1);
    __syncthreads();
    if (tid < 32) {
        const int ch = (N + 31) / 32, b = lane * ch, e = min(N, b + ch);
        int sum = 0;
        for (int j = b; j < e; ++j) sum += cur[j];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        int run = incl - sum;
        for (int j = b; j < e; ++j) { const int c = cur[j]; start[j] = run; cur[j] = run; run += c; }
        if (lane == 31) start[N] = N;
        __syncwarp();
        for (int base = 0; base < N; base += 32) {
            const int src = base + lane;
            const bool valid = src < N;
            const int key = valid ? ids[src] : -1 - lane;                  // (unique keys for the idle lanes)
            const unsigned m = __match_any_sync(0xffffffffu, key);
            const int rank = __popc(m & ((1u << lane) - 1u));
            if (valid) list[cur[key] + rank] = src;
            __syncwarp();
            if (valid && rank == __popc(m) - 1) cur[key] += rank + 1;     // the last lane of a group advances it
            __syncwarp();
        }
    }
    __syncthreads();
}

// ---- Ampere-style cp.async with zero fill (SASS LDGSTS) ----
template <int BYTES>
__device__ __forceinline__ void cp_async_zfill(void* dst_smem, const void* src_gmem, int src_bytes) {
    if constexpr (BYTES == 16) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_u32(dst_smem)), "l"(src_gmem),
                     "r"(src_bytes)
                     : "memory");
    } else if constexpr (BYTES == 8) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(smem_u32(dst_smem)), "l"(src_gmem),
                     "r"(src_bytes)
                     : "memory");
    } else {
        static_assert(BYTES == 4, "cp.async copies 4, 8 or 16 bytes");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(smem_u32(dst_smem)), "l"(src_gmem),
                     "r"(src_bytes)
                     : "memory");
    }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

#endif  // __CUDACC__
}  // namespace plsb
