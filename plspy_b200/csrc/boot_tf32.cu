// K4 fast mode: bootstrap salience moments on the 5th-generation tensor cores (tcgen05, kind::tf32) with the
// 3xTF32 split:  x = xh + xl, c = ch + cl (each TF32-exact),  x.c ~= xh.cl + xl.ch + xh.ch  (FP32 accumulate in
// TMEM), moments folded in FP64 registers.
//
// Same GEMM as boot.cu (reference: bootstrap_permutation.py:557-626, 695):
//       VS[v, (r,k)] = sum_i X[i, v] . C_r[i, k]          M = voxels, N = (resample, k) columns, K-dim = rows i
//   * M tile = 128 voxels = the 128 TMEM lanes; an epilogue thread owns one voxel and keeps its 2*Kp running
//     moments in FP64 registers for a whole work unit.
//   * N tile = `ntile` columns (240 or 256) = a whole number of resamples, so column -> k is compile-time.
//     Two accumulator stages (2 x 256 TMEM columns): the epilogue of tile t overlaps the MMAs of tile t+1.
//   * K-dim streamed in blocks of 16 rows.  Both operands are pre-split into TF32 hi/lo planes and pre-packed
//     (split_x_tf32_kernel, coef_pack_tf32_kernel) as exact images of the K-major SWIZZLE_64B shared-memory tiles
//     the MMA descriptors address, so a pipeline stage is two contiguous chunks moved by 1-D bulk copies
//     (cp.async.bulk, TMA engine) -- no tensor maps.  Per stage: Xh, Xl (128 x 16) and Ch, Cl (ntile x 16), six
//     MMAs (three products x two k-steps of 8).
//   * warps 0-3 = epilogue (tcgen05.ld 32x32b -> FADD pivot -> FP32 tile sums -> FP64 running moments), warp 4 =
//     bulk-copy producer, warp 5 = MMA issuer (one thread) + TMEM allocator: the two single-thread roles carry the
//     highest warp ids of their schedulers, which the issue arbiter favours over the epilogue warps they share with.
//   * persistent CTAs, one per SM; work unit = (voxel tile, contiguous range of column tiles); units are ordered
//     so that CTAs running concurrently stream the same coefficient range (L2-resident).
#include "common.cuh"
#include <stdlib.h>

// The probe modes that isolate the limiter of the tcgen05 kernel (free-running roles, no producer, no epilogue
// arithmetic: WRONG RESULTS by construction) exist only in builds with -DPLSB_PROBES (tools/); in the product library
// TF_DBG is the constant 0 and every probe branch is compiled out.
#ifdef PLSB_PROBES
#define TF_DBG(a) ((a).dbg)
#else
#define TF_DBG(a) 0
#endif

namespace plsb {

constexpr int TF_KB = 16;                 // rows per pipeline stage
constexpr int TF_MV = 128;                // voxels per tile
constexpr int TF_THREADS = 192;
constexpr uint32_t TF_A_PLANE = TF_MV * TF_KB * 4;     // 8 KB: one TF32 plane of the X block
constexpr uint32_t TF_A_STAGE = 2 * TF_A_PLANE;        // hi + lo

struct TfPlan {
    int Kp, period, ntile, nres, nkb, nct, nstage, nsplit, ct_per_split, nks_last;
    int cg;            // CTAs per MMA group: 2 = CTA pairs (cta_group::2, UMMA M = 256), 1 = single CTA
    int64_t nvt;       // voxel-tile groups (tiles / cg, the last group zero-padded)
    uint32_t b_plane, stage_bytes;
    size_t smem_bytes;
};

static int gcd_i(int a, int b) { return b ? gcd_i(b, a % b) : a; }

static bool tf_plan(int N, int K, int R, int64_t p, TfPlan& t) {
    static const int kps[] = {2, 3, 4, 5, 6, 8, 10, 12, 15, 16, 20, 24};
    if (K < 1 || K > 24 || N < 1 || R < 1) return false;
    t.Kp = 0;
    for (int kp : kps)
        if (kp >= K) { t.Kp = kp; break; }
    t.period = t.Kp * 16 / gcd_i(t.Kp, 16);
    t.ntile = (256 / t.period) * t.period;
    t.nres = t.ntile / t.Kp;
    t.nkb = (int)cdiv(N, TF_KB);
    t.nks_last = (int)cdiv(N - TF_KB * (t.nkb - 1), 8);
    t.nct = (int)cdiv(R, t.nres);
    t.b_plane = (uint32_t)t.ntile * TF_KB * 4;
    static const char* const env = getenv("PLSB200_TF32_CTA_GROUP");      // read once per process
    // default: CTA pairs (23.4 ms on the bench workload vs 24.2 ms single-CTA once the epilogue stopped being the
    // limiter: the pair moves a third less data through L2 and shared memory); PLSB200_TF32_CTA_GROUP=1 selects the
    // single-CTA kernel
    t.cg = (env && env[0] == '1') ? 1 : 2;
#ifdef PLSB_PROBES
    const char* dbg = getenv("PLSB200_TF32_DEBUG");     // the no-producer probe modes only make sense without the relay
    if (dbg && (dbg[0] == '2' || dbg[0] == '4')) t.cg = 1;
#endif
    t.stage_bytes = TF_A_STAGE + 2 * t.b_plane / t.cg;
    int ns = (int)((227 * 1024 - 2048) / t.stage_bytes);
    if (ns > 8) ns = 8;
    if (ns < 2) return false;
    t.nstage = ns;
    t.smem_bytes = (size_t)ns * t.stage_bytes + 1024 + 256;
    t.nvt = cdiv(cdiv(p > 0 ? p : 1, TF_MV), t.cg);
    const int nsm = num_sms() / t.cg;
    int best = 1; double best_cost = 1e30;
    for (int n = 1; n <= 8; ++n) {
        if (n > 1 && t.nct / n < 4) break;
        const double waves = (double)t.nvt * n / nsm;
        const double cost = ceil(waves) / waves + 0.01 * (n - 1);
        if (cost < best_cost - 1e-12) { best_cost = cost; best = n; }
    }
    t.ct_per_split = (int)cdiv(t.nct, best);
    t.nsplit = (int)cdiv(t.nct, t.ct_per_split);
    return true;
}

// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
__device__ __forceinline__ void split_tf32(double x, float& hi, float& lo) {
    hi = tf32_rna((float)x);
    lo = tf32_rna((float)(x - (double)hi));
}

// X (N x p, FP64, row-major) -> image [voxel tile][k-block][hi|lo][128 voxels x 16 rows], each plane in the
// K-major SWIZZLE_64B order: voxel r, row j -> r*64 + ((j/4) ^ ((r/2)&3))*16 + (j%4)*4 bytes.  T = float: X stored
// as float32; its widened value is split, so the planes are those of the widened matrix.
template <typename T>
__global__ void __launch_bounds__(TF_MV) split_x_tf32_kernel(const T* __restrict__ X, int N, long long p,
                                                            long long ldx, int nkb, float* __restrict__ img) {
    const int r = threadIdx.x;
    const long long vt = blockIdx.x;
    const int kb = blockIdx.y;
    const long long v = vt * TF_MV + r;
    float hi[TF_KB], lo[TF_KB];
#pragma unroll
    for (int j = 0; j < TF_KB; ++j) {
        const int row = kb * TF_KB + j;
        const double x = (row < N && v < p) ? (double)__ldg(X + (long long)row * ldx + v) : 0.0;
        split_tf32(x, hi[j], lo[j]);
    }
    float* base = img + ((size_t)vt * nkb + kb) * (TF_A_STAGE / 4);
    const int sw = (r >> 1) & 3;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int pos = c ^ sw;
        *reinterpret_cast<float4*>(base + r * 16 + pos * 4) = make_float4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
        *reinterpret_cast<float4*>(base + TF_A_PLANE / 4 + r * 16 + pos * 4) =
            make_float4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    }
}

// coefficients C_r = scatter(E, idx_r) -> image [column tile][k-block][hi|lo][ntile columns x 16 rows] (same
// swizzled order, column n = (r % nres)*Kp + k).  One CTA per resample; 256 target rows (16 k-blocks) per pass:
// thread j gathers target row j in index order (deterministic), the hi/lo planes of the pass are assembled in
// shared memory in image order and written out as contiguous K*64-byte runs.  The image is zeroed beforehand
// (padding rows / columns / k >= K).
constexpr int CP_ROWS = 256;                       // target rows per pass
constexpr int CP_KB = CP_ROWS / TF_KB;             // k-blocks per pass
__global__ void __launch_bounds__(CP_ROWS) coef_pack_tf32_kernel(const double* __restrict__ E, int N, int K,
                                                                const int32_t* __restrict__ idx, int Kp, int nres,
                                                                int ntile, int nkb, int stage_e,
                                                                float* __restrict__ img) {
    extern __shared__ __align__(16) double smp[];
    float* stg = reinterpret_cast<float*>(smp);                       // [2 planes][CP_KB][K][16]
    int* ids = reinterpret_cast<int*>(stg + 2 * CP_KB * K * TF_KB);   // [N], then the ordered source lists
    int* start = ids + N; int* cur = start + N + 1; int* list = cur + N;
    double* Esm = reinterpret_cast<double*>(ids + ((4 * N + 2) & ~1));
    const double* Es = stage_e ? Esm : E;           // tall designs: E stays in global memory (L2-resident)
    const int r = blockIdx.x, tid = threadIdx.x;
    const int32_t* my = idx + (size_t)r * N;
    if (stage_e)
        for (int i = tid; i < N * K; i += CP_ROWS) Esm[i] = E[i];
    build_source_lists(my, N, ids, start, cur, list);          // (ends with a block barrier: Esm is staged too)
    const int ct = r / nres, nbase = (r % nres) * Kp;
    const size_t plane = (size_t)ntile * TF_KB;      // floats
    const int pstride = CP_KB * K * TF_KB;           // floats per staged plane
    for (int j0 = 0; j0 < N; j0 += CP_ROWS) {
        const int j = j0 + tid;
        double acc[24];
#pragma unroll
        for (int k = 0; k < 24; ++k) acc[k] = 0.0;
        if (j < N) {
            for (int t = start[j]; t < start[j + 1]; ++t) {
                const int src = list[t];
#pragma unroll
                for (int k = 0; k < 24; ++k)
                    if (k < K) acc[k] += Es[src * K + k];
            }
        }
        const int kbl = tid / TF_KB, jj = tid % TF_KB;
#pragma unroll
        for (int k = 0; k < 24; ++k) {
            if (k < K) {
                const int n = nbase + k;
                const int off = (kbl * K + k) * TF_KB + (((jj >> 2) ^ ((n >> 1) & 3)) << 2) + (jj & 3);
                float h, l;
                split_tf32(acc[k], h, l);
                stg[off] = h;
                stg[pstride + off] = l;
            }
        }
        __syncthreads();
        // copy out: (plane, k-block) -> one contiguous run of K*16 floats
        const int kb0 = j0 / TF_KB;
        const int run4 = K * TF_KB / 4;              // float4 per run
        for (int i = tid; i < 2 * CP_KB * run4; i += CP_ROWS) {
            const int q = i % run4, kbl2 = (i / run4) % CP_KB, h = i / (run4 * CP_KB);
            const int kb = kb0 + kbl2;
            if (kb < nkb) {
                const float4 val = *reinterpret_cast<const float4*>(stg + h * pstride + kbl2 * K * TF_KB + 4 * q);
                float* dst = img + ((size_t)ct * nkb + kb) * (2 * plane) + h * plane + (size_t)nbase * TF_KB + 4 * q;
                *reinterpret_cast<float4*>(dst) = val;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------
// tcgen05 helpers
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    // K-major, SWIZZLE_64B: LBO (unused) = 16 B, SBO = 512 B between 8-row groups, version 1, layout type 4
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(512u >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)4 << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

struct TfArgs {
    const float* aimg;
    const float* bimg;
    const double* pivot;
    double* out1;
    double* out2;
    long long p, nvt, nunits;
    int K, R, nkb, nks_last, ntile, nres, nct, ct_per_split, nstage;
    uint32_t b_plane, stage_bytes;
    long long* trace;      // optional (PLSB200_TF32_TRACE=1): per-CTA cycle counters of the role loops, 8 per CTA
    int dbg;               // probe builds only (-DPLSB_PROBES, tools/): PLSB200_TF32_DEBUG 1 = producer and MMA issuer free-running (no full /
                           // empty hand-shake: wrong results, isolates contention from waiting), 2 = no producer at all
};

// ---- cluster helpers: cluster_ctarank, cluster_sync_all, mapa_u32, mbar_arrive_cluster live in common.cuh
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
// COLL: use of the tensor core's A-operand collector buffer -- 0 none, 1 fill (SASS A_KEEP: keep this A for the next MMA),
// 2 lastuse (A_REUSE: take A from the collector instead of shared memory).  Of the three products of a k-step two share
// the hi plane of X, so one of the three A reads from shared memory is saved.
template <int CG, int COLL = 0>
__device__ __forceinline__ void umma_tf32_cg(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1 && COLL == 1) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32.collector::a::fill [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
            "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
            : "memory");
    } else if constexpr (CG == 1 && COLL == 2) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32.collector::a::lastuse [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
            "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
            : "memory");
    } else if constexpr (CG == 1) {
        umma_tf32(d_tmem, da, db, idesc, accumulate);
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
            "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// arrive on the barrier (same offset in every CTA of the group) once all MMAs issued so far have completed
template <int CG>
__device__ __forceinline__ void umma_commit_cg(uint64_t* bar) {
    if constexpr (CG == 1) {
        umma_commit(bar);
    } else {
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
                smem_u32(bar)),
            "h"((uint16_t)3)
            : "memory");
    }
}

// CG = 1: one CTA per SM, UMMA M = 128.
// CG = 2: CTA pair (cluster of 2, cta_group::2), UMMA M = 256: the pair works on two adjacent voxel tiles against the
//   same coefficient stream; each CTA stages its own X block and HALF of the coefficient block (the tensor cores
//   of the pair share the halves), which halves the shared-memory and L2 traffic of the larger operand.
//   Rank 0 issues the MMAs; rank 1's warp 1 relays "my stage has landed" to rank 0; MMA completion is multicast
//   to the barriers of both CTAs; both epilogues report "accumulator drained" to rank 0.
template <int KP, int CG>
__global__ void __launch_bounds__(TF_THREADS, 1) boot_moments_tf32_kernel(const TfArgs a) {
    constexpr int P = KP * 16 / (KP % 16 == 0 ? 16 : (KP % 8 == 0 ? 8 : (KP % 4 == 0 ? 4 : (KP % 2 == 0 ? 2 : 1))));
    constexpr int NCH = P / 16;   // 16-column chunks per period
    extern __shared__ unsigned char smraw_[];
    // dynamic shared memory is only 16-byte aligned by contract: align the ring to 1024 B by hand
    const uint32_t s0 = smem_u32(smraw_);
    unsigned char* ring = smraw_ + ((1024u - (s0 & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)a.nstage * a.stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + 8;
    uint64_t* pfull = bars + 16;          // CG == 2, rank 0: the peer's stage has landed
    uint64_t* tfull = bars + 24;
    uint64_t* tempty = bars + 26;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 28);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
    // (CTAs of a wave stream the same coefficient tiles at the same time on purpose: starting each group at a different
    // column tile to spread the L2 load was measured 8 % SLOWER)
    const long long u_first = blockIdx.x / CG, u_step = gridDim.x / CG;
    const uint32_t bhalf = a.b_plane / CG;              // bytes of one coefficient plane staged by this CTA
    const uint32_t cta_stage_bytes = TF_A_STAGE + 2u * bhalf;

    if (tid == 0) {
        for (int s = 0; s < a.nstage; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); mbar_init(pfull + s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull + s, 1); mbar_init(tempty + s, 4 * CG); }
        mbar_fence_init();
    }
    if (warp == 5) {
        if constexpr (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n");
        }
    }
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *tmem_slot;

    if (warp == 4) {
        // ===================== producer: stream the operand images into the ring =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (long long u = u_first; u < a.nunits; u += u_step) {
                const long long vt = (u % a.nvt) * CG + rank;
                const int split = (int)(u / a.nvt);
                const int ct0 = split * a.ct_per_split, ct1 = min(a.nct, ct0 + a.ct_per_split);
                const char* asrc = reinterpret_cast<const char*>(a.aimg) + (size_t)vt * a.nkb * TF_A_STAGE;
                for (int ct = ct0; ct < ct1; ++ct) {
                    const char* bsrc = reinterpret_cast<const char*>(a.bimg) + (size_t)ct * a.nkb * (2u * a.b_plane);
                    for (int kb = 0; kb < a.nkb; ++kb) {
                        if (TF_DBG(a) == 2 || TF_DBG(a) == 4) continue;
                        if (TF_DBG(a) == 0 || TF_DBG(a) == 3 || TF_DBG(a) == 5) mbar_wait(empty + stage, phase ^ 1u);
                        unsigned char* dst = ring + (size_t)stage * a.stage_bytes;
                        mbar_expect_tx(full + stage, cta_stage_bytes);
                        bulk_g2s(dst, asrc + (size_t)kb * TF_A_STAGE, TF_A_STAGE, full + stage);
                        const char* bs = bsrc + (size_t)kb * (2u * a.b_plane) + rank * bhalf;
#pragma unroll
                        for (int h = 0; h < 2; ++h)      // hi plane, lo plane (this CTA's rows of each)
                            bulk_g2s(dst + TF_A_STAGE + h * bhalf, bs + (size_t)h * a.b_plane, bhalf, full + stage);
                        if (++stage == a.nstage) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 5) {
        if (lane == 0 && rank == 0) {
            // ===================== MMA issuer (single thread of the leader CTA) =====================
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(a.ntile >> 3) << 17) |
                                   ((uint32_t)((128 * CG) >> 4) << 24);
            int stage = 0; uint32_t phase = 0; int as = 0; uint32_t aphase = 0;
            // descriptors differ only in their 14-bit start-address field (bytes >> 4): one base per operand plane,
            // per-stage and per-k-step offsets are plain adds (the ring lies below 256 KB, so the field cannot overflow)
            const uint64_t d_ah = umma_desc_sw64(smem_u32(ring));
            const uint64_t d_al = d_ah + (TF_A_PLANE >> 4), d_bh = d_ah + (TF_A_STAGE >> 4), d_bl = d_bh + (bhalf >> 4);
            const uint64_t stage_step = a.stage_bytes >> 4;
            const int last_kb = a.nkb - 1;
            for (long long u = u_first; u < a.nunits; u += u_step) {
                const int split = (int)(u / a.nvt);
                const int ct0 = split * a.ct_per_split, ct1 = min(a.nct, ct0 + a.ct_per_split);
                for (int ct = ct0; ct < ct1; ++ct) {
                    if constexpr (CG == 2) mbar_wait_cluster(tempty + as, aphase ^ 1u);
                    else mbar_wait(tempty + as, aphase ^ 1u);
                    tc_fence_after();
                    const uint32_t d = tbase + (uint32_t)as * 256u;
                    uint32_t accum = 0u;
                    for (int kb = 0; kb <= last_kb; ++kb) {
                        if (TF_DBG(a) == 0 || TF_DBG(a) == 3 || TF_DBG(a) == 5) {
                            mbar_wait(full + stage, phase);
                            if constexpr (CG == 2) mbar_wait_cluster(pfull + stage, phase);
                        }
                        tc_fence_after();
                        const uint64_t so = (uint64_t)stage * stage_step;
                        const uint64_t ah = d_ah + so, al = d_al + so, bh = d_bh + so, bl = d_bl + so;
                        // the two products with the hi plane of X back to back: the second takes A from the collector
                        // buffer instead of shared memory
                        umma_tf32_cg<CG, 1>(d, ah, bl, idesc, accum);
                        umma_tf32_cg<CG, 2>(d, ah, bh, idesc, 1u);
                        umma_tf32_cg<CG, 0>(d, al, bh, idesc, 1u);
                        accum = 1u;
                        if (kb != last_kb || a.nks_last == 2) {          // second k-step of 8 rows (32 bytes further)
                            umma_tf32_cg<CG, 1>(d, ah + 2, bl + 2, idesc, 1u);
                            umma_tf32_cg<CG, 2>(d, ah + 2, bh + 2, idesc, 1u);
                            umma_tf32_cg<CG, 0>(d, al + 2, bh + 2, idesc, 1u);
                        }
                        umma_commit_cg<CG>(empty + stage);       // frees the smem slot (in both CTAs) once read
                        if (++stage == a.nstage) { stage = 0; phase ^= 1u; }
                    }
                    umma_commit_cg<CG>(tfull + as);              // accumulator complete -> epilogue(s)
                    if (++as == 2) { as = 0; aphase ^= 1u; }
                }
            }
        } else if (CG == 2 && lane == 0) {
            // ===================== relay (rank 1): tell the leader that my stage has landed =====================
            int stage = 0; uint32_t phase = 0;
            for (long long u = u_first; u < a.nunits; u += u_step) {
                const int split = (int)(u / a.nvt);
                const int ct0 = split * a.ct_per_split, ct1 = min(a.nct, ct0 + a.ct_per_split);
                for (int ct = ct0; ct < ct1; ++ct)
                    for (int kb = 0; kb < a.nkb; ++kb) {
                        mbar_wait(full + stage, phase);
                        mbar_arrive_cluster(mapa_u32(smem_u32(pfull + stage), 0));
                        if (++stage == a.nstage) { stage = 0; phase ^= 1u; }
                    }
            }
        }
    } else {
        // ===================== epilogue: TMEM -> FP64 running moments =====================
        const int quarter = warp & 3;                        // TMEM lane quarter this warp may access
        const int row = quarter * 32 + lane;
        int as = 0; uint32_t aphase = 0;
        const uint32_t tempty0 = CG == 2 ? mapa_u32(smem_u32(tempty), 0) : smem_u32(tempty);
        for (long long u = u_first; u < a.nunits; u += u_step) {
            const long long vt = (u % a.nvt) * CG + rank;
            const int split = (int)(u / a.nvt);
            const int ct0 = split * a.ct_per_split, ct1 = min(a.nct, ct0 + a.ct_per_split);
            const long long v = vt * TF_MV + row;
            float piv[KP];
            double s1[KP], s2[KP];
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                piv[k] = (a.pivot != nullptr && k < a.K && v < a.p) ? (float)__ldg(a.pivot + v * a.K + k) : 0.f;
                s1[k] = 0.0; s2[k] = 0.0;
            }
            for (int ct = ct0; ct < ct1; ++ct) {
                mbar_wait(tfull + as, aphase);
                tc_fence_after();
                const uint32_t t0 = tbase + ((uint32_t)(quarter * 32) << 16) + (uint32_t)as * 256u;
                const int nvalid = min(a.nres, a.R - ct * a.nres) * KP;     // valid columns of this tile
                if (TF_DBG(a) == 5) {
                    // development only: all the tensor-memory loads of a tile, none of the arithmetic
                    for (int c0 = 0; c0 < a.ntile; c0 += 16) {
                        uint32_t x[16];
                        tmem_ld16(t0 + (uint32_t)c0, x);
                        tmem_ld_wait();
                        s1[0] += (double)__uint_as_float(x[c0 & 15]);
                    }
                } else if (TF_DBG(a) >= 3) {
                    // development only: drain the accumulator without the FP64 fold
                    uint32_t x[16];
                    tmem_ld16(t0, x);
                    tmem_ld_wait();
                    s1[0] += (double)__uint_as_float(x[0]);
                } else {
                    // The <= 128 resamples of one tile are summed in FP32 (pivot-centred values: |d| ~ the bootstrap
                    // spread, 20 terms at K = 12 -> relative error ~1e-7), the tile sums are folded into the FP64
                    // running moments: one F2F / DADD pair per k and tile instead of one per element.  (With the FP64
                    // fold per element the epilogue warps slowed the MMAs down by 13 %.)
                    float f1[KP], f2[KP];
#pragma unroll
                    for (int k = 0; k < KP; ++k) { f1[k] = 0.f; f2[k] = 0.f; }
                    if (nvalid == a.ntile) {
                        for (int per = 0; per < a.ntile; per += P) {
#pragma unroll
                            for (int q = 0; q < NCH; ++q) {
                                uint32_t x[16];
                                tmem_ld16(t0 + (uint32_t)(per + 16 * q), x);
                                tmem_ld_wait();
#pragma unroll
                                for (int e = 0; e < 16; ++e) {
                                    const int k = (16 * q + e) % KP;
                                    const float dv = __uint_as_float(x[e]) - piv[k];
                                    f1[k] += dv;
                                    f2[k] = fmaf(dv, dv, f2[k]);
                                }
                            }
                        }
                    } else {
                        for (int per = 0; per < nvalid; per += P) {
#pragma unroll
                            for (int q = 0; q < NCH; ++q) {
                                uint32_t x[16];
                                tmem_ld16(t0 + (uint32_t)(per + 16 * q), x);
                                tmem_ld_wait();
#pragma unroll
                                for (int e = 0; e < 16; ++e) {
                                    const int k = (16 * q + e) % KP;
                                    if (per + 16 * q + e < nvalid) {
                                        const float dv = __uint_as_float(x[e]) - piv[k];
                                        f1[k] += dv;
                                        f2[k] = fmaf(dv, dv, f2[k]);
                                    }
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int k = 0; k < KP; ++k) { s1[k] += (double)f1[k]; s2[k] += (double)f2[k]; }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (CG == 2) mbar_arrive_cluster(tempty0 + (uint32_t)as * 8u);
                    else mbar_arrive(tempty + as);
                }
                if (++as == 2) { as = 0; aphase ^= 1u; }
            }
            if (v < a.p) {
                double* o1 = a.out1 + ((size_t)split * a.p + v) * a.K;
                double* o2 = a.out2 + ((size_t)split * a.p + v) * a.K;
#pragma unroll
                for (int k = 0; k < KP; ++k)
                    if (k < a.K) { o1[k] = s1[k]; o2[k] = s2[k]; }
            }
        }
    }
    __syncwarp();            // re-converge the warps whose lane 0 ran a role loop before the aligned barriers
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 5) {
        __syncwarp();
        if constexpr (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tbase));
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;\n" ::"r"(tbase));
    }
}

template <int KP, int CG>
static int launch_tf32_cg(const TfPlan& t, const TfArgs& a, cudaStream_t st) {
    PLSB_CUDA(cudaFuncSetAttribute(boot_moments_tf32_kernel<KP, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)t.smem_bytes));
    const long long groups = a.nunits < num_sms() / CG ? a.nunits : num_sms() / CG;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(groups * CG));
    cfg.blockDim = dim3(TF_THREADS);
    cfg.dynamicSmemBytes = t.smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CG > 1 ? 1 : 0;
    PLSB_CUDA(cudaLaunchKernelEx(&cfg, boot_moments_tf32_kernel<KP, CG>, a));
    PLSB_LAUNCH_CHECK("boot_moments_tf32_kernel");
    return PLSB200_OK;
}
template <int KP>
static int launch_tf32(const TfPlan& t, const TfArgs& a, cudaStream_t st) {
    return t.cg == 2 ? launch_tf32_cg<KP, 2>(t, a, st) : launch_tf32_cg<KP, 1>(t, a, st);
}

}  // namespace plsb

using namespace plsb;

extern "C" size_t plsb200_tf32_ximage_bytes(int N, int64_t p) {
    if (N < 1 || p < 1) return 0;
    return (size_t)(2 * cdiv(cdiv(p, TF_MV), 2)) * (size_t)cdiv(N, TF_KB) * TF_A_STAGE;   // tile count padded to even
}

template <typename T>
static int tf32_split_x(const T* X, int N, int64_t p, int64_t ldx, void* ximage, void* stream) {
    PLSB_CHECK_ARG(X && ximage, "tf32_split_x: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && ldx >= p, "tf32_split_x: bad shape");
    const int nkb = (int)cdiv(N, TF_KB);
    PLSB_CHECK_ARG(nkb <= 65535, "tf32_split_x: N too large");
    dim3 grid((unsigned)(2 * cdiv(cdiv(p, TF_MV), 2)), (unsigned)nkb);      // padding tile is written as zeros
    split_x_tf32_kernel<T><<<grid, TF_MV, 0, (cudaStream_t)stream>>>(X, N, p, ldx, nkb, (float*)ximage);
    PLSB_LAUNCH_CHECK("split_x_tf32_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_tf32_split_x(const double* X, int N, int64_t p, int64_t ldx, void* ximage, void* stream) {
    return tf32_split_x(X, N, p, ldx, ximage, stream);
}

extern "C" int plsb200_tf32_split_x32(const float* X, int N, int64_t p, int64_t ldx, void* ximage, void* stream) {
    return tf32_split_x(X, N, p, ldx, ximage, stream);
}

extern "C" size_t plsb200_boot_coef_bytes_tf32(int N, int K, int R) {
    TfPlan t;
    if (!tf_plan(N, K, R, 1, t)) return 0;
    return (size_t)t.nct * t.nkb * 2 * t.b_plane;
}

extern "C" int plsb200_boot_coef_pack_tf32(const double* E, int N, int K, const int32_t* idx, int R, void* coef,
                                           void* stream) {
    PLSB_CHECK_ARG(E && idx && coef, "boot_coef_pack_tf32: null pointer");
    TfPlan t;
    if (!tf_plan(N, K, R, 1, t)) {
        set_err("boot_coef_pack_tf32: unsupported shape N=%d K=%d R=%d (need 1 <= K <= 24)", N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t fixed = (size_t)2 * CP_KB * K * TF_KB * sizeof(float) + (size_t)((4 * N + 2) & ~1) * sizeof(int);
    const int stage_e = (size_t)N * K * sizeof(double) + fixed <= 96 * 1024;
    const size_t smem = fixed + (stage_e ? (size_t)N * K * sizeof(double) : 0);
    PLSB_CHECK_ARG(smem <= 200 * 1024, "boot_coef_pack_tf32: N=%d too large", N);
    PLSB_CUDA(cudaMemsetAsync(coef, 0, (size_t)t.nct * t.nkb * 2 * t.b_plane, st));
    PLSB_CUDA(cudaFuncSetAttribute(coef_pack_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    coef_pack_tf32_kernel<<<R, CP_ROWS, smem, st>>>(E, N, K, idx, t.Kp, t.nres, t.ntile, t.nkb, stage_e, (float*)coef);
    PLSB_LAUNCH_CHECK("coef_pack_tf32_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_boot_moments_tf32_workspace(int N, int64_t p, int K, int R) {
    TfPlan t;
    if (!tf_plan(N, K, R, p, t)) return 0;
    return t.nsplit > 1 ? (size_t)2 * t.nsplit * p * K * sizeof(double) : 16;
}

extern "C" int plsb200_boot_moments_tf32(const void* ximage, int N, int64_t p, const void* coef, int K, int R,
                                         const double* pivot, double* sum, double* sumsq, void* workspace,
                                         size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(ximage && coef && sum && sumsq, "boot_moments_tf32: null pointer");
    PLSB_CHECK_ARG(p > 0, "boot_moments_tf32: bad shape p=%lld", (long long)p);
    TfPlan t;
    if (!tf_plan(N, K, R, p, t)) {
        set_err("boot_moments_tf32: unsupported shape N=%d K=%d R=%d (need 1 <= K <= 24)", N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double *o1 = sum, *o2 = sumsq;
    if (t.nsplit > 1) {
        const size_t need = (size_t)2 * t.nsplit * p * K * sizeof(double);
        if (!workspace || workspace_bytes < need) {
            set_err("boot_moments_tf32: workspace %zu < %zu bytes", workspace_bytes, need);
            return PLSB200_EWORKSPACE;
        }
        o1 = (double*)workspace;
        o2 = o1 + (size_t)t.nsplit * p * K;
    }
    TfArgs a;
    a.aimg = (const float*)ximage; a.bimg = (const float*)coef; a.pivot = pivot; a.out1 = o1; a.out2 = o2;
    a.p = p; a.nvt = t.nvt; a.nunits = t.nvt * t.nsplit;
    a.K = K; a.R = R; a.nkb = t.nkb; a.nks_last = t.nks_last; a.ntile = t.ntile; a.nres = t.nres; a.nct = t.nct;
    a.ct_per_split = t.ct_per_split; a.nstage = t.nstage; a.b_plane = t.b_plane; a.stage_bytes = t.stage_bytes;
    a.trace = nullptr;
    a.dbg = 0;
#ifdef PLSB_PROBES
    a.dbg = getenv("PLSB200_TF32_DEBUG") ? atoi(getenv("PLSB200_TF32_DEBUG")) : 0;
#endif
    int rc;
    switch (t.Kp) {
#define PLSB_TF(kp) case kp: rc = launch_tf32<kp>(t, a, st); break;
        PLSB_TF(2) PLSB_TF(3) PLSB_TF(4) PLSB_TF(5) PLSB_TF(6) PLSB_TF(8) PLSB_TF(10) PLSB_TF(12) PLSB_TF(15)
        PLSB_TF(16) PLSB_TF(20) PLSB_TF(24)
#undef PLSB_TF
        default:
            set_err("boot_moments_tf32: no kernel for Kp=%d", t.Kp);
            return PLSB200_EUNSUPPORTED;
    }
    if (rc != PLSB200_OK) return rc;
    if (t.nsplit > 1) {
        const long long n = (long long)p * K;
        split_sum_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(o1, o2, t.nsplit, n, sum, sumsq);
        PLSB_LAUNCH_CHECK("split_sum_kernel");
    }
    return PLSB200_OK;
}
