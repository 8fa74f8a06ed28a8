// The register-resident FP64 bootstrap GEMM and what it shares with its users: the launch plan, the packed coefficient
// layout, the instantiation ladder and the pipeline body of the three kernels that stream packed coefficients through
// one shared-memory ring -- boot_moments_kernel and nspace_dmma_kernel (boot.cu) and boot_quad_kernel (boot_quad.cu).
// ring_pipeline owns the ring of bulk copies, the mbarriers, the A fragments in registers, the warp stagger and the
// DMMA stream; each kernel supplies an epilogue that says what to do with the D fragments of a period.
#pragma once
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace plsb {

constexpr int BM_WARPS = 8;          // consumer warps per CTA
constexpr int BM_THREADS = BM_WARPS * 32;
constexpr int BM_VOX = BM_WARPS * 8; // voxels per CTA

// Packed coefficients: period `per` (8*nblk columns) is the block of nks*nblk*32 doubles at per*nks*nblk*32, and in it
// the B fragment of k-step s and 8-column block c/8 is 32 consecutive doubles in lane order, lane = 4*(c%8) + q for
// row 4*s + q and column c.  Every pack writes this layout and the GEMMs read it.
__host__ __device__ __forceinline__ int bfrag_offset(int s, int c, int q, int nblk) {
    return (s * nblk + (c >> 3)) * 32 + 4 * (c & 7) + q;
}

// Column padding: the smallest padded K that divides a 24-, 16- or 8-column period (nblk = 3, 2, 1 blocks of 8), the
// wider period on a tie (more independent accumulator chains).  False when no period fits (K > 24).
__host__ __device__ inline bool pad_period(int K, int& Kp, int& nblk) {
    int best_kp = 0, best_blk = 0;
    for (int blk = 3; blk >= 1; --blk) {
        const int cols = 8 * blk;
        for (int kp = K; kp <= cols; ++kp) {
            if (cols % kp == 0) {
                if (best_kp == 0 || kp < best_kp) { best_kp = kp; best_blk = blk; }
                break;
            }
        }
    }
    Kp = best_kp; nblk = best_blk;
    return best_kp != 0;
}

struct BootPlan {
    int Kp;        // padded K (divides 8*nblk)
    int nblk;      // 8-column blocks per period
    int nb;        // resamples per period
    int nks;       // k-steps of 4 rows (multiple of 4)
    int maxks;     // template bucket
    int nper;      // periods
    int nstage;
    size_t stage_doubles;
    size_t smem_bytes;
    int nsplit;        // splits of the period range (grid.y)
    int per_per_split;
};

inline bool boot_plan(int N, int K, int R, int64_t p, BootPlan& b) {
    if (K < 1 || K > 24 || N < 1 || R < 1) return false;
    if (!pad_period(K, b.Kp, b.nblk)) return false;
    b.nb = 8 * b.nblk / b.Kp;
    b.nks = (int)cdiv(N, 16) * 4;
    if (b.nks > 80) return false;
    b.maxks = b.nks;
    b.nper = (int)cdiv(R, b.nb);
    b.stage_doubles = (size_t)b.nks * b.nblk * 32;
    const size_t red = (size_t)BM_WARPS * 8 * b.Kp * 2 * sizeof(double);
    const size_t avail = 227 * 1024 - red - 256;
    int ns = (int)(avail / (b.stage_doubles * sizeof(double)));
    if (ns > 4) ns = 4;
    if (ns < 2) return false;
    b.nstage = ns;
    b.smem_bytes = ns * b.stage_doubles * sizeof(double) + red + 256;
    // split the resample range so that tiles*nsplit fills whole waves of SMs
    const int64_t tiles = cdiv(p > 0 ? p : 1, BM_VOX);
    const int nsm = num_sms();
    int best = 1; double best_cost = 1e30;
    for (int n = 1; n <= 8; ++n) {
        if (n > 1 && b.nper / n < 8) break;
        const double waves = (double)tiles * n / nsm;
        const double cost = ceil(waves) / waves + 0.004 * (n - 1);
        if (cost < best_cost - 1e-12) { best_cost = cost; best = n; }
    }
    b.nsplit = best;
    b.per_per_split = (int)cdiv(b.nper, best);
    b.nsplit = (int)cdiv(b.nper, b.per_per_split);
    return true;
}

// Calls f(std::integral_constant<int, NKS>, std::integral_constant<int, NBLK>) for the plan's k-steps and period
// width: NKS is a compile-time constant so that a period is one straight-line stream of NKS*NBLK {LDS.64, DMMA} pairs
// that ptxas can software-pipeline, and the kernels are instantiated for every multiple of 4 up to 80 (N <= 320).
template <int NBLK, typename F>
static int ring_dispatch_nks(const BootPlan& b, const char* what, F&& f) {
    using std::integral_constant;
    switch (b.nks) {
#define PLSB_CASE(n) case n: return f(integral_constant<int, n>(), integral_constant<int, NBLK>());
        PLSB_CASE(4) PLSB_CASE(8) PLSB_CASE(12) PLSB_CASE(16) PLSB_CASE(20) PLSB_CASE(24) PLSB_CASE(28)
        PLSB_CASE(32) PLSB_CASE(36) PLSB_CASE(40) PLSB_CASE(44) PLSB_CASE(48) PLSB_CASE(52) PLSB_CASE(56)
        PLSB_CASE(60) PLSB_CASE(64) PLSB_CASE(68) PLSB_CASE(72) PLSB_CASE(76) PLSB_CASE(80)
#undef PLSB_CASE
        default:
            set_err("%s: no kernel for nks=%d", what, b.nks);
            return PLSB200_EUNSUPPORTED;
    }
}
template <typename F>
static int ring_dispatch(const BootPlan& b, const char* what, F&& f) {
    switch (b.nblk) {
        case 1: return ring_dispatch_nks<1>(b, what, f);
        case 2: return ring_dispatch_nks<2>(b, what, f);
        default: return ring_dispatch_nks<3>(b, what, f);
    }
}

#ifdef __CUDACC__

// A thread of the pipeline: its D-fragment position (row vr, columns 2q and 2q + 1 of every 8-column block) and the
// periods [per0, per0 + nit) of its CTA's split of the period range (grid.y).  tid is threadIdx.x as read in the
// kernel, where the compiler knows its range from the launch bound.
struct RingThread {
    int tid, warp, lane, q, vr, per0, nit;
    __device__ __forceinline__ RingThread(int tid_, int nper, int per_per_split)
        : tid(tid_), warp(tid >> 5), lane(tid & 31), q(lane & 3), vr(lane >> 2),
          per0(blockIdx.y * per_per_split), nit(min(nper, per0 + per_per_split) - per0) {}
};

// The epilogue hooks that do nothing; an epilogue derives from this, defines fold() and overrides what it needs:
//   d0(j, e)          the value the accumulator chains start from
//   before_wait(it)   work issued before the wait for period per0 + it (loads whose latency the wait hides)
//   read_stage(st)    reads of the period's stage in shared memory, before it is released to the producer
//   fold(d, it)       takes the period's D fragments, after the release
//   finish(red)       the final output; red: the space the kernel reserved between the ring and the barriers
struct RingEpilogue {
    __device__ __forceinline__ double d0(int, int) const { return 0.0; }
    __device__ __forceinline__ void before_wait(int) {}
    __device__ __forceinline__ void read_stage(const double*) {}
    __device__ __forceinline__ void finish(double*) {}
};

// The pipeline body.  Every warp holds the A fragments of its 8 columns of A (rows 0 .. nrows, column v; zero where
// !vok) in registers for the whole kernel; thread 0 streams the periods through an nstage-deep ring of bulk copies
// (UBLKCP, 16 KB each) with full / empty mbarriers, and each period is one chain of NKS DMMAs per 8-column block.
// Shared memory: [ring: nstage stages][red_doubles][full: nstage][empty: nstage].  The epilogue is constructed from
// `args` after the A fragments are loaded.
template <int NKS, int NBLK, typename Ep, typename T, typename V>
__device__ __forceinline__ void ring_pipeline(const RingThread& th, const T* __restrict__ A, long long lda, int nrows,
                                              V v, bool vok, const double* __restrict__ coef, int nstage,
                                              int red_doubles, const typename Ep::Args& args) {
    extern __shared__ __align__(128) unsigned char smraw[];
    constexpr int stage_doubles = NKS * NBLK * 32;
    constexpr uint32_t stage_bytes = (uint32_t)stage_doubles * 8u;
    double* ring = reinterpret_cast<double*>(smraw);
    double* red = ring + (size_t)nstage * stage_doubles;
    uint64_t* full = reinterpret_cast<uint64_t*>(red + red_doubles);
    uint64_t* empty = full + nstage;

    if (th.tid == 0) {
        for (int s = 0; s < nstage; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, BM_WARPS); }
        mbar_fence_init();
    }
    __syncthreads();

    auto issue = [&](int it, int slot) {   // thread 0 only: stream period per0+it into `slot`
        mbar_expect_tx(full + slot, stage_bytes);
        const char* src = reinterpret_cast<const char*>(coef + (size_t)(th.per0 + it) * stage_doubles);
        char* dst = reinterpret_cast<char*>(ring + (size_t)slot * stage_doubles);
#pragma unroll 1
        for (uint32_t off = 0; off < stage_bytes; off += 16384u) {
            const uint32_t n = min(16384u, stage_bytes - off);
            bulk_g2s(dst + off, src + off, n, full + slot);
        }
    };
    if (th.tid == 0)
        for (int it = 0; it < min(nstage, th.nit); ++it) issue(it, it);

    // ---- A fragments: this warp's 8 columns x all rows, resident in registers
    double a[NKS];
#pragma unroll
    for (int s = 0; s < NKS; ++s) {
        const int row = 4 * s + th.q;
        a[s] = (row < nrows && vok) ? (double)__ldg(A + (long long)row * lda + v) : 0.0;
    }
    Ep ep(args, th);

    // The two warps that share an SM sub-partition (w and w+4) run half a period apart, so that one of
    // them always has a full MMA stream in flight while the other folds its accumulators and waits on
    // the next stage (otherwise all eight warps drain the DMMA pipe at the same instant).
    if (th.warp >= 4) __nanosleep((unsigned)(NKS * NBLK * 8));

    int slot = 0, prev_slot = 0;
    uint32_t phase = 0, prev_phase = 0;
    for (int it = 0; it < th.nit; ++it) {
        if (th.tid == 0 && it > 0) {
            // refill the slot drained in the previous iteration with period it-1+nstage
            const int nx = it - 1 + nstage;
            if (nx < th.nit) {
                mbar_wait(empty + prev_slot, prev_phase);
                issue(nx, prev_slot);
            }
        }
        ep.before_wait(it);
        __syncwarp();
        mbar_wait(full + slot, phase);

        double d[NBLK][2];
#pragma unroll
        for (int j = 0; j < NBLK; ++j) { d[j][0] = ep.d0(j, 0); d[j][1] = ep.d0(j, 1); }
        // volatile: ptxas must keep these loads in program order (s-major, chains round-robin), which
        // keeps the NBLK accumulator chains interleaved; without it the straight-line stream is
        // re-ordered chain by chain (fewest live registers) and every DMMA waits on its predecessor.
        const volatile double* bs = ring + (size_t)slot * stage_doubles + th.lane;
#pragma unroll
        for (int s = 0; s < NKS; ++s) {
#pragma unroll
            for (int j = 0; j < NBLK; ++j) {
                const double b = bs[(s * NBLK + j) * 32];
                dmma884(d[j][0], d[j][1], a[s], b);
            }
        }
        ep.read_stage(ring + (size_t)slot * stage_doubles);
        __syncwarp();
        if (th.lane == 0) mbar_arrive(empty + slot);

        ep.fold(d, it);
        prev_slot = slot; prev_phase = phase;
        if (++slot == nstage) { slot = 0; phase ^= 1u; }
    }
    ep.finish(red);
}

// Folds the per-thread accumulators of NO outputs -- nb resample slots per period, slot = column / Kp -- onto k in slot
// order (deterministic) and writes the warp's 8 voxels x K of each output to out[o] + blockIdx.y * p * K, the partial
// of this CTA's split.  red: BM_WARPS * NO * 8 * Kp doubles.
template <int NO, int NBLK>
__device__ __forceinline__ void fold_slots_store(const double (&acc)[NO][NBLK][2], double* red, const RingThread& th,
                                                 int nb, int Kp, int K, long long p, double* const (&out)[NO]) {
    double* r = red + th.warp * (NO * 8 * Kp);
    for (int i = th.lane; i < NO * 8 * Kp; i += 32) r[i] = 0.0;
    __syncwarp();
    for (int round = 0; round < nb; ++round) {
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 8 * j + 2 * th.q + e;
                if (c / Kp == round) {
#pragma unroll
                    for (int o = 0; o < NO; ++o) r[o * 8 * Kp + th.vr * Kp + c % Kp] += acc[o][j][e];
                }
            }
        __syncwarp();
    }
    const long long vbase = (long long)blockIdx.x * BM_VOX + th.warp * 8;
    double* os[NO];
#pragma unroll
    for (int o = 0; o < NO; ++o) os[o] = out[o] + (size_t)blockIdx.y * p * K;
    for (int i = th.lane; i < 8 * K; i += 32) {
        const int rr = i / K, k = i % K;
        if (vbase + rr < p) {
#pragma unroll
            for (int o = 0; o < NO; ++o) os[o][(vbase + rr) * K + k] = r[o * 8 * Kp + rr * Kp + k];
        }
    }
}

#endif  // __CUDACC__

}  // namespace plsb
