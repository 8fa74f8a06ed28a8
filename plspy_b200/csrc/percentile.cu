// Percentile intervals over the resample axis of a bootstrap distribution (SURVEY section 8f rank 4).
//
// The reference's `resample.confidence_interval` (plspy/core/resample.py:171-222; its call sites on Tdistrib /
// left_sv_sampled are commented out at bootstrap_permutation.py:713-731) sorts every element's B samples in a Python
// loop and interpolates with MATLAB's `prctile` convention: sorted sample k sits at 100 (k + 0.5) / B per cent,
// linear interpolation in between, clamped to the extremes.  Here one CTA sorts one element's series in shared
// memory (bitonic network, padded with +inf to a power of two) and interpolates both bounds; the series are read
// in place through two strides, so a (B x m x n) stack -- or a voxel chunk of the explicit salience cube, which is
// how the p-sized distribution is streamed without ever holding B x p x K -- needs no transpose.
//
// Sorting network: log2(L)(log2(L)+1)/2 compare-exchange levels (91 at L = 8192).  Up to three consecutive levels of a
// merge (partner distances 4d, 2d, d) are done in registers: a thread loads the 8 elements base + {0..7} d, runs the 12
// compare-exchanges and stores them back, so the series crosses shared memory 35 times instead of 91 (the first
// version, one level per pass, ran at 99.7 % of the shared-memory pipe with 32 % bank-conflict wavefronts:
// profiles/ncu_percentile_r02.md).  One padding slot per 16 elements makes every stride conflict-free.  Warp w owns a
// contiguous span of L/8 elements, so passes whose groups fit inside a span only need a warp barrier.  Series longer
// than 16384 samples are sorted in a global-memory scratch line per CTA with the same code.
#include "common.cuh"
#include <math_constants.h>

namespace plsb {

constexpr int PC_THREADS = 256;
constexpr int PC_MAX_SMEM_L = 16384;          // 136 KB of shared memory with the padding

__device__ __forceinline__ int pc_phys(int i) { return i + (i >> 4); }       // one padding slot per 16 elements
__host__ __device__ inline size_t pc_slots(int L) { return (size_t)L + (L >> 4); }

// M consecutive levels (partner distances 2^(a+M-1) ... 2^a) of the merge of size k, on 2^M elements per group in registers
template <int M>
__device__ __forceinline__ void pc_pass(double* a_, int L, int a, int k, int warp, int lane) {
    constexpr int E = 1 << M;
    const int per_warp = (L >> M) / (PC_THREADS / 32);                 // groups per warp
    const int lowmask = (1 << a) - 1;
    for (int q = lane; q < per_warp; q += 32) {
        const int g = warp * per_warp + q;
        const int base = ((g & ~lowmask) << M) | (g & lowmask);        // M zero bits inserted at position a
        const bool asc = (base & k) == 0;
        double x[E];
#pragma unroll
        for (int e = 0; e < E; ++e) x[e] = a_[pc_phys(base + (e << a))];
#pragma unroll
        for (int lev = M - 1; lev >= 0; --lev) {
#pragma unroll
            for (int e = 0; e < E; ++e) {
                if ((e & (1 << lev)) == 0) {
                    const double lo = x[e], hi = x[e | (1 << lev)];
                    const bool sw = (lo > hi) == asc;
                    x[e] = sw ? hi : lo;
                    x[e | (1 << lev)] = sw ? lo : hi;
                }
            }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) a_[pc_phys(base + (e << a))] = x[e];
    }
}

// The three intervals one kernel takes: the plain percentile interval, the bias-corrected one and the bias-corrected and
// accelerated one.
enum PcMode { PC_PLAIN, PC_BC, PC_BCA };

// Bias-corrected bounds (BC): with prop = #{s <= theta} / B (theta = orig[s], the original value) and z0 = Phi^-1(prop),
// the levels are Phi(2 z0 + Phi^-1(q)) instead of q.  prop is counted by binary search over the first B sorted slots
// (the +inf padding never counts); prop 0 or 1 (z0 infinite) and a NaN theta give NaN bounds.
// Bias-corrected and accelerated bounds (BCa, Efron 1987): with the acceleration a = accel[s] and w = z0 + Phi^-1(q),
// the levels are Phi(z0 + w / (1 - a w)); the bound is NaN where 1 - a w <= 0 (or a is NaN).  q = 0 / 1 keep the
// minimum / maximum, as in BC.  a = 0 gives the BC levels.
template <bool GLOBAL, PcMode MODE>
__global__ void __launch_bounds__(PC_THREADS) percentile_kernel(const double* __restrict__ S, int B, long long nseries,
                                                               long long stride_sample, long long stride_series,
                                                               double q_lo, double q_hi, int L,
                                                               double* __restrict__ lower, double* __restrict__ upper,
                                                               double* __restrict__ scratch,
                                                               const double* __restrict__ orig, double* __restrict__ prop,
                                                               const double* __restrict__ accel) {
    constexpr bool BC = MODE != PC_PLAIN;
    extern __shared__ __align__(16) double pc_sm[];
    double* a = GLOBAL ? scratch + (size_t)blockIdx.x * pc_slots(L) : pc_sm;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int span = L / (PC_THREADS / 32);                 // elements owned by a warp (L >= 512: span >= 64)
    int logL = 0;
    while ((1 << logL) < L) ++logL;
    const double zq = BC && tid < 2 ? normcdfinv(tid == 0 ? q_lo : q_hi) : 0.0;   // -inf / +inf at q = 0 / 1
    for (long long s = blockIdx.x; s < nseries; s += gridDim.x) {
        const double* src = S + s * stride_series;
        for (int r = tid; r < L; r += PC_THREADS) a[pc_phys(r)] = r < B ? src[(long long)r * stride_sample] : CUDART_INF;
        bool prev_local = false;
        for (int sk = 1; sk <= logL; ++sk) {               // merge size k = 2^sk: levels 2^(sk-1) ... 1
            const int k = 1 << sk;
            int rem = sk;
            while (rem > 0) {
                const int M = rem % 3 == 0 ? 3 : rem % 3;
                const int lowest = rem - M;                 // log2 of the smallest partner distance of this pass
                const bool local = (1 << (lowest + M)) <= span;
                if (local && prev_local) __syncwarp(); else __syncthreads();
                prev_local = local;
                if (M == 3) pc_pass<3>(a, L, lowest, k, warp, lane);
                else if (M == 2) pc_pass<2>(a, L, lowest, k, warp, lane);
                else pc_pass<1>(a, L, lowest, k, warp, lane);
                rem -= M;
            }
        }
        __syncthreads();
        if (tid < 2) {
            double q = tid == 0 ? q_lo : q_hi;
            bool defined = true;
            if (BC) {                                       // both threads count (same addresses: broadcast reads)
                const double theta = orig[s];
                int lo = 0, hi = B;                         // first sorted slot > theta
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (a[pc_phys(mid)] <= theta) lo = mid + 1; else hi = mid;
                }
                const double pr = isnan(theta) ? CUDART_NAN : (double)lo / B;
                if (tid == 0) prop[s] = pr;
                defined = pr > 0.0 && pr < 1.0;             // false for NaN too
                if (MODE == PC_BCA) {
                    if (defined && q > 0.0 && q < 1.0) {
                        const double z0 = normcdfinv(pr), ac = accel[s], w = z0 + zq, den = 1.0 - ac * w;
                        defined = den > 0.0;                // false for a NaN acceleration too
                        q = normcdf(ac == 0.0 ? 2.0 * z0 + zq : z0 + w / den);   // a = 0: the BC level, bit for bit
                    }
                } else if (defined) {
                    q = normcdf(2.0 * normcdfinv(pr) + zq);
                }
            }
            double t = q * B - 0.5;                         // fractional index into the sorted samples
            t = fmin(fmax(t, 0.0), (double)(B - 1));
            const int lo = (int)floor(t), hi = min(lo + 1, B - 1);
            const double w = t - lo;
            const double v = a[pc_phys(lo)] * (1.0 - w) + a[pc_phys(hi)] * w;
            (tid == 0 ? lower : upper)[s] = defined ? v : CUDART_NAN;
        }
        __syncthreads();
    }
}

static int pc_padded(int B) {
    int L = 512;
    while (L < B) L <<= 1;
    return L;
}

}  // namespace plsb

using namespace plsb;

extern "C" size_t plsb200_percentile_f64_workspace(int B) {
    if (B < 1) return 0;
    const int L = pc_padded(B);
    return L > PC_MAX_SMEM_L ? (size_t)2 * num_sms() * pc_slots(L) * sizeof(double) : 16;
}

// one launcher for the three entry points: the plain interval (orig / prop / accel unused), the bias-corrected one
// (accel unused) and the bias-corrected and accelerated one
template <PcMode MODE>
static int pc_launch(const char* what, const double* samples, int B, int64_t nseries, int64_t stride_sample,
                     int64_t stride_series, const double* orig, const double* accel, double q_lo, double q_hi,
                     double* lower, double* upper, double* prop, void* workspace, size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(samples && lower && upper && (MODE == PC_PLAIN || (orig && prop)) && (MODE != PC_BCA || accel),
                   "%s: null pointer", what);
    PLSB_CHECK_ARG(B >= 1 && B <= (1 << 24) && nseries >= 1, "%s: bad shape B=%d nseries=%lld", what, B,
                   (long long)nseries);
    PLSB_CHECK_ARG(q_lo >= 0.0 && q_lo <= 1.0 && q_hi >= 0.0 && q_hi <= 1.0, "%s: quantiles must lie in [0, 1]", what);
    const int L = pc_padded(B);
    cudaStream_t st = (cudaStream_t)stream;
    if (L <= PC_MAX_SMEM_L) {
        const size_t smem = pc_slots(L) * sizeof(double);
        PLSB_CUDA(cudaFuncSetAttribute(percentile_kernel<false, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
        const int per_sm = (int)((220 * 1024) / smem) < 8 ? (int)((220 * 1024) / smem) : 8;
        const long long cap = (long long)num_sms() * per_sm * 4;
        const unsigned grid = (unsigned)(nseries < cap ? nseries : cap);
        percentile_kernel<false, MODE><<<grid, PC_THREADS, smem, st>>>(samples, B, nseries, stride_sample,
                                                                      stride_series, q_lo, q_hi, L, lower, upper,
                                                                      nullptr, orig, prop, accel);
    } else {
        const size_t need = (size_t)2 * num_sms() * pc_slots(L) * sizeof(double);
        if (!workspace || workspace_bytes < need) {
            set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
            return PLSB200_EWORKSPACE;
        }
        const long long cap = 2LL * num_sms();
        const unsigned grid = (unsigned)(nseries < cap ? nseries : cap);
        percentile_kernel<true, MODE><<<grid, PC_THREADS, 0, st>>>(samples, B, nseries, stride_sample, stride_series,
                                                                  q_lo, q_hi, L, lower, upper, (double*)workspace, orig,
                                                                  prop, accel);
    }
    PLSB_LAUNCH_CHECK("percentile_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_percentile_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                                      int64_t stride_series, double q_lo, double q_hi, double* lower, double* upper,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    return pc_launch<PC_PLAIN>("percentile_f64", samples, B, nseries, stride_sample, stride_series, nullptr, nullptr,
                               q_lo, q_hi, lower, upper, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int plsb200_percentile_bc_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                                         int64_t stride_series, const double* orig, double q_lo, double q_hi,
                                         double* lower, double* upper, double* prop, void* workspace,
                                         size_t workspace_bytes, void* stream) {
    return pc_launch<PC_BC>("percentile_bc_f64", samples, B, nseries, stride_sample, stride_series, orig, nullptr, q_lo,
                            q_hi, lower, upper, prop, workspace, workspace_bytes, stream);
}

extern "C" int plsb200_percentile_bca_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                                          int64_t stride_series, const double* orig, const double* accel, double q_lo,
                                          double q_hi, double* lower, double* upper, double* prop, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    return pc_launch<PC_BCA>("percentile_bca_f64", samples, B, nseries, stride_sample, stride_series, orig, accel, q_lo,
                             q_hi, lower, upper, prop, workspace, workspace_bytes, stream);
}
