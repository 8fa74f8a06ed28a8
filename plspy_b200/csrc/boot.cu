// K4: bootstrap salience moments -- the dominant kernel of the path (>99% of the algorithmic flops).
//
// Reference (bootstrap_permutation.py:557-626, 695): per bootstrap, gather N rows of X, rebuild the
// K x p cross-block matrix, VS_hat = permuted.T @ U (p x K) is stored in right_sv_sampled[B, p, K] and
// std_errs = np.std(right_sv_sampled, axis=0) at the end.  Here VS_r = X^T . C_r with
// C_r = scatter(E, idx_r) (N x K), so all resamples form ONE skinny GEMM
//       VS[v, (r,k)] = sum_i X[i, v] . C[i, (r,k)]          M = p, N = R*K, K-dim = N rows
// whose output is reduced over r on the fly: sum_r (VS - pivot), sum_r (VS - pivot)^2.
//
// Mapping onto the FP64 tensor path (DMMA.8x8x4, 37 TFLOP/s measured on B200):
//   * M (8 per MMA) = voxels.  A warp owns 8 voxels and keeps ALL its A-fragments -- X[0..N, v0..v0+8) --
//     in registers for the whole kernel (N/4 doubles per thread: 75 for N = 300).  X is read from HBM
//     exactly once per CTA row-tile and never staged in shared memory.
//   * N (8 per MMA) = flattened (resample, k) columns.  The coefficient tensor is pre-packed in the
//     exact B-fragment order (lane-major 256-byte blocks), so the TMA engine streams it into shared
//     memory with plain 1-D bulk copies (cp.async.bulk / UBLKCP, mbarrier completion) and every
//     fragment load is one conflict-free LDS.64.  It is shared by the 8 warps of the CTA.
//   * A "period" is 8*NBLK columns = nb whole resamples (K=12 -> 24 columns = 2 resamples, no padding).
//     Within a period the NBLK accumulator chains are independent, which hides the DMMA latency.
//   * After N/4 chained MMAs a D fragment holds VS - pivot (the chain starts from -pivot) for 8 voxels
//     x 8 columns; it is folded into per-thread running sums and discarded.  Column -> k is fixed per
//     thread for the whole kernel because the period is a multiple of K.
// Shared memory: nstage x (N/4 * NBLK * 256 B) ring (57.6 KB per stage at N=300, K=12 -> 3 stages).
// The ring, the A fragments and the DMMA stream are ring_pipeline (boot_plan.cuh), shared with nspace_dmma_kernel below
// and boot_quad_kernel (boot_quad.cu); boot_moments_kernel adds MomentsEpilogue: the chains start from -pivot, the D
// fragments are folded into running moments with the ragged last period masked, and fold_slots_store writes them.
#include "common.cuh"
#include "boot_plan.cuh"

namespace plsb {

// ------------------------------------------------------------------------------------------------
// coefficient packing: C_r = scatter(E, idx_r) written in B-fragment order (bfrag_offset, boot_plan.cuh): resample r
// is slot r % nb of period r / nb, column c = (r % nb)*Kp + k ; row i -> s = i/4, q = i%4.
// One CTA per PERIOD (nb resamples): thread i scans idx for sources of target row i in index order (deterministic),
// the period's block is assembled in shared memory in fragment order and written out as one contiguous, coalesced
// piece.  (Round 1 wrote every coefficient straight to its fragment position: 8-byte stores at a stride of
// 256 nblk bytes, 25 % sector efficiency -- 0.42 ms for the 146 MB of the bench workload.)
__global__ void __launch_bounds__(256) boot_coef_pack_kernel(const double* __restrict__ E, int N, int K,
                                                            const int32_t* __restrict__ idx, int R, int Kp, int nblk,
                                                            int nb, int nks, double* __restrict__ coef) {
    extern __shared__ __align__(16) double smp[];
    const int stage_doubles = nks * nblk * 32;
    double* blk = smp;                                  // [nks][nblk][32]
    int* ids = reinterpret_cast<int*>(blk + stage_doubles);
    int* start = ids + N; int* cur = start + N + 1; int* list = cur + N;
    const int per = blockIdx.x;
    for (int i = threadIdx.x; i < stage_doubles; i += blockDim.x) blk[i] = 0.0;
    for (int slot = 0; slot < nb; ++slot) {
        const int r = per * nb + slot;
        if (r >= R) break;                              // ragged last period: the remaining slots stay zero
        __syncthreads();                                // previous users of the lists are done (and blk is zeroed)
        build_source_lists(idx + (size_t)r * N, N, ids, start, cur, list);
        const int cbase = slot * Kp;
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            double acc[24];
#pragma unroll
            for (int k = 0; k < 24; ++k) acc[k] = 0.0;
            for (int t = start[i]; t < start[i + 1]; ++t) {
                const int src = list[t];
#pragma unroll
                for (int k = 0; k < 24; ++k)
                    if (k < K) acc[k] += __ldg(E + (size_t)src * K + k);
            }
            const int s = i >> 2, q = i & 3;
#pragma unroll
            for (int k = 0; k < 24; ++k) {
                if (k < K) {
                    blk[bfrag_offset(s, cbase + k, q, nblk)] = acc[k];
                }
            }
        }
    }
    __syncthreads();
    double2* out = reinterpret_cast<double2*>(coef + (size_t)per * stage_doubles);
    const double2* in = reinterpret_cast<const double2*>(blk);
    for (int i = threadIdx.x; i < stage_doubles / 2; i += blockDim.x) out[i] = in[i];
}

// The factored collapsed bootstrap (boot_quad.cu, boot_factor_kernel): pseudo-resample j has the coefficients
// c_j[n,k] = E[n,k] . L[sid[n], j] (L: ns x J, row-major), written in the layout of boot_coef_pack_kernel so that
// boot_moments_kernel runs on them unchanged.  One CTA per period; slots j >= J stay zero.
__global__ void __launch_bounds__(256) boot_factor_pack_kernel(const double* __restrict__ E, int N, int K,
                                                              const double* __restrict__ L, int J,
                                                              const int32_t* __restrict__ sid, int Kp, int nblk,
                                                              int nb, int nks, double* __restrict__ coef) {
    extern __shared__ __align__(16) double smf[];
    const int stage_doubles = nks * nblk * 32;
    const int per = blockIdx.x;
    for (int i = threadIdx.x; i < stage_doubles; i += blockDim.x) smf[i] = 0.0;
    __syncthreads();
    for (int e = threadIdx.x; e < nb * N; e += blockDim.x) {
        const int slot = e / N, i = e % N, j = per * nb + slot;
        if (j >= J) continue;
        const double w = L[(size_t)sid[i] * J + j];
        const int s = i >> 2, q = i & 3;
        for (int k = 0; k < K; ++k) smf[bfrag_offset(s, slot * Kp + k, q, nblk)] = E[(size_t)i * K + k] * w;
    }
    __syncthreads();
    double2* out = reinterpret_cast<double2*>(coef + (size_t)per * stage_doubles);
    const double2* in = reinterpret_cast<const double2*>(smf);
    for (int i = threadIdx.x; i < stage_doubles / 2; i += blockDim.x) out[i] = in[i];
}

// ------------------------------------------------------------------------------------------------
// The moments epilogue: the chains start from -pivot, so a D fragment holds VS - pivot for 8 voxels x 8 columns; it is
// folded into per-thread running sums and sums of squares (s[0], s[1]) and discarded.  Column -> k is fixed per thread
// for the whole kernel because the period is a multiple of K.  The padding slots of a ragged last period are masked.
template <int NBLK>
struct MomentsEpilogue : RingEpilogue {
    struct Args { const double* pivot; long long v, p; int R, Kp, K; double* osum; double* osumsq; };
    const Args a;
    const RingThread th;
    double piv[NBLK][2], s[2][NBLK][2];
    int nb;
    __device__ __forceinline__ MomentsEpilogue(const Args& args, const RingThread& t) : a(args), th(t) {
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 8 * j + 2 * th.q + e, k = c % a.Kp;
                piv[j][e] = (a.pivot != nullptr && k < a.K && a.v < a.p) ? __ldg(a.pivot + a.v * a.K + k) : 0.0;
                s[0][j][e] = 0.0; s[1][j][e] = 0.0;
            }
        nb = 8 * NBLK / a.Kp;
    }
    __device__ __forceinline__ double d0(int j, int e) const { return -piv[j][e]; }
    __device__ __forceinline__ void fold(const double (&d)[NBLK][2], int it) {
        if (it + 1 < th.nit || (th.per0 + it + 1) * nb <= a.R) {      // every slot of the period is a real resample
#pragma unroll
            for (int j = 0; j < NBLK; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    s[0][j][e] += d[j][e];
                    s[1][j][e] = fma(d[j][e], d[j][e], s[1][j][e]);
                }
        } else {                                                      // ragged last period: mask the padding slots
            const int rbase = (th.per0 + it) * nb;
#pragma unroll
            for (int j = 0; j < NBLK; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (rbase + (8 * j + 2 * th.q + e) / a.Kp < a.R) {
                        s[0][j][e] += d[j][e];
                        s[1][j][e] = fma(d[j][e], d[j][e], s[1][j][e]);
                    }
                }
        }
    }
    __device__ __forceinline__ void finish(double* red) {
        fold_slots_store<2, NBLK>(s, red, th, nb, a.Kp, a.K, a.p, {a.osum, a.osumsq});
    }
};

// T: element type of X (float: X stored as float32, widened as the A fragments are loaded -- the same DMMA operands as
// from the widened matrix).
template <typename T, int NKS, int NBLK>
__global__ void __launch_bounds__(BM_THREADS, 1)
boot_moments_kernel(const T* __restrict__ X, long long ldx, int N, long long p,
                    const double* __restrict__ coef, int nper, int per_per_split, int nstage,
                    int R, int Kp, int K, const double* __restrict__ pivot,
                    double* __restrict__ osum, double* __restrict__ osumsq) {
    const RingThread th(threadIdx.x, nper, per_per_split);
    const long long v = (long long)blockIdx.x * BM_VOX + th.warp * 8 + th.vr;
    ring_pipeline<NKS, NBLK, MomentsEpilogue<NBLK>>(th, X, ldx, N, v, v < p, coef, nstage, BM_WARPS * 16 * Kp,
                                                    {pivot, v, p, R, Kp, K, osum, osumsq});
}

// ------------------------------------------------------------------------------------------------
// The N-space pass (K2/K6) on the same machinery: H = G^T [C_1 | C_2 | ...] is the bootstrap GEMM with the Gram
// matrix as the data matrix (rows i, "voxels" j) and the same packed coefficient stream, and
//     d2[r,k] = C_r[:,k]^T H[:,(r,k)],      T[r,c,k] = (Lmat G C_r)[c,k] / sqrt(d2[r,k])
// come out of the epilogue: the data matrix is W = [G | 0 | (Lmat G)^T] (N rows x (Npad + Kt) columns, Npad = N rounded
// up to 8), so a warp's 8 "voxels" are either rows of H -- its D fragment is multiplied element-wise with the
// coefficients of those rows (read from the stage in shared memory), reduced over the 8 rows with shuffles and written
// as one partial per (voxel group, resample, k) -- or rows of T, which are stored as they are.  Partials are summed in
// a fixed order by nspace_finish_kernel (deterministic), which also applies 1/sqrt(d2) to T.  The pipeline is
// ring_pipeline with W as the data matrix; NspaceEpilogue adds the read of the row's own coefficients from the stage
// before it is released, and the shuffle reduction or the store of T.
// Replaces nspace_kernel (FMA, bound by the shared-memory pipe: profiles/ncu_nspace_r02.md) for N <= 320.
struct NsArgs {
    const double* W; long long ldw; int N, Nv, Npad;
    const double* coef; int nper, per_per_split, nstage, R, Kp, K, Kt;
    double* dpart;      // [ngH][R][K]
    double* Traw;       // [R][Kt][K] or NULL
};

// The N-space epilogue.  A warp over rows of H reads, before the stage is released, the coefficients of its thread's
// own row v for the thread's columns; the product with the D element is reduced over the warp's 8 rows and stored as a
// partial of d2.  A warp over rows of T stores its D elements.
template <int NBLK>
struct NspaceEpilogue : RingEpilogue {
    struct Args { const NsArgs& a; int group, v; };
    const Args x;
    const RingThread th;
    const bool is_h;                                         // warp-uniform: rows of H, else rows of T
    const int nb;
    double cv[NBLK][2];
    __device__ __forceinline__ NspaceEpilogue(const Args& args, const RingThread& t)
        : x(args), th(t), is_h(args.group * 8 < args.a.Npad), nb(8 * NBLK / args.a.Kp) {}
    __device__ __forceinline__ void read_stage(const double* stage) {
        if (is_h) {
#pragma unroll
            for (int j = 0; j < NBLK; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    cv[j][e] = x.v < x.a.N ? stage[bfrag_offset(x.v >> 2, 8 * j + 2 * th.q + e, x.v & 3, NBLK)] : 0.0;
        }
    }
    __device__ __forceinline__ void fold(const double (&d)[NBLK][2], int it) {
        const NsArgs& a = x.a;
        const int rbase = (th.per0 + it) * nb;
        if (is_h) {
#pragma unroll
            for (int j = 0; j < NBLK; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    double pr = cv[j][e] * d[j][e];
                    pr += __shfl_xor_sync(0xffffffffu, pr, 4);
                    pr += __shfl_xor_sync(0xffffffffu, pr, 8);
                    pr += __shfl_xor_sync(0xffffffffu, pr, 16);
                    const int c = 8 * j + 2 * th.q + e, r = rbase + c / a.Kp, k = c % a.Kp;
                    if (th.vr == 0 && k < a.K && r < a.R) a.dpart[((size_t)x.group * a.R + r) * a.K + k] = pr;
                }
        } else if (a.Traw != nullptr) {
            const int ci = x.v - a.Npad;
#pragma unroll
            for (int j = 0; j < NBLK; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int c = 8 * j + 2 * th.q + e, r = rbase + c / a.Kp, k = c % a.Kp;
                    if (ci < a.Kt && k < a.K && r < a.R) a.Traw[((size_t)r * a.Kt + ci) * a.K + k] = d[j][e];
                }
        }
    }
};

template <int NKS, int NBLK>
__global__ void __launch_bounds__(BM_THREADS, 1) nspace_dmma_kernel(const NsArgs a) {
    const RingThread th(threadIdx.x, a.nper, a.per_per_split);
    const int group = blockIdx.x * BM_WARPS + th.warp;      // 8 consecutive columns of W
    const int v = group * 8 + th.vr;
    ring_pipeline<NKS, NBLK, NspaceEpilogue<NBLK>>(th, a.W, a.ldw, a.N, v, v < a.Nv, a.coef, a.nstage, 0,
                                                   {a, group, v});
}

// W = [G | 0 | (Lmat G)^T]: N rows, ldw columns
__global__ void nspace_w_kernel(const double* __restrict__ G, int N, const double* __restrict__ Lmat, int Kt, int Npad,
                                long long ldw, double* __restrict__ W) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)N * ldw) return;
    const int row = (int)(i / ldw), col = (int)(i % ldw);
    double val = 0.0;
    if (col < N) val = G[(size_t)row * N + col];
    else if (col >= Npad && col - Npad < Kt) {
        const double* l = Lmat + (size_t)(col - Npad) * N;
        for (int t = 0; t < N; ++t) val = fma(l[t], G[(size_t)t * N + row], val);
    }
    W[i] = val;
}

// d2[r,k] = sum over the voxel groups (fixed order); T[r,c,k] *= 1/sqrt(d2[r,k])
__global__ void nspace_finish_kernel(const double* __restrict__ dpart, int ngroups, int R, int K, int Kt,
                                     double* __restrict__ d2, double* __restrict__ T) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)R * K) return;
    double s = 0.0;
    for (int g = 0; g < ngroups; ++g) s += dpart[(size_t)g * R * K + i];
    d2[i] = s;
    if (T != nullptr) {
        const double dn = s > 0.0 ? 1.0 / sqrt(s) : 0.0;
        const int r = (int)(i / K), k = (int)(i % K);
        for (int c = 0; c < Kt; ++c) T[((size_t)r * Kt + c) * K + k] *= dn;
    }
}

__global__ void split_sum_kernel(const double* __restrict__ part1, const double* __restrict__ part2, int nsplit,
                                 long long n, double* __restrict__ out1, double* __restrict__ out2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double a = 0.0;
    for (int s = 0; s < nsplit; ++s) a += part1[(size_t)s * n + i];
    out1[i] = a;
    if (out2 == nullptr) return;
    double b = 0.0;
    for (int s = 0; s < nsplit; ++s) b += part2[(size_t)s * n + i];
    out2[i] = b;
}

__global__ void boot_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, long long n,
                                     double R, const double* __restrict__ numer, double* __restrict__ std_errs,
                                     double* __restrict__ ratios) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double m = sum[i] / R;
    double var = sumsq[i] / R - m * m;
    if (var < 0.0) var = 0.0;
    const double sd = sqrt(var);
    std_errs[i] = sd;
    if (ratios) ratios[i] = numer[i] / sd;
}

// explicit saliences VS[r][v][k] = sum_i X[idx_r[i], v] . E[i, k]  (reference order of operations;
// small problems / debugging only -- writes R*p*K doubles)
// SERIES: output [v][k][r] (the R samples of an element contiguous: the layout percentile_kernel sorts fastest) with the
// resample as the FAST grid index, so that the CTAs running at one time share their rows of X in L2 and write
// neighbouring 8-byte slots of the same sectors.
// COEF: explicit per-sample coefficients instead of a gather, VS[r][v][k] = sum_i X[i, v] . E[r][i][k] (E: R x N x K,
// idx unused) -- the leave-one-subject-out jackknife of the saliences, whose coefficients are zero on the removed rows.
template <typename T, int KT, bool SERIES, bool COEF = false>
__global__ void __launch_bounds__(128) salience_kernel(const T* __restrict__ X, int N, long long p, long long ldx,
                                                      const double* __restrict__ E, int K,
                                                      const int32_t* __restrict__ idx, int R, double* __restrict__ VS) {
    extern __shared__ __align__(16) double sms[];
    double* Es = sms;
    int* ids = reinterpret_cast<int*>(Es + (size_t)N * K);
    const int r = SERIES ? blockIdx.x : blockIdx.y;
    const double* Er = COEF ? E + (size_t)r * N * K : E;
    for (int i = threadIdx.x; i < N * K; i += blockDim.x) Es[i] = Er[i];
    if (!COEF)
        for (int i = threadIdx.x; i < N; i += blockDim.x) ids[i] = idx[(size_t)r * N + i];
    __syncthreads();
    const long long v = (long long)(SERIES ? blockIdx.y : blockIdx.x) * blockDim.x + threadIdx.x;
    if (v >= p) return;
    for (int k0 = 0; k0 < K; k0 += KT) {
        double acc[KT];
#pragma unroll
        for (int t = 0; t < KT; ++t) acc[t] = 0.0;
        if (COEF) {
#pragma unroll 2
            for (int i = 0; i < N; ++i) {              // unrolled twice: the compiler's default unroll spills here
                const double x = (double)__ldg(X + (long long)i * ldx + v);
#pragma unroll
                for (int t = 0; t < KT; ++t)
                    if (k0 + t < K) acc[t] = fma(x, Es[i * K + k0 + t], acc[t]);
            }
        } else {
            for (int i = 0; i < N; ++i) {
                const double x = (double)__ldg(X + (long long)ids[i] * ldx + v);
#pragma unroll
                for (int t = 0; t < KT; ++t)
                    if (k0 + t < K) acc[t] = fma(x, Es[i * K + k0 + t], acc[t]);
            }
        }
#pragma unroll
        for (int t = 0; t < KT; ++t)
            if (k0 + t < K) {
                if (SERIES) VS[((size_t)v * K + k0 + t) * R + r] = acc[t];
                else VS[((size_t)r * p + v) * K + k0 + t] = acc[t];
            }
    }
}

// XL = X . V : each CTA takes a chunk of XV_CHUNK voxels; the V chunk is staged transposed in shared memory
// ([k][voxel]: conflict-free), a warp owns XV_RG rows at a time so that every V value fetched from shared
// memory feeds XV_RG FMAs (2: 24 accumulators keep the kernel at three CTAs per SM), lanes stride over the voxels (coalesced 256-B row segments of X), and the per-lane
// partial sums are combined by shuffles in a fixed order (deterministic).  HBM-bound: X is read once.
constexpr int XV_CHUNK = 512;
constexpr int XV_RG = 2;
template <typename T, int KT>
__global__ void __launch_bounds__(256, 3) xv_partial_kernel(const T* __restrict__ X, int N, long long p, long long ldx,
                                                        const double* __restrict__ V, int K,
                                                        double* __restrict__ part) {
    extern __shared__ __align__(16) double smv[];   // [KT][XV_CHUNK]
    const long long v0 = (long long)blockIdx.x * XV_CHUNK;
    const int nv = (int)min((long long)XV_CHUNK, p - v0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int k0 = 0; k0 < K; k0 += KT) {
        const int kn = min(KT, K - k0);
        __syncthreads();
        for (int i = threadIdx.x; i < XV_CHUNK * KT; i += blockDim.x) {
            const int c = i / KT, t = i % KT;
            smv[t * XV_CHUNK + c] = (c < nv && t < kn) ? V[(v0 + c) * K + k0 + t] : 0.0;
        }
        __syncthreads();
        for (int r0 = warp * XV_RG; r0 < N; r0 += nw * XV_RG) {
            double acc[XV_RG][KT];
#pragma unroll
            for (int r = 0; r < XV_RG; ++r)
#pragma unroll
                for (int t = 0; t < KT; ++t) acc[r][t] = 0.0;
            const T* x = X + (long long)r0 * ldx + v0;
#pragma unroll 2
            for (int c = lane; c < nv; c += 32) {
                double xr[XV_RG];
#pragma unroll
                for (int r = 0; r < XV_RG; ++r) xr[r] = (r0 + r < N) ? (double)__ldg(x + (long long)r * ldx + c) : 0.0;
#pragma unroll
                for (int t = 0; t < KT; ++t) {
                    const double vv = smv[t * XV_CHUNK + c];
#pragma unroll
                    for (int r = 0; r < XV_RG; ++r) acc[r][t] = fma(xr[r], vv, acc[r][t]);
                }
            }
#pragma unroll
            for (int r = 0; r < XV_RG; ++r)
#pragma unroll
                for (int t = 0; t < KT; ++t) {
                    double sacc = acc[r][t];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
                    if (lane == 0 && r0 + r < N && t < kn)
                        part[((size_t)blockIdx.x * N + r0 + r) * K + k0 + t] = sacc;
                }
        }
    }
}

__global__ void xv_reduce_kernel(const double* __restrict__ part, int nchunk, int n, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s = 0.0;
    for (int c = 0; c < nchunk; ++c) s += part[(size_t)c * n + i];
    out[i] = s;
}

// The stratified jackknife acceleration of every series: S[s][j] (J samples per series, groups [goff[g], goff[g+1])),
// one thread per series, summed with a pivot at theta[s] (translation leaves a unchanged; the pivot keeps large
// per-voxel baselines from cancelling).  With d_j = S_j - theta, m_g the mean of d over group g and
// l_j = (n_g - 1)(m_g - d_j):  a = (1/6) sum_g n_g^-3 sum l^3 / (sum_g n_g^-2 sum l^2)^(3/2), 0 where the denominator
// is 0.  The J samples of a series are read twice (mean, then moments); the second pass hits L1 / L2.
__global__ void jack_accel_kernel(const double* __restrict__ S, long long nseries, int J, const int32_t* __restrict__ goff,
                                  int G, const double* __restrict__ theta, double* __restrict__ accel) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseries) return;
    const double* row = S + s * J;
    const double th = theta[s];
    double num = 0.0, den = 0.0;
    for (int g = 0; g < G; ++g) {
        const int j0 = goff[g], j1 = goff[g + 1], n = j1 - j0;
        double m = 0.0;
        for (int j = j0; j < j1; ++j) m += row[j] - th;
        m /= n;
        double s2 = 0.0, s3 = 0.0;
        for (int j = j0; j < j1; ++j) {
            const double l = (n - 1) * (m - (row[j] - th));
            s2 = fma(l, l, s2);
            s3 = fma(l * l, l, s3);
        }
        const double inv = 1.0 / n;
        num += s3 * inv * inv * inv;
        den += s2 * inv * inv;
    }
    accel[s] = den > 0.0 ? num / (6.0 * den * sqrt(den)) : (isnan(den) ? den : 0.0);
}

}  // namespace plsb

using namespace plsb;

// N <= 320: the register-resident kernel of this file unless PLSB200_EXACT=os routes every design through boot_os.cu.
// Read once per process: the pack and the GEMM must agree on the coefficient layout.
static bool short_os() {
    static const char* const env = getenv("PLSB200_EXACT");
    return env && env[0] == 'o';
}
// tall designs (N > 320) always take the output-stationary kernel (boot_os.cu)
static bool use_os(int N) { return N > 320 || short_os(); }

extern "C" size_t plsb200_boot_coef_bytes(int N, int K, int R) {
    if (use_os(N)) return boot_os_coef_bytes(N, K, R);
    BootPlan b;
    if (!boot_plan(N, K, R, 1, b)) return 0;
    return (size_t)b.nper * b.stage_doubles * sizeof(double);
}

extern "C" int plsb200_boot_coef_pack_f64(const double* E, int N, int K, const int32_t* idx, int R, double* coef,
                                          void* stream) {
    PLSB_CHECK_ARG(E && idx && coef, "boot_coef_pack_f64: null pointer");
    if (use_os(N)) return boot_os_pack(E, N, K, idx, R, coef, (cudaStream_t)stream);
    BootPlan b;
    if (!boot_plan(N, K, R, 1, b)) {
        set_err("boot_coef_pack_f64: unsupported shape N=%d K=%d R=%d (need K<=24, N<=320)", N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    size_t smem = b.stage_doubles * sizeof(double) + (size_t)(4 * N + 1) * sizeof(int);
    PLSB_CUDA(cudaFuncSetAttribute(boot_coef_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    boot_coef_pack_kernel<<<b.nper, 256, smem, st>>>(E, N, K, idx, R, b.Kp, b.nblk, b.nb, b.nks, coef);
    PLSB_LAUNCH_CHECK("boot_coef_pack_kernel");
    return PLSB200_OK;
}

// the layout boot_moments_f64 reads: the register-resident one, else (N > 320 or PLSB200_EXACT=os) that of the
// output-stationary kernel
extern "C" size_t plsb200_boot_factor_coef_bytes(int N, int K, int J) {
    if (use_os(N)) return boot_os_coef_bytes(N, K, J);
    BootPlan b;
    if (!boot_plan(N, K, J, 1, b)) return 0;
    return (size_t)b.nper * b.stage_doubles * sizeof(double);
}

extern "C" int plsb200_boot_factor_pack_f64(const double* E, int N, int K, const double* L, int J, const int32_t* sid,
                                            double* coef, void* stream) {
    PLSB_CHECK_ARG(E && L && sid && coef, "boot_factor_pack_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && J > 0, "boot_factor_pack_f64: bad shape N=%d J=%d", N, J);
    cudaStream_t st = (cudaStream_t)stream;
    if (use_os(N)) return boot_os_factor_pack(E, N, K, L, J, sid, coef, st);
    BootPlan b;
    if (!boot_plan(N, K, J, 1, b)) {
        set_err("boot_factor_pack_f64: unsupported shape N=%d K=%d J=%d (need K<=24)", N, K, J);
        return PLSB200_EUNSUPPORTED;
    }
    const size_t smem = b.stage_doubles * sizeof(double);
    PLSB_CUDA(cudaFuncSetAttribute(boot_factor_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    boot_factor_pack_kernel<<<b.nper, 256, smem, st>>>(E, N, K, L, J, sid, b.Kp, b.nblk, b.nb, b.nks, coef);
    PLSB_LAUNCH_CHECK("boot_factor_pack_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_boot_moments_f64_workspace(int N, int64_t p, int K, int R) {
    if (use_os(N)) return boot_os_workspace(N, p, K, R);
    BootPlan b;
    if (!boot_plan(N, K, R, p, b)) return 0;
    return b.nsplit > 1 ? (size_t)2 * b.nsplit * p * K * sizeof(double) : 16;
}

template <typename T>
static int boot_moments(const T* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R,
                        const double* pivot, double* sum, double* sumsq, void* workspace, size_t workspace_bytes,
                        void* stream, const char* what) {
    PLSB_CHECK_ARG(X && coef && sum && sumsq, "%s: null pointer", what);
    PLSB_CHECK_ARG(p > 0 && ldx >= p, "%s: bad shape p=%lld ldx=%lld", what, (long long)p, (long long)ldx);
    if (use_os(N))
        return boot_os_moments(X, N, p, ldx, coef, K, R, pivot, sum, sumsq, workspace, workspace_bytes,
                               (cudaStream_t)stream, what);
    BootPlan b;
    if (!boot_plan(N, K, R, p, b)) {
        set_err("%s: unsupported shape N=%d K=%d R=%d (need K<=24, N<=320)", what, N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double *o1 = sum, *o2 = sumsq;
    if (b.nsplit > 1) {
        size_t need = (size_t)2 * b.nsplit * p * K * sizeof(double);
        if (!workspace || workspace_bytes < need) {
            set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
            return PLSB200_EWORKSPACE;
        }
        o1 = (double*)workspace;
        o2 = o1 + (size_t)b.nsplit * p * K;
    }
    const dim3 grid((unsigned)cdiv(p, BM_VOX), (unsigned)b.nsplit);
    const int rc = ring_dispatch(b, "boot_moments_f64", [&](auto nks, auto nblk) {
        const auto kernel = boot_moments_kernel<T, decltype(nks)::value, decltype(nblk)::value>;
        PLSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b.smem_bytes));
        kernel<<<grid, BM_THREADS, b.smem_bytes, st>>>(X, ldx, N, p, coef, b.nper, b.per_per_split, b.nstage, R, b.Kp,
                                                       K, pivot, o1, o2);
        PLSB_LAUNCH_CHECK("boot_moments_kernel");
        return PLSB200_OK;
    });
    if (rc != PLSB200_OK) return rc;
    if (b.nsplit > 1) {
        const long long n = (long long)p * K;
        split_sum_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(o1, o2, b.nsplit, n, sum, sumsq);
        PLSB_LAUNCH_CHECK("split_sum_kernel");
    }
    return PLSB200_OK;
}

extern "C" int plsb200_boot_moments_f64(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R,
                                        const double* pivot, double* sum, double* sumsq, void* workspace,
                                        size_t workspace_bytes, void* stream) {
    return boot_moments(X, N, p, ldx, coef, K, R, pivot, sum, sumsq, workspace, workspace_bytes, stream,
                        "boot_moments_f64");
}

extern "C" int plsb200_boot_moments_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K,
                                            int R, const double* pivot, double* sum, double* sumsq, void* workspace,
                                            size_t workspace_bytes, void* stream) {
    return boot_moments(X, N, p, ldx, coef, K, R, pivot, sum, sumsq, workspace, workspace_bytes, stream,
                        "boot_moments_x32_f64");
}

extern "C" int plsb200_boot_finalize_f64(const double* sum, const double* sumsq, int64_t p, int K, int64_t R_total,
                                         const double* numer, double* std_errs, double* boot_ratios, void* stream) {
    PLSB_CHECK_ARG(sum && sumsq && std_errs, "boot_finalize_f64: null pointer");
    PLSB_CHECK_ARG(p > 0 && K > 0 && R_total > 0, "boot_finalize_f64: bad shape");
    PLSB_CHECK_ARG(boot_ratios == nullptr || numer != nullptr, "boot_finalize_f64: ratios requested without numerator");
    const long long n = (long long)p * K;
    boot_finalize_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(sum, sumsq, n, (double)R_total, numer,
                                                                                  std_errs, boot_ratios);
    PLSB_LAUNCH_CHECK("boot_finalize_kernel");
    return PLSB200_OK;
}

template <typename T>
static int salience_launch(const T* X, int N, int64_t p, int64_t ldx, const double* E, int K, const int32_t* idx, int R,
                           double* VS, bool series, void* stream, const char* what) {
    PLSB_CHECK_ARG(X && E && idx && VS, "%s: null pointer", what);
    PLSB_CHECK_ARG(N > 0 && p > 0 && K > 0 && R >= 0 && ldx >= p, "%s: bad shape", what);
    if (R == 0) return PLSB200_OK;
    size_t smem = (size_t)N * K * sizeof(double) + (size_t)N * sizeof(int);
    if (smem > 200 * 1024) {
        set_err("%s: N*K too large", what);
        return PLSB200_EUNSUPPORTED;
    }
    if (series) {
        PLSB_CHECK_ARG(cdiv(p, 128) <= 65535, "%s: more than 65535 voxel blocks per call", what);
        PLSB_CUDA(cudaFuncSetAttribute(salience_kernel<T, 12, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid((unsigned)R, (unsigned)cdiv(p, 128));
        salience_kernel<T, 12, true><<<grid, 128, smem, (cudaStream_t)stream>>>(X, N, p, ldx, E, K, idx, R, VS);
    } else {
        PLSB_CHECK_ARG(R <= 65535, "%s: more than 65535 resamples per call", what);
        PLSB_CUDA(cudaFuncSetAttribute(salience_kernel<T, 12, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid((unsigned)cdiv(p, 128), (unsigned)R);
        salience_kernel<T, 12, false><<<grid, 128, smem, (cudaStream_t)stream>>>(X, N, p, ldx, E, K, idx, R, VS);
    }
    PLSB_LAUNCH_CHECK("salience_kernel");
    return PLSB200_OK;
}

// the jackknife pass: explicit coefficients C (J x N x K), series-major output VS[v][k][j] of the voxel window [0, p)
template <typename T>
static int salience_coef_series(const T* X, int N, int64_t p, int64_t ldx, const double* C, int K, int J, double* VS,
                                void* stream, const char* what) {
    PLSB_CHECK_ARG(X && C && VS, "%s: null pointer", what);
    PLSB_CHECK_ARG(N > 0 && p > 0 && K > 0 && J >= 0 && ldx >= p, "%s: bad shape", what);
    PLSB_CHECK_ARG(cdiv(p, 128) <= 65535, "%s: more than 65535 voxel blocks per call", what);
    if (J == 0) return PLSB200_OK;
    const size_t smem = (size_t)N * K * sizeof(double);
    if (smem > 200 * 1024) {
        set_err("%s: N*K too large", what);
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaFuncSetAttribute(salience_kernel<T, 12, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
    const dim3 grid((unsigned)J, (unsigned)cdiv(p, 128));
    salience_kernel<T, 12, true, true><<<grid, 128, smem, (cudaStream_t)stream>>>(X, N, p, ldx, C, K, nullptr, J, VS);
    PLSB_LAUNCH_CHECK("salience_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_salience_f64(const double* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                    const int32_t* idx, int R, double* VS, void* stream) {
    return salience_launch(X, N, p, ldx, E, K, idx, R, VS, false, stream, "salience_f64");
}

extern "C" int plsb200_salience_series_f64(const double* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                           const int32_t* idx, int R, double* VS, void* stream) {
    return salience_launch(X, N, p, ldx, E, K, idx, R, VS, true, stream, "salience_series_f64");
}

extern "C" int plsb200_salience_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                        const int32_t* idx, int R, double* VS, void* stream) {
    return salience_launch(X, N, p, ldx, E, K, idx, R, VS, false, stream, "salience_x32_f64");
}

extern "C" int plsb200_salience_series_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                               const int32_t* idx, int R, double* VS, void* stream) {
    return salience_launch(X, N, p, ldx, E, K, idx, R, VS, true, stream, "salience_series_x32_f64");
}

extern "C" int plsb200_salience_coef_series_f64(const double* X, int N, int64_t p, int64_t ldx, const double* C, int K,
                                                int J, double* VS, void* stream) {
    return salience_coef_series(X, N, p, ldx, C, K, J, VS, stream, "salience_coef_series_f64");
}

extern "C" int plsb200_salience_coef_series_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* C,
                                                    int K, int J, double* VS, void* stream) {
    return salience_coef_series(X, N, p, ldx, C, K, J, VS, stream, "salience_coef_series_x32_f64");
}

extern "C" int plsb200_jack_accel_f64(const double* S, int64_t nseries, int J, const int32_t* goff, int G,
                                      const double* theta, double* accel, void* stream) {
    PLSB_CHECK_ARG(S && goff && theta && accel, "jack_accel_f64: null pointer");
    PLSB_CHECK_ARG(nseries >= 1 && J >= 1 && G >= 1 && G <= J, "jack_accel_f64: bad shape nseries=%lld J=%d G=%d",
                   (long long)nseries, J, G);
    jack_accel_kernel<<<(unsigned)cdiv(nseries, 256), 256, 0, (cudaStream_t)stream>>>(S, nseries, J, goff, G, theta,
                                                                                      accel);
    PLSB_LAUNCH_CHECK("jack_accel_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_xv_f64_workspace(int N, int64_t p, int K) {
    if (N <= 0 || p <= 0 || K <= 0) return 0;
    return (size_t)cdiv(p, XV_CHUNK) * N * K * sizeof(double);
}

template <typename T>
static int xv_launch(const T* X, int N, int64_t p, int64_t ldx, const double* V, int K, double* XL, void* workspace,
                     size_t workspace_bytes, void* stream, const char* what) {
    PLSB_CHECK_ARG(X && V && XL && workspace, "%s: null pointer", what);
    PLSB_CHECK_ARG(N > 0 && p > 0 && K > 0 && ldx >= p, "%s: bad shape", what);
    const int nchunk = (int)cdiv(p, XV_CHUNK);
    size_t need = (size_t)nchunk * N * K * sizeof(double);
    if (workspace_bytes < need) {
        set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    size_t smem = (size_t)XV_CHUNK * 12 * sizeof(double);
    cudaStream_t st = (cudaStream_t)stream;
    PLSB_CUDA(cudaFuncSetAttribute(xv_partial_kernel<T, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    xv_partial_kernel<T, 12><<<nchunk, 256, smem, st>>>(X, N, p, ldx, V, K, (double*)workspace);
    PLSB_LAUNCH_CHECK("xv_partial_kernel");
    xv_reduce_kernel<<<(unsigned)cdiv((int64_t)N * K, 256), 256, 0, st>>>((const double*)workspace, nchunk, N * K, XL);
    PLSB_LAUNCH_CHECK("xv_reduce_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_xv_f64(const double* X, int N, int64_t p, int64_t ldx, const double* V, int K, double* XL,
                              void* workspace, size_t workspace_bytes, void* stream) {
    return xv_launch(X, N, p, ldx, V, K, XL, workspace, workspace_bytes, stream, "xv_f64");
}

extern "C" int plsb200_xv_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* V, int K, double* XL,
                                  void* workspace, size_t workspace_bytes, void* stream) {
    return xv_launch(X, N, p, ldx, V, K, XL, workspace, workspace_bytes, stream, "xv_x32_f64");
}

// ---- N-space pass on DMMA (see nspace_dmma_kernel) -----------------------------------------------------------
namespace plsb {
struct NsLayout { int Npad, Nv, ngH; long long ldw; size_t off_w, off_dpart, total; };
static NsLayout ns_layout(int N, int K, int Kt, int R) {
    NsLayout L;
    L.Npad = (N + 7) / 8 * 8;
    L.Nv = L.Npad + Kt;
    L.ldw = (L.Nv + 7) / 8 * 8;
    L.ngH = L.Npad / 8;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    L.off_w = 0;
    L.off_dpart = al((size_t)N * L.ldw * sizeof(double));
    L.total = L.off_dpart + al((size_t)L.ngH * R * K * sizeof(double));
    return L;
}

}  // namespace plsb

extern "C" size_t plsb200_nspace_dmma_f64_workspace(int N, int K, int Kt, int R) {
    BootPlan b;
    if (N > 320 || short_os() || Kt < 0 || !boot_plan(N, K, R, 1, b)) return 0;
    return ns_layout(N, K, Kt, R).total;
}

extern "C" int plsb200_nspace_dmma_f64(const double* G, int N, const double* Lmat, int Kt, const double* coef, int K,
                                       int R, double* d2, double* T, void* workspace, size_t workspace_bytes,
                                       void* stream) {
    PLSB_CHECK_ARG(G && coef && d2 && workspace, "nspace_dmma_f64: null pointer");
    PLSB_CHECK_ARG((T == nullptr && Kt == 0) || (T != nullptr && Lmat != nullptr && Kt > 0),
                   "nspace_dmma_f64: T, Lmat and Kt go together");
    PLSB_CHECK_ARG(N > 0 && K > 0 && R > 0, "nspace_dmma_f64: bad shape");
    BootPlan b;
    if (N > 320 || short_os() || !boot_plan(N, K, R, 1, b)) {
        set_err("nspace_dmma_f64: unsupported shape N=%d K=%d (need N<=320, K<=24): use nspace_f64", N, K);
        return PLSB200_EUNSUPPORTED;
    }
    const NsLayout L = ns_layout(N, K, Kt, R);
    if (workspace_bytes < L.total) {
        set_err("nspace_dmma_f64: workspace %zu < %zu bytes", workspace_bytes, L.total);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* W = (double*)((char*)workspace + L.off_w);
    double* dpart = (double*)((char*)workspace + L.off_dpart);
    {
        const long long n = (long long)N * L.ldw;
        nspace_w_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(G, N, Lmat, Kt, L.Npad, L.ldw, W);
        PLSB_LAUNCH_CHECK("nspace_w_kernel");
    }
    // the grid: voxel tiles of 64 columns of W x splits of the period range that fill the SMs
    const int tiles = (int)cdiv(L.Nv, BM_VOX);
    {
        const int nsm = num_sms();
        int best = 1; double best_cost = 1e30;
        for (int n = 1; n <= 64; ++n) {
            if (n > 1 && b.nper / n < 4) break;
            const double waves = (double)tiles * n / nsm;
            const double cost = ceil(waves) / waves + 0.002 * (n - 1);
            if (cost < best_cost - 1e-12) { best_cost = cost; best = n; }
        }
        b.per_per_split = (int)cdiv(b.nper, best);
        b.nsplit = (int)cdiv(b.nper, b.per_per_split);
    }
    NsArgs a;
    a.W = W; a.ldw = L.ldw; a.N = N; a.Nv = L.Nv; a.Npad = L.Npad; a.coef = coef; a.nper = b.nper;
    a.per_per_split = b.per_per_split; a.nstage = b.nstage; a.R = R; a.Kp = b.Kp; a.K = K; a.Kt = Kt;
    a.dpart = dpart; a.Traw = T;
    const dim3 grid((unsigned)tiles, (unsigned)b.nsplit);
    const int rc = ring_dispatch(b, "nspace_dmma_f64", [&](auto nks, auto nblk) {
        const auto kernel = nspace_dmma_kernel<decltype(nks)::value, decltype(nblk)::value>;
        PLSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b.smem_bytes));
        kernel<<<grid, BM_THREADS, b.smem_bytes, st>>>(a);
        PLSB_LAUNCH_CHECK("nspace_dmma_kernel");
        return PLSB200_OK;
    });
    if (rc != PLSB200_OK) return rc;
    const long long n = (long long)R * K;
    nspace_finish_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(dpart, L.ngH, R, K, Kt, d2, T);
    PLSB_LAUNCH_CHECK("nspace_finish_kernel");
    return PLSB200_OK;
}
