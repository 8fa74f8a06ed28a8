// K4 for tall designs (N > 320 rows), output-stationary variant: the exact-mode bootstrap moment GEMM as a classic
// tiled DGEMM whose epilogue folds the tile into running moments instead of storing it.
//
//   VS[v, (r,k)] = sum_i X[i, v] C_r[i, k]          M = voxels, N = R*Kp columns, K-dim = rows of X
//
// boot_moments_kernel (boot.cu) keeps a warp's A fragments -- 8 voxels x all rows -- in registers, which is ideal
// while they fit (N <= 320) and makes every coefficient byte serve only the 64 voxels of a CTA.  Taller designs would
// have to split those fragments over several warps, and a coefficient byte would serve fewer voxels still: 16 per SM,
// 63 GB/s of coefficient ingest per SM at N = 1200, which held such a kernel to 0.76 of the DGEMM peak with a fifth of
// the warp samples waiting for stages (DESIGN.md §5.1b).  Here NOTHING is register-resident except the accumulators:
// a CTA owns a tile of 128 voxels x 96 columns (4 whole resamples at K = 24), both operands stream through shared
// memory in stages of 32 rows --
//   A: 32 rows x 128 voxels of X at a pitch of 132 doubles (so that the transposed fragment loads are bank-conflict-
//      free), read from a TILE-MAJOR IMAGE of X built once per call (os_ximage_kernel: [voxel tile][32-row block]
//      [32 x 132]), so that the block is three bulk copies of contiguous memory.  Fetching the 32 row segments of the
//      row-major X with one 1 KB bulk copy each made the copy engine the limiter: 27.7 TFLOP/s, 16 % of the warp
//      samples waiting for stages; with three large copies per block the same kernel runs at 32.5,
//   B: 8 k-steps x 12 column blocks of the coefficients, pre-packed in B-fragment order (one 24 KB bulk copy) --
// and each warp (4 x 2 layout, 32 voxels x 48 columns) issues 24 independent DMMAs per k-step from 10 fragment loads.
// A coefficient byte now serves 128 voxels and an X byte 96 columns: 37 GB/s per SM at any N.  After the last row
// the 48 accumulators of a thread hold (VS) for 4 voxel rows x 12 columns; they are folded into per-thread running
// moments of (VS - pivot) -- the column -> k map is tile-invariant because 96 is a multiple of every padded K -- and
// the CTA moves to the next column tile.  There is no limit on N.
#include "common.cuh"
#include "boot_plan.cuh"

namespace plsb {

constexpr int OS_TM = 128;            // voxels per CTA tile
constexpr int OS_TN = 96;             // columns per CTA tile
constexpr int OS_NB = OS_TN / 8;      // 8-column blocks per tile
constexpr int OS_PITCH = OS_TM + 4;   // doubles between consecutive rows of the A stage
// k-steps (of 4 rows) per pipeline stage: a template parameter KS in {5, 6, 7, 8}, chosen per design so that the row
// count pads to whole stages with the least waste (N = 300: 75 k-steps = 15 stages of 5; N = 1200: 300 = 38 of 8 - 4)
constexpr int os_a_doubles(int ks) { return 4 * ks * OS_PITCH; }
constexpr int os_b_doubles(int ks) { return ks * OS_NB * 32; }
constexpr int os_stage_doubles(int ks) { return os_a_doubles(ks) + os_b_doubles(ks); }       // 7296 ks bytes
constexpr int os_nstage(int ks) { return (215 * 1024) / (os_stage_doubles(ks) * 8) > 6 ? 6 : (215 * 1024) / (os_stage_doubles(ks) * 8); }

struct OsPlan {
    int Kp, nacc, nb, nks, ks, nct, nsplit, ct_per_split;
    size_t smem_bytes;
};

static bool os_plan(int N, int K, int R, int64_t p, OsPlan& b) {
    if (K < 1 || K > 24 || N < 1 || R < 1) return false;
    if (!pad_period(K, b.Kp, b.nacc)) return false;
    b.nb = 8 * b.nacc / b.Kp;
    {
        const int need = (int)cdiv(N, 4);
        // padded k-steps are wasted DMMAs; shallower stages cost about 1.5 % per k-step below 8 (more barrier rounds
        // per column tile: measured 0.85 vs 0.96 of the DGEMM peak between 5 and 8 k-steps per stage)
        int best_ks = 8; double best_cost = 1e30;
        for (int ks = 8; ks >= 5; --ks) {
            const double cost = (double)((int)cdiv(need, ks) * ks - need) / need + 0.015 * (8 - ks);
            if (cost < best_cost - 1e-12) { best_cost = cost; best_ks = ks; }
        }
        b.ks = best_ks;
        b.nks = (int)cdiv(need, b.ks) * b.ks;
    }
    b.nct = (int)cdiv((int64_t)R * b.Kp, OS_TN);
    b.smem_bytes = (size_t)os_nstage(b.ks) * os_stage_doubles(b.ks) * sizeof(double) + 256;
    // Split of the column tiles over CTAs that work on the SAME voxel tile (consecutive block indices, i.e. resident at
    // the same time).  A CTA re-streams its X tile (128 voxels x N rows = N KB) for every column tile; with one voxel
    // tile per SM the chip-wide working set is 148 N KB (180 MB at N = 1200) -- more than the L2 -- and every pass came
    // from HBM (ncu: L2 hit rate 32 %, 89 GB of DRAM reads for a 1.4 GB X, 16 % of the warp samples waiting for
    // stages).  nsplit CTAs per voxel tile shrink the working set to 148 / nsplit tiles: kept under ~48 MB.
    const int64_t tiles = cdiv(p > 0 ? p : 1, OS_TM);
    const int nsm = num_sms();
    int want = (int)cdiv((int64_t)nsm * N * 1024, (int64_t)48 << 20);
    int best = 1; double best_cost = 1e30;
    for (int n = 1; n <= 8; ++n) {
        if (n > 1 && b.nct / n < 4) break;
        const double waves = (double)tiles * n / nsm;
        const double cost = ceil(waves) / waves + 0.004 * (n - 1) + (n < want ? 0.05 * (want - n) : 0.0);
        if (cost < best_cost - 1e-12) { best_cost = cost; best = n; }
    }
    b.ct_per_split = (int)cdiv(b.nct, best);
    b.nsplit = (int)cdiv(b.nct, b.ct_per_split);
    return true;
}

// packed layout: offset(ct, s, jb, lane) = ((ct*nks + s)*12 + jb)*32 + lane ; column j = r*Kp + k -> ct = j / 96,
// jb = (j % 96) / 8, n = j % 8 ; row i -> s = i / 4, q = i % 4 ; lane = 4n + q
__global__ void __launch_bounds__(256) boot_os_pack_kernel(const double* __restrict__ E, int N, int K,
                                                          const int32_t* __restrict__ idx, int Kp, int nks,
                                                          double* __restrict__ coef) {
    extern __shared__ int ids[];          // E (N x K) stays in global memory: L1/L2-resident, read via __ldg
    int* start = ids + N; int* cur = start + N + 1; int* list = cur + N;
    const int r = blockIdx.x;
    build_source_lists(idx + (size_t)r * N, N, ids, start, cur, list);
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
        for (int k = 0; k < 24; ++k)
            if (k < K) {
                const long long j = (long long)r * Kp + k;
                const long long ct = j / OS_TN;
                const int cin = (int)(j % OS_TN);
                coef[(((size_t)ct * nks + s) * OS_NB + (cin >> 3)) * 32 + 4 * (cin & 7) + q] = acc[k];
            }
    }
}

// The factored collapsed bootstrap (boot_quad.cu, boot_factor_kernel) for this kernel: pseudo-resample j has the
// coefficients c_j[n,k] = E[n,k] . L[sid[n], j] (L: ns x J, row-major), written at the offsets of boot_os_pack_kernel
// (r = j).  No scatter, so no source lists: one CTA per pseudo-resample, a thread per row.  The padding (rows up to
// 4 nks, k >= K inside Kp, the tail of the last column tile) is the memset of boot_os_factor_pack.
__global__ void __launch_bounds__(256) boot_os_factor_pack_kernel(const double* __restrict__ E, int N, int K,
                                                                 const double* __restrict__ L, int J,
                                                                 const int32_t* __restrict__ sid, int Kp, int nks,
                                                                 double* __restrict__ coef) {
    const int j = blockIdx.x;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const double w = __ldg(L + (size_t)__ldg(sid + i) * J + j);
        const int s = i >> 2, q = i & 3;
        for (int k = 0; k < K; ++k) {
            const long long c = (long long)j * Kp + k;
            const long long ct = c / OS_TN;
            const int cin = (int)(c % OS_TN);
            coef[(((size_t)ct * nks + s) * OS_NB + (cin >> 3)) * 32 + 4 * (cin & 7) + q] = __ldg(E + (size_t)i * K + k) * w;
        }
    }
}

// Tile-major image of X: block (t, sb) = rows [4 ks sb, 4 ks (sb + 1)) x voxels [128 t, 128 t + 128) at a pitch of 132
// doubles, zero-filled beyond N rows / p voxels (and in the 4 padding columns).  One pass over X per call
// (3.5 ms for the 9.6 GB of BASELINE config 5, against 2.4 s of GEMM).  T = float: X stored as float32, widened here,
// so the image -- and everything after it -- is that of the widened matrix.
template <typename T>
__global__ void __launch_bounds__(256) os_ximage_kernel(const T* __restrict__ X, long long ldx, int N, long long p,
                                                       int nsb, int ks, double* __restrict__ img) {
    const long long t = blockIdx.x;
    const int sb = blockIdx.y;
    const int a_doubles = 4 * ks * OS_PITCH;
    double* out = img + ((size_t)t * nsb + sb) * a_doubles;
    for (int i = threadIdx.x; i < a_doubles; i += 256) {
        const int r = i / OS_PITCH, c = i % OS_PITCH;
        const int row = sb * 4 * ks + r;
        const long long v = t * OS_TM + c;
        out[i] = (c < OS_TM && row < N && v < p) ? (double)__ldg(X + (long long)row * ldx + v) : 0.0;
    }
}

template <int NACC, int KS>
__global__ void __launch_bounds__(256, 1)
boot_moments_os_kernel(const double* __restrict__ Ximg, int N, long long p,
                       const double* __restrict__ coef, int nks, int nct, int ct_per_split, int R, int Kp, int K,
                       const double* __restrict__ pivot, double* __restrict__ osum, double* __restrict__ osumsq) {
    constexpr int OS_KS = KS, OS_A_DOUBLES = os_a_doubles(KS), OS_B_DOUBLES = os_b_doubles(KS),
                  OS_STAGE_DOUBLES = os_stage_doubles(KS), OS_NSTAGE = os_nstage(KS);
    extern __shared__ __align__(128) unsigned char smraw[];
    double* ring = reinterpret_cast<double*>(smraw);
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)OS_NSTAGE * OS_STAGE_DOUBLES);
    uint64_t* empty = full + OS_NSTAGE;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wm = warp >> 1, wn = warp & 1;             // 4 x 2 warps: 32 voxels x 48 columns each
    const int q = lane & 3, vr = lane >> 2;
    const int nsplit = (nct + ct_per_split - 1) / ct_per_split;
    const int split = (int)(blockIdx.x % nsplit);          // consecutive blocks = the splits of one voxel tile
    const long long v0 = (long long)(blockIdx.x / nsplit) * OS_TM;
    (void)N;
    const int ct0 = split * ct_per_split;
    const int ct1 = min(nct, ct0 + ct_per_split);
    const int spc = nks / OS_KS;                         // stages per column tile
    const int nit = (ct1 - ct0) * spc;

    if (tid == 0) {
        for (int s = 0; s < OS_NSTAGE; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 8); }
        mbar_fence_init();
    }
    __syncthreads();

    // warp 0 (also a consumer) is the producer: the A block of a stage is one contiguous 33 KB piece of the image
    // (one bulk copy), the coefficient block one of 24 KB (another)
    const double* atile = Ximg + (size_t)(blockIdx.x / nsplit) * spc * OS_A_DOUBLES;
    auto issue = [&](int g, int slot) {
        const int ct = ct0 + g / spc, sk = g % spc;
        double* A = ring + (size_t)slot * OS_STAGE_DOUBLES;
        if (lane == 0) mbar_expect_tx(full + slot, (uint32_t)OS_STAGE_DOUBLES * 8u);
        __syncwarp();
        const double* asrc = atile + (size_t)sk * OS_A_DOUBLES;
        const double* bsrc = coef + ((size_t)ct * nks + (size_t)sk * OS_KS) * (OS_NB * 32);
        constexpr uint32_t AB = (uint32_t)OS_A_DOUBLES * 8u, BB = (uint32_t)OS_B_DOUBLES * 8u;
        if (lane == 0) bulk_g2s(A, asrc, AB, full + slot);
        else if (lane == 1) bulk_g2s(A + OS_A_DOUBLES, bsrc, BB, full + slot);
    };
    if (warp == 0)
        for (int g = 0; g < min(OS_NSTAGE, nit); ++g) issue(g, g);

    // running moments of this thread's 4 voxel rows x (NACC blocks x 2) column classes (columns 8*NACC apart share k)
    double s1[4][NACC][2], s2[4][NACC][2];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int jm = 0; jm < NACC; ++jm) { s1[mt][jm][0] = s1[mt][jm][1] = 0.0; s2[mt][jm][0] = s2[mt][jm][1] = 0.0; }

    const int nbp = 8 * NACC / Kp;             // resamples per period of 8 NACC columns
    // the two warps of an SM sub-partition (w and w + 4) run half a stage apart, so that one of them keeps the DMMA
    // pipe busy while the other folds a finished tile or waits at a stage boundary (as in boot_moments_kernel)
    if (warp >= 4) __nanosleep((unsigned)(OS_KS * 24 * 8));      // ~ half a stage
    int slot = 0, prev_slot = 0, g = 0;
    uint32_t phase = 0, prev_phase = 0;
    for (int ct = ct0; ct < ct1; ++ct) {
        double acc[4][6][2];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
            for (int j = 0; j < 6; ++j) acc[mt][j][0] = acc[mt][j][1] = 0.0;
        for (int sk = 0; sk < spc; ++sk, ++g) {
            if (warp == 0 && g > 0) {
                const int nx = g - 1 + OS_NSTAGE;       // refill the slot drained in the previous stage
                if (nx < nit) {
                    if (lane == 0) mbar_wait(empty + prev_slot, prev_phase);
                    __syncwarp();
                    issue(nx, prev_slot);
                }
            }
            __syncwarp();
            mbar_wait(full + slot, phase);
            const double* As = ring + (size_t)slot * OS_STAGE_DOUBLES + q * OS_PITCH + wm * 32 + vr;
            const double* Bs = ring + (size_t)slot * OS_STAGE_DOUBLES + OS_A_DOUBLES + (wn * 6) * 32 + lane;
#pragma unroll
            for (int ks = 0; ks < OS_KS; ++ks) {
                double a[4], b[6];
#pragma unroll
                for (int mt = 0; mt < 4; ++mt) a[mt] = As[(4 * ks) * OS_PITCH + mt * 8];
#pragma unroll
                for (int j = 0; j < 6; ++j) b[j] = Bs[(ks * OS_NB + j) * 32];
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                    for (int j = 0; j < 6; ++j) dmma884(acc[mt][j][0], acc[mt][j][1], a[mt], b[j]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + slot);
            prev_slot = slot; prev_phase = phase;
            if (++slot == OS_NSTAGE) { slot = 0; phase ^= 1u; }
        }
        // fold the finished tile: (VS - pivot) into the running moments; padding columns (k >= K) and resamples
        // beyond R are masked.  32-bit index arithmetic only: the column of an accumulator within its period,
        // c = 8 (j mod NACC) + 2q + e, fixes k and the resample slot for the whole kernel.
        const int rbase = ct * (OS_TN / Kp) + wn * (48 / Kp);          // first resample of this warp's 48 columns
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            const long long v = v0 + wm * 32 + mt * 8 + vr;
            const bool vok = v < p;
            const double* pv = pivot != nullptr ? pivot + (vok ? v : 0) * K : nullptr;
#pragma unroll
            for (int j = 0; j < 6; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int c = 8 * (j % NACC) + 2 * q + e;
                    const int rr = c / Kp, k = c - rr * Kp;
                    const int r = rbase + (j / NACC) * nbp + rr;
                    if (k < K && r < R && vok) {
                        const double dd = acc[mt][j][e] - (pv != nullptr ? __ldg(pv + k) : 0.0);
                        s1[mt][j % NACC][e] += dd;
                        s2[mt][j % NACC][e] = fma(dd, dd, s2[mt][j % NACC][e]);
                    }
                }
        }
    }

    // ---- combine: the classes of a thread that share k (NACC*8 / Kp of them), then the two warps of a voxel row
    //      block, in a fixed order (deterministic); the ring is free now
    __syncthreads();
    double* r1 = ring;                         // [128][Kp]
    double* r2 = ring + OS_TM * Kp;
    for (int i = tid; i < 2 * OS_TM * Kp; i += 256) ring[i] = 0.0;
    __syncthreads();
    for (int half = 0; half < 2; ++half) {
        if (wn == half) {
            for (int round = 0; round < nbp; ++round) {
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                    for (int jm = 0; jm < NACC; ++jm)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int c = 8 * jm + 2 * q + e;
                            if (c / Kp == round) {
                                const int row = wm * 32 + mt * 8 + vr;
                                r1[row * Kp + c % Kp] += s1[mt][jm][e];
                                r2[row * Kp + c % Kp] += s2[mt][jm][e];
                            }
                        }
                __syncwarp();
            }
        }
        __syncthreads();
    }
    double* o1 = osum + (size_t)split * p * K;
    double* o2 = osumsq + (size_t)split * p * K;
    for (int i = tid; i < OS_TM * K; i += 256) {
        const int rr = i / K, k = i % K;
        if (v0 + rr < p) {
            o1[(v0 + rr) * K + k] = r1[rr * Kp + k];
            o2[(v0 + rr) * K + k] = r2[rr * Kp + k];
        }
    }
}

template <int NACC, int KS>
static int os_launch_ks(const OsPlan& b, const double* Ximg, int N, int64_t p, const double* coef, int K, int R,
                        const double* pivot, double* o1, double* o2, cudaStream_t st) {
    PLSB_CUDA(cudaFuncSetAttribute(boot_moments_os_kernel<NACC, KS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)b.smem_bytes));
    dim3 grid((unsigned)(cdiv(p, OS_TM) * b.nsplit));
    boot_moments_os_kernel<NACC, KS><<<grid, 256, b.smem_bytes, st>>>(Ximg, N, p, coef, b.nks, b.nct, b.ct_per_split, R,
                                                                 b.Kp, K, pivot, o1, o2);
    PLSB_LAUNCH_CHECK("boot_moments_os_kernel");
    return PLSB200_OK;
}

template <int NACC>
static int os_launch(const OsPlan& b, const double* Ximg, int N, int64_t p, const double* coef, int K, int R,
                     const double* pivot, double* o1, double* o2, cudaStream_t st) {
    switch (b.ks) {
        case 5: return os_launch_ks<NACC, 5>(b, Ximg, N, p, coef, K, R, pivot, o1, o2, st);
        case 6: return os_launch_ks<NACC, 6>(b, Ximg, N, p, coef, K, R, pivot, o1, o2, st);
        case 7: return os_launch_ks<NACC, 7>(b, Ximg, N, p, coef, K, R, pivot, o1, o2, st);
        default: return os_launch_ks<NACC, 8>(b, Ximg, N, p, coef, K, R, pivot, o1, o2, st);
    }
}

static size_t os_image_bytes(const OsPlan& b, int64_t p) {
    return (size_t)cdiv(p, OS_TM) * (b.nks / b.ks) * os_a_doubles(b.ks) * sizeof(double);
}
static size_t os_partial_bytes(const OsPlan& b, int64_t p, int K) {
    const size_t n = b.nsplit > 1 ? (size_t)2 * b.nsplit * p * K * sizeof(double) : 0;
    return (n + 255) & ~(size_t)255;
}

size_t boot_os_coef_bytes(int N, int K, int R) {
    OsPlan b;
    if (!os_plan(N, K, R, 1, b)) return 0;
    return (size_t)b.nct * b.nks * OS_NB * 32 * sizeof(double);
}

size_t boot_os_workspace(int N, int64_t p, int K, int R) {
    OsPlan b;
    if (!os_plan(N, K, R, p, b)) return 0;
    return os_partial_bytes(b, p, K) + os_image_bytes(b, p) + 256;
}

int boot_os_pack(const double* E, int N, int K, const int32_t* idx, int R, double* coef, cudaStream_t st) {
    OsPlan b;
    if (!os_plan(N, K, R, 1, b)) {
        set_err("boot_coef_pack_f64: unsupported shape N=%d K=%d R=%d (need K<=24)", N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaMemsetAsync(coef, 0, (size_t)b.nct * b.nks * OS_NB * 32 * sizeof(double), st));
    boot_os_pack_kernel<<<R, 256, (size_t)(4 * N + 1) * sizeof(int), st>>>(E, N, K, idx, b.Kp, b.nks, coef);
    PLSB_LAUNCH_CHECK("boot_os_pack_kernel");
    return PLSB200_OK;
}

// the layout is that of boot_os_pack with R = J, so boot_os_coef_bytes(N, K, J) sizes it
int boot_os_factor_pack(const double* E, int N, int K, const double* L, int J, const int32_t* sid, double* coef,
                        cudaStream_t st) {
    OsPlan b;
    if (!os_plan(N, K, J, 1, b)) {
        set_err("boot_factor_pack_f64: unsupported shape N=%d K=%d J=%d (need K<=24)", N, K, J);
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaMemsetAsync(coef, 0, (size_t)b.nct * b.nks * OS_NB * 32 * sizeof(double), st));
    boot_os_factor_pack_kernel<<<J, 256, 0, st>>>(E, N, K, L, J, sid, b.Kp, b.nks, coef);
    PLSB_LAUNCH_CHECK("boot_os_factor_pack_kernel");
    return PLSB200_OK;
}

template <typename T>
static int os_moments(const T* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R, const double* pivot,
                      double* sum, double* sumsq, void* workspace, size_t workspace_bytes, cudaStream_t st,
                      const char* what) {
    OsPlan b;
    if (!os_plan(N, K, R, p, b)) {
        set_err("%s: unsupported shape N=%d K=%d R=%d (need K<=24)", what, N, K, R);
        return PLSB200_EUNSUPPORTED;
    }
    const size_t pbytes = os_partial_bytes(b, p, K), need = pbytes + os_image_bytes(b, p);
    if (!workspace || workspace_bytes < need) {
        set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    if ((size_t)(base - (char*)workspace) + need > workspace_bytes) {
        set_err("%s: workspace too small after alignment", what);
        return PLSB200_EWORKSPACE;
    }
    double *o1 = sum, *o2 = sumsq;
    if (b.nsplit > 1) { o1 = (double*)base; o2 = o1 + (size_t)b.nsplit * p * K; }
    double* img = (double*)(base + pbytes);
    {
        dim3 grid((unsigned)cdiv(p, OS_TM), (unsigned)(b.nks / b.ks));
        os_ximage_kernel<T><<<grid, 256, 0, st>>>(X, ldx, N, p, b.nks / b.ks, b.ks, img);
        PLSB_LAUNCH_CHECK("os_ximage_kernel");
    }
    int rc;
    switch (b.nacc) {
        case 1: rc = os_launch<1>(b, img, N, p, coef, K, R, pivot, o1, o2, st); break;
        case 2: rc = os_launch<2>(b, img, N, p, coef, K, R, pivot, o1, o2, st); break;
        default: rc = os_launch<3>(b, img, N, p, coef, K, R, pivot, o1, o2, st); break;
    }
    if (rc != PLSB200_OK) return rc;
    if (b.nsplit > 1) {
        const long long n = (long long)p * K;
        split_sum_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(o1, o2, b.nsplit, n, sum, sumsq);
        PLSB_LAUNCH_CHECK("split_sum_kernel");
    }
    return PLSB200_OK;
}

int boot_os_moments(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R, const double* pivot,
                    double* sum, double* sumsq, void* workspace, size_t workspace_bytes, cudaStream_t st,
                    const char* what) {
    return os_moments(X, N, p, ldx, coef, K, R, pivot, sum, sumsq, workspace, workspace_bytes, st, what);
}

int boot_os_moments(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K, int R, const double* pivot,
                    double* sum, double* sumsq, void* workspace, size_t workspace_bytes, cudaStream_t st,
                    const char* what) {
    return os_moments(X, N, p, ldx, coef, K, R, pivot, sum, sumsq, workspace, workspace_bytes, st, what);
}

}  // namespace plsb
