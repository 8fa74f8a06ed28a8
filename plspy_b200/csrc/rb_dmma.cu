// K5 on the FP64 tensor path: the p-space bootstrap pass of behaviour / multiblock PLS (same contract as
// plsb200_rb_boot_f64 in rb.cu, which stays as the general fallback).
//
// Per bootstrap b and (group, condition) cell c (class_functions.py:219-245 as called at bootstrap_permutation.py:613):
//     P_c[v, k]  = sum_{i in c} Xc[i, v] Q_b[i, k]                      <- DMMA, M = voxels, k-dim = rows of the cell
//     m1, m2     = sum_i w_b[i] Xc[i, v], sum_i w_b[i] Xc[i, v]^2       <- FMA on the same register-resident fragments
//     VS_b[v, k] = sum_c P_c[v, k] / (sd_c(v) sqrt(n_c)),  sd_c^2 = m2 - m1^2   (1 for the trailing `unit` cells)
// and then  sum / sum of squares of (VS_b - pivot),  ||VS_b[:, k]||^2  and  T_b = Xc . VS_b  (N x K).
//
//   kernel A (rb_vs_kernel): as K4 (boot.cu) a warp owns 8 voxels and keeps its X fragments in registers for the
//     whole launch; the per-bootstrap coefficients are pre-packed in B-fragment order (cells padded to whole
//     k-steps of 4 rows) and streamed through shared memory with bulk copies.  A cell is a run of k-steps; at its
//     end the quad-reduced moments give the scale and the cell's D fragments are folded into VS.  VS_b is written
//     transposed ([column][voxel]) for kernel B, the moments are folded in registers.
//   kernel B (gemm_nt_partial_kernel): T = Xc . VS^T-transposed as a split-K DMMA GEMM over voxel chunks (the Gram
//     kernel generalised to two operand matrices), partials reduced in a fixed order.
// Columns are processed in passes of 8*NBLK (NBLK = 1, 2, 3 for K <= 8, 16, more); the running moments live in
// shared memory so that the registers are free for up to 96 k-steps of X fragments (384 padded rows).
#include "common.cuh"
#include <stdlib.h>

namespace plsb {

constexpr int RD_MAXKS = 96;

struct RdPlan {
    int nks, nblk, kcp, npass, nstage, warps;   // warps: template bucket (8 or 16) = upper bound of the launch
    int ks_unit;                                // first k-step of the trailing unit cells
    int nstd;                                   // standardised cells (the cells before the trailing unit cells)
    bool md;                                    // block moments on the tensor cores, 8 bootstraps at a time (see rb_vs_kernel)
    size_t stage_doubles;        // packed coefficients + weights of one bootstrap and one pass
    size_t smem_bytes;
    int krow[RD_MAXKS * 4];      // k-step slot -> row of Xc (-1 = padding)
    double celln[16];            // rows per cell (negative for unit cells)
    int ncell;
    uint32_t cend[3];            // bit s set: k-step s ends a cell
};

static bool rd_plan(int N, int K, const int32_t* cs, int ncell, int unit_cells, RdPlan& r) {
    if (N < 1 || K < 1 || ncell < 1 || ncell > 16 || cs[0] != 0 || cs[ncell] != N) return false;
    r.ncell = ncell;
    int s = 0;
    r.cend[0] = r.cend[1] = r.cend[2] = 0;
    r.ks_unit = -1;
    for (int c = 0; c < ncell; ++c) {
        const int n = cs[c + 1] - cs[c];
        if (n < 1) return false;
        const int ks = (n + 3) / 4;
        if (s + ks > RD_MAXKS) return false;
        if (c >= ncell - unit_cells && r.ks_unit < 0) r.ks_unit = s;
        for (int t = 0; t < ks * 4; ++t) r.krow[s * 4 + t] = t < n ? cs[c] + t : -1;
        r.celln[c] = c >= ncell - unit_cells ? -(double)n : (double)n;
        r.cend[(s + ks - 1) >> 5] |= 1u << ((s + ks - 1) & 31);
        s += ks;
    }
    r.nks = (s + 3) / 4 * 4;                       // kernels are instantiated for multiples of 4 k-steps
    if (r.ks_unit < 0) r.ks_unit = r.nks;
    for (int t = s; t < r.nks; ++t)
        for (int q = 0; q < 4; ++q) r.krow[t * 4 + q] = -1;
    r.nblk = K <= 8 ? 1 : (K <= 16 ? 2 : 3);
    r.kcp = 8 * r.nblk;
    r.npass = (int)cdiv(K, r.kcp);
    r.stage_doubles = (size_t)r.nks * r.nblk * 32 + (size_t)r.nks * 4;
    r.warps = r.nks <= 32 ? 16 : 8;
    r.nstd = ncell - unit_cells;
    const size_t coef_bytes = (size_t)r.nks * r.nblk * 32 * sizeof(double);
    // moments on DMMA: weight fragments of one batch of 8 bootstraps, block sizes, running moments, per-warp scale tables
    // of the batch ([8 bootstraps][standardised cell][8 voxels]), barriers
    const size_t fixed_md = ((size_t)r.nks * 32 + 16 + 3 * r.nblk * 2 * r.warps * 32 + (size_t)r.warps * 64 * (r.nstd > 0 ? r.nstd : 1)) * sizeof(double) + 256;
    int ns = (int)((225 * 1024 - (long long)fixed_md) / (long long)coef_bytes);
    if (ns > 4) ns = 4;
    // (only the 16-warp bucket: with 8 warps -- 2 per scheduler -- the serial moment phase of a batch is not covered by other
    // warps; cfg 4 pass 2, 92 k-steps of which 30 standardised: 7.79 ms with the scalar moments, 8.41 ms with the DMMA moments)
    r.md = ns >= 2 && r.nstd > 0 && r.warps == 16;
    if (r.md) {
        r.nstage = ns;
        r.smem_bytes = ns * coef_bytes + fixed_md;
        return true;
    }
    // scalar moments: weight ring (4 slots), block sizes, running moments, per-warp scale / moment tables, barriers
    const size_t fixed = ((size_t)4 * r.nks * 4 + 16 + 3 * r.nblk * 2 * r.warps * 32 + r.warps * 16 * 24) * sizeof(double) + 256;
    ns = (int)((225 * 1024 - (long long)fixed) / (long long)coef_bytes);
    if (ns > 4) ns = 4;
    if (ns < 2) return false;
    r.nstage = ns;
    r.smem_bytes = ns * coef_bytes + fixed;
    return true;
}

// Q (R x N x K), W (R x N) -> per (bootstrap, pass): [nks][nblk][32] B-fragments (lane = 4*col + q holds
// Q[krow[4s+q]][k0 + 8j + col]) followed by [nks][4] weights.
__global__ void rd_pack_kernel(const double* __restrict__ Q, const double* __restrict__ W, int N, int K, int b0,
                               const int* __restrict__ krow, int nks, int nblk, int npass,
                               double* __restrict__ pack) {
    const int bb = blockIdx.x, pass = blockIdx.y;
    const size_t stage = (size_t)nks * nblk * 32 + (size_t)nks * 4;
    double* out = pack + ((size_t)bb * npass + pass) * stage;
    const double* q = Q + (size_t)(b0 + bb) * N * K;
    const double* w = W ? W + (size_t)(b0 + bb) * N : nullptr;
    const int k0 = pass * 8 * nblk;
    const int nq = nks * nblk * 32;
    for (int i = threadIdx.x; i < nq; i += blockDim.x) {
        const int lane = i & 31, j = (i >> 5) % nblk, s = (i >> 5) / nblk;
        const int row = krow[4 * s + (lane & 3)], col = k0 + 8 * j + (lane >> 2);
        out[i] = (row >= 0 && col < K) ? q[(size_t)row * K + col] : 0.0;
    }
    for (int i = threadIdx.x; i < nks * 4; i += blockDim.x) {
        const int row = krow[i];
        out[nq + i] = (row >= 0 && w) ? w[row] : 0.0;
    }
}

// multiplicity weights of a batch of 8 bootstraps as DMMA B fragments: [batch][nks][32], lane = 4*col + q holds the weight
// of bootstrap 8*batch + col for row krow[4s + q] (0 for padding rows / bootstraps past the end)
__global__ void rd_wpack_kernel(const double* __restrict__ W, int N, int b0, int nbt, const int* __restrict__ krow, int nks,
                                double* __restrict__ wpack) {
    const int batch = blockIdx.x;
    double* out = wpack + (size_t)batch * nks * 32;
    for (int i = threadIdx.x; i < nks * 32; i += blockDim.x) {
        const int lane = i & 31, s = i >> 5;
        const int bb = 8 * batch + (lane >> 2), row = krow[4 * s + (lane & 3)];
        out[i] = (W && bb < nbt && row >= 0) ? W[(size_t)(b0 + bb) * N + row] : 0.0;
    }
}

struct RdArgs {
    const double* Xc2;     // rows [n1, N) of the data matrix live here (row stride ld2); n1 == N: a single matrix
    long long ld2;
    int n1;
    const double* Xc;
    const double* pack;
    const double* wpack;   // MD kernels: weight fragments per batch of 8 bootstraps
    const double* pivot;
    const int* krow;
    const double* celln;
    double* sum;
    double* sumsq;
    double* VSt;       // [nbt][kcp][p]  (may be NULL when T is not wanted)
    double* VS;        // [nbt][p][Kfull] from the launch's first bootstrap: the saliences themselves (NULL: not exported)
    double* Npart;     // [nbt][kcp][tiles*8]
    long long p;       // ONLY: the end of the voxel window
    int Kfull, k0, kc, nbt, npass, pass, nstage, ncell, nwarps;
    int ks_unit;       // first k-step of the trailing unit cells (plain linear rows: no block moments needed); nks if none
    int nstd;          // standardised cells
    uint32_t cend[3];
    long long v0;      // ONLY: first voxel of the window; VS is [nbt][p - v0][Kfull]
    long long ld1;     // ONLY: row stride of Xc (the other instantiations: p)
    int bslice;        // ONLY: bootstraps per blockIdx.y (a multiple of 8)
};

constexpr int RD_MAXCELL = 16;

// scale of one (cell, voxel): 1 / (sd sqrt(n)); same guards as rb_boot_kernel (an all-identical resampled block has
// var == 0: nan -> 0 in the reference); unit cells (n < 0) are plain linear rows.  Called from one place only (a runtime loop), so the
// FP64 sqrt / divide sequence exists once in the instruction stream.
__device__ __forceinline__ double rd_scale(double m1, double m2, double n) {
    if (n < 0.0) return 1.0;
    const double var = m2 - m1 * m1;
    return (var > 1e-13 * m2 && var > 0.0) ? 1.0 / sqrt(var * n) : 0.0;
}

// MD path: the two scales a lane owns at the end of a cell (voxel vr, bootstraps 2q and 2q+1 of the batch).  Not inlined: it is
// reached from every k-step of the unrolled moment loop and the FP64 sqrt / divide sequence should exist once.
__device__ __noinline__ void rd_store_scales(double* dst0, double* dst1, double a10, double a20, double a11, double a21, double n) {
    *dst0 = rd_scale(a10, a20, n);
    *dst1 = rd_scale(a11, a21, n);
}

// W = warps per CTA: 8 (256 registers per thread: up to 96 k-steps of fragments) or 16 (128 registers: <= 32 k-steps,
// twice the warps per scheduler to hide the serial phases between the DMMA bursts).
// MD = block moments on the tensor cores.  The scalar version (MD = false) forms the weighted block moments of bootstrap b+1
// with three FP64 operations per k-step in the shadow of the DMMAs of bootstrap b: on this GPU they share the FP64 pipe with
// the DMMAs (ncu, profiles/ncu_rb_vs_r02.md: DADD + DMUL collect 34 % of the warp samples, DMMA 22 %; math-pipe throttle is the
// top stall).  With MD the moments of EIGHT bootstraps are one DMMA chain per moment: D[voxel][bootstrap] += X-fragment x
// weight-fragment (the multiplicity weights of the 8 bootstraps packed as a B fragment, rd_wpack_kernel), once per batch of 8
// bootstraps -- 2 DMMAs + 1 DMUL per k-step and batch instead of 24 scalar operations and 8 quad reductions -- and the lane
// that ends up with (voxel, bootstraps 2q, 2q+1) stores their two scales into the batch's scale table.
// EXPORT = also store VS_b into a.VS.  A template flag, not only a run-time test of a.VS: the 8-warp bucket holds up to
// 96 k-steps of X fragments in 254 of its 255 registers, and the instantiations without the store keep exactly the
// registers (and the code) of the kernel without the feature.
// ONLY (with EXPORT) = the export alone, over the voxel window [a.v0, a.p) of a matrix whose first segment has the row
// stride a.ld1, into VS[b][v - v0][k]: no pivot moments, norms or transposed VS.  blockIdx.y takes the bootstraps
// [y * bslice, (y + 1) * bslice); bslice is a multiple of 8, so the MD path forms the batches of the whole-p pass.  The
// saliences of a voxel depend on its own column of X only, so a window's values are those of the whole-p pass.
template <int NKS, int NBLK, int W, bool MD, bool EXPORT, bool ONLY = false>
__global__ void __launch_bounds__(W * 32, 1) rb_vs_kernel(const RdArgs a) {
    static_assert(EXPORT || !ONLY, "ONLY is an export mode");
    constexpr int RD_WARPS = W, RD_THREADS = W * 32;
    extern __shared__ __align__(128) unsigned char smraw[];
    constexpr int coef_doubles = NKS * NBLK * 32;                 // B fragments of one bootstrap and pass
    constexpr int w_doubles = NKS * 4;                            // its multiplicity weights, k-step order
    constexpr int pack_doubles = coef_doubles + w_doubles;        // layout of one (bootstrap, pass) in `pack`
    constexpr uint32_t coef_bytes = (uint32_t)coef_doubles * 8u, w_bytes = (uint32_t)w_doubles * 8u;
    constexpr int WSLOTS = MD ? 1 : 4;
    constexpr int w8_doubles = NKS * 32;                          // MD: weight fragments of one batch of 8 bootstraps
    constexpr uint32_t w8_bytes = (uint32_t)w8_doubles * 8u;
    const int nstd8 = a.nstd * 8;                                 // MD: scale-table entries per bootstrap of the batch
    double* ring = reinterpret_cast<double*>(smraw);              // [nstage][coef_doubles]
    double* wring = ring + (size_t)a.nstage * coef_doubles;       // [WSLOTS][w_doubles]   (MD: [w8_doubles])
    double* celln = wring + (MD ? w8_doubles : WSLOTS * w_doubles);   // [RD_MAXCELL] rows per cell (negative: unit cell)
    double* acc = celln + RD_MAXCELL;                             // [2][NBLK*2][RD_THREADS] running moments
    double* pvs = acc + 2 * NBLK * 2 * RD_THREADS;                // [NBLK*2][RD_THREADS] pivot of this thread's elements
    double* tabs = pvs + NBLK * 2 * RD_THREADS;                   // per warp: scale[16][8], then (m1, m2)[16][8]  (MD: scale[8][nstd][8])
    uint64_t* full = reinterpret_cast<uint64_t*>(tabs + (MD ? (size_t)RD_WARPS * 8 * nstd8 : (size_t)RD_WARPS * RD_MAXCELL * 24));
    uint64_t* empty = full + a.nstage;
    uint64_t* wfull = empty + a.nstage;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = lane & 3, vr = lane >> 2;
    const int nwarps = a.nwarps;                                  // warps launched (<= W, see rd_balanced_warps)
    long long v = (long long)blockIdx.x * (nwarps * 8) + warp * 8 + vr;
    if constexpr (ONLY) v += a.v0;
    const bool ok = v < a.p;
    // ONLY: this CTA's bootstraps are [bofs, bofs + nbt_s) of the launch; everything below counts from bofs (the other
    // instantiations read a.nbt as before: bofs and nbt_s are not used there)
    const int bofs = ONLY ? (int)blockIdx.y * a.bslice : 0;
    const int nbt_s = ONLY ? min(a.bslice, a.nbt - bofs) : 0;
#define RD_NBT (ONLY ? nbt_s : a.nbt)

    if (tid == 0) {
        for (int s = 0; s < a.nstage; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, nwarps); }
        for (int s = 0; s < WSLOTS; ++s) mbar_init(wfull + s, 1);
        mbar_fence_init();
    }
    for (int i = tid; i < RD_MAXCELL; i += nwarps * 32) celln[i] = i < a.ncell ? a.celln[i] : 0.0;
    __syncthreads();

    const size_t bstride = (size_t)a.npass * pack_doubles;        // doubles between consecutive bootstraps
    auto issue = [&](int bb, int slot) {                          // coefficients of bootstrap bb -> ring slot
        mbar_expect_tx(full + slot, coef_bytes);
        const char* src = reinterpret_cast<const char*>(a.pack + (size_t)(ONLY ? bb + bofs : bb) * bstride + (size_t)a.pass * pack_doubles);
        char* dst = reinterpret_cast<char*>(ring + (size_t)slot * coef_doubles);
#pragma unroll 1
        for (uint32_t off = 0; off < coef_bytes; off += 16384u)
            bulk_g2s(dst + off, src + off, min(16384u, coef_bytes - off), full + slot);
    };
    auto issue_w = [&](int bb) {                                  // weights of bootstrap bb -> slot bb % WSLOTS
        const int ws_ = bb % WSLOTS;
        mbar_expect_tx(wfull + ws_, w_bytes);
        bulk_g2s(wring + ws_ * w_doubles,
                 a.pack + (size_t)(ONLY ? bb + bofs : bb) * bstride + (size_t)a.pass * pack_doubles + coef_doubles, w_bytes, wfull + ws_);
    };
    auto issue_w8 = [&](int batch) {                              // MD: weight fragments of bootstraps 8 batch ... 8 batch + 7
        mbar_expect_tx(wfull, w8_bytes);
        const char* src = reinterpret_cast<const char*>(a.wpack + (size_t)(ONLY ? batch + bofs / 8 : batch) * w8_doubles);
        char* dst = reinterpret_cast<char*>(wring);
#pragma unroll 1
        for (uint32_t off = 0; off < w8_bytes; off += 16384u)
            bulk_g2s(dst + off, src + off, min(16384u, w8_bytes - off), wfull);
    };
    if (tid == 0) {
        if constexpr (MD) issue_w8(0);
        else
            for (int bb = 0; bb < min(WSLOTS, RD_NBT); ++bb) issue_w(bb);
        for (int bb = 0; bb < min(a.nstage, RD_NBT); ++bb) issue(bb, bb);
    }

    double x[NKS];
#pragma unroll
    for (int s = 0; s < NKS; ++s) {
        const int row = __ldg(a.krow + 4 * s + q);
        x[s] = (row >= 0 && ok) ? __ldg((row < a.n1 ? a.Xc + (long long)row * (ONLY ? a.ld1 : a.p)
                                                     : a.Xc2 + (long long)(row - a.n1) * a.ld2) + v) : 0.0;
    }
    // running moments live in shared memory (one slot per thread and fragment element): registers are for X
    double* my1 = acc + tid;
    double* my2 = acc + NBLK * 2 * RD_THREADS + tid;
    double* myp = pvs + tid;
#pragma unroll
    for (int j = 0; j < NBLK; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int c = 8 * j + 2 * q + e;
            const bool live = !ONLY && ok && c < a.kc;                // (ONLY: no moments)
            my1[(2 * j + e) * RD_THREADS] = live ? a.sum[v * a.Kfull + a.k0 + c] : 0.0;
            my2[(2 * j + e) * RD_THREADS] = live ? a.sumsq[v * a.Kfull + a.k0 + c] : 0.0;
            // (the pivot is the same for every bootstrap: read once -- as a per-bootstrap __ldg its L2 latency sat on
            // the fold's critical path, 5 % of the warp samples)
            myp[(2 * j + e) * RD_THREADS] = (live && a.pivot) ? __ldg(a.pivot + v * a.Kfull + a.k0 + c) : 0.0;
        }
    double* sct = MD ? tabs + (size_t)warp * 8 * nstd8            // MD: scale[bootstrap of the batch][cell][voxel]
                     : tabs + warp * (RD_MAXCELL * 24);           // scale[cell][voxel] of the current bootstrap
    double* mt = sct + RD_MAXCELL * 8;                            // (m1, m2)[cell][voxel] of the next one   (not MD)
    auto scales = [&]() {       // one (cell, voxel) pair per lane, no redundancy across the quad
        __syncwarp();
        for (int i = lane; i < a.ncell * 8; i += 32) sct[i] = rd_scale(mt[2 * i], mt[2 * i + 1], celln[i >> 3]);
        __syncwarp();
    };
    // MD: moments and scales of a whole batch.  D fragment: row = voxel vr, columns 2q, 2q+1 = bootstraps of the batch.
    auto batch_scales = [&](uint32_t parity) {
        mbar_wait(wfull, parity);
        const volatile double* wl = wring + lane;
        double a1[2] = {0.0, 0.0}, a2[2] = {0.0, 0.0};
        int cell = 0;
#pragma unroll
        for (int s = 0; s < NKS; ++s) {
            if (s < a.ks_unit) {                                  // warp-uniform
                const double wf = wl[s * 32];
                dmma884(a1[0], a1[1], x[s], wf);
                dmma884(a2[0], a2[1], x[s] * x[s], wf);
            }
            if ((a.cend[s >> 5] >> (s & 31)) & 1u) {              // warp-uniform: last k-step of a cell
                if (cell < a.nstd)
                    rd_store_scales(sct + (2 * q) * nstd8 + cell * 8 + vr, sct + (2 * q + 1) * nstd8 + cell * 8 + vr,
                                    a1[0], a2[0], a1[1], a2[1], celln[cell]);
                ++cell;
                a1[0] = a1[1] = a2[0] = a2[1] = 0.0;
            }
        }
        __syncwarp();
    };

    // ---- weighted block moments of bootstrap 0 (later bootstraps: inside the DMMA loop of their predecessor)
    if constexpr (MD) {
        batch_scales(0u);
    } else {
    mbar_wait(wfull + 0, 0u);
    {
        const volatile double* ws = wring + q;
        double m1 = 0.0, m2 = 0.0;
        int cell = 0;
#pragma unroll
        for (int s = 0; s < NKS; ++s) {
            if (s < a.ks_unit) {                                  // (unit cells are not standardised: no moments)
                const double wx = ws[4 * s] * x[s];
                m1 += wx;
                m2 = fma(wx, x[s], m2);
            }
            if ((a.cend[s >> 5] >> (s & 31)) & 1u) {              // warp-uniform: last k-step of a cell
                m1 += __shfl_xor_sync(0xffffffffu, m1, 1);
                m2 += __shfl_xor_sync(0xffffffffu, m2, 1);
                m1 += __shfl_xor_sync(0xffffffffu, m1, 2);
                m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
                if (q == 0) { mt[(cell * 8 + vr) * 2] = m1; mt[(cell * 8 + vr) * 2 + 1] = m2; }
                ++cell;
                m1 = m2 = 0.0;
            }
        }
    }
    scales();
    }
    if ((warp >> 2) & 1) __nanosleep((unsigned)(NKS * NBLK * 8));     // stagger the warps of a sub-partition (see boot.cu)

    int slot = 0, prev_slot = 0;
    uint32_t phase = 0, prev_phase = 0;
    for (int bb = 0; bb < RD_NBT; ++bb) {
        if (tid == 0 && bb > 0) {
            // every warp has finished iteration bb-1: its coefficient slot is free, and so are the weight slots of
            // bootstraps <= bb (the weights of bootstrap j are read during iteration j-1); weights 0..3 were issued
            // in the prologue, bootstrap bb+3 goes into the slot bootstrap bb-1 occupied
            mbar_wait(empty + prev_slot, prev_phase);
            const int nx = bb - 1 + a.nstage;
            if (nx < RD_NBT) issue(nx, prev_slot);
            if constexpr (MD) {
                // every warp has finished iteration 8g, so it has also read the weights of batch g (before that iteration)
                if ((bb & 7) == 1 && 8 * (bb / 8 + 1) < RD_NBT) issue_w8(bb / 8 + 1);
            } else {
                if (bb + WSLOTS - 1 < RD_NBT) issue_w(bb + WSLOTS - 1);
            }
        }
        __syncwarp();
        const bool has_next = bb + 1 < RD_NBT;
        if constexpr (MD) {
            if ((bb & 7) == 0 && bb > 0) batch_scales((uint32_t)((bb >> 3) & 1));
        } else {
            if (has_next) mbar_wait(wfull + (bb + 1) % WSLOTS, (uint32_t)(((bb + 1) / WSLOTS) & 1));
        }
        mbar_wait(full + slot, phase);
        const volatile double* bs = ring + (size_t)slot * coef_doubles + lane;
        const volatile double* ws = wring + ((bb + 1) % WSLOTS) * w_doubles + q;     // (stale but harmless when !has_next)

        // ---- VS = sum_c sc_c(v) X_c^T Q_c of bootstrap bb on the tensor cores.  The (cell, voxel) scale multiplies
        //      the A fragment (a lane's element x[s] belongs to voxel `vr` and to the cell of k-step s), so the NBLK
        //      accumulator chains run through the whole bootstrap without being drained and restarted at every cell
        //      boundary (the first version folded sc * D per cell: a 5-deep chain, then a full DMMA-latency stall).
        //      In the shadow of the DMMAs: the weighted block moments of bootstrap bb+1 on the same resident fragments.
        double vs[NBLK][2], m1 = 0.0, m2 = 0.0;
#pragma unroll
        for (int j = 0; j < NBLK; ++j) vs[j][0] = vs[j][1] = 0.0;
        if constexpr (MD) {
            const double* scb = sct + (bb & 7) * nstd8 + vr;      // this bootstrap's scales of my voxel, one per cell
            int cell = 0;
            double sc = a.nstd > 0 ? scb[0] : 1.0;
#pragma unroll
            for (int s = 0; s < NKS; ++s) {
                const double xs = x[s] * sc;
#pragma unroll
                for (int j = 0; j < NBLK; ++j) {
                    const double b = bs[(s * NBLK + j) * 32];
                    dmma884(vs[j][0], vs[j][1], xs, b);
                }
                if ((a.cend[s >> 5] >> (s & 31)) & 1u) {          // warp-uniform: last k-step of a cell
                    ++cell;
                    sc = cell < a.nstd ? scb[cell * 8] : 1.0;     // unit cells: plain rows; padding k-steps: x = 0
                }
            }
        } else {
            int cell = 0;
            double sc = sct[vr];
#pragma unroll
            for (int s = 0; s < NKS; ++s) {
                const double xs = x[s] * sc;
#pragma unroll
                for (int j = 0; j < NBLK; ++j) {
                    const double b = bs[(s * NBLK + j) * 32];
                    dmma884(vs[j][0], vs[j][1], xs, b);
                }
                if (s < a.ks_unit) {                              // warp-uniform; the task rows of a multiblock pass
                    const double wx = ws[4 * s] * x[s];           // (two thirds of its k-steps) skip the moment work
                    m1 += wx;
                    m2 = fma(wx, x[s], m2);
                }
                if ((a.cend[s >> 5] >> (s & 31)) & 1u) {          // warp-uniform: last k-step of a cell
                    m1 += __shfl_xor_sync(0xffffffffu, m1, 1);
                    m2 += __shfl_xor_sync(0xffffffffu, m2, 1);
                    m1 += __shfl_xor_sync(0xffffffffu, m1, 2);
                    m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
                    if (q == 0) { mt[(cell * 8 + vr) * 2] = m1; mt[(cell * 8 + vr) * 2 + 1] = m2; }
                    ++cell;
                    m1 = m2 = 0.0;
                    sc = cell < a.ncell ? sct[cell * 8 + vr] : 0.0;   // (padding k-steps after the last cell: x = 0)
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + slot);

        // ---- fold: moments, squared column norms (this warp's 8 voxels), transposed VS for the latent GEMM, and the
        //      exported salience (before the pivot is subtracted: the reference's permuted^T U)
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 8 * j + 2 * q + e;
                const double val = ok ? vs[j][e] : 0.0;
                if constexpr (ONLY) {
                    if (ok && c < a.kc) a.VS[((size_t)(bb + bofs) * (a.p - a.v0) + (v - a.v0)) * a.Kfull + a.k0 + c] = val;
                    continue;
                }
                const double dd = val - myp[(2 * j + e) * RD_THREADS];
                my1[(2 * j + e) * RD_THREADS] += dd;
                my2[(2 * j + e) * RD_THREADS] = fma(dd, dd, my2[(2 * j + e) * RD_THREADS]);
                double n2 = val * val;
                n2 += __shfl_xor_sync(0xffffffffu, n2, 4);
                n2 += __shfl_xor_sync(0xffffffffu, n2, 8);
                n2 += __shfl_xor_sync(0xffffffffu, n2, 16);
                if (vr == 0)
                    a.Npart[((size_t)bb * (8 * NBLK) + c) * ((size_t)gridDim.x * nwarps) + blockIdx.x * nwarps + warp] = n2;
                if (a.VSt && ok) a.VSt[((size_t)bb * (8 * NBLK) + c) * a.p + v] = val;
                if constexpr (EXPORT)
                    if (ok && c < a.kc) a.VS[((size_t)bb * a.p + v) * a.Kfull + a.k0 + c] = val;
            }
        if constexpr (!MD)
            if (has_next) scales();                               // scales of bootstrap bb+1 from its moments
        prev_slot = slot; prev_phase = phase;
        if (++slot == a.nstage) { slot = 0; phase ^= 1u; }
    }
    if (!ONLY && ok) {
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 8 * j + 2 * q + e;
                if (c < a.kc) {
                    a.sum[v * a.Kfull + a.k0 + c] = my1[(2 * j + e) * RD_THREADS];
                    a.sumsq[v * a.Kfull + a.k0 + c] = my2[(2 * j + e) * RD_THREADS];
                }
            }
    }
#undef RD_NBT
}

// nrm2[b0 + bb][k0 + c] = sum over the (tile, warp) partials: one warp per output, lanes stride over the contiguous
// partials, fixed-order shuffle tree (deterministic)
__global__ void rd_norm_reduce_kernel(const double* __restrict__ Npart, int nparts, int nbt, int kcp, int kc, int K, int k0,
                                      double* __restrict__ nrm2) {
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (o >= nbt * kc) return;
    const int bb = o / kc, c = o % kc;
    const double* src = Npart + ((size_t)bb * kcp + c) * nparts;
    double s = 0.0;
    for (int t = lane; t < nparts; t += 32) s += src[t];
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) s += __shfl_xor_sync(0xffffffffu, s, w);
    if (lane == 0) nrm2[(size_t)bb * K + k0 + c] = s;
}

// ---------------------------------------------------------------------------------------------------------
// C[NA x NB] = A[NA x p] . B[NB x p]^T, both row-major (voxels contiguous), FP64 DMMA, split over voxel chunks.
// Same tiling as the Gram kernel (64 x 64 output tiles, 32-voxel stages, 3-stage cp.async ring).
constexpr int GN_T = 64, GN_KC = 32, GN_STR = GN_KC + 4, GN_STAGES = 3, GN_THREADS = 128;

template <int VEC>   // doubles per cp.async (2 when every row start is 16-byte aligned, else 1)
__global__ void __launch_bounds__(GN_THREADS) gemm_nt_partial_kernel(const double* __restrict__ A, int NA, long long lda,
                                                                    const double* __restrict__ A2, int na1, long long lda2,
                                                                    const double* __restrict__ B, int NB, long long ldb,
                                                                    long long p, long long chunk, int ntb,
                                                                    double* __restrict__ part) {
    extern __shared__ __align__(16) double sm[];
    const int ti = blockIdx.x / ntb, tj = blockIdx.x % ntb;
    const long long v0 = (long long)blockIdx.y * chunk;
    const long long v1 = min(p, v0 + chunk);
    const int nst = (int)((v1 - v0 + GN_KC - 1) / GN_KC);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wi = (warp >> 1) * 32, wj = (warp & 1) * 32;
    double* As = sm;
    double* Bs = sm + GN_STAGES * GN_T * GN_STR;
    auto load_stage = [&](int st, int kt) {
        const long long vb = v0 + (long long)kt * GN_KC;
        constexpr int CH = GN_KC / VEC;
        for (int c = tid; c < GN_T * CH; c += GN_THREADS) {
            const int r = c / CH, cc = (c % CH) * VEC;
            const long long vv = vb + cc;
            long long left = v1 - vv; if (left < 0) left = 0; if (left > VEC) left = VEC;
            {
                const int row = ti * GN_T + r;
                const int nb = row < NA ? (int)left * 8 : 0;
                const double* rp = row < na1 ? A + (long long)row * lda : A2 + (long long)(row - na1) * lda2;
                cp_async_zfill<VEC * 8>(As + (st * GN_T + r) * GN_STR + cc, nb ? rp + vv : A, nb);
            }
            {
                const int row = tj * GN_T + r;
                const int nb = row < NB ? (int)left * 8 : 0;
                cp_async_zfill<VEC * 8>(Bs + (st * GN_T + r) * GN_STR + cc, nb ? B + (long long)row * ldb + vv : B, nb);
            }
        }
    };
    double acc[4][4][2];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
#pragma unroll
    for (int s = 0; s < GN_STAGES - 1; ++s) {
        if (s < nst) load_stage(s, s);
        cp_async_commit();
    }
    const int fr = lane >> 2, fk = lane & 3;
    for (int kt = 0; kt < nst; ++kt) {
        cp_async_wait<GN_STAGES - 2>();
        __syncthreads();
        {
            const int nk = kt + GN_STAGES - 1;
            if (nk < nst) load_stage(nk % GN_STAGES, nk);
            cp_async_commit();
        }
        const int st = kt % GN_STAGES;
        const double* a_base = As + (st * GN_T + wi + fr) * GN_STR + fk;
        const double* b_base = Bs + (st * GN_T + wj + fr) * GN_STR + fk;
#pragma unroll
        for (int ks = 0; ks < GN_KC / 4; ++ks) {
            double af[4], bf[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) { af[t] = a_base[t * 8 * GN_STR + ks * 4]; bf[t] = b_base[t * 8 * GN_STR + ks * 4]; }
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) dmma884(acc[x][y][0], acc[x][y][1], af[x], bf[y]);
        }
    }
    cp_async_wait<0>();
    double* out = part + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * (GN_T * GN_T);
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int r = wi + x * 8 + fr, c = wj + y * 8 + 2 * fk;
            *reinterpret_cast<double2*>(out + r * GN_T + c) = make_double2(acc[x][y][0], acc[x][y][1]);
        }
}

// T[b0 + bb][i][k0 + c] = sum over voxel chunks of C[i][bb*kcp + c]
__global__ void rd_latent_reduce_kernel(const double* __restrict__ part, int ntiles, int ntb, int nsplit, int N, int nbt,
                                        int kcp, int kc, int K, int k0, double* __restrict__ T) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)nbt * N * kc) return;
    const int c = (int)(i % kc), row = (int)((i / kc) % N), bb = (int)(i / ((long long)kc * N));
    const int col = bb * kcp + c;
    const int tile = (row / GN_T) * ntb + col / GN_T, e = (row % GN_T) * GN_T + col % GN_T;
    double s = 0.0;
    for (int sp = 0; sp < nsplit; ++sp) s += part[((long long)sp * ntiles + tile) * (GN_T * GN_T) + e];
    T[((size_t)bb * N + row) * K + k0 + c] = s;
}

struct RdLayout {
    size_t off_krow, off_celln, off_pack, off_wpack, off_vst, off_npart, off_gpart, total;
    int ntile, nta, ntb, nsplit, nwarps;
    long long chunk;
};

// Warps (= groups of 8 voxels) per CTA actually launched.  Fewer warps than the kernel's bucket would fill the waves of
// SMs more evenly (50 000 voxels are 391 CTAs of 16 warps = 2.64 waves, 569 CTAs of 11 warps = 3.84), but the kernel
// is latency-bound, not pipe-bound: with 11 instead of 16 (5 instead of 8) warps per SM it ran 8 % (44 %) SLOWER
// (cfg 2: 21.5 -> 23.2 ms, cfg 4: 55.6 -> 80.0 ms per analysis).  The full bucket is used.
static int rd_balanced_warps(int maxw, int64_t) { return maxw; }

static RdLayout rd_layout(const RdPlan& r, int N, int64_t p, int nbt, bool want_t) {
    RdLayout L;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o = 0;
    L.off_krow = o; o = al(o + (size_t)r.nks * 4 * sizeof(int));
    L.off_celln = o; o = al(o + 16 * sizeof(double));
    L.off_pack = o; o = al(o + (size_t)nbt * r.npass * r.stage_doubles * sizeof(double));
    L.off_wpack = o; o = al(o + (size_t)cdiv(nbt, 8) * r.nks * 32 * sizeof(double));
    L.nwarps = rd_balanced_warps(r.warps, p);
    L.ntile = (int)cdiv(p, L.nwarps * 8);
    L.off_vst = o; if (want_t) o = al(o + (size_t)nbt * r.kcp * p * sizeof(double));
    L.off_npart = o; o = al(o + (size_t)L.ntile * L.nwarps * nbt * r.kcp * sizeof(double));
    L.nta = (int)cdiv(N, GN_T); L.ntb = (int)cdiv((int64_t)nbt * r.kcp, GN_T);
    const int64_t nk = cdiv(p, GN_KC);
    const int64_t max_ns = nk / 8 > 0 ? nk / 8 : 1;
    // voxel splits: the grid (output tiles x splits) should fill whole waves of the 2 CTAs an SM holds.  The first version
    // took ceil(4 SMs / tiles) splits: 70 tiles x 9 splits = 630 CTAs = 2.13 waves of 296 at the cfg-2 shape, i.e. a third
    // wave for 13 % of the CTAs (13.8 ms = 0.59 of the DGEMM peak).  Now: the split count with the best wave efficiency,
    // the smallest one among equals (fewer partial tiles to reduce).
    const int64_t tiles = (int64_t)L.nta * L.ntb, slots = 2LL * num_sms();
    int64_t ns = 1;
    double best = -1.0;
    for (int64_t c = 1; c <= max_ns && c <= 64; ++c) {
        const double waves = (double)(tiles * c) / (double)slots;
        const double eff = waves / ceil(waves);
        if (eff > best + 0.02) { best = eff; ns = c; }
    }
    L.chunk = cdiv(nk, ns) * GN_KC;
    L.nsplit = (int)cdiv(p, L.chunk);
    L.off_gpart = o; if (want_t) o = al(o + (size_t)L.nsplit * L.nta * L.ntb * GN_T * GN_T * sizeof(double));
    L.total = o;
    return L;
}

template <int NKS, int NBLK, int W, bool MD, bool EXPORT, bool ONLY>
static int launch_vs_kernel(const RdPlan& r, const RdArgs& a, dim3 grid, cudaStream_t st) {
    PLSB_CUDA(cudaFuncSetAttribute(rb_vs_kernel<NKS, NBLK, W, MD, EXPORT, ONLY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)r.smem_bytes));
    rb_vs_kernel<NKS, NBLK, W, MD, EXPORT, ONLY><<<grid, a.nwarps * 32, r.smem_bytes, st>>>(a);
    PLSB_LAUNCH_CHECK("rb_vs_kernel");
    return PLSB200_OK;
}
// only: the export-only instantiation (plsb200_rb_salience_dmma_f64), grid = (voxel tiles, bootstrap slices)
template <int NKS, int NBLK, int W, bool MD>
static int launch_vs_md(const RdPlan& r, const RdArgs& a, dim3 grid, bool only, cudaStream_t st) {
    if (only) return launch_vs_kernel<NKS, NBLK, W, MD, true, true>(r, a, grid, st);
    return a.VS ? launch_vs_kernel<NKS, NBLK, W, MD, true, false>(r, a, grid, st) : launch_vs_kernel<NKS, NBLK, W, MD, false, false>(r, a, grid, st);
}
template <int NKS, int NBLK, int W>
static int launch_vs(const RdPlan& r, const RdArgs& a, dim3 grid, bool only, cudaStream_t st) {
    if constexpr (W == 16) {
        if (r.md) return launch_vs_md<NKS, NBLK, W, true>(r, a, grid, only, st);
    }
    return launch_vs_md<NKS, NBLK, W, false>(r, a, grid, only, st);
}

template <int NBLK>
static int dispatch_vs(const RdPlan& r, const RdArgs& a, dim3 grid, bool only, cudaStream_t st) {
    if (r.warps == 16) {
        switch (r.nks) {
#define PLSB_CASE(n) case n: return launch_vs<n, NBLK, 16>(r, a, grid, only, st);
            PLSB_CASE(4) PLSB_CASE(8) PLSB_CASE(12) PLSB_CASE(16) PLSB_CASE(20) PLSB_CASE(24) PLSB_CASE(28) PLSB_CASE(32)
#undef PLSB_CASE
            default: break;
        }
    } else {
        switch (r.nks) {
#define PLSB_CASE(n) case n: return launch_vs<n, NBLK, 8>(r, a, grid, only, st);
            PLSB_CASE(36) PLSB_CASE(40) PLSB_CASE(44) PLSB_CASE(48) PLSB_CASE(52) PLSB_CASE(56) PLSB_CASE(60) PLSB_CASE(64) PLSB_CASE(68) PLSB_CASE(72)
            PLSB_CASE(76) PLSB_CASE(80) PLSB_CASE(84) PLSB_CASE(88) PLSB_CASE(92) PLSB_CASE(96)
#undef PLSB_CASE
            default: break;
        }
    }
    set_err("rb_boot_dmma_f64: no kernel for %d k-steps x %d column blocks", r.nks, NBLK);
    return PLSB200_EUNSUPPORTED;
}

}  // namespace plsb

using namespace plsb;

// cell_start_host: ncell+1 row offsets in HOST memory.  Returns 0 when the design is outside what the DMMA path is
// built for (more than 96 k-steps of 4 rows after padding every cell to a multiple of 4): use plsb200_rb_boot_f64.
extern "C" size_t plsb200_rb_boot_dmma_f64_workspace(int N, int64_t p, int K, int nbt, const int32_t* cell_start_host,
                                                     int ncell, int unit_cells, int want_t) {
    RdPlan r;
    if (!cell_start_host || p < 1 || nbt < 1 || !rd_plan(N, K, cell_start_host, ncell, unit_cells, r)) return 0;
    return rd_layout(r, N, p, nbt, want_t != 0).total;
}

extern "C" int plsb200_rb_boot_dmma_vs_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                                           const double* Q, const double* W, int K, int b0, int nbt, const int32_t* cell_start_host, int ncell, int unit_cells,
                                           const double* pivot, double* sum, double* sumsq, double* T, double* nrm2, double* VS,
                                           void* workspace, size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(Xc && Q && cell_start_host && sum && sumsq && nrm2 && workspace, "rb_boot_dmma_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && K > 0 && nbt > 0 && ncell > 0, "rb_boot_dmma_f64: bad shape");
    if (Xc2 == nullptr) { n1 = N; ld2 = p; }
    PLSB_CHECK_ARG(n1 > 0 && n1 <= N && ld2 >= p, "rb_boot_dmma_f64: bad row split");
    RdPlan r;
    if (!rd_plan(N, K, cell_start_host, ncell, unit_cells, r)) {
        set_err("rb_boot_dmma_f64: design not supported (N=%d, %d cells): use rb_boot_f64", N, ncell);
        return PLSB200_EUNSUPPORTED;
    }
    const bool want_t = T != nullptr;
    const RdLayout L = rd_layout(r, N, p, nbt, want_t);
    if (workspace_bytes < L.total) {
        set_err("rb_boot_dmma_f64: workspace %zu < %zu bytes", workspace_bytes, L.total);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    int* d_krow = (int*)(ws + L.off_krow);
    double* d_celln = (double*)(ws + L.off_celln);
    double* d_pack = (double*)(ws + L.off_pack);
    double* d_vst = want_t ? (double*)(ws + L.off_vst) : nullptr;
    double* d_npart = (double*)(ws + L.off_npart);
    double* d_gpart = (double*)(ws + L.off_gpart);
    PLSB_CUDA(cudaMemcpyAsync(d_krow, r.krow, (size_t)r.nks * 4 * sizeof(int), cudaMemcpyHostToDevice, st));
    PLSB_CUDA(cudaMemcpyAsync(d_celln, r.celln, 16 * sizeof(double), cudaMemcpyHostToDevice, st));
    rd_pack_kernel<<<dim3(nbt, r.npass), 256, 0, st>>>(Q, W, N, K, b0, d_krow, r.nks, r.nblk, r.npass, d_pack);
    PLSB_LAUNCH_CHECK("rd_pack_kernel");
    double* d_wpack = (double*)(ws + L.off_wpack);
    if (r.md) {
        rd_wpack_kernel<<<(unsigned)cdiv(nbt, 8), 256, 0, st>>>(W, N, b0, nbt, d_krow, r.nks, d_wpack);
        PLSB_LAUNCH_CHECK("rd_wpack_kernel");
    }
    for (int pass = 0; pass < r.npass; ++pass) {
        RdArgs a;
        a.Xc = Xc; a.Xc2 = Xc2; a.n1 = n1; a.ld2 = ld2; a.pack = d_pack; a.wpack = d_wpack; a.nstd = r.nstd; a.pivot = pivot; a.krow = d_krow; a.celln = d_celln; a.sum = sum; a.sumsq = sumsq;
        a.VSt = d_vst; a.VS = VS ? VS + (size_t)b0 * p * K : nullptr; a.Npart = d_npart; a.p = p; a.Kfull = K; a.k0 = pass * r.kcp;
        a.kc = K - a.k0 < r.kcp ? K - a.k0 : r.kcp;
        a.nbt = nbt; a.npass = r.npass; a.pass = pass; a.nstage = r.nstage; a.ncell = r.ncell; a.nwarps = L.nwarps; a.ks_unit = r.ks_unit;
        a.cend[0] = r.cend[0]; a.cend[1] = r.cend[1]; a.cend[2] = r.cend[2];
        a.v0 = 0; a.ld1 = p; a.bslice = nbt;
        int rc;
        switch (r.nblk) {
            case 1: rc = dispatch_vs<1>(r, a, L.ntile, false, st); break;
            case 2: rc = dispatch_vs<2>(r, a, L.ntile, false, st); break;
            default: rc = dispatch_vs<3>(r, a, L.ntile, false, st); break;
        }
        if (rc != PLSB200_OK) return rc;
        rd_norm_reduce_kernel<<<(unsigned)cdiv((int64_t)nbt * a.kc * 32, 256), 256, 0, st>>>(
            d_npart, L.ntile * L.nwarps, nbt, r.kcp, a.kc, K, a.k0, nrm2 + (size_t)b0 * K);
        PLSB_LAUNCH_CHECK("rd_norm_reduce_kernel");
        if (want_t) {
            const size_t smem = (size_t)2 * GN_STAGES * GN_T * GN_STR * sizeof(double);
            dim3 grid((unsigned)(L.nta * L.ntb), (unsigned)L.nsplit);
            const bool vec2 = (p % 2 == 0) && ((reinterpret_cast<uintptr_t>(Xc) & 15) == 0) &&
                              ((reinterpret_cast<uintptr_t>(d_vst) & 15) == 0) &&
                              (n1 == N || (((reinterpret_cast<uintptr_t>(Xc2) & 15) == 0) && ld2 % 2 == 0));
            if (vec2) {
                PLSB_CUDA(cudaFuncSetAttribute(gemm_nt_partial_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                gemm_nt_partial_kernel<2><<<grid, GN_THREADS, smem, st>>>(Xc, N, p, Xc2, n1, ld2, d_vst, nbt * r.kcp, p, p, L.chunk, L.ntb, d_gpart);
            } else {
                PLSB_CUDA(cudaFuncSetAttribute(gemm_nt_partial_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                gemm_nt_partial_kernel<1><<<grid, GN_THREADS, smem, st>>>(Xc, N, p, Xc2, n1, ld2, d_vst, nbt * r.kcp, p, p, L.chunk, L.ntb, d_gpart);
            }
            PLSB_LAUNCH_CHECK("gemm_nt_partial_kernel");
            const long long n = (long long)nbt * N * a.kc;
            rd_latent_reduce_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(d_gpart, L.nta * L.ntb, L.ntb, L.nsplit, N, nbt,
                                                                             r.kcp, a.kc, K, a.k0, T + (size_t)b0 * N * K);
            PLSB_LAUNCH_CHECK("rd_latent_reduce_kernel");
        }
    }
    return PLSB200_OK;
}

extern "C" int plsb200_rb_boot_dmma_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                                        const double* Q, const double* W, int K, int b0, int nbt, const int32_t* cell_start_host, int ncell, int unit_cells,
                                        const double* pivot, double* sum, double* sumsq, double* T, double* nrm2,
                                        void* workspace, size_t workspace_bytes, void* stream) {
    return plsb200_rb_boot_dmma_vs_f64(Xc, N, p, Xc2, n1, ld2, Q, W, K, b0, nbt, cell_start_host, ncell, unit_cells, pivot,
                                       sum, sumsq, T, nrm2, nullptr, workspace, workspace_bytes, stream);
}

// ---- export-only pass over a voxel window (right_sv_sampled in voxel chunks) -------------------------------------------
// Workspace: block rows, block sizes and the packed coefficients of all nbt bootstraps (rd_pack_kernel, and the MD weight
// fragments), filled once by plsb200_rb_salience_dmma_pack_f64 and read by every window.
struct RsLayout {
    size_t off_krow, off_celln, off_pack, off_wpack, total;
};

static RsLayout rs_layout(const RdPlan& r, int nbt) {
    RsLayout L;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o = 0;
    L.off_krow = o; o = al(o + (size_t)r.nks * 4 * sizeof(int));
    L.off_celln = o; o = al(o + 16 * sizeof(double));
    L.off_pack = o; o = al(o + (size_t)nbt * r.npass * r.stage_doubles * sizeof(double));
    L.off_wpack = o; o = al(o + (size_t)cdiv(nbt, 8) * r.nks * 32 * sizeof(double));
    L.total = o;
    return L;
}

extern "C" size_t plsb200_rb_salience_dmma_f64_workspace(int N, int K, int nbt, const int32_t* cell_start_host, int ncell,
                                                        int unit_cells) {
    RdPlan r;
    if (!cell_start_host || nbt < 1 || !rd_plan(N, K, cell_start_host, ncell, unit_cells, r)) return 0;
    return rs_layout(r, nbt).total;
}

extern "C" int plsb200_rb_salience_dmma_pack_f64(const double* Q, const double* W, int N, int K, int nbt,
                                                 const int32_t* cell_start_host, int ncell, int unit_cells, void* workspace,
                                                 size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(Q && W && cell_start_host && workspace, "rb_salience_dmma_pack_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && K > 0 && nbt > 0 && ncell > 0, "rb_salience_dmma_pack_f64: bad shape");
    RdPlan r;
    if (!rd_plan(N, K, cell_start_host, ncell, unit_cells, r)) {
        set_err("rb_salience_dmma_pack_f64: design not supported (N=%d, %d cells): use rb_salience_f64", N, ncell);
        return PLSB200_EUNSUPPORTED;
    }
    const RsLayout L = rs_layout(r, nbt);
    if (workspace_bytes < L.total) {
        set_err("rb_salience_dmma_pack_f64: workspace %zu < %zu bytes", workspace_bytes, L.total);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    int* d_krow = (int*)(ws + L.off_krow);
    PLSB_CUDA(cudaMemcpyAsync(d_krow, r.krow, (size_t)r.nks * 4 * sizeof(int), cudaMemcpyHostToDevice, st));
    PLSB_CUDA(cudaMemcpyAsync(ws + L.off_celln, r.celln, 16 * sizeof(double), cudaMemcpyHostToDevice, st));
    rd_pack_kernel<<<dim3(nbt, r.npass), 256, 0, st>>>(Q, W, N, K, 0, d_krow, r.nks, r.nblk, r.npass, (double*)(ws + L.off_pack));
    PLSB_LAUNCH_CHECK("rd_pack_kernel");
    if (r.md) {
        rd_wpack_kernel<<<(unsigned)cdiv(nbt, 8), 256, 0, st>>>(W, N, 0, nbt, d_krow, r.nks, (double*)(ws + L.off_wpack));
        PLSB_LAUNCH_CHECK("rd_wpack_kernel");
    }
    return PLSB200_OK;
}

extern "C" int plsb200_rb_salience_dmma_f64(const double* Xc, int N, int64_t ld1, const double* Xc2, int n1, int64_t ld2,
                                            int64_t v0, int64_t v1, int K, int nbt, const int32_t* cell_start_host,
                                            int ncell, int unit_cells, double* VS, const void* workspace,
                                            size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(Xc && cell_start_host && VS && workspace, "rb_salience_dmma_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && K > 0 && nbt > 0 && ncell > 0 && v0 >= 0 && v1 > v0 && ld1 >= v1,
                   "rb_salience_dmma_f64: bad shape");
    if (Xc2 == nullptr) { n1 = N; ld2 = ld1; }
    PLSB_CHECK_ARG(n1 > 0 && n1 <= N && ld2 >= v1, "rb_salience_dmma_f64: bad row split");
    RdPlan r;
    if (!rd_plan(N, K, cell_start_host, ncell, unit_cells, r)) {
        set_err("rb_salience_dmma_f64: design not supported (N=%d, %d cells): use rb_salience_f64", N, ncell);
        return PLSB200_EUNSUPPORTED;
    }
    const RsLayout L = rs_layout(r, nbt);
    if (workspace_bytes < L.total) {
        set_err("rb_salience_dmma_f64: workspace %zu < %zu bytes", workspace_bytes, L.total);
        return PLSB200_EWORKSPACE;
    }
    const char* ws = (const char*)workspace;
    const int nwarps = rd_balanced_warps(r.warps, v1 - v0);
    const int ntile = (int)cdiv(v1 - v0, nwarps * 8);
    // bootstrap slices: a window of a few thousand voxels is a few dozen tiles, too few CTAs for the SMs on their own
    // (one CTA per SM); aim for about four CTAs per SM, in slices of whole batches of 8 bootstraps
    const int nbatch = (int)cdiv(nbt, 8);
    int nsl = (int)cdiv(4LL * num_sms(), ntile);
    if (nsl > nbatch) nsl = nbatch;
    if (nsl > 65535) nsl = 65535;
    const int bslice = (int)cdiv(nbatch, nsl) * 8;
    nsl = (int)cdiv(nbt, bslice);
    for (int pass = 0; pass < r.npass; ++pass) {
        RdArgs a{};
        a.Xc = Xc; a.Xc2 = Xc2; a.n1 = n1; a.ld2 = ld2; a.pack = (const double*)(ws + L.off_pack);
        a.wpack = r.md ? (const double*)(ws + L.off_wpack) : nullptr; a.nstd = r.nstd; a.pivot = nullptr;
        a.krow = (const int*)(ws + L.off_krow); a.celln = (const double*)(ws + L.off_celln); a.sum = a.sumsq = nullptr;
        a.VSt = nullptr; a.VS = VS; a.Npart = nullptr; a.p = v1; a.Kfull = K; a.k0 = pass * r.kcp;
        a.kc = K - a.k0 < r.kcp ? K - a.k0 : r.kcp;
        a.nbt = nbt; a.npass = r.npass; a.pass = pass; a.nstage = r.nstage; a.ncell = r.ncell; a.nwarps = nwarps; a.ks_unit = r.ks_unit;
        a.cend[0] = r.cend[0]; a.cend[1] = r.cend[1]; a.cend[2] = r.cend[2];
        a.v0 = v0; a.ld1 = ld1; a.bslice = bslice;
        const dim3 grid((unsigned)ntile, (unsigned)nsl);
        cudaStream_t st = (cudaStream_t)stream;
        int rc;
        switch (r.nblk) {
            case 1: rc = dispatch_vs<1>(r, a, grid, true, st); break;
            case 2: rc = dispatch_vs<2>(r, a, grid, true, st); break;
            default: rc = dispatch_vs<3>(r, a, grid, true, st); break;
        }
        if (rc != PLSB200_OK) return rc;
    }
    return PLSB200_OK;
}
