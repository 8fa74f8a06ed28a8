// K5: behaviour-PLS (rb / csb) resampling kernels.
//
// Reference: the cross-block matrix is the stack of per-(group, condition) correlation blocks
// R_c = Yz_c^T Xz_c  (class_functions.py:185-247: z-score X and Y inside every block, ddof 0, / sqrt(n),
// nan_to_num).  Permutations permute Y only (bootstrap_permutation.py:337-340, 395-396); bootstraps
// resample X and Y rows together (:557-561, 613), so the per-voxel standard deviation of every block
// changes with the draw and X has to be streamed once per bootstrap batch.
//
// With Xc = X minus its block means (z-scoring is shift invariant) and, per resample, the small
// coefficient matrix  Q[i, k] = sum_j a_ij U[(c(i), j), k]  (a = z-scored resampled Y, summed over the
// copies of row i), the projected cross-block matrix is
//     VS[v, k] = sum_c  Q_c^T Xc_c [v, k] / (sd_c(v) sqrt(n_c)),   sd_c(v)^2 = sum_i w_i Xc[i,v]^2 - (sum_i w_i Xc[i,v])^2
// (the mean term drops because sum_i a_ij = 0).  Permutations keep sd fixed, so they collapse to
// N-space through Gz = Z Z^T, Z = block-z-scored X.
#include "common.cuh"

namespace plsb {

// ------------------------------------------------------------------------------------------------
// One thread per voxel: block means and population std (two-pass), writes Xc (centred) and
// Z = Xc / (sd sqrt(n)) (0 where sd == 0, the nan_to_num of class_functions.py:237).
__global__ void __launch_bounds__(256) cell_standardize_kernel(const double* __restrict__ X, int N, long long p,
                                                              long long ldx, const int32_t* __restrict__ cell_start,
                                                              int ncell, double* __restrict__ Xc,
                                                              double* __restrict__ Z) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= p) return;
    for (int c = 0; c < ncell; ++c) {
        const int s = cell_start[c], e = cell_start[c + 1], n = e - s;
        double m = 0.0;
        for (int i = s; i < e; ++i) m += X[(long long)i * ldx + v];
        m /= n;
        double q = 0.0;
        for (int i = s; i < e; ++i) { const double d = X[(long long)i * ldx + v] - m; q = fma(d, d, q); }
        const double sd = sqrt(q / n);
        const double sc = sd > 0.0 ? 1.0 / (sd * sqrt((double)n)) : 0.0;
        for (int i = s; i < e; ++i) {
            const double d = X[(long long)i * ldx + v] - m;
            Xc[(long long)i * p + v] = d;
            if (Z) Z[(long long)i * p + v] = d * sc;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Per-resample coefficient matrix.  One CTA per resample.
//   Ynew = Y[idx]; Yz = block z-score(Ynew) / sqrt(n) (0 where sd == 0)
//   scatter == 0 (permutation: X rows stay put):  Q[i, k] = sum_j Yz[i, j] U[(c(i), j), k]
//   scatter == 1 (bootstrap: X rows are gathered by the same idx): Q[o, k] = sum_{i: idx[i] = o} (same), and
//                W[o] = count(o) / n_c, the multiplicity weights of the resampled block moments.
__global__ void __launch_bounds__(256) rb_coef_kernel(const double* __restrict__ Y, int N, int nb,
                                                     const int32_t* __restrict__ idx,
                                                     const int32_t* __restrict__ cell_start, int ncell,
                                                     const double* __restrict__ U, int Kc, int scatter,
                                                     double* __restrict__ Q, double* __restrict__ W,
                                                     double* __restrict__ Yz_out) {
    extern __shared__ __align__(16) double smr[];
    double* Yz = smr;                         // [N][nb]
    double* mu = Yz + (size_t)N * nb;         // [ncell*nb]
    double* isd = mu + (size_t)ncell * nb;    // [ncell*nb]
    int* ids = reinterpret_cast<int*>(isd + (size_t)ncell * nb);   // [N]
    int* cid = ids + N;                                            // [N]
    const int r = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < N; i += nt) ids[i] = idx ? idx[(size_t)r * N + i] : i;
    for (int c = tid; c < ncell; c += nt)
        for (int i = cell_start[c]; i < cell_start[c + 1]; ++i) cid[i] = c;
    __syncthreads();
    for (int i = tid; i < N * nb; i += nt) Yz[i] = Y[(size_t)ids[i / nb] * nb + i % nb];
    __syncthreads();
    for (int o = tid; o < ncell * nb; o += nt) {
        const int c = o / nb, j = o % nb, s = cell_start[c], e = cell_start[c + 1], n = e - s;
        double m = 0.0;
        for (int i = s; i < e; ++i) m += Yz[i * nb + j];
        m /= n;
        double q = 0.0;
        for (int i = s; i < e; ++i) { const double d = Yz[i * nb + j] - m; q = fma(d, d, q); }
        const double sd = sqrt(q / n);
        mu[o] = m;
        isd[o] = sd > 0.0 ? 1.0 / (sd * sqrt((double)n)) : 0.0;
    }
    __syncthreads();
    for (int i = tid; i < N * nb; i += nt) {
        const int c = cid[i / nb], j = i % nb;
        Yz[i] = (Yz[i] - mu[c * nb + j]) * isd[c * nb + j];
    }
    __syncthreads();
    if (Yz_out)
        for (int i = tid; i < N * nb; i += nt) Yz_out[(size_t)r * N * nb + i] = Yz[i];
    double* Qr = Q + (size_t)r * N * Kc;
    for (int o = tid; o < N * Kc; o += nt) {
        const int row = o / Kc, k = o % Kc;
        double acc = 0.0;
        if (!scatter) {
            const int c = cid[row];
            for (int j = 0; j < nb; ++j) acc = fma(Yz[row * nb + j], U[(size_t)(c * nb + j) * Kc + k], acc);
        } else {
            const int c = cid[row];
            for (int i = cell_start[c]; i < cell_start[c + 1]; ++i)       // sources live in the same block
                if (ids[i] == row)
                    for (int j = 0; j < nb; ++j) acc = fma(Yz[i * nb + j], U[(size_t)(c * nb + j) * Kc + k], acc);
        }
        Qr[o] = acc;
    }
    if (scatter && W)
        for (int row = tid; row < N; row += nt) {
            const int c = cid[row], s = cell_start[c], e = cell_start[c + 1];
            int cnt = 0;
            for (int i = s; i < e; ++i) cnt += (ids[i] == row);
            W[(size_t)r * N + row] = (double)cnt / (double)(e - s);
        }
}

// ------------------------------------------------------------------------------------------------
// Bootstrap p-space pass.  CTA = 256 voxels; loops over the bootstraps of the chunk.
//  phase 1 (thread per voxel): block moments with multiplicity weights, VS[v, k0..k0+kc), fused
//          running sum / sum of squares of (VS - pivot), VS itself into the resample-major cube when VS != NULL;
//  phase 2 (thread per (row, 4 columns)): partial T[b] = Xc[:, tile] . VS_tile  and  ||VS||^2 partials,
//          written per (tile, bootstrap) and summed over tiles in a fixed order by rb_reduce_kernel.
constexpr int RB_VT = 256;
constexpr int RB_VCH = 32;

// ONLY (with EXPORT): phase 1 alone over the voxel window [vw0, p) of a matrix whose first segment has the row stride
// ld1, storing VS[b][v - vw0][k]; no moments, norms or phase 2.  blockIdx.y takes the bootstraps [y bslice, (y+1) bslice).
template <int KC, bool EXPORT, bool ONLY = false>     // EXPORT: also store VS into the cube (instantiations without it keep their registers)
__global__ void __launch_bounds__(RB_VT) rb_boot_kernel(const double* __restrict__ Xc, int N, long long p,
                                                       const double* __restrict__ Xc2, int n1, long long ld2,
                                                       const double* __restrict__ Q, const double* __restrict__ W,
                                                       int Kq, int k0, int kc, int b0, int nbt,
                                                       const int32_t* __restrict__ cell_start, int ncell,
                                                       int unit_cells,
                                                       const double* __restrict__ pivot, int Kfull,
                                                       double* __restrict__ sum, double* __restrict__ sumsq,
                                                       double* __restrict__ Tpart, double* __restrict__ Npart,
                                                       double* __restrict__ VS, long long vw0, long long ld1,
                                                       int bslice) {
    static_assert(EXPORT || !ONLY, "ONLY is an export mode");
    extern __shared__ __align__(16) double smb[];
    double* Qs = smb;                               // [N][KC]
    double* Ws = Qs + (size_t)N * KC;               // [N]
    double* VSs = Ws + N;                           // [KC][RB_VT]
    double* Xs = VSs + (size_t)KC * RB_VT;          // [N][RB_VCH + 1]
    const int tid = threadIdx.x;
    const long long v0 = (ONLY ? vw0 : 0) + (long long)blockIdx.x * RB_VT;
    const long long v = v0 + tid;
    const bool ok = v < p;
    double s1[KC], s2[KC];
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        s1[k] = (!ONLY && ok && k < kc) ? sum[v * Kfull + k0 + k] : 0.0;
        s2[k] = (!ONLY && ok && k < kc) ? sumsq[v * Kfull + k0 + k] : 0.0;
    }
    const int bb_lo = ONLY ? (int)blockIdx.y * bslice : 0;
    const int bb_hi = ONLY ? min(nbt, bb_lo + bslice) : nbt;
    for (int bb = bb_lo; bb < bb_hi; ++bb) {
        const int b = b0 + bb;
        __syncthreads();
        for (int i = tid; i < N * KC; i += RB_VT) {
            const int row = i / KC, k = i % KC;
            Qs[i] = k < kc ? Q[((size_t)b * N + row) * Kq + k0 + k] : 0.0;
        }
        for (int i = tid; i < N; i += RB_VT) Ws[i] = W[(size_t)b * N + i];
        __syncthreads();
        // ---- phase 1
        double vs[KC];
#pragma unroll
        for (int k = 0; k < KC; ++k) vs[k] = 0.0;
        for (int c = 0; c < ncell; ++c) {
            const int s = cell_start[c], e = cell_start[c + 1];
            double m1 = 0.0, m2 = 0.0, P[KC];
#pragma unroll
            for (int k = 0; k < KC; ++k) P[k] = 0.0;
            for (int i = s; i < e; ++i) {
                // rows [0, n1) of the data matrix live in Xc, rows [n1, N) in Xc2 (n1 == N: a single matrix)
                const double x = ok ? __ldg((i < n1 ? Xc + (long long)i * (ONLY ? ld1 : p) : Xc2 + (long long)(i - n1) * ld2) + v) : 0.0;
                const double wx = Ws[i] * x;
                m1 += wx;
                m2 = fma(wx, x, m2);
                const double* q = Qs + i * KC;
#pragma unroll
                for (int k = 0; k < KC; ++k) P[k] = fma(x, q[k], P[k]);
            }
            const double var = m2 - m1 * m1;
            // a block whose resampled rows are all identical has var == 0 in exact arithmetic (nan -> 0 in
            // the reference); guard the one-pass formula with a relative threshold.  The last `unit_cells`
            // blocks are plain linear rows (multiblock task part): no standardisation.
            const double sc = c >= ncell - unit_cells
                                  ? 1.0
                                  : ((var > 1e-13 * m2 && var > 0.0) ? 1.0 / sqrt(var * (double)(e - s)) : 0.0);
#pragma unroll
            for (int k = 0; k < KC; ++k) vs[k] = fma(sc, P[k], vs[k]);
        }
        if constexpr (ONLY) {
#pragma unroll
            for (int k = 0; k < KC; ++k)
                if (ok && k < kc) VS[((size_t)bb * (p - vw0) + (v - vw0)) * Kfull + k0 + k] = vs[k];
            continue;
        }
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            if (k < kc) {
                const double d = vs[k] - ((ok && pivot) ? __ldg(pivot + v * Kfull + k0 + k) : 0.0);
                s1[k] += d;
                s2[k] = fma(d, d, s2[k]);
                if constexpr (EXPORT)
                    if (ok) VS[((size_t)bb * p + v) * Kfull + k0 + k] = vs[k];
            }
            VSs[k * RB_VT + tid] = ok ? vs[k] : 0.0;
        }
        __syncthreads();
        // ---- squared column norms of this tile (warp per column, fixed order)
        {
            const int warp = tid >> 5, lane = tid & 31;
            for (int k = warp; k < kc; k += RB_VT / 32) {
                double a = 0.0;
                for (int j = lane; j < RB_VT; j += 32) a = fma(VSs[k * RB_VT + j], VSs[k * RB_VT + j], a);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                if (lane == 0) Npart[((size_t)blockIdx.x * nbt + bb) * Kq + k0 + k] = a;
            }
        }
        // ---- phase 2: T_tile[row, k] = sum_v Xc[row, v] VS[v, k]
        const int ngrp = (kc + 3) / 4;
        double acc[8][4];      // up to 8 tasks per thread (N*ngrp <= 2048)
        const int ntask = N * ngrp;
#pragma unroll
        for (int t = 0; t < 8; ++t)
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[t][u] = 0.0;
        for (int ch = 0; ch < RB_VT / RB_VCH; ++ch) {
            __syncthreads();
            for (int i = tid; i < N * RB_VCH; i += RB_VT) {
                const int row = i / RB_VCH, j = i % RB_VCH;
                const long long vv = v0 + ch * RB_VCH + j;
                Xs[row * (RB_VCH + 1) + j] =
                    vv < p ? __ldg((row < n1 ? Xc + (long long)row * p : Xc2 + (long long)(row - n1) * ld2) + vv) : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int task = tid + t * RB_VT;
                if (task < ntask) {
                    const int row = task % N, g = task / N;
                    const double* xr = Xs + row * (RB_VCH + 1);
                    const double* vb = VSs + (size_t)(g * 4) * RB_VT + ch * RB_VCH;
                    for (int j = 0; j < RB_VCH; ++j) {
                        const double x = xr[j];
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (g * 4 + u < kc) acc[t][u] = fma(x, vb[u * RB_VT + j], acc[t][u]);
                    }
                }
            }
        }
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int task = tid + t * RB_VT;
            if (task < ntask) {
                const int row = task % N, g = task / N;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (g * 4 + u < kc)
                        Tpart[(((size_t)blockIdx.x * nbt + bb) * N + row) * Kq + k0 + g * 4 + u] = acc[t][u];
            }
        }
    }
    if (!ONLY && ok) {
#pragma unroll
        for (int k = 0; k < KC; ++k)
            if (k < kc) { sum[v * Kfull + k0 + k] = s1[k]; sumsq[v * Kfull + k0 + k] = s2[k]; }
    }
}

// out[j] = sum over tiles of part[tile][j]  (fixed order)
__global__ void rb_reduce_kernel(const double* __restrict__ part, int ntile, long long n, double* __restrict__ out) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double a = 0.0;
    for (int t = 0; t < ntile; ++t) a += part[(size_t)t * n + j];
    out[j] = a;
}

// ------------------------------------------------------------------------------------------------
// LVcorr[b] = _compute_corr(X_new @ V_hat, Y_new): per block, Pearson correlation (with multiplicity) of
// the resampled behaviour columns with the resampled latent scores  L[i, k] = T[b, idx[i], k] / ||VS_k||
// (bootstrap_permutation.py:636-642, 668-675).  One CTA per bootstrap.  Yz is the output of rb_coef_kernel.
__global__ void __launch_bounds__(256) rb_lvcorr_kernel(const double* __restrict__ T, const double* __restrict__ nrm2,
                                                       const double* __restrict__ Yz, const int32_t* __restrict__ idx,
                                                       int N, int nb, int K, const int32_t* __restrict__ cell_start,
                                                       int ncell, double* __restrict__ LV) {
    extern __shared__ __align__(16) double sml[];
    double* L = sml;                           // [N][K] z-scored latent
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const double* Tb = T + (size_t)b * N * K;
    for (int i = tid; i < N * K; i += nt) {
        const int row = i / K, k = i % K;
        const double n2 = nrm2[(size_t)b * K + k];
        const int src = idx ? idx[(size_t)b * N + row] : row;
        L[i] = n2 > 0.0 ? Tb[(size_t)src * K + k] / sqrt(n2) : 0.0;
    }
    __syncthreads();
    for (int o = tid; o < ncell * K; o += nt) {
        const int c = o / K, k = o % K, s = cell_start[c], e = cell_start[c + 1], n = e - s;
        double m = 0.0;
        for (int i = s; i < e; ++i) m += L[i * K + k];
        m /= n;
        double q = 0.0;
        for (int i = s; i < e; ++i) { const double d = L[i * K + k] - m; q = fma(d, d, q); }
        const double sd = sqrt(q / n);
        const double sc = sd > 0.0 ? 1.0 / (sd * sqrt((double)n)) : 0.0;
        for (int i = s; i < e; ++i) L[i * K + k] = (L[i * K + k] - m) * sc;
    }
    __syncthreads();
    const double* Yb = Yz + (size_t)b * N * nb;
    for (int o = tid; o < ncell * nb * K; o += nt) {
        const int k = o % K, cj = o / K, c = cj / nb, j = cj % nb;
        double acc = 0.0;
        for (int i = cell_start[c]; i < cell_start[c + 1]; ++i) acc = fma(Yb[i * nb + j], L[i * K + k], acc);
        LV[((size_t)b * ncell * nb + cj) * K + k] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Explicit scatter of the row-space weights: C[r][o][k] = sum_{i: idx[r][i] == o} E[i][k]  (deterministic scan)
__global__ void __launch_bounds__(256) scatter_coef_kernel(const double* __restrict__ E, int N, int K,
                                                          const int32_t* __restrict__ idx, double* __restrict__ C) {
    extern __shared__ int sids[];
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < N; i += blockDim.x) sids[i] = idx[(size_t)r * N + i];
    __syncthreads();
    for (int o = threadIdx.x; o < N * K; o += blockDim.x) {
        const int row = o / K, k = o % K;
        double acc = 0.0;
        for (int i = 0; i < N; ++i)
            if (sids[i] == row) acc += E[(size_t)i * K + k];
        C[(size_t)r * N * K + o] = acc;
    }
}

// C2[r][i][k] = sum_m C1[r][i][m] * rn[r][m] * Uc[m][k],  rn = 1/sqrt(d2) (0 where d2 <= 0):
// normalise the multiblock rows (class_functions.py:503-505) and project on the design weights.
__global__ void __launch_bounds__(256) coef_project_kernel(const double* __restrict__ C1, int N, int M,
                                                          const double* __restrict__ d2, const double* __restrict__ Uc,
                                                          int K, double* __restrict__ C2) {
    extern __shared__ __align__(16) double smc[];
    double* Us = smc;              // [M][K] scaled by rn
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < M * K; i += blockDim.x) {
        const double d = d2[(size_t)r * M + i / K];
        Us[i] = Uc[i] * (d > 0.0 ? 1.0 / sqrt(d) : 0.0);
    }
    __syncthreads();
    const double* c1 = C1 + (size_t)r * N * M;
    for (int o = threadIdx.x; o < N * K; o += blockDim.x) {
        const int row = o / K, k = o % K;
        double acc = 0.0;
        for (int m = 0; m < M; ++m) acc = fma(c1[(size_t)row * M + m], Us[m * K + k], acc);
        C2[(size_t)r * N * K + o] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Split-half Gram blocks for the behaviour / multiblock family (split_half_resampling.py:198-262,
// 315-383, 615-683, 734-802).  Half h of split s is a list of positions -> data rows (ids) cut into
// blocks; the rows of its cross-block matrix are
//     M_h[k](v) = sum_c sc_{h,c}(v) sum_{pos in c} x[ids[pos], v] Q_h[pos, k]
// with sc = 1/(sd sqrt(n)) over the block's member rows for standardised blocks (x from Xstd) and sc = 1 for
// the trailing `unit_cells` blocks (plain linear rows, x from Xlin: the multiblock task part).
// CTA = 256 voxels: phase 1 forms both halves' K rows per voxel, phase 2 reduces the three K x K blocks
// S11, S12, S22 over the tile; partials per (tile, split) are summed in a fixed order afterwards.
template <int KC>
__global__ void __launch_bounds__(256) half_gram_kernel(const double* __restrict__ Xstd, const double* __restrict__ Xlin,
                                                       long long p, const int32_t* __restrict__ ids,
                                                       const double* __restrict__ Q,
                                                       const int32_t* __restrict__ cells, int ncell, int unit_cells,
                                                       int nmax, int K, int s0, int ns, double* __restrict__ part) {
    extern __shared__ __align__(16) double smh[];
    double* Rs = smh;                                   // [2][256][KC]
    double* Qs = Rs + 2 * 256 * KC;                     // [nmax][KC]
    int* sid = reinterpret_cast<int*>(Qs + (size_t)nmax * KC);   // [nmax]
    const int tid = threadIdx.x;
    const long long v = (long long)blockIdx.x * 256 + tid;
    const bool ok = v < p;
    for (int ss = 0; ss < ns; ++ss) {
        const int sp = s0 + ss;
        for (int h = 0; h < 2; ++h) {
            __syncthreads();
            const double* q = Q + ((size_t)(sp * 2 + h) * nmax) * K;
            for (int i = tid; i < nmax * KC; i += 256) {
                const int pos = i / KC, k = i % KC;
                Qs[i] = k < K ? q[(size_t)pos * K + k] : 0.0;
            }
            for (int i = tid; i < nmax; i += 256) sid[i] = ids[(size_t)(sp * 2 + h) * nmax + i];
            __syncthreads();
            double rows[KC];
#pragma unroll
            for (int k = 0; k < KC; ++k) rows[k] = 0.0;
            const int32_t* cs = cells + h * (ncell + 1);
            for (int c = 0; c < ncell; ++c) {
                const int b = cs[c], e = cs[c + 1];
                const bool unit = c >= ncell - unit_cells;
                const double* src = unit ? Xlin : Xstd;
                double m1 = 0.0, m2 = 0.0, P[KC];
#pragma unroll
                for (int k = 0; k < KC; ++k) P[k] = 0.0;
                for (int pos = b; pos < e; ++pos) {
                    const double x = ok ? __ldg(src + (long long)sid[pos] * p + v) : 0.0;
                    m1 += x;
                    m2 = fma(x, x, m2);
                    const double* qq = Qs + pos * KC;
#pragma unroll
                    for (int k = 0; k < KC; ++k) P[k] = fma(x, qq[k], P[k]);
                }
                const double n = (double)(e - b);
                m1 /= n; m2 /= n;
                const double var = m2 - m1 * m1;
                const double sc = unit ? 1.0 : ((var > 1e-13 * m2 && var > 0.0) ? 1.0 / sqrt(var * n) : 0.0);
#pragma unroll
                for (int k = 0; k < KC; ++k) rows[k] = fma(sc, P[k], rows[k]);
            }
#pragma unroll
            for (int k = 0; k < KC; ++k) Rs[(h * 256 + tid) * KC + k] = ok ? rows[k] : 0.0;
        }
        __syncthreads();
        double* out = part + ((size_t)blockIdx.x * ns + ss) * 3 * K * K;
        for (int o = tid; o < 3 * K * K; o += 256) {
            const int which = o / (K * K), a = (o % (K * K)) / K, b = o % K;
            const double* Ra = Rs + (which == 2 ? 256 * KC : 0) + a;
            const double* Rb = Rs + (which == 0 ? 0 : 256 * KC) + b;
            double acc = 0.0;
            for (int t = 0; t < 256; ++t) acc = fma(Ra[t * KC], Rb[t * KC], acc);
            out[o] = acc;
        }
    }
}

}  // namespace plsb

using namespace plsb;

extern "C" size_t plsb200_half_gram_f64_workspace(int64_t p, int K, int ns) {
    if (p <= 0 || K <= 0 || ns <= 0) return 0;
    return (size_t)cdiv(p, 256) * ns * 3 * K * K * sizeof(double);
}

extern "C" int plsb200_half_gram_f64(const double* Xstd, const double* Xlin, int64_t p, const int32_t* ids,
                                     const double* Q, const int32_t* cells, int ncell, int unit_cells, int nmax, int K,
                                     int s0, int ns, double* S3, void* workspace, size_t workspace_bytes,
                                     void* stream) {
    PLSB_CHECK_ARG(Xstd && Xlin && ids && Q && cells && S3 && workspace, "half_gram_f64: null pointer");
    PLSB_CHECK_ARG(p > 0 && ncell > 0 && nmax > 0 && K > 0 && ns > 0, "half_gram_f64: bad shape");
    if (K > 24) {
        set_err("half_gram_f64: K=%d > 24 not supported", K);
        return PLSB200_EUNSUPPORTED;
    }
    const int ntile = (int)cdiv(p, 256);
    const size_t need = (size_t)ntile * ns * 3 * K * K * sizeof(double);
    if (workspace_bytes < need) {
        set_err("half_gram_f64: workspace %zu < %zu bytes", workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
#define PLSB_HG_LAUNCH(KCV)                                                                                       \
    do {                                                                                                          \
        size_t smem = ((size_t)2 * 256 * KCV + (size_t)nmax * KCV) * sizeof(double) + (size_t)nmax * sizeof(int);  \
        if (smem > 220 * 1024) { set_err("half_gram_f64: halves too large for shared memory"); return PLSB200_EUNSUPPORTED; } \
        PLSB_CUDA(cudaFuncSetAttribute(half_gram_kernel<KCV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        half_gram_kernel<KCV><<<ntile, 256, smem, st>>>(Xstd, Xlin, p, ids, Q, cells, ncell, unit_cells, nmax, K, s0, \
                                                        ns, (double*)workspace);                                  \
    } while (0)
    if (K <= 8) PLSB_HG_LAUNCH(8);
    else if (K <= 16) PLSB_HG_LAUNCH(16);
    else PLSB_HG_LAUNCH(24);
#undef PLSB_HG_LAUNCH
    PLSB_LAUNCH_CHECK("half_gram_kernel");
    const long long n = (long long)ns * 3 * K * K;
    rb_reduce_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>((const double*)workspace, ntile, n,
                                                             S3 + (size_t)s0 * 3 * K * K);
    PLSB_LAUNCH_CHECK("rb_reduce_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_scatter_coef_f64(const double* E, int N, int K, const int32_t* idx, int R, double* C,
                                        void* stream) {
    PLSB_CHECK_ARG(E && idx && C, "scatter_coef_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && K > 0 && R >= 0, "scatter_coef_f64: bad shape");
    if (R == 0) return PLSB200_OK;
    scatter_coef_kernel<<<R, 256, (size_t)N * sizeof(int), (cudaStream_t)stream>>>(E, N, K, idx, C);
    PLSB_LAUNCH_CHECK("scatter_coef_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_coef_project_f64(const double* C1, int N, int M, const double* d2, const double* Uc, int K,
                                        int R, double* C2, void* stream) {
    PLSB_CHECK_ARG(C1 && d2 && Uc && C2, "coef_project_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && M > 0 && K > 0 && R >= 0, "coef_project_f64: bad shape");
    if (R == 0) return PLSB200_OK;
    size_t smem = (size_t)M * K * sizeof(double);
    if (smem > 200 * 1024) {
        set_err("coef_project_f64: M*K too large for shared memory");
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaFuncSetAttribute(coef_project_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    coef_project_kernel<<<R, 256, smem, (cudaStream_t)stream>>>(C1, N, M, d2, Uc, K, C2);
    PLSB_LAUNCH_CHECK("coef_project_kernel");
    return PLSB200_OK;
}


extern "C" int plsb200_cell_standardize_f64(const double* X, int N, int64_t p, int64_t ldx, const int32_t* cell_start,
                                            int ncell, double* Xc, double* Z, void* stream) {
    PLSB_CHECK_ARG(X && cell_start && Xc, "cell_standardize_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && ncell > 0 && ldx >= p, "cell_standardize_f64: bad shape");
    cell_standardize_kernel<<<(unsigned)cdiv(p, 256), 256, 0, (cudaStream_t)stream>>>(X, N, p, ldx, cell_start, ncell,
                                                                                     Xc, Z);
    PLSB_LAUNCH_CHECK("cell_standardize_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_rb_coef_f64(const double* Y, int N, int nb, const int32_t* idx, int R,
                                   const int32_t* cell_start, int ncell, const double* U, int Kc, int scatter,
                                   double* Q, double* W, double* Yz, void* stream) {
    PLSB_CHECK_ARG(Y && cell_start && U && Q, "rb_coef_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && nb > 0 && ncell > 0 && Kc > 0 && R >= 0, "rb_coef_f64: bad shape");
    PLSB_CHECK_ARG(!scatter || W, "rb_coef_f64: scatter mode needs W");
    if (R == 0) return PLSB200_OK;
    size_t smem = ((size_t)N * nb + 2 * (size_t)ncell * nb) * sizeof(double) + 2 * (size_t)N * sizeof(int);
    if (smem > 200 * 1024) {
        set_err("rb_coef_f64: N*nb too large for shared memory");
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaFuncSetAttribute(rb_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rb_coef_kernel<<<R, 256, smem, (cudaStream_t)stream>>>(Y, N, nb, idx, cell_start, ncell, U, Kc, scatter, Q, W, Yz);
    PLSB_LAUNCH_CHECK("rb_coef_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_rb_boot_f64_workspace(int N, int64_t p, int K, int nbt) {
    if (N <= 0 || p <= 0 || K <= 0 || nbt <= 0) return 0;
    const size_t ntile = (size_t)cdiv(p, RB_VT);
    return ntile * nbt * ((size_t)N * K + K) * sizeof(double);
}

extern "C" int plsb200_rb_boot_vs_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                                      const double* Q, const double* W, int K, int b0,
                                      int nbt, const int32_t* cell_start, int ncell, int unit_cells, const double* pivot,
                                      double* sum, double* sumsq, double* T, double* nrm2, double* VS, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(Xc && Q && W && cell_start && sum && sumsq && T && nrm2 && workspace, "rb_boot_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && K > 0 && nbt > 0 && ncell > 0, "rb_boot_f64: bad shape");
    if (Xc2 == nullptr) { n1 = N; ld2 = p; }
    PLSB_CHECK_ARG(n1 > 0 && n1 <= N && ld2 >= p, "rb_boot_f64: bad row split");
    const int ntile = (int)cdiv(p, RB_VT);
    const size_t need = (size_t)ntile * nbt * ((size_t)N * K + K) * sizeof(double);
    if (workspace_bytes < need) {
        set_err("rb_boot_f64: workspace %zu < %zu bytes", workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* Tpart = (double*)workspace;
    double* Npart = Tpart + (size_t)ntile * nbt * N * K;
    const int nch = (int)cdiv(K, 16);
    const int kc_max = (int)cdiv(K, nch);
    double* VSb = VS ? VS + (size_t)b0 * p * K : nullptr;
    for (int k0 = 0; k0 < K; k0 += kc_max) {
        const int kc = K - k0 < kc_max ? K - k0 : kc_max;
        if ((long long)N * ((kc + 3) / 4) > 8 * RB_VT) {
            set_err("rb_boot_f64: N=%d too large", N);
            return PLSB200_EUNSUPPORTED;
        }
#define PLSB_RB_LAUNCH(KCV)                                                                                         \
    do {                                                                                                            \
        size_t smem = ((size_t)N * KCV + N + (size_t)KCV * RB_VT + (size_t)N * (RB_VCH + 1)) * sizeof(double);      \
        if (smem > 220 * 1024) { set_err("rb_boot_f64: N=%d too large for shared memory", N); return PLSB200_EUNSUPPORTED; } \
        auto kern = VSb ? rb_boot_kernel<KCV, true> : rb_boot_kernel<KCV, false>;                                   \
        PLSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));              \
        kern<<<ntile, RB_VT, smem, st>>>(Xc, N, p, Xc2, n1, ld2, Q, W, K, k0, kc, b0, nbt, cell_start, ncell,       \
                                         unit_cells, pivot, K, sum, sumsq, Tpart, Npart, VSb, 0, 0, 0);             \
    } while (0)
        if (kc <= 8) PLSB_RB_LAUNCH(8);
        else if (kc <= 12) PLSB_RB_LAUNCH(12);
        else PLSB_RB_LAUNCH(16);
#undef PLSB_RB_LAUNCH
        PLSB_LAUNCH_CHECK("rb_boot_kernel");
    }
    const long long nT = (long long)nbt * N * K, nN = (long long)nbt * K;
    rb_reduce_kernel<<<(unsigned)cdiv(nT, 256), 256, 0, st>>>(Tpart, ntile, nT, T + (size_t)b0 * N * K);
    PLSB_LAUNCH_CHECK("rb_reduce_kernel");
    rb_reduce_kernel<<<(unsigned)cdiv(nN, 256), 256, 0, st>>>(Npart, ntile, nN, nrm2 + (size_t)b0 * K);
    PLSB_LAUNCH_CHECK("rb_reduce_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_rb_boot_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                                   const double* Q, const double* W, int K, int b0,
                                   int nbt, const int32_t* cell_start, int ncell, int unit_cells, const double* pivot,
                                   double* sum,
                                   double* sumsq, double* T, double* nrm2, void* workspace, size_t workspace_bytes,
                                   void* stream) {
    return plsb200_rb_boot_vs_f64(Xc, N, p, Xc2, n1, ld2, Q, W, K, b0, nbt, cell_start, ncell, unit_cells, pivot, sum, sumsq,
                                  T, nrm2, nullptr, workspace, workspace_bytes, stream);
}

// The export-only pass of rb_boot over the voxel window [v0, v1) (right_sv_sampled in voxel chunks): VS[b][v - v0][k]
// for the bootstraps [0, nbt) of Q / W, the same per-voxel arithmetic as plsb200_rb_boot_vs_f64.
extern "C" int plsb200_rb_salience_f64(const double* Xc, int N, int64_t ld1, const double* Xc2, int n1, int64_t ld2,
                                       int64_t v0, int64_t v1, const double* Q, const double* W, int K, int nbt,
                                       const int32_t* cell_start, int ncell, int unit_cells, double* VS, void* stream) {
    PLSB_CHECK_ARG(Xc && Q && W && cell_start && VS, "rb_salience_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && K > 0 && nbt > 0 && ncell > 0 && v0 >= 0 && v1 > v0 && ld1 >= v1, "rb_salience_f64: bad shape");
    if (Xc2 == nullptr) { n1 = N; ld2 = ld1; }
    PLSB_CHECK_ARG(n1 > 0 && n1 <= N && ld2 >= v1, "rb_salience_f64: bad row split");
    cudaStream_t st = (cudaStream_t)stream;
    const int ntile = (int)cdiv(v1 - v0, RB_VT);
    int nsl = (int)cdiv(4LL * num_sms(), ntile);          // bootstrap slices: fill the SMs when the window is narrow
    if (nsl > nbt) nsl = nbt;
    if (nsl > 65535) nsl = 65535;
    const int bslice = (int)cdiv(nbt, nsl);
    nsl = (int)cdiv(nbt, bslice);
    const int nch = (int)cdiv(K, 16);                     // the column passes of plsb200_rb_boot_vs_f64
    const int kc_max = (int)cdiv(K, nch);
    for (int k0 = 0; k0 < K; k0 += kc_max) {
        const int kc = K - k0 < kc_max ? K - k0 : kc_max;
#define PLSB_RS_LAUNCH(KCV)                                                                                         \
    do {                                                                                                            \
        size_t smem = ((size_t)N * KCV + N) * sizeof(double);                                                       \
        if (smem > 220 * 1024) { set_err("rb_salience_f64: N=%d too large for shared memory", N); return PLSB200_EUNSUPPORTED; } \
        PLSB_CUDA(cudaFuncSetAttribute(rb_boot_kernel<KCV, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        rb_boot_kernel<KCV, true, true><<<dim3(ntile, nsl), RB_VT, smem, st>>>(                                     \
            Xc, N, v1, Xc2, n1, ld2, Q, W, K, k0, kc, 0, nbt, cell_start, ncell, unit_cells, nullptr, K, nullptr,   \
            nullptr, nullptr, nullptr, VS, v0, ld1, bslice);                                                        \
    } while (0)
        if (kc <= 8) PLSB_RS_LAUNCH(8);
        else if (kc <= 12) PLSB_RS_LAUNCH(12);
        else PLSB_RS_LAUNCH(16);
#undef PLSB_RS_LAUNCH
        PLSB_LAUNCH_CHECK("rb_boot_kernel");
    }
    return PLSB200_OK;
}

extern "C" int plsb200_rb_lvcorr_f64(const double* T, const double* nrm2, const double* Yz, const int32_t* idx, int N,
                                     int nb, int K, int R, const int32_t* cell_start, int ncell, double* LVcorr,
                                     void* stream) {
    PLSB_CHECK_ARG(T && nrm2 && Yz && cell_start && LVcorr, "rb_lvcorr_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && nb > 0 && K > 0 && R >= 0 && ncell > 0, "rb_lvcorr_f64: bad shape");
    if (R == 0) return PLSB200_OK;
    size_t smem = (size_t)N * K * sizeof(double);
    if (smem > 200 * 1024) {
        set_err("rb_lvcorr_f64: N*K too large for shared memory");
        return PLSB200_EUNSUPPORTED;
    }
    PLSB_CUDA(cudaFuncSetAttribute(rb_lvcorr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rb_lvcorr_kernel<<<R, 256, smem, (cudaStream_t)stream>>>(T, nrm2, Yz, idx, N, nb, K, cell_start, ncell, LVcorr);
    PLSB_LAUNCH_CHECK("rb_lvcorr_kernel");
    return PLSB200_OK;
}
