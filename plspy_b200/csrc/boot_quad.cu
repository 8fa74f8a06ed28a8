// Collapsed bootstrap (task methods): the quadratic forms q[v,k] = x_v^T S_k x_v on the FP64 tensor cores.
//
// Every bootstrap salience is linear in the draw, VS_r[v,k] = x_v^T c_rk (c_rk = column k of C_r = scatter(E, idx_r)),
// so its spread over the resamples is a quadratic form in the covariance of the coefficients:
//       R . Var_r(VS_r[v,k]) = x_v^T S_k x_v,        S_k = sum_r d_rk d_rk^T - s1_k s1_k^T / R   (N x N)
// with d_r = C_r - E and s1_k = sum_r d_rk (DESIGN.md section 3).  Engine.boot_cov forms the S_k in N-space; this
// file evaluates the p x K quadratic forms, 2 p N^2 K flops instead of the 2 p N K B of the direct moment GEMM.
//
// The kernel is boot_moments_kernel (boot.cu) with N "pseudo-resamples" in place of the B resamples: pseudo-resample m
// has the N x K coefficient matrix P_m[n,k] = S_k[n,m], packed in the layout of boot_coef_pack_kernel (bfrag_offset),
// and the plan, the ring of bulk copies, the mbarriers and the DMMA stream are the same code, ring_pipeline
// (boot_plan.cuh).  What boot_quad_kernel adds is QuadEpilogue: a D element is (S_k x_v)[m], folded as
// acc[v,k] += X[m,v] . d with X[m,v] loaded before the period's wait, and fold_slots_store writes the one output.
// Pseudo-resamples m >= N and columns k >= K are zero in the pack.
#include <float.h>

#include "common.cuh"
#include "boot_plan.cuh"

namespace plsb {

// S ([K][N][N], row-major) -> the packed layout (bfrag_offset): element i of the pack, enumerated as period per, k-step
// s, column c and row 4*s + q in the order of the layout, is S_k[row, m] for column c = slot*Kp + k of pseudo-resample
// m = per*nb + slot.
__global__ void quad_coef_pack_kernel(const double* __restrict__ S, int N, int K, int Kp, int nblk, int nb, int nks,
                                      long long total, double* __restrict__ coef) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int q = (int)(i & 3);
    long long t = i >> 2;
    const int c = (int)(t % (8 * nblk)); t /= 8 * nblk;
    const int s = (int)(t % nks);
    const int per = (int)(t / nks);
    const int row = 4 * s + q, k = c % Kp, m = per * nb + c / Kp;
    coef[(size_t)per * nks * nblk * 32 + bfrag_offset(s, c, q, nblk)] =
        (row < N && m < N && k < K) ? S[((size_t)k * N + row) * N + m] : 0.0;
}

// The quadratic-form epilogue: the chains start from 0, so a D element is (S_k x_v)[m] for the pseudo-resample m of
// its column; it is folded as acc += X[m,v] . d.  X[m,v] comes from an __ldg issued before the period's wait (the A
// registers cannot serve it: m is a runtime index); the loads of rows m >= N are masked.
template <typename T, int NBLK>
struct QuadEpilogue : RingEpilogue {
    struct Args { const T* X; long long ldx, v, p; int N, Kp, K; double* out; };
    const Args a;
    const RingThread th;
    const long long vc;                                   // (address of the masked lanes' X loads)
    int slot_of[NBLK][2];                                 // pseudo-resample slot of each column
    double acc[1][NBLK][2], xm[NBLK][2];
    int nb;
    __device__ __forceinline__ QuadEpilogue(const Args& args, const RingThread& t)
        : a(args), th(t), vc(args.v < args.p ? args.v : 0) {
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) { slot_of[j][e] = (8 * j + 2 * th.q + e) / a.Kp; acc[0][j][e] = 0.0; }
        nb = 8 * NBLK / a.Kp;
    }
    __device__ __forceinline__ void before_wait(int it) {
        const int mbase = (th.per0 + it) * nb;
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int m = mbase + slot_of[j][e];
                xm[j][e] = m < a.N ? (double)__ldg(a.X + (long long)m * a.ldx + vc) : 0.0;
            }
    }
    __device__ __forceinline__ void fold(const double (&d)[NBLK][2], int) {
#pragma unroll
        for (int j = 0; j < NBLK; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) acc[0][j][e] = fma(xm[j][e], d[j][e], acc[0][j][e]);
    }
    __device__ __forceinline__ void finish(double* red) {
        fold_slots_store<1, NBLK>(acc, red, th, nb, a.Kp, a.K, a.p, {a.out});
    }
};

// T: element type of X (float: X stored as float32, widened at every load -- the same FP64 operations as on the
// widened matrix).  The plan reserves shared memory for two outputs per warp; this kernel uses one.
template <typename T, int NKS, int NBLK>
__global__ void __launch_bounds__(BM_THREADS, 1)
boot_quad_kernel(const T* __restrict__ X, long long ldx, int N, long long p, const double* __restrict__ coef,
                 int nper, int per_per_split, int nstage, int Kp, int K, double* __restrict__ out) {
    const RingThread th(threadIdx.x, nper, per_per_split);
    const long long v = (long long)blockIdx.x * BM_VOX + th.warp * 8 + th.vr;
    ring_pipeline<NKS, NBLK, QuadEpilogue<T, NBLK>>(th, X, ldx, N, v, v < p, coef, nstage, BM_WARPS * 16 * Kp,
                                                    {X, ldx, v, p, N, Kp, K, out});
}

// ------------------------------------------------------------------------------------------------
// Factored form (DESIGN.md section 3).  A draw of resample.bootstrap_indices keeps every row in its cell and uses one
// subject map for all conditions, and E is constant within a cell, so c_rk[n] = E[n,k] . m_r[subj(n)] with m_r the
// draw counts of the subjects and S_k = D_k P M P^T D_k, M = sum_r (m_r - 1)(m_r - 1)^T - s1 s1^T / R (ns x ns, the
// same for every k).  With M = L L^T the quadratic form is a sum of squares over ns - G "pseudo-resamples" c_jk[n] =
// E[n,k] . L[subj(n), j]: the bootstrap GEMM of boot.cu, run on those.
//
// Row layout (int32, 2N + ns): base[n] = first row of n's cell, sid[n] = subject of row n, row0[s] = row of subject s
// in the first condition of its group.  One CTA per draw: checks the structure (`bad` |= 1 when a row leaves its cell
// or its subject map differs from the first condition's) and counts the draws of each subject from the first-condition
// rows (shared-memory integer atomics: the result does not depend on their order).  counts[s][r] = m_r[s] - 1 and
// counts[ns][r] = 1, so the Gram matrix of `counts` holds sum_r (m_r - 1)(m_r - 1)^T and, in its last column, s1.
__global__ void boot_counts_kernel(const int32_t* __restrict__ idx, int N, const int32_t* __restrict__ layout, int ns,
                                   double* __restrict__ counts, long long ldc, int32_t* __restrict__ bad) {
    extern __shared__ int cnt[];
    const int32_t* base = layout;
    const int32_t* sid = layout + N;
    const int32_t* row0 = layout + 2 * N;
    const int r = blockIdx.x;
    const int32_t* id = idx + (size_t)r * N;
    for (int s = threadIdx.x; s < ns; s += blockDim.x) cnt[s] = 0;
    __syncthreads();
    bool ok = true;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const int src = id[n], n0 = row0[sid[n]];
        const int src0 = id[n0];
        const bool in = src >= 0 && src < N && src0 >= 0 && src0 < N && base[src] == base[n]
                        && src - base[n] == src0 - base[n0];
        ok = ok && in;
        if (in && n == n0) atomicAdd(&cnt[sid[src]], 1);
    }
    if (!ok && bad != nullptr) atomicOr(bad, 1);
    __syncthreads();
    if (counts == nullptr) return;
    for (int s = threadIdx.x; s <= ns; s += blockDim.x) counts[(size_t)s * ldc + r] = s < ns ? cnt[s] - 1.0 : 1.0;
}

// One CTA.  Every m_r - 1 sums to zero within each group, so M has rank <= ns - G: drop the last subject of each
// group, factor the remaining J x J block A (J = ns - G) by Cholesky, and rebuild a dropped subject's row of L as minus
// the sum of its group's other rows (L L^T = M).  A pivot <= J eps max(diag A) (a singular A: draws that do not span the
// subject space) gives a zero column -- the factor of a semidefinite matrix.  A: J x J workspace (global, L2-resident);
// every element is written by one thread in a fixed order (deterministic).
__global__ void __launch_bounds__(256) boot_factor_kernel(const double* __restrict__ Mg, int ns, double R,
                                                          const int32_t* __restrict__ gstart, int G,
                                                          double* __restrict__ A, double* __restrict__ L) {
    extern __shared__ int keep[];                       // kept index -> subject
    __shared__ double piv, tol;
    const int J = ns - G, ld = ns + 1, tid = threadIdx.x, nt = blockDim.x;
    for (int a = tid; a < J; a += nt) {
        int g = 0;
        while (a >= gstart[g + 1] - (g + 1)) ++g;        // group g keeps gstart[g+1] - gstart[g] - 1 subjects
        keep[a] = a + g;
    }
    __syncthreads();
    for (int i = tid; i < J * J; i += nt) {
        const int sa = keep[i / J], sb = keep[i % J];
        A[i] = Mg[(size_t)sa * ld + sb] - Mg[(size_t)sa * ld + ns] * Mg[(size_t)sb * ld + ns] / R;
    }
    __syncthreads();
    if (tid == 0) {
        double m = 0.0;
        for (int a = 0; a < J; ++a) m = fmax(m, A[(size_t)a * J + a]);
        tol = J * DBL_EPSILON * m;
    }
    __syncthreads();
    for (int j = 0; j < J; ++j) {
        if (tid == 0) {
            const double d = A[(size_t)j * J + j];
            piv = d > tol ? sqrt(d) : 0.0;
            A[(size_t)j * J + j] = piv;
        }
        __syncthreads();
        const double pj = piv;
        for (int i = j + 1 + tid; i < J; i += nt) A[(size_t)i * J + j] = pj > 0.0 ? A[(size_t)i * J + j] / pj : 0.0;
        __syncthreads();
        const int w = J - j - 1;
        for (int t = tid; t < w * w; t += nt) {
            const int i = j + 1 + t / w, k = j + 1 + t % w;
            if (k <= i) A[(size_t)i * J + k] -= A[(size_t)i * J + j] * A[(size_t)k * J + j];
        }
        __syncthreads();
    }
    for (int i = tid; i < ns * J; i += nt) {
        const int s = i / J, j = i % J;
        int g = 0;
        while (s >= gstart[g + 1]) ++g;
        double v = 0.0;
        if (s == gstart[g + 1] - 1) {                   // dropped subject: minus the sum of the group's kept rows
            for (int a = gstart[g] - g; a < gstart[g + 1] - g - 1; ++a) v -= j <= a ? A[(size_t)a * J + j] : 0.0;
        } else {
            const int a = s - g;
            v = j <= a ? A[(size_t)a * J + j] : 0.0;
        }
        L[i] = v;
    }
}

}  // namespace plsb

using namespace plsb;

extern "C" int plsb200_boot_counts_f64(const int32_t* idx, int N, int R, const int32_t* layout, int ns, double* counts,
                                       int64_t ldc, int32_t* bad, void* stream) {
    PLSB_CHECK_ARG(idx && layout && (counts || bad), "boot_counts_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && R >= 0 && ns > 0 && ns <= N && (counts == nullptr || ldc >= R),
                   "boot_counts_f64: bad shape N=%d R=%d ns=%d", N, R, ns);
    if (R == 0) return PLSB200_OK;
    boot_counts_kernel<<<(unsigned)R, 128, (size_t)ns * sizeof(int), (cudaStream_t)stream>>>(idx, N, layout, ns, counts,
                                                                                           (long long)ldc, bad);
    PLSB_LAUNCH_CHECK("boot_counts_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_boot_factor_f64_workspace(int ns, int G) {
    const int J = ns - G;
    return (G >= 1 && J >= 1) ? (size_t)J * J * sizeof(double) : 0;
}

extern "C" int plsb200_boot_factor_f64(const double* Mg, int ns, int64_t R_total, const int32_t* gstart, int G,
                                       double* L, void* workspace, size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(Mg && gstart && L && workspace, "boot_factor_f64: null pointer");
    PLSB_CHECK_ARG(G >= 1 && ns > G && R_total > 0, "boot_factor_f64: bad shape ns=%d G=%d", ns, G);
    const size_t need = plsb200_boot_factor_f64_workspace(ns, G);
    if (workspace_bytes < need) {
        set_err("boot_factor_f64: workspace %zu < %zu bytes", workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    boot_factor_kernel<<<1, 256, (size_t)(ns - G) * sizeof(int), (cudaStream_t)stream>>>(
        Mg, ns, (double)R_total, gstart, G, (double*)workspace, L);
    PLSB_LAUNCH_CHECK("boot_factor_kernel");
    return PLSB200_OK;
}

// the plan of the quadratic form: N pseudo-resamples of N x K coefficients
static bool quad_plan(int N, int K, int64_t p, BootPlan& b) { return N <= 320 && boot_plan(N, K, N, p, b); }

extern "C" size_t plsb200_boot_quad_coef_bytes(int N, int K) {
    BootPlan b;
    if (!quad_plan(N, K, 1, b)) return 0;
    return (size_t)b.nper * b.stage_doubles * sizeof(double);
}

extern "C" int plsb200_boot_quad_coef_pack_f64(const double* S, int N, int K, double* coef, void* stream) {
    PLSB_CHECK_ARG(S && coef, "boot_quad_coef_pack_f64: null pointer");
    BootPlan b;
    if (!quad_plan(N, K, 1, b)) {
        set_err("boot_quad_coef_pack_f64: unsupported shape N=%d K=%d (need N<=320, K<=24)", N, K);
        return PLSB200_EUNSUPPORTED;
    }
    const long long total = (long long)b.nper * b.stage_doubles;
    quad_coef_pack_kernel<<<(unsigned)cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(S, N, K, b.Kp, b.nblk, b.nb,
                                                                                       b.nks, total, coef);
    PLSB_LAUNCH_CHECK("quad_coef_pack_kernel");
    return PLSB200_OK;
}

extern "C" size_t plsb200_boot_quad_f64_workspace(int N, int64_t p, int K) {
    BootPlan b;
    if (p <= 0 || !quad_plan(N, K, p, b)) return 0;
    return b.nsplit > 1 ? (size_t)b.nsplit * p * K * sizeof(double) : 16;
}

template <typename T>
static int boot_quad(const T* X, int N, int64_t p, int64_t ldx, const double* coef, int K, double* q, void* workspace,
                     size_t workspace_bytes, void* stream, const char* what) {
    PLSB_CHECK_ARG(X && coef && q, "%s: null pointer", what);
    PLSB_CHECK_ARG(p > 0 && ldx >= p, "%s: bad shape p=%lld ldx=%lld", what, (long long)p, (long long)ldx);
    BootPlan b;
    if (!quad_plan(N, K, p, b)) {
        set_err("%s: unsupported shape N=%d K=%d (need N<=320, K<=24)", what, N, K);
        return PLSB200_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* o = q;
    if (b.nsplit > 1) {
        const size_t need = (size_t)b.nsplit * p * K * sizeof(double);
        if (!workspace || workspace_bytes < need) {
            set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
            return PLSB200_EWORKSPACE;
        }
        o = (double*)workspace;
    }
    const dim3 grid((unsigned)cdiv(p, BM_VOX), (unsigned)b.nsplit);
    const int rc = ring_dispatch(b, "boot_quad_f64", [&](auto nks, auto nblk) {
        const auto kernel = boot_quad_kernel<T, decltype(nks)::value, decltype(nblk)::value>;
        PLSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b.smem_bytes));
        kernel<<<grid, BM_THREADS, b.smem_bytes, st>>>(X, ldx, N, p, coef, b.nper, b.per_per_split, b.nstage, b.Kp, K,
                                                       o);
        PLSB_LAUNCH_CHECK("boot_quad_kernel");
        return PLSB200_OK;
    });
    if (rc != PLSB200_OK) return rc;
    if (b.nsplit > 1) {
        const long long n = (long long)p * K;
        split_sum_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(o, nullptr, b.nsplit, n, q, nullptr);
        PLSB_LAUNCH_CHECK("split_sum_kernel");
    }
    return PLSB200_OK;
}

extern "C" int plsb200_boot_quad_f64(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K,
                                     double* q, void* workspace, size_t workspace_bytes, void* stream) {
    return boot_quad(X, N, p, ldx, coef, K, q, workspace, workspace_bytes, stream, "boot_quad_f64");
}

extern "C" int plsb200_boot_quad_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K,
                                         double* q, void* workspace, size_t workspace_bytes, void* stream) {
    return boot_quad(X, N, p, ldx, coef, K, q, workspace, workspace_bytes, stream, "boot_quad_x32_f64");
}
