// K1: Gram matrix G = X . X^T in FP64 on the DMMA tensor path, split over voxel chunks.
//
// Replaces the N x p work every resample repeats in the reference (row gather resample.py:79,153;
// cell means class_functions.py:279-408; projection bootstrap_permutation.py:404): with G in hand all
// per-resample quantities except std_errs are N-space contractions (SURVEY.md App. A).
//
// Layout: X is N x p row-major (voxels contiguous).  For G[i][j] = sum_v X[i][v] X[j][v] both MMA
// operands are "K-major" rows of X, so A-fragments and B-fragments are read with the same pattern
// (row = lane/4, k = lane%4) from two shared-memory tiles of 64 rows x 32 voxels, padded to a row
// stride of 36 doubles so that the 16 lanes of an LDS.64 phase hit 16 distinct 8-byte bank pairs.
// Only tiles with tj >= ti are computed; the reduce kernel mirrors them.  Split-K partials are summed
// in a fixed order, so G is bit-reproducible run to run.
#include "common.cuh"
#include <math.h>

namespace plsb {

constexpr int GT = 64;        // output tile edge
constexpr int GKC = 32;       // voxels per pipeline stage
constexpr int GSTR = GKC + 4; // padded smem row stride (doubles)
constexpr int GSTAGES = 3;
constexpr int GTHREADS = 128; // 4 warps, each a 32x32 sub-tile

struct GramPlan {
    int ntile;      // tiles per edge
    int npair;      // upper-triangular tile pairs
    int nsplit;     // voxel chunks
    int64_t chunk;  // voxels per chunk (multiple of GKC)
};

static GramPlan gram_plan(int N, int64_t p) {
    GramPlan g;
    g.ntile = (int)cdiv(N, GT);
    g.npair = g.ntile * (g.ntile + 1) / 2;
    int64_t nk = cdiv(p, GKC);
    int64_t max_ns = nk / 8 > 0 ? nk / 8 : 1;  // at least 8 k-stages per CTA
    if (max_ns > 4096) max_ns = 4096;
    // voxel splits so that tile pairs x splits fills whole waves of the 2 CTAs an SM holds (the first version took
    // ceil(4 SMs / pairs): 15 pairs x 40 splits = 600 CTAs = 2.03 waves of 296 at N = 300 -- a third wave for 8 CTAs);
    // about two waves, the smallest count among (nearly) equally efficient ones
    const int64_t slots = 2LL * num_sms();
    int64_t ns = 1;
    double best = -1.0;
    for (int64_t c = 1; c <= max_ns && (double)(g.npair * c) <= 2.0 * slots + 0.5; ++c) {
        const double waves = (double)(g.npair * c) / (double)slots;
        const double eff = waves / ceil(waves);
        if (eff > best + 0.02) { best = eff; ns = c; }
    }
    g.chunk = cdiv(nk, ns) * GKC;
    g.nsplit = (int)cdiv(p, g.chunk);
    return g;
}

// T: element type of X (double, or float widened when the fragments are formed: the same FP64 products in the same
// order, so the same G as from the widened matrix).  VEC: elements per cp.async (16 bytes when rows are 16-B aligned,
// else one element).
template <typename T, int VEC>
__global__ void __launch_bounds__(GTHREADS) gram_partial_kernel(const T* __restrict__ X, int N, long long p,
                                                               long long ldx, const T* __restrict__ X2, int n1,
                                                               long long ld2, long long chunk, int ntile,
                                                               double* __restrict__ part) {
    extern __shared__ __align__(16) double sm[];
    // pair index -> (ti, tj) with tj >= ti
    int pair = blockIdx.x, ti = 0;
    {
        int rem = pair, row = ntile;
        while (rem >= row) { rem -= row; --row; ++ti; }
        pair = rem;
    }
    const int tj = ti + pair;
    const bool diag = (ti == tj);
    const long long v0 = (long long)blockIdx.y * chunk;
    const long long v1 = min(p, v0 + chunk);
    const int nstage_total = (int)((v1 - v0 + GKC - 1) / GKC);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wi = (warp >> 1) * 32, wj = (warp & 1) * 32;
    T* As = reinterpret_cast<T*>(sm);           // [GSTAGES][GT][GSTR]
    T* Bs = As + GSTAGES * GT * GSTR;           // same shape (unused on diagonal tiles)

    // rows [0, n1) live in X, rows [n1, N) in X2 (the Gram matrix of the stack [X; X2] without materialising it;
    // n1 == N: a single matrix)
    auto rowp = [&](int row) { return row < n1 ? X + (long long)row * ldx : X2 + (long long)(row - n1) * ld2; };
    auto load_stage = [&](int st, int kt) {
        const long long vb = v0 + (long long)kt * GKC;
        constexpr int CH = GKC / VEC;           // chunks per row
        for (int c = tid; c < GT * CH; c += GTHREADS) {
            const int r = c / CH, cc = (c % CH) * VEC;
            const long long v = vb + cc;
            long long left = v1 - v; if (left < 0) left = 0; if (left > VEC) left = VEC;
            {
                const int row = ti * GT + r;
                const int nb = row < N ? (int)left * (int)sizeof(T) : 0;
                const T* src = nb ? rowp(row) + v : X;
                cp_async_zfill<VEC * sizeof(T)>(As + (st * GT + r) * GSTR + cc, src, nb);
            }
            if (!diag) {
                const int row = tj * GT + r;
                const int nb = row < N ? (int)left * (int)sizeof(T) : 0;
                const T* src = nb ? rowp(row) + v : X;
                cp_async_zfill<VEC * sizeof(T)>(Bs + (st * GT + r) * GSTR + cc, src, nb);
            }
        }
    };

    double acc[4][4][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

#pragma unroll
    for (int s = 0; s < GSTAGES - 1; ++s) {
        if (s < nstage_total) load_stage(s, s);
        cp_async_commit();
    }
    const int fr = lane >> 2, fk = lane & 3;
    for (int kt = 0; kt < nstage_total; ++kt) {
        cp_async_wait<GSTAGES - 2>();
        __syncthreads();
        {   // prefetch stage kt + GSTAGES - 1 into the slot freed at iteration kt-1
            const int nk = kt + GSTAGES - 1;
            if (nk < nstage_total) load_stage(nk % GSTAGES, nk);
            cp_async_commit();
        }
        const int st = kt % GSTAGES;
        const T* a_base = As + (st * GT + wi + fr) * GSTR + fk;
        const T* b_base = (diag ? As : Bs) + (st * GT + wj + fr) * GSTR + fk;
#pragma unroll
        for (int ks = 0; ks < GKC / 4; ++ks) {
            double af[4], bf[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                af[t] = (double)a_base[t * 8 * GSTR + ks * 4];
                bf[t] = (double)b_base[t * 8 * GSTR + ks * 4];
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) dmma884(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
        }
    }
    cp_async_wait<0>();

    // partial tile [GT][GT] row-major
    double* out = part + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * (GT * GT);
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int r = wi + a * 8 + fr, c = wj + b * 8 + 2 * fk;
            *reinterpret_cast<double2*>(out + r * GT + c) = make_double2(acc[a][b][0], acc[a][b][1]);
        }
}

// One thread per element of a tile pair (grid: pairs x GT*GT/GRED_THREADS): the split partials of an element are summed
// in split order.  One CTA per pair (15 CTAs at N = 300) left most SMs idle while it read the partials.
constexpr int GRED_THREADS = 256;
__global__ void __launch_bounds__(GRED_THREADS) gram_reduce_kernel(const double* __restrict__ part, int npair,
                                                                   int nsplit, int ntile, int N, double* __restrict__ G) {
    const int pair = blockIdx.x;
    int ti = 0, rem = pair, row = ntile;
    while (rem >= row) { rem -= row; --row; ++ti; }
    const int tj = ti + rem;
    const int e = blockIdx.y * GRED_THREADS + threadIdx.x;
    const int r = ti * GT + e / GT, cc = tj * GT + e % GT;
    if (r >= N || cc >= N) return;
    const double* src = part + (long long)pair * (GT * GT) + e;
    const long long stride = (long long)npair * (GT * GT);
    double s = 0.0;
    for (int c = 0; c < nsplit; ++c) s += __ldg(src + c * stride);
    G[(long long)r * N + cc] = s;
    if (ti != tj) G[(long long)cc * N + r] = s;
}

}  // namespace plsb

using namespace plsb;

extern "C" size_t plsb200_gram_f64_workspace(int N, int64_t p) {
    if (N <= 0 || p <= 0) return 0;
    GramPlan g = gram_plan(N, p);
    return (size_t)g.nsplit * g.npair * GT * GT * sizeof(double);
}

template <typename T>
static int gram_launch(const T* X, int n1, int64_t ldx, const T* X2, int n2, int64_t ld2, int64_t p, double* G,
                       void* workspace, size_t workspace_bytes, void* stream, const char* what) {
    const int N = n1 + n2;
    GramPlan g = gram_plan(N, p);
    size_t need = (size_t)g.nsplit * g.npair * GT * GT * sizeof(double);
    if (workspace_bytes < need) {
        set_err("%s: workspace %zu < %zu bytes", what, workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)2 * GSTAGES * GT * GSTR * sizeof(T);
    constexpr int V = 16 / (int)sizeof(T);      // elements of a 16-byte copy
    const bool vec = ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && (ldx % V == 0) &&
                     (n2 == 0 || (((reinterpret_cast<uintptr_t>(X2) & 15) == 0) && (ld2 % V == 0)));
    dim3 grid(g.npair, g.nsplit);
    if (vec) {
        PLSB_CUDA(cudaFuncSetAttribute(gram_partial_kernel<T, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gram_partial_kernel<T, V><<<grid, GTHREADS, smem, st>>>(X, N, p, ldx, X2, n1, ld2, g.chunk, g.ntile, (double*)workspace);
    } else {
        PLSB_CUDA(cudaFuncSetAttribute(gram_partial_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gram_partial_kernel<T, 1><<<grid, GTHREADS, smem, st>>>(X, N, p, ldx, X2, n1, ld2, g.chunk, g.ntile, (double*)workspace);
    }
    PLSB_LAUNCH_CHECK("gram_partial_kernel");
    gram_reduce_kernel<<<dim3(g.npair, GT * GT / GRED_THREADS), GRED_THREADS, 0, st>>>((const double*)workspace, g.npair,
                                                                                       g.nsplit, g.ntile, N, G);
    PLSB_LAUNCH_CHECK("gram_reduce_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_gram_f64(const double* X, int N, int64_t p, int64_t ldx, double* G, void* workspace,
                                size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(X && G && workspace, "gram_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && ldx >= p, "gram_f64: bad shape N=%d p=%lld ldx=%lld", N, (long long)p,
                   (long long)ldx);
    return gram_launch<double>(X, N, ldx, nullptr, 0, 0, p, G, workspace, workspace_bytes, stream, "gram_f64");
}

// X stored as float32: the same partial sums as plsb200_gram_f64 on the widened matrix (workspace: gram_f64_workspace)
extern "C" int plsb200_gram_x32_f64(const float* X, int N, int64_t p, int64_t ldx, double* G, void* workspace,
                                    size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(X && G && workspace, "gram_x32_f64: null pointer");
    PLSB_CHECK_ARG(N > 0 && p > 0 && ldx >= p, "gram_x32_f64: bad shape N=%d p=%lld ldx=%lld", N, (long long)p,
                   (long long)ldx);
    return gram_launch<float>(X, N, ldx, nullptr, 0, 0, p, G, workspace, workspace_bytes, stream, "gram_x32_f64");
}

extern "C" int plsb200_gram_stacked_f64(const double* X1, int N1, int64_t ld1, const double* X2, int N2, int64_t ld2,
                                        int64_t p, double* G, void* workspace, size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(X1 && X2 && G && workspace, "gram_stacked_f64: null pointer");
    PLSB_CHECK_ARG(N1 > 0 && N2 > 0 && p > 0 && ld1 >= p && ld2 >= p, "gram_stacked_f64: bad shape");
    return gram_launch<double>(X1, N1, ld1, X2, N2, ld2, p, G, workspace, workspace_bytes, stream, "gram_stacked_f64");
}
