// K1: Gram matrix G = X . X^T in FP64 on the DMMA tensor path, split over voxel chunks.
//
// Replaces the N x p work every resample repeats in the reference (row gather resample.py:79,153;
// cell means class_functions.py:279-408; projection bootstrap_permutation.py:404): with G in hand all
// per-resample quantities except std_errs are N-space contractions (SURVEY.md App. A).
//
// Layout: X is N x p row-major (voxels contiguous).  For G[i][j] = sum_v X[i][v] X[j][v] both MMA
// operands are "K-major" rows of X, so A-fragments and B-fragments are read with the same pattern
// (row = lane/4, k = lane%4) from shared-memory tiles of rows x 32 voxels, padded to a row stride of
// 36 elements so that the 16 lanes of an LDS.64 phase hit 16 distinct 8-byte bank pairs.  G is cut
// into 64-row tiles; only tiles with tj >= ti are computed, and the reduce kernel mirrors them.
// Split-K partials are summed in a fixed order, so G is bit-reproducible run to run.
//
// A CTA is one pair of 128-row super tiles (two 64-row tiles each; the last one of an odd tile count
// has one) over one voxel chunk: eight MMA warps and four producer warps.  Measured at the benchmark's
// 312 x 200 000 stack on a B200, the earlier kernel (one 64 x 64 tile per CTA, the feed issued by the
// MMA warps between CTA-wide barriers) took 1.12 ms, of which the operand feed alone took 0.60 ms and
// the DMMAs with resident operands 0.71 ms: the L2 -> shared-memory feed, not the DMMA rate, held it.
// A 128 x 128 output region reads half the operand bytes per flop of a 64 x 64 one, and the producers
// stream the stages through a GSTAGES-deep ring with cp.async (16-byte copies with zero fill, or one
// element for unaligned rows) and full / empty mbarriers (cp.async.mbarrier.arrive), so the MMA warps
// neither issue the feed nor meet at a CTA-wide barrier.  A diagonal 64-row tile is symmetric: only
// its 36 blocks of 8 x 8 on and above the block diagonal are formed, and the reduce reads the mirror
// for the blocks below.
#include "common.cuh"
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <functional>
#include <queue>
#include <vector>

// Probe modes that time parts of the partial kernel in isolation (WRONG RESULTS by construction) exist only in builds
// with -DPLSB_PROBES (tools/time_gram.py); in the product library GRAM_PROBE is the constant 0 and every probe branch
// is compiled out.  PLSB200_GRAM_PROBE: 1 = operands resident after the ring is first filled (no cp.async after it),
// 2 = the feed without fragment loads or DMMAs.
#ifdef PLSB_PROBES
#define GRAM_PROBE(x) (x)
#else
#define GRAM_PROBE(x) 0
#endif

namespace plsb {

constexpr int GT = 64;         // tile edge of G (and of the split partials)
constexpr int GS = 2 * GT;     // super-tile edge: the rows of one operand region of a CTA
constexpr int GKC = 32;        // voxels per pipeline stage
constexpr int GSTR = GKC + 4;  // padded smem row stride (elements)
constexpr int GSTAGES = 3;
constexpr int GMMA_WARPS = 8;
constexpr int GPROD_WARPS = 4;                    // one producer warp issued the copies of a stage at a third of the
                                                  // rate the DMMAs consume them
constexpr int GTHREADS = (GMMA_WARPS + GPROD_WARPS) * 32;
constexpr int GSTAGE_ELEMS = 2 * GS * GSTR;       // A and B regions of one stage

// The work of one MMA warp per k-step: nf fragments (8 rows x 4 voxels of the stage; src 0 / 1 = the warp's first /
// second operand base, blk = 8-row block from it) and np DMMAs (fragment pair fa x fb, accumulated into the 8 x 8
// output block (orow, ocol) from the warp's output offset).
struct WarpTask {
    int nf, fsrc[12], fblk[12];
    int np, fa[32], fb[32], orow[32], ocol[32];
};

// Block lists (bi <= bj) of the symmetric tasks, all fragments from one base: the two halves of a diagonal 64-row
// tile (18 + 18 blocks) and its four quarters (9 each).
constexpr int kDiagHalf[2][18][2] = {
    {{0, 4}, {0, 5}, {0, 6}, {0, 7}, {1, 4}, {1, 5}, {1, 6}, {1, 7}, {2, 4}, {2, 5}, {2, 6}, {2, 7},
     {3, 4}, {3, 5}, {3, 6}, {3, 7}, {0, 0}, {1, 1}},
    {{0, 1}, {0, 2}, {0, 3}, {1, 2}, {1, 3}, {2, 2}, {2, 3}, {3, 3}, {4, 4},
     {4, 5}, {4, 6}, {4, 7}, {5, 5}, {5, 6}, {5, 7}, {6, 6}, {6, 7}, {7, 7}},
};
constexpr int kDiagQuarter[4][9][2] = {
    {{0, 5}, {0, 6}, {0, 7}, {1, 5}, {1, 6}, {1, 7}, {2, 5}, {2, 6}, {2, 7}},
    {{0, 2}, {0, 3}, {0, 4}, {1, 2}, {1, 3}, {1, 4}, {2, 2}, {2, 3}, {2, 4}},
    {{3, 3}, {3, 4}, {3, 5}, {3, 6}, {3, 7}, {4, 4}, {4, 5}, {4, 6}, {4, 7}},
    {{0, 0}, {0, 1}, {1, 1}, {5, 5}, {5, 6}, {5, 7}, {6, 6}, {6, 7}, {7, 7}},
};

// Tasks: 0 = 64 x 32 rectangle (8 x 4 blocks), 1 = 32 x 32 rectangle (4 x 4), 2..3 = halves and 4..7 = quarters of a
// diagonal 64-row tile.
__host__ __device__ constexpr WarpTask warp_task(int t) {
    WarpTask w{};
    if (t <= 1) {
        const int na = t == 0 ? 8 : 4;
        w.nf = na + 4;
        for (int i = 0; i < na; ++i) { w.fsrc[i] = 0; w.fblk[i] = i; }
        for (int i = 0; i < 4; ++i) { w.fsrc[na + i] = 1; w.fblk[na + i] = i; }
        w.np = 4 * na;
        for (int a = 0; a < na; ++a)
            for (int b = 0; b < 4; ++b) {
                w.fa[4 * a + b] = a; w.fb[4 * a + b] = na + b; w.orow[4 * a + b] = a; w.ocol[4 * a + b] = b;
            }
        return w;
    }
    int slot[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
    w.np = t <= 3 ? 18 : 9;
    for (int j = 0; j < w.np; ++j) {
        const int bi = t <= 3 ? kDiagHalf[t - 2][j][0] : kDiagQuarter[t - 4][j][0];
        const int bj = t <= 3 ? kDiagHalf[t - 2][j][1] : kDiagQuarter[t - 4][j][1];
        if (slot[bi] < 0) { slot[bi] = w.nf; w.fsrc[w.nf] = 0; w.fblk[w.nf] = bi; ++w.nf; }
        if (slot[bj] < 0) { slot[bj] = w.nf; w.fsrc[w.nf] = 0; w.fblk[w.nf] = bj; ++w.nf; }
        w.fa[j] = slot[bi]; w.fb[j] = slot[bj]; w.orow[j] = bi; w.ocol[j] = bj;
    }
    return w;
}

// CTA kinds, in the grid's order (longest first): the MMA warp with the most blocks sets a CTA's length.
//   OFF2  off-diagonal pair of two-tile super tiles: 128 x 128, 32 blocks per warp
//   DIAG2 diagonal two-tile super tile: its off-diagonal 64-row tile (16 blocks per warp, warps 0-3) and the upper
//         halves of its two diagonal tiles (18 per warp, warps 4-7)
//   OFF1  off-diagonal pair whose column super tile is the last, one-tile one (odd tile count): 128 x 64, 16 per warp
//   DIAG1 that last tile's diagonal: 9 blocks per warp, warps 0-3
enum { K_OFF2, K_DIAG2, K_OFF1, K_DIAG1, K_COUNT };
constexpr int kKindBlocks[K_COUNT] = {32, 18, 16, 9};

__host__ __device__ inline void gram_kinds(int ntile, int (&n)[K_COUNT]) {
    const int nfull = ntile / 2, odd = ntile % 2;
    n[K_OFF2] = nfull * (nfull - 1) / 2; n[K_DIAG2] = nfull; n[K_OFF1] = odd * nfull; n[K_DIAG1] = odd;
}

struct GramPlan {
    int ntile;      // 64-row tiles per edge
    int npair;      // upper-triangular tile pairs (of the partials)
    int nsplit;     // voxel chunks
    int64_t chunk;  // voxels per chunk (multiple of GKC)
    int ctas;       // CTAs per split
};

// Makespan (in units of one OFF2 CTA over all voxels) of the grid's schedule with ns voxel splits: the CTAs in grid
// order, each started on the first free one of `slots`; `fixed` is the cost of a CTA that does not shrink with its
// chunk (pipeline fill, partial tile store).
static double gram_makespan(const int (&n)[K_COUNT], int ns, int slots, double fixed) {
    std::priority_queue<double, std::vector<double>, std::greater<double>> q;
    for (int s = 0; s < slots; ++s) q.push(0.0);
    for (int k = 0; k < K_COUNT; ++k) {
        const double len = (double)kKindBlocks[k] / kKindBlocks[K_OFF2] / ns + fixed;
        for (int64_t i = 0; i < (int64_t)n[k] * ns; ++i) {
            const double t = q.top() + len;
            q.pop(); q.push(t);
        }
    }
    double end = 0.0;
    while (!q.empty()) { end = q.top(); q.pop(); }
    return end;
}

// Depends on the number of row tiles and on p only: the rows < N of a stack get the same tiles and splits as the
// matrix alone whenever the stack adds no tile.
static GramPlan gram_plan(int N, int64_t p) {
    GramPlan g;
    g.ntile = (int)cdiv(N, GT);
    g.npair = g.ntile * (g.ntile + 1) / 2;
    int n[K_COUNT];
    gram_kinds(g.ntile, n);
    g.ctas = n[K_OFF2] + n[K_DIAG2] + n[K_OFF1] + n[K_DIAG1];
    const int64_t nk = cdiv(p, GKC);
    int64_t max_ns = nk / 8 > 0 ? nk / 8 : 1;  // at least 8 k-stages per CTA
    if (max_ns > 4096) max_ns = 4096;
    const int slots = num_sms();               // one CTA an SM
    // voxel splits: the shortest simulated schedule (about 4 k-stages of fixed cost per CTA) among up to ~3 waves of
    // CTAs; the last answer is kept, since every launch and workspace query asks again
    static thread_local int64_t key[3] = {-1, -1, -1};
    static thread_local int cached = 1;
    int ns = 1;
    if (key[0] == g.ntile && key[1] == nk && key[2] == slots) {
        ns = cached;
    } else {
        const double fixed = 4.0 / (double)nk;
        const int64_t top = std::min<int64_t>(max_ns, cdiv(3LL * slots, g.ctas) + 1);
        double best = 1e30;
        for (int64_t c = 1; c <= top; ++c) {
            const double t = gram_makespan(n, (int)c, slots, fixed);
            if (t < best * (1.0 - 1e-3)) { best = t; ns = (int)c; }
        }
        key[0] = g.ntile; key[1] = nk; key[2] = slots; cached = ns;
    }
    g.chunk = cdiv(nk, ns) * GKC;
    g.nsplit = (int)cdiv(p, g.chunk);
    return g;
}

// The producer thread's cp.async copies issued so far arrive on `bar` when they have landed (the barrier counts one
// such arrival per producer thread and phase).
__device__ __forceinline__ void cp_async_mbar_arrive(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

// One MMA warp over the CTA's stages, then its blocks into the partial tiles.  a_base / b_base: this thread's fragment
// position (row lane/4, voxel lane%4) at the warp's two operand offsets in stage 0.  ti0 / tj0: the first 64-row
// tiles of the super-tile pair; orow0 / ocol0: the warp's output offset in 8-row blocks of the super-tile pair.
template <int TASK, typename T>
__device__ __forceinline__ void gram_mma(const T* a_base, const T* b_base, uint64_t* full, uint64_t* empty,
                                         int nstage_total, int pr, int lane, double* part_split, int ntile, int ti0,
                                         int tj0, int orow0, int ocol0) {
    constexpr WarpTask w = warp_task(TASK);
    double acc[w.np][2];
#pragma unroll
    for (int j = 0; j < w.np; ++j) acc[j][0] = acc[j][1] = 0.0;
    int slot = 0;
    uint32_t phase = 0;
    for (int kt = 0; kt < nstage_total; ++kt) {
        if (!(pr == 1 && kt >= GSTAGES)) mbar_wait(full + slot, phase);
        if (pr != 2) {
            const T* sa = a_base + slot * GSTAGE_ELEMS;
            const T* sb = b_base + slot * GSTAGE_ELEMS;
#pragma unroll
            for (int ks = 0; ks < GKC / 4; ++ks) {
                double f[w.nf];
#pragma unroll
                for (int i = 0; i < w.nf; ++i) f[i] = (double)(w.fsrc[i] ? sb : sa)[w.fblk[i] * 8 * GSTR + ks * 4];
#pragma unroll
                for (int j = 0; j < w.np; ++j) dmma884(acc[j][0], acc[j][1], f[w.fa[j]], f[w.fb[j]]);
            }
        }
        __syncwarp();
        if (lane == 0 && pr != 1) mbar_arrive(empty + slot);
        if (++slot == GSTAGES) { slot = 0; phase ^= 1u; }
    }
    const int fr = lane >> 2, fk = lane & 3;
#pragma unroll
    for (int j = 0; j < w.np; ++j) {
        const int R = orow0 + w.orow[j], C = ocol0 + w.ocol[j];     // 8-row blocks in the super-tile pair
        const int ti = ti0 + R / 8, tj = tj0 + C / 8;
        const int pair = ti * ntile - ti * (ti - 1) / 2 + (tj - ti);
        double* out = part_split + (long long)pair * (GT * GT);
        *reinterpret_cast<double2*>(out + ((R % 8) * 8 + fr) * GT + (C % 8) * 8 + 2 * fk) =
            make_double2(acc[j][0], acc[j][1]);
    }
}

// T: element type of X (double, or float widened when the fragments are formed: the same FP64 products in the same
// order, so the same G as from the widened matrix).  VEC: elements per cp.async (16 bytes when rows are 16-B aligned,
// else one element).
template <typename T, int VEC>
__global__ void __launch_bounds__(GTHREADS, 1) gram_partial_kernel(const T* __restrict__ X, int N, long long p,
                                                                  long long ldx, const T* __restrict__ X2, int n1,
                                                                  long long ld2, long long chunk, int ntile, int nsplit,
                                                                  double* __restrict__ part, int probe) {
    extern __shared__ __align__(16) double sm[];
    const int pr = GRAM_PROBE(probe);
    // CTA -> (kind, super-tile pair I <= J, voxel split): kinds in K_* order, within a kind splits slowest (the CTAs
    // that run together read the same voxels)
    const int nsup = (ntile + 1) / 2;
    int kind = 0, I = 0, J = 0, split = 0;
    {
        int n[K_COUNT];
        gram_kinds(ntile, n);
        int q = blockIdx.x;
        while (q >= n[kind] * nsplit) { q -= n[kind] * nsplit; ++kind; }
        split = q / n[kind];
        int rem = q % n[kind];
        if (kind == K_OFF2) {                   // pairs I < J < ntile / 2, row-major
            int row = ntile / 2 - 1;
            while (rem >= row) { rem -= row; --row; ++I; }
            J = I + 1 + rem;
        } else if (kind == K_DIAG2) {
            I = J = rem;
        } else if (kind == K_OFF1) {
            I = rem; J = nsup - 1;
        } else {
            I = J = nsup - 1;
        }
    }
    const bool diag = (I == J);
    const int rowsA = 2 * I + 1 < ntile ? GS : GT;            // rows of the A region: one or two tiles
    const int rowsB = diag ? 0 : (2 * J + 1 < ntile ? GS : GT);
    const long long v0 = (long long)split * chunk;
    const long long v1 = min(p, v0 + chunk);
    const int nstage_total = (int)((v1 - v0 + GKC - 1) / GKC);
    const int nmma = kind == K_DIAG1 ? 4 : GMMA_WARPS;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    T* As = reinterpret_cast<T*>(sm);           // [GSTAGES][A, B][GS][GSTR]
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + (GSTAGES * GSTAGE_ELEMS * sizeof(T) + 7) / 8);
    uint64_t* empty = full + GSTAGES;
    if (tid == 0) {
        for (int s = 0; s < GSTAGES; ++s) { mbar_init(full + s, 32 * GPROD_WARPS); mbar_init(empty + s, nmma); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp >= GMMA_WARPS) {
        // producers: rows [0, n1) live in X, rows [n1, N) in X2 (the Gram matrix of the stack [X; X2] without
        // materialising it; n1 == N: a single matrix)
        auto rowp = [&](int row) { return row < n1 ? X + (long long)row * ldx : X2 + (long long)(row - n1) * ld2; };
        constexpr int CH = GKC / VEC;           // copies per row
        const int nload = (pr == 1) ? min(nstage_total, GSTAGES) : nstage_total;
        const int rows = rowsA + rowsB;
        for (int kt = 0; kt < nload; ++kt) {
            const int st = kt % GSTAGES;
            if (kt >= GSTAGES) mbar_wait(empty + st, ((kt / GSTAGES) - 1) & 1);
            const long long vb = v0 + (long long)kt * GKC;
            T* dst = As + st * GSTAGE_ELEMS;
            for (int c = tid - GMMA_WARPS * 32; c < rows * CH; c += GPROD_WARPS * 32) {
                const int r = c / CH, cc = (c % CH) * VEC;
                const long long v = vb + cc;
                long long left = v1 - v; if (left < 0) left = 0; if (left > VEC) left = VEC;
                // smem row: the A region from row 0, the B region from row GS
                const bool in_a = r < rowsA;
                const int row = in_a ? I * GS + r : J * GS + (r - rowsA);
                const int srow = in_a ? r : GS + (r - rowsA);
                const int nb = row < N ? (int)left * (int)sizeof(T) : 0;
                cp_async_zfill<VEC * sizeof(T)>(dst + srow * GSTR + cc, nb ? rowp(row) + v : X, nb);
            }
            cp_async_mbar_arrive(full + st);
        }
        cp_async_wait<0>();
        return;
    }
    if (warp >= nmma) return;

    const int fr = lane >> 2, fk = lane & 3;
    const T* fa = As + fr * GSTR + fk;          // row fr, voxel fk of the A region
    const T* fb = fa + GS * GSTR;               // of the B region
    double* ps = part + (long long)split * (ntile * (ntile + 1) / 2) * (GT * GT);
    const int ti0 = 2 * I, tj0 = 2 * J, w = warp;
    switch (kind) {
        case K_OFF2:        // warp: rows 64 (w / 4) x columns 32 (w % 4)
            gram_mma<0>(fa + (w >> 2) * 64 * GSTR, fb + (w & 3) * 32 * GSTR, full, empty, nstage_total, pr, lane, ps,
                        ntile, ti0, tj0, (w >> 2) * 8, (w & 3) * 4);
            break;
        case K_OFF1:        // warp: rows 32 (w / 2) x columns 32 (w % 2)
            gram_mma<1>(fa + (w >> 1) * 32 * GSTR, fb + (w & 1) * 32 * GSTR, full, empty, nstage_total, pr, lane, ps,
                        ntile, ti0, tj0, (w >> 1) * 4, (w & 1) * 4);
            break;
        case K_DIAG2:
            if (w < 4)      // the off-diagonal tile: rows 0-63 x rows 64-127 of the A region
                gram_mma<1>(fa + (w >> 1) * 32 * GSTR, fa + (GT + (w & 1) * 32) * GSTR, full, empty, nstage_total, pr,
                            lane, ps, ntile, ti0, tj0, (w >> 1) * 4, 8 + (w & 1) * 4);
            else if (w & 1) // the halves of the two diagonal tiles
                gram_mma<3>(fa + ((w - 4) >> 1) * GT * GSTR, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0,
                            tj0, ((w - 4) >> 1) * 8, ((w - 4) >> 1) * 8);
            else
                gram_mma<2>(fa + ((w - 4) >> 1) * GT * GSTR, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0,
                            tj0, ((w - 4) >> 1) * 8, ((w - 4) >> 1) * 8);
            break;
        default:            // K_DIAG1: the quarters of the last tile's diagonal
            if (w == 0) gram_mma<4>(fa, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0, tj0, 0, 0);
            else if (w == 1) gram_mma<5>(fa, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0, tj0, 0, 0);
            else if (w == 2) gram_mma<6>(fa, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0, tj0, 0, 0);
            else gram_mma<7>(fa, fa, full, empty, nstage_total, pr, lane, ps, ntile, ti0, tj0, 0, 0);
    }
}

// One thread per element of a tile pair (grid: pairs x GT*GT/GRED_THREADS): the split partials of an element are summed
// in split order.  One CTA per pair (15 CTAs at N = 300) left most SMs idle while it read the partials.  A diagonal
// tile's partials hold only its blocks on and above the block diagonal: an element below them reads its mirror.
constexpr int GRED_THREADS = 256;
__global__ void __launch_bounds__(GRED_THREADS) gram_reduce_kernel(const double* __restrict__ part, int npair,
                                                                   int nsplit, int ntile, int N, double* __restrict__ G) {
    const int pair = blockIdx.x;
    int ti = 0, rem = pair, row = ntile;
    while (rem >= row) { rem -= row; --row; ++ti; }
    const int tj = ti + rem;
    const int e = blockIdx.y * GRED_THREADS + threadIdx.x;
    const int er = e / GT, ec = e % GT;
    const int r = ti * GT + er, cc = tj * GT + ec;
    if (r >= N || cc >= N) return;
    const int es = (ti == tj && er / 8 > ec / 8) ? ec * GT + er : e;
    const double* src = part + (long long)pair * (GT * GT) + es;
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

extern "C" int plsb200_gram_stack_fuses(int N, int K) {
    return N > 0 && K >= 0 && cdiv(N + K, GT) == cdiv(N, GT);
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
    int probe = 0;
#ifdef PLSB_PROBES
    probe = getenv("PLSB200_GRAM_PROBE") ? atoi(getenv("PLSB200_GRAM_PROBE")) : 0;
#endif
    const size_t smem = ((size_t)GSTAGES * GSTAGE_ELEMS * sizeof(T) + 7) / 8 * 8 + 2 * GSTAGES * sizeof(uint64_t);
    constexpr int V = 16 / (int)sizeof(T);      // elements of a 16-byte copy
    const bool vec = ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && (ldx % V == 0) &&
                     (n2 == 0 || (((reinterpret_cast<uintptr_t>(X2) & 15) == 0) && (ld2 % V == 0)));
    const unsigned grid = (unsigned)(g.ctas * g.nsplit);
    if (vec) {
        PLSB_CUDA(cudaFuncSetAttribute(gram_partial_kernel<T, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gram_partial_kernel<T, V><<<grid, GTHREADS, smem, st>>>(X, N, p, ldx, X2, n1, ld2, g.chunk, g.ntile, g.nsplit,
                                                                (double*)workspace, probe);
    } else {
        PLSB_CUDA(cudaFuncSetAttribute(gram_partial_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gram_partial_kernel<T, 1><<<grid, GTHREADS, smem, st>>>(X, N, p, ldx, X2, n1, ld2, g.chunk, g.ntile, g.nsplit,
                                                                (double*)workspace, probe);
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
