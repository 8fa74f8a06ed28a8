// K1 fast mode: the Gram matrix G = X X^T on the 5th-generation tensor cores (tcgen05, kind::tf32) with the 3xTF32
// split (x = xh + xl, both TF32-exact; xh.xh + xh.xl + xl.xh accumulated in FP32 in tensor memory).
//
//   G[i, j] = sum_v X[i, v] X[j, v]:   M = rows i, N = rows j, K-dim = voxels -- both operands are X itself, K-major.
//
//   * Operand image (gram_split_tf32_kernel, one pass over X): [block of 16 voxels][hi|lo][row][16 voxels] FP32, every
//     plane in the K-major SWIZZLE_64B order of a shared-memory tile, so a pipeline stage (16 voxels of every row, both
//     planes: 38 KB at 300 rows) is two contiguous bulk copies (cp.async.bulk) and both MMA operands are windows of the
//     same stage: A = the 128 rows of an M tile, B = the rows of its column range.  (The image of the bootstrap GEMM has
//     the voxels as its M dimension; read as an MN-major operand it would need no second image, but for kind::tf32 the
//     hardware only transposes the SWIZZLE_128B_BASE32B layout -- with the transpose bits of the instruction descriptor
//     set on the 64-byte-swizzled image the MMA returns zeros.)
//   * Only the upper block triangle is computed: M tile t (rows 128 t ...) against the columns 128 t ... N.  The
//     accumulators of all M tiles of a 300-row design need 304 + 176 + 48 = 528 TMEM columns, 16 more than an SM
//     has, so there are two kinds of CTAs: kind 0 owns M tile 0, kind 1 the remaining tiles (loading only the rows from
//     128 on); the groups of 128 voxels are dealt round-robin to the CTAs of a kind -- both kinds sweep the image front to
//     back at the same pace -- and the CTA counts of the two kinds are proportional to their column counts, so all CTAs
//     finish together.
//   * Precision: the tensor core truncates when it accumulates, which biases a long sum of like-signed terms (the
//     diagonal of G) by ~3e-8 per accumulation step.  The TMEM accumulators are therefore drained every `dr` groups of
//     128 voxels (192 accumulation steps at dr = 4) into a per-CTA FP32 partial block in global memory (L2-resident) with
//     round-to-nearest vector reductions (REDG.ADD.F32x4; 160 FP32 register accumulators per drain thread do not fit
//     next to the other roles), and the partial blocks are summed over the CTAs in FP64 in a fixed order.
//     Measured against the FP64 Gram: tests/test_gpu_tf32.py::test_gram_tf32.
//   * warps 0-7 = drain (two per TMEM lane quarter, alternate 16-column chunks), warp 8 = producer, warp 9 = MMA
//     issuer + TMEM allocator.  N <= 320 (three M tiles in two CTA kinds); taller designs use the exact kernel.
#include "common.cuh"
#include <stdlib.h>

namespace plsb {

constexpr int GT_KV = 16;                    // voxels per pipeline stage (one block of the image)
constexpr int GT_GROUP = 8;                  // blocks per drain unit (128 voxels)
constexpr int GT_THREADS = 320;
constexpr int GT_PSTRIDE = 320;              // columns of a CTA's partial block
constexpr uint32_t GT_ROW = GT_KV * 4;       // bytes of one row of a plane (64: the SWIZZLE_64B row)

struct GtJob { int arow, brow, nc, co; };    // first A row, first B row (relative to the kind's first row), columns, TMEM column
struct GtArgs {
    const unsigned char* img;
    float* part;
    int npad, nvb, n0, dr, nstage;            // padded rows, voxel blocks (multiple of GT_GROUP), CTAs of kind 0
    uint32_t stage_bytes;
    int r0[2], nr[2], njobs[2], tcols[2];     // per kind: first row / rows staged, M tiles, TMEM columns
    GtJob job[2][2];
};

__device__ __forceinline__ uint64_t gt_desc(uint32_t saddr) {
    // K-major, SWIZZLE_64B: LBO (unused) = 16 B, SBO = 512 B between 8-row groups, version 1, layout type 4
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(512u >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)4 << 61);
}
__device__ __forceinline__ float gt_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// X (N x p, FP64, row-major) -> image [block of 16 voxels][hi|lo][npad rows][16 voxels], each plane in the K-major
// SWIZZLE_64B order: row r, voxel j -> r*64 + ((j/4) ^ ((r/2)&3))*16 + (j%4)*4 bytes.  One thread per (row, block):
// reads one 128-byte line of X, writes one 64-byte row of each plane (consecutive rows = consecutive threads).
// T = float: X stored as float32; its widened value is split, so the planes are those of the widened matrix.
// VEC4 (float32 X whose rows are 16-byte aligned): the 64 bytes of a thread's row segment come in four 16-byte loads.
// With element loads a warp-wide load touches 32 rows for 4 bytes each, twice the instructions per byte of FP64 X:
// measured 0.307 ms (FP64) -> 0.349 ms at the bench shape with element loads, 0.233 ms with VEC4.
template <typename T, bool VEC4 = false>
__global__ void __launch_bounds__(128) gram_split_tf32_kernel(const T* __restrict__ X, int N, long long p,
                                                              long long ldx, int npad, float* __restrict__ img) {
    const int r = blockIdx.y * 128 + threadIdx.x;
    const long long vb = blockIdx.x;
    if (r >= npad) return;
    float hi[GT_KV], lo[GT_KV];
    if constexpr (VEC4) {
        static_assert(sizeof(T) == 4, "16-byte loads of four float32 elements");
#pragma unroll
        for (int c = 0; c < GT_KV / 4; ++c) {
            const long long v = vb * GT_KV + 4 * c;
            float e[4] = {0.f, 0.f, 0.f, 0.f};
            if (r < N && v + 3 < p) {
                const float4 f = __ldg(reinterpret_cast<const float4*>(X + (long long)r * ldx + v));
                e[0] = f.x; e[1] = f.y; e[2] = f.z; e[3] = f.w;
            } else if (r < N) {
#pragma unroll
                for (int t = 0; t < 4; ++t) e[t] = v + t < p ? __ldg(X + (long long)r * ldx + v + t) : 0.f;
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const double x = (double)e[t];
                hi[4 * c + t] = gt_rna((float)x);
                lo[4 * c + t] = gt_rna((float)(x - (double)hi[4 * c + t]));
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < GT_KV; ++j) {
            const long long v = vb * GT_KV + j;
            const double x = (r < N && v < p) ? (double)__ldg(X + (long long)r * ldx + v) : 0.0;
            hi[j] = gt_rna((float)x);
            lo[j] = gt_rna((float)(x - (double)hi[j]));
        }
    }
    float* base = img + ((size_t)vb * 2 * npad + r) * GT_KV;
    const int sw = (r >> 1) & 3;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int pos = c ^ sw;
        *reinterpret_cast<float4*>(base + pos * 4) = make_float4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
        *reinterpret_cast<float4*>(base + (size_t)npad * GT_KV + pos * 4) =
            make_float4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    }
}
__device__ __forceinline__ void gt_mma(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void gt_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void gt_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void gt_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void gt_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void gt_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

__global__ void __launch_bounds__(GT_THREADS, 1) gram_tf32_kernel(const GtArgs a) {
    extern __shared__ unsigned char gt_raw[];
    const uint32_t s0 = smem_u32(gt_raw);
    unsigned char* ring = gt_raw + ((1024u - (s0 & 1023u)) & 1023u);
    __shared__ __align__(8) uint64_t bars[20];
    __shared__ uint32_t tmem_slot;
    uint64_t* full = bars;
    uint64_t* empty = bars + 8;
    uint64_t* tfull = bars + 16;
    uint64_t* tempty = bars + 17;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kind = (int)blockIdx.x < a.n0 ? 0 : 1;
    const int nk = kind == 0 ? a.n0 : (int)gridDim.x - a.n0;            // CTAs of my kind
    const int me = kind == 0 ? (int)blockIdx.x : (int)blockIdx.x - a.n0;
    const int ngrp = a.nvb / GT_GROUP;                                  // groups of 128 voxels
    // groups me, me + nk, me + 2 nk, ...: the CTAs of both kinds sweep the image front to back at the same pace, so the
    // second kind to reach a block finds it in L2
    const int cnt = me < ngrp ? (ngrp - me + nk - 1) / nk : 0;
    const int nbatch = (cnt + a.dr - 1) / a.dr;
    const int nr = a.nr[kind], r0 = a.r0[kind];
    const uint32_t plane_s = (uint32_t)nr * GT_ROW;                    // bytes of one plane in a stage

    if (tid == 0) {
        for (int s = 0; s < a.nstage; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        mbar_init(tfull, 1); mbar_init(tempty, 8);
        mbar_fence_init();
    }
    if (warp == 9) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(&tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    gt_fence_before();
    __syncthreads();
    gt_fence_after();
    const uint32_t tbase = tmem_slot;

    if (warp == 8) {
        // ===================== producer: both planes of the kind's rows, 16 voxels per stage =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int it = 0; it < cnt * GT_GROUP; ++it) {
                const long long vb = (long long)(me + (it / GT_GROUP) * nk) * GT_GROUP + it % GT_GROUP;
                mbar_wait(empty + stage, phase ^ 1u);
                mbar_expect_tx(full + stage, 2u * plane_s);
                unsigned char* dst = ring + (size_t)stage * a.stage_bytes;
                const unsigned char* src = a.img + ((size_t)vb * 2 * a.npad + r0) * GT_ROW;
                bulk_g2s(dst, src, plane_s, full + stage);
                bulk_g2s(dst + plane_s, src + (size_t)a.npad * GT_ROW, plane_s, full + stage);
                if (++stage == a.nstage) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 9) {
        if (lane == 0) {
            // ===================== MMA issuer =====================
            const uint32_t ibase = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 4) << 24);
            const uint64_t d0 = gt_desc(smem_u32(ring));
            const uint64_t stage_step = a.stage_bytes >> 4, plane_step = plane_s >> 4;
            int stage = 0; uint32_t phase = 0, tph = 0;
            const int nj = a.njobs[kind];
            int vt = 0;
            for (int b = 0; b < nbatch; ++b) {
                mbar_wait(tempty, tph ^ 1u);
                gt_fence_after();
                uint32_t accum = 0u;
                const int vend = min(cnt, vt + a.dr);
                for (; vt < vend; ++vt) {
                    for (int sub = 0; sub < GT_GROUP; ++sub) {
                        mbar_wait(full + stage, phase);
                        gt_fence_after();
                        const uint64_t hi = d0 + (uint64_t)stage * stage_step, lo = hi + plane_step;
#pragma unroll
                        for (int ks = 0; ks < GT_KV / 8; ++ks) {
                            for (int j = 0; j < nj; ++j) {
                                const GtJob& jb = a.job[kind][j];
                                const uint64_t ao = (uint64_t)jb.arow * (GT_ROW >> 4) + (uint64_t)ks * 2u;    // k-step: 32 B
                                int done = 0;
                                while (done < jb.nc) {                       // UMMA N <= 256
                                    const int n = min(256, jb.nc - done);
                                    const uint64_t bo = (uint64_t)(jb.brow + done) * (GT_ROW >> 4) + (uint64_t)ks * 2u;
                                    const uint32_t idesc = ibase | ((uint32_t)(n >> 3) << 17);
                                    const uint32_t d = tbase + (uint32_t)(jb.co + done);
                                    gt_mma(d, hi + ao, lo + bo, idesc, accum);
                                    gt_mma(d, hi + ao, hi + bo, idesc, 1u);
                                    gt_mma(d, lo + ao, hi + bo, idesc, 1u);
                                    done += n;
                                }
                            }
                            accum = 1u;
                        }
                        gt_commit(empty + stage);
                        if (++stage == a.nstage) { stage = 0; phase ^= 1u; }
                    }
                }
                gt_commit(tfull);
                tph ^= 1u;
            }
        }
    } else {
        // ===================== drain: TMEM -> this CTA's FP32 partial block in global memory =====================
        // (vector reductions REDG.ADD.F32x4: round-to-nearest adds, fire-and-forget, no register accumulators; every
        // element is only ever touched by this thread, in program order -> deterministic)
        const int quarter = warp & 3, halfc = warp >> 2;
        const int nch = a.tcols[kind] / 16;
        float* out = a.part + ((size_t)blockIdx.x * 128 + quarter * 32 + lane) * GT_PSTRIDE;
        uint32_t tph = 0;
        if (nbatch == 0)                           // a CTA without voxels contributes zeros
            for (int c = halfc; c < nch; c += 2)
#pragma unroll
                for (int e = 0; e < 16; e += 4) *reinterpret_cast<float4*>(out + 16 * c + e) = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int b = 0; b < nbatch; ++b) {
            mbar_wait(tfull, tph);
            gt_fence_after();
            for (int c = halfc; c < nch; c += 2) {
                uint32_t x[16];
                gt_ld16(tbase + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(16 * c), x);
                gt_ld_wait();
                if (b == 0) {                      // the first drain initialises the block
#pragma unroll
                    for (int e = 0; e < 16; e += 4)
                        *reinterpret_cast<float4*>(out + 16 * c + e) =
                            make_float4(__uint_as_float(x[e]), __uint_as_float(x[e + 1]), __uint_as_float(x[e + 2]),
                                        __uint_as_float(x[e + 3]));
                } else {
#pragma unroll
                    for (int e = 0; e < 16; e += 4)
                        asm volatile("red.global.v4.f32.add [%0], {%1, %2, %3, %4};\n" ::"l"(out + 16 * c + e),
                                     "f"(__uint_as_float(x[e])), "f"(__uint_as_float(x[e + 1])),
                                     "f"(__uint_as_float(x[e + 2])), "f"(__uint_as_float(x[e + 3]))
                                     : "memory");
                }
            }
            gt_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
            tph ^= 1u;
        }
    }
    __syncwarp();
    gt_fence_before();
    __syncthreads();
    if (warp == 9) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tbase));
    }
}

// G[i][j] = G[j][i] = sum over the CTAs of the owning kind (fixed order).  One thread per (i, j >= i): consecutive
// threads read consecutive columns of the partial blocks.
__global__ void gram_tf32_reduce_kernel(const GtArgs a, int N, int ncta, double* __restrict__ G, int accumulate) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= N || j < i) return;
    const int t = i / 128, kind = t == 0 ? 0 : 1;
    const GtJob& jb = a.job[kind][t == 0 ? 0 : t - 1];
    const int col = jb.co + (j - 128 * t), L = i - 128 * t;      // (the job's columns start at its own first row)
    const int c0 = kind == 0 ? 0 : a.n0, c1 = kind == 0 ? a.n0 : ncta;
    double s = 0.0;
    for (int b = c0; b < c1; ++b) s += (double)a.part[((size_t)b * 128 + L) * GT_PSTRIDE + col];
    if (accumulate) s += G[(size_t)i * N + j];
    G[(size_t)i * N + j] = s;
    G[(size_t)j * N + i] = s;
}

static bool gt_plan(int N, int64_t p, GtArgs& a, int& ncta, size_t& smem) {
    if (N < 1 || N > 320 || p < 1) return false;
    a.npad = (int)cdiv(N, 16) * 16;
    a.nvb = (int)(cdiv(p, GT_KV * GT_GROUP) * GT_GROUP);
    const int npad = a.npad, nmt = (int)cdiv(N, 128);
    for (int k = 0; k < 2; ++k) { a.r0[k] = 0; a.nr[k] = 0; a.njobs[k] = 0; a.tcols[k] = 0; }
    a.r0[0] = 0; a.nr[0] = npad; a.njobs[0] = 1; a.tcols[0] = npad;
    a.job[0][0] = GtJob{0, 0, npad, 0};
    a.job[0][1] = a.job[1][0] = a.job[1][1] = GtJob{0, 0, 0, 0};
    if (nmt > 1) {
        a.r0[1] = 128; a.nr[1] = npad - 128; a.njobs[1] = nmt - 1;
        int co = 0;
        for (int t = 1; t < nmt; ++t) {
            const int nc = npad - 128 * t;
            a.job[1][t - 1] = GtJob{128 * t - 128, 128 * t - 128, nc, co};
            co += nc;
        }
        a.tcols[1] = co;
    }
    if (a.tcols[0] > GT_PSTRIDE || a.tcols[1] > GT_PSTRIDE) return false;
    const int nsm = num_sms();
    ncta = nsm;
    if (nmt > 1) {
        a.n0 = (int)((double)nsm * a.tcols[0] / (a.tcols[0] + a.tcols[1]) + 0.5);
        if (a.n0 < 1) a.n0 = 1;
        if (a.n0 > nsm - 1) a.n0 = nsm - 1;
    } else {
        a.n0 = nsm;
    }
    a.stage_bytes = 2u * (uint32_t)npad * GT_ROW;             // sized for kind 0 (kind 1 uses a part of each slot)
    const size_t slack = 128 * GT_ROW + 1024;                 // the last M tile's A window may reach 128 rows past its plane
    int ns = (int)((226 * 1024 - 1024 - slack) / a.stage_bytes);   // (static shared memory: barriers)
    if (ns > 8) ns = 8;
    if (ns < 2) return false;
    a.nstage = ns;
    smem = (size_t)ns * a.stage_bytes + slack + 1024;
    return true;
}

}  // namespace plsb

using namespace plsb;

extern "C" size_t plsb200_gram_tf32_image_bytes(int N, int64_t p) {
    GtArgs a; int ncta; size_t smem;
    if (!gt_plan(N, p, a, ncta, smem)) return 0;
    return (size_t)a.nvb * 2 * a.npad * GT_ROW;
}

template <typename T>
static int gram_tf32_split(const T* X, int N, int64_t p, int64_t ldx, void* image, void* stream) {
    PLSB_CHECK_ARG(X && image, "gram_tf32_split: null pointer");
    PLSB_CHECK_ARG(p > 0 && ldx >= p, "gram_tf32_split: bad shape");
    GtArgs a; int ncta; size_t smem;
    if (!gt_plan(N, p, a, ncta, smem)) {
        set_err("gram_tf32_split: unsupported shape N=%d (need 1 <= N <= 320)", N);
        return PLSB200_EUNSUPPORTED;
    }
    dim3 grid((unsigned)a.nvb, (unsigned)cdiv(a.npad, 128));
    if (sizeof(T) == 4 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && ldx % 4 == 0)
        gram_split_tf32_kernel<T, sizeof(T) == 4><<<grid, 128, 0, (cudaStream_t)stream>>>(X, N, p, ldx, a.npad,
                                                                                         (float*)image);
    else
        gram_split_tf32_kernel<T><<<grid, 128, 0, (cudaStream_t)stream>>>(X, N, p, ldx, a.npad, (float*)image);
    PLSB_LAUNCH_CHECK("gram_split_tf32_kernel");
    return PLSB200_OK;
}

extern "C" int plsb200_gram_tf32_split(const double* X, int N, int64_t p, int64_t ldx, void* image, void* stream) {
    return gram_tf32_split(X, N, p, ldx, image, stream);
}

extern "C" int plsb200_gram_tf32_split_x32(const float* X, int N, int64_t p, int64_t ldx, void* image, void* stream) {
    return gram_tf32_split(X, N, p, ldx, image, stream);
}

extern "C" size_t plsb200_gram_tf32_workspace(int N, int64_t p) {
    GtArgs a; int ncta; size_t smem;
    if (!gt_plan(N, p, a, ncta, smem)) return 0;
    return (size_t)ncta * 128 * GT_PSTRIDE * sizeof(float);
}

extern "C" int plsb200_gram_tf32(const void* ximage, int N, int64_t p, double* G, int accumulate, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    PLSB_CHECK_ARG(ximage && G && workspace, "gram_tf32: null pointer");
    GtArgs a; int ncta; size_t smem;
    if (!gt_plan(N, p, a, ncta, smem)) {
        set_err("gram_tf32: unsupported shape N=%d (need 1 <= N <= 320)", N);
        return PLSB200_EUNSUPPORTED;
    }
    const size_t need = (size_t)ncta * 128 * GT_PSTRIDE * sizeof(float);
    if (workspace_bytes < need) {
        set_err("gram_tf32: workspace %zu < %zu bytes", workspace_bytes, need);
        return PLSB200_EWORKSPACE;
    }
    static const char* const env = getenv("PLSB200_GRAM_TF32_DRAIN");       // voxel tiles between drains (default 4)
    a.dr = env ? atoi(env) : 4;
    if (a.dr < 1) a.dr = 1;
    a.img = (const unsigned char*)ximage;
    a.part = (float*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    PLSB_CUDA(cudaFuncSetAttribute(gram_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gram_tf32_kernel<<<ncta, GT_THREADS, smem, st>>>(a);
    PLSB_LAUNCH_CHECK("gram_tf32_kernel");
    gram_tf32_reduce_kernel<<<dim3((unsigned)cdiv(N, 64), (unsigned)N), 64, 0, st>>>(a, N, ncta, G, accumulate);
    PLSB_LAUNCH_CHECK("gram_tf32_reduce_kernel");
    return PLSB200_OK;
}
