// Launch plan of the register-resident FP64 bootstrap GEMM (boot.cu), shared with the collapsed-bootstrap quadratic
// form (boot_quad.cu), which streams its coefficients through the same ring in the same B-fragment / period order.
#pragma once
#include <math.h>

#include "common.cuh"

namespace plsb {

constexpr int BM_WARPS = 8;          // consumer warps per CTA
constexpr int BM_THREADS = BM_WARPS * 32;
constexpr int BM_VOX = BM_WARPS * 8; // voxels per CTA

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
    // smallest padded K that divides a 24-, 16- or 8-column period; prefer wider periods (more ILP)
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
    if (!best_kp) return false;
    b.Kp = best_kp; b.nblk = best_blk; b.nb = 8 * best_blk / best_kp;
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

}  // namespace plsb
