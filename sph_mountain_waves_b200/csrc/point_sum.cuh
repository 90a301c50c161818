// Point sums — the `sum(sys, f, x)` of src/core.jl:240-291 on the device: an SPH sum evaluated at a
// location that is not a particle (sampling w, u or θ′ on a section, say).  It is _apply_binary!
// (core.jl:94-112) with a point in place of p:
//   home cell  find_key(x) with the particle formula (cell_ijk_whole: IEEE x/h, floor, minus key_phase);
//   cells      the key_diff cells in the reference's order, only 1 <= key + dkey <= key_max checked
//              (neighbour_pkey), so face cells wrap exactly as they do for particles;
//   order      each cell in stored order (reference index descending);
//   accepted   r <= sys.h (Grid::r2_max: the same set, sqrt only for accepted particles), and NO
//              self-exclusion: a particle at r = 0 counts.
// Each op's sum starts at 0.0 and adds its term in that order, the terms folded left to right as Julia's
// `*` does (this file is compiled with -fmad=false):
//   count 1.0 | mW m*W | mW*f (m*f)*W | VW (m/rho)*W | VW*f ((m/rho)*f)*W,   W = wendland2/3(sys.h, r).
// A point outside the closed box (NaN coordinates included, and in 2D a third coordinate != 0) gets NaN.
// Both physical cell orders (zrun and x-chunked) are walked through pkey_ijk; in the zrun order a point
// whose home cell is not at a face walks 9 (3 in 2D) contiguous runs instead of 27 (9) cells.
// Host-includable, so the CPU tests run these kernels thread by thread (tests/emu/emu_point_sum.cpp).
#pragma once
#include "kernels_sph.cuh"
#include "sphmw_internal.h"

enum PointOpKind : int { PT_COUNT = 0, PT_MW, PT_MW_F, PT_VW, PT_VW_F };

// the decoded ops of one call, passed by value.  A null pointer is a field never written: it reads 0.
struct PointOps {
    int n;
    bool need_v;  // some op needs m/rho
    int kind[SPHMW_POINT_OPS_MAX];
    const double *f[SPHMW_POINT_OPS_MAX];  // the field of PT_MW_F / PT_VW_F
    const double *x0, *x1, *x2, *m, *rho;  // particles, physical order
};

// home cell of a point, or false: outside the box (then every output is NaN)
template <int DIM>
__host__ __device__ __forceinline__ bool point_home(const Grid &g, double x, double y, double z, CellCoord &c) {
    if (DIM == 2 && !(z == 0.0)) return false;  // the 2D box is 0 <= x[3] <= 0 (geometry.jl:24-30)
    int i, j, k;
    if (!cell_ijk_whole<DIM>(g, x, y, z, i, j, k)) return false;
    c.i = i;
    c.j = j;
    c.k = k;
    c.rest = j + (int)g.lim[1] * k;
    return true;
}

// physical home key of every point (pkey_max: outside) and the identity order the sort permutes
template <int DIM>
__global__ void k_point_keys(Grid g, const double *__restrict__ pts, int64_t n, uint32_t *__restrict__ key,
                             uint32_t *__restrict__ order) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    CellCoord c;
    key[i] = point_home<DIM>(g, pts[i], pts[n + i], pts[2 * n + i], c) ? pkey_ijk(g, c.i, c.j, c.k)
                                                                       : (uint32_t)g.pkey_max;
    order[i] = (uint32_t)i;
}

// one thread per point, points taken in `order` (sorted by home cell: a warp's points share cells);
// out[o*n + i] for the caller's index i
template <int DIM>
__global__ void __launch_bounds__(128)
k_point_sum(PointOps ops, Grid g, const uint32_t *__restrict__ cell_start, const double *__restrict__ pts, int64_t n,
            const uint32_t *__restrict__ order, double *__restrict__ out) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t i = order[t];
    const double px = pts[i], py = pts[n + i], pz = pts[2 * n + i];
    CellCoord home;
    if (!point_home<DIM>(g, px, py, pz, home)) {
        for (int o = 0; o < ops.n; ++o) out[o * n + i] = (double)NAN;
        return;
    }
    double acc[SPHMW_POINT_OPS_MAX];
#pragma unroll
    for (int o = 0; o < SPHMW_POINT_OPS_MAX; ++o) acc[o] = 0.0;
    // candidates [b, e) of the cell order, accumulated in that order
    auto visit = [&](uint32_t b, uint32_t e) {
        for (uint32_t q = b; q < e; ++q) {
            // dist(x, q) — core.jl:8-10, algebra.jl:49-60: left to right, no FMA
            const double dx = px - ops.x0[q];
            const double dy = py - ops.x1[q];
            double r2 = dx * dx + dy * dy;
            if (DIM == 3) {
                const double dz = pz - ops.x2[q];
                r2 = r2 + dz * dz;
            }
            if (r2 > g.r2_max) continue;  // r > sys.h; no p == q test
            const double W = sph_W<DIM>(g.h, sqrt(r2));
            const double mq = ops.m ? ops.m[q] : 0.0;
            const double vq = ops.need_v ? mq / (ops.rho ? ops.rho[q] : 0.0) : 0.0;
#pragma unroll
            for (int o = 0; o < SPHMW_POINT_OPS_MAX; ++o) {
                if (o < ops.n) {
                    const double fq = ops.f[o] ? ops.f[o][q] : 0.0;
                    double term;
                    switch (ops.kind[o]) {
                        case PT_COUNT: term = 1.0; break;
                        case PT_MW: term = mq * W; break;
                        case PT_MW_F: term = (mq * fq) * W; break;
                        case PT_VW: term = vq * W; break;
                        default: term = (vq * fq) * W; break;
                    }
                    acc[o] = acc[o] + term;
                }
            }
        }
    };
    const int lx = (int)g.lim[0], ly = (int)g.lim[1], lz = (int)g.lim[2];
    const bool interior = g.zrun && home.i >= 1 && home.i + 1 < lx && home.j >= 1 && home.j + 1 < ly &&
                          (DIM == 2 || (home.k >= 1 && home.k + 1 < lz));
    if (interior) {
        // zrun order, no cell near a face: the three cells of the innermost key_diff loop (dk in 3D, dj in
        // 2D) are one contiguous run stored in visiting order, so 9 (3) runs replace 27 (9) cells
        for (int di = -1; di <= 1; ++di)
            for (int dj = DIM == 3 ? -1 : 0; dj <= (DIM == 3 ? 1 : 0); ++dj) {
                const unsigned c = pkey_ijk(g, home.i + di, home.j + dj, home.k);
                visit(cell_start[c - 1], cell_start[c + 2]);
            }
    } else {
        for (int d = 0; d < g.ndiff; ++d) {
            unsigned nk;
            if (!neighbour_pkey(g, home, d, nk)) continue;  // core.jl:98 — no per-axis wrap check
            visit(cell_start[nk], cell_start[nk + 1]);
        }
    }
#pragma unroll
    for (int o = 0; o < SPHMW_POINT_OPS_MAX; ++o)
        if (o < ops.n) out[o * n + i] = acc[o];
}
