// The closures of the fused "wcsph" step as device functors — balance of
// wcsph_perturbed_witch.jl:195-303 folded into two pair passes (see DESIGN.md §4) — and the
// helpers they share with the operator menu in pair_ops.cu.  Kept in a header so that the
// pair-list kernels and these closures can also be compiled for the host by the emulation
// harness of the CPU test suite (tests/emu/), which checks them against the oracle.
//
// Arithmetic: compiled with -fmad=false; every product/sum is written in the reference's
// evaluation order (Julia's n-ary * and + fold left).
#pragma once
#include <math.h>

#include "kernels_sph.cuh"
#include "q_access.cuh"
#include "sphmw_internal.h"


// wcsph_perturbed_witch.jl:177-189
__device__ __forceinline__ double background_density(const Params &c, double y) {
    return c.rho0 * exp(-y * c.g / (c.R_mass * c.T_bg));
}
__device__ __forceinline__ double background_pressure(const Params &c, double y) {
    double rho_bg = background_density(c, y);
    return c.R_mass * c.T_bg * rho_bg;
}
__device__ __forceinline__ double background_pot_temperature(const Params &c, double y) {
    double P_bg = background_pressure(c, y);
    return c.T_bg * pow((c.T_bg * c.R_gas * c.rho0) / P_bg, 2.0 / 7.0);
}

// ---- the two unary closures of the step's kick and drift ------------------------------------
#define FLD(slot) f.s[slot][p]

// accelerate!  wcsph_perturbed_witch.jl:298-303 (+ buyoancy_force :253-256,
// damping_structure :245-251).  Vector arithmetic per component, as StaticArrays
// does: ((-g*e_a)*rho')/rho, e = VECY.
template <bool HAS_DV>
struct U_wcsph_accelerate {
    template <int DIM>
    static __device__ void apply(const Fields &f, const Params &c, int64_t p) {
        if (FLD(S_TYPE) == c.fluid) {
            const double rho_p = FLD(S_RHO_P), rho = FLD(S_RHO);
            const bool sponge = FLD(S_X1) >= c.sponge_z0;
            const double hdt = 0.5 * c.dt;
            {
                double dv = HAS_DV ? FLD(S_DV0) : 0.0;
                double buoy = -c.g * 0.0 * rho_p / rho;
                double damp = sponge ? c.sponge_y * 0.0 : 0.0;
                FLD(S_V0) += hdt * (dv + buoy + damp);
            }
            {
                double dv = HAS_DV ? FLD(S_DV1) : 0.0;
                double buoy = -c.g * 1.0 * rho_p / rho;
                double damp = sponge ? c.sponge_y * 1.0 : 0.0;
                FLD(S_V1) += hdt * (dv + buoy + damp);
            }
            if (DIM == 3) {
                double dv = HAS_DV ? FLD(S_DV2) : 0.0;
                double buoy = -c.g * 0.0 * rho_p / rho;
                double damp = sponge ? c.sponge_y * 0.0 : 0.0;
                FLD(S_V2) += hdt * (dv + buoy + damp);
            }
        }
        if (HAS_DV) {
            FLD(S_DV0) = 0.0;
            FLD(S_DV1) = 0.0;
            if (DIM == 3) FLD(S_DV2) = 0.0;
        }
    }
};
// move!  :292-296
struct U_wcsph_move {
    template <int DIM>
    static __device__ void apply(const Fields &f, const Params &c, int64_t p) {
        if (FLD(S_TYPE) == c.fluid) {
            FLD(S_X0) += c.dt * FLD(S_V0);
            FLD(S_X1) += c.dt * FLD(S_V1);
            if (DIM == 3) FLD(S_X2) += c.dt * FLD(S_V2);
        }
    }
};
#undef FLD

#define PF(slot) f.s[slot][p]
#define QF(slot) f.s[slot][q]

// particles outside the column range a pass covers (slab mode: ghost columns) are skipped
struct PairOpBase {
    template <int DIM>
    static __device__ void skip(const Fields &, const Fields &, int64_t) {}
    // packed neighbour records (pair_list.cuh): 0 the operator does not use them, 1 it needs
    // record A, 2 it needs A, B, C
    static constexpr int REC_KIND = 0;
    // true only where finish() provably discards the pair sums of a particle whose type is not
    // fluid: the replaying pass then skips the pair loop of such particles (pair_list.cuh
    // k_binary_list_fluid) and runs init() + finish() alone, which leaves the same bits behind
    static constexpr bool PAIRS_FOR_FLUID_ONLY = false;
    // run by the list and walk kernels right after finish(), with the grid at hand
    template <int DIM>
    __device__ void after(const Grid &, const Fields &, const Params &, int64_t) const {}
    // shared-memory tiles (pair_tile.cuh): number of field arrays the operator stages (0: the
    // operator has no tiled variant)
    template <int DIM>
    __host__ __device__ static constexpr int tile_fields() { return 0; }
};

// what the fused density pass leaves behind for p (shared by the strict and fast variants)
template <int DIM>
__device__ __forceinline__ void wcsph_density_finish(const Fields &f, const Params &c, int64_t p, double rho) {
    double y = PF(S_X1);
    double rbg = background_density(c, y);  // finalize_density!
    double rho_p = rho - rbg;
    double rfl = jl_max(rho, c.rho_floor);  // update_smoothing!
    double m = PF(S_M);
    double hn = DIM == 2 ? c.eta * sqrt(m / rfl) : c.eta * cbrt(m / rfl);
    double pbg = c.R_mass * c.T_bg * rbg;  // compute_pressure! (same rho_bg(y) value)
    double pp = sph_pow2(c.c) * rho_p;
    double P = pbg + pp;
    PF(S_RHO) = rho;
    PF(S_RHO_BG) = rbg;
    PF(S_RHO_P) = rho_p;
    PF(S_H) = hn;
    PF(S_P_BG) = pbg;
    PF(S_P_P) = pp;
    PF(S_P) = P;
    PF(S_PR2) = pp / sph_pow2(rfl);
    PF(S_CS) = sqrt(c.gamma * P / rfl);
}
// accelerate! folded into the force pass's finish() (wcsph_perturbed_witch.jl:298-303)
template <int DIM>
__device__ __forceinline__ void wcsph_force_finish(const Fields &f, const Fields &out, const Params &c, int64_t p,
                                                   double v0, double v1, double v2, double dv0, double dv1,
                                                   double dv2) {
    double n0 = v0, n1 = v1, n2 = v2;
    if (PF(S_TYPE) == c.fluid) {
        const double rho_p = PF(S_RHO_P), rho = PF(S_RHO);
        const bool sponge = PF(S_X1) >= c.sponge_z0;
        const double hdt = 0.5 * c.dt;
        n0 = v0 + hdt * (dv0 + -c.g * 0.0 * rho_p / rho + (sponge ? c.sponge_y * 0.0 : 0.0));
        n1 = v1 + hdt * (dv1 + -c.g * 1.0 * rho_p / rho + (sponge ? c.sponge_y * 1.0 : 0.0));
        if (DIM == 3)
            n2 = v2 + hdt * (dv2 + -c.g * 0.0 * rho_p / rho + (sponge ? c.sponge_y * 0.0 : 0.0));
    }
    out.s[S_V0][p] = n0;
    out.s[S_V1][p] = n1;
    if (DIM == 3) out.s[S_V2][p] = n2;
}

// fields the two fused passes stage in a shared-memory tile (pair_tile.cuh), in array order.
// Density: x, y, (z), m.  Force: x, y, (z), vx, vy, (vz), h, m, P'/rho^2 and, in 2D where the
// tile is small, rho and c_s as well (3D: those two are gathered from global memory, only on the
// artificial-viscosity branch).
template <int DIM>
__host__ __device__ constexpr int wcsph_density_tile_index(int slot) {
    return slot == S_X0 ? 0 : slot == S_X1 ? 1 : (DIM == 3 && slot == S_X2) ? 2 : slot == S_M ? DIM : -1;
}
template <int DIM>
__host__ __device__ constexpr int wcsph_force_tile_index(int slot) {
    return slot == S_X0 ? 0 : slot == S_X1 ? 1 : (DIM == 3 && slot == S_X2) ? 2
         : slot == S_V0 ? DIM : slot == S_V1 ? DIM + 1 : (DIM == 3 && slot == S_V2) ? DIM + 2
         : slot == S_H ? 2 * DIM : slot == S_M ? 2 * DIM + 1 : slot == S_PR2 ? 2 * DIM + 2
         : (DIM == 2 && slot == S_RHO) ? 2 * DIM + 3 : (DIM == 2 && slot == S_CS) ? 2 * DIM + 4 : -1;
}

// ---- fused operators of the fast path (sphmw_step, scheme "wcsph") --------
// reset_density! + compute_density! + finalize_density! + update_smoothing! +
// compute_pressure!  (wcsph_perturbed_witch.jl:316-323) in one pass, plus the
// per-particle invariants of the pair force.
struct B_wcsph_density_fused : PairOpBase {
    static constexpr int REC_KIND = 1;
    template <int DIM>
    __host__ __device__ static constexpr int tile_fields() { return DIM + 1; }
    template <int DIM>
    __host__ __device__ static constexpr int tile_index(int slot) { return wcsph_density_tile_index<DIM>(slot); }
    double rho, hp;
    template <int DIM>
    __device__ void init(const Fields &f, const Params &, int64_t p) {
        rho = 0.0;  // reset_density!
        hp = PF(S_H);
    }
    template <int DIM, class Q>
    __device__ void pair_q(const Params &, const Q &q, double, double, double, double r) {
        rho += QG(S_M) * sph_W<DIM>(hp, r);
    }
    template <int DIM>
    __device__ void pair(const Fields &f, const Params &c, int64_t, int64_t q, double dx, double dy,
                         double dz, double r) {
        pair_q<DIM>(c, GlobalQ{f, q}, dx, dy, dz, r);
    }
    template <int DIM>
    __device__ void finish(const Fields &f, const Fields &, const Params &c, int64_t p) {
        wcsph_density_finish<DIM>(f, c, p, rho);
    }
};

// balance_of_momentum! + accelerate!  (wcsph_perturbed_witch.jl:330-331).
// Dv starts at 0 (accelerate! zeroed it) and is never stored; the new velocity
// goes to the `out` field set because other threads still read the old one.
struct B_wcsph_momentum_fused : PairOpBase {
    static constexpr int REC_KIND = 2;
    // wcsph_force_finish keeps the old velocity of every non-fluid particle
    static constexpr bool PAIRS_FOR_FLUID_ONLY = true;
    template <int DIM>
    __host__ __device__ static constexpr int tile_fields() { return DIM == 2 ? 9 : 9; }
    template <int DIM>
    __host__ __device__ static constexpr int tile_index(int slot) { return wcsph_force_tile_index<DIM>(slot); }
    double dv0, dv1, dv2, v0, v1, v2, hp, prho, pr2, cs;
    // the velocity is double-buffered: a skipped (ghost) particle carries its value over
    template <int DIM>
    static __device__ void skip(const Fields &f, const Fields &out, int64_t p) {
        out.s[S_V0][p] = f.s[S_V0][p];
        out.s[S_V1][p] = f.s[S_V1][p];
        if (DIM == 3) out.s[S_V2][p] = f.s[S_V2][p];
    }
    template <int DIM>
    __device__ void init(const Fields &f, const Params &c, int64_t p) {
        dv0 = dv1 = dv2 = 0.0;
        v0 = PF(S_V0);
        v1 = PF(S_V1);
        v2 = DIM == 3 ? PF(S_V2) : 0.0;
        hp = PF(S_H);
        prho = jl_max(PF(S_RHO), c.rho_floor);
        pr2 = PF(S_PR2);
        cs = PF(S_CS);
    }
    template <int DIM, class Q>
    __device__ void pair_q(const Params &c, const Q &q, double dx, double dy, double dz, double r) {
        double vx = v0 - QG(S_V0), vy = v1 - QG(S_V1);
        double dot_product = dx * vx + dy * vy;
        if (DIM == 3) {
            double vz = v2 - QG(S_V2);
            dot_product = dot_product + dz * vz;
        }
        double h_ij = 0.5 * (hp + QG(S_H));
        double ker = sph_rDW<DIM>(h_ij, r);
        double qm = QG(S_M);
        double fc = -qm * (pr2 + QG(S_PR2)) * ker;
        dv0 += fc * dx;
        dv1 += fc * dy;
        if (DIM == 3) dv2 += fc * dz;
        if (dot_product < 0.0) {
            double qrho = q.rho_floored(c);
            double c_ij = 0.5 * (cs + QG(S_CS));
            double rho_ij = 0.5 * (prho + qrho);
            double mu_ij = (h_ij * dot_product) / (r * r + c.eps * h_ij * h_ij);
            double pi_ij = (-c.alpha * c_ij * mu_ij + c.beta * mu_ij * mu_ij) / rho_ij;
            double fv = -qm * pi_ij * ker;
            dv0 += fv * dx;
            dv1 += fv * dy;
            if (DIM == 3) dv2 += fv * dz;
        }
    }
    template <int DIM>
    __device__ void pair(const Fields &f, const Params &c, int64_t, int64_t q, double dx, double dy,
                         double dz, double r) {
        pair_q<DIM>(c, GlobalQ{f, q}, dx, dy, dz, r);
    }
    template <int DIM>
    __device__ void finish(const Fields &f, const Fields &out, const Params &c, int64_t p) {
        wcsph_force_finish<DIM>(f, out, c, p, v0, v1, v2, dv0, dv1, dv2);
    }
};
// Force pass of every step of a multi-step call but the last: after the kick that ends step n, the
// same thread applies the accelerate! and move! that open step n+1 (wcsph_perturbed_witch.jl:311-312)
// — the very closures the unary kernels run, on a view whose x and v live in the `out` buffers,
// because neighbours still read the old positions and velocities.  Saves two sweeps over the
// particles per step; per-particle operations, so no bit changes.
template <class Base>
struct B_force_advance : Base {
    template <int DIM>
    static __device__ void skip(const Fields &f, const Fields &out, int64_t p) {
        Base::template skip<DIM>(f, out, p);
        out.s[S_X0][p] = f.s[S_X0][p];
        out.s[S_X1][p] = f.s[S_X1][p];
        if (DIM == 3) out.s[S_X2][p] = f.s[S_X2][p];
    }
    template <int DIM>
    __device__ void finish(const Fields &f, const Fields &out, const Params &c, int64_t p) {
        Base::template finish<DIM>(f, out, c, p);  // new velocity -> out
        Fields mix = f;
        for (int s = S_X0; s <= S_X2; ++s) mix.s[s] = out.s[s];
        for (int s = S_V0; s <= S_V2; ++s) mix.s[s] = out.s[s];
        mix.s[S_X0][p] = f.s[S_X0][p];
        mix.s[S_X1][p] = f.s[S_X1][p];
        if (DIM == 3) mix.s[S_X2][p] = f.s[S_X2][p];
        U_wcsph_accelerate<false>::template apply<DIM>(mix, c, p);
        U_wcsph_move::template apply<DIM>(mix, c, p);
        if (c.esc_counter) {
            const long long i = (long long)floor(mix.s[S_X0][p] / c.esc_h) - c.esc_phase;
            if (i < c.esc_lo || i >= c.esc_hi) atomicAdd(c.esc_counter, 1u);
        }
    }
    // whole-domain call: the next cell list's key of the new position (k_keys of the next build, which
    // then skips that launch; cell_list.cu)
    template <int DIM>
    __device__ void after(const Grid &g, const Fields &out, const Params &c, int64_t p) const {
        if (c.key_out)
            cell_key_whole<DIM>(g, out.s[S_X0][p], out.s[S_X1][p], DIM == 3 ? out.s[S_X2][p] : 0.0, p, c.key_out,
                                c.cellx_out, c.key_removed, c.key_removed_cap, c.key_idx);
    }
};

// ---- fast-arithmetic variants of the two fused passes (SPHMW_FLAG_FAST_MATH) ----------
// Same neighbour set (the cut-off test stays exact) and the same summation ORDER, but the
// closure bodies use fused multiply-adds, reciprocals instead of divisions and one rsqrt,
// like the reference's own @fastmath kernels (kernels.jl:108-195).  Per particle, rho, h, P and
// v stay as close to an extended-precision evaluation as the strict path's: the median error is
// below 1.0 (rho) and 0.6 (v) units of 2^-53 times the sum of the pair terms' magnitudes
// (tests/test_xp_wcsph_emulated.py, tests/test_gpu_xp_wcsph.py; DESIGN.md §2) — while the FP64
// instruction count of the accepted-pair path drops ~2.5x.  Results remain deterministic and
// independent of the number of ranks (the code path is the same everywhere).
__device__ __forceinline__ double fast_sqrt_pos(double a) {
    // a > 0 finite in the accepted-pair path (a == 0 only for coincident particles)
    if (a <= 0.0) return a == 0.0 ? 0.0 : sqrt(a);
    double y = rsqrt(a);
    double r = a * y;
    return fma(fma(-r, r, a), 0.5 * y, r);  // one Newton step: ~0.5 ulp
}

struct B_wcsph_density_fast : PairOpBase {
    static constexpr int REC_KIND = 1;
    template <int DIM>
    __host__ __device__ static constexpr int tile_fields() { return DIM + 1; }
    template <int DIM>
    __host__ __device__ static constexpr int tile_index(int slot) { return wcsph_density_tile_index<DIM>(slot); }
    double rho, hp, inv_h, cw;
    template <int DIM>
    __device__ void init(const Fields &f, const Params &, int64_t p) {
        rho = 0.0;
        hp = PF(S_H);
        inv_h = 1.0 / hp;
        // 7/pi / h^2  or  21/(2 pi) / h^3
        cw = DIM == 2 ? 2.228169203286535 * (inv_h * inv_h) : 3.3422538049298023 * (inv_h * inv_h * inv_h);
    }
    template <int DIM, class Q>
    __device__ void pair_q(const Params &, const Q &q, double dx, double dy, double dz, double) {
        double r2 = fma(dx, dx, dy * dy);
        if (DIM == 3) r2 = fma(dz, dz, r2);
        double x = fast_sqrt_pos(r2) * inv_h;
        if (x > 1.0) return;  // kernels.jl:110-112
        double t = 1.0 - x;
        double t2 = t * t;
        double w = cw * (t2 * t2) * fma(4.0, x, 1.0);
        rho = fma(QG(S_M), w, rho);
    }
    template <int DIM>
    __device__ void pair(const Fields &f, const Params &c, int64_t, int64_t q, double dx, double dy,
                         double dz, double r) {
        pair_q<DIM>(c, GlobalQ{f, q}, dx, dy, dz, r);
    }
    template <int DIM>
    __device__ void finish(const Fields &f, const Fields &, const Params &c, int64_t p) {
        wcsph_density_finish<DIM>(f, c, p, rho);
    }
};

struct B_wcsph_momentum_fast : PairOpBase {
    static constexpr int REC_KIND = 2;
    static constexpr bool PAIRS_FOR_FLUID_ONLY = true;  // as B_wcsph_momentum_fused
    template <int DIM>
    __host__ __device__ static constexpr int tile_fields() { return DIM == 2 ? 9 : 9; }
    template <int DIM>
    __host__ __device__ static constexpr int tile_index(int slot) { return wcsph_force_tile_index<DIM>(slot); }
    double dv0, dv1, dv2, v0, v1, v2, hp, prho, pr2, cs;
    template <int DIM>
    static __device__ void skip(const Fields &f, const Fields &out, int64_t p) {
        out.s[S_V0][p] = f.s[S_V0][p];
        out.s[S_V1][p] = f.s[S_V1][p];
        if (DIM == 3) out.s[S_V2][p] = f.s[S_V2][p];
    }
    template <int DIM>
    __device__ void init(const Fields &f, const Params &c, int64_t p) {
        dv0 = dv1 = dv2 = 0.0;
        v0 = PF(S_V0);
        v1 = PF(S_V1);
        v2 = DIM == 3 ? PF(S_V2) : 0.0;
        hp = PF(S_H);
        prho = jl_max(PF(S_RHO), c.rho_floor);
        pr2 = PF(S_PR2);
        cs = PF(S_CS);
    }
    template <int DIM, class Q>
    __device__ void pair_q(const Params &c, const Q &q, double dx, double dy, double dz, double) {
        double r2 = fma(dx, dx, dy * dy);
        double dot_product = fma(dy, v1 - QG(S_V1), dx * (v0 - QG(S_V0)));
        if (DIM == 3) {
            r2 = fma(dz, dz, r2);
            dot_product = fma(dz, v2 - QG(S_V2), dot_product);
        }
        double h_ij = 0.5 * (hp + QG(S_H));
        double inv_h = 1.0 / h_ij;
        double x = fast_sqrt_pos(r2) * inv_h;
        if (x > 1.0) return;  // rDwendland: 0 outside its own support (kernels.jl:142-144)
        double t = 1.0 - x;
        double ih2 = inv_h * inv_h;
        double ih4 = ih2 * ih2;
        // -140/pi (1-x)^3 / h^4   or   -210/pi (1-x)^3 / h^5
        double ker = DIM == 2 ? -44.563384065730695 * (t * t * t) * ih4
                              : -66.84507609859604 * (t * t * t) * (ih4 * inv_h);
        double qm = QG(S_M);
        double fc = -qm * (pr2 + QG(S_PR2)) * ker;
        if (dot_product < 0.0) {
            double qrho = q.rho_floored(c);
            double c_ij = 0.5 * (cs + QG(S_CS));
            double rho_ij = 0.5 * (prho + qrho);
            // mu = h dot / D,  pi = (-alpha c mu + beta mu^2) / rho_ij, with one reciprocal
            double D = fma(c.eps * h_ij, h_ij, r2);
            double R = 1.0 / (D * rho_ij);
            double hd = h_ij * dot_product;
            double mu = hd * rho_ij * R;
            double pi_ij = hd * R * fma(c.beta, mu, -c.alpha * c_ij);
            fc = fma(-qm * pi_ij, ker, fc);
        }
        dv0 = fma(fc, dx, dv0);
        dv1 = fma(fc, dy, dv1);
        if (DIM == 3) dv2 = fma(fc, dz, dv2);
    }
    template <int DIM>
    __device__ void pair(const Fields &f, const Params &c, int64_t, int64_t q, double dx, double dy,
                         double dz, double r) {
        pair_q<DIM>(c, GlobalQ{f, q}, dx, dy, dz, r);
    }
    template <int DIM>
    __device__ void finish(const Fields &f, const Fields &out, const Params &c, int64_t p) {
        wcsph_force_finish<DIM>(f, out, c, p, v0, v1, v2, dv0, dv1, dv2);
    }
};
#undef PF
#undef QF
