// Internal declarations of libsphmw (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "sphmw.h"

// ---------------------------------------------------------------------------
// Particle fields.  One "slot" per scalar component; the union of the driver
// Particle structs (wcsph_perturbed_witch.jl:83-102, hopkins_*:103,
// collapse_dry.jl:74-82, test_collision_2d.jl:37-44) plus two derived per-particle
// invariants of the pair force (S_PR2, S_CS) that only the fused step uses.
// ---------------------------------------------------------------------------
enum Slot : int {
    S_H = 0,
    S_X0, S_X1, S_X2,
    S_M,
    S_V0, S_V1, S_V2,
    S_DV0, S_DV1, S_DV2,
    S_RHO_BG, S_RHO_P, S_RHO,
    S_P_BG, S_P_P, S_P,
    S_TH_BG, S_TH_P, S_TH,
    S_T_BG, S_T_P, S_T,
    S_TYPE,
    S_A, S_A_BG,
    S_DRHO, S_RHO0,
    S_PR2,  // P'/max(rho,floor)^2            (wcsph_perturbed_witch.jl:272)
    S_CS,   // sqrt(gamma*P/max(rho,floor))   (wcsph_perturbed_witch.jl:276)
    S_ENT, S_ENT_D,  // entropy S and entropy density s (legacy/adiabatic_flow_witch.jl:75-76)
    NSLOT
};

struct Fields {
    double *s[NSLOT];
};

// driver constants (wcsph_perturbed_witch.jl:25-75 etc.); names match sphmw_set_param
struct Params {
    double dt, g, c, gamma, alpha, beta, eps, eta, rho0, R_mass, R_gas, T_bg;
    double rho_floor, P_floor, z_t, z_b, gamma_r, fluid;
    double m, nu, mu, gx, gy, gz, kh;
    double dt_pack, c_pack, zeta_pack;
    double U_max, cp, bc_width, x_inflow, dr, inflow;  // legacy flow drivers (isothermal_flow_witch.jl:24-60)
    // derived on the host when a parameter changes
    double sponge_y;  // -gamma_r*sin(pi/2*(1-(z_t-z_b)/z_b))^2  (:245-251)
    double sponge_z0; // z_t - z_b
    // overlapped slab step: the interior force pass also runs the next step's accelerate!/move!
    // (B_force_advance) and counts particles that drift into a column whose halo records were
    // already packed (pair_ops.cu); null otherwise
    uint32_t *esc_counter;
    double esc_h;
    long long esc_phase;
    int esc_lo, esc_hi;  // legal local columns after the drift: [esc_lo, esc_hi)
    // whole-domain multi-step call: the force pass's advance also writes the next cell list's key of the
    // new position (cell_key_whole, B_force_advance::after); null otherwise
    uint32_t *key_out, *cellx_out, *key_removed;
    const uint32_t *key_idx;
    uint32_t key_removed_cap;
};

// neighbour-grid description passed to kernels by value (structs.jl:63-82)
struct Grid {
    double h;
    // largest double whose correctly rounded sqrt is <= h:  sqrt(r2) > h  <=>  r2 > r2_max,
    // so rejected candidates never pay for the FP64 square root (core.jl:104-105)
    double r2_max;
    double box[6];
    long long phase[3];
    long long lim[3];
    long long key_max;
    int key_diff[27];
    int ndiff;
    int dim;
    // PHYSICAL cell order.  The reference key is i + Lx*(j + Ly*k) (structs.jl:102): x fastest
    // over the whole domain length, so one x-y plane of cells can be tens of MB and the three
    // planes a pass needs do not stay in L2.  Physically the cells are therefore ordered in
    // x-chunks of 2^cx_shift columns: pkey = ((i >> s)*rows + rest << s) + (i & mask), with
    // rest = j + Ly*k and rows = Ly*Lz.  Only the storage order changes: neighbour cells are
    // still visited in the reference's key_diff order (nb_di/nb_drest hold each offset's
    // column and row part), so every sum keeps its order.
    int cx_shift;
    long long rows;
    long long pkey_max;
    int nb_di[27];
    int nb_drest[27];
    int nb_dj[27];  // the row part split into its y and z offsets (nb_drest = dj + Ly*dk)
    int nb_dk[27];
    // zrun (the default, DESIGN.md §3): cells stored x-outermost with the INNERMOST axis of the
    // reference's key_diff loops fastest — z in 3D, y in 2D (structs.jl:73-81: `for di, dj, dk`,
    // the last one runs fastest): pkey = i*rows + j*Lz + k.  The three cells (di, dj, -1..1) are
    // then one contiguous run of memory whose order IS the reference's visiting order, so a pair
    // pass walks 9 (3 in 2D) runs instead of 27 (9) cells, and a y-z plane of cells (a few MB)
    // stays in L2.  zrun == 0: the x-chunked order above, kept for the shared-memory variants
    // (SPHMW_FLAG_TILES, SPHMW_FLAG_CELL_PAIRS) that stage x-rows.
    int zrun;
    // slab contexts: ghost columns kept on each side of the owned ones (GHOST_COLS; three with
    // SPHMW_FLAG_GHOST3, which the Hopkins schemes need: their pressure sum reads the NEW smoothing
    // length of a particle's neighbours, i.e. complete density sums one column further out)
    int ghost;
};

#if defined(__CUDACC__) || defined(SPHMW_EMU)
// 32-bit cell arithmetic (all quantities < 2^31: sphmw_create checks pkey_max)
struct CellCoord {
    int i, rest;  // column, and the row part j + Ly*k of the reference key (structs.jl:102)
    int j, k;
};
__host__ __device__ __forceinline__ unsigned pkey_ijk(const Grid &g, int i, int j, int k) {
    if (g.zrun) return (unsigned)i * (unsigned)g.rows + (unsigned)j * (unsigned)g.lim[2] + (unsigned)k;
    const unsigned rest = (unsigned)j + (unsigned)g.lim[1] * (unsigned)k;
    return ((((unsigned)(i >> g.cx_shift) * (unsigned)g.rows) + rest) << g.cx_shift) +
           ((unsigned)i & ((1u << g.cx_shift) - 1u));
}
__host__ __device__ __forceinline__ unsigned pkey_of(const Grid &g, int i, int rest) {
    const int ly = (int)g.lim[1];
    return pkey_ijk(g, i, rest % ly, rest / ly);
}
// column i is stored per particle (cellx), the row part follows from the physical key
__host__ __device__ __forceinline__ CellCoord cell_of(const Grid &g, unsigned pk, unsigned i) {
    CellCoord c;
    c.i = (int)i;
    if (g.zrun) {
        const unsigned pr = pk - i * (unsigned)g.rows;
        c.j = (int)(pr / (unsigned)g.lim[2]);
        c.k = (int)(pr - (unsigned)c.j * (unsigned)g.lim[2]);
        c.rest = c.j + (int)g.lim[1] * c.k;
    } else {
        c.rest = (int)((pk >> g.cx_shift) - (i >> g.cx_shift) * (unsigned)g.rows);
        c.k = c.rest / (int)g.lim[1];
        c.j = c.rest - c.k * (int)g.lim[1];
    }
    return c;
}
// neighbour cell number d of the reference's key_diff table (structs.jl:73-81).  The
// reference only checks 1 <= key + dkey <= key_max (core.jl:98), so a column overflow wraps
// into the adjacent row (and a row overflow into the adjacent plane) exactly as the linear key
// arithmetic does.
__device__ __forceinline__ bool neighbour_pkey(const Grid &g, const CellCoord &c, int d, unsigned &pk) {
    int i = c.i + g.nb_di[d], j = c.j + g.nb_dj[d], k = c.k + g.nb_dk[d];
    const int lx = (int)g.lim[0], ly = (int)g.lim[1];
    if (i < 0) {
        i += lx;
        j -= 1;
    } else if (i >= lx) {
        i -= lx;
        j += 1;
    }
    while (j < 0) {
        j += ly;
        k -= 1;
    }
    while (j >= ly) {
        j -= ly;
        k += 1;
    }
    if (k < 0 || k >= (int)g.lim[2]) return false;  // <=> key + dkey outside 1..key_max
    pk = pkey_ijk(g, i, j, k);
    return true;
}
// is_inside + find_key of a whole-domain context (geometry.jl:24-30, structs.jl:97-106): false outside the
// box (closed intervals; NaN fails every comparison), else the cell (i, j, k) of the position.  Particles
// (cell_key_whole) and sample points (point_sum.cuh) both call it, so a point and a particle at the same
// coordinates get the same home cell bit for bit.
template <int DIM>
__host__ __device__ __forceinline__ bool cell_ijk_whole(const Grid &g, double x, double y, double z, int &i, int &j,
                                                        int &k) {
    if (!(g.box[0] <= x && x <= g.box[3] && g.box[1] <= y && y <= g.box[4] && g.box[2] <= z && z <= g.box[5]))
        return false;
    // IEEE division, then floor (never a reciprocal multiply)
    i = (int)((long long)floor(x / g.h) - g.phase[0]);
    j = (int)((long long)floor(y / g.h) - g.phase[1]);
    k = DIM == 3 ? (int)((long long)floor(z / g.h) - g.phase[2]) : 0;
    return true;
}
// find_key + is_inside of one particle of a whole-domain context: the physical key and column of
// position pos, or — outside the box — the dead bucket, with its reference index appended to the removed
// list.  Shared by the cell-list build (k_keys) and the force pass's advance, so both compute the same bits.
template <int DIM>
__device__ __forceinline__ void cell_key_whole(const Grid &g, double x, double y, double z, int64_t pos,
                                               uint32_t *__restrict__ key, uint32_t *__restrict__ cellx,
                                               uint32_t *__restrict__ removed, uint32_t removed_cap,
                                               const uint32_t *__restrict__ idx) {
    int i, j, kk;
    uint32_t k, ci = 0;
    if (cell_ijk_whole<DIM>(g, x, y, z, i, j, kk)) {
        // structs.jl:102 gives the reference key i + Lx*(j + Ly*k); stored is its physical image
        k = pkey_ijk(g, i, j, kk);
        ci = (uint32_t)i;
    } else {
        k = (uint32_t)g.pkey_max;  // dead bucket: sorted behind every live cell
        const uint32_t slot = atomicAdd(&removed[0], 1u);
        if (slot < removed_cap) removed[1 + slot] = idx[pos];
    }
    key[pos] = k;
    cellx[pos] = ci;
}
#endif

// slab (multi-GPU) bookkeeping: local column c <-> global column slab_lo - GHOST_COLS + c
#define GHOST_COLS 2
#define TAG_OWNED 0u
#define TAG_GHOST 1u
#define TAG_DEAD 2u
#define HALO_RECORD 13  // the base record: x0 x1 x2 v0 v1 v2 m h rho rho_p type idx kind (halo_record.cuh)
#define HALO_KIND_MIGRANT 0.0
#define HALO_KIND_GHOST 1.0
#define SLAB_LOST_CAP 4096u  // particles one rank may lose to the global box in one step (open box, slab_comm.cu)

// which cell columns a pass evaluates (slab mode): [a0,a1] U [b0,b1]; `copy` = particles outside
// the set carry double-buffered outputs over (B_*::skip)
struct ColFilter {
    int on, a0, a1, b0, b1, copy;
    int sparse;  // the set is a small part of the grid: launch over the columns' particle ranges
};
__host__ __device__ __forceinline__ bool col_selected(const ColFilter &cf, int i) {
    return (i >= cf.a0 && i <= cf.a1) || (i >= cf.b0 && i <= cf.b1);
}

// ---------------------------------------------------------------------------
// Neighbour ("pair") list of one cell-list generation.  The first binary pass after a
// create_cell_list! walks the 9/27 neighbour cells once and records, per particle and in the
// reference's traversal order (core.jl:94-112), the ACCEPTED neighbours (r <= h, the particle itself
// left out: core.jl:105); every later pass on the same cell list (the force pass of verlet_step!,
// wcsph_perturbed_witch.jl:330) reads that list instead of walking ~157 candidates again.  Order and
// accepted set are unchanged, so every sum keeps its bits.
// Layout: entry k of particle p is list[((p >> 5) * stride + k) * 32 + (p & 31)] — the 32
// particles of a warp interleaved, so a warp reads/writes one 128-byte line per k.
// ---------------------------------------------------------------------------
#define NL_NONE 0xFFFFFFFFu  // cnt value: no list for this particle (walk the cells)
#define NL_BLOCK 128
#define NL_QUEUE_SLACK 4  // room in the recording pass's queue is checked once per four slots: the last four rows are slack
// ---- 10-bit mirror of the x-chunked cell order (shared-memory tile variant, pair_tile.cuh) ----------
// Pre-test of its recording pass on the quantised mirror.  A position is cell + (q + e)/1024 with
// e in [0,1) per axis, so for a pair with r <= h the integer differences d_a (in h/1024, cell
// offsets included) satisfy |d_a| < |t_a| + 1 with sum t_a^2 <= 1024^2, hence
// sum d_a^2 < (1024 + sqrt(3))^2.  1.74 > sqrt(3) leaves room for the rounding of x/h (1e-13).
#define NL_Q10_ONE 1024
#define NL_Q10_R2MAX 1052142  // floor((1024 + 1.74)^2)
#if defined(__CUDACC__) || defined(SPHMW_EMU)
#define NL_HD __host__ __device__ __forceinline__
#else
#define NL_HD static inline
#endif
// one axis: where x sits inside its cell floor(x / h) (structs.jl:99, k_keys), in h/1024
NL_HD uint32_t nl_q10_axis(double x, double h) {
    const double t = x / h;
    const double fr = t - floor(t);  // exact, in [0, 1)
    int q = (int)(fr * (double)NL_Q10_ONE);
    q = q < 0 ? 0 : (q > NL_Q10_ONE - 1 ? NL_Q10_ONE - 1 : q);
    return (uint32_t)q;
}
// the pre-test itself: own = mirror word of p, (di, dj, dk) = cell of q minus cell of p
NL_HD bool nl_q10_pass(uint32_t own, uint32_t other, int di, int dj, int dk, int dim) {
    const int dx = (int)(own & 1023u) - NL_Q10_ONE * di - (int)(other & 1023u);
    const int dy = (int)((own >> 10) & 1023u) - NL_Q10_ONE * dj - (int)((other >> 10) & 1023u);
    int s2 = dx * dx + dy * dy;
    if (dim == 3) {
        const int dz = (int)(own >> 20) - NL_Q10_ONE * dk - (int)(other >> 20);
        s2 += dz * dz;
    }
    return !(s2 > NL_Q10_R2MAX);
}
// ---- 6-bit mirror of the zrun cell order: one packed subtract and one DP4A per candidate --------
// Word of a particle: byte 0 = x inside its cell in h/64 (0..63), byte 1 = y likewise (3D only),
// byte 2 = 0, byte 3 = the run axis (z in 3D, y in 2D) ABSOLUTE modulo four cells:
// (cell & 3) << 6 | fraction.  For a candidate q in the run (di, dj, -1..1) of p's cell:
//     t = word(q) + K,   K = 0x80808080 + 64*di + (64*dj << 8) - word(p)      (one 32-bit add)
// has in bytes 0/1 the x/y difference in h/64 biased by 128 — never a carry: 0x80 + 64*d - p_b is in
// [1, 192] and q_b < 64 — in byte 2 the bias alone, and in byte 3 the run-axis difference modulo
// 256, exact as a signed byte because two cells are 128 units (carries out of byte 3 leave the
// word).  t ^ 0x80808080 turns the biased bytes into signed ones and DP4A of that word with itself
// is the squared distance in (h/64)^2.  Conservative for the same reason as above: positions are
// cell + (q + e)/64 with e in [0,1), so |d_a| < |t_a| + 1 and sum d_a^2 < (64 + sqrt(3))^2 whenever
// r <= h.  All |d_a| <= 127 fit a signed byte.
#define NL_Q6_ONE 64
#define NL_Q6_R2MAX 4321  // floor((64 + 1.74)^2)
#define NL_Q6_BIAS 0x80808080u
NL_HD uint32_t nl_q6_axis(double x, double h) {
    const double t = x / h;
    const double fr = t - floor(t);
    int q = (int)(fr * (double)NL_Q6_ONE);
    q = q < 0 ? 0 : (q > NL_Q6_ONE - 1 ? NL_Q6_ONE - 1 : q);
    return (uint32_t)q;
}
// run-axis byte: cell index (floor(x/h) - phase, as k_keys computes it) modulo 4, and the fraction
NL_HD uint32_t nl_q6_run_axis(double x, double h, long long phase) {
    const long long cell = (long long)floor(x / h) - phase;
    return ((uint32_t)(cell & 3) << 6) | nl_q6_axis(x, h);
}
NL_HD uint32_t nl_q6_word(double x, double y, double z, double h, long long run_phase, int dim) {
    if (dim == 3) return nl_q6_axis(x, h) | (nl_q6_axis(y, h) << 8) | (nl_q6_run_axis(z, h, run_phase) << 24);
    return nl_q6_axis(x, h) | (nl_q6_run_axis(y, h, run_phase) << 24);
}
// K of a run: (di, dj) = the run's cell column minus p's (dj = 0 in 2D, where y is the run axis)
NL_HD uint32_t nl_q6_run_const(uint32_t own, int di, int dj) {
    return NL_Q6_BIAS + (uint32_t)(NL_Q6_ONE * di) + (uint32_t)(NL_Q6_ONE * dj * 256) - own;
}
NL_HD int nl_q6_dist2(uint32_t K, uint32_t other) {
    const uint32_t s = (other + K) ^ NL_Q6_BIAS;
#if defined(__CUDA_ARCH__)
    return __dp4a((int)s, (int)s, 0);
#else
    int acc = 0;
    for (int b = 0; b < 4; ++b) {
        const int v = (int)(int8_t)(s >> (8 * b));
        acc += v * v;
    }
    return acc;
#endif
}
// Packed neighbour records (SPHMW_FLAG_PACKED_RECORDS): what a replayed list entry needs from its
// neighbour, as three 32-byte records read with one 256-bit load each instead of eleven 8-byte
// gathers (profiles/microbench/gather_width.cu: 1.31x on the replay's access pattern).
//   A {x, y, z, m}          written by the cell-list gather
//   B {vx, vy, vz, h}       written by the density pass (h after update_smoothing!)
//   C {P'/rho^2, rho^, c}   written by the density pass (rho^ = max(rho, rho_floor))
// They are bit copies of the SoA fields, so results do not change.
struct __align__(32) NbRec {
    double a, b, c, d;
};
#if defined(SPHMW_EMU)  // host build of the device headers for the CPU tests (tests/emu/)
inline NbRec nb_load(const NbRec *p) { return *p; }
inline void nb_store(NbRec *p, double a, double b, double c, double d) { *p = NbRec{a, b, c, d}; }
#elif defined(__CUDACC__)
__device__ __forceinline__ NbRec nb_load(const NbRec *p) {
    NbRec r;
    asm("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.a), "=d"(r.b), "=d"(r.c), "=d"(r.d) : "l"(p));
    return r;
}
__device__ __forceinline__ void nb_store(NbRec *p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
#endif

struct PairList {
    uint32_t *list;
    uint32_t *list16;  // tiled kernels (pair_tile.cuh): 16-bit tile slots, two per word
    uint32_t *cnt;
    NbRec *recA, *recB, *recC;  // null unless SPHMW_FLAG_PACKED_RECORDS
    // quantised mirror of the positions, rebuilt by every cell-list build (cell_gather.cuh): the 6-bit
    // word of the zrun cell order (nl_q6_word above), or — x-chunked order, tile variant — 10 bits per
    // axis inside the particle's own cell, x | y<<10 | z<<20
    const uint32_t *xq;
    int stride;
    int qrows;  // rows of the recording pass's shared-memory queue (survivors of the pre-test + NL_QUEUE_SLACK)
    unsigned long long *overflow;  // counter: particles whose candidates did not fit `stride`
};

struct TimingEntry {
    int name_id;
    cudaEvent_t a, b;
};

struct sphmw_ctx {
    int device = 0;
    int flags = 0;
    int sm_count = 148;
    Grid grid{};
    Params prm{};
    int64_t n = 0;       // particles resident (incl. ghosts in slab mode)
    int64_t cap = 0;
    int64_t slab_lo = -1, slab_hi = -1;
    int64_t global_cols = 0;  // cell columns of the whole domain (slab contexts)
    // overlapped slab step (pair_ops.cu step_wcsph_overlap_*, halo.cu): 0 idle, 1 edge columns
    // advanced into the alt buffers, 2 their records packed, 3 interior advanced and buffers swapped
    int overlap_stage = 0;
    cudaEvent_t pack_event = nullptr;

    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;

    Fields cur{};  // physical (cell-sorted) order
    Fields alt{};  // reorder target / double buffer
    bool allocated[NSLOT] = {};
    bool stale[NSLOT] = {};  // contents not up to date: skip in reorder, rebuild on demand
    bool dv_zero = true;     // Dv is known to be all-zero (never written since accelerate!)
    // the keys, columns and removed list of the current positions were written by the force pass's
    // advance (whole-domain multi-step call): the next cell-list build skips k_keys.  Consumed by that
    // build; cleared by everything else that changes x
    bool keys_from_advance = false;

    uint32_t *idx = nullptr, *idx_alt = nullptr;  // reference particle index of each position
    uint32_t *pos_of_idx = nullptr;               // inverse map (whole-domain contexts only), valid iff pos_valid
    bool pos_valid = false;
    uint32_t *tag = nullptr, *tag_alt = nullptr;  // TAG_OWNED / TAG_GHOST / TAG_DEAD per position
    int64_t n_owned = 0;                          // slab mode: resident particles this rank owns
    // dead particles the next cell-list build will meet (halo.cu: ghosts and migrants of the last
    // exchange + particles dropped by the pack): with it the build needs no host round trip
    int64_t slab_dead_expected = 0;
    bool slab_dead_known = false;
    uint32_t *h_slab_check = nullptr;             // pinned ring: what the device counted, verified one build later
    cudaEvent_t slab_check_event[4] = {nullptr, nullptr, nullptr, nullptr};
    int64_t slab_check_want[4][2] = {};           // the host's figures for the same builds
    uint64_t slab_checks = 0;
    struct SlabComm *comm = nullptr;              // NCCL halo transport (slab_comm.cu)
    int halo_kind = -1;                           // halo record kind (halo_record.cuh), fixed at first use; -1: not yet
    uint32_t *lost_list = nullptr;                // open box: [0] count, [1..] global indices the last pack dropped
    struct FrameAsync *frame_async = nullptr;     // asynchronous frame output / upload prefetch (frame_async.cu)
    uint32_t *halo_counters = nullptr;            // device: [0] left records [1] right records
                                                  // [2] left migrants [3] right migrants [4] lost
    uint32_t *h_halo_counters = nullptr;          // pinned mirror
    uint32_t *key = nullptr;         // physical cell key per position (pkey_max = dead bucket)
    uint32_t *cellx = nullptr, *cellx_alt = nullptr;  // cell column i of each position
    uint32_t *rank = nullptr;        // arrival rank inside the cell
    uint32_t *src = nullptr;         // new position -> old position
    uint32_t *cell_start = nullptr;  // cells_cap + 2 entries
    int64_t cells_cap = 0;           // pkey_max of the larger of the two physical cell orders
    uint32_t *scan_tmp = nullptr;
    int64_t scan_tmp_len = 0;
    uint32_t *removed = nullptr;     // [0] = count, [1..] = removed reference indices
    int64_t removed_cap = 0;
    uint32_t *h_removed = nullptr;   // pinned mirror
    uint32_t *mv_old = nullptr, *mv_new = nullptr;
    int64_t mv_cap = 0;
    unsigned long long *d_counters = nullptr;  // [0] pair counter, [1] scratch
    unsigned long long *h_counters = nullptr;  // pinned

    // pair list (pair_list.cuh)
    PairList pl{};
    uint32_t *xq = nullptr;        // cap (+4) entries, rebuilt by every cell-list build
    NbRec *rec[3] = {nullptr, nullptr, nullptr};  // packed neighbour records A, B, C (cap entries each)
    uint64_t rec_gen = ~0ull;      // cell-list generation record A was written for
    uint64_t rec_bc_gen = ~0ull;   // ... and records B, C (by the fused density pass)
    uint64_t cell_gen = 0;         // generation of the cell list
    uint64_t pl_gen = ~0ull;       // generation the pair list was built for
    bool want_list = false;        // build the list in the next binary pass
    int passes_this_gen = 0;       // binary passes since the last cell-list build
    int64_t pl_builds = 0;
    unsigned long long pl_overflow_seen = 0;  // overflow counter at the last look (queue rows adapt, cell_list.cu)
    int pl_format = 0;             // what the valid list holds: 0 global positions, 1 tile slots
    // fluid work list of one cell-list generation (cell_list.cu, pair_list.cuh k_binary_list_fluid):
    // the positions with type == fluid ascending, then the others ascending.  Built by every cell-list
    // build once a fused WCSPH step has asked for it
    bool want_fluid_list = false;
    uint8_t *fluid_flag = nullptr;    // cap (+8): written by the gather
    uint32_t *fluid_work = nullptr;   // cap
    uint32_t *fluid_tiles = nullptr;  // fluid count per tile -> exclusive scan; fluid_tiles[tiles] = all
    int64_t fluid_tiles_cap = 0;
    const uint32_t *fluid_count = nullptr;  // device: the number of fluid positions
    uint64_t fluid_gen = ~0ull;       // cell-list generation the list was built for
    double fluid_value = 0.0;         // ... and the type value (Params::fluid) it was built with
    // neighbourhood tiles (tile_map.cuh): one record per block of TM_BLOCK particles
    uint32_t *tile_tab = nullptr;
    uint64_t tile_gen = ~0ull;     // cell-list generation the records were built for

    double *staging = nullptr;  // 3*cap doubles
    double *reduce_tmp = nullptr;
    // point sums (point_sum.cu): grow-only scratch for host points and outputs, keys and order
    double *pt_pts = nullptr, *pt_out = nullptr;
    uint32_t *pt_key = nullptr, *pt_order = nullptr;  // 2 x pt_cap each: as computed, sorted
    void *pt_sort_tmp = nullptr;
    int64_t pt_cap = 0, pt_out_cap = 0;
    size_t pt_sort_tmp_bytes = 0;

    bool cell_list_valid = false;
    bool count_pairs = false;

    // pvd output (IO.jl:9-13)
    std::string pvd_dir;
    int64_t pvd_frame = 0;
    std::vector<std::string> pvd_entries;
    bool pvd_open = false;

    // timing
    bool timing = false;
    std::string timing_prefix;  // time only kernels with this name prefix (empty: all)
    std::vector<std::string> timing_names;
    std::vector<double> timing_ms;
    std::vector<int64_t> timing_calls;
    std::vector<TimingEntry> timing_pending;
    std::vector<cudaEvent_t> event_pool;
    int64_t launches = 0;
};

// The fused pair passes read packed neighbour records unless told otherwise (sphmw.h).  Default in 3D
// only: in 2D a neighbour needs 9 fields, the records still move 96 bytes, and the SoA gathers are 6 %
// faster (4.1 M particles: 1.19 vs 1.26 ms per step, profiles/r02_pair_kernels.md); PACKED_RECORDS forces them.
static inline bool sphmw_use_records(const sphmw_ctx *c) {
    if (c->flags & (SPHMW_FLAG_NO_PACKED_RECORDS | SPHMW_FLAG_NO_PAIR_LIST | SPHMW_FLAG_CELL_PAIRS | SPHMW_FLAG_TILES |
                    SPHMW_FLAG_NO_PRETEST))
        return false;
    return c->grid.dim == 3 || (c->flags & SPHMW_FLAG_PACKED_RECORDS);
}

// which physical cell order a set of flags runs on (Grid::zrun): the shared-memory variants stage
// x-rows of cells and keep the x-chunked order; SPHMW_CELL_ORDER=xchunk forces it (A/B runs)
static inline bool sphmw_want_zrun(int flags) {
    if (flags & (SPHMW_FLAG_CELL_PAIRS | SPHMW_FLAG_TILES)) return false;
    const char *e = getenv("SPHMW_CELL_ORDER");
    return !(e && !strcmp(e, "xchunk"));
}

// error plumbing -----------------------------------------------------------
void sphmw_set_error(const char *fmt, ...);
#define CUDA_TRY(expr)                                                              \
    do {                                                                            \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess) {                                                    \
            sphmw_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                            __FILE__, __LINE__);                                    \
            return SPHMW_E_CUDA;                                                    \
        }                                                                           \
    } while (0)
#define TRY(expr)            \
    do {                     \
        int _r = (expr);     \
        if (_r != 0) return _r; \
    } while (0)

struct FieldDesc {
    const char *name;
    int slot;
    int ncomp;
};
const FieldDesc *sphmw_find_field(const char *name);

// implemented in grid_setup.cpp (host only, no CUDA calls)
void sphmw_derive_params(Params &p);
int sphmw_grid_setup(Grid &g, const double box_min[3], const double box_max[3], double h, int64_t slab_lo,
                     int64_t slab_hi, int64_t *global_cols, int ghost = GHOST_COLS);
void sphmw_grid_set_order(Grid &g, bool zrun);  // physical cell order (Grid::zrun)
// core.jl:72-81 on index space: the (old index -> new index) moves of the survivors when the
// particles `removed` (any order) leave an array of N (cell_list.cu)
void sphmw_replay_swap_removal(int64_t N, std::vector<uint32_t> &removed, std::vector<uint32_t> &mv_old,
                               std::vector<uint32_t> &mv_new);
// implemented in cell_list.cu
int sphmw_build_cell_list(sphmw_ctx *c, int64_t *n_alive);
int sphmw_ensure_slot(sphmw_ctx *c, int slot);
int sphmw_ensure_pos_of_idx(sphmw_ctx *c);  // rebuild the inverse index map if a cell-list build voided it
// implemented in pair_ops.cu
int sphmw_apply_named(sphmw_ctx *c, const char *op, int self);
int sphmw_step_scheme(sphmw_ctx *c, const char *scheme, int nsteps);
int sphmw_step_scheme_phase(sphmw_ctx *c, const char *scheme, int phase);
int sphmw_materialize(sphmw_ctx *c, int slot);
int64_t sphmw_list_ops(char *buf, int64_t cap);
int sphmw_dump_pairs(sphmw_ctx *c, int64_t *pi, int64_t *pj, int64_t cap, int64_t *n);
int sphmw_flow_add_particles(sphmw_ctx *c, int64_t *n_added, bool adiabatic);
int sphmw_flow_collect_slab(sphmw_ctx *c, uint32_t *list, uint32_t *pos, uint32_t cap, bool adiabatic);  // slab contexts (slab_comm.cu)
int sphmw_flow_spawn_slab(sphmw_ctx *c, const uint32_t *pos, const uint32_t *new_idx, int m, bool adiabatic);
int sphmw_pair_list_stats(sphmw_ctx *c, int64_t out[4]);
int sphmw_tile_stats(sphmw_ctx *c, int64_t out[6]);
int sphmw_ensure_records(sphmw_ctx *c);  // api.cu: allocate the packed neighbour records
// column sets of the overlapped slab step (local column indices)
struct SlabCols {
    ColFilter edge;      // advanced and packed first: ghost columns + the three outermost owned ones
    ColFilter interior;  // the rest
    ColFilter force_edge, force_interior;  // their owned parts (the force pass covers owned columns only)
};
SlabCols sphmw_slab_cols(const sphmw_ctx *c);
SlabCols sphmw_slab_cols_of(int W, bool has_left, bool has_right);
// implemented in cell_list.cu
int sphmw_exclusive_scan_u32(sphmw_ctx *c, uint32_t *data, int64_t n);
// implemented in halo.cu / slab_comm.cu
int sphmw_halo_pack_enqueue(sphmw_ctx *c, double *msg_left, double *msg_right, int64_t cap_records, bool edge_only);
int sphmw_halo_pack_collect_nowait(sphmw_ctx *c, int64_t cap_records, int64_t counts[5]);
int sphmw_halo_kind(sphmw_ctx *c, int *kind);  // HALO_REC_BASE / HALO_REC_ADIABATIC (halo_record.cuh)
int sphmw_comm_add_new_particles(sphmw_ctx *c, int64_t *n_added, bool adiabatic);
int sphmw_comm_step(sphmw_ctx *c, const char *scheme, int nsteps);
int sphmw_comm_create_cell_list(sphmw_ctx *c, int64_t *n_alive);
void sphmw_comm_free(sphmw_ctx *c);
int sphmw_step_wcsph_phase(sphmw_ctx *c, int phase);  // pair_ops.cu
// implemented in frame_async.cu
int sphmw_pvd_save_frame_async(sphmw_ctx *c, const char *const *fields, int nfields, const std::string &path);
int sphmw_frame_async_drain(sphmw_ctx *c);
void sphmw_frame_async_free(sphmw_ctx *c);
// implemented in frame_io.cpp
int sphmw_write_vtp(const char *path, int64_t n, const double *points3n, int nfields,
                    const char *const *names, const int *ncomps, const double *const *data);
int sphmw_write_pvd(const char *path, const std::vector<std::string> &files);

// A few words from device memory to PINNED host memory, written by a one-thread kernel through the
// unified address space instead of a cudaMemcpyAsync: the step's counters (removed particles, halo
// record counts) must not queue on the device-to-host copy engine behind a multi-gigabyte frame copy
// of another stream (measured: every step of a frame interval waited 15 ms for it; api.cu)
int sphmw_publish_words(sphmw_ctx *c, const uint32_t *dev_src, uint32_t *pinned_dst, int nwords, cudaStream_t stream);

// timing helpers (api.cu)
struct KernelTimer {
    sphmw_ctx *c;
    int pending_index;
    KernelTimer(sphmw_ctx *ctx, const char *name);
    ~KernelTimer();
};
#define TIMED(ctx, name) KernelTimer _kt_##__LINE__(ctx, name)

static inline unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }
