// Pair-list kernels: _apply_binary! (src/core.jl:94-112) split into a recording pass and
// replaying passes.  See PairList in sphmw_internal.h for the layout and the invariants.
//
//   k_binary_build  walks the 9/27 neighbour cells in key_diff order (structs.jl:73-81) — as 3/9
//                   contiguous runs of three cells in the zrun cell order — with a cheap cut-off
//                   test (one packed add + DP4A on the 6-bit mirror, or the exact FP64 one), queues
//                   the survivors per thread in shared memory, then — with the lanes of a warp
//                   compacted onto ~28 survivors instead of ~157 candidates — runs the exact test
//                   `r > sys.h` (core.jl:104-105) and the closure body, and writes the ACCEPTED
//                   neighbours (the particle itself left out, core.jl:105 `p == q`) to the list.
//   k_binary_list   replays a recorded list: exact test + closure body per entry.
//
// Both visit accepted neighbours in exactly the order of k_binary (pair_ops.cu), so every FP64
// sum is bit-identical to the cell walk.  A particle whose survivors do not fit the list
// stride, or that was outside the recording pass's column filter, has cnt == NL_NONE and
// walks the cells with the original loop.
#pragma once
#include "q_access.cuh"
#include "sphmw_internal.h"

// the loop of k_binary, for particles without a list
template <int DIM, class Op>
__device__ __forceinline__ void nl_walk(Op &op, const Fields &f, const Params &prm, const Grid &g,
                                        const CellCoord &home, int64_t p, double px, double py,
                                        double pz, const uint32_t *__restrict__ cell_start,
                                        unsigned &accepted) {
    for (int d = 0; d < g.ndiff; ++d) {
        unsigned nk;
        if (!neighbour_pkey(g, home, d, nk)) continue;  // core.jl:98
        uint32_t b = cell_start[nk], e = cell_start[nk + 1];
        for (uint32_t q = b; q < e; ++q) {
            double dx = px - f.s[S_X0][q];
            double dy = py - f.s[S_X1][q];
            double dz = 0.0;
            double r2 = dx * dx + dy * dy;
            if (DIM == 3) {
                dz = pz - f.s[S_X2][q];
                r2 = r2 + dz * dz;
            }
            if ((r2 > g.r2_max) || (q == p)) continue;
            double r = sqrt(r2);
            op.template pair<DIM>(f, prm, p, q, dx, dy, dz, r);
            ++accepted;
        }
    }
}

// what the recording pass does with an accepted neighbour before the closure body runs: append it
// to the particle's list column (entries beyond the stride are dropped; the caller then marks the
// particle NL_NONE).  The replaying pass records nothing.
struct NlNoSink {
    __device__ __forceinline__ void operator()(uint32_t) const {}
};
struct NlListSink {
    uint32_t *row;
    uint32_t left;
    __device__ __forceinline__ void operator()(uint32_t q) {
        if (left) {
            __stcs(row, q);
            row += 32;
            --left;
        }
    }
};

// exact test + closure body for one recorded candidate
template <int DIM, class Op, class Sink = NlNoSink>
__device__ __forceinline__ void nl_entry(Op &op, const Fields &f, const Params &prm, const Grid &g,
                                         int64_t p, uint32_t q, double px, double py, double pz,
                                         unsigned &accepted, Sink &&sink = Sink()) {
    // dist(p,q) — core.jl:8-10, algebra.jl:49-60: left-to-right, no FMA
    double dx = px - f.s[S_X0][q];
    double dy = py - f.s[S_X1][q];
    double dz = 0.0;
    double r2 = dx * dx + dy * dy;
    if (DIM == 3) {
        dz = pz - f.s[S_X2][q];
        r2 = r2 + dz * dz;
    }
    if ((r2 > g.r2_max) || (q == (uint32_t)p)) return;  // core.jl:105, decided on r2 (Grid::r2_max)
    sink(q);
    double r = sqrt(r2);
    op.template pair<DIM>(f, prm, p, q, dx, dy, dz, r);
    ++accepted;
}

// ---- packed-record variants (SPHMW_FLAG_PACKED_RECORDS; NbRec in sphmw_internal.h) ----------
// density closure: position and mass of q from record A
template <int DIM, class Op, class Sink = NlNoSink>
__device__ __forceinline__ void nl_entry_rec_density(Op &op, const Params &prm, const Grid &g, int64_t p,
                                                     uint32_t q, double px, double py, double pz,
                                                     const NbRec *__restrict__ recA, unsigned &accepted,
                                                     Sink &&sink = Sink()) {
    const NbRec A = nb_load(recA + q);
    double dx = px - A.a;
    double dy = py - A.b;
    double dz = 0.0;
    double r2 = dx * dx + dy * dy;
    if (DIM == 3) {
        dz = pz - A.c;
        r2 = r2 + dz * dz;
    }
    if ((r2 > g.r2_max) || (q == (uint32_t)p)) return;
    sink(q);
    double r = sqrt(r2);
    op.template pair_q<DIM>(prm, RecAQ{A.d}, dx, dy, dz, r);
    ++accepted;
}
// force closure: all three records are requested up front (the exact test rejects few entries)
template <int DIM, class Op>
__device__ __forceinline__ void nl_entry_rec_force(Op &op, const Params &prm, const Grid &g, int64_t p,
                                                   uint32_t q, double px, double py, double pz,
                                                   const PairList &pl, unsigned &accepted) {
    const NbRec A = nb_load(pl.recA + q);
    const NbRec B = nb_load(pl.recB + q);
    const NbRec C = nb_load(pl.recC + q);
    double dx = px - A.a;
    double dy = py - A.b;
    double dz = 0.0;
    double r2 = dx * dx + dy * dy;
    if (DIM == 3) {
        dz = pz - A.c;
        r2 = r2 + dz * dz;
    }
    if ((r2 > g.r2_max) || (q == (uint32_t)p)) return;
    double r = sqrt(r2);
    op.template pair_q<DIM>(prm, RecQ{A.d, B, C}, dx, dy, dz, r);
    ++accepted;
}

// per-thread queue column in shared memory, addressed with 32-bit shared-window addresses so
// that a push is one predicated st.shared and one predicated add (the queue is touched only
// through these volatile statements, which keep their order).  Room for a whole cell run is
// checked before the run starts (nl_room), not per candidate.
__device__ __forceinline__ bool nl_room(unsigned top, unsigned end, uint32_t run) {
    // run < 2^20 keeps the product inside 32 bits; longer runs never fit a stride <= 96 anyway
    return run < (1u << 20) && top + run * (NL_BLOCK * 4u) <= end;
}
#ifdef SPHMW_EMU  // host build for the CPU tests: the "shared window" is the array itself
inline void nl_push(unsigned &top, uint32_t q, bool pass) {
    if (pass) {
        *(uint32_t *)((char *)nl_queue_emu() + top) = q;
        top += NL_BLOCK * 4u;
    }
}
inline uint32_t nl_peek(unsigned addr) { return *(const uint32_t *)((const char *)nl_queue_emu() + addr); }
#else
__device__ __forceinline__ void nl_push(unsigned &top, uint32_t q, bool pass) {
    asm volatile(
        "{\n\t"
        ".reg .pred ps;\n\t"
        "setp.ne.u32 ps, %2, 0;\n\t"
        "@ps st.shared.u32 [%0], %1;\n\t"
        "@ps add.u32 %0, %0, %3;\n\t"
        "}"
        : "+r"(top)
        : "r"(q), "r"((unsigned)pass), "n"(NL_BLOCK * 4));
}
__device__ __forceinline__ uint32_t nl_peek(unsigned addr) {
    uint32_t q;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(q) : "r"(addr));
    return q;
}
#endif

__device__ __forceinline__ void nl_count_pairs(unsigned long long *pair_counter, unsigned accepted) {
    if (pair_counter) {
        unsigned m = __activemask();
        unsigned tot = __reduce_add_sync(m, accepted);
        if ((int)(threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(pair_counter, (unsigned long long)tot);
    }
}

// FILTER: how phase 1 tests a candidate — the exact FP64 test (three 8-byte loads), or integers
// on the 6-bit mirror of the zrun cell order (one 4-byte load, one add, one xor, one DP4A;
// survivors get the exact test in phase 2).  Measured alternatives: a 10-bit-per-axis mirror tested
// cell by cell (19.5 SASS instructions per candidate slot, 216 slots per particle: round 2 until the
// zrun order) and an FP32 mirror of the absolute positions (slower still, profiles/r01b_pair_list.md).
#define NL_FILTER_F64 0
#define NL_FILTER_Q6 3
// one candidate run [b, e) of the 6-bit pre-test; false: the queue is full.  Measured and set aside
// (profiles/r02b_zrun.md): requesting the next four words ahead, aligned 16-byte loads of four
// words, and two queue entries per iteration in phase 2 — the plain loop with the fewest registers
// (56: nine resident blocks) was the fastest of all.
__device__ __forceinline__ bool nl_q6_run(const uint32_t *__restrict__ xq, uint32_t b, uint32_t e, uint32_t K,
                                          unsigned &qtop, unsigned qlimit) {
    if (b >= e) return true;
    const uint32_t last = e - 1;
    for (uint32_t q = b; q < e; q += 4) {
        if (qtop > qlimit) return false;
        const uint32_t *__restrict__ cp = xq + q;  // padded: slots past the run are masked
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = cp[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int s2 = nl_q6_dist2(K, w[i]);
            const uint32_t qi = q + i;
            nl_push(qtop, qi, !((s2 > NL_Q6_R2MAX) || (i > 0 && qi > last)));
        }
    }
    return true;
}
// REC (fused density pass only): phase 2 reads q from record A, and the particle's own records B
// and C are written once its density, smoothing length and pressure are final
#ifdef NL_BUILD_MIN_BLOCKS  // A/B builds (scripts/build_variant.sh)
#define NL_BUILD_BOUNDS __launch_bounds__(NL_BLOCK, NL_BUILD_MIN_BLOCKS)
#else
#define NL_BUILD_BOUNDS __launch_bounds__(NL_BLOCK)
#endif
template <int DIM, class Op, int FILTER, bool REC = false>
__global__ void NL_BUILD_BOUNDS
k_binary_build(Fields f, Fields out, Params prm, Grid g, const uint32_t *__restrict__ key,
               const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, int64_t n,
               int self, unsigned long long *pair_counter, ColFilter cf, PairList pl) {
    // [pl.qrows][NL_BLOCK]: a private column per thread.  The queue is what limits the L1 cache the nine
    // resident blocks leave: 44 -> 36 rows took the 64 M density pass from 15.6 to 14.4 ms (16-bit
    // entries, which halve it again, lost that to their decoding: profiles/r02b_zrun.md), so the rows are
    // sized for the survivors a particle really has, independently of the list stride
    extern __shared__ uint32_t nl_queue[];
    const int64_t p = blockIdx.x * (int64_t)NL_BLOCK + threadIdx.x;
    if (p >= n) return;
    const CellCoord home = cell_of(g, key[p], cellx[p]);
    if (cf.on && !col_selected(cf, home.i)) {
        if (cf.copy) Op::template skip<DIM>(f, out, p);
        pl.cnt[p] = NL_NONE;
        return;
    }
    const uint32_t stride = (uint32_t)pl.stride;
    const unsigned qbase = (unsigned)__cvta_generic_to_shared(nl_queue + threadIdx.x);
    const unsigned qend = qbase + (unsigned)pl.qrows * (NL_BLOCK * 4u);
    unsigned qtop = qbase;
    const double px = f.s[S_X0][p], py = f.s[S_X1][p], pz = DIM == 3 ? f.s[S_X2][p] : 0.0;
    bool fits = true;
    // ---- phase 1: candidates -> queue -------------------------------------------------
    // A home cell that touches no face of the grid reaches its 9/27 neighbour cells without any
    // wrap of the linear key arithmetic (core.jl:98 has no per-axis check), and in the zrun order
    // the cells (di, dj, -1..1) are one contiguous run visited in exactly the reference's order:
    // 3/9 runs, one constant per run.  Cells on a face (and FILTER_F64) go cell by cell with the
    // exact FP64 test.
    bool by_runs = false;
    if (FILTER == NL_FILTER_Q6) {
        const int lx = (int)g.lim[0], ly = (int)g.lim[1], lz = (int)g.lim[2];
        by_runs = home.i >= 1 && home.i <= lx - 2 && home.j >= 1 && home.j <= ly - 2 &&
                  (DIM == 2 || (home.k >= 1 && home.k <= lz - 2));
    }
    if (by_runs) {
        const uint32_t ow = pl.xq[p];
        const unsigned rows = (unsigned)g.rows, lz = (unsigned)g.lim[2];
        const unsigned qlimit = qend - 4u * (NL_BLOCK * 4u);
        // first cell of the run (-1, -1): one step back along the run axis (z in 3D, y in 2D)
        const unsigned pk0 = pkey_ijk(g, home.i - 1, home.j - 1, DIM == 3 ? home.k - 1 : 0);
        for (int di = -1; di <= 1 && fits; ++di) {
            if (DIM == 3) {
                // the bounds of the plane's three runs in one go (six independent loads)
                const unsigned rk = pk0 + (unsigned)(di + 1) * rows;
                uint32_t rb[3], re[3];
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    rb[t] = cell_start[rk + (unsigned)t * lz];
                    re[t] = cell_start[rk + (unsigned)t * lz + 3];
                }
#pragma unroll
                for (int t = 0; t < 3; ++t)
                    if (fits && !nl_q6_run(pl.xq, rb[t], re[t], nl_q6_run_const(ow, di, t - 1), qtop, qlimit)) fits = false;
            } else {
                const unsigned rk = pk0 + (unsigned)(di + 1) * rows;
                if (!nl_q6_run(pl.xq, cell_start[rk], cell_start[rk + 3], nl_q6_run_const(ow, di, 0), qtop, qlimit))
                    fits = false;
            }
        }
    } else {
        for (int d = 0; d < g.ndiff; ++d) {
            unsigned nk;
            if (!neighbour_pkey(g, home, d, nk)) continue;
            const uint32_t b = cell_start[nk], e = cell_start[nk + 1];
            if (!nl_room(qtop, qend, e - b)) {
                fits = false;
                break;
            }
            for (uint32_t q = b; q < e; ++q) {
                double dx = px - f.s[S_X0][q];
                double dy = py - f.s[S_X1][q];
                double r2 = dx * dx + dy * dy;
                if (DIM == 3) {
                    double dz = pz - f.s[S_X2][q];
                    r2 = r2 + dz * dz;
                }
                nl_push(qtop, q, !(r2 > g.r2_max));
            }
        }
    }
    // ---- phase 2: exact test + closure over the queue; accepted neighbours -> list -------
    Op op;
    op.template init<DIM>(f, prm, p);
    unsigned accepted = 0;
    if (fits) {
        NlListSink sink{pl.list + ((size_t)(p >> 5) * stride) * 32 + (size_t)(p & 31), stride};
        for (unsigned a = qbase; a < qtop; a += NL_BLOCK * 4u) {
            const uint32_t q = nl_peek(a);
            if constexpr (REC && Op::REC_KIND == 1)
                nl_entry_rec_density<DIM>(op, prm, g, p, q, px, py, pz, pl.recA, accepted, sink);
            else nl_entry<DIM>(op, f, prm, g, p, q, px, py, pz, accepted, sink);
        }
        // more accepted neighbours than the list holds: this pass is complete (the closure saw
        // them all), later passes walk the cells for this particle
        if (accepted > stride) atomicAdd(pl.overflow, 1ull);
        pl.cnt[p] = accepted > stride ? NL_NONE : accepted;
    } else {
        pl.cnt[p] = NL_NONE;
        atomicAdd(pl.overflow, 1ull);
        nl_walk<DIM>(op, f, prm, g, home, p, px, py, pz, cell_start, accepted);
    }
    if (self) op.template pair<DIM>(f, prm, p, p, 0.0, 0.0, 0.0, 0.0);  // core.jl:155-157
    op.template finish<DIM>(f, out, prm, p);
    op.template after<DIM>(g, out, prm, p);
    if constexpr (REC && Op::REC_KIND == 1) {
        // what finish() just stored for p (same thread: reads see its own writes), as records
        nb_store(pl.recB + p, f.s[S_V0][p], f.s[S_V1][p], DIM == 3 ? f.s[S_V2][p] : 0.0, f.s[S_H][p]);
        const double rho = f.s[S_RHO][p];
        const double rfl = (rho != rho) ? rho : (rho < prm.rho_floor ? prm.rho_floor : rho);  // jl_max
        nb_store(pl.recC + p, f.s[S_PR2][p], rfl, f.s[S_CS][p], 0.0);
    }
    nl_count_pairs(pair_counter, accepted);
}

// REC (fused force pass only): entries are evaluated from the packed records.
// pairs == false (a non-fluid particle of an Op with PAIRS_FOR_FLUID_ONLY): the recorded entries are
// not evaluated — finish() would discard their sums — but still counted, so the pair counter keeps the
// reference's figure; a particle without a list (NL_NONE) walks the cells as always.
template <int DIM, class Op, bool REC>
__device__ __forceinline__ void nl_list_particle(int64_t p, const Fields &f, const Fields &out, const Params &prm,
                                                 const Grid &g, const uint32_t *__restrict__ key,
                                                 const uint32_t *__restrict__ cellx,
                                                 const uint32_t *__restrict__ cell_start, int self,
                                                 unsigned long long *pair_counter, const ColFilter &cf,
                                                 const PairList &pl, bool pairs = true) {
    const CellCoord home = cell_of(g, key[p], cellx[p]);
    if (cf.on && !col_selected(cf, home.i)) {
        if (cf.copy) Op::template skip<DIM>(f, out, p);
        return;
    }
    const uint32_t cnt = pl.cnt[p];
    const double px = f.s[S_X0][p], py = f.s[S_X1][p], pz = DIM == 3 ? f.s[S_X2][p] : 0.0;
    Op op;
    op.template init<DIM>(f, prm, p);
    unsigned accepted = 0;
    if (cnt != NL_NONE && !pairs) {
        accepted = cnt;  // the recording pass accepted exactly these entries (same positions)
    } else if (cnt != NL_NONE) {
        const uint32_t *row = pl.list + ((size_t)(p >> 5) * (uint32_t)pl.stride) * 32 + (size_t)(p & 31);
        // (loading the next entry's position one iteration ahead as well was measured slower:
        // profiles/r01b_pair_list.md)
        uint32_t qn = cnt ? __ldcs(row) : 0u;
        for (uint32_t k = 0; k < cnt; ++k) {
            const uint32_t q = qn;
            if (k + 1 < cnt) qn = __ldcs(row + (size_t)(k + 1) * 32);  // one entry ahead
            if constexpr (REC && Op::REC_KIND == 2)
                nl_entry_rec_force<DIM>(op, prm, g, p, q, px, py, pz, pl, accepted);
            else nl_entry<DIM>(op, f, prm, g, p, q, px, py, pz, accepted);
        }
    } else {
        nl_walk<DIM>(op, f, prm, g, home, p, px, py, pz, cell_start, accepted);
    }
    if (self) op.template pair<DIM>(f, prm, p, p, 0.0, 0.0, 0.0, 0.0);
    op.template finish<DIM>(f, out, prm, p);
    op.template after<DIM>(g, out, prm, p);
    nl_count_pairs(pair_counter, accepted);
}

#ifdef NL_LIST_MIN_BLOCKS  // A/B builds (scripts/build_variant.sh)
#define NL_LIST_BOUNDS __launch_bounds__(NL_BLOCK, NL_LIST_MIN_BLOCKS)
#else
#define NL_LIST_BOUNDS __launch_bounds__(NL_BLOCK)
#endif
template <int DIM, class Op, bool REC = false>
__global__ void NL_LIST_BOUNDS
k_binary_list(Fields f, Fields out, Params prm, Grid g, const uint32_t *__restrict__ key,
              const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, int64_t n,
              int self, unsigned long long *pair_counter, ColFilter cf, PairList pl) {
    const int64_t p = blockIdx.x * (int64_t)NL_BLOCK + threadIdx.x;
    if (p >= n) return;
    nl_list_particle<DIM, Op, REC>(p, f, out, prm, g, key, cellx, cell_start, self, pair_counter, cf, pl);
}

// Replaying pass of an Op with PAIRS_FOR_FLUID_ONLY over the fluid work list of this cell-list
// generation (cell_list.cu k_fluid_scatter): work[0, *n_fluid) are the fluid positions ascending, the
// rest the other positions ascending.  Thread t handles p = work[t]; the list row of p and the order of
// its sum are those of k_binary_list, so every bit is too.  Whole warps run the pair loop or skip it
// (only the warp that straddles *n_fluid diverges), where a per-thread test would leave every warp
// that holds a fluid particle running the loop for all its lanes.
template <int DIM, class Op, bool REC = false>
__global__ void NL_LIST_BOUNDS
k_binary_list_fluid(Fields f, Fields out, Params prm, Grid g, const uint32_t *__restrict__ key,
                    const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, int64_t n,
                    int self, unsigned long long *pair_counter, ColFilter cf, PairList pl,
                    const uint32_t *__restrict__ work, const uint32_t *__restrict__ n_fluid) {
    static_assert(Op::PAIRS_FOR_FLUID_ONLY, "k_binary_list_fluid skips the pairs of non-fluid particles");
    const int64_t t = blockIdx.x * (int64_t)NL_BLOCK + threadIdx.x;
    if (t >= n) return;
    nl_list_particle<DIM, Op, REC>((int64_t)work[t], f, out, prm, g, key, cellx, cell_start, self, pair_counter, cf, pl,
                                   t < (int64_t)*n_fluid);
}

// The particles of the cell columns [a0, a1] and [b0, b1] are two contiguous ranges of the zrun
// cell order (x outermost): col_range() reads them off the cell-start table.
struct ColRanges {
    uint32_t b0, n0, b1, n1;  // first particle and length of each range, starts rounded down to a warp
};
__device__ __forceinline__ ColRanges col_ranges(const Grid &g, const ColFilter &cf, const uint32_t *__restrict__ cell_start) {
    ColRanges r{0, 0, 0, 0};
    const unsigned rows = (unsigned)g.rows;
    uint32_t end0 = 0;
    if (cf.a0 <= cf.a1) {
        r.b0 = cell_start[(unsigned)cf.a0 * rows] & ~31u;
        end0 = (cell_start[(unsigned)(cf.a1 + 1) * rows] + 31u) & ~31u;  // whole warps: the column filter
        r.n0 = end0 - r.b0;                                               // drops what is not selected
    }
    if (cf.b0 <= cf.b1) {
        r.b1 = cell_start[(unsigned)cf.b0 * rows] & ~31u;
        if (r.b1 < end0) r.b1 = end0;  // the two ranges meet in one warp: no particle is visited twice
        const uint32_t end1 = (cell_start[(unsigned)(cf.b1 + 1) * rows] + 31u) & ~31u;
        r.n1 = end1 > r.b1 ? end1 - r.b1 : 0u;
    }
    return r;
}
// Replaying pass over a FEW cell columns (the edge columns of the overlapped slab step: 2.5 % of a
// rank's particles): a small grid strides over the columns' particle ranges instead of launching a
// block for every 128 resident particles only to see most of them fail the column filter (0.23 ms
// of a 6.4 ms step at N = 8).  zrun cell order only.
template <int DIM, class Op, bool REC = false>
__global__ void __launch_bounds__(NL_BLOCK)
k_binary_list_cols(Fields f, Fields out, Params prm, Grid g, const uint32_t *__restrict__ key,
                   const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, int64_t n,
                   int self, unsigned long long *pair_counter, ColFilter cf, PairList pl) {
    const ColRanges r = col_ranges(g, cf, cell_start);
    const uint32_t total = r.n0 + r.n1;
    for (uint32_t t = blockIdx.x * NL_BLOCK + threadIdx.x; t < total; t += gridDim.x * NL_BLOCK) {
        const int64_t p = t < r.n0 ? (int64_t)r.b0 + t : (int64_t)r.b1 + (t - r.n0);
        if (p < n)
            nl_list_particle<DIM, Op, REC>(p, f, out, prm, g, key, cellx, cell_start, self, pair_counter, cf, pl,
                                           !Op::PAIRS_FOR_FLUID_ONLY || f.s[S_TYPE][p] == prm.fluid);
    }
}
