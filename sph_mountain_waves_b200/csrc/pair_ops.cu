// Particle operators on the device — replaces apply!/apply_unary!/apply_binary!
// (src/core.jl:94-161) and the driver closures they are called with
// (src/current/wcsph_perturbed_witch.jl:195-303, src/current/hopkins_*.jl,
// sph_jl/examples/collapse_dry.jl:112-159, sph_jl/tests/test_collision_2d.jl:66-97,
// src/utils/new_packing.jl:5-60).
//
// Closures cannot cross a C ABI (and the north star forbids JIT), so the menu of
// operators below is fixed; each one restates one reference closure as a device
// functor and is applied by the same two generic kernels.
//
// Arithmetic: this file is compiled with -fmad=false.  Every product/sum below is
// written in the reference's evaluation order (Julia's n-ary * and + fold left),
// so the FP64 sums are bit-identical to an IEEE evaluation of the reference
// wherever no transcendental (exp, pow, cbrt) is involved.
#include <math.h>
#include <stdlib.h>
#include <limits.h>
#include <string.h>

#include <string>

#include "cell_pairs.cuh"
#include "kernels_sph.cuh"
#include "pair_list.cuh"
#include "pair_tile.cuh"
#include "sphmw_internal.h"
#include "ops_menu.cuh"
#include "wcsph_ops.cuh"

template <int DIM, class Op>
__global__ void __launch_bounds__(256) k_unary(Fields f, Params c, int64_t n) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p < n) Op::template apply<DIM>(f, c, p);
}

// ---------------------------------------------------------------------------
// generic neighbour traversal — _apply_binary!  src/core.jl:94-112.
// One thread per particle (positions are cell-sorted, so a warp's particles sit
// in a handful of adjacent cells and its neighbour reads hit the same lines).
// Order of accumulation = the reference's: key_diff order (di outermost,
// structs.jl:73-81), then the cell's stored order (index descending).
// ---------------------------------------------------------------------------
template <int DIM, class Op>
__global__ void __launch_bounds__(128)
k_binary(Fields f, Fields out, Params prm, Grid g, const uint32_t *__restrict__ key,
         const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, int64_t n,
         int self, unsigned long long *pair_counter, ColFilter cf) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    const CellCoord home = cell_of(g, key[p], cellx[p]);
    if (cf.on) {  // slab mode: only the selected columns are evaluated
        if (!col_selected(cf, home.i)) {
            if (cf.copy) Op::template skip<DIM>(f, out, p);
            return;
        }
    }
    Op op;
    op.template init<DIM>(f, prm, p);
    const double px = f.s[S_X0][p], py = f.s[S_X1][p], pz = DIM == 3 ? f.s[S_X2][p] : 0.0;
    unsigned long long cnt = 0;
    for (int d = 0; d < g.ndiff; ++d) {
        unsigned nk;
        if (!neighbour_pkey(g, home, d, nk)) continue;  // core.jl:98 — no per-axis wrap check
        uint32_t b = cell_start[nk], e = cell_start[nk + 1];
        for (uint32_t q = b; q < e; ++q) {
            // dist(p,q) — core.jl:8-10, algebra.jl:49-60: left-to-right, no FMA
            double dx = px - f.s[S_X0][q];
            double dy = py - f.s[S_X1][q];
            double dz = 0.0;
            double r2 = dx * dx + dy * dy;
            if (DIM == 3) {
                dz = pz - f.s[S_X2][q];
                r2 = r2 + dz * dz;
            }
            // core.jl:105 `r > sys.h || p == q`, decided on r2 (Grid::r2_max): same set, bit for bit
            if ((r2 > g.r2_max) || (q == p)) continue;
            double r = sqrt(r2);
            op.template pair<DIM>(f, prm, p, q, dx, dy, dz, r);
            ++cnt;
        }
    }
    if (self) op.template pair<DIM>(f, prm, p, p, 0.0, 0.0, 0.0, 0.0);  // core.jl:155-157
    op.template finish<DIM>(f, out, prm, p);
    op.template after<DIM>(g, out, prm, p);
    if (pair_counter) {
        unsigned m = __activemask();
        unsigned tot = __reduce_add_sync(m, (unsigned)cnt);
        if ((int)(threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(pair_counter, (unsigned long long)tot);
    }
}

// accepted pairs in traversal order (test hook)
template <int DIM>
__global__ void k_pairs(Fields f, Grid g, const uint32_t *__restrict__ key,
                        const uint32_t *__restrict__ cellx, const uint32_t *__restrict__ cell_start, const uint32_t *__restrict__ idx,
                        const uint32_t *__restrict__ pos_of_idx, int64_t n,
                        const unsigned long long *__restrict__ offsets, long long *pi, long long *pj,
                        long long cap, unsigned long long *counts) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;  // reference index
    if (i >= n) return;
    int64_t p = pos_of_idx[i];
    const double px = f.s[S_X0][p], py = f.s[S_X1][p], pz = DIM == 3 ? f.s[S_X2][p] : 0.0;
    const CellCoord home = cell_of(g, key[p], cellx[p]);
    unsigned long long cnt = 0;
    unsigned long long base = offsets ? offsets[i] : 0;
    for (int d = 0; d < g.ndiff; ++d) {
        unsigned nk;
        if (!neighbour_pkey(g, home, d, nk)) continue;
        uint32_t b = cell_start[nk], e = cell_start[nk + 1];
        for (uint32_t q = b; q < e; ++q) {
            double dx = px - f.s[S_X0][q];
            double dy = py - f.s[S_X1][q];
            double r2 = dx * dx + dy * dy;
            if (DIM == 3) {
                double dz = pz - f.s[S_X2][q];
                r2 = r2 + dz * dz;
            }
            if ((r2 > g.r2_max) || ((int64_t)q == p)) continue;
            if (offsets && (long long)(base + cnt) < cap) {
                pi[base + cnt] = i;
                pj[base + cnt] = idx[q];
            }
            ++cnt;
        }
    }
    if (!offsets) counts[i] = cnt;
}

__global__ void k_scan_u64_serial(unsigned long long *a, int64_t n, unsigned long long *total) {
    // test hook only (small n): single-thread exclusive scan
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int64_t i = 0; i < n; ++i) {
            unsigned long long v = a[i];
            a[i] = run;
            run += v;
        }
        *total = run;
    }
}

int sphmw_dump_pairs(sphmw_ctx *c, int64_t *pi, int64_t *pj, int64_t cap, int64_t *nout) {
    if (!c->cell_list_valid) { sphmw_set_error("cell list is not built"); return SPHMW_E_STATE; }
    const int64_t n = c->n;
    *nout = 0;
    if (n == 0) return SPHMW_OK;
    TRY(sphmw_ensure_pos_of_idx(c));
    unsigned long long *counts = nullptr;
    long long *dpi = nullptr, *dpj = nullptr;
    CUDA_TRY(cudaMalloc(&counts, sizeof(unsigned long long) * (n + 1)));
    int rc = [&]() -> int {
        if (c->grid.dim == 2)
            k_pairs<2><<<grid_for(n, 128), 128, 0, c->stream>>>(c->cur, c->grid, c->key, c->cellx, c->cell_start,
                                                               c->idx, c->pos_of_idx, n, nullptr,
                                                               nullptr, nullptr, 0, counts);
        else
            k_pairs<3><<<grid_for(n, 128), 128, 0, c->stream>>>(c->cur, c->grid, c->key, c->cellx, c->cell_start,
                                                               c->idx, c->pos_of_idx, n, nullptr,
                                                               nullptr, nullptr, 0, counts);
        k_scan_u64_serial<<<1, 1, 0, c->stream>>>(counts, n, counts + n);
        unsigned long long total = 0;
        CUDA_TRY(cudaMemcpyAsync(&total, counts + n, sizeof(total), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        *nout = (int64_t)total;
        int64_t m = std::min<int64_t>((int64_t)total, cap);
        if (m <= 0 || !pi || !pj) return SPHMW_OK;
        CUDA_TRY(cudaMalloc(&dpi, sizeof(long long) * m));
        CUDA_TRY(cudaMalloc(&dpj, sizeof(long long) * m));
        if (c->grid.dim == 2)
            k_pairs<2><<<grid_for(n, 128), 128, 0, c->stream>>>(c->cur, c->grid, c->key, c->cellx, c->cell_start,
                                                               c->idx, c->pos_of_idx, n, counts, dpi,
                                                               dpj, m, nullptr);
        else
            k_pairs<3><<<grid_for(n, 128), 128, 0, c->stream>>>(c->cur, c->grid, c->key, c->cellx, c->cell_start,
                                                               c->idx, c->pos_of_idx, n, counts, dpi,
                                                               dpj, m, nullptr);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(pi, dpi, sizeof(long long) * m, cudaMemcpyDefault, c->stream));
        CUDA_TRY(cudaMemcpyAsync(pj, dpj, sizeof(long long) * m, cudaMemcpyDefault, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        return SPHMW_OK;
    }();
    cudaFree(counts);
    cudaFree(dpi);
    cudaFree(dpj);
    c->launches += 3;
    return rc;
}

// ===========================================================================
// operator menu and dispatch
// ===========================================================================
struct SlotList {
    int s[16];
    int n;
};
template <class... T>
static inline SlotList make_slot_list(T... v) {
    SlotList l{{(int)v...}, (int)sizeof...(v)};
    return l;
}
#define SL(...) make_slot_list(__VA_ARGS__)

// expand vector slots for the context's dimension
static int need_slots(sphmw_ctx *c, const SlotList &reads, const SlotList &writes) {
    auto expand = [&](int s, int out[3]) -> int {
        if (s == S_X0 || s == S_V0 || s == S_DV0) {
            out[0] = s;
            out[1] = s + 1;
            if (c->grid.dim == 3) { out[2] = s + 2; return 3; }
            return 2;
        }
        out[0] = s;
        return 1;
    };
    for (int i = 0; i < reads.n; ++i) {
        int e[3];
        int m = expand(reads.s[i], e);
        for (int k = 0; k < m; ++k) {
            if (c->allocated[e[k]] && c->stale[e[k]]) TRY(sphmw_materialize(c, e[k]));
            TRY(sphmw_ensure_slot(c, e[k]));  // unset fields read as the constructor's zero
        }
    }
    for (int i = 0; i < writes.n; ++i) {
        int e[3];
        int m = expand(writes.s[i], e);
        for (int k = 0; k < m; ++k) {
            if (c->allocated[e[k]] && c->stale[e[k]]) {
                // about to be (partly) overwritten: bring it up to date first so that
                // gated writes (type == FLUID) keep the other particles' values
                TRY(sphmw_materialize(c, e[k]));
            }
            TRY(sphmw_ensure_slot(c, e[k]));
            c->stale[e[k]] = false;
        }
    }
    return SPHMW_OK;
}

template <class Op>
static int run_unary(sphmw_ctx *c, const char *name) {
    c->keys_from_advance = false;  // the operator may move particles
    if (c->n == 0) return SPHMW_OK;
    TIMED(c, name);
    if (c->grid.dim == 2)
        k_unary<2, Op><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->n);
    else
        k_unary<3, Op><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->n);
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}

// ghost_depth: how many ghost columns (from the owned range outwards) the pass must also
// evaluate in slab mode; ignored for whole-domain contexts
static ColFilter filter_for_depth(sphmw_ctx *c, int ghost_depth) {
    ColFilter cf{0, 0, (int)c->grid.lim[0] - 1, 1, 0, 1};
    if (c->slab_lo >= 0 && ghost_depth < c->grid.ghost) {
        cf.on = 1;
        cf.a0 = c->grid.ghost - ghost_depth;
        cf.a1 = (int)c->grid.lim[0] - 1 - cf.a0;
    }
    return cf;
}

template <class Op, bool REC = false>
static int run_binary_cols(sphmw_ctx *c, const char *name, int self, const Fields &out, ColFilter cf);
#define GHOST_COLS_ALL 99  // ghost_depth: every ghost column the context keeps

template <class Op, bool REC = false>
static int run_binary(sphmw_ctx *c, const char *name, int self, const Fields &out,
                      int ghost_depth = GHOST_COLS_ALL) {
    return run_binary_cols<Op, REC>(c, name, self, out, filter_for_depth(c, ghost_depth));
}

// device memory of the pair list, allocated on first use
static int ensure_pair_list(sphmw_ctx *c) {
    if (c->pl.list) return SPHMW_OK;
    int stride = c->grid.dim == 3 ? 40 : 32;
    if (const char *e = getenv("SPHMW_PAIR_LIST_STRIDE")) stride = atoi(e);
    if (stride < 4) stride = 4;
    if (stride > 92) stride = 92;  // (stride + NL_QUEUE_SLACK) rows: 48 KB of queue per block
    const size_t warps = (size_t)((c->cap + 31) / 32);
    uint32_t *list = nullptr, *cnt = nullptr;
    if (cudaMalloc(&list, sizeof(uint32_t) * warps * (size_t)stride * 32) != cudaSuccess ||
        cudaMalloc(&cnt, sizeof(uint32_t) * (size_t)c->cap) != cudaSuccess) {
        cudaFree(list);
        (void)cudaGetLastError();  // out of memory is not fatal here: the caller walks the cells instead
        sphmw_set_error("no device memory for the pair list (%zu MB)", sizeof(uint32_t) * warps * (size_t)stride * 32 >> 20);
        return SPHMW_E_CAPACITY;
    }
    c->pl.list = list;
    c->pl.cnt = cnt;
    c->pl.stride = stride;
    // queue rows: a particle of a resolved flow has 26-29 neighbours in 3D (h = 1.8 dr) and the 6-bit
    // pre-test lets ~8 % more through; one with more survivors than rows - 4 walks the cells instead
    int qrows = c->grid.dim == 3 ? 36 : 28;
    if (const char *e = getenv("SPHMW_PAIR_QUEUE_ROWS")) qrows = atoi(e);
    qrows = std::min(qrows, stride + NL_QUEUE_SLACK);
    c->pl.qrows = std::max(qrows, 2 * NL_QUEUE_SLACK);
    c->pl.overflow = c->d_counters + 2;
    return SPHMW_OK;
}

int sphmw_pair_list_stats(sphmw_ctx *c, int64_t out[4]) {
    out[0] = c->pl.stride;
    out[1] = c->pl_builds;
    CUDA_TRY(cudaMemcpyAsync(c->h_counters + 2, c->d_counters + 2, sizeof(unsigned long long),
                             cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    out[2] = (int64_t)c->h_counters[2];
    out[3] = c->pl.list ? (int64_t)(sizeof(uint32_t) * ((size_t)((c->cap + 31) / 32) * c->pl.stride * 32 + c->cap))
                        : 0;
    return SPHMW_OK;
}

// Three ways to run one binary pass (same results bit for bit):
//   list valid for this cell list      -> k_binary_list   (replay)
//   a list is wanted and none exists   -> k_binary_build  (walk once, record)
//   otherwise                          -> k_binary        (walk)
// REC (the two fused WCSPH passes with SPHMW_FLAG_PACKED_RECORDS): the list kernels read their
// neighbours from the packed records; needs record A of this cell-list generation.
template <class Op, bool REC>
static int run_binary_cols(sphmw_ctx *c, const char *name, int self, const Fields &out, ColFilter cf) {
    if (!c->cell_list_valid) {
        sphmw_set_error("%s: create_cell_list must be called after positions change", name);
        return SPHMW_E_STATE;
    }
    if (c->n == 0) return SPHMW_OK;
    unsigned long long *pc = c->count_pairs ? c->d_counters : nullptr;
    if (pc) CUDA_TRY(cudaMemsetAsync(pc, 0, sizeof(unsigned long long), c->stream));
    const bool lists = !(c->flags & SPHMW_FLAG_NO_PAIR_LIST);
    const bool replay = lists && c->pl.list && c->pl_gen == c->cell_gen && c->pl_format == 0;
    bool record = lists && !replay && (c->want_list || (c->flags & SPHMW_FLAG_PAIR_LIST_EAGER));
    if (record && ensure_pair_list(c) != SPHMW_OK) {
        // the list is an optimisation: without memory for it every pass walks the cells
        c->flags |= SPHMW_FLAG_NO_PAIR_LIST;
        record = false;
    }
    c->passes_this_gen += 1;
    const unsigned blocks = grid_for(c->n, NL_BLOCK);
    const bool rec = REC && c->rec[0] && c->rec[1] && c->rec[2] && c->rec_gen == c->cell_gen;
    c->pl.recA = c->rec[0];
    c->pl.recB = c->rec[1];
    c->pl.recC = c->rec[2];
#define NL_ARGS c->cur, out, c->prm, c->grid, c->key, c->cellx, c->cell_start, c->n, self, pc, cf
    if (replay) {
        TIMED(c, name);
        // a few columns only (edge columns of the overlapped slab step): a small grid strides over
        // their particle ranges, which are contiguous in the zrun cell order
        const bool cols = cf.on && cf.sparse && !cf.copy && c->grid.zrun && !getenv("SPHMW_NO_COLUMN_RANGES");
        const unsigned cblocks = std::min<unsigned>(blocks, (unsigned)c->sm_count * 8u);
        // an Op whose finish() discards the pair sums of non-fluid particles runs over the fluid work
        // list of this cell list: the pair loop for the fluid positions only (pair_list.cuh)
        bool fluid = false;
        if constexpr (Op::PAIRS_FOR_FLUID_ONLY)
            fluid = !cols && c->fluid_gen == c->cell_gen && c->fluid_value == c->prm.fluid;
#define NL_FLUID_ARGS NL_ARGS, c->pl, c->fluid_work, c->fluid_count
        if constexpr (REC) {
            if (rec && c->rec_bc_gen == c->cell_gen) {
                if (cols) {
                    if (c->grid.dim == 2) k_binary_list_cols<2, Op, true><<<cblocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
                    else k_binary_list_cols<3, Op, true><<<cblocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
                } else if (fluid) {
                    if constexpr (Op::PAIRS_FOR_FLUID_ONLY) {
                        if (c->grid.dim == 2) k_binary_list_fluid<2, Op, true><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_FLUID_ARGS);
                        else k_binary_list_fluid<3, Op, true><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_FLUID_ARGS);
                    }
                } else {
                    if (c->grid.dim == 2) k_binary_list<2, Op, true><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
                    else k_binary_list<3, Op, true><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
                }
                CUDA_TRY(cudaGetLastError());
                return SPHMW_OK;
            }
        }
        if (cols) {
            if (c->grid.dim == 2) k_binary_list_cols<2, Op><<<cblocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
            else k_binary_list_cols<3, Op><<<cblocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
        } else if (fluid) {
            if constexpr (Op::PAIRS_FOR_FLUID_ONLY) {
                if (c->grid.dim == 2) k_binary_list_fluid<2, Op><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_FLUID_ARGS);
                else k_binary_list_fluid<3, Op><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_FLUID_ARGS);
            }
        } else if (c->grid.dim == 2)
            k_binary_list<2, Op><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
        else
            k_binary_list<3, Op><<<blocks, NL_BLOCK, 0, c->stream>>>(NL_ARGS, c->pl);
    } else if (record) {
        c->pl.xq = c->xq;
        // pre-test of the recording pass: integers on the 6-bit mirror of the zrun cell order, or
        // (SPHMW_FLAG_NO_PRETEST, x-chunked cell order) the exact FP64 test only
        const bool q6 = c->grid.zrun && !(c->flags & SPHMW_FLAG_NO_PRETEST);
        const size_t smem = sizeof(uint32_t) * (size_t)c->pl.qrows * NL_BLOCK;
        TIMED(c, name);
        c->pl_gen = c->cell_gen;
        c->pl_format = 0;
        c->pl_builds += 1;
        if constexpr (REC) {
            if (rec && q6) {
                if (c->grid.dim == 2)
                    k_binary_build<2, Op, NL_FILTER_Q6, true><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
                else
                    k_binary_build<3, Op, NL_FILTER_Q6, true><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
                if (Op::REC_KIND == 1) c->rec_bc_gen = c->cell_gen;
                CUDA_TRY(cudaGetLastError());
                return SPHMW_OK;
            }
        }
        if (c->grid.dim == 2) {
            if (q6) k_binary_build<2, Op, NL_FILTER_Q6><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
            else k_binary_build<2, Op, NL_FILTER_F64><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
        } else {
            if (q6) k_binary_build<3, Op, NL_FILTER_Q6><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
            else k_binary_build<3, Op, NL_FILTER_F64><<<blocks, NL_BLOCK, smem, c->stream>>>(NL_ARGS, c->pl);
        }
    } else {
        // Measured on B200 (profiles/r01_tuning.md): forcing 6 or 8 resident blocks per SM
        // (64 registers), 64-thread blocks and software prefetch of the next candidate were all
        // neutral or slower than this plain configuration.
        TIMED(c, name);
        if (c->grid.dim == 2)
            k_binary<2, Op><<<blocks, 128, 0, c->stream>>>(NL_ARGS);
        else
            k_binary<3, Op><<<blocks, 128, 0, c->stream>>>(NL_ARGS);
    }
#undef NL_ARGS
#undef NL_FLUID_ARGS
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// tiled passes (pair_tile.cuh): neighbourhood of each block staged in shared memory
// ---------------------------------------------------------------------------
static int ensure_tile_buffers(sphmw_ctx *c) {
    if (c->pl.list16 && c->tile_tab) return SPHMW_OK;
    int stride = c->grid.dim == 3 ? 40 : 32;
    if (const char *e = getenv("SPHMW_PAIR_LIST_STRIDE")) stride = atoi(e);
    stride = (stride + 1) & ~1;
    if (stride < 4) stride = 4;
    if (stride > 96) stride = 96;
    if (c->pl.list && c->pl.stride != stride) stride = c->pl.stride & ~1;  // one stride per context
    const size_t warps = (size_t)((c->cap + 31) / 32);
    const size_t blocks = (size_t)((c->cap + TM_BLOCK - 1) / TM_BLOCK);
    uint32_t *l16 = nullptr, *tab = nullptr, *cnt = c->pl.cnt;
    bool ok = cudaMalloc(&l16, sizeof(uint32_t) * warps * (size_t)(stride / 2) * 32) == cudaSuccess &&
              cudaMalloc(&tab, sizeof(uint32_t) * blocks * TM_WORDS) == cudaSuccess;
    if (ok && !cnt) ok = cudaMalloc(&cnt, sizeof(uint32_t) * (size_t)c->cap) == cudaSuccess;
    if (!ok) {
        cudaFree(l16);
        cudaFree(tab);
        (void)cudaGetLastError();
        sphmw_set_error("no device memory for the tiled pair list");
        return SPHMW_E_CAPACITY;
    }
    c->pl.list16 = l16;
    c->tile_tab = tab;
    c->pl.cnt = cnt;
    c->pl.stride = stride;
    c->pl.overflow = c->d_counters + 2;
    return SPHMW_OK;
}

static int ensure_tile_map(sphmw_ctx *c) {
    if (c->tile_gen == c->cell_gen) return SPHMW_OK;
    const int64_t nblocks = (c->n + TM_BLOCK - 1) / TM_BLOCK;
    TIMED(c, "tile_map");
    k_tile_map<<<grid_for(nblocks * 32, 128), 128, 0, c->stream>>>(c->grid, c->key, c->cellx, c->cell_start, c->n,
                                                                  nblocks, c->tile_tab);
    CUDA_TRY(cudaGetLastError());
    c->tile_gen = c->cell_gen;
    return SPHMW_OK;
}

// blocks / blocks with a tile / largest tile / slots of all tiles / capacity / blocks over too many rows
__global__ void k_tile_stats(const uint32_t *__restrict__ tab, int64_t nblocks, int max_pieces, uint32_t cap,
                             unsigned long long *__restrict__ out) {
    const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const uint32_t *rec = tab + (size_t)b * TM_WORDS;
    const bool pieces_ok = rec[1] <= (uint32_t)max_pieces;
    if (pieces_ok && rec[2] <= cap) {
        atomicAdd(&out[0], 1ull);
        atomicAdd(&out[2], (unsigned long long)rec[2]);
    }
    if (pieces_ok) atomicMax(&out[1], (unsigned long long)rec[2]);
    else atomicAdd(&out[3], 1ull);
}

int sphmw_tile_stats(sphmw_ctx *c, int64_t out[6]) {
    for (int k = 0; k < 6; ++k) out[k] = 0;
    out[4] = c->grid.dim == 3 ? TileGeom<3>::CAP : TileGeom<2>::CAP;
    if (!c->tile_tab || c->tile_gen != c->cell_gen || c->n == 0) return SPHMW_OK;
    const int64_t nblocks = (c->n + TM_BLOCK - 1) / TM_BLOCK;
    unsigned long long *d = c->d_counters + 3;
    CUDA_TRY(cudaMemsetAsync(d, 0, sizeof(unsigned long long) * 4, c->stream));
    k_tile_stats<<<grid_for(nblocks, 256), 256, 0, c->stream>>>(c->tile_tab, nblocks, tm_max_pieces(c->grid),
                                                               (uint32_t)out[4], d);
    CUDA_TRY(cudaMemcpyAsync(c->h_counters + 3, d, sizeof(unsigned long long) * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    out[0] = nblocks;
    out[1] = (int64_t)c->h_counters[3];
    out[2] = (int64_t)c->h_counters[4];
    out[3] = (int64_t)c->h_counters[5];
    out[5] = (int64_t)c->h_counters[6];
    return SPHMW_OK;
}

template <class K>
static int tile_smem_attr(K kernel, int bytes) {
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return SPHMW_OK;
}

static bool tiles_enabled(const sphmw_ctx *c) {
    return (c->flags & SPHMW_FLAG_TILES) &&
           !(c->flags & (SPHMW_FLAG_NO_PAIR_LIST | SPHMW_FLAG_CELL_PAIRS | SPHMW_FLAG_NO_PRETEST));
}

// One fused pass through the tiled kernels: the first pass of a cell-list generation records
// (k_tile_build), later ones replay (k_tile_list).
template <class Op>
static int run_tiled(sphmw_ctx *c, const char *name, int self, const Fields &out, ColFilter cf) {
    if (!c->cell_list_valid) {
        sphmw_set_error("%s: create_cell_list must be called after positions change", name);
        return SPHMW_E_STATE;
    }
    if (c->n == 0) return SPHMW_OK;
    TRY(ensure_tile_buffers(c));
    TRY(ensure_tile_map(c));
    unsigned long long *pc = c->count_pairs ? c->d_counters : nullptr;
    if (pc) CUDA_TRY(cudaMemsetAsync(pc, 0, sizeof(unsigned long long), c->stream));
    c->passes_this_gen += 1;
    c->pl.xq = c->xq;
    const unsigned blocks = grid_for(c->n, TM_BLOCK);
    const bool replay = c->pl_gen == c->cell_gen && c->pl_format == 1;
#define TL_ARGS c->cur, out, c->prm, c->grid, c->key, c->cellx, c->cell_start, c->n, self, pc, cf, c->pl, c->tile_tab
    if (replay) {
        static bool attr2 = false, attr3 = false;
        TIMED(c, name);
        if (c->grid.dim == 2) {
            constexpr int smem = tile_bytes_list<2, Op>();
            if (!attr2) { TRY(tile_smem_attr(k_tile_list<2, Op>, smem)); attr2 = true; }
            k_tile_list<2, Op><<<blocks, TM_BLOCK, smem, c->stream>>>(TL_ARGS);
        } else {
            constexpr int smem = tile_bytes_list<3, Op>();
            if (!attr3) { TRY(tile_smem_attr(k_tile_list<3, Op>, smem)); attr3 = true; }
            k_tile_list<3, Op><<<blocks, TM_BLOCK, smem, c->stream>>>(TL_ARGS);
        }
    } else {
        static int attr2 = 0, attr3 = 0;
        TIMED(c, name);
        c->pl_gen = c->cell_gen;
        c->pl_format = 1;
        c->pl_builds += 1;
        if (c->grid.dim == 2) {
            const int smem = tile_bytes_build<2, Op>(c->pl.stride);
            if (attr2 != smem) { TRY(tile_smem_attr(k_tile_build<2, Op>, smem)); attr2 = smem; }
            k_tile_build<2, Op><<<blocks, TM_BLOCK, smem, c->stream>>>(TL_ARGS);
        } else {
            const int smem = tile_bytes_build<3, Op>(c->pl.stride);
            if (attr3 != smem) { TRY(tile_smem_attr(k_tile_build<3, Op>, smem)); attr3 = smem; }
            k_tile_build<3, Op><<<blocks, TM_BLOCK, smem, c->stream>>>(TL_ARGS);
        }
    }
#undef TL_ARGS
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}

// the fused WCSPH passes: cell-centric pair-parallel kernel (cell_pairs.cuh)
template <class OP>
static int run_cell_pairs(sphmw_ctx *c, const char *name, const Fields &out, int ghost_depth) {
    if (!c->cell_list_valid) {
        sphmw_set_error("%s: create_cell_list must be called after positions change", name);
        return SPHMW_E_STATE;
    }
    if (c->n == 0) return SPHMW_OK;
    unsigned long long *pc = c->count_pairs ? c->d_counters : nullptr;
    if (pc) CUDA_TRY(cudaMemsetAsync(pc, 0, sizeof(unsigned long long), c->stream));
    int col_lo = 0, col_hi = (int)c->grid.lim[0] - 1;
    if (c->slab_lo >= 0 && ghost_depth < c->grid.ghost) {
        col_lo = c->grid.ghost - ghost_depth;
        col_hi = (int)c->grid.lim[0] - 1 - col_lo;
    }
    // persistent grid: a multiple of the SM count, warps stride over the cells
    const long long warps_needed = c->grid.pkey_max;
    long long blocks = (warps_needed + CP_WARPS - 1) / CP_WARPS;
    const long long max_blocks = (long long)c->sm_count * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    TIMED(c, name);
    if (c->grid.dim == 2)
        k_cell_pairs<2, OP><<<(unsigned)blocks, CP_WARPS * 32, 0, c->stream>>>(
            c->cur, out, c->prm, c->grid, c->cell_start, c->cellx, col_lo, col_hi, pc);
    else
        k_cell_pairs<3, OP><<<(unsigned)blocks, CP_WARPS * 32, 0, c->stream>>>(
            c->cur, out, c->prm, c->grid, c->cell_start, c->cellx, col_lo, col_hi, pc);
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}

struct OpEntry {
    const char *name;
    bool binary;
    int (*run)(sphmw_ctx *, const char *, int);
};

#define UNARY_ENTRY(NAME, OP, READS, WRITES, EXTRA)                         \
    {NAME, false, [](sphmw_ctx *c, const char *nm, int) -> int {            \
         TRY(need_slots(c, READS, WRITES));                                 \
         TRY(run_unary<OP>(c, nm));                                         \
         EXTRA;                                                             \
         return SPHMW_OK;                                                   \
     }},
#define BINARY_ENTRY(NAME, OP, READS, WRITES, EXTRA)                        \
    {NAME, true, [](sphmw_ctx *c, const char *nm, int self) -> int {        \
         TRY(need_slots(c, READS, WRITES));                                 \
         TRY((run_binary<OP>(c, nm, self, c->cur)));                        \
         EXTRA;                                                             \
         return SPHMW_OK;                                                   \
     }},

static const OpEntry OPS[] = {
    SPHMW_OPERATOR_MENU(UNARY_ENTRY, BINARY_ENTRY)
    {nullptr, false, nullptr}};

int64_t sphmw_list_ops(char *buf, int64_t cap) {
    std::string all;
    for (const OpEntry *e = OPS; e->name; ++e) {
        all += e->name;
        all += e->binary ? " binary\n" : " unary\n";
    }
    if (buf && cap > 0) {
        size_t k = std::min<size_t>(all.size(), (size_t)cap - 1);
        memcpy(buf, all.data(), k);
        buf[k] = 0;
    }
    return (int64_t)all.size() + 1;
}

int sphmw_apply_named(sphmw_ctx *c, const char *op, int self) {
    for (const OpEntry *e = OPS; e->name; ++e)
        if (!strcmp(e->name, op)) {
            if (self && !e->binary) {
                // core.jl:151-161: `self` only matters for binary operators
                self = 0;
            }
            c->fluid_gen = ~0ull;  // an operator may change a particle's type (inflow conversion)
            c->keys_from_advance = false;  // ... or its position
            return e->run(c, e->name, self);
        }
    sphmw_set_error("operator '%s' is not in the device menu (no CPU fallback)", op);
    return SPHMW_E_UNSUPPORTED_OP;
}

// ---------------------------------------------------------------------------
// lazily evaluated fields.  After a fused "wcsph" step T, T', theta, theta_bg,
// theta' (diagnostics that never feed back, SURVEY quirk 11) are stale; they are
// rebuilt here by the very operators the reference runs every step
// (find_temperature!, find_pot_temp!), from P, rho, x that have not changed since.
// ---------------------------------------------------------------------------
int sphmw_materialize(sphmw_ctx *c, int slot) {
    if ((slot >= S_T_P && slot <= S_T) || (slot >= S_TH_BG && slot <= S_TH)) {
        bool want = c->allocated[slot] ? c->stale[slot] : true;
        if (!want) return SPHMW_OK;
        if (!c->allocated[S_P] || !c->allocated[S_RHO]) return SPHMW_OK;  // nothing to derive from
        for (int s : {S_T_P, S_T, S_TH_BG, S_TH_P, S_TH}) {
            TRY(sphmw_ensure_slot(c, s));
            c->stale[s] = false;
        }
        TRY(sphmw_ensure_slot(c, S_T_BG));
        TRY(run_unary<U_wcsph_find_temperature>(c, "wcsph.find_temperature"));
        TRY(run_unary<U_wcsph_find_pot_temp>(c, "wcsph.find_pot_temp"));
        return SPHMW_OK;
    }
    if (c->allocated[slot] && c->stale[slot]) {
        if (slot >= S_DV0 && slot <= S_DV2 && c->dv_zero) {
            CUDA_TRY(cudaMemsetAsync(c->cur.s[slot], 0, sizeof(double) * c->cap, c->stream));
            c->stale[slot] = false;
            return SPHMW_OK;
        }
        sphmw_set_error("internal: slot %d is stale and has no rule", slot);
        return SPHMW_E_STATE;
    }
    return SPHMW_OK;
}

// ===========================================================================
// add_new_particles!  src/legacy/isothermal_flow_witch.jl:175-186
// ===========================================================================
template <int DIM>
__global__ void k_flow_flag(Fields f, Params c, const uint32_t *__restrict__ idx, int64_t n,
                            uint32_t *__restrict__ flag_by_idx) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    flag_by_idx[idx[p]] = (f.s[S_TYPE][p] == c.inflow && f.s[S_X0][p] >= c.x_inflow) ? 1u : 0u;
}

// Particle(x - bc_width*VECX, U_max*VECX, INFLOW) of the flow drivers, built in slot s from the
// converting particle p: isothermal_flow_witch.jl:72-82; ADIABATIC: adiabatic_flow_witch.jl:82-91
// (T = T0, entropy from T and rho)
template <int DIM, bool ADIABATIC>
__device__ __forceinline__ void flow_construct(const Fields &f, const Params &c, int64_t p, int64_t s) {
    const double y = f.s[S_X1][p] - c.bc_width * 0.0;
    f.s[S_X0][s] = f.s[S_X0][p] - c.bc_width * 1.0;
    f.s[S_X1][s] = y;
    if (DIM == 3) f.s[S_X2][s] = f.s[S_X2][p] - c.bc_width * 0.0;
    f.s[S_V0][s] = c.U_max * 1.0;
    f.s[S_V1][s] = c.U_max * 0.0;
    if (DIM == 3) f.s[S_V2][s] = c.U_max * 0.0;
    const double rho = c.rho0 * exp(-y * c.g / (c.R_mass * c.T_bg));
    f.s[S_RHO][s] = rho;
    const double m = rho * sph_pow2(c.dr);
    f.s[S_M][s] = m;
    if (ADIABATIC) {
        const double T = c.T_bg, cv = c.cp - c.R_mass;
        const double P = c.R_mass * T * rho;
        const double b = (c.T_bg * c.R_gas * c.rho0) / P;
        f.s[S_T][s] = T;
        f.s[S_P][s] = P;
        f.s[S_TH][s] = T * pow(b * b, 1.0 / 7.0);
        f.s[S_ENT][s] = m * cv * log((cv * T * (c.gamma - 1.0)) / (c.gamma * pow(rho, c.gamma - 1.0)));
    } else {
        const double P = rho * c.T_bg * c.R_mass;
        f.s[S_P][s] = P;
        f.s[S_TH][s] = c.T_bg * pow((c.T_bg * c.R_gas * c.rho0) / P, c.R_gas / c.cp);
    }
    f.s[S_TYPE][s] = c.inflow;
}

// One thread per old particle; a converting particle creates its successor at index
// n + (number of converting particles with a smaller index): the order of the reference's loop.
template <int DIM, bool ADIABATIC>
__global__ void k_flow_spawn(Fields f, Params c, uint32_t *__restrict__ idx,
                             uint32_t *__restrict__ pos_of_idx, uint32_t *__restrict__ tag, int64_t n,
                             const uint32_t *__restrict__ rank_by_idx) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    if (!(f.s[S_TYPE][p] == c.inflow && f.s[S_X0][p] >= c.x_inflow)) return;
    f.s[S_TYPE][p] = c.fluid;
    const int64_t s = n + rank_by_idx[idx[p]];
    flow_construct<DIM, ADIABATIC>(f, c, p, s);
    idx[s] = (uint32_t)s;
    pos_of_idx[s] = (uint32_t)s;
    tag[s] = TAG_OWNED;
}

// ---- slab contexts (slab_comm.cu): the converting particles of ALL ranks are ranked by global
// index on the host, so the device only collects them and later builds the successors it is told to
template <int DIM>
__global__ void k_flow_collect(Fields f, Params c, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ tag,
                               int64_t n, uint32_t *__restrict__ list, uint32_t *__restrict__ pos, uint32_t cap) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n || tag[p] != TAG_OWNED) return;
    if (!(f.s[S_TYPE][p] == c.inflow && f.s[S_X0][p] >= c.x_inflow)) return;
    const uint32_t slot = atomicAdd(&list[0], 1u);
    if (slot < cap) {
        list[1 + slot] = idx[p];
        pos[slot] = (uint32_t)p;
    }
}
template <int DIM, bool ADIABATIC>
__global__ void k_flow_spawn_list(Fields f, Params c, uint32_t *__restrict__ idx, uint32_t *__restrict__ tag, int64_t n,
                                  const uint32_t *__restrict__ pos, const uint32_t *__restrict__ new_idx, int m) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int64_t p = pos[k], s = n + k;
    f.s[S_TYPE][p] = c.fluid;
    flow_construct<DIM, ADIABATIC>(f, c, p, s);
    idx[s] = new_idx[k];
    tag[s] = TAG_OWNED;
}
// collect: list[0] = count, list[1..] = global indices, pos[k] = physical position (device arrays)
int sphmw_flow_collect_slab(sphmw_ctx *c, uint32_t *list, uint32_t *pos, uint32_t cap, bool adiabatic) {
    TRY(need_slots(c, SL(S_X0, S_V0, S_TYPE, S_RHO, S_M, S_P, S_TH), SL(S_X0, S_V0, S_TYPE, S_RHO, S_M, S_P, S_TH)));
    if (adiabatic) TRY(need_slots(c, SL(S_T, S_ENT), SL(S_T, S_ENT)));
    CUDA_TRY(cudaMemsetAsync(list, 0, sizeof(uint32_t), c->stream));
    if (c->n == 0) return SPHMW_OK;
    TIMED(c, "flow.flag_inflow");
    if (c->grid.dim == 2) k_flow_collect<2><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, c->tag, c->n, list, pos, cap);
    else k_flow_collect<3><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, c->tag, c->n, list, pos, cap);
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}
// build m successors at the end of the resident set: pos[k] converts, its successor gets new_idx[k]
int sphmw_flow_spawn_slab(sphmw_ctx *c, const uint32_t *pos, const uint32_t *new_idx, int m, bool adiabatic) {
    if (m <= 0) return SPHMW_OK;
    const int64_t n = c->n;
    if (n + m > c->cap) {
        sphmw_set_error("add_new_particles: %lld + %d particles exceed capacity %lld", (long long)n, m, (long long)c->cap);
        return SPHMW_E_CAPACITY;
    }
    for (int s = 0; s < NSLOT; ++s)  // every other field of a new particle is the constructor's zero
        if (c->allocated[s]) CUDA_TRY(cudaMemsetAsync(c->cur.s[s] + n, 0, sizeof(double) * m, c->stream));
    TIMED(c, "flow.spawn_inflow");
#define SPAWN_LIST(D, A) k_flow_spawn_list<D, A><<<grid_for(m, 128), 128, 0, c->stream>>>(c->cur, c->prm, c->idx, c->tag, n, pos, new_idx, m)
    if (c->grid.dim == 2) {
        if (adiabatic) SPAWN_LIST(2, true);
        else SPAWN_LIST(2, false);
    } else {
        if (adiabatic) SPAWN_LIST(3, true);
        else SPAWN_LIST(3, false);
    }
#undef SPAWN_LIST
    CUDA_TRY(cudaGetLastError());
    c->n = n + m;
    c->keys_from_advance = false;
    c->n_owned += m;
    c->cell_list_valid = false;
    return SPHMW_OK;
}

int sphmw_flow_add_particles(sphmw_ctx *c, int64_t *n_added, bool adiabatic) {
    if (n_added) *n_added = 0;
    if (c->slab_lo >= 0) {
        // the successors' global indices follow from the converting particles of ALL ranks: collective
        // (slab_comm.cu), through the library transport with the open box
        if (!c->comm) {
            sphmw_set_error("add_new_particles: a slab context re-seeds its inflow through the library transport "
                            "(sphmw_comm_init + sphmw_comm_open_box)");
            return SPHMW_E_STATE;
        }
        return sphmw_comm_add_new_particles(c, n_added, adiabatic);
    }
    const int64_t n = c->n;
    if (n == 0) return SPHMW_OK;
    TRY(need_slots(c, SL(S_X0, S_V0, S_TYPE, S_RHO, S_M, S_P, S_TH), SL(S_X0, S_V0, S_TYPE, S_RHO, S_M, S_P, S_TH)));
    if (adiabatic) TRY(need_slots(c, SL(S_T, S_ENT), SL(S_T, S_ENT)));
    uint32_t *flags = c->rank;  // scratch of the cell-list build, free between builds
    {
        TIMED(c, "flow.flag_inflow");
        if (c->grid.dim == 2) k_flow_flag<2><<<grid_for(n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, n, flags);
        else k_flow_flag<3><<<grid_for(n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, n, flags);
    }
    // total = last flag + its exclusive prefix
    uint32_t last_flag = 0, last_rank = 0;
    CUDA_TRY(cudaMemcpyAsync(&last_flag, flags + n - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    TRY(sphmw_exclusive_scan_u32(c, flags, n));
    CUDA_TRY(cudaMemcpyAsync(&last_rank, flags + n - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int64_t m = (int64_t)last_flag + last_rank;
    if (m == 0) return SPHMW_OK;
    if (n + m > c->cap) {
        sphmw_set_error("add_new_particles: %lld + %lld particles exceed capacity %lld", (long long)n,
                        (long long)m, (long long)c->cap);
        return SPHMW_E_CAPACITY;
    }
    // every other field of a new particle is the constructor's zero
    for (int s = 0; s < NSLOT; ++s)
        if (c->allocated[s]) CUDA_TRY(cudaMemsetAsync(c->cur.s[s] + n, 0, sizeof(double) * m, c->stream));
    {
        TIMED(c, "flow.spawn_inflow");
#define SPAWN(D, A) k_flow_spawn<D, A><<<grid_for(n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, c->pos_of_idx, c->tag, n, flags)
        if (c->grid.dim == 2) {
            if (adiabatic) SPAWN(2, true);
            else SPAWN(2, false);
        } else {
            if (adiabatic) SPAWN(3, true);
            else SPAWN(3, false);
        }
#undef SPAWN
    }
    CUDA_TRY(cudaGetLastError());
    c->n = n + m;
    c->keys_from_advance = false;
    c->n_owned = c->n;
    c->cell_list_valid = false;
    if (n_added) *n_added = m;
    return SPHMW_OK;
}

// ===========================================================================
// fused stepping
// ===========================================================================
static int apply_seq(sphmw_ctx *c, std::initializer_list<const char *> ops) {
    for (const char *o : ops) {
        if (!strcmp(o, "create_cell_list")) TRY(sphmw_build_cell_list(c, nullptr));
        else if (o[0] == '+') TRY(sphmw_apply_named(c, o + 1, 1));
        else TRY(sphmw_apply_named(c, o, 0));
    }
    return SPHMW_OK;
}

// wcsph_perturbed_witch.jl:309-332 with the unary sweeps fused into the two pair
// passes; the redundant second create_cell_list! (:320, positions unchanged —
// SURVEY quirk 4) is skipped.
// bookkeeping after accelerate! + move!: positions changed, derived fields are void
static void wcsph_after_drift(sphmw_ctx *c) {
    // Dv is identically zero from here on and is not carried through the sort
    for (int s = S_DV0; s <= S_DV2; ++s)
        if (c->allocated[s]) c->stale[s] = true;
    c->cell_list_valid = false;
    // diagnostics and per-step derived fields need not travel through the reorder
    for (int s : {S_RHO_BG, S_P_BG, S_P_P, S_P, S_T_P, S_T, S_TH_BG, S_TH_P, S_TH, S_PR2, S_CS})
        if (c->allocated[s]) c->stale[s] = true;
}

// rho and rho' were last read by the kick that opened this step (and, on a slab context, by the halo
// pack that followed the drift) and are rewritten by the density pass for every particle a later
// pass reads them from: they need not travel through the sort.  (The outermost ghost column keeps
// no density at all: nothing reads it — the force pass stops one column short of it.)
static void wcsph_before_sort(sphmw_ctx *c) {
    for (int s : {S_RHO, S_RHO_P})
        if (c->allocated[s]) c->stale[s] = true;
}

static int step_wcsph_fused_pre(sphmw_ctx *c) {
    // accelerate! + move!  (:311-312)
    TRY(need_slots(c, SL(S_TYPE, S_RHO_P, S_RHO, S_X0, S_V0, S_M, S_H), SL(S_V0, S_X0)));
    if (!c->dv_zero) {
        TRY(need_slots(c, SL(S_DV0), SL(S_DV0)));
        TRY(run_unary<U_wcsph_accelerate<true>>(c, "wcsph.accelerate"));
        c->dv_zero = true;
    } else {
        TRY(run_unary<U_wcsph_accelerate<false>>(c, "wcsph.accelerate"));
    }
    TRY(run_unary<U_wcsph_move>(c, "wcsph.move"));
    wcsph_after_drift(c);
    return SPHMW_OK;
}

// the two fused pair passes of the "wcsph" step (strict / FAST_MATH closures, optionally with
// the packed neighbour records)
static int run_fused_density(sphmw_ctx *c) {
    // owned columns + the first ghost column (its sums are complete thanks to the second)
    const bool rec = sphmw_use_records(c);
    const char *name = "wcsph.density_fused";
    if (tiles_enabled(c)) {
        const ColFilter cf = filter_for_depth(c, 1);
        if (c->flags & SPHMW_FLAG_FAST_MATH) return run_tiled<B_wcsph_density_fast>(c, name, 0, c->cur, cf);
        return run_tiled<B_wcsph_density_fused>(c, name, 0, c->cur, cf);
    }
    if (c->flags & SPHMW_FLAG_FAST_MATH)
        return rec ? run_binary<B_wcsph_density_fast, true>(c, name, 0, c->cur, 1)
                   : run_binary<B_wcsph_density_fast>(c, name, 0, c->cur, 1);
    return rec ? run_binary<B_wcsph_density_fused, true>(c, name, 0, c->cur, 1)
               : run_binary<B_wcsph_density_fused>(c, name, 0, c->cur, 1);
}
static int run_force_advance(sphmw_ctx *c, const char *name, const ColFilter &cf) {
    const bool rec = sphmw_use_records(c);
    if (c->flags & SPHMW_FLAG_FAST_MATH)
        return rec ? run_binary_cols<B_force_advance<B_wcsph_momentum_fast>, true>(c, name, 0, c->alt, cf)
                   : run_binary_cols<B_force_advance<B_wcsph_momentum_fast>>(c, name, 0, c->alt, cf);
    return rec ? run_binary_cols<B_force_advance<B_wcsph_momentum_fused>, true>(c, name, 0, c->alt, cf)
               : run_binary_cols<B_force_advance<B_wcsph_momentum_fused>>(c, name, 0, c->alt, cf);
}
static int run_fused_force(sphmw_ctx *c, const char *name, const ColFilter &cf, bool advance = false) {
    const bool rec = sphmw_use_records(c);
    if (advance && c->slab_lo < 0 && c->n > 0) {
        // + the next step's accelerate! and move! in finish() (B_force_advance); x and v go to alt.  The
        // thread that drifts a particle also writes the next cell list's key of it, and the removed list
        // of the next build starts here: that build then skips k_keys (cell_list.cu)
        CUDA_TRY(cudaMemsetAsync(c->removed, 0, sizeof(uint32_t) * 2, c->stream));
        c->prm.key_out = c->key;
        c->prm.cellx_out = c->cellx;
        c->prm.key_removed = c->removed;
        c->prm.key_idx = c->idx;
        c->prm.key_removed_cap = (uint32_t)c->removed_cap;
        const int rc = run_force_advance(c, name, cf);
        c->prm.key_out = c->prm.cellx_out = c->prm.key_removed = nullptr;
        c->prm.key_idx = nullptr;
        TRY(rc);
        c->keys_from_advance = true;
        return SPHMW_OK;
    }
    if (advance) return run_force_advance(c, name, cf);  // slab: ghosts and migrants join after the drift
    if (tiles_enabled(c)) {
        if (c->flags & SPHMW_FLAG_FAST_MATH) return run_tiled<B_wcsph_momentum_fast>(c, name, 0, c->alt, cf);
        return run_tiled<B_wcsph_momentum_fused>(c, name, 0, c->alt, cf);
    }
    if (c->flags & SPHMW_FLAG_FAST_MATH)
        return rec ? run_binary_cols<B_wcsph_momentum_fast, true>(c, name, 0, c->alt, cf)
                   : run_binary_cols<B_wcsph_momentum_fast>(c, name, 0, c->alt, cf);
    return rec ? run_binary_cols<B_wcsph_momentum_fused, true>(c, name, 0, c->alt, cf)
               : run_binary_cols<B_wcsph_momentum_fused>(c, name, 0, c->alt, cf);
}

// slab mode: the halo exchange sits between the two halves (after the drift, before the sort)
// advance: the force pass also opens the next step (accelerate! + move!, B_force_advance); the
// context is then in the state step_wcsph_fused_pre leaves behind
// the force pass of the fused step replays the pair list over the fluid work list (pair_list.cuh
// k_binary_list_fluid): the cell-list builds from now on make one
static void want_fluid_list(sphmw_ctx *c) {
    c->want_fluid_list = !(c->flags & (SPHMW_FLAG_NO_PAIR_LIST | SPHMW_FLAG_CELL_PAIRS | SPHMW_FLAG_TILES));
}

static int step_wcsph_fused_post(sphmw_ctx *c, bool advance = false) {
    wcsph_before_sort(c);
    want_fluid_list(c);
    TRY(sphmw_build_cell_list(c, nullptr));  // :313
    // :316-323
    for (int s : {S_RHO_BG, S_RHO_P, S_RHO, S_P_BG, S_P_P, S_P, S_PR2, S_CS}) {
        TRY(sphmw_ensure_slot(c, s));
        c->stale[s] = false;
    }
    // owned columns + the first ghost column (its sums are complete thanks to the second).
    // The density pass records the pair list, the force pass replays it.
    c->want_list = true;
    if (c->flags & SPHMW_FLAG_CELL_PAIRS)
        TRY((run_cell_pairs<CP_Density>(c, "wcsph.density_fused", c->cur, 1)));
    else
        TRY(run_fused_density(c));
    // :326-327 find_temperature!/find_pot_temp! are diagnostics: left stale, rebuilt on demand
    // :330-331 — owned columns only
    TRY(sphmw_ensure_slot(c, S_V0));
    if (c->flags & SPHMW_FLAG_CELL_PAIRS)
        TRY((run_cell_pairs<CP_Momentum>(c, "wcsph.momentum_fused", c->alt, 0)));
    else
        TRY(run_fused_force(c, "wcsph.momentum_fused", filter_for_depth(c, 0), advance));
    std::swap(c->cur.s[S_V0], c->alt.s[S_V0]);
    std::swap(c->cur.s[S_V1], c->alt.s[S_V1]);
    if (c->grid.dim == 3) std::swap(c->cur.s[S_V2], c->alt.s[S_V2]);
    if (advance) {
        std::swap(c->cur.s[S_X0], c->alt.s[S_X0]);
        std::swap(c->cur.s[S_X1], c->alt.s[S_X1]);
        if (c->grid.dim == 3) std::swap(c->cur.s[S_X2], c->alt.s[S_X2]);
        wcsph_after_drift(c);
    }
    return SPHMW_OK;
}

// hopkins_perturbed_witch.jl:324-349 / full_hopkins_perturbed_witch.jl:350-374 with the unary
// sweeps folded into the three pair passes (ops_menu.cuh): the density pass records the pair
// list, the pressure and force passes replay it.  On a slab context the pressure sum needs the NEW
// smoothing length of a particle's neighbours, i.e. complete density sums two cell columns beyond
// the owned ones: three ghost columns (SPHMW_FLAG_GHOST3), plain schedule.
template <class Force>
static int step_hopkins_fused_post(sphmw_ctx *c) {
    if (c->slab_lo >= 0 && c->grid.ghost < 3) {
        sphmw_set_error("the Hopkins schemes need three ghost columns on a slab context (SPHMW_FLAG_GHOST3)");
        return SPHMW_E_STATE;
    }
    TRY(sphmw_build_cell_list(c, nullptr));  // :329
    TRY(need_slots(c, SL(S_X0, S_V0, S_M, S_H, S_A, S_TYPE), SL()));
    TRY(need_slots(c, SL(S_DV0), SL()));     // all zero after accelerate!; the force operator starts from it
    for (int s : {S_RHO_BG, S_RHO_P, S_RHO, S_P_BG, S_P_P, S_P}) {
        TRY(sphmw_ensure_slot(c, s));
        c->stale[s] = false;
    }
    c->want_list = true;
    // slab contexts (three ghost columns): the density sums — and with them the new smoothing lengths —
    // are complete two columns beyond the owned ones, the pressure sums one column beyond, the force
    // is needed on the owned columns only
    TRY((run_binary<B_hopkins_density_fused>(c, "hopkins.density_fused", 0, c->cur, 2)));
    TRY((run_binary<B_hopkins_pressure_fused>(c, "hopkins.pressure_fused", 0, c->cur, 1)));
    TRY((run_binary<B_force_kick_fused<Force>>(c, "hopkins.momentum_fused", 0, c->alt, 0)));
    std::swap(c->cur.s[S_V0], c->alt.s[S_V0]);
    std::swap(c->cur.s[S_V1], c->alt.s[S_V1]);
    if (c->grid.dim == 3) std::swap(c->cur.s[S_V2], c->alt.s[S_V2]);
    return SPHMW_OK;
}
template <class Force>
static int step_hopkins_fused(sphmw_ctx *c) {
    TRY(step_wcsph_fused_pre(c));           // accelerate! + move! (:325-326)
    return step_hopkins_fused_post<Force>(c);
}

// one step of a whole-domain multi-step call.  opened: the previous step's force pass already ran
// this step's accelerate! + move!; advance: do the same for the next one
static int step_wcsph_fused(sphmw_ctx *c, bool opened = false, bool advance = false) {
    if (!opened) TRY(step_wcsph_fused_pre(c));
    return step_wcsph_fused_post(c, advance);
}

// ===========================================================================
// Overlapped slab step (SURVEY.md §8e "overlap"): the halo exchange of step n+1 travels while
// the interior columns of step n are still in the force pass.
//
//   phase 2   cell list, density pass, force + kick of the EDGE columns (the three outermost
//             owned columns of each side that has a neighbour), then the next step's
//             accelerate! + move! (wcsph_perturbed_witch.jl:311-312) for the edge columns,
//             written to the alt buffers because the interior force pass still reads the
//             old positions and velocities
//   (halo.cu) sphmw_halo_pack_begin packs the edge columns' records from the alt buffers
//   phase 3   force + kick of the interior columns, their accelerate! + move!, buffer swap
//   (halo.cu) sphmw_halo_pack_finish, transport, sphmw_halo_unpack
//
// accelerate!/move! are per-particle, so doing them column set by column set changes no bit.
// Records of the next exchange can only come from particles that sit in the edge columns
// before the drift as long as nothing moves a whole cell column per step (|v| dt < h;
// dt = 0.01 h/c in the drivers); the interior kernel counts violations and
// sphmw_halo_pack_finish fails loudly on them.
// ===========================================================================
static ColFilter cols_range(int a0, int a1, int b0, int b1, int sparse = 0) {
    ColFilter cf{1, a0, a1, b0, b1, 0, sparse};
    return cf;
}

SlabCols sphmw_slab_cols(const sphmw_ctx *c) {
    return sphmw_slab_cols_of((int)c->grid.lim[0], c->slab_lo > 0, c->slab_hi < c->global_cols);
}

// W: local columns including the GHOST_COLS ghost columns per side; hl/hr: a neighbour exists
SlabCols sphmw_slab_cols_of(int W, bool hl, bool hr) {
    const int G = GHOST_COLS;
    const int il = hl ? G + 3 : 0;                     // first interior column
    const int ir = hr ? W - G - 4 : W - 1;             // last interior column
    const int er = hr ? (ir + 1 > il ? ir + 1 : il) : W;  // first column of the right edge set
    SlabCols sc;
    sc.edge = cols_range(hl ? 0 : 1, hl ? il - 1 : 0, hr ? er : 1, hr ? W - 1 : 0, 1);
    sc.interior = cols_range(il, ir, 1, 0);
    sc.force_edge = cols_range(hl ? G : 1, hl ? il - 1 : 0, hr ? er : 1, hr ? W - G - 1 : 0, 1);
    sc.force_interior = cols_range(il > G ? il : G, ir < W - G - 1 ? ir : W - G - 1, 1, 0);
    return sc;
}

// next step's accelerate! + move! for the particles of the selected columns, out of place:
// `mix` has x and v in the alt buffers (v already holds the force pass's result) and every
// other field in the current ones.  Ghosts just carry their state over (they are dropped by
// the next pack).  check_escape: count particles that end up in a column whose records were
// already packed.
template <int DIM>
__device__ __forceinline__ void advance_particle(int64_t p, const Fields &cur, const Fields &mix, const Params &prm,
                                                 const Grid &g, const uint32_t *__restrict__ cellx,
                                                 const uint32_t *__restrict__ tag, const ColFilter &cf,
                                                 int check_escape, int has_left, int has_right,
                                                 uint32_t *__restrict__ counters) {
    if (!col_selected(cf, (int)cellx[p])) return;
    mix.s[S_X0][p] = cur.s[S_X0][p];
    mix.s[S_X1][p] = cur.s[S_X1][p];
    if (DIM == 3) mix.s[S_X2][p] = cur.s[S_X2][p];
    if (tag[p] != TAG_OWNED) {
        mix.s[S_V0][p] = cur.s[S_V0][p];
        mix.s[S_V1][p] = cur.s[S_V1][p];
        if (DIM == 3) mix.s[S_V2][p] = cur.s[S_V2][p];
        return;
    }
    U_wcsph_accelerate<false>::apply<DIM>(mix, prm, p);
    U_wcsph_move::apply<DIM>(mix, prm, p);
    if (check_escape) {
        const long long W = g.lim[0];
        const long long i = (long long)floor(mix.s[S_X0][p] / g.h) - g.phase[0];
        if ((has_left && i < 2 * GHOST_COLS) || (has_right && i >= W - 2 * GHOST_COLS))
            atomicAdd(&counters[5], 1u);
    }
}
template <int DIM>
__global__ void __launch_bounds__(256)
k_advance_cols(Fields cur, Fields mix, Params prm, Grid g, const uint32_t *__restrict__ cellx,
               const uint32_t *__restrict__ tag, int64_t n, ColFilter cf, int check_escape, int has_left,
               int has_right, uint32_t *__restrict__ counters) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    advance_particle<DIM>(p, cur, mix, prm, g, cellx, tag, cf, check_escape, has_left, has_right, counters);
}
// the same over the particle ranges of a few columns (zrun cell order; pair_list.cuh col_ranges)
template <int DIM>
__global__ void __launch_bounds__(256)
k_advance_cols_ranges(Fields cur, Fields mix, Params prm, Grid g, const uint32_t *__restrict__ cellx,
                      const uint32_t *__restrict__ tag, const uint32_t *__restrict__ cell_start, int64_t n,
                      ColFilter cf, int check_escape, int has_left, int has_right, uint32_t *__restrict__ counters) {
    const ColRanges r = col_ranges(g, cf, cell_start);
    const uint32_t total = r.n0 + r.n1;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const int64_t p = t < r.n0 ? (int64_t)r.b0 + t : (int64_t)r.b1 + (t - r.n0);
        if (p < n) advance_particle<DIM>(p, cur, mix, prm, g, cellx, tag, cf, check_escape, has_left, has_right, counters);
    }
}

static Fields mixed_view(sphmw_ctx *c) {
    Fields m = c->cur;
    for (int s : {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2}) m.s[s] = c->alt.s[s];
    return m;
}

static int run_advance_cols(sphmw_ctx *c, const char *name, const ColFilter &cf, int check_escape) {
    if (c->n == 0) return SPHMW_OK;
    const int hl = c->slab_lo > 0, hr = c->slab_hi < c->global_cols;
    TIMED(c, name);
    if (cf.sparse && c->grid.zrun && !getenv("SPHMW_NO_COLUMN_RANGES")) {
        const unsigned gb = std::min<unsigned>(grid_for(c->n, 256), (unsigned)c->sm_count * 4u);
        if (c->grid.dim == 2)
            k_advance_cols_ranges<2><<<gb, 256, 0, c->stream>>>(c->cur, mixed_view(c), c->prm, c->grid, c->cellx, c->tag,
                                                                c->cell_start, c->n, cf, check_escape, hl, hr, c->halo_counters);
        else
            k_advance_cols_ranges<3><<<gb, 256, 0, c->stream>>>(c->cur, mixed_view(c), c->prm, c->grid, c->cellx, c->tag,
                                                                c->cell_start, c->n, cf, check_escape, hl, hr, c->halo_counters);
        CUDA_TRY(cudaGetLastError());
        return SPHMW_OK;
    }
    if (c->grid.dim == 2)
        k_advance_cols<2><<<grid_for(c->n, 256), 256, 0, c->stream>>>(
            c->cur, mixed_view(c), c->prm, c->grid, c->cellx, c->tag, c->n, cf, check_escape, hl, hr, c->halo_counters);
    else
        k_advance_cols<3><<<grid_for(c->n, 256), 256, 0, c->stream>>>(
            c->cur, mixed_view(c), c->prm, c->grid, c->cellx, c->tag, c->n, cf, check_escape, hl, hr, c->halo_counters);
    CUDA_TRY(cudaGetLastError());
    return SPHMW_OK;
}

static int step_wcsph_overlap_a(sphmw_ctx *c) {
    if (c->slab_lo < 0 || (c->flags & SPHMW_FLAG_CELL_PAIRS)) {
        sphmw_set_error("step_phase 2/3: the overlapped step runs on slab contexts without CELL_PAIRS");
        return SPHMW_E_STATE;
    }
    if (c->grid.ghost != GHOST_COLS) { sphmw_set_error("step_phase 2/3: the overlapped step is laid out for two ghost columns"); return SPHMW_E_STATE; }
    if (c->overlap_stage != 0) { sphmw_set_error("step_phase 2: an overlapped step is already in flight"); return SPHMW_E_STATE; }
    if (!c->dv_zero) { sphmw_set_error("step_phase 2: Dv must be zero (run step_phase 0 first)"); return SPHMW_E_STATE; }
    wcsph_before_sort(c);
    want_fluid_list(c);
    TRY(sphmw_build_cell_list(c, nullptr));
    for (int s : {S_RHO_BG, S_RHO_P, S_RHO, S_P_BG, S_P_P, S_P, S_PR2, S_CS}) {
        TRY(sphmw_ensure_slot(c, s));
        c->stale[s] = false;
    }
    c->want_list = true;
    TRY(run_fused_density(c));
    TRY(sphmw_ensure_slot(c, S_V0));
    const SlabCols sc = sphmw_slab_cols(c);
    TRY(run_fused_force(c, "wcsph.momentum_fused_edge", sc.force_edge));
    TRY(run_advance_cols(c, "wcsph.advance_edge", sc.edge, 0));
    c->overlap_stage = 1;
    return SPHMW_OK;
}

static int step_wcsph_overlap_b(sphmw_ctx *c) {
    if (c->overlap_stage != 2) {
        sphmw_set_error("step_phase 3: call step_phase 2 and halo_pack_begin first");
        return SPHMW_E_STATE;
    }
    const SlabCols sc = sphmw_slab_cols(c);
    const bool fold = !(c->flags & SPHMW_FLAG_TILES) && !getenv("SPHMW_NO_FUSED_ADVANCE");
    if (fold) {
        // the interior force pass also runs the next step's accelerate! + move! (B_force_advance)
        // and counts particles that drift into a column whose records were already packed; the
        // interior columns outside the force set (ghost columns of a rank on the global boundary:
        // empty, or nearly) get the plain advance kernel over their particle ranges
        const int W = (int)c->grid.lim[0], G = GHOST_COLS;
        c->prm.esc_counter = c->halo_counters + 5;
        c->prm.esc_h = c->grid.h;
        c->prm.esc_phase = c->grid.phase[0];
        c->prm.esc_lo = c->slab_lo > 0 ? 2 * G : INT_MIN;
        c->prm.esc_hi = c->slab_hi < c->global_cols ? W - 2 * G : INT_MAX;
        const int rc = run_fused_force(c, "wcsph.momentum_fused", sc.force_interior, true);
        c->prm.esc_counter = nullptr;
        TRY(rc);
        ColFilter rest = cols_range(sc.interior.a0, sc.force_interior.a0 - 1, sc.force_interior.a1 + 1, sc.interior.a1, 1);
        if (rest.a0 <= rest.a1 || rest.b0 <= rest.b1) TRY(run_advance_cols(c, "wcsph.advance_interior", rest, 1));
    } else {
        TRY(run_fused_force(c, "wcsph.momentum_fused", sc.force_interior));
        TRY(run_advance_cols(c, "wcsph.advance_interior", sc.interior, 1));
    }
    for (int s : {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2})
        if ((s != S_X2 && s != S_V2) || c->grid.dim == 3) std::swap(c->cur.s[s], c->alt.s[s]);
    // as after step_wcsph_fused_pre: positions changed, per-step derived fields are stale
    for (int s = S_DV0; s <= S_DV2; ++s)
        if (c->allocated[s]) c->stale[s] = true;
    c->cell_list_valid = false;
    for (int s : {S_RHO_BG, S_P_BG, S_P_P, S_P, S_T_P, S_T, S_TH_BG, S_TH_P, S_TH, S_PR2, S_CS})
        if (c->allocated[s]) c->stale[s] = true;
    c->overlap_stage = 3;
    return SPHMW_OK;
}

// hopkins_total_witch.jl:283-308 on a slab context: compute_pressure! reads the neighbours' NEW smoothing
// length, as in the other Hopkins drivers, so the context needs three ghost columns.  The base halo
// record with A in row 8 carries everything: rho, P, T and theta are recomputed for every particle type
// before they are read (U_ht_reset_density, U_ht_reset_pressure/finalize_pressure, U_ht_find_temperature,
// U_ht_find_pot_temp are not type-gated), and Dv is zero after accelerate!.  Walls move and feel gravity in
// this driver (SURVEY quirk 10): one that leaves the global box is dropped and counted as on any walled
// configuration, or renumbered like the reference with the open box (slab_comm.cu).
static int step_hopkins_total_phase(sphmw_ctx *c, int phase) {
    if (c->slab_lo >= 0 && c->grid.ghost < 3) {
        sphmw_set_error("the Hopkins schemes need three ghost columns on a slab context (SPHMW_FLAG_GHOST3)");
        return SPHMW_E_STATE;
    }
    if (phase == 0) return apply_seq(c, {"hopkins_total.accelerate", "hopkins_total.move"});
    if (phase == 1)
        return apply_seq(c, {"create_cell_list", "hopkins_total.reset_density", "wcsph.compute_density",
                             "wcsph.update_smoothing", "hopkins_total.reset_pressure", "hopkins.compute_pressure",
                             "hopkins_total.finalize_pressure", "hopkins_total.find_temperature",
                             "hopkins_total.find_pot_temp", "hopkins_total.balance_of_momentum",
                             "hopkins_total.accelerate"});
    sphmw_set_error("step_phase: the Hopkins schemes run the plain schedule (phases 0 and 1)");
    return SPHMW_E_INVALID;
}

// adiabatic_flow_witch.jl:231-243 on a slab context driven by the caller's transport.  add_new_particles!
// numbers the successors across ranks, which only the library transport can do (sphmw_comm_open_box):
// phase 0 refuses a step in which an owned INFLOW particle would convert instead of skipping it.
static int step_aflow_phase(sphmw_ctx *c, int phase) {
    if (c->slab_lo < 0) {
        sphmw_set_error("step_phase 'aflow': slab contexts only (a whole-domain context steps with sphmw_step)");
        return SPHMW_E_STATE;
    }
    if (phase == 0) {
        TRY(apply_seq(c, {"flow.accelerate", "aflow.move"}));
        TRY(need_slots(c, SL(S_X0, S_TYPE), SL()));
        uint32_t *count = c->rank;  // scratch of the cell-list build, free between builds
        CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(uint32_t), c->stream));
        if (c->n > 0) {
            TIMED(c, "flow.flag_inflow");
            if (c->grid.dim == 2) k_flow_collect<2><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, c->tag, c->n, count, nullptr, 0);
            else k_flow_collect<3><<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->cur, c->prm, c->idx, c->tag, c->n, count, nullptr, 0);
            CUDA_TRY(cudaGetLastError());
        }
        uint32_t converting = 0;
        CUDA_TRY(cudaMemcpyAsync(&converting, count, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        if (converting) {
            sphmw_set_error("step_phase 'aflow': %u INFLOW particle(s) of this rank convert in this step; their successors "
                            "are numbered across ranks, which needs the library transport with the open box "
                            "(sphmw_comm_init, sphmw_comm_open_box, sphmw_step)", converting);
            return SPHMW_E_STATE;
        }
        return SPHMW_OK;
    }
    if (phase == 1) {
        TRY(sphmw_build_cell_list(c, nullptr));
        return apply_seq(c, {"+aflow.find_density", "aflow.find_s", "aflow.find_pressure", "aflow.entropy_production",
                             "flow.internal_force", "flow.accelerate"});
    }
    sphmw_set_error("step_phase: the 'aflow' scheme runs the plain schedule (phases 0 and 1)");
    return SPHMW_E_INVALID;
}

int sphmw_step_scheme_phase(sphmw_ctx *c, const char *scheme, int phase) {
    if (!strcmp(scheme, "hopkins_total")) return step_hopkins_total_phase(c, phase);
    if (!strcmp(scheme, "aflow")) return step_aflow_phase(c, phase);
    if (!strcmp(scheme, "hopkins") || !strcmp(scheme, "hopkins_full")) {
        // plain schedule only: kick + drift | (the caller's halo exchange) | sort + three pair passes
        if (phase == 0) return step_wcsph_fused_pre(c);
        if (phase == 1)
            return !strcmp(scheme, "hopkins") ? step_hopkins_fused_post<B_wcsph_momentum>(c)
                                              : step_hopkins_fused_post<B_hf_momentum>(c);
        sphmw_set_error("step_phase: the Hopkins schemes run the plain schedule (phases 0 and 1)");
        return SPHMW_E_INVALID;
    }
    if (strcmp(scheme, "wcsph")) {
        sphmw_set_error("step_phase: only the 'wcsph', 'hopkins', 'hopkins_full', 'hopkins_total' and 'aflow' schemes "
                        "run on slabs");
        return SPHMW_E_UNSUPPORTED_OP;
    }
    switch (phase) {
        case 0: return step_wcsph_fused_pre(c);
        case 1: return step_wcsph_fused_post(c);
        case 2: return step_wcsph_overlap_a(c);
        case 3: return step_wcsph_overlap_b(c);
    }
    sphmw_set_error("step_phase: phase must be 0..3");
    return SPHMW_E_INVALID;
}

int sphmw_step_wcsph_phase(sphmw_ctx *c, int phase) { return sphmw_step_scheme_phase(c, "wcsph", phase); }

int sphmw_step_scheme(sphmw_ctx *c, const char *scheme, int nsteps) {
    c->keys_from_advance = false;  // only a step of this call may hand keys to the next build
    if (c->slab_lo >= 0 && nsteps > 0) {
        // with a communicator (sphmw_comm_init) the halo exchange is the library's business
        if (c->comm) return sphmw_comm_step(c, scheme, nsteps);
        sphmw_set_error("step: a slab context without a communicator (sphmw_comm_init) is stepped with "
                        "step_phase around the caller's halo exchange");
        return SPHMW_E_STATE;
    }
    // the fused step folds the next step's accelerate! + move! into its force pass (all steps of a
    // call but the last); not with the shared-memory variants, whose kernels have no such finish()
    const bool fold = !(c->flags & (SPHMW_FLAG_CELL_PAIRS | SPHMW_FLAG_TILES)) && !getenv("SPHMW_NO_FUSED_ADVANCE");
    bool opened = false;
    for (int k = 0; k < nsteps; ++k) {
        if (!strcmp(scheme, "wcsph")) {
            const bool advance = fold && k + 1 < nsteps;
            TRY(step_wcsph_fused(c, opened, advance));
            opened = advance;
        } else if (!strcmp(scheme, "wcsph_unfused")) {
            // the literal operator sequence of wcsph_perturbed_witch.jl:309-332
            TRY(apply_seq(c, {"wcsph.accelerate", "wcsph.move", "create_cell_list",
                              "wcsph.reset_density", "wcsph.compute_density",
                              "wcsph.finalize_density", "wcsph.update_smoothing",
                              "create_cell_list", "wcsph.compute_pressure",
                              "wcsph.find_temperature", "wcsph.find_pot_temp",
                              "wcsph.balance_of_momentum", "wcsph.accelerate"}));
        } else if (!strcmp(scheme, "hopkins") && c->slab_lo < 0 && !getenv("SPHMW_HOPKINS_UNFUSED")) {
            TRY(step_hopkins_fused<B_wcsph_momentum>(c));
        } else if (!strcmp(scheme, "hopkins_full") && c->slab_lo < 0 && !getenv("SPHMW_HOPKINS_UNFUSED")) {
            TRY(step_hopkins_fused<B_hf_momentum>(c));
        } else if (!strcmp(scheme, "hopkins") || !strcmp(scheme, "hopkins_unfused")) {
            // hopkins_perturbed_witch.jl:325-349
            TRY(apply_seq(c, {"wcsph.accelerate", "wcsph.move", "create_cell_list",
                              "wcsph.reset_density", "wcsph.compute_density",
                              "wcsph.finalize_density", "wcsph.update_smoothing",
                              "hopkins.reset_pressure", "hopkins.compute_pressure",
                              "hopkins.finalize_pressure", "wcsph.find_temperature",
                              "wcsph.find_pot_temp", "wcsph.balance_of_momentum",
                              "wcsph.accelerate"}));
        } else if (!strcmp(scheme, "hopkins_full") || !strcmp(scheme, "hopkins_full_unfused")) {
            // full_hopkins_perturbed_witch.jl:350-374
            TRY(apply_seq(c, {"wcsph.accelerate", "wcsph.move", "create_cell_list",
                              "wcsph.reset_density", "wcsph.compute_density",
                              "wcsph.finalize_density", "wcsph.update_smoothing",
                              "hopkins.reset_pressure", "hopkins.compute_pressure",
                              "hopkins.finalize_pressure", "wcsph.find_temperature",
                              "wcsph.find_pot_temp", "hopkins_full.balance_of_momentum",
                              "wcsph.accelerate"}));
        } else if (!strcmp(scheme, "hopkins_total")) {
            // hopkins_total_witch.jl:283-308
            TRY(apply_seq(c, {"hopkins_total.accelerate", "hopkins_total.move", "create_cell_list",
                              "hopkins_total.reset_density", "wcsph.compute_density",
                              "wcsph.update_smoothing", "hopkins_total.reset_pressure",
                              "hopkins.compute_pressure", "hopkins_total.finalize_pressure",
                              "hopkins_total.find_temperature", "hopkins_total.find_pot_temp",
                              "hopkins_total.balance_of_momentum", "hopkins_total.accelerate"}));
        } else if (!strcmp(scheme, "dambreak")) {
            // collapse_dry.jl:203-211
            TRY(apply_seq(c, {"dambreak.accelerate", "dambreak.move", "create_cell_list",
                              "dambreak.balance_of_mass", "dambreak.find_pressure", "dambreak.move",
                              "create_cell_list", "dambreak.internal_force", "dambreak.accelerate"}));
        } else if (!strcmp(scheme, "flow")) {
            // isothermal_flow_witch.jl:221-232
            TRY(apply_seq(c, {"flow.accelerate", "flow.move"}));
            TRY(sphmw_flow_add_particles(c, nullptr, false));
            TRY(apply_seq(c, {"create_cell_list", "flow.balance_of_mass", "flow.find_pressure",
                              "flow.find_pot_temp", "flow.internal_force", "flow.accelerate"}));
        } else if (!strcmp(scheme, "aflow")) {
            // adiabatic_flow_witch.jl:231-243
            TRY(apply_seq(c, {"flow.accelerate", "aflow.move"}));
            TRY(sphmw_flow_add_particles(c, nullptr, true));
            TRY(apply_seq(c, {"create_cell_list", "+aflow.find_density", "aflow.find_s", "aflow.find_pressure",
                              "aflow.entropy_production", "flow.internal_force", "flow.accelerate"}));
        } else if (!strcmp(scheme, "collision")) {
            // test_collision_2d.jl:106-116
            TRY(apply_seq(c, {"collision.accelerate", "collision.move", "create_cell_list",
                              "collision.reset_rho", "+collision.find_rho",
                              "collision.find_pressure", "collision.reset_a",
                              "collision.internal_force", "collision.accelerate"}));
        } else {
            sphmw_set_error("unknown scheme '%s'", scheme);
            return SPHMW_E_UNSUPPORTED_OP;
        }
    }
    return SPHMW_OK;
}
