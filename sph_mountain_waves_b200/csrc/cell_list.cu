// Cell-list construction on the device — replaces create_cell_list! (src/core.jl:51-90),
// Cell/add_index! (src/structs.jl:22-31, src/core.jl:13-41), find_key
// (src/structs.jl:97-106) and is_inside(::Box) (src/geometry.jl:24-30).
//
// Layout: particles are kept PHYSICALLY sorted by (cell key ascending, reference
// particle index descending) — the order in which the reference's cells store
// their entries (core.jl:32-37) — with a cell-start table, so a cell is the
// contiguous run [cell_start[k], cell_start[k+1]).  The sort is a one-digit
// most-significant-digit radix (counting) pass on the cell key (histogram with
// warp-aggregated ranks, exclusive scan, scatter), followed by an in-cell
// ordering by reference index that makes the result independent of the atomics'
// arrival order (deterministic, like the reference's sorted insertion under a lock).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <unordered_map>
#include <vector>

#include "cell_gather.cuh"
#include "sphmw_internal.h"

// ---------------------------------------------------------------------------
// keys + out-of-box detection
// ---------------------------------------------------------------------------
// SLAB: ghosts of the previous exchange and particles that left the local columns are
// dropped (tag == TAG_DEAD or column out of range); they are only counted, with one atomic
// per warp, because a slab drops two ghost sheets per side every step.
template <int DIM, bool SLAB>
__global__ void k_keys(const double *__restrict__ x0, const double *__restrict__ x1,
                       const double *__restrict__ x2, int64_t n, Grid g,
                       uint32_t *__restrict__ key, uint32_t *__restrict__ removed,
                       uint32_t removed_cap, const uint32_t *__restrict__ idx,
                       const uint32_t *__restrict__ tag, uint32_t *__restrict__ cellx) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (SLAB) {
        bool live = pos < n;
        bool dead = false;
        uint32_t k = 0, ci = 0;
        if (live) {
            double x = x0[pos], y = x1[pos], z = DIM == 3 ? x2[pos] : 0.0;
            bool inside = tag[pos] != TAG_DEAD && g.box[0] <= x && x <= g.box[3] && g.box[1] <= y &&
                          y <= g.box[4] && g.box[2] <= z && z <= g.box[5];
            if (inside) {
                long long i = (long long)floor(x / g.h) - g.phase[0];
                long long j = (long long)floor(y / g.h) - g.phase[1];
                long long kk = DIM == 3 ? (long long)floor(z / g.h) - g.phase[2] : 0;
                if (i < 0 || i >= g.lim[0]) inside = false;
                else {
                    k = pkey_ijk(g, (int)i, (int)j, (int)kk);
                    ci = (uint32_t)i;
                }
            }
            if (!inside) {
                k = (uint32_t)g.pkey_max;
                dead = true;
            }
            key[pos] = k;
            cellx[pos] = ci;
        }
        // removed[0]: dropped particles; removed[1]: the owned particles that stay — the rank's
        // share of the global count.  Counted per block (one pair of atomics per 256 particles:
        // per-warp atomics on two fixed addresses made this kernel 5x slower per particle)
        const int nd = __syncthreads_count(dead);
        const int no = __syncthreads_count(live && !dead && tag[pos] == TAG_OWNED);
        if (threadIdx.x == 0) {
            if (nd) atomicAdd(&removed[0], (uint32_t)nd);
            if (no) atomicAdd(&removed[1], (uint32_t)no);
        }
        return;
    }
    if (pos >= n) return;
    cell_key_whole<DIM>(g, x0[pos], x1[pos], DIM == 3 ? x2[pos] : 0.0, pos, key, cellx, removed, removed_cap, idx);
}

// ---------------------------------------------------------------------------
// histogram with warp-aggregated arrival ranks
// ---------------------------------------------------------------------------
__global__ void k_histogram(const uint32_t *__restrict__ key, int64_t n,
                            uint32_t *__restrict__ count, uint32_t *__restrict__ rank) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    bool live = pos < n;
    uint32_t k = live ? key[pos] : 0xFFFFFFFFu;
    unsigned lane = threadIdx.x & 31;
    unsigned peers = __match_any_sync(0xffffffffu, k);
    int leader = __ffs(peers) - 1;
    unsigned before = __popc(peers & ((1u << lane) - 1u));
    uint32_t base = 0;
    if (live && (int)lane == leader) base = atomicAdd(&count[k], (uint32_t)__popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (live) rank[pos] = base + before;
}

// ---------------------------------------------------------------------------
// exclusive scan (block scan + recursive block-sum scan)
// ---------------------------------------------------------------------------
#define SCAN_THREADS 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_tile(uint32_t *__restrict__ data, int64_t n, uint32_t *__restrict__ tile_sums) {
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    int64_t base = blockIdx.x * (int64_t)SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t sum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? data[base + i] : 0u;
        sum += v[i];
    }
    unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) warp_sums[w] = incl;
    __syncthreads();
    if (w == 0) {
        uint32_t ws = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0u;
        uint32_t wi = ws;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= (unsigned)o) wi += t;
        }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = wi - ws;  // exclusive
        if (lane == SCAN_THREADS / 32 - 1 && tile_sums) tile_sums[blockIdx.x] = wi;
    }
    __syncthreads();
    uint32_t run = warp_sums[w] + (incl - sum);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) data[base + i] = run;
        run += v[i];
    }
}

__global__ void k_scan_add(uint32_t *__restrict__ data, int64_t n,
                           const uint32_t *__restrict__ tile_offsets) {
    int64_t i = blockIdx.x * (int64_t)SCAN_TILE + threadIdx.x;
    uint32_t off = tile_offsets[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        int64_t j = i + (int64_t)k * SCAN_THREADS;
        if (j < n) data[j] += off;
    }
}

static int exclusive_scan(sphmw_ctx *c, uint32_t *data, int64_t n, uint32_t *tmp, int64_t tmp_len) {
    int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (tiles <= 1) {
        TIMED(c, "cell_scan");
        k_scan_tile<<<1, SCAN_THREADS, 0, c->stream>>>(data, n, nullptr);
        return SPHMW_OK;
    }
    if (tiles > tmp_len) {
        sphmw_set_error("scan scratch too small");
        return SPHMW_E_STATE;
    }
    {
        TIMED(c, "cell_scan");
        k_scan_tile<<<(unsigned)tiles, SCAN_THREADS, 0, c->stream>>>(data, n, tmp);
    }
    TRY(exclusive_scan(c, tmp, tiles, tmp + tiles, tmp_len - tiles));
    {
        TIMED(c, "cell_scan");
        k_scan_add<<<(unsigned)tiles, SCAN_THREADS, 0, c->stream>>>(data, n, tmp);
    }
    return SPHMW_OK;
}

int sphmw_exclusive_scan_u32(sphmw_ctx *c, uint32_t *data, int64_t n) {
    int64_t need = n / SCAN_TILE * 2 + 4096;
    if (!c->scan_tmp || c->scan_tmp_len < need) {
        cudaFree(c->scan_tmp);
        c->scan_tmp = nullptr;
        c->scan_tmp_len = std::max<int64_t>(need, (c->grid.pkey_max + 2) / SCAN_TILE * 2 + 4096);
        CUDA_TRY(cudaMalloc(&c->scan_tmp, sizeof(uint32_t) * c->scan_tmp_len));
    }
    return exclusive_scan(c, data, n, c->scan_tmp, c->scan_tmp_len);
}

// ---------------------------------------------------------------------------
// fluid work list (pair_list.cuh k_binary_list_fluid): a stable compaction of the gather's fluid
// flags — per-tile counts, an exclusive scan of them, then every position to its slot: a fluid one
// after the fluid positions before it, any other after all fluid ones and the others before it
// ---------------------------------------------------------------------------
#define FL_ITEMS 8
#define FL_TILE (256 * FL_ITEMS)

__device__ __forceinline__ unsigned fl_load(const uint8_t *__restrict__ fl, int64_t base, int64_t n, uint8_t v[FL_ITEMS]) {
    unsigned cnt = 0;
    if (base + FL_ITEMS <= n) {
        const uint2 w = *(const uint2 *)(fl + base);  // base is a multiple of 8
#pragma unroll
        for (int i = 0; i < FL_ITEMS; ++i) v[i] = (uint8_t)((i < 4 ? w.x >> (8 * i) : w.y >> (8 * (i - 4))) & 1u);
    } else {
#pragma unroll
        for (int i = 0; i < FL_ITEMS; ++i) v[i] = base + i < n ? fl[base + i] : 0;
    }
#pragma unroll
    for (int i = 0; i < FL_ITEMS; ++i) cnt += v[i];
    return cnt;
}

__global__ void __launch_bounds__(256) k_fluid_count(const uint8_t *__restrict__ fl, int64_t n, uint32_t *__restrict__ tiles) {
    __shared__ unsigned ws[8];
    uint8_t v[FL_ITEMS];
    unsigned cnt = fl_load(fl, blockIdx.x * (int64_t)FL_TILE + threadIdx.x * FL_ITEMS, n, v);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int w = 0; w < 8; ++w) t += ws[w];
        tiles[blockIdx.x] = t;
    }
}

// the tile's positions are ordered in shared memory (fluid ones first) and written out as two
// contiguous runs: a thread writing its own eight slots would scatter each warp store over 32 sectors
__global__ void __launch_bounds__(256) k_fluid_scatter(const uint8_t *__restrict__ fl, int64_t n,
                                                       const uint32_t *__restrict__ tiles, int64_t ntiles,
                                                       uint32_t *__restrict__ work) {
    __shared__ unsigned ws[8];
    __shared__ uint32_t stage[FL_TILE];
    const int64_t tile0 = blockIdx.x * (int64_t)FL_TILE;
    const unsigned first = threadIdx.x * FL_ITEMS;
    uint8_t v[FL_ITEMS];
    const unsigned cnt = fl_load(fl, tile0 + first, n, v);
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) ws[w] = incl;
    __syncthreads();
    unsigned fb = incl - cnt, ftile = 0;  // fluid positions of the tile before `first`, and in all
    for (unsigned k = 0; k < 8; ++k) {
        if (k < w) fb += ws[k];
        ftile += ws[k];
    }
    const unsigned len = (unsigned)(n - tile0 < FL_TILE ? n - tile0 : FL_TILE);
#pragma unroll
    for (int i = 0; i < FL_ITEMS; ++i) {
        const unsigned l = first + i;
        if (l >= len) break;
        if (v[i]) stage[fb++] = (uint32_t)(tile0 + l);
        else stage[ftile + l - fb] = (uint32_t)(tile0 + l);
    }
    __syncthreads();
    const uint32_t fbase = tiles[blockIdx.x];  // fluid positions before the tile
    const uint32_t obase = tiles[ntiles] + (uint32_t)tile0 - fbase;  // all fluid ones + the others before it
    for (unsigned l = threadIdx.x; l < len; l += 256)
        work[l < ftile ? fbase + l : obase + (l - ftile)] = stage[l];
}

static int build_fluid_list(sphmw_ctx *c, int64_t n) {
    const int64_t ntiles = (n + FL_TILE - 1) / FL_TILE;
    if (ntiles + 1 > c->fluid_tiles_cap) {
        cudaFree(c->fluid_tiles);
        c->fluid_tiles = nullptr;
        c->fluid_tiles_cap = (c->cap + FL_TILE - 1) / FL_TILE + 1;
        CUDA_TRY(cudaMalloc(&c->fluid_tiles, sizeof(uint32_t) * c->fluid_tiles_cap));
    }
    {
        TIMED(c, "fluid_list");
        k_fluid_count<<<(unsigned)ntiles, 256, 0, c->stream>>>(c->fluid_flag, n, c->fluid_tiles);
    }
    CUDA_TRY(cudaMemsetAsync(c->fluid_tiles + ntiles, 0, sizeof(uint32_t), c->stream));
    TRY(sphmw_exclusive_scan_u32(c, c->fluid_tiles, ntiles + 1));
    {
        TIMED(c, "fluid_list");
        k_fluid_scatter<<<(unsigned)ntiles, 256, 0, c->stream>>>(c->fluid_flag, n, c->fluid_tiles, ntiles, c->fluid_work);
    }
    CUDA_TRY(cudaGetLastError());
    c->fluid_count = c->fluid_tiles + ntiles;
    c->fluid_gen = c->cell_gen;
    c->fluid_value = c->prm.fluid;
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// scatter, in-cell ordering, gather
// ---------------------------------------------------------------------------
__global__ void k_scatter(const uint32_t *__restrict__ key, const uint32_t *__restrict__ rank,
                          const uint32_t *__restrict__ cell_start, int64_t n,
                          uint32_t *__restrict__ src) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos >= n) return;
    src[cell_start[key[pos]] + rank[pos]] = (uint32_t)pos;
}

// One thread per cell: order the run by reference index DESCENDING (core.jl:32-37).
// Arrival order is already nearly sorted (particles keep their previous order),
// so the insertion sort is O(run) in the common case.
__global__ void k_cell_order(const uint32_t *__restrict__ cell_start, int64_t ncells,
                             uint32_t *__restrict__ src, const uint32_t *__restrict__ idx) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= ncells) return;
    uint32_t b = cell_start[c], e = cell_start[c + 1];
    for (uint32_t i = b + 1; i < e; ++i) {
        uint32_t s = src[i];
        uint32_t id = idx[s];
        uint32_t j = i;
        while (j > b) {
            uint32_t sp = src[j - 1];
            if (idx[sp] >= id) break;
            src[j] = sp;
            --j;
        }
        src[j] = s;
    }
}

__global__ void k_renumber(uint32_t *__restrict__ idx, const uint32_t *__restrict__ pos_of_idx,
                           const uint32_t *__restrict__ mv_old, const uint32_t *__restrict__ mv_new,
                           int64_t m) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < m) idx[pos_of_idx[mv_old[t]]] = mv_new[t];
}

// reference index -> physical position.  Only the removal renumbering, the inflow spawn and the pair
// dump need it, so the cell-list build no longer writes it (a scattered 4-byte store per particle
// per step): it is rebuilt from idx on demand.
__global__ void k_inverse_map(const uint32_t *__restrict__ idx, uint32_t *__restrict__ pos_of_idx, int64_t n) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p < n) pos_of_idx[idx[p]] = (uint32_t)p;
}
int sphmw_ensure_pos_of_idx(sphmw_ctx *c) {
    if (!c->pos_of_idx || c->pos_valid || c->n == 0) return SPHMW_OK;
    TIMED(c, "inverse_map");
    k_inverse_map<<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->idx, c->pos_of_idx, c->n);
    CUDA_TRY(cudaGetLastError());
    c->pos_valid = true;
    return SPHMW_OK;
}

// core.jl:72-81 on index space.  `removed` holds the reference indices (0-based)
// of the particles outside the box.  The serial loop
//     particles[removal[i]] = particles[end+1-i]   (removal sorted DESCENDING)
// touches O(k) slots; we replay it on the host over a sparse map and return
// the (old index -> new index) moves of the surviving particles.
void sphmw_replay_swap_removal(int64_t N, std::vector<uint32_t> &removed,
                               std::vector<uint32_t> &mv_old, std::vector<uint32_t> &mv_new) {
    std::sort(removed.begin(), removed.end(), [](uint32_t a, uint32_t b) { return a > b; });
    std::unordered_map<uint32_t, uint32_t> occ;  // slot -> current occupant (original index)
    occ.reserve(removed.size() * 2);
    const int64_t k = (int64_t)removed.size();
    for (int64_t i = 1; i <= k; ++i) {
        uint32_t dst = removed[i - 1];
        uint32_t srcslot = (uint32_t)(N - i);
        auto it = occ.find(srcslot);
        uint32_t o = it == occ.end() ? srcslot : it->second;
        occ[dst] = o;
    }
    const int64_t Nn = N - k;
    for (auto &kv : occ)
        if ((int64_t)kv.first < Nn && kv.first != kv.second) {
            mv_old.push_back(kv.second);
            mv_new.push_back(kv.first);
        }
}

int sphmw_build_cell_list(sphmw_ctx *c, int64_t *n_alive) {
    const Grid &g = c->grid;
    const int64_t n = c->n;
    const int64_t ncells = g.pkey_max;  // + 1 dead bucket
    // a new generation: the pair list of the previous one is void; record a new one if the
    // previous cell list was used by two or more binary passes
    c->cell_gen += 1;
    c->want_list = c->passes_this_gen >= 2;
    c->passes_this_gen = 0;
    // The recording pass's queue (pair_list.cuh) is sized for the survivors particles really have, and a
    // particle with more walks the cells in BOTH pair passes — a cliff (64 M particles: 38.6 -> 45.5 ms
    // with 14 % such particles).  The overflow counter of the previous list (published to pinned memory
    // one build ago, so no wait) tells when the rows are too few: then they grow, up to the list stride.
    if (c->pl.list && c->h_counters) {
        const unsigned long long seen = c->h_counters[2];
        if (seen > c->pl_overflow_seen + (unsigned long long)(n >> 10) && c->pl.qrows < c->pl.stride + NL_QUEUE_SLACK)
            c->pl.qrows = std::min(c->pl.qrows + 4, c->pl.stride + NL_QUEUE_SLACK);
        c->pl_overflow_seen = seen;
        TRY(sphmw_publish_words(c, (const uint32_t *)(c->d_counters + 2), (uint32_t *)(c->h_counters + 2), 2, c->stream));
    }
    if (n == 0) {
        c->keys_from_advance = false;
        CUDA_TRY(cudaMemsetAsync(c->cell_start, 0, sizeof(uint32_t) * (ncells + 2), c->stream));
        c->cell_list_valid = true;
        c->n_owned = 0;
        if (n_alive) *n_alive = 0;
        return SPHMW_OK;
    }
    if (!c->allocated[S_X0] || !c->allocated[S_X1] || (g.dim == 3 && !c->allocated[S_X2])) {
        sphmw_set_error("create_cell_list: field x has not been set");
        return SPHMW_E_STATE;
    }
    if (!c->scan_tmp || c->scan_tmp_len < (ncells + 2) / SCAN_TILE * 2 + 4096) {
        cudaFree(c->scan_tmp);
        c->scan_tmp = nullptr;
        c->scan_tmp_len = (ncells + 2) / SCAN_TILE * 2 + 4096;
        CUDA_TRY(cudaMalloc(&c->scan_tmp, sizeof(uint32_t) * c->scan_tmp_len));
    }

    // keys written by the force pass's advance (pair_ops.cu run_fused_force): same function, same x
    const bool keyed = c->keys_from_advance && c->slab_lo < 0;
    c->keys_from_advance = false;
    if (!keyed) {
        CUDA_TRY(cudaMemsetAsync(c->removed, 0, sizeof(uint32_t) * 2, c->stream));
        TIMED(c, "cell_keys");
        const bool slab = c->slab_lo >= 0;
        const unsigned gr = grid_for(n, 256);
#define KEYS_ARGS c->cur.s[S_X0], c->cur.s[S_X1], c->cur.s[S_X2], n, g, c->key, c->removed, \
                  (uint32_t)c->removed_cap, c->idx, c->tag, c->cellx
        if (g.dim == 2 && !slab) k_keys<2, false><<<gr, 256, 0, c->stream>>>(KEYS_ARGS);
        else if (g.dim == 2) k_keys<2, true><<<gr, 256, 0, c->stream>>>(KEYS_ARGS);
        else if (!slab) k_keys<3, false><<<gr, 256, 0, c->stream>>>(KEYS_ARGS);
        else k_keys<3, true><<<gr, 256, 0, c->stream>>>(KEYS_ARGS);
#undef KEYS_ARGS
    }
    TRY(sphmw_publish_words(c, c->removed, c->h_removed, 2, c->stream));
    // overlap the host round trip with the histogram
    CUDA_TRY(cudaMemsetAsync(c->cell_start, 0, sizeof(uint32_t) * (ncells + 2), c->stream));
    {
        TIMED(c, "cell_histogram");
        k_histogram<<<grid_for(n, 256), 256, 0, c->stream>>>(c->key, n, c->cell_start, c->rank);
    }
    TRY(exclusive_scan(c, c->cell_start, ncells + 2, c->scan_tmp, c->scan_tmp_len));
    {
        TIMED(c, "cell_scatter");
        k_scatter<<<grid_for(n, 256), 256, 0, c->stream>>>(c->key, c->rank, c->cell_start, n, c->src);
    }
    // How many particles are dropped.  A whole-domain context has to ask the device (and replays
    // the reference's renumbering below).  A slab context knows from the halo pack (halo.cu:
    // ghosts and migrants of the last exchange + particles the pack dropped) and does not wait;
    // what the device counted is checked against it one build later, when the copy has long landed.
    int64_t k;
    uint32_t owned_live;
    if (c->slab_lo >= 0 && c->slab_dead_known && !getenv("SPHMW_SLAB_SYNC_BUILD")) {
        if (!c->h_slab_check) {
            CUDA_TRY(cudaMallocHost(&c->h_slab_check, sizeof(uint32_t) * 2 * 4));
            for (int e = 0; e < 4; ++e) CUDA_TRY(cudaEventCreateWithFlags(&c->slab_check_event[e], cudaEventDisableTiming));
        }
        if (c->slab_checks > 0) {
            const int prev = (int)((c->slab_checks - 1) & 3);
            CUDA_TRY(cudaEventSynchronize(c->slab_check_event[prev]));
            if ((int64_t)c->h_slab_check[2 * prev] != c->slab_check_want[prev][0] ||
                (int64_t)c->h_slab_check[2 * prev + 1] != c->slab_check_want[prev][1]) {
                sphmw_set_error("slab bookkeeping diverged: the device dropped %u particles and kept %u owned ones, "
                                "the host expected %lld and %lld", c->h_slab_check[2 * prev], c->h_slab_check[2 * prev + 1],
                                (long long)c->slab_check_want[prev][0], (long long)c->slab_check_want[prev][1]);
                return SPHMW_E_STATE;
            }
        }
        const int cur = (int)(c->slab_checks & 3);
        TRY(sphmw_publish_words(c, c->removed, c->h_slab_check + 2 * cur, 2, c->stream));
        CUDA_TRY(cudaEventRecord(c->slab_check_event[cur], c->stream));
        k = c->slab_dead_expected;
        owned_live = (uint32_t)c->n_owned;
        c->slab_check_want[cur][0] = k;
        c->slab_check_want[cur][1] = c->n_owned;
        c->slab_checks += 1;
    } else {
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        k = c->h_removed[0];
        owned_live = c->h_removed[1];  // slab mode only (else the first removed index)
    }
    c->slab_dead_known = false;
    if (k > 0 && c->slab_lo < 0) {
        if (k > c->removed_cap) {
            // the list of removed indices did not fit (the reference removes any number of
            // particles, core.jl:60-81): grow it and run the key kernel again — it rewrites the same
            // keys and fills the list; histogram and scatter did not depend on the list
            cudaFree(c->removed);
            cudaFreeHost(c->h_removed);
            c->removed = nullptr;
            c->h_removed = nullptr;
            c->removed_cap = k + k / 4 + 1024;
            CUDA_TRY(cudaMalloc(&c->removed, sizeof(uint32_t) * (c->removed_cap + 1)));
            CUDA_TRY(cudaMallocHost(&c->h_removed, sizeof(uint32_t) * (c->removed_cap + 1)));
            CUDA_TRY(cudaMemsetAsync(c->removed, 0, sizeof(uint32_t) * 2, c->stream));
            const unsigned gr = grid_for(n, 256);
            if (g.dim == 2)
                k_keys<2, false><<<gr, 256, 0, c->stream>>>(c->cur.s[S_X0], c->cur.s[S_X1], c->cur.s[S_X2], n, g, c->key,
                                                            c->removed, (uint32_t)c->removed_cap, c->idx, c->tag, c->cellx);
            else
                k_keys<3, false><<<gr, 256, 0, c->stream>>>(c->cur.s[S_X0], c->cur.s[S_X1], c->cur.s[S_X2], n, g, c->key,
                                                            c->removed, (uint32_t)c->removed_cap, c->idx, c->tag, c->cellx);
            CUDA_TRY(cudaGetLastError());
            c->launches += 1;
        }
        CUDA_TRY(cudaMemcpyAsync(c->h_removed + 1, c->removed + 1, sizeof(uint32_t) * k,
                                 cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        std::vector<uint32_t> rem(c->h_removed + 1, c->h_removed + 1 + k), mo, mn;
        sphmw_replay_swap_removal(n, rem, mo, mn);
        const int64_t m = (int64_t)mo.size();
        if (m > 0) {
            if (m > c->mv_cap) {
                cudaFree(c->mv_old);
                cudaFree(c->mv_new);
                c->mv_cap = m * 2;
                CUDA_TRY(cudaMalloc(&c->mv_old, sizeof(uint32_t) * c->mv_cap));
                CUDA_TRY(cudaMalloc(&c->mv_new, sizeof(uint32_t) * c->mv_cap));
            }
            CUDA_TRY(cudaMemcpyAsync(c->mv_old, mo.data(), sizeof(uint32_t) * m,
                                     cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaMemcpyAsync(c->mv_new, mn.data(), sizeof(uint32_t) * m,
                                     cudaMemcpyHostToDevice, c->stream));
            TRY(sphmw_ensure_pos_of_idx(c));
            TIMED(c, "cell_renumber");
            k_renumber<<<grid_for(m, 256), 256, 0, c->stream>>>(c->idx, c->pos_of_idx, c->mv_old,
                                                                c->mv_new, m);
            // mo/mn must outlive the async copies
            CUDA_TRY(cudaStreamSynchronize(c->stream));
        }
    }
    const int64_t n_new = n - k;
    {
        TIMED(c, "cell_order");
        k_cell_order<<<grid_for(ncells, 128), 128, 0, c->stream>>>(c->cell_start, ncells, c->src,
                                                                   c->idx);
    }
    GatherList gl;
    gl.count = 0;
    int gathered[NSLOT];
    gl.xq = c->xq;
    gl.h = g.h;
    gl.q6 = g.zrun;  // mirror format follows the physical cell order (sphmw_internal.h)
    gl.dim = g.dim;
    gl.run_phase = g.phase[g.dim == 3 ? 2 : 1];
    for (int a = 0; a < 3; ++a) gl.xpos[a] = -1;
    gl.mpos = -1;
    gl.recA = nullptr;
    gl.tpos = -1;
    gl.fluid = c->prm.fluid;
    gl.fl = nullptr;
    c->fluid_gen = ~0ull;
    const bool fluid_list = c->want_fluid_list && c->allocated[S_TYPE] && !c->stale[S_TYPE] && n_new > 0;
    if (fluid_list && !c->fluid_work) {
        CUDA_TRY(cudaMalloc(&c->fluid_flag, (size_t)c->cap + 8));
        CUDA_TRY(cudaMalloc(&c->fluid_work, sizeof(uint32_t) * (size_t)c->cap));
    }
    if (fluid_list) gl.fl = c->fluid_flag;
    if (sphmw_use_records(c) && c->allocated[S_M] && !c->stale[S_M]) {
        TRY(sphmw_ensure_records(c));
        gl.recA = c->rec[0];
        c->rec_gen = c->cell_gen;
    }
    for (int s = 0; s < NSLOT; ++s)
        if (c->allocated[s] && !c->stale[s]) {
            gl.from[gl.count] = c->cur.s[s];
            gl.to[gl.count] = c->alt.s[s];
            gathered[gl.count] = s;
            if (s >= S_X0 && s <= S_X2) gl.xpos[s - S_X0] = gl.count;
            if (s == S_M) gl.mpos = gl.count;
            if (s == S_TYPE) gl.tpos = gl.count;
            ++gl.count;
        }
    if (n_new > 0) {
        TIMED(c, "cell_gather");
        k_gather<<<grid_for(n_new, 256), 256, 0, c->stream>>>(gl, c->src, c->idx, c->idx_alt,
                                                              nullptr, c->key, c->rank, c->tag,
                                                              c->tag_alt, c->cellx, c->cellx_alt, n_new);
    }
    c->pos_valid = false;  // rebuilt on demand (sphmw_ensure_pos_of_idx)
    CUDA_TRY(cudaGetLastError());
    if (fluid_list) TRY(build_fluid_list(c, n_new));
    for (int f = 0; f < gl.count; ++f) std::swap(c->cur.s[gathered[f]], c->alt.s[gathered[f]]);
    std::swap(c->idx, c->idx_alt);
    std::swap(c->key, c->rank);
    std::swap(c->tag, c->tag_alt);
    std::swap(c->cellx, c->cellx_alt);
    c->n = n_new;
    c->n_owned = c->slab_lo < 0 ? n_new : (int64_t)owned_live;
    c->cell_list_valid = true;
    if (n_alive) *n_alive = n_new;
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// test hooks
// ---------------------------------------------------------------------------
// the REFERENCE key (structs.jl:102, 0-based) of every particle, in particle index order
__global__ void k_keys_by_index(const uint32_t *__restrict__ key, const uint32_t *__restrict__ cellx,
                                const uint32_t *__restrict__ idx, int64_t n, Grid g,
                                long long *__restrict__ out) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos < n) {
        CellCoord c = cell_of(g, key[pos], cellx[pos]);
        out[idx[pos]] = c.i + g.lim[0] * (long long)c.rest;
    }
}

extern "C" int sphmw_cell_keys(sphmw_ctx *c, int64_t *keys, int64_t n) {
    if (!c || !keys) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (!c->cell_list_valid) { sphmw_set_error("cell list is not built"); return SPHMW_E_STATE; }
    if (n != c->n) { sphmw_set_error("cell_keys: n mismatch"); return SPHMW_E_INVALID; }
    if (n == 0) return SPHMW_OK;
    long long *d = (long long *)c->staging;  // 3*cap doubles >= n int64
    {
        TIMED(c, "keys_by_index");
        k_keys_by_index<<<grid_for(n, 256), 256, 0, c->stream>>>(c->key, c->cellx, c->idx, n, c->grid, d);
    }
    CUDA_TRY(cudaMemcpyAsync(keys, d, sizeof(int64_t) * n, cudaMemcpyDefault, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

extern "C" int sphmw_cell_entries(sphmw_ctx *c, int64_t key, int64_t *out, int64_t cap, int64_t *n) {
    if (!c || !n) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (!c->cell_list_valid) { sphmw_set_error("cell list is not built"); return SPHMW_E_STATE; }
    if (key < 0 || key >= c->grid.key_max) { sphmw_set_error("cell key out of range"); return SPHMW_E_INVALID; }
    uint32_t be[2];
    const long long pk = pkey_of(c->grid, (int)(key % c->grid.lim[0]), (int)(key / c->grid.lim[0]));
    CUDA_TRY(cudaMemcpyAsync(be, c->cell_start + pk, sizeof(be), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    int64_t cnt = (int64_t)be[1] - (int64_t)be[0];
    *n = cnt;
    int64_t m = std::min(cnt, cap);
    if (m > 0 && out) {
        std::vector<uint32_t> tmp(m);
        CUDA_TRY(cudaMemcpy(tmp.data(), c->idx + be[0], sizeof(uint32_t) * m, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < m; ++i) out[i] = tmp[i];
    }
    return SPHMW_OK;
}
