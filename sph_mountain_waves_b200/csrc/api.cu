// libsphmw C ABI: context, parameters, field transfer, reductions, timing.
// Reference interfaces replaced: ParticleSystem (src/structs.jl:43-92),
// ParticleField (src/structs.jl:118-125), diagnostics of the drivers
// (src/current/wcsph_perturbed_witch.jl:338-350), smoothing kernels (src/kernels.jl).
#include <math.h>
#include <cmath>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "kernels_sph.cuh"
#include "sphmw_internal.h"

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

void sphmw_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char *sphmw_last_error(void) { return g_err; }
extern "C" const char *sphmw_version(void) { return "sphmw 0.1 (sm_100a)"; }

// ---------------------------------------------------------------------------
// field and parameter tables
// ---------------------------------------------------------------------------
static const FieldDesc FIELD_TABLE[] = {
    {"h", S_H, 1},
    {"x", S_X0, 3},
    {"m", S_M, 1},
    {"v", S_V0, 3},
    {"u", S_V0, 3},  // legacy drivers call the velocity `u` (isothermal_flow_witch.jl:70)
    {"Dv", S_DV0, 3},
    {"a", S_DV0, 3},  // test_collision_2d.jl:40
    {"rho_bg", S_RHO_BG, 1}, {"ρ_bg", S_RHO_BG, 1},
    {"rho_p", S_RHO_P, 1},   {"ρ′", S_RHO_P, 1},
    {"rho", S_RHO, 1},       {"ρ", S_RHO, 1},
    {"P_bg", S_P_BG, 1},
    {"P_p", S_P_P, 1},       {"P′", S_P_P, 1},
    {"P", S_P, 1},
    {"theta_bg", S_TH_BG, 1}, {"θ_bg", S_TH_BG, 1},
    {"theta_p", S_TH_P, 1},   {"θ′", S_TH_P, 1},
    {"theta", S_TH, 1},       {"θ", S_TH, 1},
    {"T_bg", S_T_BG, 1},
    {"T_p", S_T_P, 1},        {"T′", S_T_P, 1},
    {"T", S_T, 1},
    {"type", S_TYPE, 1},
    {"A", S_A, 1},
    {"A_bg", S_A_BG, 1},
    {"Drho", S_DRHO, 1},
    {"rho0", S_RHO0, 1},
    {"S", S_ENT, 1},   // adiabatic_flow_witch.jl:75-76
    {"s", S_ENT_D, 1},
    {nullptr, 0, 0}};

const FieldDesc *sphmw_find_field(const char *name) {
    for (const FieldDesc *d = FIELD_TABLE; d->name; ++d)
        if (!strcmp(d->name, name)) return d;
    return nullptr;
}

struct ParamDesc {
    const char *name;
    size_t off;
};
#define POFF(f) offsetof(Params, f)
static const ParamDesc PARAM_TABLE[] = {
    {"dt", POFF(dt)},           {"g", POFF(g)},         {"c", POFF(c)},
    {"gamma", POFF(gamma)},     {"alpha", POFF(alpha)}, {"beta", POFF(beta)},
    {"eps", POFF(eps)},         {"eta", POFF(eta)},     {"rho0", POFF(rho0)},
    {"R_mass", POFF(R_mass)},   {"R_gas", POFF(R_gas)}, {"T_bg", POFF(T_bg)},
    {"rho_floor", POFF(rho_floor)}, {"P_floor", POFF(P_floor)},
    {"z_t", POFF(z_t)},         {"z_b", POFF(z_b)},     {"gamma_r", POFF(gamma_r)},
    {"fluid", POFF(fluid)},     {"m", POFF(m)},         {"nu", POFF(nu)},
    {"mu", POFF(mu)},           {"gx", POFF(gx)},       {"gy", POFF(gy)},
    {"gz", POFF(gz)},           {"kh", POFF(kh)},       {"dt_pack", POFF(dt_pack)},
    {"c_pack", POFF(c_pack)},   {"zeta_pack", POFF(zeta_pack)}, {"U_max", POFF(U_max)},
    {"cp", POFF(cp)},           {"bc_width", POFF(bc_width)},   {"x_inflow", POFF(x_inflow)},
    {"dr", POFF(dr)},           {"inflow", POFF(inflow)},       {nullptr, 0}};

extern "C" int sphmw_set_param(sphmw_ctx *c, const char *name, double v) {
    if (!c || !name) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    for (const ParamDesc *d = PARAM_TABLE; d->name; ++d)
        if (!strcmp(d->name, name)) {
            *(double *)((char *)&c->prm + d->off) = v;
            sphmw_derive_params(c->prm);
            return SPHMW_OK;
        }
    sphmw_set_error("unknown parameter '%s'", name);
    return SPHMW_E_INVALID;
}
extern "C" int sphmw_get_param(sphmw_ctx *c, const char *name, double *v) {
    if (!c || !name || !v) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    for (const ParamDesc *d = PARAM_TABLE; d->name; ++d)
        if (!strcmp(d->name, name)) {
            *v = *(double *)((char *)&c->prm + d->off);
            return SPHMW_OK;
        }
    sphmw_set_error("unknown parameter '%s'", name);
    return SPHMW_E_INVALID;
}

__global__ void k_publish_words(const uint32_t *__restrict__ src, volatile uint32_t *dst, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
}
int sphmw_publish_words(sphmw_ctx *c, const uint32_t *dev_src, uint32_t *pinned_dst, int nwords, cudaStream_t stream) {
    k_publish_words<<<1, 32, 0, stream>>>(dev_src, pinned_dst, nwords);
    CUDA_TRY(cudaGetLastError());
    c->launches += 1;
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// timing
// ---------------------------------------------------------------------------
static int timing_name_id(sphmw_ctx *c, const char *name) {
    for (size_t i = 0; i < c->timing_names.size(); ++i)
        if (c->timing_names[i] == name) return (int)i;
    c->timing_names.push_back(name);
    c->timing_ms.push_back(0.0);
    c->timing_calls.push_back(0);
    return (int)c->timing_names.size() - 1;
}
static cudaEvent_t get_event(sphmw_ctx *c) {
    if (!c->event_pool.empty()) {
        cudaEvent_t e = c->event_pool.back();
        c->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
static void timing_resolve(sphmw_ctx *c) {
    if (c->timing_pending.empty()) return;
    cudaEventSynchronize(c->timing_pending.back().b);
    for (auto &t : c->timing_pending) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t.a, t.b);
        c->timing_ms[t.name_id] += ms;
        c->timing_calls[t.name_id] += 1;
        c->event_pool.push_back(t.a);
        c->event_pool.push_back(t.b);
    }
    c->timing_pending.clear();
}
KernelTimer::KernelTimer(sphmw_ctx *ctx, const char *name) : c(ctx), pending_index(-1) {
    c->launches += 1;
    if (!c->timing) return;
    if (!c->timing_prefix.empty() && strncmp(name, c->timing_prefix.c_str(), c->timing_prefix.size())) return;
    if (c->timing_pending.size() >= 8192) timing_resolve(c);
    TimingEntry t;
    t.name_id = timing_name_id(c, name);
    t.a = get_event(c);
    t.b = get_event(c);
    cudaEventRecord(t.a, c->stream);
    c->timing_pending.push_back(t);
    pending_index = (int)c->timing_pending.size() - 1;
}
KernelTimer::~KernelTimer() {
    if (pending_index >= 0) cudaEventRecord(c->timing_pending[pending_index].b, c->stream);
}
extern "C" int sphmw_timing_enable(sphmw_ctx *c, int32_t enable) {
    if (!c) return SPHMW_E_INVALID;
    if (!enable) timing_resolve(c);
    c->timing = enable != 0;
    return SPHMW_OK;
}
// only kernels whose name starts with `prefix` are timed (NULL or "": all) — two event records per
// launch are not free when a step is a few milliseconds of ~30 launches
extern "C" int sphmw_timing_filter(sphmw_ctx *c, const char *prefix) {
    if (!c) return SPHMW_E_INVALID;
    timing_resolve(c);
    c->timing_prefix = prefix ? prefix : "";
    return SPHMW_OK;
}
extern "C" int sphmw_timing_reset(sphmw_ctx *c) {
    if (!c) return SPHMW_E_INVALID;
    timing_resolve(c);
    std::fill(c->timing_ms.begin(), c->timing_ms.end(), 0.0);
    std::fill(c->timing_calls.begin(), c->timing_calls.end(), 0);
    return SPHMW_OK;
}
extern "C" int64_t sphmw_timing_report(sphmw_ctx *c, char *names, int64_t cap, double *ms,
                                       int64_t *calls, int32_t max_entries) {
    if (!c) return SPHMW_E_INVALID;
    timing_resolve(c);
    std::string all;
    int n = 0;
    for (size_t i = 0; i < c->timing_names.size(); ++i) {
        if (c->timing_calls[i] == 0) continue;
        if (n < max_entries) {
            if (ms) ms[n] = c->timing_ms[i];
            if (calls) calls[n] = c->timing_calls[i];
            all += c->timing_names[i];
            all += "\n";
        }
        ++n;
    }
    if (names && cap > 0) {
        size_t k = std::min<size_t>(all.size(), (size_t)cap - 1);
        memcpy(names, all.data(), k);
        names[k] = 0;
    }
    return n;
}
extern "C" int sphmw_launch_count(sphmw_ctx *c, int64_t *n) {
    if (!c || !n) return SPHMW_E_INVALID;
    *n = c->launches;
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// create / destroy
// ---------------------------------------------------------------------------
extern "C" int sphmw_create(const sphmw_config *cfg, sphmw_ctx **out) {
    if (!cfg || !out) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    *out = nullptr;
    // structs.jl:59 — @assert h > 0
    if (!(cfg->h > 0.0)) {
        sphmw_set_error("invalid ParticleSystem declaration! (h must be a positive float)");
        return SPHMW_E_INVALID;
    }
    if (cfg->capacity <= 0 || cfg->capacity >= (int64_t)0xFFFFFFF0u) {
        sphmw_set_error("capacity must be in (0, 2^32-16)");
        return SPHMW_E_INVALID;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        sphmw_set_error("no CUDA device (%s); libsphmw has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return SPHMW_E_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) {
        sphmw_set_error("device ordinal %d out of range (%d devices)", cfg->device, ndev);
        return SPHMW_E_INVALID;
    }
    CUDA_TRY(cudaSetDevice(cfg->device));

    sphmw_ctx *c = new sphmw_ctx();
    c->device = cfg->device;
    c->flags = cfg->flags;
    c->cap = cfg->capacity;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
    Grid &g = c->grid;
    c->slab_lo = cfg->slab_lo;
    c->slab_hi = cfg->slab_hi;
    {
        // key tables, neighbour offsets, physical cell order, exact cut-off (grid_setup.cpp)
        const int rc = sphmw_grid_setup(g, cfg->box_min, cfg->box_max, cfg->h, cfg->slab_lo, cfg->slab_hi,
                                        &c->global_cols, (cfg->flags & SPHMW_FLAG_GHOST3) ? 3 : GHOST_COLS);
        if (rc != SPHMW_OK) {
            delete c;
            return rc;
        }
        // physical cell order: zrun unless a shared-memory variant that stages x-rows is asked for;
        // sphmw_set_flags may switch later, so the cell-start table is sized for either order
        Grid xo = g;
        sphmw_grid_set_order(xo, false);
        c->cells_cap = std::max(g.pkey_max, xo.pkey_max);
        if (c->cells_cap >= (long long)0x7FFFFFF0) {
            sphmw_set_error("too many cells (%lld)", (long long)c->cells_cap);
            delete c;
            return SPHMW_E_INVALID;
        }
        if (!sphmw_want_zrun(c->flags)) g = xo;
    }
    memset(&c->prm, 0, sizeof(Params));

    int rc = [&]() -> int {
        CUDA_TRY(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
        c->stream = c->own_stream;
        CUDA_TRY(cudaMalloc(&c->idx, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->idx_alt, sizeof(uint32_t) * c->cap));
        if (c->slab_lo < 0) CUDA_TRY(cudaMalloc(&c->pos_of_idx, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->tag, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->tag_alt, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->halo_counters, sizeof(uint32_t) * 8));
        CUDA_TRY(cudaMemsetAsync(c->halo_counters, 0, sizeof(uint32_t) * 8, c->stream));
        CUDA_TRY(cudaEventCreateWithFlags(&c->pack_event, cudaEventDisableTiming));
        CUDA_TRY(cudaMallocHost(&c->h_halo_counters, sizeof(uint32_t) * 8));
        CUDA_TRY(cudaMalloc(&c->key, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->cellx, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->cellx_alt, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->rank, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->src, sizeof(uint32_t) * c->cap));
        CUDA_TRY(cudaMalloc(&c->cell_start, sizeof(uint32_t) * (c->cells_cap + 2)));
        c->removed_cap = 1 << 20;
        CUDA_TRY(cudaMalloc(&c->removed, sizeof(uint32_t) * (c->removed_cap + 1)));
        CUDA_TRY(cudaMallocHost(&c->h_removed, sizeof(uint32_t) * (c->removed_cap + 1)));
        CUDA_TRY(cudaMalloc(&c->d_counters, sizeof(unsigned long long) * 8));
        CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, sizeof(unsigned long long) * 8, c->stream));
        CUDA_TRY(cudaMallocHost(&c->h_counters, sizeof(unsigned long long) * 8));
        CUDA_TRY(cudaMalloc(&c->xq, sizeof(uint32_t) * (c->cap + 4)));  // +4: pair_list.cuh reads past a run
        CUDA_TRY(cudaMemsetAsync(c->xq, 0, sizeof(uint32_t) * (c->cap + 4), c->stream));
        CUDA_TRY(cudaMalloc(&c->staging, sizeof(double) * 3 * c->cap));
        CUDA_TRY(cudaMalloc(&c->reduce_tmp, sizeof(double) * 4096));
        return SPHMW_OK;
    }();
    if (rc != SPHMW_OK) {
        sphmw_destroy(c);
        return rc;
    }
    *out = c;
    return SPHMW_OK;
}

extern "C" int sphmw_destroy(sphmw_ctx *c) {
    if (!c) return SPHMW_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    sphmw_comm_free(c);
    sphmw_frame_async_free(c);
    if (c->h_slab_check) cudaFreeHost(c->h_slab_check);
    for (auto e : c->slab_check_event)
        if (e) cudaEventDestroy(e);
    for (int s = 0; s < NSLOT; ++s) {
        cudaFree(c->cur.s[s]);
        cudaFree(c->alt.s[s]);
    }
    cudaFree(c->idx); cudaFree(c->idx_alt); cudaFree(c->pos_of_idx); cudaFree(c->lost_list);
    cudaFree(c->tag); cudaFree(c->tag_alt); cudaFree(c->halo_counters);
    if (c->h_halo_counters) cudaFreeHost(c->h_halo_counters);
    cudaFree(c->key); cudaFree(c->rank); cudaFree(c->src); cudaFree(c->cellx); cudaFree(c->cellx_alt);
    cudaFree(c->cell_start); cudaFree(c->scan_tmp); cudaFree(c->removed);
    cudaFree(c->mv_old); cudaFree(c->mv_new);
    cudaFree(c->d_counters); cudaFree(c->staging); cudaFree(c->reduce_tmp);
    cudaFree(c->pt_pts); cudaFree(c->pt_out); cudaFree(c->pt_key); cudaFree(c->pt_order); cudaFree(c->pt_sort_tmp);
    cudaFree(c->fluid_flag); cudaFree(c->fluid_work); cudaFree(c->fluid_tiles);
    cudaFree(c->xq); cudaFree(c->pl.list); cudaFree(c->pl.list16); cudaFree(c->pl.cnt); cudaFree(c->tile_tab);
    for (int k = 0; k < 3; ++k) cudaFree(c->rec[k]);
    if (c->h_removed) cudaFreeHost(c->h_removed);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    for (auto &t : c->timing_pending) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    if (c->pack_event) cudaEventDestroy(c->pack_event);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return SPHMW_OK;
}

extern "C" int sphmw_set_stream(sphmw_ctx *c, void *s) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return SPHMW_OK;
}
extern "C" int sphmw_set_flags(sphmw_ctx *c, int32_t flags) {
    if (!c) return SPHMW_E_INVALID;
    c->flags = flags;
    if ((c->grid.zrun != 0) != sphmw_want_zrun(flags)) {
        // the variant asked for needs the other physical cell order: same cells, same particles,
        // stored differently — rebuild the cell list if one was valid (results do not change)
        CUDA_TRY(cudaSetDevice(c->device));
        sphmw_grid_set_order(c->grid, sphmw_want_zrun(flags));
        c->pl_gen = ~0ull;
        c->tile_gen = ~0ull;
        if (c->cell_list_valid) {
            c->cell_list_valid = false;
            if (c->slab_lo < 0) TRY(sphmw_build_cell_list(c, nullptr));
        }
    }
    return SPHMW_OK;
}
extern "C" int sphmw_sync(sphmw_ctx *c) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

extern "C" int sphmw_key_tables(sphmw_ctx *c, int64_t phase[3], int64_t lim[3], int64_t *key_max,
                                int32_t *dim) {
    if (!c) return SPHMW_E_INVALID;
    for (int a = 0; a < 3; ++a) {
        if (phase) phase[a] = c->grid.phase[a];
        if (lim) lim[a] = c->grid.lim[a];
    }
    if (key_max) *key_max = c->grid.key_max;
    if (dim) *dim = c->grid.dim;
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// particle count and field storage
// ---------------------------------------------------------------------------
__global__ void k_iota(uint32_t *a, uint32_t *b, uint32_t *tag, int64_t first, int64_t n) {
    int64_t i = first + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) {
        a[i] = (uint32_t)i;
        if (b) b[i] = (uint32_t)i;
        tag[i] = TAG_OWNED;
    }
}

int sphmw_ensure_records(sphmw_ctx *c) {
    for (int k = 0; k < 3; ++k)
        if (!c->rec[k]) {
            CUDA_TRY(cudaMalloc(&c->rec[k], sizeof(NbRec) * (size_t)c->cap));
            CUDA_TRY(cudaMemsetAsync(c->rec[k], 0, sizeof(NbRec) * (size_t)c->cap, c->stream));
        }
    return SPHMW_OK;
}

int sphmw_ensure_slot(sphmw_ctx *c, int slot) {
    if (c->allocated[slot]) return SPHMW_OK;
    // + 4: the bulk copies of the tiled pair kernels fetch whole groups of 4 particles
    CUDA_TRY(cudaMalloc(&c->cur.s[slot], sizeof(double) * (c->cap + 4)));
    CUDA_TRY(cudaMalloc(&c->alt.s[slot], sizeof(double) * (c->cap + 4)));
    CUDA_TRY(cudaMemsetAsync(c->cur.s[slot], 0, sizeof(double) * (c->cap + 4), c->stream));
    CUDA_TRY(cudaMemsetAsync(c->alt.s[slot], 0, sizeof(double) * (c->cap + 4), c->stream));
    c->allocated[slot] = true;
    c->stale[slot] = false;
    return SPHMW_OK;
}

extern "C" int sphmw_resize(sphmw_ctx *c, int64_t n) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (n < 0 || n > c->cap) {
        sphmw_set_error("resize to %lld exceeds capacity %lld", (long long)n, (long long)c->cap);
        return SPHMW_E_CAPACITY;
    }
    if (n > c->n) {
        // appended particles: index = position = old count.., all fields zero
        int64_t m = n - c->n;
        {
            TIMED(c, "iota");
            k_iota<<<grid_for(m, 256), 256, 0, c->stream>>>(c->idx, c->pos_of_idx, c->tag, c->n, n);
        }
        for (int s = 0; s < NSLOT; ++s)
            if (c->allocated[s])
                CUDA_TRY(cudaMemsetAsync(c->cur.s[s] + c->n, 0, sizeof(double) * m, c->stream));
    } else if (n < c->n) {
        if (c->n != 0 && n != 0) {
            sphmw_set_error("shrinking is only supported to 0 (use the domain box to remove particles)");
            return SPHMW_E_INVALID;
        }
    }
    c->n = n;
    c->n_owned = n;
    c->cell_list_valid = false;
    c->keys_from_advance = false;
    return SPHMW_OK;
}
extern "C" int sphmw_count(sphmw_ctx *c, int64_t *n) {
    if (!c || !n) return SPHMW_E_INVALID;
    *n = c->n;
    return SPHMW_OK;
}

// dst[pos] = staging[idx[pos]]   (upload)      — coalesced writes
__global__ void k_permute_in(double *__restrict__ dst, const double *__restrict__ stg,
                             const uint32_t *__restrict__ idx, int64_t n) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos < n) dst[pos] = stg[idx[pos]];
}
// staging[idx[pos]] = src[pos]   (download)    — coalesced reads
__global__ void k_permute_out(double *__restrict__ stg, const double *__restrict__ src,
                              const uint32_t *__restrict__ idx, int64_t n) {
    int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos < n) stg[idx[pos]] = src[pos];
}

__global__ void k_count_nonzero(const double *__restrict__ a, int64_t n, unsigned long long *__restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool nz = i < n && !(a[i] == 0.0);  // NaN counts as non-zero
    const int cnt = __syncthreads_count(nz);
    if (threadIdx.x == 0 && cnt) atomicAdd(out, (unsigned long long)cnt);
}

extern "C" int sphmw_upload(sphmw_ctx *c, const char *field, const double *buf, int64_t n,
                            int32_t ncomp) {
    if (!c || !field || !buf) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    const FieldDesc *d = sphmw_find_field(field);
    if (!d) { sphmw_set_error("Variable %s does not exist!", field); return SPHMW_E_UNKNOWN_FIELD; }
    if (ncomp != d->ncomp || n != c->n) {
        sphmw_set_error("upload(%s): expected %d x %lld values, got %d x %lld", field, d->ncomp,
                        (long long)c->n, ncomp, (long long)n);
        return SPHMW_E_INVALID;
    }
    if (n == 0) return SPHMW_OK;
    CUDA_TRY(cudaMemcpyAsync(c->staging, buf, sizeof(double) * n * ncomp, cudaMemcpyDefault,
                             c->stream));
    for (int k = 0; k < ncomp; ++k) {
        int slot = d->slot + k;
        if (c->grid.dim == 2 && ncomp == 3 && k == 2) {
            // 2D systems keep no third component.  In the reference a particle with x[3] != 0 leaves
            // the box 0 <= x[3] <= 0 (geometry.jl:24-30) and is removed, and one with v[3] != 0 does so
            // after its first move!; silently dropping the component would diverge from that, so a
            // non-zero third component is refused.
            CUDA_TRY(cudaMemsetAsync(c->d_counters + 7, 0, sizeof(unsigned long long), c->stream));
            k_count_nonzero<<<grid_for(n, 256), 256, 0, c->stream>>>(c->staging + (int64_t)k * n, n, c->d_counters + 7);
            CUDA_TRY(cudaMemcpyAsync(c->h_counters + 7, c->d_counters + 7, sizeof(unsigned long long),
                                     cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            if (c->h_counters[7] != 0) {
                sphmw_set_error("upload(%s): %llu particles have a non-zero third component in a 2D system "
                                "(the reference would remove them: box 0 <= x[3] <= 0)", field, c->h_counters[7]);
                return SPHMW_E_INVALID;
            }
            continue;
        }
        TRY(sphmw_ensure_slot(c, slot));
        TIMED(c, "upload_permute");
        k_permute_in<<<grid_for(n, 256), 256, 0, c->stream>>>(c->cur.s[slot],
                                                              c->staging + (int64_t)k * n, c->idx, n);
        c->stale[slot] = false;
    }
    if (d->slot == S_X0) c->cell_list_valid = false, c->keys_from_advance = false;
    if (d->slot == S_DV0) c->dv_zero = false;
    if (d->slot == S_TYPE) c->fluid_gen = ~0ull;  // the fluid work list no longer matches the types
    CUDA_TRY(cudaGetLastError());
    // staging is reused by the next call: the copy out of `buf` must be complete
    // before we return anyway (host memory is only borrowed).
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

extern "C" int sphmw_download(sphmw_ctx *c, const char *field, double *buf, int64_t n,
                              int32_t ncomp) {
    if (!c || !field || !buf) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    const FieldDesc *d = sphmw_find_field(field);
    if (!d) { sphmw_set_error("Variable %s does not exist!", field); return SPHMW_E_UNKNOWN_FIELD; }
    if (ncomp != d->ncomp || n != c->n) {
        sphmw_set_error("download(%s): expected %d x %lld values, got %d x %lld", field, d->ncomp,
                        (long long)c->n, ncomp, (long long)n);
        return SPHMW_E_INVALID;
    }
    if (n == 0) return SPHMW_OK;
    for (int k = 0; k < ncomp; ++k) {
        int slot = d->slot + k;
        double *stg = c->staging + (int64_t)k * n;
        bool zero = (c->grid.dim == 2 && ncomp == 3 && k == 2);
        if (!zero) {
            if (c->allocated[slot] && c->stale[slot]) TRY(sphmw_materialize(c, slot));
            if (!c->allocated[slot]) {
                if (slot >= S_DV0 && slot <= S_DV2 && c->dv_zero) zero = true;
                else TRY(sphmw_materialize(c, slot));  // may allocate derived fields
            }
        }
        if (!zero && !c->allocated[slot]) zero = true;  // never written: constructor zero
        if (zero) {
            CUDA_TRY(cudaMemsetAsync(stg, 0, sizeof(double) * n, c->stream));
        } else {
            TIMED(c, "download_permute");
            k_permute_out<<<grid_for(n, 256), 256, 0, c->stream>>>(stg, c->cur.s[slot], c->idx, n);
        }
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(buf, c->staging, sizeof(double) * n * ncomp, cudaMemcpyDefault,
                             c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// reductions — avg_velocity/max_velocity (wcsph_perturbed_witch.jl:338-350)
// ---------------------------------------------------------------------------
// mode 0: sum of a, 1: max of a, 2: sum |v|, 3: max |v|
// Julia's max propagates NaN (wcsph_perturbed_witch.jl:345-350 uses it for max_velocity); fmax drops it.
// Like Julia's max it also orders -0.0 below +0.0, so that the result does not depend on where the
// zeros sit in the reduction tree.
__device__ __forceinline__ double nanmax(double a, double b) {
    if (a != a || b != b) return a + b;
    if (a == b) return signbit(a) ? b : a;
    return a < b ? b : a;
}
__global__ void k_reduce(const double *a, const double *b, const double *cc, int64_t n, int mode,
                         double *out) {
    __shared__ double sh[32];
    double acc = (mode & 1) ? -INFINITY : 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        double v;
        if (mode >= 2) {
            double x = a[i], y = b[i], z = cc ? cc[i] : 0.0;
            v = sqrt(x * x + y * y + z * z);  // algebra.jl:49-60
        } else {
            v = a[i];
        }
        acc = (mode & 1) ? nanmax(acc, v) : acc + v;
    }
    for (int o = 16; o > 0; o >>= 1) {
        double t = __shfl_down_sync(0xffffffffu, acc, o);
        acc = (mode & 1) ? nanmax(acc, t) : acc + t;
    }
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = acc;
    __syncthreads();
    if (w == 0) {
        int nw = blockDim.x >> 5;
        acc = l < nw ? sh[l] : ((mode & 1) ? -INFINITY : 0.0);
        for (int o = 16; o > 0; o >>= 1) {
            double t = __shfl_down_sync(0xffffffffu, acc, o);
            acc = (mode & 1) ? nanmax(acc, t) : acc + t;
        }
        if (l == 0) out[blockIdx.x] = acc;
    }
}

static int reduce_run(sphmw_ctx *c, const double *a, const double *b, const double *cc, int mode,
                      double *out) {
    const int blocks = 1024, threads = 256;
    {
        TIMED(c, "reduce");
        k_reduce<<<blocks, threads, 0, c->stream>>>(a, b, cc, c->n, mode, c->reduce_tmp);
    }
    {
        TIMED(c, "reduce");
        k_reduce<<<1, 1024, 0, c->stream>>>(c->reduce_tmp, nullptr, nullptr, blocks, mode & 1,
                                             c->reduce_tmp + 2048);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, c->reduce_tmp + 2048, sizeof(double), cudaMemcpyDeviceToHost,
                             c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

extern "C" int sphmw_reduce(sphmw_ctx *c, const char *what, double *out) {
    if (!c || !what || !out) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    if (c->slab_lo >= 0) {
        // k_reduce runs over the resident particles, ghost columns included
        sphmw_set_error("reduce: x-slab contexts are not supported (the resident particles include ghost copies); "
                        "use sphmw_slab_counts for the owned count, or reduce on a whole-domain context");
        return SPHMW_E_STATE;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    if (!strcmp(what, "count")) {
        *out = (double)c->n;
        return SPHMW_OK;
    }
    if (c->n == 0) { *out = 0.0; return SPHMW_OK; }
    if (!strcmp(what, "avg_speed") || !strcmp(what, "max_speed")) {
        if (!c->allocated[S_V0]) { *out = 0.0; return SPHMW_OK; }
        int mode = !strcmp(what, "avg_speed") ? 2 : 3;
        TRY(reduce_run(c, c->cur.s[S_V0], c->cur.s[S_V1], c->cur.s[S_V2], mode, out));
        if (mode == 2) *out /= (double)c->n;
        return SPHMW_OK;
    }
    const char *colon = strchr(what, ':');
    if (colon && (!strncmp(what, "sum:", 4) || !strncmp(what, "max:", 4))) {
        const FieldDesc *d = sphmw_find_field(colon + 1);
        if (!d || d->ncomp != 1) {
            sphmw_set_error("reduce: '%s' is not a scalar field", colon + 1);
            return SPHMW_E_UNKNOWN_FIELD;
        }
        if (!c->allocated[d->slot] || c->stale[d->slot]) TRY(sphmw_materialize(c, d->slot));
        if (!c->allocated[d->slot]) { *out = 0.0; return SPHMW_OK; }
        return reduce_run(c, c->cur.s[d->slot], nullptr, nullptr, what[0] == 'm' ? 1 : 0, out);
    }
    sphmw_set_error("reduce: unknown quantity '%s'", what);
    return SPHMW_E_INVALID;
}

// ---------------------------------------------------------------------------
// smoothing kernels on the device — src/kernels.jl
// ---------------------------------------------------------------------------
__global__ void k_kernel_eval(int which, const double *h, const double *r, double *out, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = sph_kernel_by_id(which, h[i], r[i]);
}

extern "C" int sphmw_kernel_eval(const char *name, const double *h, const double *r, double *out,
                                 int64_t n, int32_t device) {
    if (!name || !h || !r || !out) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    static const char *NAMES[] = {"wendland1", "Dwendland1", "rDwendland1", "wendland2",
                                  "Dwendland2", "rDwendland2", "wendland3", "Dwendland3",
                                  "rDwendland3", "DDwendland3", "spline23", "Dspline23",
                                  "rDspline23", "spline24", "Dspline24", "rDspline24", nullptr};
    int which = -1;
    for (int i = 0; NAMES[i]; ++i)
        if (!strcmp(NAMES[i], name)) which = i;
    if (which < 0) { sphmw_set_error("unknown kernel '%s'", name); return SPHMW_E_INVALID; }
    if (n <= 0) return SPHMW_OK;
    CUDA_TRY(cudaSetDevice(device));
    double *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, sizeof(double) * 3 * n));
    cudaError_t e = cudaMemcpy(d, h, sizeof(double) * n, cudaMemcpyDefault);
    if (e == cudaSuccess) e = cudaMemcpy(d + n, r, sizeof(double) * n, cudaMemcpyDefault);
    if (e == cudaSuccess) {
        k_kernel_eval<<<grid_for(n, 256), 256>>>(which, d, d + n, d + 2 * n, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, d + 2 * n, sizeof(double) * n, cudaMemcpyDefault);
    cudaFree(d);
    if (e != cudaSuccess) {
        sphmw_set_error("kernel_eval failed: %s", cudaGetErrorString(e));
        return SPHMW_E_CUDA;
    }
    return SPHMW_OK;
}

// ---------------------------------------------------------------------------
// thin wrappers over the other translation units
// ---------------------------------------------------------------------------
extern "C" int sphmw_create_cell_list(sphmw_ctx *c, int64_t *n_alive) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->comm) return sphmw_comm_create_cell_list(c, n_alive);  // slab context: halo exchange, then the sort
    return sphmw_build_cell_list(c, n_alive);
}
extern "C" int sphmw_apply(sphmw_ctx *c, const char *op, int32_t self) {
    if (!c || !op) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_apply_named(c, op, self);
}
extern "C" int64_t sphmw_op_list(char *buf, int64_t cap) { return sphmw_list_ops(buf, cap); }
extern "C" int sphmw_step(sphmw_ctx *c, const char *scheme, int32_t nsteps) {
    if (!c || !scheme || nsteps < 0) { sphmw_set_error("bad argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_step_scheme(c, scheme, nsteps);
}
extern "C" int sphmw_step_phase(sphmw_ctx *c, const char *scheme, int32_t phase) {
    if (!c || !scheme) { sphmw_set_error("bad argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_step_scheme_phase(c, scheme, phase);
}
extern "C" int sphmw_flow_add_new_particles(sphmw_ctx *c, int64_t *n_added) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_flow_add_particles(c, n_added, false);
}
extern "C" int sphmw_aflow_add_new_particles(sphmw_ctx *c, int64_t *n_added) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_flow_add_particles(c, n_added, true);
}
extern "C" int sphmw_pairs_dump(sphmw_ctx *c, int64_t *pi, int64_t *pj, int64_t cap, int64_t *n) {
    if (!c || !n) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo >= 0) { sphmw_set_error("pairs_dump is a whole-domain test hook"); return SPHMW_E_STATE; }
    return sphmw_dump_pairs(c, pi, pj, cap, n);
}
extern "C" int sphmw_pair_list_info(sphmw_ctx *c, int64_t out[4]) {
    if (!c || !out) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_pair_list_stats(c, out);
}
extern "C" int sphmw_tile_info(sphmw_ctx *c, int64_t out[6]) {
    if (!c || !out) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    return sphmw_tile_stats(c, out);
}
// ---- host-only test hooks (no device, no context) --------------------------------------
extern "C" int sphmw_pretest_pairs(const double *xp, const double *xq, int64_t n, double h, int32_t dim,
                                   uint8_t *pass) {
    if (!xp || !xq || !pass || !(h > 0.0) || (dim != 2 && dim != 3)) return SPHMW_E_INVALID;
    for (int64_t i = 0; i < n; ++i) {
        uint32_t wp = 0, wq = 0;
        int dc[3] = {0, 0, 0};
        bool neighbour = true;
        for (int a = 0; a < dim; ++a) {
            const double p = xp[3 * i + a], q = xq[3 * i + a];
            wp |= nl_q10_axis(p, h) << (10 * a);
            wq |= nl_q10_axis(q, h) << (10 * a);
            const double d = floor(q / h) - floor(p / h);
            if (!(fabs(d) <= 1.0)) neighbour = false;
            dc[a] = (int)d;
        }
        pass[i] = !neighbour ? 2 : (nl_q10_pass(wp, wq, dc[0], dc[1], dc[2], dim) ? 1 : 0);
    }
    return SPHMW_OK;
}
// the 6-bit pre-test of the zrun cell order (the default): words as the cell-list gather writes
// them, the run constant as k_binary_build forms it
extern "C" int sphmw_pretest_pairs_q6(const double *xp, const double *xq, int64_t n, double h, int32_t dim,
                                      uint8_t *pass) {
    if (!xp || !xq || !pass || !(h > 0.0) || (dim != 2 && dim != 3)) return SPHMW_E_INVALID;
    for (int64_t i = 0; i < n; ++i) {
        int dc[3] = {0, 0, 0};
        bool neighbour = true;
        for (int a = 0; a < dim; ++a) {
            const double d = floor(xq[3 * i + a] / h) - floor(xp[3 * i + a] / h);
            if (!(fabs(d) <= 1.0)) neighbour = false;
            dc[a] = (int)d;
        }
        const long long phase = -7;  // any key_phase: the run-axis byte is taken modulo four cells
        const uint32_t wp = nl_q6_word(xp[3 * i], xp[3 * i + 1], xp[3 * i + 2], h, phase, dim);
        const uint32_t wq = nl_q6_word(xq[3 * i], xq[3 * i + 1], xq[3 * i + 2], h, phase, dim);
        const uint32_t K = nl_q6_run_const(wp, dc[0], dim == 3 ? dc[1] : 0);
        pass[i] = !neighbour ? 2 : (nl_q6_dist2(K, wq) > NL_Q6_R2MAX ? 0 : 1);
    }
    return SPHMW_OK;
}
// core.jl:72-81 replayed on index space (cell_list.cu sphmw_replay_swap_removal: what the whole-domain
// cell-list build and the open box of the slab transport both use): which survivors change their index
extern "C" int sphmw_swap_removal_moves(int64_t n, const int64_t *removed, int64_t k, int64_t *old_index,
                                        int64_t *new_index, int64_t *n_moves) {
    if (n < 0 || k < 0 || k > n || (k > 0 && !removed) || !n_moves) return SPHMW_E_INVALID;
    std::vector<uint32_t> rem(k), mo, mn;
    for (int64_t i = 0; i < k; ++i) {
        if (removed[i] < 0 || removed[i] >= n) return SPHMW_E_INVALID;
        rem[i] = (uint32_t)removed[i];
    }
    sphmw_replay_swap_removal(n, rem, mo, mn);
    *n_moves = (int64_t)mo.size();
    for (size_t i = 0; i < mo.size() && old_index && new_index; ++i) {
        old_index[i] = mo[i];
        new_index[i] = mn[i];
    }
    return SPHMW_OK;
}
extern "C" int sphmw_slab_column_sets(int32_t width, int32_t has_left, int32_t has_right, int32_t out[16]) {
    if (!out || width < 2 * GHOST_COLS + 2 * GHOST_COLS) return SPHMW_E_INVALID;
    const SlabCols sc = sphmw_slab_cols_of(width, has_left != 0, has_right != 0);
    const ColFilter *f[4] = {&sc.edge, &sc.interior, &sc.force_edge, &sc.force_interior};
    for (int k = 0; k < 4; ++k) {
        out[4 * k + 0] = f[k]->a0;
        out[4 * k + 1] = f[k]->a1;
        out[4 * k + 2] = f[k]->b0;
        out[4 * k + 3] = f[k]->b1;
    }
    return SPHMW_OK;
}

extern "C" int sphmw_count_pairs(sphmw_ctx *c, int32_t enable) {
    if (!c) return SPHMW_E_INVALID;
    c->count_pairs = enable != 0;
    return SPHMW_OK;
}
extern "C" int sphmw_pair_count(sphmw_ctx *c, int64_t *n) {
    if (!c || !n) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaMemcpyAsync(c->h_counters, c->d_counters, sizeof(unsigned long long),
                             cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    *n = (int64_t)c->h_counters[0];
    return SPHMW_OK;
}
