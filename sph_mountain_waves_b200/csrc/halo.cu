// x-slab halo exchange, device side (SURVEY.md §8e; the reference has no distributed path).
//
// A rank owns the global cell columns [slab_lo, slab_hi) and keeps Grid::ghost (2, or 3 with
// SPHMW_FLAG_GHOST3) ghost columns on each side.  Once per step, after the drift, k_halo_pack classifies every
// resident particle:
//   ghost of the previous exchange      -> dropped
//   owned, left the global box          -> dropped (counted as lost)
//   owned, now in a ghost column        -> MIGRANT record to that neighbour; kept here as a ghost
//   owned, in one of the two outermost owned columns -> GHOST record (a copy) to that neighbour
// The host moves the records between x-adjacent ranks (NCCL send/recv through
// torch.distributed, or any transport), k_halo_unpack appends what arrives, and the
// ordinary cell-list build sorts owned and ghost particles together.  Because the second
// ghost column makes the first one's density sum complete, ghost densities are recomputed
// locally and no second exchange is needed before the force pass.
#include <string.h>

#include "halo_record.cuh"
#include "sphmw_internal.h"

// cf: only the particles that sat in the selected columns BEFORE the drift (cellx is the
// column of the last cell list) are looked at — the overlapped step packs the edge columns
// while the interior is still in the force pass; cf.on == 0 looks at everybody.
template <int DIM, int KIND>
__global__ void k_halo_pack(Fields f, const uint32_t *__restrict__ idx, uint32_t *__restrict__ tag,
                            int64_t n, Grid g, int has_left, int has_right, double *buf_l,
                            double *buf_r, uint32_t cap, uint32_t *counters,
                            const uint32_t *__restrict__ cellx, ColFilter cf, uint32_t *__restrict__ lost_list,
                            uint32_t lost_cap, int carry_a) {
    constexpr int ROWS = halo_record_rows(KIND);
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    if (cf.on && !col_selected(cf, (int)cellx[p])) return;
    uint32_t t = tag[p];
    if (t != TAG_OWNED) {
        tag[p] = TAG_DEAD;
        return;
    }
    double x = f.s[S_X0][p], y = f.s[S_X1][p], z = DIM == 3 ? f.s[S_X2][p] : 0.0;
    bool inside = g.box[0] <= x && x <= g.box[3] && g.box[1] <= y && y <= g.box[4] &&
                  g.box[2] <= z && z <= g.box[5];
    if (!inside) {
        // left the GLOBAL box: removed, as create_cell_list! does (core.jl:60-66).  With an open box
        // (slab_comm.cu) its global index is kept, because the reference then moves the particles at
        // the end of sys.particles into the vacated slots (core.jl:72-81)
        tag[p] = TAG_DEAD;
        const uint32_t slot = atomicAdd(&counters[4], 1u);
        if (lost_list && slot < lost_cap) lost_list[1 + slot] = idx[p];
        return;
    }
    const long long W = g.lim[0];
    long long i = (long long)floor(x / g.h) - g.phase[0];  // local column
    int to_l = 0, to_r = 0;
    double kind = HALO_KIND_GHOST;
    const int G = g.ghost;
    if (i < G) {
        to_l = 1;
        kind = HALO_KIND_MIGRANT;
        tag[p] = (i >= 0 && has_left) ? TAG_GHOST : TAG_DEAD;
    } else if (i >= W - G) {
        to_r = 1;
        kind = HALO_KIND_MIGRANT;
        tag[p] = (i < W && has_right) ? TAG_GHOST : TAG_DEAD;
    } else {
        to_l = i < 2 * G;
        to_r = i >= W - 2 * G;
    }
    to_l = to_l && has_left;
    to_r = to_r && has_right;
    if (!to_l && !to_r) return;
    double rec[ROWS];
    halo_record_pack<DIM, KIND>(f, idx, p, x, y, z, kind, carry_a, rec);  // halo_record.cuh
    if (to_l) {
        uint32_t s = atomicAdd(&counters[0], 1u);
        if (kind == HALO_KIND_MIGRANT) atomicAdd(&counters[2], 1u);
        if (s < cap)
            for (int k = 0; k < ROWS; ++k) buf_l[(size_t)s * ROWS + k] = rec[k];
    }
    if (to_r) {
        uint32_t s = atomicAdd(&counters[1], 1u);
        if (kind == HALO_KIND_MIGRANT) atomicAdd(&counters[3], 1u);
        if (s < cap)
            for (int k = 0; k < ROWS; ++k) buf_r[(size_t)s * ROWS + k] = rec[k];
    }
}

template <int DIM, int KIND>
__global__ void k_halo_unpack(Fields f, uint32_t *__restrict__ idx, uint32_t *__restrict__ tag,
                              int64_t first, const double *__restrict__ buf, int64_t cnt, int carry_a) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const double *rec = buf + (size_t)t * halo_record_rows(KIND);
    halo_record_unpack<DIM, KIND>(f, idx, tag, first + t, rec, carry_a);  // halo_record.cuh
}

static const int CARRIED[] = {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2, S_M, S_H, S_RHO, S_RHO_P, S_TYPE};

// 0: rows 8/9 of a record are rho, rho'; 1: A; 2: A and A_bg (contexts that hold those fields)
static int carry_a(const sphmw_ctx *c) {
    if (!c->allocated[S_A]) return 0;
    return c->allocated[S_A_BG] ? 2 : 1;
}

// The record kind of a context's halo exchange (halo_record.cuh): ADIABATIC when the context holds the
// entropy S (the adiabatic flow driver), BASE otherwise.  Fixed at its first use: the first pack, unpack
// or library-transport exchange, or sphmw_halo_record_width — a caller sizes its record buffers by that
// answer, so a later pack must not write wider records into them.  Records of another width are never
// sent; a context whose fields would change the kind later fails instead.  (sphmw_comm_init does not
// decide it: a communicator may exist before the fields are uploaded.)
int sphmw_halo_kind(sphmw_ctx *c, int *kind) {
    const int want = c->allocated[S_ENT] ? HALO_REC_ADIABATIC : HALO_REC_BASE;
    if (c->halo_kind < 0) c->halo_kind = want;
    if (c->halo_kind != want) {
        sphmw_set_error("halo: the context's fields now call for %d-row records, its exchange was set up with %d rows",
                        halo_record_rows(want), halo_record_rows(c->halo_kind));
        return SPHMW_E_STATE;
    }
    *kind = want;
    return SPHMW_OK;
}

static int ensure_carried(sphmw_ctx *c, int kind) {
    for (int s : CARRIED) {
        if (c->grid.dim == 2 && (s == S_X2 || s == S_V2)) continue;
        TRY(sphmw_ensure_slot(c, s));
        if (c->stale[s]) { sphmw_set_error("halo: carried field is stale"); return SPHMW_E_STATE; }
    }
    for (int s : {S_A, S_A_BG})
        if (c->allocated[s] && c->stale[s]) { sphmw_set_error("halo: carried field is stale"); return SPHMW_E_STATE; }
    if (kind == HALO_REC_ADIABATIC)
        for (int s : {S_ENT, S_P, S_T, S_TH}) {
            TRY(sphmw_ensure_slot(c, s));
            if (c->stale[s]) { sphmw_set_error("halo: carried field is stale"); return SPHMW_E_STATE; }
        }
    return SPHMW_OK;
}

// the base record (contexts without the entropy S); sphmw_halo_record_width gives a context's own
extern "C" int sphmw_halo_record_doubles(void) { return HALO_RECORD; }

extern "C" int sphmw_halo_record_width(sphmw_ctx *c, int32_t *doubles) {
    if (!c || !doubles) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    int kind = 0;
    TRY(sphmw_halo_kind(c, &kind));
    *doubles = halo_record_rows(kind);
    return SPHMW_OK;
}

// row 0 of a message (slab_comm.cu): {records, migrants among them, record width}; the records follow
__global__ void k_halo_header(const uint32_t *__restrict__ counters, double *msg_l, double *msg_r, int width) {
    if (threadIdx.x == 0 && msg_l) {
        msg_l[0] = (double)counters[0];
        msg_l[1] = (double)counters[2];
        msg_l[2] = (double)width;
    }
    if (threadIdx.x == 1 && msg_r) {
        msg_r[0] = (double)counters[1];
        msg_r[1] = (double)counters[3];
        msg_r[2] = (double)width;
    }
}

#define HALO_LAUNCH(KERNEL, BLOCKS, ...)                                                                  \
    do {                                                                                              \
        if (c->grid.dim == 2) {                                                                       \
            if (kind == HALO_REC_ADIABATIC) KERNEL<2, HALO_REC_ADIABATIC><<<BLOCKS, 256, 0, c->stream>>>(__VA_ARGS__); \
            else KERNEL<2, HALO_REC_BASE><<<BLOCKS, 256, 0, c->stream>>>(__VA_ARGS__);                \
        } else {                                                                                      \
            if (kind == HALO_REC_ADIABATIC) KERNEL<3, HALO_REC_ADIABATIC><<<BLOCKS, 256, 0, c->stream>>>(__VA_ARGS__); \
            else KERNEL<3, HALO_REC_BASE><<<BLOCKS, 256, 0, c->stream>>>(__VA_ARGS__);                \
        }                                                                                             \
    } while (0)

// enqueue: classify + pack (all particles, or the edge columns of an overlapped step out of the
// alt buffers), then read the counters back asynchronously and mark the point with an event
// msg_left/right: when not null, the record counts are also written, on the device, to row 0 of
// these messages (the records themselves start one row further, at dev_buf_*)
static int pack_enqueue(sphmw_ctx *c, double *dev_buf_left, double *dev_buf_right, int64_t cap_records,
                        bool edge_only, double *msg_left = nullptr, double *msg_right = nullptr) {
    int kind = 0;
    TRY(sphmw_halo_kind(c, &kind));
    TRY(ensure_carried(c, kind));
    // what the next cell-list build will find dead: last exchange's ghosts and migrants, plus
    // the particles this pack is about to drop (added by pack_collect)
    c->slab_dead_expected = c->n - c->n_owned;
    const int has_left = dev_buf_left != nullptr, has_right = dev_buf_right != nullptr;
    // [0..4] belong to this pack; [5] (escapes counted by the previous interior advance) is read
    // together with them and cleared afterwards
    CUDA_TRY(cudaMemsetAsync(c->halo_counters, 0, sizeof(uint32_t) * 5, c->stream));
    if (c->n > 0) {
        Fields view = c->cur;
        ColFilter cf{0, 0, 0, 0, 0, 0};
        if (edge_only) {
            for (int s : {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2}) view.s[s] = c->alt.s[s];
            cf = sphmw_slab_cols(c).edge;
        }
        TIMED(c, "halo_pack");
        HALO_LAUNCH(k_halo_pack, grid_for(c->n, 256), view, c->idx, c->tag, c->n, c->grid, has_left, has_right, dev_buf_left,
                    dev_buf_right, (uint32_t)cap_records, c->halo_counters, c->cellx, cf, c->lost_list, SLAB_LOST_CAP,
                    carry_a(c));
        CUDA_TRY(cudaGetLastError());
    }
    if (c->lost_list)  // word 0 of the list: how many particles this pack dropped
        CUDA_TRY(cudaMemcpyAsync(c->lost_list, c->halo_counters + 4, sizeof(uint32_t), cudaMemcpyDeviceToDevice, c->stream));
    if (msg_left || msg_right) {
        k_halo_header<<<1, 32, 0, c->stream>>>(c->halo_counters, msg_left, msg_right, halo_record_rows(kind));
        c->launches += 1;
    }
    TRY(sphmw_publish_words(c, c->halo_counters, c->h_halo_counters, 8, c->stream));
    CUDA_TRY(cudaMemsetAsync(c->halo_counters + 5, 0, sizeof(uint32_t), c->stream));
    CUDA_TRY(cudaEventRecord(c->pack_event, c->stream));
    return SPHMW_OK;
}
int sphmw_halo_pack_enqueue(sphmw_ctx *c, double *msg_left, double *msg_right, int64_t cap_records, bool edge_only) {
    int kind = 0;
    TRY(sphmw_halo_kind(c, &kind));
    const int W = halo_record_rows(kind);
    return pack_enqueue(c, msg_left ? msg_left + W : nullptr, msg_right ? msg_right + W : nullptr,
                        cap_records, edge_only, msg_left, msg_right);
}

static int pack_collect(sphmw_ctx *c, int64_t cap_records, int64_t counts[5], bool wait = true) {
    if (wait) CUDA_TRY(cudaEventSynchronize(c->pack_event));
    for (int k = 0; k < 5; ++k) counts[k] = c->h_halo_counters[k];
    if (c->h_halo_counters[5] != 0) {
        sphmw_set_error("overlapped halo exchange: %u particle(s) crossed more than one cell column in a "
                        "step (it assumes |v| dt < h); use the plain step_phase 0/1 sequence",
                        c->h_halo_counters[5]);
        return SPHMW_E_STATE;
    }
    if (counts[0] > cap_records || counts[1] > cap_records) {
        sphmw_set_error("halo buffer too small: %lld/%lld records for capacity %lld",
                        (long long)counts[0], (long long)counts[1], (long long)cap_records);
        return SPHMW_E_CAPACITY;
    }
    c->n_owned -= counts[2] + counts[3] + counts[4];
    c->slab_dead_expected += counts[4];
    c->slab_dead_known = true;
    c->cell_list_valid = false;
    return SPHMW_OK;
}
// the counters are already on the host (the caller waited for something later in the stream)
int sphmw_halo_pack_collect_nowait(sphmw_ctx *c, int64_t cap_records, int64_t counts[5]) {
    return pack_collect(c, cap_records, counts, false);
}

// counts[0..4] = records to the left, to the right, migrants among them (left, right), lost.
// Blocks (reads the counters back).
extern "C" int sphmw_halo_pack(sphmw_ctx *c, double *dev_buf_left, double *dev_buf_right,
                               int64_t cap_records, int64_t counts[5]) {
    if (!c || !counts) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("halo_pack: context has no slab"); return SPHMW_E_STATE; }
    if (c->overlap_stage != 0) { sphmw_set_error("halo_pack: an overlapped step is in flight"); return SPHMW_E_STATE; }
    TRY(pack_enqueue(c, dev_buf_left, dev_buf_right, cap_records, false));
    return pack_collect(c, cap_records, counts);
}

// The two halves of sphmw_halo_pack for the overlapped step (step_phase 2 -> pack_begin ->
// step_phase 3 -> pack_finish): begin only enqueues, so the interior force pass can be queued
// behind it before the host waits for the counts.
extern "C" int sphmw_halo_pack_begin(sphmw_ctx *c, double *dev_buf_left, double *dev_buf_right,
                                     int64_t cap_records) {
    if (!c) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("halo_pack_begin: context has no slab"); return SPHMW_E_STATE; }
    if (c->overlap_stage != 1) { sphmw_set_error("halo_pack_begin: call step_phase 2 first"); return SPHMW_E_STATE; }
    TRY(pack_enqueue(c, dev_buf_left, dev_buf_right, cap_records, true));
    c->overlap_stage = 2;
    return SPHMW_OK;
}
extern "C" int sphmw_halo_pack_finish(sphmw_ctx *c, int64_t cap_records, int64_t counts[5]) {
    if (!c || !counts) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->overlap_stage != 3) { sphmw_set_error("halo_pack_finish: call step_phase 3 first"); return SPHMW_E_STATE; }
    c->overlap_stage = 0;
    return pack_collect(c, cap_records, counts);
}
// make another stream (the transport's) wait for the packed records
extern "C" int sphmw_halo_pack_wait(sphmw_ctx *c, void *cuda_stream) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)cuda_stream, c->pack_event, 0));
    return SPHMW_OK;
}

// Appends `count` records; `n_migrants` of them (the sender's count) become owned.
extern "C" int sphmw_halo_unpack(sphmw_ctx *c, const double *dev_buf, int64_t count,
                                 int64_t n_migrants) {
    if (!c) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("halo_unpack: context has no slab"); return SPHMW_E_STATE; }
    if (count <= 0) return SPHMW_OK;
    if (c->n + count > c->cap) {
        sphmw_set_error("halo_unpack: %lld + %lld particles exceed capacity %lld", (long long)c->n,
                        (long long)count, (long long)c->cap);
        return SPHMW_E_CAPACITY;
    }
    int kind = 0;
    TRY(sphmw_halo_kind(c, &kind));
    TRY(ensure_carried(c, kind));
    {
        TIMED(c, "halo_unpack");
        HALO_LAUNCH(k_halo_unpack, grid_for(count, 256), c->cur, c->idx, c->tag, c->n, dev_buf, count, carry_a(c));
        CUDA_TRY(cudaGetLastError());
    }
    c->n += count;
    c->n_owned += n_migrants;
    c->cell_list_valid = false;
    return SPHMW_OK;
}

extern "C" int sphmw_slab_counts(sphmw_ctx *c, int64_t *n_resident, int64_t *n_owned) {
    if (!c) return SPHMW_E_INVALID;
    if (n_resident) *n_resident = c->n;
    if (n_owned) *n_owned = c->n_owned;
    return SPHMW_OK;
}

// ---- physical-order access (slab contexts carry GLOBAL particle indices, so the
// index-ordered upload/download of whole-domain contexts does not apply) -----------
__global__ void k_set_index(uint32_t *idx, const long long *g, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (uint32_t)g[i];
}
__global__ void k_get_index(const uint32_t *idx, const uint32_t *tag, long long *g, int *t, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) {
        g[i] = idx[i];
        t[i] = (int)tag[i];
    }
}

// global index of every resident particle, in the current physical order
extern "C" int sphmw_set_index(sphmw_ctx *c, const int64_t *global_idx, int64_t n) {
    if (!c || !global_idx) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("set_index: context has no slab"); return SPHMW_E_STATE; }
    if (n != c->n) { sphmw_set_error("set_index: n mismatch"); return SPHMW_E_INVALID; }
    if (n == 0) return SPHMW_OK;
    long long *d = (long long *)c->staging;
    CUDA_TRY(cudaMemcpyAsync(d, global_idx, sizeof(int64_t) * n, cudaMemcpyDefault, c->stream));
    k_set_index<<<grid_for(n, 256), 256, 0, c->stream>>>(c->idx, d, n);
    c->launches += 1;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

extern "C" int sphmw_download_index(sphmw_ctx *c, int64_t *global_idx, int32_t *tag, int64_t n) {
    if (!c || !global_idx || !tag) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    if (n != c->n) { sphmw_set_error("download_index: n mismatch"); return SPHMW_E_INVALID; }
    if (n == 0) return SPHMW_OK;
    long long *d = (long long *)c->staging;
    int *dt = (int *)(c->staging + c->cap);
    k_get_index<<<grid_for(n, 256), 256, 0, c->stream>>>(c->idx, c->tag, d, dt, n);
    c->launches += 1;
    CUDA_TRY(cudaMemcpyAsync(global_idx, d, sizeof(int64_t) * n, cudaMemcpyDefault, c->stream));
    CUDA_TRY(cudaMemcpyAsync(tag, dt, sizeof(int32_t) * n, cudaMemcpyDefault, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}

// one scalar component in physical order (component-major for vectors)
extern "C" int sphmw_download_raw(sphmw_ctx *c, const char *field, double *buf, int64_t n,
                                  int32_t ncomp) {
    if (!c || !field || !buf) return SPHMW_E_INVALID;
    CUDA_TRY(cudaSetDevice(c->device));
    const FieldDesc *d = sphmw_find_field(field);
    if (!d) { sphmw_set_error("Variable %s does not exist!", field); return SPHMW_E_UNKNOWN_FIELD; }
    if (ncomp != d->ncomp || n != c->n) { sphmw_set_error("download_raw: shape mismatch"); return SPHMW_E_INVALID; }
    for (int k = 0; k < ncomp; ++k) {
        int slot = d->slot + k;
        if (c->allocated[slot] && c->stale[slot]) TRY(sphmw_materialize(c, slot));
        if (!c->allocated[slot] || (c->grid.dim == 2 && ncomp == 3 && k == 2)) {
            CUDA_TRY(cudaMemsetAsync(c->staging, 0, sizeof(double) * n, c->stream));
            CUDA_TRY(cudaMemcpyAsync(buf + (int64_t)k * n, c->staging, sizeof(double) * n,
                                     cudaMemcpyDefault, c->stream));
        } else {
            CUDA_TRY(cudaMemcpyAsync(buf + (int64_t)k * n, c->cur.s[slot], sizeof(double) * n,
                                     cudaMemcpyDefault, c->stream));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SPHMW_OK;
}
