// x-slab halo transport inside the library (SURVEY.md §8b "multi-GPU is internal to the ctx",
// §8e): ncclSend/ncclRecv between x-adjacent ranks on a second, high-priority CUDA stream,
// driven by sphmw_step / sphmw_create_cell_list themselves, so that a single-threaded caller —
// the reference's caller is one (src/core.jl:125-142) — steps a slab context with the very calls
// it uses on one GPU.
//
// One exchange = ONE ncclGroup per step.  A message is a fixed number of rows of `width` doubles (the
// context's halo record, halo_record.cuh: 13, or 17 for the adiabatic flow driver) agreed between the
// two ranks; row 0 is written on the device by the pack ({records, migrants, width}; the receiver
// checks the width against its own), so no count has to travel first and the sender's host never has to
// know it before the send is queued.  The sizes are agreed once (a header-only round at the first
// exchange: count * 1.12 + 1024 rows) and renegotiated, with one extra blocking round, only when a
// count outgrows them.  Per step the host waits once — for the two received headers, which arrive
// while the interior force pass is still running on the main stream — and the cell-list build of
// a slab context no longer waits at all (cell_list.cu: the dead count follows from the pack).
//
// NCCL is loaded with dlopen at sphmw_comm_init (libnccl.so.2 — inside a PyTorch process that is
// the copy torch already loaded), so libsphmw.so itself has no link-time dependency on it.
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "halo_record.cuh"
#include "sphmw_internal.h"

struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi g_nccl;

static int nccl_load() {
    if (g_nccl.lib) return SPHMW_OK;
    void *lib = nullptr;
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
        lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) {
        sphmw_set_error("NCCL is not available: %s", dlerror());
        return SPHMW_E_UNSUPPORTED_OP;
    }
#define NCCL_SYM(field, sym)                                                    \
    *(void **)(&g_nccl.field) = dlsym(lib, sym);                                \
    if (!g_nccl.field) {                                                        \
        sphmw_set_error("NCCL library lacks %s", sym);                          \
        return SPHMW_E_UNSUPPORTED_OP;                                          \
    }
    NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    NCCL_SYM(CommInitRank, "ncclCommInitRank")
    NCCL_SYM(CommDestroy, "ncclCommDestroy")
    NCCL_SYM(Send, "ncclSend")
    NCCL_SYM(Recv, "ncclRecv")
    NCCL_SYM(AllGather, "ncclAllGather")
    NCCL_SYM(AllReduce, "ncclAllReduce")
    NCCL_SYM(GroupStart, "ncclGroupStart")
    NCCL_SYM(GroupEnd, "ncclGroupEnd")
    NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef NCCL_SYM
    g_nccl.lib = lib;
    return SPHMW_OK;
}

#define NCCL_TRY(expr)                                                                          \
    do {                                                                                        \
        ncclResult_t _r = (expr);                                                               \
        if (_r != ncclSuccess) {                                                                \
            sphmw_set_error("%s failed: %s (%s:%d)", #expr, g_nccl.GetErrorString(_r), __FILE__, __LINE__); \
            return SPHMW_E_CUDA;                                                                \
        }                                                                                       \
    } while (0)

struct SlabComm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    bool has[2] = {false, false};  // a neighbour on the left / right
    int peer[2] = {-1, -1};
    cudaStream_t stream = nullptr;  // high priority: the transfer runs beside the interior force pass
    int64_t cap = 0;                // records a message buffer holds (+ the header row)
    int width = 0;                  // doubles per row: the context's record width; 0 until the first exchange
    double *send[2] = {nullptr, nullptr}, *recv[2] = {nullptr, nullptr};
    int64_t send_rows[2] = {0, 0}, recv_rows[2] = {0, 0};  // agreed message sizes (0: not yet)
    double *h_head = nullptr;       // pinned: the two received headers
    cudaEvent_t recv_event = nullptr;
    int64_t exchanges = 0, renegotiations = 0;
    int64_t lost = 0;
    // open box (sphmw_comm_open_box): particles may leave the global bounding box; every exchange
    // gathers the dropped global indices of all ranks and replays the reference's swap-from-end
    // renumbering (core.jl:72-81) on every rank
    bool open_box = false;
    int64_t n_global = -1;           // length of sys.particles; found with an all-reduce at the first exchange
    uint32_t *gather_dev = nullptr;  // world x (1 + SLAB_LOST_CAP) words
    uint32_t *gather_host = nullptr; // pinned
    long long *count_dev = nullptr;  // all-reduce scratch
    uint32_t *conv_list = nullptr;   // inflow: [0] count, [1..] global indices of this rank's converting particles
    uint32_t *conv_pos = nullptr;    // ... and their physical positions; then (pos, new index) pairs for the spawn
    uint32_t *h_conv = nullptr;      // pinned scratch, 2 * SLAB_LOST_CAP words
    int64_t renumbered = 0;          // survivors that changed their index so far
};

extern "C" int sphmw_comm_unique_id(void *id128) {
    if (!id128) return SPHMW_E_INVALID;
    TRY(nccl_load());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NCCL_TRY(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
    return SPHMW_OK;
}

void sphmw_comm_free(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    if (!m) return;
    if (m->stream) cudaStreamSynchronize(m->stream);
    if (m->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(m->comm);
    for (int s = 0; s < 2; ++s) {
        cudaFree(m->send[s]);
        cudaFree(m->recv[s]);
    }
    if (m->h_head) cudaFreeHost(m->h_head);
    if (m->gather_host) cudaFreeHost(m->gather_host);
    cudaFree(m->gather_dev);
    cudaFree(m->count_dev);
    cudaFree(m->conv_list);
    cudaFree(m->conv_pos);
    if (m->h_conv) cudaFreeHost(m->h_conv);
    if (m->recv_event) cudaEventDestroy(m->recv_event);
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
    c->comm = nullptr;
}

// rank r of `world` ranks holds the r-th slab from the left; halo_capacity = records one message
// buffer can hold — the SAME value on every rank (message sizes are derived from it on both ends).
// Collective: every rank of the communicator calls it.
extern "C" int sphmw_comm_init(sphmw_ctx *c, int32_t rank, int32_t world, const void *id128, int64_t halo_capacity) {
    if (!c || !id128 || world < 1 || rank < 0 || rank >= world || halo_capacity <= 0) {
        sphmw_set_error("comm_init: bad argument");
        return SPHMW_E_INVALID;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("comm_init: context has no slab"); return SPHMW_E_STATE; }
    if (c->comm) { sphmw_set_error("comm_init: context already has a communicator"); return SPHMW_E_STATE; }
    TRY(nccl_load());
    SlabComm *m = new SlabComm();
    c->comm = m;
    m->rank = rank;
    m->world = world;
    m->has[0] = c->slab_lo > 0;
    m->has[1] = c->slab_hi < c->global_cols;
    if (m->has[0] != (rank > 0) || m->has[1] != (rank < world - 1)) {
        sphmw_set_error("comm_init: rank %d of %d does not match the slab [%lld,%lld) of %lld columns", rank, world,
                        (long long)c->slab_lo, (long long)c->slab_hi, (long long)c->global_cols);
        sphmw_comm_free(c);
        return SPHMW_E_INVALID;
    }
    m->peer[0] = rank - 1;
    m->peer[1] = rank + 1;
    m->cap = halo_capacity;
    int rc = [&]() -> int {
        ncclUniqueId id;
        memcpy(&id, id128, sizeof(id));
        NCCL_TRY(g_nccl.CommInitRank(&m->comm, world, id, rank));
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&m->stream, cudaStreamNonBlocking, hi));
        CUDA_TRY(cudaEventCreateWithFlags(&m->recv_event, cudaEventDisableTiming));
        return SPHMW_OK;
    }();
    if (rc != SPHMW_OK) sphmw_comm_free(c);
    return rc;
}

// The message buffers and the pinned header rows, made at the first exchange: the record width follows
// from the fields the context holds (halo.cu sphmw_halo_kind), and a caller may create the communicator
// before it uploads them (the Julia shim does: sphmw_create, sphmw_comm_init, then the upload).
static int comm_buffers(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    if (m->width > 0) return SPHMW_OK;
    int kind = 0;
    TRY(sphmw_halo_kind(c, &kind));
    const int width = halo_record_rows(kind);
    CUDA_TRY(cudaMallocHost(&m->h_head, sizeof(double) * 2 * width));
    for (int s = 0; s < 2; ++s)
        if (m->has[s]) {
            const size_t bytes = sizeof(double) * width * (size_t)(m->cap + 1);
            CUDA_TRY(cudaMalloc(&m->send[s], bytes));
            CUDA_TRY(cudaMalloc(&m->recv[s], bytes));
            CUDA_TRY(cudaMemsetAsync(m->send[s], 0, bytes, c->stream));
            CUDA_TRY(cudaMemsetAsync(m->recv[s], 0, bytes, c->stream));
        }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    m->width = width;
    return SPHMW_OK;
}

extern "C" int sphmw_comm_info(sphmw_ctx *c, int64_t out[6]) {
    if (!c || !out) return SPHMW_E_INVALID;
    for (int k = 0; k < 6; ++k) out[k] = 0;
    if (!c->comm) return SPHMW_OK;
    out[0] = c->comm->world;
    out[1] = c->comm->exchanges;
    out[2] = c->comm->renegotiations;
    out[3] = c->comm->send_rows[0] + c->comm->send_rows[1];
    out[4] = c->comm->lost;
    out[5] = c->comm->cap;
    return SPHMW_OK;
}

static int64_t rows_for(int64_t count) { return 1 + count + count / 8 + 1024; }

// one group: `rows[s]` rows to/from each neighbour; the received headers follow to pinned memory
static int comm_round(sphmw_ctx *c, const int64_t srows[2], const int64_t rrows[2]) {
    SlabComm *m = c->comm;
    NCCL_TRY(g_nccl.GroupStart());
    for (int s = 0; s < 2; ++s) {
        if (!m->has[s]) continue;
        if (srows[s] > 0)
            NCCL_TRY(g_nccl.Send(m->send[s], (size_t)srows[s] * m->width, ncclDouble, m->peer[s], m->comm, m->stream));
        if (rrows[s] > 0)
            NCCL_TRY(g_nccl.Recv(m->recv[s], (size_t)rrows[s] * m->width, ncclDouble, m->peer[s], m->comm, m->stream));
    }
    NCCL_TRY(g_nccl.GroupEnd());
    for (int s = 0; s < 2; ++s)
        if (m->has[s] && rrows[s] > 0)  // (a kernel store, not a copy-engine transfer: see sphmw_publish_words)
            TRY(sphmw_publish_words(c, (const uint32_t *)m->recv[s], (uint32_t *)(m->h_head + s * m->width), 2 * m->width,
                                    m->stream));
    CUDA_TRY(cudaEventRecord(m->recv_event, m->stream));
    return SPHMW_OK;
}

// records packed (pack_event recorded on the main stream) -> neighbours -> unpacked.
// The host waits once, for the received headers.
static int comm_transfer_and_unpack(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    CUDA_TRY(cudaStreamWaitEvent(m->stream, c->pack_event, 0));
    const bool agreed = (!m->has[0] || m->send_rows[0] > 0) && (!m->has[1] || m->send_rows[1] > 0);
    const int64_t one[2] = {1, 1};
    if (agreed) TRY(comm_round(c, m->send_rows, m->recv_rows));
    else TRY(comm_round(c, one, one));  // first exchange: headers only
    CUDA_TRY(cudaEventSynchronize(m->recv_event));
    // the pack's counters were copied to the host before pack_event
    int64_t counts[5];
    TRY(sphmw_halo_pack_collect_nowait(c, m->cap, counts));
    m->lost += counts[4];
    int64_t in_count[2] = {0, 0}, in_migr[2] = {0, 0};
    for (int s = 0; s < 2; ++s)
        if (m->has[s]) {
            const double *head = m->h_head + s * m->width;
            if (head[2] != (double)m->width) {
                sphmw_set_error("halo message from rank %d has %g-double records, this rank's have %d (the ranks hold "
                                "different particle fields)", m->peer[s], head[2], m->width);
                return SPHMW_E_STATE;
            }
            in_count[s] = (int64_t)head[0];
            in_migr[s] = (int64_t)head[1];
            if (in_count[s] > m->cap) {
                sphmw_set_error("halo message of %lld records exceeds the buffer capacity %lld", (long long)in_count[s],
                                (long long)m->cap);
                return SPHMW_E_CAPACITY;
            }
        }
    // a count that does not fit the agreed size (or no size yet): both ends see it — the sender in
    // its own counters, the receiver in the header — and repeat that direction with a new size
    int64_t srows[2] = {0, 0}, rrows[2] = {0, 0};
    bool again = false;
    for (int s = 0; s < 2; ++s) {
        if (!m->has[s]) continue;
        if (counts[s] + 1 > m->send_rows[s]) {
            m->send_rows[s] = std::min<int64_t>(rows_for(counts[s]), m->cap + 1);
            srows[s] = m->send_rows[s];
            again = true;
        }
        if (in_count[s] + 1 > m->recv_rows[s]) {
            m->recv_rows[s] = std::min<int64_t>(rows_for(in_count[s]), m->cap + 1);
            rrows[s] = m->recv_rows[s];
            again = true;
        }
    }
    if (again) {
        m->renegotiations += agreed ? 1 : 0;
        TRY(comm_round(c, srows, rrows));
        CUDA_TRY(cudaEventSynchronize(m->recv_event));
    }
    m->exchanges += 1;
    // the main stream appends what arrived (the transfer is complete: the host has waited for it)
    for (int s = 0; s < 2; ++s)
        if (m->has[s] && in_count[s] > 0)
            TRY(sphmw_halo_unpack(c, m->recv[s] + m->width, in_count[s], in_migr[s]));
    return SPHMW_OK;
}

// ---- open box -----------------------------------------------------------------------------------
// ≙ the removal part of create_cell_list! (core.jl:60-81) on a slab decomposition.  Collective.
// After it every exchange is followed by the renumbering below and sphmw_step runs the plain
// schedule (the overlapped one packs the edge columns before the interior has drifted, so it
// cannot see an interior particle leave through the top or the sides of the box).
extern "C" int sphmw_comm_open_box(sphmw_ctx *c, int32_t on) {
    if (!c || !c->comm) { sphmw_set_error("comm_open_box: context has no communicator (sphmw_comm_init)"); return SPHMW_E_STATE; }
    CUDA_TRY(cudaSetDevice(c->device));
    SlabComm *m = c->comm;
    m->open_box = on != 0;
    if (m->open_box && !m->gather_dev) {
        const size_t words = (size_t)m->world * (1 + SLAB_LOST_CAP);
        CUDA_TRY(cudaMalloc(&m->gather_dev, sizeof(uint32_t) * words));
        CUDA_TRY(cudaMallocHost(&m->gather_host, sizeof(uint32_t) * words));
        CUDA_TRY(cudaMalloc(&m->count_dev, sizeof(long long) * 2));
        CUDA_TRY(cudaMalloc(&m->conv_list, sizeof(uint32_t) * (1 + SLAB_LOST_CAP)));
        CUDA_TRY(cudaMalloc(&m->conv_pos, sizeof(uint32_t) * 2 * SLAB_LOST_CAP));
        CUDA_TRY(cudaMallocHost(&m->h_conv, sizeof(uint32_t) * 2 * SLAB_LOST_CAP));
        CUDA_TRY(cudaMalloc(&c->lost_list, sizeof(uint32_t) * (1 + SLAB_LOST_CAP)));
        CUDA_TRY(cudaMemsetAsync(c->lost_list, 0, sizeof(uint32_t) * (1 + SLAB_LOST_CAP), c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    return SPHMW_OK;
}

// idx[p] is looked up in the sorted list of indices that move (a handful per step)
__global__ void k_renumber_sorted(uint32_t *__restrict__ idx, int64_t n, const uint32_t *__restrict__ mv_old,
                                  const uint32_t *__restrict__ mv_new, int m) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t id = idx[p];
    int lo = 0, hi = m;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (mv_old[mid] < id) lo = mid + 1;
        else hi = mid;
    }
    if (lo < m && mv_old[lo] == id) idx[p] = mv_new[lo];
}

// length of sys.particles = the owned particles of all ranks (called when nothing is in flight)
static int comm_count_global(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    const long long mine = c->n_owned;
    CUDA_TRY(cudaMemcpyAsync(m->count_dev, &mine, sizeof(mine), cudaMemcpyHostToDevice, m->stream));
    NCCL_TRY(g_nccl.AllReduce(m->count_dev, m->count_dev + 1, 1, ncclInt64, ncclSum, m->comm, m->stream));
    long long total = 0;
    CUDA_TRY(cudaMemcpyAsync(&total, m->count_dev + 1, sizeof(total), cudaMemcpyDeviceToHost, m->stream));
    CUDA_TRY(cudaStreamSynchronize(m->stream));
    m->n_global = total;
    return SPHMW_OK;
}

// after an exchange: which particles did the ranks drop, and who moves into their slots
static int comm_renumber_lost(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    const size_t block = 1 + SLAB_LOST_CAP;
    // (the comm stream has waited for the pack; the lists were complete before pack_event)
    NCCL_TRY(g_nccl.AllGather(c->lost_list, m->gather_dev, block, ncclUint32, m->comm, m->stream));
    CUDA_TRY(cudaMemcpyAsync(m->gather_host, m->gather_dev, sizeof(uint32_t) * block * m->world, cudaMemcpyDeviceToHost,
                             m->stream));
    CUDA_TRY(cudaStreamSynchronize(m->stream));
    std::vector<uint32_t> removed;
    for (int r = 0; r < m->world; ++r) {
        const uint32_t *b = m->gather_host + (size_t)r * block;
        if (b[0] > SLAB_LOST_CAP) {
            sphmw_set_error("open box: rank %d lost %u particles in one step (at most %u are tracked)", r, b[0], SLAB_LOST_CAP);
            return SPHMW_E_CAPACITY;
        }
        removed.insert(removed.end(), b + 1, b + 1 + b[0]);
    }
    if (removed.empty()) return SPHMW_OK;
    std::vector<uint32_t> mo, mn;
    sphmw_replay_swap_removal(m->n_global, removed, mo, mn);
    m->n_global -= (int64_t)removed.size();
    const int64_t k = (int64_t)mo.size();
    if (k == 0 || c->n == 0) return SPHMW_OK;
    std::vector<std::pair<uint32_t, uint32_t>> mv(k);
    for (int64_t i = 0; i < k; ++i) mv[i] = {mo[i], mn[i]};
    std::sort(mv.begin(), mv.end());
    for (int64_t i = 0; i < k; ++i) {
        mo[i] = mv[i].first;
        mn[i] = mv[i].second;
    }
    if (k > c->mv_cap) {
        cudaFree(c->mv_old);
        cudaFree(c->mv_new);
        c->mv_old = c->mv_new = nullptr;
        c->mv_cap = k * 2;
        CUDA_TRY(cudaMalloc(&c->mv_old, sizeof(uint32_t) * c->mv_cap));
        CUDA_TRY(cudaMalloc(&c->mv_new, sizeof(uint32_t) * c->mv_cap));
    }
    CUDA_TRY(cudaMemcpyAsync(c->mv_old, mo.data(), sizeof(uint32_t) * k, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->mv_new, mn.data(), sizeof(uint32_t) * k, cudaMemcpyHostToDevice, c->stream));
    {
        TIMED(c, "slab_renumber");
        k_renumber_sorted<<<grid_for(c->n, 256), 256, 0, c->stream>>>(c->idx, c->n, c->mv_old, c->mv_new, (int)k);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // mo/mn must outlive the copies
    m->renumbered += k;
    return SPHMW_OK;
}

// ≙ add_new_particles!(sys) (isothermal_flow_witch.jl:175-186; adiabatic_flow_witch.jl:197-208 with
// `adiabatic`) on a slab decomposition.  The
// reference's loop runs over sys.particles in index order and appends one successor per converting
// INFLOW particle, so successor k gets index N + k where k counts the converting particles of ALL
// ranks with a smaller index: every rank contributes its list (one all-gather per step), the merged
// list is sorted on every host, and each rank builds the successors of its own particles with the
// indices that order gives them.  *n_added (optional): successors made on all ranks.
static int comm_flow_spawn(sphmw_ctx *c, bool adiabatic, int64_t *n_added = nullptr) {
    SlabComm *m = c->comm;
    if (n_added) *n_added = 0;
    if (m->n_global < 0) TRY(comm_count_global(c));
    const size_t block = 1 + SLAB_LOST_CAP;
    TRY(sphmw_flow_collect_slab(c, m->conv_list, m->conv_pos, SLAB_LOST_CAP, adiabatic));
    CUDA_TRY(cudaEventRecord(c->pack_event, c->stream));
    CUDA_TRY(cudaStreamWaitEvent(m->stream, c->pack_event, 0));
    NCCL_TRY(g_nccl.AllGather(m->conv_list, m->gather_dev, block, ncclUint32, m->comm, m->stream));
    CUDA_TRY(cudaMemcpyAsync(m->gather_host, m->gather_dev, sizeof(uint32_t) * block * m->world, cudaMemcpyDeviceToHost,
                             m->stream));
    CUDA_TRY(cudaStreamSynchronize(m->stream));
    std::vector<uint32_t> all;
    for (int r = 0; r < m->world; ++r) {
        const uint32_t *b = m->gather_host + (size_t)r * block;
        if (b[0] > SLAB_LOST_CAP) {
            sphmw_set_error("inflow: rank %d converts %u particles in one step (at most %u are tracked)", r, b[0], SLAB_LOST_CAP);
            return SPHMW_E_CAPACITY;
        }
        all.insert(all.end(), b + 1, b + 1 + b[0]);
    }
    if (all.empty()) return SPHMW_OK;
    std::sort(all.begin(), all.end());
    const uint32_t *mine = m->gather_host + (size_t)m->rank * block;
    const int k = (int)mine[0];
    if (k > 0) {
        // my converting particles' positions stay on the device (conv_pos[0..k), in the order of my
        // list); what the host adds are their successors' indices
        for (int i = 0; i < k; ++i) {
            const size_t rank_in_all = (size_t)(std::lower_bound(all.begin(), all.end(), mine[1 + i]) - all.begin());
            m->h_conv[SLAB_LOST_CAP + i] = (uint32_t)(m->n_global + (int64_t)rank_in_all);
        }
        CUDA_TRY(cudaMemcpyAsync(m->conv_pos + SLAB_LOST_CAP, m->h_conv + SLAB_LOST_CAP, sizeof(uint32_t) * k,
                                 cudaMemcpyHostToDevice, c->stream));
        TRY(sphmw_flow_spawn_slab(c, m->conv_pos, m->conv_pos + SLAB_LOST_CAP, k, adiabatic));
    }
    m->n_global += (int64_t)all.size();
    if (n_added) *n_added = (int64_t)all.size();
    return SPHMW_OK;
}

// sphmw_flow_add_new_particles / sphmw_aflow_add_new_particles on a slab context: collective, the same
// spawn as sphmw_step(ctx, "flow" | "aflow", n); *n_added counts the particles added on all ranks
int sphmw_comm_add_new_particles(sphmw_ctx *c, int64_t *n_added, bool adiabatic) {
    if (!c->comm->open_box) {
        sphmw_set_error("add_new_particles: inflow re-seeding renumbers particles across ranks; call "
                        "sphmw_comm_open_box first");
        return SPHMW_E_STATE;
    }
    if (c->overlap_stage != 0) { sphmw_set_error("add_new_particles: an overlapped step is in flight"); return SPHMW_E_STATE; }
    return comm_flow_spawn(c, adiabatic, n_added);
}

static int comm_exchange_all(sphmw_ctx *c) {
    SlabComm *m = c->comm;
    TRY(comm_buffers(c));
    if (m->open_box && m->n_global < 0) TRY(comm_count_global(c));
    TRY(sphmw_halo_pack_enqueue(c, m->send[0], m->send[1], m->cap, false));
    TRY(comm_transfer_and_unpack(c));
    if (m->open_box) TRY(comm_renumber_lost(c));
    return SPHMW_OK;
}

// ≙ create_cell_list!(sys) on a slab context: halo exchange, then the sort
int sphmw_comm_create_cell_list(sphmw_ctx *c, int64_t *n_alive) {
    if (c->overlap_stage != 0) { sphmw_set_error("create_cell_list: an overlapped step is in flight"); return SPHMW_E_STATE; }
    TRY(comm_exchange_all(c));
    return sphmw_build_cell_list(c, n_alive);
}

// nsteps of the fused "wcsph" step (wcsph_perturbed_witch.jl:309-332) on a slab context.  All
// but the last step run the overlapped schedule of pair_ops.cu: the edge columns are advanced and
// packed first and their records travel while the interior columns are in the force pass.
int sphmw_comm_step(sphmw_ctx *c, const char *scheme, int nsteps) {
    SlabComm *m = c->comm;
    const bool hopkins = !strcmp(scheme, "hopkins") || !strcmp(scheme, "hopkins_full") || !strcmp(scheme, "hopkins_total");
    const bool aflow = !strcmp(scheme, "aflow");
    if (!strcmp(scheme, "flow") || aflow) {
        // isothermal_flow_witch.jl:221-232 / adiabatic_flow_witch.jl:231-243, operator by operator;
        // inflow re-seeding and outflow by removal renumber particles across ranks: open box only
        if (!m->open_box) {
            sphmw_set_error("step: the %s scheme loses and gains particles; call sphmw_comm_open_box first", scheme);
            return SPHMW_E_STATE;
        }
        for (int k = 0; k < nsteps; ++k) {
            TRY(sphmw_apply_named(c, "flow.accelerate", 0));
            TRY(sphmw_apply_named(c, aflow ? "aflow.move" : "flow.move", 0));
            TRY(comm_flow_spawn(c, aflow));
            TRY(comm_exchange_all(c));
            TRY(sphmw_build_cell_list(c, nullptr));
            if (aflow) {
                TRY(sphmw_apply_named(c, "aflow.find_density", 1));  // self = true (:236)
                for (const char *op : {"aflow.find_s", "aflow.find_pressure", "aflow.entropy_production",
                                       "flow.internal_force", "flow.accelerate"})
                    TRY(sphmw_apply_named(c, op, 0));
            } else {
                for (const char *op : {"flow.balance_of_mass", "flow.find_pressure", "flow.find_pot_temp",
                                       "flow.internal_force", "flow.accelerate"})
                    TRY(sphmw_apply_named(c, op, 0));
            }
        }
        return SPHMW_OK;
    }
    if (strcmp(scheme, "wcsph") && !hopkins) {
        sphmw_set_error("step: the fused 'wcsph', 'hopkins', 'hopkins_full', 'hopkins_total' and the 'flow' and "
                        "'aflow' schemes run on slabs");
        return SPHMW_E_UNSUPPORTED_OP;
    }
    if (nsteps <= 0) return SPHMW_OK;
    if (hopkins) {  // three ghost columns, plain schedule (hopkins_total: operator by operator)
        for (int k = 0; k < nsteps; ++k) {
            TRY(sphmw_step_scheme_phase(c, scheme, 0));
            TRY(comm_exchange_all(c));
            TRY(sphmw_step_scheme_phase(c, scheme, 1));
        }
        return SPHMW_OK;
    }
    const bool overlap = nsteps > 1 && c->grid.ghost == GHOST_COLS && !(c->flags & SPHMW_FLAG_CELL_PAIRS) && !m->open_box && !getenv("SPHMW_NO_OVERLAP");
    if (!overlap) {
        for (int k = 0; k < nsteps; ++k) {
            TRY(sphmw_step_wcsph_phase(c, 0));
            TRY(comm_exchange_all(c));
            TRY(sphmw_step_wcsph_phase(c, 1));
        }
        return SPHMW_OK;
    }
    TRY(sphmw_step_wcsph_phase(c, 0));
    TRY(comm_exchange_all(c));
    for (int k = 0; k + 1 < nsteps; ++k) {
        TRY(sphmw_step_wcsph_phase(c, 2));                                          // edge columns first
        TRY(sphmw_halo_pack_enqueue(c, m->send[0], m->send[1], m->cap, true));    // their records
        c->overlap_stage = 2;
        TRY(sphmw_step_wcsph_phase(c, 3));                                          // interior, enqueued only
        c->overlap_stage = 0;
        TRY(comm_transfer_and_unpack(c));  // travels beside the interior force pass
    }
    return sphmw_step_wcsph_phase(c, 1);
}
