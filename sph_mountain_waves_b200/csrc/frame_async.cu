// Asynchronous frame output and input prefetch — save_frame! (src/IO.jl:53-75) without stopping
// the time loop (SURVEY.md §8 f1).
//
// The reference gathers every exported field from the particle objects and hands the arrays to
// WriteVTK inside the time loop (wcsph_perturbed_witch.jl:375-388): the step waits for the file.
// Here a frame is CAPTURED on the device — one kernel per field permutes it into reference index
// order and interleaves its components exactly as the .vtp arrays want them (the transpose the
// host used to do) — into one of two snapshot buffers; a copy stream moves the snapshot to pinned
// host memory while the main stream goes on stepping, and a writer thread compresses and writes
// the file once the copy has landed (frame_io.cpp).  The next capture into the same buffer waits
// for that writer, nothing else ever does.
//
//   sphmw_frame_capture / sphmw_frame_wait   the same mechanism for callers that want the arrays
//                                            (bench.py's end-to-end cycle, a Julia host)
//   sphmw_upload_async / sphmw_upload_commit host -> device prefetch on the copy stream: fields are
//                                            staged while the main stream is busy and enter the
//                                            particle arrays at the commit
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "sphmw_internal.h"

struct FrameSlot {
    double *dev = nullptr, *host = nullptr;
    size_t cap = 0;  // doubles
    cudaEvent_t snapped = nullptr, copied = nullptr;
    std::thread writer;
    bool in_flight = false;
    int64_t n = 0;
    std::vector<int> ncomps;
    std::vector<size_t> offs;  // start of each array inside the buffers (doubles)
    std::vector<std::string> names;
    std::string error;  // what the writer thread had to say
};

struct UploadItem {
    int slot, ncomp;
    size_t off;
};

struct FrameAsync {
    cudaStream_t copy_stream = nullptr;  // device -> host (frames)
    cudaStream_t up_stream = nullptr;    // host -> device (prefetch): its own stream, so that a commit never waits for a frame copy
    FrameSlot slot[2];
    int next = 0;
    // upload prefetch
    double *up_dev = nullptr;
    size_t up_cap = 0, up_used = 0;
    int64_t up_n = -1;
    std::vector<UploadItem> up_items;
    cudaEvent_t up_copied = nullptr, up_consumed = nullptr;
    bool up_consumed_valid = false;
};

// dst[idx[pos] * NC + k] = src_k[pos]: index order, components interleaved (what WriteVTK stores)
template <int NC>
__global__ void k_frame_snapshot(double *__restrict__ dst, const double *__restrict__ s0, const double *__restrict__ s1,
                                 const double *__restrict__ s2, const uint32_t *__restrict__ idx, int64_t n, int by_index) {
    const int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos >= n) return;
    const size_t o = (size_t)(by_index ? idx[pos] : pos) * NC;
    dst[o] = s0 ? s0[pos] : 0.0;
    if (NC > 1) dst[o + 1] = s1 ? s1[pos] : 0.0;
    if (NC > 2) dst[o + 2] = s2 ? s2[pos] : 0.0;
}

static int fa_get(sphmw_ctx *c, FrameAsync **out) {
    if (!c->frame_async) {
        FrameAsync *fa = new FrameAsync();
        c->frame_async = fa;
        CUDA_TRY(cudaStreamCreateWithFlags(&fa->copy_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&fa->up_stream, cudaStreamNonBlocking));
        for (FrameSlot &s : fa->slot) {
            CUDA_TRY(cudaEventCreateWithFlags(&s.snapped, cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&fa->up_copied, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&fa->up_consumed, cudaEventDisableTiming));
    }
    *out = c->frame_async;
    return SPHMW_OK;
}

static int slot_finish(FrameSlot &s) {
    if (s.writer.joinable()) s.writer.join();
    s.in_flight = false;
    if (!s.error.empty()) {
        sphmw_set_error("%s", s.error.c_str());
        s.error.clear();
        return SPHMW_E_IO;
    }
    return SPHMW_OK;
}

void sphmw_frame_async_free(sphmw_ctx *c) {
    FrameAsync *fa = c->frame_async;
    if (!fa) return;
    for (FrameSlot &s : fa->slot) {
        if (s.writer.joinable()) s.writer.join();
        cudaFree(s.dev);
        if (s.host) cudaFreeHost(s.host);
        if (s.snapped) cudaEventDestroy(s.snapped);
        if (s.copied) cudaEventDestroy(s.copied);
    }
    if (fa->copy_stream) cudaStreamSynchronize(fa->copy_stream);
    if (fa->up_stream) cudaStreamSynchronize(fa->up_stream);
    cudaFree(fa->up_dev);
    if (fa->up_copied) cudaEventDestroy(fa->up_copied);
    if (fa->up_consumed) cudaEventDestroy(fa->up_consumed);
    if (fa->copy_stream) cudaStreamDestroy(fa->copy_stream);
    if (fa->up_stream) cudaStreamDestroy(fa->up_stream);
    delete fa;
    c->frame_async = nullptr;
}

// snapshot of x (first) and the named fields at this point of the main stream; the copy to pinned
// memory is queued on the copy stream.  Returns the slot through *slot_out.
int sphmw_frame_capture_impl(sphmw_ctx *c, const char *const *fields, int nfields, bool with_x, int *slot_out) {
    FrameAsync *fa;
    TRY(fa_get(c, &fa));
    FrameSlot &s = fa->slot[fa->next];
    TRY(slot_finish(s));  // the writer of two frames ago
    const int64_t n = c->n;
    std::vector<const FieldDesc *> descs;
    s.names.clear();
    s.ncomps.clear();
    s.offs.clear();
    size_t total = 0;
    for (int f = with_x ? -1 : 0; f < nfields; ++f) {
        const char *name = f < 0 ? "x" : fields[f];
        const FieldDesc *d = sphmw_find_field(name);
        if (!d) {
            sphmw_set_error("Variable %s does not exist!", name);  // structs.jl:128-133
            return SPHMW_E_UNKNOWN_FIELD;
        }
        descs.push_back(d);
        s.names.push_back(name);
        s.ncomps.push_back(d->ncomp);
        s.offs.push_back(total);
        total += (size_t)d->ncomp * (size_t)n;
    }
    if (total > s.cap) {
        cudaFree(s.dev);
        if (s.host) cudaFreeHost(s.host);
        s.dev = s.host = nullptr;
        s.cap = 0;
        const size_t want = total + total / 8 + 1024;
        CUDA_TRY(cudaMalloc(&s.dev, sizeof(double) * want));
        CUDA_TRY(cudaMallocHost(&s.host, sizeof(double) * want));
        s.cap = want;
    }
    s.n = n;
    const int by_index = c->slab_lo < 0;  // slab contexts carry global indices: physical order
    for (size_t f = 0; f < descs.size() && n > 0; ++f) {
        const FieldDesc *d = descs[f];
        const double *src[3] = {nullptr, nullptr, nullptr};
        for (int k = 0; k < d->ncomp; ++k) {
            const int sl = d->slot + k;
            if (c->grid.dim == 2 && d->ncomp == 3 && k == 2) continue;  // 2D keeps no third component
            if (c->allocated[sl] && c->stale[sl]) TRY(sphmw_materialize(c, sl));
            if (!c->allocated[sl] && !(sl >= S_DV0 && sl <= S_DV2 && c->dv_zero)) TRY(sphmw_materialize(c, sl));
            if (c->allocated[sl] && !c->stale[sl]) src[k] = c->cur.s[sl];
        }
        TIMED(c, "frame_snapshot");
        double *dst = s.dev + s.offs[f];
        if (d->ncomp == 1)
            k_frame_snapshot<1><<<grid_for(n, 256), 256, 0, c->stream>>>(dst, src[0], nullptr, nullptr, c->idx, n, by_index);
        else
            k_frame_snapshot<3><<<grid_for(n, 256), 256, 0, c->stream>>>(dst, src[0], src[1], src[2], c->idx, n, by_index);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(s.snapped, c->stream));
    CUDA_TRY(cudaStreamWaitEvent(fa->copy_stream, s.snapped, 0));
    if (total) CUDA_TRY(cudaMemcpyAsync(s.host, s.dev, sizeof(double) * total, cudaMemcpyDeviceToHost, fa->copy_stream));
    CUDA_TRY(cudaEventRecord(s.copied, fa->copy_stream));
    s.in_flight = true;
    *slot_out = fa->next;
    fa->next ^= 1;
    return SPHMW_OK;
}

extern "C" int sphmw_frame_capture(sphmw_ctx *c, const char *const *fields, int32_t nfields, int32_t *slot) {
    if (!c || (nfields > 0 && !fields) || !slot) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    int s = 0;
    TRY(sphmw_frame_capture_impl(c, fields, nfields, false, &s));
    *slot = s;
    return SPHMW_OK;
}

// Waits for the copy of that capture; host[f] points at field f (n x ncomp doubles, components
// interleaved; reference index order, physical order on a slab context) in the library's pinned
// buffer, valid until the second capture from now.
extern "C" int sphmw_frame_wait(sphmw_ctx *c, int32_t slot, const double **host, int32_t nfields, int64_t *n) {
    if (!c || slot < 0 || slot > 1 || !c->frame_async) { sphmw_set_error("frame_wait: no such capture"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    FrameSlot &s = c->frame_async->slot[slot];
    if (!s.in_flight) { sphmw_set_error("frame_wait: no such capture"); return SPHMW_E_STATE; }
    if ((int)s.names.size() != nfields) { sphmw_set_error("frame_wait: the capture has %zu fields", s.names.size()); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaEventSynchronize(s.copied));
    for (int f = 0; f < nfields; ++f)
        if (host) host[f] = s.host + s.offs[f];
    if (n) *n = s.n;
    return SPHMW_OK;
}

// ≙ save_frame!(data, sys, vars...) — IO.jl:53-75: capture now, write on a worker thread
int sphmw_pvd_save_frame_async(sphmw_ctx *c, const char *const *fields, int nfields, const std::string &path) {
    int si = 0;
    TRY(sphmw_frame_capture_impl(c, fields, nfields, true, &si));
    FrameSlot *s = &c->frame_async->slot[si];
    const int device = c->device;
    s->writer = std::thread([s, device, path]() {
        cudaSetDevice(device);
        if (cudaEventSynchronize(s->copied) != cudaSuccess) {
            s->error = "frame copy failed";
            return;
        }
        const int nf = (int)s->names.size() - 1;
        std::vector<const char *> names(nf);
        std::vector<const double *> ptrs(nf);
        for (int f = 0; f < nf; ++f) {
            names[f] = s->names[f + 1].c_str();
            ptrs[f] = s->host + s->offs[f + 1];
        }
        if (sphmw_write_vtp(path.c_str(), s->n, s->host + s->offs[0], nf, names.data(), s->ncomps.data() + 1, ptrs.data()) !=
            SPHMW_OK)
            s->error = std::string("writing ") + path + " failed: " + sphmw_last_error();
    });
    return SPHMW_OK;
}

// all writers done (save_pvd_file, sphmw_destroy); reports the first failure
int sphmw_frame_async_drain(sphmw_ctx *c) {
    if (!c->frame_async) return SPHMW_OK;
    int rc = SPHMW_OK;
    for (FrameSlot &s : c->frame_async->slot)
        if (s.writer.joinable()) {
            const int r = slot_finish(s);
            if (rc == SPHMW_OK) rc = r;
        }
    return rc;
}

// ---- host -> device prefetch ---------------------------------------------------------------------
// Stages one field on the copy stream; `buf` must stay valid until sphmw_upload_commit.  n is the
// particle count the commit will set (every field of one batch has the same n).
// slot < 0: the batch's global particle indices (slab contexts), n int64 values
static int upload_stage(sphmw_ctx *c, int slot, int ncomp, const void *buf, int64_t n, const char *what);

extern "C" int sphmw_upload_async(sphmw_ctx *c, const char *field, const double *buf, int64_t n, int32_t ncomp) {
    if (!c || !field || !buf || n < 0) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    const FieldDesc *d = sphmw_find_field(field);
    if (!d) { sphmw_set_error("Variable %s does not exist!", field); return SPHMW_E_UNKNOWN_FIELD; }
    if (ncomp != d->ncomp || n > c->cap) { sphmw_set_error("upload_async(%s): shape mismatch", field); return SPHMW_E_INVALID; }
    return upload_stage(c, d->slot, ncomp, buf, n, field);
}
// the global indices of the batch (slab contexts; ≙ sphmw_set_index after the commit, without its
// host wait): staged like a field, applied by the commit
extern "C" int sphmw_upload_index_async(sphmw_ctx *c, const int64_t *global_idx, int64_t n) {
    if (!c || !global_idx || n < 0) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo < 0) { sphmw_set_error("upload_index_async: context has no slab"); return SPHMW_E_STATE; }
    if (n > c->cap) { sphmw_set_error("upload_index_async: n exceeds the capacity"); return SPHMW_E_INVALID; }
    return upload_stage(c, -1, 1, global_idx, n, "index");
}

static int upload_stage(sphmw_ctx *c, int slot, int ncomp, const void *buf, int64_t n, const char *field) {
    FrameAsync *fa;
    TRY(fa_get(c, &fa));
    if (fa->up_items.empty()) {
        fa->up_n = n;
        fa->up_used = 0;
        // the staging area may still be read by the permute kernels of the previous commit
        if (fa->up_consumed_valid) CUDA_TRY(cudaStreamWaitEvent(fa->up_stream, fa->up_consumed, 0));
    } else if (n != fa->up_n) {
        sphmw_set_error("upload_async: all fields of one batch have the same length");
        return SPHMW_E_INVALID;
    }
    const size_t need = fa->up_used + (size_t)ncomp * (size_t)n;
    if (need > fa->up_cap) {
        if (!fa->up_items.empty()) { sphmw_set_error("upload_async: staging area too small for this batch"); return SPHMW_E_CAPACITY; }
        CUDA_TRY(cudaStreamSynchronize(fa->up_stream));
        cudaFree(fa->up_dev);
        fa->up_dev = nullptr;
        fa->up_cap = std::max<size_t>((size_t)16 * (size_t)c->cap, need);  // x, v, and ten scalars
        CUDA_TRY(cudaMalloc(&fa->up_dev, sizeof(double) * fa->up_cap));
    }
    if (n) CUDA_TRY(cudaMemcpyAsync(fa->up_dev + fa->up_used, buf, sizeof(double) * ncomp * n, cudaMemcpyHostToDevice,
                                    fa->up_stream));
    fa->up_items.push_back(UploadItem{slot, ncomp, fa->up_used});
    fa->up_used = need;
    return SPHMW_OK;
}

__global__ void k_permute_in_async(double *__restrict__ dst, const double *__restrict__ stg, int64_t n) {
    const int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos < n) dst[pos] = stg[pos];
}
__global__ void k_index_in_async(uint32_t *__restrict__ idx, const long long *__restrict__ stg, int64_t n) {
    const int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pos < n) idx[pos] = (uint32_t)stg[pos];
}

// The staged fields become the particle state: the context is resized to the batch's n (indices
// 0..n-1 in upload order, like sphmw_resize(0) + sphmw_resize(n)) and the main stream copies
// them in once the prefetch has landed.  Does not wait on the host.
extern "C" int sphmw_upload_commit(sphmw_ctx *c) {
    if (!c || !c->frame_async || c->frame_async->up_items.empty()) { sphmw_set_error("upload_commit: nothing staged"); return SPHMW_E_STATE; }
    CUDA_TRY(cudaSetDevice(c->device));
    FrameAsync *fa = c->frame_async;
    TRY(sphmw_resize(c, 0));
    TRY(sphmw_resize(c, fa->up_n));
    CUDA_TRY(cudaEventRecord(fa->up_copied, fa->up_stream));
    CUDA_TRY(cudaStreamWaitEvent(c->stream, fa->up_copied, 0));
    const int64_t n = fa->up_n;
    for (const UploadItem &it : fa->up_items)
        for (int k = 0; k < it.ncomp; ++k) {
            if (it.slot < 0) {  // global indices (sphmw_upload_index_async)
                if (n) k_index_in_async<<<grid_for(n, 256), 256, 0, c->stream>>>(c->idx, (const long long *)(fa->up_dev + it.off), n);
                continue;
            }
            if (c->grid.dim == 2 && it.ncomp == 3 && k == 2) continue;
            const int slot = it.slot + k;
            TRY(sphmw_ensure_slot(c, slot));
            if (n) {
                TIMED(c, "upload_permute");
                k_permute_in_async<<<grid_for(n, 256), 256, 0, c->stream>>>(c->cur.s[slot], fa->up_dev + it.off + (size_t)k * n, n);
            }
            c->stale[slot] = false;
            if (slot == S_X0) c->cell_list_valid = false, c->keys_from_advance = false;
            if (slot == S_DV0) c->dv_zero = false;
            if (slot == S_TYPE) c->fluid_gen = ~0ull;
        }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(fa->up_consumed, c->stream));
    fa->up_consumed_valid = true;
    fa->up_items.clear();
    return SPHMW_OK;
}
