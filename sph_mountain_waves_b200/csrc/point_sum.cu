// Point sums on the device — sphmw_point_sum, the `sum(sys, f, x)` of src/core.jl:240-291.
// The walk itself is in point_sum.cuh; this file decodes the ops, brings stale fields up to date and
// runs keys -> sort by home cell -> walk on the context's stream.
#include <string.h>

#include <string>

#include <cub/device/device_radix_sort.cuh>

#include "point_sum.cuh"
#include "sphmw_internal.h"

// "count" | "mW" | "VW" | "mW*<f>" | "VW*<f>", <f> a scalar field or a vector component "v[c]"
static int parse_point_op(const sphmw_ctx *c, const char *op, int &kind, int &slot) {
    slot = -1;
    if (!strcmp(op, "count")) {
        kind = PT_COUNT;
        return SPHMW_OK;
    }
    const bool mw = !strncmp(op, "mW", 2), vw = !strncmp(op, "VW", 2);
    if (!(mw || vw) || (op[2] != 0 && op[2] != '*') || (op[2] == '*' && op[3] == 0)) {
        sphmw_set_error("point_sum: unknown op '%s' (count | mW | VW | mW*<field> | VW*<field>)", op);
        return SPHMW_E_UNSUPPORTED_OP;
    }
    if (op[2] == 0) {
        kind = mw ? PT_MW : PT_VW;
        return SPHMW_OK;
    }
    kind = mw ? PT_MW_F : PT_VW_F;
    std::string name(op + 3);
    int comp = -1;
    const size_t br = name.find('[');
    if (br != std::string::npos) {
        if (name.size() != br + 3 || name[br + 2] != ']' || name[br + 1] < '0' || name[br + 1] > '9') {
            sphmw_set_error("point_sum: '%s': a component is written <field>[c], c = 0, 1, 2", op);
            return SPHMW_E_INVALID;
        }
        comp = name[br + 1] - '0';
        name.resize(br);
    }
    const FieldDesc *d = sphmw_find_field(name.c_str());
    if (!d) {
        sphmw_set_error("point_sum: Variable %s does not exist!", name.c_str());
        return SPHMW_E_UNKNOWN_FIELD;
    }
    if ((d->ncomp == 1) != (comp < 0) || comp > 2 || (comp == 2 && c->grid.dim == 2)) {
        sphmw_set_error("point_sum: '%s': %s", op,
                        d->ncomp == 1 ? "a scalar field has no component"
                                      : (comp < 0 ? "name a component of the vector field, e.g. v[0]"
                                                  : "no such component in this system"));
        return SPHMW_E_INVALID;
    }
    slot = d->slot + (comp < 0 ? 0 : comp);
    return SPHMW_OK;
}

// a field as sphmw_download reads it: stale -> rebuilt; never written -> null (reads as zeros)
static int point_field(sphmw_ctx *c, int slot, const double **p) {
    if (c->allocated[slot] && c->stale[slot]) TRY(sphmw_materialize(c, slot));
    if (!c->allocated[slot] && !(slot >= S_DV0 && slot <= S_DV2 && c->dv_zero))
        TRY(sphmw_materialize(c, slot));  // may derive T, theta
    *p = c->allocated[slot] ? c->cur.s[slot] : nullptr;
    return SPHMW_OK;
}

// device memory of this context's device; anything else (pageable, pinned, another device) is copied
static bool on_device(const sphmw_ctx *c, const void *p, bool *pinned) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        *pinned = false;
        return false;
    }
    *pinned = a.type == cudaMemoryTypeHost;
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == c->device;
}

static int point_scratch(sphmw_ctx *c, int64_t n, int64_t nout, int key_bits) {
    if (n > c->pt_cap) {
        cudaFree(c->pt_pts);
        cudaFree(c->pt_key);
        cudaFree(c->pt_order);
        c->pt_pts = nullptr, c->pt_key = c->pt_order = nullptr, c->pt_cap = 0;
        CUDA_TRY(cudaMalloc(&c->pt_pts, sizeof(double) * 3 * n));
        CUDA_TRY(cudaMalloc(&c->pt_key, sizeof(uint32_t) * 2 * n));
        CUDA_TRY(cudaMalloc(&c->pt_order, sizeof(uint32_t) * 2 * n));
        c->pt_cap = n;
    }
    if (nout > c->pt_out_cap) {
        cudaFree(c->pt_out);
        c->pt_out = nullptr, c->pt_out_cap = 0;
        CUDA_TRY(cudaMalloc(&c->pt_out, sizeof(double) * nout));
        c->pt_out_cap = nout;
    }
    size_t bytes = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, bytes, c->pt_key, c->pt_key + n, c->pt_order, c->pt_order + n,
                                             (int)n, 0, key_bits, c->stream));
    if (bytes > c->pt_sort_tmp_bytes) {
        cudaFree(c->pt_sort_tmp);
        c->pt_sort_tmp = nullptr, c->pt_sort_tmp_bytes = 0;
        CUDA_TRY(cudaMalloc(&c->pt_sort_tmp, bytes));
        c->pt_sort_tmp_bytes = bytes;
    }
    return SPHMW_OK;
}

extern "C" int sphmw_point_sum(sphmw_ctx *c, const char *const *ops, int32_t nops, const double *points, int64_t n,
                               double *out) {
    if (!c || !ops) { sphmw_set_error("null argument"); return SPHMW_E_INVALID; }
    if (nops < 1 || nops > SPHMW_POINT_OPS_MAX) {
        sphmw_set_error("point_sum: %d ops (1..%d per call)", (int)nops, SPHMW_POINT_OPS_MAX);
        return SPHMW_E_INVALID;
    }
    if (n < 0 || n > (int64_t)0x7FFFFFF0 || (n > 0 && (!points || !out))) {
        sphmw_set_error("point_sum: bad point buffers or count %lld", (long long)n);
        return SPHMW_E_INVALID;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    if (c->slab_lo >= 0) {
        // at the end of a step a ghost's v is not its owner's (ghosts are packed after the drift and the
        // force pass kicks owned columns only), so sums near a slab face would not be exact
        sphmw_set_error("point_sum: x-slab contexts are not supported (ghost copies are not the owners' state "
                        "at the end of a step); sample on a whole-domain context");
        return SPHMW_E_STATE;
    }
    int kind[SPHMW_POINT_OPS_MAX], slot[SPHMW_POINT_OPS_MAX];
    for (int o = 0; o < nops; ++o) {
        if (!ops[o]) { sphmw_set_error("null op"); return SPHMW_E_INVALID; }
        TRY(parse_point_op(c, ops[o], kind[o], slot[o]));
    }
    if (!c->cell_list_valid) {
        sphmw_set_error("point_sum: cell list is not built (create_cell_list after moving particles)");
        return SPHMW_E_STATE;
    }
    if (n == 0) return SPHMW_OK;

    PointOps po{};
    po.n = nops;
    for (int o = 0; o < nops; ++o) {
        po.kind[o] = kind[o];
        po.need_v = po.need_v || kind[o] == PT_VW || kind[o] == PT_VW_F;
        if (slot[o] >= 0) TRY(point_field(c, slot[o], &po.f[o]));
    }
    TRY(point_field(c, S_M, &po.m));
    if (po.need_v) TRY(point_field(c, S_RHO, &po.rho));
    TRY(point_field(c, S_X0, &po.x0));
    TRY(point_field(c, S_X1, &po.x1));
    if (c->grid.dim == 3) TRY(point_field(c, S_X2, &po.x2));

    int key_bits = 1;
    while (key_bits < 32 && (1ull << key_bits) <= (unsigned long long)c->grid.pkey_max) ++key_bits;
    bool pts_pinned = false, out_pinned = false;
    const bool pts_dev = on_device(c, points, &pts_pinned), out_dev = on_device(c, out, &out_pinned);
    TRY(point_scratch(c, n, out_dev ? 0 : (int64_t)nops * n, key_bits));
    const double *pts = points;
    if (!pts_dev) {
        CUDA_TRY(cudaMemcpyAsync(c->pt_pts, points, sizeof(double) * 3 * n, cudaMemcpyDefault, c->stream));
        pts = c->pt_pts;
    }
    double *dst = out_dev ? out : c->pt_out;
    const Grid &g = c->grid;
    {
        TIMED(c, "point_keys");
        if (g.dim == 2) k_point_keys<2><<<grid_for(n, 256), 256, 0, c->stream>>>(g, pts, n, c->pt_key, c->pt_order);
        else k_point_keys<3><<<grid_for(n, 256), 256, 0, c->stream>>>(g, pts, n, c->pt_key, c->pt_order);
    }
    CUDA_TRY(cudaGetLastError());
    {
        TIMED(c, "point_sort");
        size_t bytes = c->pt_sort_tmp_bytes;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(c->pt_sort_tmp, bytes, c->pt_key, c->pt_key + n, c->pt_order,
                                                 c->pt_order + n, (int)n, 0, key_bits, c->stream));
    }
    {
        TIMED(c, "point_sum");
        const uint32_t *order = c->pt_order + n;
        if (g.dim == 2)
            k_point_sum<2><<<grid_for(n, 128), 128, 0, c->stream>>>(po, g, c->cell_start, pts, n, order, dst);
        else
            k_point_sum<3><<<grid_for(n, 128), 128, 0, c->stream>>>(po, g, c->cell_start, pts, n, order, dst);
    }
    CUDA_TRY(cudaGetLastError());
    if (!out_dev) {
        CUDA_TRY(cudaMemcpyAsync(out, dst, sizeof(double) * nops * n, cudaMemcpyDefault, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    } else if (pts_pinned) {
        // a pinned buffer is read by the copy engine after the call returns: the caller may reuse it at once
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    return SPHMW_OK;
}
