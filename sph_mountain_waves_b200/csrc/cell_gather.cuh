// The last kernel of the cell-list build (cell_list.cu): one launch permutes every live field
// into the new physical order — (cell ascending, reference index descending), core.jl:32-37 —
// and writes the per-particle data the pair passes derive from the sorted positions (the quantised
// pre-test mirror and, when enabled, neighbour record A).  In a header so that the CPU emulation
// harness (tests/emu/) runs the same code.
#pragma once
#include "sphmw_internal.h"

struct GatherList {
    const double *from[NSLOT];
    double *to[NSLOT];
    int count;
    // quantised mirror of the sorted positions (pair_list.cuh): where the particle sits inside
    // its own cell — the 6-bit word of the zrun cell order (q6), else 10 bits per axis (h/1024)
    int xpos[3];  // entry of x0/x1/x2 in the lists above (-1: no such component)
    double h;
    uint32_t *xq;
    int q6, dim;
    long long run_phase;  // key_phase of the run axis (z in 3D, y in 2D)
    // packed neighbour record A {x, y, z, m} (SPHMW_FLAG_PACKED_RECORDS; null otherwise)
    int mpos;
    NbRec *recA;
    // fluid flag per position (type == fluid, the test of wcsph_force_finish), the input of the fluid
    // work list (cell_list.cu); null: not wanted
    int tpos;  // entry of the type field in the lists above
    double fluid;
    uint8_t *fl;
};

__global__ void k_gather(GatherList gl, const uint32_t *__restrict__ src,
                         const uint32_t *__restrict__ idx, uint32_t *__restrict__ idx_out,
                         uint32_t *__restrict__ pos_of_idx, const uint32_t *__restrict__ key,
                         uint32_t *__restrict__ key_out, const uint32_t *__restrict__ tag,
                         uint32_t *__restrict__ tag_out, const uint32_t *__restrict__ cellx,
                         uint32_t *__restrict__ cellx_out, int64_t n_new) {
    int64_t slot = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (slot >= n_new) return;
    uint32_t s = src[slot];
    uint32_t id = idx[s];
    idx_out[slot] = id;
    if (pos_of_idx) pos_of_idx[id] = (uint32_t)slot;
    key_out[slot] = key[s];
    tag_out[slot] = tag[s];
    cellx_out[slot] = cellx[s];
    uint32_t qm = 0;
    double ra[4] = {0.0, 0.0, 0.0, 0.0};
    for (int f = 0; f < gl.count; ++f) {
        const double v = gl.from[f][s];
        gl.to[f][slot] = v;
        if (f == gl.mpos) ra[3] = v;
        if (f == gl.tpos && gl.fl) gl.fl[slot] = v == gl.fluid;
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (f == gl.xpos[a]) {
                ra[a] = v;
                qm |= nl_q10_axis(v, gl.h) << (10 * a);
            }
    }
    if (gl.q6) qm = nl_q6_word(ra[0], ra[1], ra[2], gl.h, gl.run_phase, gl.dim);
    gl.xq[slot] = qm;
    if (gl.recA) nb_store(gl.recA + slot, ra[0], ra[1], ra[2], ra[3]);
}
