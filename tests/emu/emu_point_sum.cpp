// CPU emulation harness of the point sums — TEST INFRASTRUCTURE, never shipped.
//
// Compiles csrc/point_sum.cuh behind the stand-in <cuda_runtime.h> and runs what sphmw_point_sum runs,
// thread by thread: the cell list of the particles (sorted by physical key, reference index descending,
// in the zrun or the x-chunked order), k_point_keys, the sort of the points by home key (stable, as the
// radix sort is) and k_point_sum.
//
// Input (little endian): int32 {zrun, nops, nextra, 0}, int64 {n, npoints}, double box[6], double h,
// nops x int32 {kind (PointOpKind), extra field index or -1}, then in reference index order
// x0 x1 x2 m rho and the nextra fields (n doubles each), then the points (3 x npoints, SoA).
// Output: nops x npoints doubles, out[o*npoints + i].
//
// usage: emu_point_sum <input.bin> <output.bin>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "cuda_runtime.h"
#include "point_sum.cuh"

uint3 threadIdx, blockIdx, blockDim, gridDim;
uint32_t nl_queue[1];

void sphmw_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fputc('\n', stderr);
}

template <class F>
static void launch(int64_t n, unsigned block, F &&thread_body) {
    blockDim = uint3{block, 1, 1};
    for (int64_t b = 0; b * block < n; ++b) {
        blockIdx = uint3{(unsigned)b, 0, 0};
        for (unsigned t = 0; t < block; ++t) {
            threadIdx = uint3{t, 0, 0};
            thread_body();
        }
    }
}

static void read_exact(FILE *fp, void *dst, size_t bytes) {
    if (bytes && fread(dst, 1, bytes, fp) != bytes) {
        fprintf(stderr, "emu_point_sum: truncated input\n");
        exit(2);
    }
}

int main(int argc, char **argv) {
    if (argc != 3) {
        fprintf(stderr, "usage: emu_point_sum <input.bin> <output.bin>\n");
        return 2;
    }
    FILE *fp = fopen(argv[1], "rb");
    if (!fp) {
        perror(argv[1]);
        return 2;
    }
    int32_t head[4];
    int64_t sizes[2];
    double box[7];
    read_exact(fp, head, sizeof(head));
    read_exact(fp, sizes, sizeof(sizes));
    read_exact(fp, box, sizeof(box));
    const int zrun = head[0], nops = head[1], nextra = head[2];
    const int64_t n = sizes[0], np = sizes[1];
    if (nops < 1 || nops > SPHMW_POINT_OPS_MAX) return 2;
    std::vector<int32_t> opdesc(2 * nops);
    read_exact(fp, opdesc.data(), sizeof(int32_t) * 2 * nops);
    std::vector<std::vector<double>> in(5 + nextra, std::vector<double>(n));
    for (auto &a : in) read_exact(fp, a.data(), sizeof(double) * n);
    std::vector<double> pts(3 * np);
    read_exact(fp, pts.data(), sizeof(double) * 3 * np);
    fclose(fp);

    Grid g;
    memset(&g, 0, sizeof(g));
    int64_t global_cols = 0;
    if (sphmw_grid_setup(g, box, box + 3, box[6], -1, -1, &global_cols) != SPHMW_OK) return 3;
    sphmw_grid_set_order(g, zrun != 0);

    // cell list: (physical key ascending, reference index descending), as cell_list.cu leaves it
    std::vector<uint32_t> pkey(n), order(n), cs(g.pkey_max + 2, 0u);
    for (int64_t p = 0; p < n; ++p) {
        int i, j, k;
        if (g.dim == 2 ? !cell_ijk_whole<2>(g, in[0][p], in[1][p], 0.0, i, j, k)
                       : !cell_ijk_whole<3>(g, in[0][p], in[1][p], in[2][p], i, j, k)) {
            fprintf(stderr, "emu_point_sum: particle %lld is outside the box (not supported here)\n", (long long)p);
            return 3;
        }
        pkey[p] = pkey_ijk(g, i, j, k);
        cs[pkey[p] + 1] += 1;
    }
    for (long long c = 0; c <= g.pkey_max; ++c) cs[c + 1] += cs[c];
    std::iota(order.begin(), order.end(), 0u);
    std::sort(order.begin(), order.end(),
              [&](uint32_t a, uint32_t b) { return pkey[a] != pkey[b] ? pkey[a] < pkey[b] : a > b; });
    std::vector<std::vector<double>> phys(in.size(), std::vector<double>(n));
    for (size_t f = 0; f < in.size(); ++f)
        for (int64_t p = 0; p < n; ++p) phys[f][p] = in[f][order[p]];

    PointOps ops{};
    ops.n = nops;
    ops.x0 = phys[0].data();
    ops.x1 = phys[1].data();
    ops.x2 = g.dim == 3 ? phys[2].data() : nullptr;
    ops.m = phys[3].data();
    ops.rho = phys[4].data();
    for (int o = 0; o < nops; ++o) {
        ops.kind[o] = opdesc[2 * o];
        ops.need_v = ops.need_v || ops.kind[o] == PT_VW || ops.kind[o] == PT_VW_F;
        const int e = opdesc[2 * o + 1];
        ops.f[o] = e >= 0 && e < nextra ? phys[5 + e].data() : nullptr;
    }

    std::vector<uint32_t> key(np), porder(np);
    launch(np, 256, [&] {
        if (g.dim == 2) k_point_keys<2>(g, pts.data(), np, key.data(), porder.data());
        else k_point_keys<3>(g, pts.data(), np, key.data(), porder.data());
    });
    std::stable_sort(porder.begin(), porder.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
    std::vector<double> out((size_t)nops * np, -12345.0);
    launch(np, 128, [&] {
        if (g.dim == 2) k_point_sum<2>(ops, g, cs.data(), pts.data(), np, porder.data(), out.data());
        else k_point_sum<3>(ops, g, cs.data(), pts.data(), np, porder.data(), out.data());
    });
    FILE *fo = fopen(argv[2], "wb");
    if (!fo) {
        perror(argv[2]);
        return 2;
    }
    fwrite(out.data(), sizeof(double), out.size(), fo);
    fclose(fo);
    printf("emu_point_sum: n=%lld points=%lld dim=%d zrun=%d ops=%d\n", (long long)n, (long long)np, g.dim, zrun, nops);
    return 0;
}
