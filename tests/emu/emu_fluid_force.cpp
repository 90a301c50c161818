// CPU emulation harness of the fluid-only force pass — TEST INFRASTRUCTURE, never shipped.
//
// Runs whole multi-step fused WCSPH calls the way sphmw_step does on one GPU (csrc/pair_ops.cu
// step_wcsph_fused): accelerate! + move! once, then per step the cell list (the library's k_gather,
// which also writes the fluid flags), the recording density pass with the packed records, and the
// force pass replayed over the fluid work list (k_binary_list_fluid) — with B_force_advance, i.e. the
// next step's accelerate! + move! folded in, on every step but the last.  The work list is compacted
// here on the host from the gather's flags, in the order cell_list.cu k_fluid_scatter produces.  The
// advance also writes the next cell list's keys (cell_key_whole); the next step sorts by those, and they
// must equal the keys computed here from the new positions.
//
// Input: as tests/emu/emu_pairs.cpp (header, box, parameters, fields in reference index order).
// Output: meta {n, dim, force pairs, fluid positions, non-fluid warps, mixed warps — of the last step}, then
// rho, h, v (3), x (3) in reference index order.
//
// usage: emu_fluid_force <input.bin> <output.bin>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <numeric>
#include <string>
#include <type_traits>
#include <vector>

#include "cuda_runtime.h"
#include "cell_gather.cuh"
#include "pair_list.cuh"
#include "sphmw_internal.h"
#include "wcsph_ops.cuh"

uint3 threadIdx, blockIdx, blockDim, gridDim;
uint32_t nl_queue[(96 + NL_QUEUE_SLACK) * NL_BLOCK];

void sphmw_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fputc('\n', stderr);
}

template <class F>
static void launch(int64_t n, F &&thread_body) {
    blockDim = uint3{NL_BLOCK, 1, 1};
    for (int64_t b = 0; b * NL_BLOCK < n; ++b) {
        blockIdx = uint3{(unsigned)b, 0, 0};
        for (unsigned t = 0; t < NL_BLOCK; ++t) {
            threadIdx = uint3{t, 0, 0};
            thread_body();
        }
    }
}

static void read_exact(FILE *fp, void *dst, size_t bytes) {
    if (bytes && fread(dst, 1, bytes, fp) != bytes) {
        fprintf(stderr, "emu_fluid_force: truncated input\n");
        exit(2);
    }
}

// the fields a step carries, in reference index order
static const int IN_SLOTS[] = {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2, S_M, S_H, S_RHO, S_RHO_P, S_TYPE};

struct Step {
    unsigned long long pairs = 0;
    uint32_t n_fluid = 0;
    int64_t warps_nonfluid = 0, warps_mixed = 0;  // warps of the sorted order without / with some fluid particles
};

// one step of a multi-step call: cell list, density pass, force pass over the fluid work list
template <int DIM, class DensityOp, class ForceOp>
static int run_step(std::vector<double> (&in)[11], int64_t n, const Grid &g, const Params &prm_in, int stride, Step &out,
                    std::vector<uint32_t> &carry_key, std::vector<uint32_t> &carry_col) {
    Params prm = prm_in;
    std::vector<uint32_t> pkey(n), col(n), order(n);
    for (int64_t i = 0; i < n; ++i) {
        const long long ci = (long long)floor(in[0][i] / g.h) - g.phase[0];
        const long long cj = (long long)floor(in[1][i] / g.h) - g.phase[1];
        const long long ck = DIM == 3 ? (long long)floor(in[2][i] / g.h) - g.phase[2] : 0;
        if (ci < 0 || ci >= g.lim[0] || cj < 0 || cj >= g.lim[1] || ck < 0 || ck >= g.lim[2]) {
            fprintf(stderr, "emu_fluid_force: particle %lld is outside the box (not supported here)\n", (long long)i);
            return 3;
        }
        pkey[i] = pkey_ijk(g, (int)ci, (int)cj, (int)ck);
        col[i] = (uint32_t)ci;
        if (!carry_key.empty() && (carry_key[i] != pkey[i] || carry_col[i] != col[i])) {
            fprintf(stderr, "emu_fluid_force: the advance keyed particle %lld %u/%u, its position says %u/%u\n",
                    (long long)i, carry_key[i], carry_col[i], pkey[i], col[i]);
            return 1;
        }
    }
    std::iota(order.begin(), order.end(), 0u);
    std::sort(order.begin(), order.end(),
              [&](uint32_t a, uint32_t b) { return pkey[a] != pkey[b] ? pkey[a] < pkey[b] : a > b; });
    std::vector<double> cur[NSLOT], alt[NSLOT];
    for (int s = 0; s < NSLOT; ++s) {
        cur[s].assign(n + 4, 0.0);
        alt[s].assign(n + 4, 0.0);
    }
    std::vector<uint32_t> key(n), cellx(n), idx(n), xq(n + 4, 0u), cs(g.pkey_max + 2, 0u);
    std::vector<uint8_t> fl(n + 8, 0xEE);
    std::vector<NbRec> rec[3];
    for (int k = 0; k < 3; ++k) rec[k].assign(n, NbRec{0, 0, 0, 0});
    for (int64_t i = 0; i < n; ++i) cs[pkey[i] + 1] += 1;
    for (long long c = 0; c <= g.pkey_max; ++c) cs[c + 1] += cs[c];
    {
        std::vector<uint32_t> ident(n), tag_in(n, 0u), tag_out(n);
        std::iota(ident.begin(), ident.end(), 0u);
        GatherList gl;
        memset(&gl, 0, sizeof(gl));
        for (int a = 0; a < 3; ++a) gl.xpos[a] = -1;
        gl.mpos = -1;
        gl.tpos = -1;
        for (int k = 0; k < 11; ++k) {
            const int slot = IN_SLOTS[k];
            if (DIM == 2 && (slot == S_X2 || slot == S_V2)) continue;
            gl.from[gl.count] = in[k].data();
            gl.to[gl.count] = cur[slot].data();
            if (slot >= S_X0 && slot <= S_X2) gl.xpos[slot - S_X0] = gl.count;
            if (slot == S_M) gl.mpos = gl.count;
            if (slot == S_TYPE) gl.tpos = gl.count;
            ++gl.count;
        }
        gl.h = g.h;
        gl.q6 = g.zrun;
        gl.dim = DIM;
        gl.run_phase = g.phase[DIM == 3 ? 2 : 1];
        gl.xq = xq.data();
        gl.recA = rec[0].data();
        gl.fluid = prm.fluid;
        gl.fl = fl.data();
        launch(n, [&] {
            k_gather(gl, order.data(), ident.data(), idx.data(), nullptr, pkey.data(), key.data(), tag_in.data(),
                     tag_out.data(), col.data(), cellx.data(), n);
        });
    }
    // the fluid work list: fluid positions ascending, then the others ascending
    std::vector<uint32_t> work;
    for (int pass = 0; pass < 2; ++pass)
        for (int64_t p = 0; p < n; ++p) {
            if (fl[p] > 1) {
                fprintf(stderr, "emu_fluid_force: the gather left no fluid flag at position %lld\n", (long long)p);
                return 3;
            }
            if ((fl[p] == 1) == (pass == 0)) work.push_back((uint32_t)p);
        }
    uint32_t n_fluid = 0;
    for (int64_t p = 0; p < n; ++p) n_fluid += fl[p];
    out.warps_nonfluid = out.warps_mixed = 0;
    for (int64_t w = 0; w * 32 < n; ++w) {
        int k = 0, m = 0;
        for (int64_t p = w * 32; p < std::min<int64_t>(n, w * 32 + 32); ++p, ++m) k += fl[p];
        out.warps_nonfluid += k == 0;
        out.warps_mixed += k > 0 && k < m;
    }
    Fields fcur{}, falt{};
    for (int s = 0; s < NSLOT; ++s) {
        fcur.s[s] = cur[s].data();
        falt.s[s] = alt[s].data();
    }
    std::vector<uint32_t> list((size_t)((n + 31) / 32) * (size_t)stride * 32, 0u), cnt(n, 0u);
    unsigned long long counters[3] = {0, 0, 0};
    PairList pl{};
    pl.list = list.data();
    pl.cnt = cnt.data();
    pl.xq = xq.data();
    pl.stride = stride;
    pl.qrows = stride + NL_QUEUE_SLACK;
    pl.overflow = &counters[2];
    pl.recA = rec[0].data();
    pl.recB = rec[1].data();
    pl.recC = rec[2].data();
    const ColFilter cf{0, 0, (int)g.lim[0] - 1, 1, 0, 1};
    // back to reference index order: the force pass wrote v (and, with the advance, x) to alt
    constexpr bool ADV = !std::is_same<ForceOp, B_wcsph_momentum_fused>::value &&
                         !std::is_same<ForceOp, B_wcsph_momentum_fast>::value;
    std::vector<uint32_t> key_next(n, 0xFFFFFFFFu), col_next(n, 0xFFFFFFFFu), removed(16, 0u);
    if (ADV) {  // as pair_ops.cu run_fused_force on a whole-domain context
        prm.key_out = key_next.data();
        prm.cellx_out = col_next.data();
        prm.key_removed = removed.data();
        prm.key_idx = idx.data();
        prm.key_removed_cap = 15;
    }
    launch(n, [&] {
        k_binary_build<DIM, DensityOp, NL_FILTER_Q6, true>(fcur, fcur, prm, g, key.data(), cellx.data(), cs.data(), n, 0,
                                                           &counters[0], cf, pl);
    });
    launch(n, [&] {
        k_binary_list_fluid<DIM, ForceOp, true>(fcur, falt, prm, g, key.data(), cellx.data(), cs.data(), n, 0,
                                                &counters[1], cf, pl, work.data(), &n_fluid);
    });
    if (ADV && removed[0]) {
        fprintf(stderr, "emu_fluid_force: a particle left the box (not supported here)\n");
        return 3;
    }
    carry_key.assign(ADV ? n : 0, 0u);
    carry_col.assign(ADV ? n : 0, 0u);
    for (int64_t p = 0; p < n; ++p) {
        if (ADV) {
            carry_key[idx[p]] = key_next[p];
            carry_col[idx[p]] = col_next[p];
        }
        const uint32_t i = idx[p];
        in[8][i] = cur[S_RHO][p];
        in[9][i] = cur[S_RHO_P][p];
        in[7][i] = cur[S_H][p];
        for (int a = 0; a < DIM; ++a) {
            in[3 + a][i] = alt[S_V0 + a][p];
            in[a][i] = ADV ? alt[S_X0 + a][p] : cur[S_X0 + a][p];
        }
    }
    out.pairs = counters[1];
    out.n_fluid = n_fluid;
    return 0;
}

template <int DIM, class DensityOp, class ForceOp>
static int run_call(std::vector<double> (&in)[11], int64_t n, const Grid &g, const Params &prm, int stride, int nsteps,
                    Step &last) {
    // accelerate! + move! of the first step (step_wcsph_fused_pre)
    Fields master{};
    for (int k = 0; k < 11; ++k) master.s[IN_SLOTS[k]] = in[k].data();
    launch(n, [&] {
        const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
        if (p >= n) return;
        U_wcsph_accelerate<false>::apply<DIM>(master, prm, p);
        U_wcsph_move::apply<DIM>(master, prm, p);
    });
    std::vector<uint32_t> carry_key, carry_col;  // keys the previous step's advance wrote (reference order)
    for (int step = 0; step < nsteps; ++step) {
        const int rc = step + 1 < nsteps
                           ? run_step<DIM, DensityOp, B_force_advance<ForceOp>>(in, n, g, prm, stride, last, carry_key, carry_col)
                           : run_step<DIM, DensityOp, ForceOp>(in, n, g, prm, stride, last, carry_key, carry_col);
        if (rc) return rc;
    }
    return 0;
}

int main(int argc, char **argv) {
    if (argc != 3) {
        fprintf(stderr, "usage: emu_fluid_force <input.bin> <output.bin>\n");
        return 2;
    }
    FILE *fp = fopen(argv[1], "rb");
    if (!fp) {
        perror(argv[1]);
        return 2;
    }
    int32_t head[6];  // fast, stride, -, nparams, nsteps per call, calls
    int64_t n;
    double box[7];
    read_exact(fp, head, sizeof(head));
    read_exact(fp, &n, sizeof(n));
    read_exact(fp, box, sizeof(box));
    const int fast = head[0], stride = head[1], nparams = head[3], nsteps = head[4], calls = head[5];
    Params prm;
    memset(&prm, 0, sizeof(prm));
    struct Named {
        const char *name;
        double Params::*field;
    };
    static const Named TABLE[] = {{"dt", &Params::dt}, {"g", &Params::g}, {"c", &Params::c}, {"gamma", &Params::gamma},
                                  {"alpha", &Params::alpha}, {"beta", &Params::beta}, {"eps", &Params::eps},
                                  {"eta", &Params::eta}, {"rho0", &Params::rho0}, {"R_mass", &Params::R_mass},
                                  {"R_gas", &Params::R_gas}, {"T_bg", &Params::T_bg}, {"rho_floor", &Params::rho_floor},
                                  {"P_floor", &Params::P_floor}, {"z_t", &Params::z_t}, {"z_b", &Params::z_b},
                                  {"gamma_r", &Params::gamma_r}, {"fluid", &Params::fluid}};
    for (int k = 0; k < nparams; ++k) {
        char name[16];
        double value;
        read_exact(fp, name, 16);
        read_exact(fp, &value, sizeof(value));
        name[15] = 0;
        for (const Named &t : TABLE)
            if (!strcmp(t.name, name)) prm.*(t.field) = value;
    }
    sphmw_derive_params(prm);
    Grid g;
    memset(&g, 0, sizeof(g));
    int64_t global_cols = 0;
    if (sphmw_grid_setup(g, box, box + 3, box[6], -1, -1, &global_cols) != SPHMW_OK) return 3;
    sphmw_grid_set_order(g, true);
    std::vector<double> in[11];
    for (int k = 0; k < 11; ++k) {
        in[k].resize(n);
        read_exact(fp, in[k].data(), sizeof(double) * n);
    }
    fclose(fp);

    Step last;
    for (int call = 0; call < calls; ++call) {
        int rc;
        if (g.dim == 2)
            rc = fast ? run_call<2, B_wcsph_density_fast, B_wcsph_momentum_fast>(in, n, g, prm, stride, nsteps, last)
                      : run_call<2, B_wcsph_density_fused, B_wcsph_momentum_fused>(in, n, g, prm, stride, nsteps, last);
        else
            rc = fast ? run_call<3, B_wcsph_density_fast, B_wcsph_momentum_fast>(in, n, g, prm, stride, nsteps, last)
                      : run_call<3, B_wcsph_density_fused, B_wcsph_momentum_fused>(in, n, g, prm, stride, nsteps, last);
        if (rc) return rc;
    }
    FILE *out = fopen(argv[2], "wb");
    if (!out) {
        perror(argv[2]);
        return 2;
    }
    const int64_t meta[6] = {n, g.dim, (int64_t)last.pairs, (int64_t)last.n_fluid, last.warps_nonfluid, last.warps_mixed};
    fwrite(meta, sizeof(meta), 1, out);
    fwrite(in[8].data(), sizeof(double), n, out);                                  // rho
    fwrite(in[7].data(), sizeof(double), n, out);                                  // h
    for (int k = 0; k < 3; ++k) fwrite(in[3 + k].data(), sizeof(double), n, out);  // v
    for (int k = 0; k < 3; ++k) fwrite(in[k].data(), sizeof(double), n, out);      // x
    fclose(out);
    printf("emu_fluid_force: %d calls of %d steps, n=%lld dim=%d fluid=%u pairs=%llu\n", calls, nsteps, (long long)n,
           g.dim, last.n_fluid, last.pairs);
    return 0;
}
