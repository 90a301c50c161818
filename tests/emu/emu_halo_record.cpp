// The halo record layout of libsphmw (csrc/halo_record.cuh) on the host — TEST INFRASTRUCTURE, never
// shipped.  Compiled with g++ behind tests/emu/cuda_runtime.h, the very helpers k_halo_pack and
// k_halo_unpack inline are checked against
//   * the layout the base record had before it moved into the header (written out literally below):
//     row for row, for 2D and 3D and every carry_a (rho/rho', A, A + A_bg), pack and unpack;
//   * a round trip of the adiabatic record into a slot full of garbage: x, v, m, h, rho, rho', type,
//     index, S, P, T and theta come back bit for bit, s and Dv are zero, and its first rows are the
//     base record.
// usage: emu_halo_record   (prints HALO_RECORD_OK, or the failures and exits with 1)
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <random>
#include <vector>

#include "cuda_runtime.h"
#include "halo_record.cuh"

uint3 threadIdx, blockIdx, blockDim, gridDim;

static int failures = 0;
#define CHECK(cond, ...)                  \
    do {                                  \
        if (!(cond)) {                    \
            fprintf(stderr, __VA_ARGS__); \
            fputc('\n', stderr);          \
            ++failures;                   \
        }                                 \
    } while (0)

static bool same_bits(double a, double b) { return memcmp(&a, &b, sizeof(double)) == 0; }

// the base record as k_halo_pack / k_halo_unpack wrote and read it inline
template <int DIM>
static void old_pack(const Fields &f, const uint32_t *idx, int64_t p, double kind, int carry_a, double *rec) {
    rec[0] = f.s[S_X0][p];
    rec[1] = f.s[S_X1][p];
    rec[2] = DIM == 3 ? f.s[S_X2][p] : 0.0;
    rec[3] = f.s[S_V0][p];
    rec[4] = f.s[S_V1][p];
    rec[5] = DIM == 3 ? f.s[S_V2][p] : 0.0;
    rec[6] = f.s[S_M][p];
    rec[7] = f.s[S_H][p];
    rec[8] = carry_a ? f.s[S_A][p] : f.s[S_RHO][p];
    rec[9] = carry_a ? (carry_a > 1 ? f.s[S_A_BG][p] : 0.0) : f.s[S_RHO_P][p];
    rec[10] = f.s[S_TYPE][p];
    rec[11] = (double)idx[p];
    rec[12] = kind;
}
template <int DIM>
static void old_unpack(const Fields &f, uint32_t *idx, uint32_t *tag, int64_t p, const double *rec, int carry_a) {
    f.s[S_X0][p] = rec[0];
    f.s[S_X1][p] = rec[1];
    if (DIM == 3) f.s[S_X2][p] = rec[2];
    f.s[S_V0][p] = rec[3];
    f.s[S_V1][p] = rec[4];
    if (DIM == 3) f.s[S_V2][p] = rec[5];
    f.s[S_M][p] = rec[6];
    f.s[S_H][p] = rec[7];
    if (carry_a) {
        f.s[S_A][p] = rec[8];
        if (carry_a > 1) f.s[S_A_BG][p] = rec[9];
    } else {
        f.s[S_RHO][p] = rec[8];
        f.s[S_RHO_P][p] = rec[9];
    }
    f.s[S_TYPE][p] = rec[10];
    idx[p] = (uint32_t)rec[11];
    tag[p] = rec[12] == HALO_KIND_MIGRANT ? TAG_OWNED : TAG_GHOST;
    if (f.s[S_DRHO]) f.s[S_DRHO][p] = 0.0;
    if (f.s[S_DV0]) f.s[S_DV0][p] = 0.0;
    if (f.s[S_DV1]) f.s[S_DV1][p] = 0.0;
    if (DIM == 3 && f.s[S_DV2]) f.s[S_DV2][p] = 0.0;
}

// every slot of n particles holds random bits (finite or not: the copy must not care)
struct State {
    int64_t n;
    std::vector<std::vector<double>> slot;
    std::vector<uint32_t> idx, tag;
    Fields f{};
    State(int64_t n_, std::mt19937_64 &rng) : n(n_), slot(NSLOT, std::vector<double>(n_)), idx(n_), tag(n_) {
        for (int s = 0; s < NSLOT; ++s) {
            for (auto &v : slot[s]) {
                const uint64_t bits = rng();
                memcpy(&v, &bits, sizeof(v));
            }
            f.s[s] = slot[s].data();
        }
        for (auto &i : idx) i = (uint32_t)(rng() & 0xffffffu);
        for (auto &t : tag) t = (uint32_t)rng();
    }
};

template <int DIM>
static void check_base(std::mt19937_64 &rng) {
    const int64_t n = 64;
    State src(n, rng);
    for (int carry_a = 0; carry_a <= 2; ++carry_a)
        for (int64_t p = 0; p < n; ++p) {
            const double kind = (p & 1) ? HALO_KIND_GHOST : HALO_KIND_MIGRANT;
            double want[HALO_RECORD], got[HALO_RECORD];
            old_pack<DIM>(src.f, src.idx.data(), p, kind, carry_a, want);
            const double z = DIM == 3 ? src.f.s[S_X2][p] : 0.0;
            halo_record_pack<DIM, HALO_REC_BASE>(src.f, src.idx.data(), p, src.f.s[S_X0][p], src.f.s[S_X1][p], z, kind,
                                                 carry_a, got);
            for (int k = 0; k < HALO_RECORD; ++k)
                CHECK(same_bits(want[k], got[k]), "base record, %dD, carry_a %d: row %d differs from the old layout", DIM,
                      carry_a, k);
            // unpack into two copies of the same garbage: every slot, index and tag must agree
            State a(n, rng);
            State b = a;
            for (int s = 0; s < NSLOT; ++s) b.f.s[s] = b.slot[s].data();
            old_unpack<DIM>(a.f, a.idx.data(), a.tag.data(), p, want, carry_a);
            halo_record_unpack<DIM, HALO_REC_BASE>(b.f, b.idx.data(), b.tag.data(), p, want, carry_a);
            for (int s = 0; s < NSLOT; ++s)
                CHECK(same_bits(a.slot[s][p], b.slot[s][p]), "base unpack, %dD, carry_a %d: slot %d differs", DIM, carry_a, s);
            CHECK(a.idx[p] == b.idx[p] && a.tag[p] == b.tag[p], "base unpack, %dD: index or tag differs", DIM);
        }
}

template <int DIM>
static void check_adiabatic(std::mt19937_64 &rng) {
    static_assert(halo_record_rows(HALO_REC_ADIABATIC) == 17, "the adiabatic record has 17 rows");
    const int64_t n = 64;
    State src(n, rng);
    for (int64_t p = 0; p < n; ++p) {
        const double kind = (p & 1) ? HALO_KIND_GHOST : HALO_KIND_MIGRANT;
        double rec[HALO_RECORD_ADIABATIC], base[HALO_RECORD];
        const double z = DIM == 3 ? src.f.s[S_X2][p] : 0.0;
        halo_record_pack<DIM, HALO_REC_ADIABATIC>(src.f, src.idx.data(), p, src.f.s[S_X0][p], src.f.s[S_X1][p], z, kind, 0,
                                                  rec);
        halo_record_pack<DIM, HALO_REC_BASE>(src.f, src.idx.data(), p, src.f.s[S_X0][p], src.f.s[S_X1][p], z, kind, 0, base);
        for (int k = 0; k < HALO_RECORD; ++k)
            CHECK(same_bits(rec[k], base[k]), "adiabatic record, %dD: row %d is not the base record's", DIM, k);
        State dst(n, rng);
        const int64_t q = n - 1 - p;
        halo_record_unpack<DIM, HALO_REC_ADIABATIC>(dst.f, dst.idx.data(), dst.tag.data(), q, rec, 0);
        int carried[] = {S_X0, S_X1, S_X2, S_V0, S_V1, S_V2, S_M, S_H, S_RHO, S_RHO_P, S_TYPE, S_ENT, S_P, S_T, S_TH};
        for (int s : carried) {
            if (DIM == 2 && (s == S_X2 || s == S_V2)) continue;
            CHECK(same_bits(dst.slot[s][q], src.slot[s][p]), "adiabatic round trip, %dD: slot %d not restored", DIM, s);
        }
        CHECK(dst.idx[q] == src.idx[p], "adiabatic round trip, %dD: global index not restored", DIM);
        CHECK(dst.tag[q] == (kind == HALO_KIND_MIGRANT ? TAG_OWNED : TAG_GHOST), "adiabatic round trip, %dD: tag", DIM);
        for (int s : {S_ENT_D, S_DV0, S_DV1, S_DV2, S_DRHO}) {
            if (DIM == 2 && s == S_DV2) continue;
            CHECK(same_bits(dst.slot[s][q], 0.0), "adiabatic round trip, %dD: slot %d is not zero", DIM, s);
        }
    }
}

int main() {
    std::mt19937_64 rng(20261020);
    check_base<2>(rng);
    check_base<3>(rng);
    check_adiabatic<2>(rng);
    check_adiabatic<3>(rng);
    if (failures) {
        fprintf(stderr, "%d failure(s)\n", failures);
        return 1;
    }
    printf("HALO_RECORD_OK\n");
    return 0;
}
