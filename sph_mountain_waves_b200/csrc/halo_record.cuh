// Row layout of an x-slab halo record (halo.cu packs and unpacks them, slab_comm.cu sizes its NCCL
// messages by them).  Host and device: tests/emu/emu_halo_record.cpp checks the layout on the CPU.
//
// BASE record, 13 rows — every context that does not hold the entropy S:
//   0-2 x   3-5 v   6 m   7 h   8/9 rho, rho'   10 type   11 global index   12 kind (migrant / ghost)
//   For the pressure-entropy drivers (carry_a > 0) rows 8/9 are A and A_bg (or 0.0): carried state
//   there, while the densities are recomputed by the receiver.
// ADIABATIC record, 17 rows — contexts that hold S (legacy/adiabatic_flow_witch.jl, scheme "aflow"):
//   the base rows, then 13 S  14 P  15 T  16 theta
//   S      carried state: entropy_production! accumulates it (ops_menu.cuh B_aflow_entropy)
//   theta  never recomputed by the step (only make_system's find_pot_temp! sets it): a FLUID migrant
//          brings its own
//   P, T   recomputed for FLUID only (U_aflow_find_pressure is type-gated): WALL and MOUNTAIN ghosts keep
//          their constructor values, which internal_force! reads (P), and an INFLOW successor born on
//          the far side of a slab face needs its constructor P, T and theta
//   s (the entropy density) is not carried: find_s! recomputes it for FLUID before any use, so the
//   receiver sets it to the constructor's zero, like the accumulators Dv and Drho.
#pragma once
#include "sphmw_internal.h"

enum HaloRecordKind : int { HALO_REC_BASE = 0, HALO_REC_ADIABATIC = 1 };
#define HALO_RECORD_ADIABATIC 17
#define HALO_ROW_TYPE 10
#define HALO_ROW_IDX 11
#define HALO_ROW_KIND 12

__host__ __device__ constexpr int halo_record_rows(int kind) {
    return kind == HALO_REC_ADIABATIC ? HALO_RECORD_ADIABATIC : HALO_RECORD;
}

// fills rec[0 .. halo_record_rows(KIND)) for particle p at position (x, y, z); idx: global indices
template <int DIM, int KIND>
__host__ __device__ __forceinline__ void halo_record_pack(const Fields &f, const uint32_t *idx, int64_t p, double x, double y,
                                                          double z, double kind, int carry_a, double *rec) {
    rec[0] = x;
    rec[1] = y;
    rec[2] = z;
    rec[3] = f.s[S_V0][p];
    rec[4] = f.s[S_V1][p];
    rec[5] = DIM == 3 ? f.s[S_V2][p] : 0.0;
    rec[6] = f.s[S_M][p];
    rec[7] = f.s[S_H][p];
    rec[8] = carry_a ? f.s[S_A][p] : f.s[S_RHO][p];
    rec[9] = carry_a ? (carry_a > 1 ? f.s[S_A_BG][p] : 0.0) : f.s[S_RHO_P][p];
    rec[HALO_ROW_TYPE] = f.s[S_TYPE][p];
    rec[HALO_ROW_IDX] = (double)idx[p];
    rec[HALO_ROW_KIND] = kind;
    if (KIND == HALO_REC_ADIABATIC) {
        rec[13] = f.s[S_ENT][p];
        rec[14] = f.s[S_P][p];
        rec[15] = f.s[S_T][p];
        rec[16] = f.s[S_TH][p];
    }
}

// writes record rec into slot p: the carried fields, the global index and the tag (a migrant becomes
// owned, a ghost copy stays a ghost); zeroes what the receiver recomputes
template <int DIM, int KIND>
__host__ __device__ __forceinline__ void halo_record_unpack(const Fields &f, uint32_t *idx, uint32_t *tag, int64_t p,
                                                            const double *rec, int carry_a) {
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
    f.s[S_TYPE][p] = rec[HALO_ROW_TYPE];
    idx[p] = (uint32_t)rec[HALO_ROW_IDX];
    tag[p] = rec[HALO_ROW_KIND] == HALO_KIND_MIGRANT ? TAG_OWNED : TAG_GHOST;
    // accumulators of the op-by-op schemes: the sender's move! / find_pressure! left them zero
    // (isothermal_flow_witch.jl:157,205), the slot here may hold anything
    if (f.s[S_DRHO]) f.s[S_DRHO][p] = 0.0;
    if (f.s[S_DV0]) f.s[S_DV0][p] = 0.0;
    if (f.s[S_DV1]) f.s[S_DV1][p] = 0.0;
    if (DIM == 3 && f.s[S_DV2]) f.s[S_DV2][p] = 0.0;
    if (KIND == HALO_REC_ADIABATIC) {
        f.s[S_ENT][p] = rec[13];
        f.s[S_P][p] = rec[14];
        f.s[S_T][p] = rec[15];
        f.s[S_TH][p] = rec[16];
        if (f.s[S_ENT_D]) f.s[S_ENT_D][p] = 0.0;  // s: the constructor's zero until find_s!
    }
}
