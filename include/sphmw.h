/*
 * sphmw.h — C ABI of libsphmw.so, the B200-native WCSPH hot path behind the
 * SmoothedParticles.jl API used by moschehaus/sph-mountain-waves.
 *
 * The reference has no FFI boundary of its own (it is 100 % Julia); the boundary
 * it does have is its Julia API (src/SmoothedParticles.jl:14-79).  Every entry
 * point below names the reference interface it replaces (file:line under
 * /root/reference).  INTEGRATION.md shows the `ccall` shim a maintainer adds.
 *
 * Conventions
 *   - plain C: opaque handle, pointers and sizes; no C++/torch types.
 *   - every call returns 0 (SPHMW_OK) or a negative SPHMW_E_* code; the message
 *     of the last failure on the calling thread is sphmw_last_error().
 *   - host buffers are BORROWED for the duration of the call; device memory is
 *     OWNED by the context.  Buffers passed to upload/download may also be device
 *     pointers (UVA decides).
 *   - particle fields cross the ABI as structure-of-arrays, component-major:
 *     buf[c*n + i] is component c of particle i, i in the reference's particle
 *     index order (`sys.particles[i+1]`).
 *   - a context is driven by one host thread at a time (the reference's caller is
 *     single-threaded, core.jl:125-142 fans out internally).
 *   - all work is enqueued on the context's stream; only download, reduce,
 *     create_cell_list(n_alive != NULL), pairs/keys dumps and sync block.
 *   - there is NO CPU fallback: without a CUDA device sphmw_create fails.
 */
#ifndef SPHMW_H
#define SPHMW_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPHMW_OK 0
#define SPHMW_E_INVALID (-1)        /* bad argument (AssertionError in the reference) */
#define SPHMW_E_CUDA (-2)           /* CUDA runtime failure */
#define SPHMW_E_UNSUPPORTED_OP (-3) /* operator not in the menu: no CPU fallback */
#define SPHMW_E_UNKNOWN_FIELD (-4)
#define SPHMW_E_CAPACITY (-5)
#define SPHMW_E_STATE (-6)          /* e.g. binary op before create_cell_list */
#define SPHMW_E_IO (-7)

typedef struct sphmw_ctx sphmw_ctx;

/* ≙ ParticleSystem(T, domain, h) — src/structs.jl:57-91.  `box_*` is
 * boundarybox(domain) (structs.jl:63-65); 2D is detected exactly like the
 * reference: key_lim[3] == 1 (structs.jl:70).
 * Slab fields (multi-GPU, no reference equivalent): this context owns the global
 * cell columns [slab_lo, slab_hi) along x and keeps two ghost columns each side;
 * slab_lo = slab_hi = -1 means "whole domain". */
typedef struct sphmw_config {
    double box_min[3];
    double box_max[3];
    double h;
    int64_t capacity; /* max particles resident (owned + ghosts) */
    int32_t device;   /* CUDA ordinal */
    int32_t flags;    /* SPHMW_FLAG_* */
    int64_t slab_lo;
    int64_t slab_hi;
} sphmw_config;

#define SPHMW_FLAG_NONE 0
/* fused "wcsph" step only.  Default (0): strict arithmetic — no FMA contraction, IEEE
 * division/sqrt, so every FP64 sum is bit-identical to an IEEE evaluation of the reference
 * closures.  FAST_MATH: same neighbour set and summation order, but fused multiply-adds and
 * reciprocals in the closure bodies (as the reference's own @fastmath kernels allow);
 * fields agree with the strict path to ~1e-15 relative per step.  CELL_PAIRS: experimental
 * cell-centric pair-parallel kernel (strict arithmetic, bit-identical results). */
#define SPHMW_FLAG_FAST_MATH 1
#define SPHMW_FLAG_CELL_PAIRS 2
/* Pair list (no reference equivalent; results are unchanged bit for bit).  By default the first
 * binary pass after a create_cell_list! records each particle's accepted neighbours in traversal order
 * when the previous cell list saw two or more binary passes (always inside the fused "wcsph"
 * step), and later passes on the same cell list read that list instead of walking the 9/27
 * neighbour cells again.  NO_PAIR_LIST: always walk the cells.  PAIR_LIST_EAGER: record on the
 * first pass of every cell list.  NO_PRETEST: the recording pass tests candidates in FP64 only
 * (default: conservative integer pre-test on a 6-bit mirror of each particle's position inside its
 * cell — one packed add and one DP4A per candidate —, exact FP64 test for the survivors). */
#define SPHMW_FLAG_NO_PAIR_LIST 4
#define SPHMW_FLAG_PAIR_LIST_EAGER 8
#define SPHMW_FLAG_NO_PRETEST 16
/* Fused "wcsph" step only.  By default its two pair passes read their neighbours from three packed
 * 32-byte records ({x,y,z,m} written by the cell-list gather, {v,h} and {P'/rho^2, rho, c_s} written
 * by the density pass) with one 256-bit load each instead of eleven 8-byte gathers (+96 B per
 * particle; the records are bit copies of the SoA fields, so no sum changes).  Measured on B200,
 * 64 M particles: step 48.5 -> 42.1 ms (profiles/r02_pair_kernels.md).  NO_PACKED_RECORDS: gather
 * from the SoA arrays.  The records are the default in 3D; in 2D (9 neighbour fields instead of 11) the SoA
 * gathers are 6 % faster and stay the default, PACKED_RECORDS switches the records on there.
 * Ignored together with NO_PAIR_LIST / CELL_PAIRS. */
#define SPHMW_FLAG_PACKED_RECORDS 32
#define SPHMW_FLAG_NO_PACKED_RECORDS 128
/* Fused "wcsph" step only, experimental (default off).  TILES: the two pair passes stage the
 * neighbourhood of every block of 128 particles in shared memory (coalesced 16-byte copies, or
 * cp.async.bulk/TMA when built with TILE_STAGE_TMA) and gather neighbour fields from there; the
 * pair list then holds 16-bit tile slots of the accepted neighbours (same visiting order, same
 * bits).  Correct (CPU emulation and GPU tests) but 2.5x slower than the record path on B200:
 * a tile of 115 KB per 4 warps leaves 8 warps per SM and the per-thread dependent chains are no
 * longer hidden (profiles/r02_pair_kernels.md).  Ignored together with NO_PAIR_LIST / CELL_PAIRS /
 * NO_PRETEST. */
#define SPHMW_FLAG_TILES 64
/* Slab contexts, at sphmw_create only: keep THREE ghost columns per side instead of two.  Needed by
 * the pressure-entropy (Hopkins) schemes, whose pressure sum reads the new smoothing length of a
 * particle's neighbours (hopkins_perturbed_witch.jl:205-208), i.e. complete density sums two columns
 * beyond the owned ones.  Such a context steps "hopkins"/"hopkins_full" (and "wcsph", on the plain
 * schedule: the overlapped one is laid out for two ghost columns). */
#define SPHMW_FLAG_GHOST3 256

int sphmw_create(const sphmw_config *cfg, sphmw_ctx **out);
int sphmw_destroy(sphmw_ctx *ctx);
const char *sphmw_last_error(void);
const char *sphmw_version(void);

/* Use the caller's CUDA stream (cudaStream_t as void*); NULL = context's own. */
int sphmw_set_stream(sphmw_ctx *ctx, void *cuda_stream);
int sphmw_sync(sphmw_ctx *ctx);
/* switch the arithmetic / kernel variant of the fused step (SPHMW_FLAG_*) */
int sphmw_set_flags(sphmw_ctx *ctx, int32_t flags);

/* Driver constants, ≙ the module-level `const`s of a driver
 * (src/current/wcsph_perturbed_witch.jl:25-75; collapse_dry.jl:30-66).
 * Names: dt g c gamma alpha beta eps eta rho0 R_mass R_gas T_bg rho_floor P_floor
 * z_t z_b gamma_r fluid m nu mu gx gy gz kh dt_pack c_pack zeta_pack
 * U_max cp bc_width x_inflow dr inflow */
int sphmw_set_param(sphmw_ctx *ctx, const char *name, double value);
int sphmw_get_param(sphmw_ctx *ctx, const char *name, double *value);

/* key tables of the system — src/structs.jl:66-68 */
int sphmw_key_tables(sphmw_ctx *ctx, int64_t phase[3], int64_t lim[3], int64_t *key_max,
                     int32_t *dim);

/* ≙ push!(sys.particles, ...) / length(sys.particles) — src/grids.jl:305-310.
 * Sets the particle count; new particles have all fields zero. */
int sphmw_resize(sphmw_ctx *ctx, int64_t n);
int sphmw_count(sphmw_ctx *ctx, int64_t *n);

/* ≙ ParticleField(sys, :name) get/set — src/structs.jl:118-125.
 * Field names (ASCII | Julia): h x m v Dv rho_bg|ρ_bg rho_p|ρ′ rho|ρ P_bg P_p|P′ P
 * theta_bg|θ_bg theta_p|θ′ theta|θ T_bg T_p|T′ T type A A_bg Drho rho0 a(=Dv) u(=v).
 * ncomp must be 1 (scalars) or 3 (RealVector).  n must equal the particle count. */
int sphmw_upload(sphmw_ctx *ctx, const char *field, const double *buf, int64_t n, int32_t ncomp);
int sphmw_download(sphmw_ctx *ctx, const char *field, double *buf, int64_t n, int32_t ncomp);

/* ≙ create_cell_list!(sys) — src/core.jl:51-90: removal of out-of-box particles
 * with the reference's swap-from-end renumbering, cell keys (structs.jl:97-106),
 * sort by (cell, index descending), cell-start table.  n_alive may be NULL
 * (then the call does not block). */
int sphmw_create_cell_list(sphmw_ctx *ctx, int64_t *n_alive);

/* ≙ apply!(sys, f; self) / apply_unary! / apply_binary! — src/core.jl:125-161.
 * `op` is "<scheme>.<closure>" from the fixed menu (sphmw_op_list), e.g.
 * "wcsph.compute_density" ≙ wcsph_perturbed_witch.jl:226-228.  A closure that is
 * not in the menu is SPHMW_E_UNSUPPORTED_OP.  Arity (unary/binary) is a
 * property of the operator, as `hasmethod` decides in core.jl:153. */
int sphmw_apply(sphmw_ctx *ctx, const char *op, int32_t self);
/* newline-separated operator names; returns the length needed */
int64_t sphmw_op_list(char *buf, int64_t cap);

/* Fused fast path ≙ `for k in 1:nsteps verlet_step!(sys) end`
 * (wcsph_perturbed_witch.jl:309-332, :371-373).  scheme: "wcsph" | "hopkins" |
 * "hopkins_full" | "hopkins_total" | "dambreak" | "collision" | "flow".  Must leave the same state as the
 * operator-by-operator sequence. */
int sphmw_step(sphmw_ctx *ctx, const char *scheme, int32_t nsteps);

/* ≙ make_system() of the mountain-wave drivers on the device —
 * src/current/wcsph_perturbed_witch.jl:152-170 with src/grids.jl:50-93,176-196 (square,
 * hexagonal, cubic lattices) and src/geometry.jl:15-43,176-232 (Rectangle/Box domain,
 * BoundaryLayer fence, mountain Specification).  Appends, in the reference's particle order
 * (fluid bulk, wall fence, mountain; lattice index i outermost), the particles of
 *   domain - mountain (type_fluid, v = U x̂), fence (type_wall), mountain (type_mountain)
 * with the fields the step carries (h, x, m, v, rho, rho', type) set as the driver's Particle
 * constructor does (:103-145; rho0, g, R_mass, T_bg from sphmw_set_param).  mountain: 0 none,
 * 1 Witch of Agnesi y <= h_m a^2/(x^2+a^2) (2D), 2 bell hill y <= h_m/(1+(x^2+z^2)/a^2)^1.5.
 * On a slab context only the sites of the owned cell columns are generated. */
typedef struct sphmw_lattice_setup {
    int32_t grid;     /* 0 :square, 1 :hexagonal, 2 :cubic */
    int32_t mountain;
    double dr;
    double dom_min[3];
    double dom_max[3];
    double bc_width;
    double h_m, a, U;
    double type_fluid, type_wall, type_mountain;
    double h0;
} sphmw_lattice_setup;
int sphmw_generate_mountain_wave(sphmw_ctx *ctx, const sphmw_lattice_setup *setup, int64_t *n_out,
                                 int64_t group_counts[3]);

/* ≙ add_new_particles!(sys) of the constant-U flow drivers —
 * src/legacy/isothermal_flow_witch.jl:175-186: every INFLOW particle that has entered the
 * domain (x[1] >= x_inflow) becomes FLUID and a new INFLOW particle is appended bc_width
 * upstream of it, built like the driver's Particle constructor (:72-82).  New particles get
 * the next indices in the order the reference's loop would create them.  Parameters used:
 * inflow, fluid, x_inflow, bc_width, U_max, dr, rho0, g, R_mass, R_gas, cp, T_bg. */
int sphmw_flow_add_new_particles(sphmw_ctx *ctx, int64_t *n_added);
/* the same for the adiabatic variant of the driver — src/legacy/adiabatic_flow_witch.jl:197-208,
 * Particle constructor :82-91: T = T0 (parameter T_bg), hydrostatic rho, m = rho dr^2, P = R_mass T rho,
 * theta, and the entropy S = m cv log(cv T (gamma - 1) / (gamma rho^(gamma - 1))), cv = cp - R_mass.
 * Its closures are the operators "aflow.*" (+ "flow.accelerate", "flow.internal_force", which the two
 * drivers share character for character); sphmw_step(ctx, "aflow", n) is its verlet_step! (:231-243). */
int sphmw_aflow_add_new_particles(sphmw_ctx *ctx, int64_t *n_added);

/* Test hooks for bit-exact cell assignment / neighbour-pair parity. */
/* 0-based cell key of every particle, reference index order (structs.jl:97-106) */
int sphmw_cell_keys(sphmw_ctx *ctx, int64_t *keys, int64_t n);
/* particle indices stored in one cell, in stored order (core.jl:26-41) */
int sphmw_cell_entries(sphmw_ctx *ctx, int64_t key, int64_t *out, int64_t cap, int64_t *n);
/* accepted pairs (r <= h, p != q) in the reference's traversal order
 * (core.jl:94-112); fills at most cap, *n = total */
int sphmw_pairs_dump(sphmw_ctx *ctx, int64_t *pi, int64_t *pj, int64_t cap, int64_t *n);
/* accepted pairs of the last binary pass (needs sphmw_count_pairs(ctx,1)) */
int sphmw_count_pairs(sphmw_ctx *ctx, int32_t enable);
int sphmw_pair_count(sphmw_ctx *ctx, int64_t *n);

/* pair-list bookkeeping: out[0] entries per particle (stride), out[1] lists built so far,
 * out[2] particles whose candidates did not fit the stride (they walk the cells instead),
 * out[3] bytes of device memory held by the list.  Blocks. */
int sphmw_pair_list_info(sphmw_ctx *ctx, int64_t out[4]);
/* shared-memory tiles of the fused pair passes (current cell list): out[0] blocks of 128 particles,
 * out[1] blocks whose neighbourhood is staged in shared memory, out[2] slots of the largest
 * neighbourhood, out[3] slots of all staged neighbourhoods, out[4] slots a tile can hold,
 * out[5] blocks spread over too many rows of cells to be tiled.  Blocks. */
int sphmw_tile_info(sphmw_ctx *ctx, int64_t out[6]);

/* Host-only test hooks (no device, no context).
 * sphmw_pretest_pairs: the integer pre-test of the pair-list recording pass on n pairs
 * (xp, xq: n x 3 doubles): pass[i] = 1 passes, 0 rejected, 2 q is not in one of p's 27 cells.
 * Every pair with r <= h must pass.  (10-bit mirror of the x-chunked cell order, SPHMW_FLAG_TILES.)
 * sphmw_slab_column_sets: the column sets of the overlapped slab step for a context `width`
 * local columns wide (ghosts included): out = {edge, interior, force_edge, force_interior} x
 * {a0, a1, b0, b1}, each set [a0,a1] U [b0,b1] (empty when first > last). */
int sphmw_pretest_pairs(const double *xp, const double *xq, int64_t n, double h, int32_t dim,
                        uint8_t *pass);
/* the same for the 6-bit pre-test of the default (zrun) cell order: one packed add + DP4A */
int sphmw_pretest_pairs_q6(const double *xp, const double *xq, int64_t n, double h, int32_t dim,
                           uint8_t *pass);
int sphmw_slab_column_sets(int32_t width, int32_t has_left, int32_t has_right, int32_t out[16]);
/* sphmw_swap_removal_moves: the removal loop of create_cell_list! (src/core.jl:72-81) on index space —
 * `removed` (k distinct 0-based indices, any order) leave an array of n; out: the survivors whose index
 * changes, old -> new (at most k of them; arrays of k entries suffice).  What the cell-list build and
 * the open box of the slab transport replay. */
int sphmw_swap_removal_moves(int64_t n, const int64_t *removed, int64_t k, int64_t *old_index,
                             int64_t *new_index, int64_t *n_moves);

/* ≙ avg_velocity / max_velocity / length(sys.particles)
 * (wcsph_perturbed_witch.jl:338-350,377).  what: "avg_speed" | "max_speed" |
 * "count" | "sum:<field>" | "max:<field>" */
int sphmw_reduce(sphmw_ctx *ctx, const char *what, double *out);

/* ≙ the exported smoothing kernels, evaluated on the device — src/kernels.jl.
 * name: wendland1|2|3, Dwendland1|2|3, rDwendland1|2|3, DDwendland3,
 * spline23|24, Dspline23|24, rDspline23|24.  h, r, out: n doubles (host). */
int sphmw_kernel_eval(const char *name, const double *h, const double *r, double *out,
                      int64_t n, int32_t device);

/* ≙ new_pvd_file / save_frame! / save_pvd_file — src/IO.jl:20-75.  Frames are
 * written as VTK PolyData (.vtp, appended raw, one Verts cell per particle) plus
 * a .pvd collection whose timestep values are the frame counter (IO.jl:73). */
int sphmw_pvd_open(sphmw_ctx *ctx, const char *dir);
/* save_frame captures the frame on the device (reference index order, components interleaved as
 * the .vtp stores them), copies it to pinned host memory on a side stream and writes the file on a
 * worker thread: the call returns once the capture is queued and the time loop goes on.  pvd_close
 * (and sphmw_destroy) wait for the files. */
int sphmw_pvd_save_frame(sphmw_ctx *ctx, const char *const *fields, int32_t nfields);
int sphmw_pvd_close(sphmw_ctx *ctx);

/* The same capture for callers that want the arrays instead of a file.  sphmw_frame_capture: snapshot
 * of the named fields now, device -> pinned host copy queued on a side stream, *slot = 0 or 1 (two
 * captures can be in flight).  sphmw_frame_wait: waits for that copy; host[f] points at field f
 * (n x ncomp doubles, components interleaved; reference index order, physical order on a slab
 * context) inside the library's pinned buffer, valid until the second capture from now.
 * sphmw_upload_async stages a field on the copy stream (host memory borrowed until the commit);
 * sphmw_upload_commit makes the staged batch the particle state (count n, indices 0..n-1 in upload
 * order) on the main stream without waiting on the host. */
int sphmw_frame_capture(sphmw_ctx *ctx, const char *const *fields, int32_t nfields, int32_t *slot);
int sphmw_frame_wait(sphmw_ctx *ctx, int32_t slot, const double **host, int32_t nfields, int64_t *n);
int sphmw_upload_async(sphmw_ctx *ctx, const char *field, const double *buf, int64_t n, int32_t ncomp);
int sphmw_upload_commit(sphmw_ctx *ctx);
/* slab contexts: the global particle indices of the staged batch (≙ sphmw_set_index after the
 * commit, without its host wait) — staged like a field, applied by sphmw_upload_commit */
int sphmw_upload_index_async(sphmw_ctx *ctx, const int64_t *global_idx, int64_t n);

/* ≙ the file half of import_particles!(sys, path, ctor) — src/IO.jl:83-122 (ReadVTK.jl): a
 * host-only reader of the PolyData files WriteVTK (and sphmw_pvd_save_frame) writes.  Array 0
 * is "Points"; values come back as doubles, interleaved per point as stored. */
typedef struct sphmw_vtp sphmw_vtp;
int sphmw_vtp_open(const char *path, sphmw_vtp **out);
int sphmw_vtp_close(sphmw_vtp *vtp);
int sphmw_vtp_info(sphmw_vtp *vtp, int64_t *n_points, int32_t *n_arrays);
int sphmw_vtp_array(sphmw_vtp *vtp, int32_t i, char *name, int64_t cap, int32_t *ncomp);
int sphmw_vtp_read(sphmw_vtp *vtp, const char *name, double *out, int64_t n_values);
/* stand-alone writer of the same format (what save_frame! emits for one frame) */
int sphmw_vtp_write(const char *path, int64_t n, const double *points3n, int32_t nfields,
                    const char *const *names, const int32_t *ncomps, const double *const *data);

/* Per-kernel device timings accumulated since the last reset (CUDA events on the
 * context's stream).  names: newline-separated, ms/calls: one entry per name. */
int sphmw_timing_enable(sphmw_ctx *ctx, int32_t enable);
int sphmw_timing_reset(sphmw_ctx *ctx);
/* time only the kernels whose name starts with prefix (NULL or "": all) */
int sphmw_timing_filter(sphmw_ctx *ctx, const char *prefix);
int64_t sphmw_timing_report(sphmw_ctx *ctx, char *names, int64_t cap, double *ms,
                            int64_t *calls, int32_t max_entries);
/* number of kernels this library launched on ctx since creation */
int sphmw_launch_count(sphmw_ctx *ctx, int64_t *n);

/* ---- x-slab decomposition over the GPUs of one box (SURVEY.md §8e) ------------------
 * No reference equivalent: the reference is single-process (Threads.@threads,
 * src/core.jl:54-139).  A context created with slab_lo/slab_hi owns the global cell
 * columns [slab_lo, slab_hi) and keeps two ghost columns per side (three with
 * SPHMW_FLAG_GHOST3: the Hopkins schemes); it carries GLOBAL particle indices so that
 * neighbour order, and with it every FP64 sum, is the same for any number of ranks.
 * Per step the host calls
 *     sphmw_step_phase(ctx, "wcsph", 0)        accelerate! + move!
 *     sphmw_halo_pack -> transport -> sphmw_halo_unpack
 *     sphmw_step_phase(ctx, "wcsph", 1)        cell list, density pass, force pass + kick
 * (phases 2 and 3: the overlapped variant below).  The same two phases step "hopkins",
 * "hopkins_full" and "hopkins_total" (three ghost columns) and "aflow" (the adiabatic flow
 * driver; phase 0 fails when an owned INFLOW particle would convert, because the successors'
 * global indices need the library transport with the open box, below).  Host-driven steps do
 * not renumber: a particle that leaves the global box is dropped and counted (counts[4]), which
 * matches the reference's swap-from-end removal only while no particle leaves — the open box of
 * the library transport replays it.
 * A record is sphmw_halo_record_width(ctx) doubles: the base record of
 * sphmw_halo_record_doubles() (13), or 17 for a context that holds the entropy S (the
 * adiabatic flow driver: + S, P, T, theta).  The width is fixed at its first use (this query or
 * the first pack/unpack/exchange; not sphmw_comm_init), so ask after the fields are uploaded: the
 * answer is binding because buffers are sized by it.  Buffers are
 * DEVICE pointers owned by the caller (NULL = no neighbour on that side). */
int sphmw_step_phase(sphmw_ctx *ctx, const char *scheme, int32_t phase);
int sphmw_halo_record_doubles(void);
int sphmw_halo_record_width(sphmw_ctx *ctx, int32_t *doubles);
/* counts: [0] records for the left neighbour, [1] for the right, [2],[3] migrants among
 * them, [4] particles that left the global box (dropped).  Blocks. */
int sphmw_halo_pack(sphmw_ctx *ctx, double *dev_buf_left, double *dev_buf_right,
                    int64_t cap_records, int64_t counts[5]);
int sphmw_halo_unpack(sphmw_ctx *ctx, const double *dev_buf, int64_t count, int64_t n_migrants);
/* Overlapped variant for all but the last step of a run of steps: the records of the NEXT
 * exchange travel while the interior columns are still in the force pass.
 *     sphmw_step_phase(ctx, "wcsph", 2)   cell list, density pass; force pass + kick and the next
 *                                         step's accelerate! + move! for the edge columns
 *     sphmw_halo_pack_begin               pack the edge columns (enqueue only)
 *     sphmw_step_phase(ctx, "wcsph", 3)   the same for the interior columns (enqueue only)
 *     sphmw_halo_pack_finish              wait for the counts -> transport -> sphmw_halo_unpack
 * leaves the state of "phase 1; phase 0; pack" bit for bit.  Requires |v| dt < h (a particle
 * crosses at most one cell column per step); violations make pack_finish fail.
 * sphmw_halo_pack_wait lets the transport's CUDA stream wait for the packed records. */
int sphmw_halo_pack_begin(sphmw_ctx *ctx, double *dev_buf_left, double *dev_buf_right,
                          int64_t cap_records);
int sphmw_halo_pack_finish(sphmw_ctx *ctx, int64_t cap_records, int64_t counts[5]);
int sphmw_halo_pack_wait(sphmw_ctx *ctx, void *cuda_stream);
int sphmw_slab_counts(sphmw_ctx *ctx, int64_t *n_resident, int64_t *n_owned);

/* Halo transport INSIDE the library (csrc/slab_comm.cu) — what makes a slab context a drop-in for
 * the reference's single-threaded caller (its parallelism is internal to apply_binary!,
 * src/core.jl:125-142): after sphmw_comm_init, sphmw_create_cell_list and sphmw_step(ctx, "wcsph", n)
 * work on a slab context exactly as on a whole-domain one; the records travel by ncclSend/ncclRecv
 * between x-adjacent ranks on a second CUDA stream, beside the interior force pass, one NCCL group
 * per step with the record count in the first row (read on the device), one host wait per step.
 *   sphmw_comm_unique_id   128 bytes (an ncclUniqueId) made by ONE rank and handed to all others by
 *                          whatever means the host has (MPI, a file, torch.distributed ...)
 *   sphmw_comm_init        collective; rank r holds the r-th slab from the left; halo_capacity =
 *                          records one message buffer holds, the same value on every rank
 *   sphmw_comm_info        out = {world, exchanges, renegotiated message sizes, rows per step
 *                          (both directions), particles lost through the global box, capacity}
 * NCCL is loaded with dlopen("libnccl.so.2") at the first of these calls. */
int sphmw_comm_unique_id(void *id128);
int sphmw_comm_init(sphmw_ctx *ctx, int32_t rank, int32_t world, const void *id128, int64_t halo_capacity);
int sphmw_comm_info(sphmw_ctx *ctx, int64_t out[6]);
/* Open box (collective, after sphmw_comm_init): particles may leave the GLOBAL bounding box.
 * create_cell_list! removes them by moving the particles at the end of sys.particles into the
 * vacated slots (src/core.jl:72-81), which renumbers survivors that may live on any rank; since
 * neighbours are visited in index order the renumbering decides the bits of later sums.  With the
 * open box every halo exchange gathers the indices all ranks dropped (one small all-gather) and
 * replays that loop on each rank, and sphmw_step uses the plain (non-overlapped) schedule.  Without
 * it (the default: walled configurations) a particle leaving the global box of a slab context is
 * dropped and counted (sphmw_comm_info out[4]), and an interior one fails the step loudly.
 * The open box also enables sphmw_step(ctx, "flow" | "aflow", n) on slabs: the inflow re-seeding of
 * isothermal_flow_witch.jl:175-186 / adiabatic_flow_witch.jl:197-208 numbers the new particles in the
 * reference's order across ranks (one all-gather of the converting indices per step).  On such a
 * context sphmw_flow_add_new_particles / sphmw_aflow_add_new_particles are collective and return the
 * number added on all ranks, so the driver's operator-by-operator loop (sphmw_apply,
 * add_new_particles, sphmw_create_cell_list) runs unchanged.  sphmw_step(ctx, "hopkins_total", n) needs
 * three ghost columns (SPHMW_FLAG_GHOST3) and runs without the open box too: its walls move and fall
 * (SURVEY quirk 10), and one that leaves the global box is then dropped and counted. */
int sphmw_comm_open_box(sphmw_ctx *ctx, int32_t on);
/* global particle index of every resident particle (physical order) */
int sphmw_set_index(sphmw_ctx *ctx, const int64_t *global_idx, int64_t n);
/* physical-order read-back: indices + tags (0 owned, 1 ghost), and raw fields */
int sphmw_download_index(sphmw_ctx *ctx, int64_t *global_idx, int32_t *tag, int64_t n);
int sphmw_download_raw(sphmw_ctx *ctx, const char *field, double *buf, int64_t n, int32_t ncomp);

#ifdef __cplusplus
}
#endif
#endif /* SPHMW_H */
