/* wafer_b200.h — C ABI of the B200-native replacement for Wafer's imaginary-time FDTD hot path.
 *
 * The reference (Libbum/Wafer, Rust) has no FFI / plugin interface: its hot path is six private
 * functions in src/grid.rs called from `solve` (grid.rs:127,130,134,139,216) and from `evolve`
 * itself (grid.rs:677-680).  This header is the narrowest cut that replaces exactly those calls;
 * every entry point cites the reference function it stands in for.  The cgo-style binding a
 * maintainer would add on the Rust side (extern "C" block + build.rs) is in INTEGRATION.md.
 *
 * Conventions
 *  - Plain C: pointers and sizes only.  No exceptions cross the boundary; every call returns
 *    WAFER_OK (0) or a wafer_status (>0); wafer_last_error(ctx) gives a message owned by ctx.
 *  - Host arrays are the reference's `Array3<R64>` memory: C order, logical axes (x,y,z), z contiguous,
 *    PADDED shape (nx+2e, ny+2e, nz+2e) with e = ext (config.rs:222-239) unless stated "work" (nx,ny,nz).
 *    `Array3<R64>::as_ptr() as *const f64` is exactly this.
 *  - The caller owns every host buffer and may free it when the call returns; the library copies.
 *  - One wafer_ctx is used from one host thread at a time (the reference's `solve` loop is sequential).
 *  - One process per GPU.  With world > 1 the lattice is slab-decomposed along x (the slowest memory
 *    axis — the north-star's "z-slab"): rank r owns work planes [x0, x1).  Array arguments are still the
 *    GLOBAL padded arrays unless the function name ends in _slab; each rank reads / writes only its planes.
 *  - There is NO CPU fallback: wafer_create fails with WAFER_ERR_NO_DEVICE when no sm_100 GPU is present.
 */
#ifndef WAFER_B200_H
#define WAFER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wafer_ctx wafer_ctx;

typedef enum {
    WAFER_OK = 0,
    WAFER_ERR_INVALID = 1,      /* bad argument (ext not in 1..3, zero size, NULL pointer, wnum > stored states) */
    WAFER_ERR_NO_DEVICE = 2,    /* no CUDA device / not sm_100 / device ordinal out of range                   */
    WAFER_ERR_CUDA = 3,         /* a CUDA runtime call failed; see wafer_last_error                            */
    WAFER_ERR_NCCL = 4,         /* NCCL could not be loaded or a collective failed                             */
    WAFER_ERR_RING_NONZERO = 5, /* wafer_set_phi / wafer_push_lower: padding ring not 0 (config.rs:597-622)      */
    WAFER_ERR_NOT_READY = 6,    /* potential or phi not set yet                                                */
    WAFER_ERR_MAX_STEP = 7,     /* wafer_solve: not converged within max_steps (errors.rs MaxStep, grid.rs:244) */
    WAFER_ERR_NONFINITE = 8,    /* NaN/Inf met where the reference's R64 would panic (noisy_float)             */
    WAFER_ERR_IO = 9,           /* a file could not be created, written, opened or read; see wafer_last_error */
    WAFER_ERR_FORMAT = 10       /* the file is not in a layout the device decoder reads; nothing changed       */
} wafer_status;

/* flags */
#define WAFER_FLAG_AB_ARRAYS 0x1u   /* keep A and B as arrays (32 B/update) instead of recomputing them from V in the sweep */
#define WAFER_FLAG_TMA_ONE_STEP 0x8u /* one-step sweeps (5/7-point, excited states, odd tail) through the TMA-pipelined kernel;
                                        already the default unless WAFER_FLAG_SIMPLE_SWEEP or WAFER_FLAG_AB_ARRAYS is set */
#define WAFER_FLAG_NO_FUSED_CHECK 0x10u /* do not fold the check's point-wise sums into the last sweep of wafer_evolve      */
#define WAFER_FLAG_SIMPLE_SWEEP 0x4u /* force the plain register-queue sweep (no TMA pipeline, one step per pass)          */

typedef struct {
    uint64_t nx, ny, nz;   /* WORK sizes = config.grid.size.{x,y,z}            (config.rs:16-23)           */
    uint32_t ext;          /* 1|2|3 = central_difference.ext()                 (config.rs:232-238)         */
    double dn, dt, mass;   /* grid.dn, grid.dt, mass                           (config.rs:20-22,319)       */
    int32_t device;        /* CUDA device ordinal used by this process; -1 = LOCAL_RANK env or 0           */
    uint32_t rank, world;  /* slab decomposition; world = 0 or 1 means single GPU                          */
    const uint8_t *nccl_id;/* 128-byte ncclUniqueId made by wafer_nccl_unique_id on rank 0; NULL if world<=1 */
    uint32_t max_lower;    /* wavemax (config.rs:312); advisory — lower states are allocated as they are pushed */
    uint32_t flags;
} wafer_params;

/* = struct Observables, raw f64 sums on the UN-normalised work area (grid.rs:15-28) */
typedef struct { double energy, norm2, v_infinity, r2; } wafer_observables;

/* one row of the per-check table (output.rs:497-521) as recorded by wafer_solve */
typedef struct {
    uint64_t step;
    double tau, diff;
    wafer_observables obs;
} wafer_record;

/* -------- lifetime ---------------------------------------------------------------------------- */
int wafer_create(const wafer_params *params, wafer_ctx **out);
int wafer_destroy(wafer_ctx *ctx);
const char *wafer_last_error(const wafer_ctx *ctx);     /* ctx may be NULL: message of the last failed wafer_create */
int wafer_nccl_unique_id(uint8_t out[128]);             /* rank 0 calls this and ships the bytes to the other ranks  */
int wafer_slab(const wafer_ctx *ctx, uint64_t *x0, uint64_t *x1); /* this rank's work planes [x0,x1)               */
/* The decomposition rule itself (pure host arithmetic, no GPU needed): contiguous x-slabs, the first nx % world
   ranks own one plane more.  wafer_create uses exactly this. */
int wafer_slab_partition(uint64_t nx, uint32_t world, uint32_t rank, uint64_t *x0, uint64_t *x1);

/* Work distribution of the time-tiled sweep for a ny x nz plane over local x planes [xb, xe) on `slots` resident CTAs
   (pure host arithmetic, no GPU needed — the rule wafer_evolve uses, exposed for the CPU tests): segments are rows of
   5 ints {owner, y0, z0, xa, xz}; owner -1 = handed out in order through the kernel's atomic counter, owner k = static
   tail of CTA k.  *n receives the number of segments (also when it exceeds cap). */
int wafer_tb2_plan(uint32_t ny, uint32_t nz, int32_t xb, int32_t xe, uint32_t slots, int32_t *segments, uint64_t cap,
                   uint64_t *n);

/* -------- state in / out ------------------------------------------------------------------------ */
/* Potentials{v,a,b} (potential.rs:14-25): uploads V and builds b = 1/(1+dt*v/2), a = (1-dt*v/2)*b
   (potential.rs:101-110) on the device. */
int wafer_set_potential(wafer_ctx *ctx, const double *v_padded);
int wafer_get_potential(wafer_ctx *ctx, double *v_padded); /* work area only is meaningful; ring written as 0 */
int wafer_set_pot_sub_scalar(wafer_ctx *ctx, double c);           /* (None,Some(c)); c <= 0 => none (potential.rs:148-152) */
int wafer_set_pot_sub_array(wafer_ctx *ctx, const double *work);  /* (Some(arr),None): WORK sized (potential.rs:135-144)    */
int wafer_set_phi(wafer_ctx *ctx, const double *phi_padded);      /* ring must be 0 (config.rs:597-622)                     */
int wafer_get_phi(wafer_ctx *ctx, double *phi_padded);
/* Slab variants for multi-rank hosts that never hold the global array.  The chunk is a contiguous run of padded
   x-planes [p0,p1) of the global array (each (ny+2e)*(nz+2e) doubles): wafer_slab_planes(ctx, 0, ..) gives the
   run wafer_set_phi_slab reads (owned planes + ghost planes), which=1 the run wafer_get_phi_slab writes (owned
   planes, plus the outer ring planes on the first / last rank). */
int wafer_slab_planes(const wafer_ctx *ctx, int32_t which, uint64_t *p0, uint64_t *p1);
int wafer_set_phi_slab(wafer_ctx *ctx, const double *chunk);
int wafer_get_phi_slab(wafer_ctx *ctx, double *chunk);
/* The inverse of wafer_get_phi_slab: `chunk` is the which=1 run (owned planes, plus the outer ring planes on the first /
   last rank).  The ghost planes are then fetched from the x-neighbours, so this is a COLLECTIVE call when world > 1
   (every rank calls it, like the check at grid.rs:127).  get_phi_slab -> set_phi_owned round-trips the state. */
int wafer_set_phi_owned(wafer_ctx *ctx, const double *chunk);
int wafer_push_lower(wafer_ctx *ctx, const double *q_padded);     /* input::load_wavefunctions (input.rs:487-505)            */
int wafer_push_lower_from_phi(wafer_ctx *ctx);                    /* w_store.push(phi)          (grid.rs:241)                */
int wafer_get_lower(wafer_ctx *ctx, uint32_t idx, double *q_padded);
int wafer_phi_from_lower(wafer_ctx *ctx, uint32_t idx);           /* phi = w_store[idx].clone() (grid.rs:95)                 */
/* Deterministic stand-in for the clone: phi = w_store[idx] * f(x,y,z), f a fixed polynomial without symmetry.
   The reference's clone start only works through rounding noise (SURVEY F7); see generators.cuh seed_poly. */
int wafer_phi_seed_from_lower(wafer_ctx *ctx, uint32_t idx);
int wafer_clear_lowers(wafer_ctx *ctx);
uint32_t wafer_num_lowers(const wafer_ctx *ctx);

/* device-side generators (potential.rs:188-319 at padded indices; config.rs:586-622) — no host array needed.
   kind: index into PotentialType (config.rs:74-104), 100 = gen_potential.py's Poschl-Teller formula. */
int wafer_generate_potential(wafer_ctx *ctx, int32_t kind, double sig);
/* kind: InitialCondition index (config.rs:153-170): 2 Coulomb, 3 Constant, 4 Boolean */
int wafer_generate_initial_condition(wafer_ctx *ctx, int32_t kind);
/* Gaussian initial condition (config.rs:636-642) as a seeded counter-based field: every work site is N(0, sig) from
   Philox4x32-10 keyed by `seed` at the site's global index (generators.cuh gaussian_site), so the same seed gives the
   same bits at any world size.  sig must be finite and >= 0. */
int wafer_generate_gaussian(wafer_ctx *ctx, double sig, uint64_t seed);
/* symmetrise_wavefunction (config.rs:691-728) on the work area, for every ext: kind = SymmetryConstraint index
   (config.rs:186-197) 0 NotConstrained (a no-op, no launch), 1 AboutZ, 2 AntisymAboutZ, 3 AboutY, 4 AntisymAboutY.
   With n the work size of the mirrored axis, psi[.., n-1-t] = +-psi[.., t] for t < n/2; the middle index of an odd n
   is kept (symmetric) or set to +0 (antisymmetric).  Exact and idempotent; needs no communication when world > 1. */
int wafer_symmetrise(wafer_ctx *ctx, int32_t kind);
/* fill_data (input.rs:149-176) / read_csv (input.rs:641-657) on the device: `src` is the array of an input file as
   read, dense C order (sx, sy, sz), z contiguous, WORK-area data.  from_csv = 0 (Messagepack / Json): trilinear
   resample (input.rs:667-716) on a basis of padded-size many points per axis, of which the work area takes the
   first n; a source of the padded size is refused.  from_csv = 1: a work-sized source is copied, any other size
   resampled as above.  Resampling needs sx, sy, sz >= 2.  Only the source x-planes this rank's planes need are
   read, so with world > 1 every rank may pass the whole array; no communication.  Two of its x-planes must fit
   128 MB (sy*sz*8 <= 64 MB).  Each has the effects of the entry it mirrors (set_phi, set_potential, push_lower);
   bad arguments are refused with WAFER_ERR_INVALID before anything changes. */
int wafer_set_phi_resampled(wafer_ctx *ctx, const double *src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv);
int wafer_set_potential_resampled(wafer_ctx *ctx, const double *src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv);
int wafer_push_lower_resampled(wafer_ctx *ctx, const double *src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv);

/* -------- array files ------------------------------------------------------------------------------ */
typedef struct {
    uint64_t bytes;          /* bytes this rank wrote (its sites, plus the preamble on rank 0 and Json's "]}" on the last) */
    uint64_t file_bytes;     /* size of the whole file                                                                 */
    uint64_t host_formatted; /* this rank's sites whose %.17g text was made by snprintf on the host (exact ties)        */
} wafer_write_stats;
/* output::wavefunction / output::potential (output.rs:79-216): the WORK area of psi (what = 0) or V (what = 1) to `path`
   (extension included) as file_type 0 Messagepack, 1 Csv, 2 Json, byte for byte formats.hpp's write_mpk / write_csv /
   write_json (numbers as "%.17g").  The file is encoded on the device, chunk by chunk through the bounce buffers, and
   written with pwrite while the next chunk is encoded; no field-sized buffer is allocated on either side.  Ordered after
   the work already queued on the context; psi, V and the fused check sums are left as they are.
   COLLECTIVE when world > 1: every rank passes the same path and writes its planes at their offset of the one file
   (the file system must be shared by the ranks, e.g. one host).  If any rank cannot create the file, no rank writes and
   all return WAFER_ERR_IO; a failed write on one rank makes every rank return WAFER_ERR_IO.
   WAFER_ERR_INVALID, nothing created: unknown what or file_type (Yaml / Ron), NULL path, Messagepack of more than
   2^32-1 sites (its array32 header cannot count them).  WAFER_ERR_NOT_READY without psi / V.  stats may be NULL. */
int wafer_write_array(wafer_ctx *ctx, int32_t what, int32_t file_type, const char *path, wafer_write_stats *stats);

typedef struct {
    uint64_t sx, sy, sz;       /* dims of the file's array                                                           */
    uint64_t bytes_read;       /* bytes this rank read: the whole file                                               */
    uint64_t sites_converted;  /* sites of the source x-planes this rank's planes need, all converted                  */
    uint64_t host_converted;   /* of those, numbers strtod converted on the host (the device could not certify them) */
} wafer_load_stats;
/* input::load_wavefunctions / fill_data / read_csv (input.rs:113-176, 487-505, 607-662) for a file `path` of file_type
   0 Messagepack, 1 Csv, 2 Json, decoded on the device: what = 0 sets psi (= wafer_set_phi_resampled of the array that
   formats.hpp's read_mpk / read_csv / read_json return), 1 sets V (= wafer_set_potential_resampled), 2 pushes a lower
   state (= wafer_push_lower_resampled), bit for bit.  Only the canonical layouts are read: what formats.hpp's writers
   (and rmp-serde / serde_json) produce, numbers in the JSON grammar (DESIGN.md section 1.4).  The file is streamed through
   the bounce buffers with pread and checked whole before anything changes; numbers the device cannot certify are
   converted with strtod on the host.  Every rank reads the whole file and keeps the source x-planes its planes need,
   in one device buffer; no communication when world > 1.
   WAFER_ERR_IO: the file cannot be opened or read.  WAFER_ERR_FORMAT, nothing changed: the file is not canonical, or
   the rank's source planes cannot be allocated on the device (formats.hpp's readers and wafer_*_resampled still
   take such a file).  WAFER_ERR_INVALID: unknown what or file_type (Yaml / Ron), NULL path, a shape the resampling
   entries refuse.  stats may be NULL. */
int wafer_load_array(wafer_ctx *ctx, int32_t what, int32_t file_type, const char *path, wafer_load_stats *stats);

/* -------- the hot path -------------------------------------------------------------------------- */
int wafer_observables_compute(wafer_ctx *ctx, wafer_observables *out); /* compute_observables        (grid.rs:303-445) */
int wafer_norm2(wafer_ctx *ctx, double *out);                          /* get_norm_squared(work area) (grid.rs:454-457) */
int wafer_normalise(wafer_ctx *ctx, double norm2);                     /* normalise_wavefunction      (grid.rs:465-468) */
int wafer_orthogonalise(wafer_ctx *ctx, uint8_t wnum);                 /* orthogonalise_wavefunction  (grid.rs:477-492) */
int wafer_evolve(wafer_ctx *ctx, uint8_t wnum, uint64_t steps);        /* evolve; steps = screen_update (grid.rs:544-687) */
/* fused grid.rs:127-135: observables -> normalise(norm2) -> orthogonalise(wnum) without leaving the device */
int wafer_check(wafer_ctx *ctx, uint8_t wnum, wafer_observables *out);

/* -------- the immediate caller (grid.rs:50-246), re-stated on top of the calls above -------------- */
/* phi must be set.  max_steps < 0 = None; snap_update = 0 = None.  Returns WAFER_OK when converged (the state
   is then pushed to the lower-state store like grid.rs:241) or WAFER_ERR_MAX_STEP. */
int wafer_solve(wafer_ctx *ctx, uint8_t wnum, double tolerance, int64_t max_steps, uint64_t screen_update,
                uint64_t snap_update, wafer_record *records, uint64_t max_records, uint64_t *n_records);

/* -------- plumbing ------------------------------------------------------------------------------- */
int wafer_synchronize(wafer_ctx *ctx);
int wafer_timer_begin(wafer_ctx *ctx);                 /* CUDA event on the library's compute stream */
int wafer_timer_end(wafer_ctx *ctx, double *ms);       /* records, synchronises, returns elapsed ms  */
uint64_t wafer_kernel_launches(const wafer_ctx *ctx);  /* kernels launched by this ctx so far        */
int wafer_host_alloc(void **ptr, size_t bytes);        /* pinned host memory for fast host<->device copies */
int wafer_host_free(void *ptr);
/* Page-lock a buffer the CALLER owns (e.g. the memory behind an Array3<R64>) so that wafer_set_phi / wafer_get_phi and
   their slab variants copy at PCIe speed instead of through the driver's pageable path (measured 1024^3 on one B200:
   54 GB/s pinned vs 14 GB/s pageable).  Unregister before the buffer is freed. */
int wafer_host_register(void *ptr, size_t bytes);
int wafer_host_unregister(void *ptr);
int wafer_device_info(const wafer_ctx *ctx, char *name, size_t name_len, int32_t *sm_count, int32_t *cc_major,
                      int32_t *cc_minor, uint64_t *mem_bytes);
/* Fused halo exchange over NVLink peer memory (optional, world > 1).  Every rank exports 192 bytes (CUDA IPC handles of
   its two psi buffers and its flag words), the host ships rank r-1's and rank r+1's blobs to rank r (NULL at the ends of
   the chain) and calls connect.  From then on the ground-state sweep of wafer_evolve stores its first and last two output
   planes directly into the neighbours' ghost planes as it produces them, and ranks order themselves with pass counters
   in peer memory (one handshake per pass); without it the same planes travel by ncclSend/ncclRecv. */
int wafer_p2p_export(wafer_ctx *ctx, uint8_t out[192]);
int wafer_p2p_connect(wafer_ctx *ctx, const uint8_t *lower, const uint8_t *upper);
/* self-test of the sweep's division by the loop-invariant denominator: compares it bit-for-bit with IEEE
   division on n pseudo-random operands (every exponent, zeros, denormals, NaN/Inf); *mismatches must be 0 */
int wafer_selftest_division(wafer_ctx *ctx, double den, uint64_t n, uint64_t seed, uint64_t *mismatches);
/* Position-sensitive, slab-independent checksum of the work-area sites of GLOBAL work planes [x_begin, x_end) that this
   rank owns: out[0] = wrapping sum, out[1] = xor of mix64(bits(psi) + c * (global site index + 1)).  Add the out[0]s and
   xor the out[1]s of all ranks to get the checksum of the union; equal checksums <=> bit-identical wavefunctions (up to
   2^-64 collisions).  This is how multi-GPU runs are compared bit-for-bit with a single-GPU run at full size. */
int wafer_phi_checksum(wafer_ctx *ctx, uint64_t x_begin, uint64_t x_end, uint64_t out[2]);
/* Fault injection for the multi-GPU ordering tests: stall this rank by `nanoseconds` (<= 1e9) before the halo handshake
   of every pass of wafer_evolve (on the main stream before a two-step pass with fused halos, on the halo stream before
   the boundary launches of every other multi-GPU pass), so that its x-neighbours run ahead of it.  0: no stall. */
int wafer_debug_halo_delay(wafer_ctx *ctx, uint64_t nanoseconds);
const char *wafer_version(void);
const char *wafer_sweep_variant(const wafer_ctx *ctx); /* name of the sweep kernel variant in use */

#ifdef __cplusplus
}
#endif
#endif /* WAFER_B200_H */
