/* r3d_gpu.h -- C ABI of the B200-native phonon-propagate path of Radiative3D.
 *
 * This is the drop-in boundary for ONE path of the reference program: the body
 * of the per-phonon loop in Model::RunSimulation (reference model.cpp:611-625),
 * i.e. ShearDislocation::GenerateEventPhonon (events.cpp:111-124) followed by
 * Phonon::Propagate (phonons.cpp:540-682) with everything it reaches
 * (media.cpp, media_cellface.cpp, raypath.cpp, rtcoef.cpp, scatterers.cpp:297-363,
 * probability.cpp:104-129, dataout.cpp:103-216,545-617).
 *
 * The reference has no FFI for this path (the loop is hard-wired and talks to
 * global singletons), so the boundary is defined here: the host program builds
 * its model exactly as before, FLATTENS it into the plain arrays of
 * r3d_model_desc, and calls r3d_create / r3d_run / r3d_fetch in place of the
 * loop; r3d_fetch returns the seismometer bins and loss counters which the host
 * writes back into its Seismometer / DataReporter objects before calling its
 * unchanged file writers (dataout.cpp:249-406,623-694).  INTEGRATION.md shows
 * the reference-side stub.
 *
 * Conventions: plain pointers and sizes, no C++ types, no exceptions cross the
 * ABI.  Every function returning int returns 0 on success and a non-zero
 * R3D_E* code otherwise; r3d_last_error() then holds a message (thread-local).
 * All descriptor arrays are BORROWED for the duration of r3d_create only.
 * The five large tables of a descriptor (toa_theta, toa_phi, src_cdf, scat_cdf,
 * scat_spol) may live in host memory (pinned memory makes the upload direct)
 * or in DEVICE memory of any CUDA device of the process - e.g. a buffer that a
 * multi-process launcher received by an NCCL broadcast over NVLink, so that
 * the tables cross PCIe once per node and not once per GPU; all other arrays
 * are read by the host and must be host memory.
 * There is no CPU fallback: with no usable CUDA device r3d_create fails.
 */
#ifndef R3D_GPU_H_
#define R3D_GPU_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R3D_ABI_VERSION 2

/* error codes */
#define R3D_OK            0
#define R3D_EINVAL        1   /* bad descriptor / argument               */
#define R3D_ECUDA         2   /* CUDA runtime error (message has detail) */
#define R3D_ENODEV        3   /* no usable CUDA device                   */
#define R3D_ENOMEM        4
#define R3D_EUNSUPPORTED  5

/* ray types (reference raytype.hpp:12-20) */
#define R3D_RAY_P   0
#define R3D_RAY_S   1
#define R3D_RAY_SH  1
#define R3D_RAY_SV  2

/* cell kinds: one kind per model, as in the reference (model.cpp:378-411) */
#define R3D_CELL_CYLINDER 0   /* RCUCylinder, media.hpp:309  */
#define R3D_CELL_TETRA    1   /* Tetra,       media.hpp:397  */
#define R3D_CELL_SHELL    2   /* SphereShell, media.hpp:462  */

/* face flag bits (CellFace::mCollect/mReflect/mAdjoin/mGridDiscon,
 * media_cellface.hpp:120-126) */
#define R3D_FACE_COLLECT 1u
#define R3D_FACE_REFLECT 2u
#define R3D_FACE_ADJOIN  4u
#define R3D_FACE_DISCON  8u

/* faces per cell and face ids (media_cellface.hpp:96-107) */
#define R3D_CYL_NFACES    3   /* TOP=0, BOTTOM=1, SIDE=2 (shared loss face) */
#define R3D_SHELL_NFACES  2   /* TOP=0, BOTTOM=1 */
#define R3D_TETRA_NFACES  4   /* A..D = 0..3 */

/* per-cell parameter records, in doubles.
 *
 * CYLINDER (media.cpp:135-158): only the TOP velocities/Q/density are used.
 *   [0..1] vel P,S   [2] density   [3..4] Q P,S
 *   [5..7] top normal  [8..10] top point  [11..13] bottom normal  [14..16] bottom point
 * SHELL (media.cpp:578-626):  v(r) = C + A r^2
 *   [0..1] A P,S  [2..3] C P,S  [4..5] zeroRadius^2 P,S  [6] densA  [7] densC
 *   [8..9] Q P,S  [10] signed radius top (+R)  [11] signed radius bottom (-R, -0.0 at centre)
 *   [12] Rtop^2  [13] Rbot^2
 * TETRA (media.cpp:353-395):  v(x) = g.x + v0
 *   [0..2] grad P  [3..5] grad S  [6..7] v0 P,S  [8..10] density grad  [11] density0
 *   [12..13] Q P,S  [14+6f .. 14+6f+2] face f normal  [14+6f+3 .. +5] face f point
 */
#define R3D_CYL_NPARAM   17
#define R3D_SHELL_NPARAM 14
#define R3D_TETRA_NPARAM 38

/* seismometer record, in doubles (dataout.cpp:42-71):
 *   [0..2] loc  [3..5] X1  [6..8] X2  [9..11] X3
 *   [12..13] inner radius P,S  [14..15] outer radius P,S  [16..17] area P,S */
#define R3D_SEIS_NPARAM 18

/* bin record layout returned by r3d_fetch (dataout.hpp:77-93):
 *   energies[s][b][0..2] = X1,X2,X3 axis energy, [3..4] = energy by type P,S
 *   counts  [s][b][0..1] = phonon count by type P,S (u64 here; u32 in reference) */
#define R3D_BIN_NF64 5
#define R3D_BIN_NCNT 2

/* counters returned by r3d_fetch (dataout.cpp:591-617) */
#define R3D_CNT_LOST     0
#define R3D_CNT_TIMEOUT  1
#define R3D_CNT_INVALID  2
#define R3D_CNT_EVENTS   3   /* propagate-loop iterations (phonons.cpp:542), extension */
#define R3D_CNT_CATCHES  4   /* bin updates (dataout.cpp:200-212), extension            */
#define R3D_CNT_SCATTERS 5   /* scatter events (phonons.cpp:605-618), extension         */
#define R3D_CNT_PHONONS  6   /* phonons generated (model.cpp:611-614), extension        */
#define R3D_CNT_DIAG     7   /* DataReporter::mDiagInvalid: OR of (1 << R3D_INV_*); combined by OR, not by sum */
#define R3D_NCOUNTERS    8
#define R3D_NDIAG_LANES  8   /* 0/1 lanes of the diagnostic word's bits, kept after the counters on the device (see
                              * r3d_device_accumulator_blocks) */

/* invalid-phonon reasons, bit index into diag (dataout.hpp:229-237) */
#define R3D_INV_PATH_NAN      0
#define R3D_INV_TIME_NAN      1
#define R3D_INV_PATH_NEGATIVE 2
#define R3D_INV_TIME_NEGATIVE 3
#define R3D_INV_STUCK         4
#define R3D_INV_SLOW          5
#define R3D_INV_LOOP_EXCEED   6

/* fates in r3d_phonon_final */
#define R3D_FATE_LOST    1
#define R3D_FATE_TIMEOUT 2
#define R3D_FATE_INVALID 3

typedef struct r3d_model_desc {
  /* ---- globals (class statics set by the Model ctor, model.cpp:271-299) ---- */
  double   freq_hz;        /* MediumCell::cmPhononFreq                           */
  double   ttl;            /* Phonon::cm_ttl                                     */
  double   bin_dt;         /* Seismometer::cmTimePerBin                          */
  uint32_t n_bins;         /* Seismometer::cmNumBins                             */
  int32_t  ecs_radial;     /* 0: up=(0,0,1) (ENU/RAE ortho); 1: up radial from   */
  double   earth_center[3];/*    earth_center (RAE curved/spherical, ecs.cpp:147)*/
  double   min_theta;      /* Phonon::cm_min_theta (1e-7)                        */
  double   max_theta;      /* Phonon::cm_max_theta (pi-1e-7)                     */
  double   slow_concern;   /* Phonon::cm_slow_concern (0.001)                    */
  uint64_t loop_concern;   /* Phonon::cm_loop_concern (2^20)                     */
  int32_t  no_deflect;     /* Scatterer::cm_NoDeflect_b                          */
  int32_t  reserved0;
  /* ---- take-off-angle set (PhononSource::pTOA) ---- */
  uint32_t n_toa;
  uint32_t reserved1;
  const double *toa_theta; /* [n_toa] */
  const double *toa_phi;   /* [n_toa] */
  /* ---- event source (ShearDislocation, events.cpp:42-107) ---- */
  double   src_loc[3];
  uint32_t src_cell;
  uint32_t reserved2;
  const double *src_whole_cdf; /* [3]        cumulative, P,SH,SV (mWholeProbs[0]) */
  const double *src_cdf;       /* [3][n_toa] cumulative (mPDists[P|SH|SV])        */
  /* ---- scatterers (scatterers.cpp:97-220) ---- */
  uint32_t n_scat;
  uint32_t reserved3;
  const double *scat_mfp;       /* [n_scat][2]        mean free path P,S            */
  const double *scat_whole_cdf; /* [n_scat][2][4]     cumulative (mWholeProbs[in])  */
  const double *scat_cdf;       /* [n_scat][4][n_toa] cumulative PP,PS,SP,SS        */
  const double *scat_spol;      /* [n_scat][n_toa]    S->S polarisation angle       */
  /* ---- cells ---- */
  uint32_t n_cells;
  uint32_t cell_kind;      /* R3D_CELL_*                                  */
  uint32_t cell_nparam;    /* R3D_*_NPARAM matching cell_kind             */
  uint32_t faces_per_cell; /* R3D_*_NFACES matching cell_kind             */
  const double   *cell_params;     /* [n_cells][cell_nparam]              */
  const uint32_t *cell_scat;       /* [n_cells] scatterer index           */
  const uint8_t  *face_flags;      /* [n_cells][faces_per_cell] R3D_FACE_*; other bits are ignored */
  const uint32_t *face_other_cell; /* [n_cells][faces_per_cell]; ignored  */
                                   /*   unless R3D_FACE_ADJOIN is set     */
  double   cyl_radius2;    /* RCUCylinder::cmLossFace.mRad2 (cylinder only)*/
  /* ---- seismometers (dataout.cpp:42-71) ---- */
  uint32_t n_seis;
  uint32_t reserved4;
  const double *seis;      /* [n_seis][R3D_SEIS_NPARAM] */
} r3d_model_desc;

/* per-phonon end state, for parity tests (r3d_trace) */
typedef struct r3d_phonon_final {
  double   time, pathlen, amp;
  double   loc[3];
  double   theta, phi, pol;
  uint32_t moves;      /* Phonon::mMoveCount                          */
  uint32_t cell;       /* index of the cell the phonon died in        */
  uint32_t type;       /* R3D_RAY_P / R3D_RAY_S                       */
  uint32_t fate;       /* R3D_FATE_* ; for INVALID, reason in bits 8+ */
  uint32_t draws;      /* RNG draws consumed                          */
  uint32_t catches;    /* bin updates made                            */
  uint32_t scatters;   /* scatter events                              */
  uint32_t iters;      /* loop iterations                             */
} r3d_phonon_final;

/* ---- event reports (reference DataReporter::Report*, dataout.cpp:484-617; SURVEY 8a row a23) ----
 * One record per reported event, holding what output_phonon_dataline() prints: the phonon's state at the moment the
 * reference would call the matching Report* method (phonons.cpp:540-682, events.cpp:120). */
#define R3D_EV_GEN 0   /* "GEN: " new event phonon              (ReportNewEventPhonon) */
#define R3D_EV_SCT 1   /* "SCT: " after a scatter's Transform   (ReportScatterEvent)   */
#define R3D_EV_COL 2   /* "COL: " arrival at a collection face  (ReportPhononCollected)*/
#define R3D_EV_REF 3   /* "REF: " reflected at a face           (ReportReflection)     */
#define R3D_EV_CEL 4   /* "CEL: " crossed into another cell     (ReportCellToCell)     */
#define R3D_EV_LST 5   /* "LST: " left the model                (ReportLostPhonon)     */
#define R3D_EV_TMO 6   /* "TMO: " timed out                     (ReportPhononTimeout)  */
#define R3D_EV_INV 7   /* "INV: " failed a validity check       (ReportInvalidPhonon)  */
#define R3D_EV_ALL 0xFFu

typedef struct r3d_event {
  uint64_t phonon;     /* global phonon index                                   */
  uint32_t seq;        /* ordinal of this report within its phonon (0, 1, ...)  */
  uint32_t kind;       /* R3D_EV_*                                              */
  uint32_t type;       /* R3D_RAY_P / R3D_RAY_S                                 */
  uint32_t moves;      /* Phonon::mMoveCount ("it:")                            */
  uint32_t cell;       /* cell index (the reference prints the cell's address)  */
  uint32_t reason;     /* R3D_EV_INV: bit mask (1 << R3D_INV_*) of the check that failed; else 0 */
  double   time, pathlen;
  double   loc[3];     /* model coordinates (the host applies ECS.OutConvert)   */
  double   theta, phi;
  double   amp;
} r3d_event;

typedef struct r3d_handle r3d_handle;

/* Upload a model to `n_dev` CUDA devices (replicated; SURVEY 8e) and allocate
 * zeroed bins.  devices==NULL means device 0..n_dev-1.  With several devices
 * the host arrays are uploaded once, to the first device; the others copy the
 * large tables from its memory (NVLink peer copies). */
int r3d_create(const r3d_model_desc *desc, const int *devices, int n_dev,
               r3d_handle **out);

/* Trace phonons [first_phonon, first_phonon+n_phonons) and ACCUMULATE into the
 * bins / counters.  Phonon i always uses the Philox4x32-10 stream keyed by
 * (seed, i), so the result does not depend on how a range is split across
 * calls, devices or ranks (up to floating-point summation order).  The index
 * range is sharded contiguously across the handle's devices.  Asynchronous:
 * returns after enqueueing; r3d_sync / r3d_fetch wait. */
int r3d_run(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, uint64_t seed);

/* Wait for all enqueued work.  If device_seconds!=NULL it receives the device
 * time (CUDA events, max over devices) of the r3d_run calls since the last
 * r3d_sync. */
int r3d_sync(r3d_handle *h, double *device_seconds);

/* Synchronise, sum over the handle's devices, copy out.  Any pointer may be
 * NULL.  energies: [n_seis][n_bins][5] f64; counts: [n_seis][n_bins][2] u64;
 * counters: [R3D_NCOUNTERS]; diag: OR of (1<<R3D_INV_*).
 * The sum over the devices of a handle (the reference's combine.m:26-33) is
 * made ON THE DEVICE: a kernel on the first device reads the other devices'
 * accumulators through peer access (NVLink) in device order and writes the
 * sums to a staging buffer, which is then copied to the host once.  Devices
 * that are not peers are summed on the host instead. */
int r3d_fetch(r3d_handle *h, double *energies, uint64_t *counts,
              uint64_t *counters, uint32_t *diag);

/* Zero bins and counters on all devices. */
int r3d_reset(r3d_handle *h);

/* Device pointers of device `dev_slot`'s accumulators, so a multi-process
 * launcher can all-reduce them in place (e.g. torch.distributed/NCCL on a
 * tensor wrapping the memory): energies f64[n_seis*n_bins*5], counts
 * u64[n_seis*n_bins*2], counters u64[R3D_NCOUNTERS] (diag is counters[7]).
 * In-place reduction is for the END of a run: every r3d_run recomputes the
 * counters from the device's own tallies, so reduce, r3d_fetch, and call
 * r3d_reset before any further r3d_run on the handle. */
int r3d_device_accumulators(r3d_handle *h, int dev_slot, void **energies,
                            void **counts, void **counters);

/* The same accumulators as TWO blocks, so that a multi-process launcher needs two collectives (one per element type) and no
 * host synchronisation: f64_block = the energies (n_f64 doubles); i64_block (n_i64 u64 words) = counts
 * [n_seis*n_bins*2], then at word *counters_at the counters [R3D_NCOUNTERS], then R3D_NDIAG_LANES lanes holding bit b of
 * the diagnostic word as 0 / 1.  After a SUM all-reduce of i64_block every word is right except counters[R3D_CNT_DIAG]
 * (a sum of bit masks): rebuild it as OR over b of (lane[b] != 0) << b (radiative3d_b200/distributed.py does this on the
 * device).  In-place reduction is for the END of a run: the next r3d_run recomputes the counters from the device's own
 * tallies, so call r3d_fetch (and r3d_reset before any further r3d_run) right after it. */
int r3d_device_accumulator_blocks(r3d_handle *h, int dev_slot, void **f64_block, uint64_t *n_f64, void **i64_block,
                                  uint64_t *n_i64, uint64_t *counters_at);

/* The CUDA stream r3d_run launches on for `dev_slot` (a cudaStream_t). */
int r3d_stream(r3d_handle *h, int dev_slot, void **stream);

/* Number of kernels this handle has launched so far. */
int r3d_launch_count(r3d_handle *h, uint64_t *n);

/* Kernel timing for the roofline report.  Every launch of the propagate kernel is bracketed by CUDA events on
 * the launching stream, and every CTA counts the clock cycles it spends in its two phases.  r3d_set_profiling
 * resets these totals (`on` is ignored).  r3d_kernel_times returns, for device slot 0 since the last reset:
 *   seconds[0]  device seconds of the propagate kernel launches
 *   seconds[1]  the share of seconds[0] spent in phase 1 (advance + refill), averaged over CTAs
 *   seconds[2]  the share spent in phase 2 (table draws + face events)
 *   launches[0] kernel launches, launches[1] iterations of the busiest CTA, launches[2] CTAs per launch
 *   units[0]    propagate-loop events, units[1] table draws (scatter + source), units[2] bin updates
 * units are read from the handle's counters, so call r3d_reset together with r3d_set_profiling. */
int r3d_set_profiling(r3d_handle *h, int on);
int r3d_kernel_times(r3d_handle *h, double seconds[3], uint64_t launches[3], uint64_t units[3]);

/* ---- energy snapshots: phonon energy on a voxel grid at chosen lapse times ----------------------------------------------
 * The energy density E(x, t) of radiative transfer, built in the propagate kernel while each phonon is in registers.
 *
 * Contract.  The caller gives K lapse times 0 <= t_0 < t_1 < ... < t_{K-1} <= ttl (K <= R3D_SNAP_MAX_TIMES) and an
 * axis-aligned grid in model coordinates: origin[3], voxel[3] (> 0), dims[3] (>= 1).
 *   - Every move of a phonon covers the time interval [t_a, t_b): t_a is its time before Phonon::Move, t_b its time after
 *     it - the same FP64 value that is the next move's t_a - so the moves of one phonon tile [0, final time) exactly.
 *   - For every t_k in [t_a, t_b) the phonon makes one record: its position is the point on the move's ray (straight or
 *     arc) at travel time t_k - t_a from the move's start; its weight is amp^2 = exp(-2 aexp(t_k)), the square of the
 *     amplitude a seismometer bins; it goes to ray type P = 0 or S = 1.
 *   - A move makes its records whatever event ends it: scatter, face, hand-over, or loss at a face that does not collect.
 *     A phonon that times out on an infinite path makes no move and no record; NaN times make none (the comparisons fail).
 *     So a phonon contributes to snapshot k exactly when its final time is > t_k.
 *   - The voxel index on each axis is i = floor((x - origin) / voxel), IEEE division.  A record with 0 <= i < dims on all
 *     three axes goes to that voxel; any other record goes to the snapshot's "outside" cell, so every record is counted.
 *   - The point at a travel time: straight rays at constant speed (layered cells; shells without velocity gradient) are
 *     exact, len = dt v.  Curved rays (shell arcs, tetrahedral arcs) take a fixed number of Newton steps on the length
 *     with Cell::advance's own travel-time formula (radiative3d_b200/csrc/r3d_device.cuh: advance_time).
 *   - Accumulators per snapshot, voxel (and outside) and ray type: energy (sum of weights, f64) and record count (u64).
 *     They add up across r3d_run calls, devices and index ranges, like the seismometer bins.
 * r3d_run launches the kernels with the deposits while snapshots are on; r3d_trace and r3d_trace_events make no snapshot
 * records.  Snapshots do not change what a phonon does: bins and counters are those of a run without them. */
#define R3D_SNAP_MAX_TIMES 64
#define R3D_SNAP_MAX_CELLS (1u << 28)   /* cap on n_times * (dims[0] dims[1] dims[2] + 1) * 2 accumulator cells (4 GB per device) */
typedef struct r3d_snapshot_desc {
  uint32_t n_times, reserved;
  const double *times;     /* [n_times], host memory, borrowed for the call */
  double origin[3], voxel[3];
  uint32_t dims[3], reserved2;
} r3d_snapshot_desc;

/* Synchronise, then give every device of the handle zeroed snapshot accumulators (from the library's private pool),
 * replacing any earlier grid.  s == NULL or s->n_times == 0 turns snapshots off.  R3D_EINVAL for times that are not
 * increasing, not finite or outside [0, ttl]; more than R3D_SNAP_MAX_TIMES times; a voxel size that is not finite and
 * positive; a non-finite origin; a zero dimension; or more than R3D_SNAP_MAX_CELLS accumulator cells.  r3d_reset zeroes
 * the snapshot accumulators too. */
int r3d_set_snapshots(r3d_handle *h, const r3d_snapshot_desc *s);

/* Synchronise, sum over the handle's devices, copy out.  Any pointer may be NULL.  energy f64 and count u64:
 * [n_times][dims[2]][dims[1]][dims[0]][2] (x fastest, last index = ray type); outside_energy, outside_count: [n_times][2].
 * R3D_EINVAL while snapshots are off. */
int r3d_fetch_snapshots(r3d_handle *h, double *energy, uint64_t *count, double *outside_energy, uint64_t *outside_count);

/* ---- catch log: which phonons reach chosen seismometers, to be traced again by index ------------------------------------
 * The bins hold sums; the log keeps the identity of each catch, so that exactly the phonons behind a bin can be traced
 * again with full event reports (r3d_trace_events_indices).  Draws are keyed by (seed, global phonon index), so a phonon's
 * index and the run's seed are all a replay needs.
 *
 * Log.  While a log is set, every catch that r3d_run bins into a selected seismometer within the bins [bin_lo, bin_hi)
 * makes one r3d_catch record: all launches of a job, the pilot launches included, with snapshots on or off.  r3d_trace,
 * r3d_trace_events and the _indices calls make no records.
 *   - Among the runs of one seed over disjoint index ranges a record is identified uniquely by (phonon, moves, seis).
 *   - r3d_fetch_catch_log synchronises, concatenates the logs of the handle's devices and returns the kept records sorted
 *     by (phonon, moves, seis).  A log that is not truncated is therefore independent of scheduling, of how the index
 *     range was split across calls, and of the devices.
 *   - *n_matched counts every matching catch.  Each device keeps at most `capacity` records; when *n_matched exceeds the
 *     records kept, the kept records are an arbitrary subset of the matching catches.
 *   - Records accumulate across r3d_run calls.  A record does not carry the seed: replay with the seed of its run.
 *   - r3d_reset empties the log.  r3d_set_catch_log synchronises first and replaces any earlier log (NULL = off).
 *   - R3D_EINVAL: a seismometer index >= n_seis or listed twice; bin_lo >= bin_hi or bin_hi > n_bins; capacity 0 or above
 *     R3D_CATCH_LOG_MAX; r3d_fetch_catch_log while the log is off.
 * The kernels with the log are separate instantiations: with the log off r3d_run runs the same code as without this
 * feature. */
#define R3D_CATCH_LOG_MAX (1ull << 28)   /* records per device (16 GB) */
typedef struct r3d_catch {          /* 64 bytes */
  uint64_t phonon;                  /* global phonon index                                               */
  uint32_t seis, bin;               /* seismometer and time bin the catch was added to                    */
  uint32_t type;                    /* R3D_RAY_P / R3D_RAY_S                                             */
  uint32_t moves;                   /* move count at the arrival = r3d_event.moves of its COL report      */
  double   time;                    /* time alive at the arrival (before CatchPhonon's plane-wave shift)  */
  double   energy[4];               /* X1, X2, X3 and type energy, exactly the addends of the bin         */
} r3d_catch;
typedef struct r3d_catch_log_desc {
  uint32_t n_seis;                  /* entries in seis; 0 = every seismometer       */
  uint32_t bin_lo, bin_hi;          /* catches into bins [bin_lo, bin_hi)           */
  uint32_t reserved;
  const uint32_t *seis;             /* seismometer indices, host memory, borrowed   */
  uint64_t capacity;                /* records kept per device                      */
} r3d_catch_log_desc;
int r3d_set_catch_log(r3d_handle *h, const r3d_catch_log_desc *d);
/* Writes min(capacity, *n_kept) records to out (out may be NULL when capacity is 0: a query of the two counts).
 * *n_kept: records kept over all devices; *n_matched: matching catches over all devices. */
int r3d_fetch_catch_log(r3d_handle *h, r3d_catch *out, uint64_t capacity, uint64_t *n_kept, uint64_t *n_matched);

/* Replay.  r3d_trace / r3d_trace_events for the listed global phonon indices instead of a range, on device slot 0: phonon
 * indices[i] is traced exactly as r3d_trace(h, indices[i], 1, seed, ...) would trace it.  `indices` must be strictly
 * increasing (else R3D_EINVAL); an empty list is a no-op.  out[i] of r3d_trace_indices belongs to indices[i]; events are
 * sorted by (phonon, seq) with r3d_event.phonon the global index.  Bins and counters accumulate as in r3d_trace; no catch
 * log records are made.  Long lists are split into launches like long ranges. */
int r3d_trace_indices(r3d_handle *h, const uint64_t *indices, uint64_t n, uint64_t seed, r3d_phonon_final *out);
int r3d_trace_events_indices(r3d_handle *h, const uint64_t *indices, uint64_t n, uint64_t seed, uint32_t kinds_mask,
                             r3d_event *out, uint64_t capacity, uint64_t *n_events);

/* Parity hook: trace phonons [first, first+n) on device slot 0 WITHOUT touching
 * the accumulators' semantics (bins are still accumulated) and write each
 * phonon's end state to out[n] (host memory). */
int r3d_trace(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons,
              uint64_t seed, r3d_phonon_final *out);

/* Event reports for video runs: trace phonons [first, first+n) on device slot 0 (bins and counters accumulate as in
 * r3d_run) and return the events whose kind is in kinds_mask (bit R3D_EV_*), sorted by (phonon, seq) - the order in which
 * the single-threaded reference writes them.  At most `capacity` records are written to out; *n_events receives the number
 * of events that occurred (if it exceeds capacity, call again with a larger buffer or a shorter range). */
int r3d_trace_events(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, uint64_t seed, uint32_t kinds_mask,
                     r3d_event *out, uint64_t capacity, uint64_t *n_events);

/* ---- scatterer tables (SURVEY 8f-2): what the reference's Scatterer constructor computes -------------------------
 * Scatterer::PopulateProbDists / PopulateWholeProbs / ComputeMFPs (scatterers.cpp:134-220) with
 * ScatterParams::GSATO / XSATO / PSATO (scatparams.cpp:75-194, Sato & Fehler 4.50-4.52, von Karman PSDF): the G values of
 * all take-off angles are evaluated on the device; the cumulative sums are then formed on the host in index order, as
 * ProbDist::Integrate does (probability.cpp:21-35), because their rounding decides table indices.
 * This is the model-build hot spot of the reference (0.3 s per scatterer at TOA degree 9, up to 28 scatterers). */
typedef struct r3d_scatter_params {
  double nu, eps, a, kappa;   /* density/velocity scaling, RMS perturbation, correlation distance, von Karman parameter */
  double el, gam0;            /* S wavenumber omega / beta0, Vp / Vs                                                   */
} r3d_scatter_params;
/* The pieces of r3d_build_scatterer_tables for a host program that keeps the reference's own ProbDist objects (the drop-in
 * program's Scatterer::PopulateProbDists, integration/r3d_scatterer_gpu.cpp): upload the take-off angles once, then get the
 * un-integrated G values g[4][n_toa] (gpp, gps, gsp, gss) and the S->S polarisation angles spol[n_toa] of one parameter
 * set per call; the host integrates them itself (ProbDist::Integrate). */
typedef struct r3d_toa_set r3d_toa_set;
int  r3d_toa_create(const double *toa_theta, const double *toa_phi, uint32_t n_toa, int device, r3d_toa_set **out);
int  r3d_scatterer_g_values(r3d_toa_set *t, const r3d_scatter_params *par, double *g, double *spol);
void r3d_toa_destroy(r3d_toa_set *t);

/* For each of the n_par parameter sets: cdf[p][4][n_toa] (PP,PS,SP,SS, cumulative), spol[p][n_toa], whole_cdf[p][2][4]
 * (cumulative, as r3d_model_desc.scat_whole_cdf), mfp[p][2]; all host arrays, laid out as r3d_model_desc wants them.
 * The take-off angles are uploaded once; uses CUDA device `device`. */
int r3d_build_scatterer_tables(const r3d_scatter_params *par, uint32_t n_par, const double *toa_theta, const double *toa_phi,
                               uint32_t n_toa, int device, double *cdf, double *spol, double *whole_cdf, double *mfp);

/* ---- deterministic sub-kernel hooks (parity at 1e-10, SURVEY 8c) ----------
 * Each evaluates n independent cases on the device with the same device
 * functions the propagate kernel uses. */

/* ProbDist::GetRandomIndex (probability.cpp:104-129) on cdf[n_cdf] for the
 * 31-bit draws k[n]: out[i] = smallest j with cdf[n_cdf-1]*(k/RAND_MAX) <= cdf[j]. */
int r3d_test_cdf_search(const double *cdf, uint32_t n_cdf, const uint32_t *k,
                        uint32_t n, uint32_t *out, int use_guide_table);
/* use_guide_table: 0 = the reference's plain bisection, 1 = exact guide table of the default size,
 * n > 1 = exact guide table with 2^n buckets. */

/* GetPathToBoundary (media.cpp:236,518,668) for phonons in given cells:
 * in[i] = {cell, type, x,y,z, theta, phi} as 7 doubles;
 * out[i] = {pathlen, time, x,y,z, theta, phi, atten, face} as 9 doubles. */
int r3d_test_path_to_boundary(r3d_handle *h, const double *in, uint32_t n, double *out);

/* AdvanceLength (media.cpp:208,442,859): in[i] = {cell,type,x,y,z,theta,phi,len};
 * out as above with face = -1. */
int r3d_test_advance(r3d_handle *h, const double *in, uint32_t n, double *out);

/* The snapshot deposit's partial advance (see r3d_set_snapshots), with the kernel's device function:
 * in[i] = {cell, type, x,y,z, theta, phi, dt}: the point reached at travel time dt (0 <= dt < the travel time to the
 * boundary) along the move to the boundary from that state; out as r3d_test_advance. */
int r3d_test_advance_time(r3d_handle *h, const double *in, uint32_t n, double *out);

/* Phonon::Transform (phonons.cpp:116-170): in[i] = {theta,phi,pol, rtheta,rphi,rpol};
 * out[i] = {theta,phi,pol}. */
int r3d_test_transform(const double *in, uint32_t n, double *out);

/* RTCoef (rtcoef.cpp:30-588): in[i] = {nx,ny,nz, dx,dy,dz, rhoR, vpR, vsR, rhoT, vpT, vsT,
 * intype(0 P,1 SH,2 SV), notransmit, k_choose}; out[i] = {prob[6] (R_P,R_SV,R_SH,T_P,T_SV,T_SH),
 * choice, dirx,diry,dirz, pdx,pdy,pdz}. */
int r3d_test_rtcoef(const double *in, uint32_t n, double *out);

/* The straight-line division and square root of the hot paths (r3d_device.cuh: qdiv, qsqrt0) next to the compiler's own:
 * in[i] = {a, b}; out[i] = {qdiv(a, b), a / b, qsqrt0(a), sqrt(a)}.  The pairs must agree bit for bit over the operand
 * range of a phonon event. */
int r3d_test_arith(const double *in, uint32_t n, double *out);

/* The path-length draw's logarithm (Scatterer::GetRandomPathLength, scatterers.cpp:297-307): in[i] = k, a 31-bit draw as a
 * double; out[i] = {the kernel's -log(1 - k / 2^31), the math library's}. */
int r3d_test_pathlog(const double *in, uint32_t n, double *out);

/* Seismometer::CatchPhonon (dataout.cpp:103-216) for one seismometer record:
 * in[i] = {seis[18], time, x,y,z, theta,phi,pol, type, amp, vel};
 * out[i] = {caught(0/1), bin, ex,ey,ez, e}. */
int r3d_test_catch(double bin_dt, uint32_t n_bins, const double *in, uint32_t n, double *out);

void r3d_destroy(r3d_handle *h);

const char *r3d_last_error(void);

int r3d_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* R3D_GPU_H_ */
