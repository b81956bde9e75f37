// r3d_resident.cuh -- the propagate loop as a block-local wavefront over phonons that LIVE IN SHARED MEMORY.
//
// One iteration of the reference's Propagate loop (phonons.cpp:542) is one of a few very different events
// (scatter / cell-to-cell hand-over / surface reflection with a seismometer scan / loss / time-out / new phonon).
// Two earlier designs and what ncu said about them (profiles/):
//   * one phonon per thread in one fused loop: a warp holds all event kinds at once -- 5.3 of 32 lanes active,
//     instruction-fetch stalls (profiles/r1_fused_kernel.md);
//   * a wavefront over a phonon pool in HBM, three kernels per step with global index queues: lanes converge, but
//     the draw and interface kernels touch a sparse subset of the struct-of-arrays pool, so every 8-byte field
//     costs a 32-byte sector: 400 B of DRAM traffic per draw and 1.1 kB per face event, 50-67 % of DRAM
//     bandwidth spent on state that is never reused by another SM (profiles/r1_wavefront_hbm.md).
// Here every CTA is persistent (one per SM) and owns S phonon slots in its shared memory: 130 B per slot, 1504 slots in a
// 196 KB carve-out, which leaves 60 KB of the SM's 256 KB to L1.  The CTA alternates two phases, separated by
// __syncthreads():
//   phase 1  advance  (slots ready to move)  time-out / validity checks, the event's draws (path length first; all draws the
//                                            event will consume are taken from its Philox block here, in order), distance
//                                            to boundary, move, cheap hand-overs inline; classification of the event
//   (between the phases: one atomicAdd on the job's work counter grants new phonon indices for the slots that phase 1 freed)
//   phase 2  face     (queued face events)   seismometer collection by the whole warp (collect_warp: arrivals one at a time, each
//                                            one's candidates from the uniform-grid index spread over the lanes), R/T coefficients
//            draw     (queued table draws)   exact guide-table CDF search + take-off-angle fetch from HBM/L2, then
//                                            Phonon::Transform; for a freed slot: the new phonon's index and ray type
//                                            first, then its take-off angle and direction, in the same chunk - it
//                                            advances in the next phase 1, like every other slot
//            bend     (queued plain bends)   Snell bending at faces that neither collect nor reflect
// Within a phase, warps pull 32-entry chunks of ONE kind of work from index queues in shared memory, so a warp
// executes one kind of event (P and S face events are queued apart, source and scatter draws too).  State never
// leaves the SM; HBM sees only the table gathers (~150 B per draw) and the bin atomics.
// The phases are also what keeps the working set of CODE small: the same slots behind barrier-free ring queues, with
// every kind of event running at once, thrashed the instruction caches (9 cycles of fetch stall per issued instruction)
// and ran 35 % slower (profiles/r1_resident_kernel.md, which also records the other variants that were measured); one
// merged work list per iteration with the follow-ups one iteration late (round 2) ran 12-35 % slower for the same reason
// (profiles/experiments/r2_merged_worklist.md).
#pragma once
#include "r3d_device.cuh"

namespace r3d {

#define R3D_FULL 0xffffffffu
// R3D_CHECK=1 (make check -> libr3dgpu_check.so, tests/test_gpu_invariants.py): the queue invariants are asserted on the device
// and a violation traps.  Two lists share a buffer from its two ends, and a slot that is taken out of a list leaves a stale
// entry behind: an entry added to the same buffer for a slot that still has one there can make the ends meet - silently,
// unless the model frees many slots per iteration (both times this happened only the halfspace runs crashed).
#ifndef R3D_CHECK
#define R3D_CHECK 0
#endif
__device__ __noinline__ void check_fail(int what, uint32_t a, uint32_t b) {
  printf("r3d: queue invariant %d violated in block %d (%u, %u)\n", what, (int)blockIdx.x, a, b);
  __trap();
}
#ifndef R3D_MERGE_FACES
#define R3D_MERGE_FACES 0      // 1: P and S face events share chunks (one partial chunk less per iteration, but every chunk then runs the S-only code too)
#endif
#define R3D_NT 512             // most threads per CTA of any cell kind (Cell::threads sets each kernel's launch bound, one CTA per SM)

struct Job {
  unsigned long long first, n, seed;
  r3d_phonon_final *finals;                  // trace mode: per-phonon end states (or null)
  r3d_event *events;                         // trace mode: event reports (or null)
  unsigned long long *event_cursor, event_cap;
  uint32_t event_mask;
};

struct Phonon {
  double time, pathlen, recent, aexp;
  v3 loc, dir, s1;
  uint32_t moves, cell;
  int type;
};

// ---- energy snapshots (include/r3d_gpu.h r3d_set_snapshots) -----------------------------------------------------------
// The grids of one device: cell ((k * (n_vox + 1) + v) * 2 + type) holds snapshot k, voxel v (x fastest; v = n_vox is the
// snapshot's "outside" cell) and ray type.  A kernel parameter of its own, after all others, so that the kernels without
// snapshots keep their parameter layout.
struct SnapGrid {
  const double *times;              // [n_times], increasing, in [0, ttl]
  double *energy;                   // [n_times][n_vox + 1][2]  sum of amp^2
  unsigned long long *count;        // [n_times][n_vox + 1][2]  records
  double origin[3], voxel[3];
  uint32_t dims[3], n_vox, n_times;
};
// One move, as a deposit needs it: everything is what the phonon had in registers when it moved (the move's Path is
// derived again from the start point, by the same function, only for moves that straddle a snapshot time).
struct SnapMove {
  double t_a, t_b, aexp, len, time;  // time before / after Phonon::Move, attenuation exponent before, the move's length and time
  v3 loc, dir;                       // start point and direction
  uint32_t cell;
  int type;
  bool moved;
};

// ---- per-thread tallies (dataout.cpp:591-617), flushed once per CTA into its own row.  32-bit per thread (a thread
// sees a few thousand phonons per launch), 64-bit from the CTA's row onwards. ----------------------------------
struct Tally {
  uint32_t v[R3D_NCOUNTERS];
  R3D_DEV void clear() {
#pragma unroll
    for (int i = 0; i < R3D_NCOUNTERS; i++) v[i] = 0;
  }
  R3D_DEV void died(uint32_t fate) {
    const uint32_t f = fate & 0xFF;
    v[R3D_CNT_LOST] += (f == R3D_FATE_LOST);
    v[R3D_CNT_TIMEOUT] += (f == R3D_FATE_TIMEOUT);
    v[R3D_CNT_INVALID] += (f == R3D_FATE_INVALID);
    if (f == R3D_FATE_INVALID) v[R3D_CNT_DIAG] |= (fate >> 8);
  }
  // all threads of the CTA must call this
  R3D_DEV void flush(unsigned long long *row, unsigned long long (*sm)[R3D_NCOUNTERS]) {
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < R3D_NCOUNTERS; k++) {
      unsigned long long x = v[k];
      if (k == R3D_CNT_DIAG) { for (int o = 16; o > 0; o >>= 1) x |= __shfl_down_sync(R3D_FULL, x, o); }
      else { for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(R3D_FULL, x, o); }
      if (lane == 0) sm[warp][k] = x;
    }
    __syncthreads();
    if (threadIdx.x < R3D_NCOUNTERS) {
      unsigned long long x = 0;
      for (unsigned w = 0; w < nw; w++) { if (threadIdx.x == R3D_CNT_DIAG) x |= sm[w][threadIdx.x]; else x += sm[w][threadIdx.x]; }
      if (x) { if (threadIdx.x == R3D_CNT_DIAG) row[threadIdx.x] |= x; else row[threadIdx.x] += x; }
    }
  }
};

// ---- the slots (phonons.hpp:69-126): struct of arrays in shared memory, 16-byte elements where fields travel
// together.  Every accessor derives its address from the CTA's dynamic shared-memory symbol, so the compiler emits
// LDS / STS (pointers kept in a struct were treated as generic and cost a long-scoreboard wait per access).
// Per slot: 120 B of phonon state + its entries in the 5 index queues = 130 B, 1504 slots (47 chunks, three rounds of the 16
// warps of the wide builds) in the 196 KB carve-out.  Of the four running sums of a phonon, the time alive and the attenuation
// exponent feed the seismometer bins and stay FP64; the path length and the travel time since the last validity check are only
// ever tested (NaN, sign, zero, below the slow-concern threshold: phonons.cpp:554-584) and are kept as FP32 sums - in the trace
// kernels, whose end states are compared with the reference's to 1e-8, as FP64.  (The 142-byte slot of the first half of
// round 2 held 1408 slots = 44 chunks = 2.75 rounds: profiles/r2_experiments.md.)
#define R3D_SLOT_STATE 120u            // bytes of phonon state per slot (non-trace); the rest of R3D_SLOT_BYTES are its entries in the 5 index queues
#define R3D_SLOT_STATE_TRACE 128u
#define R3D_SLOT_BYTES 130u
#define R3D_SLOT_BYTES_TRACE 154u      // + FP64 path length / recent travel time (8) + four u32 per-phonon counters (16)
extern __shared__ __align__(16) unsigned char r3d_smem[];
struct Clock4 { double time, pathlen, recent, aexp; };
template <bool TRACE>
struct Slots {
  uint32_t S, table_bytes;      // table_bytes: the staged small-model tables (multiple of 16; 0 = none)
  static constexpr uint32_t kState = TRACE ? R3D_SLOT_STATE_TRACE : R3D_SLOT_STATE;
  R3D_DEV double &time(uint32_t s) const { return reinterpret_cast<double *>(r3d_smem)[s]; }                        // time alive
  R3D_DEV double &aexp(uint32_t s) const { return reinterpret_cast<double *>(r3d_smem + (size_t)S * 8)[s]; }        // attenuation exponent
  R3D_DEV double2 &lxy(uint32_t s) const { return reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 16)[s]; }   // location x, y
  R3D_DEV double2 &lzdz(uint32_t s) const { return reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 32)[s]; }  // location z, direction z
  R3D_DEV double2 &dxy(uint32_t s) const { return reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 48)[s]; }   // direction x, y (unit direction of travel, e3)
  R3D_DEV double2 &sxy(uint32_t s) const { return reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 64)[s]; }   // polarisation direction x, y (unit, s1; carried
  R3D_DEV double &sz(uint32_t s) const { return reinterpret_cast<double *>(r3d_smem + (size_t)S * 80)[s]; }      //  for P phonons too, like mPol, phonons.hpp:109-118)
  // the queued request: draw {31-bit draw, table | kind}; face {draw for the S-polarisation choice, draw for the
  // outcome choice}, exit face id in the two top bits
  R3D_DEV uint2 &req(uint32_t s) const { return reinterpret_cast<uint2 *>(r3d_smem + (size_t)S * 88)[s]; }
  R3D_DEV uint2 &mc(uint32_t s) const { return reinterpret_cast<uint2 *>(r3d_smem + (size_t)S * 96)[s]; }        // (move count, cell | ray type << 31)
  R3D_DEV uint32_t &ord(uint32_t s) const { return reinterpret_cast<uint32_t *>(r3d_smem + (size_t)S * 104)[s]; }   // draw ordinal
  R3D_DEV uint32_t &idx(uint32_t s) const { return reinterpret_cast<uint32_t *>(r3d_smem + (size_t)S * 108)[s]; }   // phonon index relative to the launch's first phonon (r3d_gpu.cu: at most 2^30 phonons per launch)
  // (path length, travel time since the last validity check): float2, trace kernels double2
  R3D_DEV Clock4 clock(uint32_t s) const {
    Clock4 c; c.time = time(s); c.aexp = aexp(s);
    if (TRACE) { const double2 v = reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 112)[s]; c.pathlen = v.x; c.recent = v.y; }
    else { const float2 v = reinterpret_cast<float2 *>(r3d_smem + (size_t)S * 112)[s]; c.pathlen = (double)v.x; c.recent = (double)v.y; }
    return c;
  }
  R3D_DEV void set_clock(uint32_t s, double t, double pathlen, double recent, double ae) const {
    time(s) = t; aexp(s) = ae;
    if (TRACE) reinterpret_cast<double2 *>(r3d_smem + (size_t)S * 112)[s] = make_double2(pathlen, recent);
    else reinterpret_cast<float2 *>(r3d_smem + (size_t)S * 112)[s] = make_float2((float)pathlen, (float)recent);
  }
  // (move count, cell, draw ordinal, ray type) as one value
  R3D_DEV uint4 meta(uint32_t s) const { const uint2 v = mc(s); return make_uint4(v.x, v.y & 0x7fffffffu, ord(s), v.y >> 31); }
  R3D_DEV void set_meta(uint32_t s, uint32_t moves, uint32_t cell, uint32_t ordinal, uint32_t type) const {
    mc(s) = make_uint2(moves, cell | (type << 31)); ord(s) = ordinal;
  }
  R3D_DEV void set_cell_type(uint32_t s, uint32_t cell, uint32_t type) const { mc(s).y = cell | (type << 31); }
  R3D_DEV unsigned char *tables() const { return r3d_smem + (size_t)S * kState; }                                   // staged small-model tables (Tab)
  // trace mode only: [4][S] catches, scatters, iterations, event reports made
  R3D_DEV uint32_t &tr(int which, uint32_t s) const { return reinterpret_cast<uint32_t *>(r3d_smem + (size_t)S * kState + table_bytes)[(uint32_t)which * S + s]; }
  // queues of slot indices: buffer 0 / 1 = [cur|next] ready-to-advance slots from the front, free slots from the back;
  // buffer 2 = table draws: scatter draws from the front, slots freed in phase 1 (waiting for a new phonon) from the back; buffer 3 = face events: P from
  // the front, S from the back; buffer 4 = plain ray bending at a face (no catch, no R/T solve)
  R3D_DEV uint16_t *queue(uint32_t buf) const {
    return reinterpret_cast<uint16_t *>(r3d_smem + (size_t)S * (kState + (TRACE ? 16u : 0u)) + table_bytes) + (size_t)buf * S;
  }
};


// ---- -log(r) for the path-length draw (Scatterer::GetRandomPathLength, scatterers.cpp:297-307), every loop event ----------
// r = 1 - k 2^-31 is a normal double in (0, 1].  The library's log() is ~80 instructions of the advance chain; this one is
// ~28: r = 2^e m with m in [0.707, 1.414]; c = the nearest multiple of 1/64 to m (exact), d = m - c (exact), t = d / c from a
// 47-entry table of (1 / c, log c) in shared memory (752 B: a larger one would cost the CTA a chunk of slots);
// log r = e log 2 + log c + log1p(t) with |t| < 0.0111 and a degree-7 series (remainder 3e-17).  For r next to 1 - short paths - e = 0, c = 1, log c = 0 and the result is log1p(d) to full
// relative accuracy; elsewhere the absolute error is ~2e-16 on values above 0.004: relative error < 1e-13, far inside the
// 1e-10 of the parity bar (checked against log() on the device: tests/test_gpu_subkernels.py::test_path_length_log).
#ifndef R3D_DIET_LOG
#define R3D_DIET_LOG 1
#endif
#define R3D_LOG_FIRST 45u
#define R3D_LOG_ENTRIES 47u          // c = 45/64 .. 91/64
R3D_DEV double2 *log_table() { __shared__ double2 tab[R3D_LOG_ENTRIES]; return tab; }
R3D_DEV void log_table_fill(double2 *tab) {          // all threads of the CTA; followed by a barrier
  for (uint32_t i = threadIdx.x; i < R3D_LOG_ENTRIES; i += blockDim.x) {
    const double c = (double)(R3D_LOG_FIRST + i) * (1.0 / 64.0);
    tab[i] = make_double2(1.0 / c, (R3D_LOG_FIRST + i == 64u) ? 0.0 : log(c));
  }
}
R3D_DEV double neg_log_unit(const double2 *tab, double r) {
#if R3D_DIET_LOG
  const int hi = __double2hiint(r);
  int e = (hi >> 20) - 1023;
  double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(r));      // [1, 2)
  if (m > 1.4142135623730951) { m *= 0.5; e += 1; }                                       // [0.7071, 1.4142]
  const int i = __double2int_rn(m * 64.0);                                                 // 45 .. 91
  const double d = m - (double)i * (1.0 / 64.0);
  const double2 cl = tab[i - (int)R3D_LOG_FIRST];
  const double t = d * cl.x;
  double p = __fma_rn(t, 1.0 / 7.0, -1.0 / 6.0);
  p = __fma_rn(p, t, 1.0 / 5.0);
  p = __fma_rn(p, t, -1.0 / 4.0);
  p = __fma_rn(p, t, 1.0 / 3.0);
  p = __fma_rn(p, t, -1.0 / 2.0);
  p = __fma_rn(p, t, 1.0);
  return -__fma_rn((double)e, 0.6931471805599453, __fma_rn(p, t, cl.y));
#else
  return -log(r);
#endif
}

// counters of the queues: cnt[0..3] = {advance, free} x {buffer 0, buffer 1}; cnt[4..8] = scatter draws, source draws, P faces,
// S faces, bends
// per-CTA clocks written at the end of a launch: [0] cycles in phase 1, [1] cycles in phase 2, [2] iterations,
// [3..6] warp-cycles inside advance / bend / face / draw chunks, [7..10] number of such chunks, [11] warp-cycles
// spent outside chunks (barriers, waiting for the last chunk of a phase)
#define R3D_NCLOCKS 12
struct Ctl {
  unsigned long long t_kind[4], t_idle;
  uint32_t n_kind[4];
  unsigned long long base;          // first phonon (relative to the job) granted to this CTA in this iteration
  uint32_t grant_a, grant_b, exhausted, done, cursor[2];       // grant_a, grant_b: new phonons for the two lists of free slots
  uint32_t cnt[9];
  unsigned long long t_phase[2];    // clock cycles spent in phase 1 / phase 2 (thread 0's view)
  uint32_t iterations;
};
enum { CNT_SCAT = 4, CNT_SRC, CNT_FP, CNT_FS, CNT_BEND };

// ---- the small per-model tables every event reads: cell parameters, cell -> scatterer, face flags and neighbours,
// mean free paths, conversion probabilities.  Layered and shell models have tens of cells (a few KB): SMALL stages
// them in shared memory, because the table gathers of phase 2 stream through the (small) L1 and would otherwise
// turn each of these reads into an L2 round trip in the middle of an event.  The tetrahedral models (2275 cells,
// 0.7 MB) read them through L1 / L2.
template <bool SMALL>
struct Tab {
  uint32_t base, np, nf, o_mfp, o_whole, o_other, o_scat, o_flags;     // byte offsets into r3d_smem
  R3D_DEV void init(const DevModel &M, uint32_t base_) {
    base = base_; np = M.cell_nparam; nf = M.faces_per_cell;
    o_mfp = base + M.n_cells * np * 8u;
    o_whole = o_mfp + M.n_scat * 16u;
    o_other = o_whole + M.n_scat * 64u;
    o_scat = o_other + M.n_cells * nf * 4u;
    o_flags = o_scat + M.n_cells * 4u;
  }
  static __host__ __device__ uint32_t bytes(uint32_t n_cells, uint32_t np, uint32_t nf, uint32_t n_scat) {
    return (n_cells * np * 8u + n_scat * 80u + n_cells * nf * 5u + n_cells * 4u + 15u) / 16u * 16u;
  }
  R3D_DEV void stage(const DevModel &M) const {          // all threads of the CTA; followed by a barrier
    if (!SMALL) return;
    double *d = reinterpret_cast<double *>(r3d_smem + base);
    for (uint32_t i = threadIdx.x; i < M.n_cells * np; i += blockDim.x) d[i] = M.cell_params[i];
    d = reinterpret_cast<double *>(r3d_smem + o_mfp);
    for (uint32_t i = threadIdx.x; i < M.n_scat * 2u; i += blockDim.x) d[i] = M.scat_mfp[i];
    d = reinterpret_cast<double *>(r3d_smem + o_whole);
    for (uint32_t i = threadIdx.x; i < M.n_scat * 8u; i += blockDim.x) d[i] = M.scat_whole[i];
    uint32_t *u = reinterpret_cast<uint32_t *>(r3d_smem + o_other);
    for (uint32_t i = threadIdx.x; i < M.n_cells * nf; i += blockDim.x) u[i] = M.face_other[i];
    u = reinterpret_cast<uint32_t *>(r3d_smem + o_scat);
    for (uint32_t i = threadIdx.x; i < M.n_cells; i += blockDim.x) u[i] = M.cell_scat[i];
    uint8_t *b = r3d_smem + o_flags;
    for (uint32_t i = threadIdx.x; i < M.n_cells * nf; i += blockDim.x) b[i] = M.face_flags[i];
  }
  R3D_DEV const double *cell(const DevModel &M, uint32_t i) const {
    if (SMALL) return reinterpret_cast<const double *>(r3d_smem + base) + i * np;
    return M.cell_params + (size_t)i * np;
  }
  R3D_DEV double mfp(const DevModel &M, uint32_t scat, int type) const {
    if (SMALL) return reinterpret_cast<const double *>(r3d_smem + o_mfp)[scat * 2u + (uint32_t)type];
    return __ldg(M.scat_mfp + scat * 2u + (uint32_t)type);
  }
  R3D_DEV const double *whole(const DevModel &M, uint32_t scat, int type) const {
    if (SMALL) return reinterpret_cast<const double *>(r3d_smem + o_whole) + (scat * 2u + (uint32_t)type) * 4u;
    return M.scat_whole + (scat * 2u + (uint32_t)type) * 4u;
  }
  R3D_DEV uint32_t other(const DevModel &M, uint32_t fi) const {
    if (SMALL) return reinterpret_cast<const uint32_t *>(r3d_smem + o_other)[fi];
    return __ldg(M.face_other + fi);
  }
  R3D_DEV uint32_t scat(const DevModel &M, uint32_t cell) const {
    if (SMALL) return reinterpret_cast<const uint32_t *>(r3d_smem + o_scat)[cell];
    return __ldg(M.cell_scat + cell);
  }
  R3D_DEV uint32_t flags(const DevModel &M, uint32_t fi) const {
    if (SMALL) return (r3d_smem + o_flags)[fi];
    return __ldg(M.face_flags + fi);
  }
};

// The first of a draw's three dependent gathers is its guide entry.  Its address is known when the draw is queued (phase
// 1), a whole phase before it is used: pull the sector into L2 then.
R3D_DEV void prefetch_guide(const DevModel &M, bool is_src, uint32_t table, uint32_t kdraw) {
  if (M.guide_shift >= 32) return;
  const uint32_t *g = (is_src ? M.src_guide : M.scat_guide) + (size_t)table * M.guide_stride + (kdraw >> M.guide_shift);
  asm volatile("prefetch.global.L2 [%0];" ::"l"(g));
}

// A warp takes the next 32-entry chunk of the current phase's work list
R3D_DEV uint32_t next_chunk(uint32_t *cursor) {
  uint32_t c = 0;
  if ((threadIdx.x & 31u) == 0) c = atomicAdd(cursor, 1u);
  return __shfl_sync(R3D_FULL, c, 0);
}

template <bool TRACE>
R3D_DEV void write_final(const Slots<TRACE> &A, const Job &J, uint32_t s, const Phonon &p, uint32_t fate, uint32_t ordinal) {
  if (!TRACE || !J.finals) return;
  r3d_phonon_final *f = J.finals + A.idx(s);
  f->time = p.time; f->pathlen = p.pathlen; f->amp = exp(-p.aexp);
  f->loc[0] = p.loc.x; f->loc[1] = p.loc.y; f->loc[2] = p.loc.z;
  angles_of(p.dir, f->theta, f->phi);
  f->pol = pol_angle_of(p.dir, p.s1);
  f->moves = p.moves; f->cell = p.cell; f->type = (uint32_t)p.type; f->fate = fate;
  f->draws = ordinal; f->catches = A.tr(0, s); f->scatters = A.tr(1, s); f->iters = A.tr(2, s);
}

// Event report (dataout.cpp:484-617): the phonon's state as output_phonon_dataline() prints it.  Trace mode only.
template <bool TRACE>
R3D_DEV void emit(const Slots<TRACE> &A, const Job &J, uint32_t s, uint32_t kind, int type, double time, double pathlen, v3 loc,
                  v3 dir, double aexp, uint32_t cell, uint32_t moves, uint32_t reason = 0) {
  if (!TRACE) return;
  if (!J.events || !((J.event_mask >> kind) & 1u)) return;
  const uint32_t seq = A.tr(3, s)++;
  const unsigned long long at = atomicAdd(J.event_cursor, 1ull);
  if (at >= J.event_cap) return;
  r3d_event *e = J.events + at;
  e->phonon = J.first + A.idx(s); e->seq = seq; e->kind = kind; e->type = (uint32_t)type; e->moves = moves; e->cell = cell; e->reason = reason;
  e->time = time; e->pathlen = pathlen; e->loc[0] = loc.x; e->loc[1] = loc.y; e->loc[2] = loc.z;
  angles_of(dir, e->theta, e->phi);
  e->amp = exp(-aexp);
}

// one 32-byte take-off-angle record through the read-only path (two 16-byte loads of the same sector)
R3D_DEV double4 load_toa(const double4 *p) {
  const double2 a = ld_table(reinterpret_cast<const double2 *>(p)), b = ld_table(reinterpret_cast<const double2 *>(p) + 1);
  return make_double4(a.x, a.y, b.x, b.y);
}

// CellFace::VelocityJump (media_cellface.cpp:83-99).  Equal velocities give exactly 0 in the reference too
// (2*(0)/(v+v)); testing for that first keeps 0/x off the slow path of the FP64 division.
template <class Cell, class TabT>
R3D_DEV double velocity_jump(const DevModel &M, const TabT &tab, uint32_t cell, uint32_t other, v3 loc) {
  const double *c = tab.cell(M, cell), *o = tab.cell(M, other);
  double v1 = Cell::veloc(c, 0, loc), v2 = Cell::veloc(o, 0, loc);
  double dvp = (v1 == v2 && v1 > 0.0) ? 0.0 : fabs(2 * (v2 - v1) / (v2 + v1));
  v1 = Cell::veloc(c, 1, loc); v2 = Cell::veloc(o, 1, loc);
  double dvs = (v1 == v2 && v1 > 0.0) ? 0.0 : fabs(2 * (v2 - v1) / (v2 + v1));
  return (dvp > dvs) ? dvp : dvs;
}

// What happens at a face (phonons.cpp:629-676), decided where the phonon arrives so that the draws the face
// event will consume can be taken from the stream in order.
enum { FACE_NONE = 0, FACE_LOST, FACE_CONTINUOUS, FACE_BEND, FACE_FULLRT };
template <class Cell, class TabT>
R3D_DEV int face_action(const DevModel &M, const TabT &tab, uint32_t fl, uint32_t cell, uint32_t other, v3 loc) {
  if (fl & R3D_FACE_REFLECT) return FACE_FULLRT;                                    // phonons.cpp:640-646
  if (fl & R3D_FACE_ADJOIN) {                                                       // Phonon::Refract, phonons.cpp:225-255
    if (fl & R3D_FACE_DISCON) return FACE_FULLRT;
    if (fl & R3D_FACE_JUMP_KNOWN) return (fl & R3D_FACE_JUMP) ? FACE_BEND : FACE_CONTINUOUS;     // layered cells: decided in r3d_create
    return (velocity_jump<Cell>(M, tab, cell, other, loc) > 0.00001) ? FACE_BEND : FACE_CONTINUOUS;
  }
  return FACE_LOST;                                                                 // phonons.cpp:675
}

// Phonon::Refraction_FullRT (phonons.cpp:429-476) + CellFace::GetRTBasis (media_cellface.cpp:122-149)
template <class Cell, class TabT>
R3D_DEV void refraction_fullrt(const DevModel &M, const TabT &tab, Phonon &p, int face, bool adjoin, uint32_t other,
                               uint32_t k_spol, uint32_t k_choose) {
  const double *c = tab.cell(M, p.cell);
  RTCoef rt;
  rt.init(Cell::normal(c, face, p.loc), p.dir);
  rt.densR = Cell::dens(c, p.loc);
  rt.velR[0] = Cell::veloc(c, 0, p.loc);
  rt.velR[1] = Cell::veloc(c, 1, p.loc);
  if (adjoin) {
    const double *o = tab.cell(M, other);
    rt.densT = Cell::dens(o, p.loc);
    rt.velT[0] = Cell::veloc(o, 0, p.loc);
    rt.velT[1] = Cell::veloc(o, 1, p.loc);
  } else {                                    // free surface
    rt.densT = 0.0; rt.velT[0] = 1e-12; rt.velT[1] = 1e-12; rt.notransmit = true;
  }
  int intype = R3D_RAY_P;
  if (p.type == R3D_RAY_S) intype = rt.choose_spol(p.s1, k_spol);          // DirectionOfMotion() of an S phonon is s1
  rt.get_coefs(intype);
  rt.choose(k_choose);
  const bool reflected = (rt.choice == R_P || rt.choice == R_SV || rt.choice == R_SH);
  const v3 outdir = unit_else(rt.chosen_ray_dir(), V(0, 0, 1));          // mDir.Set(outdir.Theta(), outdir.Phi())
  p.type = (rt.choice == R_P || rt.choice == T_P) ? R3D_RAY_P : R3D_RAY_S;
  if (p.type == R3D_RAY_S) p.s1 = pol_from_pdom(outdir, rt.chosen_pdom());  // phonons.cpp:459-465
  else p.s1 = carry_pol(p.dir, p.s1, outdir);                                 // mPol is left as it was
  p.dir = outdir;
  if (!reflected) p.cell = other;
}

// Phonon::Refraction_Bend (phonons.cpp:311-405)
template <class Cell, class TabT>
R3D_DEV void refraction_bend(const DevModel &M, const TabT &tab, Phonon &p, int face, uint32_t other) {
  const double *c = tab.cell(M, p.cell);
  const double *o = tab.cell(M, other);
  const v3 mdir = p.dir;
  const v3 fnorm = Cell::normal(c, face, p.loc);
  const v3 fpara = inplane_unit_perp(fnorm, mdir);
  const v3 fparash = cross(fnorm, fpara);
  const double veli = Cell::veloc(c, p.type, p.loc), velo = Cell::veloc(o, p.type, p.loc);
  const double sini = dot(fpara, mdir);
  double sino = (velo / veli) * sini;
  bool transfer; double coso;
  if (sino >= 1.0) { transfer = false; sino = sini; coso = -1.0 * dot(fnorm, mdir); }
  else { transfer = true; coso = sqrt(1.0 - (sino * sino)); }
  const v3 outraw = add(scal(fpara, sino), scal(fnorm, coso));
  const v3 outdir = unit_else(outraw, V(0, 0, 1));
  if (p.type != R3D_RAY_P) {
    const v3 svbasei = cross(fparash, mdir), svbaseo = cross(fparash, outraw);
    const double shcomi = dot(p.s1, fparash), svcomi = dot(p.s1, svbasei);
    p.s1 = pol_from_pdom(outdir, add(scal(fparash, shcomi), scal(svbaseo, svcomi)));
  } else {
    p.s1 = hats(outdir).th;                     // polout = 0 for P (phonons.cpp:366, 393)
  }
  p.dir = outdir;
  if (transfer) p.cell = other;
}

// kinds of follow-up work a slot can be queued for
enum { OUT_NONE = -1, OUT_ADV = 0, OUT_FREE, OUT_SCAT, OUT_SRC, OUT_FP, OUT_FS, OUT_BEND };

// Append this lane's slot to the queue of its follow-up kind: lanes of one kind find each other with one match.any,
// their leader reserves room with one shared-memory atomic.  All lanes of the warp call this.
template <bool TRACE>
R3D_DEV void route(const Slots<TRACE> &A, Ctl &C, int nxt, int out, uint32_t s) {
  const unsigned peers = __match_any_sync(R3D_FULL, out);
  if (out < 0) return;
  const unsigned lane = threadIdx.x & 31u;
  const int leader = __ffs(peers) - 1;
  const uint32_t ci = (out < 2) ? (uint32_t)(nxt * 2 + out) : (uint32_t)(2 + out);
  uint32_t base = 0;
  if ((int)lane == leader) base = atomicAdd(&C.cnt[ci], (uint32_t)__popc(peers));
  base = __shfl_sync(peers, base, leader);
  const uint32_t j = base + __popc(peers & ((1u << lane) - 1u));
  const uint32_t buf = (out < 2) ? (uint32_t)nxt : 1u + ((uint32_t)out >> 1);       // OUT_BEND = 6 -> buffer 4, from the front
  if (R3D_CHECK && (j >= A.S || s >= A.S)) check_fail(1, j, s);
  A.queue(buf)[(out & 1) ? A.S - 1u - j : j] = (uint16_t)s;
}

// =====================================================================================================
// phase 1a: one Propagate-loop iteration up to the event's classification (phonons.cpp:542-623)
// =====================================================================================================
template <class Cell, bool TRACE, bool SNAP, class TabT>
R3D_DEV int advance_one(const DevModel &M, const Job &J, const Slots<TRACE> &A, const TabT &tab, uint32_t s, Tally &T, SnapMove &D) {
  Phonon p;
  const Clock4 ck = A.clock(s);
  const double2 lxy = A.lxy(s), lzdz = A.lzdz(s), dxy = A.dxy(s);
  const uint4 meta = A.meta(s);
  p.time = ck.time; p.pathlen = ck.pathlen; p.recent = ck.recent; p.aexp = ck.aexp;
  p.loc = V(lxy.x, lxy.y, lzdz.x);
  p.dir = V(dxy.x, dxy.y, lzdz.y);
  p.moves = meta.x; p.cell = meta.y; p.type = (int)meta.w;
  uint32_t ordinal = meta.z;
  T.v[R3D_CNT_EVENTS]++;
  if (TRACE) A.tr(2, s)++;
  uint32_t fate = 0;
  int out = OUT_ADV;
  if (p.time > M.ttl) fate = R3D_FATE_TIMEOUT;                  // phonons.cpp:549-552
  else if ((p.moves % 128u) == 127u) {                          // phonons.cpp:554-584
    int why = -1;
    if (isnan(p.pathlen)) why = R3D_INV_PATH_NAN;
    else if (isnan(p.time)) why = R3D_INV_TIME_NAN;
    else if (p.pathlen < 0) why = R3D_INV_PATH_NEGATIVE;
    else if ((p.time < 0) || (p.recent < 0)) why = R3D_INV_TIME_NEGATIVE;
    else if (p.recent == 0) why = R3D_INV_STUCK;
    else if (p.recent < M.slow_concern) why = R3D_INV_SLOW;
    else if (p.moves > M.loop_concern) why = R3D_INV_LOOP_EXCEED;
    if (why >= 0) fate = R3D_FATE_INVALID | ((1u << why) << 8);
    else p.recent = 0;
  }
  bool dir_changed = false, s1_loaded = false;
  if (!fate) {
    const double *c = tab.cell(M, p.cell);
    // The event's draws come first: path length, then at most two more, all from Philox block ordinal/4 (and the next one when
    // they run over its end).  (The reference draws the path length after the distance to the boundary, phonons.cpp:590-601;
    // taking it before keeps the generator's state and the logarithm out of the registers while the ray geometry - up to 20
    // doubles of scratch for a curved ray - is live.  A phonon that times out on an infinite path has consumed no draw:
    // `ordinal` only moves further down.)
    Rng g; g.init(J.seed, J.first + A.idx(s));
    const uint32_t o = ordinal & 3u, b = ordinal >> 2;
    g.block(b);
    const uint32_t w1 = g.w[1], w2 = g.w[2], w3 = g.w[3];
    const uint32_t k_path = ((o == 0) ? g.w[0] : (o == 1) ? w1 : (o == 2) ? w2 : w3) >> 1;
    const uint32_t scat = tab.scat(M, p.cell);
    // Scatterer::GetRandomPathLength (scatterers.cpp:297-307)
    const double r = 1.0 - ((double)k_path) * (1.0 / 2147483648.0);      // k / (RAND_MAX + 1): a power of two, exact either way
    const double scatlen = neg_log_unit(log_table(), r) * tab.mfp(M, scat, p.type);
    typename Cell::Path P;
    const double edgelen = Cell::path(M, c, p.type, p.loc, p.dir, P);
    if (edgelen == pinf()) fate = R3D_FATE_TIMEOUT;             // phonons.cpp:595-598
    else {
      const bool scatter = scatlen < edgelen;
      const Travel tr = Cell::advance(M, c, p.type, scatter ? scatlen : edgelen, p.loc, p.dir, P);
      if (SNAP) {
        D.t_a = p.time; D.aexp = p.aexp; D.len = tr.len; D.time = tr.time;
        D.loc = p.loc; D.dir = p.dir; D.cell = p.cell; D.type = p.type; D.moved = true;
      }
      // Phonon::Move (phonons.cpp:62-70)
      p.pathlen += tr.len; p.time += tr.time; p.recent += tr.time;
      p.loc = tr.loc; p.aexp += tr.aexp; p.moves += 1;
      if (SNAP) D.t_b = p.time;
      if (Cell::curved) {            // the ray turned: the polarisation ANGLE is what the reference carries along
        const double2 sxy = A.sxy(s);
        p.s1 = carry_pol(p.dir, V(sxy.x, sxy.y, A.sz(s)), tr.dir);
        p.dir = tr.dir;
        dir_changed = true; s1_loaded = true;
      }
      // what follows, and how many more draws it takes
      uint32_t more = 0, fl = 0, other = 0;
      int action = FACE_NONE;
      if (scatter) {
        if (!M.no_deflect) more = 2;                              // conversion type, take-off angle (scatterers.cpp:332,336)
      } else {
        const uint32_t fi = p.cell * M.faces_per_cell + P.face;
        fl = tab.flags(M, fi);
        other = tab.other(M, fi);
        action = face_action<Cell>(M, tab, fl, p.cell, other, p.loc);
        if (action == FACE_FULLRT) more = (p.type == R3D_RAY_S) ? 2 : 1;   // [S polarisation choice,] outcome choice
      }
      uint32_t k1 = 0, k2 = 0;
      if (more) {
        uint32_t x0 = 0, x1 = 0;
        if (o + more > 3u) { g.block(b + 1); x0 = g.w[0]; x1 = g.w[1]; }
        const uint32_t i1 = o + 1, i2 = o + 2;
        k1 = ((i1 == 1) ? w1 : (i1 == 2) ? w2 : (i1 == 3) ? w3 : x0) >> 1;
        k2 = ((i2 == 2) ? w2 : (i2 == 3) ? w3 : (i2 == 4) ? x0 : x1) >> 1;
      }
      ordinal += 1 + more;
      if (scatter) {
        // Scatterer::GetRandomScatteredRelativePhonon (scatterers.cpp:318-363); the table draw is queued
        if (M.no_deflect) {
          if (!s1_loaded) { const double2 sxy = A.sxy(s); p.s1 = V(sxy.x, sxy.y, A.sz(s)); s1_loaded = true; }
          double st, ct;
          sincos(M.min_theta, &st, &ct);                          // Phonon(ThetaPhi(0,0)) nudged to min_theta, pol 0
          transform(p.dir, p.s1, st, ct, 0.0, 1.0, 0.0, 1.0);
          dir_changed = true;
          T.v[R3D_CNT_SCATTERS]++;
          if (TRACE) A.tr(1, s)++;
          emit<TRACE>(A, J, s, R3D_EV_SCT, p.type, p.time, p.pathlen, p.loc, p.dir, p.aexp, p.cell, p.moves);
        } else {
          const uint32_t conv = cdf_search_small(tab.whole(M, scat, p.type), 4, k1);
          A.req(s) = make_uint2(k2, scat * 4 + conv);
          prefetch_guide(M, false, scat * 4 + conv, k2);
          out = OUT_SCAT;
        }
      } else if (action == FACE_LOST && !(fl & R3D_FACE_COLLECT)) fate = R3D_FATE_LOST;
      else if (action == FACE_CONTINUOUS && !(fl & R3D_FACE_COLLECT)) {                 // Refraction_Continuous
        p.cell = other;
        emit<TRACE>(A, J, s, (other == meta.y) ? R3D_EV_REF : R3D_EV_CEL, p.type, p.time, p.pathlen, p.loc, p.dir, p.aexp, p.cell, p.moves);
      }
      else {
        // collection and / or R/T and / or bending: phase 2.  For P only the outcome draw exists (k1).
        const uint32_t ka = (p.type == R3D_RAY_S) ? k1 : 0u, kb = (p.type == R3D_RAY_S) ? k2 : k1;
        A.req(s) = make_uint2(ka | ((uint32_t)(P.face & 1) << 31), kb | ((uint32_t)(P.face >> 1) << 31));
        out = (action == FACE_BEND && !(fl & R3D_FACE_COLLECT)) ? OUT_BEND : (R3D_MERGE_FACES || p.type == R3D_RAY_P) ? OUT_FP : OUT_FS;
      }
    }
  }
  if (fate) {
    T.died(fate);
    if (TRACE) {
      if (!s1_loaded) { const double2 sxy = A.sxy(s); p.s1 = V(sxy.x, sxy.y, A.sz(s)); }
      const uint32_t f = fate & 0xFFu;
      emit<TRACE>(A, J, s, f == R3D_FATE_LOST ? R3D_EV_LST : f == R3D_FATE_TIMEOUT ? R3D_EV_TMO : R3D_EV_INV, p.type, p.time, p.pathlen,
                  p.loc, p.dir, p.aexp, p.cell, p.moves, fate >> 8);
      write_final<TRACE>(A, J, s, p, fate, ordinal);
    }
    return OUT_FREE;
  }
  A.set_clock(s, p.time, p.pathlen, p.recent, p.aexp);
  A.lxy(s) = make_double2(p.loc.x, p.loc.y);
  A.lzdz(s) = make_double2(p.loc.z, p.dir.z);
  if (dir_changed) {
    A.dxy(s) = make_double2(p.dir.x, p.dir.y);
    A.sxy(s) = make_double2(p.s1.x, p.s1.y);
    A.sz(s) = p.s1.z;
  }
  A.set_meta(s, p.moves, p.cell, ordinal, (uint32_t)p.type);
  return out;
}

// phase 2 (first half of a new-phonon chunk): a free slot takes the next phonon: ShearDislocation::GenerateEventPhonon (events.cpp:111-124) ->
// PhononSource::GenerateRandomPhonon (sources.cpp:156-170) -> Phonon ctor (phonons.hpp:193-207)
template <bool TRACE>
R3D_DEV void refill_one(const DevModel &M, const Job &J, const Slots<TRACE> &A, uint32_t s, unsigned long long rel, Tally &T) {
  const unsigned long long idx = J.first + rel;
  Rng g; g.init(J.seed, idx);
  g.block(0);
  const uint32_t rt3 = cdf_search_small(M.src_whole, 3, g.w[0] >> 1);
  A.req(s) = make_uint2(g.w[1] >> 1, rt3);                    // the take-off angle is drawn next, in the same chunk
  A.set_clock(s, 0.0, 0.0, 0.0, 0.0);
  A.lxy(s) = make_double2(M.src_loc[0], M.src_loc[1]);
  A.lzdz(s) = make_double2(M.src_loc[2], 0.0);
  A.idx(s) = (uint32_t)rel;
  A.set_meta(s, 0u, M.src_cell, 2u, (rt3 == R3D_RAY_P) ? R3D_RAY_P : R3D_RAY_S);
  if (TRACE) { A.tr(0, s) = 0; A.tr(1, s) = 0; A.tr(2, s) = 0; A.tr(3, s) = 0; }
  T.v[R3D_CNT_PHONONS]++;
}

// =====================================================================================================
// phase 2a: ProbDist::GetRandomIndex on the queued table + take-off angle, then either the new phonon's
// direction (sources.cpp:156-170) or Phonon::Transform (phonons.cpp:116-170).
// A draw is a chain of three dependent gathers from HBM / L2 (guide entry -> CDF entries -> take-off angle).  A thread
// works on U draws at once and issues each stage's loads for all of them before it consumes any, so a warp has
// 32 U chains in flight instead of 32 (ncu: with one draw per thread phase 2 took two thirds of the kernel, waiting).
// =====================================================================================================
#ifndef R3D_FINAL
#define R3D_FINAL 8u         // a guide span of up to this many CDF entries is read in one round trip; wider ones are narrowed
#endif                       // first (ncu: with 4, the narrowing loop ran at 4.4 of 32 lanes and cost 6 % of all instructions)
#ifndef R3D_CHUNK_CLOCKS
#define R3D_CHUNK_CLOCKS 0   // 1: every warp clocks its chunks by kind (make clocks; scripts/chunk_clocks.py); 3.7 % of all instructions
#endif
#ifndef R3D_DRAW_U
#define R3D_DRAW_U 1
#endif
template <bool TRACE, int U>
R3D_DEV void draw_batch(const DevModel &M, const Job &J, const Slots<TRACE> &A, const uint16_t *q, bool from_back, uint32_t j0, uint32_t count,
                        bool is_src, Tally &T, uint32_t (&s)[U], bool (&have)[U]) {
  const unsigned lane = threadIdx.x & 31u;
  const double *cdf0 = is_src ? M.src_cdf : M.scat_cdf;
  const uint32_t *guide0 = is_src ? M.src_guide : M.scat_guide;
  uint32_t kd[U], tbl[U], ti[U];
  const double *cdf[U];
#pragma unroll
  for (int u = 0; u < U; u++) {
    const uint32_t j = j0 + (uint32_t)u * 32u + lane;
    have[u] = j < count;
    s[u] = have[u] ? (uint32_t)q[from_back ? A.S - 1u - j : j] : 0u;
    const uint2 rq = have[u] ? A.req(s[u]) : make_uint2(0u, 0u);
    kd[u] = rq.x; tbl[u] = rq.y;
    cdf[u] = cdf0 + (size_t)tbl[u] * M.n_toa;
  }
  if (M.guide_shift < 32) {
    // cdf_search_guided (r3d_device.cuh), stage by stage over the U draws
    uint32_t k1[U], k2[U];
    double r[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t *g = guide0 + (size_t)tbl[u] * M.guide_stride + (kd[u] >> M.guide_shift);
      k1[u] = ld_table(g); k2[u] = ld_table(g + 1);
      r[u] = ld_table(cdf[u] + (M.n_toa - 1));
    }
#pragma unroll
    for (int u = 0; u < U; u++) r[u] = r[u] * over_randmax(kd[u]);
    // Wide buckets (they cover low-probability entries): narrow 8-fold per round trip with seven independent probes
    // (same predicate, cdf non-decreasing), for all U draws in lockstep so that the probes of one round overlap.
    for (;;) {
      bool wide = false;
#pragma unroll
      for (int u = 0; u < U; u++) wide |= (k2[u] - k1[u] > R3D_FINAL);
      if (!__any_sync(R3D_FULL, wide)) break;
      double pv[U][7];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t span = k2[u] - k1[u];
#pragma unroll
        for (uint32_t i = 0; i < 7; i++)
          pv[u][i] = (span > R3D_FINAL) ? ld_table(cdf[u] + k1[u] + (uint32_t)(((unsigned long long)span * (i + 1)) >> 3)) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t span = k2[u] - k1[u];
        if (span > R3D_FINAL) {
          uint32_t c = 0;
#pragma unroll
          for (uint32_t i = 0; i < 7; i++) c += (r[u] <= pv[u][i]) ? 0u : 1u;
          // probes 0..c-1 are below r, probe c (if any) is the first one at or above it
          uint32_t lo = k1[u], hi = k2[u];
#pragma unroll
          for (uint32_t i = 0; i < 7; i++) {
            const uint32_t pr = k1[u] + (uint32_t)(((unsigned long long)span * (i + 1)) >> 3);
            if (i + 1 == c) lo = pr + 1;
            if (i == c) hi = pr;
          }
          k1[u] = lo; k2[u] = hi;
        }
      }
    }
    double v[U][R3D_FINAL];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (uint32_t i = 0; i < R3D_FINAL; i++) v[u][i] = (k1[u] + i < k2[u]) ? ld_table(cdf[u] + k1[u] + i) : pinf();
#pragma unroll
    for (int u = 0; u < U; u++) {
      uint32_t c = 0;
#pragma unroll
      for (uint32_t i = 0; i < R3D_FINAL; i++) c += (r[u] <= v[u][i]) ? 0u : 1u;
      ti[u] = k1[u] + c;
    }
  } else {
#pragma unroll
    for (int u = 0; u < U; u++) ti[u] = cdf_search_plain(cdf[u], M.n_toa, kd[u]);
  }
  double4 t[U];
  double2 rp[U];
#pragma unroll
  for (int u = 0; u < U; u++) {
    t[u] = load_toa(M.toa + ti[u]);                           // sin th, cos th, sin ph, cos ph
    rp[u] = make_double2(1.0, 0.0);                           // (cos, sin) of the relative polarisation angle
    if (!is_src && (tbl[u] & 3u) == 3u) rp[u] = ld_table(M.scat_spol + (size_t)(tbl[u] >> 2) * M.n_toa + ti[u]);
  }
#pragma unroll
  for (int u = 0; u < U; u++) {
    if (!have[u]) continue;
    const uint32_t su = s[u];
    if (is_src) {
      // new phonon: direction = the drawn take-off angle, polarisation angle pi/2 for SH else 0 (phonons.hpp:193-207)
      A.dxy(su) = make_double2(t[u].x * t[u].w, t[u].x * t[u].z);
      A.lzdz(su).y = t[u].y;
      if (tbl[u] == R3D_RAY_SH) { A.sxy(su) = make_double2(-t[u].z, t[u].w); A.sz(su) = 0.0; }                     // phi-hat
      else { A.sxy(su) = make_double2(t[u].y * t[u].w, t[u].y * t[u].z); A.sz(su) = -t[u].x; }                     // theta-hat
      if (TRACE && J.events) {             // events.cpp:120
        const uint4 meta = A.meta(su);
        emit<TRACE>(A, J, su, R3D_EV_GEN, (int)meta.w, 0.0, 0.0, V(M.src_loc[0], M.src_loc[1], M.src_loc[2]),
                    V(t[u].x * t[u].w, t[u].x * t[u].z, t[u].y), 0.0, meta.y, 0u);
      }
    } else {
      const uint32_t conv = tbl[u] & 3u;
      const double2 dxy = A.dxy(su), sxy = A.sxy(su);
      v3 e3 = V(dxy.x, dxy.y, A.lzdz(su).y), s1 = V(sxy.x, sxy.y, A.sz(su));
      transform(e3, s1, t[u].x, t[u].y, t[u].z, t[u].w, rp[u].y, rp[u].x);
      A.dxy(su) = make_double2(e3.x, e3.y);
      A.lzdz(su).y = e3.z;
      A.sxy(su) = make_double2(s1.x, s1.y);
      A.sz(su) = s1.z;
      A.mc(su).y = (A.mc(su).y & 0x7fffffffu) | ((conv & 1u) << 31);       // ray type: PP,PS,SP,SS -> P,S,P,S
      T.v[R3D_CNT_SCATTERS]++;
      if (TRACE) A.tr(1, su)++;
      if (TRACE && J.events) {             // phonons.cpp:616
        const Clock4 ck = A.clock(su);
        const double2 lxy = A.lxy(su);
        const uint4 meta = A.meta(su);
        emit<TRACE>(A, J, su, R3D_EV_SCT, (int)(conv & 1u), ck.time, ck.pathlen, V(lxy.x, lxy.y, A.lzdz(su).x), e3, ck.aexp, meta.y, meta.x);
      }
    }
  }
}

// =====================================================================================================
// phase 2b, first half: DataReporter::ReportPhononCollected (dataout.cpp:545-568) + Seismometer::CatchPhonon (dataout.cpp:
// 103-216) for the slots of one face chunk - as a WARP.  Every seismometer is pass-through (dataout.cpp:50), so all that
// contain the arrival point must bin it; candidates come from the uniform grid over the seismometers' bounding spheres.
// Few lanes of a chunk arrive at a collecting face, and each has a list of 10-20 candidates: lane by lane (even with the
// lanes meeting at their n-th candidate) the scan ran at 1.4 of 32 lanes and the exact test at 1.3-2, 6.8 % of the warp
// instructions and 10 % of the stall samples of the whole-Earth model.  Here the warp takes the arrivals one at a time
// and spreads each one's candidates over its lanes: the arrival's state is read from its slot in shared memory by all
// lanes (one broadcast read per field), 32 candidates get the sphere pre-test at once, and the lanes whose candidate passed
// run the exact test and the bin update together.  The bins go straight to L2 as reductions (red.global.add.f64 / .u64:
// 5.3e7 sectors in 124 ms on that model = 0.009 % of the L1-to-L2 write throughput, profiles/r2_histogram.md), so there is
// nothing for an aggregation step in shared memory to win; catches per (seismometer, bin) are independent arrivals.
// All 32 lanes call this; `have` = the lane holds a slot of the chunk.
// =====================================================================================================
template <class Cell, bool TRACE, class TabT>
R3D_DEV void collect_warp(const DevModel &M, const Slots<TRACE> &A, const TabT &tab, bool have, uint32_t s, Tally &T) {
  if (M.n_seis == 0) return;
  const unsigned lane = threadIdx.x & 31u;
  uint32_t i0 = 0, i1 = 0;
  if (have) {
    const uint4 meta = A.meta(s);
    const uint2 q = A.req(s);
    const int face = (int)((q.x >> 31) | ((q.y >> 31) << 1));
    if (tab.flags(M, meta.y * M.faces_per_cell + face) & R3D_FACE_COLLECT) {
      const double2 lxy = A.lxy(s);
      const int cx_ = grid_axis_cell(lxy.x, M.grid_min[0], M.grid_inv_h[0]);
      const int cy_ = grid_axis_cell(lxy.y, M.grid_min[1], M.grid_inv_h[1]);
      const int cz_ = grid_axis_cell(A.lzdz(s).x, M.grid_min[2], M.grid_inv_h[2]);
      if (cx_ >= 0 && cy_ >= 0 && cz_ >= 0 && cx_ < (int)M.grid_dim[0] && cy_ < (int)M.grid_dim[1] && cz_ < (int)M.grid_dim[2]) {
        const uint32_t gcell = ((uint32_t)cz_ * M.grid_dim[1] + (uint32_t)cy_) * M.grid_dim[0] + (uint32_t)cx_;
        i0 = __ldg(M.grid_start + gcell);
        i1 = __ldg(M.grid_start + gcell + 1);
      }
    }
  }
  unsigned pending = __ballot_sync(R3D_FULL, i0 < i1);
  while (pending) {
    const int src = __ffs(pending) - 1;
    pending &= pending - 1u;
    const uint32_t ss = __shfl_sync(R3D_FULL, s, src), b0 = __shfl_sync(R3D_FULL, i0, src), b1 = __shfl_sync(R3D_FULL, i1, src);
    // the arrival (same addresses in every lane: broadcast reads)
    const double t_alive = A.time(ss), aexp = A.aexp(ss);
    const double2 lxy = A.lxy(ss), lzdz = A.lzdz(ss), dxy = A.dxy(ss), sxy = A.sxy(ss);
    const uint4 meta = A.meta(ss);
    const v3 loc = V(lxy.x, lxy.y, lzdz.x), dir = V(dxy.x, dxy.y, lzdz.y);
    const int type = (int)meta.w;
    const v3 dopm = (type == R3D_RAY_P) ? dir : V(sxy.x, sxy.y, A.sz(ss));     // Phonon::DirectionOfMotion (phonons.cpp:201-211)
    uint32_t caught = 0;
    for (uint32_t base = b0; base < b1; base += 32u) {
      const uint32_t j = base + lane;
      if (j < b1) {
        const uint32_t k2 = __ldg(M.grid_items + j);
        const double2 qa = __ldg(reinterpret_cast<const double2 *>(M.seis_sphere + k2));
        const double2 qb = __ldg(reinterpret_cast<const double2 *>(M.seis_sphere + k2) + 1);
        const double ddx = qa.x - loc.x, ddy = qa.y - loc.y, ddz = qb.x - loc.z;
        if (ddx * ddx + ddy * ddy + ddz * ddz <= qb.y) {            // may be within the gather radius: the exact CatchPhonon test
          const double vel = Cell::veloc(tab.cell(M, meta.y), type, loc);
          uint32_t bin; double e[4];
          if (seis_catch(M.seis + (size_t)k2 * R3D_SEIS_NPARAM, M.bin_dt, M.n_bins, t_alive, loc, dir, dopm, type, exp(-aexp), vel, bin, e)) {
            const size_t bb = (size_t)k2 * M.n_bins + bin;
            atomicAdd(M.energies + bb * 5 + 0, e[0]);
            atomicAdd(M.energies + bb * 5 + 1, e[1]);
            atomicAdd(M.energies + bb * 5 + 2, e[2]);
            atomicAdd(M.energies + bb * 5 + 3 + type, e[3]);
            atomicAdd(M.counts + bb * 2 + type, 1ull);
            caught++;
          }
        }
      }
    }
    T.v[R3D_CNT_CATCHES] += caught;                    // (a tally is summed over the threads at the end: whose it is does not matter)
    if (TRACE && caught) atomicAdd(&A.tr(0, ss), caught);
  }
}

// =====================================================================================================
// phase 2b: everything that happens at a face that is not a plain hand-over: collection (dataout.cpp:545-568,
// 103-216), free-surface / discontinuity R/T (phonons.cpp:429-476), Snell bending (phonons.cpp:311-405)
// =====================================================================================================
template <class Cell, bool TRACE, class TabT>
R3D_DEV int face_one(const DevModel &M, const Job &J, const Slots<TRACE> &A, const TabT &tab, uint32_t s, Tally &T) {
  Phonon p;
  const Clock4 ck = A.clock(s);
  const double2 lxy = A.lxy(s), lzdz = A.lzdz(s), dxy = A.dxy(s), sxy = A.sxy(s);
  const uint4 meta = A.meta(s);
  const uint2 q = A.req(s);
  p.time = ck.time; p.pathlen = ck.pathlen; p.recent = ck.recent; p.aexp = ck.aexp;
  p.loc = V(lxy.x, lxy.y, lzdz.x);
  p.dir = V(dxy.x, dxy.y, lzdz.y);
  p.s1 = V(sxy.x, sxy.y, A.sz(s));
  p.moves = meta.x; p.cell = meta.y; p.type = (int)meta.w;
  const int face = (int)((q.x >> 31) | ((q.y >> 31) << 1));
  const uint32_t k_spol = q.x & 0x7fffffffu, k_choose = q.y & 0x7fffffffu;
  const uint32_t fi = p.cell * M.faces_per_cell + face;
  const uint32_t fl = tab.flags(M, fi), other = tab.other(M, fi);

  if (fl & R3D_FACE_COLLECT) emit<TRACE>(A, J, s, R3D_EV_COL, p.type, p.time, p.pathlen, p.loc, p.dir, p.aexp, p.cell, p.moves);
  // ---- reflection / refraction (phonons.cpp:640-676) ---------------------------------------------------
  const int action = face_action<Cell>(M, tab, fl, p.cell, other, p.loc);
  if (action == FACE_FULLRT) refraction_fullrt<Cell>(M, tab, p, face, (fl & R3D_FACE_ADJOIN) != 0, other, k_spol, k_choose);
  else if (action == FACE_BEND) refraction_bend<Cell>(M, tab, p, face, other);
  else if (action == FACE_CONTINUOUS) p.cell = other;
  else {
    T.died(R3D_FATE_LOST);
    emit<TRACE>(A, J, s, R3D_EV_LST, p.type, p.time, p.pathlen, p.loc, p.dir, p.aexp, p.cell, p.moves);
    write_final<TRACE>(A, J, s, p, R3D_FATE_LOST, meta.z);
    return OUT_FREE;
  }
  // phonons.cpp:640-664: a reflection face always reports REF; a neighbour face REF if the cell is unchanged, else CEL
  emit<TRACE>(A, J, s, ((fl & R3D_FACE_REFLECT) || p.cell == meta.y) ? R3D_EV_REF : R3D_EV_CEL, p.type, p.time, p.pathlen, p.loc, p.dir,
              p.aexp, p.cell, p.moves);
  A.dxy(s) = make_double2(p.dir.x, p.dir.y);
  A.lzdz(s).y = p.dir.z;
  A.sxy(s) = make_double2(p.s1.x, p.s1.y);
  A.sz(s) = p.s1.z;
  A.set_cell_type(s, p.cell, (uint32_t)p.type);
  return OUT_ADV;
}

// phase 2c: Snell bending at a face that neither collects nor reflects (phonons.cpp:311-405).  Layered models with
// velocity contrasts cross such a face in half of their events; queued apart so that these cheap events do not sit in
// the same warps as R/T solves.
template <class Cell, bool TRACE, class TabT>
R3D_DEV void bend_one(const DevModel &M, const Job &J, const Slots<TRACE> &A, const TabT &tab, uint32_t s) {
  Phonon p;
  const double2 lxy = A.lxy(s), lzdz = A.lzdz(s), dxy = A.dxy(s), sxy = A.sxy(s);
  const uint4 meta = A.meta(s);
  const uint2 q = A.req(s);
  p.loc = V(lxy.x, lxy.y, lzdz.x);
  p.dir = V(dxy.x, dxy.y, lzdz.y);
  p.s1 = V(sxy.x, sxy.y, A.sz(s));
  p.cell = meta.y; p.type = (int)meta.w;
  const int face = (int)((q.x >> 31) | ((q.y >> 31) << 1));
  refraction_bend<Cell>(M, tab, p, face, tab.other(M, p.cell * M.faces_per_cell + face));
  A.dxy(s) = make_double2(p.dir.x, p.dir.y);
  A.lzdz(s).y = p.dir.z;
  A.sxy(s) = make_double2(p.s1.x, p.s1.y);
  A.sz(s) = p.s1.z;
  A.set_cell_type(s, p.cell, (uint32_t)p.type);
  if (TRACE && J.events) {
    const Clock4 ck = A.clock(s);
    emit<TRACE>(A, J, s, (p.cell == meta.y) ? R3D_EV_REF : R3D_EV_CEL, p.type, ck.time, ck.pathlen, p.loc, p.dir, ck.aexp, p.cell, meta.x);
  }
}

// =====================================================================================================
// phase 1b (SNAP kernels): the energy-snapshot records of the moves of one advance chunk.  A move over [t_a, t_b) makes
// one record for every snapshot time t_k in [t_a, t_b): the point at travel time t_k - t_a along the move (advance_time),
// weight amp^2 = exp(-2 aexp(t_k)), into the voxel floor((x - origin) / voxel) on each axis or the snapshot's outside cell.
// At early snapshot times most records of a warp fall into the same few voxels around the source, so the warp aggregates:
// lanes with the same (snapshot, voxel, type) find each other with one match.any, sum their weights in five shuffle rounds
// (pointer jumping along the lanes of the key), and the lowest lane adds the sum and the record count with one atomic each.
// A move can straddle several snapshot times: the warp repeats until no lane has a record left.  All 32 lanes call this.
// =====================================================================================================
template <class Cell, class TabT>
R3D_DEV void snap_deposit(const DevModel &M, const SnapGrid &Z, const TabT &tab, const SnapMove &D) {
  const unsigned lane = threadIdx.x & 31u;
  uint32_t k = Z.n_times;
  if (D.moved) {                                // first k with t_k >= t_a (none for a NaN t_a)
    uint32_t lo = 0, hi = Z.n_times;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(Z.times + mid) < D.t_a) lo = mid + 1; else hi = mid; }
    k = lo;
  }
  double tk = 0.0;
  if (k < Z.n_times) tk = __ldg(Z.times + k);
  bool pending = k < Z.n_times && D.t_a <= tk && tk < D.t_b;            // (false for NaN times)
  if (!__any_sync(R3D_FULL, pending)) return;
  typename Cell::Path P;
  const double *c = nullptr;
  if (pending) { c = tab.cell(M, D.cell); Cell::path(M, c, D.type, D.loc, D.dir, P); }
  do {
    uint32_t key = 0xffffffffu;
    double w = 0.0;
    if (pending) {
      const Travel tr = advance_time<Cell>(M, c, D.type, tk - D.t_a, D.loc, D.dir, P, D.len, D.time);
      w = exp(-2.0 * (D.aexp + tr.aexp));
      const double x[3] = {tr.loc.x, tr.loc.y, tr.loc.z};
      uint32_t v = 0, stride = 1;
      bool inside = true;
#pragma unroll
      for (int a = 0; a < 3; a++) {
        const double f = floor((x[a] - Z.origin[a]) / Z.voxel[a]);            // IEEE division, as the contract states
        inside = inside && f >= 0.0 && f < (double)Z.dims[a];
        if (inside) v += (uint32_t)f * stride;
        stride *= Z.dims[a];
      }
      key = ((k * (Z.n_vox + 1u) + (inside ? v : Z.n_vox)) << 1) | (uint32_t)D.type;
    }
    const unsigned peers = __match_any_sync(R3D_FULL, key);
    const unsigned above = peers & ~((2u << lane) - 1u);     // (lane 31: 2u << 31 wraps to 0, nothing above)
    int nxt = above ? __ffs(above) - 1 : -1;                  // next lane of the same key
    for (int r = 0; r < 5; r++) {                             // after round r each lane holds the sum of 2^(r+1) lanes of its key
      const int src = nxt >= 0 ? nxt : (int)lane;
      const double x = __shfl_sync(R3D_FULL, w, src);
      const int nn = __shfl_sync(R3D_FULL, nxt, src);
      if (nxt >= 0) { w += x; nxt = nn; }
    }
    if (pending && (int)lane == __ffs(peers) - 1) {
      atomicAdd(Z.energy + key, w);
      atomicAdd(Z.count + key, (unsigned long long)__popc(peers));
    }
    if (pending) {
      k++;
      if (k < Z.n_times) tk = __ldg(Z.times + k);
      pending = k < Z.n_times && tk < D.t_b;
    }
  } while (__any_sync(R3D_FULL, pending));
}

// =====================================================================================================
// the kernel: persistent CTAs, S slots each
// =====================================================================================================
template <class Cell, bool TRACE, bool SMALL, bool SNAP>
__global__ void __launch_bounds__(Cell::threads, 1)
propagate_kernel(const DevModel M, const Job J, uint32_t S, uint32_t table_bytes, unsigned long long *block_tally,
                 unsigned long long *block_clock, const SnapGrid Z) {
  __shared__ unsigned long long tally_sm[R3D_NT / 32][R3D_NCOUNTERS];
  __shared__ Ctl C;
  Slots<TRACE> A; A.S = S; A.table_bytes = table_bytes;
  Tab<SMALL> tab; tab.init(M, S * Slots<TRACE>::kState);
  tab.stage(M);
  log_table_fill(log_table());
  for (uint32_t i = threadIdx.x; i < S; i += blockDim.x) A.queue(0)[S - 1u - i] = (uint16_t)i;     // every slot starts free
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < 9; k++) C.cnt[k] = 0;
    C.cnt[OUT_FREE] = S;
    C.exhausted = 0; C.done = 0; C.grant_a = 0; C.grant_b = 0; C.t_phase[0] = 0; C.t_phase[1] = 0; C.iterations = 0;
    for (int k = 0; k < 4; k++) { C.t_kind[k] = 0; C.n_kind[k] = 0; }
    C.t_idle = 0;
  }
  const unsigned lane = threadIdx.x & 31u;
  Tally T; T.clear();
  int cur = 0;
  long long t0 = 0;
  const long long t_begin = clock64();
  __syncthreads();

  // A slot whose phonon dies in phase 1 gets its next phonon in phase 2 of the SAME iteration (grant at the phase boundary,
  // then ray type + take-off angle in one chunk), so that it advances again in the next phase 1.  (With the refill in the
  // next phase 1 and the source draw in the phase 2 after it, every phonon cost its slot one iteration in which nothing
  // advanced: 4.4 iterations for the 3.4 events of a phonon of the halfspace workload.)  Two lists of free slots: (B) the
  // slots freed in phase 1, at the back of the draw queue (buffer 2) - they cannot stay in the next advance queue's buffer,
  // which they re-enter from the front in phase 2 while their old entries still occupy its back; (A) the slots freed in
  // phase 2 (phonons lost at a collecting face: rare) and, at the start, all slots: the back of the current advance queue.
  for (;;) {
    const int nxt = cur ^ 1;
    if (threadIdx.x == 0) {
      C.cnt[nxt * 2 + OUT_ADV] = 0; C.cnt[nxt * 2 + OUT_FREE] = 0;
      C.cnt[CNT_SCAT] = 0; C.cnt[CNT_SRC] = 0; C.cnt[CNT_FP] = 0; C.cnt[CNT_FS] = 0; C.cnt[CNT_BEND] = 0;
      C.cursor[0] = 0; C.cursor[1] = 0;
      C.done = (C.cnt[cur * 2 + OUT_ADV] == 0 && C.exhausted);
      t0 = clock64();
    }
    __syncthreads();
    if (C.done) break;

    // ---- phase 1: advance chunks ---------------------------------------------------------------------------------
    {
      const uint32_t nA = C.cnt[cur * 2 + OUT_ADV];
      const uint32_t cA = (nA + 31u) >> 5;
      const uint16_t *q = A.queue((uint32_t)cur);
      for (;;) {
        const uint32_t c = next_chunk(&C.cursor[0]);
        if (c >= cA) break;
        int out = OUT_NONE;
        uint32_t s = 0;
#if R3D_CHUNK_CLOCKS
        const long long tc = clock64();
#endif
        const uint32_t j = c * 32u + lane;
        SnapMove D;
        D.moved = false;
        if (j < nA) { s = q[j]; out = advance_one<Cell, TRACE, SNAP>(M, J, A, tab, s, T, D); }
        if (SNAP) snap_deposit<Cell>(M, Z, tab, D);
        if (out == OUT_FREE) out = OUT_SRC;                     // list B: wants a new phonon in this iteration's phase 2
        route<TRACE>(A, C, nxt, out, s);
#if R3D_CHUNK_CLOCKS
        if (lane == 0) { atomicAdd(&C.t_kind[0], (unsigned long long)(clock64() - tc)); atomicAdd(&C.n_kind[0], 1u); }
#endif
      }
    }
    __syncthreads();
    // ---- grant new phonons to the free slots: one atomic on the job's work counter per CTA per iteration ------
    if (threadIdx.x == 0) {
      const long long t1 = clock64(); C.t_phase[0] += (unsigned long long)(t1 - t0); t0 = t1;
      const uint32_t nfa = C.cnt[cur * 2 + OUT_FREE], nfb = C.cnt[CNT_SRC], nf = nfa + nfb;
      if (R3D_CHECK) {                       // the two ends of every buffer, after phase 1
        if (C.cnt[nxt * 2 + OUT_ADV] + C.cnt[nxt * 2 + OUT_FREE] > S) check_fail(2, C.cnt[nxt * 2 + OUT_ADV], C.cnt[nxt * 2 + OUT_FREE]);
        if (C.cnt[CNT_SCAT] + C.cnt[CNT_SRC] > S) check_fail(3, C.cnt[CNT_SCAT], C.cnt[CNT_SRC]);
        if (C.cnt[CNT_FP] + C.cnt[CNT_FS] > S || C.cnt[CNT_BEND] > S) check_fail(4, C.cnt[CNT_FP] + C.cnt[CNT_FS], C.cnt[CNT_BEND]);
        // every slot is in exactly one list (slots are only dropped once the job has no phonon left for them)
        const uint32_t all = C.cnt[nxt * 2 + OUT_ADV] + C.cnt[nxt * 2 + OUT_FREE] + C.cnt[CNT_SCAT] + C.cnt[CNT_SRC] + C.cnt[CNT_FP] + C.cnt[CNT_FS] + C.cnt[CNT_BEND] + nfa;
        if (C.exhausted ? all > S : all != S) check_fail(5, all, S);
      }
      uint32_t grant = 0;
      if (nf && !C.exhausted) {
        const unsigned long long b = atomicAdd(M.next_phonon, (unsigned long long)nf);
        if (b < J.n) { const unsigned long long left = J.n - b; grant = (left < nf) ? (uint32_t)left : nf; C.base = b; }
        if (grant < nf) C.exhausted = 1;
      }
      C.grant_a = (grant < nfa) ? grant : nfa;
      C.grant_b = grant - C.grant_a;
    }
    __syncthreads();

    // ---- phase 2: face chunks (S, then P), then draw chunks (scatter, then new phonons), then bend chunks -----------
    {
      const uint32_t nFS = C.cnt[CNT_FS], nFP = C.cnt[CNT_FP], nDS = C.cnt[CNT_SCAT], nGA = C.grant_a, nGB = C.grant_b;
      constexpr uint32_t DB = 32u * R3D_DRAW_U;                 // draws per chunk
      const uint32_t nB = C.cnt[CNT_BEND];
      const uint32_t c0 = (nFS + 31u) >> 5, c1 = c0 + ((nFP + 31u) >> 5), c2 = c1 + (nDS + DB - 1u) / DB;
      const uint32_t c2b = c2 + (nGA + DB - 1u) / DB, c3 = c2b + (nGB + DB - 1u) / DB;
      const uint32_t c4 = c3 + ((nB + 31u) >> 5);
      const uint16_t *qd = A.queue(2), *qf = A.queue(3), *qb = A.queue(4);
      const uint16_t *qa = A.queue((uint32_t)cur);              // free lists: entry j of a list is q[S - 1 - j]
      const unsigned long long base = C.base;
      for (;;) {
        const uint32_t c = next_chunk(&C.cursor[1]);
        if (c >= c4) break;
#if R3D_CHUNK_CLOCKS
        const long long tc = clock64();
#endif
        if (c >= c3) {
          const uint32_t j = (c - c3) * 32u + lane;
          int out = OUT_NONE;
          uint32_t s = 0;
          if (j < nB) { s = qb[j]; bend_one<Cell, TRACE>(M, J, A, tab, s); out = OUT_ADV; }
          route<TRACE>(A, C, nxt, out, s);
        } else if (c < c1) {
          const bool from_back = c < c0;
          const uint32_t j = (from_back ? c : c - c0) * 32u + lane, count = from_back ? nFS : nFP;
          int out = OUT_NONE;
          uint32_t s = 0;
          const bool have = j < count;
          if (have) s = qf[from_back ? S - 1u - j : j];
          collect_warp<Cell, TRACE>(M, A, tab, have, s, T);
          if (have) out = face_one<Cell, TRACE>(M, J, A, tab, s, T);
          route<TRACE>(A, C, nxt, out, s);
        } else {
          const bool is_src = c >= c2, list_b = c >= c2b;
          const uint16_t *q = (is_src && !list_b) ? qa : qd;
          const uint32_t j0 = (is_src ? (list_b ? c - c2b : c - c2) : c - c1) * DB, count = is_src ? (list_b ? nGB : nGA) : nDS;
          if (is_src) {                       // new phonons first: index, ray type, request for the take-off angle
#pragma unroll
            for (int u = 0; u < R3D_DRAW_U; u++) {
              const uint32_t j = j0 + (uint32_t)u * 32u + lane;
              if (j < count) refill_one<TRACE>(M, J, A, q[S - 1u - j], base + (list_b ? nGA : 0u) + j, T);
            }
          }
          uint32_t s[R3D_DRAW_U];
          bool have[R3D_DRAW_U];
          draw_batch<TRACE, R3D_DRAW_U>(M, J, A, q, is_src, j0, count, is_src, T, s, have);
#pragma unroll
          for (int u = 0; u < R3D_DRAW_U; u++) route<TRACE>(A, C, nxt, have[u] ? OUT_ADV : OUT_NONE, s[u]);
        }
#if R3D_CHUNK_CLOCKS
        if (lane == 0) { const int kd = (c >= c3) ? 1 : (c < c1) ? 2 : 3; atomicAdd(&C.t_kind[kd], (unsigned long long)(clock64() - tc)); atomicAdd(&C.n_kind[kd], 1u); }
#endif
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      C.t_phase[1] += (unsigned long long)(clock64() - t0); C.iterations++;
      if (R3D_CHECK) {                       // after phase 2 every slot is ready to advance or free, in the next buffer
        const uint32_t all = C.cnt[nxt * 2 + OUT_ADV] + C.cnt[nxt * 2 + OUT_FREE];
        if (C.exhausted ? all > S : all != S) check_fail(6, C.cnt[nxt * 2 + OUT_ADV], C.cnt[nxt * 2 + OUT_FREE]);
      }
    }
    cur = nxt;
  }
  if (threadIdx.x == 0) {                    // warp time not spent inside chunks: barriers, waiting for a phase's last chunk
    const unsigned long long all = (unsigned long long)(clock64() - t_begin) * (blockDim.x >> 5);
    const unsigned long long busy = C.t_kind[0] + C.t_kind[1] + C.t_kind[2] + C.t_kind[3];
    C.t_idle = all > busy ? all - busy : 0;
  }
  T.flush(block_tally + (size_t)blockIdx.x * R3D_NCOUNTERS, tally_sm);      // (contains a barrier)
  if (threadIdx.x == 0) {
    unsigned long long *bc = block_clock + (size_t)R3D_NCLOCKS * blockIdx.x;
    bc[0] += C.t_phase[0]; bc[1] += C.t_phase[1]; bc[2] += C.iterations;
    for (int k = 0; k < 4; k++) { bc[3 + k] += C.t_kind[k]; bc[7 + k] += C.n_kind[k]; }
    bc[11] += C.t_idle;
  }
}

}  // namespace r3d
