// r3d_gpu.cu -- the C ABI of include/r3d_gpu.h and the host side of the propagate path (sm_100a only).
//
// The device work is in r3d_resident.cuh (one persistent kernel; the phonons live in shared memory) and
// r3d_device.cuh (the physics).  This file uploads a flattened model into one device arena, builds the exact
// guide tables for the CDF searches, and launches one kernel per job: every device of a handle has one worker
// thread that launches queued jobs on the device's stream, so r3d_run() returns at once and devices run
// concurrently.  There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <deque>
#include <stdlib.h>
#include <chrono>
#include <cmath>
#include "r3d_gpu.h"
#include "r3d_device.cuh"
#include "r3d_resident.cuh"

using namespace r3d;


namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(e_ == cudaErrorMemoryAllocation ? R3D_ENOMEM : R3D_ECUDA,                        \
                  std::string(#call) + ": " + cudaGetErrorString(e_));                             \
  } while (0)

// The public entry points select the device they work on; the caller's current device is put back on return.
struct DeviceGuard {
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---------------------------------------------------------------------------
// model-preparation kernels
// ---------------------------------------------------------------------------
__global__ void pack_toa_kernel(const double *th, const double *ph, double4 *out, uint32_t n, double mn, double mx) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double t = th[i];
  if (t < mn) t = mn;                    // Phonon::nudge_if_singular (phonons.hpp:335-344), applied where the
  if (t > mx) t = mx;                    // reference constructs a Phonon from a TOA entry
  double st, ct, sp, cp;
  sincos(t, &st, &ct);
  sincos(ph[i], &sp, &cp);
  out[i] = make_double4(st, ct, sp, cp);
}
__global__ void pack_spol_kernel(const double *spol, double2 *out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s_, c_;
  sincos(spol[i], &s_, &c_);
  out[i] = make_double2(c_, s_);
}
// guide[j] = lower_bound of r(k = min(j << shift, RAND_MAX)) for every table
__global__ void build_guide_kernel(const double *cdf, uint32_t n_toa, uint32_t n_tables, uint32_t shift, uint32_t stride, uint32_t *guide) {
  unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (unsigned long long)n_tables * stride) return;
  uint32_t t = (uint32_t)(i / stride), j = (uint32_t)(i % stride);
  unsigned long long k = (unsigned long long)j << shift;
  if (k > 2147483647ull) k = 2147483647ull;
  guide[i] = cdf_search_plain(cdf + (size_t)t * n_toa, n_toa, (uint32_t)k);
}
__global__ void check_monotone_kernel(const double *cdf, uint32_t n_toa, uint32_t n_tables, int *bad) {
  unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (unsigned long long)n_tables * n_toa) return;
  if ((i % n_toa) == 0) { if (!(cdf[i] >= 0.0)) *bad = 1; return; }
  if (!(cdf[i] >= cdf[i - 1])) *bad = 1;
}
__global__ void seis_sphere_kernel(const double *seis, uint32_t n, double4 *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *s = seis + (size_t)i * R3D_SEIS_NPARAM;
  double ro = fmax(s[14], s[15]);
  out[i] = make_double4(s[0], s[1], s[2], ro * ro * (1.0 + 1e-12));   // d^2 > w  =>  sqrt(d^2) > r_out for both types
}

// counters[k] = sum (OR for the diagnostic word) over the per-block tally rows
__global__ void reduce_tally_kernel(const unsigned long long *rows, uint32_t n_rows, unsigned long long *counters) {
  __shared__ unsigned long long sm[256];
  const int k = blockIdx.x;
  unsigned long long x = 0;
  for (uint32_t r = threadIdx.x; r < n_rows; r += blockDim.x) { if (k == R3D_CNT_DIAG) x |= rows[(size_t)r * R3D_NCOUNTERS + k]; else x += rows[(size_t)r * R3D_NCOUNTERS + k]; }
  sm[threadIdx.x] = x;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { if (k == R3D_CNT_DIAG) sm[threadIdx.x] |= sm[threadIdx.x + o]; else sm[threadIdx.x] += sm[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    counters[k] = sm[0];
    if (k == R3D_CNT_DIAG)                     // one 0/1 lane per reason bit, after the counters (sums of lanes survive an all-reduce)
      for (int b = 0; b < R3D_NDIAG_LANES; b++) counters[R3D_NCOUNTERS + b] = (sm[0] >> b) & 1ull;
  }
}

// Sum of the accumulators of the devices of one handle, by a kernel on device slot 0 that reads its peers' memory over
// NVLink (devices in slot order, so the sums have the bits a host loop over the devices would produce).
#define R3D_MAX_PEERS 16
struct PeerPtrs { const void *p[R3D_MAX_PEERS]; int n; };
__global__ void combine_f64_kernel(PeerPtrs P, size_t n, double *out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    double v = static_cast<const double *>(P.p[0])[i];
    for (int g = 1; g < P.n; g++) v += static_cast<const double *>(P.p[g])[i];
    out[i] = v;
  }
}
__global__ void combine_u64_kernel(PeerPtrs P, size_t n, size_t or_index, unsigned long long *out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    unsigned long long v = static_cast<const unsigned long long *>(P.p[0])[i];
    for (int g = 1; g < P.n; g++) {
      const unsigned long long x = static_cast<const unsigned long long *>(P.p[g])[i];
      if (i == or_index) v |= x; else v += x;
    }
    out[i] = v;
  }
}

// ScatterParams::GSATO with XSATO and PSATO inlined (scatparams.cpp:75-194); one take-off angle per thread.
// g[0..3][n] = gpp, gps, gsp, gss; spol[n].  `numer` = 8 pi^1.5 eps^2 a^3 Gamma(kappa+1.5) / Gamma(kappa) (host).
__global__ void gsato_kernel(r3d_scatter_params P, double numer, const double *th, const double *ph, uint32_t n, double *g, double *spol) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double psi = th[i], zeta = ph[i];
  const double gam0 = P.gam0, gam2x = gam0 * gam0, nu = P.nu, el = P.el;
  // XSATO (4.50)
  const double cpsi = cos(psi), c2psi = cos(2. * psi), spsi = sin(psi), czeta = cos(zeta), szeta = sin(zeta), spsi2 = spsi * spsi;
  const double xpp = (1. / gam2x) * (nu * (-1. + cpsi + (2. / gam2x) * spsi2) - 2. + (4. / gam2x) * spsi2);
  const double xps = -spsi * (nu * (1. - (2. / gam0) * cpsi) - (4. / gam0) * cpsi);
  const double xsp = (1. / gam2x) * spsi * czeta * (nu * (1. - (2. / gam0) * cpsi) - (4. / gam0) * cpsi);
  const double xss_psi = czeta * (nu * (cpsi - c2psi) - 2. * c2psi);
  const double xss_zeta = szeta * (nu * (cpsi - 1.) + 2. * cpsi);
  // GSATO (4.52) with PSATO (2.10, von Karman)
  const double pi4 = 4. * kPi, el4 = pow(el, 4.0), gam2 = pow(gam0, 2.0), a2 = P.a * P.a, ex = P.kappa + 1.5;
  double arg = (2. * el / gam0) * sin(psi / 2.);
  double gpp = (el4 / pi4) * (xpp * xpp) * (numer / pow(1. + a2 * arg * arg, ex));
  if (gpp < 1.e-30) gpp = 0.;
  arg = (el / gam0) * sqrt(1. + gam2 - 2. * gam0 * cos(psi));
  const double pm = numer / pow(1. + a2 * arg * arg, ex);
  double gps = (1. / gam0) * (el4 / pi4) * (xps * xps) * pm;
  if (gps < 1.e-30) gps = 0.;
  double gsp = gam0 * (el4 / pi4) * (xsp * xsp) * pm;
  if (gsp < 1.e-30) gsp = 0.;
  arg = 2. * el * sin(psi / 2.);
  double gss = (el4 / pi4) * (xss_psi * xss_psi + xss_zeta * xss_zeta) * (numer / pow(1. + a2 * arg * arg, ex));
  if (gss < 1.e-30) gss = 0.;
  g[i] = gpp; g[(size_t)n + i] = gps; g[2 * (size_t)n + i] = gsp; g[3 * (size_t)n + i] = gss;
  spol[i] = atan2(xss_zeta, xss_psi);
}

// ---------------------------------------------------------------------------
// sub-kernel hooks (r3d_test_*)
// ---------------------------------------------------------------------------
__global__ void test_cdf_kernel(const double *cdf, uint32_t n_cdf, const uint32_t *guide, uint32_t shift, const uint32_t *k, uint32_t n, uint32_t *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = (n_cdf <= 4) ? cdf_search_small(cdf, (int)n_cdf, k[i]) : cdf_search(cdf, n_cdf, guide, shift, k[i]);
}
template <class Cell>
__global__ void test_path_kernel(const DevModel M, const double *in, uint32_t n, double *out, int advance_mode) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *x = in + (advance_mode ? 8 : 7) * i;
  const double *c = M.cell_params + (size_t)(uint32_t)x[0] * M.cell_nparam;
  int rt = (int)x[1];
  v3 loc = V(x[2], x[3], x[4]);
  typename Cell::Path P;
  const v3 dir = from_thph(x[5], x[6]);
  double len = Cell::path(M, c, rt, loc, dir, P);
  Travel t = Cell::advance(M, c, rt, advance_mode ? x[7] : len, loc, dir, P);
  double *o = out + 9 * i;
  o[0] = t.len; o[1] = t.time; o[2] = t.loc.x; o[3] = t.loc.y; o[4] = t.loc.z;
  if (Cell::curved) angles_of(t.dir, o[5], o[6]); else { o[5] = x[5]; o[6] = x[6]; }
  o[7] = exp(-t.aexp);
  o[8] = advance_mode ? -1.0 : (double)P.face;
}
// in[i] = {cell, type, x,y,z, theta, phi, dt}: the snapshot deposit's partial advance (advance_time) along the move to the
// boundary from that state
template <class Cell>
__global__ void test_advance_time_kernel(const DevModel M, const double *in, uint32_t n, double *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *x = in + 8 * i;
  const double *c = M.cell_params + (size_t)(uint32_t)x[0] * M.cell_nparam;
  const int rt = (int)x[1];
  const v3 loc = V(x[2], x[3], x[4]), dir = from_thph(x[5], x[6]);
  typename Cell::Path P;
  const double len = Cell::path(M, c, rt, loc, dir, P);
  const Travel seg = Cell::advance(M, c, rt, len, loc, dir, P);
  const Travel t = advance_time<Cell>(M, c, rt, x[7], loc, dir, P, seg.len, seg.time);
  double *o = out + 9 * i;
  o[0] = t.len; o[1] = t.time; o[2] = t.loc.x; o[3] = t.loc.y; o[4] = t.loc.z;
  if (Cell::curved) angles_of(t.dir, o[5], o[6]); else { o[5] = x[5]; o[6] = x[6]; }
  o[7] = exp(-t.aexp);
  o[8] = -1.0;
}
__global__ void test_transform_kernel(const double *in, uint32_t n, double *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *x = in + 6 * i;
  v3 e3 = from_thph(x[0], x[1]), s1 = s1_from_angles(x[0], x[1], x[2]);
  double st, ct, sp, cp, sr, cr;
  sincos(x[3], &st, &ct);
  sincos(x[4], &sp, &cp);
  sincos(x[5], &sr, &cr);
  transform(e3, s1, st, ct, sp, cp, sr, cr);
  angles_of(e3, out[3 * i], out[3 * i + 1]);
  out[3 * i + 2] = pol_angle_of(e3, s1);
}
__global__ void test_rtcoef_kernel(const double *in, uint32_t n, double *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *x = in + 15 * i;
  double *o = out + 13 * i;
  RTCoef rt;
  rt.init(V(x[0], x[1], x[2]), V(x[3], x[4], x[5]));
  rt.densR = x[6]; rt.velR[0] = x[7]; rt.velR[1] = x[8];
  rt.densT = x[9]; rt.velT[0] = x[10]; rt.velT[1] = x[11];
  rt.notransmit = x[13] != 0;
  rt.get_coefs((int)x[12]);
  rt.choose((uint32_t)x[14]);
  v3 od = rt.chosen_ray_dir(), pd = rt.chosen_pdom();
  for (int k = 0; k < 6; k++) o[k] = rt.prob[k];
  o[6] = rt.choice; o[7] = od.x; o[8] = od.y; o[9] = od.z; o[10] = pd.x; o[11] = pd.y; o[12] = pd.z;
}
__global__ void test_arith_kernel(const double *in, uint32_t n, double *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double a = in[2 * i], b = in[2 * i + 1];
  out[4 * i] = qdiv(a, b); out[4 * i + 1] = a / b; out[4 * i + 2] = qsqrt0(a); out[4 * i + 3] = sqrt(a);
}
__global__ void test_pathlog_kernel(const double *in, uint32_t n, double *out) {
  log_table_fill(log_table());
  __syncthreads();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double r = 1.0 - in[i] * (1.0 / 2147483648.0);
  out[2 * i] = neg_log_unit(log_table(), r); out[2 * i + 1] = -log(r);
}
__global__ void test_catch_kernel(double bin_dt, uint32_t n_bins, const double *in, uint32_t n, double *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *x = in + 28 * i;
  double *o = out + 6 * i;
  uint32_t bin = 0; double e[4] = {0, 0, 0, 0};
  int type = (int)x[25];
  const v3 dir = from_thph(x[22], x[23]);
  bool c = seis_catch(x, bin_dt, n_bins, x[18], V(x[19], x[20], x[21]), dir,
                      (type == R3D_RAY_P) ? dir : s1_from_angles(x[22], x[23], x[24]), type, x[26], x[27], bin, e);
  o[0] = c ? 1.0 : 0.0; o[1] = c ? (double)bin : -1.0; o[2] = e[0]; o[3] = e[1]; o[4] = e[2]; o[5] = e[3];
}

// ---------------------------------------------------------------------------
// host side of the handle
// ---------------------------------------------------------------------------
struct JobReq {
  unsigned long long first, n, seed;
  r3d_phonon_final *finals;
  r3d_event *events; unsigned long long *event_cursor, event_cap; uint32_t event_mask;
  const unsigned long long *replay;        // trace: the device copy of a replayed index list (first = 0, n = its length), or null
};

struct DevState {
  int device = -1;
  cudaStream_t stream = nullptr;
  DevModel M;
  uint32_t cell_kind = 0;
  std::vector<void *> allocs;
  // launch geometry of the persistent kernel
  int grid = 0, threads = 0, blocks_per_sm = 1;
  size_t smem_block = 0;                   // dynamic shared memory available to one CTA
  uint32_t table_bytes = 0;                // small-model tables staged in shared memory (0: read through L1 / L2)
  uint32_t max_slots[2] = {0, 0};          // slots per CTA that fit [plain | trace]
  unsigned long long *block_tally = nullptr;   // [grid][R3D_NCOUNTERS], one row per CTA: no atomics
  unsigned long long *block_clock = nullptr;   // [grid][R3D_NCLOCKS] (r3d_resident.cuh)
  // worker thread: launches queued jobs on this device's stream
  std::thread worker;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<JobReq> jobs;
  bool stop = false;
  bool busy = false;
  int err_code = 0;
  std::string err;
  double seconds = 0;                      // device time of the jobs finished since the last r3d_sync
  unsigned long long launches = 0;
  double k_seconds = 0;                    // device time of the propagate kernel alone since r3d_set_profiling
  unsigned long long k_launches = 0;
  cudaEvent_t ev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};    // job begin / end, kernel begin / end, 3 for the pilot launches (made once per device)
  int wide = -1;                           // layered models: 1 = the 512-thread variant of the kernel, 0 = the 384-thread one, -1 = not decided yet
  int wide_threads = 0;
  // the integer accumulators are one allocation, so that a launcher can all-reduce them with ONE collective:
  // counts [n_seis*n_bins*2] | counters [R3D_NCOUNTERS] | diag lanes [R3D_NDIAG_LANES] (lane b = 1 if bit b of the diagnostic
  // word is set: lanes survive a SUM all-reduce, the OR-combined word does not)
  unsigned long long *ibuf = nullptr;
  size_t n_ibuf = 0, n_fbuf = 0;
  const double *raw_theta = nullptr, *raw_phi = nullptr, *raw_spol = nullptr;   // the take-off angles and S->S angles as given (sources of peer copies)
  // energy snapshots (r3d_set_snapshots): Z.n_times == 0 = off.  Z's three arrays are one pool allocation, snap_mem
  SnapGrid Z{};
  void *snap_mem = nullptr;
  size_t snap_cells = 0;                   // n_times * (n_vox + 1) * 2
  // catch log (r3d_set_catch_log): G.cap == 0 = off.  The mask, the cursor and the records are one pool allocation, log_mem
  CatchLog G{};
  void *log_mem = nullptr;
};

}  // namespace

struct r3d_handle {
  std::vector<DevState *> devs;
  uint32_t cell_kind = 0, n_seis = 0, n_bins = 0;
  double ttl = 0;
  // in-process multi-device handles: the devices' accumulators are summed by a kernel on device slot 0 that reads the
  // other devices' memory over NVLink (peer access), into these staging buffers; one device-to-host copy follows
  bool peer_ok = false;
  double *sum_f64 = nullptr;
  unsigned long long *sum_i64 = nullptr;
};

namespace {

// Device memory comes from a stream-ordered pool PRIVATE to this library (one per device, made on first use and kept for
// the life of the process, release threshold = never), so that a destroy -> create cycle (one per run of the host
// program's loop) reuses the memory instead of going to the driver - and the device's default pool, which other code of
// the process may use, keeps its own settings.
constexpr int kMaxDevices = 64;
cudaMemPool_t g_pool[kMaxDevices];
bool g_pool_made[kMaxDevices];
std::mutex g_pool_mu;
int device_pool(int dev, cudaMemPool_t *out) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  if (dev < 0 || dev >= kMaxDevices) return fail(R3D_ENODEV, "device index out of range");
  if (!g_pool_made[dev]) {
    cudaMemPoolProps props;
    memset(&props, 0, sizeof props);
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    CK(cudaMemPoolCreate(&g_pool[dev], &props));
    unsigned long long keep = ~0ull;
    CK(cudaMemPoolSetAttribute(g_pool[dev], cudaMemPoolAttrReleaseThreshold, &keep));
    g_pool_made[dev] = true;
  }
  *out = g_pool[dev];
  return 0;
}
template <class T>
int dev_alloc(DevState &D, T **p, size_t count) {
  void *q = nullptr;
  cudaMemPool_t pool;
  if (int rc = device_pool(D.device, &pool)) return rc;
  CK(cudaMallocFromPoolAsync(&q, std::max<size_t>(count, 1) * sizeof(T), pool, D.stream));
  D.allocs.push_back(q);
  *p = static_cast<T *>(q);
  return 0;
}
template <class T>
int dev_upload(DevState &D, const T **p, const T *host, size_t count) {
  T *q = nullptr;
  if (int rc = dev_alloc(D, &q, count)) return rc;
  if (count) CK(cudaMemcpyAsync(q, host, count * sizeof(T), cudaMemcpyDefault, D.stream));   // host memory, or device memory of any device
  *p = q;
  return 0;
}

typedef void (*propagate_fn)(const DevModel, const Job, uint32_t, uint32_t, unsigned long long *, unsigned long long *, const SnapGrid,
                             const CatchLog, const unsigned long long *);
// snap: the plain kernel with the energy-snapshot deposits; log: the plain kernel that writes the catch log (the trace kernels
// have neither)
template <class Cell, bool SMALL>
propagate_fn pick_plain(bool snap, bool log) {
  if (log) return snap ? propagate_kernel<Cell, false, SMALL, true, true> : propagate_kernel<Cell, false, SMALL, false, true>;
  return snap ? propagate_kernel<Cell, false, SMALL, true, false> : propagate_kernel<Cell, false, SMALL, false, false>;
}
template <class Cell>
propagate_fn pick_propagate_of(bool trace, bool small, bool snap, bool log) {
  if (trace) return small ? propagate_kernel<Cell, true, true, false, false> : propagate_kernel<Cell, true, false, false, false>;
  return small ? pick_plain<Cell, true>(snap, log) : pick_plain<Cell, false>(snap, log);
}
propagate_fn pick_propagate(uint32_t kind, bool trace, bool small, bool wide = false, bool snap = false, bool log = false) {
  switch (kind) {
    case R3D_CELL_CYLINDER:
      return wide ? pick_propagate_of<CylinderWide>(trace, small, snap, log) : pick_propagate_of<Cylinder>(trace, small, snap, log);
    case R3D_CELL_SHELL: return pick_propagate_of<Shell>(trace, small, snap, log);
    default: return pick_propagate_of<Tetra>(trace, small, snap, log);
  }
}

int validate(const r3d_model_desc *d) {
  if (!d) return fail(R3D_EINVAL, "null model descriptor");
  if (!d->n_toa || !d->n_cells || !d->n_scat) return fail(R3D_EINVAL, "model needs at least one take-off angle, cell and scatterer");
  if (!d->toa_theta || !d->toa_phi || !d->src_whole_cdf || !d->src_cdf || !d->scat_mfp || !d->scat_whole_cdf ||
      !d->scat_cdf || !d->scat_spol || !d->cell_params || !d->cell_scat || !d->face_flags || !d->face_other_cell ||
      (d->n_seis && !d->seis))
    return fail(R3D_EINVAL, "null array in model descriptor");
  uint32_t np, nf;
  switch (d->cell_kind) {
    case R3D_CELL_CYLINDER: np = R3D_CYL_NPARAM; nf = R3D_CYL_NFACES; break;
    case R3D_CELL_SHELL: np = R3D_SHELL_NPARAM; nf = R3D_SHELL_NFACES; break;
    case R3D_CELL_TETRA: np = R3D_TETRA_NPARAM; nf = R3D_TETRA_NFACES; break;
    default: return fail(R3D_EINVAL, "unknown cell_kind");
  }
  if (d->cell_nparam != np || d->faces_per_cell != nf) return fail(R3D_EINVAL, "cell_nparam / faces_per_cell do not match cell_kind");
  if (d->src_cell >= d->n_cells) return fail(R3D_EINVAL, "src_cell out of range");
  if (!(d->bin_dt > 0) || !d->n_bins) return fail(R3D_EINVAL, "bin_dt and n_bins must be positive");
  if ((uint64_t)d->n_scat * 4 > 0xffffffffull) return fail(R3D_EINVAL, "too many scatterers");
  if (d->n_cells >= 0x80000000u) return fail(R3D_EINVAL, "too many cells (the slot keeps the cell index in 31 bits)");
  for (uint32_t i = 0; i < d->n_cells; i++) {
    if (d->cell_scat[i] >= d->n_scat) return fail(R3D_EINVAL, "cell_scat out of range");
    for (uint32_t f = 0; f < nf; f++)
      if ((d->face_flags[i * nf + f] & R3D_FACE_ADJOIN) && d->face_other_cell[i * nf + f] >= d->n_cells)
        return fail(R3D_EINVAL, "face_other_cell out of range");
    if (d->cell_kind == R3D_CELL_SHELL) {
      const double *c = d->cell_params + (size_t)i * np;
      if (c[0] > 0 || c[1] > 0)        // media.cpp:675 throws for inverted radial velocity profiles
        return fail(R3D_EUNSUPPORTED, "SphereShell: no handler for inverted radial velocity profiles");
    }
  }
  return 0;
}

int env_int(const char *name, int dflt);

// Uniform grid over the seismometers' bounding spheres: cell -> list of seismometers whose (slightly inflated) sphere
// box overlaps it.  A phonon looks up the cell of its position and runs the exact CatchPhonon test only on that list.
int build_seis_grid(DevState &D, const r3d_model_desc *d) {
  DevModel &M = D.M;
  const uint32_t ns = d->n_seis;
  std::vector<uint32_t> start(2, 0), items;
  for (int a = 0; a < 3; a++) { M.grid_min[a] = 0; M.grid_inv_h[a] = 0; M.grid_dim[a] = 1; }
  if (ns) {
    std::vector<double> rad(ns);
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (uint32_t i = 0; i < ns; i++) {
      const double *s = d->seis + (size_t)i * R3D_SEIS_NPARAM;
      double r = std::max(s[14], s[15]);
      rad[i] = r * (1.0 + 1e-6) + 1e-9 * (1.0 + fabs(s[0]) + fabs(s[1]) + fabs(s[2]));     // covers r_out with margin
      for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], s[a] - rad[i]); hi[a] = std::max(hi[a], s[a] + rad[i]); }
    }
    std::vector<double> sorted(rad);
    std::sort(sorted.begin(), sorted.end());
    double h = 2.0 * sorted[ns / 2];                       // a typical sphere spans about one cell
    if (!(h > 0)) h = 1.0;
    const int max_dim = std::max(1, env_int("R3D_GRID_MAX_DIM", 128));
    for (int a = 0; a < 3; a++) {
      double ext = hi[a] - lo[a];
      double ha = std::max(h, ext / max_dim);
      uint32_t dim = (uint32_t)std::max(1.0, ceil(ext / ha) + 1.0);
      M.grid_min[a] = lo[a]; M.grid_inv_h[a] = 1.0 / ha; M.grid_dim[a] = dim;
    }
    auto cell_of = [&](double x, int a) {                  // same expression as grid_axis_cell() on the device
      long c = (long)floor((x - M.grid_min[a]) * M.grid_inv_h[a]);
      return (uint32_t)std::min<long>(std::max<long>(c, 0), (long)M.grid_dim[a] - 1);
    };
    const size_t ncell = (size_t)M.grid_dim[0] * M.grid_dim[1] * M.grid_dim[2];
    start.assign(ncell + 1, 0);
    for (int pass = 0; pass < 2; pass++) {
      std::vector<uint32_t> fill;
      if (pass == 1) {
        for (size_t c = 0, run = 0; c <= ncell; c++) { uint32_t n = c < ncell ? start[c] : 0; start[c] = (uint32_t)run; run += n; }
        items.assign(start[ncell], 0);
        fill.assign(start.begin(), start.end() - 1);
      }
      for (uint32_t i = 0; i < ns; i++) {
        const double *s = d->seis + (size_t)i * R3D_SEIS_NPARAM;
        uint32_t c0[3], c1[3];
        for (int a = 0; a < 3; a++) { c0[a] = cell_of(s[a] - rad[i], a); c1[a] = cell_of(s[a] + rad[i], a); }
        for (uint32_t z = c0[2]; z <= c1[2]; z++)
          for (uint32_t y = c0[1]; y <= c1[1]; y++)
            for (uint32_t x = c0[0]; x <= c1[0]; x++) {
              size_t c = ((size_t)z * M.grid_dim[1] + y) * M.grid_dim[0] + x;
              if (pass == 0) start[c]++; else items[fill[c]++] = i;
            }
      }
    }
  }
  if (int rc = dev_upload(D, &M.grid_start, start.data(), start.size())) return rc;
  if (int rc = dev_upload(D, &M.grid_items, items.data(), items.size())) return rc;
  CK(cudaStreamSynchronize(D.stream));                      // the host vectors go out of scope
  return 0;
}

int env_int(const char *name, int dflt) {
  const char *s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

int build_device(DevState &D, const r3d_model_desc *d) {
  CK(cudaSetDevice(D.device));
  CK(cudaStreamCreateWithFlags(&D.stream, cudaStreamNonBlocking));
  for (int i = 0; i < 7; i++) CK(cudaEventCreate(&D.ev[i]));
  const bool timing = env_int("R3D_TIMING", 0) != 0;
  auto t_start = std::chrono::steady_clock::now();
  auto lap = [&](const char *what) {
    if (!timing) return;
    cudaStreamSynchronize(D.stream);
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "r3d_create: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_start).count());
    t_start = now;
  };
  D.cell_kind = d->cell_kind;
  DevModel &M = D.M;
  memset(&M, 0, sizeof M);
  M.freq_hz = d->freq_hz; M.ttl = d->ttl; M.bin_dt = d->bin_dt;
  for (int i = 0; i < 3; i++) { M.earth_center[i] = d->earth_center[i]; M.src_loc[i] = d->src_loc[i]; M.src_whole[i] = d->src_whole_cdf[i]; }
  M.min_theta = d->min_theta; M.max_theta = d->max_theta; M.slow_concern = d->slow_concern;
  M.cyl_radius2 = d->cyl_radius2; M.loop_concern = d->loop_concern;
  M.n_bins = d->n_bins; M.n_toa = d->n_toa; M.src_cell = d->src_cell; M.n_scat = d->n_scat; M.n_cells = d->n_cells; M.n_seis = d->n_seis;
  M.ecs_radial = d->ecs_radial; M.no_deflect = d->no_deflect;
  M.cell_nparam = d->cell_nparam; M.faces_per_cell = d->faces_per_cell;
  const size_t nt = d->n_toa, ns = d->n_scat, nc = d->n_cells, nf = d->faces_per_cell;

  // take-off angles, packed (theta, phi) with the Phonon constructor's theta clamp applied
  const double *th = nullptr, *ph = nullptr;
  if (int rc = dev_upload(D, &th, d->toa_theta, nt)) return rc;
  if (int rc = dev_upload(D, &ph, d->toa_phi, nt)) return rc;
  double4 *toa = nullptr;
  if (int rc = dev_alloc(D, &toa, nt)) return rc;
  pack_toa_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, D.stream>>>(th, ph, toa, (uint32_t)nt, d->min_theta, d->max_theta);
  M.toa = toa;
  D.raw_theta = th; D.raw_phi = ph;

  lap("stream, pool, toa");
  if (int rc = dev_upload(D, &M.src_cdf, d->src_cdf, 3 * nt)) return rc;
  if (int rc = dev_upload(D, &M.scat_mfp, d->scat_mfp, 2 * ns)) return rc;
  if (int rc = dev_upload(D, &M.scat_whole, d->scat_whole_cdf, 8 * ns)) return rc;
  if (int rc = dev_upload(D, &M.scat_cdf, d->scat_cdf, 4 * ns * nt)) return rc;
  {
    const double *spol_raw = nullptr;
    double2 *spol = nullptr;
    if (int rc = dev_upload(D, &spol_raw, d->scat_spol, ns * nt)) return rc;
    if (int rc = dev_alloc(D, &spol, ns * nt)) return rc;
    pack_spol_kernel<<<(unsigned)((ns * nt + 255) / 256), 256, 0, D.stream>>>(spol_raw, spol, ns * nt);
    M.scat_spol = spol;
    D.raw_spol = spol_raw;
  }
  lap("cdf tables, spol");
  {
    // The device's cell records are the caller's, followed by a few derived constants per cell (Cell::extra doubles): reciprocals
    // and products that the reference re-derives with a division in every event (1 / v, pi f / Q, |grad v|).  Computed here
    // in plain IEEE double arithmetic; the events multiply where the reference divides (within 2 ulp of it).
    const uint32_t np = d->cell_nparam;
    const uint32_t extra = (d->cell_kind == R3D_CELL_CYLINDER) ? Cylinder::extra : (d->cell_kind == R3D_CELL_SHELL) ? Shell::extra : Tetra::extra;
    std::vector<double> rec((size_t)nc * (np + extra));
    for (size_t i = 0; i < nc; i++) {
      const double *c = d->cell_params + i * np;
      double *o = rec.data() + i * (np + extra);
      memcpy(o, c, np * sizeof(double));
      double *x = o + np;
      const double pif = kPi * d->freq_hz;
      if (d->cell_kind == R3D_CELL_CYLINDER) {
        x[0] = 1.0 / c[0]; x[1] = 1.0 / c[1]; x[2] = pif / c[3]; x[3] = pif / c[4];
      } else if (d->cell_kind == R3D_CELL_SHELL) {
        x[0] = pif / c[8]; x[1] = pif / c[9];
      } else {
        x[0] = pif / c[12]; x[1] = pif / c[13];
        for (int t = 0; t < 2; t++) {
          const double g = sqrt(c[3 * t] * c[3 * t] + c[3 * t + 1] * c[3 * t + 1] + c[3 * t + 2] * c[3 * t + 2]);
          x[2 + t] = g; x[4 + t] = 1.0 / g;
        }
      }
    }
    M.cell_nparam = np + extra;
    if (int rc = dev_upload(D, &M.cell_params, rec.data(), rec.size())) return rc;
    CK(cudaStreamSynchronize(D.stream));                      // (rec goes out of scope)
  }
  if (int rc = dev_upload(D, &M.cell_scat, d->cell_scat, nc)) return rc;
  {
    // Layered (cylinder) cells have one velocity per wave type, so whether a neighbour face bends the ray or hands it
    // over unchanged (CellFace::VelocityJump > 1e-5, phonons.cpp:225-255, media_cellface.cpp:83-99) is a property of the
    // face: evaluated once here with the reference's own expression (plain IEEE double operations, no contraction
    // possible) and kept in two library-private bits of the flag byte, instead of two divisions per face crossing.
    std::vector<uint8_t> fl(d->face_flags, d->face_flags + nc * nf);
    for (uint8_t &x : fl) x &= 0x0f;          // the ABI defines four bits (include/r3d_gpu.h:58-61)
    if (d->cell_kind == R3D_CELL_CYLINDER) {
      const size_t np = d->cell_nparam;
      for (size_t i = 0; i < nc; i++) for (size_t f = 0; f < nf; f++) {
        uint8_t &x = fl[i * nf + f];
        if (!(x & R3D_FACE_ADJOIN)) continue;
        const double *c = d->cell_params + i * np, *o = d->cell_params + (size_t)d->face_other_cell[i * nf + f] * np;
        volatile double dvp = std::fabs(2 * (o[0] - c[0]) / (o[0] + c[0])), dvs = std::fabs(2 * (o[1] - c[1]) / (o[1] + c[1]));
        const double jump = (dvp > dvs) ? dvp : dvs;
        x |= R3D_FACE_JUMP_KNOWN | ((jump > 0.00001) ? R3D_FACE_JUMP : 0);
      }
    }
    if (int rc = dev_upload(D, &M.face_flags, fl.data(), nc * nf)) return rc;
  }
  if (int rc = dev_upload(D, &M.face_other, d->face_other_cell, nc * nf)) return rc;
  if (int rc = dev_upload(D, &M.seis, d->seis, (size_t)d->n_seis * R3D_SEIS_NPARAM)) return rc;
  double4 *sph = nullptr;
  if (int rc = dev_alloc(D, &sph, d->n_seis)) return rc;
  if (d->n_seis) seis_sphere_kernel<<<(d->n_seis + 127) / 128, 128, 0, D.stream>>>(M.seis, d->n_seis, sph);
  M.seis_sphere = sph;
  if (int rc = build_seis_grid(D, d)) return rc;

  lap("cells, seismometer grid");
  // guide tables: exact only for non-decreasing CDFs; otherwise fall back to the plain bisection
  int *bad = nullptr;
  if (int rc = dev_alloc(D, &bad, 1)) return rc;
  CK(cudaMemsetAsync(bad, 0, sizeof(int), D.stream));
  check_monotone_kernel<<<(unsigned)((3 * nt + 255) / 256), 256, 0, D.stream>>>(M.src_cdf, (uint32_t)nt, 3, bad);
  check_monotone_kernel<<<(unsigned)((4 * ns * nt + 255) / 256), 256, 0, D.stream>>>(M.scat_cdf, (uint32_t)nt, (uint32_t)(4 * ns), bad);
  int hbad = 0;
  CK(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, D.stream));
  CK(cudaStreamSynchronize(D.stream));
  int bits = env_int("R3D_GUIDE_BITS", -1);
  if (bits < 0) {                         // default: about one table entry per bucket (TOA degree 9: 2^23 buckets, 32 MB per table).
    bits = 0;                             // With 4 per bucket 62-97 % of the warps of the bench workload had a lane whose bucket was
    while ((1ull << bits) < nt && bits < 24) bits++;      // wider than the final read and took the narrowing round trip; now 10-45 %
  }
  if (bits > 24) bits = 24;
  if (hbad || bits == 0 || nt < 16) {
    M.guide_shift = 32; M.guide_stride = 1;
    uint32_t *g = nullptr;
    if (int rc = dev_alloc(D, &g, 1)) return rc;
    M.src_guide = g; M.scat_guide = g;
  } else {
    M.guide_shift = 31 - bits;
    M.guide_stride = (1u << bits) + 1;
    uint32_t *gs = nullptr, *gc = nullptr;
    if (int rc = dev_alloc(D, &gs, (size_t)3 * M.guide_stride)) return rc;
    if (int rc = dev_alloc(D, &gc, (size_t)4 * ns * M.guide_stride)) return rc;
    unsigned long long tot = 3ull * M.guide_stride;
    build_guide_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, D.stream>>>(M.src_cdf, (uint32_t)nt, 3, M.guide_shift, M.guide_stride, gs);
    tot = 4ull * ns * M.guide_stride;
    build_guide_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, D.stream>>>(M.scat_cdf, (uint32_t)nt, (uint32_t)(4 * ns), M.guide_shift, M.guide_stride, gc);
    M.src_guide = gs; M.scat_guide = gc;
  }

  lap("monotone check, guide tables");
  // accumulators
  const size_t nb = std::max<size_t>((size_t)d->n_seis * d->n_bins, 1);
  D.n_fbuf = nb * R3D_BIN_NF64;
  D.n_ibuf = nb * R3D_BIN_NCNT + R3D_NCOUNTERS + R3D_NDIAG_LANES;
  if (int rc = dev_alloc(D, &M.energies, D.n_fbuf)) return rc;
  if (int rc = dev_alloc(D, &D.ibuf, D.n_ibuf)) return rc;
  M.counts = D.ibuf;
  M.counters = D.ibuf + nb * R3D_BIN_NCNT;
  if (int rc = dev_alloc(D, &M.next_phonon, (size_t)1)) return rc;
  CK(cudaMemsetAsync(M.energies, 0, D.n_fbuf * sizeof(double), D.stream));
  CK(cudaMemsetAsync(D.ibuf, 0, D.n_ibuf * sizeof(unsigned long long), D.stream));

  lap("accumulators");
  // launch geometry: persistent CTAs, `blocks_per_sm` per SM, each with an equal share of the SM's shared memory
  struct { int multiProcessorCount, sharedMemPerMultiprocessor, reservedSharedMemPerBlock, sharedMemPerBlockOptin; } prop;
  CK(cudaDeviceGetAttribute(&prop.multiProcessorCount, cudaDevAttrMultiProcessorCount, D.device));   // (cudaGetDeviceProperties takes 20+ ms)
  CK(cudaDeviceGetAttribute(&prop.sharedMemPerMultiprocessor, cudaDevAttrMaxSharedMemoryPerMultiprocessor, D.device));
  CK(cudaDeviceGetAttribute(&prop.reservedSharedMemPerBlock, cudaDevAttrReservedSharedMemoryPerBlock, D.device));
  CK(cudaDeviceGetAttribute(&prop.sharedMemPerBlockOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, D.device));
  const int kind_threads = (d->cell_kind == R3D_CELL_CYLINDER) ? Cylinder::threads : (d->cell_kind == R3D_CELL_SHELL) ? Shell::threads : Tetra::threads;
  D.threads = std::min(kind_threads, std::max(32, env_int("R3D_THREADS", kind_threads) / 32 * 32));
  D.blocks_per_sm = std::max(1, env_int("R3D_BLOCKS_PER_SM", 1));
  cudaFuncAttributes fattr;
  CK(cudaFuncGetAttributes(&fattr, pick_propagate(d->cell_kind, true, true)));
  const size_t per_block = (size_t)prop.sharedMemPerMultiprocessor / D.blocks_per_sm - (size_t)prop.reservedSharedMemPerBlock - fattr.sharedSizeBytes;
  D.smem_block = std::min(per_block, (size_t)prop.sharedMemPerBlockOptin - fattr.sharedSizeBytes) / 16 * 16;
  // Leave part of the SM's 256 KB to L1: the kernel runs at 128 registers per thread and the few values it spills
  // around the inlined event bodies must hit L1 (measured on one box: 1568 slots with 28 KB of L1 1.66e9 phonons/s,
  // 1280 slots with 60 KB 1.99e9).  The carve-out steps are 132 / 164 / 196 / 228 KB.
  const size_t smem_cap = (size_t)std::max(16, env_int("R3D_SMEM_KB", 196)) * 1024 / D.blocks_per_sm - (size_t)prop.reservedSharedMemPerBlock - fattr.sharedSizeBytes;
  D.smem_block = std::min(D.smem_block, smem_cap / 16 * 16);
  const uint32_t tb = Tab<true>::bytes(d->n_cells, M.cell_nparam, d->faces_per_cell, d->n_scat);
  D.table_bytes = ((size_t)nc * M.cell_nparam * 8 + (size_t)ns * 80 <= (size_t)env_int("R3D_SMALL_TABLE_BYTES", 24 * 1024)) ? tb : 0u;
  const size_t for_slots = D.smem_block - D.table_bytes;
  D.max_slots[0] = (uint32_t)std::min<size_t>(for_slots / R3D_SLOT_BYTES / 32 * 32, 65504);
  D.max_slots[1] = (uint32_t)std::min<size_t>(for_slots / R3D_SLOT_BYTES_TRACE / 32 * 32, 65504);
  if (int cap = env_int("R3D_SLOTS_PER_BLOCK", 0)) {
    for (int t = 0; t < 2; t++) D.max_slots[t] = std::max(32u, std::min(D.max_slots[t], (uint32_t)cap / 32 * 32));
  }
  if (D.max_slots[1] < 32) return fail(R3D_EUNSUPPORTED, "shared memory too small for the phonon slots");
  for (int variant = 0; variant < 5; variant++)          // plain, trace, plain with snapshots, with the catch log, with both
    for (int wide = 0; wide < (d->cell_kind == R3D_CELL_CYLINDER ? 2 : 1); wide++)
      CK(cudaFuncSetAttribute(pick_propagate(d->cell_kind, variant == 1, D.table_bytes != 0, wide != 0, variant == 2 || variant == 4,
                                             variant >= 3),
                              cudaFuncAttributeMaxDynamicSharedMemorySize, (int)D.smem_block));
  D.wide_threads = std::min((int)CylinderWide::threads, std::max(32, env_int("R3D_THREADS", CylinderWide::threads) / 32 * 32));
  D.wide = (d->cell_kind == R3D_CELL_CYLINDER) ? env_int("R3D_CYL_WIDE", -1) : 0;      // (-1: decided by the first large job, run_job)
  if (D.wide > 1) D.wide = 1;
  D.grid = prop.multiProcessorCount * D.blocks_per_sm;
  if (int rc = dev_alloc(D, &D.block_tally, (size_t)D.grid * R3D_NCOUNTERS)) return rc;
  if (int rc = dev_alloc(D, &D.block_clock, (size_t)D.grid * R3D_NCLOCKS)) return rc;
  CK(cudaMemsetAsync(D.block_tally, 0, (size_t)D.grid * R3D_NCOUNTERS * sizeof(unsigned long long), D.stream));
  CK(cudaMemsetAsync(D.block_clock, 0, (size_t)D.grid * R3D_NCLOCKS * sizeof(unsigned long long), D.stream));

  CK(cudaStreamSynchronize(D.stream));
  CK(cudaGetLastError());
  lap("launch geometry");
  return 0;
}

// One job on one device (called on the device's worker thread): one launch of the persistent kernel - or several, for a
// job of more than kMaxPerLaunch phonons: a slot keeps its phonon's index relative to the launch's first phonon in 32 bits,
// and the per-thread tallies are 32-bit (a thread sees phonons / (CTAs x threads) of a launch, so 2^30 phonons per launch
// leave room for 2 x 10^5 loop events per phonon on average).
// Layered models have two builds of the kernel (Cylinder, CylinderWide: r3d_device.cuh).  The first job of at least
// kPilotMin phonons starts with two pilot launches of kPilot phonons each, one per build, timed with CUDA events; the
// faster build then runs the rest of the job and everything after it on this handle.  The pilots are part of the job (their
// phonons are traced once, like all others; results do not depend on the build), so the choice costs no extra work.
constexpr unsigned long long kMaxPerLaunch = 1ull << 30;
constexpr unsigned long long kPilot = 2000000ull, kPilotMin = 8000000ull;
int run_job(DevState &D, const JobReq &jr) {
  CK(cudaSetDevice(D.device));
  cudaEvent_t ev0 = D.ev[0], ev1 = D.ev[1], ek0 = D.ev[2], ek1 = D.ev[3];
  CK(cudaEventRecord(ev0, D.stream));
  const bool trace = jr.finals != nullptr || jr.events != nullptr;
  const bool snap = !trace && D.Z.n_times > 0;        // (also the pilot launches: they trace part of the job)
  const bool log = !trace && D.G.cap > 0;             // (likewise)
  unsigned long long n_launch = 0;
  auto launch = [&](unsigned long long done, unsigned long long n, bool wide) -> int {
    Job J; J.first = jr.first + done; J.n = n; J.seed = jr.seed; J.finals = jr.finals ? jr.finals + done : nullptr;
    J.events = jr.events; J.event_cursor = jr.event_cursor; J.event_cap = jr.event_cap; J.event_mask = jr.event_mask;
    const unsigned long long *replay = jr.replay ? jr.replay + done : nullptr;      // (relative index i of this launch = list entry done + i)
    // no more slots than phonons: a small job is spread over all CTAs instead of filling the first few
    uint32_t S = D.max_slots[trace ? 1 : 0];
    const unsigned long long share = (n + (unsigned long long)D.grid - 1) / (unsigned long long)D.grid;
    if (share < S) S = (uint32_t)((share + 31ull) / 32ull * 32ull);
    const size_t smem = (size_t)S * (trace ? R3D_SLOT_BYTES_TRACE : R3D_SLOT_BYTES) + D.table_bytes;
    const unsigned long long need = (n + S - 1) / S;
    const int grid = (int)std::min<unsigned long long>((unsigned long long)D.grid, need);
    CK(cudaMemsetAsync(D.M.next_phonon, 0, sizeof(unsigned long long), D.stream));
    if (!n_launch) CK(cudaEventRecord(ek0, D.stream));
    pick_propagate(D.cell_kind, trace, D.table_bytes != 0, wide, snap, log)<<<grid, wide ? D.wide_threads : D.threads, smem, D.stream>>>(
        D.M, J, S, D.table_bytes, D.block_tally, D.block_clock, D.Z, D.G, replay);
    D.launches += 1;
    n_launch++;
    return 0;
  };
  unsigned long long done = 0;
  if (D.wide < 0 && !trace && jr.n >= kPilotMin) {
    CK(cudaEventRecord(D.ev[4], D.stream));
    if (int rc = launch(0, kPilot, false)) return rc;
    CK(cudaEventRecord(D.ev[5], D.stream));
    if (int rc = launch(kPilot, kPilot, true)) return rc;
    CK(cudaEventRecord(D.ev[6], D.stream));
    CK(cudaEventSynchronize(D.ev[6]));
    float narrow_ms = 0, wide_ms = 0;
    CK(cudaEventElapsedTime(&narrow_ms, D.ev[4], D.ev[5]));
    CK(cudaEventElapsedTime(&wide_ms, D.ev[5], D.ev[6]));
    D.wide = wide_ms < narrow_ms ? 1 : 0;
    if (env_int("R3D_TIMING", 0)) fprintf(stderr, "r3d_run: pilot launches of %llu phonons: 384 threads %.3f ms, 512 threads %.3f ms\n", kPilot, narrow_ms, wide_ms);
    done = 2 * kPilot;
  }
  const bool wide = D.wide > 0;
  while (done < jr.n) {
    const unsigned long long n = std::min(jr.n - done, kMaxPerLaunch);
    if (int rc = launch(done, n, wide)) return rc;
    done += n;
  }
  if (n_launch) CK(cudaEventRecord(ek1, D.stream));
  reduce_tally_kernel<<<R3D_NCOUNTERS, 256, 0, D.stream>>>(D.block_tally, (uint32_t)D.grid, D.M.counters);
  D.launches += 1;
  CK(cudaEventRecord(ev1, D.stream));
  CK(cudaStreamSynchronize(D.stream));
  CK(cudaGetLastError());
  float ms = 0, kms = 0;
  CK(cudaEventElapsedTime(&ms, ev0, ev1));
  if (n_launch) CK(cudaEventElapsedTime(&kms, ek0, ek1));
  {
    std::lock_guard<std::mutex> lk(D.mu);
    D.seconds += ms * 1e-3;
    if (n_launch) { D.k_seconds += kms * 1e-3; D.k_launches += n_launch; }
  }
  return 0;
}

void worker_main(DevState *D) {
  for (;;) {
    JobReq jr;
    {
      std::unique_lock<std::mutex> lk(D->mu);
      D->cv.wait(lk, [&] { return D->stop || !D->jobs.empty(); });
      if (D->jobs.empty()) return;          // stop requested and nothing left to do
      jr = D->jobs.front();
      D->jobs.pop_front();
      D->busy = true;
    }
    int rc = 0;
    {
      bool skip;
      { std::lock_guard<std::mutex> lk(D->mu); skip = D->err_code != 0; }
      if (!skip) rc = run_job(*D, jr);
    }
    {
      std::lock_guard<std::mutex> lk(D->mu);
      if (rc && !D->err_code) { D->err_code = rc; D->err = g_err; }
      D->busy = false;
    }
    D->cv.notify_all();
  }
}

void enqueue(DevState &D, const JobReq &jr) {
  { std::lock_guard<std::mutex> lk(D.mu); D.jobs.push_back(jr); }
  D.cv.notify_all();
}

// wait until the device has drained its job queue; returns its first error, if any
int drain(DevState &D) {
  std::unique_lock<std::mutex> lk(D.mu);
  D.cv.wait(lk, [&] { return D.jobs.empty() && !D.busy; });
  if (D.err_code) {
    int rc = D.err_code;
    g_err = D.err;
    D.err_code = 0; D.err.clear();
    return rc;
  }
  return 0;
}

void destroy_device(DevState *D) {
  if (!D) return;
  if (D->worker.joinable()) {
    { std::lock_guard<std::mutex> lk(D->mu); D->stop = true; }
    D->cv.notify_all();
    D->worker.join();
  }
  if (D->device >= 0) {
    cudaSetDevice(D->device);
    if (D->stream) cudaStreamSynchronize(D->stream);
    for (void *p : D->allocs) cudaFreeAsync(p, D->stream);
    if (D->snap_mem) cudaFreeAsync(D->snap_mem, D->stream);
    if (D->log_mem) cudaFreeAsync(D->log_mem, D->stream);
    if (D->stream) cudaStreamSynchronize(D->stream);
    for (int i = 0; i < 7; i++) if (D->ev[i]) cudaEventDestroy(D->ev[i]);
    if (D->stream) cudaStreamDestroy(D->stream);
  }
  delete D;
}

// The device copy of a list of phonon indices to replay, on the device's stream; freed (stream-ordered) on scope exit.
struct ReplayList {
  DevState *D = nullptr;
  unsigned long long *p = nullptr;
  int upload(DevState &dev, const uint64_t *idx, uint64_t n) {
    D = &dev;
    cudaMemPool_t pool;
    if (int rc = device_pool(D->device, &pool)) return rc;
    CK(cudaMallocFromPoolAsync(reinterpret_cast<void **>(&p), n * sizeof(unsigned long long), pool, D->stream));
    CK(cudaMemcpyAsync(p, idx, n * sizeof(unsigned long long), cudaMemcpyHostToDevice, D->stream));
    return 0;
  }
  ~ReplayList() { if (p) { cudaFreeAsync(p, D->stream); cudaStreamSynchronize(D->stream); } }
};

int check_indices(const uint64_t *idx, uint64_t n) {
  if (!idx) return fail(R3D_EINVAL, "null index list");
  for (uint64_t i = 1; i < n; i++)
    if (!(idx[i] > idx[i - 1])) return fail(R3D_EINVAL, "replayed phonon indices must be strictly increasing");
  return 0;
}

// r3d_trace / r3d_trace_indices: phonons [first, first + n), or (idx != null) the n listed ones
int trace_finals(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, const uint64_t *idx, uint64_t seed, r3d_phonon_final *out) {
  DevState &D = *h->devs[0];
  if (int rc = drain(D)) return rc;
  CK(cudaSetDevice(D.device));
  ReplayList list;
  if (idx) { if (int rc = list.upload(D, idx, n_phonons)) return rc; }
  r3d_phonon_final *dfin = nullptr;
  CK(cudaMalloc(&dfin, n_phonons * sizeof(r3d_phonon_final)));
  JobReq jr{}; jr.first = first_phonon; jr.n = n_phonons; jr.seed = seed; jr.finals = dfin; jr.replay = list.p;
  enqueue(D, jr);
  int rc = drain(D);
  cudaError_t e = cudaSuccess;
  if (!rc) e = cudaMemcpy(out, dfin, n_phonons * sizeof(r3d_phonon_final), cudaMemcpyDeviceToHost);
  cudaFree(dfin);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(R3D_ECUDA, std::string("r3d_trace: ") + cudaGetErrorString(e));
  return 0;
}

// r3d_trace_events / r3d_trace_events_indices
int trace_events(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, const uint64_t *idx, uint64_t seed, uint32_t kinds_mask,
                 r3d_event *out, uint64_t capacity, uint64_t *n_events) {
  DevState &D = *h->devs[0];
  if (int rc = drain(D)) return rc;
  CK(cudaSetDevice(D.device));
  ReplayList list;
  if (idx) { if (int rc = list.upload(D, idx, n_phonons)) return rc; }
  r3d_event *dev = nullptr;
  unsigned long long *cursor = nullptr;
  CK(cudaMalloc(&dev, std::max<uint64_t>(capacity, 1) * sizeof(r3d_event)));
  cudaError_t e = cudaMalloc(&cursor, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(cursor, 0, sizeof(unsigned long long));
  if (e != cudaSuccess) { cudaFree(dev); cudaFree(cursor); return fail(R3D_ECUDA, std::string("r3d_trace_events: ") + cudaGetErrorString(e)); }
  JobReq jr{}; jr.first = first_phonon; jr.n = n_phonons; jr.seed = seed; jr.replay = list.p;
  jr.events = dev; jr.event_cursor = cursor; jr.event_cap = capacity; jr.event_mask = kinds_mask;
  enqueue(D, jr);
  int rc = drain(D);
  unsigned long long total = 0;
  if (!rc) e = cudaMemcpy(&total, cursor, sizeof total, cudaMemcpyDeviceToHost);
  const uint64_t got = std::min<uint64_t>(total, capacity);
  if (!rc && e == cudaSuccess && got) e = cudaMemcpy(out, dev, got * sizeof(r3d_event), cudaMemcpyDeviceToHost);
  cudaFree(dev); cudaFree(cursor);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(R3D_ECUDA, std::string("r3d_trace_events: ") + cudaGetErrorString(e));
  std::sort(out, out + got, [](const r3d_event &a, const r3d_event &b) { return a.phonon != b.phonon ? a.phonon < b.phonon : a.seq < b.seq; });
  *n_events = total;
  return 0;
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

const char *r3d_last_error(void) { return g_err.c_str(); }
int r3d_abi_version(void) { return R3D_ABI_VERSION; }

int r3d_create(const r3d_model_desc *desc, const int *devices, int n_dev, r3d_handle **out) {
  DeviceGuard guard;
  if (!out) return fail(R3D_EINVAL, "null output handle");
  *out = nullptr;
  if (int rc = validate(desc)) return rc;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(R3D_ENODEV, std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
  if (n_dev <= 0) return fail(R3D_EINVAL, "n_dev must be >= 1");
  r3d_handle *h = new r3d_handle();
  h->cell_kind = desc->cell_kind; h->n_seis = desc->n_seis; h->n_bins = desc->n_bins; h->ttl = desc->ttl;
  auto bail = [&](int rc) { std::string keep = g_err; r3d_destroy(h); g_err = keep; return rc; };
  // Several devices: the host arrays cross PCIe ONCE, to device slot 0; the other devices copy the large tables from
  // slot 0's memory (NVLink when the devices are peers, else staged by the driver) and derive their own packed tables
  // and guides.  Peer access in both directions between slot 0 and every other slot also serves r3d_fetch's sum.
  r3d_model_desc from0 = *desc;
  bool peers = n_dev > 1 && n_dev <= R3D_MAX_PEERS && env_int("R3D_PEER_COMBINE", 1) != 0;
  const bool replicate = n_dev > 1 && env_int("R3D_PEER_REPLICATE", 1) != 0;
  for (int i = 0; i < n_dev; i++) {
    int dev = devices ? devices[i] : i;
    if (dev < 0 || dev >= count) { r3d_destroy(h); return fail(R3D_ENODEV, "device index out of range"); }
    for (int j = 0; j < i; j++) if (h->devs[j]->device == dev) { r3d_destroy(h); return fail(R3D_EINVAL, "device listed twice"); }
    DevState *D = new DevState();
    h->devs.push_back(D);
    D->device = dev;
    bool linked = false;                      // this device and slot 0 can read each other's pool memory
    if (i > 0 && (peers || replicate)) {
      const int d0 = h->devs[0]->device;
      int a = 0, b = 0;
      if (cudaDeviceCanAccessPeer(&a, d0, dev) == cudaSuccess && cudaDeviceCanAccessPeer(&b, dev, d0) == cudaSuccess && a && b) {
        cudaMemPool_t p0, pi;
        if (int rc = device_pool(d0, &p0)) return bail(rc);
        if (int rc = device_pool(dev, &pi)) return bail(rc);
        cudaMemAccessDesc acc;
        memset(&acc, 0, sizeof acc);
        acc.flags = cudaMemAccessFlagsProtReadWrite;
        acc.location.type = cudaMemLocationTypeDevice;
        acc.location.id = d0;
        const bool ok1 = cudaMemPoolSetAccess(pi, &acc, 1) == cudaSuccess;      // slot 0 reads this device's accumulators
        acc.location.id = dev;
        const bool ok2 = cudaMemPoolSetAccess(p0, &acc, 1) == cudaSuccess;      // this device reads slot 0's tables
        linked = ok1 && ok2;
      }
      cudaGetLastError();
      if (!linked) peers = false;
    }
    if (int rc = build_device(*D, (i > 0 && linked && replicate) ? &from0 : desc)) return bail(rc);
    if (i == 0 && replicate) {
      from0.toa_theta = D->raw_theta; from0.toa_phi = D->raw_phi; from0.src_cdf = D->M.src_cdf;
      from0.scat_cdf = D->M.scat_cdf; from0.scat_spol = D->raw_spol;
    }
    D->worker = std::thread(worker_main, D);
  }
  if (peers) {
    DevState &D0 = *h->devs[0];
    if (cudaSetDevice(D0.device) != cudaSuccess) return bail(fail(R3D_ECUDA, "cudaSetDevice"));
    if (int rc = dev_alloc(D0, &h->sum_f64, D0.n_fbuf)) return bail(rc);
    if (int rc = dev_alloc(D0, &h->sum_i64, D0.n_ibuf)) return bail(rc);
    h->peer_ok = true;
  }
  *out = h;
  return 0;
}

void r3d_destroy(r3d_handle *h) {
  DeviceGuard guard;
  if (!h) return;
  for (DevState *D : h->devs) destroy_device(D);
  delete h;
}

int r3d_run(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, uint64_t seed) {
  if (!h) return fail(R3D_EINVAL, "null handle");
  const uint64_t G = h->devs.size();
  for (uint64_t g = 0; g < G; g++) {      // contiguous index ranges (SURVEY 8e)
    uint64_t lo = n_phonons / G * g + (n_phonons % G) * g / G;
    uint64_t hi = n_phonons / G * (g + 1) + (n_phonons % G) * (g + 1) / G;
    JobReq jr{}; jr.first = first_phonon + lo; jr.n = hi - lo; jr.seed = seed;
    enqueue(*h->devs[g], jr);
  }
  return 0;
}

int r3d_sync(r3d_handle *h, double *device_seconds) {
  if (!h) return fail(R3D_EINVAL, "null handle");
  double worst = 0;
  int rc = 0;
  for (DevState *D : h->devs) {
    int r = drain(*D);
    if (r && !rc) rc = r;
    std::lock_guard<std::mutex> lk(D->mu);
    worst = std::max(worst, D->seconds);
    D->seconds = 0;
  }
  if (device_seconds) *device_seconds = worst;
  return rc;
}

int r3d_fetch(r3d_handle *h, double *energies, uint64_t *counts, uint64_t *counters, uint32_t *diag) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  const size_t nb = (size_t)h->n_seis * h->n_bins;
  unsigned long long k[R3D_NCOUNTERS], ksum[R3D_NCOUNTERS] = {0};
  if (h->devs.empty()) {
    if (energies) memset(energies, 0, nb * R3D_BIN_NF64 * sizeof(double));
    if (counts) memset(counts, 0, nb * R3D_BIN_NCNT * sizeof(uint64_t));
  }
  for (DevState *D : h->devs) {
    if (int rc = drain(*D)) return rc;
    CK(cudaSetDevice(D->device));
    CK(cudaStreamSynchronize(D->stream));
  }
  if (h->devs.size() > 1 && h->peer_ok) {
    // the sum over devices, on device slot 0 over peer memory; then ONE device-to-host copy of each array
    DevState &D0 = *h->devs[0];
    CK(cudaSetDevice(D0.device));
    PeerPtrs pf, pi;
    pf.n = pi.n = (int)h->devs.size();
    for (int g = 0; g < pf.n; g++) { pf.p[g] = h->devs[g]->M.energies; pi.p[g] = h->devs[g]->ibuf; }
    const size_t or_index = D0.n_ibuf - R3D_NDIAG_LANES - R3D_NCOUNTERS + R3D_CNT_DIAG;
    if (energies && nb) combine_f64_kernel<<<296, 256, 0, D0.stream>>>(pf, D0.n_fbuf, h->sum_f64);
    combine_u64_kernel<<<296, 256, 0, D0.stream>>>(pi, D0.n_ibuf, or_index, h->sum_i64);
    D0.launches += (energies && nb) ? 2 : 1;
    CK(cudaGetLastError());
    if (energies && nb) CK(cudaMemcpyAsync(energies, h->sum_f64, nb * R3D_BIN_NF64 * sizeof(double), cudaMemcpyDeviceToHost, D0.stream));
    if (counts && nb) CK(cudaMemcpyAsync(counts, h->sum_i64, nb * R3D_BIN_NCNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, D0.stream));
    CK(cudaMemcpyAsync(ksum, h->sum_i64 + (D0.n_ibuf - R3D_NDIAG_LANES - R3D_NCOUNTERS), sizeof ksum, cudaMemcpyDeviceToHost, D0.stream));
    CK(cudaStreamSynchronize(D0.stream));
  } else {
    // one device (or devices that are not peers: summed on the host, device by device)
    std::vector<double> e;
    std::vector<unsigned long long> c;
    for (size_t g = 0; g < h->devs.size(); g++) {
      DevState &D = *h->devs[g];
      CK(cudaSetDevice(D.device));
      if (energies && nb) {
        if (g == 0) CK(cudaMemcpyAsync(energies, D.M.energies, nb * R3D_BIN_NF64 * sizeof(double), cudaMemcpyDeviceToHost, D.stream));
        else {
          e.resize(nb * R3D_BIN_NF64);
          CK(cudaMemcpy(e.data(), D.M.energies, e.size() * sizeof(double), cudaMemcpyDeviceToHost));
          for (size_t i = 0; i < e.size(); i++) energies[i] += e[i];
        }
      }
      if (counts && nb) {
        if (g == 0) CK(cudaMemcpyAsync(counts, D.M.counts, nb * R3D_BIN_NCNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, D.stream));
        else {
          c.resize(nb * R3D_BIN_NCNT);
          CK(cudaMemcpy(c.data(), D.M.counts, c.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost));
          for (size_t i = 0; i < c.size(); i++) counts[i] += c[i];
        }
      }
      CK(cudaMemcpyAsync(k, D.M.counters, sizeof k, cudaMemcpyDeviceToHost, D.stream));
      CK(cudaStreamSynchronize(D.stream));
      for (int i = 0; i < R3D_NCOUNTERS; i++) { if (i == R3D_CNT_DIAG) ksum[i] |= k[i]; else ksum[i] += k[i]; }
    }
  }
  if (counters) for (int i = 0; i < R3D_NCOUNTERS; i++) counters[i] = ksum[i];
  if (diag) *diag = (uint32_t)ksum[R3D_CNT_DIAG];
  return 0;
}

int r3d_reset(r3d_handle *h) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  for (DevState *Dp : h->devs) {
    DevState &D = *Dp;
    if (int rc = drain(D)) return rc;
    CK(cudaSetDevice(D.device));
    CK(cudaMemsetAsync(D.M.energies, 0, D.n_fbuf * sizeof(double), D.stream));
    CK(cudaMemsetAsync(D.ibuf, 0, D.n_ibuf * sizeof(unsigned long long), D.stream));
    CK(cudaMemsetAsync(D.block_tally, 0, (size_t)D.grid * R3D_NCOUNTERS * sizeof(unsigned long long), D.stream));
    if (D.snap_mem) {
      CK(cudaMemsetAsync(D.Z.energy, 0, D.snap_cells * sizeof(double), D.stream));
      CK(cudaMemsetAsync(D.Z.count, 0, D.snap_cells * sizeof(unsigned long long), D.stream));
    }
    if (D.log_mem) CK(cudaMemsetAsync(D.G.cursor, 0, sizeof(unsigned long long), D.stream));      // (records past the cursor are never read)
    CK(cudaStreamSynchronize(D.stream));
  }
  return 0;
}

int r3d_set_snapshots(r3d_handle *h, const r3d_snapshot_desc *s) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  const bool on = s && s->n_times;
  uint64_t n_vox = 1;
  if (on) {
    if (s->n_times > R3D_SNAP_MAX_TIMES) return fail(R3D_EINVAL, "more than R3D_SNAP_MAX_TIMES snapshot times");
    if (!s->times) return fail(R3D_EINVAL, "null snapshot times");
    for (uint32_t k = 0; k < s->n_times; k++) {
      const double t = s->times[k];
      if (!std::isfinite(t) || t < 0 || t > h->ttl) return fail(R3D_EINVAL, "snapshot times must be finite and within [0, ttl]");
      if (k && !(t > s->times[k - 1])) return fail(R3D_EINVAL, "snapshot times must be increasing");
    }
    for (int a = 0; a < 3; a++) {
      if (!std::isfinite(s->origin[a])) return fail(R3D_EINVAL, "snapshot grid origin must be finite");
      if (!std::isfinite(s->voxel[a]) || !(s->voxel[a] > 0)) return fail(R3D_EINVAL, "snapshot voxel sizes must be finite and positive");
      if (!s->dims[a]) return fail(R3D_EINVAL, "snapshot grid dimensions must be at least 1");
      n_vox *= s->dims[a];
      if (n_vox > R3D_SNAP_MAX_CELLS) return fail(R3D_EINVAL, "snapshot grid exceeds R3D_SNAP_MAX_CELLS");
    }
    if ((uint64_t)s->n_times * (n_vox + 1) * 2 > R3D_SNAP_MAX_CELLS) return fail(R3D_EINVAL, "snapshot grid exceeds R3D_SNAP_MAX_CELLS");
  }
  for (DevState *Dp : h->devs) {
    DevState &D = *Dp;
    if (int rc = drain(D)) return rc;
    CK(cudaSetDevice(D.device));
    CK(cudaStreamSynchronize(D.stream));
    if (D.snap_mem) CK(cudaFreeAsync(D.snap_mem, D.stream));
    D.snap_mem = nullptr; D.snap_cells = 0;
    D.Z = SnapGrid{};
    if (!on) continue;
    const size_t cells = (size_t)s->n_times * (n_vox + 1) * 2;
    cudaMemPool_t pool;
    if (int rc = device_pool(D.device, &pool)) return rc;
    CK(cudaMallocFromPoolAsync(&D.snap_mem, cells * (sizeof(double) + sizeof(unsigned long long)) + R3D_SNAP_MAX_TIMES * sizeof(double),
                               pool, D.stream));
    double *t = static_cast<double *>(D.snap_mem);
    D.Z.times = t;
    D.Z.energy = t + R3D_SNAP_MAX_TIMES;
    D.Z.count = reinterpret_cast<unsigned long long *>(D.Z.energy + cells);
    CK(cudaMemcpyAsync(t, s->times, s->n_times * sizeof(double), cudaMemcpyHostToDevice, D.stream));
    CK(cudaMemsetAsync(D.Z.energy, 0, cells * (sizeof(double) + sizeof(unsigned long long)), D.stream));
    for (int a = 0; a < 3; a++) { D.Z.origin[a] = s->origin[a]; D.Z.voxel[a] = s->voxel[a]; D.Z.dims[a] = s->dims[a]; }
    D.Z.n_vox = (uint32_t)n_vox;
    D.Z.n_times = s->n_times;
    D.snap_cells = cells;
    CK(cudaStreamSynchronize(D.stream));                     // (s->times is borrowed)
  }
  return 0;
}

int r3d_fetch_snapshots(r3d_handle *h, double *energy, uint64_t *count, double *outside_energy, uint64_t *outside_count) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  if (h->devs.empty() || !h->devs[0]->snap_mem) return fail(R3D_EINVAL, "snapshots are off (r3d_set_snapshots)");
  const size_t cells = h->devs[0]->snap_cells, K = h->devs[0]->Z.n_times, nv = h->devs[0]->Z.n_vox;
  // the sum over the handle's devices, on the host in device order
  std::vector<double> e(cells, 0.0), eg(cells);
  std::vector<unsigned long long> c(cells, 0), cg(cells);
  for (DevState *Dp : h->devs) {
    DevState &D = *Dp;
    if (int rc = drain(D)) return rc;
    CK(cudaSetDevice(D.device));
    CK(cudaMemcpyAsync(eg.data(), D.Z.energy, cells * sizeof(double), cudaMemcpyDeviceToHost, D.stream));
    CK(cudaMemcpyAsync(cg.data(), D.Z.count, cells * sizeof(unsigned long long), cudaMemcpyDeviceToHost, D.stream));
    CK(cudaStreamSynchronize(D.stream));
    for (size_t i = 0; i < cells; i++) { e[i] += eg[i]; c[i] += cg[i]; }
  }
  for (size_t k = 0; k < K; k++) {
    const size_t at = k * (nv + 1) * 2;
    if (energy) memcpy(energy + k * nv * 2, e.data() + at, nv * 2 * sizeof(double));
    if (count) memcpy(count + k * nv * 2, c.data() + at, nv * 2 * sizeof(uint64_t));
    if (outside_energy) { outside_energy[2 * k] = e[at + nv * 2]; outside_energy[2 * k + 1] = e[at + nv * 2 + 1]; }
    if (outside_count) { outside_count[2 * k] = c[at + nv * 2]; outside_count[2 * k + 1] = c[at + nv * 2 + 1]; }
  }
  return 0;
}

int r3d_device_accumulators(r3d_handle *h, int dev_slot, void **energies, void **counts, void **counters) {
  if (!h || dev_slot < 0 || dev_slot >= (int)h->devs.size()) return fail(R3D_EINVAL, "bad handle or device slot");
  if (energies) *energies = h->devs[dev_slot]->M.energies;
  if (counts) *counts = h->devs[dev_slot]->M.counts;
  if (counters) *counters = h->devs[dev_slot]->M.counters;
  return 0;
}

int r3d_device_accumulator_blocks(r3d_handle *h, int dev_slot, void **f64_block, uint64_t *n_f64, void **i64_block,
                                  uint64_t *n_i64, uint64_t *counters_at) {
  if (!h || dev_slot < 0 || dev_slot >= (int)h->devs.size()) return fail(R3D_EINVAL, "bad handle or device slot");
  DevState &D = *h->devs[dev_slot];
  if (f64_block) *f64_block = D.M.energies;
  if (n_f64) *n_f64 = D.n_fbuf;
  if (i64_block) *i64_block = D.ibuf;
  if (n_i64) *n_i64 = D.n_ibuf;
  if (counters_at) *counters_at = D.n_ibuf - R3D_NDIAG_LANES - R3D_NCOUNTERS;
  return 0;
}

int r3d_stream(r3d_handle *h, int dev_slot, void **stream) {
  if (!h || dev_slot < 0 || dev_slot >= (int)h->devs.size() || !stream) return fail(R3D_EINVAL, "bad handle or device slot");
  *stream = h->devs[dev_slot]->stream;
  return 0;
}

int r3d_launch_count(r3d_handle *h, uint64_t *n) {
  if (!h || !n) return fail(R3D_EINVAL, "null argument");
  uint64_t tot = 0;
  for (DevState *D : h->devs) { if (int rc = drain(*D)) return rc; tot += D->launches; }
  *n = tot;
  return 0;
}

int r3d_set_profiling(r3d_handle *h, int on) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  (void)on;                                 // the kernel is always timed; this call resets the totals
  for (DevState *D : h->devs) {
    if (int rc = drain(*D)) return rc;
    CK(cudaSetDevice(D->device));
    CK(cudaMemsetAsync(D->block_clock, 0, (size_t)D->grid * R3D_NCLOCKS * sizeof(unsigned long long), D->stream));
    CK(cudaStreamSynchronize(D->stream));
    std::lock_guard<std::mutex> lk(D->mu);
    D->k_seconds = 0; D->k_launches = 0;
  }
  return 0;
}

int r3d_kernel_times(r3d_handle *h, double seconds[3], uint64_t launches[3], uint64_t units[3]) {
  DeviceGuard guard;
  if (!h || !seconds || !launches || !units) return fail(R3D_EINVAL, "null argument");
  DevState &D = *h->devs[0];
  if (int rc = drain(D)) return rc;
  unsigned long long k[R3D_NCOUNTERS];
  CK(cudaSetDevice(D.device));
  CK(cudaMemcpy(k, D.M.counters, sizeof k, cudaMemcpyDeviceToHost));
  std::vector<unsigned long long> clk((size_t)D.grid * R3D_NCLOCKS);
  CK(cudaMemcpy(clk.data(), D.block_clock, clk.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  unsigned long long c1 = 0, c2 = 0, it = 0;
  for (int b = 0; b < D.grid; b++) { c1 += clk[R3D_NCLOCKS * b]; c2 += clk[R3D_NCLOCKS * b + 1]; it = std::max(it, clk[R3D_NCLOCKS * b + 2]); }
  if (env_int("R3D_TIMING", 0)) {          // warp-cycles by kind of chunk, summed over CTAs
    unsigned long long k[R3D_NCLOCKS] = {0};
    for (int b = 0; b < D.grid; b++) for (int i = 0; i < R3D_NCLOCKS; i++) k[i] += clk[R3D_NCLOCKS * b + i];
    const char *nm[4] = {"advance", "bend", "face", "draw"};
    double tot = (double)k[11];
    for (int i = 0; i < 4; i++) tot += (double)k[3 + i];
    for (int i = 0; i < 4; i++)
      fprintf(stderr, "r3d chunks: %-8s %10llu chunks, %8.0f cycles each, %5.1f %% of warp time\n", nm[i], k[7 + i],
              k[7 + i] ? (double)k[3 + i] / (double)k[7 + i] : 0.0, 100.0 * (double)k[3 + i] / tot);
    fprintf(stderr, "r3d chunks: face_collect %8.0f cycles per face chunk, %5.1f %% of face-chunk time (the rest: face_one)\n",
            k[9] ? (double)k[12] / (double)k[9] : 0.0, k[5] ? 100.0 * (double)k[12] / (double)k[5] : 0.0);
    fprintf(stderr, "r3d chunks: waiting at barriers / for work: %5.1f %% of warp time; phase 1 %.0f, phase 2 %.0f cycles per iteration\n",
            100.0 * (double)k[11] / tot, (double)c1 / (double)std::max(1ull, k[2]), (double)c2 / (double)std::max(1ull, k[2]));
  }
  std::lock_guard<std::mutex> lk(D.mu);
  const double tot = (double)(c1 + c2);
  seconds[0] = D.k_seconds;                                   // the propagate kernel, CUDA events on its stream
  seconds[1] = tot > 0 ? D.k_seconds * (double)c1 / tot : 0;  // of which phase 1 (advance + refill), CTA-averaged
  seconds[2] = tot > 0 ? D.k_seconds * (double)c2 / tot : 0;  // of which phase 2 (table draws + face events)
  launches[0] = D.k_launches; launches[1] = it; launches[2] = (uint64_t)D.grid;
  units[0] = k[R3D_CNT_EVENTS];
  units[1] = k[R3D_CNT_SCATTERS] + k[R3D_CNT_PHONONS];                      // table draws = scatter draws + source draws
  units[2] = k[R3D_CNT_CATCHES];
  return 0;
}

int r3d_trace(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, uint64_t seed, r3d_phonon_final *out) {
  DeviceGuard guard;
  if (!h || !out) return fail(R3D_EINVAL, "null argument");
  if (!n_phonons) return 0;
  return trace_finals(h, first_phonon, n_phonons, nullptr, seed, out);
}

int r3d_trace_events(r3d_handle *h, uint64_t first_phonon, uint64_t n_phonons, uint64_t seed, uint32_t kinds_mask,
                     r3d_event *out, uint64_t capacity, uint64_t *n_events) {
  DeviceGuard guard;
  if (!h || !n_events || (capacity && !out)) return fail(R3D_EINVAL, "null argument");
  *n_events = 0;
  if (!n_phonons) return 0;
  return trace_events(h, first_phonon, n_phonons, nullptr, seed, kinds_mask, out, capacity, n_events);
}

int r3d_trace_indices(r3d_handle *h, const uint64_t *indices, uint64_t n, uint64_t seed, r3d_phonon_final *out) {
  DeviceGuard guard;
  if (!h || (n && !out)) return fail(R3D_EINVAL, "null argument");
  if (!n) return 0;
  if (int rc = check_indices(indices, n)) return rc;
  return trace_finals(h, 0, n, indices, seed, out);
}

int r3d_trace_events_indices(r3d_handle *h, const uint64_t *indices, uint64_t n, uint64_t seed, uint32_t kinds_mask,
                             r3d_event *out, uint64_t capacity, uint64_t *n_events) {
  DeviceGuard guard;
  if (!h || !n_events || (capacity && !out)) return fail(R3D_EINVAL, "null argument");
  *n_events = 0;
  if (!n) return 0;
  if (int rc = check_indices(indices, n)) return rc;
  return trace_events(h, 0, n, indices, seed, kinds_mask, out, capacity, n_events);
}

int r3d_set_catch_log(r3d_handle *h, const r3d_catch_log_desc *d) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  const size_t words = std::max<size_t>(1, ((size_t)h->n_seis + 31) / 32);
  std::vector<uint32_t> mask(words, 0u);
  if (d) {
    if (d->n_seis && !d->seis) return fail(R3D_EINVAL, "null seismometer list");
    for (uint32_t i = 0; i < (d->n_seis ? d->n_seis : h->n_seis); i++) {
      const uint32_t k = d->n_seis ? d->seis[i] : i;
      if (k >= h->n_seis) return fail(R3D_EINVAL, "catch log: seismometer index out of range");
      if ((mask[k >> 5] >> (k & 31u)) & 1u) return fail(R3D_EINVAL, "catch log: seismometer listed twice");
      mask[k >> 5] |= 1u << (k & 31u);
    }
    if (d->bin_lo >= d->bin_hi || d->bin_hi > h->n_bins) return fail(R3D_EINVAL, "catch log: need bin_lo < bin_hi <= n_bins");
    if (!d->capacity || d->capacity > R3D_CATCH_LOG_MAX) return fail(R3D_EINVAL, "catch log: capacity must be in [1, R3D_CATCH_LOG_MAX]");
  }
  for (DevState *Dp : h->devs) {
    DevState &D = *Dp;
    if (int rc = drain(D)) return rc;
    CK(cudaSetDevice(D.device));
    CK(cudaStreamSynchronize(D.stream));
    if (D.log_mem) CK(cudaFreeAsync(D.log_mem, D.stream));
    D.log_mem = nullptr;
    D.G = CatchLog{};
    if (!d) continue;
    // [capacity] records | cursor | mask words
    cudaMemPool_t pool;
    if (int rc = device_pool(D.device, &pool)) return rc;
    CK(cudaMallocFromPoolAsync(&D.log_mem, d->capacity * sizeof(r3d_catch) + sizeof(unsigned long long) + words * sizeof(uint32_t), pool,
                               D.stream));
    D.G.rec = static_cast<r3d_catch *>(D.log_mem);
    D.G.cursor = reinterpret_cast<unsigned long long *>(D.G.rec + d->capacity);
    uint32_t *m = reinterpret_cast<uint32_t *>(D.G.cursor + 1);
    D.G.mask = m;
    CK(cudaMemsetAsync(D.G.cursor, 0, sizeof(unsigned long long), D.stream));
    CK(cudaMemcpyAsync(m, mask.data(), words * sizeof(uint32_t), cudaMemcpyHostToDevice, D.stream));
    D.G.cap = d->capacity; D.G.bin_lo = d->bin_lo; D.G.bin_hi = d->bin_hi;
    CK(cudaStreamSynchronize(D.stream));                     // (mask goes out of scope)
  }
  return 0;
}

int r3d_fetch_catch_log(r3d_handle *h, r3d_catch *out, uint64_t capacity, uint64_t *n_kept, uint64_t *n_matched) {
  DeviceGuard guard;
  if (!h) return fail(R3D_EINVAL, "null handle");
  if (capacity && !out) return fail(R3D_EINVAL, "null output array");
  if (h->devs.empty() || !h->devs[0]->log_mem) return fail(R3D_EINVAL, "the catch log is off (r3d_set_catch_log)");
  const size_t G = h->devs.size();
  std::vector<unsigned long long> cur(G, 0);
  uint64_t matched = 0, kept = 0;
  for (size_t g = 0; g < G; g++) {
    DevState &D = *h->devs[g];
    if (int rc = drain(D)) return rc;
    CK(cudaSetDevice(D.device));
    CK(cudaMemcpyAsync(&cur[g], D.G.cursor, sizeof(unsigned long long), cudaMemcpyDeviceToHost, D.stream));
    CK(cudaStreamSynchronize(D.stream));
    matched += cur[g];
    kept += std::min<unsigned long long>(cur[g], D.G.cap);
  }
  if (capacity && kept) {
    // every device's kept records, in device order, then sorted: directly in `out` when it holds them all
    std::vector<r3d_catch> tmp;
    r3d_catch *all = out;
    if (capacity < kept) { tmp.resize(kept); all = tmp.data(); }
    uint64_t at = 0;
    for (size_t g = 0; g < G; g++) {
      DevState &D = *h->devs[g];
      const uint64_t k = std::min<unsigned long long>(cur[g], D.G.cap);
      CK(cudaSetDevice(D.device));
      if (k) CK(cudaMemcpyAsync(all + at, D.G.rec, k * sizeof(r3d_catch), cudaMemcpyDeviceToHost, D.stream));
      CK(cudaStreamSynchronize(D.stream));
      at += k;
    }
    std::sort(all, all + kept, [](const r3d_catch &a, const r3d_catch &b) {
      return a.phonon != b.phonon ? a.phonon < b.phonon : a.moves != b.moves ? a.moves < b.moves : a.seis < b.seis;
    });
    if (all != out) memcpy(out, all, capacity * sizeof(r3d_catch));
  }
  if (n_kept) *n_kept = kept;
  if (n_matched) *n_matched = matched;
  return 0;
}

}  // extern "C"

// ---- sub-kernel hooks --------------------------------------------------------
namespace {
struct Scratch {               // device buffers of one hook call, freed on scope exit
  std::vector<void *> p;
  ~Scratch() { for (void *q : p) cudaFree(q); }
  template <class T> int up(const T *host, size_t n, T **dev) {
    void *q = nullptr;
    CK(cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T)));
    p.push_back(q);
    if (host && n) CK(cudaMemcpy(q, host, n * sizeof(T), cudaMemcpyHostToDevice));
    *dev = static_cast<T *>(q);
    return 0;
  }
};
int need_device() {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return fail(R3D_ENODEV, "no usable CUDA device");
  return 0;
}
// advance_mode: 0 r3d_test_path_to_boundary, 1 r3d_test_advance, 2 r3d_test_advance_time
int path_hook(r3d_handle *h, const double *in, uint32_t n, double *out, int advance_mode) {
  DeviceGuard guard;
  if (!h || !in || !out) return fail(R3D_EINVAL, "null argument");
  DevState &D = *h->devs[0];
  if (int rc = drain(D)) return rc;
  CK(cudaSetDevice(D.device));
  Scratch S;
  double *din, *dout;
  if (int rc = S.up(in, (size_t)n * (advance_mode ? 8 : 7), &din)) return rc;
  if (int rc = S.up((const double *)nullptr, (size_t)n * 9, &dout)) return rc;
  unsigned g = (n + 127) / 128;
  if (advance_mode == 2) {
    switch (h->cell_kind) {
      case R3D_CELL_CYLINDER: test_advance_time_kernel<Cylinder><<<g, 128>>>(D.M, din, n, dout); break;
      case R3D_CELL_SHELL: test_advance_time_kernel<Shell><<<g, 128>>>(D.M, din, n, dout); break;
      default: test_advance_time_kernel<Tetra><<<g, 128>>>(D.M, din, n, dout); break;
    }
  } else {
    switch (h->cell_kind) {
      case R3D_CELL_CYLINDER: test_path_kernel<Cylinder><<<g, 128>>>(D.M, din, n, dout, advance_mode); break;
      case R3D_CELL_SHELL: test_path_kernel<Shell><<<g, 128>>>(D.M, din, n, dout, advance_mode); break;
      default: test_path_kernel<Tetra><<<g, 128>>>(D.M, din, n, dout, advance_mode); break;
    }
  }
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, (size_t)n * 9 * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}
template <class K>
int rows_hook(K launch_fn, const double *in, uint32_t n, int win, int wout, double *out) {
  if (!in || !out) return fail(R3D_EINVAL, "null argument");
  if (int rc = need_device()) return rc;
  Scratch S;
  double *din, *dout;
  if (int rc = S.up(in, (size_t)n * win, &din)) return rc;
  if (int rc = S.up((const double *)nullptr, (size_t)n * wout, &dout)) return rc;
  launch_fn(din, dout);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, (size_t)n * wout * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}
}  // namespace

extern "C" {

// ---- scatterer tables (SURVEY 8f-2) ----------------------------------------------------------------------------------
}  // extern "C"
struct r3d_toa_set {
  int device = 0;
  uint32_t n = 0;
  double *th = nullptr, *ph = nullptr, *g = nullptr, *spol = nullptr;      // device: angles, G values [4][n], polarisation angles
};
extern "C" {

int r3d_toa_create(const double *toa_theta, const double *toa_phi, uint32_t n_toa, int device, r3d_toa_set **out) {
  if (!toa_theta || !toa_phi || !n_toa || !out) return fail(R3D_EINVAL, "null argument");
  *out = nullptr;
  if (int rc = need_device()) return rc;
  DeviceGuard guard;
  CK(cudaSetDevice(device));
  r3d_toa_set *t = new r3d_toa_set();
  t->device = device; t->n = n_toa;
  const size_t n = n_toa;
  cudaError_t e = cudaMalloc(&t->th, n * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&t->ph, n * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&t->g, 4 * n * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&t->spol, n * sizeof(double));
  if (e == cudaSuccess) e = cudaMemcpy(t->th, toa_theta, n * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(t->ph, toa_phi, n * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { r3d_toa_destroy(t); return fail(e == cudaErrorMemoryAllocation ? R3D_ENOMEM : R3D_ECUDA, std::string("r3d_toa_create: ") + cudaGetErrorString(e)); }
  *out = t;
  return 0;
}

void r3d_toa_destroy(r3d_toa_set *t) {
  if (!t) return;
  DeviceGuard guard;
  cudaSetDevice(t->device);
  cudaFree(t->th); cudaFree(t->ph); cudaFree(t->g); cudaFree(t->spol);
  delete t;
}

int r3d_scatterer_g_values(r3d_toa_set *t, const r3d_scatter_params *par, double *g, double *spol) {
  if (!t || !par || !g || !spol) return fail(R3D_EINVAL, "null argument");
  DeviceGuard guard;
  CK(cudaSetDevice(t->device));
  const r3d_scatter_params &P = *par;
  const size_t n = t->n;
  // PSATO's numerator does not depend on the angle (scatparams.cpp:184-188)
  const double numer = (8. * pow(kPi, 1.5) * P.eps * P.eps * P.a * P.a * P.a) * tgamma(P.kappa + 1.5) / tgamma(P.kappa);
  gsato_kernel<<<(unsigned)((n + 255) / 256), 256>>>(P, numer, t->th, t->ph, t->n, t->g, t->spol);
  CK(cudaGetLastError());
  CK(cudaMemcpy(g, t->g, 4 * n * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(spol, t->spol, n * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int r3d_build_scatterer_tables(const r3d_scatter_params *par, uint32_t n_par, const double *toa_theta, const double *toa_phi,
                               uint32_t n_toa, int device, double *cdf, double *spol, double *whole_cdf, double *mfp) {
  if (!par || !toa_theta || !toa_phi || !n_toa || !cdf || !spol || !whole_cdf || !mfp) return fail(R3D_EINVAL, "null argument");
  r3d_toa_set *t = nullptr;
  if (int rc = r3d_toa_create(toa_theta, toa_phi, n_toa, device, &t)) return rc;
  const size_t n = n_toa;
  for (uint32_t p = 0; p < n_par; p++) {
    double *c = cdf + (size_t)p * 4 * n, *w = whole_cdf + (size_t)p * 8;
    if (int rc = r3d_scatterer_g_values(t, par + p, c, spol + (size_t)p * n)) { std::string keep = g_err; r3d_toa_destroy(t); g_err = keep; return rc; }
    // ProbDist::Integrate (probability.cpp:21-35): the running sum in index order decides table indices, so it is formed on
    // the host exactly as the reference forms it (one thread per table)
    std::thread scan[4];
    for (int k = 0; k < 4; k++) {
      double *ct = c + (size_t)k * n;
      scan[k] = std::thread([ct, n] { for (size_t i = 1; i < n; i++) ct[i] += ct[i - 1]; });
    }
    for (int k = 0; k < 4; k++) scan[k].join();
    const double tot[4] = {c[n - 1], c[2 * n - 1], c[3 * n - 1], c[4 * n - 1]};
    // PopulateWholeProbs (scatterers.cpp:170-183), integrated: IN_P = {gpp, gps, 0, 0}, IN_S = {0, 0, gsp, gss}
    w[0] = tot[0]; w[1] = tot[0] + tot[1]; w[2] = w[1] + 0.0; w[3] = w[2] + 0.0;
    w[4] = 0.0; w[5] = 0.0; w[6] = 0.0 + tot[2]; w[7] = w[6] + tot[3];
    // ComputeMFPs (scatterers.cpp:195-220)
    mfp[2 * p + 0] = 1.0 / (w[3] / (double)n_toa);
    mfp[2 * p + 1] = 1.0 / (w[7] / (double)n_toa);
  }
  r3d_toa_destroy(t);
  return 0;
}

int r3d_test_cdf_search(const double *cdf, uint32_t n_cdf, const uint32_t *k, uint32_t n, uint32_t *out, int use_guide_table) {
  if (!cdf || !k || !out || !n_cdf) return fail(R3D_EINVAL, "null argument");
  if (int rc = need_device()) return rc;
  Scratch S;
  double *dc; uint32_t *dk, *dout, *dg;
  if (int rc = S.up(cdf, n_cdf, &dc)) return rc;
  if (int rc = S.up(k, n, &dk)) return rc;
  if (int rc = S.up((const uint32_t *)nullptr, n, &dout)) return rc;
  uint32_t shift = 32, stride = 1;
  if (use_guide_table && n_cdf >= 16) {
    int bits = use_guide_table > 1 ? use_guide_table : 0;
    if (!bits) while ((1ull << (bits + 2)) < n_cdf && bits < 24) bits++;
    if (bits > 24) bits = 24;
    shift = 31 - bits; stride = (1u << bits) + 1;
  }
  if (int rc = S.up((const uint32_t *)nullptr, stride, &dg)) return rc;
  if (shift < 32) build_guide_kernel<<<(stride + 255) / 256, 256>>>(dc, n_cdf, 1, shift, stride, dg);
  test_cdf_kernel<<<(n + 127) / 128, 128>>>(dc, n_cdf, dg, shift, dk, n, dout);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return 0;
}

int r3d_test_path_to_boundary(r3d_handle *h, const double *in, uint32_t n, double *out) { return path_hook(h, in, n, out, 0); }
int r3d_test_advance(r3d_handle *h, const double *in, uint32_t n, double *out) { return path_hook(h, in, n, out, 1); }
int r3d_test_advance_time(r3d_handle *h, const double *in, uint32_t n, double *out) { return path_hook(h, in, n, out, 2); }

int r3d_test_transform(const double *in, uint32_t n, double *out) {
  return rows_hook([&](double *a, double *b) { test_transform_kernel<<<(n + 127) / 128, 128>>>(a, n, b); }, in, n, 6, 3, out);
}
int r3d_test_rtcoef(const double *in, uint32_t n, double *out) {
  return rows_hook([&](double *a, double *b) { test_rtcoef_kernel<<<(n + 127) / 128, 128>>>(a, n, b); }, in, n, 15, 13, out);
}
int r3d_test_arith(const double *in, uint32_t n, double *out) {
  return rows_hook([&](double *a, double *b) { test_arith_kernel<<<(n + 127) / 128, 128>>>(a, n, b); }, in, n, 2, 4, out);
}
int r3d_test_pathlog(const double *in, uint32_t n, double *out) {
  return rows_hook([&](double *a, double *b) { test_pathlog_kernel<<<(n + 127) / 128, 128>>>(a, n, b); }, in, n, 1, 2, out);
}
int r3d_test_catch(double bin_dt, uint32_t n_bins, const double *in, uint32_t n, double *out) {
  return rows_hook([&](double *a, double *b) { test_catch_kernel<<<(n + 127) / 128, 128>>>(bin_dt, n_bins, a, n, b); }, in, n, 28, 6, out);
}

}  // extern "C"
