"""Host-side binding of libr3dgpu.so (include/r3d_gpu.h) -- the product path.

`Engine` stands where the body of the reference's Model::RunSimulation loop stands
(model.cpp:611-625): give it a flattened model, ask it to trace a range of phonon
indices, fetch the seismometer bins and loss counters (what DataReporter holds after
the loop, dataout.cpp:591-694).

There is NO CPU fallback: if the CUDA library is not built, or no CUDA device is usable,
the calls raise.  Nothing in this module imports or executes anything under oracle/.
"""
import ctypes as C
import os

import numpy as np

from . import abi
from .model import FlatModel

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libr3dgpu.so")
_lib = None

EXPORTS = [
    "r3d_create", "r3d_run", "r3d_sync", "r3d_fetch", "r3d_reset", "r3d_device_accumulators", "r3d_device_accumulator_blocks", "r3d_stream",
    "r3d_launch_count", "r3d_trace", "r3d_trace_events", "r3d_build_scatterer_tables", "r3d_toa_create", "r3d_scatterer_g_values", "r3d_toa_destroy", "r3d_set_profiling", "r3d_kernel_times", "r3d_test_cdf_search", "r3d_test_path_to_boundary", "r3d_test_advance",
    "r3d_test_advance_time", "r3d_set_snapshots", "r3d_fetch_snapshots", "r3d_test_transform", "r3d_test_rtcoef", "r3d_test_catch", "r3d_test_arith", "r3d_test_pathlog", "r3d_destroy", "r3d_last_error", "r3d_abi_version",
]


class R3DError(RuntimeError):
    """Non-zero return from the C ABI; mirrors the reference's `throw Runtime(...)` convention (typedefs.hpp:123)."""

    def __init__(self, code, msg):
        super().__init__(f"r3d error {code}: {msg}")
        self.code = code


def load_library(path=None):
    """dlopen libr3dgpu.so and declare its prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("R3D_LIBRARY") or _LIB_PATH      # R3D_LIBRARY: a tuning build of the same library
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the propagate path.")
    L = C.CDLL(p)
    pd, pu32, pu64, vp = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.c_void_p
    L.r3d_create.argtypes = [C.POINTER(abi.ModelDesc), C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.r3d_run.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64]
    L.r3d_sync.argtypes = [vp, pd]
    L.r3d_fetch.argtypes = [vp, pd, pu64, pu64, pu32]
    L.r3d_reset.argtypes = [vp]
    L.r3d_device_accumulators.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.r3d_device_accumulator_blocks.argtypes = [vp, C.c_int, C.POINTER(vp), pu64, C.POINTER(vp), pu64, pu64]
    L.r3d_stream.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.r3d_launch_count.argtypes = [vp, pu64]
    L.r3d_trace.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64, vp]
    L.r3d_trace_events.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, vp, C.c_uint64, pu64]
    L.r3d_build_scatterer_tables.argtypes = [C.POINTER(abi.ScatterParams), C.c_uint32, pd, pd, C.c_uint32, C.c_int, pd, pd, pd, pd]
    L.r3d_set_profiling.argtypes = [vp, C.c_int]
    L.r3d_kernel_times.argtypes = [vp, pd, pu64, pu64]
    L.r3d_test_cdf_search.argtypes = [pd, C.c_uint32, pu32, C.c_uint32, pu32, C.c_int]
    L.r3d_test_path_to_boundary.argtypes = [vp, pd, C.c_uint32, pd]
    L.r3d_test_advance.argtypes = [vp, pd, C.c_uint32, pd]
    L.r3d_test_advance_time.argtypes = [vp, pd, C.c_uint32, pd]
    L.r3d_set_snapshots.argtypes = [vp, C.POINTER(abi.SnapshotDesc)]
    L.r3d_fetch_snapshots.argtypes = [vp, pd, pu64, pd, pu64]
    L.r3d_test_transform.argtypes = [pd, C.c_uint32, pd]
    L.r3d_test_rtcoef.argtypes = [pd, C.c_uint32, pd]
    L.r3d_test_arith.argtypes = [pd, C.c_uint32, pd]
    L.r3d_test_pathlog.argtypes = [pd, C.c_uint32, pd]
    L.r3d_test_catch.argtypes = [C.c_double, C.c_uint32, pd, C.c_uint32, pd]
    L.r3d_destroy.argtypes = [vp]
    L.r3d_destroy.restype = None
    L.r3d_last_error.restype = C.c_char_p
    L.r3d_abi_version.restype = C.c_int
    if L.r3d_abi_version() != abi.R3D_ABI_VERSION:
        raise RuntimeError("libr3dgpu.so ABI version mismatch; rebuild it")
    if path is None:
        _lib = L
    return L


def _ck(L, rc):
    if rc != 0:
        raise R3DError(rc, L.r3d_last_error().decode(errors="replace"))


def _pd(a):
    return abi.as_ptr(a, C.c_double)


class _CudaView:
    """A device allocation exposed through __cuda_array_interface__ (so torch.as_tensor can wrap it)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None}
        self._owner = owner


class Engine:
    """The GPU propagate path for one flattened model, replicated on `devices` (SURVEY 8e)."""

    def __init__(self, model: FlatModel, devices=(0,), device_tables=None):
        """device_tables: {name: device pointer or (device pointer, owner)} for any of the five large tables
        (distributed.BIG_TABLES) that are already in device memory - e.g. received by distributed.broadcast_model_tables -
        and must be complete (synchronise the producing stream first); the model's host arrays still give the shapes."""
        self._L = load_library()
        self.model = model
        self.devices = tuple(devices)
        self._h = C.c_void_p()
        d = model.desc()
        for name, ptr in (device_tables or {}).items():
            if name not in ("toa_theta", "toa_phi", "src_cdf", "scat_cdf", "scat_spol"):
                raise ValueError(f"{name} cannot be given in device memory (include/r3d_gpu.h)")
            setattr(d, name, C.cast(C.c_void_p(ptr[0] if isinstance(ptr, tuple) else ptr), C.POINTER(C.c_double)))
        dev = (C.c_int * len(self.devices))(*self.devices)
        _ck(self._L, self._L.r3d_create(C.byref(d), dev, len(self.devices), C.byref(self._h)))

    # -- lifetime --
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.r3d_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- the loop of Model::RunSimulation (model.cpp:611-625) --
    def run_simulation(self, n_phonons, seed=20261018, first_phonon=0):
        """Enqueue phonons [first_phonon, first_phonon + n_phonons); accumulates into the bins.  Asynchronous."""
        _ck(self._L, self._L.r3d_run(self._h, first_phonon, n_phonons, seed))

    def sync(self):
        """Wait; returns device seconds (CUDA events, max over devices) of the runs since the last sync."""
        t = C.c_double()
        _ck(self._L, self._L.r3d_sync(self._h, C.byref(t)))
        return t.value

    def fetch(self, out=None):
        """(energies[n_seis,n_bins,5], counts[n_seis,n_bins,2], counters[8]) summed over devices.  `out` = (energies, counts)
        host arrays of those shapes to fill instead of new ones (C-contiguous float64 / uint64; pinned memory makes the
        device-to-host copy direct)."""
        m = self.model
        if out is not None:
            e, c = out
            if (e.shape != (m.n_seis, m.n_bins, abi.R3D_BIN_NF64) or e.dtype != np.float64 or not e.flags.c_contiguous or
                    c.shape != (m.n_seis, m.n_bins, abi.R3D_BIN_NCNT) or c.dtype != np.uint64 or not c.flags.c_contiguous):
                raise ValueError("fetch(out=...): need C-contiguous float64 [n_seis,n_bins,5] and uint64 [n_seis,n_bins,2] arrays")
        else:
            e = np.zeros((m.n_seis, m.n_bins, abi.R3D_BIN_NF64))
            c = np.zeros((m.n_seis, m.n_bins, abi.R3D_BIN_NCNT), dtype=np.uint64)
        k = np.zeros(abi.R3D_NCOUNTERS, dtype=np.uint64)
        diag = C.c_uint32()
        _ck(self._L, self._L.r3d_fetch(self._h, _pd(e), abi.as_ptr(c, C.c_uint64), abi.as_ptr(k, C.c_uint64), C.byref(diag)))
        return e, c, k

    def reset(self):
        _ck(self._L, self._L.r3d_reset(self._h))

    def trace(self, n_phonons, seed=20261018, first_phonon=0):
        """Per-phonon end states (parity hook); also accumulates bins like run_simulation."""
        out = np.zeros(n_phonons, dtype=abi.PHONON_FINAL_DTYPE)
        _ck(self._L, self._L.r3d_trace(self._h, first_phonon, n_phonons, seed, out.ctypes.data))
        return out

    def trace_events(self, n_phonons, seed=20261018, first_phonon=0, kinds=abi.R3D_EV_ALL, capacity=None):
        """Event reports (DataReporter::Report*, dataout.cpp:484-617) of phonons [first, first+n), sorted by
        (phonon, seq); also accumulates bins like run_simulation.  `capacity` = records to make room for
        (default 512 per phonon); raises if more events occurred (the bins then hold this pass already)."""
        cap = int(capacity or max(4096, 512 * n_phonons))
        out = np.zeros(cap, dtype=abi.EVENT_DTYPE)
        n = C.c_uint64()
        _ck(self._L, self._L.r3d_trace_events(self._h, first_phonon, n_phonons, seed, kinds, out.ctypes.data, cap, C.byref(n)))
        if n.value > cap:
            raise R3DError(abi.R3D_EINVAL if hasattr(abi, "R3D_EINVAL") else 1, f"{n.value} events occurred, room for {cap}")
        return out[:n.value]

    # -- energy snapshots (include/r3d_gpu.h r3d_set_snapshots) --
    def set_snapshots(self, times, origin=None, voxel=None, dims=None):
        """Record phonon energy at the lapse `times` (increasing, in [0, ttl], at most 64) on the voxel grid `origin`,
        `voxel` (sizes), `dims` (nx, ny, nz), in model coordinates, during the following runs; zeroed accumulators.
        `times` None or empty turns snapshots off."""
        if times is None or len(times) == 0:
            _ck(self._L, self._L.r3d_set_snapshots(self._h, None))
            self._snap = None
            return
        d, t = abi.snapshot_desc(times, origin, voxel, dims)
        _ck(self._L, self._L.r3d_set_snapshots(self._h, C.byref(d)))
        self._snap = (t.size, tuple(int(x) for x in dims))

    def fetch_snapshots(self):
        """(energy[K, nz, ny, nx, 2] f64, count[K, nz, ny, nx, 2] u64, outside_energy[K, 2], outside_count[K, 2]) summed
        over the devices; the last axis is the ray type (P, S)."""
        if getattr(self, "_snap", None) is None:
            raise R3DError(abi.R3D_EINVAL, "snapshots are off (set_snapshots)")
        k, (nx, ny, nz) = self._snap
        e = np.zeros((k, nz, ny, nx, 2))
        c = np.zeros((k, nz, ny, nx, 2), dtype=np.uint64)
        oe = np.zeros((k, 2))
        oc = np.zeros((k, 2), dtype=np.uint64)
        _ck(self._L, self._L.r3d_fetch_snapshots(self._h, _pd(e), abi.as_ptr(c, C.c_uint64), _pd(oe), abi.as_ptr(oc, C.c_uint64)))
        return e, c, oe, oc

    @property
    def launch_count(self):
        n = C.c_uint64()
        _ck(self._L, self._L.r3d_launch_count(self._h, C.byref(n)))
        return n.value

    def set_profiling(self, on=True):
        """Reset the kernel-time totals (the propagate kernel is always event-timed; `on` is ignored)."""
        _ck(self._L, self._L.r3d_set_profiling(self._h, 1 if on else 0))

    def kernel_times(self):
        """Device slot 0 since the last set_profiling(): propagate-kernel seconds (CUDA events) and launches, the
        seconds split into the CTAs' two phases, iterations of the busiest CTA, CTAs per launch, and the units the
        kernel processed (loop events, table draws, bin updates) as tallied by the handle's counters."""
        t = np.zeros(3)
        n = np.zeros(3, dtype=np.uint64)
        u = np.zeros(3, dtype=np.uint64)
        _ck(self._L, self._L.r3d_kernel_times(self._h, _pd(t), abi.as_ptr(n, C.c_uint64), abi.as_ptr(u, C.c_uint64)))
        return {"seconds": float(t[0]), "launches": int(n[0]), "phase1_seconds": float(t[1]), "phase2_seconds": float(t[2]),
                "iterations": int(n[1]), "ctas": int(n[2]), "events": int(u[0]), "draws": int(u[1]), "catches": int(u[2])}

    def stream(self, slot=0):
        s = C.c_void_p()
        _ck(self._L, self._L.r3d_stream(self._h, slot, C.byref(s)))
        return s.value

    def device_accumulators(self, slot=0):
        """Device-resident (energies f64, counts u64 viewed as i64, counters i64) for in-place collectives."""
        e, c, k = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _ck(self._L, self._L.r3d_device_accumulators(self._h, slot, C.byref(e), C.byref(c), C.byref(k)))
        nb = self.model.n_seis * self.model.n_bins
        return (_CudaView(e.value, (nb * abi.R3D_BIN_NF64,), "<f8", self),
                _CudaView(c.value, (nb * abi.R3D_BIN_NCNT,), "<i8", self),
                _CudaView(k.value, (abi.R3D_NCOUNTERS,), "<i8", self))

    def device_accumulator_blocks(self, slot=0):
        """The same accumulators as two device-resident blocks for in-place collectives, one per element type:
        (f64 block = energies, i64 block = counts | counters | diagnostic-bit lanes, index of the counters in the i64 block)."""
        f, i = C.c_void_p(), C.c_void_p()
        nf, ni, at = C.c_uint64(), C.c_uint64(), C.c_uint64()
        _ck(self._L, self._L.r3d_device_accumulator_blocks(self._h, slot, C.byref(f), C.byref(nf), C.byref(i), C.byref(ni), C.byref(at)))
        return (_CudaView(f.value, (nf.value,), "<f8", self), _CudaView(i.value, (ni.value,), "<i8", self), int(at.value))

    # -- deterministic sub-kernels (r3d_test_*) --
    def _rows(self, fn, win, wout, x):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, win)
        out = np.zeros((x.shape[0], wout))
        _ck(self._L, fn(self._h, _pd(x), x.shape[0], _pd(out)))
        return out

    def path_to_boundary(self, x):
        return self._rows(self._L.r3d_test_path_to_boundary, 7, 9, x)

    def advance(self, x):
        return self._rows(self._L.r3d_test_advance, 8, 9, x)

    def advance_time(self, x):
        """rows {cell, type, x, y, z, theta, phi, dt} -> the snapshot deposit's point at travel time dt along the move to
        the boundary, as rows of advance()"""
        return self._rows(self._L.r3d_test_advance_time, 8, 9, x)


def _free_rows(name, win, wout, x, *pre):
    L = load_library()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, win)
    out = np.zeros((x.shape[0], wout))
    _ck(L, getattr(L, name)(*pre, _pd(x), x.shape[0], _pd(out)))
    return out


def cdf_search(cdf, k, use_guide_table=1):
    """ProbDist::GetRandomIndex on the device for 31-bit draws k.  use_guide_table: 0 plain bisection,
    1 guide table of default size, n>1 guide table with 2**n buckets."""
    L = load_library()
    cdf = np.ascontiguousarray(cdf, dtype=np.float64)
    k = np.ascontiguousarray(k, dtype=np.uint32)
    out = np.zeros(k.size, dtype=np.uint32)
    _ck(L, L.r3d_test_cdf_search(_pd(cdf), cdf.size, abi.as_ptr(k, C.c_uint32), k.size, abi.as_ptr(out, C.c_uint32),
                                 use_guide_table))
    return out


def build_scatterer_tables(params, toa_theta, toa_phi, device=0):
    """What the reference's Scatterer constructor computes (scatterers.cpp:134-220), G values on the device.
    params = (nu, eps, a, kappa, el, gam0) -> (cdf[4, n_toa], spol[n_toa], whole_cdf[2, 4], mfp[2]); a 2-D `params`
    builds the tables of several scatterers in one call (leading axis = scatterer), laid out as FlatModel wants them."""
    L = load_library()
    th = np.ascontiguousarray(toa_theta, dtype=np.float64)
    ph = np.ascontiguousarray(toa_phi, dtype=np.float64)
    p2 = np.atleast_2d(np.asarray(params, dtype=np.float64))
    n, k = th.size, p2.shape[0]
    cdf, spol, whole, mfp = np.zeros((k, 4, n)), np.zeros((k, n)), np.zeros((k, 2, 4)), np.zeros((k, 2))
    par = (abi.ScatterParams * k)(*[abi.ScatterParams(*map(float, row)) for row in p2])
    _ck(L, L.r3d_build_scatterer_tables(par, k, _pd(th), _pd(ph), n, device, _pd(cdf), _pd(spol), _pd(whole), _pd(mfp)))
    if np.ndim(params) == 1:
        return cdf[0], spol[0], whole[0], mfp[0]
    return cdf, spol, whole, mfp


def transform(x):
    return _free_rows("r3d_test_transform", 6, 3, x)


def rtcoef(x):
    return _free_rows("r3d_test_rtcoef", 15, 13, x)


def pathlog(k):
    """31-bit draws k -> rows {the kernel's -log(1 - k / 2^31), the math library's} on the device."""
    return _free_rows("r3d_test_pathlog", 1, 2, np.asarray(k, dtype=np.float64))


def arith(x):
    """rows {a, b} -> {qdiv(a, b), a / b, qsqrt0(a), sqrt(a)} on the device (r3d_device.cuh)."""
    return _free_rows("r3d_test_arith", 2, 4, x)


def catch(bin_dt, n_bins, x):
    return _free_rows("r3d_test_catch", 28, 6, x, C.c_double(bin_dt), C.c_uint32(n_bins))
