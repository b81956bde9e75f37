"""ctypes binding of snapshot_oracle/libsnaporacle.so -- the CPU restatement of the energy snapshots, for tests only."""
import ctypes as C
import os
import subprocess

import numpy as np

from radiative3d_b200 import abi

DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "snapshot_oracle")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(DIR, "libsnaporacle.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", DIR], check=True, capture_output=True)
        L = C.CDLL(path)
        pd, pu64 = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
        pdesc, psnap = C.POINTER(abi.ModelDesc), C.POINTER(abi.SnapshotDesc)
        L.r3d_oracle_check_snapshots.argtypes = [pdesc, psnap, pu64]
        L.r3d_oracle_run_snapshots.argtypes = [pdesc, C.c_uint64, C.c_uint64, C.c_uint64, psnap, pd, pu64, pd, pu64, C.c_void_p]
        L.r3d_oracle_advance_time.argtypes = [pdesc, pd, C.c_uint32, pd]
        L.r3d_oracle_advance_time.restype = None
        _LIB = L
    return _LIB


def check(model, times, origin, voxel, dims):
    """0 or the R3D_E* code r3d_set_snapshots would return for this grid"""
    d = model.desc()
    s, t = abi.snapshot_desc(times, origin, voxel, dims)
    return lib().r3d_oracle_check_snapshots(C.byref(d), C.byref(s), None)


def run(model, first, n, seed, times, origin, voxel, dims, finals=False):
    """Trace phonons [first, first+n) on the CPU with snapshot records.
    Returns (energy[K,nz,ny,nx,2], count[...] u64, outside_energy[K,2], outside_count[K,2] u64, finals|None)."""
    d = model.desc()
    s, t = abi.snapshot_desc(times, origin, voxel, dims)
    nx, ny, nz = (int(x) for x in dims)
    k = t.size
    e = np.zeros((k, nz, ny, nx, 2))
    c = np.zeros((k, nz, ny, nx, 2), dtype=np.uint64)
    oe = np.zeros((k, 2))
    oc = np.zeros((k, 2), dtype=np.uint64)
    fin = np.zeros(n, dtype=abi.PHONON_FINAL_DTYPE) if finals else None
    rc = lib().r3d_oracle_run_snapshots(C.byref(d), first, n, seed, C.byref(s), abi.as_ptr(e, C.c_double), abi.as_ptr(c, C.c_uint64),
                                        abi.as_ptr(oe, C.c_double), abi.as_ptr(oc, C.c_uint64), fin.ctypes.data if finals else None)
    if rc != 0:
        raise ValueError(f"r3d_oracle_run_snapshots returned {rc}")
    return e, c, oe, oc, fin


def advance_time(model, x):
    d = model.desc()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 8)
    out = np.zeros((x.shape[0], 9))
    lib().r3d_oracle_advance_time(C.byref(d), abi.as_ptr(x, C.c_double), x.shape[0], abi.as_ptr(out, C.c_double))
    return out
