"""ctypes mirror of include/r3d_gpu.h (structs and constants only).

Kept separate from the library loader so that the CPU-only test-suite can build
descriptors (e.g. for the oracle) without libr3dgpu.so being loadable.
"""
import ctypes as C

import numpy as np

R3D_ABI_VERSION = 2

R3D_RAY_P, R3D_RAY_S, R3D_RAY_SH, R3D_RAY_SV = 0, 1, 1, 2
R3D_CELL_CYLINDER, R3D_CELL_TETRA, R3D_CELL_SHELL = 0, 1, 2
R3D_FACE_COLLECT, R3D_FACE_REFLECT, R3D_FACE_ADJOIN, R3D_FACE_DISCON = 1, 2, 4, 8
R3D_CYL_NPARAM, R3D_SHELL_NPARAM, R3D_TETRA_NPARAM = 17, 14, 38
R3D_CYL_NFACES, R3D_SHELL_NFACES, R3D_TETRA_NFACES = 3, 2, 4
R3D_SEIS_NPARAM = 18
R3D_BIN_NF64, R3D_BIN_NCNT = 5, 2
R3D_CNT_LOST, R3D_CNT_TIMEOUT, R3D_CNT_INVALID = 0, 1, 2
R3D_CNT_EVENTS, R3D_CNT_CATCHES, R3D_CNT_SCATTERS = 3, 4, 5
R3D_CNT_PHONONS, R3D_CNT_DIAG = 6, 7
R3D_NCOUNTERS = 8
R3D_NDIAG_LANES = 8
R3D_FATE_LOST, R3D_FATE_TIMEOUT, R3D_FATE_INVALID = 1, 2, 3
(R3D_INV_PATH_NAN, R3D_INV_TIME_NAN, R3D_INV_PATH_NEGATIVE, R3D_INV_TIME_NEGATIVE, R3D_INV_STUCK, R3D_INV_SLOW,
 R3D_INV_LOOP_EXCEED) = range(7)

_pd = C.POINTER(C.c_double)
_pu32 = C.POINTER(C.c_uint32)
_pu8 = C.POINTER(C.c_uint8)


class ModelDesc(C.Structure):
    """struct r3d_model_desc"""
    _fields_ = [
        ("freq_hz", C.c_double), ("ttl", C.c_double), ("bin_dt", C.c_double),
        ("n_bins", C.c_uint32), ("ecs_radial", C.c_int32),
        ("earth_center", C.c_double * 3),
        ("min_theta", C.c_double), ("max_theta", C.c_double), ("slow_concern", C.c_double),
        ("loop_concern", C.c_uint64),
        ("no_deflect", C.c_int32), ("reserved0", C.c_int32),
        ("n_toa", C.c_uint32), ("reserved1", C.c_uint32),
        ("toa_theta", _pd), ("toa_phi", _pd),
        ("src_loc", C.c_double * 3),
        ("src_cell", C.c_uint32), ("reserved2", C.c_uint32),
        ("src_whole_cdf", _pd), ("src_cdf", _pd),
        ("n_scat", C.c_uint32), ("reserved3", C.c_uint32),
        ("scat_mfp", _pd), ("scat_whole_cdf", _pd), ("scat_cdf", _pd), ("scat_spol", _pd),
        ("n_cells", C.c_uint32), ("cell_kind", C.c_uint32),
        ("cell_nparam", C.c_uint32), ("faces_per_cell", C.c_uint32),
        ("cell_params", _pd), ("cell_scat", _pu32), ("face_flags", _pu8), ("face_other_cell", _pu32),
        ("cyl_radius2", C.c_double),
        ("n_seis", C.c_uint32), ("reserved4", C.c_uint32),
        ("seis", _pd),
    ]


class PhononFinal(C.Structure):
    """struct r3d_phonon_final"""
    _fields_ = [
        ("time", C.c_double), ("pathlen", C.c_double), ("amp", C.c_double),
        ("loc", C.c_double * 3),
        ("theta", C.c_double), ("phi", C.c_double), ("pol", C.c_double),
        ("moves", C.c_uint32), ("cell", C.c_uint32), ("type", C.c_uint32), ("fate", C.c_uint32),
        ("draws", C.c_uint32), ("catches", C.c_uint32), ("scatters", C.c_uint32), ("iters", C.c_uint32),
    ]


PHONON_FINAL_DTYPE = np.dtype([
    ("time", "<f8"), ("pathlen", "<f8"), ("amp", "<f8"), ("loc", "<f8", (3,)),
    ("theta", "<f8"), ("phi", "<f8"), ("pol", "<f8"),
    ("moves", "<u4"), ("cell", "<u4"), ("type", "<u4"), ("fate", "<u4"),
    ("draws", "<u4"), ("catches", "<u4"), ("scatters", "<u4"), ("iters", "<u4"),
])
assert PHONON_FINAL_DTYPE.itemsize == C.sizeof(PhononFinal) == 104


R3D_EV_GEN, R3D_EV_SCT, R3D_EV_COL, R3D_EV_REF, R3D_EV_CEL, R3D_EV_LST, R3D_EV_TMO, R3D_EV_INV = range(8)
R3D_EV_ALL = 0xFF
EVENT_LABELS = ("GEN", "SCT", "COL", "REF", "CEL", "LST", "TMO", "INV")      # dataout.hpp:308-324

# struct r3d_event
EVENT_DTYPE = np.dtype([
    ("phonon", "<u8"), ("seq", "<u4"), ("kind", "<u4"), ("type", "<u4"), ("moves", "<u4"), ("cell", "<u4"), ("reason", "<u4"),
    ("time", "<f8"), ("pathlen", "<f8"), ("loc", "<f8", (3,)), ("theta", "<f8"), ("phi", "<f8"), ("amp", "<f8"),
])
assert EVENT_DTYPE.itemsize == 96


R3D_EINVAL = 1
R3D_SNAP_MAX_TIMES = 64
R3D_SNAP_MAX_CELLS = 1 << 28


class SnapshotDesc(C.Structure):
    """struct r3d_snapshot_desc (energy snapshots: lapse times and voxel grid)"""
    _fields_ = [("n_times", C.c_uint32), ("reserved", C.c_uint32), ("times", _pd),
                ("origin", C.c_double * 3), ("voxel", C.c_double * 3), ("dims", C.c_uint32 * 3), ("reserved2", C.c_uint32)]


def snapshot_desc(times, origin, voxel, dims):
    """(SnapshotDesc, the float64 times array it points into: keep it alive while the descriptor is used)."""
    t = np.ascontiguousarray(times, dtype=np.float64).reshape(-1)
    d = SnapshotDesc(n_times=t.size, times=as_ptr(t, C.c_double))
    for a in range(3):
        d.origin[a], d.voxel[a], d.dims[a] = float(origin[a]), float(voxel[a]), int(dims[a])
    return d, t


class ScatterParams(C.Structure):
    """struct r3d_scatter_params (ScatterParams, scatparams.hpp:51-61)"""
    _fields_ = [("nu", C.c_double), ("eps", C.c_double), ("a", C.c_double), ("kappa", C.c_double), ("el", C.c_double), ("gam0", C.c_double)]


def as_ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))
