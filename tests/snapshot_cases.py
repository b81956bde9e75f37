"""Shared inputs of the energy-snapshot tests (tests/test_oracle_snapshots.py, tests/test_gpu_snapshots.py)."""
import numpy as np

import oracle_binding as ob


def grid_around(model, n=(8, 8, 8)):
    """A grid over the box that the seismometers and the source span (padded by 10 %), `n` voxels per axis, shifted so
    that the source is at the centre of a voxel.  (A voxel face through the source puts the early records of every phonon
    that travels along that plane on the face, where the last bit of its position decides the voxel.)"""
    src = np.asarray(model.src_loc)
    pts = np.vstack([src[None, :], model.seis.reshape(-1, 18)[:, :3]])
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    ext = np.maximum(hi - lo, 1.0)
    lo, hi = lo - 0.1 * ext, hi + 0.1 * ext
    voxel = (hi - lo) / np.asarray(n, dtype=np.float64)
    origin = src - (np.floor((src - lo) / voxel) + 0.5) * voxel
    return origin, voxel, tuple(int(x) for x in n)


def times_of(model):
    """8 snapshot times over [0, ttl], t = 0 and t = ttl included."""
    return model.ttl * np.array([0.0, 0.01, 0.03, 0.1, 0.2, 0.4, 0.7, 1.0])


def advance_time_rows(model, z, seed=1):
    """Rows {cell, type, x, y, z, theta, phi, dt} from the golden path_in, dt = u * (time to the boundary), u in [0, 1);
    also the boundary travel (oracle) of each row."""
    x = np.asarray(z["path_in"], dtype=np.float64)
    b = ob.path_to_boundary(model, x)
    ok = np.isfinite(b[:, 1]) & (b[:, 1] > 0) & np.isfinite(b[:, 0])
    x, b = x[ok], b[ok]
    u = np.random.default_rng(seed).random(len(x))
    return np.concatenate([x, (u * b[:, 1])[:, None]], axis=1), b


def time_resolved(model, rows, out):
    """Rows whose move's travel-time formula resolves time near the returned point: a step of 1e-7 of the length changes
    the time by 1e-7 length / v to 1e-3.  (Nearly straight arcs - radius far above the move's length - and moves of
    1e-12 km do not: the formulas then difference nearly equal angles, and time is only known to ~1e-5 relative.)"""
    L = out[:, 0]
    a = ob.advance(model, np.concatenate([rows[:, :7], L[:, None]], axis=1))
    b = ob.advance(model, np.concatenate([rows[:, :7], (L * (1 + 1e-7))[:, None]], axis=1))
    with np.errstate(invalid="ignore", divide="ignore"):
        ratio = (b[:, 1] - a[:, 1]) / (1e-7 * a[:, 1])
    return (L > 1e-6) & (ratio > 0.5) & (ratio < 2.0)


def dt_tolerance(cfg):
    """Relative tolerance of the travel time reached by advance_time: straight rays are exact (len = dt v); curved rays
    land on dt to the resolution of their cell's travel-time formula, a difference of nearly equal terms."""
    return 1e-12 if cfg in ("halfspace", "halfspace_nearsrc50", "lopnor") else 1e-9
