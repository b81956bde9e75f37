"""The flattened model of a BASELINE workload at any take-off-angle degree, built without the reference program.

Only three parts of a model depend on the take-off-angle (TOA) degree: the TOA set, the source's CDF tables over it and the
scatterers' CDF tables over it.  Everything else (cells, faces, seismometers, the scalars and the scatterers' parameters) is
taken from the model the reference built for the same command line, stored in tests/golden/golden_<cfg>.npz and
scat_params.npz.  The three degree-dependent parts are computed here:
  * toa_set():      the reference's icosahedral sphere tessellation (nTOA = 20 * 4^degree);
  * source_tables(): the shear-dislocation radiation pattern (P, SH, SV) over the TOA set;
  * the scatterer tables on the device (engine.build_scatterer_tables).
tests/test_workload_model.py holds the result to the models the reference built (degrees 2 and 3).
"""
import os

import numpy as np

from . import workloads
from .model import FlatModel, _ARRAYS

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# The icosahedron: 12 unit vertices and 20 faces, in the order and orientation of the reference's tessellation.
_P = (1.0 + 5.0 ** 0.5) / 2.0
_X, _Z = 1.0 / np.sqrt(1.0 + _P * _P), _P / np.sqrt(1.0 + _P * _P)
_VERTS = np.array([(_X, 0, _Z), (-_X, 0, _Z), (_X, 0, -_Z), (-_X, 0, -_Z), (_Z, _X, 0), (_Z, -_X, 0), (-_Z, _X, 0),
                   (-_Z, -_X, 0), (0, _Z, _X), (0, -_Z, _X), (0, _Z, -_X), (0, -_Z, -_X)])
_FACES = [(0, 1, 9), (0, 1, 8), (2, 3, 11), (2, 3, 10), (5, 4, 0), (5, 4, 2), (6, 7, 1), (6, 7, 3), (9, 11, 5), (9, 11, 7),
          (8, 10, 4), (8, 10, 6), (0, 9, 5), (0, 8, 4), (1, 9, 7), (1, 8, 6), (2, 11, 5), (2, 10, 4), (3, 11, 7), (3, 10, 6)]


def _unit(v):
    return v / np.sqrt((v * v).sum(-1, keepdims=True))


def toa_set(degree):
    """(theta, phi) of the 20 * 4^degree take-off angles: every face of the icosahedron split `degree` times into four
    (edge midpoints pushed out to the sphere; children in the order corner A, corner B, corner C, middle), one angle per
    final triangle at its normalised centroid.  Agrees with the reference's set to within 1e-15 rad."""
    t = _VERTS[np.array(_FACES)]
    for _ in range(int(degree)):
        a, b, c = t[:, 0], t[:, 1], t[:, 2]
        ab, bc, ca = _unit((a + b) / 2), _unit((b + c) / 2), _unit((c + a) / 2)
        t = np.stack([np.stack(k, 1) for k in ((a, ab, ca), (ab, b, bc), (ca, bc, c), (bc, ca, ab))], 1).reshape(-1, 3, 3)
    p = _unit((t[:, 0] + t[:, 1] + t[:, 2]) / 3)
    return np.arccos(p[:, 2]), np.arctan2(p[:, 1], p[:, 0])


def moment_tensor(strike, dip, rake):
    """Unit-norm double couple (Aki & Richards 4.88, M0 = 1/sqrt 2) in the model's frame: x east, y north, z up."""
    s, d, r = np.radians([strike, dip, rake])
    nn = -(np.sin(d) * np.cos(r) * np.sin(2 * s) + np.sin(2 * d) * np.sin(r) * np.sin(s) ** 2)
    ne = np.sin(d) * np.cos(r) * np.cos(2 * s) + 0.5 * np.sin(2 * d) * np.sin(r) * np.sin(2 * s)
    nd = -(np.cos(d) * np.cos(r) * np.cos(s) + np.cos(2 * d) * np.sin(r) * np.sin(s))
    ee = np.sin(d) * np.cos(r) * np.sin(2 * s) - np.sin(2 * d) * np.sin(r) * np.cos(s) ** 2
    ed = -(np.cos(d) * np.cos(r) * np.sin(s) - np.cos(2 * d) * np.sin(r) * np.cos(s))
    dd = np.sin(2 * d) * np.sin(r)
    return np.array([[ee, ne, -ed], [ne, nn, -nd], [-ed, -nd, dd]]) / np.sqrt(2.0)


def source_tables(strike, dip, rake, theta, phi):
    """(src_whole_cdf[3], src_cdf[3 * nTOA]): squared P, SH and SV radiation amplitudes over the TOA set, each summed
    cumulatively in index order, and the running sum of the three totals."""
    st, ct, sp, cp = np.sin(theta), np.cos(theta), np.sin(phi), np.cos(phi)
    n = np.stack([st * cp, st * sp, ct], -1)
    mn = n @ moment_tensor(strike, dip, rake).T
    p = (mn * n).sum(-1)
    s = mn - p[:, None] * n
    sh = -s[:, 0] * sp + s[:, 1] * cp
    sv = s[:, 0] * ct * cp + s[:, 1] * ct * sp - s[:, 2] * st
    cdf = np.cumsum(np.stack([p * p, sh * sh, sv * sv]), axis=1)
    return np.cumsum(cdf[:, -1]), cdf.ravel()


def build_model(config, toa_degree, device=0):
    """FlatModel of a workload of radiative3d_b200.workloads.CONFIGS at the given TOA degree (scatterer tables built on
    CUDA device `device`)."""
    from . import engine
    z = np.load(os.path.join(GOLDEN, f"golden_{config}.npz"))
    f, i = z["scalars_f"], z["scalars_i"]
    m = FlatModel(freq_hz=float(f[0]), ttl=float(f[1]), bin_dt=float(f[2]), earth_center=tuple(map(float, f[3:6])),
                  min_theta=float(f[6]), max_theta=float(f[7]), slow_concern=float(f[8]), src_loc=tuple(map(float, f[9:12])),
                  cyl_radius2=float(f[12]), loop_concern=int(i[0]), n_bins=int(i[1]), ecs_radial=int(i[2]),
                  no_deflect=int(i[3]), src_cell=int(i[4]), cell_kind=int(i[5]))
    for name, dt in _ARRAYS:
        setattr(m, name, np.ascontiguousarray(z[name], dtype=dt))
    m.toa_theta, m.toa_phi = toa_set(toa_degree)
    strike, dip, rake = (float(v) for v in workloads.CONFIGS[config]["source"].split(",")[1:4])
    m.src_whole_cdf, m.src_cdf = source_tables(strike, dip, rake, m.toa_theta, m.toa_phi)
    cdf, spol, whole, mfp = engine.build_scatterer_tables(np.load(os.path.join(GOLDEN, "scat_params.npz"))[config],
                                                          m.toa_theta, m.toa_phi, device)
    m.scat_cdf, m.scat_spol, m.scat_whole_cdf, m.scat_mfp = cdf.ravel(), spol.ravel(), whole.ravel(), mfp.ravel()
    return m.validate()
