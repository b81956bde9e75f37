"""GPU sub-kernels (through the C ABI's r3d_test_* hooks) against the reference golden vectors and the oracle.

Bar (BASELINE.json north_star): deterministic sub-kernels within 1e-10 relative of the reference's
double-precision results; cell / face / table indices bit-exact.
"""
import numpy as np
import pytest

import oracle_binding as ob
import seis_layouts
from conftest import CONFIGS, GOLDEN, load_golden, rel_err
from radiative3d_b200 import abi, engine

pytestmark = pytest.mark.gpu
TOL = 1e-10


@pytest.fixture(scope="module")
def free():
    return np.load(f"{GOLDEN}/golden_free.npz")


def test_transform(free):
    """Golden Transform vectors.  The reference ends Transform with theta' = acos(cos theta') (geom_r3.cpp:261), whose
    absolute error is ~eps / sin(theta'): next to a pole that exceeds 1e-10 and it is the REFERENCE's value that is
    off (the device keeps the frame as vectors).  So: compare the direction and polarisation VECTORS, with the
    tolerance widened by that conditioning term."""
    out = engine.transform(free["transform_in"])
    ref = free["transform_out"]

    def frame(a):
        st, ct, sp, cp, sr, cr = np.sin(a[:, 0]), np.cos(a[:, 0]), np.sin(a[:, 1]), np.cos(a[:, 1]), np.sin(a[:, 2]), np.cos(a[:, 2])
        return (np.stack([st * cp, st * sp, ct], 1), np.stack([cr * ct * cp - sr * sp, cr * ct * sp + sr * cp, -cr * st], 1))

    (e3a, s1a), (e3b, s1b) = frame(out), frame(ref)
    tol = TOL + 16 * np.finfo(float).eps / np.maximum(np.sin(ref[:, 0]), 1e-12)
    assert (np.abs(e3a - e3b).max(axis=1) <= tol).all()
    assert (np.abs(s1a - s1b).max(axis=1) <= tol).all()
    assert (tol <= TOL * 1.01).mean() > 0.95           # the widening only touches the few near-pole cases


def test_transform_random_vs_oracle():
    rng = np.random.default_rng(1)
    n = 200000
    x = np.stack([np.arccos(rng.uniform(-1, 1, n)), rng.uniform(-np.pi, np.pi, n), rng.uniform(-np.pi, np.pi, n),
                  np.arccos(rng.uniform(-1, 1, n)), rng.uniform(-np.pi, np.pi, n), rng.uniform(-np.pi, np.pi, n)], axis=1)
    out, ref = engine.transform(x), ob.transform(x)
    # compare the frames, not the angle charts (phi / pol are ill-conditioned next to the poles)
    def frame(a):
        st, ct, sp, cp, sr, cr = np.sin(a[:, 0]), np.cos(a[:, 0]), np.sin(a[:, 1]), np.cos(a[:, 1]), np.sin(a[:, 2]), np.cos(a[:, 2])
        e3 = np.stack([st * cp, st * sp, ct], 1)
        s1 = np.stack([cr * ct * cp - sr * sp, cr * ct * sp + sr * cp, -cr * st], 1)
        return e3, s1
    (e3a, s1a), (e3b, s1b) = frame(out), frame(ref)
    assert np.abs(e3a - e3b).max() <= TOL and np.abs(s1a - s1b).max() <= TOL


def test_rtcoef(free):
    out = engine.rtcoef(free["rtcoef_in"])
    ref = free["rtcoef_out"]
    assert np.array_equal(out[:, 6], ref[:, 6])
    scale = np.abs(ref[:, :6]).max(axis=1, keepdims=True)
    assert (np.abs(out[:, :6] - ref[:, :6]) / scale).max() <= TOL
    assert np.abs(out[:, 7:] - ref[:, 7:]).max() <= TOL


def test_rtcoef_builtin_table(free):
    t = free["rtcoef_test_table"]
    x = np.zeros((t.shape[0], 15))
    x[:, 2] = 1.0
    x[:, 3], x[:, 5] = np.sin(t[:, 1]), np.cos(t[:, 1])
    x[:, 6:12] = [10, 8, 4, 8, 4, 2]
    x[:, 12] = t[:, 0]
    x[:, 14] = 12345
    out = engine.rtcoef(x)
    ref = t[:, [3, 5, 7, 4, 6, 8]]
    scale = np.maximum(np.abs(ref).max(axis=1, keepdims=True), 1e-300)
    assert (np.abs(out[:, :6] - ref) / scale).max() <= TOL


def check_travel(out, ref, x, kind):
    """TravelRec comparison.  Lengths / positions are compared on the scale of the geometry (a phonon sitting on a
    face has a path length of ~1e-12 km that is pure cancellation noise), travel time and attenuation likewise on
    the scale of the cell.  Tetra rays that run (anti)parallel to the velocity gradient have arc radii of ~1e10 km
    and the reference's own arc-length difference keeps only ~6 digits there, so those rows get 1e-5."""
    ok = np.isfinite(ref[:, 0])
    assert np.array_equal(np.isfinite(out[:, 0]), ok)
    out, ref, x = out[ok], ref[ok], x[ok]
    L = max(1.0, np.abs(ref[:, 2:5]).max())                       # geometry scale, km
    tol_len = np.full(ref.shape[0], TOL * L)
    if kind == abi.R3D_CELL_TETRA:
        steep = np.minimum(x[:, 5], np.pi - x[:, 5]) < 1e-3        # nearly vertical = nearly along the gradient
        tol_len[steep] = 1e-5 * L
    # per-row speed (the fluid outer core carries S at 1e-5 km/s, so the same length error is a large time error)
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.where(ref[:, 1] > 1e-9, ref[:, 0] / ref[:, 1], np.inf)
    v = np.where(np.isfinite(v) & (v > 0), v, 1.0)
    tol_time = tol_len / v + 1e-9 * np.abs(ref[:, 1])
    assert (np.abs(out[:, 0] - ref[:, 0]) <= tol_len + 1e-9 * np.abs(ref[:, 0])).all()
    assert (np.abs(out[:, 1] - ref[:, 1]) <= tol_time).all()
    assert (np.abs(out[:, 2:5] - ref[:, 2:5]).max(axis=1) <= tol_len).all()
    # direction: compare unit vectors (theta, phi chart is singular at the poles)
    def unit(a):
        return np.stack([np.sin(a[:, 5]) * np.cos(a[:, 6]), np.sin(a[:, 5]) * np.sin(a[:, 6]), np.cos(a[:, 5])], 1)
    assert (np.abs(unit(out) - unit(ref)).max(axis=1) <= tol_len / L + 1e-10).all()
    # attenuation = exp(-pi f t / Q): |d atten| <= (pi f / Q) |dt| < |dt| for every model here
    assert (np.abs(out[:, 7] - ref[:, 7]) <= 1e-9 + tol_time).all()


@pytest.mark.parametrize("cfg", CONFIGS)
def test_path_and_advance(cfg):
    m, z = load_golden(cfg)
    with engine.Engine(m) as eng:
        out = eng.path_to_boundary(z["path_in"])
        assert np.array_equal(out[:, 8], z["path_out"][:, 8])      # exit face: bit-exact
        check_travel(out, z["path_out"], z["path_in"], m.cell_kind)
        check_travel(eng.advance(z["advance_in"]), z["advance_out"], z["advance_in"], m.cell_kind)


@pytest.mark.parametrize("cfg", CONFIGS)
@pytest.mark.parametrize("guide", [0, 1, 3])
def test_cdf_search_golden(cfg, guide):
    m, z = load_golden(cfg)
    nt = m.n_toa
    for which in range(9):
        rows = z["cdf_cases"][z["cdf_cases"][:, 0] == which]
        if which < 4:
            cdf = m.scat_cdf[which * nt:(which + 1) * nt]
        elif which < 6:
            cdf = m.scat_whole_cdf[(which - 4) * 4:(which - 3) * 4]
        else:
            cdf = m.src_cdf[(which - 6) * nt:(which - 5) * nt]
        out = engine.cdf_search(cdf, rows[:, 1].astype(np.uint32), guide)
        assert np.array_equal(out, rows[:, 2].astype(np.uint32)), (which, guide)


@pytest.mark.parametrize("n", [17, 1000, 5242880])
def test_cdf_search_full_size_vs_oracle(n):
    """Guide-table search == reference bisection on a table of the scripted size (TOA degree 9), incl. plateaus."""
    rng = np.random.default_rng(n)
    w = rng.random(n) ** 8                     # strongly non-uniform weights
    w[rng.integers(0, n, n // 10)] = 0.0       # zero-probability entries -> flat stretches in the CDF
    cdf = np.cumsum(w)
    k = np.concatenate([rng.integers(0, 2**31, 300000, dtype=np.uint32), np.array([0, 1, 2**31 - 1, 2**31 - 2, 2**30], dtype=np.uint32)])
    ref = ob.cdf_search(cdf, k)
    for guide in (0, 1, 8, 20):
        assert np.array_equal(engine.cdf_search(cdf, k, guide), ref), guide


@pytest.mark.parametrize("cfg", CONFIGS)
def test_catch(cfg):
    m, z = load_golden(cfg)
    out = engine.catch(m.bin_dt, m.n_bins, z["catch_in"])
    ref = ob.catch(m.bin_dt, m.n_bins, z["catch_in"])            # oracle == golden (test_oracle_golden), exact energies
    assert np.array_equal(out[:, :2], ref[:, :2])
    assert np.array_equal(out[:, :2], z["catch_out"][:, :2])
    assert rel_err(out[:, 2:], ref[:, 2:]).max() <= TOL
    # the annulus branch (r_in > 0, no shift), which no golden station has, and the radius and bin edges
    rows, want = seis_layouts.catch_edge_rows(m, z["catch_in"])
    out = engine.catch(m.bin_dt, m.n_bins, rows)
    ref = ob.catch(m.bin_dt, m.n_bins, rows)
    assert np.array_equal(out[:, :2], ref[:, :2])
    edge = want >= 0
    assert np.array_equal(out[edge, 0], want[edge])
    assert np.array_equal(out[:, 5], ref[:, 5])
    assert rel_err(out[:, 2:5], ref[:, 2:5]).max() <= TOL


def test_branch_free_arithmetic():
    """qdiv / qsqrt0 (r3d_device.cuh) are the compiler's own fast paths without the range tests: bit-identical to a / b and
    sqrt(a) over the operand range of a phonon event (and far beyond it), including zero numerators, zero radicands and NaN."""
    rng = np.random.default_rng(7)
    n = 2_000_000
    a = rng.standard_normal(n) * 10.0 ** rng.uniform(-60, 60, n)
    b = rng.standard_normal(n) * 10.0 ** rng.uniform(-60, 60, n)
    a[:1000] = 0.0                                   # 0 / b
    a[1000:2000] = rng.uniform(0, 1, 1000)           # direction cosines over lengths
    b[1000:2000] = rng.uniform(1e-7, 1, 1000)
    a[2000:2010] = np.nan
    b[2010:2020] = np.nan
    a[2020:3020] = -0.0
    b[b == 0] = 1.0
    out = engine.arith(np.stack([a, b], axis=1))
    q, q_ref, r, r_ref = out[:, 0], out[:, 1], out[:, 2], out[:, 3]
    same_q = (q.view(np.uint64) == q_ref.view(np.uint64)) | (np.isnan(q) & np.isnan(q_ref)) | ((q == 0) & (q_ref == 0))   # (+0 for -0: documented)
    assert same_q.all(), f"{(~same_q).sum()} quotients differ, e.g. {a[~same_q][:3]} / {b[~same_q][:3]}"
    same_r = (r.view(np.uint64) == r_ref.view(np.uint64)) | (np.isnan(r) & np.isnan(r_ref))
    assert same_r.all(), f"{(~same_r).sum()} roots differ, e.g. {a[~same_r][:3]}"


def test_path_length_log():
    """The kernel's -log(r) of the path-length draw against the math library's, for draws over the whole range, the smallest
    ones (r next to 1: short paths, where only a relative bound means anything) and the largest."""
    rng = np.random.default_rng(11)
    k = np.concatenate([rng.integers(0, 2**31, 1_000_000), np.arange(0, 5000), 2**31 - 1 - np.arange(0, 5000),
                        rng.integers(0, 2**12, 5000), (2**31 * (1 - 2.0 ** -rng.uniform(0, 30, 20000))).astype(np.int64)])
    out = engine.pathlog(k.astype(np.float64))
    mine, ref = out[:, 0], out[:, 1]
    assert np.all(mine[k == 0] == 0.0) and np.all(ref[k == 0] == 0.0)
    nz = k > 0
    assert (np.abs(mine[nz] - ref[nz]) / ref[nz]).max() <= 1e-13
