"""Energy snapshots on the CPU restatement (snapshot_oracle/): the exact record-count invariant, independence of how the
index range is split, the analytic ballistic case, and the argument checks of r3d_set_snapshots."""
import numpy as np
import pytest

import oracle_binding as ob
import snapshot_oracle_binding as sb
from conftest import CONFIGS, load_golden
from snapshot_cases import advance_time_rows, dt_tolerance, grid_around, time_resolved, times_of

SEED = 4242


def n_for(cfg):
    return 500 if cfg == "spherical" else 3000


@pytest.mark.parametrize("cfg", CONFIGS)
def test_record_count_invariant(cfg):
    """Snapshot k holds exactly one record per phonon whose final time is > t_k (the moves tile [0, final time))."""
    m, _ = load_golden(cfg)
    n, t = n_for(cfg), times_of(m)
    origin, voxel, dims = grid_around(m)
    e, c, oe, oc, fin = sb.run(m, 0, n, SEED, t, origin, voxel, dims, finals=True)
    per_k = c.reshape(len(t), -1).sum(axis=1) + oc.sum(axis=1)
    alive = np.array([(fin["time"] > tk).sum() for tk in t], dtype=np.uint64)
    assert np.array_equal(per_k, alive), (per_k, alive)
    assert per_k[0] == n - int(((fin["moves"] == 0)).sum())       # t_0 = 0: every phonon that moved at all
    assert np.all(e >= 0) and np.all(oe >= 0)
    # the snapshot run traces the phonons exactly as r3d_oracle_run does
    _, _, _, fin_ref = ob.run(m, 0, n, SEED, finals=True)
    for f in ("time", "moves", "fate", "draws", "cell", "type"):
        assert np.array_equal(fin[f], fin_ref[f]), f


@pytest.mark.parametrize("cfg", CONFIGS)
def test_split_ranges_add_up(cfg):
    m, _ = load_golden(cfg)
    n, t = n_for(cfg), times_of(m)
    origin, voxel, dims = grid_around(m)
    e, c, oe, oc, _ = sb.run(m, 0, n, SEED, t, origin, voxel, dims)
    cut = n // 3
    e1, c1, oe1, oc1, _ = sb.run(m, 0, cut, SEED, t, origin, voxel, dims)
    e2, c2, oe2, oc2, _ = sb.run(m, cut, n - cut, SEED, t, origin, voxel, dims)
    assert np.array_equal(c, c1 + c2) and np.array_equal(oc, oc1 + oc2)
    np.testing.assert_allclose(e, e1 + e2, rtol=1e-12, atol=0)
    np.testing.assert_allclose(oe, oe1 + oe2, rtol=1e-12, atol=0)


def ballistic_case(m):
    """The halfspace model without scattering, and 6 snapshot times before the fastest phonon can reach the nearest face
    of the source cell (layered cells: top / bottom plane, side cylinder)."""
    m.scat_mfp = np.full_like(m.scat_mfp, 1e30)
    c = m.cell_params.reshape(m.n_cells, -1)[m.src_cell]
    src = np.asarray(m.src_loc)
    d_top = abs(np.dot(c[5:8], c[8:11] - src))
    d_bot = abs(np.dot(c[11:14], c[14:17] - src))
    d_side = np.sqrt(m.cyl_radius2) - np.hypot(src[0], src[1])
    t_face = min(d_top, d_bot, d_side) / max(c[0], c[1])
    times = t_face * np.array([0.0, 0.1, 0.3, 0.5, 0.7, 0.95])
    r = max(c[0], c[1]) * times[-1]
    voxel = np.full(3, r / 6.0)
    origin = src - 8 * voxel
    return m, c, times, origin, voxel, (16, 16, 16)


def check_ballistic(m, c, times, origin, voxel, dims, e, cnt, oe, oc, n):
    src = np.asarray(m.src_loc)
    tot = cnt.reshape(len(times), -1, 2).sum(axis=1) + oc
    assert np.all(tot.sum(axis=1) == n)                   # every phonon is alive and in its first move
    assert np.all(oc == 0)
    f, Q = m.freq_hz, c[3:5]
    for k, tk in enumerate(times):
        for ty in (0, 1):
            n_rec = float(cnt[k, ..., ty].sum())
            want = n_rec * np.exp(-2 * tk * np.pi * f / Q[ty])
            got = e[k, ..., ty].sum()
            # 1e-12, or the rounding bound of a sum of n_rec terms in any order (n eps: atomics on the device)
            assert abs(got - want) <= max(1e-12, n_rec * 2.3e-16) * max(want, 1e-300), (k, ty, got, want)
            # every occupied voxel is cut by the sphere of radius v t_k around the source
            r = c[ty] * tk
            for iz, iy, ix in np.argwhere(cnt[k, ..., ty] > 0):
                lo = origin + voxel * np.array([ix, iy, iz])
                hi = lo + voxel
                near = np.linalg.norm(np.maximum(np.maximum(lo - src, src - hi), 0))
                far = np.linalg.norm(np.maximum(np.abs(lo - src), np.abs(hi - src)))
                assert near - 1e-9 * (1 + r) <= r <= far + 1e-9 * (1 + r), (k, ty, ix, iy, iz)


def test_ballistic_halfspace():
    m, _ = load_golden("halfspace")
    m, c, times, origin, voxel, dims = ballistic_case(m)
    n = 3000
    e, cnt, oe, oc, fin = sb.run(m, 0, n, SEED, times, origin, voxel, dims, finals=True)
    assert int(fin["scatters"].sum()) == 0
    check_ballistic(m, c, times, origin, voxel, dims, e, cnt, oe, oc, n)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_advance_time_reaches_dt(cfg):
    """The oracle's partial advance lands on travel time dt (where the cell's time formula resolves it) and on the point
    that advance() gives at the returned length."""
    m, z = load_golden(cfg)
    rows, _ = advance_time_rows(m, z)
    out = sb.advance_time(m, rows)
    ok = time_resolved(m, rows, out)
    assert ok.sum() >= 0.8 * len(rows)
    dt = rows[:, 7]
    assert np.all(np.abs(out[ok, 1] - dt[ok]) <= dt_tolerance(cfg) * dt[ok])
    a = ob.advance(m, np.concatenate([rows[:, :7], out[:, :1]], axis=1))
    assert np.array_equal(a[:, 2:5], out[:, 2:5])


def test_argument_checks():
    m, _ = load_golden("halfspace")
    origin, voxel, dims = grid_around(m)
    t = times_of(m)
    assert sb.check(m, t, origin, voxel, dims) == 0
    bad = [
        (t[::-1], origin, voxel, dims),                                   # not increasing
        (np.array([1.0, 1.0]), origin, voxel, dims),                      # repeated
        (np.array([-1.0, 1.0]), origin, voxel, dims),                     # below 0
        (np.array([1.0, m.ttl * 1.01]), origin, voxel, dims),             # beyond ttl
        (np.array([1.0, np.nan]), origin, voxel, dims),
        (np.array([1.0, np.inf]), origin, voxel, dims),
        (np.linspace(0, m.ttl, 65), origin, voxel, dims),                 # K > 64
        (t, origin, (0.0, 1.0, 1.0), dims),
        (t, origin, (1.0, -1.0, 1.0), dims),
        (t, origin, (1.0, 1.0, np.inf), dims),
        (t, origin, (1.0, 1.0, np.nan), dims),
        (t, (np.nan, 0.0, 0.0), voxel, dims),
        (t, origin, voxel, (0, 8, 8)),
        (t, origin, voxel, (8, 8, 0)),
        (t, origin, voxel, (1024, 1024, 1024)),                           # beyond R3D_SNAP_MAX_CELLS
        (t, origin, voxel, (4294967295, 4294967295, 4294967295)),
    ]
    for args in bad:
        assert sb.check(m, *args) == 1, args
    with pytest.raises(ValueError):
        sb.run(m, 0, 10, SEED, t[::-1], origin, voxel, dims)
    assert sb.check(m, np.linspace(0, m.ttl, 64), origin, voxel, dims) == 0
