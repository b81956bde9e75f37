"""Energy snapshots on the device: the partial advance against the CPU restatement, the exact record-count invariant, the
grids against the CPU restatement, the ballistic case, and that snapshots leave the simulation unchanged."""
import numpy as np
import pytest

import oracle_binding as ob
import snapshot_oracle_binding as sb
from conftest import CONFIGS, load_golden
from radiative3d_b200 import abi, engine
from snapshot_cases import advance_time_rows, dt_tolerance, grid_around, time_resolved, times_of
from test_oracle_snapshots import ballistic_case, check_ballistic

pytestmark = pytest.mark.gpu
SEED = 777


def n_gpus():
    import torch
    return torch.cuda.device_count()


def counts_per_snapshot(c, oc):
    return c.reshape(c.shape[0], -1).sum(axis=1) + oc.sum(axis=1)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_advance_time_vs_oracle(cfg):
    m, z = load_golden(cfg)
    rows, _ = advance_time_rows(m, z)
    with engine.Engine(m) as eng:
        g = eng.advance_time(rows)
        ga = eng.advance(np.concatenate([rows[:, :7], g[:, :1]], axis=1))
    o = sb.advance_time(m, rows)
    ok = time_resolved(m, rows, o)
    assert ok.sum() >= 0.8 * len(rows)
    dt = rows[:, 7]
    assert np.all(np.abs(g[ok, 1] - dt[ok]) <= dt_tolerance(cfg) * dt[ok])
    scale = np.maximum(1.0, np.abs(o[:, 2:5]).max(axis=1))
    # (curved rays: the two sides' travel-time formulas agree to their resolution, so the lengths they invert to do too)
    tol = np.maximum(1e-10 * scale, 2 * dt_tolerance(cfg) * np.abs(o[:, 0]))
    assert np.all(np.abs(g[ok, 2:5] - o[ok, 2:5]).max(axis=1) <= tol[ok])
    assert np.all(np.abs(ga[:, 2:5] - g[:, 2:5]).max(axis=1) <= 1e-10 * scale)


def invariant(m, n, seed, t, origin, voxel, dims):
    with engine.Engine(m) as eng:
        eng.set_snapshots(t, origin, voxel, dims)
        eng.run_simulation(n, seed)
        e, c, oe, oc = eng.fetch_snapshots()
    with engine.Engine(m) as eng:
        fin = eng.trace(n, seed)
    alive = np.array([(fin["time"] > tk).sum() for tk in t], dtype=np.uint64)
    per_k = counts_per_snapshot(c, oc)
    assert np.array_equal(per_k, alive), (per_k, alive)
    assert np.all(e >= 0) and np.all(oe >= 0)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_record_count_invariant(cfg):
    m, _ = load_golden(cfg)
    origin, voxel, dims = grid_around(m)
    invariant(m, 200000, SEED, times_of(m), origin, voxel, dims)


def test_record_count_invariant_benchmark_model():
    from radiative3d_b200 import workload_model
    m = workload_model.build_model("halfspace_nearsrc50", 9)
    origin, voxel, dims = grid_around(m, (32, 32, 32))
    invariant(m, 1000000, SEED, np.linspace(0, m.ttl, 16), origin, voxel, dims)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_grids_vs_oracle(cfg):
    m, _ = load_golden(cfg)
    n = 500 if cfg == "spherical" else 3000
    t = times_of(m)
    origin, voxel, dims = grid_around(m)
    with engine.Engine(m) as eng:
        eng.set_snapshots(t, origin, voxel, dims)
        eng.run_simulation(n, SEED)
        e, c, oe, oc = eng.fetch_snapshots()
    with engine.Engine(m) as eng:
        fin = eng.trace(n, SEED)
    e_o, c_o, oe_o, oc_o, fin_o = sb.run(m, 0, n, SEED, t, origin, voxel, dims, finals=True)
    same = np.ones(n, dtype=bool)
    for f in ("moves", "cell", "type", "fate", "draws"):
        same &= fin[f] == fin_o[f]
    same &= np.abs(fin["time"] - fin_o["time"]) <= 1e-8 * np.maximum(1.0, np.abs(fin_o["time"]))
    D = int((~same).sum())
    if cfg == "halfspace":
        assert D == 0
        assert np.array_equal(c, c_o) and np.array_equal(oc, oc_o)
        np.testing.assert_allclose(e, e_o, rtol=1e-10, atol=1e-300)
        np.testing.assert_allclose(oe, oe_o, rtol=1e-10, atol=1e-300)
    else:
        a, b = counts_per_snapshot(c, oc).astype(np.int64), counts_per_snapshot(c_o, oc_o).astype(np.int64)
        assert np.all(np.abs(a - b) <= D), (a, b, D)
        l1 = np.abs(c.astype(np.int64) - c_o.astype(np.int64)).sum() + np.abs(oc.astype(np.int64) - oc_o.astype(np.int64)).sum()
        assert l1 <= 2 * len(t) * D + 1e-4 * b.sum(), (l1, D)


def test_ballistic_on_device():
    m, _ = load_golden("halfspace")
    m, c, times, origin, voxel, dims = ballistic_case(m)
    n = 10000000
    with engine.Engine(m) as eng:
        eng.set_snapshots(times, origin, voxel, dims)
        eng.run_simulation(n, SEED)
        e, cnt, oe, oc = eng.fetch_snapshots()
        k = eng.fetch()[2]
    assert int(k[abi.R3D_CNT_SCATTERS]) == 0
    check_ballistic(m, c, times, origin, voxel, dims, e, cnt, oe, oc, n)


@pytest.mark.parametrize("cfg", ["halfspace", "crustpinch"])
def test_snapshots_leave_the_simulation_unchanged(cfg):
    m, _ = load_golden(cfg)
    n = 9000000 if cfg == "halfspace" else 500000        # halfspace: past the pilot launches of a first large job
    origin, voxel, dims = grid_around(m)
    with engine.Engine(m) as eng:
        eng.run_simulation(n, SEED)
        e0, c0, k0 = eng.fetch()
    with engine.Engine(m) as eng:
        eng.set_snapshots(times_of(m), origin, voxel, dims)
        eng.run_simulation(n, SEED)
        e1, c1, k1 = eng.fetch()
    assert np.array_equal(c0, c1) and np.array_equal(k0, k1)
    np.testing.assert_allclose(e1, e0, rtol=1e-12, atol=1e-300)


def test_additivity_reset_and_off():
    m, _ = load_golden("lopnor")
    n = 400000
    t = times_of(m)
    origin, voxel, dims = grid_around(m)
    with engine.Engine(m) as eng:
        eng.set_snapshots(t, origin, voxel, dims)
        eng.run_simulation(n, SEED)
        whole = eng.fetch_snapshots()
        eng.reset()
        z = eng.fetch_snapshots()
        assert all(not np.any(a) for a in z)
        eng.run_simulation(n // 2, SEED)
        eng.run_simulation(n - n // 2, SEED, first_phonon=n // 2)
        parts = eng.fetch_snapshots()
        assert np.array_equal(whole[1], parts[1]) and np.array_equal(whole[3], parts[3])
        np.testing.assert_allclose(parts[0], whole[0], rtol=1e-12, atol=1e-300)
        np.testing.assert_allclose(parts[2], whole[2], rtol=1e-12, atol=1e-300)
        eng.set_snapshots(None)
        with pytest.raises(engine.R3DError):
            eng.fetch_snapshots()
        eng.reset()
        eng.run_simulation(n, SEED)
        e_off, c_off, k_off = eng.fetch()
    with engine.Engine(m) as eng:
        eng.run_simulation(n, SEED)
        e_ref, c_ref, k_ref = eng.fetch()
    assert np.array_equal(c_off, c_ref) and np.array_equal(k_off, k_ref)
    np.testing.assert_allclose(e_off, e_ref, rtol=1e-12, atol=1e-300)


def test_rejections():
    m, _ = load_golden("halfspace")
    origin, voxel, dims = grid_around(m)
    t = times_of(m)
    bad = [
        (t[::-1], origin, voxel, dims), (np.array([1.0, 1.0]), origin, voxel, dims), (np.array([-1.0, 1.0]), origin, voxel, dims),
        (np.array([1.0, m.ttl * 1.01]), origin, voxel, dims), (np.array([1.0, np.nan]), origin, voxel, dims),
        (np.array([1.0, np.inf]), origin, voxel, dims), (np.linspace(0, m.ttl, 65), origin, voxel, dims),
        (t, origin, (0.0, 1.0, 1.0), dims), (t, origin, (1.0, -1.0, 1.0), dims), (t, origin, (1.0, 1.0, np.inf), dims),
        (t, origin, (1.0, 1.0, np.nan), dims), (t, (np.nan, 0.0, 0.0), voxel, dims), (t, origin, voxel, (0, 8, 8)),
        (t, origin, voxel, (8, 8, 0)), (t, origin, voxel, (1024, 1024, 1024)),
        (t, origin, voxel, (4294967295, 4294967295, 4294967295)),
    ]
    with engine.Engine(m) as eng:
        for args in bad:
            with pytest.raises(engine.R3DError) as ei:
                eng.set_snapshots(*args)
            assert ei.value.code == abi.R3D_EINVAL, args
            assert sb.check(m, *args) == abi.R3D_EINVAL
        eng.set_snapshots(np.linspace(0, m.ttl, 64), origin, voxel, dims)
        eng.run_simulation(1000, SEED)
        assert eng.fetch_snapshots()[1].shape == (64, dims[2], dims[1], dims[0], 2)


def test_two_devices_equal_one():
    if n_gpus() < 2:
        pytest.skip("needs two GPUs")
    m, _ = load_golden("crustpinch")
    n = 300000
    t = times_of(m)
    origin, voxel, dims = grid_around(m)
    out = []
    for devs in ((0,), (0, 1)):
        with engine.Engine(m, devices=devs) as eng:
            eng.set_snapshots(t, origin, voxel, dims)
            eng.run_simulation(n, SEED)
            out.append(eng.fetch_snapshots())
    (e1, c1, oe1, oc1), (e2, c2, oe2, oc2) = out
    assert np.array_equal(c1, c2) and np.array_equal(oc1, oc2)
    np.testing.assert_allclose(e2, e1, rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(oe2, oe1, rtol=1e-12, atol=1e-300)
