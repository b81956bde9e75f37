"""The catch log (r3d_set_catch_log) and replay by index (r3d_trace_indices, r3d_trace_events_indices) on the device: the
log against the bins, counters and the oracle, its filters, its independence of how a range is split, pilots and
snapshots, that it changes nothing else, and that replaying the logged phonons gives back their catches."""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import CONFIGS, load_golden
from radiative3d_b200 import abi, engine
from snapshot_cases import grid_around

pytestmark = pytest.mark.gpu
SEED = 777
U = 2.0 ** -53


def n_gpus():
    import torch
    return torch.cuda.device_count()


def logged_run(m, n, seed=SEED, seismometers=None, bins=None, capacity=1 << 24, devices=(0,), snapshots=None, parts=None):
    """(records, n_matched, (energies, counts, counters), snapshots or None) of one engine that logs while it runs [0, n),
    in one call or in the calls `parts` = [(first, count), ...]."""
    with engine.Engine(m, devices=devices) as eng:
        eng.set_catch_log(seismometers, bins, capacity)
        if snapshots is not None:
            eng.set_snapshots(*snapshots)
        for first, count in (parts or [(0, n)]):
            eng.run_simulation(count, seed, first_phonon=first)
        rec, matched = eng.fetch_catch_log()
        bins_out = eng.fetch()
        snap = eng.fetch_snapshots() if snapshots is not None else None
    return rec, matched, bins_out, snap


def plain_run(m, n, seed=SEED, snapshots=None):
    with engine.Engine(m) as eng:
        if snapshots is not None:
            eng.set_snapshots(*snapshots)
        eng.run_simulation(n, seed)
        out = eng.fetch()
        snap = eng.fetch_snapshots() if snapshots is not None else None
    return out, snap


def same_rows(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def keys_strictly_increasing(r):
    p, mv, s = r["phonon"], r["moves"], r["seis"]
    gt = (p[1:] > p[:-1]) | ((p[1:] == p[:-1]) & ((mv[1:] > mv[:-1]) | ((mv[1:] == mv[:-1]) & (s[1:] > s[:-1]))))
    return bool(np.all(gt))


def log_sums(m, r):
    """Per (seis, bin): record counts by type [.., 2], the energies summed in extended precision [.., 5] and the sums of
    their magnitudes, laid out as the bins."""
    c = np.zeros((m.n_seis, m.n_bins, 2), dtype=np.uint64)
    e = np.zeros((m.n_seis, m.n_bins, 5), dtype=np.longdouble)
    a = np.zeros((m.n_seis, m.n_bins, 5), dtype=np.longdouble)
    s, b, t = r["seis"].astype(np.intp), r["bin"].astype(np.intp), r["type"].astype(np.intp)
    np.add.at(c, (s, b, t), 1)
    for ch in range(3):
        np.add.at(e, (s, b, np.full_like(s, ch)), r["energy"][:, ch].astype(np.longdouble))
        np.add.at(a, (s, b, np.full_like(s, ch)), np.abs(r["energy"][:, ch]).astype(np.longdouble))
    np.add.at(e, (s, b, 3 + t), r["energy"][:, 3].astype(np.longdouble))
    np.add.at(a, (s, b, 3 + t), np.abs(r["energy"][:, 3]).astype(np.longdouble))
    return c, e, a


def assert_energies_within_rounding(e_bins, e_log, a_log, n_add):
    """|bin - exact sum of its addends| <= n 2^-53 sum |addends| (the sum in extended precision adds n 2^-63 of slack)."""
    bound = n_add.astype(np.longdouble) * np.longdouble(U + 2.0 ** -63) * a_log
    err = np.abs(e_bins.astype(np.longdouble) - e_log)
    assert np.all(err <= bound), float((err - bound).max())


def assert_log_equals_bins(m, rec, matched, bins_out):
    e, c, k = bins_out
    assert matched == rec.size == int(k[abi.R3D_CNT_CATCHES])
    cl, el, al = log_sums(m, rec)
    assert np.array_equal(cl, c)
    n_add = np.repeat(c.sum(axis=-1, keepdims=True), 5, axis=-1)
    assert_energies_within_rounding(e, el, al, n_add)
    assert keys_strictly_increasing(rec)


# ---- 1. the log holds exactly the catches the bins hold ----------------------------------------------------------------
@pytest.mark.parametrize("cfg", CONFIGS)
def test_log_equals_bins(cfg):
    m, _ = load_golden(cfg)
    rec, matched, out, _ = logged_run(m, 200000)
    assert rec.size > 0
    assert_log_equals_bins(m, rec, matched, out)


# ---- 2. records per phonon against the oracle's catches ---------------------------------------------------------------
@pytest.mark.parametrize("cfg", CONFIGS)
def test_records_per_phonon_equal_oracle(cfg):
    m, z = load_golden(cfg)
    n, seed = int(z["run_n"]), int(z["run_seed"])
    _, _, _, f_ref = ob.run(m, 0, n, seed, finals=True, nthreads=4)
    with engine.Engine(m) as eng:
        fin = eng.trace(n, seed)
    same = np.ones(n, dtype=bool)
    for f in ("moves", "cell", "type", "fate", "draws"):
        same &= fin[f] == f_ref[f]
    assert same.mean() >= 0.995
    rec, matched, _, _ = logged_run(m, n, seed)
    per = np.bincount(rec["phonon"].astype(np.intp), minlength=n)
    assert per.size == n and matched == rec.size
    assert per.sum() > 0
    bad = np.flatnonzero(same & (per != f_ref["catches"]))
    assert bad.size == 0, [(int(i), int(per[i]), int(f_ref["catches"][i]), int(fin["fate"][i])) for i in bad[:10]]


# ---- 3. filters: exactly the matching rows of the full log ------------------------------------------------------------
@pytest.mark.parametrize("cfg", ["lopnor", "halfspace"])
def test_filters_select_rows_of_the_full_log(cfg):
    m, _ = load_golden(cfg)
    n = 200000
    full, _, _, _ = logged_run(m, n)
    sel = np.array([m.n_seis - 1, 0, m.n_seis // 2], dtype=np.uint32)
    lo, hi = m.n_bins // 5, (4 * m.n_bins) // 5
    rec, matched, _, _ = logged_run(m, n, seismometers=sel, bins=(lo, hi))
    want = full[np.isin(full["seis"], sel) & (full["bin"] >= lo) & (full["bin"] < hi)]
    assert want.size > 0 and matched == want.size
    assert same_rows(rec, want)
    # a window nothing falls into
    empty_bins = np.setdiff1d(np.arange(m.n_bins), full["bin"])
    assert empty_bins.size > 0
    b = int(empty_bins[0])
    rec, matched, _, _ = logged_run(m, n, bins=(b, b + 1))
    assert rec.size == 0 and matched == 0


# ---- 4. independent of how the range is split, and of the devices -----------------------------------------------------
def test_split_runs_give_the_same_log():
    m, _ = load_golden("crustpinch")
    n = 300000                       # below the pilot threshold: every launch runs the same build
    whole, mw, _, _ = logged_run(m, n)
    parts = [(0, 1), (1, 123457), (123458, n - 123458)]
    split, ms, _, _ = logged_run(m, n, parts=parts)
    assert whole.size > 0 and mw == ms
    assert same_rows(whole, split)


def test_two_devices_equal_one():
    if n_gpus() < 2:
        pytest.skip("needs two GPUs")
    m, _ = load_golden("crustpinch")
    n = 300000
    one, m1, _, _ = logged_run(m, n)
    two, m2, _, _ = logged_run(m, n, devices=(0, 1))
    assert m1 == m2 and same_rows(one, two)


# ---- 5. the pilot launches of a large first job, with snapshots on ----------------------------------------------------
def test_pilots_and_snapshots_benchmark_model():
    from radiative3d_b200 import workload_model
    m = workload_model.build_model("halfspace_nearsrc50", 9)
    n = 10000000                     # >= the pilot threshold (8e6): two pilot launches, then the chosen build
    origin, voxel, dims = grid_around(m, (32, 32, 32))
    snaps = (np.linspace(0, m.ttl, 16), origin, voxel, dims)
    rec, matched, out, sn = logged_run(m, n, snapshots=snaps)
    assert rec.size > 0
    assert_log_equals_bins(m, rec, matched, out)
    _, sn0 = plain_run(m, n, snapshots=snaps)
    for a, b in zip(sn, sn0):
        if a.dtype == np.uint64:
            assert np.array_equal(a, b)
        else:
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-300)
    rec_ns, matched_ns, _, _ = logged_run(m, n)
    assert matched_ns == matched and same_rows(rec_ns, rec)


# ---- 6. no side effects; overflow, reset, off, rejections -------------------------------------------------------------
@pytest.mark.parametrize("cfg", ["halfspace", "crustpinch"])
def test_log_leaves_the_simulation_unchanged(cfg):
    m, _ = load_golden(cfg)
    n = 9000000 if cfg == "halfspace" else 500000        # halfspace: past the pilot launches of a first large job
    (e0, c0, k0), _ = plain_run(m, n)
    rec, _, (e1, c1, k1), _ = logged_run(m, n)
    assert rec.size > 0
    assert np.array_equal(c0, c1) and np.array_equal(k0, k1)
    np.testing.assert_allclose(e1, e0, rtol=1e-12, atol=1e-300)


def test_overflow_keeps_a_subset_and_counts_all():
    m, _ = load_golden("lopnor")
    n = 200000
    full, mf, _, _ = logged_run(m, n)
    assert full.size == mf and mf > 1000
    with pytest.warns(RuntimeWarning):
        rec, matched, _, _ = logged_run(m, n, capacity=100)
    assert matched == mf and rec.size == 100
    assert keys_strictly_increasing(rec)
    v = np.dtype((np.void, abi.CATCH_DTYPE.itemsize))
    assert np.all(np.isin(rec.view(v), full.view(v)))


def test_reset_off_and_rejections():
    m, _ = load_golden("lopnor")
    n = 100000
    with engine.Engine(m) as eng:
        with pytest.raises(engine.R3DError) as ei:
            eng.fetch_catch_log()                                   # never set
        assert ei.value.code == abi.R3D_EINVAL
        bad = [
            dict(seismometers=[m.n_seis]), dict(seismometers=[3, 5, 3]), dict(bins=(5, 5)), dict(bins=(7, 6)),
            dict(bins=(0, m.n_bins + 1)), dict(capacity=0), dict(capacity=abi.R3D_CATCH_LOG_MAX + 1),
        ]
        for kw in bad:
            with pytest.raises(engine.R3DError) as ei:
                eng.set_catch_log(**kw)
            assert ei.value.code == abi.R3D_EINVAL, kw
        eng.set_catch_log(capacity=abi.R3D_CATCH_LOG_MAX // 64)   # the cap is bounded, not the only size accepted
        eng.set_catch_log()
        eng.run_simulation(n, SEED)
        first, mf = eng.fetch_catch_log()
        assert mf == first.size > 0
        eng.reset()
        z, mz = eng.fetch_catch_log()
        assert z.size == 0 and mz == 0
        eng.run_simulation(n, SEED)
        again, ma = eng.fetch_catch_log()
        assert same_rows(again, first) and ma == mf
        eng.set_catch_log(capacity=None)
        with pytest.raises(engine.R3DError) as ei:
            eng.fetch_catch_log()
        assert ei.value.code == abi.R3D_EINVAL
        eng.reset()
        eng.run_simulation(n, SEED)
        e_off, c_off, k_off = eng.fetch()
    (e_ref, c_ref, k_ref), _ = plain_run(m, n)
    assert np.array_equal(c_off, c_ref) and np.array_equal(k_off, k_ref)
    np.testing.assert_allclose(e_off, e_ref, rtol=1e-12, atol=1e-300)


# ---- 7. replay by index = the range trace at those indices ------------------------------------------------------------
@pytest.mark.parametrize("cfg", CONFIGS)
def test_replay_equals_range_trace(cfg):
    m, _ = load_golden(cfg)
    n = 2000 if cfg == "spherical" else 20000
    rng = np.random.default_rng(5)
    idx = np.sort(rng.choice(n, size=n // 7, replace=False)).astype(np.uint64)
    with engine.Engine(m) as eng:
        fin = eng.trace(n, SEED)
        ev = eng.trace_events(n, SEED)
        fin_i = eng.trace_indices(idx, SEED)
        ev_i = eng.trace_events_indices(idx, SEED)
        assert same_rows(fin_i, fin[idx.astype(np.intp)])
        assert same_rows(ev_i, ev[np.isin(ev["phonon"], idx)])
        for bad in ([5, 3], [2, 2], [0, 7, 7, 9]):
            with pytest.raises(engine.R3DError) as ei:
                eng.trace_indices(bad, SEED)
            assert ei.value.code == abi.R3D_EINVAL
            with pytest.raises(engine.R3DError) as ei:
                eng.trace_events_indices(bad, SEED)
            assert ei.value.code == abi.R3D_EINVAL
        assert eng.trace_indices([], SEED).size == 0 and eng.trace_events_indices([], SEED).size == 0


# ---- 8. the log joins the replay ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", CONFIGS)
def test_log_joins_replay(cfg):
    m, _ = load_golden(cfg)
    n = 2000 if cfg == "spherical" else 20000
    with engine.Engine(m) as eng:
        eng.set_catch_log()
        eng.run_simulation(n, SEED)
        rec, matched = eng.fetch_catch_log()
        assert rec.size == matched > 0
        ph, per = np.unique(rec["phonon"], return_counts=True)
        # replay the logged phonons: their COL reports and end states, then their bins alone
        fin = eng.trace_indices(ph, SEED)
        col = eng.trace_events_indices(ph, SEED, kinds=1 << abi.R3D_EV_COL)
        eng.reset()
        eng.trace_indices(ph, SEED)
        e, c, _ = eng.fetch()
        none, n_none = eng.fetch_catch_log()
    assert none.size == 0 and n_none == 0                  # replays make no records
    fate = dict(zip(ph.tolist(), fin["fate"].tolist()))
    arrivals = {(int(p), int(mv)): t for p, mv, t in zip(col["phonon"], col["moves"], col["time"])}
    missing = [(int(r["phonon"]), int(r["moves"]), fate[int(r["phonon"])]) for r in rec
               if arrivals.get((int(r["phonon"]), int(r["moves"]))) != r["time"]]
    assert not missing, f"records without a COL report of the same move and time (phonon, moves, fate): {missing[:10]}"
    bad = np.flatnonzero(fin["catches"] != per)
    assert bad.size == 0, [(int(ph[i]), int(per[i]), int(fin["catches"][i]), int(fin["fate"][i])) for i in bad[:10]]
    # the replay's bins hold exactly the logged catches (the log selects everything)
    cl, el, al = log_sums(m, rec)
    assert np.array_equal(c, cl)
    n_add = np.repeat(c.sum(axis=-1, keepdims=True), 5, axis=-1)
    assert_energies_within_rounding(e, el, al, n_add)
