"""Seismometer collection (collect_warp, the grid of build_seis_grid, seis_catch) on adversarial station layouts
(tests/seis_layouts.py), at full occupancy (148 CTAs x 1504 slots ~ 2.2e5 phonons), held arrival by arrival to a
brute-force reference.

The reference decides every (arrival, station) pair from the kernel's own arrival states (the COL reports of a trace
over the same range) with the oracle's seis_catch.  The trajectories therefore drop out of the comparison: the kernel
and the oracle round the ray arithmetic differently, which at this size changes a few phonons' paths.  Only pairs that
lie on an edge to 1e-12 relative stay undecided; they are printed with their margins and bounded in number.
"""
import numpy as np
import pytest

import seis_layouts as sl
from conftest import CONFIGS, load_golden
from radiative3d_b200 import abi, engine
from test_gpu_catch_log import assert_energies_within_rounding, log_sums

pytestmark = pytest.mark.gpu
SEED = 4242
MAX_AMBIGUOUS = 10
EPS = np.finfo(np.float64).eps
LAYERED = ("halfspace", "halfspace_nearsrc50", "lopnor")
MAX_CELLS = 64 << 20


def n_phonons(cfg):
    """At least full occupancy; the halfspaces' small stations catch few arrivals, so they run more."""
    return 1_000_000 if cfg.startswith("halfspace") else 250_000


def void_keys(r):
    k = sl.keys(r)
    return k.view(np.dtype((np.void, k.dtype.itemsize)))


def logged(m, n, seed=SEED):
    """(catch log of every station and bin, (energies, counts, counters)) of r3d_run over [0, n)."""
    with engine.Engine(m) as eng:
        eng.set_catch_log(capacity=1 << 24)
        eng.run_simulation(n, seed)
        rec, matched = eng.fetch_catch_log()
        out = eng.fetch()
    assert matched == rec.size
    return rec, out


def col_events(m, n, seed=SEED, chunk=50_000, per_phonon=64):
    """(COL reports of [0, n), the trace's own bins).  Each chunk starts from zeroed bins, so one that overflows its
    `capacity` is traced again in halves; the chunks' bins are summed here (exact for counts)."""
    evs, e, c, k = [], 0.0, 0, 0
    todo = [(a, min(chunk, n - a)) for a in range(0, n, chunk)]
    with engine.Engine(m) as eng:
        while todo:
            a, cnt = todo.pop(0)
            eng.reset()
            try:
                ev = eng.trace_events(cnt, seed, first_phonon=a, kinds=1 << abi.R3D_EV_COL, capacity=per_phonon * cnt)
            except engine.R3DError:
                assert cnt > 1
                todo[:0] = [(a, cnt // 2), (a + cnt // 2, cnt - cnt // 2)]
                continue
            evs.append(ev)
            be, bc, bk = eng.fetch()
            e, c, k = e + be, c + bc, k + bk
    ev = np.concatenate(evs)
    assert np.all(ev["kind"] == abi.R3D_EV_COL)
    return ev, (e, c, k)


def compare_to_reference(m, rec, ev, trace_bins, label):
    """The checks of test_log_equals_reference; returns (compared catches, ambiguous pairs, coverage)."""
    ref, amb, cov = sl.reference_catches(m, ev)
    for a in amb:
        print(f"{label}: ambiguous phonon {int(a['phonon'])} move {int(a['moves'])} seis {int(a['seis'])}: margin {a['margin']:.3e}")
    assert amb.size <= MAX_AMBIGUOUS, f"{amb.size} ambiguous pairs"
    # every record joins a COL report of its phonon and move, at the same time to the bit
    ek, lk = np.zeros(ev.size, dtype=[("phonon", "<u8"), ("moves", "<u4")]), np.zeros(rec.size, dtype=[("phonon", "<u8"), ("moves", "<u4")])
    for f in ek.dtype.names:
        ek[f], lk[f] = ev[f], rec[f]
    order = np.argsort(ek, kind="stable")
    pos = np.searchsorted(ek[order], lk)
    pos = np.minimum(pos, ev.size - 1)
    hit = order[pos]
    joined = (ek[hit] == lk) & (ev["time"][hit].view(np.uint64) == rec["time"].view(np.uint64))
    assert np.all(joined), [(int(r["phonon"]), int(r["moves"]), float(r["time"])) for r in rec[~joined][:10]]
    # the log's keys = the reference's, apart from the ambiguous pairs
    keep = ~np.isin(void_keys(rec), void_keys(amb))
    got = rec[keep]
    assert got.size == ref.size, (got.size, ref.size)
    assert np.array_equal(void_keys(got), void_keys(ref))
    assert np.array_equal(got["bin"], ref["bin"]) and np.array_equal(got["type"], ref["type"])
    assert np.array_equal(got["time"].view(np.uint64), ref["time"].view(np.uint64))
    # energy[3] = exp(-aexp)^2 / bin_dt / area in the same order on both sides: bit-identical
    bad = np.flatnonzero(got["energy"][:, 3].view(np.uint64) != ref["energy"][:, 3].view(np.uint64))
    assert bad.size == 0, [(float(got["energy"][i, 3]), float(ref["energy"][i, 3])) for i in bad[:5]]
    e3 = got["energy"][:, 3]
    p = got["type"] == abi.R3D_RAY_P
    assert np.all(np.abs(got["energy"][p, :3] - ref["energy"][p, :3]) <= 1e-12 * e3[p, None])
    # S: the reference has no polarisation; the kernel's axis energies split energy[3] over three orthonormal axes by the
    # squared components of its polarisation vector, which is unit to a few ulp (measured on a B200: at most 7 ulp on the
    # layered models, 14 on the curved-ray ones, where the vector is carried along arcs)
    s_err = float((np.abs(got["energy"][~p, :3].sum(axis=1) - e3[~p]) / e3[~p]).max(initial=0.0))
    print(f"{label}: S axis energies sum to energy[3] within {s_err:.3e} relative")
    assert s_err <= 32 * EPS
    # the trace run's own bins hold exactly the catches decided (the log, which equals the reference off the edges)
    e, c, k = trace_bins
    cl, el, al = log_sums(m, rec)
    assert np.array_equal(c, cl) and int(k[abi.R3D_CNT_CATCHES]) == rec.size
    assert_energies_within_rounding(e, el, al, np.repeat(c.sum(axis=-1, keepdims=True), 5, axis=-1))
    margin = float(amb["margin"].max()) if amb.size else float("nan")
    print(f"{label}: {ref.size} catches compared ({int(p.sum())} P), {amb.size} ambiguous (largest margin {margin:.3e}), "
          f"coverage {cov}")
    return ref.size, amb.size, cov


# ---- 1. arrival-level exactness at full occupancy ----------------------------------------------------------------------
@pytest.mark.parametrize("name", sl.LAYOUTS)
@pytest.mark.parametrize("cfg", CONFIGS)
def test_log_equals_reference(cfg, name):
    m0, _ = load_golden(cfg)
    m = sl.layout(m0, name)
    n = n_phonons(cfg)
    rec, out = logged(m, n)
    ev, trace_bins = col_events(m, n)
    assert np.array_equal(out[1], log_sums(m, rec)[0])
    n_cmp, _, cov = compare_to_reference(m, rec, ev, trace_bins, f"{cfg}/{name}")
    assert n_cmp > 0
    if name == "annular":
        assert cov["annulus_catch"] > 100 and cov["inner_reject"] > 0
    if name == "edges":
        assert cov["negative_reject"] > 0 and cov["late_reject"] > 0


# ---- 2. the grid changes nothing but the candidate lists ---------------------------------------------------------------
@pytest.mark.parametrize("name", ["annular", "mixed"])
@pytest.mark.parametrize("cfg", CONFIGS)
def test_grid_invariance(cfg, name, monkeypatch):
    m0, _ = load_golden(cfg)
    m = sl.layout(m0, name)
    n = 250_000
    monkeypatch.delenv("R3D_GRID_MAX_DIM", raising=False)
    monkeypatch.delenv("R3D_CYL_WIDE", raising=False)
    base, (e0, c0, k0) = logged(m, n)
    assert base.size > 0
    cl, el, al = log_sums(m, base)
    n_add = np.repeat(c0.sum(axis=-1, keepdims=True), 5, axis=-1)
    settings = [(d, None) for d in ("1", "3", "1024")]
    if cfg in LAYERED:
        settings += [(None, w) for w in ("0", "1")] + [("1", "1"), ("3", "0")]
    ran = 0
    for dim, wide in settings:
        cells = sl.grid_size(m, int(dim) if dim else 128)[0]
        if cells > MAX_CELLS:
            print(f"{cfg}/{name}: R3D_GRID_MAX_DIM={dim}: {cells} cells, skipped")
            continue
        for var, v in (("R3D_GRID_MAX_DIM", dim), ("R3D_CYL_WIDE", wide)):
            if v is None:
                monkeypatch.delenv(var, raising=False)
            else:
                monkeypatch.setenv(var, v)
        rec, (e, c, k) = logged(m, n)
        assert rec.tobytes() == base.tobytes(), (dim, wide)
        assert np.array_equal(c, c0) and np.array_equal(k, k0), (dim, wide)
        assert_energies_within_rounding(e, el, al, n_add)
        ran += 1
    assert ran >= 2
