"""The brute-force collection reference of tests/seis_layouts.py against a plain loop over every (arrival, seismometer)
pair, one ob.catch call each, on synthetic arrivals that include rows exactly on the radius and bin edges."""
import numpy as np
import pytest

import oracle_binding as ob
import seis_layouts as sl
from conftest import load_golden
from radiative3d_b200 import abi

NP = abi.R3D_SEIS_NPARAM


def velocity(m, cell, rtype, loc):
    c = m.cell_params.reshape(m.n_cells, m.cell_nparam)[cell]
    if m.cell_kind == abi.R3D_CELL_CYLINDER:
        return c[rtype]
    if m.cell_kind == abi.R3D_CELL_SHELL:
        return c[2 + rtype] + c[rtype] * (loc[0] * loc[0] + loc[1] * loc[1] + loc[2] * loc[2])
    return loc[0] * c[3 * rtype] + loc[1] * c[3 * rtype + 1] + loc[2] * c[3 * rtype + 2] + c[6 + rtype]


def synthetic(cfg, seed=3):
    """A model with 12 stations at exactly representable positions (plane-wave and annular, P and S radii apart) and
    arrivals around them: random ones, ones exactly at r_in and r_out (offsets along one axis), ones exactly on bin
    boundaries of annular stations (no shift), past the last bin and before t = 0."""
    m, _ = load_golden(cfg)
    rng = np.random.default_rng(seed)
    base = np.round(m.seis.reshape(-1, NP)[:12, :3])
    s = np.zeros((12, NP))
    s[:, :3] = base
    s[:, 3:12] = np.eye(3).ravel()
    r_out = np.stack([np.full(12, 4.0), np.full(12, 2.5)], axis=1)
    r_out[::3] = r_out[::3, ::-1]
    r_in = np.where(np.arange(12)[:, None] % 2 == 1, 0.25 * r_out, 0.0)      # odd stations annular: 1.0 / 0.625 (exact)
    s = sl._set_radii(s, r_in, r_out)
    m = sl._with(m, s)
    n_rand, window = 600, m.n_bins * m.bin_dt
    ev = np.zeros(n_rand, dtype=abi.EVENT_DTYPE)
    k = rng.integers(0, 12, n_rand)
    u = rng.standard_normal((n_rand, 3))
    ev["loc"] = s[k, :3] + u / np.linalg.norm(u, axis=1, keepdims=True) * rng.uniform(0, 5.0, n_rand)[:, None]
    ev["time"] = rng.uniform(-0.05, 1.1, n_rand) * window
    ev["theta"] = rng.uniform(0, np.pi, n_rand)
    ev["phi"] = rng.uniform(-np.pi, np.pi, n_rand)
    ev["type"] = rng.integers(0, 2, n_rand)
    ev["amp"] = rng.uniform(0.1, 1.0, n_rand)
    ev["cell"] = rng.integers(0, m.n_cells, n_rand)
    edge = []
    for j in (1, 3, 4):                               # exactly on r_in (annular only) and r_out, P and S
        for t in (0, 1):
            for r in ([s[j, 12 + t]] if s[j, 12 + t] > 0 else []) + [s[j, 14 + t]]:
                edge.append((s[j, :3] - np.array([r, 0.0, 0.0]), 0.4 * window, t))
    for j in (1, 5):                                  # annular: arrival exactly on a boundary, the last bin, one past it
        for b in (7, m.n_bins - 1, m.n_bins):
            edge.append((s[j, :3] + np.array([0.0, 0.0, 0.8]), b * m.bin_dt, 1))
    ed = np.zeros(len(edge), dtype=abi.EVENT_DTYPE)
    for i, (loc, t, ty) in enumerate(edge):
        ed[i]["loc"], ed[i]["time"], ed[i]["type"] = loc, t, ty
    ed["theta"], ed["phi"], ed["amp"], ed["cell"] = 1.0, 0.5, 0.5, 0
    ev = np.concatenate([ev, ed])
    ev["phonon"] = np.arange(ev.size) // 2
    ev["moves"] = np.arange(ev.size) % 2 + 1
    return m, ev, n_rand


@pytest.mark.parametrize("cfg", ["halfspace", "crustpinch", "spherical"])
def test_reference_equals_all_pairs_loop(cfg):
    m, ev, n_rand = synthetic(cfg)
    s = m.seis.reshape(-1, NP)
    rec, amb, cov = sl.reference_catches(m, ev)
    rec_all, amb_all, _ = sl.reference_catches(m, ev, all_pairs=True)
    assert rec.tobytes() == rec_all.tobytes() and amb.tobytes() == amb_all.tobytes()      # the tree only filters
    loop = {}
    for i, e in enumerate(ev):
        vel = velocity(m, int(e["cell"]), int(e["type"]), e["loc"])
        for j in range(s.shape[0]):
            row = np.concatenate([s[j], [e["time"]], e["loc"], [e["theta"], e["phi"], 0.0, e["type"], e["amp"], vel]])
            o = ob.catch(m.bin_dt, m.n_bins, row)[0]
            if o[0] == 1:
                loop[(int(e["phonon"]), int(e["moves"]), j)] = (int(o[1]), o[2:6])
    amb_keys = {(int(a["phonon"]), int(a["moves"]), int(a["seis"])) for a in amb}
    got = {(int(r["phonon"]), int(r["moves"]), int(r["seis"])): (int(r["bin"]), r["energy"]) for r in rec}
    want = {key: v for key, v in loop.items() if key not in amb_keys}
    assert got.keys() == want.keys()
    for key, (b, e) in want.items():
        assert got[key][0] == b and np.array_equal(got[key][1], e), key
    # every edge row is ambiguous, and no random row is
    edge_rows = {(int(e["phonon"]), int(e["moves"])) for e in ev[n_rand:]}
    assert {k[:2] for k in amb_keys} == edge_rows
    assert np.all(amb["margin"] <= sl.AMBIG_REL)
    assert len(loop) > 50 and cov["inner_reject"] > 0 and cov["annulus_catch"] > 0
    assert cov["negative_reject"] > 0 and cov["late_reject"] > 0


@pytest.mark.parametrize("name", sl.LAYOUTS)
@pytest.mark.parametrize("cfg", ["halfspace", "lopnor", "spherical"])
def test_layouts(cfg, name):
    m, _ = load_golden(cfg)
    lm = sl.layout(m, name)
    s0, s = m.seis.reshape(-1, NP), lm.seis.reshape(-1, NP)
    assert np.all(s[:, 14:16] > s[:, 12:14]) and np.all(s[:, 16:18] > 0)
    if name == "annular":
        assert np.array_equal(s[:, 15], s0[:, 15]) and np.all(s[:, 14] < s[:, 15])
        assert np.array_equal(s[:, 12:14], 0.3 * s[:, 14:16])
    elif name == "mixed":
        assert s.shape[0] > s0.shape[0] and np.array_equal(s[:s0.shape[0]], s0)
        assert np.isin(20.0 * s0[:, 14], s[:, 14]).sum() >= 2 and np.isin(0.05 * s0[:, 14], s[:, 14]).sum() >= 2
        assert sl.grid_size(lm)[2] > 10 * sl.grid_size(m)[2]   # far stations: coarse cells, long candidate lists
    else:
        assert lm.n_bins < m.n_bins and lm.n_bins * lm.bin_dt < 0.6 * m.n_bins * m.bin_dt
        assert (s[:, 14] > s0[:, 14]).sum() == 8
    cells, items, _ = sl.grid_size(lm, 1)                  # at most 2 cells per axis, a few stations listed twice
    assert cells <= 8 and s.shape[0] <= items < 2 * s.shape[0]


@pytest.mark.parametrize("cfg", ["halfspace", "crustpinch", "spherical"])
def test_catch_edge_rows(cfg):
    """The edge rows of the sub-kernel test decide as they are meant to in the oracle, and the annulus rows from the
    golden ones both catch and reject by the inner radius."""
    m, z = load_golden(cfg)
    rows, want = sl.catch_edge_rows(m, z["catch_in"])
    out = ob.catch(m.bin_dt, m.n_bins, rows)
    edge = want >= 0
    assert np.array_equal(out[edge, 0], want[edge])
    ann = ~edge
    d = np.linalg.norm(rows[ann, :3] - rows[ann, 19:22], axis=1)
    t = rows[ann, 25].astype(int)
    r_in = rows[ann][np.arange(ann.sum()), 12 + t]
    assert out[ann, 0].sum() > 10 and (d < r_in).sum() > 10
