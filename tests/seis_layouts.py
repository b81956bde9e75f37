"""Seismometer layouts that the stock models do not have, and a brute-force restatement of seismometer collection from
the arrivals (COL event reports) to hold the kernel's collection to (tests/test_gpu_seis_layouts.py,
tests/test_gpu_collect_pairs.py, tests/test_seis_layouts_reference.py).

Layouts (each returns a copy of a golden model; the stations start from the model's own, so they stay on its
collection faces):
  annular  every station an annulus r_in = 0.3 r_out, with S gathering wider than P: the branch of CatchPhonon without
           the plane-wave shift, inner radii that differ by type, and a grid box set by the S radius.
  mixed    the stock stations, ~5 % copies at 20x radius (of stations in the smallest quarter), some at 0.05x, stations at the source's epicentre and
           stations that no arrival reaches (far outside the model, or off the collection surface): mixed radii make
           the median cell size a poor fit and the far stations stretch the grid box, so candidate lists get long.
  edges    fewer, odd-sized bins so that many arrivals fall past the last one, and plane-wave stations wide enough
           that early arrivals shift below t = 0.

The reference decides every (arrival, seismometer) pair with the oracle's seis_catch (ob.catch, compiled with
-ffp-contract=off).  Its operands are the arrival's reported state; the velocity at the arrival restates veloc_at
(include/r3d_gpu.h cell layouts).  Pairs whose deciding quantity lies within 1e-12 relative of an edge (a radius, a
bin boundary, 0 or the end of the window) are ambiguous: the kernel's state and the reported one differ in the last
bits (the direction goes through angles), so either answer is right there.  They are set apart, not decided.
"""
import copy

import numpy as np
from scipy.spatial import cKDTree

import oracle_binding as ob
from radiative3d_b200 import abi

NP = abi.R3D_SEIS_NPARAM
AMBIG_REL = 1e-12
CHUNK = 1 << 20                                     # pairs decided at a time (28 doubles each)
LAYOUTS = ["annular", "mixed", "edges"]


def _stations(m):
    return m.seis.reshape(-1, NP).copy()


def _with(m, s, **scalars):
    out = copy.deepcopy(m)
    out.seis = np.ascontiguousarray(s.reshape(-1), dtype=np.float64)
    for k, v in scalars.items():
        setattr(out, k, v)
    return out.validate()


def _set_radii(s, r_in, r_out):
    """Radii [P, S] columns (n, 2) each; the areas follow as the annuli's (dataout.cpp:42-71 divides by them)."""
    s[:, 12:14] = r_in
    s[:, 14:16] = r_out
    s[:, 16:18] = np.pi * (s[:, 14:16] ** 2 - s[:, 12:14] ** 2)
    return s


def epicentre(m):
    """The point of the collection surface above the source: radially for models with an earth centre, else straight up
    to the height of the station nearest the source's vertical."""
    s = m.seis.reshape(-1, NP)[:, :3]
    src = np.asarray(m.src_loc, dtype=np.float64)
    if m.ecs_radial:
        ec = np.asarray(m.earth_center, dtype=np.float64)
        r = np.median(np.linalg.norm(s - ec, axis=1))
        u = src - ec
        return ec + r * u / np.linalg.norm(u)
    near = np.argmin(np.hypot(s[:, 0] - src[0], s[:, 1] - src[1]))
    return np.array([src[0], src[1], s[near, 2]])


def annular(m):
    """Every station an annulus r_in = 0.3 r_out; S keeps the stock outer radius and P gets 0.6 of it (the stock
    stations have equal P and S radii), so the S radius alone sets the grid box and the pre-test."""
    s = _stations(m)
    r_out = s[:, 14:16] * np.array([0.6, 1.0])
    return _with(m, _set_radii(s, 0.3 * r_out, r_out))


def mixed(m, seed=11):
    rng = np.random.default_rng(seed)
    s = _stations(m)
    ns = s.shape[0]
    r = s[:, 14:16]
    small_r = np.argsort(r[:, 0], kind="stable")[:max(2, ns // 4)]     # (on the spherical model radii grow with distance)
    big = s[rng.choice(small_r, max(2, ns // 20), replace=False)]
    _set_radii(big, 0.0, 20.0 * big[:, 14:16])
    small = s[rng.choice(ns, max(2, ns // 20), replace=False)]
    _set_radii(small, 0.0, 0.05 * small[:, 14:16])
    epi = np.repeat(s[:1], 3, axis=0)
    epi[:, :3] = epicentre(m)
    _set_radii(epi, 0.0, np.outer([1.0, 5.0, 0.2], np.median(r, axis=0)))
    lo, hi = s[:, :3].min(axis=0), s[:, :3].max(axis=0)
    span = max(float(np.max(hi - lo)), 1.0)
    far = np.repeat(s[:1], 4, axis=0)               # never reached: far outside the model, in all directions
    far[:, :3] = (lo + hi) / 2 + span * np.array([[30.0, 0, 0], [-30.0, 25.0, 0], [0, -30.0, 40.0], [0, 0, -60.0]])
    src = np.asarray(m.src_loc, dtype=np.float64)
    h = float(np.linalg.norm(src - epicentre(m)))
    off = s[rng.choice(ns, 3, replace=False)]       # never reached: half way down to the source, off the collection surface
    off[:, :3] = 0.5 * (off[:, :3] + src)
    _set_radii(off, 0.0, np.minimum(off[:, 14:16], 0.2 * h))
    return _with(m, np.concatenate([s, big, small, epi, far, off]))


def edges(m):
    """n_bins and bin_dt cut (arrivals later than 0.55 of the stock window fall past the last bin).  The 8 stations
    whose distance L from the epicentre is nearest twice the source depth h get an outer radius 2 L + 2 h: a direct
    arrival at distance D > h^2 / L on the far side of the epicentre reaches the station, and its ray leans away from
    it by D / sqrt(D^2 + h^2), so the plane-wave shift -(D + L) D / (sqrt(D^2 + h^2) v) takes it below t = 0."""
    s = _stations(m)
    epi = epicentre(m)
    h = float(np.linalg.norm(np.asarray(m.src_loc) - epi))
    L = np.linalg.norm(s[:, :3] - epi, axis=1)
    wide = np.argsort(np.abs(L - 2 * h), kind="stable")[:8]
    ro = np.maximum(s[wide, 14:16], (2 * L[wide] + 2 * h)[:, None])
    s[wide] = _set_radii(s[wide], 0.0, ro)
    n_bins = max(8, int(m.n_bins * 0.4))
    bin_dt = m.bin_dt * 1.37
    return _with(m, s, n_bins=n_bins, bin_dt=bin_dt)


BUILDERS = {"annular": annular, "mixed": mixed, "edges": edges}


def layout(m, name):
    return BUILDERS[name](m)


# ---- the uniform grid over the stations: cells of the host formula (r3d_gpu.cu build_seis_grid) ----------------------
def grid_size(m, max_dim=128):
    """(cells, list entries, widest cell) of the seismometer grid r3d_create builds with R3D_GRID_MAX_DIM = max_dim."""
    s = m.seis.reshape(-1, NP)
    r = np.maximum(s[:, 14], s[:, 15])
    rad = r * (1.0 + 1e-6) + 1e-9 * (1.0 + np.abs(s[:, :3]).sum(axis=1))
    lo, hi = (s[:, :3] - rad[:, None]).min(axis=0), (s[:, :3] + rad[:, None]).max(axis=0)
    h = 2.0 * np.sort(rad)[s.shape[0] // 2]
    if not h > 0:
        h = 1.0
    ext = hi - lo
    ha = np.maximum(h, ext / max(1, max_dim))
    dim = np.maximum(1.0, np.ceil(ext / ha) + 1.0)
    c0 = np.clip(np.floor((s[:, :3] - rad[:, None] - lo) * (1.0 / ha)), 0, dim - 1)
    c1 = np.clip(np.floor((s[:, :3] + rad[:, None] - lo) * (1.0 / ha)), 0, dim - 1)
    return int(np.prod(dim)), int(np.prod(c1 - c0 + 1, axis=1).sum()), float(ha.max())


# ---- the reference ----------------------------------------------------------------------------------------------------
def veloc_at(m, cell, rtype, loc):
    """GetVelocAtPoint per arrival (media.cpp:185-196, 412-425, 646-660) from the cell records of include/r3d_gpu.h."""
    c = m.cell_params.reshape(m.n_cells, m.cell_nparam)[cell.astype(np.intp)]
    t = rtype.astype(np.intp)
    rows = np.arange(t.size)
    if m.cell_kind == abi.R3D_CELL_CYLINDER:
        return c[rows, t]
    if m.cell_kind == abi.R3D_CELL_SHELL:                   # C + A |x|^2
        return c[rows, 2 + t] + c[rows, t] * (loc * loc).sum(axis=1)
    g = np.stack([c[rows, 3 * t], c[rows, 3 * t + 1], c[rows, 3 * t + 2]], axis=1)
    return (loc * g).sum(axis=1) + c[rows, 6 + t]           # g.x + v0


def candidate_pairs(m, loc, all_pairs=False):
    """(arrival, seismometer) index pairs with the arrival within 1.01 x the station's larger outer radius (a filter
    only), or every pair."""
    s = m.seis.reshape(-1, NP)
    if all_pairs:
        a, k = np.meshgrid(np.arange(loc.shape[0]), np.arange(s.shape[0]), indexing="ij")
        return a.ravel(), k.ravel()
    if loc.shape[0] == 0:
        return np.zeros(0, np.intp), np.zeros(0, np.intp)
    tree = cKDTree(loc)
    lists = tree.query_ball_point(s[:, :3], r=np.maximum(s[:, 14], s[:, 15]) * 1.01 + 1e-9)
    k = np.repeat(np.arange(s.shape[0]), [len(x) for x in lists])
    a = np.concatenate([np.asarray(x, dtype=np.intp) for x in lists]) if k.size else np.zeros(0, np.intp)
    return a.astype(np.intp), k


def decide(m, ev, a, k):
    """The oracle's seis_catch on the pairs (a[i], k[i]): (out rows [caught, bin, e0..e3], ambiguity margin or +inf,
    classification dict).  pol = 0: the reports carry no polarisation, so S axis energies are not meaningful here."""
    s = m.seis.reshape(-1, NP)[k]
    e = ev[a]
    loc = np.ascontiguousarray(e["loc"], dtype=np.float64)
    t = e["type"].astype(np.intp)
    vel = veloc_at(m, e["cell"], e["type"], loc)
    rows = np.empty((a.size, 28))
    rows[:, :NP] = s
    rows[:, 18] = e["time"]
    rows[:, 19:22] = loc
    rows[:, 22] = e["theta"]
    rows[:, 23] = e["phi"]
    rows[:, 24] = 0.0
    rows[:, 25] = t
    rows[:, 26] = e["amp"]
    rows[:, 27] = vel
    out = ob.catch(m.bin_dt, m.n_bins, rows) if a.size else np.zeros((0, 6))

    # the deciding quantities, restated to find the pairs that sit on an edge
    rr = np.arange(a.size)
    r_in, r_out = s[rr, 12 + t], s[rr, 14 + t]
    toseis = s[:, :3] - loc
    d = np.sqrt((toseis * toseis).sum(axis=1))
    st, ct, sp, cp = np.sin(e["theta"]), np.cos(e["theta"]), np.sin(e["phi"]), np.cos(e["phi"])
    direc = np.stack([st * cp, st * sp, ct], axis=1)
    plane = r_in <= 0
    arv = e["time"] + np.where(plane, (toseis * direc).sum(axis=1) / vel, 0.0)
    scaled = arv / m.bin_dt
    # scales of the rounding each quantity carries: positions for d, the terms of the sum for the arrival time
    d_scale = np.maximum(np.maximum(r_out, np.abs(loc).max(axis=1)), 1e-300)
    t_scale = np.maximum((np.abs(e["time"]) + np.where(plane, d / np.abs(vel), 0.0)) / m.bin_dt, 1e-300)
    m_rin = np.where(r_in > 0, np.abs(d - r_in) / d_scale, np.inf)
    m_rout = np.abs(d - r_out) / d_scale
    kk = np.clip(np.rint(scaled), 0, m.n_bins)               # the nearest bin boundary inside [0, n_bins]
    m_t = np.abs(scaled - kk) / t_scale
    in_r = (d <= r_out * (1 + AMBIG_REL) + AMBIG_REL * d_scale) & (d >= r_in - AMBIG_REL * d_scale)
    in_t = (scaled >= -AMBIG_REL * t_scale) & (scaled < m.n_bins + AMBIG_REL * t_scale)
    margin = np.full(a.size, np.inf)
    margin = np.where(in_t, np.minimum(margin, np.minimum(m_rin, m_rout)), margin)
    margin = np.where(in_r, np.minimum(margin, m_t), margin)
    ambiguous = margin <= AMBIG_REL
    radius_ok = (d <= r_out) & (d >= r_in)
    cls = {
        "ambiguous": ambiguous,
        "inner_reject": ~ambiguous & (r_in > 0) & (d < r_in),
        "negative_reject": ~ambiguous & radius_ok & (scaled < 0),
        "late_reject": ~ambiguous & radius_ok & (scaled >= 0) & ~(np.floor(scaled) < m.n_bins),
        "annulus_catch": ~ambiguous & (out[:, 0] == 1) & (r_in > 0),
    }
    return out, margin, cls


def reference_catches(m, ev, all_pairs=False):
    """Brute-force collection of the arrivals `ev` (COL reports, abi.EVENT_DTYPE): (catches as abi.CATCH_DTYPE sorted
    by (phonon, moves, seis), ambiguous pairs as rows (phonon, moves, seis, margin), coverage counts)."""
    a, k = candidate_pairs(m, np.ascontiguousarray(ev["loc"], dtype=np.float64), all_pairs)
    parts = [decide(m, ev, a[i:i + CHUNK], k[i:i + CHUNK]) for i in range(0, max(a.size, 1), CHUNK)]
    out = np.concatenate([p[0] for p in parts])
    margin = np.concatenate([p[1] for p in parts])
    cls = {name: np.concatenate([p[2][name] for p in parts]) for name in parts[0][2]}
    amb = cls["ambiguous"]
    hit = (out[:, 0] == 1) & ~amb
    e = ev[a[hit]]
    rec = np.zeros(int(hit.sum()), dtype=abi.CATCH_DTYPE)
    rec["phonon"], rec["moves"], rec["type"], rec["time"] = e["phonon"], e["moves"], e["type"], e["time"]
    rec["seis"], rec["bin"] = k[hit], out[hit, 1].astype(np.uint32)
    rec["energy"] = out[hit, 2:6]
    rec = rec[np.lexsort((rec["seis"], rec["moves"], rec["phonon"]))]
    ea = ev[a[amb]]
    ambiguous = np.zeros(int(amb.sum()), dtype=[("phonon", "<u8"), ("moves", "<u4"), ("seis", "<u4"), ("margin", "<f8")])
    ambiguous["phonon"], ambiguous["moves"], ambiguous["seis"], ambiguous["margin"] = ea["phonon"], ea["moves"], k[amb], margin[amb]
    ambiguous = ambiguous[np.lexsort((ambiguous["seis"], ambiguous["moves"], ambiguous["phonon"]))]
    coverage = {name: int(v.sum()) for name, v in cls.items()}
    coverage["pairs"] = int(a.size)
    return rec, ambiguous, coverage


def keys(r):
    """(phonon, moves, seis) of records as one sortable void key each."""
    kt = np.dtype([("phonon", "<u8"), ("moves", "<u4"), ("seis", "<u4")])
    out = np.zeros(r.size, dtype=kt)
    for f in kt.names:
        out[f] = r[f]
    return out


# ---- sub-kernel rows of seis_catch at its edges (r3d_test_catch / ob.catch rows of 28 doubles) -------------------------
def catch_edge_rows(m, catch_in):
    """(rows, expected caught) for seis_catch: annuli with P and S radii apart (r_in 0.125 / 0.25, r_out 0.5 / 0.75 km)
    around integer station positions, so that offsets along one axis give distances exactly on r_in and r_out; arrival
    times exactly on bin boundaries with r_in > 0 (no shift), in the last bin and one past it; a plane-wave arrival
    shifted below t = 0 and one shifted inside the window.  Then the golden rows again with r_in = 0.3 r_out (expected
    -1: not asserted)."""
    x = np.asarray(catch_in, dtype=np.float64).reshape(-1, 28)
    tpl = x[0].copy()
    tpl[:3] = np.round(tpl[:3])
    _set_radii(tpl[None, :NP], np.array([0.125, 0.25]), np.array([0.5, 0.75]))
    sloc, vel, win = tpl[:3], tpl[27], m.n_bins * m.bin_dt
    rows, want = [], []

    def add(off, time, rtype, caught, plane=False, th=None, ph=None):
        r = tpl.copy()
        if plane:
            _set_radii(r[None, :NP], np.zeros(2), np.array([0.75, 0.75]))
        r[19:22] = sloc - np.asarray(off, dtype=np.float64)
        r[18], r[25] = time, rtype
        if th is not None:
            r[22], r[23] = th, ph
        rows.append(r)
        want.append(caught)

    mid = (np.floor(0.4 * m.n_bins) + 0.5) * m.bin_dt
    for t in (0, 1):
        ri, ro = tpl[12 + t], tpl[14 + t]
        add((ri, 0, 0), mid, t, 1)                              # d = r_in: inside (dist < r_in is false)
        add((0, -ro, 0), mid, t, 1)                             # d = r_out: inside (dist > r_out is false)
        add((0, 0, ri * (1 - 2.0 ** -30)), mid, t, 0)           # just inside r_in
        add((ro * (1 + 2.0 ** -30), 0, 0), mid, t, 0)           # just past r_out
        a = 0.5 * (ri + ro)
        for k in (0, 1, 17 % m.n_bins, m.n_bins - 1):
            add((0, a, 0), k * m.bin_dt, t, 1)                  # exactly on a bin's lower edge, no shift
        add((0, a, 0), m.n_bins * m.bin_dt, t, 0)               # one past the last bin, exactly on its edge
        add((0, a, 0), (m.n_bins - 0.5) * m.bin_dt, t, 1)       # the last bin
        add((0, a, 0), (m.n_bins + 0.5) * m.bin_dt, t, 0)       # past it
        add((0, a, 0), -0.5 * m.bin_dt, t, 0)                   # before t = 0
    add((0.625, 0, 0), mid, 0, 0)                               # between the P and the S outer radius
    add((0.625, 0, 0), mid, 1, 1)
    # plane wave, toseis = +0.5 x, ray along -x: the shift is -0.5 / vel
    add((0.5, 0, 0), 0.25 * 0.5 / vel, 0, 0, plane=True, th=np.pi / 2, ph=np.pi)      # shifted below t = 0
    add((0.5, 0, 0), 0.5 * win, 0, 1, plane=True, th=np.pi / 2, ph=np.pi)             # shifted within the window
    ann = x.copy()
    ann[:, :NP] = _set_radii(ann[:, :NP], 0.3 * ann[:, 14:16], ann[:, 14:16])
    return np.concatenate([np.array(rows), ann]), np.concatenate([want, np.full(ann.shape[0], -1)])
