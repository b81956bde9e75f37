"""Seismometer collection as an enumeration of (arrival, candidate) pairs over the lanes of a warp (collect_warp,
r3d_resident.cuh): the bins of r3d_run against the oracle, bin for bin.

The kernel and the oracle round FP64 differently (FMA contraction, CUDA libm), so a few phonons of a long run can take a
different discrete path.  Those are found by tracing the same range first and left out: the run and the oracle then cover
the same phonons in the same sub-ranges (draws are keyed by phonon index), and every bin must hold the same catches.
"""
import numpy as np
import pytest

import oracle_binding as ob
import seis_layouts as sl
from conftest import CONFIGS, load_golden
from radiative3d_b200 import abi, engine

pytestmark = pytest.mark.gpu


def agreeing_ranges(same):
    """Maximal runs [a, b) of phonons whose traced outcome equals the oracle's."""
    edges = np.flatnonzero(np.diff(np.concatenate(([0], same.astype(np.int8), [0]))))
    return list(zip(edges[0::2].tolist(), edges[1::2].tolist()))


def run_against_oracle(m, n, seed, nthreads=4):
    """(GPU bins, oracle bins, number of phonons compared) over the phonons of [0, n) that agree in outcome."""
    _, _, _, f_ref = ob.run(m, 0, n, seed, finals=True, nthreads=nthreads)
    with engine.Engine(m) as eng:
        fin = eng.trace(n, seed)
        same = np.ones(n, dtype=bool)
        for f in ("moves", "cell", "type", "fate", "draws"):
            same &= fin[f] == f_ref[f]
        assert same.mean() >= 0.995, f"only {same.mean():.4f} of phonons share the oracle's discrete outcome"
        # the trace kernel's catches per phonon (one shared-memory atomic per catch, added to the pair's arrival)
        assert np.array_equal(fin["catches"][same], f_ref["catches"][same])
        eng.reset()
        ranges = agreeing_ranges(same)
        for a, b in ranges:
            eng.run_simulation(b - a, seed=seed, first_phonon=a)
        gpu = eng.fetch()
    e_ref = np.zeros_like(gpu[0])
    c_ref = np.zeros_like(gpu[1])
    k_ref = np.zeros_like(gpu[2])
    for a, b in ranges:
        e, c, k, _ = ob.run(m, a, b - a, seed, nthreads=nthreads)
        e_ref += e
        c_ref += c
        k_ref += k
    return gpu, (e_ref, c_ref, k_ref), int(same.sum())


def assert_same_bins(gpu, ref, n):
    (e, c, k), (e_ref, c_ref, k_ref) = gpu, ref
    assert np.array_equal(c, c_ref)
    assert np.array_equal(k, k_ref)
    assert int(k[abi.R3D_CNT_PHONONS]) == n and int(k[abi.R3D_CNT_CATCHES]) == int(c.sum())
    # energies: each bin's channels relative to the bin's total (an axis component can be 0 in one and 1e-35 in the other).
    # The bar is the parity bar of test_gpu_propagate.py: the catches are the same, but the kernel and the oracle round the
    # FP64 ray arithmetic before them differently (up to 7e-12 of a bin on the curved-ray models).
    scale = np.maximum(e_ref[..., 3:].sum(axis=-1, keepdims=True), 1e-300)
    err = (np.abs(e - e_ref) / scale).max()
    print(f"largest energy difference: {err:.3e} of its bin")
    assert err <= 1e-8


@pytest.mark.parametrize("cfg", CONFIGS)
def test_run_bins_equal_oracle(cfg):
    m, z = load_golden(cfg)
    gpu, ref, n = run_against_oracle(m, int(z["run_n"]), int(z["run_seed"]))
    assert gpu[1].sum() > 0
    assert_same_bins(gpu, ref, n)


@pytest.mark.parametrize("copies", [11, 32])
def test_dense_seismometer_cluster(copies):
    """Every seismometer of the benchmark model `copies` times over: each grid cell then lists `copies` times its ~3
    candidates, so a face chunk with a handful of arrivals in non-empty cells has well over 96 pairs.  With 11 copies
    the passes span several arrivals (lists of 11 k pairs start anywhere in a pass); with 32 every list is a multiple of
    32 long and starts exactly at a pass boundary.  Arrivals in empty cells sit between them with no pairs."""
    m, _ = load_golden("halfspace_nearsrc50")
    ns = m.n_seis
    m.seis = np.ascontiguousarray(np.tile(m.seis.reshape(ns, abi.R3D_SEIS_NPARAM), (copies, 1)).ravel())
    gpu, ref, n = run_against_oracle(m, 10000, 77, nthreads=1)
    assert gpu[1].sum() > 0
    assert_same_bins(gpu, ref, n)
    # every copy of a seismometer is caught by exactly the same arrivals
    c = gpu[1].reshape(copies, ns, m.n_bins, 2)
    assert all(np.array_equal(c[i], c[0]) for i in range(1, copies))


LAYOUT_N = {"halfspace": 20000, "halfspace_nearsrc50": 20000, "crustpinch": 6000, "lopnor": 6000, "spherical": 1000}


@pytest.mark.parametrize("name", sl.LAYOUTS)
@pytest.mark.parametrize("cfg", CONFIGS)
def test_layout_bins_equal_oracle(cfg, name):
    """The station layouts of seis_layouts.py (annuli with S wider than P, mixed radii and far stations, a cut bin window
    with shifts below t = 0) end to end: counts exact, and the S axis energies, which depend on the polarisation the
    reports do not carry, held to the oracle with the rest."""
    m0, z = load_golden(cfg)
    m = sl.layout(m0, name)
    gpu, ref, n = run_against_oracle(m, LAYOUT_N[cfg], int(z["run_seed"]), nthreads=16)
    assert gpu[1].sum() > 0
    assert_same_bins(gpu, ref, n)
