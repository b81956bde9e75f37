"""Parity AT the benchmarked configuration: take-off-angle degree 9 (scripts/do-fundamentals.sh:82), 5 242 880 take-off
angles, 0.42 GB of CDF tables, 2^23-bucket guide tables - the configuration bench.py measures, not a reduced copy of it.

The models are built as bench.py builds them (radiative3d_b200.workload_model, held to the reference's own builds by
tests/test_workload_model.py).  Two legs:
  * phonon by phonon against the oracle on the same flattened model and the same draw stream (criteria of
    tests/test_gpu_propagate.py: discrete outcome identical for >= 99.5 %, times / path lengths / locations to 1e-8);
  * statistically against runs of the UNMODIFIED reference binary at degree 9 with its own rand() stream
    (tests/golden/stat_halfspace_nearsrc50_deg9.npz, 16 processes x 1e6 phonons, made by make_stat_golden.py): Welch
    criteria of tests/test_gpu_statistical.py.
"""
import os

import numpy as np
import pytest

import oracle_binding as ob
from radiative3d_b200 import abi, engine, workload_model
from test_gpu_propagate import compare_finals
from test_gpu_statistical import compare, gpu_batches, load_stat

pytestmark = pytest.mark.gpu

# workload -> phonons traced one by one at degree 9 (the oracle does 2e5 ... 3e2 phonons/s per host thread)
TRACE_N = {"halfspace_nearsrc50": 60000, "halfspace": 30000, "crustpinch": 6000, "lopnor": 6000, "spherical": 600}
_models = {}


def model9(cfg):
    if cfg not in _models:
        _models.clear()                         # one degree-9 model at a time (up to 4.6 GB of host arrays)
        _models[cfg] = workload_model.build_model(cfg, 9)
    return _models[cfg]


@pytest.mark.parametrize("cfg", list(TRACE_N))
def test_trace_matches_oracle_at_degree_9(cfg):
    m = model9(cfg)
    assert m.n_toa == 5242880
    n, seed, first = TRACE_N[cfg], 424242, 10_000_000
    e_ref, c_ref, k_ref, f_ref = ob.run(m, first, n, seed, finals=True, nthreads=min(16, os.cpu_count() or 1))
    with engine.Engine(m) as eng:
        fin = eng.trace(n, seed=seed, first_phonon=first)
        e, c, k = eng.fetch()
    same = compare_finals(fin, f_ref)
    n_off = int((~same).sum())
    print(cfg, f"degree 9: {int(same.sum())}/{n} phonons identical in outcome to the oracle")
    assert np.abs(c.astype(np.int64) - c_ref.astype(np.int64)).sum() <= 50 * n_off
    assert np.abs(k[:3].astype(np.int64) - k_ref[:3].astype(np.int64)).sum() <= 2 * n_off
    if n_off == 0:
        assert np.array_equal(c, c_ref) and np.array_equal(k[:3], k_ref[:3])
    assert int(k[abi.R3D_CNT_PHONONS]) == n


def test_statistics_match_reference_binary_at_degree_9():
    z = load_stat("halfspace_nearsrc50_deg9")
    assert int(z["toa_degree"]) == 9
    m = model9("halfspace_nearsrc50")
    cg, eg, kg, n = gpu_batches(m, z)
    c, e, k = z["counts"], z["energy"].astype(np.float64).sum(-1), z["counters"]
    stats, fails = compare(cg, c, eg, e, kg, k.sum(0), n, n)
    print("halfspace_nearsrc50 degree 9", stats)
    assert not fails, (stats, fails)
