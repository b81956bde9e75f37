"""The model builder of bench.py and the degree-9 tests (radiative3d_b200/workload_model.py) against the models the reference
built for the same command lines (tests/golden/golden_<cfg>.npz, TOA degrees 2 and 3).

  * not gpu: the take-off-angle set to 1e-15 rad and the source tables to 1e-14 of their totals;
  * gpu: the whole model, scatterer tables from the device included: every array other than the TOA set and the CDF tables
    identical, the tables to 1e-10, and 1e5 scripted draws per table pick the same index in both.
"""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import CONFIGS, load_golden
from radiative3d_b200 import workload_model, workloads
from radiative3d_b200.model import _ARRAYS

APPROX = ("toa_theta", "toa_phi", "src_whole_cdf", "src_cdf", "scat_cdf", "scat_spol", "scat_whole_cdf", "scat_mfp")


def degree(m):
    return {320: 2, 1280: 3}[m.n_toa]


def source_of(cfg):
    return tuple(float(v) for v in workloads.CONFIGS[cfg]["source"].split(",")[1:4])


def check_cdfs(cdf, ref, n, tol):
    cdf, ref = cdf.reshape(-1, n), ref.reshape(-1, n)
    scale = ref[:, -1:].copy()
    scale[scale == 0] = 1.0
    assert (np.abs(cdf - ref) / scale).max() <= tol
    k = np.random.default_rng(11).integers(0, 2**31, 100000, dtype=np.uint32)
    k[:3] = (0, 1, 2**31 - 1)
    for a, b in zip(cdf, ref):
        if b[-1] > 0:
            assert np.array_equal(ob.cdf_search(a, k), ob.cdf_search(b, k))


@pytest.mark.parametrize("cfg", CONFIGS)
def test_toa_set_and_source_tables_are_the_references(cfg):
    m, _ = load_golden(cfg)
    th, ph = workload_model.toa_set(degree(m))
    assert np.abs(th - m.toa_theta).max() <= 1e-15 and np.abs(ph - m.toa_phi).max() <= 1e-15
    whole, cdf = workload_model.source_tables(*source_of(cfg), th, ph)
    assert np.abs(whole / m.src_whole_cdf - 1).max() <= 1e-14
    check_cdfs(cdf, m.src_cdf, m.n_toa, 1e-14)


def test_toa_set_size_and_spread():
    th, ph = workload_model.toa_set(5)
    assert th.size == 20 * 4**5
    u = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], -1)
    assert np.abs(u.mean(0)).max() < 1e-12                    # icosahedral symmetry: the set is centred
    assert np.unique(np.round(u, 12), axis=0).shape[0] == th.size


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS)
def test_built_model_is_the_references(cfg):
    r, _ = load_golden(cfg)
    m = workload_model.build_model(cfg, degree(r))
    for name, _ in _ARRAYS:
        if name not in APPROX:
            assert np.array_equal(getattr(m, name), getattr(r, name)), name
    for k in ("freq_hz", "ttl", "bin_dt", "n_bins", "src_cell", "cell_kind", "src_loc", "earth_center", "loop_concern"):
        assert getattr(m, k) == getattr(r, k), k
    assert np.abs(m.toa_theta - r.toa_theta).max() <= 1e-15
    check_cdfs(m.src_cdf, r.src_cdf, r.n_toa, 1e-14)
    check_cdfs(m.scat_cdf, r.scat_cdf, r.n_toa, 1e-10)
    assert np.abs(m.scat_mfp / r.scat_mfp - 1).max() <= 1e-10
    assert np.abs(m.scat_whole_cdf - r.scat_whole_cdf).max() <= 1e-10 * np.abs(r.scat_whole_cdf).max()
