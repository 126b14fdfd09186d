"""CPU suite: the cluster oracle is pinned against the reference.

 * golden fixtures (tests/golden/cluster_*.npz) were produced by the UNMODIFIED reference
   (oracle/make_golden.py); the oracle must reproduce every cluster exactly;
 * the oracle also reproduces the reference's clusters of the reference's own test fixture
   (test/test_cluster.py:11-13), stored by oracle/make_golden_reference.py;
 * restated known-answer pieces: histogram edges, smoothing kernel, in-place mask array.
"""
import os

import numpy as np
import pytest
import torch

from oracle import cluster_oracle as co
from oracle import make_golden_reference as mgr
from tests import _util


@pytest.mark.parametrize("name", list(_util.CLUSTER_CASES))
def test_oracle_matches_reference_golden(name):
    g, lat, lens, rng_seed = _util.load_cluster_golden(name)
    clusters = list(co.OracleClusterGenerator(lat, lens, rng_seed=rng_seed, **_util.CLUSTER_CASES[name]))
    _util.assert_clusters_equal_golden(clusters, g)
    # partition property (test/test_cluster.py:38-55)
    allm = np.concatenate([c.members for c in clusters])
    assert len(allm) == len(lat) and set(allm.tolist()) == set(range(len(lat)))


def test_oracle_matches_live_reference_on_reference_fixture():
    g = np.load(os.path.join(_util.GOLDEN, "ref_cluster_fixture.npz"))
    data, lens = mgr.cluster_fixture()
    oc = list(co.OracleClusterGenerator(data, lens, order=g["order"]))
    _util.assert_clusters_equal_golden(oc, g)


def test_histogram_edges_are_torch_linspace():
    assert np.array_equal(co.linspace_edges(), torch.linspace(0.0, co.XMAX, co.NBINS + 1).numpy())


def test_normalpdf_is_fp32_product():
    ref = (0.005 * torch.Tensor(co._PDF_VALUES)).numpy()
    assert np.array_equal(co.NORMALPDF, ref)


def test_smoothing_matches_torch_ops():
    rng = np.random.default_rng(0)
    hist = rng.integers(0, 10 ** 7, size=60).astype(np.float32)
    pdf = torch.from_numpy(co.NORMALPDF)
    th = torch.from_numpy(hist)
    dens = torch.zeros(90)
    for i in range(60):
        dens[i:i + 31] += pdf * th[i]
    assert np.array_equal(co.smooth_histogram(hist), dens[15:-15].numpy())


def test_normalize_properties():
    rng = np.random.default_rng(1)
    m = rng.standard_normal((500, 32)).astype(np.float32)
    m[7] = 0.0
    ref = m.copy()
    co.normalize(m)
    assert np.allclose((m.astype(np.float64) ** 2).sum(1), 0.5, atol=1e-6)
    # same direction as torch's own normalisation, to fp32 accuracy
    t = torch.from_numpy(ref.copy())
    t[7] = 1 / 32
    t /= t.norm(dim=1).reshape(-1, 1) * (2 ** 0.5)
    assert np.abs(m - t.numpy()).max() < 1e-6


def test_distance_matches_fp64_dot():
    rng = np.random.default_rng(2)
    for d in (3, 32, 40, 283):
        m = rng.standard_normal((300, d)).astype(np.float32)
        co.normalize(m)
        dist = co.calc_distances(m, 17)
        exact = 0.5 - m.astype(np.float64) @ m[17].astype(np.float64)
        exact[17] = 0
        assert np.abs(dist - exact).max() < 5e-7
        assert dist[17] == 0.0


def test_inplace_maskarray_semantics():
    # test/test_vambtools.py:271-298
    from oracle import vambcore_shim

    arr = np.random.default_rng(3).random((10, 3)).astype(np.float32)
    mask = np.array([0, 1, 1, 1, 1, 0, 0, 0, 0, 0]).astype(bool)
    expect = arr[mask]
    n = vambcore_shim.overwrite_matrix(arr, mask)
    assert n == 4 and np.array_equal(arr[:n], expect)
    with pytest.raises(ValueError):
        vambcore_shim.overwrite_matrix(arr[:4], mask)
