"""CPU suite for the encode boundary: the reference's TestDataLoader (test/test_encode.py:8-119)
and the constructor / trainmodel argument checks (:127-150), which run before any GPU work."""
import numpy as np
import pytest
import torch

import vamb_b200.encode as ve
from vamb_b200 import vambtools as vt


class TestDataLoader:
    tnfs = np.random.random((111, 103)).astype(np.float32)
    rpkm = np.random.random((111, 14)).astype(np.float32)
    lens = np.random.randint(2000, 5000, size=111)

    def nearly_same(self, a, b):
        assert np.all(np.abs(a - b) < 1e-5)

    def test_bad_args(self):
        with pytest.raises(ValueError):
            ve.make_dataloader([[1, 2, 3]], self.tnfs, self.lens, batchsize=32)
        with pytest.raises(ValueError):
            ve.make_dataloader(self.rpkm, self.tnfs, self.lens, batchsize=0)
        with pytest.raises(ValueError):
            ve.make_dataloader(self.rpkm.astype(np.float64), self.tnfs, self.lens, batchsize=32)
        with pytest.raises(ValueError):
            ve.make_dataloader(self.rpkm, self.tnfs.astype(np.float64), self.lens, batchsize=32)
        with pytest.raises(ValueError):
            ve.make_dataloader(self.rpkm, self.tnfs[:-1], self.lens, batchsize=32)
        with pytest.raises(ValueError):
            cp = self.rpkm.copy()
            cp[:, 3] = 0
            ve.make_dataloader(cp, self.tnfs, self.lens, batchsize=32)

    def test_destroy(self):
        rpkm_copy, tnfs_copy = self.rpkm.copy(), self.tnfs.copy()
        ve.make_dataloader(rpkm_copy, tnfs_copy, self.lens, batchsize=32)
        assert np.all(rpkm_copy == self.rpkm) and np.all(tnfs_copy == self.tnfs)
        ve.make_dataloader(rpkm_copy, tnfs_copy, self.lens, batchsize=32, destroy=True)
        assert not np.all(rpkm_copy == self.rpkm) and not np.all(tnfs_copy == self.tnfs)

    def test_normalized(self):
        rpkm_copy, tnfs_copy = self.rpkm.copy(), self.tnfs.copy()
        ve.make_dataloader(rpkm_copy, tnfs_copy, self.lens, batchsize=32, destroy=True)
        self.nearly_same(np.mean(tnfs_copy, axis=0), np.zeros(103))
        self.nearly_same(np.std(tnfs_copy, axis=0), np.ones(103))
        self.nearly_same(np.sum(rpkm_copy, axis=1), np.ones(len(rpkm_copy)))
        assert np.all(rpkm_copy >= 0.0)

    def test_single_sample(self):
        single = self.rpkm[:, [0]].copy()
        dl = ve.make_dataloader(single, self.tnfs.copy(), self.lens, batchsize=32, destroy=True)
        depths, _, ab, _ = dl.dataset.tensors
        assert np.all(np.abs(depths.numpy() - 1.0) < 1e-6)
        assert abs(float(ab.mean())) < 1e-5

    def test_iter_and_contract(self):
        dl = ve.make_dataloader(self.rpkm, self.tnfs, self.lens, batchsize=32)
        d, t, a, w = next(iter(dl))
        assert d.dtype == t.dtype == a.dtype == w.dtype == torch.float32
        assert d.shape == (32, 14) and t.shape == (32, 103) and a.shape == (32, 1) and w.shape == (32, 1)
        assert dl.batch_size == 32 and len(dl) == 111 // 32
        dl2 = ve.set_batchsize(dl, 64, 111)
        assert dl2.batch_size == 64 and dl2.dataset is dl.dataset
        dl3 = ve.set_batchsize(dl, 64, 111, encode=True)
        assert len(dl3) == 2  # no drop_last
        assert abs(float(dl.dataset.tensors[3].mean()) - 1.0) < 1e-5


def test_matches_reference_dataloader_when_available():
    """make_dataloader's tensors == the reference's, bit for bit (tests/golden/ref_dataloader_*.npz)."""
    import os

    from oracle import make_golden_reference as mgr

    name = "uniform_300x5_zero_row"
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"ref_dataloader_{name}.npz"))
    rpkm, tnfs, lens = mgr.dataloader_inputs(name)
    b = ve.make_dataloader(rpkm.copy(), tnfs.copy(), lens, batchsize=64)
    for k, y in zip("dtaw", b.dataset.tensors):
        mgr.assert_digest_and_sample(g, k, y.numpy())


class TestVAEArgs:
    def test_bad_args(self):
        for kw in (dict(nsamples=0), dict(nsamples=3, nlatent=0), dict(nsamples=3, nhiddens=[0, 5]),
                   dict(nsamples=3, beta=0.0), dict(nsamples=3, alpha=0.0), dict(nsamples=3, alpha=1.0),
                   dict(nsamples=3, dropout=1.0), dict(nsamples=3, dropout=-0.1)):
            with pytest.raises(ValueError):
                ve.VAE(**kw)


class TestTools:
    arr = np.array([[1, 2, 2.5], [2, 4, 3], [0.9, 3.1, 2.8]])

    def test_zscore_known_answers(self):
        # test/test_vambtools.py:212-269
        z = np.array([[-1.44059316, -0.3865006, 0.14054567], [-0.3865006, 1.7216845, 0.66759195],
                      [-1.54600241, 0.77300121, 0.45677344]])
        assert np.all(np.abs(vt.zscore(self.arr) - z) < 1e-6)
        z0 = np.array([[-0.60404045, -1.26346568, -1.29777137], [1.40942772, 1.18195176, 1.13554995],
                       [-0.80538727, 0.08151391, 0.16222142]])
        assert np.all(np.abs(vt.zscore(self.arr, axis=0) - z0) < 1e-6)
        z1 = np.array([[-1.33630621, 0.26726124, 1.06904497], [-1.22474487, 1.22474487, 0.0],
                       [-1.40299112, 0.85548239, 0.54750873]])
        assert np.all(np.abs(vt.zscore(self.arr, axis=1) - z1) < 1e-6)
        with pytest.raises(np.exceptions.AxisError):
            vt.zscore(self.arr, axis=-1)
        with pytest.raises(np.exceptions.AxisError):
            vt.zscore(self.arr, axis=2)
        with pytest.raises(TypeError):
            vt.zscore(np.array([1, 2, 3]), inplace=True)
        assert np.all(vt.zscore(np.array([4, 4, 4])) == 0)
        cp = self.arr.copy()
        vt.zscore(cp, inplace=True)
        assert np.all(np.abs(cp - z) < 1e-6)

    def test_inplace_maskarray(self):
        # test/test_vambtools.py:271-298
        arr = np.random.random((10, 3)).astype(np.float32)
        mask = np.array([0, 1, 1, 1, 1, 0, 0, 0, 0, 0]).astype(bool)
        arr2 = arr[mask]
        vt.numpy_inplace_maskarray(arr, mask)
        assert np.all(np.abs(arr - arr2) < 1e-6)
        with pytest.raises(ValueError):
            vt.numpy_inplace_maskarray(arr, mask)
        t = torch.rand(10, 3)
        m = torch.tensor([0, 1, 1, 1, 1, 0, 0, 0, 0, 0], dtype=bool)
        t2 = t[m]
        vt.torch_inplace_maskarray(t, m)
        assert torch.all(torch.abs(t - t2) < 1e-6)
        with pytest.raises(ValueError):
            vt.torch_inplace_maskarray(t, m)

    def test_mask_lower_bits(self):
        x = np.random.default_rng(0).standard_normal(1000).astype(np.float32)
        y = x.copy()
        vt.mask_lower_bits(y, 12)
        assert np.all(y.view(np.uint32) & 0xFFF == 0) and np.all(np.abs(x - y) <= np.abs(x) * 2.0 ** -11)
        with pytest.raises(ValueError):
            vt.mask_lower_bits(y, 24)
