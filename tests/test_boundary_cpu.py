"""CPU suite for the drop-in boundary: the C-ABI library loads and exports every declared
symbol, and argument validation raises the reference's exceptions before any GPU work."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from vamb_b200 import _lib

    header = open(os.path.join(ROOT, "include", "vamb_b200.h")).read()
    declared = set(re.findall(r"\b(vk_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(_lib.lib, name), f"{name} declared in include/vamb_b200.h but not exported"
    assert declared == set(_lib.declared_symbols())
    assert _lib.lib.vk_abi_version() == _lib.VK_ABI_VERSION


def test_binding_constants_match_the_header():
    """The Python binding restates the header's sizes (scratch buffers are allocated from them)."""
    from vamb_b200 import _lib

    header = open(os.path.join(ROOT, "include", "vamb_b200.h")).read()
    macros = dict(re.findall(r"#define\s+(VK_[A-Z0-9_]+)\s+([0-9]+)\b", header))
    for name in ("VK_ABI_VERSION", "VK_LIST_CAND", "VK_EVAL_SUBS", "VK_NBINS", "VK_PROBE_INLINE", "VK_MAX_CAND"):
        if hasattr(_lib, name) and name in macros:
            assert int(macros[name]) == getattr(_lib, name), name
    assert "VK_LIST_CAND" in macros and "VK_EVAL_SUBS" in macros and "VK_ABI_VERSION" in macros
    assert _lib.VK_EVAL_SCRATCH_U64 == _lib.VK_EVAL_SUBS * _lib.VK_LIST_CAND * 16
    assert re.search(r"#define\s+VK_EVAL_SCRATCH_U64\s+\(VK_EVAL_SUBS \* VK_LIST_CAND \* 16\)", header)


def test_probe_header_layout_matches_binding():
    from vamb_b200 import _lib

    assert _lib.HDR_SIZE == 16 + 8 * 60 + 16 + 4 * _lib.VK_PROBE_INLINE


def test_no_cpu_fallback():
    """With no CUDA device visible, require_device() raises instead of running on the CPU.  A child process with
    CUDA_VISIBLE_DEVICES="" sees no device, so this also runs on a machine that has one."""
    code = ("from vamb_b200 import _lib\n"
            "try:\n"
            "    _lib.require_device()\n"
            "except _lib.VkError:\n"
            "    print('refused')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == "refused"


class TestClusterBadParams:
    # test/test_cluster.py:15-36
    rng = np.random.RandomState(5)
    data = rng.random((64, 40)).astype(np.float32)
    lens = rng.randint(500, 1000, size=64)

    def test_bad_params(self):
        import vamb_b200.cluster as vc

        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data.astype(np.float64), self.lens)
        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data, self.lens, maxsteps=0)
        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data, self.lens, windowsize=0)
        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data, self.lens, minsuccesses=0)
        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data, self.lens, minsuccesses=5, windowsize=4)
        with pytest.raises(ValueError):
            vc.ClusterGenerator(np.random.random((0, 40)), np.array([], dtype=int))
        with pytest.raises(ValueError):
            vc.ClusterGenerator(self.data, self.lens[:-1])

    def test_cluster_kind(self):
        import vamb_b200.cluster as vc

        assert vc.Cluster(1, 0, np.array([1]), 0.1, None, None, 0, 0).kind_str == "loner"
        assert vc.Cluster(1, 0, np.array([1]), 0.1, None, 0.06, 0, 0).kind_str == "fallback"
        assert vc.Cluster(1, 0, np.array([1]), 0.1, 0.3, 0.04, 0, 0).kind_str == "normal"

    def test_edges_and_pdf_match_oracle(self):
        import vamb_b200.cluster as vc
        from oracle import cluster_oracle as co

        assert np.array_equal(vc._histogram_edges(), co.linspace_edges())
        assert np.array_equal(vc._NORMALPDF, co.NORMALPDF)


def test_native_rng_matches_cpython_sample():
    """The C++ driver restates random.Random(seed).sample(): MT19937 + init_by_array + rejection
    _randbelow + the pool / set switch.  Must match CPython call for call."""
    import random

    from vamb_b200 import _cluster_native as cn

    for seed in (0, 1, 5, 2 ** 40 + 17, 12345678901234567890, -7):
        for k in (25, 10, 3, 40):
            ns = [0, 1, 2, 5, 24, 25, 26, 100, 277, 278, 300, 5000, 100000, 7, 1]
            got = cn.rng_selftest(seed, ns, k)
            r = random.Random(seed)
            assert got == [r.sample(list(range(n)), min(n, k)) for n in ns], (seed, k)


def test_lane_major_layout_is_a_bijection_with_the_documented_block_structure():
    """include/vamb_b200.h: A-role operands of the tensor-core GEMMs are stored in 128-row panels whose
    32-wide k-tiles are 16 KB blocks [k/4][row][k%4] -- same footprint as the row-major array."""
    import numpy as np
    from vamb_b200 import _lib

    f = _lib.lib.vk_lane_major_index
    rows, ld = 256, 96
    idx = np.array([[f(r, k, ld) for k in range(ld)] for r in range(rows)], dtype=np.int64)
    assert sorted(idx.reshape(-1).tolist()) == list(range(rows * ld))          # bijection onto the same footprint
    r, k = np.meshgrid(np.arange(rows), np.arange(ld), indexing="ij")
    expect = (r // 128) * 128 * ld + (k // 32) * 4096 + ((k % 32) // 4) * 512 + (r % 128) * 4 + (k % 4)
    assert np.array_equal(idx, expect)
    # what the producer warps rely on: for a fixed group of four k, consecutive rows are consecutive float4
    assert f(5, 8, ld) - f(4, 8, ld) == 4 and f(4, 9, ld) - f(4, 8, ld) == 1
