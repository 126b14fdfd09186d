"""CPU suite for the bench contract: the step slicing, the one-JSON-line rule of stdout and the reference arm
(which must run without the product package and without a GPU)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import importlib

    return importlib.import_module("bench")


def test_epoch_slices_partition_the_schedule():
    b = _bench()
    for nepochs, k in [(300, 20), (300, 7), (5, 5), (3, 20), (1, 1)]:
        cuts = b.epoch_slices(nepochs, k)
        assert cuts[0] == 0 and cuts[-1] == nepochs and len(cuts) == k + 1
        assert all(x <= y for x, y in zip(cuts, cuts[1:]))
    assert b.epoch_slices(300, 20) == list(range(0, 301, 15))


def test_reference_arm_prints_one_json_line_and_never_loads_the_product():
    """`bench.py --impl reference` on a small workload: stdout is exactly one JSON line with the contract's keys;
    everything else (logs, library banners) goes to stderr; vamb_b200 is never imported."""
    code = (
        "import sys, runpy\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--contigs', '20000', '--nsamples', '8', '--steps', '4', '--warmup', '1',"
        " '--cpu-seconds', '2']\n"
        "try:\n"
        "    runpy.run_path('bench.py', run_name='__main__')\n"
        "except SystemExit:\n"
        "    pass\n"
        "bad = [m for m in sys.modules if m == 'vamb_b200' or m.startswith('vamb_b200.')]\n"
        "sys.stderr.write('PRODUCT_MODULES=' + repr(bad) + '\\n')\n"
    )
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "contigs/s" and d["higher_is_better"] is True
    assert d["steps"] == 4 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "contigs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "PRODUCT_MODULES=[]" in r.stderr


def test_steps_below_one_is_rejected():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    assert r.stdout == ""


def test_dump_outputs_writes_a_fixed_sample_of_the_latent_and_the_clustering(tmp_path):
    """dump_outputs on a fake pass: one float file per output, every value finite, the same rows for the same seed,
    every sampled contig mapped to the medoid and radius of the cluster that holds it, and the 64 MB bound at the
    largest sample."""
    import types

    import numpy as np
    import torch

    b = _bench()
    n, L = 1000, 32
    latent = torch.arange(n * L, dtype=torch.float32).reshape(n, L)
    perm = np.random.default_rng(1).permutation(n)
    clusters = [types.SimpleNamespace(medoid=int(m[0]), members=m, radius=(None if k == 2 else 0.1 * k))
                for k, m in enumerate(np.array_split(perm, 7))]
    names = b.dump_outputs(str(tmp_path / "a"), latent, clusters, seed=3)
    b.dump_outputs(str(tmp_path / "b"), latent, clusters, seed=3)
    assert names == ["cluster_index", "cluster_medoid", "cluster_radius", "latent", "rows"]
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in names}
    for k in names:
        assert got[k].dtype in (np.float32, np.float64) and np.isfinite(got[k]).all(), k
        assert np.array_equal(got[k], np.load(tmp_path / "b" / f"{k}.npy"))
    rows = got["rows"].astype(np.int64)
    assert len(rows) == n and np.array_equal(rows, np.arange(n))  # n < DUMP_ROWS: every contig
    assert np.array_equal(got["latent"], latent.numpy()[rows])
    for r, k, m, rad in zip(rows, got["cluster_index"], got["cluster_medoid"], got["cluster_radius"]):
        c = clusters[int(k)]
        assert r in c.members and m == c.medoid
        assert rad == (-1.0 if c.radius is None else c.radius)
    assert b.DUMP_ROWS * (L * 4 + 4 * 8) <= 64 << 20
