"""TEST INFRASTRUCTURE -- generate tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container (needs /root/reference):  python -m oracle.make_golden
The fixtures are small and committed; tests compare the oracle (and, on the GPU box,
the CUDA path) against them.  Inputs are regenerated from oracle.synth with the
seeds stored in the fixture, so only outputs are stored.

Lengths are tie-free (``unique_lengths=True``): the reference orders seeds by
``np.argsort(lengths)[::-1]`` (vamb/cluster.py:275) whose tie order depends on the NumPy
build / CPU (AVX-512 vs AVX2 sort), so fixtures with ties would not be portable.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

CLUSTER_CASES = [
    # name, n, nlatent, data seed, spread, rng_seed, kwargs
    ("c_2k_d32", 2000, 32, 0, 0.05, 0, {}),
    ("c_5k_d32", 5000, 32, 3, 0.2, 1, {}),
    ("c_10k_d32_mixed", 10000, 32, 5, 0.3, 2, {}),
    ("c_3k_d40", 3000, 40, 7, 0.1, 3, {}),
    ("c_1500_d283", 1500, 283, 9, 0.05, 4, {}),
    ("c_2k_d3", 2000, 3, 11, 0.02, 5, {}),
    ("c_4k_d32_small_window", 4000, 32, 13, 0.3, 6, {"windowsize": 20, "minsuccesses": 5, "maxsteps": 10}),
]


def cluster_inputs(n, nlatent, data_seed, spread):
    from oracle import synth

    return synth.make_latent(n, nlatent, data_seed, spread, unique_lengths=True)


def pack_clusters(clusters):
    sizes = np.array([len(c.members) for c in clusters], dtype=np.int64)
    return dict(
        medoid=np.array([c.medoid for c in clusters], dtype=np.int64),
        seed=np.array([c.seed for c in clusters], dtype=np.int64),
        sizes=sizes,
        members=np.concatenate([np.asarray(c.members, dtype=np.int64) for c in clusters]),
        radius=np.array([np.nan if c.radius is None else c.radius for c in clusters], dtype=np.float64),
        observed_pvr=np.array([np.nan if c.observed_pvr is None else c.observed_pvr for c in clusters], dtype=np.float64),
        maximal_pvr=np.array([c.maximal_pvr for c in clusters], dtype=np.float64),
        successes=np.array([c.successes for c in clusters], dtype=np.int64),
        attempts=np.array([c.attempts for c in clusters], dtype=np.int64),
    )


def make_cluster_goldens(ref):
    for name, n, nlatent, data_seed, spread, rng_seed, kw in CLUSTER_CASES:
        lat, lens = cluster_inputs(n, nlatent, data_seed, spread)
        clusters = list(ref.cluster.ClusterGenerator(lat, lens, rng_seed=rng_seed, **kw))
        kinds = {}
        for c in clusters:
            kinds[c.kind_str] = kinds.get(c.kind_str, 0) + 1
        out = pack_clusters(clusters)
        out["params"] = np.array([n, nlatent, data_seed, rng_seed], dtype=np.int64)
        out["spread"] = np.array([spread])
        np.savez_compressed(os.path.join(GOLDEN, f"cluster_{name}.npz"), **out)
        print(f"cluster_{name}: {len(clusters)} clusters {kinds}")


def main():
    from oracle import numerics, ref_loader

    numerics.pin()
    os.makedirs(GOLDEN, exist_ok=True)
    ref = ref_loader.load()
    make_cluster_goldens(ref)
    try:
        from oracle import make_golden_vae

        make_golden_vae.make(ref, GOLDEN)
    except ImportError:
        pass


if __name__ == "__main__":
    main()
