"""TEST INFRASTRUCTURE -- fixtures of the parity checks against the UNMODIFIED reference.

Run where the reference tree is available (oracle/ref_loader.py):
    python -m oracle.make_golden_reference

Writes tests/golden/ref_*.npz: what the reference's ``make_dataloader``, VAE training steps,
``VAE.trainmodel`` and ``ClusterGenerator`` return on the inputs defined here.  The tests
rebuild the same inputs with the functions below and compare the oracle and the product
with the stored results, so they need no reference tree.

Large arrays are stored as a SHA-256 of their bytes plus a fixed sample of rows: the digest
keeps the comparison bit-exact over the whole array, the rows show where a mismatch is.
"""
from __future__ import annotations

import hashlib
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
SAMPLE_ROWS = 8

# make_dataloader cases: name -> inputs (abundance, tnf, lengths)
VAE_STEPS = dict(S=5, n=400, batch=64, seed=11, nhiddens=[64, 48], nlatent=12, nsteps=6, torch_seed0=2000)
TRAINMODEL = dict(S=4, n=1500, data_seed=8, seed=3, nhiddens=[64, 32], nlatent=8, batch=128, nepochs=4, batchsteps=[2])


def dataloader_inputs(name):
    if name == "synth_2000x3":
        from oracle import synth

        return synth.make_contigs(2000, 3, seed=5)
    if name == "uniform_300x5_zero_row":
        rng = np.random.RandomState(3)
        tnfs = rng.random((300, 103)).astype(np.float32)
        rpkm = rng.random((300, 5)).astype(np.float32)
        rpkm[7] = 0  # an all-zero abundance row
        lens = rng.randint(2000, 90000, 300)
        return rpkm, tnfs, lens
    raise KeyError(name)


DATALOADER_CASES = ["synth_2000x3", "uniform_300x5_zero_row"]


def cluster_fixture():
    """The reference's own clustering fixture (test/test_cluster.py:11-13)."""
    rng = np.random.RandomState(5)
    data = rng.random((1024, 40)).astype(np.float32)
    lens = rng.randint(500, 1000, size=1024)
    return data, lens


def sha256(x) -> str:
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


def digest_and_sample(prefix, x, rows):
    return {f"{prefix}_sha256": np.array(sha256(x)), f"{prefix}_rows": np.ascontiguousarray(x[rows])}


def assert_digest_and_sample(g, prefix, x):
    """Bit-exact comparison of ``x`` with an array stored by ``digest_and_sample``."""
    rows = g["rows"]
    assert x[rows].dtype == g[f"{prefix}_rows"].dtype, prefix
    bad = np.argwhere(x[rows] != g[f"{prefix}_rows"])
    assert len(bad) == 0, f"{prefix}: differs at (sampled row, column) {bad[:5].tolist()}"
    assert sha256(x) == str(g[f"{prefix}_sha256"]), f"{prefix}: differs outside the sampled rows"


def make_dataloader_goldens(ref):
    for name in DATALOADER_CASES:
        ab, tnf, lens = dataloader_inputs(name)
        tensors = ref.encode.make_dataloader(ab.copy(), tnf.copy(), lens).dataset.tensors
        rows = np.sort(np.random.default_rng(0).choice(len(lens), SAMPLE_ROWS, replace=False))
        out = {"rows": rows}
        for k, x in zip("dtaw", tensors):
            out.update(digest_and_sample(k, x.numpy(), rows))
        np.savez_compressed(os.path.join(GOLDEN, f"ref_dataloader_{name}.npz"), **out)
        print(f"ref_dataloader_{name}")


def make_vae_steps_golden(ref):
    """The reference VAE (with the restated DAdaptAdam) over optimiser steps under ``torch.manual_seed``."""
    from oracle import dadapt
    from oracle.make_golden_vae import vae_inputs

    c = VAE_STEPS
    rpkm, tnfs, lens = vae_inputs(c["S"], c["n"], c["seed"])
    dl = ref.encode.make_dataloader(rpkm.copy(), tnfs.copy(), lens, batchsize=c["batch"])
    d, t, a, w = dl.dataset.tensors
    vae = ref.encode.VAE(c["S"], nhiddens=c["nhiddens"], nlatent=c["nlatent"], seed=c["seed"])
    opt = dadapt.DAdaptAdam(vae.parameters(), decouple=True)
    vae.train()
    rng = np.random.default_rng(c["seed"])
    losses = []
    for step in range(c["nsteps"]):
        idx = torch.from_numpy(rng.choice(c["n"], size=c["batch"], replace=False).astype(np.int64))
        torch.manual_seed(c["torch_seed0"] + step)
        opt.zero_grad()
        do, to, ao, mu = vae(d[idx], t[idx], a[idx])
        L = vae.calc_loss(d[idx], do, t[idx], to, a[idx], ao, mu, w[idx])
        L[0].backward()
        opt.step()
        losses.append([float(x.detach()) for x in L])
    out = {"losses": np.array(losses, dtype=np.float64)}
    out.update({f"state.{k}": np.array(sha256(v.numpy())) for k, v in vae.state_dict().items()})
    vae.eval()
    rows = np.sort(np.random.default_rng(0).choice(c["n"], SAMPLE_ROWS, replace=False))
    out.update(rows=rows, **digest_and_sample("latent", vae.encode(dl), rows))
    np.savez_compressed(os.path.join(GOLDEN, "ref_vae_steps.npz"), **out)
    print(f"ref_vae_steps: losses {losses[-1][0]:.5f}")


def make_trainmodel_golden(ref):
    """The per-epoch losses that the reference's ``VAE.trainmodel`` logs."""
    from loguru import logger

    from oracle import synth

    c = TRAINMODEL
    ab, tnf, lens = synth.make_contigs(c["n"], c["S"], seed=c["data_seed"])
    rows = []
    pat = re.compile(r"Epoch:\s*(\d+)\s+Loss:\s*(\S+)")
    logger.enable("vamb")
    sink = logger.add(lambda m: rows.append(pat.search(str(m))), level="INFO")
    dl = ref.encode.make_dataloader(ab.copy(), tnf.copy(), lens, batchsize=c["batch"])
    vae = ref.encode.VAE(c["S"], nhiddens=c["nhiddens"], nlatent=c["nlatent"], seed=c["seed"])
    vae.trainmodel(dl, nepochs=c["nepochs"], batchsteps=c["batchsteps"])
    logger.remove(sink)
    logger.disable("vamb")
    logged = [float(m.group(2)) for m in rows if m]
    assert len(logged) == c["nepochs"]
    np.savez_compressed(os.path.join(GOLDEN, "ref_trainmodel_losses.npz"), epoch_loss=np.array(logged))
    print(f"ref_trainmodel_losses: {logged}")


def make_cluster_fixture_golden(ref):
    from oracle.make_golden import pack_clusters

    data, lens = cluster_fixture()
    gen = ref.cluster.ClusterGenerator(data, lens)
    order = np.array(gen.order, dtype=np.int64)  # the seed order it drew: argsort's tie order is CPU-dependent
    out = pack_clusters(list(gen))
    out["order"] = order
    np.savez_compressed(os.path.join(GOLDEN, "ref_cluster_fixture.npz"), **out)
    print(f"ref_cluster_fixture: {len(out['medoid'])} clusters")


def main():
    from oracle import numerics, ref_loader

    numerics.pin()
    os.makedirs(GOLDEN, exist_ok=True)
    ref = ref_loader.load()
    make_dataloader_goldens(ref)
    make_vae_steps_golden(ref)
    make_trainmodel_golden(ref)
    make_cluster_fixture_golden(ref)


if __name__ == "__main__":
    main()
