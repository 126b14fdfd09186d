"""CPU suite: the torch-fp32 VAE oracle is PINNED -- it reproduces the reference-made golden fixtures bit for bit
(tests/golden/vae_*.npz, written by oracle/make_golden_vae.py, and tests/golden/ref_*.npz, written by
oracle/make_golden_reference.py, both from the unmodified reference).  Also pins oracle/normalize.py."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden_reference as mgr
from oracle import vae_oracle as vo
from oracle.make_golden_vae import VAE_CASES, vae_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def unpack_keep(packed, batch, n):
    return torch.from_numpy(np.unpackbits(packed)[: batch * n].reshape(batch, n).astype(np.float32))


@pytest.mark.parametrize("case", VAE_CASES, ids=[c[0] for c in VAE_CASES])
def test_vae_oracle_reproduces_reference_goldens_bitwise(case):
    """Same batches, same recorded noise -> the reference's losses, d, parameters and latent, exactly."""
    from oracle import normalize as onorm

    name, S, nh, nl, dp, n, batch, nsteps, seed = case
    g = np.load(os.path.join(GOLDEN, f"vae_{name}.npz"))
    rpkm, tnfs, lens = vae_inputs(S, n, seed)
    d, t, a, w = (torch.from_numpy(x) for x in onorm.normalize(rpkm, tnfs, lens))
    o = vo.OracleVAE(S, nhiddens=nh, nlatent=nl, dropout=dp, seed=seed)
    hidden = o.nhiddens + o.nhiddens[::-1]
    for step in range(nsteps):
        idx = torch.from_numpy(g["batch_idx"][step])
        keeps = None
        if o.dropout > 0:
            keeps = [unpack_keep(g[f"keep{li}"][step], batch, hidden[li]) for li in range(len(hidden))]
        lo, _, _ = o.train_step(d[idx], t[idx], a[idx], w[idx], eps=torch.from_numpy(g["eps"][step]), keeps=keeps)
        assert lo == list(g["losses"][step]), (step, lo, g["losses"][step])
        assert o.d == float(g["d"][step])
    L = len(o.nhiddens)
    assert np.array_equal(o.state["mu.weight"].numpy(), g["mu_weight"])
    assert np.array_equal(o.state["outputlayer.bias"].numpy(), g["out_bias"])
    assert np.array_equal(o.state["encoderlayers.0.weight"].numpy()[:8], g["enc0_weight_head"])
    assert np.array_equal(o.state["encodernorms.0.running_mean"].numpy(), g["bn0_running_mean"])
    assert np.array_equal(o.state["encodernorms.0.running_var"].numpy(), g["bn0_running_var"])
    assert np.array_equal(o.state[f"decodernorms.{L - 1}.weight"].numpy(), g["bn_last_weight"])
    latent, _ = o.encode(d, t, a, batch=batch)
    assert np.array_equal(latent, g["latent"])


def test_normalize_restatement_matches_the_product_dataloader():
    """oracle/normalize.py (used by the reference arm of bench.py) == vamb_b200.encode.make_dataloader tensors."""
    pytest.importorskip("vamb_b200._lib")  # needs the built extension to import the package (no device needed)
    import vamb_b200.encode as ve
    from oracle import normalize as onorm
    from oracle import synth

    ab, tnf, lens = synth.make_contigs(3000, 5, seed=4)
    ab[7] = 0.0  # an all-zero abundance row takes the 1/S branch (vamb/encode.py:108-113)
    want = ve.make_dataloader(ab.copy(), tnf.copy(), lens).dataset.tensors
    got = onorm.normalize(ab, tnf, lens)
    for x, y in zip(got, want):
        assert np.array_equal(x, y.numpy())


def test_normalize_restatement_matches_the_live_reference():
    """oracle/normalize.py == the reference's make_dataloader tensors (tests/golden/ref_dataloader_*.npz)."""
    from oracle import normalize as onorm

    name = "synth_2000x3"
    g = np.load(os.path.join(GOLDEN, f"ref_dataloader_{name}.npz"))
    ab, tnf, lens = mgr.dataloader_inputs(name)
    for k, x in zip("dtaw", onorm.normalize(ab, tnf, lens)):
        mgr.assert_digest_and_sample(g, k, x)


def test_vae_oracle_equals_live_reference_over_training_steps():
    """Under the same ``torch.manual_seed`` stream the oracle and the unmodified reference stay bit-identical
    (losses, every parameter and buffer, encode) over 6 optimiser steps (tests/golden/ref_vae_steps.npz)."""
    from oracle import normalize as onorm

    c = mgr.VAE_STEPS
    g = np.load(os.path.join(GOLDEN, "ref_vae_steps.npz"))
    S, n, batch, seed = c["S"], c["n"], c["batch"], c["seed"]
    rpkm, tnfs, lens = vae_inputs(S, n, seed)
    d, t, a, w = (torch.from_numpy(x) for x in onorm.normalize(rpkm, tnfs, lens))
    o = vo.OracleVAE(S, nhiddens=c["nhiddens"], nlatent=c["nlatent"], seed=seed)
    rng = np.random.default_rng(seed)
    for step in range(c["nsteps"]):
        idx = torch.from_numpy(rng.choice(n, size=batch, replace=False).astype(np.int64))
        torch.manual_seed(c["torch_seed0"] + step)
        lo, _, _ = o.train_step(d[idx], t[idx], a[idx], w[idx])
        assert lo == list(g["losses"][step]), (step, lo, g["losses"][step])
    state_keys = sorted(k[len("state."):] for k in g.files if k.startswith("state."))
    assert state_keys == sorted(o.state)
    for k in state_keys:
        assert mgr.sha256(o.state[k].numpy()) == str(g[f"state.{k}"]), k  # every parameter and buffer, bit for bit
    mgr.assert_digest_and_sample(g, "latent", o.encode(d, t, a, batch=batch)[0])


def test_strict_rng_emulation_follows_the_live_reference_trainmodel():
    """``vamb_b200.encode.reference_epoch_noise`` (the strict-RNG parity mode of the CUDA path) consumes torch's global
    generator exactly like the reference's DataLoader + forward pass: driving the (bit-exact) oracle with it reproduces
    the per-epoch losses that the unmodified ``VAE.trainmodel`` logs, including a batch-size doubling
    (tests/golden/ref_trainmodel_losses.npz)."""
    pytest.importorskip("vamb_b200._lib")

    import vamb_b200.encode as ve
    from oracle import normalize as onorm
    from oracle import synth

    c = mgr.TRAINMODEL
    S, n, seed, nepochs, bsteps = c["S"], c["n"], c["seed"], c["nepochs"], c["batchsteps"]
    ab, tnf, lens = synth.make_contigs(n, S, seed=c["data_seed"])
    want = np.load(os.path.join(GOLDEN, "ref_trainmodel_losses.npz"))["epoch_loss"].tolist()
    assert len(want) == nepochs

    d, t, a, w = (torch.from_numpy(x) for x in onorm.normalize(ab, tnf, lens))
    o = vo.OracleVAE(S, nhiddens=c["nhiddens"], nlatent=c["nlatent"], seed=seed)  # torch.manual_seed(seed) + the reference's init draws
    batch, got = c["batch"], []
    for epoch in range(nepochs):
        if epoch in bsteps:
            batch *= 2
        tot, k = 0.0, 0
        for idx, eps, keeps in ve.reference_epoch_noise(n, batch, n > batch, o.nhiddens, o.nlatent, o.dropout):
            lo, _, _ = o.train_step(d[idx], t[idx], a[idx], w[idx], eps=eps, keeps=keeps)
            tot += lo[0]
            k += 1
        got.append(tot / k)
    assert [f"{x:.5e}" for x in got] == [f"{x:.5e}" for x in want], (got, want)
