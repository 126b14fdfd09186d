"""TEST INFRASTRUCTURE ONLY -- the CPU oracle for the vamb hot path.

Nothing under ``oracle/`` is product code.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it, and only as the checker.  The product
package (``vamb_b200``) never imports this package and fails loudly when its
CUDA extension is missing.

Contents
--------
ref_loader.py      load the UNMODIFIED reference files from /root/reference
                   (present in the build container only) under a stub ``vamb``
                   package with two shims (vambcore, dadaptation).
dadapt.py          restatement of dadaptation==3.2 DAdaptAdam (parity unpinned:
                   upstream source is not available offline).
vambcore_shim.py   restatement of vambcore.overwrite_matrix semantics.
cluster_oracle.py  restatement of vamb/cluster.py with the *defined* arithmetic
                   contract (sequential-FMA distances, exact integer density and
                   histogram sums) that the CUDA kernels implement bit-exactly.
vae_oracle.py      torch-CPU fp32 restatement of vamb/encode.py (forward, loss,
                   analytic backward, DAdaptAdam step, encode).
csrc/oracle_kernels.c   the C inner loops of cluster_oracle (gcc, -ffp-contract=off).
make_golden.py     runs the real reference (via ref_loader) and writes
                   tests/golden/*.npz; committed together with its outputs.
numerics.py        pins torch's CPU arithmetic so that bit-exact fixtures hold on
                   any x86-64 host (called by tests/conftest.py and the writers).
make_golden_reference.py   the same for the reference's dataloader, VAE steps,
                   trainmodel losses and clusters of its own test fixture.
"""
