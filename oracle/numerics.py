"""TEST INFRASTRUCTURE -- one CPU arithmetic for the torch-CPU oracle and the fixtures it is held to.

torch's float32 results on the CPU depend on the host: MKL picks a GEMM code path per processor, ATen's
vectorised kernels (reductions, exp, log) use the widest SIMD the processor has, and both split work by the
thread count; each of these moves the last bits.  The VAE fixtures in tests/golden/ are compared bit for bit,
so they are written and checked under one setting that any x86-64 host runs alike: MKL's compatible code
path, ATen's AVX2 kernels and eight threads.  One thread would be reproducible too, but its single long
accumulation over a 4096-row batch moves gradients by ~1e-3, too coarse for the GPU tests that compare
with the oracle.  MKL and ATen fix their choice at the first CPU operation of the process, so ``pin()``
must run before it (the test suite's conftest.py calls it first thing).
"""
import os

THREADS = 8  # fixed, not the host's core count: the split of a reduction over threads moves its last bits


def pin() -> None:
    os.environ["MKL_CBWR"] = "COMPATIBLE"
    os.environ["ATEN_CPU_CAPABILITY"] = "avx2"
    import torch

    torch.set_num_threads(THREADS)
    got = torch.backends.cpu.get_cpu_capability()
    if got != "AVX2":
        raise RuntimeError(f"torch CPU kernels are {got}, not AVX2: a CPU operation ran before oracle.numerics.pin()")
