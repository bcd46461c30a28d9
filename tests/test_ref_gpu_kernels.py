"""The reference's own GPU bucket kernels (oracle/_ref/libblitzar_ref_gpu.so, SURVEY §8c / Appendix
B) on the same B200, same inputs: results must agree with ours, and the timings are the
GPU-vs-GPU comparison quoted in RESULTS.md. The test compares with the results those kernels gave
on its inputs, stored in tests/golden/ref_gpu_kernels.npz (tests/golden/make_golden.py ref_gpu).
Run as a script for the C2-size numbers (needs oracle/_ref):
    python tests/test_ref_gpu_kernels.py [log2 n]"""
import os
import sys
import time

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gpu_kernels.npz")
SIZES = (1, 50, 191, 193, 20000)


def _inputs(bb, n, seed=5):
    rng = np.random.default_rng(seed)
    gens = bb.get_generators(n, 0)
    s = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    s[:, 31] &= 0x0f
    return gens, s


def test_reference_gpu_kernels_agree(bb):
    z = np.load(GOLDEN)
    for n in SIZES:
        gens, s = _inputs(bb, n, seed=n)
        want = z[f"n{n}"]  # ristretto compression of the reference GPU result
        got = bb.compute_pedersen_commitments(0, [(s, 0)], gens)
        assert np.array_equal(got, want), n


if __name__ == "__main__":
    import torch
    import blitzar_b200 as bb
    from oracle import refcpu, refgpu
    bb.sxt_init()
    for logn in ([int(a) for a in sys.argv[1:]] or [16, 18, 20]):
        n = 1 << logn
        gens, s = _inputs(bb, n)
        g = torch.empty((n, 160), dtype=torch.uint8).pin_memory(); g.numpy()[:] = gens
        sc = torch.empty((n, 32), dtype=torch.uint8).pin_memory(); sc.numpy()[:] = s
        best = (1e9, 1e9)
        for _ in range(3):
            p3, whole, kern = refgpu.bucket_msm(g.numpy(), sc.numpy())
            best = min(best, (whole, kern))
        ours = 1e9
        for _ in range(5):
            t = time.perf_counter()
            out = bb.compute_pedersen_commitments(0, [(sc.numpy(), 0)], g.numpy())
            ours = min(ours, (time.perf_counter() - t) * 1e3)
        same = np.array_equal(out, refcpu.normalize(0, p3))
        print(f"n=2^{logn}: reference kernels {best[1]:.2f} ms (+copies {best[0]:.2f} ms, "
              f"{n / best[0] * 1e3:.3e} terms/s) | this library, whole C-ABI call {ours:.2f} ms "
              f"({n / ours * 1e3:.3e} terms/s) | ratio {best[0] / ours:.1f}x | same result: {same}",
              flush=True)
