"""Parity at BASELINE.json sizes: the CUDA path (through the C ABI) against the reference's own
cpu backend on the benchmark inputs of SURVEY §8(d) — not self-consistency. The reference's results
on these seeded inputs are stored in tests/golden/baseline_sizes.npz (tests/golden/make_golden.py).

  C1  ristretto255, built-in generators, n = 2^16, mt19937{0} scalars           vs reference, full
  C2  ristretto255, explicit generators g(0..2^20), 252-bit scalars, n = 2^20   vs reference, full
  C3  bls12-381 G1, the reference's per-index generators (distinct points)      vs reference at 2^18
      and at the full 2^22 through the closed form sum_i s_i G_i = (sum_i s_i k_i mod r) G with ONE
      reference scalar multiplication (tests/common.py)
  C5  bn254 G1 fixed-base MSM over a handle of distinct generators               vs reference at 2^18,
      closed form at 2^22
The generators come from the device (b200_synthetic_generators_device) and are pinned against the
reference's generate_random_element at sample indices first. Projective results are normalised by
the oracle port, whose normaliser tests/test_oracle.py pins against the reference's.
"""
import os

import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "baseline_sizes.npz")
# (first index, offsets) at which the synthetic generators are compared with the reference's
GENERATOR_SAMPLES = ((0, 999_983, (1 << 24) - (1 << 12)), (0, 1, 1 << 11, (1 << 12) - 1))
C2_GENERATOR_SAMPLES = (0, 77_777, (1 << 20) - 1)


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


@pytest.mark.parametrize("curve", [1, 2, 3])
def test_synthetic_generators_match_the_reference(bb, port, ref, curve):
    n = 1 << 12
    want_af, want_p2 = ref[f"generators_affine{curve}"], ref[f"generators_normalized{curve}"]
    j = 0
    for first in GENERATOR_SAMPLES[0]:
        af = bb.synthetic_generators(curve, n, first, projective=False)
        p2 = bb.synthetic_generators(curve, n, first, projective=True)
        for i in GENERATOR_SAMPLES[1]:
            k = 97 if curve == 1 else 65
            assert np.array_equal(af[i, :k], want_af[j, :k]), (curve, first, i)
            assert common.same(curve, port.normalize(curve, p2[i:i + 1]), want_p2[j:j + 1]), \
                (curve, first, i)
            j += 1
    # distinct points
    assert len({bytes(r) for r in af[:, :32]}) == n


def test_synthetic_ristretto_generators(bb, port, ref):
    g = bb.synthetic_generators(0, 300, 12345)
    assert np.array_equal(port.normalize(0, g), ref["ristretto_generators_300_at_12345"])


def test_c1_builtin_generators_2_16(bb, ref):
    n = 1 << 16
    s = common.mt19937_bytes(0, n)
    got = bb.compute_pedersen_commitments(0, [(s, 0)], None, 0)
    assert np.array_equal(got, ref["c1"])


def test_c2_full_size_against_reference(bb, port, ref):
    n = 1 << 20
    s = common.mt19937_bytes(0, n)
    gens = bb.get_generators(n, 0)
    # the generators handed to the engine are the reference's own at sample indices
    for j, i in enumerate(C2_GENERATOR_SAMPLES):
        assert np.array_equal(port.normalize(0, gens[i:i + 1]), ref["c2_generators"][j:j + 1]), i
    got = bb.compute_pedersen_commitments(0, [(s, 0)], gens)
    want = ref["c2"]
    assert np.array_equal(got, want)
    # same call over the built-in generators (sxt_curve25519_compute_pedersen_commitments)
    assert np.array_equal(bb.compute_pedersen_commitments(0, [(s, 0)], None, 0), want)


def _scalars(n, seed, top_mask):
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    s[:, 31] &= top_mask
    return s


def test_c3_bls12_381_distinct_generators(bb, ref):
    n = 1 << 18
    af = bb.synthetic_generators(1, n, 0, projective=False)
    s = _scalars(n, 3, 0x7F)  # 255-bit
    got = bb.compute_pedersen_commitments(1, [(s, 0)], af)
    assert common.same(1, got, ref["c3"])
    assert common.same(1, got, ref["c3_closed_form"])


def test_c3_full_size_closed_form(bb, ref):
    n = 1 << 22
    buf = bb.DeviceBuffer(n * 104)
    bb.synthetic_generators_device(1, buf.ptr, n, 0, False)
    af = buf.to_host((n, 104))
    buf.free()
    s = _scalars(n, 4, 0x7F)
    got = bb.compute_pedersen_commitments(1, [(s, 0)], af)
    assert common.same(1, got, ref["c3_full_closed_form"])


@pytest.mark.parametrize("curve", [2, 3])
def test_c5_fixed_base_distinct_generators(bb, port, ref, curve):
    n = 1 << 18
    p2 = bb.synthetic_generators(curve, n, 0, projective=True)
    h = bb.MultiexpHandle(curve, p2)
    s = _scalars(n, 5 + curve, 0x3F)
    res = h.fixed_multiexponentiation(32, 1, n, s)
    assert common.same(curve, port.normalize(curve, res), ref[f"c5_{curve}"])
    # two outputs of different widths in one packed call, against the reference's commitments to
    # the 64-bit and 17-bit columns unpacked from the same rows
    res = h.fixed_packed_multiexponentiation(C5_BIT_TABLE, n, c5_packed_scalars(n))
    assert common.same(curve, port.normalize(curve, res), ref[f"c5_{curve}_packed"])
    h.free()


C5_BIT_TABLE = [64, 17]


def c5_packed_scalars(n):
    row = (sum(C5_BIT_TABLE) + 7) // 8
    return np.random.default_rng(9).integers(0, 256, (n, row), dtype=np.uint8)


def test_c5_full_size_closed_form(bb, port, ref):
    n = 1 << 22
    buf = bb.DeviceBuffer(n * 96)
    bb.synthetic_generators_device(2, buf.ptr, n, 0, True)
    p2 = buf.to_host((n, 96))
    buf.free()
    h = bb.MultiexpHandle(2, p2)
    del p2
    s = _scalars(n, 11, 0x3F)
    res = h.fixed_multiexponentiation(32, 1, n, s)
    h.free()
    assert common.same(2, port.normalize(2, res), ref["c5_full_closed_form"])
