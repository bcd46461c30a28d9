"""Inner-product argument (sxt_curve25519_prove_inner_product / _verify_): byte-exact against the
reference's cpu backend — committed fixtures generated from it by tests/golden/make_golden.py
(inner_product.npz: proofs and verification; inner_product_seeded.npz: proofs of seeded_cases).
Mirrors cbindings/inner_product_proof.t.cc (prove then verify, tampered inputs are rejected).
The C port of the oracle restates the protocol too and is pinned on the same fixtures."""
import os

import numpy as np
import pytest

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = os.path.join(GOLDEN_DIR, "inner_product.npz")
SEEDED_GOLDEN = os.path.join(GOLDEN_DIR, "inner_product_seeded.npz")
L = 2**252 + 27742317777372353535851937790883648493


def _check_against_fixture(engine):
    z = np.load(GOLDEN)
    off = int(z["generators_offset"])
    for ci in range(int(z["num_cases"])):
        a, b = z[f"a{ci}"], z[f"b{ci}"]
        t = z[f"t0_{ci}"].copy()
        lv, rv, ap = engine.prove_inner_product(t, a, b, off)
        assert np.array_equal(lv, z[f"l{ci}"]) and np.array_equal(rv, z[f"r{ci}"]), ci
        assert np.array_equal(ap, z[f"ap{ci}"]), ci
        assert np.array_equal(t, z[f"t1_{ci}"]), ci  # transcript advanced identically
        tv = z[f"t0_{ci}"].copy()
        assert engine.verify_inner_product(tv, b, z[f"product{ci}"], z[f"acommit{ci}"], lv, rv, ap,
                                           off) == 1, ci
        assert np.array_equal(tv, z[f"t1_{ci}"]), ci
        # tampering: product, ap, an L value, b
        bad = z[f"product{ci}"].copy()
        bad[0] ^= 1
        assert engine.verify_inner_product(z[f"t0_{ci}"].copy(), b, bad, z[f"acommit{ci}"], lv, rv,
                                           ap, off) == 0, ci
        if len(lv):
            lbad = lv.copy()
            lbad[0] = z[f"r{ci}"][0]
            assert engine.verify_inner_product(z[f"t0_{ci}"].copy(), b, z[f"product{ci}"],
                                               z[f"acommit{ci}"], lbad, rv, ap, off) == 0, ci


def test_oracle_port_matches_reference_fixture(port):
    _check_against_fixture(port)


# (rng seed, sizes, generators offset) of the seeded cases; the reference's proofs of them and its
# transcripts are in inner_product_seeded.npz
SEEDED = {"port": (15, (1, 2, 7, 12), 4), "emul": (5, (3, 8, 21), 2)}


def seeded_cases(name):
    """Yields (key, a, b, generators offset): scalars reduced mod l."""
    seed, sizes, off = SEEDED[name]
    rng = np.random.default_rng(seed)
    for n in sizes:
        av = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
        bv = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
        a = np.array([list(v.to_bytes(32, "little")) for v in av], dtype=np.uint8)
        b = np.array([list(v.to_bytes(32, "little")) for v in bv], dtype=np.uint8)
        yield f"{name}{n}", a, b, off


def _check_against_seeded(engine, name):
    z = np.load(SEEDED_GOLDEN)
    for key, a, b, off in seeded_cases(name):
        t = z["transcript_live"].copy()
        got = engine.prove_inner_product(t, a, b, off)
        want = (z[f"{key}_l"], z[f"{key}_r"], z[f"{key}_ap"])
        assert all(np.array_equal(x, y) for x, y in zip(want, got)), key
        assert np.array_equal(t, z[f"{key}_t1"]), key


def test_oracle_port_matches_reference_live(port):
    assert np.array_equal(port.transcript_new(b"xyz"), np.load(SEEDED_GOLDEN)["transcript_xyz"])
    _check_against_seeded(port, "port")


def test_emulated_pipeline_matches_reference_fixture(emul):
    _check_against_fixture(emul)


def test_emulated_pipeline_matches_oracle_port_live(emul, port):
    rng = np.random.default_rng(25)
    for n in (4, 9, 33):
        a = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        b = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        a[:, 31] &= 0x0F
        b[:, 31] &= 0x0F
        t0 = port.transcript_new(b"emul-live")
        t1, t2 = t0.copy(), t0.copy()
        want = port.prove_inner_product(t1, a, b, 1)
        got = emul.prove_inner_product(t2, a, b, 1)
        assert all(np.array_equal(x, y) for x, y in zip(want, got)) and np.array_equal(t1, t2)


def test_emulated_pipeline_matches_reference_live(emul):
    _check_against_seeded(emul, "emul")


@pytest.mark.gpu
def test_gpu_matches_reference_fixture(bb):
    _check_against_fixture(bb)


@pytest.mark.gpu
def test_gpu_matches_oracle_port_live(bb, port):
    rng = np.random.default_rng(35)
    for n in (6, 50, 300):
        a = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        b = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        a[:, 31] &= 0x0F
        b[:, 31] &= 0x0F
        t0 = port.transcript_new(b"gpu-live")
        t1, t2 = t0.copy(), t0.copy()
        want = port.prove_inner_product(t1, a, b, 70)  # straddles the 64 precomputed generators
        got = bb.prove_inner_product(t2, a, b, 70)
        assert all(np.array_equal(x, y) for x, y in zip(want, got)) and np.array_equal(t1, t2)


@pytest.mark.gpu
def test_gpu_prove_verify_roundtrip_larger(bb, port):
    rng = np.random.default_rng(6)
    n = 3000
    av = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
    bv = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
    a = np.array([list(v.to_bytes(32, "little")) for v in av], dtype=np.uint8)
    b = np.array([list(v.to_bytes(32, "little")) for v in bv], dtype=np.uint8)
    t = np.zeros(203, dtype=np.uint8)
    t[:19] = [1, 168, 1, 0, 1, 96, 83, 84, 82, 79, 66, 69, 118, 49, 46, 48, 46, 50, 0]
    t0 = t.copy()
    lv, rv, ap = bb.prove_inner_product(t, a, b, 0)
    prod = sum(x * y for x, y in zip(av, bv)) % L
    pb = np.array(list(prod.to_bytes(32, "little")), dtype=np.uint8)
    h = bb.MultiexpHandle(0, bb.get_generators(n, 0))
    acommit = h.fixed_multiexponentiation(32, 1, n, a)[0]
    h.free()
    assert bb.verify_inner_product(t0.copy(), b, pb, acommit, lv, rv, ap, 0) == 1
    pb[3] ^= 4
    assert bb.verify_inner_product(t0.copy(), b, pb, acommit, lv, rv, ap, 0) == 0
