"""The oracle itself: pinned against the reference's golden vector and the committed fixtures that
were generated from the reference's own CPU implementation (tests/golden/make_golden.py)."""
import os

import numpy as np

from tests import common

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_port_reproduces_reference_golden_commitments(port):
    out = port.commit(0, common.golden_columns())
    assert out.tolist() == common.GOLDEN_COMMITMENTS


def test_port_matches_committed_reference_fixtures(port):
    for curve in range(4):
        z = np.load(os.path.join(GOLDEN_DIR, f"commit_curve{curve}.npz"))
        cols = [(z[f"col{j}"], int(z["signed"][j])) for j in range(len(z["signed"]))]
        out = port.commit(curve, cols, z["generators"])
        assert common.same(curve, out, z["commitments"]), curve
        f = np.load(os.path.join(GOLDEN_DIR, f"fixed_curve{curve}.npz"))
        res = port.fixed_msm(curve, f["generators_p"], int(f["num_outputs"]), int(f["n"]),
                             f["scalars"], element_num_bytes=int(f["element_num_bytes"]))
        assert common.same(curve, port.normalize(curve, res), f["normalized"]), curve
        res = port.fixed_msm(curve, f["generators_p"], len(f["bit_table"]), int(f["n"]),
                             f["packed_scalars"], output_bit_table=f["bit_table"].tolist())
        assert common.same(curve, port.normalize(curve, res), f["packed_normalized"]), curve


def test_builtin_generators_fixture(port):
    z = np.load(os.path.join(GOLDEN_DIR, "ristretto_generators.npz"))
    g = port.ristretto_generators(int(z["n"]), int(z["offset"]))
    assert np.array_equal(port.normalize(0, g), z["compressed"])


def seeded_cases(port):
    """Per curve: (curve, commit generators, projective generators, columns, fixed-MSM scalars).
    tests/golden/make_golden.py runs the reference on the same cases (oracle_cases.npz)."""
    rng = np.random.default_rng(11)
    for curve in range(4):
        gens, gens_p = common.generators_for(port, curve, 120)
        cols = common.random_columns(rng, 120, [(0, 32, 0), (-7, 16, 1), (0, 3, 0), (-119, 32, 0),
                                                 (-120, 8, 0)]) + common.edge_case_columns()
        sc = rng.integers(0, 256, (40, 3 * 5), dtype=np.uint8)
        yield curve, gens, gens_p[:40], cols, sc


def test_port_matches_reference_live(port):
    z = np.load(os.path.join(GOLDEN_DIR, "oracle_cases.npz"))
    for curve, gens, gens_p, cols, sc in seeded_cases(port):
        assert common.same(curve, port.commit(curve, cols, gens), z[f"commit{curve}"])
        a = port.fixed_msm(curve, gens_p, 3, 40, sc, element_num_bytes=5)
        assert common.same(curve, port.normalize(curve, a), z[f"fixed{curve}"])
        # the two normalisers agree on the same projective input
        assert common.same(curve, port.normalize(curve, a), z[f"normalized_port_fixed{curve}"])


def test_reference_fixed_pedersen_vectors(port):
    """cbindings/fixed_pedersen.t.cc:45-135: {1,0,0,2} (1-byte x 2 outputs... as 2-byte scalars)
    gives g0 + 512 g1; packed {0b1010, 0b0101} with bit table {3,1} gives 2 g0 + 5 g1 and g0."""
    g = port.ristretto_generators(2, 0)
    # one output, element_num_bytes = 2, rows {1,0} and {0,2}: g0*1 + g1*(2<<8)
    res = port.fixed_msm(0, g, 1, 2, np.array([1, 0, 0, 2], dtype=np.uint8), element_num_bytes=2)
    want = port.commit(0, [(np.array([[1, 0], [0, 2]], dtype=np.uint8), 0)], g)
    assert np.array_equal(port.normalize(0, res), want)
    res = port.fixed_msm(0, g, 2, 2, np.array([0b1010, 0b0101], dtype=np.uint8),
                         output_bit_table=[3, 1])
    want = port.commit(0, [(np.array([[2], [5]], dtype=np.uint8), 0),
                           (np.array([[1], [0]], dtype=np.uint8), 0)], g)
    assert np.array_equal(port.normalize(0, res), want)
