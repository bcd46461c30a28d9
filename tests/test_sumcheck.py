"""Sumcheck prover (sxt_prove_sumcheck / b200_prove_sumcheck_device) over both sumcheck fields.

tests/golden/sumcheck.npz holds the reference cpu backend's proofs
(tests/golden/make_sumcheck_golden.py) of the cases below: only their specs and the outputs are stored, the inputs are
regenerated from the seeds. The reference, the pure-Python prover here, the emulated kernels and the
GPU are all driven by the same callback (`Challenger`), so every proof must match byte for byte."""
import hashlib
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sumcheck.npz")
SCALAR255, GRUMPKIN = 0, 1
MODULUS = {SCALAR255: 2**252 + 27742317777372353535851937790883648493,
           GRUMPKIN: 21888242871839275222246405745257275088548364400416034343698204186575808495617}
R = 2**256  # Montgomery radix of the grumpkin ABI form


def to_abi(field_id, x):
    """Canonical integer -> 32 ABI bytes (plain for scalar255, Montgomery for grumpkin)."""
    if field_id == GRUMPKIN:
        x = x * R % MODULUS[GRUMPKIN]
    return x.to_bytes(32, "little")


def from_abi(field_id, b):
    x = int.from_bytes(bytes(b), "little")
    if field_id == GRUMPKIN:
        x = x * pow(R, -1, MODULUS[GRUMPKIN]) % MODULUS[GRUMPKIN]
    return x


class Challenger:
    """The transcript callback: r_k = SHA-256(label | k as u32 LE | polynomial bytes) mod p, in the
    field's ABI form. Records every polynomial it is shown."""

    def __init__(self, field_id, label=b"blitzar-b200 sumcheck test"):
        self.field_id, self.label, self.seen = field_id, label, []

    def __call__(self, polynomial):
        poly = np.asarray(polynomial, dtype=np.uint8).copy()
        k = len(self.seen)
        self.seen.append(poly)
        h = hashlib.sha256(self.label + k.to_bytes(4, "little") + poly.tobytes()).digest()
        return to_abi(self.field_id, int.from_bytes(h, "little") % MODULUS[self.field_id])


# ---- cases --------------------------------------------------------------------------------------
def _spec(name, seed, n, num_mles, lengths, terms, round_degree=None, zero=(), mle_values=None,
          mults=None):
    return dict(name=name, seed=seed, n=n, num_mles=num_mles, lengths=list(lengths),
                terms=list(terms), round_degree=round_degree or max(lengths), zero=list(zero),
                mle_values=mle_values, mults=mults)


def case_specs():
    specs = [
        # cbindings/sumcheck.t.cc: n = 2, one MLE {8, 3}, one product of length 1 -> p = {8, 3 - 8}
        _spec("ref_t", 0, 2, 1, [1], [0], mle_values=[[8, 3]], mults=[1]),
    ]
    for i, n in enumerate([1, 2, 3, 5, 8, 37]):
        specs.append(_spec(f"n{n}", 100 + i, n, 3, [2, 1, 3], [0, 1, 2, 1, 0, 2]))
    for m in range(1, 8):
        lengths = [min(m, 5)] + ([2] if m > 1 else [])
        terms = list(range(min(m, 5))) + ([m - 1, m - 2] if m > 1 else [])
        specs.append(_spec(f"mles{m}", 200 + m, 29, m, lengths, terms))
    # mixed lengths 1..5, a repeated index (a square), a zero multiplier, round_degree above the
    # longest product
    specs.append(_spec("mixed", 300, 45, 5, [1, 2, 3, 4, 5, 2],
                       [4, 0, 0, 1, 2, 3, 0, 1, 3, 3, 0, 1, 2, 3, 4, 2, 2], round_degree=7,
                       zero=[3]))
    specs.append(_spec("large", 400, (1 << 18) + 3, 3, [2, 1], [0, 1, 2]))
    return specs


def case_inputs(field_id, spec):
    """(mles uint8 [num_mles, n, 32], product_table [(mult bytes, length)], terms) from the spec."""
    p = MODULUS[field_id]
    rng = np.random.default_rng(spec["seed"] * 2 + field_id)
    n, m, lengths = spec["n"], spec["num_mles"], spec["lengths"]
    raw = rng.integers(0, 256, (m, n, 32), dtype=np.uint8)
    mult_raw = rng.integers(0, 256, (len(lengths), 32), dtype=np.uint8)
    if spec["mle_values"] is not None:
        values = [[int(x) for x in col] for col in spec["mle_values"]]
    else:
        values = [[int.from_bytes(raw[j, i].tobytes(), "little") % p for i in range(n)]
                  for j in range(m)]
    if spec["mults"] is not None:
        mults = list(spec["mults"])
    else:
        mults = [int.from_bytes(mult_raw[k].tobytes(), "little") % p for k in range(len(lengths))]
    for k in spec["zero"]:
        mults[k] = 0
    mles = np.frombuffer(b"".join(to_abi(field_id, x) for col in values for x in col),
                         dtype=np.uint8).reshape(m, n, 32)
    table = [(to_abi(field_id, mults[k]), lengths[k]) for k in range(len(lengths))]
    return mles, table, list(spec["terms"]), values, mults


# ---- pure-Python restatement of the prover (integer arithmetic) -----------------------------------
def _products(lengths, terms):
    out, t = [], 0
    for length in lengths:
        out.append(terms[t:t + length])
        t += length
    return out


def python_prove(field_id, values, mults, lengths, terms, round_degree, callback):
    """sum_k mult_k prod_j f_j over max(ceil_log2(n), 1) rounds; returns (polynomials as ABI bytes
    [v, d + 1, 32], evaluation point [v, 32])."""
    p = MODULUS[field_id]
    f = [list(col) for col in values]
    n = len(f[0]) if f else 0
    v = max((n - 1).bit_length(), 1)
    prods = _products(lengths, terms)
    polys = np.zeros((v, round_degree + 1, 32), dtype=np.uint8)
    point = np.zeros((v, 32), dtype=np.uint8)
    for rnd in range(v):
        mid = 1 << (v - 1 - rnd)
        coeffs = [0] * (round_degree + 1)
        for i in range(mid):
            for mult, idx in zip(mults, prods):
                c = [mult]
                for j in idx:
                    a = f[j][i] if i < len(f[j]) else 0
                    b = (f[j][i + mid] if i + mid < len(f[j]) else 0) - a
                    nc = [0] * (len(c) + 1)
                    for d, x in enumerate(c):
                        nc[d] = (nc[d] + x * a) % p
                        nc[d + 1] = (nc[d + 1] + x * b) % p
                    c = nc
                for d, x in enumerate(c):
                    coeffs[d] = (coeffs[d] + x) % p
        poly = np.frombuffer(b"".join(to_abi(field_id, x) for x in coeffs),
                             dtype=np.uint8).reshape(-1, 32)
        polys[rnd] = poly
        rb = callback(poly)
        point[rnd] = np.frombuffer(bytes(rb), dtype=np.uint8)
        r = from_abi(field_id, rb)
        if rnd < v - 1:
            f = [[((1 - r) * col[i] + r * (col[i + mid] if i + mid < len(col) else 0)) % p
                  for i in range(mid)] for col in f]
    return polys, point


# ---- golden data ---------------------------------------------------------------------------------
def golden_cases():
    z = np.load(GOLDEN)
    for key in sorted(k for k in z.files if k.endswith("_spec")):
        spec = json.loads(bytes(z[key]).decode())
        field_id = int(key.split("_")[0][1:])
        pre = key[:-len("spec")]
        yield field_id, spec, z[pre + "polys"], z[pre + "point"]


def golden_key(field_id, spec):
    return f"f{field_id}_{spec['name']}_"


def make_fixture(prove):
    """{key: array} of the sumcheck fixture, proofs by `prove` (the reference's cpu prover)."""
    out = {}
    for field_id in (SCALAR255, GRUMPKIN):
        for spec in case_specs():
            mles, table, terms, _, _ = case_inputs(field_id, spec)
            ch = Challenger(field_id)
            polys, point = prove(field_id, mles, table, terms, ch, spec["round_degree"])
            assert all(np.array_equal(a, b) for a, b in zip(ch.seen, polys))
            key = golden_key(field_id, spec)
            out[key + "spec"] = np.frombuffer(json.dumps(spec, sort_keys=True).encode(), np.uint8)
            out[key + "polys"] = polys
            out[key + "point"] = point
    return out


def _run_case(prove, field_id, spec, polys, point):
    mles, table, terms, _, _ = case_inputs(field_id, spec)
    ch = Challenger(field_id)
    got_polys, got_point = prove(field_id, mles, table, terms, ch, spec["round_degree"])
    assert np.array_equal(got_polys, polys), spec["name"]
    assert np.array_equal(got_point, point), spec["name"]
    assert len(ch.seen) == len(polys) and all(np.array_equal(a, b) for a, b in zip(ch.seen, polys))


def test_golden_matches_specs():
    """The fixture covers exactly the cases defined here, for both fields."""
    have = {(f, json.dumps(s, sort_keys=True)) for f, s, _, _ in golden_cases()}
    want = {(f, json.dumps(s, sort_keys=True)) for f in (SCALAR255, GRUMPKIN)
            for s in case_specs()}
    assert have == want


def test_reference_unit_case():
    """cbindings/sumcheck.t.cc: p_0 = {8, 3 - 8}."""
    for field_id, spec, polys, _ in golden_cases():
        if spec["name"] == "ref_t":
            p = MODULUS[field_id]
            assert from_abi(field_id, polys[0, 0]) == 8
            assert from_abi(field_id, polys[0, 1]) == (3 - 8) % p


def test_python_prover_reproduces_golden():
    def prove(field_id, mles, table, terms, ch, round_degree):
        spec = current[0]
        _, _, _, values, mults = case_inputs(field_id, spec)
        return python_prove(field_id, values, mults, spec["lengths"], terms, round_degree, ch)

    current = [None]
    for field_id, spec, polys, point in golden_cases():
        current[0] = spec
        _run_case(prove, field_id, spec, polys, point)


@pytest.fixture(scope="module")
def emul_sc():
    """The emulated sumcheck prover (tests/emul/emul_sumcheck.cpp) — test infrastructure."""
    from tests.emul import sumcheck_harness
    return sumcheck_harness


def test_emulated_kernels_reproduce_golden(emul_sc):
    """Round 0 (sum of the plain / Montgomery input), the fold + sum of every later round, the
    grid-stride rounds of the large case and the one-block tail rounds."""
    for field_id, spec, polys, point in golden_cases():
        _run_case(emul_sc.prove_sumcheck, field_id, spec, polys, point)


def test_validation_codes(emul_sc):
    ok = dict(field_id=0, n=4, num_mles=2, product_table=[(bytes(32), 2), (bytes(32), 1)],
              product_terms=[0, 1, 1], round_degree=2)
    assert emul_sc.sumcheck_check(**ok) == 0
    assert emul_sc.sumcheck_check(**{**ok, "field_id": 1}) == 0

    def code(**kw):
        return emul_sc.sumcheck_check(**{**ok, **kw})

    codes = {
        "field": code(field_id=2),
        "n": code(n=0),
        "degree0": code(product_table=[], product_terms=[], round_degree=0),
        "length0": code(product_table=[(bytes(32), 0), (bytes(32), 3)]),
        "above_degree": code(product_table=[(bytes(32), 3), (bytes(32), 0)], product_terms=[0, 1, 1]),
        "above_cap": code(product_table=[(bytes(32), 6)], product_terms=[0] * 6, round_degree=6),
        "term_count": code(product_terms=[0, 1]),
        "term_index": code(product_terms=[0, 1, 2]),
    }
    assert all(c != 0 for c in codes.values()), codes
    assert len(set(codes.values())) == len(codes), codes
    # the grumpkin table stride (40 bytes) is honoured
    assert code(field_id=1, product_table=[(bytes(32), 2), (bytes(32), 4)]) == codes["above_degree"]


# ---- GPU -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_matches_golden(bb):
    for field_id, spec, polys, point in golden_cases():
        _run_case(bb.prove_sumcheck, field_id, spec, polys, point)


@pytest.mark.gpu
def test_gpu_device_resident_matches_golden(bb):
    def prove(field_id, mles, table, terms, ch, round_degree):
        buf = bb.DeviceBuffer(host=np.ascontiguousarray(mles))
        try:
            return bb.prove_sumcheck_device(field_id, buf.ptr, mles.shape[1], mles.shape[0], table,
                                            terms, ch, round_degree)
        finally:
            buf.free()

    for field_id, spec, polys, point in golden_cases():
        _run_case(prove, field_id, spec, polys, point)


def _mle_eval(p, col, rs):
    """f(r_0, ..., r_{v-1}) with r_0 folding the top half first (the prover's order)."""
    f = list(col)
    for r in rs:
        mid = 1 << max((len(f) - 1).bit_length() - 1, 0)
        f = [((1 - r) * f[i] + r * (f[i + mid] if i + mid < len(f) else 0)) % p for i in range(mid)]
    return f[0]


def _poly_eval(p, coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % p
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("field_id", [SCALAR255, GRUMPKIN])
def test_gpu_large_verifier_identities(bb, field_id):
    """n = 2^20 + 5, degree 4: p_0(0) + p_0(1) is the full sum, p_k(0) + p_k(1) = p_{k-1}(r_{k-1}),
    and p_last(r_last) is the polynomial evaluated at the MLEs' values at r."""
    spec = _spec("big", 900, (1 << 20) + 5, 4, [4, 3, 1], [0, 1, 2, 3, 3, 3, 1, 2])
    p = MODULUS[field_id]
    mles, table, terms, values, mults = case_inputs(field_id, spec)
    polys, point = bb.prove_sumcheck(field_id, mles, table, terms, Challenger(field_id))
    coeffs = [[from_abi(field_id, c) for c in poly] for poly in polys]
    rs = [from_abi(field_id, x) for x in point]
    prods = _products(spec["lengths"], terms)
    total = 0
    for i in range(spec["n"]):
        for mult, idx in zip(mults, prods):
            t = mult
            for j in idx:
                t = t * values[j][i] % p
            total += t
    assert (coeffs[0][0] + sum(coeffs[0])) % p == total % p
    for k in range(1, len(coeffs)):
        assert (coeffs[k][0] + sum(coeffs[k])) % p == _poly_eval(p, coeffs[k - 1], rs[k - 1]), k
    fr = [_mle_eval(p, col, rs) for col in values]
    want = 0
    for mult, idx in zip(mults, prods):
        t = mult
        for j in idx:
            t = t * fr[j] % p
        want += t
    assert _poly_eval(p, coeffs[-1], rs[-1]) == want % p


@pytest.mark.gpu
def test_gpu_other_entry_points_after_sumcheck(bb):
    """A sumcheck leaves the shared stream, pool and lock clean: a commitment and an inner-product
    proof afterwards still match their fixtures."""
    for field_id, spec, polys, point in golden_cases():
        if spec["name"] == "mixed":
            _run_case(bb.prove_sumcheck, field_id, spec, polys, point)
    gdir = os.path.dirname(GOLDEN)
    z = np.load(os.path.join(gdir, "commit_curve0.npz"))
    cols = [(z[f"col{j}"], int(s)) for j, s in enumerate(z["signed"])]
    assert np.array_equal(bb.compute_pedersen_commitments(0, cols, z["generators"]),
                          z["commitments"])
    z = np.load(os.path.join(gdir, "inner_product.npz"))
    t = z["t0_0"].copy()
    lv, rv, ap = bb.prove_inner_product(t, z["a0"], z["b0"], int(z["generators_offset"]))
    assert np.array_equal(lv, z["l0"]) and np.array_equal(rv, z["r0"])
    assert np.array_equal(ap, z["ap0"]) and np.array_equal(t, z["t1_0"])
