"""Generates the committed golden fixtures from the REFERENCE's own CPU implementation
(oracle/_ref, built from the reference's sources by oracle/ref_build/Makefile):

    python tests/golden/make_golden.py [fixture ...] [--out DIR]

(default fixture: commit). `ref_gpu` runs the reference's GPU kernels and so needs a B200.

Inputs are seeded; generators for the Weierstrass curves come from the reference's
fast_random_number_generator{i+1,i+2} -> generate_random_element scheme
(cbindings/pedersen.t.cc:81-123)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refcpu  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    rng = np.random.default_rng(20260922)
    n = 96
    for curve in range(4):
        if curve == 0:
            gens = refcpu.ristretto_generators(n, 7)
            gens_p = gens
        else:
            gens_p, gens = refcpu.random_elements(curve, n, first=5)
        cols = [(rng.integers(0, 256, (n, 32), dtype=np.uint8), 0),
                (rng.integers(0, 256, (n - 5, 16), dtype=np.uint8), 1),
                (rng.integers(0, 256, (n, 1), dtype=np.uint8), 0),
                (rng.integers(0, 256, (1, 8), dtype=np.uint8), 1),
                (np.zeros((0, 4), dtype=np.uint8), 0)]
        out = refcpu.commit(curve, cols, gens)
        np.savez_compressed(os.path.join(HERE, f"commit_curve{curve}.npz"), generators=gens,
                            commitments=out, signed=np.array([c[1] for c in cols]),
                            **{f"col{j}": c[0] for j, c in enumerate(cols)})
        m, outs, nb = 24, 3, 4
        sc = rng.integers(0, 256, (m, outs * nb), dtype=np.uint8)
        res = refcpu.fixed_msm(curve, gens_p[:m], outs, m, sc, element_num_bytes=nb)
        bt = [3, 11, 1, 9]
        row = (sum(bt) + 7) // 8
        psc = rng.integers(0, 256, (m, row), dtype=np.uint8)
        pres = refcpu.fixed_msm(curve, gens_p[:m], len(bt), m, psc, output_bit_table=bt)
        np.savez_compressed(os.path.join(HERE, f"fixed_curve{curve}.npz"), generators_p=gens_p[:m],
                            scalars=sc, num_outputs=outs, n=m, element_num_bytes=nb,
                            normalized=refcpu.normalize(curve, res), bit_table=np.array(bt),
                            packed_scalars=psc, packed_normalized=refcpu.normalize(curve, pres))
    g = refcpu.ristretto_generators(16, 1000)
    np.savez_compressed(os.path.join(HERE, "ristretto_generators.npz"), n=16, offset=1000,
                        compressed=refcpu.normalize(0, g))


def make_inner_product_fixture():
    """tests/golden/inner_product.npz: proofs produced by the reference's cpu backend
    (sxt_curve25519_prove_inner_product semantics) for n = 1, 2, 5, 16, 37 with a transcript
    labelled b"golden-ipa" and generators_offset = 11: inputs, the transcript before / after, the
    proof, <a,b> and the commitment <a, G> that the verifier takes."""
    L = 2**252 + 27742317777372353535851937790883648493
    rng = np.random.default_rng(777)
    out = {}
    cases = [1, 2, 5, 16, 37]
    for ci, n in enumerate(cases):
        av = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
        bv = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(n)]
        a = np.array([list(v.to_bytes(32, "little")) for v in av], dtype=np.uint8)
        b = np.array([list(v.to_bytes(32, "little")) for v in bv], dtype=np.uint8)
        t0 = refcpu.transcript_new(b"golden-ipa")
        t = t0.copy()
        lv, rv, ap = refcpu.prove_inner_product(t, a, b, generators_offset=11)
        prod = sum(x * y for x, y in zip(av, bv)) % L
        np_ = 1 << max(0, (n - 1).bit_length())
        g = refcpu.ristretto_generators(np_, 11)
        acommit = refcpu.fixed_msm(0, g[:n], 1, n, a, element_num_bytes=32)[0]
        out.update({f"n{ci}": n, f"a{ci}": a, f"b{ci}": b, f"t0_{ci}": t0, f"t1_{ci}": t,
                    f"l{ci}": lv, f"r{ci}": rv, f"ap{ci}": ap,
                    f"product{ci}": np.array(list(prod.to_bytes(32, "little")), dtype=np.uint8),
                    f"acommit{ci}": acommit})
    out["num_cases"] = len(cases)
    out["generators_offset"] = 11
    np.savez_compressed(os.path.join(HERE, "inner_product.npz"), **out)


def make_oracle_cases_fixture():
    """tests/golden/oracle_cases.npz: the reference's commitments, fixed-base MSMs and normalisation
    on the seeded cases of tests/test_oracle.py."""
    from oracle import port
    from tests import common, test_oracle
    assert refcpu.commit(0, common.golden_columns()).tolist() == common.GOLDEN_COMMITMENTS
    out = {}
    for curve, gens, gens_p, cols, sc in test_oracle.seeded_cases(port):
        out[f"commit{curve}"] = refcpu.commit(curve, cols, gens)
        b = refcpu.fixed_msm(curve, gens_p, 3, 40, sc, element_num_bytes=5)
        out[f"fixed{curve}"] = refcpu.normalize(curve, b)
        a = port.fixed_msm(curve, gens_p, 3, 40, sc, element_num_bytes=5)
        out[f"normalized_port_fixed{curve}"] = refcpu.normalize(curve, a)
    np.savez_compressed(os.path.join(HERE, "oracle_cases.npz"), **out)


def make_inner_product_seeded_fixture():
    """tests/golden/inner_product_seeded.npz: the reference's proofs of the seeded cases of
    tests/test_inner_product.py, from a transcript labelled b"live"."""
    from tests import test_inner_product as tip
    out = {"transcript_xyz": refcpu.transcript_new(b"xyz"),
           "transcript_live": refcpu.transcript_new(b"live")}
    for name in tip.SEEDED:
        for key, a, b, off in tip.seeded_cases(name):
            t = out["transcript_live"].copy()
            lv, rv, ap = refcpu.prove_inner_product(t, a, b, off)
            out.update({f"{key}_l": lv, f"{key}_r": rv, f"{key}_ap": ap, f"{key}_t1": t})
    np.savez_compressed(os.path.join(HERE, "inner_product_seeded.npz"), **out)


def _baseline_generators(curve):
    from tests import test_gpu_baseline_sizes as t
    af, p2 = [], []
    for first in t.GENERATOR_SAMPLES[0]:
        for i in t.GENERATOR_SAMPLES[1]:
            rp2, raf = refcpu.random_elements(curve, 1, first + i)
            af.append(raf[0])
            p2.append(refcpu.normalize(curve, rp2)[0])
    return {f"generators_affine{curve}": np.array(af), f"generators_normalized{curve}": np.array(p2)}


def _baseline_c1_c2(_):
    from tests import common, test_gpu_baseline_sizes as t
    out = {"ristretto_generators_300_at_12345":
           refcpu.normalize(0, refcpu.ristretto_generators(300, 12345))}
    s = common.mt19937_bytes(0, 1 << 16)
    out["c1"] = refcpu.commit(0, [(s, 0)], None, 0)
    s = common.mt19937_bytes(0, 1 << 20)
    out["c2_generators"] = np.concatenate(
        [refcpu.normalize(0, refcpu.ristretto_generators(1, i)) for i in t.C2_GENERATOR_SAMPLES])
    out["c2"] = refcpu.commit(0, [(s, 0)], refcpu.ristretto_generators(1 << 20, 0))
    return out


def _baseline_c3(_):
    from tests import common, test_gpu_baseline_sizes as t
    n = 1 << 18
    s = t._scalars(n, 3, 0x7F)
    af = refcpu.random_elements(1, n, 0)[1]
    return {"c3": refcpu.commit(1, [(s, 0)], af),
            "c3_closed_form": common.closed_form_commitment(refcpu, 1, s),
            "c3_full_closed_form": common.closed_form_commitment(refcpu, 1,
                                                                 t._scalars(1 << 22, 4, 0x7F))}


def _baseline_c5(curve):
    from tests import common, test_gpu_baseline_sizes as t
    n = 1 << 18
    af = refcpu.random_elements(curve, n, 0)[1]
    s = t._scalars(n, 5 + curve, 0x3F)
    bits = np.unpackbits(t.c5_packed_scalars(n), axis=1, bitorder="little")
    cols, lo = [], 0
    for w in t.C5_BIT_TABLE:  # the packed rows as one column per output width
        b = np.zeros((n, 8 * ((w + 7) // 8)), dtype=np.uint8)
        b[:, :w] = bits[:, lo:lo + w]
        cols.append((np.packbits(b, axis=1, bitorder="little"), 0))
        lo += w
    out = {f"c5_{curve}": refcpu.commit(curve, [(s, 0)], af),
           f"c5_{curve}_packed": refcpu.commit(curve, cols, af)}
    if curve == 2:
        out["c5_full_closed_form"] = common.closed_form_commitment(refcpu, 2,
                                                                   t._scalars(1 << 22, 11, 0x3F))
    return out


def _run(job):
    fn, arg = job
    return fn(arg)


def make_baseline_sizes_fixture():
    """tests/golden/baseline_sizes.npz: the reference's results on the inputs of
    tests/test_gpu_baseline_sizes.py (its generators at sample indices, its commitments at the
    BASELINE sizes, one closed-form scalar multiplication for each 2^22 case)."""
    import multiprocessing as mp
    jobs = [(_baseline_generators, c) for c in (1, 2, 3)] + \
        [(_baseline_c1_c2, None), (_baseline_c3, None), (_baseline_c5, 2), (_baseline_c5, 3)]
    out = {}
    with mp.get_context("spawn").Pool(len(jobs)) as pool:
        for part in pool.map(_run, jobs):
            out.update(part)
    np.savez_compressed(os.path.join(HERE, "baseline_sizes.npz"), **out)


def make_ref_gpu_fixture():
    """tests/golden/ref_gpu_kernels.npz: the reference's GPU bucket kernels (oracle/_ref/
    libblitzar_ref_gpu.so) on the inputs of tests/test_ref_gpu_kernels.py, ristretto-compressed."""
    import blitzar_b200 as bb
    from oracle import refgpu
    from tests import test_ref_gpu_kernels as t
    assert bb.sxt_init(num_precomputed_generators=64) == 0
    out = {}
    for n in t.SIZES:
        gens, s = t._inputs(bb, n, seed=n)
        p3, _, _ = refgpu.bucket_msm(gens, s)
        out[f"n{n}"] = refcpu.normalize(0, p3)
        assert np.array_equal(out[f"n{n}"], refcpu.commit(0, [(s, 0)], gens)), n
    np.savez_compressed(os.path.join(HERE, "ref_gpu_kernels.npz"), **out)


FIXTURES = {"commit": main, "inner_product": make_inner_product_fixture,
            "oracle_cases": make_oracle_cases_fixture,
            "inner_product_seeded": make_inner_product_seeded_fixture,
            "baseline_sizes": make_baseline_sizes_fixture, "ref_gpu": make_ref_gpu_fixture}

if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("fixtures", nargs="*", default=["commit"], choices=sorted(FIXTURES))
    ap.add_argument("--out", default=HERE, help="directory the .npz files are written to")
    args = ap.parse_args()
    HERE = args.out
    for name in args.fixtures:
        FIXTURES[name]()
