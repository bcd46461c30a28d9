"""Generates tests/golden/sumcheck.npz from the REFERENCE's own cpu sumcheck prover (oracle/_ref,
built from the reference's sources by oracle/ref_build/sumcheck.mk):

    python tests/golden/make_sumcheck_golden.py [--out DIR]

The cases are tests/test_sumcheck.py's `case_specs`; the file stores their specs (seeds,
descriptors) and the reference's proofs only, the tests regenerate the inputs from the seeds."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refsumcheck  # noqa: E402
from tests import test_sumcheck  # noqa: E402

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.dirname(os.path.abspath(__file__)),
                    help="directory sumcheck.npz is written to")
    args = ap.parse_args()
    np.savez_compressed(os.path.join(args.out, "sumcheck.npz"),
                        **test_sumcheck.make_fixture(refsumcheck.prove_sumcheck))
