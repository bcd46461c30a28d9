"""TEST INFRASTRUCTURE — Python side of the emulated sumcheck prover (tests/emul/emul_sumcheck.cpp,
linked into the emulation library of harness.py). Same arguments and results as
blitzar_b200.prove_sumcheck; used only by the `not gpu` tests."""
import ctypes as C

import numpy as np

from blitzar_b200 import api
from tests.emul import harness


def prove_sumcheck(field_id, mles, product_table, product_terms, callback, round_degree=None):
    """Emulated sxt_prove_sumcheck. mles: uint8 [num_mles, n, 32]."""
    mles = np.ascontiguousarray(mles, dtype=np.uint8)
    args, polys, point, _keep = api.sumcheck_args(field_id, mles.ctypes.data, mles.shape[1],
                                                  mles.shape[0], product_table, product_terms,
                                                  callback, round_degree)
    harness.lib().emul_prove_sumcheck(*args)
    return polys, point


def sumcheck_check(field_id, n, num_mles, product_table, product_terms, round_degree=None):
    """The descriptor checks of sxt_prove_sumcheck as a return code (0 = valid). The MLE pointer is
    a non-null placeholder: the checks never read the MLEs."""
    args, _, _, _keep = api.sumcheck_args(field_id, 1, n, num_mles, product_table, product_terms,
                                          lambda p: bytes(32), round_degree)
    fn = harness.lib().emul_sumcheck_check
    fn.restype = C.c_int
    return int(fn(*args[:5]))
