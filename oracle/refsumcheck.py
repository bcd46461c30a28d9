"""TEST INFRASTRUCTURE — ctypes binding of oracle/_ref/libblitzar_ref_sumcheck.so, the reference's
own cpu sumcheck prover (oracle/ref_build/ref_sumcheck.cc, built by oracle/ref_build/sumcheck.mk).
Only tests/ may import this module; the product never does."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libblitzar_ref_sumcheck.so")

_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(LIB_PATH)
    return _lib


def prove_sumcheck(field_id, mles, product_table, product_terms, callback, round_degree=None):
    """Same arguments and results as blitzar_b200.prove_sumcheck (mles: uint8 [num_mles, n, 32])."""
    from blitzar_b200 import api
    mles = np.ascontiguousarray(mles, dtype=np.uint8)
    args, polys, point, _keep = api.sumcheck_args(field_id, mles.ctypes.data, mles.shape[1],
                                                  mles.shape[0], product_table, product_terms,
                                                  callback, round_degree)
    lib().ref_prove_sumcheck(*args)
    return polys, point
