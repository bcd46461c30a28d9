"""ctypes mirror of include/blitzar_b200.h (same names, argument meaning and error behaviour as the
reference's cbindings/blitzar_api.h for the `sxt_*` part).

Loading fails loudly if the CUDA library has not been built; there is no Python / CPU fallback.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libblitzar_b200.so")

SXT_CPU_BACKEND, SXT_GPU_BACKEND = 1, 2
SXT_CURVE_RISTRETTO255, SXT_CURVE_BLS_381, SXT_CURVE_BN_254, SXT_CURVE_GRUMPKIN = 0, 1, 2, 3
SXT_FIELD_SCALAR255, SXT_FIELD_GRUMPKIN = 0, 1
# per curve: (projective ABI bytes, commitment-generator stride, commitment output bytes)
CURVE_SIZES = {0: (160, 160, 32), 1: (144, 104, 48), 2: (96, 72, 72), 3: (96, 72, 72)}

SXT_SYMBOLS = [
    "sxt_init", "sxt_curve25519_compute_pedersen_commitments",
    "sxt_curve25519_compute_pedersen_commitments_with_generators",
    "sxt_bls12_381_g1_compute_pedersen_commitments_with_generators",
    "sxt_bn254_g1_uncompressed_compute_pedersen_commitments_with_generators",
    "sxt_grumpkin_uncompressed_compute_pedersen_commitments_with_generators",
    "sxt_ristretto255_get_generators", "sxt_curve25519_get_one_commit",
    "sxt_curve25519_prove_inner_product", "sxt_curve25519_verify_inner_product",
    "sxt_multiexp_handle_new", "sxt_multiexp_handle_new_from_file",
    "sxt_multiexp_handle_write_to_file", "sxt_multiexp_handle_free",
    "sxt_fixed_multiexponentiation", "sxt_fixed_packed_multiexponentiation",
    "sxt_fixed_vlen_multiexponentiation", "sxt_prove_sumcheck",
]
B200_SYMBOLS = [
    "b200_set_device", "b200_launch_count", "b200_point_bytes", "b200_malloc", "b200_free",
    "b200_memcpy_h2d", "b200_memcpy_d2h", "b200_synchronize", "b200_event_create",
    "b200_event_record", "b200_event_elapsed_ms", "b200_event_destroy", "b200_commit_device",
    "b200_combine_partials_device", "b200_fixed_msm_device",
    "b200_combine_partials_projective_device", "b200_set_tuning", "b200_profile_accumulate",
    "b200_profile_read", "b200_set_reduce_groups", "b200_stream",
    "b200_synthetic_generators_device", "b200_commit_host_partials",
    "b200_fixed_msm_host_partials", "b200_multiexp_handle_new_device",
    "b200_selftest_lane_arithmetic", "b200_prove_sumcheck_device",
]


class sxt_config(C.Structure):
    _fields_ = [("backend", C.c_int), ("num_precomputed_generators", C.c_uint64)]


class sxt_sequence_descriptor(C.Structure):
    _fields_ = [("element_nbytes", C.c_uint8), ("n", C.c_uint64), ("data", C.c_void_p),
                ("is_signed", C.c_int)]


_lib = None


def lib():
    """The loaded C-ABI library (raises if it was not built — no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m blitzar_b200.build` "
                               "(blitzar_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.sxt_init.restype = C.c_int
        L.sxt_ristretto255_get_generators.restype = C.c_int
        L.sxt_curve25519_get_one_commit.restype = C.c_int
        L.sxt_multiexp_handle_new.restype = C.c_void_p
        L.sxt_multiexp_handle_new_from_file.restype = C.c_void_p
        L.b200_launch_count.restype = C.c_ulonglong
        L.b200_point_bytes.restype = C.c_uint
        L.b200_malloc.restype = C.c_void_p
        L.b200_multiexp_handle_new_device.restype = C.c_void_p
        L.b200_event_create.restype = C.c_void_p
        L.b200_stream.restype = C.c_void_p
        L.b200_event_elapsed_ms.restype = C.c_float
        _lib = L
    return _lib


_initialized = False


def sxt_init(backend=SXT_GPU_BACKEND, num_precomputed_generators=0, device=None):
    """sxt_init (blitzar_api.h:200). Safe to call repeatedly from Python (initialises once)."""
    global _initialized
    if _initialized:
        return 0
    if device is not None:
        lib().b200_set_device(C.c_int(device))
    cfg = sxt_config(backend, num_precomputed_generators)
    rc = lib().sxt_init(C.byref(cfg))
    if rc == 0:
        _initialized = True
    return rc


def make_descriptors(columns, device_ptrs=None):
    """columns: list of (uint8 array [n, element_nbytes], is_signed). Returns (ctypes array, keepalive)."""
    arr = (sxt_sequence_descriptor * max(1, len(columns)))()
    keep = []
    for i, (data, is_signed) in enumerate(columns):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        keep.append(data)
        arr[i].element_nbytes = data.shape[1]
        arr[i].n = data.shape[0]
        if device_ptrs is not None:
            arr[i].data = device_ptrs[i]
        else:
            arr[i].data = data.ctypes.data if data.shape[0] else None
        arr[i].is_signed = int(is_signed)
    return arr, keep


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(None)


def compute_pedersen_commitments(curve_id, columns, generators=None, offset_generators=0):
    """The five sxt_*_compute_pedersen_commitments* entry points behind one Python call.

    generators: uint8 array [n, stride] in the ABI layout of the curve (None = built-in ristretto
    generators at offset_generators). Returns uint8 [num_columns, commitment bytes].
    """
    L = lib()
    desc, keep = make_descriptors(columns)
    out = np.zeros((len(columns), CURVE_SIZES[curve_id][2]), dtype=np.uint8)
    num = C.c_uint32(len(columns))
    if curve_id == SXT_CURVE_RISTRETTO255:
        if generators is None:
            L.sxt_curve25519_compute_pedersen_commitments(_ptr(out), num, desc,
                                                          C.c_uint64(offset_generators))
        else:
            L.sxt_curve25519_compute_pedersen_commitments_with_generators(_ptr(out), num, desc,
                                                                          _ptr(generators))
    else:
        fn = {1: L.sxt_bls12_381_g1_compute_pedersen_commitments_with_generators,
              2: L.sxt_bn254_g1_uncompressed_compute_pedersen_commitments_with_generators,
              3: L.sxt_grumpkin_uncompressed_compute_pedersen_commitments_with_generators}[curve_id]
        fn(_ptr(out), num, desc, _ptr(generators))
    return out


def get_generators(num_generators, offset_generators=0):
    """sxt_ristretto255_get_generators (count, offset — the implemented argument order)."""
    out = np.zeros((num_generators, 160), dtype=np.uint8)
    rc = lib().sxt_ristretto255_get_generators(_ptr(out), C.c_uint64(num_generators),
                                               C.c_uint64(offset_generators))
    if rc != 0:
        raise RuntimeError("sxt_ristretto255_get_generators failed")
    return out


def get_one_commit(n):
    out = np.zeros((1, 160), dtype=np.uint8)
    rc = lib().sxt_curve25519_get_one_commit(_ptr(out), C.c_uint64(n))
    if rc != 0:
        raise RuntimeError("sxt_curve25519_get_one_commit failed")
    return out


class MultiexpHandle:
    """sxt_multiexp_handle: device-resident generators for fixed-base MSM."""

    def __init__(self, curve_id, generators=None, filename=None, device_ptr=None, n=None):
        self.curve_id = curve_id
        if device_ptr is not None:  # projective ABI structs already in HBM
            self.h = lib().b200_multiexp_handle_new_device(C.c_uint(curve_id),
                                                           C.c_void_p(device_ptr), C.c_uint(n))
        elif filename is not None:
            self.h = lib().sxt_multiexp_handle_new_from_file(C.c_uint(curve_id),
                                                             filename.encode())
        else:
            generators = np.ascontiguousarray(generators, dtype=np.uint8)
            self.h = lib().sxt_multiexp_handle_new(C.c_uint(curve_id), _ptr(generators),
                                                   C.c_uint(generators.shape[0]))

    def write_to_file(self, filename):
        lib().sxt_multiexp_handle_write_to_file(C.c_void_p(self.h), filename.encode())

    def free(self):
        if self.h:
            lib().sxt_multiexp_handle_free(C.c_void_p(self.h))
            self.h = None

    def _res(self, num_outputs):
        return np.zeros((num_outputs, CURVE_SIZES[self.curve_id][0]), dtype=np.uint8)

    def fixed_multiexponentiation(self, element_num_bytes, num_outputs, n, scalars):
        res = self._res(num_outputs)
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        lib().sxt_fixed_multiexponentiation(_ptr(res), C.c_void_p(self.h),
                                            C.c_uint(element_num_bytes), C.c_uint(num_outputs),
                                            C.c_uint(n), _ptr(scalars))
        return res

    def fixed_packed_multiexponentiation(self, output_bit_table, n, scalars):
        num_outputs = len(output_bit_table)
        res = self._res(num_outputs)
        bt = (C.c_uint * num_outputs)(*output_bit_table)
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        lib().sxt_fixed_packed_multiexponentiation(_ptr(res), C.c_void_p(self.h), bt,
                                                   C.c_uint(num_outputs), C.c_uint(n),
                                                   _ptr(scalars))
        return res

    def fixed_vlen_multiexponentiation(self, output_bit_table, output_lengths, scalars):
        num_outputs = len(output_bit_table)
        res = self._res(num_outputs)
        bt = (C.c_uint * num_outputs)(*output_bit_table)
        ol = (C.c_uint * num_outputs)(*output_lengths)
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        lib().sxt_fixed_vlen_multiexponentiation(_ptr(res), C.c_void_p(self.h), bt, ol,
                                                 C.c_uint(num_outputs), _ptr(scalars))
        return res


# ---- device-resident extension -----------------------------------------------------------------
class DeviceBuffer:
    def __init__(self, nbytes=None, host=None):
        if host is not None:
            host = np.ascontiguousarray(host)
            nbytes = host.nbytes
        self.nbytes = nbytes
        self.ptr = lib().b200_malloc(C.c_uint64(max(nbytes, 16)))
        if host is not None and nbytes:
            lib().b200_memcpy_h2d(C.c_void_p(self.ptr), _ptr(host), C.c_uint64(nbytes))

    def to_host(self, shape=None, dtype=np.uint8):
        out = np.zeros(self.nbytes, dtype=np.uint8)
        lib().b200_memcpy_d2h(_ptr(out), C.c_void_p(self.ptr), C.c_uint64(self.nbytes))
        out = out.view(dtype)
        return out.reshape(shape) if shape is not None else out

    def free(self):
        if self.ptr:
            lib().b200_free(C.c_void_p(self.ptr))
            self.ptr = None


class Event:
    def __init__(self):
        self.e = lib().b200_event_create()

    def record(self):
        lib().b200_event_record(C.c_void_p(self.e))

    def elapsed_ms(self, stop):
        return float(lib().b200_event_elapsed_ms(C.c_void_p(self.e), C.c_void_p(stop.e)))


def commit_device(curve_id, columns_shape, scalar_ptrs, generators_ptr, out_commit_ptr=None,
                  out_partial_ptr=None, offset_generators=0):
    """b200_commit_device. columns_shape: list of (n, element_nbytes, is_signed)."""
    num = len(columns_shape)
    arr = (sxt_sequence_descriptor * max(1, num))()
    for i, (n, nbytes, is_signed) in enumerate(columns_shape):
        arr[i].element_nbytes = nbytes
        arr[i].n = n
        arr[i].data = scalar_ptrs[i]
        arr[i].is_signed = int(is_signed)
    lib().b200_commit_device(C.c_uint(curve_id), C.c_void_p(out_commit_ptr),
                             C.c_void_p(out_partial_ptr), C.c_uint32(num), arr,
                             C.c_void_p(generators_ptr), C.c_uint64(offset_generators))


def selftest_lane_arithmetic(warps=64, seed=1):
    lib().b200_selftest_lane_arithmetic.restype = C.c_uint
    return int(lib().b200_selftest_lane_arithmetic(C.c_uint(warps), C.c_uint(seed)))


def synthetic_generators_device(curve_id, out_ptr, n, first=0, projective=False):
    """b200_synthetic_generators_device: the reference benchmarks' generators, produced in HBM."""
    lib().b200_synthetic_generators_device(C.c_uint(curve_id), C.c_void_p(out_ptr), C.c_uint64(n),
                                           C.c_uint64(first), C.c_int(1 if projective else 0))


def synthetic_generators(curve_id, n, first=0, projective=False):
    """Host copy of synthetic_generators_device (uint8 [n, stride])."""
    stride = CURVE_SIZES[curve_id][0 if (projective or curve_id == 0) else 1]
    buf = DeviceBuffer(n * stride)
    synthetic_generators_device(curve_id, buf.ptr, n, first, projective)
    out = buf.to_host((n, stride))
    buf.free()
    return out


def commit_host_partials(curve_id, columns, generators, out_partial_ptr, offset_generators=0):
    """b200_commit_host_partials: host columns / generators in, partial points in HBM out."""
    desc, keep = make_descriptors(columns)
    lib().b200_commit_host_partials(C.c_uint(curve_id), C.c_void_p(out_partial_ptr),
                                    C.c_uint32(len(columns)), desc, _ptr(generators),
                                    C.c_uint64(offset_generators))


def fixed_msm_device(handle, out_res_ptr, out_partial_ptr, element_num_bytes, num_outputs, n,
                     scalars_ptr):
    """b200_fixed_msm_device, fixed-width mode."""
    lib().b200_fixed_msm_device(C.c_void_p(out_res_ptr), C.c_void_p(out_partial_ptr),
                                C.c_void_p(handle.h), C.c_int(0), C.c_uint(element_num_bytes),
                                None, None, C.c_uint(num_outputs), C.c_uint(n),
                                C.c_void_p(scalars_ptr))


def fixed_msm_host_partials(handle, out_partial_ptr, element_num_bytes, num_outputs, n, scalars):
    lib().b200_fixed_msm_host_partials(C.c_void_p(out_partial_ptr), C.c_void_p(handle.h),
                                       C.c_int(0), C.c_uint(element_num_bytes), None, None,
                                       C.c_uint(num_outputs), C.c_uint(n), _ptr(scalars))


def combine_partials_projective_device(curve_id, out_ptr, partials_ptr, num_parts, count):
    lib().b200_combine_partials_projective_device(C.c_uint(curve_id), C.c_void_p(out_ptr),
                                                  C.c_void_p(partials_ptr), C.c_uint32(num_parts),
                                                  C.c_uint32(count))


def synchronize():
    lib().b200_synchronize()


def launch_count():
    return int(lib().b200_launch_count())


def profile_accumulate(enable):
    lib().b200_profile_accumulate(C.c_int(1 if enable else 0))


def profile_read():
    """(total milliseconds, launches) of the level-1 accumulation kernel since the last read."""
    ms, cnt = C.c_float(0), C.c_uint(0)
    lib().b200_profile_read(C.byref(ms), C.byref(cnt))
    return float(ms.value), int(cnt.value)


def set_tuning(window_bits=0, chunk1=0, chunkn=0):
    lib().b200_set_tuning(C.c_uint(window_bits), C.c_uint(chunk1), C.c_uint(chunkn))


def combine_partials_device(curve_id, out_ptr, partials_ptr, num_parts, count):
    lib().b200_combine_partials_device(C.c_uint(curve_id), C.c_void_p(out_ptr),
                                       C.c_void_p(partials_ptr), C.c_uint32(num_parts),
                                       C.c_uint32(count))


def point_bytes(curve_id):
    return int(lib().b200_point_bytes(C.c_uint(curve_id)))


def set_reduce_groups(g1=0, gn=0):
    lib().b200_set_reduce_groups(C.c_uint(g1), C.c_uint(gn))


def stream_ptr():
    """cudaStream_t of the library (int), e.g. for torch.cuda.ExternalStream."""
    return int(lib().b200_stream())


def prove_inner_product(transcript, a, b, generators_offset=0):
    """sxt_curve25519_prove_inner_product. transcript: uint8[203] (advanced in place); a, b:
    uint8 [n, 32] scalars. Returns (l_vector [rounds, 32], r_vector, ap_value [32])."""
    n = a.shape[0]
    rounds = max(0, (n - 1).bit_length())
    lv = np.zeros((max(rounds, 1), 32), dtype=np.uint8)
    rv = np.zeros((max(rounds, 1), 32), dtype=np.uint8)
    ap = np.zeros(32, dtype=np.uint8)
    a = np.ascontiguousarray(a, dtype=np.uint8)
    b = np.ascontiguousarray(b, dtype=np.uint8)
    lib().sxt_curve25519_prove_inner_product(_ptr(lv), _ptr(rv), _ptr(ap), _ptr(transcript),
                                             C.c_uint64(n), C.c_uint64(generators_offset),
                                             _ptr(a), _ptr(b))
    return lv[:rounds], rv[:rounds], ap


def verify_inner_product(transcript, b, product, a_commit, l_vector, r_vector, ap_value,
                         generators_offset=0):
    """sxt_curve25519_verify_inner_product -> 1 / 0."""
    n = b.shape[0]
    b = np.ascontiguousarray(b, dtype=np.uint8)
    lv = np.ascontiguousarray(l_vector if len(l_vector) else np.zeros((1, 32), np.uint8))
    rv = np.ascontiguousarray(r_vector if len(r_vector) else np.zeros((1, 32), np.uint8))
    lib().sxt_curve25519_verify_inner_product.restype = C.c_int
    return int(lib().sxt_curve25519_verify_inner_product(
        _ptr(transcript), C.c_uint64(n), C.c_uint64(generators_offset), _ptr(b),
        _ptr(np.ascontiguousarray(product)), _ptr(np.ascontiguousarray(a_commit)), _ptr(lv),
        _ptr(rv), _ptr(np.ascontiguousarray(ap_value))))


# ---- sumcheck (blitzar_api.h:133-183, :766) --------------------------------------------------------
class sumcheck_descriptor(C.Structure):
    _fields_ = [("mles", C.c_void_p), ("product_table", C.c_void_p),
                ("product_terms", C.POINTER(C.c_uint)), ("n", C.c_uint), ("num_mles", C.c_uint),
                ("num_products", C.c_uint), ("num_product_terms", C.c_uint),
                ("round_degree", C.c_uint)]


# void (FIELD* r, void* context, const FIELD* polynomial, unsigned polynomial_len)
SUMCHECK_CALLBACK = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint)


def sumcheck_num_variables(n):
    return max((n - 1).bit_length(), 1)


def pack_product_table(field_id, product_table):
    """product_table: [(multiplier as 32 ABI bytes, product_length)] -> the C layout of
    std::pair<FIELD, unsigned>: 36-byte entries for scalar255, 40-byte entries for grumpkin (the
    length at byte 32, padding zero)."""
    stride = 36 if field_id == SXT_FIELD_SCALAR255 else 40
    out = np.zeros((max(len(product_table), 1), stride), dtype=np.uint8)
    for k, (mult, length) in enumerate(product_table):
        out[k, :32] = np.frombuffer(bytes(mult), dtype=np.uint8)
        out[k, 32:36] = np.frombuffer(np.uint32(length).tobytes(), dtype=np.uint8)
    return out


def sumcheck_args(field_id, mles_ptr, n, num_mles, product_table, product_terms, callback,
                  round_degree=None):
    """ctypes arguments of sxt_prove_sumcheck / b200_prove_sumcheck_device (and the emulated
    prover). callback(polynomial uint8 [len, 32]) returns the round's challenge r as 32 ABI bytes.
    Returns (args, polynomials [num_variables, round_degree + 1, 32], evaluation_point
    [num_variables, 32], keepalive)."""
    if round_degree is None:
        round_degree = max([length for _, length in product_table], default=1)
    v = sumcheck_num_variables(n)
    polys = np.zeros((v, round_degree + 1, 32), dtype=np.uint8)
    point = np.zeros((v, 32), dtype=np.uint8)
    table = pack_product_table(field_id, product_table)
    terms = (C.c_uint * max(len(product_terms), 1))(*product_terms)

    def trampoline(r, _ctx, poly, length):
        p = np.ctypeslib.as_array(C.cast(poly, C.POINTER(C.c_uint8)), shape=(length * 32,))
        C.memmove(r, bytes(callback(p.reshape(length, 32).copy())), 32)

    cb = SUMCHECK_CALLBACK(trampoline)
    desc = sumcheck_descriptor(mles_ptr, table.ctypes.data, terms, n, num_mles, len(product_table),
                               len(product_terms), round_degree)
    args = (_ptr(polys), _ptr(point), C.c_uint(field_id), C.byref(desc), C.cast(cb, C.c_void_p),
            C.c_void_p(None))
    return args, polys, point, (table, terms, cb, desc)


def prove_sumcheck(field_id, mles, product_table, product_terms, callback, round_degree=None):
    """sxt_prove_sumcheck. mles: uint8 [num_mles, n, 32] (MLE j is mles[j], ABI form of the field);
    product_table: [(multiplier 32 bytes, product_length)]; product_terms: MLE indices of every
    product, concatenated; callback(polynomial uint8 [len, 32]) -> r (32 bytes).
    Returns (polynomials [num_variables, round_degree + 1, 32], evaluation_point [num_variables, 32])."""
    mles = np.ascontiguousarray(mles, dtype=np.uint8)
    args, polys, point, _keep = sumcheck_args(field_id, mles.ctypes.data, mles.shape[1],
                                              mles.shape[0], product_table, product_terms,
                                              callback, round_degree)
    lib().sxt_prove_sumcheck(*args)
    return polys, point


def prove_sumcheck_device(field_id, mles_ptr, n, num_mles, product_table, product_terms, callback,
                          round_degree=None):
    """b200_prove_sumcheck_device: as prove_sumcheck with the MLEs already in HBM (device pointer,
    the same column-major layout)."""
    args, polys, point, _keep = sumcheck_args(field_id, mles_ptr, n, num_mles, product_table,
                                              product_terms, callback, round_degree)
    lib().b200_prove_sumcheck_device(*args)
    return polys, point
