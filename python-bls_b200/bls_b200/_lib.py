"""ctypes binding of libb200bls.so (include/b200bls.h).  No CPU fallback: if the library
or a CUDA device is missing, importing / initialising raises."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200BLS_LIB") or os.path.join(_HERE, "libb200bls.so")


class B200BlsError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise B200BlsError(
            "%s not found: build it with `python python-bls_b200/build.py` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, sz, i32 = c.c_void_p, c.c_size_t, c.c_int
    sig = {
        "b200bls_init": (i32, [i32]),
        "b200bls_shutdown": (None, []),
        "b200bls_last_error": (c.c_char_p, []),
        "b200bls_sm_count": (i32, []),
        "b200bls_sync": (i32, []),
        "b200bls_set_stream": (i32, [i32]),
        "b200bls_stream_count": (i32, []),
        "b200bls_set_ctas_per_sm": (i32, [i32]),
        "b200bls_get_ctas_per_sm": (i32, []),
        "b200bls_malloc": (vp, [sz]),
        "b200bls_free": (None, [vp]),
        "b200bls_host_alloc": (vp, [sz]),
        "b200bls_host_free": (None, [vp]),
        "b200bls_h2d": (i32, [vp, vp, sz]),
        "b200bls_d2h": (i32, [vp, vp, sz]),
        "b200bls_timer_start": (i32, []),
        "b200bls_timer_stop": (i32, [c.POINTER(c.c_float)]),
        "b200bls_launch_count": (c.c_uint64, []),
        "b200bls_microbench_imad": (i32, [i32, i32, i32, i32, c.POINTER(c.c_double), c.POINTER(c.c_float)]),
        "b200bls_run_program_dev": (i32, [c.c_char_p, sz, c.POINTER(vp), c.POINTER(c.c_int64), i32]),
        "b200bls_program_info": (i32, [c.c_char_p, c.POINTER(i32), c.POINTER(i32), c.POINTER(i32)]),
        "b200bls_field_op_batch": (i32, [i32, i32, vp, vp, vp, sz]),
        "b200bls_field_op_batch_dev": (i32, [i32, i32, vp, vp, vp, sz]),
        "b200bls_field_frob_batch": (i32, [i32, i32, vp, vp, sz]),
        "b200bls_field_pow_batch": (i32, [i32, vp, vp, vp, sz]),
        "b200bls_field_sqrt_batch": (i32, [i32, vp, vp, vp, sz]),
        "b200bls_sw_encode_g2_batch": (i32, [vp, vp, sz]),
        "b200bls_jacobian_op_batch": (i32, [i32, i32, vp, vp, vp, sz]),
        "b200bls_g2_untwist_batch": (i32, [vp, vp, sz]),
        "b200bls_fq12_twist_batch": (i32, [vp, vp, sz]),
        "b200bls_g2_psi_batch": (i32, [vp, vp, sz]),
        "b200bls_pairing_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_pairing_batch_async": (i32, [vp, vp, vp, sz]),
        "b200bls_pairing_batch_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_final_exp_batch": (i32, [vp, vp, sz]),
        "b200bls_final_exp_batch_dev": (i32, [vp, vp, sz]),
        "b200bls_miller_loop_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_miller_loop_batch_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_miller_product": (i32, [vp, vp, vp, sz]),
        "b200bls_miller_product_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_pairing_multi": (i32, [vp, vp, vp, sz]),
        "b200bls_pairing_multi_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_pairing_multi_batch": (i32, [i32, vp, vp, vp, sz, vp]),
        "b200bls_pairing_multi_batch_dev": (i32, [i32, vp, vp, vp, sz, vp]),
        "b200bls_g1_scalar_mul_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g1_scalar_mul_batch_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_scalar_mul_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_scalar_mul_batch_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_g1_add_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_add_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g1_sum": (i32, [vp, vp, sz]),
        "b200bls_g1_sum_dev": (i32, [vp, vp, sz]),
        "b200bls_g2_sum": (i32, [vp, vp, sz]),
        "b200bls_g2_sum_dev": (i32, [vp, vp, sz]),
        "b200bls_g1_decompress_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_decompress_batch": (i32, [vp, vp, vp, sz]),
        "b200bls_g1_compress_batch": (i32, [vp, vp, sz]),
        "b200bls_g2_compress_batch": (i32, [vp, vp, sz]),
        "b200bls_subgroup_check_batch": (i32, [i32, vp, vp, sz]),
        "b200bls_subgroup_check_batch_dev": (i32, [i32, vp, vp, sz]),
        "b200bls_key_validate_batch": (i32, [vp, vp, sz]),
        "b200bls_key_validate_batch_dev": (i32, [vp, vp, sz]),
        "b200bls_verify_batch_strict": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_verify_batch_strict_dev": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_verify_batch_wire_strict": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_verify_batch_wire_strict_dev": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_g1_msm": (i32, [vp, vp, vp, sz]),
        "b200bls_g1_msm_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_msm": (i32, [vp, vp, vp, sz]),
        "b200bls_g2_msm_dev": (i32, [vp, vp, vp, sz]),
        "b200bls_aggregate_miller": (i32, [vp, vp, vp, sz, vp]),
        "b200bls_aggregate_verify_async": (i32, [vp, vp, vp, sz, vp]),
        "b200bls_verify_batch_wire": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_verify_batch_wire_dev": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_hash_pks": (i32, [vp, ctypes.c_uint32, vp, sz]),
        "b200bls_hash_pks_dev": (i32, [vp, ctypes.c_uint32, vp, sz]),
        "b200bls_hash_to_g2_batch": (i32, [vp, vp, sz]),
        "b200bls_hash_to_g2_batch_dev": (i32, [vp, vp, sz]),
        "b200bls_sign_batch": (i32, [i32, vp, vp, vp, sz]),
        "b200bls_sign_batch_dev": (i32, [i32, vp, vp, vp, sz]),
        "b200bls_public_key_batch": (i32, [i32, vp, vp, sz]),
        "b200bls_public_key_batch_dev": (i32, [i32, vp, vp, sz]),
        "b200bls_verify_batch": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_verify_batch_dev": (i32, [vp, vp, vp, vp, sz]),
        "b200bls_aggregate_verify": (i32, [vp, vp, vp, sz, vp]),
        "b200bls_comm_init": (i32, [i32, i32, c.c_char_p, c.c_char_p]),
        "b200bls_comm_shutdown": (None, []),
        "b200bls_comm_has_nccl": (i32, []),
        "b200bls_comm_world": (i32, []),
        "b200bls_comm_rank": (i32, []),
        "b200bls_allgather_host": (i32, [vp, vp, sz]),
        "b200bls_aggregate_verify_sharded": (i32, [vp, vp, vp, sz, i32, vp]),
        "b200bls_point_sum_sharded_dev": (i32, [i32, vp, sz, i32, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, sig


lib, SIGNATURES = _load()
_initialised = False


def check(rc):
    if rc != 0:
        raise B200BlsError("b200bls error %d: %s" % (rc, lib.b200bls_last_error().decode()))


def init(device=None):
    """Bind this process to one GPU (default: LOCAL_RANK or 0)."""
    global _initialised
    if _initialised:
        return
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    check(lib.b200bls_init(device))
    _initialised = True


def as_u8(buf, n_bytes=None):
    """bytes / bytearray / ndarray -> contiguous uint8 ndarray (no copy when possible)"""
    if isinstance(buf, np.ndarray):
        arr = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    else:
        arr = np.frombuffer(bytes(buf), dtype=np.uint8)
    if n_bytes is not None and arr.size != n_bytes:
        raise ValueError("expected %d bytes, got %d" % (n_bytes, arr.size))
    return arr


def ptr(arr):
    return ctypes.c_void_p(arr.ctypes.data)
