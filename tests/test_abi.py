"""The C-ABI library loads and exports every symbol that include/b200bls.h declares; no
compute call works without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200bls.h")
LIB = os.path.join(ROOT, "python-bls_b200", "bls_b200", "libb200bls.so")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200bls_\w+)\s*\(", src)))


def test_header_declares_the_hot_path():
    syms = declared_symbols()
    for must in ("b200bls_pairing_batch", "b200bls_pairing_multi", "b200bls_verify_batch",
                 "b200bls_aggregate_verify", "b200bls_g1_sum", "b200bls_g2_sum",
                 "b200bls_hash_to_g2_batch", "b200bls_g2_scalar_mul_batch",
                 "b200bls_final_exp_batch", "b200bls_field_op_batch"):
        assert must in syms
    assert len(syms) >= 50


def test_library_exports_every_declared_symbol():
    if not os.path.exists(LIB):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(LIB)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, missing


def test_python_binding_covers_the_header():
    from bls_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()


def test_no_cpu_fallback():
    """without a CUDA device init fails loudly and compute entry points refuse to run"""
    lib = ctypes.CDLL(LIB)
    lib.b200bls_last_error.restype = ctypes.c_char_p
    if lib.b200bls_init(0) == 0:
        lib.b200bls_shutdown()
        pytest.skip("GPU present")
    assert b"no CPU path" in lib.b200bls_last_error()
    buf = (ctypes.c_uint8 * 576)()
    assert lib.b200bls_pairing_batch(buf, buf, buf, ctypes.c_size_t(1)) == -1   # B200BLS_E_NOT_INIT
    from bls_b200 import _lib
    with pytest.raises(_lib.B200BlsError):
        from bls_b200 import engine
        engine.pairing_batch(bytes(96), bytes(192))


def test_plugin_seam_signatures_match_the_reference():
    """bls_b200.fields_t_c offers functions of the reference's accelerator seam (fields_t.py:1218-1265)
    under the same names and parameter lists, recorded from the reference"""
    import inspect
    from bls_b200 import fields_t_c as C
    recorded = {
        "fq_ate_pairing_multi": ["Ps", "Qs"],
        "fq_miller_loop": ["px", "py", "pinf", "qx_t", "qy_t", "qinf"],
        "fq12_final_exp": ["t_x"],
        "fq_scalar_mult_jacobian": ["c", "x1", "y1", "z1", "inf1"],
        "fq2_scalar_mult_jacobian": ["c", "x1", "y1", "z1", "inf1"],
    }
    for name, params in recorded.items():
        assert list(inspect.signature(getattr(C, name)).parameters) == params, name
