"""The Fq primitives ON THE DEVICE, bit for bit against the exact integer model (tests/fp_exact.py).

tests/fp_probe.cu is compiled here with the library's own nvcc flags (python-bls_b200/build.py NVCC_FLAGS, which
include -DB200BLS_MUL_CALL: fp_mul is then the out-of-line fp_mul_call the kernels execute) into a test-only shared
object in a temporary directory, and runs one thread per case.  This checks what the host build cannot: that
ptxas's fused IMAD.WIDE carry chains give the emulated integers at the ends of every domain.  Only in-domain
operands are sent; out-of-domain behaviour is pinned on the host (test_fp_bounds_cpu.py)."""
import ctypes
import importlib.util
import os
import shutil
import subprocess

import numpy as np
import pytest

import fp_exact as E

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _nvcc():
    return shutil.which("nvcc") or next((p for p in ("/usr/local/cuda/bin/nvcc",) if os.path.exists(p)), None)


def build_probe(outdir):
    spec = importlib.util.spec_from_file_location("b200bls_build", os.path.join(ROOT, "python-bls_b200", "build.py"))
    build = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(build)
    assert "-DB200BLS_MUL_CALL" in build.NVCC_FLAGS and "arch=compute_100a,code=sm_100a" in build.NVCC_FLAGS
    so = os.path.join(str(outdir), "fp_probe.so")
    res = subprocess.run([_nvcc()] + build.NVCC_FLAGS + ["-shared", "-o", so, os.path.join(HERE, "fp_probe.cu")],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-4000:]
    return so, res.stdout


@pytest.mark.skipif(_nvcc() is None, reason="nvcc not installed")
def test_probe_compiles_for_sm100a(tmp_path):
    """CPU: the probe must keep compiling with the library's flags, so that the device test cannot rot"""
    so, log = build_probe(tmp_path)
    assert os.path.getsize(so) > 0
    assert "fp_probe_kernel" in log and "fp_mul_call" in log     # ptxas -v lists both: fp_mul is the call form


@pytest.mark.gpu
def test_device_primitives_exact(tmp_path):
    so, _ = build_probe(tmp_path)
    lib = ctypes.CDLL(so)
    names, ops, cases = E.build_suite(seed=0xB200, n_random=6000, n_worst=3000)
    assert len(cases) > 250_000
    inp = E.pack_inputs(cases)
    out = np.zeros(len(cases) * 24, dtype=np.uint32)
    vp = ctypes.c_void_p
    rc = lib.fp_probe_run(ctypes.c_longlong(len(cases)), vp(ops.ctypes.data), vp(inp.ctypes.data), vp(out.ctypes.data))
    assert rc == 0, "CUDA error %d" % rc
    outs = E.unpack_outputs(out, len(cases))
    bad = E.check_results(names, cases, outs)
    assert not bad, "%d of %d device cases differ from the model, first: %s" % (len(bad), len(cases), bad[:3])
    print("device cases compared bit-exactly: %d" % len(cases))
