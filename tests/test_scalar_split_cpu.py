"""The scalar split of the signing ladders (python-bls_b200/csrc/scalar_split.h) on the CPU: g++ builds the header's
__host__ __device__ function behind a small C shim, and every record must hold the exact Python-integer digits of
sk mod n in base a = |x|, each below a, with sum d_i a^i = sk mod n."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from sign_corpus import digits, edge_keys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "python-bls_b200", "csrc")

A = 0xd201000000010000
N = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001

SHIM = r"""
#include "scalar_split.h"
extern "C" void shim_split(const unsigned char* sk, unsigned char* out, long long n) {
  for (long long i = 0; i < n; i++) b200bls::scalar_split(sk + 32 * i, out + 32 * i);
}
"""


@pytest.fixture(scope="module")
def split(tmp_path_factory):
    d = tmp_path_factory.mktemp("split")
    src, so = d / "shim.cpp", d / "split.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    lib.shim_split.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong]

    def run(sks):
        buf = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in sks), dtype=np.uint8).copy()
        out = np.full(buf.size, 0xa5, dtype=np.uint8)
        lib.shim_split(buf.ctypes.data, out.ctypes.data, len(sks))
        raw = out.tobytes()
        return [int.from_bytes(raw[32 * i:32 * (i + 1)], "big") for i in range(len(sks))]
    return run


def test_edge_keys(split):
    ks = edge_keys()
    assert (A - 1) * sum(A ** i for i in range(4)) > N          # all four digits at a - 1 is not below n
    for sk, rec in zip(ks, split(ks)):
        assert rec == sum(d << (64 * i) for i, d in enumerate(digits(sk))), hex(sk)


def test_seeded_random_keys(split):
    rng = random.Random(20261021)
    ks = [rng.getrandbits(256) for _ in range(10000)] + [rng.randrange(N) for _ in range(1000)]
    for sk, rec in zip(ks, split(ks)):
        ds = [(rec >> (64 * i)) & (2 ** 64 - 1) for i in range(4)]
        assert all(d < A for d in ds), hex(sk)
        assert sum(d * A ** i for i, d in enumerate(ds)) == sk % N, hex(sk)
        assert ds == digits(sk), hex(sk)
