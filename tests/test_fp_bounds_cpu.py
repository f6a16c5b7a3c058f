"""The Fq core at its reduction bounds, on the host build of the limb code (tests/hostsim/hostsim_fp.cpp: fp.cuh,
vm_exec.cuh and vm_exec2.cuh with the PTX emulated, carry flag included).

Every primitive must return exactly the integer of the model in tests/fp_exact.py -- not just the right value mod
q -- on a corpus that reaches the ends of each input domain (0 and q as zero, 2q - 1, 4q - 1, 2^384 - 1, limb
patterns, operands whose Montgomery reduction quotient is R - 1), and every output must stay below the bound the
source comments claim for it.  Those bounds are what lets the products skip their final subtraction."""
import ctypes
import os
import random
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import fp_exact as E

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "python-bls_b200", "csrc")


@pytest.fixture(scope="module")
def probe():
    """the host build, rebuilt when a source is newer than the library (as tests/hostsim/__init__.py does)"""
    so = os.path.join(HERE, "hostsim", "_hostsim_fp.so")
    srcs = [os.path.join(HERE, "hostsim", "hostsim_fp.cpp")]
    deps = srcs + [os.path.join(HERE, "fp_probe.cu")] + [
        os.path.join(CSRC, f) for f in ("fp.cuh", "vm_exec.cuh", "vm_exec2.cuh", "gen/vm_isa.h", "gen/fp_consts.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so] + srcs)
    lib = ctypes.CDLL(so)

    def run(ops, cases):
        ops = np.ascontiguousarray(ops, dtype=np.int32)
        inp = E.pack_inputs(cases)
        out = np.zeros(len(cases) * 24, dtype=np.uint32)
        vp = ctypes.c_void_p
        assert lib.hs_fp_probe_run(ctypes.c_longlong(len(cases)), vp(ops.ctypes.data), vp(inp.ctypes.data),
                                   vp(out.ctypes.data)) == 0
        return E.unpack_outputs(out, len(cases))
    return run


def _bound_ok(bound, v):
    if bound is None:
        return True
    if bound == "2q]":
        return v <= E.Q2
    return Fraction(v, E.Q) < Fraction(bound).limit_denominator(1000)


def test_every_primitive_exact_and_within_its_bound(probe):
    names, ops, cases = E.build_suite(seed=0xF00D, n_random=1500, n_worst=1500)
    assert len(cases) > 100_000
    outs = probe(ops, cases)
    bad = E.check_results(names, cases, outs)
    assert not bad, "%d mismatches, first: %s" % (len(bad), bad[:3])
    seen = set()
    for name, got in zip(names, outs):
        bound = E.FP_OPS[name][3]
        for v in got[:2 if name in E.TWO_OUT else 1]:
            assert _bound_ok(bound, v), "%s output %s above its bound %s (%s)" % (name, hex(v), bound, E.FP_OPS[name][4])
        seen.add(name)
    assert seen == set(E.FP_OPS)


def test_corpus_reaches_the_extremes():
    """the corpus is only worth something if it gets close to the claimed bounds and holds the worst quotients"""
    rnd = random.Random(1)
    top = {}
    for name in ("mul_u4", "mul2", "pair_mul2", "fp2_sqr"):
        for args in E.corpus(name, rnd, 300, 600):
            top[name] = max([top.get(name, 0)] + [v / E.Q for v in E.expected(name, args)])
    assert top["mul_u4"] > 2.6 and top["mul2"] > 1.6 and top["pair_mul2"] > 1.75 and top["fp2_sqr"] > 1.8, top
    worst = E.worst_pairs(("w", "w"), rnd, 50)
    assert len(worst) == 50 and all(E.mont_quotient(a * b) == E.R - 1 for a, b in worst)
    worst2 = E.worst_pairs(("w2", "w", "w2", "w"), rnd, 50)
    assert len(worst2) == 50 and all(E.mont_quotient(a * x + b * y) == E.R - 1 for a, x, b, y in worst2)


def test_claimed_bounds_hold_in_the_model():
    """each bound stated in fp.cuh / vm_exec2.cuh, checked two ways: the supremum over the whole input domain
    (a b + (R - 1) q) / R, and the largest value on the corpus"""
    q, R = E.Q, E.R

    def sup(*pairs):   # sup of (sum of products + (R - 1) q) / R over operands below the given limits
        return Fraction(sum(x * y for x, y in pairs) + (R - 1) * q, R * q)

    assert sup((2 * q, 2 * q)) < Fraction(141, 100)                   # fp.cuh:372: weakly reduced inputs
    assert sup((4 * q, 4 * q)) < Fraction(263, 100)                   # fp.cuh:373: unreduced sums
    assert sup((2 * q, 2 * q), (2 * q + 1, 2 * q)) < Fraction(182, 100)   # fp.cuh:474: two-row product, a, b <= 2q
    assert sup((4 * q, 2 * q)) < Fraction(182, 100)                   # fp.cuh:722: (2 a0) a1
    # fp.cuh:721 / vm_exec2.cuh fp_sqr2_coeff: (a0 + a1)(a0 - a1 + 2q) <= (a0 + q)^2 < 9 q^2, so the result stays
    # below 2q and the conditional subtraction after it never fires for weakly reduced inputs
    assert sup((3 * q, 3 * q)) < Fraction(192, 100) < 2
    assert sup((E.R2, R)) < Fraction(169, 100)                         # to_mont: R^2 mod q times any 384-bit value
    assert 9 * q < R                                                   # fp.cuh:374: (alpha + 1) q < 2^384, alpha <= 8
    assert 5 * q < R // 2 + R // 50                                    # fp.cuh:474: 5q = 0.51 R
    rnd = random.Random(2)
    for label, (fn, doms, claim) in E.CLAIMS.items():
        cases = [tuple(E.draw(d, rnd) for d in doms) for _ in range(2000)]
        if label.startswith(("product", "two-row")):
            cases += E.worst_pairs(doms, rnd, 500)
        top = max(fn(*c) for c in cases)
        assert top < claim * q, (label, top / q)


def test_fp2_mul_t2_subtraction_keeps_fp_sub_in_its_domain():
    """fp2_mul's subtraction of 2q from t2 keeps fp_sub's first operand weakly reduced; it does not change the
    output integer: t2 - t0 - t1 = (a0 b1 + a1 b0 + (M - M0 - M1) q) / R < 1.81 q, so both ways give the same
    value in [0, 2q).  So the exact-output tests cannot see it; this test pins that t2 does reach [2q, 2.63q)."""
    rnd = random.Random(5)
    above = 0
    for a0, a1, b0, b1 in E.corpus("fp2_mul", rnd, 3000, 3000):
        t0, t1, t2 = E.mont(a0, b0), E.mont(a1, b1), E.mont(a0 + a1, b0 + b1)
        assert t2 < Fraction(263, 100) * E.Q
        above += t2 >= E.Q2
        assert E.sub(E.sub(t2, t0), t1) == E.fp2_mul(a0, a1, b0, b1)[1]     # the same integer without it
    assert above > 10


def test_to_mont_is_exact_for_any_384_bit_value(probe):
    """LDBE48 / LDBE32 convert raw input bytes with fp_to_mont: R^2 mod q is the first operand, so any 384-bit
    value, 2^384 - 1 included, may be the second"""
    rnd = random.Random(3)
    raws = E.edge_values("raw") + [rnd.getrandbits(384) for _ in range(3000)] + \
        [E.R - 1 - rnd.getrandbits(64) for _ in range(500)] + [k * E.Q + rnd.randrange(E.Q) for k in range(10)]
    # R^2 mod q = 2^s o is even: the largest reduction quotient of its products is R - 2^s, reached by these raws
    s = (E.R2 & -E.R2).bit_length() - 1
    base = E.Q * pow(E.R2 >> s, -1, 1 << (384 - s)) % (1 << (384 - s))
    worst = [base + (k << (384 - s)) for k in range(1 << s)][:64]
    assert all(E.mont_quotient(E.R2 * r) == E.R - (1 << s) for r in worst)
    raws += worst
    for op in (E.FP_OPS["to_mont"][0], E.FP_OPS["mul_inline"][0], E.FP_OPS["mul_looped"][0]):
        args = [(r,) if op == E.FP_OPS["to_mont"][0] else (E.R2, r) for r in raws]
        got = probe(np.full(len(args), op), args)
        for r, g in zip(raws, got):
            assert g[0] == E.to_mont(r), (op, hex(r))
            assert g[0] < E.Q2


def test_first_operand_precondition_is_real(probe):
    """the product is NOT symmetric in its limits: with 2^384 - 1 as the FIRST operand the carry chains lose a
    bit for some second operands (so fp_to_mont must keep the raw value second), while a first operand up to 8q
    is exact (checked on the corpus).  Host-only: out-of-domain operands prove nothing on the device."""
    rnd = random.Random(4)
    bs = [E.R2] + [rnd.randrange(E.Q, E.Q2) for _ in range(200)]
    for op in (E.FP_OPS["mul_inline"][0], E.FP_OPS["mul_looped"][0]):
        got = probe(np.full(len(bs), op), [(E.R - 1, b) for b in bs])
        wrong = [b for b, g in zip(bs, got) if g[0] != E.mont(E.R - 1, b)]
        assert E.R2 in wrong and len(wrong) > 10, (op, len(wrong))
