"""Both device executors at non-canonical representatives, in every launch mode.

Every Fq value inside the VM is only weakly reduced (< 2q), and which representative of x mod q a register holds
after an input load is fixed by the input's ENCODING: LDBE48 computes to_mont(x + k q) = mont(R^2 mod q, x + k q),
which is x R mod q or x R mod q + q depending on k (tests/fp_exact.py states the exact integer).  These tests
choose k so that the device holds zero as q, coefficients at the high representative (up to ~1.67 q, the highest a
load reaches), Fq2 values with a1 = 0 (the paired MUL2 then multiplies by exactly 2q) or a1 = q, and pairs whose
Karatsuba sums come near their maximum.  The outputs must equal the oracle's bytes.

The launcher picks the kernel per launch (b200bls.cu launch_program): B200BLS_KERNEL (read once, at init) forces
the one-thread (1) or the paired (2) kernel; unset, isolated launches of <= 128 items per SM with the automatic
shape go to the paired kernel and every other launch to the one-thread kernel.  So each kernel setting runs in its
own subprocess, and inside it every launch shape (b200bls_set_ctas_per_sm 0..5) and ragged batch sizes 1, 17, 129
and sm_count * 128 + 1.  Every mode must match the oracle, and all modes must be byte-identical to each other.

The subprocess entry point is this file run as a script: `python test_gpu_weak_reduction.py <expected.pkl> <out.json>`.
"""
import hashlib
import json
import os
import pickle
import random
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (os.path.join(ROOT, "python-bls_b200"), os.path.join(ROOT, "oracle"), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import bls_oracle as O  # noqa: E402
import fp_exact as E  # noqa: E402

Q = O.Q
SHAPES = (0, 1, 2, 3, 4, 5)
KERNELS = (None, "1", "2")
FIELD_OPS = ("add", "sub", "mul", "sqr", "neg", "inv")


# ---------------------------------------------------------------------------------------------------------------
# encodings: x + k q chosen for the representative the device will hold
# ---------------------------------------------------------------------------------------------------------------
def representatives(x):
    """{k: the representative LDBE48 leaves in the register for the input bytes x + k q}"""
    return {k: E.to_mont(x + k * Q) for k in range(E.R // Q + 1) if x + k * Q < E.R}


def encode(x, want):
    """x in [0, q) -> input integer: 'canon' x itself; 'low' / 'high' a k that loads the representative below /
    at or above q (the other one when that is all x has); 'zeroq' q for x = 0 (held as q)"""
    if want == "canon":
        return x
    if want == "zeroq":
        assert x == 0
        return Q
    reps = representatives(x)
    ks = [k for k, r in reps.items() if (r >= Q) == (want == "high")] or list(reps)
    return x + max(ks, key=lambda k: reps[k] if want == "high" else -reps[k]) * Q


def top_values(rnd, n):
    """values whose high representative is among the largest a load can reach (~1.6 q and above)"""
    best = []
    for _ in range(3000):
        x = rnd.randrange(Q)
        best.append((max(representatives(x).values()), x))
    best.sort(reverse=True)
    assert best[0][0] > 1.6 * Q
    return [x for _, x in best[:n]]


def field_elements(level, rnd, tops):
    """(canonical coefficient tuples, per-coefficient encodings): the representative mixes the tests are about"""
    vals, encs = [], []

    def add(v, e):
        vals.append(tuple(v))
        encs.append(tuple(e))
    for pattern in ("high", "low", "alt", "zeroq", "a1zero", "a1q", "top", "top", "canon", "mix", "mix", "mix"):
        v = [rnd.randrange(Q) for _ in range(level)]
        e = ["high"] * level
        if pattern == "low":
            e = ["low"] * level
        elif pattern == "alt":
            e = ["high" if i % 2 else "low" for i in range(level)]
        elif pattern == "zeroq":
            v = [0] * level
            e = ["zeroq"] * level
        elif pattern in ("a1zero", "a1q"):          # odd coefficients zero: every Fq2 has a1 = 0, held as 0 / q
            for i in range(1, level, 2):
                v[i] = 0
                e[i] = "canon" if pattern == "a1zero" else "zeroq"
        elif pattern == "top":
            v = [rnd.choice(tops) for _ in range(level)]
        elif pattern == "mix":
            e = [rnd.choice(("high", "low", "canon")) for _ in range(level)]
        if level == 1 and pattern in ("a1zero", "a1q"):
            v, e = [rnd.choice(tops)], ["high"]
        add(v, e)
    return vals, encs


def ser_int(xs):
    return b"".join(int(x).to_bytes(48, "big") for x in xs)


def ser_enc(vals, encs):
    return b"".join(ser_int(encode(x, e) for x, e in zip(v, en)) for v, en in zip(vals, encs))


def _field_fns(level):
    if level == 1:
        return {"add": lambda a, b: ((a[0] + b[0]) % Q,), "sub": lambda a, b: ((a[0] - b[0]) % Q,),
                "mul": lambda a, b: (a[0] * b[0] % Q,), "neg": lambda a: (-a[0] % Q,), "inv": lambda a: (O.fq_inv(a[0]),)}
    p = {2: "f2", 6: "f6", 12: "f12"}[level]
    return {k: getattr(O, "%s_%s" % (p, k)) for k in ("add", "sub", "mul", "neg", "inv")}


def _inv(fn, a):
    return tuple([0] * len(a)) if not any(a) else tuple(fn(a))


def _f2_root(x):
    """the reference's Fq2 root, None when it has none (a real input goes to the Fq root, as the library does)"""
    try:
        r = O.f2_sqrt(x)
    except ValueError:
        return None
    return (r, 0) if isinstance(r, int) else r


def _pt1(p, enc):
    """affine G1 point -> 96 bytes with coordinate encodings enc ('canon', 'high', 'low'; zero as q)"""
    return ser_int(encode(c, "zeroq" if c == 0 and e != "canon" else e) for c, e in zip(p[:2], enc))


def _pt2(p, enc):
    cs = (p[0][0], p[0][1], p[1][0], p[1][1])
    return ser_int(encode(c, "zeroq" if c == 0 and e != "canon" else e) for c, e in zip(cs, enc))


def _ser1(p):
    return bytes(96) if p[2] else ser_int(p[:2])      # infinity as zero bytes


def _ser2(p):
    return bytes(192) if p[2] else ser_int((p[0][0], p[0][1], p[1][0], p[1][1]))


def build_cases():
    """{name: (input byte strings per argument, expected output bytes, widths)}: every case set is a small list of
    items; the worker tiles it to the batch size"""
    rnd = random.Random(0x5EED)
    tops = top_values(rnd, 16)
    cases = {}
    for level in (1, 2, 6, 12):
        fns = _field_fns(level)
        a, ea = field_elements(level, rnd, tops)
        b, eb = field_elements(level, rnd, tops)
        A, B = ser_enc(a, ea), ser_enc(b, eb)
        for op in FIELD_OPS:
            if op in ("add", "sub", "mul"):
                want = [fns[op](x, y) for x, y in zip(a, b)]
                args = (A, B)
            elif op == "sqr":
                want = [fns["mul"](x, x) for x in a]
                args = (A,)
            elif op == "inv":
                want = [_inv(fns["inv"], x) for x in a]
                args = (A,)
            else:
                want = [fns["neg"](x) for x in a]
                args = (A,)
            cases["field_%d_%s" % (level, op)] = (args, b"".join(ser_int(w) for w in want))
    # Frobenius and powers on the Fq12 set, Fq / Fq2 square roots
    a12, e12 = field_elements(12, rnd, tops)
    A12 = ser_enc(a12, e12)
    for i in (1, 2, 3):
        cases["frob_12_%d" % i] = ((A12,), b"".join(ser_int(O.f12_frob(x, i)) for x in a12))
    es = [(1 << 384) - 1, Q - 1, 0, 1, 2, 5] + [rnd.getrandbits(384) for _ in range(6)]
    cases["pow_12"] = ((A12, ser_int(es)), b"".join(ser_int(O.f12_pow(x, e)) for x, e in zip(a12, es)))
    a1, e1 = field_elements(1, rnd, tops)
    cases["pow_1"] = ((ser_enc(a1, e1), ser_int(es)), ser_int(pow(x[0], e, Q) for x, e in zip(a1, es)))
    sq1 = [(x[0] * x[0] % Q,) for x in a1]
    cases["sqrt_1"] = ((ser_enc(sq1, e1),), ser_int(O.fq_sqrt(x[0]) for x in sq1) + bytes([1] * len(sq1)))
    a2, e2 = field_elements(2, rnd, tops)
    sq2 = [O.f2_mul(x, x) for x in a2]
    roots2 = [_f2_root(x) for x in sq2]
    cases["sqrt_2"] = ((ser_enc(sq2, e2),), b"".join(ser_int(r or (0, 0)) for r in roots2) +
                       bytes([int(r is not None) for r in roots2]))
    # 512 dependent Fq2 products, never canonicalised in between
    a2b, e2b = field_elements(2, rnd, tops)
    chain = [O.f2_mul(x, O.f2_pow(y, 512)) for x, y in zip(a2, a2b)]
    cases["fq2_mul_chain"] = ((ser_enc(a2, e2), ser_enc(a2b, e2b)), b"".join(ser_int(w) for w in chain))
    # affine inputs with non-canonical coordinates
    enc1 = [("high", "high"), ("low", "low"), ("high", "low"), ("low", "high")]
    enc2 = [("high",) * 4, ("low",) * 4, ("high", "low", "low", "high"), ("low", "high", "high", "low")]
    ks = [3, 5, 0xDEADBEEF, O.N - 1]
    p1 = [O.aff_mul(k, O.G1) for k in ks] + [(0, 2, False)]   # (0, 2): x = 0, held as q; order 3
    p2 = [O.aff_mul(k + 11, O.G2) for k in ks]
    sc = [7, 0, O.N - 2, rnd.getrandbits(255)]
    e1s = enc1 + [("high", "high")]
    cases["scalar_mul_g1"] = ((b"".join(_pt1(p, e) for p, e in zip(p1, enc1)), b"".join(s.to_bytes(32, "big") for s in sc)),
                              b"".join(_ser1(O.aff_mul(s, p)) for p, s in zip(p1, sc)))
    cases["scalar_mul_g2"] = ((b"".join(_pt2(p, e) for p, e in zip(p2, enc2)), b"".join(s.to_bytes(32, "big") for s in sc)),
                              b"".join(_ser2(O.aff_mul(s, p)) for p, s in zip(p2, sc)))
    q1 = [p1[0], O.aff_neg(p1[1]), p1[0], p1[2], (0, Q - 2, False)]      # P + P, P + (-P) = infinity, P + Q, T + (-T)
    cases["point_add_g1"] = ((b"".join(_pt1(p, e) for p, e in zip(p1, e1s)), b"".join(_pt1(p, e) for p, e in zip(q1, enc1[::-1] + [("high", "low")]))),
                             b"".join(_ser1(O.aff_add(p, q)) for p, q in zip(p1, q1)))
    q2 = [p2[0], O.aff_neg(p2[1]), p2[0], p2[2]]
    cases["point_add_g2"] = ((b"".join(_pt2(p, e) for p, e in zip(p2, enc2)), b"".join(_pt2(p, e) for p, e in zip(q2, enc2[::-1]))),
                             b"".join(_ser2(O.aff_add(p, q)) for p, q in zip(p2, q2)))
    cases["subgroup_g1"] = ((b"".join(_pt1(p, e) for p, e in zip(p1, e1s)),), bytes([1, 1, 1, 1, 0]))
    cases["subgroup_g2"] = ((b"".join(_pt2(p, e) for p, e in zip(p2, enc2)),), bytes([1, 1, 1, 1]))
    cases["pairing"] = ((b"".join(_pt1(p, e) for p, e in zip(p1[:4], enc1)), b"".join(_pt2(p, e) for p, e in zip(p2, enc2))),
                        b"".join(O.f12_serialize(O.ate_pairing(p, q)) for p, q in zip(p1[:4], p2)))
    sks = [O.sk_from_seed(b"weak %d" % i) for i in range(4)]
    hs = [O.hash256(b"weak message %d" % i) for i in range(4)]
    sigs = [O.sign_prehashed(sk, h) for sk, h in zip(sks, hs)]
    hs_used = [hs[0], hs[1], hs[3], hs[3]]                     # item 2: a signature on another message
    want_v = bytes([int(O.verify(O.pk_of(sk), h, s)) for sk, h, s in zip(sks, hs_used, sigs)])
    assert want_v == bytes([1, 1, 0, 1])
    cases["verify"] = ((b"".join(_pt1(O.pk_of(sk), e) for sk, e in zip(sks, enc1)), b"".join(hs_used),
                        b"".join(_pt2(s, e) for s, e in zip(sigs, enc2))), want_v)
    return cases


# ---------------------------------------------------------------------------------------------------------------
# the worker: one process per kernel setting
# ---------------------------------------------------------------------------------------------------------------
def _tile(buf, n_base, n):
    w = len(buf) // n_base
    reps = -(-n // n_base)
    return np.frombuffer((buf * reps)[:w * n], dtype=np.uint8)


def _run_case(engine, name, args, n_base, n):
    t = [_tile(a, n_base, n) for a in args]
    if name.startswith("field_"):
        _, level, op = name.split("_")
        return engine.field_op(int(level), op, *t)
    if name.startswith("frob_12_"):
        return engine.field_frob(12, int(name[-1]), t[0])
    if name.startswith("pow_"):
        return engine.field_pow(int(name[4:]), t[0], t[1])
    if name.startswith("sqrt_"):
        out, ok = engine.field_sqrt(int(name[5:]), t[0])
        return np.concatenate([out, ok])
    if name == "fq2_mul_chain":
        bufs = [engine.DeviceBuffer(96 * n).upload(t[0]), engine.DeviceBuffer(96 * n).upload(t[1]),
                engine.DeviceBuffer(96 * n)]
        try:
            engine.run_program_dev("fq2_mul_chain", n, bufs, [96, 96, 96])
            return bufs[2].download(96 * n)
        finally:
            for b in bufs:
                b.free()
    if name.startswith("scalar_mul_"):
        return engine.scalar_mul(t[0], t[1], name.endswith("g2"))
    if name.startswith("point_add_"):
        return engine.point_add(t[0], t[1], name.endswith("g2"))
    if name.startswith("subgroup_"):
        return engine.subgroup_check(t[0], name.endswith("g2"))
    if name == "pairing":
        return engine.pairing_batch(t[0], t[1])
    if name == "verify":
        return engine.verify_batch(t[0], t[1], t[2])
    raise ValueError(name)


def _expected_tiled(want, n_base, n, has_flags):
    """expected bytes for n items; sqrt outputs are roots then flags"""
    if not has_flags:
        return _tile(want, n_base, n)
    roots, flags = want[:-n_base], want[-n_base:]
    return np.concatenate([_tile(roots, n_base, n), _tile(flags, n_base, n)])


def worker(expected_path, out_path):
    from bls_b200 import _lib, engine
    _lib.init(0)
    with open(expected_path, "rb") as fh:
        cases = pickle.load(fh)
    sm = _lib.lib.b200bls_sm_count()
    batches = (1, 17, 129, sm * 128 + 1)
    res = {"kernel": os.environ.get("B200BLS_KERNEL"), "sm_count": sm, "runs": {}, "bad": []}
    for shape in SHAPES:
        _lib.check(_lib.lib.b200bls_set_ctas_per_sm(shape))
        for n in batches:
            for name, (args, want, n_base) in cases.items():
                got = _run_case(engine, name, args, n_base, n)
                exp = _expected_tiled(want, n_base, n, name.startswith("sqrt_"))
                key = "%s/shape%d/n%d" % (name, shape, n)
                res["runs"][key] = hashlib.sha256(got.tobytes()).hexdigest()
                if got.size != exp.size or not np.array_equal(got, exp):
                    idx = int(np.argmax(got != exp)) if got.size == exp.size else -1
                    res["bad"].append("%s first differing byte %d" % (key, idx))
    _lib.check(_lib.lib.b200bls_set_ctas_per_sm(0))
    with open(out_path, "w") as fh:
        json.dump(res, fh)


# ---------------------------------------------------------------------------------------------------------------
# the tests
# ---------------------------------------------------------------------------------------------------------------
WIDTHS = {"frob_12": 576, "pow_12": 576, "pow_1": 48, "sqrt_1": 48, "sqrt_2": 96, "fq2_mul_chain": 96,
          "scalar_mul_g1": 96, "scalar_mul_g2": 192, "point_add_g1": 96, "point_add_g2": 192, "subgroup_g1": 96,
          "subgroup_g2": 192, "pairing": 96, "verify": 96}   # bytes per item of each case's first argument


def _width(name):
    if name.startswith("field_"):
        return 48 * int(name.split("_")[1])
    return WIDTHS[name.rsplit("_", 1)[0] if name.startswith("frob_") else name]


@pytest.fixture(scope="module")
def expected_file(tmp_path_factory):
    """the cases with their item counts, pickled for the worker processes"""
    packed = {}
    for name, (args, want) in build_cases().items():
        nb = len(args[0]) // _width(name)
        assert len(args[0]) == nb * _width(name) and nb > 0, name
        packed[name] = (args, want, nb)
    path = tmp_path_factory.mktemp("weak") / "expected.pkl"
    with open(path, "wb") as fh:
        pickle.dump(packed, fh)
    return path


def test_encodings_reach_the_representatives():
    """CPU: the encodings do what the device tests rely on -- q loads as the representative q, high / low
    representatives are reachable for most x, and the top ones are above 1.6 q"""
    assert E.to_mont(Q) == Q and E.to_mont(0) == 0
    rnd = random.Random(7)
    both = 0
    for _ in range(300):
        x = rnd.randrange(Q)
        hi, lo = encode(x, "high"), encode(x, "low")
        assert hi % Q == x and lo % Q == x and hi < E.R and lo < E.R
        rh, rl = E.to_mont(hi), E.to_mont(lo)
        assert rh % Q == rl % Q == x * E.R % Q and rl < E.Q2 and rh < E.Q2
        both += rh >= Q > rl
    assert 120 < both < 260
    assert max(E.to_mont(encode(x, "high")) for x in top_values(rnd, 4)) > 1.6 * Q
    # Fq2 with a1 = 0 as 0: the paired MUL2's role 0 multiplies b1 by 2q - 0 = 2q exactly
    assert E.neg_raw_2q(E.to_mont(0)) == E.Q2


def test_cases_are_self_consistent():
    """CPU: the oracle side of the device test (expected bytes from canonical values, encodings that reduce to
    them), so that a failure on the device points at the device"""
    cases = build_cases()
    assert len(cases) == 4 * len(FIELD_OPS) + 3 + 2 + 2 + 1 + 2 + 2 + 2 + 1 + 1
    args, want = cases["field_2_mul"]
    a, b = args
    for i in range(len(a) // 96):
        x = [int.from_bytes(a[96 * i + 48 * k:96 * i + 48 * (k + 1)], "big") % Q for k in (0, 1)]
        y = [int.from_bytes(b[96 * i + 48 * k:96 * i + 48 * (k + 1)], "big") % Q for k in (0, 1)]
        assert want[96 * i:96 * (i + 1)] == ser_int(O.f2_mul(tuple(x), tuple(y)))
    assert any(int.from_bytes(a[k:k + 48], "big") >= Q for k in range(0, len(a), 48))   # non-canonical inputs


@pytest.mark.gpu
def test_every_mode_matches_the_oracle(expected_file, tmp_path):
    path = expected_file
    results = {}
    for kernel in KERNELS:
        env = dict(os.environ)
        env.pop("B200BLS_KERNEL", None)
        env.pop("B200BLS_CTAS_PER_SM", None)
        if kernel:
            env["B200BLS_KERNEL"] = kernel
        out = tmp_path / ("modes_%s.json" % (kernel or "auto"))
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), str(path), str(out)], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
        assert proc.returncode == 0, proc.stdout[-4000:]
        with open(out) as fh:
            results[kernel or "auto"] = json.load(fh)
    for label, res in results.items():
        assert not res["bad"], "B200BLS_KERNEL=%s: %d runs differ from the oracle, first: %s" % (
            label, len(res["bad"]), res["bad"][:5])
    # every (kernel, shape, batch) mode gives the same bytes for the same batch
    keys = results["auto"]["runs"].keys()
    for key in keys:
        digests = {label: res["runs"][key] for label, res in results.items()}
        assert len(set(digests.values())) == 1, (key, digests)
    n_modes = len(results) * len(SHAPES) * 4
    print("modes (kernel, shape, batch): %d, runs compared: %d" % (n_modes, sum(len(r["runs"]) for r in results.values())))


if __name__ == "__main__":
    worker(sys.argv[1], sys.argv[2])
