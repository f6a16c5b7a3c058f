"""GPU: the batched multi-pairing (b200bls_pairing_multi_batch and its _dev form, engine.pairing_multi_batch,
pairing.ate_pairing_multi_batch).

Every group's output must be the bytes of one b200bls_pairing_multi call on that group, in every launch mode: each
B200BLS_KERNEL setting (unset, 1, 2) runs in its own subprocess, and inside it every launch shape
(b200bls_set_ctas_per_sm 0..5) over a ragged layout -- empty groups mixed in, groups of 1, 2, L - 1, L, L + 1 and one of
more than L^2 pairs (L = 16, csrc/multi_plan.h) -- and, in the automatic shape, 65,536 groups of 2.  A loop of 65,536
per-group calls takes minutes (each call is four dependent launches of single-item latency), so the large layout is
compared with per-group calls on its first SAMPLE groups and, whole, with the product of two pairing_batch outputs per
group (canonical Fq12 values, multiplied by the f12_mul program).  The subprocess entry point is this file run as a
script: `python test_gpu_multi_pairing.py <out.json>`.
"""
import ctypes
import json
import os
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

pytestmark = pytest.mark.gpu

SHAPES = (0, 1, 2, 3, 4, 5)
KERNELS = (None, "1", "2")
RAGGED = [0, 1, 2, 0, 15, 16, 17, 1, 0, 300, 2, 3, 0, 16, 33]
SAMPLE = 256
ONE = O.f12_serialize(O.F12_ONE)
E_ARG = -3


def _points(engine, n, seed):
    """n seeded multiples of the generators, every 7th P and every 11th Q the point at infinity"""
    from bls_b200.workloads import G1_BYTES, G2_BYTES
    rng = np.random.Generator(np.random.PCG64(seed))
    P = engine.scalar_mul(np.tile(G1_BYTES, n), rng.integers(0, 256, size=32 * n, dtype=np.uint8), False)
    Q = engine.scalar_mul(np.tile(G2_BYTES, n), rng.integers(0, 256, size=32 * n, dtype=np.uint8), True)
    P.reshape(n, 96)[::7] = 0
    Q.reshape(n, 192)[3::11] = 0
    return P, Q


def _per_group(engine, P, Q, counts):
    """the reference: one b200bls_pairing_multi per group"""
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return b"".join(engine.pairing_multi(P[96 * a:96 * b], Q[192 * a:192 * b]).tobytes() for a, b in zip(off, off[1:]))


def _per_group_dev(engine, P, Q, counts):
    """the reference for many groups: a loop of b200bls_pairing_multi_dev on device-resident data"""
    from bls_b200._lib import check, lib
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    dP, dQ = engine.DeviceBuffer(P.size).upload(P), engine.DeviceBuffer(Q.size).upload(Q)
    dO = engine.DeviceBuffer(576 * len(counts))
    for g, (a, b) in enumerate(zip(off, off[1:])):
        check(lib.b200bls_pairing_multi_dev(ctypes.c_void_p(dP.ptr + 96 * int(a)), ctypes.c_void_p(dQ.ptr + 192 * int(a)),
                                            ctypes.c_void_p(dO.ptr + 576 * g), int(b - a)))
    return dO.download().tobytes()


def _flags(ref, n):
    return bytes(int(ref[576 * g:576 * (g + 1)] == ONE) for g in range(n))


def worker(out_path):
    from bls_b200 import _lib, engine
    _lib.init(0)
    bad = []
    P, Q = _points(engine, sum(RAGGED), 0xB2005EC0)
    ref = _per_group(engine, P, Q, RAGGED)
    for shape in SHAPES:
        _lib.check(_lib.lib.b200bls_set_ctas_per_sm(shape))
        if engine.pairing_multi_batch(P, Q, RAGGED).tobytes() != ref:
            bad.append(("ragged", shape))
        if engine.pairing_multi_batch(P, Q, RAGGED, check=True).tobytes() != _flags(ref, len(RAGGED)):
            bad.append(("ragged check", shape))
    _lib.check(_lib.lib.b200bls_set_ctas_per_sm(0))
    n = 65536
    P, Q = _points(engine, 2 * n, 0xB2005EC1)
    got = engine.pairing_multi_batch(P, Q, [2] * n).tobytes()
    if got[:576 * SAMPLE] != _per_group_dev(engine, P[:192 * SAMPLE], Q[:384 * SAMPLE], [2] * SAMPLE):
        bad.append(("65536 x 2: per-group sample", 0))
    e = engine.pairing_batch(P, Q).reshape(n, 2, 576)
    ref = engine.field_op(12, "mul", e[:, 0], e[:, 1]).tobytes()
    if got != ref:
        bad.append(("65536 x 2", 0))
    if engine.pairing_multi_batch(P, Q, [2] * n, check=True).tobytes() != _flags(ref, n):
        bad.append(("65536 x 2 check", 0))
    with open(out_path, "w") as fh:
        json.dump({"mismatches": bad}, fh)


@pytest.mark.parametrize("kernel", KERNELS)
def test_every_mode_matches_per_group_calls(kernel, tmp_path):
    out = tmp_path / "res.json"
    env = dict(os.environ)
    env.pop("B200BLS_KERNEL", None)
    env.pop("B200BLS_CTAS_PER_SM", None)
    if kernel:
        env["B200BLS_KERNEL"] = kernel
    subprocess.check_call([sys.executable, os.path.abspath(__file__), str(out)], env=env, cwd=ROOT)
    assert json.loads(out.read_text())["mismatches"] == []


def _ser_p(p):
    return bytes(96) if p[2] else p[0].to_bytes(48, "big") + p[1].to_bytes(48, "big")


def _ser_q(q):
    return bytes(192) if q[2] else b"".join(c.to_bytes(48, "big") for c in (q[0][0], q[0][1], q[1][0], q[1][1]))


def test_reference_vectors():
    """the reference's ate_pairing_multi outputs (tests/golden/pairing_kat.json) and an oracle group, as one batch"""
    from bls_b200 import engine
    from conftest import load_golden
    g = load_golden("pairing_kat.json")
    groups = [[g["pairs"][i] for i in m["idx"]] for m in g["multi"]]
    P = b"".join(bytes.fromhex(c["p"]["x"]) + bytes.fromhex(c["p"]["y"]) for grp in groups for c in grp)
    Q = b"".join(bytes.fromhex(c["q"]["x"]) + bytes.fromhex(c["q"]["y"]) for grp in groups for c in grp)
    ps, qs = [O.aff_mul(3, O.G1), O.aff_mul(5, O.G1)], [O.aff_mul(7, O.G2), O.aff_mul(2, O.G2)]
    P += b"".join(_ser_p(p) for p in ps)
    Q += b"".join(_ser_q(q) for q in qs)
    out = engine.pairing_multi_batch(P, Q, [len(grp) for grp in groups] + [2]).tobytes()
    for k, m in enumerate(g["multi"]):
        assert out[576 * k:576 * (k + 1)].hex() == m["out"], k
    assert out[576 * len(groups):] == O.f12_serialize(O.ate_pairing_multi(ps, qs))


def test_check_against_constructed_identities():
    from bls_b200 import engine
    a, b = 0x1234567, 0xfedcba98765
    P, Q = O.G1, O.G2
    aP, aQ, bP = O.aff_mul(a, P), O.aff_mul(a, Q), O.aff_mul(b, P)
    a1Q = O.aff_mul(a + 1, Q)
    groups = [
        [(aP, Q), (O.aff_neg(P), aQ)],                               # e(aP, Q) e(-P, aQ) = 1
        [(aP, Q), (O.aff_neg(P), a1Q)],                              # corrupted second member
        [],                                                          # empty: one
        [(P, Q)],                                                    # e(P, Q) != 1
        [((0, 0, True), Q)],                                         # infinity: 1
        [(aP, Q), (O.aff_neg(P), aQ), (bP, Q), (O.aff_neg(bP), Q)],  # two identities
        [(aP, Q), (O.aff_neg(P), aQ), (bP, Q)],                      # one member too many
        [(O.aff_neg(aP), Q), (P, aQ)],
    ]
    want = [1, 0, 1, 0, 1, 1, 0, 1]
    Pb = b"".join(_ser_p(p) for grp in groups for p, _ in grp)
    Qb = b"".join(_ser_q(q) for grp in groups for _, q in grp)
    counts = [len(grp) for grp in groups]
    assert list(engine.pairing_multi_batch(Pb, Qb, counts, check=True)) == want
    full = engine.pairing_multi_batch(Pb, Qb, counts).tobytes()
    assert [int(full[576 * g:576 * (g + 1)] == ONE) for g in range(len(groups))] == want
    off = np.concatenate([[0], np.cumsum(counts)])
    assert engine.pairing_multi_batch(Pb, Qb, off, offsets=True).tobytes() == full


def test_python_api():
    from bls_b200 import ate_pairing_multi, ec
    from bls_b200.pairing import ate_pairing_multi_batch
    g1, g2 = ec.generator_Fq(), ec.generator_Fq2()
    groups = [([g1 * 3, (g1 * 15).negate()], [g2 * 5, g2]), ([], []), ([g1 * 2], [g2 * 9]),
              ([g1, g1 * 4, g1 * 5], [g2 * 6, g2 * 7, g2 * 8])]
    got = ate_pairing_multi_batch(groups)
    assert got == [ate_pairing_multi(Ps, Qs) for Ps, Qs in groups]
    assert ate_pairing_multi_batch([]) == []
    with pytest.raises(ValueError):
        ate_pairing_multi_batch([([g1, g1], [g2])])
    with pytest.raises(Exception, match="invalid elements"):
        ate_pairing_multi_batch([([g1], [g2]), ([g2], [g1])])
    with pytest.raises(Exception, match="invalid elements"):
        ate_pairing_multi([g2], [g1])


def test_dev_form_on_two_streams():
    """two batches in flight on library streams 0 and 1, device-resident inputs, offsets and outputs"""
    from bls_b200 import engine
    from bls_b200._lib import check, lib
    layouts = [[2, 0, 17, 1, 40], [300, 0, 0, 3]]
    jobs = []
    for k, counts in enumerate(layouts):
        P, Q = _points(engine, sum(counts), 0xB2005EC2 + k)
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)
        bufs = [engine.DeviceBuffer(x.nbytes).upload(x) for x in (P, Q, off)]
        jobs.append((counts, engine.pairing_multi_batch(P, Q, counts).tobytes(), bufs,
                     engine.DeviceBuffer(576 * len(counts)), engine.DeviceBuffer(len(counts))))
    try:
        for k, (counts, _, (dP, dQ, dOff), dOut, dFlag) in enumerate(jobs):
            check(lib.b200bls_set_stream(k))
            check(lib.b200bls_pairing_multi_batch_dev(0, dP.ptr, dQ.ptr, dOff.ptr, len(counts), dOut.ptr))
            check(lib.b200bls_pairing_multi_batch_dev(1, dP.ptr, dQ.ptr, dOff.ptr, len(counts), dFlag.ptr))
        check(lib.b200bls_sync())
    finally:
        check(lib.b200bls_set_stream(0))
    for counts, ref, _, dOut, dFlag in jobs:
        assert dOut.download().tobytes() == ref
        assert dFlag.download().tobytes() == _flags(ref, len(counts))


def test_argument_errors():
    """every B200BLS_E_ARG case, in the host form (checked on the host) and in the _dev form (offsets checked on the
    device before any pairing runs)"""
    from bls_b200 import _lib, engine
    from bls_b200._lib import lib
    _lib.init()
    P, Q = _points(engine, 4, 0xB2005EC3)
    out = np.zeros(576 * 4, dtype=np.uint8)
    dP, dQ, dOut = engine.DeviceBuffer(P.size).upload(P), engine.DeviceBuffer(Q.size).upload(Q), engine.DeviceBuffer(out.size)
    bad_offsets = [[1, 4], [0, 3, 2, 4], [0, 2 ** 32], [0, 2 ** 32 + 4, 4]]
    for off in bad_offsets:
        o = np.array(off, dtype=np.uint64)
        dOff = engine.DeviceBuffer(o.nbytes).upload(o)
        for check in (0, 1):
            assert lib.b200bls_pairing_multi_batch(check, _lib.ptr(P), _lib.ptr(Q), _lib.ptr(o), o.size - 1,
                                                   _lib.ptr(out)) == E_ARG, off
            assert lib.b200bls_pairing_multi_batch_dev(check, dP.ptr, dQ.ptr, dOff.ptr, o.size - 1, dOut.ptr) == E_ARG, off
        assert b"offsets" in lib.b200bls_last_error()
    o = np.array([0, 2, 4], dtype=np.uint64)
    dOff = engine.DeviceBuffer(o.nbytes).upload(o)
    for check in (-1, 2):
        assert lib.b200bls_pairing_multi_batch(check, _lib.ptr(P), _lib.ptr(Q), _lib.ptr(o), 2, _lib.ptr(out)) == E_ARG
        assert lib.b200bls_pairing_multi_batch_dev(check, dP.ptr, dQ.ptr, dOff.ptr, 2, dOut.ptr) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, _lib.ptr(P), _lib.ptr(Q), _lib.ptr(o), 2 ** 31, _lib.ptr(out)) == E_ARG
    assert lib.b200bls_pairing_multi_batch_dev(0, dP.ptr, dQ.ptr, dOff.ptr, 2 ** 31, dOut.ptr) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, None, _lib.ptr(Q), _lib.ptr(o), 2, _lib.ptr(out)) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, _lib.ptr(P), _lib.ptr(Q), None, 2, _lib.ptr(out)) == E_ARG
    assert lib.b200bls_pairing_multi_batch_dev(0, dP.ptr, dQ.ptr, None, 2, dOut.ptr) == E_ARG
    assert lib.b200bls_pairing_multi_batch_dev(0, dP.ptr, dQ.ptr, dOff.ptr, 2, None) == E_ARG
    # n_groups = 0 does nothing; a valid call after the refusals still works
    assert lib.b200bls_pairing_multi_batch_dev(0, None, None, None, 0, None) == 0
    assert lib.b200bls_pairing_multi_batch_dev(0, dP.ptr, dQ.ptr, dOff.ptr, 2, dOut.ptr) == 0
    assert lib.b200bls_sync() == 0
    assert dOut.download(1152).tobytes() == engine.pairing_multi_batch(P, Q, [2, 2]).tobytes()
    with pytest.raises(ValueError):
        engine.pairing_multi_batch(P, Q, [2, 1])
    with pytest.raises(ValueError):
        engine.pairing_multi_batch(P, Q, [5, -1])


if __name__ == "__main__":
    worker(sys.argv[1])
