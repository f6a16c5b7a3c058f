"""Pairing entry points with the reference's names (bls_py/pairing.py:51-92) over the GPU
engine.  miller_loop() values are not byte-comparable with the reference's (see
include/b200bls.h); everything after a final exponentiation is."""
from . import engine
from .fields import Fq12


def _pack(Ps, Qs):
    if len(Ps) != len(Qs):
        raise ValueError("Ps and Qs differ in length")
    for p, q in zip(Ps, Qs):
        if p.g2 or not q.g2:
            raise Exception("invalid elements")
    return b"".join(p.raw for p in Ps), b"".join(q.raw for q in Qs)


def ate_pairing(P, Q, ec=None):
    P, Q = _pack([P], [Q])
    return Fq12(engine.pairing_batch(P, Q).tobytes())


def ate_pairing_multi(Ps, Qs, ec=None):
    """prod_i miller(P_i, Q_i) with ONE final exponentiation (pairing.py:84-92)"""
    P, Q = _pack(list(Ps), list(Qs))
    return Fq12(engine.pairing_multi(P, Q).tobytes())


def ate_pairing_multi_batch(groups):
    """[ate_pairing_multi(Ps, Qs) for (Ps, Qs) in groups] in one device pass -> list of Fq12"""
    groups = [(list(Ps), list(Qs)) for Ps, Qs in groups]
    packed = [_pack(Ps, Qs) for Ps, Qs in groups]
    P = b"".join(p for p, _ in packed)
    Q = b"".join(q for _, q in packed)
    out = engine.pairing_multi_batch(P, Q, [len(Ps) for Ps, _ in groups]).tobytes()
    return [Fq12(out[576 * i:576 * (i + 1)]) for i in range(len(groups))]


def ate_pairing_batch(Ps, Qs):
    """independent pairings, one per (P_i, Q_i) -> list of Fq12"""
    P, Q = _pack(list(Ps), list(Qs))
    out = engine.pairing_batch(P, Q).tobytes()
    return [Fq12(out[576 * i:576 * (i + 1)]) for i in range(len(Ps))]


def miller_loop(P, Q, ec=None):
    P, Q = _pack([P], [Q])
    return Fq12(engine.miller_loop_batch(P, Q).tobytes())


def final_exponentiation(element, ec=None):
    return Fq12(engine.final_exp_batch(element.raw).tobytes())
