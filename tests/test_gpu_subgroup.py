"""GPU: subgroup membership checks and strict verification against the oracle's definition of membership
(on the curve and [n] P = infinity) and the oracle's verdicts, from the corpus up to full-size batches."""
import numpy as np
import pytest

import bls_oracle as O
import subgroup_corpus as SC

pytestmark = pytest.mark.gpu

INF1 = (0, 0, True)
INF2 = (O.F2_ZERO, O.F2_ZERO, True)


def _cat(pts, ser):
    return b"".join(ser(p) for p in pts)


@pytest.mark.parametrize("g2", [False, True])
def test_subgroup_check_matches_definition(g2):
    from bls_b200 import engine
    pts = SC.g2_corpus() if g2 else SC.g1_corpus()
    got = engine.subgroup_check(_cat(pts, SC.g2_bytes if g2 else SC.g1_bytes), g2)
    assert [bool(f) for f in got] == [SC.is_member(p) for p in pts]
    assert engine.subgroup_check(b"", g2).size == 0


def _genuine(seed):
    sk = O.sk_from_seed(seed)
    h = O.hash256(seed)
    return O.pk_of(sk), h, O.sign_prehashed(sk, h)


def test_strict_verification_cases_against_oracle():
    from bls_b200 import engine
    pk, h, sig = _genuine(b"strict-1")
    pk2, h2, sig2 = _genuine(b"strict-2")
    t13 = SC.order13_point()
    pk_mal = O.aff_add(pk, SC.G1_SMALL)
    sig_t = O.aff_add(sig, t13)
    # (pk, h, sig, oracle non-strict verdict, strict verdict)
    cases = [
        (SC.G1_SMALL, h, INF2, True, False),          # universal forgery with the order-3 key
        (SC.G1_SMALL, h2, INF2, True, False),
        (INF1, h, INF2, True, False),                 # infinity key, infinity signature
        (pk_mal, h, sig, True, False),                # second key for pk's signatures
        (pk, h, sig_t, False, False),                 # signature with an order-13 component
        (pk, h, sig, True, True),
        (pk2, h2, sig2, True, True),
        (pk, h2, sig, False, False),
    ]
    for c in cases:
        assert O.verify(c[0], c[1], c[2]) is c[3]
    pks = _cat([c[0] for c in cases], SC.g1_bytes)
    hs = b"".join(c[1] for c in cases)
    sigs = _cat([c[2] for c in cases], SC.g2_bytes)
    assert [bool(v) for v in engine.verify_batch(pks, hs, sigs)] == [c[3] for c in cases]
    assert [bool(v) for v in engine.verify_batch(pks, hs, sigs, strict=True)] == [c[4] for c in cases]
    # the wire forms of the cases without infinity (whose zero bytes decode to other points)
    wire = [c for c in cases if not c[0][2] and not c[2][2]]
    pk48 = b"".join(O.g1_serialize(c[0]) for c in wire)
    sig96 = b"".join(O.g2_serialize(c[2]) for c in wire)
    hs = b"".join(c[1] for c in wire)
    assert O.g1_serialize(pk_mal) != O.g1_serialize(pk)
    assert [bool(v) for v in engine.verify_batch_wire(pk48, hs, sig96)] == [c[3] for c in wire]
    assert [bool(v) for v in engine.verify_batch_wire(pk48, hs, sig96, strict=True)] == [c[4] for c in wire]
    # infinity keys written with a coordinate q: the device reads them as infinity (non-strict accepts them with the
    # infinity signature, as the oracle does the infinity key), so strict verification rejects them too
    inf_keys = SC.g1_noncanonical_encodings()[:3]
    pks = b"".join(inf_keys)
    hs = h + h2 + h
    sigs = bytes(192 * 3)
    assert O.verify(INF1, h, INF2) and O.verify(INF1, h2, INF2)
    assert [bool(v) for v in engine.verify_batch(pks, hs, sigs)] == [True] * 3
    assert [bool(v) for v in engine.verify_batch(pks, hs, sigs, strict=True)] == [False] * 3


def test_key_validate_matches_definition():
    from bls_b200 import engine
    raws = [SC.g1_bytes(p) for p in SC.g1_corpus()] + SC.g1_noncanonical_encodings()
    pts = [SC.g1_reduced(r) for r in raws]
    member = [SC.is_member(p) for p in pts]
    assert [bool(f) for f in engine.subgroup_check(b"".join(raws), False)] == member
    assert [bool(f) for f in engine.key_validate(b"".join(raws))] == [m and not p[2] for m, p in zip(member, pts)]


def test_strict_equals_nonstrict_and_membership_over_corpus():
    """every corpus key against corpus signatures, plus triples the non-strict check accepts"""
    from bls_b200 import engine
    g1, g2 = SC.g1_corpus(), SC.g2_corpus()
    n = max(len(g1), len(g2)) * 2
    pks = [g1[i % len(g1)] for i in range(n)]
    sigs = [g2[(3 * i) % len(g2)] for i in range(n)]
    hs = [O.hash256(b"corpus %d" % i) for i in range(n)]
    pk, h, sig = _genuine(b"corpus")
    for t in ((pk, h, sig), (O.aff_add(pk, SC.G1_SMALL), h, sig), (SC.G1_SMALL, h, INF2), (INF1, h, INF2)):
        pks.append(t[0])
        hs.append(t[1])
        sigs.append(t[2])
    P, S = _cat(pks, SC.g1_bytes), _cat(sigs, SC.g2_bytes)
    loose = engine.verify_batch(P, b"".join(hs), S).astype(bool)
    strict = engine.verify_batch(P, b"".join(hs), S, strict=True).astype(bool)
    want = loose & np.array([SC.is_member(p) and not p[2] for p in pks]) & np.array([SC.is_member(s) for s in sigs])
    assert (strict == want).all()
    assert list(loose[-4:]) == [True] * 4 and list(strict[-4:]) == [True, False, False, False]


def _scale_triples(n, seed):
    """n genuine (pk, H(m), sig) triples built on the device; 1 % of the keys get the order-3 point added and 1 % of
    the signatures an order-13 point, at seeded positions -> (pk48, hashes, sig96, bad_key, bad_sig)"""
    from bls_b200 import engine, synth
    from bls_b200.workloads import dev_scalar_mul
    sks = synth.scalars(seed, n)
    hs = synth.message_hashes(seed, n)
    H = engine.hash_to_g2(hs)
    sig = engine.scalar_mul(H, sks, True).reshape(n, 192)
    pk = dev_scalar_mul(sks, False).download().reshape(n, 96)
    bad_key = np.zeros(n, dtype=bool)
    bad_sig = np.zeros(n, dtype=bool)
    kb, sb = synth.corrupted_indices(seed + 1, n), synth.corrupted_indices(seed + 2, n)
    bad_key[kb] = True
    bad_sig[sb] = True
    pk[kb] = engine.point_add(pk[kb], np.tile(np.frombuffer(SC.g1_bytes(SC.G1_SMALL), np.uint8), len(kb)),
                              False).reshape(-1, 96)
    sig[sb] = engine.point_add(sig[sb], np.tile(np.frombuffer(SC.g2_bytes(SC.order13_point()), np.uint8), len(sb)),
                               True).reshape(-1, 192)
    return engine.compress(pk, False), hs, engine.compress(sig, True), bad_key, bad_sig


def test_strict_wire_verification_at_scale():
    from bls_b200 import engine
    n = 262144
    pk48, hs, sig96, bad_key, bad_sig = _scale_triples(n, 0xB2005B01)
    assert bad_key.sum() == n // 100 and bad_sig.sum() == n // 100
    loose = engine.verify_batch_wire(pk48, hs, sig96).astype(bool)
    strict = engine.verify_batch_wire(pk48, hs, sig96, strict=True).astype(bool)
    assert (loose == ~bad_sig).all()
    assert (strict == (~bad_sig & ~bad_key)).all()


def test_subgroup_check_one_million_g2_points():
    from bls_b200 import engine, synth
    from bls_b200.workloads import dev_scalar_mul
    n = 1 << 20
    pts = dev_scalar_mul(synth.scalars(0xB2005B02, n), True).download().reshape(n, 192)
    bad = synth.corrupted_indices(0xB2005B03, n)
    half = len(bad) // 2
    t13 = np.frombuffer(SC.g2_bytes(SC.order13_point()), np.uint8)
    pts[bad[:half]] = engine.point_add(pts[bad[:half]], np.tile(t13, half), True).reshape(-1, 192)
    for i in bad[half:]:                                   # off the curve: y.c0 + 1
        y0 = (int.from_bytes(bytes(pts[i, 96:144]), "big") + 1) % O.Q
        pts[i, 96:144] = np.frombuffer(y0.to_bytes(48, "big"), np.uint8)
    want = np.ones(n, dtype=bool)
    want[bad] = False
    got = engine.subgroup_check(pts, True).astype(bool)
    assert (got == want).all()


def test_python_api_subgroup_options():
    from bls_b200 import BLS, AggregationInfo, PrivateKey, PublicKey, Signature
    from bls_b200.ec import Point
    sk = PrivateKey.from_seed(b"subgroup api")
    pk = sk.get_public_key()
    msg = b"strict"
    sig = sk.sign(msg)
    # members: the same objects as without the check
    assert PublicKey.from_bytes(pk.serialize(), check_subgroup=True) == PublicKey.from_bytes(pk.serialize())
    assert Signature.from_bytes(sig.serialize(), check_subgroup=True) == sig
    assert PublicKey.from_bytes_batch([pk.serialize()] * 3, check_subgroup=True)[2] == pk
    assert Signature.from_bytes_batch([sig.serialize()] * 2, check_subgroup=True)[1] == sig
    assert pk.value.is_in_subgroup() and sig.value.is_in_subgroup()
    # non-members decode by default and raise with the check
    pk_pt = O.g1_deserialize(pk.serialize())
    mal = O.g1_serialize(O.aff_add(pk_pt, SC.G1_SMALL))
    bad_sig = O.g2_serialize(O.aff_add(O.g2_deserialize(sig.serialize()), SC.order13_point()))
    small = bytes(48)                                      # decodes to (0, 2)
    for buf in (mal, small):
        assert not PublicKey.from_bytes(buf).value.is_in_subgroup()
        with pytest.raises(ValueError):
            PublicKey.from_bytes(buf, check_subgroup=True)
        with pytest.raises(ValueError):
            PublicKey.from_bytes_batch([pk.serialize(), buf], check_subgroup=True)
    Signature.from_bytes(bad_sig)
    with pytest.raises(ValueError):
        Signature.from_bytes(bad_sig, check_subgroup=True)
    with pytest.raises(ValueError):
        Signature.from_bytes_batch([bad_sig], check_subgroup=True)
    assert Point(bytes(96), False).is_in_subgroup()
    # BLS.verify: an aggregate whose second key is pk + (0, 2)
    sk2 = PrivateKey.from_seed(b"subgroup api 2")
    pk_mal = PublicKey.from_bytes(O.g1_serialize(O.aff_add(O.g1_deserialize(sk2.get_public_key().serialize()),
                                                           SC.G1_SMALL)))
    s2 = sk2.sign(b"other")
    s2.set_aggregation_info(AggregationInfo.from_msg(pk_mal, b"other"))
    agg = BLS.aggregate_sigs([sig, s2])
    want = O.aggregate_verify([O.g1_deserialize(pk.serialize()), O.g1_deserialize(pk_mal.serialize())],
                              [O.hash256(msg), O.hash256(b"other")], O.g2_deserialize(agg.serialize()))
    assert BLS.verify(agg) is want
    assert BLS.verify(agg, strict=True) is False
    assert BLS.verify(sig, strict=True) is True
    # the infinity key, also spelled q || 0 etc., with the infinity signature
    for raw in [bytes(96)] + SC.g1_noncanonical_encodings()[:3]:
        inf_sig = Signature.from_g2(Point(bytes(192), True))
        inf_sig.set_aggregation_info(AggregationInfo.from_msg(PublicKey.from_g1(Point(raw, False)), b"anything"))
        assert BLS.verify(inf_sig, strict=True) is False
    # batch forms: the malleated key verifies sk2's signature unless strict
    hs = [O.hash256(msg), O.hash256(b"other")]
    assert BLS.verify_batch([pk, pk_mal], hs, [sig, s2]) == [True, True]
    assert BLS.verify_batch([pk, pk_mal], hs, [sig, s2], strict=True) == [True, False]
    wire = ([pk.serialize(), pk_mal.serialize()], hs, [sig.serialize(), s2.serialize()])
    assert BLS.verify_batch_bytes(*wire) == [True, True]
    assert BLS.verify_batch_bytes(*wire, strict=True) == [True, False]
