"""The BLS scheme entry points of the reference (bls_py/bls.py:11-249) over the GPU engine.

Host side: grouping by message, collision detection, sorting, aggregation exponents (dict /
set / SHA-256 work, identical in behaviour to the reference).  Device side, one batched
call each: scalar multiplications by the exponents, point sums, hash-to-G2 of all messages,
the Miller loops and the single final exponentiation."""
from . import ec, engine
from .aggregation_info import AggregationInfo
from .keys import PrivateKey, PublicKey
from .signature import Signature
from .util import GROUP_ORDER, hash_pks, hash_pks_bytes


class BLS:
    @staticmethod
    def aggregate_sigs_simple(signatures):
        """plain sum (bls.py:13-26); NOT secure against rogue keys on equal messages"""
        return Signature.from_g2(ec.sum_points([s.value for s in signatures], True))

    @staticmethod
    def aggregate_sigs_secure(signatures, public_keys, message_hashes):
        """sum of T_i * sig_i in (message hash, pk) order (bls.py:29-56)"""
        if not (len(signatures) == len(public_keys) == len(message_hashes)):
            raise Exception("Invalid number of keys")
        ec.serialize_many([pk.value for pk in public_keys] + [s.value for s in signatures])
        order = sorted(range(len(signatures)), key=lambda i: (message_hashes[i], public_keys[i], signatures[i]))
        ts = hash_pks_bytes(len(public_keys), public_keys)
        return Signature.from_g2(ec.weighted_sum([signatures[i].value for i in order], ts, True))

    @staticmethod
    def aggregate_sigs(signatures):
        """simple aggregation for groups with disjoint messages, secure (exponentiated) for the
        groups that share one (bls.py:59-151)"""
        ec.serialize_many([pk.value for sig in signatures if sig.aggregation_info is not None
                           for pk in sig.aggregation_info.public_keys])
        infos = []
        for sig in signatures:
            if sig.aggregation_info is None or sig.aggregation_info.empty():
                raise Exception("Each signature must have a valid aggregation info")
            infos.append(sig.aggregation_info)
        seen, colliding = set(), set()
        for info in infos:
            local = set(info.message_hashes)
            colliding |= seen & local
            seen |= local
        if not colliding:
            final = BLS.aggregate_sigs_simple(signatures)
            final.set_aggregation_info(AggregationInfo.merge_infos(infos))
            return final
        hit = [s for s in signatures if any(m in colliding for m in s.aggregation_info.message_hashes)]
        rest = [s for s in signatures if not any(m in colliding for m in s.aggregation_info.message_hashes)]
        hit.sort(key=lambda s: s.aggregation_info)
        keys = sorted((mh, pk) for s in hit
                      for mh, pk in zip(s.aggregation_info.message_hashes, s.aggregation_info.public_keys))
        ts = hash_pks_bytes(len(hit), [pk for _, pk in keys])
        secure_part = ec.weighted_sum([s.value for s in hit], ts, True)
        final = Signature.from_g2(ec.sum_points([secure_part] + [s.value for s in rest], True))
        final.set_aggregation_info(AggregationInfo.merge_infos(infos))
        return final

    @staticmethod
    def verify(signature, strict=False):
        """bls.py:154-201: group keys by message, raise each to its exponent from the
        aggregation tree, one multi-pairing against the hashed messages.  strict=True: False as well when the
        signature is outside G2 or a public key is outside G1 or is infinity (the reference accepts these)"""
        info = signature.aggregation_info
        ec.serialize_many([pk.value for pk in info.public_keys])
        groups = {}
        for mh, pk in zip(info.message_hashes, info.public_keys):
            groups.setdefault(mh, []).append(pk)
        if not groups:
            raise IndexError("signature has no aggregation info entries")
        if strict:
            keys = list(set(info.public_keys))
            if not signature.value.is_in_subgroup():
                return False
            if not engine.key_validate(b"".join(pk.value.raw for pk in keys)).all():
                return False
        flat_pts, flat_exp, spans = [], [], []
        for mh, pks in groups.items():
            uniq = list(set(pks))
            start = len(flat_pts)
            for pk in uniq:
                if (mh, pk) not in info.tree:
                    return False
                flat_pts.append(pk.value)
                flat_exp.append(info.tree[(mh, pk)])
            spans.append((mh, start, len(flat_pts)))
        # pk^exponent for every (message, key) pair in one call; unit exponents pass through
        idx = [i for i, e in enumerate(flat_exp) if e != 1]
        if idx:
            powered = ec.scalar_mul_many([flat_pts[i] for i in idx], [flat_exp[i] for i in idx], False)
            for i, p in zip(idx, powered):
                flat_pts[i] = p
        pk_sums = []
        for mh, a, b in spans:
            pk_sums.append(flat_pts[a] if b - a == 1 else ec.sum_points(flat_pts[a:b], False))
        return engine.aggregate_verify(signature.value.raw, b"".join(p.raw for p in pk_sums),
                                       b"".join(mh for mh, _, _ in spans))

    @staticmethod
    def verify_batch(public_keys, message_hashes, signatures, strict=False):
        """n independent single-message verifications in one GPU pass -> list of bool
        (the data-parallel form of calling BLS.verify n times).  strict=True: False as well for a key outside G1,
        the infinity key or a signature outside G2"""
        res = engine.verify_batch(b"".join(pk.value.raw for pk in public_keys), b"".join(message_hashes),
                                  b"".join(s.value.raw for s in signatures), strict)
        return [bool(r) for r in res]

    @staticmethod
    def verify_batch_bytes(public_key_bytes, message_hashes, signature_bytes, strict=False):
        """the same from serialised keys (48 B) and signatures (96 B): PublicKey.from_bytes /
        Signature.from_bytes run on the GPU too; where the reference would raise ValueError while
        decoding, the result is False.  strict: as in verify_batch"""
        res = engine.verify_batch_wire(b"".join(public_key_bytes), b"".join(message_hashes), b"".join(signature_bytes),
                                       strict)
        return [bool(r) for r in res]

    @staticmethod
    def aggregate_pub_keys(public_keys, secure):
        """bls.py:204-223 (sorts its argument in place, like the reference)"""
        if len(public_keys) < 1:
            raise Exception("Invalid number of keys")
        ec.serialize_many([pk.value for pk in public_keys])
        public_keys.sort()
        pts = [pk.value for pk in public_keys]
        if secure:
            return PublicKey.from_g1(ec.weighted_sum(pts, hash_pks_bytes(len(public_keys), public_keys), False))
        return PublicKey.from_g1(ec.sum_points(pts, False))

    @staticmethod
    def aggregate_priv_keys(private_keys, public_keys, secure):
        """bls.py:226-249 (scalar arithmetic mod n on the host)"""
        if not secure:
            return PrivateKey(sum(sk.value for sk in private_keys) % GROUP_ORDER)
        if not public_keys:
            raise Exception("Must include public keys in secure aggregation")
        if len(private_keys) != len(public_keys):
            raise Exception("Invalid number of keys")
        ec.serialize_many([pk.value for pk in public_keys])
        pairs = sorted(zip(public_keys, private_keys), key=lambda t: (t[0], t[1]))
        ts = hash_pks(len(private_keys), public_keys)
        return PrivateKey(sum(sk.value * t for (_, sk), t in zip(pairs, ts)) % GROUP_ORDER)
