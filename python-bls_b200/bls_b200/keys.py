"""PrivateKey / PublicKey / ExtendedPrivateKey / ExtendedPublicKey with the reference's
interface (bls_py/keys.py:17-316); curve work runs on the GPU."""
import secrets

from . import ec, engine
from .aggregation_info import AggregationInfo
from .util import GROUP_ORDER, hash256, hmac256


class PublicKey:
    PUBLIC_KEY_SIZE = 48

    def __init__(self, value):
        self.value = value                      # ec.Point on G1

    @staticmethod
    def from_bytes(buffer, check_subgroup=False):
        """check_subgroup=True: ValueError also for a point outside G1 (the reference accepts it)"""
        return PublicKey(ec.point_from_bytes(bytes(buffer), False, check_subgroup))

    @staticmethod
    def from_bytes_batch(buffers, check_subgroup=False):
        """many keys decoded in one GPU call; their serialised forms are cached"""
        return [PublicKey(p) for p in ec.points_from_bytes(buffers, False, check_subgroup)]

    @staticmethod
    def from_g1(g1_el):
        assert isinstance(g1_el, ec.Point) and not g1_el.g2
        return PublicKey(g1_el)

    def serialize(self):
        return self.value.serialize()

    def get_fingerprint(self):
        return int.from_bytes(hash256(self.serialize())[:4], "big")

    def size(self):
        return self.PUBLIC_KEY_SIZE

    def __eq__(self, other):
        return self.serialize() == other.serialize()

    def __hash__(self):
        return int.from_bytes(self.serialize(), "big")

    def __lt__(self, other):
        return self.serialize() < other.serialize()

    def __repr__(self):
        return "PublicKey(%s)" % self.serialize().hex()

    __str__ = __repr__


class PrivateKey:
    PRIVATE_KEY_SIZE = 32

    def __init__(self, value):
        self.value = int(value)

    @staticmethod
    def from_bytes(buffer):
        return PrivateKey(int.from_bytes(buffer, "big"))

    @staticmethod
    def from_seed(seed):
        return PrivateKey(int.from_bytes(hmac256(seed, b"BLS private key seed"), "big") % GROUP_ORDER)

    @staticmethod
    def new_threshold(T, N, rng=None):
        """one player's dealing of a T-of-N Joint-Feldman scheme (keys.py:93-117): a random
        degree T-1 polynomial, commitments g1 * coefficient (one batched scalar multiplication)
        and the fragments P(1..N).  `rng` (random.Random-like) makes the dealing reproducible."""
        assert 1 <= T <= N
        draw = (lambda: rng.randrange(1, GROUP_ORDER)) if rng is not None else \
            (lambda: 1 + secrets.randbelow(GROUP_ORDER - 1))
        poly = [draw() for _ in range(T)]
        commitments = ec.scalar_mul_many([ec.generator_Fq()] * T, poly, False)
        fragments = [sum(c * pow(x, i, GROUP_ORDER) for i, c in enumerate(poly)) % GROUP_ORDER
                     for x in range(1, N + 1)]
        return PrivateKey(poly[0]), commitments, fragments

    def get_public_key(self):
        return PublicKey(ec.generator_Fq() * self.value)

    def sign_threshold(self, m, player, players):
        """this player's signature share, already weighted by its Lagrange coefficient
        (keys.py:137-147)"""
        from .signature import Signature
        from .threshold import Threshold
        assert player in players
        lamb = Threshold.lagrange_coeffs_at_zero(players)[players.index(player)]
        return Signature.from_g2(ec.hash_to_point_Fq2(m) * (self.value * lamb % GROUP_ORDER))

    def sign(self, m):
        return self.sign_prehashed(hash256(m))

    def sign_prehashed(self, h):
        from .signature import Signature
        r = ec.hash_to_point_prehashed_Fq2(h)
        return Signature.from_g2(r * self.value, AggregationInfo.from_msg_hash(self.get_public_key(), h))

    @staticmethod
    def get_public_key_batch(keys):
        """[k.get_public_key() for k in keys] in one device pass (and one more that fills their serialisations, which
        the scheme layer's dictionaries and sorts use)"""
        keys = list(keys)
        if not keys:
            return []
        raw = engine.public_keys([k.value for k in keys]).tobytes()
        pts = [ec.JacobianPoint(raw[96 * i:96 * (i + 1)], False) for i in range(len(keys))]
        ec.serialize_many(pts)
        return [PublicKey(p) for p in pts]

    @staticmethod
    def sign_batch(keys, messages):
        """[k.sign(m) for k, m in zip(keys, messages)]: see sign_prehashed_batch"""
        return PrivateKey.sign_prehashed_batch(keys, [hash256(m) for m in messages])

    @staticmethod
    def sign_prehashed_batch(keys, hashes):
        """[k.sign_prehashed(h) for k, h in zip(keys, hashes)] with one device pass for the signatures and one for the
        public keys of their AggregationInfo, instead of three GPU calls per signature"""
        from .signature import Signature
        keys, hashes = list(keys), [bytes(h) for h in hashes]
        if len(keys) != len(hashes):
            raise ValueError("%d keys for %d message hashes" % (len(keys), len(hashes)))
        if not keys:
            return []
        raw = engine.sign_batch([k.value for k in keys], b"".join(hashes)).tobytes()
        pks = PrivateKey.get_public_key_batch(keys)
        return [Signature.from_g2(ec.JacobianPoint(raw[192 * i:192 * (i + 1)], True),
                                  AggregationInfo.from_msg_hash(pk, h)) for i, (pk, h) in enumerate(zip(pks, hashes))]

    def serialize(self):
        return self.value.to_bytes(self.PRIVATE_KEY_SIZE, "big")

    def size(self):
        return self.PRIVATE_KEY_SIZE

    def __lt__(self, other):
        return self.value < other.value

    def __eq__(self, other):
        return self.value == other.value

    def __hash__(self):
        return self.value

    def __repr__(self):
        return "PrivateKey(%s)" % hex(self.value)

    __str__ = __repr__


def _hd_halves(data, chain_code):
    return hmac256(data + bytes([0]), chain_code), hmac256(data + bytes([1]), chain_code)


HARDENED = 1 << 31                      # child numbers from here up commit to the secret key


class _ExtendedKey:
    """what the two halves of the BIP32-style hierarchy share (keys.py:167-316): a 45-byte header
    -- version (4), depth (1), parent fingerprint (4), child number (4), chain code (32) -- in
    front of the serialised key, and value semantics on the serialisation"""

    def _set_header(self, version, depth, parent_fingerprint, child_number, chain_code):
        self.version, self.depth = version, depth
        self.parent_fingerprint, self.child_number = parent_fingerprint, child_number
        self.chain_code = bytes(chain_code)

    def _header(self):
        return b"".join((self.version.to_bytes(4, "big"), bytes([self.depth]),
                         self.parent_fingerprint.to_bytes(4, "big"), self.child_number.to_bytes(4, "big"),
                         self.chain_code))

    def _check_depth(self):
        if self.depth >= 255:
            raise Exception("Cannot go further than 255 levels")

    def _child_header(self, i, tweak_data):
        """-> (left HMAC half as an int mod n, header fields of child i)"""
        left, right = _hd_halves(tweak_data + i.to_bytes(4, "big"), self.chain_code)
        fields = (self.version, self.depth + 1, self.get_public_key().get_fingerprint(), i, right)
        return int.from_bytes(left, "big") % GROUP_ORDER, fields

    def size(self):
        return len(self.serialize())

    def __eq__(self, other):
        return self.serialize() == other.serialize()

    def __hash__(self):
        return int.from_bytes(self.serialize(), "big")


class ExtendedPrivateKey(_ExtendedKey):
    """secret half: child secret = parent secret + left HMAC half (mod n)"""
    version = 1
    EXTENDED_PRIVATE_KEY_SIZE = 77

    def __init__(self, version, depth, parent_fingerprint, child_number, chain_code, private_key):
        self._set_header(version, depth, parent_fingerprint, child_number, chain_code)
        self.private_key = private_key

    @staticmethod
    def from_seed(seed):
        left, right = _hd_halves(bytes(seed), b"BLS HD seed")
        root = PrivateKey(int.from_bytes(left, "big") % GROUP_ORDER)
        return ExtendedPrivateKey(ExtendedPrivateKey.version, 0, 0, 0, right, root)

    def get_private_key(self):
        return self.private_key

    def get_public_key(self):
        return self.private_key.get_public_key()

    def private_child(self, i):
        self._check_depth()
        committed = self.private_key.serialize() if i >= HARDENED else self.get_public_key().serialize()
        tweak, fields = self._child_header(i, committed)
        child = PrivateKey((tweak + self.private_key.value) % GROUP_ORDER)
        return ExtendedPrivateKey(ExtendedPrivateKey.version, *fields[1:], child)

    def public_child(self, i):
        return self.private_child(i).get_extended_public_key()

    def get_extended_public_key(self):
        return ExtendedPublicKey.from_bytes(self._header() + self.get_public_key().serialize())

    def serialize(self):
        return self._header() + self.private_key.serialize()


class ExtendedPublicKey(_ExtendedKey):
    """public half: non-hardened children only, child key = parent key + g1 * left HMAC half (one
    scalar multiplication and one addition on the GPU)"""
    EXTENDED_PUBLIC_KEY_SIZE = 93

    def __init__(self, version, depth, parent_fingerprint, child_number, chain_code, public_key):
        self._set_header(version, depth, parent_fingerprint, child_number, chain_code)
        self.public_key = public_key

    @staticmethod
    def from_bytes(serialized):
        raw = bytes(serialized)
        words = [int.from_bytes(raw[a:b], "big") for a, b in ((0, 4), (4, 5), (5, 9), (9, 13))]
        return ExtendedPublicKey(*words, raw[13:45], PublicKey.from_bytes(raw[45:]))

    def get_public_key(self):
        return self.public_key

    def public_child(self, i):
        self._check_depth()
        if i >= HARDENED:
            raise Exception("Cannot derive hardened children from public key")
        tweak, fields = self._child_header(i, self.public_key.serialize())
        child = PublicKey.from_g1(ec.generator_Fq() * tweak + self.public_key.value)
        return ExtendedPublicKey(*fields, child)

    def serialize(self):
        return self._header() + self.public_key.serialize()
