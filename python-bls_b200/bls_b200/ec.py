"""Curve points of the scheme layer, backed by the GPU engine.

The reference keeps points as Python objects over Fq/Fq2 ints and does every operation in
the interpreter (bls_py/ec.py:18-391).  Here a point is its canonical affine byte string
(96 bytes for G1, 192 for G2, zero bytes for infinity -- the reference's own
(0, 0, infinity=True) affine form, fields_t.py:609-622) and every operator is one call into
the batched C ABI.  Serialisation is byte-identical (ec.py:94-111)."""
import numpy as np

from . import engine
from .programs.curve import G1_GEN
from .programs.hashg2 import G2_GEN
from .util import hash256

Q = int("1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f624"
        "1eabfffeb153ffffb9feffffffffaaab", 16)
N = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


class Point:
    """affine point on E(Fq) (g2=False) or on the twist E'(Fq2) (g2=True)"""
    __slots__ = ("raw", "g2", "_ser")

    def __init__(self, raw, g2):
        raw = bytes(raw)
        if len(raw) != (192 if g2 else 96):
            raise ValueError("bad point encoding length %d" % len(raw))
        self.raw = raw
        self.g2 = g2
        self._ser = None

    # -- reference-style accessors --------------------------------------------------------
    @property
    def infinity(self):
        return not any(self.raw)

    @property
    def x(self):
        c = [int.from_bytes(self.raw[i:i + 48], "big") for i in range(0, len(self.raw) // 2, 48)]
        return tuple(c) if self.g2 else c[0]

    @property
    def y(self):
        h = len(self.raw) // 2
        c = [int.from_bytes(self.raw[i:i + 48], "big") for i in range(h, 2 * h, 48)]
        return tuple(c) if self.g2 else c[0]

    def to_affine(self):
        return self if type(self) is AffinePoint else _retype(self, AffinePoint)

    def to_jacobian(self):
        return self if type(self) is JacobianPoint else _retype(self, JacobianPoint)

    # -- arithmetic (one GPU call each; use bls_b200.engine for batches) ----------------------
    def __add__(self, other):
        if other == 0 and not isinstance(other, Point):
            return self
        if not isinstance(other, Point) or other.g2 != self.g2:
            raise TypeError("cannot add %r" % type(other))
        return JacobianPoint(engine.point_add(self.raw, other.raw, self.g2).tobytes(), self.g2)

    __radd__ = __add__

    def negate(self):
        if self.infinity:
            return self
        h = len(self.raw) // 2
        y = [(-int.from_bytes(self.raw[i:i + 48], "big")) % Q for i in range(h, 2 * h, 48)]
        return type(self)(self.raw[:h] + b"".join(v.to_bytes(48, "big") for v in y), self.g2)

    def __neg__(self):
        return self.negate()

    def __sub__(self, other):
        return self + other.negate()

    def __mul__(self, k):
        k = int(k)
        if k < 0 or k >> 256:
            k %= N                      # valid for points of order n (every public object here)
        return JacobianPoint(engine.scalar_mul(self.raw, k.to_bytes(32, "big"), self.g2).tobytes(), self.g2)

    __rmul__ = __mul__

    def __eq__(self, other):
        return isinstance(other, Point) and self.g2 == other.g2 and self.raw == other.raw

    def __ne__(self, other):
        return not self.__eq__(other)

    def __hash__(self):
        return hash((self.g2, self.raw))

    def is_in_subgroup(self):
        """on the curve and in the prime-order subgroup G1 / G2 (infinity is); the reference has no such test.
        Batches: engine.subgroup_check"""
        return bool(engine.subgroup_check(self.raw, self.g2)[0])

    def serialize(self):
        """x with the 'y is the larger root' flag in the top bit (ec.py:94-111)"""
        if self._ser is None:
            self._ser = engine.compress(self.raw, self.g2).tobytes()
        return self._ser

    def __repr__(self):
        return "%s(%s)" % ("G2" if self.g2 else "G1", self.serialize().hex())


class AffinePoint(Point):
    """ec.py:18-112.  Same storage as every Point here -- the canonical affine bytes; the class only records which
    of the reference's two coordinate systems the caller asked for (to_affine / to_jacobian convert the class,
    arithmetic returns Jacobian points like the reference's operators)."""
    __slots__ = ()


class JacobianPoint(Point):
    """ec.py:115-188: the reference's Jacobian triple, here always normalised (z = 1) and stored as affine bytes"""
    __slots__ = ()

    @property
    def z(self):
        if self.infinity:
            return (0, 0) if self.g2 else 0
        return (1, 0) if self.g2 else 1


def _retype(p, cls):
    q = cls(p.raw, p.g2)
    q._ser = p._ser
    return q


class Fq12Point:
    """an affine point with Fq12 coordinates, as ec.untwist / ec.twist return it (ec.py:402-437)"""
    __slots__ = ("x", "y", "infinity")

    def __init__(self, x, y, infinity=False):
        self.x, self.y, self.infinity = x, y, infinity

    def __eq__(self, other):
        return isinstance(other, Fq12Point) and (self.x, self.y, self.infinity) == (other.x, other.y, other.infinity)

    def __hash__(self):
        return hash((self.x, self.y, self.infinity))


def untwist(point, ec=None):
    """ec.py:402-418: a point of the twist E'(Fq2) -> (x / w^2, y / w^3) on E(Fq12)"""
    from .fields import Fq12
    if isinstance(point, Fq12Point):          # fq12_untwist: divide the Fq12 coordinates by w^2, w^3
        w2, w3 = _w_powers()
        return Fq12Point(point.x / w2, point.y / w3, False)
    if not point.g2:
        raise Exception("point should be Fq2 or Fq12 elements")
    out = engine.g2_untwist(point.raw).tobytes()
    return Fq12Point(Fq12(out[:576]), Fq12(out[576:]), False)


def twist(point, ec=None):
    """ec.py:421-437: (x, y) -> (x w^2, y w^3) over Fq12"""
    from .fields import Fq12
    if isinstance(point, Fq12Point):
        raw = point.x.raw + point.y.raw
    else:                                     # an Fq2 point: its coordinates embedded at coefficient 0
        raw = point.raw[:96] + bytes(480) + point.raw[96:] + bytes(480)
    out = engine.fq12_twist(raw).tobytes()
    return Fq12Point(Fq12(out[:576]), Fq12(out[576:]), False)


def _w_powers():
    from .fields import Fq12
    w = Fq12(Q, (0,) * 6 + (1,) + (0,) * 5)
    w2 = w * w
    return w2, w2 * w


def psi(P, ec=None):
    """ec.py:440-444: twist(Frobenius(untwist(P))) on the twist's own coordinates"""
    return JacobianPoint(engine.g2_psi(P.raw).tobytes(), True).to_affine()


def sw_encode(t, ec=None, FE=None):
    """ec.py:449-507 for t in Fq2 (an Fq2 field object, a pair of ints or 96 bytes): the Shallue-van de Woestijne
    map onto the twist; t = 0 gives infinity.  (The Fq variant onto E(Fq) belongs to the G1 hash, which nothing on
    the signature path uses: SURVEY.md section 2 marks it out of scope.)"""
    raw = t.raw if hasattr(t, "raw") else (bytes(t) if isinstance(t, (bytes, bytearray)) else
                                            b"".join((int(c) % Q).to_bytes(48, "big") for c in t))
    if len(raw) != 96:
        raise ValueError("sw_encode takes an Fq2 element")
    return AffinePoint(engine.sw_encode_g2(raw).tobytes(), True)


def generator_Fq(ec=None):
    return AffinePoint(b"".join(c.to_bytes(48, "big") for c in G1_GEN), False)


def generator_Fq2(ec=None):
    return AffinePoint(b"".join(c.to_bytes(48, "big") for c in (G2_GEN[0] + G2_GEN[1])), True)


def infinity(g2):
    return Point(bytes(192 if g2 else 96), g2)


def _canonical_encoding(data, raw, g2):
    """the bytes serialize() gives back for the point `raw` decoded from `data` -- `data` itself with its two
    spare flag bits cleared -- when `data` is the canonical encoding; None (serialize() then asks the device)
    when it is not: an x coefficient >= q (the device reduces it on load, like Fq(Q, int)), or the sign flag on
    a point whose sign coordinate is zero (lex_gt_neg is False there, ec.py:94-101).  Keys and signatures
    compare, hash and sort by these bytes, so two encodings of one point must not yield two values."""
    masked = bytes([data[0] & 0x9f]) + data[1:]
    xs = [int.from_bytes(bytes([masked[0] & 0x1f]) + masked[1:48], "big")]
    if g2:
        xs.append(int.from_bytes(masked[48:96], "big"))
    if any(x >= Q for x in xs):
        return None
    sign_coord = raw[144:192] if g2 else raw[48:96]         # y.c1 for the twist, y for E(Fq)
    if (masked[0] & 0x80) and not any(sign_coord):
        return None
    return masked


def point_from_bytes(data, g2, check_subgroup=False):
    """PublicKey.from_bytes / Signature.from_bytes decoding (keys.py:29-40, signature.py:22-38);
    raises ValueError where the reference does, and with check_subgroup=True also for a point outside G1 / G2"""
    out, ok = engine.decompress(data, g2)
    if not ok[0]:
        raise ValueError("No y for point x")
    if check_subgroup and not engine.subgroup_check(out, g2)[0]:
        raise ValueError("point is not in the prime-order subgroup")
    p = Point(out.tobytes(), g2)
    p._ser = _canonical_encoding(bytes(data), p.raw, g2)
    return p


def points_from_bytes(buffers, g2, check_subgroup=False):
    """many PublicKey.from_bytes / Signature.from_bytes decodings in ONE GPU call (row f2: the
    reference decodes, and later re-serialises, one key at a time).  The serialised form of each
    point is known at once -- the input with its two spare flag bits cleared (the reference masks
    them on input and never sets them on output) -- so sorting / hashing these points later costs
    no further GPU work.  Raises ValueError if any buffer does not decode, like the reference, and with
    check_subgroup=True also if any point is outside G1 / G2 (one more batched call)."""
    buffers = [bytes(b) for b in buffers]
    if not buffers:
        return []
    w = 192 if g2 else 96
    out, ok = engine.decompress(b"".join(buffers), g2)
    if not ok.all():
        raise ValueError("No y for point x (buffer %d)" % int(np.argmin(ok)))
    if check_subgroup:
        member = engine.subgroup_check(out, g2)
        if not member.all():
            raise ValueError("point is not in the prime-order subgroup (buffer %d)" % int(np.argmin(member)))
    raw = out.tobytes()
    pts = []
    for i, b in enumerate(buffers):
        p = Point(raw[w * i:w * (i + 1)], g2)
        p._ser = _canonical_encoding(b, p.raw, g2)
        pts.append(p)
    return pts


def serialize_many(points):
    """fill the serialisation caches of many points with one batched GPU call per group, so
    that the sorts, sets and dictionaries of the scheme layer (which compare keys by their
    serialised bytes, keys.py:57-64 in the reference) do no per-key GPU work"""
    for g2 in (False, True):
        todo = [p for p in points if p.g2 == g2 and p._ser is None]
        if len(todo) > 1:
            w = 96 if g2 else 48
            ser = engine.compress(b"".join(p.raw for p in todo), g2).tobytes()
            for i, p in enumerate(todo):
                p._ser = ser[w * i:w * (i + 1)]


def hash_to_point_prehashed_Fq2(h):
    """ec.py:528-550"""
    if not isinstance(h, (bytes, bytearray)):
        h = h.encode("utf-8")
    if len(h) != 32:
        raise ValueError("the batched hash-to-G2 takes 32-byte message hashes")
    return AffinePoint(engine.hash_to_g2(bytes(h)).tobytes(), True)


def hash_to_point_Fq2(m):
    """ec.py:553-555"""
    return hash_to_point_prehashed_Fq2(hash256(m))


def sum_points(points, g2):
    """sum of many points in one reduction on the GPU"""
    if not points:
        return infinity(g2)
    return Point(engine.point_sum(b"".join(p.raw for p in points), g2).tobytes(), g2)


def weighted_sum(points, scalars, g2):
    """sum_i k_i * P_i in one multi-scalar multiplication on the GPU.  `scalars`: ints, or
    already n x 32 big-endian bytes (e.g. straight from engine.hash_pks)."""
    if not points:
        return infinity(g2)
    if not isinstance(scalars, (bytes, bytearray, np.ndarray)):
        scalars = b"".join((int(k) % N).to_bytes(32, "big") for k in scalars)
    return Point(engine.msm(b"".join(p.raw for p in points), scalars, g2).tobytes(), g2)


def scalar_mul_many(points, scalars, g2):
    """[k_i * P_i] in one batched call"""
    if not points:
        return []
    w = 192 if g2 else 96
    # the same rule as Point.__mul__: scalars outside [0, 2^256) are reduced mod the group order
    sc = b"".join((int(k) % N if (int(k) < 0 or int(k) >> 256) else int(k)).to_bytes(32, "big") for k in scalars)
    out = engine.scalar_mul(b"".join(p.raw for p in points), sc, g2).tobytes()
    return [Point(out[w * i:w * (i + 1)], g2) for i in range(len(points))]
