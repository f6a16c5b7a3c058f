"""Points for the subgroup-membership tests: members and non-members of G1 / G2 with the expected flag taken from the
definition (on the curve and [n] P = infinity), computed by the oracle, never from the endomorphism identities."""
import bls_oracle as O
from conftest import load_golden

# cofactor of E'(Fq2) = #E'(Fq2) / n; 13^2 divides it
H2 = int("5d543a95414e7f1091d50792876a202cd91de4547085abaa68a205b2e5a7ddfa628f1cb4d9e82ef21537e293a6691ae1616ec6e7"
         "86f0c70cf1c38e31c7238e5", 16)
G1_SMALL = (0, 2, False)                 # order 3; all-zero 48-byte keys decode to it


def is_member(p):
    return O.on_curve(p) and O.aff_mul(O.N, p)[2]


def order13_point():
    """T = [h2 / 169 * n] sw_encode(7, 11): a point of order 13 on E'(Fq2)"""
    t = O.aff_mul(H2 // 169 * O.N, O.sw_encode_g2((7, 11)))
    assert not t[2] and O.aff_mul(13, t)[2]
    return t


def g1_bytes(p):
    return b"\0" * 96 if p[2] else p[0].to_bytes(48, "big") + p[1].to_bytes(48, "big")


def g2_bytes(p):
    if p[2]:
        return b"\0" * 192
    return b"".join(c.to_bytes(48, "big") for c in (p[0][0], p[0][1], p[1][0], p[1][1]))


def _bump_y(p):
    y = (p[1] + 1) % O.Q if isinstance(p[1], int) else ((p[1][0] + 1) % O.Q, p[1][1])
    return (p[0], y, False)


def g1_corpus():
    """-> list of affine G1 points (members, infinity, small order, off-curve)"""
    g = (O.G1[0], O.G1[1], False)
    sk = load_golden("sig_kat.json")
    pks = sorted({t["pk"] for t in sk["verify_table"]} | {k["pk"] for k in sk["keys"]})
    members = [g] + [O.aff_mul(k, g) for k in (2, 3, 0xdeadbeef, O.N - 1)]
    members += [O.g1_deserialize(bytes.fromhex(h)) for h in pks]
    pts = members + [(0, 0, True), G1_SMALL, O.aff_neg(G1_SMALL)]
    for x in (4, 5, 8):                   # small x: on the curve, not in G1
        pts.append((x, O.g1_y_for_x(x)[0], False))
    pts += [O.aff_add(m, G1_SMALL) for m in members[:3]]
    pts += [_bump_y(g), _bump_y(members[-1])]
    return pts


def g2_corpus():
    """-> list of affine G2 points (members, infinity, uncleared map outputs, order-13 components, off-curve)"""
    g = (O.G2[0], O.G2[1], False)
    sk = load_golden("sig_kat.json")
    sigs = sorted({t["sig"] for t in sk["verify_table"]} | {s["sig"] for s in sk["sign"]})
    members = [g] + [O.aff_mul(k, g) for k in (2, 0xdeadbeef)]
    members += [O.hash_to_g2(m) for m in (b"", b"abc", b"subgroup")]
    decoded = []
    for h in sigs:
        try:
            decoded.append(O.g2_deserialize(bytes.fromhex(h)))
        except ValueError:                # undecodable vectors of the table
            pass
    members += decoded
    t = order13_point()
    pts = members + [(O.F2_ZERO, O.F2_ZERO, True), t]
    pts += [O.sw_encode_g2(s) for s in ((3, 5), (7, 11), (123, 456))]
    pts += [O.aff_add(m, t) for m in members[:2] + decoded[:2]]
    pts += [_bump_y(g), _bump_y(members[-1])]
    return pts


def g1_noncanonical_encodings():
    """96-byte G1 encodings with a coordinate >= q: the three spellings of infinity besides zero bytes, and the
    generator with x + q.  Every affine input is read mod q, so these are infinity and a member"""
    q = O.Q.to_bytes(48, "big")
    z = bytes(48)
    g = (O.G1[0] + O.Q).to_bytes(48, "big") + O.G1[1].to_bytes(48, "big")
    return [q + z, z + q, q + q, g]


def g1_reduced(raw):
    """the affine point the device reads from 96 bytes: coordinates mod q, (0, 0) = infinity"""
    x, y = (int.from_bytes(raw[i:i + 48], "big") % O.Q for i in (0, 48))
    return (x, y, x == 0 and y == 0)
