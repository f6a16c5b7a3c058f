"""Subgroup membership without a GPU: the g1_subgroup / g2_subgroup programs on the host simulation of the VM against
the definition of membership, and the endomorphism identities they rest on against the oracle."""
import numpy as np
import pytest

import bls_oracle as O
import hostsim
import subgroup_corpus as SC

from bls_b200.programs import curve, hashg2, registry


def test_endomorphism_identities_against_oracle():
    """phi(x, y) = (BETA x, y) is [-x^2] on G1 and psi is [x] on G2 (x = -X_ABS); the other cube root of unity gives
    x^2 - 1, and points outside the subgroups fail the identities"""
    g1 = O.aff_mul(0x1234567, (O.G1[0], O.G1[1], False))
    x2 = O.aff_mul(O.X_ABS * O.X_ABS, g1)
    assert (curve.BETA * g1[0] % O.Q, g1[1], False) == O.aff_neg(x2)
    beta2 = curve.BETA * curve.BETA % O.Q
    assert (beta2 * g1[0] % O.Q, g1[1], False) == O.aff_mul(O.X_ABS * O.X_ABS - 1, g1)
    p = (4, O.g1_y_for_x(4)[0], False)
    assert (curve.BETA * p[0] % O.Q, p[1], False) != O.aff_neg(O.aff_mul(O.X_ABS * O.X_ABS, p))
    g2 = O.hash_to_g2(b"identity")
    assert O.psi(g2) == O.aff_neg(O.aff_mul(O.X_ABS, g2))
    # the program's psi constants are the oracle's psi
    x, y = g2[0], g2[1]
    conj = lambda a: (a[0], -a[1] % O.Q)                        # noqa: E731
    assert (O.f2_mul(conj(x), hashg2.PSI_CX), O.f2_mul(conj(y), hashg2.PSI_CY), False) == O.psi(g2)
    for t in ((3, 5), (7, 11), (123, 456)):
        p = O.sw_encode_g2(t)
        assert O.psi(p) != O.aff_neg(O.aff_mul(O.X_ABS, p)) and not O.aff_mul(O.N, p)[2]


@pytest.mark.parametrize("ctas", [1, 4])
@pytest.mark.parametrize("g2", [False, True])
def test_subgroup_programs_on_host_simulation(g2, ctas):
    pts = SC.g2_corpus() if g2 else SC.g1_corpus()
    want = [SC.is_member(p) for p in pts]
    assert any(want) and not all(want)
    ser = SC.g2_bytes if g2 else SC.g1_bytes
    w = 192 if g2 else 96
    buf = np.frombuffer(b"".join(ser(p) for p in pts), dtype=np.uint8).copy()
    ok = np.full(len(pts), 9, dtype=np.uint8)
    n_slots, n_tmem = registry.SHAPES[ctas]
    asm = curve.build_subgroup_check(g2)().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    hostsim.run(asm, {0: buf, 1: ok}, {0: w, 1: 1}, len(pts), n_blocks=3, nt=8)
    assert [bool(f) for f in ok] == want
    assert set(ok.tolist()) <= {0, 1}


def _ladder_reaches_p(order):
    """True iff the |x| ladder on a point of this order adds P to an accumulator equal to P"""
    k = 1
    for bit in bin(O.X_ABS)[3:]:
        k = 2 * k % order
        if bit == "1":
            if k == 1 % order:
                return True
            k = (k + 1) % order
    return False


def _order11_g1():
    h1 = (O.X_ABS + 1) ** 2 // 3
    p = (4, O.g1_y_for_x(4)[0], False)
    t = O.aff_mul(h1 // 121 * O.N, p)                    # the 11-part of E(Fq) has exponent 11
    assert not t[2] and O.aff_mul(11, t)[2]
    return t


@pytest.mark.parametrize("g2", [False, True])
def test_subgroup_ladder_exact_on_small_order_points(g2):
    """Curve.subgroup_ladder ([x^2] P on G1, [|x|] P on G2) against the oracle's scalar multiplication.  On E(Fq) the
    ladder adds P to an accumulator equal to P for the points of order 3 and 11, which only the complete additions
    get right; E'(Fq2) has no point of small order for which that happens"""
    from bls_b200.vm.builder import Program
    if g2:
        pts = SC.g2_corpus()[:-2]                          # on the curve
        k = O.X_ABS
    else:
        assert _ladder_reaches_p(3) and _ladder_reaches_p(11)
        pts = SC.g1_corpus()[:-2] + [_order11_g1(), O.aff_neg(_order11_g1())]
        k = O.X_ABS * O.X_ABS
    prog = Program("ladder_test")
    prog.begin_body()
    c = curve.Curve(prog, g2)
    x, y, inf = c.load_affine(0)
    c.store_affine(1, 0, c.to_affine(c.subgroup_ladder(x, y, inf)))
    w = 192 if g2 else 96
    ser = SC.g2_bytes if g2 else SC.g1_bytes
    buf = np.frombuffer(b"".join(ser(p) for p in pts), dtype=np.uint8).copy()
    out = np.zeros(w * len(pts), dtype=np.uint8)
    hostsim.run(prog.assemble(6, n_cold=4096, n_tmem=7), {0: buf, 1: out}, {0: w, 1: w}, len(pts), n_blocks=2, nt=8)
    raw = out.tobytes()
    for i, p in enumerate(pts):
        assert raw[w * i:w * (i + 1)] == ser(O.aff_mul(k, p)), i


@pytest.mark.parametrize("ctas", [1, 4])
def test_key_validate_program_on_reduced_coordinates(ctas):
    """g1_keyvalidate = member and not infinity; g1_subgroup = member.  Both read coordinates mod q, so q || 0,
    0 || q and q || q are infinity (a member, not a valid key) and the generator with x + q is a valid key"""
    raws = [SC.g1_bytes(p) for p in SC.g1_corpus()] + SC.g1_noncanonical_encodings()
    pts = [SC.g1_reduced(r) for r in raws]
    member = [SC.is_member(p) for p in pts]
    n_slots, n_tmem = registry.SHAPES[ctas]
    for key, want in ((False, member), (True, [m and not p[2] for m, p in zip(member, pts)])):
        buf = np.frombuffer(b"".join(raws), dtype=np.uint8).copy()
        ok = np.full(len(raws), 9, dtype=np.uint8)
        asm = curve.build_subgroup_check(False, key=key)().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
        hostsim.run(asm, {0: buf, 1: ok}, {0: 96, 1: 1}, len(raws), n_blocks=2, nt=8)
        assert [bool(f) for f in ok] == want, key
    assert want[-4:] == [False, False, False, True] and member[-4:] == [True] * 4


def test_subgroup_program_cost():
    """two |x| ladders over Fq for G1, one over Fq2 for G2: a few thousand products, about a tenth of verify_full"""
    g1 = registry.executed_mults("g1_subgroup")
    g2 = registry.executed_mults("g2_subgroup")
    assert g1 < 2500 and g2 < 2500
    assert g2 < registry.executed_mults("verify_full") / 8
