"""Ate pairing on BLS12-381 as VM programs.

What the reference computes (bls_py/fields_t.py:1091-1128, bls_py/pairing.py:51-92):
    e(P, Q) = f_{|x|,Q}(P) ^ ((q^12 - 1) / n)
with |x| = 0xd201000000010000 and NO conjugation for the negative curve parameter.  The
reference walks an affine R with dense Fq12 line values (one Fq12 inversion per line) and
raises to the 1268-bit exponent bit by bit.  Only the value AFTER the final exponentiation
is canonical, so this implementation is free to use

  * homogeneous projective R, denominator-free sparse lines scaled by w^3 and by Fq2
    factors (all killed by the final exponentiation, see DESIGN.md),
  * the exact hard-part decomposition
        (q^4 - q^2 + 1)/n = ((a+1)^2 / 3) (q - a) (a^2 + q^2 - 1) + 1,   a = |x|,
    i.e. five 64-bit exponentiations instead of one 1268-bit one.
"""
from ..vm.builder import Program, Q
from .tower import F6, F12, CompressedCyc, decompress_many, f12_one, fp_inverter

X_ABS = 0xd201000000010000
X_BITS = bin(X_ABS)[3:]                     # below the leading one, MSB first
Y_EXP = (X_ABS + 1) // 3                    # 0x460055555555aaab
assert 3 * Y_EXP == X_ABS + 1
N_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
assert (Q ** 4 - Q ** 2 + 1) // N_ORDER == Y_EXP * (X_ABS + 1) * (Q - X_ABS) * (X_ABS ** 2 + Q ** 2 - 1) + 1
assert 3 * ((Q ** 4 - Q ** 2 + 1) // N_ORDER) == (X_ABS + 1) ** 2 * (Q - X_ABS) * (X_ABS ** 2 + Q ** 2 - 1) + 3
assert N_ORDER % 3 != 0

BUF_P, BUF_Q, BUF_OUT = 0, 1, 2


def _mul12_xi(prog, c):
    """12 * xi * c  (3 b' with b' = 4 xi)"""
    t = c.mul_xi()
    t4 = t.dbl().dbl()
    return t4.dbl() + t4


def double_step(prog, r, xp, yp):
    """R <- 2R on E'(Fq2) in homogeneous projective coordinates; returns the tangent
    line at (the old) R evaluated at P as sparse coefficients (l0, l1, l4)."""
    x, y, z = r
    b = y.sqr()
    c = z.sqr()
    e = _mul12_xi(prog, c)              # 3 b' Z^2
    f = e.dbl() + e                     # 9 b' Z^2
    h = (y + z).sqr() - b - c           # 2 Y Z as (Y + Z)^2 - Y^2 - Z^2: a squaring (2 M) instead of a product (3 M)
    xx = x.sqr()
    l0 = b - e                          # Y^2 - 3 b' Z^2
    l1 = -((xx.dbl() + xx) * xp)        # -3 X^2 xP
    l4 = h * yp                         # 2 Y Z yP
    x3 = ((x * y) * (b - f)).dbl()      # 2 X Y (Y^2 - 9 b' Z^2)
    e2 = e.sqr()
    e2_4 = e2.dbl().dbl()
    y3 = (b + f).sqr() - (e2_4.dbl() + e2_4)   # (B + F)^2 - 12 E^2
    z3 = (b * h).dbl().dbl()            # 8 Y^3 Z
    return (x3, y3, z3), (l0, l1, l4)


def add_step(prog, r, q, xp, yp):
    """R <- R + Q (Q affine); returns the chord line through R and Q at P."""
    x, y, z = r
    xq, yq = q
    theta = y - yq * z
    lam = x - xq * z
    l0 = theta * xq - lam * yq
    l1 = -(theta * xp)
    l4 = lam * yp
    c = theta.sqr()
    d = lam.sqr()
    e = lam * d
    f = z * c
    g = x * d
    h = e + f - g.dbl()
    x3 = lam * h
    y3 = theta * (g - h) - e * y
    z3 = z * e
    return (x3, y3, z3), (l0, l1, l4)


def add_step_proj(prog, r, q, xp, yp):
    """R <- R + Q with Q = (Xq, Yq, Zq) homogeneous projective: the affine-Q formulas applied to
    (X Zq, Y Zq, Z Zq) and theta' = Y Zq - Yq Z, lam' = X Zq - Xq Z; the line is the affine one
    times Zq^2, an Fq2 factor the final exponentiation removes."""
    x, y, z = r
    xq, yq, zq = q
    xs, ys, zs = x * zq, y * zq, z * zq
    theta = ys - yq * z
    lam = xs - xq * z
    l0 = theta * xq - lam * yq
    l1 = -((theta * zq) * xp)
    l4 = (lam * zq) * yp
    c = theta.sqr()
    d = lam.sqr()
    e = lam * d
    f = zs * c
    g = xs * d
    h = e + f - g.dbl()
    x3 = lam * h
    y3 = theta * (g - h) - e * ys
    z3 = zs * e
    return (x3, y3, z3), (l0, l1, l4)


def miller_loop(prog, xp, yp, xq, yq):
    """f_{|x|,Q}(P) up to factors that the final exponentiation removes."""
    one = prog.const2((1, 0))
    r = (xq, yq, one)
    f = None
    for bit in X_BITS:
        r, (l0, l1, l4) = double_step(prog, r, xp, yp)
        if f is None:
            zero = prog.const2((0, 0))
            f = F12(F6(l0, l1, zero), F6(zero, l4, zero))
            if bit == "1":
                r, (l0, l1, l4) = add_step(prog, r, (xq, yq), xp, yp)
                f = f.mul_by_014(l0, l1, l4)
            continue
        f = f.sqr_x2()                                  # 2 f^2: the factor is an Fq constant
        if bit == "1":
            # tangent and chord of the same step are multiplied with each other first (23 instead of 26 products)
            r, chord = add_step(prog, r, (xq, yq), xp, yp)
            f = f.mul_by_014_pair((l0, l1, l4), chord)
        else:
            f = f.mul_by_014(l0, l1, l4)
    return f


def miller_loop_multi(prog, pairs):
    """product of Miller loops sharing the squarings of f.  pairs: list of
    (xp, yp, xq, yq, inf) with inf a flag (or None): a pair flagged infinite contributes the
    identity line (1, 0, 0) at every step, i.e. the factor 1 -- what the reference's blind
    Miller loop on (0, 0) amounts to after the final exponentiation (SURVEY.md 9.8)."""
    one = prog.const2((1, 0))
    zero = prog.const2((0, 0))

    def guard(line, inf):
        if inf is None:
            return line
        return (prog.sel2(inf, one, line[0]), prog.sel2(inf, zero, line[1]), prog.sel2(inf, zero, line[2]))

    # a pair's Q is affine (xq, yq Fq2 values) or, when xq is a 3-tuple, homogeneous projective
    def start(xq, yq):
        return tuple(xq) if isinstance(xq, tuple) else (xq, yq, one)

    rs = [start(xq, yq) for (_, _, xq, yq, _) in pairs]
    f = None

    def absorb(f, lines):
        """f times all the lines of one step; two lines at a time are multiplied with each other first"""
        k = 0
        if f is None:
            l0, l1, l4 = lines[0]
            f = F12(F6(l0, l1, zero), F6(zero, l4, zero))
            k = 1
        while k + 1 < len(lines):
            f = f.mul_by_014_pair(lines[k], lines[k + 1])
            k += 2
        if k < len(lines):
            f = f.mul_by_014(*lines[k])
        return f

    for bit in X_BITS:
        if f is not None:
            f = f.sqr_x2()                              # 2 f^2: Fq factors die in the final exponentiation
        lines = []
        for k, (xp, yp, xq, yq, inf) in enumerate(pairs):
            rs[k], line = double_step(prog, rs[k], xp, yp)
            lines.append(guard(line, inf))
        f = absorb(f, lines)
        if bit == "1":
            lines = []
            for k, (xp, yp, xq, yq, inf) in enumerate(pairs):
                if isinstance(xq, tuple):
                    rs[k], line = add_step_proj(prog, rs[k], xq, xp, yp)
                else:
                    rs[k], line = add_step(prog, rs[k], (xq, yq), xp, yp)
                lines.append(guard(line, inf))
            f = absorb(f, lines)
    return f


def _pow_bits(f, e, sqr):
    """f^e, MSB-first square and multiply"""
    acc = f
    for bit in bin(e)[3:]:
        acc = sqr(acc)
        if bit == "1":
            acc = acc * f
    return acc


X_TOP_CUT = 57                      # |x| = (0b1101001 << 57) + 2^48 + 2^16
assert ((X_ABS >> X_TOP_CUT) << X_TOP_CUT) + (1 << 48) + (1 << 16) == X_ABS


def _pow_x_compressed(prog, m, fp_inv):
    """m^|x| for m in the cyclotomic subgroup: |x| = 2^63 + 2^62 + 2^60 + 2^57 + 2^48 + 2^16.
    ONE chain of 57 squarings of m runs in Karabina's compressed form (12 M per
    squaring instead of 18 M); its members 2^16, 2^48 and 2^57 are decompressed together (one shared
    inversion = one INV1); the four top bits, which lie within six squarings of each other, are
    finished from the 2^57 member by square-and-multiply on Granger-Scott squarings (exponent
    0b1101001) -- cheaper than three more snapshots, and 12 instead of 24 values stay live through
    the chain.  About 1,190 M instead of 1,404 M for plain square-and-multiply (63 squarings at 18 M
    + 5 products)."""
    low = [i for i in range(X_TOP_CUT + 1) if (X_ABS >> i) & 1]
    assert low[0] > 0 and low[-1] == X_TOP_CUT
    c = CompressedCyc.of(m)
    snaps = []
    for i in range(1, X_TOP_CUT + 1):
        c = c.sqr()
        if i in low:
            snaps.append(c)
    fs = decompress_many(prog, snaps, fp_inv)
    acc = _pow_bits(fs[-1], X_ABS >> X_TOP_CUT, lambda x: x.cyclotomic_sqr())
    for f in fs[:-1]:
        acc = acc * f
    return acc


class _Pow:
    """a power m^e of a fixed base, carrying its exponent so that chains are self-checking"""
    __slots__ = ("v", "e", "sqr")

    def __init__(self, v, e, sqr):
        self.v, self.e, self.sqr = v, e, sqr

    def sq(self, n=1):
        v = self.v
        for _ in range(n):
            v = self.sqr(v)
        return _Pow(v, self.e << n, self.sqr)

    def __mul__(self, o):
        return _Pow(self.v * o.v, self.e + o.e, self.sqr)


def _pow_y(m, sqr):
    """m^y, y = (|x| + 1) / 3 = 0x46_00_55_55_55_55_aa_ab, byte by byte with the three byte values
    0x55, 0xaa = 2 * 0x55 and 0xab = 0xaa + 1 precomputed: 67 cyclotomic squarings (18 M) and 11
    multiplications (54 M) = 1,800 M.  Plain square-and-multiply is 62 + 27 (2,574 M); building
    0x5555 and 0x55555555 by repeated squaring first, as an earlier version did, 96 + 9 (2,214 M)."""
    m1 = _Pow(m, 1, sqr)
    m2 = m1.sq()
    m4 = m2.sq()
    x46 = m4.sq(4) * (m4 * m2)                 # 0x40 + 0x6
    x5 = m4 * m1                               # 0x5
    x55 = x5.sq(4) * x5                        # 0x55
    r = x46.sq(16) * x55                       # 0x46_00_55
    for _ in range(3):
        r = r.sq(8) * x55                      # ..._55_55_55
    xaa = x55.sq()
    r = r.sq(8) * xaa
    r = r.sq(8) * (xaa * m1)                   # ..._aa_ab
    assert r.e == Y_EXP
    return r.v


def final_exponentiation(prog, f, cyclotomic=True, cubed=False):
    """f^((q^12-1)/n) with the exact exponent (reference: fields_t.py:1124-1128).

    cubed=True computes the CUBE of that value instead, for callers that only compare with one:
    the result has order dividing n and gcd(3, n) = 1, so r^3 == 1 iff r == 1.  With
    3 E = (a+1)^2 (q-a)(a^2+q^2-1) + 3 the first exponentiation is by a+1 (63 squarings) instead
    of by y = (a+1)/3 (96 squarings on its addition chain)."""
    fp_inv = fp_inverter(prog)
    # easy part: f^((q^6 - 1)(q^2 + 1))
    t = f.conj() * f.inv(fp_inv)
    m = t.frob(prog, 2) * t
    # after the easy part m lies in the cyclotomic subgroup: cheap squarings, inverse = conj
    sqr = (lambda x: x.cyclotomic_sqr()) if cyclotomic else (lambda x: x.sqr())
    # hard part: m^(y (a+1) (q-a) (a^2+q^2-1)) * m
    pow_x = (lambda f: _pow_x_compressed(prog, f, fp_inv)) if cyclotomic else (lambda f: _pow_bits(f, X_ABS, sqr))
    t1 = (pow_x(m) * m) if cubed else _pow_y(m, sqr)
    t2 = pow_x(t1) * t1                                    # ^(a+1)
    t3 = t2.frob(prog, 1) * pow_x(t2).conj()               # ^(q-a)
    t3a = pow_x(t3)
    t4 = pow_x(t3a) * t3.frob(prog, 2) * t3.conj()         # ^(a^2+q^2-1)
    if cubed:
        return t4 * (sqr(m) * m)
    return t4 * m


def load_g1(prog, buf):
    return prog.load1_be48(buf, 0), prog.load1_be48(buf, 48)


def load_g2(prog, buf):
    return prog.load2_be48(buf, 0), prog.load2_be48(buf, 96)


def store_f12(prog, buf, f):
    for k, c in enumerate(f.coeffs()):
        prog.store2_be48(buf, 96 * k, c)


def select_f12(prog, flag, a, b):
    return F12.from_coeffs([prog.sel2(flag, x, y) for x, y in zip(a.coeffs(), b.coeffs())])


def build_pairing():
    """one full pairing per item: P (96 B) x Q (192 B) -> Fq12 (576 B).
    A point given as all-zero coordinates is the point at infinity and pairs to 1, which
    is what the reference's blind computation on (0, 0) produces (SURVEY.md 9.8)."""
    prog = Program("pairing")
    prog.begin_body()
    xp, yp = load_g1(prog, BUF_P)
    xq, yq = load_g2(prog, BUF_Q)
    inf = (xp.is_zero() & yp.is_zero()) | (xq.is_zero() & yq.is_zero())
    f = miller_loop(prog, xp, yp, xq, yq)
    e = final_exponentiation(prog, f)
    e = select_f12(prog, inf, f12_one(prog), e)
    store_f12(prog, BUF_OUT, e)
    return prog


NEG_G1 = (int("17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac58"
              "6c55e83ff97a1aeffb3af00adb22c6bb", 16),
          Q - int("08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3ed"
                  "d03cc744a2888ae40caa232946c5e7e1", 16))


def f12_is_one(prog, f):
    c = f.coeffs()
    ok = c[0].eq(prog.const2((1, 0)))
    for k in range(1, 6):
        ok = ok & c[k].is_zero()
    return ok


def build_verify_pair():
    """single-message verification core (bls_py/bls.py:194-201 with one message):
        e(-G1, sig) * e(pk, H) == 1
    buffers: 0 = pk (G1 affine, 96 B), 1 = H = hash_to_g2(message hash) (G2 affine, 192 B),
    2 = sig (G2 affine, 192 B), 3 = result byte (1 = valid).  -G1 is the constant that the
    reference recomputes as Fq(n, -1) * generator on every call (bls.py:197)."""
    prog = Program("verify_pair")
    prog.begin_body()
    xk, yk = load_g1(prog, 0)
    xh, yh = load_g2(prog, 1)
    xs, ys = load_g2(prog, 2)
    inf_pk = (xk.is_zero() & yk.is_zero()) | (xh.is_zero() & yh.is_zero())
    inf_sig = xs.is_zero() & ys.is_zero()
    ng = (prog.const1(NEG_G1[0]), prog.const1(NEG_G1[1]))
    f = miller_loop_multi(prog, [(ng[0], ng[1], xs, ys, inf_sig), (xk, yk, xh, yh, inf_pk)])
    e = final_exponentiation(prog, f, cubed=True)          # only compared with one
    prog.store_flag(3, 0, f12_is_one(prog, e))
    return prog


def build_verify_full():
    """hash-to-G2 and the verification core in ONE program: the hashed point goes into the Miller
    loop as it leaves the cofactor clearing, projective, so its inversion (to_affine, ~490 M) is
    never computed.  buffers: 0 = pk (G1 affine, 96 B), 1 = SHA stage output for the message hash
    (256 B, csrc/sha256.cuh), 2 = sig (G2 affine, 192 B), 3 = result byte."""
    from .hashg2 import hash_to_g2
    prog = Program("verify_full")
    prog.begin_body()
    hx, hy, hz = hash_to_g2(prog, 1, affine=False)           # Jacobian: x = X / Z^2, y = Y / Z^3
    hz2 = hz.sqr()
    hq = (hx * hz, hy, hz2 * hz)                              # homogeneous: x = X' / Z', y = Y' / Z'
    xk, yk = load_g1(prog, 0)
    xs, ys = load_g2(prog, 2)
    inf_pk = (xk.is_zero() & yk.is_zero()) | hq[2].is_zero()
    inf_sig = xs.is_zero() & ys.is_zero()
    ng = (prog.const1(NEG_G1[0]), prog.const1(NEG_G1[1]))
    f = miller_loop_multi(prog, [(ng[0], ng[1], xs, ys, inf_sig), (xk, yk, hq, None, inf_pk)])
    e = final_exponentiation(prog, f, cubed=True)
    prog.store_flag(3, 0, f12_is_one(prog, e))
    return prog


def build_miller_raw():
    """Miller loop per item, written as Montgomery-form SoA (no byte conversion): stage 1 of
    ate_pairing_multi (bls_py/fields_t.py:1114-1121).  buffers: 0 = P (n x 96),
    1 = Q (n x 192), 2 = raw SoA Fq12 per item.  Infinite inputs contribute 1."""
    prog = Program("miller_raw")
    prog.begin_body()
    xp, yp = load_g1(prog, BUF_P)
    xq, yq = load_g2(prog, BUF_Q)
    inf = (xp.is_zero() & yp.is_zero()) | (xq.is_zero() & yq.is_zero())
    f = miller_loop_multi(prog, [(xp, yp, xq, yq, inf)])
    for k, c in enumerate(f.coeffs()):
        prog.store_raw2(2, k, c)
    return prog


def build_miller_hash_raw():
    """stage 1 of aggregate verification: H = hash_to_g2(message hash) and the Miller loop of
    (P, H) in one program, H projective (no inversion).  buffers: 0 = P (n x 96), 1 = SHA stage
    output (n x 256), 2 = raw SoA Fq12 per item, 3 = an explicitly given affine Q per item (n x 192),
    4 = one byte per item: non-zero where buffer 3 replaces the hashed point -- that is how the
    e(-G1, signature) pair rides in the same launch as the n (pk, H(m)) pairs.  The flag is explicit
    because all-zero bytes are a legitimate given Q: the point at infinity (an aggregate signature that
    sums to infinity), which contributes the factor 1 like everywhere else."""
    from .hashg2 import hash_to_g2
    prog = Program("miller_hash_raw")
    prog.begin_body()
    hx, hy, hz = hash_to_g2(prog, 1, affine=False)
    hz2 = hz.sqr()
    xg, yg = load_g2(prog, 3)
    given = prog.flag_byte(4, 0)
    given_inf = given & xg.is_zero() & yg.is_zero()
    one = prog.const2((1, 0))
    hq = (prog.sel2(given, xg, hx * hz), prog.sel2(given, yg, hy), prog.sel2(given, one, hz2 * hz))
    xk, yk = load_g1(prog, 0)
    inf = (xk.is_zero() & yk.is_zero()) | hq[2].is_zero() | given_inf
    f = miller_loop_multi(prog, [(xk, yk, hq, None, inf)])
    for k, c in enumerate(f.coeffs()):
        prog.store_raw2(2, k, c)
    return prog


def _f12_tree_product(prog, f, nt=128):
    off = nt // 2
    while off >= 1:
        f = f * F12.from_coeffs(prog.exchange(f.coeffs(), off))
        off //= 2
    return f


def _f12_fold(prog):
    """prologue + body: every thread multiplies the raw SoA Fq12 items (buffer 0) its body
    iterations visit into a persistent accumulator that starts at one; returns the accumulator
    at the start of the epilogue"""
    one12 = f12_one(prog)
    acc = [prog.var2(c) for c in one12.coeffs()]
    prog.begin_body()
    act = prog.flag_active()
    cs = [prog.load_raw2(0, k) for k in range(6)]
    cs = [prog.sel2(act, c, o) for c, o in zip(cs, one12.coeffs())]
    r = F12.from_coeffs(list(acc)) * F12.from_coeffs(cs)
    for a, v in zip(acc, r.coeffs()):
        prog.assign(a, v)
    prog.begin_epilogue()
    return F12.from_coeffs(list(acc))


def _f12_strided_product(prog):
    """prologue + body shared by the two product passes: every thread multiplies its strided
    share of raw SoA Fq12 items (buffer 0), then a tree over the CTA"""
    return _f12_tree_product(prog, _f12_fold(prog))


def build_f12_product_pass1():
    """stage 2 of ate_pairing_multi: buffers 0 = raw SoA Fq12 items, 1 = raw SoA partial
    products, one per CTA (prod = fq12_mul(prod, ml_res), fields_t.py:1120, as a tree)."""
    prog = Program("f12_prod1")
    tot = _f12_strided_product(prog)
    for k, c in enumerate(tot.coeffs()):
        prog.store_raw2(1, k, c, block_only=True)
    return prog


def build_f12_product_pass2():
    """stage 3: buffers 0 = raw SoA partials, 1 = their product as 576 big-endian bytes (NOT
    final-exponentiated: this is the value ranks exchange in multi-GPU runs).  One CTA."""
    prog = Program("f12_prod2")
    tot = _f12_strided_product(prog)
    for k, c in enumerate(tot.coeffs()):
        prog.store2_be48(1, 96 * k, c, block_only=True)
    return prog


def build_f12_product_seg(be):
    """one pass of the batched multi-pairing's segmented product (segmented launch mode, chunk
    tables from csrc/multi_plan.h): thread t multiplies the raw SoA Fq12 items of chunk t
    (buffer 0, at most kMultiL of them, read through the index list) starting from one, so an
    empty chunk gives one.  buffer 1 = one product per chunk: raw SoA (f12_prodseg, the input
    of the next pass) or 576 big-endian bytes (f12_prodseg_be, the last pass: the input of
    final_exp / final_exp_check)."""
    def build():
        prog = Program("f12_prodseg_be" if be else "f12_prodseg")
        tot = _f12_fold(prog)
        for k, c in enumerate(tot.coeffs()):
            if be:
                prog.store2_be48(1, 96 * k, c)
            else:
                prog.store_raw2(1, k, c)
        return prog
    return build


def build_miller_only():
    """Miller loop only (debug / per-stage benchmarking); output is NOT canonical."""
    prog = Program("miller")
    prog.begin_body()
    xp, yp = load_g1(prog, BUF_P)
    xq, yq = load_g2(prog, BUF_Q)
    store_f12(prog, BUF_OUT, miller_loop(prog, xp, yp, xq, yq))
    return prog


def build_final_exp_check():
    """Fq12 (576 B) -> one byte: final_exponentiation(f) == 1, through the cheaper cube (see
    final_exponentiation); the last step of aggregate verification"""
    prog = Program("final_exp_check")
    prog.begin_body()
    f = F12.from_coeffs([prog.load2_be48(0, 96 * k) for k in range(6)])
    prog.store_flag(1, 0, f12_is_one(prog, final_exponentiation(prog, f, cubed=True)))
    return prog


def build_final_exp():
    """Fq12 (576 B) -> Fq12 (576 B)"""
    prog = Program("final_exp")
    prog.begin_body()
    f = F12.from_coeffs([prog.load2_be48(0, 96 * k) for k in range(6)])
    store_f12(prog, 1, final_exponentiation(prog, f))
    return prog
