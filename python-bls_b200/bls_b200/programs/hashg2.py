"""hash_to_point_prehashed_Fq2 (bls_py/ec.py:528-550) as a branch-free VM program.

Pipeline per 32-byte message hash h:
  1. SHA stage (csrc/sha256.cuh): 4 x hash512(h || "G2_j_ck") -> 256 bytes.
  2. this program: t_j = (int(.) mod q, int(.) mod q); P = sw(t_0) + sw(t_1);
     H = (a^2 + a - 1) P - psi((a + 1) P) + psi^2(2 P),  a = |x|   (Budroni-Pintore clearing,
     written in the reference as t2 - t3 + psi2P, ec.py:544-550);  output affine, 192 bytes.

sw_encode (ec.py:449-507) is exception driven in the reference: it tries y_for_x(x1),
y_for_x(x2) and picks index ((X1 - 1) X2) mod 3.  Here every lane decides which candidate is
used from the Legendre symbols of the norms of g(x1), g(x2) (the FSQR1 instruction: binary Jacobi
algorithm, no multiplications) and only the selected candidate pays for a square root.  Square
roots follow fields.py:463-482 ("complex method") with one exponentiation c = n^((q-3)/4) per
Fq root, which yields the root (c n), the quadratic character (c^2 n) and the inverse root (c) at
once: two exponentiations per encode.  Both roots {y, -y} are the
same set as the reference's; the sign is then fixed by the reference's own rule
(lex_gt_neg(y) == parity, looking only at y.c1, ec.py:94-101, 505-506).

Known divergence (probability ~2^-381 per candidate, unreachable by honest hashing): when
x^3 + b has a zero imaginary part the reference takes an Fq root and then raises; this
program treats the candidate as "no y".
"""
from ..vm.builder import Program, Q
from .curve import Curve
from .tower import f2_pow_int, fp_pow_chain, f2_inv, fp_inverter

X_ABS = 0xd201000000010000
SQRT_M3 = 1586958781458431025242759403266842894121773480562120986020912974854563298150952611241517463240701
SQRT_M3_M1_O2 = 793479390729215512621379701633421447060886740281060493010456487427281649075476305620758731620350
assert SQRT_M3 * SQRT_M3 % Q == Q - 3 and (2 * SQRT_M3_M1_O2 + 1) % Q == SQRT_M3
G2_GEN = ((int("024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d177"
               "0bac0326a805bbefd48056c8c121bdb8", 16),
           int("13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049"
               "334cf11213945d57e5ac7d055d042b7e", 16)),
          (int("0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c"
               "923ac9cc3baca289e193548608b82801", 16),
           int("0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab"
               "3f370d275cec1da1aaa9075ff05f79be", 16)))
B2 = (4, 4)
ROOT_EXP = (Q - 3) // 4
HALF = (Q + 1) // 2                 # 1/2 mod q


def _f2_inv_int(a):
    n = pow(a[0] * a[0] + a[1] * a[1], Q - 2, Q)
    return (a[0] * n % Q, -a[1] * n % Q)


# psi(x, y) = (conj(x) PSI_CX, conj(y) PSI_CY); psi^2(x, y) = (x PSI2_CX, -y)   (ec.py:440-444)
PSI_CX = _f2_inv_int(f2_pow_int((1, 1), (Q - 1) // 3))
PSI_CY = _f2_inv_int(f2_pow_int((1, 1), (Q - 1) // 2))
_t = (PSI_CX[0] * PSI_CX[0] + PSI_CX[1] * PSI_CX[1]) % Q       # conj(cx) * cx
PSI2_CX = _t
assert PSI_CX[0] == 0


def fq_from_digest(prog, buf, off):
    """64 big-endian bytes -> integer mod q (ec.py:531-534): hi * 2^256 + lo"""
    hi = prog.load1_be32(buf, off)
    lo = prog.load1_be32(buf, off + 32)
    return hi * prog.const1(pow(2, 256, Q)) + lo


def _root_pow(prog, n):
    """c = n^((q-3)/4) for an Fq value n"""
    return fp_pow_chain(prog, n, ROOT_EXP)


def _candidate(prog, x):
    """u = x^3 + b, its norm n, and ok = 'y_for_x(x) succeeds' = u is a square in Fq2 = n is a
    (nonzero) square in Fq -- decided by the Legendre-symbol instruction (integer pipe only),
    not by an exponentiation"""
    u = x.sqr() * x + prog.const2(B2)
    n = u.c0.sqr() + u.c1.sqr()
    ok = n.is_square() & ~u.c1.is_zero()
    return u, n, ok


def _candidate_with_root(prog, x):
    """decompression: the candidate is always used, so ONE exponentiation c = n^((q-3)/4) gives the
    character (c^2 n) and the root of the norm (c n) together: returns (u, n, c, ok)"""
    u = x.sqr() * x + prog.const2(B2)
    n = u.c0.sqr() + u.c1.sqr()
    c = _root_pow(prog, n)
    chi = c.sqr() * n                      # norm^((q-1)/2): 1 iff nonzero square
    ok = chi.eq(prog.const1(1)) & ~u.c1.is_zero()
    return u, n, c, ok


def _sqrt_selected(prog, u, alpha):
    """a square root of u in Fq2 given alpha with alpha^2 = norm(u) (either sign: exactly one of
    (u0 + alpha) / 2 and (u0 - alpha) / 2 is a square, and both branches below only use alpha^2)"""
    half = prog.const1(HALF)
    delta = (u.c0 + alpha) * half
    c1 = _root_pow(prog, delta)
    s = c1 * delta                                     # s^2 = +-delta
    chi = s * c1                                       # +1: delta is a square, -1: it is not
    hlf = (u.c1 * c1) * half
    is_sq = chi.eq(prog.const1(1))
    y0 = prog.sel1(is_sq, s, -hlf)
    y1 = prog.sel1(is_sq, hlf, s)
    return prog.pack(y0, y1)


def sw_encode(prog, t, inv_w0, inv_3t2, w0):
    """-> (x, y, is_infinity) on E'(Fq2); inv_w0 = 1/w0, inv_3t2 = 1/(3 t^2)"""
    c = Curve(prog, True)
    t_zero = t.is_zero()
    parity = t.c1.gt_half()
    w0_zero = w0.is_zero()
    s = prog.const1(SQRT_M3)
    w = (t * s) * inv_w0
    x1 = -(w * t)
    x1 = prog.pack(x1.c0 + prog.const1(SQRT_M3_M1_O2), x1.c1)
    x2 = prog.const2((Q - 1, 0)) - x1
    x3 = -(w0.sqr() * inv_3t2)                         # 1 / w^2 = - w0^2 / (3 t^2)
    x3 = prog.pack(x3.c0 + prog.const1(1), x3.c1)
    u1, n1, ok1 = _candidate(prog, x1)
    u2, n2, ok2 = _candidate(prog, x2)
    # Shallue-van de Woestijne: g(x1) g(x2) g(x3) is a square, so the third candidate is one whenever
    # the first two are not and needs no test (the reference reaches it through two exceptions)
    u3 = x3.sqr() * x3 + prog.const2(B2)
    n3 = u3.c0.sqr() + u3.c1.sqr()
    use2 = ~ok1 & ok2
    use3 = ~ok1 & ~ok2
    x = prog.sel2(use3, x3, prog.sel2(use2, x2, x1))
    u = prog.sel2(use3, u3, prog.sel2(use2, u2, u1))
    n = prog.sel1(use3, n3, prog.sel1(use2, n2, n1))
    alpha = _root_pow(prog, n) * n                     # sqrt(norm) of the SELECTED candidate only
    y = _sqrt_selected(prog, u, alpha)
    flip = y.c1.gt_half() ^ parity
    y = prog.sel2(flip, -y, y)
    # w0 == 0 -> generator (no parity negation for Fq2, ec.py:466-470)
    gx, gy = prog.const2(G2_GEN[0]), prog.const2(G2_GEN[1])
    x = prog.sel2(w0_zero, gx, x)
    y = prog.sel2(w0_zero, gy, y)
    return x, y, t_zero


def psi(prog, p):
    """Jacobian psi: (conj(X) cx, conj(Y) cy, conj(Z))"""
    x, y, z = p
    return (x.conj() * prog.const2(PSI_CX), y.conj() * prog.const2(PSI_CY), z.conj())


def psi2(prog, p):
    x, y, z = p
    return (x * prog.const1(PSI2_CX), -y, z)


def mul_by_x_abs(c, p, complete=False, inf=None):
    """|x| * P, fixed scalar, MSB first.  With `inf` given, P = (x, y) is affine with that infinity flag and the
    additions are mixed.  complete=False leaves P + P out of the additions, which is exact while the accumulator
    cannot equal P (P of large order, as in the cofactor clearing); points of small order need complete=True."""
    mixed = inf is not None
    acc = c.from_affine(p[0], p[1], inf) if mixed else p
    for bit in bin(X_ABS)[3:]:
        acc = c.double(acc)
        if bit == "1":
            acc = c.add(acc, p, mixed=mixed, inf2=inf, complete=complete)
    return acc


def hash_to_g2(prog, buf, affine=True):
    """-> affine (x, y) of the hashed point (never infinity for honest inputs); affine=False returns
    the Jacobian point before the final inversion (callers that consume it inside the same program)"""
    c = Curve(prog, True)
    ts = []
    for j in range(2):
        c0 = fq_from_digest(prog, buf, 128 * j)
        c1 = fq_from_digest(prog, buf, 128 * j + 64)
        ts.append(prog.pack(c0, c1))
    one = prog.const2((1, 0))
    # shared inversion of w0_j and 3 t_j^2 (zero factors replaced by 1 so they cannot poison it)
    facs = []
    for t in ts:
        tt = t.sqr()
        w0 = tt + prog.const2((5, 4))                  # t^2 + b + 1
        t3 = tt.dbl() + tt
        facs.append((w0, prog.sel2(w0.is_zero(), one, w0)))
        facs.append((t3, prog.sel2(t3.is_zero(), one, t3)))
    safe = [f[1] for f in facs]
    p01 = safe[0] * safe[1]
    p23 = safe[2] * safe[3]
    inv_all = f2_inv(p01 * p23, fp_inverter(prog))
    i01 = inv_all * p23
    i23 = inv_all * p01
    invs = [i01 * safe[1], i01 * safe[0], i23 * safe[3], i23 * safe[2]]
    pts = []
    for j, t in enumerate(ts):
        pts.append(sw_encode(prog, t, invs[2 * j], invs[2 * j + 1], facs[2 * j][0]))
    (x0, y0, inf0), (x1, y1, inf1) = pts
    p = c.add(c.from_affine(x0, y0, inf0), (x1, y1), mixed=True, inf2=inf1, complete=False)
    t0 = mul_by_x_abs(c, p)                             # a P
    t1 = mul_by_x_abs(c, t0)                            # a^2 P
    t2 = c.add(c.add(t1, t0, complete=False), c.neg(p), complete=False)
    t3 = psi(prog, c.add(t0, p, complete=False))        # psi((a + 1) P)
    r = c.add(c.add(t2, c.neg(t3), complete=False), psi2(prog, c.double(p)), complete=False)
    return c.to_affine(r) if affine else r


# -psi^3(x, y) = (conj(x) PSI3_CX, conj(y) PSI_CY): psi^2 scales x by the Fq constant PSI2_CX and negates y
PSI3_CX = (PSI2_CX * PSI_CX[0] % Q, PSI2_CX * PSI_CX[1] % Q)


def sign_table(c, x, y):
    """the 16-entry table of Curve.digit_ladder for an affine point P = (x, y) of G2 (not infinity):
    B = (P, -psi P, psi^2 P, -psi^3 P) = ([1] P, [a] P, [a^2] P, [a^3] P), since psi acts on G2 as [x] = [-a];
    entry m = sum of B_i over the set bits of m.  11 mixed additions, then ONE inversion for their 11 Z coordinates."""
    prog = c.prog
    cx, cy = prog.const2(PSI_CX), prog.const2(PSI_CY)
    xc, yc = x.conj(), y.conj()
    b = [(x, y), (xc * cx, -(yc * cy)), (x * prog.const1(PSI2_CX), -y), (xc * prog.const2(PSI3_CX), yc * cy)]
    one, no_inf = c.const(1), prog.flag_const(0)
    jac = {}
    for hi in range(1, 4):                       # two base points: 3, 5, 6, 9, 10, 12
        for lo in range(hi):
            jac[(1 << hi) | (1 << lo)] = c.add((b[hi][0], b[hi][1], one), b[lo], mixed=True, inf2=no_inf)
    for m, lo, hi in ((7, 3, 2), (11, 3, 3), (13, 5, 3), (14, 6, 3), (15, 7, 3)):
        jac[m] = c.add(jac[lo], b[hi], mixed=True, inf2=no_inf)
    # Montgomery's simultaneous inversion of the Z coordinates (none is zero: the entries are not infinity)
    ms = sorted(jac)
    pre = [jac[ms[0]][2]]
    for m in ms[1:]:
        pre.append(pre[-1] * jac[m][2])
    inv = c.inv(pre[-1])
    table = [None] * 16
    for k in range(len(ms) - 1, -1, -1):
        X, Y, Z = jac[ms[k]]
        zi = inv * pre[k - 1] if k else inv
        if k:
            inv = inv * Z
        zi2 = zi.sqr()
        table[ms[k]] = (X * zi2, Y * (zi2 * zi))
    for i in range(4):
        table[1 << i] = b[i]
    table[0] = b[0]
    return table


def build_sign():
    """PrivateKey.sign_prehashed (keys.py:128-132): sk * H(h) for one message hash, from the SHA stage output and the
    digit record of sk mod n (csrc/scalar_split.h).  buffers: 0 = SHA stage output (256 B), 1 = digit records (32 B),
    2 = out (affine G2, 192 B), 3 = compression flag byte (1 iff y.c1 > q//2, the flag g2_cflag computes).
    The hashed point is in G2, where psi = [-a]: k = d0 + d1 a + d2 a^2 + d3 a^3 gives
    k H = d0 H + d1 (-psi H) + d2 psi^2 H + d3 (-psi^3 H), one 64-step joint ladder (Curve.digit_ladder) instead of
    the 128-step two-bit ladder of g2_mul.  A hashed point at infinity gives the zero signature."""
    prog = Program("g2_sign")
    prog.begin_body()
    c = Curve(prog, True)
    r = hash_to_g2(prog, 0, affine=False)
    inf = r[2].is_zero()
    x, y = c.to_affine(r)
    # infinity has no table without zero Z coordinates: ladder on the generator instead and discard the result
    x = prog.sel2(inf, prog.const2(G2_GEN[0]), x)
    y = prog.sel2(inf, prog.const2(G2_GEN[1]), y)
    sx, sy = c.to_affine(c.digit_ladder(sign_table(c, x, y), 1))
    zero = prog.const2((0, 0))
    sx, sy = prog.sel2(inf, zero, sx), prog.sel2(inf, zero, sy)
    c.store_affine(2, 0, (sx, sy))
    prog.store_flag(3, 0, sy.c1.gt_half())
    return prog


def build_hash_to_g2():
    """buffers: 0 = SHA stage output (256 B per item), 1 = out (affine G2, 192 B)"""
    prog = Program("hash_to_g2")
    prog.begin_body()
    x, y = hash_to_g2(prog, 0)
    Curve(prog, True).store_affine(1, 0, (x, y))
    return prog
