"""G1 / G2 arithmetic on BLS12-381 as VM programs (Jacobian coordinates, a = 0).

Reference behaviour restated (paths relative to /root/reference):
  * add      bls_py/fields_t.py:762-875  (u1,u2,s1,s2; equal -> double; opposite -> infinity)
  * double   bls_py/fields_t.py:878-933
  * k * P    bls_py/fields_t.py:705-740  (double and add; result compared after to_affine)
  * affine   bls_py/fields_t.py:609-632  (infinity -> (0, 0))
  * sums     bls_py/bls.py:13-26 (aggregate_sigs_simple), 204-223 (aggregate_pub_keys)
The point at infinity is represented by Z = 0 in Jacobian form and by all-zero coordinates
in affine form (the reference's (0, 0, True)).  Only affine / serialised values are
canonical; Jacobian intermediates differ from the reference's whenever the order of
operations differs (tree reduction vs left fold).
"""
from ..vm.builder import Program, Q
from .tower import fp_inverter, f2_inv

G1_GEN = (int("17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac58"
              "6c55e83ff97a1aeffb3af00adb22c6bb", 16),
          int("08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3ed"
              "d03cc744a2888ae40caa232946c5e7e1", 16))
# phi(x, y) = (BETA x, y) acts on G1 as [-x^2] (x the BLS parameter); the other primitive cube root of unity, BETA^2,
# gives the eigenvalue x^2 - 1 instead
BETA = 0x5f19672fdf76ce51ba69c6076a0f77eaddb3a93be6f89688de17d813620a00022e01fffffffefffe
assert pow(BETA, 3, Q) == 1 and BETA != 1


class Curve:
    """field adapter: G1 works on V1 values, G2 on V2 values"""

    def __init__(self, prog, g2):
        self.prog = prog
        self.g2 = g2
        self.coord_bytes = 96 if g2 else 48
        self._hoisted = {}

    def const(self, x):
        if x in self._hoisted:
            return self._hoisted[x]
        if self.g2:
            return self.prog.const2(x if isinstance(x, tuple) else (x, 0))
        return self.prog.const1(x)

    def hoist_consts(self, *xs):
        """load these constants once, here (call it in the prologue of a program whose body runs per item):
        const() then hands out the same value instead of reloading it in every iteration"""
        for x in xs:
            self._hoisted[x] = self.const(x)

    def sel(self, f, a, b):
        return self.prog.sel2(f, a, b) if self.g2 else self.prog.sel1(f, a, b)

    def load(self, buf, off):
        return self.prog.load2_be48(buf, off) if self.g2 else self.prog.load1_be48(buf, off)

    def store(self, buf, off, v, block_only=False):
        if self.g2:
            self.prog.store2_be48(buf, off, v, block_only)
        else:
            self.prog.store1_be48(buf, off, v, block_only)

    def inv(self, a):
        fp_inv = fp_inverter(self.prog)
        return f2_inv(a, fp_inv) if self.g2 else fp_inv(a)

    def mov(self, a):
        if self.g2:
            r = self.prog.const2((0, 0))
            self.prog.emit("MOV2", r, a)
            return r
        return self.prog.mov1(a)

    # ---- point formulas ---------------------------------------------------------------
    def load_affine(self, buf, off=0):
        """-> (x, y, is_infinity flag)"""
        x = self.load(buf, off)
        y = self.load(buf, off + self.coord_bytes)
        return x, y, x.is_zero() & y.is_zero()

    def store_affine(self, buf, off, p, block_only=False):
        self.store(buf, off, p[0], block_only)
        self.store(buf, off + self.coord_bytes, p[1], block_only)

    def infinity(self):
        return (self.const(1), self.const(1), self.const(0))

    def from_affine(self, x, y, inf):
        """affine (with infinity flag) -> Jacobian with Z = 0 for infinity"""
        z = self.sel(inf, self.const(0), self.const(1))
        return (x, y, z)

    def double(self, p):
        x, y, z = p
        yy = y.sqr()
        s = (x * yy).dbl().dbl()
        xx = x.sqr()
        m = xx.dbl() + xx
        x3 = m.sqr() - s.dbl()
        y3 = m * (s - x3) - yy.sqr().dbl().dbl().dbl()
        z3 = (y * z).dbl()
        return (x3, y3, z3)

    def add(self, p1, p2, mixed=False, inf2=None, complete=True, rare_special=False):
        """Jacobian addition.  mixed=True: p2 = (x2, y2) affine with infinity flag inf2.
        complete=False leaves out the P + P case (callers whose operands cannot coincide:
        fixed-scalar ladders on points of large order); infinities and P + (-P) are still
        handled."""
        prog = self.prog
        x1, y1, z1 = p1
        inf1 = z1.is_zero()
        z1z1 = z1.sqr()
        if mixed:
            x2, y2 = p2
            u1, s1 = x1, y1
            u2 = x2 * z1z1
            s2 = y2 * (z1z1 * z1)
        else:
            x2, y2, z2 = p2
            inf2 = z2.is_zero()
            z2z2 = z2.sqr()
            u1 = x1 * z2z2
            u2 = x2 * z1z1
            s1 = y1 * (z2z2 * z2)
            s2 = y2 * (z1z1 * z1)
        h = u2 - u1
        r = s2 - s1
        hh = h.sqr()
        hhh = hh * h
        v = u1 * hh
        x3 = r.sqr() - hhh - v.dbl()
        y3 = r * (v - x3) - s1 * hhh
        z3 = z1 * h if mixed else (z1 * z2) * h
        both = ~(inf1 | inf2)
        h0 = h.is_zero()
        r0 = r.is_zero()
        need_dbl = both & h0 & r0
        opposite = both & h0 & ~r0
        if complete:
            # rare: P + P.  Skipped by every warp in which no lane needs it.
            with prog.skip_unless(need_dbl):
                dx, dy, dz = self.double(p1)
                prog.update_sel(x3, need_dbl, dx)
                prog.update_sel(y3, need_dbl, dy)
                prog.update_sel(z3, need_dbl, dz)
        if rare_special:
            # P + (-P) and infinite operands patched in place inside ONE region that a warp skips unless a lane
            # needs it (the per-point folds: seven selects less on the common path)
            special = opposite | inf1 | inf2
            zero, one = self.const(0), self.const(1)
            with prog.skip_unless(special):
                prog.update_sel(z3, opposite, zero)
                if mixed:
                    z2j = self.sel(inf2, zero, one)
                    p2j = (x2, y2, z2j)
                else:
                    p2j = p2
                prog.update_sel(x3, inf1, p2j[0])
                prog.update_sel(y3, inf1, p2j[1])
                prog.update_sel(z3, inf1, p2j[2])
                prog.update_sel(x3, inf2, x1)
                prog.update_sel(y3, inf2, y1)
                prog.update_sel(z3, inf2, z1)
            return (x3, y3, z3)
        # P + (-P) = infinity (Z = 0; X, Y arbitrary non-garbage)
        z3 = self.sel(opposite, self.const(0), z3)
        # identity operands
        if mixed:
            one = self.const(1)
            p2j = (x2, y2, self.sel(inf2, self.const(0), one))
        else:
            p2j = p2
        x3 = self.sel(inf1, p2j[0], x3)
        y3 = self.sel(inf1, p2j[1], y3)
        z3 = self.sel(inf1, p2j[2], z3)
        x3 = self.sel(inf2, x1, x3)
        y3 = self.sel(inf2, y1, y3)
        z3 = self.sel(inf2, z1, z3)
        return (x3, y3, z3)

    def neg(self, p):
        return (p[0], -p[1]) + tuple(p[2:])

    def to_affine(self, p):
        """-> (x, y); infinity (Z = 0) maps to (0, 0) because 0^-1 = 0 here as in
        bls_py/fields_t.py:47-55 -- but X, Y of an infinity may be arbitrary, so force it"""
        x, y, z = p
        inf = z.is_zero()
        zi = self.inv(z)
        zi2 = zi.sqr()
        ax = x * zi2
        ay = y * (zi2 * zi)
        zero = self.const(0)
        return self.sel(inf, zero, ax), self.sel(inf, zero, ay)

    def scalar_mul(self, x, y, inf, scalar_buf, n_bits=256):
        """k * (x, y) for the item's 32-byte big-endian scalar: MSB-first, two bits per step.
        P, 2P and 3P are kept affine (one shared inversion), so a step is two doublings and ONE
        mixed addition of the entry the two scalar bits select -- per-thread flags and selects, so
        every lane runs the same code (the reference's ladder, fields_t.py:705-740, adds once per
        set bit; a uniform one-bit ladder would add once per bit).  Exact for every curve point,
        small-order ones included: 2P or 3P may be infinity, which the table carries as flags."""
        assert n_bits % 2 == 0
        prog = self.prog
        one = self.const(1)
        p2 = self.double(self.from_affine(x, y, inf))
        p3 = self.add(p2, (x, y), mixed=True, inf2=inf)
        inf2p, inf3p = p2[2].is_zero(), p3[2].is_zero()
        z2 = self.sel(inf2p, one, p2[2])
        z3 = self.sel(inf3p, one, p3[2])
        w = self.inv(z2 * z3)
        zi2, zi3 = w * z3, w * z2
        zi2s, zi3s = zi2.sqr(), zi3.sqr()
        x2, y2 = p2[0] * zi2s, p2[1] * (zi2s * zi2)
        x3, y3 = p3[0] * zi3s, p3[1] * (zi3s * zi3)
        acc = self.infinity()
        for bit in range(n_bits - 2, -2, -2):
            if bit != n_bits - 2:
                acc = self.double(self.double(acc))
            d1 = prog.flag_bit(scalar_buf, bit + 1)
            d0 = prog.flag_bit(scalar_buf, bit)
            tx = self.sel(d1, self.sel(d0, x3, x2), x)
            ty = self.sel(d1, self.sel(d0, y3, y2), y)
            # infinity flag of the selected entry: d1 ? (d0 ? inf3p : inf2p) : inf
            tinf = (d1 & ((d0 & inf3p) | (~d0 & inf2p))) | (~d1 & inf)
            s = self.add(acc, (tx, ty), mixed=True, inf2=tinf)
            nz = d1 | d0
            acc = tuple(self.sel(nz, a, b) for a, b in zip(s, acc))
        return acc

    def digit_ladder(self, table, digit_buf):
        """sum_i d_i B_i for the four 64-bit digits d_i of the item's record in `digit_buf` (csrc/scalar_split.h: digit
        i in bits [64 i, 64 i + 64)), as ONE joint ladder of 64 steps, MSB first.  table[m] = (x, y) is the affine sum of
        the B_i over the set bits i of m (table[0] is never used but must be some value); an entry may be a constant
        (int for G1, pair for G2), loaded again in every step instead of being kept live.  A step is one doubling, a
        4-flag selection of the entry and one complete mixed addition; when all four bits are clear the accumulator is
        kept.  The entries must not be infinity (B_i of order n: a sum of distinct (-a)^i is a non-zero integer of
        magnitude below n).  The additions stay complete: the accumulator equals +-(entry) exactly when a relation
        sum c_i (-a)^i = 0 mod n with |c_i| < a holds, and nothing rules that out."""
        prog = self.prog
        get = (lambda v: self.const(v) if isinstance(v, (int, tuple)) else v)
        no_inf = prog.flag_const(0)
        acc = None
        for j in range(63, -1, -1):
            f = [prog.flag_bit(digit_buf, 64 * i + j) for i in range(4)]
            level = table
            for fi in f:
                level = [(self.sel(fi, get(b[0]), get(a[0])), self.sel(fi, get(b[1]), get(a[1])))
                         for a, b in zip(level[0::2], level[1::2])]
            tx, ty = level[0]
            nz = (f[0] | f[1]) | (f[2] | f[3])
            if acc is None:
                acc = (tx, ty, self.sel(nz, self.const(1), self.const(0)))
                continue
            acc = self.double(acc)
            s = self.add(acc, (tx, ty), mixed=True, inf2=no_inf)
            acc = tuple(self.sel(nz, a, b) for a, b in zip(s, acc))
        return acc

    def subgroup_ladder(self, x, y, inf):
        """the Jacobian multiple in_subgroup compares with the endomorphism image: [|x|] P on G2, [x^2] P =
        [|x|]([|x|] P) on G1.  Complete additions: on a point of small order the accumulator can equal P at an
        addition step (the order-3 and order-11 points of E(Fq) do)."""
        from .hashg2 import mul_by_x_abs
        acc = mul_by_x_abs(self, (x, y), complete=True, inf=inf)
        return acc if self.g2 else mul_by_x_abs(self, acc, complete=True)

    def in_subgroup(self, x, y, inf):
        """flag: the affine point is on the curve and in the prime-order subgroup (infinity is).  Endomorphism tests
        (Scott, "A note on group membership tests for G1, G2 and GT on BLS pairing-friendly curves", 2021):
        G2: psi(P) == [x] P = -[|x|] P;  G1: phi(P) == -[x^2] P = -[|x|]([|x|] P).
        The ladder result (X, Y, Z) is compared with the affine image (x', y') projectively: X == x' Z^2,
        Y == -y' Z^3, Z != 0.  The curve equation is checked too: the doubling formulas never use b, so an
        off-curve point would be tested on another curve."""
        from .hashg2 import PSI_CX, PSI_CY, B2
        prog = self.prog
        on_curve = y.sqr().eq(x.sqr() * x + self.const(B2 if self.g2 else 4))
        X, Y, Z = self.subgroup_ladder(x, y, inf)
        if self.g2:
            xi, yi = x.conj() * prog.const2(PSI_CX), y.conj() * prog.const2(PSI_CY)
        else:
            xi, yi = x * prog.const1(BETA), y
        zz = Z.sqr()
        same = X.eq(xi * zz) & (-Y).eq(yi * (zz * Z)) & ~Z.is_zero()
        return inf | (on_curve & same)


# ---------------------------------------------------------------------------------------
# programs
# ---------------------------------------------------------------------------------------
def build_scalar_mul(g2):
    """buffers: 0 = points (affine, 96/192 B), 1 = scalars (32 B big-endian), 2 = out (affine).
    Replaces fq_/fq2_scalar_mult_jacobian (fields_t.py:705-740) followed by to_affine."""
    def build():
        prog = Program("g2_mul" if g2 else "g1_mul")
        prog.begin_body()
        c = Curve(prog, g2)
        x, y, inf = c.load_affine(0)
        acc = c.scalar_mul(x, y, inf, 1)
        c.store_affine(2, 0, c.to_affine(acc))
        return prog
    return build


MSM_C = 11          # window bits of the multi-scalar multiplication (csrc/b200bls.cu: MSM_C, MSM_W)
MSM_W = 24


def build_bucket_scale(g2):
    """(digit << (MSM_C * window)) * P for one bucket (segment) sum P of the multi-scalar multiplication.
    buffers: 0 = points (affine), 1 = 32-byte records {digit: 2 bytes big-endian, then MSM_W - 1 bytes g[k] = (window > k)},
    2 = out (affine).  An MSM_C-bit double-and-add for the digit, then `window` blocks of MSM_C doublings, block k
    skipped by every warp in which no lane has window > k (segments are sorted by bucket, so a warp's lanes share
    their window almost always): ~2.6 k Montgomery products on average instead of the 8.4 k of the 256-bit ladder."""
    def build():
        prog = Program("g2_bscale" if g2 else "g1_bscale")
        prog.begin_body()
        c = Curve(prog, g2)
        x, y, inf = c.load_affine(0)
        acc = None
        for bit in range(MSM_C - 1, -1, -1):
            f = prog.flag_bit(1, bit, nbytes=2)
            if acc is None:
                # top bit: acc = bit ? P : infinity
                z = c.sel(f & ~inf, c.const(1), c.const(0))
                acc = (c.mov(x), c.mov(y), z)
                continue
            acc = c.double(acc)
            s = c.add(acc, (x, y), mixed=True, inf2=inf)
            acc = tuple(c.sel(f, a, b) for a, b in zip(s, acc))
        # the selects above produce fresh values; the skip regions below update three fixed values in place
        acc = tuple(c.mov(v) for v in acc)
        for k in range(MSM_W - 1):
            g = prog.flag_byte(1, 2 + k)
            with prog.skip_unless(g):
                d = acc
                for _ in range(MSM_C):
                    d = c.double(d)
                for a, v in zip(acc, d):
                    prog.update_sel(a, g, v)
        c.store_affine(2, 0, c.to_affine(acc))
        return prog
    return build


def build_add(g2):
    """buffers: 0 = a, 1 = b, 2 = out, all affine.  Replaces fq_/fq2_add_points_jacobian
    (fields_t.py:762-819) on to_jacobian'd inputs followed by to_affine."""
    def build():
        prog = Program("g2_add" if g2 else "g1_add")
        prog.begin_body()
        c = Curve(prog, g2)
        x1, y1, i1 = c.load_affine(0)
        x2, y2, i2 = c.load_affine(1)
        s = c.add(c.from_affine(x1, y1, i1), (x2, y2), mixed=True, inf2=i2)
        c.store_affine(2, 0, c.to_affine(s))
        return prog
    return build


def _pack_point(prog, c, p):
    """Jacobian point -> list of V2 for raw SoA storage"""
    if c.g2:
        return list(p)
    return [prog.pack(p[0], p[1]), prog.pack(p[2], p[2])]


def _unpack_point(prog, c, vals):
    if c.g2:
        return tuple(vals)
    return (vals[0].c0, vals[0].c1, vals[1].c0)


def _tree_reduce(prog, c, acc, nt=128):
    """sum of every thread's acc into thread 0 (all threads execute the same adds)"""
    off = nt // 2
    while off >= 1:
        other = prog.exchange(_pack_point(prog, c, acc), off)
        acc = c.add(acc, _unpack_point(prog, c, other))
        off //= 2
    return acc


def build_sum_pass1(g2):
    """buffers: 0 = affine points (n items), 1 = raw SoA partials (one Jacobian point per CTA).
    Every thread folds its strided share with mixed additions, then the CTA tree-reduces."""
    def build():
        prog = Program("g2_sum1" if g2 else "g1_sum1")
        c = Curve(prog, g2)
        c.hoist_consts(0, 1)
        inf0 = c.infinity()
        acc = [prog.var2(v) if g2 else v for v in inf0]
        if not g2:
            # G1 accumulators are Fq values: keep them as persistent Fq2-cell variables
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        x, y, inf = c.load_affine(0)
        inf = inf | ~prog.flag_active()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, (x, y), mixed=True, inf2=inf, rare_special=True)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        tot = _tree_reduce(prog, c, cur)
        for k, v in enumerate(_pack_point(prog, c, tot)):
            prog.store_raw2(1, k, v, block_only=True)
        return prog
    return build


def build_sum_fold(g2):
    """Large sums, pass A: buffers 0 = affine points (n items), 1 = raw SoA Jacobian partials, ONE PER THREAD.  No
    cross-thread step, so the program runs in the 12-warp shape with Tensor-Memory slots (g?_sum1 with its CTA
    tree is held to two CTAs of 128 threads per SM); pass B (g?_sum1j) folds and tree-reduces the partials."""
    def build():
        prog = Program("g2_sumf" if g2 else "g1_sumf")
        c = Curve(prog, g2)
        inf0 = c.infinity()
        if g2:
            acc = [prog.var2(v) for v in inf0]
        else:
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        x, y, inf = c.load_affine(0)
        inf = inf | ~prog.flag_active()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, (x, y), mixed=True, inf2=inf)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        for k, v in enumerate(_pack_point(prog, c, cur)):
            prog.store_raw2(1, k, v)
        return prog
    return build


def build_sum_pass1j(g2):
    """Large sums, pass B: buffers 0 = raw SoA Jacobian partials (n items, one per thread of pass A), 1 = raw SoA
    partials, one per CTA.  Full Jacobian additions per thread, then the CTA tree of g?_sum1."""
    def build():
        prog = Program("g2_sum1j" if g2 else "g1_sum1j")
        c = Curve(prog, g2)
        inf0 = c.infinity()
        if g2:
            acc = [prog.var2(v) for v in inf0]
        else:
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        n_vals = 3 if g2 else 2
        vals = [prog.load_raw2(0, k) for k in range(n_vals)]
        p = _unpack_point(prog, c, vals)
        act = prog.flag_active()
        p = (p[0], p[1], c.sel(act, p[2], c.const(0)))
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, p)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        tot = _tree_reduce(prog, c, cur)
        for k, v in enumerate(_pack_point(prog, c, tot)):
            prog.store_raw2(1, k, v, block_only=True)
        return prog
    return build


def build_sum_small(g2):
    """Small sums in ONE launch of one CTA: buffers 0 = affine points (n items), 1 = out (affine, one point).  The fold
    of g?_sum1 followed directly by the tree and the to_affine of g?_sum2: up to a few hundred points (the 8 per-rank
    partial sums of a sharded aggregation, the two or three signatures of an AggregationInfo merge) do not need two
    passes."""
    def build():
        prog = Program("g2_sums" if g2 else "g1_sums")
        c = Curve(prog, g2)
        inf0 = c.infinity()
        if g2:
            acc = [prog.var2(v) for v in inf0]
        else:
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        x, y, inf = c.load_affine(0)
        inf = inf | ~prog.flag_active()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, (x, y), mixed=True, inf2=inf)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        tot = _tree_reduce(prog, c, cur)
        c.store_affine(1, 0, c.to_affine(tot), block_only=True)
        return prog
    return build


def build_sum_pass2(g2):
    """buffers: 0 = raw SoA partials (n items, one per CTA of pass 1), 1 = out (affine, one
    point).  Launched with a single CTA."""
    def build():
        prog = Program("g2_sum2" if g2 else "g1_sum2")
        c = Curve(prog, g2)
        inf0 = c.infinity()
        if g2:
            acc = [prog.var2(v) for v in inf0]
        else:
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        n_vals = 3 if g2 else 2
        vals = [prog.load_raw2(0, k) for k in range(n_vals)]
        p = _unpack_point(prog, c, vals)
        act = prog.flag_active()
        p = (p[0], p[1], c.sel(act, p[2], c.const(0)))
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, p)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        tot = _tree_reduce(prog, c, cur)
        c.store_affine(1, 0, c.to_affine(tot), block_only=True)
        return prog
    return build


def build_to_mont(g2):
    """buffers: 0 = affine points (big-endian bytes), 1 = the same coordinates as raw Montgomery limbs (SoA, one Fq2
    cell per item and element: G2 x, y; G1 (x, y) packed).  The multi-scalar multiplication reads every point once per
    window (24 times): converting once here takes the byte swap and the to-Montgomery product out of its fold."""
    def build():
        prog = Program("g2_tomont" if g2 else "g1_tomont")
        prog.begin_body()
        c = Curve(prog, g2)
        x = c.load(0, 0)
        y = c.load(0, c.coord_bytes)
        if g2:
            prog.store_raw2(1, 0, x)
            prog.store_raw2(1, 1, y)
        else:
            prog.store_raw2(1, 0, prog.pack(x, y))
        return prog
    return build


def build_bucket_fold(g2, raw=False):
    """One bucket of the multi-scalar multiplication per thread (segmented launch mode of the
    kernel): buffers 0 = affine points, read through the sorted index list (raw=True: the Montgomery-form copy
    written by g?_tomont), 1 = out, one affine bucket sum per thread.  The accumulator stays Jacobian across the
    segment; one inversion per bucket at the end.  Used by secure aggregation, sum_i T_i * P_i (bls_py/bls.py:29-56,
    132-144, 217-221)."""
    def build():
        prog = Program(("g2_bucket" if g2 else "g1_bucket") + ("r" if raw else ""))
        c = Curve(prog, g2)
        inf0 = c.infinity()
        if g2:
            acc = [prog.var2(v) for v in inf0]
        else:
            acc = [prog.var2(prog.pack(v, v)) for v in inf0]
        prog.begin_body()
        if not raw:
            x, y, inf = c.load_affine(0)
        elif g2:
            x, y = prog.load_raw2(0, 0), prog.load_raw2(0, 1)
            inf = x.is_zero() & y.is_zero()
        else:
            xy = prog.load_raw2(0, 0)
            x, y = xy.c0, xy.c1
            inf = x.is_zero() & y.is_zero()
        inf = inf | ~prog.flag_active()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        s = c.add(cur, (x, y), mixed=True, inf2=inf)
        for a, v in zip(acc, s):
            if g2:
                prog.assign(a, v)
            else:
                prog.emit("MOV1", a.c0, v)
        prog.begin_epilogue()
        cur = tuple(acc) if g2 else tuple(a.c0 for a in acc)
        c.store_affine(1, 0, c.to_affine(cur))
        return prog
    return build


def build_jacobian_op(g2, op):
    """The reference's Jacobian-coordinate functions on JACOBIAN inputs (fields_t.py:609-632 to_affine, 705-740
    scalar_mult_jacobian, 762-819 add_points_jacobian, 878-933 double_point_jacobian): buffers 0 = a = (X, Y, Z),
    three coordinates of 48 / 96 bytes each (infinity: Z = 0), 1 = b (a second Jacobian point for "add", a 32-byte
    scalar for "mul", unused otherwise), 2 = out, the result as an AFFINE point (zero bytes = infinity) -- the
    normalised representative (x, y, 1) of the Jacobian triple the reference returns."""
    def build():
        prog = Program("%s_j%s" % ("g2" if g2 else "g1", op))
        prog.begin_body()
        c = Curve(prog, g2)
        w = c.coord_bytes
        p1 = (c.load(0, 0), c.load(0, w), c.load(0, 2 * w))
        if op == "affine":
            r = c.to_affine(p1)
        elif op == "dbl":
            r = c.to_affine(c.add(p1, p1))            # the complete addition: P + P doubles, infinity stays
        elif op == "add":
            p2 = (c.load(1, 0), c.load(1, w), c.load(1, 2 * w))
            r = c.to_affine(c.add(p1, p2))
        elif op == "mul":
            x, y = c.to_affine(p1)
            inf = x.is_zero() & y.is_zero()
            r = c.to_affine(c.scalar_mul(x, y, inf, 1))
        else:
            raise ValueError(op)
        c.store_affine(2, 0, r)
        return prog
    return build


def build_decompress(g2):
    """Signature.from_bytes (bls_py/signature.py:22-38) / PublicKey.from_bytes
    (bls_py/keys.py:29-40): compressed x with the 'big y' flag in the top bit ->
    affine point.  buffers: 0 = compressed (96 / 48 B), 1 = out affine (192 / 96 B),
    2 = ok byte (0 where the reference raises 'No sqrt exists' / 'No y for point x')."""
    from .hashg2 import _candidate_with_root, _sqrt_selected, ROOT_EXP
    from .tower import fp_pow_chain

    def build():
        prog = Program("g2_decompress" if g2 else "g1_decompress")
        prog.begin_body()
        big = prog.flag_bit(0, 255)                  # top bit of byte 0
        if g2:
            x = prog.load2_be48(0, 0, mask_top=True)
            u, n, cc, ok = _candidate_with_root(prog, x)
            y = _sqrt_selected(prog, u, cc * n)
            flip = y.c1.gt_half() ^ big              # want (y.c1 > q//2) == big
            y = prog.sel2(flip, -y, y)
            zero = prog.const2((0, 0))
            prog.store2_be48(1, 0, prog.sel2(ok, x, zero))
            prog.store2_be48(1, 96, prog.sel2(ok, y, zero))
        else:
            x = prog.load1_be48(0, 0, mask_top=True)
            u = x.sqr() * x + prog.const1(4)
            cc = fp_pow_chain(prog, u, ROOT_EXP)
            r = cc * u
            ok = (r * cc).eq(prog.const1(1))         # u is a nonzero square
            flip = r.gt_half() ^ big
            y = prog.sel1(flip, -r, r)
            zero = prog.const1(0)
            prog.store1_be48(1, 0, prog.sel1(ok, x, zero))
            prog.store1_be48(1, 48, prog.sel1(ok, y, zero))
        prog.store_flag(2, 0, ok)
        return prog
    return build


def build_subgroup_check(g2, key=False):
    """buffers: 0 = affine points (96 / 192 B), 1 = flag byte: 1 iff the point is on the curve and in G1 / G2
    (Curve.in_subgroup; infinity counts as a member).  Coordinates are read mod q like every affine input, so
    infinity is any pair of coordinates that reduces to (0, 0): zero bytes, and also q || 0, 0 || q, q || q.
    key=True (G1, "g1_keyvalidate"): the public-key rule of strict verification, a member that is NOT infinity,
    decided on the same reduced coordinates.  The reference checks neither."""
    def build():
        prog = Program("g1_keyvalidate" if key else ("g2_subgroup" if g2 else "g1_subgroup"))
        prog.begin_body()
        c = Curve(prog, g2)
        x, y, inf = c.load_affine(0)
        f = c.in_subgroup(x, y, inf)
        prog.store_flag(1, 0, f & ~inf if key else f)
        return prog
    return build


def _g1_aff_add(p, q):
    """affine sum of two distinct, non-opposite points of E(Fq) (build-time constants only)"""
    lam = (q[1] - p[1]) * pow(q[0] - p[0], -1, Q) % Q
    x = (lam * lam - p[0] - q[0]) % Q
    return (x, (lam * (p[0] - x) - p[1]) % Q)


def _g1_aff_mul(k, p):
    """k P for 0 < k < n by double-and-add on affine points (build-time constants only)"""
    acc = None
    for bit in bin(k)[2:]:
        if acc is not None:
            lam = 3 * acc[0] * acc[0] * pow(2 * acc[1], -1, Q) % Q
            x = (lam * lam - 2 * acc[0]) % Q
            acc = (x, (lam * (acc[0] - x) - acc[1]) % Q)
        if bit == "1":
            acc = p if acc is None else _g1_aff_add(acc, p)
    return acc


def _g1_pubkey_table():
    """entry m = sum of [a^i] G1 over the set bits i of m (a = |x|); entry 0 repeats G1 (never selected)"""
    from .hashg2 import X_ABS
    base = [G1_GEN]
    for _ in range(3):
        base.append(_g1_aff_mul(X_ABS, base[-1]))
    table = [G1_GEN]
    for m in range(1, 16):
        pt = None
        for i in range(4):
            if m >> i & 1:
                pt = base[i] if pt is None else _g1_aff_add(pt, base[i])
        table.append(pt)
    return table


G1_PUBKEY_TABLE = _g1_pubkey_table()


def build_pubkey():
    """PrivateKey.get_public_key (keys.py:119-121): sk * G1 from the digit record of sk mod n (csrc/scalar_split.h).
    buffers: 0 = digit records (32 B), 1 = out (affine G1, 96 B), 2 = compression flag byte (1 iff y > q//2, the
    flag g1_cflag computes).  The base point is fixed, so the table of the joint ladder ([a^i] G1 and their subset
    sums, G1_PUBKEY_TABLE) is constants: 64 doublings and 64 mixed additions, against 255 doublings and 128 additions
    of g1_mul."""
    prog = Program("g1_pubkey")
    prog.begin_body()
    c = Curve(prog, False)
    x, y = c.to_affine(c.digit_ladder(G1_PUBKEY_TABLE, 0))
    c.store_affine(1, 0, (x, y))
    prog.store_flag(2, 0, y.gt_half())
    return prog


def build_compress_flag(g2):
    """AffinePoint.lex_gt_neg (bls_py/ec.py:94-101): the serialisation flag of an affine
    point.  buffers: 0 = affine point, 1 = flag byte (1 iff y > q//2, resp. y.c1 > q//2).
    The compressed form is the x bytes with (flag << 7) OR-ed into byte 0 (ec.py:103-111)."""
    def build():
        prog = Program("g2_cflag" if g2 else "g1_cflag")
        prog.begin_body()
        if g2:
            y = prog.load2_be48(0, 96)
            f = y.c1.gt_half()
        else:
            y = prog.load1_be48(0, 48)
            f = y.gt_half()
        prog.store_flag(1, 0, f)
        return prog
    return build
