"""Exact integer model of the Fq core: what every primitive of csrc/fp.cuh, vm_exec.cuh and vm_exec2.cuh returns
as an integer (not just its value mod q), the input domain each one is written for, the output bound its comments
claim, and an operand corpus per domain that reaches the ends of those domains.

Values are Python ints in [0, 2^384): the 12-limb registers of the device code.  The limb code of tests/fp_probe.cu
(host build: tests/hostsim/hostsim_fp.cpp; device build: tests/test_gpu_fp_probe.py) must return exactly these
integers on the whole corpus."""
import random

import numpy as np

Q = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
R = 1 << 384
Q2 = 2 * Q
MASK = R - 1
QINV_NEG = -pow(Q, -1, R) % R
R2 = R * R % Q
NL = 12

# ---------------------------------------------------------------------------------------------------------------
# the primitives, as integers
# ---------------------------------------------------------------------------------------------------------------


def mont(a, b):
    """fp_mul_inline / fp_mul_looped / fp_mul: (a b + M q) / R with M = -a b q^-1 mod R, no final subtraction"""
    t = a * b
    return (t + (t * QINV_NEG % R) * Q) >> 384


def mont2(a, x, b, y):
    """fp_mul2_looped: one reduction of a x + b y"""
    t = a * x + b * y
    return (t + (t * QINV_NEG % R) * Q) >> 384


def mont_quotient(t):
    """M of the reduction of t: R - 1 is the worst case"""
    return t * QINV_NEG % R


def cond_sub_2q(x):
    return x - Q2 if x >= Q2 else x


def canonical(x):
    return x - Q if x >= Q else x


def add(a, b):
    return cond_sub_2q((a + b) & MASK)


def sub(a, b):
    d = a - b
    return (d + Q2) & MASK if d < 0 else d


def neg(a):
    return 0 if a == 0 else (Q2 - a) & MASK


def sub_raw_2q(a, b):
    return (a + Q2 - b) & MASK


def neg_raw_2q(x):
    return (Q2 - x) & MASK


def xi_coeff(role, own, oth):
    """vm_exec2.cuh fp_xi_coeff: coefficient `role` of (x0 + x1 u)(1 + u), own = x_role, oth = x_(1-role)"""
    return add(own, oth if role else neg_raw_2q(oth))


def to_mont(raw):
    return mont(R2, raw)


def from_mont(a):
    return canonical(mont(a, 1))


def is_zero(a):
    return int(a == 0 or a == Q)


def eq(a, b):
    return is_zero(sub(a, b))


def raw_gt(a, b):
    return int(a > b)


def fp2_mul(a0, a1, b0, b1):
    """fp.cuh fp2_mul, Karatsuba exactly as written"""
    sa, sb = a0 + a1, b0 + b1
    t0, t1 = mont(a0, b0), mont(a1, b1)
    t2 = cond_sub_2q(mont(sa, sb))
    return sub(t0, t1), sub(sub(t2, t0), t1)


def fp2_sqr(a0, a1):
    return cond_sub_2q(mont(a0 + a1, sub_raw_2q(a0, a1))), mont(a0 + a0, a1)


def fp2_mul_xi(a0, a1):
    return sub(a0, a1), add(a0, a1)


def pair_mul2(a0, a1, b0, b1):
    """vm_exec2.cuh MUL2: role 0 a0 b0 + (2q - a1) b1, role 1 a1 b0 + a0 b1, one two-row product each"""
    return mont2(a0, b0, neg_raw_2q(a1), b1), mont2(a1, b0, a0, b1)


def pair_sqr2(a0, a1):
    """vm_exec2.cuh SQR2 (fp_sqr2_coeff): role 0 (a0 + a1)(a0 - a1 + 2q), role 1 (a1 + a1) a0"""
    return cond_sub_2q(mont(a0 + a1, sub_raw_2q(a0, a1))), cond_sub_2q(mont(a1 + a1, a0))


def pair_xi(a0, a1):
    """vm_exec2.cuh MULXI2, and POST_XI on a result held by the pair"""
    return xi_coeff(0, a0, a1), xi_coeff(1, a1, a0)


def inv_value(a):
    """fp_inv, mod q (Montgomery form in and out, 0 -> 0)"""
    x = a * pow(R, -1, Q) % Q
    return 0 if x == 0 else pow(x, -1, Q) * R % Q


def is_square(a):
    x = a % Q
    return int(x != 0 and pow(x, (Q - 1) // 2, Q) == 1)


# ---------------------------------------------------------------------------------------------------------------
# op table: probe op number (tests/fp_probe.cu enum ProbeOp), model, number of operands, per-operand domains,
# claimed output bound (exclusive unless noted), and where the claim is written
# ---------------------------------------------------------------------------------------------------------------
# Domains: "w" weakly reduced [0, 2q); "w2" (0, 2q], the 2q - value operands of the paired MUL2; "u4" unreduced
# sums [0, 4q); "u8" [0, 8q], the largest first operand the product comment allows; "raw" [0, 2^384);
# "q" canonical [0, q); "r2" the single value R^2 mod q; "bit" 0 / 1.
DOMAINS = {"w": (0, Q2), "w2": (1, Q2 + 1), "u4": (0, 4 * Q), "u8": (0, 8 * Q + 1), "raw": (0, R), "q": (0, Q),
           "bit": (0, 2)}

FP_OPS = {
    # name: (op, model, domains, bound, citation)
    "mul":        (0, mont, ("w", "w"), 1.41, "fp.cuh:372-373 (inputs < 2q -> < 1.41 q)"),
    "mul_inline": (1, mont, ("w", "w"), 1.41, "fp.cuh:372-373"),
    "mul_looped": (2, mont, ("w", "w"), 1.41, "fp.cuh:372-373"),
    "mul_u4":     (0, mont, ("u4", "u4"), 2.63, "fp.cuh:372-373 (sums of two, < 4q each -> < 2.63 q)"),
    "mul_u8":     (1, mont, ("u8", "w"), None, "fp.cuh:373-374 (intermediates < (alpha + 1) q < 2^384 for alpha <= 8)"),
    "mul_u8_looped": (2, mont, ("u8", "w"), None, "fp.cuh:373-374"),
    "mul2":       (3, mont2, ("w2", "w", "w2", "w"), 1.82, "fp.cuh:473-475 (a, b <= 2q, x, y < 2q -> < 1.82 q)"),
    "add":        (4, add, ("w", "w"), 2, "fp.cuh:216-220"),
    "sub":        (5, sub, ("w", "w"), 2, "fp.cuh:235-245"),
    "neg":        (6, neg, ("w",), 2, "fp.cuh:254-266"),
    "cond_sub_2q": (7, cond_sub_2q, ("u4",), 2, "fp.cuh:186 (x < 4q)"),
    "canonical":  (8, canonical, ("w",), 1, "fp.cuh:197 (weakly reduced -> [0, q))"),
    "sub_raw_2q": (9, sub_raw_2q, ("w", "w"), 4, "fp.cuh:222 (in (0, 4q))"),
    "neg_raw_2q": (10, neg_raw_2q, ("w",), "2q]", "vm_exec2.cuh:24 (in (0, 2q])"),
    "xi_coeff":   (11, lambda own, oth, role: xi_coeff(role, own, oth), ("w", "w", "bit"), 2,
                   "vm_exec2.cuh:37 (own < 2q, t <= 2q)"),
    "to_mont":    (12, to_mont, ("raw",), 2, "vm_exec.cuh:43 (first operand < q, the second any 384-bit value)"),
    "from_mont":  (13, from_mont, ("w",), 1, "vm_exec.cuh:46 (canonical form [0, q))"),
    "is_zero":    (14, is_zero, ("w",), None, "fp.cuh:175"),
    "eq":         (15, eq, ("w", "w"), None, "fp.cuh:247"),
    "raw_gt":     (16, raw_gt, ("raw", "raw"), None, "fp.cuh:270"),
    "fp2_mul":    (17, fp2_mul, ("w", "w", "w", "w"), 2, "fp.cuh:701-702"),
    "fp2_sqr":    (18, fp2_sqr, ("w", "w"), 2, "fp.cuh:715-723 (c0 < 1.92 q: its subtraction never fires, c1 < 1.82 q)"),
    "fp2_mul_xi": (19, fp2_mul_xi, ("w", "w"), 2, "fp.cuh:725"),
    "pair_mul2":  (20, pair_mul2, ("w", "w", "w", "w"), 1.82, "vm_exec2.cuh:8, fp.cuh:473-475"),
    "pair_sqr2":  (21, pair_sqr2, ("w", "w"), 2, "vm_exec2.cuh:10, fp_sqr2_coeff"),
    "pair_xi":    (22, pair_xi, ("w", "w"), 2, "vm_exec2.cuh:32-38"),
    "inv":        (23, inv_value, ("w",), 2, "fp.cuh:571 (Montgomery form in and out)"),
    "is_square":  (24, is_square, ("w",), None, "fp.cuh:278"),
}
TWO_OUT = {"fp2_mul", "fp2_sqr", "fp2_mul_xi", "pair_mul2", "pair_sqr2", "pair_xi"}
MOD_Q_ONLY = {"inv"}   # the model gives the value mod q; the device integer is only bounded

# claimed bounds, in units of q, that the model checks on the corpus (name -> (model of the bounded value, claim))
CLAIMS = {
    "product of weakly reduced operands < 1.41 q": (lambda a, b: mont(a, b), ("w", "w"), 1.41),
    "product of unreduced sums (< 4q) < 2.63 q": (lambda a, b: mont(a, b), ("u4", "u4"), 2.63),
    "two-row product < 1.82 q": (lambda a, x, b, y: mont2(a, x, b, y), ("w2", "w", "w2", "w"), 1.82),
    "fp2_sqr c1 = (2 a0) a1 < 1.82 q": (lambda a0, a1: mont(2 * a0, a1), ("w", "w"), 1.82),
    "paired SQR2 role 1 = (2 a1) a0 < 1.82 q": (lambda a0, a1: mont(2 * a1, a0), ("w", "w"), 1.82),
    "SQR2 role 0 / fp2_sqr c0 = (a0 + a1)(a0 - a1 + 2q) < 1.92 q": (
        lambda a0, a1: mont(a0 + a1, sub_raw_2q(a0, a1)), ("w", "w"), 1.92),
    "to_mont of any 384-bit value < 1.69 q": (lambda raw: to_mont(raw), ("raw",), 1.69),
}

# ---------------------------------------------------------------------------------------------------------------
# operand corpus
# ---------------------------------------------------------------------------------------------------------------


def _limb_patterns(hi):
    """runs of 0xffffffff limbs and single high limbs, kept below hi"""
    out = []
    for k in range(1, NL + 1):
        out.append((1 << (32 * k)) - 1)                      # k low limbs of ones
        out.append(MASK ^ ((1 << (32 * (NL - k))) - 1))      # k high limbs of ones
    for i in range(NL):
        out.append(0xFFFFFFFF << (32 * i))
        out.append(1 << (32 * i))
        out.append(1 << (32 * i + 31))
    res = []
    for v in out:
        while v >= hi:
            v >>= 1            # keep the pattern's low end, below the bound
        res.append(v)
    return res


def edge_values(dom):
    lo, hi = DOMAINS[dom]
    consts = [0, 1, 2, Q - 1, Q, Q + 1, Q2 - 1, Q2, Q2 + 1, 3 * Q, 4 * Q - 2, 4 * Q - 1, 8 * Q, R2, R - 1, R - 2,
              (Q - 1) // 2, (Q + 1) // 2, R % Q, (R - 1) % Q]
    vals = [v for v in consts if lo <= v < hi]
    vals += [v for v in _limb_patterns(hi) if lo <= v]
    return sorted(set(vals))


def band_values(dom, rnd, n):
    """random values in each band of the domain: [0, q), [q, 2q), [2q, 4q), [4q, 8q], [8q, 2^384)"""
    lo, hi = DOMAINS[dom]
    bands = [(0, Q), (Q, Q2), (Q2, 4 * Q), (4 * Q, 8 * Q), (8 * Q, R)]
    out = []
    for a, b in bands:
        a, b = max(a, lo), min(b, hi)
        if a < b:
            out += [rnd.randrange(a, b) for _ in range(n)]
    return out


def draw(dom, rnd):
    """one operand: an edge value a quarter of the time, else a random value from a random band"""
    if rnd.random() < 0.25:
        return rnd.choice(edge_values(dom))
    return rnd.choice(band_values(dom, rnd, 1))


def worst_pairs(doms, rnd, n):
    """operands of a product or a two-row product with reduction quotient M = R - 1: the largest (a b + M q) / R.
    For a b: given odd a, b = q a^-1 mod R.  For a x + b y: given a, x and odd b, y = (q - a x) b^-1 mod R."""
    out = []
    tries = 0
    while len(out) < n and tries < 400 * n:
        tries += 1
        if len(doms) == 2:
            a = draw(doms[0], rnd) | 1
            b = Q * pow(a, -1, R) % R
            args = (a, b)
        else:
            a, x = draw(doms[0], rnd), draw(doms[1], rnd)
            b = draw(doms[2], rnd) | 1
            y = (Q - a * x) * pow(b, -1, R) % R
            args = (a, x, b, y)
        if all(DOMAINS[d][0] <= v < DOMAINS[d][1] for d, v in zip(doms, args)):
            out.append(args)
    return out


def _fq2_worst(name, rnd, n):
    """Fq2 operands whose products reach the extremes: Karatsuba sums near 4q, and b1 solved so that one product
    has reduction quotient R - 1 (fp2_mul: the (a0 + a1)(b0 + b1) product; pair_mul2: either role's two-row
    product)"""
    top = Q2 - (1 << 300)
    out = []
    for _ in range(n):
        a0, a1, b0 = (rnd.randrange(top, Q2) if rnd.random() < 0.5 else draw("w", rnd) for _ in range(3))
        out.append((a0, a1, b0, rnd.randrange(top, Q2)))
        if name == "fp2_mul":
            sa = a0 + a1
            b1 = (Q * pow(sa, -1, R) - b0) % R if sa % 2 else None
        elif rnd.random() < 0.5:
            n0 = neg_raw_2q(a1)
            b1 = (Q - a0 * b0) * pow(n0, -1, R) % R if n0 % 2 else None
        else:
            b1 = (Q - a1 * b0) * pow(a0, -1, R) % R if a0 % 2 else None
        if b1 is not None and b1 < Q2:
            out.append((a0, a1, b0, b1))
    return out


def corpus(name, rnd, n_random, n_worst=0):
    """operand tuples for FP_OPS[name]: edge values (every combination for up to two operands, random combinations
    for more), random draws, and for the products operands with worst-case reduction quotients"""
    doms = FP_OPS[name][2]
    cases = []
    if len(doms) == 1:
        cases += [(v,) for v in edge_values(doms[0])]
    elif len(doms) == 2:
        e0, e1 = edge_values(doms[0]), edge_values(doms[1])
        cases += [(a, b) for a in e0 for b in e1]
    else:
        es = [edge_values(d) for d in doms]
        cases += [tuple(rnd.choice(e) for e in es) for _ in range(n_random)]
    cases += [tuple(draw(d, rnd) for d in doms) for _ in range(n_random)]
    if n_worst and FP_OPS[name][1] in (mont, mont2):
        cases += worst_pairs(doms, rnd, n_worst)
    if n_worst and name in ("fp2_mul", "pair_mul2"):
        cases += _fq2_worst(name, rnd, n_worst)
    return cases


def expected(name, args):
    """the exact output integers (one or two) of FP_OPS[name] on args"""
    r = FP_OPS[name][1](*args)
    return r if isinstance(r, tuple) else (r,)


# ---------------------------------------------------------------------------------------------------------------
# limb packing for the probe's records: in[4][12], out[2][12] uint32 per case
# ---------------------------------------------------------------------------------------------------------------


def pack_inputs(cases):
    buf = bytearray(len(cases) * 4 * 48)
    for i, args in enumerate(cases):
        for k, v in enumerate(args):
            buf[(4 * i + k) * 48:(4 * i + k + 1) * 48] = v.to_bytes(48, "little")
    return np.frombuffer(bytes(buf), dtype="<u4").copy()


def unpack_outputs(out, n):
    raw = out.astype("<u4").tobytes()
    return [(int.from_bytes(raw[96 * i:96 * i + 48], "little"), int.from_bytes(raw[96 * i + 48:96 * i + 96], "little"))
            for i in range(n)]


def check_results(names, cases, outs):
    """compares probe outputs with the model; returns a list of mismatch descriptions (empty: all exact)"""
    bad = []
    for name, args, got in zip(names, cases, outs):
        want = expected(name, args)
        if name in MOD_Q_ONLY:
            ok = got[0] % Q == want[0] and got[0] < Q2
        else:
            ok = tuple(got[:len(want)]) == want
        if not ok:
            bad.append("%s%s: got %s want %s" % (name, tuple(hex(a) for a in args), tuple(hex(g) for g in got[:len(want)]),
                                                 tuple(hex(w) for w in want)))
    return bad


def build_suite(seed, n_random, n_worst):
    """(names, ops, cases) over every op of FP_OPS"""
    rnd = random.Random(seed)
    names, ops, cases = [], [], []
    for name, spec in FP_OPS.items():
        cs = corpus(name, rnd, n_random, n_worst)
        names += [name] * len(cs)
        ops += [spec[0]] * len(cs)
        cases += cs
    return names, np.array(ops, dtype=np.int32), cases
