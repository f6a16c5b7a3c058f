"""Name -> builder table of every VM program embedded into libb200bls.so."""
import os

from . import curve, extras, fieldops, hashg2, pairing

# Launch shapes: CTAs (of 128 threads) per SM -> (Fq2 slots per thread in shared memory, slots in
# Tensor Memory).  Shared memory: ctas * slots * 96 B * 128 <= 227 KB; TMEM: ctas * pow2(24 *
# slots) <= 512 columns.  Every program is assembled for every shape ("<name>@<ctas>"); when a
# program cannot use TMEM (cross-thread reads) the shared-memory-only shape is used, and when
# it does not fit a shape at all the launcher falls back to fewer CTAs per SM.
N_SLOTS = 18
SHAPES = {1: (18, 21), 2: (9, 10), 3: (6, 5), 4: (6, 7), 5: (4, 5)}
# Shape 4 is the "wide" shape: ONE CTA of 384 threads per SM (same 12 warps as shape 3) that owns all
# 512 TMEM columns, 168 per group of four warps = 7 slots instead of 5.  TMEM programs only.
# Shape 5 is ONE CTA of 512 threads per SM (16 warps, 128 registers): 4 + 5 slots per item, more spills, but
# 75,776 items in one pass -- the shape of an isolated batch that is a little more than one 384-thread wave
# (BASELINE config 2: 65,536 pairings = 1.15 waves of shape 4, 0.86 of shape 5).
WIDE_SHAPES = {4, 5}
if os.environ.get("B200BLS_SHAPES"):          # experiments: "ctas:smem_slots:tmem_slots,..."
    SHAPES = {int(c): (int(a), int(b)) for c, a, b in
              (item.split(":") for item in os.environ["B200BLS_SHAPES"].split(","))}

PROGRAMS = {}
for _level in (1, 2, 6, 12):
    for _op in ("add", "sub", "mul", "sqr", "neg", "inv"):
        PROGRAMS["f%d_%s" % (_level, _op)] = fieldops.build_field_op(_level, _op)
PROGRAMS["f1_is_square"] = fieldops.build_is_square
PROGRAMS["fq2_mul_chain"] = fieldops.build_fq2_mul_chain(512)
PROGRAMS["pairing"] = pairing.build_pairing
PROGRAMS["miller_loop"] = pairing.build_miller_only
PROGRAMS["final_exp"] = pairing.build_final_exp
PROGRAMS["final_exp_check"] = pairing.build_final_exp_check
PROGRAMS["verify_pair"] = pairing.build_verify_pair
PROGRAMS["verify_full"] = pairing.build_verify_full
PROGRAMS["miller_raw"] = pairing.build_miller_raw
PROGRAMS["miller_hash_raw"] = pairing.build_miller_hash_raw
PROGRAMS["f12_prod1"] = pairing.build_f12_product_pass1
PROGRAMS["f12_prod2"] = pairing.build_f12_product_pass2
PROGRAMS["hash_to_g2"] = hashg2.build_hash_to_g2
# single-function parity programs (golden-vector replay of reference functions the hot programs only use inside
# larger computations); pow is 384 square-and-multiply steps: assembled for the one-CTA-per-SM shape only
PROGRAMS["sw_encode_g2"] = extras.build_sw_encode
for _level in (2, 6, 12):
    for _i in range(_level):
        PROGRAMS["f%d_frob%d" % (_level, _i)] = extras.build_frob(_level, _i)
for _level in (1, 2, 6, 12):
    PROGRAMS["f%d_pow" % _level] = extras.build_pow(_level)
for _level in (1, 2):
    PROGRAMS["f%d_sqrt" % _level] = extras.build_sqrt(_level)
PROGRAMS["g2_untwist"] = extras.build_untwist
PROGRAMS["f12_twist"] = extras.build_twist12
PROGRAMS["g2_psi"] = extras.build_psi
for _g2 in (False, True):
    _p = "g2" if _g2 else "g1"
    PROGRAMS[_p + "_mul"] = curve.build_scalar_mul(_g2)
    PROGRAMS[_p + "_add"] = curve.build_add(_g2)
    PROGRAMS[_p + "_sum1"] = curve.build_sum_pass1(_g2)
    PROGRAMS[_p + "_sum2"] = curve.build_sum_pass2(_g2)
    PROGRAMS[_p + "_sums"] = curve.build_sum_small(_g2)
    PROGRAMS[_p + "_sumf"] = curve.build_sum_fold(_g2)
    PROGRAMS[_p + "_sum1j"] = curve.build_sum_pass1j(_g2)
    PROGRAMS[_p + "_bucket"] = curve.build_bucket_fold(_g2)
    PROGRAMS[_p + "_bscale"] = curve.build_bucket_scale(_g2)
    PROGRAMS[_p + "_tomont"] = curve.build_to_mont(_g2)
    PROGRAMS[_p + "_bucketr"] = curve.build_bucket_fold(_g2, raw=True)
    PROGRAMS[_p + "_decompress"] = curve.build_decompress(_g2)
    for _op in ("affine", "dbl", "add", "mul"):        # the plugin seam's Jacobian-coordinate functions
        PROGRAMS[_p + "_j" + _op] = curve.build_jacobian_op(_g2, _op)
    PROGRAMS[_p + "_cflag"] = curve.build_compress_flag(_g2)
    PROGRAMS[_p + "_subgroup"] = curve.build_subgroup_check(_g2)
PROGRAMS["g1_keyvalidate"] = curve.build_subgroup_check(False, key=True)
PROGRAMS["g2_sign"] = hashg2.build_sign
PROGRAMS["g1_pubkey"] = curve.build_pubkey


# programs assembled for the one-CTA-per-SM shape only (seam / parity utilities, never launched in bulk)
SHAPE1_ONLY = {"f1_pow", "f2_pow", "f6_pow", "f12_pow"} | {n for n in PROGRAMS if "_frob" in n or "_j" in n}

_M_WEIGHT = {"MUL2": 3, "SQR2": 2, "MULFP2": 2, "MUL1": 1, "SQR1": 1, "LDBE48": 1, "LDBE32": 1, "STBE48": 1, "FGTHALF": 1,
             "INV1": 2}


def executed_mults(name, shape=4):
    """Montgomery products one item of program `name` really executes in launch shape `shape`
    (counted on the assembled code; the ALU-only loops of INV1 / FSQR1 are not multiplications and
    count only their two fix-up products).  bench.py reports the roofline fraction both with
    SURVEY 8d's frozen efficient-algorithm constant and with this number."""
    from ..vm import isa
    n_slots, n_tmem = SHAPES[shape]
    asm = PROGRAMS[name]().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    total = 0
    for w in asm.code[:, 0]:
        total += _M_WEIGHT.get(isa.OPNAME[int(w) & 0xff], 0)
    return total
