// fp.cuh -- BLS12-381 base field Fq on 12 x 32-bit limbs, Montgomery form (R = 2^384).
//
// Device code is hand-written PTX carry chains: every 32x32->64 limb product is a
// mad.lo.cc / madc.hi.cc pair that ptxas fuses into one IMAD.WIDE.U32 with a
// predicate carry, accumulated into two interleaved ("even" / "odd" aligned)
// 64-bit column sets so that no carry ever has to be rippled by hand.
//
// Replaces (reference, /root/reference): the Python big-int arithmetic behind
// bls_py/fields.py:35-243 (class Fq) and the `% Q` reductions all over
// bls_py/fields_t.py.  Values are always fully reduced to [0, q) so that equality and
// zero tests are limb comparisons.
//
// The same header compiles for the host (B200BLS_HOSTSIM) with the PTX instructions
// emulated one by one, carry flag included.  That build exists ONLY so that tests can
// exercise the exact instruction sequences on the CPU-only development box
// (tests/hostsim); the product library never contains or calls it.
#pragma once
#include <stdint.h>

#include "gen/fp_consts.h"

#ifdef B200BLS_HOSTSIM
#define FP_DEV inline
#define FP_CONST static const
#else
#define FP_DEV __device__ __forceinline__
#define FP_CONST __device__ __constant__ const
#endif

namespace b200bls {

constexpr int NL = 12;  // limbs

struct fp {
  uint32_t v[NL];
};
struct fp2 {
  fp c0, c1;
};

// q, little-endian limbs
#define B200BLS_Q_LIMBS                                                                        \
  {0xffffaaabu, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u, 0xf38512bfu, \
   0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau}
constexpr uint32_t Q_INV_NEG = 0xfffcfffdu;  // -q^-1 mod 2^32

#ifdef B200BLS_HOSTSIM
static const uint32_t kQ[NL] = B200BLS_Q_LIMBS;
static const uint32_t kQ2[NL] = B200BLS_2Q_LIMBS;
#define QL(i) kQ[i]
#define Q2L(i) kQ2[i]
#else
// Compile-time immediates: the modulus limbs become instruction immediates / constant
// bank operands instead of live registers.
__device__ __forceinline__ constexpr uint32_t q_limb(int i) {
  constexpr uint32_t t[NL] = B200BLS_Q_LIMBS;
  return t[i];
}
__device__ __forceinline__ constexpr uint32_t q2_limb(int i) {
  constexpr uint32_t t[NL] = B200BLS_2Q_LIMBS;
  return t[i];
}
#define QL(i) q_limb(i)
#define Q2L(i) q2_limb(i)
#endif

// ---------------------------------------------------------------------------------------
// PTX primitives (and their host emulation)
// ---------------------------------------------------------------------------------------
#ifdef B200BLS_HOSTSIM
static thread_local uint32_t g_cf = 0;  // emulated CC.CF
inline uint32_t add_cc(uint32_t a, uint32_t b) {
  uint64_t s = (uint64_t)a + b;
  g_cf = (uint32_t)(s >> 32);
  return (uint32_t)s;
}
inline uint32_t addc_cc(uint32_t a, uint32_t b) {
  uint64_t s = (uint64_t)a + b + g_cf;
  g_cf = (uint32_t)(s >> 32);
  return (uint32_t)s;
}
inline uint32_t addc(uint32_t a, uint32_t b) { return a + b + g_cf; }
inline uint32_t sub_cc(uint32_t a, uint32_t b) {
  uint64_t s = (uint64_t)a - b;
  g_cf = (uint32_t)(s >> 63);  // borrow
  return (uint32_t)s;
}
inline uint32_t subc_cc(uint32_t a, uint32_t b) {
  uint64_t s = (uint64_t)a - b - g_cf;
  g_cf = (uint32_t)(s >> 63);
  return (uint32_t)s;
}
inline uint32_t subc(uint32_t a, uint32_t b) { return a - b - g_cf; }
inline uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
inline uint32_t mul_hi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
inline uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return add_cc(a * b, c); }
inline uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return addc_cc(a * b, c); }
inline uint32_t mad_hi_cc(uint32_t a, uint32_t b, uint32_t c) { return add_cc(mul_hi(a, b), c); }
inline uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { return addc_cc(mul_hi(a, b), c); }
inline uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) { return mul_hi(a, b) + c + g_cf; }
#else
// NB: borrow semantics of sub.cc/subc on the GPU: CC.CF holds the borrow.
__device__ __forceinline__ uint32_t add_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t addc_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t addc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t sub_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t subc_cc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t subc(uint32_t a, uint32_t b) {
  uint32_t r;
  asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
__device__ __forceinline__ uint32_t mul_hi(uint32_t a, uint32_t b) { return __umulhi(a, b); }
__device__ __forceinline__ uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t mad_hi_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("mad.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm volatile("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
#endif

// ---------------------------------------------------------------------------------------
// Value discipline: every stored Fq value x is "weakly reduced", 0 <= x < 2q (zero is 0 or
// q).  With R = 2^384 and q ~ 0.1016 R this lets a Montgomery product skip its final
// subtraction (inputs < 2q -> output < 1.41 q) and lets Fq2 products be reduced once per
// coefficient from unreduced 768-bit sums (output < 2.63 q, one conditional subtraction of
// 2q).  Canonical form [0, q) is produced only where it is observable: comparisons, the
// sign rule (FGTHALF) and serialisation.
// ---------------------------------------------------------------------------------------
FP_DEV void fp_set_zero(fp& r) {
#pragma unroll
  for (int i = 0; i < NL; i++) r.v[i] = 0;
}

// x == 0 (mod q) for weakly reduced x: x is 0 or q
FP_DEV bool fp_is_zero(const fp& a) {
  uint32_t t = 0, u = 0;
#pragma unroll
  for (int i = 0; i < NL; i++) {
    t |= a.v[i];
    u |= a.v[i] ^ QL(i);
  }
  return t == 0 || u == 0;
}

// r = x - 2q if x >= 2q else x, for x < 4q
FP_DEV void fp_cond_sub_2q(fp& r, const fp& x) {
  fp t;
  t.v[0] = sub_cc(x.v[0], Q2L(0));
#pragma unroll
  for (int i = 1; i < NL; i++) t.v[i] = subc_cc(x.v[i], Q2L(i));
  uint32_t borrow = subc(0, 0);  // 0xffffffff when x < 2q
#pragma unroll
  for (int i = 0; i < NL; i++) r.v[i] = borrow ? x.v[i] : t.v[i];
}

// canonical form: weakly reduced x -> [0, q)
FP_DEV void fp_canonical(fp& r, const fp& x) {
  fp t;
  t.v[0] = sub_cc(x.v[0], QL(0));
#pragma unroll
  for (int i = 1; i < NL; i++) t.v[i] = subc_cc(x.v[i], QL(i));
  uint32_t borrow = subc(0, 0);  // 0xffffffff when x < q
#pragma unroll
  for (int i = 0; i < NL; i++) r.v[i] = borrow ? x.v[i] : t.v[i];
}

// plain 384-bit sum, no reduction (callers guarantee a + b < 2^384)
FP_DEV void fp_add_raw(fp& r, const fp& a, const fp& b) {
  r.v[0] = add_cc(a.v[0], b.v[0]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) r.v[i] = addc_cc(a.v[i], b.v[i]);
  r.v[NL - 1] = addc(a.v[NL - 1], b.v[NL - 1]);
}

FP_DEV void fp_add(fp& r, const fp& a, const fp& b) {
  fp s;
  fp_add_raw(s, a, b);  // < 4q < 2^384
  fp_cond_sub_2q(r, s);
}

// a - b + 2q, no reduction: in (0, 4q) for weakly reduced a, b
FP_DEV void fp_sub_raw_2q(fp& r, const fp& a, const fp& b) {
  fp t;
  t.v[0] = add_cc(a.v[0], Q2L(0));
#pragma unroll
  for (int i = 1; i < NL - 1; i++) t.v[i] = addc_cc(a.v[i], Q2L(i));
  t.v[NL - 1] = addc(a.v[NL - 1], Q2L(NL - 1));
  r.v[0] = sub_cc(t.v[0], b.v[0]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) r.v[i] = subc_cc(t.v[i], b.v[i]);
  r.v[NL - 1] = subc(t.v[NL - 1], b.v[NL - 1]);
}

FP_DEV void fp_sub(fp& r, const fp& a, const fp& b) {
  fp d;
  d.v[0] = sub_cc(a.v[0], b.v[0]);
#pragma unroll
  for (int i = 1; i < NL; i++) d.v[i] = subc_cc(a.v[i], b.v[i]);
  uint32_t mask = subc(0, 0);  // all ones when a < b
  r.v[0] = add_cc(d.v[0], Q2L(0) & mask);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) r.v[i] = addc_cc(d.v[i], Q2L(i) & mask);
  r.v[NL - 1] = addc(d.v[NL - 1], Q2L(NL - 1) & mask);
}

// a == b (mod q)
FP_DEV bool fp_eq(const fp& a, const fp& b) {
  fp d;
  fp_sub(d, a, b);
  return fp_is_zero(d);
}

FP_DEV void fp_neg(fp& r, const fp& a) {
  uint32_t nz = 0;
#pragma unroll
  for (int i = 0; i < NL; i++) nz |= a.v[i];
  uint32_t mask = nz ? 0xffffffffu : 0u;
  fp d;
  d.v[0] = sub_cc(Q2L(0), a.v[0]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) d.v[i] = subc_cc(Q2L(i), a.v[i]);
  d.v[NL - 1] = subc(Q2L(NL - 1), a.v[NL - 1]);
#pragma unroll
  for (int i = 0; i < NL; i++) r.v[i] = d.v[i] & mask;
}

FP_DEV void fp_dbl(fp& r, const fp& a) { fp_add(r, a, a); }

// a > b as plain 384-bit integers (used on canonical values taken out of Montgomery form)
FP_DEV bool fp_raw_gt(const fp& a, const fp& b) {
  sub_cc(b.v[0], a.v[0]);
#pragma unroll
  for (int i = 1; i < NL; i++) subc_cc(b.v[i], a.v[i]);
  return subc(0, 0) != 0;  // borrow <=> b < a
}

// ---------------------------------------------------------------------------------------
// Legendre symbol (x / q) == +1, i.e. x is a nonzero square, WITHOUT an exponentiation: the
// binary Jacobi algorithm on 12-limb integers -- shifts, subtractions and selects only, so it
// runs on the ALU pipe beside the other warps' multiplications (the Euler criterion costs
// ~467 Montgomery products on the multiply pipe; this is ~550 rounds of ~75 ALU instructions).
//   (2 / n) = -1  iff  n = 3, 5 (mod 8);   a, n odd, a < n: (a / n) = (n - a / a) * (-1 iff
//   a = n = 3 (mod 4));   a >= n: (a / n) = (a - n / n).
// The Montgomery form x R has the same character as x because R = 2^384 is a square.
// Replaces the character tests inside the reference's Fq2.modsqrt when it is called on a
// non-residue (bls_py/fields.py:463-482 via ec.py:255-269).
// ---------------------------------------------------------------------------------------
#ifdef B200BLS_HOSTSIM
inline int fp_ctz(uint32_t x) { return __builtin_ctz(x); }
inline uint32_t fp_funnel_r(uint32_t lo, uint32_t hi, int s) {
  return (uint32_t)((((uint64_t)hi << 32) | lo) >> (s & 31));
}
inline uint32_t fp_funnel_l(uint32_t lo, uint32_t hi, int s) {
  return (uint32_t)(((((uint64_t)hi << 32) | lo) << (s & 31)) >> 32);
}
#else
__device__ __forceinline__ uint32_t fp_funnel_l(uint32_t lo, uint32_t hi, int s) {
  return __funnelshift_l(lo, hi, s);
}
__device__ __forceinline__ int fp_ctz(uint32_t x) { return __ffs((int)x) - 1; }
__device__ __forceinline__ uint32_t fp_funnel_r(uint32_t lo, uint32_t hi, int s) {
  return __funnelshift_r(lo, hi, s);
}
#endif

#ifdef B200BLS_HOSTSIM
inline
#else
// out of line: a cold loop that must not perturb the interpreter's register allocation or sit
// between its hot opcode bodies in the instruction cache (internal linkage: one copy per kernel translation unit)
static __device__ __noinline__
#endif
bool fp_is_square(fp x) {
  fp a, n;
  fp_canonical(a, x);
#pragma unroll
  for (int i = 0; i < NL; i++) n.v[i] = QL(i);
  uint32_t flip = 0;
  for (;;) {
    uint32_t nz = 0;
#pragma unroll
    for (int i = 0; i < NL; i++) nz |= a.v[i];
    if (nz == 0) break;
    if (a.v[0] == 0) {  // 32 factors of two: an even number of sign changes
#pragma unroll
      for (int i = 0; i < NL - 1; i++) a.v[i] = a.v[i + 1];
      a.v[NL - 1] = 0;
      continue;
    }
    const int z = fp_ctz(a.v[0]);
#pragma unroll
    for (int i = 0; i < NL - 1; i++) a.v[i] = fp_funnel_r(a.v[i], a.v[i + 1], z);
    a.v[NL - 1] >>= z;
    flip ^= (uint32_t)z & ((n.v[0] >> 1) ^ (n.v[0] >> 2));  // bit 0: z odd and n = 3, 5 (mod 8)
    // a is odd now: (a, n) <- (|a - n|, min(a, n)), in place (the state is two values, not three: this
    // function has to fit the paired kernel's 80-register budget next to its caller's live state)
    const uint32_t a0 = a.v[0];
    a.v[0] = sub_cc(a.v[0], n.v[0]);
#pragma unroll
    for (int i = 1; i < NL; i++) a.v[i] = subc_cc(a.v[i], n.v[i]);
    const uint32_t lt = subc(0, 0);  // all ones when a < n: swap (reciprocity), then n - a
    flip ^= lt & ((a0 & n.v[0]) >> 1);
    n.v[0] = add_cc(n.v[0], a.v[0] & lt);  // n + (a - n) = the old a
#pragma unroll
    for (int i = 1; i < NL - 1; i++) n.v[i] = addc_cc(n.v[i], a.v[i] & lt);
    n.v[NL - 1] = addc(n.v[NL - 1], a.v[NL - 1] & lt);
    a.v[0] = add_cc(a.v[0] ^ lt, lt & 1u);
#pragma unroll
    for (int i = 1; i < NL - 1; i++) a.v[i] = addc_cc(a.v[i] ^ lt, 0);
    a.v[NL - 1] = addc(a.v[NL - 1] ^ lt, 0);
  }
  uint32_t rest = n.v[0] ^ 1u;  // gcd(x, q) = 1 always unless x = 0
#pragma unroll
  for (int i = 1; i < NL; i++) rest |= n.v[i];
  return rest == 0 && (flip & 1u) == 0;
}

// ---------------------------------------------------------------------------------------
// Montgomery multiplication: r = a * b / R mod q, coarsely integrated operand scanning.
//
// State T = E + O * 2^32.  E = ev[0..11] holds 64-bit columns at even word positions,
// O = od[0..11] the columns at odd positions (od[k] has weight 2^(32(k+1))).  One round
// adds a * b_i and m * q to both sets with four carry chains of six lo/hi pairs each and
// then divides by 2^32 by *renaming*: the odd set becomes the even set of the next round
// and the even set, shifted down two words, becomes the odd one.  The word that falls
// between the two (ev[1]) is folded in by the first add of the next round, whose carry is
// consumed by the following chain -- the trick known from CGBN / sppark's mont_t.  ptxas
// fuses every lo/hi pair into one IMAD.WIDE.U32.X with a predicate carry and keeps 3-4 of
// the chains in flight.
//
// Bounds: for a < alpha q, b < beta q the result is < q (0.1016 alpha beta + 1): weakly
// reduced inputs give < 1.41 q, sums of two (< 4q each) give < 2.63 q; intermediates stay
// below (alpha + 1) q < 2^384 for alpha <= 8.  No final subtraction.
// The limit is on the FIRST operand only: the second may be any 384-bit value (fp_to_mont passes
// the raw input there, R^2 mod q first), but a first operand of 2^384 - 1 gives a wrong integer.
// Every call site passes a first operand <= 4q: weakly reduced values, sums of two, R^2 mod q,
// and in fp_inv a canonical r0.  tests/fp_exact.py models the exact integer and
// tests/test_fp_bounds_cpu.py pins both sides of the limit.
//
// (Tried and rejected, measured on B200: separate 768-bit products + one Montgomery reduction
// per Fq2 coefficient -- 744 instead of 900 limb products per Fq2 multiplication, but as many
// instructions in total and less instruction-level parallelism in the reduction rounds:
// 1.20 M vs 1.27 M pairings/s in the same launch shape.  The kernel is bound by dependent-
// issue latency, not by the multiply pipe's throughput.)
// ---------------------------------------------------------------------------------------
// acc[0..11] (+)= x[j] * y for j = start, start+2, ..., 6 columns; continues an open carry
template <bool CARRY_IN>
FP_DEV void mad_row(uint32_t* acc, const uint32_t* x, uint32_t y) {
#pragma unroll
  for (int j = 0; j < NL; j += 2) {
    if (j == 0 && !CARRY_IN)
      acc[j] = mad_lo_cc(x[j], y, acc[j]);
    else
      acc[j] = madc_lo_cc(x[j], y, acc[j]);
    acc[j + 1] = madc_hi_cc(x[j], y, acc[j + 1]);
  }
}

// same with the constant modulus as multiplicand; OFF selects even (0) / odd (1) limbs
template <int OFF>
FP_DEV void mad_row_q(uint32_t* acc, uint32_t y) {
#pragma unroll
  for (int j = 0; j < NL; j += 2) {
    if (j == 0)
      acc[j] = mad_lo_cc(QL(j + OFF), y, acc[j]);
    else
      acc[j] = madc_lo_cc(QL(j + OFF), y, acc[j]);
    acc[j + 1] = madc_hi_cc(QL(j + OFF), y, acc[j + 1]);
  }
}

// acc_new[k] = acc[k+2] + x[j]*y columns, i.e. accumulate while shifting down two words;
// starts with an incoming carry (from the fold of the dropped word)
FP_DEV void madc_row_rshift(uint32_t* acc, const uint32_t* x, uint32_t y) {
#pragma unroll
  for (int j = 0; j < NL - 2; j += 2) {
    acc[j] = madc_lo_cc(x[j], y, acc[j + 2]);
    acc[j + 1] = madc_hi_cc(x[j], y, acc[j + 3]);
  }
  acc[NL - 2] = madc_lo_cc(x[NL - 2], y, 0);
  acc[NL - 1] = madc_hi(x[NL - 2], y, 0);
}

FP_DEV void mont_round_first(uint32_t* ev, uint32_t* od, const uint32_t* a, uint32_t bi) {
#pragma unroll
  for (int j = 0; j < NL; j += 2) {
    ev[j] = mul_lo(a[j], bi);
    ev[j + 1] = mul_hi(a[j], bi);
    od[j] = mul_lo(a[j + 1], bi);
    od[j + 1] = mul_hi(a[j + 1], bi);
  }
  uint32_t m = mul_lo(ev[0], Q_INV_NEG);
  mad_row_q<1>(od, m);  // no carry out: T < 2^(32*13)
  mad_row_q<0>(ev, m);
  od[NL - 1] = addc(od[NL - 1], 0);
}

// ev: set that is even-aligned in THIS round; od: last round's even set (od[0] == 0,
// od[1] is the word to fold, od[2..] become this round's odd columns)
FP_DEV void mont_round(uint32_t* ev, uint32_t* od, const uint32_t* a, uint32_t bi) {
  ev[0] = add_cc(ev[0], od[1]);
  madc_row_rshift(od, a + 1, bi);
  mad_row<false>(ev, a, bi);
  od[NL - 1] = addc(od[NL - 1], 0);
  uint32_t m = mul_lo(ev[0], Q_INV_NEG);
  mad_row_q<1>(od, m);
  mad_row_q<0>(ev, m);
  od[NL - 1] = addc(od[NL - 1], 0);
}

FP_DEV void fp_mul_inline(fp& r, const fp& a, const fp& b) {
  uint32_t ev[NL], od[NL];
  mont_round_first(ev, od, a.v, b.v[0]);
#pragma unroll
  for (int i = 1; i < NL; i += 2) {
    mont_round(od, ev, a.v, b.v[i]);
    if (i + 1 < NL) mont_round(ev, od, a.v, b.v[i + 1]);
  }
  // 12 rounds: the last one ran with (od, ev) roles, so `od` was the even-aligned set
  // (od[0] == 0 now) and `ev` holds the odd columns: T / 2^32 = ev + (od >> one word)
  fp t;
  t.v[0] = add_cc(ev[0], od[1]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) t.v[i] = addc_cc(ev[i], od[i + 1]);
  t.v[NL - 1] = addc(ev[NL - 1], 0);
  r = t;  // < 1.41 q for weakly reduced inputs (< 2.63 q for inputs < 4q): no final subtraction
}

// ---------------------------------------------------------------------------------------
// Two-row Montgomery product: r = (a * x + b * y) / R mod q with ONE reduction -- the lazily
// reduced form of an Fq2 coefficient (c0 = a0 b0 + (2q - a1) b1, c1 = a1 b0 + a0 b1,
// fields_t.py:157-161 computes the same four products and reduces each).  Per round both product
// rows and the reduction row go into the same even / odd column sets: 36 limb products + m.
// 444 limb products per coefficient, 888 per Fq2 product (Karatsuba: 900 + the operand sums),
// and the two coefficients share nothing -- the paired kernel gives one to each thread of a pair.
//
// Bounds: a, b <= 2q (weakly reduced, or 2q - value), x, y < 2q: the running value stays below
// 2^32 (a + b + q) < 2^416 (5q = 0.51 R), the result below 8 q^2 / R + q = 1.82 q: weakly reduced
// without a final subtraction.
// ---------------------------------------------------------------------------------------
FP_DEV void mont_round2(uint32_t* ev, uint32_t* od, const uint32_t* a, uint32_t xi, const uint32_t* b, uint32_t yi) {
  ev[0] = add_cc(ev[0], od[1]);
  madc_row_rshift(od, a + 1, xi);
  mad_row<false>(ev, a, xi);
  od[NL - 1] = addc(od[NL - 1], 0);
  mad_row<false>(od, b + 1, yi);
  mad_row<false>(ev, b, yi);
  od[NL - 1] = addc(od[NL - 1], 0);
  uint32_t m = mul_lo(ev[0], Q_INV_NEG);
  mad_row_q<1>(od, m);
  mad_row_q<0>(ev, m);
  od[NL - 1] = addc(od[NL - 1], 0);
}

// the last step of either product: T / 2^32 = ev + (od >> one word) after an even number of rounds
FP_DEV void mont_finish(fp& r, const uint32_t* ev, const uint32_t* od) {
  r.v[0] = add_cc(ev[0], od[1]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) r.v[i] = addc_cc(ev[i], od[i + 1]);
  r.v[NL - 1] = addc(ev[NL - 1], 0);
}

// x, y arrive four words at a time (the streaming form: the kernel loads one 16-byte chunk of each
// per four rounds, so only a and b are held in registers for the whole product); the accumulators
// start at zero, so that every round is the general one and the twelve rounds are a loop of three passes
struct Mul2State {
  uint32_t ev[NL], od[NL];
};
// four general rounds (accumulators may start at zero): the body of the looped streaming product
FP_DEV void fp_mul2_rounds4(Mul2State& s, const fp& a, const fp& b, const uint32_t* x4, const uint32_t* y4) {
  mont_round2(s.ev, s.od, a.v, x4[0], b.v, y4[0]);
  mont_round2(s.od, s.ev, a.v, x4[1], b.v, y4[1]);
  mont_round2(s.ev, s.od, a.v, x4[2], b.v, y4[2]);
  mont_round2(s.od, s.ev, a.v, x4[3], b.v, y4[3]);
}

// The twelve rounds as a LOOP of three passes over four rounds (b rotates down four limbs per pass, the
// accumulators start at zero so that every round is the general one): ~130 instructions instead of ~350.
// With 24 warps per SM at 24 different places of the program the hot code has to fit the 32 KB instruction
// cache (ncu: 81 % hit rate and `no_instruction` the top stall with the unrolled products).  This is the
// product the kernel AND the host simulation run; fp_mul_inline is the unrolled statement of the same thing.
FP_DEV void fp_mul_looped(fp& r, const fp& a, fp b) {
  uint32_t ev[NL], od[NL];
#pragma unroll
  for (int i = 0; i < NL; i++) ev[i] = od[i] = 0;
#pragma unroll 1
  for (int k = 0; k < 3; k++) {
    mont_round(ev, od, a.v, b.v[0]);
    mont_round(od, ev, a.v, b.v[1]);
    mont_round(ev, od, a.v, b.v[2]);
    mont_round(od, ev, a.v, b.v[3]);
#pragma unroll
    for (int i = 0; i < 8; i++) b.v[i] = b.v[i + 4];
  }
  mont_finish(r, ev, od);
}

// the two-row product in the same looped form (the kernel streams x and y from the workspace instead)
FP_DEV void fp_mul2_looped(fp& r, const fp& a, const fp& x, const fp& b, const fp& y) {
  Mul2State s;
#pragma unroll
  for (int i = 0; i < NL; i++) s.ev[i] = s.od[i] = 0;
#pragma unroll 1
  for (int k = 0; k < 3; k++) fp_mul2_rounds4(s, a, b, x.v + 4 * k, y.v + 4 * k);
  mont_finish(r, s.ev, s.od);
}

#if defined(B200BLS_HOSTSIM)
// the host simulation runs the unrolled and the looped product alternately and checks that they agree
FP_DEV void fp_mul(fp& r, const fp& a, const fp& b) {
  fp u;
  fp_mul_inline(r, a, b);
  fp_mul_looped(u, a, b);
  for (int i = 0; i < NL; i++)
    if (u.v[i] != r.v[i]) __builtin_trap();
}
#elif !defined(B200BLS_MUL_CALL)
FP_DEV void fp_mul(fp& r, const fp& a, const fp& b) { fp_mul_inline(r, a, b); }
#else
// ONE copy of the multiplication in the whole kernel: operands and result travel in registers
// (ptxas: 0 bytes stack).  Unrolled: measured against the looped form (531 instead of ~400 executed
// instructions per call through the rotation of b and the zeroed accumulators; the 150 instructions it saves
// do not decide whether the hot code fits the instruction cache).
static __device__ __noinline__ fp fp_mul_call(fp a, fp b) {
  fp r;
  fp_mul_inline(r, a, b);
  return r;
}
__device__ __forceinline__ void fp_mul(fp& r, const fp& a, const fp& b) { r = fp_mul_call(a, b); }
#endif

FP_DEV void fp_sqr(fp& r, const fp& a) { fp_mul(r, a, a); }

// ---------------------------------------------------------------------------------------
// Inversion: r = 1 / x in Fq, Montgomery form in and out, 0 -> 0  (reference: fq_invert,
// bls_py/fields_t.py:47-55, extended Euclid on Python ints).
//
// Binary "almost inverse" (Kaliski) with the shifts batched by trailing-zero count.  State:
// a, n (n odd) and cofactors ra, rn with
//     n * ra + a * rn == q,     x * ra == sa * a * 2^k,     x * rn == -sa * n * 2^k   (mod q),
// so every quantity stays in [0, q] and needs no modular reduction inside the loop: a round is
// ~105 shift / subtract / select instructions on the ALU pipe, ~550 rounds per inversion, and
// no multiplication at all -- the multiply pipe stays free for the other warps, where the
// Fermat chain x^(q-2) occupied it for 465 Montgomery products.  At the end a = 0, n = 1 and
// 1 / x == -sa * rn * 2^-k; the factor 2^-k and the Montgomery scaling are applied together by
// two products: (r0 * 2^(768-k) / R) * (R^2 mod q) / R == r0 * 2^-k * R^2 (as integers mod q).
// ---------------------------------------------------------------------------------------
#ifdef B200BLS_HOSTSIM
static const uint32_t kR2inv[NL] = B200BLS_R2_LIMBS;
#define R2INVL(i) kR2inv[i]
inline
#else
__device__ __forceinline__ constexpr uint32_t r2inv_limb(int i) {
  constexpr uint32_t t[NL] = B200BLS_R2_LIMBS;
  return t[i];
}
#define R2INVL(i) r2inv_limb(i)
static __device__ __noinline__
#endif
fp fp_inv(fp x) {
  fp a, n, ra, rn;
  fp_canonical(a, x);
  fp_set_zero(ra);
  fp_set_zero(rn);
  ra.v[0] = 1;
#pragma unroll
  for (int i = 0; i < NL; i++) n.v[i] = QL(i);
  uint32_t swaps = 0;
  int k = 0;
  for (;;) {
    uint32_t nz = 0;
#pragma unroll
    for (int i = 0; i < NL; i++) nz |= a.v[i];
    if (nz == 0) break;
    if (a.v[0] == 0) {  // a whole limb of zero bits
#pragma unroll
      for (int i = 0; i < NL - 1; i++) a.v[i] = a.v[i + 1];
      a.v[NL - 1] = 0;
#pragma unroll
      for (int i = NL - 1; i > 0; i--) rn.v[i] = rn.v[i - 1];
      rn.v[0] = 0;
      k += 32;
      continue;
    }
    const int z = fp_ctz(a.v[0]);
#pragma unroll
    for (int i = 0; i < NL - 1; i++) a.v[i] = fp_funnel_r(a.v[i], a.v[i + 1], z);
    a.v[NL - 1] >>= z;
#pragma unroll
    for (int i = NL - 1; i > 0; i--) rn.v[i] = fp_funnel_l(rn.v[i - 1], rn.v[i], z);
    rn.v[0] <<= z;
    k += z;
    // a, n odd: (a, n) <- (|a - n|, min(a, n)); the cofactor of the difference is ra + rn either way.
    // Everything in place -- four 12-limb values of state and no 12-limb temporary: with the caller's live
    // registers this has to fit the paired kernel's 80-register budget.
    a.v[0] = sub_cc(a.v[0], n.v[0]);
#pragma unroll
    for (int i = 1; i < NL; i++) a.v[i] = subc_cc(a.v[i], n.v[i]);
    const uint32_t lt = subc(0, 0);  // all ones when a < n
    swaps ^= lt;
    n.v[0] = add_cc(n.v[0], a.v[0] & lt);  // n + (a - n) = the old a
#pragma unroll
    for (int i = 1; i < NL - 1; i++) n.v[i] = addc_cc(n.v[i], a.v[i] & lt);
    n.v[NL - 1] = addc(n.v[NL - 1], a.v[NL - 1] & lt);
    a.v[0] = add_cc(a.v[0] ^ lt, lt & 1u);
#pragma unroll
    for (int i = 1; i < NL - 1; i++) a.v[i] = addc_cc(a.v[i] ^ lt, 0);
    a.v[NL - 1] = addc(a.v[NL - 1] ^ lt, 0);
    fp_add_raw(ra, ra, rn);
    {  // rn <- a < n ? the old ra = (ra + rn) - rn : rn
      uint32_t t = sub_cc(ra.v[0], rn.v[0]);
      rn.v[0] = lt ? t : rn.v[0];
#pragma unroll
      for (int i = 1; i < NL - 1; i++) {
        t = subc_cc(ra.v[i], rn.v[i]);
        rn.v[i] = lt ? t : rn.v[i];
      }
      t = subc(ra.v[NL - 1], rn.v[NL - 1]);
      rn.v[NL - 1] = lt ? t : rn.v[NL - 1];
    }
  }
  // 1 / x == sn * rn * 2^-k with sn = -1 initially and negated by every swap
  fp r0;
  if (swaps & 1u) {
    r0 = rn;
  } else {
    r0.v[0] = sub_cc(QL(0), rn.v[0]);
#pragma unroll
    for (int i = 1; i < NL - 1; i++) r0.v[i] = subc_cc(QL(i), rn.v[i]);
    r0.v[NL - 1] = subc(QL(NL - 1), rn.v[NL - 1]);
  }
  while (k < 385) {  // tiny inputs (x = 1: k = 381): bring 768 - k below 384
    fp t;
    fp_add_raw(t, r0, r0);
    fp_canonical(r0, t);
    k++;
  }
  const int e = 768 - k;  // 0 <= e <= 383 since k <= 2 * 381
  fp w;
#pragma unroll
  for (int i = 0; i < NL; i++) w.v[i] = (i == (e >> 5)) ? (1u << (e & 31)) : 0u;
  fp t, r2, r;
  fp_mul(t, r0, w);
#pragma unroll
  for (int i = 0; i < NL; i++) r2.v[i] = R2INVL(i);
  fp_mul(r, t, r2);
  return r;
}

// ---------------------------------------------------------------------------------------
// Fq2 = Fq[u]/(u^2+1)  (reference: bls_py/fields.py:321-482, fields_t.py:75-161)
// ---------------------------------------------------------------------------------------
FP_DEV void fp2_add(fp2& r, const fp2& a, const fp2& b) {
  fp_add(r.c0, a.c0, b.c0);
  fp_add(r.c1, a.c1, b.c1);
}
FP_DEV void fp2_sub(fp2& r, const fp2& a, const fp2& b) {
  fp_sub(r.c0, a.c0, b.c0);
  fp_sub(r.c1, a.c1, b.c1);
}
FP_DEV void fp2_neg(fp2& r, const fp2& a) {
  fp_neg(r.c0, a.c0);
  fp_neg(r.c1, a.c1);
}
// Karatsuba, 3 base multiplications (fields_t.py:157-161 uses 4).  The operand sums are left
// unreduced (< 4q), so their product is < 2.63 q and takes one conditional subtraction of 2q.
FP_DEV void fp2_mul(fp2& r, const fp2& a, const fp2& b) {
  fp sa, sb, t0, t1, t2;
  fp_add_raw(sa, a.c0, a.c1);
  fp_add_raw(sb, b.c0, b.c1);
  fp_mul(t0, a.c0, b.c0);
  fp_mul(t1, a.c1, b.c1);
  fp_mul(t2, sa, sb);
  fp_cond_sub_2q(t2, t2);  // keeps fp_sub's input < 2q; c1 = t2 - t0 - t1 < 1.81 q either way
  fp_sub(r.c0, t0, t1);
  fp_sub(t2, t2, t0);
  fp_sub(r.c1, t2, t1);
}
// (a0 + a1)(a0 - a1 + 2q), (2 a0) a1 with unreduced sums
FP_DEV void fp2_sqr(fp2& r, const fp2& a) {
  fp s, d, e, c0;
  fp_add_raw(s, a.c0, a.c1);        // < 4q
  fp_sub_raw_2q(d, a.c0, a.c1);     // in (0, 4q)
  fp_add_raw(e, a.c0, a.c0);        // < 4q
  fp_mul(c0, s, d);                 // s d <= (a0 + q)^2 < 9 q^2: < 1.92 q, the subtraction below never fires
  fp_mul(r.c1, e, a.c1);            // < 1.82 q
  fp_cond_sub_2q(r.c0, c0);
}
// times xi = 1 + u  (fields_t.py:113-116)
FP_DEV void fp2_mul_xi(fp2& r, const fp2& a) {
  fp t;
  fp_sub(t, a.c0, a.c1);
  fp_add(r.c1, a.c0, a.c1);
  r.c0 = t;
}

}  // namespace b200bls
