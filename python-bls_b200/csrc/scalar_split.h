// scalar_split.h -- a secret key in base a = |x| = 0xd201000000010000, the digits of the signing ladders.
//
// k = sk mod n is written k = d0 + d1 a + d2 a^2 + d3 a^3 with every digit below a < 2^64: n = a^4 - a^2 + 1 < a^4,
// so four digits suffice.  The g2_sign and g1_pubkey programs (programs/curve.py: build_sign, build_pubkey) run one
// 64-step joint ladder over the four digits; they read bit j of digit i with FBIT at bit 64 i + j, so the record is
// the 256-bit big-endian integer d0 + d1 2^64 + d2 2^128 + d3 2^192.  Host and device code with 64-bit integer
// operations only (no 128-bit type, no division instruction beyond 64 / 32 bits), so that g++ builds the same
// function for tests/test_scalar_split_cpu.py.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define SPLIT_HD __host__ __device__ __forceinline__
#else
#define SPLIT_HD inline
#endif

namespace b200bls {

constexpr uint64_t kSplitA = 0xd201000000010000ull;   // |x|; its top bit is set, as the division below requires

// (u1 * 2^64 + u0) / v for u1 < v and v >= 2^63; *r = the remainder.  Two-digit long division in base 2^32
// (Hacker's Delight, divlu, with the divisor already normalised).  Each quotient estimate is at most b + 1, so
// q * vn0 stays below 2^64.
SPLIT_HD uint64_t split_divlu(uint64_t u1, uint64_t u0, uint64_t v, uint64_t* r) {
  const uint64_t b = 1ull << 32;
  const uint64_t vn1 = v >> 32, vn0 = v & 0xffffffffull;
  const uint64_t un1 = u0 >> 32, un0 = u0 & 0xffffffffull;
  uint64_t q1 = u1 / vn1, rhat = u1 - q1 * vn1;
  while (q1 >= b || q1 * vn0 > b * rhat + un1) {
    q1--;
    rhat += vn1;
    if (rhat >= b) break;
  }
  const uint64_t un21 = u1 * b + un1 - q1 * v;   // exact mod 2^64: the true value is below v
  uint64_t q0 = un21 / vn1;
  rhat = un21 - q0 * vn1;
  while (q0 >= b || q0 * vn0 > b * rhat + un0) {
    q0--;
    rhat += vn1;
    if (rhat >= b) break;
  }
  *r = un21 * b + un0 - q0 * v;
  return q1 * b + q0;
}

// k (four limbs, least significant first) -> k / a in place; returns k mod a
SPLIT_HD uint64_t split_div_a(uint64_t* k) {
  uint64_t r = 0;
  for (int i = 3; i >= 0; i--) k[i] = split_divlu(r, k[i], kSplitA, &r);
  return r;
}

// sk: 32 bytes big-endian, any value below 2^256.  out: the 32-byte digit record described above.
SPLIT_HD void scalar_split(const uint8_t* sk, uint8_t* out) {
  const uint64_t nl[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull,
                          0x73eda753299d7d48ull};   // the group order n, least significant limb first
  uint64_t k[4];
  for (int i = 0; i < 4; i++) {
    uint64_t v = 0;
    for (int j = 0; j < 8; j++) v = (v << 8) | sk[8 * (3 - i) + j];
    k[i] = v;
  }
  // 2^256 < 3 n: two conditional subtractions reduce k mod n
  for (int round = 0; round < 2; round++) {
    uint64_t d[4], borrow = 0;
    for (int i = 0; i < 4; i++) {
      const uint64_t t = k[i] - nl[i];
      const uint64_t b1 = k[i] < nl[i];
      d[i] = t - borrow;
      borrow = b1 | (t < borrow);
    }
    for (int i = 0; i < 4; i++) k[i] = borrow ? k[i] : d[i];
  }
  uint64_t dig[4];
  dig[0] = split_div_a(k);
  dig[1] = split_div_a(k);
  dig[2] = split_div_a(k);
  dig[3] = k[0];   // k < n < a^4 leaves a quotient below a, in the lowest limb
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 8; j++) out[8 * (3 - i) + j] = (uint8_t)(dig[i] >> (56 - 8 * j));
}

}  // namespace b200bls
