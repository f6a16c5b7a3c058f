// multi_plan.h -- chunk tables of the batched multi-pairing (b200bls_pairing_multi_batch).
//
// Group g holds the pairs [off[g], off[g + 1]).  Their Miller values are multiplied in passes of the segmented
// f12_prodseg program: in every pass one thread multiplies one chunk of at most kMultiL consecutive values of one group,
// starting from one, so an empty group has one chunk that gives one.  The chunk products of a pass stay in group order
// and are the values of the next pass; the passes end when every group is down to one value.  No thread multiplies more
// than kMultiL values, so one long group does not serialise on one thread.  The group of a chunk never has to be looked
// up: a pass's values of group g are the range [start of g, start of g + 1) of the previous pass's prefix table.
//
// Tables:
//   prefix[r][g]  index of the first chunk of group g in pass r; prefix[r][n_groups] = the chunks of pass r
//   seg_start     for the pass being run: chunk c covers the values [seg_start[c], seg_start[c + 1])
//   idx           the index list of the segmented launch: idx[i] = i (the values of a chunk are consecutive)
// Host and device code, so that g++ builds the same functions for tests/test_multi_plan_cpu.py.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define MULTI_HD __host__ __device__ __forceinline__
#else
#define MULTI_HD inline
#endif

namespace b200bls {

constexpr uint32_t kMultiL = 16;                 // longest chunk (DESIGN §5: why 16)
constexpr int kMultiMaxPasses = 8;               // 16^8 = 2^32 > the most pairs a batch may hold
constexpr uint64_t kMultiMaxPairs = 0xffffffffull;   // segment starts are 32-bit
constexpr uint64_t kMultiMaxGroups = 0x7fffffffull;  // final_exp runs one item per group (paired kernel: 2^31 - 1);
                                                     // with the pair bound, pass 0 has < 2^28 + 2^31 chunks

// chunks of a group that holds n values in a pass: ceil(n / kMultiL), and one for an empty group
MULTI_HD uint32_t multi_chunks(uint64_t n) { return n == 0 ? 1u : (uint32_t)((n + kMultiL - 1) / kMultiL); }

// counts[r] = the chunks of a group of len pairs in pass r, for every r < kMultiMaxPasses (1 once it is down to one)
MULTI_HD void multi_group_chunks(uint64_t len, uint32_t* counts) {
  uint64_t n = len;
  for (int r = 0; r < kMultiMaxPasses; r++) {
    counts[r] = multi_chunks(n);
    n = counts[r];
  }
}

// passes to run, from the chunk totals of every pass: up to and including the first pass with one chunk per group
MULTI_HD int multi_passes(const uint32_t* chunks, uint64_t n_groups) {
  for (int r = 0; r < kMultiMaxPasses; r++)
    if (chunks[r] == n_groups) return r + 1;
  return kMultiMaxPasses;
}

// 0 for valid offsets of n_groups groups: off[0] = 0, never decreasing, at most kMultiMaxPairs pairs; else 1
MULTI_HD int multi_offsets_bad(const uint64_t* off, uint64_t n_groups) {
  if (n_groups > kMultiMaxGroups || off[0] != 0 || off[n_groups] > kMultiMaxPairs) return 1;
  for (uint64_t g = 0; g < n_groups; g++)
    if (off[g + 1] < off[g]) return 1;
  return 0;
}

// the segment starts of group g's chunks in pass r, and after the last group the end of the last chunk.  The values of
// group g in pass r: its pairs in pass 0, its chunk products of pass r - 1 afterwards.  Chunk k covers
// [base + k L, base + min((k + 1) L, n)): the start of chunk k + 1 is its end.
MULTI_HD void multi_segments_group(int r, uint64_t g, uint64_t n_groups, const uint64_t* off, const uint32_t* prefix,
                                   uint32_t* seg_start) {
  const uint32_t* row = prefix + (size_t)r * (n_groups + 1);
  uint64_t base, n;
  if (r == 0) {
    base = off[g];
    n = off[g + 1] - off[g];
  } else {
    const uint32_t* prev = row - (n_groups + 1);
    base = prev[g];
    n = prev[g + 1] - prev[g];
  }
  const uint32_t c0 = row[g], c = multi_chunks(n);
  for (uint32_t k = 0; k < c; k++) seg_start[c0 + k] = (uint32_t)(base + (uint64_t)k * kMultiL);
  if (g + 1 == n_groups) seg_start[row[n_groups]] = (uint32_t)(base + n);
}

}  // namespace b200bls
