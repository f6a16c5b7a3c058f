// vm_plan.h -- launch policy of the interpreter kernels: which shape, kernel, grid and item blocks a launch gets.
// Host code only, with no CUDA call, so that tests/test_launch_plan_cpu.py pins the policy with g++.
#pragma once
#include <stddef.h>

#include "../../include/b200bls.h"
#include "vm_params.h"

namespace b200bls {

// Launch shapes, by the id the program blob stores per program (programs/registry.py SHAPES).
struct Shape {
  int threads, ctas;     // one-thread kernel: threads per CTA, CTAs per SM
  int items, ctas2;      // paired kernel: items per CTA (two threads each), CTAs per SM; ctas2 = 0: no paired form
  int tmem_group_cols;   // one-thread kernel, CTAs wider than 128 threads: the CTA owns all 512 TMEM columns and gives
                         // each group of four warps this many; 0: the CTA allocates the columns its slots need
};
constexpr int N_SHAPES = 5;
constexpr Shape kShapes[N_SHAPES + 1] = {
    {0, 0, 0, 0, 0},   // no shape 0: 0 selects the automatic policy
    {VM_NT, 1, VM2_NT / 2, 1, 0},
    {VM_NT, 2, VM2_NT / 2, 2, 0},
    {VM_NT, 3, VM2_NT / 2, 3, 0},
    // wide: 384 items per SM, one CTA of 384 threads (three groups of 168 columns = 7 Fq2 slots) or two paired CTAs
    {VM_NT_WIDE, 1, VM2_NT_WIDE / 2, 2, 168},
    // one CTA of 512 threads (kernel3.cu): four groups of 128 columns = 5 Fq2 slots; one-thread kernel only
    {VM_NT_XWIDE, 1, 0, 0, 128},
};

struct Policy {
  int sm_count = 0;
  // 1 = one thread per item (vm_kernel.cuh: the throughput kernel, 1.7 M pairings/s on whole waves); 2 = two
  // threads per item (vm_kernel2.cuh: 0.7x the throughput, but 0.7x the latency of a pass -- 14.0 instead of
  // 20.0 ms for up to 9,472 pairings); 0 = choose per launch: the paired kernel for isolated batches that leave
  // most of the GPU empty, the one-thread kernel otherwise.  Environment variable B200BLS_KERNEL.
  int kernel = 0;
  int ctas_per_sm = 0;   // the shape id of every launch (b200bls_set_ctas_per_sm); 0 = automatic
};

// What the planner needs to know of an assembled program.
struct ProgramShape {
  int shape = 1;              // the shape id it was assembled for
  int n_slots = 0, n_tmem = 0, n_cold = 0;
  bool cross_thread = false;  // block barriers / cross-thread reads: CTA-wide item blocks
};

inline long long ceil_div(long long a, long long b) { return (a + b - 1) / b; }

// The shape a launch of n items runs in.  have: bit s set where the program was assembled for shape s.  The shape
// the policy wants, else the nearest one with fewer CTAs per SM; 0 if there is none.
inline int choose_shape(const Policy& pol, size_t n, unsigned have) {
  const long long sm = pol.sm_count, items = n ? (long long)n : 1;
  int want = pol.ctas_per_sm;
  if (want == 0) {
    // An isolated batch: more CTAs per SM raise throughput but also the latency of one pass (measured pairing pass:
    // 1 : 1.3 : 1.85 for 1 : 2 : 3 CTAs/SM), so the best shape minimises passes x latency.  Pipelines that keep
    // several batches in flight (bench.py) select the wide shape (4) explicitly.
    static const double kLat[4] = {0, 1.0, 1.3, 1.85};
    double best_cost = 1e300;
    for (int c = 1; c <= 3; c++) {
      const double cost = (double)ceil_div(items, sm * VM_NT * c) * kLat[c];
      if (cost < best_cost - 1e-9) {
        best_cost = cost;
        want = c;
      }
    }
    // the wide shape holds as many items per SM as three narrow CTAs and is faster where it exists
    if (want == 3) want = 4;
    // a little more than whole 384-item waves: fewer passes on the 512-thread shape
    if (pol.kernel != 2 && items > sm * VM_NT && ceil_div(items, sm * VM_NT_XWIDE) < ceil_div(items, sm * VM_NT_WIDE))
      want = 5;
  }
  if (want == 5 && pol.kernel == 2) want = 4;   // the paired kernel has no 512-thread shape
  for (; want >= 1; want--)
    if (have >> want & 1) return want;
  return 0;
}

struct Plan {
  int family = 0;                  // 1: vm1_launch (kernel1.cu), 2: vm2_launch (kernel2.cu), 3: vm3_launch (kernel3.cu)
  bool use_tmem = false, wide = false, seg = false;   // template selectors of vm1_launch / vm2_launch
  int block = 0, grid = 0;
  size_t smem = 0;                 // dynamic shared memory per CTA
  size_t cold_bytes = 0;           // cold area: n_cold cells for every thread of the largest grid of the shape
  long long n_blocks = 0;          // VmParams fields
  int warp_fetch = 0, active_warps = 0;
  int tmem_cols = 0, tmem_group_cols = 0;
};

inline int tmem_alloc_cols(int cols) { return cols == 0 ? 0 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512; }

// The launch of n_items items of a program.  grid_override > 0 fixes the grid (block reductions that write one
// partial per CTA); segmented: one thread (pair) per segment, statically assigned.  Returns 0, B200BLS_E_PROGRAM
// when the program's TMEM slots do not fit the shape, or B200BLS_E_ARG for more items than the paired kernel's
// 32-bit item index holds.
inline int plan_launch(const Policy& pol, const ProgramShape& pr, size_t n_items, int grid_override, bool segmented,
                       Plan& p) {
  const Shape& s = kShapes[pr.shape];
  p = Plan();
  // the paired kernel where the policy forces it, and for latency-bound launches of the automatic policy: at most
  // one 128-item block per SM and no block reduction
  const bool paired = s.ctas2 > 0 && (pol.kernel == 2 || (pol.kernel == 0 && pol.ctas_per_sm == 0 && grid_override == 0 &&
                                                          !segmented && !pr.cross_thread &&
                                                          n_items <= (size_t)pol.sm_count * 128));
  if (paired && n_items > 0x7fffffffull) return B200BLS_E_ARG;
  const int per_cta = paired ? s.items : s.threads;
  p.family = paired ? 2 : s.threads == VM_NT_XWIDE ? 3 : 1;
  p.block = paired ? 2 * s.items : s.threads;
  p.seg = segmented;
  const long long n = (long long)n_items, max_grid = (long long)pol.sm_count * (paired ? s.ctas2 : s.ctas);
  const long long cta_blocks = ceil_div(n, per_cta);
  if (segmented) grid_override = (int)cta_blocks;
  p.grid = grid_override > 0 ? grid_override : (int)(cta_blocks < 1 ? 1 : cta_blocks < max_grid ? cta_blocks : max_grid);
  // (sized for the largest grid of the shape: the balancing below may spread a small batch over more CTAs)
  const long long cold_threads = (p.grid > max_grid ? p.grid : max_grid) * p.block;
  p.cold_bytes = (size_t)pr.n_cold * (paired ? 3 : 6) * sizeof(uint4) * (size_t)cold_threads;
  p.smem = (size_t)pr.n_slots * (paired ? 3 : 6) * sizeof(uint4) * (size_t)p.block;

  // Item blocks per WARP (32 items, 16 pairs) instead of per CTA, for programs without block reductions.  The paired
  // kernel always fetches so; the one-thread kernel for an isolated batch (automatic shape) and not in shape 5: with
  // 16 warps per CTA some scheduler holds four warps whether the batch is spread or not, and CTA-wide blocks keep the
  // warps of a CTA together in the program (65,536 pairings 45.6 instead of 47.3 ms).  With an explicit shape
  // (pipelines that keep launches in flight) blocks stay CTA-wide: the barrier per block keeps a CTA's warps near
  // each other in the program, which the instruction cache rewards (33.1 vs 34.3 ms).
  const int warps = p.block / 32;
  const bool automatic = pol.ctas_per_sm == 0 && grid_override == 0;
  p.n_blocks = cta_blocks;
  if (!pr.cross_thread && !segmented && (paired || (automatic && s.threads != VM_NT_XWIDE))) {
    p.warp_fetch = 1;
    p.n_blocks = ceil_div(n, paired ? VM2_ITEMS_PER_WARP : 32);
    p.active_warps = warps;
    if (automatic) {
      // An isolated batch is spread over ALL SMs and, when it is w.f waves long, runs as ceil(w.f) EQUAL waves on
      // fewer warps per CTA: a warp is faster at lower occupancy, so neither a partly filled last wave nor a handful
      // of full CTAs on a few SMs is left (65,536 pairings = 1.15 waves took 33 + 32 ms, two passes at 7 of 12
      // warps take 52).
      const long long waves = ceil_div(p.n_blocks, max_grid * warps);
      const long long per_wave = ceil_div(p.n_blocks, waves < 1 ? 1 : waves);   // warps busy at a time
      p.grid = (int)(per_wave < max_grid ? per_wave : max_grid);
      const long long act = ceil_div(per_wave, p.grid);
      p.active_warps = act < 1 ? 1 : act < warps ? (int)act : warps;
    }
  } else if (paired) {
    p.active_warps = warps;
  }

  if (paired) {
    // 12 columns per Fq cell: each thread of a pair holds one coefficient of every Fq2 slot
    p.tmem_group_cols = pr.n_tmem * 12;
    const int cols = p.block / 128 * p.tmem_group_cols;
    if (cols > 512) return B200BLS_E_PROGRAM;
    p.tmem_cols = tmem_alloc_cols(cols);
  } else if (s.tmem_group_cols) {
    if (pr.n_tmem * 24 > s.tmem_group_cols) return B200BLS_E_PROGRAM;
    p.tmem_cols = 512;
    p.tmem_group_cols = s.tmem_group_cols;
  } else {
    p.tmem_cols = tmem_alloc_cols(pr.n_tmem * 24);
  }
  p.use_tmem = p.tmem_cols != 0;
  p.wide = paired ? p.block == VM2_NT_WIDE : s.threads == VM_NT_WIDE;
  return 0;
}

}  // namespace b200bls
