// b200bls.cu -- C ABI (include/b200bls.h) over the field-VM kernel.
//
// Host side of the library: owns the CUDA context objects (one device per process), the
// embedded field programs (csrc/gen/programs.bin, linked in as a binary object), staging
// buffers for the host-pointer entry points, and the launch logic.  No CPU compute path
// exists here: every entry point either launches vm_kernel on the GPU or fails.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200bls.h"
#include "comm.cuh"
#include "sha256.cuh"
#include "gen/vm_isa.h"
#include "multi_plan.h"
#include "scalar_split.h"
#include "vm_launch.h"
#include "vm_plan.h"

using namespace b200bls;

extern "C" {
extern const unsigned char _binary_programs_bin_start[];
extern const unsigned char _binary_programs_bin_end[];
}

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(B200BLS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                    \
  } while (0)

struct BlobEntry {
  char name[32];
  uint32_t n_ins, body_start, epi_start, n_consts, n_slots, n_cold, n_tmem, shape;
  uint64_t code_off, consts_off;
};
static_assert(sizeof(BlobEntry) == 32 + 32 + 16, "blob entry layout");

struct DevProgram : ProgramShape {
  uint2* code = nullptr;
  uint4* consts = nullptr;
  int n_ins = 0, body_start = 0, epi_start = 0;
};

struct Staging {
  void* ptr = nullptr;
  size_t cap = 0;
};

// Per-stream device buffers of the host-pointer entry points and the multi-stage pipelines, grown on demand and
// kept.  Names with the same value share one buffer: their pipelines never run inside one another.
enum Buf {
  HOST_IO = 0,   // with_staging: the device copy of host argument i is buffer HOST_IO + i (i < VM_MAX_BUFS)
  // aggregate_miller_host: the aggregate entry points stage their inputs themselves, never inside with_staging
  AGG_P = HOST_IO, AGG_MH, AGG_Q, AGG_MILLER, AGG_GIVEN,
  GATHERED = HOST_IO + 5,   // gather_partials: all ranks' partials (host gather)
  SHARD_ACC,                // sharded entry points: this rank's partial, then the combined result
  // device pipelines, each of which may run inside the ones above
  SUM_PARTS = HOST_IO + VM_MAX_BUFS,   // sum_dev: one partial per CTA
  SUM_THREAD_PARTS,         // sum_dev in three passes: one partial per thread
  MILLER_RAW,               // miller_product_dev, aggregate_miller_dev: one raw Miller value per item
  PROD_PARTS,               // raw_product_dev (inside the two above): one partial product per CTA
  SHA_OUT,                  // sha_stage_dev output: aggregate_miller_dev, hash_to_g2_dev, verify_dev
  MSM_MONT,                 // msm_dev (calls sum_dev): the points in Montgomery limbs
  MSM_SEG_SUMS,             //   segment sums (or the per-point products of a small MSM)
  MSM_COUNT,                //   bucket counts / cursors
  MSM_OFFSETS,              //   bucket offsets, segment counts
  MSM_IDX,                  //   point indices grouped by bucket
  MSM_SEGMENTS,             //   segment offsets and scalars
  MSM_SCALED,               //   segment sums times their bucket scalars
  // verify_wire_dev (calls verify_dev and strict_flags_dev) and msm_dev never run inside one another
  WIRE_PK = MSM_SEG_SUMS,   // decoded keys
  WIRE_PK_OK = MSM_COUNT,   // key decoding flags
  WIRE_SIG_OK = MSM_OFFSETS,   // signature decoding flags
  WIRE_SIG = MSM_SCALED,    // decoded signatures
  STRICT_FLAGS,             // strict_flags_dev: key and signature subgroup flags
  CFLAGS,                   // compress_dev: the flag bit of every point
  MULTI_PRODUCT = CFLAGS,   // b200bls_pairing_multi_dev (calls miller_product_dev): the Miller product
  // sign_dev and public_key_dev call neither msm_dev nor verify_wire_dev, and neither runs inside them; they take the
  // three MSM buffers that verify_wire_dev leaves alone
  SIGN_DIGITS = MSM_MONT,   // the base-a digits of sk mod n (scalar_split.h): secret, zeroed after the program
  SIGN_AFFINE = MSM_IDX,    // wire output: the affine points before the compression pack
  SIGN_FLAGS = MSM_SEGMENTS,   // the compression flag of every point
  // pairing_multi_batch_dev calls none of msm_dev, verify_wire_dev, sign_dev, public_key_dev, miller_product_dev, and
  // none of them calls it: it takes the MSM buffers (and MILLER_RAW for the Miller values)
  MULTI_TABLES = MSM_OFFSETS,  //   the header (validity, pairs, chunks per pass) and the prefix tables (multi_plan.h)
  MULTI_SEG = MSM_SEGMENTS,    //   the segment starts of the pass being run
  MULTI_IDX = MSM_IDX,         //   the index list of the segmented launches
  MULTI_PARTS = MSM_SEG_SUMS,  //   raw chunk products of the even passes
  MULTI_PARTS2 = MSM_SCALED,   //   raw chunk products of the odd passes
  MULTI_FINAL = MSM_MONT,      //   one product per group, big-endian: the input of the final exponentiation
  N_BUFS = MULTI_PRODUCT + 1
};

constexpr int N_STREAMS = 8;

// Everything a launch needs privately, so that launches on different streams can overlap:
// the spill (cold) area, the item-block counter and the multi-stage buffers.
struct StreamCtx {
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  uint4* cold = nullptr;
  size_t cold_bytes = 0;
  int* counters = nullptr;   // ring of item-block counters, one per launch in flight
  unsigned counter_pos = 0;
  Staging bufs[N_BUFS];
};
constexpr int N_COUNTERS = 256;

struct Context {
  bool ready = false;
  int device = -1;
  Policy policy;   // sm_count, B200BLS_KERNEL, b200bls_set_ctas_per_sm
  StreamCtx sc[N_STREAMS];
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::map<std::string, DevProgram> programs;
  uint64_t launches = 0;
  // segment tables of the serial tiny sums (sum_dev): idx[16] = 0..15, then for n = 0..16 the pair {0, n}
  unsigned* tiny_seg = nullptr;
};

Context g_ctx;
Comm g_comm;
std::mutex g_mu;
// stream used by the calling THREAD's API calls (b200bls_set_stream): host threads that drive different
// library streams do not disturb each other's selection
thread_local int t_stream = 0;

StreamCtx& cur() { return g_ctx.sc[t_stream]; }
#define STREAM (cur().stream)

void* dbuf(Buf b) { return cur().bufs[b].ptr; }

int ensure(Buf b, size_t bytes) {
  Staging& s = cur().bufs[b];
  if (s.cap >= bytes) return 0;
  if (s.ptr) cudaFree(s.ptr);
  s.ptr = nullptr;
  s.cap = 0;
  size_t cap = bytes + bytes / 4 + 4096;
  cudaError_t e = cudaMalloc(&s.ptr, cap);
  if (e != cudaSuccess) return fail(B200BLS_E_NOMEM, "cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(e));
  s.cap = cap;
  return 0;
}

struct SegArgs {
  const unsigned* start;  // n_items + 1 offsets
  const unsigned* idx;
};

int launch_program(const DevProgram& pr, size_t n_items, const VmBuf* bufs, int n_bufs, int grid_override = 0,
                   const SegArgs* seg = nullptr) {
  Plan pl;
  int rc = plan_launch(g_ctx.policy, pr, n_items, grid_override, seg != nullptr, pl);
  if (rc == B200BLS_E_ARG) return fail(rc, "%zu items exceed the paired kernel's 2^31 - 1", n_items);
  if (rc) return fail(rc, "shape %d: %d TMEM slots do not fit its columns", pr.shape, pr.n_tmem);
  StreamCtx& sc = cur();
  if (pl.cold_bytes > sc.cold_bytes) {
    CU(cudaStreamSynchronize(sc.stream));
    if (sc.cold) cudaFree(sc.cold);
    sc.cold = nullptr;
    sc.cold_bytes = 0;
    cudaError_t e = cudaMalloc(&sc.cold, pl.cold_bytes);
    if (e != cudaSuccess) return fail(B200BLS_E_NOMEM, "cold area cudaMalloc(%zu) failed", pl.cold_bytes);
    sc.cold_bytes = pl.cold_bytes;
  }
  int* counter = sc.counters + (sc.counter_pos++ % N_COUNTERS);
  CU(cudaMemsetAsync(counter, 0, sizeof(int), sc.stream));
  VmParams p;
  memset(&p, 0, sizeof(p));
  p.code = pr.code;
  p.body_start = pr.body_start;
  p.epi_start = pr.epi_start;
  p.n_ins = pr.n_ins;
  p.consts = pr.consts;
  p.cold = sc.cold;
  p.n_items = (long long)n_items;
  p.n_blocks = pl.n_blocks;
  p.counter = counter;
  if (seg) {
    p.seg_start = seg->start;
    p.seg_idx = seg->idx;
  }
  p.smem_cells = 2 * pr.n_slots;
  p.tmem_cols = pl.tmem_cols;
  p.tmem_group_cols = pl.tmem_group_cols;
  p.warp_fetch = pl.warp_fetch;
  p.active_warps = pl.active_warps;
  for (int i = 0; i < n_bufs && i < VM_MAX_BUFS; i++) p.bufs[i] = bufs[i];
  if (pl.family == 2)
    vm2_launch(pl.use_tmem, pl.wide, pl.seg, pl.grid, pl.smem, sc.stream, p);
  else if (pl.family == 3)
    vm3_launch(pl.grid, pl.smem, sc.stream, p);
  else
    vm1_launch(pl.use_tmem, pl.wide, pl.grid, pl.smem, sc.stream, p);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

// "<name>@<shape>": that program; "<name>": the shape choose_shape picks for n_items among those it was assembled for
const DevProgram* find_program(const char* base, size_t n_items = 0) {
  std::string name(base);
  if (name.find('@') == std::string::npos) {
    unsigned have = 0;
    for (int s = 1; s <= N_SHAPES; s++)
      if (g_ctx.programs.count(name + "@" + std::to_string(s))) have |= 1u << s;
    if (int s = choose_shape(g_ctx.policy, n_items, have)) name += "@" + std::to_string(s);
  }
  auto it = g_ctx.programs.find(name);
  if (it != g_ctx.programs.end()) return &it->second;
  fail(B200BLS_E_PROGRAM, "unknown program '%s'", base);
  return nullptr;
}

// Every compute entry point runs under the library mutex, after its own argument checks, and only once
// b200bls_init() has succeeded: there is no CPU path.
template <class F>
int locked(F&& body) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "b200bls_init() has not succeeded");
  return body();
}

struct HostIO {
  const void* in;   // host source (nullptr for pure outputs)
  void* out;        // host destination (nullptr for pure inputs)
  size_t bytes;
};

// The host-pointer form of a device pipeline: copies the inputs up into buffers HOST_IO + i, runs body on the device
// pointers and copies the outputs back on the calling thread's stream.  Synchronises unless async: then
// b200bls_sync() must precede any use of the outputs, and pinned host buffers let the copies overlap other streams'
// kernels.
template <class F>
int with_staging(const HostIO* io, int n_io, F&& body, bool async = false) {
  return locked([&] {
    void* dev[VM_MAX_BUFS];
    for (int i = 0; i < n_io; i++) {
      int rc = ensure(Buf(HOST_IO + i), io[i].bytes ? io[i].bytes : 1);
      if (rc) return rc;
      dev[i] = dbuf(Buf(HOST_IO + i));
      if (io[i].in && io[i].bytes) CU(cudaMemcpyAsync(dev[i], io[i].in, io[i].bytes, cudaMemcpyHostToDevice, STREAM));
    }
    int rc = body(dev);
    if (rc) return rc;
    for (int i = 0; i < n_io; i++)
      if (io[i].out && io[i].bytes) CU(cudaMemcpyAsync(io[i].out, dev[i], io[i].bytes, cudaMemcpyDeviceToHost, STREAM));
    if (!async) CU(cudaStreamSynchronize(STREAM));
    return 0;
  });
}

struct DevBuf {
  const void* ptr;
  size_t stride;
};

int run_dev(const char* name, size_t n, const DevBuf* db, int n_bufs) {
  const DevProgram* pr = find_program(name, n);
  if (!pr) return B200BLS_E_PROGRAM;
  if (n == 0) return 0;
  VmBuf bufs[VM_MAX_BUFS];
  memset(bufs, 0, sizeof(bufs));
  for (int i = 0; i < n_bufs; i++) {
    bufs[i].ptr = (unsigned char*)db[i].ptr;
    bufs[i].stride = (long long)db[i].stride;
  }
  return launch_program(*pr, n, bufs, n_bufs);
}

// one program on host buffers: io[i].bytes is the size of ONE item of argument i
int run_host(const char* name, size_t n, std::initializer_list<HostIO> per_item, bool async = false) {
  HostIO io[VM_MAX_BUFS];
  DevBuf db[VM_MAX_BUFS];
  const int k = (int)per_item.size();
  for (int i = 0; i < k; i++) {
    io[i] = per_item.begin()[i];
    db[i].stride = io[i].bytes;
    io[i].bytes *= n;
  }
  return with_staging(io, k, [&](void** d) {
    for (int i = 0; i < k; i++) db[i].ptr = d[i];
    return run_dev(name, n, db, k);
  }, async);
}

int launch_named(const char* name, size_t n, const VmBuf* bufs, int n_bufs, int grid_override = 0) {
  const DevProgram* pr = find_program(name, n);
  if (!pr) return B200BLS_E_PROGRAM;
  return launch_program(*pr, n, bufs, n_bufs, grid_override);
}

// the grid of a launch without override: block reductions size their per-CTA partials with it and fix it
int grid_of(const DevProgram& pr, size_t n_items) {
  Plan pl;
  plan_launch(g_ctx.policy, pr, n_items, 0, false, pl);
  return pl.grid;
}

VmBuf vb(const void* p, long long stride) {
  VmBuf b;
  b.ptr = (unsigned char*)p;
  b.stride = stride;
  return b;
}

// ---- point sums: strided fold per thread + CTA tree (pass 1), then one CTA (pass 2) --------
// From 2 M points on, three passes (below): measured 1 M G2 points 2.81 ms in two passes, 2.95 in three; 8 M points
// 19 ms in two, 13.7 in three (the third pass costs ~0.8 ms, the 12-warp fold saves 0.7 ms per million points).
constexpr size_t kSumThreePassMin = 2000000;
// Up to 1,024 points (eight per thread of one CTA) in ONE launch: the second pass costs more than the serial adds it saves.
constexpr size_t kSumOnePassMax = 1024;
// Up to 6 points: one thread adds them one after the other (measured below that: 7 tree levels cost more).
constexpr size_t kSumSerialMax = 6;
int sum_dev(bool g2, const void* pts, void* out, size_t n) {
  const char* n1 = g2 ? "g2_sum1" : "g1_sum1";
  const char* n2 = g2 ? "g2_sum2" : "g1_sum2";
  size_t w = g2 ? 192 : 96;
  if (n == 0) {  // empty sum = point at infinity = zero bytes
    CU(cudaMemsetAsync(out, 0, w, STREAM));
    return 0;
  }
  if (n <= kSumSerialMax) {   // a handful of points: ONE thread folds them (the bucket program on one segment)
    const DevProgram* pb = find_program(g2 ? "g2_bucket" : "g1_bucket", 1);
    if (!pb) return B200BLS_E_PROGRAM;
    SegArgs seg = {g_ctx.tiny_seg + 16 + 2 * n, g_ctx.tiny_seg};
    VmBuf bs[2] = {vb(pts, (long long)w), vb(out, (long long)w)};
    return launch_program(*pb, 1, bs, 2, 0, &seg);
  }
  if (n <= kSumOnePassMax) {   // one CTA, one launch: fold, tree and to_affine in the same program
    VmBuf bs[2] = {vb(pts, (long long)w), vb(out, (long long)w)};
    return launch_named(g2 ? "g2_sums" : "g1_sums", n, bs, 2, 1);
  }
  if (n >= kSumThreePassMin && g_ctx.policy.kernel != 2) {
    // Large sums in three passes.  A: every thread of the 12-warp shape folds its share with mixed additions and
    // stores its Jacobian partial (g?_sumf has no cross-thread step, so it is not held to two 128-thread CTAs per
    // SM like g?_sum1 with its tree); B: the partials are folded and tree-reduced per CTA (g?_sum1j); C: one CTA.
    const DevProgram* pf = find_program(g2 ? "g2_sumf@4" : "g1_sumf@4", n);
    const int nt = pf ? kShapes[pf->shape].threads : 0;
    const DevProgram* pj = pf ? find_program(g2 ? "g2_sum1j" : "g1_sum1j", (size_t)g_ctx.policy.sm_count * nt) : nullptr;
    if (pf && pj) {
      const int grid_a = grid_of(*pf, n);
      const size_t parts = (size_t)grid_a * nt;   // n >= parts: every thread is active in the epilogue
      const size_t elems = g2 ? 3 : 2;
      int rc = ensure(SUM_THREAD_PARTS, elems * 6 * sizeof(uint4) * parts);
      if (rc) return rc;
      VmBuf ba[2] = {vb(pts, (long long)w), vb(dbuf(SUM_THREAD_PARTS), (long long)parts)};
      rc = launch_program(*pf, n, ba, 2, grid_a);
      if (rc) return rc;
      const int grid_b = grid_of(*pj, parts);
      rc = ensure(SUM_PARTS, elems * 6 * sizeof(uint4) * grid_b);
      if (rc) return rc;
      VmBuf bb[2] = {vb(dbuf(SUM_THREAD_PARTS), (long long)parts), vb(dbuf(SUM_PARTS), grid_b)};
      rc = launch_program(*pj, parts, bb, 2, grid_b);
      if (rc) return rc;
      VmBuf bc[2] = {vb(dbuf(SUM_PARTS), grid_b), vb(out, (long long)w)};
      return launch_named(n2, (size_t)grid_b, bc, 2, 1);
    }
  }
  const DevProgram* p1 = find_program(n1, n);
  if (!p1) return B200BLS_E_PROGRAM;
  int grid = grid_of(*p1, n);
  size_t raw_bytes = (size_t)(g2 ? 3 : 2) * 6 * sizeof(uint4) * grid;
  int rc = ensure(SUM_PARTS, raw_bytes);
  if (rc) return rc;
  VmBuf b1[2] = {vb(pts, (long long)w), vb(dbuf(SUM_PARTS), grid)};
  rc = launch_program(*p1, n, b1, 2, grid);
  if (rc) return rc;
  VmBuf b2[2] = {vb(dbuf(SUM_PARTS), grid), vb(out, (long long)w)};
  return launch_named(n2, (size_t)grid, b2, 2, 1);
}

// ---- multi-scalar multiplication sum_i k_i P_i (secure aggregation, bls.py:29-56, 132-144,
// 217-221): bucket method.  Scalars are cut into MSM_W windows of MSM_C bits; a counting sort
// groups the (point, window) pairs by bucket = (window, digit); buckets are cut into segments
// of bounded length and one thread per segment folds its points (g?_bucket program, segmented
// launch); the segment sums are then multiplied by digit << (MSM_C * window) -- an MSM_C-bit ladder and `window`
// blocks of MSM_C doublings, warp-uniformly skipped (g?_bscale) -- and summed by the ordinary reduction.  24 mixed additions per
// point instead of 255 doublings + ~128 additions.
constexpr int MSM_C = 11;
constexpr int MSM_W = 24;                  // 24 * 11 = 264 >= 256 bits
constexpr int MSM_B = MSM_W << MSM_C;      // 49,152 buckets (digit 0 stays empty)
constexpr size_t MSM_MIN_N = 65536;        // below this the per-point ladder is as fast

__device__ __forceinline__ unsigned msm_digit(const uint8_t* sc, int w) {
  const int lo = w * MSM_C, byte = lo >> 3;
  unsigned v = 0;
#pragma unroll
  for (int k = 0; k < 3; k++)
    if (byte + k < 32) v |= (unsigned)sc[31 - (byte + k)] << (8 * k);  // scalars are big-endian
  return (v >> (lo & 7)) & ((1u << MSM_C) - 1);
}

__global__ void msm_count_kernel(const uint8_t* __restrict__ scalars, unsigned* __restrict__ count, long long n) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * MSM_W) return;
  const long long i = t / MSM_W;
  const int w = (int)(t % MSM_W);
  const unsigned d = msm_digit(scalars + i * 32, w);
  if (d) atomicAdd(count + ((unsigned)w << MSM_C) + d, 1u);
}

// exclusive scans over the MSM_B bucket counts, one block of 1024 threads:
//   start[b]     offset of bucket b in the grouped index list (start[MSM_B] = number of pairs)
//   seg_first[b] number of segments before bucket b, a bucket of c points being cut into
//                ceil(c / seg_len) segments so that no thread folds more than seg_len points
//                (scalars are caller data: a skewed digit distribution -- equal scalars, or the
//                2-bit top window of a 255-bit scalar -- must not serialise the fold)
// Clears count so that the scatter pass can reuse it as the per-bucket cursor.
__global__ void __launch_bounds__(1024) msm_scan_kernel(unsigned* __restrict__ count, unsigned* __restrict__ start,
                                                        unsigned* __restrict__ seg_first, unsigned seg_len) {
  constexpr int PER = MSM_B / 1024;
  __shared__ unsigned part[1024], part2[1024];
  const int t = threadIdx.x;
  unsigned sum = 0, sum2 = 0;
  for (int k = 0; k < PER; k++) {
    const unsigned c = count[t * PER + k];
    sum += c;
    sum2 += (c + seg_len - 1) / seg_len;
  }
  part[t] = sum;
  part2[t] = sum2;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    unsigned v = t >= off ? part[t - off] : 0, v2 = t >= off ? part2[t - off] : 0;
    __syncthreads();
    part[t] += v;
    part2[t] += v2;
    __syncthreads();
  }
  unsigned run = part[t] - sum, run2 = part2[t] - sum2;
  for (int k = 0; k < PER; k++) {
    const unsigned c = count[t * PER + k];   // second pass over this thread's 48 counts (L1 resident)
    count[t * PER + k] = 0;
    start[t * PER + k] = run;
    seg_first[t * PER + k] = run2;
    run += c;
    run2 += (c + seg_len - 1) / seg_len;
  }
  if (t == 1023) {
    start[MSM_B] = run;
    seg_first[MSM_B] = run2;
  }
}

// segment table: seg_start[s] = first position of segment s in the index list, seg_scalar[s] = the bucket's scalar
// digit << (MSM_C * window) as a 32-byte record {digit: 2 bytes big-endian, g[k] = (window > k) for k < MSM_W - 1}.
// One thread per bucket.
__global__ void msm_segments_kernel(const unsigned* __restrict__ start, const unsigned* __restrict__ seg_first,
                                    unsigned seg_len, unsigned* __restrict__ seg_start, uint8_t* __restrict__ seg_scalar) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= MSM_B) return;
  const unsigned s0 = seg_first[b], s1 = seg_first[b + 1];
  const int w = b >> MSM_C;
  const unsigned d = (unsigned)(b & ((1 << MSM_C) - 1));
  for (unsigned s = s0; s < s1; s++) {
    seg_start[s] = start[b] + (s - s0) * seg_len;
    // the record the g?_bscale program reads (programs/curve.py: build_bucket_scale)
    uint8_t* o = seg_scalar + (size_t)s * 32;
    o[0] = (uint8_t)(d >> 8);
    o[1] = (uint8_t)d;
    for (int k = 0; k < 30; k++) o[2 + k] = (k < MSM_W - 1 && w > k) ? 1 : 0;
  }
  if (b == MSM_B - 1) seg_start[s1] = start[MSM_B];
}

__global__ void msm_scatter_kernel(const uint8_t* __restrict__ scalars, const unsigned* __restrict__ start,
                                   unsigned* __restrict__ cursor, unsigned* __restrict__ idx, long long n) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * MSM_W) return;
  const long long i = t / MSM_W;
  const int w = (int)(t % MSM_W);
  const unsigned d = msm_digit(scalars + i * 32, w);
  if (!d) return;
  const unsigned b = ((unsigned)w << MSM_C) + d;
  idx[start[b] + atomicAdd(cursor + b, 1u)] = (unsigned)i;
}

int msm_dev(bool g2, const void* pts, const void* scalars, void* out, size_t n) {
  const size_t w = g2 ? 192 : 96;
  const char* mul = g2 ? "g2_mul" : "g1_mul";
  if (n >= 0xffffffffull / MSM_W) return fail(B200BLS_E_ARG, "msm: too many points");
  if (n < MSM_MIN_N) {  // per-point ladder, then the reduction
    if (n == 0) return sum_dev(g2, pts, out, 0);
    int rc = ensure(MSM_SEG_SUMS, w * n);
    if (rc) return rc;
    VmBuf b[3] = {vb(pts, (long long)w), vb(scalars, 32), vb(dbuf(MSM_SEG_SUMS), (long long)w)};
    rc = launch_named(mul, n, b, 3);
    if (rc) return rc;
    return sum_dev(g2, dbuf(MSM_SEG_SUMS), out, n);
  }
  // longest run one thread folds: the mean bucket size plus seven standard deviations, so that
  // uniformly distributed digits are never cut and skewed ones are spread over many threads
  const double mean = (double)n / (1 << MSM_C);
  const unsigned seg_len = (unsigned)(mean + 7.0 * sqrt(mean) + 16.0);
  const long long pairs = (long long)n * MSM_W;
  const size_t seg_cap = (size_t)MSM_B + (size_t)(pairs / seg_len) + 1;     // upper bound on the number of segments
  int rc = ensure(MSM_SEG_SUMS, w * seg_cap);                                  // segment sums
  if (!rc) rc = ensure(MSM_COUNT, sizeof(unsigned) * (size_t)MSM_B);        // counts / cursors
  if (!rc) rc = ensure(MSM_OFFSETS, sizeof(unsigned) * 2 * ((size_t)MSM_B + 1));  // bucket offsets, segment counts
  if (!rc) rc = ensure(MSM_IDX, sizeof(unsigned) * (size_t)pairs);        // point indices grouped by bucket
  if (!rc) rc = ensure(MSM_SEGMENTS, (size_t)36 * (seg_cap + 1));             // segment offsets + scalars
  if (!rc) rc = ensure(MSM_SCALED, w * seg_cap);                            // segment sums times bucket scalars
  if (rc) return rc;
  StreamCtx& sc = cur();
  unsigned* count = (unsigned*)dbuf(MSM_COUNT);
  unsigned* start = (unsigned*)dbuf(MSM_OFFSETS);
  unsigned* seg_first = start + MSM_B + 1;
  unsigned* idx = (unsigned*)dbuf(MSM_IDX);
  unsigned* seg_start = (unsigned*)dbuf(MSM_SEGMENTS);
  uint8_t* seg_scalar = (uint8_t*)(seg_start + ((seg_cap + 1 + 7) & ~(size_t)7));
  const unsigned pair_grid = (unsigned)((pairs + 255) / 256);
  CU(cudaMemsetAsync(count, 0, sizeof(unsigned) * MSM_B, STREAM));
  msm_count_kernel<<<pair_grid, 256, 0, STREAM>>>((const uint8_t*)scalars, count, (long long)n);
  msm_scan_kernel<<<1, 1024, 0, STREAM>>>(count, start, seg_first, seg_len);
  msm_scatter_kernel<<<pair_grid, 256, 0, STREAM>>>((const uint8_t*)scalars, start, count, idx, (long long)n);
  msm_segments_kernel<<<(MSM_B + 255) / 256, 256, 0, STREAM>>>(start, seg_first, seg_len, seg_start, seg_scalar);
  CU(cudaGetLastError());
  g_ctx.launches += 4;
  unsigned n_seg = 0;
  CU(cudaMemcpyAsync(&n_seg, seg_first + MSM_B, sizeof(unsigned), cudaMemcpyDeviceToHost, STREAM));
  CU(cudaStreamSynchronize(STREAM));
  if (n_seg == 0) return sum_dev(g2, pts, out, 0);  // every scalar is zero
  if (n_seg > seg_cap) return fail(B200BLS_E_CUDA, "msm: segment count %u exceeds its bound %zu", n_seg, seg_cap);
  // every point is read once per window: convert it to Montgomery limbs once (SoA copy), not MSM_W times in the fold
  rc = ensure(MSM_MONT, w * n);
  if (rc) return rc;
  VmBuf bt[2] = {vb(pts, (long long)w), vb(dbuf(MSM_MONT), (long long)n)};
  rc = launch_named(g2 ? "g2_tomont" : "g1_tomont", n, bt, 2);
  if (rc) return rc;
  const DevProgram* fold = find_program(g2 ? "g2_bucketr" : "g1_bucketr", n_seg);
  if (!fold) return B200BLS_E_PROGRAM;
  SegArgs seg = {seg_start, idx};
  VmBuf bf[2] = {vb(dbuf(MSM_MONT), (long long)n), vb(dbuf(MSM_SEG_SUMS), (long long)w)};
  rc = launch_program(*fold, n_seg, bf, 2, 0, &seg);
  if (rc) return rc;
  VmBuf bm[3] = {vb(dbuf(MSM_SEG_SUMS), (long long)w), vb(seg_scalar, 32), vb(dbuf(MSM_SCALED), (long long)w)};
  rc = launch_named(g2 ? "g2_bscale" : "g1_bscale", n_seg, bm, 3);
  if (rc) return rc;
  return sum_dev(g2, dbuf(MSM_SCALED), out, n_seg);
}

// ---- multi-pairing: Miller loops -> raw Fq12 per item -> product tree ------------------------
// out576: big-endian product of the Miller values (not final-exponentiated)
// product of the n raw Miller values in buffer MILLER_RAW -> out576 (big-endian, not final-exponentiated)
int raw_product_dev(void* out576, size_t n) {
  const DevProgram* p1 = find_program("f12_prod1", n);
  if (!p1) return B200BLS_E_PROGRAM;
  int grid = grid_of(*p1, n);
  int rc = ensure(PROD_PARTS, (size_t)576 * grid);
  if (rc) return rc;
  VmBuf bb[2] = {vb(dbuf(MILLER_RAW), (long long)n), vb(dbuf(PROD_PARTS), grid)};
  rc = launch_program(*p1, n, bb, 2, grid);
  if (rc) return rc;
  VmBuf bc[2] = {vb(dbuf(PROD_PARTS), grid), vb(out576, 576)};
  return launch_named("f12_prod2", (size_t)grid, bc, 2, 1);
}

// the Fq12 one (big-endian) -> out576: the empty product
int fq12_one_dev(void* out576) {
  static const uint8_t kOne[48] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                   0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1};
  CU(cudaMemsetAsync(out576, 0, 576, STREAM));
  CU(cudaMemcpyAsync(out576, kOne, 48, cudaMemcpyHostToDevice, STREAM));
  return 0;
}

int miller_product_dev(const void* P, const void* Q, void* out576, size_t n) {
  if (n == 0) return fq12_one_dev(out576);   // fields_t.py:1117: prod starts at one
  int rc = ensure(MILLER_RAW, (size_t)576 * n);
  if (rc) return rc;
  VmBuf ba[3] = {vb(P, 96), vb(Q, 192), vb(dbuf(MILLER_RAW), (long long)n)};
  rc = launch_named("miller_raw", n, ba, 3);
  if (rc) return rc;
  return raw_product_dev(out576, n);
}

// the final exponentiation of the Miller product: prod_i e(P_i, Q_i) -> out576
int pairing_multi_dev(const void* P, const void* Q, void* out576, size_t n) {
  int rc = ensure(MULTI_PRODUCT, 576);
  if (!rc) rc = miller_product_dev(P, Q, dbuf(MULTI_PRODUCT), n);
  if (rc) return rc;
  VmBuf b[2] = {vb(dbuf(MULTI_PRODUCT), 576), vb(out576, 576)};
  return launch_named("final_exp", 1, b, 2);
}

// ---- batched multi-pairing: ragged groups of pairs, one product and one final exponentiation per group ---------------
// What the host reads back after the scan: whether the offsets are valid, the number of pairs, the chunks of each pass.
struct MultiHeader {
  uint32_t bad;
  uint32_t chunks[kMultiMaxPasses];
  uint32_t pad;
  uint64_t total;
};
constexpr size_t kMultiHeaderBytes = 64;
static_assert(sizeof(MultiHeader) <= kMultiHeaderBytes, "multi-pairing header");

// One block: validates the n + 1 offsets and writes the prefix tables of every pass (multi_plan.h).  Thread t owns a
// contiguous range of groups: their chunk counts, a scan over the threads' sums per pass, then the table entries.
__global__ void __launch_bounds__(1024) multi_scan_kernel(const uint64_t* __restrict__ off, unsigned long long n,
                                                          uint32_t* __restrict__ prefix, MultiHeader* __restrict__ hdr) {
  __shared__ uint32_t part[kMultiMaxPasses][1024];
  __shared__ int s_bad;
  const int t = threadIdx.x;
  if (t == 0) s_bad = 0;
  __syncthreads();
  const unsigned long long per = (n + 1023) / 1024;
  const unsigned long long g0 = min(n, (unsigned long long)t * per), g1 = min(n, g0 + per);
  uint32_t sum[kMultiMaxPasses] = {}, cnt[kMultiMaxPasses];
  bool bad = t == 0 && (off[0] != 0 || off[n] > kMultiMaxPairs);
  for (unsigned long long g = g0; g < g1; g++) {
    const uint64_t a = off[g], b = off[g + 1];
    bad = bad || b < a;
    multi_group_chunks(b - a, cnt);
#pragma unroll
    for (int r = 0; r < kMultiMaxPasses; r++) sum[r] += cnt[r];
  }
  if (bad) s_bad = 1;
#pragma unroll
  for (int r = 0; r < kMultiMaxPasses; r++) part[r][t] = sum[r];
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {
    uint32_t v[kMultiMaxPasses];
#pragma unroll
    for (int r = 0; r < kMultiMaxPasses; r++) v[r] = t >= d ? part[r][t - d] : 0;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kMultiMaxPasses; r++) part[r][t] += v[r];
    __syncthreads();
  }
  uint32_t run[kMultiMaxPasses];
#pragma unroll
  for (int r = 0; r < kMultiMaxPasses; r++) run[r] = part[r][t] - sum[r];
  for (unsigned long long g = g0; g < g1; g++) {
    multi_group_chunks(off[g + 1] - off[g], cnt);
#pragma unroll
    for (int r = 0; r < kMultiMaxPasses; r++) {
      prefix[r * (n + 1) + g] = run[r];
      run[r] += cnt[r];
    }
  }
  if (t == 1023) {
#pragma unroll
    for (int r = 0; r < kMultiMaxPasses; r++) {
      prefix[r * (n + 1) + n] = run[r];
      hdr->chunks[r] = run[r];
    }
    hdr->total = off[n];
    hdr->bad = (uint32_t)s_bad;
  }
}

// the segment starts of pass r, one thread per group, and (n_idx > 0) the index list idx[i] = i for i < n_idx
__global__ void multi_tables_kernel(int r, const uint64_t* __restrict__ off, unsigned long long n,
                                    const uint32_t* __restrict__ prefix, uint32_t* __restrict__ seg_start,
                                    uint32_t* __restrict__ idx, unsigned long long n_idx) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) multi_segments_group(r, t, n, off, prefix, seg_start);
  if (t < n_idx) idx[t] = (uint32_t)t;
}

// n_groups products prod_{j in [off[g], off[g + 1])} e(P_j, Q_j) -> out: 576 bytes each (check = false) or one byte,
// 1 iff the product is one (check = true).  Offsets that are not valid (multi_offsets_bad) are refused before any
// program runs; the one host synchronisation reads the scan's header.
int pairing_multi_batch_dev(bool check, const void* P, const void* Q, const uint64_t* off, size_t n_groups, void* out) {
  if (n_groups == 0) return 0;
  if (n_groups > kMultiMaxGroups) return fail(B200BLS_E_ARG, "pairing_multi_batch: more than 2^31 - 1 groups");
  const size_t n = n_groups, rows = (size_t)kMultiMaxPasses * (n + 1);
  int rc = ensure(MULTI_TABLES, kMultiHeaderBytes + sizeof(uint32_t) * rows);
  if (rc) return rc;
  MultiHeader* dhdr = (MultiHeader*)dbuf(MULTI_TABLES);
  uint32_t* prefix = (uint32_t*)((uint8_t*)dhdr + kMultiHeaderBytes);
  multi_scan_kernel<<<1, 1024, 0, STREAM>>>(off, n, prefix, dhdr);
  CU(cudaGetLastError());
  g_ctx.launches++;
  MultiHeader h;
  CU(cudaMemcpyAsync(&h, dhdr, sizeof(h), cudaMemcpyDeviceToHost, STREAM));
  CU(cudaStreamSynchronize(STREAM));
  if (h.bad)
    return fail(B200BLS_E_ARG, "pairing_multi_batch: offsets must start at 0, never decrease and hold at most 2^32 - 1 "
                               "pairs");
  const size_t total = (size_t)h.total, c0 = h.chunks[0];
  const int passes = multi_passes(h.chunks, n);
  const size_t n_idx = total > c0 ? total : c0;
  rc = ensure(MILLER_RAW, (size_t)576 * (total ? total : 1));
  if (!rc) rc = ensure(MULTI_SEG, sizeof(uint32_t) * (c0 + 1));
  if (!rc) rc = ensure(MULTI_IDX, sizeof(uint32_t) * n_idx);
  if (!rc && passes > 1) rc = ensure(MULTI_PARTS, (size_t)576 * c0);
  if (!rc && passes > 2) rc = ensure(MULTI_PARTS2, (size_t)576 * h.chunks[1]);
  if (!rc) rc = ensure(MULTI_FINAL, (size_t)576 * n);
  if (rc) return rc;
  if (total) {
    VmBuf bm[3] = {vb(P, 96), vb(Q, 192), vb(dbuf(MILLER_RAW), (long long)total)};
    if ((rc = launch_named("miller_raw", total, bm, 3))) return rc;
  }
  uint32_t* seg_start = (uint32_t*)dbuf(MULTI_SEG);
  uint32_t* idx = (uint32_t*)dbuf(MULTI_IDX);
  VmBuf in = vb(dbuf(MILLER_RAW), (long long)total);
  for (int r = 0; r < passes; r++) {
    const size_t chunks = h.chunks[r], threads = r == 0 && n_idx > n ? n_idx : n;
    multi_tables_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, STREAM>>>(r, off, n, prefix, seg_start, idx,
                                                                               r == 0 ? n_idx : 0);
    CU(cudaGetLastError());
    g_ctx.launches++;
    const bool last = r + 1 == passes;
    const DevProgram* pr = find_program(last ? "f12_prodseg_be" : "f12_prodseg", chunks);
    if (!pr) return B200BLS_E_PROGRAM;
    const VmBuf res = last ? vb(dbuf(MULTI_FINAL), 576) : vb(dbuf(r % 2 ? MULTI_PARTS2 : MULTI_PARTS), (long long)chunks);
    VmBuf bp[2] = {in, res};
    SegArgs seg = {seg_start, idx};
    if ((rc = launch_program(*pr, chunks, bp, 2, 0, &seg))) return rc;
    in = res;
  }
  VmBuf bf[2] = {vb(dbuf(MULTI_FINAL), 576), vb(out, check ? 1 : 576)};
  return launch_named(check ? "final_exp_check" : "final_exp", n, bf, 2);
}

int sha_stage_dev(const void* hashes, void* out256, size_t n);

// Miller product of aggregate verification over m = n + 1 items in ONE launch: item 0 is the pair
// (-G1, signature), given explicitly in Qgiven; items 1..n are (pk_i, H(mh_i)), hashed and paired
// in the same program with H projective.  P: m x 96, mh: m x 32 (item 0 unused), Qgiven: m x 192
// (used where given[i] != 0), given: m bytes.
int aggregate_miller_dev(const void* P, const void* mh, const void* Qgiven, const void* given, void* out576, size_t m) {
  int rc = ensure(MILLER_RAW, (size_t)576 * m);
  if (!rc) rc = ensure(SHA_OUT, (size_t)256 * m);
  if (rc) return rc;
  rc = sha_stage_dev(mh, dbuf(SHA_OUT), m);
  if (rc) return rc;
  VmBuf bb[5] = {vb(P, 96), vb(dbuf(SHA_OUT), 256), vb(dbuf(MILLER_RAW), (long long)m), vb(Qgiven, 192),
                 vb(given, 1)};
  rc = launch_named("miller_hash_raw", m, bb, 5);
  if (rc) return rc;
  return raw_product_dev(out576, m);
}

int sha_stage_dev(const void* hashes, void* out256, size_t n) {
  long long threads = (long long)n * 8;
  int block = 256;
  long long grid = (threads + block - 1) / block;
  sha_stage_kernel<<<(unsigned)grid, block, 0, STREAM>>>((const uint8_t*)hashes, (uint8_t*)out256, (long long)n);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

// aggregation exponents T_i = H(i || pk_hash) mod n for i in [first, first + n) (util.py:46-49)
int hash_pks_dev(const void* pk_hash32, uint32_t first, void* out, size_t n) {
  if (n == 0) return 0;
  int block = 256;
  long long grid = ((long long)n + block - 1) / block;
  hash_pks_kernel<<<(unsigned)grid, block, 0, STREAM>>>((const uint8_t*)pk_hash32, first, (uint8_t*)out, (long long)n);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

int hash_to_g2_dev(const void* hashes, void* out, size_t n) {
  if (n == 0) return 0;
  int rc = ensure(SHA_OUT, (size_t)256 * n);
  if (rc) return rc;
  rc = sha_stage_dev(hashes, dbuf(SHA_OUT), n);
  if (rc) return rc;
  VmBuf b[2] = {vb(dbuf(SHA_OUT), 256), vb(out, 192)};
  return launch_named("hash_to_g2", n, b, 2);
}

int verify_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n) {
  if (n == 0) return 0;
  // SHA stage, then ONE program that hashes to G2 and verifies: the hashed point enters the Miller
  // loop projective, its to_affine inversion is never computed
  int rc = ensure(SHA_OUT, (size_t)256 * n);
  if (rc) return rc;
  rc = sha_stage_dev(mh, dbuf(SHA_OUT), n);
  if (rc) return rc;
  VmBuf b[4] = {vb(pk, 96), vb(dbuf(SHA_OUT), 256), vb(sig, 192), vb(ok, 1)};
  return launch_named("verify_full", n, b, 4);
}

// one flag byte per affine point from a g?_subgroup-style program (programs/curve.py: build_subgroup_check)
int point_flags_dev(const char* program, bool g2, const void* pts, void* ok, size_t n) {
  if (n == 0) return 0;
  VmBuf b[2] = {vb(pts, g2 ? 192 : 96), vb(ok, 1)};
  return launch_named(program, n, b, 2);
}

// ok[i] = 1 iff point i is on the curve and in G1 / G2 (Curve.in_subgroup; infinity counts as a member)
int subgroup_check_dev(bool g2, const void* pts, void* ok, size_t n) {
  return point_flags_dev(g2 ? "g2_subgroup" : "g1_subgroup", g2, pts, ok, n);
}

struct FlagList {
  const uint8_t* f[4];
  int n;
};

// ok[i] &= byte i of every flag array
__global__ void and_flags_kernel(uint8_t* __restrict__ ok, FlagList fl, long long n) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  bool v = ok[t] != 0;
#pragma unroll
  for (int i = 0; i < 4; i++)
    if (i < fl.n) v = v && fl.f[i][t];
  ok[t] = v ? 1 : 0;
}

int and_flags_dev(void* ok, const FlagList& fl, size_t n) {
  and_flags_kernel<<<(unsigned)((n + 255) / 256), 256, 0, STREAM>>>((uint8_t*)ok, fl, (long long)n);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

// strict verification: "pk in G1 and not infinity" (g1_keyvalidate, decided on the coordinates reduced mod q as the
// pairing reads them) and "sig in G2" for the affine keys and signatures into buffer STRICT_FLAGS, appended to fl
int strict_flags_dev(const void* pk, const void* sig, size_t n, FlagList& fl) {
  int rc = ensure(STRICT_FLAGS, 2 * n);
  if (rc) return rc;
  uint8_t* f = (uint8_t*)dbuf(STRICT_FLAGS);
  rc = point_flags_dev("g1_keyvalidate", false, pk, f, n);
  if (!rc) rc = subgroup_check_dev(true, sig, f + n, n);
  fl.f[fl.n++] = f;
  fl.f[fl.n++] = f + n;
  return rc;
}

// strict: the verdict AND-ed with "pk in G1, pk not infinity, sig in G2" (b200bls.h)
int verify_strict_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n) {
  if (n == 0) return 0;
  int rc = verify_dev(pk, mh, sig, ok, n);
  FlagList fl = {};
  if (!rc) rc = strict_flags_dev(pk, sig, n, fl);
  if (rc) return rc;
  return and_flags_dev(ok, fl, n);
}

// verification straight from the wire formats: PublicKey.from_bytes (keys.py:29-40) and
// Signature.from_bytes (signature.py:22-38) on the device, then the pairing check; a key or
// signature that does not decode (the reference raises ValueError) counts as a rejection.
// strict: the subgroup checks of verify_strict_dev on the decoded points as well.
int verify_wire_dev(const void* pk48, const void* mh, const void* sig96, void* ok, size_t n, bool strict = false) {
  if (n == 0) return 0;
  int rc = ensure(WIRE_PK, (size_t)96 * n);
  if (!rc) rc = ensure(WIRE_SIG, (size_t)192 * n);
  if (!rc) rc = ensure(WIRE_PK_OK, n);
  if (!rc) rc = ensure(WIRE_SIG_OK, n);
  if (rc) return rc;
  StreamCtx& sc = cur();
  VmBuf b1[3] = {vb(pk48, 48), vb(dbuf(WIRE_PK), 96), vb(dbuf(WIRE_PK_OK), 1)};
  rc = launch_named("g1_decompress", n, b1, 3);
  if (rc) return rc;
  VmBuf b2[3] = {vb(sig96, 96), vb(dbuf(WIRE_SIG), 192), vb(dbuf(WIRE_SIG_OK), 1)};
  rc = launch_named("g2_decompress", n, b2, 3);
  if (rc) return rc;
  rc = verify_dev(dbuf(WIRE_PK), mh, dbuf(WIRE_SIG), ok, n);
  if (rc) return rc;
  FlagList fl = {{(const uint8_t*)dbuf(WIRE_PK_OK), (const uint8_t*)dbuf(WIRE_SIG_OK)}, 2};
  if (strict) {
    rc = strict_flags_dev(dbuf(WIRE_PK), dbuf(WIRE_SIG), n, fl);
    if (rc) return rc;
  }
  return and_flags_dev(ok, fl, n);
}

// x bytes of each affine point with (flag << 7) OR-ed into byte 0 (bls_py/ec.py:103-111)
__global__ void compress_pack_kernel(const uint8_t* __restrict__ aff, const uint8_t* __restrict__ flag,
                                     uint8_t* __restrict__ out, long long n, int xbytes) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long words = (long long)xbytes / 4;
  if (t >= n * words) return;
  long long item = t / words;
  int wi = (int)(t % words);
  uint32_t v = reinterpret_cast<const uint32_t*>(aff + item * 2 * xbytes)[wi];
  if (wi == 0 && flag[item]) v |= 0x80u;  // byte 0 is the low byte of the first little-endian word
  reinterpret_cast<uint32_t*>(out + item * xbytes)[wi] = v;
}

// the compressed points from the affine points and their flags; xb = 48 (G1) or 96 (G2)
int pack_dev(const void* aff, const void* flag, void* out, size_t n, int xb) {
  long long threads = (long long)n * (xb / 4);
  compress_pack_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, STREAM>>>(
      (const uint8_t*)aff, (const uint8_t*)flag, (uint8_t*)out, (long long)n, xb);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

int compress_dev(bool g2, const void* aff, void* out, size_t n) {
  if (n == 0) return 0;
  int rc = ensure(CFLAGS, n);
  if (rc) return rc;
  int xb = g2 ? 96 : 48;
  VmBuf b[2] = {vb(aff, 2 * xb), vb(dbuf(CFLAGS), 1)};
  rc = launch_named(g2 ? "g2_cflag" : "g1_cflag", n, b, 2);
  if (rc) return rc;
  return pack_dev(aff, dbuf(CFLAGS), out, n, xb);
}

// ---- signing and public keys (PrivateKey.sign_prehashed / get_public_key, keys.py:119-132) ------------------------
// sk (n x 32 bytes big-endian, any value) -> the digit records of the g2_sign / g1_pubkey ladders, one thread each
__global__ void scalar_split_kernel(const uint8_t* __restrict__ sk, uint8_t* __restrict__ out, long long n) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  scalar_split(sk + t * 32, out + t * 32);
}

int split_dev(const void* sk, void* digits, size_t n) {
  scalar_split_kernel<<<(unsigned)((n + 255) / 256), 256, 0, STREAM>>>((const uint8_t*)sk, (uint8_t*)digits,
                                                                        (long long)n);
  CU(cudaGetLastError());
  g_ctx.launches++;
  return 0;
}

// zeroes a device copy of secret data once the work enqueued before it has read it; keeps the first error
int wipe(int rc, void* p, size_t bytes) {
  if (!bytes) return rc;
  cudaError_t e = cudaMemsetAsync(p, 0, bytes, STREAM);
  if (!rc && e != cudaSuccess) return fail(B200BLS_E_CUDA, "wiping secret data failed: %s", cudaGetErrorString(e));
  return rc;
}

// split, then `program` on {extra..., digits, affine out, flags}, then (wire) the compression pack; the digits are
// zeroed after the program whatever happens
int digits_pipeline(const char* program, bool g2, bool wire, const void* sk, const VmBuf* extra, int n_extra, void* out,
                    size_t n) {
  const size_t w = g2 ? 192 : 96;
  int rc = ensure(SIGN_DIGITS, 32 * n);
  if (!rc) rc = ensure(SIGN_FLAGS, n);
  if (!rc && wire) rc = ensure(SIGN_AFFINE, w * n);
  if (rc) return rc;
  void* aff = wire ? dbuf(SIGN_AFFINE) : out;
  rc = split_dev(sk, dbuf(SIGN_DIGITS), n);
  if (!rc) {
    VmBuf b[VM_MAX_BUFS];
    for (int i = 0; i < n_extra; i++) b[i] = extra[i];
    b[n_extra] = vb(dbuf(SIGN_DIGITS), 32);
    b[n_extra + 1] = vb(aff, (long long)w);
    b[n_extra + 2] = vb(dbuf(SIGN_FLAGS), 1);
    rc = launch_named(program, n, b, n_extra + 3);
  }
  rc = wipe(rc, dbuf(SIGN_DIGITS), 32 * n);
  if (rc || !wire) return rc;
  return pack_dev(aff, dbuf(SIGN_FLAGS), out, n, (int)w / 2);
}

// sk_i * H(mh_i): the SHA stage, the split, g2_sign (hash, psi-split ladder, to_affine, flag), the pack
int sign_dev(bool wire, const void* sk, const void* mh, void* sig, size_t n) {
  if (n == 0) return 0;
  int rc = ensure(SHA_OUT, (size_t)256 * n);
  if (!rc) rc = sha_stage_dev(mh, dbuf(SHA_OUT), n);
  if (rc) return rc;
  VmBuf sha = vb(dbuf(SHA_OUT), 256);
  return digits_pipeline("g2_sign", true, wire, sk, &sha, 1, sig, n);
}

// sk_i * G1: the split, g1_pubkey (fixed-base ladder, to_affine, flag), the pack
int public_key_dev(bool wire, const void* sk, void* pk, size_t n) {
  if (n == 0) return 0;
  return digits_pipeline("g1_pubkey", false, wire, sk, nullptr, 0, pk, n);
}

const char* kFieldOps[] = {"add", "sub", "mul", "sqr", "neg", "inv"};

int field_prog_name(int level, int op, char* out, size_t cap) {
  if (!(level == 1 || level == 2 || level == 6 || level == 12) || op < 0 || op > 5)
    return fail(B200BLS_E_ARG, "field_op: bad level %d or op %d", level, op);
  snprintf(out, cap, "f%d_%s", level, kFieldOps[op]);
  return 0;
}

}  // namespace

extern "C" {

const char* b200bls_last_error(void) { return g_err; }

int b200bls_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  Context& c = g_ctx;
  if (c.ready) {
    if (c.device == device) return 0;
    return fail(B200BLS_E_ARG, "already initialised on device %d", c.device);
  }
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(B200BLS_E_CUDA, "no CUDA device available (%s); this library has no CPU path",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return fail(B200BLS_E_ARG, "device %d out of range (0..%d)", device, n_dev - 1);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  c.policy.sm_count = prop.multiProcessorCount;
  for (auto& sc : c.sc) {
    CU(cudaStreamCreateWithFlags(&sc.stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&sc.done, cudaEventDisableTiming));
    CU(cudaMalloc(&sc.counters, N_COUNTERS * sizeof(int)));
  }
  CU(cudaEventCreate(&c.ev0));
  CU(cudaEventCreate(&c.ev1));
  {
    unsigned tab[16 + 2 * 17];
    for (unsigned i = 0; i < 16; i++) tab[i] = i;
    for (unsigned n = 0; n <= 16; n++) {
      tab[16 + 2 * n] = 0;
      tab[16 + 2 * n + 1] = n;
    }
    CU(cudaMalloc(&c.tiny_seg, sizeof(tab)));
    CU(cudaMemcpy(c.tiny_seg, tab, sizeof(tab), cudaMemcpyHostToDevice));
  }
  CU(vm1_configure());
  CU(vm2_configure());
  CU(vm3_configure());
  // parse the embedded program blob
  const unsigned char* blob = _binary_programs_bin_start;
  size_t blob_len = (size_t)(_binary_programs_bin_end - _binary_programs_bin_start);
  uint32_t blob_version = 0;
  if (blob_len >= 16) memcpy(&blob_version, blob + 8, 4);
  if (blob_len < 16 || memcmp(blob, "B2BLSPRG", 8) != 0 || blob_version != 2)
    return fail(B200BLS_E_PROGRAM, "bad program blob");
  uint32_t n_prog;
  memcpy(&n_prog, blob + 12, 4);
  for (uint32_t i = 0; i < n_prog; i++) {
    BlobEntry en;
    memcpy(&en, blob + 16 + i * sizeof(BlobEntry), sizeof(en));
    if (en.shape < 1 || en.shape > N_SHAPES) return fail(B200BLS_E_PROGRAM, "bad program blob: shape %u", en.shape);
    DevProgram dp;
    dp.n_ins = (int)en.n_ins;
    dp.body_start = (int)en.body_start;
    dp.epi_start = (int)en.epi_start;
    dp.n_slots = (int)en.n_slots;
    dp.n_cold = (int)en.n_cold;
    dp.n_tmem = (int)en.n_tmem;
    dp.shape = (int)en.shape;
    {
      const unsigned char* code = blob + en.code_off;
      for (uint32_t k = 0; k < en.n_ins; k++) {
        const int op = code[8 * k];
        if (op == OP_SYNC || op == OP_XMOV2 || op == OP_STRAWB2) dp.cross_thread = true;
      }
    }
    size_t code_bytes = (size_t)(en.n_ins + 1) * sizeof(uint2);
    size_t const_bytes = (size_t)en.n_consts * 3 * sizeof(uint4);
    // 64 instructions of slack: the interpreter prefetches the instruction stream two L1 lines ahead
    CU(cudaMalloc(&dp.code, code_bytes + 64 * sizeof(uint2)));
    CU(cudaMemset(dp.code, 0, code_bytes + 64 * sizeof(uint2)));
    CU(cudaMalloc(&dp.consts, const_bytes));
    CU(cudaMemcpy(dp.code, blob + en.code_off, code_bytes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dp.consts, blob + en.consts_off, const_bytes, cudaMemcpyHostToDevice));
    char nm[33];
    memcpy(nm, en.name, 32);
    nm[32] = 0;
    c.programs[nm] = dp;
  }
  const char* kenv = getenv("B200BLS_KERNEL");
  if (kenv && kenv[0] >= '0' && kenv[0] <= '2') c.policy.kernel = kenv[0] - '0';
  const char* env = getenv("B200BLS_CTAS_PER_SM");
  if (env && env[0] >= '0' && env[0] <= '5') c.policy.ctas_per_sm = env[0] - '0';
  c.device = device;
  c.ready = true;
  return 0;
}

void b200bls_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  Context& c = g_ctx;
  if (!c.ready) return;
  for (auto& sc : c.sc) cudaStreamSynchronize(sc.stream);
  for (auto& kv : c.programs) {
    cudaFree(kv.second.code);
    cudaFree(kv.second.consts);
  }
  c.programs.clear();
  for (auto& sc : c.sc) {
    for (auto& s : sc.bufs) {
      if (s.ptr) cudaFree(s.ptr);
      s = Staging();
    }
    if (sc.cold) cudaFree(sc.cold);
    sc.cold = nullptr;
    sc.cold_bytes = 0;
    cudaFree(sc.counters);
    cudaEventDestroy(sc.done);
    cudaStreamDestroy(sc.stream);
  }
  cudaEventDestroy(c.ev0);
  cudaEventDestroy(c.ev1);
  if (c.tiny_seg) cudaFree(c.tiny_seg);
  c.tiny_seg = nullptr;
  c.ready = false;
  c.device = -1;
}

int b200bls_sm_count(void) { return g_ctx.ready ? g_ctx.policy.sm_count : 0; }

int b200bls_set_ctas_per_sm(int n) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (n < 0 || n > 5)
    return fail(B200BLS_E_ARG, "ctas_per_sm must be 0 (auto), 1, 2, 3, 4 (one CTA of 384 threads) or 5 (one of 512)");
  g_ctx.policy.ctas_per_sm = n;
  return 0;
}

int b200bls_get_ctas_per_sm(void) { return g_ctx.policy.ctas_per_sm; }

int b200bls_sync(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "not initialised");
  for (auto& sc : g_ctx.sc) CU(cudaStreamSynchronize(sc.stream));
  return 0;
}

int b200bls_set_stream(int idx) {
  if (idx < 0 || idx >= N_STREAMS) return fail(B200BLS_E_ARG, "stream index out of range (0..%d)", N_STREAMS - 1);
  t_stream = idx;   // per calling thread
  return 0;
}

int b200bls_stream_count(void) { return N_STREAMS; }

void* b200bls_malloc(size_t bytes) {
  if (!g_ctx.ready) {
    fail(B200BLS_E_NOT_INIT, "not initialised");
    return nullptr;
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    fail(B200BLS_E_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return nullptr;
  }
  return p;
}

void b200bls_free(void* p) {
  if (p) cudaFree(p);
}

void* b200bls_host_alloc(size_t bytes) {
  if (!g_ctx.ready) {
    fail(B200BLS_E_NOT_INIT, "not initialised");
    return nullptr;
  }
  void* p = nullptr;
  cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    fail(B200BLS_E_NOMEM, "cudaMallocHost(%zu): %s", bytes, cudaGetErrorString(e));
    return nullptr;
  }
  return p;
}

void b200bls_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int b200bls_h2d(void* dst, const void* src, size_t bytes) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "not initialised");
  CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, STREAM));
  return 0;
}

int b200bls_d2h(void* dst, const void* src, size_t bytes) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "not initialised");
  CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, STREAM));
  return 0;
}

// The timed region covers ALL library streams: every stream waits for the start event, and
// the stop event is recorded on stream 0 after it has waited for the work of every other one.
int b200bls_timer_start(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "not initialised");
  CU(cudaEventRecord(g_ctx.ev0, g_ctx.sc[0].stream));
  for (int i = 1; i < N_STREAMS; i++) CU(cudaStreamWaitEvent(g_ctx.sc[i].stream, g_ctx.ev0, 0));
  return 0;
}

int b200bls_timer_stop(float* ms) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.ready) return fail(B200BLS_E_NOT_INIT, "not initialised");
  for (int i = 1; i < N_STREAMS; i++) {
    CU(cudaEventRecord(g_ctx.sc[i].done, g_ctx.sc[i].stream));
    CU(cudaStreamWaitEvent(g_ctx.sc[0].stream, g_ctx.sc[i].done, 0));
  }
  CU(cudaEventRecord(g_ctx.ev1, g_ctx.sc[0].stream));
  CU(cudaEventSynchronize(g_ctx.ev1));
  CU(cudaEventElapsedTime(ms, g_ctx.ev0, g_ctx.ev1));
  return 0;
}

uint64_t b200bls_launch_count(void) { return g_ctx.launches; }

int b200bls_run_program_dev(const char* name, size_t n_items, void* const* bufs, const int64_t* strides, int n_bufs) {
  if (n_bufs < 0 || n_bufs > VM_MAX_BUFS) return fail(B200BLS_E_ARG, "n_bufs out of range");
  DevBuf db[VM_MAX_BUFS];
  for (int i = 0; i < n_bufs; i++) {
    db[i].ptr = bufs[i];
    db[i].stride = (size_t)strides[i];
  }
  return locked([&] { return run_dev(name, n_items, db, n_bufs); });
}

int b200bls_program_info(const char* name, int* n_ins, int* n_slots, int* n_cold) {
  return locked([&] {
    const DevProgram* pr = find_program(name);
    if (!pr) return B200BLS_E_PROGRAM;
    if (n_ins) *n_ins = pr->n_ins;
    if (n_slots) *n_slots = pr->n_slots;
    if (n_cold) *n_cold = pr->n_cold;
    return 0;
  });
}

int b200bls_field_op_batch(int level, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  char name[32];
  int rc = field_prog_name(level, op, name, sizeof(name));
  if (rc) return rc;
  if (!a || !out || (op <= 2 && !b)) return fail(B200BLS_E_ARG, "null buffer");
  const size_t w = 48 * (size_t)level;
  return run_host(name, n, {{a, nullptr, w}, {op <= 2 ? b : nullptr, nullptr, w}, {nullptr, out, w}});
}

int b200bls_field_op_batch_dev(int level, int op, const void* a, const void* b, void* out, size_t n) {
  char name[32];
  int rc = field_prog_name(level, op, name, sizeof(name));
  if (rc) return rc;
  size_t w = 48 * (size_t)level;
  DevBuf db[3] = {{a, w}, {b ? b : a, w}, {out, w}};
  return locked([&] { return run_dev(name, n, db, 3); });
}

// ---- single-function parity entry points (programs/extras.py) ------------------------------------------
int b200bls_field_frob_batch(int level, int i, const uint8_t* a, uint8_t* out, size_t n) {
  if (!(level == 2 || level == 6 || level == 12) || i < 0 || i >= level)
    return fail(B200BLS_E_ARG, "field_frob: level %d, power %d (want level 2, 6 or 12 and 0 <= i < level)", level, i);
  if (!a || !out) return fail(B200BLS_E_ARG, "null buffer");
  char name[32];
  snprintf(name, sizeof(name), "f%d_frob%d", level, i);
  const size_t w = 48 * (size_t)level;
  return run_host(name, n, {{a, nullptr, w}, {nullptr, out, w}});
}

int b200bls_field_pow_batch(int level, const uint8_t* a, const uint8_t* e48, uint8_t* out, size_t n) {
  if (!(level == 1 || level == 2 || level == 6 || level == 12)) return fail(B200BLS_E_ARG, "field_pow: bad level %d", level);
  if (!a || !e48 || !out) return fail(B200BLS_E_ARG, "null buffer");
  char name[32];
  snprintf(name, sizeof(name), "f%d_pow", level);
  const size_t w = 48 * (size_t)level;
  return run_host(name, n, {{a, nullptr, w}, {e48, nullptr, 48}, {nullptr, out, w}});
}

int b200bls_field_sqrt_batch(int level, const uint8_t* a, uint8_t* out, uint8_t* ok, size_t n) {
  if (!(level == 1 || level == 2)) return fail(B200BLS_E_ARG, "field_sqrt: level %d (want 1 or 2)", level);
  if (!a || !out || !ok) return fail(B200BLS_E_ARG, "null buffer");
  const size_t w = 48 * (size_t)level;
  return run_host(level == 1 ? "f1_sqrt" : "f2_sqrt", n, {{a, nullptr, w}, {nullptr, out, w}, {nullptr, ok, 1}});
}

int b200bls_jacobian_op_batch(int g2, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  static const char* kOps[4] = {"affine", "dbl", "add", "mul"};
  if (op < 0 || op > 3) return fail(B200BLS_E_ARG, "jacobian_op: op %d (0 to_affine, 1 double, 2 add, 3 scalar mult)", op);
  if (!a || !out || (op >= 2 && !b)) return fail(B200BLS_E_ARG, "null buffer");
  char name[32];
  snprintf(name, sizeof(name), "%s_j%s", g2 ? "g2" : "g1", kOps[op]);
  const size_t w = g2 ? 96 : 48;
  return run_host(name, n, {{a, nullptr, 3 * w}, {op >= 2 ? b : nullptr, nullptr, op == 3 ? (size_t)32 : 3 * w},
                            {nullptr, out, 2 * w}});
}

int b200bls_sw_encode_g2_batch(const uint8_t* t, uint8_t* out, size_t n) {
  if (!t || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("sw_encode_g2", n, {{t, nullptr, 96}, {nullptr, out, 192}});
}

int b200bls_g2_untwist_batch(const uint8_t* pts, uint8_t* out, size_t n) {
  if (!pts || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g2_untwist", n, {{pts, nullptr, 192}, {nullptr, out, 1152}});
}

int b200bls_fq12_twist_batch(const uint8_t* pts, uint8_t* out, size_t n) {
  if (!pts || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("f12_twist", n, {{pts, nullptr, 1152}, {nullptr, out, 1152}});
}

int b200bls_g2_psi_batch(const uint8_t* pts, uint8_t* out, size_t n) {
  if (!pts || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g2_psi", n, {{pts, nullptr, 192}, {nullptr, out, 192}});
}

int b200bls_pairing_batch(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n) {
  if (!P || !Q || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("pairing", n, {{P, nullptr, 96}, {Q, nullptr, 192}, {nullptr, out, 576}});
}

int b200bls_pairing_batch_async(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n) {
  if (!P || !Q || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("pairing", n, {{P, nullptr, 96}, {Q, nullptr, 192}, {nullptr, out, 576}}, true);
}

int b200bls_pairing_batch_dev(const void* P, const void* Q, void* out, size_t n) {
  DevBuf db[3] = {{P, 96}, {Q, 192}, {out, 576}};
  return locked([&] { return run_dev("pairing", n, db, 3); });
}

int b200bls_final_exp_batch(const uint8_t* in, uint8_t* out, size_t n) {
  if (!in || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("final_exp", n, {{in, nullptr, 576}, {nullptr, out, 576}});
}

int b200bls_final_exp_batch_dev(const void* in, void* out, size_t n) {
  DevBuf db[2] = {{in, 576}, {out, 576}};
  return locked([&] { return run_dev("final_exp", n, db, 2); });
}

int b200bls_miller_loop_batch(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n) {
  if (!P || !Q || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("miller_loop", n, {{P, nullptr, 96}, {Q, nullptr, 192}, {nullptr, out, 576}});
}

int b200bls_miller_loop_batch_dev(const void* P, const void* Q, void* out, size_t n) {
  DevBuf db[3] = {{P, 96}, {Q, 192}, {out, 576}};
  return locked([&] { return run_dev("miller_loop", n, db, 3); });
}


// ---- curve ---------------------------------------------------------------------------------
int b200bls_g1_scalar_mul_batch(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n) {
  if (!pts || !scalars || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g1_mul", n, {{pts, nullptr, 96}, {scalars, nullptr, 32}, {nullptr, out, 96}});
}
int b200bls_g1_scalar_mul_batch_dev(const void* pts, const void* scalars, void* out, size_t n) {
  DevBuf db[3] = {{pts, 96}, {scalars, 32}, {out, 96}};
  return locked([&] { return run_dev("g1_mul", n, db, 3); });
}
int b200bls_g2_scalar_mul_batch(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n) {
  if (!pts || !scalars || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g2_mul", n, {{pts, nullptr, 192}, {scalars, nullptr, 32}, {nullptr, out, 192}});
}
int b200bls_g2_scalar_mul_batch_dev(const void* pts, const void* scalars, void* out, size_t n) {
  DevBuf db[3] = {{pts, 192}, {scalars, 32}, {out, 192}};
  return locked([&] { return run_dev("g2_mul", n, db, 3); });
}
int b200bls_g1_add_batch(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  if (!a || !b || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g1_add", n, {{a, nullptr, 96}, {b, nullptr, 96}, {nullptr, out, 96}});
}
int b200bls_g2_add_batch(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  if (!a || !b || !out) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g2_add", n, {{a, nullptr, 192}, {b, nullptr, 192}, {nullptr, out, 192}});
}
int b200bls_g1_sum_dev(const void* pts, void* out, size_t n) {
  return locked([&] { return sum_dev(false, pts, out, n); });
}
int b200bls_g2_sum_dev(const void* pts, void* out, size_t n) {
  return locked([&] { return sum_dev(true, pts, out, n); });
}
int b200bls_g1_sum(const uint8_t* pts, uint8_t* out, size_t n) {
  if (!out || (n && !pts)) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{pts, nullptr, 96 * n}, {nullptr, out, 96}};
  return with_staging(io, 2, [&](void** d) { return sum_dev(false, d[0], d[1], n); });
}
int b200bls_g2_sum(const uint8_t* pts, uint8_t* out, size_t n) {
  if (!out || (n && !pts)) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{pts, nullptr, 192 * n}, {nullptr, out, 192}};
  return with_staging(io, 2, [&](void** d) { return sum_dev(true, d[0], d[1], n); });
}
int b200bls_g1_decompress_batch(const uint8_t* in, uint8_t* out, uint8_t* ok, size_t n) {
  if (!in || !out || !ok) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g1_decompress", n, {{in, nullptr, 48}, {nullptr, out, 96}, {nullptr, ok, 1}});
}
int b200bls_g2_decompress_batch(const uint8_t* in, uint8_t* out, uint8_t* ok, size_t n) {
  if (!in || !out || !ok) return fail(B200BLS_E_ARG, "null buffer");
  return run_host("g2_decompress", n, {{in, nullptr, 96}, {nullptr, out, 192}, {nullptr, ok, 1}});
}
int b200bls_g1_compress_batch(const uint8_t* in, uint8_t* out, size_t n) {
  if (!in || !out) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{in, nullptr, 96 * n}, {nullptr, out, 48 * n}};
  return with_staging(io, 2, [&](void** d) { return compress_dev(false, d[0], d[1], n); });
}
int b200bls_g2_compress_batch(const uint8_t* in, uint8_t* out, size_t n) {
  if (!in || !out) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{in, nullptr, 192 * n}, {nullptr, out, 96 * n}};
  return with_staging(io, 2, [&](void** d) { return compress_dev(true, d[0], d[1], n); });
}
int b200bls_subgroup_check_batch(int g2, const uint8_t* pts, uint8_t* ok, size_t n) {
  if (!pts || !ok) return fail(B200BLS_E_ARG, "null buffer");
  size_t w = g2 ? 192 : 96;
  HostIO io[2] = {{pts, nullptr, w * n}, {nullptr, ok, n}};
  return with_staging(io, 2, [&](void** d) { return subgroup_check_dev(g2 != 0, d[0], d[1], n); });
}
int b200bls_subgroup_check_batch_dev(int g2, const void* pts, void* ok, size_t n) {
  return locked([&] { return subgroup_check_dev(g2 != 0, pts, ok, n); });
}
int b200bls_key_validate_batch(const uint8_t* pts, uint8_t* ok, size_t n) {
  if (!pts || !ok) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{pts, nullptr, 96 * n}, {nullptr, ok, n}};
  return with_staging(io, 2, [&](void** d) { return point_flags_dev("g1_keyvalidate", false, d[0], d[1], n); });
}
int b200bls_key_validate_batch_dev(const void* pts, void* ok, size_t n) {
  return locked([&] { return point_flags_dev("g1_keyvalidate", false, pts, ok, n); });
}

// ---- signing and public keys ----------------------------------------------------------------------
int b200bls_sign_batch(int wire, const uint8_t* sk32, const uint8_t* mh32, uint8_t* sig, size_t n) {
  if (wire != 0 && wire != 1) return fail(B200BLS_E_ARG, "sign: wire must be 0 (affine) or 1 (compressed)");
  if (n && (!sk32 || !mh32 || !sig)) return fail(B200BLS_E_ARG, "null buffer");
  if (n == 0) return 0;
  HostIO io[3] = {{sk32, nullptr, 32 * n}, {mh32, nullptr, 32 * n}, {nullptr, sig, (wire ? 96 : 192) * n}};
  return with_staging(io, 3, [&](void** d) { return wipe(sign_dev(wire != 0, d[0], d[1], d[2], n), d[0], 32 * n); });
}
int b200bls_sign_batch_dev(int wire, const void* sk32, const void* mh32, void* sig, size_t n) {
  if (wire != 0 && wire != 1) return fail(B200BLS_E_ARG, "sign: wire must be 0 (affine) or 1 (compressed)");
  if (n && (!sk32 || !mh32 || !sig)) return fail(B200BLS_E_ARG, "null buffer");
  return locked([&] { return sign_dev(wire != 0, sk32, mh32, sig, n); });
}
int b200bls_public_key_batch(int wire, const uint8_t* sk32, uint8_t* pk, size_t n) {
  if (wire != 0 && wire != 1) return fail(B200BLS_E_ARG, "public_key: wire must be 0 (affine) or 1 (compressed)");
  if (n && (!sk32 || !pk)) return fail(B200BLS_E_ARG, "null buffer");
  if (n == 0) return 0;
  HostIO io[2] = {{sk32, nullptr, 32 * n}, {nullptr, pk, (wire ? 48 : 96) * n}};
  return with_staging(io, 2, [&](void** d) { return wipe(public_key_dev(wire != 0, d[0], d[1], n), d[0], 32 * n); });
}
int b200bls_public_key_batch_dev(int wire, const void* sk32, void* pk, size_t n) {
  if (wire != 0 && wire != 1) return fail(B200BLS_E_ARG, "public_key: wire must be 0 (affine) or 1 (compressed)");
  if (n && (!sk32 || !pk)) return fail(B200BLS_E_ARG, "null buffer");
  return locked([&] { return public_key_dev(wire != 0, sk32, pk, n); });
}

// ---- hashing, multi-pairing, verification ----------------------------------------------------
int b200bls_hash_to_g2_batch(const uint8_t* hashes, uint8_t* out, size_t n) {
  if (!hashes || !out) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[2] = {{hashes, nullptr, 32 * n}, {nullptr, out, 192 * n}};
  return with_staging(io, 2, [&](void** d) { return hash_to_g2_dev(d[0], d[1], n); });
}
int b200bls_hash_to_g2_batch_dev(const void* hashes, void* out, size_t n) {
  return locked([&] { return hash_to_g2_dev(hashes, out, n); });
}
int b200bls_g1_msm(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n) {
  if (!out || (n && (!pts || !scalars))) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[3] = {{pts, nullptr, 96 * n}, {scalars, nullptr, 32 * n}, {nullptr, out, 96}};
  return with_staging(io, 3, [&](void** d) { return msm_dev(false, d[0], d[1], d[2], n); });
}
int b200bls_g1_msm_dev(const void* pts, const void* scalars, void* out, size_t n) {
  return locked([&] { return msm_dev(false, pts, scalars, out, n); });
}
int b200bls_g2_msm(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n) {
  if (!out || (n && (!pts || !scalars))) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[3] = {{pts, nullptr, 192 * n}, {scalars, nullptr, 32 * n}, {nullptr, out, 192}};
  return with_staging(io, 3, [&](void** d) { return msm_dev(true, d[0], d[1], d[2], n); });
}
int b200bls_g2_msm_dev(const void* pts, const void* scalars, void* out, size_t n) {
  return locked([&] { return msm_dev(true, pts, scalars, out, n); });
}
int b200bls_hash_pks(const uint8_t* pk_hash32, uint32_t first_index, uint8_t* out, size_t n) {
  if (!pk_hash32 || !out) return fail(B200BLS_E_ARG, "null buffer");
  if ((unsigned long long)first_index + n > 0x100000000ull) return fail(B200BLS_E_ARG, "index does not fit 4 bytes");
  HostIO io[2] = {{pk_hash32, nullptr, 32}, {nullptr, out, 32 * n}};
  return with_staging(io, 2, [&](void** d) { return hash_pks_dev(d[0], first_index, d[1], n); });
}
int b200bls_hash_pks_dev(const void* pk_hash32, uint32_t first_index, void* out, size_t n) {
  if ((unsigned long long)first_index + n > 0x100000000ull) return fail(B200BLS_E_ARG, "index does not fit 4 bytes");
  return locked([&] { return hash_pks_dev(pk_hash32, first_index, out, n); });
}
int b200bls_miller_product(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n) {
  if (!out || (n && (!P || !Q))) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[3] = {{P, nullptr, 96 * n}, {Q, nullptr, 192 * n}, {nullptr, out, 576}};
  return with_staging(io, 3, [&](void** d) { return miller_product_dev(d[0], d[1], d[2], n); });
}
int b200bls_miller_product_dev(const void* P, const void* Q, void* out, size_t n) {
  return locked([&] { return miller_product_dev(P, Q, out, n); });
}
int b200bls_pairing_multi(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n) {
  if (!out || (n && (!P || !Q))) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[3] = {{P, nullptr, 96 * n}, {Q, nullptr, 192 * n}, {nullptr, out, 576}};
  return with_staging(io, 3, [&](void** d) { return pairing_multi_dev(d[0], d[1], d[2], n); });
}
int b200bls_pairing_multi_dev(const void* P, const void* Q, void* out, size_t n) {
  return locked([&] { return pairing_multi_dev(P, Q, out, n); });
}
int b200bls_pairing_multi_batch(int check, const uint8_t* P, const uint8_t* Q, const uint64_t* off, size_t n_groups,
                                uint8_t* out) {
  if (check != 0 && check != 1) return fail(B200BLS_E_ARG, "pairing_multi_batch: check must be 0 (Fq12) or 1 (is one)");
  if (n_groups == 0) return 0;
  if (!off || !out) return fail(B200BLS_E_ARG, "null buffer");
  if (multi_offsets_bad(off, n_groups))
    return fail(B200BLS_E_ARG, "pairing_multi_batch: offsets must start at 0, never decrease and hold at most 2^32 - 1 "
                               "pairs in at most 2^31 - 1 groups");
  const size_t total = (size_t)off[n_groups];
  if (total && (!P || !Q)) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[4] = {{P, nullptr, 96 * total}, {Q, nullptr, 192 * total}, {off, nullptr, 8 * (n_groups + 1)},
                  {nullptr, out, (check ? 1 : 576) * n_groups}};
  return with_staging(io, 4, [&](void** d) {
    return pairing_multi_batch_dev(check != 0, d[0], d[1], (const uint64_t*)d[2], n_groups, d[3]);
  });
}
int b200bls_pairing_multi_batch_dev(int check, const void* P, const void* Q, const void* off, size_t n_groups,
                                    void* out) {
  if (check != 0 && check != 1) return fail(B200BLS_E_ARG, "pairing_multi_batch: check must be 0 (Fq12) or 1 (is one)");
  if (n_groups == 0) return 0;
  if (!off || !out) return fail(B200BLS_E_ARG, "null buffer");
  return locked([&] { return pairing_multi_batch_dev(check != 0, P, Q, (const uint64_t*)off, n_groups, out); });
}
int b200bls_verify_batch(const uint8_t* pk, const uint8_t* mh, const uint8_t* sig, uint8_t* ok, size_t n) {
  if (!pk || !mh || !sig || !ok) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[4] = {{pk, nullptr, 96 * n}, {mh, nullptr, 32 * n}, {sig, nullptr, 192 * n}, {nullptr, ok, n}};
  return with_staging(io, 4, [&](void** d) { return verify_dev(d[0], d[1], d[2], d[3], n); });
}
int b200bls_verify_batch_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n) {
  return locked([&] { return verify_dev(pk, mh, sig, ok, n); });
}

int b200bls_verify_batch_wire(const uint8_t* pk48, const uint8_t* mh, const uint8_t* sig96, uint8_t* ok, size_t n) {
  if (!pk48 || !mh || !sig96 || !ok) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[4] = {{pk48, nullptr, 48 * n}, {mh, nullptr, 32 * n}, {sig96, nullptr, 96 * n}, {nullptr, ok, n}};
  return with_staging(io, 4, [&](void** d) { return verify_wire_dev(d[0], d[1], d[2], d[3], n); });
}
int b200bls_verify_batch_wire_dev(const void* pk48, const void* mh, const void* sig96, void* ok, size_t n) {
  return locked([&] { return verify_wire_dev(pk48, mh, sig96, ok, n); });
}
int b200bls_verify_batch_strict(const uint8_t* pk, const uint8_t* mh, const uint8_t* sig, uint8_t* ok, size_t n) {
  if (!pk || !mh || !sig || !ok) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[4] = {{pk, nullptr, 96 * n}, {mh, nullptr, 32 * n}, {sig, nullptr, 192 * n}, {nullptr, ok, n}};
  return with_staging(io, 4, [&](void** d) { return verify_strict_dev(d[0], d[1], d[2], d[3], n); });
}
int b200bls_verify_batch_strict_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n) {
  return locked([&] { return verify_strict_dev(pk, mh, sig, ok, n); });
}
int b200bls_verify_batch_wire_strict(const uint8_t* pk48, const uint8_t* mh, const uint8_t* sig96, uint8_t* ok,
                                     size_t n) {
  if (!pk48 || !mh || !sig96 || !ok) return fail(B200BLS_E_ARG, "null buffer");
  HostIO io[4] = {{pk48, nullptr, 48 * n}, {mh, nullptr, 32 * n}, {sig96, nullptr, 96 * n}, {nullptr, ok, n}};
  return with_staging(io, 4, [&](void** d) { return verify_wire_dev(d[0], d[1], d[2], d[3], n, true); });
}
int b200bls_verify_batch_wire_strict_dev(const void* pk48, const void* mh, const void* sig96, void* ok, size_t n) {
  return locked([&] { return verify_wire_dev(pk48, mh, sig96, ok, n, true); });
}

namespace {
const uint8_t kNegG1[96] = {
    0x17, 0xf1, 0xd3, 0xa7, 0x31, 0x97, 0xd7, 0x94, 0x26, 0x95, 0x63, 0x8c, 0x4f, 0xa9, 0xac, 0x0f,
    0xc3, 0x68, 0x8c, 0x4f, 0x97, 0x74, 0xb9, 0x05, 0xa1, 0x4e, 0x3a, 0x3f, 0x17, 0x1b, 0xac, 0x58,
    0x6c, 0x55, 0xe8, 0x3f, 0xf9, 0x7a, 0x1a, 0xef, 0xfb, 0x3a, 0xf0, 0x0a, 0xdb, 0x22, 0xc6, 0xbb,
    0x11, 0x4d, 0x1d, 0x68, 0x55, 0xd5, 0x45, 0xa8, 0xaa, 0x7d, 0x76, 0xc8, 0xcf, 0x2e, 0x21, 0xf2,
    0x67, 0x81, 0x6a, 0xef, 0x1d, 0xb5, 0x07, 0xc9, 0x66, 0x55, 0xb9, 0xd5, 0xca, 0xac, 0x42, 0x36,
    0x4e, 0x6f, 0x38, 0xba, 0x0e, 0xcb, 0x75, 0x1b, 0xad, 0x54, 0xdc, 0xd6, 0xb9, 0x39, 0xc2, 0xca};

// stages host inputs and leaves [e(-G1, sig) *] prod_i miller(pk_i, H(mh_i)) (big-endian, not
// final-exponentiated) in buffer AGG_MILLER; sig may be null (a rank that does not own that pair)
int aggregate_miller_host(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n) {
  const size_t lead = sig ? 1 : 0, m = n + lead;
  int rc;
  if ((rc = ensure(AGG_MILLER, 576 * 2))) return rc;
  // an empty slice (a rank of a sharded verification that owns no pair) contributes the empty product: one, so that
  // every rank still reaches the exchange
  if (m == 0) return fq12_one_dev(dbuf(AGG_MILLER));
  if ((rc = ensure(AGG_P, 96 * m))) return rc;
  if ((rc = ensure(AGG_MH, 32 * m))) return rc;
  if ((rc = ensure(AGG_Q, 192 * m))) return rc;
  if ((rc = ensure(AGG_GIVEN, m))) return rc;
  uint8_t* dP = (uint8_t*)dbuf(AGG_P);
  uint8_t* dM = (uint8_t*)dbuf(AGG_MH);
  uint8_t* dQ = (uint8_t*)dbuf(AGG_Q);
  uint8_t* dG = (uint8_t*)dbuf(AGG_GIVEN);
  CU(cudaMemsetAsync(dQ, 0, 192 * m, STREAM));
  CU(cudaMemsetAsync(dG, 0, m, STREAM));
  if (sig) {
    CU(cudaMemsetAsync(dG, 1, 1, STREAM));   // item 0 is the explicitly given (-G1, signature) pair
    CU(cudaMemcpyAsync(dP, kNegG1, 96, cudaMemcpyHostToDevice, STREAM));
    CU(cudaMemcpyAsync(dQ, sig, 192, cudaMemcpyHostToDevice, STREAM));
    CU(cudaMemsetAsync(dM, 0, 32, STREAM));
  }
  if (n) {
    CU(cudaMemcpyAsync(dP + 96 * lead, pks, 96 * n, cudaMemcpyHostToDevice, STREAM));
    CU(cudaMemcpyAsync(dM + 32 * lead, mhs, 32 * n, cudaMemcpyHostToDevice, STREAM));
  }
  return aggregate_miller_dev(dP, dM, dQ, dG, dbuf(AGG_MILLER), m);
}
}  // namespace

// [e(-G1, sig) *] prod_i miller(pk_i, H(mh_i)), NOT final-exponentiated: one rank's partial of a
// sharded aggregate verification (sig = NULL on the ranks that do not own the signature pair)
int b200bls_aggregate_miller(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* out576) {
  return locked([&] {
    if (!out576 || (n && (!pks || !mhs))) return fail(B200BLS_E_ARG, "null buffer");
    int rc = aggregate_miller_host(sig, pks, mhs, n);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out576, dbuf(AGG_MILLER), 576, cudaMemcpyDeviceToHost, STREAM));
    CU(cudaStreamSynchronize(STREAM));
    return 0;
  });
}

namespace {
// enqueues the whole aggregate verification on the selected stream, result byte -> *ok (host)
int aggregate_verify_enqueue(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* ok) {
  if (!sig || !ok || (n && (!pks || !mhs))) return fail(B200BLS_E_ARG, "null buffer");
  int rc = aggregate_miller_host(sig, pks, mhs, n);
  if (rc) return rc;
  uint8_t* dF = (uint8_t*)dbuf(AGG_MILLER);
  VmBuf b[2] = {vb(dF, 576), vb(dF + 576, 1)};
  if ((rc = launch_named("final_exp_check", 1, b, 2))) return rc;
  CU(cudaMemcpyAsync(ok, dF + 576, 1, cudaMemcpyDeviceToHost, STREAM));
  return 0;
}
}  // namespace

// e(-G1, sig) * prod_i e(pk_i, H(mh_i)) == 1 for distinct message hashes and unit exponents:
// the core of BLS.verify (bls_py/bls.py:194-201) after its host-side grouping
int b200bls_aggregate_verify(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* ok) {
  return locked([&] {
    int rc = aggregate_verify_enqueue(sig, pks, mhs, n, ok);
    if (rc) return rc;
    CU(cudaStreamSynchronize(STREAM));
    return 0;
  });
}

// the same without waiting: several aggregate verifications (on different library streams,
// b200bls_set_stream) overlap -- a 10,000-message job fills a fifth of the GPU.  *ok is valid after
// b200bls_sync(); the input buffers must stay untouched until then (pinned memory lets the copies
// overlap other streams' kernels).
int b200bls_aggregate_verify_async(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* ok) {
  return locked([&] { return aggregate_verify_enqueue(sig, pks, mhs, n, ok); });
}

// ---- multi-GPU: one process per GPU, one tiny all-gather per sharded reduction (comm.cuh) -------------------
int b200bls_comm_init(int rank, int world, const char* key, const char* nccl_lib_path) {
  std::lock_guard<std::mutex> lk(g_mu);
  Comm& c = g_comm;   // (the host gather needs no GPU: the CPU-side tests of the multi-rank logic run it as is)
  if (c.shm || c.world > 1) return fail(B200BLS_E_ARG, "communicator already initialised");
  if (world < 1 || world > COMM_MAX_RANKS || rank < 0 || rank >= world) return fail(B200BLS_E_ARG, "bad rank %d / world %d", rank, world);
  c.rank = rank;
  c.world = world;
  c.seq = 0;
  if (world == 1) return 0;
  snprintf(c.shm_name, sizeof(c.shm_name), "/b200bls_%s", key && key[0] ? key : "default");
  int fd = -1;
  if (rank == 0) {
    shm_unlink(c.shm_name);   // a stale segment of a crashed run
    fd = shm_open(c.shm_name, O_CREAT | O_EXCL | O_RDWR, 0600);
    if (fd < 0 || ftruncate(fd, sizeof(CommShm)) != 0) return fail(B200BLS_E_ARG, "shm_open(%s) failed", c.shm_name);
  } else {
    for (int tries = 0; tries < 20000 && fd < 0; tries++) {   // wait for rank 0 (up to ~100 s)
      fd = shm_open(c.shm_name, O_RDWR, 0600);
      struct stat st;
      if (fd >= 0 && (fstat(fd, &st) != 0 || (size_t)st.st_size < sizeof(CommShm))) {
        close(fd);
        fd = -1;
      }
      if (fd < 0) usleep(5000);
    }
    if (fd < 0) return fail(B200BLS_E_ARG, "shared segment %s did not appear", c.shm_name);
  }
  void* m = mmap(nullptr, sizeof(CommShm), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (m == MAP_FAILED) return fail(B200BLS_E_ARG, "mmap of %s failed", c.shm_name);
  c.shm = (CommShm*)m;   // a fresh segment is zero-filled: every flag starts at 0
  c.shm->attached.fetch_add(1, std::memory_order_acq_rel);
  if (!comm_wait(c.shm->attached, (uint32_t)world, 120.0)) return fail(B200BLS_E_ARG, "only %u of %d ranks attached", c.shm->attached.load(), world);
  // NCCL (optional: the host gather works without it; needs an initialised GPU)
  const char* names[3] = {nccl_lib_path, "libnccl.so.2", "libnccl.so"};
  const bool want_nccl = g_ctx.ready && !getenv("B200BLS_NO_NCCL");   // (two ranks on ONE device: NCCL refuses)
  for (int i = 0; i < 3 && !c.nccl_lib && want_nccl; i++)
    if (names[i] && names[i][0]) c.nccl_lib = dlopen(names[i], RTLD_NOW | RTLD_LOCAL);
  if (c.nccl_lib) {
    c.p_get_unique_id = (int (*)(NcclUniqueId*))dlsym(c.nccl_lib, "ncclGetUniqueId");
    c.p_comm_init_rank = (int (*)(void**, int, NcclUniqueId, int))dlsym(c.nccl_lib, "ncclCommInitRank");
    c.p_all_gather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(c.nccl_lib, "ncclAllGather");
    c.p_comm_destroy = (int (*)(void*))dlsym(c.nccl_lib, "ncclCommDestroy");
    c.p_error_string = (const char* (*)(int))dlsym(c.nccl_lib, "ncclGetErrorString");
    const bool have = c.p_get_unique_id && c.p_comm_init_rank && c.p_all_gather && c.p_comm_destroy;
    int rcn = have ? 0 : -1;
    if (have && rank == 0) {
      rcn = c.p_get_unique_id(&c.shm->nccl_id);
      c.shm->id_ready.store(rcn == 0 ? 1u : 2u, std::memory_order_release);
    }
    if (have && rank != 0) {
      if (!comm_wait(c.shm->id_ready, 1u, 120.0) || c.shm->id_ready.load() != 1u) rcn = -1;
    }
    if (rcn == 0) rcn = c.p_comm_init_rank(&c.nccl_comm, world, c.shm->nccl_id, rank);
    if (rcn != 0) {
      c.nccl_comm = nullptr;
      fail(B200BLS_E_CUDA, "NCCL initialisation failed (%s); the host gather remains available",
           c.p_error_string && rcn > 0 ? c.p_error_string(rcn) : "missing symbol or unique id");
    } else {
      CU(cudaMalloc(&c.gather_dev, (size_t)world * COMM_SLOT_BYTES));
      CU(cudaMalloc(&c.send_dev, COMM_SLOT_BYTES));
    }
  }
  return 0;
}

int b200bls_comm_has_nccl(void) { return g_comm.nccl_comm != nullptr; }

// all-gather of `bytes` (<= 4096) host bytes per rank through the node's shared-memory segment
int b200bls_allgather_host(const uint8_t* send, uint8_t* recv, size_t bytes) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!send || !recv) return fail(B200BLS_E_ARG, "null buffer");
  if (bytes > COMM_SLOT_BYTES) return fail(B200BLS_E_ARG, "payload of %zu bytes exceeds the exchange slot", bytes);
  if (g_comm.world > 1 && !g_comm.shm) return fail(B200BLS_E_NOT_INIT, "communicator not initialised");
  if (comm_allgather_host(g_comm, send, recv, bytes) != 0) return fail(B200BLS_E_CUDA, "host gather timed out");
  return 0;
}
int b200bls_comm_world(void) { return g_comm.world; }
int b200bls_comm_rank(void) { return g_comm.rank; }

void b200bls_comm_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  Comm& c = g_comm;
  if (c.nccl_comm && c.p_comm_destroy) c.p_comm_destroy(c.nccl_comm);
  if (c.gather_dev) cudaFree(c.gather_dev);
  if (c.send_dev) cudaFree(c.send_dev);
  if (c.shm) {
    munmap(c.shm, sizeof(CommShm));
    if (c.rank == 0) shm_unlink(c.shm_name);
  }
  c = Comm();
}

namespace {
// all ranks' `bytes` (device, at src_dev) -> gathered_dev[world][bytes] on this rank, through NCCL or the host
int gather_partials(const void* src_dev, size_t bytes, int use_nccl, void** gathered_dev) {
  Comm& c = g_comm;
  if (bytes > COMM_SLOT_BYTES) return fail(B200BLS_E_ARG, "partial of %zu bytes exceeds the exchange slot", bytes);
  if (c.world == 1) {
    *gathered_dev = (void*)src_dev;
    return 0;
  }
  if (use_nccl) {
    if (!c.nccl_comm) return fail(B200BLS_E_ARG, "NCCL gather requested but NCCL is not initialised");
    int rc = c.p_all_gather(src_dev, c.gather_dev, bytes, /* ncclUint8 */ 1, c.nccl_comm, STREAM);
    if (rc != 0) return fail(B200BLS_E_CUDA, "ncclAllGather failed: %s", c.p_error_string ? c.p_error_string(rc) : "?");
    *gathered_dev = c.gather_dev;
    return 0;
  }
  int rc = ensure(GATHERED, (size_t)c.world * bytes);
  if (rc) return rc;
  static thread_local unsigned char mine[COMM_SLOT_BYTES];
  static thread_local unsigned char all[COMM_MAX_RANKS * 1024];
  if ((size_t)c.world * bytes > sizeof(all)) return fail(B200BLS_E_ARG, "host gather payload too large");
  CU(cudaMemcpyAsync(mine, src_dev, bytes, cudaMemcpyDeviceToHost, STREAM));
  CU(cudaStreamSynchronize(STREAM));
  if (comm_allgather_host(c, mine, all, bytes) != 0) return fail(B200BLS_E_CUDA, "host gather timed out");
  CU(cudaMemcpyAsync(dbuf(GATHERED), all, (size_t)c.world * bytes, cudaMemcpyHostToDevice, STREAM));
  *gathered_dev = dbuf(GATHERED);
  return 0;
}
}  // namespace

// Aggregate verification with the (pk_i, message hash_i) pairs sharded over the ranks: pks / mhs are THIS
// rank's slice (n may be 0), sig the aggregate signature (read on rank 0 only).  Every rank hashes and pairs
// its slice in one fused launch, the 576-byte Miller products are all-gathered (use_nccl: ncclAllGather over
// NVLink, else the shared-memory host gather), multiplied, and final-exponentiated once -- on every rank, so
// every rank returns the same *ok (bls_py/bls.py:194-201 over a sharded message list).
int b200bls_aggregate_verify_sharded(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, int use_nccl,
                                     uint8_t* ok) {
  return locked([&] {
    if (!ok || (n && (!pks || !mhs))) return fail(B200BLS_E_ARG, "null buffer");
    if (g_comm.rank == 0 && !sig) return fail(B200BLS_E_ARG, "rank 0 needs the signature");
    int rc = aggregate_miller_host(g_comm.rank == 0 ? sig : nullptr, pks, mhs, n);
    if (rc) return rc;
    void* parts = nullptr;
    if ((rc = gather_partials(dbuf(AGG_MILLER), 576, use_nccl, &parts))) return rc;
    // product of the per-rank values: world - 1 Fq12 products on the device, then the final exponentiation check
    if ((rc = ensure(SHARD_ACC, 576 + 16))) return rc;
    uint8_t* acc = (uint8_t*)dbuf(SHARD_ACC);
    CU(cudaMemcpyAsync(acc, parts, 576, cudaMemcpyDeviceToDevice, STREAM));
    for (int r = 1; r < g_comm.world; r++) {
      DevBuf db[3] = {{acc, 576}, {(uint8_t*)parts + 576 * (size_t)r, 576}, {acc, 576}};
      if ((rc = run_dev("f12_mul", 1, db, 3))) return rc;
    }
    VmBuf b[2] = {vb(acc, 576), vb(acc + 576, 1)};
    if ((rc = launch_named("final_exp_check", 1, b, 2))) return rc;
    CU(cudaMemcpyAsync(ok, acc + 576, 1, cudaMemcpyDeviceToHost, STREAM));
    CU(cudaStreamSynchronize(STREAM));
    return 0;
  });
}

// Sum of points sharded over the ranks (BLS.aggregate_sigs_simple / aggregate_pub_keys(secure=False),
// bls.py:13-26, 204-223): pts_dev is THIS rank's device-resident slice of n affine points; every rank reduces
// its slice to one affine point, the points are all-gathered and summed on every rank.  out: 96 / 192 host bytes.
int b200bls_point_sum_sharded_dev(int g2, const void* pts_dev, size_t n, int use_nccl, uint8_t* out) {
  return locked([&] {
    if (!out) return fail(B200BLS_E_ARG, "null buffer");
    const size_t w = g2 ? 192 : 96;
    int rc = ensure(SHARD_ACC, 2 * w);
    if (rc) return rc;
    uint8_t* part = (uint8_t*)dbuf(SHARD_ACC);
    if ((rc = sum_dev(g2 != 0, pts_dev, part, n))) return rc;
    void* parts = nullptr;
    if ((rc = gather_partials(part, w, use_nccl, &parts))) return rc;
    if (g_comm.world > 1) {
      if ((rc = sum_dev(g2 != 0, parts, part + w, (size_t)g_comm.world))) return rc;
      part += w;
    }
    CU(cudaMemcpyAsync(out, part, w, cudaMemcpyDeviceToHost, STREAM));
    CU(cudaStreamSynchronize(STREAM));
    return 0;
  });
}

}  // extern "C"
