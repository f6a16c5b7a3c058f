// Segmented launch mode (VmParams::seg_start / seg_idx) on the host simulation, for both executors.
// TEST INFRASTRUCTURE: the drivers of hostsim_vm.cpp / hostsim_vm2.cpp with the segment loop of vm_kernel.cuh /
// vm_kernel2.cuh.  One CTA per `nt` segments (one-thread executor) or `items_per_block` segments (paired executor), as
// the launcher plans a segmented launch: thread (pair) t owns segment t; body iteration k reads record
// seg_idx[seg_start[t] + k] and is inactive (FACTIVE false, record 0) once k reaches the segment's length; the CTA runs
// as many iterations as its longest segment; prologue and epilogue address record t.
// Built as its own translation units: SEG1 includes the one-thread driver, SEG2 the paired one.
#if defined(HOSTSIM_SEG1)
#include "hostsim_vm.cpp"

extern "C" int hs_vm_run_seg(const uint32_t* code, int n_ins, int body_start, int epi_start, const uint32_t* consts,
                             int n_slots, int n_tmem, int n_cold, uint8_t** bufs, const long* strides, long n_items,
                             int nt, const unsigned* seg_start, const unsigned* seg_idx) {
  Shared sh;
  sh.consts = consts;
  for (int i = 0; i < 8; i++) { sh.bufs[i] = bufs[i]; sh.strides[i] = strides[i]; }
  sh.n_items = n_items;
  sh.nt = nt;
  sh.n_blocks = (int)((n_items + nt - 1) / nt);
  if (sh.n_blocks < 1) sh.n_blocks = 1;
  const int n_blocks = sh.n_blocks;
  sh.total = nt * n_blocks;
  sh.n_cells = 2 * (n_slots + n_tmem);
  sh.smem_cells = 2 * n_slots;
  sh.written.assign(sh.n_cells, 0);
  sh.xread.assign(sh.n_cells, 0);
  std::vector<std::vector<uint32_t>> smem(n_blocks);
  for (auto& s : smem) s.assign((size_t)sh.n_cells * 3 * nt * 4, 0xdeadbeefu);
  sh.smem = smem.data();
  sh.cold.assign((size_t)n_cold * 6 * sh.total * 4, 0xdeadbeefu);
  std::vector<HostEnv> env(sh.total);
  const long last = n_items > 0 ? n_items - 1 : 0;
  auto own_record = [&]() {
    for (int g = 0; g < sh.total; g++) {
      env[g].item_raw = g;
      env[g].item = g < last ? g : last;
    }
  };
  for (int g = 0; g < sh.total; g++) {
    env[g].sh = &sh;
    env[g].gtid = g;
    env[g].blk = g / nt;
    env[g].tid = g % nt;
    env[g].flags = 0;
  }
  auto exec = [&](int blk, int lo, int hi) {
    for (int pc = lo; pc < hi; pc++) {
      uint32_t w0 = code[2 * pc], w1 = code[2 * pc + 1];
      if ((w0 & 0xff) == OP_SKIPZ) {
        bool any = false;
        for (int t = 0; t < nt; t++) any = any || env[blk * nt + t].get_flag(w0 >> 16);
        if (!any) pc += (int)(w1 & 0xffff);
        continue;
      }
      for (int t = 0; t < nt; t++) vm_exec(env[blk * nt + t], w0, w1);
    }
  };
  auto seg_len = [&](long g) -> unsigned { return g < n_items ? seg_start[g + 1] - seg_start[g] : 0u; };
  own_record();
  for (int blk = 0; blk < n_blocks; blk++) exec(blk, 0, body_start);
  for (int blk = 0; blk < n_blocks; blk++) {
    unsigned iters = 0;
    for (int t = 0; t < nt; t++) iters = std::max(iters, seg_len(blk * nt + t));
    for (unsigned k = 0; k < iters; k++) {
      for (int t = 0; t < nt; t++) {
        const long g = blk * nt + t;
        const bool act = k < seg_len(g);
        env[g].item = act ? (long)seg_idx[seg_start[g] + k] : 0;
        env[g].item_raw = act ? 0 : n_items;
      }
      exec(blk, body_start, epi_start);
    }
  }
  own_record();
  for (int blk = 0; blk < n_blocks; blk++) exec(blk, epi_start, n_ins);
  return 0;
}

#elif defined(HOSTSIM_SEG2)
#include "hostsim_vm2.cpp"

extern "C" int hs_vm2_run_seg(const uint32_t* code, int n_ins, int body_start, int epi_start, const uint32_t* consts,
                              int n_slots, int n_tmem, int n_cold, uint8_t** bufs, const long* strides, long n_items,
                              int items_per_block, const unsigned* seg_start, const unsigned* seg_idx) {
  (void)n_ins;
  Shared sh;
  sh.consts = consts;
  for (int i = 0; i < 8; i++) {
    sh.bufs[i] = bufs[i];
    sh.strides[i] = strides[i];
  }
  sh.n_items = n_items;
  sh.items_per_block = items_per_block;
  int n_blocks = (int)((n_items + items_per_block - 1) / items_per_block);
  if (n_blocks < 1) n_blocks = 1;
  sh.n_blocks = n_blocks;
  sh.total_items = items_per_block * n_blocks;
  sh.n_slots_all = n_slots + n_tmem;
  sh.smem_slots = n_slots;
  sh.written.assign(sh.n_slots_all, 0);
  sh.xread.assign(sh.n_slots_all, 0);
  const int nt = 2 * items_per_block;
  std::vector<std::vector<uint32_t>> ws(n_blocks);
  for (auto& s : ws) s.assign((size_t)sh.n_slots_all * 3 * nt * 4, 0xdeadbeefu);
  sh.ws = ws.data();
  sh.cold.assign((size_t)n_cold * 3 * nt * n_blocks * 4, 0xdeadbeefu);
  std::vector<PairHostEnv> env((size_t)nt * n_blocks);
  for (int b = 0; b < n_blocks; b++)
    for (int t = 0; t < nt; t++) {
      PairHostEnv& e = env[(size_t)b * nt + t];
      e.sh = &sh;
      e.blk = b;
      e.tid = t;
      e.flags = 0;
    }
  const long last = n_items > 0 ? n_items - 1 : 0;
  auto own_record = [&]() {
    for (int b = 0; b < n_blocks; b++)
      for (int t = 0; t < nt; t++) {
        PairHostEnv& e = env[(size_t)b * nt + t];
        e.item_raw = (long)b * items_per_block + (t >> 1);
        e.item = e.item_raw < last ? e.item_raw : last;
      }
  };
  // one section of block b, from lo to its END instruction (the driver loop of hs_vm2_run)
  auto exec = [&](int b, int lo) {
    for (int pc = lo;; pc++) {
      const uint32_t w0 = code[2 * pc], w1 = code[2 * pc + 1];
      const int op = w0 & 0xff;
      if (op == OP_END) break;
      if (op == OP_SKIPZ) {
        bool any = false;
        for (int t = 0; t < nt; t++) any = any || env[(size_t)b * nt + t].get_flag(w0 >> 16);
        if (!any) pc += (int)(w1 & 0xffff);
        continue;
      }
      sh.stores.clear();
      sh.byte_stores.clear();
      for (int item = 0; item < items_per_block; item++) {
        PairHostEnv* pr = &env[(size_t)b * nt + 2 * item];
        const uint32_t f0 = pr[0].flags, f1 = pr[1].flags;
        sh.xchg_count[0] = sh.xchg_count[1] = 0;
        sh.pass = 0;
        vm_exec2(pr[0], w0, w1);
        vm_exec2(pr[1], w0, w1);
        pr[0].flags = f0;
        pr[1].flags = f1;
        sh.pass = 1;
        vm_exec2(pr[0], w0, w1);
        vm_exec2(pr[1], w0, w1);
        if (pr[0].flags != pr[1].flags) abort();
      }
      for (const Store& s : sh.stores) memcpy(s.dst, s.v, 16);
      for (const ByteStore& s : sh.byte_stores) *s.dst = s.v;
    }
  };
  auto seg_len = [&](long g) -> unsigned { return g < n_items ? seg_start[g + 1] - seg_start[g] : 0u; };
  own_record();
  for (int b = 0; b < n_blocks; b++) exec(b, 0);
  for (int b = 0; b < n_blocks; b++) {
    unsigned iters = 0;
    for (int i = 0; i < items_per_block; i++) iters = std::max(iters, seg_len((long)b * items_per_block + i));
    for (unsigned k = 0; k < iters; k++) {
      for (int t = 0; t < nt; t++) {
        PairHostEnv& e = env[(size_t)b * nt + t];
        const long g = (long)b * items_per_block + (t >> 1);
        const bool act = k < seg_len(g);
        e.item = act ? (long)seg_idx[seg_start[g] + k] : 0;
        e.item_raw = act ? 0 : n_items;
      }
      exec(b, body_start);
    }
  }
  own_record();
  for (int b = 0; b < n_blocks; b++) exec(b, epi_start);
  return 0;
}
#endif
