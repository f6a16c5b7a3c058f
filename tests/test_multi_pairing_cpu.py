"""The batched multi-pairing without a GPU: the segmented product programs f12_prodseg / f12_prodseg_be on the host
simulation of the VM (both executors, segmented launch mode) against the oracle's Fq12 products, the chunk tables of
python-bls_b200/csrc/multi_plan.h built with g++ against literal tables, and the argument checks of the C ABI."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import bls_oracle as O
import hostsim

from bls_b200.programs import pairing, registry
from bls_b200.vm.builder import Program

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "python-bls_b200", "csrc")
SEG_SRC = os.path.join(ROOT, "tests", "hostsim", "hostsim_seg.cpp")
L = 16
PASSES = 8
E_ARG = -3


# ---- segmented launches on the host simulation --------------------------------------------------------------------
@pytest.fixture(scope="module")
def seg_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("seg")
    objs = []
    for k in (1, 2):
        o = str(d / ("seg%d.o" % k))
        subprocess.check_call(["g++", "-O2", "-fPIC", "-c", "-DHOSTSIM_SEG%d" % k, "-o", o, SEG_SRC])
        objs.append(o)
    so = str(d / "seg.so")
    subprocess.check_call(["g++", "-shared", "-o", so] + objs)
    return ctypes.CDLL(so)


def _run_seg(lib, asm, bufs, strides, seg_start, seg_idx, per_block=4):
    """one segmented launch of len(seg_start) - 1 segments on both executors -> the buffers of each.  Byte buffers
    must agree byte for byte; raw SoA values are only weakly reduced, and the executors' representatives may differ"""
    n = len(seg_start) - 1
    start = np.ascontiguousarray(seg_start, dtype=np.uint32)
    idx = np.ascontiguousarray(seg_idx if len(seg_idx) else [0], dtype=np.uint32)
    code = np.ascontiguousarray(asm.code).view(np.uint32).reshape(-1)
    consts = np.ascontiguousarray(asm.const_limbs())
    results = []
    for fn in (lib.hs_vm_run_seg, lib.hs_vm2_run_seg):
        own = {i: b.copy() for i, b in bufs.items()}
        ptrs = (ctypes.c_void_p * 8)()
        st = (ctypes.c_long * 8)()
        for i, b in own.items():
            ptrs[i] = b.ctypes.data
            st[i] = strides[i]
        rc = fn(code.ctypes.data_as(ctypes.c_void_p), len(asm.code), asm.body_start, asm.epilogue_start,
                consts.ctypes.data_as(ctypes.c_void_p), asm.n_slots, asm.n_tmem, max(asm.stats["max_cold"], 1), ptrs,
                st, ctypes.c_long(n), per_block, start.ctypes.data_as(ctypes.c_void_p),
                idx.ctypes.data_as(ctypes.c_void_p))
        assert rc == 0
        results.append(own)
    for i in bufs:
        if strides[i] == 576:
            assert np.array_equal(results[0][i], results[1][i]), "executors disagree on buffer %d" % i
    return results


def _to_raw_program():
    """test helper: 576 big-endian bytes (buffer 0) -> raw SoA Fq12 (buffer 1), the layout miller_raw writes"""
    prog = Program("test_f12_to_raw")
    prog.begin_body()
    for k in range(6):
        prog.store_raw2(1, k, prog.load2_be48(0, 96 * k))
    return prog


def _f12_prod(vals):
    r = O.F12_ONE
    for v in vals:
        r = O.f12_mul(r, v)
    return r


@pytest.mark.parametrize("ctas", [1, 4])
def test_prodseg_on_host_simulation(seg_lib, ctas):
    """two passes over ragged chunks read through a shuffled index list: empty chunks, chunks of one, chunks of L, more
    chunks than one CTA holds; the first pass writes raw products (f12_prodseg), the second multiplies them in groups
    and writes bytes (f12_prodseg_be)"""
    rng = random.Random(20261022 + ctas)
    lens = [0, 1, 3, L, 0, 2, 1, L - 1, 5, 0, 1, 7, 4]
    m = sum(lens)
    vals = [tuple(rng.randrange(O.Q) for _ in range(12)) for _ in range(m - 2)] + [O.F12_ONE, (0,) * 12]
    n_slots, n_tmem = registry.SHAPES[ctas]
    be = np.frombuffer(b"".join(O.f12_serialize(v) for v in vals), dtype=np.uint8).copy()
    raw = np.zeros(576 * m, dtype=np.uint8)
    hostsim.run(_to_raw_program().assemble(n_slots, n_cold=4096, n_tmem=n_tmem), {0: be, 1: raw}, {0: 576, 1: m}, m,
                n_blocks=2, nt=4)
    order = list(range(m))
    rng.shuffle(order)
    starts = list(np.cumsum([0] + lens))
    want1 = [_f12_prod(vals[j] for j in order[starts[c]:starts[c + 1]]) for c in range(len(lens))]

    seg = registry.PROGRAMS["f12_prodseg"]().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    n1 = len(lens)
    part = np.full(576 * n1, 0x5a, dtype=np.uint8)
    parts = [r[1] for r in _run_seg(seg_lib, seg, {0: raw, 1: part}, {0: m, 1: n1}, starts, order)]

    groups = [[0, 1, 2], [], [3], [4, 5, 6, 7, 8, 9, 10, 11, 12]]
    gstarts = list(np.cumsum([0] + [len(g) for g in groups]))
    gorder = [c for g in groups for c in g]
    segbe = registry.PROGRAMS["f12_prodseg_be"]().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    for part in parts:      # the raw products of either executor
        out = np.full(576 * len(groups), 0x5a, dtype=np.uint8)
        out = _run_seg(seg_lib, segbe, {0: part, 1: out}, {0: n1, 1: 576}, gstarts, gorder)[0][1].tobytes()
        for g, cs in enumerate(groups):
            assert out[576 * g:576 * (g + 1)] == O.f12_serialize(_f12_prod(want1[c] for c in cs)), (ctas, g)
        # the chunk products themselves, through a byte-writing pass of one value per segment
        out1 = np.full(576 * n1, 0x5a, dtype=np.uint8)
        out1 = _run_seg(seg_lib, segbe, {0: part, 1: out1}, {0: n1, 1: 576}, list(range(n1 + 1)), list(range(n1)))
        for c in range(n1):
            assert out1[0][1].tobytes()[576 * c:576 * (c + 1)] == O.f12_serialize(want1[c]), (ctas, c)


def test_prodseg_programs_share_the_product_body():
    """one Fq12 product per value (18 Fq2 products), and the byte form adds only the conversion of its output"""
    assert registry.executed_mults("f12_prodseg") == 54
    assert registry.executed_mults("f12_prodseg_be") - registry.executed_mults("f12_prodseg") <= 12
    assert 16 * registry.executed_mults("f12_prodseg") <= 0.15 * registry.executed_mults("miller_raw")
    assert pairing.build_f12_product_seg(True)().name == "f12_prodseg_be"


# ---- the chunk tables (multi_plan.h) built with g++ ---------------------------------------------------------------
SHIM = r"""
#include "multi_plan.h"
using namespace b200bls;
extern "C" int shim_bad(const uint64_t* off, uint64_t n) { return multi_offsets_bad(off, n); }
extern "C" unsigned shim_L(void) { return kMultiL; }
// the prefix tables as multi_scan_kernel writes them (a serial scan of the same per-group counts); returns the passes
extern "C" int shim_prefix(const uint64_t* off, uint64_t n, uint32_t* prefix) {
  uint32_t run[kMultiMaxPasses] = {}, cnt[kMultiMaxPasses];
  for (uint64_t g = 0; g <= n; g++) {
    for (int r = 0; r < kMultiMaxPasses; r++) prefix[r * (n + 1) + g] = run[r];
    if (g == n) break;
    multi_group_chunks(off[g + 1] - off[g], cnt);
    for (int r = 0; r < kMultiMaxPasses; r++) run[r] += cnt[r];
  }
  return multi_passes(run, n);
}
// the segment starts of pass r, one call per group as multi_tables_kernel runs them
extern "C" void shim_segments(int r, const uint64_t* off, uint64_t n, const uint32_t* prefix, uint32_t* seg) {
  for (uint64_t g = 0; g < n; g++) multi_segments_group(r, g, n, off, prefix, seg);
}
"""


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    d = tmp_path_factory.mktemp("multi_plan")
    src, so = d / "shim.cpp", d / "plan.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    lib.shim_bad.argtypes = [ctypes.c_void_p, ctypes.c_uint64]
    lib.shim_prefix.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]
    lib.shim_segments.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
    assert lib.shim_L() == L

    def tables(off):
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = off.size - 1
        prefix = np.zeros(PASSES * (n + 1), dtype=np.uint32)
        passes = lib.shim_prefix(off.ctypes.data, n, prefix.ctypes.data)
        rows = prefix.reshape(PASSES, n + 1)
        segs = []
        for r in range(passes):
            seg = np.full(int(rows[r][n]) + 1, 0xffffffff, dtype=np.uint32)
            lib.shim_segments(r, off.ctypes.data, n, prefix.ctypes.data, seg.ctypes.data)
            segs.append(seg.tolist())
        return [row.tolist() for row in rows[:passes]], segs

    def bad(off, n=None):
        off = np.ascontiguousarray(off, dtype=np.uint64)
        return lib.shim_bad(off.ctypes.data, off.size - 1 if n is None else n)
    return tables, bad


def test_tables_all_empty(plan):
    tables, _ = plan
    assert tables([0, 0, 0, 0]) == ([[0, 1, 2, 3]], [[0, 0, 0, 0]])


def test_tables_one_huge_group(plan):
    tables, _ = plan
    prefix, segs = tables([0, 1000])
    assert prefix == [[0, 63], [0, 4], [0, 1]]
    assert segs == [list(range(0, 1000, 16)) + [1000], [0, 16, 32, 48, 63], [0, 4]]


def test_tables_groups_of_L_and_L_plus_1(plan):
    tables, _ = plan
    assert tables([0, 16, 33]) == ([[0, 1, 3], [0, 1, 2]], [[0, 16, 32, 33], [0, 1, 3]])
    assert tables([0, 16, 32]) == ([[0, 1, 2]], [[0, 16, 32]])


def test_tables_more_than_L_squared_pairs(plan):
    """257 pairs in a group after an empty one: 17 chunks, then 2, then 1"""
    tables, _ = plan
    prefix, segs = tables([0, 3, 3, 260])
    assert prefix == [[0, 1, 2, 19], [0, 1, 2, 4], [0, 1, 2, 3]]
    assert segs == [[0, 3] + list(range(3, 260, 16)) + [260], [0, 1, 2, 18, 19], [0, 1, 2, 4]]


def test_tables_cover_every_value_once(plan):
    """seeded ragged layouts: every pass's chunks tile its values in order, each chunk within one group and at most
    L long, and the last pass has one chunk per group"""
    tables, _ = plan
    rng = random.Random(7)
    for _ in range(50):
        lens = [rng.choice([0, 0, 1, 2, 15, 16, 17, 255, 256, 257, rng.randrange(5000)]) for _ in range(rng.randrange(1, 30))]
        off = [0] + list(np.cumsum(lens))
        prefix, segs = tables(off)
        bounds = off
        for r, seg in enumerate(segs):
            n_chunks = prefix[r][-1]
            assert len(seg) == n_chunks + 1 and seg[0] == 0 and seg[-1] == bounds[-1]
            assert all(0 <= b - a <= L for a, b in zip(seg, seg[1:]))
            for g in range(len(lens)):
                c0, c1 = prefix[r][g], prefix[r][g + 1]
                assert seg[c0] == bounds[g] and seg[c1] == bounds[g + 1]
            bounds = prefix[r]
        assert prefix[-1] == list(range(len(lens) + 1))


def test_offsets_refused(plan):
    _, bad = plan
    assert bad([0]) == 0 and bad([0, 0]) == 0 and bad([0, 2, 2, 5]) == 0
    assert bad([1, 2]) == 1                              # off[0] != 0
    assert bad([0, 3, 2]) == 1                           # decreasing
    assert bad([0, 2 ** 32 - 1]) == 0
    assert bad([0, 2 ** 32]) == 1                        # more pairs than 32-bit segment starts index
    assert bad([0, 0], n=2 ** 31) == 1                   # more groups than final_exp runs items (not read)


# ---- the C ABI ---------------------------------------------------------------------------------------------------
def _lib():
    so = os.path.join(ROOT, "python-bls_b200", "bls_b200", "libb200bls.so")
    if not os.path.exists(so):
        import __graft_entry__
        __graft_entry__.build()
    return ctypes.CDLL(so)


def test_abi_symbols():
    from test_abi import declared_symbols
    from bls_b200 import _lib as L_
    lib = _lib()
    for s in ("b200bls_pairing_multi_batch", "b200bls_pairing_multi_batch_dev"):
        assert s in declared_symbols() and hasattr(lib, s) and s in L_.SIGNATURES


def test_argument_checks_need_no_device():
    """bad check values, null buffers and bad offsets are refused before the library looks for a GPU; n_groups = 0 does
    nothing"""
    lib = _lib()
    buf = (ctypes.c_uint8 * 576)()
    zero, one, two = ctypes.c_size_t(0), ctypes.c_size_t(1), ctypes.c_size_t(2)

    def offs(*v):
        return (ctypes.c_uint64 * len(v))(*v)
    for check in (-1, 2):
        assert lib.b200bls_pairing_multi_batch(check, buf, buf, offs(0, 1), one, buf) == E_ARG
        assert lib.b200bls_pairing_multi_batch_dev(check, buf, buf, offs(0, 1), one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, None, None, None, zero, None) == 0
    assert lib.b200bls_pairing_multi_batch_dev(1, None, None, None, zero, None) == 0
    assert lib.b200bls_pairing_multi_batch(0, buf, buf, None, one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, buf, buf, offs(0, 1), one, None) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, None, buf, offs(0, 1), one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch_dev(0, buf, buf, None, one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, buf, buf, offs(1, 1), one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(1, buf, buf, offs(0, 2, 1), two, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, buf, buf, offs(0, 2 ** 32), one, buf) == E_ARG
    assert lib.b200bls_pairing_multi_batch(0, buf, buf, offs(0, 0), ctypes.c_size_t(2 ** 31), buf) == E_ARG
