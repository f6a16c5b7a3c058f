#!/usr/bin/env python3
"""Benchmark of the b200-bls hot path (BASELINE.json: pairings/s and signatures verified/s vs host CPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one batch of 65,536 independent full ate pairings (Miller loop + exact final exponentiation,
BASELINE config 2) per GPU on synthetic seeded inputs; weak scaling: every rank owns its own batch, no data-path
collective on this metric (SURVEY.md 8e).  Rank 0 prints ONE JSON line:
  value        pairings/s with inputs resident in HBM, CUDA events over the library streams
  e2e          the same through the C-ABI host-buffer call (pinned HOST buffers: H2D, kernel, D2H in the timed region)
  roofline     integer-multiply roofline: limb products the program executes / measured IMAD.WIDE peak
  cpu_baseline the reference's own CPU implementation (unmodified, oracle/_ref) on all host cores, bounded sample;
               its outputs double as the parity oracle for the sampled indices
  extra        signatures verified/s, BASELINE configs 3 / 4 / 5 at full size with their parity booleans, the
               isolated synchronous call, and -- under N > 1 -- the sharded reductions over BOTH exchange transports
`--impl reference` times that CPU path alone with the same metric and config.
`--dump-outputs DIR` writes what the last timed step computed (see dump_outputs) so that two builds can be compared
output for output: the inputs depend only on the seeds and the rank.
"""
import argparse
import hashlib
import json
import os
import struct
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "python-bls_b200"))

BATCH = 65536
M_NOMINAL = 15200                # SURVEY.md 8d, frozen: efficient-algorithm Fq products per pairing
M_VERIFY_NOMINAL = 30400
LIMB_PRODUCTS_PER_M = 300        # 12x12 limbs: 144 + 144 + 12
METRIC = "pairings/s"
WORKLOAD = "config2: 65,536 independent ate pairings (Miller loop + final exponentiation) per GPU"


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/_ref, installed by tools/install_reference.py), else the oracle port
# ---------------------------------------------------------------------------------------------
def cpu_impl_kind():
    return "reference" if os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "bls_py")) else "port"


def extmod_note():
    try:
        with open(os.path.join(ROOT, "oracle", "_ref", "STATUS.json")) as fh:
            return json.load(fh)["extmod"]
    except (OSError, ValueError, KeyError):
        return "extmod: does not build in this image (no gmp.h; CPython-3.12-incompatible int access, SURVEY.md 8c)"


_CPU = {}


def _cpu_load(kind):
    """per worker process: import the CPU implementation once"""
    if kind in _CPU:
        return _CPU[kind]
    if kind == "reference":
        import logging
        logging.disable(logging.CRITICAL)          # the reference logs that its Cython accelerator is absent
        sys.dont_write_bytecode = True
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        from bls_py import ec, pairing
        from bls_py.fields import Fq, Fq2
        q = ec.default_ec.q

        def g1(raw):
            return ec.AffinePoint(Fq(q, int.from_bytes(raw[:48], "big")), Fq(q, int.from_bytes(raw[48:], "big")),
                                  False, ec.default_ec)

        def g2(raw):
            c = [int.from_bytes(raw[i:i + 48], "big") for i in range(0, 192, 48)]
            return ec.AffinePoint(Fq2(q, c[0], c[1]), Fq2(q, c[2], c[3]), False, ec.default_ec_twist)

        def mul1(k):
            return (ec.generator_Fq().to_jacobian() * k).to_affine()

        def mul2(k):
            return (ec.generator_Fq2().to_jacobian() * k).to_affine()

        def pair(p, qq):
            return b"".join(c.to_bytes(48, "big") for c in pairing.ate_pairing(p, qq).ZT)

        def verify(pk96, h, sig192):
            from bls_py.aggregation_info import AggregationInfo
            from bls_py.bls import BLS
            from bls_py.keys import PublicKey
            from bls_py.signature import Signature
            pk = PublicKey.from_g1(g1(pk96).to_jacobian())
            sig = Signature.from_g2(g2(sig192).to_jacobian(), AggregationInfo.from_msg_hash(pk, h))
            return bool(BLS.verify(sig))
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import bls_oracle as O

        def g1(raw):
            return (int.from_bytes(raw[:48], "big"), int.from_bytes(raw[48:], "big"), False)

        def g2(raw):
            c = [int.from_bytes(raw[i:i + 48], "big") for i in range(0, 192, 48)]
            return ((c[0], c[1]), (c[2], c[3]), False)

        def mul1(k):
            return O.aff_mul(k, O.G1)

        def mul2(k):
            return O.aff_mul(k, O.G2)

        def pair(p, qq):
            return O.f12_serialize(O.ate_pairing(p, qq))

        def verify(pk96, h, sig192):
            return bool(O.verify(g1(pk96), h, g2(sig192)))
    _CPU[kind] = (g1, g2, mul1, mul2, pair, verify)
    return _CPU[kind]


def _cpu_pair_worker(task):
    """task = (kind, [(idx, a, b, P bytes or None, Q bytes or None)]): inputs are built untimed (from the GPU's
    own input bytes, or by the CPU implementation's scalar multiplication), only ate_pairing is timed"""
    kind, items = task
    g1, g2, mul1, mul2, pair, _ = _cpu_load(kind)
    pts = [(idx, g1(bytes(P)) if P is not None else mul1(a), g2(bytes(Q)) if Q is not None else mul2(b))
           for idx, a, b, P, Q in items]
    t0 = time.perf_counter()
    out = [(idx, pair(p, q)) for idx, p, q in pts]
    return time.perf_counter() - t0, out


def _cpu_verify_worker(task):
    kind, items = task
    verify = _cpu_load(kind)[5]
    return [(idx, verify(bytes(pk), bytes(h), bytes(sig))) for idx, pk, h, sig in items]


_POOL = {}


def cpu_pool(cores):
    import multiprocessing as mp
    if cores not in _POOL:
        _POOL[cores] = mp.get_context("fork").Pool(cores)
    return _POOL[cores]


def cpu_pairings(items, cores=None, kind=None):
    """ate_pairing of `items` = [(idx, a, b, P, Q)] on every host core -> (pairings/s, cores, {idx: 576 bytes}).
    Throughput = items / max over workers of the time spent inside ate_pairing (one worker per core)."""
    kind = kind or cpu_impl_kind()
    cores = cores or os.cpu_count() or 1
    pool = cpu_pool(cores)
    chunks = [items[k::cores] for k in range(cores)]
    res = pool.map(_cpu_pair_worker, [(kind, c) for c in chunks if c])
    slowest = max(dt for dt, _ in res)
    outs = {idx: raw for _, part in res for idx, raw in part}
    return len(items) / slowest, cores, outs


def sample_indices(seed, n, k):
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    return sorted(int(i) for i in rng.choice(n, size=min(k, n), replace=False))


DUMP_ROWS = 16384                # a quarter of the batch: 16,384 x 144 float64 words = 18.9 MB


def dump_outputs(path, out):
    """--dump-outputs: the GT elements of one batch (out: uint8, 576 bytes per pairing = 12 Fq coefficients of 48
    big-endian bytes) at DUMP_ROWS seeded row indices, written as
      DIR/pairings.npy         float64 (rows, 12, 12): each coefficient's big-endian 32-bit words, most significant
                               first (exact: every word < 2^53)
      DIR/pairing_rows.npy     float64 (rows,): the batch indices of those rows, ascending"""
    import numpy as np
    n = out.size // 576
    rows = np.array(sample_indices(0xD0D0, n, DUMP_ROWS), dtype=np.int64)
    words = out.view(">u4").reshape(n, 12, 12)[rows]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pairings.npy"), words.astype(np.float64))
    np.save(os.path.join(path, "pairing_rows.npy"), rows.astype(np.float64))


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (rank 0 only), a bounded sample of the
    same workload per step: inputs P_i = a_i G1, Q_i = b_i G2 for seeded indices of config 2's scalars"""
    if rank != 0:
        return
    from bls_b200 import synth
    kind = cpu_impl_kind()
    cores = os.cpu_count() or 1
    a = synth.scalars(synth.SEED_PAIRING, BATCH)
    b = synth.scalars(synth.SEED_PAIRING + 1, BATCH)
    per_core = 2
    idx_all = sample_indices(0xCB0, BATCH, per_core * cores * (args.warmup + args.steps))
    vals = []
    for step in range(args.warmup + args.steps):
        idx = idx_all[step * per_core * cores:(step + 1) * per_core * cores]
        items = [(i, int.from_bytes(bytes(a[i]), "big"), int.from_bytes(bytes(b[i]), "big"), None, None) for i in idx]
        v, cores, _ = cpu_pairings(items, cores, kind)
        if step >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    sample = "%d pairings per step (%d per core on %d cores) of the same seeded inputs" % (per_core * cores, per_core, cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * BATCH / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "python int (381-bit)",
            "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": value, "unit": METRIC, "cores": cores, "kind": kind, "sample": sample,
                             "extmod": extmod_note()},
            "e2e": {"value": value, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 8:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        pw = [float(s[3]) for s in self.samples if s[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples), "power_w_max": max(pw) if pw else None}


def build_id():
    """identity of the kernel sources + embedded programs: an ncu capture only speaks for the build it was taken from"""
    h = hashlib.sha256()
    base = os.path.join(ROOT, "python-bls_b200", "csrc")
    for nm in sorted(os.listdir(base)):
        if nm.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(base, nm), "rb").read())
    h.update(open(os.path.join(base, "gen", "programs.bin"), "rb").read())
    return h.hexdigest()[:16]


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_gpu(args, rank, world):
    import ctypes
    import numpy as np
    from bls_b200 import _lib, distributed as D, engine, synth, workloads as W
    from bls_b200._lib import check, lib
    from bls_b200.programs import registry
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.init(local)
    if world > 1:
        D.init(rank, world)

    def allmax(vals):
        """max over ranks of a list of floats (host gather: timing plumbing only)"""
        if world == 1:
            return list(vals)
        parts = D.gather_bytes(struct.pack("<%dd" % len(vals), *vals))
        cols = [struct.unpack("<%dd" % len(vals), p) for p in parts]
        return [max(c[k] for c in cols) for k in range(len(vals))]

    def barrier():
        check(lib.b200bls_sync())
        if world > 1:
            D.gather_bytes(b"\0")

    # throughput shape (4 = 384 items per SM, CTA-wide item blocks) and two streams: consecutive batches overlap
    SHAPE = int(os.environ.get("B200BLS_BENCH_SHAPE", "4"))
    N_STREAMS = int(os.environ.get("B200BLS_BENCH_STREAMS", "2"))
    check(lib.b200bls_set_ctas_per_sm(SHAPE))
    n = BATCH
    NSETS = 4                      # rotating buffer sets: NSETS * 56.6 MB of inputs + outputs exceed the 126 MB L2
    dP, dQ, a_sc, b_sc = W.config2_inputs(n, rank)
    sets = [(dP, dQ, engine.DeviceBuffer(576 * n))]
    hP, hQ = dP.download(), dQ.download()
    for _ in range(NSETS - 1):
        sets.append((engine.DeviceBuffer(96 * n).upload(hP), engine.DeviceBuffer(192 * n).upload(hQ),
                     engine.DeviceBuffer(576 * n)))

    def step(i):
        p, q, o = sets[i % NSETS]
        check(lib.b200bls_set_stream(i % N_STREAMS))
        check(lib.b200bls_pairing_batch_dev(p.ptr, q.ptr, o.ptr, n))

    peak_ops, _ = engine.microbench_imad(3, 8, 256, 200)     # integer-multiply peak, measured live

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = lib.b200bls_launch_count()
    engine.timer_start()
    for i in range(args.steps):
        step(args.warmup + i)
    ms = engine.timer_stop()
    launches = lib.b200bls_launch_count() - launches0
    barrier()
    clocks = sampler.stop()
    check(lib.b200bls_set_stream(0))
    last_out = sets[(args.warmup + args.steps - 1) % NSETS][2].download() if rank == 0 else None

    # --- end to end through the host-buffer C ABI call, pinned host memory, one buffer set per stream
    def pinned(nbytes):
        p = lib.b200bls_host_alloc(nbytes)
        if not p:
            raise RuntimeError("pinned allocation failed")
        return p, np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(nbytes,))
    host_sets = []
    for _ in range(N_STREAMS):
        pP, aP = pinned(96 * n)
        pQ, aQ = pinned(192 * n)
        pO, aO = pinned(576 * n)
        aP[:] = hP
        aQ[:] = hQ
        host_sets.append((pP, pQ, pO, aO))
    e2e_steps = max(2, min(args.steps, 24))
    for k in range(N_STREAMS):                                   # warm-up (staging allocation)
        check(lib.b200bls_set_stream(k))
        check(lib.b200bls_pairing_batch_async(host_sets[k][0], host_sets[k][1], host_sets[k][2], n))
    barrier()
    engine.timer_start()
    for i in range(e2e_steps):
        k = i % N_STREAMS
        check(lib.b200bls_set_stream(k))
        check(lib.b200bls_pairing_batch_async(host_sets[k][0], host_sets[k][1], host_sets[k][2], n))
    e2e_ms = engine.timer_stop()
    barrier()
    check(lib.b200bls_set_stream(0))
    aO = host_sets[(e2e_steps - 1) % N_STREAMS][3]

    # --- the isolated synchronous call a drop-in caller makes (automatic shape: balanced waves), host buffers
    check(lib.b200bls_set_ctas_per_sm(0))
    check(lib.b200bls_pairing_batch(host_sets[0][0], host_sets[0][1], host_sets[0][2], n))
    lone = 1e30
    for _ in range(2):
        t0 = time.perf_counter()
        check(lib.b200bls_pairing_batch(host_sets[0][0], host_sets[0][1], host_sets[0][2], n))
        lone = min(lone, time.perf_counter() - t0)
    lone_same = bool(np.array_equal(host_sets[0][3], aO))

    # --- parity (rank 0): sampled outputs vs the CPU implementation on the SAME input bytes (its timing is the
    # cpu_baseline), device-resident result == host-path result, digest of the whole output buffer
    parity, cpu = None, None
    if rank == 0:
        cores = os.cpu_count() or 1
        idx = sample_indices(0xB2C, n, 4 * cores)
        items = [(i, 0, 0, hP[96 * i:96 * (i + 1)].tobytes(), hQ[192 * i:192 * (i + 1)].tobytes()) for i in idx]
        cpu_v, cpu_cores, outs = cpu_pairings(items, cores)
        match = all(aO[576 * i:576 * (i + 1)].tobytes() == outs[i] for i in idx)
        parity = {"sampled_outputs_equal_cpu_%s" % cpu_impl_kind(): bool(match), "samples": len(idx),
                  "device_path_equals_host_path": bool(np.array_equal(last_out, aO)),
                  "isolated_call_equals_streamed": lone_same,
                  "output_sha256": hashlib.sha256(aO.tobytes()).hexdigest()}
        cpu = {"value": cpu_v, "unit": METRIC, "cores": cpu_cores, "kind": cpu_impl_kind(),
               "sample": "%d pairings (%d per core on %d cores) of this run's inputs at seeded indices; outputs compared "
                         "with the GPU's" % (len(idx), len(idx) // cpu_cores, cpu_cores),
               "extmod": extmod_note()}

    # --- signatures verified/s (hash-to-G2 + 2 Miller loops + final exponentiation): one full wave of VALID
    # signatures sig_i = a_i H(m_i) for the public keys pk_i = a_i G1 = P_i, throughput shape
    check(lib.b200bls_set_ctas_per_sm(SHAPE))
    nv = lib.b200bls_sm_count() * 384
    mh = synth.message_hashes(synth.SEED_BATCH_VERIFY + rank, nv)
    d_mh = engine.DeviceBuffer(32 * nv).upload(mh)
    d_pk = engine.DeviceBuffer(96 * nv).upload(hP[:96 * nv])
    d_h = engine.DeviceBuffer(192 * nv)
    check(lib.b200bls_hash_to_g2_batch_dev(d_mh.ptr, d_h.ptr, nv))
    d_sig = W.dev_scalar_mul(a_sc[:nv], True, base=d_h)
    d_ok = engine.DeviceBuffer(nv)
    check(lib.b200bls_verify_batch_dev(d_pk.ptr, d_mh.ptr, d_sig.ptr, d_ok.ptr, nv))
    verify_ms = W.timed(lambda: check(lib.b200bls_verify_batch_dev(d_pk.ptr, d_mh.ptr, d_sig.ptr, d_ok.ptr, nv)))
    verify_all_ok = bool(d_ok.download().all())
    pk48 = engine.compress(d_pk.download(), False)
    sig96 = engine.compress(d_sig.download(), True)
    ok_wire = np.empty(nv, dtype=np.uint8)
    check(lib.b200bls_verify_batch_wire(_lib.ptr(pk48), _lib.ptr(mh), _lib.ptr(sig96), _lib.ptr(ok_wire), nv))
    verify_wire_ms = W.timed(lambda: check(lib.b200bls_verify_batch_wire(_lib.ptr(pk48), _lib.ptr(mh), _lib.ptr(sig96),
                                                                         _lib.ptr(ok_wire), nv)), reps=1)
    verify_all_ok = verify_all_ok and bool(ok_wire.all())
    d_wo = engine.DeviceBuffer(576 * nv)
    check(lib.b200bls_pairing_batch_dev(d_pk.ptr, d_sig.ptr, d_wo.ptr, nv))
    wave_ms = W.timed(lambda: check(lib.b200bls_pairing_batch_dev(d_pk.ptr, d_sig.ptr, d_wo.ptr, nv)))
    for d in (d_mh, d_pk, d_h, d_sig, d_ok, d_wo):
        d.free()

    # --- BASELINE configs 3, 4, 5 at full size (per GPU: the path shards by contiguous slices)
    extra_cfg = run_configs(rank, world, allmax, barrier, D, W, engine, lib, check, np, synth, SHAPE)

    t = allmax([ms, e2e_ms, verify_ms, verify_wire_ms, wave_ms, lone * 1e3])
    ms, e2e_ms, verify_ms, verify_wire_ms, wave_ms, lone_ms = t
    if world > 1:
        barrier()
        D.shutdown()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_out)
    if world > 1:
        time.sleep(1.0)      # let the other ranks' exit chatter (NCCL_DEBUG lines share this stdout) precede the JSON line
    value = world * n * args.steps / (ms * 1e-3)
    e2e = world * n * e2e_steps / (e2e_ms * 1e-3)
    per_gpu = value / world
    executed_m = registry.executed_mults("pairing", 4)
    executed_m_verify = registry.executed_mults("verify_full", 4)
    achieved = per_gpu * executed_m * LIMB_PRODUCTS_PER_M
    hbm_bytes = n * (96 + 192 + 576)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # DRAM bytes of one launch of the pairing kernel at this batch size from the committed `ncu --set full` capture,
    # reported only if that capture was taken from THIS build (kernel sources + embedded programs)
    traffic, traffic_note = None, "no ncu capture of this build under profiles/"
    try:
        with open(os.path.join(ROOT, "profiles", "r2_pairing_ncu.json")) as fh:
            cap = json.load(fh)
        if cap.get("build_id") == build_id():
            traffic = cap["dram_bytes_per_launch"]
            traffic_note = "dram__bytes_read.sum + dram__bytes_write.sum of one launch, profiles/r2_pairing_ncu.json (same build)"
        else:
            traffic_note = "profiles/r2_pairing_ncu.json is from build %s, this is %s: not reported" % (cap.get("build_id"), build_id())
    except (OSError, ValueError, KeyError):
        pass
    line = {
        "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (381-bit Montgomery)",
        "data": "synthetic", "gpu_launches": int(launches),
        "config": {"workload": WORKLOAD, "batch_per_gpu": n, "l2": "inputs rotate over %d buffer sets (%d MB > L2)"
                   % (NSETS, NSETS * hbm_bytes // 2 ** 20), "ctas_per_sm": SHAPE, "streams": N_STREAMS, "parity": parity},
        "e2e": {"value": e2e, "unit": METRIC, "h2d_bytes_per_step": n * 288, "d2h_bytes_per_step": n * 576,
                "steps": e2e_steps, "api": "b200bls_pairing_batch_async + b200bls_sync (pinned host buffers, %d streams)" % N_STREAMS},
        "roofline": {"bound": "int32_mul", "achieved": achieved / 1e12, "peak": peak_ops / 1e12,
                     "unit": "T limb-products/s", "frac": achieved / peak_ops, "traffic": traffic,
                     "executed_M_per_unit": executed_m,
                     "frac_nominal": per_gpu * M_NOMINAL * LIMB_PRODUCTS_PER_M / peak_ops,
                     "note": "frac = pairings/s/GPU x the Montgomery products the pairing program really executes "
                             "(executed_M_per_unit, counted on the assembled code; inversions are ALU-pipe loops) x 300 limb "
                             "products / the IMAD.WIDE.U32.X carry-chain peak measured in this run; frac_nominal uses SURVEY "
                             "8d's frozen 15,200 M (work the program no longer does counts as done); algorithmic HBM bytes per "
                             "launch %d (%.4f of the measured HBM peak at this rate); traffic: %s"
                             % (hbm_bytes, (per_gpu * 864 / 1e9) / peaks.get("hbm_gbs", 6553.3), traffic_note)},
        "cpu_baseline": cpu,
        "clocks": clocks,
        "extra": dict({
            "verify_signatures_per_s": world * nv / (verify_ms * 1e-3), "verify_batch_per_gpu": nv,
            "verify_all_accepted": verify_all_ok,
            "verify_e2e_from_wire_bytes_per_s": world * nv / (verify_wire_ms * 1e-3),
            "verify_executed_M_per_unit": executed_m_verify,
            "verify_roofline_frac": (nv / (verify_ms * 1e-3)) * executed_m_verify * 300 / peak_ops,
            "verify_roofline_frac_nominal": (nv / (verify_ms * 1e-3)) * M_VERIFY_NOMINAL * 300 / peak_ops,
            "pairings_per_s_whole_wave_batches": world * nv / (wave_ms * 1e-3),
            "whole_wave_roofline_frac": (nv / (wave_ms * 1e-3)) * executed_m * 300 / peak_ops,
            "isolated_synchronous_call": {"api": "b200bls_pairing_batch (pinned host buffers, automatic shape)",
                                          "pairings": n, "ms": lone_ms, "pairings_per_s_per_gpu": n / (lone_ms * 1e-3)},
            "build_id": build_id()}, **extra_cfg),
    }
    print(json.dumps(line), flush=True)


def run_configs(rank, world, allmax, barrier, D, W, engine, lib, check, np, synth, shape):
    """BASELINE configs 3, 4, 5 at full size.  Single-GPU numbers on every rank's own data (weak), and under N > 1
    the SHARDED reductions (config 3 and 4 over all ranks' slices) through both exchange transports."""
    out = {}
    check(lib.b200bls_set_ctas_per_sm(0))
    # ---- config 3: 1 M G2 signatures + 1 M G1 keys, plain sums (this GPU alone)
    n3 = 1_000_000
    c3 = {"n_points": n3}
    for name, g2 in (("g2_signatures", True), ("g1_public_keys", False)):
        w = 192 if g2 else 96
        d_pts, cnt, tot = W.config3_slice(n3, g2)
        d_sum = engine.DeviceBuffer(w)
        fn = lib.b200bls_g2_sum_dev if g2 else lib.b200bls_g1_sum_dev
        check(fn(d_pts.ptr, d_sum.ptr, cnt))
        ms = W.timed(lambda: check(fn(d_pts.ptr, d_sum.ptr, cnt)))
        ok = d_sum.download().tobytes() == W.expected_multiple(tot, g2)
        ms = allmax([ms])[0]
        c3[name] = {"ms": ms, "adds_per_s_per_gpu": (n3 - 1) / (ms * 1e-3), "parity_sum_equals_scalar_sum_times_G": bool(ok)}
        # secure aggregation: the same points under 254-bit exponents t_i, sum_i t_i P_i as ONE multi-scalar
        # multiplication (bls.py:29-56, 217-221 multiply every point by its exponent and fold)
        tsc = synth.scalars(synth.SEED_AGGREGATE + 17, n3)
        d_t = engine.DeviceBuffer(32 * n3).upload(tsc)
        fm = lib.b200bls_g2_msm_dev if g2 else lib.b200bls_g1_msm_dev
        check(fm(d_pts.ptr, d_t.ptr, d_sum.ptr, cnt))
        ms_m = allmax([W.timed(lambda: check(fm(d_pts.ptr, d_t.ptr, d_sum.ptr, cnt)), reps=2)])[0]
        dot = sum(a * b for a, b in zip(W.ints(synth.scalars(synth.SEED_AGGREGATE, n3)), W.ints(tsc))) % W.N
        c3[name]["secure_msm"] = {"ms": ms_m, "points_per_s_per_gpu": n3 / (ms_m * 1e-3),
                                  "parity_equals_dot_product_times_G": bool(d_sum.download().tobytes() == W.expected_multiple(dot, g2))}
        d_t.free()
        d_pts.free()
        d_sum.free()
    out["config3_aggregate_1M"] = c3
    # ---- config 4: aggregate verification of 10,000 distinct messages (10,001 Miller loops, one final exponentiation)
    n4 = 10_000
    agg, pks, hs, _ = W.config4_inputs(n4)
    ok = engine.aggregate_verify(agg, pks, hs)
    best = 1e30
    for _ in range(3):
        t0 = time.perf_counter()
        ok = engine.aggregate_verify(agg, pks, hs) and ok
        best = min(best, time.perf_counter() - t0)
    hs_bad = hs.copy()
    hs_bad[7] = hs[8]
    rejected = not engine.aggregate_verify(agg, pks, hs_bad)
    jobs = [(agg, pks, hs)] * 16
    engine.aggregate_verify_many(jobs[:8])
    dt = 1e30
    for _ in range(2):
        t0 = time.perf_counter()
        res = engine.aggregate_verify_many(jobs)
        dt = min(dt, time.perf_counter() - t0)
    best, dt = allmax([best, dt])
    out["config4_aggregate_verify_10k"] = {
        "n_messages": n4, "accepts": bool(ok), "rejects_swapped_message": bool(rejected),
        "one_job_host_to_bool_ms": best * 1e3, "one_job_miller_loops_per_s": (n4 + 1) / best,
        "jobs_in_flight": {"jobs": len(jobs), "all_accept": bool(all(res)), "seconds": dt,
                           "miller_loops_per_s_per_gpu": len(jobs) * (n4 + 1) / dt}}
    # ---- config 5: this GPU's share (500,000 = 4 M / 8) of independent verifications, 1 % corrupted
    n5 = 500_000
    check(lib.b200bls_set_ctas_per_sm(shape))
    d_pk, d_hs, d_sig, want, (pk_h, hs_h, sig_h) = W.config5_inputs(n5, rank)
    d_ok = engine.DeviceBuffer(n5)
    check(lib.b200bls_verify_batch_dev(d_pk.ptr, d_hs.ptr, d_sig.ptr, d_ok.ptr, n5))
    ms5 = W.timed(lambda: check(lib.b200bls_verify_batch_dev(d_pk.ptr, d_hs.ptr, d_sig.ptr, d_ok.ptr, n5)), reps=2)
    res5 = d_ok.download()
    all_match = bool(np.array_equal(res5, want))
    cpu_ok = None
    if rank == 0:            # CPU implementation's BLS.verify on 8 accepted + 8 corrupted triples
        bad = np.flatnonzero(want == 0)[:8]
        good = np.flatnonzero(want == 1)[:8]
        items = [(int(i), pk_h[i].tobytes(), hs_h[i].tobytes(), sig_h[i].tobytes()) for i in list(good) + list(bad)]
        cores = os.cpu_count() or 1
        parts = cpu_pool(cores).map(_cpu_verify_worker, [(cpu_impl_kind(), items[k::cores]) for k in range(cores) if items[k::cores]])
        cpu_ok = all(bool(res5[i]) == v for part in parts for i, v in part)
    ms5 = allmax([ms5])[0]
    out["config5_batch_verify"] = {"n_per_gpu": n5, "corrupted_per_gpu": int((want == 0).sum()), "ms": ms5,
                                   "signatures_per_s": world * n5 / (ms5 * 1e-3),
                                   "all_booleans_match_ground_truth": all_match,
                                   "cpu_%s_verify_agrees_on_16_samples" % cpu_impl_kind(): cpu_ok}
    for d in (d_pk, d_hs, d_sig, d_ok):
        d.free()
    check(lib.b200bls_set_ctas_per_sm(0))
    # ---- N > 1: the sharded reductions, both transports (max over ranks; host buffers -> result on every rank)
    if world > 1:
        sh = {"nccl_initialised": bool(D.has_nccl()), "ranks": world}
        transports = [("host_gather", False)] + ([("nccl_allgather", True)] if D.has_nccl() else [])
        for n_tot in (1_000_000, 8_000_000):
            d_pts, cnt, tot = W.config3_slice(n_tot, True, rank, world)
            want_sum = W.expected_multiple(tot, True)
            row = {}
            for tname, nccl in transports:
                got = D.point_sum(d_pts, True, use_nccl=nccl) if cnt else D.point_sum(b"", True, use_nccl=nccl)
                barrier()
                best = 1e30
                for _ in range(3):
                    t0 = time.perf_counter()
                    got = D.point_sum(d_pts, True, use_nccl=nccl) if cnt else D.point_sum(b"", True, use_nccl=nccl)
                    best = min(best, time.perf_counter() - t0)
                    barrier()
                row[tname] = {"ms": allmax([best * 1e3])[0], "parity": bool(got == want_sum)}
            sh["config3_g2_sum_%dM_points" % (n_tot // 1_000_000)] = row
            d_pts.free()
        for n_tot in (10_000, 400_000):
            agg, pks, hs, _ = W.config4_inputs(n_tot, seed=synth.SEED_AGG_VERIFY + (1 if n_tot > 10_000 else 0))
            lo, hi = D.shard_range(n_tot, rank, world)
            row = {}
            for tname, nccl in transports:
                ok = D.aggregate_verify(agg, pks[96 * lo:96 * hi], hs[lo:hi], use_nccl=nccl)
                barrier()
                best = 1e30
                for _ in range(2):
                    t0 = time.perf_counter()
                    ok = D.aggregate_verify(agg, pks[96 * lo:96 * hi], hs[lo:hi], use_nccl=nccl) and ok
                    best = min(best, time.perf_counter() - t0)
                    barrier()
                ms_ = allmax([best * 1e3])[0]
                row[tname] = {"ms": ms_, "accepts": bool(ok), "miller_loops_per_s": (n_tot + 1) / (ms_ * 1e-3)}
            sh["config4_aggregate_verify_%d_messages" % n_tot] = row
        out["sharded_reductions"] = sh
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # default 12: K batches of 65,536 are K x 170.7 item blocks on 148 SMs, and the timed region ends with
    # a partly filled round (K = 5: 5.77 rounds -> 96 % of the steady-state rate, K = 12: 13.84 -> 98.9 %)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's output of the last timed step as .npy files into DIR (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    os.environ.setdefault("MASTER_PORT", "29533")
    run_gpu(args, rank, world)


if __name__ == "__main__":
    main()
