#!/usr/bin/env python3
"""Batched multi-pairing on one GPU, device-resident inputs, CUDA-event times.

Three workloads: 65,536 groups of 2 pairs (verifications), 4,096 groups of 16 (aggregates over a few messages) and one
group of 10,001 pairs.  The points are multiples of the generators by seeded scalars, computed on the device.  Each
workload compares one b200bls_pairing_multi_batch_dev call (check = 0) against a loop of b200bls_pairing_multi_dev, one
call per group: the way k products had to be computed before.  A per-group call is four dependent launches, so the loop
takes minutes for 65,536 groups; the loop arm therefore runs on the first LOOP_GROUPS groups of a workload, and the batch
arm is timed both on those groups (the comparison) and on the whole workload.  The arms alternate over REPS repetitions
and every time is kept; the launches of one call of each arm are counted, and the outputs of the loop's groups are
compared byte for byte.  The card's name and power limit are read in the same run.  Usage: bench_pairing_multi.py
OUT.json"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "python-bls_b200"))
from bls_b200 import _lib, engine, synth                    # noqa: E402
from bls_b200._lib import check, lib                        # noqa: E402
from bls_b200.workloads import G1_BYTES, G2_BYTES           # noqa: E402

WORKLOADS = [(65536, 2), (4096, 16), (1, 10001)]
REPS = 7
LOOP_GROUPS = 1024
SEED = 0xB2005EC5


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, check=True).stdout
    name, power, sm_max = [x.strip() for x in q.strip().split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": sm_max}


def time_ms(fn):
    engine.timer_start()
    fn()
    return engine.timer_stop()


def launches(fn):
    before = lib.b200bls_launch_count()
    fn()
    check(lib.b200bls_sync())
    return int(lib.b200bls_launch_count() - before)


def workload(n_groups, size, seed):
    total = n_groups * size
    d_p = engine.DeviceBuffer(96 * total)
    d_q = engine.DeviceBuffer(192 * total)
    d_gen1 = engine.DeviceBuffer(96 * total).upload(np.tile(G1_BYTES, total))
    d_gen2 = engine.DeviceBuffer(192 * total).upload(np.tile(G2_BYTES, total))
    d_k = engine.DeviceBuffer(32 * total).upload(synth.scalars(seed, total))
    check(lib.b200bls_g1_scalar_mul_batch_dev(d_gen1.ptr, d_k.ptr, d_p.ptr, total))
    d_k.upload(synth.scalars(seed + 1, total))
    check(lib.b200bls_g2_scalar_mul_batch_dev(d_gen2.ptr, d_k.ptr, d_q.ptr, total))
    check(lib.b200bls_sync())
    for b in (d_gen1, d_gen2, d_k):
        b.free()
    m = min(n_groups, LOOP_GROUPS)
    off = np.arange(n_groups + 1, dtype=np.uint64) * np.uint64(size)
    d_off = engine.DeviceBuffer(off.nbytes).upload(off)
    d_new = engine.DeviceBuffer(576 * n_groups)
    d_old = engine.DeviceBuffer(576 * m)

    def batch(k):
        return lambda: check(lib.b200bls_pairing_multi_batch_dev(0, d_p.ptr, d_q.ptr, d_off.ptr, k, d_new.ptr))

    def loop():
        for g in range(m):
            a = g * size
            check(lib.b200bls_pairing_multi_dev(ctypes.c_void_p(d_p.ptr + 96 * a), ctypes.c_void_p(d_q.ptr + 192 * a),
                                                ctypes.c_void_p(d_old.ptr + 576 * g), size))

    arms = {"per_group_loop": loop, "batch_same_groups": batch(m)}
    counts = {k: launches(fn) for k, fn in arms.items()}        # (also the warm-up)
    equal = bool(np.array_equal(d_old.download(), d_new.download(576 * m)))
    ms = {k: [] for k in arms}
    labels = list(arms)
    for r in range(REPS):
        for k in (labels if r % 2 == 0 else labels[::-1]):
            ms[k].append(time_ms(arms[k]))
    whole = batch(n_groups)
    counts["batch_whole"] = launches(whole)
    ms["batch_whole"] = [time_ms(whole) for _ in range(REPS)]
    ratios = [a / b for a, b in zip(ms["per_group_loop"], ms["batch_same_groups"])]
    pairs = {"per_group_loop": m * size, "batch_same_groups": m * size, "batch_whole": n_groups * size}
    res = {"groups": n_groups, "pairs_per_group": size, "loop_groups": m, "launches_per_call": counts, "ms": ms,
           "pairs_per_s_median": {k: pairs[k] / (np.median(v) / 1e3) for k, v in ms.items()},
           "speedup_same_groups": {"median": float(np.median(ratios)), "min": min(ratios), "max": max(ratios)},
           "bytes_equal": equal}
    for b in (d_p, d_q, d_off, d_new, d_old):
        b.free()
    return res


def main(out_path):
    _lib.init(0)
    res = {"card": card(), "reps": REPS, "workloads": []}
    for k, (n_groups, size) in enumerate(WORKLOADS):
        res["workloads"].append(workload(n_groups, size, SEED + 2 * k))
        print(json.dumps(res["workloads"][-1]), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)
    if not all(w["bytes_equal"] for w in res["workloads"]):
        sys.exit("the two arms' outputs differ")


if __name__ == "__main__":
    main(sys.argv[1])
