#!/usr/bin/env python3
"""Subgroup checks and strict verification on one GPU, device-resident inputs, CUDA-event times:

  (a) b200bls_subgroup_check_batch_dev on 1 M G1 and 1 M G2 points (k_i G);
  (b) b200bls_verify_batch_wire_dev against b200bls_verify_batch_wire_strict_dev on the same 262,144 seeded wire
      triples, alternated over several repetitions (each repetition's time is kept, so the spread is visible).

The card's name and power limit are read in the same run.  Usage: bench_subgroup.py OUT.json"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "python-bls_b200"))
from bls_b200 import _lib, engine, synth                    # noqa: E402
from bls_b200._lib import check, lib                        # noqa: E402
from bls_b200.programs import registry                      # noqa: E402
from bls_b200.workloads import dev_scalar_mul               # noqa: E402

N_POINTS = 1 << 20
N_VERIFY = 262144
REPS = 7


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, check=True).stdout
    name, power, sm_max = [x.strip() for x in q.strip().split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": sm_max}


def time_ms(fn):
    engine.timer_start()
    fn()
    return engine.timer_stop()


def bench_subgroup(g2):
    d_pts = dev_scalar_mul(synth.scalars(0xB2005B10 + g2, N_POINTS), bool(g2))
    d_ok = engine.DeviceBuffer(N_POINTS)
    run = lambda: check(lib.b200bls_subgroup_check_batch_dev(g2, d_pts.ptr, d_ok.ptr, N_POINTS))  # noqa: E731
    run()                                                   # warm-up
    ms = [time_ms(run) for _ in range(REPS)]
    ok = d_ok.download()
    d_pts.free()
    d_ok.free()
    return {"points": N_POINTS, "ms": ms, "all_members": bool(ok.all()),
            "points_per_s_best": N_POINTS / (min(ms) / 1e3), "points_per_s_median": N_POINTS / (np.median(ms) / 1e3)}


def bench_verify():
    sks = synth.scalars(synth.SEED_BATCH_VERIFY, N_VERIFY)
    hs = synth.message_hashes(synth.SEED_BATCH_VERIFY, N_VERIFY)
    sig96 = engine.compress(engine.scalar_mul(engine.hash_to_g2(hs), sks, True), True)
    pk48 = engine.compress(dev_scalar_mul(sks, False).download(), False)
    d_pk, d_hs, d_sig = (engine.DeviceBuffer(a.size).upload(a) for a in (pk48, hs, sig96))
    d_ok = {s: engine.DeviceBuffer(N_VERIFY) for s in (False, True)}
    fns = {False: lib.b200bls_verify_batch_wire_dev, True: lib.b200bls_verify_batch_wire_strict_dev}

    def run(strict):
        check(fns[strict](d_pk.ptr, d_hs.ptr, d_sig.ptr, d_ok[strict].ptr, N_VERIFY))
    run(False)
    run(True)
    ms = {False: [], True: []}
    for r in range(REPS):
        for strict in ((False, True) if r % 2 == 0 else (True, False)):
            ms[strict].append(time_ms(lambda: run(strict)))
    ok = {s: d_ok[s].download() for s in (False, True)}
    ratios = [a / b for a, b in zip(ms[False], ms[True])]     # strict rate / non-strict rate, per repetition
    out = {"triples": N_VERIFY, "all_true": bool(ok[False].all() and ok[True].all()),
           "nonstrict_ms": ms[False], "strict_ms": ms[True],
           "nonstrict_per_s_median": N_VERIFY / (np.median(ms[False]) / 1e3),
           "strict_per_s_median": N_VERIFY / (np.median(ms[True]) / 1e3),
           "strict_over_nonstrict_rate": {"median": float(np.median(ratios)), "min": min(ratios), "max": max(ratios)}}
    for b in (d_pk, d_hs, d_sig, *d_ok.values()):
        b.free()
    return out


def main(out_path):
    _lib.init(0)
    res = {"card": card(),
           "executed_mults_per_item": {n: registry.executed_mults(n) for n in
                                       ("g1_subgroup", "g2_subgroup", "g1_decompress", "g2_decompress",
                                        "verify_full")},
           "subgroup_check_g1": bench_subgroup(0), "subgroup_check_g2": bench_subgroup(1),
           "verify_wire": bench_verify()}
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main(sys.argv[1])
