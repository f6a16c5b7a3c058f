#!/usr/bin/env python3
"""Batched signing and public-key derivation on one GPU, device-resident inputs, CUDA-event times.

  (a) signatures of 2^20 seeded (secret key, message hash) pairs in wire form: the composition that existed before
      (b200bls_hash_to_g2_batch_dev, b200bls_g2_scalar_mul_batch_dev, then the g2_cflag program for the compression
      flags) against b200bls_sign_batch_dev(wire = 1);
  (b) public keys of the same 2^20 keys: b200bls_g1_scalar_mul_batch_dev on copies of the generator plus g1_cflag
      against b200bls_public_key_batch_dev(wire = 1).

The composition arms stop at the flags: the library has no device-pointer form of the compression pack, a byte copy
that the new arms do include.  The arms alternate over REPS repetitions and every time is kept.  The outputs are
compared byte for byte (the composition's bytes packed on the host).  The card's name and power limit are read in the
same run.  Usage: bench_sign.py OUT.json"""
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
from bls_b200.workloads import G1_BYTES                     # noqa: E402

N = 1 << 20
REPS = 7
SEED = 0xB2005167


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, check=True).stdout
    name, power, sm_max = [x.strip() for x in q.strip().split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": sm_max}


def time_ms(fn):
    engine.timer_start()
    fn()
    return engine.timer_stop()


def pack(aff, flags, xb):
    """the compressed points from affine points and flag bytes (the compression pack, on the host)"""
    out = aff.reshape(-1, 2 * xb)[:, :xb].copy()
    out[:, 0] |= (flags.reshape(-1) != 0).astype(np.uint8) << 7
    return out.reshape(-1)


def run_program(name, bufs, strides):
    engine.run_program_dev(name, N, bufs, strides)


def alternate(arms):
    """arms: {label: fn}; every repetition runs each arm once, the order reversed on odd repetitions"""
    for fn in arms.values():
        fn()                                                # warm-up
    ms = {k: [] for k in arms}
    labels = list(arms)
    for r in range(REPS):
        for k in (labels if r % 2 == 0 else labels[::-1]):
            ms[k].append(time_ms(arms[k]))
    return ms


def summary(ms_old, ms_new):
    ratios = [a / b for a, b in zip(ms_old, ms_new)]        # new rate / old rate, per repetition
    return {"items": N, "composition_ms": ms_old, "new_ms": ms_new,
            "composition_per_s_median": N / (np.median(ms_old) / 1e3), "new_per_s_median": N / (np.median(ms_new) / 1e3),
            "speedup": {"median": float(np.median(ratios)), "min": min(ratios), "max": max(ratios)}}


def main(out_path):
    _lib.init(0)
    sks = synth.scalars(SEED, N)
    hs = synth.message_hashes(SEED, N)
    d_sk = engine.DeviceBuffer(32 * N).upload(sks)
    d_h = engine.DeviceBuffer(32 * N).upload(hs)
    d_gen = engine.DeviceBuffer(96 * N).upload(np.tile(G1_BYTES, N))
    d_hash = engine.DeviceBuffer(192 * N)
    d_sig = engine.DeviceBuffer(192 * N)
    d_pk = engine.DeviceBuffer(96 * N)
    d_flag = engine.DeviceBuffer(N)
    d_new_sig = engine.DeviceBuffer(96 * N)
    d_new_pk = engine.DeviceBuffer(48 * N)

    def old_sign():
        check(lib.b200bls_hash_to_g2_batch_dev(d_h.ptr, d_hash.ptr, N))
        check(lib.b200bls_g2_scalar_mul_batch_dev(d_hash.ptr, d_sk.ptr, d_sig.ptr, N))
        run_program("g2_cflag", [d_sig, d_flag], [192, 1])

    def new_sign():
        check(lib.b200bls_sign_batch_dev(1, d_sk.ptr, d_h.ptr, d_new_sig.ptr, N))

    def old_pk():
        check(lib.b200bls_g1_scalar_mul_batch_dev(d_gen.ptr, d_sk.ptr, d_pk.ptr, N))
        run_program("g1_cflag", [d_pk, d_flag], [96, 1])

    def new_pk():
        check(lib.b200bls_public_key_batch_dev(1, d_sk.ptr, d_new_pk.ptr, N))

    res = {"card": card(),
           "executed_mults_per_item": {n: registry.executed_mults(n) for n in
                                       ("hash_to_g2", "g2_mul", "g2_sign", "g1_mul", "g1_pubkey")}}
    ms = alternate({"old": old_sign, "new": new_sign})
    res["sign"] = summary(ms["old"], ms["new"])
    old_sign()
    check(lib.b200bls_sync())
    res["sign"]["bytes_equal"] = bool(np.array_equal(pack(d_sig.download(), d_flag.download(), 96),
                                                     d_new_sig.download()))
    ms = alternate({"old": old_pk, "new": new_pk})
    res["public_key"] = summary(ms["old"], ms["new"])
    old_pk()
    check(lib.b200bls_sync())
    res["public_key"]["bytes_equal"] = bool(np.array_equal(pack(d_pk.download(), d_flag.download(), 48),
                                                           d_new_pk.download()))
    res["card_after"] = card()
    for b in (d_sk, d_h, d_gen, d_hash, d_sig, d_pk, d_flag, d_new_sig, d_new_pk):
        b.free()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))
    if not (res["sign"]["bytes_equal"] and res["public_key"]["bytes_equal"]):
        sys.exit("the two arms' outputs differ")


if __name__ == "__main__":
    main(sys.argv[1])
