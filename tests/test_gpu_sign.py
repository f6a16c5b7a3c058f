"""GPU: batched signing and public-key derivation (b200bls_sign_batch / b200bls_public_key_batch and their _dev forms,
engine.sign_batch / public_keys, PrivateKey.sign_batch / sign_prehashed_batch / get_public_key_batch).

The new paths must give the bytes of the composition they replace -- hash_to_g2 + g2_scalar_mul + compress for
signatures, g1_scalar_mul on the generator + compress for public keys -- in every launch mode: each B200BLS_KERNEL
setting (unset, 1, 2) runs in its own subprocess, and inside it every launch shape (b200bls_set_ctas_per_sm 0..5) and
batches of 0, 1, 17, 129 and sm_count * 128 + 1, and one batch of 65,536 seeded pairs plus every edge key.  The
subprocess entry point is this file run as a script: `python test_gpu_sign.py <inputs.npz> <out.json>`.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (os.path.join(ROOT, "python-bls_b200"), os.path.join(ROOT, "oracle"), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import bls_oracle as O  # noqa: E402
import sign_corpus as SC  # noqa: E402

pytestmark = pytest.mark.gpu

SHAPES = (0, 1, 2, 3, 4, 5)
KERNELS = (None, "1", "2")
N_SEEDED = 65536


def _sk_bytes(keys):
    return np.frombuffer(b"".join(k.to_bytes(32, "big") for k in keys), dtype=np.uint8)


def _inputs():
    """every edge key, then seeded keys over the whole 32-byte range; seeded message hashes"""
    rng = np.random.Generator(np.random.PCG64(0xB2005160))
    keys = _sk_bytes(SC.edge_keys())
    sks = np.concatenate([keys, rng.integers(0, 256, size=32 * N_SEEDED, dtype=np.uint8)])
    hs = rng.integers(0, 256, size=sks.size, dtype=np.uint8)
    return sks, hs


def _composition(engine, sks, hs):
    """what the new calls replace: (affine signatures, wire signatures, affine keys, wire keys)"""
    from bls_b200.workloads import G1_BYTES
    n = sks.size // 32
    sig = engine.scalar_mul(engine.hash_to_g2(hs), sks, True)
    pk = engine.scalar_mul(np.tile(G1_BYTES, n), sks, False)
    return sig, engine.compress(sig, True), pk, engine.compress(pk, False)


def worker(in_path, out_path):
    from bls_b200 import _lib, engine
    _lib.init(0)
    data = np.load(in_path)
    sks, hs = data["sks"], data["hs"]
    sm = _lib.lib.b200bls_sm_count()
    res = {"kernel": os.environ.get("B200BLS_KERNEL"), "sm_count": sm, "bad": [], "runs": 0}
    ref = _composition(engine, sks, hs)
    widths = (192, 96, 96, 48)

    def compare(label, n):
        got = (engine.sign_batch(sks[:32 * n], hs[:32 * n]), engine.sign_batch(sks[:32 * n], hs[:32 * n], wire=True),
               engine.public_keys(sks[:32 * n]), engine.public_keys(sks[:32 * n], wire=True))
        for g, r, w, form in zip(got, ref, widths, ("sig", "sig_wire", "pk", "pk_wire")):
            res["runs"] += 1
            if g.size != n * w or not np.array_equal(g, r[:n * w]):
                idx = int(np.argmax(g != r[:n * w]) // w) if g.size == n * w else -1
                res["bad"].append("%s %s n=%d: first differing item %d" % (label, form, n, idx))
    compare("auto", sks.size // 32)
    for shape in SHAPES:
        _lib.check(_lib.lib.b200bls_set_ctas_per_sm(shape))
        for n in (0, 1, 17, 129, sm * 128 + 1):
            compare("shape%d" % shape, n)
    _lib.check(_lib.lib.b200bls_set_ctas_per_sm(0))
    with open(out_path, "w") as fh:
        json.dump(res, fh)


def test_every_mode_matches_the_composition(tmp_path):
    sks, hs = _inputs()
    path = tmp_path / "inputs.npz"
    np.savez(path, sks=sks, hs=hs)
    for kernel in KERNELS:
        env = dict(os.environ)
        env.pop("B200BLS_KERNEL", None)
        env.pop("B200BLS_CTAS_PER_SM", None)
        if kernel:
            env["B200BLS_KERNEL"] = kernel
        out = tmp_path / ("sign_%s.json" % (kernel or "auto"))
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), str(path), str(out)], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
        assert proc.returncode == 0, proc.stdout[-4000:]
        with open(out) as fh:
            res = json.load(fh)
        assert res["runs"] == 4 * (1 + len(SHAPES) * 5)
        assert not res["bad"], "B200BLS_KERNEL=%s: %s" % (kernel, res["bad"][:5])


def test_reference_vectors_both_forms():
    from bls_b200 import engine
    from conftest import load_golden
    g = load_golden("sig_kat.json")
    sks = [int(k["sk"], 16) for k in g["keys"]]
    assert engine.public_keys(sks, wire=True).tobytes().hex() == "".join(k["pk"] for k in g["keys"])
    aff = engine.public_keys(sks).tobytes()
    assert [aff[96 * i:96 * (i + 1)] for i in range(len(sks))] == [SC.g1_bytes(O.pk_of(k)) for k in sks]
    keys = [sks[s["key"]] for s in g["sign"]]
    hs = b"".join(O.hash256(bytes.fromhex(s["msg"])) for s in g["sign"])
    assert engine.sign_batch(keys, hs, wire=True).tobytes().hex() == "".join(s["sig"] for s in g["sign"])
    sig = engine.sign_batch(_sk_bytes(keys), hs).tobytes()
    assert engine.compress(sig, True).tobytes().hex() == "".join(s["sig"] for s in g["sign"])
    assert sig[:192] == SC.g2_bytes(O.sign_prehashed(keys[0], hs[:32]))


def test_oracle_samples():
    from bls_b200 import engine
    keys = SC.random_keys(64, 0x5167)
    hs = [O.hash256(b"sample %d" % i) for i in range(64)]
    sig = engine.sign_batch(keys, b"".join(hs)).tobytes()
    pk = engine.public_keys(keys).tobytes()
    for i, (k, h) in enumerate(zip(keys, hs)):
        assert sig[192 * i:192 * (i + 1)] == SC.g2_bytes(O.sign_prehashed(k, h)), i
        assert pk[96 * i:96 * (i + 1)] == SC.g1_bytes(O.pk_of(k)), i


def test_wire_round_trip_verifies():
    """wire outputs pass verification and its strict form; the zero key (sk = 0 mod n: infinity key and signature)
    is what strict verification rejects"""
    from bls_b200 import engine
    keys = SC.edge_keys() + SC.random_keys(200, 0x7717)
    hs = b"".join(O.hash256(b"round trip %d" % i) for i in range(len(keys)))
    sig = engine.sign_batch(keys, hs, wire=True)
    pk = engine.public_keys(keys, wire=True)
    zero = [k % O.N == 0 for k in keys]
    assert sum(zero) == 3
    ok = engine.verify_batch_wire(pk, hs, sig)
    strict = engine.verify_batch_wire(pk, hs, sig, strict=True)
    for i, z in enumerate(zero):
        if z:
            assert strict[i] == 0, i
        else:
            assert ok[i] == 1 and strict[i] == 1, (i, hex(keys[i]))


def test_python_batch_api_equals_per_call_signing():
    from bls_b200 import BLS
    from bls_b200 import PrivateKey as PK
    keys = [PK.from_seed(b"batch %d" % i) for i in range(6)] + [PK(0), PK(O.N + 3)]
    msgs = [b"message %d" % i for i in range(len(keys))]
    batch = PK.sign_batch(keys, msgs)
    one = [k.sign(m) for k, m in zip(keys, msgs)]
    for b, o in zip(batch, one):
        assert b.serialize() == o.serialize()
        assert b.value == o.value
        assert b.aggregation_info == o.aggregation_info
        assert b.aggregation_info.tree == o.aggregation_info.tree
    pks = PK.get_public_key_batch(keys)
    assert [p.serialize() for p in pks] == [k.get_public_key().serialize() for k in keys]
    hs = [O.hash256(m) for m in msgs]
    pre = PK.sign_prehashed_batch(keys, hs)
    assert [s.serialize() for s in pre] == [s.serialize() for s in one]
    assert PK.sign_batch([], []) == [] and PK.get_public_key_batch([]) == []
    with pytest.raises(ValueError):
        PK.sign_prehashed_batch(keys, hs[:-1])
    agg = BLS.aggregate_sigs(batch[:6])
    assert BLS.verify(agg)
    assert BLS.aggregate_sigs(batch[:6]).serialize() == BLS.aggregate_sigs(one[:6]).serialize()


def test_dev_forms_on_two_streams():
    from bls_b200 import _lib, engine
    from bls_b200._lib import check, lib
    keys = SC.random_keys(3000, 0x2222)
    hs = np.frombuffer(b"".join(O.hash256(b"stream %d" % i) for i in range(len(keys))), dtype=np.uint8)
    sks = _sk_bytes(keys)
    want_sig = engine.sign_batch(sks, hs, wire=True)
    want_pk = engine.public_keys(sks)
    n = len(keys)
    half = n // 2
    d_sk = engine.DeviceBuffer(sks.size).upload(sks)
    d_h = engine.DeviceBuffer(hs.size).upload(hs)
    d_sig = engine.DeviceBuffer(96 * n)
    d_pk = engine.DeviceBuffer(96 * n)
    try:
        for s, lo, hi in ((0, 0, half), (1, half, n)):
            check(lib.b200bls_set_stream(s))
            check(lib.b200bls_sign_batch_dev(1, d_sk.ptr + 32 * lo, d_h.ptr + 32 * lo, d_sig.ptr + 96 * lo, hi - lo))
            check(lib.b200bls_public_key_batch_dev(0, d_sk.ptr + 32 * lo, d_pk.ptr + 96 * lo, hi - lo))
        check(lib.b200bls_sync())
    finally:
        check(lib.b200bls_set_stream(0))
    assert np.array_equal(d_sig.download(), want_sig)
    assert np.array_equal(d_pk.download(), want_pk)
    # the caller's key buffer is untouched (only the library's own copies are zeroed); n = 0 does nothing
    assert np.array_equal(d_sk.download(), sks)
    check(lib.b200bls_sign_batch_dev(1, d_sk.ptr, d_h.ptr, d_sig.ptr, 0))
    assert lib.b200bls_sign_batch_dev(2, d_sk.ptr, d_h.ptr, d_sig.ptr, 1) == -3     # B200BLS_E_ARG
    assert lib.b200bls_public_key_batch(1, None, None, 1) == -3
    for b in (d_sk, d_h, d_sig, d_pk):
        b.free()
    assert _lib.lib.b200bls_sync() == 0


if __name__ == "__main__":
    worker(sys.argv[1], sys.argv[2])
