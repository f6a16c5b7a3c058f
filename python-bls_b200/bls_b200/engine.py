"""Batched byte-buffer operations on the GPU (thin, typed layer over the C ABI).

All inputs/outputs are numpy uint8 arrays (or bytes) in the reference's serialisation
(48-byte big-endian coefficients).  This is the layer the bls_py-compatible classes and
bench.py call; it owns no arithmetic.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import as_u8, check, lib, ptr
from .util import GROUP_ORDER

FIELD_OPS = {"add": 0, "sub": 1, "mul": 2, "sqr": 3, "neg": 4, "inv": 5}


def field_op(level, op, a, b=None):
    """n elements of tower level 1/2/6/12 -> n results; a, b: n * 48 * level bytes"""
    _lib.init()
    a = as_u8(a)
    w = 48 * level
    n = a.size // w
    if a.size != n * w:
        raise ValueError("operand size is not a multiple of %d" % w)
    opc = FIELD_OPS[op]
    bb = as_u8(b, a.size) if opc <= 2 else None
    out = np.empty(n * w, dtype=np.uint8)
    check(lib.b200bls_field_op_batch(level, opc, ptr(a), ptr(bb) if bb is not None else None, ptr(out), n))
    return out


def field_frob(level, i, a):
    """x -> x^(q^i) for n elements of tower level 2 / 6 / 12 (qi_pow, fields_t.py:104-110, 203-212, 355-364)"""
    _lib.init()
    a = as_u8(a)
    w = 48 * level
    n = a.size // w
    if a.size != n * w:
        raise ValueError("operand size is not a multiple of %d" % w)
    out = np.empty(n * w, dtype=np.uint8)
    check(lib.b200bls_field_frob_batch(level, i, ptr(a), ptr(out), n))
    return out


def field_pow(level, a, exponents):
    """x_k -> x_k^(e_k): exponents is a list of non-negative ints < 2^384, or n x 48 big-endian bytes"""
    _lib.init()
    a = as_u8(a)
    w = 48 * level
    n = a.size // w
    if a.size != n * w:
        raise ValueError("operand size is not a multiple of %d" % w)
    if not isinstance(exponents, (bytes, bytearray, np.ndarray)):
        exponents = b"".join(int(e).to_bytes(48, "big") for e in exponents)
    e = as_u8(exponents, 48 * n)
    out = np.empty(n * w, dtype=np.uint8)
    check(lib.b200bls_field_pow_batch(level, ptr(a), ptr(e), ptr(out), n))
    return out


def field_sqrt(level, a):
    """the reference's modsqrt on n elements of Fq (level 1) or Fq2 (level 2) -> (roots, ok flags)"""
    _lib.init()
    a = as_u8(a)
    w = 48 * level
    n = a.size // w
    if a.size != n * w:
        raise ValueError("operand size is not a multiple of %d" % w)
    out = np.empty(n * w, dtype=np.uint8)
    ok = np.empty(n, dtype=np.uint8)
    check(lib.b200bls_field_sqrt_batch(level, ptr(a), ptr(out), ptr(ok), n))
    return out, ok


def _map(fn, data, w_in, w_out):
    _lib.init()
    data = as_u8(data)
    n = data.size // w_in
    if data.size != n * w_in:
        raise ValueError("buffer size is not a multiple of %d" % w_in)
    out = np.empty(n * w_out, dtype=np.uint8)
    check(fn(ptr(data), ptr(out), n))
    return out


JACOBIAN_OPS = {"affine": 0, "dbl": 1, "add": 2, "mul": 3}


def jacobian_op(op, a, b, g2):
    """the reference's Jacobian-coordinate functions on n JACOBIAN points a = (X, Y, Z) (3 x 48 / 96 bytes, Z = 0 for
    infinity): to_affine, double, add (b = n Jacobian points), scalar mult (b = n x 32-byte scalars) -> n AFFINE points"""
    _lib.init()
    a = as_u8(a)
    w = 96 if g2 else 48
    n = a.size // (3 * w)
    if a.size != n * 3 * w:
        raise ValueError("Jacobian points are %d bytes" % (3 * w))
    opc = JACOBIAN_OPS[op]
    bb = as_u8(b, n * (32 if opc == 3 else 3 * w)) if opc >= 2 else None
    out = np.empty(n * 2 * w, dtype=np.uint8)
    check(lib.b200bls_jacobian_op_batch(int(bool(g2)), opc, ptr(a), ptr(bb) if bb is not None else None, ptr(out), n))
    return out


def sw_encode_g2(t):
    """n x 96-byte Fq2 values -> n affine points of the twist (ec.py:449-507; infinity = zero bytes)"""
    return _map(lib.b200bls_sw_encode_g2_batch, t, 96, 192)


def g2_untwist(points):
    """n affine twist points (192 B) -> n x (x', y') over Fq12 (2 x 576 B): fq2_untwist, fields_t.py:936-943"""
    return _map(lib.b200bls_g2_untwist_batch, points, 192, 1152)


def fq12_twist(points):
    """n x (x, y) over Fq12 -> n x (x w^2, y w^3): fq12_twist, fields_t.py:1018-1031"""
    return _map(lib.b200bls_fq12_twist_batch, points, 1152, 1152)


def g2_psi(points):
    """psi = twist . Frobenius . untwist on n affine twist points (ec.py:440-444)"""
    return _map(lib.b200bls_g2_psi_batch, points, 192, 192)


def _pq(P, Q):
    P, Q = as_u8(P), as_u8(Q)
    n = P.size // 96
    if P.size != n * 96 or Q.size != n * 192:
        raise ValueError("P must be n*96 bytes and Q n*192 bytes")
    return P, Q, n


def pairing_batch(P, Q):
    """n independent ate pairings -> n * 576 bytes (bls_py.pairing.ate_pairing per pair)"""
    _lib.init()
    P, Q, n = _pq(P, Q)
    out = np.empty(n * 576, dtype=np.uint8)
    check(lib.b200bls_pairing_batch(ptr(P), ptr(Q), ptr(out), n))
    return out


def miller_loop_batch(P, Q):
    _lib.init()
    P, Q, n = _pq(P, Q)
    out = np.empty(n * 576, dtype=np.uint8)
    check(lib.b200bls_miller_loop_batch(ptr(P), ptr(Q), ptr(out), n))
    return out


def final_exp_batch(f):
    _lib.init()
    f = as_u8(f)
    n = f.size // 576
    out = np.empty(n * 576, dtype=np.uint8)
    check(lib.b200bls_final_exp_batch(ptr(f), ptr(out), n))
    return out


def miller_product(P, Q):
    """prod_i miller(P_i, Q_i) as 576 bytes, NOT final-exponentiated (rank partial)"""
    _lib.init()
    P, Q, n = _pq(P, Q)
    out = np.empty(576, dtype=np.uint8)
    check(lib.b200bls_miller_product(ptr(P) if n else None, ptr(Q) if n else None, ptr(out), n))
    return out


def pairing_multi(P, Q):
    """bls_py.pairing.ate_pairing_multi on byte buffers -> 576 bytes"""
    _lib.init()
    P, Q, n = _pq(P, Q)
    out = np.empty(576, dtype=np.uint8)
    check(lib.b200bls_pairing_multi(ptr(P) if n else None, ptr(Q) if n else None, ptr(out), n))
    return out


def _g(g2):
    return ("g2", 192) if g2 else ("g1", 96)


def scalar_mul(points, scalars, g2):
    """n affine points x n 32-byte big-endian scalars -> n affine points"""
    _lib.init()
    name, w = _g(g2)
    points, scalars = as_u8(points), as_u8(scalars)
    n = points.size // w
    if points.size != n * w or scalars.size != n * 32:
        raise ValueError("bad buffer sizes")
    out = np.empty(n * w, dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_scalar_mul_batch" % name)(ptr(points), ptr(scalars), ptr(out), n))
    return out


def point_add(a, b, g2):
    _lib.init()
    name, w = _g(g2)
    a, b = as_u8(a), as_u8(b)
    n = a.size // w
    if a.size != n * w or b.size != a.size:
        raise ValueError("bad buffer sizes")
    out = np.empty(n * w, dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_add_batch" % name)(ptr(a), ptr(b), ptr(out), n))
    return out


def point_sum(points, g2):
    """sum of n affine points -> one affine point (infinity = zero bytes)"""
    _lib.init()
    name, w = _g(g2)
    points = as_u8(points)
    n = points.size // w
    if points.size != n * w:
        raise ValueError("bad buffer size")
    out = np.empty(w, dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_sum" % name)(ptr(points) if n else None, ptr(out), n))
    return out


def decompress(data, g2):
    """compressed points -> (affine bytes, ok flags)"""
    _lib.init()
    name, w = _g(g2)
    data = as_u8(data)
    n = data.size // (w // 2)
    if data.size != n * (w // 2):
        raise ValueError("bad buffer size")
    out = np.empty(n * w, dtype=np.uint8)
    ok = np.empty(n, dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_decompress_batch" % name)(ptr(data), ptr(out), ptr(ok), n))
    return out, ok


def subgroup_check(points, g2):
    """n affine points (96 / 192 B) -> n flag bytes: 1 iff the point is on the curve and in G1 / G2.  Coordinates are
    read mod q like every affine input here, and infinity counts as a member: any coordinates that reduce to (0, 0),
    zero bytes as well as q per coordinate"""
    _lib.init()
    w = _g(g2)[1]
    points = as_u8(points)
    n = points.size // w
    if points.size != n * w:
        raise ValueError("bad buffer size")
    ok = np.empty(n, dtype=np.uint8)
    check(lib.b200bls_subgroup_check_batch(int(bool(g2)), ptr(points), ptr(ok), n))
    return ok


def key_validate(points):
    """n affine G1 points (96 B) -> n flag bytes: 1 iff the point is in G1 and is not infinity (the public-key rule of
    strict verification), decided on the coordinates reduced mod q"""
    _lib.init()
    points = as_u8(points)
    n = points.size // 96
    if points.size != n * 96:
        raise ValueError("bad buffer size")
    ok = np.empty(n, dtype=np.uint8)
    check(lib.b200bls_key_validate_batch(ptr(points), ptr(ok), n))
    return ok


def compress(points, g2):
    _lib.init()
    name, w = _g(g2)
    points = as_u8(points)
    n = points.size // w
    if points.size != n * w:
        raise ValueError("bad buffer size")
    out = np.empty(n * (w // 2), dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_compress_batch" % name)(ptr(points), ptr(out), n))
    return out


def msm(points, scalars, g2):
    """sum_i k_i * P_i: n affine points x n 32-byte big-endian scalars -> one affine point"""
    _lib.init()
    name, w = _g(g2)
    points, scalars = as_u8(points), as_u8(scalars)
    n = points.size // w
    if points.size != n * w or scalars.size != n * 32:
        raise ValueError("bad buffer sizes")
    out = np.empty(w, dtype=np.uint8)
    check(getattr(lib, "b200bls_%s_msm" % name)(ptr(points), ptr(scalars), ptr(out), n))
    return out


def hash_pks(pk_hash, n, first=0):
    """aggregation exponents T_first .. T_(first+n-1) = SHA256(i || pk_hash) mod n -> n x 32 bytes
    (the per-key part of bls_py.util.hash_pks, util.py:46-49)"""
    _lib.init()
    pk_hash = as_u8(pk_hash, 32)
    out = np.empty(n * 32, dtype=np.uint8)
    check(lib.b200bls_hash_pks(ptr(pk_hash), first, ptr(out), n))
    return out


def hash_to_g2(hashes):
    """n x 32-byte message hashes -> n x 192 bytes (hash_to_point_prehashed_Fq2)"""
    _lib.init()
    hashes = as_u8(hashes)
    n = hashes.size // 32
    if hashes.size != n * 32:
        raise ValueError("bad buffer size")
    out = np.empty(n * 192, dtype=np.uint8)
    check(lib.b200bls_hash_to_g2_batch(ptr(hashes), ptr(out), n))
    return out


def _secret_keys(sks):
    """ints (taken mod the group order) or n x 32 big-endian bytes -> uint8 array of n x 32 bytes"""
    if isinstance(sks, (bytes, bytearray, np.ndarray)):
        sks = as_u8(sks)
        if sks.size % 32:
            raise ValueError("secret keys are 32 bytes each")
        return sks
    return np.frombuffer(b"".join((int(k) % GROUP_ORDER).to_bytes(32, "big") for k in sks), dtype=np.uint8)


def sign_batch(sks, hashes, wire=False):
    """PrivateKey.sign_prehashed for n (secret key, 32-byte message hash) pairs in one device pass: sks are ints or
    n x 32 big-endian bytes -> n x 192 affine bytes, or n x 96 Signature.serialize() bytes with wire=True"""
    _lib.init()
    sks, hashes = _secret_keys(sks), as_u8(hashes)
    n = hashes.size // 32
    if hashes.size != 32 * n or sks.size != 32 * n:
        raise ValueError("bad buffer sizes")
    out = np.empty(n * (96 if wire else 192), dtype=np.uint8)
    check(lib.b200bls_sign_batch(int(bool(wire)), ptr(sks), ptr(hashes), ptr(out), n))
    return out


def public_keys(sks, wire=False):
    """PrivateKey.get_public_key for n secret keys (ints or n x 32 big-endian bytes) in one device pass -> n x 96
    affine bytes, or n x 48 PublicKey.serialize() bytes with wire=True"""
    _lib.init()
    sks = _secret_keys(sks)
    n = sks.size // 32
    out = np.empty(n * (48 if wire else 96), dtype=np.uint8)
    check(lib.b200bls_public_key_batch(int(bool(wire)), ptr(sks), ptr(out), n))
    return out


def aggregate_miller(sig, pks, hashes):
    """[e(-G1, sig) *] prod_i miller(pk_i, H(hash_i)) as 576 bytes, not final-exponentiated: one
    rank's partial of a sharded aggregate verification (sig = None: no signature pair)"""
    _lib.init()
    pks, hashes = as_u8(pks), as_u8(hashes)
    n = hashes.size // 32
    if pks.size != 96 * n or hashes.size != 32 * n:
        raise ValueError("bad buffer sizes")
    s = as_u8(sig, 192) if sig is not None else None
    out = np.empty(576, dtype=np.uint8)
    check(lib.b200bls_aggregate_miller(ptr(s) if s is not None else None, ptr(pks) if n else None,
                                       ptr(hashes) if n else None, n, ptr(out)))
    return out


def verify_batch_wire(pks48, hashes, sigs96, strict=False):
    """n x (serialised pk 48 B, message hash 32 B, serialised sig 96 B) -> n result bytes; inputs that
    do not decode are rejections.  strict=True: also rejects keys outside G1, the infinity key and
    signatures outside G2 (the reference accepts them)"""
    _lib.init()
    pks48, hashes, sigs96 = as_u8(pks48), as_u8(hashes), as_u8(sigs96)
    n = hashes.size // 32
    if pks48.size != 48 * n or hashes.size != 32 * n or sigs96.size != 96 * n:
        raise ValueError("bad buffer sizes")
    out = np.empty(n, dtype=np.uint8)
    fn = lib.b200bls_verify_batch_wire_strict if strict else lib.b200bls_verify_batch_wire
    check(fn(ptr(pks48), ptr(hashes), ptr(sigs96), ptr(out), n))
    return out


def verify_batch(pks, hashes, sigs, strict=False):
    """n x (pk 96 B, message hash 32 B, sig 192 B) -> n result bytes.  strict=True: also rejects keys
    outside G1, the infinity key and signatures outside G2 (the reference accepts them)"""
    _lib.init()
    pks, hashes, sigs = as_u8(pks), as_u8(hashes), as_u8(sigs)
    n = hashes.size // 32
    if pks.size != 96 * n or hashes.size != 32 * n or sigs.size != 192 * n:
        raise ValueError("bad buffer sizes")
    ok = np.empty(n, dtype=np.uint8)
    fn = lib.b200bls_verify_batch_strict if strict else lib.b200bls_verify_batch
    check(fn(ptr(pks), ptr(hashes), ptr(sigs), ptr(ok), n))
    return ok


def aggregate_verify(sig, pks, hashes):
    """one aggregate signature (192 B affine) over n distinct message hashes -> bool"""
    _lib.init()
    sig, pks, hashes = as_u8(sig, 192), as_u8(pks), as_u8(hashes)
    n = hashes.size // 32
    if pks.size != 96 * n or hashes.size != 32 * n:
        raise ValueError("bad buffer sizes")
    ok = np.zeros(1, dtype=np.uint8)
    check(lib.b200bls_aggregate_verify(ptr(sig), ptr(pks) if n else None, ptr(hashes) if n else None, n, ptr(ok)))
    return bool(ok[0])


_PINNED = {}                # slot -> [pointer, capacity]: pinned staging, grown on demand, kept for the process


def _pinned_array(slot, nbytes):
    """uint8 view of nbytes of pinned host memory owned by `slot` (cudaHostAlloc / cudaFreeHost
    synchronise the device, so the buffers are cached instead of allocated per call)"""
    ent = _PINNED.get(slot)
    if ent is None or ent[1] < nbytes:
        if ent is not None:
            lib.b200bls_host_free(ctypes.c_void_p(ent[0]))
        cap = max(4096, nbytes + nbytes // 4)
        p = lib.b200bls_host_alloc(cap)
        if not p:
            _PINNED.pop(slot, None)
            raise _lib.B200BlsError("pinned allocation of %d bytes failed" % cap)
        ent = _PINNED[slot] = [p, cap]
    return np.ctypeslib.as_array(ctypes.cast(ent[0], ctypes.POINTER(ctypes.c_uint8)), shape=(ent[1],))[:nbytes]


def aggregate_verify_many(jobs):
    """several aggregate verifications in flight at once: jobs = [(sig 192 B, pks n x 96 B, hashes
    n x 32 B), ...] are enqueued round-robin on the library's streams and waited for together ->
    list of bool.  A 10,000-message job fills about a fifth of a B200, so sequential calls leave
    most of it idle.  Inputs are staged through pinned memory (one cached buffer per stream) and the
    result bytes land in pinned memory: copies from / to pageable memory block the host until they
    have run, which serialises the jobs and made the throughput jitter by 2-4x."""
    _lib.init()
    jobs = list(jobs)
    if not jobs:
        return []
    n_streams = lib.b200bls_stream_count()
    res = _pinned_array("res", len(jobs))
    res[:] = 0
    # throughput shape for jobs that share the GPU (the automatic choice is the lowest-latency shape,
    # whose CTAs take a whole SM each and do not leave room for a second job)
    prev_shape = lib.b200bls_get_ctas_per_sm()
    if prev_shape == 0 and len(jobs) > 1:
        check(lib.b200bls_set_ctas_per_sm(4))
    try:
        for k, (sig, pks, hashes) in enumerate(jobs):
            sig, pks, hashes = as_u8(sig, 192), as_u8(pks), as_u8(hashes)
            n = hashes.size // 32
            if pks.size != 96 * n or hashes.size != 32 * n:
                raise ValueError("bad buffer sizes")
            if k >= n_streams and k % n_streams == 0:
                check(lib.b200bls_sync())            # staging buffers are per stream: one job per stream in flight
            stage = _pinned_array(("in", k % n_streams), 192 + 128 * n)
            stage[:192] = sig
            stage[192:192 + 96 * n] = pks
            stage[192 + 96 * n:] = hashes
            base = stage.ctypes.data
            check(lib.b200bls_set_stream(k % n_streams))
            check(lib.b200bls_aggregate_verify_async(ctypes.c_void_p(base), ctypes.c_void_p(base + 192) if n else None,
                                                     ctypes.c_void_p(base + 192 + 96 * n) if n else None,
                                                     n, ctypes.c_void_p(res.ctypes.data + k)))
        check(lib.b200bls_sync())
        out = [bool(v) for v in res]
    finally:
        check(lib.b200bls_set_stream(0))
        lib.b200bls_sync()
        lib.b200bls_set_ctas_per_sm(prev_shape)
    return out


class DeviceBuffer:
    """device memory owned by the library (for resident-data pipelines and benchmarks)"""

    def __init__(self, nbytes):
        _lib.init()
        self.nbytes = nbytes
        self.ptr = lib.b200bls_malloc(nbytes)
        if not self.ptr:
            raise _lib.B200BlsError(lib.b200bls_last_error().decode())

    def upload(self, host):
        host = as_u8(host)
        assert host.size <= self.nbytes
        check(lib.b200bls_h2d(self.ptr, ptr(host), host.size))
        check(lib.b200bls_sync())
        return self

    def download(self, nbytes=None):
        out = np.empty(nbytes or self.nbytes, dtype=np.uint8)
        check(lib.b200bls_d2h(ptr(out), self.ptr, out.size))
        check(lib.b200bls_sync())
        return out

    def free(self):
        if self.ptr:
            lib.b200bls_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def run_program_dev(name, n_items, bufs, strides):
    arr = (ctypes.c_void_p * len(bufs))(*[b.ptr if isinstance(b, DeviceBuffer) else b for b in bufs])
    st = (ctypes.c_int64 * len(bufs))(*strides)
    check(lib.b200bls_run_program_dev(name.encode(), n_items, arr, st, len(bufs)))


def timer_start():
    check(lib.b200bls_timer_start())


def timer_stop():
    ms = ctypes.c_float()
    check(lib.b200bls_timer_stop(ctypes.byref(ms)))
    return ms.value


def microbench_imad(variant, blocks_per_sm=8, threads=256, iters=200):
    _lib.init()
    ops = ctypes.c_double()
    ms = ctypes.c_float()
    check(lib.b200bls_microbench_imad(variant, blocks_per_sm, threads, iters, ctypes.byref(ops), ctypes.byref(ms)))
    return ops.value, ms.value
