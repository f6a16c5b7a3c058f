"""Batched signing and public-key derivation without a GPU: the g2_sign and g1_pubkey programs on the host simulation of
the VM (both executors) against the oracle's sign_prehashed / pk_of, the endomorphism signs and the G1 table constants
they rest on against the oracle, and their cost against the generic ladders they replace."""
import ctypes
import os

import numpy as np
import pytest

import bls_oracle as O
import hostsim
import sign_corpus as SC
from conftest import load_golden

from bls_b200.programs import curve, hashg2, registry


def _conj(a):
    return (a[0], -a[1] % O.Q)


def test_psi_signs_against_oracle():
    """(P, -psi P, psi^2 P, -psi^3 P) = ([1] P, [a] P, [a^2] P, [a^3] P) on G2, and the program's constants for them"""
    for msg in (b"psi signs", b"another"):
        h = O.hash_to_g2(msg)
        p1 = O.psi(h)
        p2 = O.psi(p1)
        p3 = O.psi(p2)
        assert O.aff_neg(p1) == O.aff_mul(SC.A, h)
        assert p2 == O.aff_mul(SC.A ** 2, h)
        assert O.aff_neg(p3) == O.aff_mul(SC.A ** 3, h)
        x, y = h[0], h[1]
        assert (O.f2_mul(_conj(x), hashg2.PSI3_CX), O.f2_mul(_conj(y), hashg2.PSI_CY), False) == O.aff_neg(p3)
        assert ((x[0] * hashg2.PSI2_CX % O.Q, x[1] * hashg2.PSI2_CX % O.Q), O.f2_neg(y), False) == p2


def test_pubkey_table_against_oracle():
    assert curve.G1_PUBKEY_TABLE[0] == O.G1[:2]
    for m in range(1, 16):
        k = sum(SC.A ** i for i in range(4) if m >> i & 1)
        assert curve.G1_PUBKEY_TABLE[m] == O.aff_mul(k, O.G1)[:2], m


def _sha(hashes):
    sha = np.zeros(256 * len(hashes), dtype=np.uint8)
    hostsim.lib().hs_sha_stage(b"".join(hashes), sha.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(len(hashes)))
    return sha


def _digits(keys):
    return np.frombuffer(b"".join(SC.digit_record(k) for k in keys), dtype=np.uint8).copy()


def _kat():
    g = load_golden("sig_kat.json")
    sks = [int(k["sk"], 16) for k in g["keys"]]
    signs = [(sks[s["key"]], O.hash256(bytes.fromhex(s["msg"])), bytes.fromhex(s["sig"])) for s in g["sign"]]
    return g, sks, signs


@pytest.mark.parametrize("ctas", [1, 4])
def test_sign_program_on_host_simulation(ctas):
    """edge keys, the reference's signatures, random keys, and an all-zero SHA record (both field elements 0: the
    hashed point is infinity, and so is the signature)"""
    _, _, signs = _kat()
    rnd = SC.random_keys(4, 7)
    items = [(sk, O.hash256(b"edge %d" % i)) for i, sk in enumerate(SC.edge_keys())]
    items += [(sk, h) for sk, h, _ in signs[:6]] + [(sk, O.hash256(b"rnd %d" % sk)) for sk in rnd]
    sha = _sha([h for _, h in items])
    sha = np.concatenate([sha, np.zeros(256 * 2, dtype=np.uint8)])
    keys = [sk for sk, _ in items] + [5, O.N - 1]
    out = np.full(192 * len(keys), 0x5a, dtype=np.uint8)
    flag = np.full(len(keys), 9, dtype=np.uint8)
    n_slots, n_tmem = registry.SHAPES[ctas]
    asm = hashg2.build_sign().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    hostsim.run(asm, {0: sha, 1: _digits(keys), 2: out, 3: flag}, {0: 256, 1: 32, 2: 192, 3: 1}, len(keys),
                n_blocks=3, nt=8)
    raw = out.tobytes()
    for i, (sk, h) in enumerate(items):
        want = O.sign_prehashed(sk, h)
        assert raw[192 * i:192 * (i + 1)] == SC.g2_bytes(want), (ctas, i, hex(sk))
        assert flag[i] == (0 if want[2] else int(want[1][1] > O.Q // 2)), (ctas, i)
        comp = bytes([raw[192 * i] | (flag[i] << 7)]) + raw[192 * i + 1:192 * i + 96]
        assert comp == O.g2_serialize(want)
    for i, (sk, h, sig) in enumerate(signs[:6]):
        j = len(SC.edge_keys()) + i
        assert bytes([raw[192 * j] | (flag[j] << 7)]) + raw[192 * j + 1:192 * j + 96] == sig
    assert raw[192 * len(items):] == bytes(384) and list(flag[len(items):]) == [0, 0]


@pytest.mark.parametrize("ctas", [1, 4])
def test_pubkey_program_on_host_simulation(ctas):
    g, sks, _ = _kat()
    keys = SC.edge_keys() + sks + SC.random_keys(6, 11)
    out = np.full(96 * len(keys), 0x5a, dtype=np.uint8)
    flag = np.full(len(keys), 9, dtype=np.uint8)
    n_slots, n_tmem = registry.SHAPES[ctas]
    asm = curve.build_pubkey().assemble(n_slots, n_cold=4096, n_tmem=n_tmem)
    hostsim.run(asm, {0: _digits(keys), 1: out, 2: flag}, {0: 32, 1: 96, 2: 1}, len(keys), n_blocks=3, nt=8)
    raw = out.tobytes()
    for i, sk in enumerate(keys):
        want = O.pk_of(sk)
        assert raw[96 * i:96 * (i + 1)] == SC.g1_bytes(want), (ctas, i, hex(sk))
        comp = bytes([raw[96 * i] | (flag[i] << 7)]) + raw[96 * i + 1:96 * i + 48]
        assert comp == O.g1_serialize(want), (ctas, i)
    for k, key in enumerate(g["keys"]):
        j = len(SC.edge_keys()) + k
        assert (bytes([raw[96 * j] | (flag[j] << 7)]) + raw[96 * j + 1:96 * j + 48]).hex() == key["pk"]


def test_sign_and_pubkey_cost():
    """the joint ladders against the generic ones they replace: 0.63x of hash_to_g2 + g2_mul, 0.38x of g1_mul"""
    sign = registry.executed_mults("g2_sign")
    assert sign <= 0.70 * (registry.executed_mults("hash_to_g2") + registry.executed_mults("g2_mul"))
    assert registry.executed_mults("g1_pubkey") <= 0.45 * registry.executed_mults("g1_mul")


def test_argument_checks_need_no_device():
    """bad wire forms and null buffers are refused before the library looks for a GPU; n = 0 does nothing"""
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "python-bls_b200", "bls_b200",
                      "libb200bls.so")
    if not os.path.exists(so):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(so)
    buf = (ctypes.c_uint8 * 192)()
    one, zero = ctypes.c_size_t(1), ctypes.c_size_t(0)
    for wire in (-1, 2):
        assert lib.b200bls_sign_batch(wire, buf, buf, buf, one) == -3             # B200BLS_E_ARG
        assert lib.b200bls_sign_batch_dev(wire, buf, buf, buf, one) == -3
        assert lib.b200bls_public_key_batch(wire, buf, buf, one) == -3
        assert lib.b200bls_public_key_batch_dev(wire, buf, buf, one) == -3
    assert lib.b200bls_sign_batch(1, None, buf, buf, one) == -3
    assert lib.b200bls_public_key_batch(0, buf, None, one) == -3
    assert lib.b200bls_sign_batch(0, None, None, None, zero) == 0
    assert lib.b200bls_public_key_batch(1, None, None, zero) == 0
