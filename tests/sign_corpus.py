"""Secret keys that reach the edges of the signing ladders (csrc/scalar_split.h, Curve.digit_ladder), shared by the CPU
and GPU tests of batched signing and public-key derivation."""
import random

import bls_oracle as O

A = O.X_ABS


def digits(sk):
    """the four base-a digits of sk mod n, least significant first"""
    k = sk % O.N
    return [k // A ** i % A for i in range(4)]


def digit_record(sk):
    """the 32-byte record the split kernel writes: digit i in bits [64 i, 64 i + 64) of a big-endian integer"""
    return sum(d << (64 * i) for i, d in enumerate(digits(sk))).to_bytes(32, "big")


def edge_keys():
    """sk in {0, 1, a - 1, a, a + 1, a^2, a^3, n - 1, n, n + 1, 2n, 2n + 5, 2^256 - 1}, every k with a single
    non-zero digit (1, 2 or a - 1 at each position), and every non-zero k below n whose digits are each 0 or a - 1
    (no key is listed twice)"""
    n = O.N
    ks = [0, 1, A - 1, A, A + 1, A ** 2, A ** 3, n - 1, n, n + 1, 2 * n, 2 * n + 5, 2 ** 256 - 1]
    for i in range(4):
        ks += [d * A ** i for d in (1, 2, A - 1)]
    for mask in range(1, 16):
        k = sum((A - 1) * A ** i for i in range(4) if mask >> i & 1)
        if k < n:
            ks.append(k)
    return list(dict.fromkeys(ks))


def random_keys(count, seed):
    """seeded keys over the whole 32-byte range, so that the reduction mod n is exercised too"""
    rng = random.Random(seed)
    return [rng.getrandbits(256) for _ in range(count)]


def g1_bytes(p):
    """affine G1 point -> 96 bytes (infinity: zero bytes)"""
    if p[2]:
        return bytes(96)
    return p[0].to_bytes(48, "big") + p[1].to_bytes(48, "big")


def g2_bytes(p):
    """affine G2 point -> 192 bytes (infinity: zero bytes)"""
    if p[2]:
        return bytes(192)
    return b"".join(c.to_bytes(48, "big") for c in (p[0][0], p[0][1], p[1][0], p[1][1]))
