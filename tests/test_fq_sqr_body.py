"""The dedicated F_q squaring (fq.cuh fq_sqr_inl) against fq_mul(a, a) and against a^2 R^-1 mod q, on inputs chosen to
drive its carries to their limits: limb patterns from {0, 1, 2^31, 2^32 - 1, q_i, q_i +- 1}, the ends of the field, operands
whose rows of the square and Montgomery rows carry into the top of the window (all-ones prefixes, q minus small values), and
10^5 seeded random values.  The host build runs the emulated carry chains; the GPU test runs the same inputs through the
device's asm blocks."""
import itertools
import random

import numpy as np
import pytest

import hostlib as H
import vectors as V

Q = H.Q
RADIX = 1 << 256
RINV = pow(RADIX, -1, Q)
QL = [(Q >> (32 * i)) & 0xFFFFFFFF for i in range(8)]
M32 = (1 << 32) - 1


def from_limbs(ls):
    return sum(v << (32 * i) for i, v in enumerate(ls))


def inputs():
    """canonical inputs (< q: the squaring's contract, as for every F_q routine)"""
    base = {0, 1, 1 << 31, M32}
    for v in QL:
        base |= {v, (v + 1) & M32, (v - 1) & M32}
    base = sorted(base)
    xs = set()
    for v in base:  # every limb the same value, and one limb set in an otherwise zero / all-ones / q-shaped operand
        xs.add(from_limbs([v] * 8))
        for i, fill in itertools.product(range(8), ([0] * 8, [M32] * 8, QL)):
            ls = list(fill)
            ls[i] = v
            xs.add(from_limbs(ls))
    rnd = random.Random(20)
    for _ in range(20000):  # random limb patterns from the set
        xs.add(from_limbs([rnd.choice(base) for _ in range(8)]))
    xs |= {Q - 1, Q - 2, RADIX - 2 * Q, 1, RADIX % Q, (RADIX - Q) % Q, Q >> 1, (Q >> 1) + 1}
    for k in range(1, 256):  # all-ones low limbs: every product and reduction chain carries to its top
        xs |= {(1 << k) - 1, Q - (1 << k) + 1 if (1 << k) < Q else 0, (1 << k) % Q}
    for d in range(0, 64):  # all-ones below the top bits, and values just below q
        xs |= {(1 << 254) + d, (1 << 254) - 1 - d, (1 << 254) - (1 << (4 * d)) if 4 * d < 254 else 0, Q - 1 - (d << 200)}
    xs |= {(1 << 254) | ((1 << 224) - 1), ((1 << 254) - 1) ^ (1 << 223)}
    for _ in range(100000):
        xs.add(rnd.randrange(Q))
    return sorted(x % Q for x in xs)


@pytest.fixture(scope="module")
def lib():
    return H.build()


def test_inputs_cover_the_field_ends():
    xs = set(inputs())
    assert len(xs) > 100000 and max(xs) == Q - 1 and min(xs) == 0
    assert {1, Q - 2, RADIX % Q, (1 << 255) % Q} <= xs


def test_sqr_equals_mul_and_big_int(lib):
    out, ref = np.zeros(8, np.uint32), np.zeros(8, np.uint32)
    bad = []
    for a in inputs():
        al = H.limbs(a)
        lib.h_fq_sqr(H.ptr(al), H.ptr(out))
        lib.h_fq_mul(H.ptr(al), H.ptr(al), H.ptr(ref))
        got = H.to_int(out)
        if got != a * a * RINV % Q or got != H.to_int(ref):
            bad.append(hex(a))
    assert not bad, bad[:8]


def test_sqr_counts_84_limb_products(lib):
    """the square stays at 36 product + 48 reduction limb products (profiles/op_counts.json prices it so)"""
    cnt = np.zeros(10, np.uint64)
    out = np.zeros(8, np.uint32)
    lib.h_counts_reset()
    lib.h_fq_sqr(H.ptr(H.limbs(Q - 2)), H.ptr(out))
    lib.h_counts_get(H.ptr(cnt))
    assert int(cnt[0]) == 84 and int(cnt[2]) == 1


@pytest.mark.gpu
def test_device_sqr_equals_mul_and_big_int(engine):
    xs = inputs()
    A = V.scalars(xs)
    sq = V.ints_out(engine.dbg_fq(4, A))
    mul = V.ints_out(engine.dbg_fq(0, A, A))
    bad = [hex(a) for a, s, m in zip(xs, sq, mul) if s != a * a * RINV % Q or s != m]
    assert not bad, bad[:8]
