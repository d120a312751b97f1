"""The small-integer form of the Hades permutation (csrc/hades.cuh hades_perm_int, csrc/params_host.cuh derive_int_tables).

When every MDS entry is 1/d for a small integer d, C = L * MDS (L = lcm of the d) is a matrix of small integers and each
round runs s <- C s on the FP64 pipe, the factor L tracked in a per-round scale.  CPU part: the C++ derivation equals
its Python twin (tools/gen_constants.py) under both round-constant rules; the host build of the permutation equals the
dense one and the oracle on random and extreme states; detection accepts the default Cauchy matrix and rejects others;
the layer's exactness bounds hold.  GPU part: dbg_hades of a default context equals the oracle above one wave."""
import ctypes
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import hostlib as H
import schnorr_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_constants as G  # noqa: E402

Q = o.Q


@pytest.fixture(scope="module")
def lib():
    so = os.path.join(ROOT, "build", "host_int_layer.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-include", os.path.join(ROOT, "tests", "host_shim.h"),
                           "-o", so, os.path.join(ROOT, "tests", "host_int_layer.cpp")])
    return ctypes.CDLL(so)


def _setup(lib, rc, mds):
    """derive the host build's tables from plain-integer round constants / MDS, as sb200_init_ex does"""
    rca = np.stack([H.mont(c) for c in rc[:335]])
    mda = np.stack([H.mont(mds[i][j]) for i in range(5) for j in range(5)])
    return lib.h_setup_hades(H.ptr(rca), H.ptr(mda))


def _int_tables(lib):
    cmat, src, fix, uns, flag = np.zeros(25), np.zeros((335, 8), np.uint32), np.zeros((59, 8), np.uint32), np.zeros(8, np.uint32), np.zeros(1, np.uint32)
    lib.h_int_tables(H.ptr(cmat), H.ptr(src), H.ptr(fix), H.ptr(uns), H.ptr(flag))
    ints = lambda a: [H.to_int(r) for r in a.reshape(-1, 8)]
    return int(flag[0]), {"cmat": [int(x) for x in cmat], "src": ints(src), "fix": ints(fix), "unscale": ints(uns)}


def _perm(lib, state, dense):
    st = np.concatenate([H.mont(x) for x in state])
    lib.h_hades(H.ptr(st), int(dense))
    return [H.unmont(st[8 * k:8 * k + 8]) for k in range(5)]


def _counts(lib, state):
    cnt = np.zeros(10, np.uint64)
    lib.h_counts_reset()
    _perm(lib, state, False)
    lib.h_counts_get(H.ptr(cnt))
    return {"wide": int(cnt[0]), "fq_mul": int(cnt[1]), "fq_dot5": int(cnt[5]), "dfma": int(cnt[6])}


def _cauchy(xs, ys):
    return [[pow(x + y, -1, Q) for y in ys] for x in xs]


def _edge_states():
    top = Q - 1
    return [[0] * 5, [top] * 5, [top, 0, top, 0, top], [0, top, 0, top, 0], [1, top, 2, top, 3], [top, top, top, top, 0]]


@pytest.mark.parametrize("rule", ["cumsum", "plain"])
def test_tables_equal_python_twin(lib, rule):
    rc = o._round_constants(rule)
    assert _setup(lib, rc, o.MDS) == 0
    flag, got = _int_tables(lib)
    want = G.int_layer_tables(rc, o.MDS)
    assert flag == 1 and want is not None
    for k in ("cmat", "src", "fix", "unscale"):
        assert got[k] == want[k], k
    assert G.int_layer_matrix(o.MDS)[0] == 360360 and max(want["cmat"]) == 72072


@pytest.mark.parametrize("rule", ["cumsum", "plain"])
def test_permutation_equals_dense_and_oracle(lib, rule):
    prev = o.set_ark_rule(rule)
    try:
        assert _setup(lib, o.ROUND_CONSTANTS, o.MDS) == 0
        rnd = random.Random(5 if rule == "cumsum" else 6)
        states = _edge_states() + [[rnd.randrange(Q) for _ in range(5)] for _ in range(24)]
        for s in states:
            want = o.hades_perm(s)
            assert _perm(lib, s, False) == want, s
            assert _perm(lib, s, True) == want, s
        assert G.hades_int(states[1], G.int_layer_tables(o.ROUND_CONSTANTS, o.MDS)) == o.hades_perm(states[1])
        # the small-integer path ran: no Montgomery dot product, the layers on DFMA, one product per partial round
        # plus the S-boxes and the final unscale
        c = _counts(lib, states[0])
        assert c["fq_dot5"] == 0 and c["dfma"] > 67 * 200 and c["fq_mul"] == 8 * 5 + 59 + 59 + 5
    finally:
        o.set_ark_rule(prev)


def test_detection(lib):
    """the default Cauchy matrix qualifies; a random Cauchy matrix (entries not inverses of small integers) and one whose
    lcm makes C too large do not, and keep running the sparse rounds exactly"""
    rc = o._round_constants("plain")
    assert _setup(lib, rc, o.MDS) == 0 and _int_tables(lib)[0] == 1
    rnd = random.Random(11)  # the random Cauchy matrix of test_params.test_arbitrary_tables_are_accepted_and_bad_ones_rejected
    rc_rand = [rnd.randrange(Q) for _ in range(335)]
    xs, ys = [rnd.randrange(Q) for _ in range(5)], [rnd.randrange(Q) for _ in range(5)]
    others = [(rc_rand, _cauchy(xs, ys)), (rc, _cauchy(range(5), range(9, 14)))]   # denominators 9..17: max C = 1361360
    for rcx, mds in others:
        assert G.int_layer_matrix(mds) is None
        assert _setup(lib, rcx, mds) == 0
        flag, _ = _int_tables(lib)
        assert flag == 0
        s = [rnd.randrange(Q) for _ in range(5)]
        assert _perm(lib, s, False) == _perm(lib, s, True)
        assert _counts(lib, s)["dfma"] == 0
    # denominators 8..16: L = 720720, max C = 90090 -- qualifies, and stays exact on the extreme states
    mds = _cauchy(range(5), range(8, 13))
    L, C = G.int_layer_matrix(mds)
    assert (L, max(max(r) for r in C)) == (720720, 90090)
    assert _setup(lib, rc, mds) == 0 and _int_tables(lib)[0] == 1
    for s in _edge_states():
        assert _perm(lib, s, False) == _perm(lib, s, True), s


def test_layer_bounds(lib):
    """a column of the layer (five products of a 32-bit limb with an entry of C, plus the previous column's carry) must
    stay below 2^52 for the DFMA chain to hold it exactly; the reduction's quotient estimate must stay within one"""
    bound = lib.h_int_bound()
    assert bound == G.INT_LAYER_CMAX_BOUND and 5 * bound * (1 << 32) <= 1 << 52
    _, C = G.int_layer_matrix(o.MDS)
    lim = (1 << 32) - 1
    carry = 0
    for _ in range(8):  # worst case: every limb 2^32 - 1 (a bound on every canonical state)
        col = max(sum(r) for r in C) * lim + carry
        assert col < 1 << 52
        carry = col >> 32
    assert carry < 1 << 20
    assert _setup(lib, o.ROUND_CONSTANTS, o.MDS) == 0
    rnd = random.Random(9)
    for s in _edge_states() + [[rnd.randrange(Q) for _ in range(5)] for _ in range(16)]:
        st = np.concatenate([H.limbs(x) for x in s])
        lib.h_int_layer(H.ptr(st))
        assert [H.to_int(st[8 * k:8 * k + 8]) for k in range(5)] == [sum(C[k][j] * s[j] for j in range(5)) % Q for k in range(5)]
    # the reduction alone over its whole input range, values below 2^20 q (also those next to a multiple of q)
    vmax = (1 << 20) * Q
    tops = [0, 1, 5 * 72072 // 2, (vmax >> 256) - 1, vmax >> 256] + [rnd.randrange(vmax >> 256) for _ in range(8)]
    for top in tops:
        for low in [0, (1 << 256) - 1, Q - 1, Q, 2 * Q - 1] + [((top << 256) // Q + e) * Q - (top << 256) + d for e in (0, 1) for d in (-1, 0, 1)]:
            low %= 1 << 256
            if (top << 256) + low >= vmax:
                continue
            r = H.limbs(low)
            lib.h_int_reduce(H.ptr(r), top)
            assert H.to_int(r) == ((top << 256) + low) % Q, (top, low)


# ----------------------------------------------------------------------------------------------------- GPU
def _oracle_chunk(states):
    return [o.hades_perm(s) for s in states]


@pytest.mark.gpu
def test_dbg_hades_default_context_above_one_wave(engine):
    """dbg_hades of a default context (small-integer layers) equals the oracle over more than one wave of CTAs"""
    import multiprocessing as mp
    import torch
    import vectors as V
    n = 4 * torch.cuda.get_device_properties(0).multi_processor_count * 128 + 333
    rnd = random.Random(41)
    states = _edge_states() + [[rnd.randrange(Q) for _ in range(5)] for _ in range(n - len(_edge_states()))]
    arr = np.stack([np.concatenate([V.mont(x) for x in s]) for s in states])
    out = engine.dbg_hades(arr)
    got = [[V.unmont(r[8 * k:8 * k + 8]) for k in range(5)] for r in out]
    step = 2048
    with mp.get_context("fork").Pool(min(32, os.cpu_count() or 1)) as pool:
        want = sum(pool.map(_oracle_chunk, [states[i:i + step] for i in range(0, n, step)]), [])
    assert got == want
