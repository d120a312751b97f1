"""Nonces drawn on the device from a caller-owned StdRng position (csrc/rng.cuh, sb200_stdrng_random, sb200_sign_stdrng).

CPU part: the host build of rng.cuh equals the oracle's ChaCha12 and api.StdRng at block-aligned positions, at every
offset inside a block, across the carry from counter word 12 into word 13 and near 2^63 words; both fields; a mixed
sequence of next_u64 and draws is reproduced from its word positions; the argument checks that fail before any device
is touched.  GPU part: the device draws against the numpy stream over ragged multi-chunk batches, host and device
pointers, multi-device contexts; the seeded signers against the host-drawn-nonce calls, byte for byte; the typed
mirrors (api.py, include/schnorr_b200.hpp) against their host-draw path."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import schnorr_oracle as o
import vectors as V
from schnorr_b200 import api
from schnorr_b200._lib import DEVICE_PTRS, ERR_ARG, POINTS_AFFINE, SIGN_OBLIVIOUS, StdRngPos, aligned_empty, load_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R
STRADDLE = 16 * (2**32 - 1) + 5           # its two blocks are 2^32 - 1 and 2^32: the carry from counter word 12 into 13
NEAR_2_63 = 2**63 + 9
POSITIONS = [0, 16, 32, 16 * 777] + list(range(1, 16)) + [16 * 777 + 11, STRADDLE, 16 * (2**32 - 1), 16 * 2**32,
                                                           NEAR_2_63, 2**63 - 16, 2**64 - 16 - 7]
N_RAGGED = 3 * 2**16 + 77                # > 3 pipeline chunks of CHUNK_MIN = 2^14 ... and not a multiple of 32


def _key(seed=2321):
    return np.frombuffer(o.seed_from_u64(seed), "<u4").astype(np.uint32)


def _words_oracle(key, word_pos, nwords=16):
    b0, off = divmod(word_pos, 16)
    raw = b"".join(o.chacha_block([int(k) for k in key], b0 + j) for j in range((off + nwords + 15) // 16))
    return np.frombuffer(raw, "<u4")[off:off + nwords]


def _draws_numpy(key, word_pos, n):
    """[n, 16] keystream words of draws 0..n-1 at word_pos (api.StdRng's vectorised ChaCha12)"""
    b0, off = divmod(word_pos, 16)
    w = api.StdRng(key.tobytes()).blocks(b0, n + (1 if off else 0)).reshape(-1)
    return np.ascontiguousarray(w[off:off + 16 * n].reshape(n, 16))


def _reduce(words, field):
    out = np.empty((len(words), 8), np.uint32)
    for i, row in enumerate(words):
        x = int.from_bytes(row.tobytes(), "little")
        out[i] = V.limbs(x % R) if field == 0 else V.mont(x % Q)
    return out


@pytest.fixture(scope="module")
def hlib():
    so = os.path.join(ROOT, "build", "host_rng.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-include", os.path.join(ROOT, "tests", "host_shim.h"),
                           "-o", so, os.path.join(ROOT, "tests", "host_rng.cpp")])
    lib = ctypes.CDLL(so)
    for f in (lib.h_chacha12_block, lib.h_stdrng_draw):
        f.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]
    lib.h_stdrng_random.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p]
    lib.h_from_wide.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    lib.h_stdrng_random_args.argtypes = [ctypes.c_int64, ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.h_sign_stdrng_args.argtypes = [ctypes.c_int64, ctypes.c_uint32, ctypes.c_int] + [ctypes.c_void_p] * 7
    return lib


def _h(fn, key, pos, *extra, words=16):
    out = np.zeros(words, np.uint32)
    fn(key.ctypes.data, pos, *extra, out.ctypes.data)
    return out


# ----------------------------------------------------------------------------------------------------- CPU
def test_chacha12_block_matches_oracle_and_api(hlib):
    key = _key()
    for ctr in (0, 1, 777, 2**32 - 1, 2**32, 2**59 + 3, 2**64 - 1):
        got = _h(hlib.h_chacha12_block, key, ctr)
        assert got.tobytes() == o.chacha_block([int(k) for k in key], ctr), ctr
        assert (got == api.StdRng(key.tobytes()).blocks(ctr, 1)[0]).all(), ctr


@pytest.mark.parametrize("seed", [2321, 0xC3])
def test_draw_at_every_position_kind(hlib, seed):
    """aligned words, every offset 1..15, the 2^32-block straddle, near 2^63 words; against the oracle's blocks, the
    seeked api.StdRng and (aligned) the oracle's nonce_from_block"""
    key = _key(seed)
    for wp in POSITIONS:
        want = _words_oracle(key, wp)
        assert (_h(hlib.h_stdrng_draw, key, wp) == want).all(), wp
        rng = api.StdRng(key.tobytes())
        rng.seek(wp)
        assert rng.word_pos == wp
        assert np.frombuffer(rng.fill_bytes(64), "<u4").tolist() == want.tolist(), wp
        assert rng.word_pos == wp + 16
        x = int.from_bytes(want.tobytes(), "little")
        assert V.to_int(_h(hlib.h_stdrng_random, key, wp, 0, words=8)) == x % R, wp
        assert V.unmont(_h(hlib.h_stdrng_random, key, wp, 1, words=8)) == x % Q, wp
        if wp % 16 == 0:
            assert V.to_int(_h(hlib.h_stdrng_random, key, wp, 0, words=8)) == o.nonce_from_block([int(k) for k in key], wp // 16)


def test_reduction_extremes(hlib):
    """the from_bytes_wide the device draws go through (wire.cuh fr_from_wide / fq_from_wide), on the all-ones draw, halves
    at 2^256 - 1 and draws next to multiples of r and q in either half: both fields exact"""
    top = 2**256
    xs = [0, 1, 2**512 - 1, top - 1, top, (top - 1) * top, R - 1, R, 2 * R, Q - 1, Q, 2 * Q, 3 * Q - 1, Q * top, (Q - 1) * top + Q,
          R * top + R - 1, (2**512 // R) * R - 1, (2**512 // R) * R, (2**512 // Q) * Q - 1, (2**512 // Q) * Q]
    for x in xs:
        w = np.frombuffer(x.to_bytes(64, "little"), "<u4").copy()
        out = np.zeros(8, np.uint32)
        hlib.h_from_wide(w.ctypes.data, 0, out.ctypes.data)
        assert V.to_int(out) == x % R, hex(x)
        hlib.h_from_wide(w.ctypes.data, 1, out.ctypes.data)
        assert out.tolist() == V.mont(x % Q).tolist(), hex(x)


def test_word_position_reproduces_mixed_sequence(hlib):
    """next_u64 (2 words) and Field::random draws (16 words) interleaved: each draw equals the device function at the
    stream's word position, and a generator seeked there continues identically"""
    key = _key()
    orng, arng = o.StdRng.seed_from_u64(2321), api.StdRng.seed_from_u64(2321)
    ops = ["u64", "fr", "u64", "u64", "fq", "fr", "u64"] + ["fr"] * 9 + ["u64", "fq", "u64", "u64", "u64", "fr"]
    wp = 0
    for op in ops:
        assert arng.word_pos == wp
        if op == "u64":
            v = orng.next_u64()
            assert arng.next_u64() == v
            assert _words_oracle(key, wp, 2).tobytes() == v.to_bytes(8, "little")
            wp += 2
            continue
        field = 0 if op == "fr" else 1
        want = orng.random_fr() if field == 0 else orng.random_fq()
        dev = _h(hlib.h_stdrng_random, key, wp, field, words=8)
        assert (V.to_int(dev) if field == 0 else V.unmont(dev)) == want, (op, wp)
        assert (arng.random_scalar() if field == 0 else arng.random_bls()) == want
        twin = api.StdRng(key.tobytes())
        twin.seek(wp)
        assert (twin.random_scalar() if field == 0 else twin.random_bls()) == want
        wp += 16
    arng.fill_bytes(3)  # an odd byte draw leaves the stream inside a word: no word position
    assert arng.word_pos is None


def _arg_cases(ctx, n, bufs):
    """(name, call(pos)) pairs that must return SB200_ERR_ARG without touching anything; bufs: pointers of n-tuple arrays"""
    lib = load_library()
    sk, msg, gen, u, R_, Rp, c, out = (bufs[k] for k in ("sk", "msg", "gen", "u", "R", "Rp", "c", "out"))
    rnd = lambda n_=n, fl=0, field=0, o_=out: (lambda pos: lib.sb200_stdrng_random(ctx, n_, fl, field, pos, o_))
    sgn = lambda n_=n, fl=0, scheme=0, g=gen, rp=Rp, u_=u, s=sk: (
        lambda pos: lib.sb200_sign_stdrng(ctx, n_, fl, scheme, s, msg, g, pos, u_, R_, rp, c))
    return [
        ("random: n < 0", rnd(n_=-1)), ("random: field 2", rnd(field=2)), ("random: field -1", rnd(field=-1)),
        ("random: SIGN_OBLIVIOUS", rnd(fl=SIGN_OBLIVIOUS)), ("random: POINTS_AFFINE", rnd(fl=POINTS_AFFINE)),
        ("random: out NULL", rnd(o_=None)),
        ("sign: n < 0", sgn(n_=-1)), ("sign: scheme 3", sgn(scheme=3)), ("sign: scheme -1", sgn(scheme=-1)),
        ("sign: scheme 2 without generator", sgn(scheme=2, g=None)), ("sign: scheme 1 without R'", sgn(scheme=1, rp=None)),
        ("sign: POINTS_AFFINE on scheme 0", sgn(fl=POINTS_AFFINE)), ("sign: POINTS_AFFINE on scheme 1", sgn(scheme=1, fl=POINTS_AFFINE)),
        ("sign: CHECK_POINTS", sgn(fl=8)), ("sign: VERIFY_DUAL_PIPE", sgn(fl=4)), ("sign: unknown flag", sgn(scheme=2, fl=64)),
        ("sign: u_out NULL", sgn(u_=None)), ("sign: sk NULL", sgn(s=None)),
    ]


def _overflow_cases(ctx, bufs):
    """word_pos + 16 n must fit in 64 bits: (word_pos, n) pairs just over the limit"""
    lib = load_library()
    return [(2**64 - 64, 4, lambda pos: lib.sb200_stdrng_random(ctx, 4, 0, 0, pos, bufs["out"])),
            (2**64 - 1, 1, lambda pos: lib.sb200_sign_stdrng(ctx, 1, 0, 0, bufs["sk"], bufs["msg"], None, pos, bufs["u"],
                                                             bufs["R"], None, bufs["c"])),
            (0, 2**60, lambda pos: lib.sb200_stdrng_random(ctx, 2**60, 0, 0, pos, bufs["out"]))]


def _host_bufs(n):
    arrs = {k: aligned_empty((n, w)) for k, w in (("sk", 8), ("msg", 8), ("gen", 16), ("u", 8), ("R", 16), ("Rp", 16),
                                                  ("c", 8), ("out", 8))}
    for a in arrs.values():
        a[...] = 0
    return arrs, {k: a.ctypes.data for k, a in arrs.items()}


def _check_rejections(ctx, n):
    _, bufs = _host_bufs(max(n, 1))
    key = _key()
    lib = load_library()
    for name, call in _arg_cases(ctx, n, bufs):
        pos = StdRngPos.of(key, 12345)
        assert call(ctypes.byref(pos)) == ERR_ARG, name
        assert pos.word_pos == 12345, name
    for wp, nn, call in _overflow_cases(ctx, bufs):
        pos = StdRngPos.of(key, wp)
        assert call(ctypes.byref(pos)) == ERR_ARG, (wp, nn)
        assert pos.word_pos == wp
    assert lib.sb200_stdrng_random(ctx, n, 0, 0, None, bufs["out"]) == ERR_ARG
    assert lib.sb200_sign_stdrng(ctx, n, 0, 0, bufs["sk"], bufs["msg"], None, None, bufs["u"], bufs["R"], None, bufs["c"]) == ERR_ARG


def test_argument_checks_host_build(hlib):
    """the entry points' own argument checks (csrc/rng.cuh, run before any context is looked at), in the host build: each
    rejected case is rejected for its own reason -- the same call with that one argument corrected passes"""
    key = _key()
    P = ctypes.c_void_p(64)  # any non-null buffer: the checks never dereference it
    pos = lambda wp=12345: ctypes.byref(StdRngPos.of(key, wp))

    def rnd(n=4, fl=0, field=0, rng=True, out=P, wp=12345):
        return hlib.h_stdrng_random_args(n, fl, field, pos(wp) if rng else None, out)

    def sgn(n=4, fl=0, scheme=0, sk=P, msg=P, gen=P, rng=True, u=P, R_=P, Rp=P, wp=12345):
        return hlib.h_sign_stdrng_args(n, fl, scheme, sk, msg, gen, pos(wp) if rng else None, u, R_, Rp)

    ok = [rnd(), rnd(field=1), rnd(fl=DEVICE_PTRS), rnd(n=0), rnd(n=4, wp=2**64 - 65), rnd(n=2**60 - 1, wp=15)]
    ok += [sgn(scheme=s) for s in (0, 1, 2)] + [sgn(fl=SIGN_OBLIVIOUS | DEVICE_PTRS), sgn(scheme=2, fl=POINTS_AFFINE | SIGN_OBLIVIOUS),
                                                sgn(scheme=0, gen=None, Rp=None), sgn(scheme=2, Rp=None), sgn(n=1, wp=2**64 - 17)]
    assert ok == [0] * len(ok)
    bad = {"random: n < 0": rnd(n=-1), "random: field 2": rnd(field=2), "random: field -1": rnd(field=-1),
           "random: SIGN_OBLIVIOUS": rnd(fl=SIGN_OBLIVIOUS), "random: POINTS_AFFINE": rnd(fl=POINTS_AFFINE),
           "random: out NULL": rnd(out=None), "random: rng NULL": rnd(rng=False), "random: overflow": rnd(n=4, wp=2**64 - 64),
           "random: overflow of 16 n": rnd(n=2**60, wp=0),
           "sign: n < 0": sgn(n=-1), "sign: scheme 3": sgn(scheme=3), "sign: scheme -1": sgn(scheme=-1),
           "sign: scheme 2 without generator": sgn(scheme=2, gen=None), "sign: scheme 1 without R'": sgn(scheme=1, Rp=None),
           "sign: POINTS_AFFINE on scheme 0": sgn(fl=POINTS_AFFINE), "sign: POINTS_AFFINE on scheme 1": sgn(scheme=1, fl=POINTS_AFFINE),
           "sign: CHECK_POINTS": sgn(fl=8), "sign: VERIFY_DUAL_PIPE": sgn(fl=4), "sign: unknown flag": sgn(scheme=2, fl=64),
           "sign: u_out NULL": sgn(u=None), "sign: R_out NULL": sgn(R_=None), "sign: sk NULL": sgn(sk=None),
           "sign: msg NULL": sgn(msg=None), "sign: rng NULL": sgn(rng=False), "sign: overflow": sgn(n=1, wp=2**64 - 16)}
    assert {k: v for k, v in bad.items() if v != ERR_ARG} == {}


def test_rejected_calls_leave_the_position_alone():
    """through the library's ABI (no context: nothing to run), every rejected call returns SB200_ERR_ARG and leaves
    rng->word_pos unchanged; the GPU twin below repeats this with a live context, where valid calls succeed"""
    _check_rejections(None, 4)


# ----------------------------------------------------------------------------------------------------- GPU
def _synth(n, seed):
    rs = np.random.RandomState(seed)
    sk = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    sk[:, 7] &= 0x07FFFFFF                      # < 2^251 < r
    msg = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    msg[:, 7] &= 0x3FFFFFFF                     # Montgomery limbs of some field element (< 2^254 < q)
    return sk, msg


_NONCES = {}


def _nonces(key, wp, n):
    k = (key.tobytes(), wp, n)
    if k not in _NONCES:
        _NONCES[k] = _reduce(_draws_numpy(key, wp, n), 0)
    return _NONCES[k]


def _gens(engine, n, seed, affine):
    rs = np.random.RandomState(seed)
    s = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    s[:, 7] &= 0x07FFFFFF
    g = engine.keygen(s)                        # affine Montgomery (u, v) of s G
    if affine:
        return g
    z = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    z[:, 7] &= 0x3FFFFFFF
    z[:, 0] |= 1
    return np.ascontiguousarray(np.concatenate([engine.dbg_fq(0, g[:, :8], z), engine.dbg_fq(0, g[:, 8:], z), z], axis=1))


@pytest.mark.gpu
def test_device_argument_checks_and_position(engine):
    _check_rejections(engine._h, 4)
    key, n = _key(), 1000
    out, wp = engine.stdrng_random(key, 2**64 - 16 * n - 1, n, 0)   # the largest position with room for n draws
    assert wp == 2**64 - 1
    assert (out == _reduce(_draws_numpy(key, 2**64 - 16 * n - 1, n), 0)).all()
    _, wp = engine.stdrng_random(key, 77, 0, 1)
    assert wp == 77


@pytest.mark.gpu
@pytest.mark.parametrize("word_pos,n", [(0, 4096 + 3), (7, 4096 + 3), (STRADDLE, 4096 + 3), (NEAR_2_63, 1000),
                                        (16 * 5 + 9, N_RAGGED)])
@pytest.mark.parametrize("field", [0, 1])
def test_stdrng_random_matches_stream(engine, word_pos, n, field):
    key = _key(0xC3)
    got, wp = engine.stdrng_random(key, word_pos, n, field)
    assert wp == word_pos + 16 * n
    assert (got == _reduce(_draws_numpy(key, word_pos, n), field)).all()


@pytest.mark.gpu
def test_stdrng_random_device_pointers_and_launches(engine):
    import torch
    key, n, wp0 = _key(7), N_RAGGED, STRADDLE
    out = torch.zeros((n, 8), dtype=torch.int32, device="cuda:0")
    before = engine.launch_count
    wp = engine.stdrng_random(key, wp0, n, 1, flags=DEVICE_PTRS, out=out.data_ptr())
    torch.cuda.synchronize()
    assert engine.launch_count - before == 1 and wp == wp0 + 16 * n
    host, _ = engine.stdrng_random(key, wp0, n, 1)
    assert (out.cpu().numpy().view(np.uint32) == host).all()
    assert (host == _reduce(_draws_numpy(key, wp0, n), 1)).all()


@pytest.mark.gpu
def test_multi_device_context_gives_the_same_draws_and_signatures(engine):
    import torch
    from schnorr_b200 import Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    e = Engine(devs, ark=o.ARK_RULE)
    try:
        key, n, wp0 = _key(11), N_RAGGED, 16 * 3 + 13
        a, wa = e.stdrng_random(key, wp0, n, 0)
        b, wb = engine.stdrng_random(key, wp0, n, 0)
        assert wa == wb and (a == b).all()
        sk, msg = _synth(n, 21)
        ra, rb = e.sign_stdrng(0, sk, msg, key, wp0), engine.sign_stdrng(0, sk, msg, key, wp0)
        assert ra[-1] == rb[-1] == wp0 + 16 * n
        assert all((x == y).all() for x, y in zip(ra[:-1], rb[:-1]))
    finally:
        e.close()


def _host_sign(engine, scheme, sk, msg, nonce, gen, affine, oblivious):
    if scheme == 0:
        return engine.sign(sk, msg, nonce, oblivious=oblivious)
    if scheme == 1:
        return engine.sign_double(sk, msg, nonce, oblivious=oblivious)
    return engine.sign_vargen(sk, gen, msg, nonce, affine=affine, oblivious=oblivious)


SIGN_CASES = [(0, True, False), (0, True, True), (1, True, False), (1, True, True),
              (2, True, False), (2, False, False), (2, True, True), (2, False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("scheme,affine,oblivious", SIGN_CASES)
def test_sign_stdrng_equals_host_drawn_nonces(engine, scheme, affine, oblivious):
    """u, R, R', c byte-identical to the scheme's sign call fed the host-drawn nonces, over a ragged multi-chunk batch;
    one sample against ref_cpu"""
    import ref_cpu
    key, n = _key(0xC3), N_RAGGED
    wp0 = STRADDLE if scheme != 1 else 16 * 9 + 3
    sk, msg = _synth(n, 100 + scheme)
    gen = _gens(engine, n, 200 + scheme, affine) if scheme == 2 else None
    nonce = _nonces(key, wp0, n)
    got = engine.sign_stdrng(scheme, sk, msg, key, wp0, gen=gen, affine=affine, oblivious=oblivious)
    want = _host_sign(engine, scheme, sk, msg, nonce, gen, affine, oblivious)
    assert got[-1] == wp0 + 16 * n
    assert len(got) - 1 == len(want)
    for g, w in zip(got[:-1], want):
        assert (g == w).all()
    k = 64
    ref = (ref_cpu.sign(sk[:k], msg[:k], nonce[:k]) if scheme == 0 else
           ref_cpu.sign_double(sk[:k], msg[:k], nonce[:k]) if scheme == 1 else
           ref_cpu.sign_vargen(sk[:k], gen[:k], msg[:k], nonce[:k], affine=affine))
    for g, w in zip(got[:-1], ref):
        assert (g[:k] == w).all()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme,affine,oblivious", [(0, True, False), (1, True, True), (2, False, False), (2, True, True)])
def test_sign_stdrng_device_pointers(engine, scheme, affine, oblivious):
    import torch
    key, n, wp0 = _key(5), 5000 + 11, 16 * 41 + 15
    sk, msg = _synth(n, 300 + scheme)
    gen = _gens(engine, n, 400 + scheme, affine) if scheme == 2 else None
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda()
    d_sk, d_msg = dev(sk), dev(msg)
    d_gen = dev(gen) if gen is not None else None
    outs = [torch.zeros((n, w), dtype=torch.int32, device="cuda:0") for w in (8, 16, 16, 8)]
    fl = DEVICE_PTRS | (SIGN_OBLIVIOUS if oblivious else 0) | (POINTS_AFFINE if scheme == 2 and affine else 0)
    pos = StdRngPos.of(key, wp0)
    before = engine.launch_count
    rc = engine._lib.sb200_sign_stdrng(engine._h, n, fl, scheme, d_sk.data_ptr(), d_msg.data_ptr(),
                                       d_gen.data_ptr() if d_gen is not None else None, ctypes.byref(pos),
                                       outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr() if scheme == 1 else None,
                                       outs[3].data_ptr())
    torch.cuda.synchronize()
    assert rc == 0 and pos.word_pos == wp0 + 16 * n
    assert engine.launch_count - before == 2  # the draw kernel + the scheme's sign kernel
    want = _host_sign(engine, scheme, sk, msg, _nonces(key, wp0, n), gen, affine, oblivious)
    got = [outs[0], outs[1]] + ([outs[2]] if scheme == 1 else []) + [outs[3]]
    for g, w in zip(got, want):
        assert (g.cpu().numpy().view(np.uint32) == w).all()


# ---- typed mirrors --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("prefix", [0, 1, 3])
def test_python_typed_signers_keep_the_host_stream(engine, prefix):
    """SecretKey.sign_batch / sign_double_batch / SecretKeyVarGen.sign_batch at the reference's recipe
    (seed_from_u64(2321)) after `prefix` next_u64 calls (odd prefixes leave the stream mid-block): the signatures and
    the stream position afterwards equal those of drawing the nonces on the host"""
    api.set_engine(engine)
    try:
        for kind in ("single", "double", "vargen"):
            a, b = api.StdRng.seed_from_u64(2321), api.StdRng.seed_from_u64(2321)
            for _ in range(prefix):
                assert a.next_u64() == b.next_u64()
            n = 37
            sks = [api.SecretKey.random(a) for _ in range(n)]
            assert [api.SecretKey.random(b) for _ in range(n)] == sks
            msgs = [a.random_bls() for _ in range(n)]
            assert [b.random_bls() for _ in range(n)] == msgs
            wp = a.word_pos
            assert wp == b.word_pos == 2 * prefix + 32 * n
            sk_l, m_l = api._scalars([k.as_scalar() for k in sks]), api._fqs(msgs)
            if kind == "single":
                got = api.SecretKey.sign_batch(sks, a, msgs)
                u, Rr, _ = engine.sign(sk_l, m_l, api._scalars(b.random_scalars(n)))
                want = [api.Signature(api._int(u[i]), p) for i, p in enumerate(api._points_out(Rr))]
            elif kind == "double":
                got = api.SecretKey.sign_double_batch(sks, a, msgs)
                u, Rr, Rp, _ = engine.sign_double(sk_l, m_l, api._scalars(b.random_scalars(n)))
                want = [api.SignatureDouble(api._int(u[i]), x, y) for i, (x, y) in enumerate(zip(api._points_out(Rr), api._points_out(Rp)))]
            else:
                gk = [api.JubJubExtended(*o.pt_mul_fast(o.G, 1000 + i)) for i in range(n)]
                vks = [api.SecretKeyVarGen(k.as_scalar(), g) for k, g in zip(sks, gk)]
                got = api.SecretKeyVarGen.sign_batch(vks, a, msgs)
                u, Rr, _ = engine.sign_vargen(sk_l, api._points(gk), m_l, api._scalars(b.random_scalars(n)), affine=False)
                want = [api.SignatureVarGen(api._int(u[i]), p) for i, p in enumerate(api._points_out(Rr))]
            assert [s.to_bytes() for s in got] == [s.to_bytes() for s in want], kind
            assert a.word_pos == b.word_pos == wp + 16 * n
            assert [a.next_u64() for _ in range(9)] == [b.next_u64() for _ in range(9)]
        # the reference's recipe, against the oracle: sk, message, one signature
        rng, orng = api.StdRng.seed_from_u64(2321), o.StdRng.seed_from_u64(2321)
        for _ in range(prefix):
            rng.next_u64(), orng.next_u64()
        sk, message = api.SecretKey.random(rng), rng.random_bls()
        sig = sk.sign(rng, message)
        osk, om = orng.random_fr(), orng.random_fq()
        ou, oR, _ = o.sign(osk, orng.random_fr(), om)
        assert (sk.as_scalar(), message, sig.u(), sig.R().affine()) == (osk, om, ou, oR)
        assert rng.next_u64() == orng.next_u64()
        # a stream left inside a word signs with host-drawn nonces, still the same stream
        a, b = api.StdRng.seed_from_u64(9), api.StdRng.seed_from_u64(9)
        a.fill_bytes(3), b.fill_bytes(3)
        assert a.word_pos is None
        got = api.SecretKey.sign_batch([sk] * 5, a, [message] * 5)
        u, Rr, _ = engine.sign(api._scalars([sk.as_scalar()] * 5), api._fqs([message] * 5), api._scalars(b.random_scalars(5)))
        assert [s.u() for s in got] == [api._int(x) for x in u]
        assert a.fill_bytes(64) == b.fill_bytes(64)
    finally:
        api.set_engine(None)


@pytest.mark.gpu
def test_cpp_typed_signers_keep_the_host_stream():
    """include/schnorr_b200.hpp: the seeded batch signers (device-drawn nonces) equal the host-drawn path and leave the
    generator where the host draws would have"""
    exe = os.path.join(ROOT, "build", "test_stdrng_cpp")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe, os.path.join(ROOT, "tests", "cpp", "test_stdrng.cpp"),
                           "-L" + os.path.join(ROOT, "schnorr_b200"), "-lschnorr_b200",
                           "-Wl,-rpath," + os.path.join(ROOT, "schnorr_b200")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "ALL OK" in out.stdout
