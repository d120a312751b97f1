"""Witness rows of received signatures (include/schnorr_b200_witness.h, core.cuh verify_witness_core).

From the public tuple (PK, u, R[, R'], m) alone: the row sb200_sign_witness returns to the signer (u, R, PK, m, c,
SA = u B, SB = c PK ...) and the verdict SA + SB == R.  The CPU tests run the host build of the core against the Python
oracle; the GPU tests pin the two entry points' argument rules and launches, the round trip against the signer's rows,
the verdicts against sb200_verify* on the adversarial batches of test_gpu_scale_parity, and the byte-level call.
"""
import ctypes
import os
import random
import re
import subprocess

import numpy as np
import pytest

import hostlib as H
import schnorr_oracle as o
import vectors as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R
WIDTH = (11, 19, 13)


# ---- the oracle's row ---------------------------------------------------------------------------------------------
def oracle_row(scheme, pk, pk2, u, Rr, Rp, m, mul=o.pt_mul):
    """(row as integers, verdict) from the Python oracle; pk2 = PK' (1) or the generator (2), Rp = R' (1)"""
    if u >= R:
        return [0] * WIDTH[scheme], False
    if scheme == 1:
        c = o.challenge_hash_double(Rr, Rp, m)
        sa, sb, sa2, sb2 = mul(o.G, u), mul(pk, c), mul(o.G_NUMS, u), mul(pk2, c)
        row = [u, *Rr, *Rp, *pk, *pk2, m, c, *sa, *sb, *sa2, *sb2]
        return row, o.pt_add(sa, sb) == Rr and o.pt_add(sa2, sb2) == Rp
    c = o.challenge_hash(Rr, m)
    base = o.G if scheme == 0 else pk2
    sa, sb = mul(base, u), mul(pk, c)
    row = [u, *Rr, *pk] + ([*pk2] if scheme == 2 else []) + [m, c, *sa, *sb]
    return row, o.pt_add(sa, sb) == Rr


# ---- CPU: host build of the core ----------------------------------------------------------------------------------
def _host_lib():
    so = os.path.join(ROOT, "build", "host_witness.so")
    srcs = [os.path.join(ROOT, "tests", f) for f in ("host_witness.cpp", "host_arith.cpp", "host_shim.h")]
    csrc = os.path.join(ROOT, "schnorr_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-include", os.path.join(ROOT, "tests", "host_shim.h"),
                               "-o", so, os.path.join(ROOT, "tests", "host_witness.cpp")])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def hlib():
    return _host_lib()


@pytest.fixture(scope="module")
def htabs(hlib):
    return H.comb_tables(hlib)


def _host_row(hlib, tabs, scheme, pk, pk2, u, Rr, Rp, m, zs=None):
    """h_verify_witness on affine points (zs None) or projective ones with the given Z per point (pk, pk2, R, R')"""
    def enc(p, k):
        return H.pt_mont(p) if zs is None else H.pt_mont(p, zs[k])
    pts = [enc(p, k) if p is not None else np.zeros(24, np.uint32) for k, p in enumerate((pk, pk2, Rr, Rp))]
    rows = np.zeros(8 * WIDTH[scheme], np.uint32)
    ok = hlib.h_verify_witness(scheme, H.ptr(pts[0]), H.ptr(pts[1]), H.ptr(H.limbs(u)), H.ptr(pts[2]), H.ptr(pts[3]),
                               H.ptr(H.mont(m)), int(zs is None), 0, H.ptr(tabs[0]), H.ptr(tabs[1]), H.ptr(rows))
    return rows, bool(ok)


def _host_verify(hlib, tabs, scheme, pk, pk2, u, Rr, Rp, m):
    """the verdict of the host build of verify*_core: what sb200_verify* decides"""
    c = np.zeros(8, np.uint32)
    if scheme == 0:
        return bool(hlib.h_verify(H.ptr(H.pt_mont(pk)), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rr)), H.ptr(H.mont(m)), 1,
                                  H.ptr(tabs[0]), H.ptr(c)))
    if scheme == 1:
        return bool(hlib.h_verify_double(H.ptr(H.pt_mont(pk)), H.ptr(H.pt_mont(pk2)), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rr)),
                                         H.ptr(H.pt_mont(Rp)), H.ptr(H.mont(m)), 1, H.ptr(tabs[0]), H.ptr(tabs[1]), H.ptr(c)))
    return bool(hlib.h_verify_vargen(H.ptr(H.pt_mont(pk)), H.ptr(H.pt_mont(pk2)), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rr)),
                                     H.ptr(H.mont(m)), 1, H.ptr(c)))


def _signed(scheme, rnd):
    """one signature made by the host signer's arithmetic (oracle), as (sk, nonce, gen, tuple dict)"""
    sk, nonce, m = rnd.randrange(1, R), rnd.randrange(1, R), rnd.randrange(Q)
    gen = V.mul(o.G, rnd.randrange(1, R)) if scheme == 2 else None
    if scheme == 0:
        u, Rr, _ = o.sign(sk, nonce, m, mul=V.mul)
        t = dict(pk=V.mul(o.G, sk), pk2=None, u=u, Rr=Rr, Rp=None, m=m)
    elif scheme == 1:
        u, Rr, Rp, _ = o.sign_double(sk, nonce, m, mul=V.mul)
        t = dict(pk=V.mul(o.G, sk), pk2=V.mul(o.G_NUMS, sk), u=u, Rr=Rr, Rp=Rp, m=m)
    else:
        u, Rr, _ = o.sign_vargen(sk, gen, nonce, m, mul=V.mul)
        t = dict(pk=V.mul(gen, sk), pk2=gen, u=u, Rr=Rr, Rp=None, m=m)
    return sk, nonce, gen, t


def _host_cases(scheme, rnd):
    """(label, tuple) pairs: valid signatures and each corruption the issue of received signatures brings"""
    out = []
    for k in range(2):
        out.append((f"valid{k}", _signed(scheme, rnd)[3]))
    _, _, _, nb = _signed(scheme, rnd)
    tors = V.torsion_points()
    base = o.G if scheme != 2 else None
    for label in ("u+1", "m+1", "R+B", "neighbour key", "torsion key", "small-order key", "identity key", "u=0", "u=r-1",
                  "u=r", "u=2^256-1"):
        sk, nonce, gen, t = _signed(scheme, rnd)
        B = base if base is not None else gen
        if label == "u+1":
            t["u"] = (t["u"] + 1) % R
        elif label == "m+1":
            t["m"] = (t["m"] + 1) % Q
        elif label == "R+B":
            t["Rr"] = o.pt_add(t["Rr"], B)
        elif label == "neighbour key":
            t["pk"], t["pk2"] = nb["pk"], (nb["pk2"] if scheme == 1 else t["pk2"])
        elif label == "torsion key":  # PK = sk B + T: valid iff c T = O
            T = tors[rnd.randrange(1, len(tors))]
            t["pk"] = o.pt_add(t["pk"], T)
            if scheme == 1:
                t["pk2"] = o.pt_add(t["pk2"], T)
        elif label in ("small-order key", "identity key"):  # R = u B: valid iff c PK = O
            T = tors[rnd.randrange(1, len(tors))] if label == "small-order key" else o.IDENTITY
            t["pk"], t["u"] = T, nonce
            if scheme == 1:
                t["pk2"] = T
        elif label == "u=0":
            t["u"] = 0
        elif label == "u=r-1":
            t["u"] = R - 1
        elif label == "u=r":
            t["u"] = R
        else:
            t["u"] = (1 << 256) - 1
        out.append((label, t))
    return out


@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_host_rows_match_oracle(hlib, htabs, ark, scheme):
    H.setup_hades(hlib)  # the host build's Hades tables under the rule the `ark` fixture selected
    rnd = random.Random(700 + 10 * scheme + (ark == "plain"))
    seen = set()
    for label, t in _host_cases(scheme, rnd):
        args = (scheme, t["pk"], t["pk2"], t["u"], t["Rr"], t["Rp"], t["m"])
        rows, ok = _host_row(hlib, htabs, *args)
        got = [H.unmont(rows[8 * k:8 * k + 8]) for k in range(WIDTH[scheme])]
        want, want_ok = oracle_row(*args)
        assert got == want, (label, [k for k in range(len(want)) if got[k] != want[k]])
        assert ok == want_ok, label
        if t["u"] < R:
            assert ok == _host_verify(hlib, htabs, *args), label
        else:
            assert not (rows.any() or ok), label
        if label.startswith("valid"):
            assert ok
        seen.add(ok)
        # projective inputs: random Z per point, the same row and verdict
        zs = [rnd.randrange(1, Q) for _ in range(4)]
        prow, pok = _host_row(hlib, htabs, *args, zs=zs)
        assert (prow == rows).all() and pok == ok, label
    assert seen == {True, False}


@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_host_rows_equal_the_signers_rows(hlib, htabs, ark, scheme):
    """the central property: the row from the public tuple is bit-identical to the row witness_core gives the signer"""
    H.setup_hades(hlib)
    rnd = random.Random(800 + 10 * scheme + (ark == "plain"))
    for _ in range(3):
        sk, nonce, gen, t = _signed(scheme, rnd)
        zg = rnd.randrange(1, Q)
        signer = np.zeros(8 * WIDTH[scheme], np.uint32)
        hlib.h_witness(scheme, H.ptr(H.limbs(sk)), H.ptr(H.limbs(nonce)), H.ptr(H.mont(t["m"])),
                       H.ptr(H.pt_mont(gen, zg) if gen is not None else np.zeros(24, np.uint32)), 0, H.ptr(htabs[0]),
                       H.ptr(htabs[1]), H.ptr(signer))
        rows, ok = _host_row(hlib, htabs, scheme, t["pk"], t["pk2"], t["u"], t["Rr"], t["Rp"], t["m"])
        assert ok and (rows == signer).all()


def test_header_declares_exactly_the_bound_symbols():
    """include/schnorr_b200_witness.h declares the keys of _lib's second prototype table, the library exports them, and
    the main header's symbol list stays what schnorr_b200.h declares"""
    lib_path = os.path.join(ROOT, "schnorr_b200", "libschnorr_b200.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    from schnorr_b200 import _lib
    decl = lambda f: sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", f)).read())))
    assert decl("schnorr_b200_witness.h") == sorted(_lib._WITNESS_PROTOTYPES) == ["sb200_verify_witness", "sb200_verify_witness_bytes"]
    assert sorted(_lib.EXPORTED_SYMBOLS) == decl("schnorr_b200.h")
    assert not set(_lib._WITNESS_PROTOTYPES) & set(_lib.EXPORTED_SYMBOLS)
    lib = ctypes.CDLL(lib_path)
    assert all(hasattr(lib, s) for s in _lib._WITNESS_PROTOTYPES)
    bound = _lib.load_library()
    assert bound.sb200_verify_witness.argtypes is not None and bound.sb200_verify_witness_bytes.argtypes is not None


# ---- GPU ----------------------------------------------------------------------------------------------------------
OK, ARG = 0, -1
SPECS = [
    (f"verify_witness[{s}]", "verify_witness", True, (s,),
     [("in", "pk"), ("in", "gen" if s == 2 else "pkp"), ("in", "u"), ("in", "R"), ("in", "Rp"), ("in", "msg"), ("bm",),
      ("out", 8 * WIDTH[s])])
    for s in range(3)
] + [
    (f"verify_witness_bytes[{s}]", "verify_witness_bytes", True, (s,),
     [("in", ("pk32", "pk64", "pkg64")[s]), ("in", ("sig64", "sig96", "sig64")[s]), ("in", "msg32"), ("bm",),
      ("out", 8 * WIDTH[s]), ("bm",)])
    for s in range(3)
]
# flags: POINTS_AFFINE, DEVICE_PTRS, VERIFY_DUAL_PIPE, CHECK_POINTS, SIGN_OBLIVIOUS, unknown; null and misaligned per argument
EXPECTED = {
    "verify_witness[0]":       ((OK, OK, ARG, OK, ARG, ARG), (ARG, OK, ARG, ARG, OK, ARG, ARG, ARG), (ARG, OK, ARG, ARG, OK, ARG, OK, ARG)),
    "verify_witness[1]":       ((OK, OK, ARG, OK, ARG, ARG), (ARG,) * 8, (ARG,) * 6 + (OK, ARG)),
    "verify_witness[2]":       ((OK, OK, ARG, OK, ARG, ARG), (ARG, ARG, ARG, ARG, OK, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK, ARG, OK, ARG)),
    "verify_witness_bytes[0]": ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG, ARG)),
    "verify_witness_bytes[1]": ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG, ARG)),
    "verify_witness_bytes[2]": ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG, ARG)),
}
LAUNCHES = {**{f"verify_witness[{s}]": 1 for s in range(3)},         # the witness kernel
            **{f"verify_witness_bytes[{s}]": 2 for s in range(3)}}   # decode, witness


def _gpu_imports():
    import test_gpu_dispatch as D
    import test_gpu_scale_parity as SP
    return D, SP


# the dispatch test's call harness and fixtures (importing them needs no GPU)
from test_gpu_dispatch import Call, _cases, base  # noqa: E402,F401
from test_gpu_scale_parity import sizes  # noqa: E402,F401


@pytest.fixture
def witness_tables(monkeypatch):
    """this file's literal rows, visible to the dispatch test's harness (_cases reads its module's tables)"""
    D, _ = _gpu_imports()
    for sid in EXPECTED:
        monkeypatch.setitem(D.EXPECTED, sid, EXPECTED[sid])
        monkeypatch.setitem(D.LAUNCHES, sid, LAUNCHES[sid])
    return D


def test_tables_cover_both_calls():
    assert {s[1] for s in SPECS} == {s[len("sb200_"):] for s in re.findall(
        r"\b(sb200_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "schnorr_b200_witness.h")).read())}
    assert [s[0] for s in SPECS] == list(EXPECTED) and set(LAUNCHES) == set(EXPECTED)
    for sid, _n, _f, _i, args in SPECS:
        assert all(len(x) == len(args) for x in EXPECTED[sid][1:]) and len(EXPECTED[sid][0]) == 6, sid


@pytest.mark.gpu
@pytest.mark.parametrize("spec", SPECS, ids=[s[0] for s in SPECS])
def test_accept_reject_matrix(engine, base, spec, witness_tables):
    """each flag bit, each null and misaligned pointer, n = 0 and n = -1: the literal codes above; a rejected call writes
    and launches nothing and the valid call repeats bit for bit (test_gpu_dispatch's harness)"""
    witness_tables.test_accept_reject_matrix_and_the_context_stays_usable(engine, base, spec)
    assert [label for label, _kw, _rc in _cases(spec[0], len(spec[4]), True)][:6] == [f"flag {f}" for f in (1, 2, 4, 8, 16, 64)]
    for s in (3, -1):  # scheme outside {0, 1, 2}
        c = Call(engine, (spec[0], spec[1], spec[2], (s,), spec[4]), base, 32)
        assert c() == (ARG, 0)
        assert all((x == y).all() for x, y in zip(c.outputs(), c.initial_outputs()))


@pytest.mark.gpu
@pytest.mark.parametrize("spec", SPECS, ids=[s[0] for s in SPECS])
def test_launches_per_chunk(engine, base, spec, witness_tables):
    witness_tables.test_launch_counts_per_chunk(engine, base, spec)


def _rand_scalars(rs, n, bits=251):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << (bits - 224)) - 1
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_round_trip_with_the_signer(engine, scheme):
    """keygen / sign_witness on the device, then verify_witness on the public tuple: bit-identical rows, every verdict 1;
    affine and projective, host buffers over several ragged chunks, and one device-pointer call"""
    import torch
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE
    D, SP = _gpu_imports()
    n = D.N_CHUNKS
    assert len(SP.host_chunks(n)) > 1
    rs = np.random.RandomState(900 + scheme)
    sk, nonce, msg = _rand_scalars(rs, n), _rand_scalars(rs, n), _rand_scalars(rs, n, 254)
    gen = engine.keygen(_rand_scalars(rs, n)) if scheme == 2 else None
    rows = engine.sign_witness(scheme, sk, msg, nonce, gen=gen, affine=True)
    u = engine.fq_from_mont(np.ascontiguousarray(rows[:, 0]))  # u < r < q: the embedding is the integer itself
    Rr = np.ascontiguousarray(rows[:, 1:3].reshape(n, 16))
    if scheme == 0:
        pk, pk2, Rp = engine.keygen(sk), None, None
    elif scheme == 1:
        (pk, pk2), Rp = engine.keygen_double(sk), np.ascontiguousarray(rows[:, 3:5].reshape(n, 16))
    else:
        pk, pk2, Rp = engine.keygen_vargen(sk, gen), gen, None
    ok, got = engine.verify_witness(scheme, pk, u, Rr, msg, pk2=pk2, Rp=Rp)
    assert ok.all() and (got == rows).all()
    zs = [int(z) for z in rs.randint(2, 1 << 62, size=n, dtype=np.int64)]
    proj = lambda p: SP.projective(p, zs) if p is not None else None
    ok, got = engine.verify_witness(scheme, proj(pk), u, proj(Rr), msg, pk2=proj(pk2), Rp=proj(Rp), affine=False)
    assert ok.all() and (got == rows).all()
    # one device-pointer call
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev) if a is not None else None
    ins = [t(pk), t(pk2), t(u), t(Rr), t(Rp), t(msg)]
    bm = torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev)
    out = torch.zeros((n, WIDTH[scheme] * 8), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    rc = engine._lib.sb200_verify_witness(engine._h, n, POINTS_AFFINE | DEVICE_PTRS, scheme,
                                          *[ctypes.c_void_p(x.data_ptr()) if x is not None else None for x in ins],
                                          ctypes.c_void_p(bm.data_ptr()), ctypes.c_void_p(out.data_ptr()))
    torch.cuda.synchronize()
    assert rc == 0
    assert np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")[:n].all()
    assert (out.cpu().numpy().view(np.uint32).reshape(rows.shape) == rows).all()


# ---- adversarial batches above four waves (test_gpu_scale_parity's construction) ------------------------------------
def _split(scheme, arr):
    """(pk, pk2, u, R, R', m) from a scale-parity batch's verify arrays"""
    if scheme == 0:
        return arr[0], None, arr[1], arr[2], None, arr[3]
    if scheme == 1:
        return arr[0], arr[1], arr[2], arr[3], arr[4], arr[5]
    return arr[0], arr[1], arr[2], arr[3], None, arr[4]


def _witness(eng, scheme, arr, **kw):
    pk, pk2, u, Rr, Rp, m = _split(scheme, arr)
    return eng.verify_witness(scheme, pk, u, Rr, m, pk2=pk2, Rp=Rp, **kw)


def _sample(n, count=160):
    return np.unique(np.linspace(0, n - 1, count).astype(np.int64))


def _check_rows_against_oracle(scheme, arr, rows, idx):
    pk, pk2, u, Rr, Rp, m = _split(scheme, arr)
    pt = lambda a, i: (V.unmont(a[i, :8]), V.unmont(a[i, 8:16])) if a is not None else None
    for i in idx:
        want, _ = oracle_row(scheme, pt(pk, i), pt(pk2, i), V.to_int(u[i]), pt(Rr, i), pt(Rp, i), V.unmont(m[i]), mul=V.mul)
        got = [V.unmont(rows[i, k]) for k in range(WIDTH[scheme])]
        assert got == want, (scheme, int(i))


@pytest.fixture(scope="module")
def batches(sizes):
    _, SP = _gpu_imports()
    N = sizes[1]
    return [SP.make_single(N), SP.make_double(N), SP.make_vargen(N)]


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_adversarial_batches(engine, batches, sizes, scheme):
    _, SP = _gpu_imports()
    b = batches[scheme]
    assert b.N > 4 * sizes[0]
    ok, rows = _witness(engine, scheme, b.arr)
    ok_verify, _ = SP._verify(engine, scheme, b.arr)
    assert (ok == ok_verify).all(), np.nonzero(ok != ok_verify)[0][:8]
    SP._assert_same(b, ok)
    _check_rows_against_oracle(scheme, b.arr, rows, np.concatenate([_sample(b.N), np.nonzero(~b.want)[0][::997]]))
    assert b.ge_r.any() and not rows[b.ge_r].any()
    assert rows[~b.ge_r][:, 0].any(axis=1).all()  # every other tuple keeps its row, u included (u = 0 has probability 2^-251)


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_check_points_zeroes_malformed_tuples(engine, batches, scheme):
    """projective inputs with Z = 0 and off-curve points scattered: verdict 0 and a zero row there, the true row elsewhere"""
    _, SP = _gpu_imports()
    b = batches[scheme]
    arr = SP._proj_arrays(b, 47 + scheme)
    rs = np.random.RandomState(57 + scheme)
    bad = np.zeros(b.N, bool)
    for k in b.point_pos:
        sel = rs.randint(0, 64, size=b.N)
        zero, off = np.nonzero(sel == 0)[0], np.nonzero(sel == 1)[0]
        arr[k][zero, 16:] = 0
        arr[k][off, 8:16] = SP.from_ints([(v + 1) % Q for v in SP.to_ints(arr[k][off, 8:16])])
        bad[zero] = bad[off] = True
    ok, rows = _witness(engine, scheme, arr, affine=False, check_points=True)
    SP._assert_same(b, ok, want=b.want & ~bad)
    assert not rows[bad].any() and (b.want & bad).any()
    good = ~bad & ~b.ge_r
    _, plain = _witness(engine, scheme, b.arr)
    assert (rows[good] == plain[good]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_byte_level_call(engine, batches, scheme):
    """`invalid` and verdicts equal sb200_verify*_bytes' (non-canonical v, v that does not decode, u >= r, m >= q); rows
    of decoded tuples equal the limb call's, the others are zero; `invalid` may be NULL"""
    _, SP = _gpu_imports()
    b = batches[scheme]
    rs = np.random.RandomState(67 + scheme)
    pk, pk2, u, Rr, Rp, m = _split(scheme, b.arr)
    pts = [SP._enc_points(p) for p in (pk, pk2, Rr, Rp) if p is not None]
    ub, mb = SP._enc_scalars(u), SP._enc_scalars(m, mont=True)
    for p in pts:
        sel = rs.randint(0, 96, size=b.N)
        for i in np.nonzero(sel == 0)[0]:
            p[i] = np.frombuffer((Q + int(i) % 4096 | (int(i) >> 1 & 1) << 255).to_bytes(32, "little"), np.uint8)
        for i in np.nonzero(sel == 1)[0]:
            p[i] = np.frombuffer((SP.BAD_V[i % len(SP.BAD_V)] | (int(i) & 1) << 255).to_bytes(32, "little"), np.uint8)
    sel = rs.randint(0, 96, size=b.N)
    for i in np.nonzero(sel == 0)[0]:
        mb[i] = np.frombuffer((int.from_bytes(mb[i].tobytes(), "little") + Q).to_bytes(32, "little"), np.uint8)
    npk = 1 if scheme == 0 else 2
    pkb = np.concatenate(pts[:npk], axis=1)
    sig = np.concatenate([ub] + pts[npk:], axis=1)
    before = engine.launch_count
    ok, inv, rows = engine.verify_witness_bytes(scheme, pkb, sig, mb)
    assert engine.launch_count - before == 2 * len(SP.host_chunks(b.N))
    ok_v, inv_v = getattr(engine, ("verify_bytes", "verify_double_bytes", "verify_vargen_bytes")[scheme])(pkb, sig, mb)
    assert (inv == inv_v).all() and (ok == ok_v).all()
    assert inv.any() and (~inv).any() and (b.want & inv).any()
    assert not rows[inv].any()
    _, limb = _witness(engine, scheme, b.arr)
    assert (rows[~inv] == limb[~inv]).all()
    # invalid = NULL
    from schnorr_b200 import _lib
    bm = _lib.aligned_empty(((b.N + 31) // 32,)); bm[...] = 0
    rows2 = _lib.aligned_empty(rows.shape)
    pkb_, sig_, mb_ = (engine._bytes_arr(x, x.shape[1], "x") for x in (pkb, sig, mb))
    rc = engine._lib.sb200_verify_witness_bytes(engine._h, b.N, 0, scheme, pkb_.ctypes.data, sig_.ctypes.data, mb_.ctypes.data,
                                                bm.ctypes.data, rows2.ctypes.data, None)
    assert rc == 0
    assert (engine._unpack_bits(bm, b.N) == ok).all() and (rows2 == rows).all()


@pytest.mark.gpu
def test_multi_device_context(engine, batches):
    """a context over several devices gives the rows and verdicts of one device (with one GPU, as in the other
    multi-device tests, a context that lists device 0 twice still splits every call in two)"""
    import torch
    from schnorr_b200 import Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    one = [_witness(engine, scheme, b.arr) for scheme, b in enumerate(batches)]
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for scheme, b in enumerate(batches):
            ok, rows = _witness(eng, scheme, b.arr)
            assert (ok == one[scheme][0]).all() and (rows == one[scheme][1]).all(), scheme
    finally:
        eng.close()
