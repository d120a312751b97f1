"""Witness rows of received signatures against a keyset (include/schnorr_b200_keyset_witness.h, core.cuh
verify_witness_keyset_core).

The rows are those of sb200_verify_witness on the gathered keys, with c PK (c PK', u GEN) from the keyset's per-key combs
and the key's coordinates read back from its comb.  On the CPU: the header declares exactly the bound symbols, and the
host build of the core gives the host build of verify_witness_core's rows and the oracle's, bit for bit, for all three
schemes, affine and projective R, edge keys and wrong signatures; zero rows for an index past the keyset, a key without
its key_ok bit and u >= r.  On the GPU, for all three schemes over batches above four waves: parity with
Engine.verify_witness (affine, projective, SB200_CHECK_POINTS), with KeySet.verify's verdicts and challenges, rejected
keys, the byte-level call, updates and revocation, a multi-device context, the return codes and launches, and the typed
PublicKeySet.
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
import test_keyset as TK
import test_verify_witness as TW
from test_keyset import kbatches, make_keys, make_tuples, small  # noqa: F401
from test_keyset_live import bbatches, key_bytes, verify_bytes_ref  # noqa: F401
from test_gpu_scale_parity import sizes  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R
WIDTH = (11, 19, 13)
C_COL = (6, 10, 8)  # the row's c column per scheme
OK, ARG = 0, -1
SCHEMES = dict(argvalues=[0, 1, 2], ids=["single", "double", "vargen"])


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_header_declares_exactly_the_bound_symbols():
    lib_path = os.path.join(ROOT, "schnorr_b200", "libschnorr_b200.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    from schnorr_b200 import _lib
    text = open(os.path.join(ROOT, "include", "schnorr_b200_keyset_witness.h")).read()
    decl = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", text)))
    assert decl == sorted(_lib._KEYSET_WITNESS_PROTOTYPES) == ["sb200_verify_witness_keyset", "sb200_verify_witness_keyset_bytes"]
    others = set(_lib.EXPORTED_SYMBOLS) | set(_lib._WITNESS_PROTOTYPES) | set(_lib._KEYSET_PROTOTYPES) | set(_lib._KEYSET_LIVE_PROTOTYPES)
    assert not set(decl) & others
    assert all(hasattr(ctypes.CDLL(lib_path), s) for s in decl)


def _host_lib():
    """tests/host_keyset_witness.cpp: the keyset host build (host_keyset.cpp) and h_verify_witness_keyset"""
    so = os.path.join(ROOT, "build", "host_keyset_witness.so")
    srcs = [os.path.join(ROOT, "tests", f) for f in ("host_keyset_witness.cpp", "host_keyset.cpp", "host_arith.cpp", "host_shim.h")]
    csrc = os.path.join(ROOT, "schnorr_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-include", os.path.join(ROOT, "tests", "host_shim.h"),
                               "-o", so, os.path.join(ROOT, "tests", "host_keyset_witness.cpp")])
    lib = ctypes.CDLL(so)
    lib.h_verify_witness_keyset.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_uint32] + \
        [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
    return lib


@pytest.fixture(scope="module")
def klib():
    return _host_lib()


@pytest.fixture(scope="module")
def wlib():
    return TW._host_lib()


@pytest.fixture(scope="module")
def htabs(klib):
    return H.comb_tables(klib)


def _ks_row(klib, htabs, scheme, tabs, n_keys, key_ok, key, t, zs=None, check=0):
    """h_verify_witness_keyset: (row limbs, verdict); zs = Z of R (R') for projective input"""
    enc = lambda p, k: (H.pt_mont(p) if zs is None else H.pt_mont(p, zs[k])) if p is not None else np.zeros(24, np.uint32)
    rows = np.zeros(8 * WIDTH[scheme], np.uint32)
    ok = klib.h_verify_witness_keyset(scheme, H.ptr(tabs), n_keys, H.ptr(key_ok), key, H.ptr(H.limbs(t["u"])), H.ptr(enc(t["Rr"], 0)),
                                      H.ptr(enc(t["Rp"], 1)), H.ptr(H.mont(t["m"])), int(zs is None), check, H.ptr(htabs[0]),
                                      H.ptr(htabs[1]), H.ptr(rows))
    return rows, bool(ok)


@pytest.mark.parametrize("scheme", **SCHEMES)
def test_host_rows_equal_verify_witness_and_oracle(klib, wlib, htabs, ark, scheme):
    """every case of test_verify_witness (edge keys, wrong signatures, u = 0, u >= r) as a one-key keyset: the row and
    verdict of h_verify_witness and of the oracle, for affine and projective R, with and without SB200_CHECK_POINTS"""
    H.setup_hades(klib)
    H.setup_hades(wlib)
    rnd = random.Random(900 + 10 * scheme + (ark == "plain"))
    ok_one = np.ones(1, np.uint32)
    seen = set()
    for label, t in TW._host_cases(scheme, rnd):
        pts = (t["pk"], t["pk2"])[:1 if scheme == 0 else 2]
        z = rnd.randrange(2, Q) if label == "torsion key" else None  # one keyset built from a projective key
        tabs = np.concatenate([TK.host_table(klib, p, z) for p in pts])
        args = (scheme, t["pk"], t["pk2"], t["u"], t["Rr"], t["Rp"], t["m"])
        want_rows, want_ok = TW._host_row(wlib, htabs, *args)
        rows, ok = _ks_row(klib, htabs, scheme, tabs, 1, ok_one, 0, t)
        assert (rows == want_rows).all() and ok == want_ok, (label, [k for k in range(WIDTH[scheme])
                                                                     if (rows[8 * k:8 * k + 8] != want_rows[8 * k:8 * k + 8]).any()])
        orow, ook = TW.oracle_row(*args)
        assert [H.unmont(rows[8 * k:8 * k + 8]) for k in range(WIDTH[scheme])] == orow and ok == ook, label
        if t["u"] >= R:
            assert not rows.any() and not ok, label
        if label.startswith("valid"):
            assert ok, label
        seen.add(ok)
        zs = [rnd.randrange(1, Q) for _ in range(2)]
        assert _ks_row(klib, htabs, scheme, tabs, 1, ok_one, 0, t, zs=zs)[0].tobytes() == rows.tobytes(), label
        prow, pok = _ks_row(klib, htabs, scheme, tabs, 1, ok_one, 0, t, zs=zs, check=1)
        assert (prow == rows).all() and pok == ok, label
    assert seen == {True, False}


@pytest.mark.parametrize("scheme", **SCHEMES)
def test_host_zero_rows(klib, htabs, scheme):
    """an index past the keyset, a key without its key_ok bit, u >= r and (with SB200_CHECK_POINTS) a malformed R give
    an all-zero row and verdict 0; the same tuple against its key gives its true row"""
    H.setup_hades(klib)
    rnd = random.Random(950 + scheme)
    _, _, _, t = TW._signed(scheme, rnd)
    pts = (t["pk"], t["pk2"])[:1 if scheme == 0 else 2]
    tabs = np.concatenate([TK.host_table(klib, p) for p in pts] * 2)  # two keys: the same key twice
    good = np.full(1, 3, np.uint32)
    rows, ok = _ks_row(klib, htabs, scheme, tabs, 2, good, 1, t)
    assert ok and rows.any()
    for label, (okw, key, tt, chk) in {"index = n_keys": (good, 2, t, 0), "index = 2^32 - 1": (good, 2**32 - 1, t, 0),
                                       "key_ok clear": (np.full(1, 1, np.uint32), 1, t, 0), "u = r": (good, 1, dict(t, u=R), 0),
                                       "R off the curve": (good, 1, dict(t, Rr=(t["Rr"][0], (t["Rr"][1] + 1) % Q)), 1)}.items():
        zrows, zok = _ks_row(klib, htabs, scheme, tabs, 2, okw, key, tt, check=chk)
        assert not zrows.any() and not zok, label
    if scheme == 1:  # R' off the curve
        zrows, zok = _ks_row(klib, htabs, scheme, tabs, 2, good, 1, dict(t, Rp=(t["Rp"][0], (t["Rp"][1] + 1) % Q)), check=1)
        assert not zrows.any() and not zok


# ---- GPU ----------------------------------------------------------------------------------------------------------
def gathered_witness(eng, scheme, keys, t, affine=True, zk=None, **kw):
    """Engine.verify_witness on the gathered keys (projective keys with Z zk[key] when zk is given)"""
    import test_gpu_scale_parity as SP
    idx, u, Rr, Rp, m, _ = t
    g = np.minimum(idx, keys.K - 1)
    pk, pk2 = keys.pk[g], (keys.pk2[g] if keys.pk2 is not None else None)
    if zk is not None:
        zs = [zk[k] for k in g]
        pk, pk2 = SP.projective(pk, zs), (SP.projective(pk2, zs) if pk2 is not None else None)
    return eng.verify_witness(scheme, pk, u, Rr, m, pk2=pk2, Rp=Rp, affine=affine, **kw)


def _assert_rows(ok, rows, want_ok, want_rows, sel):
    bad = np.nonzero((ok != want_ok)[sel])[0]
    assert len(bad) == 0, f"{len(bad)} verdicts differ, first at {np.nonzero(sel)[0][bad[:8]].tolist()}"
    diff = np.nonzero((rows != want_rows).reshape(len(rows), -1)[sel].any(axis=1))[0]
    assert len(diff) == 0, f"{len(diff)} rows differ, first at {np.nonzero(sel)[0][diff[:8]].tolist()}"


def _assert_zero(ok, rows, sel):
    assert not ok[sel].any() and not rows[sel].any()


def _named(keys, ks, idx):
    """tuples whose key index is in the keyset and whose key holds its key_ok bit"""
    return (idx < keys.K) & ks.key_ok[np.minimum(idx, keys.K - 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_parity_with_verify_witness(engine, kbatches, sizes, scheme):
    """affine host buffers over several chunks, device pointers, projective inputs and SB200_CHECK_POINTS on malformed R:
    rows and verdicts of Engine.verify_witness on the gathered keys; verdicts and c of KeySet.verify"""
    import torch
    import test_gpu_scale_parity as SP
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE
    keys, t = kbatches[scheme]
    idx, u, Rr, Rp, m, cat = t
    N = sizes[1]
    with engine.keyset(scheme, keys.pk, keys.pk2) as ks:
        named = _named(keys, ks, idx)
        assert (~named & (idx < keys.K)).any() and (idx >= keys.K).any()
        want_ok, want_rows = gathered_witness(engine, scheme, keys, t)
        before = engine.launch_count
        ok, rows = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
        assert engine.launch_count - before == len(SP.host_chunks(N)) > 1
        _assert_rows(ok, rows, want_ok, want_rows, named)
        _assert_zero(ok, rows, ~named)
        assert 0.15 < ok.mean() < 0.6, ok.mean()
        live = named & (cat != 5)  # u + r: zero rows
        assert rows[live].reshape(live.sum(), -1).any(axis=1).all() and not rows[cat == 5].any()
        assert (~ok & live).sum() > N // 10  # wrong signatures keep their true rows
        kok, c = ks.verify(idx, u, Rr, m, Rp=Rp)
        assert (kok == ok).all()
        assert (rows[live, C_COL[scheme]] == engine.fq_to_mont(c[live])).all()
        # device pointers: one launch, the same bits
        dev = torch.device("cuda:0")
        td = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev) if a is not None else None
        ins = [td(idx), td(u), td(Rr), td(Rp), td(m)]
        bm = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
        rd = torch.zeros((N, WIDTH[scheme] * 8), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        before = engine.launch_count
        rc = engine._lib.sb200_verify_witness_keyset(engine._h, ks._h, N, POINTS_AFFINE | DEVICE_PTRS,
                                                     *[ctypes.c_void_p(x.data_ptr()) if x is not None else None for x in ins],
                                                     ctypes.c_void_p(bm.data_ptr()), ctypes.c_void_p(rd.data_ptr()))
        torch.cuda.synchronize()
        assert rc == OK and engine.launch_count - before == 1
        okd = np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool)
        assert (okd == ok).all() and (rd.cpu().numpy().view(np.uint32) == rows.reshape(N, -1)).all()
        # projective R (R') against projective gathered keys: the same rows
        rs = np.random.RandomState(500 + scheme)
        zs = [int(z) for z in rs.randint(2, 1 << 62, size=N, dtype=np.int64)]
        zk = [int(z) for z in rs.randint(2, 1 << 62, size=keys.K, dtype=np.int64)]
        tp = (idx, u, SP.projective(Rr, zs), SP.projective(Rp, zs) if Rp is not None else None, m, cat)
        pok, prow = ks.verify_witness(idx, u, tp[2], m, Rp=tp[3], affine=False)
        assert (pok == ok).all() and (prow == rows).all()
        # SB200_CHECK_POINTS with R (R') off the curve or Z = 0 scattered
        bad = np.zeros(N, bool)
        for k in ((2, 3) if scheme == 1 else (2,)):
            sel = rs.randint(0, 64, size=N)
            z0, off = np.nonzero(sel == 0)[0], np.nonzero(sel == 1)[0]
            tp[k][z0, 16:] = 0
            tp[k][off, 8:16] = SP.from_ints([(v + 1) % Q for v in SP.to_ints(tp[k][off, 8:16])])
            bad[z0] = bad[off] = True
        want_ok, want_rows = gathered_witness(engine, scheme, keys, tp, affine=False, zk=zk, check_points=True)
        cok, crow = ks.verify_witness(idx, u, tp[2], m, Rp=tp[3], affine=False, check_points=True)
        _assert_rows(cok, crow, want_ok, want_rows, named)
        _assert_zero(cok, crow, ~named | bad)
        assert (ok & bad).any()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_rejected_keys_leave_other_tuples_unchanged(engine, kbatches, scheme):
    """malformed keys, revoked slots and indices past the keyset: zero rows and verdict 0; every other tuple's row is the
    one a keyset without those keys gives"""
    keys, t = kbatches[scheme]
    idx, u, Rr, Rp, m, _ = t
    clean_pk, clean_pk2 = keys.pk.copy(), (keys.pk2.copy() if keys.pk2 is not None else None)
    off = np.nonzero(keys.kind == "off-curve")[0]
    g0 = np.nonzero(keys.kind == "plain")[0][0]
    clean_pk[off] = keys.pk[g0]
    if clean_pk2 is not None:
        clean_pk2[off] = keys.pk2[g0]
    gone = np.random.RandomState(600 + scheme).choice(np.nonzero(keys.kind == "plain")[0], size=30, replace=False).astype(np.uint32)
    with engine.keyset(scheme, keys.pk, keys.pk2) as a, engine.keyset(scheme, clean_pk, clean_pk2) as b:
        a.revoke(gone)
        oka, ra = a.verify_witness(idx, u, Rr, m, Rp=Rp)
        okb, rb = b.verify_witness(idx, u, Rr, m, Rp=Rp)
        g = np.minimum(idx, keys.K - 1)
        rejected = (idx >= keys.K) | np.isin(g, off) | np.isin(g, gone)
        assert rejected.any() and np.isin(g, gone).any() and np.isin(g, off).any()
        _assert_zero(oka, ra, rejected)
        _assert_rows(oka, ra, okb, rb, ~rejected)
        assert okb[np.isin(g, gone) & (idx < keys.K)].any()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_bytes_parity(engine, bbatches, scheme):
    """the byte-level call against Engine.verify_witness_bytes on the gathered key bytes, for every key that decodes;
    invalid bits of the signature and message alone; zero rows for undecodable tuples; two launches per chunk"""
    import torch
    import test_gpu_scale_parity as SP
    from schnorr_b200 import DEVICE_PTRS
    keys, t, pkb, sig, msg, bad = bbatches[scheme]
    idx, K, N = t[0], keys.K, len(t[0])
    g = np.minimum(idx, K - 1)
    with engine.keyset_from_bytes(scheme, pkb) as ks:
        named = _named(keys, ks, idx)
        before = engine.launch_count
        ok, inv, rows = ks.verify_witness_bytes(idx, sig, msg)
        assert engine.launch_count - before == 2 * len(SP.host_chunks(N))
        ref_ok, ref_inv, ref_rows = engine.verify_witness_bytes(scheme, pkb[g], sig, msg)
        _assert_rows(ok, rows, ref_ok, ref_rows, named)
        assert (inv[named] == ref_inv[named]).all()
        good_key = np.nonzero(ks.key_ok)[0][0]
        _, sig_inv = verify_bytes_ref(engine, scheme, pkb[np.full(N, good_key)], sig, msg)
        assert (inv == sig_inv).all() and bad.any() and inv[bad].all()
        _assert_zero(ok, rows, ~named | inv)
        assert 0.1 < ok.mean() < 0.6, ok.mean()
        okv, invv = ks.verify_bytes(idx, sig, msg)
        assert (okv == ok).all() and (invv == inv).all()
        # device pointers: one call, two launches; `invalid` may be null
        dev = torch.device("cuda:0")
        td = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
        ins = [td(idx), td(sig), td(msg)]
        bm = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
        rd = torch.zeros((N, WIDTH[scheme] * 8), dtype=torch.int32, device=dev)
        for with_inv in (True, False):
            ib = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            before = engine.launch_count
            rc = engine._lib.sb200_verify_witness_keyset_bytes(engine._h, ks._h, N, DEVICE_PTRS,
                                                               *[ctypes.c_void_p(x.data_ptr()) for x in ins + [bm, rd]],
                                                               ctypes.c_void_p(ib.data_ptr()) if with_inv else None)
            torch.cuda.synchronize()
            assert rc == OK and engine.launch_count - before == 2
            bits = lambda x: np.unpackbits(x.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool)
            assert (bits(bm) == ok).all() and (rd.cpu().numpy().view(np.uint32) == rows.reshape(N, -1)).all()
            assert (bits(ib) == inv).all() if with_inv else not bits(ib).any()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_update_and_revoke(engine, sizes, scheme):
    """after update the rows are verify_witness's on the new keys; after revoke they are zero; an update registers the
    revoked slots again"""
    rs = np.random.RandomState(700 + scheme)
    a = make_keys(engine, scheme, 200, 710 + scheme)
    b = make_keys(engine, scheme, 200, 720 + scheme)
    slots = rs.choice(200, size=60, replace=False).astype(np.uint32)
    final = TK.Keys()
    final.K, final.sk, final.kind = a.K, a.sk.copy(), a.kind.copy()
    final.pk, final.pk2 = a.pk.copy(), (a.pk2.copy() if a.pk2 is not None else None)
    final.sk[slots], final.kind[slots], final.pk[slots] = b.sk[slots], b.kind[slots], b.pk[slots]
    if final.pk2 is not None:
        final.pk2[slots] = b.pk2[slots]
    t = make_tuples(engine, scheme, final, sizes[1] // 2, 730 + scheme)
    idx, u, Rr, Rp, m, _ = t
    with engine.keyset(scheme, a.pk, a.pk2) as ks:
        ks.update(slots, b.pk[slots], b.pk2[slots] if b.pk2 is not None else None)
        named = _named(final, ks, idx)
        ok, rows = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
        want_ok, want_rows = gathered_witness(engine, scheme, final, t)
        _assert_rows(ok, rows, want_ok, want_rows, named)
        _assert_zero(ok, rows, ~named)
        hit = np.isin(idx, slots) & named
        assert ok[hit].any()
        ks.revoke(slots)
        ok2, rows2 = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
        _assert_zero(ok2, rows2, np.isin(idx, slots))
        _assert_rows(ok2, rows2, ok, rows, ~np.isin(idx, slots))
        ks.update(slots, b.pk[slots], b.pk2[slots] if b.pk2 is not None else None)
        ok3, rows3 = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
        assert (ok3 == ok).all() and (rows3 == rows).all()


@pytest.mark.gpu
def test_multi_device_context(engine, kbatches):
    """a context over several devices (device 0 twice on a one-GPU box) gives the rows of one device"""
    import torch
    from schnorr_b200 import Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for scheme, (keys, t) in enumerate(kbatches):
            idx, u, Rr, Rp, m, _ = t
            with engine.keyset(scheme, keys.pk, keys.pk2) as k1, eng.keyset(scheme, keys.pk, keys.pk2) as k2:
                ok1, r1 = k1.verify_witness(idx, u, Rr, m, Rp=Rp)
                ok2, r2 = k2.verify_witness(idx, u, Rr, m, Rp=Rp)
                assert (ok1 == ok2).all() and (r1 == r2).all(), scheme
    finally:
        eng.close()


SENTINEL = 0xA5A5A5A5


def _bufs(arrs):
    from schnorr_b200 import _lib
    out = []
    for a in arrs:
        if a is None:
            out.append(None)
            continue
        v = np.ascontiguousarray(a).view(np.uint32).reshape(-1)
        b = _lib.aligned_empty((v.size + 4,))
        b[:v.size] = v
        out.append(b)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_return_codes_write_and_launch_nothing(engine, small, scheme):
    """each rejected call of both entry points against a valid control: SB200_ERR_ARG, nothing written, nothing
    launched; n = 0 launches nothing; a foreign or destroyed keyset is rejected"""
    from schnorr_b200 import Engine
    import test_keyset_live as TL
    rs = np.random.RandomState(800 + scheme)
    keys, t = small[scheme]
    idx, u, Rr, Rp, m, _ = t
    n, w = len(idx), WIDTH[scheme]
    sig, msg, _ = TL.wire(engine, scheme, t, rs)
    lib = engine._lib
    ks = engine.keyset(scheme, keys.pk, keys.pk2)
    outs0 = lambda: [np.full((n + 31) // 32, SENTINEL, np.uint32), np.full((n, w * 8), SENTINEL, np.uint32),
                     np.full((n + 31) // 32, SENTINEL, np.uint32)]

    def call(byte, ks_h=None, n_=n, flags=None, null=None, mis=None, eng=engine):
        ins = [idx, sig, msg] if byte else [idx, u, Rr, Rp if scheme == 1 else None, m]
        bufs = _bufs(ins + outs0()[:3 if byte else 2])
        ptrs = [ctypes.c_void_p(b.ctypes.data) if b is not None else None for b in bufs]
        if null is not None:
            ptrs[null] = None
        if mis is not None:
            ptrs[mis] = ctypes.c_void_p(bufs[mis].ctypes.data + 4)
        fl = (0 if byte else 1) if flags is None else flags
        before = eng.launch_count
        f = lib.sb200_verify_witness_keyset_bytes if byte else lib.sb200_verify_witness_keyset
        rc = f(eng._h, ks._h if ks_h is None else ks_h, n_, fl, *ptrs)
        return rc, eng.launch_count - before, [b[:-4].copy() for b in bufs[len(ins):]]

    initial = [x.reshape(-1) for x in outs0()]
    for byte in (False, True):
        rc, launched, ref = call(byte)
        assert (rc, launched) == (OK, 2 if byte else 1)
        nin = 3 if byte else 5
        base = 0 if byte else 1
        cases = {"n = -1": dict(n_=-1)}
        for f in ((1, 4, 16, 64) if byte else (4, 16, 64)):  # the byte call takes SB200_DEVICE_PTRS only
            cases[f"flag {f}"] = dict(flags=base | f)
        if byte:
            cases["flag 8"] = dict(flags=8)
        for k in range(nin + (3 if byte else 2)):
            if not byte and k == 3 and scheme != 1:
                continue  # R' is read for scheme 1 only
            cases[f"null {k}"] = dict(null=k)
            cases[f"misaligned {k}"] = dict(mis=k)
        for label, kw in cases.items():
            rc, launched, outs = call(byte, **kw)
            if label in (f"null {nin + 2}", f"misaligned {nin}"):
                # `invalid` is optional; the verdict bitmap is written by words, as in the other calls
                assert (rc, launched) == (OK, 2 if byte else 1), (byte, label)
                continue
            assert (rc, launched) == (ARG, 0), (byte, label)
            assert all((x == y[:x.size]).all() for x, y in zip(outs, initial)), (byte, label)
        rc, launched, outs = call(byte, n_=0)
        assert (rc, launched) == (OK, 0) and all((x == y[:x.size]).all() for x, y in zip(outs, initial))
        other = Engine([0], ark=o.ARK_RULE)
        try:
            ks2 = other.keyset(scheme, keys.pk, keys.pk2)
            rc, launched, outs = call(byte, ks_h=ks2._h)
            assert (rc, launched) == (ARG, 0) and all((x == y[:x.size]).all() for x, y in zip(outs, initial))
            rc, _, outs2 = call(byte, ks_h=ks2._h, eng=other)
            assert rc == OK and all((x == y).all() for x, y in zip(outs2, ref))
            ks2.close()
        finally:
            other.close()
        rc, launched, outs = call(byte)
        assert (rc, launched) == (OK, 2 if byte else 1) and all((x == y).all() for x, y in zip(outs, ref))
    assert lib.sb200_verify_witness_keyset(engine._h, None, n, 1, *[None] * 7) == ARG
    assert lib.sb200_verify_witness_keyset_bytes(engine._h, None, n, 0, *[None] * 6) == ARG
    dead = ks._h
    ks.close()  # a destroyed keyset
    rc, launched, outs = call(False, ks_h=dead)
    assert (rc, launched) == (ARG, 0) and all((x == y[:x.size]).all() for x, y in zip(outs, initial))


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_typed_public_key_set(engine, scheme):
    """PublicKeySet.witness_batch / _bytes == Engine.verify_witness / _bytes on the gathered keys"""
    from schnorr_b200 import api
    import vectors as V
    prev = api._engine
    api.set_engine(engine)
    try:
        rng = api.StdRng.seed_from_u64(4321 + scheme)
        n_keys, n = 12, 200
        if scheme == 0:
            sks = [api.SecretKey.random(rng) for _ in range(n_keys)]
            keys = api.PublicKey.from_secret_keys(sks)
            keys[3] = api.PublicKey.from_raw_unchecked(api.JubJubExtended(*V.torsion_points()[5]))
        elif scheme == 1:
            sks = [api.SecretKey.random(rng) for _ in range(n_keys)]
            keys = [api.PublicKeyDouble.from_secret_key(k) for k in sks]
        else:
            sks = [api.SecretKeyVarGen.random(rng) for _ in range(n_keys)]
            keys = [api.PublicKeyVarGen.from_secret_key(k) for k in sks]
        rs = np.random.RandomState(scheme)
        idx = rs.randint(0, n_keys, size=n)
        msgs = [int(x) for x in rs.randint(0, 1 << 62, size=n, dtype=np.int64)]
        if scheme == 0:
            sigs = api.SecretKey.sign_batch([sks[i] for i in idx], rng, msgs)
        elif scheme == 1:
            sigs = api.SecretKey.sign_double_batch([sks[i] for i in idx], rng, msgs)
        else:
            sigs = api.SecretKeyVarGen.sign_batch([sks[i] for i in idx], rng, msgs)
        msgs = [mm + (k % 3 == 0) for k, mm in enumerate(msgs)]  # a third corrupted
        with api.PublicKeySet(keys) as ks:
            ok, rows = ks.witness_batch(idx, sigs, msgs)
            assert (ok == ks.verify_batch(idx, sigs, msgs)).all() and ok.any() and not ok.all()
            pkb = np.stack([np.frombuffer(keys[i].to_bytes(), np.uint8) for i in idx])
            sigb = [s.to_bytes() for s in sigs]
            msgb = [int(mm).to_bytes(32, "little") for mm in msgs]
            want_ok, _, want_rows = engine.verify_witness_bytes(scheme, pkb, b"".join(sigb), b"".join(msgb))
            assert (ok == want_ok).all() and (rows == want_rows).all()
            bok, binv, brows = ks.witness_batch_bytes(idx, sigb, msgb)
            assert (bok == ok).all() and not binv.any() and (brows == rows).all()
            with pytest.raises(IndexError):
                ks.witness_batch([n_keys], sigs[:1], msgs[:1])
            with pytest.raises(IndexError):
                ks.witness_batch_bytes([-1], sigb[:1], msgb[:1])
    finally:
        api.set_engine(prev)
