"""Byte-level keysets and live keysets (include/schnorr_b200_keyset_live.h).

On the CPU: the header declares exactly the bound symbols, and the library exports them.  On the GPU, for all three
schemes: sb200_verify_keyset_bytes against sb200_verify*_bytes on the gathered key bytes (malformed signatures and
messages included), sb200_keyset_create_bytes against sb200_keyset_create on the decoded keys, an updated keyset against
one freshly created from the final key list, revocation, the ordering of updates against enqueued verifications, a
multi-device context, the return codes and launches, and the typed PublicKeySet.
"""
import ctypes
import os
import re

import numpy as np
import pytest

import schnorr_oracle as o
import vectors as V
from test_keyset import Keys, _assert_ok, _ks_verify, _rand_scalars, make_keys, make_tuples, reference
from test_gpu_scale_parity import sizes  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R
OK, ARG = 0, -1
KEY_BYTES, SIG_BYTES = (32, 64, 64), (64, 96, 64)
SCHEMES = dict(argvalues=[0, 1, 2], ids=["single", "double", "vargen"])


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_header_declares_exactly_the_bound_symbols():
    lib_path = os.path.join(ROOT, "schnorr_b200", "libschnorr_b200.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    from schnorr_b200 import _lib
    text = open(os.path.join(ROOT, "include", "schnorr_b200_keyset_live.h")).read()
    decl = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", text)))
    assert decl == sorted(_lib._KEYSET_LIVE_PROTOTYPES) == ["sb200_keyset_create_bytes", "sb200_keyset_revoke", "sb200_keyset_update",
                                                            "sb200_keyset_update_bytes", "sb200_verify_keyset_bytes"]
    live = set(_lib._KEYSET_LIVE_PROTOTYPES)
    assert not live & (set(_lib.EXPORTED_SYMBOLS) | set(_lib._WITNESS_PROTOTYPES) | set(_lib._KEYSET_PROTOTYPES))
    assert all(hasattr(ctypes.CDLL(lib_path), s) for s in decl)


# ---- wire-format helpers --------------------------------------------------------------------------------------------
def _nonresidue_v():
    """a v < q whose point does not decompress ((v^2 - 1) / (1 + d v^2) is not a square)"""
    from schnorr_b200 import api
    for v in range(2, 1000):
        try:
            api.JubJubExtended.from_bytes(v.to_bytes(32, "little"))
        except api.InvalidData:
            return v
    raise AssertionError("no non-residue below 1000")


BAD_POINTS = [Q.to_bytes(32, "little"), (Q | 1 << 255).to_bytes(32, "little"), ((1 << 255) - 1).to_bytes(32, "little")]


def key_bytes(eng, pk, pk2):
    """the keys' to_bytes(): [K, 32 | 64] uint8"""
    b = eng.points_compress(pk)
    return b if pk2 is None else np.concatenate([b, eng.points_compress(pk2)], axis=1)


def wire(eng, scheme, t, rs, frac=0.06):
    """(sig bytes, msg bytes, malformed) of tuples t, with a fraction of the rows made undecodable: u >= r, v >= q in R (R'),
    R (R') that does not decompress, msg >= q"""
    idx, u, Rr, Rp, m, _ = t
    N = len(idx)
    parts = [np.ascontiguousarray(u).view(np.uint8).reshape(N, 32), eng.points_compress(Rr)]
    if scheme == 1:
        parts.append(eng.points_compress(Rp))
    sig = np.ascontiguousarray(np.concatenate(parts, axis=1))
    msg = np.ascontiguousarray(eng.fq_from_mont(m).view(np.uint8).reshape(N, 32))
    kinds = 6 if scheme == 1 else 4
    sel = np.nonzero(rs.rand(N) < frac)[0]
    kind = rs.randint(0, kinds, size=len(sel))
    nonres = _nonresidue_v().to_bytes(32, "little")
    for i, k in zip(sel, kind):
        if k == 0:
            sig[i, :32] = np.frombuffer(((1 << 256) - 1 - int(rs.randint(0, 1000))).to_bytes(32, "little"), np.uint8)
        elif k in (1, 4):  # v >= q in R / R'
            off = 32 if k == 1 else 64
            sig[i, off:off + 32] = np.frombuffer(BAD_POINTS[int(rs.randint(0, 3))], np.uint8)
        elif k in (2, 5):  # v < q, not on the curve
            off = 32 if k == 2 else 64
            sig[i, off:off + 32] = np.frombuffer(nonres, np.uint8)
        else:
            msg[i] = np.frombuffer((Q + int(rs.randint(0, 1000))).to_bytes(32, "little"), np.uint8)
    bad = np.zeros(N, bool)
    bad[sel] = True
    return sig, msg, bad


def verify_bytes_ref(eng, scheme, pkb, sig, msg):
    f = (eng.verify_bytes, eng.verify_double_bytes, eng.verify_vargen_bytes)[scheme]
    return f(pkb, sig, msg)


_BB = {}


@pytest.fixture
def bbatches(engine, sizes):
    """per scheme: 300 keys (10 % off the curve: bytes that decode to another point or not at all) and a batch above four
    waves with 10 % semantic corruption and 6 % undecodable rows, as bytes"""
    if "b" not in _BB:
        out = []
        for scheme in range(3):
            keys = make_keys(engine, scheme, 300, 140 + scheme)
            t = make_tuples(engine, scheme, keys, sizes[1], 150 + scheme)
            sig, msg, bad = wire(engine, scheme, t, np.random.RandomState(160 + scheme))
            out.append((keys, t, key_bytes(engine, keys.pk, keys.pk2), sig, msg, bad))
        _BB["b"] = out
    return _BB["b"]


# ---- 1. byte-level parity -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_verify_bytes_parity(engine, bbatches, sizes, scheme):
    import test_gpu_scale_parity as SP
    keys, t, pkb, sig, msg, bad = bbatches[scheme]
    idx, K, N = t[0], keys.K, len(t[0])
    g = np.minimum(idx, K - 1)
    with engine.keyset_from_bytes(scheme, pkb) as ks, engine.keyset(scheme, keys.pk, keys.pk2) as kl:
        dec = ks.key_ok
        assert dec.any() and not dec.all()
        before = engine.launch_count
        ok, inv = ks.verify_bytes(idx, sig, msg)
        assert engine.launch_count - before == 2 * len(SP.host_chunks(N))
        ref_ok, ref_inv = verify_bytes_ref(engine, scheme, pkb[g], sig, msg)
        good_key = np.nonzero(dec)[0][0]  # the signature's and message's own from_bytes, whatever key a tuple names
        _, sig_inv = verify_bytes_ref(engine, scheme, pkb[np.full(N, good_key)], sig, msg)
        named = (idx < K) & dec[g]
        _assert_ok(ok[named], ref_ok[named])
        _assert_ok(inv[named], ref_inv[named])
        _assert_ok(inv, sig_inv)
        assert not ok[~named].any() and not ok[inv].any()
        assert bad.any() and inv[bad].all() and (inv & ~bad).any()  # u + r rows are undecodable too
        assert (ref_inv & ~sig_inv & (idx < K)).any()  # keys whose bytes do not decode: invalid there, not here
        assert 0.1 < ok.mean() < 0.6, ok.mean()
        # valid rows whose key is the registered limb key: the limb-level keyset's verdicts
        same = ~inv & (keys.kind[g] != "off-curve")
        okl, _ = _ks_verify(kl, t)
        _assert_ok(ok[same], okl[same])
        # device pointers: one call, two launches, the same bits
        import torch
        from schnorr_b200 import DEVICE_PTRS
        dev = torch.device("cuda:0")
        td = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
        ins = [td(idx), td(sig), td(msg)]
        bm = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
        ib = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        before = engine.launch_count
        rc = engine._lib.sb200_verify_keyset_bytes(engine._h, ks._h, N, DEVICE_PTRS, *[ctypes.c_void_p(x.data_ptr()) for x in ins + [bm, ib]])
        torch.cuda.synchronize()
        assert rc == OK and engine.launch_count - before == 2
        bits = lambda x: np.unpackbits(x.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool)
        _assert_ok(bits(bm), ok)
        _assert_ok(bits(ib), inv)


# ---- 2. create_bytes against create ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_create_bytes_equals_create(engine, bbatches, scheme):
    keys, t, pkb, _, _, _ = bbatches[scheme]
    K, idx = keys.K, t[0]
    pts, dok = engine.points_decompress(pkb[:, :32].copy())
    pts2, dok2 = (engine.points_decompress(pkb[:, 32:].copy()) if scheme else (None, True))
    with engine.keyset_from_bytes(scheme, pkb) as kb, engine.keyset(scheme, pts, pts2) as kl:
        assert (kb.key_ok == (dok & dok2)).all()
        for kind in ("torsion", "small-order", "identity", "plain"):
            assert kb.key_ok[keys.kind == kind].all(), kind
        okb, cb = _ks_verify(kb, t)
        okl, cl = _ks_verify(kl, t)
        g = np.minimum(idx, K - 1)
        dec = (idx < K) & kb.key_ok[g]
        _assert_ok(okb[dec], okl[dec])
        assert (cb == cl).all() and not okb[~dec].any()
        for kind in ("torsion", "small-order", "identity"):  # edge keys verify exactly as the limb keyset says
            sel = dec & (keys.kind[g] == kind) & (t[5] < 4)
            assert okb[sel].any(), kind


# ---- 3. update equals rebuild ---------------------------------------------------------------------------------------
def _replaced(a, b, slots):
    """the key list a with rows `slots` taken from b"""
    k = Keys()
    k.K, k.sk, k.kind = a.K, a.sk.copy(), a.kind.copy()
    k.pk = a.pk.copy()
    k.pk2 = a.pk2.copy() if a.pk2 is not None else None
    k.sk[slots], k.kind[slots], k.pk[slots] = b.sk[slots], b.kind[slots], b.pk[slots]
    if k.pk2 is not None:
        k.pk2[slots] = b.pk2[slots]
    return k


def _update_slots(a, b, rs):
    """scattered slots, with malformed -> good and good -> malformed among them"""
    K = a.K
    to_good = np.nonzero((a.kind == "off-curve") & (b.kind == "plain"))[0][:6]
    to_bad = np.nonzero((a.kind == "plain") & (b.kind == "off-curve"))[0][:6]
    rest = rs.choice(np.setdiff1d(np.arange(K), np.concatenate([to_good, to_bad])), size=48, replace=False)
    s = np.concatenate([to_good, to_bad, rest])
    rs.shuffle(s)
    assert len(to_good) >= 3 and len(to_bad) >= 3
    return s.astype(np.uint32), to_good, to_bad


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_update_equals_rebuild(engine, sizes, scheme):
    import test_gpu_scale_parity as SP
    rs = np.random.RandomState(200 + scheme)
    a = make_keys(engine, scheme, 300, 210 + scheme)
    b = make_keys(engine, scheme, 300, 220 + scheme)
    slots, to_good, to_bad = _update_slots(a, b, rs)
    final = _replaced(a, b, slots)
    # three groups: affine limbs, projective limbs, bytes (keys off the curve as bytes that do not decode)
    g1, g2, g3 = slots[:20], slots[20:40], slots[40:]
    zs = [int(z) for z in rs.randint(2, 1 << 62, size=len(g2), dtype=np.int64)]
    bb = key_bytes(engine, b.pk[g3], b.pk2[g3] if b.pk2 is not None else None)
    bb[b.kind[g3] == "off-curve", :32] = np.frombuffer(BAD_POINTS[0], np.uint8)
    N = sizes[1] // 2
    t_old, t_new = make_tuples(engine, scheme, a, N, 230 + scheme), make_tuples(engine, scheme, final, N, 240 + scheme)
    t = tuple(np.concatenate([x, y]) if x is not None else None for x, y in zip(t_old, t_new))
    with engine.keyset(scheme, a.pk, a.pk2) as ka, engine.keyset(scheme, final.pk, final.pk2) as kf:
        ok_before, _ = _ks_verify(ka, t)
        n1 = ka.update(g1, b.pk[g1], b.pk2[g1] if b.pk2 is not None else None)
        n2 = ka.update(g2, SP.projective(b.pk[g2], zs), SP.projective(b.pk2[g2], zs) if b.pk2 is not None else None, affine=False)
        before = engine.launch_count
        n3 = ka.update_bytes(g3, bb)
        assert engine.launch_count - before == 2  # decode + one build launch
        assert (np.concatenate([n1, n2, n3]) == (final.kind[slots] != "off-curve")).all()
        assert (ka.key_ok == kf.key_ok).all() and ka.key_ok[to_good].all() and not ka.key_ok[to_bad].any()
        ok_a, c_a = _ks_verify(ka, t)
        ok_f, c_f = _ks_verify(kf, t)
        _assert_ok(ok_a, ok_f, c_a, c_f)
        want, _ = reference(engine, scheme, final, t, kf.key_ok)
        _assert_ok(ok_a, want)
        idx, cat = t[0], t[5]
        g = np.minimum(idx, a.K - 1)
        # signed tuples that must verify: prime-order keys, and for the variable generator not the whole-curve generators
        # of make_keys (every fourth key), where u GEN + c PK == R does not follow from signing mod r
        signed = (cat < 4) & ((g % 4 != 0) if scheme == 2 else True)
        upd, first = np.isin(idx, slots) & signed, np.arange(2 * N) < N
        old = upd & first & (a.kind[g] == "plain") & (final.kind[g] == "plain")
        new = upd & ~first & (final.kind[g] == "plain")
        assert old.sum() > 100 and ok_before[old].all() and not ok_a[old].any()  # the old keys' signatures now fail
        assert new.sum() > 100 and ok_a[new].all()
        assert ok_a[np.isin(idx, to_good) & ~first & signed].all()


# ---- 4. revoke ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_revoke(engine, bbatches, scheme):
    keys, t, pkb, sig, msg, _ = bbatches[scheme]
    rs = np.random.RandomState(300 + scheme)
    gone = rs.choice(keys.K, size=40, replace=False).astype(np.uint32)
    idx = t[0]
    with engine.keyset(scheme, keys.pk, keys.pk2) as ks, engine.keyset_from_bytes(scheme, pkb) as kb:
        ok0, c0 = _ks_verify(ks, t)
        okb0, inv0 = kb.verify_bytes(idx, sig, msg)
        before = engine.launch_count
        ks.revoke(gone)
        kb.revoke(gone)
        assert engine.launch_count - before == 2 and not ks.key_ok[gone].any() and not kb.key_ok[gone].any()
        ok1, c1 = _ks_verify(ks, t)
        okb1, inv1 = kb.verify_bytes(idx, sig, msg)
        hit = np.isin(idx, gone)
        assert (ok0[hit].any() and okb0[hit].any()) and not ok1[hit].any() and not okb1[hit].any()
        _assert_ok(ok1[~hit], ok0[~hit], c1, c0)
        _assert_ok(okb1[~hit], okb0[~hit])
        _assert_ok(inv1, inv0)
        # an update registers the keys again
        ks.update(gone, keys.pk[gone], keys.pk2[gone] if keys.pk2 is not None else None)
        kb.update_bytes(gone, pkb[gone])
        ok2, c2 = _ks_verify(ks, t)
        okb2, _ = kb.verify_bytes(idx, sig, msg)
        _assert_ok(ok2, ok0, c2, c0)
        _assert_ok(okb2, okb0)


# ---- 5. ordering ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_update_is_ordered_after_enqueued_verifications(engine, sizes, scheme):
    """verify -> update -> verify with SB200_DEVICE_PTRS on a user stream and no synchronisation in between: the first
    verification sees the old keys, the second the new ones; once with host keys, once with device keys"""
    import torch
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE
    a = make_keys(engine, scheme, 64, 400 + scheme)
    b = make_keys(engine, scheme, 64, 410 + scheme)
    N = sizes[1]
    t = make_tuples(engine, scheme, a, N, 420 + scheme)
    all_slots = np.arange(64, dtype=np.uint32)
    dev = torch.device("cuda:0")
    td = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int32).reshape(-1)).to(dev) if x is not None else None
    idx, u, Rr, Rp, m, _ = t
    ins = [td(idx), td(u), td(Rr), td(Rp), td(m)]
    with engine.keyset(scheme, a.pk, a.pk2) as ka, engine.keyset(scheme, b.pk, b.pk2) as kb:
        want_a, c_a = _ks_verify(ka, t)
        want_b, _ = _ks_verify(kb, t)
        assert (want_a != want_b).sum() > N // 8
        st = torch.cuda.Stream()
        engine.set_stream(st.cuda_stream)
        try:
            for step, (src, dst) in enumerate(((a, b), (b, a))):
                bms = [torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev) for _ in range(2)]
                keys_dev = [td(dst.pk), td(dst.pk2)]
                torch.cuda.synchronize()
                call = lambda bm: engine._lib.sb200_verify_keyset(engine._h, ka._h, N, POINTS_AFFINE | DEVICE_PTRS,
                                                                  *[ctypes.c_void_p(x.data_ptr()) if x is not None else None for x in ins],
                                                                  ctypes.c_void_p(bm.data_ptr()), None)
                assert call(bms[0]) == OK
                if step == 0:  # keys from host memory
                    ka.update(all_slots, dst.pk, dst.pk2)
                else:  # keys on the device, read on the caller's stream
                    s = _aligned(all_slots)
                    rc = engine._lib.sb200_keyset_update(ka._h, 64, POINTS_AFFINE | DEVICE_PTRS, s.ctypes.data,
                                                         *[ctypes.c_void_p(x.data_ptr()) if x is not None else None for x in keys_dev], None)
                    assert rc == OK
                assert call(bms[1]) == OK
                st.synchronize()
                got = [np.unpackbits(x.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool) for x in bms]
                first, second = (want_a, want_b) if step == 0 else (want_b, want_a)
                _assert_ok(got[0], first)
                _assert_ok(got[1], second)
        finally:
            engine.set_stream(0)


def _aligned(a):
    from schnorr_b200 import _lib
    a = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1)
    b = _lib.aligned_empty((a.size + 4,))
    b[:a.size] = a
    return b


# ---- 6. multi-device context ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_multi_device_context(engine, bbatches):
    """update and revoke reach every device of a context over several devices (device 0 twice on a one-GPU box): the
    sharded verdicts equal one device's; SB200_DEVICE_PTRS is refused there for create_bytes and update"""
    import torch
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE, Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for scheme, (keys, t, pkb, sig, msg, _) in enumerate(bbatches):
            rs = np.random.RandomState(500 + scheme)
            new = make_keys(engine, scheme, keys.K, 510 + scheme)
            slots = rs.choice(keys.K, size=50, replace=False).astype(np.uint32)
            gone = np.setdiff1d(rs.choice(keys.K, size=30, replace=False), slots).astype(np.uint32)
            pair = []
            for e in (engine, eng):
                ks = e.keyset_from_bytes(scheme, pkb)
                ks.update(slots[:25], new.pk[slots[:25]], new.pk2[slots[:25]] if new.pk2 is not None else None)
                ks.update_bytes(slots[25:], key_bytes(engine, new.pk[slots[25:]], new.pk2[slots[25:]] if new.pk2 is not None else None))
                ks.revoke(gone)
                pair.append((ks, _ks_verify(ks, t), ks.verify_bytes(t[0], sig, msg)))
            (k1, (ok1, c1), (b1, i1)), (k2, (ok2, c2), (b2, i2)) = pair
            assert (k1.key_ok == k2.key_ok).all() and not k2.key_ok[gone].any()
            _assert_ok(ok2, ok1, c2, c1)
            _assert_ok(b2, b1)
            _assert_ok(i2, i1)
            assert ok1.any() and not ok2[np.isin(t[0], gone)].any()
            for ks, *_ in pair:
                ks.close()
        keys = bbatches[0][0]
        d = torch.from_numpy(bbatches[0][2].reshape(-1)).cuda()
        h = ctypes.c_void_p()
        assert eng._lib.sb200_keyset_create_bytes(eng._h, 0, keys.K, DEVICE_PTRS, ctypes.c_void_p(d.data_ptr()), None, ctypes.byref(h)) == ARG
        assert not h.value
        with eng.keyset(0, keys.pk) as ks:
            dp = torch.from_numpy(keys.pk[:4].view(np.int32)).cuda()
            s = _aligned(np.arange(4))
            before = eng.launch_count
            assert eng._lib.sb200_keyset_update(ks._h, 4, POINTS_AFFINE | DEVICE_PTRS, s.ctypes.data, ctypes.c_void_p(dp.data_ptr()),
                                                None, None) == ARG
            assert eng._lib.sb200_keyset_update_bytes(ks._h, 4, DEVICE_PTRS, s.ctypes.data, ctypes.c_void_p(d.data_ptr()), None) == ARG
            assert eng.launch_count == before
    finally:
        eng.close()


# ---- 7. return codes and launches -----------------------------------------------------------------------------------
SENTINEL = 0xA5A5A5A5


def plain_keys(eng, scheme, K, seed):
    """K prime-order keys"""
    rs = np.random.RandomState(seed)
    k = Keys()
    k.K, k.sk, k.kind = K, _rand_scalars(rs, K), np.array(["plain"] * K)
    if scheme == 0:
        k.pk, k.pk2 = eng.keygen(k.sk), None
    elif scheme == 1:
        k.pk, k.pk2 = eng.keygen_double(k.sk)
    else:
        k.pk2 = eng.keygen(_rand_scalars(rs, K))
        k.pk = eng.keygen_vargen(k.sk, k.pk2)
    return k


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_return_codes_write_and_launch_nothing(engine, scheme):
    from schnorr_b200 import Engine
    lib = engine._lib
    rs = np.random.RandomState(600 + scheme)
    keys = plain_keys(engine, scheme, 40, 610 + scheme)
    t = make_tuples(engine, scheme, keys, 70, 620 + scheme)
    t = (t[0] % 40,) + t[1:]
    sig, msg, _ = wire(engine, scheme, t, rs)
    pkb = key_bytes(engine, keys.pk, keys.pk2)
    n, K = 70, 40
    ks = engine.keyset_from_bytes(scheme, pkb)

    # sb200_verify_keyset_bytes: key_index, sig, msg, verdicts, invalid
    def vcall(ks_h=None, n_=n, flags=0, null=None, mis=None, eng=engine):
        bufs = [_aligned(t[0]), _aligned(sig.view(np.uint32)), _aligned(msg.view(np.uint32)),
                _aligned(np.full((n + 31) // 32, SENTINEL)), _aligned(np.full((n + 31) // 32, SENTINEL))]
        ptrs = [ctypes.c_void_p(b.ctypes.data) for b in bufs]
        if null is not None:
            ptrs[null] = None
        if mis is not None:
            ptrs[mis] = ctypes.c_void_p(bufs[mis].ctypes.data + 4)
        before = eng.launch_count
        rc = lib.sb200_verify_keyset_bytes(eng._h, ks._h if ks_h is None else ks_h, n_, flags, *ptrs)
        return rc, eng.launch_count - before, [b[:-4].copy() for b in bufs[3:]]

    rc, launched, ref = vcall()
    assert (rc, launched) == (OK, 2)
    initial = [np.full((n + 31) // 32, SENTINEL, np.uint32)] * 2
    cases = {"flag AFFINE": dict(flags=1), "flag CHECK_POINTS": dict(flags=8), "flag 64": dict(flags=64), "n = -1": dict(n_=-1)}
    for k in range(5):
        cases[f"null {k}"] = dict(null=k)
        cases[f"misaligned {k}"] = dict(mis=k)
    for label, kw in cases.items():
        rc, launched, outs = vcall(**kw)
        if label in ("null 4", "misaligned 3"):  # invalid is optional; the verdict bitmap is written by words, as in sb200_verify
            assert (rc, launched) == (OK, 2), label
            continue
        assert (rc, launched) == (ARG, 0), label
        assert all((x == y).all() for x, y in zip(outs, initial)), label
    rc, launched, outs = vcall(n_=0)
    assert (rc, launched) == (OK, 0) and all((x == y).all() for x, y in zip(outs, initial))
    assert lib.sb200_verify_keyset_bytes(engine._h, None, n, 0, *[None] * 5) == ARG
    other = Engine([0], ark=o.ARK_RULE)
    try:
        ks2 = other.keyset_from_bytes(scheme, pkb)
        rc, launched, outs = vcall(ks_h=ks2._h)
        assert (rc, launched) == (ARG, 0) and all((x == y).all() for x, y in zip(outs, initial))
        rc, _, outs2 = vcall(ks_h=ks2._h, eng=other)
        assert rc == OK and all((x == y).all() for x, y in zip(outs2, ref))
        ks2.close()
    finally:
        other.close()

    # sb200_keyset_create_bytes
    pb = _aligned(pkb.view(np.uint32))

    def create(sch=scheme, nk=K, flags=0, null=False, mis=False):
        h = ctypes.c_void_p(1)
        ok = _aligned(np.full((nk + 31) // 32 if 0 < nk < 1 << 20 else 1, SENTINEL))
        ptr = None if null else ctypes.c_void_p(pb.ctypes.data + (4 if mis else 0))
        before = engine.launch_count
        rc = lib.sb200_keyset_create_bytes(engine._h, sch, nk, flags, ptr, ok.ctypes.data, ctypes.byref(h))
        launched = engine.launch_count - before
        if rc == OK:
            lib.sb200_keyset_destroy(h)
        else:
            assert not h.value and (ok[:-4] == SENTINEL).all()
        return rc, launched

    assert create() == (OK, 2)  # decode + one build launch
    for label, kw in [("n_keys = 0", dict(nk=0)), ("n_keys = -1", dict(nk=-1)), ("n_keys = 2^32", dict(nk=1 << 32)),
                      ("scheme 3", dict(sch=3)), ("scheme -1", dict(sch=-1)), ("flag AFFINE", dict(flags=1)),
                      ("flag 64", dict(flags=64)), ("null", dict(null=True)), ("misaligned", dict(mis=True))]:
        assert create(**kw) == (ARG, 0), label
    assert lib.sb200_keyset_create_bytes(None, scheme, K, 0, ctypes.c_void_p(pb.ctypes.data), None, ctypes.byref(ctypes.c_void_p())) == ARG

    # sb200_keyset_update / _update_bytes / _revoke
    nt = 1 if scheme == 0 else 2
    pk = _aligned(keys.pk[:8])
    pk2 = _aligned(keys.pk2[:8]) if nt == 2 else None

    def state():
        okb, inv = ks.verify_bytes(t[0], sig, msg)
        return okb, inv, ks.key_ok.copy()

    s0 = state()

    def upd(kind, m=4, flags=None, slots=None, null=None, mis=None, h=None):
        s = _aligned(np.arange(m) if slots is None else slots)
        okw = _aligned(np.full(2, SENTINEL))
        fl = (1 if kind == "update" else 0) if flags is None else flags
        ptrs = {"slots": ctypes.c_void_p(s.ctypes.data)}
        if kind == "update":
            ptrs["pk"] = ctypes.c_void_p(pk.ctypes.data)
            ptrs["pk2"] = ctypes.c_void_p(pk2.ctypes.data) if pk2 is not None else None
        elif kind == "update_bytes":
            ptrs["pkb"] = ctypes.c_void_p(pb.ctypes.data)
        if null is not None:
            ptrs[null] = None
        if mis is not None:
            ptrs[mis] = ctypes.c_void_p(ptrs[mis].value + 4)
        hh = ks._h if h is None else h
        before = engine.launch_count
        if kind == "update":
            rc = lib.sb200_keyset_update(hh, m, fl, ptrs["slots"], ptrs["pk"], ptrs["pk2"], okw.ctypes.data)
        elif kind == "update_bytes":
            rc = lib.sb200_keyset_update_bytes(hh, m, fl, ptrs["slots"], ptrs["pkb"], okw.ctypes.data)
        else:
            rc = lib.sb200_keyset_revoke(hh, m, ptrs["slots"])
        return rc, engine.launch_count - before, okw[:2]

    dead = engine.keyset_from_bytes(scheme, pkb)
    dead_h = dead._h
    dead.close()
    for kind in ("update", "update_bytes", "revoke"):
        cases = {"null keyset": dict(h=ctypes.c_void_p(0)), "destroyed keyset": dict(h=dead_h), "m = -1": dict(m=-1),
                 "slot >= n_keys": dict(slots=[0, 1, K, 3]), "slot 2^32-1": dict(slots=[0, 1, 2, 0xFFFFFFFF]),
                 "duplicate slots": dict(slots=[5, 1, 2, 5]), "null slots": dict(null="slots"), "misaligned slots": dict(mis="slots")}
        if kind != "revoke":
            cases.update({"flag CHECK_POINTS": dict(flags=8), "flag 64": dict(flags=64), "flag 16": dict(flags=16)})
        if kind == "update":
            cases.update({"null pk": dict(null="pk"), "misaligned pk": dict(mis="pk")})
            if nt == 2:
                cases.update({"null pk2": dict(null="pk2"), "misaligned pk2": dict(mis="pk2")})
        if kind == "update_bytes":
            cases.update({"flag AFFINE": dict(flags=1), "null bytes": dict(null="pkb"), "misaligned bytes": dict(mis="pkb")})
        for label, kw in cases.items():
            rc, launched, okw = upd(kind, **kw)
            assert (rc, launched) == (ARG, 0), (kind, label)
            assert (okw == SENTINEL).all(), (kind, label)
        rc, launched, okw = upd(kind, m=0)
        assert (rc, launched) == (OK, 0) and (okw == SENTINEL).all(), kind
        s = state()
        assert all((x == y).all() for x, y in zip(s, s0)), kind  # nothing changed
    # valid calls: launches and key_ok words
    rc, launched, okw = upd("update")
    assert (rc, launched, okw[0], okw[1]) == (OK, 1, 0xF, SENTINEL)  # ceil(m/32) words written
    rc, launched, okw = upd("update_bytes", m=5)
    assert (rc, launched, okw[0], okw[1]) == (OK, 2, 0x1F, SENTINEL)
    rc, launched, _ = upd("revoke", m=3)
    assert (rc, launched) == (OK, 1)
    ks.close()
    # more slots than one build launch takes (2048): two launches
    big = plain_keys(engine, 0, 2100, 630)
    with engine.keyset(0, np.zeros_like(big.pk)) as kb:  # (0, 0): every key malformed
        assert not kb.key_ok.any()
        slots = np.arange(2049, dtype=np.uint32)[::-1].copy()
        before = engine.launch_count
        okn = kb.update(slots, big.pk[slots])
        assert engine.launch_count - before == 2 and okn.all() and kb.key_ok.sum() == 2049
        bb = key_bytes(engine, big.pk[:2052], None)
        before = engine.launch_count
        okn = kb.update_bytes(np.arange(2052, dtype=np.uint32), bb)
        assert engine.launch_count - before == 3 and okn.all() and kb.key_ok.sum() == 2052


# ---- 8. typed API ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_typed_public_key_set_bytes_replace_remove(engine, scheme):
    from schnorr_b200 import api
    prev = api._engine
    api.set_engine(engine)
    try:
        rng = api.StdRng.seed_from_u64(4321 + scheme)
        n_keys, n = 12, 200
        if scheme == 0:
            sks = [api.SecretKey.random(rng) for _ in range(2 * n_keys)]
            allk = api.PublicKey.from_secret_keys(sks)
        elif scheme == 1:
            sks = [api.SecretKey.random(rng) for _ in range(2 * n_keys)]
            allk = [api.PublicKeyDouble.from_secret_key(k) for k in sks]
        else:
            sks = [api.SecretKeyVarGen.random(rng) for _ in range(2 * n_keys)]
            allk = [api.PublicKeyVarGen.from_secret_key(k) for k in sks]
        keys, spare = allk[:n_keys], allk[n_keys:]
        rs = np.random.RandomState(700 + scheme)
        idx = rs.randint(0, n_keys, size=n)
        msgs = [int(x) for x in rs.randint(0, 1 << 62, size=n, dtype=np.int64)]
        swap = [1, 4, 7]
        chosen = [sks[n_keys + i] if (i in swap and k % 2) else sks[i] for k, i in enumerate(idx)]  # odd tuples of swapped slots: the new key signs
        if scheme == 0:
            sigs = api.SecretKey.sign_batch(chosen, rng, msgs)
        elif scheme == 1:
            sigs = api.SecretKey.sign_double_batch(chosen, rng, msgs)
        else:
            sigs = api.SecretKeyVarGen.sign_batch(chosen, rng, msgs)
        msgs = [mm + (k % 5 == 0) for k, mm in enumerate(msgs)]
        sb = [s.to_bytes() for s in sigs]
        mb = [mm.to_bytes(32, "little") for mm in msgs]
        sb[3] = sb[3][:32] + (api.Q).to_bytes(32, "little") + sb[3][64:]  # R does not decode
        mb[5] = (api.Q + 1).to_bytes(32, "little")                           # msg >= q
        with api.PublicKeySet(keys) as ks:
            ok, inv = ks.verify_batch_bytes(idx, sb, mb)
            want = type(keys[0]).verify_batch([keys[i] for i in idx], sigs, msgs)
            assert list(np.nonzero(inv)[0]) == [3, 5]
            want[[3, 5]] = False
            assert (ok == want).all() and ok.any() and not ok.all()
            ks.replace(swap, [spare[i] for i in swap])
            cur = [ks.keys[i] for i in idx]
            want2 = type(keys[0]).verify_batch(cur, sigs, msgs)
            assert (ks.verify_batch(idx, sigs, msgs) == want2).all()
            assert (ks.verify_batch_bytes(idx, sb, mb)[0] == (want2 & ~inv)).all()
            hit = np.isin(idx, swap)
            assert want2[hit & (np.arange(n) % 2 == 1) & (np.arange(n) % 5 != 0)].all()
            assert not want2[hit & (np.arange(n) % 2 == 0)].any()
            ks.remove([0, 7])
            gone = np.isin(idx, [0, 7])
            got = ks.verify_batch(idx, sigs, msgs)
            assert not got[gone].any() and (got[~gone] == want2[~gone]).all()
            assert not ks.verify_batch_bytes(idx, sb, mb)[0][gone].any()
            with pytest.raises(IndexError):
                ks.remove([n_keys])
            # the oracle on a small batch: tuples of the replaced slots against the new keys
            for k in np.nonzero(hit)[0][:6]:
                key = ks.keys[idx[k]]
                s = sigs[k]
                if scheme == 0:
                    exp = o.verify(key._p.affine(), s._u, s._R.affine(), msgs[k], mul=V.mul)
                elif scheme == 1:
                    exp = o.verify_double(key._p.affine(), key._pp.affine(), s._u, s._R.affine(), s._Rp.affine(), msgs[k], mul=V.mul)
                else:
                    exp = o.verify_vargen(key._p.affine(), key._g.affine(), s._u, s._R.affine(), msgs[k], mul=V.mul)
                assert exp == bool(want2[k]) and bool(got[k]) == (exp and idx[k] not in (0, 7))
    finally:
        api.set_engine(prev)
