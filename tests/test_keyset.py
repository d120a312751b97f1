"""Verification against registered keys (include/schnorr_b200_keyset.h, core.cuh keyset_build_window / verify_keyset_core).

A keyset gives every point of every key an 8-bit comb (entry e of window j = e 2^(8j) P), and a verification is then the
challenge hash, the comb of G (or of the key's generator) and the key's comb.  The CPU tests run the host build against
the Python oracle: the table entries, and the verdicts and challenges of all three schemes under both round-constant
rules.  The GPU tests pin the verdicts and challenges against sb200_verify* on the gathered keys over batches above four
waves, the key_ok bitmap, isolation of malformed keys, the return codes and launches, the lifetime rules and the typed
PublicKeySet.
"""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import hostlib as H
import schnorr_oracle as o
import vectors as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R
KS_WINDOWS, KS_ENTRIES = 32, 129
KS_TABLE_WORDS = KS_WINDOWS * KS_ENTRIES * 24
OK, ARG, NOMEM = 0, -1, -4


# ---- CPU: host build --------------------------------------------------------------------------------------------------
def _host_lib():
    so = os.path.join(ROOT, "build", "host_keyset.so")
    srcs = [os.path.join(ROOT, "tests", f) for f in ("host_keyset.cpp", "host_arith.cpp", "host_shim.h")]
    csrc = os.path.join(ROOT, "schnorr_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in srcs):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-include", os.path.join(ROOT, "tests", "host_shim.h"),
                               "-o", so, os.path.join(ROOT, "tests", "host_keyset.cpp")])
    lib = ctypes.CDLL(so)
    lib.h_verify_keyset.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_uint32] + \
        [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
    return lib


@pytest.fixture(scope="module")
def hlib():
    return _host_lib()


@pytest.fixture(scope="module")
def htabs(hlib):
    return H.comb_tables(hlib)


def host_table(hlib, p, z=None):
    t = np.zeros(KS_TABLE_WORDS, np.uint32)
    hlib.h_keyset_table(H.ptr(H.pt_mont(p, z)), int(z is None), H.ptr(t))
    return t


def niels(p):
    """affine Niels form (v + u, v - u, 2 d u v) as Montgomery limbs"""
    u, v = p
    return np.concatenate([H.mont((v + u) % Q), H.mont((v - u) % Q), H.mont(2 * o.D * u * v % Q)])


def test_host_table_entries_match_oracle(hlib):
    rnd = random.Random(11)
    tors = V.torsion_points()
    order = lambda t: next(k for k in (1, 2, 4, 8) if V.mul(t, k) == o.IDENTITY)
    keys = [("random", V.mul(o.G, rnd.randrange(1, R))), ("random + 8-torsion", o.pt_add(V.mul(o.G, rnd.randrange(1, R)),
                                                                                          next(t for t in tors if order(t) == 8)))]
    keys += [(f"order {k}", next(t for t in tors if order(t) == k)) for k in (2, 4, 8)] + [("identity", o.IDENTITY)]
    for label, P in keys:
        for z in (None, rnd.randrange(2, Q)):  # affine and projective input: the same table
            t = host_table(hlib, P, z).reshape(KS_WINDOWS, KS_ENTRIES, 24)
            for j in range(KS_WINDOWS):
                for e in sorted({0, 1, 2, 3, 127, 128, rnd.randrange(4, 127)}):
                    want = niels(V.mul(P, e << (8 * j)) if e else o.IDENTITY)
                    assert (t[j, e] == want).all(), (label, z is not None, j, e)


def _signed(scheme, rnd):
    sk, nonce, m = rnd.randrange(1, R), rnd.randrange(1, R), rnd.randrange(Q)
    if scheme == 0:
        u, Rr, _ = o.sign(sk, nonce, m, mul=V.mul)
        return sk, nonce, dict(pk=V.mul(o.G, sk), pk2=None, u=u, Rr=Rr, Rp=None, m=m)
    if scheme == 1:
        u, Rr, Rp, _ = o.sign_double(sk, nonce, m, mul=V.mul)
        return sk, nonce, dict(pk=V.mul(o.G, sk), pk2=V.mul(o.G_NUMS, sk), u=u, Rr=Rr, Rp=Rp, m=m)
    gen = V.mul(o.G, rnd.randrange(1, R))
    u, Rr, _ = o.sign_vargen(sk, gen, nonce, m, mul=V.mul)
    return sk, nonce, dict(pk=V.mul(gen, sk), pk2=gen, u=u, Rr=Rr, Rp=None, m=m)


CASES = ["valid", "valid2", "u+1", "m+1", "R+B", "wrong key", "u=0", "u=r-1", "u=r", "u=2^256-1", "torsion key", "torsion R",
         "small-order key", "identity key", "whole-curve generator"]


def _host_cases(scheme, rnd):
    tors = V.torsion_points()
    out = []
    for label in CASES:
        sk, nonce, t = _signed(scheme, rnd)
        B = o.G if scheme != 2 else t["pk2"]
        if label == "u+1":
            t["u"] = (t["u"] + 1) % R
        elif label == "m+1":
            t["m"] = (t["m"] + 1) % Q
        elif label == "R+B":
            t["Rr"] = o.pt_add(t["Rr"], B)
        elif label == "wrong key":
            t["wrong"] = True
        elif label == "u=0":
            t["u"] = 0
        elif label == "u=r-1":
            t["u"] = R - 1
        elif label == "u=r":
            t["u"] = R
        elif label == "u=2^256-1":
            t["u"] = (1 << 256) - 1
        elif label == "torsion key":  # valid iff c T = O
            T = tors[rnd.randrange(1, len(tors))]
            t["pk"] = o.pt_add(t["pk"], T)
            if scheme == 1:
                t["pk2"] = o.pt_add(t["pk2"], T)
        elif label == "torsion R":
            t["Rr"] = o.pt_add(t["Rr"], tors[rnd.randrange(1, len(tors))])
        elif label in ("small-order key", "identity key"):  # R = u B: valid iff c PK = O
            T = tors[rnd.randrange(1, len(tors))] if label == "small-order key" else o.IDENTITY
            t["pk"], t["u"] = T, nonce
            if scheme == 1:
                t["pk2"] = T
        elif label == "whole-curve generator" and scheme == 2:  # GEN = G' + T: u GEN + c PK = R exactly as the oracle says
            gen = o.pt_add(V.mul(o.G, rnd.randrange(1, R)), tors[rnd.randrange(1, len(tors))])
            u, Rr, _ = o.sign_vargen(sk, gen, nonce, t["m"], mul=V.mul)
            t.update(pk=V.mul(gen, sk), pk2=gen, u=u, Rr=Rr)
        out.append((label, t))
    return out


def _oracle(scheme, t, pk, pk2):
    """(verdict, c) of the oracle's verify on the tuple with the key (pk, pk2)"""
    if scheme == 1:
        c = o.challenge_hash_double(t["Rr"], t["Rp"], t["m"])
    else:
        c = o.challenge_hash(t["Rr"], t["m"])
    if t["u"] >= R:
        return False, c
    f = (lambda: o.verify(pk, t["u"], t["Rr"], t["m"], mul=V.mul), lambda: o.verify_double(pk, pk2, t["u"], t["Rr"], t["Rp"], t["m"], mul=V.mul),
         lambda: o.verify_vargen(pk, pk2, t["u"], t["Rr"], t["m"], mul=V.mul))[scheme]
    return f(), c


def _host_verify(hlib, htabs, scheme, tabs, n_keys, key_ok, key, t, zs=None, check=0):
    enc = lambda p, k: (H.pt_mont(p) if zs is None else H.pt_mont(p, zs[k])) if p is not None else np.zeros(24, np.uint32)
    c = np.zeros(8, np.uint32)
    u = np.frombuffer(int(t["u"]).to_bytes(32, "little"), np.uint32).copy()
    ok = hlib.h_verify_keyset(scheme, H.ptr(tabs), n_keys, H.ptr(key_ok), key, H.ptr(u), H.ptr(enc(t["Rr"], 0)), H.ptr(enc(t["Rp"], 1)),
                              H.ptr(H.mont(t["m"])), int(zs is None), check, H.ptr(htabs[0]), H.ptr(htabs[1]), H.ptr(c))
    return bool(ok), H.to_int(c)


@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_host_verdicts_and_challenges_match_oracle(hlib, htabs, ark, scheme):
    H.setup_hades(hlib)  # the host build's Hades tables under the rule the `ark` fixture selected
    rnd = random.Random(300 + 10 * scheme + (ark == "plain"))
    cases = _host_cases(scheme, rnd)
    keys = [(t["pk"], t["pk2"]) for _, t in cases]
    nt = 1 if scheme == 0 else 2
    tabs = np.concatenate([host_table(hlib, p) for k in keys for p in k[:nt]])
    n = len(keys)
    key_ok = np.full((n + 31) // 32, 0xFFFFFFFF, np.uint32)
    seen = set()
    for i, (label, t) in enumerate(cases):
        key = (i + 1) % n if t.get("wrong") else i
        want = _oracle(scheme, t, *keys[key])
        got = _host_verify(hlib, htabs, scheme, tabs, n, key_ok, key, t)
        assert got == want, label
        seen.add(got[0])
        if label.startswith("valid"):
            assert got[0], label
        zs = [rnd.randrange(2, Q) for _ in range(2)]  # projective R (R')
        assert _host_verify(hlib, htabs, scheme, tabs, n, key_ok, key, t, zs=zs) == want, label
        assert _host_verify(hlib, htabs, scheme, tabs, n, key_ok, key, t, check=1) == want, label
        # an index past the keyset and a key recorded as malformed: verdict 0, the same challenge
        for k, okw in ((n, key_ok), (2**32 - 1, key_ok), (key, np.zeros_like(key_ok))):
            assert _host_verify(hlib, htabs, scheme, tabs, n, okw, k, t) == (False, want[1]), (label, k)
    assert seen == {True, False}


def test_host_check_points_rejects_malformed_R(hlib, htabs):
    H.setup_hades(hlib)
    rnd = random.Random(5)
    for scheme in range(3):
        _, _, t = _signed(scheme, rnd)
        tabs = np.concatenate([host_table(hlib, p) for p in (t["pk"], t["pk2"])[:1 if scheme == 0 else 2]])
        key_ok = np.ones(1, np.uint32)
        assert _host_verify(hlib, htabs, scheme, tabs, 1, key_ok, 0, t, check=1)[0]
        bad = dict(t, Rr=(t["Rr"][0], (t["Rr"][1] + 1) % Q))
        assert not _host_verify(hlib, htabs, scheme, tabs, 1, key_ok, 0, bad, check=1)[0]


def test_header_declares_exactly_the_bound_symbols():
    import re
    lib_path = os.path.join(ROOT, "schnorr_b200", "libschnorr_b200.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    from schnorr_b200 import _lib
    decl = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "schnorr_b200_keyset.h")).read())))
    assert decl == sorted(_lib._KEYSET_PROTOTYPES) == ["sb200_keyset_create", "sb200_keyset_destroy", "sb200_verify_keyset"]
    assert not set(_lib._KEYSET_PROTOTYPES) & set(_lib.EXPORTED_SYMBOLS)
    assert all(hasattr(ctypes.CDLL(lib_path), s) for s in decl)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _sp():
    import test_gpu_scale_parity as SP
    return SP


from test_gpu_scale_parity import sizes  # noqa: E402,F401


def _rand_scalars(rs, n, bits=251):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << (bits - 224)) - 1
    return a


class Keys:
    pass


KEY_KINDS = ["plain"] * 6 + ["torsion", "small-order", "identity", "off-curve"]


def make_keys(eng, scheme, K, seed):
    """K keys: prime-order keys, keys + torsion, small-order and identity keys, and keys with a point off the curve;
    sk per key (the secret the signatures below use)"""
    SP = _sp()
    rs, rnd = np.random.RandomState(seed), random.Random(seed)
    k = Keys()
    k.sk = _rand_scalars(rs, K)
    k.kind = np.array([KEY_KINDS[i % len(KEY_KINDS)] for i in rnd.sample(range(10 * K), K)])
    tors = V.torsion_points()
    if scheme == 0:
        pk, pk2 = eng.keygen(k.sk), None
    elif scheme == 1:
        pk, pk2 = eng.keygen_double(k.sk)
    else:
        pk2 = eng.keygen(_rand_scalars(rs, K))  # generators: prime order, every fourth with a torsion component
        wc = np.arange(0, K, 4)
        pk2[wc] = SP._add_points(pk2[wc], [tors[1 + i % 7] for i in wc])
        pk = eng.keygen_vargen(k.sk, pk2)
    for name, f in (("torsion", lambda rows, i: SP._add_points(rows, [tors[1 + j % 7] for j in i])),
                    ("small-order", lambda rows, i: V.points([tors[1 + j % 7] for j in i])),
                    ("identity", lambda rows, i: V.points([o.IDENTITY] * len(i)))):
        i = np.nonzero(k.kind == name)[0]
        pk[i] = f(pk[i], i)
        if scheme == 1 and name != "torsion":
            pk2[i] = pk[i]
    off = np.nonzero(k.kind == "off-curve")[0]  # v + 1: off the curve (the first point, or the second one for odd keys)
    tgt = [pk if (scheme == 0 or i % 2 == 0) else pk2 for i in off]
    for a, i in zip(tgt, off):
        a[i, 8:16] = SP.from_ints([(SP.to_ints(a[i, 8:16])[0] + 1) % Q])[0]
    k.pk, k.pk2, k.K = pk, pk2, K
    return k


def make_tuples(eng, scheme, keys, N, seed):
    """N tuples signed by keys[idx] and the corruption categories of test_gpu_scale_parity: u+1, u+r, m+1, R+B, a
    neighbour's key index; plus indices past the keyset.  Returns (idx, u, R, R' or None, m, category)."""
    SP = _sp()
    rs = np.random.RandomState(seed)
    K = keys.K
    idx = rs.randint(0, K, size=N).astype(np.uint32)
    nonce, m = _rand_scalars(rs, N), _rand_scalars(rs, N, 254)
    Rp = None
    if scheme == 0:
        u, Rr, _ = eng.sign(keys.sk[idx], m, nonce)
    elif scheme == 1:
        u, Rr, Rp, _ = eng.sign_double(keys.sk[idx], m, nonce)
    else:
        u, Rr, _ = eng.sign_vargen(keys.sk[idx], keys.pk2[idx], m, nonce)
    so = np.nonzero(np.isin(keys.kind[idx], ["small-order", "identity"]))[0]
    u[so] = nonce[so]  # R = nonce B: valid iff c PK = O
    cat = rs.randint(0, 10, size=N)  # 0-3 untouched, 4 u+1, 5 u+r, 6 m+1, 7 R+B, 8 neighbour key, 9 index past the keyset
    i = np.nonzero(cat == 4)[0]
    u[i] = SP.from_ints([(x + 1) % R for x in SP.to_ints(u[i])])
    i = np.nonzero(cat == 5)[0]
    u[i] = SP.from_ints([x + R for x in SP.to_ints(u[i])])
    i = np.nonzero(cat == 6)[0]
    m[i] = SP.from_ints([x + 1 for x in SP.to_ints(m[i])])
    i = np.nonzero(cat == 7)[0]
    B = [o.G] * len(i) if scheme != 2 else [SP.aff(g) for g in keys.pk2[idx[i]]]
    Rr[i] = SP._add_points(Rr[i], B)
    i = np.nonzero(cat == 8)[0]
    idx[i] = (idx[i] + 1) % K
    i = np.nonzero(cat == 9)[0]
    idx[i] = K + rs.randint(0, 1 << 20, size=len(i)).astype(np.uint32)
    idx[i[::7]] = 0xFFFFFFFF
    return idx, u, Rr, Rp, m, cat


def reference(eng, scheme, keys, t, key_ok, **kw):
    """sb200_verify* on the gathered keys: (expected verdicts, challenges)"""
    idx, u, Rr, Rp, m, _ = t
    g = np.minimum(idx, keys.K - 1)
    known = idx < keys.K
    if scheme == 0:
        ok, c = eng.verify(keys.pk[g], u, Rr, m, **kw)
    elif scheme == 1:
        ok, c = eng.verify_double(keys.pk[g], keys.pk2[g], u, Rr, Rp, m, **kw)
    else:
        ok, c = eng.verify_vargen(keys.pk[g], keys.pk2[g], u, Rr, m, **kw)
    return ok & known & key_ok[g], c


def _ks_verify(ks, t, **kw):
    idx, u, Rr, Rp, m, _ = t
    return ks.verify(idx, u, Rr, m, Rp=Rp, **kw)


_KB = {}


@pytest.fixture
def kbatches(engine, sizes):
    """300 keys and a batch above four waves per scheme (built once per module)"""
    if "b" not in _KB:
        out = []
        for scheme in range(3):
            keys = make_keys(engine, scheme, 300, 40 + scheme)
            out.append((keys, make_tuples(engine, scheme, keys, sizes[1], 50 + scheme)))
        _KB["b"] = out
    return _KB["b"]


def _assert_ok(ok, want, c=None, c_want=None):
    bad = np.nonzero(ok != want)[0]
    assert len(bad) == 0, f"{len(bad)} verdicts differ, first at {bad[:8].tolist()}"
    if c is not None:
        diff = np.nonzero((c != c_want).any(axis=1))[0]
        assert len(diff) == 0, f"{len(diff)} challenge rows differ, first at {diff[:8].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_parity_with_verify_on_gathered_keys(engine, kbatches, sizes, scheme):
    """host buffers over several chunks (one launch each) and in one chunk, and device pointers; key_ok equals
    sb200_points_check on the keys"""
    import torch
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE
    SP = _sp()
    keys, t = kbatches[scheme]
    N = sizes[1]
    assert N > 4 * sizes[0]
    with engine.keyset(scheme, keys.pk, keys.pk2) as ks:
        chk = engine.points_check(keys.pk) & (engine.points_check(keys.pk2) if scheme else True)
        assert (ks.key_ok == chk).all() and (~chk).any() and (keys.kind != "off-curve").sum() == chk.sum()
        want, c_want = reference(engine, scheme, keys, t, ks.key_ok)
        assert 0.15 < want.mean() < 0.6, want.mean()
        for kind in ("torsion", "small-order", "identity"):  # valid iff c T = O: mixed, and always for the identity
            sel = (keys.kind[np.minimum(t[0], keys.K - 1)] == kind) & (t[5] < 4) & (t[0] < keys.K)
            assert want[sel].any() and (want[sel].all() == (kind == "identity")), kind
        chunks = SP.host_chunks(N)
        assert len(chunks) > 1
        before = engine.launch_count
        ok, c = _ks_verify(ks, t)
        assert engine.launch_count - before == len(chunks)
        _assert_ok(ok, want, c, c_want)
        assert not ok[t[0] >= keys.K].any() and not ok[t[5] == 5].any()
        # one chunk, ragged
        n1 = 2000 + 13
        t1 = tuple(x[:n1] if x is not None else None for x in t)
        before = engine.launch_count
        ok1, c1 = _ks_verify(ks, t1)
        assert engine.launch_count - before == 1
        _assert_ok(ok1, want[:n1], c1, c_want[:n1])
        # device pointers, one launch
        dev = torch.device("cuda:0")
        td = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev) if a is not None else None
        idx, u, Rr, Rp, m, _ = t
        ins = [td(idx), td(u), td(Rr), td(Rp), td(m)]
        bm = torch.zeros((N + 31) // 32, dtype=torch.int32, device=dev)
        cd = torch.zeros((N, 8), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        before = engine.launch_count
        rc = engine._lib.sb200_verify_keyset(engine._h, ks._h, N, POINTS_AFFINE | DEVICE_PTRS,
                                             *[ctypes.c_void_p(x.data_ptr()) if x is not None else None for x in ins],
                                             ctypes.c_void_p(bm.data_ptr()), ctypes.c_void_p(cd.data_ptr()))
        torch.cuda.synchronize()
        assert rc == 0 and engine.launch_count - before == 1
        okd = np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool)
        _assert_ok(okd, want, cd.cpu().numpy().view(np.uint32), c_want)


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_projective_keys_and_check_points(engine, kbatches, scheme):
    """a keyset built from projective keys (some with Z = 0: malformed), projective R; then SB200_CHECK_POINTS with R
    off the curve or Z = 0 scattered: verdict 0 there, sb200_verify's everywhere else"""
    SP = _sp()
    keys, t = kbatches[scheme]
    rs = np.random.RandomState(60 + scheme)
    zk = [int(z) for z in rs.randint(2, 1 << 62, size=keys.K, dtype=np.int64)]
    pk, pk2 = SP.projective(keys.pk, zk), (SP.projective(keys.pk2, zk) if keys.pk2 is not None else None)
    zero = np.nonzero(keys.kind == "plain")[0][::9]
    pk[zero, 16:] = 0
    N = len(t[0])
    zs = [int(z) for z in rs.randint(2, 1 << 62, size=N, dtype=np.int64)]
    idx, u, Rr, Rp, m, cat = t
    tp = (idx, u, SP.projective(Rr, zs), SP.projective(Rp, zs) if Rp is not None else None, m, cat)
    with engine.keyset(scheme, pk, pk2, affine=False) as ks:
        assert not ks.key_ok[zero].any() and (ks.key_ok == engine.points_check(pk, affine=False) &
                                              (engine.points_check(pk2, affine=False) if scheme else True)).all()
        g = np.minimum(idx, keys.K - 1)
        want, c_want = reference(engine, scheme, keys, t, ks.key_ok)
        ok, c = _ks_verify(ks, tp, affine=False)
        _assert_ok(ok, want, c, c_want)
        assert not ok[np.isin(g, zero) & (idx < keys.K)].any()
        # SB200_CHECK_POINTS
        bad = np.zeros(N, bool)
        for k in ((2, 3) if scheme == 1 else (2,)):
            sel = rs.randint(0, 64, size=N)
            z0, off = np.nonzero(sel == 0)[0], np.nonzero(sel == 1)[0]
            tp[k][z0, 16:] = 0
            tp[k][off, 8:16] = SP.from_ints([(v + 1) % Q for v in SP.to_ints(tp[k][off, 8:16])])
            bad[z0] = bad[off] = True
        ok, _ = _ks_verify(ks, tp, affine=False, check_points=True)
        _assert_ok(ok[~bad], want[~bad])
        assert not ok[bad].any() and (want & bad).any()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_malformed_keys_do_not_touch_other_keys(engine, kbatches, scheme):
    keys, t = kbatches[scheme]
    clean_pk, clean_pk2 = keys.pk.copy(), (keys.pk2.copy() if keys.pk2 is not None else None)
    off = np.nonzero(keys.kind == "off-curve")[0]
    g0 = np.nonzero(keys.kind == "plain")[0][0]  # a well-formed key in their place
    clean_pk[off] = keys.pk[g0]
    if clean_pk2 is not None:
        clean_pk2[off] = keys.pk2[g0]
    with engine.keyset(scheme, keys.pk, keys.pk2) as a, engine.keyset(scheme, clean_pk, clean_pk2) as b:
        assert b.key_ok.all() and not a.key_ok[off].any()
        oka, ca = _ks_verify(a, t)
        okb, cb = _ks_verify(b, t)
        good = (t[0] < keys.K) & a.key_ok[np.minimum(t[0], keys.K - 1)]
        assert (oka[good] == okb[good]).all() and not oka[~good].any() and (ca == cb).all()


@pytest.mark.gpu
def test_multi_device_context(engine, kbatches):
    """a context over several devices (device 0 twice on a one-GPU box) keeps a copy per device and gives the verdicts
    and challenges of one device; SB200_DEVICE_PTRS on it is rejected at creation"""
    import torch
    from schnorr_b200 import Engine, SchnorrB200Error
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for scheme, (keys, t) in enumerate(kbatches):
            with engine.keyset(scheme, keys.pk, keys.pk2) as ks1, eng.keyset(scheme, keys.pk, keys.pk2) as ks2:
                ok1, c1 = _ks_verify(ks1, t)
                ok2, c2 = _ks_verify(ks2, t)
                assert (ok1 == ok2).all() and (c1 == c2).all() and (ks1.key_ok == ks2.key_ok).all(), scheme
        h = ctypes.c_void_p()
        pk = kbatches[0][0].pk
        d = torch.from_numpy(pk.view(np.int32)).cuda()
        assert eng._lib.sb200_keyset_create(eng._h, 0, len(pk), 3, ctypes.c_void_p(d.data_ptr()), None, None, ctypes.byref(h)) == ARG
        assert not h.value
    finally:
        eng.close()
    with pytest.raises(SchnorrB200Error):
        engine.keyset(0, np.zeros((0, 16), np.uint32))


SENTINEL = 0xA5A5A5A5


@pytest.fixture
def small(engine):
    """a 10-key keyset of each scheme (prime-order keys) and 70 tuples per scheme (ragged warp, one chunk)"""
    out = []
    for scheme in range(3):
        rs = np.random.RandomState(80 + scheme)
        k = Keys()
        k.K, k.sk, k.kind = 10, _rand_scalars(rs, 10), np.array(["plain"] * 10)
        if scheme == 0:
            k.pk, k.pk2 = engine.keygen(k.sk), None
        elif scheme == 1:
            k.pk, k.pk2 = engine.keygen_double(k.sk)
        else:
            k.pk2 = engine.keygen(_rand_scalars(rs, 10))
            k.pk = engine.keygen_vargen(k.sk, k.pk2)
        t = make_tuples(engine, scheme, k, 70, 90 + scheme)
        out.append((k, (t[0] % 10,) + t[1:]))
    return out


def _args(scheme, t):
    """the pointer arguments of sb200_verify_keyset after the keyset: key_index, u, R, R', msg, verdicts, c_out"""
    from schnorr_b200 import _lib
    idx, u, Rr, Rp, m, _ = t
    n = len(idx)
    arrs = [idx, u, Rr, Rp if scheme == 1 else None, m, np.full((n + 31) // 32, SENTINEL, np.uint32), np.full((n, 8), SENTINEL, np.uint32)]
    bufs = []
    for a in arrs:
        if a is None:
            bufs.append(None)
            continue
        b = _lib.aligned_empty((a.size + 4,))
        b[:a.size] = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1)
        bufs.append(b)
    return bufs


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_return_codes_write_and_launch_nothing(engine, small, scheme):
    """each rejected call against a valid control: nothing written, nothing launched, the context still repeats the
    valid call bit for bit"""
    from schnorr_b200 import Engine, _lib
    keys, t = small[scheme]
    lib = engine._lib
    n = len(t[0])
    ks = engine.keyset(scheme, keys.pk, keys.pk2)

    def call(ks_h=None, n_=n, flags=1, null=None, mis=None, eng=engine):
        bufs = _args(scheme, t)
        ptrs = [ctypes.c_void_p(b.ctypes.data) if b is not None else None for b in bufs]
        if null is not None:
            ptrs[null] = None
        if mis is not None:
            ptrs[mis] = ctypes.c_void_p(bufs[mis].ctypes.data + 4)
        before = eng.launch_count
        rc = lib.sb200_verify_keyset(eng._h, ks._h if ks_h is None else ks_h, n_, flags, *ptrs)
        return rc, eng.launch_count - before, [b[:-4].copy() for b in bufs[5:]]

    rc, launched, ref = call()
    assert (rc, launched) == (OK, 1)
    initial = [b[:-4].copy() for b in _args(scheme, t)[5:]]
    cases = {"flag 4": dict(flags=1 | 4), "flag 16": dict(flags=1 | 16), "flag 64": dict(flags=1 | 64), "n = -1": dict(n_=-1)}
    for k in range(7):
        if k == 3 and scheme != 1:
            continue  # R' is read for scheme 1 only
        cases[f"null {k}"] = dict(null=k)
        cases[f"misaligned {k}"] = dict(mis=k)
    for label, kw in cases.items():
        rc, launched, outs = call(**kw)
        if label in ("null 6", "misaligned 5"):  # c_out is optional; the verdict bitmap is written by words, as in sb200_verify
            assert (rc, launched) == (OK, 1), label
            continue
        assert (rc, launched) == (ARG, 0), label
        assert all((x == y).all() for x, y in zip(outs, initial)), label
    rc, launched, outs = call(n_=0)
    assert (rc, launched) == (OK, 0) and all((x == y).all() for x, y in zip(outs, initial))
    assert lib.sb200_verify_keyset(engine._h, None, n, 1, *[None] * 7) == ARG
    # a keyset of another context
    other = Engine([0], ark=o.ARK_RULE)
    try:
        ks2 = other.keyset(scheme, keys.pk, keys.pk2)
        rc, launched, outs = call(ks_h=ks2._h)
        assert (rc, launched) == (ARG, 0) and all((x == y).all() for x, y in zip(outs, initial))
        rc, _, outs2 = call(ks_h=ks2._h, eng=other)
        assert rc == OK and all((x == y).all() for x, y in zip(outs2, ref))
        ks2.close()
    finally:
        other.close()
    rc, launched, outs = call()
    assert (rc, launched) == (OK, 1) and all((x == y).all() for x, y in zip(outs, ref))
    ks.close()

    # sb200_keyset_create
    pk = _lib.aligned_empty((keys.pk.size + 4,)); pk[:keys.pk.size] = keys.pk.reshape(-1)
    pk2 = None
    if keys.pk2 is not None:
        pk2 = _lib.aligned_empty((keys.pk2.size + 4,)); pk2[:keys.pk2.size] = keys.pk2.reshape(-1)

    def create(sch=scheme, nk=10, flags=1, p=None, p2=None, nullpk=False, nullpk2=False, mis=False):
        h = ctypes.c_void_p(1)
        ptr = None if nullpk else ctypes.c_void_p((p if p is not None else pk).ctypes.data + (4 if mis else 0))
        ptr2 = None if (nullpk2 or pk2 is None) else ctypes.c_void_p(pk2.ctypes.data)
        before = engine.launch_count
        rc = lib.sb200_keyset_create(engine._h, sch, nk, flags, ptr, ptr2, None, ctypes.byref(h))
        launched = engine.launch_count - before
        if rc == OK:
            lib.sb200_keyset_destroy(h)
        else:
            assert not h.value
        return rc, launched

    assert create() == (OK, 1)
    for label, kw, want in [("n_keys = 0", dict(nk=0), ARG), ("n_keys = -1", dict(nk=-1), ARG), ("n_keys = 2^32", dict(nk=1 << 32), ARG),
                            ("scheme 3", dict(sch=3), ARG), ("scheme -1", dict(sch=-1), ARG), ("flag CHECK_POINTS", dict(flags=1 | 8), ARG),
                            ("flag 64", dict(flags=1 | 64), ARG), ("null pk", dict(nullpk=True), ARG), ("misaligned pk", dict(mis=True), ARG)]:
        assert create(**kw) == (want, 0), label
    if scheme:
        assert create(nullpk2=True) == (ARG, 0)
    import torch
    free0 = torch.cuda.mem_get_info()[0]
    assert create(nk=(1 << 32) - 1) == (NOMEM, 0)  # 1.7 PB of tables
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)  # nothing stays allocated
    assert create() == (OK, 1)
    lib.sb200_keyset_destroy(None)


@pytest.mark.gpu
def test_lifetime(engine, small):
    """destroying a keyset then the context, and the context with live keysets, leave no error; the session's context
    still works"""
    from schnorr_b200 import Engine
    keys, t = small[0]
    e = Engine([0], ark=o.ARK_RULE)
    ks = e.keyset(0, keys.pk)
    ks.close()
    e.close()
    e = Engine([0], ark=o.ARK_RULE)
    kss = [e.keyset(s, k.pk, k.pk2) for s, (k, _) in enumerate(small)]
    e.close()  # frees the three keysets
    for ks in kss:
        ks.close()  # a no-op now: the handles died with the context
    e = engine
    with e.keyset(0, keys.pk) as ks:
        ok, _ = _ks_verify(ks, t)
        want, _ = reference(e, 0, keys, t, ks.key_ok)
        assert (ok == want).all() and ok.any()


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_typed_public_key_set(engine, scheme):
    """PublicKeySet.verify_batch == the type's verify_batch on the gathered keys"""
    from schnorr_b200 import api
    prev = api._engine
    api.set_engine(engine)
    try:
        rng = api.StdRng.seed_from_u64(1234 + scheme)
        tors = [api.JubJubExtended(*p) for p in V.torsion_points()]
        n_keys, n = 12, 200
        if scheme == 0:
            sks = [api.SecretKey.random(rng) for _ in range(n_keys)]
            keys = api.PublicKey.from_secret_keys(sks)
            keys[3] = api.PublicKey.from_raw_unchecked(tors[5])
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
        msgs = [m + (k % 3 == 0) for k, m in enumerate(msgs)]  # a third corrupted
        with api.PublicKeySet(keys) as ks:
            got = ks.verify_batch(idx, sigs, msgs)
            want = type(keys[0]).verify_batch([keys[i] for i in idx], sigs, msgs)
            assert (got == want).all() and got.any() and not got.all()
            with pytest.raises(IndexError):
                ks.verify_batch([n_keys], sigs[:1], msgs[:1])
    finally:
        api.set_engine(prev)
