"""Every reachable entry of every comb table the device builds, and keysets whose tables lie past 2^32 words.

A scalar multiple by a known base is a sum of comb entries, one per window, picked by the signed digits of
recode_offset<W> / recode_digit<W> (ed.cuh).  A wrong entry only shows when a tuple reads it, so these tests choose the
scalars: digit sweeps whose digits, over the batch, run through every (window, digit) that a scalar below its bound can
produce.  The CPU tests restate the recoding and prove that the sweeps cover those sets exactly.  On the GPU:
  - the 16-bit combs of G and G' (k_comb_build) through keygen, keygen_double and dbg_scalar_mul, and the 4-bit combs of
    the oblivious signer (k_comb4_build) through the same keygens with SB200_SIGN_OBLIVIOUS, against ref_cpu, on one
    device and on every device of a multi-device context;
  - the 8-bit per-key combs (k_keyset_build, k_keyset_update) of keysets past one build launch and past 2^32 words of
    tables, read at probe keys on every launch and offset boundary through KeySet.verify_witness and KeySet.verify:
    challenges that cover every reachable digit, and for the variable generator a u sweep, against ref_cpu.
ref_cpu (oracle/ref_cpu.c) is a 256-bit double-and-add ladder that shares no code with the CUDA headers; every
comparison is bit for bit.
"""
import random

import numpy as np
import pytest

import ref_cpu
import schnorr_oracle as o
import vectors as V
from test_gpu_scale_parity import _cu_value, from_ints, rand_scalars, to_ints

Q, R = o.Q, o.R
KS_TABLE_WORDS = 32 * 129 * 24  # words per point of a keyset (ed.cuh KS_TABLE_WORDS)
KS_BUILD_KEYS = _cu_value(r"^constexpr int64_t KS_BUILD_KEYS = ([0-9 <]+);")  # keys per build launch
SCHEMES = dict(argvalues=[0, 1, 2], ids=["single", "double", "vargen"])
WIDTH = (11, 19, 13)


# ---- the recoding, restated ----------------------------------------------------------------------------------------
def offset(W, windows=None):
    """sum of 2^(W-1) 2^(W i) over the first `windows` windows (all 256 / W by default): recode_offset<W>'s addend"""
    return sum(1 << (W * i + W - 1) for i in range(256 // W if windows is None else windows))


def recode(k, W):
    """[n, 256 / W] signed digits of recode_offset<W> then recode_digit<W> for canonical scalar limbs k [n, 8]"""
    k = np.ascontiguousarray(k, np.uint32).reshape(-1, 8)
    add = {4: 0x88888888, 8: 0x80808080, 16: 0x80008000}[W]
    s, carry = np.empty_like(k), np.zeros(len(k), np.uint64)
    for i in range(8):
        t = k[:, i].astype(np.uint64) + add + carry
        s[:, i], carry = (t & 0xFFFFFFFF).astype(np.uint32), t >> 32
    assert not carry.any()  # k < 2^252: no carry out of the top limb
    b = s.view(np.uint8)
    w = s.view(np.uint16) if W == 16 else b if W == 8 else np.stack([b & 15, b >> 4], axis=2).reshape(len(k), 64)
    return w.astype(np.int32) - (1 << (W - 1))


def reachable(W, bound):
    """{(window, digit)} over all scalars 0 <= k < bound: window j of x = k + offset(W) runs over x in one interval, so
    x >> (W j) runs over [lo >> W j, hi >> W j] and the window takes exactly those values mod 2^W"""
    lo, hi, half = offset(W), bound - 1 + offset(W), 1 << (W - 1)
    out = set()
    for j in range(256 // W):
        ylo, yhi = lo >> (W * j), hi >> (W * j)
        vals = range(1 << W) if yhi - ylo + 1 >= 1 << W else {y % (1 << W) for y in range(ylo, yhi + 1)}
        out |= {(j, v - half) for v in vals}
    return out


def covered(digits):
    """{(window, digit)} read by rows of recoded digits"""
    return {(j, d) for j in range(digits.shape[1]) for d in np.unique(digits[:, j]).tolist()}


def sweep(W, bound, delta, seed):
    """Scalars below `bound`: scalar i (0 <= i < 2^W) has digit ((i + j delta) mod 2^W) - 2^(W-1) in window j < n - 1, so
    every such window sees every digit once and the windows of one scalar differ (delta odd); its top digit t is drawn
    from those that keep it in [0, bound).  Then one scalar per top digit that a scalar below `bound` can have.
    Returns (limbs [m, 8], the intended digits [2^W, n] of the first 2^W scalars)."""
    rnd = random.Random(seed)
    n, half, top = 256 // W, 1 << (W - 1), W * (256 // W - 1)
    low_off = offset(W, n - 1)
    ks, want = [], []
    for i in range(1 << W):
        d = [((i + j * delta) % (1 << W)) - half for j in range(n - 1)]
        low = sum(x << (W * j) for j, x in enumerate(d))
        t = rnd.randint(1 if low < 0 else 0, (bound - 1 - low) >> top)
        ks.append((t << top) + low)
        want.append(d + [t])
    for t in range(low_off >> top, ((bound - 1 + low_off) >> top) + 1):  # k + low_off in [t 2^top, (t + 1) 2^top)
        ks.append(rnd.randrange(max(0, (t << top) - low_off), min(bound, ((t + 1) << top) - low_off)))
    assert all(0 <= k < bound for k in ks)
    return from_ints(ks), np.array(want, np.int32)


SWEEPS = {16: (R, 0x9E37), 8: (R, 0x6B), "c": (1 << 250, 0x35)}


def sweep_of(key):
    W = 8 if key == "c" else key
    bound, delta = SWEEPS[key]
    return W, bound, sweep(W, bound, delta, seed=W * 7 + (key == "c"))


# ---- CPU: the sweeps read what they claim --------------------------------------------------------------------------
@pytest.mark.parametrize("key", [16, 8, "c"], ids=["W16 k<r", "W8 u<r", "W8 c<2^250"])
def test_sweep_recodes_to_its_digits_and_covers_the_reachable_set(key):
    W, bound, (k, want) = sweep_of(key)
    d = recode(k, W)
    assert (d[:len(want)] == want).all()
    n = 256 // W
    for j in range(n - 1):  # every digit once per window, and no two windows of one scalar alike
        assert sorted(want[:, j].tolist()) == list(range(-(1 << (W - 1)), 1 << (W - 1)))
    assert all(len(set(r[:n - 1].tolist())) == n - 1 for r in want[:512])
    # value of the digits = the scalar (the recoding is exact)
    ints = to_ints(k)
    for i in range(0, len(ints), 97):
        assert sum(int(x) << (W * j) for j, x in enumerate(d[i])) == ints[i]
    reach = reachable(W, bound)
    assert covered(d) == reach
    # the top window: exactly the digits of [0, bound); every other window: all 2^W digits
    top = sorted(x for j, x in reach if j == n - 1)
    assert top[0] == 0 and top[-1] == (bound - 1 + offset(W, n - 1)) >> (W * (n - 1)) and len(top) == top[-1] + 1
    assert all(sum(1 for jj, _ in reach if jj == j) == 1 << W for j in range(n - 1))
    # nothing outside the set: random scalars below the bound and the bound's neighbours stay inside
    rs = np.random.RandomState(W)
    edge = from_ints([0, 1, bound - 1, bound - 2, (bound - 1) & ~((1 << (W * (n - 1))) - 1)])
    lim = rand_scalars(rs, 20000, bound.bit_length())
    lim = lim[np.array([x < bound for x in to_ints(lim)])]
    assert covered(recode(np.concatenate([lim, edge]), W)) <= reach


def test_comb4_entries_covered_by_the_16_bit_sweep():
    """the scalars of the W = 16 sweep read every entry of the 4-bit combs that a scalar below r can read"""
    _, _, (k, _) = sweep_of(16)
    assert covered(recode(k, 4)) == reachable(4, R)
    assert len(k) % (8 * 128)  # ragged against k_fixed_batch's 8 tuples x 128 threads per CTA


# ---- GPU: generator combs, every entry -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gen_sweep():
    _, _, (k, _) = sweep_of(16)
    return k, ref_cpu.keygen(k, double=True)


def _first_diff(got, want):
    bad = np.nonzero((np.asarray(got) != want).reshape(len(want), -1).any(axis=1))[0]
    return f"{len(bad)} of {len(want)} differ, first at {bad[:8].tolist()}"


@pytest.mark.gpu
def test_generator_combs_every_entry(engine, gen_sweep):
    k, (pk, pkp) = gen_sweep
    for obl in (False, True):
        got = engine.keygen(k, oblivious=obl)
        assert (got == pk).all(), ("keygen", obl, _first_diff(got, pk))
        g0, g1 = engine.keygen_double(k, oblivious=obl)
        assert (g0 == pk).all() and (g1 == pkp).all(), ("keygen_double", obl, _first_diff(g0, pk), _first_diff(g1, pkp))
    for base, want in ((0, pk), (1, pkp)):
        got = engine.dbg_scalar_mul(base, k)
        assert (got == want).all(), ("dbg_scalar_mul", base, _first_diff(got, want))


@pytest.mark.gpu
def test_generator_combs_every_entry_on_every_device(gen_sweep):
    """a context over several devices (device 0 twice on a one-GPU box): the sweep, padded to a whole share, once per
    device, so that each device's copy of the tables serves the whole sweep"""
    import torch
    from schnorr_b200 import Engine
    k, (pk, pkp) = gen_sweep
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    pad = -len(k) % 32  # the per-device share is rounded up to 32 tuples
    kk = np.concatenate([k, k[:pad]] * len(devs))
    wk, wp = np.concatenate([pk, pk[:pad]] * len(devs)), np.concatenate([pkp, pkp[:pad]] * len(devs))
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for obl in (False, True):
            g0, g1 = eng.keygen_double(kk, oblivious=obl)
            assert (g0 == wk).all() and (g1 == wp).all(), (obl, _first_diff(g0, wk), _first_diff(g1, wp))
    finally:
        eng.close()


# ---- GPU: keysets past one build launch and past 2^32 words of tables ----------------------------------------------
K_KEYS = (43363, 21683, 21683)  # key K - 1's first table starts past 2^32 words; K is not a multiple of 32 or 2048
N_BLOCK = 4096                  # random tuples per probe key (more when their challenges miss a reachable digit)
N_SIGNED = 128                  # signed tuples per probe key


def probe_keys(K, nt):
    """keys at the build launches' boundaries, K - 1, and on either side of 2^31 and 2^32 bytes and 2^31 and 2^32 words
    of table offset (key k's tables start at word (nt k + p) KS_TABLE_WORDS)"""
    B = KS_BUILD_KEYS
    keys = {0, 1, B - 1, B, B + 1, (K - 1) // B * B, K - 1}
    for words in (1 << 29, 1 << 30, 1 << 31, 1 << 32):
        t = words // KS_TABLE_WORDS  # the table holding that word
        keys |= {(t - 1) // nt, t // nt, (t + 1) // nt}
    assert max(keys) == K - 1
    return sorted(keys)


KINDS = {1: "torsion", 3: "off-curve", 6: "small-order", 9: "identity", 11: "torsion", -2: "torsion"}  # by probe rank


def _kinds(probes, roll=0):
    kinds = {p: "plain" for p in probes}
    for i, kind in KINDS.items():
        kinds[probes[(i + roll) % len(probes)]] = kind
    return kinds


def _points(rows):
    return [(V.unmont(r[:8]), V.unmont(r[8:16])) for r in rows]


class Keys:
    pass


def make_keyset_keys(engine, scheme, K, probes, kinds, seed):
    """K keys from the device's keygen; the probe keys from ref_cpu, with the probe kinds applied"""
    rs = np.random.RandomState(seed)
    tors = V.torsion_points()
    k = Keys()
    k.sk = rand_scalars(rs, K)
    gsk = rand_scalars(rs, K)
    if scheme == 0:
        k.pk, k.pk2 = engine.keygen(k.sk), None
    elif scheme == 1:
        k.pk, k.pk2 = engine.keygen_double(k.sk)
    else:
        k.pk2 = engine.keygen(gsk)
        k.pk = engine.keygen_vargen(k.sk, k.pk2)
    p = np.array(probes)
    if scheme == 0:
        k.pk[p] = ref_cpu.keygen(k.sk[p])
    elif scheme == 1:
        k.pk[p], k.pk2[p] = ref_cpu.keygen(k.sk[p], double=True)
    else:
        k.pk2[p] = ref_cpu.keygen(gsk[p])
        k.pk[p] = ref_cpu.keygen(k.sk[p], gen=k.pk2[p])
    torsion = [q for q in probes if kinds[q] == "torsion"]
    for i, q in enumerate(probes):
        T = tors[1 + i % 7]
        kind = kinds[q]
        if kind == "torsion" and scheme == 2 and q == torsion[-1]:  # a whole-curve generator: PK = sk (G' + T)
            k.pk2[q] = V.points([o.pt_add(_points(k.pk2[q:q + 1])[0], T)])[0]
            k.pk[q] = ref_cpu.keygen(k.sk[q:q + 1], gen=k.pk2[q:q + 1])[0]
        elif kind == "torsion":
            k.pk[q] = V.points([o.pt_add(_points(k.pk[q:q + 1])[0], T)])[0]
        elif kind in ("small-order", "identity"):
            k.pk[q] = V.points([T if kind == "small-order" else o.IDENTITY])[0]
            if scheme == 1:
                k.pk2[q] = k.pk[q]
        elif kind == "off-curve":
            tgt = k.pk2 if scheme == 1 else k.pk  # the second point of a double key
            tgt[q, 8:16] = from_ints([(V.unmont(tgt[q, 8:16]) + 1) * V.RADIX % Q])[0]
    return k


def _ref_verify(scheme, pk, pk2, u, Rr, Rp, m):
    if scheme == 0:
        return ref_cpu.verify(pk, u, Rr, m)
    if scheme == 1:
        return ref_cpu.verify_double(pk, pk2, u, Rr, Rp, m)
    return ref_cpu.verify_vargen(pk, pk2, u, Rr, m)


def _mont(a):
    return from_ints([x * V.RADIX % Q for x in to_ints(a)])


def random_block(scheme, n, seed):
    """n tuples with random u < r, R (R') = random multiples of G and m < q, extended until their challenges read every
    (window, digit) of the 8-bit comb that a challenge (< 2^250) can read: (u, R, R' or None, m)"""
    rs = np.random.RandomState(seed)
    target = reachable(8, 1 << 250)
    u, Rr, Rp, m = [], [], [], []
    seen = set()
    while True:
        uu, mm = rand_scalars(rs, n), rand_scalars(rs, n, 254)
        r1 = ref_cpu.keygen(rand_scalars(rs, n))
        r2 = ref_cpu.keygen(rand_scalars(rs, n)) if scheme == 1 else None
        _, c = _ref_verify(scheme, r1, r1, uu, r1, r2, mm)  # the challenge does not depend on the key
        u.append(uu); Rr.append(r1); Rp.append(r2); m.append(mm)
        seen |= covered(recode(c, 8))
        if seen == target:
            break
        n = 512
    cat = lambda xs: np.concatenate(xs) if xs[0] is not None else None
    return cat(u), cat(Rr), cat(Rp), cat(m)


def probe_tuples(scheme, keys, probes, kinds, block, n_block, n_signed, seed):
    """per probe key: the first n_block tuples of the block, n_signed tuples signed by the key (u = nonce and R = nonce B
    for small-order and identity keys: valid iff c PK = O) and, for the variable generator, the W = 8 u sweep on the
    block's R and m.  Returns (idx, u, R, R' or None, m)."""
    rs = np.random.RandomState(seed)
    bu, bR, bRp, bm = (x[:n_block] if x is not None else None for x in block)
    u8 = sweep_of(8)[2][0] if scheme == 2 else None
    parts = []
    for q in probes:
        parts.append((np.full(n_block, q), bu, bR, bRp, bm))
        if kinds[q] == "off-curve":
            continue
        sk = np.repeat(keys.sk[q:q + 1], n_signed, axis=0)
        nonce, m = rand_scalars(rs, n_signed), rand_scalars(rs, n_signed, 254)
        Rp = None
        if kinds[q] in ("small-order", "identity"):
            u = nonce
            if scheme == 2:
                Rr = ref_cpu.scalar_mul(np.repeat(keys.pk2[q:q + 1], n_signed, axis=0), nonce)
            else:
                Rr, Rp = ref_cpu.keygen(nonce, double=True)
        elif scheme == 0:
            u, Rr, _ = ref_cpu.sign(sk, m, nonce)
        elif scheme == 1:
            u, Rr, Rp, _ = ref_cpu.sign_double(sk, m, nonce)
        else:
            u, Rr, _ = ref_cpu.sign_vargen(sk, np.repeat(keys.pk2[q:q + 1], n_signed, axis=0), m, nonce)
        parts.append((np.full(n_signed, q), u, Rr, Rp if scheme == 1 else None, m))
        if u8 is not None:
            n8 = len(u8)
            parts.append((np.full(n8, q), u8, bR[:n8], None, bm[:n8]))
    cat = lambda i: np.concatenate([p[i] for p in parts]) if parts[0][i] is not None else None
    return (cat(0).astype(np.uint32),) + tuple(cat(i) for i in range(1, 5))


def check_probe_rows(ks, scheme, keys, probes, kinds, t):
    """KeySet.verify_witness and KeySet.verify on the probe tuples t against ref_cpu on the gathered keys"""
    idx, u, Rr, Rp, m = t
    pk, pk2 = keys.pk[idx], (keys.pk2[idx] if keys.pk2 is not None else None)
    ok, rows = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
    kok, kc = ks.verify(idx, u, Rr, m, Rp=Rp)
    want_ok, c = _ref_verify(scheme, pk, pk2, u, Rr, Rp, m)
    good = np.array([kinds[q] != "off-curve" for q in idx])
    assert (kc == c).all(), _first_diff(kc, c)
    # the expected row (Engine.sign_witness's layout): u, R (, R'), PK (, PK' | GEN), m, c, SA, SB (, SA', SB')
    if scheme == 2:
        sa = [ref_cpu.scalar_mul(pk2, u)]
    else:
        uniq, inv = np.unique(u, axis=0, return_inverse=True)  # the block's u recur for every probe key
        g, gp = ref_cpu.keygen(uniq, double=True)
        sa = [g[inv.reshape(-1)], gp[inv.reshape(-1)]]
    sb = [ref_cpu.scalar_mul(pk, c)] + ([ref_cpu.scalar_mul(pk2, c)] if scheme == 1 else [])
    if scheme == 1:
        cols = [_mont(u), Rr, Rp, pk, pk2, m, _mont(c), sa[0], sb[0], sa[1], sb[1]]
    else:
        cols = [_mont(u), Rr, pk] + ([pk2] if scheme == 2 else []) + [m, _mont(c), sa[0], sb[0]]
    want = np.concatenate(cols, axis=1)
    got = rows.reshape(len(idx), -1)
    for q in probes:
        sel = idx == q
        if kinds[q] == "off-curve":
            assert not ks.key_ok[q] and not ok[sel].any() and not kok[sel].any() and not got[sel].any(), q
            continue
        assert ks.key_ok[q], (q, kinds[q])
        bad = np.nonzero((got[sel] != want[sel]).any(axis=1))[0]
        assert len(bad) == 0, (q, kinds[q], f"{len(bad)} rows differ, first at {bad[:4].tolist()}",
                               [k for k in range(WIDTH[scheme]) if (got[sel][bad[0], 8 * k:8 * k + 8] != want[sel][bad[0], 8 * k:8 * k + 8]).any()])
        assert (ok[sel] == want_ok[sel]).all() and (kok[sel] == want_ok[sel]).all(), (q, kinds[q])
    assert want_ok[good].any() and not want_ok[good].all()
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("scheme", **SCHEMES)
def test_keyset_tables_past_2_32_words(engine, scheme):
    import torch
    nt = 1 if scheme == 0 else 2
    K = K_KEYS[scheme]
    assert (K - 1) * nt * KS_TABLE_WORDS > 1 << 32 and K % 32 and K % KS_BUILD_KEYS
    need = K * nt * KS_TABLE_WORDS * 4 + KS_BUILD_KEYS * 32 * 2 * 128 * 32 + (1 << 30)  # tables, build scratch, batches
    free = torch.cuda.mem_get_info()[0]
    if free < need:
        pytest.skip(f"a keyset of {K} keys needs {need} B of device memory; {free} B are free")
    probes = probe_keys(K, nt)
    kinds = _kinds(probes)
    keys = make_keyset_keys(engine, scheme, K, probes, kinds, 1100 + scheme)
    block = random_block(scheme, N_BLOCK, 1200 + scheme)
    target = reachable(8, 1 << 250)
    with engine.keyset(scheme, keys.pk, keys.pk2) as ks:
        assert ks.key_ok.sum() == K - 1
        t = probe_tuples(scheme, keys, probes, kinds, block, len(block[0]), N_SIGNED, 1300 + scheme)
        c = check_probe_rows(ks, scheme, keys, probes, kinds, t)
        for q in probes:  # each good probe key's SB read every entry a challenge can read ...
            if kinds[q] != "off-curve":
                assert covered(recode(c[t[0] == q], 8)) == target, q
                if scheme == 2:  # ... and its SA every entry of its generator's comb a u < r can read
                    assert covered(recode(t[1][t[0] == q], 8)) == reachable(8, R), q
        # replace more than one build launch of slots, probe slots included, in shuffled order; the probe kinds move on by
        # one probe, so the off-curve slot gets a good key and a good one an off-curve key
        rs = np.random.RandomState(1400 + scheme)
        others = np.setdiff1d(np.arange(K), probes)
        slots = np.concatenate([probes, rs.choice(others, KS_BUILD_KEYS + 450, replace=False)]).astype(np.uint32)
        rs.shuffle(slots)
        kinds2 = _kinds(probes, roll=1)
        new = make_keyset_keys(engine, scheme, K, probes, kinds2, 1500 + scheme)
        before = engine.launch_count
        new_ok = ks.update(slots, new.pk[slots], new.pk2[slots] if new.pk2 is not None else None)
        assert engine.launch_count - before == -(-len(slots) // KS_BUILD_KEYS) == 2
        assert (new_ok == np.array([kinds2.get(int(s), "plain") != "off-curve" for s in slots])).all()
        cur = Keys()
        cur.sk, cur.pk, cur.pk2 = keys.sk.copy(), keys.pk.copy(), (keys.pk2.copy() if keys.pk2 is not None else None)
        cur.sk[slots], cur.pk[slots] = new.sk[slots], new.pk[slots]
        if cur.pk2 is not None:
            cur.pk2[slots] = new.pk2[slots]
        t2 = probe_tuples(scheme, cur, probes, kinds2, block, 1024, 64, 1600 + scheme)
        check_probe_rows(ks, scheme, cur, probes, kinds2, t2)
        # revoke the last key: zero rows and verdict 0
        hi = np.array([K - 1], np.uint32)
        assert kinds2[K - 1] != "off-curve"
        ks.revoke(hi)
        idx, u, Rr, Rp, m = (x[t2[0] == K - 1] if x is not None else None for x in t2)
        ok, rows = ks.verify_witness(idx, u, Rr, m, Rp=Rp)
        assert len(idx) > 1000 and not ok.any() and not rows.any()
