"""Verdicts and challenges of batches larger than one wave of resident CTAs, tuple for tuple against ref_cpu.

Above one wave (W = 4 CTAs x SMs x 128 tuples) the curve kernels run in their persistent form (k_curve_p): window tables in
thread-major global scratch rows reused from one tuple to the next, entries staged through shared memory by cp.async, work
handed out per warp from a counter.  Here each scheme gets one seeded adversarial batch of N tuples, N chosen so that every
pipeline chunk of the host-buffer path is above a wave, with every category scattered over the whole range; ref_cpu
(oracle/ref_cpu.c: 252-step double-and-add, projective equality) judges each tuple once, and the GPU runs the same tuples
through every entry point that reaches those kernels.

Where ref_cpu and the product legitimately differ, the expected verdict says so:
  - u >= r: ref_cpu reads 252 bits of u; the product rejects u >= r (JubJubScalar::from_bytes) -> ref_ok & (u < r);
  - SB200_CHECK_POINTS: ref_ok & every point well formed;
  - byte-level calls: `invalid` from the construction, ok = ref_ok of the decoded tuple & ~invalid.
"""
import os
import random
import re

import numpy as np
import pytest

import ref_cpu
import schnorr_oracle as o
import vectors as V

pytestmark = pytest.mark.gpu
Q, R = o.Q, o.R
TPB = 128
_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "schnorr_b200", "csrc", "schnorr_b200.cu")


def _cu_value(pattern):
    """an integer constant of schnorr_b200.cu ("1 << 18" or "4"), read from the source the library is built from, so that
    retuning it resizes these batches instead of quietly moving them below the persistent form"""
    with open(_CU) as f:
        m = re.search(pattern, f.read(), re.M)
    assert m, pattern
    terms = [int(t) for t in m.group(1).split("<<")]
    return terms[0] << terms[1] if len(terms) == 2 else terms[0]


CHUNK = _cu_value(r"^constexpr int64_t CHUNK = ([0-9 <]+);")          # run_device's pipeline chunk ...
CHUNK_MIN = _cu_value(r"^constexpr int64_t CHUNK_MIN = ([0-9 <]+);")  # ... and its floor
EC_P_CTAS0 = _cu_value(r"^#define SB_EC_P_CTAS0 ([0-9]+)")
EC_P_CTAS_ALL4 = _cu_value(r"^#define SB_EC_P_CTAS_ALL4 ([0-9]+)")


def ec_p_ctas(scheme):
    """resident CTAs per SM of k_curve_p<scheme> (same formula as schnorr_b200.cu): one wave is this x SMs x 128 tuples"""
    return EC_P_CTAS0 if (EC_P_CTAS0 != 4 and scheme == 0) else (4 if EC_P_CTAS_ALL4 else (4 if scheme == 0 else 3))


def host_chunks(share):
    """the chunk sizes run_device splits one device's share into (same formula as schnorr_b200.cu)"""
    chunk = CHUNK if share >= 4 * CHUNK else max(CHUNK_MIN, ((share + 3) // 4 + 31) & ~31)
    return [min(chunk, share - c0) for c0 in range(0, share, chunk)]


@pytest.fixture(scope="module")
def sizes():
    import torch
    W = max(ec_p_ctas(s) for s in range(3)) * torch.cuda.get_device_properties(0).multi_processor_count * TPB
    N = 4 * W + 429  # chunk <= N / 4 + 32, so the last of four chunks is >= N / 4 - 96 > W; N = 13 (mod 32): ragged
    chunks = host_chunks(N)
    assert min(chunks) > W, (N, W, chunks)  # every chunk runs the persistent kernel
    return W, N


# ---- limb helpers -------------------------------------------------------------------------------------------------
def rand_scalars(rs, n, bits=251):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << (bits - 224)) - 1
    return a


def to_ints(a):
    raw = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, 8).tobytes()
    return [int.from_bytes(raw[k:k + 32], "little") for k in range(0, len(raw), 32)]


def from_ints(xs):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in xs), dtype=np.uint32).reshape(-1, 8).copy()


def aff(row):
    return V.unmont(row[:8]), V.unmont(row[8:16])


def projective(pts, zs):
    """(U : V : Z) = (u z, v z, z) rows from affine Montgomery rows, per-tuple z (Montgomery scaling by a plain integer)"""
    n = len(pts)
    U, Vv = to_ints(pts[:, :8]), to_ints(pts[:, 8:16])
    out = np.empty((n, 24), np.uint32)
    out[:, :8] = from_ints([x * z % Q for x, z in zip(U, zs)])
    out[:, 8:16] = from_ints([x * z % Q for x, z in zip(Vv, zs)])
    out[:, 16:] = from_ints([z * V.RADIX % Q for z in zs])
    return out


def scatter(rs, n, ncat):
    """category of each tuple: hashed over the whole range, never in blocks"""
    return rs.randint(0, ncat, size=n)


def check_spread(cat, names, N):
    """every category reaches every pipeline chunk and both lane halves of a warp"""
    bounds = np.cumsum([0] + host_chunks(N))
    lane = np.arange(N) % 32
    for k, name in enumerate(names):
        idx = np.nonzero(cat == k)[0]
        assert all(((idx >= lo) & (idx < hi)).any() for lo, hi in zip(bounds[:-1], bounds[1:])), name
        assert (lane[idx] < 16).any() and (lane[idx] >= 16).any() and idx.max() > N - 4096, name


def order8_point():
    return next(t for t in V.torsion_points() if all(V.mul(t, k) != o.IDENTITY for k in (1, 2, 4)))


# ---- the three adversarial batches (built and judged once per module) -------------------------------------------
class Batch:
    pass


SINGLE_CATS = ["valid", "valid2", "valid3", "valid4", "valid5", "u+1", "u+r", "m+1", "R+G", "neighbour key", "torsion base key",
               "small-order key", "torsion on R", "valid6", "valid7", "valid8"]
DOUBLE_CATS = ["valid", "valid2", "valid3", "valid4", "u+1", "u+r", "m+1", "R+G", "neighbour keys", "only R' corrupted",
               "only PK' swapped", "torsion base key", "small-order keys", "torsion on R'", "valid5", "valid6"]
VARGEN_CATS = ["valid", "valid2", "valid3", "valid4", "u+1", "u+r", "m+1", "R+gen", "neighbour key", "generator swapped",
               "torsion on key", "forced fallback", "forced fallback2", "whole-curve generator", "valid5", "valid6"]


def torsion_bases(rnd, J=32):
    """whole-curve bases W_j = a_j G + T_j (T_j runs over all 8 torsion points)"""
    tors = V.torsion_points()
    a = [rnd.randrange(1, R) for _ in range(J)]
    return a, V.points([o.pt_add(V.mul(o.G, a[j]), tors[j % len(tors)]) for j in range(J)])


def _common_corruptions(b, cat, names, upos, mpos, rnd):
    """u+1, u+r, m+1 on the category rows (python ints on those rows only)"""
    for name, f in (("u+1", lambda x: (x + 1) % R), ("u+r", lambda x: x + R)):
        idx = np.nonzero(cat == names.index(name))[0]
        b.arr[upos][idx] = from_ints([f(x) for x in to_ints(b.arr[upos][idx])])
    idx = np.nonzero(cat == names.index("m+1"))[0]
    b.arr[mpos][idx] = from_ints([x + 1 for x in to_ints(b.arr[mpos][idx])])  # m < 2^254: still canonical


def _add_points(rows, pts):
    return V.points([o.pt_add(aff(r), p) for r, p in zip(rows, pts)])


def make_single(N):
    rs, rnd = np.random.RandomState(101), random.Random(101)
    names = SINGLE_CATS
    cat = scatter(rs, N, len(names))
    check_spread(cat, names, N)
    s, nonce, m = rand_scalars(rs, N), rand_scalars(rs, N), rand_scalars(rs, N, 254)
    # torsion base keys: PK = s W_j, signed with the secret x = s a_j, so u G + c PK = R + c s T_j
    a, Wrows = torsion_bases(rnd)
    tb = np.nonzero(cat == names.index("torsion base key"))[0]
    x = s.copy()
    x[tb] = from_ints([si * a[i % len(a)] % R for si, i in zip(to_ints(s[tb]), tb)])
    pk = ref_cpu.keygen(x)
    pk[tb] = ref_cpu.keygen(s[tb], gen=Wrows[tb % len(a)])
    u, Rr, c_sign = ref_cpu.sign(x, m, nonce)
    b = Batch()
    b.sign_in, b.sign_out = (x.copy(), m.copy(), nonce.copy()), (u.copy(), Rr.copy(), c_sign)
    b.arr = [pk, u, Rr, m]
    # small-order / identity keys with R = u G (the signature's R is nonce G: u = nonce)
    tors = V.points(V.torsion_points())
    so = np.nonzero(cat == names.index("small-order key"))[0]
    pk[so], u[so] = tors[so % len(tors)], nonce[so]
    # torsion on R: PK = x G + T8, R = k G + j T8, u = k - c x with c = H(R, m); valid iff c = j (mod 8)
    T8 = order8_point()
    rt = np.nonzero(cat == names.index("torsion on R"))[0]
    pk[rt] = _add_points(pk[rt], [T8] * len(rt))
    Rr[rt] = _add_points(Rr[rt], [V.mul(T8, int(i) % 8) for i in rt])
    u1, _, _ = ref_cpu.sign_vargen(x[rt], Rr[rt], m[rt], from_ints([1] * len(rt)))  # R' = 1 * R: u1 = 1 - c x
    u[rt] = from_ints([(v + k - 1) % R for v, k in zip(to_ints(u1), to_ints(nonce[rt]))])
    _common_corruptions(b, cat, names, 1, 3, rnd)
    rg = np.nonzero(cat == names.index("R+G"))[0]
    Rr[rg] = _add_points(Rr[rg], [o.G] * len(rg))
    nb = np.nonzero(cat == names.index("neighbour key"))[0]
    pk[nb] = pk[(nb + 1) % N]
    ok, c = ref_cpu.verify(pk, u, Rr, m)
    b.ge_r = cat == names.index("u+r")
    b.want, b.c, b.cat, b.names, b.N = ok & ~b.ge_r, c, cat, names, N
    b.point_pos, b.R_pos = (0, 2), (2,)
    _check_batch(b)
    return b


def make_double(N):
    rs, rnd = np.random.RandomState(102), random.Random(102)
    names = DOUBLE_CATS
    cat = scatter(rs, N, len(names))
    check_spread(cat, names, N)
    s, nonce, m = rand_scalars(rs, N), rand_scalars(rs, N), rand_scalars(rs, N, 254)
    a, Wrows = torsion_bases(rnd)
    tb = np.nonzero(cat == names.index("torsion base key"))[0]
    x = s.copy()
    x[tb] = from_ints([si * a[i % len(a)] % R for si, i in zip(to_ints(s[tb]), tb)])
    pk, pkp = ref_cpu.keygen(x, double=True)
    pk[tb] = ref_cpu.keygen(s[tb], gen=Wrows[tb % len(a)])
    u, R1, R2, c_sign = ref_cpu.sign_double(x, m, nonce)
    b = Batch()
    b.sign_in, b.sign_out = (x.copy(), m.copy(), nonce.copy()), (u.copy(), R1.copy(), R2.copy(), c_sign)
    b.arr = [pk, pkp, u, R1, R2, m]
    tors = V.points(V.torsion_points())
    so = np.nonzero(cat == names.index("small-order keys"))[0]  # R = u G, R' = u G'
    pk[so], pkp[so], u[so] = tors[so % len(tors)], tors[(so // 8) % len(tors)], nonce[so]
    # torsion on R': PK' = x G' + T8, R' = k G' + j T8, u = k - c x; c from ref_cpu's challenge of the new tuple
    T8 = order8_point()
    rt = np.nonzero(cat == names.index("torsion on R'"))[0]
    pkp[rt] = _add_points(pkp[rt], [T8] * len(rt))
    R2[rt] = _add_points(R2[rt], [V.mul(T8, int(i) % 8) for i in rt])
    _, c_rt = ref_cpu.verify_double(pk[rt], pkp[rt], u[rt], R1[rt], R2[rt], m[rt])
    u[rt] = from_ints([(k - c * xi) % R for k, c, xi in zip(to_ints(nonce[rt]), to_ints(c_rt), to_ints(x[rt]))])
    _common_corruptions(b, cat, names, 2, 5, rnd)
    rg = np.nonzero(cat == names.index("R+G"))[0]
    R1[rg] = _add_points(R1[rg], [o.G] * len(rg))
    rp = np.nonzero(cat == names.index("only R' corrupted"))[0]
    R2[rp] = _add_points(R2[rp], [o.G_NUMS] * len(rp))
    nb = np.nonzero(cat == names.index("neighbour keys"))[0]
    pk[nb], pkp[nb] = pk[(nb + 1) % N], pkp[(nb + 1) % N]
    sw = np.nonzero(cat == names.index("only PK' swapped"))[0]
    pkp[sw] = pkp[(sw + 1) % N]
    ok, c = ref_cpu.verify_double(pk, pkp, u, R1, R2, m)
    b.ge_r = cat == names.index("u+r")
    b.want, b.c, b.cat, b.names, b.N = ok & ~b.ge_r, c, cat, names, N
    b.point_pos, b.R_pos = (0, 1, 3, 4), (3, 4)
    _check_batch(b)
    return b


def generator_pool(rnd, rs, size=2048):
    """prime-order generators, the identity (last row), and whole-curve generators (torsion component: rows 0, 4, 8 ...)"""
    k = rand_scalars(rs, size)
    pool = ref_cpu.keygen(k)
    whole = np.arange(0, size, 4)
    pool[whole] = ref_cpu.scalar_mul(V.points([V.rand_curve_point(rnd) for _ in range(16)])[whole % 16], k[whole])
    pool[size - 1] = V.points([o.IDENTITY])[0]
    return pool, whole


def make_vargen(N):
    rs, rnd = np.random.RandomState(103), random.Random(103)
    names = VARGEN_CATS
    cat = scatter(rs, N, len(names))
    check_spread(cat, names, N)
    x, nonce, m = rand_scalars(rs, N), rand_scalars(rs, N), rand_scalars(rs, N, 254)
    pool, whole = generator_pool(rnd, rs)
    prime = np.setdiff1d(np.arange(len(pool)), whole)
    gidx = prime[rs.randint(0, len(prime), size=N)]
    wc = np.nonzero(cat == names.index("whole-curve generator"))[0]
    gidx[wc] = whole[rs.randint(0, len(whole), size=len(wc))]  # u g + c x g = (k + t r) g: valid iff t r g = O
    gen = pool[gidx]
    pk = ref_cpu.keygen(x, gen=gen)
    u, Rr, c_sign = ref_cpu.sign_vargen(x, gen, m, nonce)
    b = Batch()
    b.sign_in, b.sign_out = (x.copy(), gen.copy(), m.copy(), nonce.copy()), (u.copy(), Rr.copy(), c_sign)
    b.arr = [pk, gen, u, Rr, m]
    # forced full-size fallback: u = r - 1, PK = (k - u) / c * gen for R = k gen (valid by construction)
    ff = np.nonzero((cat == names.index("forced fallback")) | (cat == names.index("forced fallback2")))[0]
    ff = ff[gidx[ff] != len(pool) - 1]  # prime-order generators: (k - u) / c is taken mod r
    xf = [(k - (R - 1)) * pow(c, -1, R) % R for k, c in zip(to_ints(nonce[ff]), to_ints(c_sign[ff]))]
    pk[ff] = ref_cpu.keygen(from_ints(xf), gen=gen[ff])
    u[ff] = from_ints([R - 1] * len(ff))
    tk = np.nonzero(cat == names.index("torsion on key"))[0]
    tors = V.torsion_points()
    pk[tk] = _add_points(pk[tk], [tors[i % len(tors)] for i in tk])
    _common_corruptions(b, cat, names, 2, 4, rnd)
    rg = np.nonzero(cat == names.index("R+gen"))[0]
    Rr[rg] = V.points([o.pt_add(aff(r), aff(g)) for r, g in zip(Rr[rg], gen[rg])])
    nb = np.nonzero(cat == names.index("neighbour key"))[0]
    pk[nb] = pk[(nb + 1) % N]
    gs = np.nonzero(cat == names.index("generator swapped"))[0]
    gen[gs] = gen[(gs + 1) % N]
    ok, c = ref_cpu.verify_vargen(pk, gen, u, Rr, m)
    b.ge_r = cat == names.index("u+r")
    b.want, b.c, b.cat, b.names, b.N = ok & ~b.ge_r, c, cat, names, N
    b.point_pos, b.R_pos = (0, 1, 3), (3,)
    _check_batch(b)
    assert b.want[ff].all() and len(ff) > 0.1 * N
    return b


MIXED = {"torsion base key", "small-order key", "small-order keys", "torsion on R", "torsion on R'", "torsion on key",
         "whole-curve generator"}


def _check_batch(b):
    """the batch is not vacuous: a stated accept band, each category with the verdicts its construction allows"""
    assert 0.3 < b.want.mean() < 0.75, b.want.mean()
    for k, name in enumerate(b.names):
        w = b.want[b.cat == k]
        if name.startswith("valid") or name.startswith("forced fallback"):
            assert w.all(), name
        elif name in MIXED:
            assert 0.05 < w.mean() < 0.95, (name, w.mean())
        else:  # (a neighbour drawn with the same generator from the pool, or the identity generator, keeps a few valid)
            assert w.mean() < 0.01, name


def _assert_same(b, ok, c=None, rows=None, want=None):
    want = b.want if want is None else want
    bad = np.nonzero(ok != want)[0]
    assert len(bad) == 0, f"{len(bad)} verdicts differ, first at {bad[:8].tolist()}: {[b.names[k] for k in b.cat[bad[:8]]]}"
    if c is not None:
        rows = slice(None) if rows is None else rows
        diff = np.nonzero((c[rows] != b.c[rows]).any(axis=1))[0]
        assert len(diff) == 0, f"{len(diff)} challenge rows differ, first at {diff[:8].tolist()}"


@pytest.fixture(scope="module")
def single(sizes):
    return make_single(sizes[1])


@pytest.fixture(scope="module")
def double(sizes):
    return make_double(sizes[1])


@pytest.fixture(scope="module")
def vargen(sizes):
    return make_vargen(sizes[1])


def _verify(eng, scheme, arr, **kw):
    return (eng.verify, eng.verify_double, eng.verify_vargen)[scheme](*arr, **kw)


SCHEMES = ["single", "double", "vargen"]


@pytest.fixture(params=SCHEMES)
def batch(request):
    return SCHEMES.index(request.param), request.getfixturevalue(request.param)


# ---- 1. host buffers, affine, session engine ---------------------------------------------------------------------
def test_host_buffers_affine(engine, batch):
    """also pins the chunking: two launches (challenge, curve) per pipeline chunk, as many chunks as host_chunks says"""
    scheme, b = batch
    before = engine.launch_count
    ok, c = _verify(engine, scheme, b.arr)
    assert engine.launch_count - before == 2 * len(host_chunks(b.N))
    _assert_same(b, ok, c)


# ---- 2. device pointers: one call above a wave ---------------------------------------------------------------------
def _device_call(eng, name, n, flags, arrays, nbitmaps=1, want_c=False):
    """one SB200_DEVICE_PTRS call over the whole batch (the persistent kernel runs several waves, reusing its scratch rows):
    inputs copied to the device, then `nbitmaps` bitmaps [and the challenge rows] back"""
    import torch
    from schnorr_b200 import DEVICE_PTRS
    dev = torch.device("cuda:0")
    ins = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).view(np.int32)).to(dev) for a in arrays]
    bms = [torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev) for _ in range(nbitmaps)]
    c = torch.zeros((n, 8), dtype=torch.int32, device=dev) if want_c else None
    torch.cuda.synchronize()
    eng.call(name, n, flags | DEVICE_PTRS, *[x.data_ptr() for x in ins + bms], *([c.data_ptr()] if want_c else []))
    torch.cuda.synchronize()
    out = [np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool) for bm in bms]
    return out + ([c.cpu().numpy().view(np.uint32)] if want_c else [])


def _device_verify(eng, scheme, arr, flags):
    return _device_call(eng, ("verify", "verify_double", "verify_vargen")[scheme], len(arr[-1]), flags, arr, want_c=True)


def test_device_pointers_one_call(engine, batch, sizes):
    from schnorr_b200 import POINTS_AFFINE
    scheme, b = batch
    assert b.N > 4 * sizes[0]  # about four waves in one launch
    ok, c = _device_verify(engine, scheme, b.arr, POINTS_AFFINE)
    _assert_same(b, ok, c)


# ---- 3. projective inputs, per-tuple Z != 1 ------------------------------------------------------------------------
def _proj_arrays(b, seed):
    rs = np.random.RandomState(seed)
    out = list(b.arr)
    for k in b.point_pos:
        zs = [int(z) for z in rs.randint(2, 1 << 62, size=b.N, dtype=np.int64)]
        out[k] = projective(b.arr[k], zs)
    return out


def test_projective_inputs(engine, batch):
    from schnorr_b200 import POINTS_PROJECTIVE
    scheme, b = batch
    arr = _proj_arrays(b, 7 + scheme)
    ok, c = _verify(engine, scheme, arr, affine=False)
    _assert_same(b, ok, c)
    ok, c = _device_verify(engine, scheme, arr, POINTS_PROJECTIVE)
    _assert_same(b, ok, c)


# ---- 4. SB200_CHECK_POINTS: off-curve points and Z = 0 scattered ---------------------------------------------------
def test_check_points(engine, batch):
    scheme, b = batch
    arr = _proj_arrays(b, 17 + scheme)
    rs = np.random.RandomState(27 + scheme)
    bad = np.zeros(b.N, bool)
    bad_R = np.zeros(b.N, bool)
    for k in b.point_pos:
        sel = rs.randint(0, 64, size=b.N)
        zero, off = np.nonzero(sel == 0)[0], np.nonzero(sel == 1)[0]
        arr[k][zero, 16:] = 0
        V_ = to_ints(arr[k][off, 8:16])
        arr[k][off, 8:16] = from_ints([(v + 1) % Q for v in V_])  # (U : V + 1 : Z): checked below to be off the curve
        for i in off[:64]:
            zi = pow(V.unmont(arr[k][i, 16:]), -1, Q)
            assert not o.on_curve((V.unmont(arr[k][i, :8]) * zi % Q, V.unmont(arr[k][i, 8:16]) * zi % Q))
        bad[zero] = bad[off] = True
        if k in b.R_pos:  # the challenge hashes the nonce points
            bad_R[zero] = bad_R[off] = True
    from schnorr_b200 import CHECK_POINTS, POINTS_PROJECTIVE
    ok, c = _verify(engine, scheme, arr, affine=False, check_points=True)
    _assert_same(b, ok, c, rows=~bad_R, want=b.want & ~bad)
    ok, c = _device_verify(engine, scheme, arr, POINTS_PROJECTIVE | CHECK_POINTS)
    _assert_same(b, ok, c, rows=~bad_R, want=b.want & ~bad)
    assert (b.want & bad).any()  # some rejections come from the check alone


# ---- 5. second contexts with the curve kernel form forced ------------------------------------------------------------
@pytest.mark.parametrize("mode", ["always", "never"])
def test_forced_kernel_form(mode, monkeypatch, single, double, vargen):
    from schnorr_b200 import Engine
    monkeypatch.setenv("SB200_CURVE_PERSISTENT", mode)
    eng = Engine([0], ark=o.ARK_RULE)
    try:
        for scheme, b in enumerate((single, double, vargen)):
            ok, c = _verify(eng, scheme, b.arr)
            _assert_same(b, ok, c)
    finally:
        eng.close()


# ---- byte-level verifies: the same tuples encoded on the host ------------------------------------------------------
def _enc_points(rows):
    """JubJubAffine::to_bytes from canonical coordinates: v little-endian, bit 255 = lowest bit of u"""
    us, vs = to_ints(rows[:, :8]), to_ints(rows[:, 8:16])
    return np.frombuffer(b"".join((v * V.RINV % Q | ((u * V.RINV % Q) & 1) << 255).to_bytes(32, "little") for u, v in zip(us, vs)),
                         np.uint8).reshape(-1, 32).copy()


def _enc_scalars(rows, mont=False):
    xs = to_ints(rows)
    return np.frombuffer(b"".join((x * V.RINV % Q if mont else x).to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32).copy()


BAD_V = [v for v in range(2, 400) if o.affine_from_bytes(v.to_bytes(32, "little")) is None][:8]


def test_byte_level_verifies(engine, batch):
    scheme, b = batch
    rs = np.random.RandomState(37 + scheme)
    if scheme == 0:
        pts = [_enc_points(b.arr[0]), _enc_points(b.arr[2])]
        u, m = b.arr[1], b.arr[3]
    elif scheme == 1:
        pts = [_enc_points(b.arr[k]) for k in (0, 1, 3, 4)]
        u, m = b.arr[2], b.arr[5]
    else:
        pts = [_enc_points(b.arr[k]) for k in (0, 1, 3)]
        u, m = b.arr[2], b.arr[4]
    ub, mb = _enc_scalars(u), _enc_scalars(m, mont=True)
    invalid = b.ge_r.copy()  # u + r is already there: JubJubScalar::from_bytes fails
    for p in pts:  # each key and each nonce point: v >= q, or a v that does not decode
        sel = rs.randint(0, 96, size=b.N)
        for i in np.nonzero(sel == 0)[0]:  # q <= v < 2^255 (q is 255 bits: v + q could wrap past bit 255)
            p[i] = np.frombuffer((Q + int(i) % 4096 | (int(i) >> 1 & 1) << 255).to_bytes(32, "little"), np.uint8)
        for i in np.nonzero(sel == 1)[0]:
            p[i] = np.frombuffer((BAD_V[i % len(BAD_V)] | (int(i) & 1) << 255).to_bytes(32, "little"), np.uint8)
        invalid |= sel < 2
    sel = rs.randint(0, 96, size=b.N)
    for i in np.nonzero(sel == 0)[0]:  # m >= q
        mb[i] = np.frombuffer((int.from_bytes(mb[i].tobytes(), "little") + Q).to_bytes(32, "little"), np.uint8)
    invalid |= sel == 0
    if scheme == 0:
        pk, sig = pts[0], np.concatenate([ub, pts[1]], axis=1)
    elif scheme == 1:
        pk, sig = np.concatenate(pts[:2], axis=1), np.concatenate([ub, pts[2], pts[3]], axis=1)
    else:
        pk, sig = np.concatenate(pts[:2], axis=1), np.concatenate([ub, pts[2]], axis=1)
    name = ("verify_bytes", "verify_double_bytes", "verify_vargen_bytes")[scheme]
    before = engine.launch_count
    ok, inv = getattr(engine, name)(pk, sig, mb)
    assert engine.launch_count - before == 3 * len(host_chunks(b.N))  # decode, challenge, curve per pipeline chunk
    assert (inv == invalid).all(), np.nonzero(inv != invalid)[0][:8]
    _assert_same(b, ok, want=b.want & ~invalid)
    ok, inv = _device_call(engine, name, b.N, 0, [pk, sig, mb], nbitmaps=2)
    assert (inv == invalid).all(), np.nonzero(inv != invalid)[0][:8]
    _assert_same(b, ok, want=b.want & ~invalid)
    assert (b.want & invalid).any()


# ---- multi-device context: per-device split of sign, the three verifies and verify_bytes --------------------------
def test_multi_device_context(single, double, vargen):
    import torch
    from schnorr_b200 import Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    eng = Engine(devs, ark=o.ARK_RULE)
    try:
        for scheme, b in enumerate((single, double, vargen)):
            ok, c = _verify(eng, scheme, b.arr)
            _assert_same(b, ok, c)
        x, m, nonce = single.sign_in
        got = eng.sign(x, m, nonce)
        assert all((g == w).all() for g, w in zip(got, single.sign_out))
        pk = _enc_points(single.arr[0])
        sig = np.concatenate([_enc_scalars(single.arr[1]), _enc_points(single.arr[2])], axis=1)
        ok, inv = eng.verify_bytes(pk, sig, _enc_scalars(single.arr[3], mont=True))
        assert (inv == single.ge_r).all()
        _assert_same(single, ok)
    finally:
        eng.close()


def test_sign_at_scale_matches_construction(engine, single, double, vargen):
    """the batches were signed by ref_cpu: the GPU signs the same N tuples (several chunks, each above a wave)"""
    got = engine.sign(*single.sign_in)
    assert all((g == w).all() for g, w in zip(got, single.sign_out))
    got = engine.sign_double(*double.sign_in)
    assert all((g == w).all() for g, w in zip(got, double.sign_out))
    x, gen, m, nonce = vargen.sign_in
    got = engine.sign_vargen(x, gen, m, nonce)
    assert all((g == w).all() for g, w in zip(got, vargen.sign_out))


# ---- signing and key generation, whole batch against ref_cpu ------------------------------------------------------
EDGE = [0, 1, R - 1, (1 << 251) - 1]


def _edge_positions(n):
    """every j-slot (base + j * 128) of one thread, for 4 tuples per thread (sign) and 8 (keygen), and the last partial CTA"""
    pos = [3 * 512 + j * TPB + 5 for j in range(4)] + [2 * 1024 + j * TPB + 9 for j in range(8)]
    last = (n // 512) * 512
    pos += [last, last + 1, last + TPB, n - 1]
    return pos


@pytest.mark.parametrize("oblivious", [False, True], ids=["default", "oblivious"])
def test_sign_and_keygen_whole_batch(engine, oblivious):
    rs, rnd = np.random.RandomState(104), random.Random(104)
    n = 40 * 1024 + 300  # ragged against 512 (sign: 4 per thread) and 1024 (keygen: 8 per thread)
    assert n % 512 and n % 1024
    sk, nonce, m = rand_scalars(rs, n, 252), rand_scalars(rs, n, 252), rand_scalars(rs, n, 254)
    sk[sk[:, 7] >= (R >> 224)] >>= 1  # keep them below r
    nonce[nonce[:, 7] >= (R >> 224)] >>= 1
    pos = _edge_positions(n)
    sk[pos] = from_ints([EDGE[k % 4] for k in range(len(pos))])
    nonce[pos] = from_ints([EDGE[(k + 1) % 4] for k in range(len(pos))])
    assert max(to_ints(sk)) < R and max(to_ints(nonce)) < R
    want = ref_cpu.sign(sk, m, nonce)
    assert all((g == w).all() for g, w in zip(engine.sign(sk, m, nonce, oblivious=oblivious), want))
    want = ref_cpu.sign_double(sk, m, nonce)
    assert all((g == w).all() for g, w in zip(engine.sign_double(sk, m, nonce, oblivious=oblivious), want))
    pk, pkp = ref_cpu.keygen(sk, double=True)
    assert (engine.keygen(sk, oblivious=oblivious) == pk).all()
    got = engine.keygen_double(sk, oblivious=oblivious)
    assert (got[0] == pk).all() and (got[1] == pkp).all()
    # variable generator: prime-order, whole-curve and identity generators, affine and (U : V : Z)
    gen = generator_pool(rnd, rs, 1024)[0][rs.randint(0, 1024, size=n)]
    gen[pos] = V.points([o.IDENTITY])[0]
    want = ref_cpu.sign_vargen(sk, gen, m, nonce)
    assert all((g == w).all() for g, w in zip(engine.sign_vargen(sk, gen, m, nonce, oblivious=oblivious), want))
    pkv = ref_cpu.keygen(sk, gen=gen)
    assert (engine.keygen_vargen(sk, gen, oblivious=oblivious) == pkv).all()
    zs = [int(z) for z in rs.randint(2, 1 << 62, size=n, dtype=np.int64)]
    genp = projective(gen, zs)
    assert all((g == w).all() for g, w in zip(engine.sign_vargen(sk, genp, m, nonce, affine=False, oblivious=oblivious), want))
    assert (engine.keygen_vargen(sk, genp, affine=False, oblivious=oblivious) == pkv).all()


def test_byte_level_signers_whole_batch(engine):
    rs, rnd = np.random.RandomState(105), random.Random(105)
    n = 40 * 1024 + 300
    sk, nonce, m = rand_scalars(rs, n), rand_scalars(rs, n), rand_scalars(rs, n, 254)
    pos = _edge_positions(n)
    sk[pos] = from_ints([EDGE[k % 4] for k in range(len(pos))])
    nonce[pos] = from_ints([EDGE[(k + 3) % 4] for k in range(len(pos))])
    u, Rr, _ = ref_cpu.sign(sk, m, nonce)
    ud, R1, R2, _ = ref_cpu.sign_double(sk, m, nonce)
    gen = generator_pool(rnd, rs, 1024)[0][rs.randint(0, 1024, size=n)]
    uv, Rv, _ = ref_cpu.sign_vargen(sk, gen, m, nonce)
    skb, nb, mb = _enc_scalars(sk), _enc_scalars(nonce), _enc_scalars(m, mont=True)
    sel = rs.randint(0, 128, size=n)  # invalid scalars scattered: sk >= r, nonce >= r, m >= q, all-ones
    for i in np.nonzero(sel == 0)[0]:
        skb[i] = np.frombuffer((R + int(i)).to_bytes(32, "little"), np.uint8)
    for i in np.nonzero(sel == 1)[0]:
        nb[i] = np.frombuffer((R + int(i)).to_bytes(32, "little"), np.uint8)
    for i in np.nonzero(sel == 2)[0]:
        mb[i] = np.frombuffer((Q + int(i)).to_bytes(32, "little"), np.uint8)
    for i in np.nonzero(sel == 3)[0]:
        nb[i] = 0xFF
    invalid = sel < 4
    good = ~invalid
    sig, inv = engine.sign_bytes(skb, mb, nb, want_invalid=True)
    assert (inv == invalid).all() and not sig[invalid].any()
    assert (sig[good] == np.concatenate([_enc_scalars(u), _enc_points(Rr)], axis=1)[good]).all()
    sig, inv = engine.sign_double_bytes(skb, mb, nb, want_invalid=True)
    assert (inv == invalid).all() and not sig[invalid].any()
    assert (sig[good] == np.concatenate([_enc_scalars(ud), _enc_points(R1), _enc_points(R2)], axis=1)[good]).all()
    gb = _enc_points(gen)
    bad_g = np.nonzero(sel == 4)[0]
    gb[bad_g] = np.frombuffer(BAD_V[0].to_bytes(32, "little"), np.uint8)
    sig, okv = engine.sign_vargen_bytes(np.concatenate([skb, gb], axis=1), mb, nb)
    good_v = good & (sel != 4)
    assert (okv == good_v).all() and not sig[~good_v].any()
    assert (sig[good_v] == np.concatenate([_enc_scalars(uv), _enc_points(Rv)], axis=1)[good_v]).all()


# ---- the debug hook reaches the persistent kernel: half-size fallback forced above a wave -----------------------------
def test_hostile_challenges_reach_the_persistent_kernel(engine, sizes, monkeypatch):
    """sb200_dbg_verify_ec launches what sb200_verify launches at that size: above one wave, k_curve_p<0>.  Every third lane
    gets a challenge for which the half-size path gives up; keys carry torsion, half the R are corrupted.  Expected verdicts
    from the construction R = (u + c s) G + c T (+ G when corrupted)."""
    import torch
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE, Engine
    W, _ = sizes
    n = W + 1013
    rs, rnd = np.random.RandomState(106), random.Random(106)
    hostile = V.hgcd_hostile_challenges(256)
    c = [hostile[(i // 3) % len(hostile)] if i % 3 == 0 else rnd.randrange(1 << 250) for i in range(n)]
    s, u = rand_scalars(rs, n), rand_scalars(rs, n)
    corrupt = rs.randint(0, 2, size=n).astype(bool)
    e = [(ui + ci * si + int(k)) % R for ui, ci, si, k in zip(to_ints(u), c, to_ints(s), corrupt)]  # + G when corrupted
    pk, Rr = ref_cpu.keygen(s), ref_cpu.keygen(from_ints(e))
    tors = V.torsion_points()
    tk = np.arange(1, n, 5)  # keys with a torsion component, c T folded into R so that the verdict stays by construction
    T = [tors[i % len(tors)] for i in tk]
    pk[tk] = _add_points(pk[tk], T)
    Rr[tk] = _add_points(Rr[tk], [V.mul(t, c[i]) for t, i in zip(T, tk)])
    want = ~corrupt
    cs = from_ints(c)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev)
    ins = [t(a) for a in (pk, u, Rr, cs)]
    bm = torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    engine.call("dbg_verify_ec", n, POINTS_AFFINE | DEVICE_PTRS, *[x.data_ptr() for x in ins], bm.data_ptr())
    torch.cuda.synchronize()
    ok = np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
    assert (ok == want).all(), np.nonzero(ok != want)[0][:8]
    monkeypatch.setenv("SB200_CURVE_PERSISTENT", "always")
    eng = Engine([0], ark=o.ARK_RULE)
    try:
        assert (eng.dbg_verify_ec(pk, u, Rr, cs) == want).all()
    finally:
        eng.close()
