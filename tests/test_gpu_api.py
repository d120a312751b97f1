"""GPU twins of the reference's own tests, through the host mirror of its API (schnorr_b200/api.py), plus
full-size batches checked through size-independent properties and against the multi-threaded C restatement."""
import random

import numpy as np
import pytest

import ref_cpu
import schnorr_oracle as o
import vectors as V
from schnorr_b200 import api

pytestmark = pytest.mark.gpu
Q, R = o.Q, o.R


@pytest.fixture(autouse=True)
def _use_engine(engine):
    api.set_engine(engine)
    yield
    api.set_engine(None)


# ---- /root/reference/tests/schnorr.rs ------------------------------------------------------------
def test_sign_verify():
    rng = api.StdRng.seed_from_u64(2321)
    sk = api.SecretKey.random(rng)
    message = rng.random_bls()
    pk = api.PublicKey.from_secret_key(sk)
    sig = sk.sign(rng, message)
    assert pk.verify(sig, message)
    # bit-exact with the oracle on the same seeded stream
    orng = o.StdRng.seed_from_u64(2321)
    osk, om = orng.random_fr(), orng.random_fq()
    ou, oR, _ = o.sign(osk, orng.random_fr(), om)
    assert (sk.as_scalar(), message, sig.u(), sig.R().affine()) == (osk, om, ou, oR)
    assert pk.as_ref().affine() == o.keygen(osk)
    assert sig.to_bytes() == ou.to_bytes(32, "little") + o.affine_to_bytes(oR)


def test_wrong_keys():
    rng = api.StdRng.seed_from_u64(2321)
    sk = api.SecretKey.random(rng)
    message = rng.random_bls()
    sig = sk.sign(rng, message)
    pk = api.PublicKey.from_secret_key(api.SecretKey.random(rng))
    assert not pk.verify(sig, message)


def test_to_from_bytes():
    rng = api.StdRng.seed_from_u64(2321)
    sk = api.SecretKey.random(rng)
    message = rng.random_bls()
    sig = sk.sign(rng, message)
    assert sig == api.Signature.from_bytes(sig.to_bytes())
    pk = api.PublicKey.from_secret_key(sk)
    assert api.PublicKey.from_bytes(pk.to_bytes()).verify(api.Signature.from_bytes(sig.to_bytes()), message)
    assert api.SecretKey.from_bytes(sk.to_bytes()) == sk


# ---- /root/reference/tests/schnorr_double.rs -----------------------------------------------------
def test_double_sign_verify_wrong_keys_bytes():
    rng = api.StdRng.seed_from_u64(2321)
    sk = api.SecretKey.random(rng)
    message = rng.random_bls()
    pk = api.PublicKeyDouble.from_secret_key(sk)
    sig = sk.sign_double(rng, message)
    assert pk.verify(sig, message)
    assert not api.PublicKeyDouble.from_secret_key(api.SecretKey.random(rng)).verify(sig, message)
    assert sig == api.SignatureDouble.from_bytes(sig.to_bytes())
    assert api.PublicKeyDouble.from_bytes(pk.to_bytes()) == pk
    orng = o.StdRng.seed_from_u64(2321)
    osk, om = orng.random_fr(), orng.random_fq()
    ou, oR, oRp, _ = o.sign_double(osk, orng.random_fr(), om, mul=V.mul)
    assert (sig.u(), sig.R().affine(), sig.R_prime().affine()) == (ou, oR, oRp)


# ---- /root/reference/tests/schnorr_var_generator.rs ----------------------------------------------
def test_var_generator_sign_verify_wrong_keys_bytes():
    rng = api.StdRng.seed_from_u64(2321)
    sk = api.SecretKeyVarGen.random(rng)
    message = rng.random_bls()
    pk = api.PublicKeyVarGen.from_secret_key(sk)
    sig = sk.sign(rng, message)
    assert pk.verify(sig, message)
    assert not api.PublicKeyVarGen.from_secret_key(api.SecretKeyVarGen.random(rng)).verify(sig, message)
    assert sig == api.SignatureVarGen.from_bytes(sig.to_bytes())
    assert api.PublicKeyVarGen.from_bytes(pk.to_bytes()) == pk
    assert api.SecretKeyVarGen.from_bytes(sk.to_bytes()) == sk
    orng = o.StdRng.seed_from_u64(2321)
    osk, os_ = orng.random_fr(), orng.random_fr()
    ogen = V.mul(o.G, os_)
    om = orng.random_fq()
    ou, oR, _ = o.sign_vargen(osk, ogen, orng.random_fr(), om, mul=V.mul)
    assert (sk.generator().affine(), sig.u(), sig.R().affine()) == (ogen, ou, oR)
    # with_variable_generator builds the same key type
    assert api.SecretKey(osk).with_variable_generator(api.JubJubExtended(*ogen)) == sk


# ---- /root/reference/tests/keys.rs ---------------------------------------------------------------
def test_partial_eq_pk():
    g = lambda k: api.JubJubExtended(*V.mul(o.G, k))
    s = lambda a, b: api.JubJubExtended(*o.pt_add(V.mul(o.G, a), V.mul(o.G, b)))
    left, right, wrong = api.PublicKey(s(2, 7)), api.PublicKey(s(4, 5)), api.PublicKey(s(4, 567758785))
    assert left == right and left != wrong
    a = left.as_ref()
    scaled = api.PublicKey.from_raw_unchecked(api.JubJubExtended(a.U * 777, a.V * 777, 777))
    assert scaled.as_ref().U != a.U and scaled == left and g(9) == a


def test_batch_api_consumes_rng_in_order():
    rng1, rng2 = api.StdRng.seed_from_u64(77), api.StdRng.seed_from_u64(77)
    sks = [api.SecretKey.random(rng1) for _ in range(5)]
    [api.SecretKey.random(rng2) for _ in range(5)]
    msgs = [rng1.random_bls() for _ in range(5)]
    [rng2.random_bls() for _ in range(5)]
    batch = api.SecretKey.sign_batch(sks, rng1, msgs)
    single = [sk.sign(rng2, m) for sk, m in zip(sks, msgs)]
    assert batch == single
    pks = api.PublicKey.from_secret_keys(sks)
    assert api.PublicKey.verify_batch(pks, batch, msgs).all()
    assert not api.PublicKey.verify_batch(pks[1:] + pks[:1], batch, msgs).any()


# ---- BASELINE.json configs at full size: properties + the C restatement on a sample --------------
def _synth(n, seed):
    rs = np.random.RandomState(seed)
    def sc(bits):
        a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
        a[:, 7] &= (1 << bits) - 1
        return a
    return sc(27), sc(27), sc(30)


def test_config1_single_verify_2_16_vs_cpu_restatement(engine):
    """configs[1]: single-key verify, batch 2^16, all valid -> all true; full batch also run on the CPU restatement"""
    n = 1 << 16
    sk, nonce, msg = _synth(n, 0xC1)
    pk = engine.keygen(sk)
    u, R_, c = engine.sign(sk, msg, nonce)
    ok, c2 = engine.verify(pk, u, R_, msg)
    assert ok.all() and (c2 == c).all()
    bad = u.copy()
    bad[::10, 0] ^= 1
    ok_a, c_a = engine.verify(pk, bad, R_, msg)
    assert (c_a == c).all() and not ok_a[::10].any() and ok_a[1::10].all()
    s = np.arange(0, n, n // 4096)  # strided over the whole batch: every pipeline chunk and late work items
    okc, cc = ref_cpu.verify(pk[s], bad[s], R_[s], msg[s])
    assert (okc == ok_a[s]).all() and okc.any() and not okc.all() and (cc == c[s]).all()
    s2 = s[::2]
    uc, Rc, _ = ref_cpu.sign(sk[s2], msg[s2], nonce[s2])
    assert (uc == u[s2]).all() and (Rc == R_[s2]).all()
    assert (ref_cpu.keygen(sk[s2]) == pk[s2]).all()


def test_ragged_batch_across_pipeline_chunks(engine):
    """n = 2^18 + 33: the host-buffer path splits it into a full 2^18 chunk and a 33-tuple tail on the second stream;
    verdict words, challenge rows and the projective (Z != 1) path must line up across the chunk boundary"""
    n = (1 << 18) + 33
    sk, nonce, msg = _synth(n, 0xC5)
    pk = engine.keygen(sk)
    u, R_, c = engine.sign(sk, msg, nonce)
    bad = (np.arange(n) % 7) == 3
    u[bad, 0] ^= 1
    ok, c2 = engine.verify(pk, u, R_, msg)
    assert (ok == ~bad).all() and (c2 == c).all()
    # the same points as (U : V : Z) with a per-tuple Z: multiply by z = 2 (Montgomery limbs of 2, 4 ...) on the host
    m = 4096  # a slice that straddles nothing special; projective inputs cost an inversion each
    z = np.array([(2 + i % 5) for i in range(m)], dtype=object)
    Q = o.Q
    def scale(pts):
        out = np.zeros((m, 24), np.uint32)
        for i in range(m):
            x, y = V.unmont(pts[i, :8]), V.unmont(pts[i, 8:])
            out[i] = np.concatenate([V.mont(x * z[i] % Q), V.mont(y * z[i] % Q), V.mont(int(z[i]))])
        return out
    s0 = n - m
    okp, cp = engine.verify(scale(pk[s0:]), u[s0:], scale(R_[s0:]), msg[s0:], affine=False)
    assert (okp == ok[s0:]).all() and (cp == c[s0:]).all()
    # without c_out the challenges travel between the two kernels in device scratch only
    ok3, none = engine.verify(pk, u, R_, msg, want_c=False)
    assert none is None and (ok3 == ok).all()
    pkd, pkdp = engine.keygen_double(sk[:m])
    ud, Rd, Rdp, cd = engine.sign_double(sk[:m], msg[:m], nonce[:m])
    okd, _ = engine.verify_double(pkd, pkdp, ud, Rd, Rdp, msg[:m], want_c=False)
    okv, _ = engine.verify_vargen(pk[:m], pkd, ud, Rd, msg[:m], want_c=False)  # generator = G-keys: u Gen + c PK != R in general
    assert okd.all() and not okv.all()


def test_config2_double_verify_2_20_properties(engine):
    n = 1 << 20
    sk, nonce, msg = _synth(n, 0xC2)
    pk, pkp = engine.keygen_double(sk)
    u, R_, Rp, c = engine.sign_double(sk, msg, nonce)
    bad = (np.arange(n) % 7) == 3
    u2 = u.copy(); u2[bad, 1] ^= 4
    ok, c2 = engine.verify_double(pk, pkp, u2, R_, Rp, msg)
    assert (ok == ~bad).all() and (c2 == c).all()
    s = np.arange(0, n, n // 1024)  # strided over the whole batch: every pipeline chunk and late work items
    okc, _ = ref_cpu.verify_double(pk[s], pkp[s], u2[s], R_[s], Rp[s], msg[s])
    assert (okc == ok[s]).all()
    # swapping the two halves of the key breaks exactly the valid ones
    ok, _ = engine.verify_double(pkp[:4096], pk[:4096], u[:4096], R_[:4096], Rp[:4096], msg[:4096])
    assert not ok.any()


def test_config3_sign_2_20_seeded_nonces(engine):
    """configs[3]: nonce i = JubJubScalar::random of a StdRng consumed in tuple order = from_bytes_wide(block i)"""
    n = 1 << 20
    sk, _, msg = _synth(n, 0xC3)
    rng = api.StdRng.seed_from_u64(0xC3)
    blocks = rng.blocks(0, n)  # [n,16] u32: the 64-byte draws
    sample = list(range(0, n, n // 512))
    nonce_s = [int.from_bytes(blocks[i].tobytes(), "little") % R for i in sample]
    assert nonce_s[:3] == [o.nonce_from_block(o.StdRng.seed_from_u64(0xC3).key, i) for i in sample[:3]]
    # whole batch: nonces reduced on the host (Python ints) only for the sample; the rest use a cheap valid stand-in
    nonce = _synth(n, 0xC33)[0]
    nonce[sample] = V.scalars(nonce_s)
    u, R_, c = engine.sign(sk, msg, nonce)
    pk = engine.keygen(sk)
    ok, c2 = engine.verify(pk, u, R_, msg)
    assert ok.all() and (c2 == c).all()
    uc, Rc, cc = ref_cpu.sign(sk[sample], msg[sample], nonce[sample])
    assert (uc == u[sample]).all() and (Rc == R_[sample]).all() and (cc == c[sample]).all()


def test_config4_vargen_verify_2_22_ten_percent_corrupted(engine):
    n = 1 << 22
    sk, nonce, msg = _synth(n, 0xC4)
    gscal = _synth(n, 0xC44)[0]
    gen = engine.keygen(gscal)                       # gen_i = s_i * G   (SecretKeyVarGen::random)
    pk = engine.keygen_vargen(sk, gen)
    u, R_, c = engine.sign_vargen(sk, gen, msg, nonce)
    idx = np.arange(n, dtype=np.int64)
    bad = (idx * 2654435761 % 10) == 0
    mode = (idx // 10) % 4
    u2, msg2, pk2, gen2 = u.copy(), msg.copy(), pk.copy(), gen.copy()
    u2[bad & (mode == 0), 0] ^= 1
    msg2[bad & (mode == 1), 0] ^= 1
    sel = bad & (mode == 2); pk2[sel] = np.roll(pk, -1, axis=0)[sel]
    sel = bad & (mode == 3); gen2[sel] = np.roll(gen, -1, axis=0)[sel]
    ok, _ = engine.verify_vargen(pk2, gen2, u2, R_, msg2)
    assert (ok == ~bad).all()
    assert 0.09 < bad.mean() < 0.11
    s = np.arange(0, n, 4093)  # strided over the whole batch (every chunk, late work items); odd: all four corruption kinds
    okc, _ = ref_cpu.verify_vargen(pk2[s], gen2[s], u2[s], R_[s], msg2[s])
    assert (okc == ok[s]).all()
    assert all((bad[s] & (mode[s] == k)).any() for k in range(4))


def test_multi_device_context_shards_without_collective():
    """a context over several devices splits by tuple index (one host thread per device, no collective): distinct
    ordinals when the box has more than one GPU, else device 0 listed twice (same split and threading logic)"""
    import torch
    from schnorr_b200 import Engine
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    e = Engine(devs, ark=o.ARK_RULE)
    n = 5000 + 7
    sk, nonce, msg = _synth(n, 9)
    pk = e.keygen(sk)
    u, R_, _ = e.sign(sk, msg, nonce)
    u[::3, 0] ^= 1
    ok, _ = e.verify(pk, u, R_, msg)
    assert ok.tolist() == [(i % 3) != 0 for i in range(n)]
    e.close()


def test_cpp_api_mirror_runs_reference_tests():
    """include/schnorr_b200.hpp (the C++ host layer above the C ABI) re-runs the reference's tests on the GPU;
    its seeded outputs must equal the oracle's bytes."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "test_api_cpp")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe, os.path.join(root, "tests", "cpp", "test_api.cpp"),
                           "-L" + os.path.join(root, "schnorr_b200"), "-lschnorr_b200",
                           "-Wl,-rpath," + os.path.join(root, "schnorr_b200")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "ALL OK" in out.stdout
    kv = dict(l.split("=", 1) for l in out.stdout.splitlines() if "=" in l)
    rng = o.StdRng.seed_from_u64(2321)
    sk, m = rng.random_fr(), rng.random_fq()
    u, Rp, _ = o.sign(sk, rng.random_fr(), m, mul=V.mul)
    assert kv["sk"] == sk.to_bytes(32, "little").hex() and kv["msg"] == m.to_bytes(32, "little").hex()
    assert kv["pk"] == o.affine_to_bytes(V.mul(o.G, sk)).hex()
    assert kv["sig"] == (u.to_bytes(32, "little") + o.affine_to_bytes(Rp)).hex()
    rng = o.StdRng.seed_from_u64(2321)
    sk, m = rng.random_fr(), rng.random_fq()
    u, Rp, Rpp, _ = o.sign_double(sk, rng.random_fr(), m, mul=V.mul)
    assert kv["sig_double"] == (u.to_bytes(32, "little") + o.affine_to_bytes(Rp) + o.affine_to_bytes(Rpp)).hex()
    rng = o.StdRng.seed_from_u64(2321)
    sk, s = rng.random_fr(), rng.random_fr()
    gen = V.mul(o.G, s)
    m = rng.random_fq()
    u, Rp, _ = o.sign_vargen(sk, gen, rng.random_fr(), m, mul=V.mul)
    assert kv["vargen_generator"] == o.affine_to_bytes(gen).hex()
    assert kv["sig_vargen"] == (u.to_bytes(32, "little") + o.affine_to_bytes(Rp)).hex()


@pytest.mark.parametrize("scheme", [0, 1, 2], ids=["single", "double", "vargen"])
def test_sign_witness_rows_match_oracle(engine, scheme):
    """SURVEY 8(f) row 4: the values Signature*::append and gadgets::verify_signature* allocate
    (/root/reference/src/signatures.rs:97-103, src/gadgets.rs:48-68), one row per signature"""
    import random
    rnd = random.Random(60 + scheme)
    n = 37
    Q, R = o.Q, o.R
    sk, nonce, msg = ([rnd.randrange(1, R) for _ in range(n)], [rnd.randrange(R) for _ in range(n)], [rnd.randrange(Q) for _ in range(n)])
    msg[0], msg[1] = 0, Q - 1
    gens = [V.mul(o.G, rnd.randrange(1, R)) for _ in range(n)]
    zs = [rnd.randrange(1, Q) for _ in range(n)]
    rows = engine.sign_witness(scheme, V.scalars(sk), V.fqs(msg), V.scalars(nonce),
                               gen=V.points(gens, zs) if scheme == 2 else None, affine=False)
    assert rows.shape == (n, (11, 19, 13)[scheme], 8)
    for i in range(n):
        got = [V.unmont(rows[i, k]) for k in range(rows.shape[1])]
        if scheme == 0:
            u, Rp, c = o.sign(sk[i], nonce[i], msg[i], mul=V.mul)
            pk = V.mul(o.G, sk[i])
            sa, sb = V.mul(o.G, u), V.mul(pk, c)
            want = [u, *Rp, *pk, msg[i], c, *sa, *sb]
            assert o.pt_add(sa, sb) == Rp
        elif scheme == 1:
            u, Rp, Rpp, c = o.sign_double(sk[i], nonce[i], msg[i], mul=V.mul)
            pk, pkp = V.mul(o.G, sk[i]), V.mul(o.G_NUMS, sk[i])
            want = [u, *Rp, *Rpp, *pk, *pkp, msg[i], c, *V.mul(o.G, u), *V.mul(pk, c), *V.mul(o.G_NUMS, u), *V.mul(pkp, c)]
        else:
            u, Rp, c = o.sign_vargen(sk[i], gens[i], nonce[i], msg[i], mul=V.mul)
            pk = V.mul(gens[i], sk[i])
            want = [u, *Rp, *pk, *gens[i], msg[i], c, *V.mul(gens[i], u), *V.mul(pk, c)]
        assert got == want, (scheme, i)
