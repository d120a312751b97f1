"""Pin the oracle: self-validating constants, known-answer vectors of its RNG, the fingerprints recorded in
SURVEY.md 8(c), and agreement between its three formulations (affine ladder / fast projective / C restatement)."""
import random

import pytest

import numpy as np

import ref_cpu
import schnorr_oracle as o
import vectors as V

Q, R = o.Q, o.R


def test_field_and_curve_constants():
    assert pow(2, Q - 1, Q) == 1 and pow(2, R - 1, R) == 1 and Q.bit_length() == 255 and R.bit_length() == 252
    assert (1 << 250) < R
    assert o.D == 0x2A9318E74BFA2B48F5FD9207E6BD7FD4292D7F6D37579D2601065FD6D6343EB1
    assert pow(o.D, (Q - 1) // 2, Q) == Q - 1 and pow(Q - 1, (Q - 1) // 2, Q) == 1  # d non-square, -1 square: complete law
    for P in (o.G, o.G_NUMS):
        assert o.on_curve(P)
        assert o.pt_mul_fast(P, R) == o.IDENTITY and o.pt_mul_fast(P, 8) != o.IDENTITY
    assert o.G_NUMS not in (o.G, o.pt_neg(o.G))


def test_chacha_and_stdrng_known_answers():
    # ChaCha20, all-zero key/nonce, block 0 (the classic test vector) -- validates the block function
    assert o.chacha_block([0] * 8, 0, 0, rounds=20).hex() == (
        "76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7"
        "da41597c5157488d7724e03fb8d84a376a43b8f41518a11cc387b669b2ee6586")
    # ChaCha12, same inputs (draft-strombergson-chacha-test-vectors TC1, 12 rounds)
    assert o.chacha_block([0] * 8, 0, 0, rounds=12).hex().startswith("9bf49a6a0755f953811fce125f2683d50429c3bb49e07414")
    # rand 0.8 `test_stdrng_construction`: from_seed -> next_u64, then from_rng -> next_u64
    seed = bytes([1, 0, 0, 0, 23, 0, 0, 0, 200, 1, 0, 0, 210, 30, 0, 0] + [0] * 16)
    rng0 = o.StdRng(seed)
    assert rng0.next_u64() == 10719222850664546238
    rng1 = o.StdRng(rng0.fill_bytes(32))
    assert rng1.next_u64() == 14064965282130556830


def test_round_constant_rules():
    """the two recalled forms of dusk-hades' ark.bin: "cumsum" is the running sum of "plain", seeded with one"""
    plain, cumsum = o._round_constants("plain"), o._round_constants("cumsum")
    assert cumsum[0] == (plain[0] + 1) % Q
    assert all(cumsum[i] == (cumsum[i - 1] + plain[i]) % Q for i in range(1, 960))
    prev = o.set_ark_rule("plain")
    assert o.ROUND_CONSTANTS == plain
    o.set_ark_rule("cumsum")
    assert o.ROUND_CONSTANTS == cumsum and o.ARK_RULE == "cumsum"
    o.set_ark_rule(prev)


@pytest.fixture
def plain_rule():
    prev = o.set_ark_rule("plain")
    yield
    o.set_ark_rule(prev)


def test_poseidon_fingerprints(plain_rule):
    """SURVEY.md 8(c): these pin THIS restatement under the "plain" rule (drift detection), not the un-buildable crates."""
    assert o.ROUND_CONSTANTS[0] == 0x4929E824CAE3E5B6915AF89C2B2EF56233518DA79404494933A12BB7322DD246
    assert o.ROUND_CONSTANTS[1] == 0x16C704062C23752559D045399F2FC29CA7DB44D857DC2A6A7385F58EBA0D4801
    assert o.ROUND_CONSTANTS[334] == 0x069D59D29D2260B3510923EE9D8845734A67B558BAFD4BE62DCFC3CF34028BE9
    assert o.MDS[0][0] == pow(5, -1, Q) and o.MDS[4][4] == pow(13, -1, Q)
    assert o.hades_perm([0] * 5)[1] == 0x3A5B3B13DF69CA0F7708BB54D966C884D0D07394A00540A9F739B100CC021217
    assert o.sponge_hash([1, 2, 3]) == 0x6930089D9345A313BB691AC82F21B504AA4DFB0A6F9F4BC9519C89243E70B367
    assert o.truncated_hash([1, 2, 3]) == 0x0130089D9345A313BB691AC82F21B504AA4DFB0A6F9F4BC9519C89243E70B367
    assert o.sponge_hash([1, 2, 3, 4, 5]) == 0x6AE5A1CC67B5F6FE3D9A3F4BFC0289F653BD00262A10E31EBC0861132F83566E


def test_sponge_shapes():
    # 3 inputs = one permutation of [0, a, b, c, 1]; 5 inputs = two permutations with the padding rule
    a, b, c, d, e = 11, 22, 33, 44, 55
    assert o.sponge_hash([a, b, c]) == o.hades_perm([0, a, b, c, 1])[1]
    s = o.hades_perm([0, a, b, c, d])
    s[1] = (s[1] + e) % Q
    s[2] = (s[2] + 1) % Q
    assert o.sponge_hash([a, b, c, d, e]) == o.hades_perm(s)[1]
    # a full last chunk is followed by a padding-only permutation
    s = o.hades_perm([0, a, b, c, d])
    s[1] = (s[1] + 1) % Q
    assert o.sponge_hash([a, b, c, d]) == o.hades_perm(s)[1]


def test_ladder_equals_fast_mul():
    rnd = random.Random(3)
    for P in (o.G, o.G_NUMS, V.rand_curve_point(rnd), (0, Q - 1)):
        for k in (0, 1, 2, R - 1, (1 << 252) - 1, rnd.randrange(1 << 252)):
            assert o.pt_mul(P, k) == o.pt_mul_fast(P, k)


def test_compress_roundtrip_and_rejects():
    rnd = random.Random(4)
    for _ in range(20):
        P = V.rand_curve_point(rnd)
        assert o.affine_from_bytes(o.affine_to_bytes(P)) == P
    assert o.affine_from_bytes(Q.to_bytes(32, "little")) is None  # non-canonical v
    bad = next(v for v in range(2, 100) if o.affine_from_bytes(v.to_bytes(32, "little")) is None)
    assert bad  # some v are not on the curve
    assert o.scalar_from_bytes(R.to_bytes(32, "little")) is None and o.scalar_from_bytes((R - 1).to_bytes(32, "little")) == R - 1


def test_c_restatement_matches_python_oracle():
    rnd = random.Random(5)
    n = 24
    sk = [rnd.randrange(R) for _ in range(n)]
    nonce = [rnd.randrange(R) for _ in range(n)]
    m = [rnd.randrange(Q) for _ in range(n)]
    sk[0], nonce[0], m[0] = 0, 0, 0
    sk[1], nonce[1], m[1] = R - 1, R - 1, Q - 1
    u, Rr, c = ref_cpu.sign(V.scalars(sk), V.fqs(m), V.scalars(nonce))
    exp = [o.sign(a, b, mm) for a, b, mm in zip(sk, nonce, m)]  # the reference-shaped 252-step ladder
    assert V.ints_out(u) == [e[0] for e in exp] and V.points_out(Rr) == [e[1] for e in exp] and V.ints_out(c) == [e[2] for e in exp]
    pk = ref_cpu.keygen(V.scalars(sk))
    assert V.points_out(pk) == [o.keygen(a) for a in sk]
    uu = V.ints_out(u)
    uu[2] = (uu[2] + 1) % R
    ok, c2 = ref_cpu.verify(pk, V.scalars(uu), Rr, V.fqs(m))
    assert ok.tolist() == [i != 2 for i in range(n)] and V.ints_out(c2) == [e[2] for e in exp]
    zs = [rnd.randrange(1, Q) for _ in range(n)]
    okp, _ = ref_cpu.verify(V.points(V.points_out(pk), zs), V.scalars(uu), V.points(V.points_out(Rr), zs[::-1]), V.fqs(m), affine=False)
    assert okp.tolist() == ok.tolist()
    # double and var-generator variants
    u, Rr, Rp, c = ref_cpu.sign_double(V.scalars(sk), V.fqs(m), V.scalars(nonce))
    expd = [o.sign_double(a, b, mm, mul=V.mul) for a, b, mm in zip(sk, nonce, m)]
    assert V.ints_out(u) == [e[0] for e in expd] and V.points_out(Rp) == [e[2] for e in expd] and V.ints_out(c) == [e[3] for e in expd]
    pk, pkp = ref_cpu.keygen(V.scalars(sk), double=True)
    ok, _ = ref_cpu.verify_double(pk, pkp, u, Rr, Rp, V.fqs(m))
    assert ok.all()
    ok, _ = ref_cpu.verify_double(pk, pk, u, Rr, Rp, V.fqs(m))
    assert ok.tolist() == [a == 0 for a in sk]  # sk = 0: both keys are the identity
    gens = [V.mul(o.G, rnd.randrange(R)) for _ in range(n)]
    u, Rr, c = ref_cpu.sign_vargen(V.scalars(sk), V.points(gens), V.fqs(m), V.scalars(nonce))
    expv = [o.sign_vargen(a, g, b, mm, mul=V.mul) for a, g, b, mm in zip(sk, gens, nonce, m)]
    assert V.ints_out(u) == [e[0] for e in expv] and V.points_out(Rr) == [e[1] for e in expv]
    pkv = ref_cpu.keygen(V.scalars(sk), gen=V.points(gens))
    ok, _ = ref_cpu.verify_vargen(pkv, V.points(gens), u, Rr, V.fqs(m))
    assert ok.all()


def _whole_curve_cases(rnd, n):
    """points the scale tests hand to ref_cpu: prime-order multiples, whole-curve points, sk G + torsion, the
    small-order points and the identity"""
    tors = V.torsion_points()
    out = []
    for i in range(n):
        k = i % 4
        if k == 0:
            out.append(V.mul(o.G, rnd.randrange(R)))
        elif k == 1:
            out.append(V.rand_curve_point(rnd))
        elif k == 2:
            out.append(o.pt_add(V.mul(o.G, rnd.randrange(R)), tors[i % len(tors)]))
        else:
            out.append(tors[(i // 4) % len(tors)])
    return out


def _maybe_proj(rnd, pts, proj):
    return V.points(pts, [rnd.randrange(1, Q) for _ in pts] if proj else None)


@pytest.mark.parametrize("proj", [False, True], ids=["affine", "projective"])
def test_c_restatement_on_the_whole_curve(proj):
    """ref_cpu is the reference the large GPU batches are judged by: pin its verdicts and challenges against the Python
    oracle on keys, nonce points and generators off the prime-order subgroup, small-order keys, the identity, (U : V : Z)
    inputs with random Z, and variable-generator tuples with u = r - 1"""
    rnd = random.Random(6 + proj)
    n = 144
    tors = V.torsion_points()
    # single-key: valid by construction on the prime-order part, so keys with a torsion part pass iff c T = O
    sk = [rnd.randrange(R) for _ in range(n)]
    nonce = [rnd.randrange(R) for _ in range(n)]
    m = [rnd.randrange(Q) for _ in range(n)]
    pk, u, Rr = [], [], []
    for i in range(n):
        a, b, mm = sk[i], nonce[i], m[i]
        ui, Ri, _ = o.sign(a, b, mm, mul=V.mul)
        P = V.mul(o.G, a)
        k = i % 6
        if k == 1:
            P = o.pt_add(P, tors[i % len(tors)])
        elif k == 2:
            P, ui, Ri = tors[i % len(tors)], b, V.mul(o.G, b)  # small-order key with R = u G
        elif k == 3:
            Ri = o.pt_add(Ri, tors[(i + 3) % len(tors)])
        elif k == 4:
            P = V.rand_curve_point(rnd)
        elif k == 5:
            ui = (ui + 1) % R
        pk.append(P); u.append(ui); Rr.append(Ri)
    want = [o.verify(*t, mul=V.mul) for t in zip(pk, u, Rr, m)]
    ok, c = ref_cpu.verify(_maybe_proj(rnd, pk, proj), V.scalars(u), _maybe_proj(rnd, Rr, proj), V.fqs(m), affine=not proj)
    assert ok.tolist() == want and any(want[1::6]) and not all(want[1::6]) and any(want[2::6]) and not all(want[2::6])
    assert V.ints_out(c) == [o.challenge_hash(r_, mm) for r_, mm in zip(Rr, m)]
    # double-key over whole-curve points in every position
    P1, P2, R1, R2 = (_whole_curve_cases(rnd, n) for _ in range(4))
    for i in range(0, n, 3):  # a third valid by construction, some with a torsion part on one key only
        ui, R1[i], R2[i], _ = o.sign_double(sk[i], nonce[i], m[i], mul=V.mul)
        P1[i], P2[i], u[i] = V.mul(o.G, sk[i]), V.mul(o.G_NUMS, sk[i]), ui
        if i % 2:
            P2[i] = o.pt_add(P2[i], tors[i % len(tors)])
    want = [o.verify_double(*t, mul=V.mul) for t in zip(P1, P2, u, R1, R2, m)]
    ok, c = ref_cpu.verify_double(*(_maybe_proj(rnd, x, proj) for x in (P1, P2)), V.scalars(u),
                                  *(_maybe_proj(rnd, x, proj) for x in (R1, R2)), V.fqs(m), affine=not proj)
    assert ok.tolist() == want and any(want) and not all(want)
    assert V.ints_out(c) == [o.challenge_hash_double(a, b, mm) for a, b, mm in zip(R1, R2, m)]
    # variable generator: whole-curve generators and keys, and the forced-fallback lanes u = r - 1 (valid by construction)
    gens, pkv, Rv = (_whole_curve_cases(rnd, n) for _ in range(3))
    uv = [rnd.randrange(R) for _ in range(n)]
    for i in range(n):
        g = gens[i]
        if i % 3 == 0:
            uv[i], Rv[i], _ = o.sign_vargen(sk[i], g, nonce[i], m[i], mul=V.mul)
            pkv[i] = V.mul(g, sk[i])
        elif i % 3 == 1 and g != o.IDENTITY:
            k = rnd.randrange(1, R)
            Rv[i] = V.mul(g, k)
            c_ = o.challenge_hash(Rv[i], m[i])
            uv[i], pkv[i] = R - 1, V.mul(g, (k - (R - 1)) * pow(c_, -1, R) % R)
    want = [o.verify_vargen(*t, mul=V.mul) for t in zip(pkv, gens, uv, Rv, m)]
    ok, c = ref_cpu.verify_vargen(*(_maybe_proj(rnd, x, proj) for x in (pkv, gens)), V.scalars(uv), _maybe_proj(rnd, Rv, proj),
                                  V.fqs(m), affine=not proj)
    assert ok.tolist() == want and any(want) and not all(want)
    assert V.ints_out(c) == [o.challenge_hash(r_, mm) for r_, mm in zip(Rv, m)]


def test_c_restatement_reads_only_252_scalar_bits():
    """ref_cpu's multiplication walks bits 251..0 of u, as the reference's does, so it cannot judge a non-canonical u:
    its verdict on u >= r is the verdict on u mod 2^252.  The product rejects u >= r (JubJubScalar::from_bytes), so a
    GPU verdict is compared with ref_cpu's verdict AND u < r."""
    rnd = random.Random(9)
    n = 64
    sk, nonce, m = [rnd.randrange(R) for _ in range(n)], [rnd.randrange(R) for _ in range(n)], [rnd.randrange(Q) for _ in range(n)]
    for i in range(1, n, 8):  # u = nonce below 2^252 - r: u + r still fits the 252 bits
        sk[i], nonce[i] = 0, rnd.randrange((1 << 252) - R)
    sigs = [o.sign(a, b, mm, mul=V.mul) for a, b, mm in zip(sk, nonce, m)]
    pk = [V.mul(o.G, a) for a in sk]
    # u + r: bit 252 set or clear depending on u; u + r - 2^252 when set; the largest 256-bit values
    big = [s[0] + R for s in sigs]
    big[::8] = [(s[0] % (1 << 252)) | (0xF << 252) for s in sigs[::8]]  # same low 252 bits as a valid u
    ok, _ = ref_cpu.verify(V.points(pk), V.scalars(big), V.points([s[1] for s in sigs]), V.fqs(m))
    want = [o.verify(pk[i], big[i] % (1 << 252), sigs[i][1], m[i], mul=V.mul) for i in range(n)]
    assert ok.tolist() == want
    assert all(ok[::8]) and all(ok[1::8]) and not all(ok)  # so `& (u < r)` is what makes the expected verdict false
    assert all(b < (1 << 252) for b in big[1::8])
