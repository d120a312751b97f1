#!/usr/bin/env python3
"""Generate schnorr_b200/csrc/constants_gen.cuh -- the field / curve constants the CUDA path bakes in.

Product-side tool (does NOT import oracle/): the derivations are restated here so the kernels
and the test oracle are independent.  tests/test_abi_and_constants.py cross-checks the two.

What is baked: the two field moduli and their Montgomery constants, the curve constant d, square-root
tables, and the DEFAULT coordinates of the two generators.  What is NOT baked any more: the Hades round
constants, the MDS matrix and the sparse factorisation of the partial rounds -- those are inputs of
`sb200_init_ex` (include/schnorr_b200.h `sb200_params`) and are derived at context creation by
csrc/params_host.cuh.  This file keeps the Python twin of that derivation (`hades_tables(rule)`, and
`int_layer_tables` for the small-integer layers), which tests/test_params.py and tests/test_hades_cauchy.py compare
bit-for-bit with what the library derives, and emits the tables of the
compiled-out FP64 experiment (csrc/experimental/constants_fd_gen.cuh).

Round-constant rule (`--ark`, SURVEY.md 8(c) recall-risk item 1; both recalled from dusk-hades assets/HOWTO.md):
    cumsum (default)  p = 1;  c_i = from_bytes_wide(SHA512^(i+1)(seed)) + p;  p = c_i
    plain             c_i = from_bytes_wide(SHA512^(i+1)(seed))

Field elements are emitted as 8 x u32 little-endian limbs in Montgomery form (x * 2^256 mod p), the layout the
kernels compute in and the same bit pattern as dusk_bls12_381::BlsScalar's internal [u64; 4].

Usage:  python tools/gen_constants.py [--ark cumsum|plain]     (rewrites the headers in place)
"""
import hashlib
import os

Q = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
R = 0x0E7DB4EA6533AFA906673B0101343B00A6682093CCC81082D0970E5ED6F72CB7
RADIX = 1 << 256
WIDTH, FULL, PARTIAL = 5, 8, 59
P = WIDTH - 1  # index of the word that gets the S-box in partial rounds (dusk-hades: the LAST word)


def limbs(x):
    return [(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)]


def mont(x, p=Q):
    return x * RADIX % p


def fmt(x):
    return "{" + ", ".join("0x%08xu" % w for w in limbs(x)) + "}"


def inv(x):
    return pow(x, -1, Q)


# ---- FP64-pipe representation (csrc/fd.cuh): 5 x 52-bit limbs, Montgomery radix 2^260 ------------
RADIX260 = 1 << 260


def limbs52(x):
    return [(x >> (52 * i)) & ((1 << 52) - 1) for i in range(5)]


def m260(x):
    return x * RADIX260 % Q


def fmt_d(x):  # operand form: limbs as exactly representable doubles
    return "{" + ", ".join("%d.0" % w for w in limbs52(x)) + "}"


def fmt_u(x):  # integer form
    return "{" + ", ".join("0x%013xull" % w for w in limbs52(x)) + "}"


# ---- Hades252 (dusk-hades): round constants and MDS --------------------------------------
ARK_RULES = ("cumsum", "plain")
DEFAULT_ARK = "cumsum"


def round_constants(rule=DEFAULT_ARK):
    assert rule in ARK_RULES
    out, b, p = [], b"poseidon-for-plonk", 1
    for _ in range(960):
        b = hashlib.sha512(b).digest()
        c = int.from_bytes(b, "little") % Q
        if rule == "cumsum":
            c = (c + p) % Q
            p = c
        out.append(c)
    return out


RC = round_constants()
MDS = [[inv(i + j + WIDTH) for j in range(WIDTH)] for i in range(WIDTH)]


def set_ark(rule):
    global RC
    RC = round_constants(rule)


# ---- small exact linear algebra over F_q ---------------------------------------------------
def mat_mul(a, b):
    n, m, k = len(a), len(b[0]), len(b)
    return [[sum(a[i][t] * b[t][j] for t in range(k)) % Q for j in range(m)] for i in range(n)]


def mat_vec(a, v):
    return [sum(a[i][j] * v[j] for j in range(len(v))) % Q for i in range(len(a))]


def mat_inv(a):
    n = len(a)
    m = [list(row) + [1 if i == j else 0 for j in range(n)] for i, row in enumerate(a)]
    for c in range(n):
        piv = next(r for r in range(c, n) if m[r][c] % Q)
        m[c], m[piv] = m[piv], m[c]
        iv = inv(m[c][c])
        m[c] = [x * iv % Q for x in m[c]]
        for r in range(n):
            if r != c and m[r][c]:
                f = m[r][c]
                m[r] = [(x - f * y) % Q for x, y in zip(m[r], m[c])]
    return [row[n:] for row in m]


def ident(n):
    return [[1 if i == j else 0 for j in range(n)] for i in range(n)]


# ---- sparse factorisation of the 59 partial rounds -----------------------------------------
# Partial round t (t = 0..58):  x <- M * S_P(x + c_t), S_P = x^5 on word P only.
# Write x = (others o in F^4, p in F).  Any matrix of the form L = diag-block(Mhat on `others`,
# 1 on word P) commutes with S_P and with "add a constant" up to changing the constant.
# Factor M = L_t' * Sp_t where Sp_t is sparse (identity on `others` except column/row P); push the
# dense block forward into the next round's matrix.  After the 59 rounds one dense 5x5 matrix
# remains; it is applied once.  Algebraically identical to the dense rounds => bit-exact.
#
# Emitted form, executed by the kernel for t = 0..58 on a state y:
#     y[P] = (y[P] + k_t)^5
#     newP = sum_j row_t[j] * y[j]                (5 products, one word)
#     y[j] = y[j] + col_t[j] * y[P]   (j != P)    (4 products)       [uses the post-S-box y[P]]
#     y[P] = newP
# preceded by   y += pre_add   (vector; folds the `others` parts of all 59 round keys)
# and followed by   y = POST * y   (dense, once).
def build_sparse_partial():
    others = [i for i in range(WIDTH) if i != P]
    consts = [RC[(FULL // 2 + t) * WIDTH:(FULL // 2 + t + 1) * WIDTH] for t in range(PARTIAL)]
    B = ident(WIDTH - 1)  # acts on `others`
    # Invariant before round t: true state x = (B_t y_o ; y_P), B_0 = I.  With the MDS split into
    # (others, P) blocks M = [[Moo, Mop], [Mpo, Mpp]], z = (y_P + c_P)^5 and f_t = B_t^-1 c_o(t):
    #     y_next_P = (Mpo B_t) (y_o + f_t) + Mpp z          -> row_t = Mpo B_t (and Mpp on word P)
    #     y_next_o = (y_o + f_t) + B_{t+1}^-1 Mop z         -> col_t,  B_{t+1} = Moo B_t
    # The `others` never mix among themselves, so all folds f_t are added up-front as
    # Ftot = sum_t f_t; the excess E_t = Ftot - sum_{s<=t} f_s pollutes only y_next_P by row_t . E_t,
    # which is subtracted from the next round's key on word P (E_58 = 0).
    Moo = [[MDS[i][j] for j in others] for i in others]
    Mop = [MDS[i][P] for i in others]
    Mpo = [MDS[P][j] for j in others]
    Mpp = MDS[P][P]
    folds, ks, rows, cols = [], [], [], []
    Bs = [B]
    for t in range(PARTIAL):
        Bt = Bs[-1]
        Binv = mat_inv(Bt)
        c = consts[t]
        folds.append(mat_vec(Binv, [c[i] for i in others]))
        Bn = mat_mul(Moo, Bt)
        Bn_inv = mat_inv(Bn)
        cols.append(mat_vec(Bn_inv, Mop))
        rows.append(([sum(Mpo[k] * Bt[k][j] for k in range(WIDTH - 1)) % Q for j in range(WIDTH - 1)], Mpp))
        Bs.append(Bn)
    F = [[0] * (WIDTH - 1)]
    for t in range(PARTIAL):
        F.append([(F[-1][k] + folds[t][k]) % Q for k in range(WIDTH - 1)])
    Ftot = F[-1]
    # kernel adds Ftot to y_o up-front.  At round t the exact y'_o should contain only F[t+1]; the excess
    # E_t = Ftot - F[t+1] sits in y_o and pollutes P_next by row_t . E_t ; it never pollutes `others`
    # (no mixing).  P_next then receives key c_P(t+1) before its S-box, so fold the correction there.
    # For the last round the correction is E_58 = 0.
    for t in range(PARTIAL):
        kP = consts[t][P]
        if t > 0:
            E = [(Ftot[k] - F[t][k]) % Q for k in range(WIDTH - 1)]
            kP = (kP - sum(rows[t - 1][0][k] * E[k] for k in range(WIDTH - 1))) % Q
        ks.append(kP)
    pre_add = [0] * WIDTH
    for idx, i in enumerate(others):
        pre_add[i] = Ftot[idx]
    # POST = blockdiag(B_59, 1)
    post = [[0] * WIDTH for _ in range(WIDTH)]
    for a_, i in enumerate(others):
        for b_, j in enumerate(others):
            post[i][j] = Bs[-1][a_][b_]
    post[P][P] = 1
    row_full, col_full = [], []
    for t in range(PARTIAL):
        rw = [0] * WIDTH
        for idx, j in enumerate(others):
            rw[j] = rows[t][0][idx]
        rw[P] = rows[t][1]
        cl = [0] * WIDTH
        for idx, j in enumerate(others):
            cl[j] = cols[t][idx]
        row_full.append(rw)
        col_full.append(cl)
    return pre_add, ks, row_full, col_full, post


def hades_dense(state):
    s, ci = list(state), 0
    for rnd in range(FULL + PARTIAL):
        s = [(x + RC[ci + k]) % Q for k, x in enumerate(s)]
        ci += WIDTH
        if rnd < FULL // 2 or rnd >= FULL // 2 + PARTIAL:
            s = [pow(x, 5, Q) for x in s]
        else:
            s[P] = pow(s[P], 5, Q)
        s = mat_vec(MDS, s)
    return s


def hades_sparse(state, sp):
    pre_add, ks, rows, cols, post = sp
    s, ci = list(state), 0
    for rnd in range(FULL // 2):
        s = [pow((x + RC[ci + k]) % Q, 5, Q) for k, x in enumerate(s)]
        ci += WIDTH
        s = mat_vec(MDS, s)
    s = [(x + a) % Q for x, a in zip(s, pre_add)]
    for t in range(PARTIAL):
        s[P] = pow((s[P] + ks[t]) % Q, 5, Q)
        newp = sum(rows[t][j] * s[j] for j in range(WIDTH)) % Q
        for j in range(WIDTH):
            if j != P:
                s[j] = (s[j] + cols[t][j] * s[P]) % Q
        s[P] = newp
    s = mat_vec(post, s)
    ci += WIDTH * PARTIAL
    for rnd in range(FULL // 2):
        s = [pow((x + RC[ci + k]) % Q, 5, Q) for k, x in enumerate(s)]
        ci += WIDTH
        s = mat_vec(MDS, s)
    return s


def hades_tables(rule=DEFAULT_ARK):
    """The tables csrc/params_host.cuh derives at context creation, as Montgomery integers in the library's layout:
    rc[335], mds[25], pre[5], sparse[59 * 11] (key, row[5], col[5] with col[P] = 0), post[25]."""
    set_ark(rule)
    pre_add, ks, rows, cols, post = build_sparse_partial()
    sparse = []
    for t in range(PARTIAL):
        sparse += [ks[t]] + rows[t] + cols[t]
    out = {"rc": RC[:(FULL + PARTIAL) * WIDTH], "mds": [MDS[i][j] for i in range(WIDTH) for j in range(WIDTH)],
           "pre": pre_add, "sparse": sparse, "post": [post[i][j] for i in range(WIDTH) for j in range(WIDTH)]}
    return {k: [mont(x) for x in v] for k, v in out.items()}


INT_LAYER_CMAX_BOUND = (1 << 20) // 5  # max C below this <=> 5 * max C * 2^32 < 2^52 (a layer column fits a double)


def int_layer_matrix(mds):
    """(L, C) with C = L * mds a matrix of small integers, if mds qualifies for the small-integer layers, else None
    (twin of csrc/params_host.cuh derive_int_tables)."""
    import math
    d = []
    for row in mds:
        for x in row:
            v = inv(x) if x % Q else 0
            if not 0 < v < INT_LAYER_CMAX_BOUND:
                return None
            d.append(v)
    L = 1
    for v in d:
        L = math.lcm(L, v)
        if L >= 1 << 32:
            return None
    C = [[L // d[k * WIDTH + j] for j in range(WIDTH)] for k in range(WIDTH)]
    if max(max(r) for r in C) >= INT_LAYER_CMAX_BOUND:
        return None
    return L, C


def int_layer_tables(rc=None, mds=None):
    """The small-integer tables (cmat, src, fix, unscale) for the given round constants / MDS (plain integers),
    scaled values as Montgomery integers; None when the MDS does not qualify."""
    rc, mds = (RC if rc is None else rc), (MDS if mds is None else mds)
    lc = int_layer_matrix(mds)
    if lc is None:
        return None
    L, C = lc
    tau, src, fix = 1, [], []
    for rnd in range(FULL + PARTIAL):
        src += [tau * rc[rnd * WIDTH + k] % Q for k in range(WIDTH)]
        if rnd < FULL // 2 or rnd >= FULL // 2 + PARTIAL:
            tau = pow(tau, 5, Q)
        else:
            fix.append(inv(pow(tau, 4, Q)))
        tau = tau * L % Q
    return {"cmat": [C[k][j] for k in range(WIDTH) for j in range(WIDTH)], "src": [mont(x) for x in src],
            "fix": [mont(x) for x in fix], "unscale": [mont(inv(tau))]}


def hades_int(state, tabs):
    """The permutation as hades.cuh hades_perm_int runs it (plain integers in and out)."""
    C = [tabs["cmat"][k * WIDTH:(k + 1) * WIDTH] for k in range(WIDTH)]
    unm = lambda x: x * pow(RADIX, -1, Q) % Q
    s = list(state)
    for rnd in range(FULL + PARTIAL):
        s = [(x + unm(tabs["src"][rnd * WIDTH + k])) % Q for k, x in enumerate(s)]
        if rnd < FULL // 2 or rnd >= FULL // 2 + PARTIAL:
            s = [pow(x, 5, Q) for x in s]
        else:
            s[P] = pow(s[P], 5, Q) * unm(tabs["fix"][rnd - FULL // 2]) % Q
        s = [sum(C[k][j] * s[j] for j in range(WIDTH)) % Q for k in range(WIDTH)]
    return [x * unm(tabs["unscale"][0]) % Q for x in s]


def main():
    import argparse
    import random
    ap = argparse.ArgumentParser()
    ap.add_argument("--ark", default=DEFAULT_ARK, choices=ARK_RULES)
    rule = ap.parse_args().ark
    set_ark(rule)
    sp = build_sparse_partial()
    rnd = random.Random(7)
    for _ in range(8):
        st = [rnd.randrange(Q) for _ in range(WIDTH)]
        assert hades_dense(st) == hades_sparse(st, sp), "sparse Hades factorisation is not exact"
    assert hades_dense([0] * 5) == hades_sparse([0] * 5, sp)
    it = int_layer_tables()
    assert it is not None and all(hades_dense(s) == hades_int(s, it) for s in ([0] * 5, [Q - 1] * 5, list(range(5)))), \
        "small-integer Hades form is not exact"
    pre_add, ks, rows, cols, post = sp

    D = (-10240 * inv(10241)) % Q
    G = (0x3FD2814C43AC65A6F1FBF02D0FD6CCE62E3EBB21FD6C54ED4DF7B7FFEC7BEACA, 0x12)
    GP = (0x5E67B8F316F414F7BD9514C773FD4456931E316A39FE4541921710179DF76377,
          0x43D80EB3B2F3EB1B7B162DBEEB3B34FD9949BA0F82A5507A6705B707162E3EF8)
    for (u, v) in (G, GP):
        assert (-u * u + v * v - 1 - D * u * u * v * v) % Q == 0

    o = []
    w = o.append
    w("// GENERATED by tools/gen_constants.py -- do not edit.  Montgomery form (x * 2^256 mod p), 8 x u32 LE limbs.")
    w("#pragma once")
    w("#include <cstdint>")
    w("namespace sb200 {")
    w("// q = BLS12-381 scalar field (dusk_bls12_381::BlsScalar); r = JubJub scalar field (dusk_jubjub::JubJubScalar)")
    w("#define SB200_FQ_MOD_INIT %s" % fmt(Q))
    w("#define SB200_FR_MOD_INIT %s" % fmt(R))
    w("#define SB200_8R_INIT %s   // 8 r = the order of the whole curve group (cofactor 8)" % fmt(8 * R))
    w("#define SB200_FQ_ONE_INIT %s   // 2^256 mod q" % fmt(RADIX % Q))
    w("#define SB200_FQ_R2_INIT %s    // 2^512 mod q" % fmt(RADIX * RADIX % Q))
    # fq_sqr reduces every row with m + 1 = 2^32 - t0 and leaves out the part of (m + 1) q that does not depend on t0,
    # 2^32 + (q >> 64) 2^64 per row.  It feeds the sum of those parts over its 8 rows into its window instead, as
    # K = that sum + l q with l < 2^224 chosen so that limbs 0..6 of K are zero (l q only adds l < 2^224 to M).
    K = sum(((1 << 32) + ((Q >> 64) << 64)) << (32 * i) for i in range(8))
    K += (-K * pow(Q, -1, 1 << 224)) % (1 << 224) * Q
    assert K % (1 << 224) == 0 and K >> 480 == 0
    w("#define SB200_FQ_SQR_K_INIT {%s}   // fq_sqr's row constants (limbs 0..15)"
      % ", ".join("0x%08xu" % ((K >> (32 * i)) & 0xFFFFFFFF) for i in range(16)))
    w("#define SB200_FR_R2_INIT %s    // 2^512 mod r" % fmt(RADIX * RADIX % R))
    w("#define SB200_FR_NINV 0x%08xu  // -r^-1 mod 2^32" % ((-pow(R, -1, 1 << 32)) % (1 << 32)))
    w("#define SB200_FQ_NINV 0x%08xu  // -q^-1 mod 2^32" % ((-pow(Q, -1, 1 << 32)) % (1 << 32)))
    w("// JubJub  -u^2 + v^2 = 1 + d u^2 v^2,  d = -10240/10241 (dusk-jubjub EDWARDS_D)")
    w("#define SB200_ED_D_INIT %s" % fmt(mont(D)))
    w("#define SB200_ED_2D_INIT %s" % fmt(mont(2 * D % Q)))
    w("// dusk_jubjub::GENERATOR and GENERATOR_NUMS, affine (u, v): DEFAULTS of sb200_default_params (inputs of sb200_init_ex)")
    w("#define SB200_G_U_INIT %s" % fmt(mont(G[0])))
    w("#define SB200_G_V_INIT %s" % fmt(mont(G[1])))
    w("#define SB200_GP_U_INIT %s" % fmt(mont(GP[0])))
    w("#define SB200_GP_V_INIT %s" % fmt(mont(GP[1])))
    # Tonelli-Shanks data for F_q (q - 1 = 2^32 * t, t odd): 2^32-th primitive root g = 7^t (7 is a generator,
    # as in dusk-bls12_381's ROOT_OF_UNITY derivation; any primitive root gives the same decompressed point
    # because the sign bit picks the root) and the exponent (t - 1) / 2.
    t_odd = (Q - 1) >> 32
    assert t_odd & 1 and pow(7, (Q - 1) // 2, Q) == Q - 1
    g_root = pow(7, t_odd, Q)
    assert pow(g_root, 1 << 31, Q) == Q - 1
    w("// Tonelli-Shanks in F_q: 2-adicity 32, g = 7^t primitive 2^32-th root of unity, e = (t-1)/2")
    w("#define SB200_FQ_ROOT_OF_UNITY_INIT %s" % fmt(mont(g_root)))
    w("#define SB200_FQ_SQRT_EXP_INIT %s   // (t - 1) / 2, plain integer" % fmt((t_odd - 1) // 2))
    w("#define SB200_FQ_SQRT_EXP_BITS %d" % ((t_odd - 1) // 2).bit_length())
    # Inverse square root with a table-driven discrete logarithm in the 2^32-order subgroup (csrc/wire.cuh):
    #   y^(-(t+1)/2) by one exponentiation, then Pohlig-Hellman over eight 4-bit digits of k where y^-t = g^k.
    isqrt_exp = (Q - 1) - (t_odd + 1) // 2
    assert pow(5, isqrt_exp, Q) == pow(pow(5, (t_odd + 1) // 2, Q), -1, Q)
    w("// y^ISQRT_EXP = y^(-(t+1)/2); digit tables: W[d] = g^(d 2^28), P[i][d] = g^(-d 16^i), Q[i][d] = g^(-d 16^i / 2)")
    w("#define SB200_FQ_ISQRT_EXP_INIT %s   // q - 1 - (t + 1)/2, plain integer" % fmt(isqrt_exp))
    w("#define SB200_FQ_ISQRT_EXP_BITS %d" % isqrt_exp.bit_length())
    omega = pow(g_root, 1 << 28, Q)
    ginv = pow(g_root, -1, Q)
    w("#define SB200_FQ_DLOG_W_INIT { \\")
    for d in range(16):
        w("  %s, \\" % fmt(mont(pow(omega, d, Q))))
    w("}")
    w("#define SB200_FQ_DLOG_P_INIT { \\")
    for i in range(8):
        for d in range(16):
            w("  %s, \\" % fmt(mont(pow(ginv, d * 16 ** i, Q))))
    w("}")
    w("#define SB200_FQ_DLOG_Q_INIT { \\")
    for i in range(8):
        for d in range(16):
            ex = d * 16 ** i
            w("  %s, \\" % fmt(mont(pow(ginv, ex // 2, Q) if ex % 2 == 0 else 1)))  # odd total exponent: non-residue, caught by the final check
    w("}")
    w("}  // namespace sb200")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "schnorr_b200", "csrc", "constants_gen.cuh")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        f.write("\n".join(o) + "\n")
    print("wrote", os.path.normpath(path))

    # ---- tables of the compiled-out FP64 experiment (csrc/experimental/), under the selected round-constant rule ----
    o = []
    w = o.append
    w("// GENERATED by tools/gen_constants.py --ark %s -- do not edit.  Tables of the FP64-pipe experiment (SB_EXPERIMENTAL_FD)." % rule)
    w("#pragma once")
    w("#include <cstdint>")
    w("namespace sb200 {")
    w("// FP64-pipe field arithmetic (csrc/fd.cuh): 5 x 52-bit limbs, Montgomery radix 2^260")
    w("#define SB200_FD_Q_D_INIT %s" % fmt_d(Q))
    w("#define SB200_FD_Q_U_INIT %s" % fmt_u(Q))
    w("#define SB200_FD_KIN_D_INIT %s   // 2^264 mod q: mont260(x * 2^256, .) = x * 2^260" % fmt_d((1 << 264) % Q))
    w("#define SB200_FD_ONE_U_INIT %s   // 2^260 mod q" % fmt_u(RADIX260 % Q))
    assert Q % (1 << 52) == (1 << 52) - (1 << 32) + 1 and (Q * (1 + (1 << 32))) % (1 << 52) == 1
    w("// Hades252 tables for hades_fd.cuh, Montgomery-2^260: 9 groups of 5 additive words")
    groups = [RC[0:5], RC[5:10], RC[10:15], RC[15:20], list(pre_add[:4]) + [ks[0]],
              RC[63 * 5:64 * 5], RC[64 * 5:65 * 5], RC[65 * 5:66 * 5], RC[66 * 5:67 * 5]]
    w("#define SB200_FDH_ADD_INIT { \\")
    for g in groups:
        for x in g:
            w("  %s, \\" % fmt_u(m260(x)))
    w("}")
    w("#define SB200_FDH_MDS_INIT { \\")
    for i in range(WIDTH):
        for j in range(WIDTH):
            w("  %s, \\" % fmt_d(m260(MDS[i][j])))
    w("}")
    w("#define SB200_FDH_POST_INIT { \\")
    for i in range(WIDTH):
        for j in range(WIDTH):
            w("  %s, \\" % fmt_d(m260(post[i][j])))
    w("}")
    w("// per sparse round t: the key of round t + 1 (carried by the row product), then row[0..4], col[0..3]")
    w("#define SB200_FDH_SP_ADD_INIT { \\")
    for t in range(PARTIAL):
        w("  %s, \\" % (fmt_u(m260(ks[t + 1])) if t + 1 < PARTIAL else fmt_u(0)))
    w("}")
    w("#define SB200_FDH_SP_MAT_INIT { \\")
    for t in range(PARTIAL):
        for j in range(WIDTH):
            w("  %s, \\" % fmt_d(m260(rows[t][j])))
        for j in range(WIDTH - 1):
            w("  %s, \\" % fmt_d(m260(cols[t][j])))
    w("}")
    w("}  // namespace sb200")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "schnorr_b200", "csrc", "experimental", "constants_fd_gen.cuh")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        f.write("\n".join(o) + "\n")
    print("wrote", os.path.normpath(path))


if __name__ == "__main__":
    main()
