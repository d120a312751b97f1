// Host-side handling of the scheme parameters (include/schnorr_b200.h: sb200_params, sb200_default_params,
// sb200_init_ex).  Everything the un-vendored dependency crates define numerically -- the Hades round constants and
// MDS matrix (dusk-hades `ROUND_CONSTANTS`, `MDS_MATRIX`), the two JubJub generators (dusk-jubjub `GENERATOR`,
// `GENERATOR_NUMS`) -- is an INPUT of context creation, not a baked constant: the values used at
// /root/reference/src/signatures.rs:133,283-289 and /root/reference/src/keys/public.rs:127,239 come from crates that
// cannot be built in this image (SURVEY.md 8(c)), so a host with the real crate hands over the crate's own tables
// (rust/src/cuda.rs `params_from_crate`) and nothing here has to be trusted.
//
// This file: (1) the published recipes for the defaults (SHA-512 chain for the round constants in both recalled forms,
// Cauchy MDS), (2) validation of supplied parameters, (3) the exact sparse factorisation of the 59 partial rounds that
// the kernels run (same algebra as tools/gen_constants.py build_sparse_partial, re-derived here at init because the
// inputs are only known then), (4) the small-integer form of the rounds when the MDS qualifies (derive_int_tables),
// (5) a self-check of the production form against the dense permutation.  Host code only; runs once per context.
#pragma once
#include <cstring>

#include "wire.cuh"

namespace sb200 {
namespace params {

// ---- SHA-512 (FIPS 180-4), for the round-constant recipe only --------------------------------------------------
struct Sha512 {
  static uint64_t rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
  static void digest(const uint8_t* msg, size_t len, uint8_t out[64]) {
    static const uint64_t K[80] = {
        0x428a2f98d728ae22ull, 0x7137449123ef65cdull, 0xb5c0fbcfec4d3b2full, 0xe9b5dba58189dbbcull, 0x3956c25bf348b538ull,
        0x59f111f1b605d019ull, 0x923f82a4af194f9bull, 0xab1c5ed5da6d8118ull, 0xd807aa98a3030242ull, 0x12835b0145706fbeull,
        0x243185be4ee4b28cull, 0x550c7dc3d5ffb4e2ull, 0x72be5d74f27b896full, 0x80deb1fe3b1696b1ull, 0x9bdc06a725c71235ull,
        0xc19bf174cf692694ull, 0xe49b69c19ef14ad2ull, 0xefbe4786384f25e3ull, 0x0fc19dc68b8cd5b5ull, 0x240ca1cc77ac9c65ull,
        0x2de92c6f592b0275ull, 0x4a7484aa6ea6e483ull, 0x5cb0a9dcbd41fbd4ull, 0x76f988da831153b5ull, 0x983e5152ee66dfabull,
        0xa831c66d2db43210ull, 0xb00327c898fb213full, 0xbf597fc7beef0ee4ull, 0xc6e00bf33da88fc2ull, 0xd5a79147930aa725ull,
        0x06ca6351e003826full, 0x142929670a0e6e70ull, 0x27b70a8546d22ffcull, 0x2e1b21385c26c926ull, 0x4d2c6dfc5ac42aedull,
        0x53380d139d95b3dfull, 0x650a73548baf63deull, 0x766a0abb3c77b2a8ull, 0x81c2c92e47edaee6ull, 0x92722c851482353bull,
        0xa2bfe8a14cf10364ull, 0xa81a664bbc423001ull, 0xc24b8b70d0f89791ull, 0xc76c51a30654be30ull, 0xd192e819d6ef5218ull,
        0xd69906245565a910ull, 0xf40e35855771202aull, 0x106aa07032bbd1b8ull, 0x19a4c116b8d2d0c8ull, 0x1e376c085141ab53ull,
        0x2748774cdf8eeb99ull, 0x34b0bcb5e19b48a8ull, 0x391c0cb3c5c95a63ull, 0x4ed8aa4ae3418acbull, 0x5b9cca4f7763e373ull,
        0x682e6ff3d6b2b8a3ull, 0x748f82ee5defb2fcull, 0x78a5636f43172f60ull, 0x84c87814a1f0ab72ull, 0x8cc702081a6439ecull,
        0x90befffa23631e28ull, 0xa4506cebde82bde9ull, 0xbef9a3f7b2c67915ull, 0xc67178f2e372532bull, 0xca273eceea26619cull,
        0xd186b8c721c0c207ull, 0xeada7dd6cde0eb1eull, 0xf57d4f7fee6ed178ull, 0x06f067aa72176fbaull, 0x0a637dc5a2c898a6ull,
        0x113f9804bef90daeull, 0x1b710b35131c471bull, 0x28db77f523047d84ull, 0x32caab7b40c72493ull, 0x3c9ebe0a15c9bebcull,
        0x431d67c49c100d4cull, 0x4cc5d4becb3e42b6ull, 0x597f299cfc657e2aull, 0x5fcb6fab3ad6faecull, 0x6c44198c4a475817ull};
    uint64_t h[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                     0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    uint8_t buf[256];  // messages here are <= 64 bytes: at most one padded 128-byte block (two for safety)
    size_t total = ((len + 17 + 127) / 128) * 128;
    if (total > sizeof(buf)) return;
    memset(buf, 0, total);
    memcpy(buf, msg, len);
    buf[len] = 0x80;
    uint64_t bits = (uint64_t)len * 8;
    for (int i = 0; i < 8; i++) buf[total - 1 - i] = (uint8_t)(bits >> (8 * i));
    for (size_t off = 0; off < total; off += 128) {
      uint64_t w[80];
      for (int i = 0; i < 16; i++) {
        uint64_t x = 0;
        for (int k = 0; k < 8; k++) x = (x << 8) | buf[off + 8 * i + k];
        w[i] = x;
      }
      for (int i = 16; i < 80; i++) {
        uint64_t s0 = rotr(w[i - 15], 1) ^ rotr(w[i - 15], 8) ^ (w[i - 15] >> 7);
        uint64_t s1 = rotr(w[i - 2], 19) ^ rotr(w[i - 2], 61) ^ (w[i - 2] >> 6);
        w[i] = w[i - 16] + s0 + w[i - 7] + s1;
      }
      uint64_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
      for (int i = 0; i < 80; i++) {
        uint64_t S1 = rotr(e, 14) ^ rotr(e, 18) ^ rotr(e, 41), ch = (e & f) ^ (~e & g);
        uint64_t t1 = hh + S1 + ch + K[i] + w[i];
        uint64_t S0 = rotr(a, 28) ^ rotr(a, 34) ^ rotr(a, 39), mj = (a & b) ^ (a & c) ^ (b & c);
        uint64_t t2 = S0 + mj;
        hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
      }
      h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    for (int i = 0; i < 8; i++)
      for (int k = 0; k < 8; k++) out[8 * i + k] = (uint8_t)(h[i] >> (56 - 8 * k));
  }
};

inline fq ld(const uint32_t* p) { fq r; memcpy(r.v, p, 32); return r; }
inline void st(uint32_t* p, const fq& a) { memcpy(p, a.v, 32); }
inline fq fq_small(uint32_t x) {  // Montgomery form of a small integer
  fq c = fq_zero();
  c.v[0] = x;
  return fq_to_mont(c);
}

// dusk-hades `ark.bin` (assets/HOWTO.md), first `n` constants, Montgomery limbs.
//   bytes = "poseidon-for-plonk"; repeat: bytes = SHA-512(bytes); h = BlsScalar::from_bytes_wide(bytes)
//   rule SB200_ARK_CUMSUM:  p = 1;  c_i = h_i + p;  p = c_i      (running sum seeded with one)
//   rule SB200_ARK_PLAIN :  c_i = h_i
// Both are recollections of an un-vendored crate (SURVEY.md 8(c) item 1); which one the real crate uses is settled
// by rust/tests/dump_golden.rs, and a caller with the crate passes ROUND_CONSTANTS itself.
inline void default_round_constants(int rule, uint32_t (*out)[8], int n) {
  uint8_t bytes[64];
  const char* seed = "poseidon-for-plonk";
  size_t len = strlen(seed);
  memcpy(bytes, seed, len);
  fq p = fq_one();
  for (int i = 0; i < n; i++) {
    uint8_t d[64];
    Sha512::digest(bytes, len, d);
    memcpy(bytes, d, 64);
    len = 64;
    uint32_t w[16];
    memcpy(w, d, 64);  // little-endian host (the ABI's limb layout already assumes it)
    fq h = fq_from_wide(w);
    if (rule == SB200_ARK_CUMSUM) {
      h = fq_add(h, p);
      p = h;
    }
    st(out[i], h);
  }
}

// dusk-hades `mds.bin`: Cauchy matrix 1 / (x_i + y_j), x_i = i, y_j = WIDTH + j
inline void default_mds(uint32_t (*out)[5][8]) {
  for (int i = 0; i < 5; i++)
    for (int j = 0; j < 5; j++) st(out[i][j], fq_inv(fq_small((uint32_t)(i + j + 5))));
}

// ---- 4x4 linear algebra over F_q (Montgomery values) ------------------------------------------------------------
struct Mat4 {
  fq a[4][4];
};
inline Mat4 mat_ident() {
  Mat4 m;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) m.a[i][j] = i == j ? fq_one() : fq_zero();
  return m;
}
inline Mat4 mat_mul(const Mat4& x, const Mat4& y) {
  Mat4 r;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      fq s = fq_zero();
      for (int k = 0; k < 4; k++) s = fq_add(s, fq_mul(x.a[i][k], y.a[k][j]));
      r.a[i][j] = s;
    }
  return r;
}
inline void mat_vec(const Mat4& m, const fq* v, fq* out) {
  for (int i = 0; i < 4; i++) {
    fq s = fq_zero();
    for (int k = 0; k < 4; k++) s = fq_add(s, fq_mul(m.a[i][k], v[k]));
    out[i] = s;
  }
}
inline bool mat_inv(const Mat4& m, Mat4& out) {  // Gauss-Jordan; false if singular
  fq w[4][8];
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 8; j++) w[i][j] = j < 4 ? m.a[i][j] : (j - 4 == i ? fq_one() : fq_zero());
  for (int c = 0; c < 4; c++) {
    int piv = -1;
    for (int r = c; r < 4 && piv < 0; r++)
      if (!fq_is_zero(w[r][c])) piv = r;
    if (piv < 0) return false;
    if (piv != c)
      for (int j = 0; j < 8; j++) { fq t = w[c][j]; w[c][j] = w[piv][j]; w[piv][j] = t; }
    fq iv = fq_inv(w[c][c]);
    for (int j = 0; j < 8; j++) w[c][j] = fq_mul(w[c][j], iv);
    for (int r = 0; r < 4; r++) {
      if (r == c || fq_is_zero(w[r][c])) continue;
      fq f = w[r][c];
      for (int j = 0; j < 8; j++) w[r][j] = fq_sub(w[r][j], fq_mul(f, w[c][j]));
    }
  }
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) out.a[i][j] = w[i][4 + j];
  return true;
}

// Small-integer form of the rounds (hades.cuh hades_perm_int).  The MDS qualifies when every entry is 1/d for an integer
// d and, with L = lcm of the d, the matrix C = L * MDS (C[k][j] = L / d[k][j]) keeps a five-term column of the layer
// exact in a double: 5 * max C * 2^32 < 2^52.  The state then runs at a scale tau (the kernels hold tau * x):
//   round r adds tau_r * rc[r];  a full S-box makes the scale tau_r^5;  in a partial round the S-box word is brought back
//   from tau_r^5 to tau_r by fix = tau_r^-4;  the layer C multiplies the scale by L;  at the end, unscale = tau_67^-1.
// Sets T.int_layers = 0 and leaves the other new fields zero when the MDS does not qualify.
constexpr uint32_t INT_LAYER_CMAX_BOUND = (1u << 20) / 5;  // max C < this  <=>  5 * max C * 2^32 < 2^52

inline void derive_int_tables(HadesTables& T) {
  constexpr int W = 5, NP = 59, NF = 4;
  memset(T.cmat, 0, sizeof(T.cmat));
  memset(T.src, 0, sizeof(T.src));
  memset(T.fix, 0, sizeof(T.fix));
  memset(T.unscale, 0, sizeof(T.unscale));
  T.int_layers = 0;
  uint64_t d[25], L = 1, cmax = 0;
  for (int e = 0; e < 25; e++) {
    const fq iv = fq_from_mont(fq_inv(ld(T.mds[e])));
    for (int i = 1; i < 8; i++)
      if (iv.v[i]) return;
    if (iv.v[0] == 0 || iv.v[0] >= INT_LAYER_CMAX_BOUND) return;
    d[e] = iv.v[0];
    uint64_t a = L, b = d[e];
    while (b) { uint64_t t = a % b; a = b; b = t; }
    L = L / a * d[e];
    if (L >= (1ull << 32)) return;
  }
  for (int e = 0; e < 25; e++) cmax = L / d[e] > cmax ? L / d[e] : cmax;
  if (cmax >= INT_LAYER_CMAX_BOUND) return;
  for (int e = 0; e < 25; e++) T.cmat[e] = (double)(L / d[e]);
  const fq Lf = fq_small((uint32_t)L);
  fq tau = fq_one();
  for (int r = 0; r < 2 * NF + NP; r++) {
    for (int k = 0; k < W; k++) st(T.src[r * W + k], fq_mul(ld(T.rc[r * W + k]), tau));
    if (r < NF || r >= NF + NP) {
      tau = fq_mul(fq_sqr(fq_sqr(tau)), tau);
    } else {
      st(T.fix[r - NF], fq_inv(fq_sqr(fq_sqr(tau))));
    }
    tau = fq_mul(tau, Lf);
  }
  st(T.unscale, fq_inv(tau));
  T.int_layers = 1;
}

// Sparse factorisation of the 59 partial rounds (S-box on the LAST word, index P = 4).
// Partial round t:  x <- M * S_P(x + c_t).  With x = (B_t y_o ; y_P) (B_0 = I) and the MDS split into blocks
// M = [[Moo, Mop], [Mpo, Mpp]] over (others, P):
//     y_P' = (Mpo B_t) (y_o + f_t) + Mpp z,   z = (y_P + c_P)^5,  f_t = B_t^-1 c_o(t)
//     y_o' = (y_o + f_t) + B_{t+1}^-1 Mop z,  B_{t+1} = Moo B_t
// The `others` never mix among themselves, so all f_t are added up-front (pre); the excess that sits in y_o at round t
// pollutes only y_P' and is folded into the next round's key on word P.  After the rounds POST = blockdiag(B_59, 1).
// Algebraically identical to the dense rounds, hence bit-exact.  false <=> a block is singular (not an MDS matrix).
inline bool derive_hades_tables(const uint32_t (*rc)[8], const uint32_t (*mds)[5][8], HadesTables& T) {
  constexpr int W = 5, P = 4, NP = 59, NF = 4;
  memcpy(T.rc, rc, sizeof(T.rc));
  memcpy(T.mds, mds, sizeof(T.mds));
  Mat4 Moo;
  fq Mop[4], Mpo[4], Mpp = ld(mds[P][P]);
  for (int i = 0; i < 4; i++) {
    for (int j = 0; j < 4; j++) Moo.a[i][j] = ld(mds[i][j]);
    Mop[i] = ld(mds[i][P]);
    Mpo[i] = ld(mds[P][i]);
  }
  static thread_local fq folds[NP][4], rows[NP][4], cols[NP][4], F[NP + 1][4];
  Mat4 B = mat_ident();
  for (int t = 0; t < NP; t++) {
    const uint32_t(*c)[8] = rc + (NF + t) * W;
    Mat4 Binv, Bn, Bninv;
    if (!mat_inv(B, Binv)) return false;
    fq co[4];
    for (int i = 0; i < 4; i++) co[i] = ld(c[i]);
    mat_vec(Binv, co, folds[t]);
    Bn = mat_mul(Moo, B);
    if (!mat_inv(Bn, Bninv)) return false;
    mat_vec(Bninv, Mop, cols[t]);
    for (int j = 0; j < 4; j++) {
      fq s = fq_zero();
      for (int k = 0; k < 4; k++) s = fq_add(s, fq_mul(Mpo[k], B.a[k][j]));
      rows[t][j] = s;
    }
    B = Bn;
  }
  for (int k = 0; k < 4; k++) F[0][k] = fq_zero();
  for (int t = 0; t < NP; t++)
    for (int k = 0; k < 4; k++) F[t + 1][k] = fq_add(F[t][k], folds[t][k]);
  for (int k = 0; k < 4; k++) st(T.pre[k], F[NP][k]);
  st(T.pre[P], fq_zero());
  for (int t = 0; t < NP; t++) {
    fq kP = ld(rc[(NF + t) * W + P]);
    if (t > 0) {
      fq corr = fq_zero();
      for (int k = 0; k < 4; k++) corr = fq_add(corr, fq_mul(rows[t - 1][k], fq_sub(F[NP][k], F[t][k])));
      kP = fq_sub(kP, corr);
    }
    uint32_t(*o)[8] = &T.sparse[t * 11];
    st(o[0], kP);
    for (int j = 0; j < 4; j++) st(o[1 + j], rows[t][j]);
    st(o[1 + P], Mpp);
    for (int j = 0; j < 4; j++) st(o[6 + j], cols[t][j]);
    st(o[6 + P], fq_zero());
  }
  for (int i = 0; i < W; i++)
    for (int j = 0; j < W; j++) {
      fq v = (i < 4 && j < 4) ? B.a[i][j] : (i == P && j == P ? fq_one() : fq_zero());
      st(T.post[i * W + j], v);
    }
  derive_int_tables(T);
  return true;
}

// -u^2 + v^2 == 1 + d u^2 v^2
inline bool on_curve(const fq& u, const fq& v) {
  fq u2 = fq_sqr(u), v2 = fq_sqr(v);
  return fq_eq(fq_sub(v2, u2), fq_add(fq_one(), fq_mul(ed_d(), fq_mul(u2, v2))));
}
// r * P == identity and P != identity (a generator of the prime-order subgroup)
inline bool prime_order(const fq& u, const fq& v) {
  const uint32_t rr[8] = SB200_FR_MOD_INIT;
  ext base = affine_to_ext(u, v), acc = ext_identity();
  pniels nb = ext_to_pniels(base);
  for (int bit = 251; bit >= 0; bit--) {
    acc = p1p1_to_ext(ed_dbl(acc.X, acc.Y, acc.Z));
    if ((rr[bit >> 5] >> (bit & 31)) & 1u) acc = p1p1_to_ext(ed_add(acc, nb));
  }
  const bool is_id = fq_is_zero(acc.X) && fq_eq(acc.Y, acc.Z);
  const bool base_id = fq_is_zero(u) && fq_eq(v, fq_one());
  return is_id && !base_id;
}
inline bool canonical_fq(const uint32_t* p) { return lt_q(p); }

}  // namespace params
}  // namespace sb200
