// Hades252 permutation (width 5, x^5, 8 full + 59 partial rounds) and the Poseidon sponge shapes the
// Schnorr challenge uses.  Replaces `dusk_poseidon::sponge::truncated::hash` as called from
// challenge_hash / challenge_hash_double: /root/reference/src/signatures.rs:127-134, 275-290.
//
// One permutation per thread, state in registers (5 x 8 limbs), constants broadcast from
// __constant__ memory (every lane reads the same address in lock-step).
// When the MDS matrix is L^-1 times a matrix C of small integers (the default Cauchy matrix 1/(i+j+5): L = 360360,
// entries of C at most 72072), every round runs dense with C s in place of M s: 200 exact DFMAs and one reduction per
// word instead of five Montgomery dot products (hades_perm_int).  Any other MDS runs the 59 partial rounds in the
// sparse factorisation derived at context creation (params_host.cuh; 9 products per round instead of 25).  Both are
// algebraically identical to the dense rounds, hence bit-exact; the dense form is kept as hades_perm_dense for the
// parity tests and the self-check of the derivation.
#pragma once
#include <cstddef>
#include <cstring>
#if !defined(__CUDA_ARCH__)
#include <cmath>
#endif
#include "fq.cuh"

namespace sb200 {

#define SB_HADES_W 5

// Every Hades table is an INPUT of context creation (include/schnorr_b200.h sb200_params -> params_host.cuh
// derive_hades_tables), uploaded once per device; nothing numeric from dusk-hades is baked into the kernels.
struct HadesTables {
  uint32_t rc[335][8];         // ROUND_CONSTANTS[0..335): 67 rounds x 5 words, consumed in order
  uint32_t mds[25][8];         // MDS_MATRIX, row-major
  uint32_t pre[5][8];          // sparse form: added to the state before the partial rounds
  uint32_t sparse[59 * 11][8]; // per partial round: key (1), row (5), column (5; entry 4 unused)
  uint32_t post[25][8];        // dense matrix applied once after the partial rounds
  // Small-integer form (params_host.cuh derive_int_tables), valid when `int_layers` != 0: MDS = C / L with C a matrix
  // of small integers, the state kept at a known per-round scale tau (Montgomery limbs of tau * x).
  double cmat[25];             // C = L * MDS, row-major, exact small integers
  uint32_t src[335][8];        // round constants times the scale of their round
  uint32_t fix[59][8];         // per partial round: tau^-4 (brings the S-box word from tau^5 back to tau)
  uint32_t unscale[8];         // tau^-1 of the scale after the last layer
  uint32_t int_layers;         // 1: hades_perm runs the small-integer layers
};
// What sb200_params_check / sb200_dbg_hades_tables hand out (include/schnorr_b200.h: 1039 x 8 words)
constexpr size_t HADES_ABI_BYTES = 1039 * 32;
static_assert(offsetof(HadesTables, cmat) == HADES_ABI_BYTES, "the public table views keep their offsets");
#if defined(__CUDACC__)
__constant__ HadesTables d_hades;
#endif
static HadesTables h_hades;  // host build (parameter derivation self-check, tests/host_arith): filled by the same derivation

#if defined(__CUDA_ARCH__)
#define SB_CONST(name) d_##name
#define SB_HADES(field) d_hades.field
#else
#define SB_CONST(name) h_##name
#define SB_HADES(field) h_hades.field
#endif

SB_HD fq ld8(const uint32_t* p) {
  fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = p[i];
  return r;
}

SB_HD fq fq_pow5(const fq& x) {
  fq x2 = fq_sqr(x);
  fq x4 = fq_sqr(x2);
  return fq_mul(x4, x);
}

// s <- M * s with M a dense 5x5 matrix in constant memory (row-major)
// (each row is one lazily reduced dot product: 5 x 64 + 56 wide products instead of 5 x 120)
#define SB_MATMUL5(s, mat)                                                                  \
  do {                                                                                      \
    fq _r[5];                                                                               \
    _Pragma("unroll") for (int _k = 0; _k < 5; _k++)                                        \
        _r[_k] = fq_dot5(&SB_HADES(mat)[_k * 5], s[0], s[1], s[2], s[3], s[4]);             \
    _Pragma("unroll") for (int _k = 0; _k < 5; _k++) s[_k] = _r[_k];                        \
  } while (0)

// plain version (one reduction per product) for the reference-shaped dense permutation
#define SB_MATMUL5_PLAIN(s, mat)                                        \
  do {                                                                  \
    fq _r[5];                                                           \
    _Pragma("unroll 1") for (int _k = 0; _k < 5; _k++) {                \
      fq _a = fq_mul(ld8(SB_HADES(mat)[_k * 5]), s[0]);                 \
      _Pragma("unroll") for (int _j = 1; _j < 5; _j++)                  \
          _a = fq_add(_a, fq_mul(ld8(SB_HADES(mat)[_k * 5 + _j]), s[_j])); \
      _r[_k] = _a;                                                      \
    }                                                                   \
    _Pragma("unroll") for (int _k = 0; _k < 5; _k++) s[_k] = _r[_k];    \
  } while (0)

template <bool LAZY = true>
SB_HD void hades_full_round(fq* s, int rc_base) {
#pragma unroll
  for (int k = 0; k < 5; k++) s[k] = fq_pow5(fq_add(s[k], ld8(SB_HADES(rc)[rc_base + k])));
  if (LAZY) SB_MATMUL5(s, mds); else SB_MATMUL5_PLAIN(s, mds);
}

// Reference-shaped permutation (ScalarStrategy::perm of dusk-hades): used by parity tests.
SB_HD void hades_perm_dense(fq* s) {
  int rc = 0;
#pragma unroll 1
  for (int r = 0; r < 4; r++, rc += 5) hades_full_round<false>(s, rc);
#pragma unroll 1
  for (int r = 0; r < 59; r++, rc += 5) {
#pragma unroll
    for (int k = 0; k < 5; k++) s[k] = fq_add(s[k], ld8(SB_HADES(rc)[rc + k]));
    s[4] = fq_pow5(s[4]);
    SB_MATMUL5_PLAIN(s, mds);
  }
#pragma unroll 1
  for (int r = 0; r < 4; r++, rc += 5) hades_full_round<false>(s, rc);
}

// ---- small-integer layers on the FP64 pipe -------------------------------------------------------------------------
// A limb times an entry of C is below 2^32 * 2^20 / 5, so a five-term column plus the carry of the previous column
// stays below 2^52: a DFMA chain seeded with 2^52 holds it exactly, the integer in the low mantissa bits.  Every DFMA
// here is exact, so the host build (std::fma on the same doubles) computes the same bits.
constexpr uint32_t HI_2P52 = 0x43300000u;  // high word of 2^52
constexpr double RECIP_Q224 = 0x1.1aa84a76ff6f1p-31;  // largest double <= 2^224 / q

SB_HD double hl_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  SB_COUNT(dfma, 1);
  return std::fma(a, b, c);
#endif
}
SB_HD double hl_pair(uint32_t hi, uint32_t lo) {  // the double with these bits
#if defined(__CUDA_ARCH__)
  return __hiloint2double((int)hi, (int)lo);
#else
  uint64_t b = (uint64_t)hi << 32 | lo;
  double d;
  memcpy(&d, &b, 8);
  return d;
#endif
}
SB_HD uint64_t hl_bits(double d) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(d);
#else
  uint64_t b;
  memcpy(&b, &d, 8);
  return b;
#endif
}
SB_HD double hl_sub52(double d) {  // d - 2^52, exact for d in [2^52, 2^53)
#if defined(__CUDA_ARCH__)
  return __dsub_rn(d, 0x1p+52);
#else
  return d - 0x1p+52;
#endif
}

// r <- (top * 2^256 + r) mod q, canonical, for a value below 2^20 q (a layer row is below 5 * max C * q).
// Q = floor(T * RECIP_Q224) with T = top * 2^32 + r[7] is the quotient or one less (T * 2^224 <= value, and the error of
// the estimate is below 2^-30), so value - Q q is in [0, 2q).  Q < 2^20 and every limb of q is below 2^32, so each
// Q q_i is one exact DFMA.
SB_HD void hl_reduce(fq& r, uint32_t top) {
  const double T = hl_sub52(hl_pair(HI_2P52 | top, r.v[7]));
#if defined(__CUDA_ARCH__)
  const double h = __fma_rz(T, RECIP_Q224, 0x1p+52);  // 2^52 + floor(T * RECIP_Q224)
#else
  SB_COUNT(dfma, 1);  // the same floor, from the 53-bit significand of RECIP_Q224 (= m * 2^-83)
  const uint64_t Ti = (uint64_t)top << 32 | r.v[7];
  const double h = 0x1p+52 + (double)(uint64_t)(((unsigned __int128)Ti * 0x11aa84a76ff6f1ull) >> 83);
#endif
  const double Qd = hl_sub52(h);
  uint32_t lo[8], hi[8];
  lo[0] = (uint32_t)hl_bits(h);  // q_0 = 1
  hi[0] = 0;
#pragma unroll
  for (int i = 1; i < 8; i++) {
    const uint64_t b = hl_bits(hl_fma(Qd, (double)FqP::p(i), 0x1p+52));
    lo[i] = (uint32_t)b;
    hi[i] = (uint32_t)(b >> 32) & 0xfffffu;
  }
  uint32_t qq[8], sh[8];  // Q q mod 2^256 = lo + hi * 2^32; the difference is below 2q < 2^256
  sh[0] = 0;
#pragma unroll
  for (int i = 1; i < 8; i++) sh[i] = hi[i - 1];
  add8(qq, lo, sh);
  sub8(r.v, r.v, qq);
  cond_sub_p<FqP>(r.v);
}

// s <- C s mod q, in place.  Columns in increasing limb order; each output limb overwrites the input limb of the same
// column, whose five readers have all run, and the column's carry seeds the next column's chain.
SB_HD void hades_int_layer(fq* s) {
  uint32_t c[5];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    double x[5];
#pragma unroll
    for (int j = 0; j < 5; j++) x[j] = hl_sub52(hl_pair(HI_2P52, s[j].v[i]));
#pragma unroll
    for (int k = 0; k < 5; k++) {
      double acc = hl_pair(HI_2P52, i ? c[k] : 0u);
#pragma unroll
      for (int j = 0; j < 5; j++) acc = hl_fma(SB_HADES(cmat)[k * 5 + j], x[j], acc);
      const uint64_t b = hl_bits(acc);
      s[k].v[i] = (uint32_t)b;
      c[k] = (uint32_t)(b >> 32) & 0xfffffu;
    }
  }
#pragma unroll
  for (int k = 0; k < 5; k++) hl_reduce(s[k], c[k]);
}

// All 67 rounds dense, with M s computed as C s and the factor L tracked in the scale: round constants are pre-scaled,
// a full S-box raises the scale to its fifth power, and in a partial round one product by tau^-4 returns the S-box
// word to the scale of the others.  Exact arithmetic in F_q, so the result equals hades_perm_dense bit for bit.
SB_HD void hades_perm_int(fq* s) {
#pragma unroll 1
  for (int r = 0; r < 67; r++) {
#pragma unroll
    for (int k = 0; k < 5; k++) s[k] = fq_add(s[k], ld8(SB_HADES(src)[r * 5 + k]));
    if (r < 4 || r >= 63) {
#pragma unroll
      for (int k = 0; k < 5; k++) s[k] = fq_pow5(s[k]);
    } else {
      s[4] = fq_mul(fq_pow5(s[4]), ld8(SB_HADES(fix)[r - 4]));
    }
    hades_int_layer(s);
  }
#pragma unroll
  for (int k = 0; k < 5; k++) s[k] = fq_mul(s[k], ld8(SB_HADES(unscale)));
}

// Production permutation: the small-integer layers when the context's MDS qualifies, else sparse partial rounds.
SB_HD void hades_perm(fq* s) {
  if (SB_HADES(int_layers)) {
    hades_perm_int(s);
    return;
  }
  int rc = 0;
#pragma unroll 1
  for (int r = 0; r < 4; r++, rc += 5) hades_full_round(s, rc);
#pragma unroll
  for (int k = 0; k < 4; k++) s[k] = fq_add(s[k], ld8(SB_HADES(pre)[k]));
#pragma unroll 1
  for (int t = 0; t < 59; t++) {
    const uint32_t(*c)[8] = &SB_HADES(sparse)[t * 11];
    s[4] = fq_pow5(fq_add(s[4], ld8(c[0])));
    fq np = fq_dot5(&c[1], s[0], s[1], s[2], s[3], s[4]);  // row . state, one reduction
#pragma unroll
    for (int j = 0; j < 4; j++) s[j] = fq_add(s[j], fq_mul(ld8(c[6 + j]), s[4]));
    s[4] = np;
  }
  SB_MATMUL5(s, post);
  rc += 59 * 5;
#pragma unroll 1
  for (int r = 0; r < 4; r++, rc += 5) hades_full_round(s, rc);
}

// low 250 bits of the canonical integer (dusk_poseidon::sponge::truncated), as a scalar
SB_HD void truncate250(const fq& mont_word, uint32_t* c) {
  fq x = fq_from_mont(mont_word);
#pragma unroll
  for (int i = 0; i < 8; i++) c[i] = x.v[i];
  c[7] &= 0x03ffffffu;
}

// c = H(Ru, Rv, m): sponge state [0, Ru, Rv, m, 1], one permutation, word 1.
template <bool DENSE = false>
SB_HD void challenge3(const fq& Ru, const fq& Rv, const fq& m, uint32_t* c) {
  fq s[5] = {fq_zero(), Ru, Rv, m, fq_one()};
  if (DENSE) hades_perm_dense(s); else hades_perm(s);
  truncate250(s[1], c);
}

// c = H(Ru, Rv, R'u, R'v, m): [0, Ru, Rv, R'u, R'v] -> perm -> word1 += m, word2 += 1 -> perm -> word 1.
template <bool DENSE = false>
SB_HD void challenge5(const fq& Ru, const fq& Rv, const fq& Rpu, const fq& Rpv, const fq& m, uint32_t* c) {
  fq s[5] = {fq_zero(), Ru, Rv, Rpu, Rpv};
  if (DENSE) hades_perm_dense(s); else hades_perm(s);
  s[1] = fq_add(s[1], m);
  s[2] = fq_add(s[2], fq_one());
  if (DENSE) hades_perm_dense(s); else hades_perm(s);
  truncate250(s[1], c);
}

}  // namespace sb200
