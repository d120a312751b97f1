// Per-tuple sign / verify / keygen bodies (one tuple per thread).  Host+device so the exact code
// the kernels run is also exercised on the CPU by tests/host_arith (test scaffolding only).
//
//   verify_core         PublicKey::verify        /root/reference/src/keys/public.rs:121-130
//   verify_double_core  PublicKeyDouble::verify  /root/reference/src/keys/public.rs:222-244
//   verify_vargen_core  PublicKeyVarGen::verify  /root/reference/src/keys/public.rs:401-415
//   sign_core           SecretKey::sign          /root/reference/src/keys/secret.rs:150-168
//   sign_double_core    SecretKey::sign_double   /root/reference/src/keys/secret.rs:217-240
//   sign_vargen_core    SecretKeyVarGen::sign    /root/reference/src/keys/secret.rs:433-451
//   keygen*_core        PublicKey*::from         /root/reference/src/keys/public.rs:61-67,265-272,337-344
#pragma once
#include "ed.cuh"
#include "hades.cuh"
#include "hgcd.cuh"
#include "lat3.cuh"
#include "inv.cuh"
// The FP64-pipe permutation (DESIGN.md 4.4) is a measured experiment that lost; it is compiled only with
// -DSB_EXPERIMENTAL_FD=1 (its tables are baked by tools/gen_constants.py, not context parameters).
#ifndef SB_EXPERIMENTAL_FD
#define SB_EXPERIMENTAL_FD 0
#endif
#if SB_EXPERIMENTAL_FD
#include "experimental/hades_fd.cuh"
#endif

namespace sb200 {

// Challenge hash of the one-tuple-per-thread kernels: the IMAD.WIDE permutation of hades.cuh.  SB_HADES_FD=1 selects
// the FP64-pipe permutation (hades_fd.cuh) instead -- same scalar; measured slower when every warp runs both halves
// (the win comes from dedicating warps to it: k_verify_ws in schnorr_b200.cu).
#ifndef SB_HADES_FD
#define SB_HADES_FD 0
#endif
#if SB_HADES_FD && !SB_EXPERIMENTAL_FD
#error "SB_HADES_FD needs SB_EXPERIMENTAL_FD"
#endif
SB_HD void chal3(const fq& Ru, const fq& Rv, const fq& m, uint32_t* c) {
#if SB_HADES_FD
  challenge3_fd(Ru, Rv, m, c);
#else
  challenge3(Ru, Rv, m, c);
#endif
}
SB_HD void chal5(const fq& Ru, const fq& Rv, const fq& Rpu, const fq& Rpv, const fq& m, uint32_t* c) {
#if SB_HADES_FD
  challenge5_fd(Ru, Rv, Rpu, Rpv, m, c);
#else
  challenge5(Ru, Rv, Rpu, Rpv, m, c);
#endif
}

struct point_in {  // a point as handed over the ABI: affine (Z absent => 1) or projective (U : V : Z)
  fq U, V, Z;
  bool affine;
};

SB_HD ext point_to_ext(const point_in& p) { return p.affine ? affine_to_ext(p.U, p.V) : proj_to_ext(p.U, p.V, p.Z); }

// affine coordinates for hashing = `to_hash_inputs()` (JubJubAffine::from(extended): one inversion)
SB_HD void point_to_affine(const point_in& p, fq& u, fq& v) {
  if (p.affine) {
    u = p.U;
    v = p.V;
  } else {
    fq zi = fq_inv_fast(p.Z);  // public data: the Euclidean inversion (inv.cuh)
    u = fq_mul(p.U, zi);
    v = fq_mul(p.V, zi);
  }
}

// well-formed input point: on the curve and Z != 0 (SB200_CHECK_POINTS, sb200_points_check).  The reference's
// constructors only produce such points; `from_raw_unchecked` (/root/reference/src/keys/public.rs:142,256,427) can
// supply anything.   -U^2 Z^2 + V^2 Z^2 == Z^4 + d U^2 V^2   (Z = 1 when affine)
SB_HD bool point_well_formed(const point_in& p) {
  fq u2 = fq_sqr(p.U), v2 = fq_sqr(p.V);
  fq lhs = fq_sub(v2, u2), duv = fq_mul(ed_d(), fq_mul(u2, v2));
  if (p.affine) return fq_eq(lhs, fq_add(fq_one(), duv));
  fq z2 = fq_sqr(p.Z);
  return fq_eq(fq_mul(lhs, z2), fq_add(fq_sqr(z2), duv)) & !fq_is_zero(p.Z);
}

// completed point == R (projective equality u1*z2 == u2*z1 && v1*z2 == v2*z1, /root/reference/tests/keys.rs:52-58);
// with (X : Y : Z) = (E*F : G*H : F*G) this is E*Rz == Ru*G && H*Rz == Rv*F.
SB_HD bool p1p1_equals(const p1p1& c, const point_in& R) {
  fq l1 = R.affine ? c.E : fq_mul(c.E, R.Z);
  fq l2 = R.affine ? c.H : fq_mul(c.H, R.Z);
  return fq_eq(l1, fq_mul(R.U, c.G)) & fq_eq(l2, fq_mul(R.V, c.F));
}

SB_HD bool scalar_lt_r(const uint32_t* k) {
  uint32_t t[8];
  const uint32_t rr[8] = SB200_FR_MOD_INIT;
  return sub8(t, k, rr) != 0;  // borrow <=> k < r
}

// the curve half of a verification: c*PK + u*G == R for a challenge computed elsewhere
SB_HD bool verify_ec_core(const point_in& PK, const uint32_t* u_in, const point_in& R, const uint32_t* c_in,
                          const uint32_t* combG) {
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u[i] = ok ? u_in[i] : 0u;
    c[i] = c_in[i];
  }
  pniels tab[9];
  vartable_build(tab, point_to_ext(PK));
  recode_offset<4>(c);
  p1p1 cp = ed_mul_var(tab, c, 63);  // c < 2^250: 63 windows
  recode_offset<COMB_BITS>(u);
  cp = ed_comb_add(p1p1_to_ext(cp), combG, u);
  return ok & p1p1_equals(cp, R);
}

// The same predicate with half-size scalars (hgcd.cuh):  (b u mod r) G + a PK - b R == identity  for  a = b c (mod 8r),
// b odd: two variable-base tables, 34 windows (132 doublings) instead of 63 (248).  `fast_ok` = false where the
// short vector does not fit the window budget; the caller then uses verify_ec_core for that tuple.
SB_HD point_in point_neg(const point_in& p) {
  point_in r = p;
  r.U = fq_neg(p.U);
  return r;
}
// shared part: the short vector (a, b) for the challenge and  w = b u mod r
struct half_scalars {
  hgcd_res h;      // a, |b| (offset-recoded for 4-bit windows), sign of b, ok
  uint32_t w[8];   // b u mod r, offset-recoded for the comb
};
SB_HD half_scalars half_scalars_prepare(const uint32_t* u, const uint32_t* c_in) {
  half_scalars hs;
  hs.h = half_gcd_8r(c_in);
  fr bb, uu;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    bb.v[i] = hs.h.b[i];
    uu.v[i] = u[i];
  }
  fr w = fr_mul(bb, uu);  // |b| u mod r
  if (hs.h.bneg) {        // b u = -(|b| u)
    fr z;
#pragma unroll
    for (int i = 0; i < 8; i++) z.v[i] = 0;
    w = fr_sub(z, w);
  }
#pragma unroll
  for (int i = 0; i < 8; i++) hs.w[i] = w.v[i];
  recode_offset<4>(hs.h.a);
  recode_offset<4>(hs.h.b);
  recode_offset<COMB_BITS>(hs.w);
  return hs;
}
// (b u) B + a PK - b R == identity  for the generator B whose comb table is `comb`
// `store` = 18 table entries of this thread in caller-provided memory, or nullptr for a local array.  Local memory is
// word-interleaved across a warp, so a lookup with a per-lane index pulls a different 32-byte sector for every word of
// every lane; a thread-major region in global memory serves each lookup with four full sectors instead.
#ifndef SB_TABLE_STAGE
#define SB_TABLE_STAGE 1  // with SB_EC_GLOBAL_TABLES: stage each window's two entries into shared memory by cp.async (ed.cuh)
#endif
template <bool EXT = false>
SB_HD bool verify_ec_half(const point_in& PK, const point_in& R, const half_scalars& hs, const uint32_t* comb,
                          pniels* store = nullptr, uint4* stage = nullptr) {
  (void)stage;
  pniels local_tabs[EXT ? 1 : 18];
  pniels* tabs0 = EXT ? store : local_tabs;  // [0..9): multiples of -sign(b) R (|b| of them make -b R)
  pniels* tabs1 = tabs0 + 9;                 // [9..18): multiples of PK
  {
    const point_in nR = hs.h.bneg ? R : point_neg(R);
#pragma unroll 1
    for (int t = 0; t < 2; t++) vartable_build(t ? tabs1 : tabs0, point_to_ext(t ? PK : nR));  // one copy of the table code
  }
#if defined(__CUDA_ARCH__) && SB_TABLE_STAGE
  p1p1 cp = EXT ? ed_mul_var2_staged(tabs0, hs.h.b, tabs1, hs.h.a, 34, stage) : ed_mul_var2_rolled(tabs0, hs.h.b, tabs1, hs.h.a, 34);
#else
  p1p1 cp = ed_mul_var2_rolled(tabs0, hs.h.b, tabs1, hs.h.a, 34);
#endif
  cp = ed_comb_add(p1p1_to_ext(cp), comb, hs.w);
  // identity <=> X = E F = 0 and Y = G H = Z = F G with F, G != 0 (complete addition) <=> E = 0 and H = F
  return fq_is_zero(cp.E) & fq_eq(cp.H, cp.F);
}
template <bool EXT = false>
SB_HD bool verify_ec_core_fast(const point_in& PK, const uint32_t* u_in, const point_in& R, const uint32_t* c_in,
                               const uint32_t* combG, bool& fast_ok, pniels* store = nullptr, uint4* stage = nullptr) {
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; i++) u[i] = ok ? u_in[i] : 0u;
  half_scalars hs = half_scalars_prepare(u, c_in);
  fast_ok = hs.h.ok;
  return ok & verify_ec_half<EXT>(PK, R, hs, combG, store, stage);
}

#ifndef SB_VERIFY_HGCD
#define SB_VERIFY_HGCD 1
#endif
// c PK + u G == R, by the half-size form where it applies
template <bool EXT = false>
SB_HD bool verify_ec(const point_in& PK, const uint32_t* u_in, const point_in& R, const uint32_t* c_in, const uint32_t* combG,
                     pniels* store = nullptr, uint4* stage = nullptr) {
#if SB_VERIFY_HGCD
  bool fast_ok;
  bool ok = verify_ec_core_fast<EXT>(PK, u_in, R, c_in, combG, fast_ok, store, stage);
  if (SB_WARP_ANY(!fast_ok)) {
    bool slow = verify_ec_core(PK, u_in, R, c_in, combG);
    ok = fast_ok ? ok : slow;
  }
  return ok;
#else
  return verify_ec_core(PK, u_in, R, c_in, combG);
#endif
}

// the hash half: c = H(R_affine, m)
SB_HD void verify_hash_core(const point_in& R, const fq& m, uint32_t* c_out) {
  fq ru, rv;
  point_to_affine(R, ru, rv);
  chal3(ru, rv, m, c_out);
}
#if SB_EXPERIMENTAL_FD
// ... on the FP64 pipe, permutation state in caller-provided slot storage (hades_fd.cuh)
SB_HD void verify_hash_core_fd(const point_in& R, const fq& m, uint32_t* c_out, double* slots, int ls) {
  fq ru, rv;
  point_to_affine(R, ru, rv);
  challenge3_fd_p(ru, rv, m, c_out, slots, ls);
}
#endif

SB_HD bool verify_core(const point_in& PK, const uint32_t* u_in, const point_in& R, const fq& m, const uint32_t* combG,
                       uint32_t* c_out) {
  verify_hash_core(R, m, c_out);
  return verify_ec(PK, u_in, R, c_out, combG);
}

// curve half of the variable-generator verification: u Gen + c PK == R (Straus, both bases variable; the half-size
// trick does not apply: the generator's scalar b u mod r would be full-size again)
SB_HD bool verify_vargen_ec(const point_in& PK, const point_in& GEN, const uint32_t* u_in, const point_in& R,
                            const uint32_t* c_in) {
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u[i] = ok ? u_in[i] : 0u;
    c[i] = c_in[i];
  }
  pniels tabs[2][9];
#pragma unroll 1
  for (int t = 0; t < 2; t++) vartable_build(tabs[t], point_to_ext(t ? PK : GEN));
  recode_offset<4>(c);
  recode_offset<4>(u);
  p1p1 cp = ed_mul_var2_rolled(tabs[0], u, tabs[1], c, 64);
  return ok & p1p1_equals(cp, R);
}
// The same predicate with short scalars (lat3.cuh):  d Gen + a PK - b R == identity  for a lattice vector (b, a, d),
// a = b c, d = b u (mod 8r), b odd: three variable-base tables, 44 windows (172 doublings) instead of 64 (252).
// `fast_ok` = false where no basis vector fits the window budget; the caller then uses verify_vargen_ec.
#ifndef SB_VARGEN_LAT3
#define SB_VARGEN_LAT3 1
#endif
template <bool EXT = false>
SB_HD bool verify_vargen_ec_fast(const point_in& PK, const point_in& GEN, const uint32_t* u_in, const point_in& R,
                                 const uint32_t* c_in, bool& fast_ok, pniels* store = nullptr, uint4* stage = nullptr) {
  (void)stage;
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; i++) u[i] = ok ? u_in[i] : 0u;
  lat3_res L = lattice3_8r_call(c_in, u);
  fast_ok = L.ok;
  uint32_t kr[24];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    kr[i] = L.d[i];
    kr[8 + i] = L.a[i];
    kr[16 + i] = L.b[i];
  }
  pniels local_tabs[EXT ? 1 : 27];  // multiples of sgn(d) Gen, sgn(a) PK, -sgn(b) R (EXT: in the caller's global scratch)
  pniels* tabs = EXT ? store : local_tabs;
#pragma unroll 1
  for (int t = 0; t < 3; t++) {
    const point_in& P = t == 0 ? GEN : t == 1 ? PK : R;
    const bool neg = t == 0 ? L.dneg : t == 1 ? L.aneg : !L.bneg;
    vartable_build(tabs + 9 * t, point_to_ext(neg ? point_neg(P) : P));
    recode_offset<4>(kr + 8 * t);
  }
#if defined(__CUDA_ARCH__) && SB_TABLE_STAGE
  p1p1 cp = EXT ? ed_mul_var3_staged(tabs, kr, LAT3_WINDOWS, stage) : ed_mul_var3_rolled(tabs, kr, LAT3_WINDOWS);
#else
  p1p1 cp = ed_mul_var3_rolled(tabs, kr, LAT3_WINDOWS);
#endif
  // identity <=> E = 0 and H = F (see verify_ec_half)
  return ok & fq_is_zero(cp.E) & fq_eq(cp.H, cp.F);
}
// u Gen + c PK == R, by the short-scalar form where it applies
template <bool EXT = false>
SB_HD bool verify_vargen_ec_auto(const point_in& PK, const point_in& GEN, const uint32_t* u_in, const point_in& R,
                                 const uint32_t* c_in, pniels* store = nullptr, uint4* stage = nullptr) {
#if SB_VARGEN_LAT3
  bool fast_ok;
  bool ok = verify_vargen_ec_fast<EXT>(PK, GEN, u_in, R, c_in, fast_ok, store, stage);
  if (SB_WARP_ANY(!fast_ok)) {
    bool slow = verify_vargen_ec(PK, GEN, u_in, R, c_in);
    ok = fast_ok ? ok : slow;
  }
  return ok;
#else
  return verify_vargen_ec(PK, GEN, u_in, R, c_in);
#endif
}
SB_HD bool verify_vargen_core(const point_in& PK, const point_in& GEN, const uint32_t* u_in, const point_in& R,
                              const fq& m, uint32_t* c_out) {
  verify_hash_core(R, m, c_out);
  return verify_vargen_ec_auto(PK, GEN, u_in, R, c_out);
}

// hash half of the double-key verification: c = H(R, R', m)
SB_HD void verify_double_hash_core(const point_in& R, const point_in& Rp, const fq& m, uint32_t* c_out) {
  fq ru, rv, rpu, rpv;
  if (R.affine) {
    ru = R.U; rv = R.V; rpu = Rp.U; rpv = Rp.V;
  } else {  // one shared inversion for Z and Z'
    fq zz = fq_mul(R.Z, Rp.Z);
    fq zi = fq_inv_fast(zz);
    fq zi1 = fq_mul(zi, Rp.Z), zi2 = fq_mul(zi, R.Z);
    ru = fq_mul(R.U, zi1); rv = fq_mul(R.V, zi1);
    rpu = fq_mul(Rp.U, zi2); rpv = fq_mul(Rp.V, zi2);
  }
  chal5(ru, rv, rpu, rpv, m, c_out);
}
// curve half, full-size scalars: u G + c PK == R  and  u G' + c PK' == R'
SB_HD bool verify_double_ec_core(const point_in& PK, const point_in& PKp, const uint32_t* u_in, const point_in& R,
                                 const point_in& Rp, const uint32_t* c_in, const uint32_t* combG, const uint32_t* combGp) {
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u[i] = ok ? u_in[i] : 0u;
    c[i] = c_in[i];
  }
  recode_offset<4>(c);
  recode_offset<COMB_BITS>(u);
  // the two key / nonce-point pairs run through ONE copy of the curve code (a 2-trip loop): two inlined copies double
  // the hot code and warps in different halves evict each other from the instruction cache
#pragma unroll 1
  for (int k = 0; k < 2; k++) {
    const point_in& key = k ? PKp : PK;
    const point_in& rr = k ? Rp : R;
    pniels tab[9];
    vartable_build(tab, point_to_ext(key));
    p1p1 cp = ed_mul_var(tab, c, 63);
    cp = ed_comb_add(p1p1_to_ext(cp), k ? combGp : combG, u);
    ok &= p1p1_equals(cp, rr);
  }
  return ok;
}
// ... with half-size scalars where they fit (one short vector serves both equations: same c, same u)
template <bool EXT = false>
SB_HD bool verify_double_ec(const point_in& PK, const point_in& PKp, const uint32_t* u_in, const point_in& R, const point_in& Rp,
                            const uint32_t* c_in, const uint32_t* combG, const uint32_t* combGp, pniels* store = nullptr,
                            uint4* stage = nullptr) {
#if SB_VERIFY_HGCD
  bool ok = scalar_lt_r(u_in);
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; i++) u[i] = ok ? u_in[i] : 0u;
  half_scalars hs = half_scalars_prepare(u, c_in);
#pragma unroll 1
  for (int k = 0; k < 2; k++) ok &= verify_ec_half<EXT>(k ? PKp : PK, k ? Rp : R, hs, k ? combGp : combG, store, stage);
  if (SB_WARP_ANY(!hs.h.ok)) {
    bool slow = verify_double_ec_core(PK, PKp, u_in, R, Rp, c_in, combG, combGp);
    ok = hs.h.ok ? ok : slow;
  }
  return ok;
#else
  return verify_double_ec_core(PK, PKp, u_in, R, Rp, c_in, combG, combGp);
#endif
}
SB_HD bool verify_double_core(const point_in& PK, const point_in& PKp, const uint32_t* u_in, const point_in& R,
                              const point_in& Rp, const fq& m, const uint32_t* combG, const uint32_t* combGp,
                              uint32_t* c_out) {
  verify_double_hash_core(R, Rp, m, c_out);
  return verify_double_ec(PK, PKp, u_in, R, Rp, c_out, combG, combGp);
}

// oblivious = true keeps Fermat's constant-time a^(q-2) (Z depends on the nonce / secret key when signing)
SB_HD void ext_to_affine(const ext& p, fq& u, fq& v, bool oblivious = false) {
  fq zi = oblivious ? fq_inv(p.Z) : fq_inv_fast(p.Z);
  u = fq_mul(p.X, zi);
  v = fq_mul(p.Y, zi);
}

// Montgomery's trick: z[0..n) <- 1/z[0..n) with ONE inversion and 3(n-1) multiplications (all z[j] != 0:
// Z coordinates of complete-addition results).  Used to convert several points per thread to affine.
// FAST: the Euclidean inversion of inv.cuh (data-dependent running time); otherwise Fermat's a^(q-2) (the address-oblivious paths).
template <bool FAST = true>
SB_HD void batch_inverse(fq* z, fq* pre, int n) {
  fq acc = z[0];
  pre[0] = fq_one();
#pragma unroll 1
  for (int j = 1; j < n; j++) {
    pre[j] = acc;
    acc = fq_mul(acc, z[j]);
  }
  fq inv = FAST ? fq_inv_fast(acc) : fq_inv(acc);
#pragma unroll 1
  for (int j = n - 1; j > 0; j--) {
    fq zj = z[j];
    z[j] = fq_mul(inv, pre[j]);
    inv = fq_mul(inv, zj);
  }
  z[0] = inv;
}

// Window j of P's per-key comb (ed.cuh, KS_*) into `win` (KS_ENTRIES x 24 words): B = 2^(8j) P by 8j doublings, then
// 2B .. 128B by repeated addition, held as (X, Y) in the entry's own words and Z in z[e - 1]; one batched inversion of the
// 128 Z (z and pre: KS_ENTRIES - 1 fq each of caller memory) and the affine Niels form in place.  Only public data enters:
// the Euclidean inversion.  A P off the curve or with Z = 0 leaves garbage in this window and nowhere else.
SB_HD void keyset_build_window(const ext& P, int j, uint32_t* win, fq* z, fq* pre) {
  constexpr int NE = KS_ENTRIES - 1;  // entries 1..128
  ext B = P;
#pragma unroll 1
  for (int i = 0; i < KS_BITS * j; i++) B = p1p1_to_ext(ed_dbl(B.X, B.Y, B.Z));
  const pniels nb = ext_to_pniels(B);
  ext cur = B;
#pragma unroll 1
  for (int e = 1; e <= NE; e++) {
    if (e > 1) cur = p1p1_to_ext(ed_add(cur, nb));
#pragma unroll
    for (int i = 0; i < 8; i++) {
      win[24 * e + i] = cur.X.v[i];
      win[24 * e + 8 + i] = cur.Y.v[i];
    }
    z[e - 1] = cur.Z;
  }
  batch_inverse(z, pre, NE);
#pragma unroll 1
  for (int e = 1; e <= NE; e++) {
    fq X, Y;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      X.v[i] = win[24 * e + i];
      Y.v[i] = win[24 * e + 8 + i];
    }
    const fq zi = z[e - 1], x = fq_mul(X, zi), y = fq_mul(Y, zi);
    const fq ypx = fq_add(y, x), ymx = fq_sub(y, x), t2d = fq_mul(fq_mul(x, y), ed_2d());
#pragma unroll
    for (int i = 0; i < 8; i++) {
      win[24 * e + i] = ypx.v[i];
      win[24 * e + 8 + i] = ymx.v[i];
      win[24 * e + 16 + i] = t2d.v[i];
    }
  }
  const fq one = fq_one();  // entry 0: the identity (1, 1, 0)
#pragma unroll
  for (int i = 0; i < 8; i++) {
    win[i] = one.v[i];
    win[8 + i] = one.v[i];
    win[16 + i] = 0u;
  }
}

// u = nonce - c * sk  (mod r)
SB_HD void sign_finish(const uint32_t* nonce, const uint32_t* c, const uint32_t* sk, uint32_t* u_out) {
  fr a, b, n;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    a.v[i] = c[i];
    b.v[i] = sk[i];
    n.v[i] = nonce[i];
  }
  fr u = fr_sub(n, fr_mul(a, b));
#pragma unroll
  for (int i = 0; i < 8; i++) u_out[i] = u.v[i];
}

// k*B for the fixed generator whose comb table is `comb`; k canonical (< 2^252)
SB_HD ext fixed_base_mul(const uint32_t* comb, const uint32_t* k) {
  uint32_t kr[8];
#pragma unroll
  for (int i = 0; i < 8; i++) kr[i] = k[i];
  recode_offset<COMB_BITS>(kr);
  return p1p1_to_ext(ed_comb_add(ext_identity(), comb, kr));
}

SB_HD ext var_base_mul(const point_in& P, const uint32_t* k) {
  uint32_t kr[8];
#pragma unroll
  for (int i = 0; i < 8; i++) kr[i] = k[i];
  recode_offset<4>(kr);
  pniels tab[9];
  vartable_build(tab, point_to_ext(P));
  return p1p1_to_ext(ed_mul_var(tab, kr, 64));
}

// k * P with the window table scanned instead of indexed (SB200_SIGN_OBLIVIOUS: k is a nonce or a secret key)
SB_HD ext var_base_mul_oblivious(const point_in& P, const uint32_t* k) {
  uint32_t kr[8];
#pragma unroll
  for (int i = 0; i < 8; i++) kr[i] = k[i];
  recode_offset<4>(kr);
  pniels tab[9];
  vartable_build(tab, point_to_ext(P));
  return p1p1_to_ext(ed_mul_var_oblivious(tab, kr));
}

SB_HD void sign_core(const uint32_t* sk, const uint32_t* nonce, const fq& m, const uint32_t* combG, uint32_t* u_out,
                     fq& Ru, fq& Rv, uint32_t* c_out) {
  ext_to_affine(fixed_base_mul(combG, nonce), Ru, Rv);
  chal3(Ru, Rv, m, c_out);
  sign_finish(nonce, c_out, sk, u_out);
}

SB_HD void sign_double_core(const uint32_t* sk, const uint32_t* nonce, const fq& m, const uint32_t* combG,
                            const uint32_t* combGp, uint32_t* u_out, fq& Ru, fq& Rv, fq& Rpu, fq& Rpv, uint32_t* c_out) {
  ext a = fixed_base_mul(combG, nonce), b = fixed_base_mul(combGp, nonce);
  fq zi = fq_inv_fast(fq_mul(a.Z, b.Z));  // one inversion for both
  fq zi1 = fq_mul(zi, b.Z), zi2 = fq_mul(zi, a.Z);
  Ru = fq_mul(a.X, zi1); Rv = fq_mul(a.Y, zi1);
  Rpu = fq_mul(b.X, zi2); Rpv = fq_mul(b.Y, zi2);
  chal5(Ru, Rv, Rpu, Rpv, m, c_out);
  sign_finish(nonce, c_out, sk, u_out);
}

SB_HD void sign_vargen_core(const uint32_t* sk, const point_in& GEN, const uint32_t* nonce, const fq& m, uint32_t* u_out,
                            fq& Ru, fq& Rv, uint32_t* c_out, bool oblivious = false) {
  ext_to_affine(oblivious ? var_base_mul_oblivious(GEN, nonce) : var_base_mul(GEN, nonce), Ru, Rv, oblivious);
  chal3(Ru, Rv, m, c_out);
  sign_finish(nonce, c_out, sk, u_out);
}

// ------------------------------------------------------------------------------------------------------------
// PLONK witness pre-computation (SURVEY.md 8(f) row 4).  The reference's circuits allocate, per signature,
//   Signature::append        u as a BlsScalar witness + R as a witness point   /root/reference/src/signatures.rs:97-103,
//                            (+ R' for the double scheme)                       231-241, 377-383
//   gadgets::verify_signature*   pk (pk', generator) as witness points, msg, and as component outputs the challenge
//                            c = H(...) (sponge::truncated::gadget), s_a = u * G, s_b = c * PK, and their sum,
//                            which assert_equal_point ties to R            /root/reference/src/gadgets.rs:48-68, 99-130, 162-184
// All of them are BlsScalar values (affine coordinates, scalars embedded in F_q).  One row per signature, Montgomery
// limbs like every field element of the ABI:
//   single  (11):  u, R.u, R.v, PK.u, PK.v, m, c, SA.u, SA.v, SB.u, SB.v
//   double  (19):  u, R, R', PK, PK', m, c, SA, SB, SA', SB'            (points as (u, v))
//   vargen  (13):  u, R, PK, GEN, m, c, SA, SB
// SB = c * PK is obtained as R - SA (one addition instead of a 250-bit variable-base multiplication): the signer
// knows sk, so R = SA + SB holds by construction.  Signing itself is sign*_core's; u and c are the same scalars.
// ------------------------------------------------------------------------------------------------------------
SB_HD fq scalar_to_bls(const uint32_t* k) {  // JubJubScalar -> BlsScalar (the integer, embedded in F_q; k < r < q)
  fq x;
#pragma unroll
  for (int i = 0; i < 8; i++) x.v[i] = k[i];
  return fq_to_mont(x);
}
SB_HD ext ext_sub(const ext& a, const ext& b) { return p1p1_to_ext(ed_add(a, pniels_cneg(ext_to_pniels(b), true))); }

// SCHEME 0 single, 1 double, 2 vargen (GEN = the key's generator).  row: 11 / 19 / 13 field elements, written through
// `emit(k, value)` as they are produced (the kernel stores straight to the output array; no per-thread row buffer).
template <int SCHEME, class Emit>
SB_HD void witness_core(const uint32_t* sk, const uint32_t* nonce, const fq& m, const point_in& GEN, const uint32_t* combG,
                        const uint32_t* combGp, Emit&& emit) {
  constexpr int NB = SCHEME == 1 ? 2 : 1;  // bases
  fq Ru[NB], Rv[NB];
  int o = 1;  // slot 0 (u) is written once the challenge is known
  {
    ext P[2 * NB];  // R, PK per base
    fq z[2 * NB + 1], pre[2 * NB + 1];
#pragma unroll
    for (int b = 0; b < NB; b++) {
      P[2 * b] = SCHEME == 2 ? var_base_mul(GEN, nonce) : fixed_base_mul(b ? combGp : combG, nonce);
      P[2 * b + 1] = SCHEME == 2 ? var_base_mul(GEN, sk) : fixed_base_mul(b ? combGp : combG, sk);
    }
#pragma unroll
    for (int k = 0; k < 2 * NB; k++) z[k] = P[k].Z;
    z[2 * NB] = (SCHEME == 2 && !GEN.affine) ? GEN.Z : fq_one();
    batch_inverse(z, pre, 2 * NB + 1);
#pragma unroll
    for (int b = 0; b < NB; b++) {  // R (, R')
      Ru[b] = fq_mul(P[2 * b].X, z[2 * b]);
      Rv[b] = fq_mul(P[2 * b].Y, z[2 * b]);
      emit(o++, Ru[b]);
      emit(o++, Rv[b]);
    }
#pragma unroll
    for (int b = 0; b < NB; b++) {  // PK (, PK')
      emit(o++, fq_mul(P[2 * b + 1].X, z[2 * b + 1]));
      emit(o++, fq_mul(P[2 * b + 1].Y, z[2 * b + 1]));
    }
    if (SCHEME == 2) {  // GEN, affine
      emit(o++, fq_mul(GEN.U, z[2 * NB]));
      emit(o++, fq_mul(GEN.V, z[2 * NB]));
    }
  }
  uint32_t c[8], u[8];
  if (SCHEME == 1) chal5(Ru[0], Rv[0], Ru[NB - 1], Rv[NB - 1], m, c); else chal3(Ru[0], Rv[0], m, c);
  sign_finish(nonce, c, sk, u);
  emit(0, scalar_to_bls(u));
  emit(o++, m);
  emit(o++, scalar_to_bls(c));
  // SA = u * base, SB = R - SA
  ext S[2 * NB];
  fq z[2 * NB], pre[2 * NB];
#pragma unroll
  for (int b = 0; b < NB; b++) {
    S[2 * b] = SCHEME == 2 ? var_base_mul(GEN, u) : fixed_base_mul(b ? combGp : combG, u);
    S[2 * b + 1] = ext_sub(affine_to_ext(Ru[b], Rv[b]), S[2 * b]);
  }
#pragma unroll
  for (int k = 0; k < 2 * NB; k++) z[k] = S[k].Z;
  batch_inverse(z, pre, 2 * NB);
#pragma unroll
  for (int k = 0; k < 2 * NB; k++) {
    emit(o++, fq_mul(S[k].X, z[k]));
    emit(o++, fq_mul(S[k].Y, z[k]));
  }
}

// The same rows for a party that did not sign: from the public tuple (PK, u, R, m) alone.  PK2 = PK' (SCHEME 1) or GEN
// (SCHEME 2), Rp = R' (SCHEME 1); unused arguments are not read.  SA = u B and SB = c PK are both computed as scalar
// multiples (never SB = R - SA: R is only claimed here), and the return value is the verdict SA + SB == R (and
// SA' + SB' == R'), the same predicate sb200_verify* decides.  A tuple that fails keeps its true row; the row is zero
// (and the verdict 0) when u >= r or, with `check_points`, when an input point is not well formed.  Only public data
// enters, so both inversions are the Euclidean one.  Emits like witness_core; the zeroing masks the stores, the work
// runs for every lane.
template <int SCHEME, class Emit>
SB_HD bool verify_witness_core(const point_in& PK, const point_in& PK2, const uint32_t* u_in, const point_in& R,
                               const point_in& Rp, const fq& m, bool check_points, const uint32_t* combG,
                               const uint32_t* combGp, Emit&& emit) {
  constexpr int NB = SCHEME == 1 ? 2 : 1;                      // bases
  constexpr int NP = SCHEME == 0 ? 2 : SCHEME == 1 ? 4 : 3;    // input points, in row order: R (, R'), PK (, PK' | GEN)
  const point_in* P[4] = {&R, SCHEME == 1 ? &Rp : &PK, SCHEME == 1 ? &PK : &PK2, &PK2};
  const bool lt = scalar_lt_r(u_in);
  bool live = lt;
  if (check_points) {  // warp-uniform
#pragma unroll
    for (int k = 0; k < NP; k++) live &= point_well_formed(*P[k]);
  }
  auto put = [&](int k, const fq& v) { emit(k, live ? v : fq_zero()); };
  uint32_t u[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) u[i] = lt ? u_in[i] : 0u;  // in range for the comb; the row is zero anyway
  put(0, scalar_to_bls(u));
  // 1. the inputs in affine form: one inversion for all of them when they are projective (one flag for every point)
  fq au[NP], av[NP];
  if (R.affine) {
#pragma unroll
    for (int k = 0; k < NP; k++) {
      au[k] = P[k]->U;
      av[k] = P[k]->V;
    }
  } else {
    fq z[NP], pre[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) z[k] = P[k]->Z;
    batch_inverse(z, pre, NP);
#pragma unroll
    for (int k = 0; k < NP; k++) {
      au[k] = fq_mul(P[k]->U, z[k]);
      av[k] = fq_mul(P[k]->V, z[k]);
    }
  }
  int o = 1;
#pragma unroll
  for (int k = 0; k < NP; k++) {
    put(o++, au[k]);
    put(o++, av[k]);
  }
  // 2. the challenge
  if (SCHEME == 1) chal5(au[0], av[0], au[1], av[1], m, c); else chal3(au[0], av[0], m, c);
  put(o++, m);
  put(o++, scalar_to_bls(c));
  // 3. SA = u B (comb for G and G', window table for a variable generator), SB = c PK; 5. verdict SA + SB == R
  ext S[2 * NB];
  bool ok = live;
#pragma unroll
  for (int b = 0; b < NB; b++) {
    const point_in key = {au[NB + b], av[NB + b], fq_one(), true};
    if (SCHEME == 2) {
      const point_in gen = {au[2], av[2], fq_one(), true};
      S[2 * b] = var_base_mul(gen, u);
    } else {
      S[2 * b] = fixed_base_mul(b ? combGp : combG, u);
    }
    S[2 * b + 1] = var_base_mul(key, c);
    const point_in rr = {au[b], av[b], fq_one(), true};
    ok &= p1p1_equals(ed_add(S[2 * b], ext_to_pniels(S[2 * b + 1])), rr);
  }
  // 4. the outputs in affine form: one inversion
  fq z[2 * NB], pre[2 * NB];
#pragma unroll
  for (int k = 0; k < 2 * NB; k++) z[k] = S[k].Z;
  batch_inverse(z, pre, 2 * NB);
#pragma unroll
  for (int k = 0; k < 2 * NB; k++) {
    put(o++, fq_mul(S[k].X, z[k]));
    put(o++, fq_mul(S[k].Y, z[k]));
  }
  return ok;
}

// Verification against a registered key (include/schnorr_b200_keyset.h).  `tabs`: the keyset's per-key combs, key k's
// at tabs + k * NT * KS_TABLE_WORDS (NT = 1 for SCHEME 0: PK; 2 for SCHEME 1: PK, PK'; 2 for SCHEME 2: PK, GEN), `key_ok`
// bit k = every point of key k is well formed.  c_out = the challenge sb200_verify* writes; the verdict is the predicate
// it decides (u B + c PK == R, and u G' + c PK' == R' for SCHEME 1), with u B by the 16-bit comb of G / G' or, for a
// variable generator, by the key's own comb of GEN.  Exact on the whole curve: no short vector, no fallback.  The verdict
// is 0 when u >= r, key >= n_keys (key 0's table is read instead, never past the end), key_ok is clear, or with
// `check_points` R (R') is not well formed -- by mask: every lane runs the same work.
template <int SCHEME>
SB_HD bool verify_keyset_core(const uint32_t* tabs, int64_t n_keys, const uint32_t* key_ok, uint32_t key, const uint32_t* u_in,
                              const point_in& R, const point_in& Rp, const fq& m, bool check_points, const uint32_t* combG,
                              const uint32_t* combGp, uint32_t* c_out) {
  constexpr int NT = SCHEME == 0 ? 1 : 2;
  if (SCHEME == 1) verify_double_hash_core(R, Rp, m, c_out); else verify_hash_core(R, m, c_out);
  const bool known = (int64_t)key < n_keys;
  const uint64_t k = known ? key : 0u;
  const bool lt = scalar_lt_r(u_in);
  bool ok = known & ((key_ok[k >> 5] >> (k & 31) & 1u) != 0) & lt;
  uint32_t u[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u[i] = lt ? u_in[i] : 0u;  // in range for the recoding; the verdict is 0 anyway
    c[i] = c_out[i];
  }
  recode_offset<KS_BITS>(c);
  const uint32_t* tab = tabs + k * NT * KS_TABLE_WORDS;
  if (SCHEME == 2) {  // u GEN + c PK, both from the key's combs
    recode_offset<KS_BITS>(u);
    p1p1 s = ed_comb_add_w<KS_BITS>(ext_identity(), tab + KS_TABLE_WORDS, u);
    s = ed_comb_add_w<KS_BITS>(p1p1_to_ext(s), tab, c);
    ok &= p1p1_equals(s, R);
  } else {  // u G + c PK (and u G' + c PK'): one copy of the curve code
    recode_offset<COMB_BITS>(u);
#pragma unroll 1
    for (int b = 0; b < NT; b++) {
      p1p1 s = ed_comb_add(ext_identity(), b ? combGp : combG, u);
      s = ed_comb_add_w<KS_BITS>(p1p1_to_ext(s), tab + b * KS_TABLE_WORDS, c);
      ok &= p1p1_equals(s, b ? Rp : R);
    }
  }
  if (check_points) {  // warp-uniform
    ok &= point_well_formed(R);
    if (SCHEME == 1) ok &= point_well_formed(Rp);
  }
  return ok;
}

}  // namespace sb200
