// JubJub group law for sm_100a: a = -1 twisted Edwards  -u^2 + v^2 = 1 + d u^2 v^2  over Fq.
//
// Replaces `JubJubExtended: Mul<JubJubScalar>, Add, PartialEq` (dusk-jubjub ^0.14) as used at
// /root/reference/src/keys/public.rs:63,127-129,236-243,340,411-414 and
// /root/reference/src/keys/secret.rs:159,231-232,373,440.
//
// -1 is a square and d a non-square in Fq, so the unified extended addition below is complete: no
// exceptional cases for any pair of curve points (identity, small-order points, P + P, P - P).
// The reference's `*` computes the integer multiple s*P with a 252-step double-and-add; any
// algorithm that returns the same group element gives an equal point under its projective `==`
// (/root/reference/tests/keys.rs:52-58), so the schedules here are free to differ:
//   * variable base  : signed fixed windows (regular recoding, identical control flow in all 32
//                      lanes -- a wNAF's data-dependent add positions would diverge per lane);
//   * fixed base G/G': comb of 16-bit signed windows, 16 mixed additions and no doublings.
#pragma once
#include "fq.cuh"

namespace sb200 {

struct proj {  // (X : Y : Z), x = X/Z, y = Y/Z
  fq X, Y, Z;
};
struct ext {  // extended: T = X*Y/Z
  fq X, Y, Z, T;
};
struct p1p1 {  // completed point: X = E*F, Y = G*H, Z = F*G, T = E*H
  fq E, F, G, H;
};
struct pniels {  // projective Niels form of a point: (Y+X, Y-X, Z, 2d*T)
  fq YpX, YmX, Z, T2d;
};
struct aniels {  // affine Niels form (Z = 1): (y+x, y-x, 2d*x*y)
  fq YpX, YmX, T2d;
};

// INL = true: multiplier bodies inlined (used inside the "fat" out-of-line point operations below);
// INL = false: the out-of-line multiplier.
template <bool INL>
SB_HD fq mulT(const fq& a, const fq& b) {
  if (INL) return fq_mul_inl(a, b);
  return fq_mul(a, b);
}
template <bool INL>
SB_HD fq sqrT(const fq& a) {
  if (INL) return fq_sqr_inl(a);
  return fq_sqr(a);
}

SB_HD fq ed_2d() {
  const fq c = {SB200_ED_2D_INIT};
  return c;
}
SB_HD fq ed_d() {
  const fq c = {SB200_ED_D_INIT};
  return c;
}

SB_HD ext ext_identity() {
  ext r;
  r.X = fq_zero();
  r.Y = fq_one();
  r.Z = fq_one();
  r.T = fq_zero();
  return r;
}

template <bool INL = false>
SB_HD proj p1p1_to_proj(const p1p1& c) {
  proj r;
  if (INL) {
    r.X = fq_mul_inl(c.E, c.F);
    r.Y = fq_mul_inl(c.G, c.H);
  } else {
    fq_mul2(c.E, c.F, c.G, c.H, r.X, r.Y);
  }
  r.Z = mulT<INL>(c.F, c.G);
  return r;
}
template <bool INL = false>
SB_HD ext p1p1_to_ext(const p1p1& c) {
  ext r;
  if (INL) {
    r.X = fq_mul_inl(c.E, c.F);
    r.Y = fq_mul_inl(c.G, c.H);
    r.Z = fq_mul_inl(c.F, c.G);
    r.T = fq_mul_inl(c.E, c.H);
  } else {
    fq_mul2(c.E, c.F, c.G, c.H, r.X, r.Y);
    fq_mul2(c.F, c.G, c.E, c.H, r.Z, r.T);
  }
  return r;
}

// 2P, 4 squarings (dbl-2008-hwcd with a = -1, signs arranged so H = A + B, F = C - G)
template <bool INL = false>
SB_HD p1p1 ed_dbl(const fq& X, const fq& Y, const fq& Z) {
  fq A, B, C, S;
  if (INL) {
    A = fq_sqr_inl(X);
    B = fq_sqr_inl(Y);
    C = fq_sqr_inl(Z);
    S = fq_sqr_inl(fq_add(X, Y));
  } else {
    fq_sqr2(X, Y, A, B);
    fq_sqr2(Z, fq_add(X, Y), C, S);
  }
  C = fq_dbl(C);
  p1p1 r;
  r.H = fq_add(A, B);
  r.G = fq_sub(B, A);
  r.E = fq_sub(S, r.H);
  r.F = fq_sub(C, r.G);
  return r;
}

// P + Q, Q in projective Niels form: 4 multiplications (add-2008-hwcd-3, k = 2d)
template <bool INL = false>
SB_HD p1p1 ed_add(const ext& p, const pniels& q) {
  fq A, B, C, D;
  if (INL) {
    A = fq_mul_inl(fq_sub(p.Y, p.X), q.YmX);
    B = fq_mul_inl(fq_add(p.Y, p.X), q.YpX);
    C = fq_mul_inl(p.T, q.T2d);
    D = fq_mul_inl(p.Z, q.Z);
  } else {
    fq_mul2(fq_sub(p.Y, p.X), q.YmX, fq_add(p.Y, p.X), q.YpX, A, B);
    fq_mul2(p.T, q.T2d, p.Z, q.Z, C, D);
  }
  D = fq_dbl(D);
  p1p1 r;
  r.E = fq_sub(B, A);
  r.F = fq_sub(D, C);
  r.G = fq_add(D, C);
  r.H = fq_add(B, A);
  return r;
}

// P + Q, Q affine Niels: 3 multiplications
template <bool INL = false>
SB_HD p1p1 ed_add(const ext& p, const aniels& q) {
  fq A, B;
  if (INL) {
    A = fq_mul_inl(fq_sub(p.Y, p.X), q.YmX);
    B = fq_mul_inl(fq_add(p.Y, p.X), q.YpX);
  } else {
    fq_mul2(fq_sub(p.Y, p.X), q.YmX, fq_add(p.Y, p.X), q.YpX, A, B);
  }
  fq C = mulT<INL>(p.T, q.T2d);
  fq D = fq_dbl(p.Z);
  p1p1 r;
  r.E = fq_sub(B, A);
  r.F = fq_sub(D, C);
  r.G = fq_add(D, C);
  r.H = fq_add(B, A);
  return r;
}

SB_HD pniels ext_to_pniels(const ext& p) {
  pniels r;
  r.YpX = fq_add(p.Y, p.X);
  r.YmX = fq_sub(p.Y, p.X);
  r.Z = p.Z;
  r.T2d = fq_mul(p.T, ed_2d());
  return r;
}

SB_HD pniels pniels_identity() {
  pniels r;
  r.YpX = fq_one();
  r.YmX = fq_one();
  r.Z = fq_one();
  r.T2d = fq_zero();
  return r;
}

// -Q:  swap (Y+X, Y-X), negate 2dT.  Branch-free select.
SB_HD pniels pniels_cneg(const pniels& q, bool neg) {
  pniels r;
  r.YpX = fq_select(q.YpX, q.YmX, neg);
  r.YmX = fq_select(q.YmX, q.YpX, neg);
  r.Z = q.Z;
  r.T2d = fq_select(q.T2d, fq_neg(q.T2d), neg);
  return r;
}
SB_HD aniels aniels_cneg(const aniels& q, bool neg) {
  aniels r;
  r.YpX = fq_select(q.YpX, q.YmX, neg);
  r.YmX = fq_select(q.YmX, q.YpX, neg);
  r.T2d = fq_select(q.T2d, fq_neg(q.T2d), neg);
  return r;
}

// (U : V : Z) with Z != 0  ->  extended (U*Z : V*Z : Z^2 : U*V)
SB_HD ext proj_to_ext(const fq& U, const fq& V, const fq& Z) {
  ext r;
  r.X = fq_mul(U, Z);
  r.Y = fq_mul(V, Z);
  r.Z = fq_sqr(Z);
  r.T = fq_mul(U, V);
  return r;
}
SB_HD ext affine_to_ext(const fq& u, const fq& v) {
  ext r;
  r.X = u;
  r.Y = v;
  r.Z = fq_one();
  r.T = fq_mul(u, v);
  return r;
}

// ------------------------------------------------------------------------------------------
// scalar recoding.  k (canonical, 8 x u32 LE) + "all halves" offset; window i of the sum minus
// 2^(W-1) is the signed digit, so no carries are needed when walking windows MSB-first.
// ------------------------------------------------------------------------------------------
template <int W>
SB_HD void recode_offset(uint32_t* k) {  // k += sum_i 2^(W-1) * 2^(W*i) over all windows that fit in 256 bits
  static_assert(W == 4 || W == 8 || W == 16, "window widths that tile 32-bit limbs");
  const uint32_t c = (W == 4) ? 0x88888888u : (W == 8) ? 0x80808080u : 0x80008000u;
  const uint32_t off[8] = {c, c, c, c, c, c, c, c};
  add8(k, k, off);  // k < 2^252 => no carry out
}
template <int W>
SB_HD int recode_digit(const uint32_t* k, int i) {  // signed digit of window i, in [-2^(W-1), 2^(W-1))
  const int per = 32 / W;
  uint32_t w = (k[i / per] >> ((i % per) * W)) & ((1u << W) - 1u);
  return (int)w - (1 << (W - 1));
}

// ------------------------------------------------------------------------------------------
// variable-base:  acc = k * P, k < 2^252 given already offset-recoded for W = 4 (64 windows; digits
// in [-8, 7]).  `tab` holds 0P..8P in projective Niels form (9 entries, thread-private).
// `nwin` windows are processed (63 is enough for a challenge c < 2^250, 64 for any k < 2^252).
// Returns the completed form of the last addition.
// ------------------------------------------------------------------------------------------
SB_HD void vartable_build(pniels* tab, const ext& P) {
  tab[0] = pniels_identity();
  tab[1] = ext_to_pniels(P);
  ext cur = P;
#pragma unroll 1
  for (int i = 2; i <= 8; i++) {
    cur = p1p1_to_ext(ed_add(cur, tab[1]));
    tab[i] = ext_to_pniels(cur);
  }
}

// ---- "fat" out-of-line point steps --------------------------------------------------------------
// One call per point operation with the 7-8 multiplications inlined inside: the completed point travels
// in registers (32 in, 32 out), so the per-multiplication argument shuffling of the out-of-line
// multiplier (ptxas emits half of those moves as IMAD.MOV on the saturated FMA-heavy pipe) disappears
// from the hot loops, while the code stays small enough for the instruction cache.
#ifndef SB_FAT_OOL
#define SB_FAT_OOL 0  // measured: 27 KB per fat step thrashes the instruction cache (stall_no_instruction 0.12 -> 1.24); kept for experiments
#endif
#if defined(__CUDACC__) && SB_FAT_OOL
static __device__ __noinline__ p1p1 pt_dbl_ool(p1p1 c) {
  proj p = p1p1_to_proj<true>(c);
  return ed_dbl<true>(p.X, p.Y, p.Z);
}
#endif
// c <- 2c   (3M + 4S)
SB_HD p1p1 pt_dbl(const p1p1& c) {
#if defined(__CUDA_ARCH__) && SB_FAT_OOL
  return pt_dbl_ool(c);
#else
  proj p = p1p1_to_proj(c);
  return ed_dbl(p.X, p.Y, p.Z);
#endif
}

#ifndef SB_TABLE_PREFETCH
#define SB_TABLE_PREFETCH 0
#endif
#ifndef SB_DBL_ROLL
#define SB_DBL_ROLL 4  // how many of the 4 doublings per window run as a rolled loop
#endif
SB_HD pniels vartable_lookup(const pniels* tab, int d) {
  bool neg = d < 0;
  int idx = neg ? -d : d;
  return pniels_cneg(tab[idx], neg);
}

SB_HD p1p1 ed_mul_var(const pniels* tab, const uint32_t* k_rec, int nwin) {
  // top window: acc = digit * P directly (identity + entry)
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tab, recode_digit<4>(k_rec, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
    // rolled: four copies of the doubling's call sequence make the loop body 25 KB, and together with the
    // multiplier bodies it no longer fits the 32 KB L1.5 instruction cache (ncu: stall_no_instruction 1.3 per issue)
#pragma unroll 1
    for (int k = 0; k < SB_DBL_ROLL; k++) c = pt_dbl(c);
#if SB_DBL_ROLL < 4
#pragma unroll
    for (int k = SB_DBL_ROLL; k < 4; k++) c = pt_dbl(c);
#endif
    ext e = p1p1_to_ext(c);
    c = ed_add(e, vartable_lookup(tab, recode_digit<4>(k_rec, i)));
  }
  return c;
}

// Straus: k1*P1 + k2*P2 with shared doublings (variable-generator verification,
// /root/reference/src/keys/public.rs:411-412).
SB_HD p1p1 ed_mul_var2(const pniels* tab1, const uint32_t* k1_rec, const pniels* tab2, const uint32_t* k2_rec, int nwin) {
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tab1, recode_digit<4>(k1_rec, nwin - 1)));
  c = ed_add(p1p1_to_ext(c), vartable_lookup(tab2, recode_digit<4>(k2_rec, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
    // rolled: four copies of the doubling's call sequence make the loop body 25 KB, and together with the
    // multiplier bodies it no longer fits the 32 KB L1.5 instruction cache (ncu: stall_no_instruction 1.3 per issue)
#pragma unroll 1
    for (int k = 0; k < SB_DBL_ROLL; k++) c = pt_dbl(c);
#if SB_DBL_ROLL < 4
#pragma unroll
    for (int k = SB_DBL_ROLL; k < 4; k++) c = pt_dbl(c);
#endif
    ext e = p1p1_to_ext(c);
    c = ed_add(e, vartable_lookup(tab1, recode_digit<4>(k1_rec, i)));
    e = p1p1_to_ext(c);
    c = ed_add(e, vartable_lookup(tab2, recode_digit<4>(k2_rec, i)));
  }
  return c;
}

// The same with the two additions of a window as a 2-trip loop: one copy of the conversion + lookup + addition
// sequence in the hot loop (7 KB less code in a 32 KB instruction cache).
SB_HD p1p1 ed_mul_var2_rolled(const pniels* tab1, const uint32_t* k1_rec, const pniels* tab2, const uint32_t* k2_rec, int nwin) {
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tab1, recode_digit<4>(k1_rec, nwin - 1)));
  c = ed_add(p1p1_to_ext(c), vartable_lookup(tab2, recode_digit<4>(k2_rec, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
#if defined(__CUDA_ARCH__) && SB_TABLE_PREFETCH
    // tables in global memory (SB_EC_GLOBAL_TABLES): the two entries this window will add are known now -- pull their
    // 128-byte lines into L1 while the four doublings run
    {
      int d1 = recode_digit<4>(k1_rec, i), d2 = recode_digit<4>(k2_rec, i);
      asm volatile("prefetch.global.L1 [%0];" ::"l"(tab1 + (d1 < 0 ? -d1 : d1)));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(tab2 + (d2 < 0 ? -d2 : d2)));
    }
#endif
#pragma unroll 1
    for (int k = 0; k < 4; k++) c = pt_dbl(c);
#pragma unroll 1
    for (int t = 0; t < 2; t++) {
      const pniels* tab = t ? tab2 : tab1;
      const uint32_t* kr = t ? k2_rec : k1_rec;
      ext e = p1p1_to_ext(c);
      c = ed_add(e, vartable_lookup(tab, recode_digit<4>(kr, i)));
    }
  }
  return c;
}

#if defined(__CUDACC__)
// The same loop for window tables that live in GLOBAL memory (thread-major, one contiguous 128-byte entry per lookup:
// SB_EC_GLOBAL_TABLES), with the two entries of a window staged into shared memory by cp.async while its four doublings
// run: the lookups become conflict-free LDS.128 of data that is already on chip, and no register is held for them.
// `stage` = this CTA's 2 x 8 x blockDim.x uint4 (each thread only ever touches its own slots: no barrier needed).
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ p1p1 ed_mul_var2_staged(const pniels* tab1, const uint32_t* k1_rec, const pniels* tab2, const uint32_t* k2_rec,
                                                   int nwin, uint4* stage) {
  const int nthr = blockDim.x, tid = threadIdx.x;
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tab1, recode_digit<4>(k1_rec, nwin - 1)));
  c = ed_add(p1p1_to_ext(c), vartable_lookup(tab2, recode_digit<4>(k2_rec, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
    const int d1 = recode_digit<4>(k1_rec, i), d2 = recode_digit<4>(k2_rec, i);
    {
      const uint4* s1 = reinterpret_cast<const uint4*>(tab1 + (d1 < 0 ? -d1 : d1));
      const uint4* s2 = reinterpret_cast<const uint4*>(tab2 + (d2 < 0 ? -d2 : d2));
#pragma unroll
      for (int k = 0; k < 8; k++) {
        cp_async16(stage + k * nthr + tid, s1 + k);
        cp_async16(stage + (8 + k) * nthr + tid, s2 + k);
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
#pragma unroll 1
    for (int k = 0; k < 4; k++) c = pt_dbl(c);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll 1
    for (int t = 0; t < 2; t++) {
      const uint4* sp = stage + (8 * t) * nthr + tid;
      pniels q;
      uint4 v0 = sp[0], v1 = sp[nthr], v2 = sp[2 * nthr], v3 = sp[3 * nthr], v4 = sp[4 * nthr], v5 = sp[5 * nthr], v6 = sp[6 * nthr],
            v7 = sp[7 * nthr];
      q.YpX = {{v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w}};
      q.YmX = {{v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w}};
      q.Z = {{v4.x, v4.y, v4.z, v4.w, v5.x, v5.y, v5.z, v5.w}};
      q.T2d = {{v6.x, v6.y, v6.z, v6.w, v7.x, v7.y, v7.z, v7.w}};
      ext e = p1p1_to_ext(c);
      c = ed_add(e, pniels_cneg(q, (t ? d2 : d1) < 0));
    }
  }
  return c;
}
// three tables (lat3.cuh): 24 staged uint4 per thread and window
__device__ __forceinline__ p1p1 ed_mul_var3_staged(const pniels* tabs, const uint32_t* kr, int nwin, uint4* stage);
#endif

// Straus over THREE variable points (the variable-generator verification with short scalars, lat3.cuh):
// tabs = 27 entries (three 9-entry tables back to back), kr = three offset-recoded scalars (8 limbs each).
// One copy of the conversion + lookup + addition sequence, as in ed_mul_var2_rolled.
SB_HD p1p1 ed_mul_var3_rolled(const pniels* tabs, const uint32_t* kr, int nwin) {
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tabs, recode_digit<4>(kr, nwin - 1)));
#pragma unroll 1
  for (int t = 1; t < 3; t++) c = ed_add(p1p1_to_ext(c), vartable_lookup(tabs + 9 * t, recode_digit<4>(kr + 8 * t, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
#pragma unroll 1
    for (int k = 0; k < 4; k++) c = pt_dbl(c);
#pragma unroll 1
    for (int t = 0; t < 3; t++) {
      ext e = p1p1_to_ext(c);
      c = ed_add(e, vartable_lookup(tabs + 9 * t, recode_digit<4>(kr + 8 * t, i)));
    }
  }
  return c;
}

#if defined(__CUDACC__)
__device__ __forceinline__ p1p1 ed_mul_var3_staged(const pniels* tabs, const uint32_t* kr, int nwin, uint4* stage) {
  const int nthr = blockDim.x, tid = threadIdx.x;
  p1p1 c = ed_add(ext_identity(), vartable_lookup(tabs, recode_digit<4>(kr, nwin - 1)));
#pragma unroll 1
  for (int t = 1; t < 3; t++) c = ed_add(p1p1_to_ext(c), vartable_lookup(tabs + 9 * t, recode_digit<4>(kr + 8 * t, nwin - 1)));
#pragma unroll 1
  for (int i = nwin - 2; i >= 0; i--) {
    int d[3];
#pragma unroll
    for (int t = 0; t < 3; t++) {
      d[t] = recode_digit<4>(kr + 8 * t, i);
      const uint4* sp = reinterpret_cast<const uint4*>(tabs + 9 * t + (d[t] < 0 ? -d[t] : d[t]));
#pragma unroll
      for (int k = 0; k < 8; k++) cp_async16(stage + (8 * t + k) * nthr + tid, sp + k);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll 1
    for (int k = 0; k < 4; k++) c = pt_dbl(c);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    const unsigned negs = (d[0] < 0 ? 1u : 0u) | (d[1] < 0 ? 2u : 0u) | (d[2] < 0 ? 4u : 0u);
#pragma unroll 1
    for (int t = 0; t < 3; t++) {
      const uint4* sp = stage + (8 * t) * nthr + tid;
      pniels q;
      uint4 v0 = sp[0], v1 = sp[nthr], v2 = sp[2 * nthr], v3 = sp[3 * nthr], v4 = sp[4 * nthr], v5 = sp[5 * nthr], v6 = sp[6 * nthr],
            v7 = sp[7 * nthr];
      q.YpX = {{v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w}};
      q.YmX = {{v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w}};
      q.Z = {{v4.x, v4.y, v4.z, v4.w, v5.x, v5.y, v5.z, v5.w}};
      q.T2d = {{v6.x, v6.y, v6.z, v6.w, v7.x, v7.y, v7.z, v7.w}};
      ext e = p1p1_to_ext(c);
      c = ed_add(e, pniels_cneg(q, ((negs >> t) & 1u) != 0));
    }
  }
  return c;
}
#endif

// ------------------------------------------------------------------------------------------
// fixed-base comb.  Table layout: window j, entry e (0..2^(W-1)) = e * 2^(W*j) * B in affine Niels form,
// entry 0 = identity; 96 bytes per entry.  acc += k * B with k offset-recoded (W = COMB_BITS).
// ------------------------------------------------------------------------------------------
// Window width of the fixed-base comb.  16 bits on the device: 16 additions per scalar and a 50 MB table per
// generator (16 x 32769 x 96 B) that simply lives in HBM/L2 -- a lookup is 96 bytes per ~4000 cycles of
// addition, 30 GB/s at full speed.  The CPU test build uses 8 bits (the emulated table build is slow).
#ifndef SB_COMB_BITS
#if defined(__CUDACC__)
#define SB_COMB_BITS 16
#else
#define SB_COMB_BITS 8
#endif
#endif
constexpr int COMB_BITS = SB_COMB_BITS;
constexpr int COMB_WINDOWS = 256 / COMB_BITS;
constexpr int COMB_ENTRIES = (1 << (COMB_BITS - 1)) + 1;

SB_HD aniels comb_load(const uint32_t* table, int j, int e) {
  const uint4* p = reinterpret_cast<const uint4*>(table) + (size_t)(j * COMB_ENTRIES + e) * 6;
  uint4 q0 = p[0], q1 = p[1], q2 = p[2], q3 = p[3], q4 = p[4], q5 = p[5];
  aniels r;
  r.YpX = {{q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w}};
  r.YmX = {{q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, q3.z, q3.w}};
  r.T2d = {{q4.x, q4.y, q4.z, q4.w, q5.x, q5.y, q5.z, q5.w}};
  return r;
}

// acc (extended) += k*B ; returns completed form of the last addition (use p1p1_to_ext / compare).
SB_HD p1p1 ed_comb_add(ext acc, const uint32_t* table, const uint32_t* k_rec) {
  p1p1 c;
#pragma unroll 1
  for (int j = 0; j < COMB_WINDOWS; j++) {
    int d = recode_digit<COMB_BITS>(k_rec, j);
    bool neg = d < 0;
    aniels n = aniels_cneg(comb_load(table, j, neg ? -d : d), neg);
    c = ed_add(acc, n);
    if (j + 1 < COMB_WINDOWS) acc = p1p1_to_ext(c);
  }
  return c;
}

// ------------------------------------------------------------------------------------------
// per-key comb of a registered public key (include/schnorr_b200_keyset.h): the layout of the G comb with a fixed 8-bit
// window on the device and in the host build alike (independent of SB_COMB_BITS).  Window j, entry e (0..128) =
// e * 2^(8j) * P in affine Niels form, entry 0 = identity: 32 windows x 129 entries x 96 B = 396 288 B per point, and
// k * P (k < 2^252: 32 signed digits in [-128, 127]) is 32 mixed additions with no doubling.  Every entry is an exact
// integer multiple of P, so the sum is k * P on the whole curve, torsion points included.  Width 4 would take 55 KB and
// 64 additions per point; width 8 halves the additions for 7x the memory.  180 GB hold about 450 000 single-key keys
// (225 000 double-key or variable-generator keys, which have two points each) less the batch buffers: 2^16 single-key
// keys take 26 GB.
// ------------------------------------------------------------------------------------------
constexpr int KS_BITS = 8;
constexpr int KS_WINDOWS = 256 / KS_BITS;
constexpr int KS_ENTRIES = (1 << (KS_BITS - 1)) + 1;
constexpr size_t KS_TABLE_WORDS = (size_t)KS_WINDOWS * KS_ENTRIES * 24;  // 99 072 words per point

SB_HD aniels aniels_load(const uint32_t* entry) {  // one 96-byte affine Niels entry (six 16-byte loads)
  const uint4* p = reinterpret_cast<const uint4*>(entry);
  uint4 q0 = p[0], q1 = p[1], q2 = p[2], q3 = p[3], q4 = p[4], q5 = p[5];
  aniels r;
  r.YpX = {{q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w}};
  r.YmX = {{q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, q3.z, q3.w}};
  r.T2d = {{q4.x, q4.y, q4.z, q4.w, q5.x, q5.y, q5.z, q5.w}};
  return r;
}

// acc (extended) += k*B for the comb of W-bit windows (2^(W-1) + 1 entries each) at `table`; k offset-recoded for W.
// ed_comb_add's loop with the table layout as a parameter.
template <int W>
SB_HD p1p1 ed_comb_add_w(ext acc, const uint32_t* table, const uint32_t* k_rec) {
  constexpr int NW = 256 / W, NE = (1 << (W - 1)) + 1;
  p1p1 c;
#pragma unroll 1
  for (int j = 0; j < NW; j++) {
    const int d = recode_digit<W>(k_rec, j);
    const bool neg = d < 0;
    c = ed_add(acc, aniels_cneg(aniels_load(table + (size_t)(j * NE + (neg ? -d : d)) * 24), neg));
    if (j + 1 < NW) acc = p1p1_to_ext(c);
  }
  return c;
}

// ------------------------------------------------------------------------------------------
// Address-oblivious scalar multiplication (SB200_SIGN_OBLIVIOUS): the same group elements as above with no
// memory address and no branch depending on the (secret) scalar -- the property of the reference's ladder
// (`acc += select(identity, P, bit)`, dusk-jubjub) that the 16-bit comb gives up by indexing a 50 MB table with
// nonce / key digits.
//   fixed base : comb of 4-bit signed windows, 64 windows x 8 entries (1..8) x 96 B = 48 KB per generator, staged in
//                SHARED memory; every lane reads all 8 entries of the window (same addresses in all lanes: a
//                broadcast, conflict-free) and keeps one by mask; 64 mixed additions, no doublings.
//   variable   : the 9-entry window table is scanned with masks instead of being indexed.
// ------------------------------------------------------------------------------------------
constexpr int CT_WINDOWS = 64, CT_ENTRIES = 8;
constexpr int CT_TABLE_WORDS = CT_WINDOWS * CT_ENTRIES * 24;  // 12 288 words = 48 KB

SB_HD aniels comb4_lookup_oblivious(const uint32_t* tab, int j, int d) {
  const uint32_t neg = (uint32_t)(d >> 31);             // all ones if d < 0
  const uint32_t idx = ((uint32_t)d ^ neg) - neg;        // |d| in 0..8
  uint32_t w[24];
#pragma unroll
  for (int k = 0; k < 24; k++) w[k] = 0;
  const uint4* base = reinterpret_cast<const uint4*>(tab) + (size_t)j * CT_ENTRIES * 6;
#pragma unroll 1
  for (uint32_t e = 1; e <= (uint32_t)CT_ENTRIES; e++) {
    const uint32_t x = idx ^ e;
    const uint32_t mask = (uint32_t)((int32_t)((x | (0u - x)) ^ 0x80000000u) >> 31);  // all ones iff idx == e
#pragma unroll
    for (int q = 0; q < 6; q++) {
      const uint4 v = base[(e - 1) * 6 + q];
      w[4 * q] |= v.x & mask; w[4 * q + 1] |= v.y & mask; w[4 * q + 2] |= v.z & mask; w[4 * q + 3] |= v.w & mask;
    }
  }
  const bool zero = idx == 0;  // digit 0: the identity (1, 1, 0)
  aniels r;
  const fq one = fq_one();
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const uint32_t a = zero ? one.v[k] : w[k], b = zero ? one.v[k] : w[8 + k];
    r.YpX.v[k] = neg ? b : a;   // -Q: swap (y + x, y - x) ...
    r.YmX.v[k] = neg ? a : b;
    r.T2d.v[k] = w[16 + k];
  }
  r.T2d = fq_select(r.T2d, fq_neg(r.T2d), neg != 0);  // ... and negate 2d x y
  return r;
}

// k * B for the generator whose 4-bit comb table is `tab` (shared memory on the device); k < 2^252 canonical
SB_HD ext fixed_base_mul_oblivious(const uint32_t* tab, const uint32_t* k) {
  uint32_t kr[8];
#pragma unroll
  for (int i = 0; i < 8; i++) kr[i] = k[i];
  recode_offset<4>(kr);
  ext acc = ext_identity();
#pragma unroll 1
  for (int j = 0; j < CT_WINDOWS; j++) acc = p1p1_to_ext(ed_add(acc, comb4_lookup_oblivious(tab, j, recode_digit<4>(kr, j))));
  return acc;
}

SB_HD pniels vartable_lookup_oblivious(const pniels* tab, int d) {
  const uint32_t neg = (uint32_t)(d >> 31);
  const uint32_t idx = ((uint32_t)d ^ neg) - neg;
  pniels r;
#pragma unroll
  for (int k = 0; k < 8; k++) r.YpX.v[k] = r.YmX.v[k] = r.Z.v[k] = r.T2d.v[k] = 0;
#pragma unroll 1
  for (uint32_t e = 0; e <= 8; e++) {
    const uint32_t x = idx ^ e;
    const uint32_t mask = (uint32_t)((int32_t)((x | (0u - x)) ^ 0x80000000u) >> 31);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      r.YpX.v[k] |= tab[e].YpX.v[k] & mask; r.YmX.v[k] |= tab[e].YmX.v[k] & mask;
      r.Z.v[k] |= tab[e].Z.v[k] & mask; r.T2d.v[k] |= tab[e].T2d.v[k] & mask;
    }
  }
  return pniels_cneg(r, neg != 0);
}

// k * P with the table scanned, not indexed (64 windows; k < 2^252, offset-recoded for W = 4 by the caller)
SB_HD p1p1 ed_mul_var_oblivious(const pniels* tab, const uint32_t* k_rec) {
  p1p1 c = ed_add(ext_identity(), vartable_lookup_oblivious(tab, recode_digit<4>(k_rec, 63)));
#pragma unroll 1
  for (int i = 62; i >= 0; i--) {
#pragma unroll 1
    for (int k = 0; k < 4; k++) c = pt_dbl(c);
    c = ed_add(p1p1_to_ext(c), vartable_lookup_oblivious(tab, recode_digit<4>(k_rec, i)));
  }
  return c;
}

}  // namespace sb200

namespace sb200 {

// One comb-table entry: e * 2^(W*j) * B in affine Niels form (entry 0 = identity), written as 24 limbs.
// Run once per (j, e) at context creation (init kernel) -- plain double-and-add, speed irrelevant.
SB_HD void comb_build_entry_w(const fq& Bu, const fq& Bv, int j, int e, uint32_t* out24, const int BITS) {
  ext base = affine_to_ext(Bu, Bv);
  pniels nb = ext_to_pniels(base);
  ext acc = ext_identity();
  // scalar = e << (8*j); walk its bits MSB-first: bits 8*j+7 .. 0
#pragma unroll 1
  for (int bit = BITS * j + BITS - 1; bit >= 0; bit--) {
    acc = p1p1_to_ext(ed_dbl(acc.X, acc.Y, acc.Z));
    int eb = bit - BITS * j;
    bool set = (eb >= 0) && ((e >> eb) & 1);
    ext sum = p1p1_to_ext(ed_add(acc, nb));
    acc.X = fq_select(acc.X, sum.X, set);
    acc.Y = fq_select(acc.Y, sum.Y, set);
    acc.Z = fq_select(acc.Z, sum.Z, set);
    acc.T = fq_select(acc.T, sum.T, set);
  }
  fq zi = fq_inv(acc.Z);
  fq x = fq_mul(acc.X, zi), y = fq_mul(acc.Y, zi);
  fq ypx = fq_add(y, x), ymx = fq_sub(y, x), t2d = fq_mul(fq_mul(x, y), ed_2d());
#pragma unroll
  for (int i = 0; i < 8; i++) {
    out24[i] = ypx.v[i];
    out24[8 + i] = ymx.v[i];
    out24[16 + i] = t2d.v[i];
  }
}
SB_HD void comb_build_entry(const fq& Bu, const fq& Bv, int j, int e, uint32_t* out24) { comb_build_entry_w(Bu, Bv, j, e, out24, COMB_BITS); }
// entry of the oblivious path's 4-bit comb: e * 16^j * B, e = 1..8
SB_HD void comb4_build_entry(const fq& Bu, const fq& Bv, int j, int e, uint32_t* out24) { comb_build_entry_w(Bu, Bv, j, e, out24, 4); }

}  // namespace sb200
