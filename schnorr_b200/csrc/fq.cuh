// 255-bit Montgomery arithmetic on 8 x 32-bit limbs for sm_100a.
//
//   Fq  = BLS12-381 scalar field  (dusk_bls12_381::BlsScalar; JubJub's base field)
//   Fr  = JubJub scalar field     (dusk_jubjub::JubJubScalar)
//
// Replaces the arithmetic the reference reaches through `BlsScalar`/`JubJubScalar` operators at
// every call site of /root/reference/src/keys/public.rs:121-130 and
// /root/reference/src/keys/secret.rs:150-168.
//
// The multiplier is an interleaved (CIOS-style) Montgomery product built from carry chains of
// `mad.lo.cc.u32 / madc.hi.cc.u32` pairs, which ptxas fuses into IMAD.WIDE.U32(.X) with the carry
// in a predicate.  The running value lives in two register arrays X (64-bit pairs aligned to even
// limb positions) and Y (pairs aligned to odd positions) so every pair keeps the same two
// registers for the whole product (no MOV traffic); the per-row right shift by one limb swaps the
// roles of X and Y.  q = 1 (mod 2^32) makes the Montgomery factor m = -t0 (no multiply) and
// q[1] = 2^32 - 1 turns two more columns of the reduction into adds: 8 + 7 wide multiplies / row (q[1] is a plain multiply: chains that start with adds do not fuse).
//
// Every chain is one asm block on the device and one emulation routine on the host, so the row
// structure (folds, shifts, carries) is unit-tested on the CPU as well (tests/host_arith_test.cpp);
// the host build is test scaffolding and is never linked into the product library's compute path.
#pragma once
#include <cstdint>

#include "constants_gen.cuh"

#if defined(__CUDACC__)
#define SB_HD __host__ __device__ __forceinline__
#define SB_D __device__ __forceinline__
#else
#define SB_HD inline
#define SB_D inline
#endif

namespace sb200 {

#ifndef SB_Q1_SHORTCUT
#define SB_Q1_SHORTCUT 0  // (measured slower: -7% products but a longer dependent chain per row)  replace the m*q[1] product (q[1] = 2^32-1) of every reduction row by two additions
#endif

struct fq {
  uint32_t v[8];
};

// ------------------------------------------------------------------------------------------
// carry-chain blocks
// ------------------------------------------------------------------------------------------
#if !defined(__CUDA_ARCH__)
namespace emu {
// op counters of the host (test) build: the roofline's "work per tuple" is counted, not estimated
struct counters { unsigned long long wide, fq_mul, fq_sqr, fq_addsub, fr_mul, fq_dot5, dfma, fd_mul, fd_sqr, fd_dot5; };
inline counters& cnt() { static thread_local counters c = {}; return c; }
#define SB_COUNT(field, k) (::sb200::emu::cnt().field += (k))
// acc[0..n) += addend (little-endian limbs) starting at limb `at`; returns carry out of limb n-1
static inline uint32_t add_at(uint32_t* acc, int n, int at, uint64_t val, uint32_t cin) {
  unsigned __int128 carry = cin;
  for (int i = at; i < n; i++) {
    unsigned __int128 t = (unsigned __int128)acc[i] + carry;
    if (i == at) t += (uint32_t)val;
    if (i == at + 1) t += (uint32_t)(val >> 32);
    acc[i] = (uint32_t)t;
    carry = t >> 32;
  }
  return (uint32_t)carry;
}
}  // namespace emu
#else
#define SB_COUNT(field, k) ((void)0)
#endif

// Block A:  x0 += xf + (tprev != 0)   (xf = the limb that fell off the even array at the last shift,
//           tprev = the limb the previous row cancelled: adding m = -tprev to it carries iff tprev != 0);
//           the carry of that addition enters the odd chain:  y[0..7] += a * (b1, b3, b5, b7).
//           No carry out of y[7] (the running value fits 9 limbs).
SB_HD void blk_fold_mac_odd(uint32_t& x0, uint32_t xf, uint32_t tprev, uint32_t* y, uint32_t a, uint32_t b1, uint32_t b3,
                            uint32_t b5, uint32_t b7) {
#if defined(__CUDA_ARCH__)
  asm("{\n\t.reg .u32 t;\n\t"
      "add.cc.u32 t, %10, 0xffffffff;\n\t"
      "addc.cc.u32 %0, %0, %9;\n\t"
      "madc.lo.cc.u32 %1, %11, %12, %1;\n\t"
      "madc.hi.cc.u32 %2, %11, %12, %2;\n\t"
      "madc.lo.cc.u32 %3, %11, %13, %3;\n\t"
      "madc.hi.cc.u32 %4, %11, %13, %4;\n\t"
      "madc.lo.cc.u32 %5, %11, %14, %5;\n\t"
      "madc.hi.cc.u32 %6, %11, %14, %6;\n\t"
      "madc.lo.cc.u32 %7, %11, %15, %7;\n\t"
      "madc.hi.u32 %8, %11, %15, %8;\n\t}"
      : "+r"(x0), "+r"(y[0]), "+r"(y[1]), "+r"(y[2]), "+r"(y[3]), "+r"(y[4]), "+r"(y[5]), "+r"(y[6]), "+r"(y[7])
      : "r"(xf), "r"(tprev), "r"(a), "r"(b1), "r"(b3), "r"(b5), "r"(b7));
#else
  SB_COUNT(wide, 4);
  uint64_t t = (uint64_t)x0 + xf + (tprev != 0 ? 1u : 0u);
  x0 = (uint32_t)t;
  uint32_t c = (uint32_t)(t >> 32);
  c = emu::add_at(y, 8, 0, (uint64_t)a * b1, c);
  c += emu::add_at(y, 8, 2, (uint64_t)a * b3, 0);
  c += emu::add_at(y, 8, 4, (uint64_t)a * b5, 0);
  c += emu::add_at(y, 8, 6, (uint64_t)a * b7, 0);
  (void)c;
#endif
}

// Block B:  x[0..7] += a * (b0, b2, b4, b6); the carry out of x[7] (limb position 8) is added to ytop
//           (= y[7], the odd array's register for position 8).
SB_HD void blk_mac_even(uint32_t* x, uint32_t& ytop, uint32_t a, uint32_t b0, uint32_t b2, uint32_t b4, uint32_t b6) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %9, %10, %0;\n\t"
      "madc.hi.cc.u32 %1, %9, %10, %1;\n\t"
      "madc.lo.cc.u32 %2, %9, %11, %2;\n\t"
      "madc.hi.cc.u32 %3, %9, %11, %3;\n\t"
      "madc.lo.cc.u32 %4, %9, %12, %4;\n\t"
      "madc.hi.cc.u32 %5, %9, %12, %5;\n\t"
      "madc.lo.cc.u32 %6, %9, %13, %6;\n\t"
      "madc.hi.cc.u32 %7, %9, %13, %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(x[0]), "+r"(x[1]), "+r"(x[2]), "+r"(x[3]), "+r"(x[4]), "+r"(x[5]), "+r"(x[6]), "+r"(x[7]), "+r"(ytop)
      : "r"(a), "r"(b0), "r"(b2), "r"(b4), "r"(b6));
#else
  SB_COUNT(wide, 4);
  uint32_t c = emu::add_at(x, 8, 0, (uint64_t)a * b0, 0);
  c += emu::add_at(x, 8, 2, (uint64_t)a * b2, 0);
  c += emu::add_at(x, 8, 4, (uint64_t)a * b4, 0);
  c += emu::add_at(x, 8, 6, (uint64_t)a * b6, 0);
  ytop += c;
#endif
}

// Generic reduction blocks (any odd modulus p with limbs p0..p7): x += m * (p0,p2,p4,p6), y += m * (p1,p3,p5,p7)
SB_HD void blk_mac_odd(uint32_t* y, uint32_t a, uint32_t b1, uint32_t b3, uint32_t b5, uint32_t b7) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %8, %9, %0;\n\t"
      "madc.hi.cc.u32 %1, %8, %9, %1;\n\t"
      "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
      "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
      "madc.lo.cc.u32 %4, %8, %11, %4;\n\t"
      "madc.hi.cc.u32 %5, %8, %11, %5;\n\t"
      "madc.lo.cc.u32 %6, %8, %12, %6;\n\t"
      "madc.hi.u32 %7, %8, %12, %7;"
      : "+r"(y[0]), "+r"(y[1]), "+r"(y[2]), "+r"(y[3]), "+r"(y[4]), "+r"(y[5]), "+r"(y[6]), "+r"(y[7])
      : "r"(a), "r"(b1), "r"(b3), "r"(b5), "r"(b7));
#else
  SB_COUNT(wide, 4);
  uint32_t c = emu::add_at(y, 8, 0, (uint64_t)a * b1, 0);
  c += emu::add_at(y, 8, 2, (uint64_t)a * b3, 0);
  c += emu::add_at(y, 8, 4, (uint64_t)a * b5, 0);
  c += emu::add_at(y, 8, 6, (uint64_t)a * b7, 0);
  (void)c;
#endif
}

// Fq-specific reduction, even half.  q0 = 1 and m = -x0, so x0 + m*q0 = 0 with carry (x0 != 0): that limb
// pair is not touched here at all (the carry is injected by the next row's fold); the chain starts fresh at
// limb 2:  x[2..7] += m * (q2, q4, q6), carry out of x[7] goes to ytop.
SB_HD void blk_red_even_q(uint32_t* x, uint32_t& ytop, uint32_t m, uint32_t q2, uint32_t q4, uint32_t q6) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %7, %8, %0;\n\t"
      "madc.hi.cc.u32 %1, %7, %8, %1;\n\t"
      "madc.lo.cc.u32 %2, %7, %9, %2;\n\t"
      "madc.hi.cc.u32 %3, %7, %9, %3;\n\t"
      "madc.lo.cc.u32 %4, %7, %10, %4;\n\t"
      "madc.hi.cc.u32 %5, %7, %10, %5;\n\t"
      "addc.u32 %6, %6, 0;"
      : "+r"(x[2]), "+r"(x[3]), "+r"(x[4]), "+r"(x[5]), "+r"(x[6]), "+r"(x[7]), "+r"(ytop)
      : "r"(m), "r"(q2), "r"(q4), "r"(q6));
#else
  SB_COUNT(wide, 3);
  uint32_t c = emu::add_at(x, 8, 2, (uint64_t)m * q2, 0);
  c += emu::add_at(x, 8, 4, (uint64_t)m * q4, 0);
  c += emu::add_at(x, 8, 6, (uint64_t)m * q6, 0);
  ytop += c;
#endif
}

// y[0..7] += m * (q1, q3, q5, q7) with q1 = 2^32 - 1:  m*q1 = (m << 32) - m has low word t0 (= -m) and high word
// m - (m != 0), so the first product is two additions; three wide products remain.
SB_HD void blk_red_odd_q(uint32_t* y, uint32_t m, uint32_t t0, uint32_t q3, uint32_t q5, uint32_t q7) {
#if defined(__CUDA_ARCH__)
  asm("{\n\t.reg .u32 h;\n\t"
      "min.u32 h, %8, 1;\n\t"
      "sub.u32 h, %8, h;\n\t"
      "add.cc.u32 %0, %0, %9;\n\t"
      "addc.cc.u32 %1, %1, h;\n\t"
      "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
      "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
      "madc.lo.cc.u32 %4, %8, %11, %4;\n\t"
      "madc.hi.cc.u32 %5, %8, %11, %5;\n\t"
      "madc.lo.cc.u32 %6, %8, %12, %6;\n\t"
      "madc.hi.u32 %7, %8, %12, %7;\n\t}"
      : "+r"(y[0]), "+r"(y[1]), "+r"(y[2]), "+r"(y[3]), "+r"(y[4]), "+r"(y[5]), "+r"(y[6]), "+r"(y[7])
      : "r"(m), "r"(t0), "r"(q3), "r"(q5), "r"(q7));
#else
  SB_COUNT(wide, 3);
  uint32_t hi1 = m - (m != 0 ? 1u : 0u);
  uint32_t c = emu::add_at(y, 8, 0, ((uint64_t)hi1 << 32) | t0, 0);
  c += emu::add_at(y, 8, 2, (uint64_t)m * q3, 0);
  c += emu::add_at(y, 8, 4, (uint64_t)m * q5, 0);
  c += emu::add_at(y, 8, 6, (uint64_t)m * q7, 0);
  (void)c;
#endif
}

// ------------------------------------------------------------------------------------------
// blocks of the dedicated squaring and of the schoolbook products / separated Montgomery reduction
// ------------------------------------------------------------------------------------------
// acc[0..2N) += a * (b0, b1, .. at 64-bit strides), carry out added to `top` (a limb the caller knows cannot overflow)
SB_HD void blk_mac1c(uint32_t* acc, uint32_t& top, uint32_t a, uint32_t b0) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
      "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
      "addc.u32 %2, %2, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(top)
      : "r"(a), "r"(b0));
#else
  SB_COUNT(wide, 1);
  top += emu::add_at(acc, 2, 0, (uint64_t)a * b0, 0);
#endif
}
SB_HD void blk_mac2c(uint32_t* acc, uint32_t& top, uint32_t a, uint32_t b0, uint32_t b1) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %5, %6, %0;\n\t"
      "madc.hi.cc.u32 %1, %5, %6, %1;\n\t"
      "madc.lo.cc.u32 %2, %5, %7, %2;\n\t"
      "madc.hi.cc.u32 %3, %5, %7, %3;\n\t"
      "addc.u32 %4, %4, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(top)
      : "r"(a), "r"(b0), "r"(b1));
#else
  SB_COUNT(wide, 2);
  uint32_t c = emu::add_at(acc, 4, 0, (uint64_t)a * b0, 0);
  c += emu::add_at(acc, 4, 2, (uint64_t)a * b1, 0);
  top += c;
#endif
}
SB_HD void blk_mac3c(uint32_t* acc, uint32_t& top, uint32_t a, uint32_t b0, uint32_t b1, uint32_t b2) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %7, %8, %0;\n\t"
      "madc.hi.cc.u32 %1, %7, %8, %1;\n\t"
      "madc.lo.cc.u32 %2, %7, %9, %2;\n\t"
      "madc.hi.cc.u32 %3, %7, %9, %3;\n\t"
      "madc.lo.cc.u32 %4, %7, %10, %4;\n\t"
      "madc.hi.cc.u32 %5, %7, %10, %5;\n\t"
      "addc.u32 %6, %6, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(top)
      : "r"(a), "r"(b0), "r"(b1), "r"(b2));
#else
  SB_COUNT(wide, 3);
  uint32_t c = emu::add_at(acc, 6, 0, (uint64_t)a * b0, 0);
  c += emu::add_at(acc, 6, 2, (uint64_t)a * b1, 0);
  c += emu::add_at(acc, 6, 4, (uint64_t)a * b2, 0);
  top += c;
#endif
}
SB_HD void blk_mac4c(uint32_t* acc, uint32_t a, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) {  // top = acc[8]
  blk_mac_even(acc, acc[8], a, b0, b1, b2, b3);
}

// acc[0..2N) += a * (b0, b1, .. at 64-bit strides); the caller knows the sum fits (no carry out of acc[2N - 1])
SB_HD void blk_mac1(uint32_t* acc, uint32_t a, uint32_t b0) {
#if defined(__CUDA_ARCH__)
  asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t"
      "madc.hi.u32 %1, %2, %3, %1;"
      : "+r"(acc[0]), "+r"(acc[1])
      : "r"(a), "r"(b0));
#else
  SB_COUNT(wide, 1);
  emu::add_at(acc, 2, 0, (uint64_t)a * b0, 0);
#endif
}

// One Montgomery row of the squaring.  The row adds (m + 1) q with m + 1 = 2^32 - t0 in [1, 2^32] (t0 = the window's limb 0
// after the fold), so limb 0 always carries exactly 1 and no carry is deferred to the next row.  With q0 = 1 and
// q1 = 2^32 - 1:  t0 + (m + 1)(q0 + q1 2^32) = (t0 + 1) 2^32 + m 2^64, and m = ~t0 fits 32 bits.  The part of (m + 1) q that
// does not depend on t0, 2^32 + (q >> 64) 2^64, is left out of every row (fq_sqr_inl feeds the sum over its rows into the
// window instead); what remains is t0 at limb 1 and m (q2 + 1, q3, .., q7) from limb 2:
//   x0 += xf;  t0 = x0;  m = ~t0;  x1 += t0 + (carry of the fold);  x[2..7] += m (q2 + 1, q4, q6), carry out into y[7];
//   y[2..7] += m (q3, q5, q7)  (the window fits 9 limbs: no carry out).
// Six wide products and four other instructions; m is formed as t0 ^ q1 with q1 in a register (see fq_mul_inl).
SB_HD void blk_sqr_red_row(uint32_t* x, uint32_t* y, uint32_t xf, uint32_t q1, uint32_t q2p, uint32_t q3, uint32_t q4,
                           uint32_t q5, uint32_t q6, uint32_t q7) {
#if defined(__CUDA_ARCH__)
  asm("{\n\t.reg .u32 m;\n\t"
      "add.cc.u32 %0, %0, %14;\n\t"
      "xor.b32 m, %0, %15;\n\t"
      "addc.cc.u32 %1, %1, %0;\n\t"
      "madc.lo.cc.u32 %2, m, %16, %2;\n\t"
      "madc.hi.cc.u32 %3, m, %16, %3;\n\t"
      "madc.lo.cc.u32 %4, m, %18, %4;\n\t"
      "madc.hi.cc.u32 %5, m, %18, %5;\n\t"
      "madc.lo.cc.u32 %6, m, %20, %6;\n\t"
      "madc.hi.cc.u32 %7, m, %20, %7;\n\t"
      "addc.u32 %13, %13, 0;\n\t"
      "mad.lo.cc.u32 %8, m, %17, %8;\n\t"
      "madc.hi.cc.u32 %9, m, %17, %9;\n\t"
      "madc.lo.cc.u32 %10, m, %19, %10;\n\t"
      "madc.hi.cc.u32 %11, m, %19, %11;\n\t"
      "madc.lo.cc.u32 %12, m, %21, %12;\n\t"
      "madc.hi.u32 %13, m, %21, %13;\n\t}"
      : "+r"(x[0]), "+r"(x[1]), "+r"(x[2]), "+r"(x[3]), "+r"(x[4]), "+r"(x[5]), "+r"(x[6]), "+r"(x[7]), "+r"(y[2]),
        "+r"(y[3]), "+r"(y[4]), "+r"(y[5]), "+r"(y[6]), "+r"(y[7])
      : "r"(xf), "r"(q1), "r"(q2p), "r"(q3), "r"(q4), "r"(q5), "r"(q6), "r"(q7));
#else
  SB_COUNT(wide, 6);
  uint64_t t = (uint64_t)x[0] + xf;
  x[0] = (uint32_t)t;
  const uint32_t m = x[0] ^ q1;
  uint32_t c = emu::add_at(x, 8, 1, x[0], (uint32_t)(t >> 32));
  c += emu::add_at(x, 8, 2, (uint64_t)m * q2p, 0);
  c += emu::add_at(x, 8, 4, (uint64_t)m * q4, 0);
  c += emu::add_at(x, 8, 6, (uint64_t)m * q6, 0);
  y[7] += c;
  emu::add_at(y, 8, 2, (uint64_t)m * q3, 0);
  emu::add_at(y, 8, 4, (uint64_t)m * q5, 0);
  emu::add_at(y, 8, 6, (uint64_t)m * q7, 0);
#endif
}

// r[0..15] = e[0..15] + (o[0..14] << 32)   (o[k] sits at limb position k + 1); the sum fits 16 limbs
SB_HD void merge_eo16(uint32_t* r, const uint32_t* e, const uint32_t* o) {
#if defined(__CUDA_ARCH__)
  r[0] = e[0];
  asm("add.cc.u32 %0, %15, %30;\n\t"
      "addc.cc.u32 %1, %16, %31;\n\t"
      "addc.cc.u32 %2, %17, %32;\n\t"
      "addc.cc.u32 %3, %18, %33;\n\t"
      "addc.cc.u32 %4, %19, %34;\n\t"
      "addc.cc.u32 %5, %20, %35;\n\t"
      "addc.cc.u32 %6, %21, %36;\n\t"
      "addc.cc.u32 %7, %22, %37;\n\t"
      "addc.cc.u32 %8, %23, %38;\n\t"
      "addc.cc.u32 %9, %24, %39;\n\t"
      "addc.cc.u32 %10, %25, %40;\n\t"
      "addc.cc.u32 %11, %26, %41;\n\t"
      "addc.cc.u32 %12, %27, %42;\n\t"
      "addc.cc.u32 %13, %28, %43;\n\t"
      "addc.u32 %14, %29, %44;"
      : "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]), "r"(e[8]), "r"(e[9]), "r"(e[10]),
        "r"(e[11]), "r"(e[12]), "r"(e[13]), "r"(e[14]), "r"(e[15]), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]),
        "r"(o[5]), "r"(o[6]), "r"(o[7]), "r"(o[8]), "r"(o[9]), "r"(o[10]), "r"(o[11]), "r"(o[12]), "r"(o[13]), "r"(o[14]));
#else
  r[0] = e[0];
  uint64_t c = 0;
  for (int i = 1; i < 16; i++) {
    c += (uint64_t)e[i] + o[i - 1];
    r[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
}

// One row of the separated Montgomery reduction, odd half, fused with the fold:
//   x0 += xf + (tprev != 0);  m = -x0;  y[0..7] += m * (q1, q3, q5, q7) + carry of the fold
//   (m * q1 by the two-addition shortcut of blk_red_odd_q).
SB_HD uint32_t blk_fold_red_odd(uint32_t& x0, uint32_t xf, uint32_t tprev, uint32_t* y, uint32_t q1, uint32_t q3,
                                uint32_t q5, uint32_t q7) {
  uint32_t m;
#if defined(__CUDA_ARCH__)
  asm("{\n\t.reg .u32 t, h;\n\t"
      "add.cc.u32 t, %11, 0xffffffff;\n\t"
      "addc.cc.u32 %0, %0, %10;\n\t"
      "xor.b32 %9, %0, %12;\n\t"
      "add.u32 %9, %9, 1;\n\t"
      "min.u32 h, %9, 1;\n\t"
      "sub.u32 h, %9, h;\n\t"
      "addc.cc.u32 %1, %1, %0;\n\t"
      "addc.cc.u32 %2, %2, h;\n\t"
      "madc.lo.cc.u32 %3, %9, %13, %3;\n\t"
      "madc.hi.cc.u32 %4, %9, %13, %4;\n\t"
      "madc.lo.cc.u32 %5, %9, %14, %5;\n\t"
      "madc.hi.cc.u32 %6, %9, %14, %6;\n\t"
      "madc.lo.cc.u32 %7, %9, %15, %7;\n\t"
      "madc.hi.u32 %8, %9, %15, %8;\n\t}"
      : "+r"(x0), "+r"(y[0]), "+r"(y[1]), "+r"(y[2]), "+r"(y[3]), "+r"(y[4]), "+r"(y[5]), "+r"(y[6]), "+r"(y[7]), "=&r"(m)
      : "r"(xf), "r"(tprev), "r"(q1), "r"(q3), "r"(q5), "r"(q7));
#else
  SB_COUNT(wide, 4);
  uint64_t t = (uint64_t)x0 + xf + (tprev != 0 ? 1u : 0u);
  x0 = (uint32_t)t;
  uint32_t c = (uint32_t)(t >> 32);
  m = 0u - x0;
  SB_COUNT(wide, -1);
  (void)q1;
  c = emu::add_at(y, 8, 0, ((uint64_t)(m - (m != 0 ? 1u : 0u)) << 32) | x0, c);
  c += emu::add_at(y, 8, 2, (uint64_t)m * q3, 0);
  c += emu::add_at(y, 8, 4, (uint64_t)m * q5, 0);
  c += emu::add_at(y, 8, 6, (uint64_t)m * q7, 0);
  (void)c;
#endif
  return m;
}

// r = a + b (8 limbs), returns carry
SB_HD uint32_t add8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t c;
#if defined(__CUDA_ARCH__)
  asm("add.cc.u32 %0, %9, %17;\n\t"
      "addc.cc.u32 %1, %10, %18;\n\t"
      "addc.cc.u32 %2, %11, %19;\n\t"
      "addc.cc.u32 %3, %12, %20;\n\t"
      "addc.cc.u32 %4, %13, %21;\n\t"
      "addc.cc.u32 %5, %14, %22;\n\t"
      "addc.cc.u32 %6, %15, %23;\n\t"
      "addc.cc.u32 %7, %16, %24;\n\t"
      "addc.u32 %8, 0, 0;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(c)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]),
        "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
#else
  uint64_t t = 0;
  for (int i = 0; i < 8; i++) {
    t += (uint64_t)a[i] + b[i];
    r[i] = (uint32_t)t;
    t >>= 32;
  }
  c = (uint32_t)t;
#endif
  return c;
}

// r = a + b + (t != 0) (8 limbs); the sum is known to fit
SB_HD void add8c(uint32_t* r, const uint32_t* a, const uint32_t* b, uint32_t t) {
#if defined(__CUDA_ARCH__)
  asm("{\n\t.reg .u32 t;\n\t"
      "add.cc.u32 t, %24, 0xffffffff;\n\t"
      "addc.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;\n\t}"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]),
        "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(t));
#else
  uint64_t c = t != 0 ? 1 : 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a[i] + b[i];
    r[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
}

// r = a - b (8 limbs), returns borrow mask (0 or 0xffffffff)
SB_HD uint32_t sub8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t c;
#if defined(__CUDA_ARCH__)
  asm("sub.cc.u32 %0, %9, %17;\n\t"
      "subc.cc.u32 %1, %10, %18;\n\t"
      "subc.cc.u32 %2, %11, %19;\n\t"
      "subc.cc.u32 %3, %12, %20;\n\t"
      "subc.cc.u32 %4, %13, %21;\n\t"
      "subc.cc.u32 %5, %14, %22;\n\t"
      "subc.cc.u32 %6, %15, %23;\n\t"
      "subc.cc.u32 %7, %16, %24;\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(c)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]),
        "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
#else
  int64_t t = 0;
  for (int i = 0; i < 8; i++) {
    t += (int64_t)a[i] - (int64_t)b[i];
    r[i] = (uint32_t)t;
    t >>= 32;  // arithmetic shift keeps the borrow as -1
  }
  c = (uint32_t)t;
#endif
  return c;
}

// ------------------------------------------------------------------------------------------
// moduli
// ------------------------------------------------------------------------------------------
struct FqP {
  static SB_HD constexpr uint32_t p(int i) {
    constexpr uint32_t t[8] = SB200_FQ_MOD_INIT;
    return t[i];
  }
};
struct FrP {
  static SB_HD constexpr uint32_t p(int i) {
    constexpr uint32_t t[8] = SB200_FR_MOD_INIT;
    return t[i];
  }
  static constexpr uint32_t ninv = SB200_FR_NINV;
};

// q's limbs for the multiplier must sit in ordinary registers: with immediate or uniform-register
// multiplicands ptxas emits IMAD + IMAD.HI pairs instead of one IMAD.WIDE.U32.X per product.
#if defined(__CUDACC__)
// One copy of the modulus per lane: the lane-dependent address makes the loaded limbs "divergent" for
// ptxas' uniformity analysis, so they stay in ordinary registers.  (With immediate, constant-bank or
// uniform-register multiplicands ptxas emits IMAD + IMAD.HI.U32.X instead of one IMAD.WIDE.U32.X.)
#define SB_X32(v) v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v, v
__device__ uint32_t d_fq_mod_lane[8 * 32] = {SB_X32(0x00000001u), SB_X32(0xffffffffu), SB_X32(0xfffe5bfeu), SB_X32(0x53bda402u),
                                            SB_X32(0x09a1d805u), SB_X32(0x3339d808u), SB_X32(0x299d7d48u), SB_X32(0x73eda753u)};
__device__ uint32_t d_fr_mod_lane[8 * 32] = {SB_X32(0xd6f72cb7u), SB_X32(0xd0970e5eu), SB_X32(0xccc81082u), SB_X32(0xa6682093u),
                                            SB_X32(0x01343b00u), SB_X32(0x06673b01u), SB_X32(0x6533afa9u), SB_X32(0x0e7db4eau)};
#endif
#ifndef SB_FQ_MOD_IMM
#define SB_FQ_MOD_IMM 1  // modulus limbs as immediates (q1 through c_fq_q1); 0 = the per-lane copy in global memory (round 1)
#endif
#if defined(__CUDACC__)
// q1 = 2^32 - 1 must stay a value ptxas does not know: as a literal, every product with it is strength-reduced to
// IMAD.HI + IMAD.IADD (5 issue cycles instead of 4).  A __constant__ word is opaque (the host could change it) and costs one
// uniform load per multiplier body.
__constant__ uint32_t c_fq_q1 = 0xffffffffu;
#endif
#if defined(__CUDA_ARCH__) && SB_FQ_MOD_IMM
#define SB_FQ_MOD(i) ((i) == 1 ? c_fq_q1 : FqP::p(i))
#define SB_FR_MOD(i) __ldg(&d_fr_mod_lane[(i) * 32 + (threadIdx.x & 31)])
#elif defined(__CUDA_ARCH__)
#define SB_FQ_MOD(i) __ldg(&d_fq_mod_lane[(i) * 32 + (threadIdx.x & 31)])
#define SB_FR_MOD(i) __ldg(&d_fr_mod_lane[(i) * 32 + (threadIdx.x & 31)])
#else
#define SB_FQ_MOD(i) FqP::p(i)
#define SB_FR_MOD(i) FrP::p(i)
#endif

template <class P>
SB_HD void cond_sub_p(uint32_t* r) {  // r in [0, 2p) -> [0, p)
  uint32_t t[8];
  const uint32_t pp[8] = {P::p(0), P::p(1), P::p(2), P::p(3), P::p(4), P::p(5), P::p(6), P::p(7)};
  uint32_t borrow = sub8(t, r, pp);
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = borrow ? r[i] : t[i];
}

// ------------------------------------------------------------------------------------------
// Fq
// ------------------------------------------------------------------------------------------
SB_HD fq fq_zero() {
  fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = 0;
  return r;
}
SB_HD fq fq_one() {  // Montgomery 1
  const uint32_t c[8] = SB200_FQ_ONE_INIT;
  fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = c[i];
  return r;
}

SB_HD fq fq_add(const fq& a, const fq& b) {
  SB_COUNT(fq_addsub, 1);
  fq r;
  add8(r.v, a.v, b.v);  // a + b < 2q < 2^256: no carry
  cond_sub_p<FqP>(r.v);
  return r;
}

#ifndef SB_SUB_PREDICATED
#define SB_SUB_PREDICATED 1
#endif
SB_HD fq fq_sub(const fq& a, const fq& b) {
  SB_COUNT(fq_addsub, 1);
  fq r;
  uint32_t borrow = sub8(r.v, a.v, b.v);
#if defined(__CUDA_ARCH__) && SB_SUB_PREDICATED
  // add q back under a predicate (8 predicated additions with immediate limbs) instead of masking q first (8 AND + 8 additions)
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ne.u32 p, %8, 0;\n\t"
      "@p add.cc.u32 %0, %0, %9;\n\t"
      "@p addc.cc.u32 %1, %1, %10;\n\t"
      "@p addc.cc.u32 %2, %2, %11;\n\t"
      "@p addc.cc.u32 %3, %3, %12;\n\t"
      "@p addc.cc.u32 %4, %4, %13;\n\t"
      "@p addc.cc.u32 %5, %5, %14;\n\t"
      "@p addc.cc.u32 %6, %6, %15;\n\t"
      "@p addc.u32 %7, %7, %16;\n\t}"
      : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]), "+r"(r.v[3]), "+r"(r.v[4]), "+r"(r.v[5]), "+r"(r.v[6]), "+r"(r.v[7])
      : "r"(borrow), "n"(FqP::p(0)), "n"(FqP::p(1)), "n"(FqP::p(2)), "n"(FqP::p(3)), "n"(FqP::p(4)), "n"(FqP::p(5)), "n"(FqP::p(6)),
        "n"(FqP::p(7)));
  return r;
#endif
  uint32_t t[8];
#pragma unroll
  for (int i = 0; i < 8; i++) t[i] = FqP::p(i) & borrow;
  add8(r.v, r.v, t);
  return r;
}

SB_HD fq fq_neg(const fq& a) { return fq_sub(fq_zero(), a); }

SB_HD fq fq_dbl(const fq& a) { return fq_add(a, a); }

SB_HD bool fq_is_zero(const fq& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i];
  return o == 0;
}

SB_HD bool fq_eq(const fq& a, const fq& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i] ^ b.v[i];
  return o == 0;
}

SB_HD fq fq_select(const fq& a, const fq& b, bool take_b) {
  fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = take_b ? b.v[i] : a.v[i];
  return r;
}

// Montgomery product a * b * 2^-256 mod q, inputs and output canonical (< q).
// 8 rows x (8 + 6) wide products.
SB_HD void mul_wide16(uint32_t* T, const uint32_t* a, const uint32_t* b);
SB_HD fq mont_reduce16(const uint32_t* t);
#ifndef SB_MUL_SEPARATED
#define SB_MUL_SEPARATED 0  // experiment: schoolbook product (64) + separated reduction (48) instead of the interleaved 120
#endif
SB_HD fq fq_mul_inl(const fq& a, const fq& b) {
  SB_COUNT(fq_mul, 1);
#if SB_MUL_SEPARATED
  uint32_t T[16];
  mul_wide16(T, a.v, b.v);
  return mont_reduce16(T);
#endif
  uint32_t X[8], Y[8], xf = 0, tprev = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) X[i] = Y[i] = 0;
  const uint32_t q1 = SB_FQ_MOD(1), q2 = SB_FQ_MOD(2), q3 = SB_FQ_MOD(3), q4 = SB_FQ_MOD(4), q5 = SB_FQ_MOD(5),
                 q6 = SB_FQ_MOD(6), q7 = SB_FQ_MOD(7);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t ai = a.v[i];
    blk_fold_mac_odd(X[0], xf, tprev, Y, ai, b.v[1], b.v[3], b.v[5], b.v[7]);
    blk_mac_even(X, Y[7], ai, b.v[0], b.v[2], b.v[4], b.v[6]);
    tprev = X[0];
    // m = -tprev (-q^-1 = 2^32 - 1).  Written as (tprev ^ q1) + 1 with the register copy of q1 = 2^32 - 1,
    // which ptxas cannot recognise as a negation: when it does, it folds the negation into the multiplies
    // below and emits IMAD + IMAD.HI.U32 pairs for every product with m instead of IMAD.WIDE.U32.X.
    // (Two ALU-pipe instructions; a multiply by q1 would cost the saturated FMA-heavy pipe instead.)
#if defined(__CUDA_ARCH__) && SB_FQ_MOD_IMM
    uint32_t m;
    asm("xor.b32 %0, %1, %2;\n\tadd.u32 %0, %0, 1;" : "=r"(m) : "r"(tprev), "r"(q1));
#else
    uint32_t m = (tprev ^ q1) + 1u;
#endif
    blk_red_even_q(X, Y[7], m, q2, q4, q6);
#if SB_Q1_SHORTCUT
    blk_red_odd_q(Y, m, tprev, q3, q5, q7);
#else
    blk_mac_odd(Y, m, q1, q3, q5, q7);
#endif
    // divide by 2^32: the odd array becomes the even one; X[1] (+ the carry of the cancelled limb) is
    // folded in by the next row
    xf = X[1];
    uint32_t nx[8], ny[8];
#pragma unroll
    for (int k = 0; k < 8; k++) nx[k] = Y[k];
#pragma unroll
    for (int k = 0; k < 6; k++) ny[k] = X[k + 2];
    ny[6] = 0;
    ny[7] = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      X[k] = nx[k];
      Y[k] = ny[k];
    }
  }
  // value = X + xf + (tprev != 0) + (Y << 32)  (< 2q)
  fq r;
  uint32_t s[8] = {xf, Y[0], Y[1], Y[2], Y[3], Y[4], Y[5], Y[6]};
  add8c(r.v, X, s, tprev);
  cond_sub_p<FqP>(r.v);
  return r;
}

// Montgomery reduction of a 16-limb T < q * 2^256:  (T_lo + M q) / 2^256 + T_hi, conditional subtraction.
// M depends on T_lo only, so the 8 rows run on a 9-limb window seeded with T_lo (7 wide products each) and
// T_hi is added once at the end.
SB_HD fq mont_reduce16(const uint32_t* t) {
  uint32_t X[8], Y[8], xf = 0, tprev = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    X[i] = t[i];
    Y[i] = 0;
  }
  const uint32_t q1 = SB_FQ_MOD(1), q2 = SB_FQ_MOD(2), q3 = SB_FQ_MOD(3), q4 = SB_FQ_MOD(4), q5 = SB_FQ_MOD(5),
                 q6 = SB_FQ_MOD(6), q7 = SB_FQ_MOD(7);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t m = blk_fold_red_odd(X[0], xf, tprev, Y, q1, q3, q5, q7);
    tprev = X[0];
    blk_red_even_q(X, Y[7], m, q2, q4, q6);
    xf = X[1];
    uint32_t nx[8], ny[8];
#pragma unroll
    for (int k = 0; k < 8; k++) nx[k] = Y[k];
#pragma unroll
    for (int k = 0; k < 6; k++) ny[k] = X[k + 2];
    ny[6] = 0;
    ny[7] = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      X[k] = nx[k];
      Y[k] = ny[k];
    }
  }
  // V = X + xf + (tprev != 0) + (Y << 32) <= q;  result = V + T_hi < 2q
  fq v, r;
  uint32_t s[8] = {xf, Y[0], Y[1], Y[2], Y[3], Y[4], Y[5], Y[6]};
  add8c(v.v, X, s, tprev);
  add8(r.v, v.v, t + 8);
  cond_sub_p<FqP>(r.v);
  return r;
}

// Row r < 7 of the square, one limb later than its place (see fq_sqr_inl): a_r times b = (a_r, 2 a_{r+1} mod 2^32,
// d_{r+2}, .., d_7) with the limbs d_j of 2a (d_{r+1} also holds a_r's top bit, which belongs to a_r * a_r);
// sum_r a_r b 2^(64 r) = a^2.  Limb j of b lands on window limb j - 1: odd j on X (carry out into Y[7]), even j on Y
// (carry out into Y[6]; both are limbs the previous shift left holding only a constant).  Row 0 leaves out a_0 * a_0.
SB_HD void sqr_row(uint32_t* X, uint32_t* Y, const uint32_t* a, const uint32_t* d, int r) {
  uint32_t b[8];
#pragma unroll
  for (int j = 0; j < 8; j++) b[j] = j == r ? a[r] : j == r + 1 ? a[j] << 1 : d[j];
  const uint32_t ar = a[r];
  switch ((r | 1) / 2) {  // first odd limb: (r | 1), X pair (r | 1) / 2 .. 3
    case 0: blk_mac_even(X, Y[7], ar, b[1], b[3], b[5], b[7]); break;
    case 1: blk_mac3c(X + 2, Y[7], ar, b[3], b[5], b[7]); break;
    case 2: blk_mac2c(X + 4, Y[7], ar, b[5], b[7]); break;
    default: blk_mac1c(X + 6, Y[7], ar, b[7]); break;
  }
  switch ((r + 1) / 2) {  // first even limb: 2 (r + 1) / 2, 2 at least; Y pair (r + 1) / 2 - 1 .. 2
    case 0:
    case 1: blk_mac3c(Y, Y[6], ar, b[2], b[4], b[6]); break;
    case 2: blk_mac2c(Y + 2, Y[6], ar, b[4], b[6]); break;
    default: blk_mac1c(Y + 4, Y[6], ar, b[6]); break;
  }
}

// Dedicated squaring, a < q: the rows of the square interleaved with Montgomery rows on the 9-limb window of fq_mul_inl
// (X = even-aligned limb pairs, Y = odd-aligned).  36 + 8 x 6 = 84 wide products; besides them, four instructions per
// Montgomery row, two carries per row of the square, the limbs of 2a, the final merge and subtraction.
//  * Row r of the square is added after Montgomery row r, one limb right of its schoolbook place.  Before the shift of
//    row i >= 1 the window then holds (A (2a - A) + M q) / 2^(32 i) + (part of K, below), with A = a mod 2^(32 i) (rows
//    0..i-1 of the square) and M = sum_{j <= i} (m_j + 1) 2^(32 j) < 2^(32 (i+1)) (1 + 2^-31): below 2a + 2^32 q (1 + 2^-31)
//    + 2^257 < 2^288.  At its place, row i (a_i times about 2a) would bring it to 2^32 (2a + q), which does not fit 9 limbs.
//    Only a_0 * a_0 goes in first: limb 0 sets the first m.
//  * blk_sqr_red_row leaves the t0-independent part of every row's (m + 1) q out.  Their sum over the 8 rows plus l q
//    (l < 2^224, which only adds to M), K = SB200_FQ_SQR_K_INIT, has limbs 0..6 zero; it enters the window limb by limb,
//    limb i + 7 as the constant on the limb that the shift before row i frees (Y[6]).  It adds < 2^257 to the window.
//  * Result (a^2 + M q) / 2^256 < q^2 / 2^256 + q (1 + 2^-31) < 1.46 q: one conditional subtraction.
SB_HD fq fq_sqr_inl(const fq& x) {
  SB_COUNT(fq_sqr, 1);
  const uint32_t* a = x.v;
  const uint32_t k[16] = SB200_FQ_SQR_K_INIT;
  uint32_t d[8], X[8], Y[8], xf = 0;
  d[0] = 0;
#pragma unroll
  for (int j = 1; j < 8; j++) {
#if defined(__CUDA_ARCH__)
    d[j] = __funnelshift_l(a[j - 1], a[j], 1);
#else
    d[j] = (a[j] << 1) | (a[j - 1] >> 31);
#endif
  }
#pragma unroll
  for (int i = 0; i < 8; i++) X[i] = Y[i] = 0;
  Y[6] = k[7];
  const uint32_t q1 = SB_FQ_MOD(1), q2p = FqP::p(2) + 1u, q3 = SB_FQ_MOD(3), q4 = SB_FQ_MOD(4), q5 = SB_FQ_MOD(5),
                 q6 = SB_FQ_MOD(6), q7 = SB_FQ_MOD(7);
  blk_mac1(X, a[0], a[0]);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    if (i > 0) sqr_row(X, Y, a, d, i - 1);
    blk_sqr_red_row(X, Y, xf, q1, q2p, q3, q4, q5, q6, q7);
    // divide by 2^32 (limb 0 is t0 + m + 1 = 2^32: its carry is in X[1] already); X[1] is folded in by the next row
    xf = X[1];
    uint32_t nx[8], ny[8];
#pragma unroll
    for (int j = 0; j < 8; j++) nx[j] = Y[j];
#pragma unroll
    for (int j = 0; j < 6; j++) ny[j] = X[j + 2];
    ny[6] = k[i + 8];
    ny[7] = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      X[j] = nx[j];
      Y[j] = ny[j];
    }
  }
  blk_mac1(X + 6, a[7], a[7]);  // row 7, a_7 * a_7 (limb 14 = limb 6 of the result)
  fq r;
  const uint32_t s[8] = {xf, Y[0], Y[1], Y[2], Y[3], Y[4], Y[5], Y[6]};
  add8(r.v, X, s);
  cond_sub_p<FqP>(r.v);
  return r;
}

// ------------------------------------------------------------------------------------------
// Lazy-reduced dot product  sum_j c_j * s_j  (n <= 5 terms): n full products (64 wide each) accumulated as
// one 17-limb integer and ONE Montgomery reduction (56 wide), instead of n * 120.  Used by the Hades MDS
// layers.  5 q^2 < 2^513, result before the final subtractions < q + 5 q^2 / 2^256 < 3.27 q.
// ------------------------------------------------------------------------------------------
// T[0..15] = a * b : schoolbook product in an even- and an odd-aligned array (all chains fuse; every carry
// lands on a limb that holds at most earlier carries), merged once.
SB_HD void mul_wide16(uint32_t* T, const uint32_t* a, const uint32_t* b) {
  uint32_t E[18], O[18];
#pragma unroll
  for (int i = 0; i < 18; i++) E[i] = O[i] = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    if ((i & 1) == 0) {
      blk_mac4c(E + i, a[i], b[0], b[2], b[4], b[6]);
      blk_mac4c(O + i, a[i], b[1], b[3], b[5], b[7]);
    } else {
      blk_mac4c(O + i - 1, a[i], b[0], b[2], b[4], b[6]);
      blk_mac4c(E + i + 1, a[i], b[1], b[3], b[5], b[7]);
    }
  }
  merge_eo16(T, E, O);
}

// S[0..16] += T[0..15]
SB_HD void acc17(uint32_t* S, const uint32_t* T) {
#if defined(__CUDA_ARCH__)
  asm("add.cc.u32 %0, %0, %17;\n\t"
      "addc.cc.u32 %1, %1, %18;\n\t"
      "addc.cc.u32 %2, %2, %19;\n\t"
      "addc.cc.u32 %3, %3, %20;\n\t"
      "addc.cc.u32 %4, %4, %21;\n\t"
      "addc.cc.u32 %5, %5, %22;\n\t"
      "addc.cc.u32 %6, %6, %23;\n\t"
      "addc.cc.u32 %7, %7, %24;\n\t"
      "addc.cc.u32 %8, %8, %25;\n\t"
      "addc.cc.u32 %9, %9, %26;\n\t"
      "addc.cc.u32 %10, %10, %27;\n\t"
      "addc.cc.u32 %11, %11, %28;\n\t"
      "addc.cc.u32 %12, %12, %29;\n\t"
      "addc.cc.u32 %13, %13, %30;\n\t"
      "addc.cc.u32 %14, %14, %31;\n\t"
      "addc.cc.u32 %15, %15, %32;\n\t"
      "addc.u32 %16, %16, 0;"
      : "+r"(S[0]), "+r"(S[1]), "+r"(S[2]), "+r"(S[3]), "+r"(S[4]), "+r"(S[5]), "+r"(S[6]), "+r"(S[7]), "+r"(S[8]),
        "+r"(S[9]), "+r"(S[10]), "+r"(S[11]), "+r"(S[12]), "+r"(S[13]), "+r"(S[14]), "+r"(S[15]), "+r"(S[16])
      : "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]),
        "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
#else
  uint64_t c = 0;
  for (int i = 0; i < 16; i++) {
    c += (uint64_t)S[i] + T[i];
    S[i] = (uint32_t)c;
    c >>= 32;
  }
  S[16] += (uint32_t)c;
#endif
}

// Montgomery reduction of a 17-limb S < 5 q^2 to the canonical representative.
SB_HD fq mont_reduce17(const uint32_t* S) {
  uint32_t X[8], Y[8], xf = 0, tprev = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    X[i] = S[i];
    Y[i] = 0;
  }
  const uint32_t q1 = SB_FQ_MOD(1), q2 = SB_FQ_MOD(2), q3 = SB_FQ_MOD(3), q4 = SB_FQ_MOD(4), q5 = SB_FQ_MOD(5),
                 q6 = SB_FQ_MOD(6), q7 = SB_FQ_MOD(7);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t m = blk_fold_red_odd(X[0], xf, tprev, Y, q1, q3, q5, q7);
    tprev = X[0];
    blk_red_even_q(X, Y[7], m, q2, q4, q6);
    xf = X[1];
    uint32_t nx[8], ny[8];
#pragma unroll
    for (int k = 0; k < 8; k++) nx[k] = Y[k];
#pragma unroll
    for (int k = 0; k < 6; k++) ny[k] = X[k + 2];
    ny[6] = 0;
    ny[7] = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      X[k] = nx[k];
      Y[k] = ny[k];
    }
  }
  fq v, r;
  uint32_t s[8] = {xf, Y[0], Y[1], Y[2], Y[3], Y[4], Y[5], Y[6]};
  add8c(v.v, X, s, tprev);                   // V0 <= q
  uint32_t top = S[16] + add8(r.v, v.v, S + 8);  // 9-limb value r + top * 2^256 < 3.27 q
  // >= 2q ?  (2q < 2^256)
  uint32_t t[8], q2x[8];
#pragma unroll
  for (int i = 0; i < 8; i++) q2x[i] = (FqP::p(i) << 1) | (i ? FqP::p(i - 1) >> 31 : 0u);
  uint32_t borrow = sub8(t, r.v, q2x);
  bool ge = (top != 0) | (borrow == 0);
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = ge ? t[i] : r.v[i];
  cond_sub_p<FqP>(r.v);
  return r;
}

// S[0..16] = E[0..16] + (O[0..15] << 32)   (O[k] sits at limb position k + 1); the sum fits 17 limbs
SB_HD void merge_eo17(uint32_t* S, const uint32_t* E, const uint32_t* O) {
  S[0] = E[0];
#if defined(__CUDA_ARCH__)
  asm("add.cc.u32 %0, %16, %32;\n\t"
      "addc.cc.u32 %1, %17, %33;\n\t"
      "addc.cc.u32 %2, %18, %34;\n\t"
      "addc.cc.u32 %3, %19, %35;\n\t"
      "addc.cc.u32 %4, %20, %36;\n\t"
      "addc.cc.u32 %5, %21, %37;\n\t"
      "addc.cc.u32 %6, %22, %38;\n\t"
      "addc.cc.u32 %7, %23, %39;\n\t"
      "addc.cc.u32 %8, %24, %40;\n\t"
      "addc.cc.u32 %9, %25, %41;\n\t"
      "addc.cc.u32 %10, %26, %42;\n\t"
      "addc.cc.u32 %11, %27, %43;\n\t"
      "addc.cc.u32 %12, %28, %44;\n\t"
      "addc.cc.u32 %13, %29, %45;\n\t"
      "addc.cc.u32 %14, %30, %46;\n\t"
      "addc.u32 %15, %31, %47;"
      : "=r"(S[1]), "=r"(S[2]), "=r"(S[3]), "=r"(S[4]), "=r"(S[5]), "=r"(S[6]), "=r"(S[7]), "=r"(S[8]), "=r"(S[9]), "=r"(S[10]),
        "=r"(S[11]), "=r"(S[12]), "=r"(S[13]), "=r"(S[14]), "=r"(S[15]), "=r"(S[16])
      : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]), "r"(E[10]), "r"(E[11]),
        "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]), "r"(E[16]), "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]),
        "r"(O[6]), "r"(O[7]), "r"(O[8]), "r"(O[9]), "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]), "r"(O[15]));
#else
  uint64_t c = 0;
  for (int i = 1; i < 17; i++) {
    c += (uint64_t)E[i] + O[i - 1];
    S[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
}

#ifndef SB_DOT5_ROWMAJOR
#define SB_DOT5_ROWMAJOR 1
#endif
// sum_{j<5} c_j * s_j with the constants c_j read through `cst` (5 consecutive field elements)
SB_HD fq fq_dot5_inl(const uint32_t (*cst)[8], const fq& s0, const fq& s1, const fq& s2, const fq& s3, const fq& s4) {
  SB_COUNT(fq_dot5, 1);
#if SB_DOT5_ROWMAJOR
  // All five products accumulate into ONE pair of even- / odd-aligned arrays, limb row by limb row (row i of every product
  // before row i + 1 of any): the limb that takes a block's carry-out (position i + 8 or i + 9) has then only ever received
  // carry-outs (at most ten of them), so the plain `addc` at the end of a block cannot overflow -- and the per-product
  // merge (15 additions) and accumulation (17) of the product-by-product form disappear: 143 instructions less per call.
  {
    uint32_t E[18], O[18], S[17];
#pragma unroll
    for (int i = 0; i < 18; i++) E[i] = O[i] = 0;
    const fq* sv[5] = {&s0, &s1, &s2, &s3, &s4};
#pragma unroll
    for (int i = 0; i < 8; i++) {
#pragma unroll
      for (int j = 0; j < 5; j++) {
        const uint32_t a = sv[j]->v[i];
        if ((i & 1) == 0) {
          blk_mac4c(E + i, a, cst[j][0], cst[j][2], cst[j][4], cst[j][6]);
          blk_mac4c(O + i, a, cst[j][1], cst[j][3], cst[j][5], cst[j][7]);
        } else {
          blk_mac4c(O + i - 1, a, cst[j][0], cst[j][2], cst[j][4], cst[j][6]);
          blk_mac4c(E + i + 1, a, cst[j][1], cst[j][3], cst[j][5], cst[j][7]);
        }
      }
    }
    merge_eo17(S, E, O);
    return mont_reduce17(S);
  }
#endif
  uint32_t S[17], T[16], c[8];
#pragma unroll
  for (int i = 0; i < 17; i++) S[i] = 0;
  const fq* sv[5] = {&s0, &s1, &s2, &s3, &s4};
#pragma unroll
  for (int j = 0; j < 5; j++) {
#pragma unroll
    for (int i = 0; i < 8; i++) c[i] = cst[j][i];
    mul_wide16(T, sv[j]->v, c);
    acc17(S, T);
  }
  return mont_reduce17(S);
}

// The kernels call the multiplier out of line: a verification is ~3600 products, and with every one
// inlined the kernel is 650 KB of SASS and stalls on instruction fetch (ncu: stall_no_instruction was the
// top stall reason).  Arguments and result travel in registers (no stack traffic).
#ifndef SB_MUL_NOINLINE
#define SB_MUL_NOINLINE 1
#endif
#if defined(__CUDACC__) && SB_MUL_NOINLINE
#ifndef SB_MUL_BYPTR
#define SB_MUL_BYPTR 0  // experiment: operands through local memory instead of the register ABI
#endif
#if SB_MUL_BYPTR
static __device__ __noinline__ void fq_mul_ptr(fq* r, const fq* a, const fq* b) { *r = fq_mul_inl(*a, *b); }
static __device__ __noinline__ void fq_sqr_ptr(fq* r, const fq* a) { *r = fq_sqr_inl(*a); }
static __device__ __forceinline__ fq fq_mul_ool(const fq& a, const fq& b) { fq r; fq_mul_ptr(&r, &a, &b); return r; }
static __device__ __forceinline__ fq fq_sqr_ool(const fq& a) { fq r; fq_sqr_ptr(&r, &a); return r; }
#else
static __device__ __noinline__ fq fq_mul_ool(fq a, fq b) { return fq_mul_inl(a, b); }
static __device__ __noinline__ fq fq_sqr_ool(fq a) { return fq_sqr_inl(a); }
#endif
static __device__ __noinline__ fq fq_dot5_ool(const uint32_t (*cst)[8], fq s0, fq s1, fq s2, fq s3, fq s4) {
  return fq_dot5_inl(cst, s0, s1, s2, s3, s4);
}
#endif
SB_HD fq fq_mul(const fq& a, const fq& b) {
#if defined(__CUDA_ARCH__) && SB_MUL_NOINLINE
  return fq_mul_ool(a, b);
#else
  return fq_mul_inl(a, b);
#endif
}
SB_HD fq fq_dot5(const uint32_t (*cst)[8], const fq& s0, const fq& s1, const fq& s2, const fq& s3, const fq& s4) {
#if defined(__CUDA_ARCH__) && SB_MUL_NOINLINE
  return fq_dot5_ool(cst, s0, s1, s2, s3, s4);
#else
  return fq_dot5_inl(cst, s0, s1, s2, s3, s4);
#endif
}
SB_HD fq fq_sqr(const fq& a) {
#if defined(__CUDA_ARCH__) && SB_MUL_NOINLINE
  return fq_sqr_ool(a);
#else
  return fq_sqr_inl(a);
#endif
}

// Two independent products (or squares) per out-of-line call: the two carry-chain streams sit in one basic block,
// so ptxas interleaves them and a warp waits less on the fixed latency of its own IMAD.WIDE chains (`wait` is the
// top stall of the curve code); it also halves the calls.  Used where a point operation has independent pairs.
#ifndef SB_PAIRED_MUL
#define SB_PAIRED_MUL 0  // measured: verify 18.2 -> 16.3 M/s (32 argument registers per call: more spills around the calls than stalls saved)
#endif
struct fq2 {
  fq a, b;
};
#if defined(__CUDACC__) && SB_MUL_NOINLINE
static __device__ __noinline__ fq2 fq_mul2_ool(fq a, fq b, fq c, fq d) {
  fq2 r;
  r.a = fq_mul_inl(a, b);
  r.b = fq_mul_inl(c, d);
  return r;
}
static __device__ __noinline__ fq2 fq_sqr2_ool(fq a, fq b) {
  fq2 r;
  r.a = fq_sqr_inl(a);
  r.b = fq_sqr_inl(b);
  return r;
}
#endif
SB_HD void fq_mul2(const fq& a, const fq& b, const fq& c, const fq& d, fq& r0, fq& r1) {
#if defined(__CUDA_ARCH__) && SB_MUL_NOINLINE && SB_PAIRED_MUL
  fq2 r = fq_mul2_ool(a, b, c, d);
  r0 = r.a;
  r1 = r.b;
#else
  r0 = fq_mul(a, b);
  r1 = fq_mul(c, d);
#endif
}
SB_HD void fq_sqr2(const fq& a, const fq& b, fq& r0, fq& r1) {
#if defined(__CUDA_ARCH__) && SB_MUL_NOINLINE && SB_PAIRED_MUL
  fq2 r = fq_sqr2_ool(a, b);
  r0 = r.a;
  r1 = r.b;
#else
  r0 = fq_sqr(a);
  r1 = fq_sqr(b);
#endif
}

SB_HD fq fq_to_mont(const fq& a) {
  const fq r2 = {SB200_FQ_R2_INIT};
  return fq_mul(a, r2);
}
SB_HD fq fq_from_mont(const fq& a) {
  fq one = fq_zero();
  one.v[0] = 1;
  return fq_mul(a, one);
}

// a^(q-2): 4-bit fixed windows over the constant exponent (255 squarings + 64 + 14 multiplies).
SB_HD fq fq_inv(const fq& a) {
  fq tab[16];
  tab[0] = fq_one();
  tab[1] = a;
#pragma unroll 1
  for (int i = 2; i < 16; i++) tab[i] = fq_mul(tab[i - 1], a);
  // q - 2, little-endian limbs
  const uint32_t e[8] = {0xffffffffu, 0xfffffffeu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
  fq acc = fq_one();
#pragma unroll 1
  for (int w = 63; w >= 0; w--) {
    acc = fq_sqr(acc);
    acc = fq_sqr(acc);
    acc = fq_sqr(acc);
    acc = fq_sqr(acc);
    uint32_t d = (e[w >> 3] >> ((w & 7) * 4)) & 15u;
    acc = fq_mul(acc, tab[d]);
  }
  return acc;
}

// ------------------------------------------------------------------------------------------
// Fr (generic Montgomery; only u = r - c*sk needs it: one product + one subtraction per signature,
// /root/reference/src/keys/secret.rs:165,237,448)
// ------------------------------------------------------------------------------------------
struct fr {
  uint32_t v[8];
};

SB_HD fr fr_mont_mul(const fr& a, const fr& b) {
  SB_COUNT(fr_mul, 1);
  uint32_t X[8], Y[8], xf = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) X[i] = Y[i] = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t ai = a.v[i];
    blk_fold_mac_odd(X[0], xf, 0u, Y, ai, b.v[1], b.v[3], b.v[5], b.v[7]);
    blk_mac_even(X, Y[7], ai, b.v[0], b.v[2], b.v[4], b.v[6]);
    uint32_t m = X[0] * FrP::ninv;
    blk_mac_even(X, Y[7], m, SB_FR_MOD(0), SB_FR_MOD(2), SB_FR_MOD(4), SB_FR_MOD(6));
    blk_mac_odd(Y, m, SB_FR_MOD(1), SB_FR_MOD(3), SB_FR_MOD(5), SB_FR_MOD(7));
    xf = X[1];
    uint32_t nx[8], ny[8];
#pragma unroll
    for (int k = 0; k < 8; k++) nx[k] = Y[k];
#pragma unroll
    for (int k = 0; k < 6; k++) ny[k] = X[k + 2];
    ny[6] = 0;
    ny[7] = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      X[k] = nx[k];
      Y[k] = ny[k];
    }
  }
  fr r;
  uint32_t s[8] = {xf, Y[0], Y[1], Y[2], Y[3], Y[4], Y[5], Y[6]};
  add8(r.v, X, s);
  cond_sub_p<FrP>(r.v);
  return r;
}

// canonical a * b mod r for canonical inputs:  mont(mont(a, b), R^2) = a*b*R^-1 * R^2 * R^-1
SB_HD fr fr_mul(const fr& a, const fr& b) {
  const fr r2 = {SB200_FR_R2_INIT};
  return fr_mont_mul(fr_mont_mul(a, b), r2);
}

SB_HD fr fr_sub(const fr& a, const fr& b) {
  fr r;
  uint32_t borrow = sub8(r.v, a.v, b.v);
  uint32_t t[8];
#pragma unroll
  for (int i = 0; i < 8; i++) t[i] = FrP::p(i) & borrow;
  add8(r.v, r.v, t);
  return r;
}

}  // namespace sb200
