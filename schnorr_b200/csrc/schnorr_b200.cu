// libschnorr_b200.so: sm_100a kernels + the C ABI declared in include/schnorr_b200.h.
//
// One tuple per thread, 128 threads per CTA.  Every kernel is integer-multiply bound (~3e5
// IMAD.WIDE per verification against ~300 bytes of input), so the inputs are read straight from the
// tuple-major arrays with two 128-bit loads per field element (every 32-byte sector fully used) and
// the fixed-base comb tables stay L2-resident.  Host buffers are pipelined through two streams per
// device in chunks (H2D / kernel / D2H overlap); tuples shard by index over the context's devices
// with no inter-GPU traffic.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include <map>
#include <thread>

#include "../../include/schnorr_b200.h"
#include "../../include/schnorr_b200_witness.h"
#include "../../include/schnorr_b200_keyset.h"
#include "wire.cuh"
#include "rng.cuh"
#include "params_host.cuh"

using namespace sb200;

namespace {

#ifndef SB_EC_GLOBAL_TABLES
// 1: the curve kernel of the single-key verification is PERSISTENT, keeps its two window tables in a thread-major global
// scratch region (one contiguous 128-byte entry per lookup: no sector over-fetch, 175 MB per stream that stay in L2 far better
// than 4-byte-interleaved local memory) and stages each window's two entries into shared memory with cp.async while the four
// doublings run (SB_TABLE_STAGE).  History: static tile split 20.4-22.8 M/s (the warps the scheduler favours finish early and
// leave the SM under-occupied), + L1 prefetch: no change, + cp.async staging 23.2, + work handed out per warp from a
// counter: 24.83 M verifies/s against 24.79 with local-memory tables, at 34 GB instead of 168 GB of DRAM traffic per 2^22 launch.
#define SB_EC_GLOBAL_TABLES 1
#endif
constexpr int TPB = 128;
#ifndef SB_CHALLENGE_FD
#define SB_CHALLENGE_FD 0  // the stand-alone challenge kernel on the FP64 pipe instead of IMAD.WIDE: measured equal (182.94 vs 182.91 ms per 2^22 verifications); needs SB_EXPERIMENTAL_FD
#endif
#if SB_CHALLENGE_FD && !SB_EXPERIMENTAL_FD
#error "SB_CHALLENGE_FD needs SB_EXPERIMENTAL_FD"
#endif
#ifndef SB_MIN_CTAS
#define SB_MIN_CTAS 4
#endif
// CTAs per SM the register allocator must allow: 4 (128 registers/thread) everywhere except the two kernels that
// keep a second point table live, which measure faster at 3 (168 registers, fewer spills).  [A/B timed on B200]
// The verifier-side witness kernel (op 37, OP_VERIFY_WITNESS) spills 3.9 KB per thread at 128 registers: also 3.
#ifndef SB_VERIFY_CTAS
#define SB_VERIFY_CTAS SB_MIN_CTAS
#endif
constexpr int min_ctas(int op) { return (op == 0 || op == 19) ? SB_VERIFY_CTAS : (op == 25 || op == 27 || op == 37) ? SB_MIN_CTAS - 1 : (op == 1 || op == 2) ? SB_MIN_CTAS - 1 : SB_MIN_CTAS; }
constexpr int MAX_IN = 6, MAX_OUT = 4;
constexpr int64_t CHUNK = 1 << 18;      // tuples per pipeline stage ...
constexpr int64_t CHUNK_MIN = 1 << 14;  // ... shrunk towards this when a device's share is under 4 chunks, so that H2D still overlaps compute

enum Op : int {
  OP_VERIFY = 0, OP_VERIFY_DOUBLE, OP_VERIFY_VARGEN, OP_SIGN, OP_SIGN_DOUBLE, OP_SIGN_VARGEN,
  OP_KEYGEN, OP_KEYGEN_DOUBLE, OP_KEYGEN_VARGEN, OP_DBG_FQ, OP_DBG_FR_MUL, OP_DBG_HADES, OP_DBG_SMUL,
  OP_DECOMPRESS, OP_COMPRESS, OP_FROM_WIDE, OP_VERIFY_BYTES, OP_SIGN_BYTES, OP_CHALLENGE, OP_VERIFY_EC,
  OP_VERIFY_DOUBLE_BYTES, OP_VERIFY_VARGEN_BYTES, OP_SIGN_DOUBLE_BYTES, OP_SIGN_VARGEN_BYTES,
  OP_CHALLENGE_DOUBLE, OP_VERIFY_DOUBLE_EC, OP_CHALLENGE_VARGEN, OP_VERIFY_VARGEN_EC, OP_POINTS_CHECK, OP_DBG_VERIFY_EC,
  OP_DECODE_VERIFY, OP_WITNESS, OP_DBG_LAT3,
  OP_STDRNG, OP_SIGN_STDRNG, OP_SIGN_DOUBLE_STDRNG, OP_SIGN_VARGEN_STDRNG,
  OP_VERIFY_WITNESS, OP_VERIFY_WITNESS_BYTES, OP_VERIFY_KEYSET
};
static_assert(OP_VERIFY_WITNESS == 37, "min_ctas names the op by number");

struct KArgs {
  int64_t n;
  uint32_t flags;
  int aux;
  const uint32_t* in[MAX_IN];
  uint32_t* out[MAX_OUT];
  uint32_t* bitmap;
  const uint32_t* combG;
  const uint32_t* combGp;
  const uint32_t* comb4G;   // 4-bit combs (48 KB each) of the address-oblivious path, staged into shared memory
  const uint32_t* comb4Gp;
  struct WsState* ws;
  int nsm;
  int persist;  // curve kernels: 0 = persistent form for batches above one wave (default), 1 = always, 2 = never (SB200_CURVE_PERSISTENT)
  pniels* ec_scratch;  // window tables of k_curve_p: 4 * nsm * TPB threads x EC_P_ENTRIES entries (per stream)
  uint8_t* scratch;          // device-only rows between the kernels of one call (challenges, decoded byte-level inputs)
  const uint32_t* inv_mask;  // curve kernels: verdict word &= ~inv_mask word (tuples whose from_bytes failed)
  uint32_t* dec[MAX_IN];     // decode kernel: where the decoded arrays of the byte-level verify calls go
  uint32_t rng_key[8];       // OP_STDRNG: the StdRng seed (secret: it reaches the device only as this kernel parameter)
  uint64_t rng_word;         // OP_STDRNG: keystream word position of tuple 0 of this launch
};
// The keyset of an OP_VERIFY_KEYSET launch, as this device's copy: a second kernel parameter rather than more KArgs
// fields, so that the parameter offsets of the existing two-parameter kernels (k_curve_p) stay where they are.
struct KsArgs {
  const uint32_t* tab = nullptr;  // per-key combs
  int64_t n = 0;                  // number of keys
  const uint32_t* ok = nullptr;   // key_ok bitmap
};

// scheduling state of one warp-specialised launch (k_verify_ws): the next-tile counter, reset before every launch,
// and one monotonic CTA-arrival counter per SM that rotates the hash-warp position among an SM's resident CTAs
struct WsState {
  unsigned tile;
  unsigned pad[31];
  unsigned sm_slot[512];
};

__device__ __forceinline__ fq ldg_fq(const uint32_t* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = __ldg(q), b = __ldg(q + 1);
  fq r = {{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
  return r;
}
__device__ __forceinline__ void ldg_scalar(const uint32_t* p, uint32_t* k) {
  fq t = ldg_fq(p);
#pragma unroll
  for (int i = 0; i < 8; i++) k[i] = t.v[i];
}
__device__ __forceinline__ void stg8(uint32_t* p, const uint32_t* v) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(v[0], v[1], v[2], v[3]);
  q[1] = make_uint4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ point_in ldg_point(const uint32_t* base, int64_t i, bool affine) {
  point_in p;
  const uint32_t* q = base + i * (affine ? 16 : 24);
  p.U = ldg_fq(q);
  p.V = ldg_fq(q + 8);
  p.Z = affine ? fq_one() : ldg_fq(q + 16);
  p.affine = affine;
  return p;
}
__device__ __forceinline__ void stg_point(uint32_t* base, int64_t i, const fq& u, const fq& v) {
  stg8(base + i * 16, u.v);
  stg8(base + i * 16 + 8, v.v);
}

template <int OP>
__global__ void __launch_bounds__(TPB, min_ctas(OP)) k_run(const KArgs a) {
  int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  const bool active = i < a.n;
  if (!active) i = a.n - 1;  // idle lanes redo the last tuple so the warp stays converged
  const bool aff = (a.flags & SB200_POINTS_AFFINE) != 0;
  uint32_t c[8];

  if (OP == OP_VERIFY || OP == OP_VERIFY_DOUBLE || OP == OP_VERIFY_VARGEN) {
    bool ok;
    if (OP == OP_VERIFY) {  // in: pk, u, R, m
      uint32_t u[8];
      ldg_scalar(a.in[1] + i * 8, u);
      ok = verify_core(ldg_point(a.in[0], i, aff), u, ldg_point(a.in[2], i, aff), ldg_fq(a.in[3] + i * 8), a.combG, c);
    } else if (OP == OP_VERIFY_DOUBLE) {  // in: pk, pk', u, R, R', m
      uint32_t u[8];
      ldg_scalar(a.in[2] + i * 8, u);
      ok = verify_double_core(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                              ldg_point(a.in[4], i, aff), ldg_fq(a.in[5] + i * 8), a.combG, a.combGp, c);
    } else {  // in: pk, gen, u, R, m
      uint32_t u[8];
      ldg_scalar(a.in[2] + i * 8, u);
      ok = verify_vargen_core(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                              ldg_fq(a.in[4] + i * 8), c);
    }
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = word;
    if (a.out[0] && active) stg8(a.out[0] + i * 8, c);
    return;
  }

  // single-key verification as two launches (SB_VERIFY_SPLIT): all warps of an SM are then in the same phase, and each
  // phase's code (hash: 26 KB, curve: 19 KB) fits the 32 KB L1.5 instruction cache by itself
  if (OP == OP_CHALLENGE) {  // in: -, -, R, m -> out0: c
#if SB_CHALLENGE_FD
    {  // the challenge kernel on the FP64 pipe (hades_fd.cuh): nothing else competes for issue slots here
      fq ru, rv;
      point_to_affine(ldg_point(a.in[2], i, aff), ru, rv);
      challenge3_fd(ru, rv, ldg_fq(a.in[3] + i * 8), c);
    }
#else
    verify_hash_core(ldg_point(a.in[2], i, aff), ldg_fq(a.in[3] + i * 8), c);
#endif
    if (active) stg8(a.out[0] + i * 8, c);
#if SB_EC_GLOBAL_TABLES
    if (blockIdx.x == 0 && threadIdx.x == 0) a.ws->tile = 0;  // the persistent curve kernel's work counter
#endif
    return;
  }
  if (OP == OP_VERIFY_EC) {  // in: pk, u, R, - ; out0 (as input): c -> bitmap
    uint32_t u[8];
    ldg_scalar(a.in[1] + i * 8, u);
    ldg_scalar(a.out[0] + i * 8, c);
    bool ok = verify_ec(ldg_point(a.in[0], i, aff), u, ldg_point(a.in[2], i, aff), c, a.combG);
    if (a.flags & SB200_CHECK_POINTS) {  // warp-uniform
#pragma unroll 1
      for (int k = 0; k < 3; k += 2) ok &= point_well_formed(ldg_point(a.in[k], i, aff));
    }
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = a.inv_mask ? word & ~a.inv_mask[i >> 5] : word;
    return;
  }
  if (OP == OP_POINTS_CHECK) {  // in: points -> bitmap
    bool ok = point_well_formed(ldg_point(a.in[0], i, aff));
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = word;
    return;
  }

  if (OP == OP_CHALLENGE_VARGEN) {  // in: -, -, -, R, m -> out0: c
    verify_hash_core(ldg_point(a.in[3], i, aff), ldg_fq(a.in[4] + i * 8), c);
    if (active) stg8(a.out[0] + i * 8, c);
#if SB_EC_GLOBAL_TABLES
    if (blockIdx.x == 0 && threadIdx.x == 0) a.ws->tile = 0;  // the persistent curve kernel's work counter
#endif
    return;
  }
  if (OP == OP_VERIFY_VARGEN_EC) {  // in: pk, gen, u, R, - ; out0 (as input): c -> bitmap
    uint32_t u[8];
    ldg_scalar(a.in[2] + i * 8, u);
    ldg_scalar(a.out[0] + i * 8, c);
    bool ok = verify_vargen_ec_auto(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff), c);
    if (a.flags & SB200_CHECK_POINTS) {
#pragma unroll 1
      for (int k = 0; k < 4; k++)
        if (k != 2) ok &= point_well_formed(ldg_point(a.in[k], i, aff));
    }
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = a.inv_mask ? word & ~a.inv_mask[i >> 5] : word;
    return;
  }
  if (OP == OP_CHALLENGE_DOUBLE) {  // in: -, -, -, R, R', m -> out0: c
    verify_double_hash_core(ldg_point(a.in[3], i, aff), ldg_point(a.in[4], i, aff), ldg_fq(a.in[5] + i * 8), c);
    if (active) stg8(a.out[0] + i * 8, c);
#if SB_EC_GLOBAL_TABLES
    if (blockIdx.x == 0 && threadIdx.x == 0) a.ws->tile = 0;  // the persistent curve kernel's work counter
#endif
    return;
  }
  if (OP == OP_VERIFY_DOUBLE_EC) {  // in: pk, pk', u, R, R', - ; out0 (as input): c -> bitmap
    uint32_t u[8];
    ldg_scalar(a.in[2] + i * 8, u);
    ldg_scalar(a.out[0] + i * 8, c);
    bool ok = verify_double_ec(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                               ldg_point(a.in[4], i, aff), c, a.combG, a.combGp);
    if (a.flags & SB200_CHECK_POINTS) {
#pragma unroll 1
      for (int k = 0; k < 5; k++)
        if (k != 2) ok &= point_well_formed(ldg_point(a.in[k], i, aff));
    }
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = a.inv_mask ? word & ~a.inv_mask[i >> 5] : word;
    return;
  }

  // First kernel of the byte-level verify calls (sb200_verify{,_double,_vargen}_bytes): every from_bytes of the tuple
  // -- JubJubAffine::from_bytes for the points (/root/reference/src/keys/public.rs:94-100, signatures.rs:119-122),
  // JubJubScalar::from_bytes for u, BlsScalar::from_bytes for the message -- writing the decoded arrays in the layout
  // the challenge and curve kernels read (affine Montgomery points, canonical u, Montgomery m) and the invalid bitmap.
  // Its own launch: decompression (one 255-bit exponentiation per point) is a different code phase from the
  // permutation and the curve loop, and the three do not fit the instruction cache together (DESIGN.md 4.5).
  // aux: 0 single (pk32, sig64 -> pk, u, R, m), 1 double (pk64, sig96 -> pk, pk', u, R, R', m),
  //      2 vargen (pk64, sig64 -> pk, gen, u, R, m).  in: pk bytes, sig bytes, msg32.
  if (OP == OP_DECODE_VERIFY) {
    const int npk = a.aux == 0 ? 1 : 2, nr = a.aux == 1 ? 2 : 1;
    bool ok = true;
#pragma unroll 1
    for (int k = 0; k < npk + nr; k++) {  // one copy of the decompression code
      const uint32_t* src = k < npk ? a.in[0] + i * (8 * npk) + 8 * k : a.in[1] + i * (8 + 8 * nr) + 8 + 8 * (k - npk);
      uint32_t* dst = k < npk ? a.dec[k] : a.dec[npk + 1 + (k - npk)];
      uint32_t b[8];
      fq u, v;
      ldg_scalar(src, b);
      ok &= point_decompress(b, u, v);
      if (active) stg_point(dst, i, u, v);
    }
    uint32_t us[8], mb[8];
    fq m;
    ldg_scalar(a.in[1] + i * (8 + 8 * nr), us);
    ldg_scalar(a.in[2] + i * 8, mb);
    ok &= scalar_lt_r(us);
    ok &= msg_from_bytes(mb, m);
    if (active) {
      stg8(a.dec[npk] + i * 8, us);
      stg8(a.dec[npk + 1 + nr] + i * 8, m.v);
    }
    unsigned inv = __ballot_sync(0xffffffffu, !ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = inv;
    return;
  }

  if (OP == OP_SIGN || OP == OP_SIGN_DOUBLE || OP == OP_SIGN_VARGEN) {
    // out: u, R, (R'), c
    uint32_t sk[8], nonce[8], u[8];
    fq Ru, Rv;
    ldg_scalar(a.in[0] + i * 8, sk);
    if (OP == OP_SIGN) {  // in: sk, m, nonce
      ldg_scalar(a.in[2] + i * 8, nonce);
      sign_core(sk, nonce, ldg_fq(a.in[1] + i * 8), a.combG, u, Ru, Rv, c);
    } else if (OP == OP_SIGN_DOUBLE) {
      fq Rpu, Rpv;
      ldg_scalar(a.in[2] + i * 8, nonce);
      sign_double_core(sk, nonce, ldg_fq(a.in[1] + i * 8), a.combG, a.combGp, u, Ru, Rv, Rpu, Rpv, c);
      if (active) stg_point(a.out[2], i, Rpu, Rpv);
    } else {  // in: sk, gen, m, nonce
      ldg_scalar(a.in[3] + i * 8, nonce);
      sign_vargen_core(sk, ldg_point(a.in[1], i, aff), nonce, ldg_fq(a.in[2] + i * 8), u, Ru, Rv, c, (a.flags & SB200_SIGN_OBLIVIOUS) != 0);
    }
    if (active) {
      stg8(a.out[0] + i * 8, u);
      stg_point(a.out[1], i, Ru, Rv);
      if (a.out[3]) stg8(a.out[3] + i * 8, c);
    }
    return;
  }

  if (OP == OP_KEYGEN || OP == OP_KEYGEN_DOUBLE || OP == OP_KEYGEN_VARGEN) {
    uint32_t sk[8];
    fq u, v;
    ldg_scalar(a.in[0] + i * 8, sk);
    if (OP == OP_KEYGEN_VARGEN) {
      const point_in g = ldg_point(a.in[1], i, aff);
      ext_to_affine((a.flags & SB200_SIGN_OBLIVIOUS) ? var_base_mul_oblivious(g, sk) : var_base_mul(g, sk), u, v,
                    (a.flags & SB200_SIGN_OBLIVIOUS) != 0);
    } else {
      ext_to_affine(fixed_base_mul(a.combG, sk), u, v);
    }
    if (active) stg_point(a.out[0], i, u, v);
    if (OP == OP_KEYGEN_DOUBLE) {
      ext_to_affine(fixed_base_mul(a.combGp, sk), u, v);
      if (active) stg_point(a.out[1], i, u, v);
    }
    return;
  }

  if (OP == OP_WITNESS) {  // in: sk, msg, nonce (, generator) -> out0: witness rows; aux = scheme
    uint32_t sk[8], nonce[8];
    ldg_scalar(a.in[0] + i * 8, sk);
    ldg_scalar(a.in[2] + i * 8, nonce);
    const fq m = ldg_fq(a.in[1] + i * 8);
    const int w = a.aux == 0 ? 11 : a.aux == 1 ? 19 : 13;
    uint32_t* dst = a.out[0] + i * w * 8;
    auto emit = [&](int k, const fq& v) { if (active) stg8(dst + k * 8, v.v); };
    if (a.aux == 0) witness_core<0>(sk, nonce, m, point_in(), a.combG, a.combGp, emit);
    else if (a.aux == 1) witness_core<1>(sk, nonce, m, point_in(), a.combG, a.combGp, emit);
    else witness_core<2>(sk, nonce, m, ldg_point(a.in[3], i, aff), a.combG, a.combGp, emit);
    return;
  }
  if (OP == OP_VERIFY_WITNESS) {  // aux = scheme; in: pk, u, R, m | pk, pk', u, R, R', m | pk, gen, u, R, m -> out0: rows, bitmap
    // inv_mask (byte-level call): tuples whose from_bytes failed get a zero row and verdict 0, like the core's own zeroing
    const bool keep = !a.inv_mask || !(a.inv_mask[i >> 5] >> (i & 31) & 1u);
    const bool chk = (a.flags & SB200_CHECK_POINTS) != 0;
    uint32_t u[8];
    ldg_scalar(a.in[a.aux == 0 ? 1 : 2] + i * 8, u);
    uint32_t* dst = a.out[0] + i * SB200_WITNESS_WIDTH(a.aux) * 8;
    auto emit = [&](int k, const fq& v) {
      const fq x = keep ? v : fq_zero();
      if (active) stg8(dst + k * 8, x.v);
    };
    bool ok;
    if (a.aux == 0)
      ok = verify_witness_core<0>(ldg_point(a.in[0], i, aff), point_in(), u, ldg_point(a.in[2], i, aff), point_in(),
                                  ldg_fq(a.in[3] + i * 8), chk, a.combG, a.combGp, emit);
    else if (a.aux == 1)
      ok = verify_witness_core<1>(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                                  ldg_point(a.in[4], i, aff), ldg_fq(a.in[5] + i * 8), chk, a.combG, a.combGp, emit);
    else
      ok = verify_witness_core<2>(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                                  point_in(), ldg_fq(a.in[4] + i * 8), chk, a.combG, a.combGp, emit);
    unsigned word = __ballot_sync(0xffffffffu, ok && keep && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = word;
    return;
  }
  if (OP == OP_DBG_FQ) {
    fq x = ldg_fq(a.in[0] + i * 8), y = a.in[1] ? ldg_fq(a.in[1] + i * 8) : fq_zero(), r;
    switch (a.aux) {
      case 0: r = fq_mul(x, y); break;
      case 1: r = fq_add(x, y); break;
      case 2: r = fq_sub(x, y); break;
      case 3: r = fq_inv(x); break;
      case 4: r = fq_sqr(x); break;
      case 5: r = fq_to_mont(x); break;
      case 7: r = fq_inv_fast(x); break;
      default: r = fq_from_mont(x); break;
    }
    if (active) stg8(a.out[0] + i * 8, r.v);
    return;
  }
  if (OP == OP_DBG_LAT3) {  // in: c, u (canonical scalars) -> a | b | d | (aneg, bneg, dneg, ok, 0, 0, 0, 0)
    uint32_t c[8], u[8];
    ldg_scalar(a.in[0] + i * 8, c);
    ldg_scalar(a.in[1] + i * 8, u);
    lat3_res r = lattice3_8r(c, u);
    const uint32_t f[8] = {r.aneg, r.bneg, r.dneg, r.ok, 0u, 0u, 0u, 0u};
    if (active) {
      stg8(a.out[0] + i * 32, r.a);
      stg8(a.out[0] + i * 32 + 8, r.b);
      stg8(a.out[0] + i * 32 + 16, r.d);
      stg8(a.out[0] + i * 32 + 24, f);
    }
    return;
  }
  if (OP == OP_DBG_FR_MUL) {
    fr x, y;
    ldg_scalar(a.in[0] + i * 8, x.v);
    ldg_scalar(a.in[1] + i * 8, y.v);
    fr r = fr_mul(x, y);
    if (active) stg8(a.out[0] + i * 8, r.v);
    return;
  }
  if (OP == OP_DBG_HADES) {
    fq s[5];
#pragma unroll
    for (int k = 0; k < 5; k++) s[k] = ldg_fq(a.in[0] + i * 40 + k * 8);
#if SB_EXPERIMENTAL_FD
    if (a.aux == 2) {  // FP64-pipe permutation (hades_fd.cuh); same Montgomery-2^256 words in and out
      fd t[5];
#pragma unroll 1
      for (int k = 0; k < 5; k++) t[k] = fd_from_fq(s[k]);
      hades_perm_fd(t);
#pragma unroll 1
      for (int k = 0; k < 5; k++) {
        fd_to_canonical(t[k], s[k].v);
        s[k] = fq_to_mont(s[k]);
      }
    } else
#endif
    if (a.aux) hades_perm_dense(s); else hades_perm(s);
    if (active) {
#pragma unroll
      for (int k = 0; k < 5; k++) stg8(a.out[0] + i * 40 + k * 8, s[k].v);
    }
    return;
  }
  if (OP == OP_DBG_SMUL) {  // in: points (base 2 only), k
    uint32_t k[8];
    fq u, v;
    ldg_scalar(a.in[1] + i * 8, k);
    if (a.aux == 2) ext_to_affine(var_base_mul(ldg_point(a.in[0], i, aff), k), u, v);
    else ext_to_affine(fixed_base_mul(a.aux == 0 ? a.combG : a.combGp, k), u, v);
    if (active) stg_point(a.out[0], i, u, v);
    return;
  }
  if (OP == OP_DECOMPRESS) {  // in: bytes32 -> out0: affine points, bitmap: ok
    uint32_t b[8];
    fq u, v;
    ldg_scalar(a.in[0] + i * 8, b);
    bool ok = point_decompress(b, u, v);
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = word;
    if (active) stg_point(a.out[0], i, u, v);
    return;
  }
  if (OP == OP_COMPRESS) {  // in: points -> out0: bytes32
    point_in p = ldg_point(a.in[0], i, aff);
    fq u, v;
    point_to_affine(p, u, v);
    uint32_t b[8];
    point_compress(u, v, b);
    if (active) stg8(a.out[0] + i * 8, b);
    return;
  }
  if (OP == OP_FROM_WIDE) {  // in: 64-byte draws -> out0: scalar (aux 0: mod r canonical, aux 1: mod q Montgomery)
    uint32_t w[16], r[8];
    ldg_scalar(a.in[0] + i * 16, w);
    ldg_scalar(a.in[0] + i * 16 + 8, w + 8);
    if (a.aux == 0) {
      fr_from_wide(w, r);
    } else {
      fq x = fq_from_wide(w);
#pragma unroll
      for (int k = 0; k < 8; k++) r[k] = x.v[k];
    }
    if (active) stg8(a.out[0] + i * 8, r);
    return;
  }
  if (OP == OP_STDRNG) {  // -> out0: Field::random draw i at word rng_word + 16 i (aux 0: mod r canonical, aux 1: mod q Montgomery)
    uint32_t r[8];
    stdrng_random(a.rng_key, a.rng_word + 16u * (uint64_t)i, a.aux, r);
    if (active) stg8(a.out[0] + i * 8, r);
    return;
  }
  if (OP == OP_SIGN_DOUBLE_BYTES) {  // in: sk32, msg32, nonce32 -> out0: sig96 = u || R || R', bitmap (nullable): invalid
    uint32_t sk[8], nonce[8], mb[8], sig[24];
    ldg_scalar(a.in[0] + i * 8, sk);
    ldg_scalar(a.in[1] + i * 8, mb);
    ldg_scalar(a.in[2] + i * 8, nonce);
    bool ok = sign_double_bytes_core(sk, mb, nonce, a.combG, a.combGp, sig);
    unsigned inv = __ballot_sync(0xffffffffu, !ok && active);
    if ((threadIdx.x & 31) == 0 && active && a.bitmap) a.bitmap[i >> 5] = inv;
    if (active) {
#pragma unroll
      for (int k = 0; k < 3; k++) stg8(a.out[0] + i * 24 + 8 * k, sig + 8 * k);
    }
    return;
  }
  if (OP == OP_SIGN_VARGEN_BYTES) {  // in: sk64 (sk || generator), msg32, nonce32 -> out0: sig64, bitmap (nullable): invalid
    uint32_t sk[16], nonce[8], mb[8], sig[16];
    ldg_scalar(a.in[0] + i * 16, sk);
    ldg_scalar(a.in[0] + i * 16 + 8, sk + 8);
    ldg_scalar(a.in[1] + i * 8, mb);
    ldg_scalar(a.in[2] + i * 8, nonce);
    bool ok = sign_vargen_bytes_core(sk, mb, nonce, sig);
    unsigned inv = __ballot_sync(0xffffffffu, !ok && active);
    if ((threadIdx.x & 31) == 0 && active && a.bitmap) a.bitmap[i >> 5] = inv;
    if (active) {
      stg8(a.out[0] + i * 16, sig);
      stg8(a.out[0] + i * 16 + 8, sig + 8);
    }
    return;
  }
}

// ------------------------------------------------------------------------------------------------
// Warp-specialised single-key verification: one persistent 512-thread CTA per SM = 8 hash warps + 8 curve warps,
// i.e. on every SM sub-partition (warp w runs on sub-partition w % 4) 2 hash warps beside 2 curve warps.
//
// The curve half of a verification (c*PK + u*G == R) saturates the FMA-heavy pipe with IMAD.WIDE while using ~40 %
// of the issue slots; the Poseidon challenge on the FP64 pipe (hades_fd.cuh) needs issue slots and the FP64 / ALU
// pipes only.  Keeping both kinds of warp on every sub-partition at all times overlaps the two: the hash warps
// compute the challenges of the CTA's NEXT tile into shared memory while the curve warps verify the current tile.
// Two curve warps per sub-partition already drive the FMA-heavy pipe to 94 % of what four do (measured with the
// single-role kernel at 2 CTAs/SM), so the other two warp slots of the 128-register budget go to hash warps; a hash
// warp alone is latency-bound (IPC ~0.17 measured), two per sub-partition keep up with one challenge per
// verification.  Tile = 8 x 32 = 256 tuples per iteration, handed out by a global counter; verdict words never
// straddle warps.
// ------------------------------------------------------------------------------------------------
#ifndef SB_VERIFY_WS
#define SB_VERIFY_WS SB_EXPERIMENTAL_FD  // compiled out of the product library: measured 22 % slower than the default path
#endif
#ifndef SB_VARGEN_SPLIT
#define SB_VARGEN_SPLIT 1
#endif
#ifndef SB_VERIFY_SPLIT
#define SB_VERIFY_SPLIT 1  // hash and curve halves as two launches: with the half-size curve path the single kernel's phases evict each other from the instruction cache (21.1 -> 22.9 M verifies/s)
#endif
#ifndef SB_WS_SETMAXNREG
#define SB_WS_SETMAXNREG 0
#endif
#ifndef SB_WS_HREGS
#define SB_WS_HREGS 56
#endif
#ifndef SB_WS_EREGS
#define SB_WS_EREGS 120
#endif
#if SB_VERIFY_WS
constexpr int WS_HW = 8, WS_EW = 8, WS_THREADS = (WS_HW + WS_EW) * 32, WS_EPER = 1;
constexpr int WS_TILE = WS_EW * 32 * WS_EPER;       // 256 tuples per iteration
constexpr int WS_HPER = WS_TILE / (WS_HW * 32);     // 1 hash per hash lane
constexpr size_t WS_SMEM = (size_t)2 * WS_TILE * 8 * sizeof(uint32_t);
static_assert(WS_HPER * WS_HW * 32 == WS_TILE, "hash and curve warps must cover the same tile");
__global__ void __launch_bounds__(WS_THREADS, 1) k_verify_ws(const KArgs a) {
  extern __shared__ __align__(16) uint32_t ws_smem[];
  uint32_t(*cbuf)[WS_TILE][8] = reinterpret_cast<uint32_t(*)[WS_TILE][8]>(ws_smem);
  __shared__ unsigned tiles[2];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool aff = (a.flags & SB200_POINTS_AFFINE) != 0;
  const unsigned ntiles = (unsigned)((a.n + WS_TILE - 1) / WS_TILE);
  if (tid == 0) tiles[0] = atomicAdd(&a.ws->tile, 1u);
  __syncthreads();
  const bool is_hash = warp < WS_HW;
#if SB_WS_SETMAXNREG
  // register re-partitioning between warpgroups: the hash warps give up what the curve warps need
  if (is_hash) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(SB_WS_HREGS));
  else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(SB_WS_EREGS));
#endif

  auto hash_tile = [&](unsigned t, uint32_t (*buf)[8]) {
#pragma unroll 1
    for (int s = 0; s < WS_HPER; s++) {
      const int local = (s * WS_HW + warp) * 32 + lane;
      int64_t i = (int64_t)t * WS_TILE + local;
      const bool act = i < a.n;
      if (!act) i = a.n - 1;
      uint32_t c[8];
      fq ru, rv;
      point_to_affine(ldg_point(a.in[2], i, aff), ru, rv);
      challenge3_fd(ru, rv, ldg_fq(a.in[3] + i * 8), c);
      stg8(buf[local], c);
      if (a.out[0] && act) stg8(a.out[0] + i * 8, c);
    }
  };

  int cur = 0;
  if (is_hash && tiles[0] < ntiles) hash_tile(tiles[0], cbuf[0]);
  if (tid == 0) tiles[1] = atomicAdd(&a.ws->tile, 1u);
  __syncthreads();
  while (tiles[cur] < ntiles) {
    const unsigned t = tiles[cur], tn = tiles[cur ^ 1];
    if (is_hash) {
      if (tn < ntiles) hash_tile(tn, cbuf[cur ^ 1]);
    } else {
#pragma unroll 1
      for (int s = 0; s < WS_EPER; s++) {
        const int local0 = (s * WS_EW + (warp - WS_HW)) * 32;
        const int64_t i0 = (int64_t)t * WS_TILE + local0;
        if (i0 >= a.n) break;  // warp-uniform
        int64_t i = i0 + lane;
        const bool act = i < a.n;
        if (!act) i = a.n - 1;
        uint32_t u[8], c[8];
        ldg_scalar(a.in[1] + i * 8, u);
        const uint4* cp = reinterpret_cast<const uint4*>(cbuf[cur][act ? local0 + lane : local0]);
        uint4 c0 = cp[0], c1 = cp[1];
        c[0] = c0.x; c[1] = c0.y; c[2] = c0.z; c[3] = c0.w; c[4] = c1.x; c[5] = c1.y; c[6] = c1.z; c[7] = c1.w;
        bool ok = verify_ec_core(ldg_point(a.in[0], i, aff), u, ldg_point(a.in[2], i, aff), c, a.combG);
        unsigned word = __ballot_sync(0xffffffffu, ok && act);
        if (lane == 0) a.bitmap[i0 >> 5] = word;
      }
    }
    __syncthreads();
    if (tid == 0) tiles[cur] = atomicAdd(&a.ws->tile, 1u);
    cur ^= 1;
    __syncthreads();
  }
}

#endif  // SB_VERIFY_WS

// Curve half of the single-key verification as a persistent kernel whose window tables live in a thread-major global
// scratch region (18 entries x 128 B per resident thread) instead of local memory: see verify_ec_half.
#if SB_EC_GLOBAL_TABLES
// Persistent curve kernels of the three verifications (SCHEME 0 single-key, 1 double-key, 2 variable-generator): window tables
// in a thread-major global scratch region (EC_P_ENTRIES x 128 B per resident thread), the coming window's entries staged into
// dynamic shared memory by cp.async (16 or 24 uint4 per thread), work handed out per warp from a counter that the preceding
// challenge kernel reset.
#ifndef SB_EC_P_CTAS0
#define SB_EC_P_CTAS0 4  // resident CTAs per SM of the single-key curve kernel; measured 4 / 5 / 6 (128 / 96 / 80 registers): 24.93 / 24.95 / 25.02 M verifies/s -- occupancy is not the limiter
#endif
#ifndef SB_EC_P_CTAS_ALL4
#define SB_EC_P_CTAS_ALL4 1  // 4 CTAs per SM (128 registers) for the double-key and variable-generator forms too: with the tables out of
                             // local memory the spills are cheap -- measured 12.07 -> 12.50 and 18.05 -> 18.45 M verifies/s against 3 CTAs at 168
#endif
constexpr int EC_P_ENTRIES = 27;  // three 9-entry tables (the single- and double-key forms use 18)
constexpr int ec_p_ctas(int scheme) { return (SB_EC_P_CTAS0 != 4 && scheme == 0) ? SB_EC_P_CTAS0 : (SB_EC_P_CTAS_ALL4 ? 4 : (scheme == 0 ? 4 : 3)); }
constexpr size_t ec_p_smem(int scheme) { return (size_t)(scheme == 2 ? 24 : 16) * TPB * sizeof(uint4); }
template <int SCHEME>
__global__ void __launch_bounds__(TPB, ec_p_ctas(SCHEME)) k_curve_p(const KArgs a, pniels* scratch) {
  const bool aff = (a.flags & SB200_POINTS_AFFINE) != 0;
  pniels* store = scratch + ((size_t)blockIdx.x * TPB + threadIdx.x) * EC_P_ENTRIES;
  extern __shared__ __align__(16) uint4 stage_buf[];
#if SB_TABLE_STAGE
  uint4* stage = stage_buf;
#else
  uint4* stage = nullptr;
#endif
  // work is handed out per WARP from a counter (reset by the challenge kernel that precedes this one on the stream): with a
  // static split the warps the scheduler favours run ahead, finish their share early and leave the SM under-occupied for the
  // rest of the launch (measured: 20 % of the warp slots active instead of 24 %)
  const unsigned nwt = (unsigned)((a.n + 31) / 32);
#pragma unroll 1
  for (;;) {
    unsigned w = 0;
    if ((threadIdx.x & 31) == 0) w = atomicAdd(&a.ws->tile, 1u);
    w = __shfl_sync(0xffffffffu, w, 0);
    if (w >= nwt) break;
    int64_t i = (int64_t)w * 32 + (threadIdx.x & 31);
    const bool active = i < a.n;
    if (!active) i = a.n - 1;
    uint32_t u[8], c[8];
    ldg_scalar(a.in[SCHEME == 0 ? 1 : 2] + i * 8, u);
    ldg_scalar(a.out[0] + i * 8, c);
    bool ok;
    if (SCHEME == 0) {  // in: pk, u, R
      ok = verify_ec<true>(ldg_point(a.in[0], i, aff), u, ldg_point(a.in[2], i, aff), c, a.combG, store, stage);
    } else if (SCHEME == 1) {  // in: pk, pk', u, R, R'
      ok = verify_double_ec<true>(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff),
                                  ldg_point(a.in[4], i, aff), c, a.combG, a.combGp, store, stage);
    } else {  // in: pk, gen, u, R
      ok = verify_vargen_ec_auto<true>(ldg_point(a.in[0], i, aff), ldg_point(a.in[1], i, aff), u, ldg_point(a.in[3], i, aff), c, store,
                                       stage);
    }
    if (a.flags & SB200_CHECK_POINTS) {  // warp-uniform
      constexpr int NPT = SCHEME == 0 ? 3 : SCHEME == 1 ? 5 : 4, SKIP = SCHEME == 0 ? 1 : 2;
#pragma unroll 1
      for (int k = 0; k < NPT; k++)
        if (k != SKIP) ok &= point_well_formed(ldg_point(a.in[k], i, aff));
    }
    unsigned word = __ballot_sync(0xffffffffu, ok && active);
    if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = a.inv_mask ? word & ~a.inv_mask[i >> 5] : word;
  }
}
#endif  // SB_EC_GLOBAL_TABLES

// Fixed-base signing / key generation with several tuples per thread: the scalar multiples of G (and G') are
// computed first, all their Z coordinates are inverted together (one field inversion per thread instead of one
// per point: the inversion is a third of a single signature's work), then each tuple is finished.
// Thread t of a CTA handles tuples base + j * TPB + t (j < K): loads and stores stay coalesced.
// Tuples per thread: 4 when signing (the hash dominates, more only adds local-memory traffic), SB_KEYGEN_K for key
// generation, where the shared inversion is a quarter of the work at 4 (measured: 311 M keys/s at 4, 369 at 8, 351 at 16).
#ifndef SB_SIGN_K
#define SB_SIGN_K 4
#endif
#ifndef SB_KEYGEN_K
#define SB_KEYGEN_K 8
#endif
__host__ __device__ constexpr int fixed_k(int op) { return (op == OP_KEYGEN || op == OP_KEYGEN_DOUBLE) ? SB_KEYGEN_K : SB_SIGN_K; }
// CT = true (SB200_SIGN_OBLIVIOUS): the scalar multiples come from 4-bit combs staged in shared memory and read
// by masked scan (ed.cuh), so no address depends on a nonce or key -- the "branch-free fixed-base comb tables staged in
// shared memory" form; 64 additions per multiple instead of 16 (measured: DESIGN.md 4.2).
#ifndef SB_CTA_INVERSE
#define SB_CTA_INVERSE 0  // measured with Fermat's inversion: sign 65.4 -> 67.2 M/s, keygen 411 -> 462 M/s, sign_double -0.8 % (the lone inverting warp per sub-partition runs at ~57 % efficiency); superseded by the Euclidean inversion (inv.cuh), which leaves nothing worth sharing
#endif
// One field inversion per CTA instead of one per warp.  In SIMT terms the 32 lanes of a warp already share the instruction
// stream of "their" inversion; what can still be shared is the stream itself, between the four warps of a CTA: every thread
// leaves the product it wants inverted in shared memory, ONE warp (rotating with the CTA index, so that the four SM
// sub-partitions take turns) multiplies the four values of its lane position together, inverts once (78 multiplications +
// 256 squarings) and unfolds the four inverses with six more multiplications, while the other three warps wait at the
// barrier without issuing anything.  Saves 3 of 4 inversions per CTA: 6.5 % of a signature's issue time, 20 % of a key's.
__device__ __forceinline__ fq cta_shared_inverse(const fq& acc) {
#if SB_CTA_INVERSE
  static_assert(TPB == 128, "four warps per CTA");
  __shared__ uint32_t sh[8][TPB];  // limb-major: conflict-free
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, lead = blockIdx.x & 3;
#pragma unroll
  for (int k = 0; k < 8; k++) sh[k][threadIdx.x] = acc.v[k];
  __syncthreads();
  if (warp == lead) {  // warp-uniform
    fq v[4];
#pragma unroll
    for (int w = 0; w < 4; w++)
#pragma unroll
      for (int k = 0; k < 8; k++) v[w].v[k] = sh[k][w * 32 + lane];
    const fq p1 = fq_mul(v[0], v[1]), p2 = fq_mul(p1, v[2]);
    fq t = fq_inv(fq_mul(p2, v[3]));
    const fq i3 = fq_mul(t, p2);
    t = fq_mul(t, v[3]);
    const fq i2 = fq_mul(t, p1);
    t = fq_mul(t, v[2]);
    const fq i1 = fq_mul(t, v[0]), i0 = fq_mul(t, v[1]);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      sh[k][lane] = i0.v[k];
      sh[k][32 + lane] = i1.v[k];
      sh[k][64 + lane] = i2.v[k];
      sh[k][96 + lane] = i3.v[k];
    }
  }
  __syncthreads();
  fq r;
#pragma unroll
  for (int k = 0; k < 8; k++) r.v[k] = sh[k][threadIdx.x];
  return r;
#else
  return fq_inv(acc);
#endif
}
// z[0..n) <- 1 / z[0..n): Montgomery's trick inside the thread (core.cuh batch_inverse) around the CTA-shared inversion
template <bool FAST>
__device__ __forceinline__ void batch_inverse_cta(fq* z, fq* pre, int n) {
  fq acc = z[0];
  pre[0] = fq_one();
#pragma unroll 1
  for (int j = 1; j < n; j++) {
    pre[j] = acc;
    acc = fq_mul(acc, z[j]);
  }
  fq inv = SB_CTA_INVERSE ? cta_shared_inverse(acc) : (FAST ? fq_inv_fast(acc) : fq_inv(acc));
#pragma unroll 1
  for (int j = n - 1; j > 0; j--) {
    fq zj = z[j];
    z[j] = fq_mul(inv, pre[j]);
    inv = fq_mul(inv, zj);
  }
  z[0] = inv;
}

template <int OP, bool CT = false>
__global__ void __launch_bounds__(TPB, CT ? 2 : 4) k_fixed_batch(const KArgs a) {
  constexpr int SIGN_K = fixed_k(OP);
  constexpr bool DOUBLE = (OP == OP_SIGN_DOUBLE || OP == OP_KEYGEN_DOUBLE);
  extern __shared__ __align__(16) uint32_t ct_tab[];  // CT: [G | G'] 4-bit combs
  if (CT) {
    const uint4* src[2] = {reinterpret_cast<const uint4*>(a.comb4G), reinterpret_cast<const uint4*>(a.comb4Gp)};
    uint4* dst = reinterpret_cast<uint4*>(ct_tab);
#pragma unroll 1
    for (int t = 0; t < (DOUBLE ? 2 : 1); t++)
      for (int k = threadIdx.x; k < CT_TABLE_WORDS / 4; k += TPB) dst[t * (CT_TABLE_WORDS / 4) + k] = __ldg(src[t] + k);
    __syncthreads();
  }
  constexpr bool SIGN = (OP == OP_SIGN || OP == OP_SIGN_DOUBLE || OP == OP_SIGN_BYTES);
  constexpr int NP = DOUBLE ? 2 * SIGN_K : SIGN_K;
  const int64_t base = (int64_t)blockIdx.x * TPB * SIGN_K + threadIdx.x;
  fq X[NP], Y[NP], Z[NP], pre[NP];
  // scalar whose multiple is needed: the nonce when signing, the secret key for keygen
  const uint32_t* kin = SIGN ? a.in[2] : a.in[0];
#pragma unroll 1
  for (int j = 0; j < SIGN_K; j++) {
    int64_t i = base + (int64_t)j * TPB;
    if (i >= a.n) i = a.n - 1;
    uint32_t k[8];
    ldg_scalar(kin + i * 8, k);
    if (OP == OP_SIGN_BYTES) {  // JubJubScalar::from_bytes of the nonce: >= r is reported invalid below, 0 keeps the recoding in range
      const bool lt = scalar_lt_r(k);
#pragma unroll
      for (int w = 0; w < 8; w++) k[w] = lt ? k[w] : 0u;
    }
    ext p = CT ? fixed_base_mul_oblivious(ct_tab, k) : fixed_base_mul(a.combG, k);
    X[j] = p.X; Y[j] = p.Y; Z[j] = p.Z;
    if (DOUBLE) {
      ext q = CT ? fixed_base_mul_oblivious(ct_tab + CT_TABLE_WORDS, k) : fixed_base_mul(a.combGp, k);
      X[SIGN_K + j] = q.X; Y[SIGN_K + j] = q.Y; Z[SIGN_K + j] = q.Z;
    }
  }
  batch_inverse_cta<!CT>(Z, pre, NP);  // the address-oblivious signer keeps Fermat's constant-time inversion
#pragma unroll 1
  for (int j = 0; j < SIGN_K; j++) {
    int64_t i = base + (int64_t)j * TPB;
    const bool active = i < a.n;
    if (!active) i = a.n - 1;
    fq Ru = fq_mul(X[j], Z[j]), Rv = fq_mul(Y[j], Z[j]), Rpu, Rpv;
    if (DOUBLE) {
      Rpu = fq_mul(X[SIGN_K + j], Z[SIGN_K + j]);
      Rpv = fq_mul(Y[SIGN_K + j], Z[SIGN_K + j]);
    }
    if (!SIGN) {
      if (active) {
        stg_point(a.out[0], i, Ru, Rv);
        if (DOUBLE) stg_point(a.out[1], i, Rpu, Rpv);
      }
      continue;
    }
    uint32_t sk[8], nonce[8], u[8], c[8];
    ldg_scalar(a.in[0] + i * 8, sk);
    ldg_scalar(a.in[2] + i * 8, nonce);
    fq m;
    bool valid = true;
    if (OP == OP_SIGN_BYTES) {  // the three from_bytes of the tuple; an invalid tuple gets an all-zero signature and its bit set
      uint32_t mb[8], skb[8], nb[8];
      ldg_scalar(a.in[1] + i * 8, mb);
#pragma unroll
      for (int w = 0; w < 8; w++) { skb[w] = sk[w]; nb[w] = nonce[w]; }
      valid = sign_inputs_from_bytes(skb, nb, mb, sk, nonce, m);
    } else {
      m = ldg_fq(a.in[1] + i * 8);
    }
    if (DOUBLE) chal5(Ru, Rv, Rpu, Rpv, m, c); else chal3(Ru, Rv, m, c);
    sign_finish(nonce, c, sk, u);
    if (OP == OP_SIGN_BYTES) {
      const unsigned inv = __ballot_sync(0xffffffffu, !valid && active);
      if ((threadIdx.x & 31) == 0 && active && a.bitmap) a.bitmap[i >> 5] = inv;
    }
    if (!active) continue;
    if (OP == OP_SIGN_BYTES) {
      uint32_t rb[8];
      point_compress(Ru, Rv, rb);
#pragma unroll
      for (int w = 0; w < 8; w++) { u[w] = valid ? u[w] : 0u; rb[w] = valid ? rb[w] : 0u; }
      stg8(a.out[0] + i * 16, u);
      stg8(a.out[0] + i * 16 + 8, rb);
    } else {
      stg8(a.out[0] + i * 8, u);
      stg_point(a.out[1], i, Ru, Rv);
      if (DOUBLE) stg_point(a.out[2], i, Rpu, Rpv);
      if (a.out[3]) stg8(a.out[3] + i * 8, c);
    }
  }
}

__global__ void __launch_bounds__(TPB) k_comb4_build(uint32_t* table, const fq bu, const fq bv) {
  int t = blockIdx.x * TPB + threadIdx.x;
  if (t >= CT_WINDOWS * CT_ENTRIES) return;
  comb4_build_entry(bu, bv, t / CT_ENTRIES, t % CT_ENTRIES + 1, table + (size_t)t * 24);
}
__global__ void __launch_bounds__(TPB) k_comb_build(uint32_t* table, const fq bu, const fq bv) {
  int t = blockIdx.x * TPB + threadIdx.x;
  if (t >= COMB_WINDOWS * COMB_ENTRIES) return;  // 524 304 entries at 16-bit windows
  comb_build_entry(bu, bv, t / COMB_ENTRIES, t % COMB_ENTRIES, table + (size_t)t * 24);
}

// Verification against a keyset (include/schnorr_b200_keyset.h).  aux = scheme; in: key index, u, R, (R',) m -> bitmap,
// out0 (nullable): c
__global__ void __launch_bounds__(TPB, SB_MIN_CTAS) k_verify_keyset(const KArgs a, const KsArgs ks) {
  int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  const bool active = i < a.n;
  if (!active) i = a.n - 1;  // idle lanes redo the last tuple so the warp stays converged
  const bool aff = (a.flags & SB200_POINTS_AFFINE) != 0, chk = (a.flags & SB200_CHECK_POINTS) != 0;
  const uint32_t key = __ldg(a.in[0] + i);
  uint32_t u[8], c[8];
  ldg_scalar(a.in[1] + i * 8, u);
  bool ok;
  if (a.aux == 0)
    ok = verify_keyset_core<0>(ks.tab, ks.n, ks.ok, key, u, ldg_point(a.in[2], i, aff), point_in(), ldg_fq(a.in[3] + i * 8), chk,
                               a.combG, a.combGp, c);
  else if (a.aux == 1)
    ok = verify_keyset_core<1>(ks.tab, ks.n, ks.ok, key, u, ldg_point(a.in[2], i, aff), ldg_point(a.in[3], i, aff),
                               ldg_fq(a.in[4] + i * 8), chk, a.combG, a.combGp, c);
  else
    ok = verify_keyset_core<2>(ks.tab, ks.n, ks.ok, key, u, ldg_point(a.in[2], i, aff), point_in(), ldg_fq(a.in[3] + i * 8), chk,
                               a.combG, a.combGp, c);
  unsigned word = __ballot_sync(0xffffffffu, ok && active);
  if ((threadIdx.x & 31) == 0 && active) a.bitmap[i >> 5] = word;
  if (a.out[0] && active) stg8(a.out[0] + i * 8, c);
}

// Per-key combs of a keyset (include/schnorr_b200_keyset.h): one warp per key of [key0, key0 + nk), one lane per window
// (keyset_build_window), the key's NT points one after the other, then its key_ok bit.  Lane-divergent doubling counts
// (8 j for window j): a one-off build, not a hot path.  scratch: 2 x (KS_ENTRIES - 1) fq per thread of the launch.
constexpr int64_t KS_BUILD_KEYS = 2048;  // keys per build launch: 536 MB of scratch
struct KsBuild {
  uint32_t* tab;
  uint32_t* ok;
  const uint32_t* pk;
  const uint32_t* pk2;
  int64_t key0, nk;
  int nt;
  bool aff;
  fq* scratch;
};
__global__ void __launch_bounds__(TPB) k_keyset_build(const KsBuild b) {
  static_assert(KS_WINDOWS == 32, "one lane per window");
  const int64_t t = (int64_t)blockIdx.x * TPB + threadIdx.x, w = t >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= b.nk) return;  // warp-uniform
  const int64_t k = b.key0 + w;
  fq* z = b.scratch + (size_t)t * 2 * (KS_ENTRIES - 1);
  bool well = true;
#pragma unroll 1
  for (int p = 0; p < b.nt; p++) {
    const point_in P = ldg_point(p ? b.pk2 : b.pk, k, b.aff);
    well &= point_well_formed(P);
    keyset_build_window(point_to_ext(P), lane, b.tab + ((size_t)k * b.nt + p) * KS_TABLE_WORDS + (size_t)lane * KS_ENTRIES * 24, z,
                        z + (KS_ENTRIES - 1));
  }
  if (lane == 0 && well) atomicOr(b.ok + (k >> 5), 1u << (k & 31));
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct Stage {  // pinned staging buffer for pageable host memory
  uint8_t* p = nullptr;
  size_t cap = 0;
};
struct PendingCopy {  // results sitting in a pinned out-stage until their D2H has landed
  uint8_t* dst;
  const uint8_t* src;
  size_t bytes;
};
struct DevCtx {
  int dev = 0;
  cudaStream_t stream[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};  // end of the work enqueued for a pipeline slot
  uint32_t* combG = nullptr;
  uint32_t* combGp = nullptr;
  uint32_t* comb4 = nullptr;  // [G | G'] 4-bit combs of the oblivious path (2 x 48 KB)
  uint8_t* arena[2] = {nullptr, nullptr};
  size_t arena_cap[2] = {0, 0};
  Stage hin[2], hout[2];
  std::vector<PendingCopy> pending[2];
  WsState* ws[3] = {nullptr, nullptr, nullptr};  // per pipeline stream, [2] = caller's stream (SB200_DEVICE_PTRS)
  pniels* ec_scratch[3] = {nullptr, nullptr, nullptr};  // k_curve_p window tables (SB_EC_GLOBAL_TABLES)
  uint32_t* cscratch = nullptr;                  // device-only rows of a SB200_DEVICE_PTRS call (scratch_bytes)
  size_t cscratch_cap = 0;
  cudaEvent_t user_ev = nullptr;                 // last SB200_DEVICE_PTRS work of this context (orders a stream switch)
  cudaStream_t last_user_stream = nullptr;
  bool user_ev_valid = false;
  bool registered = false;                       // holds a reference on this device's constant-memory parameters
  int nsm = 0;
};

struct Desc {
  Op op;
  uint32_t flags;
  int aux = 0;
  int nin = 0, nout = 0;
  const uint32_t* in[MAX_IN] = {};
  int in_words[MAX_IN] = {};
  uint32_t* out[MAX_OUT] = {};
  int out_words[MAX_OUT] = {};
  uint32_t* bitmap = nullptr;
  const sb200_stdrng* rng = nullptr;  // OP_STDRNG and the seeded signers: key and word position of tuple 0
  const sb200_keyset* ks = nullptr;   // OP_VERIFY_KEYSET: whose per-device tables the kernels read
  unsigned need = 0;  // outputs that may not be null: bit k for out[k], bit MAX_OUT for the bitmap
};

// Hades tables live in each device's constant memory: one parameter set per process and device.
struct DevParams {
  uint64_t hash = 0;
  int refs = 0;
};
std::mutex g_params_mu;
std::map<int, DevParams> g_dev_params;

uint64_t fnv1a(const void* p, size_t n) {
  const uint8_t* b = (const uint8_t*)p;
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}

struct DeviceGuard {  // the caller's current device is restored when a call returns
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

struct sb200_ctx {
  std::vector<DevCtx> devs;
  std::mutex mu, err_mu;
  std::string err;
  cudaStream_t user_stream = nullptr;
  std::atomic<uint64_t> launches{0};
  sb200_params params;
  HadesTables tables;
  int persist = 0;  // environment variable SB200_CURVE_PERSISTENT at context creation: "always" | "never" | unset (by batch size)
  std::vector<sb200_keyset*> keysets;  // alive keysets of this context (sb200_destroy frees them)
  void set_err(const std::string& e) {
    std::lock_guard<std::mutex> l(err_mu);
    if (err.empty() || e.empty()) err = e;
  }
};

struct sb200_keyset {
  struct Dev {
    uint32_t* tab = nullptr;  // n_keys x (scheme == 0 ? 1 : 2) x KS_TABLE_WORDS
    uint32_t* ok = nullptr;   // key_ok bitmap
  };
  sb200_ctx* ctx;
  int scheme;
  int64_t n_keys;
  std::vector<Dev> dev;  // one copy per device of ctx, in ctx->devs order
};

namespace {

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      ctx->set_err(std::string(#call) + ": " + cudaGetErrorString(_e));                       \
      return SB200_ERR_CUDA;                                                                  \
    }                                                                                         \
  } while (0)

// ---- what the library knows about each operation: one row per Op, in Op order ------------------------------------------
// How an op launches.  INTERNAL: a stage of other ops, never called by itself.  ONE: `kernel`, one tuple per thread.
// FIXED: the k_fixed_batch `kernel` (or its SB200_SIGN_OBLIVIOUS form `ct`), fixed_k(op) tuples per thread.  VERIFY:
// challenge kernel, then curve kernel, the challenges through c_out or scratch.  VERIFY_BYTES: decode kernel, then VERIFY
// on the decoded rows.  SIGN_STDRNG: the nonces drawn into scratch, then the scheme's sign op.  DBG_VERIFY_EC: the curve
// kernel alone, on the caller's challenges.  WITNESS_BYTES: decode kernel, then `kernel` on the decoded rows.  KEYSET:
// k_verify_keyset, one tuple per thread, with the keyset's tables of the launching device.
enum Form : uint8_t { INTERNAL, ONE, FIXED, VERIFY, VERIFY_BYTES, SIGN_STDRNG, DBG_VERIFY_EC, WITNESS_BYTES, KEYSET };
using KFn = void (*)(KArgs);
struct OpInfo {
  Form form;
  uint32_t flags;       // the SB200_* flags the op accepts: any other one is SB200_ERR_ARG
  int scheme;           // VERIFY*, SIGN_STDRNG, FIXED: 0 single-key, 1 double-key (two combs), 2 variable generator
  KFn kernel, ct;
  size_t ct_smem;       // shared memory of `ct`: one or two 4-bit combs
  uint32_t forced;      // flags the op always runs with: the byte-level verifications hand affine points between kernels
  unsigned scratch;     // device-only bytes per tuple between the kernels of one call, in `scratch_arrays` arrays: the
  int scratch_arrays;   // challenges or nonces, and the decoded rows (points 64 B, u and m 32 B) and invalid bitmap
};
constexpr OpInfo row(Form form, uint32_t flags = 0, int scheme = 0, KFn kernel = nullptr, KFn ct = nullptr) {
  const bool decode = form == VERIFY_BYTES || form == WITNESS_BYTES;
  const unsigned points = scheme == 0 ? 2 : scheme == 1 ? 4 : 3, rows = decode ? 64 * points + 64 : 0;
  const bool handover = form == VERIFY || form == VERIFY_BYTES || form == SIGN_STDRNG;  // + 32 B: the challenge row
  return {form, flags, scheme, kernel, ct, ct ? (size_t)(scheme == 1 ? 2 : 1) * CT_TABLE_WORDS * 4 : 0,
          decode ? (uint32_t)SB200_POINTS_AFFINE : 0u, (handover ? 32u : 0u) + rows,
          (handover ? 1 : 0) + (rows ? (int)points + 3 : 0)};
}
constexpr uint32_t D = SB200_DEVICE_PTRS, AD = SB200_POINTS_AFFINE | D, CHK = AD | SB200_CHECK_POINTS;
constexpr uint32_t OBL = AD | SB200_SIGN_OBLIVIOUS, DUAL = SB_VERIFY_WS ? SB200_VERIFY_DUAL_PIPE : 0;
constexpr OpInfo OPS[] = {
#if SB_VERIFY_SPLIT
    row(VERIFY, CHK | DUAL, 0),  // OP_VERIFY
    row(VERIFY, CHK, 1),         // OP_VERIFY_DOUBLE
#else  // the fused one-launch verification kernels are only built when the split form is switched off
    row(ONE, CHK | DUAL, 0, k_run<OP_VERIFY>),
    row(ONE, CHK, 1, k_run<OP_VERIFY_DOUBLE>),
#endif
#if SB_VERIFY_SPLIT && SB_VARGEN_SPLIT
    row(VERIFY, CHK, 2),  // OP_VERIFY_VARGEN
#else
    row(ONE, CHK, 2, k_run<OP_VERIFY_VARGEN>),
#endif
    row(FIXED, OBL, 0, k_fixed_batch<OP_SIGN>, k_fixed_batch<OP_SIGN, true>),
    row(FIXED, OBL, 1, k_fixed_batch<OP_SIGN_DOUBLE>, k_fixed_batch<OP_SIGN_DOUBLE, true>),
    row(ONE, OBL, 0, k_run<OP_SIGN_VARGEN>),
    row(FIXED, OBL, 0, k_fixed_batch<OP_KEYGEN>, k_fixed_batch<OP_KEYGEN, true>),
    row(FIXED, OBL, 1, k_fixed_batch<OP_KEYGEN_DOUBLE>, k_fixed_batch<OP_KEYGEN_DOUBLE, true>),
    row(ONE, OBL, 0, k_run<OP_KEYGEN_VARGEN>),
    row(ONE, D, 0, k_run<OP_DBG_FQ>),
    row(ONE, AD, 0, k_run<OP_DBG_FR_MUL>),
    row(ONE, AD, 0, k_run<OP_DBG_HADES>),
    row(ONE, AD, 0, k_run<OP_DBG_SMUL>),
    row(ONE, D, 0, k_run<OP_DECOMPRESS>),
    row(ONE, AD, 0, k_run<OP_COMPRESS>),
    row(ONE, D, 0, k_run<OP_FROM_WIDE>),
    row(VERIFY_BYTES, D, 0),  // OP_VERIFY_BYTES
    row(FIXED, D, 0, k_fixed_batch<OP_SIGN_BYTES>),
    row(INTERNAL),  // OP_CHALLENGE
    row(INTERNAL),  // OP_VERIFY_EC
    row(VERIFY_BYTES, D, 1),  // OP_VERIFY_DOUBLE_BYTES
    row(VERIFY_BYTES, D, 2),  // OP_VERIFY_VARGEN_BYTES
    row(ONE, D, 0, k_run<OP_SIGN_DOUBLE_BYTES>),
    row(ONE, D, 0, k_run<OP_SIGN_VARGEN_BYTES>),
    row(INTERNAL),  // OP_CHALLENGE_DOUBLE
    row(INTERNAL),  // OP_VERIFY_DOUBLE_EC
    row(INTERNAL),  // OP_CHALLENGE_VARGEN
    row(INTERNAL),  // OP_VERIFY_VARGEN_EC
    row(ONE, AD, 0, k_run<OP_POINTS_CHECK>),
    row(DBG_VERIFY_EC, AD, 0),  // OP_DBG_VERIFY_EC
    row(INTERNAL),  // OP_DECODE_VERIFY
    row(ONE, AD, 0, k_run<OP_WITNESS>),
    row(ONE, AD, 0, k_run<OP_DBG_LAT3>),
    row(ONE, D, 0, k_run<OP_STDRNG>),
    row(SIGN_STDRNG, D | SB200_SIGN_OBLIVIOUS, 0),  // OP_SIGN_STDRNG
    row(SIGN_STDRNG, D | SB200_SIGN_OBLIVIOUS, 1),  // OP_SIGN_DOUBLE_STDRNG
    row(SIGN_STDRNG, OBL, 2),                       // OP_SIGN_VARGEN_STDRNG
    row(ONE, CHK, 0, k_run<OP_VERIFY_WITNESS>),     // the scheme is the call's aux
    row(WITNESS_BYTES, D, 1, k_run<OP_VERIFY_WITNESS>),  // scheme 1: scratch for the widest decoded rows; the call's scheme is its aux
    row(KEYSET, CHK),                               // OP_VERIFY_KEYSET: the keyset's scheme is the call's aux
};
static_assert(sizeof(OPS) / sizeof(OPS[0]) == OP_VERIFY_KEYSET + 1, "one row per Op");

// ---- launches ---------------------------------------------------------------------------------------------------------
struct Launcher {  // issues kernels on one stream and counts them (sb200_launch_count)
  sb200_ctx* ctx;
  cudaStream_t st;
  template <class... P, class... A>
  void operator()(void (*k)(P...), unsigned grid, unsigned block, size_t smem, const A&... args) const {
    k<<<grid, block, smem, st>>>(args...);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
  }
};

// The curve half of a verification.  With SB_EC_GLOBAL_TABLES a batch above one wave of resident CTAs runs the persistent
// form, which takes its tuples from the counter a.ws->tile: the challenge kernel before it resets the counter, without one
// (reset_tile) it is cleared here.  A batch that fits one wave gains nothing from the persistent form (no slot is reused,
// the scratch region is cold in L2): it runs the local-memory kernel (measured at 2^16 tuples: 16.4 vs 15.0 M verifies/s).
int launch_curve(const Launcher& go, int scheme, const KArgs& a, unsigned grid, bool reset_tile = false) {
  static const KFn one_shot[3] = {k_run<OP_VERIFY_EC>, k_run<OP_VERIFY_DOUBLE_EC>, k_run<OP_VERIFY_VARGEN_EC>};
#if SB_EC_GLOBAL_TABLES
  static void (*const persistent[3])(KArgs, pniels*) = {k_curve_p<0>, k_curve_p<1>, k_curve_p<2>};
  sb200_ctx* ctx = go.ctx;
  if (reset_tile) CU(cudaMemsetAsync(&a.ws->tile, 0, sizeof(unsigned), go.st));
  const unsigned wave = (unsigned)(ec_p_ctas(scheme) * a.nsm);
  if (a.persist == 1 || (a.persist == 0 && grid > wave)) {
    go(persistent[scheme], std::min(grid, wave), TPB, ec_p_smem(scheme), a, a.ec_scratch);
    return SB200_OK;
  }
#endif
  go(one_shot[scheme], grid, TPB, 0, a);
  return SB200_OK;
}

int launch_verify(const Launcher& go, int scheme, const KArgs& a, unsigned grid) {  // a.out[0]: where the challenges go
  static const KFn challenge[3] = {k_run<OP_CHALLENGE>, k_run<OP_CHALLENGE_DOUBLE>, k_run<OP_CHALLENGE_VARGEN>};
  go(challenge[scheme], grid, TPB, 0, a);
  return launch_curve(go, scheme, a, grid);
}

int launch(sb200_ctx* ctx, Op op, const KArgs& a, cudaStream_t st, const KsArgs& ks = KsArgs()) {
  if (a.n <= 0) return SB200_OK;
  const OpInfo& o = OPS[op];
  const Launcher go{ctx, st};
  const unsigned grid = (unsigned)((a.n + TPB - 1) / TPB);
  int rc = SB200_OK;
#if SB_VERIFY_WS
  if (op == OP_VERIFY && (a.flags & SB200_VERIFY_DUAL_PIPE)) {  // persistent warp-specialised kernel, one CTA per SM
    CU(cudaMemsetAsync(&a.ws->tile, 0, sizeof(unsigned), st));
    go(k_verify_ws, std::min<unsigned>((unsigned)((a.n + WS_TILE - 1) / WS_TILE), (unsigned)a.nsm), WS_THREADS, WS_SMEM, a);
    CU(cudaGetLastError());
    return SB200_OK;
  }
#endif
  switch (o.form) {
    case ONE:
    case FIXED: {
      const bool ct = o.ct && (a.flags & SB200_SIGN_OBLIVIOUS);
      const int64_t per_cta = TPB * (o.form == FIXED ? fixed_k(op) : 1);
      go(ct ? o.ct : o.kernel, (unsigned)((a.n + per_cta - 1) / per_cta), TPB, ct ? o.ct_smem : 0, a);
      break;
    }
    case VERIFY:  // a.out[0] is always set here: the caller's c_out or scratch
      rc = launch_verify(go, o.scheme, a, grid);
      break;
    case VERIFY_BYTES:      // decode kernel -> challenge kernel -> curve kernel, the decoded rows and the challenges in a.scratch
    case WITNESS_BYTES: {   // decode kernel -> o.kernel (rows to out[0], `invalid` in out[1]), the decoded rows in a.scratch
      const bool wit = o.form == WITNESS_BYTES;
      const int scheme = wit ? a.aux : o.scheme;
      const int npk = scheme == 0 ? 1 : 2, nr = scheme == 1 ? 2 : 1, narr = npk + 1 + nr + 1;
      uint8_t* p = a.scratch;
      auto carve = [&](size_t bytes) { uint8_t* r = p; p += (bytes + 63) & ~(size_t)63; return (uint32_t*)r; };
      KArgs dk = a, v = a;
      dk.aux = scheme;
      if (!wit) v.out[0] = carve((size_t)a.n * 32);
      for (int k = 0; k < narr; k++) {
        const bool is_scalar = (k == npk) || (k == narr - 1);  // u and m are 8 words, points 16
        dk.dec[k] = carve((size_t)a.n * (is_scalar ? 32 : 64));
        v.in[k] = dk.dec[k];
      }
      uint32_t* invalid = a.out[wit ? 1 : 0];
      dk.bitmap = invalid ? invalid : carve((size_t)((a.n + 31) / 32) * 4);  // the caller's `invalid` or scratch
      v.inv_mask = dk.bitmap;
      for (int k = 1; k < MAX_OUT; k++) v.out[k] = nullptr;
      go(k_run<OP_DECODE_VERIFY>, grid, TPB, 0, dk);
      if (wit) go(o.kernel, grid, TPB, 0, v);
      else rc = launch_verify(go, o.scheme, v, grid);
      break;
    }
    case KEYSET:
      go(k_verify_keyset, grid, TPB, 0, a, ks);
      break;
    case DBG_VERIFY_EC: {  // in: pk, u, R, c -> bitmap: the production curve kernel, in the form the batch size picks,
                           // fed the caller's challenges where the challenge kernel would have written them
      KArgs v = a;
      v.out[0] = const_cast<uint32_t*>(a.in[3]);
      v.in[3] = nullptr;
      rc = launch_curve(go, 0, v, grid, true);
      break;
    }
    case SIGN_STDRNG: {  // the chunk's nonces into a.scratch, then the unchanged sign kernel reads them from there as its nonce input
      KArgs g{};
      g.n = a.n;
      g.out[0] = (uint32_t*)a.scratch;
      memcpy(g.rng_key, a.rng_key, sizeof(g.rng_key));
      g.rng_word = a.rng_word;
      go(k_run<OP_STDRNG>, grid, TPB, 0, g);
      CU(cudaGetLastError());  // no signature from a failed draw: the scratch row would still hold an earlier call's nonces
      KArgs s = a;
      memset(s.rng_key, 0, sizeof(s.rng_key));
      s.in[o.scheme == 2 ? 3 : 2] = (const uint32_t*)a.scratch;
      static const Op sign_op[3] = {OP_SIGN, OP_SIGN_DOUBLE, OP_SIGN_VARGEN};
      return launch(ctx, sign_op[o.scheme], s, st);
    }
    default:
      return SB200_ERR_ARG;
  }
  if (rc) return rc;
  CU(cudaGetLastError());
  return SB200_OK;
}

bool splits_with_scratch(const Desc& d) {  // hash and curve kernels hand c over in memory
  return OPS[d.op].form == VERIFY && !(d.flags & SB200_VERIFY_DUAL_PIPE) && !d.out[0];
}

// device-only bytes between the kernels of one call over n tuples
size_t scratch_bytes(const Desc& d, int64_t n) {
  const OpInfo& o = OPS[d.op];
  if (!o.scratch || (o.form == VERIFY && !splits_with_scratch(d))) return 0;
  return (size_t)n * o.scratch + (size_t)((n + 31) / 32) * 4 + 64 * (o.scratch_arrays + 1);
}

// the kernel arguments every launch of a call shares; `first`: index of the launch's tuple 0 in the call
KArgs kargs(const sb200_ctx* ctx, const DevCtx& dc, int slot, const Desc& d, int64_t n, int64_t first) {
  KArgs a{};
  a.n = n; a.flags = d.flags; a.aux = d.aux; a.combG = dc.combG; a.combGp = dc.combGp;
  a.comb4G = dc.comb4; a.comb4Gp = dc.comb4 + CT_TABLE_WORDS;
  a.ws = dc.ws[slot]; a.nsm = dc.nsm; a.ec_scratch = dc.ec_scratch[slot]; a.persist = ctx->persist;
  if (d.rng) {  // draw i belongs to tuple i: tuple `first` is that many draws into the stream
    memcpy(a.rng_key, d.rng->key, sizeof(a.rng_key));
    a.rng_word = d.rng->word_pos + 16u * (uint64_t)first;
  }
  return a;
}
// the keyset tables of one device's copy (OP_VERIFY_KEYSET), none for every other op
KsArgs ks_args(const sb200_ctx* ctx, const DevCtx& dc, const Desc& d) {
  KsArgs k;
  if (d.ks) {
    const sb200_keyset::Dev& kd = d.ks->dev[&dc - ctx->devs.data()];
    k.tab = kd.tab; k.n = d.ks->n_keys; k.ok = kd.ok;
  }
  return k;
}

bool host_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

int grow_stage(sb200_ctx* ctx, Stage& s, size_t need) {
  if (s.cap >= need) return SB200_OK;
  if (s.p) cudaFreeHost(s.p);
  s.p = nullptr; s.cap = 0;
  if (cudaHostAlloc((void**)&s.p, need, cudaHostAllocPortable) != cudaSuccess) { ctx->set_err("cudaHostAlloc staging"); return SB200_ERR_NOMEM; }
  s.cap = need;
  return SB200_OK;
}

// wait for a pipeline slot's work and move its staged results to the caller's (pageable) buffers
int drain_slot(sb200_ctx* ctx, DevCtx& dc, int slot) {
  if (dc.pending[slot].empty()) return SB200_OK;
  CU(cudaEventSynchronize(dc.done[slot]));
  for (auto& c : dc.pending[slot]) memcpy(c.dst, c.src, c.bytes);
  dc.pending[slot].clear();
  return SB200_OK;
}

// One device's share [lo, hi) of a host-buffer call: chunks alternate between two streams (H2D / kernels / D2H of
// consecutive chunks overlap); pageable host arrays go through the slot's pinned stage.
int run_device(sb200_ctx* ctx, DevCtx& dc, const Desc& d, int64_t lo, int64_t hi, size_t per_tuple,
               const bool* in_pinned, const bool* out_pinned, bool bm_pinned) {
  CU(cudaSetDevice(dc.dev));
  const int64_t share = hi - lo;
  int64_t chunk = CHUNK;
  if (share < 4 * CHUNK) chunk = std::max<int64_t>(CHUNK_MIN, (((share + 3) / 4) + 31) & ~(int64_t)31);
  size_t in_stage = 0, out_stage = 0;  // staging bytes per tuple
  for (int k = 0; k < d.nin; k++) if (d.in_words[k] && !in_pinned[k]) in_stage += (size_t)d.in_words[k] * 4;
  for (int k = 0; k < d.nout; k++) if (d.out[k] && d.out_words[k] > 0 && !out_pinned[k]) out_stage += (size_t)d.out_words[k] * 4;
  int slot = 0;
  for (int64_t c0 = lo; c0 < hi; c0 += chunk, slot ^= 1) {
    const int64_t cn = std::min<int64_t>(chunk, hi - c0);
    const size_t bm_bytes = (size_t)((cn + 31) / 32) * 4;
    int rc = drain_slot(ctx, dc, slot);  // also frees the slot's stages
    if (rc) return rc;
    if (in_stage) CU(cudaEventSynchronize(dc.done[slot]));  // the in-stage may still be read by the slot's previous H2D
    const size_t scr = scratch_bytes(d, cn);
    size_t need = (size_t)cn * per_tuple + scr + bm_bytes * (1 + MAX_OUT) + 64 * (MAX_IN + MAX_OUT + 2);
    if (dc.arena_cap[slot] < need) {
      CU(cudaStreamSynchronize(dc.stream[slot]));
      if (dc.arena[slot]) CU(cudaFree(dc.arena[slot]));
      dc.arena[slot] = nullptr; dc.arena_cap[slot] = 0;
      const int64_t full = std::min<int64_t>(chunk, share);
      size_t cap = std::max(need, (size_t)full * per_tuple + scratch_bytes(d, full) + (1 << 20));
      if (cudaMalloc(&dc.arena[slot], cap) != cudaSuccess) { ctx->set_err("cudaMalloc arena"); return SB200_ERR_NOMEM; }
      dc.arena_cap[slot] = cap;
    }
    if (in_stage && (rc = grow_stage(ctx, dc.hin[slot], (size_t)chunk * in_stage + 64 * MAX_IN))) return rc;
    if ((out_stage || !bm_pinned) && (rc = grow_stage(ctx, dc.hout[slot], (size_t)chunk * out_stage + ((size_t)(chunk + 31) / 32 * 4 + 64) * (MAX_OUT + 1)))) return rc;
    cudaStream_t st = dc.stream[slot];
    uint8_t *p = dc.arena[slot], *hi_p = dc.hin[slot].p, *ho_p = dc.hout[slot].p;
    auto carve = [](uint8_t*& q, size_t bytes) { uint8_t* r = q; q += (bytes + 63) & ~(size_t)63; return r; };
    KArgs a = kargs(ctx, dc, slot, d, cn, c0);
    for (int k = 0; k < d.nin; k++) {
      if (!d.in_words[k]) continue;
      size_t bytes = (size_t)cn * d.in_words[k] * 4;
      uint32_t* dp = (uint32_t*)carve(p, bytes);
      const uint8_t* src = (const uint8_t*)(d.in[k] + (size_t)c0 * d.in_words[k]);
      if (!in_pinned[k]) {
        uint8_t* sp = carve(hi_p, bytes);
        memcpy(sp, src, bytes);
        src = sp;
      }
      CU(cudaMemcpyAsync(dp, src, bytes, cudaMemcpyHostToDevice, st));
      a.in[k] = dp;
    }
    uint32_t* dout[MAX_OUT] = {};
    auto out_bytes = [&](int k) {  // out_words == -1: bitmap-shaped output (one word per 32 tuples)
      return d.out_words[k] < 0 ? bm_bytes : (size_t)cn * d.out_words[k] * 4;
    };
    for (int k = 0; k < d.nout; k++)
      if (d.out[k]) a.out[k] = dout[k] = (uint32_t*)carve(p, out_bytes(k));
    if (scr) {
      a.scratch = carve(p, scr);
      if (splits_with_scratch(d)) a.out[0] = (uint32_t*)a.scratch;
    }
    uint32_t* dbm = nullptr;
    if (d.bitmap) a.bitmap = dbm = (uint32_t*)carve(p, bm_bytes);
    if ((rc = launch(ctx, d.op, a, st, ks_args(ctx, dc, d)))) return rc;
    auto d2h = [&](uint32_t* host_dst, const uint32_t* dev_src, size_t bytes, bool pinned) -> int {
      uint8_t* dst = (uint8_t*)host_dst;
      if (!pinned) {
        uint8_t* sp = carve(ho_p, bytes);
        dc.pending[slot].push_back({dst, sp, bytes});
        dst = sp;
      }
      CU(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToHost, st));
      return SB200_OK;
    };
    for (int k = 0; k < d.nout; k++)
      if (d.out[k] && (rc = d2h(d.out_words[k] < 0 ? d.out[k] + c0 / 32 : d.out[k] + (size_t)c0 * d.out_words[k], dout[k],
                                out_bytes(k), d.out_words[k] < 0 ? bm_pinned : out_pinned[k])))
        return rc;
    if (d.bitmap && (rc = d2h(d.bitmap + c0 / 32, dbm, bm_bytes, bm_pinned))) return rc;
    CU(cudaEventRecord(dc.done[slot], st));
  }
  for (int s = 0; s < 2; s++) {
    int rc = drain_slot(ctx, dc, s);
    if (rc) return rc;
    CU(cudaStreamSynchronize(dc.stream[s]));
  }
  return SB200_OK;
}

// after a failure nothing may still be reading or writing the caller's buffers when the call returns
void quiesce(DevCtx& dc) {
  cudaSetDevice(dc.dev);
  for (int s = 0; s < 2; s++) {
    if (dc.stream[s]) cudaStreamSynchronize(dc.stream[s]);
    dc.pending[s].clear();
  }
  cudaGetLastError();
}

int run(sb200_ctx* ctx, int64_t n, Desc d) {
  if (!ctx || n < 0 || (d.flags & ~OPS[d.op].flags)) return SB200_ERR_ARG;
  d.flags |= OPS[d.op].forced;
  for (int k = 0; k < d.nin; k++)
    if (d.in_words[k] && (!d.in[k] || ((uintptr_t)d.in[k] & 15))) return SB200_ERR_ARG;
  for (int k = 0; k < d.nout; k++)
    if (d.out[k] ? ((uintptr_t)d.out[k] & 15) : (d.need >> k & 1)) return SB200_ERR_ARG;
  if (!d.bitmap && (d.need >> MAX_OUT & 1)) return SB200_ERR_ARG;
  if (n == 0) return SB200_OK;
  std::lock_guard<std::mutex> lock(ctx->mu);
  ctx->set_err("");
  DeviceGuard guard;

  if (d.flags & SB200_DEVICE_PTRS) {
    if (ctx->devs.size() != 1) return SB200_ERR_ARG;
    DevCtx& dc = ctx->devs[0];
    CU(cudaSetDevice(dc.dev));
    cudaStream_t st = ctx->user_stream;
    // the scratch buffers below are shared by all SB200_DEVICE_PTRS calls of this context: order a stream switch
    if (dc.user_ev_valid && dc.last_user_stream != st) CU(cudaStreamWaitEvent(st, dc.user_ev, 0));
    KArgs a = kargs(ctx, dc, 2, d, n, 0);
    a.bitmap = d.bitmap;
    for (int k = 0; k < d.nin; k++) a.in[k] = d.in[k];
    for (int k = 0; k < d.nout; k++) a.out[k] = d.out[k];
    if (const size_t need = scratch_bytes(d, n)) {
      if (dc.cscratch_cap < need) {  // grows on first use / larger batches only (a cudaMalloc in the call path)
        if (dc.user_ev_valid) CU(cudaEventSynchronize(dc.user_ev));
        if (dc.cscratch) CU(cudaFree(dc.cscratch));
        dc.cscratch = nullptr; dc.cscratch_cap = 0;
        if (cudaMalloc(&dc.cscratch, need) != cudaSuccess) { ctx->set_err("cudaMalloc scratch"); return SB200_ERR_NOMEM; }
        dc.cscratch_cap = need;
      }
      a.scratch = (uint8_t*)dc.cscratch;
      if (splits_with_scratch(d)) a.out[0] = dc.cscratch;
    }
    int rc = launch(ctx, d.op, a, st, ks_args(ctx, dc, d));
    if (rc) return rc;
    CU(cudaEventRecord(dc.user_ev, st));
    dc.user_ev_valid = true;
    dc.last_user_stream = st;
    return SB200_OK;
  }

  // bytes per tuple on the device arena (every array padded to 16 B; bitmap = 4 B per 32 tuples)
  size_t per_tuple = 0;
  bool in_pinned[MAX_IN] = {}, out_pinned[MAX_OUT] = {}, bm_pinned = true;
  for (int k = 0; k < d.nin; k++) {
    per_tuple += (size_t)d.in_words[k] * 4;
    if (d.in_words[k]) in_pinned[k] = host_pinned(d.in[k]);
  }
  for (int k = 0; k < d.nout; k++) {
    per_tuple += (d.out[k] && d.out_words[k] > 0) ? (size_t)d.out_words[k] * 4 : 0;
    if (d.out[k]) out_pinned[k] = host_pinned(d.out[k]);
    if (d.out[k] && d.out_words[k] < 0) bm_pinned = bm_pinned && out_pinned[k];
  }
  if (d.bitmap) bm_pinned = bm_pinned && host_pinned(d.bitmap);

  const int ndev = (int)ctx->devs.size();
  const int64_t per_dev = ((n + ndev - 1) / ndev + 31) & ~(int64_t)31;
  std::vector<int> rcs(ndev, SB200_OK);
  auto work = [&](int di) {
    const int64_t lo = std::min<int64_t>(n, di * per_dev), hi = std::min<int64_t>(n, lo + per_dev);
    if (lo < hi) rcs[di] = run_device(ctx, ctx->devs[di], d, lo, hi, per_tuple, in_pinned, out_pinned, bm_pinned);
  };
  if (ndev == 1) {
    work(0);
  } else {  // one host thread per device: staging copies and (for pageable memory, blocking) transfers run in parallel
    std::vector<std::thread> th;
    for (int di = 1; di < ndev; di++) th.emplace_back(work, di);
    work(0);
    for (auto& t : th) t.join();
  }
  int rc = SB200_OK;
  for (int di = 0; di < ndev; di++)
    if (rcs[di] && !rc) rc = rcs[di];
  if (rc)
    for (auto& dc : ctx->devs) quiesce(dc);
  return rc;
}

int pt_words(uint32_t flags) { return (flags & SB200_POINTS_AFFINE) ? 16 : 24; }

void release_device(DevCtx& dc) {
  cudaSetDevice(dc.dev);
  for (int s = 0; s < 2; s++) {
    if (dc.stream[s]) { cudaStreamSynchronize(dc.stream[s]); cudaStreamDestroy(dc.stream[s]); }
    if (dc.done[s]) cudaEventDestroy(dc.done[s]);
    if (dc.arena[s]) cudaFree(dc.arena[s]);
    if (dc.hin[s].p) cudaFreeHost(dc.hin[s].p);
    if (dc.hout[s].p) cudaFreeHost(dc.hout[s].p);
  }
  if (dc.user_ev) { if (dc.user_ev_valid) cudaEventSynchronize(dc.user_ev); cudaEventDestroy(dc.user_ev); }
  if (dc.combG) cudaFree(dc.combG);
  if (dc.combGp) cudaFree(dc.combGp);
  if (dc.comb4) cudaFree(dc.comb4);
  for (int s = 0; s < 3; s++) {
    if (dc.ws[s]) cudaFree(dc.ws[s]);
    if (dc.ec_scratch[s]) cudaFree(dc.ec_scratch[s]);
  }
  if (dc.cscratch) cudaFree(dc.cscratch);
  if (dc.registered) {
    std::lock_guard<std::mutex> l(g_params_mu);
    auto it = g_dev_params.find(dc.dev);
    if (it != g_dev_params.end() && --it->second.refs <= 0) g_dev_params.erase(it);
  }
  dc = DevCtx();
}

// a keyset's device memory on every device of its context (work of earlier SB200_DEVICE_PTRS calls may still read it)
void keyset_free(sb200_keyset* ks) {
  for (size_t di = 0; di < ks->dev.size(); di++) {
    DevCtx& dc = ks->ctx->devs[di];
    cudaSetDevice(dc.dev);
    if (dc.user_ev_valid) cudaEventSynchronize(dc.user_ev);
    if (ks->dev[di].tab) cudaFree(ks->dev[di].tab);
    if (ks->dev[di].ok) cudaFree(ks->dev[di].ok);
  }
  delete ks;
}

// parameters -> validated, derived, self-checked tables.  Host only.
int prepare_params(const sb200_params* p, HadesTables& T) {
  if (!p || p->struct_size != sizeof(sb200_params) || p->reserved != 0) return SB200_ERR_ARG;
  const uint32_t* all = p->generator;
  const size_t nfe = (sizeof(sb200_params) - 8) / 32;
  for (size_t i = 0; i < nfe; i++)
    if (!params::canonical_fq(all + 8 * i)) return SB200_ERR_PARAMS;
  const fq gu = params::ld(p->generator), gv = params::ld(p->generator + 8);
  const fq hu = params::ld(p->generator_nums), hv = params::ld(p->generator_nums + 8);
  if (!params::on_curve(gu, gv) || !params::on_curve(hu, hv)) return SB200_ERR_PARAMS;
  if (!params::prime_order(gu, gv) || !params::prime_order(hu, hv)) return SB200_ERR_PARAMS;
  if (!params::derive_hades_tables(p->round_constants, p->mds, T)) return SB200_ERR_PARAMS;
  // self-check: the production form (small-integer layers or sparse rounds) must reproduce the reference-shaped dense
  // permutation (host build of the same code)
  h_hades = T;
  uint64_t s = 0x9e3779b97f4a7c15ull;
  for (int trial = 0; trial < 3; trial++) {
    fq a[5], b[5];
    for (int k = 0; k < 5; k++) {
      for (int j = 0; j < 8; j++) { s ^= s << 13; s ^= s >> 7; s ^= s << 17; a[k].v[j] = trial ? (uint32_t)s : 0u; }
      a[k].v[7] &= 0x3fffffffu;
      b[k] = a[k];
    }
    hades_perm_dense(a);
    hades_perm(b);
    for (int k = 0; k < 5; k++)
      if (!fq_eq(a[k], b[k])) return SB200_ERR_PARAMS;
  }
  return SB200_OK;
}

}  // namespace

extern "C" {

int sb200_default_params(int ark_rule, sb200_params* out) {
  if (!out) return SB200_ERR_ARG;
  if (ark_rule == SB200_ARK_ENV) {
    const char* e = getenv("SB200_ARK");
    ark_rule = (e && !strcmp(e, "plain")) ? SB200_ARK_PLAIN : SB200_ARK_CUMSUM;
    if (e && strcmp(e, "plain") && strcmp(e, "cumsum") && *e) return SB200_ERR_ARG;
  }
  if (ark_rule != SB200_ARK_CUMSUM && ark_rule != SB200_ARK_PLAIN) return SB200_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->struct_size = sizeof(sb200_params);
  const uint32_t g[4][8] = {SB200_G_U_INIT, SB200_G_V_INIT, SB200_GP_U_INIT, SB200_GP_V_INIT};
  memcpy(out->generator, g[0], 32); memcpy(out->generator + 8, g[1], 32);
  memcpy(out->generator_nums, g[2], 32); memcpy(out->generator_nums + 8, g[3], 32);
  params::default_round_constants(ark_rule, out->round_constants, 335);
  params::default_mds(out->mds);
  return SB200_OK;
}

int sb200_init(const int* devices, int n_devices, sb200_ctx** out) {
  sb200_params p;
  int rc = sb200_default_params(SB200_ARK_ENV, &p);
  if (rc) return rc;
  return sb200_init_ex(&p, devices, n_devices, out);
}

int sb200_init_ex(const sb200_params* params_in, const int* devices, int n_devices, sb200_ctx** out) {
  if (!out || n_devices < 0 || (n_devices > 0 && !devices)) return SB200_ERR_ARG;
  *out = nullptr;
  sb200_ctx* ctx = new sb200_ctx();
  auto fail = [&](int code) { sb200_destroy(ctx); return code; };
  int rc = prepare_params(params_in, ctx->tables);
  if (rc) return fail(rc);
  ctx->params = *params_in;
  if (const char* e = getenv("SB200_CURVE_PERSISTENT")) ctx->persist = !strcmp(e, "always") ? 1 : !strcmp(e, "never") ? 2 : 0;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(SB200_ERR_NODEV);
  DeviceGuard guard;
  int dflt = 0;
  if (n_devices == 0) { devices = &dflt; n_devices = 1; }
  const uint64_t hash = fnv1a(params_in, sizeof(*params_in));
  const fq gu = params::ld(params_in->generator), gv = params::ld(params_in->generator + 8);
  const fq hu = params::ld(params_in->generator_nums), hv = params::ld(params_in->generator_nums + 8);
  ctx->devs.reserve(n_devices);
  for (int i = 0; i < n_devices; i++) {
    if (devices[i] < 0 || devices[i] >= count) return fail(SB200_ERR_ARG);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, devices[i]) != cudaSuccess || prop.major < 10) return fail(SB200_ERR_NODEV);
    ctx->devs.emplace_back();  // owned by the context from here on: sb200_destroy releases whatever got allocated
    DevCtx& dc = ctx->devs.back();
    dc.dev = devices[i];
    if (cudaSetDevice(dc.dev) != cudaSuccess) return fail(SB200_ERR_CUDA);
    {  // this device's constant memory holds one parameter set
      std::lock_guard<std::mutex> l(g_params_mu);
      DevParams& dp = g_dev_params[dc.dev];
      if (dp.refs > 0 && dp.hash != hash) return fail(SB200_ERR_BUSY);
      if (dp.refs == 0 || dp.hash != hash) {
        if (cudaMemcpyToSymbol(d_hades, &ctx->tables, sizeof(HadesTables)) != cudaSuccess) return fail(SB200_ERR_CUDA);
        dp.hash = hash;
      }
      dp.refs++;
      dc.registered = true;
    }
    for (int s = 0; s < 2; s++) {
      if (cudaStreamCreateWithFlags(&dc.stream[s], cudaStreamNonBlocking) != cudaSuccess) return fail(SB200_ERR_CUDA);
      if (cudaEventCreateWithFlags(&dc.done[s], cudaEventDisableTiming) != cudaSuccess) return fail(SB200_ERR_CUDA);
    }
    if (cudaEventCreateWithFlags(&dc.user_ev, cudaEventDisableTiming) != cudaSuccess) return fail(SB200_ERR_CUDA);
    size_t tb = (size_t)COMB_WINDOWS * COMB_ENTRIES * 24 * 4;
    if (cudaMalloc(&dc.combG, tb) != cudaSuccess || cudaMalloc(&dc.combGp, tb) != cudaSuccess) return fail(SB200_ERR_NOMEM);
    if (cudaMalloc(&dc.comb4, (size_t)2 * CT_TABLE_WORDS * 4) != cudaSuccess) return fail(SB200_ERR_NOMEM);
    for (const OpInfo& o : OPS)
      if (o.ct && cudaFuncSetAttribute(o.ct, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)o.ct_smem) != cudaSuccess)
        return fail(SB200_ERR_CUDA);
    dc.nsm = prop.multiProcessorCount;
#if SB_VERIFY_WS
    if (cudaFuncSetAttribute(k_verify_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WS_SMEM) != cudaSuccess) return fail(SB200_ERR_CUDA);
#endif
#if SB_VERIFY_WS || SB_EC_GLOBAL_TABLES
    for (int s = 0; s < 3; s++)
      if (cudaMalloc(&dc.ws[s], sizeof(WsState)) != cudaSuccess || cudaMemset(dc.ws[s], 0, sizeof(WsState)) != cudaSuccess)
        return fail(SB200_ERR_NOMEM);
#endif
#if SB_EC_GLOBAL_TABLES
    for (int s = 0; s < 3; s++)  // 4 x 148 x 128 threads x 27 entries x 128 B = 262 MB per stream
      if (cudaMalloc(&dc.ec_scratch[s], (size_t)(SB_EC_P_CTAS0 > 4 ? SB_EC_P_CTAS0 : 4) * dc.nsm * TPB * EC_P_ENTRIES * sizeof(pniels)) != cudaSuccess) return fail(SB200_ERR_NOMEM);
    if (cudaFuncSetAttribute(k_curve_p<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ec_p_smem(2)) != cudaSuccess) return fail(SB200_ERR_CUDA);
#endif
    int grid = (COMB_WINDOWS * COMB_ENTRIES + TPB - 1) / TPB;
    k_comb_build<<<grid, TPB, 0, dc.stream[0]>>>(dc.combG, gu, gv);
    k_comb_build<<<grid, TPB, 0, dc.stream[0]>>>(dc.combGp, hu, hv);
    k_comb4_build<<<(CT_WINDOWS * CT_ENTRIES + TPB - 1) / TPB, TPB, 0, dc.stream[0]>>>(dc.comb4, gu, gv);
    k_comb4_build<<<(CT_WINDOWS * CT_ENTRIES + TPB - 1) / TPB, TPB, 0, dc.stream[0]>>>(dc.comb4 + CT_TABLE_WORDS, hu, hv);
    ctx->launches += 4;
  }
  for (auto& dc : ctx->devs)  // the table builds of all devices run concurrently
    if (cudaSetDevice(dc.dev) != cudaSuccess || cudaStreamSynchronize(dc.stream[0]) != cudaSuccess) return fail(SB200_ERR_CUDA);
  *out = ctx;
  return SB200_OK;
}

void sb200_destroy(sb200_ctx* ctx) {
  if (!ctx) return;
  {
    DeviceGuard guard;
    for (sb200_keyset* ks : ctx->keysets) keyset_free(ks);
    for (auto& dc : ctx->devs) release_device(dc);
  }
  delete ctx;
}

int sb200_params_check(const sb200_params* params_in, uint32_t* tables_out) {
  HadesTables* T = new HadesTables();
  int rc = prepare_params(params_in, *T);
  if (!rc && tables_out) memcpy(tables_out, T, HADES_ABI_BYTES);
  delete T;
  return rc;
}
int sb200_get_params(const sb200_ctx* ctx, sb200_params* out) {
  if (!ctx || !out) return SB200_ERR_ARG;
  *out = ctx->params;
  return SB200_OK;
}
int sb200_dbg_hades_tables(const sb200_ctx* ctx, uint32_t* out) {
  if (!ctx || !out) return SB200_ERR_ARG;
  memcpy(out, &ctx->tables, HADES_ABI_BYTES);
  return SB200_OK;
}

const char* sb200_strerror(int code) {
  switch (code) {
    case SB200_OK: return "ok";
    case SB200_ERR_ARG: return "invalid argument";
    case SB200_ERR_CUDA: return "CUDA error";
    case SB200_ERR_NODEV: return "no usable sm_100 CUDA device";
    case SB200_ERR_NOMEM: return "out of device memory";
    case SB200_ERR_PARAMS: return "scheme parameters rejected";
    case SB200_ERR_BUSY: return "device already holds different scheme parameters";
    default: return "unknown error";
  }
}
const char* sb200_last_error(const sb200_ctx* ctx) { return ctx ? ctx->err.c_str() : ""; }  // valid until the context's next call
int sb200_device_count(const sb200_ctx* ctx) { return ctx ? (int)ctx->devs.size() : 0; }
int sb200_set_stream(sb200_ctx* ctx, void* s) {
  if (!ctx) return SB200_ERR_ARG;
  ctx->user_stream = (cudaStream_t)s;
  return SB200_OK;
}
uint64_t sb200_launch_count(const sb200_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }
int sb200_host_alloc(size_t bytes, void** out) {
  if (!out) return SB200_ERR_ARG;
  return cudaHostAlloc(out, bytes, cudaHostAllocPortable) == cudaSuccess ? SB200_OK : SB200_ERR_NOMEM;
}
void sb200_host_free(void* p) { if (p) cudaFreeHost(p); }

#define IN(k, ptr, words) d.in[k] = (ptr); d.in_words[k] = (words)
#define OPT_OUT(k, ptr, words) d.out[k] = (ptr); d.out_words[k] = (words)
#define OUT(k, ptr, words) OPT_OUT(k, ptr, words); d.need |= 1u << (k)
#define BITMAP(ptr) d.bitmap = (ptr); d.need |= 1u << MAX_OUT

int sb200_verify(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* sig_u, const uint32_t* sig_R,
                 const uint32_t* msg, uint32_t* verdicts, uint32_t* c_out) {
  Desc d; d.op = OP_VERIFY; d.flags = flags; d.nin = 4; d.nout = 1; BITMAP(verdicts);
  IN(0, pk, pt_words(flags)); IN(1, sig_u, 8); IN(2, sig_R, pt_words(flags)); IN(3, msg, 8); OPT_OUT(0, c_out, 8);
  return run(ctx, n, d);
}
int sb200_verify_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* pkp, const uint32_t* sig_u,
                        const uint32_t* sig_R, const uint32_t* sig_Rp, const uint32_t* msg, uint32_t* verdicts, uint32_t* c_out) {
  Desc d; d.op = OP_VERIFY_DOUBLE; d.flags = flags; d.nin = 6; d.nout = 1; BITMAP(verdicts);
  int pw = pt_words(flags);
  IN(0, pk, pw); IN(1, pkp, pw); IN(2, sig_u, 8); IN(3, sig_R, pw); IN(4, sig_Rp, pw); IN(5, msg, 8); OPT_OUT(0, c_out, 8);
  return run(ctx, n, d);
}
int sb200_verify_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* gen, const uint32_t* sig_u,
                        const uint32_t* sig_R, const uint32_t* msg, uint32_t* verdicts, uint32_t* c_out) {
  Desc d; d.op = OP_VERIFY_VARGEN; d.flags = flags; d.nin = 5; d.nout = 1; BITMAP(verdicts);
  int pw = pt_words(flags);
  IN(0, pk, pw); IN(1, gen, pw); IN(2, sig_u, 8); IN(3, sig_R, pw); IN(4, msg, 8); OPT_OUT(0, c_out, 8);
  return run(ctx, n, d);
}
// the signers of one scheme: sk, (generator,) msg, nonce -> u, R, (R',) c; with `rng` the nonces are drawn on the device
static int sign_call(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* sk, const uint32_t* gen, const uint32_t* msg,
                     const uint32_t* nonce, sb200_stdrng* rng, uint32_t* u_out, uint32_t* R_out, uint32_t* Rp_out, uint32_t* c_out) {
  static const Op ops[2][3] = {{OP_SIGN, OP_SIGN_DOUBLE, OP_SIGN_VARGEN}, {OP_SIGN_STDRNG, OP_SIGN_DOUBLE_STDRNG, OP_SIGN_VARGEN_STDRNG}};
  const int g = scheme == 2;  // the generator comes second
  Desc d; d.op = ops[rng != nullptr][scheme]; d.flags = flags; d.nin = 3 + g; d.nout = 4; d.rng = rng;
  IN(0, sk, 8); IN(1, gen, g ? pt_words(flags) : 0); IN(1 + g, msg, 8); IN(2 + g, nonce, rng ? 0 : 8);
  OUT(0, u_out, 8); OUT(1, R_out, 16); OPT_OUT(3, c_out, 8);
  if (scheme == 1) { OUT(2, Rp_out, 16); }
  const int rc = run(ctx, n, d);
  if (rc == SB200_OK && rng) rng->word_pos += 16u * (uint64_t)n;  // only on success, as `&mut rng` would
  return rc;
}
int sb200_sign(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* msg, const uint32_t* nonce,
               uint32_t* u_out, uint32_t* R_out, uint32_t* c_out) {
  return sign_call(ctx, n, flags, 0, sk, nullptr, msg, nonce, nullptr, u_out, R_out, nullptr, c_out);
}
int sb200_sign_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* msg, const uint32_t* nonce,
                      uint32_t* u_out, uint32_t* R_out, uint32_t* Rp_out, uint32_t* c_out) {
  return sign_call(ctx, n, flags, 1, sk, nullptr, msg, nonce, nullptr, u_out, R_out, Rp_out, c_out);
}
int sb200_sign_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* gen, const uint32_t* msg,
                      const uint32_t* nonce, uint32_t* u_out, uint32_t* R_out, uint32_t* c_out) {
  return sign_call(ctx, n, flags, 2, sk, gen, msg, nonce, nullptr, u_out, R_out, nullptr, c_out);
}
int sb200_sign_stdrng(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* sk, const uint32_t* msg,
                      const uint32_t* gen, sb200_stdrng* rng, uint32_t* u_out, uint32_t* R_out, uint32_t* Rp_out, uint32_t* c_out) {
  if (sign_stdrng_args(n, flags, scheme, sk, msg, gen, rng, u_out, R_out, Rp_out) != SB200_OK) return SB200_ERR_ARG;
  return sign_call(ctx, n, flags, scheme, sk, gen, msg, nullptr, rng, u_out, R_out, Rp_out, c_out);
}
int sb200_keygen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, uint32_t* pk_out) {
  Desc d; d.op = OP_KEYGEN; d.flags = flags; d.nin = 1; d.nout = 1;
  IN(0, sk, 8); OUT(0, pk_out, 16);
  return run(ctx, n, d);
}
int sb200_keygen_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, uint32_t* pk_out, uint32_t* pkp_out) {
  Desc d; d.op = OP_KEYGEN_DOUBLE; d.flags = flags; d.nin = 1; d.nout = 2;
  IN(0, sk, 8); OUT(0, pk_out, 16); OUT(1, pkp_out, 16);
  return run(ctx, n, d);
}
int sb200_keygen_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* gen, uint32_t* pk_out) {
  Desc d; d.op = OP_KEYGEN_VARGEN; d.flags = flags; d.nin = 2; d.nout = 1;
  IN(0, sk, 8); IN(1, gen, pt_words(flags)); OUT(0, pk_out, 16);
  return run(ctx, n, d);
}
int sb200_points_decompress(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* bytes, uint32_t* points_out, uint32_t* ok_bitmap) {
  Desc d; d.op = OP_DECOMPRESS; d.flags = flags; d.nin = 1; d.nout = 1; BITMAP(ok_bitmap);
  IN(0, (const uint32_t*)bytes, 8); OUT(0, points_out, 16);
  return run(ctx, n, d);
}
int sb200_points_compress(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* points, uint8_t* bytes_out) {
  Desc d; d.op = OP_COMPRESS; d.flags = flags; d.nin = 1; d.nout = 1;
  IN(0, points, pt_words(flags)); OUT(0, (uint32_t*)bytes_out, 8);
  return run(ctx, n, d);
}
int sb200_scalars_from_wide(sb200_ctx* ctx, int64_t n, uint32_t flags, int field, const uint8_t* wide, uint32_t* out) {
  if (field < 0 || field > 1) return SB200_ERR_ARG;
  Desc d; d.op = OP_FROM_WIDE; d.flags = flags; d.aux = field; d.nin = 1; d.nout = 1;
  IN(0, (const uint32_t*)wide, 16); OUT(0, out, 8);
  return run(ctx, n, d);
}
int sb200_stdrng_random(sb200_ctx* ctx, int64_t n, uint32_t flags, int field, sb200_stdrng* rng, uint32_t* out) {
  if (stdrng_random_args(n, flags, field, rng, out) != SB200_OK) return SB200_ERR_ARG;
  Desc d; d.op = OP_STDRNG; d.flags = flags; d.aux = field; d.nin = 0; d.nout = 1; d.rng = rng;
  OUT(0, out, 8);
  const int rc = run(ctx, n, d);
  if (rc == SB200_OK) rng->word_pos += 16u * (uint64_t)n;  // only on success, as `&mut rng` would
  return rc;
}
static int fq_mont(sb200_ctx* ctx, int64_t n, uint32_t flags, int aux, const uint32_t* in, uint32_t* out) {
  Desc d; d.op = OP_DBG_FQ; d.flags = flags; d.aux = aux; d.nin = 2; d.nout = 1;
  IN(0, in, 8); IN(1, nullptr, 0); OUT(0, out, 8);
  return run(ctx, n, d);
}
int sb200_fq_to_mont(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* in, uint32_t* out) { return fq_mont(ctx, n, flags, 5, in, out); }
int sb200_fq_from_mont(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* in, uint32_t* out) { return fq_mont(ctx, n, flags, 6, in, out); }
// the byte-level calls of one scheme: pk_words / sk_words, sig_words and 8 words (msg, nonce) per tuple
static int verify_bytes_call(sb200_ctx* ctx, int64_t n, uint32_t flags, Op op, int pk_words, int sig_words, const uint8_t* pk,
                             const uint8_t* sig, const uint8_t* msg, uint32_t* verdicts, uint32_t* invalid) {
  Desc d; d.op = op; d.flags = flags; d.nin = 3; d.nout = 1; BITMAP(verdicts);
  IN(0, (const uint32_t*)pk, pk_words); IN(1, (const uint32_t*)sig, sig_words); IN(2, (const uint32_t*)msg, 8);
  OPT_OUT(0, invalid, -1);  // bitmap-shaped output: one word per 32 tuples
  return run(ctx, n, d);
}
static int sign_bytes_call(sb200_ctx* ctx, int64_t n, uint32_t flags, Op op, int sk_words, int sig_words, const uint8_t* sk,
                           const uint8_t* msg, const uint8_t* nonce, uint8_t* sig_out, uint32_t* invalid) {
  Desc d; d.op = op; d.flags = flags; d.nin = 3; d.nout = 1; d.bitmap = invalid;
  IN(0, (const uint32_t*)sk, sk_words); IN(1, (const uint32_t*)msg, 8); IN(2, (const uint32_t*)nonce, 8); OUT(0, (uint32_t*)sig_out, sig_words);
  return run(ctx, n, d);
}
int sb200_verify_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg,
                       uint32_t* verdicts, uint32_t* invalid) {
  return verify_bytes_call(ctx, n, flags, OP_VERIFY_BYTES, 8, 16, pk, sig, msg, verdicts, invalid);
}
int sb200_sign_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk, const uint8_t* msg, const uint8_t* nonce,
                     uint8_t* sig_out, uint32_t* invalid) {
  return sign_bytes_call(ctx, n, flags, OP_SIGN_BYTES, 8, 16, sk, msg, nonce, sig_out, invalid);
}
int sb200_verify_double_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg,
                              uint32_t* verdicts, uint32_t* invalid) {
  return verify_bytes_call(ctx, n, flags, OP_VERIFY_DOUBLE_BYTES, 16, 24, pk, sig, msg, verdicts, invalid);
}
int sb200_verify_vargen_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg,
                              uint32_t* verdicts, uint32_t* invalid) {
  return verify_bytes_call(ctx, n, flags, OP_VERIFY_VARGEN_BYTES, 16, 16, pk, sig, msg, verdicts, invalid);
}
int sb200_sign_double_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk, const uint8_t* msg, const uint8_t* nonce,
                            uint8_t* sig_out, uint32_t* invalid) {
  return sign_bytes_call(ctx, n, flags, OP_SIGN_DOUBLE_BYTES, 8, 24, sk, msg, nonce, sig_out, invalid);
}
int sb200_sign_vargen_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk, const uint8_t* msg, const uint8_t* nonce,
                            uint8_t* sig_out, uint32_t* invalid) {
  return sign_bytes_call(ctx, n, flags, OP_SIGN_VARGEN_BYTES, 16, 16, sk, msg, nonce, sig_out, invalid);
}
int sb200_sign_witness(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* sk, const uint32_t* msg,
                       const uint32_t* nonce, const uint32_t* generator, uint32_t* rows_out) {
  if (scheme < 0 || scheme > 2 || (scheme == 2 && !generator) || (scheme != 2 && (flags & SB200_POINTS_AFFINE))) return SB200_ERR_ARG;
  static const int width[3] = {11, 19, 13};
  Desc d; d.op = OP_WITNESS; d.flags = flags; d.aux = scheme; d.nin = 4; d.nout = 1;
  IN(0, sk, 8); IN(1, msg, 8); IN(2, nonce, 8); IN(3, scheme == 2 ? generator : nullptr, scheme == 2 ? pt_words(flags) : 0);
  OUT(0, rows_out, 8 * width[scheme]);
  return run(ctx, n, d);
}
int sb200_verify_witness(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* pk, const uint32_t* pk2,
                         const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                         uint32_t* verdicts, uint32_t* rows_out) {
  if (scheme < 0 || scheme > 2) return SB200_ERR_ARG;
  const int pw = pt_words(flags);
  Desc d; d.op = OP_VERIFY_WITNESS; d.flags = flags; d.aux = scheme; d.nout = 1; BITMAP(verdicts);
  int k = 0;  // the verify kernels' layout: pk, u, R, m | pk, pk', u, R, R', m | pk, gen, u, R, m
  IN(k, pk, pw); k++;
  if (scheme) { IN(k, pk2, pw); k++; }
  IN(k, sig_u, 8); k++;
  IN(k, sig_R, pw); k++;
  if (scheme == 1) { IN(k, sig_R_prime, pw); k++; }
  IN(k, msg, 8); k++;
  d.nin = k;
  OUT(0, rows_out, 8 * SB200_WITNESS_WIDTH(scheme));
  return run(ctx, n, d);
}
int sb200_verify_witness_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint8_t* pk_bytes,
                               const uint8_t* sig_bytes, const uint8_t* msg32, uint32_t* verdicts, uint32_t* rows_out,
                               uint32_t* invalid) {
  if (scheme < 0 || scheme > 2) return SB200_ERR_ARG;
  Desc d; d.op = OP_VERIFY_WITNESS_BYTES; d.flags = flags; d.aux = scheme; d.nin = 3; d.nout = 2; BITMAP(verdicts);
  IN(0, (const uint32_t*)pk_bytes, scheme == 0 ? 8 : 16); IN(1, (const uint32_t*)sig_bytes, scheme == 1 ? 24 : 16);
  IN(2, (const uint32_t*)msg32, 8);
  OUT(0, rows_out, 8 * SB200_WITNESS_WIDTH(scheme)); OPT_OUT(1, invalid, -1);
  return run(ctx, n, d);
}
int sb200_keyset_create(sb200_ctx* ctx, int scheme, int64_t n_keys, uint32_t flags, const uint32_t* pk, const uint32_t* pk2,
                        uint32_t* key_ok, sb200_keyset** out) {
  if (out) *out = nullptr;
  const int nt = scheme == 0 ? 1 : 2;
  const bool devptrs = (flags & SB200_DEVICE_PTRS) != 0;
  if (!ctx || !out || scheme < 0 || scheme > 2 || n_keys < 1 || n_keys > (int64_t)UINT32_MAX ||
      (flags & ~(SB200_POINTS_AFFINE | SB200_DEVICE_PTRS)))
    return SB200_ERR_ARG;
  if (!pk || ((uintptr_t)pk & 15) || (nt == 2 && (!pk2 || ((uintptr_t)pk2 & 15)))) return SB200_ERR_ARG;
  if (devptrs && ctx->devs.size() != 1) return SB200_ERR_ARG;
  std::lock_guard<std::mutex> lock(ctx->mu);
  ctx->set_err("");
  DeviceGuard guard;
  const size_t ndev = ctx->devs.size(), pt_bytes = (size_t)n_keys * pt_words(flags) * 4;
  const size_t tab_bytes = (size_t)n_keys * nt * KS_TABLE_WORDS * 4, ok_bytes = (size_t)((n_keys + 31) / 32) * 4;
  const int64_t batch = std::min<int64_t>(n_keys, KS_BUILD_KEYS);
  const size_t scr_bytes = (size_t)batch * 32 * 2 * (KS_ENTRIES - 1) * sizeof(fq);
  sb200_keyset* ks = new sb200_keyset{ctx, scheme, n_keys, std::vector<sb200_keyset::Dev>(ndev)};
  std::vector<uint8_t*> tmp(3 * ndev, nullptr);  // per device: scratch, and the copies of pk, pk2 (host inputs)
  auto fail = [&](int code, const char* what) {
    for (size_t di = 0; di < ndev; di++) {
      cudaSetDevice(ctx->devs[di].dev);
      if (devptrs) cudaStreamSynchronize(ctx->user_stream);
      for (int k = 0; k < 3; k++)
        if (tmp[3 * di + k]) cudaFree(tmp[3 * di + k]);
    }
    if (code != SB200_OK) {
      cudaGetLastError();  // a failed allocation is not the next call's error
      keyset_free(ks);
      ctx->set_err(what);
    }
    return code;
  };
  for (size_t di = 0; di < ndev; di++) {
    DevCtx& dc = ctx->devs[di];
    if (cudaSetDevice(dc.dev) != cudaSuccess) return fail(SB200_ERR_CUDA, "cudaSetDevice");
    sb200_keyset::Dev& kd = ks->dev[di];
    if (cudaMalloc(&kd.tab, tab_bytes) != cudaSuccess || cudaMalloc(&kd.ok, ok_bytes) != cudaSuccess ||
        cudaMalloc(&tmp[3 * di], scr_bytes) != cudaSuccess)
      return fail(SB200_ERR_NOMEM, "cudaMalloc keyset");
    // SB200_DEVICE_PTRS: on the caller's stream, after the work that produced the keys
    cudaStream_t st = devptrs ? ctx->user_stream : dc.stream[0];
    const uint32_t* src[2] = {pk, pk2};
    if (!devptrs)
      for (int p = 0; p < nt; p++) {
        if (cudaMalloc(&tmp[3 * di + 1 + p], pt_bytes) != cudaSuccess) return fail(SB200_ERR_NOMEM, "cudaMalloc keyset input");
        if (cudaMemcpyAsync(tmp[3 * di + 1 + p], src[p], pt_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess)
          return fail(SB200_ERR_CUDA, "cudaMemcpyAsync keyset input");
        src[p] = (const uint32_t*)tmp[3 * di + 1 + p];
      }
    if (cudaMemsetAsync(kd.ok, 0, ok_bytes, st) != cudaSuccess) return fail(SB200_ERR_CUDA, "cudaMemsetAsync key_ok");
    const Launcher go{ctx, st};
    for (int64_t k0 = 0; k0 < n_keys; k0 += batch) {
      const KsBuild b{kd.tab, kd.ok, src[0], nt == 2 ? src[1] : nullptr, k0, std::min(batch, n_keys - k0), nt,
                      (flags & SB200_POINTS_AFFINE) != 0, (fq*)tmp[3 * di]};
      go(k_keyset_build, (unsigned)((b.nk * 32 + TPB - 1) / TPB), TPB, 0, b);
    }
    if (cudaGetLastError() != cudaSuccess) return fail(SB200_ERR_CUDA, "k_keyset_build launch");
  }
  for (size_t di = 0; di < ndev; di++) {  // the builds of all devices run concurrently
    DevCtx& dc = ctx->devs[di];
    if (cudaSetDevice(dc.dev) != cudaSuccess || cudaStreamSynchronize(devptrs ? ctx->user_stream : dc.stream[0]) != cudaSuccess)
      return fail(SB200_ERR_CUDA, "k_keyset_build");
  }
  if (key_ok) {
    cudaSetDevice(ctx->devs[0].dev);
    if (cudaMemcpy(key_ok, ks->dev[0].ok, ok_bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return fail(SB200_ERR_CUDA, "key_ok copy");
  }
  fail(SB200_OK, "");  // frees the temporaries only
  ctx->keysets.push_back(ks);
  *out = ks;
  return SB200_OK;
}
void sb200_keyset_destroy(sb200_keyset* ks) {
  if (!ks) return;
  sb200_ctx* ctx = ks->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  DeviceGuard guard;
  ctx->keysets.erase(std::remove(ctx->keysets.begin(), ctx->keysets.end(), ks), ctx->keysets.end());
  keyset_free(ks);
}
int sb200_verify_keyset(sb200_ctx* ctx, const sb200_keyset* ks, int64_t n, uint32_t flags, const uint32_t* key_index,
                        const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                        uint32_t* verdicts, uint32_t* c_out) {
  if (!ctx || !ks) return SB200_ERR_ARG;
  {  // a keyset of this context that is still alive
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (std::find(ctx->keysets.begin(), ctx->keysets.end(), ks) == ctx->keysets.end()) return SB200_ERR_ARG;
  }
  const int pw = pt_words(flags);
  Desc d; d.op = OP_VERIFY_KEYSET; d.flags = flags; d.aux = ks->scheme; d.ks = ks; d.nout = 1; BITMAP(verdicts);
  int k = 0;  // key index, u, R, (R',) m
  IN(k, key_index, 1); k++;
  IN(k, sig_u, 8); k++;
  IN(k, sig_R, pw); k++;
  if (ks->scheme == 1) { IN(k, sig_R_prime, pw); k++; }
  IN(k, msg, 8); k++;
  d.nin = k;
  OPT_OUT(0, c_out, 8);
  return run(ctx, n, d);
}
int sb200_points_check(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* points, uint32_t* ok_bitmap) {
  Desc d; d.op = OP_POINTS_CHECK; d.flags = flags; d.nin = 1; d.nout = 0; BITMAP(ok_bitmap);
  IN(0, points, pt_words(flags));
  return run(ctx, n, d);
}
int sb200_dbg_verify_ec(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* sig_u, const uint32_t* sig_R,
                        const uint32_t* c, uint32_t* verdicts) {
  Desc d; d.op = OP_DBG_VERIFY_EC; d.flags = flags; d.nin = 4; d.nout = 0; BITMAP(verdicts);
  IN(0, pk, pt_words(flags)); IN(1, sig_u, 8); IN(2, sig_R, pt_words(flags)); IN(3, c, 8);
  return run(ctx, n, d);
}
int sb200_dbg_fq(sb200_ctx* ctx, int64_t n, int op, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  if (op < 0 || op > 7) return SB200_ERR_ARG;
  Desc d; d.op = OP_DBG_FQ; d.flags = 0; d.aux = op; d.nin = 2; d.nout = 1;
  IN(0, a, 8); IN(1, b, b ? 8 : 0); OUT(0, out, 8);
  return run(ctx, n, d);
}
int sb200_dbg_lattice3(sb200_ctx* ctx, int64_t n, const uint32_t* c, const uint32_t* u, uint32_t* out) {
  Desc d; d.op = OP_DBG_LAT3; d.flags = 0; d.nin = 2; d.nout = 1;
  IN(0, c, 8); IN(1, u, 8); OUT(0, out, 32);
  return run(ctx, n, d);
}
int sb200_dbg_fr_mul(sb200_ctx* ctx, int64_t n, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  Desc d; d.op = OP_DBG_FR_MUL; d.flags = 0; d.nin = 2; d.nout = 1;
  IN(0, a, 8); IN(1, b, 8); OUT(0, out, 8);
  return run(ctx, n, d);
}
int sb200_dbg_hades(sb200_ctx* ctx, int64_t n, int dense, uint32_t* states) {
  if (dense < 0 || dense > (SB_EXPERIMENTAL_FD ? 2 : 1)) return SB200_ERR_ARG;
  Desc d; d.op = OP_DBG_HADES; d.flags = 0; d.aux = dense; d.nin = 1; d.nout = 1;
  IN(0, states, 40); OUT(0, states, 40);
  return run(ctx, n, d);
}
int sb200_dbg_scalar_mul(sb200_ctx* ctx, int64_t n, uint32_t flags, int base, const uint32_t* points, const uint32_t* k, uint32_t* out) {
  if (base < 0 || base > 2 || (base == 2 && !points)) return SB200_ERR_ARG;
  Desc d; d.op = OP_DBG_SMUL; d.flags = flags; d.aux = base; d.nin = 2; d.nout = 1;
  IN(0, points, base == 2 ? pt_words(flags) : 0); IN(1, k, 8); OUT(0, out, 16);
  return run(ctx, n, d);
}

}  // extern "C"
