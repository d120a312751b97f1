// Host build of the device-side StdRng (csrc/rng.cuh): ChaCha12 blocks, the 16 keystream words at any word position,
// Field::random at a position, from_bytes_wide alone and the entry points' argument checks, exported with C linkage for tests/test_stdrng.py.
// Test scaffolding: never linked into libschnorr_b200.so.
#include <cstring>
#include "../include/schnorr_b200.h"
#include "../schnorr_b200/csrc/rng.cuh"
using namespace sb200;

extern "C" {
void h_chacha12_block(const uint32_t* key, uint64_t counter, uint32_t* out16) { chacha12_block(key, counter, out16); }
void h_stdrng_draw(const uint32_t* key, uint64_t word_pos, uint32_t* out16) { stdrng_draw(key, word_pos, out16); }
void h_stdrng_random(const uint32_t* key, uint64_t word_pos, int field, uint32_t* out8) { stdrng_random(key, word_pos, field, out8); }
// from_bytes_wide of one 64-byte draw (16 LE words): field 0 -> canonical mod r, 1 -> Montgomery mod q
void h_from_wide(const uint32_t* w16, int field, uint32_t* out8) {
  if (field == 0) {
    fr_from_wide(w16, out8);
  } else {
    const fq x = fq_from_wide(w16);
    memcpy(out8, x.v, 32);
  }
}
// the argument checks of the two entry points, as they run before any context is looked at
int h_stdrng_random_args(int64_t n, uint32_t flags, int field, const sb200_stdrng* rng, const void* out) {
  return stdrng_random_args(n, flags, field, rng, out);
}
int h_sign_stdrng_args(int64_t n, uint32_t flags, int scheme, const void* sk, const void* msg, const void* gen, const sb200_stdrng* rng,
                       const void* u_out, const void* R_out, const void* Rp_out) {
  return sign_stdrng_args(n, flags, scheme, sk, msg, gen, rng, u_out, R_out, Rp_out);
}
}
