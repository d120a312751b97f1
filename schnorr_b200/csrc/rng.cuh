// Field::random over a rand 0.8 `StdRng` on the device: the ChaCha12 keystream at any position, reduced with the
// from_bytes_wide of wire.cuh (/root/reference/src/keys/secret.rs:83,155).
//
// StdRng = rand_chacha's ChaCha12 with stream 0: constants "expand 32-byte k", the 32-byte seed as 8 little-endian key
// words, a 64-bit block counter in words 12-13, words 14-15 = 0, six double rounds and the feed-forward.  rand_core's
// BlockRng hands the keystream out in whole 32-bit words, so a word position (16 x block + word within the block)
// describes a generator's state exactly, and block k depends on the key and k only: any draw is computed without the
// ones before it.  The library keeps no RNG state; the caller hands in a position and gets the advanced one back.
//
// No branch and no address depends on the key or on the drawn words (ChaCha is add-rotate-xor, the reduction is
// select-based), so the seeded signers keep SB200_SIGN_OBLIVIOUS's promise.  The only branch is on the word offset
// within a block, which is part of the public position and the same for every draw of a call.
#pragma once
#include "../../include/schnorr_b200.h"
#include "wire.cuh"

namespace sb200 {

SB_HD uint32_t chacha_rotl(uint32_t v, int n) { return (v << n) | (v >> (32 - n)); }

SB_HD void chacha_qr(uint32_t* x, int a, int b, int c, int d) {
  x[a] += x[b]; x[d] = chacha_rotl(x[d] ^ x[a], 16);
  x[c] += x[d]; x[b] = chacha_rotl(x[b] ^ x[c], 12);
  x[a] += x[b]; x[d] = chacha_rotl(x[d] ^ x[a], 8);
  x[c] += x[d]; x[b] = chacha_rotl(x[b] ^ x[c], 7);
}

// ChaCha12 block `counter` of the stream-0 keystream under `key`: 16 little-endian words
SB_HD void chacha12_block(const uint32_t* key, uint64_t counter, uint32_t* out) {
  uint32_t st[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u};
#pragma unroll
  for (int i = 0; i < 8; i++) st[4 + i] = key[i];
  st[12] = (uint32_t)counter;
  st[13] = (uint32_t)(counter >> 32);
  st[14] = st[15] = 0u;
  uint32_t x[16];
#pragma unroll
  for (int i = 0; i < 16; i++) x[i] = st[i];
#pragma unroll
  for (int r = 0; r < 6; r++) {
    chacha_qr(x, 0, 4, 8, 12); chacha_qr(x, 1, 5, 9, 13); chacha_qr(x, 2, 6, 10, 14); chacha_qr(x, 3, 7, 11, 15);
    chacha_qr(x, 0, 5, 10, 15); chacha_qr(x, 1, 6, 11, 12); chacha_qr(x, 2, 7, 8, 13); chacha_qr(x, 3, 4, 9, 14);
  }
#pragma unroll
  for (int i = 0; i < 16; i++) out[i] = x[i] + st[i];
}

// The 16 keystream words starting at word `word_pos`: words off..15 of block b = word_pos / 16, then words 0..off-1 of
// block b + 1.  The two blocks are shifted into place by a barrel shifter of selects on the bits of off, so the words
// stay in registers (a dynamic index would put them in local memory).
SB_HD void stdrng_draw(const uint32_t* key, uint64_t word_pos, uint32_t* out) {
  const uint64_t b = word_pos >> 4;
  const int off = (int)(word_pos & 15u);
  uint32_t w[32];
  chacha12_block(key, b, w);
  if (off) {
    chacha12_block(key, b + 1, w + 16);
  } else {
#pragma unroll
    for (int i = 16; i < 32; i++) w[i] = 0u;
  }
#pragma unroll
  for (int s = 1; s < 16; s <<= 1) {
    const bool take = (off & s) != 0;
#pragma unroll
    for (int j = 0; j + s < 32; j++) w[j] = take ? w[j + s] : w[j];  // ascending j: w[j + s] is still the old word
  }
#pragma unroll
  for (int i = 0; i < 16; i++) out[i] = w[i];
}

// Field::random at `word_pos`: field 0 -> JubJubScalar (canonical limbs), 1 -> BlsScalar (Montgomery limbs)
SB_HD void stdrng_random(const uint32_t* key, uint64_t word_pos, int field, uint32_t* out) {
  uint32_t w[16];
  stdrng_draw(key, word_pos, w);
  if (field == 0) {
    fr_from_wide(w, out);
  } else {
    const fq x = fq_from_wide(w);
#pragma unroll
    for (int k = 0; k < 8; k++) out[k] = x.v[k];
  }
}

// Argument checks of sb200_stdrng_random / sb200_sign_stdrng (host only; shared with the host build the tests drive):
// SB200_OK or SB200_ERR_ARG, decided before any context or device is looked at.  word_pos + 16 n must fit in 64 bits.
inline bool stdrng_span_ok(const sb200_stdrng* rng, int64_t n) {
  return rng && n >= 0 && (uint64_t)n <= (UINT64_MAX - rng->word_pos) / 16u;
}
inline int stdrng_random_args(int64_t n, uint32_t flags, int field, const sb200_stdrng* rng, const void* out) {
  return (out && stdrng_span_ok(rng, n) && field >= 0 && field <= 1 && !(flags & ~SB200_DEVICE_PTRS)) ? SB200_OK : SB200_ERR_ARG;
}
// the flags of the scheme's sign entry point: SB200_POINTS_AFFINE only where a generator is read (scheme 2)
inline int sign_stdrng_args(int64_t n, uint32_t flags, int scheme, const void* sk, const void* msg, const void* gen,
                            const sb200_stdrng* rng, const void* u_out, const void* R_out, const void* Rp_out) {
  if (!stdrng_span_ok(rng, n) || scheme < 0 || scheme > 2 || !sk || !msg || !u_out || !R_out) return SB200_ERR_ARG;
  if ((scheme == 1 && !Rp_out) || (scheme == 2 && !gen)) return SB200_ERR_ARG;
  const uint32_t allowed = SB200_DEVICE_PTRS | SB200_SIGN_OBLIVIOUS | (scheme == 2 ? SB200_POINTS_AFFINE : 0u);
  return (flags & ~allowed) ? SB200_ERR_ARG : SB200_OK;
}

}  // namespace sb200
