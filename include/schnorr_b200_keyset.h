/* schnorr_b200_keyset -- verification against registered public keys, from per-key fixed-base tables on the device.
 *
 * sb200_verify* treat every public key as a fresh variable base: per tuple they build a window table of PK, shorten the
 * scalars and run the doublings of a variable-base multiplication.  Real batches repeat keys -- a node that verifies
 * every block's transactions from a stable set of accounts, a proving service that re-checks its customers' signatures,
 * a provisioner set that signs every round.  A keyset registers such keys once: each point gets a comb of 8-bit windows
 * (32 windows x 129 entries x 96 B = 396 288 B; entry e of window j = e 2^(8j) P in affine Niels form), so that c PK is
 * 32 mixed additions from memory.  u G comes from the context's comb of G as before; a verification is then the
 * challenge hash, two fixed-base combs and one projective compare.  Every tuple keeps its own verdict and challenge:
 * this is not random-linear-combination batch verification.
 *
 * Schemes: 0 single key (pk), 1 double key (pk, pk2 = PK'), 2 variable generator (pk, pk2 = the key's generator, whose
 * multiples u GEN also come from a per-key comb).
 *
 * Memory: every device of the context holds the whole keyset -- tuples are sharded by index and may name any key --
 * (scheme == 0 ? 1 : 2) x n_keys x 396 288 B, plus the key_ok bitmap (4 B per 32 keys).  Creation also takes a
 * temporary scratch region of up to 536 MB per device, freed before it returns.
 *
 * Exactness: every comb entry is an exact integer multiple of its point, so the verdicts are those of sb200_verify* on the
 * whole curve: torsion keys, small-order and identity keys, torsion components in R.  A key with a point off the curve
 * or with Z = 0 is recorded as malformed (key_ok bit clear); its own table may hold garbage, no other key's does, and
 * every tuple that names it gets verdict 0 whatever the flags.  sb200_verify's result for such a key is undefined, so
 * this is one of its behaviours.
 *
 * Lifetime: a keyset belongs to the context it was created on and is destroyed before it.  sb200_destroy frees any
 * keyset of the context that is still alive; their handles are invalid afterwards.
 *
 * These calls have a header of their own, like schnorr_b200_witness.h: schnorr_b200.h is the ABI whose every
 * declaration has a row in the tables that pin its return codes and launch counts; the calls here are pinned by their
 * own tests and bound by their own prototype table in schnorr_b200/_lib.py.  The library exports both sets. */
#ifndef SCHNORR_B200_KEYSET_H
#define SCHNORR_B200_KEYSET_H

#include "schnorr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb200_keyset sb200_keyset;

/* scheme 0 / 1 / 2.  pk: n_keys points; pk2 = PK' (scheme 1) or the generator (scheme 2), NULL for scheme 0.
 * flags: SB200_POINTS_AFFINE | SB200_DEVICE_PTRS (the layout and location of pk / pk2 only).
 * key_ok (nullable, host memory): ceil(n_keys/32) words, bit k = every point of key k is on the curve with Z != 0.
 * Builds the tables on every device of ctx (one kernel launch per 2048 keys and device) and returns when they are built.
 * SB200_ERR_ARG, with nothing allocated and nothing launched: null ctx or out, n_keys < 1 or n_keys > 2^32 - 1, a scheme
 * outside {0, 1, 2}, an unknown flag, a missing or not 16-byte aligned pk / pk2, SB200_DEVICE_PTRS on a multi-device
 * context.  SB200_ERR_NOMEM if any device cannot hold the keyset: nothing stays allocated.  *out is NULL on failure. */
int sb200_keyset_create(sb200_ctx* ctx, int scheme, int64_t n_keys, uint32_t flags, const uint32_t* pk,
                        const uint32_t* pk2, uint32_t* key_ok, sb200_keyset** out);

/* frees the keyset's device memory on every device; NULL: no-op */
void sb200_keyset_destroy(sb200_keyset* ks);

/* verdict i == sb200_verify*(pk[key_index[i]], ...) and c_out row i == its c_out row, for every well-formed key.
 * key_index: one u32 per tuple; an index >= n_keys gives verdict 0 (no table is read past the keyset), as does a
 * malformed key or u >= r.  sig_u, sig_R, sig_R_prime (scheme 1 only, else ignored), msg, verdicts and c_out (nullable)
 * have the layout of sb200_verify*.  flags: SB200_POINTS_AFFINE | SB200_DEVICE_PTRS | SB200_CHECK_POINTS (R, R').
 * One kernel launch per pipeline chunk.  SB200_ERR_ARG, with nothing written and nothing launched: a null or foreign
 * keyset (one of another context), an unknown flag, a missing or misaligned array, n < 0.  n = 0 -> SB200_OK. */
int sb200_verify_keyset(sb200_ctx* ctx, const sb200_keyset* ks, int64_t n, uint32_t flags, const uint32_t* key_index,
                        const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                        uint32_t* verdicts, uint32_t* c_out);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_KEYSET_H */
