/* schnorr_b200_keyset_witness -- PLONK witness rows of received signatures, from the per-key tables of a keyset.
 *
 * sb200_verify_witness, in schnorr_b200_witness.h, serves a prover that received signatures, but treats every public key as
 * a fresh variable base: per tuple it multiplies c PK (and, for a variable generator, u GEN) by a window table of the
 * point.  A proving service that re-proves the signatures of a stable set of customers' keys has those keys registered
 * in a keyset (schnorr_b200_keyset.h), whose 8-bit combs give c PK, c PK' and u GEN as 32 mixed additions.  The calls
 * below return the rows and verdicts of sb200_verify_witness from the keyset instead:
 *   - PK (PK', GEN) are the key's affine coordinates, read back from entry 1 of window 0 of its comb;
 *   - c is the challenge sb200_verify* and sb200_verify_keyset write to c_out;
 *   - SA = u G (u G') by the context's comb, or u GEN by the key's comb of its generator, and SB = c PK (c PK') by the key's
 *     comb -- both computed as exact multiples, never derived from R;
 *   - verdict bit i = (SA + SB == R [and SA' + SB' == R']).
 * Row layout and width are those of sb200_verify_witness: SB200_WITNESS_WIDTH(scheme) field elements per tuple.
 *
 * Parity: for every tuple whose key index is below n_keys and whose key has its key_ok bit set, the row and the verdict
 * equal those of sb200_verify_witness*(pk[key_index[i]], ...) on the gathered keys, bit for bit, with the same flags.
 * (One exception, outside that contract's inputs: a projective R or R' with Z = 0 and no SB200_CHECK_POINTS.  The key's
 * columns then hold the key, where sb200_verify_witness's shared inversion leaves garbage.)
 * A tuple with a good key and a wrong signature keeps its true row and gets verdict 0.  The row is all zero and the verdict
 * 0 when u >= r, the key index is >= n_keys, the key's key_ok bit is clear (a malformed key, or a slot revoked by
 * sb200_keyset_revoke), or, with SB200_CHECK_POINTS, R (R') is off the curve or has Z = 0.
 *
 * Arguments and errors follow sb200_verify_keyset: arrays 16-byte aligned and tuple-major, a keyset alive and of ctx.
 * SB200_ERR_ARG, with nothing written and nothing launched: a null, foreign or destroyed keyset, a flag not listed for the
 * call (SB200_SIGN_OBLIVIOUS and SB200_VERIFY_DUAL_PIPE included), a missing or misaligned required array, n < 0.
 * n = 0 -> SB200_OK with no launch.  sig_R_prime is read for scheme 1 only.  Calls are ordered against
 * sb200_keyset_update* and _revoke by the context's lock: a call issued after one of them returns reads the new tables.
 *
 * These calls have a header of their own and their own prototype table in schnorr_b200/_lib.py; the library exports them
 * beside the calls of schnorr_b200.h, schnorr_b200_witness.h, schnorr_b200_keyset.h and schnorr_b200_keyset_live.h. */
#ifndef SCHNORR_B200_KEYSET_WITNESS_H
#define SCHNORR_B200_KEYSET_WITNESS_H

#include "schnorr_b200_witness.h"
#include "schnorr_b200_keyset.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Limb-level call.  key_index: one u32 per tuple; sig_u, sig_R, sig_R_prime, msg: the layout of sb200_verify_keyset.
 * flags: SB200_POINTS_AFFINE | SB200_DEVICE_PTRS | SB200_CHECK_POINTS (R, R').  verdicts and rows_out are required;
 * rows_out: n x 8 * SB200_WITNESS_WIDTH(scheme of ks) u32.  One kernel launch per pipeline chunk. */
int sb200_verify_witness_keyset(sb200_ctx* ctx, const sb200_keyset* ks, int64_t n, uint32_t flags, const uint32_t* key_index,
                                const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                                uint32_t* verdicts, uint32_t* rows_out);

/* Byte-level call: the signature and message bytes of sb200_verify_keyset_bytes.  flags: SB200_DEVICE_PTRS only.
 * invalid (nullable): bit i = a from_bytes of the tuple's signature or message fails; such a tuple gets verdict 0 and an
 * all-zero row.  For every key that decoded and holds its key_ok bit, rows, verdicts and invalid bits equal
 * sb200_verify_witness_bytes on the gathered key bytes.  Two kernel launches per pipeline chunk: the decode of
 * sb200_verify_keyset_bytes, then the kernel of sb200_verify_witness_keyset. */
int sb200_verify_witness_keyset_bytes(sb200_ctx* ctx, const sb200_keyset* ks, int64_t n, uint32_t flags,
                                      const uint32_t* key_index, const uint8_t* sig_bytes, const uint8_t* msg32,
                                      uint32_t* verdicts, uint32_t* rows_out, uint32_t* invalid);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_KEYSET_WITNESS_H */
