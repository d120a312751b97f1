/* schnorr_b200_witness -- PLONK witness rows of RECEIVED signatures (verifier side of SURVEY.md 8(f) row 4).
 *
 * sb200_sign_witness, in schnorr_b200.h, returns the witness rows of signatures the caller makes itself: it needs the
 * secret key and the nonce.  A prover that did not sign -- a proving service that receives signed transactions, a
 * circuit that re-proves signatures it collected -- holds only (PK, signature, message).  The two calls below compute
 * the same rows from that public tuple, together with the verdict of sb200_verify*, on the device.
 *
 * These calls have a header of their own.  schnorr_b200.h is the ABI whose every declaration has a row in the test
 * tables that pin its return codes and launch counts, and whose declarations `_lib.EXPORTED_SYMBOLS` lists; the calls
 * here are pinned by their own tests and bound by their own prototype table in schnorr_b200/_lib.py.  The library
 * exports both sets.  sb200_sign_witness stays in schnorr_b200.h.
 *
 * Row layout and width are those of sb200_sign_witness: SB200_WITNESS_WIDTH(scheme) = 11 / 19 / 13 field elements
 * (Montgomery, 8 x u32 each) for scheme 0 single, 1 double, 2 variable generator:
 *   scheme 0:  u, R, PK, m, c, SA, SB                  (points as (u, v))
 *   scheme 1:  u, R, R', PK, PK', m, c, SA, SB, SA', SB'
 *   scheme 2:  u, R, PK, GEN, m, c, SA, SB
 * R, R', PK, PK', GEN are the inputs in affine form (projective inputs are normalised on the device); u and c are
 * embedded in F_q as in sb200_sign_witness, c being the challenge sb200_verify* writes to c_out.  SA = u B (B = G, G'
 * or GEN) and SB = c PK (SA' = u G', SB' = c PK') are computed as scalar multiples, never derived from R.
 *
 * verdicts: bit i = (SA + SB == R [and SA' + SB' == R']), which equals sb200_verify*'s verdict of the tuple.  A tuple
 * that fails still gets its true row.  The row is all zero, with verdict 0, when u >= r (no JubJubScalar has that
 * value) and, with SB200_CHECK_POINTS, when an input point is off the curve or has Z = 0.  For a signature made by
 * sb200_sign_witness the row is bit-identical to the signer's.
 *
 * Arguments: scheme outside {0, 1, 2}, a flag not listed for the call, a missing required array, an array that is not
 * 16-byte aligned or n < 0 -> SB200_ERR_ARG, with nothing written and nothing launched; n = 0 -> SB200_OK.  Every input
 * is public: SB200_SIGN_OBLIVIOUS is not accepted. */
#ifndef SCHNORR_B200_WITNESS_H
#define SCHNORR_B200_WITNESS_H

#include "schnorr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Limb-level call.  flags: SB200_POINTS_AFFINE | SB200_DEVICE_PTRS | SB200_CHECK_POINTS.
 * pk2 = PK' (scheme 1) or the generator (scheme 2), ignored for scheme 0; sig_R_prime only for scheme 1.  Arguments a
 * scheme does not read may be NULL; pk, sig_u, sig_R, msg, verdicts and rows_out are required.
 * rows_out: n x 8 * SB200_WITNESS_WIDTH(scheme) u32.  One kernel launch per pipeline chunk. */
int sb200_verify_witness(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* pk, const uint32_t* pk2,
                         const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                         uint32_t* verdicts, uint32_t* rows_out);

/* Byte-level call: the inputs of sb200_verify_bytes / _double_bytes / _vargen_bytes (pk 32 | 64 | 64 B, sig 64 | 96 |
 * 64 B, msg32 canonical).  flags: SB200_DEVICE_PTRS only.  A tuple whose from_bytes fails has its bit set in `invalid`
 * (nullable), verdict 0 and an all-zero row; the other rows are those of sb200_verify_witness on the decoded tuple.
 * Two kernel launches per pipeline chunk (decode, witness). */
int sb200_verify_witness_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint8_t* pk_bytes,
                               const uint8_t* sig_bytes, const uint8_t* msg32, uint32_t* verdicts, uint32_t* rows_out,
                               uint32_t* invalid);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_WITNESS_H */
