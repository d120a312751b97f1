/* schnorr_b200_keyset_live -- keysets fed with wire-format bytes, and keysets that change while they are in use.
 *
 * The calls of schnorr_b200_keyset.h take keys and signatures as Montgomery limbs and freeze a keyset at creation.  A node
 * receives bytes -- PublicKey::to_bytes() (32 B), PublicKeyDouble / PublicKeyVarGen::to_bytes() (64 B), Signature /
 * SignatureVarGen::to_bytes() (64 B), SignatureDouble::to_bytes() (96 B), messages as 32 canonical bytes -- and its key set
 * changes: provisioner sets rotate, accounts are opened and closed.  The calls below decode on the device and rebuild or
 * revoke single slots of a live keyset in place, instead of rebuilding the whole keyset.
 *
 * Capacity is fixed at creation.  To add keys later, register spare slots with placeholder keys (undecodable bytes or any
 * point), revoke them, and fill them with sb200_keyset_update* as keys arrive.
 *
 * Ordering: sb200_keyset_update, _update_bytes and _revoke take the context's lock, are ordered after all work the context
 * has already enqueued (SB200_DEVICE_PTRS work on the caller's stream included) and return when every device of the
 * context has finished.  A verification enqueued before the call reads the old keys; one issued after it returns reads the
 * new ones.  After an update or a revoke the keyset answers bit for bit as a keyset freshly created from the resulting key
 * list, with the revoked slots' keys malformed.
 *
 * Arguments follow schnorr_b200_keyset.h: arrays 16-byte aligned and tuple-major, int64_t counts, a keyset alive and (for
 * the calls that take ctx) of ctx.  SB200_ERR_ARG: nothing written, nothing allocated, nothing launched.  n = 0 / m = 0 ->
 * SB200_OK with no launch.  These calls have a header of their own and their own prototype table in schnorr_b200/_lib.py;
 * the library exports them beside the calls of schnorr_b200.h and schnorr_b200_keyset.h. */
#ifndef SCHNORR_B200_KEYSET_LIVE_H
#define SCHNORR_B200_KEYSET_LIVE_H

#include "schnorr_b200_keyset.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Verification of wire-format signatures against a keyset.  key_index: one u32 per tuple; sig_bytes: sig64 (u || R) for
 * schemes 0 and 2, sig96 (u || R || R') for scheme 1, laid out as in sb200_verify*_bytes; msg32: canonical.
 * flags: SB200_DEVICE_PTRS only.  invalid (nullable): bit i = a from_bytes of the tuple's signature or message fails
 * (u >= r, R or R' does not decompress, msg >= q); such a tuple gets verdict 0.
 * For every key whose bytes decode, verdict i and invalid bit i equal those of sb200_verify*_bytes(pk_bytes[key_index[i]],
 * sig_bytes[i], msg32[i]).  Verdict 0 with invalid bit 0 -- the key is not part of the tuple's bytes -- for an index >=
 * n_keys, a key without its key_ok bit (sb200_verify*_bytes would set `invalid` for a key that does not decode) and a
 * revoked slot.  Two kernel launches per pipeline chunk: the decode of the tuple, then the kernel of sb200_verify_keyset. */
int sb200_verify_keyset_bytes(sb200_ctx* ctx, const sb200_keyset* ks, int64_t n, uint32_t flags, const uint32_t* key_index,
                              const uint8_t* sig_bytes, const uint8_t* msg32, uint32_t* verdicts, uint32_t* invalid);

/* sb200_keyset_create from the keys' to_bytes() form: 32 B per key for scheme 0 (PublicKey), 64 B for scheme 1 (pk || pk')
 * and scheme 2 (pk || generator).  flags: SB200_DEVICE_PTRS only (refused on a multi-device context).  key_ok (nullable,
 * host): bit k = the key's from_bytes succeeds.  A key that decodes behaves exactly as the same key given to
 * sb200_keyset_create as affine points; one that does not is a malformed key.  One decode launch per device, then the build
 * launches of sb200_keyset_create. */
int sb200_keyset_create_bytes(sb200_ctx* ctx, int scheme, int64_t n_keys, uint32_t flags, const uint8_t* pk_bytes,
                              uint32_t* key_ok, sb200_keyset** out);

/* Rebuilds the tables of m slots in place with new keys, on every device of the keyset's context.  slots: host memory, m
 * distinct indices below n_keys (else SB200_ERR_ARG, checked before anything is allocated or launched).  pk / pk2: m keys
 * in the layout of sb200_keyset_create; flags: SB200_POINTS_AFFINE | SB200_DEVICE_PTRS (the location of pk / pk2; refused
 * on a multi-device context).  key_ok (nullable, host): ceil(m/32) words, bit j = the new key_ok bit of slots[j] -- set for
 * a good key written over a malformed or revoked one, cleared for a malformed key written over a good one.  Build scratch as
 * at creation (up to 536 MB per device for 2048 slots per launch), freed before return.  SB200_ERR_NOMEM: the keyset is
 * unchanged. */
int sb200_keyset_update(sb200_keyset* ks, int64_t m, uint32_t flags, const uint32_t* slots, const uint32_t* pk,
                        const uint32_t* pk2, uint32_t* key_ok);

/* sb200_keyset_update with the keys in the byte form of sb200_keyset_create_bytes.  flags: SB200_DEVICE_PTRS only. */
int sb200_keyset_update_bytes(sb200_keyset* ks, int64_t m, uint32_t flags, const uint32_t* slots, const uint8_t* pk_bytes,
                              uint32_t* key_ok);

/* Clears the key_ok bits of m slots (host memory, checked as in sb200_keyset_update) on every device: tuples that name them
 * get verdict 0 from both verify calls; no table is rebuilt, and every other tuple's verdict and c_out are unchanged.  A
 * later update of a slot registers a key there again.  One kernel launch per device. */
int sb200_keyset_revoke(sb200_keyset* ks, int64_t m, const uint32_t* slots);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_KEYSET_LIVE_H */
