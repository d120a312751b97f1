/* schnorr_b200 -- C ABI of the B200 batch engine for dusk-schnorr's sign / verify hot path.
 *
 * The reference (dusk-schnorr 0.18.0, pure Rust) has no FFI; its boundary for this path is the
 * crate's public API.  Each entry point below is the batch form of one reference method and is what
 * a `#[link(name = "schnorr_b200")] extern "C"` block in the crate would bind (INTEGRATION.md):
 *
 *   sb200_verify          PublicKey::verify            /root/reference/src/keys/public.rs:121-130
 *   sb200_verify_double   PublicKeyDouble::verify      /root/reference/src/keys/public.rs:222-244
 *   sb200_verify_vargen   PublicKeyVarGen::verify      /root/reference/src/keys/public.rs:401-415
 *   sb200_sign            SecretKey::sign              /root/reference/src/keys/secret.rs:150-168
 *   sb200_sign_double     SecretKey::sign_double       /root/reference/src/keys/secret.rs:217-240
 *   sb200_sign_vargen     SecretKeyVarGen::sign        /root/reference/src/keys/secret.rs:433-451
 *   sb200_keygen          PublicKey::from(&SecretKey)          /root/reference/src/keys/public.rs:61-67
 *   sb200_keygen_double   PublicKeyDouble::from(&SecretKey)    /root/reference/src/keys/public.rs:265-272
 *   sb200_keygen_vargen   PublicKeyVarGen::from(&SecretKeyVarGen) /root/reference/src/keys/public.rs:337-344
 *
 * Data layout (all arrays are caller-owned, tuple-major, tightly packed, 16-byte aligned):
 *   field element (BlsScalar: message, point coordinates) = 8 x u32 little-endian limbs in
 *       MONTGOMERY form (x * 2^256 mod q) -- bit-identical to `BlsScalar.0: [u64; 4]` on a
 *       little-endian host, so Rust hands over its internal limbs without conversion.  Must be < q.
 *   scalar (JubJubScalar: sk, nonce, u, c) = 8 x u32 little-endian limbs of the CANONICAL integer
 *       (= `JubJubScalar::to_bytes()`), must be < r.  A `u` >= r makes that tuple's verdict 0.
 *   point  = SB200_POINTS_AFFINE:      (u, v)      2 field elements (64 B);
 *            SB200_POINTS_PROJECTIVE:  (U, V, Z)   3 field elements (96 B), Z != 0 -- the
 *            (u, v, z) of a JubJubExtended; t1/t2 are not needed.  Points must be on the curve
 *            (the reference can only produce on-curve points outside `from_raw_unchecked`).
 *       One flag applies to every point array of the call.  Points written by the library are
 *       always affine (u, v), Montgomery form.
 *   verdicts = bitmap, bit (i & 31) of word (i >> 5) is tuple i's `verify` result; ceil(n/32) words.
 *
 * Nonces are an INPUT (`nonce[i]` is the one `JubJubScalar::random(rng)` draw of signature i,
 * /root/reference/src/keys/secret.rs:155): the RNG state stays with the caller.  The library generates no
 * randomness of its own; sb200_stdrng_random and sb200_sign_stdrng expand a caller-owned StdRng position
 * (seed + keystream word) deterministically on the device into exactly the draws the caller's generator would
 * have made, and hand back the advanced position.
 *
 * Threading: one batch in flight per context (calls on one context are serialised by an internal
 * mutex); distinct contexts are independent.  Calls block until the outputs are in host memory,
 * except with SB200_DEVICE_PTRS (see below).  No call aborts; errors are return codes.
 * There is no CPU fallback: without a usable CUDA device sb200_init fails with SB200_ERR_NODEV.
 */
#ifndef SCHNORR_B200_H
#define SCHNORR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb200_ctx sb200_ctx;

enum {
  SB200_OK = 0,
  SB200_ERR_ARG = -1,    /* null pointer, n < 0, unknown flag, misaligned buffer */
  SB200_ERR_CUDA = -2,   /* a CUDA call failed; sb200_last_error() has the text */
  SB200_ERR_NODEV = -3,  /* no usable sm_100 device */
  SB200_ERR_NOMEM = -4,
  SB200_ERR_PARAMS = -5, /* sb200_params rejected: generator off the curve / not of prime order, non-canonical field
                            element, singular MDS block, or the sparse form failed its self-check */
  SB200_ERR_BUSY = -6    /* a live context on the same device was created with different parameters (the Hades
                            tables live in that device's constant memory, one set per process and device) */
};

#define SB200_POINTS_PROJECTIVE 0u
#define SB200_POINTS_AFFINE 1u
/* All buffers are device pointers on the context's (single) device; the call enqueues its kernel on
 * the stream set with sb200_set_stream and returns without synchronising. */
#define SB200_DEVICE_PTRS 2u
/* sb200_verify only, and only in builds with -DSB_EXPERIMENTAL_FD=1 (otherwise SB200_ERR_ARG): the warp-specialised
 * kernel with hash warps on the FP64 pipe (DESIGN.md 4.4).  Same verdicts; measured 22 % slower than the default. */
#define SB200_VERIFY_DUAL_PIPE 4u
/* sb200_verify / _double / _vargen: additionally check every input point (on the curve, Z != 0) on the device; a
 * tuple with a failing point gets verdict 0 instead of undefined behaviour.  For callers that build keys with
 * `from_raw_unchecked` (/root/reference/src/keys/public.rs:142,256,427).  See also sb200_points_check. */
#define SB200_CHECK_POINTS 8u

/* sb200_sign / _sign_double / _sign_vargen / _keygen*: address-oblivious scalar multiplication -- no memory address and
 * no branch depends on the nonce or the secret key (the reference's ladder is a constant-time select).  Fixed base:
 * 4-bit combs of G and G' staged in shared memory and read by masked scan (64 additions instead of the 16 of the
 * default 16-bit comb, whose 50 MB table in HBM is indexed with scalar digits); variable base: the window table is
 * scanned instead of indexed; the conversion to affine form keeps Fermat's fixed-length a^(q-2) instead of the Euclidean
 * inversion (whose running time depends on its input).  Same outputs bit for bit; slower (DESIGN.md 4.2 has the measured ratio). */
#define SB200_SIGN_OBLIVIOUS 16u

/* ---- scheme parameters ------------------------------------------------------------------------------------------
 * Everything numeric that dusk-schnorr takes from its un-vendored dependency crates and that cannot be checked in
 * this build environment (SURVEY.md 8(b), 8(c)) is an INPUT of context creation:
 *   generator, generator_nums   dusk_jubjub::GENERATOR / GENERATOR_NUMS, affine (u, v)
 *                               (GENERATOR_EXTENDED, GENERATOR_NUMS_EXTENDED at /root/reference/src/keys/secret.rs:159,231-232,
 *                               /root/reference/src/keys/public.rs:63,127,236-239,267-268)
 *   round_constants             dusk_hades ROUND_CONSTANTS[0 .. 335) (67 rounds x 5 words, consumed in order)
 *   mds                         dusk_hades MDS_MATRIX[i][j]; a round computes result[i] = sum_j mds[i][j] * state[j]
 *                               (both used by sponge::truncated::hash at /root/reference/src/signatures.rs:133,283-289)
 * All field elements are 8 x u32 Montgomery limbs = the crate's own `BlsScalar.0`, so a Rust host copies its tables
 * verbatim (rust/src/cuda.rs `params_from_crate`).  The sparse factorisation of the partial rounds that the kernels
 * run is derived from these at sb200_init_ex and checked against the dense permutation before anything is uploaded. */
typedef struct sb200_params {
  uint32_t struct_size; /* = sizeof(sb200_params) */
  uint32_t reserved;    /* 0 */
  uint32_t generator[16];
  uint32_t generator_nums[16];
  uint32_t round_constants[335][8];
  uint32_t mds[5][5][8];
} sb200_params;

/* Rules for the DEFAULT round constants.  Both are recollections of dusk-hades' published recipe (assets/HOWTO.md:
 * bytes = "poseidon-for-plonk"; repeat bytes = SHA-512(bytes), h_i = BlsScalar::from_bytes_wide(bytes)); they differ in
 * whether the table is the running sum seeded with one.  Which one the crate uses is unverifiable here
 * (DESIGN.md section 2); rust/tests/dump_golden.rs settles it, and a host with the crate passes its own table. */
#define SB200_ARK_CUMSUM 0 /* p = 1; c_i = h_i + p; p = c_i   (default) */
#define SB200_ARK_PLAIN 1  /* c_i = h_i */
#define SB200_ARK_ENV (-1) /* the rule named by the environment variable SB200_ARK ("cumsum" | "plain"), else CUMSUM */
/* Fill *out with the default parameters: recalled generators, recipe-derived round constants, Cauchy MDS 1/(i+j+5).
 * Host-only (no CUDA call). */
int sb200_default_params(int ark_rule, sb200_params* out);

/* devices: CUDA ordinals to shard over (tuples are split into contiguous blocks, multiples of 32);
 * n_devices = 0 means "device 0".  Validates the parameters, derives and uploads the Hades tables and builds the comb
 * tables of both generators on every device. */
/* Environment variable read at context creation: SB200_CURVE_PERSISTENT = "always" | "never" selects the form of the curve
 * kernels of the three verifications regardless of batch size (default: the persistent global-table kernel for batches above one
 * wave of resident CTAs, the local-memory kernel below; results are identical -- tests run both). */
int sb200_init_ex(const sb200_params* params, const int* devices, int n_devices, sb200_ctx** out);
/* = sb200_init_ex(sb200_default_params(SB200_ARK_ENV), ...) */
int sb200_init(const int* devices, int n_devices, sb200_ctx** out);
/* Validate parameters exactly as sb200_init_ex does, without touching a GPU: canonical field elements, both generators
 * on the curve and of prime order r, the partial-round blocks invertible, sparse form == dense permutation.
 * tables_out (nullable, 1039 x 8 u32) receives the derived Hades tables (layout of sb200_dbg_hades_tables). */
int sb200_params_check(const sb200_params* params, uint32_t* tables_out);
/* the parameters a context was created with */
int sb200_get_params(const sb200_ctx* ctx, sb200_params* out);
void sb200_destroy(sb200_ctx* ctx);
const char* sb200_strerror(int code);
const char* sb200_last_error(const sb200_ctx* ctx);
int sb200_device_count(const sb200_ctx* ctx);
/* stream (a cudaStream_t) used by SB200_DEVICE_PTRS calls; NULL = the legacy default stream.  The split kernels of
 * one context share a scratch buffer, so DEVICE_PTRS work of one context is ordered: after a switch, the new stream
 * first waits (cudaStreamWaitEvent) for what the context enqueued on the previous one. */
int sb200_set_stream(sb200_ctx* ctx, void* cuda_stream);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
uint64_t sb200_launch_count(const sb200_ctx* ctx);
/* pinned host memory for full-speed host<->device copies.  Pageable buffers also work: the library detects them and
 * stages every chunk through its own pinned ring, so the copy/compute overlap is kept (one extra host memcpy). */
int sb200_host_alloc(size_t bytes, void** out);
void sb200_host_free(void* p);

/* c_out (n x 8 u32, canonical challenge scalars) may be NULL in every call below. */
int sb200_verify(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* sig_u,
                 const uint32_t* sig_R, const uint32_t* msg, uint32_t* verdicts, uint32_t* c_out);
int sb200_verify_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* pk_prime,
                        const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* sig_R_prime, const uint32_t* msg,
                        uint32_t* verdicts, uint32_t* c_out);
int sb200_verify_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* generator,
                        const uint32_t* sig_u, const uint32_t* sig_R, const uint32_t* msg, uint32_t* verdicts,
                        uint32_t* c_out);

/* u_out: n x 8 u32 canonical; R_out (and R_prime_out): n x 16 u32 affine (u, v) Montgomery. */
int sb200_sign(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* msg, const uint32_t* nonce,
               uint32_t* u_out, uint32_t* R_out, uint32_t* c_out);
int sb200_sign_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* msg,
                      const uint32_t* nonce, uint32_t* u_out, uint32_t* R_out, uint32_t* R_prime_out, uint32_t* c_out);
int sb200_sign_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* generator,
                      const uint32_t* msg, const uint32_t* nonce, uint32_t* u_out, uint32_t* R_out, uint32_t* c_out);

/* pk_out: n x 16 u32 affine (u, v) Montgomery */
int sb200_keygen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, uint32_t* pk_out);
int sb200_keygen_double(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, uint32_t* pk_out,
                        uint32_t* pk_prime_out);
int sb200_keygen_vargen(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* sk, const uint32_t* generator,
                        uint32_t* pk_out);

/* ---- wire formats on the device (the reference's serialised forms, SURVEY.md 8(f)) ---------------------
 * bytes32 point  = JubJubAffine::to_bytes (v little-endian, bit 255 = low bit of u);
 * sig64          = Signature::to_bytes = u (32 B canonical) || compressed R   /root/reference/src/signatures.rs:106-123
 * msg32 / sk32   = BlsScalar::to_bytes / SecretKey::to_bytes (32 B canonical little-endian)
 * `flags` here may only carry SB200_DEVICE_PTRS. */
/* JubJubAffine::from_bytes for n points; ok bit i = 0 where the reference returns None (v >= q or not on the
 * curve).  No subgroup check, as in the reference (/root/reference/src/keys/public.rs:94-100). */
int sb200_points_decompress(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* bytes32, uint32_t* points_out,
                            uint32_t* ok_bitmap);
/* JubJubAffine::from(point).to_bytes(); points per SB200_POINTS_AFFINE / PROJECTIVE in flags */
int sb200_points_compress(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* points, uint8_t* bytes32_out);
/* Field::random's from_bytes_wide on n 64-byte draws: field 0 -> JubJubScalar (canonical limbs),
 * field 1 -> BlsScalar (Montgomery limbs).  /root/reference/src/keys/secret.rs:83,155 */
int sb200_scalars_from_wide(sb200_ctx* ctx, int64_t n, uint32_t flags, int field, const uint8_t* wide64, uint32_t* out);
/* Position in a rand 0.8 StdRng (ChaCha12, stream 0): the 32-byte seed as 8 LE words, and the index of the next
 * unread 32-bit word of the keystream (16 x block counter + word within the block).  rand_core hands the keystream out
 * in whole words, so this is the generator's complete state.  The key determines every nonce drawn from it: it reaches
 * the device only as a kernel parameter, is never written to device memory and never appears in sb200_last_error. */
typedef struct sb200_stdrng {
  uint32_t key[8];
  uint64_t word_pos;
} sb200_stdrng;
/* n consecutive Field::random draws: out[i] = from_bytes_wide(the 16 words at word_pos + 16 i);
 * field 0 -> JubJubScalar (canonical), 1 -> BlsScalar (Montgomery).  flags: SB200_DEVICE_PTRS only.
 * On SB200_OK rng->word_pos has advanced by 16 n; on any error it is unchanged.  SB200_ERR_ARG also for a null rng
 * and for word_pos + 16 n overflowing 2^64.  Draw i belongs to tuple i however the batch is chunked or split over
 * devices.  /root/reference/src/keys/secret.rs:83,155 */
int sb200_stdrng_random(sb200_ctx* ctx, int64_t n, uint32_t flags, int field, sb200_stdrng* rng, uint32_t* out);
/* sb200_sign / _sign_double / _sign_vargen (scheme 0 / 1 / 2) with nonce i = JubJubScalar::random draw i of *rng.
 * Same outputs, bit for bit, as drawing the nonces on the host and calling the scheme's sign entry point.  flags:
 * SB200_DEVICE_PTRS, SB200_SIGN_OBLIVIOUS, and for scheme 2 SB200_POINTS_AFFINE (the layout of `generator`, which
 * only scheme 2 reads).  R_prime_out only for scheme 1.  rng->word_pos advances by 16 n on SB200_OK only.
 * Two launches: the draws into a device-only row, then the scheme's sign kernel reading its nonces from there. */
int sb200_sign_stdrng(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* sk, const uint32_t* msg,
                      const uint32_t* generator, sb200_stdrng* rng, uint32_t* u_out, uint32_t* R_out,
                      uint32_t* R_prime_out, uint32_t* c_out);
/* canonical <-> Montgomery limbs of n field elements (BlsScalar::from_bytes / to_bytes minus the range check) */
int sb200_fq_to_mont(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* in, uint32_t* out);
int sb200_fq_from_mont(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* in, uint32_t* out);
/* PublicKey::from_bytes(pk)?.verify(&Signature::from_bytes(sig)?, BlsScalar::from_bytes(msg)?) for n tuples.
 * invalid bit i = 1 where any of the three from_bytes would return Err(InvalidData); its verdict bit is 0.
 * `invalid` may be NULL. */
int sb200_verify_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk32, const uint8_t* sig64,
                       const uint8_t* msg32, uint32_t* verdicts, uint32_t* invalid);
/* SecretKey::from_bytes(sk)?.sign(nonce, BlsScalar::from_bytes(msg)?).to_bytes() for n tuples.
 * All three byte-level signers: invalid bit i = 1 where a from_bytes of the reference would return Err(InvalidData)
 * -- sk >= r, nonce >= r (JubJubScalar::from_bytes, /root/reference/src/keys/secret.rs:96-102), msg >= q, or (vargen)
 * a generator that does not decode; that tuple's signature bytes are all zero.  `invalid` may be NULL. */
int sb200_sign_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk32, const uint8_t* msg32,
                     const uint8_t* nonce32, uint8_t* sig64_out, uint32_t* invalid);

/* The same for the other two schemes:
 * pk64  = PublicKeyDouble::to_bytes = pk || pk'           /root/reference/src/keys/public.rs:282-299
 *       | PublicKeyVarGen::to_bytes = pk || generator     /root/reference/src/keys/public.rs:347-372
 * sig96 = SignatureDouble::to_bytes = u || R || R'        /root/reference/src/signatures.rs:245-270
 * sig64 = SignatureVarGen::to_bytes = u || R              /root/reference/src/signatures.rs:387-404
 * sk64  = SecretKeyVarGen::to_bytes = sk || generator     /root/reference/src/keys/secret.rs:313-336 */
int sb200_verify_double_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk64, const uint8_t* sig96,
                              const uint8_t* msg32, uint32_t* verdicts, uint32_t* invalid);
int sb200_verify_vargen_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* pk64, const uint8_t* sig64,
                              const uint8_t* msg32, uint32_t* verdicts, uint32_t* invalid);
/* SecretKey::from_bytes(sk).sign_double(nonce, msg).to_bytes() */
int sb200_sign_double_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk32, const uint8_t* msg32,
                            const uint8_t* nonce32, uint8_t* sig96_out, uint32_t* invalid);
/* SecretKeyVarGen::from_bytes(sk64)?.sign(nonce, msg).to_bytes() */
int sb200_sign_vargen_bytes(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint8_t* sk64, const uint8_t* msg32,
                            const uint8_t* nonce32, uint8_t* sig64_out, uint32_t* invalid);

/* ---- PLONK witness pre-computation (SURVEY.md 8(f)) ---------------------------------------------------------------
 * Signs n tuples like sb200_sign / _sign_double / _sign_vargen (scheme 0 / 1 / 2; `generator` only for 2, its layout
 * per SB200_POINTS_* in flags) and returns, per signature, exactly the BlsScalar values the reference's circuits
 * allocate for it -- Signature*::append (/root/reference/src/signatures.rs:97-103, 231-241, 377-383: u, R, R') and
 * gadgets::verify_signature* (/root/reference/src/gadgets.rs:48-68, 99-130, 162-184: pk, pk', generator, msg, the
 * challenge, s_a = u G, s_b = c PK) -- as rows of Montgomery field elements (8 x u32 each):
 *   scheme 0, 11 per row:  u, R.u, R.v, PK.u, PK.v, m, c, SA.u, SA.v, SB.u, SB.v
 *   scheme 1, 19 per row:  u, R, R', PK, PK', m, c, SA, SB, SA', SB'      (points as (u, v); primed = generator G')
 *   scheme 2, 13 per row:  u, R, PK, GEN, m, c, SA, SB
 * u and c are the signature's scalars embedded in F_q (`BlsScalar::from(JubJubScalar)`); SA + SB == R. */
#define SB200_WITNESS_WIDTH(scheme) ((scheme) == 0 ? 11 : (scheme) == 1 ? 19 : 13)
int sb200_sign_witness(sb200_ctx* ctx, int64_t n, uint32_t flags, int scheme, const uint32_t* sk, const uint32_t* msg,
                       const uint32_t* nonce, const uint32_t* generator, uint32_t* rows_out);

/* on-curve and Z != 0 check of n points (what SB200_CHECK_POINTS applies inside the verify calls); ok bit i = 1 if
 * point i is a well-formed curve point.  No subgroup check (the reference has none either). */
int sb200_points_check(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* points, uint32_t* ok_bitmap);

/* Building-block probes for the parity tests (same kernels' device functions, one element per thread).
 * op: 0 mul (Montgomery product), 1 add, 2 sub, 3 inverse by Fermat (b ignored), 4 square, 5 to_mont, 6 from_mont,
 * 7 inverse by the two-level Euclid of csrc/inv.cuh (what the kernels use on public data) */
int sb200_dbg_fq(sb200_ctx* ctx, int64_t n, int op, const uint32_t* a, const uint32_t* b, uint32_t* out);
/* csrc/lat3.cuh on the device: the short vector (b, a, d) of the variable-generator verification for challenges c and
 * responses u (canonical scalars).  out: 32 words per tuple = |a| (8) | |b| (8) | |d| (8) | aneg, bneg, dneg, ok, 0, 0, 0, 0 */
int sb200_dbg_lattice3(sb200_ctx* ctx, int64_t n, const uint32_t* c, const uint32_t* u, uint32_t* out);
/* canonical product a*b mod r */
int sb200_dbg_fr_mul(sb200_ctx* ctx, int64_t n, const uint32_t* a, const uint32_t* b, uint32_t* out);
/* Hades252 permutation of n states (5 field elements each, in place); dense != 0 runs the
 * reference-shaped dense partial rounds instead of the sparse factorisation. */
int sb200_dbg_hades(sb200_ctx* ctx, int64_t n, int dense, uint32_t* states);  /* dense: 0 = production form (small-integer layers when the MDS qualifies, else sparse rounds), 1 = dense (reference-shaped), 2 = FP64 pipe */
/* out[i] = k[i] * P[i] (affine); base: 0 = fixed G, 1 = fixed G', 2 = variable (points given) */
int sb200_dbg_scalar_mul(sb200_ctx* ctx, int64_t n, uint32_t flags, int base, const uint32_t* points,
                         const uint32_t* k, uint32_t* out);
/* the curve half of sb200_verify alone, with caller-supplied challenges c (n x 8 u32, any integer < 2^252): verdict
 * i = (u G + c PK == R).  Runs the curve kernel sb200_verify runs for a batch of this size (the persistent form above one
 * wave of resident CTAs, or as SB200_CURVE_PERSISTENT forces it).  Lets a test drive the half-size-scalar path and its
 * full-size fallback with chosen c. */
int sb200_dbg_verify_ec(sb200_ctx* ctx, int64_t n, uint32_t flags, const uint32_t* pk, const uint32_t* sig_u,
                        const uint32_t* sig_R, const uint32_t* c, uint32_t* verdicts);
/* the Hades tables the context derived from its parameters (rc 335, mds 25, pre 5, sparse 649, post 25 field
 * elements, in that order, 1039 x 8 u32): compared with the Python twin of the derivation in the tests */
int sb200_dbg_hades_tables(const sb200_ctx* ctx, uint32_t* out);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_H */
