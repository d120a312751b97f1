//! Batch sign / verify on B200 for dusk-schnorr (`--features cuda`).
//!
//! NOT compiled in this image (no Rust toolchain); this is the reference-side half of the C ABI in
//! `include/schnorr_b200.h`.  Marshalling copies internal limbs -- straight into page-locked, aligned buffers
//! (`Pinned`, from `sb200_host_alloc`) -- and nothing else:
//!   * `BlsScalar.0: [u64; 4]` is Montgomery (R = 2^256) little-endian  = the ABI's field element;
//!   * `JubJubExtended::{get_u, get_v, get_z}` give the projective triple = the ABI's PROJECTIVE point;
//!   * `JubJubScalar::to_bytes()` is the canonical scalar                = the ABI's scalar.
//! Verdicts / signatures are bit-exact with the single-tuple methods of the crate (src/keys/public.rs:121-130,
//! src/keys/secret.rs:150-168) at the level the crate defines equality (projective points, canonical scalars).
#![cfg(feature = "cuda")]
#![allow(non_snake_case)]

use core::ffi::{c_char, c_int, c_void};
use dusk_bls12_381::BlsScalar;
use dusk_bytes::Serializable;
use dusk_jubjub::{JubJubAffine, JubJubExtended, JubJubScalar};
use ff::Field;
use rand_core::{CryptoRng, RngCore};

use crate::{PublicKey, SecretKey, Signature};
#[cfg(feature = "double")]
use crate::{PublicKeyDouble, SignatureDouble};
#[cfg(feature = "var_generator")]
use crate::{PublicKeyVarGen, SecretKeyVarGen, SignatureVarGen};

#[repr(C)]
pub struct Sb200Ctx {
    _private: [u8; 0],
}
pub const SB200_POINTS_PROJECTIVE: u32 = 0;
pub const SB200_POINTS_AFFINE: u32 = 1;
pub const SB200_DEVICE_PTRS: u32 = 2;
/// verify calls: on-curve / Z != 0 check of every input point on the device (keys built with `from_raw_unchecked`).
pub const SB200_CHECK_POINTS: u32 = 8;
pub const SB200_ARK_CUMSUM: c_int = 0;
pub const SB200_ARK_PLAIN: c_int = 1;

/// `sb200_params` (include/schnorr_b200.h): the scheme's numeric parameters as INPUTS of context creation.  Every
/// field element is `BlsScalar.0` (Montgomery limbs) split into little-endian u32 halves, so a host with the crates
/// fills this from the crates' own tables -- nothing recalled has to be trusted.
#[repr(C)]
#[derive(Clone)]
pub struct Sb200Params {
    pub struct_size: u32,
    pub reserved: u32,
    pub generator: [u32; 16],
    pub generator_nums: [u32; 16],
    pub round_constants: [[u32; 8]; 335],
    pub mds: [[[u32; 8]; 5]; 5],
}

fn limbs(x: &BlsScalar) -> [u32; 8] {
    let mut o = [0u32; 8];
    for (i, w) in x.0.iter().enumerate() {
        o[2 * i] = *w as u32;
        o[2 * i + 1] = (*w >> 32) as u32;
    }
    o
}

impl Sb200Params {
    /// From the crates' tables: `round_constants` = dusk-hades `ROUND_CONSTANTS` (at least the first 335),
    /// `mds` = dusk-hades `MDS_MATRIX`; the generators are `dusk_jubjub::GENERATOR` / `GENERATOR_NUMS`.
    /// (If the installed dusk-hades does not export the two tables, read its `assets/ark.bin` / `assets/mds.bin`
    /// the way its `round_constants.rs` / `mds_matrix.rs` do, or use `Sb200Params::recalled` after
    /// `tests/dump_golden.rs` has shown which rule matches.)
    pub fn from_tables(round_constants: &[BlsScalar], mds: &[[BlsScalar; 5]; 5]) -> Self {
        assert!(round_constants.len() >= 335);
        let mut p = Sb200Params {
            struct_size: core::mem::size_of::<Sb200Params>() as u32,
            reserved: 0,
            generator: [0; 16],
            generator_nums: [0; 16],
            round_constants: [[0; 8]; 335],
            mds: [[[0; 8]; 5]; 5],
        };
        let put = |dst: &mut [u32; 16], a: &JubJubAffine| {
            dst[..8].copy_from_slice(&limbs(&a.get_u()));
            dst[8..].copy_from_slice(&limbs(&a.get_v()));
        };
        put(&mut p.generator, &dusk_jubjub::GENERATOR);
        put(&mut p.generator_nums, &dusk_jubjub::GENERATOR_NUMS);
        for i in 0..335 {
            p.round_constants[i] = limbs(&round_constants[i]);
        }
        for i in 0..5 {
            for j in 0..5 {
                p.mds[i][j] = limbs(&mds[i][j]);
            }
        }
        p
    }
    /// The library's recipe-derived defaults (`SB200_ARK_CUMSUM` | `SB200_ARK_PLAIN`).
    pub fn recalled(ark_rule: c_int) -> Self {
        let mut p = core::mem::MaybeUninit::<Sb200Params>::zeroed();
        let rc = unsafe { sb200_default_params(ark_rule, p.as_mut_ptr()) };
        assert_eq!(rc, 0);
        unsafe { p.assume_init() }
    }
}

/// `sb200_stdrng`: a rand 0.8 `StdRng` (= `rand_chacha::ChaCha12Rng`, stream 0) as its seed (8 little-endian words)
/// and the index of the next unread 32-bit keystream word.
#[repr(C)]
struct Sb200StdRng {
    key: [u32; 8],
    word_pos: u64,
}

#[link(name = "schnorr_b200")]
extern "C" {
    fn sb200_init(devices: *const c_int, n_devices: c_int, out: *mut *mut Sb200Ctx) -> c_int;
    fn sb200_init_ex(params: *const Sb200Params, devices: *const c_int, n_devices: c_int, out: *mut *mut Sb200Ctx) -> c_int;
    fn sb200_default_params(ark_rule: c_int, out: *mut Sb200Params) -> c_int;
    fn sb200_params_check(params: *const Sb200Params, tables_out: *mut u32) -> c_int;
    fn sb200_get_params(ctx: *const Sb200Ctx, out: *mut Sb200Params) -> c_int;
    fn sb200_points_check(ctx: *mut Sb200Ctx, n: i64, flags: u32, points: *const u32, ok_bitmap: *mut u32) -> c_int;
    fn sb200_destroy(ctx: *mut Sb200Ctx);
    fn sb200_strerror(code: c_int) -> *const c_char;
    fn sb200_last_error(ctx: *const Sb200Ctx) -> *const c_char;
    fn sb200_device_count(ctx: *const Sb200Ctx) -> c_int;
    fn sb200_set_stream(ctx: *mut Sb200Ctx, stream: *mut c_void) -> c_int;
    fn sb200_launch_count(ctx: *const Sb200Ctx) -> u64;
    fn sb200_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    fn sb200_host_free(p: *mut c_void);
    fn sb200_verify(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk: *const u32, sig_u: *const u32, sig_R: *const u32,
                    msg: *const u32, verdicts: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_verify_double(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk: *const u32, pk_prime: *const u32,
                           sig_u: *const u32, sig_R: *const u32, sig_R_prime: *const u32, msg: *const u32,
                           verdicts: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_verify_vargen(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk: *const u32, generator: *const u32,
                           sig_u: *const u32, sig_R: *const u32, msg: *const u32, verdicts: *mut u32,
                           c_out: *mut u32) -> c_int;
    fn sb200_sign(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, msg: *const u32, nonce: *const u32,
                  u_out: *mut u32, R_out: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_sign_double(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, msg: *const u32, nonce: *const u32,
                         u_out: *mut u32, R_out: *mut u32, R_prime_out: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_sign_vargen(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, generator: *const u32,
                         msg: *const u32, nonce: *const u32, u_out: *mut u32, R_out: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_sign_witness(ctx: *mut Sb200Ctx, n: i64, flags: u32, scheme: c_int, sk: *const u32, msg: *const u32,
                          nonce: *const u32, generator: *const u32, rows_out: *mut u32) -> c_int;
    fn sb200_keygen(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, pk_out: *mut u32) -> c_int;
    fn sb200_keygen_double(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, pk_out: *mut u32,
                           pk_prime_out: *mut u32) -> c_int;
    fn sb200_keygen_vargen(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk: *const u32, generator: *const u32,
                           pk_out: *mut u32) -> c_int;
    fn sb200_points_decompress(ctx: *mut Sb200Ctx, n: i64, flags: u32, bytes32: *const u8, points_out: *mut u32,
                               ok_bitmap: *mut u32) -> c_int;
    fn sb200_points_compress(ctx: *mut Sb200Ctx, n: i64, flags: u32, points: *const u32, bytes32_out: *mut u8) -> c_int;
    fn sb200_scalars_from_wide(ctx: *mut Sb200Ctx, n: i64, flags: u32, field: c_int, wide64: *const u8,
                               out: *mut u32) -> c_int;
    fn sb200_stdrng_random(ctx: *mut Sb200Ctx, n: i64, flags: u32, field: c_int, rng: *mut Sb200StdRng, out: *mut u32) -> c_int;
    fn sb200_sign_stdrng(ctx: *mut Sb200Ctx, n: i64, flags: u32, scheme: c_int, sk: *const u32, msg: *const u32,
                         generator: *const u32, rng: *mut Sb200StdRng, u_out: *mut u32, R_out: *mut u32,
                         R_prime_out: *mut u32, c_out: *mut u32) -> c_int;
    fn sb200_fq_to_mont(ctx: *mut Sb200Ctx, n: i64, flags: u32, input: *const u32, out: *mut u32) -> c_int;
    fn sb200_fq_from_mont(ctx: *mut Sb200Ctx, n: i64, flags: u32, input: *const u32, out: *mut u32) -> c_int;
    fn sb200_verify_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk32: *const u8, sig64: *const u8, msg32: *const u8,
                          verdicts: *mut u32, invalid: *mut u32) -> c_int;
    fn sb200_sign_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk32: *const u8, msg32: *const u8, nonce32: *const u8,
                        sig64_out: *mut u8, invalid: *mut u32) -> c_int;
    // the double-key and variable-generator schemes in their `Serializable` forms
    // (pk64 = pk || pk' | pk || generator; sig96 = u || R || R'; sk64 = sk || generator)
    fn sb200_verify_double_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk64: *const u8, sig96: *const u8,
                                 msg32: *const u8, verdicts: *mut u32, invalid: *mut u32) -> c_int;
    fn sb200_verify_vargen_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, pk64: *const u8, sig64: *const u8,
                                 msg32: *const u8, verdicts: *mut u32, invalid: *mut u32) -> c_int;
    fn sb200_sign_double_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk32: *const u8, msg32: *const u8,
                               nonce32: *const u8, sig96_out: *mut u8, invalid: *mut u32) -> c_int;
    fn sb200_sign_vargen_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, sk64: *const u8, msg32: *const u8,
                               nonce32: *const u8, sig64_out: *mut u8, invalid: *mut u32) -> c_int;
    // include/schnorr_b200_witness.h: witness rows of received signatures (pk2 = PK' | generator, sig_R_prime: double only)
    fn sb200_verify_witness(ctx: *mut Sb200Ctx, n: i64, flags: u32, scheme: c_int, pk: *const u32, pk2: *const u32,
                            sig_u: *const u32, sig_R: *const u32, sig_R_prime: *const u32, msg: *const u32,
                            verdicts: *mut u32, rows_out: *mut u32) -> c_int;
    fn sb200_verify_witness_bytes(ctx: *mut Sb200Ctx, n: i64, flags: u32, scheme: c_int, pk_bytes: *const u8,
                                  sig_bytes: *const u8, msg32: *const u8, verdicts: *mut u32, rows_out: *mut u32,
                                  invalid: *mut u32) -> c_int;
}

/// Owns one `sb200_ctx` (comb tables of G and G' resident on each listed device).  There is no CPU
/// fallback: `new` fails without a B200.
pub struct CudaCtx {
    raw: *mut Sb200Ctx,
}
unsafe impl Send for CudaCtx {}
unsafe impl Sync for CudaCtx {} // calls on one context are serialised inside the library

#[derive(Debug)]
pub struct CudaError(pub i32, pub String);

impl CudaCtx {
    /// Default (recalled) parameters; see `with_params` for the crate's own tables.
    pub fn new(devices: &[i32]) -> Result<Self, CudaError> {
        let mut raw = core::ptr::null_mut();
        let rc = unsafe { sb200_init(devices.as_ptr(), devices.len() as c_int, &mut raw) };
        if rc != 0 {
            return Err(CudaError(rc, cstr(unsafe { sb200_strerror(rc) })));
        }
        Ok(Self { raw })
    }
    /// Context over caller-supplied parameters (`Sb200Params::from_tables` with the crates' tables).  The library
    /// validates them (generators on the curve and of prime order, canonical field elements, invertible MDS blocks)
    /// and checks its derived sparse Hades form against the dense permutation before anything runs.
    pub fn with_params(params: &Sb200Params, devices: &[i32]) -> Result<Self, CudaError> {
        let mut raw = core::ptr::null_mut();
        let rc = unsafe { sb200_init_ex(params, devices.as_ptr(), devices.len() as c_int, &mut raw) };
        if rc != 0 {
            return Err(CudaError(rc, cstr(unsafe { sb200_strerror(rc) })));
        }
        Ok(Self { raw })
    }
    fn check(&self, rc: c_int) -> Result<(), CudaError> {
        if rc == 0 { Ok(()) } else { Err(CudaError(rc, cstr(unsafe { sb200_last_error(self.raw) }))) }
    }
}
impl Drop for CudaCtx {
    fn drop(&mut self) {
        unsafe { sb200_destroy(self.raw) }
    }
}
fn cstr(p: *const c_char) -> String {
    unsafe { std::ffi::CStr::from_ptr(p) }.to_string_lossy().into_owned()
}

// ---- marshalling: copies of internal limbs, straight into page-locked memory ------------------------------------
/// A `Vec<u32>`-like buffer in memory from `sb200_host_alloc`: page-locked (the library copies it to the device
/// without staging) and aligned far beyond the ABI's 16-byte requirement (a plain `Vec<u32>` guarantees 4).
pub struct Pinned<T: Copy> {
    ptr: *mut T,
    len: usize,
    cap: usize,
}
impl<T: Copy> Pinned<T> {
    pub fn with_capacity(cap: usize) -> Self {
        let mut p: *mut c_void = core::ptr::null_mut();
        let rc = unsafe { sb200_host_alloc(core::cmp::max(cap, 1) * core::mem::size_of::<T>(), &mut p) };
        assert_eq!(rc, 0, "sb200_host_alloc failed");
        Pinned { ptr: p as *mut T, len: 0, cap }
    }
    pub fn zeroed(len: usize) -> Self {
        let mut b = Self::with_capacity(len);
        unsafe { core::ptr::write_bytes(b.ptr, 0, len) };
        b.len = len;
        b
    }
    pub fn from_slice(src: &[T]) -> Self {
        let mut b = Self::with_capacity(src.len());
        unsafe { core::ptr::copy_nonoverlapping(src.as_ptr(), b.ptr, src.len()) };
        b.len = src.len();
        b
    }
    pub fn push(&mut self, x: T) {
        assert!(self.len < self.cap);
        unsafe { self.ptr.add(self.len).write(x) };
        self.len += 1;
    }
    pub fn as_ptr(&self) -> *const T { self.ptr }
    pub fn as_mut_ptr(&mut self) -> *mut T { self.ptr }
    pub fn as_slice(&self) -> &[T] { unsafe { core::slice::from_raw_parts(self.ptr, self.len) } }
}
impl<T: Copy> Drop for Pinned<T> {
    fn drop(&mut self) { unsafe { sb200_host_free(self.ptr as *mut c_void) } }
}
impl<T: Copy> core::ops::Index<core::ops::Range<usize>> for Pinned<T> {
    type Output = [T];
    fn index(&self, r: core::ops::Range<usize>) -> &[T] { &self.as_slice()[r] }
}
impl<T: Copy> core::ops::Index<usize> for Pinned<T> {
    type Output = T;
    fn index(&self, i: usize) -> &T { &self.as_slice()[i] }
}
type Vec32 = Pinned<u32>;

fn push_fq(v: &mut Vec32, x: &BlsScalar) {
    for w in x.0 {
        v.push(w as u32);
        v.push((w >> 32) as u32);
    }
}
fn push_point(v: &mut Vec32, p: &JubJubExtended) {
    push_fq(v, &p.get_u());
    push_fq(v, &p.get_v());
    push_fq(v, &p.get_z());
}
fn push_scalar(v: &mut Vec32, s: &JubJubScalar) {
    for c in s.to_bytes().chunks_exact(4) {
        v.push(u32::from_le_bytes([c[0], c[1], c[2], c[3]]));
    }
}
fn fq_at(a: &Vec32, i: usize) -> BlsScalar {
    let w = &a[8 * i..8 * i + 8];
    BlsScalar([
        w[0] as u64 | (w[1] as u64) << 32,
        w[2] as u64 | (w[3] as u64) << 32,
        w[4] as u64 | (w[5] as u64) << 32,
        w[6] as u64 | (w[7] as u64) << 32,
    ])
}
fn point_at(a: &Vec32, i: usize) -> JubJubExtended {
    JubJubAffine::from_raw_unchecked(fq_at(a, 2 * i), fq_at(a, 2 * i + 1)).into()
}
fn scalar_at(a: &Vec32, i: usize) -> JubJubScalar {
    let mut b = [0u8; 32];
    for (k, w) in a[8 * i..8 * i + 8].iter().enumerate() {
        b[4 * k..4 * k + 4].copy_from_slice(&w.to_le_bytes());
    }
    JubJubScalar::from_bytes(&b).expect("the library returns canonical scalars")
}
fn bits(words: &Vec32, n: usize) -> Vec<bool> {
    (0..n).map(|i| (words[i >> 5] >> (i & 31)) & 1 == 1).collect()
}
fn witness_rows<const W: usize>(rows: &Vec32, n: usize) -> Vec<[BlsScalar; W]> {
    (0..n).map(|i| {
        let mut w = [BlsScalar::zero(); W];
        for (k, x) in w.iter_mut().enumerate() { *x = fq_at(rows, W * i + k); }
        w
    }).collect()
}

impl PublicKey {
    /// `out[i] == pks[i].verify(&sigs[i], msgs[i])` (src/keys/public.rs:121-130) for every i.
    pub fn verify_batch(ctx: &CudaCtx, pks: &[PublicKey], sigs: &[Signature], msgs: &[BlsScalar]) -> Result<Vec<bool>, CudaError> {
        let n = pks.len();
        assert!(sigs.len() == n && msgs.len() == n);
        let (mut pk, mut u, mut r, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].as_ref());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_fq(&mut m, &msgs[i]);
        }
        let mut words = Vec32::zeroed((n + 31) / 32);
        ctx.check(unsafe {
            sb200_verify(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, pk.as_ptr(), u.as_ptr(), r.as_ptr(), m.as_ptr(),
                         words.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok(bits(&words, n))
    }

    /// Verifier-side counterpart of `SecretKey::sign_batch_witness`: for signatures the caller received rather than made,
    /// `verify_batch`'s verdicts together with the rows `u, R.u, R.v, PK.u, PK.v, m, c, SA.u, SA.v, SB.u, SB.v` that
    /// `Signature::append` and `gadgets::verify_signature` allocate, SA = u G and SB = c PK computed on the device
    /// (`sb200_verify_witness`).  A signature that fails keeps its true row; the row of a signature made by
    /// `sign_batch_witness` equals the signer's.
    pub fn verify_batch_witness(ctx: &CudaCtx, pks: &[PublicKey], sigs: &[Signature], msgs: &[BlsScalar])
                                -> Result<(Vec<bool>, Vec<[BlsScalar; 11]>), CudaError> {
        let n = pks.len();
        assert!(sigs.len() == n && msgs.len() == n);
        let (mut pk, mut u, mut r, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].as_ref());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_fq(&mut m, &msgs[i]);
        }
        let (mut words, mut rows) = (Vec32::zeroed((n + 31) / 32), Vec32::zeroed(8 * 11 * n));
        ctx.check(unsafe {
            sb200_verify_witness(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, 0, pk.as_ptr(), core::ptr::null(), u.as_ptr(),
                                 r.as_ptr(), core::ptr::null(), m.as_ptr(), words.as_mut_ptr(), rows.as_mut_ptr())
        })?;
        Ok((bits(&words, n), witness_rows::<11>(&rows, n)))
    }

    /// Byte-level form: `PublicKey::from_bytes(pk)?.verify(&Signature::from_bytes(sig)?, BlsScalar::from_bytes(msg)?)`;
    /// returns (verdicts, invalid) where `invalid[i]` marks tuples whose decoding would be `Err(InvalidData)`.
    pub fn verify_bytes_batch(ctx: &CudaCtx, pk32: &[[u8; 32]], sig64: &[[u8; 64]], msg32: &[[u8; 32]]) -> Result<(Vec<bool>, Vec<bool>), CudaError> {
        let n = pk32.len();
        let (mut v, mut inv) = (Vec32::zeroed((n + 31) / 32), Vec32::zeroed((n + 31) / 32));
        // `&[[u8; 32]]` has alignment 1: copy into aligned, page-locked buffers (the ABI wants 16-byte alignment)
        let (pk32, sig64, msg32) = (Pinned::from_slice(pk32), Pinned::from_slice(sig64), Pinned::from_slice(msg32));
        ctx.check(unsafe {
            sb200_verify_bytes(ctx.raw, n as i64, 0, pk32.as_ptr() as *const u8, sig64.as_ptr() as *const u8,
                               msg32.as_ptr() as *const u8, v.as_mut_ptr(), inv.as_mut_ptr())
        })?;
        Ok((bits(&v, n), bits(&inv, n)))
    }

    /// `PublicKey::from(&sk)` for every key (src/keys/public.rs:61-67).
    pub fn from_secret_keys(ctx: &CudaCtx, sks: &[SecretKey]) -> Result<Vec<PublicKey>, CudaError> {
        let n = sks.len();
        let mut k = Vec32::with_capacity(8 * n);
        sks.iter().for_each(|s| push_scalar(&mut k, s.as_ref()));
        let mut out = Vec32::zeroed(16 * n);
        ctx.check(unsafe { sb200_keygen(ctx.raw, n as i64, 0, k.as_ptr(), out.as_mut_ptr()) })?;
        Ok((0..n).map(|i| PublicKey::from(point_at(&out, i))).collect())
    }
}

impl SecretKey {
    /// Batch form of `sign` (src/keys/secret.rs:150-168).  Signature i consumes the rng's i-th
    /// `JubJubScalar::random` draw, in order, exactly like n consecutive `sign` calls.
    pub fn sign_batch<R: RngCore + CryptoRng>(ctx: &CudaCtx, sks: &[SecretKey], rng: &mut R, msgs: &[BlsScalar]) -> Result<Vec<Signature>, CudaError> {
        let n = sks.len();
        let (mut sk, mut m, mut nonce) = (Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_scalar(&mut sk, sks[i].as_ref());
            push_fq(&mut m, &msgs[i]);
            push_scalar(&mut nonce, &JubJubScalar::random(&mut *rng));
        }
        let (mut u, mut r) = (Vec32::zeroed(8 * n), Vec32::zeroed(16 * n));
        ctx.check(unsafe {
            sb200_sign(ctx.raw, n as i64, 0, sk.as_ptr(), m.as_ptr(), nonce.as_ptr(), u.as_mut_ptr(), r.as_mut_ptr(),
                       core::ptr::null_mut())
        })?;
        Ok((0..n).map(|i| Signature::new(scalar_at(&u, i), point_at(&r, i))).collect())
    }

    /// `sign_batch` over the generator rand 0.8's `StdRng` wraps (`rand_chacha::ChaCha12Rng`): the nonces are drawn on the
    /// device from the generator's seed and word position (`sb200_sign_stdrng`) instead of on the host, and the generator
    /// is moved past them -- it ends exactly where n `JubJubScalar::random` draws would have left it, and the signatures
    /// are the same.  A generic `RngCore` exposes no position; it keeps `sign_batch`, and so does a `ChaCha12Rng` on a
    /// stream other than 0 or past 2^64 words (the library's positions are 64-bit).  Uncompiled, like the rest of this
    /// file: the four `ChaCha12Rng` methods are rand_chacha 0.3's as recalled.
    pub fn sign_batch_chacha12(ctx: &CudaCtx, sks: &[SecretKey], rng: &mut rand_chacha::ChaCha12Rng, msgs: &[BlsScalar])
                               -> Result<Vec<Signature>, CudaError> {
        let n = sks.len();
        assert!(msgs.len() == n);
        // the library expands stream 0 at 64-bit word positions; any other generator state keeps the host draw
        let word_pos = match u64::try_from(rng.get_word_pos()) {
            Ok(w) if rng.get_stream() == 0 => w,
            _ => return Self::sign_batch(ctx, sks, rng, msgs),
        };
        let seed = rng.get_seed();
        let mut pos = Sb200StdRng { key: [0u32; 8], word_pos: 0 };
        for i in 0..8 {
            pos.key[i] = u32::from_le_bytes([seed[4 * i], seed[4 * i + 1], seed[4 * i + 2], seed[4 * i + 3]]);
        }
        pos.word_pos = word_pos;
        let (mut sk, mut m) = (Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_scalar(&mut sk, sks[i].as_ref());
            push_fq(&mut m, &msgs[i]);
        }
        let (mut u, mut r) = (Vec32::zeroed(8 * n), Vec32::zeroed(16 * n));
        ctx.check(unsafe {
            sb200_sign_stdrng(ctx.raw, n as i64, 0, 0, sk.as_ptr(), m.as_ptr(), core::ptr::null(), &mut pos, u.as_mut_ptr(),
                              r.as_mut_ptr(), core::ptr::null_mut(), core::ptr::null_mut())
        })?;
        rng.set_word_pos(pos.word_pos as u128);
        Ok((0..n).map(|i| Signature::new(scalar_at(&u, i), point_at(&r, i))).collect())
    }

    /// Batch signing that also returns, per signature, the BlsScalar values `Signature::append` (src/signatures.rs:97-103) and
    /// `gadgets::verify_signature` (src/gadgets.rs:48-68) allocate as witnesses: one row of 11 field elements
    /// `u, R.u, R.v, PK.u, PK.v, m, c, SA.u, SA.v, SB.u, SB.v` (SA = u G, SB = c PK, SA + SB = R), computed on the device next to
    /// the signature so that the prover does not repeat the two scalar multiplications on the CPU.
    pub fn sign_batch_witness<R: RngCore + CryptoRng>(ctx: &CudaCtx, sks: &[SecretKey], rng: &mut R, msgs: &[BlsScalar])
                                                      -> Result<Vec<(Signature, [BlsScalar; 11])>, CudaError> {
        let n = sks.len();
        let (mut sk, mut m, mut nonce) = (Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_scalar(&mut sk, sks[i].as_ref());
            push_fq(&mut m, &msgs[i]);
            push_scalar(&mut nonce, &JubJubScalar::random(&mut *rng));
        }
        let mut rows = Vec32::zeroed(8 * 11 * n);
        ctx.check(unsafe {
            sb200_sign_witness(ctx.raw, n as i64, 0, 0, sk.as_ptr(), m.as_ptr(), nonce.as_ptr(), core::ptr::null(), rows.as_mut_ptr())
        })?;
        Ok((0..n).map(|i| {
            let mut w = [BlsScalar::zero(); 11];
            for (k, x) in w.iter_mut().enumerate() { *x = fq_at(&rows, 11 * i + k); }
            // u as a JubJubScalar: the row holds its embedding in F_q (`BlsScalar::from(JubJubScalar)`), i.e. the same integer
            let u = JubJubScalar::from_bytes(&w[0].to_bytes()).expect("u < r");
            let r = JubJubExtended::from(JubJubAffine::from_raw_unchecked(w[1], w[2]));
            (Signature::new(u, r), w)
        }).collect())
    }

    #[cfg(feature = "double")]
    pub fn sign_double_batch<R: RngCore + CryptoRng>(ctx: &CudaCtx, sks: &[SecretKey], rng: &mut R, msgs: &[BlsScalar]) -> Result<Vec<SignatureDouble>, CudaError> {
        let n = sks.len();
        let (mut sk, mut m, mut nonce) = (Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_scalar(&mut sk, sks[i].as_ref());
            push_fq(&mut m, &msgs[i]);
            push_scalar(&mut nonce, &JubJubScalar::random(&mut *rng));
        }
        let (mut u, mut r, mut rp) = (Vec32::zeroed(8 * n), Vec32::zeroed(16 * n), Vec32::zeroed(16 * n));
        ctx.check(unsafe {
            sb200_sign_double(ctx.raw, n as i64, 0, sk.as_ptr(), m.as_ptr(), nonce.as_ptr(), u.as_mut_ptr(),
                              r.as_mut_ptr(), rp.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok((0..n).map(|i| SignatureDouble::new(scalar_at(&u, i), point_at(&r, i), point_at(&rp, i))).collect())
    }
}

#[cfg(feature = "double")]
impl PublicKeyDouble {
    /// Batch form of `verify` (src/keys/public.rs:222-244).
    pub fn verify_batch(ctx: &CudaCtx, pks: &[PublicKeyDouble], sigs: &[SignatureDouble], msgs: &[BlsScalar]) -> Result<Vec<bool>, CudaError> {
        let n = pks.len();
        let (mut pk, mut pkp, mut u, mut r, mut rp, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n),
                                                              Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].pk());
            push_point(&mut pkp, pks[i].pk_prime());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_point(&mut rp, sigs[i].R_prime());
            push_fq(&mut m, &msgs[i]);
        }
        let mut words = Vec32::zeroed((n + 31) / 32);
        ctx.check(unsafe {
            sb200_verify_double(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, pk.as_ptr(), pkp.as_ptr(), u.as_ptr(),
                                r.as_ptr(), rp.as_ptr(), m.as_ptr(), words.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok(bits(&words, n))
    }

    /// `verify_batch` with the witness rows of each signature (`sb200_verify_witness`, scheme 1):
    /// `u, R, R', PK, PK', m, c, SA, SB, SA', SB'` (points as (u, v); SA' = u G', SB' = c PK').
    pub fn verify_batch_witness(ctx: &CudaCtx, pks: &[PublicKeyDouble], sigs: &[SignatureDouble], msgs: &[BlsScalar])
                                -> Result<(Vec<bool>, Vec<[BlsScalar; 19]>), CudaError> {
        let n = pks.len();
        assert!(sigs.len() == n && msgs.len() == n);
        let (mut pk, mut pkp, mut u, mut r, mut rp, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n),
                                                              Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].pk());
            push_point(&mut pkp, pks[i].pk_prime());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_point(&mut rp, sigs[i].R_prime());
            push_fq(&mut m, &msgs[i]);
        }
        let (mut words, mut rows) = (Vec32::zeroed((n + 31) / 32), Vec32::zeroed(8 * 19 * n));
        ctx.check(unsafe {
            sb200_verify_witness(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, 1, pk.as_ptr(), pkp.as_ptr(), u.as_ptr(),
                                 r.as_ptr(), rp.as_ptr(), m.as_ptr(), words.as_mut_ptr(), rows.as_mut_ptr())
        })?;
        Ok((bits(&words, n), witness_rows::<19>(&rows, n)))
    }
}

#[cfg(feature = "var_generator")]
impl PublicKeyVarGen {
    /// Batch form of `verify` (src/keys/public.rs:401-415).
    pub fn verify_batch(ctx: &CudaCtx, pks: &[PublicKeyVarGen], sigs: &[SignatureVarGen], msgs: &[BlsScalar]) -> Result<Vec<bool>, CudaError> {
        let n = pks.len();
        let (mut pk, mut g, mut u, mut r, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n),
                                                    Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].public_key());
            push_point(&mut g, pks[i].generator());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_fq(&mut m, &msgs[i]);
        }
        let mut words = Vec32::zeroed((n + 31) / 32);
        ctx.check(unsafe {
            sb200_verify_vargen(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, pk.as_ptr(), g.as_ptr(), u.as_ptr(),
                                r.as_ptr(), m.as_ptr(), words.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok(bits(&words, n))
    }

    /// `verify_batch` with the witness rows of each signature (`sb200_verify_witness`, scheme 2):
    /// `u, R, PK, GEN, m, c, SA, SB` (points as (u, v); SA = u GEN).
    pub fn verify_batch_witness(ctx: &CudaCtx, pks: &[PublicKeyVarGen], sigs: &[SignatureVarGen], msgs: &[BlsScalar])
                                -> Result<(Vec<bool>, Vec<[BlsScalar; 13]>), CudaError> {
        let n = pks.len();
        assert!(sigs.len() == n && msgs.len() == n);
        let (mut pk, mut g, mut u, mut r, mut m) = (Vec32::with_capacity(24 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n),
                                                    Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_point(&mut pk, pks[i].public_key());
            push_point(&mut g, pks[i].generator());
            push_scalar(&mut u, sigs[i].u());
            push_point(&mut r, sigs[i].R());
            push_fq(&mut m, &msgs[i]);
        }
        let (mut words, mut rows) = (Vec32::zeroed((n + 31) / 32), Vec32::zeroed(8 * 13 * n));
        ctx.check(unsafe {
            sb200_verify_witness(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, 2, pk.as_ptr(), g.as_ptr(), u.as_ptr(),
                                 r.as_ptr(), core::ptr::null(), m.as_ptr(), words.as_mut_ptr(), rows.as_mut_ptr())
        })?;
        Ok((bits(&words, n), witness_rows::<13>(&rows, n)))
    }
}

#[cfg(feature = "var_generator")]
impl SecretKeyVarGen {
    /// Batch form of `sign` (src/keys/secret.rs:433-451).
    pub fn sign_batch<R: RngCore + CryptoRng>(ctx: &CudaCtx, sks: &[SecretKeyVarGen], rng: &mut R, msgs: &[BlsScalar]) -> Result<Vec<SignatureVarGen>, CudaError> {
        let n = sks.len();
        let (mut sk, mut g, mut m, mut nonce) = (Vec32::with_capacity(8 * n), Vec32::with_capacity(24 * n), Vec32::with_capacity(8 * n), Vec32::with_capacity(8 * n));
        for i in 0..n {
            push_scalar(&mut sk, sks[i].secret_key());
            push_point(&mut g, sks[i].generator());
            push_fq(&mut m, &msgs[i]);
            push_scalar(&mut nonce, &JubJubScalar::random(&mut *rng));
        }
        let (mut u, mut r) = (Vec32::zeroed(8 * n), Vec32::zeroed(16 * n));
        ctx.check(unsafe {
            sb200_sign_vargen(ctx.raw, n as i64, SB200_POINTS_PROJECTIVE, sk.as_ptr(), g.as_ptr(), m.as_ptr(),
                              nonce.as_ptr(), u.as_mut_ptr(), r.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok((0..n).map(|i| SignatureVarGen::new(scalar_at(&u, i), point_at(&r, i))).collect())
    }
}
