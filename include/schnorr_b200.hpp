// schnorr_b200.hpp -- C++ host-side mirror of dusk-schnorr's public API on top of the C ABI.
//
// The reference is compiled code (Rust); its toolchain is not in this image, so the reference-facing host
// layer is written in C++ with the reference's type names, method names, argument meaning and error
// behaviour.  Header-only; link with -lschnorr_b200.  Everything arithmetic happens on the GPU through
// include/schnorr_b200.h (single calls are batches of one); the host only moves bytes and keeps the RNG state,
// exactly the split the reference has between `dusk-schnorr` and its arithmetic crates.  The batch signers hand the
// RNG's position to the device, which draws the nonces (sb200_sign_stdrng) and returns the advanced position.
//
//   SecretKey        /root/reference/src/keys/secret.rs:56-263      random, sign, sign_double, with_variable_generator, to/from_bytes
//   SecretKeyVarGen  /root/reference/src/keys/secret.rs:307-451     new, random, sign, to/from_bytes
//   PublicKey        /root/reference/src/keys/public.rs:59-145      from(&SecretKey), verify, from_raw_unchecked, to/from_bytes
//   PublicKeyDouble  /root/reference/src/keys/public.rs:189-299
//   PublicKeyVarGen  /root/reference/src/keys/public.rs:331-433
//   Signature, SignatureDouble, SignatureVarGen   /root/reference/src/signatures.rs:58-404
//   StdRng = rand 0.8 StdRng (ChaCha12), the RNG the reference's tests seed (/root/reference/tests/schnorr.rs:16)
//
// Error behaviour: `from_bytes` throws BytesError{InvalidData} where the reference returns
// Err(dusk_bytes::Error::InvalidData) (non-canonical scalar, bytes that are not a curve point) and
// BytesError{BadLength} for a wrong size; `verify` returns bool and never throws on bad signatures.
// New relative to the reference: the `*_batch` static methods.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "schnorr_b200.h"

namespace dusk_schnorr {

struct BytesError : std::runtime_error {
  enum Kind { InvalidData, BadLength } kind;
  explicit BytesError(Kind k) : std::runtime_error(k == InvalidData ? "InvalidData" : "BadLength"), kind(k) {}
};
struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

// Aligned host vector for the ABI's arrays.  Small ones (single-tuple calls) are ordinary 64-byte aligned heap
// memory, which the library stages through its pinned ring; batch-sized ones come from sb200_host_alloc (page-locked:
// copied to and from the device directly, no staging pass) and are recycled through a per-thread pool, because
// pinning memory costs far more than the batch's arithmetic.
template <class T>
struct avec {
  T* p = nullptr;
  size_t n = 0;
  bool pinned = false;
  static constexpr size_t PIN_BYTES = 1 << 16;
  struct Pool {
    std::vector<std::pair<void*, size_t>> free_list;
    ~Pool() { for (auto& e : free_list) sb200_host_free(e.first); }
  };
  static Pool& pool() { thread_local Pool pl; return pl; }
  explicit avec(size_t count) : n(count) {
    const size_t bytes = count * sizeof(T);
    if (bytes >= PIN_BYTES) {
      auto& fl = pool().free_list;
      size_t best = fl.size();
      for (size_t i = 0; i < fl.size(); i++)
        if (fl[i].second >= bytes && (best == fl.size() || fl[i].second < fl[best].second)) best = i;
      if (best != fl.size()) {
        p = static_cast<T*>(fl[best].first); cap_ = fl[best].second;
        fl.erase(fl.begin() + best);
        pinned = true;
      } else {
        void* q = nullptr;
        if (sb200_host_alloc(bytes, &q) == SB200_OK) { p = static_cast<T*>(q); cap_ = bytes; pinned = true; }
      }
    }
    if (!p && count) {
      p = static_cast<T*>(::operator new[](bytes, std::align_val_t(64)));
      std::memset(p, 0, bytes);
    }
  }
  ~avec() {
    if (pinned) pool().free_list.emplace_back(p, cap_);
    else ::operator delete[](p, std::align_val_t(64));
  }
  avec(const avec&) = delete;
  avec& operator=(const avec&) = delete;
  T* data() { return p; }
  T& operator[](size_t i) { return p[i]; }

 private:
  size_t cap_ = 0;
};

namespace detail {
// marshalling loops of the batch calls: split over the host's cores once a batch is large enough to pay for threads
template <class F>
inline void parallel_for(size_t n, F&& f) {
  unsigned hw = std::thread::hardware_concurrency();
  size_t nt = n < (1u << 14) ? 1 : std::min<size_t>(hw ? hw : 1, 16);
  if (nt <= 1) { f(0, n); return; }
  std::vector<std::thread> th;
  size_t per = (n + nt - 1) / nt;
  for (size_t t = 1; t < nt; t++) {
    size_t lo = std::min(n, t * per), hi = std::min(n, lo + per);
    if (lo < hi) th.emplace_back([&f, lo, hi] { f(lo, hi); });
  }
  f(0, std::min(n, per));
  for (auto& x : th) x.join();
}
}  // namespace detail

// One engine per process by default (device 0); there is no CPU fallback: construction throws without a GPU.
class Context {
 public:
  explicit Context(std::vector<int> devices = {0}) {
    int rc = sb200_init(devices.data(), (int)devices.size(), &ctx_);
    if (rc != SB200_OK) throw CudaError(std::string("sb200_init: ") + sb200_strerror(rc) + " (no CPU fallback)");
  }
  ~Context() { sb200_destroy(ctx_); }
  Context(const Context&) = delete;
  sb200_ctx* raw() const { return ctx_; }
  void check(int rc, const char* what) const {
    if (rc != SB200_OK) throw CudaError(std::string(what) + ": " + sb200_strerror(rc) + " " + sb200_last_error(ctx_));
  }
  static Context& global() {
    static Context c;
    return c;
  }

 private:
  sb200_ctx* ctx_ = nullptr;
};

using Bytes32 = std::array<uint8_t, 32>;

// rand 0.8 `StdRng`: ChaCha12, 64-bit block counter, words consumed in order, little-endian.
class StdRng {
 public:
  explicit StdRng(const std::array<uint8_t, 32>& seed) { std::memcpy(key_, seed.data(), 32); }
  static StdRng seed_from_u64(uint64_t state) {  // rand_core 0.6 SeedableRng::seed_from_u64 (PCG32 expansion)
    std::array<uint8_t, 32> seed{};
    for (int i = 0; i < 8; i++) {
      state = state * 6364136223846793005ULL + 11634580027462260723ULL;
      uint32_t xs = (uint32_t)(((state >> 18) ^ state) >> 27), rot = (uint32_t)(state >> 59);
      uint32_t x = (xs >> rot) | (xs << ((32 - rot) & 31));
      std::memcpy(seed.data() + 4 * i, &x, 4);
    }
    return StdRng(seed);
  }
  void fill_bytes(uint8_t* out, size_t n) {
    size_t i = 0;
    for (; i < n && pos_ != 64; i++) out[i] = buf_[pos_++];  // drain the current block
    // whole blocks: ChaCha is seekable (block k depends on the key and k only), so a bulk draw -- the nonces of a
    // batch -- is computed in parallel and still equals the sequential stream byte for byte
    const size_t blocks = (n - i) / 64;
    if (blocks) {
      const uint64_t first = block_;
      uint8_t* dst = out + i;
      detail::parallel_for(blocks, [&](size_t lo, size_t hi) {
        for (size_t b = lo; b < hi; b++) block(first + b, dst + 64 * b);
      });
      block_ += blocks;
      i += 64 * blocks;
    }
    for (; i < n; i++) {
      if (pos_ == 64) refill();
      out[i] = buf_[pos_++];
    }
  }
  uint64_t next_u64() {
    uint8_t b[8];
    fill_bytes(b, 8);
    uint64_t v;
    std::memcpy(&v, b, 8);
    return v;
  }
  // Position of the next unread 32-bit keystream word (16 x block + word within the block), rand_chacha's get_word_pos.
  // Meaningful on a word boundary only: every draw of this API is 8 or 64 bytes, so only a caller's own fill_bytes
  // of a length that is not a multiple of 4 leaves the stream inside a word.
  bool on_word_boundary() const { return pos_ % 4 == 0; }
  uint64_t word_pos() const { return 16 * block_ - (64 - pos_) / 4; }
  // continue the stream at keystream word `w` (rand_chacha's set_word_pos)
  void seek(uint64_t w) {
    block_ = w / 16;
    pos_ = 64;
    if (w % 16) {
      refill();
      pos_ = 4 * (size_t)(w % 16);
    }
  }
  // the device-side generator's view of this stream: seed and current word position
  sb200_stdrng position() const {
    sb200_stdrng p;
    std::memcpy(p.key, key_, 32);
    p.word_pos = word_pos();
    return p;
  }

 private:
  static uint32_t rotl(uint32_t v, int n) { return (v << n) | (v >> (32 - n)); }
  void refill() {
    block(block_, buf_);
    block_++;
    pos_ = 0;
  }
  void block(uint64_t counter, uint8_t* out64) const {
    uint32_t st[16] = {0x61707865, 0x3320646e, 0x79622d32, 0x6b206574};
    std::memcpy(st + 4, key_, 32);
    st[12] = (uint32_t)counter; st[13] = (uint32_t)(counter >> 32); st[14] = st[15] = 0;
    uint32_t x[16];
    std::memcpy(x, st, 64);
    auto qr = [&](int a, int b, int c, int d) {
      x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16); x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12);
      x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8);  x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7);
    };
    for (int r = 0; r < 6; r++) {
      qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15);
      qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14);
    }
    for (int i = 0; i < 16; i++) x[i] += st[i];
    std::memcpy(out64, x, 64);
  }
  uint32_t key_[8];
  uint64_t block_ = 0;
  uint8_t buf_[64];
  size_t pos_ = 64;
};

namespace detail {
// nonce i of a batch signer = the i-th JubJubScalar::random draw of rng.  On a word boundary the device draws them
// from the stream's position (sb200_sign_stdrng), and the stream is moved to where the host draws would have left it;
// otherwise the host draws them.  Returns false when the caller must sign with host-drawn nonces.
inline bool sign_stdrng(StdRng& rng, int scheme, size_t n, uint32_t flags, const uint32_t* sk, const uint32_t* msg,
                        const uint32_t* gen, uint32_t* u, uint32_t* R, uint32_t* Rp) {
  if (!rng.on_word_boundary()) return false;
  sb200_stdrng pos = rng.position();
  Context& c = Context::global();
  c.check(sb200_sign_stdrng(c.raw(), (int64_t)n, flags, scheme, sk, msg, gen, &pos, u, R, Rp, nullptr), "sign_stdrng");
  rng.seek(pos.word_pos);
  return true;
}
inline void wide_draws(StdRng& rng, size_t n, int field, uint32_t* out /* n x 8 */) {
  avec<uint8_t> w(64 * n);
  rng.fill_bytes(w.data(), 64 * n);
  Context& c = Context::global();
  c.check(sb200_scalars_from_wide(c.raw(), (int64_t)n, 0, field, w.data(), out), "scalars_from_wide");
}
}  // namespace detail

// dusk_bls12_381::BlsScalar: 8 x u32 Montgomery limbs (bit-identical to the crate's [u64; 4])
struct BlsScalar {
  uint32_t l[8] = {};
  static BlsScalar random(StdRng& rng) {  // ff::Field::random = from_bytes_wide(64 rng bytes)
    avec<uint32_t> o(8);
    detail::wide_draws(rng, 1, 1, o.data());
    BlsScalar s;
    std::memcpy(s.l, o.data(), 32);
    return s;
  }
  static BlsScalar from_bytes(const Bytes32& b) {  // rejects >= q
    static const uint32_t q[8] = {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
    uint32_t w[8];
    std::memcpy(w, b.data(), 32);
    bool lt = false;
    for (int i = 7; i >= 0; i--) {
      if (w[i] != q[i]) { lt = w[i] < q[i]; break; }
    }
    if (!lt) throw BytesError(BytesError::InvalidData);
    avec<uint32_t> in(8), out(8);
    std::memcpy(in.data(), w, 32);
    Context& c = Context::global();
    c.check(sb200_fq_to_mont(c.raw(), 1, 0, in.data(), out.data()), "fq_to_mont");
    BlsScalar s;
    std::memcpy(s.l, out.data(), 32);
    return s;
  }
  Bytes32 to_bytes() const {
    avec<uint32_t> in(8), out(8);
    std::memcpy(in.data(), l, 32);
    Context& c = Context::global();
    c.check(sb200_fq_from_mont(c.raw(), 1, 0, in.data(), out.data()), "fq_from_mont");
    Bytes32 b;
    std::memcpy(b.data(), out.data(), 32);
    return b;
  }
  bool operator==(const BlsScalar& o) const { return std::memcmp(l, o.l, 32) == 0; }
};

// dusk_jubjub::JubJubScalar: canonical 8 x u32 limbs (= to_bytes())
struct JubJubScalar {
  uint32_t l[8] = {};
  static JubJubScalar random(StdRng& rng) {
    avec<uint32_t> o(8);
    detail::wide_draws(rng, 1, 0, o.data());
    JubJubScalar s;
    std::memcpy(s.l, o.data(), 32);
    return s;
  }
  static JubJubScalar from_bytes(const Bytes32& b) {  // rejects >= r
    static const uint32_t r[8] = {0xd6f72cb7u, 0xd0970e5eu, 0xccc81082u, 0xa6682093u, 0x01343b00u, 0x06673b01u, 0x6533afa9u, 0x0e7db4eau};
    JubJubScalar s;
    std::memcpy(s.l, b.data(), 32);
    bool lt = false;
    for (int i = 7; i >= 0; i--) {
      if (s.l[i] != r[i]) { lt = s.l[i] < r[i]; break; }
    }
    if (!lt) throw BytesError(BytesError::InvalidData);
    return s;
  }
  Bytes32 to_bytes() const {
    Bytes32 b;
    std::memcpy(b.data(), l, 32);
    return b;
  }
  bool operator==(const JubJubScalar& o) const { return std::memcmp(l, o.l, 32) == 0; }
};

// dusk_jubjub::JubJubExtended as the projective triple (U : V : Z), Montgomery limbs.  `==` is projective
// (/root/reference/tests/keys.rs:52-58): decided on the canonical compressed form computed by the GPU.
struct JubJubExtended {
  uint32_t l[24] = {};
  static JubJubExtended from_affine_limbs(const uint32_t* uv16) {
    static const uint32_t one[8] = {0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau, 0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u};
    JubJubExtended p;
    std::memcpy(p.l, uv16, 64);
    std::memcpy(p.l + 16, one, 32);
    return p;
  }
  Bytes32 to_bytes() const {  // JubJubAffine::from(self).to_bytes()
    avec<uint32_t> in(24);
    avec<uint8_t> out(32);
    std::memcpy(in.data(), l, 96);
    Context& c = Context::global();
    c.check(sb200_points_compress(c.raw(), 1, SB200_POINTS_PROJECTIVE, in.data(), out.data()), "points_compress");
    Bytes32 b;
    std::memcpy(b.data(), out.data(), 32);
    return b;
  }
  static JubJubExtended from_bytes(const uint8_t* b32) {  // JubJubAffine::from_bytes(..)?.into()
    avec<uint8_t> in(32);
    avec<uint32_t> out(16), ok(1);
    std::memcpy(in.data(), b32, 32);
    Context& c = Context::global();
    c.check(sb200_points_decompress(c.raw(), 1, 0, in.data(), out.data(), ok.data()), "points_decompress");
    if (!(ok[0] & 1)) throw BytesError(BytesError::InvalidData);
    return from_affine_limbs(out.data());
  }
  bool operator==(const JubJubExtended& o) const { return to_bytes() == o.to_bytes(); }
  bool operator!=(const JubJubExtended& o) const { return !(*this == o); }
};

inline std::vector<bool> unpack_bits(const uint32_t* words, size_t n) {
  std::vector<bool> v(n);
  for (size_t i = 0; i < n; i++) v[i] = (words[i >> 5] >> (i & 31)) & 1;  // vector<bool> packs bits: not thread-safe per element
  return v;
}

// ---------------------------------------------------------------------------------------------------------
struct Signature {  // /root/reference/src/signatures.rs:58-123
  static constexpr size_t SIZE = 64;
  JubJubScalar u_;
  JubJubExtended R_;
  const JubJubScalar& u() const { return u_; }
  const JubJubExtended& R() const { return R_; }
  std::array<uint8_t, 64> to_bytes() const {
    std::array<uint8_t, 64> b;
    std::memcpy(b.data(), u_.l, 32);
    auto r = R_.to_bytes();
    std::memcpy(b.data() + 32, r.data(), 32);
    return b;
  }
  static Signature from_bytes(const uint8_t* b, size_t len) {
    if (len != SIZE) throw BytesError(BytesError::BadLength);
    Bytes32 ub;
    std::memcpy(ub.data(), b, 32);
    return Signature{JubJubScalar::from_bytes(ub), JubJubExtended::from_bytes(b + 32)};
  }
  bool operator==(const Signature& o) const { return u_ == o.u_ && R_ == o.R_; }
};
struct SignatureVarGen : Signature {};  // /root/reference/src/signatures.rs:337-404 (same layout)

struct SignatureDouble {  // /root/reference/src/signatures.rs:180-270
  static constexpr size_t SIZE = 96;
  JubJubScalar u_;
  JubJubExtended R_, R_prime_;
  const JubJubScalar& u() const { return u_; }
  const JubJubExtended& R() const { return R_; }
  const JubJubExtended& R_prime() const { return R_prime_; }
  std::array<uint8_t, 96> to_bytes() const {
    std::array<uint8_t, 96> b;
    std::memcpy(b.data(), u_.l, 32);
    auto r = R_.to_bytes(), rp = R_prime_.to_bytes();
    std::memcpy(b.data() + 32, r.data(), 32);
    std::memcpy(b.data() + 64, rp.data(), 32);
    return b;
  }
  static SignatureDouble from_bytes(const uint8_t* b, size_t len) {
    if (len != SIZE) throw BytesError(BytesError::BadLength);
    Bytes32 ub;
    std::memcpy(ub.data(), b, 32);
    return SignatureDouble{JubJubScalar::from_bytes(ub), JubJubExtended::from_bytes(b + 32), JubJubExtended::from_bytes(b + 64)};
  }
  bool operator==(const SignatureDouble& o) const { return u_ == o.u_ && R_ == o.R_ && R_prime_ == o.R_prime_; }
};

class SecretKeyVarGen;

class SecretKey {  // /root/reference/src/keys/secret.rs:56-263
 public:
  static constexpr size_t SIZE = 32;
  SecretKey() = default;
  explicit SecretKey(const JubJubScalar& s) : s_(s) {}
  static SecretKey random(StdRng& rng) { return SecretKey(JubJubScalar::random(rng)); }
  const JubJubScalar& as_ref() const { return s_; }
  Bytes32 to_bytes() const { return s_.to_bytes(); }
  static SecretKey from_bytes(const Bytes32& b) { return SecretKey(JubJubScalar::from_bytes(b)); }
  bool operator==(const SecretKey& o) const { return s_ == o.s_; }

  Signature sign(StdRng& rng, const BlsScalar& msg) const { return sign_batch({*this}, rng, {msg})[0]; }
  SignatureDouble sign_double(StdRng& rng, const BlsScalar& message) const { return sign_double_batch({*this}, rng, {message})[0]; }
  inline SecretKeyVarGen with_variable_generator(const JubJubExtended& generator) const;

  // batch: signature i consumes the rng's i-th JubJubScalar::random draw, in order (secret.rs:155)
  static std::vector<Signature> sign_batch(const std::vector<SecretKey>& sks, StdRng& rng, const std::vector<BlsScalar>& msgs) {
    size_t n = sks.size();
    avec<uint32_t> sk(8 * n), m(8 * n), u(8 * n), R(16 * n);
    detail::parallel_for(n, [&](size_t lo, size_t hi) {
      for (size_t i = lo; i < hi; i++) { std::memcpy(&sk[8 * i], sks[i].s_.l, 32); std::memcpy(&m[8 * i], msgs[i].l, 32); }
    });
    if (!detail::sign_stdrng(rng, 0, n, 0, sk.data(), m.data(), nullptr, u.data(), R.data(), nullptr)) {
      avec<uint32_t> nonce(8 * n);
      detail::wide_draws(rng, n, 0, nonce.data());
      Context& c = Context::global();
      c.check(sb200_sign(c.raw(), (int64_t)n, 0, sk.data(), m.data(), nonce.data(), u.data(), R.data(), nullptr), "sign");
    }
    std::vector<Signature> out(n);
    detail::parallel_for(n, [&](size_t lo, size_t hi) {
      for (size_t i = lo; i < hi; i++) { std::memcpy(out[i].u_.l, &u[8 * i], 32); out[i].R_ = JubJubExtended::from_affine_limbs(&R[16 * i]); }
    });
    return out;
  }
  static std::vector<SignatureDouble> sign_double_batch(const std::vector<SecretKey>& sks, StdRng& rng, const std::vector<BlsScalar>& msgs) {
    size_t n = sks.size();
    avec<uint32_t> sk(8 * n), m(8 * n), u(8 * n), R(16 * n), Rp(16 * n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&sk[8 * i], sks[i].s_.l, 32); std::memcpy(&m[8 * i], msgs[i].l, 32); }
    if (!detail::sign_stdrng(rng, 1, n, 0, sk.data(), m.data(), nullptr, u.data(), R.data(), Rp.data())) {
      avec<uint32_t> nonce(8 * n);
      detail::wide_draws(rng, n, 0, nonce.data());
      Context& c = Context::global();
      c.check(sb200_sign_double(c.raw(), (int64_t)n, 0, sk.data(), m.data(), nonce.data(), u.data(), R.data(), Rp.data(), nullptr), "sign_double");
    }
    std::vector<SignatureDouble> out(n);
    for (size_t i = 0; i < n; i++) {
      std::memcpy(out[i].u_.l, &u[8 * i], 32);
      out[i].R_ = JubJubExtended::from_affine_limbs(&R[16 * i]);
      out[i].R_prime_ = JubJubExtended::from_affine_limbs(&Rp[16 * i]);
    }
    return out;
  }

 private:
  JubJubScalar s_;
  friend class PublicKey;
  friend class PublicKeyDouble;
};

class SecretKeyVarGen {  // /root/reference/src/keys/secret.rs:307-451
 public:
  static constexpr size_t SIZE = 64;
  SecretKeyVarGen(const JubJubScalar& sk, const JubJubExtended& generator) : sk_(sk), generator_(generator) {}
  static SecretKeyVarGen random(StdRng& rng) {  // draws sk, then the generator scalar (secret.rs:371-373)
    JubJubScalar sk = JubJubScalar::random(rng), scalar = JubJubScalar::random(rng);
    avec<uint32_t> k(8), out(16);
    std::memcpy(k.data(), scalar.l, 32);
    Context& c = Context::global();
    c.check(sb200_keygen(c.raw(), 1, 0, k.data(), out.data()), "keygen");  // GENERATOR_EXTENDED * scalar
    return SecretKeyVarGen(sk, JubJubExtended::from_affine_limbs(out.data()));
  }
  const JubJubScalar& secret_key() const { return sk_; }
  const JubJubExtended& generator() const { return generator_; }
  std::array<uint8_t, 64> to_bytes() const {
    std::array<uint8_t, 64> b;
    std::memcpy(b.data(), sk_.l, 32);
    auto g = generator_.to_bytes();
    std::memcpy(b.data() + 32, g.data(), 32);
    return b;
  }
  static SecretKeyVarGen from_bytes(const uint8_t* b, size_t len) {
    if (len != SIZE) throw BytesError(BytesError::BadLength);
    Bytes32 sb;
    std::memcpy(sb.data(), b, 32);
    return SecretKeyVarGen(JubJubScalar::from_bytes(sb), JubJubExtended::from_bytes(b + 32));
  }
  bool operator==(const SecretKeyVarGen& o) const { return sk_ == o.sk_ && generator_ == o.generator_; }
  SignatureVarGen sign(StdRng& rng, const BlsScalar& msg) const {
    avec<uint32_t> sk(8), g(24), m(8), u(8), R(16);
    std::memcpy(sk.data(), sk_.l, 32); std::memcpy(g.data(), generator_.l, 96); std::memcpy(m.data(), msg.l, 32);
    if (!detail::sign_stdrng(rng, 2, 1, SB200_POINTS_PROJECTIVE, sk.data(), m.data(), g.data(), u.data(), R.data(), nullptr)) {
      avec<uint32_t> nonce(8);
      detail::wide_draws(rng, 1, 0, nonce.data());
      Context& c = Context::global();
      c.check(sb200_sign_vargen(c.raw(), 1, SB200_POINTS_PROJECTIVE, sk.data(), g.data(), m.data(), nonce.data(), u.data(), R.data(), nullptr), "sign_vargen");
    }
    SignatureVarGen s;
    std::memcpy(s.u_.l, u.data(), 32);
    s.R_ = JubJubExtended::from_affine_limbs(R.data());
    return s;
  }

 private:
  JubJubScalar sk_;
  JubJubExtended generator_;
};
inline SecretKeyVarGen SecretKey::with_variable_generator(const JubJubExtended& generator) const { return SecretKeyVarGen(s_, generator); }

class PublicKey {  // /root/reference/src/keys/public.rs:59-145
 public:
  static constexpr size_t SIZE = 32;
  PublicKey() = default;
  explicit PublicKey(const JubJubExtended& p) : p_(p) {}
  static PublicKey from(const SecretKey& sk) { return from_batch({sk})[0]; }
  static std::vector<PublicKey> from_batch(const std::vector<SecretKey>& sks) {
    size_t n = sks.size();
    avec<uint32_t> k(8 * n), out(16 * n);
    for (size_t i = 0; i < n; i++) std::memcpy(&k[8 * i], sks[i].s_.l, 32);
    Context& c = Context::global();
    c.check(sb200_keygen(c.raw(), (int64_t)n, 0, k.data(), out.data()), "keygen");
    std::vector<PublicKey> pk(n);
    for (size_t i = 0; i < n; i++) pk[i].p_ = JubJubExtended::from_affine_limbs(&out[16 * i]);
    return pk;
  }
  static PublicKey from_raw_unchecked(const JubJubExtended& key) { return PublicKey(key); }
  const JubJubExtended& as_ref() const { return p_; }
  Bytes32 to_bytes() const { return p_.to_bytes(); }
  static PublicKey from_bytes(const Bytes32& b) { return PublicKey(JubJubExtended::from_bytes(b.data())); }
  bool operator==(const PublicKey& o) const { return p_ == o.p_; }
  bool operator!=(const PublicKey& o) const { return !(*this == o); }

  bool verify(const Signature& sig, const BlsScalar& message) const { return verify_batch({*this}, {sig}, {message})[0]; }
  static std::vector<bool> verify_batch(const std::vector<PublicKey>& pks, const std::vector<Signature>& sigs,
                                        const std::vector<BlsScalar>& msgs) {
    size_t n = pks.size();
    avec<uint32_t> pk(24 * n), u(8 * n), R(24 * n), m(8 * n), bits((n + 31) / 32);
    detail::parallel_for(n, [&](size_t lo, size_t hi) {
      for (size_t i = lo; i < hi; i++) {
        std::memcpy(&pk[24 * i], pks[i].p_.l, 96); std::memcpy(&u[8 * i], sigs[i].u_.l, 32);
        std::memcpy(&R[24 * i], sigs[i].R_.l, 96); std::memcpy(&m[8 * i], msgs[i].l, 32);
      }
    });
    Context& c = Context::global();
    c.check(sb200_verify(c.raw(), (int64_t)n, SB200_POINTS_PROJECTIVE, pk.data(), u.data(), R.data(), m.data(), bits.data(), nullptr), "verify");
    return unpack_bits(bits.data(), n);
  }

 private:
  JubJubExtended p_;
};

class PublicKeyDouble {  // /root/reference/src/keys/public.rs:189-299
 public:
  static constexpr size_t SIZE = 64;
  PublicKeyDouble(const JubJubExtended& pk, const JubJubExtended& pk_prime) : pk_(pk), pk_prime_(pk_prime) {}
  static PublicKeyDouble from(const SecretKey& sk) {
    avec<uint32_t> k(8), a(16), b(16);
    std::memcpy(k.data(), sk.s_.l, 32);
    Context& c = Context::global();
    c.check(sb200_keygen_double(c.raw(), 1, 0, k.data(), a.data(), b.data()), "keygen_double");
    return PublicKeyDouble(JubJubExtended::from_affine_limbs(a.data()), JubJubExtended::from_affine_limbs(b.data()));
  }
  static PublicKeyDouble from_raw_unchecked(const JubJubExtended& pk, const JubJubExtended& pk_prime) { return PublicKeyDouble(pk, pk_prime); }
  const JubJubExtended& pk() const { return pk_; }
  const JubJubExtended& pk_prime() const { return pk_prime_; }
  std::array<uint8_t, 64> to_bytes() const {
    std::array<uint8_t, 64> b;
    auto x = pk_.to_bytes(), y = pk_prime_.to_bytes();
    std::memcpy(b.data(), x.data(), 32); std::memcpy(b.data() + 32, y.data(), 32);
    return b;
  }
  static PublicKeyDouble from_bytes(const uint8_t* b, size_t len) {
    if (len != SIZE) throw BytesError(BytesError::BadLength);
    return PublicKeyDouble(JubJubExtended::from_bytes(b), JubJubExtended::from_bytes(b + 32));
  }
  bool operator==(const PublicKeyDouble& o) const { return pk_ == o.pk_ && pk_prime_ == o.pk_prime_; }
  bool verify(const SignatureDouble& sig_double, const BlsScalar& message) const {
    avec<uint32_t> pk(24), pkp(24), u(8), R(24), Rp(24), m(8), bits(1);
    std::memcpy(pk.data(), pk_.l, 96); std::memcpy(pkp.data(), pk_prime_.l, 96); std::memcpy(u.data(), sig_double.u_.l, 32);
    std::memcpy(R.data(), sig_double.R_.l, 96); std::memcpy(Rp.data(), sig_double.R_prime_.l, 96); std::memcpy(m.data(), message.l, 32);
    Context& c = Context::global();
    c.check(sb200_verify_double(c.raw(), 1, SB200_POINTS_PROJECTIVE, pk.data(), pkp.data(), u.data(), R.data(), Rp.data(), m.data(), bits.data(), nullptr), "verify_double");
    return bits[0] & 1;
  }

 private:
  JubJubExtended pk_, pk_prime_;
};

class PublicKeyVarGen {  // /root/reference/src/keys/public.rs:331-433
 public:
  static constexpr size_t SIZE = 64;
  PublicKeyVarGen(const JubJubExtended& pk, const JubJubExtended& generator) : pk_(pk), generator_(generator) {}
  static PublicKeyVarGen from(const SecretKeyVarGen& sk) {
    avec<uint32_t> k(8), g(24), out(16);
    std::memcpy(k.data(), sk.secret_key().l, 32); std::memcpy(g.data(), sk.generator().l, 96);
    Context& c = Context::global();
    c.check(sb200_keygen_vargen(c.raw(), 1, SB200_POINTS_PROJECTIVE, k.data(), g.data(), out.data()), "keygen_vargen");
    return PublicKeyVarGen(JubJubExtended::from_affine_limbs(out.data()), sk.generator());
  }
  static PublicKeyVarGen from_raw_unchecked(const JubJubExtended& pk, const JubJubExtended& generator) { return PublicKeyVarGen(pk, generator); }
  const JubJubExtended& public_key() const { return pk_; }
  const JubJubExtended& generator() const { return generator_; }
  std::array<uint8_t, 64> to_bytes() const {
    std::array<uint8_t, 64> b;
    auto x = pk_.to_bytes(), y = generator_.to_bytes();
    std::memcpy(b.data(), x.data(), 32); std::memcpy(b.data() + 32, y.data(), 32);
    return b;
  }
  static PublicKeyVarGen from_bytes(const uint8_t* b, size_t len) {
    if (len != SIZE) throw BytesError(BytesError::BadLength);
    return PublicKeyVarGen(JubJubExtended::from_bytes(b), JubJubExtended::from_bytes(b + 32));
  }
  bool operator==(const PublicKeyVarGen& o) const { return pk_ == o.pk_ && generator_ == o.generator_; }
  bool verify(const SignatureVarGen& sig_var_gen, const BlsScalar& message) const {
    avec<uint32_t> pk(24), g(24), u(8), R(24), m(8), bits(1);
    std::memcpy(pk.data(), pk_.l, 96); std::memcpy(g.data(), generator_.l, 96); std::memcpy(u.data(), sig_var_gen.u_.l, 32);
    std::memcpy(R.data(), sig_var_gen.R_.l, 96); std::memcpy(m.data(), message.l, 32);
    Context& c = Context::global();
    c.check(sb200_verify_vargen(c.raw(), 1, SB200_POINTS_PROJECTIVE, pk.data(), g.data(), u.data(), R.data(), m.data(), bits.data(), nullptr), "verify_vargen");
    return bits[0] & 1;
  }

 private:
  JubJubExtended pk_, generator_;
};

}  // namespace dusk_schnorr
