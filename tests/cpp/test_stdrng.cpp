// The seeded batch signers of include/schnorr_b200.hpp draw their nonces on the device from the StdRng's word
// position (sb200_sign_stdrng).  Checked here against the host-drawn path on a twin generator: same signatures, and
// the generator left exactly where the host draws leave it -- also after next_u64 calls that end mid-block, and for
// a stream left inside a word (which keeps the host draw).  Exit code != 0 on any failed check.
#include <cstdio>
#include <cstdlib>

#include "../../include/schnorr_b200.hpp"
using namespace dusk_schnorr;

#define CHECK(cond)                                                   \
  do {                                                                \
    if (!(cond)) {                                                    \
      std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      std::exit(1);                                                   \
    }                                                                 \
  } while (0)

static bool same_point(const JubJubExtended& p, const uint32_t* affine16) { return std::memcmp(p.l, affine16, 64) == 0; }

// keys and messages drawn identically from both generators
static void keys(StdRng& a, StdRng& b, size_t n, std::vector<SecretKey>& sks, std::vector<BlsScalar>& msgs) {
  avec<uint32_t> k(8 * n), m(8 * n), k2(8 * n), m2(8 * n);
  detail::wide_draws(a, n, 0, k.data());
  detail::wide_draws(a, n, 1, m.data());
  detail::wide_draws(b, n, 0, k2.data());
  detail::wide_draws(b, n, 1, m2.data());
  CHECK(std::memcmp(k.data(), k2.data(), 32 * n) == 0 && std::memcmp(m.data(), m2.data(), 32 * n) == 0);
  sks.resize(n);
  msgs.resize(n);
  for (size_t i = 0; i < n; i++) {
    JubJubScalar s;
    std::memcpy(s.l, &k[8 * i], 32);
    sks[i] = SecretKey(s);
    std::memcpy(msgs[i].l, &m[8 * i], 32);
  }
}

static void same_stream(StdRng& a, StdRng& b) {
  CHECK(a.on_word_boundary() == b.on_word_boundary());
  if (a.on_word_boundary()) CHECK(a.word_pos() == b.word_pos());
  for (int i = 0; i < 11; i++) CHECK(a.next_u64() == b.next_u64());
}

static void batch_signers(int prefix, size_t n) {
  Context& c = Context::global();
  StdRng a = StdRng::seed_from_u64(2321), b = StdRng::seed_from_u64(2321);
  for (int i = 0; i < prefix; i++) CHECK(a.next_u64() == b.next_u64());
  std::vector<SecretKey> sks;
  std::vector<BlsScalar> msgs;
  keys(a, b, n, sks, msgs);
  avec<uint32_t> sk(8 * n), m(8 * n), nonce(8 * n), u(8 * n), R(16 * n), Rp(16 * n);
  for (size_t i = 0; i < n; i++) { std::memcpy(&sk[8 * i], sks[i].as_ref().l, 32); std::memcpy(&m[8 * i], msgs[i].l, 32); }

  std::vector<Signature> s1 = SecretKey::sign_batch(sks, a, msgs);
  detail::wide_draws(b, n, 0, nonce.data());
  c.check(sb200_sign(c.raw(), (int64_t)n, 0, sk.data(), m.data(), nonce.data(), u.data(), R.data(), nullptr), "sign");
  for (size_t i = 0; i < n; i++) CHECK(std::memcmp(s1[i].u_.l, &u[8 * i], 32) == 0 && same_point(s1[i].R_, &R[16 * i]));
  CHECK(a.word_pos() == b.word_pos());

  std::vector<SignatureDouble> s2 = SecretKey::sign_double_batch(sks, a, msgs);
  detail::wide_draws(b, n, 0, nonce.data());
  c.check(sb200_sign_double(c.raw(), (int64_t)n, 0, sk.data(), m.data(), nonce.data(), u.data(), R.data(), Rp.data(), nullptr), "sign_double");
  for (size_t i = 0; i < n; i++)
    CHECK(std::memcmp(s2[i].u_.l, &u[8 * i], 32) == 0 && same_point(s2[i].R_, &R[16 * i]) && same_point(s2[i].R_prime_, &Rp[16 * i]));
  CHECK(a.word_pos() == b.word_pos());

  // SecretKeyVarGen::sign: one signature per call, generator = a key's public point
  PublicKey gen = PublicKey::from(sks[0]);
  SecretKeyVarGen vk(sks[1].as_ref(), gen.as_ref());
  for (int r = 0; r < 3; r++) {
    SignatureVarGen sv = vk.sign(a, msgs[r]);
    avec<uint32_t> g(24), one_sk(8), one_m(8), one_n(8), one_u(8), one_R(16);
    std::memcpy(g.data(), gen.as_ref().l, 96); std::memcpy(one_sk.data(), sks[1].as_ref().l, 32); std::memcpy(one_m.data(), msgs[r].l, 32);
    detail::wide_draws(b, 1, 0, one_n.data());
    c.check(sb200_sign_vargen(c.raw(), 1, SB200_POINTS_PROJECTIVE, one_sk.data(), g.data(), one_m.data(), one_n.data(), one_u.data(),
                              one_R.data(), nullptr), "sign_vargen");
    CHECK(std::memcmp(sv.u_.l, one_u.data(), 32) == 0 && same_point(sv.R_, one_R.data()));
  }
  same_stream(a, b);
  std::printf("batch signers, %d next_u64 first, n = %zu: ok\n", prefix, n);
}

static void seek_and_word_pos() {
  StdRng a = StdRng::seed_from_u64(7);
  uint8_t buf[200];
  for (uint64_t w : {0ull, 1ull, 15ull, 16ull, 33ull, 16ull * 0xffffffffull + 5, (1ull << 63) + 9}) {
    StdRng s = StdRng::seed_from_u64(7), t = StdRng::seed_from_u64(7);
    s.seek(w);
    CHECK(s.on_word_boundary() && s.word_pos() == w);
    if (w < 64) {  // sequential twin: skip w words
      for (uint64_t i = 0; i < w; i++) t.fill_bytes(buf, 4);
      CHECK(t.word_pos() == w);
      same_stream(s, t);
    }
  }
  a.fill_bytes(buf, 3);
  CHECK(!a.on_word_boundary());
  std::printf("seek / word_pos: ok\n");
}

// a stream inside a word keeps the host draw and stays the same stream
static void mid_word() {
  StdRng a = StdRng::seed_from_u64(9), b = StdRng::seed_from_u64(9);
  uint8_t buf[3];
  a.fill_bytes(buf, 3);
  b.fill_bytes(buf, 3);
  std::vector<SecretKey> sks(4, SecretKey::random(a));
  (void)SecretKey::random(b);
  std::vector<BlsScalar> msgs(4, BlsScalar::random(a));
  (void)BlsScalar::random(b);
  CHECK(!a.on_word_boundary());
  std::vector<Signature> s = SecretKey::sign_batch(sks, a, msgs);
  avec<uint32_t> sk(32), m(32), nonce(32), u(32), R(64);
  for (size_t i = 0; i < 4; i++) { std::memcpy(&sk[8 * i], sks[i].as_ref().l, 32); std::memcpy(&m[8 * i], msgs[i].l, 32); }
  detail::wide_draws(b, 4, 0, nonce.data());
  Context& c = Context::global();
  c.check(sb200_sign(c.raw(), 4, 0, sk.data(), m.data(), nonce.data(), u.data(), R.data(), nullptr), "sign");
  for (size_t i = 0; i < 4; i++) CHECK(std::memcmp(s[i].u_.l, &u[8 * i], 32) == 0 && same_point(s[i].R_, &R[16 * i]));
  same_stream(a, b);
  std::printf("mid-word stream: ok\n");
}

int main() {
  try {
    seek_and_word_pos();
    batch_signers(0, 1000 + 37);
    batch_signers(1, 1000 + 37);
    batch_signers(3, 1 << 15);
    batch_signers(5, 1);
    mid_word();
    std::printf("ALL OK\n");
    return 0;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "test_stdrng: %s\n", e.what());
    return 2;
  }
}
