// Host build of the witness rows against a keyset (core.cuh verify_witness_keyset_core) on top of everything
// host_keyset.cpp exports (the per-key combs and the keyset verification), for tests/test_keyset_witness.py and
// tools/op_counts.py.  Test scaffolding: never linked into libschnorr_b200.so.
#include "host_keyset.cpp"

extern "C" {
// the witness row of a tuple against key `key` of the keyset: 11 / 19 / 13 field elements -> rows; returns the verdict
int h_verify_witness_keyset(int scheme, const uint32_t* tabs, int64_t n_keys, const uint32_t* key_ok, uint32_t key,
                            const uint32_t* u, const uint32_t* R, const uint32_t* Rp, const uint32_t* m, int affine,
                            int check_points, const uint32_t* combG, const uint32_t* combGp, uint32_t* rows) {
  auto emit = [&](int k, const fq& v) { S(rows + 8 * k, v); };
  if (scheme == 0)
    return verify_witness_keyset_core<0>(tabs, n_keys, key_ok, key, u, P(R, affine), point_in(), L(m), check_points, combG, combGp,
                                         emit);
  if (scheme == 1)
    return verify_witness_keyset_core<1>(tabs, n_keys, key_ok, key, u, P(R, affine), P(Rp, affine), L(m), check_points, combG,
                                         combGp, emit);
  return verify_witness_keyset_core<2>(tabs, n_keys, key_ok, key, u, P(R, affine), point_in(), L(m), check_points, combG, combGp,
                                       emit);
}
}
