// Host build of the verifier-side witness rows (core.cuh verify_witness_core) on top of everything host_arith.cpp
// exports, for tests/test_verify_witness.py and tools/op_counts.py.  Test scaffolding: never linked into
// libschnorr_b200.so.
#include "host_arith.cpp"

extern "C" {
// scheme 0 / 1 / 2 -> 11 / 19 / 13 field elements; pk2 = PK' (1) or the generator (2), Rp = R' (1); returns the verdict
int h_verify_witness(int scheme, const uint32_t* pk, const uint32_t* pk2, const uint32_t* u, const uint32_t* R,
                     const uint32_t* Rp, const uint32_t* m, int affine, int check_points, const uint32_t* combG,
                     const uint32_t* combGp, uint32_t* rows) {
  auto emit = [&](int k, const fq& v) { S(rows + 8 * k, v); };
  if (scheme == 0)
    return verify_witness_core<0>(P(pk, affine), point_in(), u, P(R, affine), point_in(), L(m), check_points, combG, combGp, emit);
  if (scheme == 1)
    return verify_witness_core<1>(P(pk, affine), P(pk2, affine), u, P(R, affine), P(Rp, affine), L(m), check_points, combG,
                                  combGp, emit);
  return verify_witness_core<2>(P(pk, affine), P(pk2, affine), u, P(R, affine), point_in(), L(m), check_points, combG, combGp, emit);
}
}
