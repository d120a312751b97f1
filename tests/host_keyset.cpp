// Host build of the keyset verification (per-key combs, core.cuh keyset_build_window / verify_keyset_core) on top of
// everything host_arith.cpp exports, for tests/test_keyset.py and tools/op_counts.py.  Test scaffolding: never linked
// into libschnorr_b200.so.
#include "host_arith.cpp"

extern "C" {
// one point's comb (KS_TABLE_WORDS limbs), window by window as the device's lanes build it
void h_keyset_table(const uint32_t* p, int affine, uint32_t* table) {
  std::vector<fq> scratch(2 * (KS_ENTRIES - 1));
  const ext e = point_to_ext(P(p, affine));
  for (int j = 0; j < KS_WINDOWS; j++)
    keyset_build_window(e, j, table + (size_t)j * KS_ENTRIES * 24, scratch.data(), scratch.data() + (KS_ENTRIES - 1));
}
// scheme 0 / 1 / 2; tabs: n_keys keys of (scheme == 0 ? 1 : 2) tables; Rp = R' (1); returns the verdict, c -> c_out
int h_verify_keyset(int scheme, const uint32_t* tabs, int64_t n_keys, const uint32_t* key_ok, uint32_t key, const uint32_t* u,
                    const uint32_t* R, const uint32_t* Rp, const uint32_t* m, int affine, int check_points, const uint32_t* combG,
                    const uint32_t* combGp, uint32_t* c_out) {
  if (scheme == 0)
    return verify_keyset_core<0>(tabs, n_keys, key_ok, key, u, P(R, affine), point_in(), L(m), check_points, combG, combGp, c_out);
  if (scheme == 1)
    return verify_keyset_core<1>(tabs, n_keys, key_ok, key, u, P(R, affine), P(Rp, affine), L(m), check_points, combG, combGp, c_out);
  return verify_keyset_core<2>(tabs, n_keys, key_ok, key, u, P(R, affine), point_in(), L(m), check_points, combG, combGp, c_out);
}
}
