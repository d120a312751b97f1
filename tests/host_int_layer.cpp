// Host build of the small-integer Hades layers (csrc/hades.cuh hades_perm_int, csrc/params_host.cuh
// derive_int_tables): the exports of host_arith.cpp plus views of the new tables and the layer alone.
// Test scaffolding for tests/test_hades_cauchy.py: never linked into libschnorr_b200.so.
#include "host_arith.cpp"

extern "C" {
// cmat (25 doubles), src (335 x 8), fix (59 x 8), unscale (8), int_layers: the tables after the public view
void h_int_tables(double* cmat, uint32_t* src, uint32_t* fix, uint32_t* unscale, uint32_t* flag) {
  memcpy(cmat, sb200::h_hades.cmat, sizeof(sb200::h_hades.cmat));
  memcpy(src, sb200::h_hades.src, sizeof(sb200::h_hades.src));
  memcpy(fix, sb200::h_hades.fix, sizeof(sb200::h_hades.fix));
  memcpy(unscale, sb200::h_hades.unscale, sizeof(sb200::h_hades.unscale));
  *flag = sb200::h_hades.int_layers;
}
// one layer s <- C s mod q on five canonical words (any representation: the layer is linear over the integers)
void h_int_layer(uint32_t* st) {
  fq s[5];
  for (int i = 0; i < 5; i++) s[i] = L(st + 8 * i);
  hades_int_layer(s);
  for (int i = 0; i < 5; i++) S(st + 8 * i, s[i]);
}
// the reduction alone: (top * 2^256 + r) mod q
void h_int_reduce(uint32_t* r, uint32_t top) {
  fq x = L(r);
  hl_reduce(x, top);
  S(r, x);
}
int h_int_bound() { return (int)params::INT_LAYER_CMAX_BOUND; }
}
