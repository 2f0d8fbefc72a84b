// fixed_base_sim.cpp -- TEST INFRASTRUCTURE ONLY.  The CPU simulation of hostsim.cpp plus the device code of registered bases
// (fq_base_create / fq_dh_fixed / fq_mul_fixed): k_comb_build for a given point and k_comb + k_dh_finish on its tables.
// Built by build_fixed_base.sh in place of hostsim.cpp; it is NOT linked into, loaded by, or a fallback for libfourq_b200.so.
#include "hostsim.cpp"

extern "C" {

// k_comb_build (kernels_comb.cu): out = [2][FQ_COMB_WORDS] words, the tables of P and [392]P for P = the canonical affine
// point xy (64 bytes, a registered base), or for P = G from the curve constants (xy = NULL, the tables of context creation)
int sim_comb_tables(const uint8_t* xy, u32* out) {
  u32 w[16] = {0};
  if (xy) memcpy(w, xy, 64);
  const fp2 x = xy ? row_load_fp2(w) : curve_gx(), y = xy ? row_load_fp2(w + 8) : curve_gy();
  for (int which = 0; which < 2; which++)
    for (int i = 0; i < FQ_COMB_DIGITS; i++) comb_build_digit(comb_base(which, x, y), i, out + which * FQ_COMB_WORDS + i * FQ_COMB_DIGIT_WORDS);
  return 0;
}
// fq_dh_fixed (dh = 1) / fq_mul_fixed (dh = 0): k_comb_build for the point xy (NULL = G), then k_comb + k_dh_finish on the
// table of [392]P or of P
int sim_comb_point(int dh, const uint8_t* xy, const uint8_t* k, uint8_t* out, uint8_t* status, size_t n) {
  std::vector<u32> tabs(2 * FQ_COMB_WORDS);
  sim_comb_tables(xy, tabs.data());
  SimScratch sc(n);
  for (size_t i = 0; i < n; i++) {
    u32 wk[8]; memcpy(wk, k + 32 * i, 32);
    sc.put(i, mul_comb(row_load_scalar(wk), tabs.data() + (dh ? FQ_COMB_WORDS : 0)), 0);
  }
  if (dh) sim_finish<false, true>(sc, out, status, n, FQ_BATCHINV_ROWS); else sim_finish<false, false>(sc, out, status, n, FQ_BATCHINV_ROWS);
  return 0;
}

}  // extern "C"
