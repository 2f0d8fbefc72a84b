// comb.cuh -- fixed-base scalar multiplication with one precomputed table per digit (SURVEY.md 8f-2).
//
// The reference's fixed-base entry points are MUL_*(m, G, table=T) = [m]G (curve4q.py:582-584) and
// DH_*(m, G, table=T392) = [392 m]G (curve4q.py:743-762); the draft points to "FourQlib's fixed-base algorithm" for key
// generation (draft-ladd-cfrg-4q.md:702-705, :727-729).  The affine result is canonical, so any correct algorithm gives
// the reference's bytes.  Here the base point B is fixed, so all doublings are precomputed:
//
//     r = m mod N (+N if even) = sum_{i=0}^{62} d_i 16^i,  d_i odd in [-15, 15], d_62 = 1      (scalar.cuh, curve4q.py:216-226)
//     [r]B = [16^62]B + sum_{i=0}^{61} sign(d_i) * T_i[(|d_i|-1)/2],      T_i[j] = [(2j+1) 16^i]B
//
// 62 mixed additions (7 GF(p^2) multiplications each, the table entries have Z = 1) and no doubling: 20,832 32x32->64
// multiply-adds per row instead of 92,624 for MUL_windowed with a table (SURVEY 8d).  T_i[j] is stored as
// (x+y, y-x, 2dxy) = 96 B; a base needs 63 x 8 x 96 B = 47.25 KiB, which a CTA copies from global to shared memory.
// The scan over the 8 entries of T_i reads the SAME addresses in every thread (broadcast LDS) and keeps one entry with
// predicated selects: no secret-dependent address or branch.
#pragma once
#include "dh.cuh"

struct ptA3 { fp2 N, D, F; };                        // affine point as (x+y, y-x, 2dxy)

#define FQ_COMB_DIGITS 63
#define FQ_COMB_ENTRY_WORDS 24                       // N.re N.im D.re D.im F.re F.im, 4 words each
#define FQ_COMB_DIGIT_WORDS (8 * FQ_COMB_ENTRY_WORDS)
#define FQ_COMB_WORDS (FQ_COMB_DIGITS * FQ_COMB_DIGIT_WORDS)      // 12,096 words = 48,384 B per base point

// R1 + (affine, Z = 1) -> R1: ADD_core (curve4q.py:155-171) with E2 = 2 Z2 = 2, so D = Z1 * E2 is a doubling.
FQ_FN ptR1 pt_madd(const ptR1& Q, const ptA3& S) {
  fp2b N1 = fp2_prep(fp2_add(Q.X, Q.Y)), D1 = fp2_prep(fp2_sub(Q.Y, Q.X)), T1 = fp2_prep(fp2_mul(Q.Ta, Q.Tb));
  fp2 A = fp2_mul_prep(S.D, D1), B = fp2_mul_prep(S.N, N1), C = fp2_mul_prep(S.F, T1), D = fp2_dbl(Q.Z);
  fp2 E = fp2_sub(B, A), F = fp2_sub(D, C), G = fp2_add(D, C), H = fp2_add(B, A);
  fp2b Fp = fp2_prep(F), Gp = fp2_prep(G);
  ptR1 R;
  R.X = fp2_mul_prep(E, Fp); R.Y = fp2_mul_prep(H, Gp); R.Z = fp2_mul_prep(G, Fp); R.Ta = E; R.Tb = H;
  return R;
}

FQ_FN ptA3 a3_load(const u32* w) {
  ptA3 P;
  P.N = fp2_set(fp_set(w[0], w[1], w[2], w[3]), fp_set(w[4], w[5], w[6], w[7]));
  P.D = fp2_set(fp_set(w[8], w[9], w[10], w[11]), fp_set(w[12], w[13], w[14], w[15]));
  P.F = fp2_set(fp_set(w[16], w[17], w[18], w[19]), fp_set(w[20], w[21], w[22], w[23]));
  return P;
}

// constant-time T_i[idx] with the sign applied (curve4q.py:193-195: -(N, D, F) = (D, N, -F)); tab = the 192 words of T_i in
// shared memory (16-byte aligned).  Entry 7 is loaded unconditionally, entries 0..6 under the digit's predicate (dh.cuh
// quad_take): 6 LDS.128 per entry, the same addresses in every thread (broadcast).
template <bool STRICT = FQ_STRICT_DEFAULT> FQ_FN ptA3 comb_select(const u32* tab, u32 idx, u32 neg) {
  const uint4* t4 = reinterpret_cast<const uint4*>(tab);
  fp w[6];
  FQ_UNROLL
  for (int q = 0; q < 6; q++) { uint4 v = t4[7 * 6 + q]; w[q] = fp_set(v.x, v.y, v.z, v.w); }
  FQ_UNROLL
  for (int e = 0; e < 7; e++) {
    const bool c = idx == (u32)e;
    FQ_UNROLL
    for (int q = 0; q < 6; q++) quad_take<STRICT>(t4 + e * 6 + q, w[q], c);
  }
  ptA3 P, R;
  P.N = fp2_set(w[0], w[1]); P.D = fp2_set(w[2], w[3]); P.F = fp2_set(w[4], w[5]);
  R.N = fp2_select(neg, P.D, P.N); R.D = fp2_select(neg, P.N, P.D);
  R.F.re = fp_set(P.F.re.v[0] ^ neg, P.F.re.v[1] ^ neg, P.F.re.v[2] ^ neg, P.F.re.v[3] ^ (neg & FQ_P3));
  R.F.im = fp_set(P.F.im.v[0] ^ neg, P.F.im.v[1] ^ neg, P.F.im.v[2] ^ neg, P.F.im.v[3] ^ (neg & FQ_P3));
  return R;
}

// [k]B for the base point whose tables are `tab` (FQ_COMB_WORDS words); returns R1
template <bool STRICT = FQ_STRICT_DEFAULT> FQ_FN ptR1 mul_comb(const scal& k, const u32* tab) {
  MulPlan pl = plan_windowed(k);
  // leading digit d_62 = +1: start from T_62[0] = [16^62]B, back in (x, y) from (x+y, y-x)
  ptA3 S = a3_load(tab + 62 * FQ_COMB_DIGIT_WORDS);
  fp2 x = fp2_set(fp_half(fp_sub(S.N.re, S.D.re)), fp_half(fp_sub(S.N.im, S.D.im)));
  fp2 y = fp2_set(fp_half(fp_add(S.N.re, S.D.re)), fp_half(fp_add(S.N.im, S.D.im)));
  ptR1 Q = pt_from_affine(x, y);
  FQ_NOUNROLL
  for (int i = 61; i >= 0; i--) {
    u32 idx, neg;
    scal_next_digit(pl.S, idx, neg);
    Q = pt_madd(Q, comb_select<STRICT>(tab + i * FQ_COMB_DIGIT_WORDS, idx, neg));
  }
  return Q;
}

// The base whose tables give MUL (dh = 0: B = P, curve4q.py:582-584) or DH (dh = 1: B = [392]P, curve4q.py:450-460) of the
// point P = (x, y).  The tables of G built at context creation and those of a caller-registered point both start here.
FQ_FN ptR1 comb_base(int dh, const fp2& x, const fp2& y) { return dh ? pt_clear_cofactor(x, y) : pt_from_affine(x, y); }

// Table construction, one call per (base, digit): out = the 192 words of T_i for the base B (comb_base).
// P = [16^i]B by 4 i doublings, then the odd multiples as in table_windowed (curve4q.py:179-185), each normalised to
// affine.  Every entry is canonical affine, so the words depend only on the group element B, not on its coordinates.
// Run once per device at context creation for G (k_comb_build, 126 threads), once per device for a registered point, and
// by the CPU simulation in tests/hostsim.
FQ_FN void comb_build_digit(const ptR1& B, int i, u32* out) {
  ptR1 P = B;
  FQ_NOUNROLL
  for (int t = 0; t < 4 * i; t++) pt_dbl_c(&P);
  ptR1 P2 = P;
  pt_dbl_c(&P2);
  ptR3 P23; pt_r1_to_r3_c(&P23, &P2);
  ptR1 M = P;
  FQ_NOUNROLL
  for (int j = 0; j < 8; j++) {
    fp2 x, y;
    pt_to_affine(M, x, y);
    fp2 N = fp2_canon(fp2_add(x, y)), D = fp2_canon(fp2_sub(y, x));
    fp2 F = fp2_canon(fp2_mul_c(fp2_mul_c(x, y), curve_2d()));
    u32* w = out + j * FQ_COMB_ENTRY_WORDS;
    FQ_UNROLL
    for (int l = 0; l < 4; l++) {
      w[l] = N.re.v[l]; w[4 + l] = N.im.v[l]; w[8 + l] = D.re.v[l]; w[12 + l] = D.im.v[l]; w[16 + l] = F.re.v[l]; w[20 + l] = F.im.v[l];
    }
    if (j < 7) { ptR2 Mr2; pt_r1_to_r2_c(&Mr2, &M); pt_add_core_c(&M, &P23, &Mr2); }     // M += 2P
  }
}
// the same for the tables of G (which = 0) and [392]G (which = 1), as the CPU simulation of tests/hostsim builds them
FQ_FN void comb_build_digit(int which, int i, u32* out) { comb_build_digit(comb_base(which, curve_gx(), curve_gy()), i, out); }
