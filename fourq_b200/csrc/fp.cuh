// fp.cuh -- GF(p), p = 2^127 - 1, on 4 x 32-bit limbs held in registers.
// Replaces the Python-bigint arithmetic of the reference's impl/fields.py:29-132 (GFp.add/sub/mul/sqr/neg/select/
// inv/invsqrt); results are identical after canonicalisation (fp_canon).
//
// Representation.  fp = {v[0..3]}, little-endian limbs.  "tight" = value <= p (p itself is an alias of 0);
// "loose" = any value < 2^128.  Unless a comment says otherwise every function takes and returns tight values.
//
// Multiplication.  a*b mod p with 2^128 = 2 (mod p).  The b operand is "prepared" once (fp_prep): for row i the
// multiplier limb a_i meets the 4-limb vector  rot_i(b) = b * 2^(32 i) mod p  =  (low limbs of b shifted up) +
// 2 * (high limbs of b), which is exact in 4 limbs because b < 2^127.  All 16 products of a multiplication therefore
// land in ONE 5-limb window (+ small overflow counters) instead of an 8-limb product that would need a lo + 2*hi
// pass.  Products are accumulated in two 64-bit-aligned lattices (even limb positions E, odd positions O) by
// mad.lo.cc/madc.hi.cc pairs = IMAD.WIDE.U32[.X] with predicate carries; E and O are merged once per result.
//
// Cost of one 4x4 product: 16 IMAD.WIDE + 6 carry catches; merge 5; reduction to tight 11 (see fp_fold).
#pragma once
#include "arith.cuh"

struct fp { u32 v[4]; };

// b-side operand: limbs of b and of its rotations by 32/64/96 bits
struct fpb { u32 b0, b1, b2, b3, e1, e2, e3, d2, d3; };

// product accumulator: value = E + (O << 32);  E = e0..e4 (e4 counts carries), O = o1..o5 (o5 counts carries)
struct facc { u32 e0, e1, e2, e3, e4, o1, o2, o3, o4, o5; };

// merged accumulator, value = sum w[i] 2^(32 i), w[5] small
struct fpw { u32 w[6]; };

#define FQ_P3 0x7fffffffu

FQ_FN fp fp_set(u32 a0, u32 a1, u32 a2, u32 a3) { fp r; r.v[0] = a0; r.v[1] = a1; r.v[2] = a2; r.v[3] = a3; return r; }
FQ_FN fp fp_zero() { return fp_set(0, 0, 0, 0); }
FQ_FN fp fp_one() { return fp_set(1, 0, 0, 0); }

// ---------------------------------------------------------------- additive group

// tight + tight -> loose (< 2^128).  Only valid as the multiplier ("a") side of fp_mul / as input of fp_fold1.
FQ_FN fp fp_add_loose(const fp& a, const fp& b) {
  fp r;
  r.v[0] = add_cc(a.v[0], b.v[0]); r.v[1] = addc_cc(a.v[1], b.v[1]);
  r.v[2] = addc_cc(a.v[2], b.v[2]); r.v[3] = addc(a.v[3], b.v[3]);
  return r;
}

// loose (<= 2p) -> tight:  x mod 2^127 + (x >> 127)
FQ_FN fp fp_fold1(const fp& x) {
  fp r; u32 t = x.v[3] >> 31;
  r.v[0] = add_cc(x.v[0], t); r.v[1] = addc_cc(x.v[1], 0);
  r.v[2] = addc_cc(x.v[2], 0); r.v[3] = addc(x.v[3] & FQ_P3, 0);
  return r;
}

// fields.py:30-33
FQ_FN fp fp_add(const fp& a, const fp& b) { return fp_fold1(fp_add_loose(a, b)); }

// fields.py:36-39.  a - b, +p when it borrows: the wrapped difference minus 1 with bit 127 cleared.
FQ_FN fp fp_sub(const fp& a, const fp& b) {
  fp r;
  r.v[0] = sub_cc(a.v[0], b.v[0]); r.v[1] = subc_cc(a.v[1], b.v[1]);
  r.v[2] = subc_cc(a.v[2], b.v[2]); r.v[3] = subc_cc(a.v[3], b.v[3]);
  r.v[0] = subc_cc(r.v[0], 0); r.v[1] = subc_cc(r.v[1], 0);
  r.v[2] = subc_cc(r.v[2], 0); r.v[3] = subc(r.v[3], 0) & FQ_P3;
  return r;
}

// fields.py:54-57.  p - a = a xor p
FQ_FN fp fp_neg(const fp& a) { return fp_set(~a.v[0], ~a.v[1], ~a.v[2], a.v[3] ^ FQ_P3); }

// 2a and a/2 are rotations of the 127-bit string
FQ_FN fp fp_dbl(const fp& a) {
  return fp_set((a.v[0] << 1) | (a.v[3] >> 30), shl_pair(a.v[0], a.v[1], 1), shl_pair(a.v[1], a.v[2], 1),
                shl_pair(a.v[2], a.v[3], 1) & FQ_P3);
}
FQ_FN fp fp_half(const fp& a) {   // curve4q.py:82 multiplies by GFp.half = 2^126
  return fp_set(shr_pair(a.v[0], a.v[1], 1), shr_pair(a.v[1], a.v[2], 1), shr_pair(a.v[2], a.v[3], 1),
                (a.v[3] >> 1) | ((a.v[0] & 1) << 30));
}

// tight -> canonical (p -> 0).  All ones mask if a == p.
FQ_FN fp fp_canon(const fp& a) {
  u32 allones = a.v[0] & a.v[1] & a.v[2] & (a.v[3] | 0x80000000u);
  u32 m = (allones == 0xffffffffu) ? 0u : 0xffffffffu;
  return fp_set(a.v[0] & m, a.v[1] & m, a.v[2] & m, a.v[3] & m);
}
// inputs canonical
FQ_FN bool fp_eq_canon(const fp& a, const fp& b) {
  return ((a.v[0] ^ b.v[0]) | (a.v[1] ^ b.v[1]) | (a.v[2] ^ b.v[2]) | (a.v[3] ^ b.v[3])) == 0;
}
FQ_FN bool fp_is_zero(const fp& a) {   // a tight: zero is 0 or p
  u32 o = a.v[0] | a.v[1] | a.v[2] | a.v[3];
  u32 n = a.v[0] & a.v[1] & a.v[2] & (a.v[3] | 0x80000000u);
  return (o == 0) | (n == 0xffffffffu);
}
// fields.py:60-64: m all-ones -> x, m zero -> y
FQ_FN fp fp_select(u32 m, const fp& x, const fp& y) {
  return fp_set(y.v[0] ^ (m & (x.v[0] ^ y.v[0])), y.v[1] ^ (m & (x.v[1] ^ y.v[1])),
                y.v[2] ^ (m & (x.v[2] ^ y.v[2])), y.v[3] ^ (m & (x.v[3] ^ y.v[3])));
}
// any 128-bit value -> tight (used on untrusted inputs of the field-op entry points)
FQ_FN fp fp_from_u128(const fp& x) { return fp_fold1(fp_fold1(x)); }

// ---------------------------------------------------------------- multiplication

// b tight
FQ_FN fpb fp_prep(const fp& b) {
  fpb B;
  B.b0 = b.v[0]; B.b1 = b.v[1]; B.b2 = b.v[2]; B.b3 = b.v[3];
  B.e1 = b.v[1] << 1; B.e2 = b.v[2] << 1; B.e3 = b.v[3] << 1;
  B.d2 = shl_pair(b.v[1], b.v[2], 1); B.d3 = shl_pair(b.v[2], b.v[3], 1);
  return B;
}

FQ_FN void facc_zero(facc& A) { A.e0 = A.e1 = A.e2 = A.e3 = A.e4 = A.o1 = A.o2 = A.o3 = A.o4 = A.o5 = 0; }

// A = 2^k * p spread over the lattices so that later limb sums are exact: value 2^(127+k) - 2^k, 32 < k < 64.
// Used as a positivity offset for lazy subtractions (it is 0 mod p).
template <int K> FQ_FN void facc_init_kp(facc& A) {
  A.e0 = 0; A.e1 = 0u - (1u << (K - 32)); A.e2 = 0xffffffffu; A.e3 = 0xffffffffu; A.e4 = 0;
  A.o1 = 0; A.o2 = 0; A.o3 = 0; A.o4 = 0xffffffffu; A.o5 = (1u << (K - 33)) - 1u;
}

// first row into a fresh accumulator: no carries to catch
FQ_FN void facc_row0(facc& A, u32 a, u32 v0, u32 v1, u32 v2, u32 v3) {
  mul_wide(A.e0, A.e1, a, v0); mul_wide(A.e2, A.e3, a, v2); A.e4 = 0;
  mul_wide(A.o1, A.o2, a, v1); mul_wide(A.o3, A.o4, a, v3); A.o5 = 0;
}
// A += a * (v0 + v1 2^32 + v2 2^64 + v3 2^96)
FQ_FN void facc_row(facc& A, u32 a, u32 v0, u32 v1, u32 v2, u32 v3) {
  A.e0 = mad_lo_cc(a, v0, A.e0); A.e1 = madc_hi_cc(a, v0, A.e1);
  A.e2 = madc_lo_cc(a, v2, A.e2); A.e3 = madc_hi_cc(a, v2, A.e3); A.e4 = addc(A.e4, 0);
  A.o1 = mad_lo_cc(a, v1, A.o1); A.o2 = madc_hi_cc(a, v1, A.o2);
  A.o3 = madc_lo_cc(a, v3, A.o3); A.o4 = madc_hi_cc(a, v3, A.o4); A.o5 = addc(A.o5, 0);
}

// A (+)= a * b mod-p-folded; a loose allowed, B = fp_prep(tight b).  FRESH: A is overwritten.
template <bool FRESH> FQ_FN void facc_mul(facc& A, const fp& a, const fpb& B) {
  if (FRESH) facc_row0(A, a.v[0], B.b0, B.b1, B.b2, B.b3);
  else facc_row(A, a.v[0], B.b0, B.b1, B.b2, B.b3);
  facc_row(A, a.v[1], B.e3, B.b0, B.b1, B.b2);
  facc_row(A, a.v[2], B.e2, B.d3, B.b0, B.b1);
  facc_row(A, a.v[3], B.e1, B.d2, B.d3, B.b0);
}

FQ_FN fpw facc_merge(const facc& A) {
  fpw r;
  r.w[0] = A.e0; r.w[1] = add_cc(A.e1, A.o1); r.w[2] = addc_cc(A.e2, A.o2); r.w[3] = addc_cc(A.e3, A.o3);
  r.w[4] = addc_cc(A.e4, A.o4); r.w[5] = addc(A.o5, 0);
  return r;
}
// a - b, caller guarantees a >= b
FQ_FN fpw fpw_sub(const fpw& a, const fpw& b) {
  fpw r;
  r.w[0] = sub_cc(a.w[0], b.w[0]); r.w[1] = subc_cc(a.w[1], b.w[1]); r.w[2] = subc_cc(a.w[2], b.w[2]);
  r.w[3] = subc_cc(a.w[3], b.w[3]); r.w[4] = subc_cc(a.w[4], b.w[4]); r.w[5] = subc(a.w[5], b.w[5]);
  return r;
}

// wide (< 2^166) -> tight.  Pass 1: x mod 2^127 + (x >> 127) < 2^127 + 2^39.  Pass 2: the same again; when bit 127
// is set the rest is < 2^39, so the +1 can ripple into limb 1 at most.
FQ_FN fp fp_fold(const fpw& x) {
  fp r;
  u32 tlo = shr_pair(x.w[3], x.w[4], 31), thi = shr_pair(x.w[4], x.w[5], 31);
  r.v[0] = add_cc(x.w[0], tlo); r.v[1] = addc_cc(x.w[1], thi);
  r.v[2] = addc_cc(x.w[2], 0); r.v[3] = addc(x.w[3] & FQ_P3, 0);
  u32 top = r.v[3] >> 31;
  r.v[3] &= FQ_P3;
  r.v[0] = add_cc(r.v[0], top); r.v[1] = addc(r.v[1], 0);
  return r;
}

// fields.py:42-45.  a loose allowed; b tight.
FQ_FN fp fp_mul_prep(const fp& a, const fpb& B) {
  facc A; facc_mul<true>(A, a, B);
  return fp_fold(facc_merge(A));
}
FQ_FN fp fp_mul(const fp& a, const fp& b) { return fp_mul_prep(a, fp_prep(b)); }
// fields.py:48-51.  a tight.  Dedicated squaring: the 6 cross products are taken once against the doubled tail of a,
//     a^2 = a0 (a0 + 2 a[1..3]) + a1 W (a1 W + 2 a[2..3]) + a2 W^2 (a2 W^2 + 2 a3 W^3) + a3^2 W^6,      W = 2^32,
// where 2 a[1..3] = e1 W + d2 W^2 + d3 W^3, 2 a[2..3] = e2 W^2 + d3 W^3, 2 a3 = e3 (all exact: a < 2^127) and
// a3^2 W^6 = (a3 e3) W^2 (mod p).  10 IMAD.WIDE instead of 16; the products at W^4 and W^5 stay where they are and the
// 7-limb sum (< 2^226) is folded in one wider pass (fp_fold7).
FQ_FN fp fp_fold7(u32 w0, u32 w1, u32 w2, u32 w3, u32 w4, u32 w5, u32 w6) {
  fp r;
  u32 t0 = shr_pair(w3, w4, 31), t1 = shr_pair(w4, w5, 31), t2 = shr_pair(w5, w6, 31), t3 = w6 >> 31;    // x >> 127 < 2^99
  r.v[0] = add_cc(w0, t0); r.v[1] = addc_cc(w1, t1); r.v[2] = addc_cc(w2, t2); r.v[3] = addc(w3 & FQ_P3, t3);
  u32 top = r.v[3] >> 31;                    // when set, the rest is < 2^99: the +1 cannot leave limb 3
  r.v[3] &= FQ_P3;
  r.v[0] = add_cc(r.v[0], top); r.v[1] = addc_cc(r.v[1], 0); r.v[2] = addc_cc(r.v[2], 0); r.v[3] = addc(r.v[3], 0);
  return r;
}
FQ_FN fp fp_sqr(const fp& a) {
  const u32 a0 = a.v[0], a1 = a.v[1], a2 = a.v[2], a3 = a.v[3];
  const u32 e1 = a1 << 1, e2 = a2 << 1, e3 = a3 << 1, d2 = shl_pair(a1, a2, 1), d3 = shl_pair(a2, a3, 1);
  u32 E0, E1, E2, E3, E4, E5, E6, O1, O2, O3, O4, O5, O6;
  // even lattice: W^0, W^2, W^4
  mul_wide(E0, E1, a0, a0); mul_wide(E2, E3, a0, d2); mul_wide(E4, E5, a1, d3);
  E2 = mad_lo_cc(a1, a1, E2); E3 = madc_hi_cc(a1, a1, E3); E4 = madc_lo_cc(a2, a2, E4); E5 = madc_hi_cc(a2, a2, E5); E6 = addc(0, 0);
  E2 = mad_lo_cc(a3, e3, E2); E3 = madc_hi_cc(a3, e3, E3); E4 = addc_cc(E4, 0); E5 = addc_cc(E5, 0); E6 = addc(E6, 0);
  // odd lattice: W^1, W^3, W^5
  mul_wide(O1, O2, a0, e1); mul_wide(O3, O4, a0, d3); mul_wide(O5, O6, a2, e3);
  O3 = mad_lo_cc(a1, e2, O3); O4 = madc_hi_cc(a1, e2, O4); O5 = addc_cc(O5, 0); O6 = addc(O6, 0);
  u32 w1 = add_cc(E1, O1), w2 = addc_cc(E2, O2), w3 = addc_cc(E3, O3), w4 = addc_cc(E4, O4), w5 = addc_cc(E5, O5), w6 = addc(E6, O6);
  return fp_fold7(E0, w1, w2, w3, w4, w5, w6);
}

FQ_FN fp fp_nsqr(fp x, int n) {
  FQ_NOUNROLL
  for (int i = 0; i < n; i++) x = fp_sqr(x);
  return x;
}

// fields.py:67-106: x^(2^127-3) by the reference's addition chain (126 S + 12 M); inv(0) = 0.
FQ_FN fp fp_inv(const fp& x) {
  fp x3 = fp_mul(fp_sqr(x), x);                 // 2^2 - 1
  fp xf = fp_mul(fp_nsqr(x3, 2), x3);           // 2^4 - 1
  fp x8 = fp_mul(fp_nsqr(xf, 4), xf);           // 2^8 - 1
  fp x16 = fp_mul(fp_nsqr(x8, 8), x8);          // 2^16 - 1
  fp x32 = fp_mul(fp_nsqr(x16, 16), x16);       // 2^32 - 1
  fp t = fp_mul(fp_nsqr(x32, 32), x32);         // 2^64 - 1
  t = fp_mul(fp_nsqr(t, 32), x32);              // 2^96 - 1
  t = fp_mul(fp_nsqr(t, 16), x16);              // 2^112 - 1
  t = fp_mul(fp_nsqr(t, 8), x8);                // 2^120 - 1
  t = fp_mul(fp_nsqr(t, 4), xf);                // 2^124 - 1
  t = fp_mul(fp_sqr(t), x);                     // 2^125 - 1
  return fp_mul(fp_nsqr(t, 2), x);              // 2^127 - 3
}

// fields.py:110-122: x^(2^125-1) = x^((p-3)/4).  Same exponent, so the same value as the reference's chain.
FQ_FN fp fp_invsqrt(const fp& x) {
  fp x3 = fp_mul(fp_sqr(x), x);                 // 2^2 - 1
  fp xf = fp_mul(fp_nsqr(x3, 2), x3);           // 2^4 - 1
  fp x5 = fp_mul(fp_sqr(xf), x);                // 2^5 - 1
  fp x10 = fp_mul(fp_nsqr(x5, 5), x5);          // 2^10 - 1
  fp x20 = fp_mul(fp_nsqr(x10, 10), x10);       // 2^20 - 1
  fp x25 = fp_mul(fp_nsqr(x20, 5), x5);         // 2^25 - 1
  fp x50 = fp_mul(fp_nsqr(x25, 25), x25);       // 2^50 - 1
  fp x100 = fp_mul(fp_nsqr(x50, 50), x50);      // 2^100 - 1
  fp x125 = fp_mul(fp_nsqr(x100, 25), x25);     // 2^125 - 1
  return x125;
}
