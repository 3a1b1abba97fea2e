// pair_tower.cuh -- the Fq2/Fq6/Fq12 tower on LANE PAIRS.
//
// Two adjacent lanes (2p, 2p+1) of a warp work on one element: lane c holds coefficient c of every
// Fq2 value (x = x_0 + x_1 u), so an Fq2 is 12 registers per lane, an Fq12 72.  The partner's
// coefficient travels by `shfl.sync.bfly 1`.  Why (measured on B200, profiles/):
//   * the carry-linked IMAD.WIDE.U32.X that Montgomery products are made of issues once per 4
//     cycles per SM sub-partition; one warp alone reaches ~65 % of that, so the kernel needs >= 2-4
//     resident warps per sub-partition, and a thread-per-pairing kernel needs 255 registers (2 warps);
//   * halving the state per lane halves the registers, and halves the length of a warp task, which
//     also fixes the 2^16-batch tail (2048 warp tasks over 592 sub-partitions quantise to 86 %).
// An Fq2 product costs each lane ONE lazily-reduced dual product (fp_mul2: 444 MAC32), i.e. 888 per
// pair against 900 for the reference's Karatsuba (fq2.rs:123-136); a squaring costs one fp_mul per lane.
// Every function returns the same canonical value as the cited reference routine.
#pragma once
#include "tower.cuh"

namespace bls {

struct P2 { Fp v; };                 // own coefficient of an Fq2
struct P6 { P2 c0, c1, c2; };
struct P12 { P6 c0, c1; };

__device__ __forceinline__ int pair_c() { return threadIdx.x & 1; }

// partner lane's coefficient
__device__ __forceinline__ Fp pair_xchg(const Fp& a) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = __shfl_xor_sync(0xffffffffu, a.v[i], 1);
  return r;
}
__device__ __forceinline__ Fp fp_select(bool take_a, const Fp& a, const Fp& b) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = take_a ? a.v[i] : b.v[i];
  return r;
}

__device__ __forceinline__ P2 p2_zero() { return P2{fp_zero()}; }
__device__ __forceinline__ P2 p2_one() { return P2{pair_c() ? fp_zero() : fp_one()}; }
__device__ __forceinline__ P2 p2_add(const P2& a, const P2& b) { return P2{fp_add(a.v, b.v)}; }
__device__ __forceinline__ P2 p2_sub(const P2& a, const P2& b) { return P2{fp_sub(a.v, b.v)}; }
__device__ __forceinline__ P2 p2_dbl(const P2& a) { return P2{fp_dbl(a.v)}; }
__device__ __forceinline__ P2 p2_neg(const P2& a) { return P2{fp_neg(a.v)}; }
// both lanes learn whether the Fq2 value is zero
__device__ __forceinline__ bool p2_is_zero(const P2& a) {
  const bool z = fp_is_zero(a.v);
  const int zo = __shfl_xor_sync(0xffffffffu, (int)z, 1);      // unconditionally: `z && shfl(..)` would keep lanes with z == false out of the shuffle
  return z && zo;
}
// x (1 + u) = (c0 - c1) + (c0 + c1) u   (fq2.rs:41-45)
__device__ __forceinline__ P2 p2_mul_by_nonresidue(P2 a) {
  Fp oth = pair_xchg(a.v);
  // lane 0: c0 - c1 = own + (2q - oth);  lane 1: c1 + c0 = own + oth   (one folded addition instead of add, sub, select)
  return P2{fp_add(a.v, fp_select(pair_c() == 0, fp_neg(oth), oth))};
}
// fq2.rs:123-136: c0 = a0 b0 - a1 b1, c1 = a0 b1 + a1 b0, one lazily reduced dual product per lane
__device__ __forceinline__ P2 p2_mul(P2 a, P2 b) {
  Fp ao = pair_xchg(a.v), bo = pair_xchg(b.v);
  bool c0 = pair_c() == 0;
  // lane 0: a0 * b0 + (-a1) * b1        lane 1: a0 * b1 + a1 * b0   (X * b_own + Y * b_oth)
  Fp x = fp_select(c0, a.v, ao);
  Fp y = fp_select(c0, fp_neg(ao), a.v);
  return P2{fp_mul2(x, b.v, y, bo)};
}
// fq2.rs:87-101: c0 = (a0 + a1)(a0 - a1), c1 = 2 a0 a1
__device__ __forceinline__ P2 p2_sqr(P2 a) {
  Fp oth = pair_xchg(a.v);
  bool c0 = pair_c() == 0;
  Fp u = fp_add(fp_select(c0, a.v, oth), oth);           // lane 0: a0 + a1, lane 1: a0 + a0
  Fp w = fp_select(c0, fp_sub(a.v, oth), a.v);           // lane 0: a0 - a1, lane 1: a1
  return P2{fp_mul(u, w)};
}
// Fq2 x Fq: both coefficients scaled (mod.rs:61-65)
__device__ __forceinline__ P2 p2_mul_fp(const P2& a, const Fp& s) { return P2{fp_mul(a.v, s)}; }
// fq2.rs:138-155; returns false for zero.  Both lanes run the Fq inversion of the norm.
static __device__ __noinline__ bool p2_inv(P2& out, const P2& a) {
  Fp sq = fp_sqr(a.v);
  Fp t = fp_add(sq, pair_xchg(sq));
  Fp ti;
  bool ok = fp_inv(ti, t);       // lanes diverge inside (variable-time division steps) and re-converge at the next shuffle
  Fp r = fp_mul(a.v, ti);
  out.v = fp_select(pair_c() == 0, r, fp_neg(r));
  return ok;
}
// fq2.rs:157-159: c1 *= (-1)^((q^power - 1)/2)
__device__ __forceinline__ P2 p2_frobenius(const P2& a, int power) {
  return (power & 1) ? P2{fp_select(pair_c() == 0, a.v, fp_neg(a.v))} : a;
}
// constant Fq2 from a table entry: own coefficient
__device__ __forceinline__ P2 p2_from_const(const uint32_t (*p)[12]) { return P2{fp_from_const(p[pair_c()])}; }

// ------------------------------------------------------------------------------------------ Fq6
__device__ __forceinline__ void p6_add(P6& r, const P6& a, const P6& b) { r.c0 = p2_add(a.c0, b.c0); r.c1 = p2_add(a.c1, b.c1); r.c2 = p2_add(a.c2, b.c2); }
__device__ __forceinline__ void p6_sub(P6& r, const P6& a, const P6& b) { r.c0 = p2_sub(a.c0, b.c0); r.c1 = p2_sub(a.c1, b.c1); r.c2 = p2_sub(a.c2, b.c2); }
__device__ __forceinline__ void p6_neg(P6& r, const P6& a) { r.c0 = p2_neg(a.c0); r.c1 = p2_neg(a.c1); r.c2 = p2_neg(a.c2); }
__device__ __forceinline__ void p6_zero(P6& r) { r.c0 = p2_zero(); r.c1 = p2_zero(); r.c2 = p2_zero(); }
// fq6.rs:32-38
__device__ __forceinline__ void p6_mul_by_nonresidue(P6& r, const P6& a) {
  P2 t = p2_mul_by_nonresidue(a.c2);
  r.c2 = a.c1; r.c1 = a.c0; r.c0 = t;
}
// fq6.rs:199-248
static __device__ __noinline__ void p6_mul(P6& r, const P6& a, const P6& b) {
  P2 aa = p2_mul(a.c0, b.c0), bb = p2_mul(a.c1, b.c1), cc = p2_mul(a.c2, b.c2);
  P2 t1 = p2_mul(p2_add(b.c1, b.c2), p2_add(a.c1, a.c2));
  t1 = p2_add(p2_mul_by_nonresidue(p2_sub(p2_sub(t1, bb), cc)), aa);
  P2 t3 = p2_mul(p2_add(b.c0, b.c2), p2_add(a.c0, a.c2));
  t3 = p2_sub(p2_add(p2_sub(t3, aa), bb), cc);
  P2 t2 = p2_mul(p2_add(b.c0, b.c1), p2_add(a.c0, a.c1));
  t2 = p2_add(p2_sub(p2_sub(t2, aa), bb), p2_mul_by_nonresidue(cc));
  r.c0 = t1; r.c1 = t2; r.c2 = t3;
}
// fq6.rs:166-197
static __device__ __noinline__ void p6_sqr(P6& r, const P6& a) {
  P2 s0 = p2_sqr(a.c0);
  P2 s1 = p2_dbl(p2_mul(a.c0, a.c1));
  P2 s2 = p2_sqr(p2_add(p2_sub(a.c0, a.c1), a.c2));
  P2 s3 = p2_dbl(p2_mul(a.c1, a.c2));
  P2 s4 = p2_sqr(a.c2);
  r.c0 = p2_add(p2_mul_by_nonresidue(s3), s0);
  r.c1 = p2_add(p2_mul_by_nonresidue(s4), s1);
  r.c2 = p2_sub(p2_sub(p2_add(p2_add(s1, s2), s3), s0), s4);
}
// fq6.rs:40-66
__device__ __forceinline__ void p6_mul_by_1(P6& r, const P6& a, const P2& c1) {
  P2 bb = p2_mul(a.c1, c1);
  P2 t1 = p2_mul_by_nonresidue(p2_sub(p2_mul(c1, p2_add(a.c1, a.c2)), bb));
  P2 t2 = p2_sub(p2_mul(c1, p2_add(a.c0, a.c1)), bb);
  r.c0 = t1; r.c1 = t2; r.c2 = bb;
}
// fq6.rs:68-109
__device__ __forceinline__ void p6_mul_by_01(P6& r, const P6& a, const P2& c0, const P2& c1) {
  P2 aa = p2_mul(a.c0, c0);
  P2 bb = p2_mul(a.c1, c1);
  P2 t1 = p2_add(p2_mul_by_nonresidue(p2_sub(p2_mul(c1, p2_add(a.c1, a.c2)), bb)), aa);
  P2 t3 = p2_add(p2_sub(p2_mul(c0, p2_add(a.c0, a.c2)), aa), bb);
  P2 t2 = p2_sub(p2_sub(p2_mul(p2_add(c0, c1), p2_add(a.c0, a.c1)), aa), bb);
  r.c0 = t1; r.c1 = t2; r.c2 = t3;
}
// fq6.rs:250-301
static __device__ __noinline__ bool p6_inv(P6& r, const P6& a) {
  P2 c0 = p2_add(p2_neg(p2_mul(p2_mul_by_nonresidue(a.c2), a.c1)), p2_sqr(a.c0));
  P2 c1 = p2_sub(p2_mul_by_nonresidue(p2_sqr(a.c2)), p2_mul(a.c0, a.c1));
  P2 c2 = p2_sub(p2_sqr(a.c1), p2_mul(a.c0, a.c2));
  P2 t = p2_mul_by_nonresidue(p2_add(p2_mul(a.c2, c1), p2_mul(a.c1, c2)));
  t = p2_add(t, p2_mul(a.c0, c0));
  P2 ti;
  bool ok = p2_inv(ti, t);
  r.c0 = p2_mul(ti, c0); r.c1 = p2_mul(ti, c1); r.c2 = p2_mul(ti, c2);
  return ok;
}
// fq6.rs:157-164
static __device__ __noinline__ void p6_frobenius(P6& r, const P6& a, int power) {
  P2 c0 = p2_frobenius(a.c0, power);
  P2 c1 = p2_mul(p2_frobenius(a.c1, power), p2_from_const(BLS_FROB_FQ6_C1[power % 6]));
  P2 c2 = p2_mul(p2_frobenius(a.c2, power), p2_from_const(BLS_FROB_FQ6_C2[power % 6]));
  r.c0 = c0; r.c1 = c1; r.c2 = c2;
}

// ------------------------------------------------------------------------------------------ Fq12
__device__ __forceinline__ void p12_one(P12& r) { p6_zero(r.c0); p6_zero(r.c1); r.c0.c0 = p2_one(); }
__device__ __forceinline__ void p12_conjugate(P12& a) { p6_neg(a.c1, a.c1); }   // fq12.rs:30-32
__device__ __forceinline__ void p6_select(P6& r, bool take_a, const P6& a, const P6& b) {
  r.c0.v = fp_select(take_a, a.c0.v, b.c0.v); r.c1.v = fp_select(take_a, a.c1.v, b.c1.v); r.c2.v = fp_select(take_a, a.c2.v, b.c2.v);
}
__device__ __forceinline__ void p12_select(P12& r, bool take_a, const P12& a, const P12& b) { p6_select(r.c0, take_a, a.c0, b.c0); p6_select(r.c1, take_a, a.c1, b.c1); }
// fq12.rs:116-130 (r may alias a or b)
static __device__ __noinline__ void p12_mul(P12& r, const P12& a, const P12& b) {
  P6 aa, bb, o, s;
  p6_mul(aa, a.c0, b.c0);
  p6_mul(bb, a.c1, b.c1);
  p6_add(o, b.c0, b.c1);
  p6_add(s, a.c1, a.c0);
  p6_mul(s, s, o);
  p6_sub(s, s, aa);
  p6_sub(r.c1, s, bb);
  p6_mul_by_nonresidue(bb, bb);
  p6_add(r.c0, bb, aa);
}
// fq12.rs:99-114
__device__ __forceinline__ void p12_sqr(P12& r, const P12& a) {
  P6 ab, c0c1, c0;
  p6_mul(ab, a.c0, a.c1);
  p6_add(c0c1, a.c0, a.c1);
  p6_mul_by_nonresidue(c0, a.c1);
  p6_add(c0, c0, a.c0);
  p6_mul(c0, c0, c0c1);
  p6_sub(c0, c0, ab);
  p6_add(r.c1, ab, ab);
  p6_mul_by_nonresidue(ab, ab);
  p6_sub(r.c0, c0, ab);
}
// Squaring for elements of the cyclotomic subgroup (Granger-Scott, "Faster squaring in the cyclotomic subgroup of sixth
// degree extensions"): three Fq4 squarings, 18 M instead of the 36 M of the generic fq12.rs:99-114.  Only used inside
// exp_by_x, whose operand lies in the cyclotomic subgroup after the easy part of the final exponentiation, where it
// returns the same field value as `square`.  z' = 3t - 2z for the "real" parts, 3t + 2z for the "imaginary" ones.
__device__ __forceinline__ void p4_sqr(P2& t0, P2& t1, const P2& a, const P2& b) {
  P2 tmp = p2_mul(a, b);
  P2 s = p2_mul(p2_add(a, b), p2_add(p2_mul_by_nonresidue(b), a));
  t0 = p2_sub(p2_sub(s, tmp), p2_mul_by_nonresidue(tmp));
  t1 = p2_dbl(tmp);
}
static __device__ __noinline__ void p12_cyclotomic_sqr(P12& r, const P12& f) {
  P2 t0, t1, t2, t3, t4, t5;
  p4_sqr(t0, t1, f.c0.c0, f.c1.c1);
  p4_sqr(t2, t3, f.c1.c0, f.c0.c2);
  p4_sqr(t4, t5, f.c0.c1, f.c1.c2);
  P2 z0 = p2_sub(t0, f.c0.c0); z0 = p2_add(p2_dbl(z0), t0);
  P2 z1 = p2_add(t1, f.c1.c1); z1 = p2_add(p2_dbl(z1), t1);
  P2 x5 = p2_mul_by_nonresidue(t5);
  P2 z2 = p2_add(x5, f.c1.c0); z2 = p2_add(p2_dbl(z2), x5);
  P2 z3 = p2_sub(t4, f.c0.c2); z3 = p2_add(p2_dbl(z3), t4);
  P2 z4 = p2_sub(t2, f.c0.c1); z4 = p2_add(p2_dbl(z4), t2);
  P2 z5 = p2_add(t3, f.c1.c2); z5 = p2_add(p2_dbl(z5), t3);
  r.c0.c0 = z0; r.c0.c1 = z4; r.c0.c2 = z3;
  r.c1.c0 = z2; r.c1.c1 = z1; r.c1.c2 = z5;
}
// fq12.rs:34-48
static __device__ __noinline__ void p12_mul_by_014(P12& f, const P2& c0, const P2& c1, const P2& c4) {
  P6 aa, bb, s;
  p6_mul_by_01(aa, f.c0, c0, c1);
  p6_mul_by_1(bb, f.c1, c4);
  P2 o = p2_add(c1, c4);
  p6_add(s, f.c1, f.c0);
  p6_mul_by_01(s, s, c0, o);
  p6_sub(s, s, aa);
  p6_sub(f.c1, s, bb);
  p6_mul_by_nonresidue(bb, bb);
  p6_add(f.c0, bb, aa);
}
// fq12.rs:132-148
static __device__ __noinline__ bool p12_inv(P12& r, const P12& a) {
  P6 c0s, c1s, t;
  p6_sqr(c0s, a.c0);
  p6_sqr(c1s, a.c1);
  p6_mul_by_nonresidue(c1s, c1s);
  p6_sub(c0s, c0s, c1s);
  bool ok = p6_inv(t, c0s);
  p6_mul(c0s, t, a.c0);
  p6_mul(c1s, t, a.c1);
  r.c0 = c0s;
  p6_neg(r.c1, c1s);
  return ok;
}
// fq12.rs:90-97
static __device__ __noinline__ void p12_frobenius(P12& r, const P12& a, int power) {
  p6_frobenius(r.c0, a.c0, power);
  p6_frobenius(r.c1, a.c1, power);
  P2 k = p2_from_const(BLS_FROB_FQ12_C1[power % 12]);
  r.c1.c0 = p2_mul(r.c1.c0, k);
  r.c1.c1 = p2_mul(r.c1.c1, k);
  r.c1.c2 = p2_mul(r.c1.c2, k);
}

// ------------------------------------------------------------------------------------------ pairing on lane pairs
struct PCoeffs { P2 c0, c1, c2; };
struct PJac { P2 x, y, z; };

// mod.rs:176-245
static __device__ __noinline__ void pg2_doubling_step(PJac& r, PCoeffs& out) {
  P2 tmp0 = p2_sqr(r.x);
  P2 tmp1 = p2_sqr(r.y);
  P2 tmp2 = p2_sqr(tmp1);
  P2 tmp3 = p2_dbl(p2_sub(p2_sub(p2_sqr(p2_add(tmp1, r.x)), tmp0), tmp2));
  P2 tmp4 = p2_add(p2_dbl(tmp0), tmp0);
  P2 tmp6 = p2_add(r.x, tmp4);
  P2 tmp5 = p2_sqr(tmp4);
  P2 zsq = p2_sqr(r.z);
  r.x = p2_sub(p2_sub(tmp5, tmp3), tmp3);
  r.z = p2_sub(p2_sub(p2_sqr(p2_add(r.z, r.y)), tmp1), zsq);
  r.y = p2_sub(p2_mul(p2_sub(tmp3, r.x), tmp4), p2_dbl(p2_dbl(p2_dbl(tmp2))));
  out.c1 = p2_neg(p2_dbl(p2_mul(tmp4, zsq)));
  out.c2 = p2_sub(p2_sub(p2_sub(p2_sqr(tmp6), tmp0), tmp5), p2_dbl(p2_dbl(tmp1)));
  out.c0 = p2_dbl(p2_mul(r.z, zsq));
}
// mod.rs:247-333
static __device__ __noinline__ void pg2_addition_step(PJac& r, const P2& qx, const P2& qy, PCoeffs& out) {
  P2 zsq = p2_sqr(r.z);
  P2 ysq = p2_sqr(qy);
  P2 t0 = p2_mul(zsq, qx);
  P2 t1 = p2_mul(p2_sub(p2_sub(p2_sqr(p2_add(qy, r.z)), ysq), zsq), zsq);
  P2 t2 = p2_sub(t0, r.x);
  P2 t3 = p2_sqr(t2);
  P2 t4 = p2_dbl(p2_dbl(t3));
  P2 t5 = p2_mul(t4, t2);
  P2 t6 = p2_sub(p2_sub(t1, r.y), r.y);
  P2 t9 = p2_mul(t6, qx);
  P2 t7 = p2_mul(t4, r.x);
  r.x = p2_sub(p2_sub(p2_sub(p2_sqr(t6), t5), t7), t7);
  r.z = p2_sub(p2_sub(p2_sqr(p2_add(r.z, t2)), zsq), t3);
  P2 t10 = p2_add(qy, r.z);
  P2 t8 = p2_mul(p2_sub(t7, r.x), t6);
  r.y = p2_sub(t8, p2_dbl(p2_mul(r.y, t5)));
  t10 = p2_sub(p2_sub(p2_sqr(t10), ysq), p2_sqr(r.z));
  out.c2 = p2_sub(p2_dbl(t9), t10);
  out.c0 = p2_dbl(r.z);
  out.c1 = p2_dbl(p2_neg(t6));
}
// mod.rs:57-69
__device__ __forceinline__ void p_ell(P12& f, const PCoeffs& c, const Fp& px, const Fp& py) {
  P2 c0 = p2_mul_fp(c.c0, py);
  P2 c1 = p2_mul_fp(c.c1, px);
  p12_mul_by_014(f, c.c2, c1, c0);
}

// Multi-pairing only: the line values of TWO pairs are multiplied with each other before they touch the accumulator.
// A line is the sparse Fq12 element (c0 + c1 v) + (c4 v) w of fq12.rs:34-48 (w^2 = v, v^3 = xi), so
//   l * m = (l0 m0 + xi l4 m4) + (l0 m1 + l1 m0) v + (l1 m1) v^2 + [(l0 m4 + l4 m0) v + (l1 m4 + l4 m1) v^2] w
// costs six Fq2 products (Karatsuba on the three cross terms) and f * (l m), with the w-part's constant coefficient zero,
// 6 + 5 + 6 = 17: 23 Fq2 products for two pairs instead of 2 x 13 with mul_by_014.  The VALUE of f is the same product
// of the same field elements (multiplication in Fq12 is associative and commutative), so the canonical output is
// identical to the reference's bit for bit.
struct PLine { P2 c0, c1, c4; };
__device__ __forceinline__ PLine p_line(const PCoeffs& c, const Fp& px, const Fp& py) {
  return PLine{c.c2, p2_mul_fp(c.c1, px), p2_mul_fp(c.c0, py)};
}
// `single` (warp-uniform): only the line l is multiplied in (the odd pair left over at the end of a trip sequence).  It costs 17 Fq2
// products instead of the 13 of mul_by_014, but stays on the instruction stream the pairs use: with mul_by_014 as the leftover path
// every (bit, phase) of an odd trip count pulled another ~40 KB of code through the instruction cache (+ 2.4 ms per 2^17-pair launch).
static __device__ __noinline__ void p12_mul_by_line_pair(P12& f, const PLine& l, const PLine& m, bool single = false) {
  P12 lm;
  if (!single) {
    P2 m00 = p2_mul(l.c0, m.c0), m11 = p2_mul(l.c1, m.c1), m44 = p2_mul(l.c4, m.c4);
    lm.c0.c1 = p2_sub(p2_sub(p2_mul(p2_add(l.c0, l.c1), p2_add(m.c0, m.c1)), m00), m11);
    lm.c1.c1 = p2_sub(p2_sub(p2_mul(p2_add(l.c0, l.c4), p2_add(m.c0, m.c4)), m00), m44);
    lm.c1.c2 = p2_sub(p2_sub(p2_mul(p2_add(l.c1, l.c4), p2_add(m.c1, m.c4)), m11), m44);
    lm.c0.c0 = p2_add(m00, p2_mul_by_nonresidue(m44));
    lm.c0.c2 = m11;
  } else {                                       // l * one
    lm.c0.c0 = l.c0; lm.c0.c1 = l.c1; lm.c0.c2 = p2_zero();
    lm.c1.c1 = l.c4; lm.c1.c2 = p2_zero();
  }
  P6 aa, bb, s;
  p6_mul(aa, f.c0, lm.c0);
  p6_mul_by_01(bb, f.c1, lm.c1.c1, lm.c1.c2);    // f.c1 * (0, d1, d2) = v * (f.c1 * (d1, d2, 0))
  p6_mul_by_nonresidue(bb, bb);
  lm.c0.c1 = p2_add(lm.c0.c1, lm.c1.c1);         // lm.c0 + lm.c1 (the w-part has no constant coefficient)
  lm.c0.c2 = p2_add(lm.c0.c2, lm.c1.c2);
  p6_add(s, f.c1, f.c0);
  p6_mul(s, s, lm.c0);
  p6_sub(s, s, aa);
  p6_sub(f.c1, s, bb);
  p6_mul_by_nonresidue(bb, bb);
  p6_add(f.c0, bb, aa);
}

// The loop schedule: bits of BLS_X >> 1 = 0x6900800000008000 below the leading one, MSB first (mod.rs:72-78)
#define BLS_LOOP_BITS (BLS_X_ABS >> 1)
#define BLS_LOOP_TOP 61   /* bit 62 is the leading one */

// mod.rs:40-102 for one pair, G2 steps on the fly
// (no early exit for pairs with an infinity member: every lane must reach every shuffle; the
// caller overwrites f with one for those pairs)
__device__ __forceinline__ void p_miller_loop_single(P12& f, const Fp& px, const Fp& py, const P2& qx, const P2& qy) {
  p12_one(f);
  PCoeffs c;
  PJac r;
  r.x = qx; r.y = qy; r.z = p2_one();
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= 0; b--) {
    pg2_doubling_step(r, c);
    p_ell(f, c, px, py);
    if ((BLS_LOOP_BITS >> b) & 1ull) {
      pg2_addition_step(r, qx, qy, c);
      p_ell(f, c, px, py);
    }
    p12_sqr(f, f);
  }
  pg2_doubling_step(r, c);
  p_ell(f, c, px, py);
  p12_conjugate(f);
}

// exp_by_x (mod.rs:116-121): Field::pow(&[x]) (lib.rs:306-324) followed by a conjugation.  Two value-preserving
// shortcuts (SURVEY.md 8c "latitude"): the leading `one * self` product of pow is a copy, and -- the operand being
// in the cyclotomic subgroup (exp_by_x is only called after the easy part) -- every squaring is a Granger-Scott
// cyclotomic squaring.
static __device__ __noinline__ void p12_exp_by_x(P12& out, const P12& a, uint64_t x) {
  P12 res = a;
  const int top = 63 - __clzll((long long)x);
#pragma unroll 1
  for (int n = top - 1; n >= 0; n--) {
    p12_cyclotomic_sqr(res, res);
    if ((x >> n) & 1ull) p12_mul(res, res, a);
  }
  p12_conjugate(res);
  out = res;
}

// exp_by_x on COMPRESSED cyclotomic elements (Karabina, "Squaring in cyclotomic subgroups", Math. Comp. 2013).  With
// Fq12 = Fq4[w]/(w^3 - s), Fq4 = Fq2[s]/(s^2 - xi) the element is G0 + G1 w + G2 w^2 with G0 = (c0.c0, c1.c1),
// G1 = (c1.c0, c0.c2), G2 = (c0.c1, c1.c2), and the Granger-Scott squaring above computes the new G1, G2 from the old
// G1, G2 alone: dropping G0 leaves two Fq4 squarings -- FOUR Fq2 products per squaring instead of six.  G0 is recovered
// when a power is needed in full:
//   g1 = (xi g5^2 + 3 g4^2 - 2 g3) / (4 g2),   g0 = (2 g1^2 + g2 g5 - 3 g3 g4) xi + 1
// (g2 = c1.c0, g3 = c0.c2, g4 = c0.c1, g5 = c1.c2, g0 = c0.c0, g1 = c1.c1).  The exponent is walked from its LOW end:
// the powers a^(2^b) of the set bits b are kept compressed, decompressed together (one Fq2 inversion for all of them,
// Montgomery's trick) and multiplied -- as many Fq12 products as the square-and-multiply of lib.rs:306-324 needs, the
// same field value, hence the same canonical output.  A zero denominator (g2 = 0: the element one, e.g. a pair with a
// point at infinity) cannot be decompressed this way: the warp then also runs the uncompressed p12_exp_by_x and the
// lane pairs concerned take its result (warp-uniform control flow: every lane reaches every shuffle).
struct PK4 { P2 g2, g3, g4, g5; };
static __device__ __noinline__ void pk4_sqr(PK4& c) {
  P2 t2, t3, t4, t5;
  p4_sqr(t2, t3, c.g2, c.g3);
  p4_sqr(t4, t5, c.g4, c.g5);
  const P2 x5 = p2_mul_by_nonresidue(t5);
  P2 z2 = p2_add(x5, c.g2); z2 = p2_add(p2_dbl(z2), x5);
  P2 z3 = p2_sub(t4, c.g3); z3 = p2_add(p2_dbl(z3), t4);
  P2 z4 = p2_sub(t2, c.g4); z4 = p2_add(p2_dbl(z4), t2);
  P2 z5 = p2_add(t3, c.g5); z5 = p2_add(p2_dbl(z5), t3);
  c.g2 = z2; c.g3 = z3; c.g4 = z4; c.g5 = z5;
}
// BLS_EXP_NCOMP: how many of the set bits (from the low end) are reached by compressed squarings.  3: the powers at
// bits 16, 48, 57 are decompressed and the three close bits above (60, 62, 63) are reached from the decompressed a^(2^57) by six
// uncompressed cyclotomic squarings -- 12 Fq2 products fewer per call than decompressing all six powers (BLS_EXP_NCOMP = 6) and
// half the stored powers: 42.6 - 43.4 ms against 45.4 ms per 2^16 pairings for 6 in this code shape (4: 43.4 - 44.1 ms), same GPU call;
// the earlier all-six build measured 43.1 - 44.6 ms over its boxes, this one 42.6 - 44.0 ms.
#define BLS_EXP_NCOMP 3
static __device__ __noinline__ void p12_exp_by_x_compressed(P12& out, const P12& a, uint64_t x) {
  PK4 pts[BLS_EXP_NCOMP];
  P2 pre[BLS_EXP_NCOMP];
  PK4 c{a.c1.c0, a.c0.c2, a.c0.c1, a.c1.c2};
  const int top = 63 - __clzll((long long)x);
  int k = 0, b = 1;
#pragma unroll 1
  for (; b <= top && k < BLS_EXP_NCOMP; b++) {
    pk4_sqr(c);
    if ((x >> b) & 1ull) {
      pts[k] = c;
      const P2 den = p2_dbl(p2_dbl(c.g2));
      pre[k] = k ? p2_mul(pre[k - 1], den) : den;            // prefix products of the denominators 4 g2
      k++;
    }
  }
  const bool bad = p2_is_zero(pre[k - 1]);
  P2 inv;
  p2_inv(inv, pre[k - 1]);
  P12 res, hi;
#pragma unroll 1
  for (int i = k - 1; i >= 0; i--) {
    const PK4 g = pts[i];
    P2 dinv = inv;
    if (i) { dinv = p2_mul(inv, pre[i - 1]); inv = p2_mul(inv, p2_dbl(p2_dbl(g.g2))); }
    const P2 s4 = p2_sqr(g.g4);
    const P2 num = p2_sub(p2_add(p2_mul_by_nonresidue(p2_sqr(g.g5)), p2_add(p2_dbl(s4), s4)), p2_dbl(g.g3));
    const P2 g1 = p2_mul(num, dinv);
    const P2 m34 = p2_mul(g.g3, g.g4);
    const P2 t = p2_sub(p2_add(p2_dbl(p2_sqr(g1)), p2_mul(g.g2, g.g5)), p2_add(p2_dbl(m34), m34));
    P12 e;
    e.c0.c0 = p2_add(p2_mul_by_nonresidue(t), p2_one());
    e.c0.c1 = g.g4; e.c0.c2 = g.g3;
    e.c1.c0 = g.g2; e.c1.c1 = g1; e.c1.c2 = g.g5;
    if (i == k - 1) { res = e; hi = e; } else p12_mul(res, res, e);
  }
#pragma unroll 1
  for (; b <= top; b++) {                                    // the set bits above the last compressed one: uncompressed squarings
    p12_cyclotomic_sqr(hi, hi);
    if ((x >> b) & 1ull) p12_mul(res, res, hi);
  }
  if (x & 1ull) p12_mul(res, res, a);
  p12_conjugate(res);
  if (__any_sync(0xffffffffu, bad)) {
    P12 alt;
    p12_exp_by_x(alt, a, x);
    p12_select(res, bad, alt, res);
  }
  out = res;
}

// both lanes learn whether the Fq12 value is zero
__device__ __forceinline__ bool p12_is_zero(const P12& a) {
  bool z = fp_is_zero(a.c0.c0.v) && fp_is_zero(a.c0.c1.v) && fp_is_zero(a.c0.c2.v) &&
           fp_is_zero(a.c1.c0.v) && fp_is_zero(a.c1.c1.v) && fp_is_zero(a.c1.c2.v);
  const int zo = __shfl_xor_sync(0xffffffffu, (int)z, 1);
  return z && zo;
}

// both lanes learn whether the two Fq12 values are equal
__device__ __forceinline__ bool p12_eq(const P12& a, const P12& b) {
  const bool e = fp_eq(a.c0.c0.v, b.c0.c0.v) && fp_eq(a.c0.c1.v, b.c0.c1.v) && fp_eq(a.c0.c2.v, b.c0.c2.v) &&
                 fp_eq(a.c1.c0.v, b.c1.c0.v) && fp_eq(a.c1.c1.v, b.c1.c1.v) && fp_eq(a.c1.c2.v, b.c1.c2.v);
  const int eo = __shfl_xor_sync(0xffffffffu, (int)e, 1);
  return e && eo;
}

// mod.rs:104-160
// y0 = r^2 by the generic 12-product squaring.  The 6-product cyclotomic squaring gives the same value (r is in the cyclotomic
// subgroup after the easy part) but lost: under bench.py's conditions (L2 flushed between launches) the fused kernel measured
// 45.3 - 45.5 ms with it and 43.1 - 44.6 ms without, three boxes; back to back without the flush the two builds are equal
// (43.2 ms).  That variant was removed; it can be recovered from git history at commit 7b088bd.
__device__ __forceinline__ bool p_final_exponentiation(P12& out, const P12& in) {
  P12 f1 = in, f2, r;
  p12_conjugate(f1);
  const bool ok = p12_inv(f2, in);      // no early exit (shuffles below); a zero input is patched at the end
  p12_mul(r, f1, f2);
  f2 = r;
  p12_frobenius(r, r, 2);
  p12_mul(r, r, f2);
  const uint64_t x = BLS_X_ABS;
  P12 y0, y1, y2, y3;
  p12_sqr(y0, r);
  p12_exp_by_x_compressed(y1, y0, x);
  p12_exp_by_x_compressed(y2, y1, x >> 1);
  y3 = r; p12_conjugate(y3);
  p12_mul(y1, y1, y3);
  p12_conjugate(y1);
  p12_mul(y1, y1, y2);
  p12_exp_by_x_compressed(y2, y1, x);
  p12_exp_by_x_compressed(y3, y2, x);
  p12_conjugate(y1);
  p12_mul(y3, y3, y1);
  p12_conjugate(y1);
  p12_frobenius(y1, y1, 3);
  p12_frobenius(y2, y2, 2);
  p12_mul(y1, y1, y2);
  p12_exp_by_x_compressed(y2, y3, x);
  p12_mul(y2, y2, y0);
  p12_mul(y2, y2, r);
  p12_mul(y1, y1, y2);
  p12_frobenius(y2, y3, 1);
  p12_mul(y1, y1, y2);
  out = y1;
  if (!ok) { p6_zero(out.c0); p6_zero(out.c1); }
  return ok;
}

}  // namespace bls
