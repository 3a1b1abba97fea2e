// tower.cuh -- Fq2 / Fq6 / Fq12 on top of fp.cuh.
//   Fq2  = Fq[u]/(u^2+1)          (reference: bls12_381/fq2.rs)
//   Fq6  = Fq2[v]/(v^3-(1+u))     (bls12_381/fq6.rs)
//   Fq12 = Fq6[w]/(w^2-v)         (bls12_381/fq12.rs)
// Every function returns the same canonical field value as the cited reference routine; the
// operation order inside a routine is free (values are canonical after every Fq op).
#pragma once
#include "constants.cuh"
#include "fp.cuh"
#include "fp_inv_gcd.cuh"

namespace bls {

struct Fp2 { Fp c0, c1; };
struct Fp6 { Fp2 c0, c1, c2; };
struct Fp12 { Fp6 c0, c1; };

__device__ __forceinline__ Fp fp_from_const(const uint32_t* p) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = p[i];
  return r;
}

// ------------------------------------------------------------------------------------------ Fq2
__device__ __forceinline__ Fp2 fp2_zero() { return Fp2{fp_zero(), fp_zero()}; }
__device__ __forceinline__ Fp2 fp2_one() { return Fp2{fp_one(), fp_zero()}; }
__device__ __forceinline__ bool fp2_is_zero(const Fp2& a) { return fp_is_zero(a.c0) && fp_is_zero(a.c1); }
__device__ __forceinline__ bool fp2_eq(const Fp2& a, const Fp2& b) { return fp_eq(a.c0, b.c0) && fp_eq(a.c1, b.c1); }
__device__ __forceinline__ Fp2 fp2_add(const Fp2& a, const Fp2& b) { return Fp2{fp_add(a.c0, b.c0), fp_add(a.c1, b.c1)}; }
__device__ __forceinline__ Fp2 fp2_sub(const Fp2& a, const Fp2& b) { return Fp2{fp_sub(a.c0, b.c0), fp_sub(a.c1, b.c1)}; }
__device__ __forceinline__ Fp2 fp2_dbl(const Fp2& a) { return Fp2{fp_dbl(a.c0), fp_dbl(a.c1)}; }
__device__ __forceinline__ Fp2 fp2_neg(const Fp2& a) { return Fp2{fp_neg(a.c0), fp_neg(a.c1)}; }
// x (1 + u): fq2.rs:41-45
__device__ __forceinline__ Fp2 fp2_mul_by_nonresidue(const Fp2& a) { return Fp2{fp_sub(a.c0, a.c1), fp_add(a.c0, a.c1)}; }

// Karatsuba, fq2.rs:123-136
static __device__ __noinline__ Fp2 fp2_mul(Fp2 a, Fp2 b) {
  Fp aa = fp_mul(a.c0, b.c0);
  Fp bb = fp_mul(a.c1, b.c1);
  Fp s = fp_mul(fp_add(a.c0, a.c1), fp_add(b.c0, b.c1));
  return Fp2{fp_sub(aa, bb), fp_sub(fp_sub(s, aa), bb)};
}
// complex squaring, fq2.rs:87-101
static __device__ __noinline__ Fp2 fp2_sqr(Fp2 a) {
  Fp ab = fp_mul(a.c0, a.c1);
  Fp t = fp_mul(fp_add(a.c0, a.c1), fp_sub(a.c0, a.c1));
  return Fp2{t, fp_dbl(ab)};
}
// Fq2 x Fq (the `ell` scalings, mod.rs:61-65)
__device__ __forceinline__ Fp2 fp2_mul_fp(const Fp2& a, const Fp& s) { return Fp2{fp_mul(a.c0, s), fp_mul(a.c1, s)}; }

// Fq inversion (fq.rs:849-902).  The reference runs a binary extended Euclid; the inverse is unique and the result is
// canonical, so the algorithm is free: Bernstein-Yang division steps on signed 30-bit limbs (fp_inv_gcd.cuh), about a
// tenth of the multiplier work of the Fermat power a^(q-2) that round 1 used (removed; it can be recovered from git history
// at commit 7b088bd).  Returns false (and zero) for a == 0, the reference's `None`.
static __device__ __noinline__ bool fp_inv(Fp& out, const Fp& a) {
  const Fp c = fp_canon(a);
  gcd30::invert_words(out.v, c.v);
  return !fp_is_zero_raw(c);
}

// fq2.rs:138-155
__device__ __forceinline__ bool fp2_inv(Fp2& out, const Fp2& a) {
  Fp t = fp_add(fp_sqr(a.c0), fp_sqr(a.c1));
  Fp ti;
  bool ok = fp_inv(ti, t);
  out = Fp2{fp_mul(a.c0, ti), fp_neg(fp_mul(a.c1, ti))};
  return ok;
}
// fq2.rs:157-159
__device__ __forceinline__ Fp2 fp2_frobenius(const Fp2& a, int power) {
  return Fp2{a.c0, fp_mul(a.c1, fp_from_const(BLS_FROB_FQ2_C1[power & 1]))};
}
__device__ __forceinline__ Fp2 fp2_from_const(const uint32_t (*p)[12]) { return Fp2{fp_from_const(p[0]), fp_from_const(p[1])}; }

// ------------------------------------------------------------------------------------------ Fq6
__device__ __forceinline__ Fp6 fp6_zero() { return Fp6{fp2_zero(), fp2_zero(), fp2_zero()}; }
__device__ __forceinline__ Fp6 fp6_one() { return Fp6{fp2_one(), fp2_zero(), fp2_zero()}; }
__device__ __forceinline__ bool fp6_is_zero(const Fp6& a) { return fp2_is_zero(a.c0) && fp2_is_zero(a.c1) && fp2_is_zero(a.c2); }
__device__ __forceinline__ void fp6_add(Fp6& r, const Fp6& a, const Fp6& b) { r.c0 = fp2_add(a.c0, b.c0); r.c1 = fp2_add(a.c1, b.c1); r.c2 = fp2_add(a.c2, b.c2); }
__device__ __forceinline__ void fp6_sub(Fp6& r, const Fp6& a, const Fp6& b) { r.c0 = fp2_sub(a.c0, b.c0); r.c1 = fp2_sub(a.c1, b.c1); r.c2 = fp2_sub(a.c2, b.c2); }
__device__ __forceinline__ void fp6_neg(Fp6& r, const Fp6& a) { r.c0 = fp2_neg(a.c0); r.c1 = fp2_neg(a.c1); r.c2 = fp2_neg(a.c2); }
// x v: fq6.rs:32-38
__device__ __forceinline__ void fp6_mul_by_nonresidue(Fp6& r, const Fp6& a) {
  Fp2 t = fp2_mul_by_nonresidue(a.c2);
  r.c2 = a.c1; r.c1 = a.c0; r.c0 = t;
}
// fq6.rs:199-248
static __device__ __noinline__ void fp6_mul(Fp6& r, const Fp6& a, const Fp6& b) {
  Fp2 aa = fp2_mul(a.c0, b.c0), bb = fp2_mul(a.c1, b.c1), cc = fp2_mul(a.c2, b.c2);
  Fp2 t1 = fp2_mul(fp2_add(b.c1, b.c2), fp2_add(a.c1, a.c2));
  t1 = fp2_add(fp2_mul_by_nonresidue(fp2_sub(fp2_sub(t1, bb), cc)), aa);
  Fp2 t3 = fp2_mul(fp2_add(b.c0, b.c2), fp2_add(a.c0, a.c2));
  t3 = fp2_sub(fp2_add(fp2_sub(t3, aa), bb), cc);
  Fp2 t2 = fp2_mul(fp2_add(b.c0, b.c1), fp2_add(a.c0, a.c1));
  t2 = fp2_add(fp2_sub(fp2_sub(t2, aa), bb), fp2_mul_by_nonresidue(cc));
  r.c0 = t1; r.c1 = t2; r.c2 = t3;
}
// fq6.rs:166-197
static __device__ __noinline__ void fp6_sqr(Fp6& r, const Fp6& a) {
  Fp2 s0 = fp2_sqr(a.c0);
  Fp2 s1 = fp2_dbl(fp2_mul(a.c0, a.c1));
  Fp2 s2 = fp2_sqr(fp2_add(fp2_sub(a.c0, a.c1), a.c2));
  Fp2 s3 = fp2_dbl(fp2_mul(a.c1, a.c2));
  Fp2 s4 = fp2_sqr(a.c2);
  r.c0 = fp2_add(fp2_mul_by_nonresidue(s3), s0);
  r.c1 = fp2_add(fp2_mul_by_nonresidue(s4), s1);
  r.c2 = fp2_sub(fp2_sub(fp2_add(fp2_add(s1, s2), s3), s0), s4);
}
// fq6.rs:40-66
static __device__ __noinline__ void fp6_mul_by_1(Fp6& r, const Fp6& a, const Fp2& c1) {
  Fp2 bb = fp2_mul(a.c1, c1);
  Fp2 t1 = fp2_mul_by_nonresidue(fp2_sub(fp2_mul(c1, fp2_add(a.c1, a.c2)), bb));
  Fp2 t2 = fp2_sub(fp2_mul(c1, fp2_add(a.c0, a.c1)), bb);
  r.c0 = t1; r.c1 = t2; r.c2 = bb;
}
// fq6.rs:68-109
static __device__ __noinline__ void fp6_mul_by_01(Fp6& r, const Fp6& a, const Fp2& c0, const Fp2& c1) {
  Fp2 aa = fp2_mul(a.c0, c0);
  Fp2 bb = fp2_mul(a.c1, c1);
  Fp2 t1 = fp2_add(fp2_mul_by_nonresidue(fp2_sub(fp2_mul(c1, fp2_add(a.c1, a.c2)), bb)), aa);
  Fp2 t3 = fp2_add(fp2_sub(fp2_mul(c0, fp2_add(a.c0, a.c2)), aa), bb);
  Fp2 t2 = fp2_sub(fp2_sub(fp2_mul(fp2_add(c0, c1), fp2_add(a.c0, a.c1)), aa), bb);
  r.c0 = t1; r.c1 = t2; r.c2 = t3;
}
// fq6.rs:250-301
static __device__ __noinline__ bool fp6_inv(Fp6& r, const Fp6& a) {
  Fp2 c0 = fp2_add(fp2_neg(fp2_mul(fp2_mul_by_nonresidue(a.c2), a.c1)), fp2_sqr(a.c0));
  Fp2 c1 = fp2_sub(fp2_mul_by_nonresidue(fp2_sqr(a.c2)), fp2_mul(a.c0, a.c1));
  Fp2 c2 = fp2_sub(fp2_sqr(a.c1), fp2_mul(a.c0, a.c2));
  Fp2 t = fp2_mul_by_nonresidue(fp2_add(fp2_mul(a.c2, c1), fp2_mul(a.c1, c2)));
  t = fp2_add(t, fp2_mul(a.c0, c0));
  Fp2 ti;
  bool ok = fp2_inv(ti, t);
  r.c0 = fp2_mul(ti, c0); r.c1 = fp2_mul(ti, c1); r.c2 = fp2_mul(ti, c2);
  return ok;
}
// fq6.rs:157-164
static __device__ __noinline__ void fp6_frobenius(Fp6& r, const Fp6& a, int power) {
  Fp2 c0 = fp2_frobenius(a.c0, power);
  Fp2 c1 = fp2_mul(fp2_frobenius(a.c1, power), fp2_from_const(BLS_FROB_FQ6_C1[power % 6]));
  Fp2 c2 = fp2_mul(fp2_frobenius(a.c2, power), fp2_from_const(BLS_FROB_FQ6_C2[power % 6]));
  r.c0 = c0; r.c1 = c1; r.c2 = c2;
}

// ------------------------------------------------------------------------------------------ Fq12
__device__ __forceinline__ void fp12_one(Fp12& r) { r.c0 = fp6_one(); r.c1 = fp6_zero(); }
__device__ __forceinline__ bool fp12_is_zero(const Fp12& a) { return fp6_is_zero(a.c0) && fp6_is_zero(a.c1); }
// fq12.rs:30-32
__device__ __forceinline__ void fp12_conjugate(Fp12& a) { fp6_neg(a.c1, a.c1); }
// fq12.rs:116-130 (r may alias a or b)
static __device__ __noinline__ void fp12_mul(Fp12& r, const Fp12& a, const Fp12& b) {
  Fp6 aa, bb, o, s;
  fp6_mul(aa, a.c0, b.c0);
  fp6_mul(bb, a.c1, b.c1);
  fp6_add(o, b.c0, b.c1);
  fp6_add(s, a.c1, a.c0);
  fp6_mul(s, s, o);
  fp6_sub(s, s, aa);
  fp6_sub(r.c1, s, bb);
  fp6_mul_by_nonresidue(bb, bb);
  fp6_add(r.c0, bb, aa);
}
// fq12.rs:99-114 (generic complex squaring; r may alias a)
static __device__ __noinline__ void fp12_sqr(Fp12& r, const Fp12& a) {
  Fp6 ab, c0c1, c0;
  fp6_mul(ab, a.c0, a.c1);
  fp6_add(c0c1, a.c0, a.c1);
  fp6_mul_by_nonresidue(c0, a.c1);
  fp6_add(c0, c0, a.c0);
  fp6_mul(c0, c0, c0c1);
  fp6_sub(c0, c0, ab);
  fp6_add(r.c1, ab, ab);
  fp6_mul_by_nonresidue(ab, ab);
  fp6_sub(r.c0, c0, ab);
}
// fq12.rs:34-48 (in place on f)
static __device__ __noinline__ void fp12_mul_by_014(Fp12& f, const Fp2& c0, const Fp2& c1, const Fp2& c4) {
  Fp6 aa, bb, s;
  fp6_mul_by_01(aa, f.c0, c0, c1);
  fp6_mul_by_1(bb, f.c1, c4);
  Fp2 o = fp2_add(c1, c4);
  fp6_add(s, f.c1, f.c0);
  fp6_mul_by_01(s, s, c0, o);
  fp6_sub(s, s, aa);
  fp6_sub(f.c1, s, bb);
  fp6_mul_by_nonresidue(bb, bb);
  fp6_add(f.c0, bb, aa);
}
// fq12.rs:132-148
static __device__ __noinline__ bool fp12_inv(Fp12& r, const Fp12& a) {
  Fp6 c0s, c1s, t;
  fp6_sqr(c0s, a.c0);
  fp6_sqr(c1s, a.c1);
  fp6_mul_by_nonresidue(c1s, c1s);
  fp6_sub(c0s, c0s, c1s);
  bool ok = fp6_inv(t, c0s);
  fp6_mul(c0s, t, a.c0);
  fp6_mul(c1s, t, a.c1);
  r.c0 = c0s;
  fp6_neg(r.c1, c1s);
  return ok;
}
// fq12.rs:90-97 (r may alias a)
static __device__ __noinline__ void fp12_frobenius(Fp12& r, const Fp12& a, int power) {
  fp6_frobenius(r.c0, a.c0, power);
  fp6_frobenius(r.c1, a.c1, power);
  Fp2 k = fp2_from_const(BLS_FROB_FQ12_C1[power % 12]);
  r.c1.c0 = fp2_mul(r.c1.c0, k);
  r.c1.c1 = fp2_mul(r.c1.c1, k);
  r.c1.c2 = fp2_mul(r.c1.c2, k);
}

}  // namespace bls
