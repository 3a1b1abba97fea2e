// codec.cuh -- point encodings and their validation: the step before the pairing path in batch verification
// (bytes -> affine points) and after it (affine points -> bytes).
//   G1Uncompressed / G1Compressed   bls12_381/ec.rs:645-868
//   G2Uncompressed / G2Compressed   bls12_381/ec.rs:1292-1540
//   get_point_from_x, is_on_curve, is_in_correct_subgroup_assuming_on_curve   ec.rs:97-144
//   Fq::sqrt fq.rs:1147-1170, Fq2::sqrt fq2.rs:167-221, orderings fq.rs:703-708 / fq2.rs:20-31
// Decoded points are canonical field values, so any exponentiation schedule gives the reference's bits; the
// ROOT that `sqrt` returns is fixed by the algorithm (a^((q+1)/4), resp. Algorithm 9 of eprint 2012/685) and
// is reproduced exactly, then the lexicographic rule picks y or -y.
#pragma once
#include "curve.cuh"

namespace bls {

// status of one decoded element (0 = Ok; mirrors GroupDecodingError, src/lib.rs:468-497)
enum {
  DEC_OK = 0,
  DEC_UNEXPECTED_COMPRESSION_MODE = 1,
  DEC_UNEXPECTED_INFORMATION = 2,
  DEC_NOT_ON_CURVE = 3,
  DEC_NOT_IN_SUBGROUP = 4,
  DEC_COORDINATE = 16   // + index of the coordinate whose integer is >= q (see include/pairing_b200.h)
};

// 48 big-endian bytes -> 12 little-endian 32-bit limbs of the integer (FqRepr::read_be, lib.rs:391-432)
__device__ __forceinline__ Fp fp_from_be(const uint8_t* b, uint8_t first_byte_mask) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    const uint8_t* p = b + 44 - 4 * i;
    uint32_t b0 = p[0];
    if (i == 11) b0 &= first_byte_mask;
    r.v[i] = (b0 << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
  }
  return r;
}
__device__ __forceinline__ void fp_to_be(uint8_t* b, const Fp& a) {
#pragma unroll
  for (int i = 0; i < 12; i++) {
    uint8_t* p = b + 44 - 4 * i;
    p[0] = (uint8_t)(a.v[i] >> 24); p[1] = (uint8_t)(a.v[i] >> 16); p[2] = (uint8_t)(a.v[i] >> 8); p[3] = (uint8_t)a.v[i];
  }
}
// Fq::from_repr validity (fq.rs:747-756): the integer is < q
__device__ __forceinline__ bool fp_repr_is_valid(const Fp& a) {
  Fp t = a;
  fp_final_sub(t);          // "unchanged by one conditional subtraction" <=> a < q
  return fp_eq_raw(t, a);
}
__device__ __forceinline__ Fp fp_to_mont(const Fp& raw) { return fp_mul(raw, fp_r2()); }
__device__ __forceinline__ Fp fp_from_mont(const Fp& a) { Fp one = fp_zero(); one.v[0] = 1; return fp_canon(fp_mul(a, one)); }   // into_repr, fq.rs:758-777
// integer comparison of two canonical integers: a > b
__device__ __forceinline__ bool fp_repr_gt(const Fp& a, const Fp& b) {
#pragma unroll
  for (int i = 11; i >= 0; i--) {
    if (a.v[i] != b.v[i]) return a.v[i] > b.v[i];
  }
  return false;
}
// Ord for Fq (fq.rs:703-708): compares into_repr()
__device__ __forceinline__ bool f_gt(const Fp& a, const Fp& b) { return fp_repr_gt(fp_from_mont(a), fp_from_mont(b)); }
// Ord for Fq2 (fq2.rs:20-31): c1 first, then c0
__device__ __forceinline__ bool f_gt(const Fp2& a, const Fp2& b) {
  Fp a1 = fp_from_mont(a.c1), b1 = fp_from_mont(b.c1);
  if (!fp_eq_raw(a1, b1)) return fp_repr_gt(a1, b1);
  return fp_repr_gt(fp_from_mont(a.c0), fp_from_mont(b.c0));
}

// x^e for a fixed exponent given as 12 little-endian words, 4-bit fixed window (Field::pow, lib.rs:306-324, is
// plain square-and-multiply; the value is the same)
template <class F> __device__ __noinline__ void f_pow_words(F& out, const F& a, const uint32_t* e) {
  F tbl[16];
  f_set_one(tbl[0]);
  tbl[1] = a;
#pragma unroll 1
  for (int i = 2; i < 16; i++) tbl[i] = f_mul(tbl[i - 1], a);
  F r; f_set_one(r);
  bool started = false;
#pragma unroll 1
  for (int i = 95; i >= 0; i--) {
    uint32_t nib = (e[i >> 3] >> ((i & 7) * 4)) & 0xf;
    if (started) { r = f_sqr(r); r = f_sqr(r); r = f_sqr(r); r = f_sqr(r); }
    if (nib) { r = started ? f_mul(r, tbl[nib]) : tbl[nib]; started = true; }
  }
  out = r;
}
// (q - 3) / 4 (fq.rs:1152-1159) and (q - 1) / 2 (fq2.rs:206-213), little-endian 32-bit words
__device__ const uint32_t BLS_EXP_Q_MINUS_3_OVER_4[12] = {0xffffeaaau, 0xee7fbfffu, 0xac54ffffu, 0x07aaffffu, 0x3dac3d89u, 0xd9cc34a8u,
                                                          0x3ce144afu, 0xd91dd2e1u, 0x90d2eb35u, 0x92c6e9edu, 0x8e5ff9a6u, 0x0680447au};
__device__ const uint32_t BLS_EXP_Q_MINUS_1_OVER_2[12] = {0xffffd555u, 0xdcff7fffu, 0x58a9ffffu, 0x0f55ffffu, 0x7b587b12u, 0xb3986950u,
                                                          0x79c2895fu, 0xb23ba5c2u, 0x21a5d66bu, 0x258dd3dbu, 0x1cbff34du, 0x0d0088f5u};

// fq.rs:1147-1170
__device__ __forceinline__ bool f_sqrt(Fp& out, const Fp& a) {
  Fp a1;
  f_pow_words(a1, a, BLS_EXP_Q_MINUS_3_OVER_4);
  Fp a0 = fp_mul(fp_sqr(a1), a);
  if (fp_eq(a0, fp_neg(fp_one()))) return false;      // NEGATIVE_ONE: not a square
  out = fp_mul(a1, a);
  return true;
}
// fq2.rs:167-221
__device__ __forceinline__ bool f_sqrt(Fp2& out, const Fp2& a) {
  if (fp2_is_zero(a)) { out = fp2_zero(); return true; }
  Fp2 a1;
  f_pow_words(a1, a, BLS_EXP_Q_MINUS_3_OVER_4);
  Fp2 alpha = fp2_mul(fp2_sqr(a1), a);
  Fp2 a0 = fp2_mul(fp2_frobenius(alpha, 1), alpha);
  const Fp2 neg1 = Fp2{fp_neg(fp_one()), fp_zero()};
  if (fp2_eq(a0, neg1)) return false;
  a1 = fp2_mul(a1, a);
  if (fp2_eq(alpha, neg1)) {
    out = fp2_mul(a1, Fp2{fp_zero(), fp_one()});
  } else {
    Fp2 t;
    f_pow_words(t, fp2_add(alpha, fp2_one()), BLS_EXP_Q_MINUS_1_OVER_2);
    out = fp2_mul(a1, t);
  }
  return true;
}

// curve constant b: 4 for G1 (fq.rs:76 B_COEFF), 4(1 + u) for G2 (fq.rs:79-82)
__device__ __forceinline__ void f_coeff_b(Fp& b) { Fp four = fp_zero(); four.v[0] = 4; b = fp_to_mont(four); }
__device__ __forceinline__ void f_coeff_b(Fp2& b) { Fp t; f_coeff_b(t); b = Fp2{t, t}; }

// x^3 + b
template <class F> __device__ __forceinline__ F curve_rhs(const F& x) {
  F b; f_coeff_b(b);
  return f_add(f_mul(f_sqr(x), x), b);
}
// ec.rs:102-123
template <class F> __device__ __forceinline__ bool get_point_from_x(Aff<F>& p, const F& x, bool greatest) {
  F y;
  if (!f_sqrt(y, curve_rhs(x))) return false;
  F negy = f_neg(y);
  const bool y_less = f_gt(negy, y);                 // y < negy
  p.x = x; p.y = (y_less != greatest) ? y : negy; p.inf = false;
  return true;
}
// ec.rs:125-140
template <class F> __device__ __forceinline__ bool is_on_curve(const Aff<F>& p) {
  if (p.inf) return true;
  return f_eq(f_sqr(p.y), curve_rhs(p.x));
}
// ec.rs:142-144: self.mul(Fr::char()).is_zero() -- a 255-bit double-and-add (~120 general additions) in the reference.  The
// ANSWER is what has to match, and for BLS12-381 it is decided by an endomorphism (M. Scott, "A note on group membership tests
// for G1, G2 and GT on BLS pairing-friendly curves", eprint 2021/1130, sections 4 and 6, proved necessary and sufficient there):
//   G1:  (beta x, y) = [-u^2] P      beta = the primitive cube root of unity acting as -u^2 on G1 (BLS_ENDO_BETA)
//   G2:  psi(Q) = [u] Q              psi = twist o Frobenius o untwist: (conj(x) BLS_PSI_X, conj(y) BLS_FROB_FQ12_C1[3])
// with u = -0xd201000000010000: one (G2) or two (G1) 64-bit multiplications by |u| -- 63 doublings and 5 additions each.
// tests/test_gpu_codec.py compares the answers with the big-integer model on points inside and outside the subgroup.  The
// reference's multiplication by r was removed from this file; it can be recovered from git history at commit 7b088bd.
// [|u|] P for an affine P (mixed additions) and for a Jacobian P (general additions); |u| = 2^63 + 2^62 + 2^60 + 2^57 + 2^48 + 2^16
template <class F> __device__ __noinline__ void pt_mul_u_abs(Jac<F>& out, const Aff<F>& p) {
  Jac<F> res;
  res.x = p.x; res.y = p.y; f_set_one(res.z);
#pragma unroll 1
  for (int n = 62; n >= 0; n--) {
    pt_double(res);
    if ((BLS_X_ABS >> n) & 1ull) pt_add_mixed(res, p);
  }
  out = res;
}
template <class F> __device__ __noinline__ void pt_mul_u_abs(Jac<F>& out, const Jac<F>& p) {
  Jac<F> res = p;
#pragma unroll 1
  for (int n = 62; n >= 0; n--) {
    pt_double(res);
    if ((BLS_X_ABS >> n) & 1ull) pt_add(res, p);
  }
  out = res;
}
// -t == (x, y) for a Jacobian t = (X, Y, Z), Z != 0:  X = x Z^2 and -Y = y Z^3
template <class F> __device__ __forceinline__ bool jac_neg_equals_affine(const Jac<F>& t, const F& x, const F& y) {
  if (pt_is_zero(t)) return false;
  const F zz = f_sqr(t.z);
  return f_eq(t.x, f_mul(x, zz)) && f_eq(f_neg(t.y), f_mul(y, f_mul(zz, t.z)));
}
__device__ __forceinline__ bool is_in_correct_subgroup(const Aff<Fp>& p) {
  if (p.inf) return true;
  Jac<Fp> t, t2;
  pt_mul_u_abs(t, p);
  pt_mul_u_abs(t2, t);                                   // [u^2] P
  return jac_neg_equals_affine(t2, fp_mul(p.x, fp_from_const(BLS_ENDO_BETA)), p.y);
}
__device__ __forceinline__ bool is_in_correct_subgroup(const Aff<Fp2>& p) {
  if (p.inf) return true;
  Jac<Fp2> t;
  pt_mul_u_abs(t, p);                                    // [|u|] Q = -[u] Q
  const Fp2 px = fp2_mul(Fp2{p.x.c0, fp_neg(p.x.c1)}, fp2_from_const(BLS_PSI_X[0]));
  const Fp2 py = fp2_mul(Fp2{p.y.c0, fp_neg(p.y.c1)}, fp2_from_const(BLS_FROB_FQ12_C1[3]));
  return jac_neg_equals_affine(t, px, py);
}

// $affine::mul_bits with the cofactor (ec.rs:86-94, 871-875, 1564-1578): MSB-first over ALL bits of the limb array,
// doubling a (still infinite) accumulator included, mixed additions -- the second half of G::rand (ec.rs:199-214).
__device__ const uint32_t BLS_G1_COFACTOR[4] = {0x0000aaabu, 0x8c00aaabu, 0x5555e156u, 0x396c8c00u};
__device__ const uint32_t BLS_G2_COFACTOR[16] = {0x1c7238e5u, 0xcf1c38e3u, 0x786f0c70u, 0x1616ec6eu, 0x3a6691aeu, 0x21537e29u, 0x4d9e82efu, 0xa628f1cbu,
                                                 0x2e5a7ddfu, 0xa68a205bu, 0x47085abau, 0xcd91de45u, 0x2876a202u, 0x091d5079u, 0x5414e7f1u, 0x05d543a9u};
// (also CurveAffine::mul, ec.rs:174-177, with the 8 words of an FrRepr)
template <class F> __device__ __forceinline__ void scale_by_cofactor(Jac<F>& res, const Aff<F>& p, const uint32_t* cof, int words) {
  pt_set_zero(res);
#pragma unroll 1
  for (int i = 32 * words - 1; i >= 0; i--) {
    pt_double(res);
    if ((cof[i >> 5] >> (i & 31)) & 1u) pt_add_mixed(res, p);
  }
}

// field-generic byte I/O: one "coordinate" is 48 bytes for Fq, 96 for Fq2 (c1 first: ec.rs:1371-1374)
struct CoordLoad { bool ok; int bad_index; };
__device__ __forceinline__ void f_load_be(Fp& out, const uint8_t* b, uint8_t mask, int coord, CoordLoad& st) {
  Fp raw = fp_from_be(b, mask);
  if (st.ok && !fp_repr_is_valid(raw)) { st.ok = false; st.bad_index = coord; }
  out = fp_to_mont(raw);
}
__device__ __forceinline__ void f_load_be(Fp2& out, const uint8_t* b, uint8_t mask, int coord, CoordLoad& st) {
  Fp c1 = fp_from_be(b, mask), c0 = fp_from_be(b + 48, 0xff);
  // the reference converts c0 first, then c1 (ec.rs:1378-1393): report in that order
  if (st.ok && !fp_repr_is_valid(c0)) { st.ok = false; st.bad_index = 2 * coord; }
  if (st.ok && !fp_repr_is_valid(c1)) { st.ok = false; st.bad_index = 2 * coord + 1; }
  out = Fp2{fp_to_mont(c0), fp_to_mont(c1)};
}
__device__ __forceinline__ void f_store_be(uint8_t* b, const Fp& a) { fp_to_be(b, fp_from_mont(a)); }
__device__ __forceinline__ void f_store_be(uint8_t* b, const Fp2& a) { fp_to_be(b, fp_from_mont(a.c1)); fp_to_be(b + 48, fp_from_mont(a.c0)); }
template <class F> struct FBytes;
template <> struct FBytes<Fp> { static const int N = 48; };
template <> struct FBytes<Fp2> { static const int N = 96; };

// EncodedPoint::into_affine / into_affine_unchecked for one element.  G2 coordinate indices for the error code:
// 0 = x (c0), 1 = x (c1), 2 = y (c0), 3 = y (c1); G1: 0 = x, 1 = y.
template <class F> __device__ __forceinline__ int decode_point(Aff<F>& p, const uint8_t* b, bool compressed, bool checked) {
  const int CB = FBytes<F>::N;
  const int size = compressed ? CB : 2 * CB;
  f_set_zero(p.x); f_set_one(p.y); p.inf = true;
  const uint8_t flags = b[0];
  if (((flags & 0x80) != 0) != compressed) return DEC_UNEXPECTED_COMPRESSION_MODE;
  if (flags & 0x40) {
    uint32_t any = flags & 0x3f;
    for (int i = 1; i < size; i++) any |= b[i];
    return any ? DEC_UNEXPECTED_INFORMATION : DEC_OK;          // G::zero()
  }
  const bool greatest = (flags & 0x20) != 0;
  if (greatest && !compressed) return DEC_UNEXPECTED_INFORMATION;
  CoordLoad st{true, 0};
  F x, y;
  f_load_be(x, b, 0x1f, 0, st);
  if (!compressed) f_load_be(y, b + CB, 0xff, 1, st);
  if (!st.ok) return DEC_COORDINATE + st.bad_index;
  if (compressed) {
    if (!get_point_from_x(p, x, greatest)) { f_set_zero(p.x); f_set_one(p.y); p.inf = true; return DEC_NOT_ON_CURVE; }
  } else {
    p.x = x; p.y = y; p.inf = false;
  }
  int status = DEC_OK;
  if (checked) {
    if (!compressed && !is_on_curve(p)) status = DEC_NOT_ON_CURVE;       // decompression is on the curve by construction
    else if (!is_in_correct_subgroup(p)) status = DEC_NOT_IN_SUBGROUP;
  }
  if (status != DEC_OK) { f_set_zero(p.x); f_set_one(p.y); p.inf = true; }
  return status;
}

// EncodedPoint::from_affine (ec.rs:739-757, 846-867, 1397-1416, 1519-1540)
template <class F> __device__ __forceinline__ void encode_point(uint8_t* b, const Aff<F>& p, bool compressed) {
  const int CB = FBytes<F>::N;
  const int size = compressed ? CB : 2 * CB;
  if (p.inf) {
    for (int i = 0; i < size; i++) b[i] = 0;
    b[0] = compressed ? 0xc0 : 0x40;
    return;
  }
  f_store_be(b, p.x);
  if (!compressed) { f_store_be(b + CB, p.y); return; }
  uint8_t f = 0x80;
  if (f_gt(p.y, f_neg(p.y))) f |= 0x20;
  b[0] |= f;
}

}  // namespace bls
