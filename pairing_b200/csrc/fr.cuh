// fr.cuh -- the scalar field Fr of BLS12-381 (255-bit r) in Montgomery form, 8 x 32-bit limbs (bls12_381/fr.rs:324-572).
// Callers combine scalars (c * d in the reference's bilinearity test, tests/engine.rs:117-119), and the FFT of
// kernels_fft.cu runs its butterflies on it.  Results are canonical (< r) after every operation.
//
// The product is fp.cuh's construction on 8 limbs: a word-serial (CIOS) Montgomery product whose partial products are
// accumulated in two 8-word carry chains -- even-indexed and odd-indexed limbs -- so that every `mad.lo.cc / madc.hi.cc`
// pair becomes one IMAD.WIDE.U32(.X): 64 (a*b) + 64 (m*r) MAC32 + 8 IMAD (m = t0 * inv).  For a, b < r the merged
// result is < 2r < 2^256 (r < 2^255), so one conditional subtraction makes it canonical.
#pragma once
#include <stdint.h>

namespace bls {

struct Fr { uint32_t v[8]; };

// r (fr.rs:5-12), R = 2^256 mod r (fr.rs:20-26), R^2 mod r (fr.rs:28-34), -r^-1 mod 2^32 (low half of INV, fr.rs:36)
__device__ __forceinline__ Fr fr_modulus() { return Fr{{0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u}}; }
__device__ __forceinline__ Fr fr_one() { return Fr{{0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau, 0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u}}; }
__device__ __forceinline__ Fr fr_r2() { return Fr{{0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu, 0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u}}; }
#define BLS_FR_NINV 0xffffffffu
__device__ __forceinline__ Fr fr_zero() { return Fr{{0, 0, 0, 0, 0, 0, 0, 0}}; }

__device__ __forceinline__ bool fr_is_zero(const Fr& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i];
  return o == 0;
}
__device__ __forceinline__ bool fr_eq(const Fr& a, const Fr& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i] ^ b.v[i];
  return o == 0;
}
// a >= b as 256-bit integers
__device__ __forceinline__ bool fr_geq(const Fr& a, const Fr& b) {
#pragma unroll
  for (int i = 7; i >= 0; i--) {
    if (a.v[i] != b.v[i]) return a.v[i] > b.v[i];
  }
  return true;
}
__device__ __forceinline__ Fr fr_raw_sub(const Fr& a, const Fr& b) {
  Fr r; uint64_t borrow = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) { uint64_t t = (uint64_t)a.v[i] - b.v[i] - borrow; r.v[i] = (uint32_t)t; borrow = (t >> 32) & 1; }
  return r;
}
// r as 32-bit immediates (fr.rs:5-12)
#define BLS_R0 0x00000001
#define BLS_R1 0xffffffff
#define BLS_R2 0xfffe5bfe
#define BLS_R3 0x53bda402
#define BLS_R4 0x09a1d805
#define BLS_R5 0x3339d808
#define BLS_R6 0x299d7d48
#define BLS_R7 0x73eda753
#define BLS_FR_STR2(x) #x
#define BLS_FR_STR(x) BLS_FR_STR2(x)

// t = a - r; keep a if that borrows (fr.rs:513-518 reduce)
__device__ __forceinline__ Fr fr_reduce(const Fr& a) {
  uint32_t t[8], borrow;
  asm("sub.cc.u32 %0, %9, " BLS_FR_STR(BLS_R0) ";\n\t"
      "subc.cc.u32 %1, %10, " BLS_FR_STR(BLS_R1) ";\n\t"
      "subc.cc.u32 %2, %11, " BLS_FR_STR(BLS_R2) ";\n\t"
      "subc.cc.u32 %3, %12, " BLS_FR_STR(BLS_R3) ";\n\t"
      "subc.cc.u32 %4, %13, " BLS_FR_STR(BLS_R4) ";\n\t"
      "subc.cc.u32 %5, %14, " BLS_FR_STR(BLS_R5) ";\n\t"
      "subc.cc.u32 %6, %15, " BLS_FR_STR(BLS_R6) ";\n\t"
      "subc.cc.u32 %7, %16, " BLS_FR_STR(BLS_R7) ";\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(borrow)
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]));
  Fr r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = borrow ? a.v[i] : t[i];
  return r;
}
// fr.rs:341-348 (a + b < 2r < 2^256: no carry out)
__device__ __forceinline__ Fr fr_add(const Fr& a, const Fr& b) {
  Fr r;
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
        "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
  return fr_reduce(r);
}
// fr.rs:359-367: a - b, plus r when it borrows
__device__ __forceinline__ Fr fr_sub(const Fr& a, const Fr& b) {
  Fr r;
  uint32_t borrow;
  asm("sub.cc.u32 %0, %9, %17;\n\t"
      "subc.cc.u32 %1, %10, %18;\n\t"
      "subc.cc.u32 %2, %11, %19;\n\t"
      "subc.cc.u32 %3, %12, %20;\n\t"
      "subc.cc.u32 %4, %13, %21;\n\t"
      "subc.cc.u32 %5, %14, %22;\n\t"
      "subc.cc.u32 %6, %15, %23;\n\t"
      "subc.cc.u32 %7, %16, %24;\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7]), "=r"(borrow)
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
        "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
  // borrow is 0 or 0xffffffff: add (r & borrow)
  asm("add.cc.u32 %0, %0, %8;\n\t"
      "addc.cc.u32 %1, %1, %9;\n\t"
      "addc.cc.u32 %2, %2, %10;\n\t"
      "addc.cc.u32 %3, %3, %11;\n\t"
      "addc.cc.u32 %4, %4, %12;\n\t"
      "addc.cc.u32 %5, %5, %13;\n\t"
      "addc.cc.u32 %6, %6, %14;\n\t"
      "addc.u32 %7, %7, %15;"
      : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]), "+r"(r.v[3]), "+r"(r.v[4]), "+r"(r.v[5]), "+r"(r.v[6]), "+r"(r.v[7])
      : "r"(BLS_R0 & borrow), "r"(BLS_R1 & borrow), "r"(BLS_R2 & borrow), "r"(BLS_R3 & borrow),
        "r"(BLS_R4 & borrow), "r"(BLS_R5 & borrow), "r"(BLS_R6 & borrow), "r"(BLS_R7 & borrow));
  return r;
}
// fr.rs:369-375
__device__ __forceinline__ Fr fr_neg(const Fr& a) { return fr_is_zero(a) ? a : fr_raw_sub(fr_modulus(), a); }

// acc += (x[0], x[2], x[4], x[6]) * b as one 8-word carry chain, then top += carry-out
__device__ __forceinline__ void fr_cmad_row(uint32_t (&acc)[8], const uint32_t* x, uint32_t b, uint32_t& top) {
  asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
      "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
      "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
      "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
      "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
      "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
      "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
      "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
      : "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(b));
}
// w0 += add0 (word 0 of the other accumulator's successor); the carry out of that addition enters this chain, which
// computes acc = (acc >> 64) + (x[0], x[2], x[4], x[6]) * b
__device__ __forceinline__ void fr_madc_rshift_row(uint32_t& w0, uint32_t add0, uint32_t (&acc)[8], const uint32_t* x, uint32_t b) {
  asm("add.cc.u32 %0, %0, %9;\n\t"
      "madc.lo.cc.u32 %1, %10, %14, %3;\n\t"
      "madc.hi.cc.u32 %2, %10, %14, %4;\n\t"
      "madc.lo.cc.u32 %3, %11, %14, %5;\n\t"
      "madc.hi.cc.u32 %4, %11, %14, %6;\n\t"
      "madc.lo.cc.u32 %5, %12, %14, %7;\n\t"
      "madc.hi.cc.u32 %6, %12, %14, %8;\n\t"
      "madc.lo.cc.u32 %7, %13, %14, 0;\n\t"
      "madc.hi.u32 %8, %13, %14, 0;"
      : "+r"(w0), "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7])
      : "r"(add0), "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(b));
}
// One Montgomery reduction step on (e, o): m = e[0] * (-r^-1); o += (r1, r3, r5, r7) * m (its carry-out is zero);
// e += (r0, r2, r4, r6) * m with the carry-out into o[7].  Afterwards e[0] == 0.
__device__ __forceinline__ void fr_redc_row(uint32_t (&e)[8], uint32_t (&o)[8]) {
  const uint32_t m = e[0] * BLS_FR_NINV;
  asm("mad.lo.cc.u32 %0, %8, " BLS_FR_STR(BLS_R1) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %8, " BLS_FR_STR(BLS_R1) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %8, " BLS_FR_STR(BLS_R3) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %8, " BLS_FR_STR(BLS_R3) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %8, " BLS_FR_STR(BLS_R5) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %8, " BLS_FR_STR(BLS_R5) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %8, " BLS_FR_STR(BLS_R7) ", %6;\n\t"
      "madc.hi.u32 %7, %8, " BLS_FR_STR(BLS_R7) ", %7;"
      : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7])
      : "r"(m));
  asm("mad.lo.cc.u32 %0, %9, " BLS_FR_STR(BLS_R0) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %9, " BLS_FR_STR(BLS_R0) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %9, " BLS_FR_STR(BLS_R2) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %9, " BLS_FR_STR(BLS_R2) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %9, " BLS_FR_STR(BLS_R4) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %9, " BLS_FR_STR(BLS_R4) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %9, " BLS_FR_STR(BLS_R6) ", %6;\n\t"
      "madc.hi.cc.u32 %7, %9, " BLS_FR_STR(BLS_R6) ", %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(e[0]), "+r"(e[1]), "+r"(e[2]), "+r"(e[3]), "+r"(e[4]), "+r"(e[5]), "+r"(e[6]), "+r"(e[7]), "+r"(o[7])
      : "r"(m));
}
// fr.rs:438-465 + 520-572: a * b * 2^-256 mod r for a, b < r
__device__ __forceinline__ Fr fr_mul(const Fr& a, const Fr& b) {
  uint32_t e[8], o[8];
  // row 0: fresh products
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    const uint64_t t = (uint64_t)a.v[j] * b.v[0];
    e[j] = (uint32_t)t; e[j + 1] = (uint32_t)(t >> 32);
    const uint64_t u = (uint64_t)a.v[j + 1] * b.v[0];
    o[j] = (uint32_t)u; o[j + 1] = (uint32_t)(u >> 32);
  }
  fr_redc_row(e, o);
#pragma unroll
  for (int i = 1; i < 8; i += 2) {
    // odd row: roles swapped -- o is now word-0 aligned, e (with e[0] == 0) shifts down by 64 bits
    fr_madc_rshift_row(o[0], e[1], e, &a.v[1], b.v[i]);
    fr_cmad_row(o, &a.v[0], b.v[i], e[7]);
    fr_redc_row(o, e);
    if (i + 1 < 8) {
      fr_madc_rshift_row(e[0], o[1], o, &a.v[1], b.v[i + 1]);
      fr_cmad_row(e, &a.v[0], b.v[i + 1], o[7]);
      fr_redc_row(e, o);
    }
  }
  // 8 rows: the last one left `o` word-0 aligned with o[0] == 0; r = (o >> 32) + e < 2r
  Fr r;
  asm("add.cc.u32 %0, %8, %15;\n\t"
      "addc.cc.u32 %1, %9, %16;\n\t"
      "addc.cc.u32 %2, %10, %17;\n\t"
      "addc.cc.u32 %3, %11, %18;\n\t"
      "addc.cc.u32 %4, %12, %19;\n\t"
      "addc.cc.u32 %5, %13, %20;\n\t"
      "addc.cc.u32 %6, %14, %21;\n\t"
      "addc.u32 %7, %22, 0;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
      : "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]),
        "r"(e[0]), "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]));
  return fr_reduce(r);
}
__device__ __forceinline__ Fr fr_sqr(const Fr& a) { return fr_mul(a, a); }
// fr.rs:377-431 computes the inverse by binary extended Euclid; a^(r-2) is the same field value.  false for zero.
static __device__ __noinline__ bool fr_inv(Fr& out, const Fr& a) {
  if (fr_is_zero(a)) { out = fr_zero(); return false; }
  const Fr e = fr_raw_sub(fr_modulus(), Fr{{2, 0, 0, 0, 0, 0, 0, 0}});   // r - 2
  Fr res = fr_one();
  bool started = false;
#pragma unroll 1
  for (int i = 254; i >= 0; i--) {
    if (started) res = fr_sqr(res);
    if ((e.v[i >> 5] >> (i & 31)) & 1u) { res = started ? fr_mul(res, a) : a; started = true; }
  }
  out = res;
  return true;
}

}  // namespace bls
