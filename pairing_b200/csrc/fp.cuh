// fp.cuh -- Fq (the 381-bit BLS12-381 base field) on sm_100a: 12 x 32-bit limbs in registers,
// Montgomery form (x * 2^384 mod q) (reference: bls12_381/fq.rs:796-1123; the reference works on 6 x u64
// limbs -- byte-for-byte the same little-endian layout).
//
// Register values live in the RELAXED range [0, 2q] (2q < 2^382): every routine accepts and returns
// representatives in that range, and the value is made canonical (< q, the reference's representation) only
// where bits are observable -- stores to ABI memory (st_fp in kernels.cu), equality and zero tests.  That
// removes the conditional subtraction (13 carry-linked subtractions + 12 selects, a serial tail) from every
// Montgomery product and the zero test from every negation:
//   product of a, b <= 2q:  a b / R + q  <=  4 q^2 / R + q  <  1.41 q        (q / R < 0.1021)
//   dual product:           (x bx + y by) / R + q  <=  8 q^2 / R + q  <  1.82 q
//   add: a + b <= 4q, minus 2q if >= 2q;  sub: a - b, plus 2q if negative;  neg: 2q - a
// tools/emulate_fp.py replays the exact carry schedule on operands up to 2q and checks both the bounds and
// that every carry the PTX drops is zero.
//
// Multiplication is a word-serial (CIOS) Montgomery product on 32-bit limbs whose partial products
// are accumulated in two independent 12-word carry chains -- products of even-indexed limbs and of
// odd-indexed limbs -- so that every `mad.lo.cc / madc.hi.cc` pair is fused by ptxas into a single
// IMAD.WIDE.U32(.X) and no carry has to ripple between the two chains inside a row.
// 144 (a*b) + 144 (m*q) wide multiply-accumulates + 12 IMAD (m = t0 * inv) = 300 MAC32 per product,
// which is the unit the roofline in bench.py / DESIGN.md is counted in.
#pragma once
#include <stdint.h>

namespace bls {

struct Fp { uint32_t v[12]; };

// q as 32-bit immediates (bls12_381/fq.rs:6-13) and -q^-1 mod 2^32 (low half of fq.rs:43)
#define BLS_Q0 0xffffaaab
#define BLS_Q1 0xb9feffff
#define BLS_Q2 0xb153ffff
#define BLS_Q3 0x1eabfffe
#define BLS_Q4 0xf6b0f624
#define BLS_Q5 0x6730d2a0
#define BLS_Q6 0xf38512bf
#define BLS_Q7 0x64774b84
#define BLS_Q8 0x434bacd7
#define BLS_Q9 0x4b1ba7b6
#define BLS_Q10 0x397fe69a
#define BLS_Q11 0x1a0111ea
#define BLS_NINV 0xfffcfffdu
// 2q
#define BLS_2Q0 0xffff5556
#define BLS_2Q1 0x73fdffff
#define BLS_2Q2 0x62a7ffff
#define BLS_2Q3 0x3d57fffd
#define BLS_2Q4 0xed61ec48
#define BLS_2Q5 0xce61a541
#define BLS_2Q6 0xe70a257e
#define BLS_2Q7 0xc8ee9709
#define BLS_2Q8 0x869759ae
#define BLS_2Q9 0x96374f6c
#define BLS_2Q10 0x72ffcd34
#define BLS_2Q11 0x340223d4
#define BLS_STR2(x) #x
#define BLS_STR(x) BLS_STR2(x)

__device__ __forceinline__ Fp fp_modulus() {
  return Fp{{BLS_Q0, BLS_Q1, BLS_Q2, BLS_Q3, BLS_Q4, BLS_Q5, BLS_Q6, BLS_Q7, BLS_Q8, BLS_Q9, BLS_Q10, BLS_Q11}};
}
__device__ __forceinline__ Fp fp_zero() { return Fp{{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}}; }
// Montgomery one, R = 2^384 mod q (fq.rs:22-30)
__device__ __forceinline__ Fp fp_one() {
  return Fp{{0x0002fffdu, 0x76090000u, 0xc40c0002u, 0xebf4000bu, 0x53c758bau, 0x5f489857u,
             0x70525745u, 0x77ce5853u, 0xa256ec6du, 0x5c071a97u, 0xfa80e493u, 0x15f65ec3u}};
}
// R^2 mod q (fq.rs:33-40)
__device__ __forceinline__ Fp fp_r2() {
  return Fp{{0x1c341746u, 0xf4df1f34u, 0x09d104f1u, 0x0a76e6a6u, 0x4c95b6d5u, 0x8de5476cu,
             0x939d83c0u, 0x67eb88a9u, 0xb519952du, 0x9a793e85u, 0x92cae3aau, 0x11988fe5u}};
}

// bit-pattern tests (for canonical values and raw integers)
__device__ __forceinline__ bool fp_is_zero_raw(const Fp& a) {
  uint32_t o = a.v[0];
#pragma unroll
  for (int i = 1; i < 12; i++) o |= a.v[i];
  return o == 0;
}
__device__ __forceinline__ bool fp_eq_raw(const Fp& a, const Fp& b) {
  uint32_t o = a.v[0] ^ b.v[0];
#pragma unroll
  for (int i = 1; i < 12; i++) o |= a.v[i] ^ b.v[i];
  return o == 0;
}

// r = a - q if a >= q else a   (fq.rs:1030-1034 `reduce`)
__device__ __forceinline__ void fp_final_sub(Fp& a) {
  uint32_t t[12], borrow;
  asm("sub.cc.u32 %0, %13, " BLS_STR(BLS_Q0) ";\n\t"
      "subc.cc.u32 %1, %14, " BLS_STR(BLS_Q1) ";\n\t"
      "subc.cc.u32 %2, %15, " BLS_STR(BLS_Q2) ";\n\t"
      "subc.cc.u32 %3, %16, " BLS_STR(BLS_Q3) ";\n\t"
      "subc.cc.u32 %4, %17, " BLS_STR(BLS_Q4) ";\n\t"
      "subc.cc.u32 %5, %18, " BLS_STR(BLS_Q5) ";\n\t"
      "subc.cc.u32 %6, %19, " BLS_STR(BLS_Q6) ";\n\t"
      "subc.cc.u32 %7, %20, " BLS_STR(BLS_Q7) ";\n\t"
      "subc.cc.u32 %8, %21, " BLS_STR(BLS_Q8) ";\n\t"
      "subc.cc.u32 %9, %22, " BLS_STR(BLS_Q9) ";\n\t"
      "subc.cc.u32 %10, %23, " BLS_STR(BLS_Q10) ";\n\t"
      "subc.cc.u32 %11, %24, " BLS_STR(BLS_Q11) ";\n\t"
      "subc.u32 %12, 0, 0;"
      : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]),
        "=r"(t[8]), "=r"(t[9]), "=r"(t[10]), "=r"(t[11]), "=r"(borrow)
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]),
        "r"(a.v[7]), "r"(a.v[8]), "r"(a.v[9]), "r"(a.v[10]), "r"(a.v[11]));
  // borrow == 0xffffffff iff a < q
#pragma unroll
  for (int i = 0; i < 12; i++) a.v[i] = borrow ? a.v[i] : t[i];
}

// the canonical representative (< q) of a value in [0, 2q]
__device__ __forceinline__ Fp fp_canon(const Fp& a) {
  Fp r = a;
  fp_final_sub(r);
  fp_final_sub(r);
  return r;
}
__device__ __forceinline__ bool fp_is_zero(const Fp& a) { return fp_is_zero_raw(fp_canon(a)); }
__device__ __forceinline__ bool fp_eq(const Fp& a, const Fp& b) { return fp_eq_raw(fp_canon(a), fp_canon(b)); }

// r = a - 2q if a >= 2q else a;  a <= 4q < 2^384
__device__ __forceinline__ void fp_cond_sub_2q(Fp& a) {
  uint32_t t[12], borrow;
  asm("sub.cc.u32 %0, %13, " BLS_STR(BLS_2Q0) ";\n\t"
      "subc.cc.u32 %1, %14, " BLS_STR(BLS_2Q1) ";\n\t"
      "subc.cc.u32 %2, %15, " BLS_STR(BLS_2Q2) ";\n\t"
      "subc.cc.u32 %3, %16, " BLS_STR(BLS_2Q3) ";\n\t"
      "subc.cc.u32 %4, %17, " BLS_STR(BLS_2Q4) ";\n\t"
      "subc.cc.u32 %5, %18, " BLS_STR(BLS_2Q5) ";\n\t"
      "subc.cc.u32 %6, %19, " BLS_STR(BLS_2Q6) ";\n\t"
      "subc.cc.u32 %7, %20, " BLS_STR(BLS_2Q7) ";\n\t"
      "subc.cc.u32 %8, %21, " BLS_STR(BLS_2Q8) ";\n\t"
      "subc.cc.u32 %9, %22, " BLS_STR(BLS_2Q9) ";\n\t"
      "subc.cc.u32 %10, %23, " BLS_STR(BLS_2Q10) ";\n\t"
      "subc.cc.u32 %11, %24, " BLS_STR(BLS_2Q11) ";\n\t"
      "subc.u32 %12, 0, 0;"
      : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]),
        "=r"(t[8]), "=r"(t[9]), "=r"(t[10]), "=r"(t[11]), "=r"(borrow)
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]),
        "r"(a.v[7]), "r"(a.v[8]), "r"(a.v[9]), "r"(a.v[10]), "r"(a.v[11]));
#pragma unroll
  for (int i = 0; i < 12; i++) a.v[i] = borrow ? a.v[i] : t[i];
}

// fq.rs:813-819 add_assign.  a, b <= 2q -> result <= 2q.
__device__ __forceinline__ Fp fp_add(const Fp& a, const Fp& b) {
  Fp r;
  asm("add.cc.u32 %0, %12, %24;\n\t"
      "addc.cc.u32 %1, %13, %25;\n\t"
      "addc.cc.u32 %2, %14, %26;\n\t"
      "addc.cc.u32 %3, %15, %27;\n\t"
      "addc.cc.u32 %4, %16, %28;\n\t"
      "addc.cc.u32 %5, %17, %29;\n\t"
      "addc.cc.u32 %6, %18, %30;\n\t"
      "addc.cc.u32 %7, %19, %31;\n\t"
      "addc.cc.u32 %8, %20, %32;\n\t"
      "addc.cc.u32 %9, %21, %33;\n\t"
      "addc.cc.u32 %10, %22, %34;\n\t"
      "addc.u32 %11, %23, %35;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
        "=r"(r.v[7]), "=r"(r.v[8]), "=r"(r.v[9]), "=r"(r.v[10]), "=r"(r.v[11])
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]),
        "r"(a.v[7]), "r"(a.v[8]), "r"(a.v[9]), "r"(a.v[10]), "r"(a.v[11]),
        "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]),
        "r"(b.v[7]), "r"(b.v[8]), "r"(b.v[9]), "r"(b.v[10]), "r"(b.v[11]));
  fp_cond_sub_2q(r);
  return r;
}

// fq.rs:822-828 double
__device__ __forceinline__ Fp fp_dbl(const Fp& a) { return fp_add(a, a); }

// fq.rs:831-838 sub_assign: a - b, adding 2q back when it borrows.  a, b <= 2q -> result <= 2q.
__device__ __forceinline__ Fp fp_sub(const Fp& a, const Fp& b) {
  Fp r;
  uint32_t borrow;
  asm("sub.cc.u32 %0, %13, %25;\n\t"
      "subc.cc.u32 %1, %14, %26;\n\t"
      "subc.cc.u32 %2, %15, %27;\n\t"
      "subc.cc.u32 %3, %16, %28;\n\t"
      "subc.cc.u32 %4, %17, %29;\n\t"
      "subc.cc.u32 %5, %18, %30;\n\t"
      "subc.cc.u32 %6, %19, %31;\n\t"
      "subc.cc.u32 %7, %20, %32;\n\t"
      "subc.cc.u32 %8, %21, %33;\n\t"
      "subc.cc.u32 %9, %22, %34;\n\t"
      "subc.cc.u32 %10, %23, %35;\n\t"
      "subc.cc.u32 %11, %24, %36;\n\t"
      "subc.u32 %12, 0, 0;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
        "=r"(r.v[7]), "=r"(r.v[8]), "=r"(r.v[9]), "=r"(r.v[10]), "=r"(r.v[11]), "=r"(borrow)
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]),
        "r"(a.v[7]), "r"(a.v[8]), "r"(a.v[9]), "r"(a.v[10]), "r"(a.v[11]),
        "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]),
        "r"(b.v[7]), "r"(b.v[8]), "r"(b.v[9]), "r"(b.v[10]), "r"(b.v[11]));
  // borrow is 0 or 0xffffffff: add (q & borrow)
  asm("add.cc.u32 %0, %0, %12;\n\t"
      "addc.cc.u32 %1, %1, %13;\n\t"
      "addc.cc.u32 %2, %2, %14;\n\t"
      "addc.cc.u32 %3, %3, %15;\n\t"
      "addc.cc.u32 %4, %4, %16;\n\t"
      "addc.cc.u32 %5, %5, %17;\n\t"
      "addc.cc.u32 %6, %6, %18;\n\t"
      "addc.cc.u32 %7, %7, %19;\n\t"
      "addc.cc.u32 %8, %8, %20;\n\t"
      "addc.cc.u32 %9, %9, %21;\n\t"
      "addc.cc.u32 %10, %10, %22;\n\t"
      "addc.u32 %11, %11, %23;"
      : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]), "+r"(r.v[3]), "+r"(r.v[4]), "+r"(r.v[5]), "+r"(r.v[6]),
        "+r"(r.v[7]), "+r"(r.v[8]), "+r"(r.v[9]), "+r"(r.v[10]), "+r"(r.v[11])
      : "r"(BLS_2Q0 & borrow), "r"(BLS_2Q1 & borrow), "r"(BLS_2Q2 & borrow), "r"(BLS_2Q3 & borrow),
        "r"(BLS_2Q4 & borrow), "r"(BLS_2Q5 & borrow), "r"(BLS_2Q6 & borrow), "r"(BLS_2Q7 & borrow),
        "r"(BLS_2Q8 & borrow), "r"(BLS_2Q9 & borrow), "r"(BLS_2Q10 & borrow), "r"(BLS_2Q11 & borrow));
  return r;
}

// fq.rs:841-847 negate: 2q - a (a <= 2q -> result <= 2q; the reference's 0 -> 0 special case is a matter of the
// canonical representative only: 2q is 0)
__device__ __forceinline__ Fp fp_neg(const Fp& a) {
  Fp r;
  asm("sub.cc.u32 %0, " BLS_STR(BLS_2Q0) ", %12;\n\t"
      "subc.cc.u32 %1, " BLS_STR(BLS_2Q1) ", %13;\n\t"
      "subc.cc.u32 %2, " BLS_STR(BLS_2Q2) ", %14;\n\t"
      "subc.cc.u32 %3, " BLS_STR(BLS_2Q3) ", %15;\n\t"
      "subc.cc.u32 %4, " BLS_STR(BLS_2Q4) ", %16;\n\t"
      "subc.cc.u32 %5, " BLS_STR(BLS_2Q5) ", %17;\n\t"
      "subc.cc.u32 %6, " BLS_STR(BLS_2Q6) ", %18;\n\t"
      "subc.cc.u32 %7, " BLS_STR(BLS_2Q7) ", %19;\n\t"
      "subc.cc.u32 %8, " BLS_STR(BLS_2Q8) ", %20;\n\t"
      "subc.cc.u32 %9, " BLS_STR(BLS_2Q9) ", %21;\n\t"
      "subc.cc.u32 %10, " BLS_STR(BLS_2Q10) ", %22;\n\t"
      "subc.u32 %11, " BLS_STR(BLS_2Q11) ", %23;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
        "=r"(r.v[7]), "=r"(r.v[8]), "=r"(r.v[9]), "=r"(r.v[10]), "=r"(r.v[11])
      : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]),
        "r"(a.v[7]), "r"(a.v[8]), "r"(a.v[9]), "r"(a.v[10]), "r"(a.v[11]));
  return r;
}

// ---------------------------------------------------------------------------------------------
// Montgomery product building blocks.  Two 12-word accumulators: `e` aligned with word 0 of the
// running total and `o` aligned with word 1 (total = e + (o << 32)).
// ---------------------------------------------------------------------------------------------

// acc += (x[0], x[2], ..., x[10]) * b as one 12-word carry chain, then top += carry-out.
// (x points at limb 0 for the even products, at limb 1 for the odd ones.)
__device__ __forceinline__ void fp_cmad_row(uint32_t (&acc)[12], const uint32_t* x, uint32_t b, uint32_t& top) {
  asm("mad.lo.cc.u32 %0, %13, %19, %0;\n\t"
      "madc.hi.cc.u32 %1, %13, %19, %1;\n\t"
      "madc.lo.cc.u32 %2, %14, %19, %2;\n\t"
      "madc.hi.cc.u32 %3, %14, %19, %3;\n\t"
      "madc.lo.cc.u32 %4, %15, %19, %4;\n\t"
      "madc.hi.cc.u32 %5, %15, %19, %5;\n\t"
      "madc.lo.cc.u32 %6, %16, %19, %6;\n\t"
      "madc.hi.cc.u32 %7, %16, %19, %7;\n\t"
      "madc.lo.cc.u32 %8, %17, %19, %8;\n\t"
      "madc.hi.cc.u32 %9, %17, %19, %9;\n\t"
      "madc.lo.cc.u32 %10, %18, %19, %10;\n\t"
      "madc.hi.cc.u32 %11, %18, %19, %11;\n\t"
      "addc.u32 %12, %12, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]),
        "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11]), "+r"(top)
      : "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(x[8]), "r"(x[10]), "r"(b));
}

// w0 += carry_in_word (word 0 of the other accumulator's successor); the carry out of that
// addition enters this chain, which computes acc = (acc >> 64) + (x[0], x[2], ..., x[10]) * b.
__device__ __forceinline__ void fp_madc_rshift_row(uint32_t& w0, uint32_t add0, uint32_t (&acc)[12],
                                                   const uint32_t* x, uint32_t b) {
  asm("add.cc.u32 %0, %0, %13;\n\t"
      "madc.lo.cc.u32 %1, %14, %20, %3;\n\t"
      "madc.hi.cc.u32 %2, %14, %20, %4;\n\t"
      "madc.lo.cc.u32 %3, %15, %20, %5;\n\t"
      "madc.hi.cc.u32 %4, %15, %20, %6;\n\t"
      "madc.lo.cc.u32 %5, %16, %20, %7;\n\t"
      "madc.hi.cc.u32 %6, %16, %20, %8;\n\t"
      "madc.lo.cc.u32 %7, %17, %20, %9;\n\t"
      "madc.hi.cc.u32 %8, %17, %20, %10;\n\t"
      "madc.lo.cc.u32 %9, %18, %20, %11;\n\t"
      "madc.hi.cc.u32 %10, %18, %20, %12;\n\t"
      "madc.lo.cc.u32 %11, %19, %20, 0;\n\t"
      "madc.hi.u32 %12, %19, %20, 0;"
      : "+r"(w0), "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]),
        "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11])
      : "r"(add0), "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(x[8]), "r"(x[10]), "r"(b));
}

// acc += (q1, q3, ..., q11) * m   (odd-aligned accumulator; carry-out is provably zero)
__device__ __forceinline__ void fp_cmad_q_odd(uint32_t (&acc)[12], uint32_t m) {
  asm("mad.lo.cc.u32 %0, %12, " BLS_STR(BLS_Q1) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %12, " BLS_STR(BLS_Q1) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %12, " BLS_STR(BLS_Q3) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %12, " BLS_STR(BLS_Q3) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %12, " BLS_STR(BLS_Q5) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %12, " BLS_STR(BLS_Q5) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %12, " BLS_STR(BLS_Q7) ", %6;\n\t"
      "madc.hi.cc.u32 %7, %12, " BLS_STR(BLS_Q7) ", %7;\n\t"
      "madc.lo.cc.u32 %8, %12, " BLS_STR(BLS_Q9) ", %8;\n\t"
      "madc.hi.cc.u32 %9, %12, " BLS_STR(BLS_Q9) ", %9;\n\t"
      "madc.lo.cc.u32 %10, %12, " BLS_STR(BLS_Q11) ", %10;\n\t"
      "madc.hi.u32 %11, %12, " BLS_STR(BLS_Q11) ", %11;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]),
        "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11])
      : "r"(m));
}
// acc += (q0, q2, ..., q10) * m, then top += carry-out   (even-aligned accumulator; acc[0] becomes 0)
__device__ __forceinline__ void fp_cmad_q_even(uint32_t (&acc)[12], uint32_t m, uint32_t& top) {
  asm("mad.lo.cc.u32 %0, %13, " BLS_STR(BLS_Q0) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %13, " BLS_STR(BLS_Q0) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %13, " BLS_STR(BLS_Q2) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %13, " BLS_STR(BLS_Q2) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %13, " BLS_STR(BLS_Q4) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %13, " BLS_STR(BLS_Q4) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %13, " BLS_STR(BLS_Q6) ", %6;\n\t"
      "madc.hi.cc.u32 %7, %13, " BLS_STR(BLS_Q6) ", %7;\n\t"
      "madc.lo.cc.u32 %8, %13, " BLS_STR(BLS_Q8) ", %8;\n\t"
      "madc.hi.cc.u32 %9, %13, " BLS_STR(BLS_Q8) ", %9;\n\t"
      "madc.lo.cc.u32 %10, %13, " BLS_STR(BLS_Q10) ", %10;\n\t"
      "madc.hi.cc.u32 %11, %13, " BLS_STR(BLS_Q10) ", %11;\n\t"
      "addc.u32 %12, %12, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]),
        "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11]), "+r"(top)
      : "r"(m));
}

// One Montgomery reduction step on (e, o): m = e[0] * (-q^-1); (e, o) += m * q.  Afterwards e[0] == 0.
__device__ __forceinline__ void fp_redc_row(uint32_t (&e)[12], uint32_t (&o)[12]) {
  uint32_t m = e[0] * BLS_NINV;
  fp_cmad_q_odd(o, m);
  fp_cmad_q_even(e, m, o[11]);
}

// r = (e >> 32) + o  (<= 2q by the bounds in the header: no conditional subtraction)
__device__ __forceinline__ Fp fp_merge(const uint32_t (&e)[12], const uint32_t (&o)[12]) {
  Fp r;
  asm("add.cc.u32 %0, %12, %23;\n\t"
      "addc.cc.u32 %1, %13, %24;\n\t"
      "addc.cc.u32 %2, %14, %25;\n\t"
      "addc.cc.u32 %3, %15, %26;\n\t"
      "addc.cc.u32 %4, %16, %27;\n\t"
      "addc.cc.u32 %5, %17, %28;\n\t"
      "addc.cc.u32 %6, %18, %29;\n\t"
      "addc.cc.u32 %7, %19, %30;\n\t"
      "addc.cc.u32 %8, %20, %31;\n\t"
      "addc.cc.u32 %9, %21, %32;\n\t"
      "addc.cc.u32 %10, %22, %33;\n\t"
      "addc.u32 %11, %34, 0;"
      : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
        "=r"(r.v[7]), "=r"(r.v[8]), "=r"(r.v[9]), "=r"(r.v[10]), "=r"(r.v[11])
      : "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]), "r"(e[8]), "r"(e[9]),
        "r"(e[10]), "r"(e[11]),
        "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]), "r"(o[8]),
        "r"(o[9]), "r"(o[10]), "r"(o[11]));
  return r;
}

// a * b * 2^-384 mod q   (fq.rs:910-960 mul_assign + 1037-1122 mont_reduce)
__device__ __forceinline__ Fp fp_mul_inline(const Fp& a, const Fp& b) {
  uint32_t e[12], o[12];
  // row 0: fresh products
#pragma unroll
  for (int j = 0; j < 12; j += 2) {
    uint64_t t = (uint64_t)a.v[j] * b.v[0];
    e[j] = (uint32_t)t; e[j + 1] = (uint32_t)(t >> 32);
    uint64_t u = (uint64_t)a.v[j + 1] * b.v[0];
    o[j] = (uint32_t)u; o[j + 1] = (uint32_t)(u >> 32);
  }
  fp_redc_row(e, o);
#pragma unroll
  for (int i = 1; i < 12; i += 2) {
    // odd row: roles swapped -- o is now word-0 aligned, e (with e[0] == 0) shifts down by 64 bits
    fp_madc_rshift_row(o[0], e[1], e, &a.v[1], b.v[i]);
    fp_cmad_row(o, &a.v[0], b.v[i], e[11]);
    fp_redc_row(o, e);
    if (i + 1 < 12) {
      fp_madc_rshift_row(e[0], o[1], o, &a.v[1], b.v[i + 1]);
      fp_cmad_row(e, &a.v[0], b.v[i + 1], o[11]);
      fp_redc_row(e, o);
    }
  }
  // 12 rows: the last one left `o` word-0 aligned with o[0] == 0
  return fp_merge(o, e);
}

// (x * bx + y * by) * 2^-384 mod q with ONE Montgomery reduction (lazy reduction of a sum of two
// products): each row accumulates both partial products before the m*q row.  With all four operands
// <= 2q the sum is <= 8 q^2 and the result < 1.82 q.
// Used by the lane-pair Fq2 arithmetic: c0 = a0 b0 + (-a1) b1, c1 = a0 b1 + a1 b0.
// 288 (products) + 144 (m*q) wide MACs + 12 IMAD = 444 instead of 2 x 300.
// Carry analysis: tools/emulate_fp.py replays this schedule word by word and asserts that every
// carry the PTX drops is zero.
__device__ __forceinline__ Fp fp_mul2_inline(const Fp& x, const Fp& bx, const Fp& y, const Fp& by) {
  uint32_t e[12], o[12], dummy = 0;
#pragma unroll
  for (int j = 0; j < 12; j += 2) {
    uint64_t t = (uint64_t)x.v[j] * bx.v[0];
    e[j] = (uint32_t)t; e[j + 1] = (uint32_t)(t >> 32);
    uint64_t u = (uint64_t)x.v[j + 1] * bx.v[0];
    o[j] = (uint32_t)u; o[j + 1] = (uint32_t)(u >> 32);
  }
  fp_cmad_row(o, &y.v[1], by.v[0], dummy);
  fp_cmad_row(e, &y.v[0], by.v[0], o[11]);
  fp_redc_row(e, o);
#pragma unroll
  for (int i = 1; i < 12; i += 2) {
    fp_madc_rshift_row(o[0], e[1], e, &x.v[1], bx.v[i]);
    fp_cmad_row(o, &x.v[0], bx.v[i], e[11]);
    fp_cmad_row(e, &y.v[1], by.v[i], dummy);
    fp_cmad_row(o, &y.v[0], by.v[i], e[11]);
    fp_redc_row(o, e);
    if (i + 1 < 12) {
      fp_madc_rshift_row(e[0], o[1], o, &x.v[1], bx.v[i + 1]);
      fp_cmad_row(e, &x.v[0], bx.v[i + 1], o[11]);
      fp_cmad_row(o, &y.v[1], by.v[i + 1], dummy);
      fp_cmad_row(e, &y.v[0], by.v[i + 1], o[11]);
      fp_redc_row(e, o);
    }
  }
  return fp_merge(o, e);
}

static __device__ __noinline__ Fp fp_mul(Fp a, Fp b) { return fp_mul_inline(a, b); }
static __device__ __noinline__ Fp fp_mul2(Fp x, Fp bx, Fp y, Fp by) { return fp_mul2_inline(x, bx, y, by); }

}  // namespace bls
#include "fp_sqr_gen.cuh"
namespace bls {
// fq.rs:963-1016 `square`: the dedicated 234-MAC32 routine of fp_sqr_gen.cuh (generated and emulated by
// tools/gen_fp_sqr.py).  The fallback to fp_mul(a, a) -- one copy of the product code, the same canonical value -- was
// removed; it can be recovered from git history at commit 7b088bd.
static __device__ __noinline__ Fp fp_sqr(Fp a) { return fp_sqr_inline(a); }

// FrRepr (fr.rs:57-58): a canonical 256-bit integer as 8 x u32 -- scalars and GT exponents
struct Scalar { uint32_t v[8]; };

}  // namespace bls
