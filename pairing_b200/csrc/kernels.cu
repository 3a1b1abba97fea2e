// kernels.cu -- curve, field-op, codec and measurement kernels (one thread per element: tower.cuh, curve.cuh,
// codec.cuh), the context, and every host-buffer entry point of include/pairing_b200.h.  The pairing engine
// (Miller loops, final exponentiation, G2Prepared, GT powers) runs on LANE PAIRS and lives in kernels_pair.cu.
// Inputs and outputs use the ABI's array-of-structs layout directly: the path is integer-multiply
// bound (SURVEY.md section 8d: <= 880 B of HBM traffic per 6.19 M-MAC32 pairing), so HBM layout is
// not what limits it.
#include "abi_common.cuh"

#include <new>

#include "curve_io.cuh"
#include "codec.cuh"
#include "fr.cuh"

// ------------------------------------------------------------------------------------------------
// Field-op kernels (tower parity tests; `Field` trait methods, src/lib.rs:267-325)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_fq_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp x = ld_fp(a + 6 * i), y = b ? ld_fp(b + 6 * i) : fp_zero(), r = fp_zero();
  bool good = true;
  switch (op) {
    case BLS_OP_ADD: r = fp_add(x, y); break;
    case BLS_OP_SUB: r = fp_sub(x, y); break;
    case BLS_OP_MUL: r = fp_mul(x, y); break;
    case BLS_OP_SQR: r = fp_sqr(x); break;
    case BLS_OP_NEG: r = fp_neg(x); break;
    case BLS_OP_DBL: r = fp_dbl(x); break;
    case BLS_OP_INV: good = fp_inv(r, x); break;
    case BLS_OP_FROM_REPR: {   // fq.rs:747-756: valid iff x < q, then x * R2
      Fp t = x; fp_final_sub(t);
      good = fp_eq_raw(t, x);
      r = good ? fp_mul(x, fp_r2()) : fp_zero();
      break;
    }
    case BLS_OP_INTO_REPR: {   // fq.rs:758-777: Montgomery reduction of the padded value == x * 1 * R^-1
      Fp one = fp_zero(); one.v[0] = 1;
      r = fp_mul(x, one);
      break;
    }
    case BLS_OP_SQRT: good = f_sqrt(r, x); if (!good) r = fp_zero(); break;
  }
  st_fp(out + 6 * i, r);
  if (ok) ok[i] = good;
}

// scalar field Fr (fr.rs:324-572): `b` may be NULL for unary operations
__global__ void __launch_bounds__(128) k_fr_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr x, y = fr_zero(), r = fr_zero();
  {
    const uint2* q = reinterpret_cast<const uint2*>(a + 4 * i);
#pragma unroll
    for (int k = 0; k < 4; k++) { uint2 t = q[k]; x.v[2 * k] = t.x; x.v[2 * k + 1] = t.y; }
    if (b) {
      const uint2* qb = reinterpret_cast<const uint2*>(b + 4 * i);
#pragma unroll
      for (int k = 0; k < 4; k++) { uint2 t = qb[k]; y.v[2 * k] = t.x; y.v[2 * k + 1] = t.y; }
    }
  }
  bool good = true;
  switch (op) {
    case BLS_OP_ADD: r = fr_add(x, y); break;
    case BLS_OP_SUB: r = fr_sub(x, y); break;
    case BLS_OP_MUL: r = fr_mul(x, y); break;
    case BLS_OP_SQR: r = fr_sqr(x); break;
    case BLS_OP_NEG: r = fr_neg(x); break;
    case BLS_OP_DBL: r = fr_add(x, x); break;
    case BLS_OP_INV: good = fr_inv(r, x); break;
    case BLS_OP_FROM_REPR: good = !fr_geq(x, fr_modulus()); r = good ? fr_mul(x, fr_r2()) : fr_zero(); break;   // fr.rs:279-288
    case BLS_OP_INTO_REPR: { Fr one = fr_zero(); one.v[0] = 1; r = fr_mul(x, one); break; }                     // fr.rs:290-303
  }
  uint2* o = reinterpret_cast<uint2*>(out + 4 * i);
#pragma unroll
  for (int k = 0; k < 4; k++) o[k] = make_uint2(r.v[2 * k], r.v[2 * k + 1]);
  if (ok) ok[i] = good;
}

__global__ void __launch_bounds__(128) k_fq2_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp2 x = ld_fp2(a + 12 * i), y = b ? ld_fp2(b + 12 * i) : fp2_zero(), r = fp2_zero();
  bool good = true;
  switch (op) {
    case BLS_OP_ADD: r = fp2_add(x, y); break;
    case BLS_OP_SUB: r = fp2_sub(x, y); break;
    case BLS_OP_MUL: r = fp2_mul(x, y); break;
    case BLS_OP_SQR: r = fp2_sqr(x); break;
    case BLS_OP_NEG: r = fp2_neg(x); break;
    case BLS_OP_DBL: r = fp2_dbl(x); break;
    case BLS_OP_INV: good = fp2_inv(r, x); if (!good) r = fp2_zero(); break;
    case BLS_OP_MUL_NONRES: r = fp2_mul_by_nonresidue(x); break;
    case BLS_OP_FROB1: r = fp2_frobenius(x, 1); break;
    case BLS_OP_SQRT: good = f_sqrt(r, x); if (!good) r = fp2_zero(); break;
  }
  st_fp2(out + 12 * i, r);
  if (ok) ok[i] = good;
}

__global__ void __launch_bounds__(128) k_fq6_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp6 x, y, r;
  ld_fp6(x, a + 36 * i);
  if (b) ld_fp6(y, b + 36 * i); else y = fp6_zero();
  r = fp6_zero();
  bool good = true;
  switch (op) {
    case BLS_OP_ADD: fp6_add(r, x, y); break;
    case BLS_OP_SUB: fp6_sub(r, x, y); break;
    case BLS_OP_MUL: fp6_mul(r, x, y); break;
    case BLS_OP_SQR: fp6_sqr(r, x); break;
    case BLS_OP_NEG: fp6_neg(r, x); break;
    case BLS_OP_INV: good = fp6_inv(r, x); if (!good) r = fp6_zero(); break;
    case BLS_OP_MUL_NONRES: fp6_mul_by_nonresidue(r, x); break;
    case BLS_OP_FROB1: fp6_frobenius(r, x, 1); break;
    case BLS_OP_FROB2: fp6_frobenius(r, x, 2); break;
    case BLS_OP_FROB3: fp6_frobenius(r, x, 3); break;
    case BLS_OP_MUL_BY_01: fp6_mul_by_01(r, x, y.c0, y.c1); break;
    case BLS_OP_MUL_BY_1: fp6_mul_by_1(r, x, y.c1); break;
  }
  st_fp6(out + 36 * i, r);
  if (ok) ok[i] = good;
}

__global__ void __launch_bounds__(128) k_fq12_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp12 x, y, r;
  ld_fp12(x, a + 72 * i);
  if (b) ld_fp12(y, b + 72 * i); else { y.c0 = fp6_zero(); y.c1 = fp6_zero(); }
  r.c0 = fp6_zero(); r.c1 = fp6_zero();
  bool good = true;
  switch (op) {
    case BLS_OP_MUL: fp12_mul(r, x, y); break;
    case BLS_OP_SQR: fp12_sqr(r, x); break;
    case BLS_OP_INV: good = fp12_inv(r, x); if (!good) { r.c0 = fp6_zero(); r.c1 = fp6_zero(); } break;
    case BLS_OP_CONJ: r = x; fp12_conjugate(r); break;
    case BLS_OP_FROB1: fp12_frobenius(r, x, 1); break;
    case BLS_OP_FROB2: fp12_frobenius(r, x, 2); break;
    case BLS_OP_FROB3: fp12_frobenius(r, x, 3); break;
    case BLS_OP_MUL_BY_014: r = x; fp12_mul_by_014(r, y.c0.c0, y.c0.c1, y.c1.c1); break;
  }
  st_fp12(out + 72 * i, r);
  if (ok) ok[i] = good;
}

// ------------------------------------------------------------------------------------------------
// Pairing kernels
// ------------------------------------------------------------------------------------------------

// Product of `count` Fq12 values: each of T threads multiplies a strided subset of <= 8 factors; the
// host repeats the pass (count -> ceil(count/8)) until one value is left.
__global__ void __launch_bounds__(128) k_fq12_product(const uint64_t* in, size_t count, uint64_t* out, size_t T) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  Fp12 acc, x;
  fp12_one(acc);
#pragma unroll 1
  for (size_t i = t; i < count; i += T) {
    ld_fp12(x, in + FQ12_W * i);
    fp12_mul(acc, acc, x);
  }
  st_fp12(out + FQ12_W * t, acc);
}

// ------------------------------------------------------------------------------------------------
// Curve kernels
// ------------------------------------------------------------------------------------------------
#define BLS_WNAF_MINB 3
template <class F, int K, int MAXT> struct LocalTables {
  Jac<F> t[K][MAXT];
  __device__ __forceinline__ Jac<F> get(int j, int e) const { return t[j][e]; }
};
template <class F> struct SharedTable {
  const uint64_t* p;   // 2^(w-1) Jacobian points in the ABI layout
  __device__ __forceinline__ Jac<F> get(int, int e) const { Jac<F> r; ld_jac(r, p + (size_t)(3 * FW<F>::W) * e); return r; }
};

// K points per thread (pt_wnaf_run_lazy): thread t owns points t, t + T, ..., t + (K-1) T
#define BLS_WNAF_K 3      /* G1: 9.57 M muls/s at 2^22 against 9.33 M for K = 2 (lane efficiency 95 % vs 91 %) */
#define BLS_WNAF_K_G2 2
// blocks per SM: 3 for G2 (168 registers; 3.29 M muls/s at 2^20 against 3.19 M with 2 and 2.90 M with 4), BLS_WNAF_MINB_G1 for G1
#define BLS_WNAF_MINB_G1 4   /* 128 registers.  With the dedicated squaring (r2, 2^22 points, one box): 398.8 ms with 4 blocks, 405.1 with 5 (96 registers), 415.2 with 3, 425.7 with 6; K = 2 at 4 blocks 404.4 */
// MAXT = table entries per point: 8 for the windows the per-scalar heuristics pick (2..4, ec.rs:895-905, 1586-1596),
// 64 (K = 1) for the explicit windows 5..7 of wnaf_table / wnaf_exp
template <class F, bool IS_G2, int K, int MAXT>
__global__ void __launch_bounds__(128, IS_G2 ? BLS_WNAF_MINB : BLS_WNAF_MINB_G1) k_wnaf_mul_lazyk(const uint64_t* bases, const uint64_t* k, uint64_t* out, size_t n, int window) {
  const size_t T = (size_t)gridDim.x * blockDim.x;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  Jac<F> res[K];
  LocalTables<F, K, MAXT> table;
  int8_t digits[K][260];
  WnafState<K> st;
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t i = t + (size_t)j * T;
    const bool active = i < n;
    if (!active) i = n - 1;
    Jac<F> base;
    ld_jac(base, bases + (size_t)PW * i);
    Scalar s = ld_scalar(k + 4 * i);
    if (!active) {
#pragma unroll
      for (int w = 0; w < 8; w++) s.v[w] = 0;
    }
    int w = window;
    if (w == 0) {
      int nb = scalar_num_bits(s);
      w = IS_G2 ? g2_window_for_bits(nb) : g1_window_for_bits(nb);
    }
    const int tsize = 1 << (w - 1);
    Jac<F> b = base, dbl = base;
    pt_double(dbl);
#pragma unroll 1
    for (int e = 0; e < MAXT; e++) {       // wnaf_table, wnaf.rs:4-15 (the last add is unused)
      if (e < tsize) { table.t[j][e] = b; if (e + 1 < tsize) pt_add(b, dbl); }
    }
    st.i[j] = wnaf_form(digits[j], s, w) - 1;
    st.found[j] = false; st.doubled[j] = false;
    pt_set_zero(res[j]);
  }
  pt_wnaf_run_lazy<F, K>(res, table, digits, st);
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t i = t + (size_t)j * T;
    if (i < n) st_jac(out + (size_t)PW * i, res[j]);
  }
}

// Explicit windows 8..13 of wnaf_table / wnaf_exp (the reference's own test sweeps 2..13, src/tests/curve.rs:78): 2^(w-1) entries
// per point no longer fit per-thread local memory (590 KB per G1 point at w = 13), so every thread builds its table in a
// global-memory scratch row and walks it with the same decoupled-lane runner (K = 1).
template <class F>
__global__ void __launch_bounds__(128, BLS_WNAF_MINB) k_wnaf_mul_bigwindow(const uint64_t* bases, const uint64_t* k, uint64_t* out, size_t n, int window, uint64_t* tables) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  const size_t tsize = (size_t)1 << (window - 1);
  const bool active = t < n;
  const size_t i = active ? t : n - 1;
  uint64_t* mine = tables + t * tsize * PW;             // rows exist for every launched thread
  Jac<F> res[1];
  int32_t digits[1][260];
  WnafState<1> st;
  Jac<F> b, dbl;
  ld_jac(b, bases + (size_t)PW * i);
  dbl = b;
  pt_double(dbl);
#pragma unroll 1
  for (size_t e = 0; e < tsize; e++) {                  // wnaf_table, wnaf.rs:4-15
    st_jac(mine + e * PW, b);
    if (e + 1 < tsize) pt_add(b, dbl);
  }
  Scalar s = ld_scalar(k + 4 * i);
  if (!active) {
#pragma unroll
    for (int w = 0; w < 8; w++) s.v[w] = 0;
  }
  st.i[0] = wnaf_form(digits[0], s, window) - 1;
  st.found[0] = false; st.doubled[0] = false;
  pt_set_zero(res[0]);
  SharedTable<F> tab{mine};
  pt_wnaf_run_lazy<F, 1>(res, tab, digits, st);
  if (active) st_jac(out + (size_t)PW * i, res[0]);
}

// Fixed-base mode, Wnaf::new().base(g, num_scalars) then .scalar(s_i) per scalar (wnaf.rs:93-107, 169-178):
// ONE window table shared by all scalars, window 2..16 from recommended_wnaf_for_num_scalars.
// k_wnaf_table builds it: table[i] = (2i+1) g by repeated projective additions of 2g -- a chain of 2^(w-1)
// dependent additions (each entry's Jacobian representative depends on the previous one): ONE warp, whose lanes split
// the independent products inside each addition (curve.cuh: pt_add_fixed_coop).
template <class F>
__global__ void __launch_bounds__(32) k_wnaf_table(const uint64_t* base, uint64_t* table, int window) {
  const int PW = 3 * FW<F>::W;
  Jac<F> b, dbl;
  ld_jac(b, base);
  dbl = b;
  pt_double(dbl);
  const F z2z2 = f_sqr(dbl.z), z2c = f_mul(dbl.z, z2z2);
  const int tsize = 1 << (window - 1);
#pragma unroll 1
  for (int e = 0; e < tsize; e++) {
    if (threadIdx.x == 0) st_jac(table + (size_t)PW * e, b);
    if (e + 1 < tsize) pt_add_fixed_coop(b, dbl, z2z2, z2c);
  }
}
template <class F, int K>
__global__ void __launch_bounds__(128, BLS_WNAF_MINB) k_wnaf_fixed_base(const uint64_t* table, int window, const uint64_t* k, uint64_t* out, size_t n) {
  const size_t T = (size_t)gridDim.x * blockDim.x;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  Jac<F> res[K];
  SharedTable<F> tab{table};
  int32_t digits[K][260];
  WnafState<K> st;
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t i = t + (size_t)j * T;
    const bool active = i < n;
    Scalar s = ld_scalar(k + 4 * (active ? i : n - 1));
    if (!active) {
#pragma unroll
      for (int w = 0; w < 8; w++) s.v[w] = 0;
    }
    st.i[j] = wnaf_form(digits[j], s, window) - 1;
    st.found[j] = false; st.doubled[j] = false;
    pt_set_zero(res[j]);
  }
  pt_wnaf_run_lazy<F, K>(res, tab, digits, st);
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t i = t + (size_t)j * T;
    if (i < n) st_jac(out + (size_t)PW * i, res[j]);
  }
}

// CurveProjective::mul_assign (ec.rs:534-553): MSB-first double-and-add.  Its operation sequence -- a doubling per bit once the
// leading one has been seen, an addition of the base when the bit is set -- is wnaf_exp's (wnaf.rs:49-71) with digits in {0, 1} and a
// one-entry table, so it runs on the decoupled-lane runner of the wNAF kernel (K points per lane; lock-step SIMT would execute an
// addition for every bit position as long as ANY lane of the warp has that bit set).  Same Jacobian triple as the reference.
template <class F, int K> struct BaseTable {
  Jac<F> b[K];
  __device__ __forceinline__ Jac<F> get(int j, int) const { return b[j]; }
};
template <class F, bool IS_G2, int K>
__global__ void __launch_bounds__(128, IS_G2 ? BLS_WNAF_MINB : BLS_WNAF_MINB_G1) k_pt_mul(const uint64_t* bases, const uint64_t* k, uint64_t* out, size_t n) {
  const size_t T = (size_t)gridDim.x * blockDim.x;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  Jac<F> res[K];
  BaseTable<F, K> table;
  int8_t digits[K][260];
  WnafState<K> st;
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t i = t + (size_t)j * T;
    const bool active = i < n;
    if (!active) i = n - 1;
    ld_jac(table.b[j], bases + (size_t)PW * i);
    Scalar s = ld_scalar(k + 4 * i);
    if (!active) {
#pragma unroll
      for (int w = 0; w < 8; w++) s.v[w] = 0;
    }
    const int nb = scalar_num_bits(s);
#pragma unroll 1
    for (int b = 0; b < nb; b++) digits[j][b] = (int8_t)((s.v[b >> 5] >> (b & 31)) & 1u);
    st.i[j] = nb - 1;
    st.found[j] = false; st.doubled[j] = false;
    pt_set_zero(res[j]);
  }
  pt_wnaf_run_lazy<F, K>(res, table, digits, st);
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    const size_t i = t + (size_t)j * T;
    if (i < n) st_jac(out + (size_t)PW * i, res[j]);
  }
}

template <class F>
__global__ void __launch_bounds__(128) k_pt_op(int op, const uint64_t* a, const uint64_t* b, uint64_t* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int PW = 3 * FW<F>::W, AW = 2 * FW<F>::W + 1;
  Jac<F> x, y;
  ld_jac(x, a + (size_t)PW * i);
  switch (op) {
    case BLS_PT_DOUBLE: pt_double(x); break;
    case BLS_PT_ADD: ld_jac(y, b + (size_t)PW * i); pt_add(x, y); break;
    case BLS_PT_SUB: ld_jac(y, b + (size_t)PW * i); pt_negate(y); pt_add(x, y); break;
    case BLS_PT_ADD_MIXED: { Aff<F> o; ld_aff(o, b + (size_t)AW * i); pt_add_mixed(x, o); break; }
    case BLS_PT_NEGATE: pt_negate(x); break;
  }
  st_jac(out + (size_t)PW * i, x);
}

template <class F>
__global__ void __launch_bounds__(128) k_into_affine(const uint64_t* in, uint64_t* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int PW = 3 * FW<F>::W, AW = 2 * FW<F>::W + 1;
  Jac<F> x;
  Aff<F> o;
  ld_jac(x, in + (size_t)PW * i);
  pt_into_affine(o, x);
  st_aff(out + (size_t)AW * i, o);
}

// CurveProjective::batch_normalization (ec.rs:246-294).  The reference runs Montgomery's trick over
// the whole slice with one inversion; the outputs (x/z^2, y/z^3, one) are canonical field values, so
// any partition of the trick gives the same bits.  Here thread t owns points t, t+T, ... : a forward
// pass of prefix products of z (kept in `scratch`, one coordinate per point), one inversion per
// thread, and a backward pass that yields 1/z and applies the affine map at once.
template <class F>
__global__ void __launch_bounds__(128) k_batch_normalization(uint64_t* pts, size_t n, uint64_t* scratch) {
  const size_t T = (size_t)gridDim.x * blockDim.x;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int W = FW<F>::W, PW = 3 * W;
  F one; f_set_one(one);
  F acc = one;
  size_t last = t;
  bool any = false;
  // forward pass; the next z is loaded before the current product so that the load latency overlaps the arithmetic
  F znext; ld_F(znext, pts + (size_t)PW * t + 2 * W);
#pragma unroll 1
  for (size_t i = t; i < n; i += T) {
    const F z = znext;
    if (i + T < n) ld_F(znext, pts + (size_t)PW * (i + T) + 2 * W);
    last = i;
    if (f_is_zero(z) || f_eq(z, one)) continue;   // is_normalized, ec.rs:242-244
    st_F(scratch + (size_t)W * i, acc);           // product of the previous live z's
    acc = f_mul(acc, z);
    any = true;
  }
  if (!any) return;
  F inv; f_inv(inv, acc);
  // backward pass, same prefetching: (z, prefix, x, y) of the next point are in flight during the 6 products
  F zn, pn, xn, yn;
  ld_F(zn, pts + (size_t)PW * last + 2 * W); ld_F(pn, scratch + (size_t)W * last);
  ld_F(xn, pts + (size_t)PW * last); ld_F(yn, pts + (size_t)PW * last + W);
#pragma unroll 1
  for (size_t i = last;; i -= T) {
    uint64_t* pi = pts + (size_t)PW * i;
    const F z = zn, prev = pn, x = xn, y = yn;
    const bool more = i >= T + t;                 // i == t was the first point of this thread
    if (more) {
      const size_t j = i - T;
      ld_F(zn, pts + (size_t)PW * j + 2 * W); ld_F(pn, scratch + (size_t)W * j);
      ld_F(xn, pts + (size_t)PW * j); ld_F(yn, pts + (size_t)PW * j + W);
    }
    if (!(f_is_zero(z) || f_eq(z, one))) {
      F zinv = f_mul(inv, prev);
      inv = f_mul(inv, z);
      F zz = f_sqr(zinv);
      st_F(pi, f_mul(x, zz));
      st_F(pi + W, f_mul(y, f_mul(zz, zinv)));
      st_F(pi + 2 * W, one);
    }
    if (!more) break;
  }
}

// ------------------------------------------------------------------------------------------------
// Point encodings (codec.cuh): thread per element
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(128) k_decode(const uint8_t* bytes, int compressed, int checked, uint64_t* out, uint8_t* status, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int AW = 2 * FW<F>::W + 1;
  const size_t size = (size_t)FBytes<F>::N * (compressed ? 1 : 2);
  Aff<F> p;
  int st = decode_point(p, bytes + size * i, compressed != 0, checked != 0);
  st_aff(out + (size_t)AW * i, p);
  status[i] = (uint8_t)st;
}
template <class F>
__global__ void __launch_bounds__(128) k_encode(const uint64_t* in, int compressed, uint8_t* bytes, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int AW = 2 * FW<F>::W + 1;
  const size_t size = (size_t)FBytes<F>::N * (compressed ? 1 : 2);
  Aff<F> p;
  ld_aff(p, in + (size_t)AW * i);
  encode_point(bytes + size * i, p, compressed != 0);
}

// $affine::get_point_from_x (ec.rs:102-123) and scale_by_cofactor: G::rand with the randomness supplied by the caller
template <class F>
__global__ void __launch_bounds__(128) k_point_from_x(const uint64_t* x, const uint8_t* greatest, uint64_t* out, uint8_t* is_some, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int AW = 2 * FW<F>::W + 1;
  F xv; ld_F(xv, x + (size_t)FW<F>::W * i);
  Aff<F> p;
  const bool ok = get_point_from_x(p, xv, greatest[i] != 0);
  if (!ok) { f_set_zero(p.x); f_set_one(p.y); p.inf = true; }
  st_aff(out + (size_t)AW * i, p);
  is_some[i] = ok;
}
template <class F, bool IS_G2>
__global__ void __launch_bounds__(128) k_scale_by_cofactor(const uint64_t* in, uint64_t* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int AW = 2 * FW<F>::W + 1, PW = 3 * FW<F>::W;
  Aff<F> p; ld_aff(p, in + (size_t)AW * i);
  Jac<F> r;
  scale_by_cofactor(r, p, IS_G2 ? BLS_G2_COFACTOR : BLS_G1_COFACTOR, IS_G2 ? 16 : 4);
  st_jac(out + (size_t)PW * i, r);
}

// CurveAffine::mul (ec.rs:174-177): $affine::mul_bits over all 256 bits of the scalar, MSB first, mixed additions
template <class F>
__global__ void __launch_bounds__(128) k_affine_mul(const uint64_t* in, const uint64_t* k, uint64_t* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int AW = 2 * FW<F>::W + 1, PW = 3 * FW<F>::W;
  Aff<F> p; ld_aff(p, in + (size_t)AW * i);
  const Scalar s = ld_scalar(k + 4 * i);
  Jac<F> r;
  scale_by_cofactor(r, p, s.v, 8);
  st_jac(out + (size_t)PW * i, r);
}

// ------------------------------------------------------------------------------------------------
// Integer-multiply peak microbenchmarks (roofline denominator)
// ------------------------------------------------------------------------------------------------
#define PEAK_CHAINS 8
#define PEAK_UNROLL 32
// 32x32->64 multiplies only: each chain squares its own 64-bit value, (lo, hi) <- lo * hi, so that both halves
// of every product are consumed by the next multiply and nothing but IMAD.WIDE.U32 is left in the loop
// (tests/test_abi.py disassembles the library and checks this).  A loop-invariant `mad.wide acc, a, b, acc`
// is NOT a multiply benchmark: ptxas hoists a*b and the loop degenerates into 64-bit adds on the alu pipe.
__global__ void __launch_bounds__(256) k_imad_wide_peak(uint32_t seed, int iters, uint64_t* sink) {
  uint32_t lo[PEAK_CHAINS], hi[PEAK_CHAINS];
  uint32_t b = seed ^ (threadIdx.x * 2654435761u);
#pragma unroll
  for (int k = 0; k < PEAK_CHAINS; k++) { lo[k] = b * (2 * k + 3) + 1; hi[k] = (b ^ seed) + 77 * k; }
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < PEAK_UNROLL; u++) {
#pragma unroll
      for (int k = 0; k < PEAK_CHAINS; k++)
        asm volatile("{.reg .u64 t; mul.wide.u32 t, %1, %0; mov.b64 {%0, %1}, t;}" : "+r"(lo[k]), "+r"(hi[k]));
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < PEAK_CHAINS; k++) s ^= lo[k] ^ hi[k];
  if (s == 0x1234567u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_imad32_peak(uint32_t seed, int iters, uint64_t* sink) {
  uint32_t acc[PEAK_CHAINS];
  uint32_t a[PEAK_CHAINS];
  uint32_t b = seed ^ (threadIdx.x * 2654435761u);
#pragma unroll
  for (int k = 0; k < PEAK_CHAINS; k++) { acc[k] = seed + k; a[k] = b * (k + 3) + 1; }
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < PEAK_UNROLL; u++) {
#pragma unroll
      for (int k = 0; k < PEAK_CHAINS; k++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[k]) : "r"(a[k]), "r"(b));
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < PEAK_CHAINS; k++) s ^= acc[k];
  if (s == 0x1234567u) sink[0] = s;
}
// the shape fp_mul issues: carry-linked IMAD.WIDE.U32.X rows; 300 MAC32 per fp_mul
__global__ void __launch_bounds__(256) k_fpmul_peak(uint32_t seed, int iters, uint64_t* sink) {
  Fp x = fp_one(), y = fp_r2();
  x.v[0] ^= seed ^ threadIdx.x;
  y.v[1] ^= seed;
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
    x = fp_mul_inline(x, y);
    y = fp_mul_inline(y, x);
  }
  if (x.v[0] == 0x1234567u && y.v[3] == 7u) sink[0] = x.v[1];
}

// the dedicated squaring (fp_sqr_gen.cuh): 222 wide MACs + 12 IMAD = 234 MAC32 per squaring, two independent chains
__global__ void __launch_bounds__(256) k_fpsqr_peak(uint32_t seed, int iters, uint64_t* sink) {
  Fp x = fp_one(), y = fp_r2();
  x.v[0] ^= seed ^ threadIdx.x;
  y.v[1] ^= seed + 77u * threadIdx.x;
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
    x = fp_sqr_inline(x);
    y = fp_sqr_inline(y);
  }
  if (x.v[0] == 0x1234567u && y.v[3] == 7u) sink[0] = x.v[1];
}

// carry-linked rows only: 2 x (12-word mad.lo.cc/madc.hi.cc chain) per step, no reduction, no adds
__global__ void __launch_bounds__(256) k_carry_row_peak(uint32_t seed, int iters, uint64_t* sink) {
  uint32_t e[12], o[12], x[12];
#pragma unroll
  for (int k = 0; k < 12; k++) { e[k] = seed + k; o[k] = seed * 3 + k; x[k] = (seed ^ threadIdx.x) * (2 * k + 1) + 1; }
  uint32_t b = seed ^ (threadIdx.x * 2654435761u);
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      fp_cmad_row(e, &x[0], b, o[11]);
      fp_cmad_row(o, &x[1], b, e[11]);
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 12; k++) s ^= e[k] ^ o[k];
  if (s == 0x1234567u) sink[0] = s;
}

// ------------------------------------------------------------------------------------------------
// Host side: context + C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

void bls_ctx_destroy(bls_ctx* ctx);
bls_ctx* bls_ctx_create(int device, int* err) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) { if (err) *err = BLS_ERR_NO_DEVICE; return nullptr; }
  if (device < 0 || device >= count) { if (err) *err = BLS_ERR_INVALID_ARGUMENT; return nullptr; }
  bls_ctx* ctx = new (std::nothrow) bls_ctx();
  if (!ctx) { if (err) *err = BLS_ERR_OUT_OF_MEMORY; return nullptr; }
  ctx->device = device;
  ctx->launches = 0;
  ctx->mm_smem_ready = false;
  ctx->wide_pairing_max = BLS_WIDE_PAIRING_MAX;
  ctx->wide_final_exp_max = BLS_WIDE_FINAL_EXP_MAX;
  ctx->last_error[0] = 0;
  DevGuard guard;
  ctx->stream = ctx->stream2 = ctx->copy_in = ctx->copy_out = nullptr;
  ctx->pool = nullptr;
  for (int k = 0; k < 2; k++) ctx->ev_in[k] = ctx->ev_k[k] = ctx->ev_out[k] = nullptr;
  cudaMemPoolProps props = {};
  props.allocType = cudaMemAllocationTypePinned;
  props.handleTypes = cudaMemHandleTypeNone;
  props.location.type = cudaMemLocationTypeDevice;
  props.location.id = device;
  uint64_t keep = UINT64_MAX;                       // never hand cached staging memory back at a synchronisation point
  bool ok = guard.enter(device) == cudaSuccess &&
            cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) == cudaSuccess &&
            cudaMemPoolCreate(&ctx->pool, &props) == cudaSuccess &&
            cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep) == cudaSuccess;
  for (int k = 0; k < 2 && ok; k++)
    ok = cudaEventCreateWithFlags(&ctx->ev_in[k], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_k[k], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_out[k], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    if (err) *err = BLS_ERR_CUDA;
    bls_ctx_destroy(ctx);
    return nullptr;
  }
  if (err) *err = BLS_OK;
  return ctx;
}

void bls_ctx_destroy(bls_ctx* ctx) {
  if (!ctx) return;
  DevGuard guard;
  guard.enter(ctx->device);
  for (cudaStream_t s : {ctx->stream, ctx->stream2, ctx->copy_in, ctx->copy_out})
    if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  for (int k = 0; k < 2; k++)
    for (cudaEvent_t e : {ctx->ev_in[k], ctx->ev_k[k], ctx->ev_out[k]})
      if (e) cudaEventDestroy(e);
  if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
  delete ctx;
}
// hand the staging memory the context caches between calls back to the driver (keep at most keep_bytes)
int bls_ctx_trim(bls_ctx* ctx, size_t keep_bytes) {
  if (!ctx) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemPoolTrimTo(ctx->pool, keep_bytes));
  return BLS_OK;
}

const char* bls_strerror(int status) {
  switch (status) {
    case BLS_OK: return "ok";
    case BLS_ERR_INVALID_ARGUMENT: return "invalid argument";
    case BLS_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
    case BLS_ERR_CUDA: return "CUDA error (see bls_ctx_last_error)";
    case BLS_ERR_OUT_OF_MEMORY: return "out of device memory";
    case BLS_ERR_UNSUPPORTED: return "unsupported";
  }
  return "unknown status";
}
const char* bls_ctx_last_error(const bls_ctx* ctx) { return ctx ? ctx->last_error : ""; }
int bls_ctx_device(const bls_ctx* ctx) { return ctx ? ctx->device : -1; }
int bls_ctx_sm_count(const bls_ctx* ctx) { return ctx ? ctx->sm_count : 0; }
uint64_t bls_ctx_launch_count(const bls_ctx* ctx) { return ctx ? ctx->launches : 0; }
int bls_ctx_set_latency_path_limits(bls_ctx* ctx, size_t max_pairings, size_t max_final_exps) {
  if (!ctx) return BLS_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  ctx->wide_pairing_max = max_pairings;
  ctx->wide_final_exp_max = max_final_exps;
  return BLS_OK;
}

}  // extern "C"

// ---- device-pointer entry points --------------------------------------------------------------
template <class F, bool IS_G2, int KSMALL>
static int wnaf_mul_dev_impl(bls_ctx* ctx, const void* bases, const bls_fr_repr* k, void* out, size_t n, int window, void* stream) {
  if (!ctx || (n && (!bases || !k || !out)) || (window != 0 && (window < 2 || window > BLS_MAX_WNAF_EXPLICIT_WINDOW))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  cudaStream_t s = pick(ctx, stream);
  if (window <= 4) {
    k_wnaf_mul_lazyk<F, IS_G2, KSMALL, 8><<<blocks_for((n + KSMALL - 1) / KSMALL, TPB), TPB, 0, s>>>((const uint64_t*)bases, (const uint64_t*)k, (uint64_t*)out, n, window);
  } else if (window <= BLS_MAX_WNAF_WINDOW) {
    k_wnaf_mul_lazyk<F, IS_G2, 1, BLS_MAX_WNAF_TABLE><<<blocks_for(n, TPB), TPB, 0, s>>>((const uint64_t*)bases, (const uint64_t*)k, (uint64_t*)out, n, window);
  } else {
    // per-point tables in a stream-ordered scratch allocation from the context's pool
    const unsigned blocks = blocks_for(n, TPB);
    const size_t rows = (size_t)blocks * TPB, row_bytes = ((size_t)1 << (window - 1)) * (IS_G2 ? sizeof(bls_g2) : sizeof(bls_g1));
    void* tables = nullptr;
    CK(cudaMallocFromPoolAsync(&tables, rows * row_bytes, ctx->pool, s));
    k_wnaf_mul_bigwindow<F><<<blocks, TPB, 0, s>>>((const uint64_t*)bases, (const uint64_t*)k, (uint64_t*)out, n, window, (uint64_t*)tables);
    cudaError_t le = cudaGetLastError();
    cudaFreeAsync(tables, s);
    ctx->launches++;
    CK(le);
    return BLS_OK;
  }
  LAUNCH_CHECK();
  return BLS_OK;
}
extern "C" {
// product tree: a pass over `count` factors uses ceil(count/8) threads
static size_t prod_threads(size_t count) { return count ? (count + 7) / 8 : 1; }
size_t bls_fq12_product_scratch_bytes(const bls_ctx* ctx, size_t n) {
  (void)ctx;
  return 2 * prod_threads(n) * sizeof(bls_fq12);
}
int bls_internal_product_passes(bls_ctx* ctx, const uint64_t* in, size_t count, bls_fq12* out1, uint64_t* scratch, cudaStream_t s) {
  // scratch holds two ping-pong arrays of prod_threads(count) Fq12 each
  const size_t cap = prod_threads(count);
  uint64_t* bufs[2] = {scratch, scratch + cap * FQ12_W};
  int which = 0;
  const uint64_t* src = in;
  while (true) {
    size_t T = prod_threads(count);
    uint64_t* dst = T == 1 ? (uint64_t*)out1 : bufs[which];
    k_fq12_product<<<blocks_for(T, TPB), TPB, 0, s>>>(src, count, dst, T);
    LAUNCH_CHECK();
    if (T == 1) return BLS_OK;
    src = dst;
    count = T;
    which ^= 1;
  }
}

// Engine::pairing(p, q) with p: Into<G1Affine>, q: Into<G2Affine> on PROJECTIVE inputs (lib.rs:101-109; the crate's bench_pairing_full
// calls it this way): small batches run the conversions inside the warp-cooperative pairing kernel, large ones convert with
// k_into_affine into pool-allocated affine rows and run the throughput kernel
int bls_pairing_projective_dev(bls_ctx* ctx, const bls_g1* p, const bls_g2* q, bls_fq12* out, size_t n, void* stream) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  cudaStream_t s = pick(ctx, stream);
  if (n <= ctx->wide_pairing_max) return bls_internal_wide_pairing_projective(ctx, p, q, out, n, s);
  void *pa = nullptr, *qa = nullptr;
  CK(cudaMallocFromPoolAsync(&pa, n * sizeof(bls_g1_affine), ctx->pool, s));
  cudaError_t e = cudaMallocFromPoolAsync(&qa, n * sizeof(bls_g2_affine), ctx->pool, s);
  if (e != cudaSuccess) { cudaFreeAsync(pa, s); CK(e); }
  k_into_affine<Fp><<<blocks_for(n, TPB), TPB, 0, s>>>((const uint64_t*)p, (uint64_t*)pa, n);
  k_into_affine<Fp2><<<blocks_for(n, TPB), TPB, 0, s>>>((const uint64_t*)q, (uint64_t*)qa, n);
  ctx->launches += 2;
  int rc = cudaGetLastError() == cudaSuccess ? bls_pairing_dev(ctx, (const bls_g1_affine*)pa, (const bls_g2_affine*)qa, out, n, stream) : BLS_ERR_CUDA;
  cudaFreeAsync(pa, s);
  cudaFreeAsync(qa, s);
  return rc;
}

int bls_fq12_product_dev(bls_ctx* ctx, const bls_fq12* in, size_t n, bls_fq12* out1, void* scratch, void* stream) {
  if (!ctx || !out1 || (n && (!in || !scratch))) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t s = pick(ctx, stream);
  if (n == 0) {   // empty product = one
    k_fq12_product<<<1, TPB, 0, s>>>((const uint64_t*)in, 0, (uint64_t*)out1, 1);
    LAUNCH_CHECK();
    return BLS_OK;
  }
  return bls_internal_product_passes(ctx, (const uint64_t*)in, n, out1, (uint64_t*)scratch, s);
}

int bls_g1_wnaf_mul_dev(bls_ctx* ctx, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n, int window, void* stream) {
  return wnaf_mul_dev_impl<Fp, false, BLS_WNAF_K>(ctx, bases, k, out, n, window, stream);
}
int bls_g2_wnaf_mul_dev(bls_ctx* ctx, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n, int window, void* stream) {
  return wnaf_mul_dev_impl<Fp2, true, BLS_WNAF_K_G2>(ctx, bases, k, out, n, window, stream);
}

int bls_g1_wnaf_table_dev(bls_ctx* ctx, const bls_g1* base, int window, bls_g1* table, void* stream) {
  if (!ctx || !base || !table || window < 2 || window > BLS_MAX_WNAF_FIXED_WINDOW) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  k_wnaf_table<Fp><<<1, 32, 0, pick(ctx, stream)>>>((const uint64_t*)base, (uint64_t*)table, window);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_g2_wnaf_table_dev(bls_ctx* ctx, const bls_g2* base, int window, bls_g2* table, void* stream) {
  if (!ctx || !base || !table || window < 2 || window > BLS_MAX_WNAF_FIXED_WINDOW) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  k_wnaf_table<Fp2><<<1, 32, 0, pick(ctx, stream)>>>((const uint64_t*)base, (uint64_t*)table, window);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_g1_wnaf_fixed_base_dev(bls_ctx* ctx, const bls_g1* table, int window, const bls_fr_repr* k, bls_g1* out, size_t n, void* stream) {
  if (!ctx || window < 2 || window > BLS_MAX_WNAF_FIXED_WINDOW || (n && (!table || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_wnaf_fixed_base<Fp, 2><<<blocks_for((n + 1) / 2, TPB), TPB, 0, pick(ctx, stream)>>>((const uint64_t*)table, window, (const uint64_t*)k, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_g2_wnaf_fixed_base_dev(bls_ctx* ctx, const bls_g2* table, int window, const bls_fr_repr* k, bls_g2* out, size_t n, void* stream) {
  if (!ctx || window < 2 || window > BLS_MAX_WNAF_FIXED_WINDOW || (n && (!table || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_wnaf_fixed_base<Fp2, 2><<<blocks_for((n + 1) / 2, TPB), TPB, 0, pick(ctx, stream)>>>((const uint64_t*)table, window, (const uint64_t*)k, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}

// threads for batch normalisation: >= 64 points per thread when n allows it
static size_t bn_threads(const bls_ctx* ctx, size_t n) {
  size_t t = (n + 63) / 64;
  size_t cap = (size_t)ctx->sm_count * 4 * TPB;   // more points per thread for huge batches: the per-thread inversion (476 M) amortises better
  if (t > cap) t = cap;
  t = (t + TPB - 1) / TPB * TPB;
  return t ? t : TPB;
}
size_t bls_batch_normalization_scratch_bytes(const bls_ctx* ctx, int degree, size_t n) {
  (void)ctx;
  return n * (degree == 2 ? sizeof(bls_fq2) : sizeof(bls_fq));
}
int bls_g1_batch_normalization_dev(bls_ctx* ctx, bls_g1* inout, size_t n, void* scratch, void* stream) {
  if (!ctx || (n && (!inout || !scratch))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t T = bn_threads(ctx, n);
  k_batch_normalization<Fp><<<(unsigned)(T / TPB), TPB, 0, pick(ctx, stream)>>>((uint64_t*)inout, n, (uint64_t*)scratch);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_g2_batch_normalization_dev(bls_ctx* ctx, bls_g2* inout, size_t n, void* scratch, void* stream) {
  if (!ctx || (n && (!inout || !scratch))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t T = bn_threads(ctx, n);
  k_batch_normalization<Fp2><<<(unsigned)(T / TPB), TPB, 0, pick(ctx, stream)>>>((uint64_t*)inout, n, (uint64_t*)scratch);
  LAUNCH_CHECK();
  return BLS_OK;
}

}  // extern "C"

// ---- host-pointer entry points: stage through stream-ordered device buffers (DevBuf, H2D/D2H: abi_common.cuh)
// Large element-wise batches run as a two-deep pipeline of chunks: the H2D copy of chunk i + 1 (stream copy_in) and the
// D2H copy of chunk i - 1 (stream copy_out) overlap the kernel of chunk i (ctx->stream), with two sets of staging buffers.
// With pinned host memory all three legs are asynchronous; with pageable memory the copies block the host while the
// kernel of the neighbouring chunk runs, which overlaps just the same.  For config 4 (2^24 G1 points: 2.95 GB in, 2.4 GB out)
// the copies are 13 % of the kernel time when run back to back.
namespace {
struct PipeIn { const void* host; size_t stride; };
template <class Launch>
int run_pipelined(bls_ctx* ctx, size_t n, size_t chunk, const PipeIn* in, int n_in, void* host_out, size_t out_stride, Launch launch, bool two_kernel_streams = false) {
  const size_t nchunks = (n + chunk - 1) / chunk;
  // two_kernel_streams: the kernels of consecutive chunks go to two streams, so that the blocks of chunk c + 1 fill the SMs as the
  // last wave of chunk c drains (one launch over the whole batch would do the same) while the D2H of chunk c already runs.  Only
  // for launches that share no scratch between chunks.
  cudaStream_t ks[2] = {ctx->stream, two_kernel_streams ? ctx->stream2 : ctx->stream};
  DevBuf din[2][3] = {{DevBuf(ctx), DevBuf(ctx), DevBuf(ctx)}, {DevBuf(ctx), DevBuf(ctx), DevBuf(ctx)}};
  DevBuf dout[2] = {DevBuf(ctx), DevBuf(ctx)};
  const size_t csz = n < chunk ? n : chunk;
  for (int b = 0; b < (nchunks > 1 ? 2 : 1); b++) {
    for (int k = 0; k < n_in; k++) CK(din[b][k].alloc(csz * in[k].stride));
    CK(dout[b].alloc(csz * out_stride));
  }
  CK(cudaEventRecord(ctx->ev_k[0], ctx->stream));      // the allocations are ordered on ctx->stream: the copy streams wait for them
  CK(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[0], 0));
  CK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[0], 0));
  if (two_kernel_streams) CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_k[0], 0));
  for (size_t c = 0; c < nchunks; c++) {
    const int b = (int)(c & 1);
    const size_t lo = c * chunk, cn = (n - lo) < chunk ? (n - lo) : chunk;
    if (c >= 2) CK(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[b], 0));          // the kernel of chunk c - 2 has read this input set
    for (int k = 0; k < n_in; k++)
      CK(cudaMemcpyAsync(din[b][k].p, (const char*)in[k].host + lo * in[k].stride, cn * in[k].stride, cudaMemcpyHostToDevice, ctx->copy_in));
    CK(cudaEventRecord(ctx->ev_in[b], ctx->copy_in));
    CK(cudaStreamWaitEvent(ks[b], ctx->ev_in[b], 0));
    if (c >= 2) CK(cudaStreamWaitEvent(ks[b], ctx->ev_out[b], 0));                // the D2H of chunk c - 2 has drained this output set
    const void* ptrs[3] = {din[b][0].p, din[b][1].p, din[b][2].p};
    TRY(launch(ptrs, dout[b].p, cn, ks[b]));
    CK(cudaEventRecord(ctx->ev_k[b], ks[b]));
    CK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[b], 0));
    CK(cudaMemcpyAsync((char*)host_out + lo * out_stride, dout[b].p, cn * out_stride, cudaMemcpyDeviceToHost, ctx->copy_out));
    CK(cudaEventRecord(ctx->ev_out[b], ctx->copy_out));
  }
  CK(cudaStreamSynchronize(ctx->copy_out));
  if (two_kernel_streams) CK(cudaStreamSynchronize(ctx->stream2));
  CK(cudaStreamSynchronize(ctx->stream));              // the staging buffers are freed in ctx->stream order
  return BLS_OK;
}
// pairings per chunk of the host-buffer pairing / Miller-loop calls: ONE wave of the lane-pair kernels (2 blocks of 64 lane pairs
// per SM, pair_io.cuh) -- 18 944 on a B200.  The chunk kernels alternate between two streams (run_pipelined), so a 2^16 batch still
// runs as 3.46 back-to-back waves, but only the first chunk's H2D (5.8 MB) and the last chunk's D2H are exposed instead of the
// whole 19.9 MB in and 37.7 MB out.
static size_t pipe_chunk_pairings(const bls_ctx* ctx) { return (size_t)ctx->sm_count * 128; }
const size_t PIPE_CHUNK_POINTS = (size_t)1 << 21;
}  // namespace

extern "C" {

int bls_g2_prepare_batch(bls_ctx* ctx, const bls_g2_affine* q, bls_g2_prepared* out, size_t n) {
  if (!ctx || (n && (!q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(dq, q, n * sizeof(*q));
  DALLOC(dout, n * sizeof(*out));
  TRY(bls_g2_prepare_dev(ctx, (const bls_g2_affine*)dq.p, (bls_g2_prepared*)dout.p, n, nullptr));
  D2H(out, dout, n * sizeof(*out));
  SYNC();
  return BLS_OK;
}

static int miller_like(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, bool final_exp) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const PipeIn in[2] = {{p, sizeof(*p)}, {q, sizeof(*q)}};
  return run_pipelined(ctx, n, pipe_chunk_pairings(ctx), in, 2, out, sizeof(*out), [&](const void* const* d, void* o, size_t cn, cudaStream_t s) -> int {
    return final_exp ? bls_pairing_dev(ctx, (const bls_g1_affine*)d[0], (const bls_g2_affine*)d[1], (bls_fq12*)o, cn, s)
                     : bls_miller_loop_dev(ctx, (const bls_g1_affine*)d[0], (const bls_g2_affine*)d[1], (bls_fq12*)o, cn, s);
  }, true);
}
int bls_pairing_projective_batch(bls_ctx* ctx, const bls_g1* p, const bls_g2* q, bls_fq12* out, size_t n) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const PipeIn in[2] = {{p, sizeof(*p)}, {q, sizeof(*q)}};
  return run_pipelined(ctx, n, (size_t)1 << 16, in, 2, out, sizeof(*out), [&](const void* const* d, void* o, size_t cn, cudaStream_t s) -> int {
    return bls_pairing_projective_dev(ctx, (const bls_g1*)d[0], (const bls_g2*)d[1], (bls_fq12*)o, cn, s);
  });
}
int bls_miller_loop_batch(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n) { return miller_like(ctx, p, q, out, n, false); }
int bls_pairing_batch(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n) { return miller_like(ctx, p, q, out, n, true); }

int bls_miller_loop_prepared_batch(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q, bls_fq12* out, size_t n) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(dp, p, n * sizeof(*p));
  H2D(dq, q, n * sizeof(*q));
  DALLOC(dout, n * sizeof(*out));
  TRY(bls_miller_loop_prepared_dev(ctx, (const bls_g1_affine*)dp.p, (const bls_g2_prepared*)dq.p, (bls_fq12*)dout.p, n, nullptr));
  D2H(out, dout, n * sizeof(*out));
  SYNC();
  return BLS_OK;
}

static int shared_q_host(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n, int final_exp) {
  if (!ctx || !q1 || (n && (!p || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(dp, p, n * sizeof(*p));
  H2D(dq, q1, sizeof(*q1));
  DALLOC(dout, n * sizeof(*out));
  TRY(bls_miller_loop_shared_q_dev(ctx, (const bls_g1_affine*)dp.p, (const bls_g2_prepared*)dq.p, (bls_fq12*)dout.p, n, final_exp, nullptr));
  D2H(out, dout, n * sizeof(*out));
  SYNC();
  return BLS_OK;
}
int bls_miller_loop_shared_q_batch(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n) { return shared_q_host(ctx, p, q1, out, n, 0); }
int bls_pairing_shared_q_batch(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n) { return shared_q_host(ctx, p, q1, out, n, 1); }

static int multi_miller_host(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, int final_exp, uint8_t* is_some) {
  if (!ctx || !out1 || (n && (!p || !q))) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  H2D(dp, p, n * sizeof(*p));
  H2D(dq, q, n * sizeof(*q));
  DALLOC(dscr, bls_multi_miller_scratch_bytes(ctx, n));
  DALLOC(dout, sizeof(*out1) + 8);
  uint8_t* dsome = (uint8_t*)dout.p + sizeof(*out1);
  if (final_exp) TRY(bls_pairing_product_dev(ctx, (const bls_g1_affine*)dp.p, (const bls_g2_affine*)dq.p, n, (bls_fq12*)dout.p, dsome, dscr.p, nullptr));
  else TRY(bls_multi_miller_loop_dev(ctx, (const bls_g1_affine*)dp.p, (const bls_g2_affine*)dq.p, n, (bls_fq12*)dout.p, dscr.p, nullptr));
  D2H(out1, dout, sizeof(*out1));
  if (final_exp && is_some) CK(cudaMemcpyAsync(is_some, dsome, 1, cudaMemcpyDeviceToHost, ctx->stream));
  SYNC();
  return BLS_OK;
}
int bls_multi_miller_loop(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1) { return multi_miller_host(ctx, p, q, n, out1, 0, nullptr); }
// final_exponentiation(miller_loop(pairs)) in one call -- the batch-verification shape of BASELINE configs[2]
int bls_pairing_product(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, uint8_t* is_some) { return multi_miller_host(ctx, p, q, n, out1, 1, is_some); }

int bls_multi_miller_loop_prepared(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q, size_t n, bls_fq12* out1) {
  if (!ctx || !out1 || (n && (!p || !q))) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  H2D(dp, p, n * sizeof(*p));
  H2D(dq, q, n * sizeof(*q));
  size_t T = bls_internal_mm_lane_pairs(ctx, n);      // one partial product per block
  DALLOC(dpart, T * sizeof(bls_fq12));
  DALLOC(dout, sizeof(*out1));
  if (n) TRY(bls_internal_multi_miller_prepared(ctx, (const bls_g1_affine*)dp.p, (const bls_g2_prepared*)dq.p, n, (bls_fq12*)dpart.p, ctx->stream));
  TRY(bls_internal_product_tail(ctx, (const bls_fq12*)dpart.p, n ? T : 0, (bls_fq12*)dout.p, 0, nullptr, ctx->stream));
  D2H(out1, dout, sizeof(*out1));
  SYNC();
  return BLS_OK;
}

int bls_final_exponentiation_batch(bls_ctx* ctx, const bls_fq12* in, bls_fq12* out, uint8_t* is_some, size_t n) {
  if (!ctx || (n && (!in || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(din, in, n * sizeof(*in));
  DALLOC(dout, n * sizeof(*out));
  DALLOC(dok, n);
  TRY(bls_final_exponentiation_dev(ctx, (const bls_fq12*)din.p, (bls_fq12*)dout.p, (uint8_t*)dok.p, n, nullptr));
  D2H(out, dout, n * sizeof(*out));
  if (is_some) D2H(is_some, dok, n);
  SYNC();
  return BLS_OK;
}

int bls_fq12_product(bls_ctx* ctx, const bls_fq12* in, size_t n, bls_fq12* out1) {
  if (!ctx || !out1 || (n && !in)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  H2D(din, in, n * sizeof(*in));
  DALLOC(dscr, bls_fq12_product_scratch_bytes(ctx, n));
  DALLOC(dout, sizeof(*out1));
  TRY(bls_fq12_product_dev(ctx, (const bls_fq12*)din.p, n, (bls_fq12*)dout.p, dscr.p, nullptr));
  D2H(out1, dout, sizeof(*out1));
  SYNC();
  return BLS_OK;
}

int bls_fq12_pow_batch(bls_ctx* ctx, const bls_fq12* a, const bls_fr_repr* k, bls_fq12* out, size_t n) {
  if (!ctx || (n && (!a || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(da, a, n * sizeof(*a));
  H2D(dk, k, n * sizeof(*k));
  DALLOC(dout, n * sizeof(*out));
  TRY(bls_fq12_pow_dev(ctx, (const bls_fq12*)da.p, (const bls_fr_repr*)dk.p, (bls_fq12*)dout.p, n, nullptr));
  D2H(out, dout, n * sizeof(*out));
  SYNC();
  return BLS_OK;
}

static int wnaf_host(bls_ctx* ctx, int degree, const void* bases, const bls_fr_repr* k, void* out, size_t n, int window, int mode) {
  if (!ctx || (n && (!bases || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const PipeIn in[2] = {{bases, pb}, {k, sizeof(*k)}};
  return run_pipelined(ctx, n, PIPE_CHUNK_POINTS, in, 2, out, pb, [&](const void* const* d, void* o, size_t cn, cudaStream_t ks) -> int {
    if (mode == 0) {
      if (degree == 2) return bls_g2_wnaf_mul_dev(ctx, (const bls_g2*)d[0], (const bls_fr_repr*)d[1], (bls_g2*)o, cn, window, ks);
      return bls_g1_wnaf_mul_dev(ctx, (const bls_g1*)d[0], (const bls_fr_repr*)d[1], (bls_g1*)o, cn, window, ks);
    }
    if (degree == 2) k_pt_mul<Fp2, true, BLS_WNAF_K_G2><<<blocks_for((cn + BLS_WNAF_K_G2 - 1) / BLS_WNAF_K_G2, TPB), TPB, 0, ks>>>((const uint64_t*)d[0], (const uint64_t*)d[1], (uint64_t*)o, cn);
    else k_pt_mul<Fp, false, BLS_WNAF_K><<<blocks_for((cn + BLS_WNAF_K - 1) / BLS_WNAF_K, TPB), TPB, 0, ks>>>((const uint64_t*)d[0], (const uint64_t*)d[1], (uint64_t*)o, cn);
    LAUNCH_CHECK();
    return BLS_OK;
  }, true);
}
int bls_g1_wnaf_mul_batch(bls_ctx* ctx, const bls_g1* b, const bls_fr_repr* k, bls_g1* out, size_t n) { return wnaf_host(ctx, 1, b, k, out, n, 0, 0); }
int bls_g2_wnaf_mul_batch(bls_ctx* ctx, const bls_g2* b, const bls_fr_repr* k, bls_g2* out, size_t n) { return wnaf_host(ctx, 2, b, k, out, n, 0, 0); }
int bls_g1_wnaf_mul_window_batch(bls_ctx* ctx, const bls_g1* b, const bls_fr_repr* k, bls_g1* out, size_t n, int window) {
  if (window < 2 || window > BLS_MAX_WNAF_EXPLICIT_WINDOW) return BLS_ERR_INVALID_ARGUMENT;
  return wnaf_host(ctx, 1, b, k, out, n, window, 0);
}
int bls_g2_wnaf_mul_window_batch(bls_ctx* ctx, const bls_g2* b, const bls_fr_repr* k, bls_g2* out, size_t n, int window) {
  if (window < 2 || window > BLS_MAX_WNAF_EXPLICIT_WINDOW) return BLS_ERR_INVALID_ARGUMENT;
  return wnaf_host(ctx, 2, b, k, out, n, window, 0);
}
int bls_g1_mul_batch(bls_ctx* ctx, const bls_g1* b, const bls_fr_repr* k, bls_g1* out, size_t n) { return wnaf_host(ctx, 1, b, k, out, n, 0, 1); }
int bls_g2_mul_batch(bls_ctx* ctx, const bls_g2* b, const bls_fr_repr* k, bls_g2* out, size_t n) { return wnaf_host(ctx, 2, b, k, out, n, 0, 1); }

// Wnaf::new().base(g, num_scalars).scalar(k_i): table built on the device, then every scalar against it
static int wnaf_fixed_host(bls_ctx* ctx, int degree, const void* base, int window, const bls_fr_repr* k, void* out, size_t n, void* table_out) {
  if (!ctx || !base || window < 2 || window > BLS_MAX_WNAF_FIXED_WINDOW || (n && (!k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  size_t tsize = (size_t)1 << (window - 1);
  H2D(db, base, pb);
  DALLOC(dt, tsize * pb);
  if (degree == 2) TRY(bls_g2_wnaf_table_dev(ctx, (const bls_g2*)db.p, window, (bls_g2*)dt.p, nullptr));
  else TRY(bls_g1_wnaf_table_dev(ctx, (const bls_g1*)db.p, window, (bls_g1*)dt.p, nullptr));
  if (table_out) D2H(table_out, dt, tsize * pb);
  if (n) {
    H2D(dk, k, n * sizeof(*k));
    DALLOC(dout, n * pb);
    if (degree == 2) TRY(bls_g2_wnaf_fixed_base_dev(ctx, (const bls_g2*)dt.p, window, (const bls_fr_repr*)dk.p, (bls_g2*)dout.p, n, nullptr));
    else TRY(bls_g1_wnaf_fixed_base_dev(ctx, (const bls_g1*)dt.p, window, (const bls_fr_repr*)dk.p, (bls_g1*)dout.p, n, nullptr));
    D2H(out, dout, n * pb);
    SYNC();
    return BLS_OK;
  }
  SYNC();
  return BLS_OK;
}
int bls_g1_wnaf_fixed_base_batch(bls_ctx* ctx, const bls_g1* base, int window, const bls_fr_repr* k, bls_g1* out, size_t n) { return wnaf_fixed_host(ctx, 1, base, window, k, out, n, nullptr); }
int bls_g2_wnaf_fixed_base_batch(bls_ctx* ctx, const bls_g2* base, int window, const bls_fr_repr* k, bls_g2* out, size_t n) { return wnaf_fixed_host(ctx, 2, base, window, k, out, n, nullptr); }
int bls_g1_wnaf_table(bls_ctx* ctx, const bls_g1* base, int window, bls_g1* table) { return wnaf_fixed_host(ctx, 1, base, window, nullptr, nullptr, 0, table); }
int bls_g2_wnaf_table(bls_ctx* ctx, const bls_g2* base, int window, bls_g2* table) { return wnaf_fixed_host(ctx, 2, base, window, nullptr, nullptr, 0, table); }

static int codec_host(bls_ctx* ctx, int degree, bool decode, const void* in, int compressed, int checked, void* out, uint8_t* status, size_t n) {
  if (!ctx || (n && (!in || !out || (decode && !status)))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  const size_t eb = (size_t)(degree == 2 ? 96 : 48) * (compressed ? 1 : 2);
  if (decode) {
    H2D(din, in, n * eb);
    DALLOC(dout, n * ab);
    DALLOC(dst, n);
    if (degree == 2) k_decode<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint8_t*)din.p, compressed, checked, (uint64_t*)dout.p, (uint8_t*)dst.p, n);
    else k_decode<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint8_t*)din.p, compressed, checked, (uint64_t*)dout.p, (uint8_t*)dst.p, n);
    LAUNCH_CHECK();
    D2H(out, dout, n * ab);
    D2H(status, dst, n);
    SYNC();
  } else {
    H2D(din, in, n * ab);
    DALLOC(dout, n * eb);
    if (degree == 2) k_encode<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, compressed, (uint8_t*)dout.p, n);
    else k_encode<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, compressed, (uint8_t*)dout.p, n);
    LAUNCH_CHECK();
    D2H(out, dout, n * eb);
    SYNC();
  }
  return BLS_OK;
}
int bls_g1_decode_batch(bls_ctx* ctx, const uint8_t* bytes, int compressed, int checked, bls_g1_affine* out, uint8_t* status, size_t n) { return codec_host(ctx, 1, true, bytes, compressed, checked, out, status, n); }
int bls_g2_decode_batch(bls_ctx* ctx, const uint8_t* bytes, int compressed, int checked, bls_g2_affine* out, uint8_t* status, size_t n) { return codec_host(ctx, 2, true, bytes, compressed, checked, out, status, n); }
int bls_g1_encode_batch(bls_ctx* ctx, const bls_g1_affine* in, int compressed, uint8_t* bytes, size_t n) { return codec_host(ctx, 1, false, in, compressed, 0, bytes, nullptr, n); }
int bls_g2_encode_batch(bls_ctx* ctx, const bls_g2_affine* in, int compressed, uint8_t* bytes, size_t n) { return codec_host(ctx, 2, false, in, compressed, 0, bytes, nullptr, n); }

static int from_x_host(bls_ctx* ctx, int degree, const void* x, const uint8_t* greatest, void* out, uint8_t* is_some, size_t n) {
  if (!ctx || (n && (!x || !greatest || !out || !is_some))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t xb = degree == 2 ? sizeof(bls_fq2) : sizeof(bls_fq);
  const size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  H2D(dx, x, n * xb);
  H2D(dg, greatest, n);
  DALLOC(dout, n * ab);
  DALLOC(dok, n);
  if (degree == 2) k_point_from_x<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)dx.p, (const uint8_t*)dg.p, (uint64_t*)dout.p, (uint8_t*)dok.p, n);
  else k_point_from_x<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)dx.p, (const uint8_t*)dg.p, (uint64_t*)dout.p, (uint8_t*)dok.p, n);
  LAUNCH_CHECK();
  D2H(out, dout, n * ab);
  D2H(is_some, dok, n);
  SYNC();
  return BLS_OK;
}
int bls_g1_point_from_x_batch(bls_ctx* ctx, const bls_fq* x, const uint8_t* greatest, bls_g1_affine* out, uint8_t* is_some, size_t n) { return from_x_host(ctx, 1, x, greatest, out, is_some, n); }
int bls_g2_point_from_x_batch(bls_ctx* ctx, const bls_fq2* x, const uint8_t* greatest, bls_g2_affine* out, uint8_t* is_some, size_t n) { return from_x_host(ctx, 2, x, greatest, out, is_some, n); }

static int cofactor_host(bls_ctx* ctx, int degree, const void* in, void* out, size_t n) {
  if (!ctx || (n && (!in || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  H2D(din, in, n * ab);
  DALLOC(dout, n * pb);
  if (degree == 2) k_scale_by_cofactor<Fp2, true><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, (uint64_t*)dout.p, n);
  else k_scale_by_cofactor<Fp, false><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, (uint64_t*)dout.p, n);
  LAUNCH_CHECK();
  D2H(out, dout, n * pb);
  SYNC();
  return BLS_OK;
}
int bls_g1_scale_by_cofactor_batch(bls_ctx* ctx, const bls_g1_affine* in, bls_g1* out, size_t n) { return cofactor_host(ctx, 1, in, out, n); }
int bls_g2_scale_by_cofactor_batch(bls_ctx* ctx, const bls_g2_affine* in, bls_g2* out, size_t n) { return cofactor_host(ctx, 2, in, out, n); }

static int affine_mul_host(bls_ctx* ctx, int degree, const void* a, const bls_fr_repr* k, void* out, size_t n) {
  if (!ctx || (n && (!a || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  H2D(da, a, n * ab);
  H2D(dk, k, n * sizeof(*k));
  DALLOC(dout, n * pb);
  if (degree == 2) k_affine_mul<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)da.p, (const uint64_t*)dk.p, (uint64_t*)dout.p, n);
  else k_affine_mul<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)da.p, (const uint64_t*)dk.p, (uint64_t*)dout.p, n);
  LAUNCH_CHECK();
  D2H(out, dout, n * pb);
  SYNC();
  return BLS_OK;
}
int bls_g1_affine_mul_batch(bls_ctx* ctx, const bls_g1_affine* a, const bls_fr_repr* k, bls_g1* out, size_t n) { return affine_mul_host(ctx, 1, a, k, out, n); }
int bls_g2_affine_mul_batch(bls_ctx* ctx, const bls_g2_affine* a, const bls_fr_repr* k, bls_g2* out, size_t n) { return affine_mul_host(ctx, 2, a, k, out, n); }

// Chunks are normalised independently (Montgomery's trick per chunk): the outputs are canonical, so the partition does not show
static int bn_host(bls_ctx* ctx, int degree, void* inout, size_t n) {
  if (!ctx || (n && !inout)) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const size_t csz = n < PIPE_CHUNK_POINTS ? n : PIPE_CHUNK_POINTS;
  DALLOC(dscr, bls_batch_normalization_scratch_bytes(ctx, degree, csz));
  const PipeIn in[1] = {{inout, pb}};
  return run_pipelined(ctx, n, PIPE_CHUNK_POINTS, in, 1, inout, pb, [&](const void* const* d, void* o, size_t cn, cudaStream_t ks) -> int {
    CK(cudaMemcpyAsync(o, d[0], cn * pb, cudaMemcpyDeviceToDevice, ks));
    if (degree == 2) return bls_g2_batch_normalization_dev(ctx, (bls_g2*)o, cn, dscr.p, ks);
    return bls_g1_batch_normalization_dev(ctx, (bls_g1*)o, cn, dscr.p, ks);
  });
}
int bls_g1_batch_normalization(bls_ctx* ctx, bls_g1* inout, size_t n) { return bn_host(ctx, 1, inout, n); }
int bls_g2_batch_normalization(bls_ctx* ctx, bls_g2* inout, size_t n) { return bn_host(ctx, 2, inout, n); }

static int into_affine_host(bls_ctx* ctx, int degree, const void* in, void* out, size_t n) {
  if (!ctx || (n && (!in || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  H2D(din, in, n * pb);
  DALLOC(dout, n * ab);
  if (degree == 2) k_into_affine<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, (uint64_t*)dout.p, n);
  else k_into_affine<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>((const uint64_t*)din.p, (uint64_t*)dout.p, n);
  LAUNCH_CHECK();
  D2H(out, dout, n * ab);
  SYNC();
  return BLS_OK;
}
int bls_g1_into_affine_batch(bls_ctx* ctx, const bls_g1* in, bls_g1_affine* out, size_t n) { return into_affine_host(ctx, 1, in, out, n); }
int bls_g2_into_affine_batch(bls_ctx* ctx, const bls_g2* in, bls_g2_affine* out, size_t n) { return into_affine_host(ctx, 2, in, out, n); }

static int pt_op_host(bls_ctx* ctx, int degree, int op, const void* a, const void* b, void* out, size_t n) {
  bool needs_b = op == BLS_PT_ADD || op == BLS_PT_SUB || op == BLS_PT_ADD_MIXED;
  bool known = needs_b || op == BLS_PT_DOUBLE || op == BLS_PT_NEGATE;
  if (!ctx || !known || (n && (!a || !out || (needs_b && !b)))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  H2D(da, a, n * pb);
  H2D(db, needs_b ? b : nullptr, needs_b ? n * (op == BLS_PT_ADD_MIXED ? ab : pb) : 1);
  DALLOC(dout, n * pb);
  if (degree == 2) k_pt_op<Fp2><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, (const uint64_t*)db.p, (uint64_t*)dout.p, n);
  else k_pt_op<Fp><<<blocks_for(n, TPB), TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, (const uint64_t*)db.p, (uint64_t*)dout.p, n);
  LAUNCH_CHECK();
  D2H(out, dout, n * pb);
  SYNC();
  return BLS_OK;
}
int bls_g1_op_batch(bls_ctx* ctx, int op, const bls_g1* a, const void* b, bls_g1* out, size_t n) { return pt_op_host(ctx, 1, op, a, b, out, n); }
int bls_g2_op_batch(bls_ctx* ctx, int op, const bls_g2* a, const void* b, bls_g2* out, size_t n) { return pt_op_host(ctx, 2, op, a, b, out, n); }

int bls_field_op_batch(bls_ctx* ctx, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n) {
  if (!ctx || (n && (!a || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (degree != 1 && degree != 2 && degree != 6 && degree != 12) return BLS_ERR_INVALID_ARGUMENT;
  // which ops exist at which degree (mirrors the switch statements of the kernels)
  bool valid = false, binary = false;
  switch (op) {
    case BLS_OP_ADD: case BLS_OP_SUB: valid = degree != 12; binary = true; break;
    case BLS_OP_MUL: valid = true; binary = true; break;
    case BLS_OP_SQR: case BLS_OP_INV: valid = true; break;
    case BLS_OP_NEG: valid = degree != 12; break;
    case BLS_OP_DBL: valid = degree <= 2; break;
    case BLS_OP_FROM_REPR: case BLS_OP_INTO_REPR: valid = degree == 1; break;
    case BLS_OP_SQRT: valid = degree <= 2; break;
    case BLS_OP_MUL_NONRES: valid = degree == 2 || degree == 6; break;
    case BLS_OP_FROB1: valid = degree >= 2; break;
    case BLS_OP_FROB2: case BLS_OP_FROB3: valid = degree >= 6; break;
    case BLS_OP_CONJ: valid = degree == 12; break;
    case BLS_OP_MUL_BY_014: valid = degree == 12; binary = true; break;
    case BLS_OP_MUL_BY_01: case BLS_OP_MUL_BY_1: valid = degree == 6; binary = true; break;
  }
  if (!valid || (binary && n && !b)) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t eb = (size_t)degree * sizeof(bls_fq);
  H2D(da, a, n * eb);
  H2D(db, binary ? b : nullptr, binary ? n * eb : 1);
  DALLOC(dout, n * eb);
  DALLOC(dok, n);
  const uint64_t* pb = binary ? (const uint64_t*)db.p : nullptr;
  unsigned g = blocks_for(n, TPB);
  switch (degree) {
    case 1: k_fq_op<<<g, TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, pb, (uint64_t*)dout.p, (uint8_t*)dok.p, n); break;
    case 2: k_fq2_op<<<g, TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, pb, (uint64_t*)dout.p, (uint8_t*)dok.p, n); break;
    case 6: k_fq6_op<<<g, TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, pb, (uint64_t*)dout.p, (uint8_t*)dok.p, n); break;
    case 12: k_fq12_op<<<g, TPB, 0, ctx->stream>>>(op, (const uint64_t*)da.p, pb, (uint64_t*)dout.p, (uint8_t*)dok.p, n); break;
  }
  LAUNCH_CHECK();
  D2H(out, dout, n * eb);
  if (ok) D2H(ok, dok, n);
  SYNC();
  return BLS_OK;
}

int bls_pair_field_op_batch(bls_ctx* ctx, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n) {
  if (!ctx || (degree != 2 && degree != 6 && degree != 12) || (n && (!a || !out))) return BLS_ERR_INVALID_ARGUMENT;
  bool valid = false, binary = false;
  switch (op) {
    case BLS_OP_ADD: case BLS_OP_SUB: valid = degree != 12; binary = true; break;
    case BLS_OP_MUL: valid = true; binary = true; break;
    case BLS_OP_SQR: case BLS_OP_INV: valid = true; break;
    case BLS_OP_NEG: valid = degree != 12; break;
    case BLS_OP_DBL: valid = degree == 2; break;
    case BLS_OP_MUL_NONRES: valid = degree != 12; break;
    case BLS_OP_FROB1: valid = true; break;
    case BLS_OP_FROB2: case BLS_OP_FROB3: valid = degree >= 6; break;
    case BLS_OP_CONJ: case BLS_OP_CYCLOTOMIC_SQR: valid = degree == 12; break;
    case BLS_OP_MUL_BY_014: case BLS_OP_MUL_BY_LINE_PAIR: valid = degree == 12; binary = true; break;
    case BLS_OP_MUL_BY_01: case BLS_OP_MUL_BY_1: valid = degree == 6; binary = true; break;
  }
  if (!valid || (binary && n && !b)) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  size_t eb = (size_t)degree * sizeof(bls_fq);
  H2D(da, a, n * eb);
  H2D(db, binary ? b : nullptr, binary ? n * eb : 1);
  DALLOC(dout, n * eb);
  DALLOC(dok, n);
  TRY(bls_pair_field_op_dev(ctx, degree, op, da.p, binary ? db.p : nullptr, dout.p, (uint8_t*)dok.p, n, nullptr));
  D2H(out, dout, n * eb);
  if (ok) D2H(ok, dok, n);
  SYNC();
  return BLS_OK;
}

// bls_fr_op_batch / _dev argument rules; *binary: the op reads b
static bool fr_op_args_ok(bls_ctx* ctx, int op, const void* a, const void* b, const void* out, size_t n, bool* binary) {
  *binary = op == BLS_OP_ADD || op == BLS_OP_SUB || op == BLS_OP_MUL;
  const bool unary = op == BLS_OP_SQR || op == BLS_OP_NEG || op == BLS_OP_DBL || op == BLS_OP_INV || op == BLS_OP_FROM_REPR || op == BLS_OP_INTO_REPR;
  return ctx && !(n && (!a || !out)) && (*binary || unary) && !(*binary && n && !b);
}

int bls_fr_op_dev(bls_ctx* ctx, int op, const bls_fr* a, const bls_fr* b, bls_fr* out, uint8_t* ok, size_t n, void* stream) {
  bool binary;
  if (!fr_op_args_ok(ctx, op, a, b, out, n, &binary)) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_fr_op<<<blocks_for(n, TPB), TPB, 0, pick(ctx, stream)>>>(op, (const uint64_t*)a, binary ? (const uint64_t*)b : nullptr, (uint64_t*)out, ok, n);
  LAUNCH_CHECK();
  return BLS_OK;
}

int bls_fr_op_batch(bls_ctx* ctx, int op, const bls_fr* a, const bls_fr* b, bls_fr* out, uint8_t* ok, size_t n) {
  bool binary;
  if (!fr_op_args_ok(ctx, op, a, b, out, n, &binary)) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  H2D(da, a, n * sizeof(*a));
  H2D(db, binary ? b : nullptr, binary ? n * sizeof(*b) : 1);
  DALLOC(dout, n * sizeof(*out));
  DALLOC(dok, n);
  TRY(bls_fr_op_dev(ctx, op, (const bls_fr*)da.p, binary ? (const bls_fr*)db.p : nullptr, (bls_fr*)dout.p, (uint8_t*)dok.p, n, ctx->stream));
  D2H(out, dout, n * sizeof(*out));
  if (ok) D2H(ok, dok, n);
  SYNC();
  return BLS_OK;
}

int bls_imad_peak(bls_ctx* ctx, int variant, int iters, double* macs_per_s, double* ms_out) {
  if (!ctx || !macs_per_s || iters <= 0 || variant < 0 || variant > 4) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  DALLOC(sink, 8);
  const int threads = 256;
  const unsigned blocks = (unsigned)ctx->sm_count * 8;   // 2048 threads per SM: full occupancy
  struct Events {   // destroyed on every exit path, CK failures included
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~Events() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
  } ev;
  CK(cudaEventCreate(&ev.e0));
  CK(cudaEventCreate(&ev.e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {   // rep 0 is the warm-up
    CK(cudaEventRecord(ev.e0, ctx->stream));
    if (variant == 0) k_imad_wide_peak<<<blocks, threads, 0, ctx->stream>>>(12345u, iters, (uint64_t*)sink.p);
    else if (variant == 1) k_fpmul_peak<<<blocks, threads, 0, ctx->stream>>>(12345u, iters, (uint64_t*)sink.p);
    else if (variant == 3) k_carry_row_peak<<<blocks, threads, 0, ctx->stream>>>(12345u, iters, (uint64_t*)sink.p);
    else if (variant == 4) k_fpsqr_peak<<<blocks, threads, 0, ctx->stream>>>(12345u, iters, (uint64_t*)sink.p);
    else k_imad32_peak<<<blocks, threads, 0, ctx->stream>>>(12345u, iters, (uint64_t*)sink.p);
    LAUNCH_CHECK();
    CK(cudaEventRecord(ev.e1, ctx->stream));
    CK(cudaEventSynchronize(ev.e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ev.e0, ev.e1));
    if (rep > 0 && ms < best) best = ms;
  }
  double per_thread = variant == 1 ? 2.0 * 300.0 * iters : variant == 4 ? 2.0 * 234.0 * iters : variant == 3 ? 8.0 * 24.0 * iters : (double)PEAK_CHAINS * PEAK_UNROLL * iters;
  double total = per_thread * threads * blocks;
  *macs_per_s = total / (best * 1e-3);
  if (ms_out) *ms_out = best;
  return BLS_OK;
}

}  // extern "C"
