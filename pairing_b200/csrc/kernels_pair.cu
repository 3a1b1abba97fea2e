// kernels_pair.cu -- the pairing engine on LANE PAIRS (pair_tower.cuh): Miller loops, final exponentiation, the fused
// pairing kernel, G2Prepared, GT powers, and their device-pointer entry points (the multi-pairing Miller loop: kernels_mm.cu).
// Its own translation unit: see abi_common.cuh.

#include "pair_io.cuh"

template <bool FINAL_EXP>
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_miller(const uint64_t* p, const uint64_t* q, uint64_t* out, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  const uint64_t* pi = p + G1A_W * i;
  const uint64_t* qi = q + G2A_W * i;
  const bool live = pi[12] == 0 && qi[24] == 0;
  Fp px = ld_fp(pi), py = ld_fp(pi + 6);
  P2 qx = ld_p2(qi), qy = ld_p2(qi + 12);
  P12 f;
  p_miller_loop_single(f, px, py, qx, qy);
  if (!live) p12_one(f);                       // mod.rs:49-54: skipped pair, f stays one
  if (FINAL_EXP) {
    P12 g;
    p_final_exponentiation(g, f);
    if (active) st_p12(out + FQ12_W * i, g);
  } else {
    if (active) st_p12(out + FQ12_W * i, f);
  }
}

__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_g2_prepare(const uint64_t* q, uint64_t* out, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  const uint64_t* qi = q + G2A_W * i;
  uint64_t* o = out + (size_t)G2P_W * i;
  const bool inf = qi[24] != 0;      // infinity: empty coefficient list + flag (mod.rs:169-174); the slots are zero-filled
  const P2 qx = ld_p2(qi), qy = ld_p2(qi + 12);
  PJac r; r.x = qx; r.y = qy; r.z = p2_one();
  PCoeffs c;
  const P2 zero = p2_zero();
  int idx = 0;
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= -1; b--) {
    pg2_doubling_step(r, c);
    if (inf) { c.c0 = zero; c.c1 = zero; c.c2 = zero; }
    if (active) st_pcoeffs(o + 36 * idx, c);
    idx++;
    if (b >= 0 && ((BLS_LOOP_BITS >> b) & 1ull)) {
      pg2_addition_step(r, qx, qy, c);
      if (inf) { c.c0 = zero; c.c1 = zero; c.c2 = zero; }
      if (active) st_pcoeffs(o + 36 * idx, c);
      idx++;
    }
  }
  if (active && pair_c() == 0) o[G2P_W - 1] = inf ? 1ull : 0ull;
}

// the reference's literal miller_loop (mod.rs:40-102) for n independent pairs, coefficients read from memory
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_miller_prepared(const uint64_t* p, const uint64_t* qp, uint64_t* out, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  const uint64_t* pi = p + G1A_W * i;
  const uint64_t* qi = qp + (size_t)G2P_W * i;
  const bool live = pi[12] == 0 && qi[G2P_W - 1] == 0;
  const Fp px = ld_fp(pi), py = ld_fp(pi + 6);
  P12 f;
  p12_one(f);
  PCoeffs c;
  int idx = 0;
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= -1; b--) {
    ld_pcoeffs(c, qi + 36 * idx); idx++;
    p_ell(f, c, px, py);
    if (b >= 0 && ((BLS_LOOP_BITS >> b) & 1ull)) {
      ld_pcoeffs(c, qi + 36 * idx); idx++;
      p_ell(f, c, px, py);
    }
    if (b >= 0) p12_sqr(f, f);
  }
  p12_conjugate(f);
  if (!live) p12_one(f);
  if (active) st_p12(out + FQ12_W * i, f);
}

// n Miller loops / pairings e(P_i, Q) against ONE prepared G2 point -- the shape G2Prepared exists for in the reference
// (verification against a fixed key or generator: `prepare` once, `miller_loop(&[(&p_i, &q)])` many times).  The 19 584
// bytes of line coefficients are staged ONCE per block in shared memory by a TMA bulk copy (cp.async.bulk, completion on
// an mbarrier); every lane pair then reads them as shared-memory broadcasts and does only `ell` and the squarings
// (5156 M per Miller loop instead of 6916 M with the G2 steps).
template <bool FINAL_EXP>
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_miller_shared_q(const uint64_t* p, const uint64_t* qp, uint64_t* out, size_t n) {
  __shared__ __align__(128) uint64_t s_coeffs[68 * 36];
  __shared__ __align__(8) uint64_t s_bar;
  const uint32_t bar = smem_u32(&s_bar);
  const uint32_t bytes = 68 * 36 * 8;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_coeffs)), "l"(qp), "r"(bytes), "r"(bar) : "memory");
  }
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  const uint64_t* pi = p + G1A_W * i;
  const bool live = pi[12] == 0 && qp[G2P_W - 1] == 0;
  const Fp px = ld_fp(pi), py = ld_fp(pi + 6);
  mbar_wait_phase0(bar);                       // the bulk copy has landed
  P12 f;
  p12_one(f);
  PCoeffs c;
  int idx = 0;
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= -1; b--) {
    const uint64_t* ci = s_coeffs + 36 * idx; idx++;
    c.c0 = ld_p2_smem(ci); c.c1 = ld_p2_smem(ci + 12); c.c2 = ld_p2_smem(ci + 24);
    p_ell(f, c, px, py);
    if (b >= 0 && ((BLS_LOOP_BITS >> b) & 1ull)) {
      const uint64_t* cj = s_coeffs + 36 * idx; idx++;
      c.c0 = ld_p2_smem(cj); c.c1 = ld_p2_smem(cj + 12); c.c2 = ld_p2_smem(cj + 24);
      p_ell(f, c, px, py);
    }
    if (b >= 0) p12_sqr(f, f);
  }
  p12_conjugate(f);
  if (!live) p12_one(f);
  if (FINAL_EXP) {
    P12 g;
    p_final_exponentiation(g, f);
    if (active) st_p12(out + FQ12_W * i, g);
  } else {
    if (active) st_p12(out + FQ12_W * i, f);
  }
}

__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_final_exp(const uint64_t* in, uint64_t* out, uint8_t* is_some, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  P12 f, g;
  ld_p12(f, in + FQ12_W * i);
  bool ok = p_final_exponentiation(g, f);
  if (active) {
    st_p12(out + FQ12_W * i, g);
    if (is_some && pair_c() == 0) is_some[i] = ok;
  }
}

// Field::pow on Fq12 with an FrRepr exponent (lib.rs:306-324; GT exponentiation, tests/engine.rs:121).  The reference
// is MSB-first square-and-multiply; the value of a power does not depend on the addition chain, so this is a 4-bit
// fixed window: 252 squarings + 64 table products, and -- the exponent differing per lane pair while every lane has to
// reach every shuffle -- completely uniform control flow (a zero window multiplies by table[0] = one).
// The operand of Field::pow may be any Fq12 element, but what callers raise to powers are GT elements (pairing values),
// which lie in the cyclotomic subgroup a^(q^4 - q^2 + 1) = 1.  One Frobenius test per operand -- a^(q^4) a == a^(q^2),
// about 1 % of the work -- tells: when it holds for every lane pair of the WARP, the 252 squarings are Granger-Scott
// cyclotomic squarings (6 Fq2 products instead of 12, the same value there); otherwise the warp squares generically.
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_fq12_pow(const uint64_t* in, const uint64_t* k, uint64_t* out, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  P12 tbl[16];
  p12_one(tbl[0]);
  ld_p12(tbl[1], in + FQ12_W * i);
  bool cyclotomic;
  {
    P12 f4, f2;
    p12_frobenius(f4, tbl[1], 4);
    p12_frobenius(f2, tbl[1], 2);
    p12_mul(f4, f4, tbl[1]);
    cyclotomic = __all_sync(0xffffffffu, p12_eq(f4, f2));
  }
#pragma unroll 1
  for (int e = 2; e < 16; e++) {
    if (cyclotomic && !(e & 1)) p12_cyclotomic_sqr(tbl[e], tbl[e >> 1]);      // even entries by a 6-product squaring instead of an 18-product multiplication
    else p12_mul(tbl[e], tbl[e - 1], tbl[1]);
  }
  const Scalar s = ld_scalar(k + 4 * i);
  P12 res = tbl[(s.v[7] >> 28) & 0xf];
#pragma unroll 1
  for (int w = 62; w >= 0; w--) {
    if (cyclotomic) { p12_cyclotomic_sqr(res, res); p12_cyclotomic_sqr(res, res); p12_cyclotomic_sqr(res, res); p12_cyclotomic_sqr(res, res); }
    else { p12_sqr(res, res); p12_sqr(res, res); p12_sqr(res, res); p12_sqr(res, res); }
    const uint32_t nib = (s.v[w >> 3] >> ((w & 7) * 4)) & 0xf;
    p12_mul(res, res, tbl[nib]);
  }
  if (active) st_p12(out + FQ12_W * i, res);
}

// Field-tower operations ON LANE PAIRS (pair_tower.cuh -- the code the pairing kernels run), element-wise, for parity
// tests on edge operands: the thread-per-element tower behind bls_field_op_batch is a different implementation.
// Operands may be any representative in [0, 2q] (the relaxed range of fp.cuh); results are stored canonical.
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_pair_field_op(int degree, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint8_t* ok, size_t n) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = t >> 1;
  const bool active = i < n;
  if (!active) i = n - 1;
  bool good = true;
  if (degree == 2) {
    const P2 x = ld_p2(a + 12 * i), y = b ? ld_p2(b + 12 * i) : p2_zero();
    P2 r = p2_zero();
    switch (op) {
      case BLS_OP_ADD: r = p2_add(x, y); break;
      case BLS_OP_SUB: r = p2_sub(x, y); break;
      case BLS_OP_MUL: r = p2_mul(x, y); break;
      case BLS_OP_SQR: r = p2_sqr(x); break;
      case BLS_OP_NEG: r = p2_neg(x); break;
      case BLS_OP_DBL: r = p2_dbl(x); break;
      case BLS_OP_INV: good = p2_inv(r, x); if (!good) r = p2_zero(); break;
      case BLS_OP_MUL_NONRES: r = p2_mul_by_nonresidue(x); break;
      case BLS_OP_FROB1: r = p2_frobenius(x, 1); break;
    }
    if (active) st_p2(out + 12 * i, r);
  } else if (degree == 6) {
    P6 x, y, r;
    x.c0 = ld_p2(a + 36 * i); x.c1 = ld_p2(a + 36 * i + 12); x.c2 = ld_p2(a + 36 * i + 24);
    if (b) { y.c0 = ld_p2(b + 36 * i); y.c1 = ld_p2(b + 36 * i + 12); y.c2 = ld_p2(b + 36 * i + 24); } else p6_zero(y);
    p6_zero(r);
    switch (op) {
      case BLS_OP_ADD: p6_add(r, x, y); break;
      case BLS_OP_SUB: p6_sub(r, x, y); break;
      case BLS_OP_MUL: p6_mul(r, x, y); break;
      case BLS_OP_SQR: p6_sqr(r, x); break;
      case BLS_OP_NEG: p6_neg(r, x); break;
      case BLS_OP_INV: good = p6_inv(r, x); if (!good) p6_zero(r); break;
      case BLS_OP_MUL_NONRES: p6_mul_by_nonresidue(r, x); break;
      case BLS_OP_FROB1: p6_frobenius(r, x, 1); break;
      case BLS_OP_FROB2: p6_frobenius(r, x, 2); break;
      case BLS_OP_FROB3: p6_frobenius(r, x, 3); break;
      case BLS_OP_MUL_BY_01: p6_mul_by_01(r, x, y.c0, y.c1); break;
      case BLS_OP_MUL_BY_1: p6_mul_by_1(r, x, y.c1); break;
    }
    if (active) { st_p2(out + 36 * i, r.c0); st_p2(out + 36 * i + 12, r.c1); st_p2(out + 36 * i + 24, r.c2); }
  } else {
    P12 x, y, r;
    ld_p12(x, a + FQ12_W * i);
    if (b) ld_p12(y, b + FQ12_W * i); else p12_one(y);
    p6_zero(r.c0); p6_zero(r.c1);
    switch (op) {
      case BLS_OP_MUL: p12_mul(r, x, y); break;
      case BLS_OP_SQR: p12_sqr(r, x); break;
      case BLS_OP_CYCLOTOMIC_SQR: p12_cyclotomic_sqr(r, x); break;
      case BLS_OP_INV: good = p12_inv(r, x); if (!good) { p6_zero(r.c0); p6_zero(r.c1); } break;
      case BLS_OP_CONJ: r = x; p12_conjugate(r); break;
      case BLS_OP_FROB1: p12_frobenius(r, x, 1); break;
      case BLS_OP_FROB2: p12_frobenius(r, x, 2); break;
      case BLS_OP_FROB3: p12_frobenius(r, x, 3); break;
      case BLS_OP_MUL_BY_014: r = x; p12_mul_by_014(r, y.c0.c0, y.c0.c1, y.c1.c1); break;
      case BLS_OP_MUL_BY_LINE_PAIR: {      // b packs two lines: (l.c0, l.c1, l.c4, m.c0, m.c1, m.c4)
        r = x;
        p12_mul_by_line_pair(r, PLine{y.c0.c0, y.c0.c1, y.c0.c2}, PLine{y.c1.c0, y.c1.c1, y.c1.c2});
        break;
      }
    }
    if (active) st_p12(out + FQ12_W * i, r);
  }
  if (active && ok && pair_c() == 0) ok[i] = good;
}

extern "C" {

int bls_pair_field_op_dev(bls_ctx* ctx, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n, void* stream) {
  if (!ctx || (degree != 2 && degree != 6 && degree != 12) || (n && (!a || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_pair_field_op<<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>(degree, op, (const uint64_t*)a, (const uint64_t*)b, (uint64_t*)out, ok, n);
  LAUNCH_CHECK();
  return BLS_OK;
}

int bls_g2_prepare_dev(bls_ctx* ctx, const bls_g2_affine* q, bls_g2_prepared* out, size_t n, void* stream) {
  if (!ctx || (n && (!q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_pair_g2_prepare<<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)q, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_miller_loop_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, void* stream) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  if (n <= ctx->wide_pairing_max) return bls_internal_wide_miller(ctx, p, q, out, n, pick(ctx, stream));
  k_pair_miller<false><<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)p, (const uint64_t*)q, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_miller_loop_prepared_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q, bls_fq12* out, size_t n, void* stream) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_pair_miller_prepared<<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)p, (const uint64_t*)q, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_final_exponentiation_dev(bls_ctx* ctx, const bls_fq12* in, bls_fq12* out, uint8_t* is_some, size_t n, void* stream) {
  if (!ctx || (n && (!in || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  if (n <= ctx->wide_final_exp_max) return bls_internal_wide_final_exp(ctx, in, out, is_some, n, pick(ctx, stream));
  k_pair_final_exp<<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)in, (uint64_t*)out, is_some, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_pairing_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, void* stream) {
  if (!ctx || (n && (!p || !q || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  if (n <= ctx->wide_pairing_max) return bls_internal_wide_pairing(ctx, p, q, out, n, pick(ctx, stream));
  k_pair_miller<true><<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)p, (const uint64_t*)q, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}

int bls_miller_loop_shared_q_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n, int final_exp, void* stream) {
  if (!ctx || !q1 || (n && (!p || !out)) || ((uintptr_t)q1 & 15)) return BLS_ERR_INVALID_ARGUMENT;   // the bulk copy needs 16-byte alignment
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  if (final_exp) k_pair_miller_shared_q<true><<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)p, (const uint64_t*)q1, (uint64_t*)out, n);
  else k_pair_miller_shared_q<false><<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)p, (const uint64_t*)q1, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_fq12_pow_dev(bls_ctx* ctx, const bls_fq12* a, const bls_fr_repr* k, bls_fq12* out, size_t n, void* stream) {
  if (!ctx || (n && (!a || !k || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (!n) return BLS_OK;
  USE_DEVICE(ctx);
  k_pair_fq12_pow<<<blocks_for(2 * n, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, pick(ctx, stream)>>>((const uint64_t*)a, (const uint64_t*)k, (uint64_t*)out, n);
  LAUNCH_CHECK();
  return BLS_OK;
}
int bls_fq12_product_tail_dev(bls_ctx* ctx, const bls_fq12* in, size_t n, bls_fq12* out1, int final_exp, uint8_t* is_some, void* stream) {
  if (!ctx || !out1 || (n && !in)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  return bls_internal_product_tail(ctx, in, n, out1, final_exp, is_some, pick(ctx, stream));
}

}  // extern "C"
