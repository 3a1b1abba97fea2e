// kernels_groth16_verify.cu -- bellman's groth16::{prepare_verifying_key, verify_proof} for m proofs of one circuit, and the
// randomized batch check (bls_groth16_prepare_verifying_key, bls_groth16_verify_*, bls_groth16_verify_rlc_*).  Its own
// translation unit (see abi_common.cuh): the multiexps, the pairing product, the G2 preparation and the GT power are the
// other units' entry points, called through the C ABI, so no existing kernel is recompiled.
//
// Per-proof pipeline, all on the call's stream:
//   1. k_g16v_scalars: one thread per (proof, scalar): [into_repr(1), into_repr(x_j1), ...], the msm scalars of proof j.
//   2. bls_g1_msm_batch_dev with the shared bases ic: acc_j = ic_0 + sum_i x_ji ic_i, normalised (z = one, or z = 0 for
//      infinity), so the next kernel reads it as an affine point without an into_affine pass.
//   3. k_groth16_verify: one lane pair per proof (pair_tower.cuh), the three Miller loops of verify_proof fused into one:
//      the coefficients of -gamma and -delta are staged once per block in shared memory by two TMA bulk copies; per step of
//      the loop schedule the lane pair takes the doubling / addition step on B_j on the fly, multiplies f by l_A l_gamma
//      (one line-pair product) and by l_delta, and squares f once per bit for all three pairs.  Then the conjugation, the
//      final exponentiation, the comparison with alpha_g1_beta_g2 and one byte per proof.
//
// Randomized check: k_g16v_rlc_terms (rho_j A_j by curve.cuh's double-and-add, one thread per proof; B_j and C_j gathered),
// k_g16v_rlc_sums (the Fr column sums s_i), two bls_g1_msm_dev calls (sum_i s_i ic_i and sum_j rho_j C_j), k_g16v_rlc_pairs
// (the two sums in affine form next to -gamma and -delta), bls_pairing_product_dev over m + 2 pairs, bls_fq12_pow_dev for
// alpha_g1_beta_g2^(sum rho) and k_g16v_rlc_compare.
#include <stddef.h>

#include <vector>

#include "curve_io.cuh"
#include "fr.cuh"
#include "pair_io.cuh"

#define G16V_TPB 128
#define G16V_TAIL_TPB 32                  /* k_g16v_rlc_terms runs a single-thread chain per proof: spread them over the SMs */
#define G16V_SUM_TPB 256
#define G16V_MAX_M ((size_t)1 << 16)      /* per-proof path: bls_g1_msm_batch_dev's limits */
#define G16V_MAX_MN ((size_t)1 << 26)
#define G16V_RLC_MAX ((size_t)1 << 26)    /* randomized check: bls_g1_msm_dev's limit, for m and for num_inputs + 1 */

// bls_groth16_pvk in u64 words
#define PVK_GAMMA 0
#define PVK_DELTA (G2P_W + 1)
#define PVK_AB (2 * (G2P_W + 1))
#define PVK_GAMMA_AFF (PVK_AB + FQ12_W)
#define PVK_DELTA_AFF (PVK_GAMMA_AFF + G2A_W)
#define PVK_W (PVK_DELTA_AFF + G2A_W)
#define PROOF_W (2 * G1A_W + G2A_W)
#define G16V_COEFF_BYTES (68 * 36 * 8)
static_assert(sizeof(bls_groth16_pvk) == PVK_W * 8, "bls_groth16_pvk layout");
static_assert(offsetof(bls_groth16_pvk, neg_delta_g2) == PVK_DELTA * 8 && PVK_DELTA * 8 % 16 == 0, "neg_delta_g2 must be 16-byte aligned");
static_assert(offsetof(bls_groth16_pvk, alpha_g1_beta_g2) == PVK_AB * 8, "bls_groth16_pvk layout");
static_assert(offsetof(bls_groth16_pvk, neg_delta_g2_affine) == PVK_DELTA_AFF * 8, "bls_groth16_pvk layout");
static_assert(sizeof(bls_groth16_proof) == PROOF_W * 8, "bls_groth16_proof layout");

// ---- Fr scalars -----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ Fr g16v_ld_fr(const uint64_t* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void g16v_st_fr(uint64_t* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
// the Montgomery product with the integer 1: into_repr() of a Montgomery value; of a plain value x, x R^-1
__device__ __forceinline__ Fr g16v_int_one() {
  Fr one = fr_zero();
  one.v[0] = 1;
  return one;
}

// t = j (ni + 1) + i: scalar i of proof j, 1 for i = 0 (bellman's leading one), else into_repr(inputs[j ni + i - 1])
__global__ void __launch_bounds__(G16V_TPB) k_g16v_scalars(const uint64_t* inputs, size_t ni, size_t m, uint64_t* k) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = ni + 1;
  if (t >= m * n) return;
  const size_t j = t / n, i = t - j * n;
  const Fr x = i == 0 ? g16v_int_one() : fr_mul(g16v_ld_fr(inputs + 4 * (j * ni + i - 1)), g16v_int_one());
  g16v_st_fr(k + 4 * t, x);
}

// ---- the fused verification kernel ------------------------------------------------------------------------------------------
// line value of a pair with coefficients c at the G1 point at p; a dead pair's line is the sparse element one
__device__ __forceinline__ PLine g16v_line(PCoeffs c, const uint64_t* p, bool dead) {
  pcoeffs_set_one_if(dead, c);
  return p_line(c, ld_fp(p), ld_fp(p + 6));
}
__device__ __forceinline__ PCoeffs g16v_smem_coeffs(const uint64_t* s) {
  PCoeffs c;
  c.c0 = ld_p2_smem(s); c.c1 = ld_p2_smem(s + 12); c.c2 = ld_p2_smem(s + 24);
  return c;
}

// Lane pair i verifies proof i: final_exponentiation(miller_loop([(A, B), (acc, -gamma), (C, -delta)])) == alpha_g1_beta_g2.
// The G1 points are read from global memory at each line instead of being kept live (-Xptxas -v: DESIGN.md).
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_groth16_verify(const uint64_t* pvk, const uint64_t* proofs, const uint64_t* acc,
                                                                               size_t m, uint8_t* ok) {
  __shared__ __align__(128) uint64_t s_coeffs[2][68 * 36];
  __shared__ __align__(8) uint64_t s_bar;
  const uint32_t bar = smem_u32(&s_bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2 * G16V_COEFF_BYTES) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_coeffs[0])), "l"(pvk + PVK_GAMMA), "r"(G16V_COEFF_BYTES), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_coeffs[1])), "l"(pvk + PVK_DELTA), "r"(G16V_COEFF_BYTES), "r"(bar) : "memory");
  }
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
  const bool active = i < m;
  if (!active) i = m - 1;
  const uint64_t* a = proofs + PROOF_W * i;
  const uint64_t* b = a + G1A_W;
  const uint64_t* c = b + G2A_W;
  const uint64_t* x = acc + G1_W * i;
  uint64_t z = 0;
#pragma unroll
  for (int w = 12; w < 18; w++) z |= x[w];
  const bool dead_a = a[12] != 0 || b[24] != 0;           // mod.rs:49-54: a pair with a member at infinity is skipped
  const bool dead_g = z == 0 || pvk[PVK_GAMMA + G2P_W - 1] != 0;
  const bool dead_d = c[12] != 0 || pvk[PVK_DELTA + G2P_W - 1] != 0;
  PJac r;
  r.x = ld_p2(b); r.y = ld_p2(b + 12); r.z = p2_one();
  mbar_wait_phase0(bar);
  P12 f;
  p12_one(f);
  PCoeffs cb;
  int idx = 0;
#pragma unroll 1
  for (int bit = BLS_LOOP_TOP; bit >= -1; bit--) {       // bit == -1 is the trailing doubling step (mod.rs:92-94)
    const bool add = bit >= 0 && ((BLS_LOOP_BITS >> bit) & 1ull);
#pragma unroll 1
    for (int phase = 0; phase < (add ? 2 : 1); phase++) {
      if (phase == 0) pg2_doubling_step(r, cb);
      else pg2_addition_step(r, ld_p2(b), ld_p2(b + 12), cb);
      p12_mul_by_line_pair(f, g16v_line(cb, a, dead_a), g16v_line(g16v_smem_coeffs(s_coeffs[0] + 36 * idx), x, dead_g));
      const PLine ld = g16v_line(g16v_smem_coeffs(s_coeffs[1] + 36 * idx), c, dead_d);
      p12_mul_by_line_pair(f, ld, ld, true);               // measured against p12_mul_by_014: profiles/groth16_verify.md
      idx++;
    }
    if (bit >= 0) p12_sqr(f, f);
  }
  p12_conjugate(f);
  P12 g, ab;
  const bool some = p_final_exponentiation(g, f);
  ld_p12(ab, pvk + PVK_AB);
  const bool eq = p12_eq(g, ab);
  if (active && pair_c() == 0) ok[i] = some && eq;
}

// ---- the randomized check -------------------------------------------------------------------------------------------------
// one thread per proof j: pa[j] = into_affine(rho_j A_j), qb[j] = B_j, pc[j] = C_j
__global__ void __launch_bounds__(G16V_TAIL_TPB) k_g16v_rlc_terms(const uint64_t* proofs, const uint64_t* rho, size_t m, uint64_t* pa, uint64_t* qb,
                                                                  uint64_t* pc) {
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint64_t* row = proofs + PROOF_W * j;
  Aff<Fp> a;
  ld_aff(a, row);
  Jac<Fp> p;
  if (a.inf) pt_set_zero(p);
  else { p.x = a.x; p.y = a.y; f_set_one(p.z); }
  pt_mul(p, ld_scalar(rho + 4 * j));
  pt_into_affine(a, p);
  st_aff(pa + G1A_W * j, a);
  for (int w = 0; w < G2A_W; w++) qb[G2A_W * j + w] = row[G1A_W + w];
  for (int w = 0; w < G1A_W; w++) pc[G1A_W * j + w] = row[G1A_W + G2A_W + w];
}

// block i: s[i] = sum_j rho_j (i = 0) or sum_j rho_j x_j(i-1) (mod r), canonical.  fr_mul(x R, rho) = x rho: the plain product.
__global__ void __launch_bounds__(G16V_SUM_TPB) k_g16v_rlc_sums(const uint64_t* inputs, const uint64_t* rho, size_t ni, size_t m, uint64_t* s) {
  __shared__ Fr part[G16V_SUM_TPB];
  const size_t i = blockIdx.x;
  Fr acc = fr_zero();
#pragma unroll 1
  for (size_t j = threadIdx.x; j < m; j += G16V_SUM_TPB) {
    const Fr r = g16v_ld_fr(rho + 4 * j);
    acc = fr_add(acc, i == 0 ? r : fr_mul(g16v_ld_fr(inputs + 4 * (j * ni + i - 1)), r));
  }
  part[threadIdx.x] = acc;
  __syncthreads();
#pragma unroll 1
  for (int h = G16V_SUM_TPB / 2; h >= 1; h >>= 1) {
    if (threadIdx.x < h) part[threadIdx.x] = fr_add(part[threadIdx.x], part[threadIdx.x + h]);
    __syncthreads();
  }
  if (threadIdx.x == 0) g16v_st_fr(s + 4 * i, part[0]);
}

// pairs m and m + 1 of the product: (sum_i s_i ic_i, -gamma), (sum_j rho_j C_j, -delta).  The sums are normalised Jacobian
// points, so their affine form is (x, y) and the infinity flag z == 0.
__global__ void k_g16v_rlc_pairs(const uint64_t* pvk, const uint64_t* sums, size_t m, uint64_t* p, uint64_t* q) {
  const int t = threadIdx.x;
  if (t >= 2) return;
  const uint64_t* src = sums + G1_W * t;
  uint64_t* dst = p + G1A_W * (m + t);
  uint64_t z = 0;
  for (int w = 0; w < 12; w++) dst[w] = src[w];
  for (int w = 12; w < 18; w++) z |= src[w];
  dst[12] = z == 0;
  for (int w = 0; w < G2A_W; w++) q[G2A_W * (m + t) + w] = pvk[(t ? PVK_DELTA_AFF : PVK_GAMMA_AFF) + w];
}

__global__ void k_g16v_rlc_compare(const uint64_t* prod, const uint8_t* some, const uint64_t* pw, uint8_t* ok1) {
  bool eq = *some != 0;
  for (int w = 0; w < FQ12_W; w++) eq = eq && prod[w] == pw[w];   // canonical values: equal iff the same words
  *ok1 = eq;
}

// ---- host side ------------------------------------------------------------------------------------------------------------

static size_t g16v_align(size_t x) { return (x + 255) & ~(size_t)255; }

namespace {
struct G16vLayout {
  size_t off_k, off_acc, off_work, total;                                              // per-proof path
  size_t off_pa, off_qb, off_pc, off_s, off_sums, off_gt, off_flag, off_rwork;         // randomized check
};
}  // namespace

static bool g16v_args_ok(const bls_ctx* ctx, size_t ni, size_t m) {
  return ctx && m <= G16V_MAX_M && ni < G16V_MAX_MN && m * (ni + 1) <= G16V_MAX_MN;
}
static bool g16v_rlc_args_ok(const bls_ctx* ctx, size_t ni, size_t m) { return ctx && m <= G16V_RLC_MAX && ni < G16V_RLC_MAX; }

// scratch of the per-proof path: the msm scalars, the m sums acc_j, the msm's work region.  0 on failure.
static size_t g16v_layout(bls_ctx* ctx, size_t ni, size_t m, G16vLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += g16v_align(bytes); return at; };
  l.off_k = take(m * (ni + 1) * sizeof(bls_fr_repr));
  l.off_acc = take(m * sizeof(bls_g1));
  const size_t work = bls_msm_batch_scratch_bytes(ctx, 1, ni + 1, m, 0);
  if (!work) return 0;
  l.off_work = take(work);
  return l.total = o;
}
// scratch of the randomized check: the m + 2 pairs of the product, the C_j, s, the two sums, the two GT values and the
// is_some flag, then one region for each msm and the product in turn.  0 on failure.
static size_t g16v_rlc_layout(bls_ctx* ctx, size_t ni, size_t m, G16vLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += g16v_align(bytes); return at; };
  l.off_pa = take((m + 2) * sizeof(bls_g1_affine));
  l.off_qb = take((m + 2) * sizeof(bls_g2_affine));
  l.off_pc = take(m * sizeof(bls_g1_affine));
  l.off_s = take((ni + 1) * sizeof(bls_fr_repr));
  l.off_sums = take(2 * sizeof(bls_g1));
  l.off_gt = take(2 * sizeof(bls_fq12));
  l.off_flag = take(1);
  size_t work = bls_multi_miller_scratch_bytes(ctx, m + 2);
  for (size_t n : {ni + 1, m}) {
    const size_t b = bls_msm_scratch_bytes(ctx, 1, n, 0);
    if (!b) return 0;
    work = b > work ? b : work;
  }
  if (!work) return 0;
  l.off_rwork = take(work);
  return l.total = o;
}

static int g16v_dev_impl(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t ni, const bls_groth16_proof* proofs,
                         const bls_fr* inputs, size_t m, uint8_t* ok, void* scratch, void* stream) {
  if (!g16v_args_ok(ctx, ni, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!pvk || ((uintptr_t)pvk & 15) || !ic || !proofs || (ni && !inputs) || !ok || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  G16vLayout l;
  if (!g16v_layout(ctx, ni, m, l)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  uint64_t *k = (uint64_t*)(base + l.off_k), *acc = (uint64_t*)(base + l.off_acc);
  k_g16v_scalars<<<blocks_for(m * (ni + 1), G16V_TPB), G16V_TPB, 0, st>>>((const uint64_t*)inputs, ni, m, k);
  LAUNCH_CHECK();
  TRY(bls_g1_msm_batch_dev(ctx, ic, 1, (const bls_fr_repr*)k, ni + 1, m, 0, (bls_g1*)acc, base + l.off_work, st));
  k_groth16_verify<<<blocks_for(2 * m, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, st>>>((const uint64_t*)pvk, (const uint64_t*)proofs, acc, m, ok);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int g16v_rlc_dev_impl(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t ni, const bls_groth16_proof* proofs,
                             const bls_fr* inputs, const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream) {
  if (!g16v_rlc_args_ok(ctx, ni, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) {                                                   // the empty batch: FE(one) == alpha_g1_beta_g2^0 holds
    if (!ok1) return BLS_OK;
    USE_DEVICE(ctx);
    CK(cudaMemsetAsync(ok1, 1, 1, pick(ctx, stream)));
    return BLS_OK;
  }
  if (!pvk || ((uintptr_t)pvk & 15) || !ic || !proofs || (ni && !inputs) || !rho || !ok1 || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  G16vLayout l;
  if (!g16v_rlc_layout(ctx, ni, m, l)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint64_t *pa = at(l.off_pa), *qb = at(l.off_qb), *pc = at(l.off_pc), *s = at(l.off_s), *sums = at(l.off_sums), *gt = at(l.off_gt);
  uint8_t* flag = (uint8_t*)at(l.off_flag);
  void* work = at(l.off_rwork);
  const uint64_t* vk = (const uint64_t*)pvk;
  k_g16v_rlc_terms<<<blocks_for(m, G16V_TAIL_TPB), G16V_TAIL_TPB, 0, st>>>((const uint64_t*)proofs, (const uint64_t*)rho, m, pa, qb, pc);
  LAUNCH_CHECK();
  k_g16v_rlc_sums<<<(unsigned)(ni + 1), G16V_SUM_TPB, 0, st>>>((const uint64_t*)inputs, (const uint64_t*)rho, ni, m, s);
  LAUNCH_CHECK();
  TRY(bls_g1_msm_dev(ctx, ic, (const bls_fr_repr*)s, ni + 1, 0, (bls_g1*)sums, work, st));
  TRY(bls_g1_msm_dev(ctx, (const bls_g1_affine*)pc, rho, m, 0, (bls_g1*)(sums + G1_W), work, st));
  k_g16v_rlc_pairs<<<1, 32, 0, st>>>(vk, sums, m, pa, qb);
  LAUNCH_CHECK();
  TRY(bls_pairing_product_dev(ctx, (const bls_g1_affine*)pa, (const bls_g2_affine*)qb, m + 2, (bls_fq12*)gt, flag, work, st));
  TRY(bls_fq12_pow_dev(ctx, &pvk->alpha_g1_beta_g2, (const bls_fr_repr*)s, (bls_fq12*)(gt + FQ12_W), 1, st));
  k_g16v_rlc_compare<<<1, 1, 0, st>>>(gt, flag, gt + FQ12_W, ok1);
  LAUNCH_CHECK();
  return BLS_OK;
}

extern "C" {

int bls_groth16_prepare_verifying_key(bls_ctx* ctx, const bls_g1_affine* alpha_g1, const bls_g2_affine* beta_g2, const bls_g2_affine* gamma_g2,
                                      const bls_g2_affine* delta_g2, bls_groth16_pvk* out) {
  if (!ctx || !alpha_g1 || !beta_g2 || !gamma_g2 || !delta_g2 || !out) return BLS_ERR_INVALID_ARGUMENT;
  bls_g2_affine neg[2] = {*gamma_g2, *delta_g2};
  for (bls_g2_affine& q : neg) {                                  // CurveAffine::negate: the identity stays as it is
    if (q.infinity) continue;
    bls_fq2 y;
    TRY(bls_field_op_batch(ctx, 2, BLS_OP_NEG, &q.y, nullptr, &y, nullptr, 1));
    q.y = y;
  }
  std::vector<bls_g2_prepared> prep(2);
  TRY(bls_g2_prepare_batch(ctx, neg, prep.data(), 2));
  bls_fq12 ab;
  TRY(bls_pairing_batch(ctx, alpha_g1, beta_g2, &ab, 1));
  memset(out, 0, sizeof(*out));
  out->neg_gamma_g2 = prep[0];
  out->neg_delta_g2 = prep[1];
  out->alpha_g1_beta_g2 = ab;
  out->neg_gamma_g2_affine = neg[0];
  out->neg_delta_g2_affine = neg[1];
  return BLS_OK;
}

size_t bls_groth16_verify_scratch_bytes(const bls_ctx* cctx, size_t num_inputs, size_t m) {
  if (!g16v_args_ok(cctx, num_inputs, m)) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  G16vLayout l;
  return g16v_layout(ctx, num_inputs, m, l);
}
int bls_groth16_verify_dev(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                           const bls_fr* inputs, size_t m, uint8_t* ok, void* scratch, void* stream) {
  return g16v_dev_impl(ctx, pvk, ic, num_inputs, proofs, inputs, m, ok, scratch, stream);
}
int bls_groth16_verify_batch(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                             const bls_fr* inputs, size_t m, uint8_t* ok) {
  if (!g16v_args_ok(ctx, num_inputs, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!pvk || !ic || !proofs || (num_inputs && !inputs) || !ok) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  G16vLayout l;
  if (!g16v_layout(ctx, num_inputs, m, l)) return BLS_ERR_CUDA;
  H2D(dpvk, pvk, sizeof(bls_groth16_pvk));                        // pool allocations are 256-byte aligned
  H2D(dic, ic, (num_inputs + 1) * sizeof(bls_g1_affine));
  H2D(dpr, proofs, m * sizeof(bls_groth16_proof));
  H2D(din, num_inputs ? inputs : nullptr, m * num_inputs * sizeof(bls_fr));
  DALLOC(dok, m);
  DALLOC(dscr, l.total);
  TRY(g16v_dev_impl(ctx, (const bls_groth16_pvk*)dpvk.p, (const bls_g1_affine*)dic.p, num_inputs, (const bls_groth16_proof*)dpr.p,
                    (const bls_fr*)din.p, m, (uint8_t*)dok.p, dscr.p, ctx->stream));
  D2H(ok, dok, m);
  SYNC();
  return BLS_OK;
}

size_t bls_groth16_verify_rlc_scratch_bytes(const bls_ctx* cctx, size_t num_inputs, size_t m) {
  if (!g16v_rlc_args_ok(cctx, num_inputs, m)) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  G16vLayout l;
  return g16v_rlc_layout(ctx, num_inputs, m, l);
}
int bls_groth16_verify_rlc_dev(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                               const bls_fr* inputs, const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream) {
  return g16v_rlc_dev_impl(ctx, pvk, ic, num_inputs, proofs, inputs, rho, m, ok1, scratch, stream);
}
int bls_groth16_verify_rlc_batch(bls_ctx* ctx, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                                 const bls_fr* inputs, const bls_fr_repr* rho, size_t m, uint8_t* ok1) {
  if (!g16v_rlc_args_ok(ctx, num_inputs, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) {                                                   // the empty batch: the equation holds
    if (ok1) *ok1 = 1;
    return BLS_OK;
  }
  if (!pvk || !ic || !proofs || (num_inputs && !inputs) || !rho || !ok1) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  G16vLayout l;
  if (!g16v_rlc_layout(ctx, num_inputs, m, l)) return BLS_ERR_CUDA;
  H2D(dpvk, pvk, sizeof(bls_groth16_pvk));
  H2D(dic, ic, (num_inputs + 1) * sizeof(bls_g1_affine));
  H2D(dpr, proofs, m * sizeof(bls_groth16_proof));
  H2D(din, num_inputs ? inputs : nullptr, m * num_inputs * sizeof(bls_fr));
  H2D(drho, rho, m * sizeof(bls_fr_repr));
  DALLOC(dok, 1);
  DALLOC(dscr, l.total);
  TRY(g16v_rlc_dev_impl(ctx, (const bls_groth16_pvk*)dpvk.p, (const bls_g1_affine*)dic.p, num_inputs, (const bls_groth16_proof*)dpr.p,
                        (const bls_fr*)din.p, (const bls_fr_repr*)drho.p, m, (uint8_t*)dok.p, dscr.p, ctx->stream));
  D2H(ok1, dok, 1);
  SYNC();
  return BLS_OK;
}

}  // extern "C"
