// kernels_groth16_mpc.cu -- phase 2 of the Groth16 ceremony after the initial key (include/pairing_b200_mpc.h):
// phase2's MPCParameters::contribute (bls_groth16_mpc_contribute_*) and MPCParameters::verify (bls_groth16_mpc_verify_*).
// bls_groth16_mpc_new_* lives with the generator in kernels_groth16_setup.cu, whose scan and emit kernels it shares.
// Its own translation unit (see abi_common.cuh): the inversion, the multiexp, the normalisation, the Miller loop, the Fq12
// products and the final exponentiation are the other units' entry points, called through the C ABI.
//
// contribute: h_len + l_len multiplications by ONE scalar d = delta^-1, plus [delta] delta_g1, [delta] s, [delta] delta_g2,
//   [delta] r: k_mpc_prep lays the rows out as Jacobian bases with the scalar replicated, bls_g*_wnaf_mul_dev multiplies,
//   then bls_g*_batch_normalization_dev and k_mpc_emit (canonical affine rows).  A kernel that recoded the one scalar per
//   block into shared memory and ran every lane through the same double / add sequence was 1.06x slower than the wNAF
//   batch with the scalar replicated at 2^21 rows on a B200 (DESIGN.md), so it was removed.
// verify: k_mpcv_diff compares the unchanged queries word by word; bls_g1_msm_dev forms the four merged sums;
//   k_mpcv_pairs lays out, for the C = 2k + 3 checks e(A, B) = e(C, D), the pairs (A, B) and (-C, D); one Miller loop over
//   the 2C pairs, one Fq12 product per check, one final exponentiation per check, and k_mpcv_finish folds everything into
//   *ok1.
#include "curve_io.cuh"
#include "fr.cuh"
#include "../../include/pairing_b200_mpc.h"

#define MPC_TPB 128
#define MPC_MAX_ROWS ((size_t)1 << 26)
#define MPC_MAX_K ((size_t)1 << 16)
// bls_groth16_mpc_pubkey in u64 words
#define PK_DA 0
#define PK_S G1A_W
#define PK_SD (2 * G1A_W)
#define PK_R (3 * G1A_W)
#define PK_RD (3 * G1A_W + G2A_W)
#define PK_W (3 * G1A_W + 2 * G2A_W)
// bls_groth16_vk_points in u64 words
#define VK_DELTA1 (2 * G1A_W)
#define VK_DELTA2 (3 * G1A_W + 2 * G2A_W)

__device__ __forceinline__ Scalar mpc_repr(const uint64_t* p) {
  Fr a, one = fr_zero();
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; a.v[2 * i] = t.x; a.v[2 * i + 1] = t.y; }
  one.v[0] = 1;
  const Fr c = fr_mul(a, one);
  Scalar s;
#pragma unroll
  for (int i = 0; i < 8; i++) s.v[i] = c.v[i];
  return s;
}

// the input of bls_g*_wnaf_mul_dev: out[t] = in[t] as a Jacobian row, k[t] = into_repr of the Montgomery Fr at `scalar`
template <class F>
__global__ void __launch_bounds__(MPC_TPB) k_mpc_prep(const uint64_t* in, size_t n, const uint64_t* scalar, uint64_t* out, uint64_t* k) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int W = FW<F>::W;
  Aff<F> a;
  ld_aff(a, in + (size_t)(2 * W + 1) * t);
  Jac<F> b;
  pt_set_zero(b);
  if (!a.inf) { b.x = a.x; b.y = a.y; f_set_one(b.z); }
  st_jac(out + (size_t)(3 * W) * t, b);
  const Scalar s = mpc_repr(scalar);
#pragma unroll
  for (int i = 0; i < 4; i++) k[4 * t + i] = (uint64_t)s.v[2 * i] | ((uint64_t)s.v[2 * i + 1] << 32);
}

// normalised Jacobian rows -> canonical affine rows (the identity is (0, one, infinity = 1))
template <class F>
__global__ void __launch_bounds__(MPC_TPB) k_mpc_emit(const uint64_t* in, size_t n, uint64_t* out) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int W = FW<F>::W;
  Jac<F> p;
  ld_jac(p, in + (size_t)(3 * W) * t);
  Aff<F> a;
  a.inf = pt_is_zero(p);
  if (a.inf) { f_set_zero(a.x); f_set_one(a.y); }
  else { a.x = p.x; a.y = p.y; }
  st_aff(out + (size_t)(2 * W + 1) * t, a);
}

// *flag |= 1 when x and y differ in any of `words` words
__global__ void __launch_bounds__(MPC_TPB) k_mpcv_diff(const uint64_t* x, const uint64_t* y, size_t words, uint32_t* flag) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool d = t < words && x[t] != y[t];
  if (__any_sync(0xffffffffu, d) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}

__device__ __forceinline__ void mpcv_copy(uint64_t* dst, const uint64_t* src, int words) {
#pragma unroll 1
  for (int i = 0; i < words; i++) dst[i] = src[i];
}
// an affine G1 row of a normalised Jacobian point, negated when neg
__device__ __forceinline__ void mpcv_g1(uint64_t* dst, const uint64_t* src, bool jac, bool neg) {
  Aff<Fp> a;
  if (jac) {
    Jac<Fp> p;
    ld_jac(p, src);
    a.inf = pt_is_zero(p);
    if (a.inf) { f_set_zero(a.x); f_set_one(a.y); } else { a.x = p.x; a.y = p.y; }
  } else {
    ld_aff(a, src);
  }
  if (neg && !a.inf) a.y = fp_neg(a.y);
  st_aff(dst, a);
}

// One thread per check c < C = 2k + 3: P[c], Q[c] = (A, B) and P[C + c], Q[C + c] = (-C, D) of e(A, B) = e(C, D).
// vkp: before.delta_g1 | after.delta_g1 (G1 rows), then before.delta_g2 | after.delta_g2 (G2 rows); sums: the four merged
// sums (normalised Jacobian) before.h, after.h, before.l, after.l.
__global__ void __launch_bounds__(MPC_TPB) k_mpcv_pairs(const uint64_t* pk, size_t k, const uint64_t* vkp, const uint64_t* sums, uint64_t* P,
                                                        uint64_t* Q) {
  const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x, C = 2 * k + 3;
  if (c >= C) return;
  const uint64_t *bd1 = vkp, *bd2 = vkp + 2 * G1A_W, *ad2 = bd2 + G2A_W;
  const uint64_t *A, *B, *Cc, *D;
  bool ajac = false, cjac = false;
  if (c < 2 * k) {
    const size_t j = c >> 1;
    const uint64_t* p = pk + PK_W * j;
    if ((c & 1) == 0) { A = p + PK_SD; B = p + PK_R; Cc = p + PK_S; D = p + PK_RD; }
    else { A = j ? pk + PK_W * (j - 1) + PK_DA : bd1; B = p + PK_RD; Cc = p + PK_DA; D = p + PK_R; }
  } else if (c == 2 * k) {
    A = bd1; B = ad2; Cc = k ? pk + PK_W * (k - 1) + PK_DA : bd1; D = bd2;
  } else {
    const size_t m = c - 2 * k - 1;                   // 0: h, 1: l
    A = sums + G1_W * (2 * m); B = bd2; Cc = sums + G1_W * (2 * m + 1); D = ad2;
    ajac = cjac = true;
  }
  mpcv_g1(P + G1A_W * c, A, ajac, false);
  mpcv_copy(Q + G2A_W * c, B, G2A_W);
  mpcv_g1(P + G1A_W * (C + c), Cc, cjac, true);
  mpcv_copy(Q + G2A_W * (C + c), D, G2A_W);
}

// One block: *ok1 = no flag, every check's final exponentiation is Some(one), and after.delta_g1 == d_(k-1) bytewise
__global__ void __launch_bounds__(MPC_TPB) k_mpcv_finish(const uint64_t* fe, const uint8_t* is_some, size_t C, const uint32_t* flags,
                                                         const uint64_t* pk, size_t k, const uint64_t* vkp, uint8_t* ok1) {
  __shared__ int bad;
  if (threadIdx.x == 0) bad = *flags != 0;
  __syncthreads();
  uint64_t one[6];
  st_fp(one, fp_one());
  int b = 0;
  for (size_t c = threadIdx.x; c < C; c += blockDim.x) {
    const uint64_t* f = fe + FQ12_W * c;
    b |= !is_some[c];
    for (int i = 0; i < FQ12_W; i++) b |= f[i] != (i < 6 ? one[i] : 0ull);
  }
  const uint64_t *last = k ? pk + PK_W * (k - 1) + PK_DA : vkp, *ad1 = vkp + G1A_W;
  for (int i = threadIdx.x; i < G1A_W; i += blockDim.x) b |= last[i] != ad1[i];
  if (b) atomicOr(&bad, 1);
  __syncthreads();
  if (threadIdx.x == 0) *ok1 = bad == 0;
}

// ---- host side ----------------------------------------------------------------------------------------------------------

static size_t mpc_align(size_t x) { return (x + 255) & ~(size_t)255; }

static bool mpc_fr_canonical_nonzero(const bls_fr* x) {
  static const uint64_t R[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
  if (!(x->l[0] | x->l[1] | x->l[2] | x->l[3])) return false;
  for (int i = 3; i >= 0; i--)
    if (x->l[i] != R[i]) return x->l[i] < R[i];
  return false;
}

namespace {
struct McPlan {
  size_t n1;                                      // h_len + l_len + 2 G1 products
  size_t off_fr, off_aff, off_j1, off_o1, off_k1, off_j2, off_o2, off_k2, off_bn, total;
};
}  // namespace

static size_t mc_layout(bls_ctx* ctx, size_t h_len, size_t l_len, McPlan& p) {
  p.n1 = h_len + l_len + 2;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += mpc_align(bytes ? bytes : 1); return at; };
  p.off_fr = take(2 * sizeof(bls_fr));
  p.off_aff = take(2 * sizeof(bls_g1_affine) + 2 * sizeof(bls_g2_affine));
  p.off_j1 = take(p.n1 * sizeof(bls_g1));
  p.off_o1 = take(p.n1 * sizeof(bls_g1));
  p.off_k1 = take(p.n1 * sizeof(bls_fr_repr));
  p.off_j2 = take(2 * sizeof(bls_g2));
  p.off_o2 = take(2 * sizeof(bls_g2));
  p.off_k2 = take(2 * sizeof(bls_fr_repr));
  const size_t b1 = bls_batch_normalization_scratch_bytes(ctx, 1, p.n1), b2 = bls_batch_normalization_scratch_bytes(ctx, 2, 2);
  if (!b1 || !b2) return 0;
  p.off_bn = take(b1 > b2 ? b1 : b2);
  p.total = o;
  return o;
}

static bool mc_args_ok(const bls_ctx* ctx, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, const bls_groth16_vk_points* vk,
                       const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, const bls_g1_affine* h_out,
                       const bls_g1_affine* l_out, const bls_groth16_mpc_pubkey* pubkey) {
  if (!ctx || !delta || !mpc_fr_canonical_nonzero(delta) || !s || !r || !vk || !pubkey) return false;
  if (h_len > MPC_MAX_ROWS || l_len > MPC_MAX_ROWS) return false;
  if ((h_len && (!h || !h_out)) || (l_len && (!l || !l_out))) return false;
  return true;
}

template <class F> static void mc_emit(cudaStream_t st, const uint64_t* in, size_t n, void* out) {
  if (n) k_mpc_emit<F><<<blocks_for(n, MPC_TPB), MPC_TPB, 0, st>>>(in, n, (uint64_t*)out);
}

static int mc_dev_impl(bls_ctx* ctx, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, bls_groth16_vk_points* vk,
                       const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, bls_g1_affine* h_out, bls_g1_affine* l_out,
                       bls_groth16_mpc_pubkey* pubkey, void* scratch, void* stream) {
  if (!mc_args_ok(ctx, delta, s, r, vk, h, h_len, l, l_len, h_out, l_out, pubkey) || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  McPlan p;
  if (!mc_layout(ctx, h_len, l_len, p)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  uint64_t *fr = (uint64_t*)(base + p.off_fr), *aff = (uint64_t*)(base + p.off_aff), *j1 = (uint64_t*)(base + p.off_j1), *j2 = (uint64_t*)(base + p.off_j2);
  uint64_t *a1 = aff, *a2 = aff + 2 * G1A_W;     // [delta_g1, s], [delta_g2, r]
  uint64_t* dvk = (uint64_t*)vk;
  // delta, then d = delta^-1; s and r from the host (a pageable source has been staged when cudaMemcpyAsync returns)
  CK(cudaMemcpyAsync(fr, delta, sizeof(bls_fr), cudaMemcpyHostToDevice, st));
  TRY(bls_fr_op_dev(ctx, BLS_OP_INV, (const bls_fr*)fr, nullptr, (bls_fr*)(fr + 4), nullptr, 1, st));
  CK(cudaMemcpyAsync(a1, dvk + VK_DELTA1, sizeof(bls_g1_affine), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(a1 + G1A_W, s, sizeof(bls_g1_affine), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(a2, dvk + VK_DELTA2, sizeof(bls_g2_affine), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(a2 + G2A_W, r, sizeof(bls_g2_affine), cudaMemcpyHostToDevice, st));
  // G1 products [h | l | delta_g1 | s_delta], G2 products [delta_g2 | r_delta]
  uint64_t *o1 = (uint64_t*)(base + p.off_o1), *k1 = (uint64_t*)(base + p.off_k1), *o2 = (uint64_t*)(base + p.off_o2), *k2 = (uint64_t*)(base + p.off_k2);
  if (h_len) {
    k_mpc_prep<Fp><<<blocks_for(h_len, MPC_TPB), MPC_TPB, 0, st>>>((const uint64_t*)h, h_len, fr + 4, j1, k1);
    LAUNCH_CHECK();
  }
  if (l_len) {
    k_mpc_prep<Fp><<<blocks_for(l_len, MPC_TPB), MPC_TPB, 0, st>>>((const uint64_t*)l, l_len, fr + 4, j1 + G1_W * h_len, k1 + 4 * h_len);
    LAUNCH_CHECK();
  }
  k_mpc_prep<Fp><<<1, MPC_TPB, 0, st>>>(a1, 2, fr, j1 + G1_W * (h_len + l_len), k1 + 4 * (h_len + l_len));
  LAUNCH_CHECK();
  k_mpc_prep<Fp2><<<1, MPC_TPB, 0, st>>>(a2, 2, fr, j2, k2);
  LAUNCH_CHECK();
  TRY(bls_g1_wnaf_mul_dev(ctx, (const bls_g1*)j1, (const bls_fr_repr*)k1, (bls_g1*)o1, p.n1, 0, st));
  TRY(bls_g2_wnaf_mul_dev(ctx, (const bls_g2*)j2, (const bls_fr_repr*)k2, (bls_g2*)o2, 2, 0, st));
  j1 = o1;
  j2 = o2;
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)j1, p.n1, base + p.off_bn, st));
  TRY(bls_g2_batch_normalization_dev(ctx, (bls_g2*)j2, 2, base + p.off_bn, st));
  uint64_t* pk = (uint64_t*)pubkey;
  const uint64_t* x1 = j1 + G1_W * (h_len + l_len);
  mc_emit<Fp>(st, j1, h_len, h_out);
  mc_emit<Fp>(st, j1 + G1_W * h_len, l_len, l_out);
  mc_emit<Fp>(st, x1, 1, dvk + VK_DELTA1);
  mc_emit<Fp>(st, x1, 1, pk + PK_DA);
  mc_emit<Fp>(st, x1 + G1_W, 1, pk + PK_SD);
  mc_emit<Fp2>(st, j2, 1, dvk + VK_DELTA2);
  mc_emit<Fp2>(st, j2 + G2_W, 1, pk + PK_RD);
  LAUNCH_CHECK();
  CK(cudaMemcpyAsync(pk + PK_S, a1 + G1A_W, sizeof(bls_g1_affine), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(pk + PK_R, a2 + G2A_W, sizeof(bls_g2_affine), cudaMemcpyDeviceToDevice, st));
  return BLS_OK;
}

// ---- verify ----
namespace {
struct MvPlan {
  size_t C;                                        // checks: 2k + 3
  size_t off_flags, off_vkp, off_sums, off_msm, off_bn, off_P, off_Q, off_ml, off_prod, off_fe, off_some, total;
};
}  // namespace

static bool mv_key_ok(const bls_groth16_key* key) {
  if (!key) return false;
  const size_t lens[5] = {key->ic_len, key->h_len, key->l_len, key->a_len, key->b_len};
  for (size_t x : lens)
    if (x > MPC_MAX_ROWS) return false;
  return (!key->ic_len || key->ic) && (!key->h_len || key->h) && (!key->l_len || key->l) && (!key->a_len || key->a) &&
         (!key->b_len || (key->b_g1 && key->b_g2));
}

static bool mv_args_ok(const bls_ctx* ctx, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                       const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, const uint8_t* ok1) {
  if (!ctx || !mv_key_ok(before) || !mv_key_ok(after) || !ok1 || k > MPC_MAX_K || (k && !pk)) return false;
  if ((before->h_len || after->h_len) && !rho_h) return false;
  if ((before->l_len || after->l_len) && !rho_l) return false;
  return true;
}

// the parts compared on the host: lengths and the vk points that must not change
static bool mv_same_shape(const bls_groth16_key* b, const bls_groth16_key* a) {
  return b->ic_len == a->ic_len && b->h_len == a->h_len && b->l_len == a->l_len && b->a_len == a->a_len && b->b_len == a->b_len &&
         !memcmp(&b->vk.alpha_g1, &a->vk.alpha_g1, sizeof(bls_g1_affine)) && !memcmp(&b->vk.beta_g1, &a->vk.beta_g1, sizeof(bls_g1_affine)) &&
         !memcmp(&b->vk.beta_g2, &a->vk.beta_g2, sizeof(bls_g2_affine)) && !memcmp(&b->vk.gamma_g2, &a->vk.gamma_g2, sizeof(bls_g2_affine));
}

static size_t mv_layout(bls_ctx* ctx, const bls_groth16_key* before, size_t k, MvPlan& p) {
  p.C = 2 * k + 3;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += mpc_align(bytes ? bytes : 1); return at; };
  p.off_flags = take(sizeof(uint32_t));
  p.off_vkp = take(2 * sizeof(bls_g1_affine) + 2 * sizeof(bls_g2_affine));
  p.off_sums = take(4 * sizeof(bls_g1));
  size_t msm = 0;
  for (size_t n : {before->h_len, before->l_len}) {
    if (!n) continue;
    const size_t b = bls_msm_scratch_bytes(ctx, 1, n, 0);
    if (!b) return 0;
    msm = b > msm ? b : msm;
  }
  p.off_msm = take(msm);
  const size_t bn = bls_batch_normalization_scratch_bytes(ctx, 1, 4);
  if (!bn) return 0;
  p.off_bn = take(bn);
  p.off_P = take(2 * p.C * sizeof(bls_g1_affine));
  p.off_Q = take(2 * p.C * sizeof(bls_g2_affine));
  p.off_ml = take(2 * p.C * sizeof(bls_fq12));
  p.off_prod = take(p.C * sizeof(bls_fq12));
  p.off_fe = take(p.C * sizeof(bls_fq12));
  p.off_some = take(p.C);
  p.total = o;
  return o;
}

static int mv_dev_impl(bls_ctx* ctx, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                       const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, uint8_t* ok1, void* scratch, void* stream) {
  if (!mv_args_ok(ctx, before, after, pk, k, rho_h, rho_l, ok1) || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  MvPlan p;
  if (!mv_layout(ctx, before, k, p)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  if (!mv_same_shape(before, after)) {
    CK(cudaMemsetAsync(ok1, 0, 1, st));
    return BLS_OK;
  }
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint32_t* flags = (uint32_t*)(base + p.off_flags);
  uint64_t *vkp = at(p.off_vkp), *sums = at(p.off_sums), *P = at(p.off_P), *Q = at(p.off_Q), *ml = at(p.off_ml), *prod = at(p.off_prod),
           *fe = at(p.off_fe);
  uint8_t* some = (uint8_t*)(base + p.off_some);
  uint64_t up[2 * G1A_W + 2 * G2A_W];
  memcpy(up, &before->vk.delta_g1, sizeof(bls_g1_affine));
  memcpy(up + G1A_W, &after->vk.delta_g1, sizeof(bls_g1_affine));
  memcpy(up + 2 * G1A_W, &before->vk.delta_g2, sizeof(bls_g2_affine));
  memcpy(up + 2 * G1A_W + G2A_W, &after->vk.delta_g2, sizeof(bls_g2_affine));
  CK(cudaMemcpyAsync(vkp, up, sizeof(up), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(flags, 0, sizeof(uint32_t), st));
  CK(cudaMemsetAsync(sums, 0, 4 * sizeof(bls_g1), st));            // z = 0: the identity when a query is empty
  // 1. the unchanged queries
  const struct { const void *x, *y; size_t words; } same[4] = {
      {before->ic, after->ic, before->ic_len * G1A_W}, {before->a, after->a, before->a_len * G1A_W},
      {before->b_g1, after->b_g1, before->b_len * G1A_W}, {before->b_g2, after->b_g2, before->b_len * G2A_W}};
  for (const auto& d : same) {
    if (!d.words) continue;
    k_mpcv_diff<<<blocks_for(d.words, MPC_TPB), MPC_TPB, 0, st>>>((const uint64_t*)d.x, (const uint64_t*)d.y, d.words, flags);
    LAUNCH_CHECK();
  }
  // 4. the merged sums: before.h, after.h, before.l, after.l
  const struct { const bls_g1_affine* rows; const bls_fr_repr* rho; size_t n; } msm[4] = {
      {before->h, rho_h, before->h_len}, {after->h, rho_h, after->h_len}, {before->l, rho_l, before->l_len}, {after->l, rho_l, after->l_len}};
  for (int i = 0; i < 4; i++) {
    if (!msm[i].n) continue;
    TRY(bls_g1_msm_dev(ctx, msm[i].rows, msm[i].rho, msm[i].n, 0, (bls_g1*)(sums + G1_W * i), base + p.off_msm, st));
  }
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)sums, 4, base + p.off_bn, st));
  // 2., 3., 4.: the pairing checks
  k_mpcv_pairs<<<blocks_for(p.C, MPC_TPB), MPC_TPB, 0, st>>>((const uint64_t*)pk, k, vkp, sums, P, Q);
  LAUNCH_CHECK();
  TRY(bls_miller_loop_dev(ctx, (const bls_g1_affine*)P, (const bls_g2_affine*)Q, (bls_fq12*)ml, 2 * p.C, st));
  TRY(bls_pair_field_op_dev(ctx, 12, BLS_OP_MUL, ml, ml + FQ12_W * p.C, prod, nullptr, p.C, st));
  TRY(bls_final_exponentiation_dev(ctx, (const bls_fq12*)prod, (bls_fq12*)fe, some, p.C, st));
  k_mpcv_finish<<<1, MPC_TPB, 0, st>>>(fe, some, p.C, flags, (const uint64_t*)pk, k, vkp, ok1);
  LAUNCH_CHECK();
  return BLS_OK;
}

extern "C" {

size_t bls_groth16_mpc_contribute_scratch_bytes(const bls_ctx* cctx, size_t h_len, size_t l_len) {
  if (!cctx || h_len > MPC_MAX_ROWS || l_len > MPC_MAX_ROWS) return 0;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  McPlan p;
  return mc_layout(ctx, h_len, l_len, p);
}

int bls_groth16_mpc_contribute_dev(bls_ctx* ctx, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, bls_groth16_vk_points* vk,
                                   const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, bls_g1_affine* h_out,
                                   bls_g1_affine* l_out, bls_groth16_mpc_pubkey* pubkey, void* scratch, void* stream) {
  return mc_dev_impl(ctx, delta, s, r, vk, h, h_len, l, l_len, h_out, l_out, pubkey, scratch, stream);
}

int bls_groth16_mpc_contribute_batch(bls_ctx* ctx, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, bls_groth16_vk_points* vk,
                                     const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, bls_g1_affine* h_out,
                                     bls_g1_affine* l_out, bls_groth16_mpc_pubkey* pubkey) {
  if (!mc_args_ok(ctx, delta, s, r, vk, h, h_len, l, l_len, h_out, l_out, pubkey)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  McPlan p;
  if (!mc_layout(ctx, h_len, l_len, p)) return BLS_ERR_CUDA;
  const size_t ga = sizeof(bls_g1_affine);
  H2D(dvk, vk, sizeof(bls_groth16_vk_points));
  H2D(dh, h_len ? h : nullptr, h_len * ga);
  H2D(dl, l_len ? l : nullptr, l_len * ga);
  DALLOC(dpk, sizeof(bls_groth16_mpc_pubkey));
  DALLOC(dscr, p.total);
  TRY(mc_dev_impl(ctx, delta, s, r, (bls_groth16_vk_points*)dvk.p, (const bls_g1_affine*)dh.p, h_len, (const bls_g1_affine*)dl.p, l_len,
                  (bls_g1_affine*)dh.p, (bls_g1_affine*)dl.p, (bls_groth16_mpc_pubkey*)dpk.p, dscr.p, ctx->stream));
  CK(cudaMemcpyAsync(vk, dvk.p, sizeof(bls_groth16_vk_points), cudaMemcpyDeviceToHost, ctx->stream));
  if (h_len) CK(cudaMemcpyAsync(h_out, dh.p, h_len * ga, cudaMemcpyDeviceToHost, ctx->stream));
  if (l_len) CK(cudaMemcpyAsync(l_out, dl.p, l_len * ga, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(pubkey, dpk.p, sizeof(bls_groth16_mpc_pubkey), cudaMemcpyDeviceToHost, ctx->stream));
  SYNC();
  return BLS_OK;
}

size_t bls_groth16_mpc_verify_scratch_bytes(const bls_ctx* cctx, const bls_groth16_key* before, const bls_groth16_key* after, size_t k) {
  if (!cctx || !before || !after || k > MPC_MAX_K) return 0;
  for (const bls_groth16_key* key : {before, after}) {
    const size_t lens[5] = {key->ic_len, key->h_len, key->l_len, key->a_len, key->b_len};
    for (size_t x : lens)
      if (x > MPC_MAX_ROWS) return 0;
  }
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  MvPlan p;
  return mv_layout(ctx, before, k, p);
}

int bls_groth16_mpc_verify_dev(bls_ctx* ctx, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                               const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, uint8_t* ok1, void* scratch, void* stream) {
  return mv_dev_impl(ctx, before, after, pk, k, rho_h, rho_l, ok1, scratch, stream);
}

int bls_groth16_mpc_verify_batch(bls_ctx* ctx, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                                 const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, uint8_t* ok1) {
  if (!mv_args_ok(ctx, before, after, pk, k, rho_h, rho_l, ok1)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  MvPlan p;
  if (!mv_layout(ctx, before, k, p)) return BLS_ERR_CUDA;
  const size_t ga = sizeof(bls_g1_affine), g2a = sizeof(bls_g2_affine);
  // both keys' queries, pk and the randomizers on the device
  bls_groth16_key dk[2] = {*before, *after};
  DevBuf bufs[2][6] = {{DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx)},
                       {DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx), DevBuf(ctx)}};
  for (int i = 0; i < 2; i++) {
    bls_groth16_key& K = dk[i];
    const struct { const void** ptr; size_t bytes; } q[6] = {
        {(const void**)&K.ic, K.ic_len * ga}, {(const void**)&K.h, K.h_len * ga}, {(const void**)&K.l, K.l_len * ga},
        {(const void**)&K.a, K.a_len * ga}, {(const void**)&K.b_g1, K.b_len * ga}, {(const void**)&K.b_g2, K.b_len * g2a}};
    for (int j = 0; j < 6; j++) {
      CK(bufs[i][j].alloc(q[j].bytes));
      if (q[j].bytes) CK(cudaMemcpyAsync(bufs[i][j].p, *q[j].ptr, q[j].bytes, cudaMemcpyHostToDevice, ctx->stream));
      *q[j].ptr = bufs[i][j].p;
    }
  }
  H2D(dpk, k ? pk : nullptr, k * sizeof(bls_groth16_mpc_pubkey));
  H2D(drh, before->h_len ? rho_h : nullptr, before->h_len * sizeof(bls_fr_repr));
  H2D(drl, before->l_len ? rho_l : nullptr, before->l_len * sizeof(bls_fr_repr));
  DALLOC(dok, 1);
  DALLOC(dscr, p.total);
  TRY(mv_dev_impl(ctx, &dk[0], &dk[1], (const bls_groth16_mpc_pubkey*)dpk.p, k, (const bls_fr_repr*)drh.p, (const bls_fr_repr*)drl.p,
                  (uint8_t*)dok.p, dscr.p, ctx->stream));
  CK(cudaMemcpyAsync(ok1, dok.p, 1, cudaMemcpyDeviceToHost, ctx->stream));
  SYNC();
  return BLS_OK;
}

}  // extern "C"
