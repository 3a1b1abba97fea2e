// kernels_kzg.cu -- KZG polynomial commitments for m polynomials in one call: commit, open (evaluation and quotient proof),
// prepare_verifying_key, verify and the randomized batch check (bls_kzg_*).  Its own translation unit (see abi_common.cuh):
// the multiexps, the Fr ops, the G2 preparation and the normalisation are the other units' entry points, called through the
// C ABI, so no existing kernel is recompiled.
//
// commit: bls_fr_op_dev(INTO_REPR) -> bls_g1_msm_batch_dev(srs, shared) -> k_kzg_emit (normalised Jacobian -> affine rows).
// open:   the quotient q = (p - p(z)) / (X - z) and y = p(z) by a suffix scan, s_i = sum_{k >= i} p_k z^(k-i), so that y = s_0
//         and q_(i-1) = s_i.  s is a linear recurrence s_i = p_i + z s_(i+1); the scan runs it in chunks of KZG_CHUNK
//         coefficients per thread: k_kzg_scan_up reduces every chunk to its Horner value (the next level's entries, whose
//         multiplier is z^KZG_CHUNK), level after level until one chunk is left per polynomial; k_kzg_scan_down then walks
//         the levels back, each chunk running Horner again from the carry of the chunks above it.  Level 0's pass writes the
//         q_i as canonical bls_fr_repr -- the scalars bls_g1_msm_batch_dev(srs, shared, q, n - 1, m) reads -- and y_j.
//         Then the multiexp and k_kzg_emit.
// verify: k_kzg_term (one thread per proof: P_j = C_j - y_j g + z_j pi_j by one joint double-and-add over {g, pi_j, g + pi_j}),
//         bls_g1_batch_normalization_dev, k_kzg_verify (one lane pair per proof: the Miller loops of (P_j, h) and
//         (pi_j, -tau h) fused, both prepared points staged once per block by two TMA bulk copies; final exponentiation;
//         comparison with one).
// verify_rlc: k_kzg_rlc_scalars / k_kzg_rlc_sum (the msm scalars [rho_j], [rho_j z_j], -sum rho_j y_j), one bls_g1_msm_dev
//         over [C, pi, g], one over (pi, rho), k_kzg_emit, and k_kzg_verify on the two sums (m = 1).
#include <stddef.h>

#include <vector>

#include "curve_io.cuh"
#include "fr.cuh"
#include "pair_io.cuh"

#define KZG_TPB 128
#define KZG_CHUNK_LOG 5
#define KZG_CHUNK (1 << KZG_CHUNK_LOG)    /* coefficients per thread at every level of the scan */
#define KZG_MAX_LEVELS 8                  /* n <= 2^26: at most 6 levels */
#define KZG_TERM_TPB 32                   /* k_kzg_term runs a single-thread chain per proof: spread them over the SMs */
#define KZG_SUM_TPB 256
#define KZG_MAX_M ((size_t)1 << 16)       /* commit / open: bls_g1_msm_batch_dev's limits */
#define KZG_MAX_MN ((size_t)1 << 26)
#define KZG_VERIFY_MAX ((size_t)1 << 26)  /* per-proof verify */
#define KZG_RLC_MAX (((size_t)1 << 25) - 1) /* randomized check: 2m + 1 bases for bls_g1_msm_dev (<= 2^26) */

// bls_kzg_pvk in u64 words
#define KPVK_H 0
#define KPVK_NTH (G2P_W + 1)
#define KPVK_G (2 * (G2P_W + 1))
#define KPVK_H_AFF (KPVK_G + G1A_W)
#define KPVK_NTH_AFF (KPVK_H_AFF + G2A_W)
#define KPVK_W (KPVK_NTH_AFF + G2A_W)
#define KZG_COEFF_BYTES (68 * 36 * 8)
static_assert(sizeof(bls_kzg_pvk) == KPVK_W * 8, "bls_kzg_pvk layout");
static_assert(offsetof(bls_kzg_pvk, neg_tau_h_prepared) == KPVK_NTH * 8 && KPVK_NTH * 8 % 16 == 0, "neg_tau_h_prepared must be 16-byte aligned");
static_assert(offsetof(bls_kzg_pvk, g) == KPVK_G * 8 && offsetof(bls_kzg_pvk, neg_tau_h) == KPVK_NTH_AFF * 8, "bls_kzg_pvk layout");

// ---- Fr scalars -----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ Fr kzg_ld_fr(const uint64_t* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void kzg_st_fr(uint64_t* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
// into_repr(): the Montgomery product with the integer 1
__device__ __forceinline__ Fr kzg_into_repr(const Fr& a) {
  Fr one = fr_zero();
  one.v[0] = 1;
  return fr_mul(a, one);
}
__device__ __forceinline__ bool kzg_lt_r(const Fr& a) { return !fr_geq(a, fr_modulus()); }

// ---- open: the suffix scan ------------------------------------------------------------------------------------------------
// the multiplier of level l: z^(KZG_CHUNK^l) = z^(2^(5 l)), by squarings
__device__ __forceinline__ Fr kzg_level_mul(const uint64_t* z, int level) {
  Fr w = kzg_ld_fr(z);
#pragma unroll 1
  for (int i = 0; i < KZG_CHUNK_LOG * level; i++) w = fr_sqr(w);
  return w;
}

// Level l holds m rows of len entries (row j at x + 4 j len).  Thread t = j lc + c owns chunk c of row j, entries
// [c KZG_CHUNK, min(len, (c + 1) KZG_CHUNK)), and writes its Horner value sum_i x_i w^(i - c KZG_CHUNK) to entry t of level l + 1.
__global__ void __launch_bounds__(KZG_TPB) k_kzg_scan_up(const uint64_t* x, size_t len, size_t m, const uint64_t* z, int level, uint64_t* up) {
  const size_t lc = (len + KZG_CHUNK - 1) / KZG_CHUNK;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m * lc) return;
  const size_t j = t / lc, lo = (t - j * lc) * KZG_CHUNK, hi = lo + KZG_CHUNK < len ? lo + KZG_CHUNK : len;
  const Fr w = kzg_level_mul(z + 4 * j, level);
  const uint64_t* row = x + 4 * j * len;
  Fr acc = fr_zero();
#pragma unroll 1
  for (size_t i = hi; i-- > lo;) acc = fr_add(fr_mul(acc, w), kzg_ld_fr(row + 4 * i));
  kzg_st_fr(up + 4 * t, acc);
}

// The same chunks, run again from the carry s_(hi) -- entry c + 1 of level l + 1 after its own down pass, zero for the last
// chunk -- so that every entry becomes its suffix value s_i.  Levels >= 1 are overwritten in place (Q = false).  Level 0
// (Q = true) reads the coefficients and writes q_(i-1) = into_repr(s_i) at q[j (len - 1) + i - 1] and y_j = s_0.
template <bool Q>
__global__ void __launch_bounds__(KZG_TPB) k_kzg_scan_down(uint64_t* x, size_t len, size_t m, const uint64_t* z, int level, const uint64_t* up,
                                                           uint64_t* q, uint64_t* y) {
  const size_t lc = (len + KZG_CHUNK - 1) / KZG_CHUNK;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m * lc) return;
  const size_t j = t / lc, c = t - j * lc, lo = c * KZG_CHUNK, hi = lo + KZG_CHUNK < len ? lo + KZG_CHUNK : len;
  const Fr w = kzg_level_mul(z + 4 * j, level);
  uint64_t* row = x + 4 * j * len;
  Fr acc = c + 1 < lc ? kzg_ld_fr(up + 4 * (t + 1)) : fr_zero();
#pragma unroll 1
  for (size_t i = hi; i-- > lo;) {
    acc = fr_add(fr_mul(acc, w), kzg_ld_fr(row + 4 * i));
    if (!Q) kzg_st_fr(row + 4 * i, acc);
    else if (i > 0) kzg_st_fr(q + 4 * (j * (len - 1) + i - 1), kzg_into_repr(acc));
  }
  if (Q && lo == 0) kzg_st_fr(y + 4 * j, acc);
}

// normalised Jacobian rows (z = one, or z = 0 for the identity) -> affine rows (x, y, infinity = (z == 0))
__global__ void k_kzg_emit(const uint64_t* jac, size_t m, uint64_t* aff) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const uint64_t* src = jac + G1_W * t;
  uint64_t* dst = aff + G1A_W * t;
  uint64_t z = 0;
  for (int w = 0; w < 12; w++) dst[w] = src[w];
  for (int w = 12; w < 18; w++) z |= src[w];
  dst[12] = z == 0;
}

// ---- verify ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void kzg_jac_of(Jac<Fp>& p, const Aff<Fp>& a) {
  if (a.inf) pt_set_zero(p);
  else { p.x = a.x; p.y = a.y; f_set_one(p.z); }
}
__device__ __forceinline__ int kzg_bit(const Fr& k, int i) { return (k.v[i >> 5] >> (i & 31)) & 1u; }

// one thread per proof: pt[j] = C_j + (r - y_j) g + z_j pi_j (Jacobian) by one chain of doublings with the additions of
// g, pi_j or g + pi_j (Straus / Shamir), good[j] = y_j < r and z_j < r
__global__ void __launch_bounds__(KZG_TERM_TPB) k_kzg_term(const uint64_t* g, const uint64_t* c, const uint64_t* y, const uint64_t* z,
                                                           const uint64_t* pi, size_t m, uint64_t* pt, uint8_t* good) {
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const Fr yv = kzg_ld_fr(y + 4 * j), zv = kzg_ld_fr(z + 4 * j);
  good[j] = kzg_lt_r(yv) && kzg_lt_r(zv);
  const Fr a = fr_neg(kzg_into_repr(yv)), b = kzg_into_repr(zv);
  Aff<Fp> ga, pa, ca;
  ld_aff(ga, g);
  ld_aff(pa, pi + G1A_W * j);
  Jac<Fp> tg, tp, tgp, r;
  kzg_jac_of(tg, ga);
  kzg_jac_of(tp, pa);
  tgp = tg;
  pt_add(tgp, tp);
  pt_set_zero(r);
#pragma unroll 1
  for (int i = 254; i >= 0; i--) {                        // r < 2^255
    pt_double(r);
    const int sel = kzg_bit(a, i) | kzg_bit(b, i) << 1;
    if (sel) pt_add(r, sel == 1 ? tg : sel == 2 ? tp : tgp);
  }
  ld_aff(ca, c + G1A_W * j);
  pt_add_mixed(r, ca);
  st_jac(pt + G1_W * j, r);
}

__device__ __forceinline__ PLine kzg_line(const uint64_t* s, const uint64_t* p, bool dead) {
  PCoeffs c;
  c.c0 = ld_p2_smem(s); c.c1 = ld_p2_smem(s + 12); c.c2 = ld_p2_smem(s + 24);
  pcoeffs_set_one_if(dead, c);
  return p_line(c, ld_fp(p), ld_fp(p + 6));
}

// Lane pair i: ok[i] = good[i] && final_exponentiation(miller_loop([(P_i, h), (pi_i, -tau h)])) == one.  P_i is a normalised
// Jacobian row (infinity iff z == 0), pi_i an affine row.  Both G2 points are fixed: their prepared coefficients are staged
// once per block, and the loop does no G2 arithmetic -- one line-pair product per step, one squaring per bit.
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_PAIR_MINB) k_kzg_verify(const uint64_t* pvk, const uint64_t* pt, const uint64_t* pi,
                                                                           const uint8_t* good, size_t m, uint8_t* ok) {
  __shared__ __align__(128) uint64_t s_coeffs[2][68 * 36];
  __shared__ __align__(8) uint64_t s_bar;
  const uint32_t bar = smem_u32(&s_bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2 * KZG_COEFF_BYTES) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_coeffs[0])), "l"(pvk + KPVK_H), "r"(KZG_COEFF_BYTES), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_coeffs[1])), "l"(pvk + KPVK_NTH), "r"(KZG_COEFF_BYTES), "r"(bar) : "memory");
  }
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
  const bool active = i < m;
  if (!active) i = m - 1;
  const uint64_t* p = pt + G1_W * i;
  const uint64_t* w = pi + G1A_W * i;
  uint64_t pz = 0;
#pragma unroll
  for (int k = 12; k < 18; k++) pz |= p[k];
  const bool dead_p = pz == 0 || pvk[KPVK_H + G2P_W - 1] != 0;   // mod.rs:49-54: a pair with a member at infinity is skipped
  const bool dead_w = w[12] != 0 || pvk[KPVK_NTH + G2P_W - 1] != 0;
  mbar_wait_phase0(bar);
  P12 f;
  p12_one(f);
  int idx = 0;
#pragma unroll 1
  for (int bit = BLS_LOOP_TOP; bit >= -1; bit--) {       // bit == -1 is the trailing doubling step (mod.rs:92-94)
    const bool add = bit >= 0 && ((BLS_LOOP_BITS >> bit) & 1ull);
#pragma unroll 1
    for (int phase = 0; phase < (add ? 2 : 1); phase++) {
      p12_mul_by_line_pair(f, kzg_line(s_coeffs[0] + 36 * idx, p, dead_p), kzg_line(s_coeffs[1] + 36 * idx, w, dead_w));
      idx++;
    }
    if (bit >= 0) p12_sqr(f, f);
  }
  p12_conjugate(f);
  P12 e, one;
  const bool some = p_final_exponentiation(e, f);
  p12_one(one);
  const bool eq = p12_eq(e, one);
  if (active && pair_c() == 0) ok[i] = good[i] && some && eq;
}

// ---- the randomized check -------------------------------------------------------------------------------------------------
// one thread per proof: bases [C_0 .. C_(m-1), pi_0 .. pi_(m-1), g], scalars k[j] = rho_j, k[m + j] = rho_j z_j (mod r);
// *good = 0 when some y_j or z_j is not < r.  fr_mul(z R, rho) = z rho: the plain product.
__global__ void __launch_bounds__(KZG_TPB) k_kzg_rlc_scalars(const uint64_t* g, const uint64_t* c, const uint64_t* y, const uint64_t* z,
                                                             const uint64_t* pi, const uint64_t* rho, size_t m, uint64_t* bases, uint64_t* k,
                                                             uint8_t* good) {
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > m) return;
  if (j == m) {
    for (int w = 0; w < G1A_W; w++) bases[G1A_W * 2 * m + w] = g[w];
    return;
  }
  const Fr r = kzg_ld_fr(rho + 4 * j), zv = kzg_ld_fr(z + 4 * j);
  if (!kzg_lt_r(kzg_ld_fr(y + 4 * j)) || !kzg_lt_r(zv)) *good = 0;
  kzg_st_fr(k + 4 * j, r);
  kzg_st_fr(k + 4 * (m + j), fr_mul(zv, r));
  for (int w = 0; w < G1A_W; w++) bases[G1A_W * j + w] = c[G1A_W * j + w];
  for (int w = 0; w < G1A_W; w++) bases[G1A_W * (m + j) + w] = pi[G1A_W * j + w];
}

// one block: k[2m] = -sum_j rho_j y_j (mod r), canonical
__global__ void __launch_bounds__(KZG_SUM_TPB) k_kzg_rlc_sum(const uint64_t* y, const uint64_t* rho, size_t m, uint64_t* k) {
  __shared__ Fr part[KZG_SUM_TPB];
  Fr acc = fr_zero();
#pragma unroll 1
  for (size_t j = threadIdx.x; j < m; j += KZG_SUM_TPB) acc = fr_add(acc, fr_mul(kzg_ld_fr(y + 4 * j), kzg_ld_fr(rho + 4 * j)));
  part[threadIdx.x] = acc;
  __syncthreads();
#pragma unroll 1
  for (int h = KZG_SUM_TPB / 2; h >= 1; h >>= 1) {
    if (threadIdx.x < h) part[threadIdx.x] = fr_add(part[threadIdx.x], part[threadIdx.x + h]);
    __syncthreads();
  }
  if (threadIdx.x == 0) kzg_st_fr(k + 4 * 2 * m, fr_neg(part[0]));
}

// ---- host side ------------------------------------------------------------------------------------------------------------

static size_t kzg_align(size_t x) { return (x + 255) & ~(size_t)255; }

namespace {
struct KzgLayout {
  size_t off_k, off_lv[KZG_MAX_LEVELS], off_jac, off_work, total;   // commit / open
  size_t len[KZG_MAX_LEVELS];                                       // open: entries per row of each scan level
  int levels;
  size_t off_pt, off_good, off_bases, off_sums, off_w;              // verify / verify_rlc
};
}  // namespace

static bool kzg_args_ok(const bls_ctx* ctx, size_t n, size_t m) { return ctx && m <= KZG_MAX_M && n <= KZG_MAX_MN && m * n <= KZG_MAX_MN; }

// commit (open = false): the msm scalars, the m sums, the msm's work region.  open: the q_i (n - 1 per row), the scan
// levels 1.. (level 0 is p), the m sums, the msm's work region.  0 on failure.
static size_t kzg_layout(bls_ctx* ctx, size_t n, size_t m, bool open, KzgLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += kzg_align(bytes); return at; };
  const size_t nk = open ? (n ? n - 1 : 0) : n;
  l.off_k = take(m * nk * sizeof(bls_fr_repr));
  l.levels = 0;
  l.len[0] = n;
  if (open) {
    while (l.len[l.levels] > KZG_CHUNK) {
      l.len[l.levels + 1] = (l.len[l.levels] + KZG_CHUNK - 1) / KZG_CHUNK;
      l.levels++;
      l.off_lv[l.levels] = take(m * l.len[l.levels] * sizeof(bls_fr));
    }
  }
  l.off_jac = take(m * sizeof(bls_g1));
  const size_t work = bls_msm_batch_scratch_bytes(ctx, 1, nk, m, 0);
  if (!work) return 0;
  l.off_work = take(work);
  return l.total = o;
}
static size_t kzg_verify_layout(size_t m, KzgLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += kzg_align(bytes); return at; };
  l.off_pt = take(m * sizeof(bls_g1));
  l.off_good = take(m);
  l.off_work = take(bls_batch_normalization_scratch_bytes(nullptr, 1, m));
  return l.total = o;
}
static size_t kzg_rlc_layout(bls_ctx* ctx, size_t m, KzgLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += kzg_align(bytes); return at; };
  l.off_bases = take((2 * m + 1) * sizeof(bls_g1_affine));
  l.off_k = take((2 * m + 1) * sizeof(bls_fr_repr));
  l.off_sums = take(2 * sizeof(bls_g1));
  l.off_w = take(sizeof(bls_g1_affine));
  l.off_good = take(1);
  size_t work = 0;
  for (size_t n : {2 * m + 1, m}) {                                   // one region for each multiexp in turn
    const size_t b = bls_msm_scratch_bytes(ctx, 1, n, 0);
    if (!b) return 0;
    work = b > work ? b : work;
  }
  l.off_work = take(work);
  return l.total = o;
}

static int kzg_commit_dev_impl(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, size_t m, bls_g1_affine* c,
                               void* scratch, void* stream) {
  if (!kzg_args_ok(ctx, n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (srs_len < n || (n && (!srs || !p)) || !c || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_layout(ctx, n, m, false, l)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  bls_fr* k = (bls_fr*)(base + l.off_k);
  uint64_t* jac = (uint64_t*)(base + l.off_jac);
  if (n) TRY(bls_fr_op_dev(ctx, BLS_OP_INTO_REPR, p, nullptr, k, nullptr, m * n, st));
  TRY(bls_g1_msm_batch_dev(ctx, srs, 1, (const bls_fr_repr*)k, n, m, 0, (bls_g1*)jac, base + l.off_work, st));
  k_kzg_emit<<<blocks_for(m, KZG_TPB), KZG_TPB, 0, st>>>(jac, m, (uint64_t*)c);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int kzg_open_dev_impl(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, const bls_fr* z, size_t m,
                             bls_fr* y, bls_g1_affine* proof, void* scratch, void* stream) {
  if (!kzg_args_ok(ctx, n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (srs_len + 1 < n || (n > 1 && !srs) || (n && !p) || !z || !y || !proof || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_layout(ctx, n, m, true, l)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint64_t *q = at(l.off_k), *jac = at(l.off_jac);
  const uint64_t* zz = (const uint64_t*)z;
  auto level = [&](int i) { return i == 0 ? (uint64_t*)p : at(l.off_lv[i]); };
  if (n == 0) CK(cudaMemsetAsync(y, 0, m * sizeof(bls_fr), st));
  for (int i = 0; i < l.levels; i++) {
    k_kzg_scan_up<<<blocks_for(m * l.len[i + 1], KZG_TPB), KZG_TPB, 0, st>>>(level(i), l.len[i], m, zz, i, level(i + 1));
    LAUNCH_CHECK();
  }
  for (int i = l.levels; i >= 1; i--) {
    const uint64_t* up = i < l.levels ? level(i + 1) : nullptr;       // the top level is one chunk per row: no carry
    k_kzg_scan_down<false><<<blocks_for(m * ((l.len[i] + KZG_CHUNK - 1) / KZG_CHUNK), KZG_TPB), KZG_TPB, 0, st>>>(level(i), l.len[i], m, zz, i, up,
                                                                                                             nullptr, nullptr);
    LAUNCH_CHECK();
  }
  if (n) {
    k_kzg_scan_down<true><<<blocks_for(m * ((n + KZG_CHUNK - 1) / KZG_CHUNK), KZG_TPB), KZG_TPB, 0, st>>>((uint64_t*)p, n, m, zz, 0,
                                                                                                     l.levels ? level(1) : nullptr, q, (uint64_t*)y);
    LAUNCH_CHECK();
  }
  TRY(bls_g1_msm_batch_dev(ctx, srs, 1, (const bls_fr_repr*)q, n ? n - 1 : 0, m, 0, (bls_g1*)jac, base + l.off_work, st));
  k_kzg_emit<<<blocks_for(m, KZG_TPB), KZG_TPB, 0, st>>>(jac, m, (uint64_t*)proof);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int kzg_verify_dev_impl(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z,
                               const bls_g1_affine* proof, size_t m, uint8_t* ok, void* scratch, void* stream) {
  if (!ctx || m > KZG_VERIFY_MAX) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!pvk || ((uintptr_t)pvk & 15) || !c || !y || !z || !proof || !ok || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  kzg_verify_layout(m, l);
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  uint64_t* pt = (uint64_t*)(base + l.off_pt);
  uint8_t* good = (uint8_t*)(base + l.off_good);
  const uint64_t* vk = (const uint64_t*)pvk;
  k_kzg_term<<<blocks_for(m, KZG_TERM_TPB), KZG_TERM_TPB, 0, st>>>(vk + KPVK_G, (const uint64_t*)c, (const uint64_t*)y, (const uint64_t*)z,
                                                                   (const uint64_t*)proof, m, pt, good);
  LAUNCH_CHECK();
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)pt, m, base + l.off_work, st));
  k_kzg_verify<<<blocks_for(2 * m, BLS_PAIR_TPB), BLS_PAIR_TPB, 0, st>>>(vk, pt, (const uint64_t*)proof, good, m, ok);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int kzg_rlc_dev_impl(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z,
                            const bls_g1_affine* proof, const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream) {
  if (!ctx || m > KZG_RLC_MAX) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) {                                                   // the empty batch: FE(one) == one
    if (!ok1) return BLS_OK;
    USE_DEVICE(ctx);
    CK(cudaMemsetAsync(ok1, 1, 1, pick(ctx, stream)));
    return BLS_OK;
  }
  if (!pvk || ((uintptr_t)pvk & 15) || !c || !y || !z || !proof || !rho || !ok1 || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_rlc_layout(ctx, m, l)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint64_t *bases = at(l.off_bases), *k = at(l.off_k), *sums = at(l.off_sums), *w = at(l.off_w);
  uint8_t* good = (uint8_t*)at(l.off_good);
  const uint64_t* vk = (const uint64_t*)pvk;
  CK(cudaMemsetAsync(good, 1, 1, st));
  k_kzg_rlc_scalars<<<blocks_for(m + 1, KZG_TPB), KZG_TPB, 0, st>>>(vk + KPVK_G, (const uint64_t*)c, (const uint64_t*)y, (const uint64_t*)z,
                                                                   (const uint64_t*)proof, (const uint64_t*)rho, m, bases, k, good);
  LAUNCH_CHECK();
  k_kzg_rlc_sum<<<1, KZG_SUM_TPB, 0, st>>>((const uint64_t*)y, (const uint64_t*)rho, m, k);
  LAUNCH_CHECK();
  TRY(bls_g1_msm_dev(ctx, (const bls_g1_affine*)bases, (const bls_fr_repr*)k, 2 * m + 1, 0, (bls_g1*)sums, at(l.off_work), st));
  TRY(bls_g1_msm_dev(ctx, (const bls_g1_affine*)(bases + G1A_W * m), rho, m, 0, (bls_g1*)(sums + G1_W), at(l.off_work), st));
  k_kzg_emit<<<1, 32, 0, st>>>(sums + G1_W, 1, w);
  LAUNCH_CHECK();
  k_kzg_verify<<<1, BLS_PAIR_TPB, 0, st>>>(vk, sums, w, good, 1, ok1);
  LAUNCH_CHECK();
  return BLS_OK;
}

extern "C" {

size_t bls_kzg_commit_scratch_bytes(const bls_ctx* cctx, size_t n, size_t m) {
  if (!kzg_args_ok(cctx, n, m)) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  KzgLayout l;
  return kzg_layout(ctx, n, m, false, l);
}
int bls_kzg_commit_dev(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, size_t m, bls_g1_affine* c,
                       void* scratch, void* stream) {
  return kzg_commit_dev_impl(ctx, srs, srs_len, p, n, m, c, scratch, stream);
}
int bls_kzg_commit_batch(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, size_t m, bls_g1_affine* c) {
  if (!kzg_args_ok(ctx, n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (srs_len < n || (n && (!srs || !p)) || !c) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_layout(ctx, n, m, false, l)) return BLS_ERR_CUDA;
  H2D(dsrs, n ? srs : nullptr, n * sizeof(bls_g1_affine));
  H2D(dp, n ? p : nullptr, m * n * sizeof(bls_fr));
  DALLOC(dc, m * sizeof(bls_g1_affine));
  DALLOC(dscr, l.total);
  TRY(kzg_commit_dev_impl(ctx, (const bls_g1_affine*)dsrs.p, n, (const bls_fr*)dp.p, n, m, (bls_g1_affine*)dc.p, dscr.p, ctx->stream));
  D2H(c, dc, m * sizeof(bls_g1_affine));
  SYNC();
  return BLS_OK;
}

size_t bls_kzg_open_scratch_bytes(const bls_ctx* cctx, size_t n, size_t m) {
  if (!kzg_args_ok(cctx, n, m)) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  KzgLayout l;
  return kzg_layout(ctx, n, m, true, l);
}
int bls_kzg_open_dev(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, const bls_fr* z, size_t m, bls_fr* y,
                     bls_g1_affine* proof, void* scratch, void* stream) {
  return kzg_open_dev_impl(ctx, srs, srs_len, p, n, z, m, y, proof, scratch, stream);
}
int bls_kzg_open_batch(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, const bls_fr* z, size_t m, bls_fr* y,
                       bls_g1_affine* proof) {
  if (!kzg_args_ok(ctx, n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (srs_len + 1 < n || (n > 1 && !srs) || (n && !p) || !z || !y || !proof) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_layout(ctx, n, m, true, l)) return BLS_ERR_CUDA;
  const size_t nq = n ? n - 1 : 0;
  H2D(dsrs, nq ? srs : nullptr, nq * sizeof(bls_g1_affine));
  H2D(dp, n ? p : nullptr, m * n * sizeof(bls_fr));
  H2D(dz, z, m * sizeof(bls_fr));
  DALLOC(dy, m * sizeof(bls_fr));
  DALLOC(dpr, m * sizeof(bls_g1_affine));
  DALLOC(dscr, l.total);
  TRY(kzg_open_dev_impl(ctx, (const bls_g1_affine*)dsrs.p, nq, (const bls_fr*)dp.p, n, (const bls_fr*)dz.p, m, (bls_fr*)dy.p,
                        (bls_g1_affine*)dpr.p, dscr.p, ctx->stream));
  D2H(y, dy, m * sizeof(bls_fr));
  D2H(proof, dpr, m * sizeof(bls_g1_affine));
  SYNC();
  return BLS_OK;
}

int bls_kzg_prepare_verifying_key(bls_ctx* ctx, const bls_g1_affine* g, const bls_g2_affine* h, const bls_g2_affine* tau_h, bls_kzg_pvk* out) {
  if (!ctx || !g || !h || !tau_h || !out) return BLS_ERR_INVALID_ARGUMENT;
  bls_g2_affine q[2] = {*h, *tau_h};
  if (!q[1].infinity) {                                           // CurveAffine::negate: the identity stays as it is
    bls_fq2 ny;
    TRY(bls_field_op_batch(ctx, 2, BLS_OP_NEG, &q[1].y, nullptr, &ny, nullptr, 1));
    q[1].y = ny;
  }
  std::vector<bls_g2_prepared> prep(2);
  TRY(bls_g2_prepare_batch(ctx, q, prep.data(), 2));
  memset(out, 0, sizeof(*out));
  out->h_prepared = prep[0];
  out->neg_tau_h_prepared = prep[1];
  out->g = *g;
  out->h = q[0];
  out->neg_tau_h = q[1];
  return BLS_OK;
}

size_t bls_kzg_verify_scratch_bytes(const bls_ctx* ctx, size_t m) {
  if (!ctx || m > KZG_VERIFY_MAX) return 0;
  if (m == 0) return 1;
  KzgLayout l;
  return kzg_verify_layout(m, l);
}
int bls_kzg_verify_dev(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                       size_t m, uint8_t* ok, void* scratch, void* stream) {
  return kzg_verify_dev_impl(ctx, pvk, c, y, z, proof, m, ok, scratch, stream);
}
int bls_kzg_verify_batch(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                         size_t m, uint8_t* ok) {
  if (!ctx || m > KZG_VERIFY_MAX) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!pvk || !c || !y || !z || !proof || !ok) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  kzg_verify_layout(m, l);
  H2D(dpvk, pvk, sizeof(bls_kzg_pvk));                            // pool allocations are 256-byte aligned
  H2D(dc, c, m * sizeof(bls_g1_affine));
  H2D(dy, y, m * sizeof(bls_fr));
  H2D(dz, z, m * sizeof(bls_fr));
  H2D(dpr, proof, m * sizeof(bls_g1_affine));
  DALLOC(dok, m);
  DALLOC(dscr, l.total);
  TRY(kzg_verify_dev_impl(ctx, (const bls_kzg_pvk*)dpvk.p, (const bls_g1_affine*)dc.p, (const bls_fr*)dy.p, (const bls_fr*)dz.p,
                          (const bls_g1_affine*)dpr.p, m, (uint8_t*)dok.p, dscr.p, ctx->stream));
  D2H(ok, dok, m);
  SYNC();
  return BLS_OK;
}

size_t bls_kzg_verify_rlc_scratch_bytes(const bls_ctx* cctx, size_t m) {
  if (!cctx || m > KZG_RLC_MAX) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  KzgLayout l;
  return kzg_rlc_layout(ctx, m, l);
}
int bls_kzg_verify_rlc_dev(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z,
                           const bls_g1_affine* proof, const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream) {
  return kzg_rlc_dev_impl(ctx, pvk, c, y, z, proof, rho, m, ok1, scratch, stream);
}
int bls_kzg_verify_rlc_batch(bls_ctx* ctx, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z,
                             const bls_g1_affine* proof, const bls_fr_repr* rho, size_t m, uint8_t* ok1) {
  if (!ctx || m > KZG_RLC_MAX) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) {                                                   // the empty batch: the equation holds
    if (ok1) *ok1 = 1;
    return BLS_OK;
  }
  if (!pvk || !c || !y || !z || !proof || !rho || !ok1) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  KzgLayout l;
  if (!kzg_rlc_layout(ctx, m, l)) return BLS_ERR_CUDA;
  H2D(dpvk, pvk, sizeof(bls_kzg_pvk));
  H2D(dc, c, m * sizeof(bls_g1_affine));
  H2D(dy, y, m * sizeof(bls_fr));
  H2D(dz, z, m * sizeof(bls_fr));
  H2D(dpr, proof, m * sizeof(bls_g1_affine));
  H2D(drho, rho, m * sizeof(bls_fr_repr));
  DALLOC(dok, 1);
  DALLOC(dscr, l.total);
  TRY(kzg_rlc_dev_impl(ctx, (const bls_kzg_pvk*)dpvk.p, (const bls_g1_affine*)dc.p, (const bls_fr*)dy.p, (const bls_fr*)dz.p,
                       (const bls_g1_affine*)dpr.p, (const bls_fr_repr*)drho.p, m, (uint8_t*)dok.p, dscr.p, ctx->stream));
  D2H(ok1, dok, 1);
  SYNC();
  return BLS_OK;
}

}  // extern "C"
