// kernels_groth16.cu -- bellman's groth16::create_proof for m proofs of one circuit (bls_groth16_prove_*).  Its own
// translation unit (see abi_common.cuh): the transforms and the multiexps are the other units' entry points, called through
// the C ABI, so no existing kernel is recompiled.  The group law is curve.cuh's, unchanged.
//
// Pipeline, all on the call's stream:
//   1. bls_fr_groth16_h_dev: H, m * (n - 1) FrRepr.
//   2. k_groth16_gather: one thread per (proof, variable): into_repr of input_i / aux_i to its compacted place in
//      sa (the a query's scalars), sb (b_g1 and b_g2) and sl (l).  rank_D(i) = prefix[i / 32] + popc(word & below(i)); the
//      exclusive word prefixes come with the bitmap words, computed on the host in the pass that counts the set bits.
//   3. five bls_g*_msm_batch_dev calls with shared bases: (h, H), (l, sl), (a, sa), (b_g1, sb) in G1, (b_g2, sb) in G2.
//   4. k_groth16_mul: one thread per (proof, scalar multiplication), double-and-add (pt_mul): r delta_g1, (r s) delta_g1,
//      s (alpha_g1 + a_ans), r (beta_g1 + b1_ans) in G1 and s delta_g2 in G2, the G2 products in the grid's second row so
//      both run at once.  bellman's g_c = rs delta_g1 + s alpha_g1 + r beta_g1 + s a_ans + r b1_ans + h + l, regrouped so
//      that the four G1 products are independent.
//   5. k_groth16_assemble: one thread per proof: the sums of A, B and C, pt_into_affine, the bls_groth16_proof row.
#include "curve_io.cuh"
#include "fr.cuh"

#include <vector>

#define G16_TPB 128
#define G16_TAIL_TPB 32                   /* the tail kernels run single-thread chains: spread them over the SMs */
#define G16_MAX_M ((size_t)1 << 16)
#define G16_MAX_MN ((size_t)1 << 26)      /* m * (each multiexp's length): bls_g*_msm_batch_dev's limit */

// the vk points in scratch, u64 offsets: alpha_g1, beta_g1, delta_g1, beta_g2, delta_g2 (bls_g*_affine rows)
#define G16_ALPHA 0
#define G16_BETA1 G1A_W
#define G16_DELTA1 (2 * G1A_W)
#define G16_BETA (3 * G1A_W)
#define G16_DELTA2 (3 * G1A_W + G2A_W)
#define G16_VK_W (3 * G1A_W + 2 * G2A_W)

__device__ __forceinline__ Fr g16_ld_fr(const uint64_t* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void g16_st_fr(uint64_t* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
// into_repr(): the Montgomery product with 1
__device__ __forceinline__ Fr g16_into_repr(const Fr& x) {
  Fr one = fr_zero();
  one.v[0] = 1;
  return fr_mul(x, one);
}
// rank_D(i) and bit i of D; bm holds (word, exclusive prefix of the word popcounts) pairs
__device__ __forceinline__ Scalar g16_scalar(const Fr& k) {
  Scalar r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = k.v[i];
  return r;
}
__device__ __forceinline__ bool g16_bit(const uint2* bm, size_t i, uint32_t& rank) {
  const uint2 w = bm[i >> 5];
  const uint32_t below = (1u << (i & 31)) - 1u;
  rank = w.y + __popc(w.x & below);
  return (w.x >> (i & 31)) & 1u;
}

// t = j (ni + na) + v: variable v of proof j, v < ni an input, else aux v - ni
__global__ void __launch_bounds__(G16_TPB) k_groth16_gather(const uint64_t* input, const uint64_t* aux, size_t ni, size_t na, size_t m,
                                                            const uint2* a_aux, const uint2* b_in, const uint2* b_aux, uint32_t pop_b_in,
                                                            size_t la, size_t lb, uint64_t* sa, uint64_t* sb, uint64_t* sl) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nv = ni + na;
  if (t >= m * nv) return;
  const size_t j = t / nv, v = t - j * nv;
  uint32_t rank;
  if (v < ni) {
    const Fr x = g16_into_repr(g16_ld_fr(input + 4 * (j * ni + v)));
    g16_st_fr(sa + 4 * (j * la + v), x);
    if (g16_bit(b_in, v, rank)) g16_st_fr(sb + 4 * (j * lb + rank), x);
    return;
  }
  const size_t i = v - ni;
  const Fr x = g16_into_repr(g16_ld_fr(aux + 4 * (j * na + i)));
  g16_st_fr(sl + 4 * (j * na + i), x);
  if (g16_bit(a_aux, i, rank)) g16_st_fr(sa + 4 * (j * la + ni + rank), x);
  if (g16_bit(b_aux, i, rank)) g16_st_fr(sb + 4 * (j * lb + pop_b_in + rank), x);
}

// blockIdx.y = 0: t = 4 j + q, G1 product q of proof j into prod1[t]: r delta_g1, (r s) delta_g1, s (alpha_g1 + a_ans),
// r (beta_g1 + b1_ans);
// blockIdx.y = 1: t = j, s delta_g2 into prod2[j].  a_ans and b1_ans are the normalised Jacobian sums of the multiexps.
__global__ void __launch_bounds__(G16_TAIL_TPB) k_groth16_mul(const uint64_t* vk, const uint64_t* r, const uint64_t* s, const uint64_t* a_ans,
                                                              const uint64_t* b1_ans, size_t m, uint64_t* prod1, uint64_t* prod2) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 1) {
    if (t >= m) return;
    Aff<Fp2> d;
    ld_aff(d, vk + G16_DELTA2);
    Jac<Fp2> p;
    p.x = d.x; p.y = d.y; f_set_one(p.z);                // delta_g2 is not infinity (checked on the host)
    const Fr k = g16_into_repr(g16_ld_fr(s + 4 * t));
    pt_mul(p, g16_scalar(k));
    st_jac(prod2 + (size_t)G2_W * t, p);
    return;
  }
  if (t >= 4 * m) return;
  const size_t j = t >> 2;
  const int q = (int)(t & 3);
  const Fr fr_r = g16_ld_fr(r + 4 * j), fr_s = g16_ld_fr(s + 4 * j);
  Fr k;
  Jac<Fp> p;
  if (q < 2) {
    Aff<Fp> d;
    ld_aff(d, vk + G16_DELTA1);
    p.x = d.x; p.y = d.y; f_set_one(p.z);
    k = q == 0 ? fr_r : fr_mul(fr_r, fr_s);
  } else {
    Aff<Fp> o;
    ld_jac(p, (q == 2 ? a_ans : b1_ans) + (size_t)G1_W * j);
    ld_aff(o, vk + (q == 2 ? G16_ALPHA : G16_BETA1));
    pt_add_mixed(p, o);
    k = q == 2 ? fr_s : fr_r;
  }
  k = g16_into_repr(k);
  pt_mul(p, g16_scalar(k));
  st_jac(prod1 + (size_t)G1_W * t, p);
}

// one thread per proof: A = r delta_g1 + alpha_g1 + a_ans, B = s delta_g2 + beta_g2 + b2_ans,
// C = (r s) delta_g1 + s (alpha_g1 + a_ans) + r (beta_g1 + b1_ans) + h_ans + l_ans, each stored as bellman's into_affine()
__global__ void __launch_bounds__(G16_TAIL_TPB) k_groth16_assemble(const uint64_t* vk, const uint64_t* prod1, const uint64_t* prod2, const uint64_t* h_ans,
                                                                   const uint64_t* l_ans, const uint64_t* a_ans, const uint64_t* b2_ans, size_t m,
                                                                   uint64_t* out) {
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const size_t PW = sizeof(bls_groth16_proof) / 8;
  uint64_t* row = out + PW * j;
  const uint64_t* p1 = prod1 + (size_t)G1_W * 4 * j;
  Jac<Fp> acc, x;
  Aff<Fp> a1;
  ld_jac(acc, p1);
  ld_aff(a1, vk + G16_ALPHA);
  pt_add_mixed(acc, a1);
  ld_jac(x, a_ans + (size_t)G1_W * j);
  pt_add(acc, x);
  pt_into_affine(a1, acc);
  st_aff(row, a1);

  Jac<Fp2> acc2, x2;
  Aff<Fp2> a2;
  ld_jac(acc2, prod2 + (size_t)G2_W * j);
  ld_aff(a2, vk + G16_BETA);
  pt_add_mixed(acc2, a2);
  ld_jac(x2, b2_ans + (size_t)G2_W * j);
  pt_add(acc2, x2);
  pt_into_affine(a2, acc2);
  st_aff(row + G1A_W, a2);

  ld_jac(acc, p1 + G1_W);
#pragma unroll 1
  for (int q = 2; q < 4; q++) {
    ld_jac(x, p1 + G1_W * q);
    pt_add(acc, x);
  }
  ld_jac(x, h_ans + (size_t)G1_W * j);
  pt_add(acc, x);
  ld_jac(x, l_ans + (size_t)G1_W * j);
  pt_add(acc, x);
  pt_into_affine(a1, acc);
  st_aff(row + G1A_W + G2A_W, a1);
}

// ---- host side ----------------------------------------------------------------------------------------------------------

static size_t g16_align(size_t x) { return (x + 255) & ~(size_t)255; }
static size_t g16_words(size_t bits) { return (bits + 31) / 32; }

namespace {
// The shape of one call, from the arguments and the popcounts of the density bitmaps.
struct G16Plan {
  size_t n1;                                     // n - 1: H's coefficients per proof
  size_t la, lb, pop_b_in;                       // the a and b multiexp lengths, popcount(b_input_density)
  size_t w_a, w_bi, w_ba;                        // words of the three bitmaps
  size_t off_up, off_sums, off_prod1, off_prod2, off_h, off_sa, off_sb, off_sl, off_work, total;
};
}  // namespace

// word i of a bitmap of `bits` bits, the bits past the end cleared
static uint32_t g16_word(const uint32_t* d, size_t bits, size_t i) {
  const size_t rest = bits - 32 * i;
  return rest >= 32 ? d[i] : d[i] & ((1u << rest) - 1u);
}
static size_t g16_popcount(const uint32_t* d, size_t bits) {
  size_t c = 0;
  for (size_t i = 0; i < g16_words(bits); i++) c += (size_t)__builtin_popcount(g16_word(d, bits, i));
  return c;
}

// argument checks (no device work) and, when they pass, the plan without the scratch offsets
static bool g16_args_ok(const bls_ctx* ctx, const bls_groth16_params* pp, size_t len, size_t ni, size_t na, const uint32_t* a_aux,
                        const uint32_t* b_in, const uint32_t* b_aux, size_t m, G16Plan& p) {
  if (!ctx || !pp || m > G16_MAX_M || len > G16_MAX_MN || ni + na > G16_MAX_MN) return false;
  if (pp->delta_g1.infinity || pp->delta_g2.infinity) return false;
  if ((na && (!a_aux || !b_aux)) || (ni && !b_in)) return false;
  size_t n = 1;
  while (n < len) n <<= 1;
  p.n1 = n - 1;
  p.pop_b_in = ni ? g16_popcount(b_in, ni) : 0;
  p.la = ni + (na ? g16_popcount(a_aux, na) : 0);
  p.lb = p.pop_b_in + (na ? g16_popcount(b_aux, na) : 0);
  if (pp->h_len < p.n1 || pp->l_len < na || pp->a_len < p.la || pp->b_len < p.lb) return false;
  for (size_t l : {p.n1, na, p.la, p.lb})
    if (l > G16_MAX_MN || m * l > G16_MAX_MN) return false;
  if (p.n1 && !pp->h) return false;
  if (na && !pp->l) return false;
  if (p.la && !pp->a) return false;
  if (p.lb && (!pp->b_g1 || !pp->b_g2)) return false;
  p.w_a = g16_words(na);
  p.w_bi = g16_words(ni);
  p.w_ba = g16_words(na);
  return true;
}

// scratch layout: the vk points and the bitmap (word, prefix) pairs, the five multiexp sums, the products of k_groth16_mul, the scalars H, sa, sb,
// sl, then one work region that serves H's transforms and then each multiexp in turn.  0 on failure.
static size_t g16_layout(bls_ctx* ctx, size_t len, size_t na, size_t m, G16Plan& p) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += g16_align(bytes); return at; };
  p.off_up = take((G16_VK_W + p.w_a + p.w_bi + p.w_ba) * sizeof(uint64_t));
  p.off_sums = take(m * (4 * sizeof(bls_g1) + sizeof(bls_g2)));
  p.off_prod1 = take(4 * m * sizeof(bls_g1));
  p.off_prod2 = take(m * sizeof(bls_g2));
  p.off_h = take(m * p.n1 * sizeof(bls_fr_repr));
  p.off_sa = take(m * p.la * sizeof(bls_fr_repr));
  p.off_sb = take(m * p.lb * sizeof(bls_fr_repr));
  p.off_sl = take(m * na * sizeof(bls_fr_repr));
  size_t work = len > 1 ? bls_fr_groth16_h_scratch_bytes(ctx, len, m) : 1;
  const size_t need[5][2] = {{1, p.n1}, {1, na}, {1, p.la}, {1, p.lb}, {2, p.lb}};
  for (const auto& d : need) {
    const size_t b = bls_msm_batch_scratch_bytes(ctx, (int)d[0], d[1], m, 0);
    if (!b) return 0;
    work = b > work ? b : work;
  }
  if (!work) return 0;
  p.off_work = take(work);
  p.total = o;
  return o;
}

static int g16_dev_impl(bls_ctx* ctx, const bls_groth16_params* pp, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                        const bls_fr* input, size_t ni, const bls_fr* aux, size_t na, const uint32_t* a_aux, const uint32_t* b_in,
                        const uint32_t* b_aux, const bls_fr* r, const bls_fr* s, size_t m, bls_groth16_proof* out, void* scratch, void* stream) {
  G16Plan p;
  if (!g16_args_ok(ctx, pp, len, ni, na, a_aux, b_in, b_aux, m, p)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!out || !r || !s || !scratch || (p.n1 && (!a || !b || !c)) || (ni && !input) || (na && !aux)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!g16_layout(ctx, len, na, m, p)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };

  // the vk points, then every bitmap word with the exclusive prefix of the word popcounts as one u64 (an uint2 on the
  // device).  One copy; a pageable source has been staged when cudaMemcpyAsync returns, so `up` may go out of scope.
  std::vector<uint64_t> up(G16_VK_W + p.w_a + p.w_bi + p.w_ba);
  memcpy(up.data() + G16_ALPHA, &pp->alpha_g1, sizeof(bls_g1_affine));
  memcpy(up.data() + G16_BETA1, &pp->beta_g1, sizeof(bls_g1_affine));
  memcpy(up.data() + G16_DELTA1, &pp->delta_g1, sizeof(bls_g1_affine));
  memcpy(up.data() + G16_BETA, &pp->beta_g2, sizeof(bls_g2_affine));
  memcpy(up.data() + G16_DELTA2, &pp->delta_g2, sizeof(bls_g2_affine));
  auto pack = [&](const uint32_t* d, size_t bits, uint64_t* dst) {
    uint32_t acc = 0;
    for (size_t i = 0; i < g16_words(bits); i++) {
      const uint32_t w = g16_word(d, bits, i);
      dst[i] = w | (uint64_t)acc << 32;
      acc += (uint32_t)__builtin_popcount(w);
    }
  };
  pack(a_aux, na, up.data() + G16_VK_W);
  pack(b_in, ni, up.data() + G16_VK_W + p.w_a);
  pack(b_aux, na, up.data() + G16_VK_W + p.w_a + p.w_bi);
  CK(cudaMemcpyAsync(base + p.off_up, up.data(), up.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  const uint64_t* vk = at(p.off_up);
  const uint2* d_bm = (const uint2*)(vk + G16_VK_W);

  uint64_t *h = at(p.off_h), *sa = at(p.off_sa), *sb = at(p.off_sb), *sl = at(p.off_sl), *sums = at(p.off_sums);
  uint64_t *h_ans = sums, *l_ans = h_ans + G1_W * m, *a_ans = l_ans + G1_W * m, *b1_ans = a_ans + G1_W * m, *b2_ans = b1_ans + G1_W * m;
  void* work = base + p.off_work;
  TRY(bls_fr_groth16_h_dev(ctx, a, b, c, len, m, (bls_fr_repr*)h, work, st));
  if (ni + na) {
    k_groth16_gather<<<blocks_for(m * (ni + na), G16_TPB), G16_TPB, 0, st>>>((const uint64_t*)input, (const uint64_t*)aux, ni, na, m, d_bm,
                                                                             d_bm + p.w_a, d_bm + p.w_a + p.w_bi, (uint32_t)p.pop_b_in,
                                                                             p.la, p.lb, sa, sb, sl);
    LAUNCH_CHECK();
  }
  TRY(bls_g1_msm_batch_dev(ctx, pp->h, 1, (const bls_fr_repr*)h, p.n1, m, 0, (bls_g1*)h_ans, work, st));
  TRY(bls_g1_msm_batch_dev(ctx, pp->l, 1, (const bls_fr_repr*)sl, na, m, 0, (bls_g1*)l_ans, work, st));
  TRY(bls_g1_msm_batch_dev(ctx, pp->a, 1, (const bls_fr_repr*)sa, p.la, m, 0, (bls_g1*)a_ans, work, st));
  TRY(bls_g1_msm_batch_dev(ctx, pp->b_g1, 1, (const bls_fr_repr*)sb, p.lb, m, 0, (bls_g1*)b1_ans, work, st));
  TRY(bls_g2_msm_batch_dev(ctx, pp->b_g2, 1, (const bls_fr_repr*)sb, p.lb, m, 0, (bls_g2*)b2_ans, work, st));

  uint64_t *prod1 = at(p.off_prod1), *prod2 = at(p.off_prod2);
  k_groth16_mul<<<dim3(blocks_for(4 * m, G16_TAIL_TPB), 2), G16_TAIL_TPB, 0, st>>>(vk, (const uint64_t*)r, (const uint64_t*)s, a_ans, b1_ans, m,
                                                                                   prod1, prod2);
  LAUNCH_CHECK();
  k_groth16_assemble<<<blocks_for(m, G16_TAIL_TPB), G16_TAIL_TPB, 0, st>>>(vk, prod1, prod2, h_ans, l_ans, a_ans, b2_ans, m, (uint64_t*)out);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int g16_host(bls_ctx* ctx, const bls_groth16_params* pp, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                    const bls_fr* input, size_t ni, const bls_fr* aux, size_t na, const uint32_t* a_aux, const uint32_t* b_in,
                    const uint32_t* b_aux, const bls_fr* r, const bls_fr* s, size_t m, bls_groth16_proof* out) {
  G16Plan p;
  if (!g16_args_ok(ctx, pp, len, ni, na, a_aux, b_in, b_aux, m, p)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!out || !r || !s || (p.n1 && (!a || !b || !c)) || (ni && !input) || (na && !aux)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!g16_layout(ctx, len, na, m, p)) return BLS_ERR_CUDA;
  const size_t fb = sizeof(bls_fr), ga = sizeof(bls_g1_affine), g2a = sizeof(bls_g2_affine);
  const bool h_in = p.n1 != 0;
  H2D(da, h_in ? a : nullptr, h_in ? m * len * fb : 1);
  H2D(db, h_in ? b : nullptr, h_in ? m * len * fb : 1);
  H2D(dc, h_in ? c : nullptr, h_in ? m * len * fb : 1);
  H2D(din, ni ? input : nullptr, m * ni * fb);
  H2D(daux, na ? aux : nullptr, m * na * fb);
  H2D(dr, r, m * fb);
  H2D(ds, s, m * fb);
  H2D(qh, p.n1 ? pp->h : nullptr, p.n1 * ga);                   // the used prefix of every query
  H2D(ql, na ? pp->l : nullptr, na * ga);
  H2D(qa, p.la ? pp->a : nullptr, p.la * ga);
  H2D(qb1, p.lb ? pp->b_g1 : nullptr, p.lb * ga);
  H2D(qb2, p.lb ? pp->b_g2 : nullptr, p.lb * g2a);
  DALLOC(dout, m * sizeof(bls_groth16_proof));
  DALLOC(dscr, p.total);
  bls_groth16_params dp = *pp;
  dp.h = (const bls_g1_affine*)qh.p; dp.l = (const bls_g1_affine*)ql.p; dp.a = (const bls_g1_affine*)qa.p;
  dp.b_g1 = (const bls_g1_affine*)qb1.p; dp.b_g2 = (const bls_g2_affine*)qb2.p;
  TRY(g16_dev_impl(ctx, &dp, (const bls_fr*)da.p, (const bls_fr*)db.p, (const bls_fr*)dc.p, len, (const bls_fr*)din.p, ni, (const bls_fr*)daux.p, na,
                   a_aux, b_in, b_aux, (const bls_fr*)dr.p, (const bls_fr*)ds.p, m, (bls_groth16_proof*)dout.p, dscr.p, ctx->stream));
  D2H(out, dout, m * sizeof(bls_groth16_proof));
  SYNC();
  return BLS_OK;
}

extern "C" {

size_t bls_groth16_prove_scratch_bytes(const bls_ctx* cctx, const bls_groth16_params* pp, size_t len, size_t num_inputs, size_t num_aux,
                                       const uint32_t* a_aux_density, const uint32_t* b_input_density, const uint32_t* b_aux_density, size_t m) {
  G16Plan p;
  if (!g16_args_ok(cctx, pp, len, num_inputs, num_aux, a_aux_density, b_input_density, b_aux_density, m, p)) return 0;
  if (m == 0) return 1;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  return g16_layout(ctx, len, num_aux, m, p);
}
int bls_groth16_prove_dev(bls_ctx* ctx, const bls_groth16_params* params, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                          const bls_fr* input, size_t num_inputs, const bls_fr* aux, size_t num_aux, const uint32_t* a_aux_density,
                          const uint32_t* b_input_density, const uint32_t* b_aux_density, const bls_fr* r, const bls_fr* s, size_t m,
                          bls_groth16_proof* out, void* scratch, void* stream) {
  return g16_dev_impl(ctx, params, a, b, c, len, input, num_inputs, aux, num_aux, a_aux_density, b_input_density, b_aux_density, r, s, m, out,
                      scratch, stream);
}
int bls_groth16_prove_batch(bls_ctx* ctx, const bls_groth16_params* params, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                            const bls_fr* input, size_t num_inputs, const bls_fr* aux, size_t num_aux, const uint32_t* a_aux_density,
                            const uint32_t* b_input_density, const uint32_t* b_aux_density, const bls_fr* r, const bls_fr* s, size_t m,
                            bls_groth16_proof* out) {
  return g16_host(ctx, params, a, b, c, len, input, num_inputs, aux, num_aux, a_aux_density, b_input_density, b_aux_density, r, s, m, out);
}

}  // extern "C"
