// kernels_mm.cu -- the multi-pairing Miller loop on lane pairs (Engine::miller_loop over MANY pairs, bls12_381/mod.rs:40-102):
// one accumulator per lane pair, running G2 points in a scratch array, one partial product per block; and its device-pointer
// entry points.  Its own translation unit (see abi_common.cuh): the kernel keeps its accumulator and the Fq6 temporaries of the
// products in SHARED memory, and pointers into shared memory must not turn the local-memory accesses of the other kernels
// sharing these out-of-line tower routines into generic ones.
#include "pair_io.cuh"

// The odd pair left over by a trip sequence goes through p12_mul_by_line_pair(.., single) instead of mul_by_014 when the trip
// count is short (below BLS_MM_SINGLE_VIA_PAIR_BELOW): there the leftover is a seventh of the work and mul_by_014 -- code no other
// step of the loop executes -- costs 45 % more per product than the pair path (instruction-cache misses); for long trip counts the
// leftover is negligible and the cheaper 13-product path stays.
#define BLS_MM_SINGLE_VIA_PAIR_BELOW 32
#define BLS_MM_MINB 2      /* blocks per SM of the multi-pairing kernels; 3 (168 registers) measured 3.22 vs 4.87 M pairs/s at 2^20 */

// The accumulator f and the three Fq6 temporaries of the products that update it live in SHARED memory (181 words per lane: an
// odd stride, conflict-free 32-bit accesses; 92.7 KB per block, two blocks per SM) instead of the per-thread stack.
// Why here and not in the fused pairing kernel (DESIGN.md 8.1): this kernel streams 302 MB of running points through L2 per loop
// bit, next to 73 MB of stack that wants to stay there -- ncu showed 72 GB of the 113 GB of DRAM traffic per 2^20-pair launch to be
// evicted and re-fetched stack lines.
#define BLS_MM_SMEM_WORDS 181   /* P12 (72) + 3 x P6 (108) + 1 */
struct MmTmp { P6 a, b, s; };
// fq12.rs:34-48 x 2 (pair_tower.cuh: p12_mul_by_line_pair) with the temporaries supplied by the caller
static __device__ __noinline__ void mm_mul_by_line_pair(P12& f, MmTmp& t, const PLine& l, const PLine& m, bool single) {
  P6 lm0;              // (l m).c0
  P2 d1, d2;           // (l m).c1 = (0, d1, d2)
  if (!single) {
    P2 m00 = p2_mul(l.c0, m.c0), m11 = p2_mul(l.c1, m.c1), m44 = p2_mul(l.c4, m.c4);
    lm0.c1 = p2_sub(p2_sub(p2_mul(p2_add(l.c0, l.c1), p2_add(m.c0, m.c1)), m00), m11);
    d1 = p2_sub(p2_sub(p2_mul(p2_add(l.c0, l.c4), p2_add(m.c0, m.c4)), m00), m44);
    d2 = p2_sub(p2_sub(p2_mul(p2_add(l.c1, l.c4), p2_add(m.c1, m.c4)), m11), m44);
    lm0.c0 = p2_add(m00, p2_mul_by_nonresidue(m44));
    lm0.c2 = m11;
  } else {                                       // l * one
    lm0.c0 = l.c0; lm0.c1 = l.c1; lm0.c2 = p2_zero();
    d1 = l.c4; d2 = p2_zero();
  }
  p6_mul(t.a, f.c0, lm0);
  p6_mul_by_01(t.b, f.c1, d1, d2);               // f.c1 * (0, d1, d2) = v * (f.c1 * (d1, d2, 0))
  p6_mul_by_nonresidue(t.b, t.b);
  lm0.c1 = p2_add(lm0.c1, d1);                   // (l m).c0 + (l m).c1
  lm0.c2 = p2_add(lm0.c2, d2);
  p6_add(t.s, f.c1, f.c0);
  p6_mul(t.s, t.s, lm0);
  p6_sub(t.s, t.s, t.a);
  p6_sub(f.c1, t.s, t.b);
  p6_mul_by_nonresidue(t.b, t.b);
  p6_add(f.c0, t.b, t.a);
}
// fq12.rs:34-48
static __device__ __noinline__ void mm_mul_by_014(P12& f, MmTmp& t, const P2& c0, const P2& c1, const P2& c4) {
  p6_mul_by_01(t.a, f.c0, c0, c1);
  p6_mul_by_1(t.b, f.c1, c4);
  const P2 o = p2_add(c1, c4);
  p6_add(t.s, f.c1, f.c0);
  p6_mul_by_01(t.s, t.s, c0, o);
  p6_sub(t.s, t.s, t.a);
  p6_sub(f.c1, t.s, t.b);
  p6_mul_by_nonresidue(t.b, t.b);
  p6_add(f.c0, t.b, t.a);
}
// fq12.rs:99-114, in place
__device__ __forceinline__ void mm_sqr(P12& f, MmTmp& t) {
  p6_mul(t.a, f.c0, f.c1);                       // ab
  p6_add(t.b, f.c0, f.c1);                       // c0 + c1
  p6_mul_by_nonresidue(t.s, f.c1);
  p6_add(t.s, t.s, f.c0);
  p6_mul(t.s, t.s, t.b);
  p6_sub(t.s, t.s, t.a);
  p6_add(f.c1, t.a, t.a);
  p6_mul_by_nonresidue(t.a, t.a);
  p6_sub(f.c0, t.s, t.a);
}
extern __shared__ __align__(16) uint32_t mm_smem[];
#define MM_STATE(f, t)                                                                  \
  P12& f = *reinterpret_cast<P12*>(mm_smem + BLS_MM_SMEM_WORDS * threadIdx.x);          \
  MmTmp& t = *reinterpret_cast<MmTmp*>(mm_smem + BLS_MM_SMEM_WORDS * threadIdx.x + 72)
static size_t mm_smem_bytes() { return (size_t)BLS_MM_SMEM_WORDS * 4 * BLS_PAIR_TPB; }

// One partial product per BLOCK: the 64 lane pairs of a block fold their accumulators by a shared-memory tree (6 levels of
// Fq12 products) and lane pair 0 stores the result -- 296 partials per launch instead of 18 944, so that ONE small tail
// kernel (kernels_wide.cu: k_pair_product_tail) finishes the product.  Whole warps only: below 16 lane pairs the other lane
// pairs of warp 0 multiply along (every lane of a warp has to reach the shuffles inside p2_mul); their results are unused.
#define MM_LP (BLS_PAIR_TPB / 2)
__device__ __forceinline__ void mm_block_reduce_store(const P12& fin, uint64_t* partial) {
  P12 f = fin;                                         // off the shared state area, which the tree is about to reuse
  uint32_t* s_tree = mm_smem;                          // (MM_LP / 2) * 144 words = 18 KB of the 92.7 KB
  __syncthreads();
  const int lp = threadIdx.x >> 1;
#pragma unroll 1
  for (int s = MM_LP / 2; s >= 1; s >>= 1) {         // at level s the lane pairs [s, 2s) publish, the lane pairs [0, s) multiply
    __syncthreads();
    if (lp >= s && lp < 2 * s) {
      uint32_t* dst = s_tree + (lp - s) * 144 + pair_c() * 72;
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&f);
#pragma unroll
      for (int k = 0; k < 72; k++) dst[k] = w[k];
    }
    __syncthreads();
    if (lp < (s < 16 ? 16 : s)) {
      P12 x;
      const uint32_t* src = s_tree + lp * 144 + pair_c() * 72;
      uint32_t* w = reinterpret_cast<uint32_t*>(&x);
#pragma unroll
      for (int k = 0; k < 72; k++) w[k] = src[k];
      p12_mul(f, f, x);
    }
  }
  if (lp == 0) st_p12(partial, f);
}

// ONE miller_loop over n prepared pairs: lane pair t owns pairs t, t+T, ... and one accumulator (see k_pair_multi_miller)
__device__ __forceinline__ PLine mm_prepared_line(const uint64_t* p, const uint64_t* qp, size_t n, size_t i, int idx) {
  const bool in_range = i < n;
  if (!in_range) i = n - 1;
  const uint64_t* pi = p + G1A_W * i;
  const uint64_t* qi = qp + (size_t)G2P_W * i;
  const bool dead = !in_range || pi[12] != 0 || qi[G2P_W - 1] != 0;
  PCoeffs c;
  ld_pcoeffs(c, qi + 36 * idx);
  pcoeffs_set_one_if(dead, c);
  return p_line(c, ld_fp(pi), ld_fp(pi + 6));
}
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_MM_MINB) k_pair_multi_miller_prepared(const uint64_t* p, const uint64_t* qp, size_t n, uint64_t* partials) {
  const size_t T = ((size_t)gridDim.x * blockDim.x) >> 1;
  const size_t t = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
  const size_t per = (n + T - 1) / T;
  MM_STATE(f, tmp);
  p12_one(f);
  int idx = 0;
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= -1; b--) {
    const bool bit = b >= 0 && ((BLS_LOOP_BITS >> b) & 1ull);
#pragma unroll 1
    for (int rep = 0; rep < (bit ? 2 : 1); rep++) {
#pragma unroll 1
      for (size_t j = 0; j < per; j += 2) {          // two pairs at a time: see p12_mul_by_line_pair
        const PLine l = mm_prepared_line(p, qp, n, t + j * T, idx);
        if (j + 1 < per) mm_mul_by_line_pair(f, tmp, l, mm_prepared_line(p, qp, n, t + (j + 1) * T, idx), false);
        else if (per < BLS_MM_SINGLE_VIA_PAIR_BELOW) mm_mul_by_line_pair(f, tmp, l, l, true); else mm_mul_by_014(f, tmp, l.c0, l.c1, l.c4);
      }
      idx++;
    }
    if (b >= 0) mm_sqr(f, tmp);
  }
  p12_conjugate(f);
  mm_block_reduce_store(f, partials + FQ12_W * blockIdx.x);
}

// Lane-pair form of the multi-pairing Miller loop (the production path of bls_multi_miller_loop*):
// lane pair t owns pairs t, t+T, ... and ONE accumulator f.  Lane c keeps coefficient c of the running
// G2 point R_j in the scratch array `rstate` (layout: ld_pjac_blk).
// Every lane has to reach every shuffle, so there is no `continue`: a pair with an infinity member
// (mod.rs:49-54) or past the end of the batch multiplies f by the sparse element (1, 0, 0) = one instead,
// which leaves the canonical value of f unchanged.
// Scratch layout of the running points: blocks of 16 consecutive pairs (the 16 lane pairs of a warp work on 16 consecutive
// pairs in every trip: T is a multiple of 64), 36 lines of 128 bytes per block; line k holds word k of both coefficients
// of the 16 pairs in lane order, so every load / store instruction of a warp moves exactly one full line and a step
// touches one contiguous 4608-byte block.  (A word-major array over all n -- plane stride n words -- measured bimodal,
// 222 or 252 ms per 2^20 pairs from one process to the next.)
__host__ __device__ __forceinline__ size_t mm_rstate_words(size_t n) { return ((n + 15) / 16) * (36 * 32); }
__device__ __forceinline__ void ld_pjac_blk(PJac& r, const uint32_t* s, size_t pair) {
  uint32_t* w = reinterpret_cast<uint32_t*>(&r);
  const uint32_t* b = s + (pair >> 4) * (36 * 32) + 2 * (pair & 15) + pair_c();
#pragma unroll
  for (int k = 0; k < 36; k++) w[k] = b[k * 32];
}
__device__ __forceinline__ void st_pjac_blk(uint32_t* s, size_t pair, const PJac& r) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&r);
  uint32_t* b = s + (pair >> 4) * (36 * 32) + 2 * (pair & 15) + pair_c();
#pragma unroll
  for (int k = 0; k < 36; k++) b[k * 32] = w[k];
}
// one step (phase 0: doubling, phase 1: addition) of pair i's running point, and its line value at P_i
__device__ __forceinline__ PLine mm_step_line(const uint64_t* p, const uint64_t* q, size_t n, uint32_t* rstate, size_t i, int phase, int b) {
  const bool in_range = i < n;
  if (!in_range) i = n - 1;
  const uint64_t* pi = p + G1A_W * i;
  const uint64_t* qi = q + G2A_W * i;
  const bool dead = !in_range || pi[12] != 0 || qi[24] != 0;
  PJac r;
  PCoeffs c;
  if (phase == 0) {
    if (b == BLS_LOOP_TOP) { r.x = ld_p2(qi); r.y = ld_p2(qi + 12); r.z = p2_one(); }
    else ld_pjac_blk(r, rstate, i);
    pg2_doubling_step(r, c);
    if (b >= 0 && in_range) st_pjac_blk(rstate, i, r);
  } else {
    ld_pjac_blk(r, rstate, i);
    pg2_addition_step(r, ld_p2(qi), ld_p2(qi + 12), c);
    if (in_range) st_pjac_blk(rstate, i, r);
  }
  pcoeffs_set_one_if(dead, c);
  return p_line(c, ld_fp(pi), ld_fp(pi + 6));
}
__global__ void __launch_bounds__(BLS_PAIR_TPB, BLS_MM_MINB) k_pair_multi_miller(const uint64_t* p, const uint64_t* q, size_t n, uint32_t* rstate, uint64_t* partials) {
  const size_t T = ((size_t)gridDim.x * blockDim.x) >> 1;                       // lane pairs
  const size_t t = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
  const size_t per = (n + T - 1) / T;                                            // loop trips, uniform over the grid
  MM_STATE(f, tmp);
  p12_one(f);
#pragma unroll 1
  for (int b = BLS_LOOP_TOP; b >= -1; b--) {   // b == -1 is the trailing doubling step (mod.rs:92-94)
    const bool bit = b >= 0 && ((BLS_LOOP_BITS >> b) & 1ull);
#pragma unroll 1
    for (int phase = 0; phase < (bit ? 2 : 1); phase++) {
#pragma unroll 1
      for (size_t j = 0; j < per; j += 2) {          // two pairs at a time: see p12_mul_by_line_pair
        const PLine l = mm_step_line(p, q, n, rstate, t + j * T, phase, b);
        if (j + 1 < per) mm_mul_by_line_pair(f, tmp, l, mm_step_line(p, q, n, rstate, t + (j + 1) * T, phase, b), false);
        else if (per < BLS_MM_SINGLE_VIA_PAIR_BELOW) mm_mul_by_line_pair(f, tmp, l, l, true); else mm_mul_by_014(f, tmp, l.c0, l.c1, l.c4);
      }
    }
    if (b >= 0) mm_sqr(f, tmp);
  }
  p12_conjugate(f);
  mm_block_reduce_store(f, partials + FQ12_W * blockIdx.x);
}

// more than 48 KB of dynamic shared memory per block needs an opt-in per function and per DEVICE: once per context
static cudaError_t mm_smem_optin(bls_ctx* ctx) {
  if (ctx->mm_smem_ready) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(k_pair_multi_miller, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mm_smem_bytes());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_pair_multi_miller_prepared, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mm_smem_bytes());
  ctx->mm_smem_ready = e == cudaSuccess;
  return e;
}

extern "C" {

// lane pairs (= partial products) used by the multi-Miller kernel for n pairs: enough pairs per lane pair to
// amortise the shared squarings, never more lane pairs than pairs; a multiple of the 64 lane pairs of a block
static size_t mm_threads(const bls_ctx* ctx, size_t n) {
  const size_t per_block = BLS_PAIR_TPB / 2;
  size_t full = (size_t)ctx->sm_count * BLS_MM_MINB * per_block;
  size_t t = n < full ? n : full;
  t = (t + per_block - 1) / per_block * per_block;
  return t ? t : per_block;
}
// Products of at most this many pairs run their Miller loops one WARP per pair (kernels_wide.cu: k_wide_miller, ~1 ms) instead of one
// lane pair per pair (4.5 ms of latency): the signature-verification shape -- a product of two or a few pairings -- is latency-bound.
// Follows the context's latency-path limit for pairings, capped here because the single-block tail folds the values serially
// (47 us per 64 values).
#define BLS_WIDE_PRODUCT_CAP 1024
static size_t mm_wide_limit(const bls_ctx* ctx) { return ctx->wide_pairing_max < BLS_WIDE_PRODUCT_CAP ? ctx->wide_pairing_max : BLS_WIDE_PRODUCT_CAP; }
size_t bls_multi_miller_scratch_bytes(const bls_ctx* ctx, size_t n) {
  if (!ctx) return 0;
  size_t T = mm_threads(ctx, n);
  size_t bytes = mm_rstate_words(n) * sizeof(uint32_t) + (T / MM_LP) * sizeof(bls_fq12);
  const size_t wide = (n <= BLS_WIDE_PRODUCT_CAP ? n : 0) * sizeof(bls_fq12);      // one Miller value per pair on the latency path
  return bytes > wide ? bytes : wide;
}

// mod.rs:40-102 over ONE n-pair call: the Miller kernel leaves one partial product per block, the tail kernel folds them
// (and, for bls_pairing_product_dev, runs the single final exponentiation on the warp-cooperative engine)
static int multi_miller_impl(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, void* scratch, void* stream, int final_exp, uint8_t* is_some) {
  if (!ctx || !out1 || (n && (!p || !q || !scratch))) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t s = pick(ctx, stream);
  if (n == 0) return bls_internal_product_tail(ctx, nullptr, 0, out1, final_exp, is_some, s);   // the empty product: one
  if (n <= mm_wide_limit(ctx)) {                                                                // latency path: one warp per pair, then the tail
    TRY(bls_internal_wide_miller(ctx, p, q, (bls_fq12*)scratch, n, s));
    return bls_internal_product_tail(ctx, (const bls_fq12*)scratch, n, out1, final_exp, is_some, s);
  }
  size_t T = mm_threads(ctx, n);
  uint32_t* rstate = (uint32_t*)scratch;
  uint64_t* partials = (uint64_t*)((char*)scratch + mm_rstate_words(n) * sizeof(uint32_t));
  CK(mm_smem_optin(ctx));
  k_pair_multi_miller<<<(unsigned)(T / MM_LP), BLS_PAIR_TPB, mm_smem_bytes(), s>>>((const uint64_t*)p, (const uint64_t*)q, n, rstate, partials);
  LAUNCH_CHECK();
  return bls_internal_product_tail(ctx, (const bls_fq12*)partials, T / MM_LP, out1, final_exp, is_some, s);
}
int bls_multi_miller_loop_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, void* scratch, void* stream) {
  return multi_miller_impl(ctx, p, q, n, out1, scratch, stream, 0, nullptr);
}
int bls_pairing_product_dev(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, uint8_t* is_some, void* scratch, void* stream) {
  return multi_miller_impl(ctx, p, q, n, out1, scratch, stream, 1, is_some);
}
}  // extern "C"

size_t bls_internal_mm_lane_pairs(const bls_ctx* ctx, size_t n) { return mm_threads(ctx, n) / MM_LP; }   // = partial products (one per block)
int bls_internal_multi_miller_prepared(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* qp, size_t n, bls_fq12* partials, cudaStream_t s) {
  const size_t T = mm_threads(ctx, n);
  CK(mm_smem_optin(ctx));
  k_pair_multi_miller_prepared<<<(unsigned)(T / MM_LP), BLS_PAIR_TPB, mm_smem_bytes(), s>>>((const uint64_t*)p, (const uint64_t*)qp, n, (uint64_t*)partials);
  LAUNCH_CHECK();
  return BLS_OK;
}
