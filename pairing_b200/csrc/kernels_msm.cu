// kernels_msm.cu -- multi-scalar multiplication S = sum_i k_i * P_i over affine bases in G1 and G2 by the bucket (Pippenger)
// method, and its entry points.  Its own translation unit (see abi_common.cuh) so that ptxas' allocation of the existing
// curve kernels cannot move.  The group law is curve.cuh's, unchanged: pt_add_mixed / pt_add / pt_double / pt_into_affine.
//
// One call computes m independent sums of n points (m = 1: bls_g*_msm).  Pipeline for a c-bit window (W = ceil(257 / c)
// windows per sum, B = 2^(c-1) buckets per window); the m * W (sum, window) pairs are the "windows" of steps 2-4:
//   1. k_msm_recode: signed c-bit digits in [-2^(c-1), 2^(c-1)] per scalar; one (key, base index | sign) entry per (sum j,
//      window w, point i) at (j W + w) n + i, key = (j W + w) B + |digit| - 1, or the sentinel m W B for a zero digit or an
//      infinity base (sorted behind every real key).
//   2. cub::DeviceRadixSort over the key bits in use (stable), so that every bucket is one contiguous run of entries.
//   3. k_msm_accumulate: thread t adds the t-th fixed-length slice of the non-sentinel entries by mixed additions; buckets that
//      start and end inside the slice are stored at once, the first and the last bucket of the slice form a "node".
//      k_msm_merge folds the nodes pairwise in log2(T) rounds and stores each bucket whose sum it completes -- work follows
//      the entry count, not the bucket count: all n entries of a window in one bucket cost n / T additions + the tree.
//   4. k_msm_bucket_segments / k_msm_segment_merge: sum_b b * S_b per window by running sums over G segments of B / G buckets,
//      then a tree over the segments (acc = acc_lo + acc_hi + len_lo * run_hi, len_lo a power of two: doublings).
//   5. k_msm_final: one block per sum, Horner over its W windows (c doublings each), pt_into_affine and the normalised store.
#include "curve_io.cuh"

#include <cub/device/device_radix_sort.cuh>

#define MSM_TPB 128
#define BLS_MSM_MINB_G1 4
#define BLS_MSM_MINB_G2 3
#define MSM_NONE 0xffffffffu              /* key of an empty node */
#define MSM_SIGN 0x80000000u              /* entry value: point index | sign of the digit */
#define BLS_MSM_MAX_N ((size_t)1 << 26)   /* m * n points; W m n < 2^31 entries and m W B < 2^31 keys (32-bit indices and keys) */
#define BLS_MSM_MAX_M ((size_t)1 << 16)

template <class F> struct MsmMinB;
template <> struct MsmMinB<Fp> { static const int V = BLS_MSM_MINB_G1; };
template <> struct MsmMinB<Fp2> { static const int V = BLS_MSM_MINB_G2; };

template <class F> __device__ __forceinline__ void msm_cp_row(uint64_t* dst, const uint64_t* src) {
#pragma unroll
  for (int w = 0; w < 3 * FW<F>::W; w++) dst[w] = src[w];
}

// one thread per (sum j, point i), t = j n + i: W signed digits of k[t], base b(j, i) = shared ? i : t, entry (j, w, i) at (j W + w) n + i
__global__ void __launch_bounds__(MSM_TPB) k_msm_recode(const uint64_t* bases, int aw, int shared, const uint64_t* k, uint32_t n, uint32_t m, int c, int nwin,
                                                        uint32_t* keys, uint32_t* vals, uint32_t* count) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t mine = 0;
  if (t < m * n) {
    const uint32_t j = t / n, i = t - j * n, bi = shared ? i : t;
    const uint32_t B = 1u << (c - 1), sentinel = m * (uint32_t)nwin * B, mask = (1u << c) - 1;
    const bool inf = bases[(size_t)aw * bi + aw - 1] != 0;
    const Scalar s = ld_scalar(k + 4 * (size_t)t);
    const size_t row = (size_t)j * nwin;
    uint32_t carry = 0;
#pragma unroll 1
    for (int w = 0; w < nwin; w++) {
      const int bit = w * c, l = bit >> 5;
      uint32_t raw = 0;
      if (bit < 256) {
        const uint64_t two = (uint64_t)s.v[l] | (l < 7 ? (uint64_t)s.v[l + 1] << 32 : 0);
        raw = (uint32_t)(two >> (bit & 31)) & mask;
      }
      const uint32_t d = raw + carry;                    // <= 2^c
      carry = d > B;                                     // digit d - 2^c in [-2^(c-1), 0], borrow into the next window
      const int digit = carry ? (int)d - (int)(1u << c) : (int)d;
      uint32_t key = sentinel, val = bi;
      if (digit != 0 && !inf) {
        key = (uint32_t)(row + w) * B + (uint32_t)(digit < 0 ? -digit : digit) - 1;
        val |= digit < 0 ? MSM_SIGN : 0u;
        mine++;
      }
      keys[(row + w) * n + i] = key;
      vals[(row + w) * n + i] = val;
    }
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(count, mine);
}

// Thread t adds entries [t * per, (t + 1) * per) of the *count non-sentinel sorted entries.  Node t: kf / first = key and sum of
// the first bucket of the slice (it may continue in slice t - 1), kl / last = the last one (it may continue in slice t + 1);
// kf == kl: one bucket only, its sum in `first`; kf == MSM_NONE: empty slice (only at the end).  Buckets strictly inside the
// slice are complete and go to `buckets` directly.
template <class F>
__global__ void __launch_bounds__(MSM_TPB, MsmMinB<F>::V) k_msm_accumulate(const uint64_t* bases, const uint32_t* keys, const uint32_t* vals, const uint32_t* count, uint32_t T,
                                                                           uint32_t* kf, uint32_t* kl, uint64_t* first, uint64_t* last, uint64_t* buckets) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const int PW = 3 * FW<F>::W, AW = 2 * FW<F>::W + 1;
  const uint32_t cnt = *count, per = (cnt + T - 1) / T;
  const uint32_t begin = (uint32_t)min((uint64_t)t * per, (uint64_t)cnt), end = (uint32_t)min((uint64_t)begin + per, (uint64_t)cnt);
  uint32_t cur = MSM_NONE, k0 = MSM_NONE;
  Jac<F> acc;
  pt_set_zero(acc);
#pragma unroll 1
  for (uint32_t e = begin; e < end; e++) {
    const uint32_t key = keys[e], v = vals[e];
    if (key != cur) {
      if (cur != MSM_NONE) {
        if (k0 == MSM_NONE) { k0 = cur; st_jac(first + (size_t)PW * t, acc); }
        else st_jac(buckets + (size_t)PW * cur, acc);
      }
      cur = key;
      pt_set_zero(acc);
    }
    Aff<F> p;
    const uint64_t* row = bases + (size_t)AW * (v & ~MSM_SIGN);
    ld_F(p.x, row); ld_F(p.y, row + FW<F>::W);
    p.inf = false;                                       // infinity bases have no entries
    if (v & MSM_SIGN) p.y = f_neg(p.y);                  // negative digit: add -P
    pt_add_mixed(acc, p);
  }
  if (cur == MSM_NONE) { kf[t] = kl[t] = MSM_NONE; return; }
  if (k0 == MSM_NONE) { kf[t] = kl[t] = cur; st_jac(first + (size_t)PW * t, acc); return; }
  kf[t] = k0; kl[t] = cur;
  st_jac(last + (size_t)PW * t, acc);
}

// One round of the pairwise fold of the nodes: node a = 2 * half * i absorbs node a + half.  A bucket whose sum is complete
// (bounded by other keys on both sides) is stored; in the last round (root) node 0's own buckets are complete too.
template <class F>
__global__ void __launch_bounds__(MSM_TPB) k_msm_merge(uint32_t T, uint32_t half, int root, uint32_t* kf, uint32_t* kl, uint64_t* first, uint64_t* last, uint64_t* buckets) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t a = 2 * half * i, b = a + half;
  if (a >= T) return;
  const size_t PW = 3 * FW<F>::W;
  uint64_t *fa = first + PW * a, *la = last + PW * a;
  if (b < T && kf[b] != MSM_NONE) {                      // nodes are non-empty up to some index: node a is non-empty here
    const uint32_t lkf = kf[a], lkl = kl[a], rkf = kf[b], rkl = kl[b];
    const bool ls = lkf == lkl, rs = rkf == rkl;
    const uint64_t *fb = first + PW * b, *lb = last + PW * b;
    if (lkl == rkf) {                                    // the bucket continues across the boundary
      Jac<F> m, o;
      ld_jac(m, ls ? fa : la);
      ld_jac(o, fb);
      pt_add(m, o);
      if (ls && rs) {
        st_jac(fa, m);
      } else if (ls) {
        st_jac(fa, m); msm_cp_row<F>(la, lb); kl[a] = rkl;
      } else if (rs) {
        st_jac(la, m);
      } else {
        st_jac(buckets + PW * lkl, m); msm_cp_row<F>(la, lb); kl[a] = rkl;
      }
    } else {
      if (!ls) msm_cp_row<F>(buckets + PW * lkl, la);
      if (!rs) msm_cp_row<F>(buckets + PW * rkf, fb);
      msm_cp_row<F>(la, rs ? fb : lb);
      kl[a] = rkl;
    }
  }
  if (root && a == 0 && kf[0] != MSM_NONE) {
    msm_cp_row<F>(buckets + PW * kf[0], fa);
    if (kl[0] != kf[0]) msm_cp_row<F>(buckets + PW * kl[0], la);
  }
}

// Segment s of window j covers buckets b = s L + 1 .. (s + 1) L (L = B / G): run = sum S_b, acc = sum (b - s L) S_b.
template <class F>
__global__ void __launch_bounds__(MSM_TPB) k_msm_bucket_segments(const uint64_t* buckets, int nwin, int c, uint32_t G, uint64_t* sacc, uint64_t* srun) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (uint64_t)nwin * G) return;
  const size_t PW = 3 * FW<F>::W;
  const uint64_t B = 1ull << (c - 1), L = B / G, j = t / G, s = t % G;
  Jac<F> run, acc, sb;
  pt_set_zero(run);
  pt_set_zero(acc);
#pragma unroll 1
  for (uint64_t b = (s + 1) * L; b > s * L; b--) {
    ld_jac(sb, buckets + PW * (j * B + b - 1));
    pt_add(run, sb);
    pt_add(acc, run);
  }
  st_jac(sacc + PW * t, acc);
  st_jac(srun + PW * t, run);
}

// Segments a (lower, 2^lg_len buckets) and a + half (upper) of one window: acc_a += acc_b + 2^lg_len run_b, run_a += run_b.
template <class F>
__global__ void __launch_bounds__(MSM_TPB) k_msm_segment_merge(int nwin, uint32_t G, uint32_t half, int lg_len, uint64_t* sacc, uint64_t* srun) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, pairs = G / (2 * half);
  if (t >= (uint64_t)nwin * pairs) return;
  const size_t PW = 3 * FW<F>::W;
  const uint64_t a = (t / pairs) * G + (t % pairs) * 2 * half, b = a + half;
  Jac<F> acc, x, rb;
  ld_jac(rb, srun + PW * b);
  ld_jac(acc, sacc + PW * a);
  ld_jac(x, sacc + PW * b);
  pt_add(acc, x);
  x = rb;
#pragma unroll 1
  for (int d = 0; d < lg_len; d++) pt_double(x);
  pt_add(acc, x);
  st_jac(sacc + PW * a, acc);
  ld_jac(x, srun + PW * a);
  pt_add(x, rb);
  st_jac(srun + PW * a, x);
}

// Sum j = blockIdx.x, on thread 0 of a block of 32: Horner over its window sums (segment 0 of windows j W .. j W + W - 1 after
// the tree), then the normalised representative: (x, y, one), or G::zero() = (0, one, 0).  nwin = 0 (n = 0) stores G::zero().
// One thread per sum instead (32 sums per block) perturbs ptxas' allocation of the inlined group law (G2: spills) and made
// the single MSM 15 us slower at 2^12 points; this form compiles to the m = 1 kernel's code.
template <class F>
__global__ void __launch_bounds__(32) k_msm_final(const uint64_t* sacc, int nwin, uint32_t G, int c, uint64_t* out) {
  if (threadIdx.x != 0) return;
  const size_t PW = 3 * FW<F>::W;
  sacc += PW * G * nwin * blockIdx.x;
  Jac<F> s, t;
  pt_set_zero(s);
#pragma unroll 1
  for (int j = nwin - 1; j >= 0; j--) {
#pragma unroll 1
    for (int d = 0; d < c; d++) pt_double(s);
    ld_jac(t, sacc + PW * (size_t)j * G);
    pt_add(s, t);
  }
  Aff<F> a;
  pt_into_affine(a, s);
  F one, zero;
  f_set_one(one);
  f_set_zero(zero);
  out += PW * blockIdx.x;
  st_F(out, a.x);
  st_F(out + FW<F>::W, a.y);
  st_F(out + 2 * FW<F>::W, a.inf ? zero : one);
}

// ---- host side ----------------------------------------------------------------------------------------------------------

// Window for window = 0: c = floor(log2 n) - 5 in 8..20, the best or within 2 % of the best c of the sweep of
// tools/bench_msm.py at every size from 2^10 to 2^24 points, in G1 and in G2 (profiles/msm.md).  Below 2^14 points the
// time is the latency of the reduction chain and hardly depends on c.  For m > 1 sums the tail is paid once and the additions
// dominate: the sweep of tools/bench_msm.py --batch (profiles/msm_batch.md) keeps the rule within 1 % of the best c except
// below 2^11 points, where c = 7 is 4 % faster than 8.  Then c is raised until W m n < 2^31: c = 9 always fits the limits
// (29 * 2^26 entries, 2^16 * 29 * 2^8 keys).
static int msm_default_window(int degree, size_t n, size_t m) {
  (void)degree;
  int lg = 0;
  while (((size_t)1 << (lg + 1)) <= n) lg++;
  const int lo = m > 1 && lg <= 10 ? 7 : 8;
  int c = lg - 5;
  c = c < lo ? lo : (c > 20 ? 20 : c);
  while ((size_t)((257 + c - 1) / c) * m * n >= ((size_t)1 << 31)) c++;
  return c;
}

// m <= 2^16, m n <= 2^26, W m n < 2^31 (32-bit entry indices, CUB's int item count), m W B < 2^31 (32-bit keys)
static bool msm_args_ok(int degree, size_t n, size_t m, int window) {
  if (window != 0 && (window < 2 || window > 20)) return false;
  if (m > BLS_MSM_MAX_M || n > BLS_MSM_MAX_N || m * n > BLS_MSM_MAX_N) return false;
  const int c = window ? window : msm_default_window(degree, n, m);
  const size_t nwin = (257 + c - 1) / c;
  return nwin * m * n < ((size_t)1 << 31) && (m * nwin << (c - 1)) < ((size_t)1 << 31);
}

namespace {
struct MsmPlan {
  int c, nwin, end_bit;                          // nwin = W, the windows of one sum
  uint32_t B, G, T;
  size_t nw, E, pw;                              // m W windows in all, entries, bytes per Jacobian point
  size_t off_keys[2], off_vals[2], off_cub, cub_bytes, off_count, off_buckets, off_kf, off_kl, off_first, off_last, off_sacc, off_srun, total;
};
}  // namespace

static size_t msm_align(size_t x) { return (x + 255) & ~(size_t)255; }

// Scratch layout and launch shape of one call (the CUB size query needs the context's device to be current).
static cudaError_t msm_plan(const bls_ctx* ctx, int degree, size_t n, size_t m, int window, MsmPlan& p) {
  p.c = window ? window : msm_default_window(degree, n, m);
  p.nwin = (257 + p.c - 1) / p.c;
  p.B = 1u << (p.c - 1);
  p.nw = m * p.nwin;
  p.E = p.nw * n;
  p.pw = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const uint32_t sentinel = (uint32_t)p.nw * p.B;
  p.end_bit = 0;
  while (p.end_bit < 32 && (sentinel >> p.end_bit)) p.end_bit++;
  const size_t cap = (size_t)ctx->sm_count * MSM_TPB * (degree == 2 ? BLS_MSM_MINB_G2 : BLS_MSM_MINB_G1);
  p.T = (uint32_t)(p.E < cap ? (p.E ? p.E : 1) : cap);
  p.G = 1;
  const size_t seg_target = (size_t)ctx->sm_count * MSM_TPB * 2;
  while (p.G * 2 <= p.B && p.nw * p.G * 2 <= seg_target) p.G *= 2;
  cub::DoubleBuffer<uint32_t> dk(nullptr, nullptr), dv(nullptr, nullptr);
  p.cub_bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, p.cub_bytes, dk, dv, (int)p.E, 0, p.end_bit);
  if (e != cudaSuccess) return e;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += msm_align(bytes); return at; };
  for (int i = 0; i < 2; i++) p.off_keys[i] = take(p.E * 4);
  for (int i = 0; i < 2; i++) p.off_vals[i] = take(p.E * 4);
  p.off_cub = take(p.cub_bytes);
  p.off_count = take(4);
  p.off_buckets = take(p.nw * p.B * p.pw);
  p.off_kf = take((size_t)p.T * 4);
  p.off_kl = take((size_t)p.T * 4);
  p.off_first = take((size_t)p.T * p.pw);
  p.off_last = take((size_t)p.T * p.pw);
  p.off_sacc = take(p.nw * p.G * p.pw);
  p.off_srun = take(p.nw * p.G * p.pw);
  p.total = o;
  return cudaSuccess;
}

template <class F>
static int msm_dev_impl(bls_ctx* ctx, int degree, const void* bases, int shared, const bls_fr_repr* k, size_t n, size_t m, int window, void* out,
                        void* scratch, void* stream) {
  if (!ctx || (m && !out) || (n && m && (!bases || !k || !scratch)) || !msm_args_ok(degree, n, m, window)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  USE_DEVICE(ctx);
  cudaStream_t s = pick(ctx, stream);
  if (n == 0) {
    k_msm_final<F><<<(unsigned)m, 32, 0, s>>>(nullptr, 0, 1, 2, (uint64_t*)out);
    LAUNCH_CHECK();
    return BLS_OK;
  }
  MsmPlan p;
  CK(msm_plan(ctx, degree, n, m, window, p));
  char* base = (char*)scratch;
  uint32_t* keys[2] = {(uint32_t*)(base + p.off_keys[0]), (uint32_t*)(base + p.off_keys[1])};
  uint32_t* vals[2] = {(uint32_t*)(base + p.off_vals[0]), (uint32_t*)(base + p.off_vals[1])};
  uint32_t* count = (uint32_t*)(base + p.off_count);
  uint32_t *kf = (uint32_t*)(base + p.off_kf), *kl = (uint32_t*)(base + p.off_kl);
  uint64_t* buckets = (uint64_t*)(base + p.off_buckets);
  uint64_t *first = (uint64_t*)(base + p.off_first), *last = (uint64_t*)(base + p.off_last);
  uint64_t *sacc = (uint64_t*)(base + p.off_sacc), *srun = (uint64_t*)(base + p.off_srun);
  CK(cudaMemsetAsync(count, 0, 4, s));
  CK(cudaMemsetAsync(buckets, 0, p.nw * p.B * p.pw, s));                // z = 0: every bucket starts as zero
  const int aw = degree == 2 ? sizeof(bls_g2_affine) / 8 : sizeof(bls_g1_affine) / 8;
  k_msm_recode<<<blocks_for(m * n, MSM_TPB), MSM_TPB, 0, s>>>((const uint64_t*)bases, aw, shared != 0, (const uint64_t*)k, (uint32_t)n, (uint32_t)m, p.c, p.nwin,
                                                              keys[0], vals[0], count);
  LAUNCH_CHECK();
  cub::DoubleBuffer<uint32_t> dk(keys[0], keys[1]), dv(vals[0], vals[1]);
  size_t cub_bytes = p.cub_bytes;
  CK(cub::DeviceRadixSort::SortPairs(base + p.off_cub, cub_bytes, dk, dv, (int)p.E, 0, p.end_bit, s));
  LAUNCH_CHECK();                                                        // the sort's kernels count as one launch
  k_msm_accumulate<F><<<blocks_for(p.T, MSM_TPB), MSM_TPB, 0, s>>>((const uint64_t*)bases, dk.Current(), dv.Current(), count, p.T, kf, kl, first, last, buckets);
  LAUNCH_CHECK();
  for (uint32_t half = 1;; half *= 2) {
    const int root = 2 * (uint64_t)half >= p.T;
    const uint64_t threads = (p.T + 2 * (uint64_t)half - 1) / (2 * (uint64_t)half);
    k_msm_merge<F><<<blocks_for(threads, MSM_TPB), MSM_TPB, 0, s>>>(p.T, half, root, kf, kl, first, last, buckets);
    LAUNCH_CHECK();
    if (root) break;
  }
  k_msm_bucket_segments<F><<<blocks_for(p.nw * p.G, MSM_TPB), MSM_TPB, 0, s>>>(buckets, (int)p.nw, p.c, p.G, sacc, srun);
  LAUNCH_CHECK();
  int lg_len = p.c - 1;                                                  // log2(B / G) + log2(half)
  for (uint32_t g = p.G; g > 1; g >>= 1) lg_len--;
  for (uint32_t half = 1; half < p.G; half *= 2, lg_len++) {
    k_msm_segment_merge<F><<<blocks_for(p.nw * p.G / (2 * half), MSM_TPB), MSM_TPB, 0, s>>>((int)p.nw, p.G, half, lg_len, sacc, srun);
    LAUNCH_CHECK();
  }
  k_msm_final<F><<<(unsigned)m, 32, 0, s>>>(sacc, p.nwin, p.G, p.c, (uint64_t*)out);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int msm_host(bls_ctx* ctx, int degree, const void* bases, int shared, const bls_fr_repr* k, size_t n, size_t m, void* out) {
  if (!ctx || (m && !out) || (n && m && (!bases || !k)) || !msm_args_ok(degree, n, m, 0)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t ab = degree == 2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine);
  const size_t pb = degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1);
  const size_t nb = shared ? n : m * n;
  const size_t scratch = bls_msm_batch_scratch_bytes(ctx, degree, n, m, 0);
  if (!scratch) return BLS_ERR_CUDA;
  H2D(db, nb ? bases : nullptr, nb * ab);
  H2D(dk, n ? k : nullptr, m * n * sizeof(bls_fr_repr));
  DALLOC(dscr, scratch);
  DALLOC(dout, m * pb);
  int rc = degree == 2 ? bls_g2_msm_batch_dev(ctx, (const bls_g2_affine*)db.p, shared, (const bls_fr_repr*)dk.p, n, m, 0, (bls_g2*)dout.p, dscr.p, ctx->stream)
                       : bls_g1_msm_batch_dev(ctx, (const bls_g1_affine*)db.p, shared, (const bls_fr_repr*)dk.p, n, m, 0, (bls_g1*)dout.p, dscr.p, ctx->stream);
  TRY(rc);
  D2H(out, dout, m * pb);
  SYNC();
  return BLS_OK;
}

extern "C" {

size_t bls_msm_batch_scratch_bytes(const bls_ctx* ctx, int degree, size_t n, size_t m, int window) {
  if (!ctx || (degree != 1 && degree != 2) || !msm_args_ok(degree, n, m, window)) return 0;
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  MsmPlan p;
  if (n == 0 || m == 0) return 1;
  return msm_plan(ctx, degree, n, m, window, p) == cudaSuccess ? p.total : 0;
}
size_t bls_msm_scratch_bytes(const bls_ctx* ctx, int degree, size_t n, int window) { return bls_msm_batch_scratch_bytes(ctx, degree, n, 1, window); }
int bls_g1_msm_batch_dev(bls_ctx* ctx, const bls_g1_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, int window, bls_g1* out, void* scratch,
                         void* stream) {
  return msm_dev_impl<Fp>(ctx, 1, bases, shared_bases, k, n, m, window, out, scratch, stream);
}
int bls_g2_msm_batch_dev(bls_ctx* ctx, const bls_g2_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, int window, bls_g2* out, void* scratch,
                         void* stream) {
  return msm_dev_impl<Fp2>(ctx, 2, bases, shared_bases, k, n, m, window, out, scratch, stream);
}
int bls_g1_msm_dev(bls_ctx* ctx, const bls_g1_affine* bases, const bls_fr_repr* k, size_t n, int window, bls_g1* out1, void* scratch, void* stream) {
  return msm_dev_impl<Fp>(ctx, 1, bases, 1, k, n, 1, window, out1, scratch, stream);
}
int bls_g2_msm_dev(bls_ctx* ctx, const bls_g2_affine* bases, const bls_fr_repr* k, size_t n, int window, bls_g2* out1, void* scratch, void* stream) {
  return msm_dev_impl<Fp2>(ctx, 2, bases, 1, k, n, 1, window, out1, scratch, stream);
}
int bls_g1_msm_batch(bls_ctx* ctx, const bls_g1_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, bls_g1* out) {
  return msm_host(ctx, 1, bases, shared_bases, k, n, m, out);
}
int bls_g2_msm_batch(bls_ctx* ctx, const bls_g2_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, bls_g2* out) {
  return msm_host(ctx, 2, bases, shared_bases, k, n, m, out);
}
int bls_g1_msm(bls_ctx* ctx, const bls_g1_affine* bases, const bls_fr_repr* k, size_t n, bls_g1* out1) { return msm_host(ctx, 1, bases, 1, k, n, 1, out1); }
int bls_g2_msm(bls_ctx* ctx, const bls_g2_affine* bases, const bls_fr_repr* k, size_t n, bls_g2* out1) { return msm_host(ctx, 2, bases, 1, k, n, 1, out1); }

}  // extern "C"
