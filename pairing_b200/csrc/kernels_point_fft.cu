// kernels_point_fft.cu -- the FFT over G1 and G2 points (bellman's EvaluationDomain<Point<G>>: fft, ifft, coset_fft,
// icoset_fft, where group_mul_assign is a scalar multiplication) and KZG openings at every point of the domain by the
// FK20 method (bls_kzg_open_all_*).  Its own translation unit (see abi_common.cuh): the Fr FFT and the normalisation are
// the other units' entry points, called through the C ABI, so no existing kernel is recompiled.
//
// A transform of n = 2^L points per row runs on a Jacobian scratch buffer, radix 2, decimation in time:
//   k_pfft_load     affine rows -> Jacobian, row position bitrev(i) <- input i (one row may feed all m rows: FK20's table)
//   k_pfft_mul      buf[p] = c_p buf[p] for a scalar table c (the coset scaling g^i, n^-1, n^-1 g^-i; FK20's c-hat)
//   per stage s = 0 .. L-1 (half-width h = 2^s), over the butterflies (i0, i0 + h), twiddle omega_(2h)^j = omega^(j n / 2h):
//     k_pfft_bfly0  j = 0: the twiddle is one, a + b and a - b only
//     k_pfft_bfly   j >= 1: t = omega^(j n / 2h) b by wNAF, then a + t and a - t
//   bls_g*_batch_normalization_dev, then k_pfft_emit (canonical affine rows; the identity is (0, one, infinity = 1)).
// Every scalar multiplication (the butterflies' and k_pfft_mul's) runs curve.cuh's decoupled wNAF runner, K points per
// thread with per-thread tables, the same schedule as the library's wNAF kernels: lanes hold different twiddles and
// therefore different digit patterns, and the runner only ever issues one of double / add across the warp.
#include <stddef.h>

#include "curve_io.cuh"
#include "fr_fft_consts.cuh"

#define PFFT_TPB 128
#define PFFT_MINB_G1 4
#define PFFT_MINB_G2 3
#define PFFT_K_G1 3                           /* points per thread, as the wNAF kernels (BLS_WNAF_K, BLS_WNAF_K_G2) */
#define PFFT_K_G2 2
#define PFFT_MAXT 8                           /* wNAF table entries: window <= 4 for scalars of < 2^256 */
#define PFFT_MAX_LOG_N 26                     /* the multiexp's limits */
#define PFFT_MAX_ELEMS ((size_t)1 << 26)
#define FK_MAX_LOG_N 24
#define FK_MAX_ELEMS ((size_t)1 << 26)        /* m * 2n */

// ---- scalars --------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ Fr pf_ld_fr(const uint64_t* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void pf_st_fr(uint64_t* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
// Montgomery Fr -> the canonical integer (into_repr: the Montgomery product with the integer 1)
__device__ __forceinline__ Scalar pf_repr(const Fr& a) {
  Fr one = fr_zero();
  one.v[0] = 1;
  const Fr c = fr_mul(a, one);
  Scalar s;
#pragma unroll
  for (int i = 0; i < 8; i++) s.v[i] = c.v[i];
  return s;
}
// x^e from the table pw[b] = x^(2^b)
__device__ __forceinline__ Fr pf_pow_bits(const Fr* pw, uint32_t e) {
  Fr r = fr_one();
#pragma unroll 1
  for (int b = 0; e; b++, e >>= 1)
    if (e & 1) r = fr_mul(r, pw[b]);
  return r;
}
__device__ __forceinline__ size_t pf_rev(size_t i, int L) { return L ? (size_t)(__brevll((unsigned long long)i) >> (64 - L)) : 0; }

// One thread per entry: tw[e] = omega^(+-e), e < n / 2 (inv: omega^-1), and -- cs != NULL -- the scaling table of the kind:
// coset_fft cs[i] = g^i (i < n), ifft cs[0] = n^-1, icoset_fft cs[i] = n^-1 g^-i.  Montgomery form.
__global__ void __launch_bounds__(PFFT_TPB) k_pfft_tables(int L, int inv, int kind, uint64_t* tw, uint64_t* cs) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x, half = ((size_t)1 << L) >> 1, n = (size_t)1 << L;
  if (id < half) {
    pf_st_fr(tw + 4 * id, pf_pow_bits((inv ? FR_ROOT_INV_POW : FR_ROOT_POW) + 32 - L, (uint32_t)id));
    return;
  }
  const size_t i = id - half;
  if (!cs || i >= n) return;
  if (kind == BLS_IFFT) {
    if (i == 0) pf_st_fr(cs, FR_INV_2POW[L]);
  } else if (kind == BLS_COSET_FFT) {
    pf_st_fr(cs + 4 * i, pf_pow_bits(FR_GEN_POW, (uint32_t)i));
  } else if (kind == BLS_ICOSET_FFT) {
    pf_st_fr(cs + 4 * i, fr_mul(FR_INV_2POW[L], pf_pow_bits(FR_GEN_INV_POW, (uint32_t)i)));
  }
}

// ---- the group law --------------------------------------------------------------------------------------------------------
template <class F, int K> struct PfTables {
  Jac<F> t[K][PFFT_MAXT];
  __device__ __forceinline__ Jac<F> get(int j, int e) const { return t[j][e]; }
};

// res[j] = k[j] base[j] for the K points of this thread: wnaf_table / wnaf_form with the reference's window for the scalar's
// length, then the decoupled runner.  Every lane of the warp must call it (the runner votes with __ballot_sync).
template <class F, bool IS_G2, int K>
__device__ __forceinline__ void pf_mul(Jac<F> (&res)[K], const Jac<F> (&base)[K], const Scalar (&k)[K]) {
  PfTables<F, K> table;
  int8_t digits[K][260];
  WnafState<K> st;
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    const int nb = scalar_num_bits(k[j]);
    const int w = IS_G2 ? g2_window_for_bits(nb) : g1_window_for_bits(nb), tsize = 1 << (w - 1);
    Jac<F> b = base[j], dbl = base[j];
    pt_double(dbl);
#pragma unroll 1
    for (int e = 0; e < PFFT_MAXT; e++) {
      if (e < tsize) { table.t[j][e] = b; if (e + 1 < tsize) pt_add(b, dbl); }
    }
    st.i[j] = wnaf_form(digits[j], k[j], w) - 1;
    st.found[j] = false; st.doubled[j] = false;
    pt_set_zero(res[j]);
  }
  pt_wnaf_run_lazy<F, K>(res, table, digits, st);
}

// (a, b) <- (a + t, a - t)
template <class F> __device__ __forceinline__ void pf_bfly(uint64_t* pa, uint64_t* pb, Jac<F> t) {
  Jac<F> a, d;
  ld_jac(a, pa);
  d = a;
  pt_add(a, t);
  pt_negate(t);
  pt_add(d, t);
  st_jac(pa, a);
  st_jac(pb, d);
}

// m rows of n = 2^L: buf[row n + bitrev(i)] = in[(shared ? 0 : row) n + i] as a Jacobian point
template <class F>
__global__ void __launch_bounds__(PFFT_TPB) k_pfft_load(const uint64_t* in, int shared, int L, size_t total, uint64_t* buf) {
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int W = FW<F>::W;
  const size_t n = (size_t)1 << L, row = p >> L, i = p & (n - 1);
  Aff<F> a;
  ld_aff(a, in + (size_t)(2 * W + 1) * ((shared ? 0 : row) * n + i));
  Jac<F> r;
  if (a.inf) pt_set_zero(r);
  else { r.x = a.x; r.y = a.y; f_set_one(r.z); }
  st_jac(buf + (size_t)(3 * W) * (row * n + pf_rev(i, L)), r);
}

// buf[p] = c[idx] buf[p] for p < total: idx = (p >> L) kstride + ((rev ? bitrev(local) : local) & kmask), local = p mod 2^L;
// c holds Montgomery Fr
template <class F, bool IS_G2, int K>
__global__ void __launch_bounds__(PFFT_TPB, IS_G2 ? PFFT_MINB_G2 : PFFT_MINB_G1)
    k_pfft_mul(uint64_t* buf, const uint64_t* c, size_t total, int L, size_t kstride, size_t kmask, int rev) {
  const size_t T = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  Jac<F> base[K], res[K];
  Scalar k[K];
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t p = t + (size_t)j * T;
    const bool active = p < total;
    if (!active) p = total - 1;
    ld_jac(base[j], buf + (size_t)PW * p);
    const size_t local = p & (((size_t)1 << L) - 1);
    const size_t idx = (p >> L) * kstride + ((rev ? pf_rev(local, L) : local) & kmask);
    k[j] = pf_repr(pf_ld_fr(c + 4 * idx));
    if (!active) {
#pragma unroll
      for (int w = 0; w < 8; w++) k[j].v[w] = 0;
    }
  }
  pf_mul<F, IS_G2, K>(res, base, k);
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    const size_t p = t + (size_t)j * T;
    if (p < total) st_jac(buf + (size_t)PW * p, res[j]);
  }
}

// stage s, the butterflies with twiddle one: m n / 2h of them, (i0, i0 + h) with i0 = 2h g
template <class F>
__global__ void __launch_bounds__(PFFT_TPB) k_pfft_bfly0(uint64_t* buf, size_t count, int L, int s) {
  const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= count) return;
  const int PW = 3 * FW<F>::W;
  const size_t i0 = u << (s + 1);                                  // rows are whole multiples of 2h
  Jac<F> b;
  ld_jac(b, buf + (size_t)PW * (i0 + ((size_t)1 << s)));
  pf_bfly<F>(buf + (size_t)PW * i0, buf + (size_t)PW * (i0 + ((size_t)1 << s)), b);
}

// stage s >= 1, the butterflies with j >= 1: h - 1 per group of 2h, m n / 2h groups; tw[e] = omega^e (Montgomery), e < n / 2
template <class F, bool IS_G2, int K>
__global__ void __launch_bounds__(PFFT_TPB, IS_G2 ? PFFT_MINB_G2 : PFFT_MINB_G1)
    k_pfft_bfly(uint64_t* buf, const uint64_t* tw, size_t count, int L, int s) {
  const size_t T = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int PW = 3 * FW<F>::W;
  const size_t h = (size_t)1 << s, hm1 = h - 1;
  Jac<F> base[K], res[K];
  Scalar k[K];
  size_t i0[K];
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    size_t u = t + (size_t)j * T;
    const bool active = u < count;
    if (!active) u = count - 1;
    const size_t g = u / hm1, jj = 1 + (u - g * hm1);
    i0[j] = (g << (s + 1)) + jj;
    ld_jac(base[j], buf + (size_t)PW * (i0[j] + h));
    k[j] = pf_repr(pf_ld_fr(tw + 4 * (jj << (L - 1 - s))));
    if (!active) {
#pragma unroll
      for (int w = 0; w < 8; w++) k[j].v[w] = 0;
    }
  }
  pf_mul<F, IS_G2, K>(res, base, k);
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    if (t + (size_t)j * T < count) pf_bfly<F>(buf + (size_t)PW * i0[j], buf + (size_t)PW * (i0[j] + h), res[j]);
  }
}

// normalised Jacobian rows -> canonical affine rows; the identity is (0, one, infinity = 1) whatever its x and y
template <class F>
__global__ void __launch_bounds__(PFFT_TPB) k_pfft_emit(const uint64_t* buf, size_t count, uint64_t* out) {
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= count) return;
  const int W = FW<F>::W;
  Jac<F> r;
  ld_jac(r, buf + (size_t)(3 * W) * p);
  Aff<F> a;
  a.inf = pt_is_zero(r);
  if (a.inf) { f_set_zero(a.x); f_set_one(a.y); }
  else { a.x = r.x; a.y = r.y; }
  st_aff(out + (size_t)(2 * W + 1) * p, a);
}

// ---- FK20 ---------------------------------------------------------------------------------------------------------------
// w_t = srs[2n - 1 - t] for n + 1 <= t <= 2n - 1, the identity for t <= n (affine rows, t < 2n)
__global__ void __launch_bounds__(PFFT_TPB) k_fk_w(const uint64_t* srs, size_t n, uint64_t* w) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * n) return;
  uint64_t* d = w + G1A_W * t;
  if (t <= n) {
    Aff<Fp> a;
    a.inf = true; f_set_zero(a.x); f_set_one(a.y);
    st_aff(d, a);
  } else {
    const uint64_t* s = srs + G1A_W * (2 * n - 1 - t);
#pragma unroll 1
    for (int k = 0; k < G1A_W; k++) d[k] = s[k];
  }
}

// c-hat input: row j of 2n = (p_j zero-padded) (2n)^-1, Montgomery Fr
__global__ void __launch_bounds__(PFFT_TPB) k_fk_pad(const uint64_t* p, int L, size_t m, uint64_t* out) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)1 << L;
  if (id >= 2 * m * n) return;
  const size_t j = id >> (L + 1), i = id & (2 * n - 1);
  pf_st_fr(out + 4 * id, i < n ? fr_mul(pf_ld_fr(p + 4 * (j * n + i)), FR_INV_2POW[L + 1]) : fr_zero());
}

// H: the first n of every row of 2n, bit-reversed into rows of n (the input order of the next transform's stages)
template <class F>
__global__ void __launch_bounds__(PFFT_TPB) k_pfft_take_rev(const uint64_t* src, int L, size_t total, uint64_t* dst) {
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int PW = 3 * FW<F>::W;
  const size_t row = p >> L, i = p & (((size_t)1 << L) - 1);
  const uint64_t* s = src + (size_t)PW * ((row << (L + 1)) + i);
  uint64_t* d = dst + (size_t)PW * ((row << L) + pf_rev(i, L));
#pragma unroll 1
  for (int k = 0; k < PW; k++) d[k] = s[k];
}

// ---- host side ------------------------------------------------------------------------------------------------------------

static size_t pf_align(size_t x) { return (x + 255) & ~(size_t)255; }

namespace {
struct PfLayout {
  size_t off_buf, off_tw, off_cs, off_norm, total;
};
struct FkLayout {
  size_t off_chat, off_buf, off_h, off_tw2, off_tw1, off_norm, off_fft, total;
};
}  // namespace

static bool pf_args_ok(int log_n, size_t m) { return log_n >= 0 && log_n <= PFFT_MAX_LOG_N && m <= (PFFT_MAX_ELEMS >> log_n); }
static bool fk_args_ok(int log_n, size_t m) { return log_n >= 0 && log_n <= FK_MAX_LOG_N && m <= (FK_MAX_ELEMS >> (log_n + 1)); }
static bool pf_kind_ok(int kind) { return kind >= BLS_FFT && kind <= BLS_ICOSET_FFT; }

// the Jacobian buffer (m n points), the twiddles (n / 2), the scaling table (n), the normalisation's work region
static size_t pf_layout(bls_ctx* ctx, int degree, int L, size_t m, PfLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += pf_align(bytes); return at; };
  const size_t n = (size_t)1 << L, mn = m << L;
  l.off_buf = take(mn * (degree == 2 ? sizeof(bls_g2) : sizeof(bls_g1)));
  l.off_tw = take((n / 2) * sizeof(bls_fr));
  l.off_cs = take(n * sizeof(bls_fr));
  l.off_norm = take(bls_batch_normalization_scratch_bytes(ctx, degree, mn));
  return l.total = o;
}

template <class F, bool IS_G2> static int pf_launch_mul(bls_ctx* ctx, uint64_t* buf, const uint64_t* c, size_t total, int L, size_t kstride,
                                                        size_t kmask, int rev, cudaStream_t st) {
  const int K = IS_G2 ? PFFT_K_G2 : PFFT_K_G1;
  k_pfft_mul<F, IS_G2, K><<<blocks_for((total + K - 1) / K, PFFT_TPB), PFFT_TPB, 0, st>>>(buf, c, total, L, kstride, kmask, rev);
  LAUNCH_CHECK();
  return BLS_OK;
}

// the L radix-2 stages over m bit-reversed rows of 2^L Jacobian points in buf; tw = omega^(+-e), e < 2^(L-1).  Results in
// natural order.
template <class F, bool IS_G2> static int pf_stages(bls_ctx* ctx, uint64_t* buf, const uint64_t* tw, int L, size_t m, cudaStream_t st) {
  const int K = IS_G2 ? PFFT_K_G2 : PFFT_K_G1;
  const size_t mn = m << L;
  for (int s = 0; s < L; s++) {
    const size_t groups = mn >> (s + 1);
    k_pfft_bfly0<F><<<blocks_for(groups, PFFT_TPB), PFFT_TPB, 0, st>>>(buf, groups, L, s);
    LAUNCH_CHECK();
    const size_t count = groups * (((size_t)1 << s) - 1);
    if (count) {
      k_pfft_bfly<F, IS_G2, K><<<blocks_for((count + K - 1) / K, PFFT_TPB), PFFT_TPB, 0, st>>>(buf, tw, count, L, s);
      LAUNCH_CHECK();
    }
  }
  return BLS_OK;
}

template <class F, bool IS_G2> static int pf_normalize(bls_ctx* ctx, uint64_t* buf, size_t n, void* scratch, cudaStream_t st) {
  if (IS_G2) return bls_g2_batch_normalization_dev(ctx, (bls_g2*)buf, n, scratch, st);
  return bls_g1_batch_normalization_dev(ctx, (bls_g1*)buf, n, scratch, st);
}

template <class F, bool IS_G2>
static int pf_dev_impl(bls_ctx* ctx, int kind, const void* in, void* out, int log_n, size_t m, void* scratch, void* stream) {
  if (!ctx || !pf_kind_ok(kind) || !pf_args_ok(log_n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!in || !out || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t st = pick(ctx, stream);
  PfLayout l;
  pf_layout(ctx, IS_G2 ? 2 : 1, log_n, m, l);
  char* base = (char*)scratch;
  uint64_t *buf = (uint64_t*)(base + l.off_buf), *tw = (uint64_t*)(base + l.off_tw), *cs = (uint64_t*)(base + l.off_cs);
  const size_t n = (size_t)1 << log_n, mn = m << log_n;
  const bool inv = kind == BLS_IFFT || kind == BLS_ICOSET_FFT;
  k_pfft_tables<<<blocks_for(n / 2 + n, PFFT_TPB), PFFT_TPB, 0, st>>>(log_n, inv, kind, tw, kind == BLS_FFT ? nullptr : cs);
  LAUNCH_CHECK();
  k_pfft_load<F><<<blocks_for(mn, PFFT_TPB), PFFT_TPB, 0, st>>>((const uint64_t*)in, 0, log_n, mn, buf);
  LAUNCH_CHECK();
  if (kind == BLS_COSET_FFT) {                                     // element i (at row position bitrev(i)) times g^i
    TRY((pf_launch_mul<F, IS_G2>(ctx, buf, cs, mn, log_n, 0, n - 1, 1, st)));
  }
  TRY((pf_stages<F, IS_G2>(ctx, buf, tw, log_n, m, st)));
  if (inv) {                                                       // output i times n^-1 (ifft) or n^-1 g^-i (icoset_fft)
    TRY((pf_launch_mul<F, IS_G2>(ctx, buf, cs, mn, log_n, 0, kind == BLS_IFFT ? 0 : n - 1, 0, st)));
  }
  TRY((pf_normalize<F, IS_G2>(ctx, buf, mn, base + l.off_norm, st)));
  k_pfft_emit<F><<<blocks_for(mn, PFFT_TPB), PFFT_TPB, 0, st>>>(buf, mn, (uint64_t*)out);
  LAUNCH_CHECK();
  return BLS_OK;
}

template <class F, bool IS_G2> static int pf_host(bls_ctx* ctx, int kind, const void* in, void* out, int log_n, size_t m) {
  if (!ctx || !pf_kind_ok(kind) || !pf_args_ok(log_n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!in || !out) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  const size_t bytes = (m << log_n) * (IS_G2 ? sizeof(bls_g2_affine) : sizeof(bls_g1_affine));
  PfLayout l;
  pf_layout(ctx, IS_G2 ? 2 : 1, log_n, m, l);
  H2D(din, in, bytes);
  DALLOC(dscr, l.total);
  TRY((pf_dev_impl<F, IS_G2>(ctx, kind, din.p, din.p, log_n, m, dscr.p, ctx->stream)));
  D2H(out, din, bytes);
  SYNC();
  return BLS_OK;
}

// ---- FK20 ---------------------------------------------------------------------------------------------------------------
// prepare: the w rows (2n), then the point FFT's scratch for one row of 2n
static size_t fk_prepare_layout(bls_ctx* ctx, int L, size_t& off_fft) {
  PfLayout l;
  const size_t w = pf_align(((size_t)2 << L) * sizeof(bls_g1_affine));
  off_fft = w;
  return w + pf_layout(ctx, 1, L + 1, 1, l);
}

static int fk_prepare_dev_impl(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, int log_n, bls_g1_affine* table, void* scratch,
                               void* stream) {
  if (!ctx || log_n < 0 || log_n > FK_MAX_LOG_N) return BLS_ERR_INVALID_ARGUMENT;
  const size_t n = (size_t)1 << log_n;
  if (srs_len + 1 < n || (n > 1 && !srs) || !table || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t st = pick(ctx, stream);
  size_t off_fft;
  fk_prepare_layout(ctx, log_n, off_fft);
  uint64_t* w = (uint64_t*)scratch;
  k_fk_w<<<blocks_for(2 * n, PFFT_TPB), PFFT_TPB, 0, st>>>((const uint64_t*)srs, n, w);
  LAUNCH_CHECK();
  return pf_dev_impl<Fp, false>(ctx, BLS_FFT, w, table, log_n + 1, 1, (char*)scratch + off_fft, st);
}

// open_all: c-hat (m 2n Fr), the Jacobian buffer (m 2n), H bit-reversed (m n), the twiddles of 2n and of n, the
// normalisation's work region (m n), the Fr FFT's scratch (the larger of the two transforms)
static size_t fk_layout(bls_ctx* ctx, int L, size_t m, FkLayout& l) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += pf_align(bytes); return at; };
  const size_t n = (size_t)1 << L;
  l.off_chat = take(2 * m * n * sizeof(bls_fr));
  l.off_buf = take(2 * m * n * sizeof(bls_g1));
  l.off_h = take(m * n * sizeof(bls_g1));
  l.off_tw2 = take(n * sizeof(bls_fr));
  l.off_tw1 = take((n / 2) * sizeof(bls_fr));
  l.off_norm = take(bls_batch_normalization_scratch_bytes(ctx, 1, m * n));
  const size_t f2 = bls_fr_fft_scratch_bytes(ctx, L + 1, m), f1 = bls_fr_fft_scratch_bytes(ctx, L, m);
  if (!f2 || !f1) return 0;
  l.off_fft = take(f2 > f1 ? f2 : f1);
  return l.total = o;
}

static int fk_open_all_dev_impl(bls_ctx* ctx, const bls_g1_affine* table, const bls_fr* p, int log_n, size_t m, bls_fr* y, bls_g1_affine* proof,
                                void* scratch, void* stream) {
  if (!ctx || !fk_args_ok(log_n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!table || !p || !y || !proof || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t st = pick(ctx, stream);
  FkLayout l;
  if (!fk_layout(ctx, log_n, m, l)) return BLS_ERR_CUDA;
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint64_t *chat = at(l.off_chat), *buf = at(l.off_buf), *hb = at(l.off_h), *tw2 = at(l.off_tw2), *tw1 = at(l.off_tw1);
  const int L2 = log_n + 1;
  const size_t n = (size_t)1 << log_n, m2n = 2 * m * n, mn = m * n;
  // y = FFT_n(p); c-hat = FFT_2n(p zero-padded, times (2n)^-1)
  TRY(bls_fr_fft_dev(ctx, BLS_FFT, p, y, log_n, m, base + l.off_fft, st));
  k_fk_pad<<<blocks_for(m2n, PFFT_TPB), PFFT_TPB, 0, st>>>((const uint64_t*)p, log_n, m, chat);
  LAUNCH_CHECK();
  TRY(bls_fr_fft_dev(ctx, BLS_FFT, (const bls_fr*)chat, (bls_fr*)chat, L2, m, base + l.off_fft, st));
  // twiddles of the inverse transform of 2n and the forward one of n
  k_pfft_tables<<<blocks_for(n, PFFT_TPB), PFFT_TPB, 0, st>>>(L2, 1, BLS_IFFT, tw2, nullptr);
  LAUNCH_CHECK();
  k_pfft_tables<<<blocks_for(n / 2 + 1, PFFT_TPB), PFFT_TPB, 0, st>>>(log_n, 0, BLS_FFT, tw1, nullptr);
  LAUNCH_CHECK();
  // every row: table bit-reversed, times c-hat (the scalar of position p is c-hat[bitrev(p)]), the unscaled inverse stages
  k_pfft_load<Fp><<<blocks_for(m2n, PFFT_TPB), PFFT_TPB, 0, st>>>((const uint64_t*)table, 1, L2, m2n, buf);
  LAUNCH_CHECK();
  TRY((pf_launch_mul<Fp, false>(ctx, buf, chat, m2n, L2, 2 * n, 2 * n - 1, 1, st)));
  TRY((pf_stages<Fp, false>(ctx, buf, tw2, L2, m, st)));
  // H = the first n outputs, then proofs = FFT_n(H)
  k_pfft_take_rev<Fp><<<blocks_for(mn, PFFT_TPB), PFFT_TPB, 0, st>>>(buf, log_n, mn, hb);
  LAUNCH_CHECK();
  TRY((pf_stages<Fp, false>(ctx, hb, tw1, log_n, m, st)));
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)hb, mn, base + l.off_norm, st));
  k_pfft_emit<Fp><<<blocks_for(mn, PFFT_TPB), PFFT_TPB, 0, st>>>(hb, mn, (uint64_t*)proof);
  LAUNCH_CHECK();
  return BLS_OK;
}

extern "C" {

size_t bls_point_fft_scratch_bytes(const bls_ctx* ctx, int degree, int log_n, size_t m) {
  if (!ctx || (degree != 1 && degree != 2) || !pf_args_ok(log_n, m)) return 0;
  if (m == 0) return 1;
  PfLayout l;
  return pf_layout(const_cast<bls_ctx*>(ctx), degree, log_n, m, l);
}
int bls_g1_fft_dev(bls_ctx* ctx, int kind, const bls_g1_affine* in, bls_g1_affine* out, int log_n, size_t m, void* scratch, void* stream) {
  return pf_dev_impl<Fp, false>(ctx, kind, in, out, log_n, m, scratch, stream);
}
int bls_g2_fft_dev(bls_ctx* ctx, int kind, const bls_g2_affine* in, bls_g2_affine* out, int log_n, size_t m, void* scratch, void* stream) {
  return pf_dev_impl<Fp2, true>(ctx, kind, in, out, log_n, m, scratch, stream);
}
int bls_g1_fft_batch(bls_ctx* ctx, int kind, const bls_g1_affine* in, bls_g1_affine* out, int log_n, size_t m) {
  return pf_host<Fp, false>(ctx, kind, in, out, log_n, m);
}
int bls_g2_fft_batch(bls_ctx* ctx, int kind, const bls_g2_affine* in, bls_g2_affine* out, int log_n, size_t m) {
  return pf_host<Fp2, true>(ctx, kind, in, out, log_n, m);
}

size_t bls_kzg_open_all_prepare_scratch_bytes(const bls_ctx* ctx, int log_n) {
  if (!ctx || log_n < 0 || log_n > FK_MAX_LOG_N) return 0;
  size_t off_fft;
  return fk_prepare_layout(const_cast<bls_ctx*>(ctx), log_n, off_fft);
}
int bls_kzg_open_all_prepare_dev(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, int log_n, bls_g1_affine* table, void* scratch,
                                 void* stream) {
  return fk_prepare_dev_impl(ctx, srs, srs_len, log_n, table, scratch, stream);
}
int bls_kzg_open_all_prepare(bls_ctx* ctx, const bls_g1_affine* srs, size_t srs_len, int log_n, bls_g1_affine* table) {
  if (!ctx || log_n < 0 || log_n > FK_MAX_LOG_N) return BLS_ERR_INVALID_ARGUMENT;
  const size_t n = (size_t)1 << log_n, ns = n > 1 ? n - 1 : 0;
  if (srs_len < ns || (ns && !srs) || !table) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  size_t off_fft;
  const size_t total = fk_prepare_layout(ctx, log_n, off_fft);
  H2D(dsrs, ns ? srs : nullptr, ns * sizeof(bls_g1_affine));
  DALLOC(dt, 2 * n * sizeof(bls_g1_affine));
  DALLOC(dscr, total);
  TRY(fk_prepare_dev_impl(ctx, (const bls_g1_affine*)dsrs.p, ns, log_n, (bls_g1_affine*)dt.p, dscr.p, ctx->stream));
  D2H(table, dt, 2 * n * sizeof(bls_g1_affine));
  SYNC();
  return BLS_OK;
}

size_t bls_kzg_open_all_scratch_bytes(const bls_ctx* ctx, int log_n, size_t m) {
  if (!ctx || !fk_args_ok(log_n, m)) return 0;
  if (m == 0) return 1;
  FkLayout l;
  return fk_layout(const_cast<bls_ctx*>(ctx), log_n, m, l);
}
int bls_kzg_open_all_dev(bls_ctx* ctx, const bls_g1_affine* table, const bls_fr* p, int log_n, size_t m, bls_fr* y, bls_g1_affine* proof,
                         void* scratch, void* stream) {
  return fk_open_all_dev_impl(ctx, table, p, log_n, m, y, proof, scratch, stream);
}
int bls_kzg_open_all_batch(bls_ctx* ctx, const bls_g1_affine* table, const bls_fr* p, int log_n, size_t m, bls_fr* y, bls_g1_affine* proof) {
  if (!ctx || !fk_args_ok(log_n, m)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  if (!table || !p || !y || !proof) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  FkLayout l;
  if (!fk_layout(ctx, log_n, m, l)) return BLS_ERR_CUDA;
  const size_t n = (size_t)1 << log_n;
  H2D(dt, table, 2 * n * sizeof(bls_g1_affine));
  H2D(dp, p, m * n * sizeof(bls_fr));
  DALLOC(dy, m * n * sizeof(bls_fr));
  DALLOC(dpr, m * n * sizeof(bls_g1_affine));
  DALLOC(dscr, l.total);
  TRY(fk_open_all_dev_impl(ctx, (const bls_g1_affine*)dt.p, (const bls_fr*)dp.p, log_n, m, (bls_fr*)dy.p, (bls_g1_affine*)dpr.p, dscr.p,
                           ctx->stream));
  D2H(y, dy, m * n * sizeof(bls_fr));
  D2H(proof, dpr, m * n * sizeof(bls_g1_affine));
  SYNC();
  return BLS_OK;
}

}  // extern "C"
