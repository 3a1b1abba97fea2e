// kernels_fft.cu -- radix-2 FFT over Fr for batches of polynomials (bellman's EvaluationDomain: fft, ifft, coset_fft,
// icoset_fft) and its entry points.  Its own translation unit (see abi_common.cuh) so that ptxas' allocation of the
// existing kernels cannot move.  The arithmetic is fr.cuh's: every value is canonical (< r) between operations.
//
// A transform of n = 2^L points runs as P = ceil(L / 10) Stockham passes of radix 2^deg (deg <= 10, the L stages split
// evenly), natural order in and out, each pass one read and one write of HBM:
//   pass (lgp = stages already done, deg): group gp (of n / 2^deg per polynomial) reads x[gp + i * n / 2^deg], i < 2^deg,
//   scales element i by w^(e), e = (k * i) << (L - lgp - deg) with k = gp mod 2^lgp (the inter-pass twiddle; none in the
//   first pass), runs deg decimation-in-frequency stages in shared memory and writes its outputs in bit-reversed order
//   to y[((gp - k) << deg) + k + j * 2^lgp], j < 2^deg.
// A block holds 2^10 elements: 2^(10 - deg) consecutive groups, which for a one-pass transform (L <= 10) are
// 2^(10 - L) whole polynomials.  The coset scaling g^j rides on the first pass's loads, the n^-1 and g^-j scaling of
// the inverse kinds on the last pass's stores.
//
// Twiddles are built on the device by k_fft_tables into the caller's scratch, every entry a product of the powers
// x^(2^b) of fr_fft_consts.cuh: w^e = T_hi[e >> s] * T_lo[e & (2^s - 1)] (s = ceil(L / 2)), the same two-level scheme
// for g^(+-j), and the stage table S[bit + di] = omega_(2 bit)^di that the butterflies read.
//
// Groth16's quotient polynomial (bls_fr_groth16_h_*) runs on the same transforms: gather and pad, ifft and coset_fft of
// all 3m polynomials in two calls, the element-wise (A B - C) z(g)^-1, icoset_fft of the m results, conversion to
// FrRepr without the last coefficient.  The element-wise steps are kernels of their own, not fused into k_fr_fft_pass.
#include "abi_common.cuh"
#include "fr_fft_consts.cuh"

#define FFT_D 10                           /* stages per pass at most */
#define FFT_ELEMS (1u << FFT_D)            /* elements in a block's shared memory (32 KB) */
#define FFT_TPB 256
#define FFT_MINB 3
#define FFT_MAX_LOG_N 28
#define FFT_MAX_ELEMS ((size_t)1 << 30)    /* m * 2^log_n */

// 8-byte loads and stores: the ABI's bls_fr rows are arrays of u64
__device__ __forceinline__ Fr ld_fr(const Fr* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void st_fr(Fr* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}

// x^e for e < 2^32 from the table pw[b] = x^(2^b): the product of the entries at the set bits of e
__device__ __forceinline__ Fr fft_pow_bits(const Fr* pw, uint32_t e) {
  Fr r = fr_one();
  bool started = false;
#pragma unroll 1
  for (int b = 0; e; b++, e >>= 1) {
    if (e & 1) { r = started ? fr_mul(r, pw[b]) : pw[b]; started = true; }
  }
  return r;
}

// One thread per table entry: tw_lo[i] = w^i (i < 2^s), tw_hi[i] = w^(i 2^s), stage[bit + di] = omega_(2 bit)^di, and for
// the coset kinds cs_lo[i] = g^(+-i) (times n^-1 for icoset_fft), cs_hi[i] = g^(+-i 2^s).  w = omega^(+-1).
__global__ void __launch_bounds__(128) k_fft_tables(int kind, int L, int s, Fr* tw_lo, Fr* tw_hi, Fr* stage, Fr* cs_lo, Fr* cs_hi) {
  uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  const bool inv = kind == BLS_IFFT || kind == BLS_ICOSET_FFT;
  const Fr* rp = inv ? FR_ROOT_INV_POW : FR_ROOT_POW;
  const uint32_t nlo = 1u << s, nhi = 1u << (L - s);
  if (id < nlo) { tw_lo[id] = fft_pow_bits(rp + 32 - L, id); return; }
  id -= nlo;
  if (id < nhi) { tw_hi[id] = fft_pow_bits(rp + 32 - L + s, id); return; }
  id -= nhi;
  if (id < FFT_ELEMS) {
    if (id == 0) { stage[0] = fr_one(); return; }
    const int lb = 31 - __clz(id);                      // bit = 2^lb, omega_(2 bit) = omega_32^(2^(31 - lb))
    stage[id] = fft_pow_bits(rp + 31 - lb, id - (1u << lb));
    return;
  }
  id -= FFT_ELEMS;
  if (kind != BLS_COSET_FFT && kind != BLS_ICOSET_FFT) return;
  const Fr* gp = kind == BLS_COSET_FFT ? FR_GEN_POW : FR_GEN_INV_POW;
  if (id < nlo) {
    const Fr v = fft_pow_bits(gp, id);
    cs_lo[id] = kind == BLS_ICOSET_FFT ? fr_mul(v, FR_INV_2POW[L]) : v;
    return;
  }
  id -= nlo;
  if (id < nhi) cs_hi[id] = fft_pow_bits(gp + s, id);
}

// x^e from a two-level table (lo[0] may carry a factor, so only the hi == 0 case skips the product)
__device__ __forceinline__ Fr fft_pow2(const Fr* lo, const Fr* hi, uint32_t e, int s) {
  const uint32_t h = e >> s;
  const Fr l = ld_fr(lo + (e & ((1u << s) - 1)));
  return h ? fr_mul(l, ld_fr(hi + h)) : l;
}

struct FftPass {
  const Fr* x;
  Fr* y;
  const Fr *tw_lo, *tw_hi, *stage, *cs_lo, *cs_hi;
  size_t groups;         // m * 2^(L - deg)
  int L, s, lgp, deg;
  int pre;               // 1: element j of the input times g^j (coset_fft, first pass)
  int post;              // 1: output times n^-1 (ifft); 2: output o times g^-o n^-1 (icoset_fft); last pass only
};

// Shared memory is word-sliced (word w of element e at sm[w][e]) and XOR-swizzled within each group, so that the
// loads (consecutive groups), the butterflies (consecutive i) and the bit-reversed stores (consecutive j) of a warp
// fall on distinct banks.
__device__ __forceinline__ uint32_t fft_pos(uint32_t gl, uint32_t i, int deg) {
  return (gl << deg) | (i ^ (((i >> 5) ^ (__brev(gl) >> 27)) & 31u & ((1u << deg) - 1)));
}
__device__ __forceinline__ Fr ld_sm(const uint32_t (*sm)[FFT_ELEMS], uint32_t pos) {
  Fr r;
#pragma unroll
  for (int w = 0; w < 8; w++) r.v[w] = sm[w][pos];
  return r;
}
__device__ __forceinline__ void st_sm(uint32_t (*sm)[FFT_ELEMS], uint32_t pos, const Fr& a) {
#pragma unroll
  for (int w = 0; w < 8; w++) sm[w][pos] = a.v[w];
}

__global__ void __launch_bounds__(FFT_TPB, FFT_MINB) k_fr_fft_pass(const FftPass P) {
  __shared__ uint32_t sm[8][FFT_ELEMS];
  const int deg = P.deg, lgG = FFT_D - deg, lgq = P.L - deg;     // 2^lgG groups per block, 2^lgq groups per polynomial
  const uint32_t R = 1u << deg, G = 1u << lgG, p = 1u << P.lgp;
  const size_t g0 = (size_t)blockIdx.x << lgG, n = (size_t)1 << P.L, t = n >> deg, qmask = ((size_t)1 << lgq) - 1;
#pragma unroll 1
  for (uint32_t idx = threadIdx.x; idx < FFT_ELEMS; idx += FFT_TPB) {
    const uint32_t i = idx >> lgG, gl = idx & (G - 1);
    const size_t g = g0 + gl;
    if (g >= P.groups) continue;
    const size_t gp = g & qmask, j = gp + (size_t)i * t;
    Fr v = ld_fr(P.x + (g >> lgq) * n + j);
    if (P.pre) v = fr_mul(v, fft_pow2(P.cs_lo, P.cs_hi, (uint32_t)j, P.s));
    if (P.lgp) {
      const uint32_t e = (((uint32_t)gp & (p - 1)) * i) << (P.L - P.lgp - deg);
      if (e) v = fr_mul(v, fft_pow2(P.tw_lo, P.tw_hi, e, P.s));
    }
    st_sm(sm, fft_pos(gl, i, deg), v);
  }
  __syncthreads();
#pragma unroll 1
  for (int rnd = 0; rnd < deg; rnd++) {
    const uint32_t bit = (R >> 1) >> rnd;
#pragma unroll 1
    for (uint32_t b = threadIdx.x; b < FFT_ELEMS / 2; b += FFT_TPB) {
      const uint32_t gl = b >> (deg - 1), i = b & ((R >> 1) - 1);
      const uint32_t di = i & (bit - 1), i0 = (i << 1) - di;
      const uint32_t p0 = fft_pos(gl, i0, deg), p1 = fft_pos(gl, i0 + bit, deg);
      const Fr a = ld_sm(sm, p0), c = ld_sm(sm, p1);
      st_sm(sm, p0, fr_add(a, c));
      Fr d = fr_sub(a, c);
      if (di) d = fr_mul(d, ld_fr(P.stage + bit + di));
      st_sm(sm, p1, d);
    }
    __syncthreads();
  }
  // output slot (group gl, j) in the order of the destination addresses: runs of min(2^lgp, G) groups, then j
  const int lP = P.lgp < lgG ? P.lgp : lgG;
#pragma unroll 1
  for (uint32_t idx = threadIdx.x; idx < FFT_ELEMS; idx += FFT_TPB) {
    const uint32_t lo = idx & ((1u << lP) - 1), jj = (idx >> lP) & (R - 1), gl = ((idx >> (lP + deg)) << lP) | lo;
    const size_t g = g0 + gl;
    if (g >= P.groups) continue;
    const size_t gp = g & qmask, k = gp & (p - 1), o = ((gp - k) << deg) + k + (size_t)jj * p;
    Fr v = ld_sm(sm, fft_pos(gl, deg ? __brev(jj) >> (32 - deg) : 0, deg));
    if (P.post == 1) v = fr_mul(v, FR_INV_2POW[P.L]);
    else if (P.post == 2) v = fr_mul(v, fft_pow2(P.cs_lo, P.cs_hi, (uint32_t)o, P.s));
    st_fr(P.y + (g >> lgq) * n + o, v);
  }
}

// ---- Groth16's quotient polynomial H (bellman's groth16::create_proof, the `h` block) ---------------------------------
// m proofs of len evaluations in each of a, b, c; the work buffer holds 3m polynomials of n = 2^L: A_0 .. A_(m-1),
// B_0 .. B_(m-1), C_0 .. C_(m-1), so that one transform call covers all 3m and the A regions are the first m.

// one thread per element of the work buffer: EvaluationDomain::from_coeffs (copy, zero-pad to n)
__global__ void __launch_bounds__(128) k_fr_h_gather(const Fr* a, const Fr* b, const Fr* c, size_t len, size_t m, int L, Fr* w) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= 3 * (m << L)) return;
  const size_t poly = id >> L, i = id & (((size_t)1 << L) - 1), which = poly / m, j = poly - which * m;
  const Fr* src = which == 0 ? a : which == 1 ? b : c;
  st_fr(w + id, i < len ? ld_fr(src + j * len + i) : fr_zero());
}

// one thread per element of the A regions: a.mul_assign(&b), a.sub_assign(&c), divide_by_z_on_coset -- (A B - C) z(g)^-1
__global__ void __launch_bounds__(128) k_fr_h_combine(Fr* w, size_t mn, int L) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= mn) return;
  const Fr x = fr_mul(ld_fr(w + id), ld_fr(w + mn + id));
  st_fr(w + id, fr_mul(fr_sub(x, ld_fr(w + 2 * mn + id)), FR_Z_INV[L]));
}

// one thread per element of the A regions: coefficient i < n - 1 of proof j to h[j (n - 1) + i] as into_repr() (x * 1 R^-1)
__global__ void __launch_bounds__(128) k_fr_into_repr_truncate(const Fr* w, size_t mn, int L, Fr* h) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= mn) return;
  const size_t j = id >> L, i = id & (((size_t)1 << L) - 1);
  if (i == ((size_t)1 << L) - 1) return;                   // the dropped coefficient n - 1
  Fr one = fr_zero();
  one.v[0] = 1;
  st_fr(h + id - j, fr_mul(ld_fr(w + id), one));
}

// ---- host side ----------------------------------------------------------------------------------------------------------

static bool fft_args_ok(int log_n, size_t m) { return log_n >= 0 && log_n <= FFT_MAX_LOG_N && m <= (FFT_MAX_ELEMS >> log_n); }

namespace {
struct FftPlan {
  int L, s, passes, deg[3];
  size_t off_tw_lo, off_tw_hi, off_stage, off_cs_lo, off_cs_hi, off_buf, total;
};
}  // namespace

static size_t fft_align(size_t x) { return (x + 255) & ~(size_t)255; }

// Pass split and scratch layout: the tables, then (two or more passes) one buffer of m * n elements between passes
static void fft_plan(int log_n, size_t m, FftPlan& p) {
  p.L = log_n;
  p.s = (log_n + 1) / 2;
  p.passes = log_n <= FFT_D ? 1 : (log_n + FFT_D - 1) / FFT_D;
  for (int i = 0; i < p.passes; i++) p.deg[i] = log_n / p.passes + (i < log_n % p.passes ? 1 : 0);
  const size_t e = sizeof(bls_fr), nlo = (size_t)1 << p.s, nhi = (size_t)1 << (log_n - p.s);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += fft_align(bytes); return at; };
  p.off_tw_lo = take(nlo * e);
  p.off_tw_hi = take(nhi * e);
  p.off_stage = take(FFT_ELEMS * e);
  p.off_cs_lo = take(nlo * e);
  p.off_cs_hi = take(nhi * e);
  p.off_buf = take(p.passes > 1 ? (m << log_n) * e : 0);
  p.total = o;
}

static int fft_dev_impl(bls_ctx* ctx, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m, void* scratch, void* stream) {
  if (!ctx || kind < BLS_FFT || kind > BLS_ICOSET_FFT || !fft_args_ok(log_n, m) || (m && (!in || !out || !scratch))) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  USE_DEVICE(ctx);
  cudaStream_t st = pick(ctx, stream);
  FftPlan p;
  fft_plan(log_n, m, p);
  char* base = (char*)scratch;
  Fr *tw_lo = (Fr*)(base + p.off_tw_lo), *tw_hi = (Fr*)(base + p.off_tw_hi), *stage = (Fr*)(base + p.off_stage);
  Fr *cs_lo = (Fr*)(base + p.off_cs_lo), *cs_hi = (Fr*)(base + p.off_cs_hi), *buf = (Fr*)(base + p.off_buf);
  const size_t ntab = ((size_t)2 << p.s) + ((size_t)2 << (log_n - p.s)) + FFT_ELEMS;
  k_fft_tables<<<blocks_for(ntab, 128), 128, 0, st>>>(kind, log_n, p.s, tw_lo, tw_hi, stage, cs_lo, cs_hi);
  LAUNCH_CHECK();
  // Buffers of the passes: the last one writes `out`, none reads the buffer it writes.  Three passes in place go
  // through a copy of the input, so that the first pass does not overwrite what the others have yet to read.
  const Fr* src[3];
  Fr* dst[3];
  const size_t bytes = (m << log_n) * sizeof(bls_fr);
  if (p.passes == 1) { src[0] = (const Fr*)in; dst[0] = (Fr*)out; }
  else if (p.passes == 2) { src[0] = (const Fr*)in; dst[0] = buf; src[1] = buf; dst[1] = (Fr*)out; }
  else {
    const Fr* first = (const Fr*)in;
    if ((const void*)in == (void*)out) {
      CK(cudaMemcpyAsync(buf, in, bytes, cudaMemcpyDeviceToDevice, st));
      first = buf;
    }
    src[0] = first; dst[0] = (Fr*)out; src[1] = (Fr*)out; dst[1] = buf; src[2] = buf; dst[2] = (Fr*)out;
  }
  FftPass a;
  a.tw_lo = tw_lo; a.tw_hi = tw_hi; a.stage = stage; a.cs_lo = cs_lo; a.cs_hi = cs_hi;
  a.L = log_n; a.s = p.s;
  int lgp = 0;
  for (int i = 0; i < p.passes; i++) {
    a.x = src[i]; a.y = dst[i];
    a.deg = p.deg[i]; a.lgp = lgp;
    a.groups = m << (log_n - p.deg[i]);
    a.pre = i == 0 && kind == BLS_COSET_FFT;
    a.post = i + 1 < p.passes ? 0 : kind == BLS_IFFT ? 1 : kind == BLS_ICOSET_FFT ? 2 : 0;
    k_fr_fft_pass<<<blocks_for(a.groups, 1 << (FFT_D - p.deg[i])), FFT_TPB, 0, st>>>(a);
    LAUNCH_CHECK();
    lgp += p.deg[i];
  }
  return BLS_OK;
}

static int fft_host(bls_ctx* ctx, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m) {
  if (!ctx || kind < BLS_FFT || kind > BLS_ICOSET_FFT || !fft_args_ok(log_n, m) || (m && (!in || !out))) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0) return BLS_OK;
  USE_DEVICE(ctx);
  const size_t bytes = (m << log_n) * sizeof(bls_fr);
  FftPlan p;
  fft_plan(log_n, m, p);
  H2D(din, in, bytes);
  DALLOC(dout, bytes);
  DALLOC(dscr, p.total);
  TRY(fft_dev_impl(ctx, kind, (const bls_fr*)din.p, (bls_fr*)dout.p, log_n, m, dscr.p, ctx->stream));
  D2H(out, dout, bytes);
  SYNC();
  return BLS_OK;
}

#define GH_MAX_ELEMS ((size_t)1 << 28)     /* m * n, so that the 3m polynomials stay within FFT_MAX_ELEMS */

// n = 2^L, the smallest power of two >= len (1 for len <= 1); false for L > 28 or m * n > 2^28
static bool gh_args_ok(size_t len, size_t m, int& L) {
  if (len > ((size_t)1 << FFT_MAX_LOG_N)) return false;
  for (L = 0; ((size_t)1 << L) < len; L++) {}
  return m <= (GH_MAX_ELEMS >> L);
}

// scratch: the work buffer of 3m * n elements, then the scratch of the 3m-polynomial transforms
static size_t gh_scratch_bytes(int L, size_t m) {
  FftPlan p;
  fft_plan(L, 3 * m, p);
  return fft_align(3 * (m << L) * sizeof(bls_fr)) + p.total;
}

static int groth16_h_dev_impl(bls_ctx* ctx, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h,
                              void* scratch, void* stream) {
  int L;
  if (!ctx || !gh_args_ok(len, m, L)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0 || len <= 1) return BLS_OK;                   // nothing to store: n - 1 = 0 coefficients per proof
  if (!a || !b || !c || !h || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  cudaStream_t st = pick(ctx, stream);
  const size_t mn = m << L, work = fft_align(3 * mn * sizeof(bls_fr));
  Fr* w = (Fr*)scratch;
  void* fscr = (char*)scratch + work;
  k_fr_h_gather<<<blocks_for(3 * mn, 128), 128, 0, st>>>((const Fr*)a, (const Fr*)b, (const Fr*)c, len, m, L, w);
  LAUNCH_CHECK();
  TRY(fft_dev_impl(ctx, BLS_IFFT, (bls_fr*)w, (bls_fr*)w, L, 3 * m, fscr, st));
  TRY(fft_dev_impl(ctx, BLS_COSET_FFT, (bls_fr*)w, (bls_fr*)w, L, 3 * m, fscr, st));
  k_fr_h_combine<<<blocks_for(mn, 128), 128, 0, st>>>(w, mn, L);
  LAUNCH_CHECK();
  TRY(fft_dev_impl(ctx, BLS_ICOSET_FFT, (bls_fr*)w, (bls_fr*)w, L, m, fscr, st));   // the m-polynomial plan fits in the 3m one
  k_fr_into_repr_truncate<<<blocks_for(mn, 128), 128, 0, st>>>(w, mn, L, (Fr*)h);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int groth16_h_host(bls_ctx* ctx, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h) {
  int L;
  if (!ctx || !gh_args_ok(len, m, L)) return BLS_ERR_INVALID_ARGUMENT;
  if (m == 0 || len <= 1) return BLS_OK;
  if (!a || !b || !c || !h) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  const size_t in_bytes = m * len * sizeof(bls_fr), out_bytes = m * (((size_t)1 << L) - 1) * sizeof(bls_fr_repr);
  H2D(da, a, in_bytes);
  H2D(db, b, in_bytes);
  H2D(dc, c, in_bytes);
  DALLOC(dh, out_bytes);
  DALLOC(dscr, gh_scratch_bytes(L, m));
  TRY(groth16_h_dev_impl(ctx, (const bls_fr*)da.p, (const bls_fr*)db.p, (const bls_fr*)dc.p, len, m, (bls_fr_repr*)dh.p, dscr.p, ctx->stream));
  D2H(h, dh, out_bytes);
  SYNC();
  return BLS_OK;
}

extern "C" {

size_t bls_fr_fft_scratch_bytes(const bls_ctx* ctx, int log_n, size_t m) {
  if (!ctx || !fft_args_ok(log_n, m)) return 0;
  FftPlan p;
  fft_plan(log_n, m, p);
  return p.total;
}
int bls_fr_fft_dev(bls_ctx* ctx, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m, void* scratch, void* stream) {
  return fft_dev_impl(ctx, kind, in, out, log_n, m, scratch, stream);
}
int bls_fr_fft_batch(bls_ctx* ctx, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m) { return fft_host(ctx, kind, in, out, log_n, m); }

size_t bls_fr_groth16_h_scratch_bytes(const bls_ctx* ctx, size_t len, size_t m) {
  int L;
  if (!ctx || !gh_args_ok(len, m, L)) return 0;
  return gh_scratch_bytes(L, m);
}
int bls_fr_groth16_h_dev(bls_ctx* ctx, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h,
                         void* scratch, void* stream) {
  return groth16_h_dev_impl(ctx, a, b, c, len, m, h, scratch, stream);
}
int bls_fr_groth16_h_batch(bls_ctx* ctx, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h) {
  return groth16_h_host(ctx, a, b, c, len, m, h);
}

}  // extern "C"
