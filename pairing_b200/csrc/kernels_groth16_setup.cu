// kernels_groth16_setup.cu -- bellman's groth16::generate_parameters from the constraint system and the toxic waste
// (bls_groth16_generate_parameters_*).  Its own translation unit (see abi_common.cuh): the inversions, the inverse FFT, the
// fixed-base wNAF tables and exponentiations and the batch normalisations are the other units' entry points, called through
// the C ABI, so no existing kernel is recompiled.
//
// Pipeline, all on the call's stream (n = 2^L the domain size, nv = num_inputs + num_aux):
//   1. bls_fr_op_dev(INV): gamma^-1, delta^-1.  k_gs_pre (one thread): tau^(2^b) for b <= L by L squarings, z(tau) delta^-1
//      = (tau^n - 1) delta^-1, the six vk scalars, g1 and g2 as Jacobian points.  k_gs_tau_tables: lo[i] = tau^i (i < 2^s),
//      hi[j] = tau^(j 2^s), each a product of at most L entries of the tau^(2^b) table (k_fft_tables' scheme for omega).
//      k_gs_powers: tau^i = lo * hi into the Lagrange buffer, and the h scalars tau^i z(tau) delta^-1, i < n - 1.
//   2. bls_fr_fft_dev(IFFT) in place: Lq = L_q(tau), the Lagrange basis of the omega^q (bellman's powers_of_tau.ifft()).
//   3. k_gs_qap: for A, B and C, one thread per chunk of GS_CHUNK consecutive terms in the variable-major (CSR) order, so the
//      work follows the terms whatever their distribution over the variables.  A thread sums coeff * L[constraint] over each
//      run of one variable in its chunk.  A variable whose terms all lie in the chunk is stored; the runs of a variable that
//      crosses chunk boundaries are added, as their 8 32-bit limbs, into 8 u64 counters owned by the chunk that holds the
//      variable's first term (atomicAdd; at most 2^31 terms, so no counter overflows).  Integer sums are exact, so the
//      result does not depend on the order of the atomics.
//   4. k_gs_query: one thread per variable: u, v, w (the spanning ones reduced mod r from the counters), the scalars
//      into_repr((beta u + alpha v + w) gamma^-1) (ic) or delta^-1 (l), into_repr(u) (a) and into_repr(v) (b_g1, b_g2), and a
//      warp ballot of u != 0 and v != 0: the density words over all variables.  It also flags malformed CSR (the _dev form)
//      and l scalars equal to zero (UnconstrainedVariable).
//   5. bls_g*_wnaf_table_dev on g1 and g2, bls_g*_wnaf_fixed_base_dev over every G1 and every G2 scalar.  The G1 batch is
//      [alpha, beta, delta | ic | l | h | u for every variable | v for every variable], the G2 batch [beta, gamma, delta | v
//      for every variable]: zero scalars give the identity.
//   6. k_gs_scan (one block): exclusive prefixes of the density words' popcounts, a_len and b_len, and the three density
//      bitmaps of the key in the prover's format.
//   7. bls_g*_batch_normalization_dev, then k_gs_emit: one thread per point: the affine row, the a and b rows at their ranks
//      (rank = prefix of the word + popcount below the bit) with the identities dropped, and `ok`.
// g1 and g2 have order r (bellman's generators), so [k]g is the identity exactly when k = 0: the filters are decided on the
// scalars, which is bellman's rule on the points.
//
// bls_groth16_mpc_new_* (phase 2 of the ceremony, include/pairing_b200_mpc.h) shares steps 6 and 7: its sums are points
// from the start (k_mpc_qap, k_mpc_fix and k_mpc_combine below), so the filters are decided on the Jacobian sums.
#include "curve_io.cuh"
#include "fr.cuh"
#include "../../include/pairing_b200_mpc.h"

#define GS_TPB 128
#define GS_SCAN_TPB 1024
#define GS_CHUNK 32                        /* terms per thread of k_gs_qap */
#define GS_MAX_N ((size_t)1 << 26)         /* domain size and number of variables: every query fits the prover's 2^26 */
#define GS_MAX_NNZ ((size_t)1 << 31)       /* terms per matrix, exclusive */
// Fixed-base windows.  Not chosen by a measurement: the sweep of tools/bench_groth16_setup.py --sweep has not been run on a
// GPU yet (DESIGN.md "Groth16 generator").  12 / 11 trade the one-warp table build (2^(w-1) sequential additions) against
// the ~256 / (w + 1) additions per scalar that the doublings of every scalar dwarf anyway.
#define GS_WINDOW_G1 12
#define GS_WINDOW_G2 11

// the small scalars in scratch, Fr (4 u64) slots
#define GS_ALPHA 0
#define GS_BETA 1
#define GS_GAMMA 2
#define GS_DELTA 3
#define GS_TAU 4
#define GS_GAMMA_INV 5
#define GS_DELTA_INV 6
#define GS_ZD 7                            /* (tau^n - 1) delta^-1 */
#define GS_TPOW 8                          /* tau^(2^b), b = 0 .. L */
#define GS_NSC (GS_TPOW + 27)
// flags word: bit 0 = malformed CSR term or offsets, bit 1 = an l scalar is zero
#define GS_BAD_CSR 1u
#define GS_UNCONSTRAINED 2u

// bls_groth16_vk_points in u64 words
#define GSV_ALPHA1 0
#define GSV_BETA1 G1A_W
#define GSV_DELTA1 (2 * G1A_W)
#define GSV_BETA2 (3 * G1A_W)
#define GSV_GAMMA2 (3 * G1A_W + G2A_W)
#define GSV_DELTA2 (3 * G1A_W + 2 * G2A_W)

__device__ __forceinline__ Fr gs_ld_fr(const uint64_t* p) {
  Fr r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { const uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
__device__ __forceinline__ void gs_st_fr(uint64_t* p, const Fr& a) {
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
// into_repr(): the Montgomery product with 1
__device__ __forceinline__ Fr gs_into_repr(const Fr& x) {
  Fr one = fr_zero();
  one.v[0] = 1;
  return fr_mul(x, one);
}
// x^e for e < 2^32 from pw[b] = x^(2^b)
__device__ __forceinline__ Fr gs_pow_bits(const uint64_t* pw, uint32_t e) {
  Fr r = fr_one();
  bool started = false;
#pragma unroll 1
  for (int b = 0; e; b++, e >>= 1) {
    if (e & 1) {
      const Fr x = gs_ld_fr(pw + 4 * b);
      r = started ? fr_mul(r, x) : x;
      started = true;
    }
  }
  return r;
}

// One thread: the tau^(2^b) table, z(tau) delta^-1, the vk scalars (G1: alpha, beta, delta; G2: beta, gamma, delta) and
// the Jacobian bases of the wNAF tables.
__global__ void k_gs_pre(uint64_t* sc, int L, const uint64_t* g1a, const uint64_t* g2a, uint64_t* g1j, uint64_t* g2j, uint64_t* s1,
                         uint64_t* s2) {
  Fr t = gs_ld_fr(sc + 4 * GS_TAU);
#pragma unroll 1
  for (int b = 0; b <= L; b++) {
    gs_st_fr(sc + 4 * (GS_TPOW + b), t);
    t = fr_sqr(t);
  }
  const Fr tn = gs_ld_fr(sc + 4 * (GS_TPOW + L));
  gs_st_fr(sc + 4 * GS_ZD, fr_mul(fr_sub(tn, fr_one()), gs_ld_fr(sc + 4 * GS_DELTA_INV)));
  const int g1s[3] = {GS_ALPHA, GS_BETA, GS_DELTA}, g2s[3] = {GS_BETA, GS_GAMMA, GS_DELTA};
#pragma unroll
  for (int i = 0; i < 3; i++) {
    gs_st_fr(s1 + 4 * i, gs_into_repr(gs_ld_fr(sc + 4 * g1s[i])));
    gs_st_fr(s2 + 4 * i, gs_into_repr(gs_ld_fr(sc + 4 * g2s[i])));
  }
  Aff<Fp> a1;
  ld_aff(a1, g1a);
  Jac<Fp> j1{a1.x, a1.y, fp_one()};
  st_jac(g1j, j1);
  Aff<Fp2> a2;
  ld_aff(a2, g2a);
  Jac<Fp2> j2;
  j2.x = a2.x; j2.y = a2.y; f_set_one(j2.z);
  st_jac(g2j, j2);
}

__global__ void __launch_bounds__(GS_TPB) k_gs_tau_tables(const uint64_t* sc, int L, int s, uint64_t* lo, uint64_t* hi) {
  uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t nlo = 1u << s, nhi = 1u << (L - s);
  if (id < nlo) { gs_st_fr(lo + 4 * (size_t)id, gs_pow_bits(sc + 4 * GS_TPOW, id)); return; }
  id -= nlo;
  if (id < nhi) gs_st_fr(hi + 4 * (size_t)id, gs_pow_bits(sc + 4 * (GS_TPOW + s), id));
}

// tau^i into lag[i] (Montgomery, the IFFT's input) and, for i < n - 1, into_repr(tau^i z(tau) delta^-1) into hs[i]
__global__ void __launch_bounds__(GS_TPB) k_gs_powers(const uint64_t* sc, const uint64_t* lo, const uint64_t* hi, int s, size_t n, uint64_t* lag,
                                                      uint64_t* hs) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Fr p = fr_mul(gs_ld_fr(lo + 4 * (i & ((1u << s) - 1))), gs_ld_fr(hi + 4 * (i >> s)));
  gs_st_fr(lag + 4 * i, p);
  if (i + 1 < n) gs_st_fr(hs + 4 * i, gs_into_repr(fr_mul(p, gs_ld_fr(sc + 4 * GS_ZD))));
}

// One matrix of the system in device memory, with the clamped reads every kernel uses: whatever the offsets hold, an offset
// read is at most nnz and every term index stays below nnz.
struct GsMat {
  const uint64_t* off;
  const uint32_t* cons;
  const uint64_t* coeff;
  size_t nnz;
  __device__ __forceinline__ size_t ov(size_t v) const { const uint64_t o = off[v]; return o < nnz ? (size_t)o : nnz; }
};
struct GsMats { GsMat m[3]; };

// the last variable v in [lo, hi] with offset <= e (lo when there is none): a binary search, O(log nv) reads
__device__ __forceinline__ size_t gs_last_at(const GsMat& M, size_t lo, size_t hi, size_t e) {
  while (lo < hi) {
    const size_t mid = (lo + hi + 1) >> 1;
    if (M.ov(mid) <= e) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Adds the runs of one slot to their counters: the lanes of a warp that hold the same counter index are summed first (16-bit
// halves of the limbs, so the 32-bit warp reduction cannot overflow), and one lane of each group does the 8 atomicAdds.
// A variable such as ONE that spans the chunks of a whole warp thus costs one set of atomics per warp, not per thread.
// Every lane of the warp calls it; key = ~0 marks a lane without a run in this slot.
__device__ __forceinline__ void gs_flush_runs(unsigned long long* ac, unsigned long long key, const Fr& sum) {
  const unsigned lane = threadIdx.x & 31;
  const unsigned m = __match_any_sync(0xffffffffu, key == ~0ull ? ~0ull - 1 - lane : key);
  if (key == ~0ull) return;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const unsigned lo = __reduce_add_sync(m, sum.v[i] & 0xffffu), hi = __reduce_add_sync(m, sum.v[i] >> 16);
    if (lane == (unsigned)(__ffs(m) - 1)) atomicAdd(ac + 8 * key + i, (unsigned long long)lo + ((unsigned long long)hi << 16));
  }
}

// blockIdx.y = matrix (A, B, C).  Thread k sums the terms kC .. kC + C - 1; uvw[mat * nv + v] receives the complete
// variables, acc[(mat * chunks_max + kf) * 8 + limb] the runs of the others (kf = chunk of the variable's first term).
__global__ void __launch_bounds__(GS_TPB) k_gs_qap(GsMats mats, size_t nv, size_t nc, size_t chunks_max, const uint64_t* lag, uint64_t* uvw,
                                                   unsigned long long* acc, uint32_t* flags) {
  const GsMat M = blockIdx.y == 0 ? mats.m[0] : blockIdx.y == 1 ? mats.m[1] : mats.m[2];   // constant indices: no local copy
  const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t chunks = (M.nnz + GS_CHUNK - 1) / GS_CHUNK;
  // no early return: the warp aggregates its counter additions below with full-warp intrinsics
  const bool active = k < chunks && nv != 0;
  const size_t e0 = k * GS_CHUNK, e1 = !active ? e0 : e0 + GS_CHUNK < M.nnz ? e0 + GS_CHUNK : M.nnz;
  uint64_t* out = uvw + 4 * nv * blockIdx.y;
  unsigned long long* ac = acc + 8 * chunks_max * blockIdx.y;
  uint32_t bad = 0;
  // a well-formed chunk has at most two runs that cross its boundaries (its first and its last): they wait here
  unsigned long long key0 = ~0ull, key1 = ~0ull;
  Fr sum0 = fr_zero(), sum1 = fr_zero();
  size_t e = e0, v = active ? gs_last_at(M, 0, nv - 1, e0) : 0;
#pragma unroll 1
  while (e < e1) {
    const size_t o1 = M.ov(v + 1);
    const size_t end = o1 < e ? e : (o1 < e1 ? o1 : e1);
    if (end > e) {
      Fr sum = fr_zero();
#pragma unroll 1
      for (; e < end; e++) {
        const uint32_t q = M.cons[e];
        const Fr c = gs_ld_fr(M.coeff + 4 * e);
        if (q >= nc || fr_geq(c, fr_modulus())) { bad = 1; continue; }   // a malformed term contributes zero
        sum = fr_add(sum, fr_mul(c, gs_ld_fr(lag + 4 * (size_t)q)));
      }
      size_t kf = M.ov(v) / GS_CHUNK;
      if (kf >= chunks) kf = chunks - 1;
      if (kf == (o1 - 1) / GS_CHUNK) {
        gs_st_fr(out + 4 * v, sum);
      } else if (key0 == ~0ull) {
        key0 = kf; sum0 = sum;
      } else if (key1 == ~0ull) {
        key1 = kf; sum1 = sum;
      } else {                                                            // only malformed offsets get here
#pragma unroll
        for (int i = 0; i < 8; i++) atomicAdd(ac + 8 * kf + i, (unsigned long long)sum.v[i]);
      }
    }
    if (v + 1 >= nv) break;
    v = gs_last_at(M, v + 1, nv - 1, e);   // the variables without terms at offset e are jumped over, not walked
  }
  gs_flush_runs(ac, key0, sum0);
  gs_flush_runs(ac, key1, sum1);
  if (bad) atomicOr(flags, GS_BAD_CSR);
}

// sum_i c[i] 2^(32 i) mod r (Montgomery representations add as integers): the low 256 bits are < 3r, the rest h < 2^64 is
// h 2^256 = fr_mul(h, R^2)
__device__ __forceinline__ Fr gs_reduce_counters(const unsigned long long* c) {
  Fr lo;
  unsigned long long carry = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const unsigned long long t = c[i] + carry;
    lo.v[i] = (uint32_t)t;
    carry = t >> 32;
  }
  Fr h = fr_zero();
  h.v[0] = (uint32_t)carry;
  h.v[1] = (uint32_t)(carry >> 32);
  return fr_add(fr_reduce(fr_reduce(lo)), fr_mul(h, fr_r2()));
}

// u, v or w of variable t from the outputs of k_gs_qap; flags offsets that are not a CSR index
__device__ __forceinline__ Fr gs_qap_value(const GsMat& M, size_t t, size_t nv, const uint64_t* uvw, const unsigned long long* ac, uint32_t& bad) {
  const uint64_t a = M.off[t], b = M.off[t + 1];
  if (a > b || b > M.nnz || (t == 0 && a != 0) || (t + 1 == nv && b != M.nnz)) bad = 1;
  const size_t o0 = M.ov(t), o1 = M.ov(t + 1);
  if (o1 <= o0) return fr_zero();
  const size_t chunks = (M.nnz + GS_CHUNK - 1) / GS_CHUNK;
  size_t kf = o0 / GS_CHUNK;
  if (kf >= chunks) kf = chunks - 1;
  if (kf == (o1 - 1) / GS_CHUNK) return gs_ld_fr(uvw + 4 * t);
  return gs_reduce_counters(ac + 8 * kf);
}

// one thread per variable; s1 points at the G1 batch's ic block (ic | l | h | a | b follow), sb2 at the G2 batch's b block
__global__ void __launch_bounds__(GS_TPB) k_gs_query(GsMats mats, size_t ni, size_t nv, size_t n1, size_t chunks_max, const uint64_t* sc,
                                                     const uint64_t* uvw, const unsigned long long* acc, uint64_t* s1, uint64_t* sb2,
                                                     uint32_t* wa, uint32_t* wb, uint32_t* flags) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool nz_u = false, nz_v = false;
  if (t < nv) {
    uint32_t bad = 0;
    Fr x[3];
#pragma unroll
    for (int m = 0; m < 3; m++) x[m] = gs_qap_value(mats.m[m], t, nv, uvw + 4 * nv * m, acc + 8 * chunks_max * m, bad);
    const Fr k = fr_add(fr_add(fr_mul(gs_ld_fr(sc + 4 * GS_BETA), x[0]), fr_mul(gs_ld_fr(sc + 4 * GS_ALPHA), x[1])), x[2]);
    const Fr sk = fr_mul(k, gs_ld_fr(sc + 4 * (t < ni ? GS_GAMMA_INV : GS_DELTA_INV)));
    if (t >= ni && fr_is_zero(sk)) bad |= 2;
    gs_st_fr(s1 + 4 * t, gs_into_repr(sk));
    uint64_t* sa = s1 + 4 * (nv + n1);
    gs_st_fr(sa + 4 * t, gs_into_repr(x[0]));
    const Fr rv = gs_into_repr(x[1]);
    gs_st_fr(sa + 4 * (nv + t), rv);
    gs_st_fr(sb2 + 4 * t, rv);
    nz_u = !fr_is_zero(x[0]);
    nz_v = !fr_is_zero(x[1]);
    if (bad) atomicOr(flags, (bad & 1 ? GS_BAD_CSR : 0u) | (bad & 2 ? GS_UNCONSTRAINED : 0u));
  }
  const uint32_t ba = __ballot_sync(0xffffffffu, nz_u), bb = __ballot_sync(0xffffffffu, nz_v);
  if ((threadIdx.x & 31) == 0 && t < nv) { wa[t >> 5] = ba; wb[t >> 5] = bb; }
}

// bits [bit, bit + 32) of a bitmap of `words` words
__device__ __forceinline__ uint32_t gs_bits_at(const uint32_t* w, size_t words, size_t bit) {
  const size_t i = bit >> 5;
  const uint32_t sh = bit & 31, a = i < words ? w[i] : 0u, b = i + 1 < words ? w[i + 1] : 0u;
  return sh ? (a >> sh) | (b << (32 - sh)) : a;
}

// One block: exclusive word prefixes pa, pb of popc(wa), popc(wb), lens = [a_len, b_len], and the key's density bitmaps
__global__ void __launch_bounds__(GS_SCAN_TPB) k_gs_scan(const uint32_t* wa, const uint32_t* wb, size_t words, size_t ni, size_t na, uint32_t* pa,
                                                         uint32_t* pb, uint64_t* lens, uint32_t* a_aux, uint32_t* b_in, uint32_t* b_aux) {
  __shared__ uint32_t sa[GS_SCAN_TPB], sb[GS_SCAN_TPB];
  const size_t per = (words + GS_SCAN_TPB - 1) / GS_SCAN_TPB, w0 = threadIdx.x * per;
  const size_t w1 = w0 + per < words ? w0 + per : words;
  uint32_t ca = 0, cb = 0;
  for (size_t i = w0; i < w1; i++) { ca += __popc(wa[i]); cb += __popc(wb[i]); }
  sa[threadIdx.x] = ca;
  sb[threadIdx.x] = cb;
  __syncthreads();
  for (int d = 1; d < GS_SCAN_TPB; d <<= 1) {    // inclusive Hillis-Steele scan
    const uint32_t xa = threadIdx.x >= d ? sa[threadIdx.x - d] : 0u, xb = threadIdx.x >= d ? sb[threadIdx.x - d] : 0u;
    __syncthreads();
    sa[threadIdx.x] += xa;
    sb[threadIdx.x] += xb;
    __syncthreads();
  }
  ca = sa[threadIdx.x] - ca;
  cb = sb[threadIdx.x] - cb;
  for (size_t i = w0; i < w1; i++) {
    pa[i] = ca; pb[i] = cb;
    ca += __popc(wa[i]); cb += __popc(wb[i]);
  }
  if (threadIdx.x == 0) { lens[0] = sa[GS_SCAN_TPB - 1]; lens[1] = sb[GS_SCAN_TPB - 1]; }
  const size_t wi = (ni + 31) / 32, wx = (na + 31) / 32;
  for (size_t i = threadIdx.x; i < wi; i += GS_SCAN_TPB) {
    const size_t rest = ni - 32 * i;
    b_in[i] = rest >= 32 ? wb[i] : wb[i] & ((1u << rest) - 1u);
  }
  for (size_t i = threadIdx.x; i < wx; i += GS_SCAN_TPB) {    // bits past nv are zero in wa and wb
    a_aux[i] = gs_bits_at(wa, words, ni + 32 * i);
    b_aux[i] = gs_bits_at(wb, words, ni + 32 * i);
  }
}

template <class F> __device__ __forceinline__ void gs_emit_row(uint64_t* dst, const uint64_t* src) {
  Jac<F> p;
  ld_jac(p, src);
  Aff<F> a;
  if (pt_is_zero(p)) { f_set_zero(a.x); f_set_one(a.y); a.inf = true; }   // normalised: z is one or zero
  else { a.x = p.x; a.y = p.y; a.inf = false; }
  st_aff(dst, a);
}
// rank of bit i among the set bits, or -1 when it is clear
__device__ __forceinline__ long long gs_rank(const uint32_t* w, const uint32_t* pre, size_t i) {
  const uint32_t x = w[i >> 5], bit = 1u << (i & 31);
  return (x & bit) ? (long long)(pre[i >> 5] + __popc(x & (bit - 1u))) : -1;
}

struct GsOut {
  uint64_t *vk, *ic, *h, *l, *a, *b_g1, *b_g2;
  uint8_t* ok;
};
// blockIdx.y = 0: G1 rows [alpha, beta, delta | ic | l | h | a | b]; 1: G2 rows [beta, gamma, delta | b]
__global__ void __launch_bounds__(GS_TPB) k_gs_emit(const uint64_t* p1, const uint64_t* p2, size_t ni, size_t na, size_t n1, const uint32_t* wa,
                                                    const uint32_t* pa, const uint32_t* wb, const uint32_t* pb, const uint32_t* flags, GsOut o) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nv = ni + na;
  if (blockIdx.y == 1) {
    if (t >= 3 + nv) return;
    uint64_t* dst;
    if (t < 3) dst = o.vk + (t == 0 ? GSV_BETA2 : t == 1 ? GSV_GAMMA2 : GSV_DELTA2);
    else {
      const long long r = gs_rank(wb, pb, t - 3);
      if (r < 0) return;
      dst = o.b_g2 + (size_t)G2A_W * r;
    }
    gs_emit_row<Fp2>(dst, p2 + (size_t)G2_W * t);
    return;
  }
  if (t == 0) *o.ok = *flags == 0;
  if (t >= 3 + 2 * nv + n1 + nv) return;
  uint64_t* dst;
  size_t i = t;
  if (i < 3) dst = o.vk + (i == 0 ? GSV_ALPHA1 : i == 1 ? GSV_BETA1 : GSV_DELTA1);
  else if ((i -= 3) < ni) dst = o.ic + (size_t)G1A_W * i;
  else if ((i -= ni) < na) dst = o.l + (size_t)G1A_W * i;
  else if ((i -= na) < n1) dst = o.h + (size_t)G1A_W * i;
  else if ((i -= n1) < nv) {
    const long long r = gs_rank(wa, pa, i);
    if (r < 0) return;
    dst = o.a + (size_t)G1A_W * r;
  } else {
    const long long r = gs_rank(wb, pb, i - nv);
    if (r < 0) return;
    dst = o.b_g1 + (size_t)G1A_W * r;
  }
  gs_emit_row<Fp>(dst, p1 + (size_t)G1_W * t);
}

// ---- phase 2 of the ceremony (bls_groth16_mpc_new_*) ----------------------------------------------------------------------
// The group-valued k_gs_qap: the same per-chunk walk over the CSR terms, with c [L_q(tau)] (a scalar multiplication of the
// transcript's row q) in place of c L_q(tau).  Points cannot be added atomically, so a run of a variable that crosses chunk
// boundaries goes to one of the chunk's two boundary slots (0: the variable started in an earlier chunk, 1: it starts here
// and goes on), and k_mpc_fix adds the slots up.  One launch per (matrix, transcript row set):
//   G1: A x coeffs -> a, A x beta_coeffs, B x coeffs -> b_g1, B x alpha_coeffs, C x coeffs; G2: B x coeffs_g2 -> b_g2.
// k_mpc_combine then adds the three ext parts, and decides densities and flags on the Jacobian sums (z = 0 is exact).
#define MPC_CHUNK 12                       /* terms per thread: 4 groups of MPC_K_G1, 6 of MPC_K_G2 */
#define MPC_K_G1 3                         /* points per thread of the wNAF runner, as the library's wNAF kernels */
#define MPC_K_G2 2
#define MPC_MAXT 8                         /* wNAF table entries: window <= 4 */
#define MPC_INCONSISTENT 4u                /* flags bit: bg1_v and bg2_v disagree on being the identity */

template <class F, int K> struct MpcTables {
  Jac<F> t[K][MPC_MAXT];
  __device__ __forceinline__ Jac<F> get(int j, int e) const { return t[j][e]; }
};

// c (Montgomery) as the integer min(c, r - c); neg when r - c was taken.  -1 and -2^k become 1 and 2^k: the window and the
// doublings follow the short value.  [r - c](-P) = [c] P holds for P of order r.
__device__ __forceinline__ Scalar mpc_signed(const Fr& c, bool& neg) {
  const Fr x = gs_into_repr(c), y = gs_into_repr(fr_neg(c));
  neg = !fr_geq(y, x);
  Scalar s;
#pragma unroll
  for (int i = 0; i < 8; i++) s.v[i] = neg ? y.v[i] : x.v[i];
  return s;
}

// a boundary or complete run of variable v from chunk k: complete variables go to sums[v], the others to a boundary slot
template <class F>
__device__ __forceinline__ void mpc_flush(const GsMat& M, size_t v, size_t k, size_t chunks, const Jac<F>& sum, uint64_t* sums, uint64_t* bnd) {
  const int PW = 3 * FW<F>::W;
  size_t kf = M.ov(v) / MPC_CHUNK;
  if (kf >= chunks) kf = chunks - 1;
  const size_t o1 = M.ov(v + 1);
  if (o1 && kf == (o1 - 1) / MPC_CHUNK) st_jac(sums + (size_t)PW * v, sum);
  else st_jac(bnd + (size_t)PW * (2 * k + (kf < k ? 0 : 1)), sum);
}

// Thread k sums c [rows[q]] over the terms kC .. kC + C - 1 of M, K terms at a time through the decoupled wNAF runner.
template <class F, bool IS_G2, int K>
__global__ void __launch_bounds__(GS_TPB, IS_G2 ? 3 : 4)
    k_mpc_qap(GsMat M, size_t nv, size_t nc, const uint64_t* rows, uint64_t* sums, uint64_t* bnd, uint32_t* flags) {
  const int W = FW<F>::W, PW = 3 * W;
  const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t chunks = (M.nnz + MPC_CHUNK - 1) / MPC_CHUNK;
  // no early return: the runner votes with __ballot_sync, so every lane runs the same number of groups
  const bool active = k < chunks && nv != 0;
  const size_t e0 = k * MPC_CHUNK, e1 = !active ? e0 : e0 + MPC_CHUNK < M.nnz ? e0 + MPC_CHUNK : M.nnz;
  Jac<F> sum;
  pt_set_zero(sum);
  if (active) {
    st_jac(bnd + (size_t)PW * 2 * k, sum);
    st_jac(bnd + (size_t)PW * (2 * k + 1), sum);
  }
  uint32_t bad = 0;
  bool open = false;                                        // sum holds terms of v
  size_t v = active ? gs_last_at(M, 0, nv - 1, e0) : 0;
  size_t o1 = active ? M.ov(v + 1) : 0;
#pragma unroll 1
  for (size_t g = e0; g < e0 + MPC_CHUNK; g += K) {
    MpcTables<F, K> table;
    int8_t digits[K][260];
    WnafState<K> st;
    Jac<F> res[K];
    bool neg[K];
#pragma unroll 1
    for (int j = 0; j < K; j++) {
      const size_t e = g + j;
      Scalar s;
#pragma unroll
      for (int i = 0; i < 8; i++) s.v[i] = 0;
      Jac<F> b;
      pt_set_zero(b);
      neg[j] = false;
      if (e < e1) {
        const uint32_t q = M.cons[e];
        const Fr c = gs_ld_fr(M.coeff + 4 * e);
        if (q >= nc || fr_geq(c, fr_modulus())) bad = 1;   // a malformed term contributes the identity
        else {
          s = mpc_signed(c, neg[j]);
          Aff<F> a;
          ld_aff(a, rows + (size_t)(2 * W + 1) * q);
          if (!a.inf) { b.x = a.x; b.y = a.y; f_set_one(b.z); }
        }
      }
      const int w = IS_G2 ? g2_window_for_bits(scalar_num_bits(s)) : g1_window_for_bits(scalar_num_bits(s)), tsize = 1 << (w - 1);
      Jac<F> dbl = b;
      pt_double(dbl);
#pragma unroll 1
      for (int t = 0; t < MPC_MAXT; t++) {
        if (t < tsize) { table.t[j][t] = b; if (t + 1 < tsize) pt_add(b, dbl); }
      }
      st.i[j] = wnaf_form(digits[j], s, w) - 1;
      st.found[j] = false; st.doubled[j] = false;
      pt_set_zero(res[j]);
    }
    pt_wnaf_run_lazy<F, K>(res, table, digits, st);
#pragma unroll 1
    for (int j = 0; j < K; j++) {
      const size_t e = g + j;
      if (e >= e1) break;
      while (e >= o1 && v + 1 < nv) {                       // the run of v ends before term e
        if (open) mpc_flush<F>(M, v, k, chunks, sum, sums, bnd);
        open = false;
        pt_set_zero(sum);
        v = gs_last_at(M, v + 1, nv - 1, e);
        o1 = M.ov(v + 1);
      }
      if (e >= o1) continue;                                // past the last variable: only malformed offsets get here
      if (neg[j]) pt_negate(res[j]);
      pt_add(sum, res[j]);
      open = true;
    }
  }
  if (open) mpc_flush<F>(M, v, k, chunks, sum, sums, bnd);
  if (bad) atomicOr(flags, GS_BAD_CSR);
}

// One block per variable: the identity for a variable without terms; for one whose terms cross chunk boundaries, slot 1 of
// its first chunk plus slot 0 of every later chunk it reaches, strided over the block's threads.  A variable with all terms in
// one chunk was stored by k_mpc_qap.
template <class F>
__global__ void __launch_bounds__(GS_TPB) k_mpc_fix(GsMat M, size_t nv, uint64_t* bnd, uint64_t* sums) {
  const int PW = 3 * FW<F>::W;
  const size_t v = blockIdx.x;
  const int tid = threadIdx.x;
  if (v >= nv) return;                                      // block-uniform, as every return before the barrier
  Jac<F> s;
  pt_set_zero(s);
  const size_t o0 = M.ov(v), o1 = M.ov(v + 1);
  if (o1 <= o0) {
    if (tid == 0) st_jac(sums + (size_t)PW * v, s);
    return;
  }
  const size_t chunks = (M.nnz + MPC_CHUNK - 1) / MPC_CHUNK, kl = (o1 - 1) / MPC_CHUNK;
  size_t kf = o0 / MPC_CHUNK;
  if (kf >= chunks) kf = chunks - 1;
  if (kf == kl) return;
  if (tid == 0) ld_jac(s, bnd + (size_t)PW * (2 * kf + 1));
#pragma unroll 1
  for (size_t k = kf + 1 + tid; k <= kl; k += GS_TPB) {
    Jac<F> t;
    ld_jac(t, bnd + (size_t)PW * 2 * k);
    pt_add(s, t);
  }
  // each thread's partial into the slot of the first chunk it read (no other thread reads it), then thread 0 adds them up
  const size_t span = kl - kf;
  if (tid && (size_t)tid < span) st_jac(bnd + (size_t)PW * 2 * (kf + 1 + tid), s);
  __syncthreads();
  if (tid) return;
#pragma unroll 1
  for (size_t l = 1; l < GS_TPB && l < span; l++) {
    Jac<F> t;
    ld_jac(t, bnd + (size_t)PW * 2 * (kf + 1 + l));
    pt_add(s, t);
  }
  st_jac(sums + (size_t)PW * v, s);
}

// One thread per variable: ext = A x beta_coeffs + B x alpha_coeffs + C x coeffs into the ic | l block of the G1 batch, the
// density ballots (a != O, bg1 != O), and the flags: malformed offsets, an l row at the identity (phase2's
// UnconstrainedVariable), bg1 and bg2 disagreeing on the identity.
__global__ void __launch_bounds__(GS_TPB) k_mpc_combine(GsMats mats, size_t ni, size_t nv, const uint64_t* x1, uint64_t* ext, const uint64_t* a,
                                                        const uint64_t* b1, const uint64_t* b2, uint32_t* wa, uint32_t* wb, uint32_t* flags) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool nz_a = false, nz_b = false;
  if (t < nv) {
    uint32_t bad = 0;
#pragma unroll
    for (int m = 0; m < 3; m++) {
      const GsMat& M = mats.m[m];
      const uint64_t lo = M.off[t], hi = M.off[t + 1];
      if (lo > hi || hi > M.nnz || (t == 0 && lo != 0) || (t + 1 == nv && hi != M.nnz)) bad |= GS_BAD_CSR;
    }
    Jac<Fp> e, x;
    ld_jac(e, x1 + (size_t)G1_W * t);
    ld_jac(x, x1 + (size_t)G1_W * (nv + t));
    pt_add(e, x);
    ld_jac(x, x1 + (size_t)G1_W * (2 * nv + t));
    pt_add(e, x);
    st_jac(ext + (size_t)G1_W * t, e);
    if (t >= ni && pt_is_zero(e)) bad |= GS_UNCONSTRAINED;
    Fp z;
    ld_F(z, a + (size_t)G1_W * t + 2 * FW<Fp>::W);
    nz_a = !f_is_zero(z);
    ld_F(z, b1 + (size_t)G1_W * t + 2 * FW<Fp>::W);
    nz_b = !f_is_zero(z);
    Fp2 z2;
    ld_F(z2, b2 + (size_t)G2_W * t + 2 * FW<Fp2>::W);
    if (nz_b == f_is_zero(z2)) bad |= MPC_INCONSISTENT;
    if (bad) atomicOr(flags, bad);
  }
  const uint32_t ba = __ballot_sync(0xffffffffu, nz_a), bb = __ballot_sync(0xffffffffu, nz_b);
  if ((threadIdx.x & 31) == 0 && t < nv) { wa[t >> 5] = ba; wb[t >> 5] = bb; }
}

// affine rows -> Jacobian rows (the identity as (0, 1, 0))
template <class F>
__global__ void __launch_bounds__(GS_TPB) k_mpc_load(const uint64_t* in, size_t count, uint64_t* out) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int W = FW<F>::W;
  Aff<F> a;
  ld_aff(a, in + (size_t)(2 * W + 1) * t);
  Jac<F> r;
  pt_set_zero(r);
  if (!a.inf) { r.x = a.x; r.y = a.y; f_set_one(r.z); }
  st_jac(out + (size_t)(3 * W) * t, r);
}

// ---- host side ----------------------------------------------------------------------------------------------------------

static size_t gs_align(size_t x) { return (x + 255) & ~(size_t)255; }

namespace {
struct GsPlan {
  int L, s;                                      // log2 n, the split of the tau tables
  size_t n, nv, n1, words, chunks_max;           // domain, variables, n - 1, density words, k_gs_qap chunks of the longest matrix
  size_t N1, N2;                                 // G1 and G2 exponentiations
  size_t off_sc, off_flags, off_g, off_lo, off_hi, off_lag, off_fft, off_uvw, off_acc, off_words, off_s1, off_s2, off_p1, off_p2, off_t1,
      off_t2, off_bn, total;
};
}  // namespace

// shape checks (no device work, no reads of the matrices' contents)
static bool gs_shape_ok(const bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, GsPlan& p) {
  if (!ctx || !abc) return false;
  p.nv = ni + na;
  if (ni > GS_MAX_N || na > GS_MAX_N || p.nv > GS_MAX_N || nc > GS_MAX_N) return false;
  p.n = 1;
  p.L = 0;
  while (p.n < nc) { p.n <<= 1; p.L++; }
  p.s = (p.L + 1) / 2;
  p.n1 = p.n - 1;
  p.chunks_max = 0;
  for (int m = 0; m < 3; m++) {
    const bls_r1cs_matrix& M = abc[m];
    if (M.nnz >= GS_MAX_NNZ || !M.offsets || (M.nnz && (!M.constraint || !M.coeff)) || (p.nv == 0 && M.nnz)) return false;
    const size_t c = (M.nnz + GS_CHUNK - 1) / GS_CHUNK;
    p.chunks_max = c > p.chunks_max ? c : p.chunks_max;
  }
  p.words = (p.nv + 31) / 32;
  p.N1 = 3 + p.nv + p.n1 + 2 * p.nv;
  p.N2 = 3 + p.nv;
  return true;
}

static bool gs_fr_canonical_nonzero(const bls_fr* x, bool& zero) {
  static const uint64_t R[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
  zero = !(x->l[0] | x->l[1] | x->l[2] | x->l[3]);
  for (int i = 3; i >= 0; i--)
    if (x->l[i] != R[i]) return x->l[i] < R[i];
  return false;
}

static bool gs_out_ok(const bls_groth16_parameters_out* out, size_t ni, size_t na, const GsPlan& p) {
  if (!out || !out->vk || !out->lens || !out->ok) return false;
  if ((ni && (!out->ic || !out->b_input_density)) || (na && (!out->l || !out->a_aux_density || !out->b_aux_density))) return false;
  if (p.n1 && !out->h) return false;
  if (p.nv && (!out->a || !out->b_g1 || !out->b_g2)) return false;
  return true;
}

static bool gs_args_ok(const bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_g1_affine* g1,
                       const bls_g2_affine* g2, const bls_fr* const sc[5], const bls_groth16_parameters_out* out, GsPlan& p) {
  if (!gs_shape_ok(ctx, abc, nc, ni, na, p)) return false;
  if (!g1 || !g2 || g1->infinity || g2->infinity) return false;
  for (int i = 0; i < 5; i++) {
    bool zero;
    if (!sc[i] || !gs_fr_canonical_nonzero(sc[i], zero)) return false;
    if (zero && (i == GS_GAMMA || i == GS_DELTA)) return false;            // bellman's UnexpectedIdentity from inverse()
  }
  return gs_out_ok(out, ni, na, p);
}

static size_t gs_layout(bls_ctx* ctx, GsPlan& p) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += gs_align(bytes ? bytes : 1); return at; };
  const size_t fr = sizeof(bls_fr);
  p.off_sc = take(GS_NSC * fr);
  p.off_flags = take(sizeof(uint32_t));
  p.off_g = take(sizeof(bls_g1_affine) + sizeof(bls_g2_affine) + sizeof(bls_g1) + sizeof(bls_g2));
  p.off_lo = take(((size_t)1 << p.s) * fr);
  p.off_hi = take(((size_t)1 << (p.L - p.s)) * fr);
  p.off_lag = take(p.n * fr);
  const size_t fft = bls_fr_fft_scratch_bytes(ctx, p.L, 1);
  if (!fft) return 0;
  p.off_fft = take(fft);
  p.off_uvw = take(3 * p.nv * fr);
  p.off_acc = take(3 * p.chunks_max * 8 * sizeof(unsigned long long));
  p.off_words = take(4 * p.words * sizeof(uint32_t));
  p.off_s1 = take(p.N1 * sizeof(bls_fr_repr));
  p.off_s2 = take(p.N2 * sizeof(bls_fr_repr));
  p.off_p1 = take(p.N1 * sizeof(bls_g1));
  p.off_p2 = take(p.N2 * sizeof(bls_g2));
  p.off_t1 = take(((size_t)1 << (GS_WINDOW_G1 - 1)) * sizeof(bls_g1));
  p.off_t2 = take(((size_t)1 << (GS_WINDOW_G2 - 1)) * sizeof(bls_g2));
  const size_t b1 = bls_batch_normalization_scratch_bytes(ctx, 1, p.N1), b2 = bls_batch_normalization_scratch_bytes(ctx, 2, p.N2);
  p.off_bn = take(b1 > b2 ? b1 : b2);
  p.total = o;
  return o;
}

static int gs_dev_impl(bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_g1_affine* g1, const bls_g2_affine* g2,
                       const bls_fr* const sc5[5], const bls_groth16_parameters_out* out, void* scratch, void* stream) {
  GsPlan p;
  if (!gs_args_ok(ctx, abc, nc, ni, na, g1, g2, sc5, out, p) || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!gs_layout(ctx, p)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  uint64_t* sc = at(p.off_sc);
  uint32_t* flags = (uint32_t*)(base + p.off_flags);
  uint64_t *g1a = at(p.off_g), *g2a = g1a + G1A_W, *g1j = g2a + G2A_W, *g2j = g1j + G1_W;
  uint64_t *lo = at(p.off_lo), *hi = at(p.off_hi), *lag = at(p.off_lag), *uvw = at(p.off_uvw);
  unsigned long long* acc = (unsigned long long*)(base + p.off_acc);
  uint32_t *wa = (uint32_t*)(base + p.off_words), *wb = wa + p.words, *pa = wb + p.words, *pb = pa + p.words;
  uint64_t *s1 = at(p.off_s1), *s2 = at(p.off_s2), *p1 = at(p.off_p1), *p2 = at(p.off_p2);

  // the five scalars and g1, g2 in one copy (a pageable source has been staged when cudaMemcpyAsync returns)
  uint64_t up[5 * 4 + G1A_W + G2A_W];
  for (int i = 0; i < 5; i++) memcpy(up + 4 * i, sc5[i], sizeof(bls_fr));
  memcpy(up + 20, g1, sizeof(bls_g1_affine));
  memcpy(up + 20 + G1A_W, g2, sizeof(bls_g2_affine));
  CK(cudaMemcpyAsync(sc, up, 20 * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(g1a, up + 20, (G1A_W + G2A_W) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(flags, 0, sizeof(uint32_t), st));
  CK(cudaMemsetAsync(acc, 0, 3 * p.chunks_max * 8 * sizeof(unsigned long long), st));
  TRY(bls_fr_op_dev(ctx, BLS_OP_INV, (const bls_fr*)(sc + 4 * GS_GAMMA), nullptr, (bls_fr*)(sc + 4 * GS_GAMMA_INV), nullptr, 2, st));

  // G1 batch: [alpha, beta, delta | ic | l | h | a | b]
  uint64_t *s_ic = s1 + 4 * 3, *s_h = s_ic + 4 * p.nv;
  k_gs_pre<<<1, 1, 0, st>>>(sc, p.L, g1a, g2a, g1j, g2j, s1, s2);
  LAUNCH_CHECK();
  k_gs_tau_tables<<<blocks_for(((size_t)1 << p.s) + ((size_t)1 << (p.L - p.s)), GS_TPB), GS_TPB, 0, st>>>(sc, p.L, p.s, lo, hi);
  LAUNCH_CHECK();
  k_gs_powers<<<blocks_for(p.n, GS_TPB), GS_TPB, 0, st>>>(sc, lo, hi, p.s, p.n, lag, s_h);
  LAUNCH_CHECK();
  TRY(bls_fr_fft_dev(ctx, BLS_IFFT, (const bls_fr*)lag, (bls_fr*)lag, p.L, 1, base + p.off_fft, st));

  if (p.nv) {
    GsMats mats;
    for (int m = 0; m < 3; m++)
      mats.m[m] = GsMat{abc[m].offsets, abc[m].constraint, (const uint64_t*)abc[m].coeff, abc[m].nnz};
    if (p.chunks_max) {
      k_gs_qap<<<dim3(blocks_for(p.chunks_max, GS_TPB), 3), GS_TPB, 0, st>>>(mats, p.nv, nc, p.chunks_max, lag, uvw, acc, flags);
      LAUNCH_CHECK();
    }
    k_gs_query<<<blocks_for(p.nv, GS_TPB), GS_TPB, 0, st>>>(mats, ni, p.nv, p.n1, p.chunks_max, sc, uvw, acc, s_ic, s2 + 4 * 3, wa, wb, flags);
    LAUNCH_CHECK();
  }
  k_gs_scan<<<1, GS_SCAN_TPB, 0, st>>>(wa, wb, p.words, ni, na, pa, pb, out->lens, out->a_aux_density, out->b_input_density, out->b_aux_density);
  LAUNCH_CHECK();

  bls_g1* t1 = (bls_g1*)at(p.off_t1);
  bls_g2* t2 = (bls_g2*)at(p.off_t2);
  TRY(bls_g1_wnaf_table_dev(ctx, (const bls_g1*)g1j, GS_WINDOW_G1, t1, st));
  TRY(bls_g2_wnaf_table_dev(ctx, (const bls_g2*)g2j, GS_WINDOW_G2, t2, st));
  TRY(bls_g1_wnaf_fixed_base_dev(ctx, t1, GS_WINDOW_G1, (const bls_fr_repr*)s1, (bls_g1*)p1, p.N1, st));
  TRY(bls_g2_wnaf_fixed_base_dev(ctx, t2, GS_WINDOW_G2, (const bls_fr_repr*)s2, (bls_g2*)p2, p.N2, st));
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)p1, p.N1, base + p.off_bn, st));
  TRY(bls_g2_batch_normalization_dev(ctx, (bls_g2*)p2, p.N2, base + p.off_bn, st));

  GsOut o{(uint64_t*)out->vk, (uint64_t*)out->ic, (uint64_t*)out->h, (uint64_t*)out->l, (uint64_t*)out->a, (uint64_t*)out->b_g1,
          (uint64_t*)out->b_g2, out->ok};
  k_gs_emit<<<dim3(blocks_for(p.N1, GS_TPB), 2), GS_TPB, 0, st>>>(p1, p2, ni, na, p.n1, wa, pa, wb, pb, flags, o);
  LAUNCH_CHECK();
  return BLS_OK;
}

// the host form's checks of the matrices: offsets non-decreasing from 0 to nnz, constraint indices < num_constraints,
// coefficients < r
static bool gs_matrices_ok(const bls_r1cs_matrix* abc, size_t nc, size_t nv) {
  static const uint64_t R[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
  for (int m = 0; m < 3; m++) {
    const bls_r1cs_matrix& M = abc[m];
    if (M.offsets[0] != 0 || M.offsets[nv] != M.nnz) return false;
    for (size_t v = 0; v < nv; v++)
      if (M.offsets[v] > M.offsets[v + 1]) return false;
    for (size_t e = 0; e < M.nnz; e++) {
      if (M.constraint[e] >= nc) return false;
      const uint64_t* c = M.coeff[e].l;
      bool lt = false;
      for (int i = 3; i >= 0; i--)
        if (c[i] != R[i]) { lt = c[i] < R[i]; break; }
      if (!lt) return false;
    }
  }
  return true;
}

// The host forms: the matrices and a staging buffer for the outputs on the device, dev(matrices, outputs, scratch) for the
// _dev form's work, then the outputs back (of the queries a, b_g1 and b_g2 only the rows the compaction wrote).
template <class Dev>
static int gs_host_run(bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t ni, size_t na, const GsPlan& p, size_t scratch,
                       const bls_groth16_parameters_out* out, Dev dev) {
  const size_t ga = sizeof(bls_g1_affine), g2a = sizeof(bls_g2_affine), nv = p.nv;
  H2D(o0, abc[0].offsets, (nv + 1) * sizeof(uint64_t));
  H2D(o1, abc[1].offsets, (nv + 1) * sizeof(uint64_t));
  H2D(o2, abc[2].offsets, (nv + 1) * sizeof(uint64_t));
  H2D(c0, abc[0].nnz ? abc[0].constraint : nullptr, abc[0].nnz * sizeof(uint32_t));
  H2D(c1, abc[1].nnz ? abc[1].constraint : nullptr, abc[1].nnz * sizeof(uint32_t));
  H2D(c2, abc[2].nnz ? abc[2].constraint : nullptr, abc[2].nnz * sizeof(uint32_t));
  H2D(k0, abc[0].nnz ? abc[0].coeff : nullptr, abc[0].nnz * sizeof(bls_fr));
  H2D(k1, abc[1].nnz ? abc[1].coeff : nullptr, abc[1].nnz * sizeof(bls_fr));
  H2D(k2, abc[2].nnz ? abc[2].coeff : nullptr, abc[2].nnz * sizeof(bls_fr));
  const size_t wi = (ni + 31) / 32, wx = (na + 31) / 32;
  // the outputs in one staging buffer: vk | ic | h | l | a | b_g1 | b_g2 | densities | lens | ok
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t a = o; o += gs_align(bytes); return a; };
  const size_t f_vk = take(sizeof(bls_groth16_vk_points)), f_ic = take(ni * ga), f_h = take(p.n1 * ga), f_l = take(na * ga), f_a = take(nv * ga),
               f_b1 = take(nv * ga), f_b2 = take(nv * g2a), f_da = take(wx * 4), f_dbi = take(wi * 4), f_dba = take(wx * 4), f_lens = take(16),
               f_ok = take(1);
  DALLOC(dout, o);
  DALLOC(dscr, scratch);
  char* d = (char*)dout.p;
  bls_groth16_parameters_out dp{(bls_groth16_vk_points*)(d + f_vk), (bls_g1_affine*)(d + f_ic), (bls_g1_affine*)(d + f_h), (bls_g1_affine*)(d + f_l),
                                (bls_g1_affine*)(d + f_a), (bls_g1_affine*)(d + f_b1), (bls_g2_affine*)(d + f_b2), (uint32_t*)(d + f_da),
                                (uint32_t*)(d + f_dbi), (uint32_t*)(d + f_dba), (uint64_t*)(d + f_lens), (uint8_t*)(d + f_ok)};
  bls_r1cs_matrix dm[3] = {{(const uint64_t*)o0.p, (const uint32_t*)c0.p, (const bls_fr*)k0.p, abc[0].nnz},
                           {(const uint64_t*)o1.p, (const uint32_t*)c1.p, (const bls_fr*)k1.p, abc[1].nnz},
                           {(const uint64_t*)o2.p, (const uint32_t*)c2.p, (const bls_fr*)k2.p, abc[2].nnz}};
  TRY(dev(dm, &dp, dscr.p));
  uint64_t lens[2];
  CK(cudaMemcpyAsync(lens, dp.lens, sizeof(lens), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out->vk, dp.vk, sizeof(bls_groth16_vk_points), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out->ok, dp.ok, 1, cudaMemcpyDeviceToHost, ctx->stream));
  if (ni) CK(cudaMemcpyAsync(out->ic, dp.ic, ni * ga, cudaMemcpyDeviceToHost, ctx->stream));
  if (p.n1) CK(cudaMemcpyAsync(out->h, dp.h, p.n1 * ga, cudaMemcpyDeviceToHost, ctx->stream));
  if (na) {
    CK(cudaMemcpyAsync(out->l, dp.l, na * ga, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out->a_aux_density, dp.a_aux_density, wx * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out->b_aux_density, dp.b_aux_density, wx * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (ni) CK(cudaMemcpyAsync(out->b_input_density, dp.b_input_density, wi * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SYNC();
  memcpy(out->lens, lens, sizeof(lens));
  // the queries: only the rows the compaction wrote
  if (lens[0]) CK(cudaMemcpyAsync(out->a, dp.a, lens[0] * ga, cudaMemcpyDeviceToHost, ctx->stream));
  if (lens[1]) {
    CK(cudaMemcpyAsync(out->b_g1, dp.b_g1, lens[1] * ga, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out->b_g2, dp.b_g2, lens[1] * g2a, cudaMemcpyDeviceToHost, ctx->stream));
  }
  SYNC();
  return BLS_OK;
}

static int gs_host(bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_g1_affine* g1, const bls_g2_affine* g2,
                   const bls_fr* const sc5[5], const bls_groth16_parameters_out* out) {
  GsPlan p;
  if (!gs_args_ok(ctx, abc, nc, ni, na, g1, g2, sc5, out, p)) return BLS_ERR_INVALID_ARGUMENT;
  if (!gs_matrices_ok(abc, nc, p.nv)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!gs_layout(ctx, p)) return BLS_ERR_CUDA;
  return gs_host_run(ctx, abc, ni, na, p, p.total, out, [&](const bls_r1cs_matrix* dm, const bls_groth16_parameters_out* dp, void* scr) {
    return gs_dev_impl(ctx, dm, nc, ni, na, g1, g2, sc5, dp, scr, ctx->stream);
  });
}

// ---- phase 2: bls_groth16_mpc_new_* ----
namespace {
struct MpcPlan {
  GsPlan g;                                      // shape, n, N1 = 3 + nv + n1 + 2 nv, N2 = 3 + nv, density words
  size_t chunks_max;                             // k_mpc_qap chunks of the longest matrix
  size_t off_flags, off_pts, off_p1, off_p2, off_x1, off_bnd, off_words, off_bn, total;
};
}  // namespace

static bool mpc_args_ok(const bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_groth16_phase1* ph,
                        const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_groth16_parameters_out* out, MpcPlan& p) {
  if (!gs_shape_ok(ctx, abc, nc, ni, na, p.g)) return false;
  if (!g1 || !g2 || g1->infinity || g2->infinity || !ph || ph->n != p.g.n) return false;
  if ((abc[0].nnz || abc[1].nnz || abc[2].nnz) && (!ph->coeffs_g1 || !ph->alpha_coeffs_g1 || !ph->beta_coeffs_g1 || !ph->coeffs_g2)) return false;
  if (p.g.n1 && !ph->h) return false;
  return gs_out_ok(out, ni, na, p.g);
}

static size_t mpc_layout(bls_ctx* ctx, const bls_r1cs_matrix* abc, MpcPlan& p) {
  p.chunks_max = 0;
  for (int m = 0; m < 3; m++) {
    const size_t c = (abc[m].nnz + MPC_CHUNK - 1) / MPC_CHUNK;
    p.chunks_max = c > p.chunks_max ? c : p.chunks_max;
  }
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += gs_align(bytes ? bytes : 1); return at; };
  p.off_flags = take(sizeof(uint32_t));
  p.off_pts = take(3 * sizeof(bls_g1_affine) + 3 * sizeof(bls_g2_affine));
  p.off_p1 = take(p.g.N1 * sizeof(bls_g1));
  p.off_p2 = take(p.g.N2 * sizeof(bls_g2));
  p.off_x1 = take(3 * p.g.nv * sizeof(bls_g1));
  p.off_bnd = take(2 * p.chunks_max * sizeof(bls_g2));
  p.off_words = take(4 * p.g.words * sizeof(uint32_t));
  const size_t b1 = bls_batch_normalization_scratch_bytes(ctx, 1, p.g.N1), b2 = bls_batch_normalization_scratch_bytes(ctx, 2, p.g.N2);
  if (!b1 || !b2) return 0;
  p.off_bn = take(b1 > b2 ? b1 : b2);
  p.total = o;
  return o;
}

static int mpc_dev_impl(bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_groth16_phase1* ph,
                        const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_groth16_parameters_out* out, void* scratch, void* stream) {
  MpcPlan p;
  if (!mpc_args_ok(ctx, abc, nc, ni, na, ph, g1, g2, out, p) || !scratch) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!mpc_layout(ctx, abc, p)) return BLS_ERR_CUDA;
  cudaStream_t st = pick(ctx, stream);
  char* base = (char*)scratch;
  auto at = [&](size_t off) { return (uint64_t*)(base + off); };
  const size_t nv = p.g.nv, n1 = p.g.n1;
  uint32_t* flags = (uint32_t*)(base + p.off_flags);
  uint64_t *pts = at(p.off_pts), *p1 = at(p.off_p1), *p2 = at(p.off_p2), *x1 = at(p.off_x1), *bnd = at(p.off_bnd);
  uint32_t *wa = (uint32_t*)(base + p.off_words), *wb = wa + p.g.words, *pa = wb + p.g.words, *pb = pa + p.g.words;
  // G1 batch [alpha, beta, delta | ic | l | h | a | b], G2 batch [beta, gamma, delta | b]: k_gs_emit's layout
  uint64_t *p1_ext = p1 + G1_W * 3, *p1_h = p1_ext + G1_W * nv, *p1_a = p1_h + G1_W * n1, *p1_b = p1_a + G1_W * nv, *p2_b = p2 + G2_W * 3;

  // vk points in one copy (a pageable source has been staged when cudaMemcpyAsync returns): alpha_g1, beta_g1, delta_g1 = g1,
  // then beta_g2, gamma_g2 = delta_g2 = g2
  uint64_t up[3 * G1A_W + 3 * G2A_W];
  memcpy(up, &ph->alpha_g1, sizeof(bls_g1_affine));
  memcpy(up + G1A_W, &ph->beta_g1, sizeof(bls_g1_affine));
  memcpy(up + 2 * G1A_W, g1, sizeof(bls_g1_affine));
  memcpy(up + 3 * G1A_W, &ph->beta_g2, sizeof(bls_g2_affine));
  memcpy(up + 3 * G1A_W + G2A_W, g2, sizeof(bls_g2_affine));
  memcpy(up + 3 * G1A_W + 2 * G2A_W, g2, sizeof(bls_g2_affine));
  CK(cudaMemcpyAsync(pts, up, sizeof(up), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(flags, 0, sizeof(uint32_t), st));
  k_mpc_load<Fp><<<1, GS_TPB, 0, st>>>(pts, 3, p1);
  LAUNCH_CHECK();
  k_mpc_load<Fp2><<<1, GS_TPB, 0, st>>>(pts + 3 * G1A_W, 3, p2);
  LAUNCH_CHECK();
  if (n1) {
    k_mpc_load<Fp><<<blocks_for(n1, GS_TPB), GS_TPB, 0, st>>>((const uint64_t*)ph->h, n1, p1_h);
    LAUNCH_CHECK();
  }

  if (nv) {
    GsMats mats;
    for (int m = 0; m < 3; m++) mats.m[m] = GsMat{abc[m].offsets, abc[m].constraint, (const uint64_t*)abc[m].coeff, abc[m].nnz};
    const uint64_t *c1 = (const uint64_t*)ph->coeffs_g1, *al1 = (const uint64_t*)ph->alpha_coeffs_g1, *be1 = (const uint64_t*)ph->beta_coeffs_g1;
    struct { int m; const uint64_t* rows; uint64_t* sums; } g1pass[5] = {
        {0, c1, p1_a}, {0, be1, x1}, {1, c1, p1_b}, {1, al1, x1 + G1_W * nv}, {2, c1, x1 + 2 * G1_W * nv}};
    for (const auto& ps : g1pass) {
      const GsMat& M = mats.m[ps.m];
      if (M.nnz) {
        k_mpc_qap<Fp, false, MPC_K_G1><<<blocks_for((M.nnz + MPC_CHUNK - 1) / MPC_CHUNK, GS_TPB), GS_TPB, 0, st>>>(M, nv, nc, ps.rows, ps.sums, bnd, flags);
        LAUNCH_CHECK();
      }
      k_mpc_fix<Fp><<<(unsigned)nv, GS_TPB, 0, st>>>(M, nv, bnd, ps.sums);
      LAUNCH_CHECK();
    }
    if (mats.m[1].nnz) {
      k_mpc_qap<Fp2, true, MPC_K_G2><<<blocks_for((mats.m[1].nnz + MPC_CHUNK - 1) / MPC_CHUNK, GS_TPB), GS_TPB, 0, st>>>(
          mats.m[1], nv, nc, (const uint64_t*)ph->coeffs_g2, p2_b, bnd, flags);
      LAUNCH_CHECK();
    }
    k_mpc_fix<Fp2><<<(unsigned)nv, GS_TPB, 0, st>>>(mats.m[1], nv, bnd, p2_b);
    LAUNCH_CHECK();
    k_mpc_combine<<<blocks_for(nv, GS_TPB), GS_TPB, 0, st>>>(mats, ni, nv, x1, p1_ext, p1_a, p1_b, p2_b, wa, wb, flags);
    LAUNCH_CHECK();
  }
  k_gs_scan<<<1, GS_SCAN_TPB, 0, st>>>(wa, wb, p.g.words, ni, na, pa, pb, out->lens, out->a_aux_density, out->b_input_density, out->b_aux_density);
  LAUNCH_CHECK();
  TRY(bls_g1_batch_normalization_dev(ctx, (bls_g1*)p1, p.g.N1, base + p.off_bn, st));
  TRY(bls_g2_batch_normalization_dev(ctx, (bls_g2*)p2, p.g.N2, base + p.off_bn, st));
  GsOut o{(uint64_t*)out->vk, (uint64_t*)out->ic, (uint64_t*)out->h, (uint64_t*)out->l, (uint64_t*)out->a, (uint64_t*)out->b_g1,
          (uint64_t*)out->b_g2, out->ok};
  k_gs_emit<<<dim3(blocks_for(p.g.N1, GS_TPB), 2), GS_TPB, 0, st>>>(p1, p2, ni, na, n1, wa, pa, wb, pb, flags, o);
  LAUNCH_CHECK();
  return BLS_OK;
}

static int mpc_host(bls_ctx* ctx, const bls_r1cs_matrix* abc, size_t nc, size_t ni, size_t na, const bls_groth16_phase1* ph,
                    const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_groth16_parameters_out* out) {
  MpcPlan p;
  if (!mpc_args_ok(ctx, abc, nc, ni, na, ph, g1, g2, out, p)) return BLS_ERR_INVALID_ARGUMENT;
  if (!gs_matrices_ok(abc, nc, p.g.nv)) return BLS_ERR_INVALID_ARGUMENT;
  USE_DEVICE(ctx);
  if (!mpc_layout(ctx, abc, p)) return BLS_ERR_CUDA;
  const size_t n = p.g.n, rows = (abc[0].nnz || abc[1].nnz || abc[2].nnz) ? n : 0, ga = sizeof(bls_g1_affine);
  H2D(r1, rows ? ph->coeffs_g1 : nullptr, rows * ga);
  H2D(ra, rows ? ph->alpha_coeffs_g1 : nullptr, rows * ga);
  H2D(rb, rows ? ph->beta_coeffs_g1 : nullptr, rows * ga);
  H2D(r2, rows ? ph->coeffs_g2 : nullptr, rows * sizeof(bls_g2_affine));
  H2D(rh, p.g.n1 ? ph->h : nullptr, p.g.n1 * ga);
  bls_groth16_phase1 dph = *ph;
  dph.coeffs_g1 = (const bls_g1_affine*)r1.p;
  dph.alpha_coeffs_g1 = (const bls_g1_affine*)ra.p;
  dph.beta_coeffs_g1 = (const bls_g1_affine*)rb.p;
  dph.coeffs_g2 = (const bls_g2_affine*)r2.p;
  dph.h = (const bls_g1_affine*)rh.p;
  return gs_host_run(ctx, abc, ni, na, p.g, p.total, out, [&](const bls_r1cs_matrix* dm, const bls_groth16_parameters_out* dp, void* scr) {
    return mpc_dev_impl(ctx, dm, nc, ni, na, &dph, g1, g2, dp, scr, ctx->stream);
  });
}

extern "C" {

size_t bls_groth16_generate_parameters_scratch_bytes(const bls_ctx* cctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs,
                                                     size_t num_aux) {
  GsPlan p;
  if (!gs_shape_ok(cctx, abc, num_constraints, num_inputs, num_aux, p)) return 0;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  return gs_layout(ctx, p);
}
int bls_groth16_generate_parameters_dev(bls_ctx* ctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                                        const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_fr* alpha, const bls_fr* beta, const bls_fr* gamma,
                                        const bls_fr* delta, const bls_fr* tau, const bls_groth16_parameters_out* out, void* scratch, void* stream) {
  const bls_fr* const sc[5] = {alpha, beta, gamma, delta, tau};
  return gs_dev_impl(ctx, abc, num_constraints, num_inputs, num_aux, g1, g2, sc, out, scratch, stream);
}
int bls_groth16_generate_parameters_batch(bls_ctx* ctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                                          const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_fr* alpha, const bls_fr* beta,
                                          const bls_fr* gamma, const bls_fr* delta, const bls_fr* tau, const bls_groth16_parameters_out* out) {
  const bls_fr* const sc[5] = {alpha, beta, gamma, delta, tau};
  return gs_host(ctx, abc, num_constraints, num_inputs, num_aux, g1, g2, sc, out);
}

size_t bls_groth16_mpc_new_scratch_bytes(const bls_ctx* cctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux) {
  MpcPlan p;
  if (!gs_shape_ok(cctx, abc, num_constraints, num_inputs, num_aux, p.g)) return 0;
  bls_ctx* ctx = const_cast<bls_ctx*>(cctx);
  DevGuard g;
  if (g.enter(ctx->device) != cudaSuccess) return 0;
  return mpc_layout(ctx, abc, p);
}
int bls_groth16_mpc_new_dev(bls_ctx* ctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                            const bls_groth16_phase1* phase1, const bls_g1_affine* g1, const bls_g2_affine* g2,
                            const bls_groth16_parameters_out* out, void* scratch, void* stream) {
  return mpc_dev_impl(ctx, abc, num_constraints, num_inputs, num_aux, phase1, g1, g2, out, scratch, stream);
}
int bls_groth16_mpc_new_batch(bls_ctx* ctx, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                              const bls_groth16_phase1* phase1, const bls_g1_affine* g1, const bls_g2_affine* g2,
                              const bls_groth16_parameters_out* out) {
  return mpc_host(ctx, abc, num_constraints, num_inputs, num_aux, phase1, g1, g2, out);
}

}  // extern "C"
