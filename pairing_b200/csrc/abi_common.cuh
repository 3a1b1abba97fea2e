// abi_common.cuh -- shared by the translation units of the library (kernels_pair.cu: the lane-pair pairing engine; kernels_mm.cu: the
// multi-pairing Miller loop; kernels_wide.cu: the warp-cooperative engine; kernels.cu: curve, field-op, codec and measurement kernels +
// the host-buffer entry points; mgpu.cu: several devices behind one call).
// The pairing engine is compiled on its own so that ptxas' register allocation of the routines it shares with
// nothing else (fp_mul2, p6_mul, ...) cannot be perturbed by unrelated kernels: a two-line change in curve.cuh was
// measured to slow the fused pairing kernel by 4 % when everything lived in one module.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "../../include/pairing_b200.h"
#include "tower.cuh"

using namespace bls;

// ------------------------------------------------------------------------------------------------
// ABI <-> register conversions.  ABI structs are arrays of u64 (8-byte aligned).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ Fp ld_fp(const uint64_t* p) {
  Fp r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 6; i++) { uint2 t = q[i]; r.v[2 * i] = t.x; r.v[2 * i + 1] = t.y; }
  return r;
}
// every value that leaves through the ABI is the canonical representative (< q), as in the reference
__device__ __forceinline__ void st_fp(uint64_t* p, const Fp& x) {
  const Fp a = fp_canon(x);
  uint2* q = reinterpret_cast<uint2*>(p);
#pragma unroll
  for (int i = 0; i < 6; i++) q[i] = make_uint2(a.v[2 * i], a.v[2 * i + 1]);
}
__device__ __forceinline__ Fp2 ld_fp2(const uint64_t* p) { return Fp2{ld_fp(p), ld_fp(p + 6)}; }
__device__ __forceinline__ void st_fp2(uint64_t* p, const Fp2& a) { st_fp(p, a.c0); st_fp(p + 6, a.c1); }
__device__ __forceinline__ void ld_fp6(Fp6& r, const uint64_t* p) { r.c0 = ld_fp2(p); r.c1 = ld_fp2(p + 12); r.c2 = ld_fp2(p + 24); }
__device__ __forceinline__ void st_fp6(uint64_t* p, const Fp6& a) { st_fp2(p, a.c0); st_fp2(p + 12, a.c1); st_fp2(p + 24, a.c2); }
__device__ __forceinline__ void ld_fp12(Fp12& r, const uint64_t* p) { ld_fp6(r.c0, p); ld_fp6(r.c1, p + 36); }
__device__ __forceinline__ void st_fp12(uint64_t* p, const Fp12& a) { st_fp6(p, a.c0); st_fp6(p + 36, a.c1); }

__device__ __forceinline__ Scalar ld_scalar(const uint64_t* p) {
  Scalar s;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) { uint2 t = q[i]; s.v[2 * i] = t.x; s.v[2 * i + 1] = t.y; }
  return s;
}

#define G1A_W 13
#define G1_W 18
#define G2A_W 25
#define G2_W 36
#define FQ12_W 72
#define G2P_W (68 * 36 + 1)

// ------------------------------------------------------------------------------------------------
// Host side: context
// ------------------------------------------------------------------------------------------------
struct bls_ctx {
  std::recursive_mutex mu;                       // every entry point holds it while it runs on the host (USE_DEVICE): calls from several threads serialise
  int device;
  int sm_count;
  cudaStream_t stream;
  cudaStream_t stream2;                          // second kernel stream of run_pipelined (kernels of consecutive chunks overlap their tails)
  cudaStream_t copy_in, copy_out;                // the H2D / D2H legs of the chunked host-buffer entry points (run_pipelined)
  cudaEvent_t ev_in[2], ev_k[2], ev_out[2];
  cudaMemPool_t pool;                            // staging buffers of the host-buffer entry points: cached across calls
  uint64_t launches;
  bool mm_smem_ready;                            // kernels_mm.cu: the > 48 KB dynamic shared memory opt-in has been made on this device
  size_t wide_pairing_max, wide_final_exp_max;   // batches up to these sizes run on the warp-cooperative engine (kernels_wide.cu)
  char last_error[256];
};
// Defaults of the two limits: below them one WARP per element (~2 ms for one pairing or for a thousand) beats the lane-pair
// throughput kernels (8.8 ms of latency, 1.49 M pairings/s); bls_ctx_set_latency_path_limits overrides them per context.
#define BLS_WIDE_PAIRING_MAX 2560
#define BLS_WIDE_FINAL_EXP_MAX 2560

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t e_ = (call);                                                          \
    if (e_ != cudaSuccess) {                                                          \
      snprintf(ctx->last_error, sizeof(ctx->last_error), "%s: %s", #call, cudaGetErrorString(e_)); \
      return e_ == cudaErrorMemoryAllocation ? BLS_ERR_OUT_OF_MEMORY : BLS_ERR_CUDA;  \
    }                                                                                 \
  } while (0)

// Every entry point runs on ctx->device and leaves the caller's current device as it found it (a host that shares the
// process with torch or with another context must not have its current device switched under it).
struct DevGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t enter(int dev) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev == dev) return cudaSuccess;
    e = cudaSetDevice(dev);
    switched = e == cudaSuccess;
    return e;
  }
  ~DevGuard() { if (switched) cudaSetDevice(prev); }
};
#define USE_DEVICE(ctx)                                          \
  std::lock_guard<std::recursive_mutex> ctx_lock_((ctx)->mu);    \
  DevGuard dev_guard_;                                           \
  CK(dev_guard_.enter((ctx)->device))

static inline unsigned blocks_for(size_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }
static const int TPB = 128;

static inline cudaStream_t pick(bls_ctx* ctx, void* stream) { return stream ? (cudaStream_t)stream : ctx->stream; }

#define LAUNCH_CHECK()                                  \
  do {                                                  \
    ctx->launches++;                                    \
    CK(cudaGetLastError());                             \
  } while (0)

// ---- host-buffer entry points stage through stream-ordered device buffers
namespace {
struct DevBuf {
  void* p = nullptr;
  cudaStream_t s;
  cudaMemPool_t pool;
  explicit DevBuf(bls_ctx* c) : s(c->stream), pool(c->pool) {}
  // the context's own pool (release threshold: never), so that a call does not pay cudaMalloc / cudaFree of its staging
  // buffers again: the first call grows the pool, later calls of the same size find the memory cached
  cudaError_t alloc(size_t bytes) { return cudaMallocFromPoolAsync(&p, bytes ? bytes : 1, pool, s); }
  ~DevBuf() { if (p) cudaFreeAsync(p, s); }
};
}  // namespace

#define H2D(buf, host, bytes)                                                          \
  DevBuf buf(ctx);                                                                     \
  CK(buf.alloc(bytes));                                                                \
  if (host) CK(cudaMemcpyAsync(buf.p, host, bytes, cudaMemcpyHostToDevice, ctx->stream))
#define DALLOC(buf, bytes) \
  DevBuf buf(ctx);         \
  CK(buf.alloc(bytes))
#define D2H(host, buf, bytes) CK(cudaMemcpyAsync(host, buf.p, bytes, cudaMemcpyDeviceToHost, ctx->stream))
#define SYNC() CK(cudaStreamSynchronize(ctx->stream))
#define TRY(call)            \
  do {                       \
    int rc_ = (call);        \
    if (rc_ != BLS_OK) return rc_; \
  } while (0)


#define BLS_INTERNAL __attribute__((visibility("hidden")))
// cross-unit helpers (not part of the ABI)
extern "C" {
BLS_INTERNAL int bls_internal_product_passes(bls_ctx* ctx, const uint64_t* in, size_t count, bls_fq12* out1, uint64_t* scratch, cudaStream_t s);
BLS_INTERNAL size_t bls_internal_mm_lane_pairs(const bls_ctx* ctx, size_t n);
BLS_INTERNAL int bls_internal_wide_final_exp(bls_ctx* ctx, const bls_fq12* in, bls_fq12* out, uint8_t* is_some, size_t n, cudaStream_t s);
BLS_INTERNAL int bls_internal_wide_pairing(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, cudaStream_t s);
BLS_INTERNAL int bls_internal_wide_miller(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, cudaStream_t s);
BLS_INTERNAL int bls_internal_wide_pairing_projective(bls_ctx* ctx, const bls_g1* p, const bls_g2* q, bls_fq12* out, size_t n, cudaStream_t s);
BLS_INTERNAL int bls_internal_product_tail(bls_ctx* ctx, const bls_fq12* in, size_t count, bls_fq12* out1, int final_exp, uint8_t* is_some, cudaStream_t s);
BLS_INTERNAL int bls_internal_multi_miller_prepared(bls_ctx* ctx, const bls_g1_affine* p, const bls_g2_prepared* qp, size_t n, bls_fq12* partials, cudaStream_t s);
}
