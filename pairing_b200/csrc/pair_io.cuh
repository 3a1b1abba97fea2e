// pair_io.cuh -- ABI <-> lane-pair register conversions and the launch shape shared by the lane-pair translation units
// (kernels_pair.cu, kernels_mm.cu, kernels_groth16_verify.cu).
#pragma once
#include "abi_common.cuh"
#include "pair_tower.cuh"

// ---- lane-pair kernels (pair_tower.cuh): two adjacent lanes per pairing, lane c owns coefficient c
// of every Fq2.  Threads past the end of the batch recompute the last element (every lane has to
// reach every shuffle) and skip the store.
__device__ __forceinline__ P2 ld_p2(const uint64_t* p) { return P2{ld_fp(p + 6 * pair_c())}; }
__device__ __forceinline__ void st_p2(uint64_t* p, const P2& a) { st_fp(p + 6 * pair_c(), a.v); }
__device__ __forceinline__ void ld_p12(P12& r, const uint64_t* p) {
  r.c0.c0 = ld_p2(p); r.c0.c1 = ld_p2(p + 12); r.c0.c2 = ld_p2(p + 24);
  r.c1.c0 = ld_p2(p + 36); r.c1.c1 = ld_p2(p + 48); r.c1.c2 = ld_p2(p + 60);
}
__device__ __forceinline__ void st_p12(uint64_t* p, const P12& a) {
  st_p2(p, a.c0.c0); st_p2(p + 12, a.c0.c1); st_p2(p + 24, a.c0.c2);
  st_p2(p + 36, a.c1.c0); st_p2(p + 48, a.c1.c1); st_p2(p + 60, a.c1.c2);
}

// launch shape of the lane-pair kernels: BLS_PAIR_TPB threads per block, BLS_PAIR_MINB blocks per SM
// (registers per thread <= 65536 / (TPB * MINB)).  Small blocks keep the tail of a 2^16 batch short.
#define BLS_PAIR_TPB 128
#define BLS_PAIR_MINB 2

// line coefficients of a pair that does not count (infinity member, past the end): the sparse element one
__device__ __forceinline__ void pcoeffs_set_one_if(bool dead, PCoeffs& c) {
  const P2 one = p2_one(), zero = p2_zero();
  c.c0.v = fp_select(dead, zero.v, c.c0.v);
  c.c1.v = fp_select(dead, zero.v, c.c1.v);
  c.c2.v = fp_select(dead, one.v, c.c2.v);
}

// G2Prepared::from_affine (mod.rs:168-358) on lane pairs: lane c writes coefficient c of every Fq2 of the 68 triples
__device__ __forceinline__ void st_pcoeffs(uint64_t* p, const PCoeffs& c) { st_p2(p, c.c0); st_p2(p + 12, c.c1); st_p2(p + 24, c.c2); }
__device__ __forceinline__ void ld_pcoeffs(PCoeffs& c, const uint64_t* p) { c.c0 = ld_p2(p); c.c1 = ld_p2(p + 12); c.c2 = ld_p2(p + 24); }

// prepared coefficients staged in shared memory (a TMA bulk copy completing on an mbarrier): lane c reads coefficient c
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ P2 ld_p2_smem(const uint64_t* p) {
  P2 r;
  const uint2* q = reinterpret_cast<const uint2*>(p + 6 * pair_c());
#pragma unroll
  for (int i = 0; i < 6; i++) { uint2 t = q[i]; r.v.v[2 * i] = t.x; r.v.v[2 * i + 1] = t.y; }
  return r;
}
// spin until phase 0 of the mbarrier at shared address `bar` has completed
__device__ __forceinline__ void mbar_wait_phase0(uint32_t bar) {
  asm volatile("{\n\t.reg .pred ready;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 ready, [%0], 0;\n\t@ready bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar) : "memory");
}
