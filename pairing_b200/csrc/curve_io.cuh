// curve_io.cuh -- ABI rows <-> curve.cuh points (Jacobian bls_g1 / bls_g2, affine bls_g*_affine), for F = Fp (G1) and Fp2 (G2).
// Shared by the translation units that run the group law (kernels.cu, kernels_msm.cu).
#pragma once
#include "abi_common.cuh"
#include "curve.cuh"

__device__ __forceinline__ void ld_F(Fp& r, const uint64_t* p) { r = ld_fp(p); }
__device__ __forceinline__ void ld_F(Fp2& r, const uint64_t* p) { r = ld_fp2(p); }
__device__ __forceinline__ void st_F(uint64_t* p, const Fp& a) { st_fp(p, a); }
__device__ __forceinline__ void st_F(uint64_t* p, const Fp2& a) { st_fp2(p, a); }
template <class F> struct FW;   // words (u64) per coordinate
template <> struct FW<Fp> { static const int W = 6; };
template <> struct FW<Fp2> { static const int W = 12; };

template <class F> __device__ __forceinline__ void ld_jac(Jac<F>& r, const uint64_t* p) {
  ld_F(r.x, p); ld_F(r.y, p + FW<F>::W); ld_F(r.z, p + 2 * FW<F>::W);
}
template <class F> __device__ __forceinline__ void st_jac(uint64_t* p, const Jac<F>& a) {
  st_F(p, a.x); st_F(p + FW<F>::W, a.y); st_F(p + 2 * FW<F>::W, a.z);
}
template <class F> __device__ __forceinline__ void ld_aff(Aff<F>& r, const uint64_t* p) {
  ld_F(r.x, p); ld_F(r.y, p + FW<F>::W); r.inf = p[2 * FW<F>::W] != 0;
}
template <class F> __device__ __forceinline__ void st_aff(uint64_t* p, const Aff<F>& a) {
  st_F(p, a.x); st_F(p + FW<F>::W, a.y); p[2 * FW<F>::W] = a.inf ? 1ull : 0ull;
}
