/* pairing_b200_mpc.h -- C ABI of phase 2 of the Groth16 setup ceremony (the `phase2` crate, on pairing 0.14 and bellman).
 *
 * An extension of pairing_b200.h, with the same layouts, errors, threading and device-pointer contract; include it after
 * that header.  tests/test_gpu_groth16_mpc.py holds the completeness checks of this header's entry points (every symbol
 * bound by pairing_b200._native.MPC_SYMBOLS, every scratch-taking `_dev` call covered by a device-contract case).
 *
 * Phase 1 (powers of tau) publishes [tau^i] rows; powersoftau's prepare_phase2 turns them into the Lagrange rows of the
 * circuit's domain (bls_g1_fft_* / bls_g2_fft_* IFFT), which bls_groth16_mpc_new_* takes.  The library hashes nothing and
 * draws no randomness: phase2's BLAKE2b transcript hashes, hash_to_g2 and the randomizers stay with the caller.
 */
#ifndef PAIRING_B200_MPC_H
#define PAIRING_B200_MPC_H

#include "pairing_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ Groth16 ceremony, phase 2
 * powersoftau's prepare_phase2 output for the domain of n points (the phase1radix2m file, decoded): alpha_g1, beta_g1 and
 * beta_g2 by value, then n rows each of [L_q(tau)] g1, [alpha L_q(tau)] g1, [beta L_q(tau)] g1 and [L_q(tau)] g2, and n - 1
 * rows [tau^i (tau^n - 1)] g1.  The row pointers are host memory for _batch, device memory for _dev. */
typedef struct {
  bls_g1_affine alpha_g1, beta_g1;
  bls_g2_affine beta_g2;
  const bls_g1_affine *coeffs_g1, *alpha_coeffs_g1, *beta_coeffs_g1;
  const bls_g2_affine* coeffs_g2;
  const bls_g1_affine* h;
  size_t n;
} bls_groth16_phase1;

/* phase2's MPCParameters::new: the circuit's key from a phase-1 transcript, before any contribution.
 * abc, num_constraints, num_inputs, num_aux and out are those of bls_groth16_generate_parameters_batch (the CSR layout,
 * inputs first, the input_i * 0 = 0 constraints included).  n is the smallest power of two >= num_constraints (1 for 0 or
 * 1 constraints) and phase1->n must equal it.  For each variable v over its terms (q, c):
 *   a_v = sum_A c coeffs_g1[q], bg1_v = sum_B c coeffs_g1[q], bg2_v = sum_B c coeffs_g2[q],
 *   ext_v = sum_A c beta_coeffs_g1[q] + sum_B c alpha_coeffs_g1[q] + sum_C c coeffs_g1[q].
 * The key: vk alpha_g1, beta_g1, beta_g2 from the transcript, gamma_g2 = delta_g2 = g2, delta_g1 = g1; ic = ext of the
 * inputs, l = ext of the aux variables, h = the transcript's h rows; a, b_g1, b_g2 = a_v, bg1_v, bg2_v with the identities
 * dropped; the densities as generate_parameters emits them, decided on the points (a_aux bit: a_v != O; b bits: bg1_v != O);
 * lens = [a_len, b_len].  ok = 0 (the key is still written) when an l row is the identity (phase2's UnconstrainedVariable),
 * when bg1_v and bg2_v disagree on being the identity (an inconsistent transcript), or when the _dev form finds a malformed
 * matrix.  An honest transcript of (tau, alpha, beta) on generators g1, g2 gives, byte for byte, the key of
 * bls_groth16_generate_parameters_batch for (alpha, beta, gamma = 1, delta = 1, tau).
 * Every point is a canonical affine row (the identity is (0, one, infinity = 1)), so the key does not depend on the
 * summation order.  Results are defined for transcript rows of order dividing r; the call validates no row (phase2 reads
 * them unchecked): check them with bls_g1_decode_batch / bls_g2_decode_batch first.  Coefficients are multiplied in signed
 * form, min(c, r - c), so -1 and -2^k cost what 1 and 2^k cost.
 * BLS_ERR_INVALID_ARGUMENT, before any work: g1 or g2 NULL or at infinity, phase1 NULL or phase1->n wrong, a NULL row
 * pointer where there is something to read (the four coefficient row sets when a matrix has terms, h when n > 1), a NULL
 * output where there is something to write, and the limits and (host form) the matrix checks of
 * bls_groth16_generate_parameters_batch. */
int bls_groth16_mpc_new_batch(bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                              const bls_groth16_phase1* phase1, const bls_g1_affine* g1, const bls_g2_affine* g2,
                              const bls_groth16_parameters_out* out);

/* bls_groth16_mpc_new_batch on device pointers: the matrices' arrays, phase1's row pointers and every pointer of `out`; abc,
 * phase1 itself (with its alpha_g1, beta_g1 and beta_g2), g1 and g2 stay in host memory.  The matrices' contents are not
 * validated up front; reads are clamped as in bls_groth16_generate_parameters_dev, and a malformed matrix sets ok = 0.
 * Only the first a_len rows of a and b_len rows of b_g1 and b_g2 are written.  scratch:
 * bls_groth16_mpc_new_scratch_bytes(ctx, abc, num_constraints, num_inputs, num_aux) bytes (0 for invalid arguments): the
 * Jacobian G1 and G2 batches, the three ext parts, the boundary slots of the chunks, the density words and the
 * normalisation's work region.  The call allocates nothing and does not synchronise. */
size_t bls_groth16_mpc_new_scratch_bytes(const bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux);
int bls_groth16_mpc_new_dev(bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                            const bls_groth16_phase1* phase1, const bls_g1_affine* g1, const bls_g2_affine* g2,
                            const bls_groth16_parameters_out* out, void* scratch, void* stream);

/* ------------------------------------------------------------------ contributions
 * phase2's PublicKey without its transcript hash, plus r = hash_to_g2(transcript), which the caller derives. */
typedef struct { bls_g1_affine delta_after, s, s_delta; bls_g2_affine r, r_delta; } bls_groth16_mpc_pubkey;

/* phase2's MPCParameters::contribute for a caller-supplied secret delta and the caller's s and r.  delta is a Montgomery
 * bls_fr, canonical and nonzero.  With d = delta^-1: h_out[i] = [d] h[i], l_out[i] = [d] l[i] (h_out == h and l_out == l are
 * allowed); vk->delta_g1 and vk->delta_g2 are multiplied by delta in place; pubkey = (the new delta_g1, s, [delta] s, r,
 * [delta] r).  Every point leaves as a canonical affine row.  phase2 hashes s_delta into the transcript that r is derived
 * from, so the caller first computes s_delta = [delta] s (bls_g1_affine_mul_batch, then into_affine: the same point this
 * call stores), hashes, derives r with hash_to_g2, then calls this.  Results are defined for points of order dividing r.
 * BLS_ERR_INVALID_ARGUMENT, before any work: delta NULL, >= r or zero; s, r or vk NULL; a NULL row pointer where there is
 * work; h_len or l_len > 2^26. */
int bls_groth16_mpc_contribute_batch(bls_ctx*, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, bls_groth16_vk_points* vk,
                                     const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, bls_g1_affine* h_out,
                                     bls_g1_affine* l_out, bls_groth16_mpc_pubkey* pubkey);
/* bls_groth16_mpc_contribute_batch on device pointers: vk (read and written), h, l, h_out, l_out and pubkey; delta, s and r
 * stay in host memory.  scratch: bls_groth16_mpc_contribute_scratch_bytes(ctx, h_len, l_len) bytes (0 for invalid
 * arguments): delta and its inverse, the Jacobian bases with the replicated scalars, the products and the normalisation's
 * work region.  The call allocates nothing
 * and does not synchronise. */
size_t bls_groth16_mpc_contribute_scratch_bytes(const bls_ctx*, size_t h_len, size_t l_len);
int bls_groth16_mpc_contribute_dev(bls_ctx*, const bls_fr* delta, const bls_g1_affine* s, const bls_g2_affine* r, bls_groth16_vk_points* vk,
                                   const bls_g1_affine* h, size_t h_len, const bls_g1_affine* l, size_t l_len, bls_g1_affine* h_out,
                                   bls_g1_affine* l_out, bls_groth16_mpc_pubkey* pubkey, void* scratch, void* stream);

/* ------------------------------------------------------------------ verification
 * bellman's Parameters<Bls12>: the vk by value, the queries in host (_batch) or device (_dev) memory. */
typedef struct {
  bls_groth16_vk_points vk;
  const bls_g1_affine *ic, *h, *l, *a, *b_g1;
  const bls_g2_affine* b_g2;
  size_t ic_len, h_len, l_len, a_len, b_len;
} bls_groth16_key;

/* phase2's MPCParameters::verify, given the r of each of the k contributions.  `before` is the output of
 * bls_groth16_mpc_new_*; its delta_g1 and delta_g2 are the generators phase2 calls one().  "e(A, B) = e(C, D)" below is
 * FE(ML(A, B) ML(-C, D)) == 1, phase2's same_ratio for points of order r, with pairs at infinity contributing one.
 * *ok1 = 1 iff all hold:
 *   1. before and after have equal ic, a, b_g1, b_g2 (lengths and bytes), equal alpha_g1, beta_g1, beta_g2 and gamma_g2,
 *      and equal h_len and l_len;
 *   2. with d_(-1) = before.delta_g1 and d_j = pk[j].delta_after: e(s_delta_j, r_j) = e(s_j, r_delta_j) and
 *      e(d_(j-1), r_delta_j) = e(d_j, r_j) for every j < k;
 *   3. after.delta_g1 == d_(k-1) bytewise, and e(before.delta_g1, after.delta_g2) = e(d_(k-1), before.delta_g2);
 *   4. e(sum rho_h_i before.h_i, before.delta_g2) = e(sum rho_h_i after.h_i, after.delta_g2), and the same for l with rho_l
 *      (phase2's merge_pairs with the caller's randomizers; rho_i = 0 leaves row i out).
 * k = 0 is valid.  The caller keeps phase2's hash checks (each r_j against its transcript).  BLS_ERR_INVALID_ARGUMENT,
 * before any work: a NULL pointer where there is something to read or write, k > 2^16, a query of more than 2^26 rows. */
int bls_groth16_mpc_verify_batch(bls_ctx*, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                                 const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, uint8_t* ok1);
/* bls_groth16_mpc_verify_batch on device pointers: the query rows of both keys, pk, rho_h, rho_l and ok1; before and after
 * themselves (with their vk) stay in host memory.  scratch: bls_groth16_mpc_verify_scratch_bytes(ctx, before, after, k)
 * bytes (0 for invalid arguments): the four sums and the multiexp's work region, the pairs, the Miller loop and final
 * exponentiation values, and the flags.  The call allocates nothing and does not synchronise. */
size_t bls_groth16_mpc_verify_scratch_bytes(const bls_ctx*, const bls_groth16_key* before, const bls_groth16_key* after, size_t k);
int bls_groth16_mpc_verify_dev(bls_ctx*, const bls_groth16_key* before, const bls_groth16_key* after, const bls_groth16_mpc_pubkey* pk, size_t k,
                               const bls_fr_repr* rho_h, const bls_fr_repr* rho_l, uint8_t* ok1, void* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PAIRING_B200_MPC_H */
