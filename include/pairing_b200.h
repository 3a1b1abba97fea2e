/* pairing_b200.h -- C ABI of the B200-native batched BLS12-381 pairing / wNAF engine.
 *
 * This is the drop-in boundary beneath the `pairing` crate's trait surface (v0.14.2).  The
 * reference has no FFI of its own: its boundary is the Rust traits `Engine` (src/lib.rs:34-110),
 * `CurveProjective` (src/lib.rs:114-181), `CurveAffine` (src/lib.rs:185-234) and `Wnaf`
 * (src/wnaf.rs:75-179).  Each entry point below names the reference routine it replaces; the Rust
 * shim that binds them is shown in INTEGRATION.md and rust/src/ffi.rs.
 *
 * Data layout (all little-endian, identical byte-for-byte to the crate's in-memory values):
 *   Fq      6 x u64 limbs, Montgomery form (x * 2^384 mod q), always < q   (bls12_381/fq.rs:510,699)
 *   Fq2     c0 | c1                                                        (fq2.rs:8-12)
 *   Fq6     c0 | c1 | c2                                                   (fq6.rs:8-12)
 *   Fq12    c0 | c1                                                        (fq12.rs:8-12)
 *   FrRepr  4 x u64 limbs, canonical integer, NOT Montgomery               (fr.rs:58)
 * Ownership: the caller owns every buffer; nothing is retained after a call returns.
 * Errors: every function returns 0 on success or a negative bls_status; nothing unwinds across
 * the ABI.  There is no CPU fallback: without a CUDA device bls_ctx_create fails.
 * Threading: a bls_ctx may be shared by several host threads -- every entry point holds the context's lock while it runs on the
 * host, so concurrent calls serialise (one ordered stream per device); use one context per thread for concurrency.
 */
#ifndef PAIRING_B200_H
#define PAIRING_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { uint64_t l[6]; } bls_fq;
typedef struct { bls_fq c0, c1; } bls_fq2;
typedef struct { bls_fq2 c0, c1, c2; } bls_fq6;
typedef struct { bls_fq6 c0, c1; } bls_fq12;                       /* 576 B */
typedef struct { bls_fq x, y; uint64_t infinity; } bls_g1_affine;  /* 104 B; ec.rs:13-18 */
typedef struct { bls_fq x, y, z; } bls_g1;                         /* 144 B; Jacobian, z == 0 <=> infinity; ec.rs:31-36 */
typedef struct { bls_fq2 x, y; uint64_t infinity; } bls_g2_affine; /* 200 B */
typedef struct { bls_fq2 x, y, z; } bls_g2;                        /* 288 B */
typedef struct { uint64_t l[4]; } bls_fr_repr;                     /* 32 B */
typedef struct { uint64_t l[4]; } bls_fr;                          /* Fr(FrRepr): Montgomery form (x * 2^256 mod r), < r; fr.rs:54-58 */
/* G2Prepared (ec.rs:1615-1619): 68 = 63 doubling + 5 addition coefficient triples in loop order */
typedef struct { bls_fq2 coeffs[68][3]; uint64_t infinity; } bls_g2_prepared; /* 19 592 B */

typedef struct bls_ctx bls_ctx;

typedef enum {
  BLS_OK = 0,
  BLS_ERR_INVALID_ARGUMENT = -1,
  BLS_ERR_NO_DEVICE = -2,
  BLS_ERR_CUDA = -3,
  BLS_ERR_OUT_OF_MEMORY = -4,
  BLS_ERR_UNSUPPORTED = -5
} bls_status;

/* One context = one CUDA device + one ordered stream + reusable device scratch.  `device` is a CUDA
 * ordinal.  Multi-GPU callers create one context per device (one process per GPU under
 * torch.distributed / NCCL, or several contexts in one process) and shard batches themselves;
 * see bls_fq12_product for the only cross-device reduction the path has. */
bls_ctx* bls_ctx_create(int device, int* err);
void bls_ctx_destroy(bls_ctx* ctx);
const char* bls_strerror(int status);
/* text of the last CUDA error seen by this context (empty string if none) */
const char* bls_ctx_last_error(const bls_ctx* ctx);
int bls_ctx_device(const bls_ctx* ctx);
int bls_ctx_sm_count(const bls_ctx* ctx);
/* number of kernel launches issued through this context so far (bench.py's gpu_launches) */
uint64_t bls_ctx_launch_count(const bls_ctx* ctx);
/* The host-buffer entry points stage through device buffers from a per-context memory pool that keeps its memory between
 * calls (no cudaMalloc / cudaFree per call after the first); bls_ctx_trim hands it back, keeping at most keep_bytes. */
int bls_ctx_trim(bls_ctx*, size_t keep_bytes);
/* bls_pairing_* / bls_final_exponentiation_* pick between two kernels by batch size: up to these many elements one WARP
 * works on each element (latency path: ~2 ms for one pairing or for a thousand, the crate's bench_pairing_full shape),
 * above them one lane pair does (throughput path: 8.8 ms of latency, 1.49 M pairings/s).  Same bits either way.
 * 0 disables the latency path.  Defaults: 2560 / 2560 (where the two curves cross on a B200). */
int bls_ctx_set_latency_path_limits(bls_ctx*, size_t max_pairings, size_t max_final_exps);

/* ------------------------------------------------------------------ pairing engine (host buffers) */

/* G2Affine::prepare / G2Prepared::from_affine, bls12_381/mod.rs:168-358, for n points. */
int bls_g2_prepare_batch(bls_ctx*, const bls_g2_affine* q, bls_g2_prepared* out, size_t n);
/* n independent Engine::miller_loop(&[(&p_i.prepare(), &q_i.prepare())]), mod.rs:40-102.
 * Pairs with an infinity member give Fq12::one() (mod.rs:49-54). */
int bls_miller_loop_batch(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n);
/* same, from already prepared G2 coefficients (the reference's actual miller_loop signature) */
int bls_miller_loop_prepared_batch(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q, bls_fq12* out, size_t n);
/* n independent Miller loops / pairings e(P_i, Q) against ONE prepared G2 point: the reference's
 * `let q = Q.prepare(); for p_i { Engine::miller_loop(&[(&p_i.prepare(), &q)]) }` (the reason G2Prepared exists,
 * ec.rs:1615-1619).  The coefficients are staged once per block in shared memory by a TMA bulk copy. */
int bls_miller_loop_shared_q_batch(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n);
int bls_pairing_shared_q_batch(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n);
/* ONE Engine::miller_loop over n pairs: the product of the n Miller values (mod.rs:80-95). */
int bls_multi_miller_loop(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1);
int bls_multi_miller_loop_prepared(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q, size_t n, bls_fq12* out1);
/* Engine::final_exponentiation(&Engine::miller_loop(pairs)) in ONE call -- the batch-verification shape (BASELINE
 * configs[2]): the Miller kernel leaves one partial product per block, one tail kernel folds them and runs the single
 * final exponentiation on the warp-cooperative engine.  *is_some = 0 marks the reference's None (product 0). */
int bls_pairing_product(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, uint8_t* is_some);
/* Engine::final_exponentiation, mod.rs:104-160; is_some[i] = 0 marks the reference's None (input 0),
 * in which case out[i] is all-zero.  is_some may be NULL. */
int bls_final_exponentiation_batch(bls_ctx*, const bls_fq12* in, bls_fq12* out, uint8_t* is_some, size_t n);
/* Engine::pairing on affine inputs, lib.rs:101-109 (Miller loop + final exponentiation). */
int bls_pairing_batch(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n);
/* Engine::pairing(p, q) with PROJECTIVE arguments (`G1: Into<G1Affine>`, `G2: Into<G2Affine>`, lib.rs:101-109) -- how the crate's
 * own bench_pairing_full calls it (benches/bls12_381/mod.rs:91-107): the two into_affine conversions (ec.rs:586-619) are fused in
 * front of the pairing.  A pair with an infinity member gives Fq12::one(). */
int bls_pairing_projective_batch(bls_ctx*, const bls_g1* p, const bls_g2* q, bls_fq12* out, size_t n);
/* product of n Fq12 values (Fq12::mul_assign, fq12.rs:116-130): merges per-device partial Miller
 * products before the single final exponentiation of a sharded multi_miller_loop. */
int bls_fq12_product(bls_ctx*, const bls_fq12* in, size_t n, bls_fq12* out1);

/* Field::pow on Fq12 with an FrRepr exponent (lib.rs:306-324): GT exponentiation e(P,Q)^k, the step after
 * the path in the reference's bilinearity test (tests/engine.rs:93-126). */
int bls_fq12_pow_batch(bls_ctx*, const bls_fq12* a, const bls_fr_repr* k, bls_fq12* out, size_t n);

/* ------------------------------------------------------------------ curve groups (host buffers) */

/* Wnaf::new().scalar(k_i).base(g_i): window from the scalar (ec.rs:895-905 / 1586-1596),
 * wnaf_table + wnaf_form + wnaf_exp (wnaf.rs:4-71).  Output Jacobian triples are bit-identical
 * to the reference's. */
int bls_g1_wnaf_mul_batch(bls_ctx*, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n);
int bls_g2_wnaf_mul_batch(bls_ctx*, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n);
/* same with an explicit window 2..13 (the crate-internal wnaf_table/wnaf_form/wnaf_exp triple, as swept by
 * src/tests/curve.rs:78; windows above 7 keep their 2^(w-1)-entry tables in a per-call global-memory scratch) */
int bls_g1_wnaf_mul_window_batch(bls_ctx*, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n, int window);
int bls_g2_wnaf_mul_window_batch(bls_ctx*, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n, int window);
/* Fixed-base mode Wnaf::new().base(g, num_scalars) then .scalar(k_i) for every scalar (wnaf.rs:93-107,
 * 169-178): ONE window table of 2^(window-1) entries (wnaf_table, wnaf.rs:4-15) shared by all scalars;
 * `window` = recommended_wnaf_for_num_scalars(n) (ec.rs:907-921 / 1598-1612), 2..16.
 * bls_g*_wnaf_table returns the table itself (2^(window-1) Jacobian points, bit-identical to the crate's). */
int bls_g1_wnaf_fixed_base_batch(bls_ctx*, const bls_g1* base, int window, const bls_fr_repr* k, bls_g1* out, size_t n);
int bls_g2_wnaf_fixed_base_batch(bls_ctx*, const bls_g2* base, int window, const bls_fr_repr* k, bls_g2* out, size_t n);
int bls_g1_wnaf_table(bls_ctx*, const bls_g1* base, int window, bls_g1* table);
int bls_g2_wnaf_table(bls_ctx*, const bls_g2* base, int window, bls_g2* table);
/* CurveProjective::mul_assign (double-and-add), ec.rs:534-553 */
int bls_g1_mul_batch(bls_ctx*, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n);
int bls_g2_mul_batch(bls_ctx*, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n);
/* CurveAffine::mul, ec.rs:174-177: $affine::mul_bits (MSB-first over all 256 bits, mixed additions) -- a different
 * Jacobian representative of the same point as mul_assign on the projective form */
int bls_g1_affine_mul_batch(bls_ctx*, const bls_g1_affine* a, const bls_fr_repr* k, bls_g1* out, size_t n);
int bls_g2_affine_mul_batch(bls_ctx*, const bls_g2_affine* a, const bls_fr_repr* k, bls_g2* out, size_t n);
/* CurveProjective::batch_normalization, ec.rs:246-294, in place */
int bls_g1_batch_normalization(bls_ctx*, bls_g1* inout, size_t n);
int bls_g2_batch_normalization(bls_ctx*, bls_g2* inout, size_t n);
/* From<projective> for affine / CurveProjective::into_affine, ec.rs:586-619 */
int bls_g1_into_affine_batch(bls_ctx*, const bls_g1* in, bls_g1_affine* out, size_t n);
int bls_g2_into_affine_batch(bls_ctx*, const bls_g2* in, bls_g2_affine* out, size_t n);
/* element-wise group law: op = BLS_PT_*.  b is bls_g1/bls_g2 (ADD, SUB), bls_g*_affine (ADD_MIXED)
 * or NULL (DOUBLE, NEGATE).  ec.rs:296-532, lib.rs:156-160 */
enum { BLS_PT_DOUBLE = 0, BLS_PT_ADD = 1, BLS_PT_ADD_MIXED = 2, BLS_PT_NEGATE = 3, BLS_PT_SUB = 6 };
int bls_g1_op_batch(bls_ctx*, int op, const bls_g1* a, const void* b, bls_g1* out, size_t n);
int bls_g2_op_batch(bls_ctx*, int op, const bls_g2* a, const void* b, bls_g2* out, size_t n);
/* Multi-scalar multiplication: out1 = sum_i k_i * bases_i (the shape downstream provers and batch verifiers build from
 * CurveAffine::add_assign_mixed, ec.rs:446-526), by the bucket (Pippenger) method.  k_i is the full 256-bit integer of the
 * FrRepr, NOT reduced mod r, so the sum is exact for bases outside the r-order subgroup as well.  Infinity bases and zero
 * scalars contribute nothing.  out1 is the NORMALISED representative -- (x, y, one) as into_projective(into_affine(S)) gives
 * it, or G::zero() = (0, one, 0) -- unique, hence bit-exact whatever the summation order.  n = 0 gives G::zero().
 * n is at most 2^26 (BLS_ERR_INVALID_ARGUMENT above). */
int bls_g1_msm(bls_ctx*, const bls_g1_affine* bases, const bls_fr_repr* k, size_t n, bls_g1* out1);
int bls_g2_msm(bls_ctx*, const bls_g2_affine* bases, const bls_fr_repr* k, size_t n, bls_g2* out1);
/* m independent sums in one call: out[j] = sum_{i<n} k[j*n + i] * bases[b(j, i)] for j < m, where b(j, i) = i if
 * shared_bases != 0 (one set of n bases for every sum: one SRS or proving key) and j*n + i otherwise (m sets of n bases back
 * to back: the different base sets of one proof).  Each out[j] is exactly what bls_g*_msm returns for its n bases and
 * scalars: full 256-bit FrRepr scalars, infinity bases and zero scalars contribute nothing, the normalised representative is
 * stored.  n = 0 stores m zeros; m = 0 does nothing.  Sums of different lengths are padded with zero scalars: a zero digit
 * costs sort work but no addition.  m <= 2^16 and m * n <= 2^26, else BLS_ERR_INVALID_ARGUMENT.  A loop of m bls_g*_msm
 * calls pays the latency of the reduction m times; one batch pays it once. */
int bls_g1_msm_batch(bls_ctx*, const bls_g1_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, bls_g1* out);
int bls_g2_msm_batch(bls_ctx*, const bls_g2_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, bls_g2* out);

/* ------------------------------------------------------------------ point encodings (host buffers)
 * EncodedPoint::into_affine (checked != 0: on-curve and r-order-subgroup checks) / into_affine_unchecked and
 * EncodedPoint::from_affine for G1Uncompressed (96 B) / G1Compressed (48 B) (ec.rs:645-868) and
 * G2Uncompressed (192 B) / G2Compressed (96 B) (ec.rs:1292-1540).  `bytes` holds n encodings back to back.
 * status[i] mirrors GroupDecodingError (src/lib.rs:468-497); a rejected element decodes to the zero point. */
enum {
  BLS_DEC_OK = 0, BLS_DEC_UNEXPECTED_COMPRESSION_MODE = 1, BLS_DEC_UNEXPECTED_INFORMATION = 2,
  BLS_DEC_NOT_ON_CURVE = 3, BLS_DEC_NOT_IN_SUBGROUP = 4,
  BLS_DEC_COORDINATE = 16 /* + coordinate: G1 0 = x, 1 = y; G2 0 = x (c0), 1 = x (c1), 2 = y (c0), 3 = y (c1) */
};
int bls_g1_decode_batch(bls_ctx*, const uint8_t* bytes, int compressed, int checked, bls_g1_affine* out, uint8_t* status, size_t n);
int bls_g2_decode_batch(bls_ctx*, const uint8_t* bytes, int compressed, int checked, bls_g2_affine* out, uint8_t* status, size_t n);
int bls_g1_encode_batch(bls_ctx*, const bls_g1_affine* in, int compressed, uint8_t* bytes, size_t n);
int bls_g2_encode_batch(bls_ctx*, const bls_g2_affine* in, int compressed, uint8_t* bytes, size_t n);

/* G::rand with the randomness supplied by the caller (ec.rs:199-214): $affine::get_point_from_x (ec.rs:102-123; is_some = 0
 * when x^3 + b has no square root) and $affine::scale_by_cofactor (mul_bits with the cofactor, ec.rs:86-94, 871-875,
 * 1564-1578: Jacobian output, infinity possible -- the reference retries). */
int bls_g1_point_from_x_batch(bls_ctx*, const bls_fq* x, const uint8_t* greatest, bls_g1_affine* out, uint8_t* is_some, size_t n);
int bls_g2_point_from_x_batch(bls_ctx*, const bls_fq2* x, const uint8_t* greatest, bls_g2_affine* out, uint8_t* is_some, size_t n);
int bls_g1_scale_by_cofactor_batch(bls_ctx*, const bls_g1_affine* in, bls_g1* out, size_t n);
int bls_g2_scale_by_cofactor_batch(bls_ctx*, const bls_g2_affine* in, bls_g2* out, size_t n);

/* ------------------------------------------------------------------ field tower (host buffers) */
/* Element-wise field operations, the `Field` trait methods of src/lib.rs:267-325 on
 * Fq (degree 1), Fq2 (2), Fq6 (6), Fq12 (12).  `b` is an array of the same element type or NULL.
 * ok[i] = 0 marks None (inverse of 0, from_repr of a non-canonical value); may be NULL. */
enum {
  BLS_OP_ADD = 0, BLS_OP_SUB = 1, BLS_OP_MUL = 2, BLS_OP_SQR = 3, BLS_OP_NEG = 4, BLS_OP_DBL = 5,
  BLS_OP_INV = 6, BLS_OP_FROM_REPR = 7, BLS_OP_INTO_REPR = 8, BLS_OP_MUL_NONRES = 9,
  BLS_OP_FROB1 = 10, BLS_OP_FROB2 = 11, BLS_OP_FROB3 = 12, BLS_OP_CONJ = 13,
  BLS_OP_MUL_BY_014 = 14, /* Fq12 only: sparse operands b.c0.c0, b.c0.c1, b.c1.c1 (fq12.rs:34-48) */
  BLS_OP_MUL_BY_01 = 15,  /* Fq6 only: b.c0, b.c1 (fq6.rs:68-109) */
  BLS_OP_MUL_BY_1 = 16,   /* Fq6 only: b.c1 (fq6.rs:40-66) */
  BLS_OP_SQRT = 17,       /* Fq, Fq2: SqrtField::sqrt (fq.rs:1147-1170, fq2.rs:167-221); ok = 0 for a non-residue */
  /* lane-pair tower only (bls_pair_field_op_batch): */
  BLS_OP_MUL_BY_LINE_PAIR = 18,  /* Fq12: a * l * m for two sparse lines packed in b as (l.c0, l.c1, l.c4, m.c0, m.c1, m.c4) */
  BLS_OP_CYCLOTOMIC_SQR = 19     /* Fq12: Granger-Scott squaring; equals `square` for elements of the cyclotomic subgroup */
};
int bls_field_op_batch(bls_ctx*, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n);
/* The same element-wise operations (degree 2, 6, 12) on the LANE-PAIR tower the pairing kernels run (two lanes per element,
 * lazily reduced dual products): a separate implementation of fq2.rs / fq6.rs / fq12.rs, so it gets its own parity entry.
 * Operands may be any representative in [0, 2q]; results are canonical. */
int bls_pair_field_op_batch(bls_ctx*, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n);
int bls_pair_field_op_dev(bls_ctx*, int degree, int op, const void* a, const void* b, void* out, uint8_t* ok, size_t n, void* stream);

/* The scalar field Fr (fr.rs:324-572), element-wise: op is BLS_OP_ADD / SUB / MUL / SQR / NEG / DBL / INV /
 * FROM_REPR (bls_fr_repr -> bls_fr; ok = 0 for values >= r) / INTO_REPR (bls_fr -> bls_fr_repr).  The step after the
 * path: callers combine scalars (c * d in the reference's bilinearity test, tests/engine.rs:117-119). */
int bls_fr_op_batch(bls_ctx*, int op, const bls_fr* a, const bls_fr* b, bls_fr* out, uint8_t* ok, size_t n);
/* Radix-2 FFT over Fr for m polynomials of n = 2^log_n coefficients each, back to back (m * n bls_fr, natural order in
 * and out): bellman's EvaluationDomain with the crate's constants (fr.rs: S = 32, multiplicative_generator() g = 7,
 * root_of_unity() = 7^t, r - 1 = t * 2^32), omega = root_of_unity() squared (32 - log_n) times.  For i < n:
 *   BLS_FFT         out[i] = sum_j a_j omega^(ij)
 *   BLS_IFFT        out[i] = n^-1 sum_j a_j omega^(-ij)
 *   BLS_COSET_FFT   out[i] = sum_j a_j (g omega^i)^j              (distribute_powers(g), then fft)
 *   BLS_ICOSET_FFT  out[i] = g^-i n^-1 sum_j a_j omega^(-ij)      (ifft, then distribute_powers(g^-1))
 * Inputs must be canonical (< r); outputs are canonical.  in == out (in place) is allowed, otherwise the buffers must not
 * overlap and `in` is left unchanged.  m = 0 does nothing.  log_n in 0..28 and m * 2^log_n <= 2^30, kind in 0..3, else
 * BLS_ERR_INVALID_ARGUMENT. */
enum { BLS_FFT = 0, BLS_IFFT = 1, BLS_COSET_FFT = 2, BLS_ICOSET_FFT = 3 };
int bls_fr_fft_batch(bls_ctx*, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m);
/* Groth16's quotient polynomial H for m proofs: the `h` block of bellman's groth16::create_proof.  Proof j has len
 * evaluations in each of a, b, c (the ProvingAssignment vectors, Montgomery bls_fr, canonical) at a[j*len + i], and so on.
 * With n = 2^log_n the smallest power of two >= len (n = 1 for len <= 1), each proof computes
 *   A, B, C = coset_fft(ifft(x zero-padded to n))                  (EvaluationDomain::from_coeffs, ifft, coset_fft)
 *   H = icoset_fft((A B - C) z(g)^-1), z(g) = g^n - 1, g = 7        (mul_assign, sub_assign, divide_by_z_on_coset)
 * and stores coefficients 0 .. n - 2 of H as canonical bls_fr_repr (coefficient n - 1 is dropped, every one goes through
 * into_repr()) at h[j*(n-1) + i]: the scalars of bls_g1_msm_batch(h_bases, shared_bases = 1, h, n - 1, m, ...).  Outputs are
 * canonical, so bit-exact with any correct evaluation order.  The inputs are left unchanged; h must not overlap them.
 * m = 0 does nothing; len <= 1 stores nothing (n - 1 = 0).  log_n <= 28 and m * n <= 2^28, else BLS_ERR_INVALID_ARGUMENT,
 * as for a NULL pointer when there is something to store. */
int bls_fr_groth16_h_batch(bls_ctx*, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h);
/* Groth16 proofs: bellman's groth16::create_proof for m proofs of one circuit, from the assignments to the proofs.
 * Proof j: a, b, c as for bls_fr_groth16_h_batch (len each, the input constraints create_proof appends included); its
 * input_assignment at input[j*num_inputs + i] (input[0] = one by bellman's convention, not enforced) and aux_assignment at
 * aux[j*num_aux + i]; the blinding values r[j], s[j].  All Montgomery bls_fr.  Density bitmaps (DensityTracker, shared by the
 * m proofs): 32-bit words, bit i at word i / 32, bit i % 32 (bit-vec's BitVec<u32> storage); bits past the end are ignored.
 * With rank_D(i) the number of set bits of D below i and every scalar through into_repr():
 *   h_ans  = sum_{i < n-1} H_i h[i]                                  (H: bls_fr_groth16_h_batch, n the smallest power of two >= len)
 *   l_ans  = sum_{i < num_aux} aux_i l[i]
 *   a_ans  = sum_{i < num_inputs} input_i a[i] + sum_{a_aux_density[i]} aux_i a[num_inputs + rank_a_aux(i)]
 *   b1_ans = sum_{b_input_density[i]} input_i b_g1[rank_b_in(i)] + sum_{b_aux_density[i]} aux_i b_g1[popcount(b_in) + rank_b_aux(i)]
 *   b2_ans = the same over b_g2
 *   A = r delta_g1 + alpha_g1 + a_ans,  B = s delta_g2 + beta_g2 + b2_ans,
 *   C = (r s) delta_g1 + s alpha_g1 + r beta_g1 + s a_ans + r b1_ans + h_ans + l_ans   (bellman's g_c; C = s A + r B_g1 - rs delta_g1)
 * out[j] = (A, B, C) in affine form (into_affine(); the identity is (0, one, infinity = 1)).  Outputs are canonical, so
 * bit-exact with any correct summation order.  Entries of a query past the used prefix are ignored.
 * Differences from bellman: a query base at infinity is summed as zero (bellman stops with UnexpectedIdentity; a key from
 * its generator has none), and one density set serves every proof (the m proofs come from one circuit).
 * BLS_ERR_INVALID_ARGUMENT, before any work: delta_g1 or delta_g2 at infinity (bellman's UnexpectedIdentity); a query
 * shorter than the formula indexes (h_len < n - 1, l_len < num_aux, a_len < num_inputs + popcount(a_aux), b_len <
 * popcount(b_in) + popcount(b_aux)); m > 2^16 or m times one multiexp's length (n - 1, num_aux, a's or b's) > 2^26; a NULL
 * pointer where there is work.  m = 0 does nothing. */
typedef struct { bls_g1_affine a; bls_g2_affine b; bls_g1_affine c; } bls_groth16_proof;   /* 408 B: bellman's Proof<Bls12> */
typedef struct {
  bls_g1_affine alpha_g1, beta_g1, delta_g1;                            /* by value: host memory in both variants */
  bls_g2_affine beta_g2, delta_g2;
  const bls_g1_affine *h, *l, *a, *b_g1;                                /* host pointers for _batch, device pointers for _dev */
  const bls_g2_affine* b_g2;
  size_t h_len, l_len, a_len, b_len;                                    /* b_len: b_g1 and b_g2 have the same length */
} bls_groth16_params;
int bls_groth16_prove_batch(bls_ctx*, const bls_groth16_params* params, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                            const bls_fr* input, size_t num_inputs, const bls_fr* aux, size_t num_aux, const uint32_t* a_aux_density,
                            const uint32_t* b_input_density, const uint32_t* b_aux_density, const bls_fr* r, const bls_fr* s, size_t m,
                            bls_groth16_proof* out);
/* Groth16 verification: bellman's groth16::{prepare_verifying_key, verify_proof} for proofs of one circuit.
 * bls_groth16_pvk is bellman's PreparedVerifyingKey without ic (passed separately, like the prover's queries), plus the two
 * negated G2 points in affine form.  Both prepared points start at a multiple of 16 bytes (the pads), so that the
 * verification kernel can stage their coefficients by TMA bulk copies.  bls_groth16_prepare_verifying_key fills it from the
 * vk points: alpha_g1_beta_g2 = pairing(alpha_g1, beta_g2), neg_gamma_g2 = prepare(-gamma_g2), neg_delta_g2 =
 * prepare(-delta_g2), bit-exact with bellman; the pads are zero.  NULL pointers give BLS_ERR_INVALID_ARGUMENT. */
typedef struct {
  bls_g2_prepared neg_gamma_g2;                                      /* offset 0 */
  uint64_t pad0;
  bls_g2_prepared neg_delta_g2;                                      /* offset 19 600 */
  uint64_t pad1;
  bls_fq12 alpha_g1_beta_g2;                                         /* offset 39 200 */
  bls_g2_affine neg_gamma_g2_affine, neg_delta_g2_affine;            /* offsets 39 776, 39 976 */
} bls_groth16_pvk;                                                   /* 40 176 B */
int bls_groth16_prepare_verifying_key(bls_ctx*, const bls_g1_affine* alpha_g1, const bls_g2_affine* beta_g2, const bls_g2_affine* gamma_g2,
                                      const bls_g2_affine* delta_g2, bls_groth16_pvk* out);
/* bellman's verify_proof for m proofs of one circuit.  ic holds the vk's num_inputs + 1 points; proof j's public inputs are
 * inputs[j*num_inputs + i], Montgomery bls_fr without bellman's leading one, as verify_proof takes them.  With
 * acc_j = ic[0] + sum_i x_ji ic[i + 1]:
 *   ok[j] = 1  iff  final_exponentiation(miller_loop([(A_j, B_j), (acc_j, -gamma), (C_j, -delta)])) == alpha_g1_beta_g2,
 * else 0 (a None from the final exponentiation gives 0).  A pair with a member at infinity (A_j, B_j, acc_j or C_j) contributes
 * one, as in Engine::miller_loop.  Like bellman, the call does not validate points: decode proofs with
 * bls_g*_decode_batch(checked = 1).  m <= 2^16 and m * (num_inputs + 1) <= 2^26 (bls_g1_msm_batch's limits); outside them,
 * or for a NULL pointer where there is work, BLS_ERR_INVALID_ARGUMENT before any work.  m = 0 does nothing. */
int bls_groth16_verify_batch(bls_ctx*, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                             const bls_fr* inputs, size_t m, uint8_t* ok);
/* Randomized batch verification (bellperson's verify_proofs_batch): one verdict for m proofs, with the caller's randomizers
 * rho[j] (canonical bls_fr_repr, < r; the library has no RNG).  With s_0 = sum_j rho_j and s_i = sum_j rho_j x_j(i-1) (mod r):
 *   *ok1 = 1  iff  FE( prod_j ML(rho_j A_j, B_j) * ML(sum_i s_i ic_i, -gamma) * ML(sum_j rho_j C_j, -delta) )
 *                  == alpha_g1_beta_g2 ^ (sum_j rho_j),
 * exactly this equation; else 0.  A proof with rho_j = 0 is left out of it.  With random rho an invalid proof makes the
 * verdict 0 except with probability about 1/r.  Limits are those of the multiexps and the product: m <= 2^26 and
 * num_inputs + 1 <= 2^26, else BLS_ERR_INVALID_ARGUMENT, as for a NULL pointer where there is work.  m = 0 sets *ok1 = 1
 * (the equation holds for the empty batch: both sides are one) when ok1 is not NULL, and does nothing else. */
int bls_groth16_verify_rlc_batch(bls_ctx*, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                                 const bls_fr* inputs, const bls_fr_repr* rho, size_t m, uint8_t* ok1);
/* Groth16 parameters: bellman's groth16::generate_parameters(circuit, g1, g2, alpha, beta, gamma, delta, tau), bit-exact, with
 * the toxic waste and the bases supplied by the caller (generate_random_parameters is the caller drawing them).
 * The circuit: num_inputs input variables (input 0 is ONE by bellman's convention, not enforced), num_aux aux variables and
 * num_constraints constraints, the input_i * 0 = 0 constraints the generator appends included (the prover's len).  abc holds
 * A, B and C as KeypairAssembly records them (at_inputs / at_aux ...), variable-major: variable v (inputs, then aux) owns
 * the terms offsets[v] .. offsets[v + 1] - 1, each a constraint index and a Montgomery bls_fr coefficient.  Terms are not
 * merged: a variable may have several terms in one constraint, and coefficients may be zero.
 * With n the smallest power of two >= num_constraints (1 for 0 or 1), Lq = ifft(tau^0 .. tau^(n-1)) (the Lagrange basis at
 * tau of the omega^q), u_v = sum coeff Lq[constraint] over A's terms of v, and v_v, w_v the same over B and C:
 *   h[i]  = [tau^i (tau^n - 1) delta^-1] g1                for i < n - 1 (never filtered)
 *   ic[i] = [(beta u_i + alpha v_i + w_i) gamma^-1] g1     for each input i
 *   l[i]  = [(beta u + alpha v + w) delta^-1] g1          for each aux i
 *   a     = [u_v] g1 over every variable, inputs then aux, identities dropped (the inputs too, as in bellman)
 *   b_g1, b_g2 = [v_v] g1, [v_v] g2 over every variable, identities dropped (one length: g1, g2 are not the identity)
 *   vk    = alpha_g1 = [alpha] g1, beta_g1 = [beta] g1, beta_g2 = [beta] g2, gamma_g2 = [gamma] g2, delta_g1, delta_g2
 *   a_aux_density bit i = (u of aux i != 0), b_input_density bit i = (v of input i != 0), b_aux_density bit i = (v of aux
 *   i != 0): BitVec<u32> words as bls_groth16_prove_* takes them, unused high bits of the last word zero
 *   lens  = [a_len, b_len];  ok = 0 iff some l[i] is the identity (bellman's SynthesisError::UnconstrainedVariable; the rest of
 *   the key is still written), else 1.
 * Every point is a canonical affine row; the identity is (0, one, infinity = 1).  g1 and g2 must have order r (bellman's
 * generators do), for which [k] g is the identity exactly when k = 0.
 * BLS_ERR_INVALID_ARGUMENT, before any work: gamma or delta zero (bellman's UnexpectedIdentity from inverse()); a scalar
 * >= r; g1 or g2 at infinity (a difference from bellman, whose key would then have b_g1 and b_g2 of different lengths); a
 * NULL pointer where there is something to read or write; n > 2^26, num_inputs + num_aux > 2^26 (so that every query fits
 * the prover's m * multiexp length <= 2^26) or a matrix with 2^31 terms or more, or with terms but no variables.  The host
 * form also rejects offsets that do not rise from 0 to nnz, a constraint index >= num_constraints and a coefficient >= r.
 * Shared with bellman: when an input's u_i(tau) = 0 (probability about 1/r, or an adversarial tau such as a domain point
 * omega^k), a is shorter than num_inputs + popcount(a_aux_density); bls_groth16_prove_* rejects such a key. */
typedef struct { const uint64_t* offsets; const uint32_t* constraint; const bls_fr* coeff; size_t nnz; } bls_r1cs_matrix;  /* offsets: nv + 1 */
typedef struct { bls_g1_affine alpha_g1, beta_g1, delta_g1; bls_g2_affine beta_g2, gamma_g2, delta_g2; } bls_groth16_vk_points;  /* 114 u64 */
typedef struct {                                   /* host pointers for _batch, device pointers for _dev */
  bls_groth16_vk_points* vk;
  bls_g1_affine *ic, *h, *l, *a, *b_g1;            /* num_inputs, n - 1, num_aux, and num_inputs + num_aux for a and b_g1 */
  bls_g2_affine* b_g2;                             /* num_inputs + num_aux */
  uint32_t *a_aux_density, *b_input_density, *b_aux_density;   /* ceil(num_aux / 32), ceil(num_inputs / 32), ceil(num_aux / 32) */
  uint64_t* lens;                                  /* [a_len, b_len] */
  uint8_t* ok;
} bls_groth16_parameters_out;
int bls_groth16_generate_parameters_batch(bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                                          const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_fr* alpha, const bls_fr* beta,
                                          const bls_fr* gamma, const bls_fr* delta, const bls_fr* tau, const bls_groth16_parameters_out* out);

/* ------------------------------------------------------------------ KZG polynomial commitments
 * The SRS is srs[i] = [tau^i] g in G1 for i < srs_len (affine rows), plus h and [tau] h in G2; the caller supplies all of it
 * (the library has no RNG and no setup file), and the Fiat-Shamir challenges z_j and randomizers rho_j as well.  Polynomials
 * are in coefficient form, p(X) = sum_{i<n} p_i X^i, Montgomery bls_fr, canonical, m polynomials back to back (p[j*n + i]:
 * the layout bls_fr_fft_* produces).  n is any length.  Points leave as canonical affine rows (the identity is (0, one,
 * infinity = 1)), so outputs are bit-exact whatever the summation order.  m = 0 does nothing.  BLS_ERR_INVALID_ARGUMENT,
 * before any work: a NULL pointer where there is work, an SRS shorter than the formula indexes, sizes over the limits.
 *
 * commit: c[j] = sum_{i<n} p_ji srs[i].  srs_len >= n; m <= 2^16 and m * n <= 2^26 (bls_g1_msm_batch's limits). */
int bls_kzg_commit_batch(bls_ctx*, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, size_t m, bls_g1_affine* c);
/* open at z_j (Montgomery bls_fr): y[j] = p_j(z_j) (Montgomery bls_fr) and proof[j] = sum_{i<n-1} q_ji srs[i] with
 * q_j(X) = (p_j(X) - y_j) / (X - z_j), q_i = sum_{k>i} p_k z^(k-i-1): the unique [q(tau)] g.  n = 0 gives y = 0 and the
 * identity, n = 1 gives y = p_0 and the identity.  srs_len >= n - 1; the limits of commit. */
int bls_kzg_open_batch(bls_ctx*, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, const bls_fr* z, size_t m, bls_fr* y,
                       bls_g1_affine* proof);
/* The verifying key: prepare(h) at offset 0 and prepare(-tau h) at a 16-byte aligned offset (the pads; zero), so that the
 * verification kernel can stage both coefficient arrays by bulk copies, then g, h and -tau h in affine form.  NULL pointers
 * give BLS_ERR_INVALID_ARGUMENT. */
typedef struct {
  bls_g2_prepared h_prepared;                                        /* offset 0 */
  uint64_t pad0;
  bls_g2_prepared neg_tau_h_prepared;                                /* offset 19 600 */
  uint64_t pad1;
  bls_g1_affine g;                                                   /* offset 39 200 */
  bls_g2_affine h, neg_tau_h;                                        /* offsets 39 304, 39 504 */
} bls_kzg_pvk;                                                       /* 39 704 B */
int bls_kzg_prepare_verifying_key(bls_ctx*, const bls_g1_affine* g, const bls_g2_affine* h, const bls_g2_affine* tau_h, bls_kzg_pvk* out);
/* verify, one byte per proof:
 *   ok[j] = 1  iff  FE(ML(C_j - y_j g + z_j proof_j, h) * ML(proof_j, -tau h)) == 1   (e(C - y g, h) == e(proof, tau h - z h)),
 * else 0; also 0 when y_j or z_j is not < r (rejected, not reduced).  A pair with a member at infinity contributes one, as in
 * Engine::miller_loop.  Points are not validated: decode them with bls_g*_decode_batch(checked = 1).  m <= 2^26. */
int bls_kzg_verify_batch(bls_ctx*, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                         size_t m, uint8_t* ok);
/* randomized check, one verdict for m proofs with the caller's randomizers rho[j] (canonical bls_fr_repr, < r):
 *   *ok1 = 1  iff  FE(ML(sum_j rho_j (C_j - y_j g + z_j proof_j), h) * ML(sum_j rho_j proof_j, -tau h)) == 1,
 * exactly this equation (for points of order r), else 0; 0 as well when some y_j or z_j is not < r.  rho_j = 0 leaves proof j
 * out.  The first sum is one bls_g1_msm over the 2m + 1 bases [C_0 .. C_(m-1), proof_0 .. proof_(m-1), g], so m < 2^25
 * (2m + 1 <= 2^26, bls_g1_msm's limit).  m = 0 sets *ok1 = 1 when ok1 is not NULL. */
int bls_kzg_verify_rlc_batch(bls_ctx*, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                             const bls_fr_repr* rho, size_t m, uint8_t* ok1);

/* ------------------------------------------------------------------ device-pointer variants
 * Same semantics; every pointer is a device pointer on the context's device, the work is enqueued
 * on `stream` (a cudaStream_t, NULL = the context's own stream) and NOT synchronised.  `scratch`
 * arguments are caller-provided device buffers of the stated size (so no allocation happens on the
 * timed path). */
int bls_g2_prepare_dev(bls_ctx*, const bls_g2_affine* q, bls_g2_prepared* out, size_t n, void* stream);
int bls_miller_loop_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, void* stream);
int bls_miller_loop_prepared_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q, bls_fq12* out, size_t n, void* stream);
int bls_final_exponentiation_dev(bls_ctx*, const bls_fq12* in, bls_fq12* out, uint8_t* is_some, size_t n, void* stream);
int bls_pairing_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n, void* stream);
int bls_pairing_projective_dev(bls_ctx*, const bls_g1* p, const bls_g2* q, bls_fq12* out, size_t n, void* stream);
/* q1: ONE prepared point in device memory, 16-byte aligned; final_exp != 0 adds the final exponentiation */
int bls_miller_loop_shared_q_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_prepared* q1, bls_fq12* out, size_t n, int final_exp, void* stream);
int bls_fq12_pow_dev(bls_ctx*, const bls_fq12* a, const bls_fr_repr* k, bls_fq12* out, size_t n, void* stream);
/* scratch: bls_multi_miller_scratch_bytes(ctx, n) bytes */
size_t bls_multi_miller_scratch_bytes(const bls_ctx*, size_t n);
int bls_multi_miller_loop_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, void* scratch, void* stream);
int bls_pairing_product_dev(bls_ctx*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, uint8_t* is_some, void* scratch, void* stream);
/* product of n Fq12 values by ONE block (n up to a few thousand: the per-block or per-device partials of a sharded
 * multi_miller_loop), then -- final_exp != 0 -- Engine::final_exponentiation of the product (mod.rs:104-160) on the
 * warp-cooperative engine.  No scratch.  is_some (device pointer, may be NULL) as in bls_final_exponentiation_dev. */
int bls_fq12_product_tail_dev(bls_ctx*, const bls_fq12* in, size_t n, bls_fq12* out1, int final_exp, uint8_t* is_some, void* stream);
size_t bls_fq12_product_scratch_bytes(const bls_ctx*, size_t n);
int bls_fq12_product_dev(bls_ctx*, const bls_fq12* in, size_t n, bls_fq12* out1, void* scratch, void* stream);
int bls_g1_wnaf_mul_dev(bls_ctx*, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n, int window, void* stream);
int bls_g2_wnaf_mul_dev(bls_ctx*, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n, int window, void* stream);
/* fixed-base mode on the device: `table` holds 2^(window-1) points, built by bls_g*_wnaf_table_dev */
int bls_g1_wnaf_table_dev(bls_ctx*, const bls_g1* base, int window, bls_g1* table, void* stream);
int bls_g2_wnaf_table_dev(bls_ctx*, const bls_g2* base, int window, bls_g2* table, void* stream);
int bls_g1_wnaf_fixed_base_dev(bls_ctx*, const bls_g1* table, int window, const bls_fr_repr* k, bls_g1* out, size_t n, void* stream);
int bls_g2_wnaf_fixed_base_dev(bls_ctx*, const bls_g2* table, int window, const bls_fr_repr* k, bls_g2* out, size_t n, void* stream);
/* scratch: bls_batch_normalization_scratch_bytes(ctx, degree, n) bytes; degree 1 = G1, 2 = G2 */
size_t bls_batch_normalization_scratch_bytes(const bls_ctx*, int degree, size_t n);
int bls_g1_batch_normalization_dev(bls_ctx*, bls_g1* inout, size_t n, void* scratch, void* stream);
int bls_g2_batch_normalization_dev(bls_ctx*, bls_g2* inout, size_t n, void* scratch, void* stream);
/* bls_g*_msm on device pointers; out1 is one device point.  window = bucket width c in bits, 2..20, or 0 = the library's
 * choice for n.  n <= 2^26 and ceil(257 / c) * n < 2^31, else BLS_ERR_INVALID_ARGUMENT.  scratch: bls_msm_scratch_bytes(ctx,
 * degree, n, window) bytes (degree 1 = G1, 2 = G2; 0 for invalid arguments); it holds everything, including the radix sort's
 * temporary storage: the call allocates nothing. */
size_t bls_msm_scratch_bytes(const bls_ctx*, int degree, size_t n, int window);
int bls_g1_msm_dev(bls_ctx*, const bls_g1_affine* bases, const bls_fr_repr* k, size_t n, int window, bls_g1* out1, void* scratch, void* stream);
int bls_g2_msm_dev(bls_ctx*, const bls_g2_affine* bases, const bls_fr_repr* k, size_t n, int window, bls_g2* out1, void* scratch, void* stream);
/* bls_g*_msm_batch on device pointers; out holds m device points.  window as for bls_g*_msm_dev, with W = ceil(257 / c):
 * m <= 2^16, m * n <= 2^26, W * m * n < 2^31 and m * W * 2^(c-1) < 2^31, else BLS_ERR_INVALID_ARGUMENT; window = 0 is
 * valid for every such m and n.  scratch: bls_msm_batch_scratch_bytes(ctx, degree, n, m, window) bytes (0 for invalid
 * arguments); bls_msm_scratch_bytes(ctx, degree, n, window) equals it for m = 1, and bls_g*_msm_dev is the m = 1 call. */
size_t bls_msm_batch_scratch_bytes(const bls_ctx*, int degree, size_t n, size_t m, int window);
int bls_g1_msm_batch_dev(bls_ctx*, const bls_g1_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, int window, bls_g1* out, void* scratch, void* stream);
int bls_g2_msm_batch_dev(bls_ctx*, const bls_g2_affine* bases, int shared_bases, const bls_fr_repr* k, size_t n, size_t m, int window, bls_g2* out, void* scratch, void* stream);
/* bls_fr_fft_batch on device pointers, same arguments and limits.  scratch: bls_fr_fft_scratch_bytes(ctx, log_n, m)
 * bytes (0 for invalid arguments; the same for every kind); it holds the twiddle tables the call builds and, for
 * log_n > 10, one buffer of m * 2^log_n elements between passes: the call allocates nothing. */
size_t bls_fr_fft_scratch_bytes(const bls_ctx*, int log_n, size_t m);
int bls_fr_fft_dev(bls_ctx*, int kind, const bls_fr* in, bls_fr* out, int log_n, size_t m, void* scratch, void* stream);
/* bls_fr_groth16_h_batch on device pointers, same arguments and limits.  scratch: bls_fr_groth16_h_scratch_bytes(ctx, len,
 * m) bytes (0 for invalid arguments): 3m * n elements for A, B and C of every proof, then bls_fr_fft_scratch_bytes(ctx,
 * log_n, 3m) for the transforms; it must not overlap the other buffers.  The call allocates nothing. */
size_t bls_fr_groth16_h_scratch_bytes(const bls_ctx*, size_t len, size_t m);
int bls_fr_groth16_h_dev(bls_ctx*, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len, size_t m, bls_fr_repr* h, void* scratch, void* stream);
/* bls_fr_op_batch on device pointers: the same ops, NULL rules for b and ok, and results.  out may equal a or b.  The way
 * between Montgomery bls_fr and bls_fr_repr (FROM_REPR / INTO_REPR) for data that stays on the device. */
int bls_fr_op_dev(bls_ctx*, int op, const bls_fr* a, const bls_fr* b, bls_fr* out, uint8_t* ok, size_t n, void* stream);
/* bls_groth16_prove_batch on device pointers: a, b, c, input, aux, r, s, out and the params' query pointers; params and
 * the density bitmaps stay in host memory (their popcounts set the multiexp lengths).  Same limits.  scratch:
 * bls_groth16_prove_scratch_bytes(ctx, the same arguments) bytes (0 for invalid arguments): the vk points and bitmap words
 * (copied with cudaMemcpyAsync on `stream`), the five sums and the r / s products, the scalars of the five multiexps, and
 * one region for H's transforms and each multiexp in turn.  The call allocates nothing and does not synchronise. */
size_t bls_groth16_prove_scratch_bytes(const bls_ctx*, const bls_groth16_params* params, size_t len, size_t num_inputs, size_t num_aux,
                                       const uint32_t* a_aux_density, const uint32_t* b_input_density, const uint32_t* b_aux_density, size_t m);
int bls_groth16_prove_dev(bls_ctx*, const bls_groth16_params* params, const bls_fr* a, const bls_fr* b, const bls_fr* c, size_t len,
                          const bls_fr* input, size_t num_inputs, const bls_fr* aux, size_t num_aux, const uint32_t* a_aux_density,
                          const uint32_t* b_input_density, const uint32_t* b_aux_density, const bls_fr* r, const bls_fr* s, size_t m,
                          bls_groth16_proof* out, void* scratch, void* stream);
/* bls_groth16_verify_batch / bls_groth16_verify_rlc_batch on device pointers: pvk, ic, proofs, inputs, rho and ok / ok1 (one
 * byte).  pvk must be 16-byte aligned.  Same limits.  scratch: bls_groth16_verify_scratch_bytes(ctx, num_inputs, m) (the msm
 * scalars and sums and the msm's work region) or bls_groth16_verify_rlc_scratch_bytes(ctx, num_inputs, m) (the pairs of the
 * product, the scalars s and the msm and product work regions) bytes, 0 for invalid arguments.  The calls allocate nothing
 * and do not synchronise. */
size_t bls_groth16_verify_scratch_bytes(const bls_ctx*, size_t num_inputs, size_t m);
int bls_groth16_verify_dev(bls_ctx*, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                           const bls_fr* inputs, size_t m, uint8_t* ok, void* scratch, void* stream);
size_t bls_groth16_verify_rlc_scratch_bytes(const bls_ctx*, size_t num_inputs, size_t m);
int bls_groth16_verify_rlc_dev(bls_ctx*, const bls_groth16_pvk* pvk, const bls_g1_affine* ic, size_t num_inputs, const bls_groth16_proof* proofs,
                               const bls_fr* inputs, const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream);
/* bls_groth16_generate_parameters_batch on device pointers: the matrices' offsets, constraint and coeff arrays and every
 * pointer of `out`; abc itself, g1, g2 and the five scalars stay in host memory, so their checks happen before any work.
 * The matrices' contents are NOT validated up front, but every device read stays inside the caller's buffers whatever they
 * hold (offsets are clamped to nnz, a constraint index >= num_constraints or a coefficient >= r makes its term contribute
 * zero) and a malformed matrix sets ok = 0.  Only the first a_len rows of a and b_len rows of b_g1 and b_g2 are written.
 * scratch: bls_groth16_generate_parameters_scratch_bytes(ctx, abc, num_constraints, num_inputs, num_aux) bytes (0 for
 * invalid arguments): the scalars, the Lagrange basis and its transform's work region, the QAP sums, the G1 and G2 scalars
 * and points of the exponentiations, the two wNAF tables and the normalisation's work region.  The call allocates nothing
 * and does not synchronise. */
size_t bls_groth16_generate_parameters_scratch_bytes(const bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs,
                                                     size_t num_aux);
int bls_groth16_generate_parameters_dev(bls_ctx*, const bls_r1cs_matrix abc[3], size_t num_constraints, size_t num_inputs, size_t num_aux,
                                        const bls_g1_affine* g1, const bls_g2_affine* g2, const bls_fr* alpha, const bls_fr* beta, const bls_fr* gamma,
                                        const bls_fr* delta, const bls_fr* tau, const bls_groth16_parameters_out* out, void* scratch, void* stream);
/* bls_kzg_* on device pointers: srs, p, z, y, c / proof, pvk (16-byte aligned), rho and ok / ok1.  Same limits.  scratch:
 * bls_kzg_*_scratch_bytes(ctx, ...) bytes, 0 for invalid arguments -- commit: the msm scalars, the m sums and the multiexp's
 * work region; open: the quotient coefficients, the scan's upper levels (about m n / 31 elements), the sums and the
 * multiexp's; verify: the m G1 terms, the range flags and the normalisation's; verify_rlc: the 2m + 1 bases and scalars, the
 * two sums and the multiexp's.  The calls allocate nothing and do not synchronise. */
size_t bls_kzg_commit_scratch_bytes(const bls_ctx*, size_t n, size_t m);
int bls_kzg_commit_dev(bls_ctx*, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, size_t m, bls_g1_affine* c, void* scratch,
                       void* stream);
size_t bls_kzg_open_scratch_bytes(const bls_ctx*, size_t n, size_t m);
int bls_kzg_open_dev(bls_ctx*, const bls_g1_affine* srs, size_t srs_len, const bls_fr* p, size_t n, const bls_fr* z, size_t m, bls_fr* y,
                     bls_g1_affine* proof, void* scratch, void* stream);
size_t bls_kzg_verify_scratch_bytes(const bls_ctx*, size_t m);
int bls_kzg_verify_dev(bls_ctx*, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                       size_t m, uint8_t* ok, void* scratch, void* stream);
size_t bls_kzg_verify_rlc_scratch_bytes(const bls_ctx*, size_t m);
int bls_kzg_verify_rlc_dev(bls_ctx*, const bls_kzg_pvk* pvk, const bls_g1_affine* c, const bls_fr* y, const bls_fr* z, const bls_g1_affine* proof,
                           const bls_fr_repr* rho, size_t m, uint8_t* ok1, void* scratch, void* stream);

/* ------------------------------------------------------------------ several GPUs behind ONE call
 * Engine::miller_loop takes ALL pairs of a product in one call (mod.rs:40-102), and a Rust / C caller is one process.
 * A bls_mgpu binds n devices of one node.  An n-pair product is split into contiguous shards, one host thread per
 * device; every device reduces its shard to ONE 576-byte partial product, the partials travel to the first device by
 * peer copies (NVLink; staged through the host where peer access is unavailable), and the first device folds them and
 * runs the single final exponentiation.  Independent batches (pairings, wNAF multiplications) are sharded the same
 * way with no exchange step.  devices == NULL selects devices 0 .. n_devices-1. */
typedef struct bls_mgpu bls_mgpu;
bls_mgpu* bls_mgpu_create(const int* devices, int n_devices, int* err);
void bls_mgpu_destroy(bls_mgpu*);
int bls_mgpu_device_count(const bls_mgpu*);
bls_ctx* bls_mgpu_ctx(bls_mgpu*, int i);   /* the single-device context of shard i (owned by the bls_mgpu) */
int bls_mgpu_multi_miller_loop(bls_mgpu*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1);
int bls_mgpu_pairing_product(bls_mgpu*, const bls_g1_affine* p, const bls_g2_affine* q, size_t n, bls_fq12* out1, uint8_t* is_some);
int bls_mgpu_pairing_batch(bls_mgpu*, const bls_g1_affine* p, const bls_g2_affine* q, bls_fq12* out, size_t n);
int bls_mgpu_g1_wnaf_mul_batch(bls_mgpu*, const bls_g1* bases, const bls_fr_repr* k, bls_g1* out, size_t n);
int bls_mgpu_g2_wnaf_mul_batch(bls_mgpu*, const bls_g2* bases, const bls_fr_repr* k, bls_g2* out, size_t n);
/* host wall-clock phases of the last product call, milliseconds: ms3[0] = shards (H2D + Miller kernel + per-device
 * fold + peer copy, slowest device), ms3[1] = fold of the partials + final exponentiation + D2H, ms3[2] = whole call */
int bls_mgpu_last_phase_ms(const bls_mgpu*, double* ms3);

/* ------------------------------------------------------------------ measurement
 * Register-resident integer-multiply microbenchmark: the roofline denominator for this path
 * (MEASURED_PEAKS.json has no integer figure).  variant 0 = chains of dependent IMAD.WIDE.U32
 * (32x32->64, the only multiply in the loop -- checked on the SASS by tests/test_abi.py),
 * 1 = back-to-back fp_mul (300 MAC32 each), 2 = 32-bit IMAD, 3 = carry-linked
 * IMAD.WIDE.U32.X rows only (mad.lo.cc / madc.hi.cc chains, no reduction), 4 = back-to-back dedicated squarings
 * (fq.rs:963-1016; 234 MAC32 each).
 * Returns multiply-accumulates per second in *macs_per_s and the kernel time in *ms. */
int bls_imad_peak(bls_ctx*, int variant, int iters, double* macs_per_s, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* PAIRING_B200_H */
