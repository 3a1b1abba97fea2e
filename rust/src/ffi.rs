//! Raw bindings of include/pairing_b200.h.  POD mirrors are `#[repr(C)]`; the crate's own `Fq`,
//! `G1Affine`, ... are NOT (`pub(crate)` fields, no repr), so `lib.rs` marshals explicitly.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] #[derive(Copy, Clone)] pub struct bls_fq { pub l: [u64; 6] }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_fq2 { pub c0: bls_fq, pub c1: bls_fq }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_fq6 { pub c0: bls_fq2, pub c1: bls_fq2, pub c2: bls_fq2 }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_fq12 { pub c0: bls_fq6, pub c1: bls_fq6 }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_g1_affine { pub x: bls_fq, pub y: bls_fq, pub infinity: u64 }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_g1 { pub x: bls_fq, pub y: bls_fq, pub z: bls_fq }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_g2_affine { pub x: bls_fq2, pub y: bls_fq2, pub infinity: u64 }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_g2 { pub x: bls_fq2, pub y: bls_fq2, pub z: bls_fq2 }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_fr_repr { pub l: [u64; 4] }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_groth16_proof { pub a: bls_g1_affine, pub b: bls_g2_affine, pub c: bls_g1_affine }
#[repr(C)] pub struct bls_groth16_params {
    pub alpha_g1: bls_g1_affine, pub beta_g1: bls_g1_affine, pub delta_g1: bls_g1_affine,
    pub beta_g2: bls_g2_affine, pub delta_g2: bls_g2_affine,
    pub h: *const bls_g1_affine, pub l: *const bls_g1_affine, pub a: *const bls_g1_affine, pub b_g1: *const bls_g1_affine,
    pub b_g2: *const bls_g2_affine,
    pub h_len: usize, pub l_len: usize, pub a_len: usize, pub b_len: usize,
}
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_g2_prepared { pub coeffs: [[bls_fq2; 3]; 68], pub infinity: u64 }
/// bellman's PreparedVerifyingKey without ic, plus -gamma_g2 and -delta_g2 in affine form; the pads keep both prepared points
/// 16-byte aligned (40 176 bytes)
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_groth16_pvk {
    pub neg_gamma_g2: bls_g2_prepared, pub pad0: u64, pub neg_delta_g2: bls_g2_prepared, pub pad1: u64,
    pub alpha_g1_beta_g2: bls_fq12, pub neg_gamma_g2_affine: bls_g2_affine, pub neg_delta_g2_affine: bls_g2_affine,
}
/// KZG verifying key: prepare(h) and prepare(-tau h) at 16-byte aligned offsets (the pads), then g, h, -tau h (39 704 bytes)
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_kzg_pvk {
    pub h_prepared: bls_g2_prepared, pub pad0: u64, pub neg_tau_h_prepared: bls_g2_prepared, pub pad1: u64,
    pub g: bls_g1_affine, pub h: bls_g2_affine, pub neg_tau_h: bls_g2_affine,
}
/// one of A, B, C variable-major, as KeypairAssembly records it: the terms of variable v are offsets[v] .. offsets[v + 1]
#[repr(C)] pub struct bls_r1cs_matrix { pub offsets: *const u64, pub constraint: *const u32, pub coeff: *const bls_fr_repr, pub nnz: usize }
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_groth16_vk_points {
    pub alpha_g1: bls_g1_affine, pub beta_g1: bls_g1_affine, pub delta_g1: bls_g1_affine,
    pub beta_g2: bls_g2_affine, pub gamma_g2: bls_g2_affine, pub delta_g2: bls_g2_affine,
}
#[repr(C)] pub struct bls_groth16_parameters_out {
    pub vk: *mut bls_groth16_vk_points,
    pub ic: *mut bls_g1_affine, pub h: *mut bls_g1_affine, pub l: *mut bls_g1_affine, pub a: *mut bls_g1_affine, pub b_g1: *mut bls_g1_affine,
    pub b_g2: *mut bls_g2_affine,
    pub a_aux_density: *mut u32, pub b_input_density: *mut u32, pub b_aux_density: *mut u32,
    pub lens: *mut u64, pub ok: *mut u8,
}
/// powersoftau's prepare_phase2 rows for a domain of n points (include/pairing_b200_mpc.h): n rows per coefficient set, n - 1 h rows
#[repr(C)] pub struct bls_groth16_phase1 {
    pub alpha_g1: bls_g1_affine, pub beta_g1: bls_g1_affine, pub beta_g2: bls_g2_affine,
    pub coeffs_g1: *const bls_g1_affine, pub alpha_coeffs_g1: *const bls_g1_affine, pub beta_coeffs_g1: *const bls_g1_affine,
    pub coeffs_g2: *const bls_g2_affine, pub h: *const bls_g1_affine, pub n: usize,
}
/// phase2's PublicKey without its transcript hash, plus r = hash_to_g2(transcript)
#[repr(C)] #[derive(Copy, Clone)] pub struct bls_groth16_mpc_pubkey {
    pub delta_after: bls_g1_affine, pub s: bls_g1_affine, pub s_delta: bls_g1_affine, pub r: bls_g2_affine, pub r_delta: bls_g2_affine,
}
/// bellman's Parameters<Bls12> for bls_groth16_mpc_verify_batch: the vk by value, the queries by pointer
#[repr(C)] pub struct bls_groth16_key {
    pub vk: bls_groth16_vk_points,
    pub ic: *const bls_g1_affine, pub h: *const bls_g1_affine, pub l: *const bls_g1_affine, pub a: *const bls_g1_affine,
    pub b_g1: *const bls_g1_affine, pub b_g2: *const bls_g2_affine,
    pub ic_len: usize, pub h_len: usize, pub l_len: usize, pub a_len: usize, pub b_len: usize,
}
pub enum bls_ctx {}
/// several devices of one node behind one call (include/pairing_b200.h, "several GPUs")
pub enum bls_mgpu {}

pub const BLS_OK: c_int = 0;
pub const BLS_ERR_INVALID_ARGUMENT: c_int = -1;

extern "C" {
    pub fn bls_ctx_create(device: c_int, err: *mut c_int) -> *mut bls_ctx;
    pub fn bls_ctx_destroy(ctx: *mut bls_ctx);
    pub fn bls_strerror(status: c_int) -> *const c_char;
    pub fn bls_ctx_last_error(ctx: *const bls_ctx) -> *const c_char;

    pub fn bls_g2_prepare_batch(ctx: *mut bls_ctx, q: *const bls_g2_affine, out: *mut bls_g2_prepared, n: usize) -> c_int;
    pub fn bls_miller_loop_batch(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_affine, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_miller_loop_prepared_batch(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_prepared, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_miller_loop_shared_q_batch(ctx: *mut bls_ctx, p: *const bls_g1_affine, q1: *const bls_g2_prepared, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_pairing_shared_q_batch(ctx: *mut bls_ctx, p: *const bls_g1_affine, q1: *const bls_g2_prepared, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_multi_miller_loop(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_affine, n: usize, out1: *mut bls_fq12) -> c_int;
    pub fn bls_multi_miller_loop_prepared(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_prepared, n: usize, out1: *mut bls_fq12) -> c_int;
    pub fn bls_pairing_projective_batch(ctx: *mut bls_ctx, p: *const bls_g1, q: *const bls_g2, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_pairing_product(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_affine, n: usize, out1: *mut bls_fq12, is_some: *mut u8) -> c_int;
    pub fn bls_mgpu_create(devices: *const c_int, n_devices: c_int, err: *mut c_int) -> *mut bls_mgpu;
    pub fn bls_mgpu_destroy(m: *mut bls_mgpu);
    pub fn bls_mgpu_device_count(m: *const bls_mgpu) -> c_int;
    pub fn bls_mgpu_multi_miller_loop(m: *mut bls_mgpu, p: *const bls_g1_affine, q: *const bls_g2_affine, n: usize, out1: *mut bls_fq12) -> c_int;
    pub fn bls_mgpu_pairing_product(m: *mut bls_mgpu, p: *const bls_g1_affine, q: *const bls_g2_affine, n: usize, out1: *mut bls_fq12, is_some: *mut u8) -> c_int;
    pub fn bls_mgpu_pairing_batch(m: *mut bls_mgpu, p: *const bls_g1_affine, q: *const bls_g2_affine, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_mgpu_g1_wnaf_mul_batch(m: *mut bls_mgpu, bases: *const bls_g1, k: *const bls_fr_repr, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_mgpu_g2_wnaf_mul_batch(m: *mut bls_mgpu, bases: *const bls_g2, k: *const bls_fr_repr, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_final_exponentiation_batch(ctx: *mut bls_ctx, input: *const bls_fq12, out: *mut bls_fq12, is_some: *mut u8, n: usize) -> c_int;
    pub fn bls_pairing_batch(ctx: *mut bls_ctx, p: *const bls_g1_affine, q: *const bls_g2_affine, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_g1_decode_batch(ctx: *mut bls_ctx, bytes: *const u8, compressed: c_int, checked: c_int, out: *mut bls_g1_affine, status: *mut u8, n: usize) -> c_int;
    pub fn bls_g2_decode_batch(ctx: *mut bls_ctx, bytes: *const u8, compressed: c_int, checked: c_int, out: *mut bls_g2_affine, status: *mut u8, n: usize) -> c_int;
    pub fn bls_g1_encode_batch(ctx: *mut bls_ctx, input: *const bls_g1_affine, compressed: c_int, bytes: *mut u8, n: usize) -> c_int;
    pub fn bls_g2_encode_batch(ctx: *mut bls_ctx, input: *const bls_g2_affine, compressed: c_int, bytes: *mut u8, n: usize) -> c_int;
    pub fn bls_g1_affine_mul_batch(ctx: *mut bls_ctx, a: *const bls_g1_affine, k: *const bls_fr_repr, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_affine_mul_batch(ctx: *mut bls_ctx, a: *const bls_g2_affine, k: *const bls_fr_repr, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_point_from_x_batch(ctx: *mut bls_ctx, x: *const bls_fq, greatest: *const u8, out: *mut bls_g1_affine, is_some: *mut u8, n: usize) -> c_int;
    pub fn bls_g2_point_from_x_batch(ctx: *mut bls_ctx, x: *const bls_fq2, greatest: *const u8, out: *mut bls_g2_affine, is_some: *mut u8, n: usize) -> c_int;
    pub fn bls_g1_scale_by_cofactor_batch(ctx: *mut bls_ctx, input: *const bls_g1_affine, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_scale_by_cofactor_batch(ctx: *mut bls_ctx, input: *const bls_g2_affine, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_fr_op_batch(ctx: *mut bls_ctx, op: c_int, a: *const bls_fr_repr, b: *const bls_fr_repr, out: *mut bls_fr_repr, ok: *mut u8, n: usize) -> c_int;
    pub fn bls_fr_fft_batch(ctx: *mut bls_ctx, kind: c_int, input: *const bls_fr_repr, out: *mut bls_fr_repr, log_n: c_int, m: usize) -> c_int;
    pub fn bls_groth16_prove_batch(ctx: *mut bls_ctx, params: *const bls_groth16_params, a: *const bls_fr_repr, b: *const bls_fr_repr, c: *const bls_fr_repr, len: usize,
                                   input: *const bls_fr_repr, num_inputs: usize, aux: *const bls_fr_repr, num_aux: usize, a_aux_density: *const u32,
                                   b_input_density: *const u32, b_aux_density: *const u32, r: *const bls_fr_repr, s: *const bls_fr_repr, m: usize,
                                   out: *mut bls_groth16_proof) -> c_int;
    pub fn bls_groth16_prepare_verifying_key(ctx: *mut bls_ctx, alpha_g1: *const bls_g1_affine, beta_g2: *const bls_g2_affine, gamma_g2: *const bls_g2_affine,
                                             delta_g2: *const bls_g2_affine, out: *mut bls_groth16_pvk) -> c_int;
    pub fn bls_groth16_verify_batch(ctx: *mut bls_ctx, pvk: *const bls_groth16_pvk, ic: *const bls_g1_affine, num_inputs: usize, proofs: *const bls_groth16_proof,
                                    inputs: *const bls_fr_repr, m: usize, ok: *mut u8) -> c_int;
    pub fn bls_groth16_verify_rlc_batch(ctx: *mut bls_ctx, pvk: *const bls_groth16_pvk, ic: *const bls_g1_affine, num_inputs: usize, proofs: *const bls_groth16_proof,
                                        inputs: *const bls_fr_repr, rho: *const bls_fr_repr, m: usize, ok1: *mut u8) -> c_int;
    pub fn bls_groth16_generate_parameters_batch(ctx: *mut bls_ctx, abc: *const bls_r1cs_matrix, num_constraints: usize, num_inputs: usize,
                                                 num_aux: usize, g1: *const bls_g1_affine, g2: *const bls_g2_affine, alpha: *const bls_fr_repr,
                                                 beta: *const bls_fr_repr, gamma: *const bls_fr_repr, delta: *const bls_fr_repr, tau: *const bls_fr_repr,
                                                 out: *const bls_groth16_parameters_out) -> c_int;
    pub fn bls_groth16_mpc_contribute_batch(ctx: *mut bls_ctx, delta: *const bls_fr_repr, s: *const bls_g1_affine, r: *const bls_g2_affine,
                                            vk: *mut bls_groth16_vk_points, h: *const bls_g1_affine, h_len: usize, l: *const bls_g1_affine,
                                            l_len: usize, h_out: *mut bls_g1_affine, l_out: *mut bls_g1_affine,
                                            pubkey: *mut bls_groth16_mpc_pubkey) -> c_int;
    pub fn bls_groth16_mpc_verify_batch(ctx: *mut bls_ctx, before: *const bls_groth16_key, after: *const bls_groth16_key,
                                        pk: *const bls_groth16_mpc_pubkey, k: usize, rho_h: *const bls_fr_repr, rho_l: *const bls_fr_repr,
                                        ok1: *mut u8) -> c_int;
    pub fn bls_groth16_mpc_new_batch(ctx: *mut bls_ctx, abc: *const bls_r1cs_matrix, num_constraints: usize, num_inputs: usize, num_aux: usize,
                                     phase1: *const bls_groth16_phase1, g1: *const bls_g1_affine, g2: *const bls_g2_affine,
                                     out: *const bls_groth16_parameters_out) -> c_int;
    pub fn bls_kzg_commit_batch(ctx: *mut bls_ctx, srs: *const bls_g1_affine, srs_len: usize, p: *const bls_fr_repr, n: usize, m: usize,
                                c: *mut bls_g1_affine) -> c_int;
    pub fn bls_kzg_open_batch(ctx: *mut bls_ctx, srs: *const bls_g1_affine, srs_len: usize, p: *const bls_fr_repr, n: usize, z: *const bls_fr_repr,
                              m: usize, y: *mut bls_fr_repr, proof: *mut bls_g1_affine) -> c_int;
    pub fn bls_kzg_prepare_verifying_key(ctx: *mut bls_ctx, g: *const bls_g1_affine, h: *const bls_g2_affine, tau_h: *const bls_g2_affine,
                                         out: *mut bls_kzg_pvk) -> c_int;
    pub fn bls_kzg_verify_batch(ctx: *mut bls_ctx, pvk: *const bls_kzg_pvk, c: *const bls_g1_affine, y: *const bls_fr_repr, z: *const bls_fr_repr,
                                proof: *const bls_g1_affine, m: usize, ok: *mut u8) -> c_int;
    pub fn bls_kzg_verify_rlc_batch(ctx: *mut bls_ctx, pvk: *const bls_kzg_pvk, c: *const bls_g1_affine, y: *const bls_fr_repr, z: *const bls_fr_repr,
                                    proof: *const bls_g1_affine, rho: *const bls_fr_repr, m: usize, ok1: *mut u8) -> c_int;
    pub fn bls_kzg_open_all_prepare(ctx: *mut bls_ctx, srs: *const bls_g1_affine, srs_len: usize, log_n: c_int, table: *mut bls_g1_affine) -> c_int;
    pub fn bls_kzg_open_all_batch(ctx: *mut bls_ctx, table: *const bls_g1_affine, p: *const bls_fr_repr, log_n: c_int, m: usize, y: *mut bls_fr_repr,
                                  proof: *mut bls_g1_affine) -> c_int;
    pub fn bls_g1_fft_batch(ctx: *mut bls_ctx, kind: c_int, input: *const bls_g1_affine, out: *mut bls_g1_affine, log_n: c_int, m: usize) -> c_int;
    pub fn bls_g2_fft_batch(ctx: *mut bls_ctx, kind: c_int, input: *const bls_g2_affine, out: *mut bls_g2_affine, log_n: c_int, m: usize) -> c_int;
    pub fn bls_fr_groth16_h_batch(ctx: *mut bls_ctx, a: *const bls_fr_repr, b: *const bls_fr_repr, c: *const bls_fr_repr, len: usize, m: usize, h: *mut bls_fr_repr) -> c_int;
    pub fn bls_fq12_pow_batch(ctx: *mut bls_ctx, a: *const bls_fq12, k: *const bls_fr_repr, out: *mut bls_fq12, n: usize) -> c_int;
    pub fn bls_fq12_product(ctx: *mut bls_ctx, input: *const bls_fq12, n: usize, out1: *mut bls_fq12) -> c_int;

    pub fn bls_g1_wnaf_mul_batch(ctx: *mut bls_ctx, bases: *const bls_g1, k: *const bls_fr_repr, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_wnaf_mul_batch(ctx: *mut bls_ctx, bases: *const bls_g2, k: *const bls_fr_repr, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_wnaf_mul_window_batch(ctx: *mut bls_ctx, bases: *const bls_g1, k: *const bls_fr_repr, out: *mut bls_g1, n: usize, window: c_int) -> c_int;
    pub fn bls_g2_wnaf_mul_window_batch(ctx: *mut bls_ctx, bases: *const bls_g2, k: *const bls_fr_repr, out: *mut bls_g2, n: usize, window: c_int) -> c_int;
    pub fn bls_g1_wnaf_fixed_base_batch(ctx: *mut bls_ctx, base: *const bls_g1, window: c_int, k: *const bls_fr_repr, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_wnaf_fixed_base_batch(ctx: *mut bls_ctx, base: *const bls_g2, window: c_int, k: *const bls_fr_repr, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_wnaf_table(ctx: *mut bls_ctx, base: *const bls_g1, window: c_int, table: *mut bls_g1) -> c_int;
    pub fn bls_g2_wnaf_table(ctx: *mut bls_ctx, base: *const bls_g2, window: c_int, table: *mut bls_g2) -> c_int;
    pub fn bls_g1_mul_batch(ctx: *mut bls_ctx, bases: *const bls_g1, k: *const bls_fr_repr, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_mul_batch(ctx: *mut bls_ctx, bases: *const bls_g2, k: *const bls_fr_repr, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_batch_normalization(ctx: *mut bls_ctx, inout: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_batch_normalization(ctx: *mut bls_ctx, inout: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_into_affine_batch(ctx: *mut bls_ctx, input: *const bls_g1, out: *mut bls_g1_affine, n: usize) -> c_int;
    pub fn bls_g2_into_affine_batch(ctx: *mut bls_ctx, input: *const bls_g2, out: *mut bls_g2_affine, n: usize) -> c_int;
    pub fn bls_g1_op_batch(ctx: *mut bls_ctx, op: c_int, a: *const bls_g1, b: *const c_void, out: *mut bls_g1, n: usize) -> c_int;
    pub fn bls_g2_op_batch(ctx: *mut bls_ctx, op: c_int, a: *const bls_g2, b: *const c_void, out: *mut bls_g2, n: usize) -> c_int;
    pub fn bls_g1_msm(ctx: *mut bls_ctx, bases: *const bls_g1_affine, k: *const bls_fr_repr, n: usize, out1: *mut bls_g1) -> c_int;
    pub fn bls_g2_msm(ctx: *mut bls_ctx, bases: *const bls_g2_affine, k: *const bls_fr_repr, n: usize, out1: *mut bls_g2) -> c_int;
    pub fn bls_g1_msm_batch(ctx: *mut bls_ctx, bases: *const bls_g1_affine, shared_bases: c_int, k: *const bls_fr_repr, n: usize, m: usize, out: *mut bls_g1) -> c_int;
    pub fn bls_g2_msm_batch(ctx: *mut bls_ctx, bases: *const bls_g2_affine, shared_bases: c_int, k: *const bls_fr_repr, n: usize, m: usize, out: *mut bls_g2) -> c_int;
}
