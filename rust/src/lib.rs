//! Slice-level GPU entry points next to the `pairing` crate's scalar trait methods.
//!
//! This file lives INSIDE a fork of the crate, as the module `crate::bls12_381::gpu` (`mod gpu;` in
//! src/bls12_381/mod.rs, `ffi.rs` next to it as `gpu/ffi.rs`): the point fields are `pub(crate)`
//! (src/bls12_381/ec.rs:15-17, 33-35), so marshalling needs crate visibility, and the two accessors it
//! uses on `Fq` / `Fr` -- `mont_limbs()` and `from_mont_limbs()`, raw access to the Montgomery limbs --
//! are the two-line patch shown in INTEGRATION.md (the upstream fields are private to fq.rs / fr.rs).
//! Marshalling through the public API instead (`into_repr` / `from_repr`) would cost a Montgomery
//! conversion per coordinate in each direction.  The
//! scalar trait methods (`Engine::pairing`, `CurveProjective::mul_assign`, ...) stay as they are;
//! callers with batches use the functions below.  One `Gpu` = one `bls_ctx`; it is `Send` and is
//! wrapped in a `Mutex` because calls on a context must be serialised.
//!
//! Authored, not compiled here (no Rust toolchain in the build image) -- see INTEGRATION.md.
pub mod ffi;

use self::ffi::*;
use crate::bls12_381::{Fq12, Fr, FrRepr, G1Affine, G2Affine, G1, G2};
use std::os::raw::c_int;
use std::sync::Mutex;

#[derive(Debug)]
pub struct GpuError(pub i32, pub String);

pub struct Gpu { ctx: Mutex<*mut bls_ctx> }
unsafe impl Send for Gpu {}
unsafe impl Sync for Gpu {}

impl Gpu {
    /// One context per CUDA device; there is no CPU fallback (fails without a device).
    pub fn new(device: i32) -> Result<Gpu, GpuError> {
        let mut err = 0;
        let ctx = unsafe { bls_ctx_create(device, &mut err) };
        if ctx.is_null() { return Err(GpuError(err, strerror(err))); }
        Ok(Gpu { ctx: Mutex::new(ctx) })
    }

    /// `Bls12::pairing(p_i, q_i)` for every i (src/lib.rs:101-109).
    pub fn pairing_batch(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Vec<Fq12>, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let mut out = vec![marshal::FQ12_ZERO; p.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_pairing_batch(*ctx, pp.as_ptr(), qq.as_ptr(), out.as_mut_ptr(), p.len()) }, *ctx)?;
        Ok(out.iter().map(marshal::fq12_back).collect())
    }

    /// `Bls12::pairing(p_i, q_i)` with projective arguments (`Into<G1Affine>`, `Into<G2Affine>`): conversions fused in front.
    pub fn pairing_projective_batch(&self, p: &[G1], q: &[G2]) -> Result<Vec<Fq12>, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1> = p.iter().map(marshal::g1).collect();
        let qq: Vec<bls_g2> = q.iter().map(marshal::g2).collect();
        let mut out = vec![marshal::FQ12_ZERO; p.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_pairing_projective_batch(*ctx, pp.as_ptr(), qq.as_ptr(), out.as_mut_ptr(), p.len()) }, *ctx)?;
        Ok(out.iter().map(marshal::fq12_back).collect())
    }

    /// `Bls12::miller_loop(&[(&p_0.prepare(), &q_0.prepare()), ...])`: one shared accumulator (mod.rs:40-102).
    pub fn multi_miller_loop(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Fq12, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let mut out = marshal::FQ12_ZERO;
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_multi_miller_loop(*ctx, pp.as_ptr(), qq.as_ptr(), p.len(), &mut out) }, *ctx)?;
        Ok(marshal::fq12_back(&out))
    }

    /// `Bls12::final_exponentiation(&Bls12::miller_loop(pairs))` in one call: the batch-verification shape.
    pub fn pairing_product(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Option<Fq12>, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let (mut out, mut some) = (marshal::FQ12_ZERO, 0u8);
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_pairing_product(*ctx, pp.as_ptr(), qq.as_ptr(), p.len(), &mut out, &mut some) }, *ctx)?;
        Ok(if some != 0 { Some(marshal::fq12_back(&out)) } else { None })
    }

    /// `Bls12::final_exponentiation` per element; `None` where the input is zero (mod.rs:104-160).
    pub fn final_exponentiation_batch(&self, f: &[Fq12]) -> Result<Vec<Option<Fq12>>, GpuError> {
        let ff: Vec<bls_fq12> = f.iter().map(marshal::fq12).collect();
        let mut out = vec![marshal::FQ12_ZERO; f.len()];
        let mut some = vec![0u8; f.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_final_exponentiation_batch(*ctx, ff.as_ptr(), out.as_mut_ptr(), some.as_mut_ptr(), f.len()) }, *ctx)?;
        Ok(out.iter().zip(some).map(|(v, s)| if s != 0 { Some(marshal::fq12_back(v)) } else { None }).collect())
    }

    /// `Wnaf::new().scalar(k_i).base(g_i)` per element (wnaf.rs:111-128, 158-164); Jacobian outputs are
    /// the reference's exact (X, Y, Z) triples.
    pub fn g1_wnaf_mul_batch(&self, bases: &[G1], k: &[FrRepr]) -> Result<Vec<G1>, GpuError> {
        assert_eq!(bases.len(), k.len());
        let bb: Vec<bls_g1> = bases.iter().map(marshal::g1).collect();
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = bb.clone();
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_wnaf_mul_batch(*ctx, bb.as_ptr(), kk.as_ptr(), out.as_mut_ptr(), bb.len()) }, *ctx)?;
        Ok(out.iter().map(marshal::g1_back).collect())
    }

    /// `G1::batch_normalization(&mut v)` (ec.rs:246-294).
    pub fn g1_batch_normalization(&self, v: &mut [G1]) -> Result<(), GpuError> {
        let mut vv: Vec<bls_g1> = v.iter().map(marshal::g1).collect();
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_batch_normalization(*ctx, vv.as_mut_ptr(), vv.len()) }, *ctx)?;
        for (dst, src) in v.iter_mut().zip(vv.iter()) { *dst = marshal::g1_back(src); }
        Ok(())
    }
    /// `Wnaf::new().base(g, k.len()).scalar(k_i)` for every scalar: one shared window table (wnaf.rs:93-107, 169-178).
    pub fn g1_wnaf_fixed_base(&self, base: &G1, k: &[FrRepr]) -> Result<Vec<G1>, GpuError> {
        use pairing::CurveProjective;
        let window = G1::recommended_wnaf_for_num_scalars(k.len()) as i32;
        let b = marshal::g1(base);
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = vec![b; k.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_wnaf_fixed_base_batch(*ctx, &b, window, kk.as_ptr(), out.as_mut_ptr(), kk.len()) }, *ctx)?;
        Ok(out.iter().map(marshal::g1_back).collect())
    }

    /// `sum_i k_i * bases_i` by the bucket method: the normalised sum (`into_projective(into_affine(S))`, or `G1::zero()`).
    /// Scalars are full 256-bit `FrRepr` integers (not reduced mod r).
    pub fn g1_multiexp(&self, bases: &[G1Affine], k: &[FrRepr]) -> Result<G1, GpuError> {
        assert_eq!(bases.len(), k.len());
        let bb: Vec<bls_g1_affine> = bases.iter().map(marshal::g1_affine).collect();
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = bls_g1 { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, z: marshal::FQ_ZERO };
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_msm(*ctx, bb.as_ptr(), kk.as_ptr(), bb.len(), &mut out) }, *ctx)?;
        Ok(marshal::g1_back(&out))
    }

    /// `m` independent multiexp sums in one call, `m = k.len() / n`: sum `j` is `sum_i k[j*n + i] * bases[b(j, i)]` with
    /// `b(j, i) = i` when `bases.len() == n` (one set of bases for every sum) and `j*n + i` when `bases.len() == k.len()`.
    /// Each result equals `g1_multiexp` of its sum; a loop of `g1_multiexp` calls becomes one call.
    pub fn g1_multiexp_batch(&self, bases: &[G1Affine], k: &[FrRepr], n: usize) -> Result<Vec<G1>, GpuError> {
        assert!(n > 0 && k.len() % n == 0 && (bases.len() == n || bases.len() == k.len()));
        let m = k.len() / n;
        let bb: Vec<bls_g1_affine> = bases.iter().map(marshal::g1_affine).collect();
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = vec![bls_g1 { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, z: marshal::FQ_ZERO }; m];
        let shared = (bases.len() == n) as i32;
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_msm_batch(*ctx, bb.as_ptr(), shared, kk.as_ptr(), n, m, out.as_mut_ptr()) }, *ctx)?;
        Ok(out.iter().map(marshal::g1_back).collect())
    }

    /// bellman's `EvaluationDomain` transforms over `Fr` for `a.len() / 2^log_n` polynomials back to back, natural order:
    /// kind 0 `fft`, 1 `ifft`, 2 `coset_fft`, 3 `icoset_fft` (`BLS_FFT` ... in the C header).
    pub fn fr_fft(&self, kind: i32, a: &[Fr], log_n: u32) -> Result<Vec<Fr>, GpuError> {
        assert!(log_n <= 28 && a.len() % (1usize << log_n) == 0);
        let aa: Vec<bls_fr_repr> = a.iter().map(marshal::fr).collect();
        let mut out = vec![bls_fr_repr { l: [0; 4] }; a.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_fr_fft_batch(*ctx, kind, aa.as_ptr(), out.as_mut_ptr(), log_n as i32, a.len() >> log_n) }, *ctx)?;
        Ok(out.iter().map(marshal::fr_back).collect())
    }

    /// Groth16's quotient polynomial for `m` proofs, the `h` block of bellman's `create_proof`: `a`, `b`, `c` are the
    /// `ProvingAssignment` evaluations of the proofs back to back (`len = a.len() / m` each).  Returns `m * (n - 1)`
    /// canonical `FrRepr` coefficients, `n` the smallest power of two `>= len`: the scalars of `g1_multiexp_batch` against
    /// the `n - 1` bases of the proving key's `h` query.
    pub fn groth16_h(&self, a: &[Fr], b: &[Fr], c: &[Fr], m: usize) -> Result<Vec<FrRepr>, GpuError> {
        assert!(m > 0 && a.len() % m == 0 && b.len() == a.len() && c.len() == a.len());
        let len = a.len() / m;
        let n = len.max(1).next_power_of_two();
        let (aa, bb, cc): (Vec<bls_fr_repr>, Vec<bls_fr_repr>, Vec<bls_fr_repr>) =
            (a.iter().map(marshal::fr).collect(), b.iter().map(marshal::fr).collect(), c.iter().map(marshal::fr).collect());
        let mut h = vec![bls_fr_repr { l: [0; 4] }; m * (n - 1)];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_fr_groth16_h_batch(*ctx, aa.as_ptr(), bb.as_ptr(), cc.as_ptr(), len, m, h.as_mut_ptr()) }, *ctx)?;
        Ok(h.iter().map(|r| FrRepr(r.l)).collect())
    }

    /// bellman's `groth16::create_proof` for `m` proofs of one circuit, after synthesis: `a`, `b`, `c` are the proofs'
    /// `ProvingAssignment` vectors back to back (`len = a.len() / m` each, input constraints included), `inputs` and `aux`
    /// their `input_assignment` / `aux_assignment`, `densities` the words of the circuit's three `DensityTracker::bv`
    /// (`a_aux`, `b_input`, `b_aux`: `BitVec<u32>` storage, shared by the proofs), `r` and `s` the blinding values.
    /// Returns `Proof { a, b, c }` of every proof as `(A, B, C)`, bit-exact with bellman.
    pub fn groth16_create_proof_batch(&self, params: &Groth16Params, a: &[Fr], b: &[Fr], c: &[Fr], inputs: &[Fr], aux: &[Fr],
                                      densities: [&[u32]; 3], r: &[Fr], s: &[Fr], m: usize)
                                      -> Result<Vec<(G1Affine, G2Affine, G1Affine)>, GpuError> {
        assert!(m > 0 && a.len() % m == 0 && inputs.len() % m == 0 && aux.len() % m == 0 && b.len() == a.len() && c.len() == a.len());
        assert!(r.len() == m && s.len() == m && params.b_g1.len() == params.b_g2.len());
        let (len, ni, na) = (a.len() / m, inputs.len() / m, aux.len() / m);
        let fr = |v: &[Fr]| -> Vec<bls_fr_repr> { v.iter().map(marshal::fr).collect() };
        let (aa, bb, cc, ii, xx, rr, ss) = (fr(a), fr(b), fr(c), fr(inputs), fr(aux), fr(r), fr(s));
        let g1s = |v: &[G1Affine]| -> Vec<bls_g1_affine> { v.iter().map(marshal::g1_affine).collect() };
        let (h, l, qa, b1) = (g1s(&params.h), g1s(&params.l), g1s(&params.a), g1s(&params.b_g1));
        let b2: Vec<bls_g2_affine> = params.b_g2.iter().map(marshal::g2_affine).collect();
        let p = bls_groth16_params {
            alpha_g1: marshal::g1_affine(&params.alpha_g1), beta_g1: marshal::g1_affine(&params.beta_g1),
            delta_g1: marshal::g1_affine(&params.delta_g1), beta_g2: marshal::g2_affine(&params.beta_g2),
            delta_g2: marshal::g2_affine(&params.delta_g2),
            h: h.as_ptr(), l: l.as_ptr(), a: qa.as_ptr(), b_g1: b1.as_ptr(), b_g2: b2.as_ptr(),
            h_len: h.len(), l_len: l.len(), a_len: qa.len(), b_len: b1.len(),
        };
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let zero2 = bls_g2_affine { x: bls_fq2 { c0: marshal::FQ_ZERO, c1: marshal::FQ_ZERO }, y: bls_fq2 { c0: marshal::FQ_ZERO, c1: marshal::FQ_ZERO }, infinity: 1 };
        let mut out = vec![bls_groth16_proof { a: zero1, b: zero2, c: zero1 }; m];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe {
            bls_groth16_prove_batch(*ctx, &p, aa.as_ptr(), bb.as_ptr(), cc.as_ptr(), len, ii.as_ptr(), ni, xx.as_ptr(), na, densities[0].as_ptr(),
                                    densities[1].as_ptr(), densities[2].as_ptr(), rr.as_ptr(), ss.as_ptr(), m, out.as_mut_ptr())
        }, *ctx)?;
        Ok(out.iter().map(|p| (marshal::g1_affine_back(&p.a), marshal::g2_affine_back(&p.b), marshal::g1_affine_back(&p.c))).collect())
    }

    /// bellman's `groth16::prepare_verifying_key` without `ic` (the caller keeps it): e(alpha_g1, beta_g2) and the prepared
    /// -gamma_g2, -delta_g2, bit-exact with bellman.  Boxed: the struct is 40 176 bytes.
    pub fn groth16_prepare_verifying_key(&self, alpha_g1: &G1Affine, beta_g2: &G2Affine, gamma_g2: &G2Affine, delta_g2: &G2Affine)
                                         -> Result<Box<bls_groth16_pvk>, GpuError> {
        let (a, b, g, d) = (marshal::g1_affine(alpha_g1), marshal::g2_affine(beta_g2), marshal::g2_affine(gamma_g2), marshal::g2_affine(delta_g2));
        let mut out: Box<bls_groth16_pvk> = Box::new(unsafe { std::mem::zeroed() });
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_groth16_prepare_verifying_key(*ctx, &a, &b, &g, &d, &mut *out) }, *ctx)?;
        Ok(out)
    }

    /// bellman's `groth16::verify_proof` for every proof: `ic` is the vk's `ic` (num_inputs + 1 points), `inputs` the proofs'
    /// public inputs back to back (num_inputs each, without the leading one).  `true` where the proof verifies.
    pub fn groth16_verify_proof_batch(&self, pvk: &bls_groth16_pvk, ic: &[G1Affine], proofs: &[(G1Affine, G2Affine, G1Affine)], inputs: &[Fr])
                                      -> Result<Vec<bool>, GpuError> {
        assert!(!ic.is_empty() && inputs.len() == proofs.len() * (ic.len() - 1));
        let icc: Vec<bls_g1_affine> = ic.iter().map(marshal::g1_affine).collect();
        let pr: Vec<bls_groth16_proof> = proofs.iter().map(|(a, b, c)| bls_groth16_proof { a: marshal::g1_affine(a), b: marshal::g2_affine(b), c: marshal::g1_affine(c) }).collect();
        let xs: Vec<bls_fr_repr> = inputs.iter().map(marshal::fr).collect();
        let mut ok = vec![0u8; proofs.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_groth16_verify_batch(*ctx, pvk, icc.as_ptr(), ic.len() - 1, pr.as_ptr(), xs.as_ptr(), proofs.len(), ok.as_mut_ptr()) }, *ctx)?;
        Ok(ok.iter().map(|&b| b != 0).collect())
    }

    /// bellperson's `verify_proofs_batch` with the caller's randomizers `rho` (one per proof; 0 leaves a proof out): one verdict.
    pub fn groth16_verify_proofs_batch(&self, pvk: &bls_groth16_pvk, ic: &[G1Affine], proofs: &[(G1Affine, G2Affine, G1Affine)], inputs: &[Fr],
                                       rho: &[FrRepr]) -> Result<bool, GpuError> {
        assert!(!ic.is_empty() && inputs.len() == proofs.len() * (ic.len() - 1) && rho.len() == proofs.len());
        let icc: Vec<bls_g1_affine> = ic.iter().map(marshal::g1_affine).collect();
        let pr: Vec<bls_groth16_proof> = proofs.iter().map(|(a, b, c)| bls_groth16_proof { a: marshal::g1_affine(a), b: marshal::g2_affine(b), c: marshal::g1_affine(c) }).collect();
        let xs: Vec<bls_fr_repr> = inputs.iter().map(marshal::fr).collect();
        let rs: Vec<bls_fr_repr> = rho.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut ok = 0u8;
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_groth16_verify_rlc_batch(*ctx, pvk, icc.as_ptr(), ic.len() - 1, pr.as_ptr(), xs.as_ptr(), rs.as_ptr(), proofs.len(), &mut ok) }, *ctx)?;
        Ok(ok != 0)
    }

    /// KZG commitments `c[j] = sum_i p[j n + i] srs[i]` for `p.len() / n` polynomials of `n` coefficients (`srs[i] = [tau^i] g`).
    pub fn kzg_commit(&self, srs: &[G1Affine], p: &[Fr], n: usize) -> Result<Vec<G1Affine>, GpuError> {
        assert!(n > 0 && p.len() % n == 0);
        let s: Vec<bls_g1_affine> = srs.iter().map(marshal::g1_affine).collect();
        let pp: Vec<bls_fr_repr> = p.iter().map(marshal::fr).collect();
        let m = p.len() / n;
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let mut c = vec![zero1; m];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_commit_batch(*ctx, s.as_ptr(), s.len(), pp.as_ptr(), n, m, c.as_mut_ptr()) }, *ctx)?;
        Ok(c.iter().map(marshal::g1_affine_back).collect())
    }

    /// KZG openings: polynomial j (`n` coefficients) at `z[j]` -> (`p_j(z_j)`, `[q_j(tau)] g`), q_j = (p_j - p_j(z_j)) / (X - z_j).
    pub fn kzg_open(&self, srs: &[G1Affine], p: &[Fr], n: usize, z: &[Fr]) -> Result<Vec<(Fr, G1Affine)>, GpuError> {
        assert!(p.len() == n * z.len());
        let s: Vec<bls_g1_affine> = srs.iter().map(marshal::g1_affine).collect();
        let pp: Vec<bls_fr_repr> = p.iter().map(marshal::fr).collect();
        let zz: Vec<bls_fr_repr> = z.iter().map(marshal::fr).collect();
        let m = z.len();
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let mut y = vec![bls_fr_repr { l: [0; 4] }; m];
        let mut proof = vec![zero1; m];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_open_batch(*ctx, s.as_ptr(), s.len(), pp.as_ptr(), n, zz.as_ptr(), m, y.as_mut_ptr(), proof.as_mut_ptr()) }, *ctx)?;
        Ok(y.iter().zip(proof.iter()).map(|(y, w)| (marshal::fr_back(y), marshal::g1_affine_back(w))).collect())
    }

    /// The KZG verifying key from `g`, `h` and `[tau] h`.  Boxed: the struct is 39 704 bytes.
    pub fn kzg_prepare_verifying_key(&self, g: &G1Affine, h: &G2Affine, tau_h: &G2Affine) -> Result<Box<bls_kzg_pvk>, GpuError> {
        let (a, b, t) = (marshal::g1_affine(g), marshal::g2_affine(h), marshal::g2_affine(tau_h));
        let mut out: Box<bls_kzg_pvk> = Box::new(unsafe { std::mem::zeroed() });
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_prepare_verifying_key(*ctx, &a, &b, &t, &mut *out) }, *ctx)?;
        Ok(out)
    }

    /// `e(C_j - y_j g, h) == e(proof_j, tau h - z_j h)` for every opening `(C_j, z_j, y_j, proof_j)`.
    pub fn kzg_verify(&self, pvk: &bls_kzg_pvk, openings: &[(G1Affine, Fr, Fr, G1Affine)]) -> Result<Vec<bool>, GpuError> {
        let c: Vec<bls_g1_affine> = openings.iter().map(|o| marshal::g1_affine(&o.0)).collect();
        let z: Vec<bls_fr_repr> = openings.iter().map(|o| marshal::fr(&o.1)).collect();
        let y: Vec<bls_fr_repr> = openings.iter().map(|o| marshal::fr(&o.2)).collect();
        let w: Vec<bls_g1_affine> = openings.iter().map(|o| marshal::g1_affine(&o.3)).collect();
        let mut ok = vec![0u8; openings.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_verify_batch(*ctx, pvk, c.as_ptr(), y.as_ptr(), z.as_ptr(), w.as_ptr(), openings.len(), ok.as_mut_ptr()) }, *ctx)?;
        Ok(ok.iter().map(|&b| b != 0).collect())
    }

    /// The randomized check of `kzg_verify`'s openings with the caller's randomizers `rho` (one per opening; 0 leaves one out).
    pub fn kzg_verify_batch(&self, pvk: &bls_kzg_pvk, openings: &[(G1Affine, Fr, Fr, G1Affine)], rho: &[FrRepr]) -> Result<bool, GpuError> {
        assert!(rho.len() == openings.len());
        let c: Vec<bls_g1_affine> = openings.iter().map(|o| marshal::g1_affine(&o.0)).collect();
        let z: Vec<bls_fr_repr> = openings.iter().map(|o| marshal::fr(&o.1)).collect();
        let y: Vec<bls_fr_repr> = openings.iter().map(|o| marshal::fr(&o.2)).collect();
        let w: Vec<bls_g1_affine> = openings.iter().map(|o| marshal::g1_affine(&o.3)).collect();
        let rs: Vec<bls_fr_repr> = rho.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut ok = 0u8;
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_verify_rlc_batch(*ctx, pvk, c.as_ptr(), y.as_ptr(), z.as_ptr(), w.as_ptr(), rs.as_ptr(), openings.len(), &mut ok) }, *ctx)?;
        Ok(ok != 0)
    }

    /// The FK20 table (2n rows) of `srs` for the domain of `n = 2^log_n`, for `kzg_open_all`.
    pub fn kzg_open_all_prepare(&self, srs: &[G1Affine], log_n: u32) -> Result<Vec<G1Affine>, GpuError> {
        let s: Vec<bls_g1_affine> = srs.iter().map(marshal::g1_affine).collect();
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let mut table = vec![zero1; 2usize << log_n];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_open_all_prepare(*ctx, s.as_ptr(), s.len(), log_n as i32, table.as_mut_ptr()) }, *ctx)?;
        Ok(table.iter().map(marshal::g1_affine_back).collect())
    }

    /// KZG openings of every polynomial of `p` (`p.len() / n` rows of `n = 2^log_n` coefficients) at every `omega^k`:
    /// entry `j n + k` is (`p_j(omega^k)`, the proof `kzg_open` returns for `z = omega^k`).
    pub fn kzg_open_all(&self, table: &[G1Affine], p: &[Fr], log_n: u32) -> Result<Vec<(Fr, G1Affine)>, GpuError> {
        let n = 1usize << log_n;
        assert!(table.len() == 2 * n && p.len() % n == 0);
        let t: Vec<bls_g1_affine> = table.iter().map(marshal::g1_affine).collect();
        let pp: Vec<bls_fr_repr> = p.iter().map(marshal::fr).collect();
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let mut y = vec![bls_fr_repr { l: [0; 4] }; p.len()];
        let mut proof = vec![zero1; p.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_kzg_open_all_batch(*ctx, t.as_ptr(), pp.as_ptr(), log_n as i32, p.len() / n, y.as_mut_ptr(), proof.as_mut_ptr()) }, *ctx)?;
        Ok(y.iter().zip(proof.iter()).map(|(y, w)| (marshal::fr_back(y), marshal::g1_affine_back(w))).collect())
    }

    /// bellman's `EvaluationDomain<Point<G1>>` transforms (`kind`: 0 fft, 1 ifft, 2 coset_fft, 3 icoset_fft) of the
    /// `a.len() / 2^log_n` rows of `a`; `ifft` of `[tau^i] g` is the Lagrange basis `[L_i(tau)] g`.
    pub fn g1_fft(&self, kind: i32, a: &[G1Affine], log_n: u32) -> Result<Vec<G1Affine>, GpuError> {
        assert!(a.len() % (1usize << log_n) == 0);
        let x: Vec<bls_g1_affine> = a.iter().map(marshal::g1_affine).collect();
        let mut out = x.clone();
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_fft_batch(*ctx, kind as i32, x.as_ptr(), out.as_mut_ptr(), log_n as i32, a.len() >> log_n) }, *ctx)?;
        Ok(out.iter().map(marshal::g1_affine_back).collect())
    }

    /// `g1_fft` over G2.
    pub fn g2_fft(&self, kind: i32, a: &[G2Affine], log_n: u32) -> Result<Vec<G2Affine>, GpuError> {
        assert!(a.len() % (1usize << log_n) == 0);
        let x: Vec<bls_g2_affine> = a.iter().map(marshal::g2_affine).collect();
        let mut out = x.clone();
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g2_fft_batch(*ctx, kind as i32, x.as_ptr(), out.as_mut_ptr(), log_n as i32, a.len() >> log_n) }, *ctx)?;
        Ok(out.iter().map(marshal::g2_affine_back).collect())
    }

    /// bellman's `groth16::generate_parameters(circuit, g1, g2, alpha, beta, gamma, delta, tau)` from the circuit's three
    /// matrices as `KeypairAssembly` records them, flattened variable-major (see INTEGRATION.md): `abc[k] = (offsets, constraint,
    /// coeff)` with `offsets` of `num_inputs + num_aux + 1` entries.  `num_constraints` counts the input constraints the generator
    /// appends.  Returns the parameters with their queries trimmed to `a_len` / `b_len`, `gamma_g2`, `ic` and the three density
    /// bitmaps (`a_aux`, `b_input`, `b_aux` words, as `groth16_create_proof_batch` takes them); `Err` on bellman's
    /// `UnconstrainedVariable`, reported as `BLS_ERR_INVALID_ARGUMENT`.
    pub fn groth16_generate_parameters(&self, abc: [(&[u64], &[u32], &[Fr]); 3], num_constraints: usize, num_inputs: usize, num_aux: usize,
                                       g1: &G1Affine, g2: &G2Affine, alpha: &Fr, beta: &Fr, gamma: &Fr, delta: &Fr, tau: &Fr)
                                       -> Result<(Groth16Params, G2Affine, Vec<G1Affine>, [Vec<u32>; 3]), GpuError> {
        let (gg1, gg2) = (marshal::g1_affine(g1), marshal::g2_affine(g2));
        let sc: Vec<bls_fr_repr> = [alpha, beta, gamma, delta, tau].iter().map(|x| marshal::fr(x)).collect();
        self.groth16_key(abc, num_constraints, num_inputs, num_aux, "UnconstrainedVariable: an l query point is the identity", |ctx, mats, out| unsafe {
            bls_groth16_generate_parameters_batch(ctx, mats, num_constraints, num_inputs, num_aux, &gg1, &gg2, &sc[0], &sc[1], &sc[2], &sc[3], &sc[4], out)
        })
    }

    /// phase2's `MPCParameters::new` (include/pairing_b200_mpc.h): the circuit's key from powersoftau's `prepare_phase2` rows
    /// for the domain of `num_constraints` (`coeffs_g1`, `alpha_coeffs_g1`, `beta_coeffs_g1`, `coeffs_g2` of n rows, `h` of
    /// n - 1), before any contribution: gamma_g2 = delta_g2 = g2, delta_g1 = g1.  Same matrices and result as
    /// `groth16_generate_parameters`; `Err` on `UnconstrainedVariable` or on a transcript whose b_g1 and b_g2 disagree on the identity.
    pub fn groth16_mpc_new(&self, abc: [(&[u64], &[u32], &[Fr]); 3], num_constraints: usize, num_inputs: usize, num_aux: usize,
                           alpha_g1: &G1Affine, beta_g1: &G1Affine, beta_g2: &G2Affine, coeffs_g1: &[G1Affine], alpha_coeffs_g1: &[G1Affine],
                           beta_coeffs_g1: &[G1Affine], coeffs_g2: &[G2Affine], h: &[G1Affine], g1: &G1Affine, g2: &G2Affine)
                           -> Result<(Groth16Params, G2Affine, Vec<G1Affine>, [Vec<u32>; 3]), GpuError> {
        let n = coeffs_g1.len();
        if alpha_coeffs_g1.len() != n || beta_coeffs_g1.len() != n || coeffs_g2.len() != n || h.len() + 1 != n {
            return Err(GpuError(BLS_ERR_INVALID_ARGUMENT, "groth16_mpc_new: n rows per coefficient set and n - 1 h rows".to_string()));
        }
        let r1 = |v: &[G1Affine]| -> Vec<bls_g1_affine> { v.iter().map(marshal::g1_affine).collect() };
        let (c1, a1, b1, hh) = (r1(coeffs_g1), r1(alpha_coeffs_g1), r1(beta_coeffs_g1), r1(h));
        let c2: Vec<bls_g2_affine> = coeffs_g2.iter().map(marshal::g2_affine).collect();
        let ph = bls_groth16_phase1 {
            alpha_g1: marshal::g1_affine(alpha_g1), beta_g1: marshal::g1_affine(beta_g1), beta_g2: marshal::g2_affine(beta_g2),
            coeffs_g1: c1.as_ptr(), alpha_coeffs_g1: a1.as_ptr(), beta_coeffs_g1: b1.as_ptr(), coeffs_g2: c2.as_ptr(), h: hh.as_ptr(), n,
        };
        let (gg1, gg2) = (marshal::g1_affine(g1), marshal::g2_affine(g2));
        self.groth16_key(abc, num_constraints, num_inputs, num_aux,
                         "UnconstrainedVariable or an inconsistent transcript: an l query point is the identity, or b_g1 and b_g2 disagree",
                         |ctx, mats, out| unsafe { bls_groth16_mpc_new_batch(ctx, mats, num_constraints, num_inputs, num_aux, &ph, &gg1, &gg2, out) })
    }

    /// phase2's `MPCParameters::contribute` (include/pairing_b200_mpc.h) for the caller's secret `delta`, `s` and `r =
    /// hash_to_g2(transcript)`: `h` and `l` are multiplied by delta^-1 and `delta_g1`, `delta_g2` by delta, in place.  The
    /// caller computes `s_delta = s * delta` first (it goes into the transcript r is derived from).  Returns phase2's public key.
    pub fn groth16_mpc_contribute(&self, params: &mut Groth16Params, delta: &Fr, s: &G1Affine, r: &G2Affine)
                                  -> Result<bls_groth16_mpc_pubkey, GpuError> {
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let zero2 = bls_g2_affine { x: marshal::FQ2_ZERO, y: marshal::FQ2_ZERO, infinity: 1 };
        let mut vk = bls_groth16_vk_points {
            alpha_g1: marshal::g1_affine(&params.alpha_g1), beta_g1: marshal::g1_affine(&params.beta_g1), delta_g1: marshal::g1_affine(&params.delta_g1),
            beta_g2: marshal::g2_affine(&params.beta_g2), gamma_g2: zero2, delta_g2: marshal::g2_affine(&params.delta_g2),
        };
        let mut h: Vec<bls_g1_affine> = params.h.iter().map(marshal::g1_affine).collect();
        let mut l: Vec<bls_g1_affine> = params.l.iter().map(marshal::g1_affine).collect();
        let mut pk = bls_groth16_mpc_pubkey { delta_after: zero1, s: zero1, s_delta: zero1, r: zero2, r_delta: zero2 };
        let (dd, ss, rr) = (marshal::fr(delta), marshal::g1_affine(s), marshal::g2_affine(r));
        let ctx = self.ctx.lock().unwrap();
        check(unsafe {
            bls_groth16_mpc_contribute_batch(*ctx, &dd, &ss, &rr, &mut vk, h.as_ptr(), h.len(), l.as_ptr(), l.len(), h.as_mut_ptr(), l.as_mut_ptr(), &mut pk)
        }, *ctx)?;
        params.h = h.iter().map(marshal::g1_affine_back).collect();
        params.l = l.iter().map(marshal::g1_affine_back).collect();
        params.delta_g1 = marshal::g1_affine_back(&vk.delta_g1);
        params.delta_g2 = marshal::g2_affine_back(&vk.delta_g2);
        Ok(pk)
    }

    /// phase2's `MPCParameters::verify`: `before` is the key of `groth16_mpc_new` and `after` the contributed key, each with
    /// its `gamma_g2` and `ic`; `pks` the contributions' public keys in order; `rho_h`, `rho_l` the caller's randomizers of
    /// the merged pairs (one per h and l row).  The transcript hash checks stay with the caller.
    pub fn groth16_mpc_verify(&self, before: (&Groth16Params, &G2Affine, &[G1Affine]), after: (&Groth16Params, &G2Affine, &[G1Affine]),
                              pks: &[bls_groth16_mpc_pubkey], rho_h: &[FrRepr], rho_l: &[FrRepr]) -> Result<bool, GpuError> {
        let g1v = |v: &[G1Affine]| -> Vec<bls_g1_affine> { v.iter().map(marshal::g1_affine).collect() };
        let rows = |k: &(&Groth16Params, &G2Affine, &[G1Affine])| {
            (g1v(k.2), g1v(&k.0.h), g1v(&k.0.l), g1v(&k.0.a), g1v(&k.0.b_g1), k.0.b_g2.iter().map(marshal::g2_affine).collect::<Vec<bls_g2_affine>>())
        };
        let key = |k: &(&Groth16Params, &G2Affine, &[G1Affine]), r: &(Vec<bls_g1_affine>, Vec<bls_g1_affine>, Vec<bls_g1_affine>, Vec<bls_g1_affine>,
                                                                    Vec<bls_g1_affine>, Vec<bls_g2_affine>)| bls_groth16_key {
            vk: bls_groth16_vk_points {
                alpha_g1: marshal::g1_affine(&k.0.alpha_g1), beta_g1: marshal::g1_affine(&k.0.beta_g1), delta_g1: marshal::g1_affine(&k.0.delta_g1),
                beta_g2: marshal::g2_affine(&k.0.beta_g2), gamma_g2: marshal::g2_affine(k.1), delta_g2: marshal::g2_affine(&k.0.delta_g2),
            },
            ic: r.0.as_ptr(), h: r.1.as_ptr(), l: r.2.as_ptr(), a: r.3.as_ptr(), b_g1: r.4.as_ptr(), b_g2: r.5.as_ptr(),
            ic_len: r.0.len(), h_len: r.1.len(), l_len: r.2.len(), a_len: r.3.len(), b_len: r.4.len(),
        };
        if rho_h.len() != before.0.h.len() || rho_l.len() != before.0.l.len() || before.0.b_g1.len() != before.0.b_g2.len()
            || after.0.b_g1.len() != after.0.b_g2.len() {
            return Err(GpuError(BLS_ERR_INVALID_ARGUMENT, "groth16_mpc_verify: one randomizer per h and l row, and b_g1 as long as b_g2".to_string()));
        }
        let (rb, ra) = (rows(&before), rows(&after));
        let (kb, ka) = (key(&before, &rb), key(&after, &ra));
        let rh: Vec<bls_fr_repr> = rho_h.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let rl: Vec<bls_fr_repr> = rho_l.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut ok = 0u8;
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_groth16_mpc_verify_batch(*ctx, &kb, &ka, pks.as_ptr(), pks.len(), rh.as_ptr(), rl.as_ptr(), &mut ok) }, *ctx)?;
        Ok(ok != 0)
    }

    fn groth16_key<F>(&self, abc: [(&[u64], &[u32], &[Fr]); 3], num_constraints: usize, num_inputs: usize, num_aux: usize, not_ok: &str, call: F)
                      -> Result<(Groth16Params, G2Affine, Vec<G1Affine>, [Vec<u32>; 3]), GpuError>
    where F: FnOnce(*mut bls_ctx, *const bls_r1cs_matrix, *const bls_groth16_parameters_out) -> c_int {
        let nv = num_inputs + num_aux;
        let coeffs: Vec<Vec<bls_fr_repr>> = abc.iter().map(|m| m.2.iter().map(marshal::fr).collect()).collect();
        let mats: Vec<bls_r1cs_matrix> = abc.iter().zip(coeffs.iter()).map(|(m, c)| {
            assert!(m.0.len() == nv + 1 && m.1.len() == c.len());
            bls_r1cs_matrix { offsets: m.0.as_ptr(), constraint: m.1.as_ptr(), coeff: c.as_ptr(), nnz: c.len() }
        }).collect();
        let n = num_constraints.max(1).next_power_of_two();
        let zero1 = bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 1 };
        let zero2 = bls_g2_affine { x: marshal::FQ2_ZERO, y: marshal::FQ2_ZERO, infinity: 1 };
        let mut vk = bls_groth16_vk_points { alpha_g1: zero1, beta_g1: zero1, delta_g1: zero1, beta_g2: zero2, gamma_g2: zero2, delta_g2: zero2 };
        let (mut ic, mut h, mut l) = (vec![zero1; num_inputs], vec![zero1; n - 1], vec![zero1; num_aux]);
        let (mut a, mut b1, mut b2) = (vec![zero1; nv], vec![zero1; nv], vec![zero2; nv]);
        let mut dens = [vec![0u32; (num_aux + 31) / 32], vec![0u32; (num_inputs + 31) / 32], vec![0u32; (num_aux + 31) / 32]];
        let (mut lens, mut ok) = ([0u64; 2], 0u8);
        let out = bls_groth16_parameters_out {
            vk: &mut vk, ic: ic.as_mut_ptr(), h: h.as_mut_ptr(), l: l.as_mut_ptr(), a: a.as_mut_ptr(), b_g1: b1.as_mut_ptr(), b_g2: b2.as_mut_ptr(),
            a_aux_density: dens[0].as_mut_ptr(), b_input_density: dens[1].as_mut_ptr(), b_aux_density: dens[2].as_mut_ptr(),
            lens: lens.as_mut_ptr(), ok: &mut ok,
        };
        let ctx = self.ctx.lock().unwrap();
        check(call(*ctx, mats.as_ptr(), &out as *const bls_groth16_parameters_out), *ctx)?;
        if ok == 0 {
            return Err(GpuError(-1, not_ok.to_string()));
        }
        let g1v = |v: &[bls_g1_affine]| -> Vec<G1Affine> { v.iter().map(marshal::g1_affine_back).collect() };
        let params = Groth16Params {
            alpha_g1: marshal::g1_affine_back(&vk.alpha_g1), beta_g1: marshal::g1_affine_back(&vk.beta_g1),
            delta_g1: marshal::g1_affine_back(&vk.delta_g1), beta_g2: marshal::g2_affine_back(&vk.beta_g2),
            delta_g2: marshal::g2_affine_back(&vk.delta_g2),
            h: g1v(&h), l: g1v(&l), a: g1v(&a[..lens[0] as usize]), b_g1: g1v(&b1[..lens[1] as usize]),
            b_g2: b2[..lens[1] as usize].iter().map(marshal::g2_affine_back).collect(),
        };
        Ok((params, marshal::g2_affine_back(&vk.gamma_g2), g1v(&ic), dens))
    }

    /// `let q = Q.prepare(); ps.iter().map(|p| Bls12::pairing(p, Q))` with the one `G2Prepared` staged on the device.
    pub fn pairing_shared_q(&self, p: &[G1Affine], q: &G2Affine) -> Result<Vec<Fq12>, GpuError> {
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq = marshal::g2_affine(q);
        let mut prepared: Box<bls_g2_prepared> = Box::new(unsafe { std::mem::zeroed() });
        let mut out = vec![marshal::FQ12_ZERO; p.len()];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g2_prepare_batch(*ctx, &qq, &mut *prepared, 1) }, *ctx)?;
        check(unsafe { bls_pairing_shared_q_batch(*ctx, pp.as_ptr(), &*prepared, out.as_mut_ptr(), pp.len()) }, *ctx)?;
        Ok(out.iter().map(marshal::fq12_back).collect())
    }

    /// `G1Compressed::into_affine` for every 48-byte encoding: `Err(code)` carries the reference's `GroupDecodingError`
    /// as the status byte of include/pairing_b200.h (BLS_DEC_*).
    pub fn g1_decode_compressed(&self, bytes: &[u8]) -> Result<Vec<Result<G1Affine, u8>>, GpuError> {
        assert_eq!(bytes.len() % 48, 0);
        let n = bytes.len() / 48;
        let mut out = vec![bls_g1_affine { x: marshal::FQ_ZERO, y: marshal::FQ_ZERO, infinity: 0 }; n];
        let mut status = vec![0u8; n];
        let ctx = self.ctx.lock().unwrap();
        check(unsafe { bls_g1_decode_batch(*ctx, bytes.as_ptr(), 1, 1, out.as_mut_ptr(), status.as_mut_ptr(), n) }, *ctx)?;
        Ok(out.iter().zip(status).map(|(a, s)| if s == 0 { Ok(marshal::g1_affine_back(a)) } else { Err(s) }).collect())
    }
    // g2_wnaf_mul_batch, g2_batch_normalization, g2_prepare_batch, miller_loop_batch, g2_multiexp, the other encodings: same pattern.
}

impl Drop for Gpu {
    fn drop(&mut self) { unsafe { bls_ctx_destroy(*self.ctx.lock().unwrap()) } }
}

fn strerror(e: i32) -> String {
    unsafe { std::ffi::CStr::from_ptr(bls_strerror(e)).to_string_lossy().into_owned() }
}
fn check(rc: i32, ctx: *mut bls_ctx) -> Result<(), GpuError> {
    if rc == BLS_OK { return Ok(()); }
    let detail = unsafe { std::ffi::CStr::from_ptr(bls_ctx_last_error(ctx)).to_string_lossy().into_owned() };
    Err(GpuError(rc, format!("{} [{}]", strerror(rc), detail)))
}

/// Explicit field-by-field copies between the crate's types and the `#[repr(C)]` mirrors.  `Fq` is
/// `Fq(FqRepr([u64; 6]))` in Montgomery form (fq.rs:699-700), which is exactly `bls_fq`.
/// The part of bellman's `groth16::Parameters` that `create_proof` reads: the verifying key's alpha_g1, beta_g1, delta_g1,
/// beta_g2, delta_g2 and the `h`, `l`, `a`, `b_g1`, `b_g2` queries.
pub struct Groth16Params {
    pub alpha_g1: G1Affine, pub beta_g1: G1Affine, pub delta_g1: G1Affine, pub beta_g2: G2Affine, pub delta_g2: G2Affine,
    pub h: Vec<G1Affine>, pub l: Vec<G1Affine>, pub a: Vec<G1Affine>, pub b_g1: Vec<G1Affine>, pub b_g2: Vec<G2Affine>,
}

mod marshal {
    use super::ffi::*;
    use pairing::bls12_381::*;
    pub const FQ_ZERO: bls_fq = bls_fq { l: [0; 6] };
    pub const FQ2_ZERO: bls_fq2 = bls_fq2 { c0: FQ_ZERO, c1: FQ_ZERO };
    pub const FQ6_ZERO: bls_fq6 = bls_fq6 { c0: FQ2_ZERO, c1: FQ2_ZERO, c2: FQ2_ZERO };
    pub const FQ12_ZERO: bls_fq12 = bls_fq12 { c0: FQ6_ZERO, c1: FQ6_ZERO };
    // In the fork these use the crate-private accessors `Fq::mont_limbs()` / `Fq::from_mont_limbs()`
    // (two one-line additions to fq.rs) so that no Montgomery conversion happens at the boundary.
    pub fn fq(x: &Fq) -> bls_fq { bls_fq { l: x.mont_limbs() } }
    pub fn fq_back(x: &bls_fq) -> Fq { Fq::from_mont_limbs(x.l) }
    // `Fr(FrRepr)` in Montgomery form (fr.rs:54-58), through the same kind of accessors on fr.rs
    pub fn fr(x: &Fr) -> bls_fr_repr { bls_fr_repr { l: x.mont_limbs() } }
    pub fn fr_back(x: &bls_fr_repr) -> Fr { Fr::from_mont_limbs(x.l) }
    pub fn fq2(x: &Fq2) -> bls_fq2 { bls_fq2 { c0: fq(&x.c0), c1: fq(&x.c1) } }
    pub fn fq2_back(x: &bls_fq2) -> Fq2 { Fq2 { c0: fq_back(&x.c0), c1: fq_back(&x.c1) } }
    pub fn fq6(x: &Fq6) -> bls_fq6 { bls_fq6 { c0: fq2(&x.c0), c1: fq2(&x.c1), c2: fq2(&x.c2) } }
    pub fn fq6_back(x: &bls_fq6) -> Fq6 { Fq6 { c0: fq2_back(&x.c0), c1: fq2_back(&x.c1), c2: fq2_back(&x.c2) } }
    pub fn fq12(x: &Fq12) -> bls_fq12 { bls_fq12 { c0: fq6(&x.c0), c1: fq6(&x.c1) } }
    pub fn fq12_back(x: &bls_fq12) -> Fq12 { Fq12 { c0: fq6_back(&x.c0), c1: fq6_back(&x.c1) } }
    pub fn g1_affine(p: &G1Affine) -> bls_g1_affine { bls_g1_affine { x: fq(&p.x), y: fq(&p.y), infinity: p.infinity as u64 } }
    pub fn g2_affine(p: &G2Affine) -> bls_g2_affine { bls_g2_affine { x: fq2(&p.x), y: fq2(&p.y), infinity: p.infinity as u64 } }
    pub fn g2_affine_back(p: &bls_g2_affine) -> G2Affine { G2Affine { x: fq2_back(&p.x), y: fq2_back(&p.y), infinity: p.infinity != 0 } }
    pub fn g1_affine_back(p: &bls_g1_affine) -> G1Affine { G1Affine { x: fq_back(&p.x), y: fq_back(&p.y), infinity: p.infinity != 0 } }
    pub fn g1(p: &G1) -> bls_g1 { bls_g1 { x: fq(&p.x), y: fq(&p.y), z: fq(&p.z) } }
    pub fn g1_back(p: &bls_g1) -> G1 { G1 { x: fq_back(&p.x), y: fq_back(&p.y), z: fq_back(&p.z) } }
}


/// Several GPUs of one node behind one call: `Engine::miller_loop` takes all pairs of a product at once
/// (src/bls12_381/mod.rs:40-102), so the sharding, the 576-byte exchange and the single final
/// exponentiation happen inside the library (pairing_b200/csrc/mgpu.cu).
pub struct MultiGpu { m: Mutex<*mut bls_mgpu> }
unsafe impl Send for MultiGpu {}
unsafe impl Sync for MultiGpu {}

impl MultiGpu {
    pub fn new(devices: &[i32]) -> Result<MultiGpu, GpuError> {
        let mut err = 0;
        let m = unsafe { bls_mgpu_create(devices.as_ptr(), devices.len() as i32, &mut err) };
        if m.is_null() { return Err(GpuError(err, strerror(err))); }
        Ok(MultiGpu { m: Mutex::new(m) })
    }

    /// One `miller_loop` over all pairs, sharded over the devices.
    pub fn multi_miller_loop(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Fq12, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let mut out = marshal::FQ12_ZERO;
        let m = self.m.lock().unwrap();
        let rc = unsafe { bls_mgpu_multi_miller_loop(*m, pp.as_ptr(), qq.as_ptr(), p.len(), &mut out) };
        if rc != 0 { return Err(GpuError(rc, strerror(rc))); }
        Ok(marshal::fq12_back(&out))
    }

    /// `final_exponentiation(miller_loop(pairs))` over all devices.
    pub fn pairing_product(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Option<Fq12>, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let (mut out, mut some) = (marshal::FQ12_ZERO, 0u8);
        let m = self.m.lock().unwrap();
        let rc = unsafe { bls_mgpu_pairing_product(*m, pp.as_ptr(), qq.as_ptr(), p.len(), &mut out, &mut some) };
        if rc != 0 { return Err(GpuError(rc, strerror(rc))); }
        Ok(if some != 0 { Some(marshal::fq12_back(&out)) } else { None })
    }

    /// Independent pairings, sharded over the devices (no exchange step).
    pub fn pairing_batch(&self, p: &[G1Affine], q: &[G2Affine]) -> Result<Vec<Fq12>, GpuError> {
        assert_eq!(p.len(), q.len());
        let pp: Vec<bls_g1_affine> = p.iter().map(marshal::g1_affine).collect();
        let qq: Vec<bls_g2_affine> = q.iter().map(marshal::g2_affine).collect();
        let mut out = vec![marshal::FQ12_ZERO; p.len()];
        let m = self.m.lock().unwrap();
        let rc = unsafe { bls_mgpu_pairing_batch(*m, pp.as_ptr(), qq.as_ptr(), out.as_mut_ptr(), p.len()) };
        if rc != 0 { return Err(GpuError(rc, strerror(rc))); }
        Ok(out.iter().map(marshal::fq12_back).collect())
    }

    pub fn g1_wnaf_mul_batch(&self, bases: &[G1], k: &[FrRepr]) -> Result<Vec<G1>, GpuError> {
        assert_eq!(bases.len(), k.len());
        let bb: Vec<bls_g1> = bases.iter().map(marshal::g1).collect();
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = bb.clone();
        let m = self.m.lock().unwrap();
        let rc = unsafe { bls_mgpu_g1_wnaf_mul_batch(*m, bb.as_ptr(), kk.as_ptr(), out.as_mut_ptr(), bb.len()) };
        if rc != 0 { return Err(GpuError(rc, strerror(rc))); }
        Ok(out.iter().map(marshal::g1_back).collect())
    }

    pub fn g2_wnaf_mul_batch(&self, bases: &[G2], k: &[FrRepr]) -> Result<Vec<G2>, GpuError> {
        assert_eq!(bases.len(), k.len());
        let bb: Vec<bls_g2> = bases.iter().map(marshal::g2).collect();
        let kk: Vec<bls_fr_repr> = k.iter().map(|r| bls_fr_repr { l: r.0 }).collect();
        let mut out = bb.clone();
        let m = self.m.lock().unwrap();
        let rc = unsafe { bls_mgpu_g2_wnaf_mul_batch(*m, bb.as_ptr(), kk.as_ptr(), out.as_mut_ptr(), bb.len()) };
        if rc != 0 { return Err(GpuError(rc, strerror(rc))); }
        Ok(out.iter().map(marshal::g2_back).collect())
    }
}

impl Drop for MultiGpu {
    fn drop(&mut self) { unsafe { bls_mgpu_destroy(*self.m.lock().unwrap()) } }
}
