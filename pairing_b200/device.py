"""Device-resident batch API: torch CUDA tensors in, torch CUDA tensors out, no host copies.

torch is plumbing only (device memory, streams, torch.distributed); every kernel is launched
through the C ABI's `*_dev` entry points on torch's current stream.  Tensors are int64 with the
ABI's u64 word layout, one row per element (same shapes as the numpy API: (n, 13) G1Affine, ...).
"""
import ctypes

import torch

from . import _native as nat


def _check(t, w, name):
    if not (t.is_cuda and t.dtype == torch.int64 and t.dim() == 2 and t.shape[1] == w and t.is_contiguous()):
        raise ValueError("%s must be a contiguous CUDA int64 tensor of shape (n, %d)" % (name, w))


class DeviceEngine:
    def __init__(self, ctx=None, device=None):
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        self.ctx = ctx if ctx is not None else nat.Context(self.device.index or 0)
        self._scratch = {}

    def _stream(self):
        # torch's default stream has handle 0, which the C ABI reads as "use the context's own stream";
        # name the legacy default stream explicitly (cudaStreamLegacy == 0x1) so that the kernels are
        # ordered with torch's events and collectives.
        return torch.cuda.current_stream(self.device).cuda_stream or 1

    def _buf(self, key, nbytes):
        """Grow-only named scratch buffer, so the timed path never allocates."""
        t = self._scratch.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
            self._scratch[key] = t
        return t

    # ---------------------------------------------------------------- pairing engine
    def pairing(self, p, q, out=None):
        _check(p, nat.W_G1A, "p"); _check(q, nat.W_G2A, "q")
        n = p.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_FQ12), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_pairing_dev", p.data_ptr(), q.data_ptr(), out.data_ptr(), n, self._stream())
        return out

    def pairing_projective(self, p, q, out=None):
        """Engine::pairing on Jacobian rows (n,18),(n,36): into_affine fused in front of the pairing."""
        _check(p, nat.W_G1, "p"); _check(q, nat.W_G2, "q")
        n = p.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_FQ12), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_pairing_projective_dev", p.data_ptr(), q.data_ptr(), out.data_ptr(), n, self._stream())
        return out

    def miller_loop_batch(self, p, q, out=None):
        _check(p, nat.W_G1A, "p"); _check(q, nat.W_G2A, "q")
        n = p.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_FQ12), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_miller_loop_dev", p.data_ptr(), q.data_ptr(), out.data_ptr(), n, self._stream())
        return out

    def g2_prepare(self, q, out=None):
        _check(q, nat.W_G2A, "q")
        n = q.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_G2P), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_g2_prepare_dev", q.data_ptr(), out.data_ptr(), n, self._stream())
        return out

    def miller_loop_prepared_batch(self, p, qp, out=None):
        _check(p, nat.W_G1A, "p"); _check(qp, nat.W_G2P, "qp")
        n = p.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_FQ12), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_miller_loop_prepared_dev", p.data_ptr(), qp.data_ptr(), out.data_ptr(), n, self._stream())
        return out

    def pairing_shared_q(self, p, q1_prepared, out=None, final_exp=True):
        """e(P_i, Q) for every P_i against ONE prepared Q ((1, 2449) tensor): coefficients staged in shared memory by TMA."""
        _check(p, nat.W_G1A, "p"); _check(q1_prepared, nat.W_G2P, "q1_prepared")
        n = p.shape[0]
        if out is None:
            out = torch.empty((n, nat.W_FQ12), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_miller_loop_shared_q_dev", p.data_ptr(), q1_prepared.data_ptr(), out.data_ptr(), n, 1 if final_exp else 0, self._stream())
        return out

    def final_exponentiation(self, f, out=None):
        _check(f, nat.W_FQ12, "f")
        n = f.shape[0]
        if out is None:
            out = torch.empty_like(f)
        ok = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.ctx.call_dev("bls_final_exponentiation_dev", f.data_ptr(), out.data_ptr(), ok.data_ptr(), n, self._stream())
        return out, ok

    def multi_miller_loop(self, p, q, out=None):
        """Product of the Miller values of all pairs of this device's shard -> (1, 72)."""
        _check(p, nat.W_G1A, "p"); _check(q, nat.W_G2A, "q")
        n = p.shape[0]
        if out is None:
            out = torch.empty((1, nat.W_FQ12), dtype=torch.int64, device=self.device)
        scr = self._buf("mm", self.ctx.multi_miller_scratch_bytes(n))
        self.ctx.call_dev("bls_multi_miller_loop_dev", p.data_ptr(), q.data_ptr(), n, out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    def pairing_product(self, p, q, out=None):
        """final_exponentiation(miller_loop(all pairs of this device)) -> ((1, 72), is_some (1,) uint8)."""
        _check(p, nat.W_G1A, "p"); _check(q, nat.W_G2A, "q")
        n = p.shape[0]
        if out is None:
            out = torch.empty((1, nat.W_FQ12), dtype=torch.int64, device=self.device)
        ok = torch.empty(1, dtype=torch.uint8, device=self.device)
        scr = self._buf("mm", self.ctx.multi_miller_scratch_bytes(n))
        self.ctx.call_dev("bls_pairing_product_dev", p.data_ptr(), q.data_ptr(), n, out.data_ptr(), ok.data_ptr(), scr.data_ptr(), self._stream())
        return out, ok

    def fq12_product_tail(self, f, final_exp=False, out=None):
        """Product of a few Fq12 values (per-device partials) by one block, optionally followed by the single final
        exponentiation on the warp-cooperative engine -> ((1, 72), is_some)."""
        _check(f, nat.W_FQ12, "f")
        if out is None:
            out = torch.empty((1, nat.W_FQ12), dtype=torch.int64, device=self.device)
        ok = torch.ones(1, dtype=torch.uint8, device=self.device)
        self.ctx.call_dev("bls_fq12_product_tail_dev", f.data_ptr(), f.shape[0], out.data_ptr(), 1 if final_exp else 0, ok.data_ptr(), self._stream())
        return out, ok

    def fq12_pow(self, a, k, out=None):
        _check(a, nat.W_FQ12, "a"); _check(k, nat.W_FR, "k")
        if out is None:
            out = torch.empty_like(a)
        self.ctx.call_dev("bls_fq12_pow_dev", a.data_ptr(), k.data_ptr(), out.data_ptr(), a.shape[0], self._stream())
        return out

    def fq12_product(self, f, out=None):
        _check(f, nat.W_FQ12, "f")
        n = f.shape[0]
        if out is None:
            out = torch.empty((1, nat.W_FQ12), dtype=torch.int64, device=self.device)
        scr = self._buf("prod", self.ctx.fq12_product_scratch_bytes(n))
        self.ctx.call_dev("bls_fq12_product_dev", f.data_ptr(), n, out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    # ---------------------------------------------------------------- curves
    def g1_wnaf_mul(self, bases, k, window=0, out=None):
        _check(bases, nat.W_G1, "bases"); _check(k, nat.W_FR, "k")
        if out is None:
            out = torch.empty_like(bases)
        self.ctx.call_dev("bls_g1_wnaf_mul_dev", bases.data_ptr(), k.data_ptr(), out.data_ptr(), bases.shape[0], window, self._stream())
        return out

    def g2_wnaf_mul(self, bases, k, window=0, out=None):
        _check(bases, nat.W_G2, "bases"); _check(k, nat.W_FR, "k")
        if out is None:
            out = torch.empty_like(bases)
        self.ctx.call_dev("bls_g2_wnaf_mul_dev", bases.data_ptr(), k.data_ptr(), out.data_ptr(), bases.shape[0], window, self._stream())
        return out

    def msm(self, bases, k, g2=False, window=0, out=None):
        """sum_i k_i * bases_i over affine rows ((n, 13) G1 / (n, 25) G2) and (n, 4) FrRepr scalars -> one normalised
        Jacobian row (1, 18) / (1, 36).  window: bucket width c in 2..20, 0 = the library's choice for n."""
        _check(bases, nat.W_G2A if g2 else nat.W_G1A, "bases"); _check(k, nat.W_FR, "k")
        n = bases.shape[0]
        if k.shape[0] != n:
            raise ValueError("bases and k must have the same length")
        if out is None:
            out = torch.empty((1, nat.W_G2 if g2 else nat.W_G1), dtype=torch.int64, device=self.device)
        else:
            _check(out, nat.W_G2 if g2 else nat.W_G1, "out")
        scr = self._buf("msm", self.ctx.msm_scratch_bytes(2 if g2 else 1, n, window))
        self.ctx.call_dev("bls_g2_msm_dev" if g2 else "bls_g1_msm_dev", bases.data_ptr(), k.data_ptr(), n, window, out.data_ptr(),
                          scr.data_ptr(), self._stream())
        return out

    def msm_batch(self, bases, k, g2=False, window=0, out=None):
        """m independent sums: k (m, n, 4) FrRepr scalars against affine bases shared by every sum ((n, 13) G1 / (n, 25) G2)
        or one set per sum ((m, n, 13) / (m, n, 25)) -> (m, 18) / (m, 36) normalised Jacobian rows.  window as for msm."""
        wa, w = (nat.W_G2A, nat.W_G2) if g2 else (nat.W_G1A, nat.W_G1)
        if not (k.is_cuda and k.dtype == torch.int64 and k.dim() == 3 and k.shape[2] == nat.W_FR and k.is_contiguous()):
            raise ValueError("k must be a contiguous CUDA int64 tensor of shape (m, n, 4)")
        m, n = k.shape[:2]
        if not (bases.is_cuda and bases.dtype == torch.int64 and tuple(bases.shape) in ((n, wa), (m, n, wa)) and bases.is_contiguous()):
            raise ValueError("bases must be a contiguous CUDA int64 tensor of shape (%d, %d) or (%d, %d, %d)" % (n, wa, m, n, wa))
        if out is None:
            out = torch.empty((m, w), dtype=torch.int64, device=self.device)
        elif not (out.is_cuda and out.dtype == torch.int64 and tuple(out.shape) == (m, w) and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape (%d, %d)" % (m, w))
        scr = self._buf("msm", self.ctx.msm_batch_scratch_bytes(2 if g2 else 1, n, m, window))
        self.ctx.call_dev("bls_g2_msm_batch_dev" if g2 else "bls_g1_msm_batch_dev", bases.data_ptr(), 1 if bases.dim() == 2 else 0,
                          k.data_ptr(), n, m, window, out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    def fr_fft(self, a, kind="fft", out=None):
        """bellman's EvaluationDomain transforms over Fr on the device: kind "fft" | "ifft" | "coset_fft" | "icoset_fft"
        on one polynomial (n, 4) or m polynomials (m, n, 4) of Montgomery-form values, n a power of two.  out may be a
        (contiguous, same-shape) tensor, `a` itself included (in place)."""
        if not (a.is_cuda and a.dtype == torch.int64 and a.dim() in (2, 3) and a.shape[-1] == nat.W_FR and a.is_contiguous()):
            raise ValueError("a must be a contiguous CUDA int64 tensor of shape (n, 4) or (m, n, 4)")
        n = a.shape[-2]
        log_n = n.bit_length() - 1
        if n != 1 << log_n:
            raise ValueError("the polynomial length must be a power of two, got %d" % n)
        m = a.shape[0] if a.dim() == 3 else 1
        if out is None:
            out = torch.empty_like(a)
        elif not (out.is_cuda and out.dtype == torch.int64 and out.shape == a.shape and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape %r" % (tuple(a.shape),))
        scr = self._buf("fft", self.ctx.fr_fft_scratch_bytes(log_n, m))
        self.ctx.call_dev("bls_fr_fft_dev", nat.FFT_KINDS[kind], a.data_ptr(), out.data_ptr(), log_n, m, scr.data_ptr(), self._stream())
        return out

    def groth16_h(self, a, b, c, out=None):
        """Groth16's quotient polynomial on the device (the `h` block of bellman's create_proof): a, b, c are the
        evaluations of one proof (len, 4) or of m proofs (m, len, 4), Montgomery-form values -> H's coefficients 0 .. n - 2
        as canonical FrRepr, (n - 1, 4) or (m, n - 1, 4), n the smallest power of two >= len.  The (m, n - 1, 4) result is
        the k of msm_batch against n - 1 shared bases."""
        if not (a.is_cuda and a.dtype == torch.int64 and a.dim() in (2, 3) and a.shape[-1] == nat.W_FR and a.is_contiguous()):
            raise ValueError("a must be a contiguous CUDA int64 tensor of shape (len, 4) or (m, len, 4)")
        for t, name in ((b, "b"), (c, "c")):
            if not (t.is_cuda and t.dtype == torch.int64 and t.shape == a.shape and t.is_contiguous()):
                raise ValueError("%s must be a contiguous CUDA int64 tensor of shape %r" % (name, tuple(a.shape)))
        length = a.shape[-2]
        m = a.shape[0] if a.dim() == 3 else 1
        shape = tuple(a.shape[:-2]) + ((1 << max(length - 1, 0).bit_length()) - 1, nat.W_FR)
        if out is None:
            out = torch.empty(shape, dtype=torch.int64, device=self.device)
        elif not (out.is_cuda and out.dtype == torch.int64 and tuple(out.shape) == shape and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape %r" % (shape,))
        scr = self._buf("groth16_h", self.ctx.fr_groth16_h_scratch_bytes(length, m))
        self.ctx.call_dev("bls_fr_groth16_h_dev", a.data_ptr(), b.data_ptr(), c.data_ptr(), length, m, out.data_ptr(), scr.data_ptr(),
                          self._stream())
        return out

    def groth16_prove(self, params, a, b, c, input, aux, densities, r, s, out=None):
        """bellman's groth16::create_proof for m proofs of one circuit on the device (bls_groth16_prove_dev): the arguments
        of Context.groth16_prove as contiguous CUDA int64 tensors -- a, b, c (m, len, 4), input (m, num_inputs, 4), aux
        (m, num_aux, 4), r, s (m, 4) and params' queries -- except params' vk rows and the densities (numpy bool arrays),
        which stay on the host.  Returns (A (m, 13), B (m, 25), C (m, 13)), views of one (m, 51) tensor (`out` if given)."""
        for t, name in ((a, "a"), (b, "b"), (c, "c"), (input, "input"), (aux, "aux")):
            if not (t.is_cuda and t.dtype == torch.int64 and t.dim() == 3 and t.shape[2] == nat.W_FR and t.is_contiguous()):
                raise ValueError("%s must be a contiguous CUDA int64 tensor of shape (m, n, 4)" % name)
        m, length = a.shape[:2]
        if b.shape != a.shape or c.shape != a.shape or input.shape[0] != m or aux.shape[0] != m:
            raise ValueError("a, b, c must have one shape (m, len, 4) and input, aux m rows: %r %r %r %r %r"
                             % tuple(tuple(x.shape) for x in (a, b, c, input, aux)))
        for t, name in ((r, "r"), (s, "s")):
            _check(t, nat.W_FR, name)
            if t.shape[0] != m:
                raise ValueError("%s must have %d rows" % (name, m))
        for name, w in (("h", nat.W_G1A), ("l", nat.W_G1A), ("a", nat.W_G1A), ("b_g1", nat.W_G1A), ("b_g2", nat.W_G2A)):
            _check(getattr(params, name), w, "params." + name)
        ni, na = input.shape[1], aux.shape[1]
        vk = [x.cpu().numpy() if isinstance(x, torch.Tensor) else x for x in (params.alpha_g1, params.beta_g1, params.delta_g1, params.beta_g2, params.delta_g2)]
        pc = nat.groth16_params_c(nat.Groth16Params(*vk, params.h, params.l, params.a, params.b_g1, params.b_g2),
                                  lambda t: t.data_ptr(), lambda t: t.shape[0])
        dw = [nat.density_words(d, bits, name) for d, bits, name in zip(densities, (na, ni, na), ("a_aux_density", "b_input_density", "b_aux_density"))]
        if out is None:
            out = torch.empty((m, nat.W_PROOF), dtype=torch.int64, device=self.device)
        elif not (out.is_cuda and out.dtype == torch.int64 and tuple(out.shape) == (m, nat.W_PROOF) and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape (%d, %d)" % (m, nat.W_PROOF))
        scr = self._buf("groth16", self.ctx.groth16_prove_scratch_bytes(pc, length, ni, na, dw, m))
        self.ctx.call_dev("bls_groth16_prove_dev", ctypes.byref(pc), a.data_ptr(), b.data_ptr(), c.data_ptr(), length, input.data_ptr(), ni,
                          aux.data_ptr(), na, *[nat._p(w) for w in dw], r.data_ptr(), s.data_ptr(), m, out.data_ptr(), scr.data_ptr(),
                          self._stream())
        return out[:, :nat.W_G1A], out[:, nat.W_G1A:nat.W_G1A + nat.W_G2A], out[:, nat.W_G1A + nat.W_G2A:]

    def groth16_generate_parameters(self, abc, num_constraints, num_inputs, num_aux, g1, g2, alpha, beta, gamma, delta, tau):
        """bellman's groth16::generate_parameters on the device (bls_groth16_generate_parameters_dev): abc three (offsets,
        constraint, coeff) contiguous CUDA tensors -- int64 (nv + 1,), int32 (nnz,), int64 (nnz, 4) -- and g1, g2, alpha ..
        tau as for Context.groth16_generate_parameters (host memory).  Returns a Groth16Parameters whose rows are CUDA int64
        tensors and whose densities are numpy bool arrays, so it goes to groth16_prove unchanged.  Reading a_len and b_len to
        trim the queries synchronises the stream."""
        ni, na = int(num_inputs), int(num_aux)
        mats = self._r1cs_mats(abc, ni + na)
        host = [nat._arr(nat.np.reshape(x, (1, -1)), w, name) for x, w, name in
                ((g1, nat.W_G1A, "g1"), (g2, nat.W_G2A, "g2"), (alpha, nat.W_FR, "alpha"), (beta, nat.W_FR, "beta"), (gamma, nat.W_FR, "gamma"),
                 (delta, nat.W_FR, "delta"), (tau, nat.W_FR, "tau"))]
        bufs, out = self._parameters_out(num_constraints, ni, na)
        scr = self._buf("groth16_setup", self.ctx.groth16_generate_parameters_scratch_bytes(mats, num_constraints, ni, na))
        self.ctx.call_dev("bls_groth16_generate_parameters_dev", mats, num_constraints, ni, na, *[nat._p(x) for x in host], ctypes.byref(out),
                          scr.data_ptr(), self._stream())
        return self._parameters(bufs, ni, na)

    def groth16_mpc_new(self, abc, num_constraints, num_inputs, num_aux, phase1, g1, g2):
        """phase2's MPCParameters::new on the device (bls_groth16_mpc_new_dev): abc as for groth16_generate_parameters, phase1
        a Groth16Phase1 whose row sets are contiguous CUDA int64 tensors ((n, 13), (n, 25) for coeffs_g2, (n - 1, 13) for h)
        and whose vk points are host rows; g1 and g2 host rows.  Returns a Groth16Parameters as groth16_generate_parameters
        does; reading a_len and b_len synchronises the stream."""
        ni, na = int(num_inputs), int(num_aux)
        mats = self._r1cs_mats(abc, ni + na)
        for name in ("coeffs_g1", "alpha_coeffs_g1", "beta_coeffs_g1", "coeffs_g2", "h"):
            _check(getattr(phase1, name), nat.W_G2A if name == "coeffs_g2" else nat.W_G1A, name)
        ph = nat.groth16_phase1_c(phase1, num_constraints, lambda t: t.data_ptr(), lambda t: int(t.shape[0]))
        g1 = nat._arr(nat.np.reshape(g1, (1, -1)), nat.W_G1A, "g1")
        g2 = nat._arr(nat.np.reshape(g2, (1, -1)), nat.W_G2A, "g2")
        bufs, out = self._parameters_out(num_constraints, ni, na)
        scr = self._buf("groth16_mpc", self.ctx.groth16_mpc_new_scratch_bytes(mats, num_constraints, ni, na))
        self.ctx.call_dev("bls_groth16_mpc_new_dev", mats, num_constraints, ni, na, ctypes.byref(ph), nat._p(g1), nat._p(g2), ctypes.byref(out),
                          scr.data_ptr(), self._stream())
        return self._parameters(bufs, ni, na)

    def groth16_mpc_contribute(self, params, delta, s, r, in_place=False):
        """phase2's MPCParameters::contribute on the device (bls_groth16_mpc_contribute_dev): params a Groth16Parameters whose
        vk rows and queries are CUDA int64 tensors; delta, s and r host rows as for Context.groth16_mpc_contribute.  Returns
        (the contributed Groth16Parameters, the (89,) pubkey as a CUDA int64 tensor); in_place writes h and l over the inputs."""
        _check(params.h, nat.W_G1A, "h"); _check(params.l, nat.W_G1A, "l")
        host = [nat._arr(nat.np.reshape(x, (1, -1)), w, name) for x, w, name in ((delta, nat.W_FR, "delta"), (s, nat.W_G1A, "s"), (r, nat.W_G2A, "r"))]
        vk = torch.cat([getattr(params, name).reshape(-1) for name, _, _ in nat.VK_POINT_ROWS]).contiguous()
        h, l = (params.h, params.l) if in_place else (torch.empty_like(params.h), torch.empty_like(params.l))
        pk = torch.zeros(nat.W_MPC_PUBKEY, dtype=torch.int64, device=self.device)
        scr = self._buf("groth16_mpc", self.ctx.groth16_mpc_contribute_scratch_bytes(params.h.shape[0], params.l.shape[0]))
        self.ctx.call_dev("bls_groth16_mpc_contribute_dev", *[nat._p(x) for x in host], vk.data_ptr(), params.h.data_ptr(), params.h.shape[0],
                          params.l.data_ptr(), params.l.shape[0], h.data_ptr(), l.data_ptr(), pk.data_ptr(), scr.data_ptr(), self._stream())
        return nat.contributed(params, vk, h, l), pk

    def groth16_mpc_verify(self, before, after, pubkeys, rho_h, rho_l):
        """phase2's MPCParameters::verify on the device (bls_groth16_mpc_verify_dev): before and after Groth16Parameters of CUDA
        tensors, pubkeys a (k, 89) CUDA int64 tensor, rho_h and rho_l (h_len, 4) / (l_len, 4) CUDA int64 tensors.  Returns a
        bool (reading it synchronises the stream)."""
        row = lambda t: t.cpu().numpy().view(nat.np.uint64)
        kb, ka = (nat.groth16_key_c(k, lambda t: t.data_ptr(), lambda t: int(t.shape[0]), row) for k in (before, after))
        _check(pubkeys, nat.W_MPC_PUBKEY, "pubkeys"); _check(rho_h, nat.W_FR, "rho_h"); _check(rho_l, nat.W_FR, "rho_l")
        ok = torch.zeros(1, dtype=torch.uint8, device=self.device)
        scr = self._buf("groth16_mpc", self.ctx.groth16_mpc_verify_scratch_bytes(kb, ka, pubkeys.shape[0]))
        self.ctx.call_dev("bls_groth16_mpc_verify_dev", ctypes.byref(kb), ctypes.byref(ka), pubkeys.data_ptr(), pubkeys.shape[0], rho_h.data_ptr(),
                          rho_l.data_ptr(), ok.data_ptr(), scr.data_ptr(), self._stream())
        return bool(ok.cpu()[0])

    @staticmethod
    def _r1cs_mats(abc, nv):
        if len(abc) != 3:
            raise ValueError("abc must hold the three matrices A, B and C")
        mats = (nat.R1csMatrixC * 3)()
        for i, (off, cons, coeff) in enumerate(abc):
            ok = all(t.is_cuda and t.is_contiguous() for t in (off, cons, coeff)) and off.dtype == torch.int64 and cons.dtype == torch.int32 \
                and coeff.dtype == torch.int64 and tuple(off.shape) == (nv + 1,) and coeff.dim() == 2 and coeff.shape[1] == nat.W_FR \
                and tuple(cons.shape) == (coeff.shape[0],)
            if not ok:
                raise ValueError("matrix %d: offsets, constraint, coeff must be contiguous CUDA tensors int64 (%d,), int32 (nnz,), int64 (nnz, 4)"
                                 % (i, nv + 1))
            mats[i] = nat.R1csMatrixC(off.data_ptr(), cons.data_ptr(), coeff.data_ptr(), cons.shape[0])
        return mats

    def _parameters_out(self, num_constraints, ni, na):
        nv, n1 = ni + na, nat.domain_size(num_constraints) - 1
        e = lambda *shape: torch.zeros(shape, dtype=torch.int64, device=self.device)
        vk, ic, h, l, a, b_g1, b_g2 = e(nat.W_VK_POINTS), e(ni, nat.W_G1A), e(n1, nat.W_G1A), e(na, nat.W_G1A), e(nv, nat.W_G1A), e(nv, nat.W_G1A), e(nv, nat.W_G2A)
        dens = [torch.zeros((k + 31) // 32, dtype=torch.int32, device=self.device) for k in (na, ni, na)]
        lens = e(2)
        ok = torch.zeros(1, dtype=torch.uint8, device=self.device)
        out = nat.Groth16ParametersOutC(*[t.data_ptr() for t in (vk, ic, h, l, a, b_g1, b_g2, *dens, lens, ok)])
        return (vk, ic, h, l, a, b_g1, b_g2, dens, lens, ok), out

    @staticmethod
    def _parameters(bufs, ni, na):
        vk, ic, h, l, a, b_g1, b_g2, dens, lens, ok = bufs
        words = [d.cpu().numpy().view(nat.np.uint32) for d in dens]
        return nat.groth16_parameters(vk, ic, h, l, a, b_g1, b_g2, words, lens.cpu().numpy(), int(ok.cpu()[0]), ni, na)

    def _verify_args(self, pvk, ic, proofs, inputs):
        if not (pvk.is_cuda and pvk.dtype == torch.int64 and tuple(pvk.shape) == (nat.W_PVK,) and pvk.is_contiguous()):
            raise ValueError("pvk must be a contiguous CUDA int64 tensor of shape (%d,)" % nat.W_PVK)
        _check(ic, nat.W_G1A, "ic"); _check(proofs, nat.W_PROOF, "proofs")
        m, ni = proofs.shape[0], ic.shape[0] - 1
        if not (inputs.is_cuda and inputs.dtype == torch.int64 and tuple(inputs.shape) == (m, max(ni, 0), nat.W_FR) and inputs.is_contiguous()) or ni < 0:
            raise ValueError("ic must hold num_inputs + 1 points and inputs be a contiguous CUDA int64 tensor of shape (m, num_inputs, 4)")
        return m, ni

    def groth16_verify(self, pvk, ic, proofs, inputs, out=None):
        """bellman's verify_proof for m proofs on the device (bls_groth16_verify_dev): pvk the (5022,) tensor of
        Context.groth16_prepare_verifying_key, ic (num_inputs + 1, 13), proofs (m, 51), inputs (m, num_inputs, 4) -> (m,)
        uint8 tensor, 1 where the proof verifies."""
        m, ni = self._verify_args(pvk, ic, proofs, inputs)
        if out is None:
            out = torch.empty(m, dtype=torch.uint8, device=self.device)
        scr = self._buf("groth16_verify", self.ctx.groth16_verify_scratch_bytes(ni, m))
        self.ctx.call_dev("bls_groth16_verify_dev", pvk.data_ptr(), ic.data_ptr(), ni, proofs.data_ptr(), inputs.data_ptr(), m, out.data_ptr(),
                          scr.data_ptr(), self._stream())
        return out

    def groth16_verify_rlc(self, pvk, ic, proofs, inputs, rho, out=None):
        """the randomized batch check on the device (bls_groth16_verify_rlc_dev): groth16_verify's arguments and rho (m, 4)
        canonical FrRepr -> (1,) uint8 tensor (1 for m = 0)"""
        m, ni = self._verify_args(pvk, ic, proofs, inputs)
        _check(rho, nat.W_FR, "rho")
        if rho.shape[0] != m:
            raise ValueError("rho must have %d rows" % m)
        if out is None:
            out = torch.zeros(1, dtype=torch.uint8, device=self.device)
        scr = self._buf("groth16_verify_rlc", self.ctx.groth16_verify_rlc_scratch_bytes(ni, m))
        self.ctx.call_dev("bls_groth16_verify_rlc_dev", pvk.data_ptr(), ic.data_ptr(), ni, proofs.data_ptr(), inputs.data_ptr(), rho.data_ptr(), m,
                          out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    # ---------------------------------------------------------------- KZG commitments
    def _kzg_poly(self, srs, p, open_):
        _check(srs, nat.W_G1A, "srs")
        if not (p.is_cuda and p.dtype == torch.int64 and p.is_contiguous()):
            raise ValueError("p must be a contiguous CUDA int64 tensor of shape (m, n, 4)")
        return nat.kzg_poly_shape(tuple(p.shape), srs.shape[0], open_)

    def kzg_commit(self, srs, p, out=None):
        """c[j] = sum_i p[j, i] srs[i] on the device (bls_kzg_commit_dev): srs (>= n, 13), p (m, n, 4) Montgomery -> (m, 13)."""
        m, n = self._kzg_poly(srs, p, False)
        if out is None:
            out = torch.empty((m, nat.W_G1A), dtype=torch.int64, device=self.device)
        _check(out, nat.W_G1A, "out")
        scr = self._buf("kzg", self.ctx.kzg_scratch_bytes("commit", n, m))
        self.ctx.call_dev("bls_kzg_commit_dev", srs.data_ptr(), srs.shape[0], p.data_ptr(), n, m, out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    def kzg_open(self, srs, p, z):
        """open polynomial j at z[j] on the device (bls_kzg_open_dev): srs (>= n - 1, 13), p (m, n, 4), z (m, 4) Montgomery ->
        (y (m, 4) Montgomery, proof (m, 13) affine)."""
        m, n = self._kzg_poly(srs, p, True)
        _check(z, nat.W_FR, "z")
        if z.shape[0] != m:
            raise ValueError("z must have %d rows" % m)
        y = torch.empty((m, nat.W_FR), dtype=torch.int64, device=self.device)
        proof = torch.empty((m, nat.W_G1A), dtype=torch.int64, device=self.device)
        scr = self._buf("kzg", self.ctx.kzg_scratch_bytes("open", n, m))
        self.ctx.call_dev("bls_kzg_open_dev", srs.data_ptr(), srs.shape[0], p.data_ptr(), n, z.data_ptr(), m, y.data_ptr(), proof.data_ptr(),
                          scr.data_ptr(), self._stream())
        return y, proof

    def kzg_open_all_prepare(self, srs, log_n, out=None):
        """the FK20 table on the device (bls_kzg_open_all_prepare_dev): srs (>= n - 1, 13), n = 2^log_n -> (2n, 13)"""
        _check(srs, nat.W_G1A, "srs")
        n = 1 << log_n
        if srs.shape[0] < n - 1:
            raise ValueError("the SRS has %d points, the domain of %d needs %d" % (srs.shape[0], n, n - 1))
        if out is None:
            out = torch.empty((2 * n, nat.W_G1A), dtype=torch.int64, device=self.device)
        _check(out, nat.W_G1A, "out")
        if out.shape[0] != 2 * n:
            raise ValueError("out must have %d rows" % (2 * n))
        scr = self._buf("kzg_open_all_prepare", self.ctx.kzg_scratch_bytes("open_all_prepare", log_n))
        self.ctx.call_dev("bls_kzg_open_all_prepare_dev", srs.data_ptr(), srs.shape[0], log_n, out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    def kzg_open_all(self, table, p):
        """open every polynomial at every omega^k on the device (bls_kzg_open_all_dev): table (2n, 13), p (m, n, 4) Montgomery ->
        (y (m, n, 4) Montgomery, proof (m, n, 13) affine)"""
        _check(table, nat.W_G1A, "table")
        if not (p.is_cuda and p.dtype == torch.int64 and p.is_contiguous()):
            raise ValueError("p must be a contiguous CUDA int64 tensor of shape (m, n, 4)")
        m, n, log_n = nat.open_all_shape(tuple(p.shape), table.shape[0])
        y = torch.empty((m, n, nat.W_FR), dtype=torch.int64, device=self.device)
        proof = torch.empty((m, n, nat.W_G1A), dtype=torch.int64, device=self.device)
        scr = self._buf("kzg_open_all", self.ctx.kzg_scratch_bytes("open_all", log_n, m))
        self.ctx.call_dev("bls_kzg_open_all_dev", table.data_ptr(), p.data_ptr(), log_n, m, y.data_ptr(), proof.data_ptr(), scr.data_ptr(),
                          self._stream())
        return y, proof

    def _point_fft(self, g2, a, kind, out):
        w = nat.W_G2A if g2 else nat.W_G1A
        if not (a.is_cuda and a.dtype == torch.int64 and a.dim() in (2, 3) and a.shape[-1] == w and a.is_contiguous()):
            raise ValueError("a must be a contiguous CUDA int64 tensor of shape (n, %d) or (m, n, %d)" % (w, w))
        n = a.shape[-2]
        log_n = n.bit_length() - 1
        if n != 1 << log_n:
            raise ValueError("the row length must be a power of two, got %d" % n)
        m = a.shape[0] if a.dim() == 3 else 1
        if out is None:
            out = torch.empty_like(a)
        elif not (out.is_cuda and out.dtype == torch.int64 and out.shape == a.shape and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape %r" % (tuple(a.shape),))
        scr = self._buf("point_fft", self.ctx.point_fft_scratch_bytes(2 if g2 else 1, log_n, m))
        self.ctx.call_dev("bls_g2_fft_dev" if g2 else "bls_g1_fft_dev", nat.FFT_KINDS[kind], a.data_ptr(), out.data_ptr(), log_n, m,
                          scr.data_ptr(), self._stream())
        return out

    def g1_fft(self, a, kind="fft", out=None):
        """bellman's EvaluationDomain<Point<G1>> transforms on the device: kind "fft" | "ifft" | "coset_fft" | "icoset_fft" on
        (n, 13) or (m, n, 13) affine rows, n a power of two -> canonical affine rows.  out may be `a` itself (in place)."""
        return self._point_fft(False, a, kind, out)

    def g2_fft(self, a, kind="fft", out=None):
        """g1_fft over G2: (n, 25) or (m, n, 25) affine rows"""
        return self._point_fft(True, a, kind, out)

    def kzg_prepare_verifying_key(self, g, h, tau_h):
        """the (4963,) bls_kzg_pvk of Context.kzg_prepare_verifying_key as a CUDA tensor (rows in host or device memory)"""
        rows = [x.cpu().numpy() if isinstance(x, torch.Tensor) else x for x in (g, h, tau_h)]
        return torch.from_numpy(self.ctx.kzg_prepare_verifying_key(*rows).view(nat.np.int64)).to(self.device)

    def _kzg_verify_args(self, pvk, c, y, z, proof):
        if not (pvk.is_cuda and pvk.dtype == torch.int64 and tuple(pvk.shape) == (nat.W_KZG_PVK,) and pvk.is_contiguous()):
            raise ValueError("pvk must be a contiguous CUDA int64 tensor of shape (%d,)" % nat.W_KZG_PVK)
        _check(c, nat.W_G1A, "c"); _check(proof, nat.W_G1A, "proof"); _check(y, nat.W_FR, "y"); _check(z, nat.W_FR, "z")
        m = c.shape[0]
        if not (proof.shape[0] == y.shape[0] == z.shape[0] == m):
            raise ValueError("c, y, z and proof must have the same number of rows")
        return m

    def kzg_verify(self, pvk, c, y, z, proof, out=None):
        """bls_kzg_verify_dev: pvk (4963,), c and proof (m, 13), y and z (m, 4) Montgomery -> (m,) uint8 tensor, 1 where the
        opening verifies."""
        m = self._kzg_verify_args(pvk, c, y, z, proof)
        if out is None:
            out = torch.empty(m, dtype=torch.uint8, device=self.device)
        scr = self._buf("kzg_verify", self.ctx.kzg_scratch_bytes("verify", m))
        self.ctx.call_dev("bls_kzg_verify_dev", pvk.data_ptr(), c.data_ptr(), y.data_ptr(), z.data_ptr(), proof.data_ptr(), m, out.data_ptr(),
                          scr.data_ptr(), self._stream())
        return out

    def kzg_verify_rlc(self, pvk, c, y, z, proof, rho, out=None):
        """the randomized check on the device (bls_kzg_verify_rlc_dev): kzg_verify's arguments and rho (m, 4) canonical
        FrRepr -> (1,) uint8 tensor (1 for m = 0)"""
        m = self._kzg_verify_args(pvk, c, y, z, proof)
        _check(rho, nat.W_FR, "rho")
        if rho.shape[0] != m:
            raise ValueError("rho must have %d rows" % m)
        if out is None:
            out = torch.zeros(1, dtype=torch.uint8, device=self.device)
        scr = self._buf("kzg_verify_rlc", self.ctx.kzg_scratch_bytes("verify_rlc", m))
        self.ctx.call_dev("bls_kzg_verify_rlc_dev", pvk.data_ptr(), c.data_ptr(), y.data_ptr(), z.data_ptr(), proof.data_ptr(), rho.data_ptr(), m,
                          out.data_ptr(), scr.data_ptr(), self._stream())
        return out

    def fr_op(self, op, a, b=None, out=None):
        """Fr element-wise operation on (n, 4) tensors (bls_fr_op_batch's ops: "add", "mul", ..., "from_repr", "into_repr")
        -> (out, ok), ok an (n,) uint8 tensor, 0 for the inverse of zero or from_repr of a value >= r.  out may be a or b."""
        _check(a, nat.W_FR, "a")
        if b is not None:
            _check(b, nat.W_FR, "b")
            if b.shape != a.shape:
                raise ValueError("a and b must have the same length")
        if out is None:
            out = torch.empty_like(a)
        elif not (out.is_cuda and out.dtype == torch.int64 and out.shape == a.shape and out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA int64 tensor of shape %r" % (tuple(a.shape),))
        ok = torch.empty(a.shape[0], dtype=torch.uint8, device=self.device)
        self.ctx.call_dev("bls_fr_op_dev", nat.OPS[op], a.data_ptr(), b.data_ptr() if b is not None else None, out.data_ptr(),
                          ok.data_ptr(), a.shape[0], self._stream())
        return out, ok

    def wnaf_table(self, base, window, g2=False):
        """Wnaf::base(g, n): the shared window table (2^(window-1), W) on the device."""
        w = nat.W_G2 if g2 else nat.W_G1
        _check(base, w, "base")
        table = torch.empty((1 << (window - 1), w), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_g2_wnaf_table_dev" if g2 else "bls_g1_wnaf_table_dev", base.data_ptr(), window, table.data_ptr(), self._stream())
        return table

    def wnaf_fixed_base(self, table, window, k, g2=False, out=None):
        """`.scalar(k_i)` for every scalar against one shared table."""
        w = nat.W_G2 if g2 else nat.W_G1
        _check(table, w, "table"); _check(k, nat.W_FR, "k")
        if table.shape[0] != 1 << (window - 1):
            raise ValueError("table has %d entries, window %d needs %d" % (table.shape[0], window, 1 << (window - 1)))
        if out is None:
            out = torch.empty((k.shape[0], w), dtype=torch.int64, device=self.device)
        self.ctx.call_dev("bls_g2_wnaf_fixed_base_dev" if g2 else "bls_g1_wnaf_fixed_base_dev", table.data_ptr(), window, k.data_ptr(), out.data_ptr(), k.shape[0], self._stream())
        return out

    def g1_batch_normalization_(self, v):
        _check(v, nat.W_G1, "v")
        scr = self._buf("bn", self.ctx.batch_normalization_scratch_bytes(1, v.shape[0]))
        self.ctx.call_dev("bls_g1_batch_normalization_dev", v.data_ptr(), v.shape[0], scr.data_ptr(), self._stream())
        return v

    def g2_batch_normalization_(self, v):
        _check(v, nat.W_G2, "v")
        scr = self._buf("bn", self.ctx.batch_normalization_scratch_bytes(2, v.shape[0]))
        self.ctx.call_dev("bls_g2_batch_normalization_dev", v.data_ptr(), v.shape[0], scr.data_ptr(), self._stream())
        return v

    # normalised Jacobian -> affine rows (pure data movement: x, y, infinity flag = (z == 0))
    @staticmethod
    def jacobian_to_affine_rows(v, coord_words):
        n = v.shape[0]
        out = torch.zeros((n, 2 * coord_words + 1), dtype=torch.int64, device=v.device)
        out[:, :2 * coord_words] = v[:, :2 * coord_words]
        out[:, 2 * coord_words] = (v[:, 2 * coord_words:] == 0).all(dim=1).to(torch.int64)
        return out
