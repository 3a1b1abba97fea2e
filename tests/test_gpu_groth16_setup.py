"""Groth16 parameters (bls_groth16_generate_parameters_batch / _dev, Context.groth16_generate_parameters,
DeviceEngine.groth16_generate_parameters, Groth16::generate_parameters).

Every point of a key is [e]g for an exponent e the model (tests/groth16_setup_model.py) computes, so the GPU's bytes are
compared with [e]g from the oracle on toy circuits and from bls_g*_mul_batch at full size.  The generated keys then go
through the prover and both verifiers: the first end-to-end check of the three calls together."""
import ctypes
import os
import random
import re
import subprocess
import tempfile
import time

import numpy as np
import pytest

import bls_model as bm
import groth16_prove_model as gp
import groth16_setup_model as gs
import oracle_lib as o
from fr_fft_model import fr_root
from groth16_h_model import domain_log
from test_gpu_groth16_prove import SHAPES, W1, W2, _ints, _limbs, _mont_rows, _points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER


def _scalars(rng, tau=None):
    """alpha, beta, gamma, delta, tau (canonical ints)"""
    s = [rng.randrange(1, R) for _ in range(5)]
    if tau is not None:
        s[4] = tau % R
    return s


def _mont1(x):
    return _mont_rows([x])[0]


def _call(ctx, abc, nc, ni, na, sc, g1=None, g2=None):
    g1_, g2_ = o.generators()
    return ctx.groth16_generate_parameters(abc, nc, ni, na, g1_[0] if g1 is None else g1, g2_[0] if g2 is None else g2,
                                           *[_mont1(x) for x in sc])


def _expect(key, t1=1, t2=1, points=_points):
    """the rows a key with these exponents has on the bases [t1] G1, [t2] G2"""
    m1 = lambda e: points(False, [x * t1 % R for x in e])
    m2 = lambda e: points(True, [x * t2 % R for x in e])
    return {"alpha_g1": m1([key["alpha"]])[0], "beta_g1": m1([key["beta"]])[0], "delta_g1": m1([key["delta"]])[0],
            "beta_g2": m2([key["beta"]])[0], "gamma_g2": m2([key["gamma"]])[0], "delta_g2": m2([key["delta"]])[0],
            "h": m1(key["h"]), "ic": m1(key["ic"]), "l": m1(key["l"]), "a": m1(key["a"]), "b_g1": m1(key["b"]), "b_g2": m2(key["b"])}


def _assert_key(got, key, t1=1, t2=1, points=_points):
    want = _expect(key, t1, t2, points)
    for name, rows in want.items():
        g = np.asarray(getattr(got, name).cpu() if hasattr(getattr(got, name), "cpu") else getattr(got, name), dtype=np.uint64)
        assert g.tobytes() == np.asarray(rows, dtype=np.uint64).tobytes(), name
    for d, w, name in zip(got.densities, key["densities"], ("a_aux", "b_input", "b_aux")):
        assert list(np.asarray(d, dtype=bool)) == list(w), name
    assert (len(got.a), len(got.b_g1), len(got.b_g2)) == (key["lens"][0], key["lens"][1], key["lens"][1])
    assert got.ok == key["ok"]


def _toy(nc, ni, na, seed, dup=False):
    c = gp.ToyCircuit(nc, ni, na, seed)
    return c, gs.csr_from_cons(c.all_cons, ni + na, seed if dup else None)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_model_agrees_with_toy_setup(nc, ni, na):
    rng = random.Random(nc * 31 + ni * 7 + na)
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
    al, be, ga, de, tau = _scalars(rng)
    key = gs.generate(abc, circ.length, ni, na, tau, al, be, ga, de)
    toy = circ.setup(tau, al, be, ga, de)
    for name in ("h", "ic", "l"):
        assert key[name] == toy[name], name
    assert key["b"] == toy["b_g1"] and tuple(key["densities"]) == tuple(toy["densities"])
    assert key["a"] == [x for x in toy["a"] if x]                  # bellman drops zero inputs from a too
    assert key["ok"] == all(toy["l"])


@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_model_keys_give_verifying_proofs(nc, ni, na):
    rng = random.Random(nc * 17 + ni + na)
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30))
    sc = _scalars(rng)
    key = gs.as_prove_key(gs.generate(abc, circ.length, ni, na, sc[4], *sc[:4]))
    for j in range(2):
        inputs, aux = circ.witness(j)
        ev = circ.evaluations(inputs, aux)
        proof = gp.create_proof(key, *[gp.mont(e) for e in ev], gp.mont(inputs), gp.mont(aux), key["densities"],
                                bm.fr_to_mont(rng.randrange(R)), bm.fr_to_mont(rng.randrange(R)))
        assert gp.verifies(key, inputs, proof)
        assert not gp.verifies(key, inputs, (proof[0], proof[1], proof[2] + 1))


def test_csr_helper_keeps_the_sums():
    circ = gp.ToyCircuit(20, 3, 30, 4)
    plain, dup = gs.csr_from_cons(circ.all_cons, 33), gs.csr_from_cons(circ.all_cons, 33, seed=9)
    for (o0, c0, k0), (o1, c1, k1) in zip(plain, dup):
        assert o0[0] == 0 and o0[-1] == len(c0) and np.all(np.diff(o0.astype(np.int64)) >= 0) and k0.shape == (len(c0), 4)
        assert len(c1) > len(c0) and np.any(np.all(k1 == 0, axis=1))     # split terms and zero coefficients
    tau = 123456789
    assert gs.qap(plain, circ.length, 33, tau) == gs.qap(dup, circ.length, 33, tau)


def test_lagrange_at_a_domain_point_is_a_unit_vector():
    for log_n, k in ((0, 0), (3, 5), (5, 0)):
        tau = pow(fr_root(log_n), k, R)
        lag = gs.lagrange(log_n, tau)
        assert lag == [1 if q == k else 0 for q in range(1 << log_n)]


def _sizes_program():
    return r'''
#include <stddef.h>
#include <stdio.h>
#include "pairing_b200.h"
int main() {
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(bls_r1cs_matrix), offsetof(bls_r1cs_matrix, nnz), sizeof(bls_groth16_vk_points),
         offsetof(bls_groth16_vk_points, gamma_g2), sizeof(bls_groth16_parameters_out), offsetof(bls_groth16_parameters_out, lens),
         offsetof(bls_groth16_parameters_out, b_g2));
  return 0;
}
'''


def test_struct_layouts_match_the_bindings():
    import pairing_b200._native as nat
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(src, "w").write(_sizes_program())
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, src])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    want = [ctypes.sizeof(nat.R1csMatrixC), nat.R1csMatrixC.nnz.offset, ctypes.sizeof(nat.Groth16VkPointsC), nat.Groth16VkPointsC.gamma_g2.offset,
            ctypes.sizeof(nat.Groth16ParametersOutC), nat.Groth16ParametersOutC.lens.offset, nat.Groth16ParametersOutC.b_g2.offset]
    assert got == want
    assert nat.W_VK_POINTS == 3 * W1 + 3 * W2


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_groth16_generate_parameters_batch(None, None, 4, 1, 0, *[None] * 8) == -1
    assert lib.bls_groth16_generate_parameters_dev(None, None, 4, 1, 0, *[None] * 10) == -1
    assert lib.bls_groth16_generate_parameters_scratch_bytes(None, None, 4, 1, 0) == 0


def test_setup_kernels_do_not_spill():
    """the new kernels keep their state in registers: no local memory and no stack (cuobjdump --dump-resource-usage)"""
    import shutil
    import pairing_b200._native as nat
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(nat.LIB_PATH):
        pytest.skip("cuobjdump or the built library not available")
    out = subprocess.check_output([exe, "--dump-resource-usage", nat.LIB_PATH], text=True)
    usage, name = {}, None
    for line in out.splitlines():
        if "Function " in line:
            name = line.split("Function ")[1].rstrip(":").strip()
        elif "REG:" in line and name:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL|SHARED):(\d+)", line)}
    for kernel in ("k_gs_pre", "k_gs_tau_tables", "k_gs_powers", "k_gs_qap", "k_gs_query", "k_gs_scan", "k_gs_emit"):
        found = [v for k, v in usage.items() if kernel in k]
        assert len(found) == 1, (kernel, sorted(usage))
        assert found[0]["LOCAL"] == 0 and found[0]["STACK"] == 0, (kernel, found[0])


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", SHAPES)
@pytest.mark.parametrize("bases", ["generators", "multiples"])
def test_toy_keys_are_bit_exact(ctx, nc, ni, na, bases):
    rng = random.Random(nc * 1000 + ni * 100 + na + (bases == "multiples"))
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
    sc = _scalars(rng)
    t1, t2 = (1, 1) if bases == "generators" else (rng.randrange(2, R), rng.randrange(2, R))
    got = _call(ctx, abc, circ.length, ni, na, sc, _points(False, [t1])[0], _points(True, [t2])[0])
    _assert_key(got, gs.generate(abc, circ.length, ni, na, sc[4], *sc[:4]), t1, t2)


def _verify_all(ctx, params, proofs, inputs):
    pvk = ctx.groth16_prepare_verifying_key(params.alpha_g1, params.beta_g2, params.gamma_g2, params.delta_g2)
    return ctx.groth16_verify(pvk, params.ic, proofs, inputs), ctx.groth16_verify_rlc(pvk, params.ic, proofs, inputs, _limbs(range(3, 3 + len(proofs))))


@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_generated_keys_prove_and_verify(ctx, nc, ni, na):
    rng = random.Random(nc * 7 + ni * 3 + na)
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30))
    sc = _scalars(rng)
    params = _call(ctx, abc, circ.length, ni, na, sc)
    key = gs.as_prove_key(gs.generate(abc, circ.length, ni, na, sc[4], *sc[:4]))
    m = 3
    wit = [circ.witness(j) for j in range(m)]
    evals = [circ.evaluations(*w) for w in wit]
    abc_ev = [np.stack([_mont_rows(e[q]) for e in evals]).reshape(m, circ.length, 4) for q in range(3)]
    inp = np.stack([_mont_rows(w[0]) for w in wit]).reshape(m, ni, 4)
    aux = np.stack([_mont_rows(w[1]) for w in wit]).reshape(m, na, 4)
    r, s = _mont_rows([rng.randrange(R) for _ in range(m)]), _mont_rows([rng.randrange(R) for _ in range(m)])
    proofs = np.concatenate(ctx.groth16_prove(params, *abc_ev, inp, aux, params.densities, r, s), axis=1)
    for j in range(m):
        e = gp.create_proof(key, *[_ints(x[j]) for x in abc_ev], _ints(inp[j]), _ints(aux[j]), key["densities"], _ints(r[j])[0], _ints(s[j])[0])
        want = np.concatenate([_points(False, [e[0]]), _points(True, [e[1]]), _points(False, [e[2]])], axis=1)
        assert proofs[j].tobytes() == want[0].tobytes(), j
    pub = inp[:, 1:]
    ok, ok1 = _verify_all(ctx, params, proofs, pub)
    assert ok.all() and ok1
    for part, sl in (("A", slice(0, W1)), ("B", slice(W1, W1 + W2)), ("C", slice(W1 + W2, None))):
        bad = proofs.copy()
        bad[1, sl] = _points(part == "B", [777])[0]
        ok, ok1 = _verify_all(ctx, params, bad, pub)
        assert list(ok) == [True, False, True] and not ok1, part
    if ni > 1:
        bad_in = pub.copy()
        bad_in[0, 0] = _mont1(_ints(pub[0, :1])[0] + 1)
        ok, ok1 = _verify_all(ctx, params, proofs, bad_in)
        assert list(ok) == [False, True, True] and not ok1


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["zero", "domain_point", "domain_point_0"])
def test_degenerate_tau(ctx, which):
    ni, na = 3, 12
    circ, abc = _toy(12, ni, na, 77)
    log_n = domain_log(circ.length)
    tau = {"zero": 0, "domain_point": pow(fr_root(log_n), 5, R), "domain_point_0": 1}[which]
    sc = _scalars(random.Random(5), tau)
    got = _call(ctx, abc, circ.length, ni, na, sc)
    key = gs.generate(abc, circ.length, ni, na, sc[4], *sc[:4])
    _assert_key(got, key)
    if which != "zero":
        assert not any(key["h"])                                     # tau^n = 1: every h point is the identity
        assert key["lens"][0] < ni + na                              # a unit Lagrange vector filters heavily


@pytest.mark.gpu
def test_unconstrained_aux_gives_ok_0(ctx):
    circ = gp.ToyCircuit(12, 2, 6, 3)
    cons = [[{v: c for v, c in lc.items() if v != 2 + 6} for lc in con] for con in circ.all_cons]   # no term of the new aux 6
    abc = gs.csr_from_cons(cons, 2 + 7)
    sc = _scalars(random.Random(1))
    got = _call(ctx, abc, len(cons), 2, 7, sc)
    key = gs.generate(abc, len(cons), 2, 7, sc[4], *sc[:4])
    assert not key["ok"] and not got.ok
    _assert_key(got, key)


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [0, 1])
def test_domain_of_one_point(ctx, nc):
    ni, na = 1, 2
    cons = [[{0: 5, 1: 1}, {2: 3}, {1: 7, 2: 2}]][:nc]
    abc = gs.csr_from_cons(cons, ni + na, seed=3)
    sc = _scalars(random.Random(nc))
    got = _call(ctx, abc, nc, ni, na, sc)
    key = gs.generate(abc, nc, ni, na, sc[4], *sc[:4])
    assert len(got.h) == 0
    _assert_key(got, key)


# ---- full size: a seeded random circuit built in CSR, with a witness, in the layout KeypairAssembly records

def random_circuit(log_c, ni, seed):
    """2^log_c constraints (the ni input constraints included) over ni inputs and about as many aux variables: constraint q
    has ~3 terms in A and B (ONE in about half of them) and C = (A.z)(B.z) through a fresh aux variable o_q with coefficient
    c_q, so the witness z satisfies every constraint.  Returns abc (CSR triples), num_aux, the witness (inputs, aux) and the
    evaluations a, b, c (canonical ints)."""
    rng = np.random.default_rng(seed)
    nc = 1 << log_c
    nq = nc - ni
    na = nq
    nv = ni + na
    pool = [int(x) for x in rng.integers(1, 2 ** 62, 64)] + [1, R - 1]
    z = [1] + [int(x) for x in rng.integers(1, 2 ** 62, ni - 1)]
    z += [0] * na
    terms = [[], [], []]             # (variable, constraint, coefficient) per matrix
    evals = [[0] * nc for _ in range(3)]
    var = rng.integers(0, ni, size=(nq, 2, 3))
    prev = rng.random((nq, 2, 3))
    has_one = rng.random((nq, 2)) < 0.25
    cidx = rng.integers(0, len(pool), size=(nq, 2, 3))
    for q in range(nq):
        o_q = ni + q
        for k in range(2):
            s = 0
            for t in range(3):
                v = 0 if (t == 0 and has_one[q, k]) else (int(var[q, k, t]) if q < 8 or prev[q, k, t] < 0.3 else ni + int(prev[q, k, t] * q) % q)
                c = pool[cidx[q, k, t]]
                terms[k].append((v, q, c))
                s += c * z[v]
            evals[k][q] = s % R
        cq = pool[cidx[q, 0, 0]]
        z[o_q] = evals[0][q] * evals[1][q] * pow(cq, -1, R) % R
        terms[2].append((o_q, q, cq))
        evals[2][q] = evals[0][q] * evals[1][q] % R
    for i in range(ni):                                             # bellman's input_i * 0 = 0
        terms[0].append((i, nq + i, 1))
        evals[0][nq + i] = z[i]
    abc = []
    for k in range(3):
        t = np.array([(v, q) for v, q, _ in terms[k]], dtype=np.int64).reshape(-1, 2)
        order = np.argsort(t[:, 0], kind="stable")
        offsets = np.zeros(nv + 1, dtype=np.uint64)
        offsets[1:] = np.cumsum(np.bincount(t[:, 0], minlength=nv))
        coeff = _limbs([bm.fr_to_mont(terms[k][i][2]) for i in order])
        abc.append((offsets, t[order, 1].astype(np.uint32), coeff))
    return abc, na, (z[:ni], z[ni:]), evals


def _points_gpu(ctx, g2, exps):
    """[e]g through bls_g*_mul_batch (pinned to the oracle by its own tests), affine rows"""
    if not exps:
        return np.zeros((0, W2 if g2 else W1), dtype=np.uint64)
    from_aff = o.g2_from_affine if g2 else o.g1_from_affine
    g = np.repeat(from_aff(o.generators()[1 if g2 else 0]), len(exps), 0)
    k = _limbs([e % R for e in exps])
    return ctx.g2_into_affine(ctx.g2_mul(g, k)) if g2 else ctx.g1_into_affine(ctx.g1_mul(g, k))


@pytest.mark.gpu
def test_full_size_2_20_generate_prove_verify(ctx):
    ni = 4
    abc, na, (inputs, aux), evals = random_circuit(20, ni, 2020)
    nc = 1 << 20
    sc = _scalars(random.Random(11))
    got = _call(ctx, abc, nc, ni, na, sc)
    key = gs.generate(abc, nc, ni, na, sc[4], *sc[:4])
    assert got.ok and key["ok"]
    _assert_key(got, key, points=lambda g2, e: _points_gpu(ctx, g2, e))
    m = 4
    abc_ev = [np.broadcast_to(_mont_rows(e), (m, nc, 4)).copy() for e in evals]
    inp = np.broadcast_to(_mont_rows(inputs), (m, ni, 4)).copy()
    ax = np.broadcast_to(_mont_rows(aux), (m, na, 4)).copy()
    rng = random.Random(3)
    r, s = _mont_rows([rng.randrange(R) for _ in range(m)]), _mont_rows([rng.randrange(R) for _ in range(m)])
    proofs = np.concatenate(ctx.groth16_prove(got, *abc_ev, inp, ax, got.densities, r, s), axis=1)
    ok, ok1 = _verify_all(ctx, got, proofs, inp[:, 1:])
    assert ok.all() and ok1
    bad = proofs.copy()
    bad[2, W1 + W2:] = proofs[1, W1 + W2:]
    ok, ok1 = _verify_all(ctx, got, bad, inp[:, 1:])
    assert list(ok) == [True, True, False, True] and not ok1


def _one_heavy(nc, nv, concentrated):
    """nc terms per matrix: all on ONE (concentrated) or spread evenly over the nv variables"""
    rng = np.random.default_rng(nc)
    var = np.zeros(nc, dtype=np.int64) if concentrated else np.arange(nc) % nv
    order = np.argsort(var, kind="stable")
    offsets = np.zeros(nv + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(np.bincount(var, minlength=nv))
    cons = rng.permutation(nc).astype(np.uint32)[order]
    coeff = _limbs([bm.fr_to_mont(int(x)) for x in rng.integers(1, 2 ** 62, nc)])
    return [(offsets, cons, coeff)] * 3


def _dev_abc(abc):
    import torch
    return [(torch.from_numpy(off.view(np.int64)).cuda(), torch.from_numpy(c.view(np.int32)).cuda(), torch.from_numpy(k.view(np.int64)).cuda())
            for off, c, k in abc]


@pytest.mark.gpu
def test_terms_on_one_variable_are_correct_and_not_slow(ctx):
    """ONE in every constraint of A, B and C (and 2^16 - 1 variables without terms after it) against the same number of terms
    spread evenly over the variables: k_gs_qap, timed alone by the profiler, takes less than twice as long, and the key of
    the concentrated circuit is bit-exact"""
    import torch
    from pairing_b200.device import DeviceEngine
    nc, ni, na = 1 << 18, 1, (1 << 16) - 1
    sc = _scalars(random.Random(2))
    g1, g2 = o.generators()
    eng = DeviceEngine(ctx)
    times = {}
    for conc in (False, True, False, True):
        abc = _one_heavy(nc, ni + na, conc)
        dabc = _dev_abc(abc)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            got = eng.groth16_generate_parameters(dabc, nc, ni, na, g1[0], g2[0], *[_mont1(x) for x in sc])
            torch.cuda.synchronize()
        qap = sum(ev.self_device_time_total for ev in prof.key_averages() if "k_gs_qap" in ev.key)
        assert qap > 0
        times.setdefault(conc, []).append(qap)
    key = gs.generate(abc, nc, ni, na, sc[4], *sc[:4])
    host = type("K", (), {})()
    for name in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "gamma_g2", "delta_g2", "h", "ic", "l", "a", "b_g1", "b_g2"):
        setattr(host, name, getattr(got, name).cpu().numpy().view(np.uint64))
    host.densities, host.ok = got.densities, got.ok
    _assert_key(host, key, points=lambda g2_, e: _points_gpu(ctx, g2_, e))
    assert min(times[True]) < 2 * min(times[False]), times


@pytest.mark.gpu
def test_host_dev_engine_and_cpp_agree(ctx):
    import torch
    from pairing_b200.device import DeviceEngine
    ni, na = 3, 40
    circ, abc = _toy(40, ni, na, 8, dup=True)
    sc = _scalars(random.Random(8))
    host = _call(ctx, abc, circ.length, ni, na, sc)
    eng = DeviceEngine(ctx)
    dabc = [(torch.from_numpy(off.view(np.int64)).cuda(), torch.from_numpy(c.view(np.int32)).cuda(), torch.from_numpy(k.view(np.int64)).cuda())
            for off, c, k in abc]
    g1, g2 = o.generators()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dev = eng.groth16_generate_parameters(dabc, circ.length, ni, na, g1[0], g2[0], *[_mont1(x) for x in sc])
    for name in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "gamma_g2", "delta_g2", "h", "ic", "l", "a", "b_g1", "b_g2"):
        assert getattr(dev, name).cpu().numpy().view(np.uint64).tobytes() == np.asarray(getattr(host, name)).tobytes(), name
    assert all(np.array_equal(x, y) for x, y in zip(dev.densities, host.densities)) and dev.ok == host.ok
    with tempfile.TemporaryDirectory() as d:
        inp = os.path.join(d, "in.bin")
        with open(inp, "wb") as f:
            f.write(np.array([circ.length, ni, na], dtype=np.uint64).tobytes())
            for off, c, k in abc:
                f.write(np.array([len(c)], dtype=np.uint64).tobytes() + off.tobytes() + c.tobytes() + k.tobytes())
            f.write(np.concatenate([g1[0], g2[0]] + [_mont1(x) for x in sc]).astype(np.uint64).tobytes())
        exe = os.path.join(d, "setup")
        import pairing_b200._native as nat
        libdir = os.path.dirname(nat.LIB_PATH)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe,
                               os.path.join(ROOT, "tests", "cpp", "test_groth16_setup.cpp"), "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        out = os.path.join(d, "out.bin")
        subprocess.check_call([exe, inp, out])
        want = np.concatenate([np.asarray(getattr(host, q), dtype=np.uint64).reshape(-1) for q in
                               ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "gamma_g2", "delta_g2", "ic", "h", "l", "a", "b_g1", "b_g2")])
        assert open(out, "rb").read() == want.tobytes()


@pytest.mark.gpu
def test_invalid_arguments(ctx):
    import pairing_b200._native as nat
    ni, na = 2, 5
    circ, abc = _toy(8, ni, na, 1)
    sc = _scalars(random.Random(4))
    g1, g2 = o.generators()
    inf1, inf2 = g1[0].copy(), g2[0].copy()
    inf1[-1] = inf2[-1] = 1

    def rejects(abc_, nc=circ.length, ni_=ni, na_=na, sc_=sc, g1_=g1[0], g2_=g2[0]):
        with pytest.raises(nat.BlsError, match="invalid"):
            _call(ctx, abc_, nc, ni_, na_, sc_, g1_, g2_)

    for i in (2, 3):                                            # gamma = 0, delta = 0
        rejects(abc, sc_=[0 if j == i else x for j, x in enumerate(sc)])
    rejects(abc, g1_=inf1)
    rejects(abc, g2_=inf2)
    for k in range(3):
        off, cons, coeff = abc[k]
        if len(cons) == 0:
            continue
        bad_off = off.copy(); bad_off[0] = 1
        rejects([x if j != k else (bad_off, cons, coeff) for j, x in enumerate(abc)])
        bad_off = off.copy(); bad_off[1], bad_off[2] = off[2] + 1, off[2]
        rejects([x if j != k else (bad_off, cons, coeff) for j, x in enumerate(abc)])
        bad_c = cons.copy(); bad_c[0] = circ.length
        rejects([x if j != k else (off, bad_c, coeff) for j, x in enumerate(abc)])
        bad_k = coeff.copy(); bad_k[0] = _limbs([R])[0]
        rejects([x if j != k else (off, cons, bad_k) for j, x in enumerate(abc)])
    keep, mats = nat.r1cs_matrices(abc, circ.length, ni + na)
    lib = nat.load()
    assert lib.bls_groth16_generate_parameters_scratch_bytes(ctx._ctx, mats, circ.length, ni, na) > 0
    assert lib.bls_groth16_generate_parameters_scratch_bytes(ctx._ctx, mats, (1 << 26) + 1, ni, na) == 0    # n > 2^26
    assert lib.bls_groth16_generate_parameters_scratch_bytes(ctx._ctx, mats, circ.length, 1 << 26, na) == 0  # too many variables
    # _dev: an out-of-range constraint index is not checked up front; it contributes zero and sets ok = 0
    import torch
    from pairing_b200.device import DeviceEngine
    off, cons, coeff = abc[0]
    bad_c = cons.copy(); bad_c[0] = 1 << 30
    dabc = [(torch.from_numpy(o_.view(np.int64)).cuda(), torch.from_numpy(c.view(np.int32)).cuda(), torch.from_numpy(k.view(np.int64)).cuda())
            for o_, c, k in [(off, bad_c, coeff)] + abc[1:]]
    dev = DeviceEngine(ctx).groth16_generate_parameters(dabc, circ.length, ni, na, g1[0], g2[0], *[_mont1(x) for x in sc])
    assert not dev.ok
