"""Groth16 verification (bls_groth16_prepare_verifying_key, bls_groth16_verify_* and bls_groth16_verify_rlc_*, their Context,
DeviceEngine and C++ bindings).

Every point is [e]g for a known exponent e, so the verdict of any proof, honest, tampered or built from arbitrary exponents,
is known from tests/groth16_verify_model.py: every verdict the GPU returns is compared with the model's."""
import ctypes
import os
import random
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import bls_model as bm
import groth16_prove_model as gp
import groth16_verify_model as gv
import oracle_lib as o
from test_gpu_groth16_prove import SHAPES, Toy, _ints, _proof

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER
W1, W2, WP, W12 = 13, 25, 51, 72


def _limbs(values):
    return np.array([bm.limbs64(v % (1 << 256), 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _mont(values):
    return _limbs([bm.fr_to_mont(x % R) for x in values])


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_model_agrees_with_the_prover_model(nc, ni, na):
    """the prover model's proofs verify in the verifier model (ic_0 carries bellman's leading one); every tampering is
    caught; the randomized verdict is 1 for valid proofs, 0 with one invalid proof and random rho, and 1 for two errors
    that cancel under the chosen rho"""
    rng = random.Random(nc * 1000 + ni * 100 + na)
    circuit = gp.ToyCircuit(nc, ni, na, rng.randrange(1 << 30))
    key = circuit.setup(*[rng.randrange(1, R) for _ in range(5)])
    proofs, xs = [], []
    for w in range(3):
        inputs, aux = circuit.witness(w)
        a, b, c = circuit.evaluations(inputs, aux)
        p = gp.create_proof(key, gp.mont(a), gp.mont(b), gp.mont(c), gp.mont(inputs), gp.mont(aux), key["densities"],
                            gp.mont([rng.randrange(R)])[0], gp.mont([rng.randrange(R)])[0])
        assert gv.verifies(key, inputs[1:], p) == gp.verifies(key, inputs, p) is True
        proofs.append(p)
        xs.append(inputs[1:])
        ea, eb, ec = p
        for bad in ((ea + 1, eb, ec), (ea, eb + 1, ec), (ea, eb, ec + 1)):
            assert not gv.verifies(key, inputs[1:], bad)
        if xs[-1]:
            assert not gv.verifies(key, [xs[-1][0] + 1] + xs[-1][1:], p)
    rho = [rng.randrange(1, R) for _ in proofs]
    assert gv.rlc_verifies(key, xs, proofs, rho)
    bad = list(proofs)
    bad[1] = (bad[1][0], bad[1][1], bad[1][2] + 5)
    assert not gv.rlc_verifies(key, xs, bad, rho)
    assert gv.rlc_verifies(key, xs, bad, [rho[0], 0, rho[2]])            # rho_j = 0 leaves proof j out
    bad[2] = (bad[2][0], bad[2][1], (bad[2][2] - 5 * rho[1] * pow(rho[2], -1, R)) % R)
    assert gv.rlc_verifies(key, xs, bad, rho) and not gv.verifies(key, xs[2], bad[2])


def test_model_solvers():
    rng = random.Random(3)
    key = {"alpha": rng.randrange(R), "beta": rng.randrange(R), "gamma": rng.randrange(1, R), "delta": rng.randrange(1, R),
           "ic": [rng.randrange(1, R) for _ in range(4)]}
    x = [rng.randrange(R) for _ in range(3)]
    a, b = rng.randrange(R), rng.randrange(R)
    assert gv.verifies(key, x, (a, b, gv.solve_c(key, x, a, b)))
    assert gv.verifies(key, x, (a, gv.solve_b(key, x, a, 0), 0))
    z = gv.inputs_with_zero_acc(key, x)
    assert gv.acc(key, z) == 0 and z[1:] == x[1:]


def test_pvk_layout_matches_the_bindings():
    """sizeof / offsetof of bls_groth16_pvk equal the ctypes mirror, and both coefficient arrays are 16-byte aligned"""
    import pairing_b200._native as nat
    fields = ("neg_gamma_g2", "neg_delta_g2", "alpha_g1_beta_g2", "neg_gamma_g2_affine", "neg_delta_g2_affine")
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "pairing_b200.h"\nint main(){printf("%zu' + ' %zu' * len(fields) + '\\n",' \
          'sizeof(bls_groth16_pvk)' + ''.join(',offsetof(bls_groth16_pvk,%s)' % f for f in fields) + ');return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(c, "w").write(src)
        subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert got == [ctypes.sizeof(nat.Groth16PvkC)] + [getattr(nat.Groth16PvkC, f).offset for f in fields]
    assert got == [40176, 0, 19600, 39200, 39776, 39976]
    assert got[1] % 16 == 0 and got[2] % 16 == 0 and nat.W_PVK * 8 == 40176


def _resource_usage():
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
    return exe, nat.LIB_PATH, usage


def test_verify_kernels_resources_and_bulk_copy():
    """the new kernels' registers, stack and shared memory (DESIGN.md), no local memory, and the TMA bulk copies with their
    mbarrier in k_groth16_verify's SASS"""
    exe, lib, usage = _resource_usage()
    #               kernel                 max REG  max STACK  min SHARED
    limits = {"k_groth16_verify": (255, 6640, 2 * 19584),
              "k_g16v_scalars": (64, 0, 0), "k_g16v_rlc_sums": (64, 0, 256 * 32), "k_g16v_rlc_terms": (255, 472, 0),
              "k_g16v_rlc_pairs": (64, 0, 0), "k_g16v_rlc_compare": (64, 0, 0)}
    for kernel, (reg, stack, shared) in limits.items():
        found = [(k, v) for k, v in usage.items() if kernel in k]
        assert len(found) == 1, (kernel, sorted(usage))
        u = found[0][1]
        assert u["LOCAL"] == 0 and u["REG"] <= reg and u["STACK"] <= stack and u["SHARED"] >= shared, (kernel, u)
    name = [k for k in usage if "k_groth16_verify" in k][0]
    sass = subprocess.check_output([exe, "-sass", "-fun", name, lib], text=True)
    assert len(re.findall(r"\bUBLKCP\b", sass)) == 2 and "SYNCS" in sass


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_groth16_prepare_verifying_key(None, None, None, None, None, None) == -1
    assert lib.bls_groth16_verify_batch(None, None, None, 1, None, None, 1, None) == -1
    assert lib.bls_groth16_verify_dev(None, None, None, 1, None, None, 1, None, None, None) == -1
    assert lib.bls_groth16_verify_rlc_batch(None, None, None, 1, None, None, None, 1, None) == -1
    assert lib.bls_groth16_verify_rlc_dev(None, None, None, 1, None, None, None, 1, None, None, None) == -1
    assert lib.bls_groth16_verify_scratch_bytes(None, 1, 1) == 0
    assert lib.bls_groth16_verify_rlc_scratch_bytes(None, 1, 1) == 0


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def eng(ctx):
    from pairing_b200.device import DeviceEngine
    return DeviceEngine(ctx=ctx)


def _pts(ctx, g2, exps):
    """[e]g for every exponent as affine rows (e = 0: the identity), by double-and-add from the generator on the GPU"""
    exps = [e % R for e in exps]
    if not exps:
        return np.zeros((0, W2 if g2 else W1), dtype=np.uint64)
    gen = (o.g2_from_affine if g2 else o.g1_from_affine)(o.generators()[1 if g2 else 0])
    mul, into = (ctx.g2_mul, ctx.g2_into_affine) if g2 else (ctx.g1_mul, ctx.g1_into_affine)
    return into(mul(np.repeat(gen, len(exps), 0), _limbs(exps)))


class Vk:
    """a verifying key with known exponents, its points and its prepared form"""

    def __init__(self, ctx, ni, seed, key=None):
        rng = random.Random(seed)
        self.key = key or {"alpha": rng.randrange(1, R), "beta": rng.randrange(1, R), "gamma": rng.randrange(1, R),
                           "delta": rng.randrange(1, R), "ic": [rng.randrange(1, R) for _ in range(ni + 1)]}
        k = self.key
        g1 = _pts(ctx, False, [k["alpha"]] + k["ic"])
        self.alpha, self.ic = g1[0], g1[1:]
        self.beta, self.gamma, self.delta = _pts(ctx, True, [k["beta"], k["gamma"], k["delta"]])
        self.pvk = ctx.groth16_prepare_verifying_key(self.alpha, self.beta, self.gamma, self.delta)
        self.ni = len(k["ic"]) - 1

    def rows(self, ctx, exps):
        """proof rows (A, B, C) of the exponent triples"""
        if not exps:
            return np.zeros((0, WP), dtype=np.uint64)
        return np.concatenate([_pts(ctx, q == 1, [e[q] for e in exps]) for q in range(3)], axis=1)

    def model(self, xs, exps):
        return np.array([gv.verifies(self.key, x, e) for x, e in zip(xs, exps)], dtype=bool)


def _inputs(xs, ni):
    return (_mont([v for x in xs for v in x]) if ni else np.zeros((0, 4), np.uint64)).reshape(len(xs), ni, 4)


def _pvk_field(pvk, name):
    import pairing_b200._native as nat
    f = getattr(nat.Groth16PvkC, name)
    return pvk[f.offset // 8:(f.offset + f.size) // 8]


@pytest.mark.gpu
def test_pvk_is_bit_exact(ctx):
    """alpha_g1_beta_g2 = bls_pairing_batch(alpha, beta); the prepared parts = bls_g2_prepare_batch of -gamma, -delta (the
    oracle's points); the affine parts are those points; the pads are zero"""
    vk = Vk(ctx, 2, 0xAB)
    k = vk.key
    neg = o.g2_into_affine(o.g2_op("mul", np.repeat(o.g2_from_affine(o.generators()[1]), 2, 0),
                                   k=_limbs([-k["gamma"] % R, -k["delta"] % R]), threads=o.default_threads()))
    assert np.array_equal(_pvk_field(vk.pvk, "alpha_g1_beta_g2"), ctx.pairing(vk.alpha[None], vk.beta[None])[0])
    prep = ctx.g2_prepare(neg)
    assert np.array_equal(_pvk_field(vk.pvk, "neg_gamma_g2"), prep[0])
    assert np.array_equal(_pvk_field(vk.pvk, "neg_delta_g2"), prep[1])
    assert np.array_equal(_pvk_field(vk.pvk, "neg_gamma_g2_affine"), neg[0])
    assert np.array_equal(_pvk_field(vk.pvk, "neg_delta_g2_affine"), neg[1])
    assert _pvk_field(vk.pvk, "pad0")[0] == 0 and _pvk_field(vk.pvk, "pad1")[0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_prover_proofs_verify_and_tampered_ones_do_not(ctx, nc, ni, na):
    """proofs of bls_groth16_prove_batch on the prover tests' toy shapes, and the same proofs with A or C shifted by G, B of
    another proof, a changed public input, two proofs swapped: every verdict equals the model's"""
    m = 3
    toy = Toy(nc, ni, na, m, nc * 97 + ni * 13 + na)
    key = toy.key
    vk = Vk(ctx, ni - 1, 0, key={q: key[q] for q in ("alpha", "beta", "gamma", "delta", "ic")})
    got = _proof(toy.prove(ctx))
    exps = [gp.create_proof(key, *[_ints(x[j]) for x in toy.abc], _ints(toy.input[j]), _ints(toy.aux[j]), key["densities"],
                            _ints(toy.r[j])[0], _ints(toy.s[j])[0]) for j in range(m)]
    xs = [toy.witnesses[j][0][1:] for j in range(m)]
    rows, cases, cx = [got], list(exps), list(xs)
    tampered = [(exps[0][0] + 1, exps[0][1], exps[0][2]), (exps[1][0], exps[1][1], exps[1][2] + 1),
                (exps[2][0], exps[0][1], exps[2][2])]
    rows.append(vk.rows(ctx, tampered))
    cases += tampered
    cx += xs
    rows.append(got[::-1])                                                # swapped: proofs 2 and 0 with the inputs of 0 and 2
    cases += exps[::-1]
    cx += xs
    if ni > 1:
        rows.append(got[:1])
        cases.append(exps[0])
        cx.append([(xs[0][0] + 1) % R] + xs[0][1:])
    proofs = np.concatenate(rows)
    want = vk.model(cx, cases)
    assert want[:m].all() and not want[m + 1]                          # C + G never verifies (delta != 0)
    assert np.array_equal(ctx.groth16_verify(vk.pvk, vk.ic, proofs, _inputs(cx, ni - 1)), want)


def _dead_pair_cases(vk, rng):
    """exponent triples and inputs that verify (and their invalid neighbours) with A, B, C or acc_j at infinity"""
    k, ni = vk.key, vk.ni
    xs, exps = [], []
    for kind in ("a0", "b0", "c0", "acc0", "plain"):
        x = [rng.randrange(R) for _ in range(ni)]
        if kind == "acc0":
            if ni == 0:
                continue
            x = gv.inputs_with_zero_acc(k, x)
            assert gv.acc(k, x) == 0
        a, b = rng.randrange(1, R), rng.randrange(1, R)
        if kind == "a0":
            a = 0
        if kind == "b0":
            b = 0
        if kind == "c0":
            e = (a, gv.solve_b(k, x, a, 0), 0)
        else:
            e = (a, b, gv.solve_c(k, x, a, b))
        xs += [x, x]
        exps += [e, (e[0], e[1], (e[2] + 1) % R)]
    return xs, exps


@pytest.mark.gpu
@pytest.mark.parametrize("ni", [0, 1, 8])
def test_constructed_proofs_with_points_at_infinity(ctx, ni):
    """proofs solved from the equation with A, B, C or acc_j at infinity verify (each slot's dead-pair rule), a shifted C
    does not"""
    rng = random.Random(ni + 40)
    vk = Vk(ctx, ni, 0x1000 + ni)
    xs, exps = _dead_pair_cases(vk, rng)
    want = vk.model(xs, exps)
    assert list(want) == [True, False] * (len(exps) // 2)
    got = ctx.groth16_verify(vk.pvk, vk.ic, vk.rows(ctx, exps), _inputs(xs, ni))
    assert np.array_equal(got, want)


def _batch(ctx, vk, m, seed, pool=61):
    """m constructed proofs, about half invalid (c shifted, or a, b changed); the public inputs cycle through `pool` rows"""
    rng = random.Random(seed)
    k, ni = vk.key, vk.ni
    rows_x = [[rng.choice([0, 1, rng.randrange(R)]) for _ in range(ni)] for _ in range(pool)]
    acc = [gv.acc(k, x) for x in rows_x]
    ab = k["alpha"] * k["beta"]
    dinv = pow(k["delta"], -1, R)
    exps = []
    for j in range(m):
        a, b = rng.randrange(R), rng.randrange(R)
        c = (a * b - ab - k["gamma"] * acc[j % pool]) * dinv % R
        kind = rng.randrange(4)
        if kind == 1:
            c = (c + rng.randrange(1, R)) % R
        elif kind == 2:
            a = (a + 1) % R
        exps.append((a, b, c))
    xs = [rows_x[j % pool] for j in range(m)]
    pool_rows = _inputs(rows_x, ni)
    inputs = pool_rows[np.arange(m) % pool] if m else np.zeros((0, ni, 4), np.uint64)
    return xs, exps, vk.rows(ctx, exps), inputs


@pytest.mark.gpu
@pytest.mark.parametrize("ni", [1, 8])
def test_2_16_proofs_half_invalid(ctx, ni):
    vk = Vk(ctx, ni, 0x216 + ni)
    xs, exps, proofs, inputs = _batch(ctx, vk, 1 << 16, 0x5EED + ni)
    want = vk.model(xs, exps)
    assert 0.3 < want.mean() < 0.7
    assert np.array_equal(ctx.groth16_verify(vk.pvk, vk.ic, proofs, inputs), want)


@pytest.mark.gpu
@pytest.mark.parametrize("ni", [0, 1, 8, 64])
def test_ragged_batches(ctx, ni):
    vk = Vk(ctx, ni, 0x3A + ni)
    xs, exps, proofs, inputs = _batch(ctx, vk, (1 << 16) - 1, 0x77 + ni)
    want = vk.model(xs, exps)
    for m in (0, 1, 2, 63, 64, 65, 129, (1 << 16) - 1):
        assert np.array_equal(ctx.groth16_verify(vk.pvk, vk.ic, proofs[:m], inputs[:m]), want[:m]), m


CPP_VERIFY = r"""
#include <cstring>
#include <fstream>
#include "pairing_b200.hpp"
using namespace pairing_b200;
template <class T> std::vector<T> rd(std::ifstream& f) {
  uint64_t n; f.read(reinterpret_cast<char*>(&n), 8);
  std::vector<T> v(n / sizeof(T)); f.read(reinterpret_cast<char*>(v.data()), n);
  return v;
}
int main(int, char** argv) {
  Gpu gpu(0);
  std::ifstream f(argv[1], std::ios::binary);
  auto g1 = rd<G1AffinePoint>(f); auto g2 = rd<G2AffinePoint>(f); auto ic = rd<G1AffinePoint>(f);
  auto proofs = rd<Groth16::Proof>(f); auto inputs = rd<bls_fr>(f); auto rho = rd<bls_fr_repr>(f);
  auto pvk = Groth16::prepare_verifying_key(gpu, g1[0], g2[0], g2[1], g2[2]);
  std::vector<bool> ok = Groth16::verify_proof(gpu, *pvk, ic, proofs, inputs);
  const bool rlc = Groth16::verify_proofs_batch(gpu, *pvk, ic, proofs, inputs, rho);
  std::ofstream o(argv[2], std::ios::binary);
  o.write(reinterpret_cast<const char*>(pvk.get()), sizeof(Groth16::PreparedVerifyingKey));
  for (bool b : ok) o.put(b ? 1 : 0);
  o.put(rlc ? 1 : 0);
  return 0;
}
"""


@pytest.mark.gpu
def test_host_dev_engine_cpp_and_the_chain_agree(ctx, eng):
    """Context (host _batch), bls_groth16_verify_dev on a stream of its own, DeviceEngine, Groth16::verify_proof and the chain
    of existing calls (msm -> three Miller-loop calls -> Fq12 products -> final exponentiation -> compare) give the same
    verdicts; the same for the randomized check"""
    import torch
    import pairing_b200._native as nat
    ni = 3
    vk = Vk(ctx, ni, 0xC4A1)
    xs, exps, proofs, inputs = _batch(ctx, vk, 40, 0xC4A2, pool=7)
    d_xs, d_exps = _dead_pair_cases(vk, random.Random(9))
    xs, exps = xs + d_xs, exps + d_exps
    proofs, inputs = np.concatenate([proofs, vk.rows(ctx, d_exps)]), np.concatenate([inputs, _inputs(d_xs, ni)])
    m = len(exps)
    want = vk.model(xs, exps)
    host = ctx.groth16_verify(vk.pvk, vk.ic, proofs, inputs)
    assert np.array_equal(host, want)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to(eng.device)  # noqa: E731
    dpvk, dic, dpr, din = dev(vk.pvk), dev(vk.ic), dev(proofs), dev(inputs)
    assert np.array_equal(eng.groth16_verify(dpvk, dic, dpr, din).cpu().numpy().astype(bool), want)
    scratch = torch.empty(ctx.groth16_verify_scratch_bytes(ni, m), dtype=torch.uint8, device=eng.device)
    out = torch.zeros(m, dtype=torch.uint8, device=eng.device)
    st = torch.cuda.Stream(eng.device)
    st.wait_stream(torch.cuda.current_stream(eng.device))
    with torch.cuda.stream(st):
        ctx.call_dev("bls_groth16_verify_dev", dpvk.data_ptr(), dic.data_ptr(), ni, dpr.data_ptr(), din.data_ptr(), m, out.data_ptr(),
                     scratch.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert np.array_equal(out.cpu().numpy().astype(bool), want)
    # the randomized check over the valid proofs, host, engine and _dev
    rng = random.Random(5)
    good = np.flatnonzero(want)
    rho = _limbs([rng.randrange(1, R) for _ in good])
    assert ctx.groth16_verify_rlc(vk.pvk, vk.ic, proofs[good], inputs[good], rho)
    assert eng.groth16_verify_rlc(dpvk, dic, dev(proofs[good]), dev(inputs[good]), dev(rho)).item() == 1
    rho_all = _limbs([rng.randrange(1, R) for _ in range(m)])
    assert not ctx.groth16_verify_rlc(vk.pvk, vk.ic, proofs, inputs, rho_all)
    rscr = torch.empty(ctx.groth16_verify_rlc_scratch_bytes(ni, m), dtype=torch.uint8, device=eng.device)
    out1 = torch.full((1,), 7, dtype=torch.uint8, device=eng.device)
    with torch.cuda.stream(st):
        ctx.call_dev("bls_groth16_verify_rlc_dev", dpvk.data_ptr(), dic.data_ptr(), ni, dpr.data_ptr(), din.data_ptr(), dev(rho_all).data_ptr(), m,
                     out1.data_ptr(), rscr.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert out1.item() == 0
    # the C++ mirror: prepare_verifying_key, verify_proof, verify_proofs_batch
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe, fin, fout = (os.path.join(d, x) for x in ("v.cpp", "v", "in", "out"))
        open(src, "w").write(CPP_VERIFY)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        with open(fin, "wb") as f:
            for x in (vk.alpha[None], np.stack([vk.beta, vk.gamma, vk.delta]), vk.ic, proofs, inputs, rho_all):
                raw = np.ascontiguousarray(x).tobytes()
                f.write(np.uint64(len(raw)).tobytes() + raw)
        subprocess.check_call([exe, fin, fout], timeout=300)
        res = np.fromfile(fout, dtype=np.uint8)
    assert res[:40176].tobytes() == vk.pvk.tobytes()
    assert np.array_equal(res[40176:40176 + m].astype(bool), want) and res[-1] == 0
    # the chain of existing calls
    scal = np.concatenate([np.tile(_limbs([1]), (m, 1, 1)), _limbs([v for x in xs for v in x]).reshape(m, ni, 4)], axis=1)
    acc = ctx.g1_into_affine(ctx.g1_msm_batch(vk.ic, scal))
    ng = np.repeat(_pvk_field(vk.pvk, "neg_gamma_g2_affine")[None], m, 0)
    nd = np.repeat(_pvk_field(vk.pvk, "neg_delta_g2_affine")[None], m, 0)
    f = ctx.miller_loop(proofs[:, :W1], proofs[:, W1:W1 + W2])
    f = ctx.field_op(12, "mul", f, ctx.miller_loop(acc, ng))[0]
    f = ctx.field_op(12, "mul", f, ctx.miller_loop(proofs[:, W1 + W2:], nd))[0]
    fe, some = ctx.final_exponentiation(f)
    chain = (some != 0) & (fe == _pvk_field(vk.pvk, "alpha_g1_beta_g2")[None]).all(axis=1)
    assert np.array_equal(chain, want)


@pytest.mark.gpu
@pytest.mark.parametrize("at_infinity", ["gamma", "delta"])
def test_key_with_gamma_or_delta_at_infinity(ctx, at_infinity):
    """a key whose gamma (or delta) is the identity: its prepared point carries the infinity flag, the pair (acc_j, -gamma)
    (or (C_j, -delta)) contributes one, and both verdicts follow the model"""
    ni = 2
    rng = random.Random(0x1F + len(at_infinity))
    key = {"alpha": rng.randrange(1, R), "beta": rng.randrange(1, R), "gamma": rng.randrange(1, R), "delta": rng.randrange(1, R),
           "ic": [rng.randrange(1, R) for _ in range(ni + 1)]}
    key[at_infinity] = 0
    vk = Vk(ctx, ni, 0, key=key)
    assert _pvk_field(vk.pvk, "neg_%s_g2" % at_infinity)[-1] == 1
    xs, exps = [], []
    for j in range(8):
        x = [rng.randrange(R) for _ in range(ni)]
        a, c = rng.randrange(1, R), rng.randrange(R)
        b = gv.solve_b(key, x, a, c)
        xs.append(x)
        exps.append((a, b, c) if j % 2 == 0 else (a, (b + 1) % R, c))
    want = vk.model(xs, exps)
    assert list(want) == [True, False] * 4
    proofs, inputs = vk.rows(ctx, exps), _inputs(xs, ni)
    assert np.array_equal(ctx.groth16_verify(vk.pvk, vk.ic, proofs, inputs), want)
    rho = [rng.randrange(1, R) for _ in exps]
    for sel in (np.flatnonzero(want), np.arange(len(exps))):
        r = [rho[j] for j in sel]
        assert ctx.groth16_verify_rlc(vk.pvk, vk.ic, proofs[sel], inputs[sel], _limbs(r)) == \
            gv.rlc_verifies(key, [xs[j] for j in sel], [exps[j] for j in sel], r) == (len(sel) < len(exps))


@pytest.mark.gpu
def test_randomized_check(ctx):
    """all valid: 1; one invalid proof at 0, in the middle or at m - 1: 0; two invalid proofs whose errors cancel under the
    chosen rho: 1 as in the model; rho_j = 0 leaves an invalid proof out; m = 1 agrees with the per-proof verdict"""
    ni = 2
    vk = Vk(ctx, ni, 0x21C)
    k = vk.key
    rng = random.Random(0x21D)
    m = 33
    xs = [[rng.randrange(R) for _ in range(ni)] for _ in range(m)]
    exps = []
    for x in xs:
        a, b = rng.randrange(R), rng.randrange(R)
        exps.append((a, b, gv.solve_c(k, x, a, b)))
    inputs = _inputs(xs, ni)
    rho = [rng.randrange(1, R) for _ in range(m)]

    def run(ex, rh):
        want = gv.rlc_verifies(k, xs, ex, rh)
        got = ctx.groth16_verify_rlc(vk.pvk, vk.ic, vk.rows(ctx, ex), inputs, _limbs(rh))
        assert got == want
        return got

    assert run(exps, rho)
    for j in (0, m // 2, m - 1):
        bad = list(exps)
        bad[j] = (bad[j][0], bad[j][1], bad[j][2] + 1)
        assert not run(bad, rho), j
        zero = list(rho)
        zero[j] = 0
        assert run(bad, zero), j
    bad = list(exps)
    j1, j2, dlt = 3, 20, rng.randrange(1, R)
    bad[j1] = (bad[j1][0], bad[j1][1], (bad[j1][2] + dlt) % R)
    bad[j2] = (bad[j2][0], bad[j2][1], (bad[j2][2] - dlt * rho[j1] * pow(rho[j2], -1, R)) % R)
    assert not vk.model(xs, bad)[[j1, j2]].any()
    assert run(bad, rho)
    for j in (0, j1):
        one = ctx.groth16_verify_rlc(vk.pvk, vk.ic, vk.rows(ctx, [bad[j]]), inputs[j:j + 1], _limbs([rho[j]]))
        assert one == bool(ctx.groth16_verify(vk.pvk, vk.ic, vk.rows(ctx, [bad[j]]), inputs[j:j + 1])[0]) == (j == 0)


@pytest.mark.gpu
def test_invalid_arguments(ctx):
    """NULL pointers where there is work, the limits, a misaligned _dev pvk; m = 0 does nothing"""
    import torch
    lib, cx = ctx._lib, ctx._ctx
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    vk = Vk(ctx, 1, 0xBAD)
    proofs = vk.rows(ctx, [(1, 2, 3)])
    inputs, ok, rho = _mont([5]), np.zeros(1, np.uint8), _limbs([9])
    args = [p(vk.pvk), p(vk.ic), 1, p(proofs), p(inputs), 1, p(ok)]
    assert lib.bls_groth16_verify_batch(cx, *args) == 0
    for i in (0, 1, 3, 4, 6):
        a = list(args)
        a[i] = None
        assert lib.bls_groth16_verify_batch(cx, *a) == -1, i
        ra = a[:5] + [p(rho)] + a[5:]
        assert lib.bls_groth16_verify_rlc_batch(cx, *ra) == -1, i
    assert lib.bls_groth16_verify_rlc_batch(cx, *args[:5], None, *args[5:]) == -1
    a0 = list(args)
    a0[2], a0[4] = 0, None                                      # no inputs: inputs may be NULL
    assert lib.bls_groth16_verify_batch(cx, *a0) == 0
    # m = 0: nothing to do, every pointer may be NULL
    assert lib.bls_groth16_verify_batch(cx, None, None, 5, None, None, 0, None) == 0
    assert lib.bls_groth16_verify_rlc_batch(cx, None, None, 5, None, None, None, 0, None) == 0
    assert lib.bls_groth16_verify_dev(cx, None, None, 5, None, None, 0, None, None, None) == 0
    assert lib.bls_groth16_verify_scratch_bytes(cx, 5, 0) == 1
    # the empty randomized batch satisfies its equation (both sides are one): the verdict is 1
    ok0 = np.zeros(1, np.uint8)
    assert lib.bls_groth16_verify_rlc_batch(cx, None, None, 5, None, None, None, 0, p(ok0)) == 0 and ok0[0] == 1
    assert ctx.groth16_verify_rlc(vk.pvk, vk.ic, proofs[:0], np.zeros((0, 1, 4), np.uint64), np.zeros((0, 4), np.uint64)) is True
    # limits (checked before any pointer is used)
    assert lib.bls_groth16_verify_scratch_bytes(cx, 1, (1 << 16) + 1) == 0
    assert lib.bls_groth16_verify_scratch_bytes(cx, 63, 1 << 16) > 0
    assert lib.bls_groth16_verify_scratch_bytes(cx, 1 << 10, 1 << 16) == 0
    assert lib.bls_groth16_verify_batch(cx, None, None, 1, None, None, (1 << 16) + 1, None) == -1
    assert lib.bls_groth16_verify_rlc_scratch_bytes(cx, 1 << 26, 1) == 0
    assert lib.bls_groth16_verify_rlc_scratch_bytes(cx, 1, (1 << 26) + 1) == 0
    assert lib.bls_groth16_verify_rlc_batch(cx, None, None, 1, None, None, None, (1 << 26) + 1, None) == -1
    # a pvk that is not 16-byte aligned is rejected before any work
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to("cuda")  # noqa: E731
    raw = torch.zeros(40176 + 16, dtype=torch.uint8, device="cuda")
    dic, dpr, din, dok, drho = dev(vk.ic), dev(proofs), dev(inputs), torch.zeros(1, dtype=torch.uint8, device="cuda"), dev(rho)
    scr = torch.empty(ctx.groth16_verify_rlc_scratch_bytes(1, 1) + ctx.groth16_verify_scratch_bytes(1, 1), dtype=torch.uint8, device="cuda")
    for off, rc in ((8, -1), (0, 0)):
        raw[off:off + 40176].copy_(torch.from_numpy(vk.pvk.view(np.uint8)).to("cuda"))
        torch.cuda.synchronize()                                        # the calls below run on the context's own stream
        assert lib.bls_groth16_verify_dev(cx, raw.data_ptr() + off, dic.data_ptr(), 1, dpr.data_ptr(), din.data_ptr(), 1, dok.data_ptr(),
                                          scr.data_ptr(), None) == rc, off
        assert lib.bls_groth16_verify_rlc_dev(cx, raw.data_ptr() + off, dic.data_ptr(), 1, dpr.data_ptr(), din.data_ptr(), drho.data_ptr(), 1,
                                              dok.data_ptr(), scr.data_ptr(), None) == rc, off
    torch.cuda.synchronize()
    dev_args = [raw.data_ptr(), dic.data_ptr(), 1, dpr.data_ptr(), din.data_ptr(), 1, dok.data_ptr(), scr.data_ptr(), None]
    for i in (0, 1, 3, 4, 6, 7):
        a = list(dev_args)
        a[i] = None
        assert lib.bls_groth16_verify_dev(cx, *a) == -1, i
    rlc_args = dev_args[:5] + [drho.data_ptr()] + dev_args[5:]
    for i in (0, 1, 3, 4, 5, 7, 8):                                   # pvk, ic, proofs, inputs, rho, ok1, scratch
        a = list(rlc_args)
        a[i] = None
        assert lib.bls_groth16_verify_rlc_dev(cx, *a) == -1, i
    dok.zero_()
    torch.cuda.synchronize()
    assert lib.bls_groth16_verify_rlc_dev(cx, None, None, 1, None, None, None, 0, dok.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    assert dok.item() == 1
    assert lib.bls_groth16_prepare_verifying_key(cx, p(vk.alpha), p(vk.beta), None, p(vk.delta), p(np.zeros(5022, np.uint64))) == -1
    with pytest.raises(ValueError):
        ctx.groth16_verify(vk.pvk, vk.ic, proofs, np.zeros((1, 2, 4), np.uint64))
    with pytest.raises(ValueError):
        ctx.groth16_verify_rlc(vk.pvk, vk.ic, proofs, inputs.reshape(1, 1, 4), np.zeros((2, 4), np.uint64))
