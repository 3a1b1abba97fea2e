"""Phase 2 of the Groth16 ceremony (bls_groth16_mpc_new_batch / _dev, Context.groth16_mpc_new, DeviceEngine.groth16_mpc_new),
declared in include/pairing_b200_mpc.h.

Every transcript row is [e]g for an exponent e of tests/groth16_mpc_model.py, so a key is compared bit for bit with the
model's exponents on the generators, and with bls_groth16_generate_parameters_batch for (alpha, beta, gamma = 1, delta = 1,
tau), which an honest transcript must reproduce byte for byte."""
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
import groth16_mpc_model as mm
import groth16_prove_model as gp
import groth16_setup_model as gs
import oracle_lib as o
from fr_fft_model import fr_root
from groth16_h_model import domain_log
from test_gpu_dev_contract import Case, _out, run_dev
from test_gpu_groth16_prove import SHAPES, W1, W2, _limbs, _mont_rows, _points
from test_gpu_groth16_setup import _assert_key, _dev_abc, _expect, _mont1, _one_heavy, _points_gpu, _toy, _verify_all, random_circuit
from test_gpu_kzg import _resource_usage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pairing_b200_mpc.h")
R = bm.R_ORDER
KEY_ROWS = ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "gamma_g2", "delta_g2", "h", "ic", "l", "a", "b_g1", "b_g2")


def _header_functions():
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(bls_[a-z0-9_]+)\s*\(", src))), src


def _phase1(ctx, ph, points=None):
    """a Groth16Phase1 of affine rows from the model's exponents"""
    import pairing_b200._native as nat
    pts = points or (lambda g2, e: _points(g2, e))
    one = lambda g2, e: pts(g2, [e])[0]                                                   # noqa: E731
    return nat.Groth16Phase1(one(False, ph["alpha_g1"]), one(False, ph["beta_g1"]), one(True, ph["beta_g2"]), pts(False, ph["coeffs_g1"]),
                             pts(False, ph["alpha_coeffs_g1"]), pts(False, ph["beta_coeffs_g1"]), pts(True, ph["coeffs_g2"]), pts(False, ph["h"]))


def _gens():
    g1, g2 = o.generators()
    return g1[0], g2[0]


def _generate(ctx, abc, nc, ni, na, alpha, beta, tau):
    return ctx.groth16_generate_parameters(abc, nc, ni, na, *_gens(), *[_mont1(x) for x in (alpha, beta, 1, 1, tau)])


def _same_key(got, want):
    for name in KEY_ROWS:
        g, w = (np.ascontiguousarray(getattr(k, name).cpu() if hasattr(getattr(k, name), "cpu") else getattr(k, name)) for k in (got, want))
        assert g.view(np.uint64).tobytes() == w.view(np.uint64).tobytes(), name
    for d, w in zip(got.densities, want.densities):
        assert list(d) == list(w)
    assert got.ok == want.ok


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_model_new_is_generate_with_gamma_delta_one(nc, ni, na):
    rng = random.Random(nc * 131 + ni * 7 + na)
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
    alpha, beta, tau = (rng.randrange(1, R) for _ in range(3))
    key = mm.new(abc, circ.length, ni, na, mm.transcript(circ.length, tau, alpha, beta))
    want = gs.generate(abc, circ.length, ni, na, tau, alpha, beta, 1, 1)
    for name in ("alpha", "beta", "gamma", "delta", "h", "ic", "l", "a", "b", "densities", "lens", "ok"):
        assert key[name] == want[name], name
    assert key["b_g2"] == key["b"]


def test_header_symbols_are_bound_and_exported():
    import pairing_b200._native as nat
    lib = nat.load()
    names, _ = _header_functions()
    assert names == sorted(nat.MPC_SYMBOLS)
    assert not set(names) & set(nat.SYMBOLS)
    out = subprocess.check_output(["nm", "-D", "--defined-only", nat.LIB_PATH], text=True)
    assert set(names) <= set(re.findall(r" T (bls_[a-z0-9_]+)", out))
    for n in names:
        assert hasattr(lib, n)


def test_every_scratch_entry_point_of_the_header_has_a_contract_case():
    _, src = _header_functions()
    decls = re.findall(r"\bint\s+(bls_\w+_dev)\s*\(([^;]*)\)\s*;", src)
    scratch_dev = {name for name, params in decls if re.search(r"void\s*\*\s*scratch\b", params)}
    sizers = set(re.findall(r"\bsize_t\s+(bls_\w+_scratch_bytes)\s*\(", src))
    assert scratch_dev == {fn for fn, _ in CONTRACT_CASES} and sizers == {sb for _, sb in CONTRACT_CASES}


def test_struct_layouts_match_the_bindings():
    import pairing_b200._native as nat
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "pairing_b200_mpc.h"
int main() {
  printf("%zu %zu %zu %zu %zu %zu\n", sizeof(bls_groth16_phase1), offsetof(bls_groth16_phase1, beta_g2), offsetof(bls_groth16_phase1, coeffs_g1),
         offsetof(bls_groth16_phase1, coeffs_g2), offsetof(bls_groth16_phase1, h), offsetof(bls_groth16_phase1, n));
  return 0;
}
'''
    with tempfile.TemporaryDirectory() as d:
        path, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(path, "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, path])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    C = nat.Groth16Phase1C
    assert got == [ctypes.sizeof(C), C.beta_g2.offset, C.coeffs_g1.offset, C.coeffs_g2.offset, C.h.offset, C.n.offset]
    src2 = src.replace('printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(bls_groth16_phase1), offsetof(bls_groth16_phase1, beta_g2), offsetof(bls_groth16_phase1, coeffs_g1),\n         offsetof(bls_groth16_phase1, coeffs_g2), offsetof(bls_groth16_phase1, h), offsetof(bls_groth16_phase1, n));',
                       'printf("%zu %zu %zu %zu %zu\\n", sizeof(bls_groth16_mpc_pubkey), offsetof(bls_groth16_mpc_pubkey, r), sizeof(bls_groth16_key), offsetof(bls_groth16_key, ic), offsetof(bls_groth16_key, ic_len));')
    assert src2 != src
    with tempfile.TemporaryDirectory() as d:
        path, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(path, "w").write(src2)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, path])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    K = nat.Groth16KeyC
    assert got == [8 * nat.W_MPC_PUBKEY, 8 * 3 * W1, ctypes.sizeof(K), K.ic.offset, K.ic_len.offset]


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_groth16_mpc_new_batch(None, None, 4, 1, 0, None, None, None, None) == -1
    assert lib.bls_groth16_mpc_new_dev(None, None, 4, 1, 0, None, None, None, None, None, None) == -1
    assert lib.bls_groth16_mpc_new_scratch_bytes(None, None, 4, 1, 0) == 0
    assert lib.bls_groth16_mpc_contribute_batch(None, *[None] * 5, 0, None, 0, None, None, None) == -1
    assert lib.bls_groth16_mpc_contribute_dev(None, *[None] * 5, 0, None, 0, None, None, None, None, None) == -1
    assert lib.bls_groth16_mpc_contribute_scratch_bytes(None, 1, 1) == 0
    assert lib.bls_groth16_mpc_verify_batch(None, None, None, None, 0, None, None, None) == -1
    assert lib.bls_groth16_mpc_verify_dev(None, None, None, None, 0, None, None, None, None, None) == -1
    assert lib.bls_groth16_mpc_verify_scratch_bytes(None, None, None, 0) == 0


def test_mpc_kernels_resources():
    """the new kernels use no local memory and no shared memory, and stay within DESIGN.md's registers and stack"""
    _, _, usage = _resource_usage()
    #        kernel (G1 = Fp, G2 = Fp2)          max REG  max STACK
    limits = {"k_mpc_qapIN3bls2Fp": (128, 6144, 0), "k_mpc_qapIN3bls3Fp2": (168, 8448, 0), "k_mpc_fixIN3bls2Fp": (255, 512, 0),
              "k_mpc_fixIN3bls3Fp2": (255, 1536, 0), "k_mpc_loadIN3bls2Fp": (96, 0, 0), "k_mpc_loadIN3bls3Fp2": (96, 0, 0),
              "k_mpc_combine": (255, 512, 0), "k_mpc_prepIN3bls2Fp": (96, 0, 0), "k_mpc_prepIN3bls3Fp2": (96, 0, 0),
              "k_mpc_emitIN3bls2Fp": (96, 0, 0), "k_mpc_emitIN3bls3Fp2": (96, 0, 0), "k_mpcv_diff": (64, 0, 0), "k_mpcv_pairs": (96, 0, 0),
              "k_mpcv_finish": (64, 0, 2048)}
    for kernel, (reg, stack, shared) in limits.items():
        found = [v for k, v in usage.items() if kernel + ("E" if "IN3bls" in kernel else "") in k]
        assert len(found) == 1, (kernel, sorted(k for k in usage if "k_mpc" in k))
        u = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL|SHARED):(\d+)", found[0])}
        assert u["LOCAL"] == 0 and u["SHARED"] <= shared and u["REG"] <= reg and u["STACK"] <= stack, (kernel, u)
    assert len([k for k in usage if "k_mpc" in k]) == len(limits)


def test_preexisting_kernels_resources_unchanged():
    """every kernel the library had before phase 2 keeps its cuobjdump --dump-resource-usage line
    (tests/golden/resource_usage_pre_mpc.txt: the dump of the parent commit's build)"""
    _, _, usage = _resource_usage()
    before = dict(line.split(" ", 1) for line in open(os.path.join(ROOT, "tests", "golden", "resource_usage_pre_mpc.txt")).read().splitlines())
    assert len(before) >= 110 and any("k_pfft_" in k for k in before) and any("k_gs_qap" in k for k in before)
    changed = {k: (v, usage.get(k)) for k, v in before.items() if usage.get(k) != v}
    assert not changed, changed


# ---------------------------------------------------------------------------------------------------------------- GPU

def _check_new(ctx, abc, nc, ni, na, alpha, beta, tau):
    ph = mm.transcript(nc, tau, alpha, beta)
    got = ctx.groth16_mpc_new(abc, nc, ni, na, _phase1(ctx, ph), *_gens())
    _assert_key(got, mm.new(abc, nc, ni, na, ph))
    _same_key(got, _generate(ctx, abc, nc, ni, na, alpha, beta, tau))
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_new_is_generate_parameters_byte_for_byte(ctx, nc, ni, na):
    rng = random.Random(nc * 1000 + ni * 100 + na)
    circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
    _check_new(ctx, abc, circ.length, ni, na, *(rng.randrange(1, R) for _ in range(3)))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["zero", "domain_point", "domain_point_0"])
def test_degenerate_tau(ctx, which):
    ni, na = 3, 12
    circ, abc = _toy(12, ni, na, 77)
    tau = {"zero": 0, "domain_point": pow(fr_root(domain_log(circ.length)), 5, R), "domain_point_0": 1}[which]
    _check_new(ctx, abc, circ.length, ni, na, 11, 13, tau)


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [0, 1])
def test_domain_of_one_point(ctx, nc):
    ni, na = 1, 2
    cons = [[{0: 5, 1: 1}, {2: 3}, {1: 7, 2: 2}]][:nc]
    abc = gs.csr_from_cons(cons, ni + na, seed=3)
    got = _check_new(ctx, abc, nc, ni, na, 5, 6, 7)
    assert len(got.h) == 0


def _classes_circuit(nc, ni, na, seed):
    """every constraint's A, B and C over random variables with coefficients from one class each: random, +-1, +-2^k, r - 1,
    zero, and a variable repeated in one constraint"""
    rng = random.Random(seed)
    nv = ni + na
    pick = [lambda: rng.randrange(R), lambda: rng.choice([1, R - 1]), lambda: (rng.choice([1, -1]) * (1 << rng.randrange(1, 255))) % R,
            lambda: R - 1, lambda: 0, lambda: rng.choice([2, R - 2, 3])]
    cons = []
    for q in range(nc):
        con = []
        for _ in range(3):
            lc = {}
            for _ in range(rng.randrange(1, 5)):
                lc[rng.randrange(nv)] = pick[rng.randrange(len(pick))]()
            con.append(lc)
        cons.append(con)
    for i in range(ni):                                               # bellman's input_i * 0 = 0
        cons.append([{i: 1}, {}, {}])
    abc = gs.csr_from_cons(cons, nv, seed=seed)                       # split terms and zero terms: repeated (variable, constraint)
    return abc, len(cons)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_coefficient_classes(ctx, seed):
    abc, nc = _classes_circuit(40, 3, 40, seed)
    _check_new(ctx, abc, nc, 3, 40, 17, 19, random.Random(seed).randrange(R))


@pytest.mark.gpu
def test_transcript_from_the_point_ifft_gives_the_same_key(ctx):
    """prepare_phase2's own construction: the IFFT of the [tau^i] rows (bls_g*_fft_batch), and alpha and beta times them,
    against the fixed-base [L_q(tau)] rows"""
    import pairing_b200._native as nat
    ni, na = 3, 30
    circ, abc = _toy(20, ni, na, 5, dup=True)
    nc, alpha, beta, tau = circ.length, 23, 29, 987654321
    n = 1 << domain_log(nc)
    powers = [pow(tau, i, R) for i in range(n)]
    coeffs_g1 = ctx.g1_fft("ifft", _points(False, powers))
    ph = mm.transcript(nc, tau, alpha, beta)
    p1 = nat.Groth16Phase1(_points(False, [alpha])[0], _points(False, [beta])[0], _points(True, [beta])[0], coeffs_g1,
                           ctx.g1_fft("ifft", _points(False, [alpha * x for x in powers])), ctx.g1_fft("ifft", _points(False, [beta * x for x in powers])),
                           ctx.g2_fft("ifft", _points(True, powers)), _points(False, ph["h"]))
    assert coeffs_g1.tobytes() == _points(False, ph["coeffs_g1"]).tobytes()
    got = ctx.groth16_mpc_new(abc, nc, ni, na, p1, *_gens())
    _same_key(got, ctx.groth16_mpc_new(abc, nc, ni, na, _phase1(ctx, ph), *_gens()))
    _same_key(got, _generate(ctx, abc, nc, ni, na, alpha, beta, tau))


@pytest.mark.gpu
def test_unconstrained_aux_gives_ok_0(ctx):
    circ = gp.ToyCircuit(12, 2, 6, 3)
    cons = [[{v: c for v, c in lc.items() if v != 2 + 6} for lc in con] for con in circ.all_cons]
    abc = gs.csr_from_cons(cons, 2 + 7)
    ph = mm.transcript(len(cons), 31, 37, 41)
    got = ctx.groth16_mpc_new(abc, len(cons), 2, 7, _phase1(ctx, ph), *_gens())
    key = mm.new(abc, len(cons), 2, 7, ph)
    assert not key["ok"] and not got.ok
    _assert_key(got, key)


@pytest.mark.gpu
def test_inconsistent_g2_row_gives_ok_0(ctx):
    """coeffs_g2[q] replaced by the identity where one variable has its only B term: bg1 != O but bg2 = O"""
    ni, na = 1, 3
    cons = [[{0: 1}, {1: 2}, {2: 1}], [{1: 1}, {2: 5}, {3: 1}], [{0: 1}, {}, {}]]
    abc = gs.csr_from_cons(cons, ni + na)
    ph = mm.transcript(len(cons), 43, 47, 53)
    good = ctx.groth16_mpc_new(abc, len(cons), ni, na, _phase1(ctx, ph), *_gens())
    assert good.ok
    ph["coeffs_g2"][0] = 0
    bad = ctx.groth16_mpc_new(abc, len(cons), ni, na, _phase1(ctx, ph), *_gens())
    assert not mm.new(abc, len(cons), ni, na, ph)["ok"] and not bad.ok
    for name in ("ic", "l", "h", "a", "b_g1"):
        assert getattr(bad, name).tobytes() == getattr(good, name).tobytes(), name


@pytest.mark.gpu
def test_terms_on_one_variable_are_correct_and_not_slow(ctx):
    """2^20 terms per matrix on ONE against the same terms spread evenly over 2^16 variables: the k_mpc_ kernels, timed by
    the profiler, take less than twice as long, and the concentrated key equals generate_parameters' byte for byte"""
    import torch
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    nc, ni, na = 1 << 20, 1, (1 << 16) - 1
    alpha, beta, tau = 3, 5, 1234567
    ph = mm.transcript(nc, tau, alpha, beta)
    rows = _phase1(ctx, ph, lambda g2, e: _points_gpu(ctx, g2, e))
    drows = nat.Groth16Phase1(rows.alpha_g1, rows.beta_g1, rows.beta_g2,
                              *[torch.from_numpy(getattr(rows, k).view(np.int64)).cuda() for k in ("coeffs_g1", "alpha_coeffs_g1", "beta_coeffs_g1", "coeffs_g2", "h")])
    eng = DeviceEngine(ctx)
    times = {}
    for conc in (False, True, False, True):
        abc = _one_heavy(nc, ni + na, conc)
        dabc = _dev_abc(abc)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            got = eng.groth16_mpc_new(dabc, nc, ni, na, drows, *_gens())
            torch.cuda.synchronize()
        t = sum(ev.self_device_time_total for ev in prof.key_averages() if "k_mpc_" in ev.key)
        assert t > 0
        times.setdefault(conc, []).append(t)
    want = _generate(ctx, abc, nc, ni, na, alpha, beta, tau)
    _same_key(got, want)
    assert min(times[True]) < 2 * min(times[False]), times


@pytest.mark.gpu
def test_full_size_2_20_new_prove_verify(ctx):
    """at 2^20 constraints the key equals generate_parameters' byte for byte, proves, and both verifiers accept"""
    ni, nc = 4, 1 << 20
    abc, na, (inputs, aux), evals = random_circuit(20, ni, 2020)
    alpha, beta, tau = 101, 103, 1 << 200
    ph = mm.transcript(nc, tau, alpha, beta)
    got = ctx.groth16_mpc_new(abc, nc, ni, na, _phase1(ctx, ph, lambda g2, e: _points_gpu(ctx, g2, e)), *_gens())
    assert got.ok
    _same_key(got, _generate(ctx, abc, nc, ni, na, alpha, beta, tau))
    m = 2
    abc_ev = [np.broadcast_to(_mont_rows(e), (m, nc, 4)).copy() for e in evals]
    inp = np.broadcast_to(_mont_rows(inputs), (m, ni, 4)).copy()
    ax = np.broadcast_to(_mont_rows(aux), (m, na, 4)).copy()
    r, s = _mont_rows([7, 8]), _mont_rows([9, 10])
    proofs = np.concatenate(ctx.groth16_prove(got, *abc_ev, inp, ax, got.densities, r, s), axis=1)
    ok, ok1 = _verify_all(ctx, got, proofs, inp[:, 1:])
    assert ok.all() and ok1


def _dev_case(ctx, nc, ni, na):
    """a device-contract case of bls_groth16_mpc_new_dev (tests/test_gpu_dev_contract.py's run_dev)"""
    import pairing_b200._native as nat
    rng = random.Random(nc * 100 + ni * 10 + na)
    if nc <= 1:
        cons = [[{0: 5, 1: 1}, {2: 3}, {1: 7, 2: 2}]][:nc]
        abc, length = gs.csr_from_cons(cons, ni + na, seed=3), nc
    else:
        circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
        length = circ.length
    nv = ni + na
    alpha, beta, tau = (rng.randrange(1, R) for _ in range(3))
    ph = mm.transcript(length, tau, alpha, beta)
    rows = _phase1(ctx, ph)
    other = _phase1(ctx, mm.transcript(length, tau + 1, alpha + 1, beta + 1))
    real, decoy = {}, {}
    for i, (off, cons_, coeff) in enumerate(abc):
        real.update({"off%d" % i: off, "cons%d" % i: cons_, "coeff%d" % i: coeff})
        decoy.update({"off%d" % i: off, "cons%d" % i: cons_, "coeff%d" % i: _limbs([bm.fr_to_mont(rng.randrange(R)) for _ in range(len(cons_))]).reshape(-1, 4)})
    names = ("coeffs_g1", "alpha_coeffs_g1", "beta_coeffs_g1", "coeffs_g2", "h")
    for k in names:
        real[k], decoy[k] = getattr(rows, k), getattr(other, k)
    nnz = [len(c) for _, c, _ in abc]
    host_mats = nat.r1cs_matrices(abc, length, nv)
    scratch = int(ctx.groth16_mpc_new_scratch_bytes(host_mats[1], length, ni, na))
    key = mm.new(abc, length, ni, na, ph)
    n1 = nat.domain_size(length) - 1
    a_len, b_len = key["lens"]
    outs = {"vk": _out(nat.W_VK_POINTS * 8), "ic": _out(ni * W1 * 8), "h_out": _out(n1 * W1 * 8), "l": _out(na * W1 * 8),
            "a": _out(nv * W1 * 8, written=a_len * W1 * 8), "b_g1": _out(nv * W1 * 8, written=b_len * W1 * 8),
            "b_g2": _out(nv * W2 * 8, written=b_len * W2 * 8), "d0": _out((na + 31) // 32 * 4, 4), "d1": _out((ni + 31) // 32 * 4, 4),
            "d2": _out((na + 31) // 32 * 4, 4), "lens": _out(16), "ok": _out(1, 1)}
    g1, g2 = (np.ascontiguousarray(x) for x in _gens())

    def args(P):
        mats = (nat.R1csMatrixC * 3)()
        for i in range(3):
            mats[i] = nat.R1csMatrixC(P("off%d" % i), P("cons%d" % i), P("coeff%d" % i), nnz[i])
        p = nat.Groth16Phase1(rows.alpha_g1, rows.beta_g1, rows.beta_g2, *[k for k in names])
        c = nat.groth16_phase1_c(p, length, P, lambda k: len(real[k]))
        out = nat.Groth16ParametersOutC(*[P(x) for x in ("vk", "ic", "h_out", "l", "a", "b_g1", "b_g2", "d0", "d1", "d2", "lens", "ok")])
        return [mats, length, ni, na, ctypes.byref(c), nat._p(g1), nat._p(g2), ctypes.byref(out), P("scratch"), P("stream")]

    def want():
        e = _expect(key)
        w = {"vk": np.concatenate([e[name] for name, _, _ in nat.VK_POINT_ROWS]), "ic": e["ic"], "h_out": e["h"], "l": e["l"], "a": e["a"],
             "b_g1": e["b_g1"], "b_g2": e["b_g2"], "lens": np.array(key["lens"], np.uint64), "ok": np.array([key["ok"]], np.uint8)}
        for i, (d, bits) in enumerate(zip(key["densities"], (na, ni, na))):
            w["d%d" % i] = nat.density_words(np.array(d, dtype=bool), bits, "d")
        return w
    return Case("bls_groth16_mpc_new_dev", args, real, decoy, outs, want, scratch)


CONTRACT_SHAPES = [(0, 1, 2), (1, 1, 2), (5, 2, 3), (33, 1, 5), (40, 3, 40)]
CONTRACT_CASES = [("bls_groth16_mpc_new_dev", "bls_groth16_mpc_new_scratch_bytes"),
                  ("bls_groth16_mpc_contribute_dev", "bls_groth16_mpc_contribute_scratch_bytes"),
                  ("bls_groth16_mpc_verify_dev", "bls_groth16_mpc_verify_scratch_bytes")]


@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", CONTRACT_SHAPES)
def test_dev_contract(ctx, nc, ni, na):
    run_dev(ctx, _dev_case(ctx, nc, ni, na))


@pytest.mark.gpu
def test_host_dev_and_engine_agree(ctx):
    from pairing_b200.device import DeviceEngine
    import torch
    import pairing_b200._native as nat
    ni, na = 3, 40
    circ, abc = _toy(40, ni, na, 8, dup=True)
    nc = circ.length
    ph = _phase1(ctx, mm.transcript(nc, 99, 98, 97))
    host = ctx.groth16_mpc_new(abc, nc, ni, na, ph, *_gens())
    dph = nat.Groth16Phase1(ph.alpha_g1, ph.beta_g1, ph.beta_g2,
                            *[torch.from_numpy(getattr(ph, k).view(np.int64)).cuda() for k in ("coeffs_g1", "alpha_coeffs_g1", "beta_coeffs_g1", "coeffs_g2", "h")])
    dev = DeviceEngine(ctx).groth16_mpc_new(_dev_abc(abc), nc, ni, na, dph, *_gens())
    for name in KEY_ROWS:
        assert np.ascontiguousarray(getattr(dev, name).cpu()).view(np.uint64).tobytes() == np.ascontiguousarray(getattr(host, name)).tobytes(), name
    assert [list(d) for d in dev.densities] == [list(d) for d in host.densities] and dev.ok == host.ok


@pytest.mark.gpu
def test_invalid_arguments_are_rejected_before_any_work(ctx):
    import pairing_b200._native as nat
    lib = nat.load()
    ni, na = 1, 2
    cons = [[{0: 5, 1: 1}, {2: 3}, {1: 7, 2: 2}], [{0: 1}, {}, {}], [{1: 1}, {2: 1}, {2: 1}]]
    abc = gs.csr_from_cons(cons, ni + na)
    ph = _phase1(ctx, mm.transcript(3, 5, 6, 7))
    g1, g2 = _gens()
    with pytest.raises(ValueError):
        ctx.groth16_mpc_new(abc, 5, ni, na, ph, g1, g2)                 # rows of n = 4, the domain of 5 constraints is 8
    keep, mats = nat.r1cs_matrices(abc, 3, ni + na)
    c = nat.groth16_phase1_c(ph, 3, nat._p, len)
    bufs, out = ctx._parameters_out(3, ni, na)
    inf1, inf2 = g1.copy(), g2.copy()
    inf1[-1], inf2[-1] = 1, 1
    call = lambda c_, a, b, o_=out: lib.bls_groth16_mpc_new_batch(ctx._ctx, mats, 3, ni, na, c_ if c_ is None else ctypes.byref(c_),  # noqa: E731
                                                                 nat._p(a), nat._p(b), o_ if o_ is None else ctypes.byref(o_))
    assert call(c, g1, g2) == 0
    assert call(c, inf1, g2) == -1 and call(c, g1, inf2) == -1 and call(None, g1, g2) == -1 and call(c, g1, g2, None) == -1
    wrong_n = nat.groth16_phase1_c(ph, 3, nat._p, len)
    wrong_n.n = 8
    bads = [wrong_n]
    for field in ("coeffs_g1", "alpha_coeffs_g1", "beta_coeffs_g1", "coeffs_g2", "h"):
        c_ = nat.groth16_phase1_c(ph, 3, nat._p, len)
        setattr(c_, field, None)
        bads.append(c_)
    for bad in bads:                                              # every output poisoned and left as it was
        for b in bufs:
            for x in (b if isinstance(b, list) else [b]):
                x.view(np.uint8).fill(0x5A)
        assert call(bad, g1, g2) == -1
        for b in bufs:
            for x in (b if isinstance(b, list) else [b]):
                assert (x.view(np.uint8) == 0x5A).all()
    for field in ("vk", "ic", "h", "l", "a", "b_g1", "b_g2", "a_aux_density", "b_input_density", "b_aux_density", "lens", "ok"):
        _, o2 = ctx._parameters_out(3, ni, na)
        setattr(o2, field, None)
        assert call(c, g1, g2, o2) == -1, field
    assert ctx._lib.bls_groth16_mpc_new_scratch_bytes(ctx._ctx, mats, (1 << 26) + 1, ni, na) == 0     # the domain limit
    assert lib.bls_groth16_mpc_new_dev(ctx._ctx, mats, 3, ni, na, ctypes.byref(wrong_n), nat._p(g1), nat._p(g2), ctypes.byref(out), None, None) == -1
    del keep


# ---------------------------------------------------------------------------------------------------------------- contributions and verification

def _chain(key, k, seed):
    """k honest contributions in exponents: the keys after each and the pubkey exponents"""
    rng = random.Random(seed)
    keys, pks = [key], []
    for _ in range(k):
        nk, pk = mm.contribute(keys[-1], rng.randrange(1, R), rng.randrange(1, R), rng.randrange(1, R))
        keys.append(nk)
        pks.append(pk)
    return keys, pks


def _tampers(before, after, pks):
    """(name, before, after, pks) for every single tamper of the issue's list, in exponents"""
    out = []
    for q in ("h", "l", "ic", "a", "b", "b_g2"):
        if after[q]:
            t = dict(after)
            t[q] = [after[q][0] + 1] + after[q][1:]
            out.append(("row-" + q, before, t, pks))
    for q in ("h", "l"):
        t = dict(after)
        t[q] = after[q][:-1]
        out.append(("len-" + q, before, t, pks))
    out.append(("gamma_g2", before, dict(after, gamma=after["gamma"] + 1), pks))
    out.append(("delta_g1", before, dict(after, delta=after["delta"] + 1), pks))
    out.append(("delta_g2", before, dict(after, delta_g2=after["delta"] + 1), pks))
    if len(pks) >= 2:
        for i, name in ((1, "s_delta"), (4, "r_delta"), (0, "delta_after")):
            bad = [list(p) for p in pks]
            bad[1][2 if i == 1 else i] = bad[1][2 if i == 1 else i] + 1
            out.append(("mid-" + name, before, after, [tuple(p) for p in bad]))
        out.append(("swapped", before, after, [pks[1], pks[0]] + pks[2:]))
    return out


def _model_key(nc=20, ni=3, na=30, seed=4):
    circ, abc = _toy(nc, ni, na, seed, dup=True)
    return mm.new(abc, circ.length, ni, na, mm.transcript(circ.length, 1234567, 89, 97))


@pytest.mark.parametrize("k", [0, 1, 3])
def test_model_verify_accepts_honest_chains_and_rejects_each_tamper(k):
    key = _model_key()
    keys, pks = _chain(key, k, k)
    rng = random.Random(9)
    rho_h, rho_l = [rng.randrange(1, R) for _ in key["h"]], [rng.randrange(1, R) for _ in key["l"]]
    assert mm.verify(key, keys[-1], pks, rho_h, rho_l)
    for name, b, a, p in _tampers(key, keys[-1], pks):
        if name.startswith("len-"):
            continue                                                   # the model's merged sums would zip-truncate
        assert not mm.verify(b, a, p, rho_h, rho_l), name


def _rows(g2, exps):
    return _points(g2, exps)


def _params(ctx, key, ni, na):
    """a Groth16Parameters of points for the model key (its queries in the key's order)"""
    import pairing_b200._native as nat
    one = lambda g2, e: _points(g2, [e])[0]                                                 # noqa: E731
    dens = tuple(np.array(d, dtype=bool) for d in key["densities"])
    return nat.Groth16Parameters(one(False, key["alpha"]), one(False, key["beta"]), one(False, key["delta"]), one(True, key["beta"]),
                                 one(True, key.get("delta_g2", key["delta"])), _rows(False, key["h"]), _rows(False, key["l"]), _rows(False, key["a"]),
                                 _rows(False, key["b"]), _rows(True, key["b_g2"]), gamma_g2=one(True, key["gamma"]), ic=_rows(False, key["ic"]),
                                 densities=dens, ok=True)


def _pk_rows(pk):
    da, s, sd, r, rd = pk
    return np.concatenate([_points(False, [da])[0], _points(False, [s])[0], _points(False, [sd])[0], _points(True, [r])[0], _points(True, [rd])[0]])


def _contribute_chain(ctx, before, k, seed):
    rng = random.Random(seed)
    params, pks, exps = before, [], []
    for _ in range(k):
        delta, s, r = rng.randrange(1, R), rng.randrange(1, R), rng.randrange(1, R)
        params, pk = ctx.groth16_mpc_contribute(params, _mont1(delta), _points(False, [s])[0], _points(True, [r])[0])
        pks.append(pk)
        exps.append((delta, s, r))
    return params, np.stack(pks) if pks else np.zeros((0, 89), dtype=np.uint64), exps


def _rho(n, seed):
    rng = random.Random(seed)
    return _limbs([rng.randrange(R) for _ in range(n)] if n < 3 else [0] + [rng.randrange(R) for _ in range(n - 1)])


@pytest.mark.gpu
def test_contribute_chain_of_three_matches_the_model(ctx):
    key = _model_key()
    before = _params(ctx, key, 3, 30)
    after, pks, exps = _contribute_chain(ctx, before, 3, 1)
    want, wpk = key, []
    for delta, s, r in exps:
        want, pk = mm.contribute(want, delta, s, r)
        wpk.append(pk)
    for name, ex in (("h", want["h"]), ("l", want["l"])):
        assert np.ascontiguousarray(getattr(after, name)).tobytes() == _rows(False, ex).tobytes(), name
    assert after.delta_g1.tobytes() == _points(False, [want["delta"]])[0].tobytes()
    assert after.delta_g2.tobytes() == _points(True, [want["delta"]])[0].tobytes()
    for j in range(3):
        assert pks[j].tobytes() == _pk_rows(wpk[j]).tobytes(), j
    for name in ("alpha_g1", "beta_g1", "beta_g2", "gamma_g2", "ic", "a", "b_g1", "b_g2"):
        assert np.ascontiguousarray(getattr(after, name)).tobytes() == np.ascontiguousarray(getattr(before, name)).tobytes(), name


@pytest.mark.gpu
def test_contribute_matches_the_replicated_wnaf_batch_and_runs_in_place(ctx):
    import torch
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    key = _model_key(40, 3, 40, 6)
    before = _params(ctx, key, 3, 40)
    delta = 0x1234567890ABCDEF1234567890ABCDEF % R
    d = pow(delta, -1, R)
    s, r = _points(False, [5])[0], _points(True, [7])[0]
    after, pk = ctx.groth16_mpc_contribute(before, _mont1(delta), s, r)
    rows = np.concatenate([before.h, before.l])
    want = ctx.g1_into_affine(ctx.g1_wnaf_mul(np.ascontiguousarray(o.g1_from_affine(rows)), _limbs([d] * len(rows))))
    assert np.concatenate([after.h, after.l]).tobytes() == want.tobytes()
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).cuda()          # noqa: E731
    dparams = nat.Groth16Parameters(*[dev(getattr(before, n)) for n in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2", "h", "l", "a", "b_g1", "b_g2")],
                                    gamma_g2=dev(before.gamma_g2), ic=dev(before.ic), densities=before.densities, ok=True)
    eng = DeviceEngine(ctx)
    out_of_place, dpk = eng.groth16_mpc_contribute(dparams, _mont1(delta), s, r)
    in_place, dpk2 = eng.groth16_mpc_contribute(dparams, _mont1(delta), s, r, in_place=True)
    for name in ("h", "l", "delta_g1", "delta_g2"):
        a, b = (np.ascontiguousarray(getattr(x, name).cpu()).view(np.uint64).tobytes() for x in (out_of_place, in_place))
        c = np.ascontiguousarray(getattr(after, name)).tobytes()
        assert a == b == c, name
    assert dpk.cpu().numpy().view(np.uint64).tobytes() == pk.tobytes() == dpk2.cpu().numpy().view(np.uint64).tobytes()


def _tamper_params(ctx, before, after, pks, name):
    """the point form of each tamper of _tampers"""
    import dataclasses
    a, p = after, pks.copy()
    other = _points(False, [424242])[0]
    if name.startswith("row-"):
        q = {"b": "b_g1"}.get(name[4:], name[4:])
        rows = np.ascontiguousarray(getattr(after, q)).copy()
        rows[-1] = _points(q == "b_g2", [424242])[0]                   # the last row: rho_0 = 0 leaves row 0 out
        a = dataclasses.replace(after, **{q: rows} if q != "ic" else {}) if q != "ic" else dataclasses.replace(after, ic=rows)
    elif name.startswith("len-"):
        q = name[4:]
        a = dataclasses.replace(after, **{q: np.ascontiguousarray(getattr(after, q))[:-1]})
    elif name == "gamma_g2":
        a = dataclasses.replace(after, gamma_g2=_points(True, [3])[0])
    elif name == "delta_g1":
        a = dataclasses.replace(after, delta_g1=other)
    elif name == "delta_g2":
        a = dataclasses.replace(after, delta_g2=_points(True, [424242])[0])
    elif name.startswith("mid-"):
        off = {"mid-s_delta": (2 * W1, W1, False), "mid-r_delta": (3 * W1 + W2, W2, True), "mid-delta_after": (0, W1, False)}[name]
        p[1, off[0]:off[0] + off[1]] = _points(off[2], [424242])[0]
    elif name == "swapped":
        p = p[[1, 0, 2]]
    return before, a, p


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1, 3])
def test_verify_accepts_an_honest_chain(ctx, k):
    key = _model_key()
    before = _params(ctx, key, 3, 30)
    after, pks, _ = _contribute_chain(ctx, before, k, 10 + k)
    assert ctx.groth16_mpc_verify(before, after, pks, _rho(len(before.h), 1), _rho(len(before.l), 2))


TAMPERS = ["row-h", "row-l", "row-ic", "row-a", "row-b", "row-b_g2", "len-h", "len-l", "gamma_g2", "delta_g1", "delta_g2", "mid-s_delta",
           "mid-r_delta", "mid-delta_after", "swapped"]


@pytest.mark.gpu
def test_verify_rejects_each_tamper(ctx):
    key = _model_key()
    before = _params(ctx, key, 3, 30)
    after, pks, _ = _contribute_chain(ctx, before, 3, 20)
    rh, rl = _rho(len(before.h), 1), _rho(len(before.l), 2)
    assert ctx.groth16_mpc_verify(before, after, pks, rh, rl)
    for name in TAMPERS:
        b, a, p = _tamper_params(ctx, before, after, pks, name)
        assert not ctx.groth16_mpc_verify(b, a, p, rh, rl), name


@pytest.mark.gpu
def test_verify_host_and_device_agree(ctx):
    import torch
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    key = _model_key()
    before = _params(ctx, key, 3, 30)
    after, pks, _ = _contribute_chain(ctx, before, 2, 30)
    rh, rl = _rho(len(before.h), 1), _rho(len(before.l), 2)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).cuda()          # noqa: E731
    names = ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2", "h", "l", "a", "b_g1", "b_g2")
    todev = lambda P: nat.Groth16Parameters(*[dev(getattr(P, n)) for n in names], gamma_g2=dev(P.gamma_g2), ic=dev(P.ic),   # noqa: E731
                                            densities=P.densities, ok=True)
    eng = DeviceEngine(ctx)
    for b, a, p in ((before, after, pks), _tamper_params(ctx, before, after, pks, "row-l")):
        assert ctx.groth16_mpc_verify(b, a, p, rh, rl) == eng.groth16_mpc_verify(todev(b), todev(a), dev(p), dev(rh), dev(rl))


@pytest.mark.gpu
def test_full_size_2_20_contributions_verify_and_prove(ctx):
    """at 2^20 constraints: mpc_new, three contributions, verify gives 1, and a proof from the contributed key passes both
    verifiers while failing against the pre-contribution vk"""
    ni, nc = 4, 1 << 20
    abc, na, (inputs, aux), evals = random_circuit(20, ni, 2020)
    ph = mm.transcript(nc, 1 << 200, 101, 103)
    before = ctx.groth16_mpc_new(abc, nc, ni, na, _phase1(ctx, ph, lambda g2, e: _points_gpu(ctx, g2, e)), *_gens())
    assert before.ok
    after, pks, _ = _contribute_chain(ctx, before, 3, 7)
    assert ctx.groth16_mpc_verify(before, after, pks, _rho(len(before.h), 3), _rho(len(before.l), 4))
    m = 2
    abc_ev = [np.broadcast_to(_mont_rows(e), (m, nc, 4)).copy() for e in evals]
    inp = np.broadcast_to(_mont_rows(inputs), (m, ni, 4)).copy()
    ax = np.broadcast_to(_mont_rows(aux), (m, na, 4)).copy()
    proofs = np.concatenate(ctx.groth16_prove(after, *abc_ev, inp, ax, after.densities, _mont_rows([7, 8]), _mont_rows([9, 10])), axis=1)
    ok, ok1 = _verify_all(ctx, after, proofs, inp[:, 1:])
    assert ok.all() and ok1
    ok, ok1 = _verify_all(ctx, before, proofs, inp[:, 1:])
    assert not ok.any() and not ok1


def _contribute_case(ctx, h_len, l_len):
    import pairing_b200._native as nat
    pool = _points(False, list(range(1, h_len + l_len + 9)))
    h, l = pool[:h_len], pool[h_len:h_len + l_len]
    dh, dl = pool[::-1][:h_len].copy(), pool[::-1][h_len:h_len + l_len].copy()
    vk = np.concatenate([_points(False, [2])[0], _points(False, [3])[0], _points(False, [4])[0], _points(True, [5])[0], _points(True, [6])[0],
                         _points(True, [4])[0]])
    delta, s, r = _mont1(77), _points(False, [8])[0], _points(True, [9])[0]
    real, decoy = {"h": h, "l": l, "vk": vk}, {"h": dh, "l": dl, "vk": np.concatenate([vk[:2 * W1], _points(False, [11])[0], vk[3 * W1:]])}
    outs = {"h_out": _out(h.nbytes), "l_out": _out(l.nbytes), "pk": _out(8 * nat.W_MPC_PUBKEY)}
    host = [np.ascontiguousarray(x) for x in (delta, s, r)]

    def args(P):
        return [*[nat._p(x) for x in host], P("vk"), P("h"), h_len, P("l"), l_len, P("h_out"), P("l_out"), P("pk"), P("scratch"), P("stream")]

    def want():
        vk2 = vk.copy()
        h2, l2, pk = h.copy(), l.copy(), np.zeros(nat.W_MPC_PUBKEY, dtype=np.uint64)
        ctx._check(ctx._lib.bls_groth16_mpc_contribute_batch(ctx._ctx, *[nat._p(x) for x in host], nat._p(vk2), nat._p(h2), h_len, nat._p(l2), l_len,
                                                             nat._p(h2), nat._p(l2), nat._p(pk)))
        return {"vk": vk2, "h_out": h2, "l_out": l2, "pk": pk}
    return Case("bls_groth16_mpc_contribute_dev", args, real, decoy, outs, want, int(ctx.groth16_mpc_contribute_scratch_bytes(h_len, l_len)),
                inout=("vk",))


def _verify_case(ctx, k, valid):
    import pairing_b200._native as nat
    key = _model_key()
    before = _params(ctx, key, 3, 30)
    after, pks, _ = _contribute_chain(ctx, before, k, 40 + k)
    if not valid:
        _, after, pks = _tamper_params(ctx, before, after, pks, "row-l")
    rh, rl = _rho(len(before.h), 1), _rho(len(before.l), 2)
    names = ("ic", "h", "l", "a", "b_g1", "b_g2")
    real = {"b_" + n: np.ascontiguousarray(getattr(before, n)) for n in names}
    real.update({"a_" + n: np.ascontiguousarray(getattr(after, n)) for n in names})
    real.update({"pk": pks if k else np.zeros((1, 89), np.uint64), "rh": rh, "rl": rl})
    decoy = {n: v[::-1].copy() for n, v in real.items()}
    kb, ka = nat.groth16_key_c(before, nat._p, len), nat.groth16_key_c(after, nat._p, len)

    def args(P):
        for c_, pre in ((kb, "b_"), (ka, "a_")):
            for n in names:
                setattr(c_, n, P(pre + n))
        return [ctypes.byref(kb), ctypes.byref(ka), P("pk"), k, P("rh"), P("rl"), P("ok"), P("scratch"), P("stream")]

    def want():
        return {"ok": np.array([ctx.groth16_mpc_verify(before, after, pks, rh, rl)], np.uint8)}
    sb = nat.groth16_key_c(before, nat._p, len), nat.groth16_key_c(after, nat._p, len)
    return Case("bls_groth16_mpc_verify_dev", args, real, decoy, {"ok": _out(1, 1)}, want, int(ctx.groth16_mpc_verify_scratch_bytes(*sb, k)))


@pytest.mark.gpu
@pytest.mark.parametrize("h_len,l_len", [(0, 0), (1, 0), (3, 5), (200, 130)])
def test_dev_contract_contribute(ctx, h_len, l_len):
    run_dev(ctx, _contribute_case(ctx, h_len, l_len))


@pytest.mark.gpu
@pytest.mark.parametrize("k,valid", [(0, True), (3, True), (3, False)])
def test_dev_contract_verify(ctx, k, valid):
    case = _verify_case(ctx, k, valid)
    assert case.want()["ok"][0] == valid
    run_dev(ctx, case)
