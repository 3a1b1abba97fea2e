"""Groth16 proofs (bls_groth16_prove_batch / _dev, Context.groth16_prove, DeviceEngine.groth16_prove, Groth16::create_proof).

Every key point is [e]g with a known exponent e, so a proof is known by the exponents of A, B and C: the GPU's bytes are
compared with [e]g from the oracle.  On toy circuits the exponents come from tests/groth16_prove_model.py, which is checked
here against the verification equation; at full size they come from the closed form over the known exponents of
bench.make_inputs' points, with H from bls_fr_groth16_h (tests/test_gpu_groth16_h.py pins it to its model).  Outputs are
canonical affine points, so every comparison is bit for bit whatever order the kernels sum in."""
import ctypes
import os
import random
import re
import subprocess
import tempfile

import numpy as np
import pytest

import bls_model as bm
import groth16_prove_model as gp
import oracle_lib as o
from test_gpu_msm import N_MAX, _base_exponents, eng, inputs  # noqa: F401 -- eng and inputs are fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER
W1, W2 = 13, 25


def _limbs(values):
    return np.array([bm.limbs64(v % (1 << 256), 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _ints(a):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).astype(object)
    return list(a[:, 0] + (a[:, 1] << 64) + (a[:, 2] << 128) + (a[:, 3] << 192))


def _points(g2, exps):
    """[e]g for every exponent, affine rows (the identity for e = 0)"""
    exps = [e % R for e in exps]
    if not exps:
        return np.zeros((0, W2 if g2 else W1), dtype=np.uint64)
    op, from_aff, into_aff = (o.g2_op, o.g2_from_affine, o.g2_into_affine) if g2 else (o.g1_op, o.g1_from_affine, o.g1_into_affine)
    g = np.repeat(from_aff(o.generators()[1 if g2 else 0]), len(exps), 0)
    return into_aff(op("mul", g, k=_limbs(exps), threads=o.default_threads()))


def _mont_rows(values):
    return _limbs(gp.mont(values))


class Toy:
    """a toy circuit, its key (exponents and points) and m witnesses"""

    def __init__(self, nc, ni, na, m, seed):
        rng = random.Random(seed)
        self.circuit = gp.ToyCircuit(nc, ni, na, seed)
        self.key = self.circuit.setup(*[rng.randrange(1, R) for _ in range(5)])
        k = self.key
        self.witnesses = [self.circuit.witness(seed * 101 + j) for j in range(m)]
        evals = [self.circuit.evaluations(*w) for w in self.witnesses]
        self.m, self.len = m, self.circuit.length
        self.abc = [np.stack([_mont_rows(e[q]) for e in evals]).reshape(m, self.len, 4) for q in range(3)]
        self.input = np.stack([_mont_rows(w[0]) for w in self.witnesses]).reshape(m, ni, 4)
        self.aux = np.stack([_mont_rows(w[1]) for w in self.witnesses]).reshape(m, na, 4)
        rs = [rng.choice([0, 1, rng.randrange(R)]) for _ in range(2 * m)]
        self.r, self.s = _mont_rows(rs[:m]), _mont_rows(rs[m:])
        self.densities = tuple(np.array(d, dtype=bool) for d in k["densities"])
        self.params = gp_params(k["alpha"], k["beta"], k["delta"], k["h"], k["l"], k["a"], k["b_g1"], k["b_g2"])

    def model(self):
        """the (m, 51) proof rows of the model"""
        rows = []
        for j in range(self.m):
            e = gp.create_proof(self.key, *[_ints(x[j]) for x in self.abc], _ints(self.input[j]), _ints(self.aux[j]),
                                self.key["densities"], _ints(self.r[j])[0], _ints(self.s[j])[0])
            rows.append(np.concatenate([_points(False, [e[0]]), _points(True, [e[1]]), _points(False, [e[2]])], axis=1))
        return np.concatenate(rows) if rows else np.zeros((0, 2 * W1 + W2), dtype=np.uint64)

    def prove(self, ctx):
        return ctx.groth16_prove(self.params, *self.abc, self.input, self.aux, self.densities, self.r, self.s)


def gp_params(alpha, beta, delta, h, l, a, b_g1, b_g2):
    import pairing_b200._native as nat
    one = _points(False, [alpha, beta, delta])
    two = _points(True, [beta, delta])
    return nat.Groth16Params(one[0], one[1], one[2], two[0], two[1], _points(False, h), _points(False, l), _points(False, a),
                             _points(False, b_g1), _points(True, b_g2))


def _proof(parts):
    return np.concatenate([np.asarray(x) for x in parts], axis=1)


# ---------------------------------------------------------------------------------------------------------------- CPU

SHAPES = [(1, 1, 0), (2, 1, 1), (5, 2, 3), (7, 3, 0), (12, 1, 12), (20, 3, 30), (40, 3, 40), (3, 2, 10), (33, 1, 5)]


@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_model_proofs_satisfy_the_verification_equation(nc, ni, na):
    """A B = alpha beta + gamma sum_i input_i ic_i + delta C (mod r) for several r and s (0 included), and not for a changed C"""
    rng = random.Random(nc * 1000 + ni * 100 + na)
    circuit = gp.ToyCircuit(nc, ni, na, rng.randrange(1 << 30))
    key = circuit.setup(*[rng.randrange(1, R) for _ in range(5)])
    for w in range(2):
        inputs, aux = circuit.witness(w)
        a, b, c = circuit.evaluations(inputs, aux)
        assert all(x * y % R == z for x, y, z in zip(a, b, c))
        for r, s in ((0, 0), (0, 1), (1, 0), (rng.randrange(R), rng.randrange(R))):
            proof = gp.create_proof(key, gp.mont(a), gp.mont(b), gp.mont(c), gp.mont(inputs), gp.mont(aux), key["densities"],
                                    gp.mont([r])[0], gp.mont([s])[0])
            assert gp.verifies(key, inputs, proof), (w, r, s)
            assert not gp.verifies(key, inputs, (proof[0], proof[1], (proof[2] + 1) % R))


def test_density_words_are_bitvec_u32_storage():
    import pairing_b200._native as nat
    rng = np.random.default_rng(5)
    for bits in (0, 1, 31, 32, 33, 100):
        d = rng.random(bits) < 0.5
        w = nat.density_words(d, bits, "d")
        assert len(w) == (bits + 31) // 32
        assert [bool((w[i // 32] >> (i % 32)) & 1) for i in range(bits)] == list(d)
    with pytest.raises(ValueError):
        nat.density_words(np.zeros(5, dtype=bool), 6, "d")


def test_groth16_kernels_do_not_spill():
    """k_groth16_gather keeps its state in registers; the tail kernels use no local memory and no more stack than the
    call frames of curve.cuh's group law stated in DESIGN.md (cuobjdump --dump-resource-usage)"""
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
    limits = {"k_groth16_gather": 0, "k_groth16_mul": 1176, "k_groth16_assemble": 1696}
    for kernel, stack in limits.items():
        found = [v for k, v in usage.items() if kernel in k]
        assert len(found) == 1, (kernel, sorted(usage))
        assert found[0]["LOCAL"] == 0 and found[0]["STACK"] <= stack, (kernel, found[0])


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    args = [None, None, None, None, 4, None, 1, None, 0, None, None, None, None, None, 1, None]
    assert lib.bls_groth16_prove_batch(None, *args) == -1
    assert lib.bls_groth16_prove_dev(None, *args, None, None) == -1
    assert lib.bls_groth16_prove_scratch_bytes(None, None, 4, 1, 0, None, None, None, 1) == 0


def test_struct_sizes_match_the_bindings():
    """sizeof(bls_groth16_proof) = 408 (bellman's Proof<Bls12>: 2 G1Affine + 1 G2Affine) and bls_groth16_params' layout
    equals the ctypes structure of the Python binding"""
    import pairing_b200._native as nat
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "pairing_b200.h"\nint main(){printf("%zu %zu %zu\\n",' \
          'sizeof(bls_groth16_proof),sizeof(bls_groth16_params),offsetof(bls_groth16_params,h));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(c, "w").write(src)
        subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        sizes = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert sizes == [8 * nat.W_PROOF, ctypes.sizeof(nat._Groth16ParamsC), nat._Groth16ParamsC.h.offset]
    assert nat.W_PROOF * 8 == 408


# ---------------------------------------------------------------------------------------------------------------- GPU

def _verify(ctx, key, proof_row, inputs):
    """e(A, B) e(-alpha, beta) e(-IC, gamma) e(-C, delta) = 1 through the library's pairing_product"""
    ic = sum(x * e for x, e in zip(inputs, key["ic"]))
    c_neg = ctx.g1_into_affine(ctx.g1_op("negate", o.g1_from_affine(proof_row[None, W1 + W2:])))
    p = np.concatenate([proof_row[None, :W1], _points(False, [-key["alpha"], -ic]), c_neg])
    q = np.concatenate([proof_row[None, W1:W1 + W2], _points(True, [key["beta"], key["gamma"], key["delta"]])])
    got, some = ctx.pairing_product(p, q)
    g1, g2 = o.generators()
    one, _ = ctx.pairing_product(np.concatenate([g1, _points(False, [-1])]), np.concatenate([g2, g2]))
    return some and np.array_equal(got, one)


@pytest.mark.gpu
@pytest.mark.parametrize("nc,ni,na", SHAPES)
def test_toy_circuits_match_the_model_and_verify(ctx, nc, ni, na):
    m = 3
    toy = Toy(nc, ni, na, m, nc * 97 + ni * 13 + na)
    a, b, c = toy.prove(ctx)
    got = _proof((a, b, c))
    assert got.tobytes() == toy.model().tobytes()
    for j in range(m):
        assert _verify(ctx, toy.key, got[j], toy.witnesses[j][0]), j
    bad = got[0].copy()
    bad[W1 + W2:] = _points(False, [12345])[0]
    assert not _verify(ctx, toy.key, bad, toy.witnesses[0][0])


@pytest.fixture(scope="module")
def full(inputs):
    """the 2^20 G1 and G2 points and their exponents"""
    return {False: (inputs["host"][False], _ints(_base_exponents(False, N_MAX))),
            True: (inputs["host"][True], _ints(_base_exponents(True, N_MAX)))}


def _rot(full, g2, off, count):
    pts, ex = full[g2]
    idx = (np.arange(count) + off) % N_MAX
    return pts[idx], [ex[i] for i in idx]


def _rand_fr(rng, count):
    """Montgomery-form values < r (canonical): random 252-bit integers"""
    k = rng.integers(0, 1 << 63, size=(count, 4), dtype=np.uint64) * 2 + rng.integers(0, 2, size=(count, 4), dtype=np.uint64)
    k[:, 3] &= np.uint64((1 << 60) - 1)
    return k


def _run_full(ctx, eng, full, length, ni, na, m, dens, seed):
    """prove through the DeviceEngine and compare with [closed-form exponent] g; returns the proof rows"""
    import torch
    import pairing_b200._native as nat
    rng = np.random.default_rng(seed)
    a_aux, b_in, b_aux = dens
    la, lb = ni + int(a_aux.sum()), int(b_in.sum()) + int(b_aux.sum())
    n1 = (1 << max(length - 1, 0).bit_length()) - 1
    hq, he = _rot(full, False, 11, n1)
    lq, le = _rot(full, False, 3 * N_MAX // 7, na)
    aq, ae = _rot(full, False, N_MAX // 3, la)
    b1q, b1e = _rot(full, False, N_MAX // 2, lb)
    b2q, b2e = _rot(full, True, 77, lb)
    vk = [int(x) for x in rng.integers(1, 1 << 62, size=5)]
    one, two = _points(False, vk[:3]), _points(True, vk[3:])
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to(eng.device)  # noqa: E731
    params = nat.Groth16Params(one[0], one[1], one[2], two[0], two[1], dev(hq), dev(lq), dev(aq), dev(b1q), dev(b2q))
    abc = [_rand_fr(rng, m * length).reshape(m, length, 4) for _ in range(3)]
    inp, aux = _rand_fr(rng, m * ni).reshape(m, ni, 4), _rand_fr(rng, m * na).reshape(m, na, 4)
    r, s = _rand_fr(rng, m), _rand_fr(rng, m)
    if m:
        r[0] = 0
    got = eng.groth16_prove(params, *(dev(x) for x in abc), dev(inp), dev(aux), dens, dev(r), dev(s))
    got = _proof([t.cpu().numpy().view(np.uint64) for t in got])
    h = eng.groth16_h(*(dev(x) for x in abc)).cpu().numpy().view(np.uint64).reshape(m, n1, 4) if n1 else np.zeros((m, 0, 4), np.uint64)
    ia, ib, ibx = np.flatnonzero(a_aux), np.flatnonzero(b_in), np.flatnonzero(b_aux)
    want = []
    for j in range(m):
        x_in = [bm.fr_from_mont(v) for v in _ints(inp[j])]
        x_aux = [bm.fr_from_mont(v) for v in _ints(aux[j])]
        sa = x_in + [x_aux[i] for i in ia]
        sb = [x_in[i] for i in ib] + [x_aux[i] for i in ibx]
        dot = lambda xs, es: sum(x * e for x, e in zip(xs, es))  # noqa: E731
        a_ans, b1, b2 = dot(sa, ae), dot(sb, b1e), dot(sb, b2e)
        rr, ss = bm.fr_from_mont(_ints(r[j])[0]), bm.fr_from_mont(_ints(s[j])[0])
        alpha, beta1, delta1, beta2, delta2 = vk
        ea = rr * delta1 + alpha + a_ans
        eb = ss * delta2 + beta2 + b2
        ec = rr * ss * delta1 + ss * (alpha + a_ans) + rr * (beta1 + b1) + dot(_ints(h[j]), he) + dot(x_aux, le)
        want.append((ea, eb, ec))
    rows = [np.concatenate([_points(False, [w[0]]), _points(True, [w[1]]), _points(False, [w[2]])], axis=1) for w in want]
    assert got.tobytes() == (np.concatenate(rows) if rows else np.zeros((0, 51), np.uint64)).tobytes()
    return got


def _dens(rng, ni, na, p):
    return (rng.random(na) < p, rng.random(ni) < p, rng.random(na) < p)


@pytest.mark.gpu
def test_one_proof_of_2_20_against_the_closed_form(ctx, eng, full):
    rng = np.random.default_rng(20)
    length, ni, na = 1 << 20, 3, (1 << 20) - 3
    _run_full(ctx, eng, full, length, ni, na, 1, _dens(rng, ni, na, 0.7), 0x220)


@pytest.mark.gpu
def test_64_proofs_of_2_12_against_the_closed_form(ctx, eng, full):
    rng = np.random.default_rng(12)
    length, ni, na = 1 << 12, 2, 4000
    _run_full(ctx, eng, full, length, ni, na, 64, _dens(rng, ni, na, 0.5), 0x212)


@pytest.mark.gpu
def test_ragged_shapes_against_the_closed_form(ctx, eng, full):
    """len 1, 2, 7, 129; num_aux = 0; num_inputs = 1; all-zero and all-one densities; bitmap lengths that are not a
    multiple of 32; m = 0"""
    rng = np.random.default_rng(7)
    for length, ni, na, m, kind in ((1, 1, 0, 2, "rand"), (2, 1, 1, 3, "ones"), (7, 2, 5, 2, "zeros"), (129, 3, 100, 3, "rand"),
                                    (129, 1, 33, 2, "ones"), (64, 33, 65, 2, "rand"), (7, 1, 0, 0, "rand"), (1000, 1, 31, 5, "zeros")):
        if kind == "rand":
            dens = _dens(rng, ni, na, 0.5)
        else:
            v = kind == "ones"
            dens = (np.full(na, v), np.full(ni, v), np.full(na, v))
        _run_full(ctx, eng, full, length, ni, na, m, dens, length * 7 + na)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_random_densities_against_the_closed_form(ctx, eng, full, p):
    rng = np.random.default_rng(int(p * 100))
    _run_full(ctx, eng, full, 3000, 3, 2900, 4, _dens(rng, 3, 2900, p), int(p * 1000))


CPP_PROVE = r"""
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
  Groth16::Params p;
  auto vk1 = rd<G1AffinePoint>(f); auto vk2 = rd<G2AffinePoint>(f);
  p.alpha_g1 = vk1[0]; p.beta_g1 = vk1[1]; p.delta_g1 = vk1[2]; p.beta_g2 = vk2[0]; p.delta_g2 = vk2[1];
  p.h = rd<G1AffinePoint>(f); p.l = rd<G1AffinePoint>(f); p.a = rd<G1AffinePoint>(f); p.b_g1 = rd<G1AffinePoint>(f); p.b_g2 = rd<G2AffinePoint>(f);
  auto a = rd<bls_fr>(f); auto b = rd<bls_fr>(f); auto c = rd<bls_fr>(f); auto in = rd<bls_fr>(f); auto aux = rd<bls_fr>(f);
  auto d0 = rd<uint32_t>(f); auto d1 = rd<uint32_t>(f); auto d2 = rd<uint32_t>(f);
  auto r = rd<bls_fr>(f); auto s = rd<bls_fr>(f);
  auto proofs = Groth16::create_proof(gpu, p, a, b, c, in, aux, d0, d1, d2, r, s, r.size());
  std::ofstream o(argv[2], std::ios::binary);
  o.write(reinterpret_cast<const char*>(proofs.data()), proofs.size() * sizeof(Groth16::Proof));
  return 0;
}
"""


@pytest.mark.gpu
def test_host_dev_engine_cpp_and_the_chain_agree(ctx, eng):
    """Context (host _batch), bls_groth16_prove_dev, DeviceEngine and Groth16::create_proof give the same bytes, and they
    equal the chain groth16_h + five msm_batch calls + the assembly from the existing point ops on the host"""
    import torch
    import pairing_b200._native as nat
    toy = Toy(40, 3, 40, 5, 0x5151)
    host = _proof(toy.prove(ctx))
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to(eng.device)  # noqa: E731
    pr = toy.params
    dparams = nat.Groth16Params(pr.alpha_g1, pr.beta_g1, pr.delta_g1, pr.beta_g2, pr.delta_g2, *(dev(getattr(pr, q)) for q in ("h", "l", "a", "b_g1", "b_g2")))
    targs = [dev(x) for x in (*toy.abc, toy.input, toy.aux)]
    got = eng.groth16_prove(dparams, *targs, toy.densities, dev(toy.r), dev(toy.s))
    assert _proof([t.cpu().numpy().view(np.uint64) for t in got]).tobytes() == host.tobytes()
    # the raw _dev call on a stream of its own, with the scratch the query states
    m, length, ni, na = toy.m, toy.len, toy.input.shape[1], toy.aux.shape[1]
    pc = nat.groth16_params_c(dparams, lambda t: t.data_ptr(), lambda t: t.shape[0])
    dw = [nat.density_words(d, bits, "d") for d, bits in zip(toy.densities, (na, ni, na))]
    scratch = torch.empty(ctx.groth16_prove_scratch_bytes(pc, length, ni, na, dw, m), dtype=torch.uint8, device=eng.device)
    out = torch.empty((m, nat.W_PROOF), dtype=torch.int64, device=eng.device)
    tr, ts = dev(toy.r), dev(toy.s)
    st = torch.cuda.Stream(eng.device)
    st.wait_stream(torch.cuda.current_stream(eng.device))
    with torch.cuda.stream(st):
        ctx.call_dev("bls_groth16_prove_dev", ctypes.byref(pc), targs[0].data_ptr(), targs[1].data_ptr(), targs[2].data_ptr(), length,
                     targs[3].data_ptr(), ni, targs[4].data_ptr(), na, *[nat._p(w) for w in dw], tr.data_ptr(), ts.data_ptr(), m,
                     out.data_ptr(), scratch.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert out.cpu().numpy().view(np.uint64).tobytes() == host.tobytes()
    # the C++ mirror
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe, fin, fout = (os.path.join(d, x) for x in ("p.cpp", "p", "in", "out"))
        open(src, "w").write(CPP_PROVE)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        with open(fin, "wb") as f:
            for x in (np.stack([pr.alpha_g1, pr.beta_g1, pr.delta_g1]), np.stack([pr.beta_g2, pr.delta_g2]), pr.h, pr.l, pr.a, pr.b_g1, pr.b_g2,
                      *toy.abc, toy.input, toy.aux, *dw, toy.r, toy.s):
                raw = np.ascontiguousarray(x).tobytes()
                f.write(np.uint64(len(raw)).tobytes() + raw)
        subprocess.check_call([exe, fin, fout], timeout=300)
        assert np.fromfile(fout, dtype=np.uint64).tobytes() == host.tobytes()
    # the chain: H, the five multiexps over host-compacted scalars, the r / s terms and sums with the point ops
    repr_ = lambda x: _limbs([bm.fr_from_mont(v) for v in _ints(x)])  # noqa: E731
    h = eng.groth16_h(*targs[:3]).cpu().numpy().view(np.uint64)
    a_aux, b_in, b_aux = toy.densities
    sa = np.stack([np.concatenate([repr_(toy.input[j]), repr_(toy.aux[j])[a_aux]]) for j in range(m)])
    sb = np.stack([np.concatenate([repr_(toy.input[j])[b_in], repr_(toy.aux[j])[b_aux]]) for j in range(m)])
    sl = np.stack([repr_(toy.aux[j]) for j in range(m)])
    h_ans, l_ans = ctx.g1_msm_batch(pr.h, h), ctx.g1_msm_batch(pr.l, sl)
    a_ans, b1_ans, b2_ans = ctx.g1_msm_batch(pr.a, sa), ctx.g1_msm_batch(pr.b_g1, sb), ctx.g2_msm_batch(pr.b_g2, sb)
    rk, sk = repr_(toy.r), repr_(toy.s)
    rsk = _limbs([x * y % R for x, y in zip(_ints(rk), _ints(sk))])
    rep = lambda row, g2=False: np.repeat((o.g2_from_affine if g2 else o.g1_from_affine)(row[None]), m, 0)  # noqa: E731
    add = lambda x, y, g2=False: (ctx.g2_op if g2 else ctx.g1_op)("add", x, y)  # noqa: E731
    A = add(add(ctx.g1_mul(rep(pr.delta_g1), rk), rep(pr.alpha_g1)), a_ans)
    B = add(add(ctx.g2_mul(rep(pr.delta_g2, True), sk), rep(pr.beta_g2, True), True), b2_ans, True)
    C = ctx.g1_mul(rep(pr.delta_g1), rsk)
    C = add(C, ctx.g1_mul(add(a_ans, rep(pr.alpha_g1)), sk))
    C = add(C, ctx.g1_mul(add(b1_ans, rep(pr.beta_g1)), rk))
    C = add(add(C, h_ans), l_ans)
    chain = _proof((ctx.g1_into_affine(A), ctx.g2_into_affine(B), ctx.g1_into_affine(C)))
    assert chain.tobytes() == host.tobytes()


@pytest.mark.gpu
def test_invalid_arguments(ctx):
    """delta at infinity, each query too short, NULL pointers where there is work, m and lengths past the limits"""
    import pairing_b200._native as nat
    lib, cx = ctx._lib, ctx._ctx
    toy = Toy(5, 2, 3, 2, 0x1BAE)
    m, length, ni, na = toy.m, toy.len, 2, 3
    assert sum(toy.densities[0]) > 0 and sum(toy.densities[2]) > 0 and sum(toy.densities[1]) > 0
    dw = [nat.density_words(d, bits, "d") for d, bits in zip(toy.densities, (na, ni, na))]
    arrs = [*toy.abc, toy.input, toy.aux]

    def call(pc, ptrs=None, m_=m, length_=length, ni_=ni, na_=na, dens=None, rs=None):
        p = [nat._p(x) for x in arrs] if ptrs is None else ptrs
        d = [nat._p(w) for w in dw] if dens is None else dens
        r_, s_ = (nat._p(toy.r), nat._p(toy.s)) if rs is None else rs
        out = np.zeros((max(m_, 1), nat.W_PROOF), dtype=np.uint64)
        rc = lib.bls_groth16_prove_batch(cx, ctypes.byref(pc), p[0], p[1], p[2], length_, p[3], ni_, p[4], na_, *d, r_, s_, m_, nat._p(out))
        sb = lib.bls_groth16_prove_scratch_bytes(cx, ctypes.byref(pc), length_, ni_, na_, *d, m_)
        # the _dev call only where the arguments are rejected: it returns before any work, so the placeholder device
        # pointers are never used
        rcd = lib.bls_groth16_prove_dev(cx, ctypes.byref(pc), 1, 1, 1, length_, 1, ni_, 1, na_, *d, 1, 1, m_, 1, 1, None) if sb == 0 else None
        return rc, rcd, sb

    good = nat.groth16_params_c(toy.params, nat._p, len)
    assert call(good)[0] == 0 and call(good)[2] > 0
    for field in ("delta_g1", "delta_g2"):
        pc = nat.groth16_params_c(toy.params, nat._p, len)
        getattr(pc, field)[-1] = 1
        assert call(pc) == (-1, -1, 0), field
    needs = {"h_len": (1 << (length - 1).bit_length()) - 1, "l_len": na, "a_len": ni + int(toy.densities[0].sum()),
             "b_len": int(toy.densities[1].sum() + toy.densities[2].sum())}
    for field, need in needs.items():
        pc = nat.groth16_params_c(toy.params, nat._p, len)
        setattr(pc, field, need - 1)
        assert call(pc) == (-1, -1, 0), field
        setattr(pc, field, need)
        assert call(pc)[0] == 0, field
    for q in ("h", "l", "a", "b_g1", "b_g2"):
        pc = nat.groth16_params_c(toy.params, nat._p, len)
        setattr(pc, q, None)
        assert call(pc) == (-1, -1, 0), q
    for i in range(5):
        ptrs = [nat._p(x) for x in arrs]
        ptrs[i] = None
        assert call(good, ptrs=ptrs)[0] == -1, i
    dev_args = [1, 1, 1, length, 1, ni, 1, na, *[nat._p(w) for w in dw], 1, 1, m, 1, 1, None]
    for i in (0, 1, 2, 4, 6, 11, 12, 14, 15):                            # a, b, c, input, aux, r, s, out, scratch
        args = list(dev_args)
        args[i] = None
        assert lib.bls_groth16_prove_dev(cx, ctypes.byref(good), *args) == -1, i
    for i in range(3):
        d = [nat._p(w) for w in dw]
        d[i] = None
        assert call(good, dens=d) == (-1, -1, 0), i
    assert call(good, rs=(None, nat._p(toy.s)))[0] == -1
    assert call(good, rs=(nat._p(toy.r), None))[0] == -1
    # limits: m <= 2^16, m * (each multiexp length) <= 2^26
    big = nat.groth16_params_c(toy.params, nat._p, len)
    big.h_len = big.l_len = big.a_len = big.b_len = 1 << 27
    assert lib.bls_groth16_prove_scratch_bytes(cx, ctypes.byref(big), 1, 1, 0, None, nat._p(np.ones(1, np.uint32)), None, (1 << 16) + 1) == 0
    assert lib.bls_groth16_prove_scratch_bytes(cx, ctypes.byref(big), (1 << 20) + 1, 1, 0, None, nat._p(np.ones(1, np.uint32)), None, 64) == 0
    many = np.zeros((1 << 21) // 32 + 1, dtype=np.uint32)
    assert lib.bls_groth16_prove_scratch_bytes(cx, ctypes.byref(big), 2, 1, 1 << 21, nat._p(many), nat._p(np.ones(1, np.uint32)), nat._p(many), 64) == 0
    assert lib.bls_groth16_prove_scratch_bytes(cx, ctypes.byref(big), 2, 1, 1 << 20, nat._p(many), nat._p(np.ones(1, np.uint32)), nat._p(many), 64) > 0
    with pytest.raises(ValueError):
        ctx.groth16_prove(toy.params, *toy.abc[:2], toy.abc[2][:, :-1], toy.input, toy.aux, toy.densities, toy.r, toy.s)
    with pytest.raises(ValueError):
        ctx.groth16_prove(toy.params, *toy.abc, toy.input, toy.aux, (toy.densities[0][:-1],) + toy.densities[1:], toy.r, toy.s)
