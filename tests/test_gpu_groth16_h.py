"""Groth16's quotient polynomial H (bls_fr_groth16_h_batch / _dev, DeviceEngine.groth16_h) and the Fr element-wise ops on
device pointers (bls_fr_op_dev).  H is byte-compared with the big-int model tests/groth16_h_model.py, which is itself
checked here against the defining identity H(tau) (tau^n - 1) = A(tau) B(tau) - C(tau) of satisfied inputs.  Outputs are
canonical FrRepr, so every comparison is bit for bit whatever order the kernels compute in."""
import ctypes
import os
import random
import re
import subprocess
import tempfile

import numpy as np
import pytest

import bls_model as m
import datagen as dg
import fr_fft_model as fm
import groth16_h_model as gm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = m.R_ORDER


def _ints(a):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).astype(object)
    return list(a[:, 0] + (a[:, 1] << 64) + (a[:, 2] << 128) + (a[:, 3] << 192))


def _limbs(values):
    return np.array([m.limbs64(v, 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _eval(coeffs, x):
    """Horner: sum_i coeffs[i] x^i mod r (canonical coefficients)"""
    s = 0
    for c in reversed(coeffs):
        s = (s * x + c) % R
    return s


def _lagrange_eval(values, log_n, tau):
    """the polynomial of degree < n through (omega^i, values[i]) (canonical values, zero-padded to n) at tau, tau^n != 1:
    sum_i v_i omega^i (tau^n - 1) / (n (tau - omega^i))"""
    n = 1 << log_n
    w = fm.fr_root(log_n)
    zt = (pow(tau, n, R) - 1) % R
    s, wi = 0, 1
    for v in list(values) + [0] * (n - len(values)):
        s += v * wi * pow(tau - wi, -1, R)
        wi = wi * w % R
    return s * zt * pow(n, -1, R) % R


def _proofs(m_proofs, length, seed, satisfied):
    """(m, len, 4) Montgomery a, b, c: random (an unsatisfied system) or with c_i = a_i b_i; 0, one and r - 1 planted in"""
    total = m_proofs * length
    a = dg.rand_scalars(total, seed, edge_cases=False)
    b = dg.rand_scalars(total, seed + 1, edge_cases=False)
    for i, v in enumerate([0, m.FR_MONT_R, R - 1][:total]):
        a[(i * 0x9E37) % total] = m.limbs64(v, 4)
        b[(i * 0x7F4B + 1) % total] = m.limbs64(v, 4)
    if satisfied:
        c = _limbs([m.fr_to_mont(m.fr_from_mont(x) * m.fr_from_mont(y) % R) for x, y in zip(_ints(a), _ints(b))])
    else:
        c = dg.rand_scalars(total, seed + 2, edge_cases=False)
    return tuple(x.reshape(m_proofs, length, 4) for x in (a, b, c))


def _model(a, b, c):
    """(m, len, 4) inputs -> (m, n - 1, 4) model output"""
    n1 = (1 << gm.domain_log(a.shape[1])) - 1
    return np.stack([_limbs(gm.groth16_h(_ints(x), _ints(y), _ints(z))) for x, y, z in zip(a, b, c)]).reshape(a.shape[0], n1, 4)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("length", range(1, 41))
def test_model_against_the_definition(length):
    """satisfied inputs: H(tau) (tau^n - 1) = A(tau) B(tau) - C(tau) at a random tau with A, B, C Lagrange-evaluated from
    the evaluations, and the dropped coefficient is 0; random inputs: the same identity on the coset g omega^i, where
    (A B - C) / z(g) is what H interpolates"""
    rng = random.Random(length)
    log_n = gm.domain_log(length)
    n = 1 << log_n
    for satisfied in (True, False):
        a, b, c = (_ints(x) for x in _proofs(1, length, 0x600 + length, satisfied))
        full = gm.groth16_h_full(a, b, c)
        assert len(full) == n and gm.groth16_h(a, b, c) == full[:-1]
        ca, cb, cc = ([m.fr_from_mont(v) for v in x] for x in (a, b, c))
        if satisfied:
            assert full[-1] == 0
            taus = [rng.randrange(R) for _ in range(2)]
        else:
            w = fm.fr_root(log_n)
            taus = [fm.FR_GENERATOR * pow(w, rng.randrange(n), R) % R for _ in range(2)]
        for tau in taus:
            lhs = _eval(full, tau) * (pow(tau, n, R) - 1) % R
            rhs = (_lagrange_eval(ca, log_n, tau) * _lagrange_eval(cb, log_n, tau) - _lagrange_eval(cc, log_n, tau)) % R
            assert lhs == rhs, (satisfied, tau)


def test_generated_z_inv_table_matches_the_model():
    """FR_Z_INV of pairing_b200/csrc/fr_fft_consts.cuh (tools/gen_fr_fft_consts.py) against the model"""
    src = open(os.path.join(ROOT, "pairing_b200", "csrc", "fr_fft_consts.cuh")).read()
    body = re.search(r"__constant__ Fr FR_Z_INV\[29\] = \{(.*?)\n\};", src, re.S).group(1)
    rows = re.findall(r"\{\{([^}]*)\}\}", body)
    got = [m.fr_from_mont(sum(int(x.strip().rstrip("u"), 16) << (32 * i) for i, x in enumerate(r.split(",")))) for r in rows]
    assert got == [gm.z_inv(L) for L in range(29)]
    assert all(z * (pow(fm.FR_GENERATOR, 1 << L, R) - 1) % R == 1 for L, z in enumerate(got))


def test_groth16_h_kernels_do_not_spill():
    """the gather, combine and conversion kernels keep their state in registers (cuobjdump --dump-resource-usage)"""
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
    new = {k: v for k, v in usage.items() if any(s in k for s in ("k_fr_h_gather", "k_fr_h_combine", "k_fr_into_repr_truncate"))}
    assert len(new) == 3, sorted(usage)
    for k, v in new.items():
        assert v["STACK"] == 0 and v["LOCAL"] == 0, (k, v)


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_fr_groth16_h_batch(None, None, None, None, 16, 1, None) == -1
    assert lib.bls_fr_groth16_h_dev(None, None, None, None, 16, 1, None, None, None) == -1
    assert lib.bls_fr_groth16_h_scratch_bytes(None, 16, 1) == 0
    assert lib.bls_fr_op_dev(None, 0, None, None, None, None, 4, None) == -1


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def eng(ctx):
    from pairing_b200.device import DeviceEngine
    return DeviceEngine(ctx=ctx)


def _dev(eng, a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(eng.device)


def _host(t):
    return t.cpu().numpy().view(np.uint64)


def _random_device(eng, n, seed):
    """(n, 4) canonical values (< 2^252 < r) drawn on the device"""
    import torch
    gen = torch.Generator(device=eng.device).manual_seed(seed)
    a = torch.randint(-(1 << 63), (1 << 63) - 1, (n, 4), dtype=torch.int64, device=eng.device, generator=gen)
    a[:, 3] &= (1 << 60) - 1
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("m_proofs", [1, 3])
@pytest.mark.parametrize("length", [1, 2, 3, 5, 8, 1000, 1024, 1025, 4097, 1 << 16])
def test_matches_the_model(ctx, length, m_proofs):
    """random (unsatisfied) and satisfied inputs, one- and two-pass transforms; the inputs are left unchanged"""
    for satisfied in (False, True):
        a, b, c = _proofs(m_proofs, length, 0x7000 + 17 * length + m_proofs, satisfied)
        keep = [x.copy() for x in (a, b, c)]
        got = ctx.fr_groth16_h(a, b, c)
        assert got.tobytes() == _model(a, b, c).tobytes(), satisfied
        assert all(np.array_equal(x, y) for x, y in zip((a, b, c), keep))
        if m_proofs == 1:
            assert ctx.fr_groth16_h(a[0], b[0], c[0]).tobytes() == got.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("length", [(1 << 20) + 1, 1 << 22])
def test_large_satisfied_inputs_satisfy_the_identity(eng, length):
    """n = 2^21 (three passes) and 2^22: H(tau) (tau^n - 1) = A(tau) B(tau) - C(tau) at two random tau, with A, B and C's
    coefficients from fr_fft's ifft and every polynomial evaluated by Horner; the device inputs are left unchanged"""
    import torch
    log_n = gm.domain_log(length)
    n = 1 << log_n
    a, b = _random_device(eng, length, length), _random_device(eng, length, length + 1)
    c, ok = eng.fr_op("mul", a, b)
    assert bool(ok.all())
    keep = [x.clone() for x in (a, b, c)]
    h = eng.groth16_h(a, b, c)
    assert tuple(h.shape) == (n - 1, 4)
    assert all(torch.equal(x, y) for x, y in zip((a, b, c), keep))
    rng = random.Random(length)
    taus = [rng.randrange(R) for _ in range(2)]
    evals = []
    for x in (a, b, c):
        pad = torch.zeros((n, 4), dtype=torch.int64, device=eng.device)
        pad[:length] = x
        coeffs = _ints(_host(eng.fr_op("into_repr", eng.fr_fft(pad, "ifft"))[0]))
        evals.append([_eval(coeffs, t) for t in taus])
        del pad
    hc = _ints(_host(h))
    for i, t in enumerate(taus):
        assert _eval(hc, t) * (pow(t, n, R) - 1) % R == (evals[0][i] * evals[1][i] - evals[2][i]) % R, t
    del a, b, c, h, keep
    torch.cuda.empty_cache()


CPP_H = r"""
#include <fstream>
#include "pairing_b200.hpp"
using namespace pairing_b200;
int main(int, char** argv) {
  Gpu gpu(0);
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  const size_t total = raw.size() / (3 * sizeof(bls_fr)), m = std::atoi(argv[2]);
  std::vector<bls_fr> a(total), b(total), c(total);
  std::memcpy(a.data(), raw.data(), total * sizeof(bls_fr));
  std::memcpy(b.data(), raw.data() + total * sizeof(bls_fr), total * sizeof(bls_fr));
  std::memcpy(c.data(), raw.data() + 2 * total * sizeof(bls_fr), total * sizeof(bls_fr));
  auto h = FrField::groth16_h(gpu, a, b, c, m);
  std::ofstream o(argv[3], std::ios::binary);
  o.write(reinterpret_cast<const char*>(h.data()), h.size() * sizeof(FrRepr));
  return 0;
}
"""


@pytest.mark.gpu
def test_host_dev_engine_and_cpp_agree(ctx, eng):
    import torch
    import pairing_b200._native as nat
    length, m_proofs = 1000, 3
    a, b, c = _proofs(m_proofs, length, 0x8008, False)
    host = ctx.fr_groth16_h(a, b, c)
    ta, tb, tc = (_dev(eng, x) for x in (a, b, c))
    assert _host(eng.groth16_h(ta, tb, tc)).tobytes() == host.tobytes()
    out = torch.empty((m_proofs, 1023, 4), dtype=torch.int64, device=eng.device)
    scratch = torch.empty(ctx.fr_groth16_h_scratch_bytes(length, m_proofs), dtype=torch.uint8, device=eng.device)
    ctx.call_dev("bls_fr_groth16_h_dev", ta.data_ptr(), tb.data_ptr(), tc.data_ptr(), length, m_proofs, out.data_ptr(),
                 scratch.data_ptr(), eng._stream())
    assert _host(out).tobytes() == host.tobytes()
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe, fin, fout = (os.path.join(d, x) for x in ("h.cpp", "h", "in", "out"))
        open(src, "w").write(CPP_H)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        np.concatenate([a.reshape(-1), b.reshape(-1), c.reshape(-1)]).tofile(fin)
        subprocess.check_call([exe, fin, str(m_proofs), fout], timeout=300)
        got = np.fromfile(fout, dtype=np.uint64)
    assert got.tobytes() == host.tobytes()


@pytest.mark.gpu
def test_device_resident_chain_into_msm_batch(ctx, eng):
    """groth16_h -> msm_batch against n - 1 shared G1 bases with no host copy in between equals bls_g1_msm_batch over the
    model's H"""
    length, m_proofs = 1000, 3
    a, b, c = _proofs(m_proofs, length, 0x9009, False)
    bases = dg.g1_affine_points(1023, 0x900A, infinity_at=(5,))
    h = eng.groth16_h(*(_dev(eng, x) for x in (a, b, c)))
    got = eng.msm_batch(_dev(eng, bases), h)
    assert _host(got).tobytes() == ctx.g1_msm_batch(bases, _model(a, b, c)).tobytes()


FR_OPS = ["add", "sub", "mul", "sqr", "neg", "dbl", "inv", "from_repr", "into_repr"]


@pytest.mark.gpu
@pytest.mark.parametrize("op", FR_OPS)
def test_fr_op_dev_equals_the_host_call(ctx, eng, op):
    """every op of bls_fr_op_batch, ok flags included: zero for inv, values >= r (up to 2^256 - 1) for from_repr"""
    import torch
    n = 3000
    a = dg.rand_scalars(n, 0xA000 + FR_OPS.index(op))
    b = dg.rand_scalars(n, 0xB000 + FR_OPS.index(op))
    a[5] = 0
    if op == "from_repr":
        for i, v in enumerate([R, R + 1, (1 << 256) - 1, R - 1]):
            a[10 + i] = m.limbs64(v, 4)
        a[100:200] = dg.splitmix64(0xC0, 400).reshape(100, 4)
    binary = op in ("add", "sub", "mul")
    want, want_ok = ctx.fr_op(op, a, b if binary else None)
    ta, tb = _dev(eng, a), _dev(eng, b)
    out, ok = eng.fr_op(op, ta, tb if binary else None)
    assert _host(out).tobytes() == want.tobytes()
    assert ok.cpu().numpy().tobytes() == want_ok.tobytes()
    if op == "inv":                                                       # rand_scalars' edge cases put a 0 at row 0 too
        zero = ~a.any(axis=1)
        assert zero[5] and np.array_equal(want_ok, (~zero).astype(np.uint8))
    if op == "from_repr":
        assert not want_ok[10:13].any() and want_ok[13]
    same, _ = eng.fr_op(op, ta, tb if binary else None, out=ta)          # in place
    assert same.data_ptr() == ta.data_ptr() and _host(ta).tobytes() == want.tobytes()
    ctx.call_dev("bls_fr_op_dev", 2, 0, 0, 0, None, 0, None)              # n = 0
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_zero_proofs_and_short_inputs(ctx, eng):
    import torch
    assert ctx.fr_groth16_h(*[np.zeros((0, 100, 4), dtype=np.uint64)] * 3).shape == (0, 127, 4)
    assert ctx.fr_groth16_h(*[np.ones((4, 1, 4), dtype=np.uint64)] * 3).shape == (4, 0, 4)
    assert ctx.fr_groth16_h(*[np.zeros((0, 4), dtype=np.uint64)] * 3).shape == (0, 4)
    e = torch.empty((2, 1, 4), dtype=torch.int64, device=eng.device)
    assert eng.groth16_h(e, e, e).shape == (2, 0, 4)
    ctx.call_dev("bls_fr_groth16_h_dev", None, None, None, 100, 0, None, None, None)
    ctx.call_dev("bls_fr_groth16_h_dev", None, None, None, 1, 5, None, None, None)


def _median_ms(fn, flush, reps=7):
    import torch
    fn()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


@pytest.mark.gpu
def test_one_call_costs_about_its_transforms(eng):
    """at 2^20, m = 1, the call takes at most 1.15x the fr_fft calls it contains (ifft and coset_fft of 3 polynomials,
    icoset_fft of 1), timed in the same process with 256 MiB written between launches"""
    import torch
    log_n = 20
    n = 1 << log_n
    a, b, c = (_random_device(eng, n, 0xD00 + i) for i in range(3))
    out = torch.empty((n - 1, 4), dtype=torch.int64, device=eng.device)
    abc = torch.stack([a, b, c])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)

    def transforms():
        eng.fr_fft(abc, "ifft", out=abc)
        eng.fr_fft(abc, "coset_fft", out=abc)
        eng.fr_fft(abc[0], "icoset_fft", out=abc[0])

    ms_call = _median_ms(lambda: eng.groth16_h(a, b, c, out=out), flush)
    ms_fft = _median_ms(transforms, flush)
    assert ms_call <= 1.15 * ms_fft, (ms_call, ms_fft)


@pytest.mark.gpu
def test_invalid_arguments(ctx, eng):
    lib = ctx._lib
    cx = ctx._ctx
    buf = np.zeros((64, 4), dtype=np.uint64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    # log_n > 28, m * n > 2^28
    for length, m_proofs in (((1 << 28) + 1, 1), (1 << 28, 2), ((1 << 20) + 1, 129), (1 << 20, 257), (2, (1 << 27) + 1)):
        assert lib.bls_fr_groth16_h_batch(cx, p, p, p, length, m_proofs, p) == -1
        assert lib.bls_fr_groth16_h_dev(cx, 1, 1, 1, length, m_proofs, 1, 1, None) == -1
        assert lib.bls_fr_groth16_h_scratch_bytes(cx, length, m_proofs) == 0
    assert lib.bls_fr_groth16_h_scratch_bytes(cx, 1 << 28, 1) > 0
    assert lib.bls_fr_groth16_h_scratch_bytes(cx, 1 << 20, 256) > 0
    assert lib.bls_fr_groth16_h_scratch_bytes(cx, 2, 1 << 27) > 0
    for i in range(4):
        ptrs = [p] * 4
        ptrs[i] = None
        assert lib.bls_fr_groth16_h_batch(cx, ptrs[0], ptrs[1], ptrs[2], 16, 1, ptrs[3]) == -1
    for i in range(5):
        ptrs = [1] * 5
        ptrs[i] = None
        assert lib.bls_fr_groth16_h_dev(cx, ptrs[0], ptrs[1], ptrs[2], 16, 1, ptrs[3], ptrs[4], None) == -1
    with pytest.raises(ValueError):
        ctx.fr_groth16_h_scratch_bytes((1 << 28) + 1)
    with pytest.raises(ValueError):
        ctx.fr_groth16_h(buf[:8], buf[:8], buf[:9])
    # bls_fr_op_dev: unknown ops, NULL a / out, NULL b for a binary op
    for op in (-1, 9, 17):
        assert lib.bls_fr_op_dev(cx, op, 1, 1, 1, None, 4, None) == -1
    assert lib.bls_fr_op_dev(cx, 0, None, 1, 1, None, 4, None) == -1
    assert lib.bls_fr_op_dev(cx, 0, 1, 1, None, None, 4, None) == -1
    assert lib.bls_fr_op_dev(cx, 2, 1, None, 1, None, 4, None) == -1
