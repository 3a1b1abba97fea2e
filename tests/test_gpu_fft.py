"""Radix-2 FFT over Fr (bls_fr_fft_batch / bls_fr_fft_dev): bellman's EvaluationDomain fft / ifft / coset_fft / icoset_fft,
byte-compared with the big-int model tests/fr_fft_model.py::fr_fft, which is itself checked here against a direct O(n^2) DFT.
Outputs are canonical Montgomery values, so every comparison is bit for bit whatever order the kernels compute in."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import bls_model as m
import datagen as dg
import fr_fft_model as fm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = m.R_ORDER
KINDS = ["fft", "ifft", "coset_fft", "icoset_fft"]
INVERSE = {"fft": "ifft", "coset_fft": "icoset_fft"}
# fr.rs PrimeField constants, as the crate stores them (Montgomery limbs)
ROOT_OF_UNITY = [0xb9b58d8c5f0e466a, 0x5b1b4c801819d7ec, 0x0af53ae352a31e64, 0x5bf3adda19e9b27b]
GENERATOR = [0x0000000efffffff1, 0x17e363d300189c0f, 0xff9c57876f8457b0, 0x351332208fc5a8c4]


def _ints(a):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).astype(object)
    return list(a[:, 0] + (a[:, 1] << 64) + (a[:, 2] << 128) + (a[:, 3] << 192))


def _limbs(values):
    return np.array([m.limbs64(v, 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _inputs(m_polys, log_n, seed):
    """(m, n, 4) random canonical Montgomery values with 0, Montgomery one and r - 1 planted in"""
    total = m_polys << log_n
    a = dg.rand_scalars(total, seed, edge_cases=False)
    for i, v in enumerate([0, m.FR_MONT_R, R - 1]):
        a[(i * 0x9E37) % total] = m.limbs64(v, 4)
    return a.reshape(m_polys, 1 << log_n, 4)


def _model(kind, a, log_n):
    """model transform of every polynomial of an (m, n, 4) array"""
    return np.stack([_limbs(fm.fr_fft(kind, _ints(p), log_n)) for p in a]).reshape(a.shape)


def _closed_form(kind, coeffs, log_n, idx):
    """out[i] at the indices idx of the transform of a sparse polynomial {j: Montgomery value} (the table of the header)"""
    n = 1 << log_n
    w = fm.fr_root(log_n)
    inv = kind in ("ifft", "icoset_fft")
    if inv:
        w = pow(w, -1, R)
    a = {j: m.fr_from_mont(v) for j, v in coeffs.items()}
    if kind == "coset_fft":
        a = {j: v * pow(fm.FR_GENERATOR, j, R) % R for j, v in a.items()}
    out = []
    for i in idx:
        s = sum(v * pow(w, i * j % n, R) for j, v in a.items()) % R
        if inv:
            s = s * pow(n, -1, R) % R
        if kind == "icoset_fft":
            s = s * pow(fm.FR_GENERATOR, -i, R) % R
        out.append(m.fr_to_mont(s))
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_constants_match_the_crate():
    w32 = fm.fr_root(32)
    assert m.limbs64(m.fr_to_mont(w32), 4) == ROOT_OF_UNITY
    assert m.limbs64(m.fr_to_mont(fm.FR_GENERATOR), 4) == GENERATOR
    assert pow(w32, 1 << 32, R) == 1 and pow(w32, 1 << 31, R) != 1
    assert (R - 1) % (1 << 32) == 0 and ((R - 1) >> 32) % 2 == 1
    assert pow(fm.FR_GENERATOR, (R - 1) // 2, R) == R - 1          # 7 is a quadratic non-residue


def test_generated_twiddle_constants_match_the_model():
    """pairing_b200/csrc/fr_fft_consts.cuh (tools/gen_fr_fft_consts.py) against the model's constants"""
    src = open(os.path.join(ROOT, "pairing_b200", "csrc", "fr_fft_consts.cuh")).read()
    tables = {}
    for name, body in re.findall(r"__constant__ Fr (\w+)\[\d+\] = \{(.*?)\n\};", src, re.S):
        rows = re.findall(r"\{\{([^}]*)\}\}", body)
        tables[name] = [m.fr_from_mont(sum(int(x.strip().rstrip("u"), 16) << (32 * i) for i, x in enumerate(r.split(",")))) for r in rows]
    w, g = fm.fr_root(32), fm.FR_GENERATOR
    assert tables["FR_ROOT_POW"] == [pow(w, 1 << b, R) for b in range(32)]
    assert tables["FR_ROOT_INV_POW"] == [pow(w, -(1 << b), R) for b in range(32)]
    assert tables["FR_GEN_POW"] == [pow(g, 1 << b, R) for b in range(28)]
    assert tables["FR_GEN_INV_POW"] == [pow(g, -(1 << b), R) for b in range(28)]
    assert tables["FR_INV_2POW"] == [pow(1 << L, -1, R) for L in range(29)]


@pytest.mark.parametrize("log_n", range(7))
def test_model_against_direct_dft(log_n):
    """every n = 2^log_n from 1 to 64, all four kinds, against the O(n^2) definition; the inverse kinds undo the forward ones"""
    n = 1 << log_n
    a = _ints(_inputs(1, log_n, 0x51 + log_n))
    coeffs = dict(enumerate(a))
    for kind in KINDS:
        got = fm.fr_fft(kind, a, log_n)
        assert got == _closed_form(kind, coeffs, log_n, range(n)), kind
        if kind in INVERSE:
            assert fm.fr_fft(INVERSE[kind], got, log_n) == a


def test_fft_kernels_do_not_spill():
    """the FFT kernels keep their state in registers and shared memory (cuobjdump --dump-resource-usage of the built library)"""
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
    fft = {k: v for k, v in usage.items() if "k_fr_fft_pass" in k or "k_fft_tables" in k}
    assert len(fft) == 2, sorted(usage)
    for k, v in fft.items():
        assert v["STACK"] == 0 and v["LOCAL"] == 0, (k, v)
    assert fft[[k for k in fft if "k_fr_fft_pass" in k][0]]["REG"] <= 85                # 3 blocks of 256 threads per SM


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_fr_fft_batch(None, 0, None, None, 4, 1) == -1
    assert lib.bls_fr_fft_dev(None, 0, None, None, 4, 1, None, None) == -1
    assert lib.bls_fr_fft_scratch_bytes(None, 4, 1) == 0


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


@pytest.mark.gpu
@pytest.mark.parametrize("m_polys", [1, 3])
@pytest.mark.parametrize("log_n", range(15))
def test_small_sizes_match_the_model(ctx, log_n, m_polys):
    a = _inputs(m_polys, log_n, 0x1000 + 7 * log_n + m_polys)
    for kind in KINDS:
        got = ctx.fr_fft(kind, a)
        assert got.tobytes() == _model(kind, a, log_n).tobytes(), kind


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,m_polys", [(16, 3), (20, 1)])
def test_multi_pass_sizes_match_the_model(ctx, log_n, m_polys):
    a = _inputs(m_polys, log_n, 0x2000 + log_n)
    for kind in KINDS:
        assert ctx.fr_fft(kind, a).tobytes() == _model(kind, a, log_n).tobytes(), kind


def _random_device(eng, n, seed):
    """(n, 4) canonical values (< 2^252 < r) drawn on the device"""
    import torch
    gen = torch.Generator(device=eng.device).manual_seed(seed)
    a = torch.randint(-(1 << 63), (1 << 63) - 1, (n, 4), dtype=torch.int64, device=eng.device, generator=gen)
    a[:, 3] &= (1 << 60) - 1
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [24, 28])
def test_large_round_trips(eng, log_n):
    """a dense random polynomial comes back from fft -> ifft and coset_fft -> icoset_fft, compared on the device"""
    import torch
    a = _random_device(eng, 1 << log_n, log_n)
    for fwd, inv in INVERSE.items():
        f = eng.fr_fft(a, fwd)
        assert not torch.equal(f, a)
        back = eng.fr_fft(f, inv, out=f)                 # in place
        assert torch.equal(back, a), fwd
        del f, back
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [24, 28])
def test_large_sparse_inputs_match_the_closed_form(eng, log_n):
    """64 random non-zero coefficients; every kind at 1024 sampled output indices"""
    import torch
    n = 1 << log_n
    rng = np.random.default_rng(log_n)
    pos = sorted(set(int(x) for x in rng.integers(0, n, 64)) | {0, n - 1})
    vals = _ints(dg.rand_scalars(len(pos), 0x3000 + log_n, edge_cases=False))
    a = torch.zeros((n, 4), dtype=torch.int64, device=eng.device)
    a[torch.tensor(pos, device=eng.device)] = _dev(eng, _limbs(vals))
    idx = sorted(set(int(x) for x in rng.integers(0, n, 1024 - 2)) | {0, n - 1})
    tidx = torch.tensor(idx, device=eng.device)
    coeffs = dict(zip(pos, vals))
    out = torch.empty_like(a)
    for kind in KINDS:
        got = _host(eng.fr_fft(a, kind, out=out)[tidx])
        assert got.tobytes() == _limbs(_closed_form(kind, coeffs, log_n, idx)).tobytes(), kind
    del a, out
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_dense_2_24_at_sampled_indices(eng):
    """a dense random polynomial of 2^24 coefficients, fft at 4 indices, each a Horner evaluation at omega^i"""
    import torch
    log_n = 24
    n = 1 << log_n
    a = _random_device(eng, n, 99)
    idx = [0, 1, 12345, n - 1]
    got = _host(eng.fr_fft(a, "fft")[torch.tensor(idx, device=eng.device)])
    coeffs = [m.fr_from_mont(v) for v in _ints(_host(a))]
    w = fm.fr_root(log_n)
    want = []
    for i in idx:
        x, s = pow(w, i, R), 0
        for c in reversed(coeffs):
            s = (s * x + c) % R
        want.append(m.fr_to_mont(s))
    assert got.tobytes() == _limbs(want).tobytes()


@pytest.mark.gpu
def test_polynomial_multiplication(ctx):
    """ifft(fft(a) * fft(b)) with the element-wise product of bls_fr_op_batch is the cyclic convolution of a and b"""
    log_n = 10
    n = 1 << log_n
    a, b = _inputs(1, log_n, 0x4001)[0], _inputs(1, log_n, 0x4002)[0]
    fa, fb = ctx.fr_fft("fft", a), ctx.fr_fft("fft", b)
    prod, ok = ctx.fr_op("mul", fa, fb)
    assert ok.all()
    got = ctx.fr_fft("ifft", prod)
    x, y = [m.fr_from_mont(v) for v in _ints(a)], [m.fr_from_mont(v) for v in _ints(b)]
    want = [0] * n
    for i, xi in enumerate(x):
        for j, yj in enumerate(y):
            want[(i + j) % n] += xi * yj
    assert got.tobytes() == _limbs([m.fr_to_mont(v % R) for v in want]).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,m_polys", [(6, 5), (10, 2), (16, 2), (22, 1)])      # one, two and three passes
def test_in_place_equals_out_of_place(eng, log_n, m_polys):
    import torch
    a = _random_device(eng, m_polys << log_n, log_n).reshape(m_polys, 1 << log_n, 4)
    keep = a.clone()
    for kind in KINDS:
        out = eng.fr_fft(a, kind)
        assert torch.equal(a, keep), "an out-of-place call changed its input"
        b = a.clone()
        assert eng.fr_fft(b, kind, out=b).data_ptr() == b.data_ptr()
        assert torch.equal(b, out), kind


@pytest.mark.gpu
def test_zero_polynomials(ctx, eng):
    import torch
    assert ctx.fr_fft("fft", np.zeros((0, 1024, 4), dtype=np.uint64)).shape == (0, 1024, 4)
    e = torch.empty((0, 16, 4), dtype=torch.int64, device=eng.device)
    assert eng.fr_fft(e, "icoset_fft").shape == (0, 16, 4)
    ctx.call_dev("bls_fr_fft_dev", 0, None, None, 10, 0, None, None)


CPP_FFT = r"""
#include <fstream>
#include "pairing_b200.hpp"
using namespace pairing_b200;
int main(int, char** argv) {
  Gpu gpu(0);
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<bls_fr> a(raw.size() / sizeof(bls_fr));
  std::memcpy(a.data(), raw.data(), a.size() * sizeof(bls_fr));
  const int log_n = std::atoi(argv[2]);
  std::ofstream o(argv[3], std::ios::binary);
  for (auto* fn : {&FrField::fft, &FrField::ifft, &FrField::coset_fft, &FrField::icoset_fft}) {
    auto r = fn(gpu, a, log_n);
    o.write(reinterpret_cast<const char*>(r.data()), r.size() * sizeof(bls_fr));
  }
  return 0;
}
"""


@pytest.mark.gpu
def test_host_dev_engine_and_cpp_agree(ctx, eng):
    import torch
    import pairing_b200._native as nat
    log_n, m_polys = 12, 3
    a = _inputs(m_polys, log_n, 0x5005)
    host = {k: ctx.fr_fft(k, a) for k in KINDS}
    ta = _dev(eng, a.reshape(m_polys, 1 << log_n, 4))
    scratch = torch.empty(ctx.fr_fft_scratch_bytes(log_n, m_polys), dtype=torch.uint8, device=eng.device)
    for kind in KINDS:
        assert _host(eng.fr_fft(ta, kind)).tobytes() == host[kind].tobytes(), kind
        out = torch.empty_like(ta)
        ctx.call_dev("bls_fr_fft_dev", nat.FFT_KINDS[kind], ta.data_ptr(), out.data_ptr(), log_n, m_polys, scratch.data_ptr(), eng._stream())
        assert _host(out).tobytes() == host[kind].tobytes(), kind
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe, fin, fout = (os.path.join(d, x) for x in ("fft.cpp", "fft", "in", "out"))
        open(src, "w").write(CPP_FFT)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        a.tofile(fin)
        subprocess.check_call([exe, fin, str(log_n), fout], timeout=300)
        got = np.fromfile(fout, dtype=np.uint64)
    assert got.tobytes() == b"".join(host[k].tobytes() for k in KINDS)


def _time_ms(eng, t, reps=5):
    import torch
    out = torch.empty_like(t)
    eng.fr_fft(t, "fft", out=out)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.fr_fft(t, "fft", out=out)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


@pytest.mark.gpu
def test_batch_of_small_polynomials_fills_the_gpu(eng):
    """256 polynomials of 2^10 take less than twice the time of one polynomial of 2^18 (the same number of elements)"""
    many = _random_device(eng, 1 << 18, 7).reshape(256, 1 << 10, 4)
    one = _random_device(eng, 1 << 18, 8)
    ms_many, ms_one = _time_ms(eng, many), _time_ms(eng, one)
    assert ms_many < 2 * ms_one, (ms_many, ms_one)


@pytest.mark.gpu
def test_invalid_arguments(ctx):
    lib = ctx._lib
    c = ctx._ctx
    buf = np.zeros((16, 4), dtype=np.uint64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    for kind in (-1, 4):
        assert lib.bls_fr_fft_batch(c, kind, p, p, 4, 1) == -1
        assert lib.bls_fr_fft_dev(c, kind, 1, 1, 4, 1, 1, None) == -1
    for log_n, m_polys in ((-1, 1), (29, 1), (20, 1025), (0, (1 << 30) + 1), (28, 5)):
        assert lib.bls_fr_fft_batch(c, 0, p, p, log_n, m_polys) == -1
        assert lib.bls_fr_fft_dev(c, 0, 1, 1, log_n, m_polys, 1, None) == -1
        assert lib.bls_fr_fft_scratch_bytes(c, log_n, m_polys) == 0
    assert lib.bls_fr_fft_scratch_bytes(c, 20, 1024) > 0
    assert lib.bls_fr_fft_batch(c, 0, None, p, 4, 1) == -1
    assert lib.bls_fr_fft_batch(c, 0, p, None, 4, 1) == -1
    for ptrs in ((None, 1, 1), (1, None, 1), (1, 1, None)):
        assert lib.bls_fr_fft_dev(c, 0, ptrs[0], ptrs[1], 4, 1, ptrs[2], None) == -1
    with pytest.raises(ValueError):
        ctx.fr_fft_scratch_bytes(29)
