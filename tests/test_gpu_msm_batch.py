"""Batched multi-scalar multiplication: m independent sums in one call (bls_g1_msm_batch / bls_g2_msm_batch and their _dev
forms), byte-compared with the closed form [sum_i k_ji a_ji mod r] g for bases [a_ji] g, with the direct sum per row, and with
one bls_g*_msm call per row.  The helpers and inputs are test_gpu_msm.py's."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as o
from test_gpu_msm import (CURVES, N_MAX, R, ROOT, WINDOWS, _base_exponents, _direct_sum, _host, _ints, _limbs,
                          _negate_affine, _normalise, _off_subgroup_bases, _ops, _splitmix_scalars, _window_edge_scalars,
                          _zero, eng, inputs)  # noqa: F401 -- eng and inputs are fixtures

MODES = [pytest.param(True, id="shared"), pytest.param(False, id="separate")]


def _closed_forms(g2, a, k):
    """k (m, n, 4) scalars against bases [a] g, a (n, 4) shared or (m, n, 4): the m normalised rows
    [sum_i k_ji a_ji mod r] g, all oracle multiplications in one call"""
    op, from_aff, _, idx = _ops(g2)
    m_, n = k.shape[:2]
    if m_ == 0:
        return np.zeros((0, 36 if g2 else 18), dtype=np.uint64)
    if n == 0:
        return np.repeat(_zero(g2), m_, 0)
    ki = _ints(k.reshape(-1, 4)).reshape(m_, n)
    ai = _ints(np.broadcast_to(a, k.shape).reshape(-1, 4)).reshape(m_, n)
    s = [int(x) % R for x in (ki * ai).sum(axis=1)]
    g = np.repeat(from_aff(o.generators()[idx]), m_, 0)
    return _normalise(g2, op("mul", g, k=_limbs(s), threads=o.default_threads()))


def _batch(ctx, g2, bases, k):
    return (ctx.g2_msm_batch if g2 else ctx.g1_msm_batch)(bases, k)


def _dev_batch(eng, g2, bases, k, window=0):
    import torch
    tb = torch.from_numpy(np.ascontiguousarray(bases).view(np.int64)).to(eng.device)
    tk = torch.from_numpy(np.ascontiguousarray(k).view(np.int64)).to(eng.device)
    return eng.msm_batch(tb, tk, g2=g2, window=window).cpu().numpy().view(np.uint64)


def _rows(inputs, g2, m_, n, shared):
    """bases and their exponents: the first n points (shared) or the first m n points as m rows"""
    host, a = inputs["host"][g2], _base_exponents(g2, N_MAX)
    if shared:
        return host[:n], a[:n]
    return host[:m_ * n].reshape(m_, n, host.shape[1]), a[:m_ * n].reshape(m_, n, 4)


# ------------------------------------------------------------------------------------------------ 1. the closed form
@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_separate_bases_256_rows_of_4096_against_the_closed_form(ctx, inputs, g2):
    """the 2^20 points of bench.make_inputs split into 256 rows of 4096, each row its own bases"""
    m_, n = 256, 4096
    bases, a = _rows(inputs, g2, m_, n, shared=False)
    k = inputs["k"].reshape(m_, n, 4)
    assert _batch(ctx, g2, bases, k).tobytes() == _closed_forms(g2, a, k).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_shared_bases_64_rows_of_2_14_against_the_closed_form(ctx, inputs, g2):
    m_, n = 64, 1 << 14
    bases, a = _rows(inputs, g2, m_, n, shared=True)
    k = _splitmix_scalars(0x6414, m_ * n).reshape(m_, n, 4)
    assert _batch(ctx, g2, bases, k).tobytes() == _closed_forms(g2, a, k).tobytes()


@pytest.mark.gpu
def test_g1_shared_bases_4_rows_of_2_20_against_the_closed_form(ctx, inputs):
    m_, n = 4, N_MAX
    bases, a = _rows(inputs, False, m_, n, shared=True)
    k = _splitmix_scalars(0x4220, m_ * n).reshape(m_, n, 4)
    assert _batch(ctx, False, bases, k).tobytes() == _closed_forms(False, a, k).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("shared", MODES)
@pytest.mark.parametrize("g2", CURVES)
def test_ragged_shapes_against_the_closed_form(ctx, inputs, g2, shared):
    for m_ in (1, 2, 3, 7, 129):
        for n in (0, 1, 2, 31, 1000):
            bases, a = _rows(inputs, g2, m_, n, shared)
            k = inputs["k"][:m_ * n].reshape(m_, n, 4)
            assert _batch(ctx, g2, bases, k).tobytes() == _closed_forms(g2, a, k).tobytes(), (m_, n)


# ------------------------------------------------------------------------------------------------ 2. explicit windows
@pytest.mark.gpu
@pytest.mark.parametrize("shared", MODES)
@pytest.mark.parametrize("g2", CURVES)
@pytest.mark.parametrize("c", WINDOWS)
def test_explicit_windows_through_dev(eng, inputs, g2, c, shared):
    """m = 3, n = 1000 on bls_g*_msm_batch_dev with window c: the window-edge scalars in row 0, the edge scalars
    0, 1, r - 1, r, r + 1, 2^256 - 1 in row 1, random 256-bit scalars everywhere else"""
    m_, n = 3, 1000
    k = inputs["k"][:m_ * n].reshape(m_, n, 4).copy()
    edge = _window_edge_scalars(c)
    k[0, :len(edge)] = _limbs(edge)
    k[1, :6] = _limbs([0, 1, R - 1, R, R + 1, (1 << 256) - 1])
    bases, a = _rows(inputs, g2, m_, n, shared)
    assert _dev_batch(eng, g2, bases, k, window=c).tobytes() == _closed_forms(g2, a, k).tobytes()


# ------------------------------------------------------------------------------------------------ 3. the direct sum
@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
@pytest.mark.parametrize("window", [0, 4, 7])
def test_off_subgroup_bases_against_the_direct_sum(ctx, eng, inputs, g2, window):
    """rows of subgroup and off-subgroup bases with infinity bases sprinkled in; edge, reversed edge and random scalars"""
    edge = [0, 1, R - 1, R, R + 1, (1 << 256) - 1] + _window_edge_scalars(window or 8)
    n = len(edge)
    bases = np.concatenate([inputs["host"][g2][:n], _off_subgroup_bases(ctx, g2, 2 * n, 0x61 + window)])
    bases[[5, n + 3, 2 * n + 1, 3 * n - 1]] = 0
    bases[[5, n + 3, 2 * n + 1, 3 * n - 1], -1] = 1
    k = np.concatenate([_limbs(edge), _limbs(edge[::-1]), _splitmix_scalars(0x4343, n)]).reshape(3, n, 4)
    bases = bases.reshape(3, n, -1)
    want = np.concatenate([_direct_sum(g2, bases[j], k[j]) for j in range(3)])
    assert _dev_batch(eng, g2, bases, k, window=window).tobytes() == want.tobytes()
    shared = np.concatenate([_direct_sum(g2, bases[1], k[j]) for j in range(3)])       # row 1's bases for every sum
    assert _dev_batch(eng, g2, bases[1], k, window=window).tobytes() == shared.tobytes()
    if window == 0:
        assert _batch(ctx, g2, bases, k).tobytes() == want.tobytes()


# ------------------------------------------------------------------------------------------------ 4. rows are independent
@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_degenerate_rows_equal_their_own_single_msm(ctx, inputs, g2):
    n = 1000
    host, k = inputs["host"][g2], inputs["k"]
    rows_b, rows_k = [], []
    rows_b.append(host[:n]); rows_k.append(np.zeros((n, 4), dtype=np.uint64))                          # zero scalars
    inf = host[:n].copy()
    inf[:] = 0
    inf[:, -1] = 1
    rows_b.append(inf); rows_k.append(k[:n])                                                            # infinity bases
    half = n // 2
    rows_b.append(np.concatenate([host[:half], _negate_affine(g2, host[:half])]))                      # P and -P cancel
    rows_k.append(np.concatenate([k[:half], k[:half]]))
    rows_b.append(np.repeat(host[:1], n, 0)); rows_k.append(_limbs([1] * n))                           # nP by doublings
    rows_b.append(host[n:2 * n]); rows_k.append(np.repeat(k[7:8], n, 0))                               # all-equal scalars
    for j in range(5):                                                                                  # random rows
        rows_b.append(host[(2 + j) * n:(3 + j) * n]); rows_k.append(k[(3 + j) * n:(4 + j) * n])
    bases, scalars = np.stack(rows_b), np.stack(rows_k)
    got = _batch(ctx, g2, bases, scalars)
    for j in range(len(rows_b)):
        assert got[j:j + 1].tobytes() == _host(ctx, g2, bases[j], scalars[j]).tobytes(), j
    zero = _zero(g2).tobytes()
    assert got[0:1].tobytes() == got[1:2].tobytes() == got[2:3].tobytes() == zero


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_one_row_is_the_single_msm_bit_for_bit(ctx, inputs, g2):
    n = 1 << 16
    bases, k = inputs["host"][g2][:n], inputs["k"][:n]
    single = _host(ctx, g2, bases, k).tobytes()
    assert _batch(ctx, g2, bases, k[None]).tobytes() == single
    assert _batch(ctx, g2, bases[None], k[None]).tobytes() == single


# ------------------------------------------------------------------------------------------------ 5. every layer agrees
@pytest.mark.gpu
@pytest.mark.parametrize("shared", MODES)
@pytest.mark.parametrize("g2", CURVES)
def test_host_dev_and_engine_calls_agree(ctx, eng, inputs, g2, shared):
    from pairing_b200 import engine
    m_, n = 16, 4096
    bases, _ = _rows(inputs, g2, m_, n, shared)
    k = inputs["k"][:m_ * n].reshape(m_, n, 4)
    launches = ctx.launch_count
    host = _batch(ctx, g2, bases, k)
    assert ctx.launch_count > launches
    assert _dev_batch(eng, g2, bases, k).tobytes() == host.tobytes()
    curve = engine.G2 if g2 else engine.G1
    assert curve.multiexp_batch(bases, k, ctx=ctx).tobytes() == host.tobytes()


CPP_MSM_BATCH = r"""
#include <cstdio>
#include <fstream>
#include "pairing_b200.hpp"
using namespace pairing_b200;
template <class T> static std::vector<T> load(const char* path) {
  std::ifstream f(path, std::ios::binary);
  std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<T> v(raw.size() / sizeof(T));
  std::memcpy(v.data(), raw.data(), v.size() * sizeof(T));
  return v;
}
template <class T> static void save(std::ofstream& f, const std::vector<T>& v) {
  f.write(reinterpret_cast<const char*>(v.data()), v.size() * sizeof(T));
}
int main(int, char** argv) {
  Gpu gpu(0);
  const size_t m = 8;
  auto k = load<FrRepr>(argv[3]);
  auto p1 = load<G1AffinePoint>(argv[1]);
  auto p2 = load<G2AffinePoint>(argv[2]);
  std::vector<G1AffinePoint> s1(p1.begin(), p1.begin() + k.size() / m);
  std::vector<G2AffinePoint> s2(p2.begin(), p2.begin() + k.size() / m);
  std::ofstream out(argv[4], std::ios::binary);
  save(out, G1::multiexp_batch(gpu, p1, k, m));
  save(out, G2::multiexp_batch(gpu, p2, k, m));
  save(out, G1::multiexp_batch(gpu, s1, k, m));
  save(out, G2::multiexp_batch(gpu, s2, k, m));
  try {
    G1::multiexp_batch(gpu, std::vector<G1AffinePoint>(p1.begin(), p1.begin() + 3), k, m);
    return 2;
  } catch (const Error&) {
  }
  return 0;
}
"""


@pytest.mark.gpu
def test_cpp_mirror_multiexp_batch(ctx, inputs):
    import pairing_b200._native as nat
    m_, n = 8, 512
    p1, p2 = inputs["host"][False][:m_ * n], inputs["host"][True][:m_ * n]
    k = inputs["k"][:m_ * n]
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "msm_batch.cpp"), os.path.join(d, "msm_batch")
        open(src, "w").write(CPP_MSM_BATCH)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        files = [os.path.join(d, f) for f in ("p1", "p2", "k", "out")]
        for f, a in zip(files, (p1, p2, k)):
            np.ascontiguousarray(a).tofile(f)
        subprocess.check_call([exe] + files, timeout=300)
        got = np.fromfile(files[3], dtype=np.uint64)
    k3 = k.reshape(m_, n, 4)
    want = [ctx.g1_msm_batch(p1.reshape(m_, n, -1), k3), ctx.g2_msm_batch(p2.reshape(m_, n, -1), k3),
            ctx.g1_msm_batch(p1[:n], k3), ctx.g2_msm_batch(p2[:n], k3)]
    assert got.tobytes() == b"".join(w.tobytes() for w in want)


# ------------------------------------------------------------------------------------------------ 6. timing
def _median_ms(fn, reps=3):
    import torch
    fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_a_batch_beats_a_loop_of_single_msms(eng, inputs, g2):
    """64 sums of 2^12 points over shared bases: one batch call against 64 eng.msm calls, timed with events in one test"""
    import torch
    m_, n = 64, 1 << 12
    tb = inputs[g2][:n].contiguous()
    tk = torch.from_numpy(np.ascontiguousarray(inputs["k"][:m_ * n]).view(np.int64)).to(eng.device).reshape(m_, n, 4)
    out = eng.msm_batch(tb, tk, g2=g2)
    singles = [eng.msm(tb, tk[j], g2=g2) for j in range(m_)]
    assert out.cpu().numpy().tobytes() == torch.cat(singles).cpu().numpy().tobytes()
    ms_batch = _median_ms(lambda: eng.msm_batch(tb, tk, g2=g2, out=out))
    ms_loop = _median_ms(lambda: [eng.msm(tb, tk[j], g2=g2) for j in range(m_)], reps=1)
    assert ms_batch < ms_loop / 8, (ms_batch, ms_loop)


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_all_equal_scalars_in_every_row_is_correct_and_not_slow(eng, inputs, g2):
    """every entry of a (sum, window) in ONE bucket: the accumulation is split by entries, not buckets"""
    import torch
    m_, n = 64, 1 << 12
    tb = inputs[g2][:n].contiguous()
    same = np.repeat(inputs["k"][:m_], n, 0).reshape(m_, n, 4)
    t_same = torch.from_numpy(np.ascontiguousarray(same).view(np.int64)).to(eng.device)
    t_rand = torch.from_numpy(np.ascontiguousarray(inputs["k"][:m_ * n]).view(np.int64)).to(eng.device).reshape(m_, n, 4)
    got = eng.msm_batch(tb, t_same, g2=g2).cpu().numpy().view(np.uint64)
    assert got.tobytes() == _closed_forms(g2, _base_exponents(g2, n), same).tobytes()
    ms_same = _median_ms(lambda: eng.msm_batch(tb, t_same, g2=g2))
    ms_rand = _median_ms(lambda: eng.msm_batch(tb, t_rand, g2=g2))
    assert ms_same < 5 * ms_rand, (ms_same, ms_rand)


# ------------------------------------------------------------------------------------------------ 7. invalid arguments
@pytest.mark.gpu
def test_invalid_arguments(ctx, inputs):
    import ctypes
    lib = ctx._lib
    b, k = inputs["host"][False][:8], inputs["k"][:16]
    out = np.zeros((2, 18), dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    c = ctx._ctx
    for shared in (0, 1):
        assert lib.bls_g1_msm_batch(c, None, shared, vp(k), 8, 2, vp(out)) == -1
        assert lib.bls_g1_msm_batch(c, vp(b), shared, None, 8, 2, vp(out)) == -1
        assert lib.bls_g1_msm_batch(c, vp(b), shared, vp(k), 8, 2, None) == -1
        assert lib.bls_g1_msm_batch_dev(c, None, shared, 1, 8, 2, 0, 1, 1, None) == -1
        assert lib.bls_g1_msm_batch_dev(c, 1, shared, None, 8, 2, 0, 1, 1, None) == -1
        assert lib.bls_g1_msm_batch_dev(c, 1, shared, 1, 8, 2, 0, None, 1, None) == -1
        assert lib.bls_g1_msm_batch_dev(c, 1, shared, 1, 8, 2, 0, 1, None, None) == -1
        assert lib.bls_g2_msm_batch_dev(c, None, shared, 1, 8, 2, 0, 1, 1, None) == -1
    assert lib.bls_g1_msm_batch(c, None, 1, None, 0, 2, vp(out)) == 0                  # n = 0: no pointer is read
    assert lib.bls_g1_msm_batch(c, None, 1, None, 8, 0, None) == 0                     # m = 0: nothing to do
    assert out.tobytes() == np.repeat(_zero(False), 2, 0).tobytes()
    sb = lib.bls_msm_batch_scratch_bytes
    assert sb(c, 1, 1, (1 << 16) + 1, 0) == 0                                            # m > 2^16
    assert lib.bls_g1_msm_batch(c, vp(b), 1, vp(k), 1, (1 << 16) + 1, vp(out)) == -1
    assert sb(c, 1, (1 << 10) + 1, 1 << 16, 0) == 0                                      # m n = 2^26 + 2^16
    assert sb(c, 1, (1 << 26) + 1, 1, 0) == 0 and sb(c, 2, 1 << 26, 1, 0) > 0            # m n = 2^26 + 1 / 2^26
    assert lib.bls_g1_msm_batch(c, vp(b), 1, vp(k), (1 << 26) + 1, 1, vp(out)) == -1
    assert sb(c, 1, 1, 1 << 16, 20) == 0                                                 # m W 2^(c-1) >= 2^31
    assert sb(c, 1, 1 << 10, 1 << 16, 8) == 0                                            # W m n >= 2^31
    assert sb(c, 1, 1 << 10, 1 << 16, 9) > 0
    assert sb(c, 1, 1 << 10, 1 << 16, 0) > 0 and sb(c, 2, 1 << 10, 1 << 16, 0) > 0       # the boundary, library window
    assert lib.bls_g1_msm_batch_dev(c, 1, 1, 1, 1, 1 << 16, 20, 1, 1, None) == -1
    assert sb(c, 3, 8, 2, 0) == 0
    for window in (1, 21, -1):
        assert sb(c, 1, 8, 2, window) == 0
        assert lib.bls_g1_msm_batch_dev(c, 1, 1, 1, 8, 2, window, 1, 1, None) == -1
    for n in (0, 1, 1000, 1 << 16, 1 << 20):
        for window in (0, 2, 8, 16):
            for degree in (1, 2):
                assert lib.bls_msm_scratch_bytes(c, degree, n, window) == sb(c, degree, n, 1, window), (n, window, degree)


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_g1_msm_batch(None, None, 1, None, 0, 1, None) == -1
    assert lib.bls_g2_msm_batch(None, None, 0, None, 0, 1, None) == -1
    assert lib.bls_g1_msm_batch_dev(None, None, 1, None, 0, 1, 0, None, None, None) == -1
    assert lib.bls_g2_msm_batch_dev(None, None, 0, None, 0, 1, 0, None, None, None) == -1
    assert lib.bls_msm_batch_scratch_bytes(None, 1, 16, 4, 0) == 0
