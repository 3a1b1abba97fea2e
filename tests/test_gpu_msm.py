"""Multi-scalar multiplication sum_i k_i * P_i (bls_g1_msm / bls_g2_msm and their _dev forms), byte-compared with results built
from oracle operations the KATs pin: the closed form [sum k_i a_i mod r] g for bases P_i = [a_i] g (bench.make_inputs), and the
direct sum (oracle mul per point, a pairwise tree of oracle adds, normalisation) at small n, which also covers bases outside
the r-order subgroup."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import bls_model as m
import datagen as dg
import oracle_lib as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = m.R_ORDER
SEED = 0x3A5E
N_MAX = 1 << 20
CURVES = [pytest.param(False, id="g1"), pytest.param(True, id="g2")]
WINDOWS = [2, 3, 5, 8, 11, 13, 16, 20]


def _limbs(values):
    return np.array([m.limbs64(v % (1 << 256), 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _ints(k):
    k = np.ascontiguousarray(k, dtype=np.uint64).astype(object)
    return k[:, 0] + (k[:, 1] << 64) + (k[:, 2] << 128) + (k[:, 3] << 192)


def _splitmix_scalars(seed, n, full=True):
    """full 256-bit scalars (not reduced mod r); full=False: the bench.make_inputs formula (< 2^254, bit 1 set)"""
    k = dg.splitmix64(seed, 4 * n).reshape(n, 4)
    if not full:
        k[:, 3] &= np.uint64((1 << 62) - 1)
        k[:, 0] |= np.uint64(2)
    return k


def _base_exponents(g2, n):
    """a_i of the bases P_i = [a_i] g that bench.make_inputs(eng, N_MAX, SEED) returns"""
    return _splitmix_scalars(SEED ^ (0x2222 if g2 else 0x1111), N_MAX, full=False)[:n]


def _ops(g2):
    if g2:
        return o.g2_op, o.g2_from_affine, o.g2_into_affine, 1
    return o.g1_op, o.g1_from_affine, o.g1_into_affine, 0


def _zero(g2):
    _, from_aff, _, idx = _ops(g2)
    inf = np.zeros((1, 25 if g2 else 13), dtype=np.uint64)
    inf[0, -1] = 1
    return from_aff(inf)


def _normalise(g2, p):
    _, from_aff, into_aff, _ = _ops(g2)
    return from_aff(into_aff(p))


def _closed_form(g2, a, k):
    """[sum k_i a_i mod r] g, normalised"""
    op, from_aff, _, idx = _ops(g2)
    s = int((_ints(k) * _ints(a)).sum()) % R if len(k) else 0
    g = from_aff(o.generators()[idx])
    return _normalise(g2, op("mul", g, k=_limbs([s])))


def _direct_sum(g2, bases, k):
    """oracle mul per point, pairwise tree of oracle adds, normalised"""
    op, from_aff, _, _ = _ops(g2)
    if len(k) == 0:
        return _zero(g2)
    p = op("mul", from_aff(bases), k=k, threads=o.default_threads())
    while p.shape[0] > 1:
        if p.shape[0] % 2:
            p = np.concatenate([p, _zero(g2)])
        p = op("add", p[0::2], p[1::2], threads=o.default_threads())
    return _normalise(g2, p)


@pytest.fixture(scope="module")
def eng(ctx):
    from pairing_b200.device import DeviceEngine
    return DeviceEngine(ctx=ctx)


@pytest.fixture(scope="module")
def inputs(eng):
    """bench.make_inputs' subgroup points (G1, G2 affine, device and host) and full 256-bit scalars"""
    import torch
    import bench
    pa, qa, _, _ = bench.make_inputs(eng, N_MAX, SEED, torch, np)
    k = _splitmix_scalars(0x77AA, N_MAX)
    return {False: pa, True: qa, "host": {False: pa.cpu().numpy().view(np.uint64), True: qa.cpu().numpy().view(np.uint64)}, "k": k}


def _dev(eng, g2, bases, k, window=0):
    import torch
    tb = torch.from_numpy(np.ascontiguousarray(bases).view(np.int64)).to(eng.device)
    tk = torch.from_numpy(np.ascontiguousarray(k).view(np.int64)).to(eng.device)
    return eng.msm(tb, tk, g2=g2, window=window).cpu().numpy().view(np.uint64)


def _host(ctx, g2, bases, k):
    return (ctx.g2_msm if g2 else ctx.g1_msm)(bases, k)


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
@pytest.mark.parametrize("n", [0, 1, 2, 3, 31, 1000, 1 << 16, 1 << 20])
def test_sizes_against_the_closed_form(ctx, inputs, g2, n):
    bases, k = inputs["host"][g2][:n], inputs["k"][:n]
    got = _host(ctx, g2, bases, k)
    assert got.tobytes() == _closed_form(g2, _base_exponents(g2, n), k).tobytes()


@pytest.mark.gpu
def test_g1_2_22_tiled_bases_distinct_scalars(ctx, inputs):
    n = 1 << 22
    bases = np.tile(inputs["host"][False], (4, 1))
    a = np.tile(_base_exponents(False, N_MAX), (4, 1))
    k = _splitmix_scalars(0x99CC, n)
    assert len(np.unique(k[:, 0])) > n - 16
    assert _host(ctx, False, bases, k).tobytes() == _closed_form(False, a, k).tobytes()


def _window_edge_scalars(c):
    """2^(cj), 2^(cj) - 1, every digit +2^(c-1), every raw digit 2^(c-1) + 1 (negative digits, carries), every raw digit
    2^(c-1) - 1 after a carry, for the windows of width c"""
    nwin = (257 + c - 1) // c
    out = []
    for j in range(nwin):
        out += [1 << (c * j), (1 << (c * j)) - 1]
    out.append(sum((1 << (c - 1)) << (c * j) for j in range(nwin)))
    out.append(sum(((1 << (c - 1)) + 1) << (c * j) for j in range(nwin)))
    out.append(sum(((1 << (c - 1)) - 1) << (c * j) for j in range(nwin)) + 1)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
@pytest.mark.parametrize("c", WINDOWS)
def test_explicit_windows_through_dev(eng, inputs, g2, c):
    """n = 1000 with window c on bls_g*_msm_dev: the window-specific edge scalars first, then random 256-bit ones"""
    n = 1000
    edge = [0, 1, R - 1, R, R + 1, (1 << 256) - 1] + _window_edge_scalars(c)
    k = inputs["k"][:n].copy()
    k[:len(edge)] = _limbs(edge)
    got = _dev(eng, g2, inputs["host"][g2][:n], k, window=c)
    assert got.tobytes() == _closed_form(g2, _base_exponents(g2, n), k).tobytes()


def _off_subgroup_bases(ctx, g2, n, seed):
    """get_point_from_x outputs without cofactor clearing: curve points outside the r-order subgroup"""
    x = dg.rand_field(3 * n, 2 if g2 else 1, seed)
    aff, ok = ctx.point_from_x(g2, x, np.arange(3 * n) & 1)
    aff = aff[ok.astype(bool)][:n]
    assert aff.shape[0] == n
    return aff


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
@pytest.mark.parametrize("window", [0, 4, 7])
def test_edge_scalars_and_off_subgroup_bases_against_the_direct_sum(ctx, eng, inputs, g2, window):
    edge = [0, 1, R - 1, R, R + 1, (1 << 256) - 1] + _window_edge_scalars(window or 8)
    n = 3 * len(edge)
    bases = np.concatenate([inputs["host"][g2][:len(edge)], _off_subgroup_bases(ctx, g2, 2 * len(edge), 0x51 + window)])
    bases[[5, 17, n - 1]] = 0
    bases[[5, 17, n - 1], -1] = 1                                  # infinity bases sprinkled in
    k = np.concatenate([_limbs(edge), _limbs(edge[::-1]), _splitmix_scalars(0x4242, len(edge))])
    want = _direct_sum(g2, bases, k).tobytes()
    assert _dev(eng, g2, bases, k, window=window).tobytes() == want
    if window == 0:
        assert _host(ctx, g2, bases, k).tobytes() == want


def _negate_affine(g2, aff):
    out = aff.copy()
    w = 12 if g2 else 6
    out[:, w:2 * w] = o.fq_op("neg", out[:, w:2 * w].reshape(-1, 6))[0].reshape(-1, w)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_degenerate_base_sets(ctx, inputs, g2):
    host = inputs["host"][g2]
    op, from_aff, _, _ = _ops(g2)
    zero = _zero(g2).tobytes()
    # n copies of one base with k = 1: nP, built through the doubling branch of the bucket sums
    for n in (2, 3, 1000):
        got = _host(ctx, g2, np.repeat(host[:1], n, 0), _limbs([1] * n))
        assert got.tobytes() == _normalise(g2, op("mul", from_aff(host[:1]), k=_limbs([n]))).tobytes(), n
    # P and -P with equal scalars; many pairs cancelling to G::zero(); all bases infinity; all scalars zero
    neg = _negate_affine(g2, host[:64])
    k = inputs["k"][:64]
    assert _host(ctx, g2, np.concatenate([host[:1], neg[:1]]), np.concatenate([k[:1], k[:1]])).tobytes() == zero
    assert _host(ctx, g2, np.concatenate([host[:64], neg]), np.concatenate([k, k])).tobytes() == zero
    inf = host[:64].copy()
    inf[:] = 0
    inf[:, -1] = 1
    assert _host(ctx, g2, inf, k).tobytes() == zero
    assert _host(ctx, g2, host[:64], np.zeros_like(k)).tobytes() == zero
    assert _host(ctx, g2, host[:0], k[:0]).tobytes() == zero


def _time_ms(eng, g2, tb, tk, reps=3):
    import torch
    eng.msm(tb, tk, g2=g2)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.msm(tb, tk, g2=g2)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_all_scalars_equal_is_correct_and_not_slow(eng, inputs, g2):
    """2^16 equal scalars put every entry of a window into ONE bucket: the accumulation is split by entries, not buckets"""
    import torch
    n = 1 << 16
    tb = inputs[g2][:n].contiguous()
    same = np.repeat(inputs["k"][:1], n, 0)
    rand = inputs["k"][:n]
    t_same = torch.from_numpy(same.view(np.int64)).to(eng.device)
    t_rand = torch.from_numpy(np.ascontiguousarray(rand).view(np.int64)).to(eng.device)
    got = eng.msm(tb, t_same, g2=g2).cpu().numpy().view(np.uint64)
    assert got.tobytes() == _closed_form(g2, _base_exponents(g2, n), same).tobytes()
    ms_same, ms_rand = _time_ms(eng, g2, tb, t_same), _time_ms(eng, g2, tb, t_rand)
    assert ms_same < 5 * ms_rand, (ms_same, ms_rand)


@pytest.mark.gpu
@pytest.mark.parametrize("g2", CURVES)
def test_host_dev_and_engine_calls_agree(ctx, eng, inputs, g2):
    from pairing_b200 import engine
    n = 1 << 16
    bases, k = inputs["host"][g2][:n], inputs["k"][:n]
    launches = ctx.launch_count
    host = _host(ctx, g2, bases, k)
    assert ctx.launch_count > launches
    assert _dev(eng, g2, bases, k).tobytes() == host.tobytes()
    curve = engine.G2 if g2 else engine.G1
    assert curve.multiexp(bases, k, ctx=ctx).tobytes() == host.tobytes()


@pytest.mark.gpu
def test_invalid_arguments(ctx, inputs):
    import ctypes
    lib = ctx._lib
    b, k = inputs["host"][False][:8], inputs["k"][:8]
    out = np.zeros((1, 18), dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    assert lib.bls_g1_msm(ctx._ctx, None, vp(k), 8, vp(out)) == -1
    assert lib.bls_g1_msm(ctx._ctx, vp(b), vp(k), 8, None) == -1
    assert lib.bls_g1_msm(ctx._ctx, vp(b), vp(k), (1 << 26) + 1, vp(out)) == -1
    for window in (1, 21, -1):
        assert lib.bls_msm_scratch_bytes(ctx._ctx, 1, 8, window) == 0
        assert lib.bls_g1_msm_dev(ctx._ctx, 1, 1, 8, window, 1, 1, None) == -1
    assert lib.bls_msm_scratch_bytes(ctx._ctx, 3, 8, 0) == 0
    assert lib.bls_msm_scratch_bytes(ctx._ctx, 1, 1 << 24, 2) == 0           # 129 windows x 2^24 entries: above 2^31
    assert lib.bls_msm_scratch_bytes(ctx._ctx, 2, 1 << 20, 0) > 0


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_g1_msm(None, None, None, 0, None) == -1
    assert lib.bls_g2_msm_dev(None, None, None, 0, 0, None, None, None) == -1
    assert lib.bls_msm_scratch_bytes(None, 1, 16, 0) == 0


CPP_MSM = r"""
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
int main(int, char** argv) {
  Gpu gpu(0);
  auto k = load<FrRepr>(argv[3]);
  G1Point s1 = G1::multiexp(gpu, load<G1AffinePoint>(argv[1]), k);
  G2Point s2 = G2::multiexp(gpu, load<G2AffinePoint>(argv[2]), k);
  std::ofstream(argv[4], std::ios::binary).write(reinterpret_cast<const char*>(&s1), sizeof(s1)).write(reinterpret_cast<const char*>(&s2), sizeof(s2));
  return 0;
}
"""


@pytest.mark.gpu
def test_cpp_mirror_multiexp(ctx, inputs):
    import pairing_b200._native as nat
    n = 4096
    p1, p2, k = inputs["host"][False][:n], inputs["host"][True][:n], inputs["k"][:n]
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "msm.cpp"), os.path.join(d, "msm")
        open(src, "w").write(CPP_MSM)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        files = [os.path.join(d, f) for f in ("p1", "p2", "k", "out")]
        for f, a in zip(files, (p1, p2, k)):
            np.ascontiguousarray(a).tofile(f)
        subprocess.check_call([exe] + files, timeout=300)
        got = np.fromfile(files[3], dtype=np.uint64)
    assert got.tobytes() == ctx.g1_msm(p1, k).tobytes() + ctx.g2_msm(p2, k).tobytes()
