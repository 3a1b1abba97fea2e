"""The point FFT (bls_g1_fft_*, bls_g2_fft_*) and KZG openings at every point of the domain (bls_kzg_open_all_*), with their
Context and DeviceEngine bindings.

Every input point is [a] g for a known exponent a, so a transform is compared bit for bit with [the exponents' transform] g
(tests/point_fft_model.py, itself checked against tests/fr_fft_model.py), and every FK20 proof with bls_kzg_open_batch at
z = omega^k."""
import os
import random
import re

import numpy as np
import pytest

import bls_model as bm
import fr_fft_model as fm
import kzg_model as km
import oracle_lib as o
import point_fft_model as pm
from test_gpu_kzg import Key, _fr, _limbs, _resource_usage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER
W1, W2 = 13, 25
KINDS = ("fft", "ifft", "coset_fft", "icoset_fft")


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_model_point_fft_is_the_fr_fft():
    """the kernels' evaluation order, in exponents, equals fr_fft_model.fr_fft for every kind"""
    rng = random.Random(1)
    for log_n in (0, 1, 2, 3, 5, 8):
        a = [rng.randrange(R) for _ in range(1 << log_n)]
        for kind in KINDS:
            want = [bm.fr_from_mont(v) for v in fm.fr_fft(kind, [bm.fr_to_mont(x) for x in a], log_n)]
            assert pm.point_fft(kind, a, log_n) == want, (log_n, kind)


def test_model_fk20_is_kzg_open_at_every_root():
    """the FK20 construction reproduces kzg_model.open_ at every omega^k"""
    rng = random.Random(2)
    tau = rng.randrange(R)
    for log_n in (0, 1, 2, 6):
        n = 1 << log_n
        srs = km.powers(tau, max(n - 1, 0))
        table = pm.fk20_table(srs + [0], log_n)                          # srs[n - 1] is never read
        w = fm.fr_root(log_n)
        for coeffs in ([rng.randrange(R) for _ in range(n)], [0] * n, [5] + [0] * (n - 1)):
            proofs = pm.fk20_proofs(coeffs, table, log_n)
            assert proofs == [km.open_(coeffs, pow(w, k, R), srs)[1] for k in range(n)], log_n


def test_point_fft_kernels_resources():
    """the new kernels' registers and stack are within DESIGN.md's figures, with no local memory and no shared memory"""
    _, _, usage = _resource_usage()
    #        kernel (G1 = Fp, G2 = Fp2)              max REG  max STACK
    limits = {"k_pfft_bflyIN3bls2Fp": (128, 6144), "k_pfft_bflyIN3bls3Fp2": (168, 8448),
              "k_pfft_mulIN3bls2Fp": (128, 6144), "k_pfft_mulIN3bls3Fp2": (168, 8448),
              "k_pfft_bfly0IN3bls2Fp": (255, 512), "k_pfft_bfly0IN3bls3Fp2": (255, 1536),
              "k_pfft_loadIN3bls2Fp": (96, 0), "k_pfft_loadIN3bls3Fp2": (96, 0),
              "k_pfft_emitIN3bls2Fp": (96, 0), "k_pfft_emitIN3bls3Fp2": (96, 0),
              "k_pfft_take_rev": (32, 0), "k_pfft_tables": (64, 0), "k_fk_w": (64, 0), "k_fk_pad": (64, 0)}
    for kernel, (reg, stack) in limits.items():
        found = [v for k, v in usage.items() if kernel + ("E" if "IN3bls" in kernel else "") in k]
        assert len(found) == 1, (kernel, sorted(k for k in usage if "pfft" in k or "k_fk" in k))
        u = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL|SHARED):(\d+)", found[0])}
        assert u["LOCAL"] == 0 and u["SHARED"] == 0 and u["REG"] <= reg and u["STACK"] <= stack, (kernel, u)
    assert len([k for k in usage if "k_pfft_" in k or "k_fk_" in k]) == len(limits)


def test_preexisting_kernels_resources_unchanged():
    """every kernel the library had before the point FFT unit, the KZG kernels included, keeps its cuobjdump
    --dump-resource-usage line (tests/golden/resource_usage_pre_point_fft.txt: the dump of the parent commit's build)"""
    _, _, usage = _resource_usage()
    before = dict(line.split(" ", 1) for line in open(os.path.join(ROOT, "tests", "golden", "resource_usage_pre_point_fft.txt")).read().splitlines())
    assert len(before) >= 100 and any("k_kzg_" in k for k in before)
    changed = {k: (v, usage.get(k)) for k, v in before.items() if usage.get(k) != v}
    assert not changed, changed


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    for fn in (lib.bls_g1_fft_batch, lib.bls_g2_fft_batch):
        assert fn(None, 0, None, None, 1, 1) == -1
    for fn in (lib.bls_g1_fft_dev, lib.bls_g2_fft_dev):
        assert fn(None, 0, None, None, 1, 1, None, None) == -1
    assert lib.bls_kzg_open_all_prepare(None, None, 1, 1, None) == -1
    assert lib.bls_kzg_open_all_prepare_dev(None, None, 1, 1, None, None, None) == -1
    assert lib.bls_kzg_open_all_batch(None, None, None, 1, 1, None, None) == -1
    assert lib.bls_kzg_open_all_dev(None, None, None, 1, 1, None, None, None, None) == -1
    assert lib.bls_point_fft_scratch_bytes(None, 1, 1, 1) == 0
    assert lib.bls_kzg_open_all_prepare_scratch_bytes(None, 1) == 0
    assert lib.bls_kzg_open_all_scratch_bytes(None, 1, 1) == 0


# ---------------------------------------------------------------------------------------------------------------- GPU

def _gen(g2):
    return o.g2_from_affine(o.generators()[1]) if g2 else o.g1_from_affine(o.generators()[0])


def _pts(ctx, exps, g2=False):
    """[e] g (or [e] h) as affine rows, on the GPU (bls_g*_mul_batch, parity-tested against the oracle)"""
    exps = list(exps)
    if not exps:
        return np.zeros((0, W2 if g2 else W1), np.uint64)
    k = _limbs([e % R for e in exps])
    if g2:
        return ctx.g2_into_affine(ctx.g2_mul(np.repeat(_gen(True), len(exps), 0), k))
    return ctx.g1_into_affine(ctx.g1_mul(np.repeat(_gen(False), len(exps), 0), k))


def _rows(rng, m, n, special):
    """m exponent rows: random, with the identity (0) sprinkled in; special adds a constant row and a delta row"""
    rows = [[0 if rng.random() < 0.05 else rng.randrange(R) for _ in range(n)] for _ in range(m)]
    if special and m >= 3:
        c = rng.randrange(1, R)
        rows[1] = [c] * n                                                  # P + P and P + (-P) inside the butterflies
        rows[2] = [0] * n
        rows[2][rng.randrange(n)] = rng.randrange(1, R)                   # a delta row
    return rows


@pytest.fixture(scope="module")
def eng(ctx):
    from pairing_b200.device import DeviceEngine
    return DeviceEngine(ctx=ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
@pytest.mark.parametrize("log_n", [0, 1, 2, 5, 10, 11, 12])
def test_point_fft_exponent_model(ctx, eng, g2, log_n):
    """inputs [a_j] g; every kind equals [fr_fft(kind, a)_i] g bit for bit, m in {1, 3}, out of place (Context) and in place
    (DeviceEngine, out = a); the constant row gives n P at index 0 and the identity elsewhere"""
    import torch
    rng = random.Random(log_n * 2 + g2)
    n = 1 << log_n
    rows = _rows(rng, 3, n, True)
    pts = _pts(ctx, [e for r in rows for e in r], g2).reshape(3, n, -1)
    fft = ctx.g2_fft if g2 else ctx.g1_fft
    for kind in KINDS:
        want_e = [pm.point_fft(kind, r, log_n) for r in rows]
        want = _pts(ctx, [e for r in want_e for e in r], g2).reshape(3, n, -1)
        assert np.array_equal(fft(kind, pts[0]), want[0]), kind
        assert np.array_equal(fft(kind, pts), want), kind
        if kind == "fft":
            assert want_e[1][0] == n * rows[1][0] % R and not any(want_e[1][1:])
        t = torch.from_numpy(pts.view(np.int64).copy()).to(eng.device)
        (eng.g2_fft if g2 else eng.g1_fft)(t, kind, out=t)
        assert np.array_equal(t.cpu().numpy().view(np.uint64), want), kind


@pytest.mark.gpu
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
def test_point_fft_round_trips(ctx, g2):
    """ifft(fft(x)) == x and icoset_fft(coset_fft(x)) == x as canonical affine rows, identities included"""
    rng = random.Random(0x77 + g2)
    n = 1 << 9
    x = _pts(ctx, [e for r in _rows(rng, 2, n, False) for e in r], g2).reshape(2, n, -1)
    fft = ctx.g2_fft if g2 else ctx.g1_fft
    assert np.array_equal(fft("ifft", fft("fft", x)), x)
    assert np.array_equal(fft("icoset_fft", fft("coset_fft", x)), x)
    ident = _pts(ctx, [0] * 4, g2)
    assert all(np.array_equal(fft(k, ident), ident) for k in KINDS)


@pytest.mark.gpu
def test_g1_fft_2_16_against_fr_fft_and_mul(ctx):
    """log_n = 16: every kind equals bls_fr_fft_batch of the exponents followed by bls_g1_mul_batch of g"""
    rng = random.Random(0x16)
    n = 1 << 16
    a = [rng.randrange(R) for _ in range(n)]
    x = _pts(ctx, a)
    for kind in KINDS:
        e = ctx.fr_op("into_repr", ctx.fr_fft(kind, _fr(a)))[0]
        want = ctx.g1_into_affine(ctx.g1_mul(np.repeat(_gen(False), n, 0), e))
        assert np.array_equal(ctx.g1_fft(kind, x), want), kind


@pytest.mark.gpu
def test_lagrange_srs_commitments(ctx):
    """commit(ifft(srs), evaluations) == commit(srs, coefficients) bit for bit, n = 2^12, m = 4"""
    rng = random.Random(0x1A6)
    log_n, m = 12, 4
    n = 1 << log_n
    tau = rng.randrange(R)
    srs = _pts(ctx, km.powers(tau, n))
    lagrange = ctx.g1_fft("ifft", srs)
    coeffs = _fr([rng.randrange(R) for _ in range(m * n)]).reshape(m, n, 4)
    evals = ctx.fr_fft("fft", coeffs)
    assert np.array_equal(ctx.kzg_commit(lagrange, evals), ctx.kzg_commit(srs, coeffs))


def _open_each(ctx, srs, p, log_n):
    """the chain bls_kzg_open_all replaces: bls_kzg_open_batch of every row at every omega^k"""
    m, n = p.shape[0], 1 << log_n
    w = fm.fr_root(log_n)
    z = _fr([pow(w, k, R) for k in range(n)] * m)
    y, proof = ctx.kzg_open(srs[:max(n - 1, 0)], np.repeat(p, n, axis=0), z)
    return y.reshape(m, n, 4), proof.reshape(m, n, W1), z


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [0, 1, 2, 6, 9])
def test_kzg_open_all_equals_open_at_every_root(ctx, eng, log_n):
    """y and the proofs equal bls_kzg_open_batch at every z = omega^k bit for bit, m in {1, 3} with a zero and a constant
    polynomial; a sample verifies; the table is two identities for n = 1; DeviceEngine and Context agree"""
    import torch
    rng = random.Random(0xF20 + log_n)
    n = 1 << log_n
    key = Key(ctx, 0, tau=rng.randrange(R))
    srs = _pts(ctx, km.powers(key.tau, n))
    table = ctx.kzg_open_all_prepare(srs, log_n)
    assert np.array_equal(table, _pts(ctx, pm.fk20_table(km.powers(key.tau, n), log_n)))
    coeffs = [[rng.randrange(R) for _ in range(n)], [0] * n, [rng.randrange(R)] + [0] * (n - 1)]
    p = _fr([c for r in coeffs for c in r]).reshape(3, n, 4)
    for m in (1, 3):
        y, proof = ctx.kzg_open_all(table, p[:m])
        wy, wproof, z = _open_each(ctx, srs, p[:m], log_n)
        assert np.array_equal(y, wy) and np.array_equal(proof, wproof), m
    sample = rng.sample(range(3 * n), min(8, 3 * n))
    c = np.repeat(ctx.kzg_commit(srs, p), n, axis=0)
    assert ctx.kzg_verify(key.pvk, c[sample], y.reshape(-1, 4)[sample], z[sample], proof.reshape(-1, W1)[sample]).all()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(eng.device)  # noqa: E731
    dtable = eng.kzg_open_all_prepare(dev(srs), log_n)
    assert np.array_equal(dtable.cpu().numpy().view(np.uint64), table)
    dy, dproof = eng.kzg_open_all(dtable, dev(p))
    assert np.array_equal(dy.cpu().numpy().view(np.uint64), y) and np.array_equal(dproof.cpu().numpy().view(np.uint64), proof)


@pytest.mark.gpu
def test_dev_calls_on_their_own_stream_with_exact_scratch(ctx):
    """bls_g1_fft_dev / bls_kzg_open_all_dev with a scratch of exactly _scratch_bytes on a stream of their own give the
    _batch rows"""
    import torch
    rng = random.Random(0xDE5)
    log_n, m = 7, 2
    n = 1 << log_n
    x = _pts(ctx, [rng.randrange(R) for _ in range(m * n)]).reshape(m, n, W1)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to("cuda")  # noqa: E731
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    dx = dev(x)
    out = torch.empty_like(dx)
    scr = torch.empty(ctx.point_fft_scratch_bytes(1, log_n, m), dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(st):
        ctx.call_dev("bls_g1_fft_dev", 2, dx.data_ptr(), out.data_ptr(), log_n, m, scr.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint64), ctx.g1_fft("coset_fft", x))
    srs = _pts(ctx, km.powers(rng.randrange(R), n - 1))
    table = ctx.kzg_open_all_prepare(srs, log_n)
    p = _fr([rng.randrange(R) for _ in range(m * n)]).reshape(m, n, 4)
    dp, dt = dev(p), dev(table)
    y = torch.empty((m, n, 4), dtype=torch.int64, device="cuda")
    pr = torch.empty((m, n, W1), dtype=torch.int64, device="cuda")
    scr = torch.empty(ctx.kzg_scratch_bytes("open_all", log_n, m), dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(st):
        ctx.call_dev("bls_kzg_open_all_dev", dt.data_ptr(), dp.data_ptr(), log_n, m, y.data_ptr(), pr.data_ptr(), scr.data_ptr(), st.cuda_stream)
    st.synchronize()
    wy, wp = ctx.kzg_open_all(table, p)
    assert np.array_equal(y.cpu().numpy().view(np.uint64), wy) and np.array_equal(pr.cpu().numpy().view(np.uint64), wp)


@pytest.mark.gpu
def test_invalid_arguments(ctx):
    """a bad kind, sizes over the limits and NULL pointers where there is work give BLS_ERR_INVALID_ARGUMENT and leave the
    outputs untouched; the scratch sizes of rejected arguments are 0; m = 0 does nothing"""
    lib, cx = ctx._lib, ctx._ctx
    p_ = lambda a: a.ctypes.data_as(__import__("ctypes").c_void_p)  # noqa: E731
    x = _pts(ctx, [1, 2, 3, 4])
    sentinel = np.uint64(0x5A5A5A5A5A5A5A5A)
    out = np.full_like(x, sentinel)
    for fn in (lib.bls_g1_fft_batch, lib.bls_g2_fft_batch):
        assert fn(cx, 4, p_(x), p_(out), 2, 1) == -1 and fn(cx, -1, p_(x), p_(out), 2, 1) == -1
        assert fn(cx, 0, None, p_(out), 2, 1) == -1 and fn(cx, 0, p_(x), None, 2, 1) == -1
        assert fn(cx, 0, None, None, 27, 1) == -1 and fn(cx, 0, None, None, 20, 65) == -1 and fn(cx, 0, None, None, -1, 1) == -1
        assert fn(cx, 0, None, None, 2, 0) == 0
    for fn in (lib.bls_g1_fft_dev, lib.bls_g2_fft_dev):
        assert fn(cx, 0, None, None, 2, 1, None, None) == -1 and fn(cx, 0, None, None, 2, 0, None, None) == 0
    assert (out == sentinel).all()
    for d in (1, 2):
        assert lib.bls_point_fft_scratch_bytes(cx, d, 26, 1) > 0 and lib.bls_point_fft_scratch_bytes(cx, d, 27, 1) == 0
        assert lib.bls_point_fft_scratch_bytes(cx, d, 20, 65) == 0
    assert lib.bls_point_fft_scratch_bytes(cx, 3, 2, 1) == 0
    assert lib.bls_kzg_open_all_prepare_scratch_bytes(cx, 24) > 0 and lib.bls_kzg_open_all_prepare_scratch_bytes(cx, 25) == 0
    assert lib.bls_kzg_open_all_scratch_bytes(cx, 24, 2) > 0 and lib.bls_kzg_open_all_scratch_bytes(cx, 24, 3) == 0
    assert lib.bls_kzg_open_all_scratch_bytes(cx, 25, 1) == 0
    table = np.full((8, W1), sentinel)
    assert lib.bls_kzg_open_all_prepare(cx, p_(x), 2, 2, p_(table)) == -1                  # srs_len < n - 1
    assert lib.bls_kzg_open_all_prepare(cx, None, 3, 2, p_(table)) == -1
    assert lib.bls_kzg_open_all_prepare(cx, p_(x), 3, 25, p_(table)) == -1
    assert (table == sentinel).all()
    assert lib.bls_kzg_open_all_prepare(cx, p_(x), 3, 2, p_(table)) == 0
    p = _fr(range(8)).reshape(2, 4, 4)
    y, pr = np.full((2, 4, 4), sentinel), np.full((2, 4, W1), sentinel)
    for i in (0, 1, 4, 5):
        a = [p_(table), p_(p), 2, 2, p_(y), p_(pr)]
        a[i] = None
        assert lib.bls_kzg_open_all_batch(cx, *a) == -1, i
    assert lib.bls_kzg_open_all_batch(cx, None, None, 24, 3, None, None) == -1
    assert (y == sentinel).all() and (pr == sentinel).all()
    assert lib.bls_kzg_open_all_batch(cx, None, None, 2, 0, None, None) == 0
    with pytest.raises(ValueError):
        ctx.kzg_open_all(table[:6], p)
    with pytest.raises(ValueError):
        ctx.g1_fft("fft", x[:3])
