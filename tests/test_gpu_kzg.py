"""KZG polynomial commitments (bls_kzg_commit_*, bls_kzg_open_*, bls_kzg_prepare_verifying_key, bls_kzg_verify_* and
bls_kzg_verify_rlc_*, their Context, DeviceEngine and C++ bindings).

Every point is [e] g for a known exponent e, so commitments and proofs are compared bit for bit with [closed-form exponent] g
(tests/kzg_model.py), and every verdict with the model's."""
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
import kzg_model as km
import oracle_lib as o
from test_gpu_msm import N_MAX, _base_exponents, _ints, eng, inputs  # noqa: F401 -- eng and inputs are fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER
W1 = 13
PVK_BYTES = 39704


def _limbs(values):
    return np.array([bm.limbs64(v % (1 << 256), 4) for v in values], dtype=np.uint64).reshape(-1, 4)


def _fr(values):
    """Montgomery bls_fr limbs; a value v >= r stands for the out-of-range input mont(v - r) + r (not reduced)"""
    return _limbs([bm.fr_to_mont(v) if v < R else bm.fr_to_mont(v - R) + R for v in values])


def _polys(rng, m, n):
    coeffs = [[rng.choice([0, 1, R - 1, rng.randrange(R)]) if i % 7 == 0 else rng.randrange(R) for i in range(n)] for _ in range(m)]
    return coeffs, _fr([c for row in coeffs for c in row]).reshape(m, n, 4)


def _g1(exps):
    """[e] g as affine rows, by the CPU oracle"""
    if not len(exps):
        return np.zeros((0, W1), dtype=np.uint64)
    gen = o.g1_from_affine(o.generators()[0])
    return o.g1_into_affine(o.g1_op("mul", np.repeat(gen, len(exps), 0), k=_limbs([e % R for e in exps]), threads=o.default_threads()))


def _g2(exps):
    gen = o.g2_from_affine(o.generators()[1])
    return o.g2_into_affine(o.g2_op("mul", np.repeat(gen, len(exps), 0), k=_limbs([e % R for e in exps]), threads=o.default_threads()))


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_model_quotient_and_verdicts():
    """p(X) = q(X)(X - z) + y at random points; honest openings verify; tampering c, y, z or w fails; y or z >= r fails"""
    rng = random.Random(1)
    tau = rng.randrange(R)
    for n in (0, 1, 2, 3, 17, 64):
        p = [rng.randrange(R) for _ in range(n)]
        for z in (0, 1, R - 1, rng.randrange(R)):
            y, q = km.quotient(p, z)
            assert y == km.evaluate(p, z) and len(q) == max(n - 1, 0)
            for x in (rng.randrange(R) for _ in range(3)):
                assert km.evaluate(p, x) == (km.evaluate(q, x) * (x - z) + y) % R
            c = km.commit(p, km.powers(tau, n))
            y, w = km.open_(p, z, km.powers(tau, max(n - 1, 0)))
            assert w == km.evaluate(q, tau) and km.verifies(tau, c, y, z, w)
            for bad in ((c + 1, y, z, w), (c, y + 1, z, w), (c, y, (z + 1) % R, w), (c, y, z, w + 1)):
                assert not km.verifies(tau, *bad) or (w == 0 and bad[2] != z)   # z does not matter when w = 0
            assert not km.verifies(tau, c, y + R, z, w) and not km.verifies(tau, c, y, z + R, w)


def test_model_randomized_check():
    """all valid: 1; one invalid: 0; rho_j = 0 excludes it; two errors that cancel under rho: 1; an out-of-range y: 0"""
    rng = random.Random(2)
    tau = rng.randrange(R)
    rows = []
    for _ in range(6):
        w, z, y = rng.randrange(R), rng.randrange(R), rng.randrange(R)
        rows.append(((tau * w - z * w + y) % R, y, z, w))
    rho = [rng.randrange(1, R) for _ in rows]
    assert km.rlc_verifies(tau, rows, rho)
    bad = list(rows)
    bad[2] = (bad[2][0] + 1, *bad[2][1:])
    assert not km.rlc_verifies(tau, bad, rho)
    assert km.rlc_verifies(tau, bad, rho[:2] + [0] + rho[3:])
    d = rng.randrange(1, R)
    bad[2] = (rows[2][0] + d, *rows[2][1:])
    bad[4] = ((rows[4][0] - d * rho[2] * pow(rho[4], -1, R)) % R, *rows[4][1:])
    assert km.rlc_verifies(tau, bad, rho) and not km.verifies(tau, *bad[2]) and not km.verifies(tau, *bad[4])
    oob = list(rows)
    oob[0] = (rows[0][0], rows[0][1] + R, *rows[0][2:])
    assert not km.rlc_verifies(tau, oob, rho) and km.rlc_verifies(tau, [], [])


def test_pvk_layout_matches_the_bindings():
    """sizeof / offsetof of bls_kzg_pvk equal the ctypes mirror, and both prepared arrays are 16-byte aligned"""
    import pairing_b200._native as nat
    fields = ("h_prepared", "neg_tau_h_prepared", "g", "h", "neg_tau_h")
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "pairing_b200.h"\nint main(){printf("%zu' + ' %zu' * len(fields) + '\\n",' \
          'sizeof(bls_kzg_pvk)' + ''.join(',offsetof(bls_kzg_pvk,%s)' % f for f in fields) + ');return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "s.c"), os.path.join(d, "s")
        open(c, "w").write(src)
        subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert got == [ctypes.sizeof(nat.KzgPvkC)] + [getattr(nat.KzgPvkC, f).offset for f in fields]
    assert got == [PVK_BYTES, 0, 19600, 39200, 39304, 39504]
    assert got[1] % 16 == 0 and got[2] % 16 == 0 and nat.W_KZG_PVK * 8 == PVK_BYTES


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
            usage[name] = line.strip()
    return exe, nat.LIB_PATH, usage


def test_kzg_kernels_resources_and_bulk_copy():
    """the new kernels' registers, stack and shared memory are within DESIGN.md's figures, with no local memory; the TMA bulk
    copies and their mbarrier are in k_kzg_verify's SASS"""
    exe, lib, usage = _resource_usage()
    #               kernel                 max REG  max STACK  min SHARED
    limits = {"k_kzg_verify": (255, 6112, 2 * 19584), "k_kzg_term": (184, 744, 0),
              "k_kzg_scan_up": (64, 0, 0), "k_kzg_scan_downILb0": (64, 0, 0), "k_kzg_scan_downILb1": (64, 0, 0),
              "k_kzg_emit": (32, 0, 0), "k_kzg_rlc_scalars": (64, 0, 0), "k_kzg_rlc_sum": (64, 0, 256 * 32)}
    for kernel, (reg, stack, shared) in limits.items():
        found = [v for k, v in usage.items() if kernel in k]
        assert len(found) == 1, (kernel, sorted(usage))
        u = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL|SHARED):(\d+)", found[0])}
        assert u["LOCAL"] == 0 and u["REG"] <= reg and u["STACK"] <= stack and u["SHARED"] >= shared, (kernel, u)
    assert len([k for k in usage if "k_kzg_" in k]) == len(limits)
    name = [k for k in usage if "k_kzg_verify" in k][0]
    sass = subprocess.check_output([exe, "-sass", "-fun", name, lib], text=True)
    assert len(re.findall(r"\bUBLKCP\b", sass)) == 2 and "SYNCS" in sass


def test_preexisting_kernels_resources_unchanged():
    """every kernel the library had before the KZG unit keeps its cuobjdump --dump-resource-usage line
    (tests/golden/resource_usage_pre_kzg.txt: the dump of the parent commit's build)"""
    _, _, usage = _resource_usage()
    before = dict(line.split(" ", 1) for line in open(os.path.join(ROOT, "tests", "golden", "resource_usage_pre_kzg.txt")).read().splitlines())
    assert len(before) > 80
    changed = {k: (v, usage.get(k)) for k, v in before.items() if usage.get(k) != v}
    assert not changed, changed


def test_null_context_is_an_invalid_argument():
    import pairing_b200._native as nat
    lib = nat.load()
    assert lib.bls_kzg_commit_batch(None, None, 1, None, 1, 1, None) == -1
    assert lib.bls_kzg_commit_dev(None, None, 1, None, 1, 1, None, None, None) == -1
    assert lib.bls_kzg_open_batch(None, None, 1, None, 1, None, 1, None, None) == -1
    assert lib.bls_kzg_open_dev(None, None, 1, None, 1, None, 1, None, None, None, None) == -1
    assert lib.bls_kzg_prepare_verifying_key(None, None, None, None, None) == -1
    assert lib.bls_kzg_verify_batch(None, None, None, None, None, None, 1, None) == -1
    assert lib.bls_kzg_verify_dev(None, None, None, None, None, None, 1, None, None, None) == -1
    assert lib.bls_kzg_verify_rlc_batch(None, None, None, None, None, None, None, 1, None) == -1
    assert lib.bls_kzg_verify_rlc_dev(None, None, None, None, None, None, None, 1, None, None, None) == -1
    for name, args in (("commit", (1, 1)), ("open", (1, 1)), ("verify", (1,)), ("verify_rlc", (1,))):
        assert getattr(lib, "bls_kzg_%s_scratch_bytes" % name)(None, *args) == 0


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def srs(inputs):
    """the 2^20 fixture bases [a_i] g (bench.make_inputs) and their exponents a_i"""
    return inputs["host"][False], [int(a) for a in _ints(_base_exponents(False, N_MAX))]


SIZES = [0, 1, 2, 3, 31, 32, 33, 1023, 1025, 4097]


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_commit_and_open_ragged(ctx, srs, n):
    """n on both sides of the scan's chunk (32) and level (1024) boundaries; m in {0, 1, 3, 64}; z in {0, 1, r - 1, random}:
    commitments and proofs equal [closed form] g bit for bit, y the model's Horner value"""
    bases, a = srs
    rng = random.Random(n)
    coeffs, p = _polys(rng, 64, n)
    zs = [[0, 1, R - 1][j] if j < 3 else rng.randrange(R) for j in range(64)]
    z = _fr(zs)
    want_c = [km.commit(row, a) for row in coeffs]
    want_open = [km.open_(row, zz, a) for row, zz in zip(coeffs, zs)]
    pts = _g1(want_c + [w for _, w in want_open])
    for m in (0, 1, 3, 64):
        c = ctx.kzg_commit(bases[:n], p[:m])
        assert np.array_equal(c, pts[:m]), m
        y, proof = ctx.kzg_open(bases[:max(n - 1, 0)], p[:m], z[:m])
        assert np.array_equal(y, _fr([yy for yy, _ in want_open[:m]])), m
        assert np.array_equal(proof, pts[64:64 + m]), m


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(1, 1 << 20), (64, 1 << 14)])
def test_commit_and_open_full_size(ctx, srs, m, n):
    bases, a = srs
    rng = random.Random(m * 7 + n)
    coeffs = [[rng.randrange(R) for _ in range(n)] for _ in range(m)]
    p = _fr([c for row in coeffs for c in row]).reshape(m, n, 4)
    zs = [rng.randrange(R) for _ in range(m)]
    want_open = [km.open_(row, zz, a) for row, zz in zip(coeffs, zs)]
    pts = _g1([km.commit(row, a) for row in coeffs] + [w for _, w in want_open])
    assert np.array_equal(ctx.kzg_commit(bases[:n], p), pts[:m])
    y, proof = ctx.kzg_open(bases[:n - 1], p, _fr(zs))
    assert np.array_equal(y, _fr([yy for yy, _ in want_open]))
    assert np.array_equal(proof, pts[m:])


class Key:
    """tau, the verifying key over the generators g, h and [tau] h, and proof rows from chosen exponents"""

    def __init__(self, ctx, seed, tau=None):
        self.tau = random.Random(seed).randrange(R) if tau is None else tau
        self.g = o.generators()[0].reshape(-1)
        h = _g2([1, self.tau])
        self.h, self.tau_h = h[0], h[1]
        self.pvk = ctx.kzg_prepare_verifying_key(self.g, self.h, self.tau_h)

    @staticmethod
    def rows(ctx, rows):
        """(c, y, z, w) exponent rows -> C (m, 13), y (m, 4), z (m, 4), W (m, 13); [e] g on the GPU for large batches"""
        m = len(rows)
        gen = o.g1_from_affine(o.generators()[0])
        pts = ctx.g1_into_affine(ctx.g1_mul(np.repeat(gen, 2 * m, 0), _limbs([r[0] % R for r in rows] + [r[3] % R for r in rows])))
        return pts[:m], _fr([r[1] for r in rows]), _fr([r[2] for r in rows]), pts[m:]

    def valid(self, rng, w=None, z=None, y=None):
        w = rng.randrange(R) if w is None else w
        z = rng.randrange(R) if z is None else z
        y = rng.randrange(R) if y is None else y
        return ((self.tau * w - z * w + y) % R, y, z, w)


def _cases(key, rng, m):
    """m rows, about half invalid: tampered C, y, z or W; C or W at infinity (valid and not); y or z >= r"""
    rows = []
    for j in range(m):
        kind = j % 12
        c, y, z, w = key.valid(rng)
        if kind == 1:
            c = (c + rng.randrange(1, R)) % R
        elif kind == 2:
            y = (y + 1) % R
        elif kind == 3:
            z = (z + 1) % R
        elif kind == 4:
            w = (w + 1) % R
        elif kind == 5:                                                  # C at infinity, valid
            y = (z * w - key.tau * w) % R
            c = 0
        elif kind == 6:                                                  # W at infinity: valid iff c = y
            c, y, z, w = key.valid(rng, w=0)
        elif kind == 7:
            c, y, z, w = (c, y, z, 0)
        elif kind == 8:
            y += R
        elif kind == 9:
            z += R
        elif kind == 10:                                                 # C at infinity, invalid
            c = 0
        rows.append((c, y, z, w))
    return rows


@pytest.mark.gpu
def test_verify_2_16_proofs(ctx):
    key = Key(ctx, 0xA11)
    rng = random.Random(0xA12)
    rows = _cases(key, rng, 1 << 16)
    want = np.array([km.verifies(key.tau, *r) for r in rows])
    assert 0.3 < want.mean() < 0.7
    args = Key.rows(ctx, rows)
    assert np.array_equal(ctx.kzg_verify(key.pvk, *args), want)
    for m in (0, 1, 2, 63, 65, 257):
        assert np.array_equal(ctx.kzg_verify(key.pvk, *[x[:m] for x in args]), want[:m]), m


@pytest.mark.gpu
def test_verify_rlc(ctx):
    """valid batch of 2^16: 1; one invalid: 0; rho_j = 0 on it: 1; a cancelling pair: 1; an out-of-range z: 0; m = 0: 1"""
    key = Key(ctx, 0xB11)
    rng = random.Random(0xB12)
    m = 1 << 16
    rows = [key.valid(rng) for _ in range(m)]
    rho = [rng.randrange(1, R) for _ in range(m)]
    c, y, z, w = Key.rows(ctx, rows)
    assert ctx.kzg_verify_rlc(key.pvk, c, y, z, w, _limbs(rho))
    j = 12345
    bad = rows[j][0] + 1
    c_bad = c.copy()
    c_bad[j] = _g1([bad])[0]
    assert not ctx.kzg_verify_rlc(key.pvk, c_bad, y, z, w, _limbs(rho))
    rho0 = list(rho)
    rho0[j] = 0
    assert ctx.kzg_verify_rlc(key.pvk, c_bad, y, z, w, _limbs(rho0))
    k = 77
    d = rng.randrange(1, R)
    c_pair = c.copy()
    c_pair[[j, k]] = _g1([rows[j][0] + d, rows[k][0] - d * rho[j] * pow(rho[k], -1, R)])
    assert not km.verifies(key.tau, (rows[j][0] + d) % R, *rows[j][1:])
    assert ctx.kzg_verify_rlc(key.pvk, c_pair, y, z, w, _limbs(rho))
    z_oob = z.copy()
    z_oob[5] = _fr([rows[5][2] + R])[0]
    assert not ctx.kzg_verify_rlc(key.pvk, c, y, z_oob, w, _limbs(rho))
    empty = np.zeros((0, 4), np.uint64)
    assert ctx.kzg_verify_rlc(key.pvk, np.zeros((0, W1), np.uint64), empty, empty, np.zeros((0, W1), np.uint64), empty) is True
    small = _cases(key, rng, 24)
    rh = [rng.randrange(1, R) for _ in small]
    for sel in ([0], [5], [6], list(range(24))):
        sub = [small[i] for i in sel]
        assert ctx.kzg_verify_rlc(key.pvk, *Key.rows(ctx, sub), _limbs([rh[i] for i in sel])) == km.rlc_verifies(key.tau, sub, [rh[i] for i in sel])


@pytest.mark.gpu
def test_end_to_end_with_a_real_srs(ctx):
    """random tau, 2^12 powers [tau^i] g from the oracle: commit, open and verify accept; a wrong y, or a proof for another
    z, is rejected; the randomized check agrees"""
    rng = random.Random(0xE2E)
    n = 1 << 12
    key = Key(ctx, 0, tau=rng.randrange(R))
    srs_rows = _g1(km.powers(key.tau, n))
    coeffs, p = _polys(rng, 5, n)
    zs = [rng.randrange(R) for _ in range(5)]
    c = ctx.kzg_commit(srs_rows, p)
    assert np.array_equal(c, _g1([km.evaluate(row, key.tau) for row in coeffs]))
    y, proof = ctx.kzg_open(srs_rows, p, _fr(zs))
    assert ctx.kzg_verify(key.pvk, c, y, _fr(zs), proof).all()
    y_bad = y.copy()
    y_bad[1] = _fr([(km.evaluate(coeffs[1], zs[1]) + 1) % R])[0]
    _, proof_other = ctx.kzg_open(srs_rows, p, _fr([(zz + 1) % R for zz in zs]))
    assert list(ctx.kzg_verify(key.pvk, c, y_bad, _fr(zs), proof)) == [True, False, True, True, True]
    assert not ctx.kzg_verify(key.pvk, c, y, _fr(zs), proof_other).any()
    rho = _limbs([rng.randrange(1, R) for _ in zs])
    assert ctx.kzg_verify_rlc(key.pvk, c, y, _fr(zs), proof, rho)
    assert not ctx.kzg_verify_rlc(key.pvk, c, y_bad, _fr(zs), proof, rho)


CPP_KZG = r"""
#include <fstream>
#include "pairing_b200.hpp"
using namespace pairing_b200;
template <class T> std::vector<T> rd(std::ifstream& f) {
  uint64_t n; f.read(reinterpret_cast<char*>(&n), 8);
  std::vector<T> v(n / sizeof(T)); f.read(reinterpret_cast<char*>(v.data()), n);
  return v;
}
template <class T> void wr(std::ofstream& o, const std::vector<T>& v) { o.write(reinterpret_cast<const char*>(v.data()), v.size() * sizeof(T)); }
int main(int, char** argv) {
  Gpu gpu(0);
  std::ifstream f(argv[1], std::ios::binary);
  auto srs = rd<G1AffinePoint>(f); auto p = rd<bls_fr>(f); auto z = rd<bls_fr>(f); auto g1 = rd<G1AffinePoint>(f); auto g2 = rd<G2AffinePoint>(f);
  auto rho = rd<bls_fr_repr>(f);
  const size_t n = p.size() / z.size();
  auto c = Kzg::commit(gpu, srs, p, n);
  auto op = Kzg::open(gpu, srs, p, n, z);
  auto pvk = Kzg::prepare_verifying_key(gpu, g1[0], g2[0], g2[1]);
  auto ok = Kzg::verify(gpu, *pvk, c, op.y, z, op.proof);
  const bool rlc = Kzg::verify_batch(gpu, *pvk, c, op.y, z, op.proof, rho);
  std::ofstream o(argv[2], std::ios::binary);
  wr(o, c); wr(o, op.y); wr(o, op.proof);
  o.write(reinterpret_cast<const char*>(pvk.get()), sizeof(Kzg::PreparedVerifyingKey));
  for (bool b : ok) o.put(b ? 1 : 0);
  o.put(rlc ? 1 : 0);
  return 0;
}
"""


@pytest.mark.gpu
def test_host_dev_engine_cpp_and_the_chain_agree(ctx, eng):
    """Context (host _batch), the _dev calls on a stream of their own, DeviceEngine, the C++ Kzg section and the chain of
    existing calls give identical outputs: commit (into_repr -> msm_batch -> into_affine), open (host division -> msm_batch ->
    into_affine) and verify (msm_batch over [C, g, W] with [1, r - y, z] -> two shared-Q Miller loops -> Fq12 product -> final
    exponentiation -> compare with one)"""
    import torch
    import pairing_b200._native as nat
    rng = random.Random(0xF0)
    m, n = 6, 301
    key = Key(ctx, 0xF1)
    coeffs, p = _polys(rng, m, n)
    zs = [0, 1] + [rng.randrange(R) for _ in range(m - 2)]
    z = _fr(zs)
    srs_rows = _g1(km.powers(key.tau, n))                                # the SRS of key's tau: every opening below verifies
    c = ctx.kzg_commit(srs_rows, p)
    y, proof = ctx.kzg_open(srs_rows, p, z)
    assert ctx.kzg_verify(key.pvk, c, y, z, proof).all()
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to(eng.device)  # noqa: E731
    host = lambda t: t.cpu().numpy().view(np.uint64)  # noqa: E731
    assert np.array_equal(host(eng.kzg_commit(dev(srs_rows), dev(p))), c)
    dy, dproof = eng.kzg_open(dev(srs_rows), dev(p), dev(z))
    assert np.array_equal(host(dy), y) and np.array_equal(host(dproof), proof)
    # the chain of existing calls
    k = ctx.fr_op("into_repr", p.reshape(-1, 4))[0].reshape(m, n, 4)
    assert np.array_equal(ctx.g1_into_affine(ctx.g1_msm_batch(srs_rows, k)), c)
    qs = [km.quotient(row, zz) for row, zz in zip(coeffs, zs)]
    assert np.array_equal(y, _fr([yy for yy, _ in qs]))
    q = _limbs([v for _, qq in qs for v in qq]).reshape(m, n - 1, 4)
    assert np.array_equal(ctx.g1_into_affine(ctx.g1_msm_batch(srs_rows[:n - 1], q)), proof)
    # verify: valid openings, tampered ones and edge cases
    rows = [key.valid(rng) for _ in range(8)] + _cases(key, rng, 24)
    vc, vy, vz, vw = Key.rows(ctx, rows)
    want = np.array([km.verifies(key.tau, *r) for r in rows])
    assert np.array_equal(ctx.kzg_verify(key.pvk, vc, vy, vz, vw), want)
    dpvk = dev(key.pvk)
    assert np.array_equal(eng.kzg_verify(dpvk, dev(vc), dev(vy), dev(vz), dev(vw)).cpu().numpy().astype(bool), want)
    st = torch.cuda.Stream(eng.device)
    st.wait_stream(torch.cuda.current_stream(eng.device))
    mv = len(rows)
    out = torch.zeros(mv, dtype=torch.uint8, device=eng.device)
    scr = torch.empty(ctx.kzg_scratch_bytes("verify", mv), dtype=torch.uint8, device=eng.device)
    tv = [dev(x) for x in (vc, vy, vz, vw)]
    with torch.cuda.stream(st):
        ctx.call_dev("bls_kzg_verify_dev", dpvk.data_ptr(), *[t.data_ptr() for t in tv], mv, out.data_ptr(), scr.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert np.array_equal(out.cpu().numpy().astype(bool), want)
    in_range = np.array([r[1] < R and r[2] < R for r in rows])
    cgw = np.stack([vc, np.repeat(key.g[None], mv, 0), vw], axis=1)
    sc = np.stack([_limbs([1] * mv), _limbs([(-r[1]) % R for r in rows]), _limbs([r[2] % R for r in rows])], axis=1)
    pt = ctx.g1_into_affine(ctx.g1_msm_batch(cgw, sc))
    prep = ctx.g2_prepare(np.stack([key.h, nat_neg(ctx, key.tau_h)]))
    f = ctx.field_op(12, "mul", ctx.miller_loop_shared_q(pt, prep[:1]), ctx.miller_loop_shared_q(vw, prep[1:]))[0]
    fe, some = ctx.final_exponentiation(f)
    one = ctx.pairing(np.repeat(_g1([0]), 1, 0), key.h[None])[0]
    chain = in_range & (some != 0) & (fe == one[None]).all(axis=1)
    assert np.array_equal(chain, want)
    # randomized check: host, engine, _dev
    rho = _limbs([rng.randrange(1, R) for _ in rows])
    good = np.flatnonzero(want)
    assert ctx.kzg_verify_rlc(key.pvk, vc[good], vy[good], vz[good], vw[good], rho[good])
    assert eng.kzg_verify_rlc(dpvk, *[dev(x[good]) for x in (vc, vy, vz, vw)], dev(rho[good])).item() == 1
    out1 = torch.full((1,), 7, dtype=torch.uint8, device=eng.device)
    rscr = torch.empty(ctx.kzg_scratch_bytes("verify_rlc", mv), dtype=torch.uint8, device=eng.device)
    drho = dev(rho)
    with torch.cuda.stream(st):
        ctx.call_dev("bls_kzg_verify_rlc_dev", dpvk.data_ptr(), *[t.data_ptr() for t in tv], drho.data_ptr(), mv, out1.data_ptr(), rscr.data_ptr(),
                     st.cuda_stream)
    st.synchronize()
    assert out1.item() == 0
    # the C++ mirror
    libdir = os.path.dirname(nat.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        src, exe, fin, fout = (os.path.join(d, x) for x in ("k.cpp", "k", "in", "out"))
        open(src, "w").write(CPP_KZG)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                               "-L", libdir, "-lpairing_b200", "-Wl,-rpath," + libdir])
        with open(fin, "wb") as fh:
            for x in (srs_rows, p, z, key.g[None], np.stack([key.h, key.tau_h]), _limbs([rng.randrange(1, R) for _ in range(m)])):
                raw = np.ascontiguousarray(x).tobytes()
                fh.write(np.uint64(len(raw)).tobytes() + raw)
        subprocess.check_call([exe, fin, fout], timeout=300)
        res = np.fromfile(fout, dtype=np.uint8)
    nb = [m * W1 * 8, m * 32, m * W1 * 8, PVK_BYTES]
    parts = np.split(res, np.cumsum(nb))
    assert parts[0].tobytes() == c.tobytes() and parts[1].tobytes() == y.tobytes() and parts[2].tobytes() == proof.tobytes()
    assert parts[3].tobytes() == key.pvk.tobytes()
    assert parts[4][:m].all() and parts[4][m] == 1                      # the openings of key's SRS verify, one by one and together


def nat_neg(ctx, q):
    """-q for a G2 affine row (CurveAffine::negate)"""
    out = q.copy()
    if q[24] == 0:
        out[12:24] = ctx.field_op(2, "neg", q[None, 12:24])[0][0]
    return out


@pytest.mark.gpu
def test_pvk_is_bit_exact(ctx):
    """prepared parts = bls_g2_prepare_batch of h and -tau h; the affine parts are g, h, -tau h; the pads are zero"""
    import pairing_b200._native as nat
    key = Key(ctx, 0xC0)
    f = lambda name: key.pvk[getattr(nat.KzgPvkC, name).offset // 8:(getattr(nat.KzgPvkC, name).offset + getattr(nat.KzgPvkC, name).size) // 8]  # noqa: E731
    neg = _g2([-key.tau % R])[0]
    prep = ctx.g2_prepare(np.stack([key.h, neg]))
    assert np.array_equal(f("h_prepared"), prep[0]) and np.array_equal(f("neg_tau_h_prepared"), prep[1])
    assert np.array_equal(f("g"), key.g) and np.array_equal(f("h"), key.h) and np.array_equal(f("neg_tau_h"), neg)
    assert f("pad0")[0] == 0 and f("pad1")[0] == 0


@pytest.mark.gpu
def test_invalid_arguments(ctx, srs):
    """NULL pointers where there is work, a short SRS, the limits and a misaligned _dev pvk give BLS_ERR_INVALID_ARGUMENT and
    leave the outputs untouched; m = 0 does nothing"""
    import torch
    lib, cx = ctx._lib, ctx._ctx
    p_ = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    bases, _ = srs
    n, m = 5, 2
    s = np.ascontiguousarray(bases[:n])
    p = _fr(list(range(1, m * n + 1))).reshape(m, n, 4)
    z = _fr([3, 4])
    sentinel = np.uint64(0x5A5A5A5A5A5A5A5A)
    c = np.full((m, W1), sentinel)
    y, w = np.full((m, 4), sentinel), np.full((m, W1), sentinel)
    assert lib.bls_kzg_commit_batch(cx, p_(s), n - 1, p_(p), n, m, p_(c)) == -1           # srs_len < n
    assert lib.bls_kzg_commit_batch(cx, None, n, p_(p), n, m, p_(c)) == -1
    assert lib.bls_kzg_commit_batch(cx, p_(s), n, None, n, m, p_(c)) == -1
    assert lib.bls_kzg_commit_batch(cx, p_(s), n, p_(p), n, m, None) == -1
    assert lib.bls_kzg_commit_batch(cx, None, 1, None, 1, (1 << 16) + 1, None) == -1
    assert lib.bls_kzg_commit_batch(cx, None, 1 << 20, None, 1 << 20, 65, None) == -1  # m n > 2^26
    assert (c == sentinel).all()
    assert lib.bls_kzg_open_batch(cx, p_(s), n - 2, p_(p), n, p_(z), m, p_(y), p_(w)) == -1   # srs_len < n - 1
    for i in (0, 2, 4, 6, 7):
        a = [p_(s), n, p_(p), n, p_(z), m, p_(y), p_(w)]
        a[i] = None
        assert lib.bls_kzg_open_batch(cx, *a) == -1, i
    assert (y == sentinel).all() and (w == sentinel).all()
    assert lib.bls_kzg_open_batch(cx, p_(s), n - 1, p_(p), n, p_(z), m, p_(y), p_(w)) == 0       # srs_len = n - 1 is enough
    assert lib.bls_kzg_commit_batch(cx, p_(s), n, p_(p), n, m, p_(c)) == 0
    # m = 0: nothing to do, every pointer may be NULL
    assert lib.bls_kzg_commit_batch(cx, None, 0, None, 9, 0, None) == 0
    assert lib.bls_kzg_open_batch(cx, None, 0, None, 9, None, 0, None, None) == 0
    assert lib.bls_kzg_verify_batch(cx, None, None, None, None, None, 0, None) == 0
    ok0 = np.zeros(1, np.uint8)
    assert lib.bls_kzg_verify_rlc_batch(cx, None, None, None, None, None, None, 0, p_(ok0)) == 0 and ok0[0] == 1
    assert lib.bls_kzg_commit_scratch_bytes(cx, 9, 0) == 1 and lib.bls_kzg_verify_scratch_bytes(cx, 0) == 1
    # n = 0 and n = 1 need no SRS: y = 0 / p_0 and the identity
    ident = _g1([0])
    y1, w1 = ctx.kzg_open(np.zeros((0, W1), np.uint64), p[:, :1], z)
    assert np.array_equal(y1, p[:, 0]) and (w1 == ident).all()
    y0, w0 = ctx.kzg_open(np.zeros((0, W1), np.uint64), p[:, :0], z)
    assert not y0.any() and (w0 == ident).all()
    assert (ctx.kzg_commit(np.zeros((0, W1), np.uint64), p[:, :0]) == ident).all()
    # verify
    key = Key(ctx, 0xD0)
    vc, vy, vz, vw = Key.rows(ctx, [key.valid(random.Random(1))])
    ok = np.full(1, 7, np.uint8)
    args = [p_(key.pvk), p_(vc), p_(vy), p_(vz), p_(vw), 1, p_(ok)]
    for i in (0, 1, 2, 3, 4, 6):
        a = list(args)
        a[i] = None
        assert lib.bls_kzg_verify_batch(cx, *a) == -1, i
        assert lib.bls_kzg_verify_rlc_batch(cx, *a[:5], p_(_limbs([1])), *a[5:]) == -1, i
    assert lib.bls_kzg_verify_rlc_batch(cx, *args[:5], None, *args[5:]) == -1
    assert ok[0] == 7
    assert lib.bls_kzg_verify_batch(cx, None, None, None, None, None, (1 << 26) + 1, None) == -1
    assert lib.bls_kzg_verify_rlc_batch(cx, None, None, None, None, None, None, 1 << 25, None) == -1
    assert lib.bls_kzg_verify_rlc_scratch_bytes(cx, (1 << 25) - 1) > 0 and lib.bls_kzg_verify_rlc_scratch_bytes(cx, 1 << 25) == 0
    assert lib.bls_kzg_verify_batch(cx, *args) == 0 and ok[0] == 1
    # a pvk that is not 16-byte aligned is rejected before any work
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to("cuda")  # noqa: E731
    raw = torch.zeros(PVK_BYTES + 16, dtype=torch.uint8, device="cuda")
    t = [dev(x) for x in (vc, vy, vz, vw)]
    dok = torch.full((1,), 7, dtype=torch.uint8, device="cuda")
    scr = torch.empty(ctx.kzg_scratch_bytes("verify_rlc", 1) + ctx.kzg_scratch_bytes("verify", 1), dtype=torch.uint8, device="cuda")
    drho = dev(_limbs([1]))
    for off, rc in ((8, -1), (0, 0)):
        raw[off:off + PVK_BYTES].copy_(torch.from_numpy(key.pvk.view(np.uint8)).to("cuda"))
        torch.cuda.synchronize()
        assert lib.bls_kzg_verify_dev(cx, raw.data_ptr() + off, *[x.data_ptr() for x in t], 1, dok.data_ptr(), scr.data_ptr(), None) == rc, off
        assert lib.bls_kzg_verify_rlc_dev(cx, raw.data_ptr() + off, *[x.data_ptr() for x in t], drho.data_ptr(), 1, dok.data_ptr(),
                                          scr.data_ptr(), None) == rc, off
        torch.cuda.synchronize()
        assert dok.item() == (7 if rc else 1)
    assert lib.bls_kzg_open_dev(cx, None, 0, None, 3, None, 1, None, None, None, None) == -1
    assert lib.bls_kzg_commit_dev(cx, None, 3, None, 3, 1, None, None, None) == -1
    assert lib.bls_kzg_prepare_verifying_key(cx, p_(key.g), p_(key.h), None, p_(np.zeros(PVK_BYTES // 8, np.uint64))) == -1
    with pytest.raises(ValueError):
        ctx.kzg_commit(s[:n - 1], p)
    with pytest.raises(ValueError):
        ctx.kzg_verify(key.pvk, vc, vy, vz[:0], vw)
