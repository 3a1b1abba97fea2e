"""The memory and stream contract of the device-pointer entry points (include/pairing_b200.h, "device-pointer variants").

Every case goes through run_dev, which checks what the value tests elsewhere in the suite cannot see:
- scratch of exactly the size *_scratch_bytes states, between two 64 KiB canaries of seeded random bytes: a write even one
  byte past either end is caught;
- the scratch poisoned twice, with 0xFF and with seeded random bytes: both outputs must be byte-identical and equal the
  reference, so no region may be read before the call writes it;
- every buffer carved from a larger one with guard bytes on both sides, outputs filled with the 0x5A sentinel: the guards
  stay, every word the call writes loses the sentinel, every row it leaves alone keeps it;
- every const input compared byte for byte after the call; the documented in == out forms run in place as well;
- the work enqueued on a stream of the test's own behind a sleep, the real inputs copied in on that stream after it, and the
  host not synchronised before the call: a stage on another stream, or one that reads its input early, sees the other (valid)
  input set the buffers held before and gives a wrong answer.

The reference is the model the rest of the suite uses at that shape where there is one, else the host _batch call, which the
suite pins to the models and the oracle.  test_every_scratch_entry_point_has_a_case keeps the table complete."""
import ctypes
import os
import random
import re
from dataclasses import dataclass, field

import numpy as np
import pytest

import bls_model as bm
import datagen as dg
import fr_fft_model as fm
import groth16_setup_model as gs
import kzg_model as km
import oracle_lib as o
import point_fft_model as pm
from test_gpu_groth16_h import _model as h_model, _proofs as h_proofs
from test_gpu_groth16_prove import Toy
from test_gpu_groth16_setup import _expect, _mont1, _scalars, _toy
from test_gpu_groth16_verify import Vk, _batch as verify_batch
from test_gpu_kzg import Key, _cases as kzg_cases, _fr, _limbs, _polys
from test_gpu_msm import _splitmix_scalars
from test_gpu_point_fft import _pts, _rows as pfft_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = bm.R_ORDER
W1, W2, W1J, W2J, W12, WFR = 13, 25, 18, 36, 72, 4
KINDS = ("fft", "ifft", "coset_fft", "icoset_fft")
GUARD = 4096                 # guard bytes before and after every input and output buffer
CANARY = 64 << 10            # canary bytes before and after the scratch
SENTINEL = 0x5A
SLEEP_CYCLES = 50_000_000    # about 25 ms at the B200's clocks
POOL = 1 << 14               # subgroup points of known exponents for bases, SRS and pairs


def _u8(a):
    return np.ascontiguousarray(a).view(np.uint8).reshape(-1)


@dataclass
class Case:
    """one call: fn and its arguments (args(P) with P(name) the pointer of a buffer, "scratch" or "stream"), the real input
    set and a decoy of the same shapes, the outputs as name -> (bytes, unit, bytes written from the start), the reference
    (want() -> name -> array of the written bytes), the scratch size, the inputs the call rewrites in place (inout) and the
    documented in == out form (inplace = (output, input))"""
    fn: str
    args: object
    real: dict
    decoy: dict
    outs: dict
    want: object
    scratch: int = None
    inout: tuple = ()
    inplace: tuple = None


def _run_once(ctx, case, poison, alias=None):
    import torch
    alias = alias or {}
    rng = np.random.default_rng(0xC0DE if poison == "ff" else 0xBEEF)
    dev = torch.device("cuda", ctx.device)

    def guarded(payload_bytes):
        return torch.full((2 * GUARD + payload_bytes,), SENTINEL, dtype=torch.uint8, device=dev)

    ins = {}
    for name, arr in case.real.items():
        real, decoy = _u8(arr), _u8(case.decoy[name])
        assert real.size == decoy.size, name
        t = guarded(real.size)
        t[GUARD:GUARD + real.size].copy_(torch.from_numpy(decoy.copy()))
        ins[name] = (t, torch.from_numpy(real.copy()).to(dev), real)
    outs = {name: guarded(nb) for name, (nb, _, _) in case.outs.items()}
    scr = fill = None
    if case.scratch is not None:
        S = case.scratch
        scr = torch.empty(2 * CANARY + S, dtype=torch.uint8, device=dev)
        canary = rng.integers(0, 256, 2 * CANARY, dtype=np.uint8)
        scr[:CANARY].copy_(torch.from_numpy(canary[:CANARY]))
        scr[CANARY + S:].copy_(torch.from_numpy(canary[CANARY:]))
        if poison != "ff":
            fill = torch.from_numpy(rng.integers(0, 256, S, dtype=np.uint8)).to(dev)
        assert (scr.data_ptr() + CANARY) % 256 == 0
    st = torch.cuda.Stream(dev)

    def P(name):
        if name == "stream":
            return st.cuda_stream
        if name == "scratch":
            return scr.data_ptr() + CANARY
        name = alias.get(name, name)
        return (ins[name][0] if name in ins else outs[name]).data_ptr() + GUARD

    torch.cuda.synchronize(dev)
    with torch.cuda.stream(st):
        torch.cuda._sleep(SLEEP_CYCLES)
        for t, staged, _ in ins.values():
            t[GUARD:GUARD + staged.numel()].copy_(staged)
        if scr is not None:
            mid = scr[CANARY:CANARY + case.scratch]
            mid.fill_(0xFF) if fill is None else mid.copy_(fill)
        ctx.call_dev(case.fn, *case.args(P))
    st.synchronize()

    got = {}
    if scr is not None:
        h = scr.cpu().numpy()
        assert np.array_equal(h[:CANARY], canary[:CANARY]), "%s wrote before its scratch" % case.fn
        assert np.array_equal(h[CANARY + case.scratch:], canary[CANARY:]), "%s wrote past its scratch of %d bytes" % (case.fn, case.scratch)
    rewritten = set(case.inout) | set(alias.values())
    for name, (t, _, real) in ins.items():
        h = t.cpu().numpy()
        assert (h[:GUARD] == SENTINEL).all() and (h[GUARD + real.size:] == SENTINEL).all(), "%s wrote outside input %s" % (case.fn, name)
        payload = h[GUARD:GUARD + real.size]
        if name in rewritten:
            got[name] = payload
        else:
            assert np.array_equal(payload, real), "%s changed its const input %s" % (case.fn, name)
    for name, t in outs.items():
        nb, unit, written = case.outs[name]
        h = t.cpu().numpy()
        assert (h[:GUARD] == SENTINEL).all() and (h[GUARD + nb:] == SENTINEL).all(), "%s wrote outside output %s" % (case.fn, name)
        if name in alias:
            assert (h[GUARD:GUARD + nb] == SENTINEL).all(), name
            got[name] = got[alias[name]]
            continue
        assert (h[GUARD + written:GUARD + nb] == SENTINEL).all(), "%s wrote rows of %s it leaves alone" % (case.fn, name)
        w = h[GUARD:GUARD + written]
        units = w.view({1: np.uint8, 4: np.uint32, 8: np.uint64}[unit])
        assert not (units == int.from_bytes(bytes([SENTINEL]) * unit, "little")).any(), "%s left words of %s unwritten" % (case.fn, name)
        got[name] = w
    return got


def run_dev(ctx, case):
    """the contract checks above, both poisons, the reference, and the in-place form"""
    first = _run_once(ctx, case, "ff")
    second = _run_once(ctx, case, "random")
    for name in first:
        assert first[name].tobytes() == second[name].tobytes(), "%s: %s depends on what the scratch held" % (case.fn, name)
    want = case.want()
    assert set(want) == set(first), (sorted(want), sorted(first))
    for name, w in want.items():
        assert first[name].tobytes() == _u8(w).tobytes(), "%s: %s differs from the reference" % (case.fn, name)
    if case.inplace:
        out, inp = case.inplace
        again = _run_once(ctx, case, "random", alias={out: inp})
        assert again[out].tobytes() == first[out].tobytes(), "%s in place differs from out of place" % case.fn


# ------------------------------------------------------------------------------------------------------------ the table

@dataclass
class Spec:
    fn: str                       # entry point
    sb: str                       # its *_scratch_bytes function (None for entry points without scratch)
    id: str
    build: object = field(repr=False)   # (ctx, pool) -> Case


class Pool:
    """POOL subgroup points [e_i] g in G1 and G2 (affine rows) of known exponents e_i"""

    def __init__(self, ctx):
        rng = random.Random(0xD0C)
        self.e = [rng.randrange(1, R) for _ in range(POOL)]
        self.g1, self.g2 = _pts(ctx, self.e), _pts(ctx, self.e, True)

    def take(self, g2, n, shift=0):
        return np.ascontiguousarray(np.roll(self.g2 if g2 else self.g1, -shift, axis=0)[:n])


def _sb(ctx, name, *args):
    b = int(getattr(ctx._lib, name)(ctx._ctx, *args))
    assert b > 0, (name, args)
    return b


def _out(nbytes, unit=8, written=None):
    return (nbytes, unit, nbytes if written is None else written)


# ---- Fr FFT and Groth16's H

def _fr_fft_case(kind, log_n, m):
    def build(ctx, pool):
        n = 1 << log_n
        rng = random.Random(log_n * 16 + m * 4 + KINDS.index(kind))
        vals = [[rng.choice([0, 1, R - 1, rng.randrange(R)]) for _ in range(n)] for _ in range(2 * m)]
        real, decoy = (_fr([v for row in vals[s] for v in row]).reshape(m, n, WFR) for s in (slice(0, m), slice(m, 2 * m)))

        def want():
            if log_n <= 11:
                return {"out": np.stack([_limbs(fm.fr_fft(kind, [bm.fr_to_mont(v) for v in row], log_n)) for row in vals[:m]])}
            return {"out": ctx.fr_fft(kind, real)}
        return Case("bls_fr_fft_dev", lambda P: [fm.FR_FFT_KINDS[kind], P("in"), P("out"), log_n, m, P("scratch"), P("stream")],
                    {"in": real}, {"in": decoy}, {"out": _out(real.nbytes)}, want, _sb(ctx, "bls_fr_fft_scratch_bytes", log_n, m),
                    inplace=("out", "in"))
    return Spec("bls_fr_fft_dev", "bls_fr_fft_scratch_bytes", "fr_fft-%s-log%d-m%d" % (kind, log_n, m), build)


def _groth16_h_case(length, m):
    def build(ctx, pool):
        real, decoy = h_proofs(m, length, length * 8 + m, False), h_proofs(m, length, length * 8 + m + 99, False)
        n1 = (1 << max(length - 1, 0).bit_length()) - 1

        def want():
            return {"h": h_model(*real) if length <= 1025 else ctx.fr_groth16_h(*real)}
        return Case("bls_fr_groth16_h_dev", lambda P: [P("a"), P("b"), P("c"), length, m, P("h"), P("scratch"), P("stream")],
                    dict(zip("abc", real)), dict(zip("abc", decoy)), {"h": _out(m * n1 * 32)}, want,
                    _sb(ctx, "bls_fr_groth16_h_scratch_bytes", length, m))
    return Spec("bls_fr_groth16_h_dev", "bls_fr_groth16_h_scratch_bytes", "groth16_h-len%d-m%d" % (length, m), build)


# ---- multiexps

def _msm_case(g2, mode, n, m, window):
    """mode: "single" (bls_g*_msm_dev), "shared" or "own" bases (bls_g*_msm_batch_dev)"""
    curve = "g2" if g2 else "g1"
    fn = "bls_%s_msm_dev" % curve if mode == "single" else "bls_%s_msm_batch_dev" % curve
    sbn = "bls_msm_scratch_bytes" if mode == "single" else "bls_msm_batch_scratch_bytes"

    def build(ctx, pool):
        deg, wj = (2, W2J) if g2 else (1, W1J)

        def inputs(shift, seed):
            if mode == "own":
                b = np.stack([pool.take(g2, n, shift + 977 * j) for j in range(m)]) if n else np.zeros((m, 0, W2 if g2 else W1), np.uint64)
            else:
                b = pool.take(g2, n, shift)
            k = _splitmix_scalars(seed, m * n).reshape(m, n, 4)
            if m * n:
                k.reshape(-1, 4)[::29] = 0                                 # zero scalars contribute nothing
            return b, k
        (b, k), (db, dk) = inputs(0, n * 31 + m + window), inputs(5, n * 31 + m + window + 1)

        def want():
            if mode == "single":
                return {"out": (ctx.g2_msm if g2 else ctx.g1_msm)(b, k[0])}
            if n == 0:                                                     # m zeros
                return {"out": np.repeat((ctx.g2_msm if g2 else ctx.g1_msm)(b, k[0]), m, 0)}
            return {"out": (ctx.g2_msm_batch if g2 else ctx.g1_msm_batch)(b, k)}
        if mode == "single":
            args = lambda P: [P("bases"), P("k"), n, window, P("out"), P("scratch"), P("stream")]  # noqa: E731
            scratch = _sb(ctx, sbn, deg, n, window)
        else:
            args = lambda P: [P("bases"), 1 if mode == "shared" else 0, P("k"), n, m, window, P("out"), P("scratch"), P("stream")]  # noqa: E731
            scratch = _sb(ctx, sbn, deg, n, m, window)
        return Case(fn, args, {"bases": b, "k": k}, {"bases": db, "k": dk}, {"out": _out(m * wj * 8)}, want, scratch)
    return Spec(fn, sbn, "msm-%s-%s-n%d-m%d-w%d" % (curve, mode, n, m, window), build)


def _msm_specs():
    specs = []
    for g2 in (False, True):
        for n in (1, 31, 1000, 1 << 10, 1 << 11, 1 << 13, 1 << 14):
            specs += [_msm_case(g2, "single", n, 1, 0), _msm_case(g2, "shared", n, 5, 0), _msm_case(g2, "own", n, 5, 0)]
        for n in (1, 31, 1000):
            for w in (2, 13):
                specs += [_msm_case(g2, "single", n, 1, w), _msm_case(g2, "shared", n, 5, w), _msm_case(g2, "own", n, 5, w)]
        specs += [_msm_case(g2, "own", 1 << 11, 1, 0), _msm_case(g2, "shared", 0, 3, 0), _msm_case(g2, "shared", 31, 0, 0)]
    return specs


# ---- batch normalisation

def _bn_case(g2, n):
    curve = "g2" if g2 else "g1"

    def build(ctx, pool):
        def jac(seed):
            k = dg.rand_scalars(n, seed, edge_cases=n > 1)                 # edge scalars first: 0 gives the identity
            gen = (o.g2_from_affine if g2 else o.g1_from_affine)(o.generators()[1 if g2 else 0])
            return (ctx.g2_mul if g2 else ctx.g1_mul)(np.repeat(gen, n, 0), k)
        v, dv = jac(n), jac(n + 1)
        want = lambda: {"v": (ctx.g2_batch_normalization if g2 else ctx.g1_batch_normalization)(v)}  # noqa: E731
        return Case("bls_%s_batch_normalization_dev" % curve, lambda P: [P("v"), n, P("scratch"), P("stream")], {"v": v}, {"v": dv}, {},
                    want, _sb(ctx, "bls_batch_normalization_scratch_bytes", 2 if g2 else 1, n), inout=("v",))
    return Spec("bls_%s_batch_normalization_dev" % curve, "bls_batch_normalization_scratch_bytes", "bn-%s-n%d" % (curve, n), build)


# ---- products of pairs and of Fq12 values

def _pairs(pool, n, shift):
    p, q = pool.take(False, n, shift), pool.take(True, n, shift + 3)
    if n > 2:
        p[1] = 0
        p[1, -1] = 1                                                       # a pair with P at infinity contributes one
    return p, q


def _product_case(what, n):
    fn = {"mm": "bls_multi_miller_loop_dev", "pp": "bls_pairing_product_dev", "fq12": "bls_fq12_product_dev"}[what]
    sbn = "bls_fq12_product_scratch_bytes" if what == "fq12" else "bls_multi_miller_scratch_bytes"

    def build(ctx, pool):
        scratch = _sb(ctx, sbn, n)
        if what == "fq12":
            f, df = dg.rand_field(n, 12, n), dg.rand_field(n, 12, n + 1)
            return Case(fn, lambda P: [P("f"), n, P("out"), P("scratch"), P("stream")], {"f": f}, {"f": df}, {"out": _out(W12 * 8)},
                        lambda: {"out": ctx.fq12_product(f)}, scratch)
        (p, q), (dp, dq) = _pairs(pool, n, 0), _pairs(pool, n, 11)
        if what == "mm":
            return Case(fn, lambda P: [P("p"), P("q"), n, P("out"), P("scratch"), P("stream")], {"p": p, "q": q}, {"p": dp, "q": dq},
                        {"out": _out(W12 * 8)}, lambda: {"out": ctx.multi_miller_loop(p, q)}, scratch)

        def want():
            out, some = ctx.pairing_product(p, q)
            return {"out": out, "is_some": np.array([some], np.uint8)}
        return Case(fn, lambda P: [P("p"), P("q"), n, P("out"), P("is_some"), P("scratch"), P("stream")], {"p": p, "q": q},
                    {"p": dp, "q": dq}, {"out": _out(W12 * 8), "is_some": _out(1, 1)}, want, scratch)
    return Spec(fn, sbn, "%s-n%d" % (what, n), build)


# ---- Groth16

PROVE_SHAPES = [(1, 1, 0), (5, 2, 3), (33, 1, 5), (1020, 5, 30)]          # the last has len 1025


def _prove_case(nc, ni, na, m):
    def build(ctx, pool):
        import pairing_b200._native as nat
        toy = Toy(nc, ni, na, 2 * m, nc * 7 + ni * 3 + na)                 # witnesses 0 .. m-1 are real, m .. 2m-1 the decoy
        pr = toy.params
        length = toy.len
        sets = [{"a": toy.abc[0][s], "b": toy.abc[1][s], "c": toy.abc[2][s], "input": toy.input[s], "aux": toy.aux[s], "r": toy.r[s],
                 "s": toy.s[s]} for s in (slice(0, m), slice(m, 2 * m))]
        queries = {"qh": (pr.h, False), "ql": (pr.l, False), "qa": (pr.a, False), "qb1": (pr.b_g1, False), "qb2": (pr.b_g2, True)}
        for name, (rows, g2) in queries.items():
            sets[0][name] = rows
            sets[1][name] = pool.take(g2, len(rows), 17)
        dw = [nat.density_words(d, bits, "d") for d, bits in zip(toy.densities, (na, ni, na))]
        pc_host = nat.groth16_params_c(pr, nat._p, len)
        scratch = int(ctx.groth16_prove_scratch_bytes(pc_host, length, ni, na, dw, m))
        rows = {name: len(r) for name, (r, _) in queries.items()}

        def args(P):
            pc = nat.groth16_params_c(nat.Groth16Params(pr.alpha_g1, pr.beta_g1, pr.delta_g1, pr.beta_g2, pr.delta_g2, "qh", "ql", "qa", "qb1",
                                                        "qb2"), P, lambda q: rows[q])
            return [ctypes.byref(pc), P("a"), P("b"), P("c"), length, P("input"), ni, P("aux"), na, *[nat._p(w) for w in dw], P("r"),
                    P("s"), m, P("out"), P("scratch"), P("stream")]
        return Case("bls_groth16_prove_dev", args, sets[0], sets[1], {"out": _out(m * nat.W_PROOF * 8)}, lambda: {"out": toy.model()[:m]},
                    scratch)
    return Spec("bls_groth16_prove_dev", "bls_groth16_prove_scratch_bytes", "prove-%d-%d-%d-m%d" % (nc, ni, na, m), build)


def _verify_case(ni, m, rlc, valid=False):
    fn = "bls_groth16_verify_rlc_dev" if rlc else "bls_groth16_verify_dev"
    sbn = "bls_groth16_verify_rlc_scratch_bytes" if rlc else "bls_groth16_verify_scratch_bytes"

    def build(ctx, pool):
        def batch(seed, all_valid):
            vk = Vk(ctx, ni, seed)
            xs, exps, proofs, inputs = verify_batch(ctx, vk, 4 * m, seed)
            keep = [j for j in range(4 * m) if vk.model([xs[j]], [exps[j]])[0]][:m] if all_valid else list(range(m))
            rr = random.Random(seed)
            rho = _limbs([rr.randrange(1, R) for _ in range(m)])
            return vk, [xs[j] for j in keep], [exps[j] for j in keep], {"pvk": vk.pvk, "ic": vk.ic, "proofs": proofs[keep],
                                                                         "inputs": inputs[keep], "rho": rho}
        vk, xs, exps, real = batch(ni * 10 + m, valid)
        decoy = batch(ni * 10 + m + 500, not valid)[3]
        if rlc:
            want = lambda: {"ok1": np.array([ctx.groth16_verify_rlc(real["pvk"], real["ic"], real["proofs"], real["inputs"], real["rho"])], np.uint8)}  # noqa: E731
            return Case(fn, lambda P: [P("pvk"), P("ic"), ni, P("proofs"), P("inputs"), P("rho"), m, P("ok1"), P("scratch"), P("stream")],
                        real, decoy, {"ok1": _out(1, 1)}, want, _sb(ctx, sbn, ni, m))
        for d in (real, decoy):
            del d["rho"]
        want = lambda: {"ok": vk.model(xs, exps).astype(np.uint8)}  # noqa: E731
        return Case(fn, lambda P: [P("pvk"), P("ic"), ni, P("proofs"), P("inputs"), m, P("ok"), P("scratch"), P("stream")], real, decoy,
                    {"ok": _out(m, 1)}, want, _sb(ctx, sbn, ni, m))
    return Spec(fn, sbn, "%s-ni%d-m%d%s" % ("verify_rlc" if rlc else "verify", ni, m, "-valid" if valid else ""), build)


SETUP_SHAPES = [(0, 1, 2), (1, 1, 2), (1, 1, 0), (5, 2, 3), (12, 1, 12), (33, 1, 5)]   # nc 0 and 1: a domain of one point


def _setup_case(nc, ni, na):
    def build(ctx, pool):
        import pairing_b200._native as nat
        rng = random.Random(nc * 100 + ni * 10 + na)
        if nc <= 1 and na == 2:
            cons = [[{0: 5, 1: 1}, {2: 3}, {1: 7, 2: 2}]][:nc]
            abc, length = gs.csr_from_cons(cons, ni + na, seed=3), nc
        else:
            circ, abc = _toy(nc, ni, na, rng.randrange(1 << 30), dup=True)
            length = circ.length
        nv = ni + na
        sc = _scalars(rng)
        real, decoy = {}, {}
        for i, (off, cons_, coeff) in enumerate(abc):
            real.update({"off%d" % i: off, "cons%d" % i: cons_, "coeff%d" % i: coeff})
            other = _limbs([bm.fr_to_mont(rng.randrange(R)) for _ in range(len(cons_))]).reshape(-1, 4)
            decoy.update({"off%d" % i: off, "cons%d" % i: cons_, "coeff%d" % i: other})
        g1, g2 = o.generators()
        host = [g1[0], g2[0]] + [_mont1(x) for x in sc]
        nnz = [len(c) for _, c, _ in abc]
        host_mats = nat.r1cs_matrices(abc, length, nv)
        scratch = int(ctx.groth16_generate_parameters_scratch_bytes(host_mats[1], length, ni, na))
        key = gs.generate(abc, length, ni, na, sc[4], *sc[:4])
        n1 = (1 << max(length - 1, 0).bit_length()) - 1
        a_len, b_len = key["lens"]
        outs = {"vk": _out(nat.W_VK_POINTS * 8), "ic": _out(ni * W1 * 8), "h": _out(n1 * W1 * 8), "l": _out(na * W1 * 8),
                "a": _out(nv * W1 * 8, written=a_len * W1 * 8), "b_g1": _out(nv * W1 * 8, written=b_len * W1 * 8),
                "b_g2": _out(nv * W2 * 8, written=b_len * W2 * 8), "d0": _out((na + 31) // 32 * 4, 4), "d1": _out((ni + 31) // 32 * 4, 4),
                "d2": _out((na + 31) // 32 * 4, 4), "lens": _out(16), "ok": _out(1, 1)}

        def args(P):
            mats = (nat.R1csMatrixC * 3)()
            for i in range(3):
                mats[i] = nat.R1csMatrixC(P("off%d" % i), P("cons%d" % i), P("coeff%d" % i), nnz[i])
            out = nat.Groth16ParametersOutC(*[P(x) for x in ("vk", "ic", "h", "l", "a", "b_g1", "b_g2", "d0", "d1", "d2", "lens", "ok")])
            return [mats, length, ni, na, *[nat._p(np.ascontiguousarray(x)) for x in host], ctypes.byref(out), P("scratch"), P("stream")]

        def want():
            e = _expect(key)
            w = {"vk": np.concatenate([e[name] for name, _, _ in nat.VK_POINT_ROWS]), "ic": e["ic"], "h": e["h"], "l": e["l"], "a": e["a"],
                 "b_g1": e["b_g1"], "b_g2": e["b_g2"], "lens": np.array(key["lens"], np.uint64), "ok": np.array([key["ok"]], np.uint8)}
            for i, (d, bits) in enumerate(zip(key["densities"], (na, ni, na))):
                w["d%d" % i] = nat.density_words(np.array(d, dtype=bool), bits, "d")
            return w
        return Case("bls_groth16_generate_parameters_dev", args, real, decoy, outs, want, scratch)
    return Spec("bls_groth16_generate_parameters_dev", "bls_groth16_generate_parameters_scratch_bytes", "setup-%d-%d-%d" % (nc, ni, na), build)


# ---- KZG

def _kzg_poly_case(what, n, m):
    fn = "bls_kzg_%s_dev" % what
    sbn = "bls_kzg_%s_scratch_bytes" % what

    def build(ctx, pool):
        rng = random.Random(n * 8 + m + (what == "open"))
        rows = n if what == "commit" else max(n - 1, 0)
        coeffs, p = _polys(rng, m, n)
        _, dp = _polys(rng, m, n)
        zs = [[0, 1, R - 1][j] if j < 3 and m > 1 else rng.randrange(R) for j in range(m)]
        real, decoy = {"srs": pool.take(False, rows), "p": p}, {"srs": pool.take(False, rows, 23), "p": dp}
        a = pool.e[:rows]
        scratch = _sb(ctx, sbn, n, m)
        if what == "commit":
            want = lambda: {"c": _pts(ctx, [km.commit(row, a) for row in coeffs])}  # noqa: E731
            return Case(fn, lambda P: [P("srs"), rows, P("p"), n, m, P("c"), P("scratch"), P("stream")], real, decoy,
                        {"c": _out(m * W1 * 8)}, want, scratch)
        real["z"], decoy["z"] = _fr(zs), _fr([rng.randrange(R) for _ in range(m)])

        def want():
            op = [km.open_(row, z, a) for row, z in zip(coeffs, zs)]
            return {"y": _fr([y for y, _ in op]).reshape(-1, 4)[:m], "proof": _pts(ctx, [w for _, w in op])}
        return Case(fn, lambda P: [P("srs"), rows, P("p"), n, P("z"), m, P("y"), P("proof"), P("scratch"), P("stream")], real, decoy,
                    {"y": _out(m * 32), "proof": _out(m * W1 * 8)}, want, scratch)
    return Spec(fn, sbn, "kzg_%s-n%d-m%d" % (what, n, m), build)


def _kzg_verify_case(m, rlc, valid=False):
    fn = "bls_kzg_verify_rlc_dev" if rlc else "bls_kzg_verify_dev"
    sbn = "bls_kzg_verify_rlc_scratch_bytes" if rlc else "bls_kzg_verify_scratch_bytes"

    def build(ctx, pool):
        def rows_of(seed, all_valid):
            key = Key(ctx, seed)
            rng = random.Random(seed)
            rows = [key.valid(rng) for _ in range(m)] if all_valid else kzg_cases(key, rng, m)
            c, y, z, w = Key.rows(ctx, rows)
            rho = [rng.randrange(1, R) for _ in range(m)]
            return key, rows, rho, {"pvk": key.pvk, "c": c, "y": y, "z": z, "proof": w, "rho": _limbs(rho)}
        key, rows, rho, real = rows_of(m * 3 + rlc, valid)
        decoy = rows_of(m * 3 + rlc + 100, not valid)[3]
        if rlc:
            return Case(fn, lambda P: [P("pvk"), P("c"), P("y"), P("z"), P("proof"), P("rho"), m, P("ok1"), P("scratch"), P("stream")], real,
                        decoy, {"ok1": _out(1, 1)}, lambda: {"ok1": np.array([km.rlc_verifies(key.tau, rows, rho)], np.uint8)},
                        _sb(ctx, sbn, m))
        for d in (real, decoy):
            del d["rho"]
        return Case(fn, lambda P: [P("pvk"), P("c"), P("y"), P("z"), P("proof"), m, P("ok"), P("scratch"), P("stream")], real, decoy,
                    {"ok": _out(m, 1)}, lambda: {"ok": np.array([km.verifies(key.tau, *r) for r in rows], np.uint8)}, _sb(ctx, sbn, m))
    return Spec(fn, sbn, "%s-m%d%s" % ("kzg_verify_rlc" if rlc else "kzg_verify", m, "-valid" if valid else ""), build)


# ---- point FFT and FK20

def _pfft_case(g2, kind, log_n, m):
    curve = "g2" if g2 else "g1"

    def build(ctx, pool):
        rng = random.Random(log_n * 64 + m * 8 + KINDS.index(kind) * 2 + g2)
        n = 1 << log_n
        rows = pfft_rows(rng, m, n, True)
        w = W2 if g2 else W1
        real = _pts(ctx, [e for r in rows for e in r], g2).reshape(m, n, w)
        decoy = _pts(ctx, [e for r in pfft_rows(rng, m, n, False) for e in r], g2).reshape(m, n, w)
        want = lambda: {"out": _pts(ctx, [e for r in rows for e in pm.point_fft(kind, r, log_n)], g2).reshape(m, n, w)}  # noqa: E731
        return Case("bls_%s_fft_dev" % curve, lambda P: [fm.FR_FFT_KINDS[kind], P("in"), P("out"), log_n, m, P("scratch"), P("stream")],
                    {"in": real}, {"in": decoy}, {"out": _out(real.nbytes)}, want,
                    _sb(ctx, "bls_point_fft_scratch_bytes", 2 if g2 else 1, log_n, m), inplace=("out", "in"))
    return Spec("bls_%s_fft_dev" % curve, "bls_point_fft_scratch_bytes", "pfft-%s-%s-log%d-m%d" % (curve, kind, log_n, m), build)


def _open_all_prepare_case(log_n):
    def build(ctx, pool):
        n = 1 << log_n
        tau, dtau = random.Random(log_n).randrange(R), random.Random(log_n + 50).randrange(R)
        srs, dsrs = _pts(ctx, km.powers(tau, n)), _pts(ctx, km.powers(dtau, n))
        return Case("bls_kzg_open_all_prepare_dev", lambda P: [P("srs"), n, log_n, P("table"), P("scratch"), P("stream")], {"srs": srs},
                    {"srs": dsrs}, {"table": _out(2 * n * W1 * 8)}, lambda: {"table": _pts(ctx, pm.fk20_table(km.powers(tau, n), log_n))},
                    _sb(ctx, "bls_kzg_open_all_prepare_scratch_bytes", log_n))
    return Spec("bls_kzg_open_all_prepare_dev", "bls_kzg_open_all_prepare_scratch_bytes", "open_all_prepare-log%d" % log_n, build)


def _open_all_case(log_n, m):
    def build(ctx, pool):
        n = 1 << log_n
        rng = random.Random(log_n * 4 + m)
        tables = [ctx.kzg_open_all_prepare(_pts(ctx, km.powers(rng.randrange(R), n)), log_n) for _ in range(2)]
        (_, p), (_, dp) = _polys(rng, m, n), _polys(rng, m, n)

        def want():
            y, proof = ctx.kzg_open_all(tables[0], p)
            return {"y": y, "proof": proof}
        return Case("bls_kzg_open_all_dev", lambda P: [P("table"), P("p"), log_n, m, P("y"), P("proof"), P("scratch"), P("stream")],
                    {"table": tables[0], "p": p}, {"table": tables[1], "p": dp}, {"y": _out(m * n * 32), "proof": _out(m * n * W1 * 8)}, want,
                    _sb(ctx, "bls_kzg_open_all_scratch_bytes", log_n, m))
    return Spec("bls_kzg_open_all_dev", "bls_kzg_open_all_scratch_bytes", "open_all-log%d-m%d" % (log_n, m), build)


# ---- entry points without scratch: the stream, output-guard and input checks

def _pair_case(what, n):
    fn = {"pairing": "bls_pairing_dev", "miller": "bls_miller_loop_dev", "projective": "bls_pairing_projective_dev"}[what]

    def build(ctx, pool):
        (p, q), (dp, dq) = _pairs(pool, n, 2), _pairs(pool, n, 31)
        if what == "projective":
            p, q, dp, dq = (o.g1_from_affine(x) if x.shape[1] == W1 else o.g2_from_affine(x) for x in (p, q, dp, dq))
            want = lambda: {"out": ctx.pairing_projective(p, q)}  # noqa: E731
        else:
            want = lambda: {"out": (ctx.pairing if what == "pairing" else ctx.miller_loop)(p, q)}  # noqa: E731
        return Case(fn, lambda P: [P("p"), P("q"), P("out"), n, P("stream")], {"p": p, "q": q}, {"p": dp, "q": dq},
                    {"out": _out(n * W12 * 8)}, want)
    return Spec(fn, None, "%s-n%d" % (what, n), build)


def _final_exp_case(n):
    def build(ctx, pool):
        f, df = (ctx.miller_loop(*_pairs(pool, n, s)) for s in (4, 40))
        f[n // 2] = 0                                                      # the reference's None: out all zero, is_some 0

        def want():
            out, ok = ctx.final_exponentiation(f)
            return {"out": out, "is_some": ok}
        return Case("bls_final_exponentiation_dev", lambda P: [P("f"), P("out"), P("is_some"), n, P("stream")], {"f": f}, {"f": df},
                    {"out": _out(n * W12 * 8), "is_some": _out(n, 1)}, want)
    return Spec("bls_final_exponentiation_dev", None, "final_exp-n%d" % n, build)


def _wnaf_case(g2, window, n=64):
    curve = "g2" if g2 else "g1"

    def build(ctx, pool):
        def jac(seed):
            return (o.g2_from_affine if g2 else o.g1_from_affine)(pool.take(g2, n, seed)), dg.rand_scalars(n, seed)
        (b, k), (db, dk) = jac(7), jac(8)
        want = lambda: {"out": (ctx.g2_wnaf_mul if g2 else ctx.g1_wnaf_mul)(b, k, window)}  # noqa: E731
        return Case("bls_%s_wnaf_mul_dev" % curve, lambda P: [P("bases"), P("k"), P("out"), n, window, P("stream")], {"bases": b, "k": k},
                    {"bases": db, "k": dk}, {"out": _out(b.nbytes)}, want)
    return Spec("bls_%s_wnaf_mul_dev" % curve, None, "wnaf-%s-w%d" % (curve, window), build)


def _fr_op_case(op, n=300):
    import pairing_b200._native as nat
    unary = op in ("inv", "from_repr", "sqr")

    def build(ctx, pool):
        rng = random.Random(n + len(op))
        vals = lambda: [0, 1, R - 1] + [rng.randrange(R) for _ in range(n - 3)]  # noqa: E731
        if op == "from_repr":                                              # values >= r give ok = 0
            a, da = _limbs(vals()[:-2] + [R, (1 << 256) - 1]), _limbs(vals())
        else:
            a, da = _fr(vals()), _fr(vals())
        real, decoy = {"a": a}, {"a": da}
        if not unary:
            real["b"], decoy["b"] = _fr(vals()), _fr(vals())

        def want():
            out, ok = ctx.fr_op(op, a, real.get("b"))
            return {"out": out, "ok": ok}
        return Case("bls_fr_op_dev", lambda P: [nat.OPS[op], P("a"), None if unary else P("b"), P("out"), P("ok"), n, P("stream")], real,
                    decoy, {"out": _out(a.nbytes), "ok": _out(n, 1)}, want, inplace=("out", "a"))
    return Spec("bls_fr_op_dev", None, "fr_op-%s" % op, build)


CASES = (
    [_fr_fft_case(kind, log_n, m) for kind in KINDS for log_n in (0, 1, 10, 11, 16) for m in (1, 3)]
    + [_groth16_h_case(length, m) for length in (1, 2, 1025, 4097) for m in (1, 3)]
    + _msm_specs()
    + [_bn_case(g2, n) for g2 in (False, True) for n in (1, 100, 5000)]
    + [_product_case(what, n) for what in ("mm", "pp", "fq12") for n in (1, 2, 129, 3000)]
    + [_prove_case(*shape, m) for shape in PROVE_SHAPES for m in (1, 3)]
    + [_verify_case(ni, m, rlc) for rlc in (False, True) for ni in (0, 1, 5) for m in (1, 7)]
    + [_verify_case(ni, 7, True, valid=True) for ni in (0, 5)]
    + [_setup_case(*shape) for shape in SETUP_SHAPES]
    + [_kzg_poly_case(what, n, m) for what in ("commit", "open") for n in (0, 1, 32, 33, 1024, 1025) for m in (1, 3)]
    + [_kzg_poly_case(what, 33, 0) for what in ("commit", "open")]
    + [_kzg_verify_case(m, rlc) for rlc in (False, True) for m in (1, 9)] + [_kzg_verify_case(9, True, valid=True)]
    + [_pfft_case(g2, kind, log_n, m) for g2 in (False, True) for kind in KINDS for log_n in (0, 1, 7) for m in (1, 3)]
    + [_pfft_case(False, "fft", 3, 0)]
    + [_open_all_prepare_case(log_n) for log_n in (0, 1, 5)]
    + [_open_all_case(log_n, m) for log_n in (0, 1, 5) for m in (1, 3)]
    + [_pair_case(what, n) for what in ("pairing", "miller") for n in (7, 3000)] + [_pair_case("projective", 7)]
    + [_final_exp_case(7)]
    + [_wnaf_case(g2, w) for g2 in (False, True) for w in (0, 9)]
    + [_fr_op_case(op) for op in ("mul", "sub", "inv", "from_repr")]
)


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_every_scratch_entry_point_has_a_case():
    """every *_dev declaration of the header with a `void* scratch` parameter has a case, and every *_scratch_bytes function
    sizes one"""
    header = open(os.path.join(ROOT, "include", "pairing_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    decls = re.findall(r"\bint\s+(bls_\w+_dev)\s*\(([^;]*)\)\s*;", header)
    scratch_dev = {name for name, params in decls if re.search(r"void\s*\*\s*scratch\b", params)}
    sizers = set(re.findall(r"\bsize_t\s+(bls_\w+_scratch_bytes)\s*\(", header))
    assert len(scratch_dev) >= 23 and len(sizers) >= 18, (sorted(scratch_dev), sorted(sizers))
    assert scratch_dev - {s.fn for s in CASES} == set()
    assert sizers - {s.sb for s in CASES} == set()
    assert all(s.sb for s in CASES if s.fn in scratch_dev)
    assert len({s.id for s in CASES}) == len(CASES)


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def pool(ctx):
    return Pool(ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", CASES, ids=[s.id for s in CASES])
def test_dev_contract(ctx, pool, spec):
    run_dev(ctx, spec.build(ctx, pool))
