"""Big-integer model of bellman's groth16::generate_parameters in exponent space, for a constraint system in the CSR layout
of bls_groth16_generate_parameters_*.

Every point of the key is [e]g1 or [e]g2, so the key is known by its exponents.  With n the smallest power of two >=
num_constraints, Lq = L_q(tau) the Lagrange basis of the n points omega^q, and u, v, w the sums of coeff * Lq over the terms
of each variable in A, B and C:

    h_i = tau^i (tau^n - 1) / delta (i < n - 1),  ic_i = (beta u_i + alpha v_i + w_i) / gamma,  l_i = (...) / delta
    a = [u_v for every variable if u_v != 0],  b = [v_v for every variable if v_v != 0]   (bellman drops identity points,
                                                                                           inputs included)
    densities: a_aux[i] = u_(ni+i) != 0, b_input[i] = v_i != 0, b_aux[i] = v_(ni+i) != 0;  ok = no l_i is zero

tests/groth16_prove_model.py::ToyCircuit.setup restates the same generator for its constraint-major circuits, but keeps
every input in `a`; agree() is the comparison that allows for that.

TEST INFRASTRUCTURE ONLY: tests/test_gpu_groth16_setup.py compares bls_groth16_generate_parameters_* with it.
"""
import random

import numpy as np

from bls_model import R_ORDER, fr_from_mont, fr_to_mont
from fr_fft_model import fr_root
from groth16_h_model import domain_log
from groth16_prove_model import _lagrange_at

R = R_ORDER


def lagrange(log_n, tau):
    """L_q(tau) for q < n; a unit vector when tau is a domain point omega^k (where _lagrange_at would divide by zero)"""
    n = 1 << log_n
    w, wq = fr_root(log_n), 1
    for k in range(n):
        if wq == tau % R:
            return [1 if q == k else 0 for q in range(n)]
        wq = wq * w % R
    return _lagrange_at(log_n, tau % R)


def _limbs(values):
    return np.array([[(v >> (64 * i)) & (2 ** 64 - 1) for i in range(4)] for v in values], dtype=np.uint64).reshape(-1, 4)


def csr_from_cons(all_cons, nv, seed=None):
    """constraint-major dicts (ToyCircuit.all_cons: per constraint three dicts variable -> canonical coefficient) -> the three
    (offsets uint64, constraint uint32, coeff (nnz, 4) Montgomery uint64) triples.  With a seed, some terms are split in two
    (same constraint twice) and zero-coefficient terms are added, as KeypairAssembly may record them; the sums are unchanged."""
    rng = random.Random(seed)
    out = []
    for k in range(3):
        terms = [[] for _ in range(nv)]
        for q, con in enumerate(all_cons):
            for var, co in con[k].items():
                if seed is not None and rng.random() < 0.3:
                    part = rng.randrange(R)
                    terms[var] += [(q, part), (q, (co - part) % R)]
                else:
                    terms[var].append((q, co % R))
                if seed is not None and rng.random() < 0.2:
                    terms[var].append((rng.randrange(len(all_cons)), 0))
        if seed is not None:
            for t in terms:
                rng.shuffle(t)
        offsets = np.zeros(nv + 1, dtype=np.uint64)
        offsets[1:] = np.cumsum([len(t) for t in terms]) if nv else []
        flat = [x for t in terms for x in t]
        cons = np.array([q for q, _ in flat], dtype=np.uint32)
        coeff = _limbs([fr_to_mont(c) for _, c in flat])
        out.append((offsets, cons, coeff))
    return out


def qap(abc, num_constraints, nv, tau):
    """u, v, w (canonical ints) of every variable"""
    lag = lagrange(domain_log(num_constraints), tau)
    res = []
    for offsets, cons, coeff in abc:
        c = coeff.astype(object)
        vals = [fr_from_mont(int(x)) for x in c[:, 0] + (c[:, 1] << 64) + (c[:, 2] << 128) + (c[:, 3] << 192)] if len(c) else []
        sums = [0] * nv
        for var in range(nv):
            for e in range(int(offsets[var]), int(offsets[var + 1])):
                sums[var] = (sums[var] + vals[e] * lag[int(cons[e])]) % R
        res.append(sums)
    return res


def generate(abc, num_constraints, ni, na, tau, alpha, beta, gamma, delta):
    """the key's exponents (canonical ints): alpha, beta, gamma, delta, h, ic, l, a, b (the b_g1 and b_g2 exponents), the
    densities (three bool lists), lens (a_len, b_len) and ok"""
    nv = ni + na
    u, v, w = qap(abc, num_constraints, nv, tau)
    n = 1 << domain_log(num_constraints)
    zt = (pow(tau, n, R) - 1) % R
    gi, di = pow(gamma, -1, R), pow(delta, -1, R)
    k = [(beta * u[i] + alpha * v[i] + w[i]) % R for i in range(nv)]
    a = [x for x in u if x]
    b = [x for x in v if x]
    l = [k[ni + i] * di % R for i in range(na)]
    return {
        "alpha": alpha, "beta": beta, "gamma": gamma, "delta": delta,
        "h": [pow(tau, i, R) * zt * di % R for i in range(n - 1)],
        "ic": [k[i] * gi % R for i in range(ni)], "l": l, "a": a, "b": b,
        "densities": ([u[ni + i] != 0 for i in range(na)], [v[i] != 0 for i in range(ni)], [v[ni + i] != 0 for i in range(na)]),
        "lens": (len(a), len(b)), "ok": all(l),
    }


def as_prove_key(key):
    """the dict groth16_prove_model.create_proof and verifies take"""
    return dict(key, b_g1=key["b"], b_g2=key["b"])
