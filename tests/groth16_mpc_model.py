"""Big-integer model of phase 2 of the Groth16 ceremony (phase2's MPCParameters::new) in exponent space, for a constraint
system in the CSR layout of bls_groth16_mpc_new_*.

Every transcript row is [e]g1 or [e]g2, so a transcript is known by its exponents: coeffs = L_q(tau), alpha_coeffs = alpha
L_q(tau), beta_coeffs = beta L_q(tau), coeffs_g2 (= coeffs for an honest transcript) and h_i = tau^i (tau^n - 1).  new() sums
them over the terms as the kernels do, so an honest transcript gives groth16_setup_model.generate(..., gamma = 1,
delta = 1).

TEST INFRASTRUCTURE ONLY: tests/test_gpu_groth16_mpc.py compares bls_groth16_mpc_new_* with it.
"""
from bls_model import R_ORDER, fr_from_mont
from groth16_h_model import domain_log
import groth16_setup_model as gs

R = R_ORDER


def transcript(num_constraints, tau, alpha, beta):
    """the exponents of powersoftau's prepare_phase2 rows for the domain of num_constraints"""
    log_n = domain_log(num_constraints)
    n = 1 << log_n
    lag = gs.lagrange(log_n, tau)
    zt = (pow(tau, n, R) - 1) % R
    return {"alpha_g1": alpha % R, "beta_g1": beta % R, "beta_g2": beta % R, "coeffs_g1": lag,
            "alpha_coeffs_g1": [alpha * x % R for x in lag], "beta_coeffs_g1": [beta * x % R for x in lag],
            "coeffs_g2": list(lag), "h": [pow(tau, i, R) * zt % R for i in range(n - 1)]}


def _sums(mat, nv, rows):
    offsets, cons, coeff = mat
    c = coeff.astype(object)
    vals = [fr_from_mont(int(x)) for x in c[:, 0] + (c[:, 1] << 64) + (c[:, 2] << 128) + (c[:, 3] << 192)] if len(c) else []
    out = [0] * nv
    for v in range(nv):
        for e in range(int(offsets[v]), int(offsets[v + 1])):
            out[v] = (out[v] + vals[e] * rows[int(cons[e])]) % R
    return out


def new(abc, num_constraints, ni, na, ph):
    """the key's exponents in groth16_setup_model.generate's format, with b_g2 apart (an inconsistent transcript can make it
    differ from b) and gamma = delta = 1 (the generators)"""
    nv = ni + na
    A, B, C = abc
    a = _sums(A, nv, ph["coeffs_g1"])
    bg1 = _sums(B, nv, ph["coeffs_g1"])
    bg2 = _sums(B, nv, ph["coeffs_g2"])
    ext = [(x + y + z) % R for x, y, z in zip(_sums(A, nv, ph["beta_coeffs_g1"]), _sums(B, nv, ph["alpha_coeffs_g1"]), _sums(C, nv, ph["coeffs_g1"]))]
    l = ext[ni:]
    return {
        "alpha": ph["alpha_g1"], "beta": ph["beta_g1"], "beta_g2": ph["beta_g2"], "gamma": 1, "delta": 1,
        "h": list(ph["h"]), "ic": ext[:ni], "l": l, "a": [x for x in a if x], "b": [x for x in bg1 if x], "b_g2": [x for x in bg2 if x],
        "densities": ([a[ni + i] != 0 for i in range(na)], [bg1[i] != 0 for i in range(ni)], [bg1[ni + i] != 0 for i in range(na)]),
        "lens": (len([x for x in a if x]), len([x for x in bg1 if x])),
        "ok": all(l) and all((x == 0) == (y == 0) for x, y in zip(bg1, bg2)),
    }


def contribute(key, delta, s, r):
    """phase2's contribute in exponents: (the new key, the pubkey exponents (delta_after, s, s_delta, r, r_delta))"""
    d = pow(delta, -1, R)
    new = dict(key, delta=key["delta"] * delta % R, h=[x * d % R for x in key["h"]], l=[x * d % R for x in key["l"]])
    return new, (new["delta"], s % R, s * delta % R, r % R, r * delta % R)


def verify(before, after, pks, rho_h, rho_l):
    """phase2's verify in exponents: e(A, B) = e(C, D) is a b == c d (mod r).  before / after hold h, l, ic, a, b, b_g2, alpha,
    beta, gamma, delta (delta_g1 and delta_g2 share the exponent unless delta_g2 is given)."""
    for name in ("ic", "a", "b", "b_g2", "alpha", "beta", "gamma"):
        if before[name] != after[name]:
            return False
    if len(before["h"]) != len(after["h"]) or len(before["l"]) != len(after["l"]):
        return False
    same = lambda a, b, c, d: a * b % R == c * d % R                                     # noqa: E731
    bd1, bd2 = before["delta"], before.get("delta_g2", before["delta"])
    ad1, ad2 = after["delta"], after.get("delta_g2", after["delta"])
    prev = bd1
    for da, s, sd, r, rd in pks:
        if not (same(sd, r, s, rd) and same(prev, rd, da, r)):
            return False
        prev = da
    if ad1 != prev or not same(bd1, ad2, prev, bd2):
        return False
    for q, rho in (("h", rho_h), ("l", rho_l)):
        sb = sum(x * y for x, y in zip(rho, before[q])) % R
        sa = sum(x * y for x, y in zip(rho, after[q])) % R
        if not same(sb, bd2, sa, ad2):
            return False
    return True
