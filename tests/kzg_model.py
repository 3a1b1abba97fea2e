"""KZG polynomial commitments in exponent space: every G1 point is [e] g and every G2 point [e] h, so a commitment, an opening
proof and a verdict are integers mod r.  The SRS exponents are tau^i (or any known a_i: commit and open are linear in the
bases), a commitment is p(tau), an opening (p(z), q(tau)) with q from synthetic division, and a proof verifies iff
c - y + z w == tau w (mod r), the exponent of FE(ML(C - y g + z W, h) * ML(W, -tau h)) == 1."""
from bls_model import R_ORDER

R = R_ORDER


def evaluate(p, x):
    """p(x) mod r by Horner"""
    acc = 0
    for c in reversed(p):
        acc = (acc * x + c) % R
    return acc


def quotient(p, z):
    """(y, q) with p(X) = q(X) (X - z) + y: q_(n-2) = p_(n-1), q_(i-1) = p_i + z q_i, y = p_0 + z q_0; n = 0 gives (0, [])"""
    n = len(p)
    if n == 0:
        return 0, []
    q = [0] * (n - 1)
    acc = p[n - 1] % R
    for i in range(n - 1, 0, -1):
        q[i - 1] = acc
        acc = (p[i - 1] + z * acc) % R
    return acc, q


def commit(p, bases):
    """the exponent of sum_i p_i [a_i] g for base exponents a_i (tau^i for a real SRS)"""
    return sum(c * a for c, a in zip(p, bases)) % R


def open_(p, z, bases):
    """(y, w): y = p(z), w the exponent of [q(tau)] g over the base exponents"""
    y, q = quotient(p, z)
    return y, commit(q, bases)


def powers(tau, n):
    return [pow(tau, i, R) for i in range(n)]


def residual(tau, c, y, z, w):
    return (c - y + z * w - tau * w) % R


def verifies(tau, c, y, z, w):
    """the per-proof verdict; y and z are the integers the caller passed, rejected (not reduced) when >= r"""
    return y < R and z < R and residual(tau, c, y, z, w) == 0


def rlc_verifies(tau, rows, rho):
    """the randomized verdict over rows (c, y, z, w): sum_j rho_j (c_j - y_j + z_j w_j - tau w_j) == 0, and every y, z < r"""
    if any(y >= R or z >= R for _, y, z, _ in rows):
        return False
    return sum(r * residual(tau, *row) for r, row in zip(rho, rows)) % R == 0
