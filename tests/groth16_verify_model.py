"""Big-integer model of bellman's groth16::verify_proof and of the randomized batch check, in exponent space.

Every point is [e]g for a known exponent e (a point at infinity has e = 0, and a pairing with it is one = e(g1, g2)^0, which is
the dead-pair rule of Engine::miller_loop).  With the key's exponents alpha, beta, gamma, delta and ic, and x_j the canonical
public inputs of proof j (without bellman's leading one), acc_j = ic_0 + sum_i x_ji ic_(i+1) and

    verify_proof(A, B, C)  <=>  a b == alpha beta + gamma acc_j + delta c                              (mod r)
    the randomized check    <=>  sum_j rho_j (a_j b_j - alpha beta - gamma acc_j - delta c_j) == 0     (mod r)

for any exponents, adversarial ones included: the pairing is a bijection from exponents to GT (e(g1, g2) has order r).

TEST INFRASTRUCTURE ONLY: tests/test_gpu_groth16_verify.py compares bls_groth16_verify_* with it.
"""
from bls_model import R_ORDER

R = R_ORDER


def acc(key, inputs):
    """the exponent of ic_0 + sum_i x_i ic_(i+1); key["ic"] holds len(inputs) + 1 exponents"""
    assert len(key["ic"]) == len(inputs) + 1
    return (key["ic"][0] + sum(x * e for x, e in zip(inputs, key["ic"][1:]))) % R


def residual(key, inputs, proof):
    """a b - alpha beta - gamma acc - delta c (mod r): zero iff the proof verifies"""
    a, b, c = proof
    return (a * b - key["alpha"] * key["beta"] - key["gamma"] * acc(key, inputs) - key["delta"] * c) % R


def verifies(key, inputs, proof):
    return residual(key, inputs, proof) == 0


def rlc_verifies(key, inputs, proofs, rho):
    """the verdict of FE(prod_j ML(rho_j A_j, B_j) ML(sum_i s_i ic_i, -gamma) ML(sum_j rho_j C_j, -delta)) == e(alpha, beta)^(sum rho)"""
    return sum(r * residual(key, x, p) for r, x, p in zip(rho, inputs, proofs)) % R == 0


def solve_c(key, inputs, a, b):
    """the c that makes (a, b, c) verify"""
    return (a * b - key["alpha"] * key["beta"] - key["gamma"] * acc(key, inputs)) * pow(key["delta"], -1, R) % R


def solve_b(key, inputs, a, c):
    """the b that makes (a, b, c) verify, a != 0"""
    return (key["alpha"] * key["beta"] + key["gamma"] * acc(key, inputs) + key["delta"] * c) * pow(a, -1, R) % R


def inputs_with_zero_acc(key, inputs):
    """inputs with x_0 changed so that acc == 0 (acc_j at infinity); needs len(inputs) >= 1 and ic_1 != 0"""
    rest = (key["ic"][0] + sum(x * e for x, e in zip(inputs[1:], key["ic"][2:]))) % R
    return [(-rest) * pow(key["ic"][1], -1, R) % R] + list(inputs[1:])
