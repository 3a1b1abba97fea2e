"""Big-integer model of bellman's groth16::create_proof in exponent space, and a toy trusted setup.

Every key point is [e]g for a known exponent e, so a proof is three exponents: with every scalar through into_repr() and
rank_D(i) the number of set bits of D below i,

    a_ans  = sum_{i < num_inputs} input_i a[i] + sum_{a_aux[i]} aux_i a[num_inputs + rank_a_aux(i)]
    b_ans  = sum_{b_in[i]} input_i b[rank_b_in(i)] + sum_{b_aux[i]} aux_i b[popcount(b_in) + rank_b_aux(i)]
    A = r delta + alpha + a_ans,  B = s delta + beta + b_ans (over the b_g2 exponents)
    C = (r s) delta + s (alpha + a_ans) + r (beta + b_ans over b_g1) + sum_{i < n-1} H_i h[i] + sum_{i < num_aux} aux_i l[i]
                                                                                                                (mod r)

with H from tests/groth16_h_model.py.  The toy setup follows bellman's generator with known tau, alpha, beta, gamma, delta:
u_i(tau), v_i(tau), w_i(tau) through the Lagrange basis of the size-n domain, the a and b queries filtered of zero entries
(which yields the density bitmaps), l_i = (beta u_i + alpha v_i + w_i) / delta, ic_i = (...) / gamma and
h_i = tau^i (tau^n - 1) / delta.  Its proofs satisfy A B = alpha beta + gamma sum_i input_i ic_i + delta C (mod r).

TEST INFRASTRUCTURE ONLY: tests/test_gpu_groth16_prove.py checks the model against that equation and compares
bls_groth16_prove_* with it.
"""
import random

from bls_model import R_ORDER, fr_from_mont, fr_to_mont
from fr_fft_model import fr_root
from groth16_h_model import domain_log, groth16_h

R = R_ORDER


def _rank(d, i):
    return sum(1 for x in d[:i] if x)


def create_proof(key, a, b, c, inputs, aux, densities, r, s):
    """one proof: key = dict of exponents alpha, beta, delta (ints) and h, l, a, b_g1, b_g2 (lists); a, b, c, inputs, aux
    lists of Montgomery-form ints; densities = (a_aux, b_input, b_aux) lists of bools; r, s Montgomery-form ints ->
    the exponents (A, B, C), canonical"""
    a_aux, b_in, b_aux = densities
    x_in = [fr_from_mont(v) for v in inputs]
    x_aux = [fr_from_mont(v) for v in aux]
    ni, pop_b_in = len(x_in), sum(1 for x in b_in if x)
    h = groth16_h(a, b, c) if len(a) > 1 else []
    h_ans = sum(x * e for x, e in zip(h, key["h"]))
    l_ans = sum(x * key["l"][i] for i, x in enumerate(x_aux))
    a_ans = sum(x * key["a"][i] for i, x in enumerate(x_in))
    a_ans += sum(x * key["a"][ni + _rank(a_aux, i)] for i, x in enumerate(x_aux) if a_aux[i])

    def b_ans(q):
        t = sum(x * q[_rank(b_in, i)] for i, x in enumerate(x_in) if b_in[i])
        return t + sum(x * q[pop_b_in + _rank(b_aux, i)] for i, x in enumerate(x_aux) if b_aux[i])
    rr, ss = fr_from_mont(r), fr_from_mont(s)
    ea = (rr * key["delta"] + key["alpha"] + a_ans) % R
    eb = (ss * key["delta"] + key["beta"] + b_ans(key["b_g2"])) % R
    ec = (rr * ss * key["delta"] + ss * (key["alpha"] + a_ans) + rr * (key["beta"] + b_ans(key["b_g1"])) + h_ans + l_ans) % R
    return ea, eb, ec


def _lagrange_at(log_n, tau):
    """L_q(tau) for the n points omega^q: omega^q (tau^n - 1) / (n (tau - omega^q))"""
    n = 1 << log_n
    w = fr_root(log_n)
    zt = (pow(tau, n, R) - 1) % R
    out, wq = [], 1
    for _ in range(n):
        out.append(wq * zt * pow(n * (tau - wq), -1, R) % R)
        wq = wq * w % R
    return out


class ToyCircuit:
    """A random R1CS system over num_inputs inputs (input 0 = one) and num_aux aux variables, with its toy trusted setup.
    Constraint q: (A_q . z)(B_q . z) = C_q . z, z = inputs ++ aux, each of A_q, B_q, C_q a dict variable -> coefficient.
    The last min(num_constraints, num_aux) aux variables are outputs: constraint q with output o has A_q, B_q over the
    variables before o and C_q = c o, so every choice of the inputs and the other aux values extends to a witness.  A
    constraint without an output is one * x_k = x_k scaled, which every witness satisfies."""

    def __init__(self, num_constraints, num_inputs, num_aux, seed, sparsity=0.3):
        assert num_inputs >= 1
        rng = random.Random(seed)
        self.ni, self.na = num_inputs, num_aux
        self.outputs = min(num_constraints, num_aux)
        self.free = num_aux - self.outputs
        self.cons = []
        for q in range(num_constraints):
            if q < self.outputs:
                o = num_inputs + self.free + q
                lcs = [{v: rng.choice([1, R - 1, rng.randrange(1, R)]) for v in range(o) if rng.random() < sparsity} for _ in range(2)]
                lcs.append({o: rng.randrange(1, R)})
            else:
                k, c1, c2 = rng.randrange(num_inputs), rng.randrange(1, R), rng.randrange(1, R)
                lcs = [{0: c1}, {k: c2}, {k: c1 * c2 % R}]
            self.cons.append(lcs)
        # bellman's generator and prover append input_i * 0 = 0 for every input
        self.all_cons = self.cons + [[{i: 1}, {}, {}] for i in range(num_inputs)]
        self.length = len(self.all_cons)
        self.log_n = domain_log(self.length)

    def witness(self, seed):
        """canonical (inputs, aux) that satisfy every constraint, inputs[0] = 1; 0 and 1 among the free values"""
        rng = random.Random(seed)
        z = [1] + [rng.randrange(R) for _ in range(self.ni - 1)] + [rng.choice([0, 1, rng.randrange(R)]) for _ in range(self.free)]
        for con in self.cons[:self.outputs]:
            a, b = (sum(co * z[v] for v, co in lc.items()) % R for lc in con[:2])
            (o, co), = con[2].items()
            z.append(a * b * pow(co, -1, R) % R)
        return z[:self.ni], z[self.ni:]

    def evaluations(self, inputs, aux):
        """the ProvingAssignment vectors a, b, c (canonical), the input constraints included"""
        z = inputs + aux
        ev = [[sum(co * z[v] for v, co in lc.items()) % R for lc in con] for con in self.all_cons]
        return [e[0] for e in ev], [e[1] for e in ev], [e[2] for e in ev]

    def setup(self, tau, alpha, beta, gamma, delta):
        """the key's exponents (bellman's generator): alpha, beta, gamma, delta, h, l, a, b_g1, b_g2, ic and the densities"""
        lag = _lagrange_at(self.log_n, tau)
        nv = self.ni + self.na
        u, v, w = ([0] * nv for _ in range(3))
        for q, con in enumerate(self.all_cons):
            for k, vec in enumerate((u, v, w)):
                for var, co in con[k].items():
                    vec[var] = (vec[var] + co * lag[q]) % R
        n = 1 << self.log_n
        zt = (pow(tau, n, R) - 1) % R
        di, gi = pow(delta, -1, R), pow(gamma, -1, R)
        k_all = [(beta * u[i] + alpha * v[i] + w[i]) % R for i in range(nv)]
        a_aux = [u[self.ni + i] != 0 for i in range(self.na)]
        b_in = [v[i] != 0 for i in range(self.ni)]
        b_aux = [v[self.ni + i] != 0 for i in range(self.na)]
        a_q = [u[i] for i in range(self.ni)] + [u[self.ni + i] for i in range(self.na) if a_aux[i]]
        b_q = [v[i] for i in range(self.ni) if b_in[i]] + [v[self.ni + i] for i in range(self.na) if b_aux[i]]
        return {
            "alpha": alpha, "beta": beta, "gamma": gamma, "delta": delta,
            "h": [pow(tau, i, R) * zt * di % R for i in range(n - 1)],
            "l": [k_all[self.ni + i] * di % R for i in range(self.na)],
            "ic": [k_all[i] * gi % R for i in range(self.ni)],
            "a": a_q, "b_g1": b_q, "b_g2": list(b_q),
            "densities": (a_aux, b_in, b_aux),
        }


def mont(values):
    return [fr_to_mont(x % R) for x in values]


def verifies(key, inputs, proof):
    """A B = alpha beta + gamma sum_i input_i ic_i + delta C (mod r), inputs canonical"""
    ea, eb, ec = proof
    ic = sum(x * e for x, e in zip(inputs, key["ic"]))
    return ea * eb % R == (key["alpha"] * key["beta"] + key["gamma"] * ic + key["delta"] * ec) % R
