"""Big-integer model of Groth16's quotient polynomial H: the `h` block of bellman's groth16::create_proof on top of
tests/fr_fft_model.py::fr_fft.  For the evaluations a, b, c of one proof (Montgomery-form ints, len each):

    n = the smallest power of two >= len (1 for len <= 1); A, B, C = zero-padded to n   (EvaluationDomain::from_coeffs)
    A, B, C = coset_fft(ifft(.))
    H = (A B - C) * z(g)^-1, z(g) = g^n - 1, g = 7            (mul_assign, sub_assign, divide_by_z_on_coset)
    H = icoset_fft(H); drop coefficient n - 1; into_repr() every coefficient

TEST INFRASTRUCTURE ONLY: tests/test_gpu_groth16_h.py compares bls_fr_groth16_h_* with it and checks it against the
defining identity H(tau) (tau^n - 1) = A(tau) B(tau) - C(tau) of satisfied inputs, and tools/gen_fr_fft_consts.py's
FR_Z_INV table is z_inv() of every log_n.
"""
from bls_model import R_ORDER, fr_from_mont, fr_to_mont
from fr_fft_model import FR_GENERATOR, fr_fft


def domain_log(length):
    """log_n of the domain of len evaluations: n = 2^log_n >= len, 0 for len <= 1"""
    return max(length - 1, 0).bit_length()


def z_inv(log_n):
    """(g^n - 1)^-1, canonical: divide_by_z_on_coset's constant"""
    return pow(pow(FR_GENERATOR, 1 << log_n, R_ORDER) - 1, -1, R_ORDER)


def groth16_h_full(a, b, c):
    """one proof: a, b, c lists of len Montgomery-form ints -> all n coefficients of H as canonical ints, the last one
    included (it is 0 when c_i = a_i b_i for every i)"""
    length = len(a)
    assert len(b) == length and len(c) == length
    log_n = domain_log(length)
    n = 1 << log_n
    ev = []
    for x in (a, b, c):
        x = list(x) + [0] * (n - length)
        ev.append([fr_from_mont(v) for v in fr_fft("coset_fft", fr_fft("ifft", x, log_n), log_n)])
    zi = z_inv(log_n)
    h = [fr_to_mont((x * y - z) * zi % R_ORDER) for x, y, z in zip(*ev)]
    return [fr_from_mont(v) for v in fr_fft("icoset_fft", h, log_n)]


def groth16_h(a, b, c):
    """one proof: a, b, c lists of len Montgomery-form ints -> n - 1 canonical ints, the FrRepr values bellman passes to
    the `h` multiexp"""
    return groth16_h_full(a, b, c)[:-1]
