"""Big-integer model of the radix-2 FFT over Fr: bellman's EvaluationDomain (fft / ifft / coset_fft / icoset_fft) with the
crate's PrimeField constants for Fr (fr.rs: S = 32, multiplicative_generator() = 7, root_of_unity() = 7^t with
r - 1 = t * 2^32, t odd).  Values are Montgomery-form ints, inputs and outputs in natural order.

TEST INFRASTRUCTURE ONLY, on top of oracle/bls_model.py (the modulus and the Montgomery conversions of Fr):
tests/test_gpu_fft.py compares the kernels with it and checks it against a direct O(n^2) DFT, and
tools/gen_fr_fft_consts.py derives the constants the kernels embed from it.
"""
from bls_model import R_ORDER, fr_from_mont, fr_to_mont

FR_S = 32
FR_GENERATOR = 7
FR_T = (R_ORDER - 1) >> FR_S
FR_ROOT_OF_UNITY = pow(FR_GENERATOR, FR_T, R_ORDER)    # canonical integer, a primitive 2^32-th root of unity
FR_FFT, FR_IFFT, FR_COSET_FFT, FR_ICOSET_FFT = 0, 1, 2, 3
FR_FFT_KINDS = {"fft": FR_FFT, "ifft": FR_IFFT, "coset_fft": FR_COSET_FFT, "icoset_fft": FR_ICOSET_FFT}


def fr_root(log_n):
    """canonical omega of the domain of size 2^log_n: root_of_unity() squared (32 - log_n) times"""
    w = FR_ROOT_OF_UNITY
    for _ in range(FR_S - log_n):
        w = w * w % R_ORDER
    return w


def _fr_radix2(a, w):
    """in-place iterative radix-2 transform of canonical ints: a[i] <- sum_j a[j] w^(ij) (bellman's serial_fft)"""
    n = len(a)
    log_n = n.bit_length() - 1
    for k in range(n):
        rk = int(format(k, "0%db" % log_n)[::-1], 2) if log_n else 0
        if k < rk:
            a[k], a[rk] = a[rk], a[k]
    m = 1
    while m < n:
        w_m = pow(w, n // (2 * m), R_ORDER)
        for k in range(0, n, 2 * m):
            t = 1
            for j in range(m):
                u, v = a[k + j], a[k + j + m] * t % R_ORDER
                a[k + j], a[k + j + m] = (u + v) % R_ORDER, (u - v) % R_ORDER
                t = t * w_m % R_ORDER
        m *= 2
    return a


def _fr_distribute_powers(a, g):
    """a[j] <- a[j] g^j (bellman's distribute_powers)"""
    out, u = [], 1
    for x in a:
        out.append(x * u % R_ORDER)
        u = u * g % R_ORDER
    return out


def fr_fft(kind, values, log_n):
    """One polynomial of 2^log_n Montgomery-form Fr values -> its transform (Montgomery form), natural order:
    fft: sum_j a_j w^(ij); ifft: n^-1 sum_j a_j w^(-ij); coset_fft: distribute_powers(g) then fft;
    icoset_fft: ifft then distribute_powers(g^-1)."""
    kind = FR_FFT_KINDS.get(kind, kind)
    n = 1 << log_n
    assert len(values) == n
    a = [fr_from_mont(int(v)) for v in values]
    w = fr_root(log_n)
    if kind == FR_COSET_FFT:
        a = _fr_distribute_powers(a, FR_GENERATOR)
    if kind in (FR_IFFT, FR_ICOSET_FFT):
        a = _fr_radix2(a, pow(w, -1, R_ORDER))
        ninv = pow(n, -1, R_ORDER)
        a = [x * ninv % R_ORDER for x in a]
        if kind == FR_ICOSET_FFT:
            a = _fr_distribute_powers(a, pow(FR_GENERATOR, -1, R_ORDER))
    else:
        a = _fr_radix2(a, w)
    return [fr_to_mont(x) for x in a]
