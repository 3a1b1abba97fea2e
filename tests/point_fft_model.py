"""The point FFT and FK20 in exponent space: every point is [e] g, so a point transform is a transform of the exponents mod r,
and an FK20 proof is an integer that must equal kzg_model.open_'s.

point_fft restates the kernels' evaluation order -- bit-reversed load, radix-2 decimation-in-time stages with twiddle
omega^(j n / 2h), the coset scaling g^i before the stages, one folded scalar n^-1 (g^-i) after them -- on canonical ints.
fk20_proofs restates bls_kzg_open_all_*: the table w of the SRS exponents, its FFT of size 2n, the element-wise products with
c-hat, the first n of the inverse transform (H), and FFT_n(H)."""
from bls_model import R_ORDER
from fr_fft_model import FR_GENERATOR, FR_FFT_KINDS, fr_root

R = R_ORDER
FFT, IFFT, COSET_FFT, ICOSET_FFT = 0, 1, 2, 3


def _rev(i, log_n):
    return int(format(i, "0%db" % log_n)[::-1], 2) if log_n else 0


def _stages(a, w, log_n):
    """the kernels' stages on a bit-reversed row: stage s pairs (i0, i0 + h), h = 2^s, twiddle w^(j n / 2h)"""
    n = 1 << log_n
    for s in range(log_n):
        h = 1 << s
        for g in range(0, n, 2 * h):
            for j in range(h):
                t = pow(w, j << (log_n - 1 - s), R) * a[g + j + h] % R
                a[g + j], a[g + j + h] = (a[g + j] + t) % R, (a[g + j] - t) % R
    return a


def point_fft(kind, exps, log_n, scaled=True):
    """exponents of the outputs of bls_g*_fft_* for inputs [exps[j]] g (canonical ints); scaled = False leaves out the inverse
    kinds' n^-1 (FK20's inverse transform)"""
    kind = FR_FFT_KINDS.get(kind, kind)
    n = 1 << log_n
    assert len(exps) == n
    a = [exps[_rev(p, log_n)] % R for p in range(n)]
    if kind == COSET_FFT:
        a = [a[p] * pow(FR_GENERATOR, _rev(p, log_n), R) % R for p in range(n)]
    w = fr_root(log_n)
    inv = kind in (IFFT, ICOSET_FFT)
    a = _stages(a, pow(w, -1, R) if inv else w, log_n)
    if inv and scaled:
        ninv = pow(n, -1, R)
        ginv = pow(FR_GENERATOR, -1, R)
        a = [x * ninv * (pow(ginv, i, R) if kind == ICOSET_FFT else 1) % R for i, x in enumerate(a)]
    return a


def fk20_table(srs, log_n):
    """the exponents of bls_kzg_open_all_prepare's 2n rows: FFT_2n(w), w_t = srs[2n - 1 - t] for n < t < 2n, 0 for t <= n"""
    n = 1 << log_n
    w = [srs[2 * n - 1 - t] if t > n else 0 for t in range(2 * n)]
    return point_fft(FFT, w, log_n + 1)


def fk20_proofs(coeffs, table, log_n):
    """the exponents of bls_kzg_open_all's n proofs of one polynomial, from the table's exponents"""
    n = 1 << log_n
    c = [x % R for x in coeffs] + [0] * n
    inv2n = pow(2 * n, -1, R)
    chat = [x * inv2n % R for x in point_fft(FFT, c, log_n + 1)]          # the Fr FFT: the same transform of integers
    h = point_fft(IFFT, [x * t % R for x, t in zip(chat, table)], log_n + 1, scaled=False)[:n]
    return point_fft(FFT, h, log_n)
