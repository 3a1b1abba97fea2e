"""Batch (slice-level) mirror of the reference's Engine / CurveProjective / CurveAffine / Wnaf API.

Names, argument meaning and error behaviour follow the reference; the only difference is that every
value is a *batch*: an (n, words) numpy uint64 array in the ABI layout.  `None` results of the
reference (`final_exponentiation` of zero) come back as an `is_some` mask.
"""
import numpy as np

from . import _native as nat

_default = None


def default_context():
    """The process-wide context on the current CUDA device (cuda:LOCAL_RANK under torchrun)."""
    global _default
    if _default is None:
        import os
        _default = nat.Context(int(os.environ.get("LOCAL_RANK", "0")))
    return _default


def _ctx(ctx):
    return ctx if ctx is not None else default_context()


# ---- window heuristics: pure host logic, bls12_381/ec.rs:895-921 (G1) and 1586-1612 (G2) ----------
_G1_NUM_SCALARS = [1, 3, 7, 20, 43, 120, 273, 563, 1630, 3128, 7933, 62569]
_G2_NUM_SCALARS = [1, 3, 8, 20, 47, 126, 260, 826, 1501, 4555, 84071]


def _num_bits(k):
    """FrRepr::num_bits (fr.rs:213-225) of (n,4) scalars."""
    k = np.ascontiguousarray(k, dtype=np.uint64).reshape(-1, 4)
    out = np.zeros(k.shape[0], dtype=np.int64)
    for limb in range(4):
        v = k[:, limb]
        nz = v != 0
        bl = np.zeros(k.shape[0], dtype=np.int64)
        vv = v.copy()
        for s in (32, 16, 8, 4, 2, 1):
            big = vv >= (np.uint64(1) << np.uint64(s))
            bl += np.where(big, s, 0)
            vv = np.where(big, vv >> np.uint64(s), vv)
        bl += np.where(nz, 1, 0)
        out = np.where(nz, 64 * limb + bl, out)
    return out


def _rec_num_scalars(table, n):
    ret = 4
    for r in table:
        if n > r:
            ret += 1
        else:
            break
    return ret


class _Curve:
    """Shared implementation of the CurveProjective batch methods; G1 and G2 specialise it."""
    _g2 = False
    _num_scalars_table = _G1_NUM_SCALARS
    _thresholds = (130, 34)

    # CurveProjective::double / add_assign / sub_assign / add_assign_mixed / negate  (ec.rs:296-532)
    @classmethod
    def double(cls, a, ctx=None): return cls._op("double", a, None, ctx)
    @classmethod
    def add_assign(cls, a, b, ctx=None): return cls._op("add", a, b, ctx)
    @classmethod
    def sub_assign(cls, a, b, ctx=None): return cls._op("sub", a, b, ctx)
    @classmethod
    def add_assign_mixed(cls, a, b_affine, ctx=None): return cls._op("add_mixed", a, b_affine, ctx)
    @classmethod
    def negate(cls, a, ctx=None): return cls._op("negate", a, None, ctx)

    @classmethod
    def _op(cls, op, a, b, ctx):
        c = _ctx(ctx)
        return (c.g2_op if cls._g2 else c.g1_op)(op, a, b)

    # CurveProjective::mul_assign: double-and-add (ec.rs:534-553)
    @classmethod
    def mul_assign(cls, a, scalars, ctx=None):
        c = _ctx(ctx)
        return (c.g2_mul if cls._g2 else c.g1_mul)(a, scalars)

    # CurveProjective::into_affine (ec.rs:586-619)
    @classmethod
    def into_affine(cls, a, ctx=None):
        c = _ctx(ctx)
        return (c.g2_into_affine if cls._g2 else c.g1_into_affine)(a)

    # CurveProjective::batch_normalization (ec.rs:246-294); returns the normalised copy
    @classmethod
    def batch_normalization(cls, v, ctx=None):
        c = _ctx(ctx)
        return (c.g2_batch_normalization if cls._g2 else c.g1_batch_normalization)(v)

    # sum_i k_i * bases_i over affine bases (the sum provers and batch verifiers build from add_assign_mixed, ec.rs:446-526):
    # one normalised Jacobian row, (x, y, one) or zero() = (0, one, 0).  Scalars are full 256-bit FrRepr integers.
    @classmethod
    def multiexp(cls, bases_affine, scalars, ctx=None):
        c = _ctx(ctx)
        return (c.g2_msm if cls._g2 else c.g1_msm)(bases_affine, scalars)

    # m independent multiexp sums in one call: scalars (m, n, 4); bases_affine (n, W) shared by every sum or (m, n, W), one
    # set per sum -> (m, 18|36), row j = multiexp(bases of sum j, scalars[j])
    @classmethod
    def multiexp_batch(cls, bases_affine, scalars, ctx=None):
        c = _ctx(ctx)
        return (c.g2_msm_batch if cls._g2 else c.g1_msm_batch)(bases_affine, scalars)

    # ec.rs:895-905 / 1586-1596
    @classmethod
    def recommended_wnaf_for_scalar(cls, scalars):
        nb = _num_bits(scalars)
        hi, lo = cls._thresholds
        return np.where(nb >= hi, 4, np.where(nb >= lo, 3, 2))

    # ec.rs:907-921 / 1598-1612
    @classmethod
    def recommended_wnaf_for_num_scalars(cls, num_scalars):
        return _rec_num_scalars(cls._num_scalars_table, int(num_scalars))


class G1(_Curve):
    _g2 = False
    _num_scalars_table = _G1_NUM_SCALARS
    _thresholds = (130, 34)


class G2(_Curve):
    _g2 = True
    _num_scalars_table = _G2_NUM_SCALARS
    _thresholds = (103, 37)


class G1Affine:
    """CurveAffine for G1: `prepare` is the identity wrap (G1Prepared, ec.rs:924-935)."""

    @staticmethod
    def prepare(p):
        return np.ascontiguousarray(p, dtype=np.uint64)

    @staticmethod
    def into_projective(p):
        """From<affine> for projective (ec.rs:570-582): (x, y, one) or zero() = (0, 1, 0)."""
        p = np.ascontiguousarray(p, dtype=np.uint64)
        out = np.zeros((p.shape[0], nat.W_G1), dtype=np.uint64)
        out[:, :12] = p[:, :12]
        out[:, 12:18] = _ONE
        inf = p[:, 12] != 0
        out[inf] = 0
        out[inf, 6:12] = _ONE
        return out

    @staticmethod
    def pairing_with(p, q, ctx=None):
        return Bls12.pairing(p, q, ctx)

    # CurveAffine::mul (ec.rs:174-177): mul_bits with mixed additions -> Jacobian rows
    @staticmethod
    def mul(p, scalars, ctx=None): return _ctx(ctx).affine_mul(False, p, scalars)

    # CurveAffine::into_compressed / into_uncompressed (lib.rs:226-233 -> EncodedPoint::from_affine)
    @staticmethod
    def into_compressed(p, ctx=None): return _ctx(ctx).encode(False, p, True)
    @staticmethod
    def into_uncompressed(p, ctx=None): return _ctx(ctx).encode(False, p, False)


class _Encoded:
    """EncodedPoint (lib.rs:236-263): `into_affine` checks curve + subgroup membership, `into_affine_unchecked`
    does not.  Batch-shaped: returns (affine rows, status) with status[i] = 0 for Ok, else the code of the
    reference's GroupDecodingError (include/pairing_b200.h, BLS_DEC_*)."""
    _g2, _compressed = False, False

    @classmethod
    def size(cls): return (96 if cls._g2 else 48) * (1 if cls._compressed else 2)
    @classmethod
    def into_affine(cls, data, ctx=None): return _ctx(ctx).decode(cls._g2, data, cls._compressed, True)
    @classmethod
    def into_affine_unchecked(cls, data, ctx=None): return _ctx(ctx).decode(cls._g2, data, cls._compressed, False)
    @classmethod
    def from_affine(cls, affine, ctx=None): return _ctx(ctx).encode(cls._g2, affine, cls._compressed)


class G1Uncompressed(_Encoded): _g2, _compressed = False, False
class G1Compressed(_Encoded): _g2, _compressed = False, True
class G2Uncompressed(_Encoded): _g2, _compressed = True, False
class G2Compressed(_Encoded): _g2, _compressed = True, True


class G2Affine:
    @staticmethod
    def prepare(q, ctx=None):
        """G2Affine::prepare -> G2Prepared::from_affine (mod.rs:168-358)."""
        return G2Prepared.from_affine(q, ctx)

    @staticmethod
    def into_projective(q):
        q = np.ascontiguousarray(q, dtype=np.uint64)
        out = np.zeros((q.shape[0], nat.W_G2), dtype=np.uint64)
        out[:, :24] = q[:, :24]
        out[:, 24:30] = _ONE
        inf = q[:, 24] != 0
        out[inf] = 0
        out[inf, 12:18] = _ONE
        return out

    @staticmethod
    def pairing_with(q, p, ctx=None):
        return Bls12.pairing(p, q, ctx)

    @staticmethod
    def mul(q, scalars, ctx=None): return _ctx(ctx).affine_mul(True, q, scalars)

    @staticmethod
    def into_compressed(q, ctx=None): return _ctx(ctx).encode(True, q, True)
    @staticmethod
    def into_uncompressed(q, ctx=None): return _ctx(ctx).encode(True, q, False)


# Montgomery one, R = 2^384 mod q (fq.rs:22-30)
_ONE = np.array([0x760900000002fffd, 0xebf4000bc40c0002, 0x5f48985753c758ba,
                 0x77ce585370525745, 0x5c071a97a256ec6d, 0x15f65ec3fa80e493], dtype=np.uint64)


class G2Prepared:
    """(n, 2449) arrays: 68 coefficient triples + infinity flag per point (ec.rs:1615-1619)."""

    @staticmethod
    def from_affine(q, ctx=None):
        return _ctx(ctx).g2_prepare(q)

    @staticmethod
    def is_zero(prepared):
        return np.ascontiguousarray(prepared, dtype=np.uint64)[:, -1] != 0


class Bls12:
    """Engine for BLS12-381 (bls12_381/mod.rs:30-160), batch-shaped."""

    @staticmethod
    def miller_loop(p_prepared, q_prepared, ctx=None):
        """ONE Miller loop over all n (G1Prepared, G2Prepared) pairs -- Engine::miller_loop(&[...])
        (mod.rs:40-102).  Returns a (1, 72) Fq12.  Pairs with an infinity member are skipped."""
        q = np.ascontiguousarray(q_prepared, dtype=np.uint64)
        c = _ctx(ctx)
        if q.ndim == 2 and q.shape[1] == nat.W_G2A:      # affine Q: coefficients are generated on the fly
            return c.multi_miller_loop(p_prepared, q)
        return c.multi_miller_loop_prepared(p_prepared, q)

    @staticmethod
    def miller_loop_batch(p, q, ctx=None):
        """n independent single-pair Miller loops -> (n, 72)."""
        q = np.ascontiguousarray(q, dtype=np.uint64)
        c = _ctx(ctx)
        if q.ndim == 2 and q.shape[1] == nat.W_G2A:
            return c.miller_loop(p, q)
        return c.miller_loop_prepared(p, q)

    @staticmethod
    def final_exponentiation(f, ctx=None):
        """Engine::final_exponentiation (mod.rs:104-160) -> (values, is_some)."""
        return _ctx(ctx).final_exponentiation(f)

    @staticmethod
    def pairing(p, q, ctx=None):
        """Engine::pairing (lib.rs:101-109) for n (G1Affine, G2Affine) pairs -> (n, 72)."""
        return _ctx(ctx).pairing(p, q)


class Wnaf:
    """The reference's typestate builder (wnaf.rs:75-179), batch-shaped.

    Wnaf().scalar(k).base(g)   per-(base, scalar) mode: window from each scalar's bit length
    Wnaf().base(g, n)          fixed-base mode: window from the number of scalars (4..16 for G1, 4..15 for
                               G2, ec.rs:907-921 / 1598-1612); ONE table is built on the device and shared
                               by every `.scalar(s)` (wnaf.rs:93-107, 169-178)
    """

    def __init__(self, curve=G1, ctx=None):
        self._curve = curve
        self._ctx = ctx
        self._scalars = None
        self._base = None
        self._window = 0

    def scalar(self, scalars):
        w = Wnaf(self._curve, self._ctx)
        w._scalars = np.ascontiguousarray(scalars, dtype=np.uint64)
        if self._base is not None:                      # `.base(g, n).scalar(s)`: exponentiate now, shared table
            c = _ctx(self._ctx)
            fn = c.g2_wnaf_fixed_base if self._curve._g2 else c.g1_wnaf_fixed_base
            return fn(self._base, self._window, w._scalars.reshape(-1, 4))
        return w

    def base(self, base, num_scalars=None):
        base = np.ascontiguousarray(base, dtype=np.uint64)
        if num_scalars is None:                         # `.scalar(s).base(g)`
            if self._scalars is None:
                raise ValueError("Wnaf.base(g) without num_scalars needs a preceding .scalar(s)")
            return self._run(base, self._scalars, 0)
        w = Wnaf(self._curve, self._ctx)
        if base.ndim == 1:
            base = base.reshape(1, -1)
        if base.ndim != 2 or base.shape[0] != 1:
            raise ValueError("Wnaf.base(g, n) takes one base point")
        w._base = base
        w._window = self._curve.recommended_wnaf_for_num_scalars(num_scalars)
        return w

    def shared(self):
        return self

    def _run(self, bases, scalars, window):
        c = _ctx(self._ctx)
        fn = c.g2_wnaf_mul if self._curve._g2 else c.g1_wnaf_mul
        return fn(bases, scalars, window)
