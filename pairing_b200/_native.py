"""ctypes binding of libpairing_b200.so (the C ABI of include/pairing_b200.h).

The product path has no CPU fallback: if the CUDA library is missing or no device is present every
entry point raises.  Nothing here imports or calls the oracle.
"""
import ctypes
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpairing_b200.so")

# u64 words per ABI struct
W_FQ, W_FQ2, W_FQ6, W_FQ12 = 6, 12, 36, 72
W_G1A, W_G1, W_G2A, W_G2, W_FR, W_G2P = 13, 18, 25, 36, 4, 68 * 3 * 12 + 1

OPS = dict(add=0, sub=1, mul=2, sqr=3, neg=4, dbl=5, inv=6, from_repr=7, into_repr=8, mul_nonres=9,
           frob1=10, frob2=11, frob3=12, conj=13, mul_by_014=14, mul_by_01=15, mul_by_1=16, sqrt=17,
           mul_by_line_pair=18, cyclotomic_sqr=19)
PT_OPS = dict(double=0, add=1, add_mixed=2, negate=3, sub=6)
FFT_KINDS = dict(fft=0, ifft=1, coset_fft=2, icoset_fft=3)

# every symbol include/pairing_b200.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "bls_ctx_create", "bls_ctx_destroy", "bls_strerror", "bls_ctx_last_error", "bls_ctx_device",
    "bls_ctx_sm_count", "bls_ctx_launch_count", "bls_ctx_set_latency_path_limits", "bls_ctx_trim",
    "bls_g2_prepare_batch", "bls_miller_loop_batch", "bls_miller_loop_prepared_batch",
    "bls_multi_miller_loop", "bls_multi_miller_loop_prepared", "bls_final_exponentiation_batch",
    "bls_pairing_batch", "bls_fq12_product",
    "bls_g1_wnaf_mul_batch", "bls_g2_wnaf_mul_batch", "bls_g1_wnaf_mul_window_batch",
    "bls_g2_wnaf_mul_window_batch", "bls_g1_mul_batch", "bls_g2_mul_batch",
    "bls_g1_batch_normalization", "bls_g2_batch_normalization", "bls_g1_into_affine_batch",
    "bls_g2_into_affine_batch", "bls_g1_op_batch", "bls_g2_op_batch", "bls_field_op_batch",
    "bls_g2_prepare_dev", "bls_miller_loop_dev", "bls_miller_loop_prepared_dev",
    "bls_final_exponentiation_dev", "bls_pairing_dev", "bls_multi_miller_scratch_bytes",
    "bls_multi_miller_loop_dev", "bls_fq12_product_scratch_bytes", "bls_fq12_product_dev",
    "bls_g1_wnaf_mul_dev", "bls_g2_wnaf_mul_dev", "bls_batch_normalization_scratch_bytes",
    "bls_g1_batch_normalization_dev", "bls_g2_batch_normalization_dev", "bls_imad_peak",
    "bls_g1_wnaf_fixed_base_batch", "bls_g2_wnaf_fixed_base_batch", "bls_g1_wnaf_table", "bls_g2_wnaf_table",
    "bls_fq12_pow_batch", "bls_fq12_pow_dev", "bls_fr_op_batch",
    "bls_miller_loop_shared_q_batch", "bls_pairing_shared_q_batch", "bls_miller_loop_shared_q_dev",
    "bls_g1_affine_mul_batch", "bls_g2_affine_mul_batch",
    "bls_g1_point_from_x_batch", "bls_g2_point_from_x_batch", "bls_g1_scale_by_cofactor_batch", "bls_g2_scale_by_cofactor_batch",
    "bls_g1_decode_batch", "bls_g2_decode_batch", "bls_g1_encode_batch", "bls_g2_encode_batch",
    "bls_g1_wnaf_table_dev", "bls_g2_wnaf_table_dev", "bls_g1_wnaf_fixed_base_dev", "bls_g2_wnaf_fixed_base_dev",
    "bls_pairing_product", "bls_pairing_product_dev", "bls_fq12_product_tail_dev",
    "bls_pair_field_op_batch", "bls_pair_field_op_dev", "bls_pairing_projective_batch", "bls_pairing_projective_dev",
    "bls_mgpu_create", "bls_mgpu_destroy", "bls_mgpu_device_count", "bls_mgpu_ctx", "bls_mgpu_multi_miller_loop",
    "bls_mgpu_pairing_product", "bls_mgpu_pairing_batch", "bls_mgpu_g1_wnaf_mul_batch", "bls_mgpu_g2_wnaf_mul_batch",
    "bls_mgpu_last_phase_ms",
    "bls_g1_msm", "bls_g2_msm", "bls_msm_scratch_bytes", "bls_g1_msm_dev", "bls_g2_msm_dev",
    "bls_g1_msm_batch", "bls_g2_msm_batch", "bls_msm_batch_scratch_bytes", "bls_g1_msm_batch_dev", "bls_g2_msm_batch_dev",
    "bls_fr_fft_batch", "bls_fr_fft_scratch_bytes", "bls_fr_fft_dev",
    "bls_fr_groth16_h_batch", "bls_fr_groth16_h_scratch_bytes", "bls_fr_groth16_h_dev", "bls_fr_op_dev",
    "bls_groth16_prove_batch", "bls_groth16_prove_scratch_bytes", "bls_groth16_prove_dev",
    "bls_groth16_prepare_verifying_key", "bls_groth16_verify_batch", "bls_groth16_verify_scratch_bytes", "bls_groth16_verify_dev",
    "bls_groth16_verify_rlc_batch", "bls_groth16_verify_rlc_scratch_bytes", "bls_groth16_verify_rlc_dev",
    "bls_groth16_generate_parameters_batch", "bls_groth16_generate_parameters_scratch_bytes", "bls_groth16_generate_parameters_dev",
    "bls_kzg_commit_batch", "bls_kzg_commit_scratch_bytes", "bls_kzg_commit_dev", "bls_kzg_open_batch", "bls_kzg_open_scratch_bytes",
    "bls_kzg_open_dev", "bls_kzg_prepare_verifying_key", "bls_kzg_verify_batch", "bls_kzg_verify_scratch_bytes", "bls_kzg_verify_dev",
    "bls_kzg_verify_rlc_batch", "bls_kzg_verify_rlc_scratch_bytes", "bls_kzg_verify_rlc_dev",
]


class BlsError(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BlsError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "or `make -C pairing_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.bls_ctx_create.restype = vp
    lib.bls_ctx_create.argtypes = [ci, ctypes.POINTER(ci)]
    lib.bls_ctx_destroy.argtypes = [vp]
    lib.bls_ctx_destroy.restype = None
    lib.bls_strerror.restype = ctypes.c_char_p
    lib.bls_strerror.argtypes = [ci]
    lib.bls_ctx_last_error.restype = ctypes.c_char_p
    lib.bls_ctx_last_error.argtypes = [vp]
    lib.bls_ctx_device.argtypes = [vp]
    lib.bls_ctx_sm_count.argtypes = [vp]
    lib.bls_ctx_launch_count.restype = ctypes.c_uint64
    lib.bls_ctx_launch_count.argtypes = [vp]
    lib.bls_ctx_set_latency_path_limits.argtypes = [vp, sz, sz]
    lib.bls_ctx_trim.argtypes = [vp, sz]
    for name in ("bls_multi_miller_scratch_bytes", "bls_fq12_product_scratch_bytes"):
        getattr(lib, name).restype = sz
        getattr(lib, name).argtypes = [vp, sz]
    lib.bls_batch_normalization_scratch_bytes.restype = sz
    lib.bls_batch_normalization_scratch_bytes.argtypes = [vp, ci, sz]
    lib.bls_msm_scratch_bytes.restype = sz
    lib.bls_msm_scratch_bytes.argtypes = [vp, ci, sz, ci]
    lib.bls_msm_batch_scratch_bytes.restype = sz
    lib.bls_msm_batch_scratch_bytes.argtypes = [vp, ci, sz, sz, ci]
    lib.bls_fr_fft_scratch_bytes.restype = sz
    lib.bls_fr_fft_scratch_bytes.argtypes = [vp, ci, sz]
    lib.bls_fr_groth16_h_scratch_bytes.restype = sz
    lib.bls_fr_groth16_h_scratch_bytes.argtypes = [vp, sz, sz]
    lib.bls_groth16_prove_scratch_bytes.restype = sz
    lib.bls_groth16_prove_scratch_bytes.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, sz]
    for name in ("bls_groth16_verify_scratch_bytes", "bls_groth16_verify_rlc_scratch_bytes"):
        getattr(lib, name).restype = sz
        getattr(lib, name).argtypes = [vp, sz, sz]
    lib.bls_groth16_generate_parameters_scratch_bytes.restype = sz
    lib.bls_groth16_generate_parameters_scratch_bytes.argtypes = [vp, vp, sz, sz, sz]
    for name, args in (("bls_kzg_commit_scratch_bytes", [vp, sz, sz]), ("bls_kzg_open_scratch_bytes", [vp, sz, sz]),
                       ("bls_kzg_verify_scratch_bytes", [vp, sz]), ("bls_kzg_verify_rlc_scratch_bytes", [vp, sz])):
        getattr(lib, name).restype = sz
        getattr(lib, name).argtypes = args
    sig = {
        "bls_g2_prepare_batch": [vp, vp, vp, sz],
        "bls_miller_loop_batch": [vp, vp, vp, vp, sz],
        "bls_miller_loop_prepared_batch": [vp, vp, vp, vp, sz],
        "bls_multi_miller_loop": [vp, vp, vp, sz, vp],
        "bls_multi_miller_loop_prepared": [vp, vp, vp, sz, vp],
        "bls_final_exponentiation_batch": [vp, vp, vp, vp, sz],
        "bls_pairing_batch": [vp, vp, vp, vp, sz],
        "bls_fq12_product": [vp, vp, sz, vp],
        "bls_g1_wnaf_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g2_wnaf_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g1_wnaf_mul_window_batch": [vp, vp, vp, vp, sz, ci],
        "bls_g2_wnaf_mul_window_batch": [vp, vp, vp, vp, sz, ci],
        "bls_g1_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g2_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g1_batch_normalization": [vp, vp, sz],
        "bls_g2_batch_normalization": [vp, vp, sz],
        "bls_g1_into_affine_batch": [vp, vp, vp, sz],
        "bls_g2_into_affine_batch": [vp, vp, vp, sz],
        "bls_g1_op_batch": [vp, ci, vp, vp, vp, sz],
        "bls_g2_op_batch": [vp, ci, vp, vp, vp, sz],
        "bls_field_op_batch": [vp, ci, ci, vp, vp, vp, vp, sz],
        "bls_g1_wnaf_fixed_base_batch": [vp, vp, ci, vp, vp, sz],
        "bls_g2_wnaf_fixed_base_batch": [vp, vp, ci, vp, vp, sz],
        "bls_g1_wnaf_table": [vp, vp, ci, vp],
        "bls_g2_wnaf_table": [vp, vp, ci, vp],
        "bls_g1_wnaf_table_dev": [vp, vp, ci, vp, vp],
        "bls_g2_wnaf_table_dev": [vp, vp, ci, vp, vp],
        "bls_g1_wnaf_fixed_base_dev": [vp, vp, ci, vp, vp, sz, vp],
        "bls_g2_wnaf_fixed_base_dev": [vp, vp, ci, vp, vp, sz, vp],
        "bls_g1_decode_batch": [vp, vp, ci, ci, vp, vp, sz],
        "bls_g2_decode_batch": [vp, vp, ci, ci, vp, vp, sz],
        "bls_g1_encode_batch": [vp, vp, ci, vp, sz],
        "bls_g2_encode_batch": [vp, vp, ci, vp, sz],
        "bls_fr_op_batch": [vp, ci, vp, vp, vp, vp, sz],
        "bls_miller_loop_shared_q_batch": [vp, vp, vp, vp, sz],
        "bls_pairing_shared_q_batch": [vp, vp, vp, vp, sz],
        "bls_miller_loop_shared_q_dev": [vp, vp, vp, vp, sz, ci, vp],
        "bls_g1_affine_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g2_affine_mul_batch": [vp, vp, vp, vp, sz],
        "bls_g1_point_from_x_batch": [vp, vp, vp, vp, vp, sz],
        "bls_g2_point_from_x_batch": [vp, vp, vp, vp, vp, sz],
        "bls_g1_scale_by_cofactor_batch": [vp, vp, vp, sz],
        "bls_g2_scale_by_cofactor_batch": [vp, vp, vp, sz],
        "bls_fq12_pow_batch": [vp, vp, vp, vp, sz],
        "bls_fq12_pow_dev": [vp, vp, vp, vp, sz, vp],
        "bls_g2_prepare_dev": [vp, vp, vp, sz, vp],
        "bls_miller_loop_dev": [vp, vp, vp, vp, sz, vp],
        "bls_miller_loop_prepared_dev": [vp, vp, vp, vp, sz, vp],
        "bls_final_exponentiation_dev": [vp, vp, vp, vp, sz, vp],
        "bls_pairing_dev": [vp, vp, vp, vp, sz, vp],
        "bls_multi_miller_loop_dev": [vp, vp, vp, sz, vp, vp, vp],
        "bls_fq12_product_dev": [vp, vp, sz, vp, vp, vp],
        "bls_g1_wnaf_mul_dev": [vp, vp, vp, vp, sz, ci, vp],
        "bls_g2_wnaf_mul_dev": [vp, vp, vp, vp, sz, ci, vp],
        "bls_g1_batch_normalization_dev": [vp, vp, sz, vp, vp],
        "bls_g2_batch_normalization_dev": [vp, vp, sz, vp, vp],
        "bls_imad_peak": [vp, ci, ci, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)],
        "bls_pairing_product": [vp, vp, vp, sz, vp, vp],
        "bls_pair_field_op_batch": [vp, ci, ci, vp, vp, vp, vp, sz],
        "bls_pairing_projective_batch": [vp, vp, vp, vp, sz],
        "bls_pairing_projective_dev": [vp, vp, vp, vp, sz, vp],
        "bls_pair_field_op_dev": [vp, ci, ci, vp, vp, vp, vp, sz, vp],
        "bls_pairing_product_dev": [vp, vp, vp, sz, vp, vp, vp, vp],
        "bls_fq12_product_tail_dev": [vp, vp, sz, vp, ci, vp, vp],
        "bls_mgpu_multi_miller_loop": [vp, vp, vp, sz, vp],
        "bls_mgpu_pairing_product": [vp, vp, vp, sz, vp, vp],
        "bls_mgpu_pairing_batch": [vp, vp, vp, vp, sz],
        "bls_mgpu_g1_wnaf_mul_batch": [vp, vp, vp, vp, sz],
        "bls_mgpu_g2_wnaf_mul_batch": [vp, vp, vp, vp, sz],
        "bls_mgpu_last_phase_ms": [vp, ctypes.POINTER(ctypes.c_double)],
        "bls_g1_msm": [vp, vp, vp, sz, vp],
        "bls_g2_msm": [vp, vp, vp, sz, vp],
        "bls_g1_msm_dev": [vp, vp, vp, sz, ci, vp, vp, vp],
        "bls_g2_msm_dev": [vp, vp, vp, sz, ci, vp, vp, vp],
        "bls_g1_msm_batch": [vp, vp, ci, vp, sz, sz, vp],
        "bls_g2_msm_batch": [vp, vp, ci, vp, sz, sz, vp],
        "bls_g1_msm_batch_dev": [vp, vp, ci, vp, sz, sz, ci, vp, vp, vp],
        "bls_g2_msm_batch_dev": [vp, vp, ci, vp, sz, sz, ci, vp, vp, vp],
        "bls_fr_fft_batch": [vp, ci, vp, vp, ci, sz],
        "bls_fr_fft_dev": [vp, ci, vp, vp, ci, sz, vp, vp],
        "bls_fr_groth16_h_batch": [vp, vp, vp, vp, sz, sz, vp],
        "bls_fr_groth16_h_dev": [vp, vp, vp, vp, sz, sz, vp, vp, vp],
        "bls_fr_op_dev": [vp, ci, vp, vp, vp, vp, sz, vp],
        "bls_groth16_prove_batch": [vp, vp, vp, vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, vp, sz, vp],
        "bls_groth16_prove_dev": [vp, vp, vp, vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, vp, sz, vp, vp, vp],
        "bls_groth16_prepare_verifying_key": [vp, vp, vp, vp, vp, vp],
        "bls_groth16_verify_batch": [vp, vp, vp, sz, vp, vp, sz, vp],
        "bls_groth16_verify_dev": [vp, vp, vp, sz, vp, vp, sz, vp, vp, vp],
        "bls_groth16_verify_rlc_batch": [vp, vp, vp, sz, vp, vp, vp, sz, vp],
        "bls_groth16_verify_rlc_dev": [vp, vp, vp, sz, vp, vp, vp, sz, vp, vp, vp],
        "bls_groth16_generate_parameters_batch": [vp, vp, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp],
        "bls_groth16_generate_parameters_dev": [vp, vp, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
        "bls_kzg_commit_batch": [vp, vp, sz, vp, sz, sz, vp],
        "bls_kzg_commit_dev": [vp, vp, sz, vp, sz, sz, vp, vp, vp],
        "bls_kzg_open_batch": [vp, vp, sz, vp, sz, vp, sz, vp, vp],
        "bls_kzg_open_dev": [vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp],
        "bls_kzg_prepare_verifying_key": [vp, vp, vp, vp, vp],
        "bls_kzg_verify_batch": [vp, vp, vp, vp, vp, vp, sz, vp],
        "bls_kzg_verify_dev": [vp, vp, vp, vp, vp, vp, sz, vp, vp, vp],
        "bls_kzg_verify_rlc_batch": [vp, vp, vp, vp, vp, vp, vp, sz, vp],
        "bls_kzg_verify_rlc_dev": [vp, vp, vp, vp, vp, vp, vp, sz, vp, vp, vp],
    }
    lib.bls_mgpu_create.restype = vp
    lib.bls_mgpu_create.argtypes = [ctypes.POINTER(ci), ci, ctypes.POINTER(ci)]
    lib.bls_mgpu_destroy.restype = None
    lib.bls_mgpu_destroy.argtypes = [vp]
    lib.bls_mgpu_device_count.argtypes = [vp]
    lib.bls_mgpu_ctx.restype = vp
    lib.bls_mgpu_ctx.argtypes = [vp, ci]
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = ci
    _lib = lib
    return lib


def _arr(a, w, name="array"):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    if a.ndim != 2 or a.shape[1] != w:
        raise ValueError("%s must have shape (n, %d) uint64, got %r" % (name, w, a.shape))
    return a


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


W_PROOF = 2 * W_G1A + W_G2A        # bls_groth16_proof: A (G1Affine), B (G2Affine), C (G1Affine)


@dataclass
class Groth16Params:
    """The part of bellman's groth16::Parameters that create_proof reads: the vk points alpha_g1, beta_g1, delta_g1 ((13,)
    G1Affine rows), beta_g2, delta_g2 ((25,) G2Affine rows) and the queries h, l, a, b_g1 ((n, 13)) and b_g2 ((n, 25)).  numpy
    uint64 arrays for Context.groth16_prove; for DeviceEngine.groth16_prove the queries are CUDA int64 tensors."""
    alpha_g1: object
    beta_g1: object
    delta_g1: object
    beta_g2: object
    delta_g2: object
    h: object
    l: object
    a: object
    b_g1: object
    b_g2: object


class _Groth16ParamsC(ctypes.Structure):
    _fields_ = [("alpha_g1", ctypes.c_uint64 * W_G1A), ("beta_g1", ctypes.c_uint64 * W_G1A), ("delta_g1", ctypes.c_uint64 * W_G1A),
                ("beta_g2", ctypes.c_uint64 * W_G2A), ("delta_g2", ctypes.c_uint64 * W_G2A),
                ("h", ctypes.c_void_p), ("l", ctypes.c_void_p), ("a", ctypes.c_void_p), ("b_g1", ctypes.c_void_p),
                ("b_g2", ctypes.c_void_p), ("h_len", ctypes.c_size_t), ("l_len", ctypes.c_size_t), ("a_len", ctypes.c_size_t),
                ("b_len", ctypes.c_size_t)]


def groth16_params_c(params, ptr, length):
    """the bls_groth16_params struct: vk rows by value, ptr(query) and length(query) for the five queries"""
    c = _Groth16ParamsC()
    for name, w in (("alpha_g1", W_G1A), ("beta_g1", W_G1A), ("delta_g1", W_G1A), ("beta_g2", W_G2A), ("delta_g2", W_G2A)):
        row = np.ascontiguousarray(getattr(params, name), dtype=np.uint64).reshape(-1)
        if row.shape != (w,):
            raise ValueError("%s must be one row of %d uint64, got %r" % (name, w, row.shape))
        getattr(c, name)[:] = [int(x) for x in row]
    for name in ("h", "l", "a", "b_g1", "b_g2"):
        setattr(c, name, ptr(getattr(params, name)))
    if length(params.b_g1) != length(params.b_g2):
        raise ValueError("b_g1 and b_g2 must have the same length")
    c.h_len, c.l_len, c.a_len, c.b_len = (length(getattr(params, q)) for q in ("h", "l", "a", "b_g1"))
    return c


class Groth16PvkC(ctypes.Structure):
    """bls_groth16_pvk: bellman's PreparedVerifyingKey without ic, plus -gamma_g2 and -delta_g2 in affine form.  The pads put
    both prepared points at 16-byte aligned offsets."""
    _fields_ = [("neg_gamma_g2", ctypes.c_uint64 * W_G2P), ("pad0", ctypes.c_uint64),
                ("neg_delta_g2", ctypes.c_uint64 * W_G2P), ("pad1", ctypes.c_uint64),
                ("alpha_g1_beta_g2", ctypes.c_uint64 * W_FQ12),
                ("neg_gamma_g2_affine", ctypes.c_uint64 * W_G2A), ("neg_delta_g2_affine", ctypes.c_uint64 * W_G2A)]


W_PVK = ctypes.sizeof(Groth16PvkC) // 8     # 5022 words


class KzgPvkC(ctypes.Structure):
    """bls_kzg_pvk: prepare(h) and prepare(-tau h), the pads putting both at 16-byte aligned offsets, then g, h and -tau h in
    affine form."""
    _fields_ = [("h_prepared", ctypes.c_uint64 * W_G2P), ("pad0", ctypes.c_uint64),
                ("neg_tau_h_prepared", ctypes.c_uint64 * W_G2P), ("pad1", ctypes.c_uint64),
                ("g", ctypes.c_uint64 * W_G1A), ("h", ctypes.c_uint64 * W_G2A), ("neg_tau_h", ctypes.c_uint64 * W_G2A)]


W_KZG_PVK = ctypes.sizeof(KzgPvkC) // 8     # 4963 words


def kzg_poly_shape(shape, srs_rows, open_):
    """(m, n) of an (m, n, 4) coefficient array, checked against an SRS of srs_rows rows (n rows for commit, n - 1 for open)"""
    if len(shape) != 3 or shape[2] != W_FR:
        raise ValueError("p must have shape (m, n, 4), got %r" % (tuple(shape),))
    m, n = int(shape[0]), int(shape[1])
    if srs_rows < (max(n - 1, 0) if open_ else n):
        raise ValueError("the SRS has %d points, a polynomial of %d coefficients needs %d" % (srs_rows, n, max(n - 1, 0) if open_ else n))
    return m, n


class R1csMatrixC(ctypes.Structure):
    """bls_r1cs_matrix: one of A, B, C variable-major (offsets of num_inputs + num_aux + 1 entries, then the terms)"""
    _fields_ = [("offsets", ctypes.c_void_p), ("constraint", ctypes.c_void_p), ("coeff", ctypes.c_void_p), ("nnz", ctypes.c_size_t)]


class Groth16VkPointsC(ctypes.Structure):
    """bls_groth16_vk_points"""
    _fields_ = [("alpha_g1", ctypes.c_uint64 * W_G1A), ("beta_g1", ctypes.c_uint64 * W_G1A), ("delta_g1", ctypes.c_uint64 * W_G1A),
                ("beta_g2", ctypes.c_uint64 * W_G2A), ("gamma_g2", ctypes.c_uint64 * W_G2A), ("delta_g2", ctypes.c_uint64 * W_G2A)]


W_VK_POINTS = ctypes.sizeof(Groth16VkPointsC) // 8      # 114 words
VK_POINT_ROWS = (("alpha_g1", 0, W_G1A), ("beta_g1", W_G1A, W_G1A), ("delta_g1", 2 * W_G1A, W_G1A),
                 ("beta_g2", 3 * W_G1A, W_G2A), ("gamma_g2", 3 * W_G1A + W_G2A, W_G2A), ("delta_g2", 3 * W_G1A + 2 * W_G2A, W_G2A))


class Groth16ParametersOutC(ctypes.Structure):
    """bls_groth16_parameters_out"""
    _fields_ = [(name, ctypes.c_void_p) for name in ("vk", "ic", "h", "l", "a", "b_g1", "b_g2", "a_aux_density", "b_input_density",
                                                      "b_aux_density", "lens", "ok")]


@dataclass
class Groth16Parameters(Groth16Params):
    """bellman's groth16::Parameters as generate_parameters makes them: Groth16Params (its queries trimmed to a_len and
    b_len, so it goes to groth16_prove unchanged) plus gamma_g2 ((25,) G2Affine row), ic ((num_inputs, 13)), the density
    bitmaps (a_aux_density, b_input_density, b_aux_density) as bool arrays and ok (False: bellman's UnconstrainedVariable)."""
    gamma_g2: object = None
    ic: object = None
    densities: object = None
    ok: bool = True


def r1cs_matrices(abc, num_constraints, nv):
    """abc = three (offsets, constraint, coeff) triples -> contiguous numpy arrays (uint64 (nv + 1,), uint32 (nnz,), uint64
    (nnz, 4)) and the bls_r1cs_matrix[3] array pointing at them"""
    if len(abc) != 3:
        raise ValueError("abc must hold the three matrices A, B and C")
    keep, mats = [], (R1csMatrixC * 3)()
    for i, (off, cons, coeff) in enumerate(abc):
        off = np.ascontiguousarray(off, dtype=np.uint64)
        cons = np.ascontiguousarray(cons, dtype=np.uint32)
        coeff = np.ascontiguousarray(coeff, dtype=np.uint64).reshape(-1, W_FR)
        if off.shape != (nv + 1,) or cons.shape != (coeff.shape[0],):
            raise ValueError("matrix %d: offsets must have %d entries and constraint one per coefficient row, got %r, %r, %r"
                             % (i, nv + 1, off.shape, cons.shape, coeff.shape))
        keep.append((off, cons, coeff))
        mats[i] = R1csMatrixC(_p(off), _p(cons), _p(coeff), cons.shape[0])
    return keep, mats


def unpack_density(words, bits):
    """the inverse of density_words: BitVec<u32> words -> a bool array of `bits` entries"""
    b = np.unpackbits(np.ascontiguousarray(words, dtype="<u4").view(np.uint8), bitorder="little")
    return b[:bits].astype(bool)


def groth16_parameters(vk, ic, h, l, a, b_g1, b_g2, dens, lens, ok, ni, na):
    """Groth16Parameters from the outputs of bls_groth16_generate_parameters_*: vk the 114 words of bls_groth16_vk_points,
    the queries untrimmed, dens the three word arrays (numpy), lens (a_len, b_len)"""
    rows = {name: vk[o:o + w] for name, o, w in VK_POINT_ROWS}
    a_len, b_len = int(lens[0]), int(lens[1])
    densities = (unpack_density(dens[0], na), unpack_density(dens[1], ni), unpack_density(dens[2], na))
    return Groth16Parameters(rows["alpha_g1"], rows["beta_g1"], rows["delta_g1"], rows["beta_g2"], rows["delta_g2"], h, l, a[:a_len],
                             b_g1[:b_len], b_g2[:b_len], gamma_g2=rows["gamma_g2"], ic=ic, densities=densities, ok=bool(ok))


def density_words(d, bits, name):
    """a numpy bool array of `bits` entries -> the uint32 words of bit-vec's BitVec<u32> (bit i at word i / 32, bit i % 32)"""
    d = np.ascontiguousarray(d, dtype=bool)
    if d.shape != (bits,):
        raise ValueError("%s must be a bool array of %d entries, got %r" % (name, bits, d.shape))
    b = np.packbits(d, bitorder="little")
    b = np.concatenate([b, np.zeros(-len(b) % 4, dtype=np.uint8)])
    return np.ascontiguousarray(b.view("<u4"))


class Context:
    """One CUDA device + stream (bls_ctx).  Host-array methods take and return numpy uint64 arrays
    in the ABI layouts; `*_dev` methods take raw device pointers (ints) and a CUDA stream handle."""

    def __init__(self, device=0):
        self._lib = load()
        err = ctypes.c_int(0)
        self._ctx = self._lib.bls_ctx_create(int(device), ctypes.byref(err))
        if not self._ctx:
            raise BlsError("bls_ctx_create(device=%d) failed: %s" % (device, self._lib.bls_strerror(err.value).decode()))
        self.device = int(device)

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.bls_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise BlsError("%s [%s]" % (self._lib.bls_strerror(rc).decode(),
                                        self._lib.bls_ctx_last_error(self._ctx).decode()))

    @property
    def sm_count(self):
        return self._lib.bls_ctx_sm_count(self._ctx)

    @property
    def launch_count(self):
        return int(self._lib.bls_ctx_launch_count(self._ctx))

    def trim(self, keep_bytes=0):
        """release the staging memory the context caches between host-buffer calls"""
        self._check(self._lib.bls_ctx_trim(self._ctx, int(keep_bytes)))

    def set_latency_path_limits(self, max_pairings, max_final_exps):
        """Batch sizes up to which pairing / final_exponentiation run one WARP per element (0: lane-pair kernels always)."""
        self._check(self._lib.bls_ctx_set_latency_path_limits(self._ctx, int(max_pairings), int(max_final_exps)))

    # ------------------------------------------------------------------ engine, host arrays
    def g2_prepare(self, q):
        q = _arr(q, W_G2A, "q")
        out = np.zeros((q.shape[0], W_G2P), dtype=np.uint64)
        self._check(self._lib.bls_g2_prepare_batch(self._ctx, _p(q), _p(out), q.shape[0]))
        return out

    def _pq(self, fn, p, q, wq):
        p, q = _arr(p, W_G1A, "p"), _arr(q, wq, "q")
        if p.shape[0] != q.shape[0]:
            raise ValueError("p and q must have the same length")
        out = np.zeros((p.shape[0], W_FQ12), dtype=np.uint64)
        self._check(fn(self._ctx, _p(p), _p(q), _p(out), p.shape[0]))
        return out

    def miller_loop(self, p, q):
        return self._pq(self._lib.bls_miller_loop_batch, p, q, W_G2A)

    def miller_loop_prepared(self, p, qp):
        return self._pq(self._lib.bls_miller_loop_prepared_batch, p, qp, W_G2P)

    def pairing(self, p, q):
        return self._pq(self._lib.bls_pairing_batch, p, q, W_G2A)

    def pairing_projective(self, p, q):
        """Engine::pairing on Jacobian inputs (the two into_affine conversions fused in front): (n,18),(n,36) -> (n,72)."""
        p, q = _arr(p, W_G1, "p"), _arr(q, W_G2, "q")
        if p.shape[0] != q.shape[0]:
            raise ValueError("p and q must have the same length")
        out = np.zeros((p.shape[0], W_FQ12), dtype=np.uint64)
        self._check(self._lib.bls_pairing_projective_batch(self._ctx, _p(p), _p(q), _p(out), p.shape[0]))
        return out

    def _shared_q(self, fn, p, q1):
        p, q1 = _arr(p, W_G1A, "p"), _arr(q1, W_G2P, "q1")
        if q1.shape[0] != 1:
            raise ValueError("q1 must be ONE prepared G2 point")
        out = np.zeros((p.shape[0], W_FQ12), dtype=np.uint64)
        self._check(fn(self._ctx, _p(p), _p(q1), _p(out), p.shape[0]))
        return out

    def miller_loop_shared_q(self, p, q1):
        """n Miller loops e(P_i, Q) against one prepared Q."""
        return self._shared_q(self._lib.bls_miller_loop_shared_q_batch, p, q1)

    def pairing_shared_q(self, p, q1):
        return self._shared_q(self._lib.bls_pairing_shared_q_batch, p, q1)

    def _multi(self, fn, p, q, wq):
        p, q = _arr(p, W_G1A, "p"), _arr(q, wq, "q")
        if p.shape[0] != q.shape[0]:
            raise ValueError("p and q must have the same length")
        out = np.zeros((1, W_FQ12), dtype=np.uint64)
        self._check(fn(self._ctx, _p(p), _p(q), p.shape[0], _p(out)))
        return out

    def multi_miller_loop(self, p, q):
        return self._multi(self._lib.bls_multi_miller_loop, p, q, W_G2A)

    def multi_miller_loop_prepared(self, p, qp):
        return self._multi(self._lib.bls_multi_miller_loop_prepared, p, qp, W_G2P)

    def pairing_product(self, p, q):
        """final_exponentiation(miller_loop(all pairs)) in one call -> ((1, 72) GT element, is_some)."""
        p, q = _arr(p, W_G1A, "p"), _arr(q, W_G2A, "q")
        if p.shape[0] != q.shape[0]:
            raise ValueError("p and q must have the same length")
        out = np.zeros((1, W_FQ12), dtype=np.uint64)
        ok = np.zeros(1, dtype=np.uint8)
        self._check(self._lib.bls_pairing_product(self._ctx, _p(p), _p(q), p.shape[0], _p(out), _p(ok)))
        return out, bool(ok[0])

    def final_exponentiation(self, f):
        f = _arr(f, W_FQ12, "f")
        out = np.zeros_like(f)
        ok = np.zeros(f.shape[0], dtype=np.uint8)
        self._check(self._lib.bls_final_exponentiation_batch(self._ctx, _p(f), _p(out), _p(ok), f.shape[0]))
        return out, ok

    def fq12_pow(self, a, k):
        """Fq12::pow(FrRepr) per element (lib.rs:306-324)."""
        a, k = _arr(a, W_FQ12, "a"), _arr(k, W_FR, "k")
        if a.shape[0] != k.shape[0]:
            raise ValueError("a and k must have the same length")
        out = np.zeros_like(a)
        self._check(self._lib.bls_fq12_pow_batch(self._ctx, _p(a), _p(k), _p(out), a.shape[0]))
        return out

    def fq12_product(self, f):
        f = _arr(f, W_FQ12, "f")
        out = np.zeros((1, W_FQ12), dtype=np.uint64)
        self._check(self._lib.bls_fq12_product(self._ctx, _p(f), f.shape[0], _p(out)))
        return out

    # ------------------------------------------------------------------ curves, host arrays
    def _wnaf(self, g2, bases, k, window, mode):
        w = W_G2 if g2 else W_G1
        bases, k = _arr(bases, w, "bases"), _arr(k, W_FR, "k")
        if bases.shape[0] != k.shape[0]:
            raise ValueError("bases and k must have the same length")
        out = np.zeros_like(bases)
        n = bases.shape[0]
        L = self._lib
        if mode == "mul":
            fn = L.bls_g2_mul_batch if g2 else L.bls_g1_mul_batch
            self._check(fn(self._ctx, _p(bases), _p(k), _p(out), n))
        elif window:
            fn = L.bls_g2_wnaf_mul_window_batch if g2 else L.bls_g1_wnaf_mul_window_batch
            self._check(fn(self._ctx, _p(bases), _p(k), _p(out), n, int(window)))
        else:
            fn = L.bls_g2_wnaf_mul_batch if g2 else L.bls_g1_wnaf_mul_batch
            self._check(fn(self._ctx, _p(bases), _p(k), _p(out), n))
        return out

    def decode(self, g2, data, compressed, checked=True):
        """EncodedPoint::into_affine(_unchecked) for n encodings back to back -> (affine rows, status bytes)."""
        size = (96 if g2 else 48) * (1 if compressed else 2)
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        if buf.size % size:
            raise ValueError("encoded data is not a multiple of %d bytes" % size)
        n = buf.size // size
        out = np.zeros((n, W_G2A if g2 else W_G1A), dtype=np.uint64)
        status = np.zeros(n, dtype=np.uint8)
        buf = np.ascontiguousarray(buf)
        fn = self._lib.bls_g2_decode_batch if g2 else self._lib.bls_g1_decode_batch
        self._check(fn(self._ctx, _p(buf), int(bool(compressed)), int(bool(checked)), _p(out), _p(status), n))
        return out, status

    def encode(self, g2, affine, compressed):
        """EncodedPoint::from_affine for n affine points -> bytes."""
        affine = _arr(affine, W_G2A if g2 else W_G1A, "affine")
        size = (96 if g2 else 48) * (1 if compressed else 2)
        out = np.zeros(affine.shape[0] * size, dtype=np.uint8)
        fn = self._lib.bls_g2_encode_batch if g2 else self._lib.bls_g1_encode_batch
        self._check(fn(self._ctx, _p(affine), int(bool(compressed)), _p(out), affine.shape[0]))
        return out.tobytes()

    def _wnaf_fixed(self, g2, base, window, k):
        """Wnaf::base(g, n).scalar(k_i): one shared table (window 2..16), every scalar against it."""
        w = W_G2 if g2 else W_G1
        base, k = _arr(base, w, "base"), _arr(k, W_FR, "k")
        if base.shape[0] != 1:
            raise ValueError("fixed-base mode takes exactly one base point")
        out = np.zeros((k.shape[0], w), dtype=np.uint64)
        fn = self._lib.bls_g2_wnaf_fixed_base_batch if g2 else self._lib.bls_g1_wnaf_fixed_base_batch
        self._check(fn(self._ctx, _p(base), int(window), _p(k), _p(out), k.shape[0]))
        return out

    def g1_wnaf_fixed_base(self, base, window, k): return self._wnaf_fixed(False, base, window, k)
    def g2_wnaf_fixed_base(self, base, window, k): return self._wnaf_fixed(True, base, window, k)

    def _wnaf_table(self, g2, base, window):
        w = W_G2 if g2 else W_G1
        base = _arr(base, w, "base")
        if not 2 <= int(window) <= 16:
            raise ValueError("window must be in 2..16")
        table = np.zeros((1 << (int(window) - 1), w), dtype=np.uint64)
        fn = self._lib.bls_g2_wnaf_table if g2 else self._lib.bls_g1_wnaf_table
        self._check(fn(self._ctx, _p(base), int(window), _p(table)))
        return table

    def g1_wnaf_table(self, base, window): return self._wnaf_table(False, base, window)
    def g2_wnaf_table(self, base, window): return self._wnaf_table(True, base, window)

    def g1_wnaf_mul(self, bases, k, window=0): return self._wnaf(False, bases, k, window, "wnaf")
    def g2_wnaf_mul(self, bases, k, window=0): return self._wnaf(True, bases, k, window, "wnaf")
    def g1_mul(self, bases, k): return self._wnaf(False, bases, k, 0, "mul")
    def g2_mul(self, bases, k): return self._wnaf(True, bases, k, 0, "mul")

    def g1_batch_normalization(self, v):
        v = _arr(v, W_G1, "v").copy()
        self._check(self._lib.bls_g1_batch_normalization(self._ctx, _p(v), v.shape[0]))
        return v

    def g2_batch_normalization(self, v):
        v = _arr(v, W_G2, "v").copy()
        self._check(self._lib.bls_g2_batch_normalization(self._ctx, _p(v), v.shape[0]))
        return v

    def g1_into_affine(self, v):
        v = _arr(v, W_G1, "v")
        out = np.zeros((v.shape[0], W_G1A), dtype=np.uint64)
        self._check(self._lib.bls_g1_into_affine_batch(self._ctx, _p(v), _p(out), v.shape[0]))
        return out

    def g2_into_affine(self, v):
        v = _arr(v, W_G2, "v")
        out = np.zeros((v.shape[0], W_G2A), dtype=np.uint64)
        self._check(self._lib.bls_g2_into_affine_batch(self._ctx, _p(v), _p(out), v.shape[0]))
        return out

    def _pt_op(self, g2, op, a, b):
        w, wa = (W_G2, W_G2A) if g2 else (W_G1, W_G1A)
        a = _arr(a, w, "a")
        if b is not None:
            b = _arr(b, wa if op == "add_mixed" else w, "b")
        out = np.zeros_like(a)
        fn = self._lib.bls_g2_op_batch if g2 else self._lib.bls_g1_op_batch
        self._check(fn(self._ctx, PT_OPS[op], _p(a), _p(b), _p(out), a.shape[0]))
        return out

    def g1_op(self, op, a, b=None): return self._pt_op(False, op, a, b)
    def g2_op(self, op, a, b=None): return self._pt_op(True, op, a, b)

    def _msm(self, g2, bases, k):
        bases, k = _arr(bases, W_G2A if g2 else W_G1A, "bases"), _arr(k, W_FR, "k")
        if bases.shape[0] != k.shape[0]:
            raise ValueError("bases and k must have the same length")
        out = np.zeros((1, W_G2 if g2 else W_G1), dtype=np.uint64)
        fn = self._lib.bls_g2_msm if g2 else self._lib.bls_g1_msm
        self._check(fn(self._ctx, _p(bases), _p(k), bases.shape[0], _p(out)))
        return out

    def g1_msm(self, bases, k):
        """sum_i k_i * bases_i over (n, 13) affine bases and (n, 4) FrRepr scalars -> one normalised Jacobian row (1, 18)."""
        return self._msm(False, bases, k)

    def g2_msm(self, bases, k):
        """sum_i k_i * bases_i over (n, 25) affine bases and (n, 4) FrRepr scalars -> one normalised Jacobian row (1, 36)."""
        return self._msm(True, bases, k)

    def _msm_batch(self, g2, bases, k):
        wa = W_G2A if g2 else W_G1A
        k = np.ascontiguousarray(k, dtype=np.uint64)
        bases = np.ascontiguousarray(bases, dtype=np.uint64)
        if k.ndim != 3 or k.shape[2] != W_FR:
            raise ValueError("k must have shape (m, n, %d) uint64, got %r" % (W_FR, k.shape))
        m, n = k.shape[:2]
        if bases.shape not in ((n, wa), (m, n, wa)):
            raise ValueError("bases must have shape (n, %d) (shared) or (m, n, %d), got %r for k of %r" % (wa, wa, bases.shape, k.shape))
        out = np.zeros((m, W_G2 if g2 else W_G1), dtype=np.uint64)
        fn = self._lib.bls_g2_msm_batch if g2 else self._lib.bls_g1_msm_batch
        self._check(fn(self._ctx, _p(bases), 1 if bases.ndim == 2 else 0, _p(k), n, m, _p(out)))
        return out

    def g1_msm_batch(self, bases, k):
        """m independent sums: k (m, n, 4) FrRepr scalars against (n, 13) affine bases shared by every sum or (m, n, 13),
        one set per sum -> (m, 18) normalised Jacobian rows, row j = g1_msm(bases (of sum j), k[j])."""
        return self._msm_batch(False, bases, k)

    def g2_msm_batch(self, bases, k):
        """g1_msm_batch in G2: bases (n, 25) or (m, n, 25) -> (m, 36)."""
        return self._msm_batch(True, bases, k)

    # ------------------------------------------------------------------ field tower, host arrays
    def field_op(self, degree, op, a, b=None):
        a = _arr(a, 6 * degree, "a")
        if b is not None:
            b = _arr(b, 6 * degree, "b")
        out = np.zeros_like(a)
        ok = np.zeros(a.shape[0], dtype=np.uint8)
        self._check(self._lib.bls_field_op_batch(self._ctx, degree, OPS[op], _p(a), _p(b), _p(out), _p(ok), a.shape[0]))
        return out, ok

    def pair_field_op(self, degree, op, a, b=None):
        """the same operation on the lane-pair tower of the pairing kernels (degree 2, 6, 12)"""
        a = _arr(a, 6 * degree, "a")
        if b is not None:
            b = _arr(b, 6 * degree, "b")
            if b.shape[0] != a.shape[0]:
                raise ValueError("a and b must have the same length")
        out = np.zeros_like(a)
        ok = np.zeros(a.shape[0], dtype=np.uint8)
        self._check(self._lib.bls_pair_field_op_batch(self._ctx, degree, OPS[op], _p(a), _p(b), _p(out), _p(ok), a.shape[0]))
        return out, ok

    # ------------------------------------------------------------------ device pointers
    def point_from_x(self, g2, x, greatest):
        """$affine::get_point_from_x for n x-coordinates (Montgomery limbs) -> (affine rows, is_some)."""
        x = _arr(x, W_FQ2 if g2 else W_FQ, "x")
        gr = np.ascontiguousarray(greatest, dtype=np.uint8).reshape(-1)
        if gr.shape[0] != x.shape[0]:
            raise ValueError("x and greatest must have the same length")
        out = np.zeros((x.shape[0], W_G2A if g2 else W_G1A), dtype=np.uint64)
        ok = np.zeros(x.shape[0], dtype=np.uint8)
        fn = self._lib.bls_g2_point_from_x_batch if g2 else self._lib.bls_g1_point_from_x_batch
        self._check(fn(self._ctx, _p(x), _p(gr), _p(out), _p(ok), x.shape[0]))
        return out, ok

    def affine_mul(self, g2, affine, k):
        """CurveAffine::mul for n (affine point, FrRepr) pairs -> Jacobian rows."""
        affine, k = _arr(affine, W_G2A if g2 else W_G1A, "affine"), _arr(k, W_FR, "k")
        if affine.shape[0] != k.shape[0]:
            raise ValueError("affine and k must have the same length")
        out = np.zeros((affine.shape[0], W_G2 if g2 else W_G1), dtype=np.uint64)
        fn = self._lib.bls_g2_affine_mul_batch if g2 else self._lib.bls_g1_affine_mul_batch
        self._check(fn(self._ctx, _p(affine), _p(k), _p(out), affine.shape[0]))
        return out

    def scale_by_cofactor(self, g2, affine):
        affine = _arr(affine, W_G2A if g2 else W_G1A, "affine")
        out = np.zeros((affine.shape[0], W_G2 if g2 else W_G1), dtype=np.uint64)
        fn = self._lib.bls_g2_scale_by_cofactor_batch if g2 else self._lib.bls_g1_scale_by_cofactor_batch
        self._check(fn(self._ctx, _p(affine), _p(out), affine.shape[0]))
        return out

    def fr_op(self, op, a, b=None):
        """Fr field operation (Montgomery-form (n,4) arrays; from_repr/into_repr convert) -> (values, ok)."""
        a = _arr(a, W_FR, "a")
        if b is not None:
            b = _arr(b, W_FR, "b")
        out = np.zeros_like(a)
        ok = np.zeros(a.shape[0], dtype=np.uint8)
        self._check(self._lib.bls_fr_op_batch(self._ctx, OPS[op], _p(a), _p(b) if b is not None else None, _p(out), _p(ok), a.shape[0]))
        return out, ok

    def fr_fft(self, kind, a):
        """bellman's EvaluationDomain transforms over Fr: kind "fft" | "ifft" | "coset_fft" | "icoset_fft" on one
        polynomial (n, 4) or m polynomials (m, n, 4) of Montgomery-form values, n a power of two -> same shape."""
        kind = FFT_KINDS[kind]
        a = np.ascontiguousarray(a, dtype=np.uint64)
        if a.ndim not in (2, 3) or a.shape[-1] != W_FR:
            raise ValueError("a must have shape (n, 4) or (m, n, 4) uint64, got %r" % (a.shape,))
        n = a.shape[-2]
        log_n = n.bit_length() - 1
        if n != 1 << log_n:
            raise ValueError("the polynomial length must be a power of two, got %d" % n)
        m = a.shape[0] if a.ndim == 3 else 1
        out = np.zeros_like(a)
        self._check(self._lib.bls_fr_fft_batch(self._ctx, kind, _p(a), _p(out), log_n, m))
        return out

    def fr_fft_scratch_bytes(self, log_n, m=1):
        """device scratch of bls_fr_fft_dev for m polynomials of 2^log_n; raises for arguments the call would reject"""
        b = int(self._lib.bls_fr_fft_scratch_bytes(self._ctx, log_n, m))
        if b == 0:
            raise ValueError("no FFT of log_n = %d, m = %d" % (log_n, m))
        return b

    def fr_groth16_h(self, a, b, c):
        """Groth16's quotient polynomial (the `h` block of bellman's create_proof): a, b, c are the evaluations of one
        proof (len, 4) or of m proofs (m, len, 4), Montgomery-form values -> H's coefficients 0 .. n - 2 as canonical
        FrRepr, (n - 1, 4) or (m, n - 1, 4), n the smallest power of two >= len (1 for len <= 1)."""
        a, b, c = (np.ascontiguousarray(x, dtype=np.uint64) for x in (a, b, c))
        if a.ndim not in (2, 3) or a.shape[-1] != W_FR or b.shape != a.shape or c.shape != a.shape:
            raise ValueError("a, b and c must have one shape (len, 4) or (m, len, 4) uint64, got %r, %r, %r" % (a.shape, b.shape, c.shape))
        length = a.shape[-2]
        m = a.shape[0] if a.ndim == 3 else 1
        n = 1 << max(length - 1, 0).bit_length()
        out = np.zeros(a.shape[:-2] + (n - 1, W_FR), dtype=np.uint64)
        self._check(self._lib.bls_fr_groth16_h_batch(self._ctx, _p(a), _p(b), _p(c), length, m, _p(out)))
        return out

    def fr_groth16_h_scratch_bytes(self, length, m=1):
        """device scratch of bls_fr_groth16_h_dev for m proofs of `length` evaluations; raises for arguments the call would reject"""
        b = int(self._lib.bls_fr_groth16_h_scratch_bytes(self._ctx, length, m))
        if b == 0:
            raise ValueError("no Groth16 H of len = %d, m = %d" % (length, m))
        return b

    def groth16_prove(self, params, a, b, c, input, aux, densities, r, s):
        """bellman's groth16::create_proof for m proofs of one circuit (bls_groth16_prove_batch).  params: Groth16Params of
        numpy rows; a, b, c (m, len, 4), input (m, num_inputs, 4), aux (m, num_aux, 4), r and s (m, 4), all Montgomery-form
        Fr; densities = (a_aux_density, b_input_density, b_aux_density), numpy bool arrays of num_aux, num_inputs and num_aux
        entries.  Returns the proofs (A (m, 13), B (m, 25), C (m, 13)) in affine form, views of one (m, 51) array."""
        a, b, c, input, aux = (np.ascontiguousarray(x, dtype=np.uint64) for x in (a, b, c, input, aux))
        r, s = (np.ascontiguousarray(x, dtype=np.uint64) for x in (r, s))
        if a.ndim != 3 or a.shape[2] != W_FR or b.shape != a.shape or c.shape != a.shape:
            raise ValueError("a, b and c must have one shape (m, len, 4) uint64, got %r, %r, %r" % (a.shape, b.shape, c.shape))
        m, length = a.shape[:2]
        for x, name in ((input, "input"), (aux, "aux")):
            if x.ndim != 3 or x.shape[0] != m or x.shape[2] != W_FR:
                raise ValueError("%s must have shape (%d, n, 4) uint64, got %r" % (name, m, x.shape))
        for x, name in ((r, "r"), (s, "s")):
            if x.shape != (m, W_FR):
                raise ValueError("%s must have shape (%d, 4) uint64, got %r" % (name, m, x.shape))
        ni, na = input.shape[1], aux.shape[1]
        q = {}
        for name, w in (("h", W_G1A), ("l", W_G1A), ("a", W_G1A), ("b_g1", W_G1A), ("b_g2", W_G2A)):
            q[name] = _arr(getattr(params, name), w, name)
        pc = groth16_params_c(Groth16Params(params.alpha_g1, params.beta_g1, params.delta_g1, params.beta_g2, params.delta_g2, **q), _p, len)
        dw = [density_words(d, bits, name) for d, bits, name in zip(densities, (na, ni, na), ("a_aux_density", "b_input_density", "b_aux_density"))]
        out = np.zeros((m, W_PROOF), dtype=np.uint64)
        self._check(self._lib.bls_groth16_prove_batch(self._ctx, ctypes.byref(pc), _p(a), _p(b), _p(c), length, _p(input), ni, _p(aux), na,
                                                      _p(dw[0]), _p(dw[1]), _p(dw[2]), _p(r), _p(s), m, _p(out)))
        return out[:, :W_G1A], out[:, W_G1A:W_G1A + W_G2A], out[:, W_G1A + W_G2A:]

    def groth16_prove_scratch_bytes(self, params_c, length, num_inputs, num_aux, density_words_, m):
        """device scratch of bls_groth16_prove_dev; params_c from groth16_params_c, density_words_ the three uint32 word
        arrays; raises for arguments the call would reject"""
        n = int(self._lib.bls_groth16_prove_scratch_bytes(self._ctx, ctypes.byref(params_c), length, num_inputs, num_aux,
                                                          *[_p(w) for w in density_words_], m))
        if n == 0:
            raise ValueError("no Groth16 proof of len = %d, num_inputs = %d, num_aux = %d, m = %d for these params and densities"
                             % (length, num_inputs, num_aux, m))
        return n

    def groth16_prepare_verifying_key(self, alpha_g1, beta_g2, gamma_g2, delta_g2):
        """bellman's prepare_verifying_key (bls_groth16_prepare_verifying_key): alpha_g1 a (13,) G1Affine row, beta_g2,
        gamma_g2, delta_g2 (25,) G2Affine rows -> the bls_groth16_pvk as a (5022,) uint64 array (Groth16PvkC's layout)."""
        rows = []
        for x, w, name in ((alpha_g1, W_G1A, "alpha_g1"), (beta_g2, W_G2A, "beta_g2"), (gamma_g2, W_G2A, "gamma_g2"), (delta_g2, W_G2A, "delta_g2")):
            rows.append(_arr(np.reshape(x, (1, -1)), w, name))
        out = np.zeros(W_PVK, dtype=np.uint64)
        self._check(self._lib.bls_groth16_prepare_verifying_key(self._ctx, *[_p(r) for r in rows], _p(out)))
        return out

    def _verify_args(self, pvk, ic, proofs, inputs):
        pvk = np.ascontiguousarray(pvk, dtype=np.uint64)
        if pvk.shape != (W_PVK,):
            raise ValueError("pvk must be a (%d,) uint64 array, got %r" % (W_PVK, pvk.shape))
        ic, proofs = _arr(ic, W_G1A, "ic"), _arr(proofs, W_PROOF, "proofs")
        m, ni = proofs.shape[0], ic.shape[0] - 1
        inputs = np.ascontiguousarray(inputs, dtype=np.uint64)
        if ni < 0 or inputs.shape != (m, ni, W_FR):
            raise ValueError("ic must hold num_inputs + 1 points and inputs have shape (m, num_inputs, 4) = (%d, %d, 4), got %r, %r"
                             % (m, max(ni, 0), ic.shape, inputs.shape))
        return pvk, ic, proofs, inputs, m, ni

    def groth16_verify(self, pvk, ic, proofs, inputs):
        """bellman's verify_proof for m proofs of one circuit (bls_groth16_verify_batch): pvk from
        groth16_prepare_verifying_key, ic (num_inputs + 1, 13), proofs (m, 51) rows (A, B, C), inputs (m, num_inputs, 4)
        Montgomery-form Fr without the leading one -> (m,) bool array."""
        pvk, ic, proofs, inputs, m, ni = self._verify_args(pvk, ic, proofs, inputs)
        ok = np.zeros(m, dtype=np.uint8)
        self._check(self._lib.bls_groth16_verify_batch(self._ctx, _p(pvk), _p(ic), ni, _p(proofs), _p(inputs), m, _p(ok)))
        return ok.astype(bool)

    def groth16_verify_rlc(self, pvk, ic, proofs, inputs, rho):
        """the randomized batch check (bls_groth16_verify_rlc_batch): the arguments of groth16_verify and the randomizers
        rho (m, 4) canonical FrRepr -> one bool (True for m = 0: the equation holds for the empty batch)"""
        pvk, ic, proofs, inputs, m, ni = self._verify_args(pvk, ic, proofs, inputs)
        rho = np.ascontiguousarray(rho, dtype=np.uint64)
        if rho.shape != (m, W_FR):
            raise ValueError("rho must have shape (%d, 4) uint64, got %r" % (m, rho.shape))
        ok = np.zeros(1, dtype=np.uint8)
        self._check(self._lib.bls_groth16_verify_rlc_batch(self._ctx, _p(pvk), _p(ic), ni, _p(proofs), _p(inputs), _p(rho), m, _p(ok)))
        return bool(ok[0])

    def groth16_verify_scratch_bytes(self, num_inputs, m):
        n = int(self._lib.bls_groth16_verify_scratch_bytes(self._ctx, num_inputs, m))
        if n == 0:
            raise ValueError("no Groth16 verification of m = %d proofs with num_inputs = %d" % (m, num_inputs))
        return n

    def groth16_verify_rlc_scratch_bytes(self, num_inputs, m):
        n = int(self._lib.bls_groth16_verify_rlc_scratch_bytes(self._ctx, num_inputs, m))
        if n == 0:
            raise ValueError("no randomized Groth16 check of m = %d proofs with num_inputs = %d" % (m, num_inputs))
        return n

    def groth16_generate_parameters(self, abc, num_constraints, num_inputs, num_aux, g1, g2, alpha, beta, gamma, delta, tau):
        """bellman's groth16::generate_parameters (bls_groth16_generate_parameters_batch): abc three (offsets, constraint,
        coeff) numpy triples, A, B, C variable-major over num_inputs + num_aux variables (offsets uint64, constraint uint32,
        coeff (nnz, 4) Montgomery Fr); g1 a (13,) G1Affine row, g2 a (25,) G2Affine row; alpha .. tau (4,) Montgomery Fr.
        Returns a Groth16Parameters."""
        ni, na = int(num_inputs), int(num_aux)
        nv = ni + na
        keep, mats = r1cs_matrices(abc, num_constraints, nv)
        g1 = _arr(np.reshape(g1, (1, -1)), W_G1A, "g1")
        g2 = _arr(np.reshape(g2, (1, -1)), W_G2A, "g2")
        sc = []
        for x, name in ((alpha, "alpha"), (beta, "beta"), (gamma, "gamma"), (delta, "delta"), (tau, "tau")):
            sc.append(_arr(np.reshape(x, (1, -1)), W_FR, name))
        n1 = (1 << max(int(num_constraints) - 1, 0).bit_length()) - 1
        vk = np.zeros(W_VK_POINTS, dtype=np.uint64)
        ic, h, l = (np.zeros((k, W_G1A), dtype=np.uint64) for k in (ni, n1, na))
        a, b_g1 = (np.zeros((nv, W_G1A), dtype=np.uint64) for _ in range(2))
        b_g2 = np.zeros((nv, W_G2A), dtype=np.uint64)
        dens = [np.zeros((k + 31) // 32, dtype=np.uint32) for k in (na, ni, na)]
        lens = np.zeros(2, dtype=np.uint64)
        ok = np.zeros(1, dtype=np.uint8)
        out = Groth16ParametersOutC(*[_p(x) for x in (vk, ic, h, l, a, b_g1, b_g2, *dens, lens, ok)])
        self._check(self._lib.bls_groth16_generate_parameters_batch(self._ctx, mats, num_constraints, ni, na, _p(g1), _p(g2),
                                                                    *[_p(x) for x in sc], ctypes.byref(out)))
        del keep
        return groth16_parameters(vk, ic, h, l, a, b_g1, b_g2, dens, lens, ok[0], ni, na)

    def groth16_generate_parameters_scratch_bytes(self, mats, num_constraints, num_inputs, num_aux):
        """device scratch of bls_groth16_generate_parameters_dev; mats a bls_r1cs_matrix[3] (R1csMatrixC * 3); raises for
        arguments the call would reject"""
        n = int(self._lib.bls_groth16_generate_parameters_scratch_bytes(self._ctx, mats, num_constraints, num_inputs, num_aux))
        if n == 0:
            raise ValueError("no Groth16 parameters for num_constraints = %d, num_inputs = %d, num_aux = %d and these matrices"
                             % (num_constraints, num_inputs, num_aux))
        return n

    # ------------------------------------------------------------------ KZG commitments
    def kzg_commit(self, srs, p):
        """c[j] = sum_i p[j, i] srs[i] (bls_kzg_commit_batch): srs (>= n, 13) affine rows [tau^i] g, p (m, n, 4) Montgomery
        coefficients -> (m, 13) affine rows."""
        srs, p = _arr(srs, W_G1A, "srs"), np.ascontiguousarray(p, dtype=np.uint64)
        m, n = kzg_poly_shape(p.shape, srs.shape[0], False)
        out = np.zeros((m, W_G1A), dtype=np.uint64)
        self._check(self._lib.bls_kzg_commit_batch(self._ctx, _p(srs), srs.shape[0], _p(p), n, m, _p(out)))
        return out

    def kzg_open(self, srs, p, z):
        """open polynomial j at z[j] (bls_kzg_open_batch): srs (>= n - 1, 13), p (m, n, 4), z (m, 4) Montgomery Fr -> (y (m, 4)
        Montgomery p_j(z_j), proof (m, 13) affine [q_j(tau)] g)."""
        srs, p, z = _arr(srs, W_G1A, "srs"), np.ascontiguousarray(p, dtype=np.uint64), np.ascontiguousarray(z, dtype=np.uint64)
        m, n = kzg_poly_shape(p.shape, srs.shape[0], True)
        if z.shape != (m, W_FR):
            raise ValueError("z must have shape (%d, 4) uint64, got %r" % (m, z.shape))
        y, proof = np.zeros((m, W_FR), dtype=np.uint64), np.zeros((m, W_G1A), dtype=np.uint64)
        self._check(self._lib.bls_kzg_open_batch(self._ctx, _p(srs), srs.shape[0], _p(p), n, _p(z), m, _p(y), _p(proof)))
        return y, proof

    def kzg_prepare_verifying_key(self, g, h, tau_h):
        """bls_kzg_prepare_verifying_key: g a (13,) G1Affine row, h and tau_h (25,) G2Affine rows -> the bls_kzg_pvk as a
        (4963,) uint64 array (KzgPvkC's layout)."""
        rows = [_arr(np.reshape(x, (1, -1)), w, name) for x, w, name in ((g, W_G1A, "g"), (h, W_G2A, "h"), (tau_h, W_G2A, "tau_h"))]
        out = np.zeros(W_KZG_PVK, dtype=np.uint64)
        self._check(self._lib.bls_kzg_prepare_verifying_key(self._ctx, *[_p(r) for r in rows], _p(out)))
        return out

    def _kzg_verify_args(self, pvk, c, y, z, proof):
        pvk = np.ascontiguousarray(pvk, dtype=np.uint64)
        if pvk.shape != (W_KZG_PVK,):
            raise ValueError("pvk must be a (%d,) uint64 array, got %r" % (W_KZG_PVK, pvk.shape))
        c, proof, y, z = _arr(c, W_G1A, "c"), _arr(proof, W_G1A, "proof"), _arr(y, W_FR, "y"), _arr(z, W_FR, "z")
        m = c.shape[0]
        if not (proof.shape[0] == y.shape[0] == z.shape[0] == m):
            raise ValueError("c, y, z and proof must have the same number of rows")
        return pvk, c, y, z, proof, m

    def kzg_verify(self, pvk, c, y, z, proof):
        """bls_kzg_verify_batch: pvk from kzg_prepare_verifying_key, c and proof (m, 13) affine rows, y and z (m, 4) Montgomery
        Fr -> (m,) bool array."""
        pvk, c, y, z, proof, m = self._kzg_verify_args(pvk, c, y, z, proof)
        ok = np.zeros(m, dtype=np.uint8)
        self._check(self._lib.bls_kzg_verify_batch(self._ctx, _p(pvk), _p(c), _p(y), _p(z), _p(proof), m, _p(ok)))
        return ok.astype(bool)

    def kzg_verify_rlc(self, pvk, c, y, z, proof, rho):
        """the randomized check (bls_kzg_verify_rlc_batch): kzg_verify's arguments and rho (m, 4) canonical FrRepr -> one bool
        (True for m = 0)"""
        pvk, c, y, z, proof, m = self._kzg_verify_args(pvk, c, y, z, proof)
        rho = np.ascontiguousarray(rho, dtype=np.uint64)
        if rho.shape != (m, W_FR):
            raise ValueError("rho must have shape (%d, 4) uint64, got %r" % (m, rho.shape))
        ok = np.zeros(1, dtype=np.uint8)
        self._check(self._lib.bls_kzg_verify_rlc_batch(self._ctx, _p(pvk), _p(c), _p(y), _p(z), _p(proof), _p(rho), m, _p(ok)))
        return bool(ok[0])

    def kzg_scratch_bytes(self, what, *args):
        """device scratch of bls_kzg_<what>_dev: what "commit" / "open" (args n, m), "verify" / "verify_rlc" (args m); raises
        for arguments the call would reject"""
        b = int(getattr(self._lib, "bls_kzg_%s_scratch_bytes" % what)(self._ctx, *args))
        if b == 0:
            raise ValueError("no KZG %s for %r" % (what, args))
        return b

    def call_dev(self, name, *args):
        """Raw access to a `*_dev` entry point: args are ints (device pointers / sizes / stream)."""
        self._check(getattr(self._lib, name)(self._ctx, *args))

    def multi_miller_scratch_bytes(self, n):
        return int(self._lib.bls_multi_miller_scratch_bytes(self._ctx, n))

    def fq12_product_scratch_bytes(self, n):
        return int(self._lib.bls_fq12_product_scratch_bytes(self._ctx, n))

    def batch_normalization_scratch_bytes(self, degree, n):
        return int(self._lib.bls_batch_normalization_scratch_bytes(self._ctx, degree, n))

    def msm_scratch_bytes(self, degree, n, window=0):
        """device scratch of bls_g*_msm_dev (degree 1 = G1, 2 = G2); raises for arguments the call would reject"""
        b = int(self._lib.bls_msm_scratch_bytes(self._ctx, degree, n, window))
        if b == 0:
            raise ValueError("no MSM of degree %r, n = %d, window = %d" % (degree, n, window))
        return b

    def msm_batch_scratch_bytes(self, degree, n, m, window=0):
        """device scratch of bls_g*_msm_batch_dev for m sums of n points; raises for arguments the call would reject"""
        b = int(self._lib.bls_msm_batch_scratch_bytes(self._ctx, degree, n, m, window))
        if b == 0:
            raise ValueError("no MSM batch of degree %r, n = %d, m = %d, window = %d" % (degree, n, m, window))
        return b

    def imad_peak(self, variant=0, iters=2000):
        macs, ms = ctypes.c_double(0), ctypes.c_double(0)
        self._check(self._lib.bls_imad_peak(self._ctx, variant, iters, ctypes.byref(macs), ctypes.byref(ms)))
        return macs.value, ms.value


class MultiGpu:
    """Several devices of one node behind one call (bls_mgpu): an n-pair product or batch is split into contiguous
    shards, one host thread per device inside the library; the product's 576-byte partials meet on the first device."""

    def __init__(self, devices):
        self._lib = load()
        devices = list(range(devices)) if isinstance(devices, int) else [int(d) for d in devices]
        arr = (ctypes.c_int * len(devices))(*devices)
        err = ctypes.c_int(0)
        self._m = self._lib.bls_mgpu_create(arr, len(devices), ctypes.byref(err))
        if not self._m:
            raise BlsError("bls_mgpu_create(%r) failed: %s" % (devices, self._lib.bls_strerror(err.value).decode()))
        self.devices = devices

    def close(self):
        if getattr(self, "_m", None):
            self._lib.bls_mgpu_destroy(self._m)
            self._m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            msgs = [self._lib.bls_ctx_last_error(self._lib.bls_mgpu_ctx(self._m, i)).decode() for i in range(len(self.devices))]
            raise BlsError("%s %r" % (self._lib.bls_strerror(rc).decode(), [m for m in msgs if m]))

    @property
    def device_count(self):
        return self._lib.bls_mgpu_device_count(self._m)

    def _pairs(self, p, q):
        p, q = _arr(p, W_G1A, "p"), _arr(q, W_G2A, "q")
        if p.shape[0] != q.shape[0]:
            raise ValueError("p and q must have the same length")
        return p, q

    def multi_miller_loop(self, p, q):
        p, q = self._pairs(p, q)
        out = np.zeros((1, W_FQ12), dtype=np.uint64)
        self._check(self._lib.bls_mgpu_multi_miller_loop(self._m, _p(p), _p(q), p.shape[0], _p(out)))
        return out

    def pairing_product(self, p, q):
        p, q = self._pairs(p, q)
        out = np.zeros((1, W_FQ12), dtype=np.uint64)
        ok = np.zeros(1, dtype=np.uint8)
        self._check(self._lib.bls_mgpu_pairing_product(self._m, _p(p), _p(q), p.shape[0], _p(out), _p(ok)))
        return out, bool(ok[0])

    def pairing(self, p, q):
        p, q = self._pairs(p, q)
        out = np.zeros((p.shape[0], W_FQ12), dtype=np.uint64)
        self._check(self._lib.bls_mgpu_pairing_batch(self._m, _p(p), _p(q), _p(out), p.shape[0]))
        return out

    def _wnaf(self, fn, w, bases, k):
        bases, k = _arr(bases, w, "bases"), _arr(k, W_FR, "k")
        if bases.shape[0] != k.shape[0]:
            raise ValueError("bases and k must have the same length")
        out = np.zeros_like(bases)
        self._check(fn(self._m, _p(bases), _p(k), _p(out), bases.shape[0]))
        return out

    def g1_wnaf_mul(self, bases, k):
        return self._wnaf(self._lib.bls_mgpu_g1_wnaf_mul_batch, W_G1, bases, k)

    def g2_wnaf_mul(self, bases, k):
        return self._wnaf(self._lib.bls_mgpu_g2_wnaf_mul_batch, W_G2, bases, k)

    def last_phase_ms(self):
        ms = (ctypes.c_double * 3)()
        self._check(self._lib.bls_mgpu_last_phase_ms(self._m, ms))
        return {"shards_ms": ms[0], "tail_ms": ms[1], "total_ms": ms[2]}
