"""ctypes binding of libvdfgpu.so (include/vdfgpu.h).  There is no fallback: if the library or a GPU is
missing, calls raise."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_bool, c_char_p, c_double, c_int, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libvdfgpu.so"
_lib = None


class VdfGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"vdfgpu error {code}: {msg}")
        self.code = code


# name -> (restype, argtypes); every symbol include/vdfgpu.h declares
PROTOTYPES = {
    "vdfgpu_init": (c_int, [c_int]),
    "vdfgpu_shutdown": (c_int, []),
    "vdfgpu_device_count": (c_int, []),
    "vdfgpu_last_error": (c_char_p, []),
    "vdfgpu_version": (c_char_p, []),
    "vdfgpu_set_stream": (c_int, [c_void_p]),
    "vdfgpu_synchronize": (c_int, []),
    "vdfgpu_launch_count": (c_uint64, []),
    "vdfgpu_trim": (c_int, []),
    "vdfgpu_dropin_cache_clear": (c_int, []),
    "vdfgpu_dropin_cache_stats": (c_int, [POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint64)]),
    "vdfgpu_witness_bank_create": (c_int, [c_int, c_void_p, c_uint64, c_size_t, POINTER(c_void_p)]),
    "vdfgpu_witness_bank_destroy": (c_int, [c_void_p]),
    "vdfgpu_witness_bank_read": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p]),
    "vdfgpu_running_commit_step": (c_int, [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_profile_enable": (c_int, [c_int]),
    "vdfgpu_profile_read": (c_int, [POINTER(c_double), c_int]),
    "vdfgpu_point_sum_dev": (c_int, [c_int, c_void_p, c_size_t, c_void_p]),
    "mult_pippenger_pallas": (None, [c_void_p, c_void_p, c_size_t, c_void_p, c_bool]),
    "mult_pippenger_vesta": (None, [c_void_p, c_void_p, c_size_t, c_void_p, c_bool]),
    "vdfgpu_gens_create": (c_int, [c_int, c_void_p, c_size_t, c_uint32, c_uint32, POINTER(c_void_p)]),
    "vdfgpu_gens_progression": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_uint32, c_uint32, POINTER(c_void_p)]),
    "vdfgpu_gens_export": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p]),
    "vdfgpu_gens_len": (c_size_t, [c_void_p]),
    "vdfgpu_gens_window_bits": (c_uint32, [c_void_p, c_size_t]),
    "vdfgpu_gens_affine_rounds": (c_uint32, [c_void_p, c_size_t]),
    "vdfgpu_gens_destroy": (c_int, [c_void_p]),
    "vdfgpu_msm": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_msm_submit": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
    "vdfgpu_msm_wait": (c_int, [c_int]),
    "vdfgpu_msm_dev": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_msm_batch_dev": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_size_t), c_uint32, c_void_p]),
    "vdfgpu_msm_range_dev": (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_point_normalise_host": (c_int, [c_int, c_void_p, c_size_t]),
    "vdfgpu_point_sum": (c_int, [c_int, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_r1cs_create": (c_int, [c_int, c_size_t, c_size_t, c_size_t,
                                   c_void_p, c_void_p, c_void_p, c_size_t,
                                   c_void_p, c_void_p, c_void_p, c_size_t,
                                   c_void_p, c_void_p, c_void_p, c_size_t, POINTER(c_void_p)]),
    "vdfgpu_r1cs_destroy": (c_int, [c_void_p]),
    "vdfgpu_multiply_vec": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_commit_T": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_fold": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_multiply_vec_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_r1cs_bind_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_r1cs_bind_rows_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_cross_term_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_fold_dev": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_running_create": (c_int, [c_void_p, c_void_p, POINTER(c_void_p)]),
    "vdfgpu_running_destroy": (c_int, [c_void_p]),
    "vdfgpu_running_set": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_running_get": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_running_commit": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_running_finish": (c_int, [c_void_p, c_void_p]),
    "vdfgpu_r1cs_is_sat_relaxed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           POINTER(c_uint64)]),
    "vdfgpu_r1cs_is_sat_relaxed_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_running_check": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(c_uint64)]),
    "vdfgpu_running_spartan_prove": (c_int, [c_void_p] * 8),
    "vdfgpu_r1cs_evaluate": (c_int, [c_void_p] * 4),
    "vdfgpu_r1cs_evaluate_batch": (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_spartan_verify_batch": (c_int, [c_void_p, c_void_p, c_size_t] + [c_void_p] * 6),
    "vdfgpu_eq_evals": (c_int, [c_int, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_eq_evals_dev": (c_int, [c_int, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_sumcheck_cubic": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_sumcheck_cubic_dev": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_sumcheck_quad": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_sumcheck_quad_dev": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_poly_evaluate": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_poly_evaluate_dev": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_vec_lincomb": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_inner_product": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_points_lincomb": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_ipa_prove": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_ipa_prove_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdfgpu_ipa_gens_hat": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "vdfgpu_ipa_verify_batch": (c_int, [c_void_p, c_size_t, c_size_t] + [c_void_p] * 10),
    "vdfgpu_minroot_check_batch": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_uint64, c_size_t, c_void_p]),
    "vdfgpu_minroot_check_batch_dev": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_uint64, c_size_t, c_void_p]),
    "vdfgpu_minroot_inverse_eval_batch": (c_int, [c_int, c_void_p, c_uint64, c_size_t, c_void_p]),
    "vdfgpu_minroot_witness_batch": (c_int, [c_int, c_void_p, c_uint64, c_size_t, c_void_p]),
    "vdfgpu_field_mul_batch": (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_uint32, c_void_p]),
    "vdfgpu_imad_peak": (c_int, [POINTER(c_double), POINTER(c_double), POINTER(c_double)]),
}


# int (*vdfgpu_round_fn)(void* user, size_t round, const void* evals_fe32, size_t n_evals, void* r_out_fe32)
ROUND_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p)
# int (*vdfgpu_ipa_round_fn)(void* user, size_t round, const void* L_point96, const void* R_point96, void* r_out32)
IPA_ROUND_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p)
# int (*vdfgpu_spartan_claims_fn)(void* user, int stage, const void* in_fe32, size_t n_in, void* out_fe32, size_t n_out)
CLAIMS_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_size_t)


def lib_path() -> Path:
    return Path(os.environ.get("VDFGPU_LIB", _LIB_PATH))


def load() -> ctypes.CDLL:
    """Load libvdfgpu.so (built in-tree by vdf_b200._build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not path.exists():
            raise FileNotFoundError(
                f"{path} is missing: build it with `python -m vdf_b200._build` "
                "(there is no CPU fallback for the GPU path)")
        lib = ctypes.CDLL(str(path))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().vdfgpu_last_error()
        raise VdfGpuError(rc, msg.decode() if msg else "")


def as_ptr(buf) -> c_void_p:
    """Pointer to the start of a bytes / bytearray / numpy / torch-CPU buffer (kept alive by caller)."""
    if buf is None:
        return c_void_p(None)
    if isinstance(buf, int):
        return c_void_p(buf)
    if isinstance(buf, (bytes, bytearray)):
        if isinstance(buf, bytes):
            return ctypes.cast(ctypes.c_char_p(buf), c_void_p)
        return ctypes.cast((ctypes.c_char * len(buf)).from_buffer(buf), c_void_p)
    if hasattr(buf, "data_ptr"):  # torch tensor
        return c_void_p(buf.data_ptr())
    if hasattr(buf, "ctypes"):  # numpy array
        return c_void_p(buf.ctypes.data)
    raise TypeError(f"cannot take the address of {type(buf)!r}")
