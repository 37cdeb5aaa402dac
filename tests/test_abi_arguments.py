"""CPU: every entry point that takes a field or curve id rejects an unknown one as an argument error
(VDFGPU_ERR_ARG, "<prefix>: unknown field / curve") before it touches the device, so the same answer comes back with
or without a GPU.  The other arguments are plausible host buffers and valid sizes."""
import ctypes

import pytest

from vdf_b200 import _lib

ERR_ARG = -1
BAD_IDS = (7, -1)

_buf = ctypes.create_string_buffer(1 << 16)   # host memory behind every pointer argument
_idx = (ctypes.c_uint64 * 1)(0)
_round = _lib.ROUND_FN(lambda *a: 0)


def _handle():
    return ctypes.byref(ctypes.c_void_p())


# name -> (message prefix, what is unknown, call with the id)
CALLS = {
    "gens_create": ("gens", "curve", lambda lib, i: lib.vdfgpu_gens_create(i, _buf, 4, 0, 0, _handle())),
    "gens_progression": ("gens", "curve", lambda lib, i: lib.vdfgpu_gens_progression(i, _buf, _buf, 4, 0, 0, _handle())),
    "point_sum": ("point_sum", "curve", lambda lib, i: lib.vdfgpu_point_sum(i, _buf, 2, _buf)),
    "point_sum_dev": ("point_sum_dev", "curve", lambda lib, i: lib.vdfgpu_point_sum_dev(i, _buf, 2, _buf)),
    "point_normalise_host": ("point_normalise_host", "curve", lambda lib, i: lib.vdfgpu_point_normalise_host(i, _buf, 1)),
    "r1cs_create": ("r1cs_create", "field", lambda lib, i: lib.vdfgpu_r1cs_create(
        i, 1, 1, 0, _idx, _idx, _buf, 1, _idx, _idx, _buf, 1, _idx, _idx, _buf, 1, _handle())),
    "fold": ("fold", "field", lambda lib, i: lib.vdfgpu_fold(i, _buf, _buf, 2, _buf, _buf, 2, _buf)),
    "fold_dev": ("fold_dev", "field", lambda lib, i: lib.vdfgpu_fold_dev(i, _buf, _buf, 2, _buf, _buf, 2, _buf)),
    "witness_bank_create": ("witness_bank_create", "field",
                            lambda lib, i: lib.vdfgpu_witness_bank_create(i, _buf, 1, 2, _handle())),
    "eq_evals": ("eq_evals", "field", lambda lib, i: lib.vdfgpu_eq_evals(i, _buf, 3, _buf)),
    "eq_evals_dev": ("eq_evals", "field", lambda lib, i: lib.vdfgpu_eq_evals_dev(i, _buf, 3, _buf)),
    "sumcheck_cubic": ("sumcheck", "field", lambda lib, i: lib.vdfgpu_sumcheck_cubic(
        i, _buf, _buf, _buf, _buf, 3, _round, None, _buf)),
    "sumcheck_cubic_dev": ("sumcheck", "field", lambda lib, i: lib.vdfgpu_sumcheck_cubic_dev(
        i, _buf, _buf, _buf, _buf, 3, _round, None, _buf)),
    "sumcheck_quad": ("sumcheck", "field", lambda lib, i: lib.vdfgpu_sumcheck_quad(i, _buf, _buf, 3, _round, None, _buf)),
    "sumcheck_quad_dev": ("sumcheck", "field",
                          lambda lib, i: lib.vdfgpu_sumcheck_quad_dev(i, _buf, _buf, 3, _round, None, _buf)),
    "poly_evaluate": ("poly_evaluate", "field", lambda lib, i: lib.vdfgpu_poly_evaluate(i, _buf, _buf, 3, _buf)),
    "poly_evaluate_dev": ("poly_evaluate", "field", lambda lib, i: lib.vdfgpu_poly_evaluate_dev(i, _buf, _buf, 3, _buf)),
    "vec_lincomb": ("vec_lincomb", "field", lambda lib, i: lib.vdfgpu_vec_lincomb(i, _buf, _buf, 2, _buf, _buf, _buf)),
    "inner_product": ("inner_product", "field", lambda lib, i: lib.vdfgpu_inner_product(i, _buf, _buf, 2, _buf)),
    "points_lincomb": ("points_lincomb", "curve",
                       lambda lib, i: lib.vdfgpu_points_lincomb(i, _buf, _buf, 2, _buf, _buf, _buf)),
    "minroot_check_batch": ("minroot_check", "field",
                            lambda lib, i: lib.vdfgpu_minroot_check_batch(i, _buf, _buf, None, 1, 2, _buf)),
    "minroot_check_batch_dev": ("minroot_check", "field",
                                lambda lib, i: lib.vdfgpu_minroot_check_batch_dev(i, _buf, _buf, None, 1, 2, _buf)),
    "minroot_inverse_eval_batch": ("minroot_inverse_eval", "field",
                                   lambda lib, i: lib.vdfgpu_minroot_inverse_eval_batch(i, _buf, 1, 2, _buf)),
    "minroot_witness_batch": ("minroot_witness", "field",
                              lambda lib, i: lib.vdfgpu_minroot_witness_batch(i, _buf, 1, 2, _buf)),
    "field_mul_batch": ("field_mul_batch", "field", lambda lib, i: lib.vdfgpu_field_mul_batch(i, _buf, _buf, 2, 1, _buf)),
}


def test_every_id_taking_entry_point_is_covered():
    assert len(CALLS) == 25
    lib = _lib.load()
    for name in CALLS:
        assert hasattr(lib, "vdfgpu_" + name)


@pytest.mark.parametrize("bad_id", BAD_IDS)
@pytest.mark.parametrize("name", sorted(CALLS))
def test_unknown_id_is_an_argument_error(name, bad_id):
    lib = _lib.load()
    prefix, what, call = CALLS[name]
    launches = lib.vdfgpu_launch_count()
    rc = call(lib, bad_id)
    assert (rc, lib.vdfgpu_last_error().decode()) == (ERR_ARG, f"{prefix}: unknown {what}")
    assert lib.vdfgpu_launch_count() == launches
