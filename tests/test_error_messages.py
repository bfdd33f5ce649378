"""CPU-side checks of the library's error path: encoder, GEMM and Pareto entry points reject bad arguments with the
documented code before anything is launched, and leave a message naming themselves in mtfjsp_last_error -- also when an
env call failed before them on the same thread."""
import ctypes as C
import importlib

import pytest

E_ARG, E_STATE = -1, -3
P = C.c_void_p(0x10000)   # stands for a device operand: 16-byte aligned, never dereferenced on the host
P4 = C.c_void_p(0x10004)  # 4-byte aligned only


@pytest.fixture(scope="module")
def lib():
    mod = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
    mod.build()
    return mod.lib()


# (entry point, arguments, code): a NULL operand, a misaligned pointer, K = 130, envs_per_group not dividing B, S < 0
CASES = [
    ("mtfjsp_enc_linear_tf32", (None, 4096, 128, P, None, None, None, 0, P, None, None), E_ARG),
    ("mtfjsp_enc_linear_tf32", (P, 4096, 130, P, None, None, None, 0, P, None, None), E_ARG),
    ("mtfjsp_enc_linear_tf32", (P4, 4096, 128, P, None, None, None, 0, P, None, None), E_ARG),
    ("mtfjsp_enc_linear_tf32_grouped", (P, 6, 36, 128, P, None, P, P, 1, 4, P, P, None), E_ARG),
    ("mtfjsp_enc_aggregate_linear_tf32_grouped", (P, 6, 200, P, P, P, None, P, P, 1, 2, P, P, None), E_STATE),
    ("mtfjsp_enc_head_tf32", (P, None, 4, 36, 0, None, None, 0, P, P4, 1, P, None, P, None, P, None), E_ARG),
    ("mtfjsp_enc_head_tf32_grouped", (P, None, 6, 36, 0, P, P, 1, 4, P, P, 1, P, None, P, None, P, None), E_ARG),
    ("mtfjsp_enc_gat_trunk_tf32", (P, P, P, P, None, P, P, P, None, 128, None), E_ARG),
    ("mtfjsp_enc_wgrad_tf32", (P, P, 4096, 130, P, P, P, None), E_ARG),
    ("mtfjsp_enc_aggregate", (P, P4, P, P, 4, 36, 128, None, None, 0, None), E_ARG),
    ("mtfjsp_enc_aggregate_grouped", (P, P, P, P, 6, 36, 128, P, P, 1, 4, None), E_ARG),
    ("mtfjsp_enc_aggregate_bwd", (None, P, P, P, P, 4, 36, 128, None), E_ARG),
    ("mtfjsp_enc_bn_fwd", (P, P, P, 1e-5, 0, 36, 128, 1, P, P, P, P, None), E_ARG),
    ("mtfjsp_enc_gat_attend", (P, P, P4, P, 128, 0, None), E_ARG),
    ("mtfjsp_gae4", (P, P, P, None, P, P, 8, 4, 0.99, 0.98, None), E_ARG),
    ("mtfjsp_pareto_filter", (P, P, -1, 8, P, None), E_ARG),
    ("mtfjsp_hypervolume3", (P, P, -1, P, P, None), E_ARG),
]


@pytest.mark.parametrize("name,args,code", CASES, ids=["%s-%d" % (c[0], i) for i, c in enumerate(CASES)])
def test_bad_arguments_name_the_entry_point(lib, name, args, code):
    assert getattr(lib, name)(*args) == code
    assert lib.mtfjsp_last_error().decode().startswith(name + ":")


def test_last_error_is_the_latest_failure(lib):
    assert lib.mtfjsp_step(None, None, None, None, None, None, None, None) == E_ARG
    assert lib.mtfjsp_last_error().startswith(b"mtfjsp_step:")
    assert lib.mtfjsp_enc_linear_tf32(P, 4096, 130, P, None, None, None, 0, P, None, None) == E_ARG
    assert lib.mtfjsp_last_error().startswith(b"mtfjsp_enc_linear_tf32:")
    assert lib.mtfjsp_pareto_filter(None, P, 1, 8, P, None) == E_ARG
    assert lib.mtfjsp_last_error().startswith(b"mtfjsp_pareto_filter:")
