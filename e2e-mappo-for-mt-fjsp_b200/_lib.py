"""Loader (and in-tree builder) of the C-ABI shared library ``libmtfjsp_b200.so``.

The product path fails loudly when the CUDA extension is missing or cannot be loaded: there is no CPU
fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(_HERE, "csrc")
# MTFJSP_LIB: load another build of the same library (A/B runs of kernel variants on the GPU box); default in-tree .so
LIB_PATH = os.environ.get("MTFJSP_LIB") or os.path.join(_HERE, "libmtfjsp_b200.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "mtfjsp.h")
SOURCES = ["mtfjsp_env.cu", "mtfjsp_encoder.cu", "mtfjsp_gemm.cu", "mtfjsp_pareto.cu", "mtfjsp_evolve.cu",
           "mtfjsp_mcts.cu", "mtfjsp_tabu.cu", "mtfjsp_anneal.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]
# the env kernels restate the reference's FP64 arithmetic operation by operation, and the hypervolume, the MCTS score and
# the annealer's acceptance test their numpy specifications: no FMA contraction there
EXTRA_FLAGS = {"mtfjsp_env.cu": ["-fmad=false"], "mtfjsp_pareto.cu": ["-fmad=false"], "mtfjsp_mcts.cu": ["-fmad=false"],
               "mtfjsp_anneal.cu": ["-fmad=false"]}


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    mt = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(SRC_DIR, s) for s in os.listdir(SRC_DIR)] + [HEADER, os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > mt for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc cross-compiles for sm_100a without a GPU; the .so stays in-tree so it travels to the GPU box.
    One object per source (compiled in parallel), then one shared library."""
    if force or _stale():
        obj_dir = os.path.join(_HERE, "build")
        os.makedirs(obj_dir, exist_ok=True)
        procs, objs = [], []
        for src in SOURCES:
            obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
            objs.append(obj)
            cmd = ["nvcc"] + NVCC_FLAGS + EXTRA_FLAGS.get(src, []) + (["-Xptxas", "-v"] if verbose else []) + \
                  ["-c", "-o", obj, os.path.join(SRC_DIR, src)]
            procs.append((cmd, subprocess.Popen(cmd)))
        for cmd, pr in procs:
            if pr.wait() != 0:
                raise subprocess.CalledProcessError(pr.returncode, cmd)
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs)
    return LIB_PATH


_lib = None

_VP, _I, _U64, _D = C.c_void_p, C.c_int, C.c_uint64, C.c_double

# every symbol include/mtfjsp.h declares: (argtypes, restype)
SIGNATURES = {
    "mtfjsp_create": ([C.POINTER(_VP), _I, _I, _I, _I, _I, _I], _I),
    "mtfjsp_destroy": ([_VP], _I),
    "mtfjsp_set_params": ([_VP, _D, _D, _D, _D, _D], _I),
    "mtfjsp_set_obs_incremental": ([_VP, _I], _I),
    "mtfjsp_load": ([_VP, _VP, _VP, _VP, _VP, _I, _VP], _I),
    "mtfjsp_scaler_init": ([_VP, _VP], _I),
    "mtfjsp_scaler_reset": ([_VP, _VP], _I),
    "mtfjsp_reset": ([_VP, _VP, _VP], _I),
    "mtfjsp_step": ([_VP] + [_VP] * 6 + [_VP], _I),
    "mtfjsp_obs": ([_VP] + [_VP] * 6 + [_I, _I, _VP], _I),
    "mtfjsp_step_obs": ([_VP] + [_VP] * 12 + [_I, _I, _VP], _I),
    "mtfjsp_mfea1": ([_VP, _VP, _VP, _VP, _I, _VP], _I),
    "mtfjsp_dense_adj": ([_VP, _VP, _I, _VP], _I),
    "mtfjsp_raw_adj": ([_VP, _VP, _VP], _I),
    "mtfjsp_generate_instances": ([_I, _I, _I, _I, _U64, _U64, _VP, _VP, _VP, _VP, _I, _VP], _I),
    "mtfjsp_costs": ([_VP, _VP, _VP, _VP], _I),
    "mtfjsp_export_state": ([_VP] + [_VP] * 4 + [_VP], _I),
    "mtfjsp_export_scaler": ([_VP] + [_VP] * 4 + [_VP], _I),
    "mtfjsp_gather": ([_VP, _VP, _VP, _VP], _I),
    "mtfjsp_peek": ([_VP, _VP, _VP, _I, _VP, _VP, _VP], _I),
    "mtfjsp_replay": ([_VP, _VP, _I, _VP, _I, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_replay_moves": ([_VP, _VP, _I, _VP, _VP, _I, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_complete": ([_VP, _VP, _I, _VP, _I, _I, _VP, _VP, _U64, _I, _VP, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_policy_random": ([_VP, _U64, _U64, _I, _VP, _VP, _VP], _I),
    "mtfjsp_random_step": ([_VP, _U64, _U64] + [_VP] * 14 + [_I, _I, _VP], _I),
    "mtfjsp_step_host": ([_VP] + [_VP] * 9 + [_I, _I, _VP], _I),
    "mtfjsp_step_host_packed": ([_VP] + [_VP] * 6 + [_I, _I, _VP], _I),
    "mtfjsp_host_record_bytes": ([_VP], _I),
    "mtfjsp_enc_aggregate": ([_VP, _VP, _VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _VP], _I),
    "mtfjsp_enc_ell_invert": ([_VP, _VP, C.c_int64, _I, _VP], _I),
    "mtfjsp_enc_bn_fwd": ([_VP, _VP, _VP, C.c_float, C.c_int64, C.c_int64, _I, _I, _VP, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_enc_bn_bwd": ([_VP, _VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int64, _I, _I, _VP, _VP, _VP], _I),
    "mtfjsp_enc_aggregate_bwd": ([_VP, _VP, _VP, _VP, _VP, C.c_int64, _I, _I, _VP], _I),
    "mtfjsp_enc_graph_mean": ([_VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _VP], _I),
    "mtfjsp_enc_linear_tf32": ([_VP, C.c_int64, _I, _VP, _VP, _VP, _VP, _I, _VP, _VP, _VP], _I),
    "mtfjsp_enc_gat_attend": ([_VP, _VP, _VP, _VP, C.c_int64, _I, _VP], _I),
    "mtfjsp_enc_gat_attend_bwd": ([_VP, _VP, _VP, _VP, _VP, _VP, C.c_int64, _I, _VP], _I),
    "mtfjsp_enc_gat_attend_bwd_blocks": ([C.c_int64], _I),
    "mtfjsp_enc_gat_trunk_tf32": ([_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int64, _VP], _I),
    "mtfjsp_enc_aggregate_linear_tf32": ([_VP, C.c_int64, _I, _VP, _VP, _VP, _VP, _VP, _VP, _I, _VP, _VP, _VP], _I),
    "mtfjsp_enc_select": ([_VP, _VP, _VP, C.c_float, _I, C.c_int64, _I, _U64, _VP, _I, _VP, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_enc_head_tf32": ([_VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _VP, _VP, C.c_int64, _VP, _VP, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_enc_wgrad_tf32": ([_VP, _VP, C.c_int64, _I, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_enc_wgrad_workspace_floats": ([_I], C.c_int64),
    "mtfjsp_enc_esa_mach_stats": ([_VP, _VP, C.c_int64, _I, _VP, _VP, _VP, _VP], _I),
    "mtfjsp_enc_esa_mach_stats_workspace_doubles": ([], C.c_int64),
    "mtfjsp_enc_esa_mach_fold": ([_VP, C.c_int64, _VP, _VP, _VP, _VP, C.c_float] + [_VP] * 7, _I),
    "mtfjsp_enc_esa_mach_head_tf32": ([_VP, _VP, C.c_int64, _I] + [_VP] * 8, _I),
    "mtfjsp_enc_bn_finalize": ([_VP, C.c_int64, _VP, _VP, C.c_float, _VP, _VP, _I, _VP], _I),
    "mtfjsp_enc_linear_tf32_grouped": ([_VP, C.c_int64, _I, _I, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP, _VP], _I),
    "mtfjsp_enc_aggregate_linear_tf32_grouped": ([_VP, C.c_int64, _I] + [_VP] * 6 + [_I, _I, _VP, _VP, _VP], _I),
    "mtfjsp_enc_aggregate_grouped": ([_VP, _VP, _VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _I, _VP], _I),
    "mtfjsp_enc_graph_mean_grouped": ([_VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _I, _VP], _I),
    "mtfjsp_enc_head_tf32_grouped": ([_VP, _VP, C.c_int64, _I, _I, _VP, _VP, _I, _I, _VP, _VP, C.c_int64] + [_VP] * 6, _I),
    "mtfjsp_enc_bn_finalize_grouped": ([_VP, C.c_int64, _I, _I, _VP, _VP, C.c_float, _VP, _VP, _I, _VP], _I),
    "mtfjsp_enc_gat_trunk_tf32_grouped": ([_VP] * 9 + [C.c_int64, _I, _VP], _I),
    "mtfjsp_gae4": ([_VP, _VP, _VP, _VP, _VP, _VP, _I, C.c_int64, C.c_float, C.c_float, _VP], _I),
    "mtfjsp_adv_normalize": ([_VP, _VP, C.c_double, _I, C.c_int64, _VP], _I),
    "mtfjsp_pareto_filter": ([_VP, _VP, _I, C.c_int64, _VP, _VP], _I),
    "mtfjsp_hypervolume3": ([_VP, _VP, _I, _VP, _VP, _VP], _I),
    "mtfjsp_pareto_rank": ([_VP, _VP, _I, C.c_int64, _VP, _VP], _I),
    "mtfjsp_offspring": ([_VP, _I, _I, _I, _VP, _I, _VP, _VP, _I, _U64, _D, _D, _VP, _VP], _I),
    "mtfjsp_mcts_select": ([_VP, _VP, _I, _I, _I, _VP, _I, _I, _I, _D] + [_VP] * 9, _I),
    "mtfjsp_mcts_backup": ([_I, _I, _I] + [_VP] * 8, _I),
    "mtfjsp_tabu_move": ([_I, _I, _I, _VP, C.c_int64, _VP, _VP, _VP, _I, _I, _I] + [_VP] * 10, _I),
    "mtfjsp_anneal_propose": ([_VP, _I, _I, _I, _I, _VP, _U64, _I, _VP, _VP], _I),
    "mtfjsp_anneal_step": ([_I, _I, _I, _I] + [_VP] * 5 + [_U64, _I, _I] + [_VP] * 9, _I),
    "mtfjsp_launch_overlap_error": ([_VP], _I),
    "mtfjsp_launch_count": ([_VP], C.c_int64),
    "mtfjsp_bytes_per_step": ([_VP, _I], C.c_int64),
    "mtfjsp_bytes_per_random_step": ([_VP, _I], C.c_int64),
    "mtfjsp_bytes_per_gather": ([_VP], C.c_int64),
    "mtfjsp_bytes_per_peek": ([_VP, _I], C.c_int64),
    "mtfjsp_random_step_is_fused": ([_VP], _I),
    "mtfjsp_last_error": ([], C.c_char_p),
    "mtfjsp_version": ([], C.c_char_p),
}


def lib():
    """The loaded C-ABI library.  Raises if it is absent: build it with ``__graft_entry__.build()``."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "CUDA extension %s is missing; run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(_lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.argtypes = argtypes
            fn.restype = restype
    return _lib


def _ptr(t):
    """A tensor's address for the C ABI; None passes NULL (optional operands; the library rejects a missing one)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    """The current torch stream of the current device, as the library's `void* stream`."""
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class MTFJSPError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc != 0:
        raise MTFJSPError("%s failed (%d): %s" % (what, rc, lib().mtfjsp_last_error().decode()))
