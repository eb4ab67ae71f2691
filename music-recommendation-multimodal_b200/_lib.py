"""ctypes binding of libtt_b200.so — the only door to the device code.

There is deliberately no fallback: if the shared library is missing or a launcher
returns non-zero, a TTError is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_uint32, c_uint64, c_void_p
from pathlib import Path

# TT_B200_LIB: load another build of the same ABI (A/B timing of kernel variants on one GPU box)
_LIB_PATH = Path(os.environ.get("TT_B200_LIB") or Path(__file__).resolve().parent / "libtt_b200.so")
_lib = None


class TTError(RuntimeError):
    pass


class GemmArgs(ctypes.Structure):
    """Mirror of ``tt_gemm_args`` (include/tt_b200.h)."""

    _fields_ = [
        ("A", c_void_p), ("B", c_void_p),
        ("lda", c_int32), ("ldb", c_int32),
        ("a_mn", c_int32), ("b_mn", c_int32),
        ("M", c_int32), ("N", c_int32), ("K", c_int32),
        ("alpha", c_float),
        ("bias", c_void_p),
        ("relu", c_int32),
        ("drop_p", c_float),
        ("drop_seed", c_uint64),
        ("drop_seed_dev", c_void_p),
        ("drop_site", c_uint32),
        ("gate", c_void_p),
        ("ld_gate", c_int32),
        ("gate_scale", c_float),
        ("residual", c_void_p),
        ("ld_res", c_int32),
        ("out_f32", c_void_p),
        ("ld_f32", c_int32),
        ("out_bf16", c_void_p),
        ("ld_bf16", c_int32),
        ("accumulate", c_int32),
        ("k_splits", c_int32),
        ("block_n", c_int32),
        ("a_colsum", c_void_p),
    ]


def _declare(l):
    l.tt_last_error.restype = c_char_p
    l.tt_last_error.argtypes = []
    l.tt_version.restype = c_int32
    l.tt_num_sms.restype = c_int32
    l.tt_gemm_bf16.restype = c_int32
    l.tt_gemm_bf16.argtypes = [ctypes.POINTER(GemmArgs), c_void_p]
    l.tt_attn_causal_fwd.restype = c_int32
    l.tt_attn_causal_fwd.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float,
                                     c_uint64, c_void_p, c_uint32, c_void_p]
    l.tt_attn_causal_bwd.restype = c_int32
    l.tt_attn_causal_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                     c_int32, c_float, c_uint64, c_void_p, c_uint32, c_void_p]


def lib():
    """Load (once) and return the shared library; fail loudly if it is not built."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise TTError(
                f"{_LIB_PATH} not found: build it with `python __graft_entry__.py` "
                "(there is no CPU or PyTorch fallback for the device path)")
        l = ctypes.CDLL(str(_LIB_PATH))
        _declare(l)
        _lib = l
    return _lib


#: number of kernels launched through the C ABI by this process (every launcher = 1 kernel)
launch_count = 0


def check(rc: int, what: str) -> None:
    global launch_count
    launch_count += 1
    if rc != 0:
        msg = lib().tt_last_error().decode("utf-8", "replace")
        raise TTError(f"{what} failed (code {rc}): {msg}")


class ChainArgs(ctypes.Structure):
    """Mirror of ``tt_chain_args``."""

    _fields_ = [
        ("x", c_void_p), ("rows", c_int32), ("width", c_int32),
        ("ln_w", c_void_p), ("ln_b", c_void_p), ("ln_eps", c_float),
        ("relu", c_int32),
        ("drop_p", c_float), ("drop_seed", c_uint64), ("drop_seed_dev", c_void_p), ("drop_site", c_uint32),
        ("l2norm", c_int32), ("l2_eps", c_float),
        ("out_f32", c_void_p), ("out_bf16", c_void_p),
        ("dout", c_void_p), ("resid", c_void_p), ("dx_f32", c_void_p), ("dx_bf16", c_void_p),
        ("drop2_p", c_float), ("drop2_site", c_uint32),
        ("dgamma", c_void_p), ("dbeta", c_void_p), ("dx_colsum", c_void_p),
        ("resid_rows", c_void_p), ("resid_last_idx", c_void_p), ("resid_seq_len", c_int32),
        ("dout_bf16", c_void_p),
    ]


class BnArgs(ctypes.Structure):
    """Mirror of ``tt_bn_args``."""

    _fields_ = [
        ("y", c_void_p), ("B", c_int32), ("C", c_int32),
        ("w", c_void_p), ("b", c_void_p),
        ("running_mean", c_void_p), ("running_var", c_void_p), ("num_batches_tracked", c_void_p),
        ("training", c_int32), ("momentum", c_float), ("eps", c_float),
        ("drop_p", c_float), ("drop_seed", c_uint64), ("drop_seed_dev", c_void_p), ("drop_site", c_uint32),
        ("save_mean", c_void_p), ("save_rstd", c_void_p), ("out_bf16", c_void_p),
        ("dout", c_void_p), ("dy_bf16", c_void_p), ("dgamma", c_void_p), ("dbeta", c_void_p),
        ("dy_colsum", c_void_p),
    ]


class TopkPlan(ctypes.Structure):
    """Mirror of ``tt_topk_plan``."""

    _fields_ = [("U", c_int32), ("N", c_int32), ("kprime", c_int32), ("cap", c_int32),
                ("n_ut", c_int32), ("n_ranges", c_int32), ("tiles_per_range", c_int32),
                ("sample_stride", c_int32), ("sample_rank", c_int32), ("sample_tiles", c_int32),
                ("cand_bytes", ctypes.c_int64), ("cnt_bytes", ctypes.c_int64), ("thr_bytes", ctypes.c_int64),
                ("smax_bytes", ctypes.c_int64)]


_I64 = ctypes.c_int64


class SymmTeam(ctypes.Structure):
    """Mirror of ``tt_symm_team``."""

    _fields_ = [("rank", c_int32), ("world", c_int32), ("bufs", c_void_p * 16), ("multicast", c_void_p),
                ("ctrl_offset", ctypes.c_int64)]


class SymmSegment(ctypes.Structure):
    """Mirror of ``tt_symm_segment``."""

    _fields_ = [("src", c_void_p), ("dst_offset", ctypes.c_int64), ("nbytes", ctypes.c_int64)]


_SIGNATURES = {
    "tt_symm_ctrl_bytes": [],
    "tt_symm_allgather": [ctypes.POINTER(SymmTeam), ctypes.POINTER(SymmSegment), c_int32, c_int32, c_void_p],
    "tt_dp_adamw_step": [ctypes.POINTER(SymmTeam), _I64, _I64, _I64, _I64, _I64, c_void_p, c_void_p, c_float, c_float,
                         c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, _I64, c_void_p],
    "tt_symm_barrier": [ctypes.POINTER(SymmTeam), c_void_p],
    "tt_gather_rows": [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p],
    "tt_scatter_rows_add": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p],
    "tt_attn_lastq_fwd": [c_void_p] * 5 + [c_int32, c_int32, c_int32, c_float, c_uint64, c_void_p, c_uint32, c_void_p],
    "tt_attn_lastq_bwd": [c_void_p] * 8 + [c_int32, c_int32, c_int32, c_float, c_uint64, c_void_p, c_uint32, c_void_p],
    "tt_topk_plan_make": [c_int32, c_int32, c_int32, ctypes.POINTER(TopkPlan)],
    "tt_score_topk": [c_void_p, c_void_p, c_int32, ctypes.POINTER(TopkPlan), c_void_p, c_void_p, c_void_p, c_void_p,
                      c_int32, c_void_p],
    "tt_users_prepare": [c_void_p, c_void_p, c_int32, c_void_p, c_void_p],
    "tt_topk_finalize": [ctypes.POINTER(TopkPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                         c_float, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_topk_finalize_bounded": [ctypes.POINTER(TopkPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                 c_float, c_void_p, c_float, c_float, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                                 c_int32, c_void_p],
    "tt_topk_merge_packed": [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                             c_void_p],
    "tt_topk_merge": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p],
    "tt_topk_merge_lists": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p],
    "tt_exact_topk": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_exclusions_build": [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p,
                            c_void_p],
    "tt_score_topk_excl": [c_void_p, c_void_p, c_int32, ctypes.POINTER(TopkPlan), c_void_p, c_void_p, c_void_p,
                           c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p],
    "tt_exact_topk_excl": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p],
    "tt_mmr_select": [c_void_p, c_void_p, c_int32, c_int32, c_int32, ctypes.c_double, ctypes.c_double, c_int32,
                      c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p],
    "tt_mmr_gather_rows": [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p],
    "tt_rank_metrics": [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                        c_void_p],
    "tt_cast_bf16": [c_void_p, c_void_p, _I64, c_void_p],
    "tt_last_index": [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p],
    "tt_embed_ln_fwd": [c_void_p] * 7 + [c_int32, c_int32, c_float, c_uint64, c_void_p, c_uint32,
                                         c_void_p, c_void_p, c_void_p],
    "tt_embed_ln_fwd_pos": [c_void_p] * 8 + [c_int32, c_void_p, c_void_p, c_void_p],
    "tt_session_attn": [c_void_p] * 5 + [c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p],
    "tt_embed_ln_bwd": [c_void_p] * 6 + [c_int32, c_int32, c_float, c_uint64, c_void_p, c_uint32,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_embed_ln_bwd_det": [c_void_p] * 6 + [c_int32, c_int32, c_float, c_uint64, c_void_p, c_uint32,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_rows_scatter_add_i64": [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p],
    "tt_chain_fwd": [ctypes.POINTER(ChainArgs), c_void_p],
    "tt_chain_bwd": [ctypes.POINTER(ChainArgs), c_void_p],
    "tt_gather_cat_fwd": [c_void_p] * 6 + [c_int32, c_int32, c_void_p, c_void_p],
    "tt_gather_cat_bwd": [c_void_p] * 4 + [c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_concat4_bf16": [c_void_p] * 4 + [c_int32, c_int32, c_void_p, c_void_p],
    "tt_bn_relu_fwd": [ctypes.POINTER(BnArgs), c_void_p],
    "tt_bn_relu_bwd": [ctypes.POINTER(BnArgs), c_void_p],
    "tt_adamw_step": [c_void_p] * 4 + [_I64, c_float, c_float, c_float, c_float, c_float, c_float, c_void_p, c_void_p,
                                       _I64, _I64, c_int32, c_void_p],
    "tt_ids_dedup": [c_void_p, c_int32, _I64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_rows_gather": [ctypes.POINTER(SymmTeam), _I64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p],
    "tt_rows_scatter_add": [ctypes.POINTER(SymmTeam), _I64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p],
    "tt_step_counters_advance": [c_void_p, c_void_p, c_void_p],
    "tt_infonce_rows": [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                        c_void_p],
    "tt_infonce_grad": [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_float, c_void_p,
                        c_int32, c_void_p],
    "tt_infonce_loss": [c_void_p] * 4 + [c_int32, c_float, c_void_p, c_void_p],
    "tt_infonce_rows_off": [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                            c_void_p, c_void_p],
    "tt_infonce_grad_off": [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_float, c_void_p,
                            c_void_p, c_void_p, c_int32, c_void_p],
    "tt_logq_table_gather": [c_void_p, c_int32, c_void_p, _I64, c_float, c_void_p, c_void_p],
    "tt_logq_stream_update": [c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_float, c_float,
                              c_void_p, c_void_p],
    "tt_inbatch_recall": [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p],
    "tt_index_rows": [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, _I64, c_void_p, c_void_p, c_void_p],
    "tt_score_topk_live": [c_void_p, c_void_p, c_int32, ctypes.POINTER(TopkPlan), c_void_p, c_void_p, c_void_p,
                           c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p],
    "tt_exact_topk_live": [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p, c_void_p],
    "tt_index_rows_live": [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, _I64, _I64, c_int32, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p],
    "tt_catalog_retire": [c_void_p, c_int32, _I64, _I64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p],
}

_declare_base = _declare


def _declare(l):  # noqa: F811 - extends the base declarations with the row-wise / loss entry points
    _declare_base(l)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(l, name)
        fn.restype = c_int32
        fn.argtypes = argtypes


#: every symbol include/tt_b200.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = ["tt_last_error", "tt_version", "tt_num_sms", "tt_gemm_bf16", "tt_attn_causal_fwd",
                    "tt_attn_causal_bwd", *sorted(_SIGNATURES)]
