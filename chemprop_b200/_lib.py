"""ctypes binding of libdmpnn_sm100.so (the C ABI declared in include/dmpnn.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the
product path raises.  (`oracle/` is test infrastructure and is never imported from here.)
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("DMPNN_LIB", _PKG / "lib" / "libdmpnn_sm100.so"))

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_LEAKYRELU, ACT_TANH, ACT_ELU = 0, 1, 2, 3, 4
SCALE_NONE, SCALE_DIV_CONST, SCALE_INV_COUNT = 0, 1, 2
META_N_TILES, META_FLAGS, META_MAX_INDEG, META_MAX_TILE_ROWS, META_MAX_TILE_ATOMS, META_WORDS = 0, 1, 2, 3, 4, 8
FLAG_REV_INVOLUTION, FLAG_BATCH_SORTED, FLAG_INDEX_IN_RANGE = 1, 2, 4

_vp, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/dmpnn.h one to one
SIGNATURES = {
    "dmpnn_version": (C.c_int, []),
    "dmpnn_last_error": (C.c_char_p, []),
    "dmpnn_device_ok": (C.c_int, []),
    "dmpnn_launch_count": (C.c_longlong, []),
    "dmpnn_collate_host": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_collate_host_compact": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_scale_mask": (C.c_int, [_vp, _vp, _vp, _i32, _i64, _f32, _vp]),
    "dmpnn_tile_pack_order": (C.c_int, [_i64, _vp, _vp, _vp]),
    "dmpnn_batch_meta_host": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "dmpnn_dataset_batch_meta_host": (C.c_int, [_i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_dataset_gather_host": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64]
                                  + [_vp] * 10 + [_i32]),
    "dmpnn_dataset_gather": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64,
                                       _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "dmpnn_layout_workspace_bytes": (C.c_int, [_i64, _i64, _i64, C.POINTER(_sz)]),
    "dmpnn_layout_build": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64] + [_vp] * 12 + [_vp, _vp]),
    "dmpnn_sorted_index_to_ptr": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp]),
    "dmpnn_linear_fwd": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i64, _vp,
                                   _vp, _i32, _i64, _i32, _f32, _vp, _i32, _i64, _i64, _i64, _i64, _vp]),
    "dmpnn_linear_wgrad_workspace_bytes": (C.c_int, [_i64, _i64, _i64, C.POINTER(_sz)]),
    "dmpnn_linear_wgrad": (C.c_int, [_vp, _i32, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i32, _i64, _vp, _i64,
                                     _vp, _i64, _vp, _i32, _i64, _i64, _vp, _vp]),
    "dmpnn_segment_sum": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _i64, _i64, _i32, _f32, _i32, _f32,
                                    _vp, _i32, _i64, _i64, _vp]),
    "dmpnn_segment_bcast": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _i64, _i64, _i64, _i32, _f32, _vp, _i32, _i64, _vp]),
    "dmpnn_bond_message": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _i64, _i64, _i32, _f32, _i32, _vp, _i32, _i64, _vp]),
    "dmpnn_bond_message_bwd_masked": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _i64, _i64, _vp, _i64, _i32, _f32, _vp, _i64, _vp]),
    "dmpnn_sum_act_bwd": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _f32, _vp, _i32, _i64, _i64, _i64, _vp]),
    "dmpnn_rev_average": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _i64, _i32, _f32, _vp, _i32, _i64, _vp]),
    "dmpnn_act_bwd": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _i32, _i64, _i32, _i32, _f32, _vp, _i32, _i64,
                                _vp, _i32, _i64, _i64, _i64, _vp]),
    "dmpnn_bond_step_bwd_fused_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _f32,
                                                 _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_work_table_build": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_concat_bf16": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "dmpnn_concat_f32": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "dmpnn_pack_weight_tc_bytes": (C.c_int, [_i64, _i64, C.POINTER(_sz)]),
    "dmpnn_pack_weight_tc": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _vp, _vp]),
    "dmpnn_linear_tc_bf16": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _i32, _f32, _vp, _i64, _vp]),
    "dmpnn_tiles_workspace_bytes": (C.c_int, [_i64, C.POINTER(_sz)]),
    "dmpnn_tiles_build": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "dmpnn_atom_step_fused_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _f32,
                                             _i32, _vp, _vp]),
    "dmpnn_atom_step_bwd_fused_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _f32,
                                                 _i32, _vp, _vp, _vp, _vp]),
    "dmpnn_wgrad_tc_workspace_bytes": (C.c_int, [_i64, _i64, C.POINTER(_sz)]),
    "dmpnn_wgrad_tc_bf16": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _vp]),
    "dmpnn_wgrad_tc_multi_bf16": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _vp]),
    "dmpnn_column_sum": (C.c_int, [_vp, _i32, _i64, _i64, _i64, _vp, _i32, _vp, _vp]),
    "dmpnn_set_trace_buffer": (C.c_int, [_vp, _i64]),
    "dmpnn_pack_weight_bf16_bytes": (C.c_int, [_i64, _i64, C.POINTER(_sz)]),
    "dmpnn_pack_weight_bf16": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "dmpnn_bond_step_fused_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp,
                                             _i64, _i32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _vp]),
    "dmpnn_dropout_bits": (C.c_int, [_vp, _i64, _i64, _f32, C.c_uint64, C.c_uint64, _vp]),
    "dmpnn_pack_weight_x3_bytes": (C.c_int, [_i64, _i64, C.POINTER(_sz)]),
    "dmpnn_pack_weight_x3": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _vp, _vp]),
    "dmpnn_linear_x3": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _i32, _f32, _vp, _i64, _i64, _vp]),
    "dmpnn_wgrad_x3_workspace_bytes": (C.c_int, [_i64, _i64, C.POINTER(_sz)]),
    "dmpnn_wgrad_x3": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _vp]),
    "dmpnn_bn_train_fwd": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "dmpnn_bn_bwd": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "dmpnn_mse_loss": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _vp, _vp, _i64, _vp]),
    "dmpnn_bce_loss": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _vp, _vp, _i64, _vp]),
    "dmpnn_ce_loss": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp]),
    "dmpnn_class_probs": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp]),
    "dmpnn_class_probs_bwd": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp]),
}


class DmpnnError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built -- no fallback."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise DmpnnError(
                f"{LIB_PATH} not found: build it with `python -m chemprop_b200.build` "
                "(or __graft_entry__.build()); the engine has no CPU / PyTorch fallback."
            )
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().dmpnn_last_error().decode(errors="replace")
        raise DmpnnError(f"{what} failed (rc={rc}): {msg}")
