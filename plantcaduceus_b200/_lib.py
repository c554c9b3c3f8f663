"""ctypes binding of libpcad.so (C ABI in include/pcad.h).

The library is built in-tree (plantcaduceus_b200/libpcad.so) by ``__graft_entry__.build()`` /
``make -C plantcaduceus_b200/csrc``.  There is no fallback: if the library is missing or cannot be
loaded, importing the engine raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libpcad.so"

PCAD_BF16, PCAD_F32, PCAD_F16 = 0, 1, 2
STAGES = ("embed", "norm", "in_proj", "conv", "x_proj", "dt_proj", "scan", "out_proj", "head", "misc", "gnorm")
PCAD_MIXER_MAMBA1, PCAD_MIXER_MAMBA2 = 0, 1
ABI_VERSION = 3

EXPORTS = (
    "pcad_abi_version", "pcad_create", "pcad_destroy", "pcad_last_error", "pcad_set_weight", "pcad_finalize",
    "pcad_set_tokenizer", "pcad_take_id_error", "pcad_hidden_at", "pcad_forward",
    "pcad_forward_taps", "pcad_hidden_at_layers", "pcad_hidden_mean_at_layers", "pcad_score_masked", "pcad_score_masked_at", "pcad_score_windows_host", "pcad_score_windows_dev", "pcad_extract_windows", "pcad_tokenize",
    "pcad_workspace_bytes", "pcad_set_profiling", "pcad_get_profile", "pcad_launch_count",
    "pcad_graph_replays",
    "pcad_op_linear", "pcad_op_linear_residual", "pcad_op_linear_residual_tap", "pcad_op_linear_rowscale", "pcad_op_sumsq_parts",
    "pcad_op_add_rmsnorm", "pcad_op_conv_silu", "pcad_op_biscan", "pcad_op_biscan_segmented", "pcad_op_biscan_ex",
    "pcad_op_biscan_dt",
    "pcad_op_ssd_scan", "pcad_op_gated_norm_sum", "pcad_op_hidden_mean",
)


class PcadConfig(C.Structure):
    _fields_ = [
        ("d_model", C.c_int32), ("n_layer", C.c_int32), ("vocab_size", C.c_int32), ("d_state", C.c_int32),
        ("d_conv", C.c_int32), ("expand", C.c_int32), ("dt_rank", C.c_int32), ("norm_eps", C.c_float),
        ("residual_in_fp32", C.c_int32), ("dtype", C.c_int32), ("complement_map", C.c_int32 * 16),
        ("mixer", C.c_int32), ("headdim", C.c_int32), ("ngroups", C.c_int32),
    ]


class PcadError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Load libpcad.so and declare signatures. Raises PcadError if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PCAD_LIB", str(LIB_PATH))
    if not os.path.exists(path):
        raise PcadError(
            f"{path} not found: the CUDA extension is not built. Run `python -c 'import __graft_entry__ as g; "
            f"g.build()'` or `make -C plantcaduceus_b200/csrc`. There is no CPU fallback.")
    lib = C.CDLL(path)
    vp, i32, i64, f32p = C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_float)
    lib.pcad_abi_version.restype = i32
    lib.pcad_create.argtypes = [C.POINTER(PcadConfig), i32, C.POINTER(vp)]
    lib.pcad_destroy.argtypes = [vp]
    lib.pcad_destroy.restype = None
    lib.pcad_last_error.argtypes = [vp]
    lib.pcad_last_error.restype = C.c_char_p
    lib.pcad_set_weight.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32, i32]
    lib.pcad_finalize.argtypes = [vp]
    lib.pcad_set_tokenizer.argtypes = [vp, C.POINTER(C.c_uint8), i32, C.POINTER(C.c_int32)]
    lib.pcad_take_id_error.argtypes = [vp, vp, i32]
    lib.pcad_hidden_at.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.pcad_forward.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.pcad_forward_taps.argtypes = [vp, vp, i32, i32, vp, i32, C.POINTER(C.c_int32), C.POINTER(vp), vp]
    lib.pcad_hidden_at_layers.argtypes = [vp, vp, vp, i32, i32, i32, i32, C.POINTER(C.c_int32), vp, vp]
    lib.pcad_hidden_mean_at_layers.argtypes = [vp, vp, vp, i32, i32, i32, C.POINTER(C.c_int32), vp, vp]
    lib.pcad_score_masked.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.pcad_score_masked_at.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    lib.pcad_score_windows_host.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    lib.pcad_score_windows_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    lib.pcad_extract_windows.argtypes = [vp, vp, i64, vp, i32, i32, i32, vp, vp]
    lib.pcad_tokenize.argtypes = [vp, vp, i64, vp, vp]
    lib.pcad_workspace_bytes.argtypes = [vp, i32, i32, C.POINTER(C.c_size_t)]
    lib.pcad_set_profiling.argtypes = [vp, i32]
    lib.pcad_get_profile.argtypes = [vp, f32p, C.POINTER(i64)]
    lib.pcad_launch_count.argtypes = [vp]
    lib.pcad_launch_count.restype = i64
    lib.pcad_graph_replays.argtypes = [vp]
    lib.pcad_graph_replays.restype = i64
    lib.pcad_op_linear.argtypes = [vp, vp, vp, i64, i32, i32, i64, i64, i64, i32, vp]
    lib.pcad_op_linear_residual.argtypes = [vp, vp, vp, vp, vp, i64, i32, i32, i64, i64, i64, i32, vp]
    lib.pcad_op_linear_residual_tap.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, i32, i64, i64, i64, i64, i32, vp]
    lib.pcad_op_linear_rowscale.argtypes = [vp, vp, vp, i32, C.c_float, vp, i64, i32, i32, i64, i64, i64, i32, vp]
    lib.pcad_op_sumsq_parts.argtypes = [i32]
    lib.pcad_op_add_rmsnorm.argtypes = [vp, vp, vp, vp, vp, i64, i32, C.c_float, i32, i32, vp]
    lib.pcad_op_conv_silu.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.pcad_op_biscan_dt.argtypes = [vp, vp, vp, vp, i64, i32, vp, vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.pcad_op_biscan.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp,
                                   i32, i32, i32, i32, vp]
    lib.pcad_op_biscan_segmented.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp,
                                             i32, i32, i32, i32, vp, vp, i32, vp]
    lib.pcad_op_biscan_ex.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp,
                                      i32, i32, i32, i32, vp, vp, vp, i32, i32, vp]
    lib.pcad_op_ssd_scan.argtypes = [vp, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.pcad_op_gated_norm_sum.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, i32, C.c_float, i32, vp]
    lib.pcad_op_hidden_mean.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
    for name in EXPORTS:
        getattr(lib, name)  # AttributeError here means header and library disagree
    if lib.pcad_abi_version() != ABI_VERSION:
        raise PcadError(f"{path} has ABI version {lib.pcad_abi_version()}, this package needs {ABI_VERSION}: rebuild the extension")
    _lib = lib
    return lib


def check(rc: int, handle=None) -> None:
    if rc != 0:
        msg = load().pcad_last_error(handle)
        raise PcadError(f"libpcad error {rc}: {msg.decode() if msg else '?'}")
