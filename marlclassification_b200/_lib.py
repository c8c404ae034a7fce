"""ctypes binding of libmarlc.so (the C ABI declared in include/marlc.h).

There is no fallback: if the library is missing or a call fails, a RuntimeError
is raised.  Nothing here imports the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _build

MAX_ACTIONS = 16
MAX_CNN_LAYERS = 6


class MarlcConfig(C.Structure):
    """Mirror of ``marlc_config`` (include/marlc.h)."""

    _fields_ = [
        ("na", C.c_int), ("nb", C.c_int), ("T", C.c_int), ("C", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("f", C.c_int), ("n_actions", C.c_int), ("actions", (C.c_int * 2) * MAX_ACTIONS),
        ("cnn_layers", C.c_int), ("cnn_cin", C.c_int * MAX_CNN_LAYERS), ("cnn_cout", C.c_int * MAX_CNN_LAYERS),
        ("cnn_groups", C.c_int * MAX_CNN_LAYERS),
        ("n_b", C.c_int), ("n_a", C.c_int), ("n_m", C.c_int), ("n_m_o", C.c_int), ("n_d", C.c_int),
        ("nl_b", C.c_int), ("nl_a", C.c_int), ("nb_class", C.c_int),
        ("gamma", C.c_float), ("use_tc", C.c_int), ("use_chains", C.c_int),
    ]


class MarlcPlan(C.Structure):
    """Mirror of ``marlc_plan`` (include/marlc.h): what the engine's launchers choose for its geometry."""

    _fields_ = [(name, C.c_int) for name in (
        "cnn_wide", "cnn_nw", "cnn_batches", "cnn_ctas", "cnn_passes", "cnn_tail",
        "lstm_tc", "lstm_hu", "lstm_bn", "lstm_fat", "lstm_ks", "lstm_ksplit", "lstm_tail_rows",
        "sweep_chained", "staged_step_pre", "staged_step_post", "staged_bwd_pre", "staged_bwd_post")]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


_P = C.c_void_p
_SIGS = {
    "marlc_version": (C.c_int, []),
    "marlc_selftest_fastdiv": (C.c_long, [C.c_int, C.c_int]),
    "marlc_last_error": (C.c_char_p, []),
    "marlc_patch_gather": (C.c_int, [_P, _P, _P] + [C.c_int] * 6 + [_P]),
    "marlc_patch_gather_backward": (C.c_int, [_P, _P, _P] + [C.c_int] * 6 + [_P]),
    "marlc_transition": (C.c_int, [_P, _P, _P] + [C.c_int] * 5 + [_P, _P, _P]),
    "marlc_normalized_positions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "marlc_images_u8_to_f32": (C.c_int, [_P, _P] + [C.c_int] * 5 + [_P]),
    "marlc_linear": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "marlc_ln_silu": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, _P]),
    "marlc_msg_mean": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "marlc_tc_gemm": (C.c_int, [_P, C.c_int64, C.c_int, _P, C.c_int64, C.c_int, _P, C.c_int64, _P, C.c_int64, C.c_int, _P,
                                _P, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "marlc_tc_lstm_pair": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.POINTER(_P)] * 9 + [C.c_int, _P]),
    "marlc_split_lo": (C.c_int, [_P, _P, C.c_int64, _P]),
    "marlc_tc_lstm_pair_presplit": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int] + [C.POINTER(_P)] * 13 + [_P]),
    "marlc_cnn_forward": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.c_int,
                                    C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P, _P, C.c_int, _P]),
    "marlc_engine_create": (C.c_int, [C.POINTER(MarlcConfig), C.POINTER(_P)]),
    "marlc_engine_destroy": (None, [_P]),
    "marlc_engine_plan": (C.c_int, [_P, C.POINTER(MarlcPlan)]),
    "marlc_engine_param_count": (C.c_int, [_P]),
    "marlc_engine_param_info": (C.c_int, [_P, C.c_int, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int),
                                          C.POINTER(C.c_int64)]),
    "marlc_engine_param_floats": (C.c_int64, [_P]),
    "marlc_engine_workspace_bytes": (C.c_size_t, [_P]),
    "marlc_engine_bind": (C.c_int, [_P, _P, _P, _P]),
    "marlc_engine_buffer": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "marlc_episode_forward": (C.c_int, [_P, _P, _P, C.POINTER(_P), _P, _P]),
    "marlc_model_step": (C.c_int, [_P, _P, _P, _P, C.POINTER(_P), _P]),
    "marlc_engine_seed": (C.c_int, [_P, C.c_uint64, _P]),
    "marlc_loss_phase_a": (C.c_int, [_P, _P, _P]),
    "marlc_loss_phase_b": (C.c_int, [_P, _P]),
    "marlc_episode_backward": (C.c_int, [_P, _P, C.c_int, _P]),
    "marlc_episode_image_grad": (C.c_int, [_P, _P, _P]),
    "marlc_model_step_backward": (C.c_int, [_P, _P, _P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P, _P]),
    "marlc_model_step_input_grad": (C.c_int, [_P, _P, _P, _P]),
    "marlc_adam_step": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                  _P, _P]),
    "marlc_engine_debug_stop": (C.c_int, [_P, C.c_int]),
    "marlc_engine_last_launches": (C.c_int, [_P]),
    "marlc_gemm_launch_count": (C.c_long, [C.c_int]),
}

_lib = None


def exported_symbols() -> list[str]:
    """Every symbol include/marlc.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGS)


def lib() -> C.CDLL:
    """Load (building first if the sources changed and nvcc is around) libmarlc.so."""
    global _lib
    if _lib is not None:
        return _lib
    # MARLC_LIB: an alternative build of the same sources (in-kernel trace / A-B variants; development aid)
    path = os.environ.get("MARLC_LIB") or _build.LIB
    if path == _build.LIB and _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on the box and no prebuilt library
            if not os.path.exists(path):
                raise RuntimeError(
                    "libmarlc.so is missing and could not be built; the CUDA library is mandatory "
                    f"(no CPU fallback exists): {exc}"
                ) from exc
    try:
        handle = C.CDLL(path)
    except OSError as exc:
        raise RuntimeError(f"cannot load {path}: {exc}") from exc
    for name, (res, args) in _SIGS.items():
        fn = getattr(handle, name)  # AttributeError if the ABI drifted
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(ret: int) -> None:
    if ret != 0:
        raise RuntimeError("libmarlc: " + lib().marlc_last_error().decode())


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def stream_ptr(device: torch.device | None = None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, what: str, dtype: torch.dtype | None = None) -> torch.Tensor:
    """Boundary checks shared by every operator: CUDA, dtype, contiguous."""
    if not t.is_cuda:
        raise RuntimeError(f"{what}: expected a CUDA tensor (this implementation has no CPU path), got {t.device}")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"{what}: expected dtype {dtype}, got {t.dtype}")
    return t.contiguous()
