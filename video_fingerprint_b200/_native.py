"""ctypes binding of libvfp_b200.so (include/vfp_b200.h). PyTorch only supplies device memory and streams
here; every signature is plain pointers and sizes. Importing this module never touches the GPU; calling
into it without the built library or without a CUDA device raises - there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_LIB_NAME = "libvfp_b200.so"
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, _LIB_NAME)
LIB_PATH = os.environ.get("VFP_B200_LIB", LIB_PATH)  # development aid: load an experimental build

ABI_VERSION = 5
FRAME_U8, FRAME_BF16, FRAME_F32, FRAME_U8_HWC = 0, 1, 2, 3

# every symbol include/vfp_b200.h declares (tests check the library exports exactly these)
EXPORTED_SYMBOLS = (
    "vfp_abi_version",
    "vfp_last_error",
    "vfp_device_sm_count",
    "vfp_weights_create",
    "vfp_weights_destroy",
    "vfp_weights_embedding_dim",
    "vfp_forward_workspace_bytes",
    "vfp_forward",
    "vfp_forward_clips",
    "vfp_join_workspace_bytes",
    "vfp_join_threshold",
    "vfp_topk_workspace_bytes",
    "vfp_topk_ip",
    "vfp3d_weights_create",
    "vfp3d_weights_destroy",
    "vfp3d_weights_embedding_dim",
    "vfp3d_forward_workspace_bytes",
    "vfp3d_forward",
    "vfp3d_forward_packed_workspace_bytes",
    "vfp3d_forward_packed",
    "vfp3d_forward_clips",
    "vfp_preprocess_workspace_bytes",
    "vfp_preprocess_frames",
    "vfp_pair_scores",
    "vfp_pair_stats",
    "vfp_device_error_word",
    "vfp_profile_enable",
    "vfp_profile_num_stages",
    "vfp_profile_stage_name",
    "vfp_profile_read",
    "vfp_set_tuning",
    "vfp_debug_hang_log",
)


class TensorDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_int64)]


class NativeError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library once and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} is missing - build it with `python -m video_fingerprint_b200.build` "
            "(this package has no CPU or PyTorch fallback path)"
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
    lib.vfp_abi_version.restype = i32
    lib.vfp_abi_version.argtypes = []
    lib.vfp_last_error.restype = C.c_char_p
    lib.vfp_last_error.argtypes = []
    lib.vfp_device_sm_count.restype = i32
    lib.vfp_device_sm_count.argtypes = []
    lib.vfp_weights_create.restype = i32
    lib.vfp_weights_create.argtypes = [C.POINTER(TensorDesc), i32, C.POINTER(vp)]
    lib.vfp_weights_destroy.restype = None
    lib.vfp_weights_destroy.argtypes = [vp]
    lib.vfp_weights_embedding_dim.restype = i32
    lib.vfp_weights_embedding_dim.argtypes = [vp]
    lib.vfp_forward_workspace_bytes.restype = sz
    lib.vfp_forward_workspace_bytes.argtypes = [i64, i64]
    lib.vfp_forward.restype = i32
    lib.vfp_forward.argtypes = [vp, vp, i32, vp, i32, vp, vp, vp, sz, vp]
    lib.vfp_forward_clips.restype = i32
    lib.vfp_forward_clips.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]
    lib.vfp_join_workspace_bytes.restype = sz
    lib.vfp_join_workspace_bytes.argtypes = [i64, i64, i64]
    lib.vfp_join_threshold.restype = i32
    lib.vfp_join_threshold.argtypes = [vp, vp, i64, i64, i32, i64, f32, f32, vp, vp, vp, i64, vp, vp, sz, vp]
    lib.vfp_topk_workspace_bytes.restype = sz
    lib.vfp_topk_workspace_bytes.argtypes = [i64, i64, i32]
    lib.vfp_topk_ip.restype = i32
    lib.vfp_topk_ip.argtypes = [vp, vp, i64, i64, i32, i32, f32, vp, vp, vp, vp, sz, vp]
    lib.vfp3d_weights_create.restype = i32
    lib.vfp3d_weights_create.argtypes = [C.POINTER(TensorDesc), i32, i32, C.POINTER(vp)]
    lib.vfp3d_weights_destroy.restype = None
    lib.vfp3d_weights_destroy.argtypes = [vp]
    lib.vfp3d_weights_embedding_dim.restype = i32
    lib.vfp3d_weights_embedding_dim.argtypes = [vp]
    lib.vfp3d_forward_workspace_bytes.restype = sz
    lib.vfp3d_forward_workspace_bytes.argtypes = [vp, i64, i32]
    lib.vfp3d_forward.restype = i32
    lib.vfp3d_forward.argtypes = [vp, vp, i32, i64, i32, vp, vp, sz, vp]
    lib.vfp3d_forward_packed_workspace_bytes.restype = sz
    lib.vfp3d_forward_packed_workspace_bytes.argtypes = [vp, i64, i64]
    lib.vfp3d_forward_packed.restype = i32
    lib.vfp3d_forward_packed.argtypes = [vp, vp, i32, vp, i32, vp, vp, sz, vp]
    lib.vfp3d_forward_clips.restype = i32
    lib.vfp3d_forward_clips.argtypes = [vp, vp, vp, i32, i32, vp, vp, sz, vp]
    lib.vfp_preprocess_workspace_bytes.restype = sz
    lib.vfp_preprocess_workspace_bytes.argtypes = [i32, i32]
    lib.vfp_preprocess_frames.restype = i32
    lib.vfp_preprocess_frames.argtypes = [vp, i32, i32, i32, vp, vp, sz, vp]
    lib.vfp_pair_scores.restype = i32
    lib.vfp_pair_scores.argtypes = [vp, i64, i32, vp, vp, i64, vp, vp]
    lib.vfp_pair_stats.restype = i32
    lib.vfp_pair_stats.argtypes = [vp, vp, i64, i32, vp, vp, vp, vp, i64, vp, i32, vp, vp, vp, vp, vp]
    lib.vfp_profile_enable.restype = i32
    lib.vfp_profile_enable.argtypes = [i32]
    lib.vfp_profile_num_stages.restype = i32
    lib.vfp_profile_num_stages.argtypes = []
    lib.vfp_profile_stage_name.restype = C.c_char_p
    lib.vfp_profile_stage_name.argtypes = [i32]
    lib.vfp_profile_read.restype = i32
    lib.vfp_profile_read.argtypes = [vp, i32, vp, i32]
    lib.vfp_set_tuning.restype = i32
    lib.vfp_set_tuning.argtypes = [i32, C.c_longlong]
    lib.vfp_debug_hang_log.restype = i32
    lib.vfp_debug_hang_log.argtypes = [C.c_void_p, i32]
    lib.vfp_device_error_word.restype = C.c_uint
    lib.vfp_device_error_word.argtypes = []
    if lib.vfp_abi_version() != ABI_VERSION:
        raise NativeError(f"ABI mismatch: library {lib.vfp_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().vfp_last_error().decode("utf-8", "replace")
        raise NativeError(f"{what} failed (code {rc}): {msg}")


def require_cuda() -> None:
    import torch

    if not torch.cuda.is_available():
        raise NativeError("no CUDA device: video_fingerprint_b200 runs on B200 (sm_100a) only, there is no CPU fallback")
