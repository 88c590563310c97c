"""ctypes binding of libdss_b200.so (include/dss_b200.h). Fails loudly if the CUDA library is missing: there is
no CPU or PyTorch fallback for any operator of the hot path."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import torch

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libdss_b200.so"

c_void_p, c_int, c_float, c_size_t = C.c_void_p, C.c_int, C.c_float, C.c_size_t


class VitConfig(C.Structure):
    _fields_ = [("patch", c_int), ("dim", c_int), ("depth", c_int), ("heads", c_int), ("mlp_ratio", c_int),
                ("grid0", c_int), ("ln_eps", c_float)]


class ProfileEntry(C.Structure):
    _fields_ = [("name", C.c_char_p), ("launches", C.c_longlong), ("total_ms", C.c_double)]


class VitBlockWeights(C.Structure):
    _fields_ = [(n, c_void_p) for n in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "proj_w", "proj_b", "ln2_w", "ln2_b",
                                        "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class VitWeights(C.Structure):
    _fields_ = [("patch_w", c_void_p), ("patch_b", c_void_p), ("cls_token", c_void_p), ("pos_embed", c_void_p),
                ("blocks", C.POINTER(VitBlockWeights)), ("norm_w", c_void_p), ("norm_b", c_void_p)]


# name -> (restype, argtypes); every symbol declared in include/dss_b200.h
PROTOTYPES = {
    "dss_last_error": (C.c_char_p, []),
    "dss_version": (c_int, []),
    "dss_device_sm_count": (c_int, []),
    "dss_kernel_launch_count": (C.c_longlong, []),
    "dss_profile_enable": (None, [c_int]),
    "dss_profile_read": (c_int, [C.POINTER(ProfileEntry), c_int]),
    "dss_vit_create": (c_int, [C.POINTER(VitConfig), C.POINTER(c_void_p)]),
    "dss_vit_destroy": (None, [c_void_p]),
    "dss_vit_load_weights": (c_int, [c_void_p, C.POINTER(VitWeights), c_void_p]),
    "dss_vit_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int, c_int]),
    "dss_vit_forward_k": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                  c_void_p]),
    "dss_vit_forward_tokens": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                       c_void_p]),
    "dss_vit_forward_cls": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dss_vit_pos_embed": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dss_pos_embed_interp_host": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "dss_op_gemm_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                c_int, c_void_p]),
    "dss_op_gemm_f16_simt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                     c_int, c_int, c_void_p]),
    "dss_op_gemm_ln_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                                   c_int, c_void_p]),
    "dss_op_layernorm_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "dss_op_attention_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "dss_op_attention_tc_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "dss_op_im2col_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "dss_affinity_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dss_affinity": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_int, c_void_p,
                             c_void_p, c_size_t, c_void_p]),
    "dss_knn_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dss_knn_color_counts": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dss_eigsh_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "dss_eigsh_laplacian": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dss_eigsh_topk": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_size_t, c_void_p]),
    "dss_rw_affinity_add": (c_int, [c_void_p, c_int, c_int, c_int, c_float, C.c_double, c_void_p, c_int, c_void_p,
                                    c_void_p]),
    "dss_segment_threshold": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "dss_segment_kmeans": (c_int, [c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, c_int, c_int, c_int, c_void_p,
                                   c_void_p, c_int, c_int, c_int, c_int, C.c_uint, c_int, c_float, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "dss_upsample_bilinear": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dss_normalize_rows": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
}

EPI_BIAS_F16, EPI_BIAS_GELU_F16, EPI_BIAS_RESID_F32, EPI_BIAS_F32, EPI_PATCH_F32, EPI_DROPCLS_F32 = range(6)
AFF_NORMALIZE, AFF_THRESHOLD_AT_ZERO, AFF_NO_MAX_SCALE = 1, 2, 4

_lib = None


class DssError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libdss_b200.so (building is the job of build.py / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.is_file():
        raise DssError(f"{LIB_PATH} not found: build it with `python {_HERE.name}/build.py` "
                       "(nvcc, sm_100a). There is no fallback implementation.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().dss_last_error()
        raise DssError(f"{what or 'libdss_b200'} failed (status {rc}): {msg.decode() if msg else ''}")


def ptr(t) -> int:
    """Device/host pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "libdss_b200 needs contiguous tensors"
    return t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise DssError(f"{name} must be a CUDA tensor: the hot path has no CPU implementation")


def launch_count() -> int:
    return int(load().dss_kernel_launch_count())


def profile(enable: bool) -> None:
    load().dss_profile_enable(1 if enable else 0)


def profile_read() -> dict:
    """{kernel class: (launches, total_ms)} for the recording started by profile(True)."""
    arr = (ProfileEntry * 32)()
    n = load().dss_profile_read(arr, 32)
    if n < 0:
        check(n, "dss_profile_read")
    return {arr[i].name.decode(): (int(arr[i].launches), float(arr[i].total_ms)) for i in range(n)}
