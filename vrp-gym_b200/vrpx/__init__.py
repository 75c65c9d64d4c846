"""vrpx — ctypes binding of libvrpx.so (include/vrpx.h), the hand-written sm_100a CUDA behind the
reference-shaped Python surface in `gym_vrp/` and `agents/`.

There is NO CPU fallback: if the shared library is missing, or no sm_100 device is visible, every entry
point that would compute raises `RuntimeError` loudly.  PyTorch is used only for device memory, streams
and (multi-GPU) torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvrpx.so")

TSP, VRP, IRP = 0, 1, 2
GREEDY, SAMPLE, TEACHER = 0, 1, 2
MAX_NODES = 128
EMB = 128
LAYERS = 3


ABI_VERSION = 6  # must equal VRPX_ABI_VERSION of include/vrpx.h


class VrpxError(RuntimeError):
    pass


class EnvView(C.Structure):
    """struct vrpx_env (include/vrpx.h)."""

    _fields_ = [
        ("kind", C.c_int32), ("N", C.c_int32), ("B", C.c_int64),
        ("xy", C.c_void_p), ("depot", C.c_void_p), ("demand", C.c_void_p),
        ("visited", C.c_void_p), ("mask", C.c_void_p), ("cur", C.c_void_p), ("load", C.c_void_p),
    ]


class EncoderLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "bn1_w", "bn1_b", "bn1_mean", "bn1_var",
        "ff0_w", "ff0_b", "ff2_w", "ff2_b", "bn2_w", "bn2_b", "bn2_mean", "bn2_var")]


class EncoderWeights(C.Structure):
    _fields_ = [("f", C.c_int32), ("node_w", C.c_void_p), ("node_b", C.c_void_p),
                ("depot_w", C.c_void_p), ("depot_b", C.c_void_p), ("layer", EncoderLayer * LAYERS)]


class RolloutTrace(C.Structure):
    _fields_ = [("mask_hist", C.c_void_p), ("load_hist", C.c_void_p), ("qg0", C.c_void_p)]


class DecoderWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ag_t", "af_t", "al_t", "a_c", "a_q0", "a_load", "m_t", "m_c", "qk_w")]


class DecoderBwdWeights(C.Structure):
    _fields_ = [("m_n", C.c_void_p), ("al_n", C.c_void_p)]


class DecoderGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("dH", "D0", "D1", "Dl", "d_al_t", "d_m_t", "d_m_c")]


class EncoderLayerT(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("in_proj_wT", "out_proj_wT", "ff0_wT", "ff2_wT")]


class EncoderWeightsT(C.Structure):
    _fields_ = [("layer", EncoderLayerT * LAYERS)]


class EncoderLayerGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "bn1_w", "bn1_b",
                                          "ff0_w", "ff0_b", "ff2_w", "ff2_b", "bn2_w", "bn2_b")]


class EncoderGrads(C.Structure):
    _fields_ = [("node_w", C.c_void_p), ("node_b", C.c_void_p), ("depot_w", C.c_void_p), ("depot_b", C.c_void_p),
                ("layer", EncoderLayerGrads * LAYERS)]


_lib = None


def lib():
    """Load libvrpx.so once.  Raises if it has not been built (python vrp-gym_b200/csrc/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VrpxError(
            f"{LIB_PATH} not found: build it with `python vrp-gym_b200/csrc/build.py` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.vrpx_abi_version.restype = C.c_int
    L.vrpx_last_error.restype = C.c_char_p
    L.vrpx_launch_count.restype = i64
    L.vrpx_device_check.argtypes = [C.c_int]
    L.vrpx_env_generate.argtypes = [C.POINTER(EnvView), u64, u64, vp]
    L.vrpx_env_reset.argtypes = [C.POINTER(EnvView), vp]
    L.vrpx_env_step.argtypes = [C.POINTER(EnvView), vp, vp, vp, vp, vp]
    L.vrpx_env_observe.argtypes = [C.POINTER(EnvView), vp, vp, vp, vp]
    L.vrpx_env_set_visited.argtypes = [C.POINTER(EnvView), vp, vp]
    L.vrpx_env_refresh_mask.argtypes = [C.POINTER(EnvView), vp]
    L.vrpx_mt19937_seed.argtypes = [C.c_uint32, vp, vp]
    L.vrpx_mt19937_permutation_head.argtypes = [vp, vp, i64, i64, vp]
    L.vrpx_mt19937_instances.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp]
    L.vrpx_mt19937_random_actions.argtypes = [vp, vp, vp, i64, i32, vp]
    L.vrpx_encoder_workspace_bytes.argtypes = [i64, i32]
    L.vrpx_encoder_workspace_bytes.restype = i64
    L.vrpx_encoder_forward.argtypes = [C.POINTER(EncoderWeights), C.POINTER(EnvView), vp, vp, i64, i32, i32,
                                       vp, vp, i64, i32, vp, vp]
    L.vrpx_encoder_saved_bytes.argtypes = [i64, i32]
    L.vrpx_encoder_saved_bytes.restype = i64
    L.vrpx_encoder_backward_workspace_bytes.argtypes = [i64, i32]
    L.vrpx_encoder_backward_workspace_bytes.restype = i64
    L.vrpx_encoder_backward.argtypes = [C.POINTER(EncoderWeights), C.POINTER(EncoderWeightsT), C.POINTER(EnvView), vp, vp,
                                        i64, i32, vp, vp, C.POINTER(EncoderGrads), vp, i64, i32, vp]
    L.vrpx_decoder_backward_workspace_bytes.argtypes = [i64, i32]
    L.vrpx_decoder_backward_workspace_bytes.restype = i64
    L.vrpx_decoder_backward.argtypes = [C.POINTER(EnvView), C.POINTER(DecoderWeights), C.POINTER(DecoderBwdWeights), vp, vp,
                                        i32, i64, C.POINTER(RolloutTrace), vp, vp, C.POINTER(DecoderGrads), vp, i64, vp]
    L.vrpx_decoder_backward_samples.argtypes = [C.POINTER(EnvView), C.POINTER(DecoderWeights), C.POINTER(DecoderBwdWeights),
                                                vp, i64, i32, vp, i32, i64, C.POINTER(RolloutTrace), vp, vp,
                                                C.POINTER(DecoderGrads), vp, i64, vp]
    L.vrpx_gemm_tn_accumulate.argtypes = [vp, vp, vp, i64, i32, i32, vp]
    L.vrpx_gemm_tn_colsum_accumulate.argtypes = [vp, vp, vp, vp, i64, i32, i32, vp]
    L.vrpx_colsum_accumulate.argtypes = [vp, i64, i32, vp, vp]
    L.vrpx_episode_gather.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.vrpx_episode_scatter.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.vrpx_rollout_workspace_bytes.argtypes = [i64, i32]
    L.vrpx_rollout_workspace_bytes.restype = i64
    L.vrpx_rollout_workspace_qg_offset.argtypes = []
    L.vrpx_rollout_workspace_qg_offset.restype = i64
    L.vrpx_rollout_table_workspace_bytes.argtypes = [i32, i64, i32]
    L.vrpx_rollout_table_workspace_bytes.restype = i64
    L.vrpx_rollout_samples_workspace_bytes.argtypes = [i32, i64, i32, i32]
    L.vrpx_rollout_samples_workspace_bytes.restype = i64
    L.vrpx_rollout_samples.argtypes = [C.POINTER(EnvView), C.POINTER(DecoderWeights), vp, i64, i32, i64, u64, u64, vp,
                                       i32, vp, vp, vp, vp, vp, i64, vp]
    L.vrpx_rollout_samples_traced.argtypes = [C.POINTER(EnvView), C.POINTER(DecoderWeights), vp, i64, i32, i64, u64, u64,
                                              vp, i32, vp, vp, vp, vp, C.POINTER(RolloutTrace), vp, i64, vp]
    L.vrpx_debug_rollout_profile.argtypes = [C.c_void_p]
    L.vrpx_debug_rollout_profile.restype = None
    L.vrpx_debug_rollout_split.argtypes = [i32]
    L.vrpx_debug_rollout_split.restype = None
    L.vrpx_debug_rollout_timing.argtypes = [i32]
    L.vrpx_debug_rollout_timing.restype = None
    L.vrpx_debug_rollout_kernel_ms.argtypes = []
    L.vrpx_debug_rollout_kernel_ms.restype = C.c_float
    L.vrpx_rollout.argtypes = [C.POINTER(EnvView), C.POINTER(DecoderWeights), vp, i32, i64, u64, u64, vp, i32, i32,
                               vp, vp, vp, vp, C.POINTER(RolloutTrace), vp, i64, vp]
    L.vrpx_debug_gemm.argtypes = [vp, i64, i32, vp, i32, vp, i32, vp, vp, vp, vp, i32, vp]
    L.vrpx_debug_ff_fused.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.vrpx_debug_encoder_fuse_ff.argtypes = [i32]
    L.vrpx_debug_encoder_fuse_ff.restype = None
    L.vrpx_debug_attention_backward.argtypes = [vp, vp, vp, vp, i64, i32, i32, vp]
    L.vrpx_debug_gemm_tn_path.argtypes = [i32]
    L.vrpx_debug_gemm_tn_path.restype = None
    L.vrpx_debug_qkv_attention.argtypes = [vp, vp, vp, i64, i32, vp, vp]
    L.vrpx_debug_encoder_fuse_attention.argtypes = [i32]
    L.vrpx_debug_encoder_fuse_attention.restype = None
    L.vrpx_debug_score_table.argtypes = [vp, vp, i64, i32, vp, vp]
    L.vrpx_debug_encoder_backward_stages.argtypes = [C.POINTER(EncoderWeights), C.POINTER(EncoderWeightsT),
                                                     C.POINTER(EnvView), vp, vp, i64, i32, vp, vp, C.POINTER(EncoderGrads),
                                                     vp, i64, i32, vp, i32, vp]
    if L.vrpx_abi_version() != ABI_VERSION:
        raise VrpxError("libvrpx.so ABI version mismatch")
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise VrpxError(f"libvrpx error {rc}: {lib().vrpx_last_error().decode()}")


_device_ok = {}


def require_device(device=None) -> torch.device:
    """Return the CUDA device to run on, or raise: the product path has no CPU implementation."""
    if not torch.cuda.is_available():
        raise VrpxError("no CUDA device visible: the vrpx rollout path is sm_100a CUDA only (no CPU fallback)")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise VrpxError(f"vrpx needs a CUDA device, got {dev}")
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _device_ok:
        check(lib().vrpx_device_check(idx))
        _device_ok[idx] = True
    return torch.device("cuda", idx)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "vrpx needs contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def launch_count() -> int:
    return int(lib().vrpx_launch_count())
