"""ctypes binding of libtmf_sm100a.so (declared in include/tmf.h).

There is deliberately NO fallback: if the shared library is missing, or the device is not a cc 10.x part, every
op raises.  Host code passes raw device pointers (``tensor.data_ptr()``) and the current torch CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtmf_sm100a.so")

POOL_NONE, POOL_MAX, POOL_AVG = 0, 1, 2
LRP_EPSILON, LRP_ZPLUS = 0, 1
CONV_AUTO, CONV_DIRECT, CONV_UMMA = 0, 1, 2

_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float
_pp = C.POINTER(C.c_void_p)          # host array of device pointers

# name -> argtypes  (must mirror include/tmf.h; tests/test_abi.py checks every symbol is exported)
SIGNATURES = {
    "tmf_pack_conv_weights": [_i, _pp, _pp, _pp, _i, _i, _i, _vp],
    "tmf_conv1_fwd": [_i, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _vp],
    "tmf_conv1_wgrad": [_i, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_conv1_bwd_fused": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _f, _vp, C.c_size_t, _vp],
    "tmf_conv1_dgrad_fused": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _f, _i, _vp, C.c_size_t, _vp],
    "tmf_conv3d_fwd": [_i, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "tmf_conv3d_wgrad": [_i, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_bn_finalize": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i64, _f, _f, _i, _vp],
    "tmf_bn_act_pool_fwd": [_i, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_bn_act_pool_bwd_reduce": [_i, _pp, _i, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_bn_act_pool_fwd_keepmax": [_i, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_bn_act_pool_fwd_dual": [_i, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_bn_act_pool_fwd_keepmax_dual": [_i, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_widen_bf16": [_i, _pp, _pp, _i64, _vp],
    "tmf_narrow_f32": [_i, _pp, _pp, _i64, _vp],
    "tmf_gradcam": [_i, _pp, _pp, _pp] + [_i] * 10 + [_vp, C.c_size_t, _vp],
    "tmf_map_resample": [_i, _vp, _pp] + [_i] * 8 + [_vp, C.c_size_t, _vp],
    "tmf_lrp_fold_pack": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _f, _i, _vp],
    "tmf_lrp_ratio": [_i, _pp, _pp, _i, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp, C.c_size_t, _vp],
    "tmf_lrp_conv1": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _f, _i, _vp, C.c_size_t, _vp],
    "tmf_lrp_normalize": [_i, _pp, _i, _i64, _vp],
    "tmf_ig_expand": [_i, _pp, _pp, _vp, _i, _pp, _pp, _i, _i64, _i, _f, _vp],
    "tmf_ig_combine": [_i, _pp, _pp, _pp, _vp, _vp, _i, _pp, _i, _i64, _i, _f, _vp],
    "tmf_ig_attribute": [_i, _pp, _pp, _pp, _i, _i64, _vp, C.c_size_t, _vp],
    "tmf_occ_input": [_i, _pp, _vp, _i, _f, _pp] + [_i] * 7 + [_vp],
    "tmf_occ_compose": [_i, _pp, _pp, _vp, _i, _pp] + [_i] * 12 + [_vp],
    "tmf_occ_map": [_i, _pp, _pp] + [_i] * 13 + [_vp],
    "tmf_abl_input": [_i, _pp, _vp, _i, _pp, C.POINTER(C.c_float), _i, _vp, _vp, _i, _pp] + [_i] * 7 + [_vp],
    "tmf_abl_map": [_i, _pp, _vp, _i, _i, _pp, _i, _i, _i, _i, _vp],
    "tmf_shap_input": [_i, _pp, _vp, _i, _pp, C.POINTER(C.c_float), _i, _vp, _vp, _i, _vp, _vp, _i, _pp] + [_i] * 7 + [_vp],
    "tmf_shap_compose": [_i, _pp, _vp, _pp, _vp, _i, _pp] + [_i] * 12 + [_vp],
    "tmf_attn_scores": [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_attn_relevance": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "tmf_bn_maxpool_bwd_reduce_kept": [_i, _pp, _i, _pp, _pp, _pp, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_bn_bwd_finalize": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i64, _i, _vp],
    "tmf_bn_act_pool_bwd_apply": [_i, _pp, _i, _pp, _pp, _pp, _pp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_linear_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "tmf_linear_dgrad": [_vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "tmf_linear_wgrad": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_layernorm_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp],
    "tmf_layernorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_gelu_bwd": [_vp, _vp, _vp, _i64, _vp],
    "tmf_attn_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_attn_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp],
    "tmf_encoder_pack_weights": [_vp] * 5 + [_i, _vp, _vp],
    "tmf_encoder_proj_fwd": [_vp] * 11 + [_i, _i, _f, _vp, _vp],
    "tmf_encoder_chain_fwd": [_vp] * 22 + [_i, _i, _i, _f, _f, _vp, _vp],
    "tmf_encoder_chain_bwd": [_vp] * 22 + [_i, _i, _i, _vp, _vp, C.c_size_t, _vp],
    "tmf_encoder_proj_bwd": [_vp] * 13 + [_i, _i, _vp, _vp, C.c_size_t, _vp],
    "tmf_encoder_wgrad": [_pp, _vp, _vp, _vp, _i, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_fold_bn_pack": [_i, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _pp, _i, _i, _i, _f, _vp],
    "tmf_eval_head": [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "tmf_volume_minmax": [_vp, _vp, _i, _i64, _vp],
    "tmf_augment_volumes": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "tmf_line_conv_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i64, _i, _i, _vp],
    "tmf_line_conv_dgrad": [_vp, _vp, _vp, _i, _i, _i64, _i, _i, _vp],
    "tmf_line_conv_wgrad": [_vp, _vp, _vp, _vp, _i, _i, _i64, _i, _i, _vp, C.c_size_t, _vp],
    "tmf_conv2d_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "tmf_conv2d_dgrad": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "tmf_conv2d_wgrad": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "tmf_nchw_bn_stats": [_vp, _vp, _i, _i, _i64, _vp],
    "tmf_nchw_bn_relu_fwd": [_vp, _vp, _vp, _i, _i, _i64, _vp],
    "tmf_nchw_bn_relu_bwd_reduce": [_vp, _vp, _vp, _vp, _i, _i, _i64, _vp],
    "tmf_nchw_bn_relu_bwd_apply": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i64, _vp],
    "tmf_maxpool2d_fwd": [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp],
    "tmf_maxpool2d_bwd": [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp],
    "tmf_token_pool_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "tmf_token_pool_bwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "tmf_scale": [_vp, _vp, _f, _vp, _i64, _vp],
    "tmf_adam_step": [_vp, _i, _vp, _f, _f, _f, _f, _vp, _vp, _vp],
}
PLAIN = {"tmf_last_error": (C.c_char_p, []), "tmf_version": (_i, []), "tmf_check_device": (_i, []), "tmf_stat_rows": (_i, []), "tmf_scratch_bytes": (_i64, []), "tmf_encoder_supported": (_i, [_i, _i, _i]), "tmf_encoder_pack_bytes": (C.c_size_t, [_i]),
         "tmf_launch_count": (_i64, []), "tmf_attn_impl_default": (_i, []), "tmf_conv3d_supported": (_i, [_i] * 8),
         "tmf_conv3d_wgrad_workspace_bytes": (_i64, [_i] * 9),
         "tmf_conv3d_umma_plan_info": (_i, [_i] * 8 + [C.POINTER(C.c_int)]),
         "tmf_conv3d_col_plan_info": (_i, [_i] * 7 + [C.POINTER(C.c_int)]),
         "tmf_conv1_bwd_fused_workspace_bytes": (_i64, [_i] * 6), "tmf_conv1_dgrad_fused_workspace_bytes": (_i64, [_i] * 7),
         "tmf_conv1_wgrad_workspace_bytes": (_i64, [_i] * 4), "tmf_gradcam_workspace_bytes": (_i64, [_i] * 11), "tmf_map_resample_workspace_bytes": (_i64, [_i] * 9),
         "tmf_lrp_ratio_workspace_bytes": (_i64, [_i] * 7), "tmf_lrp_conv1_workspace_bytes": (_i64, [_i] * 7),
         "tmf_lrp_conv1_impl": (_i, [_i] * 7), "tmf_ig_attribute_workspace_bytes": (_i64, [_i, _i, _i64]),
         "tmf_line_conv_wgrad_workspace_bytes": (_i64, [_i, _i]), "tmf_adam_chunk_bytes": (_i, [])}

_lib = None
_device_checked = False


def load():
    """dlopen the library (no GPU needed); raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m transmf_ad_b200.build` (there is no fallback path)")
        lib = C.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = _i
        for name, (res, argtypes) in PLAIN.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = res
        _lib = lib
    return _lib


def stat_rows():
    """TMF_STAT_ROWS: rows of a per-channel statistics buffer (include/tmf.h, DETERMINISM)."""
    return int(load().tmf_stat_rows())


def stat_buffers(ng, channels, device):
    """``ng`` statistics buffers double[TMF_STAT_ROWS][2*channels] carved out of one allocation.  Every producer kernel
    writes all rows, so the buffer is NOT zeroed; ``tmf_bn_finalize`` / ``tmf_bn_bwd_finalize`` add the rows in order."""
    return list(torch.empty((ng, stat_rows(), 2 * channels), dtype=torch.float64, device=device).unbind(0))


_SCRATCH = {}


def scratch(device):
    """(tensor, nbytes): the zero-initialised scratch buffer of include/tmf.h (tickets + deterministic partial sums), one
    per (device, stream): kernels that share it are stream-ordered, and every kernel leaves the ticket area zero."""
    dev = torch.device(device)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), torch.cuda.current_stream(dev).cuda_stream)
    buf = _SCRATCH.get(key)
    if buf is None:
        buf = torch.zeros(int(load().tmf_scratch_bytes()), dtype=torch.uint8, device=dev)
        _SCRATCH[key] = buf
    return buf, buf.numel()


def last_error():
    return load().tmf_last_error().decode()


def launch_count():
    return int(load().tmf_launch_count())


def _require_device():
    global _device_checked
    if not _device_checked:
        if not torch.cuda.is_available():
            raise RuntimeError("transmf_ad_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if load().tmf_check_device() != 0:
            raise RuntimeError(last_error())
        _device_checked = True


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_cur_device = getattr(torch._C, "_cuda_getDevice", None)


def stream_ptr():
    """cudaStream_t of torch's current stream (raw C accessors: this sits on the launch path of every kernel)."""
    if _raw_stream is not None and _cur_device is not None:
        return C.c_void_p(_raw_stream(_cur_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device pointer of a tensor (or NULL)."""
    return C.c_void_p(0 if t is None else t.data_ptr())


_PA = {1: C.c_void_p * 1, 2: C.c_void_p * 2}
_NULL_PP = C.cast(None, _pp)


def ptrs(ts):
    """host array of device pointers, one per group; ``None`` -> NULL array.  (A ctypes array instance is accepted
    where the prototype says POINTER(c_void_p); no cast needed.)"""
    if ts is None:
        return _NULL_PP
    if len(ts) == 2:
        a, b = ts
        return _PA[2](0 if a is None else a.data_ptr(), 0 if b is None else b.data_ptr())
    a = ts[0]
    return _PA[1](0 if a is None else a.data_ptr())


class KernelTimer:
    """Optional per-entry-point CUDA-event timing (bench.py's roofline leg).  Off unless ``start()`` is called;
    events are recorded on the launching (current) stream around each C-ABI call."""

    def __init__(self):
        self.records = None

    def start(self):
        self.records = []

    def stop(self):
        """-> {tag: (total_ms, calls)}; synchronises."""
        torch.cuda.synchronize()
        out = {}
        for tag, e0, e1 in self.records or []:
            ms, n = out.get(tag, (0.0, 0))
            out[tag] = (ms + e0.elapsed_time(e1), n + 1)
        self.records = None
        return out


TIMER = KernelTimer()


def call(name, *args, tag=None):
    """Invoke an entry point on the current stream; raises RuntimeError(tmf_last_error()) on failure."""
    _require_device()
    if TIMER.records is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(load(), name)(*args, stream_ptr())
        e1.record()
        TIMER.records.append((tag or name, e0, e1))
    else:
        rc = getattr(load(), name)(*args, stream_ptr())
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")
