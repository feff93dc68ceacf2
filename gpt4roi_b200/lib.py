"""ctypes binding of libgpt4roi_b200.so (the C ABI declared in include/gpt4roi_b200.h).

PyTorch is used here only for device memory and streams: every wrapper takes torch
tensors, checks device/dtype/contiguity the way the reference's dispatch does
(mmcv-1.4.7/mmcv/ops/csrc/common/pytorch_device_registry.hpp:109-139), and hands raw
pointers + the current CUDA stream to the C entry point.  There is NO fallback: if the
shared library is missing, or a tensor is not on a CUDA device, the call raises.
"""
import ctypes
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, 'libgpt4roi_b200.so')

F32, F16, BF16, F64 = 0, 1, 2, 3
NCHW, NHWC = 0, 1
POOL_MAX, POOL_AVG = 0, 1
MAX_LEVELS = 4

_DTYPE = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16, torch.float64: F64}

_c = ctypes
_vp, _i, _f, _i64 = _c.c_void_p, _c.c_int, _c.c_float, _c.c_int64
_ll = _c.c_longlong

# name -> (restype, argtypes); must list EVERY symbol include/gpt4roi_b200.h declares
# (tests/test_abi_cpu.py parses the header and checks both directions).
SIGNATURES = {
    'g4r_last_error': (_c.c_char_p, []),
    'g4r_version': (_i, []),
    'g4r_built_arch': (_i, []),
    'g4r_set_sm_reserve': (_i, [_i]),
    'g4r_set_pdl': (_i, [_i]),
    'g4r_roi_align_forward': (_i, [_vp] * 5 + [_i] * 7 + [_f] + [_i] * 5 + [_vp]),
    'g4r_roi_align_forward_workspace': (_c.c_size_t, [_i] * 11),
    'g4r_roi_align_forward_ws': (_i, [_vp] * 5 + [_i] * 7 + [_f] + [_i] * 5 + [_vp, _c.c_size_t, _vp]),
    'g4r_roi_align_backward': (_i, [_vp] * 5 + [_i] * 7 + [_f] + [_i] * 5 + [_vp]),
    'g4r_roi_align_mlvl_forward': (_i, [_vp] * 4 + [_i] + [_vp] * 2 + [_i] * 9 + [_vp] * 3),
    'g4r_roi_align_mlvl_backward': (_i, [_vp] * 4 + [_i] + [_vp] * 2 + [_i] * 8 + [_vp]),
    'g4r_splice_region_tokens': (_i, [_vp] * 8 + [_i] * 5 + [_i64] * 4 + [_vp]),
    'g4r_gemm_bf16': (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _vp, _i, _vp, _ll, _i, _i, _i, _vp]),
    'g4r_gemm_bf16_ex': (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _vp, _i, _vp, _ll, _i, _i, _i, _i, _i, _vp]),
    'g4r_gemm_bf16_t': (_i, [_vp, _ll, _i, _vp, _ll, _i, _vp, _ll, _i, _i, _i, _i, _vp]),
    'g4r_gemm_qkv_rope_bf16': (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    'g4r_decode_gemm_bf16': (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _ll, _vp, _vp, _i, _i, _vp, _vp, _vp,
                                  _i, _i, _vp]),
    'g4r_kv_append_bf16': (_i, [_vp, _ll, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp]),
    'g4r_decode_attention_bf16': (_i, [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _vp, _i, _f, _vp]),
    'g4r_conv_nhwc_bf16': (_i, [_vp] * 3 + [_i] * 7 + [_vp, _i, _i, _vp, _i, _vp]),
    'g4r_attention_bf16': (_i, [_vp] * 4 + [_ll] * 4 + [_i] * 5 + [_f, _vp, _vp]),
    'g4r_attention_tc_bf16': (_i, [_vp] * 4 + [_ll] * 4 + [_i] * 5 + [_f, _vp, _vp]),
    'g4r_layernorm_bf16': (_i, [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _f, _vp]),
    'g4r_layernorm_ex': (_i, [_vp, _ll, _i, _vp, _vp, _vp, _ll, _i, _i, _i, _f, _vp]),
    'g4r_cast_f32_bf16': (_i, [_vp, _ll, _ll, _vp, _i, _i, _i, _vp]),
    'g4r_rmsnorm_bf16': (_i, [_vp, _ll, _vp, _vp, _ll, _i, _i, _f, _vp]),
    'g4r_rmsnorm_ex': (_i, [_vp, _ll, _i, _vp, _vp, _ll, _i, _i, _f, _vp]),
    'g4r_rope_inplace_bf16': (_i, [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp]),
    'g4r_patchify_bf16': (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    'g4r_vit_embed_bf16': (_i, [_vp] * 4 + [_i] * 3 + [_vp]),
    'g4r_upsample_tokens_coords_bf16': (_i, [_vp, _ll, _ll, _vp, _i, _i, _i, _i, _i, _vp]),
    'g4r_upsample_tokens_coords_f32': (_i, [_vp, _ll, _ll, _vp, _i, _i, _i, _i, _i, _vp]),
    'g4r_fuse_gather_bf16': (_i, [_vp, _vp, _vp, _i] * 3 + [_vp, _i, _i, _vp]),
    'g4r_gn_finalize': (_i, [_vp] * 5 + [_i] * 4 + [_f, _f, _vp]),
    'g4r_conv_gn_slots': (_i, [_i, _i]),
    'g4r_pos_embed_mlp': (_i, [_vp] * 10 + [_i, _f, _vp]),
    'g4r_cross_entropy_bf16': (_i, [_vp, _ll, _vp, _i, _i, _vp, _vp, _vp, _vp, _ll, _f, _vp]),
    'g4r_rmsnorm_bwd_slabs': (_i, [_i]),
    'g4r_rmsnorm_bwd_bf16': (_i, [_vp, _ll, _vp, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _vp, _i, _i, _f, _vp]),
    'g4r_swiglu_fwd_bf16': (_i, [_vp, _ll, _vp, _ll, _ll, _i, _vp]),
    'g4r_swiglu_bwd_bf16': (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _vp]),
    'g4r_attention_tc_lse_bf16': (_i, [_vp] * 4 + [_ll] * 4 + [_i] * 5 + [_f, _vp, _vp]),
    'g4r_attention_bwd_bf16': (_i, [_vp] * 10 + [_ll] * 6 + [_i] * 5 + [_f, _vp]),
    'g4r_splice_backward': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'g4r_embed_grad_rows': (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _vp]),
    'g4r_colsum_slabs': (_i, [_i]),
    'g4r_colsum_bf16': (_i, [_vp, _ll, _i, _i, _vp, _vp, _vp]),
    'g4r_pad_nhwc_bf16': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'g4r_conv_weight_flip_t_bf16': (_i, [_vp, _ll, _vp, _i, _i, _vp]),
    'g4r_conv3x3_dw_bf16': (_i, [_vp, _vp, _vp, _ll, _i, _i, _i, _i, _vp]),
    'g4r_gn_relu_bwd_workspace': (_ll, [_i, _i, _i, _i]),
    'g4r_gn_relu_bwd_bf16': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _f, _f, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    'g4r_fuse_gather_bwd': (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp]),
    'g4r_pos_embed_mlp_grad_size': (_i, []),
    'g4r_pos_embed_mlp_bwd': (_i, [_vp] * 9 + [_ll, _vp, _vp, _i, _f, _vp]),
    'g4r_relu_bwd_bf16': (_i, [_vp, _vp, _vp, _ll, _vp]),
    'g4r_adamw_step': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _f, _i, _f, _vp]),
    'g4r_adamw_step_ex': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _f, _i, _f, _vp, _vp]),
    'g4r_sumsq_slabs': (_i, []),
    'g4r_sumsq': (_i, [_vp, _i, _ll, _vp, _vp]),
    'g4r_grad_clip_coef': (_i, [_vp, _ll, _f, _f, _vp, _vp]),
    'g4r_preprocess_images': (_i, [_vp] * 6 + [_i, _i, _vp, _vp, _i, _i, _vp]),
    'g4r_affine_relu_nhwc_bf16': (_i, [_vp, _vp, _vp, _vp, _i, _ll, _i, _vp]),
    'g4r_add_bias_pos_cast': (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _vp]),
}

# fp16 twins of the inference entry points (include/gpt4roi_b200.h, last section; csrc/act_type.cuh): same signatures.
F16_TWINS = {
    'g4r_gemm_bf16': 'g4r_gemm_f16',
    'g4r_gemm_bf16_ex': 'g4r_gemm_f16_ex',
    'g4r_gemm_qkv_rope_bf16': 'g4r_gemm_qkv_rope_f16',
    'g4r_conv_nhwc_bf16': 'g4r_conv_nhwc_f16',
    'g4r_attention_tc_bf16': 'g4r_attention_tc_f16',
    'g4r_attention_bf16': 'g4r_attention_f16',
    'g4r_layernorm_bf16': 'g4r_layernorm_f16',
    'g4r_rmsnorm_bf16': 'g4r_rmsnorm_f16',
    'g4r_rope_inplace_bf16': 'g4r_rope_inplace_f16',
    'g4r_patchify_bf16': 'g4r_patchify_f16',
    'g4r_vit_embed_bf16': 'g4r_vit_embed_f16',
    'g4r_upsample_tokens_coords_bf16': 'g4r_upsample_tokens_coords_f16',
    'g4r_upsample_tokens_coords_f32': 'g4r_upsample_tokens_coords_f32_f16',
    'g4r_layernorm_ex': 'g4r_layernorm_ex_f16',
    'g4r_rmsnorm_ex': 'g4r_rmsnorm_ex_f16',
    'g4r_cast_f32_bf16': 'g4r_cast_f32_f16',
    'g4r_fuse_gather_bf16': 'g4r_fuse_gather_f16',
    'g4r_gn_finalize': 'g4r_gn_finalize_f16',
    'g4r_pos_embed_mlp': 'g4r_pos_embed_mlp_f16',
    'g4r_affine_relu_nhwc_bf16': 'g4r_affine_relu_nhwc_f16',
    'g4r_add_bias_pos_cast': 'g4r_add_bias_pos_cast_f16',
    'g4r_decode_gemm_bf16': 'g4r_decode_gemm_f16',
    'g4r_kv_append_bf16': 'g4r_kv_append_f16',
    'g4r_decode_attention_bf16': 'g4r_decode_attention_f16',
}
SIGNATURES.update({twin: SIGNATURES[name] for name, twin in F16_TWINS.items()})


def sym(name, dtype):
    """Entry-point name for 16-bit tensors of `dtype`: the bf16 name itself, or its fp16 twin."""
    if dtype == torch.float16:
        return F16_TWINS[name]
    if dtype != torch.bfloat16:
        raise TypeError('%s: bf16 or fp16 tensors required, got %s' % (name, dtype))
    return name


_lib = None
LAUNCHES = 0  # kernels launched through the C ABI (bench.py reports it as gpu_launches)


def count_launches(n=1):
    global LAUNCHES
    LAUNCHES += n


class G4RError(RuntimeError):
    """Non-zero return of a C-ABI entry point (maps the reference's RuntimeError)."""


def load():
    """Load the shared library (once).  Raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            'gpt4roi_b200: %s is missing. Build it with `python -m gpt4roi_b200.build` '
            '(needs nvcc; cross-compiles for sm_100a without a GPU). There is no CPU or '
            'PyTorch fallback for this path.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def set_sm_reserve(n):
    """Keep n SMs free of the persistent GEMM kernels (room for an overlapped collective); returns the previous value."""
    return int(load().g4r_set_sm_reserve(int(n)))


def set_pdl(on):
    """Programmatic dependent launch for the decode step's kernel chain (include/gpt4roi_b200.h: g4r_set_pdl); returns
    the previous setting."""
    return int(load().g4r_set_pdl(int(bool(on))))


def check(rc, launches=1):
    global LAUNCHES
    LAUNCHES += launches
    if rc != 0:
        msg = load().g4r_last_error()
        raise G4RError('gpt4roi_b200 C-ABI error %d: %s' % (rc, (msg or b'').decode()))


def dtype_code(t):
    try:
        return _DTYPE[t.dtype]
    except KeyError:
        raise TypeError('gpt4roi_b200: unsupported dtype %s' % t.dtype)


def require_cuda_same_device(named):
    """pytorch_device_registry.hpp:111-124: every tensor on the device of the first one."""
    first = None
    for idx, (name, t) in enumerate(named):
        if t is None:
            continue
        if first is None:
            first = t
            if not t.is_cuda:
                raise RuntimeError(
                    'gpt4roi_b200: %s is on %s -- implementation for device %s not found '
                    '(this library is CUDA sm_100a only; no CPU fallback)' % (name, t.device, t.device.type))
        elif t.device != first.device:
            raise RuntimeError('gpt4roi_b200: arg %d (%s) is on %s but arg 0 is on %s'
                               % (idx, name, t.device, first.device))
    return first.device


def require_contiguous(named):
    for name, t in named:
        if t is not None and not t.is_contiguous():
            raise RuntimeError('gpt4roi_b200: %s must be contiguous (the reference indexes raw '
                               'data_ptr memory, roi_align_cuda.cu:21-23)' % name)


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr_array(tensors):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def int_array(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


def float_array(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])
