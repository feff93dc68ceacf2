"""Dense contractions (nn.Linear / nn.Conv2d replacements) on the tcgen05 kernels.

Thin torch-tensor front-ends of `g4r_gemm_bf16` / `g4r_conv_nhwc_bf16`
(csrc/gemm_tcgen05.cu).  bf16 operands (or fp16 throughout: the `_f16` twins, for the demo's dtype), fp32
accumulation; no library GEMM is called.
"""
import torch

from . import lib as _L

ACT = {None: 0, 'none': 0, 'relu': 1, 'quick_gelu': 2, 'swiglu': 3}

# bench.py instrumentation: when PROFILE is a list, every tensor-core launch appends
# (kind, flops, start_event, end_event) -- used for the roofline of the dominant kernel.
PROFILE = None


def _prof_begin(dev):
    if PROFILE is None:
        return None
    e = torch.cuda.Event(enable_timing=True)
    e.record(torch.cuda.current_stream(dev))
    return e


def _prof_end(dev, start, kind, flops):
    if start is None:
        return
    e = torch.cuda.Event(enable_timing=True)
    e.record(torch.cuda.current_stream(dev))
    PROFILE.append((kind, flops, start, e))


def _act16(name, *ts):
    """The one 16-bit storage type (bf16, or fp16 for the demo's dtype) of the given operands."""
    dt = ts[0].dtype
    if dt not in (torch.bfloat16, torch.float16) or any(t.dtype != dt for t in ts):
        raise TypeError('%s: bf16 (or all-fp16) operands required, got %s' % (name, ' / '.join(str(t.dtype) for t in ts)))
    return dt


def linear(x, weight, bias=None, act=None, residual=None, out=None, out_dtype=None,
           k_splits=1, round_branch=False):
    """y = act(x @ weight.T + bias) (+ residual).  x [..., K] bf16, weight [N, K] bf16.

    act='swiglu': weight rows interleaved (gate_j, up_j); returns [..., N/2].
    residual may be bf16 or fp32; round_branch=True rounds act(x@W.T+bias) to bf16 before the residual
    add (a bf16 Linear output added to an fp32 residual stream, as CLIP does under autocast).
    k_splits>1: deterministic split-K -- returns fp32 partial slabs [k_splits, M, N] (no bias);
    the caller sums them in a fixed order (kernels.add_bias_pos_cast does).
    """
    K = x.shape[-1]
    x2 = x.reshape(-1, K)
    M, N = x2.shape[0], weight.shape[0]
    named = [('x', x2), ('weight', weight), ('bias', bias), ('residual', residual)]
    dev = _L.require_cuda_same_device(named)
    a16 = _act16('linear', x2, weight)
    out_dtype = a16 if out_dtype is None else out_dtype
    if out_dtype not in (a16, torch.float32):
        raise TypeError('linear: out_dtype must be %s or fp32' % a16)
    if x2.stride(-1) != 1 or weight.stride(-1) != 1:
        raise RuntimeError('linear: operands must be K-major (unit stride on the last dim)')
    if weight.shape[1] != K:
        raise RuntimeError('linear: weight is %s but x has K=%d' % (tuple(weight.shape), K))
    n_out = N // 2 if act == 'swiglu' else N
    out_f32 = out_dtype == torch.float32
    if k_splits > 1:
        if out is not None or bias is not None:
            raise RuntimeError('linear: split-K returns its own [k_splits,M,N] slabs and takes no bias')
        slabs = torch.empty((k_splits, M, n_out), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _ps = _prof_begin(dev)
            _L.check(getattr(_L.load(), _L.sym('g4r_gemm_bf16', a16))(
                _L.ptr(x2), x2.stride(0), _L.ptr(weight), weight.stride(0), _L.ptr(slabs), n_out,
                M, N, K, None, 0, None, 0, 0, 1, int(k_splits), _L.stream_ptr(dev)))
            _prof_end(dev, _ps, 'gemm', 2.0 * M * N * K)
        return slabs
    if out is None:
        out = torch.empty((M, n_out), dtype=out_dtype, device=dev)
    else:
        if out.dtype != out_dtype or out.shape[-1] != n_out or out.stride(-1) != 1:
            raise RuntimeError('linear: bad `out`')
    out2 = out.reshape(-1, n_out) if out.is_contiguous() else out
    res2 = None
    if residual is not None:
        if residual.dtype not in (a16, torch.float32):
            raise TypeError('linear: residual must be %s or fp32' % a16)
        res2 = residual.reshape(-1, n_out) if residual.is_contiguous() else residual
    bias_f32 = 0
    if bias is not None:
        if bias.dtype == torch.float32:
            bias_f32 = 1
        elif bias.dtype != a16:
            raise TypeError('linear: bias must be %s or fp32' % a16)
    with torch.cuda.device(dev):
        _ps = _prof_begin(dev)
        _L.check(getattr(_L.load(), _L.sym('g4r_gemm_bf16_ex', a16))(
            _L.ptr(x2), x2.stride(0), _L.ptr(weight), weight.stride(0), _L.ptr(out2), out2.stride(0),
            M, N, K, _L.ptr(bias), bias_f32, _L.ptr(res2), res2.stride(0) if res2 is not None else 0,
            int(res2 is not None and res2.dtype == torch.float32), int(bool(round_branch)),
            ACT[act], int(out_f32), int(k_splits), _L.stream_ptr(dev)))
        _prof_end(dev, _ps, 'gemm', 2.0 * M * N * K)
    return out.reshape(*x.shape[:-1], n_out) if out.is_contiguous() else out


def matmul_t(a, b, a_mn=False, b_mn=False, out_dtype=torch.bfloat16, out=None):
    """D[M,N] = op(a) @ op(b).T on the tensor cores with the transposes folded into the operand descriptors.
    a: [M,K] (a_mn=False) or stored [K,M] (a_mn=True); b: [N,K] (b_mn=False) or stored [K,N] (b_mn=True).
    Linear backward:  grad_x = matmul_t(grad_y, W, b_mn=True);  grad_W = matmul_t(grad_y, x, a_mn=True, b_mn=True)."""
    dev = _L.require_cuda_same_device([('a', a), ('b', b)])
    if a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16 or a.dim() != 2 or b.dim() != 2:
        raise TypeError('matmul_t: 2-D bf16 operands required')
    if a.stride(1) != 1 or b.stride(1) != 1:
        raise RuntimeError('matmul_t: operands must have unit stride on the last dim')
    M, K = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    N, Kb = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    if K != Kb:
        raise RuntimeError('matmul_t: contraction mismatch %d vs %d' % (K, Kb))
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=dev)
    elif tuple(out.shape) != (M, N) or out.dtype != out_dtype or out.stride(1) != 1:
        raise RuntimeError('matmul_t: `out` must be [%d,%d] %s with unit inner stride' % (M, N, out_dtype))
    with torch.cuda.device(dev):
        _ps = _prof_begin(dev)
        _L.check(_L.load().g4r_gemm_bf16_t(_L.ptr(a), a.stride(0), int(a_mn), _L.ptr(b), b.stride(0), int(b_mn),
                                           _L.ptr(out), out.stride(0), M, N, K, int(out_dtype == torch.float32),
                                           _L.stream_ptr(dev)))
        _prof_end(dev, _ps, 'gemm', 2.0 * M * N * K)
    return out


def qkv_rope(x, wqkv, cos, sin, L, rope_cols, pos0=0, pos_dev=None):
    """Fused LLaMA q/k/v projection + rotary embedding: x [M,K] bf16, wqkv [N,K] (q|k|v rows), cos/sin
    bf16 [L,128]; columns [0,rope_cols) (q and k heads, head_dim 128) are rotated at position row % L."""
    M, K = x.shape
    N = wqkv.shape[0]
    dev = _L.require_cuda_same_device([('x', x), ('wqkv', wqkv), ('cos', cos), ('sin', sin)])
    a16 = _act16('qkv_rope', x, wqkv, cos, sin)
    out = torch.empty((M, N), dtype=a16, device=dev)
    with torch.cuda.device(dev):
        _ps = _prof_begin(dev)
        _L.check(getattr(_L.load(), _L.sym('g4r_gemm_qkv_rope_bf16', a16))(
            _L.ptr(x), x.stride(0), _L.ptr(wqkv), wqkv.stride(0), _L.ptr(out), N, M, N, K, _L.ptr(cos), _L.ptr(sin),
            int(rope_cols), int(L), int(pos0), _L.ptr(pos_dev), _L.stream_ptr(dev)))
        _prof_end(dev, _ps, 'gemm', 2.0 * M * N * K)
    return out


def gn_slots(h, w):
    """Number of per-(tile,warp) GroupNorm partial-sum slots the conv kernel writes for an h x w map."""
    return int(_L.load().g4r_conv_gn_slots(int(h), int(w)))


def conv_nhwc(x, weight_khwc, bias=None, act=None, gn_stats=None, out=None, levels=1):
    """NHWC conv, stride 1, 'same' padding.  x [N,H,W,Cin] bf16; weight_khwc [Cout,kh,kw,Cin] bf16.

    gn_stats: optional fp32 [N, gn_slots(H,W), groups, 2] receiving per-(tile,warp) partial sum / sumsq
    of the bf16 output per (image, 16-channel group); see kernels.gn_finalize.
    """
    dev = _L.require_cuda_same_device([('x', x), ('weight', weight_khwc), ('bias', bias), ('gn_stats', gn_stats)])
    _L.require_contiguous([('x', x), ('weight', weight_khwc)])
    n, h, w, cin = x.shape
    if levels > 1:
        # x [levels*n,H,W,Cin] level-major; weight [Cout, levels, k, k, Cin]: sum of `levels` convs
        cout, lv, kh, kw, cin2 = weight_khwc.shape
        if lv != levels or n % levels:
            raise RuntimeError('conv_nhwc: levels mismatch')
        n //= levels
    else:
        cout, kh, kw, cin2 = weight_khwc.shape
    if kh != kw or kh not in (1, 3) or cin2 != cin:
        raise RuntimeError('conv_nhwc: weight must be [Cout,k,k,Cin] with k in (1,3)')
    a16 = _act16('conv_nhwc', x, weight_khwc)
    if out is None:
        out = torch.empty((n, h, w, cout), dtype=a16, device=dev)
    bias_f32 = int(bias is not None and bias.dtype == torch.float32)
    groups = 0
    if gn_stats is not None:
        slots = gn_slots(h, w)
        if gn_stats.dtype != torch.float32 or gn_stats.dim() != 4 or gn_stats.shape[0] != n or \
                gn_stats.shape[1] != slots or gn_stats.shape[3] != 2 or not gn_stats.is_contiguous():
            raise RuntimeError('gn_stats must be contiguous fp32 [N,%d,groups,2]' % slots)
        groups = gn_stats.shape[2]
    with torch.cuda.device(dev):
        _ps = _prof_begin(dev)
        _L.check(getattr(_L.load(), _L.sym('g4r_conv_nhwc_bf16', a16))(
            _L.ptr(x), _L.ptr(weight_khwc), _L.ptr(out), n, h, w, cin, cout, kh, int(levels), _L.ptr(bias), bias_f32,
            ACT[act], _L.ptr(gn_stats), groups, _L.stream_ptr(dev)))
        _prof_end(dev, _ps, 'conv', 2.0 * n * h * w * cout * kh * kw * cin * levels)
    return out


def decode_gemm(x, weight, act=None, residual=None, rope=None, kv=None):
    """Decode-step GEMM (M = batch <= 16): out = [RoPE | SwiGLU | + residual](x @ weight.T), the rotary embedding
    and the KV-cache append folded into one weight-streaming launch (g4r_decode_gemm_bf16).
    rope = (cos, sin, rope_cols, pos0, pos_dev); kv = (kcache [B,Lmax,HD], vcache) -- needs rope on the fused q|k|v weight."""
    M, K = x.shape
    N = weight.shape[0]
    dev = _L.require_cuda_same_device([('x', x), ('weight', weight), ('residual', residual)])
    a16 = _act16('decode_gemm', x, weight)
    n_out = N // 2 if act == 'swiglu' else N
    out = torch.empty((M, n_out), dtype=a16, device=dev)
    cos = sin = pos_dev = None
    rope_cols = pos0 = 0
    if rope is not None:
        cos, sin, rope_cols, pos0, pos_dev = rope
    kc = vc = None
    lmax = hd = 0
    if kv is not None:
        kc, vc = kv
        lmax, hd = kc.shape[1], kc.shape[2]
    with torch.cuda.device(dev):
        _ps = _prof_begin(dev)
        _L.check(getattr(_L.load(), _L.sym('g4r_decode_gemm_bf16', a16))(
            _L.ptr(x), x.stride(0), _L.ptr(weight), weight.stride(0), _L.ptr(out), out.stride(0), M, N, K,
            ACT[act], _L.ptr(residual), residual.stride(0) if residual is not None else 0,
            _L.ptr(cos), _L.ptr(sin), int(rope_cols), int(pos0), _L.ptr(pos_dev), _L.ptr(kc), _L.ptr(vc), int(lmax), int(hd),
            _L.stream_ptr(dev)))
        _prof_end(dev, _ps, 'gemm', 2.0 * M * N * K)
    return out
