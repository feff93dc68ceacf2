"""Torch-tensor front-ends of the elementwise / attention entry points of the C ABI
(csrc/elementwise.cu, csrc/attention.cu).  No computation happens in Python."""
import torch

from . import lib as _L


def _call(fn_name, dev, *args, act=torch.bfloat16):
    """act: the 16-bit storage type of the call's tensors -- selects the bf16 entry point or its fp16 twin."""
    with torch.cuda.device(dev):
        _L.check(getattr(_L.load(), _L.sym(fn_name, act))(*args, _L.stream_ptr(dev)))


def _bf16(*ts):
    """All given tensors share one 16-bit storage type (bf16, or fp16 for the demo's dtype); returns it."""
    dt = None
    for t in ts:
        if t is None:
            continue
        if t.dtype not in (torch.bfloat16, torch.float16) or (dt is not None and t.dtype != dt):
            raise TypeError('bf16 (or all-fp16) tensors required, got %s' % ', '.join(str(u.dtype) for u in ts if u is not None))
        dt = t.dtype
    return dt


def layernorm(x, weight, bias, eps=1e-5, out=None):
    act = _bf16(x, weight, bias)
    D = x.shape[-1]
    x2 = x.reshape(-1, D)
    out = torch.empty_like(x2) if out is None else out
    _call('g4r_layernorm_bf16', x.device, _L.ptr(x2), x2.stride(0), _L.ptr(weight), _L.ptr(bias), _L.ptr(out),
          out.stride(0), x2.shape[0], D, float(eps), act=act)
    return out.view(x.shape) if out.is_contiguous() and out.numel() == x.numel() else out


def layernorm_ex(x, weight, bias, eps=1e-5, out_dtype=None):
    """LayerNorm with 16-bit/fp32 input rows and 16-bit/fp32 output rows (CLIP's fp32 residual stream); the 16-bit
    type is the weight's."""
    act = _bf16(weight, bias)
    out_dtype = act if out_dtype is None else out_dtype
    if x.dtype not in (act, torch.float32) or out_dtype not in (act, torch.float32):
        raise TypeError('layernorm_ex: rows must be %s or fp32, got %s -> %s' % (act, x.dtype, out_dtype))
    D = x.shape[-1]
    x2 = x.reshape(-1, D)
    out = torch.empty(x2.shape, dtype=out_dtype, device=x.device)
    _call('g4r_layernorm_ex', x.device, _L.ptr(x2), x2.stride(0), int(x.dtype == torch.float32), _L.ptr(weight),
          _L.ptr(bias), _L.ptr(out), out.stride(0), int(out_dtype == torch.float32), x2.shape[0], D, float(eps), act=act)
    return out.view(x.shape)


def cast_tokens_f32_bf16(hidden, skip_first=1, dtype=torch.bfloat16):
    """hidden fp32 [B,T,C] -> dense 16-bit [B*(T-skip_first), C] (drops the CLS row)."""
    B, T, C = hidden.shape
    out = torch.empty((B * (T - skip_first), C), dtype=dtype, device=hidden.device)
    import ctypes
    src = ctypes.c_void_p(hidden.data_ptr() + skip_first * C * 4)
    _call('g4r_cast_f32_bf16', hidden.device, src, C, T * C, _L.ptr(out), B, T - skip_first, C, act=dtype)
    return out


def rmsnorm(x, weight, eps=1e-6, out=None):
    """x 16-bit (the weight's type) or fp32 rows (an fp32 residual stream); 16-bit output."""
    act = _bf16(weight)
    if x.dtype not in (act, torch.float32):
        raise TypeError('rmsnorm: %s or fp32 rows required, got %s' % (act, x.dtype))
    D = x.shape[-1]
    x2 = x.reshape(-1, D)
    out = torch.empty(x2.shape, dtype=act, device=x.device) if out is None else out
    _call('g4r_rmsnorm_ex', x.device, _L.ptr(x2), x2.stride(0), int(x.dtype == torch.float32), _L.ptr(weight),
          _L.ptr(out), out.stride(0), x2.shape[0], D, float(eps), act=act)
    return out.view(x.shape) if out.is_contiguous() and out.numel() == x.numel() else out


def rope_inplace(qkv, cos, sin, L, n_heads_qk, head_dim):
    """qkv [rows, width] packed; rotates the first n_heads_qk heads of every row in place."""
    act = _bf16(qkv, cos, sin)
    _call('g4r_rope_inplace_bf16', qkv.device, _L.ptr(qkv), qkv.stride(0), _L.ptr(cos), _L.ptr(sin),
          qkv.shape[0], int(L), int(n_heads_qk), int(head_dim), act=act)
    return qkv


def attention(qkv, B, L, n_heads, head_dim, causal, scale, out=None, seqlens=None, impl='tc'):
    """qkv: packed bf16 [B*L, 3*n_heads*head_dim] = (q | k | v); returns [B*L, n_heads*head_dim].
    impl: 'tc' the tcgen05 kernel; 'mma' the mma.sync kernel, kept as the tests' cross-check."""
    act = _bf16(qkv)
    hd = n_heads * head_dim
    if out is None:
        out = torch.empty((B * L, hd), dtype=act, device=qkv.device)
    ld = qkv.stride(0)
    esz = 2
    base = qkv.data_ptr()
    import ctypes
    q, k, v = (ctypes.c_void_p(base + i * hd * esz) for i in range(3))
    fn = {'tc': 'g4r_attention_tc_bf16', 'mma': 'g4r_attention_bf16'}[impl]
    _call(fn, qkv.device, q, k, v, _L.ptr(out), ld, L * ld, out.stride(0), L * out.stride(0),
          B, n_heads, L, head_dim, int(bool(causal)), float(scale), _L.ptr(seqlens), act=act)
    return out


def patchify(images, ps, kpad):
    act = _bf16(images)
    B, _, S, _ = images.shape
    G = S // ps
    out = torch.empty((B * G * G, kpad), dtype=act, device=images.device)
    _call('g4r_patchify_bf16', images.device, _L.ptr(images.contiguous()), _L.ptr(out), B, S, ps, kpad, act=act)
    return out


def vit_embed(patch, cls, pos, B, P):
    act = _bf16(patch, cls, pos)
    D = patch.shape[-1]
    out = torch.empty((B, P + 1, D), dtype=act, device=patch.device)
    _call('g4r_vit_embed_bf16', patch.device, _L.ptr(patch), _L.ptr(cls), _L.ptr(pos), _L.ptr(out), B, P, D, act=act)
    return out


def upsample_tokens_coords(hidden, G, Ho, cpad, has_cls=True, dtype=None):
    """hidden: [B, 1+G*G, C] ViT hidden state, 16-bit or fp32 (CLS first; has_cls=False: [B, G*G, C]);
    returns 16-bit NHWC [B,Ho,Ho,cpad] (`dtype`: the 16-bit type for fp32 tokens, default bf16)."""
    B, T, C = hidden.shape
    skip = 1 if has_cls else 0
    if T != G * G + skip or not hidden.is_contiguous() or hidden.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        raise RuntimeError('upsample_tokens_coords: contiguous bf16/fp16/fp32 [B,%d,C] tokens required, got %s %s'
                           % (G * G + skip, tuple(hidden.shape), hidden.dtype))
    act = hidden.dtype if hidden.dtype != torch.float32 else (dtype or torch.bfloat16)
    out = torch.empty((B, Ho, Ho, cpad), dtype=act, device=hidden.device)
    import ctypes
    f32 = hidden.dtype == torch.float32
    tok = ctypes.c_void_p(hidden.data_ptr() + skip * C * (4 if f32 else 2))  # skip CLS
    _call('g4r_upsample_tokens_coords_f32' if f32 else 'g4r_upsample_tokens_coords_bf16', hidden.device, tok, C,
          T * C, _L.ptr(out), B, G, Ho, C, cpad, act=act)
    return out


def fuse_gather(own, top, down, own_ss=None, top_ss=None, down_ss=None, out=None):
    """own/top/down: NHWC bf16 [B,H,H,C]; *_ss: optional (scale, shift) fp32 [B,C] pairs."""
    act = _bf16(own, top, down)
    B, H, _, C = own.shape
    out = torch.empty_like(own) if out is None else out

    def ss(p):
        return (None, None) if p is None else (_L.ptr(p[0]), _L.ptr(p[1]))
    a, b, c = ss(own_ss), ss(top_ss), ss(down_ss)
    _call('g4r_fuse_gather_bf16', own.device, _L.ptr(own), a[0], a[1], H, _L.ptr(top), b[0], b[1], top.shape[1],
          _L.ptr(down), c[0], c[1], down.shape[1], _L.ptr(out), B, C, act=act)
    return out


def gn_finalize(stats, gamma, beta, count, eps=1e-5):
    """stats: fp32 [B, slots, groups, 2] partial sums from dense.conv_nhwc(gn_stats=...)."""
    B, slots, groups, _ = stats.shape
    C = gamma.shape[0]
    scale = torch.empty((B, C), dtype=torch.float32, device=stats.device)
    shift = torch.empty_like(scale)
    _call('g4r_gn_finalize', stats.device, _L.ptr(stats), _L.ptr(gamma), _L.ptr(beta), _L.ptr(scale),
          _L.ptr(shift), B, C, groups, slots, float(count), float(eps), act=_bf16(gamma, beta))
    return scale, shift


def affine_relu_nhwc(z, scale, shift):
    """z bf16 NHWC [B,H,W,C], scale/shift fp32 [B,C] (gn_finalize) -> relu(z*scale+shift) bf16 NHWC."""
    act = _bf16(z)
    B, H, W, C = z.shape
    out = torch.empty_like(z)
    _call('g4r_affine_relu_nhwc_bf16', z.device, _L.ptr(z), _L.ptr(scale), _L.ptr(shift), _L.ptr(out), B, H * W, C, act=act)
    return out


def pos_embed_mlp(boxes, w0, b0, g2, be2, w3, b3, g5, be5, eps=1e-5):
    K = boxes.shape[0]
    out = torch.empty((K, 1024), dtype=torch.float32, device=boxes.device)
    if K:
        _call('g4r_pos_embed_mlp', boxes.device, _L.ptr(boxes), _L.ptr(w0), _L.ptr(b0), _L.ptr(g2), _L.ptr(be2),
              _L.ptr(w3), _L.ptr(b3), _L.ptr(g5), _L.ptr(be5), _L.ptr(out), K, float(eps),
              act=_bf16(w0, b0, g2, be2, w3, b3, g5, be5))
    return out


def add_bias_pos_cast(acc, bias, pos):
    """acc: fp32 [splits, K, D] (split-K slabs) or [K, D]."""
    if acc.dim() == 2:
        acc = acc[None]
    splits, K, D = acc.shape
    act = _bf16(bias)
    out = torch.empty((K, D), dtype=act, device=acc.device)
    if K:
        _call('g4r_add_bias_pos_cast', acc.device, _L.ptr(acc), splits, _L.ptr(bias), _L.ptr(pos), _L.ptr(out), K, D, act=act)
    return out


def kv_append(qkv, kcache, vcache, B, Ln, pos0, pos_dev=None):
    """Copy the k|v parts of packed qkv rows [B*Ln, 3*HD] into caches [B, Lmax, HD] at pos0..pos0+Ln-1."""
    HD = kcache.shape[-1]
    _call('g4r_kv_append_bf16', qkv.device, _L.ptr(qkv), qkv.stride(0), _L.ptr(kcache), _L.ptr(vcache), B, Ln,
          int(pos0), _L.ptr(pos_dev), kcache.shape[1], HD, act=_bf16(qkv, kcache, vcache))


def decode_attention(qkv, kcache, vcache, B, n_heads, head_dim, kv_len, scale, pos_dev=None):
    """qkv [B, 3*HD] (one new token per sample); caches [B, Lmax, HD]; returns [B, HD]."""
    act = _bf16(qkv, kcache, vcache)
    out = torch.empty((B, n_heads * head_dim), dtype=act, device=qkv.device)
    _call('g4r_decode_attention_bf16', qkv.device, _L.ptr(qkv), qkv.stride(0), _L.ptr(kcache), _L.ptr(vcache),
          _L.ptr(out), out.stride(0), B, n_heads, head_dim, int(kv_len), _L.ptr(pos_dev), kcache.shape[1], float(scale),
          act=act)
    return out
