"""Host wrappers of the training-step kernels (SURVEY.md 8(a) row 14): cross entropy, RMSNorm / SwiGLU /
attention backward, AdamW.  Same rules as kernels.py: CUDA tensors in, raw pointers + current stream to the
C ABI, no fallback."""
import torch

from . import lib as _L

BF16 = torch.bfloat16


def _call(name, dev, *args):
    with torch.cuda.device(dev):
        _L.check(getattr(_L.load(), name)(*args, _L.stream_ptr(dev)))


def cross_entropy(logits, targets, grad_scale=1.0, want_grad=True):
    """logits [M, V] bf16 (unit stride on V); targets int64 [M] already shifted, -100 = ignore
    (llava/model/llava.py:238-249).  Returns (loss fp32 scalar tensor, valid count tensor, dlogits or None)."""
    dev = _L.require_cuda_same_device([('logits', logits), ('targets', targets)])
    if logits.dtype != BF16 or targets.dtype != torch.int64 or logits.dim() != 2 or logits.stride(1) != 1:
        raise TypeError('cross_entropy: logits [M,V] bf16 and int64 targets required')
    M, V = logits.shape
    if targets.numel() != M or not targets.is_contiguous():
        raise RuntimeError('cross_entropy: targets must be contiguous with one entry per logits row')
    row = torch.empty((2, M), dtype=torch.float32, device=dev)
    lc = torch.empty(2, dtype=torch.float32, device=dev)
    # rows padded to a multiple of 64 elements: 16-byte-aligned rows for the dW / dX GEMMs that consume dlogits
    dl = torch.empty((M, (V + 63) // 64 * 64), dtype=BF16, device=dev)[:, :V] if want_grad else None
    _call('g4r_cross_entropy_bf16', dev, _L.ptr(logits), logits.stride(0), _L.ptr(targets), M, V, _L.ptr(row[0]),
          _L.ptr(row[1]), _L.ptr(lc), _L.ptr(dl), dl.stride(0) if want_grad else 0, float(grad_scale))
    _L.count_launches(2 if want_grad else 1)
    return lc[0], lc[1], dl


def rmsnorm_bwd(x, w, dy, eps, dres=None):
    """-> (dx bf16 [M,D], dw fp32 [D]) for y = w * (x * rsqrt(mean(x^2)+eps)).to(bf16); dres (optional, bf16
    [M,D]) is added to dx: the gradient that reaches x through the residual connection around the block."""
    dev = _L.require_cuda_same_device([('x', x), ('w', w), ('dy', dy)])
    M, D = x.shape
    dx = torch.empty((M, D), dtype=BF16, device=dev)
    dw = torch.empty(D, dtype=torch.float32, device=dev)
    S = _L.load().g4r_rmsnorm_bwd_slabs(M)
    slabs = torch.empty((S, D), dtype=torch.float32, device=dev)
    _call('g4r_rmsnorm_bwd_bf16', dev, _L.ptr(x), x.stride(0), _L.ptr(w), _L.ptr(dy), dy.stride(0), _L.ptr(dres),
          dres.stride(0) if dres is not None else 0, _L.ptr(dx), dx.stride(0), _L.ptr(dw), _L.ptr(slabs), M, D,
          float(eps))
    _L.count_launches(1)
    return dx, dw


def colsum(x):
    """fp32 column sums of a bf16 matrix [M,N] (bias gradient of a Linear: sum over rows of grad_y)."""
    M, N = x.shape
    out = torch.empty(N, dtype=torch.float32, device=x.device)
    slabs = torch.empty((_L.load().g4r_colsum_slabs(M), N), dtype=torch.float32, device=x.device)
    _call('g4r_colsum_bf16', x.device, _L.ptr(x), x.stride(0), M, N, _L.ptr(out), _L.ptr(slabs))
    _L.count_launches(1)
    return out


def linear_bwd(x, w, dy, need_dx=True, has_bias=True):
    """Backward of y = x @ w.T + b (torch.nn.functional.linear): returns (dx or None, dw bf16 [N,K], db fp32 [N] or None)."""
    from . import dense
    dw = dense.matmul_t(dy, x, a_mn=True, b_mn=True)
    db = colsum(dy) if has_bias else None
    dx = dense.matmul_t(dy, w, b_mn=True) if need_dx else None
    return dx, dw, db


def pad_nhwc(x):
    """x [n,H,W,C] bf16 -> (padded rows [2*guard + n*(H+2)*(W+2), C], guard) with a zero ring and zero guards."""
    n, H, W, C = x.shape
    guard = W + 3
    out = torch.empty((2 * guard + n * (H + 2) * (W + 2), C), dtype=BF16, device=x.device)
    _call('g4r_pad_nhwc_bf16', x.device, _L.ptr(x), _L.ptr(out), n, H, W, C, guard)
    return out, guard


def conv_weight_flip_t(w):
    """w [Cout, 3, 3, Cin] (rows may be strided: a level slice of [Cout, L, 3, 3, Cin]) -> [Cin, 3, 3, Cout] flipped."""
    Cout, Cin = w.shape[0], w.shape[-1]
    wf = torch.empty((Cin, 3, 3, Cout), dtype=BF16, device=w.device)
    _call('g4r_conv_weight_flip_t_bf16', w.device, _L.ptr(w), w.stride(0), _L.ptr(wf), Cin, Cout)
    return wf


def conv3x3_bwd(x, w, dz, dw_acc=None, need_dx=True, wf=None):
    """Backward of z = conv3x3(x, w) (NHWC bf16, stride 1, pad 1, no bias): x [n,H,W,Cin], w [Cout,3,3,Cin],
    dz [n,H,W,Cout].  Returns (dx bf16 or None, dW fp32 [Cout,3,3,Cin]); dw_acc (fp32) is accumulated into."""
    from . import dense
    n, H, W, Cin = x.shape
    Cout = dz.shape[-1]
    xp, guard = pad_nhwc(x)
    dzp, _ = pad_nhwc(dz)
    rows = n * (H + 2) * (W + 2)
    acc = dw_acc is not None
    dW = dw_acc if acc else torch.empty((Cout, 3, 3, Cin), dtype=torch.float32, device=x.device)
    _call('g4r_conv3x3_dw_bf16', x.device, _L.ptr(dzp[guard:]), _L.ptr(xp[guard - (W + 2) - 1:]), _L.ptr(dW), rows, W + 2,
          Cin, Cout, int(acc))
    dx = None
    if need_dx:
        dx = dense.conv_nhwc(dz, wf if wf is not None else conv_weight_flip_t(w))
    return dx, dW


def gn_relu_bwd(z, dA, scale, shift, stats, count, gamma, dgamma, dbeta, accumulate, eps=1e-5):
    """z bf16 [B,H,W,C]; dA fp32 or bf16 (gradient w.r.t. relu(gn(z))); stats fp32 [B,slots,groups,2] of the forward.
    Returns dz bf16; dgamma / dbeta (fp32 [C]) are written or accumulated in place."""
    B, H, W, C = z.shape
    _, slots, groups, _ = stats.shape
    dz = torch.empty_like(z)
    ws = torch.empty(_L.load().g4r_gn_relu_bwd_workspace(B, H * W, C, groups), dtype=torch.float32, device=z.device)
    _call('g4r_gn_relu_bwd_bf16', z.device, _L.ptr(z), _L.ptr(dA), int(dA.dtype == torch.float32), _L.ptr(scale),
          _L.ptr(shift), _L.ptr(stats), slots, float(count), float(eps), _L.ptr(gamma), _L.ptr(dz), _L.ptr(dgamma),
          _L.ptr(dbeta), int(accumulate), _L.ptr(ws), B, H * W, C, groups)
    _L.count_launches(4)
    return dz


def fuse_consumers(n, m):
    """Inverse of MLVLFuseModule's fuse_lvl_list (layers.py:105-112: level l reads top = min(l+1, n-1) and
    down = max(l-1, 0)): the levels that read level m as their `down` source and as their `top` source."""
    dn = [l for l in range(n) if max(l - 1, 0) == m]
    tp = [l for l in range(n) if min(l + 1, n - 1) == m]
    return dn, tp


def fuse_gather_bwd(d_in, m):
    """d_in: list (per level) of conv-input gradients bf16 [B,H_l,H_l,C] of one fuse round; returns the fp32 gradient
    w.r.t. the previous round's activated maps of level m (adjoint of kernels.fuse_gather)."""
    n = len(d_in)
    B, H, _, C = d_in[m].shape
    dn, tp = fuse_consumers(n, m)
    out = torch.empty((B, H, H, C), dtype=torch.float32, device=d_in[m].device)

    def pair(ls, i):
        return (_L.ptr(d_in[ls[i]]), d_in[ls[i]].shape[1]) if i < len(ls) else (None, 0)
    a, b, c, d = pair(dn, 0), pair(dn, 1), pair(tp, 0), pair(tp, 1)
    _call('g4r_fuse_gather_bwd', out.device, _L.ptr(d_in[m]), H, a[0], a[1], b[0], b[1], c[0], c[1], d[0], d[1],
          _L.ptr(out), B, C)
    return out


def pos_embed_mlp_bwd(boxes, params, dout, eps=1e-5):
    """boxes fp32 [K,4]; params = (w0, b0, g2, be2, w3, b3, g5, be5) bf16; dout bf16 [K,1024].
    Returns a dict name -> fp32 gradient for pos_embedd.{0,2,3,5}.{weight,bias}."""
    w0, b0, g2, be2, w3, b3, g5, be5 = params
    K = boxes.shape[0]
    n = _L.load().g4r_pos_embed_mlp_grad_size()
    grads = torch.empty(n, dtype=torch.float32, device=boxes.device)
    slabs = torch.empty((K, n), dtype=torch.float32, device=boxes.device)
    _call('g4r_pos_embed_mlp_bwd', boxes.device, _L.ptr(boxes), _L.ptr(w0), _L.ptr(b0), _L.ptr(g2), _L.ptr(be2), _L.ptr(w3),
          _L.ptr(b3), _L.ptr(g5), _L.ptr(dout), dout.stride(0), _L.ptr(grads), _L.ptr(slabs), K, float(eps))
    o, out = 0, {}
    for name, shape in (('0.weight', (256, 4)), ('0.bias', (256,)), ('2.weight', (256,)), ('2.bias', (256,)),
                        ('3.weight', (1024, 256)), ('3.bias', (1024,)), ('5.weight', (1024,)), ('5.bias', (1024,))):
        cnt = 1
        for d in shape:
            cnt *= d
        out[name] = grads[o:o + cnt].view(shape)
        o += cnt
    return out


def relu_bwd(dy, y):
    out = torch.empty_like(dy)
    _call('g4r_relu_bwd_bf16', dy.device, _L.ptr(dy), _L.ptr(y), _L.ptr(out), dy.numel())
    return out


def cast_f32_bf16(x):
    """contiguous fp32 [N, D] -> bf16 [N, D] (g4r_cast_f32_bf16)."""
    N, D = x.shape
    out = torch.empty((N, D), dtype=BF16, device=x.device)
    _call('g4r_cast_f32_bf16', x.device, _L.ptr(x), D, 0, _L.ptr(out), 1, N, D)
    return out


def swiglu_fwd(gu):
    """gu [M, 2F] interleaved (gate_j, up_j) -> silu(gate) * up  [M, F]."""
    M, F2 = gu.shape
    f = torch.empty((M, F2 // 2), dtype=BF16, device=gu.device)
    _call('g4r_swiglu_fwd_bf16', gu.device, _L.ptr(gu), gu.stride(0), _L.ptr(f), f.stride(0), M, F2 // 2)
    return f


def swiglu_bwd(gu, df):
    M, F2 = gu.shape
    dgu = torch.empty((M, F2), dtype=BF16, device=gu.device)
    _call('g4r_swiglu_bwd_bf16', gu.device, _L.ptr(gu), gu.stride(0), _L.ptr(df), df.stride(0), _L.ptr(dgu),
          dgu.stride(0), M, F2 // 2)
    return dgu


def attention_fwd_lse(qkv, B, L, n_heads, head_dim, causal, scale):
    """Training forward on packed qkv rows [B*L, 3*H*D]: returns (out [B*L, H*D] bf16, lse [B,H,L] fp32)."""
    hid = n_heads * head_dim
    out = torch.empty((B * L, hid), dtype=BF16, device=qkv.device)
    lse = torch.empty((B, n_heads, L), dtype=torch.float32, device=qkv.device)
    ld = qkv.stride(0)
    _call('g4r_attention_tc_lse_bf16', qkv.device, _L.ptr(qkv), _L.ptr(qkv[:, hid:]), _L.ptr(qkv[:, 2 * hid:]),
          _L.ptr(out), ld, L * ld, hid, L * hid, B, n_heads, L, head_dim, int(causal), float(scale), _L.ptr(lse))
    return out, lse


def attention_bwd(qkv, out, dout, lse, B, L, n_heads, head_dim, causal, scale):
    """-> dqkv [B*L, 3*H*D] bf16 (dQ | dK | dV), gradients w.r.t. the post-RoPE q, k and v."""
    hid = n_heads * head_dim
    dqkv = torch.empty((B * L, 3 * hid), dtype=BF16, device=qkv.device)
    delta = torch.empty((B, n_heads, L), dtype=torch.float32, device=qkv.device)
    ld = qkv.stride(0)
    _call('g4r_attention_bwd_bf16', qkv.device, _L.ptr(qkv), _L.ptr(qkv[:, hid:]), _L.ptr(qkv[:, 2 * hid:]),
          _L.ptr(out), _L.ptr(dout), _L.ptr(lse), _L.ptr(delta), _L.ptr(dqkv), _L.ptr(dqkv[:, hid:]),
          _L.ptr(dqkv[:, 2 * hid:]), ld, L * ld, out.stride(0), L * out.stride(0), dqkv.stride(0),
          L * dqkv.stride(0), B, n_heads, L, head_dim, int(causal), float(scale))
    _L.count_launches(2)
    return dqkv


def grad_sumsq(tensors, slabs=None):
    """Per-CTA partial sums of squares of every gradient tensor (bf16 / fp32, contiguous) into one fp32 slab
    buffer [len(tensors), g4r_sumsq_slabs()]; feeds clip_coef.  Fixed summation order: reproducible."""
    n = _L.load().g4r_sumsq_slabs()
    dev = tensors[0].device
    if slabs is None:
        slabs = torch.empty((len(tensors), n), dtype=torch.float32, device=dev)
    for i, t in enumerate(tensors):
        if t.dtype not in (BF16, torch.float32) or not t.is_contiguous():
            raise TypeError('grad_sumsq: contiguous bf16/fp32 tensors required')
        _call('g4r_sumsq', dev, _L.ptr(t), int(t.dtype == BF16), t.numel(), _L.ptr(slabs[i]))
    return slabs


def clip_coef(slabs, max_norm, pre_scale=1.0):
    """-> device fp32 [2] = (total gradient norm * pre_scale, min(1, max_norm / (norm + 1e-6))):
    torch.nn.utils.clip_grad_norm_ semantics (what HF Trainer applies with max_grad_norm=1.0), no host sync."""
    out = torch.empty(2, dtype=torch.float32, device=slabs.device)
    _call('g4r_grad_clip_coef', slabs.device, _L.ptr(slabs), slabs.numel(), float(pre_scale), float(max_norm), _L.ptr(out))
    return out


def adamw_step(p32, grad, m, v, p16, lr, betas, eps, weight_decay, step, grad_scale=1.0, scale_dev=None):
    """In-place torch.optim.AdamW update of the fp32 master `p32` (+ bf16 copy `p16`, optional).
    scale_dev: optional device float multiplied into grad_scale (clip_coef(...)[1:])."""
    n = p32.numel()
    if not (p32.is_contiguous() and grad.is_contiguous() and m.is_contiguous() and v.is_contiguous()):
        raise RuntimeError('adamw_step: contiguous tensors required')
    if grad.dtype not in (BF16, torch.float32) or grad.numel() != n:
        raise TypeError('adamw_step: grad must be bf16 or fp32 with the parameter\'s size')
    _call('g4r_adamw_step_ex', p32.device, _L.ptr(p32), _L.ptr(grad), int(grad.dtype == BF16), _L.ptr(m), _L.ptr(v),
          _L.ptr(p16), n, float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step),
          float(grad_scale), _L.ptr(scale_dev))
