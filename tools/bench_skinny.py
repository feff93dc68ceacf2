"""Per-kernel timing of the decode step's kernels at 7B shapes, warm (back-to-back launches inside one
CUDA graph, weights rotated over several copies so that every launch streams from HBM, not L2).
usage: python tools/bench_skinny.py [batch] [--pdl]"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gpt4roi_b200 import dense, kernels  # noqa: E402

DEV = 'cuda:0'
BF = torch.bfloat16


def timed_graph(fn, n_iter=5):
    """fn() enqueues R launches; capture once, replay n_iter times, return ms per fn() call."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_iter):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n_iter


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('batch', nargs='?', type=int, default=8)
    ap.add_argument('--pdl', action='store_true', help='launch the chain the way the decode step does (programmatic dependent launch)')
    args = ap.parse_args()
    B = args.batch
    if args.pdl:
        from gpt4roi_b200 import lib
        lib.set_pdl(True)
    hid, ffn, H, D, V = 4096, 11008, 32, 128, 32006
    R = 8   # weight copies (>= 33 MB each -> well past the 126 MB L2 in rotation)
    torch.manual_seed(0)
    x = (torch.randn(B, hid, device=DEV) * 0.5).to(BF)
    xf = (torch.randn(B, ffn, device=DEV) * 0.5).to(BF)
    res = torch.randn(B, hid, device=DEV).to(BF)
    Lmax = 1024
    inv = 1.0 / (10000.0 ** (torch.arange(0, D, 2).float() / D))
    emb = torch.cat([torch.arange(Lmax).float()[:, None] * inv[None]] * 2, -1)
    cos, sin = emb.cos().to(DEV, BF).contiguous(), emb.sin().to(DEV, BF).contiguous()
    out = []

    def report(name, ms_total, launches, bytes_per_launch):
        us = ms_total * 1e3 / launches
        rec = dict(kernel=name, batch=B, us_per_launch=round(us, 2), MB_per_launch=round(bytes_per_launch / 1e6, 2),
                   GBps=round(bytes_per_launch / us / 1e3, 1))
        out.append(rec)
        print(json.dumps(rec), flush=True)

    def wset(n, k):
        return [(torch.randn(n, k, device=DEV) * 0.02).to(BF) for _ in range(R)]

    w = wset(3 * hid, hid)
    report('skinny qkv+rope 12288x4096', timed_graph(lambda: [dense.qkv_rope(x, wi, cos, sin, 1, 2 * hid, pos0=700) for wi in w]), R, 3 * hid * hid * 2)
    kc, vc = (torch.empty(B, Lmax, hid, device=DEV, dtype=BF) for _ in range(2))
    report('decode_gemm qkv+rope+kv 12288x4096',
           timed_graph(lambda: [dense.decode_gemm(x, wi, rope=(cos, sin, 2 * hid, 700, None), kv=(kc, vc)) for wi in w]), R,
           3 * hid * hid * 2)
    del w, kc, vc
    w = wset(hid, hid)
    report('skinny wo+residual 4096x4096', timed_graph(lambda: [dense.linear(x, wi, residual=res) for wi in w]), R, hid * hid * 2)
    del w
    w = wset(2 * ffn, hid)
    report('skinny gate/up swiglu 22016x4096', timed_graph(lambda: [dense.linear(x, wi, act='swiglu') for wi in w]), R, 2 * ffn * hid * 2)
    report('decode_gemm gate/up swiglu 22016x4096', timed_graph(lambda: [dense.decode_gemm(x, wi, act='swiglu') for wi in w]), R,
           2 * ffn * hid * 2)
    del w
    w = wset(hid, ffn)
    report('skinny down+residual 4096x11008', timed_graph(lambda: [dense.linear(xf, wi, residual=res) for wi in w]), R, ffn * hid * 2)
    del w
    w = wset(V, hid)
    report('skinny lm_head 32006x4096', timed_graph(lambda: [dense.linear(x, wi) for wi in w[:4]]), 4, V * hid * 2)
    del w
    g = torch.ones(hid, device=DEV, dtype=BF)
    report('rmsnorm', timed_graph(lambda: [kernels.rmsnorm(x, g, 1e-6) for _ in range(32)]), 32, 2 * B * hid * 2)
    for kv_len in (706, 1024):
        caches = [(torch.randn(B, Lmax, H * D, device=DEV).to(BF), torch.randn(B, Lmax, H * D, device=DEV).to(BF)) for _ in range(R)]
        qkv = torch.randn(B, 3 * H * D, device=DEV).to(BF)
        report('decode_attention kv_len=%d' % kv_len,
               timed_graph(lambda: [kernels.decode_attention(qkv, k, v, B, H, D, kv_len, D ** -0.5) for k, v in caches]), R,
               2 * B * kv_len * H * D * 2)
        report('kv_append', timed_graph(lambda: [kernels.kv_append(qkv, k, v, B, 1, 700) for k, v in caches]), R, 2 * B * H * D * 2 * 2)
        del caches
    os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)


if __name__ == '__main__':
    main()
