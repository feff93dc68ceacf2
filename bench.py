#!/usr/bin/env python
"""bench.py -- GPT4RoI region-token prefill throughput on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank/GPU)
  python bench.py --impl reference ...                     (the reference's CPU path, bounded sample)
  python bench.py ... --dump-outputs DIR                   (also save a fixed sample of the last timed step's logits)

A step = one prefill of the headline workload (configs[1]): batch 8, 336 px image, 8 RoIs per
image, 128 text tokens -> L = 706, CLIP-ViT-L/14 + SPI module + LLaMA-7B + lm_head, bf16, random-init
weights of the real architecture, synthetic inputs.  Prints ONE JSON line (rank 0).

Beside the headline the line carries, as extras measured in the same run (each under its own key, none of them
changes `value`): the RoIAlign microbench at the BASELINE size (configs[4], `roialign_roofline`), configs[2]'s
16-RoI variant (`config2_16roi`), the stage-2 / stage-1 training step of configs[3] at the rank count of the run
(`train_step`: DDP over NCCL, exposed all-reduce time), and the decode loop (`decode`, N=1 only).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(batch_per_gpu=8, image_size=336, rois_per_image=8, text_tokens=128)
# algorithmic FLOPs per sample of the headline workload (SURVEY.md App. B, 2*MAC), with the 23 CLIP layers that
# feed hidden_states[-2] (the 24th layer and post-LN are dead work for mm_vision_select_layer=-2, SURVEY 8(a)1)
FLOPS_PER_SAMPLE = 14.69e12 - (0.382e12 - 0.366e12)
METRIC = 'samples_per_sec_prefill_336px_8roi_128tok_7b'


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return p, 'measured'
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0), 'fallback'


class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 8 and r[1].replace('.', '').isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 8 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) > 8 for n, v in zip(names, r[5:9]) if v.lower().startswith('active')})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm))


def synthetic_inputs(cfg, B, k_per_img, T, seed=0):
    import torch
    g = torch.Generator().manual_seed(seed)
    P = cfg.num_patches
    L = T + P + 2
    ids = torch.randint(3, 32000, (B, L), generator=g)
    boxes = []
    for b in range(B):
        ids[b, 0] = 1
        ids[b, 1] = cfg.im_start_token
        ids[b, 2:2 + P] = cfg.im_patch_token
        ids[b, 2 + P] = cfg.im_end_token
        pos = torch.randperm(L - (3 + P), generator=g)[:k_per_img] + 3 + P
        ids[b, pos] = cfg.bbox_token
        p = torch.rand(k_per_img, 2, 2, generator=g).sort(dim=1).values
        bx = torch.cat([p[:, 0, :], p[:, 1, :]], 1)
        bx[:, 2:] = torch.maximum(bx[:, 2:], bx[:, :2] + 2.0 / cfg.image_size).clamp(max=1.0)
        boxes.append(bx)
    images = torch.randn(B, 3, cfg.image_size, cfg.image_size, generator=g).to(getattr(cfg, 'torch_dtype', torch.bfloat16))
    return ids, images, boxes


# ---------------------------------------------------------------------------------------------
# CPU baseline: the reference's path (PyTorch-CPU + transformers + mmcv-CPU RoIAlign) on a BOUNDED
# sample of ONE headline sample.
# ---------------------------------------------------------------------------------------------
def cgroup_cpu_limit():
    """CPUs this process may actually use: the cgroup CFS quota (v2 cpu.max, v1 cpu.cfs_quota_us) when one is
    set, else None.  The affinity mask alone over-counts on shared hosts (a 128-CPU mask over a 16-CPU quota makes
    a 128-thread OpenMP pool thrash -- the 60x swing of round 1's CPU arm)."""
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if q != 'max':
            return max(1, int(math.ceil(float(q) / float(p))))
    except Exception:
        pass
    for base in ('/sys/fs/cgroup/cpu', '/sys/fs/cgroup/cpu,cpuacct'):
        try:
            q = int(open(base + '/cpu.cfs_quota_us').read())
            p = int(open(base + '/cpu.cfs_period_us').read())
            if q > 0 and p > 0:
                return max(1, int(math.ceil(q / p)))
        except Exception:
            pass
    return None


def pick_cpu_threads():
    """Thread count for the CPU arm: min(affinity, cgroup quota), then a 1-second calibration over
    {n, n/2, n/4} with an fp32 GEMM keeps the fastest (hyper-thread siblings / hidden limits)."""
    import torch
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = cgroup_cpu_limit()
    cap = min(aff, quota) if quota else aff
    cands = sorted({max(1, cap), max(1, cap // 2), max(1, cap // 4)}, reverse=True)
    a, b = torch.randn(1024, 2048), torch.randn(2048, 2048)
    rates = {}
    for n in cands:
        torch.set_num_threads(n)
        torch.mm(a, b)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 0.3:
            torch.mm(a, b)
            reps += 1
        rates[n] = reps * 2.0 * 1024 * 2048 * 2048 / (time.perf_counter() - t0) / 1e9
    best = max(rates, key=lambda n: rates[n])
    torch.set_num_threads(best)
    return best, dict(affinity=aff, cgroup_quota_cpus=quota, calibration_gflops={str(k): round(v, 1) for k, v in rates.items()})


def cpu_reference_sample(repeats=3):
    """One headline sample (336 px, 8 RoIs, L = 706) on the host cores, fp32.
      * SPI module: IN FULL -- the reference's own modules (gpt4roi/models/layers.py under tests/golden/ref_shims.py)
        when /root/reference exists, else their pinned restatement oracle/spi_oracle.py; RoIAlign = the reference's
        own cpu/roi_align.cpp compiled in place (oracle/_ref) when present, else the C port;
      * mm_projector, lm_head: in full;  ViT: 1 of 24 encoder layers x24, LLaMA: 1 of 32 decoder layers x32
        (transformers' own layers; the stacks are 24 / 32 identical layers, the whole 7B fp32 forward would need
        27 GB and minutes) -- the line says `extrapolated: true` and carries the real wall-clock of the sample.
    `repeats` timed repeats after one warm-up each; value = median, spread = (max-min)/median."""
    import numpy as np
    import torch
    import torch.nn.functional as F
    from gpt4roi_b200.engine import EngineConfig, random_state_dicts
    torch.set_grad_enabled(False)
    t_wall = time.perf_counter()
    cores, cpu_info = pick_cpu_threads()
    tiny = os.environ.get('G4R_BENCH_TINY') == '1'   # CPU unit test only: same code path, toy sizes
    cfg = EngineConfig(image_size=56 if tiny else WORKLOAD['image_size'], n_layers=0, vit_layers=0)
    S, K, T = cfg.image_size, (1 if tiny else WORKLOAD['rois_per_image']), (4 if tiny else WORKLOAD['text_tokens'])
    L = T + cfg.num_patches + 2
    reps = 1 if tiny else repeats

    def timeit(fn):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return ts

    stages = {}
    # ---- ViT: 1 encoder layer of 24 (reference runs all 24, llava.py:126)
    from transformers import CLIPVisionConfig
    from transformers.models.clip.modeling_clip import CLIPEncoderLayer
    vc = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24,
                          num_attention_heads=16, image_size=S, patch_size=14)
    vc._attn_implementation = 'eager'
    vl = CLIPEncoderLayer(vc).eval()
    xv = torch.randn(1, cfg.num_patches + 1, 1024)
    try:
        vl(xv, None, None)
        stages['vit'] = [24 * t for t in timeit(lambda: vl(xv, None, None))]
    except TypeError:
        stages['vit'] = [24 * t for t in timeit(lambda: vl(xv, attention_mask=None))]
    # ---- SPI module in full
    sd, _ = random_state_dicts(cfg, 'cpu', seed=0, dtype=torch.float32)
    toks = [torch.randn(1, cfg.num_patches, 1024) for _ in range(4)]
    p = torch.rand(K, 2, 2).sort(dim=1).values
    boxes = [torch.cat([p[:, 0, :], p[:, 1, :]], 1)]
    boxes[0][:, 2:] = torch.maximum(boxes[0][:, 2:], boxes[0][:, :2] + 2.0 / S).clamp(max=1.0)
    ext, kind, spi_kind = None, 'port', None
    try:
        from oracle import build_ref
        ext = build_ref.load()
    except Exception:
        ext = None
    spi_fn, saved = None, None
    if ext is not None:
        kind = 'reference'
    if os.path.isdir('/root/reference') and not tiny:
        try:   # the reference's OWN MLVLROIQueryModule (unmodified; 336: the three literals lifted, SURVEY 8(c))
            from tests.golden import ref_shims
            mod = ref_shims.build_roi_query_module(S)
            mod.load_state_dict({k[len('model.spi_module.'):]: v for k, v in sd.items() if k.startswith('model.spi_module.')})
            mod = mod.eval()
            spi_fn = lambda: mod([t.clone() for t in toks], boxes)
            spi_kind = 'reference modules (gpt4roi/models/layers.py under ref_shims) + reference cpu/roi_align.cpp'
            spi_fn()
        except Exception as e:
            spi_fn, spi_kind = None, None
    if spi_fn is None:
        from oracle import spi_oracle
        if ext is not None:
            e0 = torch.zeros(0)

            def ref_roi_align(x, rois, out_size, scale, sampling):
                o = x.new_zeros(rois.shape[0], x.shape[1], out_size, out_size)
                ext.roi_align_forward(x.contiguous(), rois.contiguous(), o, e0, e0, aligned_height=out_size,
                                      aligned_width=out_size, spatial_scale=float(np.float32(scale)),
                                      sampling_ratio=sampling, pool_mode=1, aligned=True)
                return o
            spi_oracle_roi = ref_roi_align
        else:
            from oracle import roi_align_oracle as O

            def spi_oracle_roi(x, rois, out_size, scale, sampling):
                return torch.from_numpy(O.roi_align_forward(x.numpy(), rois.numpy(), out_size, scale, sampling, 'avg', True)[0])
        saved = spi_oracle._roi_align
        spi_oracle._roi_align = spi_oracle_roi
        spi_fn = lambda: spi_oracle.roi_query_forward(sd, toks, boxes, S)
        spi_kind = 'oracle/spi_oracle.py (restatement pinned to the reference modules by tests/golden) + %s RoIAlign' % \
                   ('reference cpu/roi_align.cpp (oracle/_ref)' if ext is not None else 'C-port')
    stages['spi_module'] = timeit(spi_fn)
    if saved is not None:
        spi_oracle._roi_align = saved
    wp = sd['model.mm_projector.weight']
    stages['mm_projector'] = timeit(lambda: F.linear(toks[0][0], wp))
    # ---- LLaMA: 1 decoder layer of 32 at L tokens + lm_head in full
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding
    hid, inter, V = (256, 512, 1000) if tiny else (4096, 11008, 32006)
    lc = LlamaConfig(hidden_size=hid, intermediate_size=inter, num_hidden_layers=32, num_attention_heads=32,
                     num_key_value_heads=32, vocab_size=V)
    lc._attn_implementation = 'eager'
    dl = LlamaDecoderLayer(lc, 0).eval()
    xl = torch.randn(1, L, hid)
    pos_ids = torch.arange(L)[None]
    pe = LlamaRotaryEmbedding(lc)(xl, pos_ids)
    mask = torch.full((L, L), float('-inf')).triu(1)[None, None]
    stages['llama'] = [32 * t for t in timeit(lambda: dl(xl, attention_mask=mask, position_ids=pos_ids, position_embeddings=pe))]
    wl = torch.randn(V, hid) * 0.02
    stages['lm_head'] = timeit(lambda: F.linear(xl[0], wl))
    per_rep = [sum(stages[k][i] for k in stages) for i in range(reps)]
    med = sorted(per_rep)[len(per_rep) // 2]
    spread = (max(per_rep) - min(per_rep)) / med if med > 0 else 0.0
    sample = ('1 sample (336px, 8 RoIs, L=%d), fp32 on %d host threads: SPI module in full [%s]; mm_projector and lm_head in '
              'full; 1 of 24 CLIP layers x24 and 1 of 32 LLaMA layers x32 (transformers layers); %d timed repeats after a '
              'warm-up, median' % (L, cores, spi_kind, reps))
    return dict(value=1.0 / med, unit='samples/s', cores=cores, kind=kind, sample=sample, extrapolated=True,
                seconds_per_sample_median=med, repeat_seconds=[round(v, 3) for v in per_rep], spread=round(spread, 4),
                wall_clock_s=round(time.perf_counter() - t_wall, 2), cpu=cpu_info,
                stage_seconds={k: round(sorted(v)[len(v) // 2], 3) for k, v in stages.items()})


def roialign_microbench(dev, pk, how, n_maps=256, rois_per_map=100):
    """BASELINE configs[4] at its full size: 256 images x 4-level 224-pyramid (128,64,32,16) x 1024 ch NHWC fp32,
    100 RoIs per image (K = 25 600), 7x7, sampling 2, ONE fused launch (43 GB of operands).  achieved = algorithmic bytes (whole maps read once + output written once + rois) / CUDA-event time.
    14x14 (the SPI module's own setting) and bf16 are reported beside it."""
    import numpy as np
    import torch
    import gpt4roi_b200 as g
    rng = np.random.default_rng(0)
    sizes, C = (128, 64, 32, 16), 1024
    rows = []
    for i in range(n_maps):
        p = np.sort(rng.uniform(0, 1, (rois_per_map, 2, 2)), axis=1)
        b = np.concatenate([p[:, 0, :], p[:, 1, :]], 1) * 224
        b[:, 2:] = np.minimum(np.maximum(b[:, 2:], b[:, :2] + 2.0), 224)
        rows.append(np.concatenate([np.full((rois_per_map, 1), i), b], 1))
    rois = torch.from_numpy(np.concatenate(rows).astype(np.float32)).to(dev)
    K = rois.shape[0]
    scales = [float(np.float32(1.0 / s)) for s in (14 / 8, 14 / 4, 14 / 2, 14)]
    flush = torch.zeros(256 * 1024 * 1024 // 4, device=dev)   # 256 MiB > 126 MB L2, rewritten between iterations

    def run(dtype, ph):
        maps = [torch.randn(n_maps, h, h, C, device=dev, dtype=dtype) for h in sizes]
        out = torch.empty((4, K, ph, ph, C), device=dev, dtype=dtype)
        for _ in range(3):
            g.roi_align_mlvl(maps, rois, ph, scales, 2, out=out)
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(5):
            flush.add_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.roi_align_mlvl(maps, rois, ph, scales, 2, out=out)
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        ms = sorted(ts)[len(ts) // 2]
        alg = sum(m.numel() for m in maps) * maps[0].element_size() + out.numel() * out.element_size() + K * 20
        del maps, out
        torch.cuda.empty_cache()
        return ms, alg
    ms, alg = run(torch.float32, 7)
    ach = alg / 1e9 / (ms / 1e3)
    others = {}
    for name, dt, ph in (('fp32_14x14', torch.float32, 14), ('bf16_7x7', torch.bfloat16, 7), ('bf16_14x14', torch.bfloat16, 14)):
        try:
            m2, a2 = run(dt, ph)
            others[name] = dict(ms=m2, achieved=a2 / 1e9 / (m2 / 1e3), frac=a2 / 1e9 / (m2 / 1e3) / pk['hbm_gbs'])
        except Exception as e:
            others[name] = dict(skipped=str(e)[:120])
    traffic, tsrc = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'r2_roialign_traffic.json')))
        traffic, tsrc = tj['traffic_bytes_per_launch'], tj['source']
    except Exception:
        pass
    del flush
    torch.cuda.empty_cache()
    return dict(bound='hbm', kernel='roi_align_fwd_nhwc_mlvl_dedup', achieved=ach, peak=pk['hbm_gbs'], unit='GB/s',
                frac=ach / pk['hbm_gbs'], peak_kind=how, ms=ms, algorithmic_GB=alg / 1e9,
                config='%d maps x %d RoIs, 7x7, 4 levels x 1024 ch (128,64,32,16), fp32 NHWC, L2 flushed between launches'
                       % (n_maps, rois_per_map),
                traffic=traffic, traffic_source=tsrc, variants=others)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t0 = time.perf_counter()
    best = cpu_reference_sample(repeats=args.steps)
    L = WORKLOAD['text_tokens'] + (WORKLOAD['image_size'] // 14) ** 2 + 2
    line = dict(impl='reference', metric=METRIC, value=best['value'],
                unit='samples/s', n_gpus=args.gpus, steps=len(best['repeat_seconds']), warmup=1,
                ms_per_step=1e3 / best['value'], higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic',
                config=dict(workload='configs[1] per-sample: 336px, 8 RoIs, 128-tok prompt (L=%d), 7B prefill; '
                                     'reference CPU path (PyTorch-CPU + transformers + mmcv-CPU RoIAlign)' % L,
                            note='bounded sample: SPI module in full, ViT / LLaMA stacks extrapolated from one layer'),
                extrapolated=True, wall_clock_s=round(time.perf_counter() - t0, 2), spread=best['spread'],
                cpu_baseline=dict(value=best['value'], unit='samples/s', cores=best['cores'], kind=best['kind'],
                                  sample=best['sample'], cpu=best['cpu']),
                e2e=dict(value=best['value'], unit='samples/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                stage_seconds=best['stage_seconds'], repeat_seconds=best['repeat_seconds'])
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# extras
# ---------------------------------------------------------------------------------------------
def time_graph(graph, steps, warmup, stream, barrier, max_over_ranks):
    import torch
    for _ in range(warmup):
        graph.graph.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        graph.graph.replay()
    e1.record(stream)
    barrier()
    return max_over_ranks(e0.elapsed_time(e1)) / steps


def decode_extra(eng, cfg, dev, pk, n_new=48):
    """ms per generated token at batch 1 and 8 after a 706-token region-token prefill (CUDA-graph decode step)."""
    import torch
    from gpt4roi_b200.engine import GraphedDecode, KVCache
    out = {}
    wbytes = sum(t.numel() * 2 for lay in eng.layers for t in lay.values()) + eng.lm_head.numel() * 2
    floor_ms = wbytes / (pk['hbm_gbs'] * 1e9) * 1e3
    for B in (1, 8):
        ids, images, boxes = synthetic_inputs(cfg, B, WORKLOAD['rois_per_image'], WORKLOAD['text_tokens'], seed=50 + B)
        ids, images = ids.to(dev), images.to(dev)
        cache = KVCache(cfg, B, ids.shape[1] + n_new + 8, dev)
        logits = eng.forward_device(ids, images, eng.plan_boxes(boxes), validate=False, last_only=True, cache=cache)
        nxt = logits[:, -1].float().argmax(-1, keepdim=True)
        stepper = GraphedDecode(eng, cache)
        for _ in range(4):
            nxt = stepper.step(nxt)[:, -1].float().argmax(-1, keepdim=True)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_new - 4):
            nxt = stepper.step(nxt)[:, -1].float().argmax(-1, keepdim=True)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / (n_new - 4)
        # bytes one step must stream: every decoder / lm_head weight once + the K and V rows of all cached positions
        kv_bytes = 2 * B * (ids.shape[1] + 4 + (n_new - 4) / 2) * cfg.hidden * 2 * cfg.n_layers
        floor_kv_ms = (wbytes + kv_bytes) / (pk['hbm_gbs'] * 1e9) * 1e3
        out['batch%d' % B] = dict(ms_per_token=ms, tokens_per_s=B * 1e3 / ms, frac_of_weight_stream_floor=floor_ms / ms,
                                  weight_plus_kv_floor_ms=floor_kv_ms, frac_of_weight_plus_kv_floor=floor_kv_ms / ms)
        del stepper, cache
    out['weight_stream_floor_ms'] = floor_ms
    out['note'] = ('floor = bf16 decoder + lm_head weight bytes / measured HBM bandwidth; greedy sampling (arg-max on the host '
                   'stream) inside the timed loop; %d tokens after a 706-token prefill' % (n_new - 4))
    return out


def train_extra(dev, world, rank, steps=4, warmup=2, batch=4, stage1=True):
    """BASELINE configs[3]: stage-2 training step (ViT frozen), bf16, per-GPU batch 4 (global 32 at 8 GPUs), DDP with
    the NCCL gradient all-reduce overlapped with the backward; the same step with the sharded optimizer (reduce-scatter
    / AdamW on slices / all-gather: what train_stage2.sh's FSDP does); and the ONLY_SPI stage-1 variant."""
    import torch
    import torch.distributed as dist
    from gpt4roi_b200 import lib
    from gpt4roi_b200.engine import EngineConfig, random_state_dicts
    from gpt4roi_b200.train import LayerBucketAllReduce, Stage2Trainer
    cfg = EngineConfig(image_size=WORKLOAD['image_size'])
    out = {}
    ids, images, boxes = synthetic_inputs(cfg, batch, WORKLOAD['rois_per_image'], WORKLOAD['text_tokens'], seed=100 + rank)
    ids, images = ids.to(dev), images.to(dev)
    labels = ids.clone()
    labels[:, :cfg.num_patches + 3] = -100
    labels[ids == cfg.bbox_token] = -100

    def timed(tr, n):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            loss = tr.step(ids, images, boxes, labels)
        tr.stack.sync_optimizer()      # the last step's side-stream AdamW belongs to the timed region
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / n
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, float(loss.item())

    variants = [('stage2', dict(trainable=('embed', 'proj', 'spi', 'llama', 'head')))]
    if world > 1:   # FSDP-equivalent of train_stage2.sh:51-52: reduce-scatter + AdamW on 1/world slices + all-gather
        variants.append(('stage2_sharded_optimizer', dict(trainable=('embed', 'proj', 'spi', 'llama', 'head'), shard_optimizer=True)))
    if stage1:
        variants.append(('stage1_only_spi', dict(trainable=('spi',), spi_decay_all=0.01)))
    for name, kw in variants:
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        sd, vit_sd = random_state_dicts(cfg, dev, seed=0)           # same weights on every rank
        red = LayerBucketAllReduce() if world > 1 else None
        tr = Stage2Trainer(cfg, sd, vit_sd, dev, lr=2e-5, reducer=red, world_size=world, max_grad_norm=1.0,
                           schedule=dict(total_steps=10000, warmup_ratio=0.003, kind='cosine'), **kw)
        del sd, vit_sd
        torch.cuda.empty_cache()
        losses = [tr.step(ids, images, boxes, labels).item() for _ in range(warmup)]
        l0 = lib.LAUNCHES
        ms, loss = timed(tr, steps)
        launches = (lib.LAUNCHES - l0) // steps
        rec = dict(ms_per_step=ms, samples_per_s=world * batch / (ms / 1e3), per_gpu_batch=batch, global_batch=world * batch,
                   g4r_launches_per_step=launches, peak_mem_GB=torch.cuda.max_memory_allocated(dev) / 1e9,
                   losses=[round(v, 4) for v in losses + [loss]],
                   grad_norm=float(tr.clip[0].item()) if tr.clip is not None else None)
        if world > 1 and not kw.get('shard_optimizer'):
            tr.reducer = None                                         # same step without the collectives
            ms_local, _ = timed(tr, max(2, steps // 2))
            rec['ms_per_step_no_allreduce'] = ms_local
            rec['exposed_allreduce_ms'] = max(0.0, ms - ms_local)
            rec['allreduce_calls_per_step'] = red.calls // (warmup + steps)
        out[name] = rec
        del tr, red
        torch.cuda.empty_cache()
    out['config'] = ('configs[3]: 336 px, 8 RoIs/img, 128 text tokens (L=706), 7B, bf16 compute, fp32 masters + AdamW, '
                     'grad-norm clip 1.0, cosine LR, DDP x%d (one flat bf16 bucket per decoder layer over NCCL)' % world)
    return out


DUMP_ROWS = 256   # sampled logit rows: 256 x 32006 fp32 = 33 MB


def dump_logits(logits, out_dir):
    """Write what the last timed step returned, the [B, L, V] logits, as float32 .npy files small enough to keep:
    logits_last.npy = every sample's last position [B, V]; logits_rows.npy = DUMP_ROWS (b, l) positions drawn once
    from a fixed seed, in ascending b * L + l order [DUMP_ROWS, V]."""
    import numpy as np
    B, L, V = logits.shape
    rows = np.sort(np.random.default_rng(0).choice(B * L, size=min(DUMP_ROWS, B * L), replace=False))
    flat = logits.reshape(B * L, V)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'logits_last.npy'), logits[:, -1].float().cpu().numpy())
    np.save(os.path.join(out_dir, 'logits_rows.npy'), flat[rows.tolist()].float().cpu().numpy())


def run_ours(args):
    # keep stdout to the single JSON line: NCCL prints its version banner there unless told otherwise
    if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
        os.environ['NCCL_DEBUG'] = 'WARN'
    import torch
    import torch.distributed as dist
    from gpt4roi_b200 import dense, dist_utils, lib
    from gpt4roi_b200.engine import EngineConfig, GraphedPrefill, PrefillEngine, random_state_dicts

    world, rank, local = dist_utils.env_world()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist_utils.init('nccl', dev)   # NCCL only for the barrier + max-over-ranks time (no data-path collective in the prefill)
    pk, how = peaks()

    cfg = EngineConfig(image_size=WORKLOAD['image_size'], n_layers=args.layers, vit_layers=24, dtype=args.dtype)
    B, K, T = WORKLOAD['batch_per_gpu'], WORKLOAD['rois_per_image'], WORKLOAD['text_tokens']
    sd, vit_sd = random_state_dicts(cfg, dev, seed=0)
    eng = PrefillEngine(cfg, sd, vit_sd, dev)
    del sd, vit_sd
    torch.cuda.empty_cache()
    ids, images, boxes = synthetic_inputs(cfg, B, K, T, seed=rank)
    L = ids.shape[1]
    h_ids, h_img = ids.pin_memory(), images.pin_memory()
    h_boxes = [b.pin_memory() for b in boxes]
    if args.ncu:
        # profiling mode (run under `ncu --profile-from-start off`): one eager forward inside the
        # cudaProfilerStart/Stop window, nothing else.
        plan = eng.plan_boxes(boxes)
        d_ids, d_img = ids.to(dev), images.to(dev)
        eng.forward_device(d_ids, d_img, plan, validate=True, last_only=False)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        eng.forward_device(d_ids, d_img, plan, validate=False, last_only=False)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return
    lib.LAUNCHES = 0
    graph = GraphedPrefill(eng, ids, images, boxes, last_only=False)
    launches_per_step = lib.LAUNCHES // 3  # 2 eager warm-ups + 1 capture
    stream = torch.cuda.current_stream(dev)

    def barrier():
        dist_utils.barrier(dev)

    def max_over_ranks(ms):
        return dist_utils.max_over_ranks(ms, dev)

    # ---- value: inputs resident in HBM, graph replays only --------------------------------
    for _ in range(max(args.warmup, 3)):
        graph.graph.replay()
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        graph.graph.replay()
    e1.record(stream)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_logits(graph.out, args.dump_outputs)

    # ---- e2e: public API with pinned HOST buffers.  Every step: H2D of ids/images/boxes, graph replay, D2H of
    #      EVERYTHING the step computes (the full [B,L,V] logits, 361 MB) into pinned host memory.  The D2H runs on a
    #      copy stream from a snapshot of the logits, double-buffered, so it overlaps the next step's compute; the
    #      timed region ends when the last copy has landed. ---
    copy_stream = torch.cuda.Stream(device=dev)
    V = cfg.vocab
    h_out = [torch.empty((B, L, V), dtype=cfg.torch_dtype).pin_memory() for _ in range(2)]
    d_snap = [torch.empty((B, L, V), dtype=cfg.torch_dtype, device=dev) for _ in range(2)]
    ev_copied = [torch.cuda.Event() for _ in range(2)]

    def e2e_step(i):
        out = graph.run(h_ids, h_img, h_boxes)
        j = i & 1
        stream.wait_event(ev_copied[j])          # the snapshot buffer is free again
        d_snap[j].copy_(out)                     # device-side snapshot (the graph's output buffer is reused next step)
        ev = torch.cuda.Event()
        ev.record(stream)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev)
            h_out[j].copy_(d_snap[j], non_blocking=True)
            ev_copied[j].record(copy_stream)
    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize(dev)
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        e2e_step(i)
    stream.wait_stream(copy_stream)
    e1.record(stream)
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    h2d = h_ids.numel() * 8 + h_img.numel() * 2 + sum(b.numel() * 4 for b in h_boxes)
    d2h = h_out[0].numel() * 2
    del h_out, d_snap
    torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv): one instrumented
    #      eager step with CUDA events around every launch on the launching stream ------------
    dense.PROFILE = []
    plan = eng.plan_boxes(boxes)
    eng.forward_device(graph.ids, graph.images, plan, validate=False, last_only=False)
    torch.cuda.synchronize(dev)
    prof, dense.PROFILE = dense.PROFILE, None
    gemm_ms = sum(s.elapsed_time(e) for _, _, s, e in prof)
    gemm_flops = sum(f for _, f, _, _ in prof)
    achieved = gemm_flops / 1e12 / (gemm_ms / 1e3)
    traffic, traffic_src = None, None
    for name in ('r2_gemm_traffic.json', 'r1_gemm_traffic.json'):
        try:  # dram__bytes_read+write per launch from the committed ncu --set full capture of this kernel
            tj = json.load(open(os.path.join(ROOT, 'profiles', name)))
            traffic, traffic_src = tj['traffic_bytes_per_launch_avg'], tj['source']
            break
        except Exception:
            pass
    roof = dict(bound='tensor', kernel='gemm_bf16_tcgen05', achieved=achieved, peak=pk['bf16_tflops_sustained'],
                unit='TFLOP/s', frac=achieved / pk['bf16_tflops_sustained'], traffic=traffic, traffic_source=traffic_src,
                peak_kind=how + ' (sustained cuBLAS bf16; kernel timed inside a long step)',
                launches=len(prof), flops_per_launch_avg=gemm_flops / max(len(prof), 1),
                avg_launch_ms=gemm_ms / max(len(prof), 1), share_of_step=gemm_ms / ms_step,
                note='events around each launch in one eager instrumented step after the timed region')

    # ---- second half of the BASELINE metric (43 GB of operands beside the 14.6 GB engine; after the headline so
    #      that its 0.6 s of sustained HBM traffic does not pre-heat the headline's power-capped clocks) ----
    roi = None
    if rank == 0 and not args.no_roialign:
        try:
            torch.cuda.synchronize(dev)
            time.sleep(3.0)    # let the power-capped SM clock recover: the kernel is L1 / issue bound, i.e. SM-clock bound
            roi = roialign_microbench(dev, pk, how)
        except Exception as e:
            roi = dict(skipped=str(e)[:200])
        torch.cuda.empty_cache()

    # ---- configs[2]'s shape: 16 RoIs per image, 8 images per GPU (batch 64 across 8 GPUs) ----------------------
    cfg2 = None
    if not args.no_extras:
        del graph
        torch.cuda.empty_cache()
        ids2, images2, boxes2 = synthetic_inputs(cfg, B, 16, T, seed=1000 + rank)
        g2 = GraphedPrefill(eng, ids2, images2, boxes2, last_only=False)
        ms2 = time_graph(g2, max(5, args.steps // 2), 3, stream, barrier, max_over_ranks)
        cfg2 = dict(samples_per_s=world * B / (ms2 / 1e3), ms_per_step=ms2, global_batch=world * B, rois_per_image=16,
                    note='configs[2] shape per GPU (8 images x 16 RoIs, L=706); at --gpus 8 this is the batch-64 configuration')
        del g2
        torch.cuda.empty_cache()

    dec = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            dec = decode_extra(eng, cfg, dev, pk)
        except Exception as e:
            dec = dict(skipped=str(e)[:200])
    del eng
    torch.cuda.empty_cache()

    train = None
    if not args.no_extras and not args.no_train:
        try:
            train = train_extra(dev, world, rank)
        except Exception as e:
            train = dict(skipped=repr(e)[:300])
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = cpu_reference_sample() if (world == 1 and not args.no_cpu_baseline) else None
    line = dict(metric=METRIC, value=value, unit='samples/s',
                n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_step,
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype=args.dtype, data='synthetic',
                config=dict(workload='configs[1]: batch %d/GPU, 336px, %d RoIs/img, %d-tok prompt (L=%d), '
                                     'CLIP-ViT-L/14 + SPI + LLaMA-7B (%d layers) + lm_head, full logits' %
                                     (B, K, T, L, cfg.n_layers),
                            global_batch=world * B, seq_len=L, parallelism='replicas x%d (batch split, no collective)' % world,
                            l2='weights (14.6 GB) >> 126 MB L2: inputs larger than L2, no explicit flush',
                            cuda_graph=True, flops_per_sample=FLOPS_PER_SAMPLE),
                clocks=clocks, gpu_launches=launches_per_step * args.steps,
                e2e=dict(value=world * B / (e2e_ms / 1e3), unit='samples/s', h2d_bytes_per_step=h2d,
                         d2h_bytes_per_step=d2h, ms_per_step=e2e_ms,
                         note='D2H = the full [B,L,V] bf16 logits of the step (everything it computes), double-buffered on a copy stream'),
                roofline=roof,
                model_tflops=value * FLOPS_PER_SAMPLE / 1e12 / world,
                roialign_roofline=roi, config2_16roi=cfg2, decode=dec, train_step=train,
                cpu_baseline=cpu)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--layers', type=int, default=32, help=argparse.SUPPRESS)  # debugging only; 32 = LLaMA-7B
    ap.add_argument('--dtype', default='bf16', choices=['bf16', 'fp16'],
                    help="16-bit storage type of the prefill / decode kernels (fp16 = the demo's mode; training extras stay bf16)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-roialign', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='headline only (no config2 / decode / train_step extras)')
    ap.add_argument('--no-train', action='store_true')
    ap.add_argument('--ncu', action='store_true', help='one eager forward inside a cudaProfiler window')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write a fixed sample of the last step\'s logits to DIR/*.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
