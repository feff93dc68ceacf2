"""Generate the committed golden fixtures under tests/golden/ FROM THE REFERENCE ITSELF.

Run in the build container (needs /root/reference; the GPU box never runs this):
    python tests/golden/make_golden.py

Fixtures:
  mmcv_roi_align_kat.json   the reference's own known-answer vectors, read from
                            mmcv-1.4.7/tests/test_ops/test_roi_align.py:14-32
                            (3 cases: input, rois -> forward output and input-gradient;
                            pool 2x2, scale 1.0, sampling 2, avg, aligned)
  roi_align_ref_cases.npz   seeded random + adversarial cases run through the reference's
                            CPU kernel compiled unmodified (oracle/_ref, see oracle/build_ref.py):
                            forward (avg/max, argmax) and backward, fp32, NCHW.
"""
import importlib.util
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import build_ref  # noqa: E402

REF = os.environ.get('GPT4ROI_REFERENCE', '/root/reference')


def kat():
    path = os.path.join(REF, 'mmcv-1.4.7', 'tests', 'test_ops', 'test_roi_align.py')
    spec = importlib.util.spec_from_file_location('ref_test_roi_align', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    cases = []
    for (inp, rois), (out, grad) in zip(mod.inputs, mod.outputs):
        cases.append(dict(input=inp, rois=rois, output=out, grad_input=grad))
    doc = dict(source='mmcv-1.4.7/tests/test_ops/test_roi_align.py:14-32',
               pool_h=mod.pool_h, pool_w=mod.pool_w, spatial_scale=mod.spatial_scale,
               sampling_ratio=mod.sampling_ratio, pool_mode='avg', aligned=True, atol=1e-3,
               cases=cases)
    with open(os.path.join(HERE, 'mmcv_roi_align_kat.json'), 'w') as f:
        json.dump(doc, f, indent=1)
    print('wrote mmcv_roi_align_kat.json (%d cases)' % len(cases))


def adversarial_boxes(S):
    """xyxy boxes in input-pixel units for an SxS image: degenerate, full-image, border cases."""
    e = 1.0
    return np.array([
        [0, 0, S, S],                    # full image
        [10.5, 20.25, 10.5, 20.25],      # zero area
        [5, 5, 5, 60],                   # zero width
        [-e, -e, S + e, S + e],          # exceeds every border by 1px
        [S - 0.4, S - 0.4, S, S],        # sub-pixel at the far corner
        [0, 0, 0.3, 0.3],                # sub-pixel at the origin
        [S * 0.5, -e, S + e, S * 0.5],   # top-right overhang
        [3.999, 7.001, 100.5, 50.499],   # generic non-aligned
        [S, S, S, S],                    # point on the far border
        [0, 0, 2, 2],                    # minimum 2px training box
    ], dtype=np.float32)


def ref_cases():
    ext = build_ref.load()
    assert ext is not None, 'reference tree not available'
    rng = np.random.default_rng(20260923)
    out = {}
    meta = []
    S = 224
    #            name         N  C   H    W   PH sr mode   stride
    configs = [('l0_224',     2, 8, 128, 128, 14, 2, 'avg', 1.75),
               ('l1_224',     2, 8, 64, 64, 14, 2, 'avg', 3.5),
               ('l2_224',     2, 8, 32, 32, 14, 2, 'avg', 7.0),
               ('l3_224',     2, 8, 16, 16, 14, 2, 'avg', 14.0),
               ('l3_336',     2, 8, 24, 24, 14, 2, 'avg', 14.0),
               ('mb7',        3, 8, 32, 32, 7, 2, 'avg', 7.0),
               ('adaptive',   2, 4, 20, 28, 3, 0, 'avg', 4.0),
               ('max2',       2, 4, 16, 16, 5, 2, 'max', 14.0),
               ('max_adapt',  2, 4, 12, 9, 4, 0, 'max', 8.0),
               ('rect',       1, 4, 10, 17, (3, 5), 3, 'avg', 2.0),
               ('unaligned',  2, 4, 16, 16, 7, 2, 'avg_unaligned', 14.0)]
    for name, N, C, H, W, PH, sr, mode, stride in configs:
        x = rng.standard_normal((N, C, H, W)).astype(np.float32)
        Sx, Sy = W * stride, H * stride
        K = 12
        p = np.sort(rng.uniform(0, 1, (K, 2, 2)), axis=1)
        boxes = np.concatenate([p[:, 0, :], p[:, 1, :]], 1) * np.array([Sx, Sy, Sx, Sy])
        boxes = boxes.astype(np.float32)
        if H == W:
            boxes = np.concatenate([boxes, adversarial_boxes(Sx)], 0)
        K = len(boxes)
        bidx = rng.integers(0, N, (K, 1)).astype(np.float32)
        rois = np.concatenate([bidx, boxes], 1).astype(np.float32)
        scale = float(np.float32(1.0 / stride))
        ph, pw = (PH, PH) if isinstance(PH, int) else PH
        aligned = mode != 'avg_unaligned'
        pm = 0 if mode == 'max' else 1
        xt, rt = torch.from_numpy(x), torch.from_numpy(rois)
        o = xt.new_zeros(K, C, ph, pw)
        ay = xt.new_zeros(K, C, ph, pw) if pm == 0 else xt.new_zeros(0)
        ax = xt.new_zeros(K, C, ph, pw) if pm == 0 else xt.new_zeros(0)
        ext.roi_align_forward(xt, rt, o, ay, ax, aligned_height=ph, aligned_width=pw,
                              spatial_scale=scale, sampling_ratio=sr, pool_mode=pm, aligned=aligned)
        g = rng.standard_normal((K, C, ph, pw)).astype(np.float32)
        gi = xt.new_zeros(N, C, H, W)
        ext.roi_align_backward(torch.from_numpy(g), rt, ay, ax, gi, aligned_height=ph,
                               aligned_width=pw, spatial_scale=scale, sampling_ratio=sr,
                               pool_mode=pm, aligned=aligned)
        out[name + '.input'] = x
        out[name + '.rois'] = rois
        out[name + '.output'] = o.numpy()
        out[name + '.grad_output'] = g
        out[name + '.grad_input'] = gi.numpy()
        if pm == 0:
            out[name + '.argmax_y'] = ay.numpy()
            out[name + '.argmax_x'] = ax.numpy()
        meta.append(dict(name=name, N=N, C=C, H=H, W=W, PH=ph, PW=pw, sampling_ratio=sr,
                         pool_mode='max' if pm == 0 else 'avg', aligned=aligned,
                         spatial_scale=scale, K=K))
    out['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'roi_align_ref_cases.npz'), **out)
    print('wrote roi_align_ref_cases.npz (%d cases)' % len(meta))


if __name__ == '__main__' and len(sys.argv) == 1:
    kat()
    ref_cases()


# ---------------------------------------------------------------------------------------
# SPI module golden: the reference's MLVLROIQueryModule run UNMODIFIED (224 px) and with the three
# literals lifted (336 px, SURVEY.md 8(c)), fp32 on CPU, with seeded weights that the tests can
# regenerate (gpt4roi_b200.engine.random_state_dicts on CPU) and seeded inputs.
# ---------------------------------------------------------------------------------------
def spi_inputs(image_size, B, ks, seed):
    g = torch.Generator().manual_seed(seed)
    G = image_size // 14
    toks = [torch.randn(B, G * G, 1024, generator=g) for _ in range(4)]
    boxes = []
    for k in ks:
        p = torch.rand(k, 2, 2, generator=g).sort(dim=1).values
        b = torch.cat([p[:, 0, :], p[:, 1, :]], 1)
        b[:, 2:] = torch.maximum(b[:, 2:], b[:, :2] + 2.0 / image_size).clamp(max=1.0)
        boxes.append(b)
    return toks, boxes


def spi_module_golden():
    sys.path.insert(0, HERE)
    import ref_shims
    from gpt4roi_b200.engine import EngineConfig, random_state_dicts
    out = {}
    for size, B, ks in ((224, 1, [3]), (336, 2, [2, 1])):
        layers = ref_shims.load_layers(size)
        cfg = EngineConfig(image_size=size, n_layers=0, vit_layers=0)
        sd, _ = random_state_dicts(cfg, 'cpu', seed=1234, dtype=torch.float32)
        mod = layers.MLVLROIQueryModule(embed_dims=1024, out_dims=4096, num_levels=4)
        spi = {k[len('model.spi_module.'):]: v for k, v in sd.items() if k.startswith('model.spi_module.')}
        missing = mod.load_state_dict(spi, strict=True)
        mod.eval()
        toks, boxes = spi_inputs(size, B, ks, seed=size)
        with torch.no_grad():
            res = mod([t.clone() for t in toks], boxes)
        out['spi%d.out' % size] = torch.cat(res, 0).numpy()
        out['spi%d.in_checksum' % size] = np.array([float(t.double().sum()) for t in toks] +
                                                   [float(torch.cat(boxes).double().sum())])
        out['spi%d.w_checksum' % size] = np.array([float(sd['model.spi_module.roi_align.flatten_linear.weight'].double().sum()),
                                                   float(sd['model.spi_module.mlvl_fuse.fuse_convs.4.conv.weight'].double().abs().sum())])
        print('spi golden %d: out %s' % (size, out['spi%d.out' % size].shape))
    np.savez_compressed(os.path.join(HERE, 'spi_module_ref.npz'), **out)
    print('wrote spi_module_ref.npz')


if __name__ == '__main__' and '--spi' in sys.argv:
    spi_module_golden()


# ---------------------------------------------------------------------------------------
# Full-model golden: the reference's OWN SPILlavaMPTForCausalLM.forward (gpt4roi/models/spi_llava.py +
# llava/model/llava.py, unmodified, 224 px, fp32, CPU) with a full-width CLIP-L/14 (24 layers) and a
# 2-layer LLaMA of hidden 4096.  Pins oracle/model_oracle.py (composition: level pick, projector,
# splice, region scatter, lm_head) to the real code path.  Stored: logits at 24 probe positions.
# ---------------------------------------------------------------------------------------
def model_inputs(cfg, ks, T, seed):
    g = torch.Generator().manual_seed(seed)
    B, P = len(ks), cfg.num_patches
    L = T + P + 2
    ids = torch.randint(3, 32000, (B, L), generator=g)
    boxes = []
    for b in range(B):
        ids[b, 0] = 1
        ids[b, 1] = cfg.im_start_token
        ids[b, 2:2 + P] = cfg.im_patch_token
        ids[b, 2 + P] = cfg.im_end_token
        pos = torch.randperm(L - (3 + P), generator=g)[:ks[b]] + 3 + P
        ids[b, pos] = cfg.bbox_token
        p = torch.rand(ks[b], 2, 2, generator=g).sort(dim=1).values
        bx = torch.cat([p[:, 0, :], p[:, 1, :]], 1)
        bx[:, 2:] = torch.maximum(bx[:, 2:], bx[:, :2] + 2.0 / cfg.image_size).clamp(max=1.0)
        boxes.append(bx)
    images = torch.randn(B, 3, cfg.image_size, cfg.image_size, generator=g)
    return ids, images, boxes


def full_model_golden():
    sys.path.insert(0, HERE)
    import importlib
    import ref_shims
    from gpt4roi_b200.engine import EngineConfig, random_state_dicts
    ref_shims.install()
    spi_llava = importlib.import_module('gpt4roi.models.spi_llava')
    llava = importlib.import_module('llava.model.llava')
    from transformers import CLIPVisionConfig, CLIPVisionModel
    cfg = EngineConfig(image_size=224, vit_layers=24, n_layers=2)
    sd, vit_sd = random_state_dicts(cfg, 'cpu', seed=4321, dtype=torch.float32)
    lc = llava.LlavaConfig(hidden_size=4096, intermediate_size=11008, num_hidden_layers=2, num_attention_heads=32,
                           num_key_value_heads=32, vocab_size=32006, rms_norm_eps=1e-6, max_position_embeddings=2048)
    lc._attn_implementation = 'eager'
    lc.mm_vision_select_layer = -2
    lc.use_mm_proj = True
    lc.mm_hidden_size = 1024
    model = spi_llava.SPILlavaMPTForCausalLM(lc)
    vc = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                          image_size=224, patch_size=14)
    vc._attn_implementation = 'eager'
    vt = CLIPVisionModel(vc)
    missing, unexpected = vt.load_state_dict(vit_sd, strict=False)
    assert not unexpected
    model.model.vision_tower = [vt.eval()]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all('rotary' in k or 'inv_freq' in k for k in missing), missing
    model.eval()
    vconf = vt.config
    vconf.im_patch_token, vconf.bbox_token = cfg.im_patch_token, cfg.bbox_token
    vconf.im_start_token, vconf.im_end_token = cfg.im_start_token, cfg.im_end_token
    vconf.use_im_start_end = True

    class Tok:
        def convert_tokens_to_ids(self, toks):
            return [cfg.bbox_token for _ in toks]
    for m in model.modules():
        m.tokenizer = Tok()
    ids, images, boxes = model_inputs(cfg, [2, 1], 20, seed=99)
    with torch.no_grad():
        out = model(input_ids=ids, images=images, img_metas=[None] * len(boxes), bboxes=boxes,
                    attention_mask=torch.ones_like(ids))
    logits = out.logits.float()
    L = ids.shape[1]
    probe = torch.unique(torch.cat([torch.arange(0, L, L // 12), torch.tensor([1, 2, cfg.num_patches + 2, L - 1]),
                                    torch.where(ids[0] == cfg.bbox_token)[0]]))
    np.savez_compressed(os.path.join(HERE, 'full_model_ref_224.npz'),
                        probe=probe.numpy(), logits=logits[:, probe].numpy(),
                        argmax=logits.argmax(-1).numpy(), lmean=np.array([float(logits.double().mean()), float(logits.double().std())]),
                        ids_checksum=np.array([int(ids.sum())]),
                        w_checksum=np.array([float(sd['lm_head.weight'].double().sum())]))
    print('wrote full_model_ref_224.npz', logits.shape, probe.tolist())


if __name__ == '__main__' and '--model' in sys.argv:
    full_model_golden()


# ---------------------------------------------------------------------------------------
# Training-step golden: the reference's OWN forward WITH labels + loss.backward() (the body of the HF Trainer step,
# gpt4roi/train/train.py:698-712) on the same unmodified modules as the full-model golden, fp32 on CPU, CLIP tower
# frozen as in stage 2.  Weights are rounded to bf16-representable values so that the sm_100a trainer starts from
# identical parameters.  Stored: the loss and the gradients of a probe set of parameters (small tensors in full,
# the first rows of the large ones).  Pins gpt4roi_b200.train.Stage2Trainer to the reference's autograd.
# ---------------------------------------------------------------------------------------
TRAIN_PROBES_FULL = [
    'model.norm.weight', 'model.layers.1.input_layernorm.weight', 'model.layers.0.post_attention_layernorm.weight',
    'model.mm_projector.bias', 'model.spi_module.roi_align.updims.bias', 'model.spi_module.roi_align.flatten_linear.bias',
    'model.spi_module.mlvl_fuse.fuse_convs.0.gn.weight', 'model.spi_module.mlvl_fuse.fuse_convs.4.gn.bias',
    'model.spi_module.roi_align.pos_embedd.5.weight', 'model.spi_module.roi_align.pos_embedd.0.weight',
    'model.spi_module.mlvl_fuse.input_conv.3.bias', 'model.spi_module.roi_align.pconvs.1.bias',
]
TRAIN_PROBES_ROWS = {   # name -> number of leading rows kept
    'lm_head.weight': 4, 'model.layers.0.self_attn.q_proj.weight': 4, 'model.layers.0.self_attn.v_proj.weight': 4,
    'model.layers.1.self_attn.o_proj.weight': 4, 'model.layers.1.mlp.gate_proj.weight': 4,
    'model.layers.1.mlp.down_proj.weight': 4, 'model.mm_projector.weight': 8,
    'model.spi_module.roi_align.updims.weight': 8, 'model.spi_module.roi_align.pconvs.2.weight': 2,
    'model.spi_module.mlvl_fuse.fuse_convs.2.conv.weight': 2, 'model.spi_module.mlvl_fuse.fuse_convs.0.conv.weight': 2,
    'model.spi_module.mlvl_fuse.input_conv.0.weight': 8,
}


def train_inputs():
    from gpt4roi_b200.engine import EngineConfig
    cfg = EngineConfig(image_size=224, vit_layers=24, n_layers=2)
    ids, images, boxes = model_inputs(cfg, [2, 1], 20, seed=77)
    labels = ids.clone()
    labels[:, : cfg.num_patches + 6] = -100                      # prompt / image part is not supervised
    labels[ids == cfg.bbox_token] = -100
    return cfg, ids, images, boxes, labels


def train_step_golden():
    sys.path.insert(0, HERE)
    import importlib
    import ref_shims
    from gpt4roi_b200.engine import random_state_dicts
    ref_shims.install()
    spi_llava = importlib.import_module('gpt4roi.models.spi_llava')
    llava = importlib.import_module('llava.model.llava')
    from transformers import CLIPVisionConfig, CLIPVisionModel
    cfg, ids, images, boxes, labels = train_inputs()
    sd, vit_sd = random_state_dicts(cfg, 'cpu', seed=1234, dtype=torch.float32)
    sd = {k: v.to(torch.bfloat16).float() for k, v in sd.items()}
    vit_sd = {k: v.to(torch.bfloat16).float() for k, v in vit_sd.items()}
    lc = llava.LlavaConfig(hidden_size=4096, intermediate_size=11008, num_hidden_layers=2, num_attention_heads=32,
                           num_key_value_heads=32, vocab_size=32006, rms_norm_eps=1e-6, max_position_embeddings=2048)
    lc._attn_implementation = 'eager'
    lc.mm_vision_select_layer = -2
    lc.use_mm_proj = True
    lc.mm_hidden_size = 1024
    model = spi_llava.SPILlavaMPTForCausalLM(lc)
    vc = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                          image_size=224, patch_size=14)
    vc._attn_implementation = 'eager'
    vt = CLIPVisionModel(vc)
    missing, unexpected = vt.load_state_dict(vit_sd, strict=False)
    assert not unexpected
    vt.requires_grad_(False)                                     # frozen tower (train.py:604-612)
    model.model.vision_tower = [vt.eval()]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    model.train()
    vconf = vt.config
    vconf.im_patch_token, vconf.bbox_token = cfg.im_patch_token, cfg.bbox_token
    vconf.im_start_token, vconf.im_end_token = cfg.im_start_token, cfg.im_end_token
    vconf.use_im_start_end = True

    class Tok:
        def convert_tokens_to_ids(self, toks):
            return [cfg.bbox_token for _ in toks]
    for m in model.modules():
        m.tokenizer = Tok()
    out = model(input_ids=ids, images=images, img_metas=[None] * len(boxes), bboxes=boxes,
                attention_mask=torch.ones_like(ids), labels=labels)
    out.loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
    trained = sorted(grads)
    store = {'loss': np.array([float(out.loss)]), 'n_trained_tensors': np.array([len(trained)]),
             'ids_checksum': np.array([int(ids.sum())]), 'w_checksum': np.array([float(sd['lm_head.weight'].double().sum())])}
    for k in TRAIN_PROBES_FULL:
        store['full/' + k] = grads[k].float().numpy()
    for k, n in TRAIN_PROBES_ROWS.items():
        store['rows/' + k] = grads[k][:n].float().numpy()
    used = torch.unique(ids[(ids < 32000)])[:6]
    store['embed_ids'] = used.numpy()
    store['embed_rows'] = grads['model.embed_tokens.weight'][used].float().numpy()
    store['norms'] = np.array([float(grads[k].double().norm()) for k in trained])
    store['norm_names'] = np.array(trained)
    np.savez_compressed(os.path.join(HERE, 'train_step_ref_224.npz'), **store)
    print('wrote train_step_ref_224.npz: loss %.6f, %d trained tensors' % (float(out.loss), len(trained)))


if __name__ == '__main__' and '--train' in sys.argv:
    train_step_golden()


# ---------------------------------------------------------------------------------------------
# Input pipeline (SURVEY.md 8(f2)): the reference's OWN transform classes (mmdet/datasets/pipelines/transforms.py,
# loading.py; mmcv.imresize / imnormalize underneath), in the order coco_det.py:60-71 lists them, on synthetic uint8
# BGR images with controlled augmentation decisions.  Stored: source images, source boxes, the decisions, the
# pipeline's image tensor and boxes -> tests/golden/input_pipeline_ref.npz.
# ---------------------------------------------------------------------------------------------
INPUT_CASES = [  # (name, src_h, src_w, S, n_boxes, shift (x, y) or None, flip)
    ('down_plain', 120, 90, 56, 3, None, False),
    ('down_shift_flip', 97, 131, 56, 4, (7, -5), True),
    ('up_shift', 37, 53, 56, 2, (-32, 11), False),
    ('square_flip', 64, 64, 112, 3, None, True),
    ('shift_kills_all_boxes', 80, 100, 56, 1, (32, 32), False),   # RandomShift must then leave image AND boxes alone
    ('wide', 33, 200, 112, 5, (3, 32), True),
]


def input_pipeline_golden():
    import importlib
    import random
    import ref_shims
    ref_shims.install()
    T = importlib.import_module('mmdet.datasets.pipelines.transforms')
    Ld = importlib.import_module('mmdet.datasets.pipelines.loading')
    rng = np.random.default_rng(7)
    mean = [0.48145466 * 255, 0.4578275 * 255, 0.40821073 * 255]
    std = [0.26862954 * 255, 0.26130258 * 255, 0.27577711 * 255]
    store = {'names': np.array([c[0] for c in INPUT_CASES])}
    for name, h, w, S, nb, shift, flip in INPUT_CASES:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        p = np.sort(rng.uniform(0, 1, (nb, 2, 2)), axis=1)
        boxes = (np.concatenate([p[:, 0, :], p[:, 1, :]], 1) * np.array([w, h, w, h])).astype(np.float32)
        if name == 'shift_kills_all_boxes':
            boxes = np.array([[w * 0.9, h * 0.9, w * 0.99, h * 0.99]], np.float32)
        res = dict(img=img.copy(), img_shape=img.shape, ori_shape=img.shape, img_fields=['img'], bbox_fields=['gt_bboxes'],
                   gt_bboxes=boxes.copy(), gt_labels=np.arange(nb))
        res = T.Resize(img_scale=(S, S), keep_ratio=False)(res)
        if shift is not None:      # RandomShift with its draws forced to the chosen shift (transforms.py uses
            draws = iter([shift[0], shift[1]])   # `from numpy import random`: random.random(), random.randint(-32, 32) x then y)
            class _Forced:
                random = staticmethod(lambda: 0.0)
                randint = staticmethod(lambda a, b: next(draws))
            orig = T.random
            T.random = _Forced
            try:
                res = T.RandomShift(shift_ratio=0.5, max_shift_px=32)(res)
            finally:
                T.random = orig
        out = Ld.FilterAnnotations(min_gt_bbox_wh=(2.0, 2.0))(res)
        kept_any = out is not None
        if kept_any:
            res = out
        res = T.RandomFlip(flip_ratio=1.0 if flip else 0.0)(res)
        res = T.Normalize(mean=mean, std=std, to_rgb=True)(res)
        res = T.Pad(size_divisor=S)(res)
        chw = np.ascontiguousarray(res['img'].transpose(2, 0, 1))       # DefaultFormatBundle: HWC -> CHW
        store[name + '.src'] = img
        store[name + '.src_boxes'] = boxes
        store[name + '.params'] = np.array([S, 0 if shift is None else shift[0], 0 if shift is None else shift[1], int(flip),
                                            int(kept_any)], np.int32)
        store[name + '.image'] = chw.astype(np.float32)
        store[name + '.boxes'] = (res['gt_bboxes'] / chw.shape[1]).astype(np.float32) if kept_any else np.zeros((0, 4), np.float32)
    np.savez_compressed(os.path.join(HERE, 'input_pipeline_ref.npz'), **store)
    print('wrote input_pipeline_ref.npz (%d cases)' % len(INPUT_CASES))


if __name__ == '__main__' and '--input' in sys.argv:
    input_pipeline_golden()


# ---------------------------------------------------------------------------------------------
# Oracle pin on adversarial boxes: seeded maps and random + adversarial RoIs (tests/helpers.make_rois) through the
# reference's CPU kernel compiled unmodified (oracle/_ref), avg with fixed and adaptive sampling and max pooling.
# Stored: inputs, outputs and argmax -> tests/golden/roi_align_adversarial_ref.npz.
# ---------------------------------------------------------------------------------------------
ADVERSARIAL_CASES = [(48, 14, 2, 'avg', 7.0), (24, 7, 0, 'avg', 14.0), (16, 3, 2, 'max', 14.0)]   # H, PH, sr, mode, stride


def adversarial_golden():
    from tests.helpers import make_rois
    ext = build_ref.load()
    assert ext is not None, 'reference tree not available'
    rng = np.random.default_rng(7)
    store, meta = {}, []
    for i, (H, PH, sr, mode, stride) in enumerate(ADVERSARIAL_CASES):
        name = 'c%d' % i
        x = rng.standard_normal((2, 5, H, H)).astype(np.float32)
        rois = make_rois(rng, 2, 6, H * stride, adversarial=True)
        scale = float(np.float32(1 / stride))
        xt, rt = torch.from_numpy(x), torch.from_numpy(rois)
        pm = 0 if mode == 'max' else 1
        o = xt.new_zeros(len(rois), 5, PH, PH)
        ay = xt.new_zeros(o.shape) if pm == 0 else xt.new_zeros(0)
        ax = xt.new_zeros(o.shape) if pm == 0 else xt.new_zeros(0)
        ext.roi_align_forward(xt, rt, o, ay, ax, aligned_height=PH, aligned_width=PH,
                              spatial_scale=scale, sampling_ratio=sr, pool_mode=pm, aligned=True)
        store[name + '.input'], store[name + '.rois'], store[name + '.output'] = x, rois, o.numpy()
        if pm == 0:
            store[name + '.argmax_y'], store[name + '.argmax_x'] = ay.numpy(), ax.numpy()
        meta.append(dict(name=name, PH=PH, sampling_ratio=sr, pool_mode=mode, spatial_scale=scale))
    store['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'roi_align_adversarial_ref.npz'), **store)
    print('wrote roi_align_adversarial_ref.npz (%d cases)' % len(meta))


if __name__ == '__main__' and '--adversarial' in sys.argv:
    adversarial_golden()


# ---------------------------------------------------------------------------------------------
# How the reference's own wrapper (mmcv-1.4.7/mmcv/ops/roi_align.py, unmodified) calls `mmcv._ext`: every symbol that
# `import mmcv.ops` asserts on (mmcv/utils/ext_loader.py), and the roi_align_forward / roi_align_backward calls of a
# RoIAlign forward + backward in 'avg' and 'max' mode (tensor arguments by shape and dtype, scalars by value).
# Recorded over the reference CPU kernel (oracle/_ref) -> tests/golden/mmcv_wrapper_calls.json.
# ---------------------------------------------------------------------------------------------
def wrapper_calls_golden():
    sys.path.insert(0, HERE)
    import importlib
    import ref_shims
    ref_shims.install()
    ext_loader = importlib.import_module('mmcv.utils.ext_loader')
    names = set()
    load_ext = ext_loader.load_ext

    def recording_load_ext(name, funcs):
        if name == '_ext':
            names.update(funcs)
        return load_ext(name, funcs)
    ext_loader.load_ext = recording_load_ext
    importlib.import_module('mmcv.ops')
    R = sys.modules['mmcv.ops.roi_align']

    def describe(v):
        if isinstance(v, torch.Tensor):
            return dict(shape=list(v.shape), dtype=str(v.dtype).replace('torch.', ''))
        return v
    calls = []
    for fn in ('roi_align_forward', 'roi_align_backward'):
        def recorder(*args, _fn=fn, _impl=getattr(R.ext_module, fn), **kwargs):
            calls.append(dict(fn=_fn, args=[describe(a) for a in args], kwargs={k: describe(v) for k, v in kwargs.items()}))
            return _impl(*args, **kwargs)
        setattr(R.ext_module, fn, recorder)
    for mode in ('avg', 'max'):
        x = torch.randn(1, 4, 8, 8, requires_grad=True)
        R.RoIAlign((7, 7), 0.5, 2, mode)(x, torch.tensor([[0., 0., 0., 4., 4.]])).sum().backward()
    doc = dict(source='mmcv-1.4.7/mmcv/ops/roi_align.py over mmcv/utils/ext_loader.py', ext_names=sorted(names), calls=calls)
    with open(os.path.join(HERE, 'mmcv_wrapper_calls.json'), 'w') as f:
        json.dump(doc, f, indent=1)
    print('wrote mmcv_wrapper_calls.json (%d symbols, %d calls)' % (len(names), len(calls)))


if __name__ == '__main__' and '--wrapper' in sys.argv:
    wrapper_calls_golden()
