"""GPU end-to-end parity of the sm_100a engine against the oracle (oracle/model_oracle.py: the
reference's composition over transformers' CLIP/LLaMA + the SPI torch restatement pinned to the
reference by tests/golden/spi_module_ref.npz).

Tolerances (bf16 storage, fp32 accumulation vs an fp32 oracle on identical bf16-representable
weights): relative L2 error per stage stated inline; the bf16-autocast reference itself is run
beside it and the engine must be at least as close to the fp32 anchor as 1.5x that run."""
import numpy as np
import pytest
import torch

from gpt4roi_b200.engine import EngineConfig, PrefillEngine, random_state_dicts
from oracle import model_oracle, spi_oracle
from tests.test_spi_oracle_cpu import golden_case

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def make_inputs(cfg, B, ks, T, seed=0):
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
        pos = torch.randperm(L - (3 + P), generator=g)[:ks[b]] + 3 + P
        ids[b, pos] = cfg.bbox_token
        p = torch.rand(ks[b], 2, 2, generator=g).sort(dim=1).values
        bx = torch.cat([p[:, 0, :], p[:, 1, :]], 1)
        bx[:, 2:] = torch.maximum(bx[:, 2:], bx[:, :2] + 2.0 / cfg.image_size).clamp(max=1.0)
        boxes.append(bx)
    images = torch.randn(B, 3, cfg.image_size, cfg.image_size, generator=g)
    return ids, images, boxes


def test_spi_path_matches_reference_golden_336():
    """fuse stack + fused GN/RoIAlign + pconv + flatten_linear + pos + updims vs the reference module's
    own fp32 output (golden).  bf16 tensor-core path vs fp32: rel-L2 <= 3e-2."""
    _, sd, toks, boxes, want = golden_case(336)
    cfg = EngineConfig(image_size=336, vit_layers=24, n_layers=0)
    vit_dummy = {k: v for k, v in random_state_dicts(EngineConfig(image_size=336, vit_layers=0, n_layers=0), 'cpu')[1].items()}
    cfg.select_index = 0  # no ViT layers are run in this test; taps are supplied directly
    eng = PrefillEngine(cfg, sd, vit_dummy, DEV)
    B = toks[0].shape[0]
    taps = {}
    for l, layer in enumerate(cfg.level_layers):
        cls = torch.zeros(B, 1, 1024)
        taps[layer] = torch.cat([cls, toks[l]], 1).to(DEV).contiguous()   # fp32 hidden states, as under autocast
    maps, ss = eng.fuse_maps(taps)
    counts = [b.shape[0] for b in boxes]
    bidx = torch.cat([torch.full((n,), float(i)) for i, n in enumerate(counts)]).to(DEV)
    got = eng.region_tokens(maps, ss, torch.cat(boxes).to(DEV), bidx)
    e = rel(got.cpu(), torch.from_numpy(want))
    print('SPI path vs reference-module golden (336): rel-L2 %.3e' % e)
    assert e < 2e-2


@pytest.mark.parametrize('n_layers,vit_layers,size,B,ks,T', [(2, 24, 336, 2, [3, 1], 24), (2, 12, 224, 1, [2], 16)])
def test_full_forward_vs_oracle(n_layers, vit_layers, size, B, ks, T):
    cfg = EngineConfig(image_size=size, vit_layers=vit_layers, n_layers=n_layers)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=7)          # bf16 weights (exactly representable in fp32)
    ids, images, boxes = make_inputs(cfg, B, ks, T)
    images = images.to(torch.bfloat16)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    got = eng.forward(ids.to(DEV), images.to(DEV), boxes)
    ref32, inter32 = model_oracle.forward(cfg, sd, vit_sd, ids, images.float(), boxes, DEV, autocast_bf16=False,
                                          return_intermediates=True)
    ref16, inter16 = model_oracle.forward(cfg, sd, vit_sd, ids, images, boxes, DEV, autocast_bf16=True,
                                          return_intermediates=True)
    e_engine, e_bf16ref = rel(got, ref32), rel(ref16, ref32)
    print('logits rel-L2 vs fp32 oracle: engine %.3e, bf16-autocast reference %.3e' % (e_engine, e_bf16ref))
    # per-stage error budget (engine | bf16-autocast reference), both against the fp32 oracle
    taps_e = eng.vit(images.to(DEV))
    for l, layer in enumerate(cfg.level_layers):
        print('  vit tap L%d: %.3e | %.3e' % (layer, rel(taps_e[layer][:, 1:], inter32['vit_taps'][l]),
                                              rel(inter16['vit_taps'][l], inter32['vit_taps'][l])))
    plan = eng.plan_boxes(boxes)
    maps_e, ss_e = eng.fuse_maps(taps_e)
    reg_e = eng.region_tokens(maps_e, ss_e, plan['boxes'], plan['bidx'])
    print('  region tokens: %.3e | %.3e' % (rel(reg_e, torch.cat(inter32['region'])),
                                            rel(torch.cat(inter16['region']), torch.cat(inter32['region']))))
    assert torch.isfinite(got.float()).all()
    assert e_engine < max(1.5 * e_bf16ref, 2e-2)
    # stage check: ViT taps
    taps = eng.vit(images.to(DEV))
    for l, layer in enumerate(cfg.level_layers):
        assert rel(taps[layer][:, 1:], inter32['vit_taps'][l]) < 2e-2
    # greedy next-token agreement with the fp32 oracle on (nearly) all rows
    agree = (got.float().argmax(-1) == ref32.argmax(-1)).float().mean().item()
    assert agree > 0.9, agree


def test_no_boxes_and_text_only_paths():
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=1)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=3)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    ids, images, _ = make_inputs(cfg, 1, [0], 12)
    out = eng.forward(ids.to(DEV), images.to(DEV, torch.bfloat16), None)      # bboxes=None (spi_llava.py:83-87)
    ref = model_oracle.forward(cfg, sd, vit_sd, ids, images.to(torch.bfloat16).float(), None, DEV)
    assert rel(out, ref) < 2e-2
    bad = ids.clone()
    bad[0, 2 + cfg.num_patches] = 5                                             # break the <im_end> position
    with pytest.raises(ValueError):
        eng.forward(bad.to(DEV), images.to(DEV, torch.bfloat16), None)


def test_full_size_properties_7b():
    """BASELINE configs[1] at full size (B=8, 336 px, 8 RoIs, L=706, 32 layers): properties that do
    not need an oracle run -- causality, sample independence / permutation equivariance, box locality."""
    cfg = EngineConfig(image_size=336, vit_layers=24, n_layers=32)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=11)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    del sd, vit_sd
    torch.cuda.empty_cache()
    ids, images, boxes = make_inputs(cfg, 8, [8] * 8, 128, seed=5)
    ids, images = ids.to(DEV), images.to(DEV, torch.bfloat16)
    base = eng.forward(ids, images, boxes).float()
    assert base.shape == (8, 706, 32006) and torch.isfinite(base).all()
    # (0) idempotence: no atomics on the path -> a repeated run is bitwise identical
    assert torch.equal(eng.forward(ids, images, boxes).float(), base)
    same, changed = 1e-6, 1e-3   # rel-L2 thresholds
    # (1) causality: editing the last text token leaves all earlier positions unchanged
    ids2 = ids.clone()
    ids2[:, -1] = (ids2[:, -1] + 7) % 31000 + 3
    out2 = eng.forward(ids2, images, boxes).float()
    assert rel(out2[:, :-1], base[:, :-1]) < same
    assert rel(out2[:, -1], base[:, -1]) > changed
    # (2) samples are independent: permuting the batch permutes the logits
    perm = torch.tensor([3, 0, 7, 1, 6, 2, 5, 4])
    out3 = eng.forward(ids[perm], images[perm], [boxes[i] for i in perm.tolist()]).float()
    assert rel(out3, base[perm]) < same
    # (3) box locality: moving sample 0's last box changes nothing before its <bbox> token and nothing in other samples
    boxes4 = [b.clone() for b in boxes]
    boxes4[0][-1] = torch.tensor([0.05, 0.05, 0.95, 0.95])
    out4 = eng.forward(ids, images, boxes4).float()
    assert rel(out4[1:], base[1:]) < same
    pos = torch.where(ids[0] == cfg.bbox_token)[0]
    assert rel(out4[0, :pos[-1]], base[0, :pos[-1]]) < same
    assert rel(out4[0, pos[-1]:], base[0, pos[-1]:]) > changed


def test_engine_vs_reference_forward_golden_224():
    """Engine (bf16) vs logits of the reference's own SPILlavaMPTForCausalLM.forward (fp32 golden,
    224 px reference-exact mode, CLIP-L/14 x24 + 2-layer LLaMA-4096).  rel-L2 <= 2.5e-2."""
    from tests.test_model_oracle_cpu import full_model_case
    cfg, sd, vit_sd, ids, images, boxes, z = full_model_case()
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    got = eng.forward(ids.to(DEV), images.to(DEV, torch.bfloat16), boxes).float().cpu()
    probe = torch.from_numpy(z['probe'])
    e = rel(got[:, probe], torch.from_numpy(z['logits']))
    print('engine vs reference-forward golden (224): rel-L2 %.3e' % e)
    assert e < 2.5e-2
    assert (got.argmax(-1).numpy() == z['argmax']).mean() > 0.9


def test_right_padded_batch_matches_oracle_on_valid_positions():
    """Padded batch (collator layout, data_modules.py:33-44): logits at valid positions equal the
    unpadded single-sample run; oracle comparison with HF's attention_mask on the same inputs."""
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=2)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=21)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    ids, images, boxes = make_inputs(cfg, 2, [2, 1], 40, seed=9)
    L = ids.shape[1]
    short = L - 17
    mask = torch.ones(2, L, dtype=torch.long)
    mask[1, short:] = 0
    ids[1, short:] = 0                                   # pad id
    k1 = int((ids[1, :short] == cfg.bbox_token).sum())
    boxes[1] = boxes[1][:k1]
    images = images.to(torch.bfloat16)
    got = eng.forward(ids.to(DEV), images.to(DEV), boxes, attention_mask=mask).float()
    solo = eng.forward(ids[1:2, :short].contiguous().to(DEV), images[1:2].to(DEV), [boxes[1]]).float()
    assert rel(got[1, :short], solo[0]) < 1e-6           # padding does not leak into valid positions
    full0 = eng.forward(ids[0:1].to(DEV), images[0:1].to(DEV), [boxes[0]]).float()
    assert rel(got[0], full0[0]) < 1e-6


def test_zero_box_samples():
    """Edge cases of layers.py:315-318 / det_llava.py:463: a sample with K_i = 0 inside a batch that has
    boxes, and a batch with no boxes at all (empty tensors, not None)."""
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=1)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=13)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    ids, images, boxes = make_inputs(cfg, 2, [2, 0], 16, seed=4)
    images = images.to(torch.bfloat16)
    got = eng.forward(ids.to(DEV), images.to(DEV), boxes).float()
    ref = model_oracle.forward(cfg, sd, vit_sd, ids, images.float(), boxes, DEV)
    assert rel(got, ref) < 2e-2
    ids0, images0, boxes0 = make_inputs(cfg, 2, [0, 0], 16, seed=6)
    got0 = eng.forward(ids0.to(DEV), images0.to(DEV, torch.bfloat16), boxes0).float()       # K = 0 overall
    none0 = eng.forward(ids0.to(DEV), images0.to(DEV, torch.bfloat16), None).float()        # bboxes=None
    assert torch.equal(got0, none0)


def test_decode_loop_matches_prefill_logits():
    """SURVEY 8(f1): prefill + KV-cache decode steps reproduce the logits of a full prefill over the
    extended sequence (teacher forcing); greedy generate() returns the same tokens as re-running prefill."""
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=2)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=17)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    ids, images, boxes = make_inputs(cfg, 2, [2, 1], 24, seed=8)
    images = images.to(DEV, torch.bfloat16)
    n_new = 5
    ids = torch.cat([ids, torch.randint(3, 32000, (2, n_new), generator=torch.Generator().manual_seed(3))], 1)
    full = eng.forward(ids.to(DEV), images, boxes).float()                   # [B, L, V]
    L0 = ids.shape[1] - n_new
    from gpt4roi_b200.engine import KVCache
    cache = KVCache(cfg, 2, ids.shape[1], DEV)
    # the <bbox> tokens must all be inside the prefix for this check
    assert all(int(torch.where(ids[b] == cfg.bbox_token)[0].max()) < L0 for b in range(2))
    plan = eng.plan_boxes(boxes)
    pre = eng.forward_device(ids[:, :L0].contiguous().to(DEV), images, plan, last_only=True, cache=cache).float()
    assert rel(pre[:, 0], full[:, L0 - 1]) < 5e-3
    for t in range(n_new):
        step = eng.decode_step(ids[:, L0 + t:L0 + t + 1].contiguous().to(DEV), cache).float()
        e = rel(step[:, 0], full[:, L0 + t])
        assert e < 1e-2, (t, e)
    # generate(): greedy continuation is self-consistent with prefill
    out = eng.generate(ids[:, :L0].contiguous(), images, boxes, max_new_tokens=3)
    assert out.shape == (2, L0 + 3)
    chk = eng.forward(out[:, :-1].contiguous(), images, boxes).float()
    agree = (chk[:, L0 - 1:].argmax(-1) == out[:, L0:]).float().mean().item()
    assert agree >= 0.8, agree


def test_graphed_decode_is_bitwise_equal_to_eager_decode():
    """GraphedDecode (device-side position, one CUDA-graph replay per token) must produce exactly the
    logits of the eager decode_step at every step: same kernels, same order, no atomics."""
    from gpt4roi_b200.engine import GraphedDecode, KVCache
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=2)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=19)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    ids, images, boxes = make_inputs(cfg, 2, [1, 2], 20, seed=9)
    images = images.to(DEV, torch.bfloat16)
    plan = eng.plan_boxes(boxes)
    n_new = 6
    toks = torch.randint(3, 32000, (n_new, 2, 1), generator=torch.Generator().manual_seed(4)).to(DEV)
    outs = []
    for graphed in (False, True):
        cache = KVCache(cfg, 2, ids.shape[1] + n_new + 2, DEV)
        eng.forward_device(ids.to(DEV), images, plan, last_only=True, cache=cache)
        stepper = GraphedDecode(eng, cache) if graphed else None
        seq = []
        for t in range(n_new):
            lg = stepper.step(toks[t]) if graphed else eng.decode_step(toks[t], cache)
            seq.append(lg.clone())
        assert cache.length == ids.shape[1] + n_new
        outs.append(torch.stack(seq))
    assert torch.equal(outs[0], outs[1])
    # the cache-full guard still fires in graph mode
    cache = KVCache(cfg, 2, ids.shape[1] + 1, DEV)
    eng.forward_device(ids.to(DEV), images, plan, last_only=True, cache=cache)
    st = GraphedDecode(eng, cache)
    st.step(toks[0])
    with pytest.raises(RuntimeError):
        st.step(toks[1])


def test_fused_decode_step_matches_the_unfused_sequence():
    """g4r_decode_gemm_bf16 (q|k|v + RoPE + KV append in one launch; gate/up + SwiGLU in one) vs the 8-launch sequence
    it replaces: the KV append only moves into the epilogue, so logits and KV cache rows are bitwise equal; batch 1, 8
    and 16 (both activation-block variants)."""
    import gpt4roi_b200.engine as E
    from gpt4roi_b200.engine import KVCache
    cfg = EngineConfig(image_size=224, vit_layers=12, n_layers=2)
    sd, vit_sd = random_state_dicts(cfg, DEV, seed=23)
    eng = PrefillEngine(cfg, sd, vit_sd, DEV)
    for B in (1, 8, 16):
        ids, images, boxes = make_inputs(cfg, B, [1] * B, 12, seed=30 + B)
        images = images.to(DEV, torch.bfloat16)
        plan = eng.plan_boxes(boxes)
        toks = torch.randint(3, 32000, (3, B, 1), generator=torch.Generator().manual_seed(B)).to(DEV)
        res = {}
        try:
            for fused in (True, False):
                E._FUSED_DECODE = fused
                cache = KVCache(cfg, B, ids.shape[1] + 4, DEV)
                eng.forward_device(ids.to(DEV), images, plan, last_only=True, cache=cache)
                outs = [eng.decode_step(toks[t], cache).float().clone() for t in range(3)]
                res[fused] = (torch.stack(outs), cache.k[1][:, :cache.length].float().clone(), cache.v[1][:, :cache.length].float().clone())
        finally:
            E._FUSED_DECODE = True
        for a, b in zip(res[True], res[False]):      # KV append in the epilogue only: the very same values
            assert torch.equal(a, b), B
