"""Region-token prefill engine: CLIP-ViT-L/14 -> MLVL fuse -> multi-level RoIAlign -> region
projector -> splice -> LLaMA prefill -> lm_head, every op a hand-written sm_100a kernel behind
the C ABI.  PyTorch supplies device memory, streams and CUDA-graph capture only.

Reference call stack reproduced (SURVEY.md 3.3):
  gpt4roi/models/spi_llava.py:23-205   SPILlavaLlamaModel.forward
  gpt4roi/models/layers.py:182-195     MLVLFuseModule.forward
  gpt4roi/models/layers.py:218-236     MLVLROIQueryModule.forward
  gpt4roi/models/layers.py:280-335     MlvlRoIExtractor.forward
  llava/model/llava.py:203-261         LlavaLlamaForCausalLM.forward (lm_head)
  transformers CLIPVisionModel / LlamaModel (third party, pyproject.toml:19)

Weights come in with the reference's parameter names (SURVEY.md App. C) and are re-laid-out
ONCE at load time (fused QKV, interleaved gate/up, NHWC conv filters, flatten_linear permuted
from (c,ph,pw) to (ph,pw,c)).  Numerics: bf16 storage, fp32 accumulation, rounding points of the
reference under bf16 autocast.
"""
import math

import torch

from . import dense, kernels
from .roi_align import roi_align_mlvl
from .splice import splice_region_tokens

BF16 = torch.bfloat16


class EngineConfig:
    def __init__(self, image_size=336, patch_size=14, vit_hidden=1024, vit_heads=16, vit_layers=24,
                 vit_mlp=4096, vit_eps=1e-5, select_layer=-2, num_levels=4,
                 hidden=4096, n_heads=32, n_layers=32, mlp=11008, vocab=32006, rms_eps=1e-6,
                 rope_theta=10000.0, roi_out=14, roi_sampling=2, spi_dim=1024, gn_groups=64,
                 im_patch_token=32001, bbox_token=32002, im_start_token=32004, im_end_token=32005,
                 llama_stream=None, dtype='bf16'):
        """dtype: the 16-bit storage type of weights and activations -- 'bf16' (training scripts, BASELINE "7B bf16
        prefill") or 'fp16' (the demo: gpt4roi/app.py:74-98,271 builds the model with .half()); fp16 runs the `_f16`
        twins of every kernel (csrc/act_type.cuh), same fp32 accumulation and rounding points.
        llama_stream: dtype of the LLaMA residual stream in the prefill -- 'bf16' (default: what the reference has
        when the model was cast to bf16, the BASELINE "7B bf16 prefill" mode) or 'fp32' (what the reference has
        whenever its parameters are fp32 under autocast; 25 % closer to the fp32 anchor at 32 layers, 2.4 % slower:
        tests/test_parity_7b_gpu.py, profiles/r2_bench_stream_ab.json).  Env G4R_LLAMA_STREAM overrides the default."""
        import os
        if llama_stream is None:
            llama_stream = os.environ.get('G4R_LLAMA_STREAM', 'bf16')
        if llama_stream not in ('fp32', 'bf16'):
            raise ValueError('llama_stream must be fp32 or bf16 (bf16 = the 16-bit storage type)')
        if dtype in (torch.bfloat16, torch.float16):
            dtype = 'bf16' if dtype == torch.bfloat16 else 'fp16'
        if dtype not in ('bf16', 'fp16'):
            raise ValueError("dtype must be 'bf16' or 'fp16'")
        self.__dict__.update(locals())
        del self.__dict__['os']
        del self.__dict__['self']
        self.torch_dtype = torch.bfloat16 if dtype == 'bf16' else torch.float16
        self.grid = image_size // patch_size
        self.num_patches = self.grid ** 2
        self.head_dim = hidden // n_heads
        self.vit_head_dim = vit_hidden // vit_heads
        self.strides = [patch_size / 8, patch_size / 4, patch_size / 2, patch_size][-num_levels:] \
            if num_levels <= 4 else None
        self.level_sizes = [self.grid * 2 ** (num_levels - 1 - l) for l in range(num_levels)]
        # spi_llava.py:68-82: hidden_states[select::-3][::-1][-num_levels:]
        sel = select_layer if select_layer >= 0 else vit_layers + 1 + select_layer
        lv = list(range(sel, -1, -3))[::-1][-num_levels:]
        self.select_index = sel
        self.level_layers = lv


def _b(t, dev, dt=BF16):
    return t.detach().to(device=dev, dtype=dt).contiguous()


class PrefillEngine:
    """Holds re-laid-out weights on one GPU and runs the fused forward."""

    def __init__(self, cfg, llm_sd, vit_sd, device, parts=('vit', 'spi', 'llm')):
        """parts: which weight groups to prepare -- ('spi',) builds an SPI-module-only engine (the model-seam
        mirrors of MLVLROIQueryModule / MLVLFuseModule / MlvlRoIExtractor run on it)."""
        self.cfg = cfg
        self.dev = torch.device(device)
        self.dt = cfg.torch_dtype          # bf16, or fp16 for the demo's dtype
        self.parts = tuple(parts)
        if 'vit' in self.parts:
            self._prepare_vit(vit_sd)
        if 'spi' in self.parts:
            self._prepare_spi(llm_sd)
        if 'llm' in self.parts:
            self._prepare_llm(llm_sd)
        self._rope_cache = {}

    # ------------------------------------------------------------------ weight preparation
    def _prepare_vit(self, sd):
        c, dev = self.cfg, self.dev
        p = 'vision_model.'
        kreal = 3 * c.patch_size ** 2
        self.vit_kpad = (kreal + 7) // 8 * 8
        w = sd[p + 'embeddings.patch_embedding.weight'].reshape(c.vit_hidden, kreal)
        wp = torch.zeros(c.vit_hidden, self.vit_kpad, dtype=self.dt, device=dev)
        wp[:, :kreal] = w.to(dev, self.dt)
        self.vit_patch_w = wp
        self.vit_cls = _b(sd[p + 'embeddings.class_embedding'], dev, self.dt)
        self.vit_pos = _b(sd[p + 'embeddings.position_embedding.weight'], dev, self.dt)
        self.vit_pre_ln = (_b(sd[p + 'pre_layrnorm.weight'], dev, self.dt), _b(sd[p + 'pre_layrnorm.bias'], dev, self.dt))
        self.vit_layers = []
        for i in range(c.select_index):  # layers beyond the selected hidden state are dead work
            q = p + 'encoder.layers.%d.' % i
            wqkv = torch.cat([sd[q + 'self_attn.%s_proj.weight' % n] for n in 'qkv'], 0)
            bqkv = torch.cat([sd[q + 'self_attn.%s_proj.bias' % n] for n in 'qkv'], 0)
            self.vit_layers.append(dict(
                ln1=(_b(sd[q + 'layer_norm1.weight'], dev, self.dt), _b(sd[q + 'layer_norm1.bias'], dev, self.dt)),
                wqkv=_b(wqkv, dev, self.dt), bqkv=_b(bqkv, dev, self.dt),
                wo=_b(sd[q + 'self_attn.out_proj.weight'], dev, self.dt), bo=_b(sd[q + 'self_attn.out_proj.bias'], dev, self.dt),
                ln2=(_b(sd[q + 'layer_norm2.weight'], dev, self.dt), _b(sd[q + 'layer_norm2.bias'], dev, self.dt)),
                w1=_b(sd[q + 'mlp.fc1.weight'], dev, self.dt), b1=_b(sd[q + 'mlp.fc1.bias'], dev, self.dt),
                w2=_b(sd[q + 'mlp.fc2.weight'], dev, self.dt), b2=_b(sd[q + 'mlp.fc2.bias'], dev, self.dt)))

    def _prepare_spi(self, sd):
        """SPI-module weights in engine layout.  The two halves are independent (a stand-alone MLVLFuseModule or
        MlvlRoIExtractor mirror owns only one of them): whatever keys are present are prepared."""
        c, dev = self.cfg, self.dev
        p = 'model.spi_module.'
        C = c.spi_dim
        self.spi_cpad = (C + 2 + 63) // 64 * 64  # 1026 -> 1088
        if p + 'mlvl_fuse.input_conv.0.weight' in sd:
            self.in_w, self.in_b = [], []
            for l in range(c.num_levels):
                w = sd[p + 'mlvl_fuse.input_conv.%d.weight' % l].reshape(C, C + 2)
                wp = torch.zeros(C, self.spi_cpad, dtype=self.dt, device=dev)
                wp[:, :C + 2] = w.to(dev, self.dt)
                self.in_w.append(wp)
                self.in_b.append(_b(sd[p + 'mlvl_fuse.input_conv.%d.bias' % l], dev, self.dt))
            self.fuse = []
            for r in range(5):
                q = p + 'mlvl_fuse.fuse_convs.%d.' % r
                w = sd[q + 'conv.weight'].to(dev, self.dt).permute(0, 2, 3, 1).contiguous()  # [Cout,kh,kw,Cin]
                self.fuse.append(dict(w=w, gamma=_b(sd[q + 'gn.weight'], dev, self.dt), beta=_b(sd[q + 'gn.bias'], dev, self.dt)))
        q = p + 'roi_align.'
        if q + 'flatten_linear.weight' in sd:
            pw = torch.stack([sd[q + 'pconvs.%d.weight' % l].to(dev, self.dt).permute(0, 2, 3, 1)
                              for l in range(c.num_levels)], 1).contiguous()  # [Cout, L, kh, kw, Cin]
            self.pconv_w = pw
            self.pconv_b = sum(sd[q + 'pconvs.%d.bias' % l].to(dev, torch.float32) for l in range(c.num_levels)).contiguous()
            R = c.roi_out
            fw = sd[q + 'flatten_linear.weight']  # [1024, C*R*R] in (c, ph, pw) order (layers.py:326)
            self.flat_w = fw.to(dev, self.dt).reshape(-1, C, R, R).permute(0, 2, 3, 1).reshape(fw.shape[0], -1).contiguous()
            self.flat_b = _b(sd[q + 'flatten_linear.bias'], dev, self.dt)
            self.pos = [_b(sd[q + 'pos_embedd.%s' % n], dev, self.dt) for n in
                        ('0.weight', '0.bias', '2.weight', '2.bias', '3.weight', '3.bias', '5.weight', '5.bias')]
            self.up_w, self.up_b = _b(sd[q + 'updims.weight'], dev, self.dt), _b(sd[q + 'updims.bias'], dev, self.dt)
            kb = self.flat_w.shape[1] // 64
            self.flat_splits = next(s for s in (16, 14, 8, 7, 4, 2, 1) if kb % s == 0)
        if 'model.mm_projector.weight' in sd:
            self.proj_w, self.proj_b = _b(sd['model.mm_projector.weight'], dev, self.dt), _b(sd['model.mm_projector.bias'], dev, self.dt)

    def _prepare_llm(self, sd):
        c, dev = self.cfg, self.dev
        self.embed = _b(sd['model.embed_tokens.weight'], dev, self.dt)
        self.layers = []
        for i in range(c.n_layers):
            q = 'model.layers.%d.' % i
            wqkv = torch.cat([sd[q + 'self_attn.%s_proj.weight' % n].to(dev, self.dt) for n in 'qkv'], 0).contiguous()
            g, u = sd[q + 'mlp.gate_proj.weight'].to(dev, self.dt), sd[q + 'mlp.up_proj.weight'].to(dev, self.dt)
            wgu = torch.stack([g, u], 1).reshape(2 * g.shape[0], g.shape[1]).contiguous()  # rows: g0,u0,g1,u1,...
            self.layers.append(dict(
                ln_in=_b(sd[q + 'input_layernorm.weight'], dev, self.dt), wqkv=wqkv,
                wo=_b(sd[q + 'self_attn.o_proj.weight'], dev, self.dt),
                ln_post=_b(sd[q + 'post_attention_layernorm.weight'], dev, self.dt), wgu=wgu,
                wdown=_b(sd[q + 'mlp.down_proj.weight'], dev, self.dt)))
            del g, u
        self.norm_w = _b(sd['model.norm.weight'], dev, self.dt)
        self.lm_head = _b(sd['lm_head.weight'], dev, self.dt) if 'lm_head.weight' in sd else None   # LlamaModel-only seam
        self.vocab_pad = (c.vocab + 63) // 64 * 64

    def _rope(self, L):
        """cos/sin tables exactly as LlamaRotaryEmbedding (modeling_llama.py:118-135): fp32 then bf16."""
        if L not in self._rope_cache:
            c = self.cfg
            inv = 1.0 / (c.rope_theta ** (torch.arange(0, c.head_dim, 2, dtype=torch.int64).float() / c.head_dim))
            freqs = torch.arange(L, dtype=torch.float32)[:, None] * inv[None, :]
            emb = torch.cat((freqs, freqs), -1)
            self._rope_cache[L] = (emb.cos().to(self.dev, self.dt).contiguous(), emb.sin().to(self.dev, self.dt).contiguous())
        return self._rope_cache[L]

    # ------------------------------------------------------------------ stages
    def vit(self, images):
        """images bf16 [B,3,S,S] -> dict{layer index: hidden state [B,P+1,C]} for the consumed layers."""
        c = self.cfg
        B = images.shape[0]
        P, T = c.num_patches, c.num_patches + 1
        patches = kernels.patchify(images, c.patch_size, self.vit_kpad)
        pe = dense.linear(patches, self.vit_patch_w)
        x = kernels.vit_embed(pe, self.vit_cls, self.vit_pos, B, P)
        # Residual stream in fp32, as the reference has it under autocast: nn.LayerNorm returns fp32
        # (pre_layrnorm turns the bf16 embeddings into an fp32 stream) and `residual + bf16_branch`
        # stays fp32; the Linears see bf16 inputs (autocast cast) and produce bf16 outputs.
        F32 = torch.float32
        x = kernels.layernorm_ex(x, *self.vit_pre_ln, eps=c.vit_eps, out_dtype=F32).view(B * T, c.vit_hidden)
        taps = {}
        scale = c.vit_head_dim ** -0.5
        for i, w in enumerate(self.vit_layers):
            h = kernels.layernorm_ex(x, *w['ln1'], eps=c.vit_eps)
            qkv = dense.linear(h, w['wqkv'], w['bqkv'])
            a = kernels.attention(qkv, B, T, c.vit_heads, c.vit_head_dim, False, scale)
            x = dense.linear(a, w['wo'], w['bo'], residual=x, out_dtype=F32, round_branch=True)
            h = kernels.layernorm_ex(x, *w['ln2'], eps=c.vit_eps)
            f = dense.linear(h, w['w1'], w['b1'], act='quick_gelu')
            x = dense.linear(f, w['w2'], w['b2'], residual=x, out_dtype=F32, round_branch=True)
            if (i + 1) in c.level_layers:
                taps[i + 1] = x.view(B, T, c.vit_hidden)
        return taps

    def fuse_maps(self, taps, has_cls=True, pre_upsampled=False):
        """MLVLROIQueryModule upsampling + MLVLFuseModule: returns the last round's raw conv outputs
        (bf16 NHWC) and the per-(image,channel) GroupNorm scale/shift still to be applied.
        taps: {layer: [B, 1+P, C]} ViT hidden states (CLS first), or with has_cls=False a list / dict of
        [B, P, C] token maps in level order (what MLVLROIQueryModule.forward receives, layers.py:218-224).
        pre_upsampled: the level-l entry already has the pyramid size [B, H_l*H_l, C] (MLVLFuseModule.forward's
        input, layers.py:182): the resampling step degenerates to the identity and only appends the coordinates."""
        c = self.cfg
        C = c.spi_dim
        if isinstance(taps, (list, tuple)):
            taps = {layer: t for layer, t in zip(c.level_layers, taps)}
        B = next(iter(taps.values())).shape[0]
        maps = []
        for l, layer in enumerate(c.level_layers):
            H = c.level_sizes[l]
            up = kernels.upsample_tokens_coords(taps[layer], H if pre_upsampled else c.grid, H, self.spi_cpad,
                                                has_cls=has_cls, dtype=self.dt)
            m = dense.linear(up.view(-1, self.spi_cpad), self.in_w[l], self.in_b[l]).view(B, H, H, C)
            maps.append(m)
        ss = [None] * c.num_levels
        n = c.num_levels
        for r in range(5):
            new, stats = [], []
            for l in range(n):
                top, down = min(l + 1, n - 1), max(l - 1, 0)
                x_in = kernels.fuse_gather(maps[l], maps[top], maps[down], ss[l], ss[top], ss[down])
                st = torch.zeros((B, dense.gn_slots(c.level_sizes[l], c.level_sizes[l]), c.gn_groups, 2),
                                 dtype=torch.float32, device=self.dev)
                new.append(dense.conv_nhwc(x_in, self.fuse[r]['w'], gn_stats=st))
                stats.append(st)
            maps = new
            ss = [kernels.gn_finalize(stats[l], self.fuse[r]['gamma'], self.fuse[r]['beta'],
                                      count=c.level_sizes[l] ** 2 * (C // c.gn_groups)) for l in range(n)]
        return maps, ss

    def region_tokens(self, maps, ss, boxes, batch_idx):
        """MlvlRoIExtractor.forward: boxes fp32 [K,4] normalised xyxy, batch_idx fp32 [K] -> [K,hidden]."""
        c = self.cfg
        K = boxes.shape[0]
        rois = torch.cat([batch_idx[:, None], boxes * float(c.image_size)], 1).contiguous()  # layers.py:294-302
        scales = [float(torch.tensor(1.0 / s, dtype=torch.float32)) for s in c.strides]
        # ss=None: the maps are already activated (MlvlRoIExtractor.forward called on its own)
        feats = roi_align_mlvl(maps, rois, c.roi_out, scales, c.roi_sampling, True, out_dtype=self.dt,
                               gn_scale=None if ss is None else [s for s, _ in ss],
                               gn_shift=None if ss is None else [b for _, b in ss])
        R = c.roi_out
        pc = dense.conv_nhwc(feats.view(c.num_levels * K, R, R, c.spi_dim), self.pconv_w, self.pconv_b,
                             act='relu', levels=c.num_levels)
        acc = dense.linear(pc.view(K, -1), self.flat_w, out_dtype=torch.float32, k_splits=self.flat_splits) \
            if self.flat_splits > 1 else dense.linear(pc.view(K, -1), self.flat_w, out_dtype=torch.float32)
        pos = kernels.pos_embed_mlp(boxes.contiguous(), *self.pos)
        t = kernels.add_bias_pos_cast(acc, self.flat_b, pos)
        return dense.linear(t, self.up_w, self.up_b)

    def llama(self, embeds, B, L, last_only=False, seqlens=None, cache=None, hidden_taps=None, want='logits'):
        """hidden_taps: optional dict {n: None}; filled with a copy of the residual stream after decoder layer n
        (1-based; the parity tests record error growth with depth).  want='hidden' returns the final-norm
        hidden states [B, L, hidden] instead of logits (LlamaModel.forward's last_hidden_state)."""
        c = self.cfg
        x = embeds.view(B * L, c.hidden)
        cos, sin = self._rope(L)
        scale = c.head_dim ** -0.5
        # fp32 residual stream: the first o_proj epilogue widens it (bf16 residual in, fp32 out); every branch output
        # is rounded to bf16 before the fp32 add, as a bf16 nn.Linear output added to an fp32 stream under autocast
        f32 = dict(out_dtype=torch.float32, round_branch=True) if c.llama_stream == 'fp32' else {}
        for li, w in enumerate(self.layers):
            h = kernels.rmsnorm(x, w['ln_in'], c.rms_eps)
            if c.head_dim == 128 and (2 * c.hidden) % 256 == 0:
                qkv = dense.qkv_rope(h, w['wqkv'], cos, sin, L, 2 * c.hidden)   # RoPE fused into the GEMM epilogue
            else:
                qkv = dense.linear(h, w['wqkv'])
                kernels.rope_inplace(qkv, cos, sin, L, 2 * c.n_heads, c.head_dim)
            if cache is not None:  # keep post-RoPE K and V for the decode loop
                kernels.kv_append(qkv, cache.k[li], cache.v[li], B, L, 0)
            a = kernels.attention(qkv, B, L, c.n_heads, c.head_dim, True, scale, seqlens=seqlens)
            x = dense.linear(a, w['wo'], residual=x, **f32)
            h = kernels.rmsnorm(x, w['ln_post'], c.rms_eps)
            f = dense.linear(h, w['wgu'], act='swiglu')
            x = dense.linear(f, w['wdown'], residual=x, **f32)
            if hidden_taps is not None and (li + 1) in hidden_taps:
                hidden_taps[li + 1] = x.view(B, L, c.hidden).clone()
        if last_only:
            x = x.view(B, L, c.hidden)[:, -1].contiguous()
        x = kernels.rmsnorm(x, self.norm_w, c.rms_eps)
        if want == 'hidden':
            return x.view(B, -1, c.hidden)
        if self.lm_head is None:
            raise RuntimeError('this engine was built without lm_head.weight (LlamaModel seam): use want="hidden"')
        rows = x.shape[0]
        # padded row stride keeps the epilogue's 128-bit stores aligned (vocab 32006 is not a multiple of 8)
        buf = torch.empty((rows, self.vocab_pad), dtype=self.dt, device=self.dev)
        dense.linear(x, self.lm_head, out=buf[:, :c.vocab])
        return buf.view(B, rows // B, self.vocab_pad)[:, :, :c.vocab]

    # ------------------------------------------------------------------ whole path
    def plan_boxes(self, bboxes):
        """Host-side packing of the per-sample box lists (the reference does this with torch.cat and
        python loops at layers.py:283-302): returns device tensors so that `forward_device` contains no
        host->device traffic and can be captured in a CUDA graph."""
        if bboxes is None or len(bboxes) == 0:
            return None
        counts = [0 if b is None else int(b.shape[0]) for b in bboxes]
        K = sum(counts)
        offs = torch.tensor([0] + list(torch.tensor(counts).cumsum(0).tolist()), dtype=torch.int32).to(self.dev)
        if K > 0:
            boxes = torch.cat([b.to(self.dev, torch.float32) for b in bboxes if b is not None and b.shape[0]], 0).contiguous()
            bidx = torch.cat([torch.full((n,), float(i)) for i, n in enumerate(counts)]).to(self.dev)
        else:
            boxes = torch.zeros((0, 4), dtype=torch.float32, device=self.dev)
            bidx = torch.zeros((0,), dtype=torch.float32, device=self.dev)
        return dict(K=K, boxes=boxes, bidx=bidx, offs=offs)

    def forward_device(self, input_ids, images, plan, validate=True, last_only=False, seqlens=None, cache=None,
                       hidden_taps=None, want='logits', stage_taps=None):
        """Device-only forward (capturable): input_ids int64 [B,L], images bf16 [B,3,S,S] on the GPU.
        images=None: text-only forward (spi_llava.py:47-48 skips the vision branch when no image is given).
        stage_taps: optional dict filled with 'vit_taps', 'region', 'embeds' (parity tests)."""
        c = self.cfg
        B, L = input_ids.shape
        if images is None:
            embeds = splice_region_tokens(input_ids, self.embed, None, None, 0, c.im_patch_token, c.im_start_token,
                                          c.im_end_token, c.bbox_token, validate=False)
            if cache is not None:
                cache.length = L
            return self.llama(embeds, B, L, last_only=last_only, seqlens=seqlens, cache=cache,
                              hidden_taps=hidden_taps, want=want)
        taps = self.vit(images)
        feat = kernels.cast_tokens_f32_bf16(taps[c.select_index], dtype=self.dt)  # spi_llava.py:68-73 (+ autocast cast, CLS dropped)
        img_rows = dense.linear(feat, self.proj_w, self.proj_b).view(B, c.num_patches, c.hidden)
        region = None
        if plan is not None:
            if plan['K'] > 0:
                maps, ss = self.fuse_maps(taps)
                rows = self.region_tokens(maps, ss, plan['boxes'], plan['bidx'])
            else:
                rows = torch.zeros((1, c.hidden), dtype=self.dt, device=self.dev)
            region = (rows, plan['offs'])
        embeds = splice_region_tokens(input_ids, self.embed, img_rows, region, c.num_patches, c.im_patch_token,
                                      c.im_start_token, c.im_end_token, c.bbox_token, validate=validate)
        if stage_taps is not None:
            stage_taps['vit_taps'] = [taps[l][:, 1:] for l in c.level_layers]
            stage_taps['region'] = region[0] if (region is not None and plan['K'] > 0) else None
            stage_taps['embeds'] = embeds
        if cache is not None:
            cache.length = L
        return self.llama(embeds, B, L, last_only=last_only, seqlens=seqlens, cache=cache, hidden_taps=hidden_taps,
                          want=want)

    def forward(self, input_ids, images, bboxes, validate=True, last_only=False, attention_mask=None,
                hidden_taps=None, want='logits', stage_taps=None, cache=None):
        """Public entry: input_ids int64 [B,L]; images [B,3,S,S]; bboxes list (len B) of [K_i,4]
        normalised xyxy or None (host or device tensors).  Returns logits [B,L,V] (bf16) -- [B,1,V]
        with last_only.  attention_mask: None / all-ones, or a RIGHT-padded 0/1 mask [B,L] (the collator's
        pad_sequence layout, data_modules.py:33-44); logits at padded positions are don't-care."""
        plan = self.plan_boxes(bboxes)
        seqlens = None
        if attention_mask is not None:
            m = attention_mask.to(self.dev).to(torch.int32)
            lens = m.sum(1)
            if not bool((m == (torch.arange(m.shape[1], device=self.dev)[None] < lens[:, None])).all()):
                raise NotImplementedError('only right-padded attention masks are supported')
            seqlens = lens.to(torch.int32).contiguous()
        return self.forward_device(input_ids.to(self.dev, non_blocking=True).contiguous(),
                                   None if images is None else images.to(self.dev, self.dt, non_blocking=True).contiguous(),
                                   plan, validate, last_only, seqlens, cache=cache, hidden_taps=hidden_taps, want=want,
                                   stage_taps=stage_taps)


# Decode steps at B <= 16 take the fused GEMMs of g4r_decode_gemm_bf16; the unfused sequence remains the path for the
# other shapes and the reference the tests compare the fused step against (they switch this off).
_FUSED_DECODE = True


class KVCache:
    """Per-layer K/V cache [B, Lmax, n_heads*head_dim] (the engine's 16-bit type, post-RoPE keys) for the decode loop."""

    def __init__(self, cfg, B, max_len, device):
        hd = cfg.n_heads * cfg.head_dim
        dt = cfg.torch_dtype
        self.k = [torch.empty((B, max_len, hd), dtype=dt, device=device) for _ in range(cfg.n_layers)]
        self.v = [torch.empty((B, max_len, hd), dtype=dt, device=device) for _ in range(cfg.n_layers)]
        self.B, self.max_len, self.length = B, max_len, 0


def _decode_step(self, token_ids, cache, pos_dev=None):
    """One decode step (SURVEY.md 8(f1)): token_ids int64 [B,1] -> logits [B,1,V]; the vision / SPI branch
    is skipped exactly as the reference does for input_ids.shape[1] == 1 (spi_llava.py:47-48).
    pos_dev: optional device int32 holding the current length (CUDA-graph replay: the kernels read the
    position from memory instead of from a launch argument)."""
    from . import lib
    if cache.length + 1 > cache.max_len:
        raise RuntimeError('KV cache is full (%d)' % cache.max_len)
    # every kernel of the step only READS weights: let each one start in its predecessor's tail and fetch its first
    # weight block before it waits for the predecessor (programmatic dependent launch, csrc/common.cuh)
    prev = lib.set_pdl(True)
    try:
        return _decode_step_chain(self, token_ids, cache, pos_dev)
    finally:
        lib.set_pdl(prev)


def _decode_step_chain(self, token_ids, cache, pos_dev):
    c = self.cfg
    B = token_ids.shape[0]
    pos = cache.length
    kv_len = cache.max_len if pos_dev is not None else pos + 1   # sizes the score buffer when device-driven
    x = splice_region_tokens(token_ids, self.embed, None, None, 0, c.im_patch_token, c.im_start_token,
                             c.im_end_token, c.bbox_token, validate=False).view(B, c.hidden)
    cos, sin = self._rope(cache.max_len)
    scale = c.head_dim ** -0.5
    fused = c.head_dim == 128 and (2 * c.hidden) % 256 == 0
    # KV-cache append folded into the q|k|v GEMM's RoPE epilogue (7 launches per layer instead of 8).  Folding the two
    # RMSNorms into the GEMMs as well (5 launches) measured SLOWER on B200 -- 4.57 vs 3.58 ms/token: the per-fragment
    # normalisation sits between the weight-streaming loads of a kernel that lives on memory-level parallelism
    # (profiles/r2_decode_fusion.md).
    fuse_step = fused and B <= 16 and c.hidden % 256 == 0 and _FUSED_DECODE
    for li, w in enumerate(self.layers):
        if fuse_step:
            h = kernels.rmsnorm(x, w['ln_in'], c.rms_eps)
            qkv = dense.decode_gemm(h, w['wqkv'], rope=(cos, sin, 2 * c.hidden, pos, pos_dev), kv=(cache.k[li], cache.v[li]))
            a = kernels.decode_attention(qkv, cache.k[li], cache.v[li], B, c.n_heads, c.head_dim, kv_len, scale, pos_dev)
            x = dense.linear(a, w['wo'], residual=x)
            h = kernels.rmsnorm(x, w['ln_post'], c.rms_eps)
            f = dense.decode_gemm(h, w['wgu'], act='swiglu')
            x = dense.linear(f, w['wdown'], residual=x)
            continue
        h = kernels.rmsnorm(x, w['ln_in'], c.rms_eps)
        if fused:
            qkv = dense.qkv_rope(h, w['wqkv'], cos, sin, 1, 2 * c.hidden, pos0=pos, pos_dev=pos_dev)
        else:
            if pos_dev is not None:
                raise NotImplementedError('graph decode needs the fused-RoPE QKV GEMM (head_dim 128)')
            qkv = dense.linear(h, w['wqkv'])
            kernels.rope_inplace(qkv, cos[pos:pos + 1].contiguous(), sin[pos:pos + 1].contiguous(), 1, 2 * c.n_heads, c.head_dim)
        kernels.kv_append(qkv, cache.k[li], cache.v[li], B, 1, pos, pos_dev)
        a = kernels.decode_attention(qkv, cache.k[li], cache.v[li], B, c.n_heads, c.head_dim, kv_len, scale, pos_dev)
        x = dense.linear(a, w['wo'], residual=x)
        h = kernels.rmsnorm(x, w['ln_post'], c.rms_eps)
        f = dense.linear(h, w['wgu'], act='swiglu')
        x = dense.linear(f, w['wdown'], residual=x)
    cache.length = pos + 1
    x = kernels.rmsnorm(x, self.norm_w, c.rms_eps)
    buf = torch.empty((B, self.vocab_pad), dtype=self.dt, device=self.dev)
    dense.linear(x, self.lm_head, out=buf[:, :c.vocab])
    return buf[:, None, :c.vocab]


@torch.no_grad()
def _generate(self, input_ids, images, bboxes, max_new_tokens=32, do_sample=False, temperature=1.0,
              stopping_criteria=None, eos_token_id=None, generator=None, use_graph=True):
    """Prefill + greedy / temperature-sampled decode (gpt4roi/app.py:286-300 calls
    model.generate(input_ids, images=..., do_sample=True, temperature=0.2, max_new_tokens=1024,
    stopping_criteria=[...]) with the boxes bound to forward).  Returns ids [B, L + new]."""
    B, L = input_ids.shape
    cache = KVCache(self.cfg, B, L + max_new_tokens, self.dev)
    plan = self.plan_boxes(bboxes)
    ids = input_ids.to(self.dev)
    logits = self.forward_device(ids, images.to(self.dev, self.dt), plan, validate=True, last_only=True, cache=cache)
    out = ids
    stepper = None
    if use_graph and max_new_tokens > 4 and self.cfg.head_dim == 128:
        stepper = GraphedDecode(self, cache)
    for step in range(max_new_tokens):
        last = logits[:, -1].float()
        if do_sample and temperature > 0:
            nxt = torch.multinomial(torch.softmax(last / temperature, -1), 1, generator=generator)
        else:
            nxt = last.argmax(-1, keepdim=True)
        out = torch.cat([out, nxt], 1)
        if eos_token_id is not None and bool((nxt == eos_token_id).all()):
            break
        if stopping_criteria is not None and any(bool(torch.as_tensor(sc(out, last)).all()) for sc in stopping_criteria):
            break
        if step + 1 < max_new_tokens:
            logits = stepper.step(nxt) if stepper is not None else self.decode_step(nxt, cache)
    return out


class GraphedDecode:
    """CUDA-graph replay of one decode step: ~260 launches become one.  The current length lives in a
    device int32 that the QKV-RoPE epilogue, kv_append and decode_attention read; `step` bumps it."""

    def __init__(self, engine, cache):
        self.eng, self.cache = engine, cache
        dev = engine.dev
        self.ids = torch.zeros((cache.B, 1), dtype=torch.int64, device=dev)
        self.pos = torch.tensor([cache.length], dtype=torch.int32, device=dev)
        start = cache.length
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):  # warm-up (writes slot `start`, overwritten by the first real step)
                engine.decode_step(self.ids, cache, self.pos)
                cache.length = start
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.logits = engine.decode_step(self.ids, cache, self.pos)
        cache.length = start

    def step(self, token_ids):
        if self.cache.length + 1 > self.cache.max_len:
            raise RuntimeError('KV cache is full (%d)' % self.cache.max_len)
        self.ids.copy_(token_ids, non_blocking=True)
        self.graph.replay()
        self.pos.add_(1)
        self.cache.length += 1
        return self.logits


PrefillEngine.decode_step = _decode_step
PrefillEngine.generate = _generate


class GraphedPrefill:
    """CUDA-graph replay of PrefillEngine.forward_device for a fixed (B, L, box counts) shape:
    the ~1500 kernel launches of one prefill become one graph launch.  Inputs are staged through
    static device buffers; `run` accepts (pinned) host tensors."""

    def __init__(self, engine, input_ids, images, bboxes, last_only=True):
        self.eng = engine
        dev = engine.dev
        self.ids = input_ids.to(dev).clone()
        self.images = images.to(dev, engine.dt).clone()
        self.plan = engine.plan_boxes(bboxes)
        self.counts = None if bboxes is None else [0 if b is None else int(b.shape[0]) for b in bboxes]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            engine.forward_device(self.ids, self.images, self.plan, validate=True, last_only=last_only)  # warm-up + validation
            engine.forward_device(self.ids, self.images, self.plan, validate=False, last_only=last_only)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = engine.forward_device(self.ids, self.images, self.plan, validate=False, last_only=last_only)

    def run(self, input_ids, images, bboxes):
        self.ids.copy_(input_ids, non_blocking=True)
        self.images.copy_(images, non_blocking=True)
        if self.plan is not None and self.plan['K'] > 0:
            counts = [0 if b is None else int(b.shape[0]) for b in bboxes]
            if counts != self.counts:
                raise ValueError('box counts differ from the captured shape')
            off = 0
            for b in bboxes:
                if b is not None and b.shape[0]:
                    self.plan['boxes'][off:off + b.shape[0]].copy_(b, non_blocking=True)
                    off += b.shape[0]
        self.graph.replay()
        return self.out


def random_state_dicts(cfg, device, seed=0, dtype=BF16):
    """Seeded random-init weights with the reference's parameter names and init scales
    (conv normal(0,0.01): layers.py:146-150,275-278; GN (1,0); HF defaults elsewhere).
    Used by bench.py / tests: no checkpoints are available offline."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def rn(*shape, std=0.02):
        return (torch.randn(*shape, generator=g, device=device, dtype=torch.float32) * std).to(dtype)

    C, D = cfg.vit_hidden, cfg.hidden
    vit = {'vision_model.embeddings.class_embedding': rn(C),
           'vision_model.embeddings.patch_embedding.weight': rn(C, 3, cfg.patch_size, cfg.patch_size),
           'vision_model.embeddings.position_embedding.weight': rn(cfg.num_patches + 1, C),
           'vision_model.pre_layrnorm.weight': torch.ones(C, device=device, dtype=dtype),
           'vision_model.pre_layrnorm.bias': torch.zeros(C, device=device, dtype=dtype)}
    for i in range(cfg.vit_layers):
        q = 'vision_model.encoder.layers.%d.' % i
        for n in ('q', 'k', 'v', 'out'):
            vit[q + 'self_attn.%s_proj.weight' % n] = rn(C, C)
            vit[q + 'self_attn.%s_proj.bias' % n] = rn(C)
        for n in ('layer_norm1', 'layer_norm2'):
            vit[q + n + '.weight'] = torch.ones(C, device=device, dtype=dtype)
            vit[q + n + '.bias'] = torch.zeros(C, device=device, dtype=dtype)
        vit[q + 'mlp.fc1.weight'], vit[q + 'mlp.fc1.bias'] = rn(cfg.vit_mlp, C), rn(cfg.vit_mlp)
        vit[q + 'mlp.fc2.weight'], vit[q + 'mlp.fc2.bias'] = rn(C, cfg.vit_mlp), rn(C)
    sd = {'model.embed_tokens.weight': rn(cfg.vocab, D), 'lm_head.weight': rn(cfg.vocab, D),
          'model.norm.weight': torch.ones(D, device=device, dtype=dtype),
          'model.mm_projector.weight': rn(D, C), 'model.mm_projector.bias': rn(D)}
    for i in range(cfg.n_layers):
        q = 'model.layers.%d.' % i
        for n in ('q', 'k', 'v', 'o'):
            sd[q + 'self_attn.%s_proj.weight' % n] = rn(D, D)
        sd[q + 'mlp.gate_proj.weight'], sd[q + 'mlp.up_proj.weight'] = rn(cfg.mlp, D), rn(cfg.mlp, D)
        sd[q + 'mlp.down_proj.weight'] = rn(D, cfg.mlp)
        sd[q + 'input_layernorm.weight'] = torch.ones(D, device=device, dtype=dtype)
        sd[q + 'post_attention_layernorm.weight'] = torch.ones(D, device=device, dtype=dtype)
    S = cfg.spi_dim
    p = 'model.spi_module.'
    for l in range(cfg.num_levels):
        sd[p + 'mlvl_fuse.input_conv.%d.weight' % l] = rn(S, S + 2, 1, 1, std=0.01)
        sd[p + 'mlvl_fuse.input_conv.%d.bias' % l] = torch.zeros(S, device=device, dtype=dtype)
        sd[p + 'roi_align.pconvs.%d.weight' % l] = rn(S, S, 3, 3, std=0.01)
        sd[p + 'roi_align.pconvs.%d.bias' % l] = torch.zeros(S, device=device, dtype=dtype)
    for r in range(5):
        sd[p + 'mlvl_fuse.fuse_convs.%d.conv.weight' % r] = rn(S, S, 3, 3, std=0.01)
        sd[p + 'mlvl_fuse.fuse_convs.%d.gn.weight' % r] = torch.ones(S, device=device, dtype=dtype)
        sd[p + 'mlvl_fuse.fuse_convs.%d.gn.bias' % r] = torch.zeros(S, device=device, dtype=dtype)
    q = p + 'roi_align.'
    sd[q + 'pos_embedd.0.weight'], sd[q + 'pos_embedd.0.bias'] = rn(256, 4, std=0.5), rn(256, std=0.1)
    sd[q + 'pos_embedd.2.weight'] = torch.ones(256, device=device, dtype=dtype)
    sd[q + 'pos_embedd.2.bias'] = torch.zeros(256, device=device, dtype=dtype)
    sd[q + 'pos_embedd.3.weight'], sd[q + 'pos_embedd.3.bias'] = rn(1024, 256, std=0.06), rn(1024, std=0.06)
    sd[q + 'pos_embedd.5.weight'] = torch.ones(1024, device=device, dtype=dtype)
    sd[q + 'pos_embedd.5.bias'] = torch.zeros(1024, device=device, dtype=dtype)
    sd[q + 'updims.weight'], sd[q + 'updims.bias'] = rn(D, 1024, std=0.03), rn(D, std=0.03)
    R = cfg.roi_out
    sd[q + 'flatten_linear.weight'] = rn(1024, S * R * R, std=0.002)
    sd[q + 'flatten_linear.bias'] = rn(1024, std=0.002)
    return sd, vit
