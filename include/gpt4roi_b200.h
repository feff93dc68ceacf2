/*
 * gpt4roi_b200.h -- C ABI of libgpt4roi_b200.so (sm_100a).
 *
 * Drop-in boundary for the GPT4RoI region-token forward path.  Every entry
 * point takes raw DEVICE pointers, plain sizes and a cudaStream_t (as void*),
 * returns 0 on success or a negative G4R_E* code (message via
 * g4r_last_error()), allocates nothing that outlives the call, and never
 * synchronises the stream unless stated.  No torch types cross this boundary.
 *
 * Each declaration cites the reference interface it replaces; paths are
 * relative to /root/reference.
 */
#ifndef GPT4ROI_B200_H_
#define GPT4ROI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- enums (ints on the wire) ------------------------------------------- */
enum { G4R_F32 = 0, G4R_F16 = 1, G4R_BF16 = 2, G4R_F64 = 3 };       /* dtype   */
enum { G4R_NCHW = 0, G4R_NHWC = 1 };                                /* layout  */
enum { G4R_POOL_MAX = 0, G4R_POOL_AVG = 1 };  /* mmcv/ops/roi_align.py:77 */

enum {
  G4R_OK = 0,
  G4R_EINVAL = -1,   /* bad argument (message says which)                  */
  G4R_ECUDA = -2,    /* CUDA runtime / launch error                        */
  G4R_EUNSUPPORTED = -3,
  G4R_ENODEVICE = -4
};

#define G4R_MAX_LEVELS 4

/* Thread-local message for the last non-zero return on this thread. */
const char* g4r_last_error(void);
/* Library/ABI version (major*1000+minor) and the SM arch it was built for. */
int g4r_version(void);
int g4r_built_arch(void); /* 100 for sm_100a */
/* Keep n_sms SMs free of the persistent (one CTA per SM) tcgen05 GEMM kernels -- room for the CTAs of a collective
 * that runs beside the backward (the DDP gradient all-reduce of gpt4roi/train/train.py:698-712).  Returns the
 * previous reserve.  Process-wide; 0 (default) = the GEMMs use every SM. */
int g4r_set_sm_reserve(int n_sms);
/* Programmatic dependent launch for the kernels of the decode step behind generate() (llava/model/llava.py:263-283;
 * gpt4roi/app.py:293-300): while on != 0, the small-M GEMM, RMSNorm and single-query attention kernels are launched so
 * that each may start during its predecessor's tail, fetch its first WEIGHT block, and only then wait for the
 * predecessor.  Sound only for a launch sequence in which no kernel writes weights (the decode step); callers switch
 * it on around such a sequence and off again.  Returns the previous setting.  Process-wide; default off. */
int g4r_set_pdl(int on);

/* ---- RoIAlign: operator seam -------------------------------------------- */
/*
 * Replaces mmcv._ext.roi_align_forward
 *   mmcv-1.4.7/mmcv/ops/csrc/pytorch/pybind.cpp:611-615  (python binding)
 *   mmcv-1.4.7/mmcv/ops/csrc/pytorch/roi_align.cpp:25-32 (dispatch)
 *   mmcv-1.4.7/mmcv/ops/csrc/pytorch/cuda/roi_align_cuda.cu:5-30 (launcher)
 *   mmcv-1.4.7/mmcv/ops/csrc/common/cuda/roi_align_cuda_kernel.cuh:17-108
 * input  [N,C,H,W] (G4R_NCHW) or [N,H,W,C] (G4R_NHWC), contiguous, `dtype`
 * rois   [K,5] = (batch_idx, x1, y1, x2, y2), SAME dtype as input (reference
 *        contract, roi_align_cuda.cu:22)
 * output [K,C,PH,PW] (NCHW) or [K,PH,PW,C] (NHWC), `dtype`; fully overwritten
 * argmax_y/argmax_x: same shape as output for G4R_POOL_MAX, ignored for AVG.
 * Arithmetic: index/bin/weight math in fp32 (fp64 for G4R_F64) with the
 * reference's association and no FMA contraction; fp16/bf16 taps are widened
 * to fp32, accumulated in fp32 and rounded once on store.
 */
int g4r_roi_align_forward(const void* input, const void* rois, void* output,
                          void* argmax_y, void* argmax_x,
                          int N, int C, int H, int W, int K,
                          int pooled_height, int pooled_width,
                          float spatial_scale, int sampling_ratio,
                          int pool_mode, int aligned,
                          int dtype, int layout, void* stream);

/*
 * Same operator with a caller-provided scratch buffer: for the NCHW drop-in layout with enough RoIs
 * (g4r_roi_align_forward_workspace() > 0: avg pooling, fp32/fp16/bf16, C a multiple of the 16-byte vector and
 * >= 64, tap work >= twice the map size) the call runs as NCHW->NHWC transpose, the coalesced NHWC kernel, and
 * the transpose back -- three streaming passes instead of the reference layout's plane gather
 * (roi_align_cuda_kernel.cuh:17-108), bit-identical results.  With workspace == NULL, too small, or a
 * configuration the fast path does not cover, it is exactly g4r_roi_align_forward.  workspace: 256-byte aligned.
 */
size_t g4r_roi_align_forward_workspace(int N, int C, int H, int W, int K, int PH, int PW, int sampling_ratio,
                                       int pool_mode, int dtype, int layout);
int g4r_roi_align_forward_ws(const void* input, const void* rois, void* output, void* argmax_y, void* argmax_x,
                             int N, int C, int H, int W, int K, int PH, int PW, float spatial_scale,
                             int sampling_ratio, int pool_mode, int aligned, int dtype, int layout,
                             void* workspace, size_t workspace_bytes, void* stream);

/*
 * Replaces mmcv._ext.roi_align_backward
 *   pybind.cpp:616-620; roi_align.cpp:34-41; roi_align_cuda.cu:32-57;
 *   roi_align_cuda_kernel.cuh:111-210.
 * grad_output contiguous in `layout`; grad_input must be ZEROED by the caller
 * (mmcv/ops/roi_align.py:113) and is accumulated with atomics.
 */
int g4r_roi_align_backward(const void* grad_output, const void* rois,
                           const void* argmax_y, const void* argmax_x,
                           void* grad_input,
                           int N, int C, int H, int W, int K,
                           int pooled_height, int pooled_width,
                           float spatial_scale, int sampling_ratio,
                           int pool_mode, int aligned,
                           int dtype, int layout, void* stream);

/*
 * Fused multi-level RoIAlign (one launch for all levels and all RoIs).
 * Replaces the per-level loop of gpt4roi/models/layers.py:307-313, i.e.
 * 4x { feats[i].to(float32) -> mmcv RoIAlign -> .to(ori_dtype) }.
 * maps[l]   : NHWC [N,H[l],W[l],C], dtype in_dtype (F32, F16 or BF16)
 * scales[l] : spatial_scale of level l as a C float (1/stride)
 * rois      : fp32 [K,5] in input-pixel units (layers.py:294-302)
 * output    : [n_levels,K,PH,PW,C] NHWC, dtype out_dtype; avg pooling only
 * Optional per-(image,channel) affine+ReLU applied to every tap BEFORE the
 * bilinear weights (fuses the last GroupNorm+ReLU of the fuse stack,
 * layers.py:178 / mmcv cnn/bricks/conv_module.py:196-208): for level l, tap
 * value v -> max(v*gn_scale[l][n*C+c] + gn_shift[l][n*C+c], 0); pass NULL
 * arrays to disable.  fp32 [N,C] each.
 */
int g4r_roi_align_mlvl_forward(const void* const* maps, const int* H, const int* W,
                               const float* scales, int n_levels,
                               const float* rois, void* output,
                               int N, int C, int K,
                               int pooled_height, int pooled_width,
                               int sampling_ratio, int aligned,
                               int in_dtype, int out_dtype,
                               const float* const* gn_scale,
                               const float* const* gn_shift,
                               void* stream);

/* Gradient of the above w.r.t. the maps (fp32 NHWC grad maps, pre-zeroed). */
int g4r_roi_align_mlvl_backward(const void* grad_output, const int* H, const int* W,
                                const float* scales, int n_levels,
                                const float* rois, float* const* grad_maps,
                                int N, int C, int K,
                                int pooled_height, int pooled_width,
                                int sampling_ratio, int aligned,
                                int grad_dtype, void* stream);

/* ---- region-token splice: model seam ------------------------------------- */
/*
 * Replaces the per-sample python loop of gpt4roi/models/spi_llava.py:99-196
 * (use_im_start_end branch) including `embed_tokens(input_ids)` (:44-45):
 *   row t of sample b <- embed_table[ids[b,t]]             (default)
 *                     <- image_rows[b, t-(s+1)]            (s = <im_start> pos, s<t<=s+P)
 *                     <- region_rows[region_offsets[b]+j]  (t is the j-th <bbox> of sample b)
 * All rows are `D` elements of a 16-bit type (bf16/fp16); data is moved, never
 * re-rounded.  status[b] (int32, device) receives 0 or the reference's error:
 *   1 = #<im_start> != #<im_end>            (spi_llava.py:114-118)
 *   2 = <im_end> not at s+P+1               (spi_llava.py:124-128)
 *   3 = #<bbox> != K_b                      (shape error at spi_llava.py:154)
 *   4 = more than one <im_start> (unsupported; see DESIGN.md)
 *   5 = <im_patch> present but no <im_start> (reference: unbound variable)
 *   6 = token id outside [0,V) (reference: embedding index error)
 * region_rows/region_offsets may be NULL (bboxes=None, spi_llava.py:83-87): then
 * a <bbox> token present in a multimodal sample is error 3 (assert :158-161).
 * plan: int32 scratch [B,L] (device).
 */
int g4r_splice_region_tokens(const int64_t* input_ids, const void* embed_table,
                             const void* image_rows, const void* region_rows,
                             const int32_t* region_offsets, void* out,
                             int32_t* plan, int32_t* status,
                             int B, int L, int P, int D, int V,
                             int64_t im_patch_token, int64_t im_start_token,
                             int64_t im_end_token, int64_t bbox_token,
                             void* stream);

/* ---- dense contractions on tcgen05 tensor cores ---------------------------- */
enum { G4R_ACT_NONE = 0, G4R_ACT_RELU = 1, G4R_ACT_QUICK_GELU = 2, G4R_ACT_SWIGLU = 3 };

/*
 * D[M,N] = epilogue(A[M,K] . B[N,K]^T): bf16 operands (both K-major, i.e. B is an
 * nn.Linear weight [out,in]), fp32 accumulation in TMEM, TMA-fed, persistent.
 * Replaces the cuBLAS calls behind torch.nn.Linear at
 *   gpt4roi/models/layers.py:260-270,326-329  (pos_embedd, flatten_linear, updims)
 *   llava/model/llava.py:52,76 / gpt4roi/models/spi_llava.py:89-97 (mm_projector)
 *   llava/model/llava.py:195,235-236 (lm_head)
 *   transformers CLIP / LLaMA q,k,v,o,fc1,fc2,gate,up,down projections (third party)
 * epilogue: (+bias[N]) -> act -> (+residual[M,N] bf16) -> store bf16 (or fp32 if out_f32).
 *   G4R_ACT_SWIGLU: B rows interleaved (2j = gate_j, 2j+1 = up_j); D is [M,N/2] = silu(g)*u.
 *   k_splits > 1: D is an fp32 buffer [k_splits][M][ldd]; split s writes slab s (no atomics, no
 *   bias/act/residual); the consumer sums the slabs in a fixed order (bitwise reproducible).
 * lda/ldb/ldd/ldr are row strides in elements; lda, ldb multiples of 8.
 */
int g4r_gemm_bf16(const void* A, long long lda, const void* B, long long ldb,
                  void* D, long long ldd, int M, int N, int K,
                  const void* bias, int bias_f32,
                  const void* residual, long long ldr,
                  int act, int out_f32, int k_splits, void* stream);

/* Extended form: residual may be fp32 (residual_f32=1; CLIP's residual stream is fp32 under autocast)
 * and the branch (acc + bias, act) can be rounded to bf16 before the residual add (bias_round_bf16=1),
 * reproducing "bf16 linear output + fp32 stream". */
int g4r_gemm_bf16_ex(const void* A, long long lda, const void* B, long long ldb,
                     void* D, long long ldd, int M, int N, int K,
                     const void* bias, int bias_f32,
                     const void* residual, long long ldr, int residual_f32, int bias_round_bf16,
                     int act, int out_f32, int k_splits, void* stream);

/* Backward-pass GEMM with operand transposes done in the tensor-core descriptors:
 *   D[M,N] = op(A) . op(B)^T ;  a_mn=0: A [M,K] K-contiguous, a_mn=1: A stored [K,M] M-contiguous (lda >= M)
 *                               b_mn=0: B [N,K] K-contiguous, b_mn=1: B stored [K,N] N-contiguous (ldb >= N)
 * For y = x.W^T (torch.nn.functional.linear; every Linear of the LLaMA stack the stage-2 step trains,
 * gpt4roi/train/train.py:698-712 + llava_trainer.py:59-144):
 *   grad_x = grad_y . W      -> g4r_gemm_bf16_t(grad_y, ., 0, W, ., 1, grad_x, ., M, K_in, N_out, ...)
 *   grad_W = grad_y^T . x    -> g4r_gemm_bf16_t(grad_y, ., 1, x, ., 1, grad_W, ., N_out, K_in, M, ...)
 * bf16 operands, fp32 accumulation, bf16 or fp32 (out_f32) output. */
int g4r_gemm_bf16_t(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn,
                    void* D, long long ldd, int M, int N, int K, int out_f32, void* stream);

/* LLaMA QKV projection with apply_rotary_pos_emb fused into the epilogue (transformers
 * modeling_llama.py:138-168): D[M,N] = A.B^T; columns [0,rope_cols) are 128-dim heads rotated with the
 * bf16 cos/sin tables [>= pos0+L, 128] at position pos0 + (row % L) (pos0 > 0: decode steps);
 * rounding points as in the reference's bf16 ops. */
int g4r_gemm_qkv_rope_bf16(const void* A, long long lda, const void* B, long long ldb,
                           void* D, long long ldd, int M, int N, int K,
                           const void* rope_cos, const void* rope_sin, int rope_cols, int L, int pos0,
                           const int* pos0_dev /* device int32 overriding pos0 (CUDA-graph decode) or NULL */,
                           void* stream);

/* ---- decode loop (KV cache) -------------------------------------------------- */
/* Decode-step GEMM (M = batch <= 16 new tokens, one per sample; the LLaMA stack behind generate(), llava.py:263-283,
 * spi_llava.py:47-48), weight-streaming, with the neighbouring memory-bound steps folded in:
 *   out = [RoPE | SwiGLU | + residual]( x . W^T )
 * rope_cos/sin (optional): rotate columns [0, rope_cols) at position pos0 / *pos_dev;
 * kcache / vcache (optional, with RoPE on the fused q|k|v projection, N == 3 * cache_hd): the rotated key and the value
 * columns of sample m are also written to cache[m, pos, :] -- replaces g4r_gemm_qkv_rope_bf16 + g4r_kv_append_bf16
 * (2 launches) of the unfused step. */
int g4r_decode_gemm_bf16(const void* x, long long ldx, const void* W, long long ldw, void* out, long long ldo, int M,
                         int N, int K, int act, const void* residual, long long ldr,
                         const void* rope_cos, const void* rope_sin, int rope_cols, int pos0, const int* pos_dev,
                         void* kcache, void* vcache, int cache_lmax, int cache_hd, void* stream);

/* Append the k and v parts of packed rows [B*Ln, (q|k|v) of width HD each] to the caches
 * [B, Lmax, HD] at positions pos0..pos0+Ln-1 (prefill: pos0=0, Ln=L; decode: Ln=1).  */
int g4r_kv_append_bf16(const void* qkv, long long ld, void* kcache, void* vcache,
                       int B, int Ln, int pos0, const int* pos_dev /* overrides pos0 when non-NULL */,
                       int Lmax, int HD, void* stream);
/* One new query per sample against the first kv_len cached positions: out[b,h,:] =
 * softmax(q.K^T*scale) V.  Replaces the decode-step attention of transformers' LlamaAttention with a
 * DynamicCache (generate() in gpt4roi/app.py:293-300; vision branch skipped, spi_llava.py:47-48). */
int g4r_decode_attention_bf16(const void* q, long long ldq, const void* kcache, const void* vcache,
                              void* out, long long ldo, int B, int H, int head_dim, int kv_len,
                              const int* pos_dev /* kv_len = *pos_dev + 1 when non-NULL; kv_len then sizes smem */,
                              int Lmax, float scale, void* stream);

/*
 * NHWC convolution as an implicit GEMM (stride 1, pad (ksize-1)/2, ksize 1 or 3):
 *   Y[n,y,x,co] = act( sum_{ky,kx,ci} X[n,y+ky-1,x+kx-1,ci] * Wt[co,(ky*ks+kx)*Cin+ci] + bias[co] )
 * X bf16 [n_img,H,W,Cin]; Wt bf16 [Cout, ks*ks*Cin] (torch [Cout,Cin,kh,kw] permuted to
 * [Cout,kh,kw,Cin] once at load time); Y bf16 [n_img,H,W,Cout].  The A operand is fetched
 * with 4-D TMA boxes shifted by the filter tap; TMA's out-of-bounds zero fill is the padding.
 * Replaces cuDNN behind nn.Conv2d at gpt4roi/models/layers.py:129-144,191,178 (input_conv,
 * fuse_convs[i].conv) and :257-259,320-325 (pconvs).
 * levels > 1 sums `levels` convolutions in one contraction (K concatenated): X is
 * [levels*n_img,H,W,Cin] (level-major), Wt [Cout, levels*ks*ks*Cin]; this is
 * sum_l pconvs[l](roi_feats[l]) of layers.py:320-325 as ONE GEMM.
 * gn_stats (optional, fp32 [n_img, g4r_conv_gn_slots(H,W), gn_groups, 2]): per-(tile,warp) partial
 * sum / sum of squares of the bf16-rounded output per (image, 16-channel group) -- the statistics
 * GroupNorm(64) needs (mmcv cnn/bricks/conv_module.py:196-208) -- written with plain stores
 * (reproducible) and summed in a fixed order by g4r_gn_finalize; no extra pass over Y.
 */
int g4r_conv_gn_slots(int H, int W);
int g4r_conv_nhwc_bf16(const void* X, const void* Wt, void* Y,
                       int n_img, int H, int W, int Cin, int Cout, int ksize, int levels,
                       const void* bias, int bias_f32, int act,
                       float* gn_stats, int gn_groups, void* stream);

/* ---- fused attention ------------------------------------------------------- */
/*
 * out[b,i,h,:] = softmax_j( (q_i.k_j) * scale [+ causal mask] ) . v_j   (scores kept in fp32)
 * q/k/v: bf16, element (b, token, head h, d) at  base + b*bs + token*ld + h*head_dim + d
 * (so the packed [B,L,(q|k|v)] output of the QKV GEMM is read in place); out likewise with
 * ldo/bso.  head_dim 64 (CLIP-ViT-L/14) or 128 (LLaMA-7B).  Replaces transformers'
 * eager_attention_forward (modeling_clip.py / modeling_llama.py:199-222), third party to the
 * reference (pyproject.toml:19).
 */
int g4r_attention_bf16(const void* q, const void* k, const void* v, void* out,
                       long long ld, long long bs, long long ldo, long long bso,
                       int B, int H, int L, int head_dim, int causal, float scale,
                       const int* seqlens /* device int32 [B] or NULL: keys >= seqlens[b] are masked */,
                       void* stream);

/*
 * Same contract on the tcgen05 tensor cores (TMA-fed, S and O accumulators in TMEM, V consumed as an
 * MN-major operand); requires the packed layout bs == L*ld.  csrc/attention_tcgen05.cu.
 */
int g4r_attention_tc_bf16(const void* q, const void* k, const void* v, void* out,
                          long long ld, long long bs, long long ldo, long long bso,
                          int B, int H, int L, int head_dim, int causal, float scale,
                          const int* seqlens, void* stream);

/* ---- HBM-bound glue (csrc/elementwise.cu); bf16 rows, fp32 math ------------- */
/* nn.LayerNorm over the last dim (CLIP layer norms; gpt4roi/models/layers.py:263,266). */
int g4r_layernorm_bf16(const void* x, long long ldx, const void* w, const void* b,
                       void* out, long long ldo, int M, int D, float eps, void* stream);
/* LayerNorm with fp32 or bf16 input/output rows (x_f32 / out_f32).  Under autocast the reference's
 * nn.LayerNorm returns fp32, so CLIP's residual stream is fp32: pre_layrnorm is bf16->fp32, layer_norm1/2
 * are fp32->bf16 (their output is cast to bf16 by the following autocast Linear). */
int g4r_layernorm_ex(const void* x, long long ldx, int x_f32, const void* w, const void* b,
                     void* out, long long ldo, int out_f32, int M, int D, float eps, void* stream);
/* fp32 rows [B][rows_per_batch][D] (row stride ld, batch stride bst) -> dense bf16 [B*rows_per_batch, D]
 * (the autocast cast at mm_projector's input, spi_llava.py:89-93, skipping the CLS row). */
int g4r_cast_f32_bf16(const void* x, long long ld, long long bst, void* out,
                      int B, int rows_per_batch, int D, void* stream);
/* LlamaRMSNorm: w * bf16(x * rsqrt(mean(x^2)+eps))  (transformers modeling_llama.py:53-67). */
int g4r_rmsnorm_bf16(const void* x, long long ldx, const void* w,
                     void* out, long long ldo, int M, int D, float eps, void* stream);
/* Same for an fp32 (x_f32=1) or bf16 residual stream; bf16 output rows (the operand of the next GEMM).  With an
 * fp32 stream the normalised value is not rounded before the weight multiply, exactly LlamaRMSNorm on an fp32
 * input (modeling_llama.py:53-67: `self.weight * hidden_states.to(input_dtype)`) -- the reference's residual stream
 * is fp32 whenever its parameters are (training under autocast), bf16 when the model was cast to bf16. */
int g4r_rmsnorm_ex(const void* x, long long ldx, int x_f32, const void* w, void* out, long long ldo, int M, int D,
                   float eps, void* stream);
/* apply_rotary_pos_emb in place on the first n_heads_qk heads of each packed row
 * (modeling_llama.py:138-168); cos/sin bf16 [L, head_dim]; position = row % L. */
int g4r_rope_inplace_bf16(void* qkv, long long ld, const void* cos_t, const void* sin_t,
                          int rows, int L, int n_heads_qk, int head_dim, void* stream);
/* CLIP patchify (im2col of the stride-14 patch_embedding conv, modeling_clip.py:148-154):
 * img bf16 [B,3,S,S] -> out bf16 [B*(S/ps)^2, Kpad], column (c*ps+ky)*ps+kx, zero padded. */
int g4r_patchify_bf16(const void* img, void* out, int B, int S, int ps, int Kpad, void* stream);
/* [CLS | patches] + position_embedding  (modeling_clip.py:209-216). */
int g4r_vit_embed_bf16(const void* patch, const void* cls, const void* pos, void* out,
                       int B, int P, int D, void* stream);
/* ViT tokens [B,G*G,C] (row stride ldt, batch stride bst) -> bilinear align_corners resize to
 * [B,Ho,Ho,Cpad] NHWC with the two coordinate channels appended and zero padding
 * (gpt4roi/models/layers.py:219-232 + :117-126,185-188). */
int g4r_upsample_tokens_coords_bf16(const void* tok, long long ldt, long long bst, void* out,
                                    int B, int G, int Ho, int C, int Cpad, void* stream);
/* same with fp32 tokens (CLIP hidden states are fp32 under autocast) */
int g4r_upsample_tokens_coords_f32(const void* tok, long long ldt, long long bst, void* out,
                                   int B, int G, int Ho, int C, int Cpad, void* stream);
/* One level of MLVLFuseModule._single_shuffle (layers.py:152-180): out = [own[:, :C/2] |
 * resize(top[:, 3C/4:]) | resize(down[:, C/2:3C/4])]; optional per-(image,channel) scale/shift
 * (fp32 [B,C]) apply the previous round's GroupNorm+ReLU to every tap first. */
int g4r_fuse_gather_bf16(const void* own, const float* own_sc, const float* own_sh, int H,
                         const void* top, const float* top_sc, const float* top_sh, int Ht,
                         const void* down, const float* down_sc, const float* down_sh, int Hd,
                         void* out, int B, int C, void* stream);
/* GroupNorm statistics -> per-(image,channel) scale/shift (torch.nn.GroupNorm semantics). */
int g4r_gn_finalize(const float* stats, const void* gamma, const void* beta,
                    float* scale, float* shift, int B, int C, int groups, int slots,
                    float count, float eps, void* stream);
/* pos_embedd MLP of MlvlRoIExtractor (layers.py:260-267,285): boxes fp32 [K,4] -> fp32 [K,1024]. */
int g4r_pos_embed_mlp(const float* boxes, const void* w0, const void* b0, const void* g2,
                      const void* be2, const void* w3, const void* b3, const void* g5,
                      const void* be5, float* out, int K, float eps, void* stream);
/* out = bf16( bf16(sum_s acc[s] + bias) + pos )  (layers.py:327-328). acc fp32 [splits,K,D]
 * (split-K slabs of flatten_linear), pos fp32 [K,D]. */
int g4r_add_bias_pos_cast(const float* acc, int splits, const void* bias, const float* pos, void* out,
                          int K, int D, void* stream);

/* ---- training step (SURVEY.md 8(a) row 14; gpt4roi/train/train.py:698-712 + HF Trainer) ----------------
 * Cross entropy of llava/model/llava.py:238-249 (CrossEntropyLoss(): mean over targets != -100) on rows of
 * bf16 logits [M,V]; `targets` are the already shifted labels (labels[..., 1:], last position -100).
 * Writes row_lse[M], row_loss[M], loss_count[2] = {mean loss, #valid rows} and, if dlogits != NULL,
 * dlogits = (softmax - onehot) * grad_scale / count (bf16, a separate buffer).  No atomics. */
int g4r_cross_entropy_bf16(const void* logits, long long ld, const long long* targets, int M, int V,
                           float* row_lse, float* row_loss, float* loss_count, void* dlogits, long long ldd,
                           float grad_scale, void* stream);

/* LlamaRMSNorm backward (transformers modeling_llama.py LlamaRMSNorm.forward): dx bf16 [M,D], dw fp32 [D].
 * dw_slabs: fp32 scratch [g4r_rmsnorm_bwd_slabs(M)][D] (per-CTA partial sums, reduced in fixed order). */
int g4r_rmsnorm_bwd_slabs(int M);
int g4r_rmsnorm_bwd_bf16(const void* x, long long ldx, const void* w, const void* dy, long long ldy,
                         const void* dres /* optional bf16 [M,D]: added to dx (gradient of the residual branch) */,
                         long long ldr, void* dx, long long ldd, float* dw, float* dw_slabs, int M, int D, float eps,
                         void* stream);

/* SwiGLU on an interleaved gate/up buffer gu [M,2F] (col 2j gate_j, 2j+1 up_j): f = silu(g)*u [M,F], and its
 * backward dgu [M,2F] from df [M,F] (transformers LlamaMLP.forward). */
int g4r_swiglu_fwd_bf16(const void* gu, long long ldg, void* f, long long ldf, long long M, int F, void* stream);
int g4r_swiglu_bwd_bf16(const void* gu, long long ldg, const void* df, long long ldf, void* dgu, long long ldd,
                        long long M, int F, void* stream);

/* Causal attention for training: forward on the tcgen05 / TMEM attention kernel that also writes lse[B,H,L] (fp32
 * log-sum-exp of the scaled scores; q, k, v must be one packed [B*L, width] buffer, bs == L*ld), and the backward
 * (autograd of transformers modeling_llama.py:199-222 eager attention): packed dQ|dK|dV rows from q,k,v (after
 * RoPE), the forward output `out`, `dout` and `lse`.  delta: fp32 scratch [B,H,L].
 * q/k/v: row stride ld, batch stride bs (elements); out/dout: ldo, bso; dq/dk/dv: ldg, bsg.  No atomics. */
int g4r_attention_tc_lse_bf16(const void* q, const void* k, const void* v, void* out, long long ld, long long bs,
                              long long ldo, long long bso, int B, int H, int L, int head_dim, int causal, float scale,
                              float* lse, void* stream);
int g4r_attention_bwd_bf16(const void* q, const void* k, const void* v, const void* out, const void* dout,
                           const float* lse, float* delta, void* dq, void* dk, void* dv, long long ld,
                           long long bs, long long ldo, long long bso, long long ldg, long long bsg, int B,
                           int H, int L, int head_dim, int causal, float scale, void* stream);

/* Backward of the splice (spi_llava.py:99-196): rows of d(inputs_embeds) [B*L, D] (16-bit) are copied back to
 * d_image [B*P, D] and d_region [K, D] following the forward's `plan` (either may be NULL to skip it).
 * g4r_embed_grad_rows accumulates the rows that came from the embedding table into a dense fp32 gradient
 * [V, D] (zeroed by the caller): `ids[n_unique]` are the distinct token ids, `order[seg[u] .. seg[u+1])` the
 * row indices (b*L + t) of id u.  One CTA per id, fixed summation order, no atomics. */
int g4r_splice_backward(const int32_t* plan, const void* d_out, void* d_image, void* d_region, int B, int L,
                        int P, int D, void* stream);
int g4r_embed_grad_rows(const void* d_out, const int32_t* order, const int32_t* seg, const int32_t* ids,
                        int n_unique, float* grad, int D, void* stream);

/* Column sums of a bf16 matrix [M,N] into fp32 out[N] (bias gradients of nn.Linear / Conv2d).
 * slabs: fp32 scratch [g4r_colsum_slabs(M)][N]. */
int g4r_colsum_slabs(int M);
int g4r_colsum_bf16(const void* x, long long ld, int M, int N, float* out, float* slabs, void* stream);

/* Backward of a 3x3 / stride 1 / pad 1 NHWC convolution (mmcv ConvModule of MLVLFuseModule, layers.py:133-145, and
 * the pconvs of MlvlRoIExtractor, layers.py:262-268):
 *   grad_x = g4r_conv_nhwc_bf16(grad_z, Wf) with Wf = g4r_conv_weight_flip_t_bf16(W): Wf[ci][ky][kx][co] = W[co][2-ky][2-kx][ci]
 *            (W rows `w_ld` elements apart, so one level of a stacked [Cout, L, 3, 3, Cin] weight works in place);
 *   grad_W = g4r_conv3x3_dw_bf16 on zero-padded copies (g4r_pad_nhwc_bf16: rows [guard | n*(H+2)*(W+2) | guard] x C,
 *            guard_rows >= W+3): one GEMM over all padded pixels, the nine taps being column blocks reached through an
 *            aliasing 4-D TMA tensor map.  x_pad_origin = x_pad + (guard_rows - (W+2) - 1) * Cin elements;
 *            dz_pad = first real row of the padded grad_z (skip its guard).  dW fp32 [Cout, 9*Cin]. */
int g4r_pad_nhwc_bf16(const void* x, void* out, int n, int H, int W, int C, int guard_rows, void* stream);
int g4r_conv_weight_flip_t_bf16(const void* w, long long w_ld, void* wf, int Cin, int Cout, void* stream);
int g4r_conv3x3_dw_bf16(const void* dz_pad, const void* x_pad_origin, float* dW, long long rows, int Wp,
                        int Cin, int Cout, int accumulate, void* stream);

/* GroupNorm(64) + ReLU backward of the fuse ConvModules (mmcv cnn/bricks/conv_module.py:196-208): z = raw conv output
 * (bf16 [B,HW,C], saved), dA = gradient w.r.t. relu(gn(z)) (fp32 when dA_f32, else bf16), scale/shift = g4r_gn_finalize
 * outputs, stats/slots/count/eps = the forward's GroupNorm statistics (mean / rstd are re-derived in the same order).
 * Writes dz (bf16) and dgamma / dbeta (fp32 [C]; accumulate != 0 adds: the four pyramid levels share one GN).
 * workspace: fp32 scratch of g4r_gn_relu_bwd_workspace(B, HW, C, groups) elements.  Fixed-order reductions only. */
long long g4r_gn_relu_bwd_workspace(int B, int HW, int C, int groups);
int g4r_gn_relu_bwd_bf16(const void* z, const void* dA, int dA_f32, const float* scale, const float* shift,
                         const float* stats, int slots, float count, float eps, const void* gamma, void* dz,
                         float* dgamma, float* dbeta, int accumulate, float* workspace, int B, int HW, int C,
                         int groups, void* stream);

/* Adjoint of g4r_fuse_gather_bf16 (MLVLFuseModule._single_shuffle, layers.py:152-180) for pyramid level m:
 * out fp32 [B,H,H,C] = gradient w.r.t. the previous round's activated maps of level m.  d_own = gradient of level
 * m's own conv input; dn0/dn1 = gradients of the conv inputs of the (<= 2) levels that read level m as their
 * `down` source, tp0/tp1 = of those that read it as their `top` source (NULL when absent), each bf16
 * [B,Hx,Hx,C].  Transposed bilinear resize evaluated as a gather (no atomics). */
int g4r_fuse_gather_bwd(const void* d_own, int H, const void* dn0, int Hdn0, const void* dn1, int Hdn1,
                        const void* tp0, int Htp0, const void* tp1, int Htp1, float* out, int B, int C, void* stream);

/* Backward of g4r_pos_embed_mlp (pos_embedd of MlvlRoIExtractor, layers.py:260-267): dout bf16 [K,1024] -> fp32
 * parameter gradients packed as [w0 256x4 | b0 256 | ln2.weight 256 | ln2.bias 256 | w3 1024x256 | b3 1024 |
 * ln5.weight 1024 | ln5.bias 1024] (g4r_pos_embed_mlp_grad_size() floats).  slabs: fp32 scratch [K][that size]. */
int g4r_pos_embed_mlp_grad_size(void);
int g4r_pos_embed_mlp_bwd(const float* boxes, const void* w0, const void* b0, const void* g2, const void* be2,
                          const void* w3, const void* b3, const void* g5, const void* dout, long long ldd,
                          float* grads, float* slabs, int K, float eps, void* stream);

/* ReLU backward from the saved output: out = y > 0 ? dy : 0 (bf16, n elements, n % 8 == 0). */
int g4r_relu_bwd_bf16(const void* dy, const void* y, void* out, long long n, void* stream);

/* ---- input pipeline (SURVEY.md 8(f2)) ------------------------------------------------------------------------
 * Image side of gpt4roi/datasets/coco_det.py:60-71 for a whole batch in one launch: Resize(S,S) [cv2 INTER_LINEAR on
 * uint8, integer-exact] -> RandomShift [zero-filled, per-image (shift_x, shift_y); NULL = none] -> horizontal
 * RandomFlip [per-image flag; NULL = none] -> Normalize(mean, std, to_rgb) [mmcv.imnormalize_ arithmetic] -> CHW.
 * src_packed: decoded uint8 HWC 3-channel images back to back (device); offsets[b] = byte offset of image b;
 * src_hw[b] = (h, w); out [B,3,S,S] fp32 (bit-identical to the reference pipeline) or bf16.  mean3 / std3: HOST float[3].
 * Replaces mmdet/datasets/pipelines/transforms.py:209-243 (Resize), :505-562 (RandomShift), :422-470 (RandomFlip),
 * Normalize / Pad / DefaultFormatBundle, which the reference runs per sample on CPU dataloader workers. */
int g4r_preprocess_images(const void* src_packed, const long long* offsets, const int* src_hw, const int* shift_xy,
                          const int* flip, void* out, int B, int S, const float* mean3, const float* std3, int to_rgb,
                          int out_dtype, void* stream);

/* Apply a pending GroupNorm affine + ReLU to an NHWC bf16 map: out = relu(z * scale[b,c] + shift[b,c]) with the
 * fp32 [B,C] scale / shift of g4r_gn_finalize.  The activated map is what MLVLFuseModule.forward returns
 * (gpt4roi/models/layers.py:182-195; mmcv ConvModule conv -> GN -> ReLU, conv_module.py:196-208); inside the fused
 * engine the affine stays folded into the consumer's taps, so only the module-level seam calls this. */
int g4r_affine_relu_nhwc_bf16(const void* z, const float* scale, const float* shift, void* out, int B,
                              long long pix_per_img, int C, void* stream);

/* torch.optim.AdamW step (HF Trainer optim="adamw_torch"; param groups llava_trainer.py:59-144): fp32 master
 * weights p and moments m, v; gradient bf16 (g_bf16=1) or fp32, multiplied by grad_scale (1/world, clip factor);
 * p_bf16 (optional) receives the bf16 copy used by the next forward.  step counts from 1. */
int g4r_adamw_step(float* p, const void* g, int g_bf16, float* m, float* v, void* p_bf16, long long n,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                   void* stream);
/* Same, with the gradient scale additionally multiplied by the device float *scale_dev (NULL = 1): the clip
 * coefficient of g4r_grad_clip_coef, so that clipping costs no host synchronisation. */
int g4r_adamw_step_ex(float* p, const void* g, int g_bf16, float* m, float* v, void* p_bf16, long long n,
                      float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                      const float* scale_dev, void* stream);

/* Global gradient-norm clip (HF Trainer max_grad_norm=1.0 -> torch.nn.utils.clip_grad_norm_, called between
 * backward and optimizer.step() by transformers Trainer.training_step; reference gpt4roi/train/train.py:698-712).
 * g4r_sumsq writes g4r_sumsq_slabs() per-CTA partial sums of squares of one gradient tensor (bf16 or fp32) to
 * slab; g4r_grad_clip_coef adds n_slabs partials in a fixed order and writes out2[0] = sqrt(sum) * pre_scale
 * (pre_scale = 1/world for summed, not averaged, DDP gradients) and out2[1] = min(1, max_norm / (out2[0] + 1e-6)). */
int g4r_sumsq_slabs(void);
int g4r_sumsq(const void* g, int g_bf16, long long n, float* slab, void* stream);
int g4r_grad_clip_coef(const float* slabs, long long n_slabs, float pre_scale, float max_norm, float* out2,
                       void* stream);

/* ---- fp16 twins of the inference entry points ---------------------------------------------
 * The demo serves the model in fp16 (gpt4roi/app.py:74-98,271: `model.half()`, `images.half()`, `bboxes.half()`).
 * Every entry point below has the signature, argument meaning and error behaviour of its `_bf16` namesake above,
 * with "bf16" read as "fp16" for every 16-bit tensor (activations, weights, norm / bias vectors, RoPE tables, KV
 * cache); fp32 arguments (statistics, scale / shift, split-K slabs, fp32 residual streams) are unchanged, and the
 * arithmetic is the same (fp32 accumulation, the same rounding points, tcgen05 kind::f16 with the F16 operand
 * format).  Built from the same sources with -DG4R_ACT_HALF (gpt4roi_b200/csrc/act_type.cuh).  RoIAlign and the
 * splice take a dtype argument / are 2-byte copies and need no twin; the training step is bf16 only
 * (train_stage*.sh --bf16 True). */
int g4r_gemm_f16(const void* A, long long lda, const void* B, long long ldb,
                  void* D, long long ldd, int M, int N, int K,
                  const void* bias, int bias_f32,
                  const void* residual, long long ldr,
                  int act, int out_f32, int k_splits, void* stream);
int g4r_gemm_f16_ex(const void* A, long long lda, const void* B, long long ldb,
                     void* D, long long ldd, int M, int N, int K,
                     const void* bias, int bias_f32,
                     const void* residual, long long ldr, int residual_f32, int bias_round_bf16,
                     int act, int out_f32, int k_splits, void* stream);
int g4r_gemm_qkv_rope_f16(const void* A, long long lda, const void* B, long long ldb,
                           void* D, long long ldd, int M, int N, int K,
                           const void* rope_cos, const void* rope_sin, int rope_cols, int L, int pos0,
                           const int* pos0_dev /* device int32 overriding pos0 (CUDA-graph decode) or NULL */,
                           void* stream);
int g4r_conv_nhwc_f16(const void* X, const void* Wt, void* Y,
                       int n_img, int H, int W, int Cin, int Cout, int ksize, int levels,
                       const void* bias, int bias_f32, int act,
                       float* gn_stats, int gn_groups, void* stream);
int g4r_attention_tc_f16(const void* q, const void* k, const void* v, void* out,
                          long long ld, long long bs, long long ldo, long long bso,
                          int B, int H, int L, int head_dim, int causal, float scale,
                          const int* seqlens, void* stream);
int g4r_attention_f16(const void* q, const void* k, const void* v, void* out,
                       long long ld, long long bs, long long ldo, long long bso,
                       int B, int H, int L, int head_dim, int causal, float scale,
                       const int* seqlens /* device int32 [B] or NULL: keys >= seqlens[b] are masked */,
                       void* stream);
int g4r_layernorm_f16(const void* x, long long ldx, const void* w, const void* b,
                       void* out, long long ldo, int M, int D, float eps, void* stream);
int g4r_rmsnorm_f16(const void* x, long long ldx, const void* w,
                     void* out, long long ldo, int M, int D, float eps, void* stream);
int g4r_rope_inplace_f16(void* qkv, long long ld, const void* cos_t, const void* sin_t,
                          int rows, int L, int n_heads_qk, int head_dim, void* stream);
int g4r_patchify_f16(const void* img, void* out, int B, int S, int ps, int Kpad, void* stream);
int g4r_vit_embed_f16(const void* patch, const void* cls, const void* pos, void* out,
                       int B, int P, int D, void* stream);
int g4r_upsample_tokens_coords_f16(const void* tok, long long ldt, long long bst, void* out,
                                    int B, int G, int Ho, int C, int Cpad, void* stream);
int g4r_upsample_tokens_coords_f32_f16(const void* tok, long long ldt, long long bst, void* out,
                                   int B, int G, int Ho, int C, int Cpad, void* stream);
int g4r_layernorm_ex_f16(const void* x, long long ldx, int x_f32, const void* w, const void* b,
                     void* out, long long ldo, int out_f32, int M, int D, float eps, void* stream);
int g4r_rmsnorm_ex_f16(const void* x, long long ldx, int x_f32, const void* w, void* out, long long ldo, int M, int D,
                   float eps, void* stream);
int g4r_cast_f32_f16(const void* x, long long ld, long long bst, void* out,
                      int B, int rows_per_batch, int D, void* stream);
int g4r_fuse_gather_f16(const void* own, const float* own_sc, const float* own_sh, int H,
                         const void* top, const float* top_sc, const float* top_sh, int Ht,
                         const void* down, const float* down_sc, const float* down_sh, int Hd,
                         void* out, int B, int C, void* stream);
int g4r_gn_finalize_f16(const float* stats, const void* gamma, const void* beta,
                    float* scale, float* shift, int B, int C, int groups, int slots,
                    float count, float eps, void* stream);
int g4r_pos_embed_mlp_f16(const float* boxes, const void* w0, const void* b0, const void* g2,
                      const void* be2, const void* w3, const void* b3, const void* g5,
                      const void* be5, float* out, int K, float eps, void* stream);
int g4r_affine_relu_nhwc_f16(const void* z, const float* scale, const float* shift, void* out, int B,
                              long long pix_per_img, int C, void* stream);
int g4r_add_bias_pos_cast_f16(const float* acc, int splits, const void* bias, const float* pos, void* out,
                          int K, int D, void* stream);
int g4r_decode_gemm_f16(const void* x, long long ldx, const void* W, long long ldw, void* out, long long ldo, int M,
                         int N, int K, int act, const void* residual, long long ldr,
                         const void* rope_cos, const void* rope_sin, int rope_cols, int pos0, const int* pos_dev,
                         void* kcache, void* vcache, int cache_lmax, int cache_hd, void* stream);
int g4r_kv_append_f16(const void* qkv, long long ld, void* kcache, void* vcache,
                       int B, int Ln, int pos0, const int* pos_dev /* overrides pos0 when non-NULL */,
                       int Lmax, int HD, void* stream);
int g4r_decode_attention_f16(const void* q, long long ldq, const void* kcache, const void* vcache,
                              void* out, long long ldo, int B, int H, int head_dim, int kv_len,
                              const int* pos_dev /* kv_len = *pos_dev + 1 when non-NULL; kv_len then sizes smem */,
                              int Lmax, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPT4ROI_B200_H_ */
