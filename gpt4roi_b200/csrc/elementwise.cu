// elementwise.cu -- the HBM-bound glue of the region-token path (sm_100a): normalisations,
// rotary embedding, patchify, bilinear resampling / channel shuffle, GroupNorm finalisation and
// the small box-position MLP.  bf16 in / bf16 out, fp32 math, 128-bit accesses.
//
// Each kernel cites the reference op sequence it replaces; rounding points follow what the
// reference produces under bf16 autocast (the only mode in which the SPI module runs, see
// DESIGN.md "numerics").
#include "common.cuh"
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void unpack8(const uint4& raw, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 raw;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; i++) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return raw;
}
// 8 consecutive elements of a bf16 or fp32 row
template <typename T> __device__ __forceinline__ void load8(const T* p, float (&f)[8]);
template <> __device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&f)[8]) {
  unpack8(*reinterpret_cast<const uint4*>(p), f);
}
template <> __device__ __forceinline__ void load8<float>(const float* p, float (&f)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
template <typename T> __device__ __forceinline__ void store8(T* p, const float (&f)[8]);
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&f)[8]) {
  *reinterpret_cast<uint4*>(p) = pack8(f);
}
template <> __device__ __forceinline__ void store8<float>(float* p, const float (&f)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// ------------------------------------------------------------------------------------------
// Row-wise LayerNorm / RMSNorm: one warp per row, the row lives in registers (D <= 8192).
//   LayerNorm: CLIP pre_layrnorm / layer_norm1 / layer_norm2 (transformers modeling_clip.py) and
//              nn.LayerNorm in pos_embedd (gpt4roi/models/layers.py:263,266)
//   RMSNorm  : LlamaRMSNorm (transformers modeling_llama.py:53-67):
//              w * (x * rsqrt(mean(x^2) + eps)).to(bf16)
// ------------------------------------------------------------------------------------------
// PER_LANE = ceil(D/8/32) vectors per lane, compile-time so the row stays in registers.
template <bool RMS, int PER_LANE, typename TI = __nv_bfloat16, typename TO = __nv_bfloat16>
__global__ void __launch_bounds__(256, (sizeof(TI) == 2 && PER_LANE >= 16 ? 2 : 1))
norm_rows_bf16(const TI* __restrict__ x, long long ldx, const __nv_bfloat16* __restrict__ w,
               const __nv_bfloat16* __restrict__ b, TO* __restrict__ out, long long ldo, int M,
               int D, float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  const int nvec = D >> 3;
  const TI* xr = x + (long long)row * ldx;
  // The row lives in registers between the statistics pass and the output pass.  16-bit rows are kept PACKED (one
  // uint4 per 8 elements, widened on use): half the registers of a widened copy, so two to three CTAs fit per SM at
  // D = 4096 instead of one -- the kernel is latency-bound, not ALU-bound (round 1: 3.0 TB/s).
  constexpr bool PACKED = sizeof(TI) == 2;
  uint4 raw[PACKED ? PER_LANE : 1];
  float v[PACKED ? 1 : PER_LANE][8];
  float sum = 0.f, sumsq = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; i++) {
    const int vi = lane + (i << 5);
    float t[8];
    if (vi < nvec) {
      if constexpr (PACKED) { raw[i] = *reinterpret_cast<const uint4*>(xr + vi * 8); unpack8(raw[i], t); }
      else load8<TI>(xr + vi * 8, t);
    } else {
      if constexpr (PACKED) raw[i] = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int j = 0; j < 8; j++) t[j] = 0.f;
    }
    if constexpr (!PACKED) {
#pragma unroll
      for (int j = 0; j < 8; j++) v[i][j] = t[j];
    }
#pragma unroll
    for (int j = 0; j < 8; j++) { sum += t[j]; sumsq += t[j] * t[j]; }
  }
  sum = warp_sum(sum);
  sumsq = warp_sum(sumsq);
  float mean = 0.f, rstd;
  if (RMS) {
    rstd = rsqrtf(sumsq / D + eps);
  } else {
    mean = sum / D;
    float var = 0.f;  // second pass over registers (two-pass variance, like torch)
#pragma unroll
    for (int i = 0; i < PER_LANE; i++) {
      if (lane + (i << 5) < nvec) {
        float t[8];
        if constexpr (PACKED) unpack8(raw[i], t);
#pragma unroll
        for (int j = 0; j < 8; j++) { const float d = (PACKED ? t[j] : v[i][j]) - mean; var += d * d; }
      }
    }
    var = warp_sum(var);
    rstd = rsqrtf(var / D + eps);
  }
  TO* orow = out + (long long)row * ldo;
  const uint4* wv = reinterpret_cast<const uint4*>(w);
  const uint4* bv = reinterpret_cast<const uint4*>(b);
#pragma unroll
  for (int i = 0; i < PER_LANE; i++) {
    const int vi = lane + (i << 5);
    if (vi >= nvec) continue;
    float wf[8], o[8], t[8];
    unpack8(wv[vi], wf);
    if constexpr (PACKED) unpack8(raw[i], t);
    else {
#pragma unroll
      for (int j = 0; j < 8; j++) t[j] = v[i][j];
    }
    if (RMS) {
#pragma unroll
      for (int j = 0; j < 8; j++)   // LlamaRMSNorm: weight * (x * rstd).to(input_dtype) -- no rounding for an fp32 stream
        o[j] = wf[j] * (sizeof(TI) == 4 ? t[j] * rstd : bf16_round(t[j] * rstd));
    } else {
      float bf[8];
      unpack8(bv[vi], bf);
#pragma unroll
      for (int j = 0; j < 8; j++) o[j] = (t[j] - mean) * rstd * wf[j] + bf[j];
    }
    store8<TO>(orow + vi * 8, o);
  }
}

// Few rows (the decode step, M = batch): one CTA per row so the row's latency is one load round, not
// PER_LANE dependent rounds of a single warp.  Same rounding points as norm_rows_bf16.
template <bool RMS, int PER>
__global__ void __launch_bounds__(256)
norm_row_cta_bf16(const __nv_bfloat16* x, long long ldx, const __nv_bfloat16* __restrict__ w,
                  const __nv_bfloat16* __restrict__ b, __nv_bfloat16* out, long long ldo, int D,
                  float eps) {
  __shared__ float red[8];
  __shared__ float stat;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nvec = D >> 3;
  const __nv_bfloat16* xr = x + (long long)blockIdx.x * ldx;
  // programmatic dependent launch (common.cuh): the norm weights are constant -- fetch them, then wait for the
  // kernel that produces x.  x carries no __restrict__ so its loads stay on the coherent path.
  const uint4* wv = reinterpret_cast<const uint4*>(w);
  const uint4* bv = reinterpret_cast<const uint4*>(b);
  uint4 wraw[PER];
#pragma unroll
  for (int i = 0; i < PER; i++) wraw[i] = tid + i * 256 < nvec ? __ldg(wv + tid + i * 256) : make_uint4(0, 0, 0, 0);
  pdl_sync();
  float v[PER][8];
  float sum = 0.f, sumsq = 0.f;
#pragma unroll
  for (int i = 0; i < PER; i++) {
    const int vi = tid + i * 256;
    if (vi < nvec) {
      load8<__nv_bfloat16>(xr + vi * 8, v[i]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; j++) v[i][j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 8; j++) { sum += v[i][j]; sumsq += v[i][j] * v[i][j]; }
  }
  auto block_sum = [&](float t) {
    t = warp_sum(t);
    __syncthreads();
    if (lane == 0) red[warp] = t;
    __syncthreads();
    if (tid == 0) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 8; k++) a += red[k];
      stat = a;
    }
    __syncthreads();
    return stat;
  };
  float mean = 0.f, rstd;
  if (RMS) {
    rstd = rsqrtf(block_sum(sumsq) / D + eps);
  } else {
    mean = block_sum(sum) / D;
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < PER; i++) {
      if (tid + i * 256 < nvec) {
#pragma unroll
        for (int j = 0; j < 8; j++) { const float d = v[i][j] - mean; var += d * d; }
      }
    }
    rstd = rsqrtf(block_sum(var) / D + eps);
  }
  __nv_bfloat16* orow = out + (long long)blockIdx.x * ldo;
#pragma unroll
  for (int i = 0; i < PER; i++) {
    const int vi = tid + i * 256;
    if (vi >= nvec) continue;
    float wf[8], o[8];
    unpack8(wraw[i], wf);
    if (RMS) {
#pragma unroll
      for (int j = 0; j < 8; j++) o[j] = wf[j] * bf16_round(v[i][j] * rstd);
    } else {
      float bf[8];
      unpack8(bv[vi], bf);
#pragma unroll
      for (int j = 0; j < 8; j++) o[j] = (v[i][j] - mean) * rstd * wf[j] + bf[j];
    }
    store8<__nv_bfloat16>(orow + vi * 8, o);
  }
}

template <bool RMS>
static int launch_norm(const void* x, long long ldx, const void* w, const void* b, void* out, long long ldo,
                       int M, int D, float eps, cudaStream_t st) {
  if (M <= 64 && D <= 8192) {
    const int per = (D / 8 + 255) / 256;
#define G4R_NORM_ROW_CASE(PR)                                                                              \
  G4R_CUDA(launch_pdl(norm_row_cta_bf16<RMS, PR>, dim3(M), dim3(256), 0, st, dim3(1, 1, 1),                \
                      (const __nv_bfloat16*)x, ldx, (const __nv_bfloat16*)w, (const __nv_bfloat16*)b,     \
                      (__nv_bfloat16*)out, ldo, D, eps))
    if (per <= 1) G4R_NORM_ROW_CASE(1);
    else if (per <= 2) G4R_NORM_ROW_CASE(2);
    else G4R_NORM_ROW_CASE(4);
#undef G4R_NORM_ROW_CASE
    G4R_LAUNCH_CHECK(RMS ? "rmsnorm" : "layernorm");
    return G4R_OK;
  }
  const int per_lane = (D / 8 + 31) / 32;
  const dim3 grid((M + 7) / 8);
#define G4R_NORM_CASE(PL)                                                                              \
  norm_rows_bf16<RMS, PL><<<grid, 256, 0, st>>>((const __nv_bfloat16*)x, ldx, (const __nv_bfloat16*)w,   \
                                                 (const __nv_bfloat16*)b, (__nv_bfloat16*)out, ldo, M, D, eps)
  if (per_lane <= 1) G4R_NORM_CASE(1);
  else if (per_lane <= 2) G4R_NORM_CASE(2);
  else if (per_lane <= 4) G4R_NORM_CASE(4);
  else if (per_lane <= 8) G4R_NORM_CASE(8);
  else if (per_lane <= 16) G4R_NORM_CASE(16);
  else G4R_NORM_CASE(32);
#undef G4R_NORM_CASE
  G4R_LAUNCH_CHECK(RMS ? "rmsnorm" : "layernorm");
  return G4R_OK;
}

template <typename TI, typename TO, bool RMS = false>
static int launch_ln_ex(const void* x, long long ldx, const void* w, const void* b, void* out, long long ldo,
                        int M, int D, float eps, cudaStream_t st) {
  const int per_lane = (D / 8 + 31) / 32;
  const dim3 grid((M + 7) / 8);
#define G4R_LN_CASE(PL)                                                                                   \
  norm_rows_bf16<RMS, PL, TI, TO><<<grid, 256, 0, st>>>((const TI*)x, ldx, (const __nv_bfloat16*)w,        \
                                                        (const __nv_bfloat16*)b, (TO*)out, ldo, M, D, eps)
  if (per_lane <= 1) G4R_LN_CASE(1);
  else if (per_lane <= 2) G4R_LN_CASE(2);
  else if (per_lane <= 4) G4R_LN_CASE(4);
  else if (per_lane <= 8) G4R_LN_CASE(8);
  else if (per_lane <= 16) G4R_LN_CASE(16);
  else G4R_LN_CASE(32);
#undef G4R_LN_CASE
  G4R_LAUNCH_CHECK("layernorm_ex");
  return G4R_OK;
}

// rows [B][rows_per_batch][D] (row stride ld, batch stride bst) fp32 -> dense bf16 [B*rows_per_batch, D]
__global__ void __launch_bounds__(256)
cast_rows_f32_bf16(const float* __restrict__ x, long long ld, long long bst, __nv_bfloat16* __restrict__ out,
                   int B, int rows_per_batch, int D) {
  const int nvec = D >> 3;
  const long long total = (long long)B * rows_per_batch * nvec;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    const int r = (int)((i / nvec) % rows_per_batch);
    const int b = (int)(i / ((long long)nvec * rows_per_batch));
    float f[8];
    load8<float>(x + (long long)b * bst + (long long)r * ld + v * 8, f);
    store8<__nv_bfloat16>(out + ((long long)b * rows_per_batch + r) * D + v * 8, f);
  }
}

// ------------------------------------------------------------------------------------------
// Rotary embedding, in place on the q and k parts of a packed [rows, (q|k|v)] buffer.
// transformers modeling_llama.py:138-168: q*cos + rotate_half(q)*sin with cos/sin already cast
// to bf16; each bf16 tensor op rounds, so: out = bf16( bf16(q*cos) + bf16(rot*sin) ).
// cos/sin: bf16 tables [L, head_dim] (computed on the host exactly as LlamaRotaryEmbedding does).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rope_inplace_bf16(__nv_bfloat16* __restrict__ qkv, long long ld, const __nv_bfloat16* __restrict__ cos_t,
                  const __nv_bfloat16* __restrict__ sin_t, int rows, int L, int n_heads_qk, int head_dim) {
  // one thread = 8 consecutive dims of the first half of a head and their partners in the second half
  const int half = head_dim >> 1;
  const int vph = half >> 3;  // 16-byte vectors per half head
  const long long total = (long long)rows * n_heads_qk * vph;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % vph);
    const int h = (int)((i / vph) % n_heads_qk);
    const long long r = i / ((long long)vph * n_heads_qk);
    const int pos = (int)(r % L);
    __nv_bfloat16* p = qkv + r * ld + (long long)h * head_dim + v * 8;
    float x1[8], x2[8], c1[8], s1[8], c2[8], s2[8], o1[8], o2[8];
    unpack8(*reinterpret_cast<const uint4*>(p), x1);
    unpack8(*reinterpret_cast<const uint4*>(p + half), x2);
    const __nv_bfloat16* ct = cos_t + (long long)pos * head_dim + v * 8;
    const __nv_bfloat16* st = sin_t + (long long)pos * head_dim + v * 8;
    unpack8(*reinterpret_cast<const uint4*>(ct), c1);
    unpack8(*reinterpret_cast<const uint4*>(st), s1);
    unpack8(*reinterpret_cast<const uint4*>(ct + half), c2);
    unpack8(*reinterpret_cast<const uint4*>(st + half), s2);
#pragma unroll
    for (int j = 0; j < 8; j++) {
      // rotate_half(x) = cat(-x2, x1)
      o1[j] = bf16_round(x1[j] * c1[j]) + bf16_round(-x2[j] * s1[j]);
      o2[j] = bf16_round(x2[j] * c2[j]) + bf16_round(x1[j] * s2[j]);
    }
    *reinterpret_cast<uint4*>(p) = pack8(o1);
    *reinterpret_cast<uint4*>(p + half) = pack8(o2);
  }
}

// ------------------------------------------------------------------------------------------
// CLIP patchify: images [B,3,S,S] (bf16, NCHW) -> rows [B*P, Kpad], column (c*ps+ky)*ps+kx
// (the flatten order of the patch_embedding conv weight [hidden,3,ps,ps]); columns >= 3*ps*ps
// are zero.  transformers modeling_clip.py:148-154,209-216 (Conv2d stride=patch, no bias).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
patchify_bf16(const __nv_bfloat16* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int S, int ps,
              int Kpad) {
  const int G = S / ps;
  const long long total = (long long)B * G * G * Kpad;
  const int kreal = 3 * ps * ps;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % Kpad);
    const long long prow = i / Kpad;
    __nv_bfloat16 v = __float2bfloat16_rn(0.f);
    if (col < kreal) {
      const int kx = col % ps, ky = (col / ps) % ps, c = col / (ps * ps);
      const int px = (int)(prow % G), py = (int)((prow / G) % G);
      const int b = (int)(prow / ((long long)G * G));
      v = img[(((long long)b * 3 + c) * S + (py * ps + ky)) * S + px * ps + kx];
    }
    out[i] = v;
  }
}

// x[b,0,:] = cls + pos[0]; x[b,1+p,:] = patch[b,p,:] + pos[1+p]  (modeling_clip.py:209-216)
__global__ void __launch_bounds__(256)
vit_embed_bf16(const __nv_bfloat16* __restrict__ patch, const __nv_bfloat16* __restrict__ cls,
               const __nv_bfloat16* __restrict__ pos, __nv_bfloat16* __restrict__ out, int B, int P, int D) {
  const int nvec = D >> 3;
  const long long total = (long long)B * (P + 1) * nvec;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    const int t = (int)((i / nvec) % (P + 1));
    const int b = (int)(i / ((long long)nvec * (P + 1)));
    float a[8], pz[8], o[8];
    if (t == 0) unpack8(reinterpret_cast<const uint4*>(cls)[v], a);
    else unpack8(reinterpret_cast<const uint4*>(patch + ((long long)b * P + t - 1) * D)[v], a);
    unpack8(reinterpret_cast<const uint4*>(pos + (long long)t * D)[v], pz);
#pragma unroll
    for (int j = 0; j < 8; j++) o[j] = a[j] + pz[j];
    reinterpret_cast<uint4*>(out + ((long long)b * (P + 1) + t) * D)[v] = pack8(o);
  }
}

// ------------------------------------------------------------------------------------------
// Bilinear resampling helpers, align_corners=True (ATen upsample_bilinear2d):
//   scale = (in-1)/(out-1) (0 if out==1); src = scale*dst; i0=(int)src; i1=i0+(i0<in-1); l1=src-i0
// ------------------------------------------------------------------------------------------
struct Lerp {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ Lerp lerp_ac(int dst, int in, int out) {
  const float scale = out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f;
  const float src = scale * dst;
  Lerp r;
  r.i0 = (int)src;
  if (r.i0 > in - 1) r.i0 = in - 1;
  r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
  r.l1 = src - r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

// ViT tokens -> pyramid level input (gpt4roi/models/layers.py:219-232 + :117-126,185-188):
//   tokens [B, G*G, C] (row stride ldt, batch stride bst; CLS already skipped by the caller) are the
//   NHWC map [B,G,G,C]; resize to [B,Ho,Ho,C] (bf16 out, fp32 math), append x = linspace(-1,1,Wo)[xo],
//   y = linspace(-1,1,Ho)[yo] as channels C, C+1 (bf16-rounded, as autocast does at the conv input)
//   and zero-pad to Cpad channels (K of the following 1x1-conv GEMM must be a multiple of 8).
template <typename TT>
__global__ void __launch_bounds__(256)
upsample_tokens_coords_bf16(const TT* __restrict__ tok, long long ldt, long long bst,
                            __nv_bfloat16* __restrict__ out, int B, int G, int Ho, int C, int Cpad) {
  const int nvec = Cpad >> 3;
  const long long total = (long long)B * Ho * Ho * nvec;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long q1, q2, bq;
    int v, xo, yo;
    divmod_idx(i, nvec, q1, v);
    divmod_idx(q1, Ho, q2, xo);
    divmod_idx(q2, Ho, bq, yo);
    const int b = (int)bq;
    float o[8];
    if (v * 8 < C) {
      const Lerp ly = lerp_ac(yo, G, Ho), lx = lerp_ac(xo, G, Ho);
      const TT* base = tok + (long long)b * bst + v * 8;
      float a[8], bb[8], c[8], d[8];
      load8<TT>(base + ((long long)ly.i0 * G + lx.i0) * ldt, a);
      load8<TT>(base + ((long long)ly.i0 * G + lx.i1) * ldt, bb);
      load8<TT>(base + ((long long)ly.i1 * G + lx.i0) * ldt, c);
      load8<TT>(base + ((long long)ly.i1 * G + lx.i1) * ldt, d);
#pragma unroll
      for (int j = 0; j < 8; j++)
        o[j] = ly.l0 * (lx.l0 * a[j] + lx.l1 * bb[j]) + ly.l1 * (lx.l0 * c[j] + lx.l1 * d[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; j++) o[j] = 0.f;
      if (v * 8 == C) {
        // torch.linspace(-1, 1, n): start + i*step for i < n/2, end - (n-1-i)*step otherwise
        const float step = Ho > 1 ? 2.f / (float)(Ho - 1) : 0.f;
        o[0] = xo < Ho / 2 ? -1.f + step * xo : 1.f - step * (Ho - 1 - xo);
        o[1] = yo < Ho / 2 ? -1.f + step * yo : 1.f - step * (Ho - 1 - yo);
      }
    }
    reinterpret_cast<uint4*>(out + (((long long)b * Ho + yo) * Ho + xo) * Cpad)[v] = pack8(o);
  }
}

// One level of MLVLFuseModule._single_shuffle (gpt4roi/models/layers.py:152-180): builds the conv
// input [own[:, :C/2] | resize(top[:, 3C/4:]) | resize(down[:, C/2:3C/4])], NHWC bf16.
// Sources are the PREVIOUS round's raw conv outputs (bf16); when sc/sh (fp32 [B,C]) are given the
// previous round's GroupNorm+ReLU is applied to every tap first: relu(v*sc + sh) in fp32 -- i.e.
// ConvModule's GN->ReLU (mmcv cnn/bricks/conv_module.py:196-208) is fused into this gather and the
// resampling runs on fp32 values exactly like F.interpolate(x.to(float32), ...) at :166-175.
struct FuseSrc {
  const __nv_bfloat16* __restrict__ p;
  const float* __restrict__ sc;
  const float* __restrict__ sh;
  int H;
};
__device__ __forceinline__ void act8(const uint4& raw, bool affine, const float (&aa)[8], const float (&dd)[8],
                                     float (&f)[8]) {
  unpack8(raw, f);
  if (affine) {
#pragma unroll
    for (int j = 0; j < 8; j++) f[j] = fmaxf(f[j] * aa[j] + dd[j], 0.f);
  }
}
__global__ void __launch_bounds__(256)
fuse_gather_bf16(FuseSrc own, FuseSrc top, FuseSrc down, __nv_bfloat16* __restrict__ out, int B, int C) {
  const int H = own.H;
  const int nvec = C >> 3;
  const int q = C >> 2;  // shuffle_channels = C/4; remain = C/2
  // a group of `nvec` consecutive threads owns one output pixel (coalesced 16-byte channel vectors);
  // the pixel decomposition is done once per thread, not per element
  const int ppb = blockDim.x / nvec;  // pixels per block (launcher guarantees blockDim % nvec == 0)
  const long long npix = (long long)B * H * H;
  const int v = threadIdx.x % nvec;
  // the channel slice -- and with it the source map and its GroupNorm scale / shift vectors -- is fixed per thread;
  // the scale / shift (64 bytes per thread, 4x the 16-byte payload of an own-channel pixel) are reloaded only when
  // the grid-stride loop crosses into another image
  const int c = v * 8;
  // out channels [0,C/2) <- own; [C/2,3C/4) <- top[:, 3C/4 + j]; [3C/4,C) <- down[:, C/2 + j]
  const bool is_own = c < 2 * q, from_top = c < 3 * q;
  const FuseSrc& s = is_own ? own : (from_top ? top : down);
  const int sc0 = is_own ? c : (from_top ? c + q : c - q);
  const bool affine = s.sc != nullptr;
  float aa[8], dd[8];
  int cur_b = -1;
  // (b, y, x) advance incrementally with the grid stride: no 64-bit div / mod per pixel (three of them cost more
  // instructions than the pixel's arithmetic); the align_corners scale is loop-invariant
  const long long pix0 = (long long)blockIdx.x * ppb + threadIdx.x / nvec;
  const long long step = (long long)gridDim.x * ppb;
  const int HH = H * H;
  int b = (int)(pix0 / HH), y = (int)((pix0 % HH) / H), x = (int)(pix0 % H);
  const int sb = (int)(step / HH), sy = (int)((step % HH) / H), sx = (int)(step % H);
  const float lscale = (H > 1 && s.H != H) ? (float)(s.H - 1) / (float)(H - 1) : 0.f;
  auto lerp = [&](int dst) {
    const float src = lscale * dst;
    Lerp r;
    r.i0 = (int)src;
    if (r.i0 > s.H - 1) r.i0 = s.H - 1;
    r.i1 = r.i0 + (r.i0 < s.H - 1 ? 1 : 0);
    r.l1 = src - r.i0;
    r.l0 = 1.f - r.l1;
    return r;
  };
  for (long long pix = pix0; pix < npix; pix += step, x += sx, y += sy, b += sb) {
    if (x >= H) { x -= H; y++; }
    if (y >= H) { y -= H; b++; }
    if (affine && b != cur_b) {
      const float4* a = reinterpret_cast<const float4*>(s.sc + (long long)b * C + sc0);
      const float4* d = reinterpret_cast<const float4*>(s.sh + (long long)b * C + sc0);
      const float4 a0 = a[0], a1 = a[1], d0 = d[0], d1 = d[1];
      aa[0] = a0.x; aa[1] = a0.y; aa[2] = a0.z; aa[3] = a0.w; aa[4] = a1.x; aa[5] = a1.y; aa[6] = a1.z; aa[7] = a1.w;
      dd[0] = d0.x; dd[1] = d0.y; dd[2] = d0.z; dd[3] = d0.w; dd[4] = d1.x; dd[5] = d1.y; dd[6] = d1.z; dd[7] = d1.w;
      cur_b = b;
    }
    const __nv_bfloat16* base = s.p + (long long)b * s.H * s.H * C + sc0;
    float o[8];
    if (s.H == H) {  // own channels, or a same-size "resize" (identity)
      act8(*reinterpret_cast<const uint4*>(base + ((long long)y * H + x) * C), affine, aa, dd, o);
    } else {
      const Lerp ly = lerp(y), lx = lerp(x);
      const uint4 r00 = *reinterpret_cast<const uint4*>(base + ((long long)ly.i0 * s.H + lx.i0) * C);
      const uint4 r01 = *reinterpret_cast<const uint4*>(base + ((long long)ly.i0 * s.H + lx.i1) * C);
      const uint4 r10 = *reinterpret_cast<const uint4*>(base + ((long long)ly.i1 * s.H + lx.i0) * C);
      const uint4 r11 = *reinterpret_cast<const uint4*>(base + ((long long)ly.i1 * s.H + lx.i1) * C);
      float a[8], bb[8], cc[8], d[8];
      act8(r00, affine, aa, dd, a);
      act8(r01, affine, aa, dd, bb);
      act8(r10, affine, aa, dd, cc);
      act8(r11, affine, aa, dd, d);
#pragma unroll
      for (int j = 0; j < 8; j++)
        o[j] = ly.l0 * (lx.l0 * a[j] + lx.l1 * bb[j]) + ly.l1 * (lx.l0 * cc[j] + lx.l1 * d[j]);
    }
    reinterpret_cast<uint4*>(out + (((long long)b * H + y) * H + x) * C)[v] = pack8(o);
  }
}

// Adjoint of fuse_gather_bf16 (training step): gradient w.r.t. the ACTIVATED maps of the previous round at
// pyramid level m, from the gradients d_in of the conv inputs of the levels that read level m:
//   channels [0, C/2)      <- d_in_m[:, 0:C/2]                                (own)
//   channels [C/2, 3C/4)   <- sum over levels l with down(l) = m of resize^T(d_in_l[:, 3C/4:C])
//   channels [3C/4, C)     <- sum over levels l with top(l)  = m of resize^T(d_in_l[:, C/2:3C/4])
// resize^T is the transpose of the align_corners bilinear resize from size H_m to H_l, evaluated as a GATHER
// per source pixel (every destination pixel whose footprint contains it), so there are no atomics and the
// summation order is fixed.  Same-size consumers are the identity.  Output fp32 [B, Hm, Hm, C].
struct FuseGrad {
  const __nv_bfloat16* __restrict__ p;   // d_in of a consumer level (bf16 NHWC), or null
  int H;
};
__device__ __forceinline__ void adjoint_resize8(const FuseGrad& gsrc, int b, int ys, int xs, int Hs, int C, int ch,
                                                float (&acc)[8]) {
  const int Hd = gsrc.H;
  const __nv_bfloat16* base = gsrc.p + (long long)b * Hd * Hd * C + ch;
  if (Hd == Hs) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(base + ((long long)ys * Hd + xs) * C), f);
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j] += f[j];
    return;
  }
  const float r = Hs > 1 ? (float)(Hd - 1) / (float)(Hs - 1) : 0.f;
  const int ylo = max(0, (int)floorf((ys - 1) * r) - 1), yhi = min(Hd - 1, (int)ceilf((ys + 1) * r) + 1);
  const int xlo = max(0, (int)floorf((xs - 1) * r) - 1), xhi = min(Hd - 1, (int)ceilf((xs + 1) * r) + 1);
  for (int yd = ylo; yd <= yhi; yd++) {
    const Lerp ly = lerp_ac(yd, Hs, Hd);
    const float wy = (ly.i0 == ys ? ly.l0 : 0.f) + (ly.i1 == ys ? ly.l1 : 0.f);
    if (wy == 0.f) continue;
    for (int xd = xlo; xd <= xhi; xd++) {
      const Lerp lx = lerp_ac(xd, Hs, Hd);
      const float wx = (lx.i0 == xs ? lx.l0 : 0.f) + (lx.i1 == xs ? lx.l1 : 0.f);
      if (wx == 0.f) continue;
      float f[8];
      unpack8(*reinterpret_cast<const uint4*>(base + ((long long)yd * Hd + xd) * C), f);
      const float wgt = wy * wx;
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] += wgt * f[j];
    }
  }
}
__global__ void __launch_bounds__(256)
fuse_gather_bwd(FuseGrad own, FuseGrad dn0, FuseGrad dn1, FuseGrad tp0, FuseGrad tp1, float* __restrict__ out, int B, int C) {
  const int H = own.H;
  const int nvec = C >> 3, q = C >> 2;
  const int ppb = blockDim.x / nvec;
  const long long npix = (long long)B * H * H;
  const int v = threadIdx.x % nvec;
  for (long long pix = (long long)blockIdx.x * ppb + threadIdx.x / nvec; pix < npix; pix += (long long)gridDim.x * ppb) {
    long long rowq, bq;
    int x, y;
    divmod_idx(pix, H, rowq, x);
    divmod_idx(rowq, H, bq, y);
    const int b = (int)bq;
    const int c = v * 8;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j] = 0.f;
    if (c < 2 * q) {
      unpack8(*reinterpret_cast<const uint4*>(own.p + (((long long)b * H + y) * H + x) * C + c), acc);
    } else if (c < 3 * q) {   // read as "down" source: consumer channel c + C/4
      if (dn0.p) adjoint_resize8(dn0, b, y, x, H, C, c + q, acc);
      if (dn1.p) adjoint_resize8(dn1, b, y, x, H, C, c + q, acc);
    } else {                  // read as "top" source: consumer channel c - C/4
      if (tp0.p) adjoint_resize8(tp0, b, y, x, H, C, c - q, acc);
      if (tp1.p) adjoint_resize8(tp1, b, y, x, H, C, c - q, acc);
    }
    float* o = out + (((long long)b * H + y) * H + x) * C + c;
    reinterpret_cast<float4*>(o)[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    reinterpret_cast<float4*>(o)[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
}

// GroupNorm finalisation: stats [B,groups,2] (sum, sumsq over H*W*cpg elements) + gamma/beta ->
// per-(image,channel) scale/shift so that GN(x) = x*scale + shift (eps inside the rsqrt, biased
// variance, like torch.nn.GroupNorm).
// One warp per (image, group): lanes stride over the per-(tile,warp) partial slots (fixed order per
// lane + fixed shuffle tree => bitwise reproducible), then the first cpg lanes write scale/shift.
__global__ void __launch_bounds__(256)
gn_finalize(const float* __restrict__ stats, const __nv_bfloat16* __restrict__ gamma,
            const __nv_bfloat16* __restrict__ beta, float* __restrict__ scale, float* __restrict__ shift, int B,
            int C, int groups, int slots, float count, float eps) {
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= B * groups) return;
  const int lane = threadIdx.x & 31;
  const int b = w / groups, g = w % groups;
  float s = 0.f, ss = 0.f;
  for (int t = lane; t < slots; t += 32) {
    const float2 v = *reinterpret_cast<const float2*>(stats + (((long long)b * slots + t) * groups + g) * 2);
    s += v.x;
    ss += v.y;
  }
  s = warp_sum(s);
  ss = warp_sum(ss);
  const float mean = s / count;
  float var = ss / count - mean * mean;
  var = var < 0.f ? 0.f : var;
  const float rstd = rsqrtf(var + eps);
  const int cpg = C / groups;
  for (int j = lane; j < cpg; j += 32) {
    const int c = g * cpg + j;
    const float a = __bfloat162float(gamma[c]) * rstd;
    scale[(long long)b * C + c] = a;
    shift[(long long)b * C + c] = __bfloat162float(beta[c]) - mean * a;
  }
}

// ------------------------------------------------------------------------------------------
// pos_embedd (gpt4roi/models/layers.py:260-267,285): Linear(4,256) ReLU LN(256) Linear(256,1024)
// ReLU LN(1024) on the normalised xyxy boxes.  One CTA (256 threads) per box.  Under autocast the
// Linears run in bf16 (inputs/weights bf16, fp32 accumulate, bf16 output) and LayerNorm in fp32;
// the output stays fp32 (it is added to flatten_linear's result in fp32, :328).
// ------------------------------------------------------------------------------------------
__device__ float block_sum_256(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) t += red[i];
  __syncthreads();
  return t;
}
__global__ void __launch_bounds__(256)
pos_embed_mlp(const float* __restrict__ boxes, const __nv_bfloat16* __restrict__ w0,
              const __nv_bfloat16* __restrict__ b0, const __nv_bfloat16* __restrict__ g2,
              const __nv_bfloat16* __restrict__ be2, const __nv_bfloat16* __restrict__ w3,
              const __nv_bfloat16* __restrict__ b3, const __nv_bfloat16* __restrict__ g5,
              const __nv_bfloat16* __restrict__ be5, float* __restrict__ out, float eps) {
  __shared__ float h1[256];
  __shared__ float red[8];
  const int k = blockIdx.x, t = threadIdx.x;
  float bx[4];
#pragma unroll
  for (int j = 0; j < 4; j++) bx[j] = bf16_round(boxes[k * 4 + j]);  // autocast: input -> bf16
  float a = __bfloat162float(b0[t]);
#pragma unroll
  for (int j = 0; j < 4; j++) a += bx[j] * __bfloat162float(w0[t * 4 + j]);
  a = fmaxf(bf16_round(a), 0.f);
  // LayerNorm(256) in fp32
  float mean = block_sum_256(a, red) / 256.f;
  float d = a - mean;
  float var = block_sum_256(d * d, red) / 256.f;
  float y = d * rsqrtf(var + eps) * __bfloat162float(g2[t]) + __bfloat162float(be2[t]);
  h1[t] = bf16_round(y);  // next Linear's input is cast to bf16
  __syncthreads();
  float o[4];
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int n = t + r * 256;
    float acc = 0.f;
    const uint4* wr = reinterpret_cast<const uint4*>(w3 + (long long)n * 256);
    for (int v = 0; v < 32; v++) {
      float wf[8];
      unpack8(wr[v], wf);
#pragma unroll
      for (int j = 0; j < 8; j++) acc += wf[j] * h1[v * 8 + j];
    }
    acc += __bfloat162float(b3[n]);
    o[r] = fmaxf(bf16_round(acc), 0.f);
  }
  float s = o[0] + o[1] + o[2] + o[3];
  mean = block_sum_256(s, red) / 1024.f;
  float vs = 0.f;
#pragma unroll
  for (int r = 0; r < 4; r++) { const float dd = o[r] - mean; vs += dd * dd; }
  var = block_sum_256(vs, red) / 1024.f;
  const float rstd = rsqrtf(var + eps);
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int n = t + r * 256;
    out[(long long)k * 1024 + n] = (o[r] - mean) * rstd * __bfloat162float(g5[n]) + __bfloat162float(be5[n]);
  }
}

// Backward of pos_embed_mlp (training step): one CTA per RoI recomputes the forward and writes that RoI's
// parameter-gradient slab [w0 4x256 | b0 | g2 | be2 | w3 1024x256 | b3 | g5 | be5] (fp32, kPosSlab floats);
// pos_slab_reduce sums the slabs over the RoIs in order.  Rounding points of the forward are treated as identity.
constexpr int kPosSlab = 1024 + 256 * 3 + 1024 * 256 + 1024 * 3;
__global__ void __launch_bounds__(256)
pos_embed_mlp_bwd(const float* __restrict__ boxes, const __nv_bfloat16* __restrict__ w0,
                  const __nv_bfloat16* __restrict__ b0, const __nv_bfloat16* __restrict__ g2,
                  const __nv_bfloat16* __restrict__ be2, const __nv_bfloat16* __restrict__ w3,
                  const __nv_bfloat16* __restrict__ b3, const __nv_bfloat16* __restrict__ g5,
                  const __nv_bfloat16* __restrict__ dout, long long ldd, float* __restrict__ slabs, float eps) {
  __shared__ float h1[256];
  __shared__ float du2s[1024];
  __shared__ float red[8];
  const int k = blockIdx.x, t = threadIdx.x;
  float* sl = slabs + (long long)k * kPosSlab;
  float bx[4];
#pragma unroll
  for (int j = 0; j < 4; j++) bx[j] = bf16_round(boxes[k * 4 + j]);
  float u1 = __bfloat162float(b0[t]);
#pragma unroll
  for (int j = 0; j < 4; j++) u1 += bx[j] * __bfloat162float(w0[t * 4 + j]);
  const float r1 = fmaxf(bf16_round(u1), 0.f);
  const float mean1 = block_sum_256(r1, red) / 256.f;
  const float d1 = r1 - mean1;
  const float rstd1 = rsqrtf(block_sum_256(d1 * d1, red) / 256.f + eps);
  const float xh1 = d1 * rstd1;
  const float g2f = __bfloat162float(g2[t]);
  h1[t] = bf16_round(xh1 * g2f + __bfloat162float(be2[t]));
  __syncthreads();
  float u2[4], r2[4];
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int n = t + r * 256;
    float acc = 0.f;
    const uint4* wr = reinterpret_cast<const uint4*>(w3 + (long long)n * 256);
    for (int v = 0; v < 32; v++) {
      float wf[8];
      unpack8(wr[v], wf);
#pragma unroll
      for (int j = 0; j < 8; j++) acc += wf[j] * h1[v * 8 + j];
    }
    u2[r] = bf16_round(acc + __bfloat162float(b3[n]));
    r2[r] = fmaxf(u2[r], 0.f);
  }
  const float mean2 = block_sum_256(r2[0] + r2[1] + r2[2] + r2[3], red) / 1024.f;
  float vs = 0.f;
#pragma unroll
  for (int r = 0; r < 4; r++) { const float dd = r2[r] - mean2; vs += dd * dd; }
  const float rstd2 = rsqrtf(block_sum_256(vs, red) / 1024.f + eps);
  // ---- LayerNorm(1024) backward
  float dxh[4], xh2[4], s1 = 0.f, s2 = 0.f;
  float* o_w3 = sl + 1024 + 768;
  float* o_b3 = o_w3 + 1024 * 256;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int n = t + r * 256;
    const float dy = __bfloat162float(dout[(long long)k * ldd + n]);
    xh2[r] = (r2[r] - mean2) * rstd2;
    o_b3[1024 + n] = dy * xh2[r];          // dg5
    o_b3[2048 + n] = dy;                   // dbe5
    dxh[r] = dy * __bfloat162float(g5[n]);
    s1 += dxh[r];
    s2 += dxh[r] * xh2[r];
  }
  s1 = block_sum_256(s1, red) / 1024.f;
  s2 = block_sum_256(s2, red) / 1024.f;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int n = t + r * 256;
    const float dr2 = rstd2 * (dxh[r] - s1 - xh2[r] * s2);
    const float du2 = u2[r] > 0.f ? dr2 : 0.f;
    du2s[n] = du2;
    o_b3[n] = du2;                         // db3
    float* row = o_w3 + (long long)n * 256;
    for (int i = 0; i < 256; i++) row[i] = du2 * h1[i];   // dW3[n, :]
  }
  __syncthreads();
  // dn1[t] = sum_n W3[n, t] * du2[n]
  float dn1 = 0.f;
  for (int n = 0; n < 1024; n++) dn1 += __bfloat162float(w3[(long long)n * 256 + t]) * du2s[n];
  // ---- LayerNorm(256) backward
  sl[1024 + 256 + t] = dn1 * xh1;          // dg2
  sl[1024 + 512 + t] = dn1;                // dbe2
  const float dx1 = dn1 * g2f;
  const float m1 = block_sum_256(dx1, red) / 256.f;
  const float m2 = block_sum_256(dx1 * xh1, red) / 256.f;
  const float dr1 = rstd1 * (dx1 - m1 - xh1 * m2);
  const float du1 = bf16_round(u1) > 0.f ? dr1 : 0.f;
  sl[1024 + t] = du1;                      // db0
#pragma unroll
  for (int j = 0; j < 4; j++) sl[t * 4 + j] = du1 * bx[j];   // dW0[t, :]
}

__global__ void __launch_bounds__(256)
pos_slab_reduce(const float* __restrict__ slabs, int K, float* __restrict__ out) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= kPosSlab) return;
  float a = 0.f;
  for (int k = 0; k < K; k++) a += slabs[(long long)k * kPosSlab + i];
  out[i] = a;
}

// t[k,:] = bf16( bf16(acc[k,:] + bias) + pos[k,:] )   (gpt4roi/models/layers.py:327-328: flatten_linear
// output is bf16 under autocast, `+ pos_embedd` promotes to fp32, updims casts its input to bf16)
__global__ void add_bias_pos_cast(const float* __restrict__ acc, int splits, const __nv_bfloat16* __restrict__ bias,
                                  const float* __restrict__ pos, __nv_bfloat16* __restrict__ out, int K, int D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * D) return;
  const int c = i % D;
  float a = 0.f;
  for (int s = 0; s < splits; s++) a += acc[(long long)s * K * D + i];  // split-K slabs, fixed order
  const float f = bf16_round(a + __bfloat162float(bias[c]));
  out[i] = __float2bfloat16_rn(f + pos[i]);
}

static inline int grid_for(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace g4r

using namespace G4R_NS;

extern "C" int g4r_layernorm_bf16(const void* x, long long ldx, const void* w, const void* b, void* out,
                                  long long ldo, int M, int D, float eps, void* stream) {
  G4R_REQUIRE(x && w && b && out && M > 0 && D > 0 && D % 8 == 0 && D <= 8192 && ldx % 8 == 0 && ldo % 8 == 0,
              "layernorm: bad arguments (D=%d must be a multiple of 8, <= 8192)", D);
  return launch_norm<false>(x, ldx, w, b, out, ldo, M, D, eps, (cudaStream_t)stream);
}

extern "C" int g4r_rmsnorm_bf16(const void* x, long long ldx, const void* w, void* out, long long ldo, int M,
                                int D, float eps, void* stream) {
  G4R_REQUIRE(x && w && out && M > 0 && D > 0 && D % 8 == 0 && D <= 8192 && ldx % 8 == 0 && ldo % 8 == 0,
              "rmsnorm: bad arguments (D=%d)", D);
  return launch_norm<true>(x, ldx, w, nullptr, out, ldo, M, D, eps, (cudaStream_t)stream);
}

extern "C" int g4r_rope_inplace_bf16(void* qkv, long long ld, const void* cos_t, const void* sin_t, int rows,
                                     int L, int n_heads_qk, int head_dim, void* stream) {
  G4R_REQUIRE(qkv && cos_t && sin_t && rows > 0 && L > 0 && n_heads_qk > 0 && head_dim % 16 == 0 && ld % 8 == 0, "rope: bad arguments");
  const long long total = (long long)rows * n_heads_qk * (head_dim / 16);
  rope_inplace_bf16<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      (__nv_bfloat16*)qkv, ld, (const __nv_bfloat16*)cos_t, (const __nv_bfloat16*)sin_t, rows, L, n_heads_qk, head_dim);
  G4R_LAUNCH_CHECK("rope");
  return G4R_OK;
}

extern "C" int g4r_patchify_bf16(const void* img, void* out, int B, int S, int ps, int Kpad, void* stream) {
  G4R_REQUIRE(img && out && B > 0 && S > 0 && ps > 0 && S % ps == 0 && Kpad >= 3 * ps * ps, "patchify: bad arguments");
  const long long total = (long long)B * (S / ps) * (S / ps) * Kpad;
  patchify_bf16<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)img, (__nv_bfloat16*)out, B, S, ps, Kpad);
  G4R_LAUNCH_CHECK("patchify");
  return G4R_OK;
}

extern "C" int g4r_vit_embed_bf16(const void* patch, const void* cls, const void* pos, void* out, int B, int P,
                                  int D, void* stream) {
  G4R_REQUIRE(patch && cls && pos && out && B > 0 && P > 0 && D % 8 == 0, "vit_embed: bad arguments");
  const long long total = (long long)B * (P + 1) * (D / 8);
  vit_embed_bf16<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)patch, (const __nv_bfloat16*)cls, (const __nv_bfloat16*)pos, (__nv_bfloat16*)out, B, P, D);
  G4R_LAUNCH_CHECK("vit_embed");
  return G4R_OK;
}

extern "C" int g4r_upsample_tokens_coords_bf16(const void* tok, long long ldt, long long bst, void* out, int B,
                                               int G, int Ho, int C, int Cpad, void* stream) {
  G4R_REQUIRE(tok && out && B > 0 && G > 0 && Ho > 0 && C % 8 == 0 && Cpad % 8 == 0 && Cpad >= C + 8 && ldt % 8 == 0 && bst % 8 == 0,
              "upsample_tokens_coords: bad arguments");
  const long long total = (long long)B * Ho * Ho * (Cpad / 8);
  upsample_tokens_coords_bf16<__nv_bfloat16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)tok, ldt, bst, (__nv_bfloat16*)out, B, G, Ho, C, Cpad);
  G4R_LAUNCH_CHECK("upsample_tokens_coords");
  return G4R_OK;
}

extern "C" int g4r_upsample_tokens_coords_f32(const void* tok, long long ldt, long long bst, void* out, int B,
                                              int G, int Ho, int C, int Cpad, void* stream) {
  G4R_REQUIRE(tok && out && B > 0 && G > 0 && Ho > 0 && C % 8 == 0 && Cpad % 8 == 0 && Cpad >= C + 8 && ldt % 4 == 0 && bst % 4 == 0,
              "upsample_tokens_coords_f32: bad arguments");
  const long long total = (long long)B * Ho * Ho * (Cpad / 8);
  upsample_tokens_coords_bf16<float><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      (const float*)tok, ldt, bst, (__nv_bfloat16*)out, B, G, Ho, C, Cpad);
  G4R_LAUNCH_CHECK("upsample_tokens_coords_f32");
  return G4R_OK;
}

extern "C" int g4r_layernorm_ex(const void* x, long long ldx, int x_f32, const void* w, const void* b, void* out,
                                long long ldo, int out_f32, int M, int D, float eps, void* stream) {
  G4R_REQUIRE(x && w && b && out && M > 0 && D > 0 && D % 8 == 0 && D <= 8192 && ldx % 8 == 0 && ldo % 8 == 0,
              "layernorm_ex: bad arguments (D=%d)", D);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_f32) return out_f32 ? launch_ln_ex<float, float>(x, ldx, w, b, out, ldo, M, D, eps, st)
                            : launch_ln_ex<float, __nv_bfloat16>(x, ldx, w, b, out, ldo, M, D, eps, st);
  return out_f32 ? launch_ln_ex<__nv_bfloat16, float>(x, ldx, w, b, out, ldo, M, D, eps, st)
                 : launch_ln_ex<__nv_bfloat16, __nv_bfloat16>(x, ldx, w, b, out, ldo, M, D, eps, st);
}

extern "C" int g4r_rmsnorm_ex(const void* x, long long ldx, int x_f32, const void* w, void* out, long long ldo, int M,
                              int D, float eps, void* stream) {
  G4R_REQUIRE(x && w && out && M > 0 && D > 0 && D % 8 == 0 && D <= 8192 && ldx % 8 == 0 && ldo % 8 == 0,
              "rmsnorm_ex: bad arguments (D=%d)", D);
  cudaStream_t st = (cudaStream_t)stream;
  if (!x_f32) return launch_norm<true>(x, ldx, w, nullptr, out, ldo, M, D, eps, st);
  return launch_ln_ex<float, __nv_bfloat16, true>(x, ldx, w, nullptr, out, ldo, M, D, eps, st);
}

extern "C" int g4r_cast_f32_bf16(const void* x, long long ld, long long bst, void* out, int B, int rows_per_batch,
                                 int D, void* stream) {
  G4R_REQUIRE(x && out && B > 0 && rows_per_batch > 0 && D % 8 == 0 && ld % 4 == 0 && bst % 4 == 0, "cast_f32_bf16: bad arguments");
  const long long total = (long long)B * rows_per_batch * (D / 8);
  cast_rows_f32_bf16<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const float*)x, ld, bst, (__nv_bfloat16*)out, B,
                                                                            rows_per_batch, D);
  G4R_LAUNCH_CHECK("cast_f32_bf16");
  return G4R_OK;
}

extern "C" int g4r_fuse_gather_bf16(const void* own, const float* own_sc, const float* own_sh, int H,
                                    const void* top, const float* top_sc, const float* top_sh, int Ht,
                                    const void* down, const float* down_sc, const float* down_sh, int Hd,
                                    void* out, int B, int C, void* stream) {
  G4R_REQUIRE(own && top && down && out && B > 0 && C % 32 == 0 && H > 0 && Ht > 0 && Hd > 0, "fuse_gather: bad arguments");
  FuseSrc a{(const __nv_bfloat16*)own, own_sc, own_sh, H};
  FuseSrc t{(const __nv_bfloat16*)top, top_sc, top_sh, Ht};
  FuseSrc d{(const __nv_bfloat16*)down, down_sc, down_sh, Hd};
  const int nvec = C / 8;
  G4R_REQUIRE(nvec <= 1024, "fuse_gather: C too large");
  const int threads = nvec >= 256 ? nvec : (256 / nvec) * nvec;  // whole pixels per block
  const long long npix = (long long)B * H * H;
  const int ppb = threads / nvec;
  long long blocks = (npix + ppb - 1) / ppb;
  const long long cap = (long long)num_sms() * 32;
  if (blocks > cap) blocks = cap;
  fuse_gather_bf16<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(a, t, d, (__nv_bfloat16*)out, B, C);
  G4R_LAUNCH_CHECK("fuse_gather");
  return G4R_OK;
}

#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_fuse_gather_bwd(const void* d_own, int H, const void* dn0, int Hdn0, const void* dn1, int Hdn1,
                                   const void* tp0, int Htp0, const void* tp1, int Htp1, float* out, int B, int C,
                                   void* stream) {
  G4R_REQUIRE(d_own && out && B > 0 && C % 32 == 0 && H > 1, "fuse_gather_bwd: bad arguments");
  FuseGrad o{(const __nv_bfloat16*)d_own, H}, a{(const __nv_bfloat16*)dn0, Hdn0}, b{(const __nv_bfloat16*)dn1, Hdn1};
  FuseGrad c{(const __nv_bfloat16*)tp0, Htp0}, d{(const __nv_bfloat16*)tp1, Htp1};
  const int nvec = C / 8;
  G4R_REQUIRE(nvec <= 1024, "fuse_gather_bwd: C too large");
  const int threads = nvec >= 256 ? nvec : (256 / nvec) * nvec;
  const long long npix = (long long)B * H * H;
  const int ppb = threads / nvec;
  long long blocks = (npix + ppb - 1) / ppb;
  const long long cap = (long long)num_sms() * 32;
  if (blocks > cap) blocks = cap;
  fuse_gather_bwd<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(o, a, b, c, d, out, B, C);
  G4R_LAUNCH_CHECK("fuse_gather_bwd");
  return G4R_OK;
}
#endif

extern "C" int g4r_gn_finalize(const float* stats, const void* gamma, const void* beta, float* scale,
                               float* shift, int B, int C, int groups, int slots, float count, float eps,
                               void* stream) {
  G4R_REQUIRE(stats && gamma && beta && scale && shift && B > 0 && C > 0 && groups > 0 && C % groups == 0 && slots > 0, "gn_finalize: bad arguments");
  gn_finalize<<<(B * groups + 7) / 8, 256, 0, (cudaStream_t)stream>>>(stats, (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta,
                                                                   scale, shift, B, C, groups, slots, count, eps);
  G4R_LAUNCH_CHECK("gn_finalize");
  return G4R_OK;
}

extern "C" int g4r_pos_embed_mlp(const float* boxes, const void* w0, const void* b0, const void* g2,
                                 const void* be2, const void* w3, const void* b3, const void* g5,
                                 const void* be5, float* out, int K, float eps, void* stream) {
  G4R_REQUIRE(boxes && w0 && b0 && g2 && be2 && w3 && b3 && g5 && be5 && out && K > 0, "pos_embed_mlp: bad arguments");
  pos_embed_mlp<<<K, 256, 0, (cudaStream_t)stream>>>(boxes, (const __nv_bfloat16*)w0, (const __nv_bfloat16*)b0,
      (const __nv_bfloat16*)g2, (const __nv_bfloat16*)be2, (const __nv_bfloat16*)w3, (const __nv_bfloat16*)b3,
      (const __nv_bfloat16*)g5, (const __nv_bfloat16*)be5, out, eps);
  G4R_LAUNCH_CHECK("pos_embed_mlp");
  return G4R_OK;
}

#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_pos_embed_mlp_grad_size(void) { return kPosSlab; }

#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_pos_embed_mlp_bwd(const float* boxes, const void* w0, const void* b0, const void* g2, const void* be2,
                                     const void* w3, const void* b3, const void* g5, const void* dout, long long ldd,
                                     float* grads, float* slabs, int K, float eps, void* stream) {
  G4R_REQUIRE(boxes && w0 && b0 && g2 && be2 && w3 && b3 && g5 && dout && grads && slabs && K > 0, "pos_embed_mlp_bwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  pos_embed_mlp_bwd<<<K, 256, 0, st>>>(boxes, (const __nv_bfloat16*)w0, (const __nv_bfloat16*)b0, (const __nv_bfloat16*)g2,
      (const __nv_bfloat16*)be2, (const __nv_bfloat16*)w3, (const __nv_bfloat16*)b3, (const __nv_bfloat16*)g5,
      (const __nv_bfloat16*)dout, ldd, slabs, eps);
  G4R_LAUNCH_CHECK("pos_embed_mlp_bwd");
  pos_slab_reduce<<<(kPosSlab + 255) / 256, 256, 0, st>>>(slabs, K, grads);
  G4R_LAUNCH_CHECK("pos_slab_reduce");
  return G4R_OK;
}
#endif
#endif

// out = relu(z * scale[b, c] + shift[b, c]) on an NHWC bf16 map: applies a pending GroupNorm affine + ReLU
// (mmcv ConvModule's norm + activation, conv_module.py:196-208) where a caller needs the activated map itself
// (MLVLFuseModule.forward returns it, gpt4roi/models/layers.py:182-195; inside the engine the affine stays
// folded into the consumer's taps instead).  8 channels (16 bytes) per thread.
__global__ void __launch_bounds__(256)
affine_relu_nhwc(const __nv_bfloat16* __restrict__ z, const float* __restrict__ scale, const float* __restrict__ shift,
                 __nv_bfloat16* __restrict__ out, long long pix_per_img, int C, long long total_vec) {
  const int nvec = C >> 3;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total_vec; i += (long long)gridDim.x * 256) {
    const int v = (int)(i % nvec);
    const long long b = (i / nvec) / pix_per_img;
    float f[8];
    load16<__nv_bfloat16>(z + i * 8, f);
    const float* sc = scale + b * C + v * 8;
    const float* sh = shift + b * C + v * 8;
#pragma unroll
    for (int j = 0; j < 8; j++) f[j] = fmaxf(fmaf(f[j], sc[j], sh[j]), 0.f);
    store16<__nv_bfloat16>(out + i * 8, f);
  }
}

extern "C" int g4r_affine_relu_nhwc_bf16(const void* z, const float* scale, const float* shift, void* out, int B,
                                         long long pix_per_img, int C, void* stream) {
  G4R_REQUIRE(z && scale && shift && out && B > 0 && pix_per_img > 0 && C > 0 && C % 8 == 0, "affine_relu_nhwc: bad arguments");
  const long long total = (long long)B * pix_per_img * (C / 8);
  long long grid = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (grid > cap) grid = cap;
  affine_relu_nhwc<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)z, scale, shift, (__nv_bfloat16*)out,
                                                                    pix_per_img, C, total);
  G4R_LAUNCH_CHECK("affine_relu_nhwc");
  return G4R_OK;
}

extern "C" int g4r_add_bias_pos_cast(const float* acc, int splits, const void* bias, const float* pos, void* out,
                                     int K, int D, void* stream) {
  G4R_REQUIRE(acc && bias && pos && out && K > 0 && D > 0 && splits >= 1, "add_bias_pos_cast: bad arguments");
  add_bias_pos_cast<<<(K * D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(acc, splits, (const __nv_bfloat16*)bias, pos, (__nv_bfloat16*)out, K, D);
  G4R_LAUNCH_CHECK("add_bias_pos_cast");
  return G4R_OK;
}
