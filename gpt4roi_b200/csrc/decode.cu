// decode.cu -- KV-cache append and single-query attention for the decode loop behind generate()
// (SURVEY.md 8(f1)): after the region-token prefill, every further step is plain LLaMA with one new
// token per sample (the vision/SPI branch is skipped, gpt4roi/models/spi_llava.py:47-48;
// llava/model/llava.py:263-283 prepare_inputs_for_generation; gpt4roi/app.py:293-300).
// Both kernels are HBM-bound: the step streams the whole KV cache of the batch once.
#include "common.cuh"
#include <cooperative_groups.h>
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

// rows [B*Ln, 3*HD] packed (q|k|v) -> caches [B, Lmax, HD] at positions pos0 .. pos0+Ln-1
__global__ void __launch_bounds__(256)
kv_append_bf16(const __nv_bfloat16* __restrict__ qkv, long long ld, __nv_bfloat16* __restrict__ kc,
               __nv_bfloat16* __restrict__ vc, int B, int Ln, int pos0, const int* __restrict__ pos_dev, int Lmax,
               int HD) {
  if (pos_dev) pos0 = *pos_dev;
  const int nvec = HD >> 3;
  const long long total = (long long)B * Ln * nvec * 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    const int which = (int)((i / nvec) & 1);  // 0 = k, 1 = v
    const long long r = i / (2LL * nvec);     // row in [0, B*Ln)
    const int t = (int)(r % Ln), b = (int)(r / Ln);
    const uint4 val = *reinterpret_cast<const uint4*>(qkv + r * ld + (long long)(1 + which) * HD + v * 8);
    __nv_bfloat16* dst = (which ? vc : kc) + ((long long)b * Lmax + pos0 + t) * HD + v * 8;
    *reinterpret_cast<uint4*>(dst) = val;
  }
}

// Single-query attention over the KV cache: out = softmax(q . K^T * scale) V for the first kv_len
// cached positions.  Grid (H, B, S) with a thread-block cluster of S CTAs along z: each CTA of the
// cluster owns a contiguous slice of the keys (split-KV), and the softmax statistics and the partial
// outputs are combined through distributed shared memory -- no workspace, no atomics, and a fixed
// summation order (bitwise reproducible).  S is chosen so that even batch 1 (32 heads) fills the GPU.
// 256 threads; a half-warp owns one key/value row (16 lanes x 16 bytes = the 256-byte row, coalesced).
// Rounding as the reference's eager attention: fp32 softmax, probabilities cast to bf16 before P.V.
template <int D>
__global__ void __launch_bounds__(256)
decode_attention_bf16(const __nv_bfloat16* q, long long ldq, const __nv_bfloat16* kc, const __nv_bfloat16* vc,
                      __nv_bfloat16* out, long long ldo, int H, int kv_len, const int* __restrict__ pos_dev, int Lmax,
                      float scale, int per_max) {
  // Programmatic dependent launch (common.cuh): q and the newest K/V row come from the q|k|v GEMM that precedes this
  // kernel in the decode step, so there is nothing to fetch ahead; the launch itself and the prologue overlap its tail.
  // q / kc / vc carry no __restrict__: their loads must stay on the coherent path.
  pdl_sync();
  static_assert(D == 128 || D == 64, "head_dim");
  constexpr int LPR = D / 8;          // lanes per row (16 or 8)
  constexpr int RPW = 32 / LPR;       // rows per warp instruction (2 or 4)
  constexpr int GROUPS = 8 * RPW;     // row groups per CTA (16 or 32)
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  if (pos_dev) kv_len = *pos_dev + 1;
  extern __shared__ float sm[];
  float* sc = sm;                       // [per_max] scores / probabilities of this CTA's slice
  float* part = sm + per_max;           // [GROUPS][D] partial outputs, then [D] CTA total in part[0..D)
  __shared__ float red[8];
  __shared__ float cl_max, cl_sum;      // this CTA's slice statistics, read by the cluster peers
  const int h = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int sub = lane % LPR, grp = warp * RPW + lane / LPR;
  const int HD = H * D;
  const int per = (kv_len + S - 1) / S;
  const int k0 = rank * per;
  const int n_loc = max(0, min(kv_len, k0 + per) - k0);

  float qf[8];
  {
    const uint4 raw = *reinterpret_cast<const uint4*>(q + (long long)b * ldq + (long long)h * D + sub * 8);
    const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const float2 f = __bfloat1622float2(hh[j]);
      qf[2 * j] = f.x * scale;
      qf[2 * j + 1] = f.y * scale;
    }
  }
  // ---- phase 1: scores of the slice
  const __nv_bfloat16* kb = kc + ((long long)b * Lmax + k0) * HD + (long long)h * D + sub * 8;
  float mx = -INFINITY;
  for (int base = 0; base < n_loc; base += GROUPS * 4) {
    uint4 raw[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int key = base + u * GROUPS + grp;
      raw[u] = key < n_loc ? *reinterpret_cast<const uint4*>(kb + (long long)key * HD) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&raw[u]);
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const float2 f = __bfloat1622float2(hh[j]);
        acc += f.x * qf[2 * j] + f.y * qf[2 * j + 1];
      }
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      const int key = base + u * GROUPS + grp;
      if (key < n_loc) {
        if (sub == 0) sc[key] = acc;
        mx = fmaxf(mx, acc);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (tid == 0) {
    float m = red[0];
#pragma unroll
    for (int w = 1; w < 8; w++) m = fmaxf(m, red[w]);
    cl_max = m;
  }
  cluster.sync();
  float gmax = -INFINITY;
  for (int r = 0; r < S; r++) gmax = fmaxf(gmax, *cluster.map_shared_rank(&cl_max, r));
  float sum = 0.f;
  for (int key = tid; key < n_loc; key += 256) {
    const float p = __expf(sc[key] - gmax);
    sc[key] = p;
    sum += p;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) t += red[w];
    cl_sum = t;
  }
  cluster.sync();
  float gsum = 0.f;
  for (int r = 0; r < S; r++) gsum += *cluster.map_shared_rank(&cl_sum, r);
  const float inv = 1.f / gsum;
  // ---- phase 2: partial P.V of the slice (probabilities rounded to bf16 like P.to(q.dtype))
  const __nv_bfloat16* vb = vc + ((long long)b * Lmax + k0) * HD + (long long)h * D + sub * 8;
  float o8[8];
#pragma unroll
  for (int j = 0; j < 8; j++) o8[j] = 0.f;
  for (int base = 0; base < n_loc; base += GROUPS * 4) {
    uint4 raw[4];
    float pk[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int key = base + u * GROUPS + grp;
      const bool ok = key < n_loc;
      raw[u] = ok ? *reinterpret_cast<const uint4*>(vb + (long long)key * HD) : make_uint4(0, 0, 0, 0);
      pk[u] = ok ? __bfloat162float(__float2bfloat16_rn(sc[key] * inv)) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&raw[u]);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const float2 f = __bfloat1622float2(hh[j]);
        o8[2 * j] += pk[u] * f.x;
        o8[2 * j + 1] += pk[u] * f.y;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) part[grp * D + sub * 8 + j] = o8[j];
  __syncthreads();
  float tot = 0.f;
  if (tid < D) {
#pragma unroll 4
    for (int g2 = 0; g2 < GROUPS; g2++) tot += part[g2 * D + tid];
  }
  __syncthreads();
  if (tid < D) part[tid] = tot;   // CTA total, visible to rank 0 after the cluster barrier
  cluster.sync();
  if (rank == 0 && tid < D) {
    float v = 0.f;
    for (int r = 0; r < S; r++) v += cluster.map_shared_rank(part, r)[tid];
    out[(long long)b * ldo + (long long)h * D + tid] = __float2bfloat16_rn(v);
  }
  cluster.sync();   // keep every CTA's shared memory alive until rank 0 has read it
}

}  // namespace g4r

using namespace G4R_NS;

extern "C" int g4r_kv_append_bf16(const void* qkv, long long ld, void* kcache, void* vcache, int B, int Ln,
                                  int pos0, const int* pos_dev, int Lmax, int HD, void* stream) {
  G4R_REQUIRE(qkv && kcache && vcache && B > 0 && Ln > 0 && pos0 >= 0 && pos0 + Ln <= Lmax && HD % 8 == 0 && ld % 8 == 0,
              "kv_append: bad arguments (pos0=%d Ln=%d Lmax=%d)", pos0, Ln, Lmax);
  const long long total = (long long)B * Ln * (HD / 8) * 2;
  long long grid = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (grid > cap) grid = cap;
  kv_append_bf16<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)qkv, ld, (__nv_bfloat16*)kcache,
                                                                  (__nv_bfloat16*)vcache, B, Ln, pos0, pos_dev, Lmax, HD);
  G4R_LAUNCH_CHECK("kv_append");
  return G4R_OK;
}

template <int D>
static int launch_decode_attention(const void* q, long long ldq, const void* kcache, const void* vcache, void* out,
                                   long long ldo, int B, int H, int kv_len, const int* pos_dev, int Lmax,
                                   float scale, cudaStream_t st) {
  // split-KV factor: enough CTAs for >= 2 per SM, slices of >= 64 keys, cluster size <= 8 (portable)
  int S = 1;
  while (S < 8 && H * B * S < 2 * num_sms() && kv_len / (2 * S) >= 64) S *= 2;
  const int per_max = (kv_len + S - 1) / S;
  const int groups = 8 * (32 / (D / 8));
  const size_t smem = ((size_t)per_max + (size_t)groups * D) * sizeof(float);
  G4R_REQUIRE(smem <= 200 * 1024, "decode_attention: kv_len %d too long for the shared-memory score buffer", kv_len);
  static bool set = false;
  if (!set) {
    G4R_CUDA(cudaFuncSetAttribute(decode_attention_bf16<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    set = true;
  }
  G4R_CUDA(launch_pdl(decode_attention_bf16<D>, dim3(H, B, S), dim3(256), smem, st, dim3(1, 1, S),
                      (const __nv_bfloat16*)q, ldq, (const __nv_bfloat16*)kcache, (const __nv_bfloat16*)vcache,
                      (__nv_bfloat16*)out, ldo, H, kv_len, pos_dev, Lmax, scale, per_max));
  return G4R_OK;
}

extern "C" int g4r_decode_attention_bf16(const void* q, long long ldq, const void* kcache, const void* vcache,
                                         void* out, long long ldo, int B, int H, int head_dim, int kv_len,
                                         const int* pos_dev, int Lmax, float scale, void* stream) {
  G4R_REQUIRE(q && kcache && vcache && out && B > 0 && H > 0 && kv_len > 0 && kv_len <= Lmax, "decode_attention: bad arguments");
  G4R_REQUIRE(head_dim == 64 || head_dim == 128, "decode_attention: head_dim %d", head_dim);
  G4R_REQUIRE(ldq % 8 == 0 && ((uintptr_t)q & 15) == 0, "decode_attention: q rows must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (head_dim == 128)
    return launch_decode_attention<128>(q, ldq, kcache, vcache, out, ldo, B, H, kv_len, pos_dev, Lmax, scale, st);
  return launch_decode_attention<64>(q, ldq, kcache, vcache, out, ldo, B, H, kv_len, pos_dev, Lmax, scale, st);
}
