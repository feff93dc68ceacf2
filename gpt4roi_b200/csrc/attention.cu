// attention.cu -- fused softmax(Q K^T * scale [+ causal mask]) V for the ViT (non-causal, d=64) and
// the LLaMA prefill (causal, d=128).  Replaces the eager attention the reference gets from
// transformers (CLIP: modeling_clip.py `eager_attention_forward`; LLaMA: modeling_llama.py:199-222),
// i.e. matmul -> *scale -> (+mask) -> softmax(fp32) -> cast -> matmul, without materialising the
// [B,H,L,L] score tensor.
//
// Round-1 implementation note (DESIGN.md "attention"): attention is ~1.5 % of the path's FLOPs
// (SURVEY.md App. B), so this first version uses warp-level mma.sync.m16n8k16 tiles (legacy tensor
// path, HMMA) with cp.async double buffering; the tcgen05/TMEM version is scheduled after the GEMMs.
// Numerics: QK^T accumulates in fp32 and the scaled scores stay fp32 through the softmax (the
// reference rounds them to bf16 twice -- after the matmul and after *scale -- which only adds
// noise); P is cast to bf16 before the PV product like the reference, the output is rounded once.
#include "common.cuh"
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

constexpr int kBM = 64;   // query rows per CTA (4 warps x 16)
constexpr int kBN = 64;   // keys per iteration
constexpr int kAttnThreads = 128;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32." G4R_ACT_PTX "." G4R_ACT_PTX ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// swizzled element offset of 16-byte chunk `chunk` of row `row` in a [rows][D] bf16 tile
template <int D>
__device__ __forceinline__ int swz(int row, int chunk) { return row * D + ((chunk ^ (row & 7)) << 3); }

template <int D>
__device__ __forceinline__ void load_tile(__nv_bfloat16* s, const __nv_bfloat16* g, long long ld, int row0,
                                          int L) {
  constexpr int CPR = D / 8;  // 16-byte chunks per row
  for (int i = threadIdx.x; i < kBN * CPR; i += kAttnThreads) {
    const int r = i / CPR, c = i % CPR;
    int gr = row0 + r;
    if (gr > L - 1) gr = L - 1;  // clamp; out-of-range keys are masked, out-of-range queries not stored
    cp_async16(smem_addr(s + swz<D>(r, c)), g + (long long)gr * ld + c * 8);
  }
}

template <int D, bool CAUSAL>
__global__ void __launch_bounds__(kAttnThreads)
flash_attn_fwd(const __nv_bfloat16* __restrict__ Q, const __nv_bfloat16* __restrict__ K,
               const __nv_bfloat16* __restrict__ V, __nv_bfloat16* __restrict__ O, long long ld, long long bs,
               long long ldo, long long bso, int L, float scale, const int* __restrict__ seqlens) {
  extern __shared__ __align__(128) uint8_t smem_attn[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* sK = sQ + kBM * D;       // 2 buffers
  __nv_bfloat16* sV = sK + 2 * kBN * D;   // 2 buffers

  const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = qb * kBM;
  const __nv_bfloat16* gq = Q + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gk = K + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gv = V + (long long)b * bs + (long long)h * D;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;

  // right-padded batches: keys >= seqlens[b] are masked (attention_mask of data_modules.py:33-44);
  // rows >= seqlens[b] produce don't-care values (their labels are -100 in the reference).
  const int Lk = seqlens ? min(max(seqlens[b], 1), L) : L;
  const int n_kv = CAUSAL ? min((Lk + kBN - 1) / kBN, (q0 + kBM + kBN - 1) / kBN) : (Lk + kBN - 1) / kBN;

  load_tile<D>(sQ, gq, ld, q0, L);
  load_tile<D>(sK, gk, ld, 0, L);
  load_tile<D>(sV, gv, ld, 0, L);
  cp_async_commit();

  uint32_t qf[D / 16][4];
  float o[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; i++) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  constexpr float kLog2e = 1.4426950408889634f;

  for (int kb = 0; kb < n_kv; kb++) {
    const int buf = kb & 1;
    if (kb + 1 < n_kv) {
      load_tile<D>(sK + (buf ^ 1) * kBN * D, gk, ld, (kb + 1) * kBN, L);
      load_tile<D>(sV + (buf ^ 1) * kBN * D, gv, ld, (kb + 1) * kBN, L);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (kb == 0) {
      // Q fragments (A operand) for this warp's 16 rows, all k-steps
#pragma unroll
      for (int kk = 0; kk < D / 16; kk++) {
        const int row = warp * 16 + (lane & 15), chunk = kk * 2 + (lane >> 4);
        ldsm_x4(smem_addr(sQ + swz<D>(row, chunk)), qf[kk][0], qf[kk][1], qf[kk][2], qf[kk][3]);
      }
    }
    const __nv_bfloat16* cK = sK + buf * kBN * D;
    const __nv_bfloat16* cV = sV + buf * kBN * D;

    float s[kBN / 8][4];
#pragma unroll
    for (int i = 0; i < kBN / 8; i++) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < D / 16; kk++) {
#pragma unroll
      for (int n2 = 0; n2 < kBN / 16; n2++) {
        uint32_t b0, b1, b2, b3;
        const int row = n2 * 16 + (lane & 7) + ((lane >> 4) << 3);
        const int chunk = kk * 2 + ((lane >> 3) & 1);
        ldsm_x4(smem_addr(cK + swz<D>(row, chunk)), b0, b1, b2, b3);
        mma_bf16(s[2 * n2], qf[kk], b0, b1);
        mma_bf16(s[2 * n2 + 1], qf[kk], b2, b3);
      }
    }
    // online softmax in fp32 on the raw fp32 scores (scale folded into the exp2 argument).
    // Only the diagonal block (causal) and the tail block (keys >= L) need masking.
    const int key0 = kb * kBN;
    const int qrow0 = q0 + warp * 16;
    if (key0 + kBN > Lk || (CAUSAL && key0 + kBN - 1 > qrow0)) {
#pragma unroll
      for (int nt = 0; nt < kBN / 8; nt++) {
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int key = key0 + nt * 8 + 2 * t + (e & 1);
          const int qrow = qrow0 + g + ((e >> 1) << 3);
          if (key >= Lk || (CAUSAL && key > qrow)) s[nt][e] = -INFINITY;
        }
      }
    }
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < kBN / 8; nt++) {
      mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
    }
    const float c = scale * kLog2e;
    float alpha[2], mc[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m_run[r], mx[r]);
      const float msub = m_new == -INFINITY ? 0.f : m_new;
      alpha[r] = exp2f((m_run[r] - msub) * c);  // m_run = -inf -> 0
      mc[r] = msub * c;
      m_run[r] = m_new;
      l_run[r] *= alpha[r];
    }
    uint32_t pf[kBN / 16][4];
#pragma unroll
    for (int nt = 0; nt < kBN / 8; nt++) {
      float p[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        p[e] = exp2f(fmaf(s[nt][e], c, -mc[e >> 1]));
        l_run[e >> 1] += p[e];
      }
      pf[nt >> 1][(nt & 1) * 2] = pack_bf16(p[0], p[1]);
      pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16(p[2], p[3]);
    }
#pragma unroll
    for (int i = 0; i < D / 8; i++) {
      o[i][0] *= alpha[0]; o[i][1] *= alpha[0];
      o[i][2] *= alpha[1]; o[i][3] *= alpha[1];
    }
#pragma unroll
    for (int kt = 0; kt < kBN / 16; kt++) {
#pragma unroll
      for (int d2 = 0; d2 < D / 16; d2++) {
        uint32_t b0, b1, b2, b3;
        const int row = kt * 16 + (lane & 7) + (((lane >> 3) & 1) << 3);
        const int chunk = d2 * 2 + (lane >> 4);
        ldsm_x4_t(smem_addr(cV + swz<D>(row, chunk)), b0, b1, b2, b3);
        mma_bf16(o[2 * d2], pf[kt], b0, b1);
        mma_bf16(o[2 * d2 + 1], pf[kt], b2, b3);
      }
    }
    __syncthreads();  // everyone done with buf before it is refilled two iterations later
  }

#pragma unroll
  for (int r = 0; r < 2; r++) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  __nv_bfloat16* go = O + (long long)b * bso + (long long)h * D;
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const int qrow = q0 + warp * 16 + g + r * 8;
    if (qrow >= L) continue;
    const float inv = 1.f / l_run[r];
#pragma unroll
    for (int i = 0; i < D / 8; i++) {
      const uint32_t pk = pack_bf16(o[i][2 * r] * inv, o[i][2 * r + 1] * inv);
      *reinterpret_cast<uint32_t*>(go + (long long)qrow * ldo + i * 8 + 2 * t) = pk;
    }
  }
}

template <int D, bool CAUSAL>
static int launch_attn(const void* q, const void* k, const void* v, void* o, long long ld, long long bs,
                       long long ldo, long long bso, int B, int H, int L, float scale, const int* seqlens,
                       cudaStream_t st) {
  const int smem = (kBM * D + 4 * kBN * D) * 2;
  static bool set = false;
  auto kern = flash_attn_fwd<D, CAUSAL>;
  if (!set) {
    G4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    set = true;
  }
  dim3 grid((L + kBM - 1) / kBM, H, B);
  kern<<<grid, kAttnThreads, smem, st>>>((const __nv_bfloat16*)q, (const __nv_bfloat16*)k,
                                          (const __nv_bfloat16*)v, (__nv_bfloat16*)o, ld, bs, ldo, bso, L, scale, seqlens);
  G4R_LAUNCH_CHECK("flash_attn_fwd");
  return G4R_OK;
}

}  // namespace g4r

using namespace G4R_NS;

extern "C" int g4r_attention_bf16(const void* q, const void* k, const void* v, void* out, long long ld,
                                  long long bs, long long ldo, long long bso, int B, int H, int L,
                                  int head_dim, int causal, float scale, const int* seqlens, void* stream) {
  G4R_REQUIRE(q && k && v && out && B > 0 && H > 0 && L > 0, "attention: bad arguments");
  G4R_REQUIRE(head_dim == 64 || head_dim == 128, "attention: head_dim %d (64 or 128)", head_dim);
  G4R_REQUIRE(ld % 8 == 0 && bs % 8 == 0 && ldo % 2 == 0 && bso % 2 == 0, "attention: strides must keep 16-byte row alignment");
  G4R_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v) & 15) == 0 && ((uintptr_t)out & 3) == 0, "attention: misaligned pointers");
  cudaStream_t st = (cudaStream_t)stream;
  if (head_dim == 64) {
    return causal ? launch_attn<64, true>(q, k, v, out, ld, bs, ldo, bso, B, H, L, scale, seqlens, st)
                  : launch_attn<64, false>(q, k, v, out, ld, bs, ldo, bso, B, H, L, scale, seqlens, st);
  }
  return causal ? launch_attn<128, true>(q, k, v, out, ld, bs, ldo, bso, B, H, L, scale, seqlens, st)
                : launch_attn<128, false>(q, k, v, out, ld, bs, ldo, bso, B, H, L, scale, seqlens, st);
}
