// attention_bwd.cu -- backward of the fused causal attention for the training step (SURVEY.md 8(a) row 14;
// the reference gets it from autograd through transformers' eager LLaMA attention, modeling_llama.py:199-222).
//
// Inputs: packed qkv rows [B*L, 3*H*D] (after RoPE), the forward output O, its log-sum-exp rows
// (g4r_attention_tc_lse_bf16) and dO.  Output: packed dqkv rows (dQ | dK | dV), bf16.
// Two kernels, both recomputing S = Q K^T from the saved LSE (no [L, L] tensor is ever stored) and both
// free of atomics, so gradients are bitwise reproducible:
//   attn_bwd_dq : one CTA per 64-query block, loops over the key blocks it can see:
//                 P = exp(S*scale - lse), dP = dO V^T, dS = P o (dP - delta), dQ += dS K
//   attn_bwd_dkv: one CTA per 64-key block, loops over the query blocks that see it:
//                 dV += P^T dO, dK += dS^T Q
// delta = rowsum(dO o O) comes from attn_bwd_delta.  Warp-level mma.sync m16n8k16 (bf16 in, fp32 accumulate)
// with cp.async double buffering, like the first forward kernel (attention.cu); P and dS are rounded to bf16
// before their second matmul exactly like the forward rounds P.
#include "common.cuh"

namespace g4r {
namespace {

constexpr int kB = 64;          // rows per block, queries and keys alike
constexpr int kThr = 128;       // 4 warps x 16 rows

__device__ __forceinline__ uint32_t saddr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pk(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <int D> __device__ __forceinline__ int swz(int row, int chunk) { return row * D + ((chunk ^ (row & 7)) << 3); }

// [kB rows][D] bf16 tile, rows row0.. of a strided matrix, clamped to L-1 (callers mask / zero what is out of range)
template <int D>
__device__ __forceinline__ void load_tile(__nv_bfloat16* s, const __nv_bfloat16* g, long long ld, int row0, int L) {
  constexpr int CPR = D / 8;
  for (int i = threadIdx.x; i < kB * CPR; i += kThr) {
    const int r = i / CPR, c = i % CPR;
    int gr = row0 + r;
    if (gr > L - 1) gr = L - 1;
    cp16(saddr(s + swz<D>(r, c)), g + (long long)gr * ld + c * 8);
  }
}

// A operand: 16 rows (row0..) x 16 k (k-step kk) of a row-major tile
template <int D>
__device__ __forceinline__ void frag_a(const __nv_bfloat16* s, int row0, int kk, int lane, uint32_t (&a)[4]) {
  ldsm4(saddr(s + swz<D>(row0 + (lane & 15), kk * 2 + (lane >> 4))), a[0], a[1], a[2], a[3]);
}
// B operand, tile rows are the n index (contraction along the row): n-rows n2*16.., k-step kk -> two n8 tiles
template <int D>
__device__ __forceinline__ void frag_b_rows_n(const __nv_bfloat16* s, int n2, int kk, int lane, uint32_t (&b)[4]) {
  ldsm4(saddr(s + swz<D>(n2 * 16 + (lane & 7) + ((lane >> 4) << 3), kk * 2 + ((lane >> 3) & 1))), b[0], b[1], b[2], b[3]);
}
// B operand, tile rows are the k index (n along the row): k-rows kt*16.., columns d2*16.. -> two n8 tiles
template <int D>
__device__ __forceinline__ void frag_b_rows_k(const __nv_bfloat16* s, int kt, int d2, int lane, uint32_t (&b)[4]) {
  ldsm4t(saddr(s + swz<D>(kt * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), d2 * 2 + (lane >> 4))), b[0], b[1], b[2], b[3]);
}

}  // namespace

// delta[b, h, q] = sum_d dO[b, q, h, d] * O[b, q, h, d]     (one warp per (b, q, h))
template <int D>
__global__ void __launch_bounds__(256)
attn_bwd_delta(const __nv_bfloat16* __restrict__ O, const __nv_bfloat16* __restrict__ dO, long long ldo, long long bso,
               float* __restrict__ delta, int B, int H, int L) {
  const long long w = (blockIdx.x * 256LL + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= (long long)B * L * H) return;
  const int h = (int)(w % H);
  const long long bq = w / H;
  const int q = (int)(bq % L), b = (int)(bq / L);
  const long long off = (long long)b * bso + (long long)q * ldo + (long long)h * D;
  float acc = 0.f;
  for (int d = lane * 2; d < D; d += 64) {
    const float2 o = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(O + off + d));
    const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(dO + off + d));
    acc += o.x * g.x + o.y * g.y;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  if (lane == 0) delta[((long long)b * H + h) * L + q] = acc;
}

template <int D, bool CAUSAL>
__global__ void __launch_bounds__(kThr)
attn_bwd_dq(const __nv_bfloat16* __restrict__ Q, const __nv_bfloat16* __restrict__ K, const __nv_bfloat16* __restrict__ V,
            const __nv_bfloat16* __restrict__ dO, const float* __restrict__ lse, const float* __restrict__ delta,
            __nv_bfloat16* __restrict__ dQ, long long ld, long long bs, long long ldo, long long bso, long long ldg,
            long long bsg, int L, float scale) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  __nv_bfloat16* sdO = sQ + kB * D;
  __nv_bfloat16* sK = sdO + kB * D;      // 2 buffers
  __nv_bfloat16* sV = sK + 2 * kB * D;   // 2 buffers
  const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z, H = gridDim.y;
  const int q0 = qb * kB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const __nv_bfloat16* gq = Q + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gk = K + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gv = V + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gdo = dO + (long long)b * bso + (long long)h * D;
  const int n_kv = CAUSAL ? min((L + kB - 1) / kB, qb + 1) : (L + kB - 1) / kB;

  load_tile<D>(sQ, gq, ld, q0, L);
  load_tile<D>(sdO, gdo, ldo, q0, L);
  load_tile<D>(sK, gk, ld, 0, L);
  load_tile<D>(sV, gv, ld, 0, L);
  cp_commit();

  constexpr float kLog2e = 1.4426950408889634f;
  const float c = scale * kLog2e;
  float lse2[2], dl[2];
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const int qrow = min(q0 + warp * 16 + g + r * 8, L - 1);
    lse2[r] = lse[((long long)b * H + h) * L + qrow] * kLog2e;
    dl[r] = delta[((long long)b * H + h) * L + qrow];
  }
  uint32_t qf[D / 16][4], dof[D / 16][4];
  float dq[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; i++) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;

  for (int kb = 0; kb < n_kv; kb++) {
    const int buf = kb & 1;
    if (kb + 1 < n_kv) {
      load_tile<D>(sK + (buf ^ 1) * kB * D, gk, ld, (kb + 1) * kB, L);
      load_tile<D>(sV + (buf ^ 1) * kB * D, gv, ld, (kb + 1) * kB, L);
      cp_commit();
      cp_wait<1>();
    } else {
      cp_wait<0>();
    }
    __syncthreads();
    if (kb == 0) {
#pragma unroll
      for (int kk = 0; kk < D / 16; kk++) {
        frag_a<D>(sQ, warp * 16, kk, lane, qf[kk]);
        frag_a<D>(sdO, warp * 16, kk, lane, dof[kk]);
      }
    }
    const __nv_bfloat16* cK = sK + buf * kB * D;
    const __nv_bfloat16* cV = sV + buf * kB * D;
    float s[kB / 8][4], dp[kB / 8][4];
#pragma unroll
    for (int i = 0; i < kB / 8; i++) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; dp[i][0] = dp[i][1] = dp[i][2] = dp[i][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < D / 16; kk++) {
#pragma unroll
      for (int n2 = 0; n2 < kB / 16; n2++) {
        uint32_t bk[4], bv[4];
        frag_b_rows_n<D>(cK, n2, kk, lane, bk);
        mma(s[2 * n2], qf[kk], bk[0], bk[1]);
        mma(s[2 * n2 + 1], qf[kk], bk[2], bk[3]);
        frag_b_rows_n<D>(cV, n2, kk, lane, bv);
        mma(dp[2 * n2], dof[kk], bv[0], bv[1]);
        mma(dp[2 * n2 + 1], dof[kk], bv[2], bv[3]);
      }
    }
    const int key0 = kb * kB, qrow0 = q0 + warp * 16;
    const bool edge = key0 + kB > L || (CAUSAL && key0 + kB - 1 > qrow0);
    uint32_t dsf[kB / 16][4];
#pragma unroll
    for (int nt = 0; nt < kB / 8; nt++) {
      float ds[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int r = e >> 1;
        float p = exp2f(fmaf(s[nt][e], c, -lse2[r]));
        if (edge) {
          const int key = key0 + nt * 8 + 2 * t + (e & 1);
          const int qrow = qrow0 + g + r * 8;
          if (key >= L || (CAUSAL && key > qrow)) p = 0.f;
        }
        ds[e] = p * (dp[nt][e] - dl[r]);
      }
      dsf[nt >> 1][(nt & 1) * 2] = pk(ds[0], ds[1]);
      dsf[nt >> 1][(nt & 1) * 2 + 1] = pk(ds[2], ds[3]);
    }
#pragma unroll
    for (int kt = 0; kt < kB / 16; kt++) {
#pragma unroll
      for (int d2 = 0; d2 < D / 16; d2++) {
        uint32_t bk[4];
        frag_b_rows_k<D>(cK, kt, d2, lane, bk);
        mma(dq[2 * d2], dsf[kt], bk[0], bk[1]);
        mma(dq[2 * d2 + 1], dsf[kt], bk[2], bk[3]);
      }
    }
    __syncthreads();
  }
  __nv_bfloat16* out = dQ + (long long)b * bsg + (long long)h * D;
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const int qrow = q0 + warp * 16 + g + r * 8;
    if (qrow >= L) continue;
#pragma unroll
    for (int i = 0; i < D / 8; i++)
      *reinterpret_cast<uint32_t*>(out + (long long)qrow * ldg + i * 8 + 2 * t) = pk(dq[i][2 * r] * scale, dq[i][2 * r + 1] * scale);
  }
}

template <int D, bool CAUSAL>
__global__ void __launch_bounds__(kThr)
attn_bwd_dkv(const __nv_bfloat16* __restrict__ Q, const __nv_bfloat16* __restrict__ K, const __nv_bfloat16* __restrict__ V,
             const __nv_bfloat16* __restrict__ dO, const float* __restrict__ lse, const float* __restrict__ delta,
             __nv_bfloat16* __restrict__ dK, __nv_bfloat16* __restrict__ dV, long long ld, long long bs, long long ldo,
             long long bso, long long ldg, long long bsg, int L, float scale) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  __nv_bfloat16* sV = sK + kB * D;
  __nv_bfloat16* sQ = sV + kB * D;        // 2 buffers
  __nv_bfloat16* sdO = sQ + 2 * kB * D;   // 2 buffers
  float* sLse = reinterpret_cast<float*>(sdO + 2 * kB * D);   // [2][kB] (already * log2e)
  float* sDl = sLse + 2 * kB;                                  // [2][kB]
  const int kvb = blockIdx.x, h = blockIdx.y, b = blockIdx.z, H = gridDim.y;
  const int k0 = kvb * kB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const __nv_bfloat16* gq = Q + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gk = K + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gv = V + (long long)b * bs + (long long)h * D;
  const __nv_bfloat16* gdo = dO + (long long)b * bso + (long long)h * D;
  const float* glse = lse + ((long long)b * H + h) * L;
  const float* gdl = delta + ((long long)b * H + h) * L;
  const int n_q = (L + kB - 1) / kB;
  const int qb0 = CAUSAL ? kvb : 0;
  constexpr float kLog2e = 1.4426950408889634f;
  const float c = scale * kLog2e;

  auto load_q = [&](int qb, int buf) {
    load_tile<D>(sQ + buf * kB * D, gq, ld, qb * kB, L);
    load_tile<D>(sdO + buf * kB * D, gdo, ldo, qb * kB, L);
    if (threadIdx.x < kB) {
      const int q = min(qb * kB + (int)threadIdx.x, L - 1);
      sLse[buf * kB + threadIdx.x] = glse[q] * kLog2e;
      sDl[buf * kB + threadIdx.x] = gdl[q];
    }
  };
  load_tile<D>(sK, gk, ld, k0, L);
  load_tile<D>(sV, gv, ld, k0, L);
  load_q(qb0, 0);
  cp_commit();

  float dk[D / 8][4], dv[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; i++) { dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f; dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f; }

  for (int qb = qb0; qb < n_q; qb++) {
    const int buf = (qb - qb0) & 1;
    if (qb + 1 < n_q) {
      load_q(qb + 1, buf ^ 1);
      cp_commit();
      cp_wait<1>();
    } else {
      cp_wait<0>();
    }
    __syncthreads();
    const __nv_bfloat16* cQ = sQ + buf * kB * D;
    const __nv_bfloat16* cdO = sdO + buf * kB * D;
    // S^T = K Q^T and dP^T = V dO^T : rows = this warp's 16 keys, columns = the 64 queries of the block
    float st[kB / 8][4], dpt[kB / 8][4];
#pragma unroll
    for (int i = 0; i < kB / 8; i++) { st[i][0] = st[i][1] = st[i][2] = st[i][3] = 0.f; dpt[i][0] = dpt[i][1] = dpt[i][2] = dpt[i][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < D / 16; kk++) {
      uint32_t ka[4], va[4];
      frag_a<D>(sK, warp * 16, kk, lane, ka);
      frag_a<D>(sV, warp * 16, kk, lane, va);
#pragma unroll
      for (int n2 = 0; n2 < kB / 16; n2++) {
        uint32_t bq[4], bo[4];
        frag_b_rows_n<D>(cQ, n2, kk, lane, bq);
        mma(st[2 * n2], ka, bq[0], bq[1]);
        mma(st[2 * n2 + 1], ka, bq[2], bq[3]);
        frag_b_rows_n<D>(cdO, n2, kk, lane, bo);
        mma(dpt[2 * n2], va, bo[0], bo[1]);
        mma(dpt[2 * n2 + 1], va, bo[2], bo[3]);
      }
    }
    const int q0 = qb * kB, krow0 = k0 + warp * 16;
    // masking is needed on the diagonal block (causal), for keys >= L and for queries >= L
    const bool edge = q0 + kB > L || k0 + kB > L || (CAUSAL && qb == kvb);
    uint32_t pf[kB / 16][4], dsf[kB / 16][4];
#pragma unroll
    for (int nt = 0; nt < kB / 8; nt++) {
      float p[4], ds[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int qc = nt * 8 + 2 * t + (e & 1);      // query column within the block
        p[e] = exp2f(fmaf(st[nt][e], c, -sLse[buf * kB + qc]));
        if (edge) {
          const int key = krow0 + g + ((e >> 1) << 3);
          const int qrow = q0 + qc;
          if (key >= L || qrow >= L || (CAUSAL && key > qrow)) p[e] = 0.f;
        }
        ds[e] = p[e] * (dpt[nt][e] - sDl[buf * kB + qc]);
      }
      pf[nt >> 1][(nt & 1) * 2] = pk(p[0], p[1]);
      pf[nt >> 1][(nt & 1) * 2 + 1] = pk(p[2], p[3]);
      dsf[nt >> 1][(nt & 1) * 2] = pk(ds[0], ds[1]);
      dsf[nt >> 1][(nt & 1) * 2 + 1] = pk(ds[2], ds[3]);
    }
    // dV += P^T dO ; dK += dS^T Q   (contraction over the block's 64 queries)
#pragma unroll
    for (int kt = 0; kt < kB / 16; kt++) {
#pragma unroll
      for (int d2 = 0; d2 < D / 16; d2++) {
        uint32_t bo[4], bq[4];
        frag_b_rows_k<D>(cdO, kt, d2, lane, bo);
        mma(dv[2 * d2], pf[kt], bo[0], bo[1]);
        mma(dv[2 * d2 + 1], pf[kt], bo[2], bo[3]);
        frag_b_rows_k<D>(cQ, kt, d2, lane, bq);
        mma(dk[2 * d2], dsf[kt], bq[0], bq[1]);
        mma(dk[2 * d2 + 1], dsf[kt], bq[2], bq[3]);
      }
    }
    __syncthreads();
  }
  __nv_bfloat16* ok = dK + (long long)b * bsg + (long long)h * D;
  __nv_bfloat16* ov = dV + (long long)b * bsg + (long long)h * D;
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const int krow = k0 + warp * 16 + g + r * 8;
    if (krow >= L) continue;
#pragma unroll
    for (int i = 0; i < D / 8; i++) {
      *reinterpret_cast<uint32_t*>(ok + (long long)krow * ldg + i * 8 + 2 * t) = pk(dk[i][2 * r] * scale, dk[i][2 * r + 1] * scale);
      *reinterpret_cast<uint32_t*>(ov + (long long)krow * ldg + i * 8 + 2 * t) = pk(dv[i][2 * r], dv[i][2 * r + 1]);
    }
  }
}

template <int D, bool CAUSAL>
static int launch_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse,
                      float* delta, void* dq, void* dk, void* dv, long long ld, long long bs, long long ldo,
                      long long bso, long long ldg, long long bsg, int B, int H, int L, float scale, cudaStream_t st) {
  const long long warps = (long long)B * L * H;
  attn_bwd_delta<D><<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)o, (const __nv_bfloat16*)dout,
                                                                       ldo, bso, delta, B, H, L);
  G4R_LAUNCH_CHECK("attn_bwd_delta");
  const int smem_dq = 6 * kB * D * 2;
  const int smem_dkv = 6 * kB * D * 2 + 4 * kB * (int)sizeof(float);
  static bool set = false;
  if (!set) {
    G4R_CUDA(cudaFuncSetAttribute(attn_bwd_dq<D, CAUSAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dq));
    G4R_CUDA(cudaFuncSetAttribute(attn_bwd_dkv<D, CAUSAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dkv));
    set = true;
  }
  dim3 grid((L + kB - 1) / kB, H, B);
  attn_bwd_dq<D, CAUSAL><<<grid, kThr, smem_dq, st>>>((const __nv_bfloat16*)q, (const __nv_bfloat16*)k, (const __nv_bfloat16*)v,
                                                      (const __nv_bfloat16*)dout, lse, delta, (__nv_bfloat16*)dq, ld, bs, ldo,
                                                      bso, ldg, bsg, L, scale);
  G4R_LAUNCH_CHECK("attn_bwd_dq");
  attn_bwd_dkv<D, CAUSAL><<<grid, kThr, smem_dkv, st>>>((const __nv_bfloat16*)q, (const __nv_bfloat16*)k, (const __nv_bfloat16*)v,
                                                        (const __nv_bfloat16*)dout, lse, delta, (__nv_bfloat16*)dk,
                                                        (__nv_bfloat16*)dv, ld, bs, ldo, bso, ldg, bsg, L, scale);
  G4R_LAUNCH_CHECK("attn_bwd_dkv");
  return G4R_OK;
}

}  // namespace g4r

using namespace g4r;

extern "C" int g4r_attention_bwd_bf16(const void* q, const void* k, const void* v, const void* out, const void* dout,
                                      const float* lse, float* delta, void* dq, void* dk, void* dv, long long ld,
                                      long long bs, long long ldo, long long bso, long long ldg, long long bsg, int B,
                                      int H, int L, int head_dim, int causal, float scale, void* stream) {
  G4R_REQUIRE(q && k && v && out && dout && lse && delta && dq && dk && dv && B > 0 && H > 0 && L > 0, "attention_bwd: bad arguments");
  G4R_REQUIRE(head_dim == 64 || head_dim == 128, "attention_bwd: head_dim %d (64 or 128)", head_dim);
  G4R_REQUIRE(ld % 8 == 0 && bs % 8 == 0 && ldo % 8 == 0 && bso % 8 == 0 && ldg % 2 == 0 && bsg % 2 == 0,
              "attention_bwd: strides must keep 16-byte row alignment");
  G4R_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)dout) & 15) == 0, "attention_bwd: misaligned pointers");
  cudaStream_t st = (cudaStream_t)stream;
  if (head_dim == 64) {
    return causal ? launch_bwd<64, true>(q, k, v, out, dout, lse, delta, dq, dk, dv, ld, bs, ldo, bso, ldg, bsg, B, H, L, scale, st)
                  : launch_bwd<64, false>(q, k, v, out, dout, lse, delta, dq, dk, dv, ld, bs, ldo, bso, ldg, bsg, B, H, L, scale, st);
  }
  return causal ? launch_bwd<128, true>(q, k, v, out, dout, lse, delta, dq, dk, dv, ld, bs, ldo, bso, ldg, bsg, B, H, L, scale, st)
                : launch_bwd<128, false>(q, k, v, out, dout, lse, delta, dq, dk, dv, ld, bs, ldo, bso, ldg, bsg, B, H, L, scale, st);
}
