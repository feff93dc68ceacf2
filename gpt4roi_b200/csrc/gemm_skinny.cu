// gemm_skinny.cu -- weight-streaming GEMM for M <= 16 activation rows (the decode step behind
// generate(), SURVEY.md 8(f1): one new token per sample, gpt4roi/models/spi_llava.py:47-48 skips the
// vision branch so the step is the 7B LLaMA stack at M = batch).
//
// D[M, N] = A[M, K] . W[N, K]^T with the epilogues of gemm_tcgen05.cu (bias, residual, SwiGLU,
// fused RoPE).  At M <= 16 a 128-row tcgen05 tile wastes the tensor pipe and, worse, gives one CTA
// per 256 weight rows: too few CTAs to keep HBM busy (measured 1.7 TB/s).  This kernel is HBM-bound
// by construction: every weight byte is read exactly once with 16-byte streaming loads
// (ld.global.nc.L1::no_allocate), hundreds of CTAs each cover 16/32 weight rows over the whole K, and
// the warps of a CTA split K.  The arithmetic rides on mma.sync m16n8k16 with the weight rows as the
// 16-row operand and the (<= 8) activation rows as the 8-column operand -- tcgen05 has no shape this
// small (M >= 64) and the kernel is nowhere near compute-bound (2*M flop per weight byte pair).
//
// k-permutation trick: the MMA contracts over "logical" k and does not care which physical k each
// slot holds as long as A and B agree.  Thread (g, t) therefore takes its 8 slots of two consecutive
// k16 steps from ONE 16-byte load at physical k0 + 8t .. 8t+7, from the weight row and from the
// activation row alike -- no shuffles, no shared-memory staging, full-sector global loads.
//
// Deterministic: the partial sums of the warps are added in a fixed order.
#include "common.cuh"
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

enum { SK_ACT_NONE = 0, SK_ACT_RELU = 1, SK_ACT_QUICK_GELU = 2, SK_ACT_SWIGLU = 3 };

struct SkinnyParams {
  const __nv_bfloat16* A; long long lda;
  const __nv_bfloat16* W; long long ldb;
  __nv_bfloat16* D; long long ldd;
  int M, N, K;
  const void* bias; int bias_f32;
  const __nv_bfloat16* residual; long long ldr;
  int act;
  const __nv_bfloat16* rope_cos; const __nv_bfloat16* rope_sin;
  int rope_cols, rope_L, rope_pos0;
  const int* rope_pos_dev;
  // decode-step fusion (optional):
  __nv_bfloat16* kcache; __nv_bfloat16* vcache;  // [M, cache_lmax, cache_hd]: k / v columns are also written at `pos`
  int cache_lmax, cache_hd;
};

// weights: constant for the lifetime of the step, read exactly once.  volatile: the first block is issued BEFORE
// pdl_wait() and must stay there.
__device__ __forceinline__ uint4 ldg_stream16(const void* ptr) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}
// activations: written by the predecessor kernel, read after pdl_wait() on the coherent path (no .nc).  volatile asm:
// keeps its order relative to griddepcontrol.wait (also volatile) and stays an unconditional, straight-line load.
__device__ __forceinline__ uint4 ldg_act16(const void* ptr) {
  uint4 v;
  asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}

__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                          uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32." G4R_ACT_PTX "." G4R_ACT_PTX ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// MT: 16-row weight tiles per CTA (1 or 2); MB: 8-row activation blocks (1: M<=8, 2: M<=16);
// ROPE: the two tiles are 64 rows apart (dims d and d+64 of one 128-dim head) so the rotation has
// both partners in the CTA.
// DEPTH: k-blocks each warp keeps in flight (register double buffering): with DEPTH = 2 a warp that owns two k-blocks
// (o_proj: K = 4096 over 16 warps) requests its whole share before the first MMA -- one HBM latency instead of two.
// DEPTH = 2 relies on 2 CTAs per SM (see gemm_skinny_run), i.e. <= 128 registers; the launch bound holds ptxas to it.
template <int MT, int MB, int WARPS, bool ROPE, int DEPTH = 1>
__global__ void __launch_bounds__(WARPS * 32, DEPTH == 2 ? 2 : 0)
gemm_skinny_bf16(const SkinnyParams p) {
  constexpr int KB = 128;        // k per warp iteration: 4 sub-blocks of 32 (one 16-byte load per row each)
  constexpr int NT = MT * 16;
  constexpr int MC = MB * 8;
  __shared__ float red[WARPS][NT][MC + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int tile_stride = ROPE ? 64 : 16;
  const int n_base = ROPE ? (int)(blockIdx.x >> 2) * 128 + (int)(blockIdx.x & 3) * 16 : (int)blockIdx.x * NT;

  float acc[MT][MB][4];
#pragma unroll
  for (int j = 0; j < MT; j++)
#pragma unroll
    for (int i = 0; i < MB; i++)
#pragma unroll
      for (int c = 0; c < 4; c++) acc[j][i][c] = 0.f;

  const __nv_bfloat16* wrow[MT][2];
  bool wok[MT][2];
#pragma unroll
  for (int j = 0; j < MT; j++)
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int n = n_base + j * tile_stride + g + 8 * h;
      wok[j][h] = n < p.N;
      wrow[j][h] = p.W + (long long)(wok[j][h] ? n : 0) * p.ldb + 8 * t;
    }
  const __nv_bfloat16* xrow[MB];
  bool xok[MB];
#pragma unroll
  for (int i = 0; i < MB; i++) {
    const int m = i * 8 + g;
    xok[i] = m < p.M;
    xrow[i] = p.A + (long long)(xok[i] ? m : 0) * p.lda + 8 * t;
  }

  // The first weight block of every warp does not depend on the predecessor kernel: issue it, then wait for the
  // predecessor (programmatic dependent launch, common.cuh) -- its tail and this kernel's ramp-up overlap.
  constexpr int kstep = WARPS * KB;
  int k0 = warp * KB;
  uint4 a[DEPTH][4][MT][2];
  auto load_w = [&](uint4 (&aw)[4][MT][2], int kb) {
#pragma unroll
    for (int s = 0; s < 4; s++) {
      // K % 32 == 0: a sub-block is whole or absent.  Loads are unconditional (absent blocks / rows re-read element 0
      // and are zeroed or never stored), so the block is straight-line code the scheduler can issue back to back.
      const bool kok = kb + 32 * s < p.K;
      const int kk = kok ? kb + 32 * s : 0;
#pragma unroll
      for (int j = 0; j < MT; j++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const uint4 v = ldg_stream16(wrow[j][h] + kk);
          aw[s][j][h] = kok ? v : make_uint4(0, 0, 0, 0);
        }
    }
  };
#pragma unroll
  for (int d = 0; d < DEPTH; d++)
    if (k0 + d * kstep < p.K) load_w(a[d], k0 + d * kstep);
  pdl_sync();

  // activation fragments of a k-block; like the weights they are fetched DEPTH blocks ahead, so that all loads of a
  // block are issued back to back (left inside the loop body, ptxas strings them out between the dependent HMMAs)
  uint4 b[DEPTH][4][MB];
  auto load_x = [&](uint4 (&bx)[4][MB], int kb) {
#pragma unroll
    for (int s = 0; s < 4; s++) {
      const bool kok = kb + 32 * s < p.K;
      const int kk = kok ? kb + 32 * s : 0;
#pragma unroll
      for (int i = 0; i < MB; i++) {
        const uint4 v = ldg_act16(xrow[i] + kk);   // rows >= M alias row 0; their outputs are never stored
        bx[s][i] = kok ? v : make_uint4(0, 0, 0, 0);
      }
    }
  };
#pragma unroll
  for (int d = 0; d < DEPTH; d++)
    if (k0 + d * kstep < p.K) load_x(b[d], k0 + d * kstep);
#pragma unroll 1
  for (; k0 < p.K; k0 += DEPTH * kstep) {
#pragma unroll
    for (int d = 0; d < DEPTH; d++) {
      const int kd = k0 + d * kstep;
      if (kd >= p.K) break;       // warp-uniform
#pragma unroll
      for (int s = 0; s < 4; s++)
#pragma unroll
        for (int j = 0; j < MT; j++)
#pragma unroll
          for (int i = 0; i < MB; i++) {
            mma_16816(acc[j][i], a[d][s][j][0].x, a[d][s][j][1].x, a[d][s][j][0].y, a[d][s][j][1].y, b[d][s][i].x, b[d][s][i].y);
            mma_16816(acc[j][i], a[d][s][j][0].z, a[d][s][j][1].z, a[d][s][j][0].w, a[d][s][j][1].w, b[d][s][i].z, b[d][s][i].w);
          }
      if (kd + DEPTH * kstep < p.K) {   // refill this slot: in flight across the loop edge
        load_w(a[d], kd + DEPTH * kstep);
        load_x(b[d], kd + DEPTH * kstep);
      }
    }
  }

  // accumulator fragment: c0,c1 = (weight row g, activation rows 2t, 2t+1); c2,c3 = (weight row g+8, ...)
#pragma unroll
  for (int j = 0; j < MT; j++)
#pragma unroll
    for (int i = 0; i < MB; i++)
#pragma unroll
      for (int c = 0; c < 4; c++) red[warp][j * 16 + g + 8 * (c >> 1)][i * 8 + 2 * t + (c & 1)] = acc[j][i][c];
  __syncthreads();

  auto total = [&](int r, int m) {   // warps in fixed order: bitwise reproducible
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; w++) v += red[w][r][m];
    return v;
  };

  if (ROPE) {
    // thread <-> (activation row m, d in [0,16) of this CTA's slice); partners r (dim d) and 16 + r (dim d+64)
    for (int e = threadIdx.x; e < 16 * MC; e += WARPS * 32) {
      const int r = e & 15, m = e >> 4;
      if (m >= p.M) continue;
      const int n1 = n_base + r, n2 = n1 + 64;
      const float v1 = total(r, m), v2 = total(16 + r, m);
      __nv_bfloat16* o = p.D + (long long)m * p.ldd;
      if (n1 < p.rope_cols) {
        // rounding points as in the tcgen05 epilogue / transformers modeling_llama.py:138-168
        const int pos = (p.rope_pos_dev ? *p.rope_pos_dev : p.rope_pos0) + m % p.rope_L;
        const int d = n1 & 127;
        const __nv_bfloat16* ct = p.rope_cos + (long long)pos * 128;
        const __nv_bfloat16* st = p.rope_sin + (long long)pos * 128;
        const float x1 = bf16r(v1), x2 = bf16r(v2);
        const float a1 = bf16r(x1 * __bfloat162float(ct[d])), b1 = bf16r(-x2 * __bfloat162float(st[d]));
        const float a2 = bf16r(x2 * __bfloat162float(ct[d + 64])), b2 = bf16r(x1 * __bfloat162float(st[d + 64]));
        const __nv_bfloat16 r1 = __float2bfloat16_rn(a1 + b1), r2 = __float2bfloat16_rn(a2 + b2);
        o[n1] = r1;
        o[n2] = r2;
        if (p.kcache != nullptr && n1 >= p.cache_hd) {   // a key column: also the cache row of sample m at this position
          __nv_bfloat16* kc = p.kcache + ((long long)m * p.cache_lmax + pos) * p.cache_hd - p.cache_hd;
          kc[n1] = r1;
          kc[n2] = r2;
        }
      } else {
        const __nv_bfloat16 r1 = __float2bfloat16_rn(v1), r2 = __float2bfloat16_rn(v2);
        o[n1] = r1;
        o[n2] = r2;
        if (p.vcache != nullptr && n1 >= 2 * p.cache_hd) {
          const int pos = (p.rope_pos_dev ? *p.rope_pos_dev : p.rope_pos0) + m % p.rope_L;
          __nv_bfloat16* vc = p.vcache + ((long long)m * p.cache_lmax + pos) * p.cache_hd - 2 * p.cache_hd;
          vc[n1] = r1;
          vc[n2] = r2;
        }
      }
    }
    return;
  }

  for (int e = threadIdx.x; e < NT * MC; e += WARPS * 32) {
    const int r = e % NT, m = e / NT;
    const int n = n_base + r;
    if (m >= p.M || n >= p.N) continue;
    if (p.act == SK_ACT_SWIGLU) {
      if (r & 1) continue;   // even row = gate_j, odd row = up_j (interleaved weights) -> out[:, j]
      float gt = total(r, m), up = total(r + 1, m);
      if (p.bias != nullptr) {
        gt += p.bias_f32 ? reinterpret_cast<const float*>(p.bias)[n] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.bias)[n]);
        up += p.bias_f32 ? reinterpret_cast<const float*>(p.bias)[n + 1] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.bias)[n + 1]);
      }
      p.D[(long long)m * p.ldd + (n >> 1)] = __float2bfloat16_rn(gt / (1.f + __expf(-gt)) * up);
      continue;
    }
    float v = total(r, m);
    if (p.bias != nullptr)
      v += p.bias_f32 ? reinterpret_cast<const float*>(p.bias)[n] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.bias)[n]);
    if (p.act == SK_ACT_RELU) v = fmaxf(v, 0.f);
    if (p.act == SK_ACT_QUICK_GELU) v = v / (1.f + __expf(-1.702f * v));
    if (p.residual != nullptr) v += __bfloat162float(p.residual[(long long)m * p.ldr + n]);
    p.D[(long long)m * p.ldd + n] = __float2bfloat16_rn(v);
  }
}

template <int MT, int MB, int WARPS, bool ROPE, int DEPTH = 1>
static int launch_skinny(const SkinnyParams& p, unsigned tiles, cudaStream_t st) {
  G4R_CUDA(launch_pdl(gemm_skinny_bf16<MT, MB, WARPS, ROPE, DEPTH>, dim3(tiles), dim3(WARPS * 32), 0, st, dim3(1, 1, 1), p));
  return G4R_OK;
}

// 32-row tiles, M <= 8: 4 warps (4 CTAs per SM) or 8 warps (2 CTAs per SM, twice the bytes in flight per CTA).  What
// separates them is the partially filled last wave: pick the CTA size whose wave count rounds up the least
// (gate/up, 688 tiles: 1.16 waves of 592 slots vs 2.32 of 296 -> 8 warps, 38.0 -> 35.4 us; lm_head, 1001 tiles:
// 1.69 vs 3.38 -> 4 warps, 45.4 vs 48.4 us).
static bool wide_prefers_8_warps(int tiles) {
  const double w4 = (double)tiles / (4.0 * num_sms()), w8 = (double)tiles / (2.0 * num_sms());
  auto waste = [](double w) { const double c = (double)(long long)(w + 0.999999); return c / w; };
  return waste(w8) < 0.95 * waste(w4);
}

// Tile selection for both entry points: gemm_impl (gemm_tcgen05.cu) and g4r_decode_gemm_*.  Returns -1 when the shape
// does not qualify.
static int gemm_skinny_run(SkinnyParams p, cudaStream_t st) {
  if (p.M > 16 || p.K % 32 != 0) return -1;
  if (p.act == SK_ACT_SWIGLU && (p.N % 2 != 0)) return -1;
  p.rope_L = p.rope_L > 0 ? p.rope_L : 1;
  if (p.rope_cos != nullptr) {
    if (p.N % 128 != 0) return -1;
    const unsigned grid = (unsigned)(p.N / 128) * 4;
    return p.M <= 8 ? launch_skinny<2, 1, 4, true>(p, grid, st) : launch_skinny<2, 2, 4, true>(p, grid, st);
  }
  // 32-row tiles halve the activation re-reads; use them once they still give >= 2 CTAs per SM
  const bool wide = (p.N + 31) / 32 >= 2 * num_sms();
  if (wide) {
    const unsigned grid = (unsigned)((p.N + 31) / 32);
    if (p.M > 8) return launch_skinny<2, 2, 4, false>(p, grid, st);
    return wide_prefers_8_warps((int)grid) ? launch_skinny<2, 1, 8, false>(p, grid, st) : launch_skinny<2, 1, 4, false>(p, grid, st);
  }
  const unsigned grid = (unsigned)((p.N + 15) / 16);
  // 16-row tiles give few CTAs (N/16 = 256 for the 4096-row projections).  M <= 8: 8 warps with two k-blocks in flight
  // each (128 registers -> 2 CTAs per SM, so all 256 CTAs are resident at once and request half the matrix up front):
  // o_proj 11.4 -> 8.4 us, down_proj 21.5 -> 17.8 us (B200, profiles/r2_decode_pdl_depth.md).  M <= 16: 16 warps.
  return p.M <= 8 ? launch_skinny<1, 1, 8, false, 2>(p, grid, st) : launch_skinny<1, 2, 16, false>(p, grid, st);
}

// Called by gemm_impl (gemm_tcgen05.cu) for M <= 16; returns -1 when the shape does not qualify.
int gemm_skinny_dispatch(const void* A, long long lda, const void* B, long long ldb, void* D, long long ldd, int M,
                         int N, int K, const void* bias, int bias_f32, const void* residual, long long ldr, int act,
                         const void* rope_cos, const void* rope_sin, int rope_cols, int rope_L, int rope_pos0,
                         const int* rope_pos_dev, void* stream) {
  SkinnyParams p{};
  p.A = (const __nv_bfloat16*)A; p.lda = lda; p.W = (const __nv_bfloat16*)B; p.ldb = ldb;
  p.D = (__nv_bfloat16*)D; p.ldd = ldd; p.M = M; p.N = N; p.K = K;
  p.bias = bias; p.bias_f32 = bias_f32; p.residual = (const __nv_bfloat16*)residual; p.ldr = ldr; p.act = act;
  p.rope_cos = (const __nv_bfloat16*)rope_cos; p.rope_sin = (const __nv_bfloat16*)rope_sin;
  p.rope_cols = rope_cols; p.rope_L = rope_L; p.rope_pos0 = rope_pos0; p.rope_pos_dev = rope_pos_dev;
  return gemm_skinny_run(p, (cudaStream_t)stream);
}

}  // namespace g4r

using namespace G4R_NS;

extern "C" int g4r_decode_gemm_bf16(const void* x, long long ldx, const void* W, long long ldw, void* out, long long ldo,
                                    int M, int N, int K, int act, const void* residual, long long ldr, const void* rope_cos, const void* rope_sin, int rope_cols, int pos0,
                                    const int* pos_dev, void* kcache, void* vcache, int cache_lmax, int cache_hd,
                                    void* stream) {
  G4R_REQUIRE(x && W && out && M > 0 && M <= 16 && N > 0 && K > 0, "decode_gemm: M must be 1..16 (got %d)", M);
  G4R_REQUIRE(ldx % 8 == 0 && ldw % 8 == 0 && K % 32 == 0, "decode_gemm: K %% 32 == 0 and 16-byte-aligned rows required");
  G4R_REQUIRE(act == SK_ACT_NONE || act == SK_ACT_SWIGLU, "decode_gemm: act must be none or swiglu");
  G4R_REQUIRE((rope_cos == nullptr) == (rope_sin == nullptr), "decode_gemm: both RoPE tables or none");
  G4R_REQUIRE(!(kcache || vcache) || (rope_cos && kcache && vcache && cache_lmax > 0 && cache_hd > 0 && N == 3 * cache_hd),
              "decode_gemm: the KV-cache write needs the fused q|k|v projection with RoPE (N == 3 * cache_hd)");
  SkinnyParams p{};
  p.A = (const __nv_bfloat16*)x; p.lda = ldx; p.W = (const __nv_bfloat16*)W; p.ldb = ldw;
  p.D = (__nv_bfloat16*)out; p.ldd = ldo; p.M = M; p.N = N; p.K = K;
  p.residual = (const __nv_bfloat16*)residual; p.ldr = ldr; p.act = act;
  p.rope_cos = (const __nv_bfloat16*)rope_cos; p.rope_sin = (const __nv_bfloat16*)rope_sin;
  p.rope_cols = rope_cols; p.rope_L = 1; p.rope_pos0 = pos0; p.rope_pos_dev = pos_dev;
  p.kcache = (__nv_bfloat16*)kcache; p.vcache = (__nv_bfloat16*)vcache; p.cache_lmax = cache_lmax; p.cache_hd = cache_hd;
  const int rc = gemm_skinny_run(p, (cudaStream_t)stream);
  if (rc == -1) { set_error("decode_gemm: shape not supported (M=%d N=%d K=%d)", M, N, K); return G4R_EUNSUPPORTED; }
  return rc;
}
