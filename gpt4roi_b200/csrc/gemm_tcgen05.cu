// gemm_tcgen05.cu -- bf16 x bf16 -> fp32 dense contraction on the 5th-gen tensor cores (sm_100a).
//
// One persistent, warp-specialised kernel serves every dense op of the region-token path:
//   D[M,N] = epilogue( A[M,K] . B[N,K]^T )           (GEMM: nn.Linear weights are [N,K] K-major)
//   D[n,y,x,:] = epilogue( conv3x3(A[n,:,:,:]) )      (implicit GEMM, NHWC, K = 9*Cin, pad 1)
// replacing the library calls the reference makes through ATen (cuBLAS / cuDNN):
//   nn.Linear            : gpt4roi/models/layers.py:260-270 (pos_embedd, updims, flatten_linear),
//                          llava/model/llava.py:52 (mm_projector), :195 (lm_head), HF CLIP / LLaMA linears
//   nn.Conv2d 1x1 / 3x3  : gpt4roi/models/layers.py:129-144 (input_conv, fuse_convs), :257-259 (pconvs)
//
// Structure (per CTA, 1 CTA / SM, persistent over output tiles):
//   warp 0     : TMA producer  -- cp.async.bulk.tensor loads of the A tile [128 x 64] and the
//                B tile [BLOCK_N x 64] (128-byte swizzle) into a kStages-deep smem ring,
//                completion signalled on `full` mbarriers (expect_tx).
//                In conv mode the A tile is a 4-D box (64 ch, BW, BH, 1) of the NHWC map shifted by
//                the filter tap; out-of-bounds coordinates are zero-filled by TMA = the padding.
//   warp 1     : MMA issuer    -- one thread issues tcgen05.mma (M=128, N=BLOCK_N, K=16) x4 per stage,
//                accumulating in TMEM; tcgen05.commit releases the smem slot (`empty`) and, after the
//                last k-block, publishes the accumulator (`tmem_full`).
//   warp 2     : TMEM allocator (2 accumulator stages x BLOCK_N fp32 columns).
//   warps 4..7 : epilogue      -- tcgen05.ld 32 columns at a time (thread = accumulator row), fused
//                bias / activation / residual / SwiGLU / GroupNorm statistics, bf16 or fp32 store;
//                the second accumulator stage lets tile i+1's MMAs overlap tile i's epilogue.
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = 128 B = one swizzle atom
constexpr int kUmmaK = 16;
constexpr int kGemmThreads = 256;
constexpr int kEpiWarp0 = 4;
constexpr int kSmemBudget = 200 * 1024;  // operand ring budget (bytes)

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_QUICK_GELU = 2, ACT_SWIGLU = 3 };

struct GemmParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles, num_k_blocks;  // num_k_blocks: per split
  int k_splits;
  int n_fast;  // tile order: 1 = n-tile index fastest (conv: the big NHWC input is read from DRAM once and
               // its <= 4 weight panels stay in L2), 0 = m fastest (GEMM: weight panels stream once)
  // epilogue
  void* D;
  long long ldd;
  const void* bias;      // [N] bf16 or fp32 (bias_f32), or null
  int bias_f32;
  const __nv_bfloat16* residual;  // same row mapping as D, or null (bf16, or fp32 when residual_f32)
  int residual_f32;
  int round_branch;  // round (acc + bias, act) to bf16 before the residual add (bf16 linear output + fp32 stream)
  long long ldr;
  int act;
  int out_f32;   // 1: fp32 output
  int atomic;    // unused (split-K writes per-split slabs)
  // conv mode
  int conv;
  int cH, cW, cBH, cBW, tiles_x, tiles_y, cin_blocks, taps;  // taps = 9 (3x3) or 1
  int a_rows;            // rows delivered by the A box (<= 128)
  int levels, lvl_img_stride;  // conv: sum over `levels` inputs (image index + lvl*stride), K concatenated
  // fused rotary embedding (LLaMA QKV GEMM): columns [0, rope_cols) are heads of 128 dims rotated with
  // bf16 cos/sin tables [rope_L][128]; row position = out_row % rope_L
  const __nv_bfloat16* rope_cos;
  const __nv_bfloat16* rope_sin;
  int rope_cols, rope_L, rope_pos0;
  const int* rope_pos_dev;  // optional device-side position base (CUDA-graph decode): pos0 = *rope_pos_dev
  // operand majorness (backward GEMMs): a_mn: A is stored [K][M] (M contiguous); b_mn: B is stored [K][N];
  // b_mn == 2 (conv weight gradient): B is the zero-padded NHWC input seen through a 4-D tensor map
  // {Cin, kx, row, ky} whose kx / ky dimensions alias the row dimension (strides of 1 and W+2 rows), so that
  // column block n = (tap, cin) of the virtual [rows, 9*Cin] matrix is the input shifted by that tap
  int a_mn, b_mn, dw_cin;
  float* gn_stats;       // optional [n_img, groups, 2] (sum, sumsq) of the bf16-rounded output
  int gn_group_ch;       // channels per group (16)
  int gn_groups;         // groups per image (64)
};

template <int BLOCK_N>
struct GemmCfg {
  static constexpr int kABytes = kBlockM * kBlockK * 2;
  static constexpr int kBBytes = BLOCK_N * kBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = kSmemBudget / kStageBytes;
  static constexpr int kAccStages = 2;
  static constexpr int kTmemCols = kAccStages * BLOCK_N;  // 256 or 512 (power of two)
  static constexpr int kBarBytes = (2 * kStages + 2 * kAccStages) * 8 + 16;
  static constexpr int kSmemBytes = kStages * kStageBytes + kBarBytes + 1024;  // +1024 alignment slack
};

__device__ __forceinline__ float act_apply(float x, int act) {
  if (act == ACT_RELU) return fmaxf(x, 0.f);
  if (act == ACT_QUICK_GELU) return x / (1.f + __expf(-1.702f * x));
  return x;
}

// Epilogue of one 128-row accumulator tile owned by this CTA: thread `row` (= TMEM lane) walks the
// BLOCK_N columns 32 at a time.  `arrive()` is called once all TMEM reads of the stage are done.
template <int BLOCK_N, bool CONV, typename Arrive>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, uint32_t taddr, int m_blk, int n_blk, int split,
                                              int row, int lane, Arrive arrive) {
  // row -> output row offset
  bool row_ok;
  long long out_row;
  int img = 0;
  if (CONV) {
    const int tx = m_blk % p.tiles_x;
    const int ty = (m_blk / p.tiles_x) % p.tiles_y;
    img = m_blk / (p.tiles_x * p.tiles_y);
    const int y = ty * p.cBH + row / p.cBW, x = tx * p.cBW + row % p.cBW;
    row_ok = m_blk < p.num_m_tiles && row < p.a_rows && y < p.cH && x < p.cW;
    out_row = ((long long)img * p.cH + y) * p.cW + x;
  } else {
    out_row = (long long)m_blk * kBlockM + row;
    row_ok = m_blk < p.num_m_tiles && out_row < p.M;
  }
  if (!CONV && p.rope_cos != nullptr && n_blk * BLOCK_N < p.rope_cols) {
    // ---- fused RoPE (transformers modeling_llama.py:138-168): the tile holds BLOCK_N/128 whole heads;
    // dims (d, d+64) of a head are 64 columns apart -> load both 32-column chunks, rotate, store.
    // Rounding as in the reference: q/k are bf16 GEMM outputs, each bf16 tensor op rounds:
    //   out = bf16( bf16(x*cos) + bf16(rot*sin) ),  rotate_half(x) = cat(-x2, x1).
    const int pos = (p.rope_pos_dev ? *p.rope_pos_dev : p.rope_pos0) + (int)(out_row % p.rope_L);
    const __nv_bfloat16* ct = p.rope_cos + (long long)pos * 128;
    const __nv_bfloat16* st = p.rope_sin + (long long)pos * 128;
#pragma unroll 1
    for (int hc = 0; hc < BLOCK_N / 64; hc++) {   // hc = head*2 + half-chunk (0: dims 0-31, 1: dims 32-63)
      const int cA = (hc >> 1) * 128 + (hc & 1) * 32, cB = cA + 64;
      uint32_t va[32], vb[32];
      ptx::tmem_ld_32x32b_x32(taddr + cA, va);
      ptx::tmem_ld_32x32b_x32(taddr + cB, vb);
      ptx::tmem_ld_wait();
      if (hc == BLOCK_N / 64 - 1) {
        ptx::tcgen05_before_thread_sync();
        arrive();
      }
      if (!row_ok) continue;
      const int d0 = (hc & 1) * 32;
      uint32_t oa[16], ob[16];
#pragma unroll
      for (int h8 = 0; h8 < 4; h8++) {
        const uint4 c1r = *reinterpret_cast<const uint4*>(ct + d0 + h8 * 8);
        const uint4 s1r = *reinterpret_cast<const uint4*>(st + d0 + h8 * 8);
        const uint4 c2r = *reinterpret_cast<const uint4*>(ct + 64 + d0 + h8 * 8);
        const uint4 s2r = *reinterpret_cast<const uint4*>(st + 64 + d0 + h8 * 8);
        const __nv_bfloat16* c1 = reinterpret_cast<const __nv_bfloat16*>(&c1r);
        const __nv_bfloat16* s1 = reinterpret_cast<const __nv_bfloat16*>(&s1r);
        const __nv_bfloat16* c2 = reinterpret_cast<const __nv_bfloat16*>(&c2r);
        const __nv_bfloat16* s2 = reinterpret_cast<const __nv_bfloat16*>(&s2r);
        float r1[8], r2[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const float x1 = __bfloat162float(__float2bfloat16_rn(__uint_as_float(va[h8 * 8 + j])));
          const float x2 = __bfloat162float(__float2bfloat16_rn(__uint_as_float(vb[h8 * 8 + j])));
          const float a1 = __bfloat162float(__float2bfloat16_rn(x1 * __bfloat162float(c1[j])));
          const float b1 = __bfloat162float(__float2bfloat16_rn(-x2 * __bfloat162float(s1[j])));
          const float a2 = __bfloat162float(__float2bfloat16_rn(x2 * __bfloat162float(c2[j])));
          const float b2 = __bfloat162float(__float2bfloat16_rn(x1 * __bfloat162float(s2[j])));
          r1[j] = a1 + b1;
          r2[j] = a2 + b2;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
          __nv_bfloat162 h1 = __floats2bfloat162_rn(r1[2 * j], r1[2 * j + 1]);
          __nv_bfloat162 h2 = __floats2bfloat162_rn(r2[2 * j], r2[2 * j + 1]);
          oa[h8 * 4 + j] = *reinterpret_cast<uint32_t*>(&h1);
          ob[h8 * 4 + j] = *reinterpret_cast<uint32_t*>(&h2);
        }
      }
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.D) + out_row * p.ldd + n_blk * BLOCK_N;
#pragma unroll
      for (int h4 = 0; h4 < 4; h4++) {
        reinterpret_cast<uint4*>(o + cA)[h4] = make_uint4(oa[4 * h4], oa[4 * h4 + 1], oa[4 * h4 + 2], oa[4 * h4 + 3]);
        reinterpret_cast<uint4*>(o + cB)[h4] = make_uint4(ob[4 * h4], ob[4 * h4 + 1], ob[4 * h4 + 2], ob[4 * h4 + 3]);
      }
    }
    return;
  }
#pragma unroll 1
  for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
    uint32_t v[32];
    ptx::tmem_ld_32x32b_x32(taddr + c0, v);
    ptx::tmem_ld_wait();
    if (c0 + 32 >= BLOCK_N) {
      // all TMEM reads of this accumulator stage are done: hand it back to the MMA warp
      ptx::tcgen05_before_thread_sync();
      arrive();
    }
    const int col0 = n_blk * BLOCK_N + c0;
    if (col0 >= p.N) continue;  // (warp-uniform)
    float f[32];
#pragma unroll
    for (int j = 0; j < 32; j++) f[j] = __uint_as_float(v[j]);
    const bool full_chunk = col0 + 32 <= p.N;
    if (p.bias != nullptr && split == 0) {
      if (p.bias_f32) {
        const float* b = reinterpret_cast<const float*>(p.bias) + col0;
#pragma unroll
        for (int j = 0; j < 32; j++) if (full_chunk || col0 + j < p.N) f[j] += b[j];
      } else {
        const __nv_bfloat16* b = reinterpret_cast<const __nv_bfloat16*>(p.bias) + col0;
#pragma unroll
        for (int j = 0; j < 32; j++) if (full_chunk || col0 + j < p.N) f[j] += __bfloat162float(b[j]);
      }
    }
    if (p.act == ACT_RELU || p.act == ACT_QUICK_GELU) {
#pragma unroll
      for (int j = 0; j < 32; j++) f[j] = act_apply(f[j], p.act);
    }
    if (p.act == ACT_SWIGLU) {
      // interleaved weights: column 2j = gate_j, 2j+1 = up_j -> out[:, j] = silu(gate) * up
      if (row_ok) {
        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.D) + out_row * p.ldd + col0 / 2;
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const float g0 = f[4 * j], u0 = f[4 * j + 1], g1 = f[4 * j + 2], u1 = f[4 * j + 3];
          const float s0 = g0 / (1.f + __expf(-g0)) * u0, s1 = g1 / (1.f + __expf(-g1)) * u1;
          __nv_bfloat162 h = __floats2bfloat162_rn(s0, s1);
          pk[j] = *reinterpret_cast<uint32_t*>(&h);
        }
        if (full_chunk && (p.ldd % 8 == 0)) {
          reinterpret_cast<uint4*>(o)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          reinterpret_cast<uint4*>(o)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        } else {
          const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(pk);
          for (int j = 0; j < 16; j++) if (col0 + 2 * j + 1 < p.N) o[j] = e[j];
        }
      }
      continue;
    }
    if (p.round_branch) {
#pragma unroll
      for (int j = 0; j < 32; j++) f[j] = __bfloat162float(__float2bfloat16_rn(f[j]));
    }
    if (p.residual != nullptr && row_ok) {
      if (p.residual_f32) {
        // fp32 residual stream (CLIP under autocast keeps it in fp32: LayerNorm outputs fp32 and
        // `residual + bf16_branch` promotes)
        const float* rr = reinterpret_cast<const float*>(p.residual) + out_row * p.ldr + col0;
        if (full_chunk && (p.ldr % 4 == 0)) {
#pragma unroll
          for (int h = 0; h < 8; h++) {
            const float4 r4 = reinterpret_cast<const float4*>(rr)[h];
            f[4 * h] += r4.x; f[4 * h + 1] += r4.y; f[4 * h + 2] += r4.z; f[4 * h + 3] += r4.w;
          }
        } else {
          for (int j = 0; j < 32; j++) if (col0 + j < p.N) f[j] += rr[j];
        }
      } else {
        const __nv_bfloat16* rr = p.residual + out_row * p.ldr + col0;
        if (full_chunk && (p.ldr % 8 == 0)) {
#pragma unroll
          for (int h = 0; h < 4; h++) {
            const uint4 raw = reinterpret_cast<const uint4*>(rr)[h];
            const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
            for (int j = 0; j < 8; j++) f[h * 8 + j] += __bfloat162float(e[j]);
          }
        } else {
          for (int j = 0; j < 32; j++) if (col0 + j < p.N) f[j] += __bfloat162float(rr[j]);
        }
      }
    }
    if (p.out_f32) {
      if (row_ok) {
        // split-K: split s writes slab s of a [k_splits][M][ldd] fp32 buffer (no atomics; the consumer
        // sums the slabs in a fixed order, so the result is bitwise reproducible)
        float* o = reinterpret_cast<float*>(p.D) + ((long long)split * p.M + out_row) * p.ldd + col0;
        if (full_chunk && (p.ldd % 4 == 0)) {
#pragma unroll
          for (int h = 0; h < 8; h++)
            reinterpret_cast<float4*>(o)[h] = make_float4(f[4 * h], f[4 * h + 1], f[4 * h + 2], f[4 * h + 3]);
        } else {
          for (int j = 0; j < 32; j++) if (col0 + j < p.N) o[j] = f[j];
        }
      }
    } else {
      uint32_t pk[16];
#pragma unroll
      for (int j = 0; j < 16; j++) {
        __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
        pk[j] = *reinterpret_cast<uint32_t*>(&h);
      }
      if (row_ok) {
        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.D) + out_row * p.ldd + col0;
        if (full_chunk && (p.ldd % 8 == 0)) {
#pragma unroll
          for (int h = 0; h < 4; h++)
            reinterpret_cast<uint4*>(o)[h] = make_uint4(pk[4 * h], pk[4 * h + 1], pk[4 * h + 2], pk[4 * h + 3]);
        } else {
          const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(pk);
          for (int j = 0; j < 32; j++) if (col0 + j < p.N) o[j] = e[j];
        }
      }
      if (CONV && p.gn_stats != nullptr) {
        // GroupNorm statistics of the bf16-rounded conv output (what the reference's GN sees:
        // mmcv cnn/bricks/conv_module.py:196-208 runs GN on the conv's bf16 result).
        // 32 columns = 2 groups of 16 channels; reduce over the 32 rows of this warp, then ONE plain
        // store per (tile, warp) slot -- no atomics, so the statistics are bitwise reproducible;
        // gn_finalize sums the slots in a fixed order.
        const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(pk);
        float s[2] = {0.f, 0.f}, ss[2] = {0.f, 0.f};
        if (row_ok) {
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const float x = __bfloat162float(e[j]);
            s[j >> 4] += x;
            ss[j >> 4] += x * x;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          s[0] += __shfl_xor_sync(0xffffffffu, s[0], o);
          s[1] += __shfl_xor_sync(0xffffffffu, s[1], o);
          ss[0] += __shfl_xor_sync(0xffffffffu, ss[0], o);
          ss[1] += __shfl_xor_sync(0xffffffffu, ss[1], o);
        }
        if (lane < 2 && full_chunk && m_blk < p.num_m_tiles) {
          const int tiles_per_img = p.tiles_x * p.tiles_y;
          const int slot = (m_blk % tiles_per_img) * 4 + (row >> 5);
          float* st = p.gn_stats + (((long long)img * (tiles_per_img * 4) + slot) * p.gn_groups +
                                    (col0 / p.gn_group_ch + lane)) * 2;
          st[0] = lane == 0 ? s[0] : s[1];
          st[1] = lane == 0 ? ss[0] : ss[1];
        }
      }
    }
  }
}

template <int BLOCK_N, bool CONV>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                  const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BLOCK_N>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + Cfg::kStages;
  uint64_t* tmem_full = bars + 2 * Cfg::kStages;
  uint64_t* tmem_empty = tmem_full + Cfg::kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + Cfg::kAccStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::kStages; i++) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < Cfg::kAccStages; i++) {
      ptx::mbar_init(&tmem_full[i], 1);
      ptx::mbar_init(&tmem_empty[i], 128);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
  ptx::tcgen05_before_thread_sync();
  __syncthreads();
  ptx::tcgen05_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles_mn = p.num_m_tiles * p.num_n_tiles;
  const int total_tiles = tiles_mn * p.k_splits;

  if (warp == 0) {
    // ============================ TMA producer ============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int split = t / tiles_mn;
        const int mn = t % tiles_mn;
        const int n_blk = p.n_fast ? mn % p.num_n_tiles : mn / p.num_m_tiles;
        const int m_blk = p.n_fast ? mn / p.num_n_tiles : mn % p.num_m_tiles;
        const int kb0 = split * p.num_k_blocks;
        int img = 0, y0 = 0, x0 = 0;
        if (CONV) {
          const int tx = m_blk % p.tiles_x;
          const int ty = (m_blk / p.tiles_x) % p.tiles_y;
          img = m_blk / (p.tiles_x * p.tiles_y);
          y0 = ty * p.cBH;
          x0 = tx * p.cBW;
        }
        for (int kb = 0; kb < p.num_k_blocks; kb++) {
          ptx::mbar_wait(&empty[stage], phase ^ 1);
          ptx::mbar_arrive_expect_tx(&full[stage], (uint32_t)(p.a_rows * kBlockK * 2 + Cfg::kBBytes));
          const int kg = kb0 + kb;
          if (CONV) {
            const int tap_all = kg / p.cin_blocks, cc = kg % p.cin_blocks;
            const int lvl = tap_all / p.taps, tap = tap_all % p.taps;
            const int dy = p.taps == 9 ? tap / 3 - 1 : 0, dx = p.taps == 9 ? tap % 3 - 1 : 0;
            ptx::tma_load_4d(smem_a + stage * Cfg::kABytes, &tmap_a, &full[stage], cc * kBlockK, x0 + dx,
                             y0 + dy, img + lvl * p.lvl_img_stride);
          } else if (p.a_mn) {
            // MN-major A: two [64 k][64 m] boxes (one 128-byte swizzle atom of m each)
#pragma unroll
            for (int a = 0; a < kBlockM / 64; a++)
              ptx::tma_load_2d(smem_a + stage * Cfg::kABytes + a * (kBlockK * 128), &tmap_a, &full[stage],
                               m_blk * kBlockM + a * 64, kg * kBlockK);
          } else {
            ptx::tma_load_2d(smem_a + stage * Cfg::kABytes, &tmap_a, &full[stage], kg * kBlockK,
                             m_blk * kBlockM);
          }
          if (!CONV && p.b_mn == 2) {
            const int n0 = n_blk * BLOCK_N, tap = n0 / p.dw_cin, c0 = n0 % p.dw_cin;
#pragma unroll
            for (int a = 0; a < BLOCK_N / 64; a++)
              ptx::tma_load_4d(smem_b + stage * Cfg::kBBytes + a * (kBlockK * 128), &tmap_b, &full[stage],
                               c0 + a * 64, tap % 3, kg * kBlockK, tap / 3);
          } else if (!CONV && p.b_mn) {
#pragma unroll
            for (int a = 0; a < BLOCK_N / 64; a++)
              ptx::tma_load_2d(smem_b + stage * Cfg::kBBytes + a * (kBlockK * 128), &tmap_b, &full[stage],
                               n_blk * BLOCK_N + a * 64, kg * kBlockK);
          } else {
            ptx::tma_load_2d(smem_b + stage * Cfg::kBBytes, &tmap_b, &full[stage], kg * kBlockK, n_blk * BLOCK_N);
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ============================
    const uint32_t idesc = ptx::make_idesc_bf16_f32(kBlockM, BLOCK_N) | (p.a_mn ? 1u << 15 : 0u) | (p.b_mn ? 1u << 16 : 0u);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, it++) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      ptx::tcgen05_after_thread_sync();
      const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
      for (int kb = 0; kb < p.num_k_blocks; kb++) {
        ptx::mbar_wait(&full[stage], phase);
        ptx::tcgen05_after_thread_sync();
        if (lane == 0) {
          // K-major: advance 16 bf16 = 32 B inside the 128 B swizzle atom: +2 in the (>>4) address field.
          // MN-major: advance 16 k-rows of 128 B: +128 in the address field; LBO = the 8 KB mn-atom stride.
          const uint32_t sa = ptx::smem_u32(smem_a + stage * Cfg::kABytes), sb = ptx::smem_u32(smem_b + stage * Cfg::kBBytes);
          const uint64_t da = p.a_mn ? ptx::make_smem_desc_mn_sw128(sa, kBlockK * 128) : ptx::make_smem_desc_sw128(sa);
          const uint64_t db = p.b_mn ? ptx::make_smem_desc_mn_sw128(sb, kBlockK * 128) : ptx::make_smem_desc_sw128(sb);
          const uint64_t ia = p.a_mn ? 128 : 2, ib = p.b_mn ? 128 : 2;
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; k++) {
            ptx::umma_f16_ss(tmem_d, da + ia * k, db + ib * k, idesc, (kb | k) != 0);
          }
          ptx::umma_commit(&empty[stage]);
          if (kb == p.num_k_blocks - 1) ptx::umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ============================ epilogue ============================
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;     // accumulator row owned by this thread
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, it++) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int split = t / tiles_mn;
      const int mn = t % tiles_mn;
      const int n_blk = p.n_fast ? mn % p.num_n_tiles : mn / p.num_m_tiles;
      const int m_blk = p.n_fast ? mn / p.num_n_tiles : mn % p.num_m_tiles;
      ptx::mbar_wait(&tmem_full[acc], acc_phase);
      ptx::tcgen05_after_thread_sync();
      const uint32_t taddr = tmem_base + acc * BLOCK_N + (static_cast<uint32_t>(q * 32) << 16);
      epilogue_tile<BLOCK_N, CONV>(p, taddr, m_blk, n_blk, split, row, lane,
                                   [&]() { ptx::mbar_arrive(&tmem_empty[acc]); });
    }
  }
  ptx::tcgen05_before_thread_sync();
  __syncthreads();
  if (warp == 2) {
    ptx::tcgen05_after_thread_sync();
    ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------
// 2-CTA variant: a cluster of two CTAs (one TPC) computes a 256 x 256 output tile with
// tcgen05.mma.cta_group::2 (UMMA_M = 256).  Each CTA TMA-loads its own 128 A rows and HALF of the
// B tile (128 of the 256 N rows), so the B operand is fetched from L2 and staged in shared memory
// once per pair instead of once per CTA; accumulators land in each CTA's own TMEM and the epilogue
// is unchanged.  Barriers: `full` (leader's, 2 arrivals + both CTAs' TMA bytes), `empty` / `tmem_full`
// (per CTA, signalled by the leader's multicast tcgen05.commit), `tmem_empty` (leader's, 2x128
// epilogue arrivals, the peer's via mapa).
// ------------------------------------------------------------------------------------------
struct Gemm2Cfg {
  static constexpr int BLOCK_N = 256;
  static constexpr int kABytes = kBlockM * kBlockK * 2;          // 16 KB: this CTA's 128 rows of A
  static constexpr int kBBytes = (BLOCK_N / 2) * kBlockK * 2;    // 16 KB: this CTA's half of B
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = kSmemBudget / kStageBytes;      // 6
  static constexpr int kAccStages = 2;
  static constexpr int kTmemCols = kAccStages * BLOCK_N;         // 512
  static constexpr int kBarBytes = (2 * kStages + 2 * kAccStages) * 8 + 16;
  static constexpr int kSmemBytes = kStages * kStageBytes + kBarBytes + 1024;
};

template <bool CONV>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05_2sm(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                      const __grid_constant__ GemmParams p) {
  using Cfg = Gemm2Cfg;
  constexpr int BLOCK_N = Cfg::BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + Cfg::kStages;
  uint64_t* tmem_full = bars + 2 * Cfg::kStages;
  uint64_t* tmem_empty = tmem_full + Cfg::kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + Cfg::kAccStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::kStages; i++) {
      ptx::mbar_init(&full[i], 2);    // leader's own arrive.expect_tx + the peer's remote arrive
      ptx::mbar_init(&empty[i], 1);   // multicast commit
    }
    for (int i = 0; i < Cfg::kAccStages; i++) {
      ptx::mbar_init(&tmem_full[i], 1);
      ptx::mbar_init(&tmem_empty[i], 256);  // epilogue threads of both CTAs
    }
    ptx::fence_barrier_init();
  }
  ptx::cluster_sync();  // barriers of both CTAs initialised before any remote signal; required before 2-CTA TMEM alloc
  if (warp == 2) ptx::tmem_alloc_2sm(tmem_slot, Cfg::kTmemCols);
  ptx::tcgen05_before_thread_sync();
  ptx::cluster_sync();
  ptx::tcgen05_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int num_m_pairs = (p.num_m_tiles + 1) >> 1;
  const int tiles_mn = num_m_pairs * p.num_n_tiles;
  const int total_tiles = tiles_mn * p.k_splits;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0) {
    // ============================ TMA producer (both CTAs) ============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = cluster_id; t < total_tiles; t += num_clusters) {
        const int split = t / tiles_mn;
        const int mn = t % tiles_mn;
        const int n_blk = p.n_fast ? mn % p.num_n_tiles : mn / num_m_pairs;
        const int m_blk = (p.n_fast ? mn / p.num_n_tiles : mn % num_m_pairs) * 2 + (int)rank;
        const int kb0 = split * p.num_k_blocks;
        int img = 0, y0 = 0, x0 = 0;
        if (CONV) {
          const int tx = m_blk % p.tiles_x;
          const int ty = (m_blk / p.tiles_x) % p.tiles_y;
          img = m_blk / (p.tiles_x * p.tiles_y);  // >= n_img for the padding tile of an odd count: TMA zero-fills
          y0 = ty * p.cBH;
          x0 = tx * p.cBW;
        }
        for (int kb = 0; kb < p.num_k_blocks; kb++) {
          ptx::mbar_wait(&empty[stage], phase ^ 1);
          const int kg = kb0 + kb;
          if (CONV) {
            const int tap_all = kg / p.cin_blocks, cc = kg % p.cin_blocks;
            const int lvl = tap_all / p.taps, tap = tap_all % p.taps;
            const int dy = p.taps == 9 ? tap / 3 - 1 : 0, dx = p.taps == 9 ? tap % 3 - 1 : 0;
            const int im = img < p.lvl_img_stride ? img + lvl * p.lvl_img_stride : p.lvl_img_stride * p.levels;
            ptx::tma_load_4d_2sm(smem_a + stage * Cfg::kABytes, &tmap_a, &full[stage], cc * kBlockK, x0 + dx,
                                 y0 + dy, im);
          } else if (p.a_mn) {
            // MN-major A (backward GEMMs): two [64 k][64 m] boxes, one 128-byte swizzle atom of m each
#pragma unroll
            for (int a = 0; a < kBlockM / 64; a++)
              ptx::tma_load_2d_2sm(smem_a + stage * Cfg::kABytes + a * (kBlockK * 128), &tmap_a, &full[stage],
                                   m_blk * kBlockM + a * 64, kg * kBlockK);
          } else {
            ptx::tma_load_2d_2sm(smem_a + stage * Cfg::kABytes, &tmap_a, &full[stage], kg * kBlockK,
                                 m_blk * kBlockM);
          }
          const int nb0 = n_blk * BLOCK_N + (int)rank * (BLOCK_N / 2);    // this CTA's half of the B tile
          if (!CONV && p.b_mn == 2) {
            const int tap = nb0 / p.dw_cin, c0 = nb0 % p.dw_cin;
#pragma unroll
            for (int a = 0; a < BLOCK_N / 2 / 64; a++)
              ptx::tma_load_4d_2sm(smem_b + stage * Cfg::kBBytes + a * (kBlockK * 128), &tmap_b, &full[stage],
                                   c0 + a * 64, tap % 3, kg * kBlockK, tap / 3);
          } else if (!CONV && p.b_mn) {
#pragma unroll
            for (int a = 0; a < BLOCK_N / 2 / 64; a++)
              ptx::tma_load_2d_2sm(smem_b + stage * Cfg::kBBytes + a * (kBlockK * 128), &tmap_b, &full[stage],
                                   nb0 + a * 64, kg * kBlockK);
          } else {
            ptx::tma_load_2d_2sm(smem_b + stage * Cfg::kBBytes, &tmap_b, &full[stage], kg * kBlockK, nb0);
          }
          if (leader) {
            ptx::mbar_arrive_expect_tx(&full[stage], 2u * (uint32_t)(p.a_rows * kBlockK * 2 + Cfg::kBBytes));
          } else {
            ptx::mbar_arrive_cluster(&full[stage], 0);
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && leader) {
    // ============================ MMA issuer (leader CTA only) ============================
    const uint32_t idesc = ptx::make_idesc_bf16_f32(2 * kBlockM, BLOCK_N) | (p.a_mn ? 1u << 15 : 0u) | (p.b_mn ? 1u << 16 : 0u);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = cluster_id; t < total_tiles; t += num_clusters, it++) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      ptx::tcgen05_after_thread_sync();
      const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
      for (int kb = 0; kb < p.num_k_blocks; kb++) {
        ptx::mbar_wait(&full[stage], phase);
        ptx::tcgen05_after_thread_sync();
        if (lane == 0) {
          const uint32_t sa = ptx::smem_u32(smem_a + stage * Cfg::kABytes), sb = ptx::smem_u32(smem_b + stage * Cfg::kBBytes);
          const uint64_t da = p.a_mn ? ptx::make_smem_desc_mn_sw128(sa, kBlockK * 128) : ptx::make_smem_desc_sw128(sa);
          const uint64_t db = p.b_mn ? ptx::make_smem_desc_mn_sw128(sb, kBlockK * 128) : ptx::make_smem_desc_sw128(sb);
          const uint64_t ia = p.a_mn ? 128 : 2, ib = p.b_mn ? 128 : 2;
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; k++)
            ptx::umma_f16_ss_2sm(tmem_d, da + ia * k, db + ib * k, idesc, (kb | k) != 0);
          ptx::umma_commit_2sm(&empty[stage], 3);
          if (kb == p.num_k_blocks - 1) ptx::umma_commit_2sm(&tmem_full[acc], 3);
        }
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ============================ epilogue (both CTAs) ============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    int it = 0;
    for (int t = cluster_id; t < total_tiles; t += num_clusters, it++) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int split = t / tiles_mn;
      const int mn = t % tiles_mn;
      const int n_blk = p.n_fast ? mn % p.num_n_tiles : mn / num_m_pairs;
      const int m_blk = (p.n_fast ? mn / p.num_n_tiles : mn % num_m_pairs) * 2 + (int)rank;
      ptx::mbar_wait(&tmem_full[acc], acc_phase);
      ptx::tcgen05_after_thread_sync();
      const uint32_t taddr = tmem_base + acc * BLOCK_N + (static_cast<uint32_t>(q * 32) << 16);
      epilogue_tile<BLOCK_N, CONV>(p, taddr, m_blk, n_blk, split, row, lane,
                                   [&]() { ptx::mbar_arrive_cluster(&tmem_empty[acc], 0); });
    }
  }
  ptx::tcgen05_before_thread_sync();
  ptx::cluster_sync();  // nobody leaves while the peer may still signal its barriers / read its TMEM
  if (warp == 2) {
    ptx::tcgen05_after_thread_sync();
    ptx::tmem_dealloc_2sm(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// bf16 tensor map, rank 2..4; dims/box innermost first; strides (bytes) for dims 1..rank-1.
static int make_tmap(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims,
                     const cuuint64_t* strides_bytes, const cuuint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled unavailable (driver entry point lookup failed)");
    return G4R_ECUDA;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims,
                   strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: CUresult %d (rank %d, dims %llu,%llu box %u,%u)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return G4R_ECUDA;
  }
  return G4R_OK;
}

template <int BLOCK_N, bool CONV>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, cudaStream_t st) {
  using Cfg = GemmCfg<BLOCK_N>;
  static bool attr_set = false;
  auto kern = gemm_bf16_tcgen05<BLOCK_N, CONV>;
  if (!attr_set) {
    G4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const int total = p.num_m_tiles * p.num_n_tiles * p.k_splits;
  const int grid = total < sm_budget() ? total : sm_budget();
  kern<<<grid, kGemmThreads, Cfg::kSmemBytes, st>>>(ta, tb, p);
  G4R_LAUNCH_CHECK("gemm_bf16_tcgen05");
  return G4R_OK;
}

template <bool CONV>
static int launch_gemm_2sm(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, cudaStream_t st) {
  using Cfg = Gemm2Cfg;
  static bool attr_set = false;
  auto kern = gemm_bf16_tcgen05_2sm<CONV>;
  if (!attr_set) {
    G4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const int pairs = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles * p.k_splits;
  const int max_clusters = sm_budget() / 2;
  const int clusters = pairs < max_clusters ? pairs : max_clusters;
  kern<<<2 * clusters, kGemmThreads, Cfg::kSmemBytes, st>>>(ta, tb, p);  // __cluster_dims__(2,1,1)
  G4R_LAUNCH_CHECK("gemm_bf16_tcgen05_2sm");
  return G4R_OK;
}

// 2-CTA tiles (cta_group::2, UMMA_M = 256) whenever there is enough work to keep all SM pairs busy.  Measured on
// B200, round 2 (profiles/r2_gemm_2sm_ab.md): the 2-CTA kernel beats the 1-CTA kernel on every LLaMA shape
// (qkv 1416 vs 1317, o 1322 vs 1253, gate/up 1470 vs 1415, down 1413 vs 1305 TFLOP/s under ncu) although
// M = B*L = 5648 rows leave a 94 %-empty last 256-row pair, and runs the convs at 1.58 PFLOP/s; whole step 106.0 vs
// 107.4 ms.
static bool use_2sm(int N, int m_tiles, int k_splits) {
  if (N <= 128 || m_tiles < 2) return false;
  const long pairs = (long)((m_tiles + 1) / 2) * ((N + 255) / 256) * k_splits;
  return pairs >= num_sms() / 2;
}

static int pick_block_n(int N, int m_tiles, int k_splits) {
  // 256-wide tiles feed the tensor core best; fall back to 128 when that leaves SMs idle.
  if (N <= 128) return 128;
  const long t256 = (long)m_tiles * ((N + 255) / 256) * k_splits;
  if (t256 >= num_sms()) return 256;
  return 128;
}

}  // namespace g4r

using namespace G4R_NS;

extern "C" int g4r_gemm_bf16(const void* A, long long lda, const void* B, long long ldb, void* D,
                             long long ldd, int M, int N, int K, const void* bias, int bias_f32,
                             const void* residual, long long ldr, int act, int out_f32, int k_splits,
                             void* stream);
extern "C" int g4r_gemm_bf16_ex(const void* A, long long lda, const void* B, long long ldb, void* D,
                                long long ldd, int M, int N, int K, const void* bias, int bias_f32,
                                const void* residual, long long ldr, int residual_f32, int bias_round_bf16,
                                int act, int out_f32, int k_splits, void* stream);
extern "C" int g4r_gemm_bf16(const void* A, long long lda, const void* B, long long ldb, void* D,
                             long long ldd, int M, int N, int K, const void* bias, int bias_f32,
                             const void* residual, long long ldr, int act, int out_f32, int k_splits,
                             void* stream) {
  return g4r_gemm_bf16_ex(A, lda, B, ldb, D, ldd, M, N, K, bias, bias_f32, residual, ldr, 0, 0, act, out_f32,
                          k_splits, stream);
}

static int gemm_impl(const void* A, long long lda, const void* B, long long ldb, void* D, long long ldd, int M,
                     int N, int K, const void* bias, int bias_f32, const void* residual, long long ldr,
                     int residual_f32, int bias_round_bf16, int act, int out_f32, int k_splits,
                     const void* rope_cos, const void* rope_sin, int rope_cols, int rope_L, void* stream,
                     int rope_pos0 = 0, const int* rope_pos_dev = nullptr);

namespace G4R_NS {
// gemm_skinny.cu: M <= 16 weight-streaming path; returns -1 when the shape does not qualify
int gemm_skinny_dispatch(const void* A, long long lda, const void* B, long long ldb, void* D, long long ldd, int M,
                         int N, int K, const void* bias, int bias_f32, const void* residual, long long ldr, int act,
                         const void* rope_cos, const void* rope_sin, int rope_cols, int rope_L, int rope_pos0,
                         const int* rope_pos_dev, void* stream);
}

extern "C" int g4r_gemm_bf16_ex(const void* A, long long lda, const void* B, long long ldb, void* D,
                                long long ldd, int M, int N, int K, const void* bias, int bias_f32,
                                const void* residual, long long ldr, int residual_f32, int bias_round_bf16,
                                int act, int out_f32, int k_splits, void* stream) {
  return gemm_impl(A, lda, B, ldb, D, ldd, M, N, K, bias, bias_f32, residual, ldr, residual_f32, bias_round_bf16,
                   act, out_f32, k_splits, nullptr, nullptr, 0, 0, stream);
}

// QKV projection with the rotary embedding fused into the epilogue: D[M, N] = A.B^T, columns
// [0, rope_cols) (the q and k heads, head_dim 128) rotated with cos/sin[row % L].  Replaces
// q_proj/k_proj/v_proj + apply_rotary_pos_emb (transformers modeling_llama.py:138-168,240-260).
extern "C" int g4r_gemm_qkv_rope_bf16(const void* A, long long lda, const void* B, long long ldb, void* D,
                                      long long ldd, int M, int N, int K, const void* rope_cos,
                                      const void* rope_sin, int rope_cols, int L, int pos0, const int* pos0_dev,
                                      void* stream) {
  G4R_REQUIRE(rope_cos && rope_sin && L > 0, "qkv_rope: null tables");
  G4R_REQUIRE(rope_cols % 256 == 0 && rope_cols <= N && N % 128 == 0 && ldd % 8 == 0, "qkv_rope: rope_cols must be a multiple of 256 (whole tiles of 128-dim heads)");
  return gemm_impl(A, lda, B, ldb, D, ldd, M, N, K, nullptr, 0, nullptr, 0, 0, 0, ACT_NONE, 0, 1, rope_cos, rope_sin,
                   rope_cols, L, stream, pos0, pos0_dev);
}

// Backward-pass GEMM: D[M, N] = op(A) . op(B)^T with either operand optionally stored "MN-major":
//   a_mn = 0: A is [M, K] (K contiguous, row stride lda);  a_mn = 1: A is stored [K, M] (M contiguous, lda >= M)
//   b_mn = 0: B is [N, K] (K contiguous, row stride ldb);  b_mn = 1: B is stored [K, N] (N contiguous, ldb >= N)
// so that for y = x W^T (W [N_out, K_in], nn.Linear):
//   dX[M, K_in]      = dY[M, N_out] . W          -> A = dY (a_mn 0), B = W  (b_mn 1, contraction N_out)
//   dW[N_out, K_in]  = dY^T . X                  -> A = dY (a_mn 1), B = X  (b_mn 1, contraction M tokens)
// The transposes happen in the tensor-core operand descriptors (UMMA major bits), never in memory.
// Replaces the autograd of F.linear inside the stage-2 training step (gpt4roi/train/train.py:698-712).
#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_gemm_bf16_t(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, void* D,
                               long long ldd, int M, int N, int K, int out_f32, void* stream) {
  G4R_REQUIRE(A && B && D, "null operand");
  G4R_REQUIRE(M > 0 && N > 0 && K > 0, "bad sizes M=%d N=%d K=%d", M, N, K);
  G4R_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "lda/ldb must be multiples of 8 (16-byte TMA strides)");
  G4R_REQUIRE(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "lda/ldb smaller than the contiguous extent");
  G4R_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0, "A/B must be 16-byte aligned");
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
  p.k_splits = 1;
  p.num_k_blocks = (K + kBlockK - 1) / kBlockK;
  p.D = D; p.ldd = ldd; p.out_f32 = out_f32;
  p.a_rows = kBlockM;
  p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0;
  // 2-CTA tiles for the backward GEMMs too; MN-major boxes are 64 x 64 either way
  const bool two = N % 256 == 0 && use_2sm(N, p.num_m_tiles, 1);
  const int bn = two ? 256 : pick_block_n(N, p.num_m_tiles, 1);
  p.num_n_tiles = (N + bn - 1) / bn;
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[2] = {(cuuint64_t)(a_mn ? M : K), (cuuint64_t)(a_mn ? K : M)};
    cuuint64_t str[1] = {(cuuint64_t)lda * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(a_mn ? kBlockK : kBlockM)};
    int rc = make_tmap(&ta, A, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)(b_mn ? N : K), (cuuint64_t)(b_mn ? K : N)};
    cuuint64_t str[1] = {(cuuint64_t)ldb * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(b_mn ? kBlockK : (two ? bn / 2 : bn))};
    int rc = make_tmap(&tb, B, 2, dims, str, box);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (two) return launch_gemm_2sm<false>(ta, tb, p, st);
  return bn == 256 ? launch_gemm<256, false>(ta, tb, p, st) : launch_gemm<128, false>(ta, tb, p, st);
}
#endif

// Weight gradient of a 3x3 / stride 1 / pad 1 convolution (NHWC, bf16) as ONE tensor-core GEMM on the
// zero-padded layout:  dW[co, ky, kx, ci] = sum_rows dz_pad[row, co] * x_pad[row + (ky-1)*(W+2) + (kx-1), ci]
// where rows run over n_img*(H+2)*(W+2) padded pixels (dz_pad is zero on the padding ring, so wrapped
// neighbours contribute nothing).  A = dz_pad as an MN-major operand; B = x_pad through an aliasing 4-D tensor
// map (b_mn == 2), so all nine taps are column blocks of one launch (8 x 36 tiles for 1024 -> 1024).
// x_pad_origin points at the row of x_pad that tap (0,0) pairs with row 0, i.e. (W+2)+1 rows before the first
// real row; the caller keeps >= (W+2)+1 zero guard rows on both ends.  dW is fp32 [Cout, 9*Cin]; accumulate != 0
// adds to it (the four pyramid levels of a fuse round share one weight, gpt4roi/models/layers.py:152-180).
#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_conv3x3_dw_bf16(const void* dz_pad, const void* x_pad_origin, float* dW, long long rows, int Wp,
                                   int Cin, int Cout, int accumulate, void* stream) {
  G4R_REQUIRE(dz_pad && x_pad_origin && dW && rows > 0 && Wp > 2, "conv3x3_dw: bad arguments");
  G4R_REQUIRE(Cin % 256 == 0 && Cout % 8 == 0, "conv3x3_dw: Cin=%d must be a multiple of 256, Cout=%d of 8", Cin, Cout);
  G4R_REQUIRE((((uintptr_t)dz_pad | (uintptr_t)x_pad_origin) & 15) == 0, "conv3x3_dw: misaligned operands");
  GemmParams p{};
  p.M = Cout; p.N = 9 * Cin; p.K = (int)rows;
  p.num_m_tiles = (Cout + kBlockM - 1) / kBlockM;
  p.k_splits = 1;
  p.num_k_blocks = (int)((rows + kBlockK - 1) / kBlockK);
  p.D = dW; p.ldd = 9LL * Cin; p.out_f32 = 1;
  if (accumulate) { p.residual = reinterpret_cast<const __nv_bfloat16*>(dW); p.residual_f32 = 1; p.ldr = p.ldd; }
  p.a_rows = kBlockM;
  p.a_mn = 1; p.b_mn = 2; p.dw_cin = Cin;
  const int bn = 256;
  p.num_n_tiles = p.N / bn;
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[2] = {(cuuint64_t)Cout, (cuuint64_t)rows};
    cuuint64_t str[1] = {(cuuint64_t)Cout * 2};
    cuuint32_t box[2] = {64, kBlockK};
    int rc = make_tmap(&ta, dz_pad, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    // dimension order {ci, kx, row, ky}: every stride is a multiple of the previous one (driver requirement)
    cuuint64_t dims[4] = {(cuuint64_t)Cin, 3, (cuuint64_t)rows, 3};
    cuuint64_t str[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cin * 2, (cuuint64_t)Wp * Cin * 2};
    cuuint32_t box[4] = {64, 1, kBlockK, 1};
    int rc = make_tmap(&tb, x_pad_origin, 4, dims, str, box);
    if (rc) return rc;
  }
  if (use_2sm(p.N, p.num_m_tiles, 1)) return launch_gemm_2sm<false>(ta, tb, p, (cudaStream_t)stream);
  return launch_gemm<256, false>(ta, tb, p, (cudaStream_t)stream);
}
#endif

static int gemm_impl(const void* A, long long lda, const void* B, long long ldb, void* D, long long ldd, int M,
                     int N, int K, const void* bias, int bias_f32, const void* residual, long long ldr,
                     int residual_f32, int bias_round_bf16, int act, int out_f32, int k_splits,
                     const void* rope_cos, const void* rope_sin, int rope_cols, int rope_L, void* stream,
                     int rope_pos0, const int* rope_pos_dev) {
  G4R_REQUIRE(A && B && D, "null operand");
  G4R_REQUIRE(M > 0 && N > 0 && K > 0, "bad sizes M=%d N=%d K=%d", M, N, K);
  G4R_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && lda >= K && ldb >= K, "lda/ldb must be >= K and multiples of 8 (16-byte TMA strides)");
  G4R_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0, "A/B must be 16-byte aligned");
  G4R_REQUIRE(act >= ACT_NONE && act <= ACT_SWIGLU, "act=%d", act);
  G4R_REQUIRE(k_splits >= 1, "k_splits=%d", k_splits);
  if (act == ACT_SWIGLU) G4R_REQUIRE(N % 2 == 0 && !out_f32 && k_splits == 1 && !residual, "SwiGLU epilogue: even N, bf16 out, no split-K/residual");
  if (k_splits > 1) G4R_REQUIRE(out_f32 && act == ACT_NONE && !residual && !bias, "split-K writes fp32 partial slabs [k_splits][M][ldd]: out_f32, no bias/act/residual");
  // M <= 16 (decode step): HBM-bound weight-streaming kernel instead of a mostly empty 128-row tile
  if (M <= 16 && !out_f32 && k_splits == 1 && !residual_f32 && !bias_round_bf16) {
    const int rc = gemm_skinny_dispatch(A, lda, B, ldb, D, ldd, M, N, K, bias, bias_f32, residual, ldr, act, rope_cos,
                                        rope_sin, rope_cols, rope_L, rope_pos0, rope_pos_dev, stream);
    if (rc >= 0) return rc;
  }
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
  const int kb_total = (K + kBlockK - 1) / kBlockK;
  G4R_REQUIRE(kb_total % k_splits == 0, "K blocks (%d) not divisible by k_splits (%d)", kb_total, k_splits);
  p.k_splits = k_splits;
  p.num_k_blocks = kb_total / k_splits;
  p.D = D; p.ldd = ldd; p.bias = bias; p.bias_f32 = bias_f32;
  p.residual = (const __nv_bfloat16*)residual; p.ldr = ldr; p.residual_f32 = residual_f32;
  p.round_branch = bias_round_bf16;
  p.rope_cos = (const __nv_bfloat16*)rope_cos; p.rope_sin = (const __nv_bfloat16*)rope_sin;
  p.rope_cols = rope_cols; p.rope_L = rope_L; p.rope_pos0 = rope_pos0; p.rope_pos_dev = rope_pos_dev;
  p.act = act; p.out_f32 = out_f32; p.atomic = k_splits > 1;
  p.conv = 0; p.a_rows = kBlockM;
  const bool two = use_2sm(N, p.num_m_tiles, k_splits);
  const int bn = two ? 256 : pick_block_n(N, p.num_m_tiles, k_splits);
  p.num_n_tiles = (N + bn - 1) / bn;
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)M};
    cuuint64_t str[1] = {(cuuint64_t)lda * 2};
    cuuint32_t box[2] = {kBlockK, kBlockM};
    int rc = make_tmap(&ta, A, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
    cuuint64_t str[1] = {(cuuint64_t)ldb * 2};
    cuuint32_t box[2] = {kBlockK, (cuuint32_t)(two ? bn / 2 : bn)};
    int rc = make_tmap(&tb, B, 2, dims, str, box);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (two) return launch_gemm_2sm<false>(ta, tb, p, st);
  return bn == 256 ? launch_gemm<256, false>(ta, tb, p, st) : launch_gemm<128, false>(ta, tb, p, st);
}

// spatial tiling used by the conv kernel for an H x W map (also tells callers how many GN partial slots exist)
static void conv_tiling(int H, int W, int* bw_out, int* bh_out) {
  int bw = W >= 16 && W % 16 == 0 ? 16 : (W >= 8 ? 8 : W);
  if (W == 14) bw = 14;
  int bh = kBlockM / bw;
  if (bh > H) bh = H;
  *bw_out = bw;
  *bh_out = bh;
}

#if G4R_BF16_ONLY   // independent of the activation type: built once
extern "C" int g4r_conv_gn_slots(int H, int W) {
  int bw, bh;
  conv_tiling(H, W, &bw, &bh);
  return ((W + bw - 1) / bw) * ((H + bh - 1) / bh) * 4;
}
#endif

extern "C" int g4r_conv_nhwc_bf16(const void* X, const void* Wt, void* Y, int n_img, int H, int W, int Cin,
                                  int Cout, int ksize, int levels, const void* bias, int bias_f32, int act,
                                  float* gn_stats, int gn_groups, void* stream) {
  G4R_REQUIRE(X && Wt && Y, "null operand");
  G4R_REQUIRE(ksize == 3 || ksize == 1, "ksize=%d (1 or 3)", ksize);
  G4R_REQUIRE(Cin % kBlockK == 0, "Cin=%d must be a multiple of 64", Cin);
  G4R_REQUIRE(Cout % 8 == 0, "Cout=%d must be a multiple of 8", Cout);
  G4R_REQUIRE(n_img > 0 && H > 0 && W > 0, "bad sizes");
  G4R_REQUIRE(levels >= 1 && levels <= 8, "levels=%d", levels);
  G4R_REQUIRE(act == ACT_NONE || act == ACT_RELU, "conv epilogue: none or relu");
  if (gn_stats) G4R_REQUIRE(gn_groups > 0 && Cout % gn_groups == 0 && Cout / gn_groups == 16, "GN stats need 16-channel groups");
  GemmParams p{};
  // spatial tile: BW x BH = 128 output pixels (or fewer for small maps)
  int bw, bh;
  conv_tiling(H, W, &bw, &bh);
  p.cBW = bw; p.cBH = bh; p.cH = H; p.cW = W;
  p.tiles_x = (W + bw - 1) / bw;
  p.tiles_y = (H + bh - 1) / bh;
  p.a_rows = bw * bh;
  p.M = n_img * H * W; p.N = Cout; p.K = levels * ksize * ksize * Cin;
  p.levels = levels; p.lvl_img_stride = n_img;
  p.num_m_tiles = n_img * p.tiles_x * p.tiles_y;
  p.cin_blocks = Cin / kBlockK;
  p.taps = ksize * ksize;
  p.num_k_blocks = levels * p.taps * p.cin_blocks;
  p.k_splits = 1;
  p.D = Y; p.ldd = Cout; p.bias = bias; p.bias_f32 = bias_f32; p.act = act;
  p.conv = 1;
  p.n_fast = 1;
  p.gn_stats = gn_stats; p.gn_groups = gn_groups; p.gn_group_ch = gn_groups ? Cout / gn_groups : 0;
  const bool two = use_2sm(Cout, p.num_m_tiles, 1);
  const int bn = two ? 256 : pick_block_n(Cout, p.num_m_tiles, 1);
  p.num_n_tiles = (Cout + bn - 1) / bn;
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_img * levels};
    cuuint64_t str[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2};
    cuuint32_t box[4] = {kBlockK, (cuuint32_t)bw, (cuuint32_t)bh, 1};
    int rc = make_tmap(&ta, X, 4, dims, str, box);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)Cout};
    cuuint64_t str[1] = {(cuuint64_t)p.K * 2};
    cuuint32_t box[2] = {kBlockK, (cuuint32_t)(two ? bn / 2 : bn)};
    int rc = make_tmap(&tb, Wt, 2, dims, str, box);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (two) return launch_gemm_2sm<true>(ta, tb, p, st);
  return bn == 256 ? launch_gemm<256, true>(ta, tb, p, st) : launch_gemm<128, true>(ta, tb, p, st);
}
