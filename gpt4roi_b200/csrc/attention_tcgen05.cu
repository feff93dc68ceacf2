// attention_tcgen05.cu -- fused attention forward on the 5th-gen tensor cores (sm_100a):
//   O = softmax(Q K^T * scale [+ causal / length mask]) V,   one CTA = 128 queries of one (batch, head)
//
// Replaces transformers' eager attention (modeling_llama.py:199-222, modeling_clip.py) that the
// reference calls for every LLaMA / CLIP layer, without materialising the [B,H,L,L] scores.
//
//   warp 0      TMA producer: Q tile once, then K_j / V_j tiles (128 keys) into 2-stage rings
//               (cp.async.bulk.tensor, 128-byte swizzle, [128 rows x 64 cols] atoms)
//   warp 1      MMA issuer (one thread):  S_j = Q K_j^T  -> TMEM (double-buffered, 128 fp32 cols each)
//                                        O  += P_j V_j  -> TMEM (D fp32 cols); V is consumed as an
//               MN-major B operand straight from its [keys][d] layout (no transpose pass)
//   warp 2      TMEM allocator (512 columns)
//   warps 4..7  softmax: thread r owns query row r == TMEM lane r -> no cross-thread reductions.
//               pass 1 tcgen05.ld S -> row max; rescale O in TMEM (tcgen05.ld/st) by exp2(m_old-m_new);
//               pass 2 tcgen05.ld S -> p = exp2(s*c - m*c) -> bf16 -> swizzled smem tile P (A operand of PV)
// QK_{j+1} is issued before PV_j so the tensor core works on the next scores while the softmax
// warps process block j.  Scores stay fp32 through the softmax (see attention.cu header).
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"
#include "act_type.cuh"   // bf16 as written; fp16 twin with -DG4R_ACT_HALF

namespace G4R_NS {

constexpr int kFaBM = 128;
// keys per block.  64 keeps a CTA at 112 KB of shared memory and 256 TMEM columns (D=128), so TWO CTAs share an SM:
// one CTA's prologue / epilogue overlaps the other's MMAs and 8 softmax warps instead of 4 hide the tcgen05.ld / MUFU
// latencies.
constexpr int kFaBN = 64;
constexpr int kFaThreads = 256;
constexpr int kAtomBytes = 128 * 128;  // [128 rows][64 bf16] swizzle-128B atom (Q, P)

struct FaParams {
  __nv_bfloat16* out;
  long long ldo, bso;
  int L, H;
  float scale;
  const int* seqlens;
  float* lse;   // optional [B, H, L]: natural-log sum-exp of the scaled scores (training forward; attention_bwd reads it)
};

__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]),
      "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]),
      "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

using ptx::make_smem_desc_mn_sw128;  // V tile [keys][d] (d contiguous) is an MN-major B operand

template <int D, bool CAUSAL>
__global__ void __launch_bounds__(kFaThreads, 2)
fa_fwd_tcgen05(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
               const __grid_constant__ CUtensorMap tm_v, const __grid_constant__ FaParams p) {
  constexpr int ATOMS = D / 64;
  constexpr int Q_BYTES = ATOMS * kAtomBytes;        // Q tile: 128 rows x D
  constexpr int KV_ATOM = kFaBN * 128;               // [kFaBN keys][64 bf16]
  constexpr int TILE_BYTES = ATOMS * KV_ATOM;        // K / V tile: kFaBN rows x D
  constexpr int P_BYTES = (kFaBN / 64) * kAtomBytes; // P: 128 x kFaBN keys
  constexpr int TMEM_COLS = (2 * kFaBN + D) <= 256 ? 256 : 512;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Q_BYTES;          // 2 stages
  uint8_t* sV = sK + 2 * TILE_BYTES;   // 2 stages
  uint8_t* sP = sV + 2 * TILE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + P_BYTES);
  uint64_t* q_full = bars;           // 1
  uint64_t* k_full = bars + 1;       // 2
  uint64_t* k_empty = bars + 3;      // 2
  uint64_t* v_full = bars + 5;       // 2
  uint64_t* v_empty = bars + 7;      // 2
  uint64_t* s_full = bars + 9;       // 2
  uint64_t* s_free = bars + 11;      // 2
  uint64_t* p_full = bars + 13;      // 1
  uint64_t* pv_done = bars + 14;     // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // heaviest query blocks first (causal: block i attends to i+1 key blocks): the long CTAs start early and the
  // short ones fill the tail of the last wave (LPT order)
  const int qb = CAUSAL ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = qb * kFaBM;
  const int row_base = b * p.L;
  const int Lk = p.seqlens ? min(max(p.seqlens[b], 1), p.L) : p.L;
  const int nblk = CAUSAL ? min((Lk + kFaBN - 1) / kFaBN, (q0 + kFaBM + kFaBN - 1) / kFaBN) : (Lk + kFaBN - 1) / kFaBN;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tm_q);
    ptx::prefetch_tensormap(&tm_k);
    ptx::prefetch_tensormap(&tm_v);
  }
  if (warp == 1 && lane == 0) {
    ptx::mbar_init(q_full, 1);
    for (int i = 0; i < 2; i++) {
      ptx::mbar_init(&k_full[i], 1);
      ptx::mbar_init(&k_empty[i], 1);
      ptx::mbar_init(&v_full[i], 1);
      ptx::mbar_init(&v_empty[i], 1);
      ptx::mbar_init(&s_full[i], 1);
      ptx::mbar_init(&s_free[i], 128);
    }
    ptx::mbar_init(p_full, 128);
    ptx::mbar_init(pv_done, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_slot, TMEM_COLS);
  ptx::tcgen05_before_thread_sync();
  __syncthreads();
  ptx::tcgen05_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_o = tmem_base + 2 * kFaBN;

  if (warp == 0) {
    // ============================ TMA producer ============================
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(q_full, Q_BYTES);
      for (int a = 0; a < ATOMS; a++)
        ptx::tma_load_2d(sQ + a * kAtomBytes, &tm_q, q_full, h * D + a * 64, row_base + q0);
      for (int j = 0; j < nblk; j++) {
        const int st = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        ptx::mbar_wait(&k_empty[st], ph ^ 1);
        ptx::mbar_arrive_expect_tx(&k_full[st], TILE_BYTES);
        for (int a = 0; a < ATOMS; a++)
          ptx::tma_load_2d(sK + st * TILE_BYTES + a * KV_ATOM, &tm_k, &k_full[st], h * D + a * 64,
                           row_base + j * kFaBN);
        ptx::mbar_wait(&v_empty[st], ph ^ 1);
        ptx::mbar_arrive_expect_tx(&v_full[st], TILE_BYTES);
        for (int a = 0; a < ATOMS; a++)
          ptx::tma_load_2d(sV + st * TILE_BYTES + a * KV_ATOM, &tm_v, &v_full[st], h * D + a * 64,
                           row_base + j * kFaBN);
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ============================
    constexpr uint32_t idesc_qk = ptx::make_idesc_bf16_f32(kFaBM, kFaBN);
    constexpr uint32_t idesc_pv = ptx::make_idesc_bf16_f32(kFaBM, D) | (1u << 16);  // B (= V) is MN-major
    ptx::mbar_wait(q_full, 0);
    auto issue_qk = [&](int j) {
      const int st = j & 1, sb = j & 1;
      const uint32_t ph = (j >> 1) & 1;
      ptx::mbar_wait(&k_full[st], ph);
      ptx::mbar_wait(&s_free[sb], ph ^ 1);
      ptx::tcgen05_after_thread_sync();
      if (lane == 0) {
#pragma unroll
        for (int kk = 0; kk < D / 16; kk++) {
          const uint64_t da = ptx::make_smem_desc_sw128(ptx::smem_u32(sQ + (kk >> 2) * kAtomBytes)) + 2 * (kk & 3);
          const uint64_t db =
              ptx::make_smem_desc_sw128(ptx::smem_u32(sK + st * TILE_BYTES + (kk >> 2) * KV_ATOM)) + 2 * (kk & 3);
          ptx::umma_f16_ss(tmem_base + sb * kFaBN, da, db, idesc_qk, kk != 0);
        }
        ptx::umma_commit(&s_full[sb]);
        ptx::umma_commit(&k_empty[st]);
      }
      __syncwarp();
    };
    issue_qk(0);
    for (int j = 0; j < nblk; j++) {
      if (j + 1 < nblk) issue_qk(j + 1);
      const int st = j & 1;
      ptx::mbar_wait(p_full, j & 1);
      ptx::mbar_wait(&v_full[st], (j >> 1) & 1);
      ptx::tcgen05_after_thread_sync();
      if (lane == 0) {
#pragma unroll
        for (int ks = 0; ks < kFaBN / 16; ks++) {
          const uint64_t da = ptx::make_smem_desc_sw128(ptx::smem_u32(sP + (ks >> 2) * kAtomBytes)) + 2 * (ks & 3);
          const uint64_t db = make_smem_desc_mn_sw128(ptx::smem_u32(sV + st * TILE_BYTES + ks * 2048), KV_ATOM);
          ptx::umma_f16_ss(tmem_o, da, db, idesc_pv, (j | ks) != 0);
        }
        ptx::umma_commit(pv_done);
        ptx::umma_commit(&v_empty[st]);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ============================ softmax / correction / epilogue ============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int qrow = q0 + row;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const float c = p.scale * 1.4426950408889634f;
    // m_used: the row maximum the running sums are expressed against.  It is only advanced (and O / l
    // rescaled) when the true maximum grew by more than 2^kTau -- exponentials stay <= 2^kTau, exact in
    // fp32 and harmless in bf16 -- so the TMEM read-modify-write of O is skipped for almost every block.
    constexpr float kTau = 8.0f;
    float m_used = -INFINITY, l_run = 0.f;
    for (int j = 0; j < nblk; j++) {
      const int sb = j & 1;
      ptx::mbar_wait(&s_full[sb], (j >> 1) & 1);
      ptx::tcgen05_after_thread_sync();
      const uint32_t ts = tmem_base + sb * kFaBN + lane_off;
      const int key0 = j * kFaBN;
      const bool need_mask = (key0 + kFaBN > Lk) || (CAUSAL && key0 + kFaBN - 1 > q0);
      // ---- one TMEM read of the score row (kept in registers for both the max and the exponentials)
      uint32_t sv[kFaBN / 32][32];
#pragma unroll
      for (int cc = 0; cc < kFaBN / 32; cc++) ptx::tmem_ld_32x32b_x32(ts + cc * 32, sv[cc]);
      ptx::tmem_ld_wait();
      ptx::tcgen05_before_thread_sync();
      ptx::mbar_arrive(&s_free[sb]);  // S buffer may be overwritten by QK_{j+2}
      float mx = -INFINITY;
#pragma unroll
      for (int cc = 0; cc < kFaBN / 32; cc++) {
#pragma unroll
        for (int i = 0; i < 32; i++) {
          float sc = __uint_as_float(sv[cc][i]);
          if (need_mask) {
            const int key = key0 + cc * 32 + i;
            if (key >= Lk || (CAUSAL && key > qrow)) sc = -INFINITY;
            sv[cc][i] = __float_as_uint(sc);
          }
          mx = fmaxf(mx, sc);
        }
      }
      const float m_new = fmaxf(m_used, mx);
      const bool grow = (m_new - m_used) * c > kTau;  // false when both are -inf (NaN compare)
      float alpha = 1.f;
      if (grow) {
        alpha = exp2f((m_used - m_new) * c);  // m_used = -inf -> 0
        m_used = m_new;
      }
      const float mc = (m_used == -INFINITY ? 0.f : m_used) * c;
      // ---- exponentials -> bf16 (registers)
      uint32_t pk[kFaBN / 2];
      float lsum = 0.f;
#pragma unroll
      for (int cc = 0; cc < kFaBN / 32; cc++) {
#pragma unroll
        for (int i = 0; i < 16; i++) {
          const float p0 = exp2f(fmaf(__uint_as_float(sv[cc][2 * i]), c, -mc));
          const float p1 = exp2f(fmaf(__uint_as_float(sv[cc][2 * i + 1]), c, -mc));
          lsum += p0 + p1;
          __nv_bfloat162 hh = __floats2bfloat162_rn(p0, p1);
          pk[cc * 16 + i] = *reinterpret_cast<uint32_t*>(&hh);
        }
      }
      l_run = l_run * alpha + lsum;
      // ---- P buffer free and O consistent once PV_{j-1} has completed
      if (j > 0) {
        ptx::mbar_wait(pv_done, (j - 1) & 1);
        ptx::tcgen05_after_thread_sync();
        if (__any_sync(0xffffffffu, grow)) {  // warp-uniform: tcgen05.ld/st are warp-collective
#pragma unroll 1
          for (int cc = 0; cc < D / 32; cc++) {
            uint32_t v[32];
            ptx::tmem_ld_32x32b_x32(tmem_o + lane_off + cc * 32, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; i++) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
            tmem_st_32x32b_x32(tmem_o + lane_off + cc * 32, v);
          }
          tmem_st_wait();
        }
      }
      // ---- P -> swizzled smem tile (A operand of the PV product): 32 keys = 4 16-byte chunks of this row
      // inside atom (cc>>1); chunk index (cc&1)*4 + t, XOR-swizzled by row&7
#pragma unroll
      for (int cc = 0; cc < kFaBN / 32; cc++) {
        uint8_t* prow = sP + (cc >> 1) * kAtomBytes + row * 128;
#pragma unroll
        for (int t = 0; t < 4; t++) {
          const int chunk = ((cc & 1) * 4 + t) ^ (row & 7);
          *reinterpret_cast<uint4*>(prow + chunk * 16) =
              make_uint4(pk[cc * 16 + 4 * t], pk[cc * 16 + 4 * t + 1], pk[cc * 16 + 4 * t + 2], pk[cc * 16 + 4 * t + 3]);
        }
      }
      ptx::tcgen05_before_thread_sync();
      ptx::fence_proxy_async_smem();
      ptx::mbar_arrive(p_full);
    }
    // ---- epilogue: O / l -> bf16 -> global (thread = row: D contiguous elements)
    ptx::mbar_wait(pv_done, (nblk - 1) & 1);
    ptx::tcgen05_after_thread_sync();
    const float inv = 1.f / l_run;
    if (p.lse != nullptr && qrow < p.L)   // p = 2^((s - m_used) c) = e^(scale (s - m_used))  =>  lse = scale m_used + ln l
      p.lse[((long long)b * p.H + h) * p.L + qrow] = (m_used == -INFINITY ? 0.f : m_used) * p.scale + logf(l_run);
    __nv_bfloat16* orow = p.out + (long long)b * p.bso + (long long)qrow * p.ldo + (long long)h * D;
#pragma unroll 1
    for (int cc = 0; cc < D / 32; cc++) {
      uint32_t v[32];
      ptx::tmem_ld_32x32b_x32(tmem_o + lane_off + cc * 32, v);
      ptx::tmem_ld_wait();
      if (qrow < p.L) {
#pragma unroll
        for (int t = 0; t < 4; t++) {
          uint32_t pk[4];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            __nv_bfloat162 hh = __floats2bfloat162_rn(__uint_as_float(v[t * 8 + 2 * i]) * inv,
                                                       __uint_as_float(v[t * 8 + 2 * i + 1]) * inv);
            pk[i] = *reinterpret_cast<uint32_t*>(&hh);
          }
          *reinterpret_cast<uint4*>(orow + cc * 32 + t * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
  }
  ptx::tcgen05_before_thread_sync();
  __syncthreads();
  if (warp == 2) {
    ptx::tcgen05_after_thread_sync();
    ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);

static int make_tmap_rows(CUtensorMap* m, const void* base, long long cols, long long rows, long long ld,
                          int box_rows) {
  static EncodeTiledFn2 enc = nullptr;
  if (!enc) {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled unavailable");
      return G4R_ECUDA;
    }
    enc = reinterpret_cast<EncodeTiledFn2>(fp);
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t str[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, str, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("attention: cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return G4R_ECUDA;
  }
  return G4R_OK;
}

template <int D, bool CAUSAL>
static int launch_fa(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const FaParams& p, int B,
                     cudaStream_t st) {
  constexpr int smem = (D / 64) * kAtomBytes + 4 * (D / 64) * kFaBN * 128 + (kFaBN / 64) * kAtomBytes + 256;
  static bool set = false;
  auto kern = fa_fwd_tcgen05<D, CAUSAL>;
  if (!set) {
    G4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    set = true;
  }
  dim3 grid((p.L + kFaBM - 1) / kFaBM, p.H, B);
  kern<<<grid, kFaThreads, smem, st>>>(tq, tk, tv, p);
  G4R_LAUNCH_CHECK("fa_fwd_tcgen05");
  return G4R_OK;
}

}  // namespace g4r

using namespace G4R_NS;

// Same contract as g4r_attention_bf16 (attention.cu), with the restriction that q/k/v are contiguous in
// the batch dimension (bs == L*ld: the packed [B*L, width] QKV buffer), which the TMA descriptors need.
static int attention_tc_impl(const void* q, const void* k, const void* v, void* out, long long ld,
                             long long bs, long long ldo, long long bso, int B, int H, int L,
                             int head_dim, int causal, float scale, const int* seqlens, float* lse, void* stream) {
  G4R_REQUIRE(q && k && v && out && B > 0 && H > 0 && L > 0, "attention_tc: bad arguments");
  G4R_REQUIRE(head_dim == 64 || head_dim == 128, "attention_tc: head_dim %d (64 or 128)", head_dim);
  G4R_REQUIRE(bs == (long long)L * ld, "attention_tc: q/k/v must be one packed [B*L, width] buffer (bs == L*ld)");
  G4R_REQUIRE(ld % 8 == 0 && ldo % 8 == 0 && bso % 8 == 0, "attention_tc: strides must keep 16-byte alignment");
  G4R_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0, "attention_tc: misaligned pointers");
  CUtensorMap tq, tk, tv;
  const long long cols = (long long)H * head_dim, rows = (long long)B * L;
  int rc;
  if ((rc = make_tmap_rows(&tq, q, cols, rows, ld, 128))) return rc;
  if ((rc = make_tmap_rows(&tk, k, cols, rows, ld, kFaBN))) return rc;
  if ((rc = make_tmap_rows(&tv, v, cols, rows, ld, kFaBN))) return rc;
  FaParams p{(__nv_bfloat16*)out, ldo, bso, L, H, scale, seqlens, lse};
  cudaStream_t st = (cudaStream_t)stream;
  if (head_dim == 64) return causal ? launch_fa<64, true>(tq, tk, tv, p, B, st) : launch_fa<64, false>(tq, tk, tv, p, B, st);
  return causal ? launch_fa<128, true>(tq, tk, tv, p, B, st) : launch_fa<128, false>(tq, tk, tv, p, B, st);
}

extern "C" int g4r_attention_tc_bf16(const void* q, const void* k, const void* v, void* out, long long ld,
                                     long long bs, long long ldo, long long bso, int B, int H, int L,
                                     int head_dim, int causal, float scale, const int* seqlens, void* stream) {
  return attention_tc_impl(q, k, v, out, ld, bs, ldo, bso, B, H, L, head_dim, causal, scale, seqlens, nullptr, stream);
}

// Training forward on the tcgen05 kernel: additionally writes lse[B, H, L] (fp32, natural log) for g4r_attention_bwd_bf16.
#if G4R_BF16_ONLY   // training-step only: no fp16 twin
extern "C" int g4r_attention_tc_lse_bf16(const void* q, const void* k, const void* v, void* out, long long ld,
                                         long long bs, long long ldo, long long bso, int B, int H, int L,
                                         int head_dim, int causal, float scale, float* lse, void* stream) {
  G4R_REQUIRE(lse, "attention_tc_lse: lse is NULL");
  return attention_tc_impl(q, k, v, out, ld, bs, ldo, bso, B, H, L, head_dim, causal, scale, nullptr, lse, stream);
}
#endif
