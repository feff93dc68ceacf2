// roi_align.cu -- RoIAlign forward/backward for sm_100a (HBM-bound gather / scatter-add).
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false: the bin / sample / weight
// arithmetic below is written with the reference's association and must not be
// contracted into FMAs, so that indices, weights and fp32 outputs are bit-identical
// to the reference CPU kernel (mmcv-1.4.7/mmcv/ops/csrc/pytorch/cpu/roi_align.cpp)
// -- checked by tests/test_roi_align_gpu.py against the CPU checker.
//
// Replaces (reference, relative to /root/reference/mmcv-1.4.7/mmcv/ops/csrc):
//   common/cuda/roi_align_cuda_kernel.cuh:17-108   roi_align_forward_cuda_kernel
//   common/cuda/roi_align_cuda_kernel.cuh:111-210  roi_align_backward_cuda_kernel
//   common/cuda/common_cuda_helper.hpp:28-119      bilinear_interpolate(_gradient)
//   pytorch/cuda/roi_align_cuda.cu:5-57            launchers
//
// Design (B200): the reference runs one thread per output scalar and recomputes the
// RoI geometry in every thread.  Here the geometry is separable: a sample's y depends
// on (ph,iy) only and its x on (pw,ix) only, so a CTA computes PH*gh + PW*gw axis
// entries {lo,hi,frac,1-frac,valid} once into shared memory and every thread reuses
// them.  Two data paths:
//   * NHWC, multi-level (the hot path): one launch covers all pyramid levels and all
//     RoIs; a thread owns 16 bytes of channels, issues the 4*g*g tap loads of a bin
//     as independent 128-bit loads (fully coalesced across the warp: consecutive lanes
//     read consecutive 16 B of the same pixel), accumulates in fp32 in the reference's
//     order and writes one 128-bit (or 64-bit, bf16 out) store per bin.
//   * NCHW (the mmcv._ext drop-in layout): CTA = (RoI, channel chunk); output writes
//     are contiguous; taps are plane gathers like the reference's but without the
//     per-thread geometry.
#include <stdlib.h>

#include "common.cuh"

namespace g4r {

constexpr int kTab = 256;      // axis-table capacity per axis (entries); else on-the-fly
constexpr int kThreads = 256;

template <typename A>
struct AxisEntry {
  A coord;  // raw sample coordinate (max-mode argmax)
  A l, h;   // frac, 1-frac
  int lo, hi;
  int valid;
};

// One axis of bilinear_interpolate: common_cuda_helper.hpp:33-55 == cpu/roi_align.cpp:44-86.
template <typename A>
__device__ __forceinline__ AxisEntry<A> axis_from_coord(A v, int size) {
  AxisEntry<A> e;
  e.coord = v;
  if (v < -1.0 || v > size) {
    e.valid = 0;
    e.lo = e.hi = 0;
    e.l = e.h = 0;
    return e;
  }
  e.valid = 1;
  if (v <= 0) v = 0;
  int lo = (int)v;
  int hi;
  if (lo >= size - 1) {
    hi = lo = size - 1;
    v = (A)lo;
  } else {
    hi = lo + 1;
  }
  e.lo = lo;
  e.hi = hi;
  e.l = v - lo;
  e.h = (A)1 - e.l;
  return e;
}

// y = roi_start_h + ph * bin_size_h + static_cast<T>(iy + .5f) * bin_size_h / static_cast<T>(grid)
// (roi_align_cuda_kernel.cuh:89-91; same expression in cpu/roi_align.cpp:33-35).
template <typename A>
__device__ __forceinline__ AxisEntry<A> axis_entry(A start, A bin, int p, int i, int grid, int size) {
  const A v = start + p * bin + static_cast<A>(i + .5f) * bin / static_cast<A>(grid);
  return axis_from_coord<A>(v, size);
}

template <typename A>
struct RoiGeom {
  int batch;
  A start_w, start_h, bin_w, bin_h;
  int gh, gw;
  A count;
};

// roi_align_cuda_kernel.cuh:31-60 (== cpu/roi_align.cpp:126-159).
template <typename A>
__device__ __forceinline__ RoiGeom<A> roi_geom(A r0, A r1, A r2, A r3, A r4, A scale, int PH, int PW,
                                               int sampling_ratio, bool aligned, bool clamp_count) {
  RoiGeom<A> g;
  g.batch = (int)r0;
  A offset = aligned ? (A)0.5 : (A)0.0;
  g.start_w = r1 * scale - offset;
  g.start_h = r2 * scale - offset;
  A end_w = r3 * scale - offset;
  A end_h = r4 * scale - offset;
  A roi_w = end_w - g.start_w;
  A roi_h = end_h - g.start_h;
  if (!aligned) {
    roi_w = roi_w > (A)1. ? roi_w : (A)1.;
    roi_h = roi_h > (A)1. ? roi_h : (A)1.;
  }
  g.bin_h = roi_h / static_cast<A>(PH);
  g.bin_w = roi_w / static_cast<A>(PW);
  g.gh = (sampling_ratio > 0) ? sampling_ratio : static_cast<int>(ceilf((float)(roi_h / PH)));
  g.gw = (sampling_ratio > 0) ? sampling_ratio : static_cast<int>(ceilf((float)(roi_w / PW)));
  if (g.gh < 0) g.gh = 0;
  if (g.gw < 0) g.gw = 0;
  int cnt = g.gh * g.gw;
  if (clamp_count && cnt < 1) cnt = 1;  // forward: max(gh*gw,1); backward divides by gh*gw
  g.count = (A)cnt;
  return g;
}

template <typename T> struct AccOf { using type = float; };
template <> struct AccOf<double> { using type = double; };

template <typename T, typename A> __device__ __forceinline__ A ld_as(const T* p) { return (A)to_f32<T>(*p); }
template <> __device__ __forceinline__ double ld_as<double, double>(const double* p) { return *p; }
template <typename T, typename A> __device__ __forceinline__ T st_as(A v) { return from_f32<T>((float)v); }
template <> __device__ __forceinline__ double st_as<double, double>(double v) { return v; }

// ------------------------------------------------------------------------------------
// NCHW forward (drop-in layout).  grid = (K, ceil(C/c_chunk)); block = kThreads.
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
roi_align_fwd_nchw(const T* __restrict__ input, const T* __restrict__ rois, T* __restrict__ output,
                   T* __restrict__ argmax_y, T* __restrict__ argmax_x, int C, int H, int W, int PH,
                   int PW, float spatial_scale, int sampling_ratio, int pool_mode, int aligned,
                   int c_chunk) {
  using A = typename AccOf<T>::type;
  __shared__ AxisEntry<A> ytab[kTab];
  __shared__ AxisEntry<A> xtab[kTab];

  const int k = blockIdx.x;
  const int c0 = blockIdx.y * c_chunk;
  const int c1 = min(C, c0 + c_chunk);
  const T* r = rois + (size_t)k * 5;
  const RoiGeom<A> g = roi_geom<A>(ld_as<T, A>(r), ld_as<T, A>(r + 1), ld_as<T, A>(r + 2),
                                   ld_as<T, A>(r + 3), ld_as<T, A>(r + 4), (A)spatial_scale, PH, PW,
                                   sampling_ratio, aligned != 0, true);
  const bool use_tab = (PH * g.gh <= kTab) && (PW * g.gw <= kTab);
  if (use_tab) {
    for (int i = threadIdx.x; i < PH * g.gh; i += blockDim.x)
      ytab[i] = axis_entry<A>(g.start_h, g.bin_h, i / g.gh, i % g.gh, g.gh, H);
    for (int i = threadIdx.x; i < PW * g.gw; i += blockDim.x)
      xtab[i] = axis_entry<A>(g.start_w, g.bin_w, i / g.gw, i % g.gw, g.gw, W);
    __syncthreads();
  }
  const int bins = PH * PW;
  const int items = (c1 - c0) * bins;
  const size_t hw = (size_t)H * W;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int c = c0 + it / bins;
    const int b = it % bins;
    const int ph = b / PW, pw = b % PW;
    const T* plane = input + ((size_t)g.batch * C + c) * hw;
    A out_val = 0;
    A maxval = -10000;  // cpu/roi_align.cpp:177 (the oracle); the CUDA reference uses -FLT_MAX
    A maxidx_y = -1.f, maxidx_x = -1.f;
    for (int iy = 0; iy < g.gh; iy++) {
      const AxisEntry<A> ey = use_tab ? ytab[ph * g.gh + iy]
                                      : axis_entry<A>(g.start_h, g.bin_h, ph, iy, g.gh, H);
      for (int ix = 0; ix < g.gw; ix++) {
        const AxisEntry<A> ex = use_tab ? xtab[pw * g.gw + ix]
                                        : axis_entry<A>(g.start_w, g.bin_w, pw, ix, g.gw, W);
        A val = 0;
        if (ey.valid && ex.valid) {
          const A w1 = ey.h * ex.h, w2 = ey.h * ex.l, w3 = ey.l * ex.h, w4 = ey.l * ex.l;
          const A v1 = ld_as<T, A>(plane + (size_t)ey.lo * W + ex.lo);
          const A v2 = ld_as<T, A>(plane + (size_t)ey.lo * W + ex.hi);
          const A v3 = ld_as<T, A>(plane + (size_t)ey.hi * W + ex.lo);
          const A v4 = ld_as<T, A>(plane + (size_t)ey.hi * W + ex.hi);
          val = w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4;
        }
        if (val > maxval) {
          maxval = val;
          maxidx_y = ey.coord;
          maxidx_x = ex.coord;
        }
        out_val += val;
      }
    }
    const size_t o = ((size_t)k * C + c) * bins + b;
    if (pool_mode == G4R_POOL_MAX) {
      output[o] = st_as<T, A>(maxval);
      argmax_y[o] = st_as<T, A>(maxidx_y);
      argmax_x[o] = st_as<T, A>(maxidx_x);
    } else {
      output[o] = st_as<T, A>(out_val / g.count);
    }
  }
}

// ---- atomics for every grad dtype -----------------------------------------------------
__device__ __forceinline__ void atomic_add_t(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void atomic_add_t(double* p, double v) { atomicAdd(p, v); }
__device__ __forceinline__ void atomic_add_t(__half* p, float v) { atomicAdd(p, __float2half_rn(v)); }
__device__ __forceinline__ void atomic_add_t(__nv_bfloat16* p, float v) { atomicAdd(p, __float2bfloat16_rn(v)); }

// ------------------------------------------------------------------------------------
// NCHW backward.  Same decomposition as forward; 4 atomics per sample like
// roi_align_cuda_kernel.cuh:191-205 (avg) / :141-150 (max).
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
roi_align_bwd_nchw(const T* __restrict__ grad_output, const T* __restrict__ rois,
                   const T* __restrict__ argmax_y, const T* __restrict__ argmax_x,
                   T* __restrict__ grad_input, int C, int H, int W, int PH, int PW,
                   float spatial_scale, int sampling_ratio, int pool_mode, int aligned, int c_chunk) {
  using A = typename AccOf<T>::type;
  __shared__ AxisEntry<A> ytab[kTab];
  __shared__ AxisEntry<A> xtab[kTab];
  const int k = blockIdx.x;
  const int c0 = blockIdx.y * c_chunk;
  const int c1 = min(C, c0 + c_chunk);
  const T* r = rois + (size_t)k * 5;
  const RoiGeom<A> g = roi_geom<A>(ld_as<T, A>(r), ld_as<T, A>(r + 1), ld_as<T, A>(r + 2),
                                   ld_as<T, A>(r + 3), ld_as<T, A>(r + 4), (A)spatial_scale, PH, PW,
                                   sampling_ratio, aligned != 0, false);
  const bool use_tab = (pool_mode == G4R_POOL_AVG) && (PH * g.gh <= kTab) && (PW * g.gw <= kTab);
  if (use_tab) {
    for (int i = threadIdx.x; i < PH * g.gh; i += blockDim.x)
      ytab[i] = axis_entry<A>(g.start_h, g.bin_h, i / g.gh, i % g.gh, g.gh, H);
    for (int i = threadIdx.x; i < PW * g.gw; i += blockDim.x)
      xtab[i] = axis_entry<A>(g.start_w, g.bin_w, i / g.gw, i % g.gw, g.gw, W);
    __syncthreads();
  }
  const int bins = PH * PW;
  const int items = (c1 - c0) * bins;
  const size_t hw = (size_t)H * W;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int c = c0 + it / bins;
    const int b = it % bins;
    const int ph = b / PW, pw = b % PW;
    const size_t o = ((size_t)k * C + c) * bins + b;
    const A go = ld_as<T, A>(grad_output + o);
    T* plane = grad_input + ((size_t)g.batch * C + c) * hw;
    if (pool_mode == G4R_POOL_MAX) {
      const A y = ld_as<T, A>(argmax_y + o), x = ld_as<T, A>(argmax_x + o);
      if (y != -1.f) {
        const AxisEntry<A> ey = axis_from_coord<A>(y, H), ex = axis_from_coord<A>(x, W);
        if (ey.valid && ex.valid) {
          atomic_add_t(plane + (size_t)ey.lo * W + ex.lo, go * (ey.h * ex.h));
          atomic_add_t(plane + (size_t)ey.lo * W + ex.hi, go * (ey.h * ex.l));
          atomic_add_t(plane + (size_t)ey.hi * W + ex.lo, go * (ey.l * ex.h));
          atomic_add_t(plane + (size_t)ey.hi * W + ex.hi, go * (ey.l * ex.l));
        }
      }
    } else {
      for (int iy = 0; iy < g.gh; iy++) {
        const AxisEntry<A> ey = use_tab ? ytab[ph * g.gh + iy]
                                        : axis_entry<A>(g.start_h, g.bin_h, ph, iy, g.gh, H);
        for (int ix = 0; ix < g.gw; ix++) {
          const AxisEntry<A> ex = use_tab ? xtab[pw * g.gw + ix]
                                          : axis_entry<A>(g.start_w, g.bin_w, pw, ix, g.gw, W);
          if (ey.valid && ex.valid) {
            atomic_add_t(plane + (size_t)ey.lo * W + ex.lo, go * (ey.h * ex.h) / g.count);
            atomic_add_t(plane + (size_t)ey.lo * W + ex.hi, go * (ey.h * ex.l) / g.count);
            atomic_add_t(plane + (size_t)ey.hi * W + ex.lo, go * (ey.l * ex.h) / g.count);
            atomic_add_t(plane + (size_t)ey.hi * W + ex.hi, go * (ey.l * ex.l) / g.count);
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// NHWC multi-level forward (hot path).
// grid = (K * ceil(PH/rows_per_cta), n_levels); block = kThreads.
// ------------------------------------------------------------------------------------
struct MlvlParams {
  const void* maps[G4R_MAX_LEVELS];
  const float* gn_scale[G4R_MAX_LEVELS];
  const float* gn_shift[G4R_MAX_LEVELS];
  float* grad_maps[G4R_MAX_LEVELS];
  int H[G4R_MAX_LEVELS], W[G4R_MAX_LEVELS];
  float scale[G4R_MAX_LEVELS];
  const float* rois;
  void* out;  // forward: output; backward: grad_output (const)
  int N, C, K, PH, PW, sampling_ratio, aligned, rows_per_cta, n_levels;
  int rows_per_cta_lvl[G4R_MAX_LEVELS];  // forward: bin rows handled by one CTA, per level
  float one;  // 1.0f, passed at run time: see add2_unfused
};

template <typename Tout, int N>
__device__ __forceinline__ void store_vec(Tout* p, const float (&v)[N]) {
  constexpr int kBytes = N * (int)sizeof(Tout);
  if constexpr (kBytes == 32) {
    uint4 a, b;
    Tout* ea = reinterpret_cast<Tout*>(&a);
    Tout* eb = reinterpret_cast<Tout*>(&b);
#pragma unroll
    for (int i = 0; i < N / 2; i++) { ea[i] = from_f32<Tout>(v[i]); eb[i] = from_f32<Tout>(v[N / 2 + i]); }
    reinterpret_cast<uint4*>(p)[0] = a;
    reinterpret_cast<uint4*>(p)[1] = b;
  } else if constexpr (kBytes == 16) {
    uint4 a;
    Tout* ea = reinterpret_cast<Tout*>(&a);
#pragma unroll
    for (int i = 0; i < N; i++) ea[i] = from_f32<Tout>(v[i]);
    *reinterpret_cast<uint4*>(p) = a;
  } else {
    static_assert(kBytes == 8, "unsupported vector store width");
    uint2 a;
    Tout* ea = reinterpret_cast<Tout*>(&a);
#pragma unroll
    for (int i = 0; i < N; i++) ea[i] = from_f32<Tout>(v[i]);
    *reinterpret_cast<uint2*>(p) = a;
  }
}

// ---- packed fp32x2 arithmetic (Blackwell FMUL2 / FFMA2: two IEEE fp32 lanes per instruction) ----------
// The forward is bound by the fma pipe, not by HBM: the reference association
//   val = ((w1*v1 + w2*v2) + w3*v3) + w4*v4;  acc += val          (roi_align.cpp:70-78 / cuda_kernel.cuh:63-66)
// is 8 dependent-rounding fp32 ops per channel-sample and must not be contracted into FMAs to stay
// bit-exact with the reference CPU kernel.  Two channels per instruction halves the pipe time.
// ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad=false (seen in SASS), so the
// unfused add is spelled fma(a, one, b) with `one` == 1.0f supplied at run time: a*1 is exact, the single
// rounding is that of a + b, and there is no multiply left to contract.
using f32x2 = unsigned long long;
__device__ __forceinline__ f32x2 pack2(float a, float b) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 add2_unfused(f32x2 a, f32x2 b, f32x2 one) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(one), "l"(b));
  return r;
}

// 16-byte read-only global load with an explicit state space (the hoisted row pointers pass through an
// optimisation barrier and would otherwise become generic LD instead of LDG).
template <typename T>
__device__ __forceinline__ void load16_global(const void* p, float (&out)[16 / sizeof(T)]) {
  uint4 raw;
  asm("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(raw.x), "=r"(raw.y), "=r"(raw.z), "=r"(raw.w) : "l"(p));
  const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
  for (int i = 0; i < 16 / (int)sizeof(T); i++) out[i] = to_f32<T>(e[i]);
}

// Packed axis entry for the hot path: element offsets pre-multiplied (y: lo*W*C, x: lo*C).
// An out-of-range sample gets offsets 0 and weights 0, exactly what the reference's pre_calc stores for it
// (cpu/roi_align.cpp:43-57: pos1..4 = 0, w1..4 = 0): its four products are (+-)0 and leave the accumulator unchanged,
// and the hot loop needs no branch (the loads of all samples of a bin can be in flight together).
struct PackedAxis {
  int off_lo, off_hi;
  float l, h;
};

__device__ __forceinline__ PackedAxis pack_axis(const AxisEntry<float>& e, int mul) {
  PackedAxis a;
  a.off_lo = e.valid ? e.lo * mul : 0;
  a.off_hi = e.valid ? e.hi * mul : 0;
  a.l = e.valid ? e.l : 0.f;
  a.h = e.valid ? e.h : 0.f;
  return a;
}

template <typename Tin, typename Tout, int G, bool AFFINE>
__global__ void __launch_bounds__(kThreads, (sizeof(Tin) == 4 && !AFFINE ? 5 : 3))
roi_align_fwd_nhwc_mlvl(const __grid_constant__ MlvlParams p) {
  constexpr int VEC = 16 / (int)sizeof(Tin);   // channels per thread: one 16-byte vector
  __shared__ PackedAxis ytab[kTab];
  __shared__ PackedAxis xtab[kTab];

  const int lvl = blockIdx.y;
  const int rpc = p.rows_per_cta_lvl[lvl];
  const int row_groups = (p.PH + rpc - 1) / rpc;
  const int k = blockIdx.x / row_groups;
  if (k >= p.K) return;  // grid.x is sized for the level with the most row groups
  const int ph0 = (blockIdx.x % row_groups) * rpc;
  const int nrows = min(rpc, p.PH - ph0);
  const int H = p.H[lvl], W = p.W[lvl], C = p.C, PW = p.PW;
  const float* r = p.rois + (size_t)k * 5;
  const RoiGeom<float> g = roi_geom<float>(r[0], r[1], r[2], r[3], r[4], p.scale[lvl], p.PH, PW,
                                           G > 0 ? G : p.sampling_ratio, p.aligned != 0, true);
  const int gh = G > 0 ? G : g.gh, gw = G > 0 ? G : g.gw;
  // tables always fit for G > 0 (launcher guarantees PH*G, PW*G <= kTab); adaptive grids that do
  // not fit are processed in chunks of kTab samples per axis.
  const int lanes = C / VEC;
  const Tin* map = reinterpret_cast<const Tin*>(p.maps[lvl]) + (size_t)g.batch * H * W * C;
  Tout* out = reinterpret_cast<Tout*>(p.out) +
              (((size_t)lvl * p.K + k) * p.PH + ph0) * (size_t)PW * C;
  const bool quarter = (gh * gw == 4);  // x/4 == x*0.25f exactly: avoids an IEEE division per value
  const f32x2 one2 = pack2(p.one, p.one);

  if (nrows * gh <= kTab && PW * gw <= kTab) {
    for (int i = threadIdx.x; i < nrows * gh; i += blockDim.x)
      ytab[i] = pack_axis(axis_entry<float>(g.start_h, g.bin_h, ph0 + i / gh, i % gh, gh, H), W * C);
    for (int i = threadIdx.x; i < PW * gw; i += blockDim.x)
      xtab[i] = pack_axis(axis_entry<float>(g.start_w, g.bin_w, i / gw, i % gw, gw, W), C * (int)sizeof(Tin) / 16);  // 16-byte units
    __syncthreads();
    // Per-bin body: `prow`, `pw`, `lane` select the bin and the channel slice.
    auto do_bin = [&](int prow, int pw, int lane, const PackedAxis* eyp, const char* const* rows) {
      const int coff = lane * VEC;
      const char* mpb = reinterpret_cast<const char*>(map + coff);
      float ga[VEC], gb[VEC];
      if constexpr (AFFINE) {
        const float* sa = p.gn_scale[lvl] + (size_t)g.batch * C + coff;
        const float* sb = p.gn_shift[lvl] + (size_t)g.batch * C + coff;
#pragma unroll
        for (int i = 0; i < VEC; i++) { ga[i] = sa[i]; gb[i] = sb[i]; }
      }
      f32x2 acc2[VEC / 2];
#pragma unroll
      for (int i = 0; i < VEC / 2; i++) acc2[i] = 0ull;   // (+0.f, +0.f)
#pragma unroll
      for (int iy = 0; iy < (G > 0 ? G : gh); iy++) {
        const PackedAxis ey = eyp ? eyp[iy] : ytab[prow * gh + iy];
        // row base pointers (hoisted by the caller when `rows` is given); each tap is then one
        // IMAD.WIDE.U32: row + x_offset * 16 (x entries are stored in 16-byte units)
        const char* r_lo = rows ? rows[2 * iy] : mpb + (size_t)(unsigned)ey.off_lo * sizeof(Tin);
        const char* r_hi = rows ? rows[2 * iy + 1] : mpb + (size_t)(unsigned)ey.off_hi * sizeof(Tin);
#pragma unroll
        for (int ix = 0; ix < (G > 0 ? G : gw); ix++) {
          const PackedAxis ex = xtab[pw * gw + ix];
          {
            const float w1 = ey.h * ex.h, w2 = ey.h * ex.l, w3 = ey.l * ex.h, w4 = ey.l * ex.l;
            float v1[VEC], v2[VEC], v3[VEC], v4[VEC];
            load16_global<Tin>(r_lo + (size_t)(unsigned)ex.off_lo * 16, v1);
            load16_global<Tin>(r_lo + (size_t)(unsigned)ex.off_hi * 16, v2);
            load16_global<Tin>(r_hi + (size_t)(unsigned)ex.off_lo * 16, v3);
            load16_global<Tin>(r_hi + (size_t)(unsigned)ex.off_hi * 16, v4);
            if constexpr (AFFINE) {
              // fused GroupNorm affine + ReLU on every tap (this engine's own fusion, tolerance-tested):
              // one FFMA2 per channel pair and tap
#pragma unroll
              for (int i = 0; i < VEC; i += 2) {
                const f32x2 GA = pack2(ga[i], ga[i + 1]), GB = pack2(gb[i], gb[i + 1]);
                float a, b;
                unpack2(fma2(pack2(v1[i], v1[i + 1]), GA, GB), a, b); v1[i] = fmaxf(a, 0.f); v1[i + 1] = fmaxf(b, 0.f);
                unpack2(fma2(pack2(v2[i], v2[i + 1]), GA, GB), a, b); v2[i] = fmaxf(a, 0.f); v2[i + 1] = fmaxf(b, 0.f);
                unpack2(fma2(pack2(v3[i], v3[i + 1]), GA, GB), a, b); v3[i] = fmaxf(a, 0.f); v3[i + 1] = fmaxf(b, 0.f);
                unpack2(fma2(pack2(v4[i], v4[i + 1]), GA, GB), a, b); v4[i] = fmaxf(a, 0.f); v4[i + 1] = fmaxf(b, 0.f);
              }
            }
            const f32x2 W1 = pack2(w1, w1), W2 = pack2(w2, w2), W3 = pack2(w3, w3), W4 = pack2(w4, w4);
#pragma unroll
            for (int i = 0; i < VEC; i += 2) {
              f32x2 t = mul2(W1, pack2(v1[i], v1[i + 1]));
              t = add2_unfused(t, mul2(W2, pack2(v2[i], v2[i + 1])), one2);
              t = add2_unfused(t, mul2(W3, pack2(v3[i], v3[i + 1])), one2);
              t = add2_unfused(t, mul2(W4, pack2(v4[i], v4[i + 1])), one2);
              acc2[i / 2] = add2_unfused(acc2[i / 2], t, one2);
            }
          }
        }
      }
      float acc[VEC];
#pragma unroll
      for (int i = 0; i < VEC; i += 2) unpack2(acc2[i / 2], acc[i], acc[i + 1]);
#pragma unroll
      for (int i = 0; i < VEC; i++) acc[i] = quarter ? acc[i] * 0.25f : acc[i] / g.count;
      store_vec<Tout, VEC>(out + ((size_t)prow * PW + pw) * C + coff, acc);
    };
    if constexpr (G > 0) {
      if (blockDim.x % lanes == 0 || lanes % blockDim.x == 0) {
        // fixed channel slice per thread, y-axis entries hoisted out of the pw loop
        const int ngrp = blockDim.x >= lanes ? blockDim.x / lanes : 1;
        const int grp = blockDim.x >= lanes ? threadIdx.x / lanes : 0;
        for (int lane = threadIdx.x % lanes; lane < lanes; lane += (blockDim.x >= lanes ? lanes : blockDim.x)) {
          for (int prow = 0; prow < nrows; prow++) {
            PackedAxis eyr[G];
            const char* rows[2 * G];
            const char* mpb = reinterpret_cast<const char*>(map + lane * VEC);
#pragma unroll
            for (int iy = 0; iy < G; iy++) {
              eyr[iy] = ytab[prow * G + iy];
              rows[2 * iy] = mpb + (size_t)(unsigned)eyr[iy].off_lo * sizeof(Tin);
              rows[2 * iy + 1] = mpb + (size_t)(unsigned)eyr[iy].off_hi * sizeof(Tin);
              // opaque to the optimiser: keeps the 64-bit row pointers in registers instead of
              // re-deriving them (3 integer instructions) at every tap
              asm volatile("" : "+l"(rows[2 * iy]), "+l"(rows[2 * iy + 1]));
            }
            for (int pw = grp; pw < PW; pw += ngrp) do_bin(prow, pw, lane, eyr, rows);
          }
        }
        return;
      }
    }
    const int items = nrows * PW * lanes;
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
      const int lane = it % lanes;
      const int b = it / lanes;  // bin within this CTA's rows
      do_bin(b / PW, b % PW, lane, nullptr, nullptr);
    }
    return;
  }

  // generic path (adaptive sampling grids too large for the tables): geometry on the fly
  const int lanes1 = C / VEC;
  const int items = nrows * PW * lanes1;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int lane = it % lanes1;
    const int b = it / lanes1;
    const int prow = b / PW, pw = b % PW;
    const int coff = lane * VEC;
    float acc[VEC];
#pragma unroll
    for (int i = 0; i < VEC; i++) acc[i] = 0.f;
    for (int iy = 0; iy < gh; iy++) {
      const AxisEntry<float> ey = axis_entry<float>(g.start_h, g.bin_h, ph0 + prow, iy, gh, H);
      for (int ix = 0; ix < gw; ix++) {
        const AxisEntry<float> ex = axis_entry<float>(g.start_w, g.bin_w, pw, ix, gw, W);
        if (!(ey.valid && ex.valid)) continue;
        const float w1 = ey.h * ex.h, w2 = ey.h * ex.l, w3 = ey.l * ex.h, w4 = ey.l * ex.l;
        float v1[VEC], v2[VEC], v3[VEC], v4[VEC];
        load16<Tin>(map + ((size_t)ey.lo * W + ex.lo) * C + coff, v1);
        load16<Tin>(map + ((size_t)ey.lo * W + ex.hi) * C + coff, v2);
        load16<Tin>(map + ((size_t)ey.hi * W + ex.lo) * C + coff, v3);
        load16<Tin>(map + ((size_t)ey.hi * W + ex.hi) * C + coff, v4);
#pragma unroll
        for (int i = 0; i < VEC; i++) {
          if constexpr (AFFINE) {
            const float a = p.gn_scale[lvl][(size_t)g.batch * C + coff + i];
            const float bb = p.gn_shift[lvl][(size_t)g.batch * C + coff + i];
            v1[i] = fmaxf(v1[i] * a + bb, 0.f);
            v2[i] = fmaxf(v2[i] * a + bb, 0.f);
            v3[i] = fmaxf(v3[i] * a + bb, 0.f);
            v4[i] = fmaxf(v4[i] * a + bb, 0.f);
          }
          const float val = w1 * v1[i] + w2 * v2[i] + w3 * v3[i] + w4 * v4[i];
          acc[i] += val;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < VEC; i++) acc[i] = acc[i] / g.count;
    store_vec<Tout, VEC>(out + ((size_t)prow * PW + pw) * C + coff, acc);
  }
}

// ------------------------------------------------------------------------------------
// Tap-deduplicating forward for the fixed 2x2 sampling grid (RoIAlign(14, sampling_ratio=2) of the SPI module,
// gpt4roi/models/layers.py:205-212, and the 7x7 BASELINE microbench).
//
// The table kernel above is bound by the L1 data pipe (ncu: l1tex__data_pipe_lsu_wavefronts 76 %, DRAM 34 %):
// every bin issues 16 16-byte tap loads per 16-byte store.  On the coarse levels the two samples of a bin axis are
// less than a pixel apart, so their (lo, hi) tap pairs overlap: per axis the four taps (lo0, hi0, lo1, hi1) are
//     P2: lo1 == lo0              -> 2 distinct columns      (taps map to slots 0,1,0,1)
//     P3: lo1 == hi0 == lo0 + 1   -> 3 distinct columns      (slots 0,1,1,2)
//     P4: anything else (>= 2 px apart, clamped at the border, out of range) -> 4 loads (slots 0,1,2,3)
// The pattern of a bin row / bin column is the same for every channel and every lane of the CTA, so it is classified
// once per (RoI, level) into shared memory and each bin branches -- uniformly -- into one of 3 x 3 straight-line
// variants that issue NSY x NSX unconditional loads (4 ... 16) and then the UNCHANGED arithmetic: every sample still
// computes w1*v1 + w2*v2 + w3*v3 + w4*v4 in the reference's association (roi_align_cuda_kernel.cuh:63-66) with the
// same weights, the duplicated taps simply read the same register.  Bit-identical to the table kernel.
// ------------------------------------------------------------------------------------
// slot of tap t in (lo0, hi0, lo1, hi1) for NS distinct rows / columns
template <int NS>
__host__ __device__ constexpr int tap_slot(int t) {
  return NS == 2 ? (t & 1) : (NS == 3 ? (t == 0 ? 0 : (t == 3 ? 2 : 1)) : t);
}

__device__ __forceinline__ int tap_pattern(const AxisEntry<float>& a, const AxisEntry<float>& b) {
  if (!a.valid || !b.valid) return 4;
  if (a.hi != a.lo + 1 || b.hi != b.lo + 1) return 4;   // clamped at the far border
  if (b.lo == a.lo) return 2;
  if (b.lo == a.hi) return 3;
  return 4;
}

template <typename Tin, typename Tout, bool AFFINE, int NSY, int NSX>
__device__ __forceinline__ void dedup_bin(const char* __restrict__ mpb, const PackedAxis& ey0, const PackedAxis& ey1,
                                          const PackedAxis& ex0, const PackedAxis& ex1, const float* __restrict__ sa,
                                          const float* __restrict__ sb, f32x2 one2, Tout* __restrict__ outp) {
  constexpr int VEC = 16 / (int)sizeof(Tin);
  // distinct row / column offsets of this bin
  unsigned yo[NSY], xo[NSX];
  yo[0] = (unsigned)ey0.off_lo; yo[1] = (unsigned)ey0.off_hi;
  if constexpr (NSY == 3) yo[2] = (unsigned)ey1.off_hi;
  if constexpr (NSY == 4) { yo[2] = (unsigned)ey1.off_lo; yo[3] = (unsigned)ey1.off_hi; }
  xo[0] = (unsigned)ex0.off_lo; xo[1] = (unsigned)ex0.off_hi;
  if constexpr (NSX == 3) xo[2] = (unsigned)ex1.off_hi;
  if constexpr (NSX == 4) { xo[2] = (unsigned)ex1.off_lo; xo[3] = (unsigned)ex1.off_hi; }
  uint4 R[NSY][NSX];   // raw 16-byte taps; widened (and, AFFINE, normalised + ReLU'd) where they are used
#pragma unroll
  for (int sy = 0; sy < NSY; sy++) {
    const char* row = mpb + (size_t)yo[sy] * sizeof(Tin);
#pragma unroll
    for (int sx = 0; sx < NSX; sx++) {
      const void* q = row + (size_t)xo[sx] * 16;
      asm("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(R[sy][sx].x), "=r"(R[sy][sx].y), "=r"(R[sy][sx].z), "=r"(R[sy][sx].w) : "l"(q));
    }
  }
  float ga[VEC], gb[VEC];
  if constexpr (AFFINE) {
#pragma unroll
    for (int i = 0; i < VEC; i++) { ga[i] = sa[i]; gb[i] = sb[i]; }
  }
  auto tap = [&](const uint4& raw, float (&v)[VEC]) {
    const Tin* e = reinterpret_cast<const Tin*>(&raw);
#pragma unroll
    for (int i = 0; i < VEC; i++) v[i] = to_f32<Tin>(e[i]);
    if constexpr (AFFINE) {   // fused GroupNorm affine + ReLU (same op on the same value as the table kernel)
#pragma unroll
      for (int i = 0; i < VEC; i += 2) {
        float a, b;
        unpack2(fma2(pack2(v[i], v[i + 1]), pack2(ga[i], ga[i + 1]), pack2(gb[i], gb[i + 1])), a, b);
        v[i] = fmaxf(a, 0.f);
        v[i + 1] = fmaxf(b, 0.f);
      }
    }
  };
  f32x2 acc2[VEC / 2];
#pragma unroll
  for (int i = 0; i < VEC / 2; i++) acc2[i] = 0ull;
#pragma unroll
  for (int iy = 0; iy < 2; iy++) {
    const PackedAxis& ey = iy ? ey1 : ey0;
#pragma unroll
    for (int ix = 0; ix < 2; ix++) {
      const PackedAxis& ex = ix ? ex1 : ex0;
      const float w1 = ey.h * ex.h, w2 = ey.h * ex.l, w3 = ey.l * ex.h, w4 = ey.l * ex.l;
      const f32x2 W1 = pack2(w1, w1), W2 = pack2(w2, w2), W3 = pack2(w3, w3), W4 = pack2(w4, w4);
      float v1[VEC], v2[VEC], v3[VEC], v4[VEC];
      tap(R[tap_slot<NSY>(2 * iy)][tap_slot<NSX>(2 * ix)], v1);
      tap(R[tap_slot<NSY>(2 * iy)][tap_slot<NSX>(2 * ix + 1)], v2);
      tap(R[tap_slot<NSY>(2 * iy + 1)][tap_slot<NSX>(2 * ix)], v3);
      tap(R[tap_slot<NSY>(2 * iy + 1)][tap_slot<NSX>(2 * ix + 1)], v4);
#pragma unroll
      for (int i = 0; i < VEC; i += 2) {
        f32x2 t = mul2(W1, pack2(v1[i], v1[i + 1]));
        t = add2_unfused(t, mul2(W2, pack2(v2[i], v2[i + 1])), one2);
        t = add2_unfused(t, mul2(W3, pack2(v3[i], v3[i + 1])), one2);
        t = add2_unfused(t, mul2(W4, pack2(v4[i], v4[i + 1])), one2);
        acc2[i / 2] = add2_unfused(acc2[i / 2], t, one2);
      }
    }
  }
  float o[VEC];
#pragma unroll
  for (int i = 0; i < VEC; i += 2) unpack2(acc2[i / 2], o[i], o[i + 1]);
#pragma unroll
  for (int i = 0; i < VEC; i++) o[i] = o[i] * 0.25f;   // / 4 exactly (count = 2 x 2)
  store_vec<Tout, VEC>(outp, o);
}

template <typename Tin, typename Tout, bool AFFINE>
__global__ void __launch_bounds__(kThreads, (sizeof(Tin) == 4 ? (AFFINE ? 3 : 4) : 2))
roi_align_fwd_nhwc_mlvl_dedup(const __grid_constant__ MlvlParams p) {
  constexpr int VEC = 16 / (int)sizeof(Tin);
  constexpr int G = 2;
  __shared__ PackedAxis ytab[kTab];
  __shared__ PackedAxis xtab[kTab];
  __shared__ unsigned char ypat[kTab / 2];
  __shared__ unsigned char xpat[kTab / 2];

  const int lvl = blockIdx.y;
  const int rpc = p.rows_per_cta_lvl[lvl];
  const int row_groups = (p.PH + rpc - 1) / rpc;
  const int k = blockIdx.x / row_groups;
  if (k >= p.K) return;
  const int ph0 = (blockIdx.x % row_groups) * rpc;
  const int nrows = min(rpc, p.PH - ph0);
  const int H = p.H[lvl], W = p.W[lvl], C = p.C, PW = p.PW;
  const float* r = p.rois + (size_t)k * 5;
  const RoiGeom<float> g = roi_geom<float>(r[0], r[1], r[2], r[3], r[4], p.scale[lvl], p.PH, PW, G, p.aligned != 0, true);
  const int lanes = C / VEC;
  const Tin* map = reinterpret_cast<const Tin*>(p.maps[lvl]) + (size_t)g.batch * H * W * C;
  Tout* out = reinterpret_cast<Tout*>(p.out) + (((size_t)lvl * p.K + k) * p.PH + ph0) * (size_t)PW * C;
  const f32x2 one2 = pack2(p.one, p.one);

  for (int i = threadIdx.x; i < nrows; i += blockDim.x) {
    const AxisEntry<float> a = axis_entry<float>(g.start_h, g.bin_h, ph0 + i, 0, G, H);
    const AxisEntry<float> b = axis_entry<float>(g.start_h, g.bin_h, ph0 + i, 1, G, H);
    ytab[2 * i] = pack_axis(a, W * C);
    ytab[2 * i + 1] = pack_axis(b, W * C);
    ypat[i] = (unsigned char)tap_pattern(a, b);
  }
  for (int i = threadIdx.x; i < PW; i += blockDim.x) {
    const AxisEntry<float> a = axis_entry<float>(g.start_w, g.bin_w, i, 0, G, W);
    const AxisEntry<float> b = axis_entry<float>(g.start_w, g.bin_w, i, 1, G, W);
    xtab[2 * i] = pack_axis(a, C * (int)sizeof(Tin) / 16);   // 16-byte units
    xtab[2 * i + 1] = pack_axis(b, C * (int)sizeof(Tin) / 16);
    xpat[i] = (unsigned char)tap_pattern(a, b);
  }
  __syncthreads();

  const int ngrp = blockDim.x >= lanes ? blockDim.x / lanes : 1;
  const int grp = blockDim.x >= lanes ? threadIdx.x / lanes : 0;
  for (int lane = threadIdx.x % lanes; lane < lanes; lane += (blockDim.x >= lanes ? lanes : blockDim.x)) {
    const int coff = lane * VEC;
    const char* mpb = reinterpret_cast<const char*>(map + coff);
    const float* sa = nullptr;
    const float* sb = nullptr;
    if constexpr (AFFINE) {
      sa = p.gn_scale[lvl] + (size_t)g.batch * C + coff;
      sb = p.gn_shift[lvl] + (size_t)g.batch * C + coff;
    }
    for (int prow = 0; prow < nrows; prow++) {
      const PackedAxis ey0 = ytab[2 * prow], ey1 = ytab[2 * prow + 1];
      const int py = ypat[prow];
      for (int pw = grp; pw < PW; pw += ngrp) {
        const PackedAxis ex0 = xtab[2 * pw], ex1 = xtab[2 * pw + 1];
        Tout* outp = out + ((size_t)prow * PW + pw) * C + coff;
        const int px = xpat[pw];
#define G4R_DEDUP_CASE(NY, NX) dedup_bin<Tin, Tout, AFFINE, NY, NX>(mpb, ey0, ey1, ex0, ex1, sa, sb, one2, outp)
        if (py == 2) {
          if (px == 2) G4R_DEDUP_CASE(2, 2); else if (px == 3) G4R_DEDUP_CASE(2, 3); else G4R_DEDUP_CASE(2, 4);
        } else if (py == 3) {
          if (px == 2) G4R_DEDUP_CASE(3, 2); else if (px == 3) G4R_DEDUP_CASE(3, 3); else G4R_DEDUP_CASE(3, 4);
        } else {
          if (px == 2) G4R_DEDUP_CASE(4, 2); else if (px == 3) G4R_DEDUP_CASE(4, 3); else G4R_DEDUP_CASE(4, 4);
        }
#undef G4R_DEDUP_CASE
      }
    }
  }
}

// NHWC multi-level backward: grad_output [Lv,K,PH,PW,C] (Tg) -> fp32 NHWC grad maps (atomics).
template <typename Tg>
__global__ void __launch_bounds__(kThreads)
roi_align_bwd_nhwc_mlvl(const __grid_constant__ MlvlParams p) {
  constexpr int VEC = 4;  // float4 vector atomics (red.global.add.v4.f32, sm_90+)
  __shared__ AxisEntry<float> ytab[kTab];
  __shared__ AxisEntry<float> xtab[kTab];
  const int lvl = blockIdx.y;
  const int row_groups = (p.PH + p.rows_per_cta - 1) / p.rows_per_cta;
  const int k = blockIdx.x / row_groups;
  const int ph0 = (blockIdx.x % row_groups) * p.rows_per_cta;
  const int nrows = min(p.rows_per_cta, p.PH - ph0);
  const int H = p.H[lvl], W = p.W[lvl], C = p.C, PW = p.PW;
  const float* r = p.rois + (size_t)k * 5;
  const RoiGeom<float> g = roi_geom<float>(r[0], r[1], r[2], r[3], r[4], p.scale[lvl], p.PH, PW,
                                           p.sampling_ratio, p.aligned != 0, false);
  const int gh = g.gh, gw = g.gw;
  const bool use_tab = (nrows * gh <= kTab) && (PW * gw <= kTab);
  if (use_tab) {
    for (int i = threadIdx.x; i < nrows * gh; i += blockDim.x)
      ytab[i] = axis_entry<float>(g.start_h, g.bin_h, ph0 + i / gh, i % gh, gh, H);
    for (int i = threadIdx.x; i < PW * gw; i += blockDim.x)
      xtab[i] = axis_entry<float>(g.start_w, g.bin_w, i / gw, i % gw, gw, W);
    __syncthreads();
  }
  const int lanes = C / VEC;
  const int items = nrows * PW * lanes;
  float* gmap = p.grad_maps[lvl] + (size_t)g.batch * H * W * C;
  const Tg* go = reinterpret_cast<const Tg*>(p.out) +
                 (((size_t)lvl * p.K + k) * p.PH + ph0) * (size_t)PW * C;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int lane = it % lanes;
    const int b = it / lanes;
    const int prow = b / PW, pw = b % PW;
    const int coff = lane * VEC;
    float gv[VEC];
    const Tg* gp = go + ((size_t)prow * PW + pw) * C + coff;
#pragma unroll
    for (int i = 0; i < VEC; i++) gv[i] = to_f32<Tg>(gp[i]);
    for (int iy = 0; iy < gh; iy++) {
      const AxisEntry<float> ey = use_tab ? ytab[prow * gh + iy]
                                          : axis_entry<float>(g.start_h, g.bin_h, ph0 + prow, iy, gh, H);
      for (int ix = 0; ix < gw; ix++) {
        const AxisEntry<float> ex = use_tab ? xtab[pw * gw + ix]
                                            : axis_entry<float>(g.start_w, g.bin_w, pw, ix, gw, W);
        if (!(ey.valid && ex.valid)) continue;
        const float w[4] = {ey.h * ex.h, ey.h * ex.l, ey.l * ex.h, ey.l * ex.l};
        const size_t off[4] = {((size_t)ey.lo * W + ex.lo) * C, ((size_t)ey.lo * W + ex.hi) * C,
                               ((size_t)ey.hi * W + ex.lo) * C, ((size_t)ey.hi * W + ex.hi) * C};
#pragma unroll
        for (int t = 0; t < 4; t++) {
          float4 a;
          a.x = gv[0] * w[t] / g.count;
          a.y = gv[1] * w[t] / g.count;
          a.z = gv[2] * w[t] / g.count;
          a.w = gv[3] * w[t] / g.count;
          atomicAdd(reinterpret_cast<float4*>(gmap + off[t] + coff), a);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------
static int pick_c_chunk(int C, int bins) {
  int c = 4096 / (bins > 0 ? bins : 1);
  if (c < 1) c = 1;
  if (c > C) c = C;
  return c;
}

template <typename T>
static int launch_fwd_nchw(const void* input, const void* rois, void* output, void* ay, void* ax,
                           int C, int H, int W, int K, int PH, int PW, float scale, int sr,
                           int pool_mode, int aligned, cudaStream_t st) {
  const int c_chunk = pick_c_chunk(C, PH * PW);
  dim3 grid(K, (C + c_chunk - 1) / c_chunk);
  roi_align_fwd_nchw<T><<<grid, kThreads, 0, st>>>((const T*)input, (const T*)rois, (T*)output, (T*)ay,
                                                   (T*)ax, C, H, W, PH, PW, scale, sr, pool_mode,
                                                   aligned, c_chunk);
  G4R_LAUNCH_CHECK("roi_align_fwd_nchw");
  return G4R_OK;
}

template <typename T>
static int launch_bwd_nchw(const void* go, const void* rois, const void* ay, const void* ax, void* gi,
                           int C, int H, int W, int K, int PH, int PW, float scale, int sr,
                           int pool_mode, int aligned, cudaStream_t st) {
  const int c_chunk = pick_c_chunk(C, PH * PW);
  dim3 grid(K, (C + c_chunk - 1) / c_chunk);
  roi_align_bwd_nchw<T><<<grid, kThreads, 0, st>>>((const T*)go, (const T*)rois, (const T*)ay,
                                                   (const T*)ax, (T*)gi, C, H, W, PH, PW, scale, sr,
                                                   pool_mode, aligned, c_chunk);
  G4R_LAUNCH_CHECK("roi_align_bwd_nchw");
  return G4R_OK;
}

static int pick_rows_per_cta(int K, int n_levels, int PH) {
  // Whole-RoI CTAs maximise L1 reuse between neighbouring bin rows; split rows only when
  // there are too few (RoI, level) pairs to give every SM a few CTAs.
  const long want = 4L * num_sms();
  int rows = PH;
  while (rows > 1 && (long)K * n_levels * ((PH + rows - 1) / rows) < want) rows = (rows + 1) / 2;
  return rows;
}

template <typename Tin, typename Tout>
static int launch_fwd_mlvl(MlvlParams& p, bool affine, cudaStream_t st) {
  // Rows per CTA, per level.  Whole-RoI CTAs amortise the table build; but on the big (fine)
  // levels a whole image-level does not fit L2 with many RoIs in flight, so those levels use one
  // bin row per CTA: ~PH x more CTAs per image => fewer images in flight => taps hit L2.
  constexpr int VEC = 16 / (int)sizeof(Tin);
  const int lanes = p.C / VEC;   // threads per bin: one 16-byte channel vector each
  int max_groups = 1;
  for (int l = 0; l < p.n_levels; l++) {
    const double map_mb = (double)p.H[l] * p.W[l] * p.C * sizeof(Tin) / 1e6;
    int rows = map_mb > 8.0 ? 1 : pick_rows_per_cta(p.K, p.n_levels, p.PH);
    // At least kThreads / lanes bin rows per CTA.  This clamp was written for a row-walk kernel that gave each group
    // of `lanes` threads its own bin row; the tap-dedup kernel was measured (DESIGN.md section 3) on the grid it shapes.
    if (lanes < kThreads && rows < kThreads / lanes) rows = kThreads / lanes;
    if (rows > p.PH) rows = p.PH;
    p.rows_per_cta_lvl[l] = rows;
    const int groups = (p.PH + rows - 1) / rows;
    if (groups > max_groups) max_groups = groups;
  }
  dim3 grid((unsigned)(p.K * max_groups), p.n_levels);
  const bool g2 = p.sampling_ratio == 2 && p.PH * 2 <= kTab && p.PW * 2 <= kTab;
  // 2x2 sampling grid: the tap-dedup kernel (12.1 ms vs 15.3 ms for the table kernel on the BASELINE microbench).
  // It maps threads to a fixed channel slice, so `lanes` must divide kThreads or be a multiple of it.
  if (g2 && (kThreads % lanes == 0 || lanes % kThreads == 0)) {
    if (affine) roi_align_fwd_nhwc_mlvl_dedup<Tin, Tout, true><<<grid, kThreads, 0, st>>>(p);
    else roi_align_fwd_nhwc_mlvl_dedup<Tin, Tout, false><<<grid, kThreads, 0, st>>>(p);
    G4R_LAUNCH_CHECK("roi_align_fwd_nhwc_mlvl_dedup");
    return G4R_OK;
  }
  if (g2) {
    if (affine) roi_align_fwd_nhwc_mlvl<Tin, Tout, 2, true><<<grid, kThreads, 0, st>>>(p);
    else roi_align_fwd_nhwc_mlvl<Tin, Tout, 2, false><<<grid, kThreads, 0, st>>>(p);
  } else {
    if (affine) roi_align_fwd_nhwc_mlvl<Tin, Tout, 0, true><<<grid, kThreads, 0, st>>>(p);
    else roi_align_fwd_nhwc_mlvl<Tin, Tout, 0, false><<<grid, kThreads, 0, st>>>(p);
  }
  G4R_LAUNCH_CHECK("roi_align_fwd_nhwc_mlvl");
  return G4R_OK;
}

// ------------------------------------------------------------------------------------
// NCHW drop-in, large-work fast path: [N,C,H,W] -> NHWC transpose (tiled through shared memory), the NHWC
// multi-level kernel above on one level (coalesced 16-byte channel vectors, tap dedup), and the [K,PH,PW,C] ->
// [K,C,PH,PW] transpose back.  Three streaming passes instead of the plane gather of the reference layout
// (roi_align_cuda_kernel.cuh:17-108: one thread per output scalar, 16 scattered 4-byte loads each): the same
// arithmetic in the same order, so the results stay bit-identical to the direct NCHW kernel.
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
transpose_batched(const T* __restrict__ in, T* __restrict__ out, int R, int S) {
  // per batch b = blockIdx.z: in [R][S] -> out [S][R].  Tile = 32 rows x 32 16-byte vectors: global reads are
  // 16-byte vectors along S (4 in flight per thread), global writes 4-byte-per-lane runs along R (coalesced);
  // the row pitch of the shared tile keeps the vector stores conflict-free and the transposed reads 4-way.
  constexpr int VEC = 16 / (int)sizeof(T);
  constexpr int TS = 32 * VEC;
  __shared__ __align__(16) T tile[32][TS + VEC];
  const size_t base = (size_t)blockIdx.z * R * S;
  const int s0 = blockIdx.x * TS, r0 = blockIdx.y * 32;
  const bool vec_ok = (S % VEC == 0) && ((reinterpret_cast<uintptr_t>(in + base) & 15) == 0);
#pragma unroll
  for (int it = 0; it < 4; it++) {
    const int idx = threadIdx.x + it * 256;
    const int row = idx >> 5, vc = idx & 31;
    const int r = r0 + row, sidx = s0 + vc * VEC;
    if (r < R && sidx < S) {
      if (vec_ok) {
        *reinterpret_cast<uint4*>(&tile[row][vc * VEC]) = *reinterpret_cast<const uint4*>(in + base + (size_t)r * S + sidx);
      } else {
#pragma unroll
        for (int i = 0; i < VEC; i++)
          if (sidx + i < S) tile[row][vc * VEC + i] = in[base + (size_t)r * S + sidx + i];
      }
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = r0 + lane;
  for (int sl = warp; sl < TS; sl += 8) {
    const int sidx = s0 + sl;
    if (sidx < S && r < R) out[base + (size_t)sidx * R + r] = tile[lane][sl];
  }
}

template <typename T>
__global__ void widen_rois(const T* __restrict__ in, float* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = to_f32<T>(in[i]);
}

static bool nchw_fast_ok(int N, int C, int H, int W, int K, int PH, int PW, int sampling_ratio, int pool_mode, int dtype) {
  if (pool_mode != G4R_POOL_AVG) return false;
  if (dtype != G4R_F32 && dtype != G4R_F16 && dtype != G4R_BF16) return false;
  const int vec = 16 / (int)dtype_size(dtype);
  if (C < 64 || C % vec != 0) return false;
  if (H > 65535 || W > 65535) return false;
  const int g = sampling_ratio > 0 ? sampling_ratio : 2;
  // worth three streaming passes only when the tap work outweighs touching every map element twice
  return (double)K * PH * PW * 4.0 * g * g >= 2.0 * (double)N * H * W;
}

static size_t nchw_fast_bytes(int N, int C, int H, int W, int K, int PH, int PW, int dtype) {
  const size_t es = dtype_size(dtype);
  auto al = [](size_t v) { return (v + 255) / 256 * 256; };
  return al((size_t)N * C * H * W * es) + al((size_t)K * C * PH * PW * es) + al((size_t)K * 5 * 4);
}

template <typename T>
static int nchw_fast_run(const void* input, const void* rois, void* output, int N, int C, int H, int W, int K, int PH,
                         int PW, float scale, int sr, int aligned, int dtype, void* ws, cudaStream_t st) {
  auto al = [](size_t v) { return (v + 255) / 256 * 256; };
  const size_t es = sizeof(T);
  char* w0 = (char*)ws;
  T* in_t = (T*)w0;
  T* out_t = (T*)(w0 + al((size_t)N * C * H * W * es));
  float* rois32 = (float*)(w0 + al((size_t)N * C * H * W * es) + al((size_t)K * C * PH * PW * es));
  const int HW = H * W;
  G4R_REQUIRE(N <= 65535 && K <= 65535 * 64, "nchw fast path: batch too large");
  transpose_batched<T><<<dim3((HW + 32 * (16 / (int)sizeof(T)) - 1) / (32 * (16 / (int)sizeof(T))), (C + 31) / 32, N), 256, 0, st>>>((const T*)input, in_t, C, HW);
  G4R_LAUNCH_CHECK("transpose_batched(in)");
  const float* rp = (const float*)rois;
  if (dtype != G4R_F32) {
    widen_rois<T><<<(K * 5 + 255) / 256, 256, 0, st>>>((const T*)rois, rois32, K * 5);
    G4R_LAUNCH_CHECK("widen_rois");
    rp = rois32;
  }
  MlvlParams p{};
  p.maps[0] = in_t; p.H[0] = H; p.W[0] = W; p.scale[0] = scale;
  p.rois = rp; p.out = out_t;
  p.N = N; p.C = C; p.K = K; p.PH = PH; p.PW = PW; p.sampling_ratio = sr; p.aligned = aligned; p.n_levels = 1;
  p.one = 1.0f;
  int rc = launch_fwd_mlvl<T, T>(p, false, st);
  if (rc) return rc;
  // out_t [K][PH*PW][C] -> output [K][C][PH*PW]; K can exceed gridDim.z: chunk it
  const int P = PH * PW;
  for (int k0 = 0; k0 < K; k0 += 65535) {
    const int kb = K - k0 < 65535 ? K - k0 : 65535;
    transpose_batched<T><<<dim3((C + 32 * (16 / (int)sizeof(T)) - 1) / (32 * (16 / (int)sizeof(T))), (P + 31) / 32, kb), 256, 0, st>>>(out_t + (size_t)k0 * P * C,
                                                                               (T*)output + (size_t)k0 * P * C, P, C);
    G4R_LAUNCH_CHECK("transpose_batched(out)");
  }
  return G4R_OK;
}

}  // namespace g4r

using namespace g4r;

extern "C" int g4r_roi_align_mlvl_forward(const void* const* maps, const int* H, const int* W,
                                          const float* scales, int n_levels, const float* rois,
                                          void* output, int N, int C, int K, int PH, int PW,
                                          int sampling_ratio, int aligned, int in_dtype, int out_dtype,
                                          const float* const* gn_scale, const float* const* gn_shift,
                                          void* stream) {
  G4R_REQUIRE(n_levels >= 1 && n_levels <= G4R_MAX_LEVELS, "n_levels=%d out of range", n_levels);
  G4R_REQUIRE(maps && H && W && scales && output, "null argument");
  G4R_REQUIRE(N > 0 && C > 0 && PH > 0 && PW > 0 && K >= 0, "bad sizes N=%d C=%d K=%d PH=%d PW=%d", N, C, K, PH, PW);
  G4R_REQUIRE(in_dtype == G4R_F32 || in_dtype == G4R_F16 || in_dtype == G4R_BF16, "in_dtype %d unsupported", in_dtype);
  G4R_REQUIRE(out_dtype == G4R_F32 || out_dtype == G4R_F16 || out_dtype == G4R_BF16, "out_dtype %d unsupported", out_dtype);
  const int vec = 16 / (int)dtype_size(in_dtype);
  G4R_REQUIRE(C % vec == 0, "C=%d must be a multiple of %d for 128-bit channel vectors", C, vec);
  G4R_REQUIRE((gn_scale == nullptr) == (gn_shift == nullptr), "gn_scale/gn_shift must both be given or both NULL");
  if (K == 0) return G4R_OK;
  G4R_REQUIRE(rois, "rois is NULL with K=%d", K);
  MlvlParams p{};
  p.one = 1.0f;
  for (int l = 0; l < n_levels; l++) {
    G4R_REQUIRE(maps[l] && H[l] > 0 && W[l] > 0, "level %d: bad map", l);
    G4R_REQUIRE(((uintptr_t)maps[l] & 15) == 0, "level %d: map not 16-byte aligned", l);
    p.maps[l] = maps[l];
    p.H[l] = H[l];
    p.W[l] = W[l];
    p.scale[l] = scales[l];
    p.gn_scale[l] = gn_scale ? gn_scale[l] : nullptr;
    p.gn_shift[l] = gn_shift ? gn_shift[l] : nullptr;
    if (gn_scale) G4R_REQUIRE(gn_scale[l] && gn_shift[l], "level %d: null gn_scale/shift", l);
  }
  G4R_REQUIRE(((uintptr_t)output & 15) == 0, "output not 16-byte aligned");
  for (int l = 0; l < n_levels; l++)
    G4R_REQUIRE((double)H[l] * W[l] * C < 2147483647.0, "level %d: H*W*C must fit int32 element offsets", l);
  p.rois = rois;
  p.out = output;
  p.N = N; p.C = C; p.K = K; p.PH = PH; p.PW = PW;
  p.sampling_ratio = sampling_ratio; p.aligned = aligned; p.n_levels = n_levels;
  p.rows_per_cta = pick_rows_per_cta(K, n_levels, PH);
  cudaStream_t st = (cudaStream_t)stream;
  const bool aff = gn_scale != nullptr;
#define G4R_DISPATCH_OUT(TIN)                                                              \
  switch (out_dtype) {                                                                     \
    case G4R_F32: return launch_fwd_mlvl<TIN, float>(p, aff, st);                          \
    case G4R_F16: return launch_fwd_mlvl<TIN, __half>(p, aff, st);                         \
    default: return launch_fwd_mlvl<TIN, __nv_bfloat16>(p, aff, st);                       \
  }
  switch (in_dtype) {
    case G4R_F32: G4R_DISPATCH_OUT(float)
    case G4R_F16: G4R_DISPATCH_OUT(__half)
    default: G4R_DISPATCH_OUT(__nv_bfloat16)
  }
#undef G4R_DISPATCH_OUT
}

extern "C" int g4r_roi_align_mlvl_backward(const void* grad_output, const int* H, const int* W,
                                           const float* scales, int n_levels, const float* rois,
                                           float* const* grad_maps, int N, int C, int K, int PH,
                                           int PW, int sampling_ratio, int aligned, int grad_dtype,
                                           void* stream) {
  G4R_REQUIRE(n_levels >= 1 && n_levels <= G4R_MAX_LEVELS, "n_levels=%d out of range", n_levels);
  G4R_REQUIRE(grad_output && H && W && scales && grad_maps, "null argument");
  G4R_REQUIRE(N > 0 && C > 0 && PH > 0 && PW > 0 && K >= 0, "bad sizes");
  G4R_REQUIRE(C % 4 == 0, "C=%d must be a multiple of 4", C);
  G4R_REQUIRE(grad_dtype == G4R_F32 || grad_dtype == G4R_F16 || grad_dtype == G4R_BF16, "grad_dtype %d unsupported", grad_dtype);
  if (K == 0) return G4R_OK;
  G4R_REQUIRE(rois, "rois is NULL");
  MlvlParams p{};
  for (int l = 0; l < n_levels; l++) {
    G4R_REQUIRE(grad_maps[l] && ((uintptr_t)grad_maps[l] & 15) == 0, "level %d: bad grad map", l);
    p.grad_maps[l] = grad_maps[l];
    p.H[l] = H[l]; p.W[l] = W[l]; p.scale[l] = scales[l];
  }
  p.rois = rois;
  p.out = const_cast<void*>(grad_output);
  p.N = N; p.C = C; p.K = K; p.PH = PH; p.PW = PW;
  p.sampling_ratio = sampling_ratio; p.aligned = aligned; p.n_levels = n_levels;
  p.rows_per_cta = pick_rows_per_cta(K, n_levels, PH);
  const int row_groups = (PH + p.rows_per_cta - 1) / p.rows_per_cta;
  dim3 grid((unsigned)(K * row_groups), n_levels);
  cudaStream_t st = (cudaStream_t)stream;
  switch (grad_dtype) {
    case G4R_F32: roi_align_bwd_nhwc_mlvl<float><<<grid, kThreads, 0, st>>>(p); break;
    case G4R_F16: roi_align_bwd_nhwc_mlvl<__half><<<grid, kThreads, 0, st>>>(p); break;
    default: roi_align_bwd_nhwc_mlvl<__nv_bfloat16><<<grid, kThreads, 0, st>>>(p); break;
  }
  G4R_LAUNCH_CHECK("roi_align_bwd_nhwc_mlvl");
  return G4R_OK;
}

static int check_common(const void* a, const void* rois, const void* b, int N, int C, int H, int W,
                        int K, int PH, int PW, int pool_mode, int dtype, int layout) {
  G4R_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0 && K >= 0 && PH > 0 && PW > 0,
              "bad sizes N=%d C=%d H=%d W=%d K=%d PH=%d PW=%d", N, C, H, W, K, PH, PW);
  G4R_REQUIRE(pool_mode == G4R_POOL_MAX || pool_mode == G4R_POOL_AVG, "pool_mode=%d", pool_mode);
  G4R_REQUIRE(dtype >= G4R_F32 && dtype <= G4R_F64, "dtype=%d", dtype);
  G4R_REQUIRE(layout == G4R_NCHW || layout == G4R_NHWC, "layout=%d", layout);
  if (K > 0) G4R_REQUIRE(a && rois && b, "null tensor pointer");
  return G4R_OK;
}

extern "C" int g4r_roi_align_forward(const void* input, const void* rois, void* output, void* argmax_y,
                                     void* argmax_x, int N, int C, int H, int W, int K, int PH, int PW,
                                     float spatial_scale, int sampling_ratio, int pool_mode,
                                     int aligned, int dtype, int layout, void* stream) {
  int rc = check_common(input, rois, output, N, C, H, W, K, PH, PW, pool_mode, dtype, layout);
  if (rc) return rc;
  if (K == 0) return G4R_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (pool_mode == G4R_POOL_MAX) G4R_REQUIRE(argmax_y && argmax_x, "max pooling needs argmax_y/argmax_x");
  if (layout == G4R_NHWC) {
    G4R_REQUIRE(pool_mode == G4R_POOL_AVG, "NHWC path implements avg pooling only");
    G4R_REQUIRE(dtype == G4R_F32, "NHWC single-level entry takes fp32 maps+rois; use g4r_roi_align_mlvl_forward for 16-bit maps");
    const void* maps[1] = {input};
    return g4r_roi_align_mlvl_forward(maps, &H, &W, &spatial_scale, 1, (const float*)rois, output, N, C,
                                      K, PH, PW, sampling_ratio, aligned, dtype, dtype, nullptr, nullptr,
                                      stream);
  }
  switch (dtype) {
    case G4R_F32: return launch_fwd_nchw<float>(input, rois, output, argmax_y, argmax_x, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    case G4R_F64: return launch_fwd_nchw<double>(input, rois, output, argmax_y, argmax_x, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    case G4R_F16: return launch_fwd_nchw<__half>(input, rois, output, argmax_y, argmax_x, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    default: return launch_fwd_nchw<__nv_bfloat16>(input, rois, output, argmax_y, argmax_x, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
  }
}

extern "C" size_t g4r_roi_align_forward_workspace(int N, int C, int H, int W, int K, int PH, int PW,
                                                  int sampling_ratio, int pool_mode, int dtype, int layout) {
  if (layout != G4R_NCHW || K <= 0) return 0;
  if (!nchw_fast_ok(N, C, H, W, K, PH, PW, sampling_ratio, pool_mode, dtype)) return 0;
  return nchw_fast_bytes(N, C, H, W, K, PH, PW, dtype);
}

extern "C" int g4r_roi_align_forward_ws(const void* input, const void* rois, void* output, void* argmax_y,
                                        void* argmax_x, int N, int C, int H, int W, int K, int PH, int PW,
                                        float spatial_scale, int sampling_ratio, int pool_mode, int aligned,
                                        int dtype, int layout, void* workspace, size_t workspace_bytes, void* stream) {
  const size_t need = g4r_roi_align_forward_workspace(N, C, H, W, K, PH, PW, sampling_ratio, pool_mode, dtype, layout);
  if (need == 0 || workspace == nullptr || workspace_bytes < need)
    return g4r_roi_align_forward(input, rois, output, argmax_y, argmax_x, N, C, H, W, K, PH, PW, spatial_scale,
                                 sampling_ratio, pool_mode, aligned, dtype, layout, stream);
  int rc = check_common(input, rois, output, N, C, H, W, K, PH, PW, pool_mode, dtype, layout);
  if (rc) return rc;
  G4R_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case G4R_F32: return nchw_fast_run<float>(input, rois, output, N, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, aligned, dtype, workspace, st);
    case G4R_F16: return nchw_fast_run<__half>(input, rois, output, N, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, aligned, dtype, workspace, st);
    default: return nchw_fast_run<__nv_bfloat16>(input, rois, output, N, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, aligned, dtype, workspace, st);
  }
}

extern "C" int g4r_roi_align_backward(const void* grad_output, const void* rois, const void* argmax_y,
                                      const void* argmax_x, void* grad_input, int N, int C, int H,
                                      int W, int K, int PH, int PW, float spatial_scale,
                                      int sampling_ratio, int pool_mode, int aligned, int dtype,
                                      int layout, void* stream) {
  int rc = check_common(grad_output, rois, grad_input, N, C, H, W, K, PH, PW, pool_mode, dtype, layout);
  if (rc) return rc;
  if (K == 0) return G4R_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (pool_mode == G4R_POOL_MAX) G4R_REQUIRE(argmax_y && argmax_x, "max pooling needs argmax_y/argmax_x");
  if (layout == G4R_NHWC) {
    G4R_REQUIRE(pool_mode == G4R_POOL_AVG && dtype == G4R_F32, "NHWC backward: fp32 avg only");
    float* gm[1] = {(float*)grad_input};
    return g4r_roi_align_mlvl_backward(grad_output, &H, &W, &spatial_scale, 1, (const float*)rois, gm, N,
                                       C, K, PH, PW, sampling_ratio, aligned, G4R_F32, stream);
  }
  switch (dtype) {
    case G4R_F32: return launch_bwd_nchw<float>(grad_output, rois, argmax_y, argmax_x, grad_input, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    case G4R_F64: return launch_bwd_nchw<double>(grad_output, rois, argmax_y, argmax_x, grad_input, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    case G4R_F16: return launch_bwd_nchw<__half>(grad_output, rois, argmax_y, argmax_x, grad_input, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
    default: return launch_bwd_nchw<__nv_bfloat16>(grad_output, rois, argmax_y, argmax_x, grad_input, C, H, W, K, PH, PW, spatial_scale, sampling_ratio, pool_mode, aligned, st);
  }
}
