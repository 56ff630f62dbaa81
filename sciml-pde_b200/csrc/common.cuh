// Shared declarations for libfno_sm100.so (B200 / sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/fno_sm100.h"

namespace fno {

// ---- plan ------------------------------------------------------------------------------------
// Immutable per-geometry tables, all in device memory.
//   twH  [NP][JP]   folded row twiddles for the strided axis of a 2-D plane, NP = H/2+1:
//                   cols 0..M1T      cos(2 pi j t / H)
//                   cols M1T+1..2M1T sin(2 pi j t / H), j = 1..M1T   (0 beyond m1)
//   twW  [2][m2][WP] cos / sin of 2 pi k2 w / W, WP = roundup(W, 4), zero padded
//   twX  [D1][2*m1][2]  (3-D only) cos / sin of 2 pi k1 d / D1 for the kept signed rows
struct Plan {
  int nd;            // 2 or 3
  int device;
  int D1;            // 3-D only: outer (strided) axis handled by the axis kernels
  int H, W;          // 2-D plane extents (3-D: D2, D3)
  int m1x;           // 3-D only: modes along D1
  int m1, m2;        // modes of the 2-D plane transform (3-D: m2, m3)
  int M1T;           // m1 rounded up to an instantiated template size
  int NP, JP, WP;
  float* twH;
  float* twW;
  float* twX;
  int G_fwd, G_inv;  // planes per CTA
  // tensor-core W-axis stage of K1 (transform2d_tc.cu): F = [cos | sin](2 pi q w / W) hi / lo in the K-major
  // UMMA layout, tc_nch 16-byte w chunks per row (0 = path not available for this geometry)
  float* tcF_hi;
  float* tcF_lo;
  float* tcF_bf;     // the same table rounded to bfloat16 (bf16 math mode)
  int tc_nch;
};

// One-time setup that must run once PER DEVICE: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the current
// device only, so a process-wide flag would leave the second GPU of a single-process multi-GPU program without it.
struct PerDeviceOnce {
  std::atomic<int> done[64];
  PerDeviceOnce() { for (auto& d : done) d.store(0); }
  static int current() { int d = 0; return cudaGetDevice(&d) == cudaSuccess ? d : -1; }
  bool need() const { const int d = current(); return d < 0 || d >= 64 || !done[d].load(); }
  void mark() { const int d = current(); if (d >= 0 && d < 64) done[d].store(1); }
};

void set_error(const char* fmt, ...);
int check_launch(const char* what);
extern std::atomic<unsigned long long> g_launches;
extern std::atomic<int> g_math_mode;     // FNO_MATH_FP32 (3xTF32 split) / FNO_MATH_TF32 (single pass)
inline void count_launch(unsigned n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- kernel launchers (one per translation unit) -------------------------------------------
int launch_fwd2d(const Plan* p, const float* x, const float* preact, float* ds_out, float* X,
                 long planes, int cmode, float scale, cudaStream_t st);
int launch_inv2d(const Plan* p, const float* Y, const float* addend, float* s_out, float* out,
                 long planes, int cmode, float scale, int apply_gelu, cudaStream_t st);
int setup_transform2d_attrs(const Plan* p);
int launch_fwd2d_ws(const Plan* p, const float* x, const float* preact, float* ds_out, float* X, float* work,
                    long planes, int cmode, float scale, cudaStream_t st);
int launch_fwd2d_tcap(const Plan* p, const float* g, const float* preact, float* ds_out, float* T1, long planes,
                      cudaStream_t st, bool attr_only);
int launch_fwd2d_tca(const Plan* p, const float* x, float* T1, long planes, cudaStream_t st, bool attr_only);
bool layer2d_tc_supported(const Plan* p, int C);
int setup_layer2d_tc_attrs();
size_t layer2d_tc_workspace_bytes(const Plan* p, int B, int C);
int launch_layer2d_tc(const Plan* p, const float* Y, const float* a, const float* Wl, const float* bias, float* s_out,
                      float* out, float* work, int B, int C, int cmode, float scale, int apply_gelu, int transpose_w,
                      cudaStream_t st);
size_t head_bwd_tc_workspace_bytes();
int head_pad_zero(float* dh, int R_in, int W_in, int R_out, int Wp, long planes, cudaStream_t st);
int launch_axis_fwd(const Plan* p, const float* S, float* X, long planes, long Q, cudaStream_t st);
int launch_axis_inv(const Plan* p, const float* Y, float* Z, long planes, long Q, cudaStream_t st);
int launch_mix_fwd(const Plan* p, const float* X, const float* const* w, float* Y, int B, int Ci,
                   int Co, cudaStream_t st);
int launch_mix_bwd_data(const Plan* p, const float* gY, const float* const* w, float* gX, int B,
                        int Ci, int Co, cudaStream_t st);
int launch_mix_bwd_weight(const Plan* p, const float* X, const float* gY, float* const* gw, int B,
                          int Ci, int Co, cudaStream_t st);
bool mix_tc_supported(const Plan* p, int Ci, int Co);
bool pointwise_tc_supported(int Cin, int Cout);
int launch_wgrad_tc_rows128(const float* ds, const float* a, float* part, int B, int Co, int Ci, long N, int max_parts,
                            int* nparts, cudaStream_t st);
int launch_wgrad_tc(const float* ds, const float* a, float* part, int B, int Co, int Ci, long N, int max_parts, int* nparts,
                    cudaStream_t st);
int launch_pointwise_tc(const float* in, const float* W, const float* bias, float* out, int B, int Co, int Ci, long N,
                        int transpose, cudaStream_t st);

// ---- split-K reduction ------------------------------------------------------------------------
// The weight gradients are computed split-K: every CTA writes a record of partial sums and one more launch sums the
// records in a fixed order, so the result is deterministic.  Output k of a segment reads record offset
//   col + k                                    (row == 0: a contiguous run), or
//   (k / row) * stride + col + k % row         (row > 0: a [n / row][row] matrix stored with pitch `stride`),
// plus q * copy_stride for each of the `copies` sub-records of one record that sum into the same output.
// A null dst skips the segment's stores; unused segments have n == 0.
struct ReduceSeg {
  float* dst = nullptr;
  int n = 0;
  int col = 0;
  int row = 0;
  int stride = 0;
  int copies = 1;
  int copy_stride = 0;
};
struct ReduceSegs {
  ReduceSeg s[4];
};
// out = sum over the nparts records of length reclen at `part`; one warp per output element.
int launch_partial_reduce(const float* part, int nparts, int reclen, const ReduceSegs& segs, cudaStream_t st);

// ---- 2-D tensor maps (cuTensorMapEncodeTiled, resolved once through the runtime: no link-time libcuda dependency) -----
bool tensor_maps_available();
// The [planes][pixels] view of a channel-first f32 tensor with a box of {box_pixels, box_planes}, zero fill outside.
// elem_bytes 4 reads a row as FLOAT32; 8 as UINT64 float pairs (pixels and box_pixels even), which fits twice the
// pixels into the 256-element box limit.  False when the entry point is missing or the encoding is rejected.
bool make_plane_map(CUtensorMap* m, const float* base, unsigned long long pixels, unsigned long long planes,
                    unsigned box_pixels, unsigned box_planes, unsigned elem_bytes, CUtensorMapL2promotion l2);

// ---- device helpers --------------------------------------------------------------------------
// exact unsigned 32-bit division by a run-time constant (Granlund-Montgomery): 4 instructions instead
// of the ~35 of a hardware-less integer division -- a loader warp is one dependent instruction stream
struct FastDiv {
  unsigned d, m, l;
  __host__ void init(unsigned div) {
    d = div;
    l = 0;
    while ((1ull << l) < div) ++l;
    m = (unsigned)(((1ull << 32) * ((1ull << l) - div)) / div + 1);
  }
  __device__ __forceinline__ unsigned div(unsigned n) const {
    const unsigned t = __umulhi(m, n);
    return l == 0 ? n : (t + ((n - t) >> 1)) >> (l - 1);
  }
};


__device__ __forceinline__ float gelu_exact(float s) {
  return 0.5f * s * (1.0f + erff(s * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_exact_grad(float s) {
  const float cdf = 0.5f * (1.0f + erff(s * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * expf(-0.5f * s * s);
  return fmaf(s, pdf, cdf);
}


// Exact-erf GELU and its derivative through the Abramowitz-Stegun 7.1.26 rational form of erfc,
//     0.5 erfc(z) = q = 0.5 t (a1 + a2 t + ... + a5 t^4) exp(-z^2),  t = 1 / (1 + p z),  z = |s| / sqrt(2)
// which shares exp(-s^2/2) with the Gaussian pdf of the derivative.  Absolute error of the cdf
// < 6e-7 in fp32 (tests/test_kernels_gpu.py bounds it through the layer / head parity tests), far
// inside the 1e-5 parity budget.  13 instructions for GELU (4 FMUL, 6 FFMA, 2 MUFU, 1 FMNMX), 16
// for GELU + GELU'; erff + expf cost ~40.  Written on |s| so that both tails are free of
// cancellation:  gelu(s) = max(s, 0) - |s| q.
__device__ __forceinline__ float gelu_half_erfc(float as, float& e) {
  const float u = as * 0.8493218002880191f;                       // u^2 = (s^2 / 2) log2(e)
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.2316418882663604f, as, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-(u * u)));    // exp(-s^2 / 2)
  float poly = fmaf(0.5307027145f, t, -0.7265760135f);
  poly = fmaf(poly, t, 0.7107068705f);
  poly = fmaf(poly, t, -0.142248368f);
  poly = fmaf(poly, t, 0.127414796f);
  return (poly * t) * e;
}
__device__ __forceinline__ float gelu_fast(float s) {
  float e;
  const float as = fabsf(s);
  const float q = gelu_half_erfc(as, e);
  return fmaf(-as, q, fmaxf(s, 0.0f));
}
__device__ __forceinline__ void gelu_fast_both(float s, float& g, float& gp) {
  float e;
  const float as = fabsf(s);
  const float q = gelu_half_erfc(as, e);
  g = fmaf(-as, q, fmaxf(s, 0.0f));
  const float cdf = 0.5f + copysignf(0.5f - q, s);
  gp = fmaf(s * 0.3989422804014327f, e, cdf);
}
__device__ __forceinline__ float gelu_fast_grad(float s) {
  float e;
  const float q = gelu_half_erfc(fabsf(s), e);
  const float cdf = 0.5f + copysignf(0.5f - q, s);
  return fmaf(s * 0.3989422804014327f, e, cdf);
}

// Two-element forms on the packed f32x2 pipe (FFMA2 / FMUL2 / FADD2): every lane is rounded exactly like the scalar
// instruction and the operations run in the scalar forms' order, so .x / .y are bit-identical to gelu_fast /
// gelu_fast_both of .x / .y, at one issue slot per two elements.  The epilogues that use them are bound by
// instruction issue, not by the FMA pipe.  Written on nas = -|s|: u = nas c gives the same u^2, fma(-c, nas, 1) the
// same 1 + c|s|, and fma(nas, q, max(s, 0)) is the scalar fma(-|s|, q, max(s, 0)); 0.5 - q is fma(q, -1, 0.5).
__device__ __forceinline__ float2 f32x2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 gelu_half_erfc2(float2 nas, float2& e) {
  const float2 u = __fmul2_rn(nas, f32x2(0.8493218002880191f));
  const float2 d = __ffma2_rn(f32x2(-0.2316418882663604f), nas, f32x2(1.0f));
  const float2 uu = __fmul2_rn(u, u);
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(d.y));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(-uu.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(-uu.y));
  float2 poly = __ffma2_rn(f32x2(0.5307027145f), t, f32x2(-0.7265760135f));
  poly = __ffma2_rn(poly, t, f32x2(0.7107068705f));
  poly = __ffma2_rn(poly, t, f32x2(-0.142248368f));
  poly = __ffma2_rn(poly, t, f32x2(0.127414796f));
  return __fmul2_rn(__fmul2_rn(poly, t), e);
}
__device__ __forceinline__ float2 gelu_fast2(float2 s) {
  float2 e;
  const float2 nas = make_float2(-fabsf(s.x), -fabsf(s.y));
  const float2 q = gelu_half_erfc2(nas, e);
  return __ffma2_rn(nas, q, make_float2(fmaxf(s.x, 0.0f), fmaxf(s.y, 0.0f)));
}
__device__ __forceinline__ void gelu_fast_both2(float2 s, float2& g, float2& gp) {
  float2 e;
  const float2 nas = make_float2(-fabsf(s.x), -fabsf(s.y));
  const float2 q = gelu_half_erfc2(nas, e);
  g = __ffma2_rn(nas, q, make_float2(fmaxf(s.x, 0.0f), fmaxf(s.y, 0.0f)));
  const float2 r = __ffma2_rn(q, f32x2(-1.0f), f32x2(0.5f));
  const float2 cdf = __fadd2_rn(f32x2(0.5f), make_float2(copysignf(r.x, s.x), copysignf(r.y, s.y)));
  gp = __ffma2_rn(__fmul2_rn(s, f32x2(0.3989422804014327f)), e, cdf);
}

// ---- mbarrier / bulk-copy (TMA, 1-D) helpers --------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug traps instead of hanging the GPU.  The suspend-time hint lets the hardware
// park the warp until the phase completes instead of returning to the spin loop every few dozen cycles
// (ncu on head_bwd_tc: a third of all issued instructions were TRYWAIT / BRA pairs of waiting warps).
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned addr = smem_u32(bar);
  unsigned long long t0 = 0;
#pragma unroll 1
  for (unsigned spin = 0;; ++spin) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(20000u)
        : "memory");
    if (ok) return;
    if ((spin & 1023u) == 1023u) {          // wall-clock bound (4 s), whatever one try_wait lasts
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 4000000000ull) __trap();
    }
  }
}
// polling wait (mbarrier.test_wait never suspends the warp): for hand-offs on the critical path of a short
// pipeline step, where the wake-up latency of a parked warp is comparable to the step itself.  Same 4 s bound.
__device__ __forceinline__ void mbar_wait_spin(unsigned long long* bar, unsigned parity) {
  const unsigned addr = smem_u32(bar);
  unsigned long long t0 = 0;
#pragma unroll 1
  for (unsigned spin = 0;; ++spin) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if ((spin & 0xfffffu) == 0xfffffu) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 4000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// one box of a 2-D tensor map at element coordinates {c0, c1}; completes on `bar` with the box's full byte count
// (elements outside the tensor are zero-filled and still counted)
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace fno
