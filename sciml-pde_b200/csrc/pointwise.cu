// 1x1-conv bypass of a Fourier layer (nn.Conv2d/3d(width, width, 1), fno/fno.py:131-134,162) on
// channel-first activations [B, C, N]: a per-pixel C x C matrix product.  FP32 CUDA-core path.
//
//   forward / data gradient: each thread owns VEC consecutive pixels and OT output channels; the
//     weight tile sits transposed in shared memory so that the OT weights of one input channel
//     are warp-uniform float4 broadcasts; every activation element is read exactly once per
//     output-channel tile with a coalesced 128-bit load.
//   weight gradient: gW[o,i] = sum_{b,p} ds[b,o,p] a[b,i,p] is a [C x K][K x C] product with a
//     huge K = B*N and a tiny output, so it is a split-K reduction: a CTA stages a K-slab of both
//     operands in shared memory, each warp owns a T x T output tile with lanes striding K, and
//     per-CTA partials are combined by a second fixed-order pass (deterministic, no atomics).
#include <cstring>

#include "common.cuh"

namespace fno {
namespace {

template <int OT, int VEC, bool TRANSPOSE>
__global__ void __launch_bounds__(256)
pointwise_kernel(const float* __restrict__ in, const float* __restrict__ Wm, const float* __restrict__ bias,
                 float* __restrict__ out, int Cin, int Cout, int Co, int Ci, long N) {
  extern __shared__ __align__(16) float ws[];  // [Cin][OT] weights, then [OT] bias
  const int o0 = blockIdx.y * OT;
  const int b = blockIdx.z;
  for (int idx = threadIdx.x; idx < Cin * OT; idx += blockDim.x) {
    const int s = idx / OT, oo = idx - s * OT;
    const int oc = o0 + oo;
    float v = 0.f;
    if (oc < Cout) v = TRANSPOSE ? Wm[(size_t)s * Ci + oc] : Wm[(size_t)oc * Ci + s];
    ws[idx] = v;
  }
  float* bs = ws + Cin * OT;
  for (int idx = threadIdx.x; idx < OT; idx += blockDim.x)
    bs[idx] = (bias != nullptr && o0 + idx < Cout) ? bias[o0 + idx] : 0.f;
  __syncthreads();

  const long p0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (p0 >= N) return;
  float acc[OT][VEC];
#pragma unroll
  for (int oo = 0; oo < OT; ++oo)
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[oo][v] = bs[oo];
  const float* __restrict__ ip = in + (size_t)b * Cin * N + p0;
#pragma unroll 4
  for (int s = 0; s < Cin; ++s) {
    float xv[VEC];
    if constexpr (VEC == 4) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(ip + (size_t)s * N));
      xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w;
    } else {
      xv[0] = __ldg(ip + (size_t)s * N);
    }
    const float* wrow = ws + s * OT;
#pragma unroll
    for (int oo = 0; oo < OT; ++oo) {
      const float wv = wrow[oo];
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[oo][v] = fmaf(wv, xv[v], acc[oo][v]);
    }
  }
  float* __restrict__ op = out + (size_t)b * Cout * N + p0;
#pragma unroll
  for (int oo = 0; oo < OT; ++oo) {
    if (o0 + oo >= Cout) break;
    if constexpr (VEC == 4) {
      *reinterpret_cast<float4*>(op + (size_t)(o0 + oo) * N) =
          make_float4(acc[oo][0], acc[oo][1], acc[oo][2], acc[oo][3]);
    } else {
      op[(size_t)(o0 + oo) * N] = acc[oo][0];
    }
  }
}

// v2 of the forward / data-gradient product for even plane sizes: two adjacent pixels per thread
// (64-bit coalesced accesses), every output channel of the CTA's tile in registers, and the input
// channels fetched in bursts of PW_CH loads that are all issued before the first FMA consumes
// them -- 16 resident warps per SM each with PW_CH x 8 bytes in flight cover the HBM latency that
// the one-load-at-a-time loop above exposes (profiles/r1_b: 183 registers, 12 % occupancy).
constexpr int PW_CH = 20;

template <int OT, bool TRANSPOSE, int CH = PW_CH>
__global__ void __launch_bounds__(256, 2)
pointwise2_kernel(const float* __restrict__ in, const float* __restrict__ Wm, const float* __restrict__ bias,
                  float* __restrict__ out, int Cin, int Cout, int Co, int Ci, long N2) {
  extern __shared__ __align__(16) float ws[];  // [Cin][OT] weights, then [OT] bias
  const int o0 = blockIdx.y * OT;
  const int b = blockIdx.z;
  for (int idx = threadIdx.x; idx < Cin * OT; idx += blockDim.x) {
    const int s = idx / OT, oo = idx - s * OT;
    const int oc = o0 + oo;
    float v = 0.f;
    if (oc < Cout) v = TRANSPOSE ? Wm[(size_t)s * Ci + oc] : Wm[(size_t)oc * Ci + s];
    ws[idx] = v;
  }
  float* bs = ws + Cin * OT;
  for (int idx = threadIdx.x; idx < OT; idx += blockDim.x)
    bs[idx] = (bias != nullptr && o0 + idx < Cout) ? bias[o0 + idx] : 0.f;
  __syncthreads();

  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= N2) return;
  float2 acc[OT];
#pragma unroll
  for (int oo = 0; oo < OT; ++oo) acc[oo] = make_float2(bs[oo], bs[oo]);
  const float2* __restrict__ ip = reinterpret_cast<const float2*>(in) + (size_t)b * Cin * N2 + p;
  for (int s0 = 0; s0 < Cin; s0 += CH) {
    float2 xv[CH];
#pragma unroll
    for (int u = 0; u < CH; ++u)
      xv[u] = (s0 + u < Cin) ? __ldg(ip + (size_t)(s0 + u) * N2) : make_float2(0.f, 0.f);
#pragma unroll
    for (int u = 0; u < CH; ++u) {
      if (s0 + u < Cin) {
        const float4* wrow = reinterpret_cast<const float4*>(ws + (s0 + u) * OT);
#pragma unroll
        for (int q = 0; q < OT / 4; ++q) {
          const float4 w = wrow[q];
          acc[4 * q + 0].x = fmaf(w.x, xv[u].x, acc[4 * q + 0].x); acc[4 * q + 0].y = fmaf(w.x, xv[u].y, acc[4 * q + 0].y);
          acc[4 * q + 1].x = fmaf(w.y, xv[u].x, acc[4 * q + 1].x); acc[4 * q + 1].y = fmaf(w.y, xv[u].y, acc[4 * q + 1].y);
          acc[4 * q + 2].x = fmaf(w.z, xv[u].x, acc[4 * q + 2].x); acc[4 * q + 2].y = fmaf(w.z, xv[u].y, acc[4 * q + 2].y);
          acc[4 * q + 3].x = fmaf(w.w, xv[u].x, acc[4 * q + 3].x); acc[4 * q + 3].y = fmaf(w.w, xv[u].y, acc[4 * q + 3].y);
        }
      }
    }
  }
  float2* __restrict__ op = reinterpret_cast<float2*>(out) + (size_t)b * Cout * N2 + p;
#pragma unroll
  for (int oo = 0; oo < OT; ++oo) {
    if (o0 + oo >= Cout) break;
    op[(size_t)(o0 + oo) * N2] = acc[oo];
  }
}

template <int OT, int CH = PW_CH>
int launch_pw2(const float* in, const float* Wm, const float* bias, float* out, int B, int Co, int Ci, long N,
               int transpose, cudaStream_t st) {
  const int Cin = transpose ? Co : Ci;
  const int Cout = transpose ? Ci : Co;
  const long N2 = N / 2;
  dim3 grid((unsigned)((N2 + 255) / 256), (Cout + OT - 1) / OT, B);
  const size_t smem = sizeof(float) * ((size_t)Cin * OT + OT);
  if (transpose)
    pointwise2_kernel<OT, true, CH><<<grid, 256, smem, st>>>(in, Wm, bias, out, Cin, Cout, Co, Ci, N2);
  else
    pointwise2_kernel<OT, false, CH><<<grid, 256, smem, st>>>(in, Wm, bias, out, Cin, Cout, Co, Ci, N2);
  count_launch();
  return check_launch("pointwise2_kernel");
}

template <int OT, int VEC>
int launch_pw(const float* in, const float* Wm, const float* bias, float* out, int B, int Co, int Ci, long N,
              int transpose, cudaStream_t st) {
  const int Cin = transpose ? Co : Ci;
  const int Cout = transpose ? Ci : Co;
  const int threads = 256;
  const long nvec = (N + VEC - 1) / VEC;
  dim3 grid((unsigned)((nvec + threads - 1) / threads), (Cout + OT - 1) / OT, B);
  const size_t smem = sizeof(float) * ((size_t)Cin * OT + OT);
  if (transpose)
    pointwise_kernel<OT, VEC, true><<<grid, threads, smem, st>>>(in, Wm, bias, out, Cin, Cout, Co, Ci, N);
  else
    pointwise_kernel<OT, VEC, false><<<grid, threads, smem, st>>>(in, Wm, bias, out, Cin, Cout, Co, Ci, N);
  count_launch();
  return check_launch("pointwise_kernel");
}

// ------------------------------------------------------------------------------------------
// weight / bias gradient
// ------------------------------------------------------------------------------------------
constexpr int KT = 128;      // pixels per shared-memory slab
constexpr int WG_T = 10;     // output tile edge per warp (register tile T x T)
constexpr int WG_MAXW = 8;   // warps (= output tiles) per CTA

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// Persistent split-K: CTA c owns the contiguous slab range [c*spc, (c+1)*spc) of the B*slabs_per_sample
// slabs (slab = KT consecutive pixels of one sample, all channels of ds and a).  Slabs stream through
// a 2-stage cp.async ring (16-byte copies, zero-filled past the end of the sample).
// part[cta][Co][Ci + 1]  (last column: bias gradient)
template <int T>
__global__ void __launch_bounds__(32 * WG_MAXW)
wgrad_partial_kernel(const float* __restrict__ ds, const float* __restrict__ a, float* __restrict__ part,
                     int Co, int Ci, long N, int slabs_per_sample, long total_slabs, long slabs_per_cta,
                     int tiles_i, int ntiles, int aligned) {
  extern __shared__ __align__(16) float sm[];  // 2 stages x ([Co][KT] ds slab, [Ci][KT] a slab)
  const int rows = Co + Ci;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  const int tile = blockIdx.y * nwarps + warp;
  const bool has_tile = tile < ntiles;
  const int to = has_tile ? (tile / tiles_i) * T : 0;
  const int ti = has_tile ? (tile % tiles_i) * T : 0;
  const bool bias_tile = has_tile && (ti == 0);
  long s_begin = (long)blockIdx.x * slabs_per_cta;
  long s_end = s_begin + slabs_per_cta;
  if (s_end > total_slabs) s_end = total_slabs;

  float acc[T][T];
  float accb[T];
#pragma unroll
  for (int r = 0; r < T; ++r) {
    accb[r] = 0.f;
#pragma unroll
    for (int c = 0; c < T; ++c) acc[r][c] = 0.f;
  }

  auto issue = [&](long slab, int stage) {
    float* dst = sm + (size_t)stage * rows * KT;
    const long b = slab / slabs_per_sample;
    const long k0 = (slab - b * slabs_per_sample) * KT;
    const float* dsb = ds + (size_t)b * Co * N;
    const float* ab = a + (size_t)b * Ci * N;
    if (aligned) {
      for (int idx = threadIdx.x; idx < rows * (KT / 4); idx += blockDim.x) {
        const int c = idx / (KT / 4), q = idx - c * (KT / 4);
        const long k = k0 + 4 * q;
        const float* src = (c < Co) ? (dsb + (size_t)c * N + k) : (ab + (size_t)(c - Co) * N + k);
        long left = (N - k) * 4;
        const int nb = left >= 16 ? 16 : (left > 0 ? (int)left : 0);
        cp_async16(dst + c * KT + 4 * q, nb > 0 ? src : ds, nb);
      }
    } else {
      for (int idx = threadIdx.x; idx < rows * KT; idx += blockDim.x) {
        const int c = idx / KT, kk = idx - c * KT;
        const long k = k0 + kk;
        const float* src = (c < Co) ? (dsb + (size_t)c * N + k) : (ab + (size_t)(c - Co) * N + k);
        dst[idx] = (k < N) ? __ldg(src) : 0.f;
      }
    }
    cp_async_commit();
  };

  if (s_begin < s_end) issue(s_begin, 0);
  for (long slab = s_begin; slab < s_end; ++slab) {
    const int stage = (int)((slab - s_begin) & 1);
    if (slab + 1 < s_end) {
      issue(slab + 1, stage ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (has_tile) {
      const float* ds_s = sm + (size_t)stage * rows * KT;
      const float* a_s = ds_s + (size_t)Co * KT;
#pragma unroll
      for (int kk = 0; kk < KT; kk += 32) {
        float dv[T], av[T];
#pragma unroll
        for (int r = 0; r < T; ++r) dv[r] = (to + r < Co) ? ds_s[(to + r) * KT + kk + lane] : 0.f;
#pragma unroll
        for (int c = 0; c < T; ++c) av[c] = (ti + c < Ci) ? a_s[(ti + c) * KT + kk + lane] : 0.f;
#pragma unroll
        for (int r = 0; r < T; ++r) {
          accb[r] += dv[r];
#pragma unroll
          for (int c = 0; c < T; ++c) acc[r][c] = fmaf(dv[r], av[c], acc[r][c]);
        }
      }
    }
    __syncthreads();  // the stage is refilled by the next iteration's issue()
  }
  if (!has_tile) return;
  float* __restrict__ pp = part + (size_t)blockIdx.x * Co * (Ci + 1);
#pragma unroll
  for (int r = 0; r < T; ++r) {
#pragma unroll
    for (int c = 0; c < T; ++c) {
      float v = acc[r][c];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0 && to + r < Co && ti + c < Ci) pp[(size_t)(to + r) * (Ci + 1) + ti + c] = v;
    }
    if (bias_tile) {
      float v = accb[r];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0 && to + r < Co) pp[(size_t)(to + r) * (Ci + 1) + Ci] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// v2 of the weight gradient: TMA-fed slabs with an mbarrier full/empty ring.  Warp 0 streams slab after slab into a
// WG2_STAGES-deep ring; the warps each own one T x T output tile with lanes over pixel quads (LDS.128: 2T loads per
// 4 T^2 FMA).  Nothing but the tensor-map copies touches global memory in the steady state, so the kernel streams at the
// HBM rate set by its 8 bytes/pixel/channel.
// ------------------------------------------------------------------------------------------
constexpr int WG2_STAGES = 2;
constexpr int WG2_KT = 512;      // pixels per slab: the 256-element box limit, in float pairs
constexpr int WG2_MAXW = 8;      // consumer warps per CTA
// A slab is TWO 2-D tensor-map copies -- box {512 pixels, C planes} of the [planes][pixels] view of ds and of a, with the row
// taken as 8-byte elements so that 512 pixels fit the 256-element box limit: 40 KB per copy at width 20 instead of Co + Ci
// bulk copies of 2 KB.  Pixels past the end of a sample are zero-filled by the TMA unit (and still counted by complete_tx).
// Measured at cfg 1 (B = 128, profiles/r2g_wgrad_forms.md): one bulk copy per channel row 124 us, the same ring fed by tensor
// maps 93 us, + FULL 89 us; a kernel that only waits for its slabs 79-85 us in every form (the TMA feed tops out at ~4.5 TB/s),
// and every bulk copy costs ~40 ns of issue on top.

// DGRAD: the same pass also produces the bypass data gradient dx[b, i, p] = sum_o W[o, i] ds[b, o, p]
// (autograd of nn.Conv2d(C, C, 1), fno/fno.py:162) from the ds slab that is already in shared memory --
// one read of the ds tensor per layer instead of two.  Thread = two adjacent pixels of the 512-pixel slab
// (8 consumer warps), all Ci outputs in registers, weight rows broadcast with LDS.128.
template <int T, bool DGRAD, bool FULL>
__global__ void __launch_bounds__(32 * WG2_MAXW)
wgrad2_partial_kernel(float* __restrict__ part, int Co, int Ci, long N, int slabs_per_sample, long total_slabs,
                      long slabs_per_cta, int tiles_i, int ntiles, int nwarps, int KH, const float* __restrict__ Wm,
                      float* __restrict__ dx, const __grid_constant__ CUtensorMap tm_ds, const __grid_constant__ CUtensorMap tm_a) {
  extern __shared__ __align__(128) float wg2_sm[];  // WG2_STAGES x ([Co][WG2_KT] ds slab, [Ci][WG2_KT] a slab), then barriers
  float* const sm = wg2_sm;
  const int rows = Co + Ci;
  unsigned long long* full = reinterpret_cast<unsigned long long*>(sm + (size_t)WG2_STAGES * rows * WG2_KT);
  unsigned long long* empty = full + WG2_STAGES;
  float* ws = reinterpret_cast<float*>(empty + WG2_STAGES);            // DGRAD: W [Co][2T] (rows zero-padded)
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int s = 0; s < WG2_STAGES; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, nwarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (DGRAD) {
    for (int i = threadIdx.x; i < Co * 2 * T; i += blockDim.x) {
      const int o = i / (2 * T), c = i - o * (2 * T);
      ws[i] = (c < Ci) ? __ldg(Wm + (size_t)o * Ci + c) : 0.f;
    }
  }
  __syncthreads();
  long s_begin = (long)blockIdx.x * slabs_per_cta;
  long s_end = s_begin + slabs_per_cta;
  if (s_end > total_slabs) s_end = total_slabs;

  // ---- producer duty (warp 0): one tensor-map copy of ds and one of a per slab.  There is no
  // dedicated producer warp: a ninth warp would put three warps on one SM sub-partition and cap the kernel at
  // 168 registers (16 K registers per sub-partition), which the fused data-gradient phase does not fit.
  auto produce = [&](long slab) {
    if (slab >= s_end) return;
    const int it = (int)(slab - s_begin);
    const int stage = it % WG2_STAGES;
    const unsigned ph = (unsigned)(it / WG2_STAGES) & 1u;
    mbar_wait(empty + stage, ph ^ 1u);            // every consumer warp is done with the slab that used this stage
    const long b = slab / slabs_per_sample;
    const long k0 = (slab - b * slabs_per_sample) * WG2_KT;
    float* dst = sm + (size_t)stage * rows * WG2_KT;
    if (lane == 0) {
      mbar_arrive_expect_tx(full + stage, (unsigned)(WG2_KT * sizeof(float)) * (unsigned)rows);   // whole boxes, zero fill included
      const int c0 = (int)(k0 >> 1);                                                           // in float pairs
      tma_load_2d(dst, &tm_ds, c0, (int)(b * Co), full + stage);
      tma_load_2d(dst + (size_t)Co * WG2_KT, &tm_a, c0, (int)(b * Ci), full + stage);
    }
    __syncwarp();
  };
  if (warp == 0) {
    for (int s = 0; s < WG2_STAGES; ++s) produce(s_begin + s);
  }

  // ---- consumer warps: (tile, pixel part) each; a tile is a T x T block of outputs ------------
  const int kh = warp % KH;                       // which 1/KH of the slab's pixels
  const int tile = blockIdx.y * (nwarps / KH) + warp / KH;
  const bool has_tile = tile < ntiles;
  const int to = has_tile ? (tile / tiles_i) * T : 0;
  const int ti = has_tile ? (tile % tiles_i) * T : 0;
  // FULL (every tile complete, two tiles per tile row): no bounds predicates, operand addresses are one base register plus
  // immediates, and the two warps of a tile row share the bias rows (T/2 each) so that all warps carry the same work
  const bool bias_hi = FULL && ti != 0;
  const bool bias_tile = has_tile && (FULL || ti == 0);
  const float* const ds_t = sm + (size_t)to * WG2_KT + 4 * lane;
  const float* const a_t = sm + (size_t)(Co + ti) * WG2_KT + 4 * lane;
  float acc[T][T];
  float accb[T];
#pragma unroll
  for (int r = 0; r < T; ++r) {
    accb[r] = 0.f;
#pragma unroll
    for (int c = 0; c < T; ++c) acc[r][c] = 0.f;
  }
  const int steps = WG2_KT / 128;                    // 128 pixels (32 lanes x 4) per step
  for (long slab = s_begin; slab < s_end; ++slab) {
    const int it = (int)(slab - s_begin);
    const int stage = it % WG2_STAGES;
    const unsigned ph = (unsigned)(it / WG2_STAGES) & 1u;
    mbar_wait(full + stage, ph);
    const long b = slab / slabs_per_sample;
    const long left = N - (slab - b * slabs_per_sample) * WG2_KT;
    if (has_tile) {
      for (int st = kh; st < steps; st += KH) {
        const int px = st * 128 + 4 * lane;       // a short slab at the end of a sample ends on a quad (N % 4 == 0)
        if (px >= left) break;
        const float* ds_s = sm + (size_t)stage * rows * WG2_KT + px;
        const float* a_s = ds_s + (size_t)Co * WG2_KT;
        const int soff = stage * rows * WG2_KT + st * 128;
        float4 dv[T];
#pragma unroll
        for (int r = 0; r < T; ++r) {
          if (FULL) dv[r] = *reinterpret_cast<const float4*>(ds_t + soff + r * WG2_KT);
          else dv[r] = (to + r < Co) ? *reinterpret_cast<const float4*>(ds_s + (to + r) * WG2_KT) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (FULL) {
          if (!bias_hi) {
#pragma unroll
            for (int r = 0; r < T / 2; ++r) accb[r] += (dv[r].x + dv[r].y) + (dv[r].z + dv[r].w);
          } else {
#pragma unroll
            for (int r = T / 2; r < T; ++r) accb[r] += (dv[r].x + dv[r].y) + (dv[r].z + dv[r].w);
          }
        } else if (bias_tile) {
#pragma unroll
          for (int r = 0; r < T; ++r) accb[r] += (dv[r].x + dv[r].y) + (dv[r].z + dv[r].w);
        }
#pragma unroll
        for (int c = 0; c < T; ++c) {
          float4 av;
          if (FULL) av = *reinterpret_cast<const float4*>(a_t + soff + c * WG2_KT);
          else av = (ti + c < Ci) ? *reinterpret_cast<const float4*>(a_s + (ti + c) * WG2_KT) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int r = 0; r < T; ++r) {
            acc[r][c] = fmaf(dv[r].x, av.x, acc[r][c]);
            acc[r][c] = fmaf(dv[r].y, av.y, acc[r][c]);
            acc[r][c] = fmaf(dv[r].z, av.z, acc[r][c]);
            acc[r][c] = fmaf(dv[r].w, av.w, acc[r][c]);
          }
        }
      }
    }
    if (DGRAD) {
      const int px = 2 * (int)threadIdx.x;       // 256 consumer threads x 2 pixels = one slab
      if (px < left) {                            // `left` is a multiple of 4
        const long k0 = (slab - b * slabs_per_sample) * WG2_KT;
        const float* dsp = sm + (size_t)stage * rows * WG2_KT + px;
        float2 o2[2 * T];
#pragma unroll
        for (int i = 0; i < 2 * T; ++i) o2[i] = make_float2(0.f, 0.f);
        for (int o = 0; o < Co; ++o) {
          const float2 d = *reinterpret_cast<const float2*>(dsp + (size_t)o * WG2_KT);
          const float4* wrow = reinterpret_cast<const float4*>(ws + o * 2 * T);
#pragma unroll
          for (int q = 0; q < 2 * T / 4; ++q) {
            const float4 w = wrow[q];
            o2[4 * q + 0].x = fmaf(w.x, d.x, o2[4 * q + 0].x); o2[4 * q + 0].y = fmaf(w.x, d.y, o2[4 * q + 0].y);
            o2[4 * q + 1].x = fmaf(w.y, d.x, o2[4 * q + 1].x); o2[4 * q + 1].y = fmaf(w.y, d.y, o2[4 * q + 1].y);
            o2[4 * q + 2].x = fmaf(w.z, d.x, o2[4 * q + 2].x); o2[4 * q + 2].y = fmaf(w.z, d.y, o2[4 * q + 2].y);
            o2[4 * q + 3].x = fmaf(w.w, d.x, o2[4 * q + 3].x); o2[4 * q + 3].y = fmaf(w.w, d.y, o2[4 * q + 3].y);
          }
        }
        float* __restrict__ op = dx + (size_t)b * Ci * N + k0 + px;
#pragma unroll
        for (int i = 0; i < 2 * T; ++i)
          if (i < Ci) *reinterpret_cast<float2*>(op + (size_t)i * N) = o2[i];
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + stage);
    if (warp == 0) produce(slab + WG2_STAGES);    // refill the stage just released (waits for the other warps)
  }
  if (!has_tile) return;
  // part[(cta * KH + kh)][Co][Ci + 1]
  float* __restrict__ pp = part + ((size_t)blockIdx.x * KH + kh) * Co * (Ci + 1);
#pragma unroll
  for (int r = 0; r < T; ++r) {
#pragma unroll
    for (int c = 0; c < T; ++c) {
      float v = acc[r][c];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0 && to + r < Co && ti + c < Ci) pp[(size_t)(to + r) * (Ci + 1) + ti + c] = v;
    }
    if (bias_tile && (!FULL || ((r >= T / 2) == bias_hi))) {
      float v = accb[r];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0 && to + r < Co) pp[(size_t)(to + r) * (Ci + 1) + Ci] = v;
    }
  }
}

// One place that names every instantiation of the TMA-fed kernel: attr_only sets the shared-memory attribute of all of them
// (once per device), otherwise the one selected by (dgrad, full) is launched.
template <int T, bool DGRAD, bool FULL, typename... Args>
void wg2_launch_one(bool attr_only, dim3 grid, int threads, size_t smem, cudaStream_t st, int& rc, Args... args) {
  auto kern = wgrad2_partial_kernel<T, DGRAD, FULL>;
  if (attr_only) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
      rc = check_launch("cudaFuncSetAttribute(wgrad2)");
    return;
  }
  kern<<<grid, threads, smem, st>>>(args...);
}
template <int T, typename... Args>
void wg2_launch(bool attr_only, bool dgrad, bool full, dim3 grid, int threads, size_t smem, cudaStream_t st, int& rc,
                Args... args) {
  if (attr_only || (dgrad && full)) wg2_launch_one<T, true, true>(attr_only, grid, threads, smem, st, rc, args...);
  if (attr_only || (dgrad && !full)) wg2_launch_one<T, true, false>(attr_only, grid, threads, smem, st, rc, args...);
  if (attr_only || (!dgrad && full)) wg2_launch_one<T, false, true>(attr_only, grid, threads, smem, st, rc, args...);
  if (attr_only || (!dgrad && !full)) wg2_launch_one<T, false, false>(attr_only, grid, threads, smem, st, rc, args...);
}

// ------------------------------------------------------------------------------------------
// Wide-channel weight gradient (20 < max(Co, Ci) <= 64: BASELINE configs[2], width 64).  The T x T-per-warp kernels above
// need Co/T x Ci/T warps per CTA; at width 64 that is 49 tiles, i.e. 7 CTA groups that each re-read the same slabs.  Here a
// CTA owns the WHOLE 64 x 64 output: 4 pixel groups x 64 threads, thread = 8 x 8 register tile (rows og + 8 j, columns
// ig + 8 j: consecutive threads touch consecutive shared-memory rows, whose 272-byte pitch spreads them over all banks), 16
// LDS.128 per 256 FMA, slabs of 64 pixels through a 2-stage cp.async ring, two CTAs per SM.  The pixel groups are summed
// through shared memory at the end; per-CTA partials go through partial_reduce_kernel like the other forms.
// ------------------------------------------------------------------------------------------
constexpr int WW_KT = 64;          // pixels per slab
constexpr int WW_P = WW_KT + 4;    // row pitch (floats)
constexpr int WW_C = 64;           // padded channels
constexpr int WW_THREADS = 256;

__global__ void __launch_bounds__(WW_THREADS, 2)
wgrad_wide_kernel(const float* __restrict__ ds, const float* __restrict__ a, float* __restrict__ part, int Co, int Ci,
                  long N, int slabs_per_sample, long total_slabs, long slabs_per_cta) {
  extern __shared__ __align__(16) float sm[];        // 2 stages x [2 * WW_C][WW_P]  (ds rows, then a rows)
  constexpr int STAGE = 2 * WW_C * WW_P;
  const int tid = threadIdx.x;
  const int kg = tid >> 6, og = (tid >> 3) & 7, ig = tid & 7;
  long s_begin = (long)blockIdx.x * slabs_per_cta;
  long s_end = s_begin + slabs_per_cta;
  if (s_end > total_slabs) s_end = total_slabs;
  // rows beyond Co / Ci are never written by the copies: zero them once
  for (int i = tid; i < 2 * STAGE; i += WW_THREADS) sm[i] = 0.f;
  __syncthreads();

  float acc[8][8];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
  float accb = 0.f;                                  // bias: thread = (row tid / 4, 16-pixel chunk tid % 4)

  auto issue = [&](long slab, int stage) {
    float* dst = sm + (size_t)stage * STAGE;
    const long b = slab / slabs_per_sample;
    const long k0 = (slab - b * slabs_per_sample) * WW_KT;
    const float* dsb = ds + (size_t)b * Co * N;
    const float* ab = a + (size_t)b * Ci * N;
    for (int idx = tid; idx < 2 * WW_C * (WW_KT / 4); idx += WW_THREADS) {
      const int c = idx / (WW_KT / 4), q = idx - c * (WW_KT / 4);
      const bool is_ds = c < WW_C;
      const int ch = is_ds ? c : c - WW_C;
      if (ch >= (is_ds ? Co : Ci)) continue;
      const long k = k0 + 4 * q;
      const float* src = (is_ds ? dsb : ab) + (size_t)ch * N + k;
      const long left = (N - k) * 4;
      const int nb = left >= 16 ? 16 : (left > 0 ? (int)left : 0);
      cp_async16(dst + c * WW_P + 4 * q, nb > 0 ? src : ds, nb);
    }
    cp_async_commit();
  };

  if (s_begin < s_end) issue(s_begin, 0);
  for (long slab = s_begin; slab < s_end; ++slab) {
    const int stage = (int)((slab - s_begin) & 1);
    if (slab + 1 < s_end) {
      issue(slab + 1, stage ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* ds_s = sm + (size_t)stage * STAGE;
    const float* a_s = ds_s + WW_C * WW_P;
    {
      const float4* br = reinterpret_cast<const float4*>(ds_s + (tid >> 2) * WW_P + (tid & 3) * 16);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = br[q];
        accb += (v.x + v.y) + (v.z + v.w);
      }
    }
#pragma unroll
    for (int st = 0; st < WW_KT / 16; ++st) {
      const int px = kg * (WW_KT / 4) + st * 4;
      float4 dv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) dv[j] = *reinterpret_cast<const float4*>(ds_s + (og + 8 * j) * WW_P + px);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 av = *reinterpret_cast<const float4*>(a_s + (ig + 8 * c) * WW_P + px);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          acc[r][c] = fmaf(dv[r].x, av.x, acc[r][c]);
          acc[r][c] = fmaf(dv[r].y, av.y, acc[r][c]);
          acc[r][c] = fmaf(dv[r].z, av.z, acc[r][c]);
          acc[r][c] = fmaf(dv[r].w, av.w, acc[r][c]);
        }
      }
    }
    __syncthreads();  // the stage is refilled by the next iteration's issue()
  }
  // combine the 4 pixel groups: red[kg][o][i] (64 KB of the 68 KB ring), bias partials behind it
  float* red = sm;
  float* redb = sm + 4 * WW_C * WW_C;                 // [64 rows][4 chunks]
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int c = 0; c < 8; ++c) red[(kg * WW_C + og + 8 * r) * WW_C + ig + 8 * c] = acc[r][c];
  redb[tid] = accb;
  __syncthreads();
  float* __restrict__ pp = part + (size_t)blockIdx.x * Co * (Ci + 1);
  for (int e = tid; e < WW_C * WW_C; e += WW_THREADS) {
    const int o = e / WW_C, i = e - o * WW_C;
    if (o < Co && i < Ci)
      pp[(size_t)o * (Ci + 1) + i] = (red[e] + red[WW_C * WW_C + e]) + (red[2 * WW_C * WW_C + e] + red[3 * WW_C * WW_C + e]);
  }
  if (tid < Co) pp[(size_t)tid * (Ci + 1) + Ci] = (redb[4 * tid] + redb[4 * tid + 1]) + (redb[4 * tid + 2] + redb[4 * tid + 3]);
}

constexpr int WG_CTAS = 148 * 2;  // persistent grid: 2 resident CTAs per SM (register-limited)

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" int fno_pointwise_fwd(const float* in, const float* W, const float* bias, float* out, int B, int Co,
                                 int Ci, long N, int transpose, fno_stream_t stream) {
  if (!in || !W || !out || B <= 0 || Co <= 0 || Ci <= 0 || N <= 0) {
    set_error("fno_pointwise_fwd: bad argument");
    return FNO_E_ARG;
  }
  if (B > 65535) { set_error("fno_pointwise_fwd: batch %d > 65535", B); return FNO_E_ARG; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int Cout = transpose ? Ci : Co;
  const int Cin = transpose ? Co : Ci;
  // wide layers (width 33..64, cfg 3): the product and its data gradient run on tcgen05 (pointwise_tc.cu)
  if (pointwise_tc_supported(Cin, Cout)) return launch_pointwise_tc(in, W, bias, out, B, Co, Ci, N, transpose, st);
  const bool vec2 = (N % 2 == 0) && ((reinterpret_cast<size_t>(in) | reinterpret_cast<size_t>(out)) % 8 == 0);
  if (vec2 && Cin <= 256) {
    if (Cout % 20 == 0) return launch_pw2<20>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    if (Cout % 16 == 0) return launch_pw2<16>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    if (Cout % 8 == 0) return launch_pw2<8>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    return launch_pw2<4>(in, W, bias, out, B, Co, Ci, N, transpose, st);
  }
  const bool vec4 = (N % 4 == 0) && ((reinterpret_cast<size_t>(in) | reinterpret_cast<size_t>(out)) % 16 == 0);
  if (vec4) {
    if (Cout % 20 == 0) return launch_pw<20, 4>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    if (Cout % 16 == 0) return launch_pw<16, 4>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    if (Cout % 8 == 0) return launch_pw<8, 4>(in, W, bias, out, B, Co, Ci, N, transpose, st);
    return launch_pw<4, 4>(in, W, bias, out, B, Co, Ci, N, transpose, st);
  }
  if (Cout % 20 == 0) return launch_pw<20, 1>(in, W, bias, out, B, Co, Ci, N, transpose, st);
  if (Cout % 16 == 0) return launch_pw<16, 1>(in, W, bias, out, B, Co, Ci, N, transpose, st);
  if (Cout % 8 == 0) return launch_pw<8, 1>(in, W, bias, out, B, Co, Ci, N, transpose, st);
  return launch_pw<4, 1>(in, W, bias, out, B, Co, Ci, N, transpose, st);
}

extern "C" size_t fno_pointwise_wgrad_workspace_bytes(int B, int Co, int Ci, long N) {
  if (B <= 0 || Co <= 0 || Ci <= 0 || N <= 0) return 0;
  return sizeof(float) * (size_t)WG_CTAS * Co * (Ci + 1);
}

// Wm / dx != nullptr: also write the data gradient dx = W^T ds when the TMA-fed kernel can carry it (returns 1 in
// *fused then); otherwise only the weight gradient is computed and the caller runs the product separately.
static int pointwise_wgrad_impl(const float* ds, const float* a, float* gW, float* gb, void* work, int B, int Co, int Ci,
                                long N, const float* Wm, float* dx, int* fused, fno_stream_t stream) {
  if (fused) *fused = 0;
  if (!ds || !a || !work || B <= 0 || Co <= 0 || Ci <= 0 || N <= 0) {
    set_error("fno_pointwise_wgrad: bad argument");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  constexpr int T = WG_T;
  const int tiles_o = (Co + T - 1) / T, tiles_i = (Ci + T - 1) / T;
  const int ntiles = tiles_o * tiles_i;
  const int warps = ntiles < WG_MAXW ? ntiles : WG_MAXW;
  const int ygroups = (ntiles + warps - 1) / warps;
  const size_t smem = sizeof(float) * 2ul * (size_t)(Co + Ci) * KT;
  if (smem > 200 * 1024) { set_error("fno_pointwise_wgrad: width %d too large", Co + Ci); return FNO_E_ARG; }
  static PerDeviceOnce attr_done;
  if (attr_done.need()) {
    if (cudaFuncSetAttribute(wgrad_partial_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) !=
        cudaSuccess)
      return check_launch("cudaFuncSetAttribute(wgrad)");
    attr_done.mark();
  }
  const int slabs_per_sample = (int)((N + KT - 1) / KT);
  const long total_slabs = (long)B * slabs_per_sample;
  long ctas = total_slabs < WG_CTAS ? total_slabs : WG_CTAS;
  const long spc = (total_slabs + ctas - 1) / ctas;
  ctas = (total_slabs + spc - 1) / spc;
  const int aligned = (N % 4 == 0) && ((reinterpret_cast<size_t>(ds) | reinterpret_cast<size_t>(a)) % 16 == 0);
  float* part = static_cast<float*>(work);
  int nparts = 0;
  // v2 (TMA-fed): persistent CTAs, one per SM, each over a contiguous range of 512-pixel slabs; the operand feed is two 2-D
  // tensor-map copies per slab (box {512 pixels as 256 8-byte elements, C planes} of ds and of a)
  const size_t smem2 = sizeof(float) * (size_t)WG2_STAGES * (Co + Ci) * WG2_KT + 2 * WG2_STAGES * sizeof(unsigned long long);
  CUtensorMap mds, ma;
  memset(&mds, 0, sizeof(mds)); memset(&ma, 0, sizeof(ma));
  const auto l2 = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
  if (aligned && smem2 <= 200 * 1024 && ntiles <= WG2_MAXW && N < (1L << 31) && (long)B * (Co > Ci ? Co : Ci) < (1L << 31) &&
      make_plane_map(&mds, ds, (unsigned long long)N, (unsigned long long)B * Co, WG2_KT, Co, 8, l2) &&
      make_plane_map(&ma, a, (unsigned long long)N, (unsigned long long)B * Ci, WG2_KT, Ci, 8, l2)) {
    const int KH = (2 * ntiles <= WG2_MAXW) ? 2 : 1;       // pixel halves per tile
    const int warps2 = ntiles * KH;
    const int sps2 = (int)((N + WG2_KT - 1) / WG2_KT);
    const long total2s = (long)B * sps2;
    long ctas2 = total2s < 148 ? total2s : 148;
    const long spc2 = (total2s + ctas2 - 1) / ctas2;
    ctas2 = (total2s + spc2 - 1) / spc2;
    // the data gradient rides along when the 8 consumer warps cover a slab two pixels per thread
    const size_t smem2d = smem2 + sizeof(float) * (size_t)Co * 2 * T;
    const bool dgrad = Wm != nullptr && dx != nullptr && warps2 == WG2_MAXW && Co <= 2 * T && Ci <= 2 * T &&
                       smem2d <= 200 * 1024 && (reinterpret_cast<size_t>(dx) % 8) == 0;
    const bool full = (T % 2 == 0) && tiles_i == 2 && Ci == 2 * T && Co % T == 0;
    static PerDeviceOnce attr2_done;
    if (attr2_done.need()) {
      int rca = FNO_OK;
      wg2_launch<T>(true, true, true, dim3(1), 0, 0, st, rca, part, Co, Ci, N, sps2, total2s, spc2, tiles_i, ntiles,
                    warps2, KH, Wm, dx, mds, ma);
      if (rca != FNO_OK) return rca;
      attr2_done.mark();
    }
    int rcl = FNO_OK;
    wg2_launch<T>(false, dgrad, full, dim3((unsigned)ctas2, 1), 32 * warps2, dgrad ? smem2d : smem2, st, rcl, part, Co,
                  Ci, N, sps2, total2s, spc2, tiles_i, ntiles, warps2, KH, dgrad ? Wm : nullptr, dgrad ? dx : nullptr, mds, ma);
    if (rcl != FNO_OK) return rcl;
    if (dgrad && fused) *fused = 1;
    count_launch();
    int rc2 = check_launch("wgrad2_partial_kernel");
    if (rc2 != FNO_OK) return rc2;
    nparts = (int)(ctas2 * KH);
  } else if (aligned && pointwise_tc_supported(Ci, Co)) {
    // wide channels on tcgen05: [ds ; a] [a ; 1]^T per 64-pixel slab, accumulator in TMEM (pointwise_tc.cu)
    int rct = launch_wgrad_tc(ds, a, part, B, Co, Ci, N, WG_CTAS, &nparts, st);
    if (rct != FNO_OK) return rct;
  } else if (aligned && ygroups > 1 && Co <= WW_C && Ci <= WW_C) {
    // wide channels: one CTA owns the whole Co x Ci output (wgrad_wide_kernel)
    const size_t smemw = sizeof(float) * 2ul * 2 * WW_C * WW_P;
    static_assert(sizeof(float) * (4ul * WW_C * WW_C + WW_THREADS) <= sizeof(float) * 2ul * 2 * WW_C * WW_P, "reduce buffer fits the ring");
    static PerDeviceOnce attrw_done;
    if (attrw_done.need()) {
      if (cudaFuncSetAttribute(wgrad_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(wgrad_wide)");
      attrw_done.mark();
    }
    const int spsw = (int)((N + WW_KT - 1) / WW_KT);
    const long totalw = (long)B * spsw;
    long ctasw = totalw < WG_CTAS ? totalw : WG_CTAS;
    const long spcw = (totalw + ctasw - 1) / ctasw;
    ctasw = (totalw + spcw - 1) / spcw;
    wgrad_wide_kernel<<<(unsigned)ctasw, WW_THREADS, smemw, st>>>(ds, a, part, Co, Ci, N, spsw, totalw, spcw);
    count_launch();
    int rcw = check_launch("wgrad_wide_kernel");
    if (rcw != FNO_OK) return rcw;
    nparts = (int)ctasw;
  } else {
    const dim3 grid((unsigned)ctas, ygroups);
    wgrad_partial_kernel<T><<<grid, 32 * warps, smem, st>>>(ds, a, part, Co, Ci, N, slabs_per_sample, total_slabs, spc,
                                                          tiles_i, ntiles, aligned);
    count_launch();
    int rc = check_launch("wgrad_partial_kernel");
    if (rc != FNO_OK) return rc;
    nparts = (int)ctas;
  }
  // records [nparts][Co][Ci + 1]: gW in the first Ci columns, gb in the last
  ReduceSegs segs;
  segs.s[0] = {gW, Co * Ci, 0, Ci, Ci + 1};
  segs.s[1] = {gb, Co, Ci, 1, Ci + 1};
  return launch_partial_reduce(part, nparts, Co * (Ci + 1), segs, st);
}

extern "C" int fno_pointwise_wgrad(const float* ds, const float* a, float* gW, float* gb, void* work, int B, int Co,
                                   int Ci, long N, fno_stream_t stream) {
  return pointwise_wgrad_impl(ds, a, gW, gb, work, B, Co, Ci, N, nullptr, nullptr, nullptr, stream);
}

extern "C" int fno_pointwise_bwd(const float* ds, const float* a, const float* W, float* dx, float* gW, float* gb,
                                 void* work, int B, int Co, int Ci, long N, fno_stream_t stream) {
  if (!W || !dx) { set_error("fno_pointwise_bwd: bad argument"); return FNO_E_ARG; }
  int fused = 0;
  int rc = pointwise_wgrad_impl(ds, a, gW, gb, work, B, Co, Ci, N, W, dx, &fused, stream);
  if (rc != FNO_OK || fused) return rc;
  return fno_pointwise_fwd(ds, W, nullptr, dx, B, Co, Ci, N, /*transpose=*/1, stream);
}
