// Projection-head backward for WIDE trunks (24 <= C <= 64: BASELINE configs[2], width 64) on the 5th-generation tensor
// cores.  Autograd of  out = (W2 gelu(W1 h + b1) + b2) * std + mean  (fno/fno.py:180-187); the hidden layer is recomputed.
//
// head_bwd_tc.cu keeps all three contractions of a tile in one CTA, which at C = 64 needs ~390 KB of staged operands.
// Here the work is cut in two launches with the hidden-layer gradient dpre [B, 128, plane] passing through HBM:
//
//   X  head_bwd_wide_kernel (this file), per 128 positions of the padded plane (thread = position = TMEM lane):
//        (a) pre[px, j]  = sum_c h[px, c] W1[j, c]        A = h hi / lo written to TENSOR MEMORY (lane = px, K along
//                                                         columns: no shared-memory staging), B = W1 in shared memory
//        epilogue: dpre = gelu'(pre + b1) * (W2^T dy),  dy = dout * std (0 in the padding); dpre goes to HBM and, split
//                  hi / lo, back into tensor memory over the pre tile it was read from -- the A operand of (b);
//                  gW2[:, j] += gelu(pre) dy^T through a lane reduce-scatter (31 shuffles per 32 hidden units), gb2
//        (b) dh[px, c]   = sum_j dpre[px, j] W1[j, c]     A = dpre from tensor memory, B = W1^T in shared memory
//      Positions in the padding take part with dy = 0, so dh gets its zero padding from the same stores.
//   Y  wgrad_tc_kernel<128, 32> (pointwise_tc.cu): gW1 | gb1 = [dpre ; h ; 1]-Gram blocks, K = pixels, as for the bypass.
//
// 3xTF32 everywhere (fp32 mode: <= 1e-5); the MMA chains are 24 / 48 instructions long, far below the length at which
// the tensor core's truncating accumulate shows (pointwise_tc.cu).
#include <cstdlib>

#include "common.cuh"
#include "tc_common.cuh"

namespace fno {
namespace {

constexpr int HW_M = 128;                 // positions per tile = TMEM lanes
constexpr int HW_HID = 128;
constexpr int HW_K = 64;                  // padded channels
constexpr int HW_VP = 4;                  // output variables (padded)
constexpr int HW_EPI_WARPS = 16;
constexpr int HW_EPI_THREADS = 32 * HW_EPI_WARPS;
constexpr int HW_THREADS = HW_EPI_THREADS + 32;
constexpr int HW_SBO_A = (HW_K / 4) * 128;            // W1   [j 128][k = c 64]: 2048
constexpr int HW_SBO_B = (HW_HID / 4) * 128;          // W1^T [c 64][k = j 128]: 4096
constexpr int HW_BA_BYTES = (HW_HID / 8) * HW_SBO_A;  // 32 KB
constexpr int HW_BB_BYTES = (HW_K / 8) * HW_SBO_B;    // 32 KB
constexpr int HW_RED_FLOATS = 4 * HW_VP * HW_HID + 4 * HW_VP;
constexpr int HW_SMEM = 2 * HW_BA_BYTES + 2 * HW_BB_BYTES + 4 * (HW_HID * HW_VP + HW_HID + HW_RED_FLOATS) + 4 * 8 + 16;
// tensor-memory columns
constexpr unsigned HW_TM_HHI = 0, HW_TM_HLO = 64, HW_TM_P = 128, HW_TM_DL = 256, HW_TM_DH = 384, HW_TM_COLS = 512;
constexpr int HW_REC = HW_VP * HW_HID + HW_VP;        // per-CTA record: gW2 [4][128] | gb2 [4]

struct HwGeo {
  int R_in, W_in, Wp;
  long npix, plane;
};

// sum over the 32 lanes of x[i] for every i, lane l ends up with the total of x[l] (reduce-scatter butterfly)
__device__ __forceinline__ float lane_reduce_scatter(float (&x)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool upper = (lane & s) != 0;
#pragma unroll
    for (int k = 0; k < s; ++k) {
      const float send = upper ? x[k] : x[k + s];
      const float keep = upper ? x[k + s] : x[k];
      x[k] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return x[0];
}

__global__ void __launch_bounds__(HW_THREADS, 1)
head_bwd_wide_kernel(const float* __restrict__ h, const float* __restrict__ dout, const float* __restrict__ W1,
                     const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ stats,
                     float* __restrict__ dh, float* __restrict__ dpre_g, float* __restrict__ rec, HwGeo g, int C, int V,
                     int tiles_per_sample, int total_tiles, int single) {
  FNO_SPLIT_CONSTS(single);
  extern __shared__ __align__(128) unsigned char hsm[];
  unsigned char* ba_hi = hsm;
  unsigned char* ba_lo = ba_hi + HW_BA_BYTES;
  unsigned char* bb_hi = ba_lo + HW_BA_BYTES;
  unsigned char* bb_lo = bb_hi + HW_BB_BYTES;
  float* W2s = reinterpret_cast<float*>(bb_lo + HW_BB_BYTES);     // [HID][VP]
  float* b1s = W2s + HW_HID * HW_VP;                              // [HID]
  float* red = b1s + HW_HID;                                      // [4 quadrants][VP][HID] | [4][VP]
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(red + HW_RED_FLOATS);
  unsigned long long* h_ready = bars;          // loaders -> MMA: h hi / lo in tensor memory
  unsigned long long* pre_full = bars + 1;     // MMA (a) done
  unsigned long long* dpre_ready = bars + 2;   // epilogue -> MMA: dpre hi / lo in tensor memory
  unsigned long long* dh_full = bars + 3;      // MMA (b) done
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 4);

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    mbar_init(h_ready, HW_EPI_WARPS);
    mbar_init(pre_full, 1);
    mbar_init(dpre_ready, HW_EPI_WARPS);
    mbar_init(dh_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == HW_EPI_WARPS) tmem_alloc(tmem_slot, HW_TM_COLS);
  // constant operands: W1 [j][c] (B of (a)) and W1^T [c][j] (B of (b)), hi / lo, zero padded to 64 channels
  for (int i = tid; i < HW_HID * HW_K; i += HW_THREADS) {
    const int j = i / HW_K, c = i - j * HW_K;
    float hi = 0.f, lo = 0.f;
    if (c < C) split_rm(__ldg(W1 + (size_t)j * C + c), hi, lo, sp_rnd, sp_msk);
    const int oa = (j & 7) * 16 + (j >> 3) * HW_SBO_A + (c >> 2) * 128 + (c & 3) * 4;
    const int ob = (c & 7) * 16 + (c >> 3) * HW_SBO_B + (j >> 2) * 128 + (j & 3) * 4;
    *reinterpret_cast<float*>(ba_hi + oa) = hi;
    *reinterpret_cast<float*>(ba_lo + oa) = lo;
    *reinterpret_cast<float*>(bb_hi + ob) = hi;
    *reinterpret_cast<float*>(bb_lo + ob) = lo;
  }
  for (int i = tid; i < HW_HID * HW_VP; i += HW_THREADS) {
    const int j = i / HW_VP, v = i - j * HW_VP;
    W2s[i] = (v < V) ? __ldg(W2 + (size_t)v * HW_HID + j) : 0.f;
  }
  for (int i = tid; i < HW_HID; i += HW_THREADS) b1s[i] = __ldg(b1 + i);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const int ksteps = (C + 7) / 8;
  const int Pl = (int)g.plane;              // 32-bit element offsets (the launcher checks 128 plane < 2^31)
  const int ntl = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA

  if (warp == HW_EPI_WARPS) {
    // ---- MMA issuer ------------------------------------------------------------------------------------
    constexpr unsigned idesc_a = umma_idesc_tf32(HW_M, HW_HID, 0, 0);
    constexpr unsigned idesc_b = umma_idesc_tf32(HW_M, HW_K, 0, 0);
    const unsigned long long d_a_h = umma_desc(ba_hi, 128, HW_SBO_A), d_a_l = umma_desc(ba_lo, 128, HW_SBO_A);
    const unsigned long long d_b_h = umma_desc(bb_hi, 128, HW_SBO_B), d_b_l = umma_desc(bb_lo, 128, HW_SBO_B);
    for (int it = 0; it < ntl; ++it) {
      const unsigned ph = (unsigned)it & 1u;
      mbar_wait(h_ready, ph);
      tc_fence_after();
      __syncwarp();
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < HW_K / 8; ++ks)
          if (ks < ksteps && (pass == 2 || !single))
            tc_mma_tf32_ts_elect(tmem_base + HW_TM_P, tmem_base + (pass == 0 ? HW_TM_HLO : HW_TM_HHI) + (unsigned)(8 * ks),
                                 (pass == 1 ? d_a_l : d_a_h) + (unsigned long long)(ks * (256 >> 4)), idesc_a,
                                 single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      tc_commit_elect(pre_full);
      mbar_wait(dpre_ready, ph);
      tc_fence_after();
      __syncwarp();
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int ks = 0; ks < HW_HID / 8; ++ks)
          if (pass == 2 || !single)
            tc_mma_tf32_ts_elect(tmem_base + HW_TM_DH, tmem_base + (pass == 0 ? HW_TM_DL : HW_TM_P) + (unsigned)(8 * ks),
                                 (pass == 1 ? d_b_l : d_b_h) + (unsigned long long)(ks * (256 >> 4)), idesc_b,
                                 single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      tc_commit_elect(dh_full);
    }
  } else {
    // ---- loader / epilogue warps: warp <-> (TMEM lane quadrant, quarter of the columns) -------------------
    const int quad = warp & 3, colq = warp >> 2;
    const int m = quad * 32 + lane;                 // position of the tile owned by this thread (= its TMEM lane)
    const unsigned tlane = tmem_base + ((unsigned)(quad * 32) << 16);
    float raw[16];                                  // channels [16 colq, 16 colq + 16) of position m, next tile
    float accw2[HW_VP], accb2[HW_VP];
#pragma unroll
    for (int v = 0; v < HW_VP; ++v) { accw2[v] = 0.f; accb2[v] = 0.f; }
    auto load_raw = [&](int it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const bool inr = it < ntl;
      const int b = inr ? tile / tiles_per_sample : 0;
      const long q = inr ? (long)(tile - b * tiles_per_sample) * HW_M + m : 0;
      const bool inplane = inr && q < g.plane;
      const float* hp = h + ((size_t)b * C + 16 * colq) * g.plane + (inplane ? q : 0);   // running pointer: 2 adds per access
      const int cmax = inplane ? C - 16 * colq : 0;
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        raw[e] = (e < cmax) ? __ldg(hp) : 0.f;
        hp += Pl;
      }
    };
    load_raw(0);
    for (int it = 0; it < ntl; ++it) {
      const unsigned ph = (unsigned)it & 1u;
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int b = tile / tiles_per_sample;
      const long q = (long)(tile - b * tiles_per_sample) * HW_M + m;
      const bool inplane = q < g.plane;
      const int r = (int)(q / g.Wp), w = (int)(q - (long)r * g.Wp);
      const bool valid = inplane && r < g.R_in && w < g.W_in;
      // -- h of this tile -> tensor memory (hi / lo), then the next tile's loads and this tile's dy go in flight
      if (16 * colq < 8 * ksteps) {
        float hi[16], lo[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) split_rm(raw[e], hi[e], lo[e], sp_rnd, sp_msk);
        tmem_st16(tlane + HW_TM_HHI + (unsigned)(16 * colq), hi);
        if (!single) tmem_st16(tlane + HW_TM_HLO + (unsigned)(16 * colq), lo);
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(h_ready);
      load_raw(it + 1);
      float dy[HW_VP];
      {
        const float* __restrict__ op = dout + ((size_t)b * g.npix + (valid ? (long)r * g.W_in + w : 0)) * V;
        const float* __restrict__ sd = stats + (size_t)b * 2 * V + V;
#pragma unroll
        for (int v = 0; v < HW_VP; ++v) dy[v] = (valid && v < V) ? __ldg(op + v) * __ldg(sd + v) : 0.f;
      }
      if (colq == 0) {
#pragma unroll
        for (int v = 0; v < HW_VP; ++v) accb2[v] += dy[v];
      }

      // -- epilogue of (a): dpre and gelu for hidden units [32 colq, 32 colq + 32) of position m
      mbar_wait(pre_full, ph);
      tc_fence_after();
      float act[32];
      float* dg = dpre_g + ((size_t)b * HW_HID + 32 * colq) * g.plane + q;     // running pointer over the hidden units
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[16], hi[16], lo[16];
        const unsigned col = HW_TM_P + (unsigned)(32 * colq + 16 * half);
        tmem_ld16(tlane + col, v);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const int j = 32 * colq + 16 * half + e;
          float gl, gp;
          gelu_fast_both(v[e] + b1s[j], gl, gp);
          const float4 w2 = *reinterpret_cast<const float4*>(W2s + j * HW_VP);
          const float dact = fmaf(w2.x, dy[0], fmaf(w2.y, dy[1], fmaf(w2.z, dy[2], w2.w * dy[3])));
          const float dpre = dact * gp;
          act[16 * half + e] = gl;
          if (inplane) *dg = dpre;
          dg += Pl;
          split_rm(dpre, hi[e], lo[e], sp_rnd, sp_msk);
        }
        tmem_st16(tlane + col, hi);
        if (!single) tmem_st16(tlane + HW_TM_DL + (unsigned)(32 * colq + 16 * half), lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dpre_ready);
      // -- gW2[:, j] += sum over this warp's 32 positions of gelu(pre) * dy  (runs under the MMAs of (b))
#pragma unroll
      for (int v = 0; v < HW_VP; ++v) {
        if (v < V) {
          float x[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) x[i] = act[i] * dy[v];
          accw2[v] += lane_reduce_scatter(x, lane);
        }
      }
      // -- epilogue of (b): dh for channels [16 colq, 16 colq + 16), zero in the padding
      mbar_wait(dh_full, ph);
      tc_fence_after();
      {
        float v[16];
        tmem_ld16(tlane + HW_TM_DH + (unsigned)(16 * colq), v);
        if (inplane) {
          float* dp = dh + ((size_t)b * C + 16 * colq) * g.plane + q;
          const int nc = C - 16 * colq;
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            if (e < nc) *dp = valid ? v[e] : 0.f;
            dp += Pl;
          }
        }
      }
      tc_fence_before();
    }
    // ---- per-CTA record: gW2 [VP][HID] (lane l of warp (quad, colq) holds hidden unit 32 colq + l), gb2 [VP] ----
#pragma unroll
    for (int v = 0; v < HW_VP; ++v) red[(quad * HW_VP + v) * HW_HID + 32 * colq + lane] = accw2[v];
    if (colq == 0) {
#pragma unroll
      for (int v = 0; v < HW_VP; ++v) {
        float t = accb2[v];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (lane == 0) red[4 * HW_VP * HW_HID + quad * HW_VP + v] = t;
      }
    }
    named_bar_sync(1, HW_EPI_THREADS);
    float* __restrict__ myrec = rec + (size_t)blockIdx.x * HW_REC;
    for (int i = tid; i < HW_VP * HW_HID; i += HW_EPI_THREADS)
      myrec[i] = (red[i] + red[HW_VP * HW_HID + i]) + (red[2 * HW_VP * HW_HID + i] + red[3 * HW_VP * HW_HID + i]);
    if (tid < HW_VP) {
      const float* rb = red + 4 * HW_VP * HW_HID;
      myrec[HW_VP * HW_HID + tid] = (rb[tid] + rb[HW_VP + tid]) + (rb[2 * HW_VP + tid] + rb[3 * HW_VP + tid]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == HW_EPI_WARPS) tmem_dealloc(tmem_base, HW_TM_COLS);
}

constexpr int HW_WG_PARTS = 148;

// ------------------------------------------------------------------------------------------
// forward for wide trunks (32 < C <= 64):  out = (W2 gelu(W1 h + b1) + b2) * std + mean  per valid pixel.
// The same (a) GEMM with h through tensor memory; the pre-activation tile is double-buffered so the MMAs of tile i+1
// run under the GELU epilogue of tile i; the four column quarters of a pixel meet in shared memory (as in head_tc.cu).
// ------------------------------------------------------------------------------------------
constexpr int HF_SMEM = 2 * HW_BA_BYTES + 4 * (HW_HID * HW_VP + HW_HID + 2 * 4 * HW_M * HW_VP) + 5 * 8 + 16;
constexpr unsigned HF_TM_P = 128;         // 2 x 128 columns

struct HfGeo {
  int W_in, Wp;
  long npix, plane;
};

__global__ void __launch_bounds__(HW_THREADS, 1)
head_fwd_wide_kernel(const float* __restrict__ h, const float* __restrict__ W1, const float* __restrict__ b1,
                     const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ stats,
                     float* __restrict__ out, HfGeo g, int C, int V, int tiles_per_sample, int total_tiles, int single) {
  FNO_SPLIT_CONSTS(single);
  extern __shared__ __align__(128) unsigned char hsm[];
  unsigned char* ba_hi = hsm;
  unsigned char* ba_lo = ba_hi + HW_BA_BYTES;
  float* W2s = reinterpret_cast<float*>(ba_lo + HW_BA_BYTES);     // [HID][VP]
  float* b1s = W2s + HW_HID * HW_VP;                              // [HID]
  float* ox = b1s + HW_HID;                                       // [2 tiles][4 quarters][M][VP]
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(ox + 2 * 4 * HW_M * HW_VP);
  unsigned long long* h_ready = bars;          // loaders -> MMA
  unsigned long long* pre_full = bars + 1;     // [2] MMA done
  unsigned long long* d_free = bars + 3;       // [2] epilogue -> MMA: the pre-activation tile may be overwritten
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 5);

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    mbar_init(h_ready, HW_EPI_WARPS);
    for (int s = 0; s < 2; ++s) {
      mbar_init(pre_full + s, 1);
      mbar_init(d_free + s, HW_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == HW_EPI_WARPS) tmem_alloc(tmem_slot, 512);
  for (int i = tid; i < HW_HID * HW_K; i += HW_THREADS) {
    const int j = i / HW_K, c = i - j * HW_K;
    float hi = 0.f, lo = 0.f;
    if (c < C) split_rm(__ldg(W1 + (size_t)j * C + c), hi, lo, sp_rnd, sp_msk);
    const int oa = (j & 7) * 16 + (j >> 3) * HW_SBO_A + (c >> 2) * 128 + (c & 3) * 4;
    *reinterpret_cast<float*>(ba_hi + oa) = hi;
    *reinterpret_cast<float*>(ba_lo + oa) = lo;
  }
  for (int i = tid; i < HW_HID * HW_VP; i += HW_THREADS) {
    const int j = i / HW_VP, v = i - j * HW_VP;
    W2s[i] = (v < V) ? __ldg(W2 + (size_t)v * HW_HID + j) : 0.f;
  }
  for (int i = tid; i < HW_HID; i += HW_THREADS) b1s[i] = __ldg(b1 + i);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const int ksteps = (C + 7) / 8;
  const int Pl = (int)g.plane;
  const int ntl = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == HW_EPI_WARPS) {
    constexpr unsigned idesc_a = umma_idesc_tf32(HW_M, HW_HID, 0, 0);
    const unsigned long long d_a_h = umma_desc(ba_hi, 128, HW_SBO_A), d_a_l = umma_desc(ba_lo, 128, HW_SBO_A);
    for (int it = 0; it < ntl; ++it) {
      const int st = it & 1;
      mbar_wait(h_ready, (unsigned)it & 1u);
      mbar_wait(d_free + st, (((unsigned)it >> 1) & 1u) ^ 1u);
      tc_fence_after();
      __syncwarp();
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < HW_K / 8; ++ks)
          if (ks < ksteps && (pass == 2 || !single))
            tc_mma_tf32_ts_elect(tmem_base + HF_TM_P + (unsigned)(st * HW_HID),
                                 tmem_base + (pass == 0 ? HW_TM_HLO : HW_TM_HHI) + (unsigned)(8 * ks),
                                 (pass == 1 ? d_a_l : d_a_h) + (unsigned long long)(ks * (256 >> 4)), idesc_a,
                                 single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      tc_commit_elect(pre_full + st);
    }
  } else {
    const int quad = warp & 3, colq = warp >> 2;
    const int m = quad * 32 + lane;
    const unsigned tlane = tmem_base + ((unsigned)(quad * 32) << 16);
    float raw[16];
    auto load_raw = [&](int it) {                   // channels [16 colq, +16) of pixel m of tile `it`
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const bool inr = it < ntl;
      const int b = inr ? tile / tiles_per_sample : 0;
      const long p = inr ? (long)(tile - b * tiles_per_sample) * HW_M + m : 0;
      const bool valid = inr && p < g.npix;
      const long r = valid ? p / g.W_in : 0;
      const float* hp = h + ((size_t)b * C + 16 * colq) * g.plane + r * g.Wp + (valid ? p - r * g.W_in : 0);
      const int cmax = valid ? C - 16 * colq : 0;
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        raw[e] = (e < cmax) ? __ldg(hp) : 0.f;
        hp += Pl;
      }
    };
    auto stage = [&]() {                            // raw -> tensor memory hi / lo, hand over to the MMA warp
      if (16 * colq < 8 * ksteps) {
        float hi[16], lo[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) split_rm(raw[e], hi[e], lo[e], sp_rnd, sp_msk);
        tmem_st16(tlane + HW_TM_HHI + (unsigned)(16 * colq), hi);
        if (!single) tmem_st16(tlane + HW_TM_HLO + (unsigned)(16 * colq), lo);
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(h_ready);
    };
    load_raw(0);
    stage();
    load_raw(1);
    for (int it = 0; it < ntl; ++it) {
      const int st = it & 1;
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int b = tile / tiles_per_sample;
      const long p0 = (long)(tile - b * tiles_per_sample) * HW_M;
      mbar_wait(pre_full + st, ((unsigned)it >> 1) & 1u);        // (a) of tile it done: h in tensor memory is free
      tc_fence_after();
      if (it + 1 < ntl) stage();                                 // tile it+1's MMAs run under this epilogue
      load_raw(it + 2);
      float o[HW_VP];
#pragma unroll
      for (int v = 0; v < HW_VP; ++v) o[v] = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[16];
        tmem_ld16(tlane + HF_TM_P + (unsigned)(st * HW_HID + 32 * colq + 16 * half), v);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const int j = 32 * colq + 16 * half + e;
          const float gl = gelu_fast(v[e] + b1s[j]);
          const float4 w2 = *reinterpret_cast<const float4*>(W2s + j * HW_VP);
          o[0] = fmaf(w2.x, gl, o[0]); o[1] = fmaf(w2.y, gl, o[1]);
          o[2] = fmaf(w2.z, gl, o[2]); o[3] = fmaf(w2.w, gl, o[3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(d_free + st);
      float* oxb = ox + (size_t)st * 4 * HW_M * HW_VP;
      *reinterpret_cast<float4*>(oxb + (colq * HW_M + m) * HW_VP) = make_float4(o[0], o[1], o[2], o[3]);
      named_bar_sync(1, HW_EPI_THREADS);
      if (colq == (it & 3)) {
        float4 t = *reinterpret_cast<const float4*>(oxb + m * HW_VP);
#pragma unroll
        for (int qq = 1; qq < 4; ++qq) {
          const float4 u = *reinterpret_cast<const float4*>(oxb + (qq * HW_M + m) * HW_VP);
          t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
        }
        const long p = p0 + m;
        if (p < g.npix) {
          const float of[4] = {t.x, t.y, t.z, t.w};
          const float* __restrict__ mean = stats + (size_t)b * 2 * V;
          const float* __restrict__ sd = mean + V;
          float* __restrict__ op = out + ((size_t)b * g.npix + p) * V;
#pragma unroll
          for (int v = 0; v < HW_VP; ++v)
            if (v < V) op[v] = fmaf(of[v] + __ldg(b2 + v), __ldg(sd + v), __ldg(mean + v));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == HW_EPI_WARPS) tmem_dealloc(tmem_base, 512);
}

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" int fno_head_bwd_wide_supported(int R_out, int Wp, int C, int HID, int V) {
  static const bool off = [] { const char* e = std::getenv("FNO_HEAD_WIDE_TC"); return e != nullptr && e[0] == '0'; }();
  return (!off && HID == HW_HID && C > 23 && C <= HW_K && V >= 1 && V <= HW_VP && R_out > 0 && Wp > 0 &&
          ((long)R_out * Wp) % 4 == 0) ? 1 : 0;
}

extern "C" size_t fno_head_bwd_wide_workspace_bytes(int B, int R_out, int Wp, int C, int V) {
  if (B <= 0 || R_out <= 0 || Wp <= 0 || C <= 0 || V <= 0) return 0;
  const size_t plane = (size_t)R_out * Wp;
  return sizeof(float) * ((size_t)B * HW_HID * plane + (size_t)HW_WG_PARTS * HW_HID * (C + 1) + (size_t)148 * HW_REC);
}

extern "C" int fno_head_bwd_wide_tc(const float* h, const float* dout, const float* W1, const float* b1, const float* W2,
                                    const float* stats, float* dh, float* gW1, float* gb1, float* gW2, float* gb2, void* work,
                                    int B, int R_in, int W_in, int R_out, int Wp, int C, int HID, int V, fno_stream_t stream) {
  if (!h || !dout || !W1 || !b1 || !W2 || !stats || !dh || !gW1 || !gb1 || !gW2 || !gb2 || !work || B <= 0 || R_in <= 0 ||
      W_in <= 0 || R_out < R_in || Wp < W_in) {
    set_error("fno_head_bwd_wide_tc: bad argument");
    return FNO_E_ARG;
  }
  if (!fno_head_bwd_wide_supported(R_out, Wp, C, HID, V)) {
    set_error("fno_head_bwd_wide_tc: supports hidden width 128, 24 <= C <= %d, V <= %d, padded plane %% 4 == 0 (got %d, %d, %d, %ld)",
              HW_K, HW_VP, HID, C, V, (long)R_out * Wp);
    return FNO_E_ARG;
  }
  if (((reinterpret_cast<size_t>(h) | reinterpret_cast<size_t>(work)) & 15u) != 0) {
    set_error("fno_head_bwd_wide_tc: h and work must be 16-byte aligned");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HwGeo g;
  g.R_in = R_in; g.W_in = W_in; g.Wp = Wp;
  g.npix = (long)R_in * W_in;
  g.plane = (long)R_out * Wp;
  const long tps = (g.plane + HW_M - 1) / HW_M;
  const long total = tps * B;
  if (total > 0x7fffffffL || g.plane > 0x7fffffffL / 128) { set_error("fno_head_bwd_wide_tc: too many tiles / plane too large"); return FNO_E_ARG; }
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(head_bwd_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HW_SMEM) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_bwd_wide)");
    done.mark();
  }
  float* dpre = static_cast<float*>(work);
  float* part = dpre + (size_t)B * HW_HID * g.plane;
  float* rec = part + (size_t)HW_WG_PARTS * HW_HID * (C + 1);
  const int ctas = (int)(total < 148 ? total : 148);
  head_bwd_wide_kernel<<<ctas, HW_THREADS, HW_SMEM, st>>>(h, dout, W1, b1, W2, stats, dh, dpre, rec, g, C, V, (int)tps,
                                                          (int)total, g_math_mode.load());
  count_launch();
  int rc = check_launch("head_bwd_wide_kernel");
  if (rc != FNO_OK) return rc;
  ReduceSegs segs2;                              // gW2 [V][128] | gb2 [V]
  segs2.s[0] = {gW2, V * HW_HID, 0};
  segs2.s[1] = {gb2, V, HW_VP * HW_HID};
  rc = launch_partial_reduce(rec, ctas, HW_REC, segs2, st);
  if (rc != FNO_OK) return rc;
  // gW1 [128][C] | gb1 [128] = sum over all positions of dpre (x) [h ; 1]  (dpre is zero in the padding)
  int nparts = 0;
  rc = launch_wgrad_tc_rows128(dpre, h, part, B, HW_HID, C, g.plane, HW_WG_PARTS, &nparts, st);
  if (rc != FNO_OK) return rc;
  ReduceSegs segs1;                              // records [nparts][128][C + 1]
  segs1.s[0] = {gW1, HW_HID * C, 0, C, C + 1};
  segs1.s[1] = {gb1, HW_HID, C, 1, C + 1};
  return launch_partial_reduce(part, nparts, HW_HID * (C + 1), segs1, st);
}

extern "C" int fno_head_fwd_wide_tc(const float* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                    const float* stats, float* out, int B, int R_in, int W_in, int R_out, int Wp, int C,
                                    int HID, int V, fno_stream_t stream) {
  if (!h || !W1 || !b1 || !W2 || !b2 || !stats || !out || B <= 0 || R_in <= 0 || W_in <= 0 || R_out < R_in || Wp < W_in) {
    set_error("fno_head_fwd_wide_tc: bad argument");
    return FNO_E_ARG;
  }
  if (HID != HW_HID || C < 1 || C > HW_K || V < 1 || V > HW_VP) {
    set_error("fno_head_fwd_wide_tc: supports hidden width 128, C <= %d, V <= %d (got %d, %d, %d)", HW_K, HW_VP, HID, C, V);
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HfGeo g;
  g.W_in = W_in; g.Wp = Wp;
  g.npix = (long)R_in * W_in;
  g.plane = (long)R_out * Wp;
  const long tps = (g.npix + HW_M - 1) / HW_M;
  const long total = tps * B;
  if (total > 0x7fffffffL || g.plane > 0x7fffffffL / 128) { set_error("fno_head_fwd_wide_tc: too many tiles / plane too large"); return FNO_E_ARG; }
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(head_fwd_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HF_SMEM) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_fwd_wide)");
    done.mark();
  }
  const int ctas = (int)(total < 148 ? total : 148);
  head_fwd_wide_kernel<<<ctas, HW_THREADS, HF_SMEM, st>>>(h, W1, b1, W2, b2, stats, out, g, C, V, (int)tps, (int)total,
                                                          g_math_mode.load());
  count_launch();
  return check_launch("head_fwd_wide_kernel");
}
