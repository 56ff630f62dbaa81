// Projection head on the 5th-generation tensor cores (tcgen05 + TMEM), fp32-accurate through a
// 3xTF32 split.
//
// The head (fno/fno.py:180-187) is the one genuinely dense contraction of the width-20 model: per
// pixel  pre[128] = W1[128 x C] h[C] + b1,  out[V] = W2 gelu(pre) + b2  -- 2 816 FMA per pixel forward,
// ~8 300 backward, half of all FMAs of a training step, and the FP32 path is bound by instruction
// issue (DESIGN.md section 5).  Here the C -> 128 product runs as  D[128 pixels x 128 hidden] =
// A[128 x K] B[K x 128]  with tcgen05.mma.kind::tf32 (b1 included as a ones column of A), accumulators in
// TMEM, and the CUDA cores keep only the element-wise part (exact-erf GELU, the 128 -> V product).
//
// fp32 mode (<= 1e-5 relative, BASELINE north_star) rules out single-pass TF32 (6e-4): every operand
// is split x = hi + lo, hi = rna_tf32(x), and three MMAs accumulate lo*hi + hi*lo + hi*hi into the
// same TMEM tile (the dropped lo*lo term is 2^-22 relative).
//
// Operand staging (no-swizzle canonical layout, 8 x 16-byte core matrices, both operands K-major --
// tools/ubench/umma_probe.cu verified this layout on the hardware and found that kind::tf32 with an
// MN-major operand returns zeros, so the channel-first activation is transposed on the way in):
// thread = pixel loads its channels (coalesced across the warp: 32 consecutive pixels per channel
// row), splits them in registers and stores four channels per 16-byte chunk
//     A[m = pixel ][k = channel]: (m % 8) * 16 + (m / 8) * 1280 + (k / 4) * 128 + (k % 4) * 4   bytes
//     B[n = hidden][k = channel]: (n % 8) * 16 + (n / 8) * 1280 + (k / 4) * 128 + (k % 4) * 4   bytes
// (W1 is staged once per CTA); LBO = 128 B between the 16-byte K chunks, SBO = 1280 B between 8-row groups
// (K = 40: up to 32 channels, then the ones column that multiplies b1 in column C of W1).
#include "common.cuh"
#include "tc_common.cuh"

namespace fno {
namespace {

constexpr int TC_M = 128;          // pixels per tile = TMEM lanes
constexpr int TC_HID = 128;        // hidden units = accumulator columns
constexpr int TC_KP = 40;          // channel padding of the staged operands: C <= 32 channels + the ones column (b1)
constexpr int TC_VP = 8;           // output variables: W2 is staged for 2, 4 or 8 of them

struct HeadGeo {
  int R_in, W_in, R_out, Wp;
  long npix, plane;
};

// byte offsets inside the staged operand buffers (see the file header); SBO = TC_KP / 4 chunks of 128 B
constexpr int TC_SBO = TC_KP / 4 * 128;
__device__ __forceinline__ int b_off_bytes(int n, int k) { return (n & 7) * 16 + (n >> 3) * TC_SBO + (k >> 2) * 128 + (k & 3) * 4; }

constexpr int A_BYTES = 16 * TC_SBO;  // [16 pixel groups ][10 channel chunks][8][4] floats
constexpr int B_BYTES = 16 * TC_SBO;  // [16 hidden groups][10 channel chunks][8][4] floats

// ------------------------------------------------------------------------------------------
// forward:  out = (W2 gelu(W1 h + b1) + b2) * std + mean
//
// Persistent CTA, one per SM; 4 groups of 4 loader / epilogue warps + 1 MMA-issue warp.  A group owns whole
// 128-pixel tiles (group g takes the CTA's tiles g, g + 4, ...), one operand slot and one TMEM accumulator
// (4 x 128 = all 512 columns).  A thread is one pixel (its TMEM lane): it walks all 128 hidden columns, so the
// 128 -> V product completes in its registers, and no barrier couples the groups.  The four groups drift apart,
// so the MUFU-heavy GELU bursts of one group overlap the staging, the MMAs and the waits of the others.  b1 rides
// in the MMA as column C of W1 against a column of ones in h.
// ------------------------------------------------------------------------------------------
constexpr int TCF_GROUPS = 4;
constexpr int TCF_EPI_WARPS = 4 * TCF_GROUPS;
constexpr int TCF_THREADS = 32 * TCF_EPI_WARPS + 32;
constexpr int TCF_MAXC = 32;               // channels a thread holds in registers (C <= 32)

template <int NV>   // output variables accumulated per hidden unit: 2 (V <= 2), 4 or 8
__global__ void __launch_bounds__(TCF_THREADS, 1)
head_fwd_tc_kernel(const float* __restrict__ h, const float* __restrict__ W1, const float* __restrict__ b1,
                   const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ stats,
                   float* __restrict__ out, HeadGeo g, int C, int V, int tiles_per_sample, int total_tiles, int single) {
  FNO_SPLIT_CONSTS(single);                  // single: 0 = 3xTF32 (fp32 mode), 1 = tf32, 2 = bf16 operands
  extern __shared__ __align__(128) unsigned char tsm[];
  unsigned char* a_hi = tsm;                       // [4 groups][A_BYTES]
  unsigned char* a_lo = a_hi + TCF_GROUPS * A_BYTES;
  unsigned char* w_hi = a_lo + TCF_GROUPS * A_BYTES;   // B_BYTES
  unsigned char* w_lo = w_hi + B_BYTES;
  float* W2s = reinterpret_cast<float*>(w_lo + B_BYTES);   // [HID / 2 column pairs][NV][2]
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(W2s + TC_HID * TC_VP);
  unsigned long long* a_ready = bars;                       // [4] group -> MMA: operands of its next tile staged
  unsigned long long* d_full = bars + TCF_GROUPS;           // [4] MMA -> group: accumulator ready, operand slot free
  unsigned long long* d_free = bars + 2 * TCF_GROUPS;       // [4] group -> MMA: accumulator read
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 3 * TCF_GROUPS);

  // warp index made provably warp-uniform (role branches non-divergent for the compiler: the MMA warp then
  // issues back-to-back UTCHMMAs from uniform registers, see tc_common.cuh)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < TCF_GROUPS; ++s) {
      mbar_init(a_ready + s, 4);
      mbar_init(d_full + s, 1);
      mbar_init(d_free + s, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == TCF_EPI_WARPS) tmem_alloc(tmem_slot, TCF_GROUPS * TC_HID);
  // stage W1 | b1 (hi / lo, K-major B operand, b1 in column C, zero padded to TC_KP channels) and W2
  for (int i = tid; i < TC_HID * TC_KP; i += TCF_THREADS) {
    const int n = i / TC_KP, k = i - n * TC_KP;
    float hi = 0.f, lo = 0.f;
    if (k < C) split_rm(__ldg(W1 + (size_t)n * C + k), hi, lo, sp_rnd, sp_msk);
    else if (k == C) split_rm(__ldg(b1 + n), hi, lo, sp_rnd, sp_msk);
    *reinterpret_cast<float*>(w_hi + b_off_bytes(n, k)) = hi;
    *reinterpret_cast<float*>(w_lo + b_off_bytes(n, k)) = lo;
  }
  for (int i = tid; i < TC_HID * NV; i += TCF_THREADS) {
    const int jp = i / (2 * NV), v = (i >> 1) % NV, j = 2 * jp + (i & 1);
    W2s[i] = (v < V) ? __ldg(W2 + (size_t)v * TC_HID + j) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const int ksteps = (C + 1 + 7) / 8;              // channels + the ones column
  const int ntl = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA

  if (warp == TCF_EPI_WARPS) {
    // ---- MMA issuer: the whole warp stays converged, one elected lane issues; groups are served in tile order
    constexpr unsigned idesc = umma_idesc_tf32(TC_M, TC_HID, /*A K-major*/ 0, /*B K-major*/ 0);
    const unsigned long long d_a_h = umma_desc(a_hi, 128, TC_SBO), d_a_l = umma_desc(a_lo, 128, TC_SBO);
    const unsigned long long d_w_h = umma_desc(w_hi, 128, TC_SBO), d_w_l = umma_desc(w_lo, 128, TC_SBO);
    for (int it = 0; it < ntl; ++it) {
      const int gr = it & (TCF_GROUPS - 1);
      const unsigned ph = (unsigned)(it / TCF_GROUPS) & 1u;
      mbar_wait(a_ready + gr, ph);
      mbar_wait(d_free + gr, ph ^ 1u);
      tc_fence_after();
      __syncwarp();
      const unsigned long long so = (unsigned long long)(gr * (A_BYTES >> 4));
      const unsigned d = tmem_base + (unsigned)gr * TC_HID;
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < TC_KP / 8; ++ks) {
          // K = 8 per instruction = two 16-byte chunks: +256 B per K step for both operands
          if (ks < ksteps && (pass == 2 || !single))     // tf32 mode: the hi*hi pass alone
            tc_mma_tf32_elect(d, (pass == 0 ? d_a_l : d_a_h) + so + (unsigned long long)(ks * (256 >> 4)),
                              (pass == 1 ? d_w_l : d_w_h) + (unsigned long long)(ks * (256 >> 4)), idesc,
                              single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
        }
      tc_commit_elect(d_full + gr);
    }
  } else {
    // ---- loader / epilogue groups ------------------------------------------------------------------
    const int quad = warp & 3;                     // TMEM lane quadrant of this warp
    const int gr = warp >> 2;                      // group: tiles gr, gr + 4, ... of the CTA
    const int m = quad * 32 + lane;                // pixel of the tile (staged and finished by this thread)
    const int nk = ntl > gr ? (ntl - gr + TCF_GROUPS - 1) / TCF_GROUPS : 0;   // tiles of this group
    const int abase = gr * A_BYTES + (m & 7) * 16 + (m >> 3) * TC_SBO;
    float raw[TCF_MAXC];
    auto load_raw = [&](int k) {                   // this thread's channels of the group's tile `k` (zeros past the end)
      const int tile = (int)blockIdx.x + (gr + TCF_GROUPS * k) * (int)gridDim.x;
      const bool in = k < nk;
      const int b = in ? tile / tiles_per_sample : 0;
      const long p = in ? (long)(tile - b * tiles_per_sample) * TC_M + m : 0;
      const bool valid = in && p < g.npix;
      const long r = valid ? p / g.W_in : 0;
      const float* hp = h + (size_t)b * C * g.plane + r * g.Wp + (valid ? p - r * g.W_in : 0);
      const int cmax = valid ? C : 0;
      const int pl = (int)g.plane;
#pragma unroll
      for (int c = 0; c < TCF_MAXC; ++c) {
        raw[c] = (c < cmax) ? __ldg(hp) : 0.f;
        hp += pl;
      }
    };
    auto store_raw = [&]() {
#pragma unroll
      for (int kc = 0; kc < TC_KP / 4; ++kc) {
        if (kc < 2 * ksteps) {
          float hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = 4 * kc + e;
            split_rm(c < TCF_MAXC && c < C ? raw[c < TCF_MAXC ? c : 0] : (c == C ? 1.f : 0.f), hi[e], lo[e], sp_rnd, sp_msk);
          }
          *reinterpret_cast<float4*>(a_hi + abase + kc * 128) = make_float4(hi[0], hi[1], hi[2], hi[3]);
          if (!single) *reinterpret_cast<float4*>(a_lo + abase + kc * 128) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready + gr);
    };
    // prologue: the group's tile 0 staged, tile 1 in flight
    if (nk > 0) {
      load_raw(0);
      store_raw();
      load_raw(1);
    }
    const float4* __restrict__ w2q = reinterpret_cast<const float4*>(W2s);
    for (int k = 0; k < nk; ++k) {
      const unsigned ph = (unsigned)k & 1u;
      const int tile = (int)blockIdx.x + (gr + TCF_GROUPS * k) * (int)gridDim.x;
      const int b = tile / tiles_per_sample;
      const long p = (long)(tile - b * tiles_per_sample) * TC_M + m;
      mbar_wait(d_full + gr, ph);
      tc_fence_after();
      // the MMAs of tile k have read the operand slot: stage tile k+1, put tile k+2's loads in flight
      if (k + 1 < nk) store_raw();
      load_raw(k + 2);

      // -- epilogue of tile k: GELU and the 128 -> V product of this thread's pixel, column pairs on the f32x2 pipe
      float2 o[NV];                                // (even, odd) hidden-column partial sums of output v
#pragma unroll
      for (int v = 0; v < NV; ++v) o[v] = f32x2(0.f);
#pragma unroll 1
      for (int j0 = 0; j0 < TC_HID; j0 += 16) {
        float v[16];
        tmem_ld16(tmem_base + ((unsigned)(quad * 32) << 16) + (unsigned)(gr * TC_HID + j0), v);
        if (j0 + 16 == TC_HID) {                   // accumulator fully read: the group's next tile may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(d_free + gr);
        }
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          const float2 gl = gelu_fast2(make_float2(v[i], v[i + 1]));
#pragma unroll
          for (int q = 0; q < NV / 2; ++q) {       // W2 of outputs 2q, 2q+1 at columns j, j+1 (warp-wide broadcast)
            const float4 w = w2q[((j0 + i) / 2) * (NV / 2) + q];
            o[2 * q] = __ffma2_rn(make_float2(w.x, w.y), gl, o[2 * q]);
            o[2 * q + 1] = __ffma2_rn(make_float2(w.z, w.w), gl, o[2 * q + 1]);
          }
        }
      }
      if (p < g.npix) {
        const float* __restrict__ mean = stats + (size_t)b * 2 * V;
        const float* __restrict__ sd = mean + V;
        float* __restrict__ op = out + ((size_t)b * g.npix + p) * V;
#pragma unroll
        for (int v = 0; v < NV; ++v)
          if (v < V) op[v] = fmaf(o[v].x + o[v].y + __ldg(b2 + v), __ldg(sd + v), __ldg(mean + v));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == TCF_EPI_WARPS) tmem_dealloc(tmem_base, TCF_GROUPS * TC_HID);
}

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" int fno_head_fwd_tc(const float* h, const float* W1, const float* b1, const float* W2, const float* b2,
                               const float* stats, float* out, int B, int R_in, int W_in, int R_out, int Wp, int C,
                               int HID, int V, fno_stream_t stream) {
  if (!h || !W1 || !b1 || !W2 || !b2 || !stats || !out || B <= 0 || R_in <= 0 || W_in <= 0 || R_out < R_in || Wp < W_in) {
    set_error("fno_head_fwd_tc: bad argument");
    return FNO_E_ARG;
  }
  if (HID != TC_HID || C > TCF_MAXC || C < 1 || V < 1 || V > TC_VP) {
    set_error("fno_head_fwd_tc: supports hidden width 128, C <= %d, V <= %d (got %d, %d, %d)", TCF_MAXC, TC_VP, HID, C, V);
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HeadGeo g;
  g.R_in = R_in; g.W_in = W_in; g.R_out = R_out; g.Wp = Wp;
  g.npix = (long)R_in * W_in;
  g.plane = (long)R_out * Wp;
  const long tps = (g.npix + TC_M - 1) / TC_M;
  const long total = tps * B;
  if (total > 0x7fffffffL || g.plane > 0x7fffffffL / 16) { set_error("fno_head_fwd_tc: too many tiles / plane too large"); return FNO_E_ARG; }
  const size_t smem = 2 * TCF_GROUPS * A_BYTES + 2 * B_BYTES + sizeof(float) * TC_HID * TC_VP +
                      3 * TCF_GROUPS * sizeof(unsigned long long) + 16;
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(head_fwd_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaFuncSetAttribute(head_fwd_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaFuncSetAttribute(head_fwd_tc_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_fwd_tc)");
    done.mark();
  }
  const int ctas = (int)(total < 148 ? total : 148);
  const int single = g_math_mode.load();
  if (V <= 2)
    head_fwd_tc_kernel<2><<<ctas, TCF_THREADS, smem, st>>>(h, W1, b1, W2, b2, stats, out, g, C, V, (int)tps, (int)total, single);
  else if (V <= 4)
    head_fwd_tc_kernel<4><<<ctas, TCF_THREADS, smem, st>>>(h, W1, b1, W2, b2, stats, out, g, C, V, (int)tps, (int)total, single);
  else
    head_fwd_tc_kernel<8><<<ctas, TCF_THREADS, smem, st>>>(h, W1, b1, W2, b2, stats, out, g, C, V, (int)tps, (int)total, single);
  count_launch();
  return check_launch("head_fwd_tc_kernel");
}
