// The 1x1-conv bypass of a wide Fourier layer (nn.Conv2d(width, width, 1), fno/fno.py:131-134,162; BASELINE configs[2]:
// width 64) and its data gradient on the 5th-generation tensor cores (tcgen05 + TMEM), fp32-accurate through the
// 3xTF32 split of head_tc.cu.
//
// At width 64 the product is 64 MACs per loaded float: the FP32 kernel (pointwise2_kernel) is bound by instruction
// issue at 0.24 of the HBM roof (DESIGN.md section 4, cfg 3).  Here a 128-pixel tile is one GEMM
//     D[128 pixels x 64 out channels] = A[128 x K] B[K x 64],   K = in channels <= 64
// with the activation tile staged K-major in shared memory (thread = pixel: coalesced 128-byte channel-row loads, split
// hi / lo in registers, four channels per 16-byte chunk -- the layout head_tc.cu verified on the hardware, SBO widened to
// 16 chunks), W (or W^T for the data gradient) hi / lo staged once per CTA, the accumulator in TMEM (double-buffered:
// the MMAs of tile i+1 run under the stores of tile i) and an epilogue that only adds the bias and writes coalesced
// channel rows.  What is left is a streaming kernel: 64 KB in + out per tile against 24 MMAs.
#include <cstdlib>

#include "common.cuh"
#include "tc_common.cuh"

namespace fno {
namespace {

constexpr int PT_M = 128;                       // pixels per tile = TMEM lanes
constexpr int PT_N = 64;                        // out channels (padded) = accumulator columns
constexpr int PT_K = 64;                        // in channels (padded)
constexpr int PT_SBO = (PT_K / 4) * 128;        // 8-row group pitch: 16 chunks of 16 bytes per row, LBO = 128
constexpr int PT_A_BYTES = (PT_M / 8) * PT_SBO; // 32 KB
constexpr int PT_B_BYTES = (PT_N / 8) * PT_SBO; // 16 KB
constexpr int PT_EPI_WARPS = 16;
constexpr int PT_EPI_THREADS = 32 * PT_EPI_WARPS;
constexpr int PT_THREADS = PT_EPI_THREADS + 32;
constexpr int PT_MAXCH = 4;                     // 16-byte channel chunks staged per thread
constexpr int PT_SMEM = 4 * PT_A_BYTES + 2 * PT_B_BYTES + PT_N * 4 + 6 * 8 + 16;

__device__ __forceinline__ int pt_off(int n, int k) { return (n & 7) * 16 + (n >> 3) * PT_SBO + (k >> 2) * 128 + (k & 3) * 4; }

// out[b, n, p] = sum_k Wm[n, k] in[b, k, p] (+ bias[n]);  Wm[n, k] = W[n * ldw + k]  (transpose == 0: the convolution)
//                                                        Wm[n, k] = W[k * ldw + n]  (transpose != 0: its data gradient)
// Persistent CTA, one per SM; 16 loader / epilogue warps (4 TMEM lane quadrants x 4 column quarters) + 1 MMA-issue warp.
__global__ void __launch_bounds__(PT_THREADS, 1)
pointwise_tc_kernel(const float* __restrict__ in, const float* __restrict__ W, const float* __restrict__ bias,
                    float* __restrict__ out, long N, int Cin, int Cout, int ldw, int transpose, int tiles_per_sample,
                    int total_tiles, int single) {
  FNO_SPLIT_CONSTS(single);                     // single: 0 = 3xTF32 (fp32 mode), 1 = tf32, 2 = bf16 operands
  extern __shared__ __align__(128) unsigned char psm[];
  unsigned char* a_hi = psm;                    // [2 stages][PT_A_BYTES]
  unsigned char* a_lo = a_hi + 2 * PT_A_BYTES;
  unsigned char* w_hi = a_lo + 2 * PT_A_BYTES;
  unsigned char* w_lo = w_hi + PT_B_BYTES;
  float* bs = reinterpret_cast<float*>(w_lo + PT_B_BYTES);            // [PT_N]
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(bs + PT_N);
  unsigned long long* a_ready = bars;           // [2]
  unsigned long long* d_full = bars + 2;        // [2]
  unsigned long long* d_free = bars + 4;        // [2]
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 6);

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(a_ready + s, PT_EPI_WARPS);
      mbar_init(d_full + s, 1);
      mbar_init(d_free + s, PT_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == PT_EPI_WARPS) tmem_alloc(tmem_slot, 2 * PT_N);
  for (int i = tid; i < PT_N * PT_K; i += PT_THREADS) {
    const int n = i / PT_K, k = i - n * PT_K;
    float hi = 0.f, lo = 0.f;
    if (n < Cout && k < Cin) split_rm(__ldg(W + (transpose ? (size_t)k * ldw + n : (size_t)n * ldw + k)), hi, lo, sp_rnd, sp_msk);
    *reinterpret_cast<float*>(w_hi + pt_off(n, k)) = hi;
    *reinterpret_cast<float*>(w_lo + pt_off(n, k)) = lo;
  }
  for (int i = tid; i < PT_N; i += PT_THREADS) bs[i] = (bias != nullptr && i < Cout) ? __ldg(bias + i) : 0.f;
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const int ksteps = (Cin + 7) / 8;
  const int ntl = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA

  if (warp == PT_EPI_WARPS) {
    // ---- MMA issuer: the whole warp stays converged, one elected lane issues ---------------------------
    constexpr unsigned idesc = umma_idesc_tf32(PT_M, PT_N, /*A K-major*/ 0, /*B K-major*/ 0);
    const unsigned long long d_a_h = umma_desc(a_hi, 128, PT_SBO), d_a_l = umma_desc(a_lo, 128, PT_SBO);
    const unsigned long long d_w_h = umma_desc(w_hi, 128, PT_SBO), d_w_l = umma_desc(w_lo, 128, PT_SBO);
    for (int it = 0; it < ntl; ++it) {
      const int st = it & 1;
      const unsigned ph = (unsigned)(it >> 1) & 1u;
      mbar_wait(a_ready + st, ph);
      mbar_wait(d_free + st, ph ^ 1u);
      tc_fence_after();
      __syncwarp();
      const unsigned long long so = (unsigned long long)(st * (PT_A_BYTES >> 4));
      const unsigned d = tmem_base + (unsigned)(st * PT_N);
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < PT_K / 8; ++ks)           // K = 8 per instruction = two 16-byte chunks: +256 B
          if (ks < ksteps && (pass == 2 || !single))
            tc_mma_tf32_elect(d, (pass == 0 ? d_a_l : d_a_h) + so + (unsigned long long)(ks * (256 >> 4)),
                              (pass == 1 ? d_w_l : d_w_h) + (unsigned long long)(ks * (256 >> 4)), idesc,
                              single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      tc_commit_elect(d_full + st);
    }
  } else {
    // ---- loader / epilogue warps ------------------------------------------------------------------
    const int quad = warp & 3;                     // TMEM lane quadrant of this warp
    const int colq = warp >> 2;                    // out channels [16 * colq, 16 * colq + 16)
    const int m = quad * 32 + lane;                // pixel of the tile owned in the epilogue
    const int pm = tid & (PT_M - 1);               // pixel of the tile staged by this thread
    const int kq = tid >> 7;                       // chunk residue staged by this thread
    const int abase = (pm & 7) * 16 + (pm >> 3) * PT_SBO;
    float raw[PT_MAXCH][4];
    // 32-bit element offsets (the launcher checks 64 N < 2^31): one IMAD per access instead of a 64-bit product -- the
    // first version spent 55 % of its issue slots on address arithmetic (profiles/r2c_wide_ncu.md)
    const int Ni = (int)N;
    auto load_raw = [&](int it) {                  // this thread's channels of tile `it` (zeros past the end)
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const bool inr = it < ntl;
      const int b = inr ? tile / tiles_per_sample : 0;
      const int p = inr ? (tile - b * tiles_per_sample) * PT_M + pm : 0;
      const bool valid = inr && p < Ni;
      // a running pointer (two adds per access): the compiler otherwise rebuilds base + index * stride from the constant
      // bank for every element (8 integer instructions per load)
      const float* ip = in + ((size_t)b * Cin + 4 * kq) * N + (valid ? p : 0);
      const int cmax = valid ? Cin - 4 * kq : 0;   // channels 4 kq + j, j < cmax, exist
#pragma unroll
      for (int u = 0; u < PT_MAXCH; ++u) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          raw[u][e] = (16 * u + e < cmax) ? __ldg(ip) : 0.f;
          ip += (e < 3) ? Ni : 13 * Ni;
        }
      }
    };
    auto store_raw = [&](int st) {
#pragma unroll
      for (int u = 0; u < PT_MAXCH; ++u) {
        const int kc = kq + 4 * u;
        if (kc < 2 * ksteps) {
          float hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) split_rm(raw[u][e], hi[e], lo[e], sp_rnd, sp_msk);
          *reinterpret_cast<float4*>(a_hi + st * PT_A_BYTES + abase + kc * 128) = make_float4(hi[0], hi[1], hi[2], hi[3]);
          if (!single) *reinterpret_cast<float4*>(a_lo + st * PT_A_BYTES + abase + kc * 128) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready + st);
    };
    // prologue: tile 0 staged, tile 1 in flight
    load_raw(0);
    store_raw(0);
    load_raw(1);
    for (int it = 0; it < ntl; ++it) {
      const int st = it & 1;
      const unsigned ph = (unsigned)(it >> 1) & 1u;
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int b = tile / tiles_per_sample;
      const int p = (tile - b * tiles_per_sample) * PT_M + m;
      // stage tile it+1 (its operand buffer was last read by the MMAs of tile it-1, whose completion this thread
      // observed in the previous epilogue), then put tile it+2's loads in flight
      if (it + 1 < ntl) store_raw(st ^ 1);
      load_raw(it + 2);

      mbar_wait(d_full + st, ph);
      tc_fence_after();
      float v[16];
      tmem_ld16(tmem_base + ((unsigned)(quad * 32) << 16) + (unsigned)(st * PT_N + colq * 16), v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(d_free + st);     // the accumulator may be overwritten by tile it+2's MMAs
      if (p < Ni) {
        float* op = out + ((size_t)b * Cout + colq * 16) * N + p;
        const int nout = Cout - colq * 16;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          if (i < nout) *op = v[i] + bs[colq * 16 + i];
          op += Ni;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == PT_EPI_WARPS) tmem_dealloc(tmem_base, 2 * PT_N);
}


// ------------------------------------------------------------------------------------------
// Weight / bias gradient of the wide 1x1 conv:  gW[o, i] = sum_{b,p} ds[b, o, p] a[b, i, p],  gb[o] = sum ds[b, o, p].
// The contraction runs over PIXELS, which are contiguous in both tensors, so a 64-pixel slab of [ds ; a] is already
// K-major: thread = (channel row, 16-byte pixel chunk) loads one float4, splits it and stores hi / lo into ONE stacked
// operand buffer  rows 0..63 = ds channels, 64..127 = a channels, 128..143 = a constant row of ones + zero padding
// (LBO = 144 B: the chunk-strided 16-byte stores of a quarter warp are conflict-free).  A = rows 0..127 and
// B = rows 64..143 of that same buffer:
//     D[128 x 80] += [ds ; a] [a ; 1]^T        M = 128, N = 80, K = 8 x 8 pixels per slab, 3xTF32
// rows 0..63 of D are gW (columns 0..63) and gb (column 64); rows 64..127 (a a^T) are the price of not staging a second
// operand -- the tensor pipe has the room (24 MMAs ~ 0.8 k cycles per slab against ~1.5 k cycles of HBM time).
// The tensor core's fp32 accumulate truncates: a chain of ~500 MMAs into one TMEM tile measured 7e-6 of relative error
// (biased, so it grows with the chain), too much for the 1e-5 fp32-mode bound.  A TMEM tile therefore only collects
// WT_CHAIN = 2 slabs (48 MMAs); the loader warps drain it into IEEE fp32 register accumulators while the next chain fills
// the other tile.  Per-CTA partials go through partial_reduce_kernel.
// ------------------------------------------------------------------------------------------
// RA = rows of the gradient (64: the bypass; 128: the projection head's hidden layer, head_wide_tc.cu -- then A is the
// ds block alone and B = [a ; 1]), KT = pixels per slab (64 / 32: the stacked buffer must fit twice, hi and lo).
constexpr int WT_LBO = 144;
constexpr int WT_N = 80;
constexpr int WT_LD_WARPS = 16;
constexpr int WT_THREADS = 32 * WT_LD_WARPS + 32;
template <int RA, int KT>
struct WtCfg {
  static constexpr int SBO = (KT / 4) * WT_LBO;          // 2304 / 1152
  static constexpr int ROWS = RA + 80;                   // ds | a (64) | ones + zero padding (16)
  static constexpr int BUF = (ROWS / 8) * SBO;           // bytes per hi / lo buffer
  static constexpr int SMEM = 4 * BUF + 8 * 8 + 16;
  static constexpr int RPP = (32 * WT_LD_WARPS) / (KT / 4);   // rows staged per pass of the loader threads
  static constexpr int NU = (RA + 64) / RPP;             // passes
  static_assert((RA + 64) % RPP == 0, "loader mapping");
};

template <int RA, int KT>
__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tc_kernel(const float* __restrict__ ds, const float* __restrict__ a, float* __restrict__ part, int Co, int Ci, long N,
                int slabs_per_sample, long total_slabs, long slabs_per_cta, int single) {
  FNO_SPLIT_CONSTS(single);
  using Cfg = WtCfg<RA, KT>;
  constexpr int WT_KT = KT, WT_SBO = Cfg::SBO, WT_BUF = Cfg::BUF;
  extern __shared__ __align__(128) unsigned char wsm[];
  unsigned char* b_hi = wsm;                     // [2 stages][WT_BUF]
  unsigned char* b_lo = wsm + 2 * WT_BUF;
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(wsm + 4 * WT_BUF);
  unsigned long long* a_ready = bars;            // [2] loaders -> MMA
  unsigned long long* a_free = bars + 2;         // [2] MMA -> loaders
  unsigned long long* d_full = bars + 4;         // [2] MMA -> drain: a chain of two slabs has landed in D[chain & 1]
  unsigned long long* d_free = bars + 6;         // [2] drain -> MMA
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 8);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(a_ready + s, WT_LD_WARPS);
      mbar_init(a_free + s, 1);
      mbar_init(d_full + s, 1);
      mbar_init(d_free + s, WT_LD_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WT_LD_WARPS) tmem_alloc(tmem_slot, 256);
  // constant rows RA+64 .. RA+79 of both stages: the first = ones (hi = 1, lo = 0), the rest zero
  for (int i = tid; i < 2 * 16 * WT_KT; i += WT_THREADS) {
    const int s = i / (16 * WT_KT), r = RA + 64 + (i / WT_KT) % 16, k = i % WT_KT;
    const int off = s * WT_BUF + (r & 7) * 16 + (r >> 3) * WT_SBO + (k >> 2) * WT_LBO + (k & 3) * 4;
    *reinterpret_cast<float*>(b_hi + off) = r == RA + 64 ? 1.0f : 0.0f;
    *reinterpret_cast<float*>(b_lo + off) = 0.0f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const long s_begin = (long)blockIdx.x * slabs_per_cta;
  long s_end = s_begin + slabs_per_cta;
  if (s_end > total_slabs) s_end = total_slabs;
  const int n = s_end > s_begin ? (int)(s_end - s_begin) : 0;

  if (warp == WT_LD_WARPS) {
    constexpr unsigned idesc = umma_idesc_tf32(128, WT_N, 0, 0);
    for (int it = 0; it < n; ++it) {
      const int st = it & 1;                       // operand stage = position inside the chain
      const int c = it >> 1, db = c & 1;           // chain and its TMEM tile
      mbar_wait(a_ready + st, (unsigned)c & 1u);
      if (st == 0 && c >= 2) mbar_wait(d_free + db, (unsigned)((c >> 1) - 1) & 1u);   // chain c-2 drained
      tc_fence_after();
      __syncwarp();
      const unsigned long long a_h = umma_desc(b_hi + st * WT_BUF, WT_LBO, WT_SBO), a_l = umma_desc(b_lo + st * WT_BUF, WT_LBO, WT_SBO);
      const unsigned long long bo = (unsigned long long)(((RA / 8) * WT_SBO) >> 4);   // B = rows RA .. RA+79
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < WT_KT / 8; ++ks)
          if (pass == 2 || !single)
            tc_mma_tf32_elect(tmem_base + (unsigned)(128 * db),
                              (pass == 0 ? a_l : a_h) + (unsigned long long)(ks * (2 * WT_LBO >> 4)),
                              (pass == 1 ? a_l : a_h) + bo + (unsigned long long)(ks * (2 * WT_LBO >> 4)), idesc,
                              (st != 0 || ks != 0 || (!single && pass != 0)) ? 1u : 0u);
      tc_commit_elect(a_free + st);
      if (st == 1 || it == n - 1) tc_commit_elect(d_full + db);
    }
  } else {
    const int q = tid % (KT / 4);                  // 16-byte pixel chunk of the slab
    const int r0 = tid / (KT / 4);                 // rows r0 + RPP u
    constexpr int NU = Cfg::NU;
    float4 raw[2][NU];
    auto load_raw = [&](int it, float4 (&v)[NU]) {
      const long slab = s_begin + it;
      const bool inr = it < n;
      const long b = inr ? slab / slabs_per_sample : 0;
      const long k = inr ? (slab - b * slabs_per_sample) * WT_KT + 4 * q : 0;
      const bool pv = inr && k < N;
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const int r = r0 + Cfg::RPP * u;
        const bool is_ds = r < RA;
        const int ch = is_ds ? r : r - RA;
        const int C = is_ds ? Co : Ci;
        const float* src = (is_ds ? ds : a) + ((size_t)b * C + ch) * N + k;
        v[u] = (pv && ch < C) ? __ldg(reinterpret_cast<const float4*>(src)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    auto store_raw = [&](int st, const float4 (&v)[NU]) {
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const int r = r0 + Cfg::RPP * u;
        const int off = st * WT_BUF + (r & 7) * 16 + (r >> 3) * WT_SBO + q * WT_LBO;
        float4 hi, lo;
        split_rm(v[u].x, hi.x, lo.x, sp_rnd, sp_msk);
        split_rm(v[u].y, hi.y, lo.y, sp_rnd, sp_msk);
        split_rm(v[u].z, hi.z, lo.z, sp_rnd, sp_msk);
        split_rm(v[u].w, hi.w, lo.w, sp_rnd, sp_msk);
        *reinterpret_cast<float4*>(b_hi + off) = hi;
        if (!single) *reinterpret_cast<float4*>(b_lo + off) = lo;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready + st);
    };
    // rows 0..RA-1 of D (TMEM lanes 0..RA-1) are gW | gb: warp <-> (quadrant, 16 columns), IEEE accumulators
    constexpr int NQ = RA / 32;
    const int quad = warp & 3, colq = warp >> 2;
    float accw[16], accb = 0.f;
#pragma unroll
    for (int e = 0; e < 16; ++e) accw[e] = 0.f;
    const int nchains = (n + 1) >> 1;
    int drained = 0;
    auto drain = [&]() {                           // chain `drained`: D[drained & 1] -> registers, tile handed back
      const int db = drained & 1;
      mbar_wait(d_full + db, (unsigned)(drained >> 1) & 1u);
      tc_fence_after();
      if (quad < NQ) {
        float v[16];
        tmem_ld16(tmem_base + ((unsigned)(quad * 32) << 16) + (unsigned)(128 * db + 16 * colq), v);
#pragma unroll
        for (int e = 0; e < 16; ++e) accw[e] += v[e];
        if (colq == 0) {
          float w[8];
          tmem_ld8(tmem_base + ((unsigned)(quad * 32) << 16) + (unsigned)(128 * db + 64), w);
          accb += w[0];
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(d_free + db);
      ++drained;
    };
    load_raw(0, raw[0]);
    load_raw(1, raw[1]);
    for (int it = 0; it < n; it += 2) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int i = it + h;
        if (i < n) {
          if (i >= 2) mbar_wait(a_free + h, (unsigned)((i >> 1) - 1) & 1u);   // slab i-2's MMAs have read stage h
          store_raw(h, raw[h]);
          load_raw(i + 2, raw[h]);
          if (h == 1 && i >= 3) drain();           // chain (i - 3) / 2 finished a whole slab ago: no wait in practice
        }
      }
    }
    while (drained < nchains) drain();
    if (quad < NQ) {
      const int o = quad * 32 + lane;
      float* __restrict__ pp = part + (size_t)blockIdx.x * Co * (Ci + 1);
      if (o < Co) {
#pragma unroll
        for (int e = 0; e < 16; ++e)
          if (16 * colq + e < Ci) pp[(size_t)o * (Ci + 1) + 16 * colq + e] = accw[e];
        if (colq == 0) pp[(size_t)o * (Ci + 1) + Ci] = accb;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == WT_LD_WARPS) tmem_dealloc(tmem_base, 256);
}

}  // namespace

bool pointwise_tc_supported(int Cin, int Cout) {
  static const bool off = [] { const char* e = std::getenv("FNO_PW_TC"); return e != nullptr && e[0] == '0'; }();
  const int wmax = Cin > Cout ? Cin : Cout;
  return !off && wmax > 32 && wmax <= PT_K;
}

int launch_pointwise_tc(const float* in, const float* W, const float* bias, float* out, int B, int Co, int Ci, long N,
                        int transpose, cudaStream_t st) {
  const int Cout = transpose ? Ci : Co, Cin = transpose ? Co : Ci;
  const long tps = (N + PT_M - 1) / PT_M;
  const long total = tps * B;
  if (total > 0x7fffffffL || N > 0x7fffffffL / 64) { set_error("fno_pointwise_fwd: too many tiles / plane too large"); return FNO_E_ARG; }
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(pointwise_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PT_SMEM) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(pointwise_tc)");
    done.mark();
  }
  const int ctas = (int)(total < 148 ? total : 148);
  pointwise_tc_kernel<<<ctas, PT_THREADS, PT_SMEM, st>>>(in, W, bias, out, N, Cin, Cout, Ci, transpose, (int)tps, (int)total,
                                                         g_math_mode.load());
  count_launch();
  return check_launch("pointwise_tc_kernel");
}

// per-CTA partial records [ctas][Co][Ci + 1] into `part` (the caller runs partial_reduce_kernel over them); returns the
// number of records through *nparts.  Needs N % 4 == 0 and 16-byte aligned tensors (the caller checks).
template <int RA, int KT>
static int launch_wgrad_tc_t(const float* ds, const float* a, float* part, int B, int Co, int Ci, long N, int max_parts,
                             int* nparts, cudaStream_t st) {
  using Cfg = WtCfg<RA, KT>;
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(wgrad_tc_kernel<RA, KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(wgrad_tc)");
    done.mark();
  }
  const int sps = (int)((N + KT - 1) / KT);
  const long total = (long)B * sps;
  long ctas = total < 148 ? total : 148;
  if (ctas > max_parts) ctas = max_parts;
  const long spc = (total + ctas - 1) / ctas;
  ctas = (total + spc - 1) / spc;
  wgrad_tc_kernel<RA, KT><<<(unsigned)ctas, WT_THREADS, Cfg::SMEM, st>>>(ds, a, part, Co, Ci, N, sps, total, spc,
                                                                                g_math_mode.load());
  count_launch();
  *nparts = (int)ctas;
  return check_launch("wgrad_tc_kernel");
}

int launch_wgrad_tc(const float* ds, const float* a, float* part, int B, int Co, int Ci, long N, int max_parts, int* nparts,
                    cudaStream_t st) {
  return launch_wgrad_tc_t<64, 64>(ds, a, part, B, Co, Ci, N, max_parts, nparts, st);
}

// Co <= 128 gradient rows (the projection head's hidden layer), Ci <= 64
int launch_wgrad_tc_rows128(const float* ds, const float* a, float* part, int B, int Co, int Ci, long N, int max_parts,
                            int* nparts, cudaStream_t st) {
  return launch_wgrad_tc_t<128, 32>(ds, a, part, B, Co, Ci, N, max_parts, nparts, st);
}

}  // namespace fno
