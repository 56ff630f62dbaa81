// Projection-head backward on the 5th-generation tensor cores (tcgen05 + TMEM), fp32-accurate through
// the 3xTF32 split of head_tc.cu.  Autograd of  out = (W2 gelu(W1 h + b1) + b2) * std + mean
// (fno/fno.py:180-187): the hidden layer is recomputed per 64-pixel tile and all three dense
// contractions run as tcgen05.mma.kind::tf32 with accumulators in TMEM:
//
//   (a) pre^T[j, px]  = sum_c  W1[j, c] h[px, c] + b1[j]      M = 128 hidden, N = 64 px, K = 24
//                        (the bias rides in the padding: column C of W1 holds b1, column C of h is 1)
//   (b) dh[px, c]      = sum_j  dpre[px, j] W1[j, c]           M = 64 px,     N = 24,    K = 128
//   (c) gW1[j, c]     += sum_px dpre[px, j] h[px, c]           M = 128 hidden, N = 32,    K = 64
//                        (accumulates in TMEM over ALL tiles of the CTA; row C of h^T is 1, so
//                         column C of the accumulator is gb1)
//
// (a) is computed transposed so that an epilogue thread owns ONE hidden unit j (its TMEM lane) and walks
// over pixels (columns): b1 / W2[:, j] are per-thread constants, gW2[:, j] = sum_px gelu(pre) * dout is
// a private register accumulator for the CTA's whole lifetime (no cross-lane reduction).  dpre is
// needed in both orientations and kind::tf32 only takes K-major operands:
//   * [j][px] for (c) never leaves tensor memory: the epilogue writes dpre hi / lo back (tcgen05.st)
//     over the pre^T tile it just read -- lane = row, K along columns is exactly the layout
//     of an A operand in TMEM (tools/ubench/umma_tmemA_probe.cu) -- and (c) runs with A from TMEM;
//   * [px][j] for (b) goes to shared memory with bank-skewed 4-byte stores (LBO = 144 B).
// M = 64 puts D row i in TMEM lane 32 * (i / 16) + i % 16 (tools/ubench/umma_m64_probe.cu,
// profiles/r1_g_umma_m64_layout_probe.txt).
//
// The kernel is bound by the shared-memory pipe (MMA operand fetches + staging stores share it;
// profiles/r1_h): every byte that stays in TMEM or is not restaged counts.
//
// Warp roles (persistent CTA, one per SM): 16 epilogue warps (4 lane quadrants x 4 pixel quarters),
// 1 MMA-issue warp, 6 loader warps (global -> split -> operand buffers); the dh accumulator is drained to
// global memory by the epilogue warps in rotation.  mbarrier hand-offs; operand slots, the pre^T / dpre^T tile and the dh
// accumulator are double-buffered so the (a) MMAs of tile i+1 run under the GELU epilogue of tile i.
#include "common.cuh"
#include "tc_common.cuh"

namespace fno {
namespace {

constexpr int BT_PX = 64;            // pixels per tile
constexpr int BT_HID = 128;
constexpr int BT_KC = 24;            // padded channels: K of (a), N of (b); C + 1 <= 24
constexpr int BT_NC = 32;            // N of (c)  (M = 128 needs N % 16 == 0)
constexpr int BT_GV = 8;             // floats per pixel of a staged dout tile / per-variable record stride (V <= 8)
constexpr int BT_EPI_WARPS = 16;
constexpr int BT_LD_WARPS = 6;
constexpr int BT_MMA_WARP = BT_EPI_WARPS;
constexpr int BT_LD_WARP0 = BT_EPI_WARPS + 1;
constexpr int BT_THREADS = 32 * (BT_EPI_WARPS + 1 + BT_LD_WARPS);   // 736

// operand buffers (bytes); every shared-memory operand is K-major, 8-row x 16-byte core matrices
constexpr int AW1_SBO = 6 * 128, AW1_BYTES = 16 * AW1_SBO;          // W1   [j 128][k 24]
constexpr int B2_SBO = 32 * 128, B2_BYTES = 3 * B2_SBO;             // W1^T [c 24][j 128]
constexpr int BH_SBO = 6 * 128, BH_BYTES = 8 * BH_SBO;              // h    [px 64][k 24]       x 2 slots
constexpr int B3_LBO = 144, B3_SBO = 16 * B3_LBO, B3_BYTES = 4 * B3_SBO;   // h^T  [c 32][px 64]  x 2 slots
constexpr int A2_LBO = 144, A2_SBO = 32 * A2_LBO, A2_BYTES = 8 * A2_SBO;   // dpre [px 64][j 128]
constexpr int GT_BYTES = 2 * BT_PX * BT_GV * 4;                     // dout * std, two slots
constexpr int BT_OPER_BYTES = 2 * (AW1_BYTES + B2_BYTES + 2 * BH_BYTES + 2 * B3_BYTES + A2_BYTES) + GT_BYTES;
constexpr int BT_NBARS = 17;
constexpr int BT_SMEM = BT_OPER_BYTES + BT_NBARS * 8 + 16;

// TMEM columns (512 allocated: the CTA owns its SM)
constexpr unsigned TM_D1 = 0;        // 2 slots x 128: [pre^T, then dpre^T hi | dpre^T lo]
constexpr unsigned TM_D2 = 256;      // 2 slots x 32: dh tile
constexpr unsigned TM_D3 = 320;      // 32: gW1 | gb1, accumulated over the CTA's lifetime
constexpr unsigned TM_COLS = 512;

// per-CTA partial record (floats): gW1|gb1 [128][32], gW2 [4 quarters][4][128], gb2 [2 warps][4] (padded to 64 x 4)
constexpr int REC_W1 = 0, REC_W2 = BT_HID * BT_NC, REC_B2 = REC_W2 + 4 * BT_GV * BT_HID;
constexpr int REC_LEN = REC_B2 + BT_PX * BT_GV;

#ifdef FNO_TRACE
__device__ long long g_trace[16 * 32];
#define TRACE(slot) do { if (blockIdx.x == 0 && lane == 0 && it >= 8 && it < 24) g_trace[(it - 8) * 32 + (slot)] = clock64(); } while (0)
#else
#define TRACE(slot) do { } while (0)
#endif

struct BtGeo {
  int R_in, W_in, R_out, Wp;
  long npix, plane;
  FastDiv by_w, by_tps;
};

template <int VP>
__global__ void __launch_bounds__(BT_THREADS, 1)
head_bwd_tc_kernel(const float* __restrict__ h, const float* __restrict__ dout, const float* __restrict__ W1,
                   const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ stats,
                   float* __restrict__ dh, float* __restrict__ rec, BtGeo g, int C, int V, int tiles_per_sample,
                   int total_tiles, int single) {
  FNO_SPLIT_CONSTS(single);                  // single: 0 = 3xTF32 (fp32 mode), 1 = tf32, 2 = bf16 operands
  extern __shared__ __align__(128) unsigned char bsm[];
  unsigned char* aw1_hi = bsm;
  unsigned char* aw1_lo = aw1_hi + AW1_BYTES;
  unsigned char* b2_hi = aw1_lo + AW1_BYTES;
  unsigned char* b2_lo = b2_hi + B2_BYTES;
  unsigned char* bh_hi = b2_lo + B2_BYTES;            // [2 slots]
  unsigned char* bh_lo = bh_hi + 2 * BH_BYTES;
  unsigned char* b3_hi = bh_lo + 2 * BH_BYTES;        // [2 slots]
  unsigned char* b3_lo = b3_hi + 2 * B3_BYTES;
  unsigned char* a2_hi = b3_lo + 2 * B3_BYTES;
  unsigned char* a2_lo = a2_hi + A2_BYTES;
  float4* gt = reinterpret_cast<float4*>(a2_lo + A2_BYTES);          // [2][32 pixel pairs][8 variables][2] dout * std
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(bsm + BT_OPER_BYTES);
  unsigned long long* bh_ready = bars;        // [2] loaders -> MMA, epilogue: h tile (a) + dout tile staged
  unsigned long long* bh_free = bars + 2;     // [2] MMA (a) done -> loaders
  unsigned long long* b3_ready = bars + 4;    // [2] loaders -> MMA: h^T tile staged for (c)
  unsigned long long* d2_full = bars + 6;     // [2] MMA (b), (c) done: h^T slot free
  unsigned long long* d2_free = bars + 8;     // [2] dh accumulator drained
  unsigned long long* g_free = bars + 10;     // [2] dout tile consumed by the epilogue
  unsigned long long* d1_full = bars + 12;    // [2] MMA (a) done: pre^T ready
  unsigned long long* a23_ready = bars + 14;  // epilogue -> MMA: dpre staged (TMEM hi / lo + shared [px][j])
  unsigned long long* b_done = bars + 15;     // MMA (b) done: the shared dpre buffer is free, the dh accumulator full
  unsigned long long* c_done = bars + 16;     // MMA (c) of the CTA's last tile done: gW1 | gb1 complete (one phase)
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + BT_NBARS);

  // the shuffle makes the warp index provably warp-uniform: role branches are then non-divergent for the
  // compiler and the MMA warp's code runs on the uniform datapath (back-to-back UTCHMMA)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  for (int i = tid; i < BT_OPER_BYTES / 16; i += BT_THREADS) reinterpret_cast<float4*>(bsm)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(bh_ready + s, BT_LD_WARPS);
      mbar_init(bh_free + s, 1);
      mbar_init(b3_ready + s, BT_LD_WARPS);
      mbar_init(d2_full + s, 1);
      mbar_init(d2_free + s, 4);
      mbar_init(g_free + s, BT_EPI_WARPS);
      mbar_init(d1_full + s, 1);
    }
    mbar_init(a23_ready, BT_EPI_WARPS);
    mbar_init(b_done, 1);
    mbar_init(c_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == BT_MMA_WARP) tmem_alloc(tmem_slot, TM_COLS);
  __syncthreads();
  // constant operands: W1 (+ b1 in column C) as A of (a), W1^T as B of (b)
  for (int i = tid; i < BT_HID * BT_KC; i += BT_THREADS) {
    const int j = i / BT_KC, k = i - j * BT_KC;
    float hi = 0.f, lo = 0.f;
    if (k < C) split_rm(__ldg(W1 + (size_t)j * C + k), hi, lo, sp_rnd, sp_msk);
    else if (k == C) split_rm(__ldg(b1 + j), hi, lo, sp_rnd, sp_msk);
    const int off = (j & 7) * 16 + (j >> 3) * AW1_SBO + (k >> 2) * 128 + (k & 3) * 4;
    *reinterpret_cast<float*>(aw1_hi + off) = hi;
    *reinterpret_cast<float*>(aw1_lo + off) = lo;
    if (k < C) {
      const int off2 = (k & 7) * 16 + (k >> 3) * B2_SBO + (j >> 2) * 128 + (j & 3) * 4;
      *reinterpret_cast<float*>(b2_hi + off2) = hi;
      *reinterpret_cast<float*>(b2_lo + off2) = lo;
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const int ntl = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA
  float* __restrict__ myrec = rec + (size_t)blockIdx.x * REC_LEN;

  if (warp == BT_MMA_WARP) {
    // ---- MMA issuer: the whole warp stays converged, one elected lane issues (tc_common.cuh) ----------
    constexpr unsigned idesc_a = umma_idesc_tf32(BT_HID, BT_PX, 0, 0);
    constexpr unsigned idesc_b = umma_idesc_tf32(BT_PX, BT_KC, 0, 0);
    constexpr unsigned idesc_c = umma_idesc_tf32(BT_HID, BT_NC, 0, 0);
    // the operand buffers never move: descriptors are built once, a K step / slot only adds to the address field
    const unsigned long long d_aw1_h = umma_desc(aw1_hi, 128, AW1_SBO), d_aw1_l = umma_desc(aw1_lo, 128, AW1_SBO);
    const unsigned long long d_bh_h = umma_desc(bh_hi, 128, BH_SBO), d_bh_l = umma_desc(bh_lo, 128, BH_SBO);
    const unsigned long long d_a2_h = umma_desc(a2_hi, A2_LBO, A2_SBO), d_a2_l = umma_desc(a2_lo, A2_LBO, A2_SBO);
    const unsigned long long d_b2_h = umma_desc(b2_hi, 128, B2_SBO), d_b2_l = umma_desc(b2_lo, 128, B2_SBO);
    const unsigned long long d_b3_h = umma_desc(b3_hi, B3_LBO, B3_SBO), d_b3_l = umma_desc(b3_lo, B3_LBO, B3_SBO);
    auto issue_a = [&](int it) {
      const int s = it & 1;
      mbar_wait(bh_ready + s, ((unsigned)it >> 1) & 1u);
      tc_fence_after();
      __syncwarp();
      TRACE(0);
      // slot s of D1 was last read by the (c) MMAs of tile it-2, issued earlier by this thread: in order
      const unsigned d = tmem_base + TM_D1 + (unsigned)s * 128u;
      const unsigned long long so = (unsigned long long)(s * (BH_BYTES >> 4));
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)              // lo*hi, hi*lo, hi*hi
#pragma unroll
        for (int ks = 0; ks < BT_KC / 8; ++ks)
          if (pass == 2 || !single)                     // tf32 mode: the hi*hi pass alone
            tc_mma_tf32_elect(d, (pass == 0 ? d_aw1_l : d_aw1_h) + (unsigned long long)(ks * (256 >> 4)),
                              (pass == 1 ? d_bh_l : d_bh_h) + so + (unsigned long long)(ks * (256 >> 4)), idesc_a,
                              single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      tc_commit_elect(d1_full + s);
      tc_commit_elect(bh_free + s);
    };
    auto issue_bc = [&](int it) {
      const int s = it & 1;
      mbar_wait(a23_ready, (unsigned)it & 1u);
      mbar_wait(b3_ready + s, ((unsigned)it >> 1) & 1u);
      mbar_wait(d2_free + s, (((unsigned)it >> 1) & 1u) ^ 1u);
      tc_fence_after();
      __syncwarp();
      TRACE(1);
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int ks = 0; ks < BT_HID / 8; ++ks)
          if (pass == 2 || !single)
            tc_mma_tf32_elect(tmem_base + TM_D2 + (unsigned)(s * 32), (pass == 0 ? d_a2_l : d_a2_h) + (unsigned long long)(ks * (2 * A2_LBO >> 4)),
                              (pass == 1 ? d_b2_l : d_b2_h) + (unsigned long long)(ks * (256 >> 4)), idesc_b,
                              single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0));
      // (b) alone reads the shared dpre buffer and writes the dh accumulator: the epilogue need not wait for (c)
      tc_commit_elect(b_done);
      const unsigned long long so = (unsigned long long)(s * (B3_BYTES >> 4));
      const unsigned at = tmem_base + TM_D1 + (unsigned)s * 128u;       // dpre^T hi at +0, lo at +64
#pragma unroll
      for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int ks = 0; ks < BT_PX / 8; ++ks)
          if (pass == 2 || !single)
            tc_mma_tf32_ts_elect(tmem_base + TM_D3, at + (unsigned)((pass == 0 ? 64 : 0) + ks * 8),
                                 (pass == 1 ? d_b3_l : d_b3_h) + so + (unsigned long long)(ks * (2 * B3_LBO >> 4)), idesc_c,
                                 (single ? (unsigned)(ks != 0) : (unsigned)((pass | ks) != 0)) | (unsigned)(it > 0));
      tc_commit_elect(d2_full + s);
      if (it == ntl - 1) tc_commit_elect(c_done);
      TRACE(2);
    };
    issue_a(0);
    for (int it = 0; it < ntl; ++it) {
      if (it + 1 < ntl) issue_a(it + 1);
      issue_bc(it);
    }
  } else if (warp < BT_EPI_WARPS) {
    // ---- epilogue: thread = hidden unit j (TMEM lane), 16 pixels (columns) of the tile ----------------
    const int quad = warp & 3, colq = warp >> 2;
    const int j = quad * 32 + lane;
    float w2r[VP];
    float2 aw2[VP];                                      // gW2[v][j] over the even / odd pixels of each pair
#pragma unroll
    for (int v = 0; v < VP; ++v) {
      w2r[v] = (v < V) ? __ldg(W2 + (size_t)v * BT_HID + j) : 0.f;
      aw2[v] = f32x2(0.f);
    }
    const int a2off = (2 * colq) * A2_SBO + (j >> 2) * A2_LBO + (j & 3) * 4;
    // dh tile of tile `t` (accumulator slot t & 1): D2 row i lives in lane 32 (i / 16) + i % 16, so the drain
    // needs one warp per lane quadrant; the duty rotates over the four pixel-quarter groups (tile t is drained
    // by the warps with colq == t % 4) so that it costs every epilogue warp the same ~5 %.  A loader warp is a
    // single dependent instruction stream and was the kernel's bottleneck when it also carried the drain.
    const int npix = (int)g.npix;
    const size_t sample_stride = (size_t)C * g.plane;
    auto drain_dh = [&](int t) {
      const int s = t & 1;
      tc_fence_after();
      const unsigned ta = tmem_base + ((unsigned)(quad * 32) << 16) + TM_D2 + (unsigned)(s * 32);
      const int tile = (int)blockIdx.x + t * (int)gridDim.x;
      const int b = (int)g.by_tps.div((unsigned)tile);
      const int p = (tile - b * tiles_per_sample) * BT_PX + 16 * quad + lane;
      const bool ok = lane < 16 && p < npix;
      const int row = (int)g.by_w.div((unsigned)(ok ? p : 0));
      float* __restrict__ dp = dh + (size_t)b * sample_stride + (size_t)(row * g.Wp + ((ok ? p : 0) - row * g.W_in));
#pragma unroll
      for (int c0 = 0; c0 < BT_KC; c0 += 8) {
        float v[8];
        tmem_ld8(ta + (unsigned)c0, v);
        if (c0 + 8 == BT_KC) {                     // accumulator fully read
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(d2_free + s);
        }
        if (ok) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            if (c0 + c < C) *dp = v[c];
            dp += g.plane;
          }
        }
      }
    };
    for (int it = 0; it < ntl; ++it) {
      const int s = it & 1;
      const unsigned ph = ((unsigned)it >> 1) & 1u;
      mbar_wait(bh_ready + s, ph);                       // dout tile
      mbar_wait(d1_full + s, ph);
      tc_fence_after();
      if (warp == 0) TRACE(8);
      const unsigned tq = tmem_base + ((unsigned)(quad * 32) << 16) + TM_D1 + (unsigned)(s * 128 + 16 * colq);
      float pre[16];
      tmem_ld16(tq, pre);
      float hi[16], lo[16];
      const float4* __restrict__ gq = gt + (s * BT_PX + 16 * colq) * (BT_GV / 4);
      // pixel pairs on the packed f32x2 pipe; the dout tile holds (pixel p, pixel p+1) pairs per variable
#pragma unroll
      for (int p = 0; p < 16; p += 2) {
        float2 gl, gp;
        gelu_fast_both2(make_float2(pre[p], pre[p + 1]), gl, gp);
        float2 da;
#pragma unroll
        for (int q = 0; q < VP / 2; ++q) {
          const float4 go = gq[(p / 2) * (BT_GV / 2) + q];   // variables 2q, 2q+1 of both pixels (warp-wide broadcast)
          const float2 g0 = make_float2(go.x, go.y), g1 = make_float2(go.z, go.w);
          da = q == 0 ? __fmul2_rn(f32x2(w2r[0]), g0) : __ffma2_rn(f32x2(w2r[2 * q]), g0, da);
          da = __ffma2_rn(f32x2(w2r[2 * q + 1]), g1, da);
          aw2[2 * q] = __ffma2_rn(gl, g0, aw2[2 * q]);
          aw2[2 * q + 1] = __ffma2_rn(gl, g1, aw2[2 * q + 1]);
        }
        const float2 dp = __fmul2_rn(da, gp);
        split_rm(dp.x, hi[p], lo[p], sp_rnd, sp_msk);
        split_rm(dp.y, hi[p + 1], lo[p + 1], sp_rnd, sp_msk);
      }
      // dpre^T for (c) goes back into tensor memory, over the pre^T values this thread just read
      tmem_st16(tq, hi);
      if (!single) tmem_st16(tq + 64u, lo);
      __syncwarp();
      if (lane == 0) mbar_arrive(g_free + s);
      if (warp == 0) TRACE(9);
      // the shared dpre buffer was last read by the (b) MMAs of the previous tile
      mbar_wait(b_done, ((unsigned)it & 1u) ^ 1u);
      if (warp == 0) TRACE(10);
#pragma unroll
      for (int p = 0; p < 16; ++p) {
        const int off = a2off + (p & 7) * 16 + (p >> 3) * A2_SBO;
        *reinterpret_cast<float*>(a2_hi + off) = hi[p];
        if (!single) *reinterpret_cast<float*>(a2_lo + off) = lo[p];
      }
      tmem_st_wait();
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a23_ready);
      if (warp == 0) TRACE(11);
      // (b) of tile it-1 is done (b_done above): its dh accumulator is complete
      if (it > 0 && colq == ((it - 1) & 3)) drain_dh(it - 1);
    }
    if (colq == ((ntl - 1) & 3)) {
      mbar_wait(b_done, (unsigned)(ntl - 1) & 1u);
      drain_dh(ntl - 1);
    }
    // partial records: gW2 share of this pixel quarter; the gW1 | gb1 accumulator (quarter 0 warps)
#pragma unroll
    for (int v = 0; v < BT_GV; ++v)
      myrec[REC_W2 + (colq * BT_GV + v) * BT_HID + j] = (v < VP) ? aw2[v < VP ? v : 0].x + aw2[v < VP ? v : 0].y : 0.f;
    if (colq == 0) {
      mbar_wait(c_done, 0u);
      tc_fence_after();
      float acc[32];
      tmem_ld32(tmem_base + ((unsigned)(quad * 32) << 16) + TM_D3, acc);
#pragma unroll
      for (int c = 0; c < 32; c += 4)
        *reinterpret_cast<float4*>(myrec + REC_W1 + j * BT_NC + c) = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
    }
  } else {
    // ---- loaders: global -> split -> operand buffers -------------------------------------------------
    // A loader warp is a single dependent instruction stream whose shared-memory stores queue behind the
    // epilogue's, so its work is ordered by urgency and runs a tile ahead: per iteration the (a) operands of
    // tile it+1 (their slot is free as soon as the (a) MMAs of tile it-1 are done), then h^T of tile it+1 (its
    // slot is free when the (c) MMAs of tile it-1 are done), then the global loads of tile it+3.
    const int lt = tid - BT_LD_WARP0 * 32;
    const int lw = lt >> 5;
    const int px = lt & (BT_PX - 1);
    const int kq = lt >> 6;                        // stages the 4-channel chunks kq and kq + 3
    const int npix = (int)g.npix;
    const size_t sample_stride = (size_t)C * g.plane;
    constexpr int GV = VP > 4 ? 8 : 4;           // variables carried by this instantiation's loaders
    float gb2[GV];
#pragma unroll
    for (int v = 0; v < GV; ++v) gb2[v] = 0.f;
    struct Raw { float x[2][4]; float go[GV]; float sd[GV]; bool valid; };
    // Loads only: nothing in load_raw may USE a loaded value (the warp would sit out the whole DRAM latency
    // there); masking and the dout * std product happen one iteration later, at staging time.  Every load is
    // executed, from a clamped in-range address (no branches, no per-element 64-bit address rebuilds).
    unsigned choff[2][4];                          // channel offsets of this thread's 8 elements (clamped to C - 1)
    unsigned creal = 0, cone = 0;                  // bit 4u+e: a real channel / the ones column C (bias, gb1)
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 4 * (kq + 3 * u) + e;
        choff[u][e] = (unsigned)(c < C ? c : C - 1) * (unsigned)g.plane;
        creal |= (c < C ? 1u : 0u) << (4 * u + e);
        cone |= (c == C ? 1u : 0u) << (4 * u + e);
      }
    auto load_raw = [&](Raw& r, int it) {
      if (lw == 0) TRACE(26);
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const bool in = it < ntl;
      const int b = in ? (int)g.by_tps.div((unsigned)tile) : 0;
      const int p0 = (tile - b * tiles_per_sample) * BT_PX + px;
      r.valid = in && p0 < npix;
      const int p = r.valid ? p0 : 0;
      const int row = (int)g.by_w.div((unsigned)p);
      const float* __restrict__ hp = h + (size_t)b * sample_stride + (size_t)(row * g.Wp + (p - row * g.W_in));
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) r.x[u][e] = __ldg(hp + choff[u][e]);
      if (kq == 0) {
        const float* __restrict__ sd = stats + (size_t)b * 2 * V + V;
        const float* __restrict__ op = dout + ((size_t)b * npix + p) * V;
#pragma unroll
        for (int v = 0; v < GV; ++v) {
          const int vc = v < V ? v : V - 1;
          r.go[v] = __ldg(op + vc);
          r.sd[v] = __ldg(sd + vc);
        }
      }
      if (lw == 0) TRACE(27);
    };
    // masked / padded channel values of a raw set
    auto chan = [&](const Raw& r, int u, int e) -> float {
      return ((creal >> (4 * u + e)) & 1u) ? (r.valid ? r.x[u][e] : 0.f) : (((cone >> (4 * u + e)) & 1u) ? 1.f : 0.f);
    };
    // operands of (a) for tile `it`: h [px][c] hi / lo, dout * std
    auto stage_a = [&](const Raw& r, int it) {
      const int s = it & 1;
      const unsigned phf = (((unsigned)it >> 1) & 1u) ^ 1u;     // the previous use of slot s
      float hi[2][4], lo[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) split_rm(chan(r, u, e), hi[u][e], lo[u][e], sp_rnd, sp_msk);
      if (lw == 0) TRACE(16);
      mbar_wait(bh_free + s, phf);
      if (lw == 0) TRACE(17);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int off = s * BH_BYTES + (px & 7) * 16 + (px >> 3) * BH_SBO + (kq + 3 * u) * 128;
        *reinterpret_cast<float4*>(bh_hi + off) = make_float4(hi[u][0], hi[u][1], hi[u][2], hi[u][3]);
        if (!single) *reinterpret_cast<float4*>(bh_lo + off) = make_float4(lo[u][0], lo[u][1], lo[u][2], lo[u][3]);
      }
      if (kq == 0) {
        mbar_wait(g_free + s, phf);
        float go[GV];
#pragma unroll
        for (int v = 0; v < GV; ++v) {
          go[v] = (r.valid && v < V) ? r.go[v] * r.sd[v] : 0.f;
          gb2[v] += go[v];
        }
        // pixel-pair layout [pair][variable][pixel of the pair]: the even lane of a pair stores variables 4r, 4r+1, the
        // odd lane 4r+2, 4r+3, each after one exchange with its partner
        const bool odd = px & 1;
#pragma unroll
        for (int r = 0; r < GV / 4; ++r) {
          const float a = __shfl_xor_sync(0xffffffffu, odd ? go[4 * r] : go[4 * r + 2], 1);
          const float c = __shfl_xor_sync(0xffffffffu, odd ? go[4 * r + 1] : go[4 * r + 3], 1);
          gt[(s * BT_PX + px - odd) * (BT_GV / 4) + 2 * r + odd] = odd ? make_float4(a, go[4 * r + 2], c, go[4 * r + 3])
                                                               : make_float4(go[4 * r], a, go[4 * r + 1], c);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bh_ready + s);
      if (lw == 0) TRACE(18);
    };
    // h^T of tile `it` for (c): its slot is free once the (b), (c) MMAs of tile it-2 are done
    auto stage_c = [&](const Raw& r, int it) {
      const int s = it & 1;
      float hi[2][4], lo[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) split_rm(chan(r, u, e), hi[u][e], lo[u][e], sp_rnd, sp_msk);
      mbar_wait(d2_full + s, (((unsigned)it >> 1) & 1u) ^ 1u);
      if (lw == 0) TRACE(19);
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int c = 4 * (kq + 3 * u) + e;
          const int off = s * B3_BYTES + (c & 7) * 16 + (c >> 3) * B3_SBO + (px >> 2) * B3_LBO + (px & 3) * 4;
          *reinterpret_cast<float*>(b3_hi + off) = hi[u][e];
          if (!single) *reinterpret_cast<float*>(b3_lo + off) = lo[u][e];
        }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(b3_ready + s);
      if (lw == 0) TRACE(20);
    };
    Raw ra, rb;
    load_raw(ra, 0);
    load_raw(rb, 1);
    stage_a(ra, 0);
    stage_c(ra, 0);
    load_raw(ra, 2);
    // iteration `it` works on tile it+1 (raw set rb for even it, ra for odd it)
    for (int it = 0; it < ntl; it += 2) {
      if (it + 1 < ntl) {
        stage_a(rb, it + 1);
        stage_c(rb, it + 1);
      }
      load_raw(rb, it + 3);
      if (it + 2 < ntl) {
        stage_a(ra, it + 2);
        stage_c(ra, it + 2);
      }
      load_raw(ra, it + 4);
    }
    if (kq == 0) {                                  // gb2: the two dout-staging warps reduce over their 32 pixels each
#pragma unroll
      for (int v = 0; v < BT_GV; ++v) {
        float t = v < GV ? gb2[v < GV ? v : 0] : 0.f;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (lane == 0) myrec[REC_B2 + lw * BT_GV + v] = t;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == BT_MMA_WARP) tmem_dealloc(tmem_base, TM_COLS);
}

}  // namespace

size_t head_bwd_tc_workspace_bytes() { return sizeof(float) * (size_t)148 * REC_LEN; }

}  // namespace fno

using namespace fno;

#ifdef FNO_TRACE
extern "C" int fno_debug_trace(long long* out) {
  return cudaMemcpyFromSymbol(out, g_trace, sizeof(long long) * 16 * 32) == cudaSuccess ? 0 : -1;
}
#endif

extern "C" int fno_head_bwd_tc(const float* h, const float* dout, const float* W1, const float* b1, const float* W2,
                               const float* stats, float* dh, float* gW1, float* gb1, float* gW2, float* gb2, void* work,
                               int B, int R_in, int W_in, int R_out, int Wp, int C, int HID, int V,
                               fno_stream_t stream) {
  if (!h || !dout || !W1 || !b1 || !W2 || !stats || !dh || !gW1 || !gb1 || !gW2 || !gb2 || !work || B <= 0 || R_in <= 0 ||
      W_in <= 0 || R_out < R_in || Wp < W_in) {
    set_error("fno_head_bwd_tc: bad argument");
    return FNO_E_ARG;
  }
  if (HID != BT_HID || C < 1 || C + 1 > BT_KC || V < 1 || V > BT_GV) {
    set_error("fno_head_bwd_tc: supports hidden width 128, C <= %d, V <= %d (got %d, %d, %d)", BT_KC - 1, BT_GV, HID, C, V);
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = head_pad_zero(dh, R_in, W_in, R_out, Wp, (long)B * C, st);
  if (rc != FNO_OK) return rc;
  BtGeo g;
  g.R_in = R_in; g.W_in = W_in; g.R_out = R_out; g.Wp = Wp;
  g.npix = (long)R_in * W_in;
  g.plane = (long)R_out * Wp;
  if (g.npix > 0x3fffffffL) { set_error("fno_head_bwd_tc: plane too large"); return FNO_E_ARG; }
  const long tps = (g.npix + BT_PX - 1) / BT_PX;
  const long total = tps * B;
  if (total > 0x7fffffffL) { set_error("fno_head_bwd_tc: too many tiles"); return FNO_E_ARG; }
  g.by_w.init((unsigned)W_in);
  g.by_tps.init((unsigned)tps);
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(head_bwd_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM) != cudaSuccess ||
        cudaFuncSetAttribute(head_bwd_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM) != cudaSuccess ||
        cudaFuncSetAttribute(head_bwd_tc_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_bwd_tc)");
    done.mark();
  }
  const int ctas = (int)(total < 148 ? total : 148);
  float* rec = static_cast<float*>(work);
  const int single = g_math_mode.load();
  if (V <= 2)
    head_bwd_tc_kernel<2><<<ctas, BT_THREADS, BT_SMEM, st>>>(h, dout, W1, b1, W2, stats, dh, rec, g, C, V, (int)tps, (int)total, single);
  else if (V <= 4)
    head_bwd_tc_kernel<4><<<ctas, BT_THREADS, BT_SMEM, st>>>(h, dout, W1, b1, W2, stats, dh, rec, g, C, V, (int)tps, (int)total, single);
  else
    head_bwd_tc_kernel<8><<<ctas, BT_THREADS, BT_SMEM, st>>>(h, dout, W1, b1, W2, stats, dh, rec, g, C, V, (int)tps, (int)total, single);
  count_launch();
  rc = check_launch("head_bwd_tc_kernel");
  if (rc != FNO_OK) return rc;
  // gW1 [128][C], gb1 [128] (column C of the gW1 rows), gW2 [V][128] summed over 4 copies, gb2 [V] over 2
  ReduceSegs segs;
  segs.s[0] = {gW1, BT_HID * C, REC_W1, C, BT_NC};
  segs.s[1] = {gb1, BT_HID, REC_W1 + C, 1, BT_NC};
  segs.s[2] = {gW2, V * BT_HID, REC_W2, 0, 0, 4, BT_GV * BT_HID};
  segs.s[3] = {gb2, V, REC_B2, 0, 0, 2, BT_GV};
  return launch_partial_reduce(rec, ctas, REC_LEN, segs, st);
}
