// K3 on the tensor cores with the 1x1-conv bypass folded into the same GEMM (fno/fno.py:161-164: x1 = conv(x),
// x2 = w(x), x = gelu(x1 + x2)) and, as its adjoint, the data gradient of a Fourier layer (K3 of gX plus W^T dS).
//
// For one row (b, h) of the padded plane the pre-activation of ALL output channels is ONE GEMM
//
//   s[w, co] = sum_q' F[w, q'] T2[b, co, h, q']  +  sum_ci a[b, ci, h, w] Wl[co, ci]  +  bias[co]
//
//   M = 128 (w: TMEM lane), N = channels, K = 2*m2 (contiguous-axis inverse DFT) + C + 1 (bypass + bias)
//
// whose A operand lives in TENSOR memory: the twiddle columns F = [cos | sin](2 pi q w / W) are written once per
// CTA, the activation columns a[b, :, h, w] are loaded straight from HBM by converter warps (lane = w: one
// coalesced 128-byte request per channel row), split hi / lo in registers (3xTF32: fp32-mode accuracy) and
// stored with tcgen05.st; the bias rides on a constant-one column.  The B operand [T2(b, h) ; Wl] sits in
// shared memory: Wl (hi / lo) once per CTA, the 2.3 KB T2 tile of the row re-split per tile by one warp.
// T2 = strided-axis inverse of the mixed spectrum (130 x 24 reals per plane instead of 130 x 130) is produced
// by hinv_tiles_kernel directly in the K-major core-matrix layout of that operand, with the C2R column
// weights, the 1/(HW) scale and the sign of the sine part folded in.  The epilogue reads D[w, co] back with
// tcgen05.ld (thread = w), stores the pre-activation and its exact-erf GELU with one coalesced 128-byte
// store per channel and warp.  The bypass output `lin`, its 173 MB round trip and the separate
// pointwise kernel of round 1 are gone; the activation is read once and each output written once.
//
// The last W - 128 columns of a row (2 for the 130-wide padded planes of cfg 1) do not fit the 128 TMEM lanes; an
// "edge" warp computes them on the FP32 pipes, 32 rows at a time (lane = row), independently of the pipeline.
//
// Pipeline (per CTA, persistent over a contiguous range of rows; every hand-off is an mbarrier):
//   2 B-prep warps   (one per row parity) bulk-copy raw T2 tiles into a 4-deep ring and    raw_full, mma_done -> ready
//                    split them hi / lo into the operand buffers (the proxy fence this needs is why they are
//                    separate warps: it is a MEMBAR that would wait for the converters' prefetched loads)
//   8 converter warps  (lane quadrant x row parity) activation columns -> TMEM with wide     mma_done -> ready
//                    tcgen05.st, 2 own rows of loads in flight
//   MMA warp         18 tcgen05.mma per row into a double-buffered accumulator         ready -> mma_done
//   8 epilogue warps tcgen05.ld, GELU, stores                                          mma_done -> ready
// (`ready[s]` collects the A buffer, the T2 operand tile and the free accumulator of a row: one wait in the MMA warp)
#include <cstdlib>
#include <cstring>

#include "tc_common.cuh"

namespace fno {
namespace {

// -DL2_TRACE: CTA 0 records clock64 at the pipeline hand-offs of its first 64 rows (tools only; off in the product build)
#ifdef L2_TRACE
#define L2TR(ev, it) do { if (p.trace != nullptr && blockIdx.x == 0 && lane == 0 && (it) < 64) p.trace[(it) * 16 + (ev)] = clock64(); } while (0)
#else
#define L2TR(ev, it) do { } while (0)
#endif
#ifdef L2_TRACE
#define L2DBG(bit) (p.dbg & (bit))
#else
#define L2DBG(bit) 0
#endif
constexpr int L2_RMAX = 4;        // edge columns (W - 128) handled on the FP32 pipes
constexpr int L2_NR = 4;          // T2 tiles in flight (bulk copies into a shared-memory ring)
constexpr int L2_NS = 6;          // activation rows in flight with the tensor-map path (3 per row parity)
constexpr int L2_PD = 3;          // own rows of activation copies in flight per converter warp (= 6 rows ahead)

// 2-D tiled TMA: box {Wm pixels, C planes} of the [planes][pixels] view of an activation tensor <-> dense [C][Wm] shared memory
// (loads through tma_load_2d).  The tensor map takes element coordinates, so the 8-byte-aligned rows of the 130-wide planes need
// no special casing.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int c0, int c1, const void* src) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
               ::"l"(map), "r"(c0), "r"(c1), "r"(smem_u32(src))
               : "memory");
}

__device__ __forceinline__ void tmem_st4(unsigned taddr, const float (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                 "r"(__float_as_uint(v[3]))
               : "memory");
}

// arguments for the spectral part of the edge columns w = Wm + j that do not fit the 128 TMEM lanes (W > 128):
//   E[plane, h, j] = Re sum_{r, q} sc_q Y[r, q] e^{+2 pi i (k_r h / H + q w_j / W)} = sum_q' F[w_j, q'] T2[h, q']
struct EdgeArgs {
  float* E;             // [planes][H][RE]
  const float* twW;
  int WP, Wm, RE, r_edge, shift;
};


// ------------------------------------------------------------------------------------------------------
// strided-axis inverse into B-operand tiles:  Z[h, q] = sum_r Y[r, q] e^{+2 pi i k_r h / H}  (k_r signed),
//   T2[(b, h)][n = c][k = q]      =  sc_q Re Z,      T2[..][c][m2 + q] = -sc_q Im Z
// (sc_q = scale * c2r weight).  Frequencies are folded onto j = |k| and rows onto pairs (t, H - t):
//   P_j = Y[+j] + Y[-j], M_j = Y[+j] - Y[-j]:   Re Z = Y0r + sum_j (Pr cos - Mi sin),  Im Z = Y0i + sum_j (Pi cos + Mr sin)
// thread = (channel of an 8-row group, q); the 4 m1 folded coefficients stay in registers.
// tile layout (floats): (c >> 3) * KQ * 8 + (k >> 2) * 32 + (c & 7) * 4 + (k & 3)   [8 x 16-byte core matrices]
// ------------------------------------------------------------------------------------------------------
template <int M1T>
__global__ void __launch_bounds__(256)
hinv_tiles_kernel(const float2* __restrict__ Y, float* __restrict__ T2g, const float* __restrict__ twH, int H, int W,
                  int m1, int m2, int C, int D1, int KQ, int tile_floats, int TL, int cmode, float scale, const EdgeArgs ea) {
  constexpr int JP = ((2 * M1T + 1) + 3) & ~3;
  // one block = (sample, slice of row pairs, 8-channel row group): its part of every operand tile is a contiguous
  // KQ * 32-byte segment, assembled in shared memory (zero padding included) and written out with 16-byte stores.
  // The spectral part of the edge columns (E[plane, h, j] = sum_q' F[w_j, q'] T2[h, q'], W > 128) falls out of the same
  // values: every thread leaves its two terms in shared memory and the write-out phase sums them over q (shared-memory
  // atomics were tried: 12-way contention made the kernel 3x slower).
  extern __shared__ float4 hs4[];
  float* hs = reinterpret_cast<float*>(hs4);
  const int q = threadIdx.x % m2, cl = threadIdx.x / m2;
  const int c = blockIdx.z * 8 + cl;
  const bool active = cl < 8 && c < C;
  const int bd = blockIdx.x;                  // b * D1 + d1
  const int NP = H / 2 + 1;
  const int t0 = blockIdx.y * TL, t1 = (t0 + TL < NP) ? t0 + TL : NP;
  const int seg = KQ * 8;                     // floats of one (row, row group) segment
  const int RE = ea.RE, r_edge = ea.r_edge;
  float* es = hs + 2 * TL * seg;              // [2 TL rows][8 channels][RE][m2] partial edge sums
  for (int i = threadIdx.x; i < 2 * TL * seg / 4; i += blockDim.x) hs4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  if (active) {
    const int b = bd / D1, d1 = bd - b * D1;
    const size_t plane = ((size_t)b * C + c) * D1 + d1;
    const float2* __restrict__ Yp = Y + plane * (size_t)(2 * m1) * m2 + q;
    float PR[M1T + 1], PI[M1T + 1], MR[M1T + 1], MI[M1T + 1];
    const float2 y0 = __ldg(Yp);
#pragma unroll
    for (int j = 1; j <= M1T; ++j) {
      float2 yp = make_float2(0.f, 0.f), yn = make_float2(0.f, 0.f);
      if (j < m1) yp = __ldg(Yp + (size_t)j * m2);
      if (j <= m1) yn = __ldg(Yp + (size_t)(2 * m1 - j) * m2);
      PR[j] = yp.x + yn.x; PI[j] = yp.y + yn.y;
      MR[j] = yp.x - yn.x; MI[j] = yp.y - yn.y;
    }
    float sc = scale;
    if (cmode && q != 0 && !((W & 1) == 0 && 2 * q == W)) sc *= 2.0f;
    // twiddles of this thread's wavenumber at the edge columns: slot u < r_edge -> w = Wm + u; with `shift`,
    // r_edge <= u < 2 r_edge -> w = u - r_edge (rows whose tensor-map window is [r_edge, Wm + r_edge))
    float fc[L2_RMAX], fs[L2_RMAX];
#pragma unroll
    for (int u = 0; u < L2_RMAX; ++u) {
      const int ncol = ea.shift ? 2 * r_edge : r_edge;
      const int wcol = u < r_edge ? ea.Wm + u : u - r_edge;
      fc[u] = (u < ncol) ? __ldg(ea.twW + (size_t)q * ea.WP + wcol) : 0.f;
      fs[u] = (u < ncol) ? __ldg(ea.twW + (size_t)(m2 + q) * ea.WP + wcol) : 0.f;
    }
    const int o_re = (q >> 2) * 32 + cl * 4 + (q & 3), o_im = ((m2 + q) >> 2) * 32 + cl * 4 + ((m2 + q) & 3);
    // all addresses advance by constants per row pair (integer index arithmetic was half of this kernel's instructions)
    float* __restrict__ o = hs;                                  // row t, then its mirror H - t: 2 seg floats per pair
    float* __restrict__ e = es + (size_t)cl * RE * m2 + q;       // [slot][ch][j][q]; the mirror row is 8 RE m2 further
    const int mo = 8 * RE * m2;
    const float4* __restrict__ r4 = reinterpret_cast<const float4*>(twH + (size_t)t0 * JP);
    // with `shift` (W % 4 == 2) a row's column window -- hence its edge column pair -- depends on the parity of the row
    const bool hodd = (H & 1) != 0;
    for (int t = t0; t < t1; ++t, o += 2 * seg, e += 2 * mo, r4 += JP / 4) {
      float tw[JP];
#pragma unroll
      for (int i = 0; i < JP / 4; ++i) {
        const float4 v = __ldg(r4 + i);
        tw[4 * i] = v.x; tw[4 * i + 1] = v.y; tw[4 * i + 2] = v.z; tw[4 * i + 3] = v.w;
      }
      float er = y0.x, ei = y0.y, odr = 0.f, odi = 0.f;
#pragma unroll
      for (int j = 1; j <= M1T; ++j) {
        er = fmaf(PR[j], tw[j], er);
        ei = fmaf(PI[j], tw[j], ei);
        odr = fmaf(MI[j], tw[M1T + j], odr);
        odi = fmaf(MR[j], tw[M1T + j], odi);
      }
      const float a_re = sc * (er - odr), a_im = -sc * (ei + odi);
      const float b_re = sc * (er + odr), b_im = -sc * (ei - odi);
      o[o_re] = a_re;
      o[o_im] = a_im;
      o[seg + o_re] = b_re;
      o[seg + o_im] = b_im;
      if (r_edge > 0) {
        if (ea.shift) {                                        // r_edge <= 2
          const bool sa = (t & 1) != 0, sb = sa != hodd;       // parity of rows t and H - t
          e[0] = fmaf(sa ? fc[2] : fc[0], a_re, (sa ? fs[2] : fs[0]) * a_im);
          e[mo] = fmaf(sb ? fc[2] : fc[0], b_re, (sb ? fs[2] : fs[0]) * b_im);
          if (RE > 1) {
            e[m2] = fmaf(sa ? fc[3] : fc[1], a_re, (sa ? fs[3] : fs[1]) * a_im);
            e[mo + m2] = fmaf(sb ? fc[3] : fc[1], b_re, (sb ? fs[3] : fs[1]) * b_im);
          }
        } else {
#pragma unroll
          for (int j = 0; j < L2_RMAX; ++j) {
            if (j < RE) {
              e[j * m2] = fmaf(fc[j], a_re, fs[j] * a_im);
              e[mo + j * m2] = fmaf(fc[j], b_re, fs[j] * b_im);
            }
          }
        }
      }
    }
  }
  __syncthreads();
  // write-out: thread f copies float4 f of every segment (running pointers: rows t ascend, their mirrors descend)
  const int seg4 = seg / 4;
  if ((int)threadIdx.x < seg4) {
    float* __restrict__ base = T2g + (size_t)bd * H * tile_floats + (size_t)blockIdx.z * seg;
    float4* __restrict__ da = reinterpret_cast<float4*>(base + (size_t)t0 * tile_floats) + threadIdx.x;
    float4* __restrict__ db = reinterpret_cast<float4*>(base + (size_t)(H - t0) * tile_floats) + threadIdx.x;
    const float4* __restrict__ src = hs4 + threadIdx.x;
    const int tf4 = tile_floats / 4;
    for (int t = t0; t < t1; ++t, da += tf4, db -= tf4, src += 2 * seg4) {
      *da = src[0];
      if (t != 0 && 2 * t != H) *db = src[seg4];               // self-paired rows have no mirror
    }
  }
  if (r_edge > 0) {
    // RE is 2 or 4: item i = (slot, channel, j)
    const int lre = RE == 4 ? 2 : 1;
    const int b = bd / D1, d1 = bd - b * D1;
    for (int i = threadIdx.x; i < 2 * (t1 - t0) * 8 * RE; i += blockDim.x) {
      const int j = i & (RE - 1), ch = (i >> lre) & 7, slot = i >> (lre + 3);
      const int t = t0 + (slot >> 1), cc = blockIdx.z * 8 + ch;
      if (cc >= C || ((slot & 1) && (t == 0 || 2 * t == H))) continue;
      const int row = (slot & 1) ? H - t : t;
      const float* __restrict__ pq = es + (size_t)i * m2;
      float sum = 0.f;
      for (int qq = 0; qq < m2; ++qq) sum += pq[qq];
      ea.E[((((size_t)b * C + cc) * D1 + d1) * H + row) * RE + j] = sum;
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------------
template <int KA, int NPAD, int CWQ>
struct L2Cfg {
  static_assert(CWQ == 2, "two converter warps per lane quadrant: one per row parity");
  static constexpr int EW = NPAD / 16;                           // epilogue warps per lane quadrant
  static constexpr int CONV_WARPS = 4 * CWQ;
  static constexpr int EPI_WARP0 = CONV_WARPS;
  static constexpr int EPI_WARPS = 4 * EW;
  static constexpr int MMA_WARP = CONV_WARPS + EPI_WARPS;
  static constexpr int EDGE_WARP = MMA_WARP + 1;
  static constexpr int BPREP_WARP0 = MMA_WARP + 2;               // 2 warps: raw T2 tile -> hi / lo operand buffers
  static constexpr int BPREP_WARPS = 2;
  static constexpr int NFB = NPAD / 4;                           // float4 of a T2 tile per B-prep lane (KQ <= 32)
  static constexpr int THREADS = 32 * (MMA_WARP + 2 + BPREP_WARPS);
  static constexpr unsigned TM_COLS = (4 * 32 + 4 * KA + 2 * NPAD <= 256) ? 256u : 512u;
};

struct L2Args {
  const float* a;       // [B, C, RS, W] activation (forward) / dS (adjoint)
  const float* T2g;     // [B * RS] tiles from hinv_tiles_kernel
  const float* E;       // [B * C * RS][RE] spectral part of the edge columns (hinv_edge_kernel)
  int RE;
  const float* Wl;      // [C, C] bypass weight
  const float* bias;    // [C] or null
  float* s_out;         // optional pre-activation
  float* out;
  const float* twW;     // [2][m2][WP] cos / sin of 2 pi q w / W
  int WP, W, m2, KQ, C, RS;
  int tile_floats;
  long total_tiles;     // B * RS
  int transpose_w, apply_gelu, single;
  int shift;            // tensor-map path, W % 4 == 2: rows with (row * W) % 4 == 2 use the column window [2, 130) (16-byte aligned)
  FastDiv rs_div;
  unsigned long long* trace;
  int dbg;   // L2_TRACE builds only: 1 no epilogue stores, 2 no activation loads, 4 no MMAs, 8 no edge, 16 no STTM, 32 no LDTM
};

template <int V>
struct IC { static constexpr int value = V; };

// waits: the single MMA / producer warps poll (they are the critical path and cost one warp's issue slots), the 16
// converter / epilogue warps park (polling would take the issue slots the working warps of their sub-partition need)
#ifndef L2WAIT_HOT
#define L2WAIT_HOT mbar_wait_spin
#endif
#ifndef L2WAIT_COLD
#define L2WAIT_COLD mbar_wait
#endif

// CX: compile-time width (0 = run-time p.C, every channel loop predicated); GELU / SOUT: epilogue form
//     TMA: activation rows come in and results go out through 2-D tensor maps (one TMA op per row for all channels)
template <int KA, int NPAD, int CWQ, int CX, bool GELU, bool SOUT, bool TMA>
__global__ void __launch_bounds__(L2Cfg<KA, NPAD, CWQ>::THREADS, 1)
layer2d_tc_kernel(const L2Args p, const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_o,
                  const __grid_constant__ CUtensorMap tm_s) {
  using Cfg = L2Cfg<KA, NPAD, CWQ>;
  extern __shared__ __align__(128) unsigned char lsm[];
  const int KQ = p.KQ, W = p.W;
  const int C = CX > 0 ? CX : p.C;
  const int CP = (C + 3) & ~3;
  const int t2_tile = NPAD * KQ;                          // floats of one hi (or lo) T2 operand tile
  float* bT2 = reinterpret_cast<float*>(lsm);             // [2 stages][hi | lo][NPAD * KQ]
  float* bW = bT2 + 4 * t2_tile;                          // [hi | lo][NPAD * KA]
  float* eW = bW + 2 * NPAD * KA;                         // [C][CP] raw weight (edge warp), zero padded rows
  float* eB = eW + C * CP;                                // [NPAD] bias
  float* eF = eB + NPAD;                                  // [L2_RMAX][KQ] twiddles of the edge columns
  float* ring = eF + L2_RMAX * KQ;                        // [L2_NR][tile_floats] raw T2 tiles (bulk-copy destination)
  // activation staging (128-byte aligned): [CONV_WARPS][L2_PD][KA][32] per-warp rows, filled by cp.async or, with tensor
  // maps, by one {32 pixels, C planes} box per warp and row; TMA only: [out | s][2][C][Wm] result boxes
  float* stage = reinterpret_cast<float*>((reinterpret_cast<size_t>(ring + (size_t)L2_NR * p.tile_floats) + 127) & ~size_t(127));
  const int box_floats = ((C * (p.W < 128 ? p.W : 128) + 31) & ~31);
  float* ostage = stage + (size_t)Cfg::CONV_WARPS * L2_PD * KA * 32;
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(
      (reinterpret_cast<size_t>(ostage + (TMA ? (size_t)4 * box_floats : 0)) + 15) & ~size_t(15));
  unsigned long long* ready = bars;                    // [2] everything MMA(row) needs: A buffer s written (4 converter warps), T2
                                                       //     operand tile s staged (1 B-prep warp), accumulator s read back (epilogue)
  unsigned long long* mma_done = bars + 2;             // [2] MMAs of the tile on buffers s complete (A / B free, D full)
  unsigned long long* raw_full = bars + 8;             // [L2_NR] bulk copy of a raw T2 tile landed
  unsigned long long* f_ready = bars + 8 + L2_NR;      // [1] the twiddle columns of A are in tensor memory (once)
  unsigned long long* raw_free = bars + 9 + L2_NR;     // [L2_NR] the B-prep warp has read ring slot
  unsigned long long* act_full = raw_free + L2_NR;     // [CONV_WARPS][L2_PD] TMA: this warp's 32 columns of a row landed
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(act_full + Cfg::CONV_WARPS * L2_PD);

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int Wm = W < 128 ? W : 128;          // columns on the tensor cores
  const int r_edge = W - Wm;                 // columns on the edge warp
  const int m2x2 = 2 * p.m2;
  const unsigned RS = (unsigned)p.RS;
  const size_t cs = (size_t)RS * W;          // channel stride (floats)
  const size_t bs = cs * C;                  // sample stride
  const FastDiv rsd = p.rs_div;
  const long t_begin = (p.total_tiles * (long)blockIdx.x) / (long)gridDim.x;          // total_tiles < 2^32, grid <= 148
  const long t_end = (p.total_tiles * (long)(blockIdx.x + 1)) / (long)gridDim.x;
  const int ntl = (int)(t_end - t_begin);
  const int single = p.single;                 // 0 = 3xTF32 (fp32 mode), 1 = tf32, 2 = bf16 operands
  FNO_SPLIT_CONSTS(single);

  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(ready + s, 4 + 1 + Cfg::EPI_WARPS);  // ONE wait per row in the MMA warp: its serial instruction stream is
      mbar_init(mma_done + s, 1);                    // the pipeline's critical path
    }
    for (int s = 0; s < L2_NR; ++s) mbar_init(raw_full + s, 1);
    mbar_init(f_ready, 4);
    for (int s = 0; s < L2_NR; ++s) mbar_init(raw_free + s, 1);
    for (int s = 0; s < Cfg::CONV_WARPS * L2_PD; ++s) mbar_init(act_full + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == Cfg::MMA_WARP) tmem_alloc(tmem_slot, Cfg::TM_COLS);
  // constant operands: Wl (+ bias row) hi / lo in the K-major core-matrix layout; T2 operand rows beyond the tile's
  // row groups stay zero
  for (int i = tid; i < 4 * t2_tile; i += Cfg::THREADS) bT2[i] = 0.f;
  for (int i = tid; i < NPAD * KA; i += Cfg::THREADS) {
    const int n = i / KA, k = i - n * KA;
    float v = 0.f;
    if (n < C) {
      if (k < C) v = __ldg(p.Wl + (p.transpose_w ? (size_t)k * C + n : (size_t)n * C + k));
      else if (k == C && p.bias != nullptr) v = __ldg(p.bias + n);
    }
    float hi, lo;
    split_rm(v, hi, lo, sp_rnd, sp_msk);
    const int off = (n >> 3) * KA * 8 + (k >> 2) * 32 + (n & 7) * 4 + (k & 3);
    bW[off] = hi;
    bW[NPAD * KA + off] = lo;
  }
  for (int i = tid; i < C * CP; i += Cfg::THREADS) {
    const int n = i / CP, k = i - n * CP;
    eW[i] = (k < C) ? __ldg(p.Wl + (p.transpose_w ? (size_t)k * C + n : (size_t)n * C + k)) : 0.f;
  }
  for (int i = tid; i < NPAD; i += Cfg::THREADS) eB[i] = (i < C && p.bias != nullptr) ? __ldg(p.bias + i) : 0.f;
  for (int i = tid; i < L2_RMAX * KQ; i += Cfg::THREADS) {
    const int j = i / KQ, k = i - j * KQ;
    eF[i] = (j < r_edge && k < m2x2) ? __ldg(p.twW + (size_t)k * p.WP + Wm + j) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  // twiddle sets: [hi | lo] for the column window [0, Wm) and, shifted rows, [2, Wm + 2)
  const unsigned TM_FHI = 0, TM_FLO = (unsigned)KQ, TM_F1 = 2u * KQ, TM_A = 4u * KQ, TM_D = 4u * KQ + 4u * KA;
  const int shift = TMA ? p.shift : 0;

  if (warp < Cfg::CONV_WARPS) {
    // ---- converters: lane = w.  Warp (quadrant, parity) owns ALL bypass columns of its 32 lanes for the rows of its
    // parity, i.e. A buffer s = parity: tcgen05.st costs ~15-30 cycles of the SM's tensor-memory store port per
    // INSTRUCTION whatever its width (48 x4 stores per row made the converters the bottleneck), so a row is written
    // with x16 / x8 stores -- 4 per warp.  L2_PD own rows (2 L2_PD rows ahead) of loads are in flight per thread.
    const int quad = warp & 3, par = warp >> 2;
    const int w = quad * 32 + lane;
    const bool wv = w < Wm;
    const unsigned ta = tmem_base + ((unsigned)(quad * 32) << 16);
    if (par == 0) {
      // twiddle columns, once: F[w, q'] = twW[q'][w]
      for (int set = 0; set <= shift; ++set)
        for (int g = 0; g < KQ / 8; ++g) {
          float hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int k = 8 * g + e;
            const float v = (wv && k < m2x2) ? __ldg(p.twW + (size_t)k * p.WP + w + 2 * set) : 0.f;
            split_rm(v, hi[e], lo[e], sp_rnd, sp_msk);
          }
          tmem_st8(ta + (set ? TM_F1 : 0u) + TM_FHI + 8u * g, hi);
          tmem_st8(ta + (set ? TM_F1 : 0u) + TM_FLO + 8u * g, lo);
        }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(f_ready);
    }
    // activation staging: cp.async (LDGSTS) into a per-warp shared-memory ring, L2_PD own rows (2 L2_PD rows) ahead.
    // Register prefetch does not work here: the loads of the row after next land on the same scoreboard as the ones
    // about to be consumed, so the warp waited a full DRAM latency per row (ncu: long_scoreboard on the first use).
    constexpr int NLD = CX > 0 ? CX : KA - 1;                 // channel slots per thread (C <= KA - 1)
    const float* __restrict__ abase = p.a + w;
    const unsigned ah = ta + TM_A + (unsigned)(par * 2 * KA), al = ah + KA;
    const int s = par;
    float* __restrict__ stg = stage + (size_t)warp * L2_PD * (KA * 32) + lane;      // [L2_PD][KA][32 lanes]
    const unsigned stg_u32 = smem_u32(stg);
    float* __restrict__ wstage = stage + (size_t)warp * L2_PD * (KA * 32);          // this warp's [L2_PD][KA][32]
    const unsigned box_bytes = (unsigned)C * 32u * 4u;
    auto load_tile = [&](int it, int slot) {
      if (TMA) {                                   // one {32 pixels, C planes} box: this warp's columns of row `it`
        if (lane == 0 && it < ntl && !L2DBG(2)) {
          const unsigned T = (unsigned)(t_begin + it);
          const unsigned b = rsd.div(T);
          const unsigned row = T - b * RS;
          unsigned long long* bar = act_full + warp * L2_PD + slot;
          mbar_arrive_expect_tx(bar, box_bytes);
          const unsigned px = row * (unsigned)W;
          tma_load_2d(wstage + (size_t)slot * (KA * 32), &tm_a, (int)(px + (shift ? (px & 3u) : 0u)) + quad * 32,
                      (int)(b * (unsigned)C), bar);
        }
        return;
      }
      if (it < ntl && wv && !L2DBG(2)) {
        const unsigned T = (unsigned)(t_begin + it);
        const unsigned b = rsd.div(T);
        const unsigned row = T - b * RS;
        const float* __restrict__ src = abase + (size_t)b * bs + (size_t)row * W;
        const unsigned dst = stg_u32 + (unsigned)(slot * KA * 32 * 4);
#pragma unroll
        for (int i = 0; i < NLD; ++i) {
          if (i < C) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + (unsigned)(i * 128)), "l"(src) : "memory");
          src += cs;
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto convert_tile = [&](int it, int slot, int use) {
      const unsigned ph = ((unsigned)it >> 1) & 1u;
      float r[NLD];
      if (TMA) {
        if (!L2DBG(2)) L2WAIT_COLD(act_full + warp * L2_PD + slot, (unsigned)use & 1u);
        if (warp == 0) L2TR(1, it);
        const float* __restrict__ sp = wstage + (size_t)slot * (KA * 32) + lane;
#pragma unroll
        for (int i = 0; i < NLD; ++i) r[i] = (wv && i < C) ? sp[i * 32] : 0.f;
        __syncwarp();                              // every lane has read the slot: load_tile below may refill it
        if (warp == 0) L2TR(2, it);
      } else {
        asm volatile("cp.async.wait_group %0;" ::"n"(L2_PD - 1) : "memory");        // this row's copies have landed
        const float* __restrict__ sp = stg + (size_t)slot * (KA * 32);
#pragma unroll
        for (int i = 0; i < NLD; ++i) r[i] = (wv && i < C) ? sp[i * 32] : 0.f;
      }
      L2WAIT_COLD(mma_done + s, ph ^ 1u);          // the MMAs of tile it - 2 no longer read A buffer s
      if (warp == 0) L2TR(0, it);
      tc_fence_after();
      auto column = [&](int col) -> float {         // col is a compile-time constant after unrolling
        return col < NLD ? ((CX == 0 && col == C) ? 1.0f : r[col < NLD ? col : 0]) : (col == C ? 1.0f : 0.f);
      };
#pragma unroll
      for (int c0 = 0; c0 < KA; c0 += 16) {
        if (KA - c0 >= 16) {
          float hi[16], lo[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) split_rm(column(c0 + e), hi[e], lo[e], sp_rnd, sp_msk);
          if (!L2DBG(16)) {
            tmem_st16(ah + (unsigned)c0, hi);
            if (!single) tmem_st16(al + (unsigned)c0, lo);
          }
        } else {
          float hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) split_rm(column(c0 + e), hi[e], lo[e], sp_rnd, sp_msk);
          if (!L2DBG(16)) {
            tmem_st8(ah + (unsigned)c0, hi);
            if (!single) tmem_st8(al + (unsigned)c0, lo);
          }
        }
      }
      if (warp == 0) L2TR(3, it);
      tmem_st_wait();                              // (no fence.proxy.async here: it compiles to MEMBAR.ALL.CTA, which would
      tc_fence_before();                           //  wait for this warp's copies in flight every row)
      __syncwarp();
      if (lane == 0) mbar_arrive(ready + s);
      if (warp == 0) L2TR(5, it);
    };
#pragma unroll
    for (int d = 0; d < L2_PD; ++d) load_tile(par + 2 * d, d);
    // T2 ring copies are issued here too (quadrant 0 of each parity), not by the B-prep warps: their proxy fence is a
    // MEMBAR that waits for the issuing thread's bulk copies in flight
    const unsigned tile_bytes = (unsigned)p.tile_floats * 4u;
    auto issue_t2 = [&](int it) {
      const int rs = it & (L2_NR - 1);
      mbar_arrive_expect_tx(raw_full + rs, tile_bytes);
      bulk_g2s(ring + (size_t)rs * p.tile_floats, p.T2g + (size_t)(t_begin + it) * p.tile_floats, tile_bytes, raw_full + rs);
    };
    if (quad == 0 && lane == 0) {
      if (par < ntl) issue_t2(par);
      if (par + 2 < ntl) issue_t2(par + 2);
    }
    int slot = 0, use = 0;                          // use = how many times this slot has been filled before
    for (int it = par; it < ntl; it += 2) {
      convert_tile(it, slot, use);
      load_tile(it + 2 * L2_PD, slot);
      if (quad == 0 && lane == 0 && it + L2_NR < ntl) {
        L2WAIT_COLD(raw_free + (it & (L2_NR - 1)), ((unsigned)it / L2_NR) & 1u);    // B-prep has read raw tile `it`
        issue_t2(it + L2_NR);
      }
      if (++slot == L2_PD) { slot = 0; ++use; }
    }
  } else if (warp < Cfg::MMA_WARP) {
    // ---- epilogue: thread = w, a slice of the output channels ------------------------------------------
    const int ew = warp - Cfg::EPI_WARP0;
    const int quad = ew & 3, e = ew >> 2;
    const int w = quad * 32 + lane;
    const bool wv = w < Wm;
    if (lane == 0) {                               // both accumulators start out free
      mbar_arrive(ready);
      mbar_arrive(ready + 1);
    }
    auto role = [&](auto Ec) {
      constexpr int E = decltype(Ec)::value;
      const int CPW = (C + Cfg::EW - 1) / Cfg::EW;
      const int c0 = E * CPW;
      const int cn = (C - c0 < CPW) ? (C - c0 > 0 ? C - c0 : 0) : CPW;
      float* __restrict__ obase = p.out + w + (size_t)c0 * cs;
      float* __restrict__ sbase = SOUT ? p.s_out + w + (size_t)c0 * cs : nullptr;
      const unsigned td = tmem_base + ((unsigned)(quad * 32) << 16) + TM_D + (unsigned)c0;
      for (int it = 0; it < ntl; ++it) {
        const int s = it & 1;
        const unsigned ph = ((unsigned)it >> 1) & 1u;
        const unsigned T = (unsigned)(t_begin + it);
        const unsigned b = rsd.div(T);
        const unsigned row = T - b * RS;
        const size_t toff = (size_t)b * bs + (size_t)row * W;
        L2WAIT_COLD(mma_done + s, ph);
        if (ew == 0) L2TR(9, it);
        tc_fence_after();
        float v[16];
        if (!L2DBG(32)) tmem_ld16(td + (unsigned)(s * NPAD), v);
        else { for (int i = 0; i < 16; ++i) v[i] = (float)i; }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ready + s);          // accumulator s is free for row it + 2
        if (ew == 0) L2TR(10, it);
        if (TMA) {
          // results -> dense [C][Wm] boxes in shared memory, one tensor-map store per row and tensor
          float* __restrict__ po = ostage + (size_t)(it & 1) * box_floats + (size_t)c0 * Wm + w;
          float* __restrict__ ps = po + 2 * box_floats;
          if (wv && !L2DBG(1)) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (i < cn) {
                const float x = v[i];
                if (SOUT) ps[i * Wm] = x;
                po[i * Wm] = GELU ? gelu_fast(x) : x;
              }
            }
          }
          fence_proxy_async();                       // staging stores -> visible to the TMA engine
          const bool issuer = (ew == 0 && lane == 0);
          if (issuer) bulk_wait_read<0>();           // the store of row it - 1 has read its boxes: row it + 1 may overwrite them
          named_bar_sync(1, Cfg::EPI_WARPS * 32);
          if (issuer && !L2DBG(1)) {
            const unsigned px = row * (unsigned)W;
            const int c0x = (int)(px + (shift ? (px & 3u) : 0u));
            tma_store_2d(&tm_o, c0x, (int)(b * (unsigned)C), ostage + (size_t)(it & 1) * box_floats);
            if (SOUT) tma_store_2d(&tm_s, c0x, (int)(b * (unsigned)C), ostage + (size_t)(2 + (it & 1)) * box_floats);
            bulk_commit();
          }
        } else if (wv && !L2DBG(1)) {
          float* __restrict__ po = obase + toff;
          float* __restrict__ ps = SOUT ? sbase + toff : nullptr;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            if (i < cn) {
              const float x = v[i];
              if (SOUT) { *ps = x; ps += cs; }
              *po = GELU ? gelu_fast(x) : x;
              po += cs;
            }
          }
        }
        if (ew == 0) L2TR(11, it);
      }
      if (TMA && ew == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    };
    if (e == 0) role(IC<0>{});
    else if (e == 1) role(IC<1>{});
    else if (e == 2) role(IC<2>{});
    else role(IC<3>{});
  } else if (warp == Cfg::MMA_WARP) {
    // ---- MMA issuer (whole warp converged, one elected lane issues) ------------------------------------
    constexpr unsigned idesc = umma_idesc_tf32(128, NPAD, 0, 0);
    const unsigned long long d_wh = umma_desc(bW, 128, KA * 32), d_wl = umma_desc(bW + NPAD * KA, 128, KA * 32);
    const unsigned long long d_t0 = umma_desc(bT2, 128, KQ * 32);
    const unsigned long long t2d = (unsigned long long)((t2_tile * 4) >> 4);       // descriptor step between T2 buffers
    const int nkq = KQ / 8;
    L2WAIT_HOT(f_ready, 0u);
    unsigned row = (unsigned)t_begin - rsd.div((unsigned)t_begin) * RS;
    for (int it = 0; it < ntl; ++it) {
      const int s = it & 1;
      const unsigned ph = ((unsigned)it >> 1) & 1u;
      const unsigned td = tmem_base + TM_D + (unsigned)(s * NPAD);
      const unsigned long long d_th = d_t0 + (unsigned long long)(2 * s) * t2d, d_tl = d_th + t2d;
      const unsigned ab = tmem_base + TM_A + (unsigned)(s * 2 * KA);
      const unsigned fbase = tmem_base + ((shift && ((row * (unsigned)W) & 3u)) ? TM_F1 : 0u);
      if (++row == RS) row = 0;
      L2WAIT_HOT(ready + s, ph);
      L2TR(6, it);
      tc_fence_after();
      __syncwarp();
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        if (ks < nkq && !L2DBG(4)) {
          const unsigned long long fo = (unsigned long long)(ks * 16);
          const unsigned fh = fbase + TM_FHI + 8u * ks, fl = fbase + TM_FLO + 8u * ks;
          if (!single) {
            tc_mma_tf32_ts_elect(td, fl, d_th + fo, idesc, ks != 0);
            tc_mma_tf32_ts_elect(td, fh, d_tl + fo, idesc, 1u);
          }
          tc_mma_tf32_ts_elect(td, fh, d_th + fo, idesc, single ? (unsigned)(ks != 0) : 1u);
        }
      }
#pragma unroll
      for (int ks = 0; ks < (L2DBG(4) ? 0 : KA / 8); ++ks) {
        const unsigned long long fo = (unsigned long long)(ks * 16);
        const unsigned ah = ab + 8u * ks, al = ah + KA;
        if (!single) {
          tc_mma_tf32_ts_elect(td, al, d_wh + fo, idesc, 1u);
          tc_mma_tf32_ts_elect(td, ah, d_wl + fo, idesc, 1u);
        }
        tc_mma_tf32_ts_elect(td, ah, d_wh + fo, idesc, 1u);
      }
      tc_commit_elect(mma_done + s);
      L2TR(8, it);
    }
  } else if (warp >= Cfg::BPREP_WARP0) {
    // ---- T2 operand tiles: warp j owns the rows of parity j, i.e. operand buffer s = j and ring slots j, j + 2: it
    // splits the raw tile (2.3 KB at cfg 1, bulk-copied into the ring by a converter warp) hi / lo into the operand
    // buffer.  These warps have no memory traffic of their own in flight -- no loads, stores or bulk copies --, so the
    // proxy fence their shared-memory stores need (MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC) is cheap here.
    constexpr int NFB = Cfg::NFB;
    const int j = warp - Cfg::BPREP_WARP0, s = j;
    const int tile_f4 = p.tile_floats >> 2;
    const float4* __restrict__ ring4 = reinterpret_cast<const float4*>(ring) + lane;
    float4* __restrict__ dh = reinterpret_cast<float4*>(bT2 + (size_t)(2 * s) * t2_tile) + lane;
    float4* __restrict__ dl = reinterpret_cast<float4*>(bT2 + (size_t)(2 * s + 1) * t2_tile) + lane;
    for (int it = j; it < ntl; it += 2) {
      const unsigned ph = ((unsigned)it >> 1) & 1u;
      const int slot = it & (L2_NR - 1);
      L2WAIT_COLD(raw_full + slot, ((unsigned)it / L2_NR) & 1u);
      if (j == 0) L2TR(12, it);
      float4 raw[NFB];
#pragma unroll
      for (int i = 0; i < NFB; ++i)
        if (lane + 32 * i < tile_f4) raw[i] = ring4[(size_t)slot * tile_f4 + 32 * i];
      __syncwarp();
      if (lane == 0) mbar_arrive(raw_free + slot);                   // the slot has been read: the converter may refill it
      L2WAIT_COLD(mma_done + s, ph ^ 1u);          // the MMAs of tile it - 2 no longer read B buffer s
      if (j == 0) L2TR(13, it);
#pragma unroll
      for (int i = 0; i < NFB; ++i) {
        if (lane + 32 * i < tile_f4) {
          float4 hi, lo;
          split_rm(raw[i].x, hi.x, lo.x, sp_rnd, sp_msk); split_rm(raw[i].y, hi.y, lo.y, sp_rnd, sp_msk);
          split_rm(raw[i].z, hi.z, lo.z, sp_rnd, sp_msk); split_rm(raw[i].w, hi.w, lo.w, sp_rnd, sp_msk);
          dh[32 * i] = hi;
          dl[32 * i] = lo;
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(ready + s);
      if (j == 0) L2TR(14, it);
    }
  } else if (r_edge > 0 && !L2DBG(8)) {
    // ---- edge warp: the W - 128 columns that do not fit the TMEM lanes, on the FP32 pipes, independent of the
    // pipeline.  lane = row, 32 rows per pass: spectral part from hinv_edge_kernel (coalesced over the rows), bypass
    // = C x C FMAs per column with the weights as shared-memory broadcasts; all loads of a pass are issued up front.
    const float* __restrict__ abase = p.a;
    float* __restrict__ obase = p.out;
    float* __restrict__ sbase = SOUT ? p.s_out : nullptr;
    const int RE = p.RE;
    const bool pair_ok = ((W & 1) == 0) && ((reinterpret_cast<size_t>(p.a) & 7) == 0);
    for (int base = 0; base < ntl; base += 32) {
      const bool live = base + lane < ntl;
      const unsigned T = (unsigned)(t_begin + (live ? base + lane : ntl - 1));
      const unsigned b = rsd.div(T);
      const unsigned row = T - b * RS;
      // this row's edge columns: [Wm, W), or [0, W - Wm) where the tensor-map window is shifted
      const size_t roff = (size_t)b * bs + (size_t)row * W + ((shift && ((row * (unsigned)W) & 3u)) ? 0 : Wm);
      const float* __restrict__ erow = p.E + ((size_t)b * C * RS + row) * RE;       // + co * RS * RE
      for (int j0 = 0; j0 < r_edge; j0 += 2) {             // two edge columns per pass
        const bool two = j0 + 1 < r_edge;
        const float* __restrict__ arow = abase + roff + j0;
        auto lda = [&](int ci) -> float2 {
          const float* __restrict__ q = arow + (size_t)ci * cs;
          if (two && pair_ok) return __ldg(reinterpret_cast<const float2*>(q));
          return make_float2(__ldg(q), two ? __ldg(q + 1) : 0.f);
        };
        float2 av[CX > 0 ? CX : 1];
        if (CX > 0) {
#pragma unroll
          for (int ci = 0; ci < (CX > 0 ? CX : 1); ++ci) av[ci] = lda(ci);
        }
#pragma unroll 4
        for (int co = 0; co < C; ++co) {
          const float2 e2 = __ldg(reinterpret_cast<const float2*>(erow + (size_t)co * RS * RE + j0));
          float acc0 = eB[co] + e2.x, acc1 = eB[co] + e2.y;
          const float4* __restrict__ w4 = reinterpret_cast<const float4*>(eW + co * CP);
          if (CX > 0) {
#pragma unroll
            for (int c4 = 0; c4 < (CX + 3) / 4; ++c4) {
              const float4 wq = w4[c4];
              const float wj[4] = {wq.x, wq.y, wq.z, wq.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (4 * c4 + e < CX) {
                  acc0 = fmaf(wj[e], av[4 * c4 + e].x, acc0);
                  acc1 = fmaf(wj[e], av[4 * c4 + e].y, acc1);
                }
              }
            }
          } else {
            for (int ci = 0; ci < C; ++ci) {
              const float wj = eW[co * CP + ci];
              const float2 a2 = lda(ci);
              acc0 = fmaf(wj, a2.x, acc0);
              acc1 = fmaf(wj, a2.y, acc1);
            }
          }
          if (live) {
            const size_t off = roff + (size_t)co * cs + j0;
            if (SOUT) {
              sbase[off] = acc0;
              if (two) sbase[off + 1] = acc1;
            }
            obase[off] = GELU ? gelu_fast(acc0) : acc0;
            if (two) obase[off + 1] = GELU ? gelu_fast(acc1) : acc1;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == Cfg::MMA_WARP) tmem_dealloc(tmem_base, Cfg::TM_COLS);
}

template <int KA, int NPAD, int CWQ>
size_t layer2d_smem_bytes(int KQ, int C, int Wm, bool tma) {
  const size_t CP = (size_t)((C + 3) & ~3);
  const size_t box = (size_t)((C * Wm + 31) & ~31);
  const size_t staging = (size_t)8 * L2_PD * KA * 32 + (tma ? 4 * box : 0);
  return sizeof(float) * ((size_t)4 * NPAD * KQ + 2 * NPAD * KA + (size_t)C * CP + NPAD + L2_RMAX * KQ +
                          (size_t)L2_NR * ((C + 7) / 8) * KQ * 8 + staging) + 128 + 16 + (9 + 2 * L2_NR + 8 * L2_PD) * 8 + 16;
}

template <int KA, int NPAD, int CWQ, int CX, bool GELU, bool SOUT, bool TMA>
int launch_layer2d_k(const L2Args& args, cudaStream_t st, bool attr_only) {
  using Cfg = L2Cfg<KA, NPAD, CWQ>;
  auto kern = layer2d_tc_kernel<KA, NPAD, CWQ, CX, GELU, SOUT, TMA>;
  if (attr_only) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(layer2d_tc)");
    return FNO_OK;
  }
  const int Wm = args.W < 128 ? args.W : 128;
  const size_t smem = layer2d_smem_bytes<KA, NPAD, CWQ>(args.KQ, args.C, Wm, TMA);
  if (smem > 200 * 1024) { set_error("layer2d_tc: shared memory %zu", smem); return FNO_E_ARG; }
  CUtensorMap ma, mo, ms;
  memset(&ma, 0, sizeof(ma)); memset(&mo, 0, sizeof(mo)); memset(&ms, 0, sizeof(ms));
  if (TMA) {
    const unsigned long long pixels = (unsigned long long)args.RS * args.W, planes = (unsigned long long)(args.total_tiles / args.RS) * args.C;
    const auto l2 = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    if (!make_plane_map(&ma, args.a, pixels, planes, 32, args.C, 4, l2) ||
        !make_plane_map(&mo, args.out, pixels, planes, Wm, args.C, 4, l2) ||
        (SOUT && !make_plane_map(&ms, args.s_out, pixels, planes, Wm, args.C, 4, l2))) {
      set_error("layer2d_tc: cuTensorMapEncodeTiled failed");
      return FNO_E_CUDA;
    }
  }
  const long ctas = args.total_tiles < 148 ? args.total_tiles : 148;
  kern<<<(unsigned)ctas, Cfg::THREADS, smem, st>>>(args, ma, mo, ms);
  count_launch();
  return check_launch("layer2d_tc_kernel");
}

// tensor-map eligibility: 16-byte aligned tensors and plane pitch, box rows a multiple of 16 bytes
bool layer2d_tma_ok(const L2Args& a) {
  static const bool off = [] { const char* e = std::getenv("FNO_LAYER_TMA"); return e != nullptr && e[0] == '0'; }();
  if (off || !tensor_maps_available()) return false;
  const int Wm = a.W < 128 ? a.W : 128;
  if (((long)a.RS * a.W) % 4 != 0 || Wm % 4 != 0 || (long)a.RS * a.W >= (1L << 31)) return false;
  // every row's column window must start 16-byte aligned: W % 4 == 0, or W = 130 (window [2, 130) on odd rows)
  if (a.W % 4 != 0 && !(a.W % 4 == 2 && a.W == Wm + 2)) return false;
  if (((reinterpret_cast<size_t>(a.a) | reinterpret_cast<size_t>(a.out) | reinterpret_cast<size_t>(a.s_out)) & 15) != 0) return false;
  return true;
}

template <int KA, int NPAD, int CWQ, int CX, bool TMA>
int launch_layer2d_m(const L2Args& args, cudaStream_t st, bool attr_only) {
  if (attr_only) {                         // once per device: raise the dynamic shared-memory limit of all four forms
    int rc = launch_layer2d_k<KA, NPAD, CWQ, CX, true, true, TMA>(args, st, true);
    if (rc == FNO_OK) rc = launch_layer2d_k<KA, NPAD, CWQ, CX, true, false, TMA>(args, st, true);
    if (rc == FNO_OK) rc = launch_layer2d_k<KA, NPAD, CWQ, CX, false, true, TMA>(args, st, true);
    if (rc == FNO_OK) rc = launch_layer2d_k<KA, NPAD, CWQ, CX, false, false, TMA>(args, st, true);
    return rc;
  }
  const bool so = args.s_out != nullptr;
  if (args.apply_gelu) return so ? launch_layer2d_k<KA, NPAD, CWQ, CX, true, true, TMA>(args, st, false)
                                 : launch_layer2d_k<KA, NPAD, CWQ, CX, true, false, TMA>(args, st, false);
  return so ? launch_layer2d_k<KA, NPAD, CWQ, CX, false, true, TMA>(args, st, false)
            : launch_layer2d_k<KA, NPAD, CWQ, CX, false, false, TMA>(args, st, false);
}

template <int KA, int NPAD, int CWQ, int CX>
int launch_layer2d_t(const L2Args& args, cudaStream_t st, bool attr_only = false) {
  if (attr_only) {
    const int rc = launch_layer2d_m<KA, NPAD, CWQ, CX, true>(args, st, true);
    return rc != FNO_OK ? rc : launch_layer2d_m<KA, NPAD, CWQ, CX, false>(args, st, true);
  }
  return layer2d_tma_ok(args) ? launch_layer2d_m<KA, NPAD, CWQ, CX, true>(args, st, false)
                              : launch_layer2d_m<KA, NPAD, CWQ, CX, false>(args, st, false);
}

template <int M1T>
int launch_hinv_t(const Plan* p, const float* Y, float* T2g, int B, int C, int KQ, int tile_floats, int cmode, float scale,
                  const EdgeArgs& ea, cudaStream_t st) {
  const int NP = p->H / 2 + 1;
  int threads = 8 * p->m2;
  threads = (threads + 31) & ~31;
  // row-pair slices: enough CTAs for ~4 waves of small blocks
  const long base = (long)B * p->D1 * ((C + 7) / 8);
  int TS = (int)((4L * 148 * 4 + base - 1) / base);
  { static const int ov = [] { const char* e = std::getenv("FNO_HINV_TS"); return e ? std::atoi(e) : 0; }(); if (ov > 0) TS = ov; }
  if (TS < 1) TS = 1;
  if (TS > NP) TS = NP;
  const int TL = (NP + TS - 1) / TS;
  TS = (NP + TL - 1) / TL;
  dim3 grid((unsigned)(B * p->D1), (unsigned)TS, (unsigned)((C + 7) / 8));
  const size_t smem = sizeof(float) * (2ul * TL * KQ * 8 + 2ul * TL * 8 * ea.RE * p->m2);
  if (smem > 48 * 1024) { set_error("hinv_tiles: row slice too large"); return FNO_E_ARG; }
  hinv_tiles_kernel<M1T><<<grid, threads, smem, st>>>(reinterpret_cast<const float2*>(Y), T2g, p->twH, p->H, p->W, p->m1, p->m2,
                                                  C, p->D1, KQ, tile_floats, TL, cmode, scale, ea);
  count_launch();
  return check_launch("hinv_tiles_kernel");
}

}  // namespace

// geometry the tensor-core layer kernel covers: one 128-lane tile (+ <= 4 edge columns) per row, 2 m2 <= 32
// twiddle columns, width + bias <= 32, 8 m2 <= 256 threads for the strided-axis stage
bool layer2d_tc_supported(const Plan* p, int C) {
  if (p == nullptr || C < 1 || C > 31) return false;
  if (p->W > 128 + L2_RMAX || 2 * p->m2 > 32 || 8 * p->m2 > 256) return false;
  if ((long)p->H * p->D1 >= (1L << 31)) return false;
  return true;
}

// raises the dynamic shared-memory limit of every instantiation on the CURRENT device (called from plan creation, which
// has made the plan's device current: the attribute is per device, so a process-wide "done" flag would be wrong)
int setup_layer2d_tc_attrs() {
  L2Args args{};
  args.KQ = 8; args.C = 1;
  int rc = launch_layer2d_t<24, 32, 2, 20>(args, nullptr, true);
  if (rc == FNO_OK) rc = launch_layer2d_t<8, 32, 2, 0>(args, nullptr, true);
  if (rc == FNO_OK) rc = launch_layer2d_t<16, 32, 2, 0>(args, nullptr, true);
  if (rc == FNO_OK) rc = launch_layer2d_t<24, 32, 2, 0>(args, nullptr, true);
  if (rc == FNO_OK) rc = launch_layer2d_t<32, 32, 2, 0>(args, nullptr, true);
  return rc;
}

static int kq_of(const Plan* p) { return (2 * p->m2 + 7) & ~7; }
static int tile_floats_of(const Plan* p, int C) { return ((C + 7) / 8) * kq_of(p) * 8; }

static int re_of(const Plan* p) { const int r = p->W > 128 ? p->W - 128 : 0; return (r + 1) & ~1; }

size_t layer2d_tc_workspace_bytes(const Plan* p, int B, int C) {
  if (!layer2d_tc_supported(p, C) || B <= 0) return 0;
  return sizeof(float) * ((size_t)B * p->D1 * p->H * tile_floats_of(p, C) + (size_t)B * C * p->D1 * p->H * re_of(p));
}

// out = act( K3(Y) + Wl a + bias ),  s_out = pre-activation (optional);  transpose_w: Wl^T a (adjoint)
int launch_layer2d_tc(const Plan* p, const float* Y, const float* a, const float* Wl, const float* bias, float* s_out,
                      float* out, float* work, int B, int C, int cmode, float scale, int apply_gelu, int transpose_w,
                      cudaStream_t st) {
  if (!layer2d_tc_supported(p, C)) { set_error("layer2d_tc: geometry not supported"); return FNO_E_ARG; }
  if ((reinterpret_cast<size_t>(work) & 15) != 0) { set_error("layer2d_tc: workspace must be 16-byte aligned"); return FNO_E_ARG; }
  const int KQ = kq_of(p), tile_floats = tile_floats_of(p, C);
  const long total = (long)B * p->D1 * p->H;
  if (total >= (1L << 32)) { set_error("layer2d_tc: too many rows"); return FNO_E_ARG; }
  float* E = work + (size_t)total * tile_floats;             // 8-byte aligned: tile_floats is a multiple of 64
  L2Args args;
  args.a = a; args.out = out; args.s_out = s_out; args.W = p->W; args.RS = p->D1 * p->H;
  const int shift = (layer2d_tma_ok(args) && p->W % 4 == 2) ? 1 : 0;
  EdgeArgs ea;
  ea.E = E; ea.twW = p->twW; ea.WP = p->WP; ea.Wm = p->W < 128 ? p->W : 128; ea.RE = re_of(p); ea.r_edge = p->W - ea.Wm;
  ea.shift = shift;
  int rc;
  switch (p->M1T) {
    case 4: rc = launch_hinv_t<4>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    case 8: rc = launch_hinv_t<8>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    case 12: rc = launch_hinv_t<12>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    case 16: rc = launch_hinv_t<16>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    case 24: rc = launch_hinv_t<24>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    case 32: rc = launch_hinv_t<32>(p, Y, work, B, C, KQ, tile_floats, cmode, scale, ea, st); break;
    default: set_error("unsupported padded modes1 %d", p->M1T); return FNO_E_ARG;
  }
  if (rc != FNO_OK) return rc;
  args.E = E; args.RE = re_of(p); args.shift = shift;
  args.a = a; args.T2g = work; args.Wl = Wl; args.bias = bias; args.s_out = s_out; args.out = out;
  args.twW = p->twW; args.WP = p->WP; args.W = p->W; args.m2 = p->m2; args.KQ = KQ; args.C = C;
  args.RS = p->D1 * p->H; args.tile_floats = tile_floats; args.total_tiles = total;
  args.transpose_w = transpose_w; args.apply_gelu = apply_gelu;
  args.single = g_math_mode.load();
  args.rs_div.init((unsigned)args.RS);
  args.trace = nullptr;
  args.dbg = 0;
#ifdef L2_TRACE
  static unsigned long long* trace_buf = nullptr;
  const bool tracing = std::getenv("FNO_L2_TRACE") != nullptr;
  { const char* e = std::getenv("FNO_L2_DBG"); args.dbg = e ? std::atoi(e) : 0; }
  if (tracing && trace_buf == nullptr) cudaMalloc(&trace_buf, 64 * 16 * 8);
  if (tracing) { cudaMemset(trace_buf, 0, 64 * 16 * 8); args.trace = trace_buf; }
#endif

  const int KA = (C + 1 + 7) & ~7;
  if (C == 20) {                                                     // the reference's width: channel loops unrolled
    rc = launch_layer2d_t<24, 32, 2, 20>(args, st);
#ifdef L2_TRACE
    static int calls = 0;
    static const int dump_call = [] { const char* e = std::getenv("FNO_L2_TRACE_CALL"); return e ? std::atoi(e) : 5; }();
    if (args.trace != nullptr && ++calls == dump_call) {
      unsigned long long h[64 * 16];
      cudaDeviceSynchronize();
      cudaMemcpy(h, args.trace, sizeof(h), cudaMemcpyDeviceToHost);
      const unsigned long long t0 = h[20 * 16 + 6];
      fprintf(stderr, "ev: 0 conv-wake 1 fenced 2 loads-in 3 sttm-issued 4 - 5 arrived | 6 mma-bready 7 mma-aready 8 committed | 9 epi-wake 10 epi-ld 11 epi-end | 12 bp-raw 13 bp-free 14 bp-arrived\n");
      fprintf(stderr, "kernel span (CTA 0, rows 0..63): first ev6 %lld, row 63 ev8 %lld\n", (long long)(h[6] - t0), (long long)(h[63 * 16 + 8] - t0));
      for (int it = 20; it < 32; ++it) {
        fprintf(stderr, "tile %2d:", it);
        for (int e = 0; e < 15; ++e) fprintf(stderr, " %6lld", h[it * 16 + e] ? (long long)(h[it * 16 + e] - t0) : -1LL);
        fprintf(stderr, "\n");
      }
    }
#endif
    return rc;
  }
  switch (KA) {
    case 8: return launch_layer2d_t<8, 32, 2, 0>(args, st);
    case 16: return launch_layer2d_t<16, 32, 2, 0>(args, st);
    case 24: return launch_layer2d_t<24, 32, 2, 0>(args, st);
    case 32: return launch_layer2d_t<32, 32, 2, 0>(args, st);
    default: set_error("layer2d_tc: width %d unsupported", C); return FNO_E_ARG;
  }
}

}  // namespace fno
