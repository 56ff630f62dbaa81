// Lift (fc0) and projection head (fc1 -> GELU -> fc2) of FNO2d / FNO3d, fused around the trunk's
// channel-first padded activation layout  h[b, c, r, w]  (r < R_out rows of pitch Wp; the valid
// region is r < R_in, w < W_in; 2-D: rows = x, 3-D: rows = (x, y) flattened, w = last axis).
//
//   lift  (fno/fno.py:140-159, :343-360): per-sample statistics -> normalise -> [x_tv, grid] ->
//         fc0 -> NCHW -> zero pad, written straight into the trunk layout (no cat / permute /
//         pad tensors); backward = fc0 weight/bias gradient, and the gradient w.r.t. x and grid when
//         they need one (only the statistics are constants, as under the reference's no_grad).
//   head  (fno/fno.py:180-188, :381-390): unpad -> NHWC -> fc1 -> exact GELU -> fc2 ->
//         de-normalise, reading the padded layout in place.  The 128-wide hidden layer
//         (8.4 MB/sample at 128x128) never exists in memory: forward keeps it in registers,
//         backward recomputes it tile by tile in shared memory.
//
// FP32 CUDA-core kernels (width 20 -> K = 20 contractions; the GELU over the hidden layer costs
// as many issue slots as the FMAs, see DESIGN.md section 5).
#include "common.cuh"

namespace fno {
namespace {

struct PixGeo {
  int R_in, W_in, R_out, Wp;
  long npix;      // R_in * W_in valid pixels per sample
  long plane;     // R_out * Wp elements per channel plane
};

__device__ __forceinline__ long pix_offset(const PixGeo& g, long p) {
  const long r = p / g.W_in;
  return r * g.Wp + (p - r * g.W_in);
}

// ------------------------------------------------------------------------------------------
// statistics: mean and unbiased std (+1e-7) over (pixels, time) per (sample, variable)
// ------------------------------------------------------------------------------------------
constexpr int ST_BLOCKS = 32;   // partial blocks per sample
constexpr int ST_THREADS = 256;
constexpr int VMAX = 8;

// part[b][blk][v][2] = sum (x - K_v), sum (x - K_v)^2 with the shift K_v = x[b, 0, v]
// (shifted-data algorithm: no cancellation when |mean| >> std)
__global__ void __launch_bounds__(ST_THREADS)
lift_stats_partial_kernel(const float* __restrict__ x, float* __restrict__ part, long entries, int V) {
  const int b = blockIdx.y;
  const float* __restrict__ xb = x + (size_t)b * entries * V;
  float K[VMAX], s1[VMAX], s2[VMAX];
#pragma unroll
  for (int v = 0; v < VMAX; ++v) {
    K[v] = (v < V) ? __ldg(xb + v) : 0.f;
    s1[v] = 0.f;
    s2[v] = 0.f;
  }
  const long per = (entries + gridDim.x - 1) / gridDim.x;
  const long e0 = (long)blockIdx.x * per;
  long e1 = e0 + per;
  if (e1 > entries) e1 = entries;
  for (long e = e0 + threadIdx.x; e < e1; e += ST_THREADS) {
    const float* __restrict__ p = xb + (size_t)e * V;
#pragma unroll
    for (int v = 0; v < VMAX; ++v) {
      if (v < V) {
        const float d = __ldg(p + v) - K[v];
        s1[v] += d;
        s2[v] = fmaf(d, d, s2[v]);
      }
    }
  }
  __shared__ float red[ST_THREADS / 32][VMAX][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int v = 0; v < VMAX; ++v) {
    float a = s1[v], c = s2[v];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, off);
      c += __shfl_xor_sync(0xffffffffu, c, off);
    }
    if (lane == 0) { red[warp][v][0] = a; red[warp][v][1] = c; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * V) {
    const int v = threadIdx.x >> 1, k = threadIdx.x & 1;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < ST_THREADS / 32; ++w) s += red[w][v][k];
    part[(((size_t)b * gridDim.x + blockIdx.x) * V + v) * 2 + k] = s;
  }
}

// The same partial sums for V = 1 / 2 / 4 from 16-byte loads: a float4 of the (entry, variable) stream holds lane k of
// variable k % V, so every lane keeps its own accumulator pair and the four are folded at the end.  Four independent loads per
// thread and iteration (the scalar form above had 8 bytes per thread in flight and ran at 2.3 TB/s).
template <int V>
__global__ void __launch_bounds__(ST_THREADS)
lift_stats_partial_vec_kernel(const float* __restrict__ x, float* __restrict__ part, long entries) {
  static_assert(V == 1 || V == 2 || V == 4, "a float4 must hold whole entries");
  const int b = blockIdx.y;
  const float* __restrict__ xb = x + (size_t)b * entries * V;
  float K[4], s1[4], s2[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    K[k] = __ldg(xb + (k % V));
    s1[k] = 0.f;
    s2[k] = 0.f;
  }
  const long total4 = entries * V / 4;             // entries * V % 4 == 0 (checked by the caller)
  const long per = (total4 + gridDim.x - 1) / gridDim.x;
  const long i0 = (long)blockIdx.x * per;
  long i1 = i0 + per;
  if (i1 > total4) i1 = total4;
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(xb);
  auto add = [&](const float4& q) {
    const float d0 = q.x - K[0], d1 = q.y - K[1], d2 = q.z - K[2], d3 = q.w - K[3];
    s1[0] += d0; s2[0] = fmaf(d0, d0, s2[0]);
    s1[1] += d1; s2[1] = fmaf(d1, d1, s2[1]);
    s1[2] += d2; s2[2] = fmaf(d2, d2, s2[2]);
    s1[3] += d3; s2[3] = fmaf(d3, d3, s2[3]);
  };
  long i = i0 + threadIdx.x;
  for (; i + 3 * ST_THREADS < i1; i += 4 * ST_THREADS) {
    const float4 q0 = __ldg(x4 + i), q1 = __ldg(x4 + i + ST_THREADS), q2 = __ldg(x4 + i + 2 * ST_THREADS),
                 q3 = __ldg(x4 + i + 3 * ST_THREADS);
    add(q0); add(q1); add(q2); add(q3);
  }
  for (; i < i1; i += ST_THREADS) add(__ldg(x4 + i));
  // fold the lanes of one variable: lane k belongs to variable k % V
  float a[V], c[V];
#pragma unroll
  for (int v = 0; v < V; ++v) { a[v] = 0.f; c[v] = 0.f; }
#pragma unroll
  for (int k = 0; k < 4; ++k) { a[k % V] += s1[k]; c[k % V] += s2[k]; }
  __shared__ float red[ST_THREADS / 32][V][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float av = a[v], cv = c[v];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      av += __shfl_xor_sync(0xffffffffu, av, off);
      cv += __shfl_xor_sync(0xffffffffu, cv, off);
    }
    if (lane == 0) { red[warp][v][0] = av; red[warp][v][1] = cv; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * V) {
    const int v = threadIdx.x >> 1, k = threadIdx.x & 1;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < ST_THREADS / 32; ++w) s += red[w][v][k];
    part[(((size_t)b * gridDim.x + blockIdx.x) * V + v) * 2 + k] = s;
  }
}

// stats[b][0][v] = mean, stats[b][1][v] = std + 1e-7   (torch.std_mean: unbiased)
__global__ void lift_stats_final_kernel(const float* __restrict__ x, const float* __restrict__ part,
                                        float* __restrict__ stats, long entries, int V, int B, int nblk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * V) return;
  const int b = i / V, v = i - b * V;
  double S1 = 0.0, S2 = 0.0;
  for (int k = 0; k < nblk; ++k) {
    S1 += (double)part[(((size_t)b * nblk + k) * V + v) * 2 + 0];
    S2 += (double)part[(((size_t)b * nblk + k) * V + v) * 2 + 1];
  }
  const double n = (double)entries;
  const double K = (double)x[(size_t)b * entries * V + v];
  const double mean = K + S1 / n;
  double var = (S2 - S1 * S1 / n) / (n - 1.0);
  if (var < 0.0) var = 0.0;
  stats[((size_t)b * 2 + 0) * V + v] = (float)mean;
  stats[((size_t)b * 2 + 1) * V + v] = (float)sqrt(var) + 1e-7f;
}

// ------------------------------------------------------------------------------------------
// zero the padding of a channel-first padded tensor: columns [W_in, Wp) of valid rows, whole
// rows [R_in, R_out)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pad_zero_kernel(float* __restrict__ h, PixGeo g, long planes) {
  const int padw = g.Wp - g.W_in;
  const long per_plane = (long)g.R_in * padw + (long)(g.R_out - g.R_in) * g.Wp;
  const long total = planes * per_plane;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pl = i / per_plane;
    long k = i - pl * per_plane;
    long off;
    if (k < (long)g.R_in * padw) {
      const long r = k / padw;
      off = r * g.Wp + g.W_in + (k - r * padw);
    } else {
      off = (long)g.R_in * g.Wp + (k - (long)g.R_in * padw);
    }
    h[(size_t)pl * g.plane + off] = 0.f;
  }
}

// ------------------------------------------------------------------------------------------
// lift forward: thread per valid pixel, CT output channels per pass
// ------------------------------------------------------------------------------------------
constexpr int LIFT_THREADS = 128;

template <int CT>
__global__ void __launch_bounds__(LIFT_THREADS)
lift_fwd_kernel(const float* __restrict__ x, const float* __restrict__ grid, const float* __restrict__ stats,
                const float* __restrict__ W0, const float* __restrict__ b0, float* __restrict__ h, PixGeo g,
                int T, int V, int G, int C) {
  extern __shared__ __align__(16) float sm[];
  const int F1 = T * V, F = F1 + G;
  float* ws = sm;                 // [F][CT]  fc0 weights of the current channel tile, transposed
  float* bs = ws + F * CT;        // [CT]
  const int b = blockIdx.y;
  const long p = (long)blockIdx.x * LIFT_THREADS + threadIdx.x;
  const bool active = p < g.npix;
  const float* __restrict__ xp = x + ((size_t)b * g.npix + (active ? p : 0)) * F1;
  const bool vec4 = (F1 % 4 == 0) && ((reinterpret_cast<size_t>(x) & 15u) == 0);
  const float* __restrict__ gp = grid + ((size_t)b * g.npix + (active ? p : 0)) * G;
  const long off = active ? pix_offset(g, p) : 0;
  float mu[VMAX], rs[VMAX];
#pragma unroll
  for (int v = 0; v < VMAX; ++v) {
    mu[v] = (v < V) ? __ldg(stats + (size_t)b * 2 * V + v) : 0.f;
    rs[v] = (v < V) ? 1.0f / __ldg(stats + (size_t)b * 2 * V + V + v) : 0.f;
  }

  for (int c0 = 0; c0 < C; c0 += CT) {
    __syncthreads();
    for (int i = threadIdx.x; i < F * CT; i += LIFT_THREADS) {
      const int f = i / CT, cc = i - f * CT;
      ws[i] = (c0 + cc < C) ? __ldg(W0 + (size_t)(c0 + cc) * F + f) : 0.f;
    }
    if (threadIdx.x < CT) bs[threadIdx.x] = (c0 + threadIdx.x < C) ? __ldg(b0 + c0 + threadIdx.x) : 0.f;
    __syncthreads();
    if (!active) continue;
    float acc[CT];
#pragma unroll
    for (int cc = 0; cc < CT; ++cc) acc[cc] = bs[cc];
    // normalised history (x - mean_v) / std_v, feature index f = t * V + v   (fno.py:143-149)
    if (vec4 && (V == 2 || V == 4)) {
      // a pixel's T * V history values are contiguous: 16-byte loads (a warp's scalar loads at an 80-byte lane stride
      // cost 20 L1 wavefronts per instruction -- the kernel was bound by them, not by HBM or the FMAs)
      for (int f4 = 0; f4 < F1; f4 += 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(xp + f4));
        const float xv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int v = V == 2 ? (j & 1) : j;                       // (f4 + j) % V for V = 2 / 4
          const float xn = (xv[j] - mu[v]) * rs[v];
          const float* wr = ws + (f4 + j) * CT;
#pragma unroll
          for (int cc = 0; cc < CT; ++cc) acc[cc] = fmaf(wr[cc], xn, acc[cc]);
        }
      }
    } else {
      for (int t = 0; t < T; ++t) {
#pragma unroll
        for (int v = 0; v < VMAX; ++v) {
          if (v < V) {
            const float xn = (__ldg(xp + t * V + v) - mu[v]) * rs[v];
            const float* wr = ws + (t * V + v) * CT;
#pragma unroll
            for (int cc = 0; cc < CT; ++cc) acc[cc] = fmaf(wr[cc], xn, acc[cc]);
          }
        }
      }
    }
    for (int f = F1; f < F; ++f) {
      const float gv = __ldg(gp + (f - F1));
      const float* wr = ws + f * CT;
#pragma unroll
      for (int cc = 0; cc < CT; ++cc) acc[cc] = fmaf(wr[cc], gv, acc[cc]);
    }
#pragma unroll
    for (int cc = 0; cc < CT; ++cc)
      if (c0 + cc < C) h[((size_t)b * C + c0 + cc) * g.plane + off] = acc[cc];
  }
}

// ------------------------------------------------------------------------------------------
// lift backward: gW0[c][f] = sum_{b,p} dh[b,c,p] feat[b,p,f],  gb0[c] = sum dh
// persistent CTAs over 64-pixel tiles; thread item = (c, 4 consecutive f) with lanes over items
// ------------------------------------------------------------------------------------------
constexpr int TILE = 64;          // pixels per tile: a 64-wide piece of one row
constexpr int TP = TILE + 4;      // shared-memory pitch (floats): rows 16-B aligned, bank-skewed
constexpr int LB_THREADS = 256;
constexpr int LB_ITEMS = 4;       // (c, f-quad) items per thread
constexpr int LB_CTAS = 148 * 3;

// tile -> (sample, row, first column); tiles never straddle rows, so a pixel's offset in the padded
// layout is r * Wp + w with no division per element
struct TileMap {
  int tiles_per_row;
  int total;
  FastDiv by_tpr, by_rows;
};
__device__ __forceinline__ void decode_tile(const TileMap& tm, const PixGeo& g, int tile, int& b, int& r, int& w0) {
  const int t = (int)tm.by_tpr.div((unsigned)tile);
  const int wc = tile - t * tm.tiles_per_row;
  b = (int)tm.by_rows.div((unsigned)t);
  r = t - b * g.R_in;
  w0 = wc * TILE;
}

__global__ void __launch_bounds__(LB_THREADS, 3)
lift_bwd_kernel(const float* __restrict__ x, const float* __restrict__ grid, const float* __restrict__ stats,
                const float* __restrict__ dh, float* __restrict__ part, PixGeo g, TileMap tm, int T, int V, int G,
                int C, int KSPL) {
  extern __shared__ __align__(16) float sm[];
  const int F1 = T * V, F = F1 + G;
  const int FQ = (F + 1 + 3) / 4;            // feature quads incl. the bias "feature" (= 1)
  const int FR = FQ * 4;
  float* dhs = sm;                            // [C][TP]
  float* fs = dhs + (size_t)C * TP;           // [FR][TP]
  const int nitems = C * FQ;
  float acc[LB_ITEMS][4];
#pragma unroll
  for (int k = 0; k < LB_ITEMS; ++k)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[k][q] = 0.f;

  const int k = threadIdx.x & (TILE - 1);     // pixel of the tile staged by this thread
  const int pt = threadIdx.x / TILE;          // which quarter of the channels / features it stages
  const int FCH = FR / 4;
  // compute-phase ownership
  const int slot = (KSPL == 2) ? (threadIdx.x & 127) : threadIdx.x;
  const int ks = (KSPL == 2) ? (threadIdx.x >> 7) : 0;
  const int q0 = ks * (TILE / 4 / KSPL), q1 = q0 + TILE / 4 / KSPL;

  for (int tile = blockIdx.x; tile < tm.total; tile += gridDim.x) {
    int b, r, w0;
    decode_tile(tm, g, tile, b, r, w0);
    const int w = w0 + k;
    const bool valid = w < g.W_in;
    const float* __restrict__ mean = stats + (size_t)b * 2 * V;
    const float* __restrict__ sd = mean + V;
    __syncthreads();
    {
      const float* __restrict__ dp = dh + (size_t)b * C * g.plane + (size_t)r * g.Wp + w;
      for (int c = pt; c < C; c += LB_THREADS / TILE) dhs[c * TP + k] = valid ? __ldg(dp + (size_t)c * g.plane) : 0.f;
      const size_t pidx = (size_t)b * g.npix + (size_t)r * g.W_in + w;
      const float* __restrict__ xp = x + pidx * F1;
      const float* __restrict__ gp = grid + pidx * G;
      const int f0 = pt * FCH;
      int vi = f0 % V;
      for (int f = f0; f < f0 + FCH; ++f) {
        float v = 0.f;
        if (valid) {
          if (f < F1) v = (__ldg(xp + f) - __ldg(mean + vi)) * (1.0f / __ldg(sd + vi));
          else if (f < F) v = __ldg(gp + (f - F1));
          else if (f == F) v = 1.f;
        }
        fs[f * TP + k] = v;
        if (++vi == V) vi = 0;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < LB_ITEMS; ++kk) {
      const int item = slot + kk * LB_THREADS;
      if (item >= nitems) break;
      const int fq = item / C, c = item - fq * C;   // lanes over channels: dh rows conflict-free, feature rows broadcast
      const float4* d4 = reinterpret_cast<const float4*>(dhs + c * TP);
      const float4* f0 = reinterpret_cast<const float4*>(fs + (4 * fq + 0) * TP);
      const float4* f1 = reinterpret_cast<const float4*>(fs + (4 * fq + 1) * TP);
      const float4* f2 = reinterpret_cast<const float4*>(fs + (4 * fq + 2) * TP);
      const float4* f3 = reinterpret_cast<const float4*>(fs + (4 * fq + 3) * TP);
#pragma unroll 4
      for (int q = q0; q < q1; ++q) {
        const float4 d = d4[q];
        const float4 a0 = f0[q], a1 = f1[q], a2 = f2[q], a3 = f3[q];
#define FNO_DOT4(P, U, Vv) P = fmaf(U.x, Vv.x, P); P = fmaf(U.y, Vv.y, P); P = fmaf(U.z, Vv.z, P); P = fmaf(U.w, Vv.w, P);
        FNO_DOT4(acc[kk][0], d, a0) FNO_DOT4(acc[kk][1], d, a1) FNO_DOT4(acc[kk][2], d, a2) FNO_DOT4(acc[kk][3], d, a3)
#undef FNO_DOT4
      }
      if (KSPL == 2) break;                   // one item per thread when the pixel range is split
    }
  }
  // part[cta * KSPL + ks][c][F + 1]
  float* __restrict__ pp = part + ((size_t)blockIdx.x * KSPL + ks) * C * (F + 1);
#pragma unroll
  for (int kk = 0; kk < LB_ITEMS; ++kk) {
    const int item = slot + kk * LB_THREADS;
    if (item >= nitems) break;
    const int fq = item / C, c = item - fq * C;   // lanes over channels: dh rows conflict-free, feature rows broadcast
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (4 * fq + q <= F) pp[(size_t)c * (F + 1) + 4 * fq + q] = acc[kk][q];
    if (KSPL == 2) break;
  }
}

// ------------------------------------------------------------------------------------------
// lift backward, register-tiled form (taken when the feature count is a multiple of 4 and the output
// tile is small): gW0[c, f] = sum_px dh[c, px] feat[px, f].
// The features are staged PIXEL-major, feat[px][FR], straight from the contiguous channels-last x tile
// with coalesced 16-byte loads (normalised on the way through registers); the gradient keeps its channel
// rows.  A thread owning a 4-channel x 4-feature block of the output needs one LDS.128 and four
// broadcast LDS.32 per pixel for its 16 FMAs (the first form: five LDS.128 per 16, bound by the
// shared-memory pipe), and the next tile's global data travels in registers under the products.
// Warp w accumulates pixels 8w..8w+7 of every tile; the eight pixel slices are combined once per CTA.
// ------------------------------------------------------------------------------------------
constexpr int LB2_THREADS = 256;
constexpr int LB2_SLICE = TILE / (LB2_THREADS / 32);    // pixels per warp and tile (8)
constexpr int LB2_TP = TILE + 2;           // channel-row pitch: lanes read rows 4 cq + a of one pixel -> banks 8 cq + 2 a + px
                                           // (pitch 68 put channel quads 0 / 2 / 4 on the same bank: 3-way conflicts)

template <int NIT>
__global__ void __launch_bounds__(LB2_THREADS, 3)
lift_bwd2_kernel(const float* __restrict__ x, const float* __restrict__ grid, const float* __restrict__ stats,
                 const float* __restrict__ dh, float* __restrict__ part, PixGeo g, TileMap tm, int T, int V, int G,
                 int C) {
  extern __shared__ __align__(16) float sm[];
  const int F1 = T * V, F = F1 + G;
  const int FR = (F + 1 + 3) & ~3, FQ = FR / 4;
  const int CQ = (C + 3) / 4, CR = 4 * CQ;
  const int nitems = CQ * FQ;
  // two tile buffers: tile i+1 is stored while tile i is multiplied -> ONE barrier per tile
  const int buf_floats = TILE * FR + CR * LB2_TP;
  float* feat0 = sm;                          // [2][ [TILE][FR] | [CR][TP] channel rows (pad rows zero) ]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // constant columns: bias feature = 1, padding = 0
  for (int bsel = 0; bsel < 2; ++bsel) {
    float* feat = feat0 + bsel * buf_floats;
    float* dhs = feat + TILE * FR;
    for (int i = tid; i < TILE * (FR - F); i += LB2_THREADS) {
      const int px = i / (FR - F), q = i - px * (FR - F);
      feat[px * FR + F + q] = (q == 0) ? 1.f : 0.f;
    }
    for (int i = tid; i < LB2_TP * (CR - C); i += LB2_THREADS) dhs[C * LB2_TP + i] = 0.f;
  }
  int cq[NIT], fq[NIT];
  float acc[NIT][4][4];
#pragma unroll
  for (int k = 0; k < NIT; ++k) {
    const int item = lane + 32 * k;
    const int it = item < nitems ? item : 0;
    fq[k] = it / CQ;
    cq[k] = it - fq[k] * CQ;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[k][a][b] = 0.f;
  }
  const int F4 = F1 / 4;
  // software pipeline: the next tile's global data travels in registers while this tile's products run.
  // Everything that does not depend on the tile (which element of the tile a thread stages, where it goes in
  // shared memory, which variable it belongs to) is computed once: run-time integer divisions inside the
  // tile loop cost more instructions than the products.
  constexpr int XR = 2;                       // float4 of x per thread and tile (TILE * F4 <= XR * 256)
  constexpr int DR = 3;                       // float2 of dh per thread and tile (C * TILE / 2 <= DR * 256)
  float4 xr[XR];
  float2 dr[DR];
  float gr;
  int xpx[XR], xdst[XR], xvi[XR];             // pixel (TILE = not staged), feat offset, variable of element 0
#pragma unroll
  for (int u = 0; u < XR; ++u) {
    const int i = tid + u * LB2_THREADS;
    const int px = i / F4, q = i - px * F4;
    xpx[u] = (i < TILE * F4) ? px : TILE;
    xdst[u] = px * FR + 4 * q;
    xvi[u] = (4 * q) % V;
  }
  const int gpx = (tid < TILE * G) ? tid / G : TILE;
  const int gdst = (tid < TILE * G) ? gpx * FR + F1 + (tid - gpx * G) : 0;
  int pb = 0, pnv = 0;
  auto prefetch = [&](int tile) {
    int b, r, w0;
    decode_tile(tm, g, tile, b, r, w0);
    pb = b;
    pnv = (g.W_in - w0 < TILE) ? g.W_in - w0 : TILE;
    const size_t pidx = (size_t)b * g.npix + (size_t)r * g.W_in + w0;
    const float4* __restrict__ xp = reinterpret_cast<const float4*>(x + pidx * F1);
#pragma unroll
    for (int u = 0; u < XR; ++u)
      xr[u] = (xpx[u] < pnv) ? __ldg(xp + tid + u * LB2_THREADS) : make_float4(0.f, 0.f, 0.f, 0.f);
    gr = (gpx < pnv) ? __ldg(grid + pidx * G + tid) : 0.f;
    // channel rows of the gradient: 8-byte coalesced loads (pixel pairs)
    const float* __restrict__ dp = dh + (size_t)b * C * g.plane + (size_t)r * g.Wp + w0 + 2 * lane;
#pragma unroll
    for (int u = 0; u < DR; ++u) {
      const int c = warp + u * (LB2_THREADS / 32);
      float2 v = make_float2(0.f, 0.f);
      if (c < C) {
        const float* __restrict__ q = dp + (size_t)c * g.plane;
        if (2 * lane + 1 < pnv) v = __ldg(reinterpret_cast<const float2*>(q));
        else if (2 * lane < pnv) v.x = __ldg(q);
      }
      dr[u] = v;
    }
  };
  // registers -> tile buffer `bsel` (normalising x on the way); uses the sample / valid count of the prefetched tile
  auto store_tile = [&](int bsel) {
    float* feat = feat0 + bsel * buf_floats;
    float* dhs = feat + TILE * FR;
    const float* __restrict__ mean = stats + (size_t)pb * 2 * V;
    const float* __restrict__ sd = mean + V;
#pragma unroll
    for (int u = 0; u < XR; ++u) {
      if (xpx[u] < TILE) {
        float4 v = xr[u];
        if (xpx[u] < pnv) {
          int vi = xvi[u];
          float* e = reinterpret_cast<float*>(&v);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            e[k] = (e[k] - __ldg(mean + vi)) * (1.0f / __ldg(sd + vi));
            if (++vi == V) vi = 0;
          }
        }
        *reinterpret_cast<float4*>(feat + xdst[u]) = v;
      }
    }
    if (gpx < TILE) feat[gdst] = gr;
#pragma unroll
    for (int u = 0; u < DR; ++u) {
      const int c = warp + u * (LB2_THREADS / 32);
      if (c < C) *reinterpret_cast<float2*>(dhs + c * LB2_TP + 2 * lane) = dr[u];
    }
  };
  int bsel = 0;
  if ((int)blockIdx.x < tm.total) {
    prefetch(blockIdx.x);
    store_tile(0);
    if ((int)(blockIdx.x + gridDim.x) < tm.total) prefetch(blockIdx.x + gridDim.x);
  }
  __syncthreads();

  for (int tile = blockIdx.x; tile < tm.total; tile += gridDim.x) {
    // the registers hold tile + gridDim.x: store it into the other buffer, then put tile + 2 gridDim.x in flight
    if (tile + (int)gridDim.x < tm.total) {
      store_tile(bsel ^ 1);
      if (tile + 2 * (int)gridDim.x < tm.total) prefetch(tile + 2 * gridDim.x);
    }
    const float* feat = feat0 + bsel * buf_floats;
    const float* dhs = feat + TILE * FR;
#pragma unroll
    for (int j = 0; j < LB2_SLICE; ++j) {
      const int px = warp * LB2_SLICE + j;
#pragma unroll
      for (int k = 0; k < NIT; ++k) {
        const float* __restrict__ dq = dhs + 4 * cq[k] * LB2_TP + px;
        const float4 f = *reinterpret_cast<const float4*>(feat + px * FR + 4 * fq[k]);
        const float dv[4] = {dq[0], dq[LB2_TP], dq[2 * LB2_TP], dq[3 * LB2_TP]}, fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int bb = 0; bb < 4; ++bb) acc[k][a][bb] = fmaf(dv[a], fv[bb], acc[k][a][bb]);
      }
    }
    __syncthreads();                          // tile done by every warp; the other buffer is complete
    bsel ^= 1;
  }
  // combine the eight pixel slices, then one partial record per CTA: part[cta][c][F + 1]
  __syncthreads();
  float* red = sm;                            // [8 warps][nitems][16]
#pragma unroll
  for (int k = 0; k < NIT; ++k) {
    const int item = lane + 32 * k;
    if (item < nitems) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
        *reinterpret_cast<float4*>(red + ((size_t)warp * nitems + item) * 16 + 4 * a) =
            make_float4(acc[k][a][0], acc[k][a][1], acc[k][a][2], acc[k][a][3]);
    }
  }
  __syncthreads();
  float* __restrict__ pp = part + (size_t)blockIdx.x * C * (F + 1);
  for (int o = tid; o < nitems * 16; o += LB2_THREADS) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < LB2_THREADS / 32; ++w) sum += red[(size_t)w * nitems * 16 + o];
    const int item = o >> 4, a = (o >> 2) & 3, bb = o & 3;
    const int f_q = item / CQ, c_q = item - f_q * CQ;
    const int c = 4 * c_q + a, f = 4 * f_q + bb;
    if (c < C && f <= F) pp[(size_t)c * (F + 1) + f] = sum;
  }
}

// ------------------------------------------------------------------------------------------
// lift data gradient (the statistics are constants, as under the reference's no_grad):
//   dx[b, p, t, v]  = (1 / sd[b, v]) sum_c W0[c, t V + v] dh[b, c, off(p)]
//   dgrid[b, p, g]  =                sum_c W0[c, T V + g] dh[b, c, off(p)]
// One CTA per 64-pixel row tile.  Only the valid columns of dh are read: whatever the adjoint of the first layer left in
// the padding never reaches dx.  Item = (feature quad, pixel pair): lanes over the 32 pixel pairs read a channel row of
// the tile as one 256-byte line, warps over quads read the W0 quad as a broadcast (2 shared loads per 8 FMAs).  The
// result goes through a feature-major tile in shared memory, because the tile's dx block is contiguous in HBM
// (nv * T * V floats): it leaves as coalesced 16-byte stores instead of per-pixel stores at a T * V * 4-byte lane stride.
// ------------------------------------------------------------------------------------------
constexpr int LD_THREADS = 256;
constexpr int LD_OP = TILE + 1;           // output-tile pitch: the transposing read of a warp spreads over the banks

size_t lift_dgrad_smem(int C, int F) {
  const int FR = 4 * ((F + 3) / 4);
  return sizeof(float) * ((size_t)C * FR + (size_t)C * TILE + (size_t)FR * LD_OP);
}

__global__ void __launch_bounds__(LD_THREADS)
lift_dgrad_kernel(const float* __restrict__ dh, const float* __restrict__ W0, const float* __restrict__ stats,
                  float* __restrict__ dx, float* __restrict__ dgrid, PixGeo g, TileMap tm, int T, int V, int G, int C,
                  int q0, int q1) {
  extern __shared__ __align__(16) float sm[];
  const int F1 = T * V, F = F1 + G, FR = 4 * ((F + 3) / 4);
  float* ws = sm;                             // [C][FR]      W0, zero beyond F
  float* dhs = ws + (size_t)C * FR;           // [C][TILE]    the tile's dh rows, zero beyond the valid columns
  float* os = dhs + (size_t)C * TILE;         // [FR][LD_OP]  dx | dgrid of the tile, feature-major
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int b, r, w0;
  decode_tile(tm, g, blockIdx.x, b, r, w0);
  const int nv = min(TILE, g.W_in - w0);
  for (int i = tid; i < C * FR; i += LD_THREADS) {
    const int c = i / FR, f = i - c * FR;
    ws[i] = f < F ? __ldg(W0 + (size_t)c * F + f) : 0.f;
  }
  {
    const int k = tid & (TILE - 1);
    const float* __restrict__ dp = dh + (size_t)b * C * g.plane + (size_t)r * g.Wp + w0 + k;
#pragma unroll 4
    for (int c = tid / TILE; c < C; c += LD_THREADS / TILE) dhs[c * TILE + k] = k < nv ? __ldg(dp + (size_t)c * g.plane) : 0.f;
  }
  __syncthreads();
  const float* __restrict__ sd = stats + (size_t)b * 2 * V + V;
  for (int q = q0 + warp; q < q1; q += LD_THREADS / 32) {
    float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int c = 0; c < C; ++c) {
      const float2 d = *reinterpret_cast<const float2*>(dhs + c * TILE + 2 * lane);
      const float4 w = *reinterpret_cast<const float4*>(ws + c * FR + 4 * q);
      a0[0] = fmaf(w.x, d.x, a0[0]); a0[1] = fmaf(w.y, d.x, a0[1]); a0[2] = fmaf(w.z, d.x, a0[2]); a0[3] = fmaf(w.w, d.x, a0[3]);
      a1[0] = fmaf(w.x, d.y, a1[0]); a1[1] = fmaf(w.y, d.y, a1[1]); a1[2] = fmaf(w.z, d.y, a1[2]); a1[3] = fmaf(w.w, d.y, a1[3]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int f = 4 * q + j;
      if (f < F) {
        const float s = f < F1 ? 1.0f / __ldg(sd + f % V) : 1.0f;   // the forward's reciprocal of std + 1e-7
        os[f * LD_OP + 2 * lane] = a0[j] * s;
        os[f * LD_OP + 2 * lane + 1] = a1[j] * s;
      }
    }
  }
  __syncthreads();
  const size_t p0 = (size_t)b * g.npix + (size_t)r * g.W_in + w0;   // first pixel of the tile
  if (dx != nullptr) {
    float* __restrict__ out = dx + p0 * F1;
    const int n = nv * F1;
    if ((F1 & 3) == 0 && (reinterpret_cast<size_t>(out) & 15) == 0) {
      for (int i = 4 * tid; i < n; i += 4 * LD_THREADS) {
        const int k = i / F1, f = i - k * F1;
        const float* o = os + f * LD_OP + k;
        *reinterpret_cast<float4*>(out + i) = make_float4(o[0], o[LD_OP], o[2 * LD_OP], o[3 * LD_OP]);
      }
    } else {
      for (int i = tid; i < n; i += LD_THREADS) {
        const int k = i / F1, f = i - k * F1;
        out[i] = os[f * LD_OP + k];
      }
    }
  }
  if (dgrid != nullptr && G > 0) {
    float* __restrict__ out = dgrid + p0 * G;
    const int n = nv * G;
    for (int i = tid; i < n; i += LD_THREADS) {
      const int k = i / G, f = i - k * G;
      out[i] = os[(F1 + f) * LD_OP + k];
    }
  }
}

// The split-K reduction of every weight gradient (common.cuh): output k of segment s, one warp per output.  Lanes stride
// the records (and, with copies > 1, the copies of one record: t = record * copies + copy), then a fixed xor tree.
__global__ void __launch_bounds__(128)
partial_reduce_kernel(const float* __restrict__ part, int nparts, int reclen, ReduceSegs segs) {
  int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  // unrolled, so that every segment is read from the parameter bank (a run-time index would copy segs to the stack)
  ReduceSeg g = segs.s[0];
#pragma unroll
  for (int s = 1; s < 4; ++s)
    if (k >= g.n) { k -= g.n; g = segs.s[s]; }
  if (k >= g.n) return;
  int src;
  if (g.row > 0) {
    const int r = k / g.row, c = k - r * g.row;
    src = r * g.stride + g.col + c;
  } else {
    src = g.col + k;
  }
  float sum = 0.f;
  if (g.copies == 1) {
    for (int p = lane; p < nparts; p += 32) sum += part[(size_t)p * reclen + src];
  } else {
    for (int t = lane; t < nparts * g.copies; t += 32) {
      const int r = t / g.copies, q = t - r * g.copies;
      sum += part[(size_t)r * reclen + src + q * g.copy_stride];
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  if (lane == 0 && g.dst != nullptr) g.dst[k] = sum;
}

// ------------------------------------------------------------------------------------------
// head forward: thread per 2 pixels, hidden units streamed, weights broadcast from shared memory
// ------------------------------------------------------------------------------------------
constexpr int HF_THREADS = 128;

template <int CP, int VP>
__global__ void __launch_bounds__(HF_THREADS)
head_fwd_kernel(const float* __restrict__ h, const float* __restrict__ W1, const float* __restrict__ b1,
                const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ stats,
                float* __restrict__ out, PixGeo g, int C, int HID, int V) {
  extern __shared__ __align__(16) float sm[];
  float* W1s = sm;                         // [HID][CP]
  float* W2s = W1s + (size_t)HID * CP;     // [HID][VP]
  float* b1s = W2s + (size_t)HID * VP;     // [HID]
  for (int i = threadIdx.x; i < HID * CP; i += HF_THREADS) {
    const int j = i / CP, c = i - j * CP;
    W1s[i] = (c < C) ? __ldg(W1 + (size_t)j * C + c) : 0.f;
  }
  for (int i = threadIdx.x; i < HID * VP; i += HF_THREADS) {
    const int j = i / VP, v = i - j * VP;
    W2s[i] = (v < V) ? __ldg(W2 + (size_t)v * HID + j) : 0.f;
  }
  for (int i = threadIdx.x; i < HID; i += HF_THREADS) b1s[i] = __ldg(b1 + i);
  __syncthreads();

  const int b = blockIdx.y;
  const long pa = (long)blockIdx.x * (2 * HF_THREADS) + threadIdx.x;
  const long pb = pa + HF_THREADS;
  const bool va = pa < g.npix, vb = pb < g.npix;
  if (!va) return;
  const float* __restrict__ hb = h + (size_t)b * C * g.plane;
  const long oa = pix_offset(g, pa), ob = vb ? pix_offset(g, pb) : oa;
  float ha[CP], hc[CP];
#pragma unroll
  for (int c = 0; c < CP; ++c) {
    ha[c] = (c < C) ? __ldg(hb + (size_t)c * g.plane + oa) : 0.f;
    hc[c] = (c < C) ? __ldg(hb + (size_t)c * g.plane + ob) : 0.f;
  }
  float o0[VP], o1[VP];
#pragma unroll
  for (int v = 0; v < VP; ++v) { o0[v] = 0.f; o1[v] = 0.f; }
#pragma unroll 2
  for (int j = 0; j < HID; ++j) {
    const float4* w4 = reinterpret_cast<const float4*>(W1s + (size_t)j * CP);
    float pa0 = b1s[j], pa1 = 0.f, pb0 = pa0, pb1 = 0.f;
#pragma unroll
    for (int q = 0; q < CP / 4; ++q) {
      const float4 w = w4[q];
      pa0 = fmaf(w.x, ha[4 * q + 0], pa0); pa1 = fmaf(w.y, ha[4 * q + 1], pa1);
      pa0 = fmaf(w.z, ha[4 * q + 2], pa0); pa1 = fmaf(w.w, ha[4 * q + 3], pa1);
      pb0 = fmaf(w.x, hc[4 * q + 0], pb0); pb1 = fmaf(w.y, hc[4 * q + 1], pb1);
      pb0 = fmaf(w.z, hc[4 * q + 2], pb0); pb1 = fmaf(w.w, hc[4 * q + 3], pb1);
    }
    const float ga = gelu_fast(pa0 + pa1), gb = gelu_fast(pb0 + pb1);
    const float4* v4 = reinterpret_cast<const float4*>(W2s + (size_t)j * VP);
#pragma unroll
    for (int q = 0; q < VP / 4; ++q) {
      const float4 w = v4[q];
      o0[4 * q + 0] = fmaf(w.x, ga, o0[4 * q + 0]); o0[4 * q + 1] = fmaf(w.y, ga, o0[4 * q + 1]);
      o0[4 * q + 2] = fmaf(w.z, ga, o0[4 * q + 2]); o0[4 * q + 3] = fmaf(w.w, ga, o0[4 * q + 3]);
      o1[4 * q + 0] = fmaf(w.x, gb, o1[4 * q + 0]); o1[4 * q + 1] = fmaf(w.y, gb, o1[4 * q + 1]);
      o1[4 * q + 2] = fmaf(w.z, gb, o1[4 * q + 2]); o1[4 * q + 3] = fmaf(w.w, gb, o1[4 * q + 3]);
    }
  }
  const float* __restrict__ mean = stats + (size_t)b * 2 * V;
  const float* __restrict__ sd = mean + V;
  float* __restrict__ outa = out + ((size_t)b * g.npix + pa) * V;
  float* __restrict__ outb = out + ((size_t)b * g.npix + pb) * V;
#pragma unroll
  for (int v = 0; v < VP; ++v) {
    if (v < V) {
      const float bias = __ldg(b2 + v), s = __ldg(sd + v), m = __ldg(mean + v);
      outa[v] = fmaf(o0[v] + bias, s, m);
      if (vb) outb[v] = fmaf(o1[v] + bias, s, m);
    }
  }
}

// ------------------------------------------------------------------------------------------
// head backward: persistent CTAs over 64-pixel tiles.
//   phase A  thread = (pixel, quarter of the hidden units): recompute pre-activation, GELU and
//            GELU', dpre = (W2^T do) * gelu'(pre); stores dpre / gelu tiles to shared memory and
//            accumulates its share of dh = W1^T dpre.
//   phase B1 thread = (2 hidden units, CP/4 channels): gW1 += dpre (x) h over the tile's pixels
//            (LDS.128 over 4 pixels; every output element has exactly one owner -> plain
//            register accumulators for the CTA's whole lifetime, no atomics).
//   phase B2 threads < HID: gb1, gW2 ; the other threads combine the four dh shares and store.
// ------------------------------------------------------------------------------------------
constexpr int HB_THREADS = 256;
constexpr int HB_JQ = HB_THREADS / TILE;   // hidden-unit groups in phase A (4)

template <int CP, int VP>
__global__ void __launch_bounds__(HB_THREADS, (CP <= 20 ? 2 : 1))
head_bwd_kernel(const float* __restrict__ h, const float* __restrict__ dout, const float* __restrict__ W1,
                const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ stats,
                float* __restrict__ dh, float* __restrict__ part, PixGeo g, TileMap tm, int C, int HID, int V) {
  constexpr int TC = CP / 4;                 // channels per phase-B1 thread
  extern __shared__ __align__(16) float sm[];
  float* W1s = sm;                           // [HID][CP]
  float* W2s = W1s + (size_t)HID * CP;       // [HID][VP]
  float* b1s = W2s + (size_t)HID * VP;       // [HID]
  float* Ds = b1s + HID;                     // [HID][TP]  dpre
  float* Gs = Ds + (size_t)HID * TP;         // [HID][TP]  gelu(pre)
  float* hs = Gs + (size_t)HID * TP;         // [CP][TP]
  float* dos = hs + (size_t)CP * TP;         // [VP][TP]
  float* dhs = dos + (size_t)VP * TP;        // [HB_JQ][CP][TP]

  for (int i = threadIdx.x; i < HID * CP; i += HB_THREADS) {
    const int j = i / CP, c = i - j * CP;
    W1s[i] = (c < C) ? __ldg(W1 + (size_t)j * C + c) : 0.f;
  }
  for (int i = threadIdx.x; i < HID * VP; i += HB_THREADS) {
    const int j = i / VP, v = i - j * VP;
    W2s[i] = (v < V) ? __ldg(W2 + (size_t)v * HID + j) : 0.f;
  }
  for (int i = threadIdx.x; i < HID; i += HB_THREADS) b1s[i] = __ldg(b1 + i);

  const int pix = threadIdx.x % TILE;
  const int jq = threadIdx.x / TILE;
  const int JPQ = HID / HB_JQ;               // hidden units per phase-A thread
  // phase B1 ownership: hidden units (2*jp, 2*jp+1) [+ multiples of HB_THREADS/2], channels cg*TC..
  const int jp = threadIdx.x >> 2, cg = threadIdx.x & 3;
  constexpr int MAXJR = 1;                   // HID <= MAXJR * HB_THREADS / 2 = 128
  float aw[MAXJR][2][TC];
#pragma unroll
  for (int r = 0; r < MAXJR; ++r)
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int c = 0; c < TC; ++c) aw[r][u][c] = 0.f;
  float ab1 = 0.f, aw2[VP], ab2 = 0.f;       // phase B2 owners: thread j < HID (gb1, gW2[:, j]); thread HB_THREADS-1-v (gb2)
#pragma unroll
  for (int v = 0; v < VP; ++v) aw2[v] = 0.f;

  // inputs of one tile for this thread's pixel: h[0..C), dout * std
  float hv[CP], dv[VP], sv[VP];     // dv * sv is formed at the start of phase A, not here: the prefetch must not wait
  auto load_tile = [&](int tile) {
    int b, r, w0;
    decode_tile(tm, g, tile, b, r, w0);
    const int w = w0 + pix;
    const bool valid = w < g.W_in;
    const float* __restrict__ hp = h + (size_t)b * C * g.plane + (size_t)r * g.Wp + w;
    const float* __restrict__ op = dout + ((size_t)b * g.npix + (size_t)r * g.W_in + w) * V;
    const float* __restrict__ sd = stats + (size_t)b * 2 * V + V;
#pragma unroll
    for (int c = 0; c < CP; ++c) hv[c] = (valid && c < C) ? __ldg(hp + (size_t)c * g.plane) : 0.f;
#pragma unroll
    for (int v = 0; v < VP; ++v) {
      dv[v] = (valid && v < V) ? __ldg(op + v) : 0.f;
      sv[v] = (v < V) ? __ldg(sd + v) : 0.f;
    }
  };
  if ((int)blockIdx.x < tm.total) load_tile(blockIdx.x);

  for (int tile = blockIdx.x; tile < tm.total; tile += gridDim.x) {
    __syncthreads();   // previous tile's phase B done (also covers the weight staging on entry)

    // ---- phase A --------------------------------------------------------------------------
    float dacc[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) dacc[c] = 0.f;
#pragma unroll
    for (int v = 0; v < VP; ++v) dv[v] *= sv[v];
    if (jq == 0) {
#pragma unroll
      for (int c = 0; c < CP; ++c) hs[c * TP + pix] = hv[c];
#pragma unroll
      for (int v = 0; v < VP; ++v) dos[v * TP + pix] = dv[v];
    }
    for (int jj = 0; jj < JPQ; ++jj) {
      const int j = jq * JPQ + jj;
      const float4* w4 = reinterpret_cast<const float4*>(W1s + (size_t)j * CP);
      float w[CP];
#pragma unroll
      for (int q = 0; q < CP / 4; ++q) {
        const float4 t = w4[q];
        w[4 * q + 0] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
      }
      float p0 = b1s[j], p1 = 0.f;
#pragma unroll
      for (int c = 0; c < CP; c += 2) {
        p0 = fmaf(w[c], hv[c], p0);
        p1 = fmaf(w[c + 1], hv[c + 1], p1);
      }
      float gl, gp;
      gelu_fast_both(p0 + p1, gl, gp);
      const float4* v4 = reinterpret_cast<const float4*>(W2s + (size_t)j * VP);
      float dg = 0.f;
#pragma unroll
      for (int q = 0; q < VP / 4; ++q) {
        const float4 t = v4[q];
        dg = fmaf(t.x, dv[4 * q + 0], dg); dg = fmaf(t.y, dv[4 * q + 1], dg);
        dg = fmaf(t.z, dv[4 * q + 2], dg); dg = fmaf(t.w, dv[4 * q + 3], dg);
      }
      const float dpre = dg * gp;
      Ds[j * TP + pix] = dpre;
      Gs[j * TP + pix] = gl;
#pragma unroll
      for (int c = 0; c < CP; ++c) dacc[c] = fmaf(w[c], dpre, dacc[c]);
    }
#pragma unroll
    for (int c = 0; c < CP; ++c) dhs[(jq * CP + c) * TP + pix] = dacc[c];
    // the next tile's inputs travel while phase B runs (hv / dv are dead until the next phase A)
    if (tile + (int)gridDim.x < tm.total) load_tile(tile + gridDim.x);
    __syncthreads();

    // ---- phase B1: gW1 ------------------------------------------------------------------------
#pragma unroll
    for (int r = 0; r < MAXJR; ++r) {
      const int j0 = 2 * (jp + r * (HB_THREADS / 4));
      if (j0 >= HID) break;
      const float4* d0 = reinterpret_cast<const float4*>(Ds + (size_t)j0 * TP);
      const float4* d1 = reinterpret_cast<const float4*>(Ds + (size_t)(j0 + 1) * TP);
#pragma unroll 2
      for (int q = 0; q < TILE / 4; ++q) {
        const float4 a = d0[q], e = d1[q];
#pragma unroll
        for (int c = 0; c < TC; ++c) {
          const float4 x4 = reinterpret_cast<const float4*>(hs + (size_t)(cg * TC + c) * TP)[q];
          aw[r][0][c] = fmaf(a.x, x4.x, aw[r][0][c]); aw[r][0][c] = fmaf(a.y, x4.y, aw[r][0][c]);
          aw[r][0][c] = fmaf(a.z, x4.z, aw[r][0][c]); aw[r][0][c] = fmaf(a.w, x4.w, aw[r][0][c]);
          aw[r][1][c] = fmaf(e.x, x4.x, aw[r][1][c]); aw[r][1][c] = fmaf(e.y, x4.y, aw[r][1][c]);
          aw[r][1][c] = fmaf(e.z, x4.z, aw[r][1][c]); aw[r][1][c] = fmaf(e.w, x4.w, aw[r][1][c]);
        }
      }
    }
    // ---- phase B2: gb1, gW2, gb2, dh ----------------------------------------------------------
    if (threadIdx.x < HID) {
      const int j = threadIdx.x;
      const float4* d4 = reinterpret_cast<const float4*>(Ds + (size_t)j * TP);
      const float4* g4 = reinterpret_cast<const float4*>(Gs + (size_t)j * TP);
#pragma unroll 2
      for (int q = 0; q < TILE / 4; ++q) {
        const float4 d = d4[q], gg = g4[q];
        ab1 += (d.x + d.y) + (d.z + d.w);
#pragma unroll
        for (int v = 0; v < VP; ++v) {
          const float4 o = reinterpret_cast<const float4*>(dos + (size_t)v * TP)[q];
          aw2[v] = fmaf(gg.x, o.x, aw2[v]); aw2[v] = fmaf(gg.y, o.y, aw2[v]);
          aw2[v] = fmaf(gg.z, o.z, aw2[v]); aw2[v] = fmaf(gg.w, o.w, aw2[v]);
        }
      }
    }
    if (threadIdx.x >= HB_THREADS - VP) {
      const int v = HB_THREADS - 1 - threadIdx.x;
      for (int k = 0; k < TILE; ++k) ab2 += dos[v * TP + k];
    }
    // dh[b, c, pixel] = sum of the four hidden-unit shares (all threads; coalesced over pixels)
    {
      int b, r, w0;
      decode_tile(tm, g, tile, b, r, w0);
      float* __restrict__ dp = dh + (size_t)b * C * g.plane + (size_t)r * g.Wp + w0;
      for (int i = threadIdx.x; i < C * TILE; i += HB_THREADS) {
        const int c = i / TILE, k = i - c * TILE;
        if (w0 + k < g.W_in) {
          float s = 0.f;
#pragma unroll
          for (int q = 0; q < HB_JQ; ++q) s += dhs[(q * CP + c) * TP + k];
          dp[(size_t)c * g.plane + k] = s;
        }
      }
    }
  }

  // per-CTA partial record: gW1 [HID][CP] | gb1 [HID] | gW2 [VP][HID] | gb2 [VP]
  const int reclen = HID * CP + HID + VP * HID + VP;
  float* __restrict__ pp = part + (size_t)blockIdx.x * reclen;
#pragma unroll
  for (int r = 0; r < MAXJR; ++r) {
    const int j0 = 2 * (jp + r * (HB_THREADS / 4));
    if (j0 >= HID) break;
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int c = 0; c < TC; ++c) pp[(size_t)(j0 + u) * CP + cg * TC + c] = aw[r][u][c];
  }
  if (threadIdx.x < HID) {
    pp[HID * CP + threadIdx.x] = ab1;
#pragma unroll
    for (int v = 0; v < VP; ++v) pp[HID * CP + HID + v * HID + threadIdx.x] = aw2[v];
  }
  if (threadIdx.x >= HB_THREADS - VP) pp[HID * CP + HID + VP * HID + (HB_THREADS - 1 - threadIdx.x)] = ab2;
}

PixGeo make_geo(int R_in, int W_in, int R_out, int Wp) {
  PixGeo g;
  g.R_in = R_in; g.W_in = W_in; g.R_out = R_out; g.Wp = Wp;
  g.npix = (long)R_in * W_in;
  g.plane = (long)R_out * Wp;
  return g;
}

bool bad_geo(int B, int R_in, int W_in, int R_out, int Wp) {
  return B <= 0 || B > 65535 || R_in <= 0 || W_in <= 0 || R_out < R_in || Wp < W_in;
}

constexpr int PERSIST_CTAS = 148 * 2;

TileMap make_tiles(const PixGeo& g, int B) {
  TileMap tm;
  tm.tiles_per_row = (g.W_in + TILE - 1) / TILE;
  const long total = (long)B * g.R_in * tm.tiles_per_row;
  tm.total = total < 0x7fffffffL ? (int)total : -1;
  tm.by_tpr.init((unsigned)tm.tiles_per_row);
  tm.by_rows.init((unsigned)g.R_in);
  return tm;
}

template <int CP, int VP>
size_t head_bwd_smem(int HID) {
  return sizeof(float) * ((size_t)HID * CP + (size_t)HID * VP + HID + 2ul * HID * TP + (size_t)CP * TP +
                          (size_t)VP * TP + (size_t)HB_JQ * CP * TP);
}

template <int CP, int VP>
int launch_head_fwd(const float* h, const float* W1, const float* b1, const float* W2, const float* b2,
                    const float* stats, float* out, const PixGeo& g, int B, int C, int HID, int V, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((size_t)HID * CP + (size_t)HID * VP + HID);
  auto k = head_fwd_kernel<CP, VP>;
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_fwd)");
    done.mark();
  }
  if (smem > 160 * 1024) { set_error("head_fwd: hidden %d x width %d too large", HID, C); return FNO_E_ARG; }
  dim3 grid((unsigned)((g.npix + 2 * HF_THREADS - 1) / (2 * HF_THREADS)), B);
  k<<<grid, HF_THREADS, smem, st>>>(h, W1, b1, W2, b2, stats, out, g, C, HID, V);
  count_launch();
  return check_launch("head_fwd_kernel");
}

template <int CP, int VP>
int launch_head_bwd(const float* h, const float* dout, const float* W1, const float* b1, const float* W2,
                    const float* stats, float* dh, float* gW1, float* gb1, float* gW2, float* gb2, float* part,
                    const PixGeo& g, int B, int C, int HID, int V, cudaStream_t st) {
  const size_t smem = head_bwd_smem<CP, VP>(HID);
  auto k = head_bwd_kernel<CP, VP>;
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(head_bwd)");
    done.mark();
  }
  if (smem > 227 * 1024) { set_error("head_bwd: hidden %d x width %d too large", HID, C); return FNO_E_ARG; }
  const TileMap tm = make_tiles(g, B);
  if (tm.total <= 0) { set_error("head_bwd: too many pixel tiles"); return FNO_E_ARG; }
  const int ctas = tm.total < PERSIST_CTAS ? tm.total : PERSIST_CTAS;
  k<<<ctas, HB_THREADS, smem, st>>>(h, dout, W1, b1, W2, stats, dh, part, g, tm, C, HID, V);
  count_launch();
  int rc = check_launch("head_bwd_kernel");
  if (rc != FNO_OK) return rc;
  const int reclen = HID * CP + HID + VP * HID + VP;
  ReduceSegs segs;
  segs.s[0] = {gW1, HID * C, 0, C, CP};
  segs.s[1] = {gb1, HID, HID * CP};
  segs.s[2] = {gW2, V * HID, HID * CP + HID};
  segs.s[3] = {gb2, V, HID * CP + HID + VP * HID};
  return launch_partial_reduce(part, ctas, reclen, segs, st);
}

int pick_cp(int C) {
  const int sizes[] = {8, 12, 20, 32, 64};
  for (int s : sizes)
    if (C <= s) return s;
  return -1;
}

int launch_pad_zero(float* h, const PixGeo& g, long planes, cudaStream_t st) {
  const long per_plane = (long)g.R_in * (g.Wp - g.W_in) + (long)(g.R_out - g.R_in) * g.Wp;
  if (per_plane == 0) return FNO_OK;
  const long total = planes * per_plane;
  long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pad_zero_kernel<<<(unsigned)blocks, 256, 0, st>>>(h, g, planes);
  count_launch();
  return check_launch("pad_zero_kernel");
}

}  // namespace
}  // namespace fno

namespace fno {
int launch_partial_reduce(const float* part, int nparts, int reclen, const ReduceSegs& segs, cudaStream_t st) {
  const int total = segs.s[0].n + segs.s[1].n + segs.s[2].n + segs.s[3].n;
  partial_reduce_kernel<<<(total * 32 + 127) / 128, 128, 0, st>>>(part, nparts, reclen, segs);
  count_launch();
  return check_launch("partial_reduce_kernel");
}

// zero padding of a trunk-layout gradient tensor (used by head_bwd_tc.cu as well)
int head_pad_zero(float* dh, int R_in, int W_in, int R_out, int Wp, long planes, cudaStream_t st) {
  return launch_pad_zero(dh, make_geo(R_in, W_in, R_out, Wp), planes, st);
}
}  // namespace fno

using namespace fno;

#define FNO_DISPATCH_CPVP(FN, ...)                                                         \
  do {                                                                                     \
    const int cp_ = pick_cp(C);                                                            \
    if (cp_ < 0 || V > 8 || V < 1) { set_error("unsupported width %d / variables %d", C, V); return FNO_E_ARG; } \
    if (V <= 4) {                                                                          \
      switch (cp_) {                                                                       \
        case 8: return FN<8, 4>(__VA_ARGS__);                                              \
        case 12: return FN<12, 4>(__VA_ARGS__);                                            \
        case 20: return FN<20, 4>(__VA_ARGS__);                                            \
        case 32: return FN<32, 4>(__VA_ARGS__);                                            \
        default: return FN<64, 4>(__VA_ARGS__);                                            \
      }                                                                                    \
    }                                                                                      \
    switch (cp_) {                                                                         \
      case 8: return FN<8, 8>(__VA_ARGS__);                                                \
      case 12: return FN<12, 8>(__VA_ARGS__);                                              \
      case 20: return FN<20, 8>(__VA_ARGS__);                                              \
      case 32: return FN<32, 8>(__VA_ARGS__);                                              \
      default: return FN<64, 8>(__VA_ARGS__);                                              \
    }                                                                                      \
  } while (0)

extern "C" size_t fno_lift_stats_workspace_bytes(int B, int V) {
  if (B <= 0 || V <= 0) return 0;
  return sizeof(float) * 2ul * (size_t)B * ST_BLOCKS * V;
}

extern "C" int fno_lift_stats(const float* x, float* stats, void* work, int B, long entries, int V,
                              fno_stream_t stream) {
  if (!x || !stats || !work || B <= 0 || B > 65535 || entries < 2 || V < 1 || V > VMAX) {
    set_error("fno_lift_stats: bad argument (need 1 <= V <= %d, entries >= 2)", VMAX);
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* part = static_cast<float*>(work);
  // 16-byte loads when a float4 holds whole entries and every sample starts 16-byte aligned
  const bool vec = (V == 1 || V == 2 || V == 4) && (entries * V) % 4 == 0 && (reinterpret_cast<size_t>(x) & 15u) == 0;
  if (vec && V == 1) lift_stats_partial_vec_kernel<1><<<dim3(ST_BLOCKS, B), ST_THREADS, 0, st>>>(x, part, entries);
  else if (vec && V == 2) lift_stats_partial_vec_kernel<2><<<dim3(ST_BLOCKS, B), ST_THREADS, 0, st>>>(x, part, entries);
  else if (vec && V == 4) lift_stats_partial_vec_kernel<4><<<dim3(ST_BLOCKS, B), ST_THREADS, 0, st>>>(x, part, entries);
  else lift_stats_partial_kernel<<<dim3(ST_BLOCKS, B), ST_THREADS, 0, st>>>(x, part, entries, V);
  count_launch();
  int rc = check_launch("lift_stats_partial_kernel");
  if (rc != FNO_OK) return rc;
  lift_stats_final_kernel<<<(B * V + 127) / 128, 128, 0, st>>>(x, part, stats, entries, V, B, ST_BLOCKS);
  count_launch();
  return check_launch("lift_stats_final_kernel");
}

extern "C" int fno_lift_fwd(const float* x, const float* grid, const float* stats, const float* W0, const float* b0,
                            float* h, int B, int R_in, int W_in, int R_out, int Wp, int T, int V, int G, int C,
                            fno_stream_t stream) {
  if (!x || !grid || !stats || !W0 || !b0 || !h || bad_geo(B, R_in, W_in, R_out, Wp) || T < 1 || V < 1 || G < 0 ||
      C < 1) {
    set_error("fno_lift_fwd: bad argument");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PixGeo g = make_geo(R_in, W_in, R_out, Wp);
  int rc = launch_pad_zero(h, g, (long)B * C, st);
  if (rc != FNO_OK) return rc;
  const int F = T * V + G;
  dim3 grid_dim((unsigned)((g.npix + LIFT_THREADS - 1) / LIFT_THREADS), B);
  if (C % 20 == 0) {
    const size_t smem = sizeof(float) * ((size_t)F * 20 + 20);
    lift_fwd_kernel<20><<<grid_dim, LIFT_THREADS, smem, st>>>(x, grid, stats, W0, b0, h, g, T, V, G, C);
  } else if (C % 16 == 0) {
    const size_t smem = sizeof(float) * ((size_t)F * 16 + 16);
    lift_fwd_kernel<16><<<grid_dim, LIFT_THREADS, smem, st>>>(x, grid, stats, W0, b0, h, g, T, V, G, C);
  } else {
    const size_t smem = sizeof(float) * ((size_t)F * 8 + 8);
    lift_fwd_kernel<8><<<grid_dim, LIFT_THREADS, smem, st>>>(x, grid, stats, W0, b0, h, g, T, V, G, C);
  }
  count_launch();
  return check_launch("lift_fwd_kernel");
}

extern "C" size_t fno_lift_bwd_workspace_bytes(int T, int V, int G, int C) {
  if (T < 1 || V < 1 || G < 0 || C < 1) return 0;
  return sizeof(float) * 2ul * (size_t)LB_CTAS * C * (T * V + G + 1);
}

extern "C" int fno_lift_bwd(const float* x, const float* grid, const float* stats, const float* dh, float* gW0,
                            float* gb0, void* work, int B, int R_in, int W_in, int R_out, int Wp, int T, int V,
                            int G, int C, fno_stream_t stream) {
  if (!x || !grid || !stats || !dh || !work || bad_geo(B, R_in, W_in, R_out, Wp) || T < 1 || V < 1 || G < 0 ||
      C < 1) {
    set_error("fno_lift_bwd: bad argument");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PixGeo g = make_geo(R_in, W_in, R_out, Wp);
  const int F = T * V + G;
  const int FQ = (F + 1 + 3) / 4;
  if (C * FQ > LB_ITEMS * LB_THREADS) {
    set_error("fno_lift_bwd: %d channels x %d features exceeds the per-CTA output tile", C, F);
    return FNO_E_ARG;
  }
  const TileMap tm0 = make_tiles(g, B);
  if (tm0.total <= 0) { set_error("fno_lift_bwd: too many pixel tiles"); return FNO_E_ARG; }
  float* part0 = static_cast<float*>(work);
  {
    // register-tiled form: contiguous 16-byte loads of the x tile need T * V % 4 == 0
    const int CQ = (C + 3) / 4, nitems = CQ * FQ, NIT = (nitems + 31) / 32;
    const bool aligned = (reinterpret_cast<size_t>(x) & 15) == 0;
    if ((T * V) % 4 == 0 && aligned && NIT <= 2 && C * (TILE / 2) <= 3 * LB2_THREADS && TILE * (T * V / 4) <= 2 * LB2_THREADS && TILE * G <= LB2_THREADS &&
        Wp % 2 == 0 && (reinterpret_cast<size_t>(dh) & 7) == 0) {
      const size_t tile_bytes = 2 * sizeof(float) * ((size_t)TILE * FQ * 4 + (size_t)CQ * 4 * LB2_TP);   // double-buffered
      const size_t red_bytes = sizeof(float) * (size_t)(LB2_THREADS / 32) * nitems * 16;
      const size_t smem2 = tile_bytes > red_bytes ? tile_bytes : red_bytes;
      const int ctas = tm0.total < LB_CTAS ? tm0.total : LB_CTAS;
      static PerDeviceOnce done2;
      if (done2.need()) {
        if (cudaFuncSetAttribute(lift_bwd2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(lift_bwd2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024) != cudaSuccess)
          return check_launch("cudaFuncSetAttribute(lift_bwd2)");
        done2.mark();
      }
      if (smem2 <= 64 * 1024) {
        if (NIT == 1) lift_bwd2_kernel<1><<<ctas, LB2_THREADS, smem2, st>>>(x, grid, stats, dh, part0, g, tm0, T, V, G, C);
        else lift_bwd2_kernel<2><<<ctas, LB2_THREADS, smem2, st>>>(x, grid, stats, dh, part0, g, tm0, T, V, G, C);
        count_launch();
        int rc2 = check_launch("lift_bwd2_kernel");
        if (rc2 != FNO_OK) return rc2;
        ReduceSegs segs2;
        segs2.s[0] = {gW0, C * F, 0, F, F + 1};
        segs2.s[1] = {gb0, C, F, 1, F + 1};
        return launch_partial_reduce(part0, ctas, C * (F + 1), segs2, st);
      }
    }
  }
  const size_t smem = sizeof(float) * ((size_t)C * TP + (size_t)FQ * 4 * TP);
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(lift_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(lift_bwd)");
    done.mark();
  }
  if (smem > 160 * 1024) { set_error("fno_lift_bwd: tile does not fit shared memory"); return FNO_E_ARG; }
  const TileMap tm = make_tiles(g, B);
  if (tm.total <= 0) { set_error("fno_lift_bwd: too many pixel tiles"); return FNO_E_ARG; }
  const int ctas = tm.total < LB_CTAS ? tm.total : LB_CTAS;
  const int KSPL = (C * FQ <= 128) ? 2 : 1;      // split the tile's pixels over two half-CTAs when outputs are few
  float* part = static_cast<float*>(work);
  lift_bwd_kernel<<<ctas, LB_THREADS, smem, st>>>(x, grid, stats, dh, part, g, tm, T, V, G, C, KSPL);
  count_launch();
  int rc = check_launch("lift_bwd_kernel");
  if (rc != FNO_OK) return rc;
  ReduceSegs segs;
  segs.s[0] = {gW0, C * F, 0, F, F + 1};
  segs.s[1] = {gb0, C, F, 1, F + 1};
  return launch_partial_reduce(part, ctas * KSPL, C * (F + 1), segs, st);
}

extern "C" int fno_lift_dgrad(const float* dh, const float* W0, const float* stats, float* dx, float* dgrid, int B,
                              int R_in, int W_in, int R_out, int Wp, int T, int V, int G, int C, fno_stream_t stream) {
  if (!dh || !W0 || !stats || (!dx && !dgrid) || bad_geo(B, R_in, W_in, R_out, Wp) || T < 1 || V < 1 || V > VMAX ||
      G < 0 || C < 1) {
    set_error("fno_lift_dgrad: bad argument (need dx or dgrid, 1 <= V <= %d)", VMAX);
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PixGeo g = make_geo(R_in, W_in, R_out, Wp);
  const int F1 = T * V, F = F1 + G;
  const size_t smem = lift_dgrad_smem(C, F);
  if (smem > 160 * 1024) { set_error("fno_lift_dgrad: %d channels x %d features do not fit shared memory", C, F); return FNO_E_ARG; }
  const TileMap tm = make_tiles(g, B);
  if (tm.total <= 0) { set_error("fno_lift_dgrad: too many pixel tiles"); return FNO_E_ARG; }
  static PerDeviceOnce done;
  if (done.need()) {
    if (cudaFuncSetAttribute(lift_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(lift_dgrad)");
    done.mark();
  }
  // feature quads to compute: those holding dx features and / or grid features
  const int q0 = dx ? 0 : F1 / 4, q1 = dgrid ? (F + 3) / 4 : (F1 + 3) / 4;
  lift_dgrad_kernel<<<tm.total, LD_THREADS, smem, st>>>(dh, W0, stats, dx, dgrid, g, tm, T, V, G, C, q0, q1);
  count_launch();
  return check_launch("lift_dgrad_kernel");
}

extern "C" int fno_head_fwd(const float* h, const float* W1, const float* b1, const float* W2, const float* b2,
                            const float* stats, float* out, int B, int R_in, int W_in, int R_out, int Wp, int C,
                            int HID, int V, fno_stream_t stream) {
  if (!h || !W1 || !b1 || !W2 || !b2 || !stats || !out || bad_geo(B, R_in, W_in, R_out, Wp) || HID < 4 ||
      HID % 4 != 0) {
    set_error("fno_head_fwd: bad argument");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PixGeo g = make_geo(R_in, W_in, R_out, Wp);
  FNO_DISPATCH_CPVP(launch_head_fwd, h, W1, b1, W2, b2, stats, out, g, B, C, HID, V, st);
}

extern "C" size_t fno_head_bwd_workspace_bytes(int C, int HID, int V) {
  const int CP = pick_cp(C);
  if (CP < 0 || HID < 1 || V < 1 || V > 8) return 0;
  const int VP = V <= 4 ? 4 : 8;
  const size_t fp32_path = sizeof(float) * (size_t)PERSIST_CTAS * ((size_t)HID * CP + HID + (size_t)VP * HID + VP);
  const size_t tc_path = head_bwd_tc_workspace_bytes();      // fno_head_bwd_tc shares the workspace contract
  return fp32_path > tc_path ? fp32_path : tc_path;
}

extern "C" int fno_head_bwd(const float* h, const float* dout, const float* W1, const float* b1, const float* W2,
                            const float* stats, float* dh, float* gW1, float* gb1, float* gW2, float* gb2, void* work,
                            int B, int R_in, int W_in, int R_out, int Wp, int C, int HID, int V,
                            fno_stream_t stream) {
  if (!h || !dout || !W1 || !b1 || !W2 || !stats || !dh || !work || bad_geo(B, R_in, W_in, R_out, Wp) ||
      HID < 8 || HID % 8 != 0 || HID > 128) {
    set_error("fno_head_bwd: bad argument (hidden width must be a multiple of 8, <= 128)");
    return FNO_E_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PixGeo g = make_geo(R_in, W_in, R_out, Wp);
  int rc = launch_pad_zero(dh, g, (long)B * C, st);
  if (rc != FNO_OK) return rc;
  float* part = static_cast<float*>(work);
  FNO_DISPATCH_CPVP(launch_head_bwd, h, dout, W1, b1, W2, stats, dh, gW1, gb1, gW2, gb2, part, g, B, C, HID, V, st);
}
