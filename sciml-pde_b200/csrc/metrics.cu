// On-device evaluation metrics (SURVEY 8f row f4): the reference's `metric_func` (pdebench/models/metrics.py:164-306,
// if_mean=True) for 2-D / 3-D fields in the loaders' layout
//     pred, target [B, nx, ny(, nz), T, V]        (channels last, time-inner; one plane of T*V values per grid point)
// and the autoregressive window shift of its rollout loop (metrics.py:341-344).  Six metrics:
//   RMSE, normalised RMSE, RMSE of the conserved (summed) variables, maximum error, RMSE at the boundaries, RMSE in
//   Fourier space (radially binned |fftn(pred) - fftn(target)|^2 over the positive quadrant, low / middle / high bands)
// plus the per-time-step RMSE the reference accumulates as `val_l2_time` (metrics.py:386-393).
//
// Kernels: one streaming pass for every point-wise sum (metric_sums_kernel: per (b, t, v): SSE, sum target^2, sum pred,
// sum target, max |err|, boundary SSE -- fp32 per thread, fp64 across blocks), the Fourier part as a separable pruned DFT of
// the error field (fftn is linear: only pred - target is transformed, and only the nx/2 x ny/2 (x nz/2) quadrant the
// reference bins is ever computed: metric_dft_axis_kernel, one launch per axis), radial binning (metric_bins_kernel) and
// a single-CTA combine (metric_final_kernel).  Evaluation is not the hot path: these kernels are written for clarity
// and to keep the whole rollout evaluation on the device without host synchronisation.
#include "common.cuh"

namespace fno {
namespace {

constexpr int MS_TV = 8;           // (t, v) pairs per pass of the sums kernel
constexpr int MS_THREADS = 256;
constexpr int MS_FIELDS = 6;       // sse, st2, sp, st, max, bd

struct MetricGeo {
  int nx, ny, nz, nd;              // nd = 2: nz == 1
  int T, V, TV;
  long S;                          // grid points per sample
};

__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x < 32) {
    s = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  }
  return s;                        // valid in thread 0
}

__global__ void __launch_bounds__(MS_THREADS)
metric_sums_kernel(const float* __restrict__ pred, const float* __restrict__ target, double* __restrict__ sums,
                   MetricGeo g, int tv0) {
  __shared__ double red[MS_THREADS / 32];
  const int b = blockIdx.y;
  const int ntv = min(MS_TV, g.TV - tv0);
  float sse[MS_TV], st2[MS_TV], sp[MS_TV], st[MS_TV], mx[MS_TV], bd[MS_TV];
#pragma unroll
  for (int i = 0; i < MS_TV; ++i) sse[i] = st2[i] = sp[i] = st[i] = mx[i] = bd[i] = 0.f;
  const long yz = (long)g.ny * g.nz;
  for (long s = (long)blockIdx.x * blockDim.x + threadIdx.x; s < g.S; s += (long)gridDim.x * blockDim.x) {
    const int x = (int)(s / yz);
    const long r = s - (long)x * yz;
    const int y = (int)(r / g.nz), z = (int)(r - (long)y * g.nz);
    // number of boundary faces through this point (corner points count once per face, as the reference's slices do)
    float faces = (float)((x == 0) + (x == g.nx - 1) + (y == 0) + (y == g.ny - 1));
    if (g.nd == 3) faces += (float)((z == 0) + (z == g.nz - 1));
    const size_t base = ((size_t)b * g.S + s) * g.TV + tv0;
#pragma unroll
    for (int i = 0; i < MS_TV; ++i)
      if (i < ntv) {
        const float p = __ldg(pred + base + i), t = __ldg(target + base + i);
        const float e = p - t;
        sse[i] = fmaf(e, e, sse[i]);
        st2[i] = fmaf(t, t, st2[i]);
        sp[i] += p;
        st[i] += t;
        mx[i] = fmaxf(mx[i], fabsf(e));
        bd[i] = fmaf(faces * e, e, bd[i]);
      }
  }
#pragma unroll
  for (int i = 0; i < MS_TV; ++i) {
    if (i >= ntv) break;                                    // uniform
    double* out = sums + ((size_t)b * g.TV + tv0 + i) * MS_FIELDS;
    double v;
    v = block_sum((double)sse[i], red); if (threadIdx.x == 0) atomicAdd(out + 0, v);
    v = block_sum((double)st2[i], red); if (threadIdx.x == 0) atomicAdd(out + 1, v);
    v = block_sum((double)sp[i], red);  if (threadIdx.x == 0) atomicAdd(out + 2, v);
    v = block_sum((double)st[i], red);  if (threadIdx.x == 0) atomicAdd(out + 3, v);
    v = block_sum((double)bd[i], red);  if (threadIdx.x == 0) atomicAdd(out + 5, v);
    float m = mx[i];
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    // non-negative doubles order like their bit patterns
    if ((threadIdx.x & 31) == 0)
      atomicMax(reinterpret_cast<unsigned long long*>(out + 4), (unsigned long long)__double_as_longlong((double)m));
  }
}

// out[o][k][i] = sum_a in[o][a][i] exp(-2 pi i k a / n),  k < m   (tensor viewed as [outer][n][inner]);
// REAL_IN: in = pred - target (real).
template <bool REAL_IN>
__global__ void __launch_bounds__(256)
metric_dft_axis_kernel(const float* __restrict__ pred, const float* __restrict__ target, const float2* __restrict__ in,
                       float2* __restrict__ out, long outer, int n, int m, long inner) {
  extern __shared__ float2 tw[];                            // exp(-2 pi i r / n), r < n
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    float s, c;
    sincospif(2.0f * (float)r / (float)n, &s, &c);
    tw[r] = make_float2(c, -s);
  }
  __syncthreads();
  const long total = outer * m * inner;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long o = idx / (m * inner);
    const long r = idx - o * (m * inner);
    const int k = (int)(r / inner);
    const long i = r - (long)k * inner;
    float re = 0.f, im = 0.f;
    int ph = 0;
    const size_t base = (size_t)o * n * inner + i;
    for (int a = 0; a < n; ++a) {
      const float2 w = tw[ph];
      if (REAL_IN) {
        const float v = __ldg(pred + base + (size_t)a * inner) - __ldg(target + base + (size_t)a * inner);
        re = fmaf(v, w.x, re);
        im = fmaf(v, w.y, im);
      } else {
        const float2 v = __ldg(in + base + (size_t)a * inner);
        re = fmaf(v.x, w.x, fmaf(-v.y, w.y, re));
        im = fmaf(v.x, w.y, fmaf(v.y, w.x, im));
      }
      ph += k;
      if (ph >= n) ph -= n;
    }
    out[idx] = make_float2(re, im);
  }
}

// D [B][hx][hy][hz][TV] -> bins[b][tv][floor(sqrt(i^2+j^2+k^2))] += |D|^2   (metrics.py:262-287)
__global__ void __launch_bounds__(256)
metric_bins_kernel(const float2* __restrict__ D, float* __restrict__ bins, int B, int hx, int hy, int hz, int TV, int nbins) {
  const long per = (long)hx * hy * hz * TV;
  const long total = (long)B * per;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / per);
    long r = idx - (long)b * per;
    const int tv = (int)(r % TV); r /= TV;
    const int k = (int)(r % hz); r /= hz;
    const int j = (int)(r % hy);
    const int i = (int)(r / hy);
    const int it = (int)floor(sqrt((double)(i * i + j * j + k * k)));
    if (it > nbins - 1) continue;
    const float2 d = D[idx];
    atomicAdd(bins + ((size_t)b * TV + tv) * nbins + it, d.x * d.x + d.y * d.y);
  }
}

// out[0..7] = RMSE, nRMSE, CSV, Max, BD, F_low, F_mid, F_high (metric_func(..., if_mean=True)); out[8 + t] = sqrt of the
// mean squared error over (b, grid, v) per time step (the `val_l2_time` increment).
__global__ void __launch_bounds__(256)
metric_final_kernel(const double* __restrict__ sums, const float* __restrict__ bins, float* __restrict__ out, int B,
                    MetricGeo g, int nbins, float Lscale, int iLow, int iHigh) {
  __shared__ double red[8];
  __shared__ double acc[5];
  const int TV = g.TV;
  const double S = (double)g.S;
  double rmse = 0, nrmse = 0;
  for (int e = threadIdx.x; e < B * TV; e += blockDim.x) {
    const double* s = sums + (size_t)e * MS_FIELDS;
    const double em = sqrt(s[0] / S);
    rmse += em;
    nrmse += em / sqrt(s[1] / S);
  }
  double v = block_sum(rmse, red);  if (threadIdx.x == 0) acc[0] = v / (B * TV);
  v = block_sum(nrmse, red);        if (threadIdx.x == 0) acc[1] = v / (B * TV);
  double csv = 0, mx = 0, bd = 0;
  for (int tv = threadIdx.x; tv < TV; tv += blockDim.x) {
    double c2 = 0, m = 0, bsum = 0;
    for (int b = 0; b < B; ++b) {
      const double* s = sums + ((size_t)b * TV + tv) * MS_FIELDS;
      const double d = s[2] - s[3];
      c2 += d * d;
      m = fmax(m, s[4]);
      if (g.nd == 2) bsum += sqrt(s[5] / (2.0 * g.nx + 2.0 * g.ny));
    }
    csv += sqrt(c2 / B) / S;
    mx += m;
    bd += bsum / B;
  }
  v = block_sum(csv, red); if (threadIdx.x == 0) acc[2] = v / TV;
  v = block_sum(mx, red);  if (threadIdx.x == 0) acc[3] = v / TV;
  if (g.nd == 3) {
    // metrics.py:243-252: the face sums are taken over the channels too, per (b, t); no mean over the batch before the sqrt
    bd = 0;
    const double den = 2.0 * ((double)g.nx * g.ny + (double)g.ny * g.nz + (double)g.nz * g.nx);
    for (int e = threadIdx.x; e < B * g.T; e += blockDim.x) {
      const int b = e / g.T, t = e - b * g.T;
      double s5 = 0;
      for (int c = 0; c < g.V; ++c) s5 += sums[((size_t)b * TV + t * g.V + c) * MS_FIELDS + 5];
      bd += sqrt(s5 / den);
    }
    v = block_sum(bd, red); if (threadIdx.x == 0) acc[4] = v / (B * g.T);
  } else {
    v = block_sum(bd, red); if (threadIdx.x == 0) acc[4] = v / TV;
  }
  // Fourier bands: _err_F[c, it, t] = sqrt(mean_b bins) * Lscale; band mean over `it`, then mean over (c, t)
  for (int band = 0; band < 3; ++band) {
    const int lo = band == 0 ? 0 : (band == 1 ? min(iLow, nbins) : min(iHigh, nbins));
    const int hi = band == 0 ? min(iLow, nbins) : (band == 1 ? min(iHigh, nbins) : nbins);
    double f = 0;
    for (int e = threadIdx.x; e < TV * max(hi - lo, 0); e += blockDim.x) {
      const int tv = e / (hi - lo), it = lo + e - tv * (hi - lo);
      double m = 0;
      for (int b = 0; b < B; ++b) m += (double)bins[((size_t)b * TV + tv) * nbins + it];
      f += sqrt(m / B) * (double)Lscale;
    }
    v = block_sum(f, red);
    // an empty band is the mean of an empty slice in the reference: NaN
    if (threadIdx.x == 0) out[5 + band] = hi > lo ? (float)(v / ((double)TV * (hi - lo))) : __int_as_float(0x7fc00000);
  }
  for (int t = 0; t < g.T; ++t) {
    double s = 0;
    for (int e = threadIdx.x; e < B * g.V; e += blockDim.x) {
      const int b = e / g.V, c = e - b * g.V;
      s += sums[((size_t)b * TV + t * g.V + c) * MS_FIELDS + 0];
    }
    v = block_sum(s, red);
    if (threadIdx.x == 0) out[8 + t] = (float)sqrt(v / (S * B * g.V));
  }
  __syncthreads();
  if (threadIdx.x < 5) out[threadIdx.x] = (float)acc[threadIdx.x];
}

// xx_out[..., t, :] = xx[..., t + 1, :] (t < T0 - 1),  xx_out[..., T0 - 1, :] = pred[..., 0, :]   (metrics.py:344)
// over a window whose first points_a points take their new frame from pred_a and the rest from pred_b (the joint
// model's primary and auxiliary rows); the single-stream shift is points_a = points
__global__ void __launch_bounds__(256)
window_shift_kernel(const float* __restrict__ xx, const float* __restrict__ pred_a, const float* __restrict__ pred_b,
                    float* __restrict__ out, long points_a, long points, int T0, int V) {
  const long total = points * T0 * V;
  const int TV = T0 * V;
  // (point, offset in the point) of o, advanced by the grid stride without a 64-bit division per element
  const long stride = (long)gridDim.x * blockDim.x, sp = stride / TV;
  const int se = (int)(stride - sp * TV);
  long o = (long)blockIdx.x * blockDim.x + threadIdx.x, pt = o / TV;
  int e = (int)(o - pt * TV);
  for (; o < total; o += stride) {
    const int v = e - (TV - V);
    const float* src = v < 0 ? xx + o + V : pt < points_a ? pred_a + pt * V + v : pred_b + (pt - points_a) * V + v;
    out[o] = __ldg(src);
    pt += sp;
    e += se;
    if (e >= TV) { e -= TV; ++pt; }
  }
}

// its adjoint: gxx[..., 0, :] = 0, gxx[..., t, :] = g[..., t - 1, :], gpred_a / gpred_b = g[..., T0 - 1, :] of their
// points (any output may be null)
__global__ void __launch_bounds__(256)
window_shift_bwd_kernel(const float* __restrict__ g, float* __restrict__ gxx, float* __restrict__ gpred_a,
                        float* __restrict__ gpred_b, long points_a, long points, int T0, int V) {
  const long total = points * T0 * V;
  const int TV = T0 * V;
  const long stride = (long)gridDim.x * blockDim.x, sp = stride / TV;
  const int se = (int)(stride - sp * TV);
  long o = (long)blockIdx.x * blockDim.x + threadIdx.x, pt = o / TV;
  int e = (int)(o - pt * TV);
  for (; o < total; o += stride) {
    if (gxx != nullptr) gxx[o] = e < V ? 0.f : __ldg(g + o - V);
    const int v = e - (TV - V);
    if (v >= 0) {
      float* dst = pt < points_a ? (gpred_a != nullptr ? gpred_a + pt * V + v : nullptr)
                                 : (gpred_b != nullptr ? gpred_b + (pt - points_a) * V + v : nullptr);
      if (dst != nullptr) *dst = __ldg(g + o);
    }
    pt += sp;
    e += se;
    if (e >= TV) { e -= TV; ++pt; }
  }
}

size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

struct MetricWork {
  size_t sums, bins, bufA, bufB, total;
};

MetricWork metric_layout(int B, int nx, int ny, int nz, int T, int V) {
  MetricWork w{};
  const size_t TV = (size_t)T * V;
  const int nbins = nz > 1 ? min(nx / 2, min(ny / 2, nz / 2)) : min(nx / 2, ny / 2);
  w.sums = 0;
  size_t off = align256(sizeof(double) * B * TV * MS_FIELDS);
  w.bins = off;
  off += align256(sizeof(float) * B * TV * (size_t)max(nbins, 1));
  // stage 1 (last spatial axis halved): B * S / 2 complex values per (t, v); stage 2 a half of that again
  const size_t S = (size_t)nx * ny * nz;
  w.bufA = off;
  off += align256(sizeof(float2) * B * (S / 2 + 1) * TV);
  w.bufB = off;
  off += align256(sizeof(float2) * B * (S / 4 + 1) * TV);
  w.total = off;
  return w;
}

unsigned grid_for(long total) {
  long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" size_t fno_metric_workspace_bytes(int B, int nx, int ny, int nz, int T, int V) {
  if (B <= 0 || nx <= 0 || ny <= 0 || nz <= 0 || T <= 0 || V <= 0) return 0;
  return metric_layout(B, nx, ny, nz, T, V).total;
}

extern "C" int fno_metric_func(const float* pred, const float* target, void* work, float* out, int B, int nx, int ny,
                               int nz, int T, int V, float Lx, float Ly, float Lz, int iLow, int iHigh,
                               fno_stream_t stream) {
  if (!pred || !target || !work || !out || B <= 0 || nx < 2 || ny < 2 || nz < 1 || nz == 2 || T <= 0 || V <= 0 ||
      iLow < 0 || iHigh < iLow) {
    set_error("fno_metric_func: bad argument (2-D: nz = 1; 3-D: nz >= 3; nx, ny >= 2)");
    return FNO_E_ARG;
  }
  if (nx > 4096 || ny > 4096 || nz > 4096) { set_error("fno_metric_func: axis longer than 4096"); return FNO_E_ARG; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MetricGeo g{};
  g.nx = nx; g.ny = ny; g.nz = nz; g.nd = nz > 1 ? 3 : 2; g.T = T; g.V = V; g.TV = T * V;
  g.S = (long)nx * ny * nz;
  const MetricWork w = metric_layout(B, nx, ny, nz, T, V);
  char* base = static_cast<char*>(work);
  double* sums = reinterpret_cast<double*>(base + w.sums);
  float* bins = reinterpret_cast<float*>(base + w.bins);
  float2* bufA = reinterpret_cast<float2*>(base + w.bufA);
  float2* bufB = reinterpret_cast<float2*>(base + w.bufB);
  const int hx = nx / 2, hy = ny / 2, hz = g.nd == 3 ? nz / 2 : 1;
  const int nbins = g.nd == 3 ? min(hx, min(hy, hz)) : min(hx, hy);
  if (cudaMemsetAsync(base, 0, w.bufA, st) != cudaSuccess) return check_launch("cudaMemsetAsync(metric workspace)");
  unsigned chunks = (unsigned)((g.S + 4 * MS_THREADS - 1) / (4 * MS_THREADS));
  if (chunks > 592) chunks = 592;
  for (int tv0 = 0; tv0 < g.TV; tv0 += MS_TV) {
    metric_sums_kernel<<<dim3(chunks, B), MS_THREADS, 0, st>>>(pred, target, sums, g, tv0);
    count_launch();
  }
  int rc = check_launch("metric_sums_kernel");
  if (rc != FNO_OK) return rc;
  const long TV = g.TV;
  const float2* D = nullptr;
  if (g.nd == 2) {
    // [B*nx][ny][TV] -> A [B*nx][hy][TV] -> B [B][hx][hy*TV]
    metric_dft_axis_kernel<true><<<grid_for((long)B * nx * hy * TV), 256, sizeof(float2) * ny, st>>>(
        pred, target, nullptr, bufA, (long)B * nx, ny, hy, TV);
    metric_dft_axis_kernel<false><<<grid_for((long)B * hx * hy * TV), 256, sizeof(float2) * nx, st>>>(
        nullptr, nullptr, bufA, bufB, (long)B, nx, hx, (long)hy * TV);
    count_launch(); count_launch();
    D = bufB;
  } else {
    // [B*nx*ny][nz][TV] -> A [..][hz][TV];  [B*nx][ny][hz*TV] -> B;  [B][nx][hy*hz*TV] -> A
    metric_dft_axis_kernel<true><<<grid_for((long)B * nx * ny * hz * TV), 256, sizeof(float2) * nz, st>>>(
        pred, target, nullptr, bufA, (long)B * nx * ny, nz, hz, TV);
    metric_dft_axis_kernel<false><<<grid_for((long)B * nx * hy * hz * TV), 256, sizeof(float2) * ny, st>>>(
        nullptr, nullptr, bufA, bufB, (long)B * nx, ny, hy, (long)hz * TV);
    metric_dft_axis_kernel<false><<<grid_for((long)B * hx * hy * hz * TV), 256, sizeof(float2) * nx, st>>>(
        nullptr, nullptr, bufB, bufA, (long)B, nx, hx, (long)hy * hz * TV);
    count_launch(); count_launch(); count_launch();
    D = bufA;
  }
  rc = check_launch("metric_dft_axis_kernel");
  if (rc != FNO_OK) return rc;
  if (nbins > 0) {
    metric_bins_kernel<<<grid_for((long)B * hx * hy * hz * TV), 256, 0, st>>>(D, bins, B, hx, hy, hz, (int)TV, nbins);
    count_launch();
  }
  const double L = g.nd == 3 ? (double)Lx * Ly * Lz : (double)Lx * Ly;
  metric_final_kernel<<<1, 256, 0, st>>>(sums, bins, out, B, g, nbins, (float)(L / (double)g.S), iLow, iHigh);
  count_launch();
  return check_launch("metric_final_kernel");
}

namespace {
int window_shift_impl(const char* name, const float* xx, const float* pred_a, const float* pred_b, float* xx_out,
                      long points_a, long points, int T0, int V, cudaStream_t st) {
  if (!xx || !xx_out || points <= 0 || T0 <= 0 || V <= 0 || points_a < 0 || points_a > points ||
      (points_a > 0 && !pred_a) || (points_a < points && !pred_b) || xx_out == xx || xx_out == pred_a ||
      xx_out == pred_b) {
    set_error("%s: bad argument (0 <= points_a <= points, a prediction for every point; in-place shift is not "
              "supported)", name);
    return FNO_E_ARG;
  }
  window_shift_kernel<<<grid_for(points * T0 * V), 256, 0, st>>>(xx, pred_a, pred_b, xx_out, points_a, points, T0, V);
  count_launch();
  return check_launch("window_shift_kernel");
}

int window_shift_bwd_impl(const char* name, const float* g, float* gxx, float* gpred_a, float* gpred_b, long points_a,
                          long points, int T0, int V, cudaStream_t st) {
  if (!g || (!gxx && !gpred_a && !gpred_b) || points <= 0 || T0 <= 0 || V <= 0 || points_a < 0 || points_a > points ||
      g == gxx || g == gpred_a || g == gpred_b) {
    set_error("%s: bad argument (need an output, 0 <= points_a <= points; in-place is not supported)", name);
    return FNO_E_ARG;
  }
  window_shift_bwd_kernel<<<grid_for(points * T0 * V), 256, 0, st>>>(g, gxx, gpred_a, gpred_b, points_a, points, T0, V);
  count_launch();
  return check_launch("window_shift_bwd_kernel");
}
}  // namespace

extern "C" int fno_window_shift(const float* xx, const float* pred, float* xx_out, long points, int T0, int V,
                                fno_stream_t stream) {
  return window_shift_impl("fno_window_shift", xx, pred, nullptr, xx_out, points, points, T0, V,
                           static_cast<cudaStream_t>(stream));
}

extern "C" int fno_window_shift_bwd(const float* g, float* gxx, float* gpred, long points, int T0, int V,
                                    fno_stream_t stream) {
  return window_shift_bwd_impl("fno_window_shift_bwd", g, gxx, gpred, nullptr, points, points, T0, V,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int fno_window_shift_split(const float* xx, const float* pred_a, const float* pred_b, float* xx_out,
                                      long points_a, long points, int T0, int V, fno_stream_t stream) {
  return window_shift_impl("fno_window_shift_split", xx, pred_a, pred_b, xx_out, points_a, points, T0, V,
                           static_cast<cudaStream_t>(stream));
}

extern "C" int fno_window_shift_split_bwd(const float* g, float* gxx, float* gpred_a, float* gpred_b, long points_a,
                                          long points, int T0, int V, fno_stream_t stream) {
  return window_shift_bwd_impl("fno_window_shift_split_bwd", g, gxx, gpred_a, gpred_b, points_a, points, T0, V,
                               static_cast<cudaStream_t>(stream));
}
