// Device-resident windowed dataset (SURVEY 8f row f4).  The reference loaders re-open the HDF5 file and read
// the WHOLE trajectory for every item (fno/utils_2d_rd_baseline.py:74-86), slice the window on the host
// and rebuild the grid per sample (:97-102).  Here the trajectories live on the GPU in a time-inner layout
//     traj [n_traj, pixels, T, V]          traj_aux [n_traj, A, pixels, T, V]   (joint model, A streams per item)
// so that the window of item (trajectory i, start s) is, per pixel, ONE contiguous run of
// (initial_step + rollout) * V floats starting at ((i * pixels + p) * T + s) * V, and a batch is
// gathered by a single streaming copy kernel straight into the layouts the lift kernel and the loss
// read:  xx [B, pixels, initial_step, V],  yy [B, pixels, rollout, V].  For the two-head joint model the
// primary and auxiliary windows go into ONE joined input xj [B + B*A, pixels, initial_step, V] (primary rows
// first, then item b's auxiliary stream k at row B + b*A + k), which the trunk reads without a concatenation.
#include "common.cuh"

namespace fno {
namespace {

// grid.y = output row (primary rows [0, B), auxiliary rows [B, B + B*A)); grid.x covers the row's
// pixels*XE window floats followed by its pixels*YE target floats, VEC consecutive output floats per thread.
// The row's source run is found once per thread, the pixel of the first float with one 32-bit FastDiv; the
// following floats step through the run and carry into the next pixel.  VEC = 4 writes 16-byte stores (host
// checks alignment and that every row segment is a multiple of 4 floats); VEC = 1 handles any size.
template <int VEC>
__global__ void __launch_bounds__(256)
window_gather_kernel(const float* __restrict__ traj, const float* __restrict__ traj_aux,
                     const long long* __restrict__ traj_idx, const int* __restrict__ t_start, float* __restrict__ xj,
                     float* __restrict__ yy, float* __restrict__ yy_aux, int B, int A, unsigned npix, int T, int V,
                     unsigned XE, unsigned YE, FastDiv by_xe, FastDiv by_ye) {
  const unsigned row = blockIdx.y;
  const unsigned nx = npix * XE, n = nx + npix * YE;        // floats of the row's window / window + targets (< 2^32)
  const unsigned o = (blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (o >= n) return;
  const bool is_x = o < nx;
  unsigned b = row, k = 0;
  if ((int)row >= B) {                                       // auxiliary row B + b*A + k
    const unsigned j = row - (unsigned)B;
    b = j / (unsigned)A;
    k = j - b * (unsigned)A;
  }
  const long long ti = __ldg(traj_idx + b);
  const float* src = (int)row < B ? traj + (size_t)ti * npix * T * V
                                  : traj_aux + ((size_t)ti * A + k) * npix * T * V;
  const unsigned r = is_x ? o : o - nx;                      // offset inside the row's xx (or yy) segment
  const unsigned E = is_x ? XE : YE;
  unsigned p = is_x ? by_xe.div(r) : by_ye.div(r);
  unsigned e = r - p * E;
  const int ts = __ldg(t_start + b) + (is_x ? 0 : (int)(XE / V));
  size_t s = ((size_t)p * T + ts) * V + e;
  const size_t jump = (size_t)T * V - E + 1;                 // end of one pixel's run -> start of the next
  float v[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    v[i] = __ldg(src + s);
    if (++e == E) { e = 0; s += jump; } else { ++s; }
  }
  float* dst = is_x ? xj + (size_t)row * nx + r
                    : ((int)row < B ? yy + (size_t)row * (n - nx) : yy_aux + (size_t)(row - B) * (n - nx)) + r;
  if constexpr (VEC == 4) {
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) dst[i] = v[i];
  }
}

bool overlaps(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
  const char *pa = static_cast<const char*>(a), *pb = static_cast<const char*>(b);
  return a && b && pa < pb + b_bytes && pb < pa + a_bytes;
}

int window_gather_impl(const char* name, const float* traj, const float* traj_aux, const long long* traj_idx,
                       const int* t_start, float* xj, float* yy, float* yy_aux, int B, int A, long npix, int T, int V,
                       int initial_step, int rollout, fno_stream_t stream) {
  if (!traj || !traj_idx || !t_start || !xj || !yy || B <= 0 || npix <= 0 || T <= 0 || V <= 0 || initial_step <= 0 ||
      rollout <= 0) {
    set_error("%s: bad argument", name);
    return FNO_E_ARG;
  }
  if (A < 0) {
    set_error("%s: A = %d auxiliary streams per item, must be >= 0", name, A);
    return FNO_E_ARG;
  }
  if (A > 0 && (!traj_aux || !yy_aux)) {
    set_error("%s: A = %d needs traj_aux and yy_aux", name, A);
    return FNO_E_ARG;
  }
  if (initial_step + rollout > T) {
    set_error("%s: window of %d + %d frames is longer than the %d-frame trajectories", name, initial_step, rollout, T);
    return FNO_E_ARG;
  }
  const long long rows = (long long)B * (1 + A);
  const long long total_x = rows * npix * initial_step * V;
  const long long total_y = (long long)B * npix * rollout * V, total_ya = total_y * A;
  const long long row_n = (long long)npix * (initial_step + rollout) * V;
  if (total_x >= (1ll << 32) || total_y >= (1ll << 32) || total_ya >= (1ll << 32) || row_n >= (1ll << 32) - 256 ||
      rows > 65535) {
    set_error("%s: batch too large (element counts must fit 32 bits, at most 65535 rows)", name);
    return FNO_E_ARG;
  }
  // outputs may not overlap a store; the number of trajectories is not passed, so the first one's extent is checked
  const size_t traj_bytes = (size_t)npix * T * V * 4;
  const float* outs[3] = {xj, yy, yy_aux};
  const size_t out_bytes[3] = {(size_t)total_x * 4, (size_t)total_y * 4, (size_t)total_ya * 4};
  for (int i = 0; i < 3; ++i) {
    if (overlaps(outs[i], out_bytes[i], traj, traj_bytes) || overlaps(outs[i], out_bytes[i], traj_aux, traj_bytes * A)) {
      set_error("%s: an output aliases a trajectory store", name);
      return FNO_E_ARG;
    }
  }
  const unsigned XE = (unsigned)(initial_step * V), YE = (unsigned)(rollout * V);
  FastDiv by_xe, by_ye;
  by_xe.init(XE);
  by_ye.init(YE);
  const bool vec = (npix * XE) % 4 == 0 && (npix * YE) % 4 == 0 && reinterpret_cast<uintptr_t>(xj) % 16 == 0 &&
                   reinterpret_cast<uintptr_t>(yy) % 16 == 0 && reinterpret_cast<uintptr_t>(yy_aux) % 16 == 0;
  const int per_thread = vec ? 4 : 1;
  const dim3 grid((unsigned)((row_n / per_thread + 255) / 256), (unsigned)rows);
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (vec)
    window_gather_kernel<4><<<grid, 256, 0, st>>>(traj, traj_aux, traj_idx, t_start, xj, yy, yy_aux, B, A,
                                                  (unsigned)npix, T, V, XE, YE, by_xe, by_ye);
  else
    window_gather_kernel<1><<<grid, 256, 0, st>>>(traj, traj_aux, traj_idx, t_start, xj, yy, yy_aux, B, A,
                                                  (unsigned)npix, T, V, XE, YE, by_xe, by_ye);
  count_launch();
  return check_launch("window_gather_kernel");
}

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" int fno_window_gather(const float* traj, const long long* traj_idx, const int* t_start, float* xx, float* yy,
                                 int B, long npix, int T, int V, int initial_step, int rollout, fno_stream_t stream) {
  return window_gather_impl("fno_window_gather", traj, nullptr, traj_idx, t_start, xx, yy, nullptr, B, 0, npix, T, V,
                            initial_step, rollout, stream);
}

extern "C" int fno_window_gather_joint(const float* traj, const float* traj_aux, const long long* traj_idx,
                                       const int* t_start, float* xj, float* yy, float* yy_aux, int B, int A, long npix,
                                       int T, int V, int initial_step, int rollout, fno_stream_t stream) {
  return window_gather_impl("fno_window_gather_joint", traj, traj_aux, traj_idx, t_start, xj, yy, yy_aux, B, A, npix, T,
                            V, initial_step, rollout, stream);
}
