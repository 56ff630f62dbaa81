// extern "C" surface of libfno_sm100.so (include/fno_sm100.h): plan management, argument
// validation, error reporting, tensor-map encoding.  No torch types, no C++ exceptions across the boundary.
#include <cmath>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"

namespace fno {

std::atomic<unsigned long long> g_launches{0};
std::atomic<int> g_math_mode{0};

namespace {
thread_local char t_err[512] = "";
std::mutex g_plan_mutex;
std::vector<Plan*> g_plans;
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return FNO_OK;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return FNO_E_CUDA;
}

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      f = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}
}  // namespace

bool tensor_maps_available() { return encode_tiled_fn() != nullptr; }

bool make_plane_map(CUtensorMap* m, const float* base, unsigned long long pixels, unsigned long long planes,
                    unsigned box_pixels, unsigned box_planes, unsigned elem_bytes, CUtensorMapL2promotion l2) {
  const EncodeTiledFn fn = encode_tiled_fn();
  const unsigned per = elem_bytes / 4;   // floats per element
  if (fn == nullptr || base == nullptr || (per != 1 && per != 2) || pixels % per != 0 || box_pixels % per != 0) return false;
  const cuuint64_t gdim[2] = {pixels / per, planes};
  const cuuint64_t gstr[1] = {pixels * 4ull};
  const cuuint32_t box[2] = {box_pixels / per, box_planes};
  const cuuint32_t estr[2] = {1, 1};
  return fn(m, per == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim,
            gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, l2,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

namespace {

int check_device(int device) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    cudaGetLastError();
    set_error("cannot query CUDA device %d (no GPU? this library has no CPU fallback)", device);
    return FNO_E_CUDA;
  }
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; libfno_sm100 is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return FNO_E_ARCH;
  }
  return FNO_OK;
}

int pad_modes(int m1) {
  const int sizes[] = {4, 8, 12, 16, 24, 32};
  for (int s : sizes)
    if (m1 <= s) return s;
  return -1;
}

int upload(float** dst, const std::vector<float>& host) {
  if (cudaMalloc(dst, host.size() * sizeof(float)) != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaMalloc of %zu-byte twiddle table failed", host.size() * sizeof(float));
    return FNO_E_NOMEM;
  }
  if (cudaMemcpy(*dst, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess)
    return check_launch("cudaMemcpy(twiddle table)");
  return FNO_OK;
}

// exact zeros / +-1 where the angle is a multiple of pi/2 would be nice-to-have; what matters for
// the folded kernels is that sin(pi * j) of the self-paired Nyquist row is exactly 0.
double cos2pi(long num, long den) { return std::cos(2.0 * M_PI * (double)(num % den) / (double)den); }
double sin2pi(long num, long den) {
  const long r = num % den;
  if (2 * r == den || r == 0) return 0.0;
  return std::sin(2.0 * M_PI * (double)r / (double)den);
}

int build_plane_tables(Plan* p) {
  const int H = p->H, W = p->W, m1 = p->m1, m2 = p->m2, M1T = p->M1T;
  p->NP = H / 2 + 1;
  p->JP = (2 * M1T + 1 + 3) & ~3;
  p->WP = (W + 3) & ~3;
  std::vector<float> th((size_t)p->NP * p->JP, 0.0f);
  for (int t = 0; t < p->NP; ++t) {
    for (int j = 0; j <= m1; ++j) th[(size_t)t * p->JP + j] = (float)cos2pi((long)j * t, H);
    for (int j = 1; j <= m1; ++j) th[(size_t)t * p->JP + M1T + j] = (float)sin2pi((long)j * t, H);
  }
  std::vector<float> tw((size_t)2 * m2 * p->WP, 0.0f);
  for (int k = 0; k < m2; ++k)
    for (int w = 0; w < W; ++w) {
      tw[(size_t)k * p->WP + w] = (float)cos2pi((long)k * w, W);
      tw[(size_t)(m2 + k) * p->WP + w] = (float)sin2pi((long)k * w, W);
    }
  int rc = upload(&p->twH, th);
  if (rc != FNO_OK) return rc;
  return upload(&p->twW, tw);
}

// hi = rna_tf32(x) (round to nearest, ties away: what cvt.rna.tf32.f32 does), lo = x - hi
void split_tf32_host(float x, float& hi, float& lo) {
  unsigned u;
  std::memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;
  std::memcpy(&hi, &u, 4);
  lo = x - hi;
}

// F[q][w] for the tensor-core W-axis stage: q < m2 cos, m2 <= q < 2*m2 sin, in the K-major UMMA B layout
//   (q % 8) * 16 + (q / 8) * (nch * 128) + (w / 4) * 128 + (w % 4) * 4  bytes, 32 rows, nch chunks
int build_tc_tables(Plan* p) {
  p->tcF_hi = p->tcF_lo = p->tcF_bf = nullptr;
  p->tc_nch = 0;
  const int W = p->W, m2 = p->m2;
  const int KP = (W + 7) & ~7;
  const int nch = KP / 4;
  if ((W & 1) || 2 * m2 > 32 || nch > 34) return FNO_OK;   // not eligible: FP32 path only
  std::vector<float> hi((size_t)4 * nch * 32, 0.0f), lo((size_t)4 * nch * 32, 0.0f), bf((size_t)4 * nch * 32, 0.0f);
  for (int q = 0; q < 2 * m2; ++q)
    for (int w = 0; w < W; ++w) {
      const int k2 = q < m2 ? q : q - m2;
      const float v = (float)(q < m2 ? cos2pi((long)k2 * w, W) : sin2pi((long)k2 * w, W));
      const size_t off = ((size_t)(q & 7) * 16 + (size_t)(q >> 3) * nch * 128 + (size_t)(w >> 2) * 128 + (w & 3) * 4) / 4;
      split_tf32_host(v, hi[off], lo[off]);
      unsigned u;
      std::memcpy(&u, &v, 4);
      u = (u + 0x8000u) & 0xFFFF0000u;
      std::memcpy(&bf[off], &u, 4);
    }
  int rc = upload(&p->tcF_hi, hi);
  if (rc == FNO_OK) rc = upload(&p->tcF_bf, bf);
  if (rc != FNO_OK) return rc;
  rc = upload(&p->tcF_lo, lo);
  if (rc != FNO_OK) return rc;
  p->tc_nch = nch;
  return launch_fwd2d_tca(p, nullptr, nullptr, 0, nullptr, true);
}

void free_plan(Plan* p) {
  if (p == nullptr) return;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaSetDevice(p->device);
  if (p->twH) cudaFree(p->twH);
  if (p->twW) cudaFree(p->twW);
  if (p->twX) cudaFree(p->twX);
  if (p->tcF_hi) cudaFree(p->tcF_hi);
  if (p->tcF_lo) cudaFree(p->tcF_lo);
  if (p->tcF_bf) cudaFree(p->tcF_bf);
  cudaSetDevice(cur);
  cudaGetLastError();
  delete p;
}

int create_common(int device, int nd, int D1, int H, int W, int m1x, int m1, int m2, fno_plan** out) {
  if (out == nullptr) { set_error("plan_create: out is NULL"); return FNO_E_ARG; }
  *out = nullptr;
  if (H < 2 || W < 2 || m1 < 1 || m2 < 1 || 2 * m1 > H || m2 > W / 2 + 1) {
    set_error("plan_create: plane %dx%d cannot hold modes (%d, %d): need 2*m1 <= H, m2 <= W/2+1", H, W, m1, m2);
    return FNO_E_ARG;
  }
  if (nd == 3 && (D1 < 2 || m1x < 1 || 2 * m1x > D1 || m1x > 16)) {
    set_error("plan_create: outer axis %d cannot hold %d modes (need 2*m <= D, m <= 16)", D1, m1x);
    return FNO_E_ARG;
  }
  const int M1T = pad_modes(m1);
  if (M1T < 0) { set_error("plan_create: modes %d > 32 unsupported", m1); return FNO_E_ARG; }
  int rc = check_device(device);
  if (rc != FNO_OK) return rc;
  int cur = 0;
  cudaGetDevice(&cur);
  if (cudaSetDevice(device) != cudaSuccess) return check_launch("cudaSetDevice");
  Plan* p = new (std::nothrow) Plan();
  if (p == nullptr) { set_error("out of host memory"); return FNO_E_NOMEM; }
  std::memset(p, 0, sizeof(Plan));
  p->nd = nd; p->device = device; p->D1 = D1; p->H = H; p->W = W;
  p->m1x = m1x; p->m1 = m1; p->m2 = m2; p->M1T = M1T;
  rc = build_plane_tables(p);
  if (rc == FNO_OK && nd == 3) {
    const int R = 2 * m1x;
    if (sizeof(float) * 2ul * D1 * R > 48 * 1024) {
      set_error("plan_create: outer axis %d x %d kept rows exceeds the twiddle staging budget", D1, R);
      rc = FNO_E_ARG;
    } else {
      std::vector<float> tx((size_t)D1 * R * 2);
      for (int d = 0; d < D1; ++d)
        for (int r = 0; r < R; ++r) {
          const long k = (r < m1x) ? r : (long)D1 + (r - R);  // wrapped kept frequency
          tx[((size_t)d * R + r) * 2 + 0] = (float)cos2pi(k * d, D1);
          tx[((size_t)d * R + r) * 2 + 1] = (float)sin2pi(k * d, D1);
        }
      rc = upload(&p->twX, tx);
    }
  }
  if (rc == FNO_OK) rc = setup_transform2d_attrs(p);
  if (rc == FNO_OK) rc = build_tc_tables(p);
  if (rc == FNO_OK) rc = setup_layer2d_tc_attrs();
  cudaSetDevice(cur);
  if (rc != FNO_OK) { free_plan(p); return rc; }
  {
    std::lock_guard<std::mutex> lk(g_plan_mutex);
    g_plans.push_back(p);
  }
  *out = reinterpret_cast<fno_plan*>(p);
  return FNO_OK;
}

inline const Plan* P(const fno_plan* plan) { return reinterpret_cast<const Plan*>(plan); }

}  // namespace
}  // namespace fno

using namespace fno;

extern "C" {

int fno_version(void) { return 100; }
int fno_sm_arch(void) { return 100; }
const char* fno_last_error(void) { return t_err; }
unsigned long long fno_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int fno_set_math_mode(int mode) {
  if (mode != FNO_MATH_FP32 && mode != FNO_MATH_TF32 && mode != FNO_MATH_BF16) { set_error("fno_set_math_mode: unknown mode %d", mode); return FNO_E_ARG; }
  return g_math_mode.exchange(mode);
}
int fno_get_math_mode(void) { return g_math_mode.load(); }

void fno_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_plan_mutex);
  for (Plan* p : g_plans) free_plan(p);
  g_plans.clear();
}

int fno_plan2d_create(int device, int H, int W, int m1, int m2, fno_plan** out) {
  return create_common(device, 2, 1, H, W, 0, m1, m2, out);
}

int fno_plan3d_create(int device, int D1, int D2, int D3, int m1, int m2, int m3, fno_plan** out) {
  return create_common(device, 3, D1, D2, D3, m1, m2, m3, out);
}

int fno_plan_destroy(fno_plan* plan) {
  if (plan == nullptr) return FNO_OK;
  Plan* p = reinterpret_cast<Plan*>(plan);
  {
    std::lock_guard<std::mutex> lk(g_plan_mutex);
    bool found = false;
    for (size_t i = 0; i < g_plans.size(); ++i)
      if (g_plans[i] == p) { g_plans.erase(g_plans.begin() + i); found = true; break; }
    if (!found) { set_error("fno_plan_destroy: unknown plan"); return FNO_E_ARG; }
  }
  free_plan(p);
  return FNO_OK;
}

size_t fno_plan_workspace_bytes(const fno_plan* plan, long planes) {
  const Plan* p = P(plan);
  if (p == nullptr || p->nd != 3 || planes <= 0) return 0;
  // per-slice plane spectra (forward: S, inverse: Z), then -- when the inner planes are inside the tensor-core envelope
  // of K1 -- the T1 scratch of its W-axis GEMM (16-byte aligned: the first part is a multiple of 16 floats)
  const size_t spectra = (sizeof(float) * 2ul * (size_t)planes * p->D1 * (2 * p->m1) * p->m2 + 255) & ~(size_t)255;
  const size_t t1 = p->tc_nch ? sizeof(float) * (size_t)planes * p->D1 * p->H * ((2 * p->m2 + 3) & ~3) : 0;
  return spectra + t1;
}

int fno_sc2d_fwd_transform(const fno_plan* plan, const float* x, const float* preact, float* ds_out, float* X,
                           long planes, int cmode, float scale, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 2 || !x || !X || planes <= 0) { set_error("fno_sc2d_fwd_transform: bad argument"); return FNO_E_ARG; }
  return launch_fwd2d(p, x, preact, ds_out, X, planes, cmode, scale, static_cast<cudaStream_t>(stream));
}

size_t fno_sc2d_fwd_workspace_bytes(const fno_plan* plan, long planes) {
  const Plan* p = P(plan);
  if (p == nullptr || p->tc_nch == 0 || planes <= 0) return 0;
  return sizeof(float) * (size_t)planes * p->H * ((2 * p->m2 + 3) & ~3);
}

int fno_sc2d_fwd_transform_ws(const fno_plan* plan, const float* x, const float* preact, float* ds_out, float* X,
                              void* work, long planes, int cmode, float scale, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 2 || !x || !X || planes <= 0) { set_error("fno_sc2d_fwd_transform_ws: bad argument"); return FNO_E_ARG; }
  return launch_fwd2d_ws(p, x, preact, ds_out, X, static_cast<float*>(work), planes, cmode, scale,
                         static_cast<cudaStream_t>(stream));
}

int fno_sc2d_inv_transform(const fno_plan* plan, const float* Y, const float* addend, float* s_out, float* out,
                           long planes, int cmode, float scale, int apply_gelu, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 2 || !Y || !out || planes <= 0) { set_error("fno_sc2d_inv_transform: bad argument"); return FNO_E_ARG; }
  return launch_inv2d(p, Y, addend, s_out, out, planes, cmode, scale, apply_gelu, static_cast<cudaStream_t>(stream));
}

int fno_sc3d_fwd_transform(const fno_plan* plan, const float* x, const float* preact, float* ds_out, float* X,
                           void* work, long planes, int cmode, float scale, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 3 || !x || !X || !work || planes <= 0) { set_error("fno_sc3d_fwd_transform: bad argument"); return FNO_E_ARG; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = static_cast<float*>(work);
  const size_t spectra = (sizeof(float) * 2ul * (size_t)planes * p->D1 * (2 * p->m1) * p->m2 + 255) & ~(size_t)255;
  float* T1 = p->tc_nch ? reinterpret_cast<float*>(static_cast<char*>(work) + spectra) : nullptr;
  // inner planes: tcgen05 W-axis GEMM + strided-axis fold when eligible (launch_fwd2d_ws falls back to the FP32 kernel)
  int rc = launch_fwd2d_ws(p, x, preact, ds_out, S, T1, planes * p->D1, cmode, scale, st);
  if (rc != FNO_OK) return rc;
  return launch_axis_fwd(p, S, X, planes, (long)(2 * p->m1) * p->m2, st);
}

int fno_sc3d_inv_transform(const fno_plan* plan, const float* Y, const float* addend, float* s_out, float* out,
                           void* work, long planes, int cmode, float scale, int apply_gelu, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 3 || !Y || !out || !work || planes <= 0) { set_error("fno_sc3d_inv_transform: bad argument"); return FNO_E_ARG; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* Z = static_cast<float*>(work);
  int rc = launch_axis_inv(p, Y, Z, planes, (long)(2 * p->m1) * p->m2, st);
  if (rc != FNO_OK) return rc;
  return launch_inv2d(p, Z, addend, s_out, out, planes * p->D1, cmode, scale, apply_gelu, st);
}

int fno_layer2d_fused_supported(const fno_plan* plan, int C) {
  const Plan* p = P(plan);
  return (p != nullptr && p->nd == 2 && layer2d_tc_supported(p, C)) ? 1 : 0;
}

size_t fno_layer2d_fused_workspace_bytes(const fno_plan* plan, int B, int C) {
  const Plan* p = P(plan);
  if (p == nullptr || p->nd != 2) return 0;
  return layer2d_tc_workspace_bytes(p, B, C);
}

int fno_layer2d_inv_fused(const fno_plan* plan, const float* Y, const float* a, const float* W, const float* bias,
                          float* s_out, float* out, void* work, int B, int C, int cmode, float scale, int apply_gelu,
                          int transpose_w, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || p->nd != 2 || !Y || !a || !W || !out || !work || B <= 0 || C <= 0) {
    set_error("fno_layer2d_inv_fused: bad argument");
    return FNO_E_ARG;
  }
  if (a == out || a == s_out) { set_error("fno_layer2d_inv_fused: the input may not alias an output"); return FNO_E_ARG; }
  return launch_layer2d_tc(p, Y, a, W, bias, s_out, out, static_cast<float*>(work), B, C, cmode, scale, apply_gelu,
                           transpose_w, static_cast<cudaStream_t>(stream));
}

int fno_mix_tc_supported(const fno_plan* plan, int Ci, int Co) {
  const Plan* p = P(plan);
  return (p != nullptr && Ci > 0 && Co > 0 && mix_tc_supported(p, Ci, Co)) ? 1 : 0;
}

int fno_mix_fwd(const fno_plan* plan, const float* X, const float* const* w, float* Y, int B, int Ci, int Co,
                fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || !X || !w || !Y || B <= 0 || Ci <= 0 || Co <= 0) { set_error("fno_mix_fwd: bad argument"); return FNO_E_ARG; }
  const int nc = p->nd == 2 ? 2 : 4;
  for (int c = 0; c < nc; ++c)
    if (!w[c]) { set_error("fno_mix_fwd: corner weight %d is NULL", c); return FNO_E_ARG; }
  return launch_mix_fwd(p, X, w, Y, B, Ci, Co, static_cast<cudaStream_t>(stream));
}

int fno_mix_bwd(const fno_plan* plan, const float* X, const float* gY, const float* const* w, float* gX,
                float* const* gw, int B, int Ci, int Co, fno_stream_t stream) {
  const Plan* p = P(plan);
  if (!p || !gY || B <= 0 || Ci <= 0 || Co <= 0) { set_error("fno_mix_bwd: bad argument"); return FNO_E_ARG; }
  const int nc = p->nd == 2 ? 2 : 4;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (gX != nullptr) {
    if (!w) { set_error("fno_mix_bwd: weights required for gX"); return FNO_E_ARG; }
    for (int c = 0; c < nc; ++c)
      if (!w[c]) { set_error("fno_mix_bwd: corner weight %d is NULL", c); return FNO_E_ARG; }
    int rc = launch_mix_bwd_data(p, gY, w, gX, B, Ci, Co, st);
    if (rc != FNO_OK) return rc;
  }
  if (gw != nullptr) {
    if (!X) { set_error("fno_mix_bwd: X required for gW"); return FNO_E_ARG; }
    for (int c = 0; c < nc; ++c)
      if (!gw[c]) { set_error("fno_mix_bwd: corner gradient %d is NULL", c); return FNO_E_ARG; }
    int rc = launch_mix_bwd_weight(p, X, gY, gw, B, Ci, Co, st);
    if (rc != FNO_OK) return rc;
  }
  return FNO_OK;
}

}  // extern "C"
