/*
 * fno_sm100.h -- C ABI of libfno_sm100.so: the B200 (sm_100a) implementation of the FNO
 * spectral-convolution training path of mehrdadmmz/SciML-PDE.
 *
 * The reference has no FFI: its seam is the Python nn.Module protocol, and all arithmetic is
 * delegated to PyTorch library calls.  Each entry point below states the reference call site(s)
 * (path:line under /root/reference/pdebench/models) whose work it replaces.  The host-side
 * mirror of the reference modules (sciml-pde_b200/fno_b200) binds exactly these symbols through
 * ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into caller-owned memory (the torch caching allocator
 *     owns all bytes); the library owns only immutable twiddle tables inside a plan;
 *   - real tensors are float32, complex tensors are interleaved (re, im) float32 pairs
 *     (= torch.complex64 storage); all tensors are dense/contiguous in the stated layout;
 *   - every compute call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *     synchronises, never allocates: safe under CUDA-graph capture and from PyTorch's autograd
 *     thread; plans may be shared between threads once created;
 *   - return value: 0 = ok, < 0 = error (FNO_E_*); fno_last_error() gives the thread-local text.
 *     There is no CPU fallback: on a device that is not sm_100 every call fails with FNO_E_ARCH.
 *
 * Spectrum layout ("retained modes"): for a 2-D plane [H, W] with modes (m1, m2) the kept
 * spectrum is X[2*m1, m2]: rows 0..m1-1 are k1 = 0..m1-1 (reference slice `:m1`, weights1), rows
 * m1..2*m1-1 are k1 = H-m1..H-1 (slice `-m1:`, weights2); columns are k2 = 0..m2-1 of the
 * half spectrum.  3-D: X[2*m1, 2*m2, m3], corner (r1 >= m1) + 2*(r2 >= m2) <-> weights1..4
 * (fno/fno.py:274-285).
 */
#ifndef FNO_SM100_H
#define FNO_SM100_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FNO_OK 0
#define FNO_E_ARG (-1)     /* bad shape / null pointer / unsupported size */
#define FNO_E_CUDA (-2)    /* CUDA runtime error (text in fno_last_error) */
#define FNO_E_ARCH (-3)    /* device is not sm_100 */
#define FNO_E_NOMEM (-4)   /* plan table allocation failed */

typedef struct fno_plan fno_plan;
typedef void* fno_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------------------------- */
int fno_version(void);                         /* 100 * major + minor */
int fno_sm_arch(void);                         /* 100: the only architecture compiled in */
const char* fno_last_error(void);              /* thread-local, never NULL */
unsigned long long fno_launch_count(void);     /* kernels launched by this library so far */
void fno_shutdown(void);                       /* destroys every live plan */
/* Arithmetic mode of the tensor-core kernels (process-wide, read at launch).  FNO_MATH_FP32 (default):
 * every tcgen05.mma operand is split hi + lo and three MMAs accumulate lo*hi + hi*lo + hi*hi ("3xTF32"):
 * results within the fp32-mode tolerance (<= 1e-5 relative).  FNO_MATH_TF32: a single kind::tf32 pass
 * (10-bit mantissa operands, fp32 accumulate); stated bound <= 2e-3 relative on the outputs and gradients of
 * the projection head and of the forward transform's truncated-DFT GEMM (tests/test_kernels_gpu.py::
 * test_head_tf32_mode, ::test_fwd_transform_tf32_mode).  FNO_MATH_BF16: every MMA operand is rounded to bfloat16
 * (8-bit significand), one pass, fp32 accumulate -- the arithmetic of a bf16 tensor-core MMA, issued on the tf32 datapath
 * (bf16 values are tf32 values), so it runs at tf32-mode speed; stated bound <= 2e-2 relative (::test_*_bf16_mode).
 * The FP32 CUDA-core kernels are not affected.  Returns the previous mode, or a negative error code.                   */
#define FNO_MATH_FP32 0
#define FNO_MATH_TF32 1
#define FNO_MATH_BF16 2
int fno_set_math_mode(int mode);
int fno_get_math_mode(void);

/* ---- plans: immutable twiddle tables for one transform geometry ---------------------------- */
/* 2-D plane [H, W], modes (m1, m2); requires 2*m1 <= H, m2 <= W/2+1, m1 <= 32.              */
int fno_plan2d_create(int device, int H, int W, int m1, int m2, fno_plan** out);
/* 3-D volume [D1, D2, D3], modes (m1, m2, m3); 2*m1 <= D1, 2*m2 <= D2, m3 <= D3/2+1.        */
int fno_plan3d_create(int device, int D1, int D2, int D3, int m1, int m2, int m3, fno_plan** out);
int fno_plan_destroy(fno_plan* plan);
/* bytes of scratch a 3-D transform call needs for `planes` volumes (0 for a 2-D plan).       */
size_t fno_plan_workspace_bytes(const fno_plan* plan, long planes);

/* ---- K1: pruned real-to-complex forward transform ------------------------------------------ */
/* Replaces torch.fft.rfft2(x)[..., kept modes] (fno/fno.py:73, slices :84-89) and, with
 * cmode = 1 / scale = 1/(H*W), the autograd backward of torch.fft.irfft2 (fno/fno.py:92).
 *   x      [planes, H, W] f32
 *   preact optional [planes, H, W] f32: if given the transform input is x * gelu'(preact)
 *          (backward of F.gelu, fno/fno.py:164) and, if ds_out is given, that product is stored
 *   X      [planes, 2*m1, m2] complex64 out, multiplied by scale (and c_k2 if cmode = 1)      */
int fno_sc2d_fwd_transform(const fno_plan* plan, const float* x, const float* preact,
                           float* ds_out, float* X, long planes, int cmode, float scale,
                           fno_stream_t stream);
/* Same contract with caller-provided scratch (fno_sc2d_fwd_workspace_bytes(plan, planes) bytes; 0 means
 * the plan has no use for it): lets the library run the contiguous-axis half as a truncated-DFT GEMM
 * on the tensor cores (tcgen05 kind::tf32, 3xTF32 split) and the strided-axis half on the reduced
 * [H, 2*m2] data.  With work = NULL it is identical to fno_sc2d_fwd_transform.                     */
size_t fno_sc2d_fwd_workspace_bytes(const fno_plan* plan, long planes);
int fno_sc2d_fwd_transform_ws(const fno_plan* plan, const float* x, const float* preact,
                              float* ds_out, float* X, void* work, long planes, int cmode,
                              float scale, fno_stream_t stream);
/* 3-D twin (torch.fft.rfftn, fno/fno.py:262): x [planes, D1, D2, D3] -> X [planes, 2m1, 2m2, m3];
 * work: fno_plan_workspace_bytes(plan, planes) bytes of scratch.                               */
int fno_sc3d_fwd_transform(const fno_plan* plan, const float* x, const float* preact,
                           float* ds_out, float* X, void* work, long planes, int cmode,
                           float scale, fno_stream_t stream);

/* ---- K2: per-mode complex channel mixing ---------------------------------------------------- */
/* compl_mul2d / compl_mul3d (fno/fno.py:66-68, :255-257) for all corners in one launch:
 *   Y[b,o,k] = sum_i X[b,i,k] * Wcorner(k)[i,o,k]
 *   X [B, Ci, M] c64, Y [B, Co, M] c64, M = modes of the plan's retained spectrum;
 *   w[0..ncorners) device pointers to the corner parameters, each [Ci, Co, m1, m2(, m3)] c64
 *   in the reference's own state_dict layout (2 corners for a 2-D plan, 4 for a 3-D plan).     */
int fno_mix_fwd(const fno_plan* plan, const float* X, const float* const* w, float* Y, int B,
                int Ci, int Co, fno_stream_t stream);
/* autograd backward of the einsum: gX[b,i,k] = sum_o gY[b,o,k] conj(W[i,o,k]);
 * gW[i,o,k] = sum_b conj(X[b,i,k]) gY[b,o,k] written per corner into gw[0..ncorners).
 * gX or gw may be NULL to skip that half.                                                      */
int fno_mix_bwd(const fno_plan* plan, const float* X, const float* gY, const float* const* w,
                float* gX, float* const* gw, int B, int Ci, int Co, fno_stream_t stream);
/* 1 if fno_mix_fwd / fno_mix_bwd run this shape on the tensor cores (tcgen05, 3xTF32 in fp32 mode):
 * 32 < max(Ci, Co) <= 64 and an even innermost mode count (BASELINE configs[2], width 64); the
 * entry points fall back to the FP32 kernels for tensors that are not 16-byte aligned.        */
int fno_mix_tc_supported(const fno_plan* plan, int Ci, int Co);

/* ---- K3: zero-padding inverse transform with fused epilogue --------------------------------- */
/* Replaces torch.zeros + slice-assign + torch.fft.irfft2 (fno/fno.py:76-92) and, when `addend`
 * / `apply_gelu` are used, also `x1 + x2` and F.gelu (fno/fno.py:163-164).
 *   Y       [planes, 2*m1, m2] c64
 *   addend  optional [planes, H, W] f32 added to the transform (may alias `out`)
 *   s_out   optional [planes, H, W] f32: receives the pre-activation (transform + addend)
 *   out     [planes, H, W] f32: gelu(pre-activation) if apply_gelu else the pre-activation
 *   cmode = 1, scale = 1/(H*W): irfft2 semantics; cmode = 0, scale = 1: adjoint of K1.        */
int fno_sc2d_inv_transform(const fno_plan* plan, const float* Y, const float* addend,
                           float* s_out, float* out, long planes, int cmode, float scale,
                           int apply_gelu, fno_stream_t stream);
int fno_sc3d_inv_transform(const fno_plan* plan, const float* Y, const float* addend,
                           float* s_out, float* out, void* work, long planes, int cmode,
                           float scale, int apply_gelu, fno_stream_t stream);

/* ---- fused Fourier-layer output: K3 + 1x1-conv bypass + bias + GELU on the tensor cores --------- */
/* Replaces, in ONE pass over the activation, everything after the mode mixing of a Fourier layer
 * (fno/fno.py:76-92 zeros + slice-assign + irfft2, :162 w_l(x), :163 x1 + x2, :164 F.gelu):
 *   s   = irfft2(scatter(Y)) + W a + bias        (pre-activation, optional output s_out)
 *   out = gelu(s) if apply_gelu else s
 * as a tcgen05 GEMM per row of the plane (layer2d_tc.cu): the contiguous-axis inverse DFT, the 1x1
 * convolution and the bias share one accumulator in tensor memory (3xTF32 split: fp32-mode accuracy;
 * FNO_MATH_TF32: single pass).  With transpose_w = 1, cmode = 0, scale = 1, bias = NULL and a = dS,
 * Y = gX it is the data gradient of the layer: K3(gX) + W^T dS (autograd of :161-163).
 *   Y [B, C, 2*m1, m2] c64,  a / s_out / out [B, C, H, W] f32 (a must not alias an output),
 *   W [C, C] (conv weight viewed 2-D), bias [C] or NULL,
 *   work: fno_layer2d_fused_workspace_bytes(plan, B, C) bytes (16-byte aligned).
 * fno_layer2d_fused_supported: 1 if the plan geometry / width can run on this path (W <= 132,
 * 2*m2 <= 32, C <= 31), else 0 -- callers then use fno_pointwise_fwd + fno_sc2d_inv_transform.     */
int fno_layer2d_fused_supported(const fno_plan* plan, int C);
size_t fno_layer2d_fused_workspace_bytes(const fno_plan* plan, int B, int C);
int fno_layer2d_inv_fused(const fno_plan* plan, const float* Y, const float* a, const float* W,
                          const float* bias, float* s_out, float* out, void* work, int B, int C,
                          int cmode, float scale, int apply_gelu, int transpose_w,
                          fno_stream_t stream);

/* ---- 1x1-conv bypass (nn.Conv2d/3d(width, width, 1); fno/fno.py:131-134,162) ----------------- */
/* out[b,o,p] = sum_i W[o,i] in[b,i,p] (+ bias[o]);  transpose != 0: out[b,i,p] = sum_o W[o,i] in[b,o,p]
 *   in [B, Cin, N], out [B, Cout, N], W [Co, Ci] (the conv weight viewed 2-D), N = pixels/sample */
int fno_pointwise_fwd(const float* in, const float* W, const float* bias, float* out, int B,
                      int Co, int Ci, long N, int transpose, fno_stream_t stream);
/* gW[o,i] = sum_{b,p} ds[b,o,p] a[b,i,p];  gb[o] = sum_{b,p} ds[b,o,p].
 * work: fno_pointwise_wgrad_workspace_bytes(B, C, C, N) bytes of scratch.                       */
size_t fno_pointwise_wgrad_workspace_bytes(int B, int Co, int Ci, long N);
int fno_pointwise_wgrad(const float* ds, const float* a, float* gW, float* gb, void* work, int B,
                        int Co, int Ci, long N, fno_stream_t stream);
/* Whole autograd of the 1x1 convolution in one call: gW, gb as above AND the data gradient
 * dx [B, Ci, N] = W^T ds.  When the TMA-fed weight-gradient kernel can carry it (width <= 20, aligned
 * tensors) dx is produced from the ds slabs already staged in shared memory -- ds is read once --;
 * otherwise the call runs fno_pointwise_wgrad followed by fno_pointwise_fwd(transpose = 1).        */
int fno_pointwise_bwd(const float* ds, const float* a, const float* W, float* dx, float* gW, float* gb,
                      void* work, int B, int Co, int Ci, long N, fno_stream_t stream);

/* ---- lift: per-sample normalisation + fc0, written into the trunk layout (SURVEY 8f row f2) ------ */
/* Trunk layout of an activation: h[b, c, r, w], r < R_out rows of pitch Wp floats per channel
 * plane; valid region r < R_in, w < W_in, zero elsewhere.  2-D: (R_in, W_in) = (X, Y), padded by
 * F.pad(x, [0, p, 0, p]) (fno/fno.py:159); 3-D: rows = (X, Y) flattened, W_in = Z, only the last
 * axis padded (fno/fno.py:360).
 *
 * torch.std_mean(x, dim=(1,2,3[,4])) + 1e-7 (fno/fno.py:140-142, :343-345):
 *   x [B, entries, V] f32 (entries = pixels * time steps) -> stats [B, 2, V] = (mean, std + 1e-7)
 *   work: fno_lift_stats_workspace_bytes(B, V) bytes                                             */
size_t fno_lift_stats_workspace_bytes(int B, int V);
int fno_lift_stats(const float* x, float* stats, void* work, int B, long entries, int V,
                   fno_stream_t stream);
/* normalise, reshape to [.., T*V], cat grid, fc0, permute to channel-first, zero pad
 * (fno/fno.py:143-159, :346-360):
 *   x [B, R_in*W_in, T, V], grid [B, R_in*W_in, G], W0 [C, T*V+G], b0 [C] -> h [B, C, R_out, Wp]   */
int fno_lift_fwd(const float* x, const float* grid, const float* stats, const float* W0,
                 const float* b0, float* h, int B, int R_in, int W_in, int R_out, int Wp, int T,
                 int V, int G, int C, fno_stream_t stream);
/* autograd backward of the above w.r.t. fc0: gW0 [C, T*V+G], gb0 [C] from dh [B, C, R_out, Wp].
 * Only the statistics are constants (computed under no_grad, fno/fno.py:140-142); the gradient
 * w.r.t. the model input is fno_lift_dgrad.                                                       */
size_t fno_lift_bwd_workspace_bytes(int T, int V, int G, int C);
int fno_lift_bwd(const float* x, const float* grid, const float* stats, const float* dh, float* gW0,
                 float* gb0, void* work, int B, int R_in, int W_in, int R_out, int Wp, int T, int V,
                 int G, int C, fno_stream_t stream);
/* autograd backward of fno_lift_fwd w.r.t. its data inputs, the statistics held constant:
 *   dx [B, R_in*W_in, T, V]:  dx[b,p,t,v] = (1 / stats[b,1,v]) sum_c W0[c, t*V+v] dh[b, c, off(p)]
 *   dgrid [B, R_in*W_in, G]:  dgrid[b,p,g] = sum_c W0[c, T*V+g] dh[b, c, off(p)]
 * Only the valid region of dh is read.  Either output may be NULL (not both); 1 <= V <= 8.
 * No workspace.                                                                                     */
int fno_lift_dgrad(const float* dh, const float* W0, const float* stats, float* dx, float* dgrid,
                   int B, int R_in, int W_in, int R_out, int Wp, int T, int V, int G, int C,
                   fno_stream_t stream);

/* ---- projection head: unpad, fc1, exact GELU, fc2, de-normalise (SURVEY 8f row f1) ---------------- */
/* fno/fno.py:180-187, :381-389.  h [B, C, R_out, Wp] (trunk layout, read in place), W1 [HID, C],
 * b1 [HID], W2 [V, HID], b2 [V], stats as above -> out [B, R_in*W_in, V]
 *   out = (W2 gelu(W1 h + b1) + b2) * std + mean.   The hidden layer never reaches memory.        */
int fno_head_fwd(const float* h, const float* W1, const float* b1, const float* W2, const float* b2,
                 const float* stats, float* out, int B, int R_in, int W_in, int R_out, int Wp, int C,
                 int HID, int V, fno_stream_t stream);
/* Same contract on the tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM) with a 3xTF32
 * split so that the result stays within fp32-mode tolerance; requires HID = 128, C <= 32, V <= 4.  */
int fno_head_fwd_tc(const float* h, const float* W1, const float* b1, const float* W2,
                    const float* b2, const float* stats, float* out, int B, int R_in, int W_in,
                    int R_out, int Wp, int C, int HID, int V, fno_stream_t stream);
/* backward: dout [B, R_in*W_in, V] -> dh [B, C, R_out, Wp] (zero in the padding), gW1, gb1, gW2,
 * gb2; the hidden layer is recomputed.  HID must be a multiple of 8, <= 128 (the reference
 * hard-codes 128).  work: fno_head_bwd_workspace_bytes(C, HID, V) bytes.                           */
size_t fno_head_bwd_workspace_bytes(int C, int HID, int V);
int fno_head_bwd(const float* h, const float* dout, const float* W1, const float* b1, const float* W2,
                 const float* stats, float* dh, float* gW1, float* gb1, float* gW2, float* gb2,
                 void* work, int B, int R_in, int W_in, int R_out, int Wp, int C, int HID, int V,
                 fno_stream_t stream);
/* Same contract on the tensor cores (head_bwd_tc.cu: the hidden-layer recompute, dh = dpre W1 and
 * gW1 = dpre^T h as tcgen05.mma kind::tf32 with a 3xTF32 split, accumulators in TMEM); requires
 * HID = 128, C <= 23, V <= 4.  Same workspace size.                                                 */
int fno_head_bwd_tc(const float* h, const float* dout, const float* W1, const float* b1,
                    const float* W2, const float* stats, float* dh, float* gW1, float* gb1,
                    float* gW2, float* gb2, void* work, int B, int R_in, int W_in, int R_out, int Wp,
                    int C, int HID, int V, fno_stream_t stream);

/* Wide trunks (24 <= C <= 64; BASELINE configs[2]: width 64), same contract in two tcgen05 launches
 * (head_wide_tc.cu): the hidden-layer recompute + dpre + dh = dpre W1 per 128 positions of the padded
 * plane (h and dpre as A operands in tensor memory), then gW1 | gb1 = dpre^T [h ; 1] with the pixels
 * as K; dpre [B, 128, R_out*Wp] passes through `work`.  Requires HID = 128, V <= 4 and
 * (R_out * Wp) % 4 == 0 (fno_head_bwd_wide_supported); work:
 * fno_head_bwd_wide_workspace_bytes(B, R_out, Wp, C, V) bytes, 16-byte aligned.
 * fno_head_fwd_wide_tc: the forward (contract of fno_head_fwd) for HID = 128, C <= 64, V <= 4.     */
int fno_head_fwd_wide_tc(const float* h, const float* W1, const float* b1, const float* W2,
                         const float* b2, const float* stats, float* out, int B, int R_in, int W_in,
                         int R_out, int Wp, int C, int HID, int V, fno_stream_t stream);
int fno_head_bwd_wide_supported(int R_out, int Wp, int C, int HID, int V);
size_t fno_head_bwd_wide_workspace_bytes(int B, int R_out, int Wp, int C, int V);
int fno_head_bwd_wide_tc(const float* h, const float* dout, const float* W1, const float* b1,
                         const float* W2, const float* stats, float* dh, float* gW1, float* gb1,
                         float* gW2, float* gb2, void* work, int B, int R_in, int W_in, int R_out,
                         int Wp, int C, int HID, int V, fno_stream_t stream);

/* ---- device-resident windowed dataset (SURVEY 8f row f4) ----------------------------------------- */
/* Replaces the per-item HDF5 read + host-side slicing of the reference loaders
 * (fno/utils_2d_rd_baseline.py:59-102): traj [n_traj, pixels, T, V] stays on the GPU (time-inner), item b of
 * a batch is (traj_idx[b], t_start[b]) (both device arrays) and one copy kernel writes
 *   xx [B, pixels, initial_step, V] = traj[traj_idx[b], :, t_start[b] : +initial_step, :]
 *   yy [B, pixels, rollout, V]      = traj[traj_idx[b], :, t_start[b]+initial_step : +rollout, :]     */
int fno_window_gather(const float* traj, const long long* traj_idx, const int* t_start, float* xx,
                      float* yy, int B, long npix, int T, int V, int initial_step, int rollout,
                      fno_stream_t stream);
/* The two-head joint model's batch (fno_aux/utils_2d_rd.py items, flattened as fno_train_aux.py:251-256 does):
 * traj_aux [n_traj, A, pixels, T, V] holds the A auxiliary trajectories of each primary trajectory, and one launch writes
 * the JOINED window the trunk runs on, primary rows first:
 *   xj [B + B*A, pixels, initial_step, V]: row b = primary window of item b,
 *                                          row B + b*A + k = window of traj_aux[traj_idx[b], k] at t_start[b]
 *   yy [B, pixels, rollout, V],  yy_aux [B*A, pixels, rollout, V]: the targets in the same order.
 * The (item, stream) of an auxiliary row is computed in the kernel.  A = 0 is fno_window_gather (traj_aux, yy_aux may be
 * NULL).  FNO_E_ARG for A < 0, a NULL traj_aux / yy_aux with A > 0, a window longer than T, element counts >= 2^32 or
 * more than 65535 rows, and an output that overlaps a store (checked against the extent of its first trajectory). */
int fno_window_gather_joint(const float* traj, const float* traj_aux, const long long* traj_idx,
                            const int* t_start, float* xj, float* yy, float* yy_aux, int B, int A,
                            long npix, int T, int V, int initial_step, int rollout, fno_stream_t stream);

/* ---- SpectralConv1d (named by north_star; the reference tree has no 1-D layer, so this follows the 2-D layer's
 * conventions, fno/fno.py:35-92, one dimension down) ---------------------------------------------------------------- */
/* X[r, k] = scale * c_k * sum_n x[r, n] exp(-2 pi i k n / N), k < m: pruned torch.fft.rfft(x)[..., :m]; with cmode = 1,
 * scale = 1/N the backward of fno_sc1d_inv_transform.  x [rows, N] f32, X [rows, m] complex64 interleaved. */
int fno_sc1d_fwd_transform(const float* x, float* X, long rows, int N, int m, int cmode, float scale,
                           fno_stream_t stream);
/* y[r, n] = scale * sum_k c_k Re(Y[r, k] exp(+2 pi i k n / N)) (+ addend): torch.fft.irfft of the zero-padded spectrum
 * (cmode = 1, scale = 1/N: c_0 = 1, c_k = 2, c_{N/2} = 1, Im of DC / Nyquist ignored); cmode = 0, scale = 1: the backward
 * of fno_sc1d_fwd_transform. */
int fno_sc1d_inv_transform(const float* Y, const float* addend, float* y, long rows, int N, int m, int cmode,
                           float scale, fno_stream_t stream);
/* einsum("bix,iox->box") over the m retained modes (X [B, Ci, m], W [Ci, Co, m], Y [B, Co, m], complex64) and its
 * gradients gX = sum_o gY conj(W), gW = sum_b conj(X) gY (either may be NULL). */
int fno_mix1d_fwd(const float* X, const float* W, float* Y, int B, int Ci, int Co, int m, fno_stream_t stream);
int fno_mix1d_bwd(const float* X, const float* gY, const float* W, float* gX, float* gW, int B, int Ci, int Co,
                  int m, fno_stream_t stream);

/* ---- on-device evaluation (SURVEY 8f row f4) -------------------------------------------------------- */
/* metric_func(pred, target, if_mean=True, Lx, Ly, Lz, iLow, iHigh) of pdebench/models/metrics.py:164-306 for fields in the
 * loaders' layout pred, target [B, nx, ny(, nz), T, V] (2-D: nz = 1):
 *   out[0..7] = RMSE, normalised RMSE, RMSE of the conserved variables, maximum error, RMSE at the boundaries,
 *               RMSE in Fourier space (low / middle / high band; NaN for an empty band, as the reference's empty mean)
 *   out[8+t]  = sqrt(mean over (b, grid, v) of (pred-target)^2) per time step: the `val_l2_time` term of metrics.py:386-393
 * `work`: fno_metric_workspace_bytes(...) bytes of device scratch (zeroed by the call). */
size_t fno_metric_workspace_bytes(int B, int nx, int ny, int nz, int T, int V);
int fno_metric_func(const float* pred, const float* target, void* work, float* out, int B, int nx, int ny,
                    int nz, int T, int V, float Lx, float Ly, float Lz, int iLow, int iHigh,
                    fno_stream_t stream);
/* The autoregressive window shift of the rollout loop, `xx = torch.cat((xx[..., 1:, :], pred), dim=-2)`
 * (metrics.py:344): xx, xx_out [points, T0, V], pred [points, 1, V]; xx_out != xx. */
int fno_window_shift(const float* xx, const float* pred, float* xx_out, long points, int T0, int V,
                     fno_stream_t stream);
/* Its adjoint, for training through a rollout: g [points, T0, V] -> gxx [points, T0, V] with
 * gxx[.., 0, :] = 0 and gxx[.., t, :] = g[.., t-1, :], and gpred [points, 1, V] = g[.., T0-1, :].
 * Either output may be NULL (not both); gxx != g.                                                   */
int fno_window_shift_bwd(const float* g, float* gxx, float* gpred, long points, int T0, int V,
                         fno_stream_t stream);
/* The same shift over the two-head model's joined window xx [points, T0, V] (primary points first,
 * then auxiliary ones): point p takes its new last frame from pred_a [points_a, 1, V] when
 * p < points_a and from pred_b [points - points_a, 1, V] otherwise, so that both streams are fed
 * back without splitting or re-joining the window.  0 <= points_a <= points; pred_a (pred_b) may be
 * NULL when points_a == 0 (== points); xx_out aliases no input.  fno_window_shift is the
 * points_a == points case of the same kernel.                                                      */
int fno_window_shift_split(const float* xx, const float* pred_a, const float* pred_b, float* xx_out,
                           long points_a, long points, int T0, int V, fno_stream_t stream);
/* Its adjoint: gxx as for fno_window_shift_bwd, gpred_a / gpred_b = g[.., T0-1, :] of their points.
 * Any output may be NULL (not all of them); no output aliases g.                                   */
int fno_window_shift_split_bwd(const float* g, float* gxx, float* gpred_a, float* gpred_b,
                               long points_a, long points, int T0, int V, fno_stream_t stream);

/* ---- step tail: loss, gradient clipping, Adam, LR schedule (SURVEY 8f row f3) --------------------- */
/* nrmse(out, target).mean() of fno/train.py:34-40,:266-267 for out / target [B, P, V] (P = pixels x
 * output steps): loss[0] = mean_{b,v} ( mean_p (out-y)^2 / (1e-7 + mean_p y^2) ).
 * work: fno_nrmse_workspace_bytes(B, V) bytes, kept for the backward call.                          */
size_t fno_nrmse_workspace_bytes(int B, int V);
int fno_nrmse_fwd(const float* out, const float* target, float* loss, void* work, int B, long P,
                  int V, fno_stream_t stream);
/* dout = gscale[0] * d loss / d out (gscale: device scalar, NULL = 1).                              */
int fno_nrmse_bwd(const float* out, const float* target, const void* work, const float* gscale,
                  float* dout, int B, long P, int V, fno_stream_t stream);
/* fno/train.py:251-259,:273-278 without the host round trip: total_norm over all chunks,
 * clip_value = max(hparams[7], hparams[8] * total_norm), clip_grad_norm_ coefficient, then
 * Adam with coupled L2 weight decay and (if hparams[2] = T_max > 0) the CosineAnnealingLR value of
 * this step, all driven by the device-resident step counter state[0].
 *   chunks   device array of { float* p; const float* g; float* m; float* v; int n; float lr0; }
 *            (fno_opt_chunk_bytes() each, n <= fno_opt_chunk_floats()); complex tensors as real pairs; lr0 = base
 *            learning rate of the chunk's parameter group (0 = hparams[0]): the three Adam groups of the joint loop
 *            (fno_aux/fno_train_aux.py:175-179) share one schedule factor
 *   partials device scratch, nchunks floats
 *   state    device float[8]: step, total_norm, clip_coef, lr, 1-beta1^t, 1-beta2^t, clip_value, clipped_norm
 *   hparams  device float[12]: lr0, eta_min, T_max, beta1, beta2, eps, weight_decay, clip_floor, clip_frac,
 *            sched_extra = scheduler steps taken besides the one per optimizer step (fno/train.py:340 steps the
 *            CosineAnnealingLR once more per epoch), 1 - beta1 and 1 - beta2 evaluated in double, then rounded
 *            (what torch.optim.Adam multiplies by; 1.0f - 0.999f differs from it by 1.3e-5)                */
int fno_opt_chunk_floats(void);
size_t fno_opt_chunk_bytes(void);
int fno_clip_adam_step(const void* chunks, int nchunks, float* partials, float* state,
                       const float* hparams, fno_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FNO_SM100_H */
