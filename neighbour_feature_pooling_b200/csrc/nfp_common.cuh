// Shared definitions for the NFP kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdint.h>

#include "nfp_b200.h"

namespace nfp {

// how `p` of the NORM measure is evaluated (torch.linalg.norm ord semantics, nfp.py:145)
enum { P_GENERAL = 0, P_ONE = 1, P_TWO = 2, P_INF = 3, P_ZERO = 4 };

// Kernel-side view of nfpb200_desc_t (validated, with derived sizes).
struct KParams {
  int B, C, H, W;
  int R, k, K;          // k = 2R+1, K = k*k-1 (nfp.py:38-39)
  int stride, pad, dil, mode;
  int Ho, Wo;
  int similarity, diff_taps, pkind;
  int layout;           // NFPB200_LAYOUT_*
  long long x_batch_stride, gx_batch_stride;  // NHWC: elements between images (0 = dense)
  int force_split;      // NFPB200_PATH_SPLIT: the cluster-split kernels or nothing
  int y_f32;            // NFPB200_FLAG_Y_F32: forward writes y as fp32 although x is bf16 / fp16
  int x_stable;         // NFPB200_HINT_X_STABLE: x is not an output of the launch that precedes this one
  int rin, Kin;         // multi-radius launch (desc.inner_R): inner radius r (0 = off) and its tap count (2r+1)^2 - 1
  float eps, p, q;
};

// Source index of padded coordinate i (already shifted by -pad); -1 = implicit zero.
// Same rule as F.pad / Conv2d(padding_mode=...) which the reference relies on (nfp.py:42-58).
__host__ __device__ __forceinline__ int map_index(int i, int n, int mode) {
  if (i >= 0 && i < n) return i;
  switch (mode) {
    case NFPB200_PAD_REFLECT:   return i < 0 ? -i : 2 * (n - 1) - i;
    case NFPB200_PAD_REPLICATE: return i < 0 ? 0 : n - 1;
    case NFPB200_PAD_CIRCULAR:  return i < 0 ? i + n : i - n;
    default:                    return -1;
  }
}

// Multi-radius launches (desc.inner_R): tap n of the radius-R window (row-major, centre removed) -> the tap number of the
// same offset in the radius-r window, or -1 when the offset lies outside it.  With padding = radius both windows see the
// same padded pixel at the same offset (reflect / replicate / zeros map an index, whatever the pad width is).
__host__ __device__ __forceinline__ int inner_tap(int n, int R, int r) {
  const int k = 2 * R + 1, o = n < (k * k) / 2 ? n : n + 1;
  const int dy = o / k - R, dx = o % k - R;
  if (dy < -r || dy > r || dx < -r || dx > r) return -1;
  const int k1 = 2 * r + 1, o1 = (dy + r) * k1 + dx + r;
  return o1 < (k1 * k1) / 2 ? o1 : o1 - 1;
}

// tap index t in [0,K) -> (row a, col b) of the k x k window, centre removed, row-major (nfp.py:64-67)
__host__ __device__ __forceinline__ void tap_rc(int t, int k, int K, int& a, int& b) {
  int tt = t < (K >> 1) ? t : t + 1;
  a = tt / k;
  b = tt - a * k;
}

// Every padded coordinate p (frame: i*stride + a*dil - pad) that the padding rule maps onto source coordinate r.
template <class F>
__device__ __forceinline__ void for_each_preimage(int r, int n, int pad, int mode, F f) {
  f(r);
  switch (mode) {
    case NFPB200_PAD_REFLECT:
      if (r >= 1 && r <= pad) f(-r);
      if (r <= n - 2 && n - 1 - r <= pad) f(2 * (n - 1) - r);
      break;
    case NFPB200_PAD_REPLICATE:
      if (r == 0) for (int p = -pad; p < 0; ++p) f(p);
      if (r == n - 1) for (int p = n; p < n + pad; ++p) f(p);
      break;
    case NFPB200_PAD_CIRCULAR:
      if (r - n >= -pad) f(r - n);
      if (r + n <= n - 1 + pad) f(r + n);
      break;
    default: break;
  }
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
// round to nearest: a value beyond 65504 becomes +-inf (as a narrowing copy does); nothing is clamped
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

__device__ __forceinline__ float sgnf(float v) { return (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f); }

// ---- host-side launch plumbing ------------------------------------------------------------

struct LaunchCtx {
  cudaStream_t stream;
  void* ws;
  size_t ws_bytes;
};

// generic (any geometry, any measure) kernels: nfp_generic.cu
size_t generic_workspace_bytes(const KParams& P, int dtype, int measure, int op);
int generic_launch_count(const KParams& P, int dtype, int measure, int op);
int generic_forward(const KParams& P, int dtype, int measure, const void* x, void* y, const LaunchCtx& ctx);
int generic_backward(const KParams& P, int dtype, int measure, const void* x, const void* gy, void* gx,
                     const LaunchCtx& ctx);
int generic_pool_forward(const KParams& P, int dtype, int measure, const void* x, float* gap_x, float* gap_nfp,
                         const LaunchCtx& ctx);
int generic_pool_backward(const KParams& P, int dtype, int measure, const void* x, const float* g_gap_x,
                          const float* g_gap_nfp, void* gx, const LaunchCtx& ctx);

// fused kernels (cosine, stride 1, dilation 1, pad = R; cluster-split and streaming-ring forms): nfp_stream.cu
bool stream_supported(const KParams& P, int dtype, int measure, int op);
const char* stream_name(const KParams& P, int dtype, int measure, int op);
int stream_forward(const KParams& P, int dtype, const void* x, void* y, const LaunchCtx& ctx);
int stream_backward(const KParams& P, int dtype, const void* x, const void* gy, void* gx, const LaunchCtx& ctx);
int stream_pool_forward(const KParams& P, int dtype, const void* x, float* gap_x, float* gap_nfp,
                        const LaunchCtx& ctx);
int stream_pool_backward(const KParams& P, int dtype, const void* x, const float* g_gap_x, const float* g_gap_nfp,
                         void* gx, const LaunchCtx& ctx);


bool stream_head_supported(const KParams& P, int dtype, int measure, int op);
int stream_head_forward(const KParams& P, int dtype, const void* x, const float* proj_w, const float* proj_b, float* out,
                        float* gap_x, float* gap_nfp, const LaunchCtx& ctx);
int stream_head_backward(const KParams& P, int dtype, const void* x, const float* proj_w, const float* proj_b,
                         const float* gap_x, const float* gap_nfp, const float* g_out, void* gx, const LaunchCtx& ctx);

// channels-last ("token") tensor-core kernels (bf16 / fp16, cosine, stride 1, dilation 1, pad = R): nfp_token.cu
bool token_supported(const KParams& P, int dtype, int measure, int op);
const char* token_name(const KParams& P);
int token_run(const KParams& P, int dtype, int op, const void* x, const void* gy, void* y, void* gx, const float* g_gap_x,
              const float* g_gap_nfp, float* gap_x, float* gap_nfp, const LaunchCtx& ctx);

int token_head_run(const KParams& P, int dtype, int op, const void* x, const float* proj_w, const float* proj_b,
                   float* out, float* gap_x, float* gap_nfp, const float* g_out, void* gx, const LaunchCtx& ctx);

// planar kernels (cosine, stride 1, dilation 1, pad = R, any map size): nfp_planar.cu.  Map mode (NFPB200_OP_FORWARD /
// _BACKWARD) in the band and table forms; pooled-map mode (GAP(NFP(x)), NFPB200_OP_POOLED_MAP_*) in the band form only
// (planar_pooled_supported).  Not used by nfpb200_pool_* / nfpb200_head_*.
bool planar_supported(const KParams& P, int dtype, int measure, int op);
bool planar_pooled_supported(const KParams& P, int dtype, int measure);
size_t planar_workspace_bytes(const KParams& P, int dtype, int op);
int planar_launch_count(const KParams& P, int dtype, int op);
const char* planar_name(const KParams& P, int dtype, int op);
int planar_forward(const KParams& P, int dtype, const void* x, void* y, const LaunchCtx& ctx);
int planar_backward(const KParams& P, int dtype, const void* x, const void* gy, void* gx, const LaunchCtx& ctx);
int planar_pooled_forward(const KParams& P, int dtype, const void* x, float* gap_nfp, const LaunchCtx& ctx);
int planar_pooled_backward(const KParams& P, int dtype, const void* x, const float* g_gap_nfp, void* gx,
                           const LaunchCtx& ctx);

// second-order kernels of the cosine measure (JVP, backward of the backward; NCHW, any geometry): nfp_second.cu
size_t second_workspace_bytes(const KParams& P, int op);
int second_jvp(const KParams& P, int dtype, const void* x, const void* v, void* ydot, int rule, const LaunchCtx& ctx);
int second_backward_backward(const KParams& P, int dtype, const void* x, const void* gy, const void* v, void* gx2,
                             const LaunchCtx& ctx);

}  // namespace nfp
