// Dispatcher of the streaming fused NFP kernels: geometry check, dtype selection, entry points used
// by the C ABI (nfp_capi.cu).  The kernels themselves live in nfp_stream_impl.cuh.
#include <stdlib.h>
#include <string.h>

#include "nfp_split.h"
#include "nfp_stream.h"

namespace nfp {
namespace stream {
std::atomic<unsigned long long*> g_debug_stamps{nullptr};
}
namespace {

bool geometry_ok(const KParams& P, int measure) {
  return measure == NFPB200_COSINE && P.stride == 1 && P.dil == 1 && P.pad == P.R &&
         P.mode != NFPB200_PAD_CIRCULAR;
}

int op_mode(int op) {
  switch (op) {
    case NFPB200_OP_FORWARD: return stream::MODE_FWD;
    case NFPB200_OP_BACKWARD: return stream::MODE_BWD;
    case NFPB200_OP_POOL_FORWARD: return stream::MODE_POOL_FWD;
    default: return stream::MODE_POOL_BWD;
  }
}

// the cluster-split kernels (nfp_split_impl.cuh) take every problem their planner accepts; the one-CTA-per-image
// ring kernels (nfp_stream_impl.cuh) remain for the rest and for A/B runs (NFPB200_FUSED_IMPL=stream)
bool split_ok(const KParams& P, int dtype, int mode) {
  static const bool want_split = [] {
    const char* e = getenv("NFPB200_FUSED_IMPL");
    return e && strcmp(e, "split") == 0;
  }();
  if (!want_split && !P.force_split) return false;
  if (P.rin) return false;  // multi-radius launches: ring kernels only
  switch (dtype) {
    case NFPB200_F32: return split::plan_f32(P, mode).ok;
    case NFPB200_BF16: return split::plan_bf16(P, mode).ok;
    default: return false;   // NFPB200_F16: the cluster-split kernels carry no fp16 instantiation
  }
}

int run(const KParams& P, int dtype, int mode, stream::StreamArgs a, cudaStream_t s) {
  if (split_ok(P, dtype, mode)) {
    split::SplitArgs sa{};
    sa.x = a.x; sa.gy = a.gy; sa.y = a.y; sa.gx = a.gx;
    sa.g_gap_x = a.g_gap_x; sa.g_gap_nfp = a.g_gap_nfp; sa.gap_x = a.gap_x; sa.gap_nfp = a.gap_nfp;
    sa.B = P.B; sa.C = P.C;
    sa.pad_mode = P.mode; sa.similarity = P.similarity; sa.eps = P.eps;
    sa.x_early = a.x_early;
    sa.y_f32 = P.y_f32;
    sa.dbg = stream::g_debug_stamps.load(std::memory_order_relaxed);
    return dtype == NFPB200_BF16 ? split::launch_bf16(P, mode, sa, s) : split::launch_f32(P, mode, sa, s);  // never F16
  }
  a.B = P.B; a.C = P.C;
  a.pad_mode = P.mode; a.similarity = P.similarity; a.eps = P.eps;
  a.y_f32 = P.y_f32;
  a.kin = P.Kin; a.rin = P.rin;
  a.dbg = stream::g_debug_stamps.load(std::memory_order_relaxed);
  switch (dtype) {
    case NFPB200_F32: return stream::launch_f32(P, mode, a, s);
    case NFPB200_BF16: return stream::launch_bf16(P, mode, a, s);
    case NFPB200_F16: return stream::launch_f16(P, mode, a, s);
    default: return NFPB200_EINVAL;
  }
}

}  // namespace

bool stream_supported(const KParams& P, int dtype, int measure, int op) {
  if (!geometry_ok(P, measure)) return false;
  const int mode = op_mode(op);
  if (dtype == NFPB200_F16) {
    // the ring kernels serve fp16 exactly where they serve bf16 (same element size, same plans); a problem the
    // cluster-split kernels would take for bf16 (NFPB200_PATH_SPLIT, NFPB200_FUSED_IMPL=split) is not served
    return !P.force_split && !split_ok(P, NFPB200_BF16, mode) && stream::plan_ok_f16(P, mode);
  }
  if (split_ok(P, dtype, mode)) return true;
  if (P.force_split) return false;
  return dtype == NFPB200_BF16 ? stream::plan_ok_bf16(P, mode) : stream::plan_ok_f32(P, mode);
}

const char* stream_name(const KParams& P, int dtype, int measure, int op) {
  (void)measure;
  const bool sp = split_ok(P, dtype, op_mode(op));
  const char* nm = "fused/stream";
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) nm = sp ? "fused/split_" #H_ "x" #W_ "_r" #R_ : "fused/stream_" #H_ "x" #W_ "_r" #R_;
  NFP_STREAM_SHAPES(X)
#undef X
  return nm;
}

int stream_forward(const KParams& P, int dtype, const void* x, void* y, const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.y = y;
  return run(P, dtype, stream::MODE_FWD, a, ctx.stream);
}
int stream_backward(const KParams& P, int dtype, const void* x, const void* gy, void* gx, const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.gy = gy; a.gx = gx;
  a.x_early = P.x_stable;
  return run(P, dtype, stream::MODE_BWD, a, ctx.stream);
}
int stream_pool_forward(const KParams& P, int dtype, const void* x, float* gap_x, float* gap_nfp,
                        const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.gap_x = gap_x; a.gap_nfp = gap_nfp;
  return run(P, dtype, stream::MODE_POOL_FWD, a, ctx.stream);
}
// fused nfp_pooling head on the ring kernels (the cluster-split experiment does not carry it)
bool stream_head_supported(const KParams& P, int dtype, int measure, int op) {
  return stream_supported(P, dtype, measure, op) && !split_ok(P, dtype, op_mode(op)) && P.K % 4 == 0;
}
int stream_head_forward(const KParams& P, int dtype, const void* x, const float* proj_w, const float* proj_b, float* out,
                        float* gap_x, float* gap_nfp, const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.gap_x = gap_x; a.gap_nfp = gap_nfp;
  a.proj_w = proj_w; a.proj_b = proj_b; a.head_out = out;
  return run(P, dtype, stream::MODE_POOL_FWD, a, ctx.stream);
}
int stream_head_backward(const KParams& P, int dtype, const void* x, const float* proj_w, const float* proj_b,
                         const float* gap_x, const float* gap_nfp, const float* g_out, void* gx, const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.gx = gx;
  a.gap_x = const_cast<float*>(gap_x); a.gap_nfp = const_cast<float*>(gap_nfp);   // read-only here: the forward's results
  a.proj_w = proj_w; a.proj_b = proj_b; a.head_gout = g_out;
  a.x_early = P.x_stable;
  a.ggx_tma = 0;
  return run(P, dtype, stream::MODE_POOL_BWD, a, ctx.stream);
}
int stream_pool_backward(const KParams& P, int dtype, const void* x, const float* g_gap_x, const float* g_gap_nfp,
                         void* gx, const LaunchCtx& ctx) {
  stream::StreamArgs a{};
  a.x = x; a.g_gap_x = g_gap_x; a.g_gap_nfp = g_gap_nfp; a.gx = gx;
  a.x_early = P.x_stable;
  a.ggx_tma = (P.C % 4 == 0) && (reinterpret_cast<uintptr_t>(g_gap_x) % 16 == 0);
  return run(P, dtype, stream::MODE_POOL_BWD, a, ctx.stream);
}

}  // namespace nfp
