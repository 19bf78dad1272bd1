// extern "C" entry points of libnfp_b200.so -- see include/nfp_b200.h for the contract.
// Validates the descriptor (same error conditions as the reference's Conv2d / reflection_pad2d
// calls, models/pooling/nfp.py:42-58), picks the fused or the generic kernel path and launches.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "nfp_common.cuh"
#include "nfp_stream.h"

using namespace nfp;

namespace {

constexpr int kPathFlags = NFPB200_HINT_X_STABLE | NFPB200_FLAG_Y_F32;

int make_params(const nfpb200_desc_t* d, KParams* out) {
  if (!d || d->struct_bytes != (int32_t)sizeof(nfpb200_desc_t)) return NFPB200_EINVAL;
  if (d->dtype != NFPB200_F32 && d->dtype != NFPB200_BF16 && d->dtype != NFPB200_F16) return NFPB200_EINVAL;
  if (d->B <= 0 || d->C <= 0 || d->H <= 0 || d->W <= 0) return NFPB200_EINVAL;
  if (d->R < 1 || d->stride < 1 || d->dilation < 1 || d->padding < 0) return NFPB200_EINVAL;
  if (d->padding_mode < NFPB200_PAD_ZEROS || d->padding_mode > NFPB200_PAD_CIRCULAR) return NFPB200_EINVAL;
  if (d->measure < 0 || d->measure >= NFPB200_NUM_MEASURES) return NFPB200_EINVAL;
  if ((d->path & ~kPathFlags) < NFPB200_PATH_AUTO || (d->path & ~kPathFlags) > NFPB200_PATH_SPLIT) return NFPB200_EINVAL;
  KParams P{};
  P.B = d->B; P.C = d->C; P.H = d->H; P.W = d->W;
  P.R = d->R; P.k = 2 * d->R + 1; P.K = P.k * P.k - 1;
  P.stride = d->stride; P.pad = d->padding; P.dil = d->dilation; P.mode = d->padding_mode;
  // ATen reflection_pad2d: "Padding size should be less than the corresponding input dimension";
  // circular: "Padding value causes wrapping around more than once."
  if (P.mode == NFPB200_PAD_REFLECT && P.pad > 0 && (P.pad >= P.H || P.pad >= P.W)) return NFPB200_EPADDING;
  if (P.mode == NFPB200_PAD_CIRCULAR && (P.pad > P.H || P.pad > P.W)) return NFPB200_EPADDING;
  const int span = P.dil * (P.k - 1) + 1;
  if (P.H + 2 * P.pad < span || P.W + 2 * P.pad < span) return NFPB200_ESHAPE;
  P.Ho = (P.H + 2 * P.pad - span) / P.stride + 1;
  P.Wo = (P.W + 2 * P.pad - span) / P.stride + 1;
  if (d->layout != NFPB200_LAYOUT_NCHW && d->layout != NFPB200_LAYOUT_NHWC) return NFPB200_EINVAL;
  if (d->inner_R < 0 || d->inner_R >= d->R || d->x_batch_stride < 0 || d->gx_batch_stride < 0) return NFPB200_EINVAL;
  P.rin = d->inner_R;
  P.Kin = d->inner_R ? (2 * d->inner_R + 1) * (2 * d->inner_R + 1) - 1 : 0;
  P.layout = d->layout;
  P.x_batch_stride = d->x_batch_stride;
  P.gx_batch_stride = d->gx_batch_stride;
  if (P.layout == NFPB200_LAYOUT_NHWC) {
    const long long dense = (long long)P.H * P.W * P.C;
    if ((P.x_batch_stride && P.x_batch_stride < dense) || (P.gx_batch_stride && P.gx_batch_stride < dense)) return NFPB200_EINVAL;
    if (P.x_batch_stride % 8 || P.gx_batch_stride % 8) return NFPB200_EALIGN;
  }
  P.similarity = d->similarity != 0;
  P.x_stable = (d->path & NFPB200_HINT_X_STABLE) != 0;
  P.force_split = (d->path & ~kPathFlags) == NFPB200_PATH_SPLIT;
  P.y_f32 = (d->path & NFPB200_FLAG_Y_F32) != 0 && (d->dtype == NFPB200_BF16 || d->dtype == NFPB200_F16);
  P.diff_taps = d->difference_taps != 0;
  P.eps = d->eps; P.p = d->p; P.q = d->q_scs;
  P.pkind = P_GENERAL;
  if (d->measure == NFPB200_NORM) {
    if (d->p == 1.f) P.pkind = P_ONE;
    else if (d->p == 2.f) P.pkind = P_TWO;
    else if (isinf(d->p) && d->p > 0) P.pkind = P_INF;
    else if (d->p == 0.f) P.pkind = P_ZERO;
    else if (!(d->p == d->p) || isinf(d->p)) return NFPB200_EINVAL;
  }
  *out = P;
  return NFPB200_OK;
}

inline bool pooled_map_op(int op) { return op == NFPB200_OP_POOLED_MAP_FORWARD || op == NFPB200_OP_POOLED_MAP_BACKWARD; }
// the pool op whose kernels a pooled-map op reuses on the ring, token and generic paths
inline int pool_op_of(int op) {
  return op == NFPB200_OP_POOLED_MAP_FORWARD ? NFPB200_OP_POOL_FORWARD
                                              : (op == NFPB200_OP_POOLED_MAP_BACKWARD ? NFPB200_OP_POOL_BACKWARD : op);
}
inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
inline bool second_op(int op) { return op == NFPB200_OP_JVP || op == NFPB200_OP_BACKWARD_BACKWARD; }
inline bool valid_op(int op) { return (op >= NFPB200_OP_FORWARD && op <= NFPB200_OP_POOLED_MAP_BACKWARD) || second_op(op); }
constexpr int kPathSecond = 5;

// The second-order ops have one path each (nfp_second.cu), whatever desc->path asks for: cosine, NCHW, single radius.
int second_path(const nfpb200_desc_t* d, const KParams& P) {
  if (d->measure != NFPB200_COSINE || P.layout != NFPB200_LAYOUT_NCHW || P.rin) return NFPB200_EUNSUPPORTED;
  return kPathSecond;
}

// fp16 is served by two kernel families only, the ones the live heads use: the NCHW streaming-ring kernels (2) and the
// channels-last token kernels (4), for every op they carry, on exactly the problems a bf16 descriptor sends to them.
// Everything else -- what bf16 sends to the planar, generic or cluster-split kernels, NFPB200_PATH_GENERIC -- is
// NFPB200_EUNSUPPORTED, and the caller widens to fp32.  Decided here, before any dispatcher that picks kernels by dtype.
int choose_path_f16(const nfpb200_desc_t* d, const KParams& P, int op) {
  const int want = d->path & ~kPathFlags;
  if (want == NFPB200_PATH_GENERIC) return NFPB200_EUNSUPPORTED;
  // multi-radius launches: map mode, ring / token kernels, not under NFPB200_PATH_SPLIT (as for bf16)
  if (P.rin && ((op != NFPB200_OP_FORWARD && op != NFPB200_OP_BACKWARD) || want == NFPB200_PATH_SPLIT))
    return NFPB200_EUNSUPPORTED;
  const int pop = pool_op_of(op);
  if (P.layout == NFPB200_LAYOUT_NHWC) return token_supported(P, NFPB200_F16, d->measure, pop) ? 4 : NFPB200_EUNSUPPORTED;
  return stream_supported(P, NFPB200_F16, d->measure, pop) ? 2 : NFPB200_EUNSUPPORTED;
}

// 4 = token (channels-last), 3 = planar, 2 = fused (cluster-split or streaming-ring kernels), 0 = generic, <0 = error
int choose_path(const nfpb200_desc_t* d, const KParams& P, int op) {
  if (second_op(op)) return second_path(d, P);
  if (d->dtype == NFPB200_F16) return choose_path_f16(d, P, op);
  if (pooled_map_op(op)) {
    // the pool ops' choice (token, ring, generic; inner_R refused), with the row-band kernels' pooled mode taking the
    // shapes whose map mode takes "planar/band" instead of the generic kernels
    const int path = choose_path(d, P, pool_op_of(op));
    const bool generic_forced = (d->path & ~kPathFlags) == NFPB200_PATH_GENERIC;
    return (path == 0 && !generic_forced && planar_pooled_supported(P, d->dtype, d->measure)) ? 3 : path;
  }
  if (P.rin) {  // multi-radius launch: the fused kernels' map modes or nothing
    if (op != NFPB200_OP_FORWARD && op != NFPB200_OP_BACKWARD) return NFPB200_EUNSUPPORTED;
    const int want = d->path & ~kPathFlags;
    if (want == NFPB200_PATH_GENERIC || want == NFPB200_PATH_SPLIT) return NFPB200_EUNSUPPORTED;
    if (P.layout == NFPB200_LAYOUT_NHWC) return token_supported(P, d->dtype, d->measure, op) ? 4 : NFPB200_EUNSUPPORTED;
    if (stream_supported(P, d->dtype, d->measure, op)) return 2;
    if (want == NFPB200_PATH_FUSED) return NFPB200_EUNSUPPORTED;
    return planar_supported(P, d->dtype, d->measure, op) ? 3 : NFPB200_EUNSUPPORTED;   // other map sizes: row-band kernels
  }
  if (P.layout == NFPB200_LAYOUT_NHWC) {
    if ((d->path & ~kPathFlags) == NFPB200_PATH_GENERIC) return NFPB200_EUNSUPPORTED;
    return token_supported(P, d->dtype, d->measure, op) ? 4 : NFPB200_EUNSUPPORTED;
  }
  const int fused = stream_supported(P, d->dtype, d->measure, op) ? 2 : 0;
  const int want = d->path & ~kPathFlags;
  if (want == NFPB200_PATH_FUSED || want == NFPB200_PATH_SPLIT) return fused ? fused : NFPB200_EUNSUPPORTED;
  if (want == NFPB200_PATH_GENERIC) return 0;
  if (fused) return fused;
  // large or odd-sized maps (the multi-stage heads' 112x112 ... 28x28 maps): per-pixel planar kernels
  return planar_supported(P, d->dtype, d->measure, op) ? 3 : 0;
}

size_t path_workspace_bytes(int path, const nfpb200_desc_t* d, const KParams& P, int op) {
  // pooled-map ops on the ring / token kernels: their GAP(x) output (forward) or zero g_gap_x input (backward), (B, C) fp32
  if (pooled_map_op(op) && (path == 2 || path == 4)) return align256((size_t)P.B * P.C * sizeof(float));
  if (path == kPathSecond) return second_workspace_bytes(P, op);
  if (path == 3) return planar_workspace_bytes(P, d->dtype, op);
  if (path == 4) return 0;
  return path ? 0 : generic_workspace_bytes(P, d->dtype, d->measure, op);
}

int check_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return (int)e;
  return major == 10 ? NFPB200_OK : NFPB200_EDEVICE;
}

}  // namespace

extern "C" {

int nfpb200_abi_version(void) { return NFPB200_ABI_VERSION; }

const char* nfpb200_status_string(int status) {
  switch (status) {
    case NFPB200_OK: return "ok";
    case NFPB200_EINVAL: return "invalid argument (null pointer, bad size, unknown enum or descriptor size mismatch)";
    case NFPB200_EPADDING:
      return "Padding size should be less than the corresponding input dimension (reflect), or wraps more than "
             "once (circular)";
    case NFPB200_ESHAPE: return "Kernel size can't be greater than actual input size";
    case NFPB200_EWORKSPACE: return "workspace missing or too small (see nfpb200_workspace_bytes)";
    case NFPB200_EUNSUPPORTED: return "the fused kernels do not cover this problem (use NFPB200_PATH_AUTO)";
    case NFPB200_EDEVICE: return "current CUDA device is not compute capability 10.x (B200, sm_100a)";
    case NFPB200_EALIGN:
      return "misaligned pointer: x, y, gy, gx, proj_w and the workspace must be 16-byte aligned, the fp32 vectors "
             "4-byte aligned";
    default: break;
  }
  if (status > 0) return cudaGetErrorString((cudaError_t)status);
  return "unknown nfpb200 status";
}

int nfpb200_debug_phase_timing(unsigned long long* device_stamps) {
  nfp::stream::g_debug_stamps.store(device_stamps, std::memory_order_relaxed);
  return NFPB200_OK;
}

int nfpb200_output_shape(const nfpb200_desc_t* desc, int32_t* Ho, int32_t* Wo) {
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  if (!Ho || !Wo) return NFPB200_EINVAL;
  *Ho = P.Ho;
  *Wo = P.Wo;
  return NFPB200_OK;
}

int nfpb200_workspace_bytes(const nfpb200_desc_t* desc, int32_t op, size_t* bytes) {
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  if (!bytes || !valid_op(op)) return NFPB200_EINVAL;
  int path = choose_path(desc, P, op);
  if (path < 0) return path;
  *bytes = path_workspace_bytes(path, desc, P, op);
  return NFPB200_OK;
}

int nfpb200_describe_path(const nfpb200_desc_t* desc, int32_t op, char* buf, size_t buf_bytes) {
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  if (!buf || buf_bytes == 0 || !valid_op(op)) return NFPB200_EINVAL;
  int path = choose_path(desc, P, op);
  if (path < 0) return path;
  snprintf(buf, buf_bytes, "%s",
           path == kPathSecond ? (op == NFPB200_OP_JVP ? "second/jvp" : "second/pairs")
           : path == 4 ? token_name(P) : path == 3 ? planar_name(P, desc->dtype, op)
                     : (path == 2 ? stream_name(P, desc->dtype, desc->measure, pool_op_of(op)) : "generic/pairs"));
  return NFPB200_OK;
}

int nfpb200_launch_count(const nfpb200_desc_t* desc, int32_t op, int32_t* launches) {
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  if (!launches || !valid_op(op)) return NFPB200_EINVAL;
  int path = choose_path(desc, P, op);
  if (path < 0) return path;
  if (path == kPathSecond) *launches = op == NFPB200_OP_JVP ? 1 : 2;
  else if (path == 3) *launches = planar_launch_count(P, desc->dtype, op);
  else if (path == 2 || path == 4) *launches = op == NFPB200_OP_POOLED_MAP_BACKWARD ? 2 : 1;   // + the g_gap_x memset
  else *launches = generic_launch_count(P, desc->dtype, desc->measure, op);
  return NFPB200_OK;
}

// The alignment each pointer needs (include/nfp_b200.h), checked before any CUDA call.  16 bytes: x, y, gy, gx and
// proj_w, which the kernels move with bulk copies and 16-byte vector accesses, and the workspace.  4 bytes: the fp32
// vectors gap_x, gap_nfp, g_gap_x, g_gap_nfp, out, g_out and proj_b, which every kernel reads and writes one float at a
// time (the ring kernels' bulk copy of a g_gap_x row is only taken when the row is 16-byte aligned and sized).
static inline bool misaligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }
static inline bool misaligned_f32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) != 0; }

// argument errors (descriptor, path, workspace size) are host-only and come before the first CUDA call
#define NFP_PROLOGUE(OP)                                                                      \
  KParams P;                                                                                  \
  int rc = make_params(desc, &P);                                                             \
  if (rc) return rc;                                                                          \
  const int path = choose_path(desc, P, OP);                                                  \
  if (path < 0) return path;                                                                  \
  const size_t need = path_workspace_bytes(path, desc, P, OP);                                \
  if (need > 0 && (!workspace || workspace_bytes < need)) return NFPB200_EWORKSPACE;          \
  rc = check_device();                                                                        \
  if (rc) return rc;                                                                          \
  LaunchCtx ctx{(cudaStream_t)stream, workspace, workspace_bytes};

int nfpb200_forward(const nfpb200_desc_t* desc, const void* x, void* y, void* workspace, size_t workspace_bytes,
                    void* stream) {
  if (!x || !y) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(y) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_FORWARD)
  if (P.y_f32 && path != 2 && path != 4) return NFPB200_EUNSUPPORTED;
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_FORWARD, x, nullptr, y, nullptr, nullptr, nullptr, nullptr, nullptr, ctx);
  if (path == 3) return planar_forward(P, desc->dtype, x, y, ctx);
  if (path == 2) return stream_forward(P, desc->dtype, x, y, ctx);
  return generic_forward(P, desc->dtype, desc->measure, x, y, ctx);
}

int nfpb200_backward(const nfpb200_desc_t* desc, const void* x, const void* gy, void* gx, void* workspace,
                     size_t workspace_bytes, void* stream) {
  if (!x || !gy || !gx) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(gy) || misaligned(gx) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_BACKWARD)
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_BACKWARD, x, gy, nullptr, gx, nullptr, nullptr, nullptr, nullptr, ctx);
  if (path == 3) return planar_backward(P, desc->dtype, x, gy, gx, ctx);
  if (path == 2) return stream_backward(P, desc->dtype, x, gy, gx, ctx);
  return generic_backward(P, desc->dtype, desc->measure, x, gy, gx, ctx);
}

int nfpb200_pool_forward(const nfpb200_desc_t* desc, const void* x, float* gap_x, float* gap_nfp, void* workspace,
                         size_t workspace_bytes, void* stream) {
  if (!x || !gap_x || !gap_nfp) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned_f32(gap_x) || misaligned_f32(gap_nfp) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_POOL_FORWARD)
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_POOL_FORWARD, x, nullptr, nullptr, nullptr, nullptr, nullptr, gap_x, gap_nfp, ctx);
  if (path == 2) return stream_pool_forward(P, desc->dtype, x, gap_x, gap_nfp, ctx);
  return generic_pool_forward(P, desc->dtype, desc->measure, x, gap_x, gap_nfp, ctx);
}

int nfpb200_pool_backward(const nfpb200_desc_t* desc, const void* x, const float* g_gap_x, const float* g_gap_nfp,
                          void* gx, void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !g_gap_x || !g_gap_nfp || !gx) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(gx) || misaligned_f32(g_gap_x) || misaligned_f32(g_gap_nfp) || misaligned(workspace))
    return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_POOL_BACKWARD)
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_POOL_BACKWARD, x, nullptr, nullptr, gx, g_gap_x, g_gap_nfp, nullptr, nullptr, ctx);
  if (path == 2) return stream_pool_backward(P, desc->dtype, x, g_gap_x, g_gap_nfp, gx, ctx);
  return generic_pool_backward(P, desc->dtype, desc->measure, x, g_gap_x, g_gap_nfp, gx, ctx);
}

// ---- pooled similarity map: GAP(NFP(x)) alone ---------------------------------------------------------------------
int nfpb200_pooled_map_forward(const nfpb200_desc_t* desc, const void* x, float* gap_nfp, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!x || !gap_nfp) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned_f32(gap_nfp) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_POOLED_MAP_FORWARD)
  if (path == 3) return planar_pooled_forward(P, desc->dtype, x, gap_nfp, ctx);
  float* gap_x = static_cast<float*>(workspace);   // ring / token kernels: GAP(x) is written to the workspace
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_POOL_FORWARD, x, nullptr, nullptr, nullptr, nullptr, nullptr, gap_x, gap_nfp, ctx);
  if (path == 2) return stream_pool_forward(P, desc->dtype, x, gap_x, gap_nfp, ctx);
  return generic_pool_forward(P, desc->dtype, desc->measure, x, nullptr, gap_nfp, ctx);
}

int nfpb200_pooled_map_backward(const nfpb200_desc_t* desc, const void* x, const float* g_gap_nfp, void* gx,
                                void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !g_gap_nfp || !gx) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(gx) || misaligned_f32(g_gap_nfp) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_POOLED_MAP_BACKWARD)
  if (path == 3) return planar_pooled_backward(P, desc->dtype, x, g_gap_nfp, gx, ctx);
  if (path == 0) return generic_pool_backward(P, desc->dtype, desc->measure, x, nullptr, g_gap_nfp, gx, ctx);
  // ring / token kernels: a zero g_gap_x (B, C) in the workspace
  float* zero = static_cast<float*>(workspace);
  if (cudaError_t e = cudaMemsetAsync(zero, 0, (size_t)P.B * P.C * sizeof(float), ctx.stream)) return (int)e;
  if (path == 4) return token_run(P, desc->dtype, NFPB200_OP_POOL_BACKWARD, x, nullptr, nullptr, gx, zero, g_gap_nfp, nullptr, nullptr, ctx);
  return stream_pool_backward(P, desc->dtype, x, zero, g_gap_nfp, gx, ctx);
}

// ---- fused nfp_pooling head -------------------------------------------------------------------------------------
static int head_path(const nfpb200_desc_t* desc, const KParams& P, int pool_op) {
  const int want = desc->path & ~kPathFlags;
  if (P.rin) return NFPB200_EUNSUPPORTED;  // multi-radius launches exist in map mode only
  if (P.layout == NFPB200_LAYOUT_NHWC)
    return (want != NFPB200_PATH_GENERIC && P.K % 4 == 0 && token_supported(P, desc->dtype, desc->measure, pool_op))
               ? 4 : NFPB200_EUNSUPPORTED;
  if (want == NFPB200_PATH_GENERIC) return NFPB200_EUNSUPPORTED;
  return stream_head_supported(P, desc->dtype, desc->measure, pool_op) ? 2 : NFPB200_EUNSUPPORTED;
}

int nfpb200_head_supported(const nfpb200_desc_t* desc) {
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  rc = head_path(desc, P, NFPB200_OP_POOL_FORWARD);
  if (rc < 0) return rc;
  rc = head_path(desc, P, NFPB200_OP_POOL_BACKWARD);
  return rc < 0 ? rc : NFPB200_OK;
}

int nfpb200_head_forward(const nfpb200_desc_t* desc, const void* x, const float* proj_w, const float* proj_b, float* out,
                         float* gap_x, float* gap_nfp, void* stream) {
  if (!x || !proj_w || !out || !gap_x || !gap_nfp) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(proj_w) || misaligned_f32(proj_b) || misaligned_f32(out) || misaligned_f32(gap_x) ||
      misaligned_f32(gap_nfp))
    return NFPB200_EALIGN;
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  rc = check_device();
  if (rc) return rc;
  rc = head_path(desc, P, NFPB200_OP_POOL_FORWARD);
  if (rc < 0) return rc;
  LaunchCtx ctx{(cudaStream_t)stream, nullptr, 0};
  if (rc == 4)
    return token_head_run(P, desc->dtype, NFPB200_OP_POOL_FORWARD, x, proj_w, proj_b, out, gap_x, gap_nfp, nullptr, nullptr, ctx);
  return stream_head_forward(P, desc->dtype, x, proj_w, proj_b, out, gap_x, gap_nfp, ctx);
}

int nfpb200_head_backward(const nfpb200_desc_t* desc, const void* x, const float* proj_w, const float* proj_b,
                          const float* gap_x, const float* gap_nfp, const float* g_out, void* gx, void* stream) {
  if (!x || !proj_w || !gap_x || !gap_nfp || !g_out || !gx) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(gx) || misaligned(proj_w) || misaligned_f32(proj_b) || misaligned_f32(gap_x) ||
      misaligned_f32(gap_nfp) || misaligned_f32(g_out))
    return NFPB200_EALIGN;
  KParams P;
  int rc = make_params(desc, &P);
  if (rc) return rc;
  rc = check_device();
  if (rc) return rc;
  rc = head_path(desc, P, NFPB200_OP_POOL_BACKWARD);
  if (rc < 0) return rc;
  LaunchCtx ctx{(cudaStream_t)stream, nullptr, 0};
  if (rc == 4)
    return token_head_run(P, desc->dtype, NFPB200_OP_POOL_BACKWARD, x, proj_w, proj_b, nullptr, const_cast<float*>(gap_x),
                          const_cast<float*>(gap_nfp), g_out, gx, ctx);
  return stream_head_backward(P, desc->dtype, x, proj_w, proj_b, gap_x, gap_nfp, g_out, gx, ctx);
}

// ---- second order of the cosine measure --------------------------------------------------------------------------
int nfpb200_jvp(const nfpb200_desc_t* desc, const void* x, const void* v, void* ydot, int32_t rule, void* workspace,
                size_t workspace_bytes, void* stream) {
  if (!x || !v || !ydot) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(v) || misaligned(ydot) || misaligned(workspace)) return NFPB200_EALIGN;
  if (rule != NFPB200_JVP_FORWARD_AD && rule != NFPB200_JVP_REVERSE) return NFPB200_EINVAL;
  NFP_PROLOGUE(NFPB200_OP_JVP)
  return second_jvp(P, desc->dtype, x, v, ydot, rule, ctx);
}

int nfpb200_backward_backward(const nfpb200_desc_t* desc, const void* x, const void* gy, const void* v, void* gx2,
                              void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !gy || !v || !gx2) return NFPB200_EINVAL;
  if (misaligned(x) || misaligned(gy) || misaligned(v) || misaligned(gx2) || misaligned(workspace)) return NFPB200_EALIGN;
  NFP_PROLOGUE(NFPB200_OP_BACKWARD_BACKWARD)
  return second_backward_backward(P, desc->dtype, x, gy, v, gx2, ctx);
}

}  // extern "C"
