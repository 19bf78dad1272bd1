// Internal interface between the dtype-specific translation units of the streaming fused kernels
// (nfp_stream_f32.cu, nfp_stream_bf16.cu, nfp_stream_f16.cu) and the dispatcher (nfp_stream.cu).
#pragma once

#include <atomic>

#include "nfp_common.cuh"

namespace nfp {
namespace stream {

enum { MODE_FWD = 0, MODE_BWD = 1, MODE_POOL_FWD = 2, MODE_POOL_BWD = 3 };

struct StreamArgs {
  const void* x;
  const void* gy;
  void* y;
  void* gx;
  const float* g_gap_x;
  const float* g_gap_nfp;
  float* gap_x;
  float* gap_nfp;
  // fused nfp_pooling head (NFP_Pooling.py:31-35): out = GAP(x) * (proj_w GAP(NFP(x)) + proj_b)
  const float* proj_w;     // (C, K) fp32, null = plain pooled mode
  const float* proj_b;     // (C) fp32 or null
  float* head_out;         // forward: (B, C) fp32
  const float* head_gout;  // backward: d loss / d out (B, C) fp32; gap_x / gap_nfp then hold the forward's saved results
  int B, C;
  int CC;        // channels per chunk (a whole number of group pairs, divides C)
  int NCH;       // chunks per image
  int nst;       // ring stages
  int resident;  // backward: the image fits in the ring, pass B re-walks the slots of pass A
  int pad_mode, similarity;
  int lanech;    // backward: lane-per-channel pass B (C a multiple of 64, chunks a whole number of 64-channel tasks)
  int x_early;   // backward: x is stable across the preceding launch -> stream it before griddepcontrol.wait
  int nsm;       // SMs of the device: CTAs with blockIdx >= nsm are the second CTA of their SM
  int y_delay_ns, y_stages;  // experiment knobs for those second CTAs (NFPB200_Y_DELAY_NS / NFPB200_Y_STAGES)
  int y_f32;     // forward: y is fp32 regardless of T
  int bdirect;   // backward: per-lane partial tables (no shuffle tree over the channel slots), see Smem
  int gy_bufs;   // backward: upstream-gradient buffers in shared memory (1 when every CTA handles a single image)
  int kin, rin;  // multi-radius launch (desc.inner_R): y / gy carry kin extra channels per image (the radius-rin map) in front
  int ggx_tma;   // pooled backward: g_gap_x rows are 16-byte aligned and sized -> fetched with one bulk copy per image
  float eps;
  unsigned long long* dbg;  // optional: 8 globaltimer stamps per CTA (first image), see nfpb200_debug_phase_timing
};

// the (H, W, R, strip width) shapes with a streaming instantiation
#define NFP_STREAM_SHAPES(X) \
  X(7, 7, 1, 7)              \
  X(14, 14, 1, 7)            \
  X(2, 2, 1, 2)              \
  X(4, 4, 1, 4)              \
  X(7, 7, 2, 7)              \
  X(14, 14, 2, 7)

bool plan_ok_f32(const KParams& P, int mode);
bool plan_ok_bf16(const KParams& P, int mode);
bool plan_ok_f16(const KParams& P, int mode);
int launch_f32(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream);
int launch_bf16(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream);
int launch_f16(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream);
// device buffer set through nfpb200_debug_phase_timing (null = off); atomic, so setting it while another host thread
// launches is a benign race: that launch stamps either into the old buffer, the new one, or not at all
extern std::atomic<unsigned long long*> g_debug_stamps;

}  // namespace stream
}  // namespace nfp
