// fp16-I/O (fp32 accumulate) instantiations of the streaming fused NFP kernels (see nfp_stream_impl.cuh).  Same element
// size as bf16, hence the same chunking and shared-memory plans: fp16 ring coverage is bf16 ring coverage.
#include "nfp_stream_impl.cuh"

namespace nfp {
namespace stream {
bool plan_ok_f16(const KParams& P, int mode) { return plan_ok_dtype<__half>(P, mode); }
int launch_f16(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream) {
  return launch_dtype<__half>(P, mode, a, stream);
}
}  // namespace stream
}  // namespace nfp
