// Second-order kernels of the cosine measure (sm_100a): forward-mode JVP and the backward of the backward.
//
// Same gather architecture as nfp_generic.cu: one thread per (centre, neighbour) pair reads both pixels straight from
// global memory, and the input-side sum is a gather through the inverse index map (for_each_preimage), in a fixed
// order and without atomics, so every result is bit-reproducible.  Any radius, stride, dilation, padding and padding
// mode; NCHW; x, v, gy in fp32, bf16 or fp16, fp32 arithmetic.
//
// Per pair (centre a, neighbour b; v_a, v_b the direction at those pixels), n = ||.||, N = max(n, eps), P = Na Nb,
// y = a.b / P, p = v_a.b + a.v_b:
//   JVP:     y' = p / P - y (t_a a.v_a + t_b b.v_b)
//            reverse rule (the map whose transpose is nfpb200_backward): t = 1 / (N n), 0 at n = 0 -- the clamped norm
//            differentiates as n, as in ATen's cosine_similarity; forward-AD rule: t = 0 where n < eps (a clamped norm
//            has a zero tangent).
//   d<v, gx(x, gy)>/dx, G = +-gy, S = t_a a.v_a + t_b b.v_b, w = t (1/N + 1/n) (x.v / n):
//            centre    += G (k_aa a + k_ab b + k_ava v_a + k_v v_b)
//            neighbour += G (k_bb b + k_ab a + k_bvb v_b + k_v v_a)
//            k_aa = -t_a p / P + y t_a S + y w_a,  k_bb likewise,  k_ab = -S / P,  k_ava = -y t_a,  k_bvb = -y t_b,
//            k_v = 1 / P.  Of the 8 coefficients two pairs coincide: 6 floats per pair are stored.
//            At an all-zero pixel x.v / n is 0/0: NaN in every channel of that pixel, as ATen's norm double backward.
#include "nfp_common.cuh"

namespace nfp {
namespace {

constexpr int kThreads = 256;
constexpr int kCoefs = 6;   // k_aa, k_bb, k_ab, k_ava, k_bvb, k_v (SoA: coef[u * npairs + pair])

inline unsigned blocks_for(long long n) { return (unsigned)((n + kThreads - 1) / kThreads); }

struct Pair {
  int b, t, i, j;
  int off_a, off_b;   // element offset inside one channel plane, -1 = implicit zero
};

__device__ __forceinline__ Pair decode(long long idx, const KParams& P) {
  Pair q;
  q.j = (int)(idx % P.Wo);
  long long r = idx / P.Wo;
  q.i = (int)(r % P.Ho);
  r /= P.Ho;
  q.t = (int)(r % P.K);
  q.b = (int)(r / P.K);
  int a, bb;
  tap_rc(q.t, P.k, P.K, a, bb);
  const int rc = map_index(q.i * P.stride + P.R * P.dil - P.pad, P.H, P.mode);
  const int cc = map_index(q.j * P.stride + P.R * P.dil - P.pad, P.W, P.mode);
  const int rn = map_index(q.i * P.stride + a * P.dil - P.pad, P.H, P.mode);
  const int cn = map_index(q.j * P.stride + bb * P.dil - P.pad, P.W, P.mode);
  q.off_a = (rc < 0 || cc < 0) ? -1 : rc * P.W + cc;
  q.off_b = (rn < 0 || cn < 0) ? -1 : rn * P.W + cn;
  return q;
}

// the seven channel sums of one pair: a.a, b.b, a.b, a.v_a, b.v_b, v_a.b + a.v_b
struct Dots {
  float aa, bb, ab, qa, qb, p;
};

template <typename T>
__device__ __forceinline__ Dots pair_dots(const T* __restrict__ x, const T* __restrict__ v, const Pair& q,
                                          const KParams& P) {
  const int HW = P.H * P.W;
  const size_t img = (size_t)q.b * P.C * HW;
  Dots d{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float pab = 0.f, pba = 0.f;
  for (int ch = 0; ch < P.C; ++ch) {
    const size_t o = img + (size_t)ch * HW;
    const float a = q.off_a >= 0 ? to_f32(x[o + q.off_a]) : 0.f;
    const float va = q.off_a >= 0 ? to_f32(v[o + q.off_a]) : 0.f;
    const float b = q.off_b >= 0 ? to_f32(x[o + q.off_b]) : 0.f;
    const float vb = q.off_b >= 0 ? to_f32(v[o + q.off_b]) : 0.f;
    d.aa = fmaf(a, a, d.aa);
    d.bb = fmaf(b, b, d.bb);
    d.ab = fmaf(a, b, d.ab);
    d.qa = fmaf(a, va, d.qa);
    d.qb = fmaf(b, vb, d.qb);
    pab = fmaf(va, b, pab);
    pba = fmaf(a, vb, pba);
  }
  d.p = pab + pba;
  return d;
}

// 1 / (N n) where the rule keeps the norm's derivative, else 0
__device__ __forceinline__ float tcoef(float n, float N, float eps, int rule) {
  const bool keep = rule == NFPB200_JVP_FORWARD_AD ? n >= eps : n > 0.f;
  return keep ? 1.f / (N * n) : 0.f;
}

template <typename T, typename YT>
__global__ void __launch_bounds__(kThreads) jvp_kernel(const T* __restrict__ x, const T* __restrict__ v,
                                                       YT* __restrict__ ydot, KParams P, int rule, long long npairs) {
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  const Pair q = decode(idx, P);
  const Dots d = pair_dots(x, v, q, P);
  const float na = sqrtf(d.aa), nb = sqrtf(d.bb);
  const float Na = fmaxf(na, P.eps), Nb = fmaxf(nb, P.eps);
  const float Pn = Na * Nb;
  const float y = d.ab / Pn;
  const float yd = d.p / Pn - y * (tcoef(na, Na, P.eps, rule) * d.qa + tcoef(nb, Nb, P.eps, rule) * d.qb);
  ydot[idx] = from_f32<YT>(P.similarity ? yd : -yd);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) bb_pair_kernel(const T* __restrict__ x, const T* __restrict__ v,
                                                           const T* __restrict__ gy, float* __restrict__ coef,
                                                           KParams P, long long npairs) {
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  const Pair q = decode(idx, P);
  const Dots d = pair_dots(x, v, q, P);
  const float G = P.similarity ? to_f32(gy[idx]) : -to_f32(gy[idx]);
  const float na = sqrtf(d.aa), nb = sqrtf(d.bb);
  const float Na = fmaxf(na, P.eps), Nb = fmaxf(nb, P.eps);
  const float Pn = Na * Nb;
  const float y = d.ab / Pn;
  const float ta = tcoef(na, Na, P.eps, NFPB200_JVP_REVERSE), tb = tcoef(nb, Nb, P.eps, NFPB200_JVP_REVERSE);
  const float S = ta * d.qa + tb * d.qb;
  // x.v / n is 0/0 = NaN at an all-zero pixel: NaN in that pixel's channels, as ATen's norm double backward
  const float wa = ta * (1.f / Na + 1.f / na) * (d.qa / na);
  const float wb = tb * (1.f / Nb + 1.f / nb) * (d.qb / nb);
  const float k[kCoefs] = {G * (-ta * d.p / Pn + y * ta * S + y * wa), G * (-tb * d.p / Pn + y * tb * S + y * wb),
                           G * (-S / Pn), G * (-y * ta), G * (-y * tb), G / Pn};
#pragma unroll
  for (int u = 0; u < kCoefs; ++u) coef[u * npairs + idx] = k[u];
}

// one thread per (b, channel, input pixel q): every pair that reads q, as a neighbour tap and as a centre, in a fixed
// order (the order of nfp_generic.cu's gather_kernel); gx2 is written once, in the dtype of x
template <typename T>
__global__ void __launch_bounds__(kThreads) bb_gather_kernel(const T* __restrict__ x, const T* __restrict__ v,
                                                             const float* __restrict__ coef, T* __restrict__ gx2,
                                                             KParams P, long long npairs, long long total) {
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= total) return;
  const int w = (int)(idx % P.W);
  long long r = idx / P.W;
  const int h = (int)(r % P.H);
  r /= P.H;
  const int ch = (int)(r % P.C);
  const int b = (int)(r / P.C);
  const size_t plane = ((size_t)b * P.C + ch) * P.H * P.W;
  const long long HoWo = (long long)P.Ho * P.Wo;
  const float xq = to_f32(x[plane + h * P.W + w]);
  const float vq = to_f32(v[plane + h * P.W + w]);
  const int ctr = P.R * P.dil;
  float acc = 0.f;
  for_each_preimage(h, P.H, P.pad, P.mode, [&](int pr) {
    for_each_preimage(w, P.W, P.pad, P.mode, [&](int pc) {
      // (1) q as the neighbour tap t of output pixel (i, j)
      for (int t = 0; t < P.K; ++t) {
        int a, bb;
        tap_rc(t, P.k, P.K, a, bb);
        const int ti = pr + P.pad - a * P.dil, tj = pc + P.pad - bb * P.dil;
        if (ti < 0 || tj < 0 || ti % P.stride || tj % P.stride) continue;
        const int i = ti / P.stride, j = tj / P.stride;
        if (i >= P.Ho || j >= P.Wo) continue;
        const int rc = map_index(i * P.stride + ctr - P.pad, P.H, P.mode);
        const int cc = map_index(j * P.stride + ctr - P.pad, P.W, P.mode);
        const bool in = rc >= 0 && cc >= 0;
        const float xa = in ? to_f32(x[plane + rc * P.W + cc]) : 0.f;
        const float va = in ? to_f32(v[plane + rc * P.W + cc]) : 0.f;
        const long long pb = (long long)b * P.K * HoWo + t * HoWo + (long long)i * P.Wo + j;
        acc += coef[1 * npairs + pb] * xq + coef[2 * npairs + pb] * xa + coef[4 * npairs + pb] * vq +
               coef[5 * npairs + pb] * va;
      }
      // (2) q as the centre of output pixel (i, j)
      const int ti = pr + P.pad - ctr, tj = pc + P.pad - ctr;
      if (ti >= 0 && tj >= 0 && ti % P.stride == 0 && tj % P.stride == 0) {
        const int i = ti / P.stride, j = tj / P.stride;
        if (i < P.Ho && j < P.Wo) {
          const long long p0 = (long long)b * P.K * HoWo + (long long)i * P.Wo + j;
          for (int t = 0; t < P.K; ++t) {
            int a, bb;
            tap_rc(t, P.k, P.K, a, bb);
            const int rn = map_index(i * P.stride + a * P.dil - P.pad, P.H, P.mode);
            const int cn = map_index(j * P.stride + bb * P.dil - P.pad, P.W, P.mode);
            const bool in = rn >= 0 && cn >= 0;
            const float xb = in ? to_f32(x[plane + rn * P.W + cn]) : 0.f;
            const float vb = in ? to_f32(v[plane + rn * P.W + cn]) : 0.f;
            const long long pb = p0 + t * HoWo;
            acc += coef[0 * npairs + pb] * xq + coef[2 * npairs + pb] * xb + coef[3 * npairs + pb] * vq +
                   coef[5 * npairs + pb] * vb;
          }
        }
      }
    });
  });
  gx2[idx] = from_f32<T>(acc);
}

template <typename T>
int jvp_t(const KParams& P, const void* x, const void* v, void* ydot, int rule, cudaStream_t stream) {
  const long long npairs = (long long)P.B * P.K * P.Ho * P.Wo;
  if (P.y_f32)
    jvp_kernel<T, float><<<blocks_for(npairs), kThreads, 0, stream>>>((const T*)x, (const T*)v, (float*)ydot, P, rule,
                                                                      npairs);
  else
    jvp_kernel<T, T><<<blocks_for(npairs), kThreads, 0, stream>>>((const T*)x, (const T*)v, (T*)ydot, P, rule, npairs);
  return (int)cudaGetLastError();
}

template <typename T>
int bb_t(const KParams& P, const void* x, const void* gy, const void* v, void* gx2, void* ws, cudaStream_t stream) {
  const long long npairs = (long long)P.B * P.K * P.Ho * P.Wo;
  const long long nx = (long long)P.B * P.C * P.H * P.W;
  float* coef = (float*)ws;
  bb_pair_kernel<T><<<blocks_for(npairs), kThreads, 0, stream>>>((const T*)x, (const T*)v, (const T*)gy, coef, P,
                                                                 npairs);
  bb_gather_kernel<T><<<blocks_for(nx), kThreads, 0, stream>>>((const T*)x, (const T*)v, coef, (T*)gx2, P, npairs,
                                                               nx);
  return (int)cudaGetLastError();
}

}  // namespace

size_t second_workspace_bytes(const KParams& P, int op) {
  if (op != NFPB200_OP_BACKWARD_BACKWARD) return 0;
  const size_t npairs = (size_t)P.B * P.K * P.Ho * P.Wo;
  return (kCoefs * sizeof(float) * npairs + 255) & ~(size_t)255;
}

int second_jvp(const KParams& P, int dtype, const void* x, const void* v, void* ydot, int rule, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16) return jvp_t<__nv_bfloat16>(P, x, v, ydot, rule, ctx.stream);
  if (dtype == NFPB200_F16) return jvp_t<__half>(P, x, v, ydot, rule, ctx.stream);
  return jvp_t<float>(P, x, v, ydot, rule, ctx.stream);
}

int second_backward_backward(const KParams& P, int dtype, const void* x, const void* gy, const void* v, void* gx2,
                             const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16) return bb_t<__nv_bfloat16>(P, x, gy, v, gx2, ctx.ws, ctx.stream);
  if (dtype == NFPB200_F16) return bb_t<__half>(P, x, gy, v, gx2, ctx.ws, ctx.stream);
  return bb_t<float>(P, x, gy, v, gx2, ctx.ws, ctx.stream);
}

}  // namespace nfp
