// Planar NFP kernels for sm_100a: cosine measure, stride 1, dilation 1, padding = R, ANY map size and channel
// count -- the shapes the streaming fused kernels (nfp_stream_impl.cuh) do not cover, in particular the large,
// shallow maps of the reference's multi-stage heads (models/texture_pooling.py:211-268: 16x112x112, 24x56x56,
// 40x28x28 ...).  An image's tables do not fit in shared memory there, so the work is cut into ROW BANDS instead of
// images.  Thread = pixel, every access coalesced along the plane, gather form throughout: no atomics,
// bit-reproducible.  Two forms:
//
//   band    ("planar/band", planes and row groups 16-byte aligned) ONE launch each way, no workspace: a CTA owns TH map
//           rows of one image and fetches them plus R halo rows of EVERY channel with TMA bulk copies (cp.async.bulk,
//           one per channel: the rows of a plane are contiguous) onto one mbarrier; inverse norms of the slab's pixels,
//           the dots of every band pixel with its whole window, the forward values or the k x k stencil coefficients
//           (closed form of ATen's cosine_similarity backward, SURVEY.md 8 a3) and the stencil application all run out of
//           that slab -- x is read from HBM once per launch, the per-pixel tables / coefficient planes never exist.
//           Pooled mode (GAP(NFP(x)) alone, nfpb200_pooled_map_*): the same band kernels sum the K values per CTA in a
//           fixed order into per-band partials (+ one tiny kernel that adds them in band order), and the backward reads the
//           upstream gradient as K fp32 constants per image instead of a map.
//   scalar  ("planar/table", any shape) separate launches exchanging per-pixel tables through the caller's workspace:
//             table    T[b][v][p]   v = 0: |x_p|^2,  v = 1..K/2: dot(x_p, x_q) for the "forward" window neighbours q,
//                                   v = K/2+1: 1 / max(|x_p|, eps)
//             forward  y[b][n][p]   = dot(p, v_n) / (max(|p|,eps) max(|v_n|,eps)),  v_n = padded tap n of p (nfp.py:150-159)
//             coef     Wd[b][o][p]  the k x k stencil of the backward, gather form
//             apply    gx[b][c][p]  = sum_o Wd[o][p] * x[c][p + off(o)]
//           forward = table + forward (2 launches); backward = table + coef + apply (3 launches, x re-read from L2).
// The window radius is a template parameter: all tap / offset loops are unrolled and the per-thread arrays live in
// registers.
#include <utility>

#include "nfp_common.cuh"
#include "nfp_ptx.cuh"

namespace nfp {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxR = 2;  // wider windows take the generic kernels (the unrolled fold code grows as k^4)

struct PlanarParams {
  int B, C, H, W, P, mode, similarity;
  float eps;
  int kin;  // multi-radius launch (desc.inner_R = 1 with R = 2): 8 planes of the radius-1 map in front of y / gy (band kernels)
};

template <int R>
struct Win {
  static constexpr int k = 2 * R + 1, KK = k * k, K = KK - 1, CTR = R * k + R, ND = K / 2, NV = ND + 1;
  static constexpr int NPL = NV + 1;  // table planes per image (the last one: inverse clamped norm)
};

// pixel (pr + dy, pc + dx) when inside the map, else -1
__device__ __forceinline__ int window_pixel(int pr, int pc, int dy, int dx, const PlanarParams& q) {
  const int r = pr + dy, c = pc + dx;
  return (r >= 0 && r < q.H && c >= 0 && c < q.W) ? r * q.W + c : -1;
}

// The padded tap (dy, dx) of pixel (pr, pc): the pixel it lands on (-1 = implicit zero) and the window entry of
// (pr, pc) that pixel corresponds to (reflect / replicate fold an outside tap back INTO the window).
template <int R>
__device__ __forceinline__ int tap_landing(int pr, int pc, int dy, int dx, const PlanarParams& q, int& o) {
  const int vr = map_index(pr + dy, q.H, q.mode), vc = map_index(pc + dx, q.W, q.mode);
  o = (vr - pr + R) * (2 * R + 1) + (vc - pc + R);
  return (vr < 0 || vc < 0) ? -1 : vr * q.W + vc;
}

// dot(x_p, x_v), v = window entry o of p (o != centre), from the symmetric table of one image
template <int R>
__device__ __forceinline__ float table_dot(const float* __restrict__ tb, int p, int v, int o, int P) {
  constexpr int CTR = Win<R>::CTR;
  return o > CTR ? tb[(size_t)(o - CTR) * P + p] : tb[(size_t)(CTR - o) * P + v];
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_table_kernel(const T* __restrict__ x, float* __restrict__ tab,
                                                                PlanarParams q) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, CTR = Wn::CTR, ND = Wn::ND;
  const int p = blockIdx.x * kThreads + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= q.P) return;
  const int pr = p / q.W, pc = p - pr * q.W;
  int off[ND];  // forward directions: window entries after the centre; outside the map: 0 (result discarded)
  bool in[ND];
  float acc[ND + 1];
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    const int o = CTR + 1 + d;
    const int v = window_pixel(pr, pc, o / k - R, o % k - R, q);
    in[d] = v >= 0;
    off[d] = in[d] ? v - p : 0;
    acc[d + 1] = 0.f;
  }
  acc[0] = 0.f;
  const T* pl = x + (size_t)b * q.C * q.P + p;
#pragma unroll(R == 1 ? 4 : (R == 2 ? 2 : 1))
  for (int c = 0; c < q.C; ++c, pl += q.P) {
    const float xc = to_f32(pl[0]);
    acc[0] = fmaf(xc, xc, acc[0]);
#pragma unroll
    for (int d = 0; d < ND; ++d) acc[d + 1] = fmaf(xc, to_f32(pl[off[d]]), acc[d + 1]);
  }
  float* tb = tab + (size_t)b * Wn::NPL * q.P + p;
  tb[0] = acc[0];
#pragma unroll
  for (int d = 0; d < ND; ++d) tb[(size_t)(d + 1) * q.P] = in[d] ? acc[d + 1] : 0.f;
  tb[(size_t)Wn::NV * q.P] = 1.f / fmaxf(sqrtf(acc[0]), q.eps);
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_forward_kernel(const float* __restrict__ tab, T* __restrict__ y,
                                                                  PlanarParams q) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, KK = Wn::KK, CTR = Wn::CTR;
  const int p = blockIdx.x * kThreads + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= q.P) return;
  const int pr = p / q.W, pc = p - pr * q.W;
  const float* tb = tab + (size_t)b * Wn::NPL * q.P;
  const float* inv = tb + (size_t)Wn::NV * q.P;
  const float ip = inv[p];
  T* yb = y + (size_t)b * Wn::K * q.P + p;
  // pixels at least R away from every border: every tap lands on its own window entry
  const bool interior = pr >= R && pr < q.H - R && pc >= R && pc < q.W - R;
#pragma unroll
  for (int t = 0; t < KK; ++t) {
    if (t == CTR) continue;
    const int dy = t / k - R, dx = t % k - R;
    float yv = 0.f;
    if (interior) {
      const int v = p + dy * q.W + dx;
      yv = table_dot<R>(tb, p, v, t, q.P) * (ip * inv[v]);
    } else {
      int o;
      const int v = tap_landing<R>(pr, pc, dy, dx, q, o);
      if (v >= 0) yv = (o == CTR ? tb[p] : table_dot<R>(tb, p, v, o, q.P)) * (ip * inv[v]);
    }
    if (!q.similarity) yv = 1.f - yv;
    yb[(size_t)(t < CTR ? t : t - 1) * q.P] = from_f32<T>(yv);
  }
}

// Fold maps: fy[i] = window row (0..k-1, relative to pixel row ar) the tap row i of a pixel in map row ar lands on,
// -1 = dropped (zero padding); same rule for columns.  Padding folds rows and columns independently.
template <int R>
__device__ __forceinline__ void fold_map(int a, int n, int mode, int (&f)[2 * R + 1]) {
#pragma unroll
  for (int i = 0; i < 2 * R + 1; ++i) {
    const int v = map_index(a + i - R, n, mode);
    f[i] = v < 0 ? -1 : v - a + R;
  }
}
// Upstream-gradient mass of the taps of a pixel (gya = gy + its index) that land on its window entry (oy, ox).
template <typename T, int R>
__device__ __forceinline__ float folded_taps(const T* __restrict__ gya, const int (&fy)[2 * R + 1],
                                             const int (&fx)[2 * R + 1], int oy, int ox, int P) {
  constexpr int k = 2 * R + 1, CTR = R * k + R;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < k; ++i)
#pragma unroll
    for (int j = 0; j < k; ++j) {
      if (i * k + j != CTR && fy[i] == oy && fx[j] == ox) {
        const int t = i * k + j;
        s += to_f32(gya[(size_t)(t < CTR ? t : t - 1) * P]);
      }
    }
  return s;
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_coef_kernel(const float* __restrict__ tab, const T* __restrict__ gy,
                                                               float* __restrict__ wd, PlanarParams q) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, KK = Wn::KK, K = Wn::K, CTR = Wn::CTR;
  const int p = blockIdx.x * kThreads + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= q.P) return;
  const int pr = p / q.W, pc = p - pr * q.W;
  const float sgn = q.similarity ? 1.f : -1.f;
  const float* tb = tab + (size_t)b * Wn::NPL * q.P;
  const float* inv = tb + (size_t)Wn::NV * q.P;
  const T* gyb = gy + (size_t)b * K * q.P;
  float* wb = wd + (size_t)b * KK * q.P + p;
  const float t0 = tb[p], ip = inv[p];
  const float nrm = sqrtf(t0);
  const float rnp = nrm > 0.f ? ip / nrm : 0.f;  // 1 / (N_p |x_p|): the norm term of ATen's backward, 0 at x = 0
  // pixels at least 2R away from every border: neither p nor any window neighbour has a folded tap
  const bool interior = pr >= 2 * R && pr < q.H - 2 * R && pc >= 2 * R && pc < q.W - 2 * R;
  float s_dot = 0.f, sw = 0.f;
  if (interior) {
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      if (o == CTR) continue;
      const int v = p + (o / k - R) * q.W + (o % k - R);
      const int n = o < CTR ? o : o - 1;  // the direct tap of p towards v, and v's direct tap back
      const float s = to_f32(gyb[(size_t)n * q.P + p]) + to_f32(gyb[(size_t)(K - 1 - n) * q.P + v]);
      const float w = sgn * s * ip * inv[v];
      s_dot = fmaf(w, table_dot<R>(tb, p, v, o, q.P), s_dot);
      wb[(size_t)o * q.P] = w;
    }
  } else {
    // S[p][o] = (taps of p folded onto p + off(o)) + (taps of q = p + off(o) folded onto p).  The row fold map of q
    // depends on q's row only, the column map on its column only: k + k maps cover the whole window.
    int FY[k][k], FX[k][k];
#pragma unroll
    for (int d = 0; d < k; ++d) {
      fold_map<R>(pr + d - R, q.H, q.mode, FY[d]);
      fold_map<R>(pc + d - R, q.W, q.mode, FX[d]);
    }
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      if (o == CTR) continue;
      const int oy = o / k, ox = o % k;
      const int v = window_pixel(pr, pc, oy - R, ox - R, q);
      float w = 0.f;
      if (v >= 0) {
        const float s = folded_taps<T, R>(gyb + p, FY[R], FX[R], oy, ox, q.P) +
                        folded_taps<T, R>(gyb + v, FY[oy], FX[ox], k - 1 - oy, k - 1 - ox, q.P);
        w = sgn * s * ip * inv[v];
        s_dot = fmaf(w, table_dot<R>(tb, p, v, o, q.P), s_dot);
      }
      wb[(size_t)o * q.P] = w;
    }
    // taps of p that land on p itself (replicate padding): y = <p,p>/(N N), gradient 2 G (1/N^2 - y/(N |p|)) x_p
    sw = 2.f * sgn * folded_taps<T, R>(gyb + p, FY[R], FX[R], R, R, q.P) * ip * ip;
  }
  wb[(size_t)CTR * q.P] = sw - rnp * (s_dot + sw * t0);
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_apply_kernel(const T* __restrict__ x, const float* __restrict__ wd,
                                                                T* __restrict__ gx, PlanarParams q) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, KK = Wn::KK;
  const int p = blockIdx.x * kThreads + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= q.P) return;
  const int pr = p / q.W, pc = p - pr * q.W;
  const float* wb = wd + (size_t)b * KK * q.P + p;
  int off[KK];
  float w[KK];
#pragma unroll
  for (int o = 0; o < KK; ++o) {
    const int v = window_pixel(pr, pc, o / k - R, o % k - R, q);
    off[o] = v >= 0 ? v - p : 0;                  // outside the map: coefficient 0 on the pixel itself
    w[o] = v >= 0 ? wb[(size_t)o * q.P] : 0.f;
  }
  const T* pl = x + (size_t)b * q.C * q.P + p;
  T* gp = gx + (size_t)b * q.C * q.P + p;
#pragma unroll(R == 1 ? 4 : 1)
  for (int c = 0; c < q.C; ++c, pl += q.P, gp += q.P) {
    float acc = 0.f;
#pragma unroll
    for (int o = 0; o < KK; ++o) acc = fmaf(w[o], to_f32(pl[off[o]]), acc);
    gp[0] = from_f32<T>(acc);
  }
}

// ---- fused band kernels: the whole forward / backward of a row band in ONE launch, no workspace -------------------
// A CTA owns TH map rows of one image and fetches them with A >= R halo rows on either side (all channels, TMA bulk
// copies as above).  Everything a band pixel needs lives inside that slab:
//   1. inverse clamped norms of every fetched pixel -> shared memory;
//   2. thread = band pixel: |x_p|^2 and the dots with ALL window neighbours (both directions: dot(p,q) is computed at p
//      and again at q, with the same operands in the same channel order, so both get identical bits);
//   forward: y from those dots and the neighbours' inverse norms;
//   backward: the k x k stencil coefficients in registers (closed form of ATen's backward, gather form; upstream
//      gradients straight from global memory, coalesced along the plane), then gx = stencil(x) out of the same slab.
// x is read from HBM once (plus the halo rows, an L2 hit), gy and gx once; the per-pixel tables / coefficient planes of
// the three-launch form never exist.  No atomics, fixed order: bit-reproducible.
template <typename T, int R>
__device__ __forceinline__ void band_fetch(const T* __restrict__ x, unsigned char* xs, uint64_t* bar, const PlanarParams& q,
                                           int b, int r0, int TH, int A, int& top, int& bot, int& pitch) {
  constexpr int ESZ = (int)sizeof(T);
  top = max(r0 - A, 0);
  bot = min(r0 + TH + A, q.H);   // image rows fetched
  pitch = (TH + 2 * A) * q.W * ESZ;
  if (threadIdx.x == 0) {
    ptx::mbar_init(bar, 1);
    ptx::fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const uint32_t bytes = (uint32_t)((bot - top) * q.W * ESZ);
    if (threadIdx.x == 0) ptx::mbar_expect_tx(bar, bytes * (uint32_t)q.C);
    __syncwarp();
    const T* src = x + (size_t)b * q.C * q.P + (size_t)top * q.W;
    unsigned char* dst = xs + (size_t)(top - (r0 - A)) * q.W * ESZ;
    for (int c = threadIdx.x; c < q.C; c += 32) ptx::bulk_g2s(dst + (size_t)c * pitch, src + (size_t)c * q.P, bytes, bar);
  }
  ptx::mbar_wait(bar, 0);
}

// inverse clamped norm of every fetched pixel (slab rows top - (r0 - A) .. bot - (r0 - A))
template <typename T>
__device__ __forceinline__ void band_norms(const unsigned char* xs, float* inv, const PlanarParams& q, int r0, int A, int top,
                                           int bot, int pitch) {
  constexpr int ESZ = (int)sizeof(T);
  const int first = (top - (r0 - A)) * q.W, last = (bot - (r0 - A)) * q.W;
  for (int t = first + threadIdx.x; t < last; t += blockDim.x) {
    const unsigned char* pl = xs + (size_t)t * ESZ;
    float s = 0.f;
#pragma unroll 4
    for (int c = 0; c < q.C; ++c, pl += pitch) {
      const float v = ptx::ldx<T>(pl);
      s = fmaf(v, v, s);
    }
    inv[t] = 1.f / fmaxf(sqrtf(s), q.eps);
  }
  __syncthreads();
}

// acc[o] = dot(x_p, x_{p + off(o)}) for the in-map window entries (acc[CTR] = |x_p|^2; outside: junk, never used)
template <typename T, int R>
__device__ __forceinline__ void band_dots(const unsigned char* pl, int pitch, int C, const int (&off)[(2 * R + 1) * (2 * R + 1)],
                                          float (&acc)[(2 * R + 1) * (2 * R + 1)]) {
  constexpr int KK = (2 * R + 1) * (2 * R + 1);
#pragma unroll
  for (int o = 0; o < KK; ++o) acc[o] = 0.f;
#pragma unroll(R == 1 ? 4 : 2)
  for (int c = 0; c < C; ++c, pl += pitch) {
    const float xc = ptx::ldx<T>(pl);
#pragma unroll
    for (int o = 0; o < KK; ++o) acc[o] = fmaf(xc, ptx::ldx<T>(pl + off[o]), acc[o]);
  }
}

// Upstream gradient of one image as the band kernels see it.  Multi-radius launch: element (tap n, pixel) of the radius-R
// block plus, for the inner taps, the same tap of the radius-r block in front of it (inner_tap folds to a constant in the
// unrolled tap loops).
template <typename T, int R>
struct GyView {
  const T* __restrict__ outer;
  const T* __restrict__ inner;  // null = single radius
  int P;
  __device__ __forceinline__ float at(int n, int pix) const {
    float v = to_f32(outer[(size_t)n * P + pix]);
    if constexpr (R >= 2) {
      if (inner) {
        const int n1 = inner_tap(n, R, 1);
        if (n1 >= 0) v += to_f32(inner[(size_t)n1 * P + pix]);
      }
    }
    return v;
  }
};
// Upstream gradient of the pooled mode (GAP(NFP(x))): d GAP / d y[n][pix] = g_gap_nfp[b][n] / (H W) for every pixel, kept
// in fp32 whatever the dtype of x (rounded to bf16, its error would be multiplied by per-tap derivatives that cancel to
// far smaller sums near the norm clamp).  `g` points at the image's K values in shared memory.
struct GapGradView {
  const float* g;
  __device__ __forceinline__ float at(int n, int) const { return g[n]; }
};
// View: GyView (map gradient) or GapGradView (pooled mode), anything with at(tap, pixel)
template <int R, typename View>
__device__ __forceinline__ float folded_taps_view(const View& gv, int pix, const int (&fy)[2 * R + 1],
                                                  const int (&fx)[2 * R + 1], int oy, int ox) {
  constexpr int k = 2 * R + 1, CTR = R * k + R;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < k; ++i)
#pragma unroll
    for (int j = 0; j < k; ++j) {
      if (i * k + j != CTR && fy[i] == oy && fx[j] == ox) {
        const int t = i * k + j;
        s += gv.at(t < CTR ? t : t - 1, pix);
      }
    }
  return s;
}

// forward values of one band pixel from its window dots: yv[n], n = tap number
template <int R, bool INTERIOR>
__device__ __forceinline__ void band_forward_pixel(const float (&acc)[(2 * R + 1) * (2 * R + 1)], const float* inv, int ps,
                                                   int p, int pr, int pc, const PlanarParams& q,
                                                   float (&yv)[(2 * R + 1) * (2 * R + 1) - 1]) {
  constexpr int k = 2 * R + 1, KK = k * k, CTR = R * k + R;
  const float ip = inv[ps];
#pragma unroll
  for (int tp = 0; tp < KK; ++tp) {
    if (tp == CTR) continue;
    const int dy = tp / k - R, dx = tp % k - R;
    float v_ = 0.f;
    if constexpr (INTERIOR) {  // at least R away from every border: every tap lands on its own window entry
      v_ = acc[tp] * (ip * inv[ps + dy * q.W + dx]);
    } else {
      int o;
      const int v = tap_landing<R>(pr, pc, dy, dx, q, o);
      if (v >= 0) {
        float d = 0.f;   // acc[o] with a run-time o: select (the array must stay in registers)
#pragma unroll
        for (int oo = 0; oo < KK; ++oo) d = (oo == o) ? acc[oo] : d;
        v_ = d * (ip * inv[ps + (v - p)]);
      }
    }
    if (!q.similarity) v_ = 1.f - v_;
    yv[tp < CTR ? tp : tp - 1] = v_;
  }
}

// the k x k stencil coefficients of one band pixel (closed form of ATen's cosine_similarity backward, gather form):
// w[o] multiplies x[p + off(o)]; outside the map: 0
template <int R, bool INTERIOR, typename View>
__device__ __forceinline__ void band_coefficients(const float (&acc)[(2 * R + 1) * (2 * R + 1)], const float* inv, int ps, int p,
                                                  int pr, int pc, const PlanarParams& q, const View& gv, float sgn,
                                                  float (&w)[(2 * R + 1) * (2 * R + 1)]) {
  constexpr int k = 2 * R + 1, KK = k * k, K = KK - 1, CTR = R * k + R;
  const float t0 = acc[CTR], ip = inv[ps];
  const float nrm = sqrtf(t0);
  const float rnp = nrm > 0.f ? ip / nrm : 0.f;  // 1 / (N_p |x_p|): the norm term of ATen's backward, 0 at x = 0
  float s_dot = 0.f, sw = 0.f;
  if constexpr (INTERIOR) {  // at least 2R away from every border: neither p nor any window neighbour has a folded tap
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      if (o == CTR) continue;
      const int dv = (o / k - R) * q.W + (o % k - R);
      const int n = o < CTR ? o : o - 1;  // the direct tap of p towards v, and v's direct tap back
      const float s = gv.at(n, p) + gv.at(K - 1 - n, p + dv);
      w[o] = sgn * s * ip * inv[ps + dv];
      s_dot = fmaf(w[o], acc[o], s_dot);
    }
  } else {
    int FY[k][k], FX[k][k];
#pragma unroll
    for (int d = 0; d < k; ++d) {
      fold_map<R>(pr + d - R, q.H, q.mode, FY[d]);
      fold_map<R>(pc + d - R, q.W, q.mode, FX[d]);
    }
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      if (o == CTR) continue;
      const int oy = o / k, ox = o % k;
      const int v = window_pixel(pr, pc, oy - R, ox - R, q);
      w[o] = 0.f;
      if (v >= 0) {
        const float s = folded_taps_view<R>(gv, p, FY[R], FX[R], oy, ox) +
                        folded_taps_view<R>(gv, v, FY[oy], FX[ox], k - 1 - oy, k - 1 - ox);
        w[o] = sgn * s * ip * inv[ps + (v - p)];
        s_dot = fmaf(w[o], acc[o], s_dot);
      }
    }
    // taps of p that land on p itself (replicate padding): y = <p,p>/(N N), gradient 2 G (1/N^2 - y/(N |p|)) x_p
    sw = 2.f * sgn * folded_taps_view<R>(gv, p, FY[R], FX[R], R, R) * ip * ip;
  }
  w[CTR] = sw - rnp * (s_dot + sw * t0);
}

// The pixels of a band in two passes: first the INTERIOR ones (at least M pixels away from every border of the map:
// straight-line code, window offsets identical for all threads, i.e. uniform-register address operands), then the few
// border pixels of the band as a compact list (M columns on either side of every row, whole rows at the top / bottom of
// the map) -- so that a warp which merely CONTAINS a border pixel does not drag all its lanes through the fold logic
// (ncu on the one-pass form: 1 080 instructions per 32 pixels, most of them border code run by 57 % of the warps).
struct BandSplit {
  int r0, r1, ir0, ir1, IW, M, W, n_int, n_brd, nbr_top, nbr_rows;
  __device__ BandSplit(int r0_, int TH, int H, int W_, int M_) {
    r0 = r0_; r1 = min(r0_ + TH, H); M = M_; W = W_;
    IW = max(W_ - 2 * M_, 0);
    ir0 = min(max(r0, M_), r1);
    ir1 = max(min(r1, H - M_), ir0);
    if (IW == 0) ir1 = ir0;
    n_int = (ir1 - ir0) * IW;
    nbr_top = ir0 - r0;
    nbr_rows = (r1 - r0) - (ir1 - ir0);
    n_brd = nbr_rows * W_ + (ir1 - ir0) * (W_ - IW);
  }
  __device__ __forceinline__ void interior(int t, int& pr, int& pc) const {
    const int lr = t / IW;
    pr = ir0 + lr;
    pc = M + (t - lr * IW);
  }
  __device__ __forceinline__ void border(int u, int& pr, int& pc) const {
    if (u < nbr_rows * W) {  // whole rows above / below the interior rows
      const int lr = u / W;
      pc = u - lr * W;
      pr = lr < nbr_top ? r0 + lr : ir1 + (lr - nbr_top);
    } else {
      const int e = W - IW, v = u - nbr_rows * W, lr = v / e, j = v - lr * e;
      pr = ir0 + lr;
      pc = j < M ? j : IW + j;
    }
  }
};

// Forward of one band: emit(yv, p) receives the K values of every band pixel p exactly once (map mode stores them, the
// pooled mode sums them).
template <typename T, int R, typename Emit>
__device__ __forceinline__ void band_forward(const T* __restrict__ x, const PlanarParams& q, int TH, int A, Emit&& emit) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, KK = Wn::KK, K = Wn::K, ESZ = (int)sizeof(T);
  extern __shared__ __align__(128) unsigned char sm[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm);
  unsigned char* xs = sm + 16;
  const int b = blockIdx.y, r0 = blockIdx.x * TH;
  int top, bot, pitch;
  band_fetch<T, R>(x, xs, bar, q, b, r0, TH, A, top, bot, pitch);
  float* inv = reinterpret_cast<float*>(xs + (size_t)q.C * pitch);
  band_norms<T>(xs, inv, q, r0, A, top, bot, pitch);
  const BandSplit bs(r0, TH, q.H, q.W, R);
  {
    int off[KK];  // the same for every interior pixel
#pragma unroll
    for (int o = 0; o < KK; ++o) off[o] = ((o / k - R) * q.W + (o % k - R)) * ESZ;
    for (int t = threadIdx.x; t < bs.n_int; t += blockDim.x) {
      int pr, pc;
      bs.interior(t, pr, pc);
      const int p = pr * q.W + pc, ps = (pr - r0 + A) * q.W + pc;   // pixel in the map / in the slab
      float acc[KK], yv[K];
      band_dots<T, R>(xs + (size_t)ps * ESZ, pitch, q.C, off, acc);
      band_forward_pixel<R, true>(acc, inv, ps, p, pr, pc, q, yv);
      emit(yv, p);
    }
  }
  for (int u = threadIdx.x; u < bs.n_brd; u += blockDim.x) {
    int pr, pc;
    bs.border(u, pr, pc);
    const int p = pr * q.W + pc, ps = (pr - r0 + A) * q.W + pc;
    int off[KK];
    float acc[KK], yv[K];
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      const int dy = o / k - R, dx = o % k - R;
      off[o] = window_pixel(pr, pc, dy, dx, q) >= 0 ? (dy * q.W + dx) * ESZ : 0;
    }
    band_dots<T, R>(xs + (size_t)ps * ESZ, pitch, q.C, off, acc);
    band_forward_pixel<R, false>(acc, inv, ps, p, pr, pc, q, yv);
    emit(yv, p);
  }
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_fused_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, PlanarParams q,
                                                                    int TH, int A) {
  constexpr int K = Win<R>::K;
  T* yb0 = y + (size_t)blockIdx.y * (K + q.kin) * q.P;   // multi-radius launch: kin planes of the inner radius in front
  band_forward<T, R>(x, q, TH, A, [&](const float (&yv)[K], int p) {
#pragma unroll
    for (int n = 0; n < K; ++n) {
      const T v = from_f32<T>(yv[n]);
      yb0[(size_t)(n + q.kin) * q.P + p] = v;
      if constexpr (R >= 2) {
        const int n1 = inner_tap(n, R, 1);   // a constant per unrolled n
        if (n1 >= 0 && q.kin) yb0[(size_t)n1 * q.P + p] = v;
      }
    }
  });
}

// Pooled mode: every thread sums the K values of its pixels in registers; the CTA reduces them in a fixed order (shuffle
// tree per warp, then the warps' sums in warp order) and writes its band's partial sums part[b][band][n].  No atomics.
template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_pooled_fwd_kernel(const T* __restrict__ x, float* __restrict__ part,
                                                                     PlanarParams q, int TH, int A) {
  constexpr int K = Win<R>::K;
  __shared__ float red[kThreads / 32][K];
  float s[K];
#pragma unroll
  for (int n = 0; n < K; ++n) s[n] = 0.f;
  band_forward<T, R>(x, q, TH, A, [&](const float (&yv)[K], int) {
#pragma unroll
    for (int n = 0; n < K; ++n) s[n] += yv[n];
  });
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int n = 0; n < K; ++n) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[n] += __shfl_xor_sync(0xffffffffu, s[n], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int n = 0; n < K; ++n) red[warp][n] = s[n];
  }
  __syncthreads();
  if (threadIdx.x < K) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w][threadIdx.x];
    part[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * K + threadIdx.x] = t;
  }
}

// gap_nfp[b][n] = (sum of the band partials, in band order) / (H W)
__global__ void __launch_bounds__(kThreads) planar_pooled_finish_kernel(const float* __restrict__ part,
                                                                        float* __restrict__ gap_nfp, int n_bands, int K,
                                                                        int BK, int P) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= BK) return;
  const int b = i / K, n = i - b * K;
  const float* pb = part + (size_t)b * n_bands * K + n;
  float t = 0.f;
  for (int j = 0; j < n_bands; ++j) t += pb[(size_t)j * K];
  gap_nfp[i] = t / (float)P;
}

// Backward of one band: gx = stencil(x) with the k x k coefficients of every band pixel, the upstream gradient read
// through gv (GyView or GapGradView).
template <typename T, int R, typename View>
__device__ __forceinline__ void band_backward(const T* __restrict__ x, T* __restrict__ gx, const PlanarParams& q, int TH,
                                              int A, const View& gv) {
  using Wn = Win<R>;
  constexpr int k = Wn::k, KK = Wn::KK, ESZ = (int)sizeof(T);
  extern __shared__ __align__(128) unsigned char sm[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm);
  unsigned char* xs = sm + 16;
  const int b = blockIdx.y, r0 = blockIdx.x * TH;
  int top, bot, pitch;
  band_fetch<T, R>(x, xs, bar, q, b, r0, TH, A, top, bot, pitch);
  float* inv = reinterpret_cast<float*>(xs + (size_t)q.C * pitch);
  band_norms<T>(xs, inv, q, r0, A, top, bot, pitch);
  const float sgn = q.similarity ? 1.f : -1.f;
  T* gxb = gx + (size_t)b * q.C * q.P;
  const BandSplit bs(r0, TH, q.H, q.W, 2 * R);
  {
    int off[KK];  // the same for every interior pixel
#pragma unroll
    for (int o = 0; o < KK; ++o) off[o] = ((o / k - R) * q.W + (o % k - R)) * ESZ;
    for (int t = threadIdx.x; t < bs.n_int; t += blockDim.x) {
      int pr, pc;
      bs.interior(t, pr, pc);
      const int p = pr * q.W + pc, ps = (pr - r0 + A) * q.W + pc;
      float acc[KK], w[KK];
      const unsigned char* pl = xs + (size_t)ps * ESZ;
      band_dots<T, R>(pl, pitch, q.C, off, acc);
      band_coefficients<R, true>(acc, inv, ps, p, pr, pc, q, gv, sgn, w);
      T* gp = gxb + p;
#pragma unroll(R == 1 ? 4 : 1)
      for (int c = 0; c < q.C; ++c, pl += pitch, gp += q.P) {
        float a = 0.f;
#pragma unroll
        for (int o = 0; o < KK; ++o) a = fmaf(w[o], ptx::ldx<T>(pl + off[o]), a);
        gp[0] = from_f32<T>(a);
      }
    }
  }
  for (int u = threadIdx.x; u < bs.n_brd; u += blockDim.x) {
    int pr, pc;
    bs.border(u, pr, pc);
    const int p = pr * q.W + pc, ps = (pr - r0 + A) * q.W + pc;
    int off[KK];
    float acc[KK], w[KK];
#pragma unroll
    for (int o = 0; o < KK; ++o) {
      const int dy = o / k - R, dx = o % k - R;
      off[o] = window_pixel(pr, pc, dy, dx, q) >= 0 ? (dy * q.W + dx) * ESZ : 0;
    }
    const unsigned char* pl = xs + (size_t)ps * ESZ;
    band_dots<T, R>(pl, pitch, q.C, off, acc);
    band_coefficients<R, false>(acc, inv, ps, p, pr, pc, q, gv, sgn, w);
    T* gp = gxb + p;
#pragma unroll(R == 1 ? 4 : 1)
    for (int c = 0; c < q.C; ++c, pl += pitch, gp += q.P) {
      float a = 0.f;
#pragma unroll
      for (int o = 0; o < KK; ++o) a = fmaf(w[o], ptx::ldx<T>(pl + off[o]), a);
      gp[0] = from_f32<T>(a);
    }
  }
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_fused_bwd_kernel(const T* __restrict__ x, const T* __restrict__ gy,
                                                                    T* __restrict__ gx, PlanarParams q, int TH, int A) {
  constexpr int K = Win<R>::K;
  const T* gyimg = gy + (size_t)blockIdx.y * (K + q.kin) * q.P;   // multi-radius launch: [kin inner planes | K planes] per image
  const GyView<T, R> gv{gyimg + (size_t)q.kin * q.P, q.kin ? gyimg : nullptr, q.P};
  band_backward<T, R>(x, gx, q, TH, A, gv);
}

// Pooled mode: the upstream gradient is K constants per image (GapGradView), so no pixel reads a gradient from memory.
template <typename T, int R>
__global__ void __launch_bounds__(kThreads) planar_pooled_bwd_kernel(const T* __restrict__ x,
                                                                     const float* __restrict__ g_gap_nfp,
                                                                     T* __restrict__ gx, PlanarParams q, int TH, int A) {
  constexpr int K = Win<R>::K;
  __shared__ float gs[K];
  if (threadIdx.x < K) gs[threadIdx.x] = g_gap_nfp[(size_t)blockIdx.y * K + threadIdx.x] / (float)q.P;   // visible after
  band_backward<T, R>(x, gx, q, TH, A, GapGradView{gs});                                             // band_fetch's barrier
}

// Band geometry: TH rows per CTA (a multiple of the row granule g that keeps every bulk copy 16-byte aligned and
// sized), A >= R halo rows (a multiple of g).  ok = false: this shape takes the scalar three-launch kernels.
struct BandPlan {
  bool ok;
  int TH, A, threads;
  size_t smem;
};
constexpr size_t kBandSmemMax = 100 * 1024;  // two CTAs per SM

inline int gcd_i(int a, int b) { return b ? gcd_i(b, a % b) : a; }

// Fused band kernels: halo rows on both sides plus the inverse-norm slab; taller bands than the three-launch form (the
// halo rows are re-read and their norms recomputed by the neighbouring CTAs: (TH + 2A) / TH of the work)
BandPlan fused_plan(const KParams& P, int esz) {
  BandPlan bp{false, 0, 0, 0, 0};
  const int rowB = P.W * esz;
  if (((size_t)P.H * rowB) % 16) return bp;  // every channel plane must start 16-byte aligned
  const int g = 16 / gcd_i(16, rowB);
  const int A = (P.R + g - 1) / g * g;
  const int Hg = (P.H + g - 1) / g * g;
  auto bytes = [&](int th) { return (size_t)P.C * (th + 2 * A) * rowB + 16 + (size_t)(th + 2 * A) * P.W * sizeof(float); };
  constexpr int th_cap = 8;  // band height before rounding to the row granule
  int TH = (th_cap + g - 1) / g * g;
  if (TH > Hg) TH = Hg;
  while (TH > g && bytes(TH) > kBandSmemMax) TH -= g;
  if (bytes(TH) > kBandSmemMax) return bp;
  while (TH - g >= 4 * A && (long)((P.H + TH - 1) / TH) * P.B < 3 * 148) TH -= g;  // enough CTAs, bounded halo overhead
  if ((size_t)P.C * (TH + 2 * A) * rowB >= (1u << 20)) return bp;  // mbarrier transaction-count range
  bp.ok = true;
  bp.TH = TH;
  bp.A = A;
  bp.threads = TH * P.W >= kThreads ? kThreads : (TH * P.W + 31) / 32 * 32;
  bp.smem = bytes(TH);
  return bp;
}

// Without the opt-in a block gets at most 48 KB of dynamic + static shared memory.  static_smem: the kernel's static
// shared memory (0 for the map kernels; the pooled kernels' reduction table / gradient constants, static_smem_of).
template <typename K>
cudaError_t allow_smem(K kern, size_t smem, size_t static_smem = 0) {
  return smem + static_smem > 48 * 1024
             ? cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBandSmemMax)
             : cudaSuccess;
}
// static shared memory of a kernel as the compiler laid it out (callers keep the answer: it never changes)
template <typename K>
std::pair<cudaError_t, size_t> static_smem_of(K kern) {
  cudaFuncAttributes fa{};
  const cudaError_t e = cudaFuncGetAttributes(&fa, kern);
  return {e, fa.sharedSizeBytes};
}

PlanarParams make(const KParams& P) {
  PlanarParams q{};
  q.B = P.B; q.C = P.C; q.H = P.H; q.W = P.W; q.P = P.H * P.W; q.mode = P.mode; q.similarity = P.similarity;
  q.eps = P.eps;
  q.kin = P.Kin;
  return q;
}
inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
size_t table_bytes(const KParams& P) { return align256((size_t)P.B * (P.K / 2 + 2) * P.H * P.W * sizeof(float)); }
size_t coef_bytes(const KParams& P) { return align256((size_t)P.B * P.k * P.k * P.H * P.W * sizeof(float)); }

template <typename T, int R>
int launch_table(const KParams& P, const PlanarParams& q, const T* x, float* tab, cudaStream_t st) {
  (void)P;
  const dim3 grid((unsigned)((q.P + kThreads - 1) / kThreads), (unsigned)q.B);
  planar_table_kernel<T, R><<<grid, kThreads, 0, st>>>(x, tab, q);
  return 0;
}

template <typename T, int R>
int forward_r(const KParams& P, const T* x, T* y, const LaunchCtx& ctx) {
  const PlanarParams q = make(P);
  const BandPlan fp = fused_plan(P, (int)sizeof(T));
  if (fp.ok) {  // one launch, no workspace
    const dim3 bgrid((unsigned)((q.H + fp.TH - 1) / fp.TH), (unsigned)q.B);
    auto kern = planar_fused_fwd_kernel<T, R>;
    if (cudaError_t e = allow_smem(kern, fp.smem)) return (int)e;
    kern<<<bgrid, fp.threads, fp.smem, ctx.stream>>>(x, y, q, fp.TH, fp.A);
    return (int)cudaGetLastError();
  }
  float* tab = reinterpret_cast<float*>(ctx.ws);
  const dim3 grid((unsigned)((q.P + kThreads - 1) / kThreads), (unsigned)q.B);
  if (int rc = launch_table<T, R>(P, q, x, tab, ctx.stream)) return rc;
  planar_forward_kernel<T, R><<<grid, kThreads, 0, ctx.stream>>>(tab, y, q);
  return (int)cudaGetLastError();
}
template <typename T, int R>
int backward_r(const KParams& P, const T* x, const T* gy, T* gx, const LaunchCtx& ctx) {
  const PlanarParams q = make(P);
  const BandPlan fp = fused_plan(P, (int)sizeof(T));
  if (fp.ok) {  // one launch, no workspace
    const dim3 bgrid((unsigned)((q.H + fp.TH - 1) / fp.TH), (unsigned)q.B);
    auto kern = planar_fused_bwd_kernel<T, R>;
    if (cudaError_t e = allow_smem(kern, fp.smem)) return (int)e;
    kern<<<bgrid, fp.threads, fp.smem, ctx.stream>>>(x, gy, gx, q, fp.TH, fp.A);
    return (int)cudaGetLastError();
  }
  float* tab = reinterpret_cast<float*>(ctx.ws);
  float* wd = reinterpret_cast<float*>(reinterpret_cast<char*>(ctx.ws) + table_bytes(P));
  const dim3 grid((unsigned)((q.P + kThreads - 1) / kThreads), (unsigned)q.B);
  if (int rc = launch_table<T, R>(P, q, x, tab, ctx.stream)) return rc;
  planar_coef_kernel<T, R><<<grid, kThreads, 0, ctx.stream>>>(tab, gy, wd, q);
  planar_apply_kernel<T, R><<<grid, kThreads, 0, ctx.stream>>>(x, wd, gx, q);
  return (int)cudaGetLastError();
}
// pooled mode (band form only): forward = band partials + finish (2 launches, partials in the workspace), backward = one
// launch without workspace
template <typename T, int R>
int pooled_forward_r(const KParams& P, const T* x, float* gap_nfp, const LaunchCtx& ctx) {
  const PlanarParams q = make(P);
  const BandPlan fp = fused_plan(P, (int)sizeof(T));
  if (!fp.ok) return NFPB200_EUNSUPPORTED;
  const int n_bands = (q.H + fp.TH - 1) / fp.TH;
  float* part = reinterpret_cast<float*>(ctx.ws);
  auto kern = planar_pooled_fwd_kernel<T, R>;
  static const auto st = static_smem_of(kern);   // one per instantiation
  if (st.first) return (int)st.first;
  if (cudaError_t e = allow_smem(kern, fp.smem, st.second)) return (int)e;
  kern<<<dim3((unsigned)n_bands, (unsigned)q.B), fp.threads, fp.smem, ctx.stream>>>(x, part, q, fp.TH, fp.A);
  const int BK = q.B * P.K;
  planar_pooled_finish_kernel<<<(BK + kThreads - 1) / kThreads, kThreads, 0, ctx.stream>>>(part, gap_nfp, n_bands, P.K,
                                                                                           BK, q.P);
  return (int)cudaGetLastError();
}
template <typename T, int R>
int pooled_backward_r(const KParams& P, const T* x, const float* g_gap_nfp, T* gx, const LaunchCtx& ctx) {
  const PlanarParams q = make(P);
  const BandPlan fp = fused_plan(P, (int)sizeof(T));
  if (!fp.ok) return NFPB200_EUNSUPPORTED;
  auto kern = planar_pooled_bwd_kernel<T, R>;
  static const auto st = static_smem_of(kern);   // one per instantiation
  if (st.first) return (int)st.first;
  if (cudaError_t e = allow_smem(kern, fp.smem, st.second)) return (int)e;
  kern<<<dim3((unsigned)((q.H + fp.TH - 1) / fp.TH), (unsigned)q.B), fp.threads, fp.smem, ctx.stream>>>(
      x, g_gap_nfp, gx, q, fp.TH, fp.A);
  return (int)cudaGetLastError();
}
template <typename T>
int pooled_forward_t(const KParams& P, const T* x, float* gap_nfp, const LaunchCtx& ctx) {
  switch (P.R) {
    case 1: return pooled_forward_r<T, 1>(P, x, gap_nfp, ctx);
    case 2: return pooled_forward_r<T, 2>(P, x, gap_nfp, ctx);
    default: return NFPB200_EUNSUPPORTED;
  }
}
template <typename T>
int pooled_backward_t(const KParams& P, const T* x, const float* g_gap_nfp, T* gx, const LaunchCtx& ctx) {
  switch (P.R) {
    case 1: return pooled_backward_r<T, 1>(P, x, g_gap_nfp, gx, ctx);
    case 2: return pooled_backward_r<T, 2>(P, x, g_gap_nfp, gx, ctx);
    default: return NFPB200_EUNSUPPORTED;
  }
}

template <typename T>
int forward_t(const KParams& P, const T* x, T* y, const LaunchCtx& ctx) {
  switch (P.R) {
    case 1: return forward_r<T, 1>(P, x, y, ctx);
    case 2: return forward_r<T, 2>(P, x, y, ctx);
    default: return NFPB200_EUNSUPPORTED;
  }
}
template <typename T>
int backward_t(const KParams& P, const T* x, const T* gy, T* gx, const LaunchCtx& ctx) {
  switch (P.R) {
    case 1: return backward_r<T, 1>(P, x, gy, gx, ctx);
    case 2: return backward_r<T, 2>(P, x, gy, gx, ctx);
    default: return NFPB200_EUNSUPPORTED;
  }
}

}  // namespace

bool planar_supported(const KParams& P, int dtype, int measure, int op) {
  if (op != NFPB200_OP_FORWARD && op != NFPB200_OP_BACKWARD) return false;
  if (!(measure == NFPB200_COSINE && P.stride == 1 && P.dil == 1 && P.pad == P.R && P.R <= kMaxR &&
        P.mode != NFPB200_PAD_CIRCULAR && P.B <= 65535))
    return false;
  // multi-radius launches (R = 2 with the radius-1 map): the one-launch band kernels only
  if (P.rin) return P.R == 2 && P.rin == 1 && fused_plan(P, dtype == NFPB200_BF16 ? 2 : 4).ok;
  return true;
}
// pooled map (GAP(NFP(x)), NFPB200_OP_POOLED_MAP_*): the band form only -- other shapes take the generic kernels
bool planar_pooled_supported(const KParams& P, int dtype, int measure) {
  return !P.rin && planar_supported(P, dtype, measure, NFPB200_OP_FORWARD) && fused_plan(P, dtype == NFPB200_BF16 ? 2 : 4).ok;
}
size_t planar_workspace_bytes(const KParams& P, int dtype, int op) {
  const BandPlan fp = fused_plan(P, dtype == NFPB200_BF16 ? 2 : 4);
  if (op == NFPB200_OP_POOLED_MAP_FORWARD)   // the band partials (B, n_bands, K)
    return fp.ok ? align256((size_t)P.B * ((P.H + fp.TH - 1) / fp.TH) * P.K * sizeof(float)) : 0;
  if (op == NFPB200_OP_POOLED_MAP_BACKWARD) return 0;
  if (fp.ok) return 0;
  return op == NFPB200_OP_FORWARD ? table_bytes(P) : table_bytes(P) + coef_bytes(P);
}
int planar_launch_count(const KParams& P, int dtype, int op) {
  if (op == NFPB200_OP_POOLED_MAP_FORWARD) return 2;
  if (op == NFPB200_OP_POOLED_MAP_BACKWARD) return 1;
  if (fused_plan(P, dtype == NFPB200_BF16 ? 2 : 4).ok) return 1;
  return op == NFPB200_OP_FORWARD ? 2 : 3;
}
const char* planar_name(const KParams& P, int dtype, int op) {
  const int esz = dtype == NFPB200_BF16 ? 2 : 4;
  (void)op;
  return fused_plan(P, esz).ok ? "planar/band" : "planar/table";
}

int planar_forward(const KParams& P, int dtype, const void* x, void* y, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16) return forward_t<__nv_bfloat16>(P, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, ctx);
  return forward_t<float>(P, (const float*)x, (float*)y, ctx);
}
int planar_backward(const KParams& P, int dtype, const void* x, const void* gy, void* gx, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return backward_t<__nv_bfloat16>(P, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gy, (__nv_bfloat16*)gx, ctx);
  return backward_t<float>(P, (const float*)x, (const float*)gy, (float*)gx, ctx);
}
int planar_pooled_forward(const KParams& P, int dtype, const void* x, float* gap_nfp, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16) return pooled_forward_t<__nv_bfloat16>(P, (const __nv_bfloat16*)x, gap_nfp, ctx);
  return pooled_forward_t<float>(P, (const float*)x, gap_nfp, ctx);
}
int planar_pooled_backward(const KParams& P, int dtype, const void* x, const float* g_gap_nfp, void* gx,
                           const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return pooled_backward_t<__nv_bfloat16>(P, (const __nv_bfloat16*)x, g_gap_nfp, (__nv_bfloat16*)gx, ctx);
  return pooled_backward_t<float>(P, (const float*)x, g_gap_nfp, (float*)gx, ctx);
}

}  // namespace nfp
