// Geometry- and measure-generic NFP kernels (sm_100a).
//
// These cover every constructor combination of the reference operator
// (models/pooling/nfp.py:16-18): any radius, stride, padding, dilation, padding mode and all 17
// measures, forward and backward.  They read x straight from global memory (L1/L2 provide the
// reuse) with one thread per (centre, neighbour) pair, so they are correct everywhere but not
// tuned; the hot configurations are taken by the fused kernels (nfp_stream_impl.cuh, nfp_token.cu).
//
// Forward:   pair kernel -> y                                   (+ a second pass for attention / scs)
// Backward:  pair kernel -> 5 coefficients per pair (workspace) (+ a second pass for attention / scs)
//            gather kernel (inverse index map, fixed order, no atomics) writes gx in its own dtype.
#include "nfp_common.cuh"

namespace nfp {
namespace {

constexpr int kThreads = 256;

__host__ __device__ constexpr bool is_gram(int M) {
  return M == NFPB200_COSINE || M == NFPB200_DOT || M == NFPB200_ATTENTION || M == NFPB200_GFC ||
         M == NFPB200_PEARSON || M == NFPB200_SCS;
}

// Decoded position of one (centre, neighbour) pair.
struct PairPos {
  int b, t, i, j;
  int off_c, off_n;  // element offset of the pixel inside one channel plane, -1 = implicit zero
};

__device__ __forceinline__ PairPos decode_pair(long long idx, const KParams& P) {
  PairPos q;
  q.j = (int)(idx % P.Wo);
  long long r = idx / P.Wo;
  q.i = (int)(r % P.Ho);
  r /= P.Ho;
  q.t = (int)(r % P.K);
  q.b = (int)(r / P.K);
  int a, bb;
  tap_rc(q.t, P.k, P.K, a, bb);
  int rc = map_index(q.i * P.stride + P.R * P.dil - P.pad, P.H, P.mode);
  int cc = map_index(q.j * P.stride + P.R * P.dil - P.pad, P.W, P.mode);
  int rn = map_index(q.i * P.stride + a * P.dil - P.pad, P.H, P.mode);
  int cn = map_index(q.j * P.stride + bb * P.dil - P.pad, P.W, P.mode);
  q.off_c = (rc < 0 || cc < 0) ? -1 : rc * P.W + cc;
  q.off_n = (rn < 0 || cn < 0) ? -1 : rn * P.W + cn;
  return q;
}

// ---- per-channel accumulation ---------------------------------------------------------------
template <int M>
__device__ __forceinline__ void accum(float c, float n, float (&s)[5], const KParams& P) {
  if constexpr (is_gram(M)) {
    s[0] = fmaf(c, n, s[0]);
    s[1] = fmaf(c, c, s[1]);
    s[2] = fmaf(n, n, s[2]);
  } else if constexpr (M == NFPB200_NORM) {
    float v = P.diff_taps ? c - n : n;
    float a = fabsf(v);
    switch (P.pkind) {
      case P_ONE: s[0] += a; break;
      case P_TWO: s[0] = fmaf(v, v, s[0]); break;
      case P_INF:
        if (a > s[0]) { s[0] = a; s[1] = 1.f; } else if (a == s[0]) { s[1] += 1.f; }
        break;
      case P_ZERO: s[0] += (v != 0.f) ? 1.f : 0.f; break;
      default: s[0] += powf(a, P.p); break;
    }
  } else if constexpr (M == NFPB200_RMSE) {
    float v = P.diff_taps ? c - n : n;
    s[0] = fmaf(v, v, s[0]);
  } else if constexpr (M == NFPB200_GEMAN) {
    float d = (c - n) * (c - n);
    s[0] += d / (d + P.eps);
  } else if constexpr (M == NFPB200_EMD) {
    s[0] += fabsf(c - n);
  } else if constexpr (M == NFPB200_CANBERRA) {
    s[0] += fabsf(c - n) / (fabsf(c) + fabsf(n) + P.eps);
  } else if constexpr (M == NFPB200_HELLINGER || M == NFPB200_SQUAREDCHORD) {
    float t = sqrtf(fabsf(c) + P.eps) - sqrtf(fabsf(n) + P.eps);
    s[0] = fmaf(t, t, s[0]);
  } else if constexpr (M == NFPB200_CHISQUARED1) {
    float d = c - n;
    s[0] += d * d / (fabsf(c) + fabsf(n) + P.eps);
  } else if constexpr (M == NFPB200_CHISQUARED2) {
    float d = c - n;
    s[0] += d * d / (fabsf(c) + P.eps);
  } else if constexpr (M == NFPB200_JEFFREY) {
    float ca = fabsf(c) + P.eps, na = fabsf(n) + P.eps;
    s[0] += ca * logf(ca / na) + na * logf(na / ca);
  } else if constexpr (M == NFPB200_SMITH) {
    float ca = fabsf(c), na = fabsf(n);
    s[0] += fminf(ca, na);
    s[1] += ca;
    s[2] += na;
  }
}

// Channel reduction for one pair.  Pearson is two-pass (means, then centred sums) to avoid the
// cancellation of the one-pass variance formula; s[3], s[4] return the two means.
template <typename T, int M>
__device__ __forceinline__ void reduce_pair(const T* __restrict__ xb, const PairPos& q, const KParams& P,
                                            float (&s)[5]) {
  const int HW = P.H * P.W;
#pragma unroll
  for (int u = 0; u < 5; ++u) s[u] = 0.f;
  const T* pc = q.off_c >= 0 ? xb + q.off_c : nullptr;
  const T* pn = q.off_n >= 0 ? xb + q.off_n : nullptr;
  float cm = 0.f, nm = 0.f;
  if constexpr (M == NFPB200_PEARSON) {
    for (int ch = 0; ch < P.C; ++ch) {
      cm += pc ? to_f32(pc[(size_t)ch * HW]) : 0.f;
      nm += pn ? to_f32(pn[(size_t)ch * HW]) : 0.f;
    }
    cm /= (float)P.C;
    nm /= (float)P.C;
  }
  for (int ch = 0; ch < P.C; ++ch) {
    float c = pc ? to_f32(pc[(size_t)ch * HW]) : 0.f;
    float n = pn ? to_f32(pn[(size_t)ch * HW]) : 0.f;
    accum<M>(c - cm, n - nm, s, P);
  }
  if constexpr (M == NFPB200_PEARSON) { s[3] = cm; s[4] = nm; }
}

// ---- forward value of one pair --------------------------------------------------------------
template <int M>
__device__ __forceinline__ float finalize(const float (&s)[5], const KParams& P) {
  const bool sim = P.similarity != 0;
  if constexpr (M == NFPB200_COSINE) {
    float y = s[0] / (fmaxf(sqrtf(s[1]), P.eps) * fmaxf(sqrtf(s[2]), P.eps));
    return sim ? y : 1.f - y;
  } else if constexpr (M == NFPB200_DOT || M == NFPB200_ATTENTION || M == NFPB200_SCS) {
    return sim ? s[0] : -s[0];  // attention / scs are finished by their second pass
  } else if constexpr (M == NFPB200_GFC) {
    float y = s[0] / (sqrtf(s[1]) * sqrtf(s[2]) + P.eps);
    return sim ? y : -y;
  } else if constexpr (M == NFPB200_PEARSON) {
    float y = s[0] / sqrtf(s[1] * s[2] + P.eps);
    return sim ? y : -y;
  } else if constexpr (M == NFPB200_NORM) {
    float y;
    switch (P.pkind) {
      case P_TWO: y = sqrtf(s[0]); break;
      case P_ONE: case P_INF: case P_ZERO: y = s[0]; break;
      default: y = powf(s[0], 1.f / P.p); break;
    }
    return sim ? -y : y;
  } else if constexpr (M == NFPB200_RMSE) {
    float y = sqrtf(s[0] / (float)P.C);
    return sim ? -y : y;
  } else if constexpr (M == NFPB200_GEMAN) {
    float y = s[0] / (float)P.C;
    return sim ? y : 1.f - y;
  } else if constexpr (M == NFPB200_HELLINGER) {
    float y = sqrtf(0.5f * s[0]);
    return sim ? -y : y;
  } else if constexpr (M == NFPB200_SMITH) {
    float y = 1.f - s[0] / (fminf(s[1], s[2]) + P.eps);
    return sim ? y : -y;
  } else {  // emd, canberra, chisquared1/2, jeffrey, squaredchord: plain sums of distances
    return sim ? -s[0] : s[0];
  }
}

// ---- backward: 5 coefficients per pair, then per-channel derivatives --------------------------
// Gram family:  d/dc = k0*n + k1*c (+ centring for pearson: k3 = mean c, k4 = mean n), d/dn = k0*c + k2*n
// others: measure-specific, see chan_grad().
template <int M>
__device__ __forceinline__ void coefs(const float (&s)[5], float g, const KParams& P, float (&k)[5]) {
  const bool sim = P.similarity != 0;
#pragma unroll
  for (int u = 0; u < 5; ++u) k[u] = 0.f;
  if constexpr (M == NFPB200_COSINE) {
    // ATen cosine_similarity: value uses the clamped norms, the gradient keeps the norm term
    // y*c/(Nc*||c||) (zero for c == 0).  SURVEY.md section 8 row a3.
    float G = sim ? g : -g;
    float nc = sqrtf(s[1]), nn = sqrtf(s[2]);
    float Nc = fmaxf(nc, P.eps), Nn = fmaxf(nn, P.eps);
    float y = s[0] / (Nc * Nn);
    k[0] = G / (Nc * Nn);
    k[1] = nc > 0.f ? -G * y / (Nc * nc) : 0.f;
    k[2] = nn > 0.f ? -G * y / (Nn * nn) : 0.f;
  } else if constexpr (M == NFPB200_DOT) {
    k[0] = sim ? g : -g;
  } else if constexpr (M == NFPB200_ATTENTION) {
    k[0] = s[0];  // raw dot; the softmax pass turns it into d/d dot
  } else if constexpr (M == NFPB200_SCS) {
    k[0] = s[0]; k[1] = sqrtf(s[1]); k[2] = sqrtf(s[2]);  // dot, ||c||, ||n||; the batch pass finishes
  } else if constexpr (M == NFPB200_GFC) {
    float G = sim ? g : -g;
    float nc = sqrtf(s[1]), nn = sqrtf(s[2]);
    float D = nc * nn + P.eps;
    k[0] = G / D;
    k[1] = nc > 0.f ? -G * s[0] / (D * D) * nn / nc : 0.f;
    k[2] = nn > 0.f ? -G * s[0] / (D * D) * nc / nn : 0.f;
  } else if constexpr (M == NFPB200_PEARSON) {
    float G = sim ? g : -g;
    float den = sqrtf(s[1] * s[2] + P.eps);
    float d3 = den * den * den;
    k[0] = G / den;
    k[1] = -G * s[0] * s[2] / d3;
    k[2] = -G * s[0] * s[1] / d3;
    k[3] = s[3];
    k[4] = s[4];
  } else if constexpr (M == NFPB200_NORM) {
    k[0] = sim ? -g : g;
    switch (P.pkind) {
      case P_TWO: k[1] = sqrtf(s[0]); break;
      case P_INF: k[1] = s[0]; k[2] = s[1]; break;
      case P_ONE: case P_ZERO: break;
      default: k[1] = powf(s[0], 1.f / P.p); break;
    }
  } else if constexpr (M == NFPB200_RMSE) {
    float G = sim ? -g : g;
    float y = sqrtf(s[0] / (float)P.C);
    k[0] = G / ((float)P.C * y);  // y == 0 -> inf, and inf*0 = NaN like sqrt'(0) in the reference
  } else if constexpr (M == NFPB200_GEMAN) {
    k[0] = (sim ? g : -g) / (float)P.C;
  } else if constexpr (M == NFPB200_HELLINGER) {
    float G = sim ? -g : g;
    k[0] = G / (4.f * sqrtf(0.5f * s[0]));
  } else if constexpr (M == NFPB200_SMITH) {
    float G = sim ? g : -g;
    float D = fminf(s[1], s[2]) + P.eps;
    float wc = s[1] < s[2] ? 1.f : (s[1] == s[2] ? 0.5f : 0.f);
    k[0] = G / D;
    k[1] = G * s[0] * wc / (D * D);
    k[2] = G * s[0] * (1.f - wc) / (D * D);
  } else {
    k[0] = sim ? -g : g;
  }
}

template <int M>
__device__ __forceinline__ void chan_grad(float c, float n, const float (&k)[5], const KParams& P, float& dc,
                                          float& dn) {
  if constexpr (M == NFPB200_PEARSON) {
    float cc = c - k[3], nc = n - k[4];
    dc = k[0] * nc + k[1] * cc;
    dn = k[0] * cc + k[2] * nc;
  } else if constexpr (is_gram(M)) {
    dc = k[0] * n + k[1] * c;
    dn = k[0] * c + k[2] * n;
  } else if constexpr (M == NFPB200_NORM) {
    float v = P.diff_taps ? c - n : n;
    float dv;
    switch (P.pkind) {
      case P_ONE: dv = k[0] * sgnf(v); break;
      case P_TWO: dv = k[1] > 0.f ? k[0] * v / k[1] : 0.f; break;
      case P_INF: dv = (fabsf(v) == k[1]) ? k[0] * sgnf(v) / k[2] : 0.f; break;
      case P_ZERO: dv = 0.f; break;
      default:
        dv = (v == 0.f || k[1] == 0.f) ? 0.f
                                       : k[0] * sgnf(v) * powf(fabsf(v), P.p - 1.f) / powf(k[1], P.p - 1.f);
        break;
    }
    dc = P.diff_taps ? dv : 0.f;
    dn = P.diff_taps ? -dv : dv;
  } else if constexpr (M == NFPB200_RMSE) {
    float v = P.diff_taps ? c - n : n;
    float dv = k[0] * v;
    dc = P.diff_taps ? dv : 0.f;
    dn = P.diff_taps ? -dv : dv;
  } else if constexpr (M == NFPB200_GEMAN) {
    float d = c - n, den = d * d + P.eps;
    dc = k[0] * 2.f * d * P.eps / (den * den);
    dn = -dc;
  } else if constexpr (M == NFPB200_EMD) {
    dc = k[0] * sgnf(c - n);
    dn = -dc;
  } else if constexpr (M == NFPB200_CANBERRA) {
    float a = fabsf(c - n), s = fabsf(c) + fabsf(n) + P.eps, sg = sgnf(c - n);
    dc = k[0] * (sg / s - a * sgnf(c) / (s * s));
    dn = k[0] * (-sg / s - a * sgnf(n) / (s * s));
  } else if constexpr (M == NFPB200_HELLINGER || M == NFPB200_SQUAREDCHORD) {
    float rc = sqrtf(fabsf(c) + P.eps), rn = sqrtf(fabsf(n) + P.eps), t = rc - rn;
    dc = k[0] * t / rc * sgnf(c);
    dn = -k[0] * t / rn * sgnf(n);
  } else if constexpr (M == NFPB200_CHISQUARED1) {
    float d = c - n, s = fabsf(c) + fabsf(n) + P.eps;
    dc = k[0] * (2.f * d / s - d * d * sgnf(c) / (s * s));
    dn = k[0] * (-2.f * d / s - d * d * sgnf(n) / (s * s));
  } else if constexpr (M == NFPB200_CHISQUARED2) {
    float d = c - n, s = fabsf(c) + P.eps;
    dc = k[0] * (2.f * d / s - d * d * sgnf(c) / (s * s));
    dn = k[0] * (-2.f * d / s);
  } else if constexpr (M == NFPB200_JEFFREY) {
    float ca = fabsf(c) + P.eps, na = fabsf(n) + P.eps;
    dc = k[0] * sgnf(c) * (logf(ca / na) + 1.f - na / ca);
    dn = k[0] * sgnf(n) * (logf(na / ca) + 1.f - ca / na);
  } else if constexpr (M == NFPB200_SMITH) {
    float ca = fabsf(c), na = fabsf(n);
    float mc = ca < na ? 1.f : (ca == na ? 0.5f : 0.f);  // d min(|c|,|n|)/d|c| as torch.minimum splits ties
    dc = sgnf(c) * (-k[0] * mc + k[1]);
    dn = sgnf(n) * (-k[0] * (1.f - mc) + k[2]);
  }
}

// ---- kernels ----------------------------------------------------------------------------------

// y (or raw fp32 values for attention / scs) for every pair
template <typename T, int M>
__global__ void __launch_bounds__(kThreads) pair_forward_kernel(const T* __restrict__ x, T* __restrict__ y,
                                                                float* __restrict__ raw, KParams P,
                                                                long long npairs) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  PairPos q = decode_pair(idx, P);
  float s[5];
  reduce_pair<T, M>(x + (size_t)q.b * P.C * P.H * P.W, q, P, s);
  if constexpr (M == NFPB200_ATTENTION) {
    raw[idx] = s[0];
  } else if constexpr (M == NFPB200_SCS) {
    raw[idx] = s[0];
    raw[npairs + idx] = (sqrtf(s[1]) + P.q) * (sqrtf(s[2]) + P.q);
  } else {
    y[idx] = from_f32<T>(finalize<M>(s, P));
  }
}

// softmax over the K neighbours of every output pixel (nfp.py:202)
template <typename T>
__global__ void __launch_bounds__(kThreads) attention_forward_kernel(const float* __restrict__ raw,
                                                                     T* __restrict__ y, KParams P) {
  long long pix = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long HoWo = (long long)P.Ho * P.Wo;
  if (pix >= (long long)P.B * HoWo) return;
  long long b = pix / HoWo, r = pix % HoWo;
  const float* d = raw + b * P.K * HoWo + r;
  float m = -INFINITY;
  for (int t = 0; t < P.K; ++t) m = fmaxf(m, d[t * HoWo]);
  float z = 0.f;
  for (int t = 0; t < P.K; ++t) z += expf(d[t * HoWo] - m);
  for (int t = 0; t < P.K; ++t) {
    float v = expf(d[t * HoWo] - m) / z;
    y[b * P.K * HoWo + t * HoWo + r] = from_f32<T>(P.similarity ? v : -v);
  }
}

__device__ __forceinline__ float scs_h(float t, float p) {
  float h = sgnf(t) * powf(fabsf(t), p);
  return isfinite(h) ? h : 0.f;  // nan_to_num(nan=0, posinf=0, neginf=0), nfp.py:369
}
__device__ __forceinline__ float scs_dh(float t, float p) {
  if (t == 0.f || !isfinite(t)) return 0.f;
  float h = powf(fabsf(t), p);
  if (!isfinite(h)) return 0.f;
  float d = p * powf(fabsf(t), p - 1.f);
  return isfinite(d) ? d : 0.f;
}

// Sharpened cosine with the reference's cross-batch broadcast (nfp.py:363-374):
// out[b] = mean_{b'} h(dot[b'] / den[b]).
template <typename T>
__global__ void __launch_bounds__(kThreads) scs_forward_kernel(const float* __restrict__ raw, T* __restrict__ y,
                                                               KParams P, long long npairs) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  const long long per = npairs / P.B;
  const long long r = idx % per;
  const float den = raw[npairs + idx];
  float acc = 0.f;
  for (int bp = 0; bp < P.B; ++bp) acc += scs_h(raw[bp * per + r] / den, P.p);
  float v = acc / (float)P.B;
  y[idx] = from_f32<T>(P.similarity ? v : 1.f - v);
}

// coefficients of every pair (SoA: coef[u * npairs + idx]); gy is T (map mode) or fp32 (pooled mode, GT = float)
template <typename T, typename GT, int M>
__global__ void __launch_bounds__(kThreads) pair_coef_kernel(const T* __restrict__ x, const GT* __restrict__ gy,
                                                             float* __restrict__ coef, KParams P,
                                                             long long npairs) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  PairPos q = decode_pair(idx, P);
  float s[5], k[5];
  reduce_pair<T, M>(x + (size_t)q.b * P.C * P.H * P.W, q, P, s);
  coefs<M>(s, to_f32(gy[idx]), P, k);
#pragma unroll
  for (int u = 0; u < 5; ++u) coef[u * npairs + idx] = k[u];
}

// attention: raw dots (coef[0]) -> d/d dot = y_t (G_t - sum_u G_u y_u)
template <typename T>
__global__ void __launch_bounds__(kThreads) attention_coef_kernel(const T* __restrict__ gy,
                                                                  float* __restrict__ coef, KParams P) {
  long long pix = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long HoWo = (long long)P.Ho * P.Wo;
  if (pix >= (long long)P.B * HoWo) return;
  long long b = pix / HoWo, r = pix % HoWo;
  float* d = coef + b * P.K * HoWo + r;
  const T* g = gy + b * P.K * HoWo + r;
  float m = -INFINITY;
  for (int t = 0; t < P.K; ++t) m = fmaxf(m, d[t * HoWo]);
  float z = 0.f;
  for (int t = 0; t < P.K; ++t) z += expf(d[t * HoWo] - m);
  float gs = 0.f;
  const float sg = P.similarity ? 1.f : -1.f;
  for (int t = 0; t < P.K; ++t) gs += sg * to_f32(g[t * HoWo]) * expf(d[t * HoWo] - m) / z;
  for (int t = 0; t < P.K; ++t) {
    float yv = expf(d[t * HoWo] - m) / z;
    d[t * HoWo] = yv * (sg * to_f32(g[t * HoWo]) - gs);
  }
}

// scs: (dot, ||c||, ||n||) in coef[0..2] -> Gram-family coefficients, through the batch coupling.
// coef[3], coef[4] are used as scratch for d/d dot and d/d den so that no pair reads a slot
// another thread has already overwritten.
template <typename T>
__global__ void __launch_bounds__(kThreads) scs_coef_kernel_a(const T* __restrict__ gy, float* __restrict__ coef,
                                                              KParams P, long long npairs) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  const long long per = npairs / P.B;
  const long long r = idx % per;
  const float* dot = coef;
  const float* nc = coef + npairs;
  const float* nn = coef + 2 * npairs;
  const float sg = P.similarity ? 1.f : -1.f;
  const float invB = 1.f / (float)P.B;
  // role b: d out[b] / d den[b]
  {
    float den = (nc[idx] + P.q) * (nn[idx] + P.q);
    float G = sg * to_f32(gy[idx]) * invB;
    float acc = 0.f;
    for (int bp = 0; bp < P.B; ++bp) {
      float dv = dot[bp * per + r];
      acc += scs_dh(dv / den, P.p) * dv;
    }
    coef[4 * npairs + idx] = -G * acc / (den * den);
  }
  // role b': d sum_b out[b] / d dot[b']
  {
    float dv = dot[idx];
    float acc = 0.f;
    for (int b = 0; b < P.B; ++b) {
      long long o = b * per + r;
      float den = (nc[o] + P.q) * (nn[o] + P.q);
      acc += sg * to_f32(gy[o]) * invB * scs_dh(dv / den, P.p) / den;
    }
    coef[3 * npairs + idx] = acc;
  }
}
__global__ void __launch_bounds__(kThreads) scs_coef_kernel_b(float* __restrict__ coef, KParams P,
                                                              long long npairs) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= npairs) return;
  float nc = coef[npairs + idx], nn = coef[2 * npairs + idx];
  float gdot = coef[3 * npairs + idx], gden = coef[4 * npairs + idx];
  coef[idx] = gdot;
  coef[npairs + idx] = nc > 0.f ? gden * (nn + P.q) / nc : 0.f;
  coef[2 * npairs + idx] = nn > 0.f ? gden * (nc + P.q) / nn : 0.f;
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

// Gather form of the backward: one thread per (b, channel, INPUT pixel q) collects, in a fixed order, every
// contribution that lands on q -- as a neighbour tap of an output pixel (d/dn) and as the centre of an output pixel
// (sum over its taps of d/dc) -- through the inverse of the padding / stride / dilation index map.  No atomics:
// bit-reproducible for every measure and geometry; gx is written once, in its own dtype.
template <typename T, int M>
__global__ void __launch_bounds__(kThreads) gather_kernel(const T* __restrict__ x, const float* __restrict__ coef,
                                                          T* __restrict__ gx, const float* __restrict__ g_gap_x,
                                                          KParams P, long long npairs, long long total) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= total) return;
  const int w = (int)(idx % P.W);
  long long r = idx / P.W;
  const int h = (int)(r % P.H);
  r /= P.H;
  const int ch = (int)(r % P.C);
  const int b = (int)(r / P.C);
  const int HW = P.H * P.W;
  const size_t plane = ((size_t)b * P.C + ch) * HW;
  const long long HoWo = (long long)P.Ho * P.Wo;
  const float xq = to_f32(x[plane + h * P.W + w]);
  float acc = g_gap_x ? g_gap_x[(size_t)b * P.C + ch] / (float)HW : 0.f;
  const int ctr = P.R * P.dil;
  for_each_preimage(h, P.H, P.pad, P.mode, [&](int pr) {
    for_each_preimage(w, P.W, P.pad, P.mode, [&](int pc) {
      // (1) q as the neighbour tap t of output pixel (i, j): i*stride + a*dil - pad == pr
      for (int t = 0; t < P.K; ++t) {
        int a, bb;
        tap_rc(t, P.k, P.K, a, bb);
        const int ti = pr + P.pad - a * P.dil, tj = pc + P.pad - bb * P.dil;
        if (ti < 0 || tj < 0 || ti % P.stride || tj % P.stride) continue;
        const int i = ti / P.stride, j = tj / P.stride;
        if (i >= P.Ho || j >= P.Wo) continue;
        const int rc = map_index(i * P.stride + ctr - P.pad, P.H, P.mode);
        const int cc = map_index(j * P.stride + ctr - P.pad, P.W, P.mode);
        const float c = (rc >= 0 && cc >= 0) ? to_f32(x[plane + rc * P.W + cc]) : 0.f;
        const long long pb = (long long)b * P.K * HoWo + (long long)i * P.Wo + j + t * HoWo;
        float k[5];
#pragma unroll
        for (int u = 0; u < 5; ++u) k[u] = coef[u * npairs + pb];
        float dc, dn;
        chan_grad<M>(c, xq, k, P, dc, dn);
        acc += dn;
      }
      // (2) q as the centre of output pixel (i, j): i*stride + R*dil - pad == pr
      const int ti = pr + P.pad - ctr, tj = pc + P.pad - ctr;
      if (ti >= 0 && tj >= 0 && ti % P.stride == 0 && tj % P.stride == 0) {
        const int i = ti / P.stride, j = tj / P.stride;
        if (i < P.Ho && j < P.Wo) {
          const long long pb = (long long)b * P.K * HoWo + (long long)i * P.Wo + j;
          for (int t = 0; t < P.K; ++t) {
            int a, bb;
            tap_rc(t, P.k, P.K, a, bb);
            const int rn = map_index(i * P.stride + a * P.dil - P.pad, P.H, P.mode);
            const int cn = map_index(j * P.stride + bb * P.dil - P.pad, P.W, P.mode);
            const float n = (rn >= 0 && cn >= 0) ? to_f32(x[plane + rn * P.W + cn]) : 0.f;
            float k[5];
#pragma unroll
            for (int u = 0; u < 5; ++u) k[u] = coef[u * npairs + pb + t * HoWo];
            float dc, dn;
            chan_grad<M>(xq, n, k, P, dc, dn);
            acc += dc;
          }
        }
      }
    });
  });
  gx[idx] = from_f32<T>(acc);
}

// mean over the spatial plane: one warp per (b, channel)
template <typename T>
__global__ void __launch_bounds__(kThreads) gap_kernel(const T* __restrict__ src, float* __restrict__ dst, int HW,
                                                       long long planes) {
  long long w = ((long long)blockIdx.x * kThreads + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= planes) return;
  const T* p = src + w * HW;
  float acc = 0.f;
  for (int e = lane; e < HW; e += 32) acc += to_f32(p[e]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) dst[w] = acc / (float)HW;
}

// gy[b,t,:,:] = g_gap_nfp[b,t] / (Ho*Wo)
template <typename T>
__global__ void __launch_bounds__(kThreads) expand_gap_grad_kernel(const float* __restrict__ g, T* __restrict__ gy,
                                                                   int HoWo, long long total) {
  long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (idx < total) gy[idx] = from_f32<T>(g[idx / HoWo] / (float)HoWo);
}

inline unsigned blocks_for(long long n) { return (unsigned)((n + kThreads - 1) / kThreads); }

#define NFP_DISPATCH_MEASURE(M_RT, ...)                                             \
  switch (M_RT) {                                                                    \
    case NFPB200_NORM: { constexpr int M = NFPB200_NORM; __VA_ARGS__; } break;        \
    case NFPB200_COSINE: { constexpr int M = NFPB200_COSINE; __VA_ARGS__; } break;    \
    case NFPB200_DOT: { constexpr int M = NFPB200_DOT; __VA_ARGS__; } break;          \
    case NFPB200_RMSE: { constexpr int M = NFPB200_RMSE; __VA_ARGS__; } break;        \
    case NFPB200_GEMAN: { constexpr int M = NFPB200_GEMAN; __VA_ARGS__; } break;      \
    case NFPB200_ATTENTION: { constexpr int M = NFPB200_ATTENTION; __VA_ARGS__; } break; \
    case NFPB200_EMD: { constexpr int M = NFPB200_EMD; __VA_ARGS__; } break;          \
    case NFPB200_CANBERRA: { constexpr int M = NFPB200_CANBERRA; __VA_ARGS__; } break; \
    case NFPB200_HELLINGER: { constexpr int M = NFPB200_HELLINGER; __VA_ARGS__; } break; \
    case NFPB200_CHISQUARED1: { constexpr int M = NFPB200_CHISQUARED1; __VA_ARGS__; } break; \
    case NFPB200_CHISQUARED2: { constexpr int M = NFPB200_CHISQUARED2; __VA_ARGS__; } break; \
    case NFPB200_GFC: { constexpr int M = NFPB200_GFC; __VA_ARGS__; } break;          \
    case NFPB200_PEARSON: { constexpr int M = NFPB200_PEARSON; __VA_ARGS__; } break;  \
    case NFPB200_JEFFREY: { constexpr int M = NFPB200_JEFFREY; __VA_ARGS__; } break;  \
    case NFPB200_SQUAREDCHORD: { constexpr int M = NFPB200_SQUAREDCHORD; __VA_ARGS__; } break; \
    case NFPB200_SMITH: { constexpr int M = NFPB200_SMITH; __VA_ARGS__; } break;      \
    case NFPB200_SCS: { constexpr int M = NFPB200_SCS; __VA_ARGS__; } break;          \
    default: return NFPB200_EINVAL;                                                  \
  }

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

template <typename T>
int forward_t(const KParams& P, int measure, const T* x, T* y, const LaunchCtx& ctx) {
  const long long npairs = (long long)P.B * P.K * P.Ho * P.Wo;
  float* raw = (float*)ctx.ws;
  NFP_DISPATCH_MEASURE(measure,
    (pair_forward_kernel<T, M><<<blocks_for(npairs), kThreads, 0, ctx.stream>>>(x, y, raw, P, npairs)));
  if (measure == NFPB200_ATTENTION) {
    long long pix = (long long)P.B * P.Ho * P.Wo;
    attention_forward_kernel<T><<<blocks_for(pix), kThreads, 0, ctx.stream>>>(raw, y, P);
  } else if (measure == NFPB200_SCS) {
    scs_forward_kernel<T><<<blocks_for(npairs), kThreads, 0, ctx.stream>>>(raw, y, P, npairs);
  }
  return (int)cudaGetLastError();
}

// workspace layout of backward: [coef: 5*npairs f32]
template <typename T, typename GT>
int backward_t(const KParams& P, int measure, const T* x, const GT* gy, T* gx, const float* g_gap_x,
               char* ws, cudaStream_t stream) {
  const long long npairs = (long long)P.B * P.K * P.Ho * P.Wo;
  const long long nx = (long long)P.B * P.C * P.H * P.W;
  float* coef = (float*)ws;
  NFP_DISPATCH_MEASURE(measure,
    (pair_coef_kernel<T, GT, M><<<blocks_for(npairs), kThreads, 0, stream>>>(x, gy, coef, P, npairs)));
  if (measure == NFPB200_ATTENTION) {
    long long pix = (long long)P.B * P.Ho * P.Wo;
    attention_coef_kernel<GT><<<blocks_for(pix), kThreads, 0, stream>>>(gy, coef, P);
  } else if (measure == NFPB200_SCS) {
    scs_coef_kernel_a<GT><<<blocks_for(npairs), kThreads, 0, stream>>>(gy, coef, P, npairs);
    scs_coef_kernel_b<<<blocks_for(npairs), kThreads, 0, stream>>>(coef, P, npairs);
  }
  NFP_DISPATCH_MEASURE(measure,
    (gather_kernel<T, M><<<blocks_for(nx), kThreads, 0, stream>>>(x, coef, gx, g_gap_x, P, npairs, nx)));
  return (int)cudaGetLastError();
}

}  // namespace

size_t generic_workspace_bytes(const KParams& P, int dtype, int measure, int op) {
  const size_t npairs = (size_t)P.B * P.K * P.Ho * P.Wo;
  const size_t nx = (size_t)P.B * P.C * P.H * P.W;
  const size_t esz = dtype == NFPB200_BF16 ? 2 : 4;
  const size_t fwd = measure == NFPB200_ATTENTION ? 4 * npairs : (measure == NFPB200_SCS ? 8 * npairs : 0);
  const size_t bwd = align256(20 * npairs);
  (void)nx;
  switch (op) {
    case NFPB200_OP_FORWARD: return fwd;
    case NFPB200_OP_BACKWARD: return bwd;
    case NFPB200_OP_POOL_FORWARD: return align256(esz * npairs) + fwd;   // [y map][forward scratch]
    case NFPB200_OP_POOL_BACKWARD: return align256(4 * npairs) + bwd;    // [fp32 gy map][backward scratch]
  }
  return 0;
}

int generic_launch_count(const KParams& P, int dtype, int measure, int op) {
  (void)P;
  const int extra_f = (measure == NFPB200_ATTENTION || measure == NFPB200_SCS) ? 1 : 0;
  const int extra_b = measure == NFPB200_ATTENTION ? 1 : (measure == NFPB200_SCS ? 2 : 0);
  const int fwd = 1 + extra_f;
  const int bwd = 2 + extra_b;
  (void)dtype;
  switch (op) {
    case NFPB200_OP_FORWARD: return fwd;
    case NFPB200_OP_BACKWARD: return bwd;
    case NFPB200_OP_POOL_FORWARD: return fwd + 2;
    case NFPB200_OP_POOL_BACKWARD: return bwd + 1;
  }
  return 0;
}

int generic_forward(const KParams& P, int dtype, int measure, const void* x, void* y, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return forward_t<__nv_bfloat16>(P, measure, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, ctx);
  return forward_t<float>(P, measure, (const float*)x, (float*)y, ctx);
}

int generic_backward(const KParams& P, int dtype, int measure, const void* x, const void* gy, void* gx,
                     const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return backward_t<__nv_bfloat16, __nv_bfloat16>(P, measure, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gy,
                                                     (__nv_bfloat16*)gx, nullptr, (char*)ctx.ws, ctx.stream);
  return backward_t<float, float>(P, measure, (const float*)x, (const float*)gy, (float*)gx, nullptr, (char*)ctx.ws,
                                  ctx.stream);
}

namespace {
template <typename T>
int pool_forward_t(const KParams& P, int measure, const T* x, float* gap_x, float* gap_nfp, const LaunchCtx& ctx) {
  const size_t npairs = (size_t)P.B * P.K * P.Ho * P.Wo;
  T* ymap = (T*)ctx.ws;
  LaunchCtx inner{ctx.stream, (char*)ctx.ws + align256(sizeof(T) * npairs), 0};
  int rc = forward_t<T>(P, measure, x, ymap, inner);
  if (rc) return rc;
  const long long px = (long long)P.B * P.C, py = (long long)P.B * P.K;
  gap_kernel<T><<<blocks_for(px * 32), kThreads, 0, ctx.stream>>>(x, gap_x, P.H * P.W, px);
  gap_kernel<T><<<blocks_for(py * 32), kThreads, 0, ctx.stream>>>(ymap, gap_nfp, P.Ho * P.Wo, py);
  return (int)cudaGetLastError();
}
template <typename T>
int pool_backward_t(const KParams& P, int measure, const T* x, const float* g_gap_x, const float* g_gap_nfp,
                    T* gx, const LaunchCtx& ctx) {
  const size_t npairs = (size_t)P.B * P.K * P.Ho * P.Wo;
  // the map gradient g_gap_nfp / (Ho*Wo) stays fp32 also for bf16 x: rounded to bf16, its 2^-9 error is multiplied by
  // the per-tap derivatives, which cancel to far smaller sums at pixels near a clamp (norm ~ eps, |c| + |n| ~ eps)
  float* gymap = (float*)ctx.ws;
  expand_gap_grad_kernel<float><<<blocks_for((long long)npairs), kThreads, 0, ctx.stream>>>(
      g_gap_nfp, gymap, P.Ho * P.Wo, (long long)npairs);
  return backward_t<T, float>(P, measure, x, gymap, gx, g_gap_x, (char*)ctx.ws + align256(sizeof(float) * npairs),
                              ctx.stream);
}
}  // namespace

int generic_pool_forward(const KParams& P, int dtype, int measure, const void* x, float* gap_x, float* gap_nfp,
                         const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return pool_forward_t<__nv_bfloat16>(P, measure, (const __nv_bfloat16*)x, gap_x, gap_nfp, ctx);
  return pool_forward_t<float>(P, measure, (const float*)x, gap_x, gap_nfp, ctx);
}

int generic_pool_backward(const KParams& P, int dtype, int measure, const void* x, const float* g_gap_x,
                          const float* g_gap_nfp, void* gx, const LaunchCtx& ctx) {
  if (dtype == NFPB200_BF16)
    return pool_backward_t<__nv_bfloat16>(P, measure, (const __nv_bfloat16*)x, g_gap_x, g_gap_nfp,
                                          (__nv_bfloat16*)gx, ctx);
  return pool_backward_t<float>(P, measure, (const float*)x, g_gap_x, g_gap_nfp, (float*)gx, ctx);
}

}  // namespace nfp
