// Channels-last ("token") fused NFP kernels for sm_100a, bf16 or fp16: cosine measure, stride 1, dilation 1, padding = R.
//
// Input layout: x[b][p][c] with the C channels of a pixel contiguous and an arbitrary batch stride -- what a
// channels_last (NHWC) feature map is in memory, and what the reference's ViT head builds as a VIEW of the backbone's
// token tensor (models/texture_pooling.py:181-188: feats[:, 1:].transpose(1, 2).reshape(B, C, H, W) has strides
// (197*C, 1, W*C, C); models/vittiny.py:129-135).  The NCHW kernels would need a repack copy each way; here the
// channel contraction runs on tensor cores straight from that layout:
//
//   load     the image's P x C bf16 / fp16 matrix X -> shared memory with 16-byte cp.async copies, 16-byte chunks XOR-swizzled
//            by (row & 7) so that every ldmatrix below is bank-conflict-free; two image buffers when they fit (the next
//            image streams in while the current one is processed).
//   Gram     G = X X^T restricted to the band the k x k window needs: mma.sync.m16n8k16 (bf16 x bf16 -> fp32: the
//            products are exact, accumulation is fp32 as in the NCHW kernels).  A = 16 pixel rows, B = the pixel rows
//            of the n-tiles at and after the diagonal (X is both operands; dot(p,q) = dot(q,p)), K = channels, split
//            over warps (fp16: mma.sync.m16n8k16 f16 x f16 -> fp32, equally exact).  The accumulator entries whose (row, column) pair is a forward window direction go to the
//            per-pixel table the NCHW kernels build with FMAs (|x_p|^2 and (k*k-1)/2 dots per pixel).
//   forward  y = dot / (max(|p|,eps) max(|q|,eps)) via the compile-time stencil tables -> (B, K, H, W) (NCHW, as the
//            reference returns it; the dtype of x or, under autocast, fp32); pooled mode reduces instead.
//   backward the closed-form stencil coefficients Wd[p][o] (same code as the NCHW kernels: gather form, no atomics)
//            are scattered into the banded P x P matrix M (bf16 hi + lo parts: 16 mantissa bits), and
//            gx = M X runs on the tensor cores again: A = M (16 rows x the 3..5 k-tiles of the band), B = X through
//            ldmatrix.trans, fp32 accumulators -> bf16 / fp16 -> per-warp staging -> 128-byte row segments of gx
//            (channels-last).  fp16 x: M stays bf16 hi + lo -- its entries reach ~1/eps^2 at degenerate pixels and span
//            ~1e6 within a row, beyond fp16's range, so an fp16 M would flush the ordinary entries to subnormals.  Each
//            X fragment is split in registers into bf16 hi + lo instead (exact: an fp16 value has 11 significant bits;
//            the f16 and bf16 m16n8k16 fragment layouts are the same), and gx = M_hi X_hi + M_hi X_lo + M_lo X_hi.
//
// Bit-reproducible: every sum has a fixed order.  fp32 channels-last inputs are not covered (TF32 would break the 1e-5
// parity bound): the host side repacks those to NCHW.
#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "nfp_common.cuh"
#include "nfp_ptx.cuh"
#include "nfp_stream.h"
#include "nfp_tables.cuh"

namespace nfp {
namespace token {

using namespace ptx;
using stream::align_up;
using stream::Cfg;
using stream::Tables;
using stream::tables_for;
using stream::MODE_BWD;
using stream::MODE_FWD;
using stream::MODE_POOL_BWD;
using stream::MODE_POOL_FWD;

typedef __nv_bfloat16 bf16;
typedef __half f16;

struct TokenArgs {
  const void* x;
  const void* gy;
  void* y;
  void* gx;
  const float* g_gap_x;
  const float* g_gap_nfp;
  float* gap_x;
  float* gap_nfp;
  // fused nfp_pooling head (NFP_Pooling.py:31-35), as in the NCHW ring kernels
  const float* proj_w;     // (C, K) fp32, null = plain pooled mode
  const float* proj_b;     // (C) fp32 or null
  float* head_out;         // forward: (B, C) fp32
  const float* head_gout;  // backward: d loss / d out (B, C) fp32; gap_x / gap_nfp then hold the forward's results
  int B, C;
  long long xbs, gxbs;  // batch strides of x / gx in elements
  int nbuf;             // image buffers in shared memory (1 or 2)
  int KS, KSlog;        // channel split of the Gram phase (a power of two) and its log2
  int pad_mode, similarity, y_f32;
  int kin, rin;         // multi-radius launch (desc.inner_R): kin planes of the radius-rin map in front of y / gy
  float eps;
  unsigned long long* dbg;  // optional: 8 globaltimer stamps per (CTA, image < 2), see nfpb200_debug_phase_timing
};

#define NFP_TSTAMP(k) do { if (a.dbg && tid == 0 && it < 2) a.dbg[((size_t)blockIdx.x * 2 + it) * 8 + (k)] = globaltimer_ns(); } while (0)

// warps per CTA: 16 with one CTA per SM (two image buffers), or 8 with two CTAs per SM (one buffer each) when both fit:
// the scalar table / coefficient phases of one image then overlap the tensor-core phases of the other
constexpr int kNWBig = 16, kNWSmall = 8;
constexpr int kSmemPerSM = 227 * 1024;
constexpr int kMaxKS = 8;
constexpr int kStgStride = 144;  // bytes per staged gx row: 64 channels + 16 (conflict-free fragment stores)

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// X X^T step in the element type of x (both operands are X)
template <typename T>
__device__ __forceinline__ void mma_x(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (std::is_same<T, f16>::value) mma_f16(d, a, b0, b1);
  else mma_bf16(d, a, b0, b1);
}
// two packed elements of x -> fp32
template <typename T>
__device__ __forceinline__ void unpack_x2(uint32_t v, float& lo, float& hi) {
  if constexpr (std::is_same<T, f16>::value) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v));
    lo = f.x; hi = f.y;
  } else {
    lo = __uint_as_float(v << 16);
    hi = __uint_as_float(v & 0xffff0000u);
  }
}
// two fp32 values -> packed elements of x (round to nearest: fp16 overflows to +-inf, nothing is clamped)
template <typename T>
__device__ __forceinline__ uint32_t pack_x2(float lo, float hi) {
  uint32_t r;
  if constexpr (std::is_same<T, f16>::value) {
    const __half2 h = __floats2half2_rn(lo, hi);
    r = *reinterpret_cast<const uint32_t*>(&h);
  } else {
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    r = *reinterpret_cast<const uint32_t*>(&h);
  }
  return r;
}
// a B fragment register of fp16 X (two halves) -> the same two values as bf16 hi + lo registers, exactly
__device__ __forceinline__ void split_f16x2(uint32_t v, uint32_t& hi, uint32_t& lo) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v));
  const __nv_bfloat162 h = __floats2bfloat162_rn(f.x, f.y);
  const float2 hf = __bfloat1622float2(h);
  const __nv_bfloat162 l = __floats2bfloat162_rn(f.x - hf.x, f.y - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

template <class C>
struct Geo {
  static constexpr int P = C::P, PPAD = align_up(C::P, 16), MT = PPAD / 16;
  static constexpr int HALO = C::R * C::W + C::R;             // pixels a window reaches before / after its centre
  static constexpr int NTN = (16 + HALO + 7) / 8;             // n-tiles (8 pixels) at and after the diagonal, Gram phase
  static constexpr int HT = (HALO + 15) / 16;                 // k-tiles (16 pixels) the band reaches on either side
  static constexpr int KTN = 1 + 2 * HT;                      // k-tiles per m-tile in gx = M X
  static constexpr int MS = KTN * 32 + 16;                    // bytes per row of an M block (padded: conflict-free ldmatrix)
};

// Shared-memory layout (byte offsets)
template <class C, int MODE, int NW>
struct Lay {
  static constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  int tfull, tpart, inv, rn, wd, gp, tabs, gyraw, ggx, mhi, mlo, stg, ytab, eidx, xs, total;
  int t_fv, t_fd, t_q, t_fsrc, t_fdst, t_fptr;
  int gy_stride, x_stride, row_bytes;
  __host__ __device__ Lay(int Cch, int nbuf, int ks, int kin = 0) {
    using G = Geo<C>;
    int o = 0;
    auto take = [&](int n) { int r = o; o += (n + 127) & ~127; return r; };
    tfull = take(C::PNV * 4);
    inv = take(C::P * 4);
    rn = take(BWD ? C::P * 4 : 0);
    wd = take(BWD ? C::H * C::RS * 4 : 0);
    // union: [Gram partial tables | gy-only stencil scratch] are dead once the coefficients exist; the per-warp gx
    // staging of the last phase lives on top of them
    const int u0 = o;
    tpart = take(ks * C::PNV * 4);
    gp = take(BWD ? C::P * C::KK * 4 : 0);
    const int u1 = o;
    o = u0;
    stg = take(BWD ? NW * 16 * kStgStride : 0);
    if (o < u1) o = u1;
    tabs = take(BWD ? Tables<C>::BWD_BYTES : Tables<C>::FWD_BYTES);
    if (BWD) {
      t_q = tabs;
      t_fsrc = t_q + Tables<C>::NQ * 2;
      t_fdst = t_fsrc + Tables<C>::NFS * 2;
      t_fptr = t_fdst + Tables<C>::NFS * 2;
      t_fv = t_fd = 0;
    } else {
      t_fv = tabs;
      t_fd = tabs + Tables<C>::NF * 2;
      t_q = t_fsrc = t_fdst = t_fptr = 0;
    }
    gy_stride = align_up((C::K + kin) * C::P * 2, 128);
    gyraw = take(MODE == MODE_BWD ? nbuf * gy_stride : (MODE == MODE_POOL_BWD ? C::K * 4 : 0));
    ggx = take(MODE == MODE_POOL_BWD ? Cch * 4 : 0);
    mhi = take(BWD ? G::MT * 16 * G::MS : 0);
    mlo = take(BWD ? G::MT * 16 * G::MS : 0);
    ytab = take(MODE == MODE_POOL_FWD ? C::K * C::P * 4 : 0);
    eidx = take(G::MT * 32 * G::NTN * 4 * 2);  // table entry of every Gram accumulator element (m-tile, lane, n-tile, e)
    row_bytes = Cch * 2;
    x_stride = G::PPAD * row_bytes;
    xs = take(nbuf * x_stride);
    total = o;
  }
};

template <typename T, class C, int MODE, int NW>
__global__ void __launch_bounds__(NW * 32, NW == kNWSmall ? 2 : 1) token_kernel(const TokenArgs a, const Tables<C>* __restrict__ gt) {
  using G = Geo<C>;
  constexpr int W = C::W, R = C::R, k = C::k, KK = C::KK, K = C::K, P = C::P, NV = C::NV, PNV = C::PNV;
  constexpr int PPAD = G::PPAD, MT = G::MT, NTN = G::NTN, HT = G::HT, KTN = G::KTN, MS = G::MS;
  constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  constexpr bool POOLED = (MODE == MODE_POOL_FWD || MODE == MODE_POOL_BWD);
  constexpr int NT = NW * 32;
  const int GY_BYTES = (K + a.kin) * P * 2;  // (multi-radius launch: kin inner-radius planes in front)

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int Cch = a.C, NBUF = a.nbuf, KS = a.KS;
  const Lay<C, MODE, NW> L(Cch, NBUF, KS, a.kin);
  float* tfull = reinterpret_cast<float*>(smem_raw + L.tfull);
  float* tpart = reinterpret_cast<float*>(smem_raw + L.tpart);
  float* inv = reinterpret_cast<float*>(smem_raw + L.inv);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int g8 = lane >> 2, t4 = lane & 3;
  const int row_bytes = L.row_bytes, chunks = Cch >> 3;  // 16-byte chunks per pixel row
  const uint32_t xs0 = smem_u32(smem_raw + L.xs);
  auto xaddr = [&](uint32_t xb, int row, int chunk) -> uint32_t {
    return xb + (uint32_t)(row * row_bytes) + (uint32_t)(((chunk ^ (row & 7)) << 4));
  };

  // ---- prologue (constants only: overlaps the tail of the preceding grid) --------------------------------------
  {
    constexpr int TAB_BYTES = BWD ? Tables<C>::BWD_BYTES : Tables<C>::FWD_BYTES;
    const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(gt) + (BWD ? Tables<C>::BWD_OFFSET : 0));
    uint4* dst = reinterpret_cast<uint4*>(smem_raw + L.tabs);
    for (int i = tid; i < TAB_BYTES / 16; i += NT) dst[i] = src[i];
    for (int i = tid; i < KS * PNV; i += NT) tpart[i] = 0.f;
    // rows P .. PPAD-1 of every image buffer stay zero (they are MMA operands, never loaded)
    for (int bf = 0; bf < NBUF; ++bf) {
      uint4* z = reinterpret_cast<uint4*>(smem_raw + L.xs + bf * L.x_stride + P * row_bytes);
      for (int i = tid; i < (PPAD - P) * row_bytes / 16; i += NT) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    // which per-pixel table entry (p * NV + dy * k + dx) a Gram accumulator element is, -1 = none: depends on the
    // geometry only, so it is worked out once here instead of per image in the accumulator epilogue
    {
      int16_t* ei = reinterpret_cast<int16_t*>(smem_raw + L.eidx);
      for (int i = tid; i < MT * 32 * NTN * 4; i += NT) {
        const int e = i & 3, j = (i >> 2) % NTN, ln = (i / (4 * NTN)) & 31, mt = i / (4 * NTN * 32);
        const int p = mt * 16 + (ln >> 2) + ((e >> 1) << 3), q = mt * 16 + 8 * j + 2 * (ln & 3) + (e & 1);
        int v = -1;
        if (p < P && q < P && q >= p) {
          const int pr = p / W, pc = p - pr * W, qr = q / W, qc = q - qr * W;
          const int dy = qr - pr, dx = qc - pc;
          if (dy <= R && dx >= -R && dx <= R && (dy > 0 || dx >= 0)) v = p * NV + dy * k + dx;
        }
        ei[i] = (int16_t)v;
      }
    }
    if constexpr (BWD) {  // M: the entries outside the band positions written below stay zero
      uint4* z = reinterpret_cast<uint4*>(smem_raw + L.mhi);
      for (int i = tid; i < 2 * G::MT * 16 * G::MS / 16; i += NT) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  grid_dependency_wait();
  if (tid == 0) grid_launch_dependents();

  const int nmine = (a.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int ld_row0 = tid / chunks, ld_ch0 = tid - ld_row0 * chunks, ld_drow = NT / chunks, ld_dch = NT - ld_drow * chunks;
  auto issue = [&](int it) {  // image `it` of this CTA -> buffer it % NBUF (all threads); two groups: gy, then x
    const int b = blockIdx.x + it * gridDim.x, bf = it % NBUF;
    if constexpr (MODE == MODE_BWD) {
      const unsigned char* gsrc = reinterpret_cast<const unsigned char*>(a.gy) + (size_t)b * GY_BYTES;
      const uint32_t gd = smem_u32(smem_raw + L.gyraw + bf * L.gy_stride);
      for (int i = tid; i < GY_BYTES / 16; i += NT) cp_async16(gd + i * 16, gsrc + i * 16);
    }
    cp_async_commit();
    const T* src = reinterpret_cast<const T*>(a.x) + (size_t)b * a.xbs;
    const uint32_t xb = xs0 + bf * L.x_stride;
    int row = ld_row0, ch = ld_ch0;
    while (row < P) {   // (row, chunk) walk in steps of NT chunks, no divisions
      cp_async16(xaddr(xb, row, ch), src + (size_t)row * Cch + ch * 8);
      row += ld_drow;
      ch += ld_dch;
      if (ch >= chunks) { ch -= chunks; ++row; }
    }
    cp_async_commit();
  };
  const float sgn = a.similarity ? 1.f : -1.f;

  for (int it = 0; it < nmine; ++it) {
    const int b = blockIdx.x + it * gridDim.x, bf = it % NBUF;
    const uint32_t xb = xs0 + bf * L.x_stride;
    const unsigned char* xbp = smem_raw + L.xs + bf * L.x_stride;
    NFP_TSTAMP(0);
    if (NBUF == 1 || it == 0) issue(it);
    const bool ahead = (NBUF == 2 && it + 1 < nmine);
    if (ahead) issue(it + 1);
    // groups in flight, oldest first: gy(it), x(it) [, gy(it+1), x(it+1)] -- the upstream gradient first: the gy-only
    // stencil part below runs while x is still streaming in
    if (ahead) cp_async_wait<3>(); else cp_async_wait<1>();
    __syncthreads();
    NFP_TSTAMP(1);  // gradient landed

    // ---- backward: the gy-only part of the stencil (as in the NCHW kernels) ---------------------------------------
    if constexpr (BWD) {
      const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
      const int16_t* fsrc = reinterpret_cast<const int16_t*>(smem_raw + L.t_fsrc);
      const int16_t* fdst = reinterpret_cast<const int16_t*>(smem_raw + L.t_fdst);
      const int16_t* fptr = reinterpret_cast<const int16_t*>(smem_raw + L.t_fptr);
      float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
      float* Gp = reinterpret_cast<float*>(smem_raw + L.gp);
      const unsigned char* gin = smem_raw + L.gyraw + (POOLED ? 0 : bf * L.gy_stride);
      const unsigned char* g = gin + a.kin * P * 2;
      if constexpr (POOLED) {
        float* gs = reinterpret_cast<float*>(smem_raw + L.ggx);
        if (a.proj_w) {
          // fused head backward: d/d GAP(x)[c] = g_out[c] (proj_w[c] . gnfp + proj_b[c]),
          // d/d GAP(NFP(x))[n] = sum_c g_out[c] GAP(x)[c] proj_w[c][n] (fixed-order block reduction)
          float gn[K], part[K];
#pragma unroll
          for (int n = 0; n < K; ++n) {
            gn[n] = a.gap_nfp[(size_t)b * K + n];
            part[n] = 0.f;
          }
          for (int c = tid; c < Cch; c += NT) {
            const float go = a.head_gout[(size_t)b * Cch + c], gxv = a.gap_x[(size_t)b * Cch + c];
            const float4* wr4 = reinterpret_cast<const float4*>(a.proj_w + (size_t)c * K);
            float proj = a.proj_b ? a.proj_b[c] : 0.f;
            const float t = go * gxv;
#pragma unroll
            for (int n4 = 0; n4 < K / 4; ++n4) {
              const float4 w4 = wr4[n4];
              proj = fmaf(w4.x, gn[4 * n4], proj); proj = fmaf(w4.y, gn[4 * n4 + 1], proj);
              proj = fmaf(w4.z, gn[4 * n4 + 2], proj); proj = fmaf(w4.w, gn[4 * n4 + 3], proj);
              part[4 * n4] = fmaf(t, w4.x, part[4 * n4]); part[4 * n4 + 1] = fmaf(t, w4.y, part[4 * n4 + 1]);
              part[4 * n4 + 2] = fmaf(t, w4.z, part[4 * n4 + 2]); part[4 * n4 + 3] = fmaf(t, w4.w, part[4 * n4 + 3]);
            }
            gs[c] = go * proj * (1.f / (float)P);
          }
#pragma unroll
          for (int n = 0; n < K; ++n) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part[n] += __shfl_xor_sync(0xffffffffu, part[n], o);
            if (lane == 0) Gp[warp * K + n] = part[n];   // Gp is free until the stencil loops below
          }
          __syncthreads();
          if (tid < K) {
            float sred = 0.f;
            for (int w = 0; w < NW; ++w) sred += Gp[w * K + tid];
            reinterpret_cast<float*>(smem_raw + L.gyraw)[tid] = sred * (1.f / (float)P);
          }
        } else {
          if (tid < K) reinterpret_cast<float*>(smem_raw + L.gyraw)[tid] = a.g_gap_nfp[(size_t)b * K + tid] * (1.f / (float)P);
          for (int i = tid; i < Cch; i += NT) gs[i] = a.g_gap_x[(size_t)b * Cch + i] * (1.f / (float)P);
        }
        __syncthreads();
      }
      auto Gv = [&](int flat) -> float {
        if constexpr (POOLED) return reinterpret_cast<const float*>(smem_raw + L.gyraw)[flat / P];
        else {
          float v = ldx<T>(g + flat * 2);
          if constexpr (R >= 2) {
            if (a.kin) {  // multi-radius launch: the same tap of the inner radius' map adds its gradient
              const int n = flat / P, n1 = inner_tap(n, R, a.rin);
              if (n1 >= 0) v += ldx<T>(gin + (n1 * P + flat - n * P) * 2);
            }
          }
          return v;
        }
      };
      for (int idx = tid; idx < P * KK; idx += NT) {
        const int p = idx / KK, o = idx - p * KK;
        float v = 0.f;
        if (o != C::CTR && qt[idx] >= 0) v = Gv((o < C::CTR ? o : o - 1) * P + p);
        Gp[idx] = v;
      }
      __syncthreads();
      const int nfd = fptr[Tables<C>::NFP - 1];
      for (int i = tid; i < nfd; i += NT) {
        const int dst = fdst[i];
        float v = Gp[dst];
        for (int j = fptr[i]; j < fptr[i + 1]; ++j) v += Gv(fsrc[j]);
        Gp[dst] = v;
      }
      __syncthreads();
      for (int idx = tid; idx < P * KK; idx += NT) {
        const int p = idx / KK, o = idx - p * KK;
        const int q = (o == C::CTR) ? -1 : (int)qt[idx];
        float v = Gp[idx];
        if (q >= 0) v += Gp[q * KK + (KK - 1 - o)];
        Wd[C::widx(p, o)] = sgn * v;
      }
    }

    if (ahead) cp_async_wait<2>(); else cp_async_wait<0>();
    __syncthreads();
    NFP_TSTAMP(2);  // gy-only stencil part done, image landed
    // ---- Gram band on the tensor cores: items (m-tile, channel split) over the warps ------------------------------
    {
      const int kper = Cch >> a.KSlog;
      for (int item = warp; item < MT * KS; item += NW) {
        const int mt = item >> a.KSlog, ks = item & (KS - 1);
        const int m0 = mt * 16, kbeg = ks * kper, kend = kbeg + kper;
        float acc[NTN][4];
#pragma unroll
        for (int j = 0; j < NTN; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
        // B rows of this lane for the n-tile pairs (clamped: tiles past the padded map are computed on junk and ignored)
        int brow[(NTN + 1) / 2];
#pragma unroll
        for (int jp = 0; jp < (NTN + 1) / 2; ++jp) {
          const int rr = m0 + 16 * jp + (lane & 7) + ((lane >> 4) << 3);
          brow[jp] = rr < PPAD ? rr : PPAD - 1;
        }
        // per-lane operand addresses: row base + swizzled 16-byte chunk; fragments of step s+1 are fetched before the
        // MMAs of step s are issued (two register sets), so ldmatrix latency overlaps the tensor-core work
        constexpr int NBP = (NTN + 1) / 2;
        const int arow = m0 + (lane & 15);
        const uint32_t abase = xb + (uint32_t)(arow * row_bytes), ax = (uint32_t)(arow & 7), ac = (uint32_t)(lane >> 4);
        uint32_t bbase[NBP], bxr[NBP];
#pragma unroll
        for (int jp = 0; jp < NBP; ++jp) {
          bbase[jp] = xb + (uint32_t)(brow[jp] * row_bytes);
          bxr[jp] = (uint32_t)(brow[jp] & 7);
        }
        const uint32_t bc = (uint32_t)((lane >> 3) & 1);
        auto fetch = [&](int k0, uint32_t (&af)[4], uint32_t (&bq)[NBP][4]) {
          const uint32_t c0 = (uint32_t)(k0 >> 3);
          ldmatrix_x4(af, abase + (((c0 + ac) ^ ax) << 4));
#pragma unroll
          for (int jp = 0; jp < NBP; ++jp) ldmatrix_x4(bq[jp], bbase[jp] + (((c0 + bc) ^ bxr[jp]) << 4));
        };
        auto compute = [&](const uint32_t (&af)[4], const uint32_t (&bq)[NBP][4]) {
#pragma unroll
          for (int jp = 0; jp < NBP; ++jp) {
            mma_x<T>(acc[2 * jp], af, bq[jp][0], bq[jp][1]);
            if (2 * jp + 1 < NTN) mma_x<T>(acc[2 * jp + 1], af, bq[jp][2], bq[jp][3]);
          }
        };
        uint32_t af0[4], bq0[NBP][4], af1[4], bq1[NBP][4];
        fetch(kbeg, af0, bq0);
        for (int k0 = kbeg; k0 < kend; k0 += 32) {   // two steps per trip (kper is a multiple of 32 or ends on step 0)
          const bool two = k0 + 16 < kend;
          if (two) fetch(k0 + 16, af1, bq1);
          compute(af0, bq0);
          if (two) {
            if (k0 + 32 < kend) fetch(k0 + 32, af0, bq0);
            compute(af1, bq1);
          }
        }
        // accumulator entries that are forward window directions -> this split's partial table
        float* tp = tpart + ks * PNV;
        const int16_t* ei = reinterpret_cast<const int16_t*>(smem_raw + L.eidx) + (mt * 32 + lane) * (NTN * 4);
#pragma unroll
        for (int j = 0; j < NTN; ++j) {
          const uint2 w = *reinterpret_cast<const uint2*>(ei + 4 * j);
          const int i0 = (int)(int16_t)(w.x & 0xffffu), i1 = (int)(int16_t)(w.x >> 16);
          const int i2 = (int)(int16_t)(w.y & 0xffffu), i3 = (int)(int16_t)(w.y >> 16);
          if (i0 >= 0) tp[i0] = acc[j][0];
          if (i1 >= 0) tp[i1] = acc[j][1];
          if (i2 >= 0) tp[i2] = acc[j][2];
          if (i3 >= 0) tp[i3] = acc[j][3];
        }
      }
    }
    __syncthreads();
    NFP_TSTAMP(3);  // Gram done
    for (int i = tid; i < PNV; i += NT) {
      float s = tpart[i];
      for (int ks = 1; ks < KS; ++ks) s += tpart[ks * PNV + i];  // fixed order: deterministic
      tfull[i] = s;
      if (i % NV == 0) {
        const int p = i / NV;
        const float nrm = sqrtf(s), N = fmaxf(nrm, a.eps);
        inv[p] = 1.f / N;
        if constexpr (BWD) reinterpret_cast<float*>(smem_raw + L.rn)[p] = nrm > 0.f ? 1.f / (N * nrm) : 0.f;
      }
    }
    if constexpr (MODE == MODE_POOL_FWD) {
      // GAP(x) (NFP_Pooling.py:27): a thread sums two adjacent channels down the P pixel rows
      for (int w2 = tid; w2 < Cch / 2; w2 += NT) {
        float s0 = 0.f, s1 = 0.f;
        for (int p = 0; p < P; ++p) {
          const uint32_t v = *reinterpret_cast<const uint32_t*>(xbp + p * row_bytes + ((((w2 >> 2) ^ (p & 7)) << 4) | ((w2 & 3) << 2)));
          float v0, v1;
          unpack_x2<T>(v, v0, v1);
          s0 += v0;
          s1 += v1;
        }
        a.gap_x[(size_t)b * Cch + 2 * w2] = s0 / (float)P;
        a.gap_x[(size_t)b * Cch + 2 * w2 + 1] = s1 / (float)P;
      }
    }
    __syncthreads();

    if constexpr (!BWD) {
      const int16_t* fv = reinterpret_cast<const int16_t*>(smem_raw + L.t_fv);
      const int16_t* fd = reinterpret_cast<const int16_t*>(smem_raw + L.t_fd);
      float* ytab = reinterpret_cast<float*>(smem_raw + L.ytab);
      for (int idx = tid; idx < K * P; idx += NT) {
        const int p = idx % P;
        const int v = fv[idx];
        float yv = 0.f;
        if (v >= 0) yv = tfull[fd[idx]] * (inv[p] * inv[v]);
        if (!a.similarity) yv = 1.f - yv;
        if constexpr (POOLED) {
          ytab[idx] = yv;
        } else {
          const size_t yb = (size_t)b * (K + a.kin) * P;
          if (a.y_f32) reinterpret_cast<float*>(a.y)[yb + a.kin * P + idx] = yv;
          else reinterpret_cast<T*>(a.y)[yb + a.kin * P + idx] = from_f32<T>(yv);
          if constexpr (R >= 2) {
            if (a.kin) {  // multi-radius launch: the inner radius' taps are the inner taps of this window
              const int n1 = inner_tap(idx / P, R, a.rin);
              if (n1 >= 0) {
                if (a.y_f32) reinterpret_cast<float*>(a.y)[yb + n1 * P + p] = yv;
                else reinterpret_cast<T*>(a.y)[yb + n1 * P + p] = from_f32<T>(yv);
              }
            }
          }
        }
      }
      if constexpr (POOLED) {
        __syncthreads();
        for (int n = warp; n < K; n += NW) {
          float s = 0.f;
          for (int p = lane; p < P; p += 32) s += ytab[n * P + p];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lane == 0) {
            a.gap_nfp[(size_t)b * K + n] = s / (float)P;
            tfull[n] = s / (float)P;   // (the table is dead: every y value has been computed)
          }
        }
        if (a.proj_w) {
          // fused head: out[c] = GAP(x)[c] * (proj_w[c] . GAP(NFP(x)) + proj_b[c])
          __syncthreads();   // tfull[0..K) and this CTA's gap_x stores are visible to the whole CTA
          for (int c = tid; c < Cch; c += NT) {
            const float4* wr4 = reinterpret_cast<const float4*>(a.proj_w + (size_t)c * K);
            float proj = a.proj_b ? a.proj_b[c] : 0.f;
#pragma unroll
            for (int n4 = 0; n4 < K / 4; ++n4) {
              const float4 w4 = wr4[n4];
              proj = fmaf(w4.x, tfull[4 * n4], proj); proj = fmaf(w4.y, tfull[4 * n4 + 1], proj);
              proj = fmaf(w4.z, tfull[4 * n4 + 2], proj); proj = fmaf(w4.w, tfull[4 * n4 + 3], proj);
            }
            a.head_out[(size_t)b * Cch + c] = a.gap_x[(size_t)b * Cch + c] * proj;
          }
        }
      }
    } else {
      // ---- stencil coefficients (closed form of ATen's cosine_similarity backward, as in the NCHW kernels) -------
      const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
      const float* rn = reinterpret_cast<const float*>(smem_raw + L.rn);
      float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
      for (int i8 = tid; i8 < align_up(P * 8, 32); i8 += NT) {
        const int p = i8 >> 3, g = i8 & 7;
        const bool valid = p < P;
        const float ip = valid ? inv[p] : 0.f;
        float s = 0.f;
        if (valid) {
#pragma unroll
          for (int t = 0; t < (K + 7) / 8; ++t) {
            const int n = g + 8 * t;
            if (n < K) {
              const int o = n < C::CTR ? n : n + 1;
              const int q = qt[p * KK + o];
              if (q >= 0) {
                const float w = Wd[C::widx(p, o)] * (ip * inv[q]);
                const float d = o > C::CTR ? tfull[p * NV + (o - C::CTR)] : tfull[q * NV + (C::CTR - o)];
                Wd[C::widx(p, o)] = w;
                s = fmaf(w, d, s);
              }
            }
          }
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if (valid && g == 0) {
          const float sw = 2.f * Wd[C::widx(p, C::CTR)] * (ip * ip);
          Wd[C::widx(p, C::CTR)] = sw - rn[p] * (s + sw * tfull[p * NV]);
        }
      }
      __syncthreads();
      NFP_TSTAMP(4);  // coefficients done
      // ---- M[p][q] = Wd[p][o] for q = p + off(o) inside the map: bf16 hi + lo, banded blocks per m-tile ------------
      unsigned char* mhi = smem_raw + L.mhi;
      unsigned char* mlo = smem_raw + L.mlo;
      for (int idx = tid; idx < P * KK; idx += NT) {
        const int p = idx / KK, o = idx - p * KK;
        const int q = (o == C::CTR) ? p : (int)qt[idx];
        if (q < 0) continue;
        const float w = Wd[C::widx(p, o)];
        const bf16 hi = __float2bfloat16_rn(w);
        const bf16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
        const int mt = p >> 4, col = q - 16 * (mt - HT);
        const int off = (mt * 16 + (p & 15)) * MS + col * 2;
        *reinterpret_cast<bf16*>(mhi + off) = hi;
        *reinterpret_cast<bf16*>(mlo + off) = lo;
      }
      __syncthreads();
      NFP_TSTAMP(5);  // M built
      // ---- gx = M X on the tensor cores: items (m-tile, 64-channel chunk) over the warps ------------------------
      const uint32_t mhi_a = smem_u32(mhi), mlo_a = smem_u32(mlo);
      unsigned char* stg = smem_raw + L.stg + warp * 16 * kStgStride;
      const float* ggx = reinterpret_cast<const float*>(smem_raw + L.ggx);
      T* gxb = reinterpret_cast<T*>(a.gx) + (size_t)b * a.gxbs;
      const int nchunk = Cch >> 6;
      for (int item = warp; item < MT * nchunk; item += NW) {
        const int mt = item / nchunk, cc = item - mt * nchunk;
        const int m0 = mt * 16, ch0 = cc * 64;
        float acc[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float i0 = 0.f, i1 = 0.f;
          if constexpr (MODE == MODE_POOL_BWD) {
            i0 = ggx[ch0 + 8 * j + 2 * t4];
            i1 = ggx[ch0 + 8 * j + 2 * t4 + 1];
          }
          acc[j][0] = i0; acc[j][1] = i1; acc[j][2] = i0; acc[j][3] = i1;
        }
        const uint32_t bch = (uint32_t)((ch0 >> 3) + (lane >> 4));
#pragma unroll
        for (int kk = 0; kk < KTN; ++kk) {
          const int kt = mt - HT + kk;
          if (kt < 0 || kt >= MT) continue;
          uint32_t ahi[4], alo[4], bx[4][4];
          const uint32_t moff = (uint32_t)((m0 + (lane & 15)) * MS + kk * 32 + ((lane >> 4) << 4));
          const int brow = 16 * kt + (lane & 7) + (((lane >> 3) & 1) << 3);
          const uint32_t bb = xb + (uint32_t)(brow * row_bytes), bxr = (uint32_t)(brow & 7);
          // all six operand fetches of the k-tile go out before its sixteen MMAs
          ldmatrix_x4(ahi, mhi_a + moff);
          ldmatrix_x4(alo, mlo_a + moff);
#pragma unroll
          for (int np = 0; np < 4; ++np) ldmatrix_x4_trans(bx[np], bb + (((bch + 2 * np) ^ bxr) << 4));
          if constexpr (std::is_same<T, f16>::value) {
            // fp16 X: bf16 hi + lo fragments in registers, M_hi X_hi + M_hi X_lo + M_lo X_hi (M_lo X_lo, ~2^-18 of a
            // term, is below the 16-bit precision M is held at)
#pragma unroll
            for (int np = 0; np < 4; ++np) {
              uint32_t xh[4], xl[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) split_f16x2(bx[np][i], xh[i], xl[i]);
              mma_bf16(acc[2 * np], ahi, xh[0], xh[1]);
              mma_bf16(acc[2 * np + 1], ahi, xh[2], xh[3]);
              mma_bf16(acc[2 * np], ahi, xl[0], xl[1]);
              mma_bf16(acc[2 * np + 1], ahi, xl[2], xl[3]);
              mma_bf16(acc[2 * np], alo, xh[0], xh[1]);
              mma_bf16(acc[2 * np + 1], alo, xh[2], xh[3]);
            }
          } else {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
              mma_bf16(acc[2 * np], ahi, bx[np][0], bx[np][1]);
              mma_bf16(acc[2 * np + 1], ahi, bx[np][2], bx[np][3]);
            }
#pragma unroll
            for (int np = 0; np < 4; ++np) {
              mma_bf16(acc[2 * np], alo, bx[np][0], bx[np][1]);
              mma_bf16(acc[2 * np + 1], alo, bx[np][2], bx[np][3]);
            }
          }
        }
        // fragments -> dtype of x -> staging (row stride 144 B: conflict-free) -> 128-byte row segments of gx
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          *reinterpret_cast<uint32_t*>(stg + g8 * kStgStride + (8 * j + 2 * t4) * 2) = pack_x2<T>(acc[j][0], acc[j][1]);
          *reinterpret_cast<uint32_t*>(stg + (g8 + 8) * kStgStride + (8 * j + 2 * t4) * 2) = pack_x2<T>(acc[j][2], acc[j][3]);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int id = i * 32 + lane, rr = id >> 3, c16 = id & 7;
          if (m0 + rr < P) {
            const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * kStgStride + c16 * 16);
            *reinterpret_cast<uint4*>(gxb + (size_t)(m0 + rr) * Cch + ch0 + c16 * 8) = v;
          }
        }
        __syncwarp();
      }
    }
    __syncthreads();  // the image buffer and the per-image tables are reused
    NFP_TSTAMP(6);  // image done
  }
}

// ---- host side --------------------------------------------------------------------------------------

struct Plan {
  bool ok;
  int nbuf, KS, nw, ctas;
  size_t smem;
};

template <class C, int MODE, int NW>
bool plan_try(const KParams& P, int nbuf, int budget, Plan& pl) {
  using G = Geo<C>;
  int ks = 1;
  while (ks < kMaxKS && ks * G::MT < NW && P.C % (2 * ks) == 0 && (P.C / (2 * ks)) % 16 == 0) ks *= 2;
  Lay<C, MODE, NW> L(P.C, nbuf, ks, P.Kin);
  if (L.total > budget) return false;
  pl.ok = true;
  pl.nbuf = nbuf;
  pl.KS = ks;
  pl.nw = NW;
  pl.smem = (size_t)L.total;
  return true;
}

template <class C, int MODE>
Plan plan_for(const KParams& P) {
  Plan pl{false, 0, 0, 0, 0, 0};
  if (P.C % 64 || P.C < 64) return pl;             // swizzle granule: 8 chunks of 8 channels
  if ((C::K * C::P * 2) % 16) return pl;           // upstream-gradient rows are fetched with 16-byte copies
  if (P.Kin && (C::R < 2 || (P.Kin * C::P * 2) % 16)) return pl;  // multi-radius: both gradient blocks
  static const int want_two = [] { const char* e = getenv("NFPB200_TOKEN_TWO_CTAS"); return e ? atoi(e) : 1; }();
  // two 8-warp CTAs per SM (one image buffer each) when they fit and there is more than one image per SM to overlap
  if (want_two && plan_try<C, MODE, kNWSmall>(P, 1, kSmemPerSM / 2 - 1024, pl)) {
    pl.ctas = 2;
    return pl;
  }
  if (plan_try<C, MODE, kNWBig>(P, 2, kSmemPerSM - 1024, pl) || plan_try<C, MODE, kNWBig>(P, 1, kSmemPerSM - 1024, pl)) pl.ctas = 1;
  return pl;
}

template <typename T, class C, int MODE, int NW>
int launch_nw(const KParams& P, const Plan& pl, TokenArgs a, cudaStream_t stream) {
  a.nbuf = pl.nbuf;
  a.KS = pl.KS;
  a.KSlog = 0;
  while ((1 << a.KSlog) < pl.KS) ++a.KSlog;
  auto kern = token_kernel<T, C, MODE, NW>;
  constexpr int kMaxDev = 64;
  static int sm_count[kMaxDev] = {0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < 0 || dev >= kMaxDev) return NFPB200_EDEVICE;
  if (sm_count[dev] == 0) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemPerSM);
    if (e != cudaSuccess) return (int)e;
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return (int)e;
    sm_count[dev] = n;
  }
  const Tables<C>* gt = tables_for<C>(a.pad_mode);
  if (!gt) return NFPB200_EINVAL;
  const int slots = sm_count[dev] * pl.ctas;
  const int grid = P.B < slots ? P.B : slots;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NW * 32);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return (int)cudaLaunchKernelEx(&cfg, kern, a, gt);
}

// the plan depends on the element size only (2 bytes for both dtypes): fp16 coverage is bf16 coverage
template <typename T, class C, int MODE>
int launch_mode(const KParams& P, TokenArgs a, cudaStream_t stream) {
  const Plan pl = plan_for<C, MODE>(P);
  if (!pl.ok) return NFPB200_EUNSUPPORTED;
  return pl.nw == kNWSmall ? launch_nw<T, C, MODE, kNWSmall>(P, pl, a, stream)
                           : launch_nw<T, C, MODE, kNWBig>(P, pl, a, stream);
}

template <typename T, class C>
int launch_cfg(const KParams& P, int mode, const TokenArgs& a, cudaStream_t stream) {
  switch (mode) {
    case MODE_FWD: return launch_mode<T, C, MODE_FWD>(P, a, stream);
    case MODE_BWD: return launch_mode<T, C, MODE_BWD>(P, a, stream);
    case MODE_POOL_FWD: return launch_mode<T, C, MODE_POOL_FWD>(P, a, stream);
    default: return launch_mode<T, C, MODE_POOL_BWD>(P, a, stream);
  }
}
template <class C>
bool plan_ok_cfg(const KParams& P, int mode) {
  switch (mode) {
    case MODE_FWD: return plan_for<C, MODE_FWD>(P).ok;
    case MODE_BWD: return plan_for<C, MODE_BWD>(P).ok;
    case MODE_POOL_FWD: return plan_for<C, MODE_POOL_FWD>(P).ok;
    default: return plan_for<C, MODE_POOL_BWD>(P).ok;
  }
}

template <typename T>
int launch_dtype(const KParams& P, int mode, const TokenArgs& a, cudaStream_t stream) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return launch_cfg<T, Cfg<H_, W_, R_, TW_>>(P, mode, a, stream);
  NFP_STREAM_SHAPES(X)
#undef X
  return NFPB200_EUNSUPPORTED;
}
int launch(const KParams& P, int dtype, int mode, const TokenArgs& a, cudaStream_t stream) {
  switch (dtype) {
    case NFPB200_BF16: return launch_dtype<bf16>(P, mode, a, stream);
    case NFPB200_F16: return launch_dtype<f16>(P, mode, a, stream);
    default: return NFPB200_EUNSUPPORTED;
  }
}
bool plan_ok(const KParams& P, int mode) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return plan_ok_cfg<Cfg<H_, W_, R_, TW_>>(P, mode);
  NFP_STREAM_SHAPES(X)
#undef X
  return false;
}

}  // namespace token

namespace {
int token_mode(int op) {
  switch (op) {
    case NFPB200_OP_FORWARD: return stream::MODE_FWD;
    case NFPB200_OP_BACKWARD: return stream::MODE_BWD;
    case NFPB200_OP_POOL_FORWARD: return stream::MODE_POOL_FWD;
    default: return stream::MODE_POOL_BWD;
  }
}
}  // namespace

bool token_supported(const KParams& P, int dtype, int measure, int op) {
  if ((dtype != NFPB200_BF16 && dtype != NFPB200_F16) || measure != NFPB200_COSINE) return false;
  if (P.stride != 1 || P.dil != 1 || P.pad != P.R || P.mode == NFPB200_PAD_CIRCULAR) return false;
  return token::plan_ok(P, token_mode(op));
}

const char* token_name(const KParams& P) {
  const char* nm = "fused/token";
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) nm = "fused/token_" #H_ "x" #W_ "_r" #R_;
  NFP_STREAM_SHAPES(X)
#undef X
  return nm;
}

int token_head_run(const KParams& P, int dtype, int op, const void* x, const float* proj_w, const float* proj_b,
                   float* out, float* gap_x, float* gap_nfp, const float* g_out, void* gx, const LaunchCtx& ctx) {
  token::TokenArgs a{};
  a.x = x; a.gx = gx; a.gap_x = gap_x; a.gap_nfp = gap_nfp;
  a.proj_w = proj_w; a.proj_b = proj_b; a.head_out = out; a.head_gout = g_out;
  a.B = P.B; a.C = P.C;
  const long long dense = (long long)P.H * P.W * P.C;
  a.xbs = P.x_batch_stride > 0 ? P.x_batch_stride : dense;
  a.gxbs = P.gx_batch_stride > 0 ? P.gx_batch_stride : dense;
  a.pad_mode = P.mode; a.similarity = P.similarity; a.eps = P.eps; a.y_f32 = 0;
  a.dbg = stream::g_debug_stamps.load(std::memory_order_relaxed);
  return token::launch(P, dtype, token_mode(op), a, ctx.stream);
}

int token_run(const KParams& P, int dtype, int op, const void* x, const void* gy, void* y, void* gx, const float* g_gap_x,
              const float* g_gap_nfp, float* gap_x, float* gap_nfp, const LaunchCtx& ctx) {
  token::TokenArgs a{};
  a.x = x; a.gy = gy; a.y = y; a.gx = gx;
  a.g_gap_x = g_gap_x; a.g_gap_nfp = g_gap_nfp; a.gap_x = gap_x; a.gap_nfp = gap_nfp;
  a.B = P.B; a.C = P.C;
  const long long dense = (long long)P.H * P.W * P.C;
  a.xbs = P.x_batch_stride > 0 ? P.x_batch_stride : dense;
  a.gxbs = P.gx_batch_stride > 0 ? P.gx_batch_stride : dense;
  a.pad_mode = P.mode; a.similarity = P.similarity; a.eps = P.eps; a.y_f32 = P.y_f32;
  a.kin = P.Kin; a.rin = P.rin;
  a.dbg = stream::g_debug_stamps.load(std::memory_order_relaxed);
  return token::launch(P, dtype, token_mode(op), a, ctx.stream);
}

}  // namespace nfp
