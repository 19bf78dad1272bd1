// Cluster-split fused NFP kernels for sm_100a: cosine measure, stride 1, dilation 1, padding = R
// (the configuration every live model path of the reference uses: models/NFP_Pooling.py:10-16,
// models/texture_pooling.py:232,302).  Included by nfp_split_f32.cu / nfp_split_bf16.cu.
//
// Work unit = (image b, channel slice s of S): a thread-block CLUSTER of S CTAs owns one image at a time, CTA `rank`
// owns the Cs = C/S channels [rank*Cs, (rank+1)*Cs) -- about 25 KB of x, which stays RESIDENT in its shared memory for
// the whole unit (one HBM read, no second pass through L2).  The grid is persistent: as many clusters as fit (3 small
// CTAs of 4 warps per SM), cluster c works on images c, c + G, ...; every CTA has NBUF = 2 unit buffers, so the next
// unit's x streams in while the current one is being processed, and the co-resident CTAs of an SM are in different
// phases: the HBM-bound streaming of one overlaps the shared-memory-bound stencil application of another
// (one-CTA-per-image grids run their phases in lock-step: B = 256 images are one wave on 148 SMs).
//
//   load     one elected thread issues NSUB TMA bulk copies (cp.async.bulk + mbarrier complete_tx), one per
//            sub-chunk of the unit, plus the stencil tables and the image's upstream gradient.
//   pass A   per-pixel |x_p|^2 and the dot products with the (k*k-1)/2 "forward" window neighbours over the unit's
//            channels, sub-chunk by sub-chunk as they land (lane = row strip x channel slot, packed fp32 pairs ->
//            FFMA2); the warps' partial tables are summed in a fixed order into the CTA's partial table.
//   exchange cluster barrier; every CTA sums the S partial tables through distributed shared memory (fixed rank
//            order: deterministic, identical bits in every CTA) -- only for the pixels it needs: CTA `rank` owns the
//            pixel slice [rank*P/S, (rank+1)*P/S) of the per-pixel work that follows (+ the window halo).
//   forward  y = dot / (max(|p|,eps) max(|q|,eps)) for the K taps of the CTA's pixel slice -> HBM; pooled mode
//            reduces over the slice and sends K partial sums to rank 0.
//   backward the closed-form stencil coefficients Wd[p][o] of ATen's cosine_similarity backward (SURVEY.md 8 a3;
//            gather form, no atomics) for the CTA's pixel slice, pushed into the shared memory of every CTA of
//            the cluster (st.shared::cluster); second cluster barrier; then
//   pass B   gx[c][p] = sum_o Wd[p][o] * x[c][p+o] on the resident channels.  7x7 maps with Cs % 64 == 0:
//            lane-per-channel form (a lane slides a k-row window down its own two planes: every x element is read
//            from shared memory once, coefficients as broadcast LDS.128, FFMA2, results in place, one TMA bulk
//            store per 64-channel task; when there are fewer tasks than warps a task is split into two row bands
//            that exchange their boundary rows through registers).  Everything else: strip form (lane = row strip x
//            channel slot, coefficients in registers, results staged per warp, TMA bulk stores).
//
// The (B, C*(k*k-1), H, W) neighbour tensor of the reference (nfp.py:153-154) never exists; x is read from HBM once
// per kernel and gx written once.
#pragma once

#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "nfp_common.cuh"
#include "nfp_ptx.cuh"
#include "nfp_split.h"
#include "nfp_stream.h"
#include "nfp_tables.cuh"

namespace nfp {
namespace split {

using namespace ptx;
using stream::align_up;
using stream::Cfg;
using stream::Tables;
using stream::tables_for;
using stream::MODE_BWD;
using stream::MODE_FWD;
using stream::MODE_POOL_BWD;
using stream::MODE_POOL_FWD;


constexpr int kNW = 4;           // warps per CTA
constexpr int kMaxS = 8;         // portable cluster size limit
constexpr int kMaxSub = 8;
constexpr int kNBuf = 2;         // unit buffers per CTA (double buffering of the resident x)
constexpr int kSmemPerSM = 227 * 1024;
constexpr int kLeadPad = 128;    // zeroed bytes in front of / behind the resident x (halo reads of the first / last plane)


// CTAs per SM the register budget is sized for (shared memory allows 3 with two 25 KB unit buffers)
template <class C>
__host__ __device__ constexpr int min_ctas() { return 3; }

// Shared-memory layout (byte offsets); everything but the resident x has a compile-time size.
template <typename T, class C, int MODE, int NW>
struct Lay {
  static constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  static constexpr int ESZ = (int)sizeof(T);
  int bars, tfull, tpart, inv, rn, wd, tabs, gp, gyraw, poolp, ggx, uni, wtab, stg, ytab, lead, xs, total;
  int t_fv, t_fd, t_q, t_fsrc, t_fdst, t_fptr;
  int stg_warp, gy_stride, x_stride;
  __host__ __device__ Lay(int Cs, bool lanech) {
    int o = 0;
    auto take = [&](int n) { int r = o; o += (n + 127) & ~127; return r; };
    bars = take((kNBuf * (kMaxSub + 2) + 2) * 8);
    tfull = take(C::PNV * 4);
    tpart = take(C::PNV * 4);
    inv = take(C::P * 4);
    rn = take(BWD ? C::P * 4 : 0);
    wd = take(BWD ? C::H * C::RS * 4 : 0);
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
    gp = take(BWD ? C::P * C::KK * 4 : 0);
    gy_stride = align_up(C::K * C::P * ESZ, 128);
    gyraw = take(MODE == MODE_BWD ? kNBuf * gy_stride : (MODE == MODE_POOL_BWD ? C::K * 4 : 0));
    poolp = take(MODE == MODE_POOL_FWD ? kMaxS * C::K * 4 : 0);
    ggx = take(MODE == MODE_POOL_BWD ? Cs * 4 : 0);
    // union: the warps' partial tables (pass A .. table sum) | store staging of the strip-form pass B | pooled y tile
    uni = o;
    wtab = take(NW * C::PNV * 4);
    const int u1 = o;
    o = uni;
    stg_warp = 2 * align_up(2 * C::CPW * C::P * ESZ, 16);
    stg = take((BWD && !lanech) ? NW * stg_warp : 0);
    const int u2 = o;
    o = uni;
    ytab = take(MODE == MODE_POOL_FWD ? C::K * C::P * 4 : 0);
    const int u3 = o;
    o = u1 > u2 ? (u1 > u3 ? u1 : u3) : (u2 > u3 ? u2 : u3);
    // [zero pad][unit buffer 0][zero pad][unit buffer 1][zero pad]: a pad serves the buffer before and after it
    lead = take(kLeadPad);
    x_stride = align_up(Cs * C::P * ESZ + kLeadPad, 128);
    xs = take(kNBuf * x_stride);
    total = o;
  }
};

// ---- lane-per-channel pass B on the rows [RB, RE) of a 64-channel task -------------------------------------------
// p0 / p1: this lane's two channel planes (resident x, overwritten in place by gx).  When the task is split into two
// row bands (another warp works on the other rows of the same planes) the R boundary rows that belong to the other
// band are read into registers BEFORE the pair barrier BAR, i.e. before either warp overwrites anything.
template <typename T, class C, int RB, int RE, int BAR>
__device__ __forceinline__ void lanech_rows(unsigned char* p0, unsigned char* p1, const float4* wd4, uint64_t gpair) {
  constexpr int W = C::W, R = C::R, k = C::k, KK = C::KK, H = C::H;
  constexpr int ESZ = (int)sizeof(T);
  constexpr bool BANDED = (RB > 0 || RE < H);
  constexpr int NLO = (RB > 0) ? R : 0, NHI = (RE < H) ? R : 0;
  auto ldrow = [&](int q, int j) -> uint64_t {
    return pack2(ldx<T>(p0 + (q * W + j) * ESZ), ldx<T>(p1 + (q * W + j) * ESZ));
  };
  uint64_t hlo[NLO ? NLO : 1][W], hhi[NHI ? NHI : 1][W];
#pragma unroll
  for (int i = 0; i < NLO; ++i)
#pragma unroll
    for (int j = 0; j < W; ++j) hlo[i][j] = (RB - R + i >= 0) ? ldrow(RB - R + i, j) : 0ull;
#pragma unroll
  for (int i = 0; i < NHI; ++i)
#pragma unroll
    for (int j = 0; j < W; ++j) hhi[i][j] = (RE + i < H) ? ldrow(RE + i, j) : 0ull;
  if constexpr (BANDED) named_sync<BAR, 64>();
  // map row q (compile-time after unrolling): zero outside the map, registers for the other band's rows
  auto fetch = [&](int q, int j) -> uint64_t {
    if (q < 0 || q >= H) return 0ull;
    if (q < RB) return hlo[q - (RB - R)][j];
    if (q >= RE) return hhi[q - RE][j];
    return ldrow(q, j);
  };
  // rows rr-R .. rr+R of the two planes, rotating: map row q lives in win[q mod k]
  uint64_t win[k][W];
#pragma unroll
  for (int q = RB - R; q < RB + R; ++q)
#pragma unroll
    for (int j = 0; j < W; ++j) win[((q % k) + k) % k][j] = fetch(q, j);
#pragma unroll
  for (int rr = RB; rr < RE; ++rr) {
#pragma unroll
    for (int j = 0; j < W; ++j) win[(rr + R) % k][j] = fetch(rr + R, j);
    uint64_t out[W];
#pragma unroll
    for (int j = 0; j < W; ++j) out[j] = gpair;
    // the row's W*KK coefficients, four at a time (warp-uniform address: one wavefront per load)
#pragma unroll
    for (int q4 = 0; q4 < C::RS4; ++q4) {
      const float4 c4 = wd4[rr * (C::RS / 4) + q4];
      const float cw[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = q4 * 4 + e;
        if (i < W * KK) {
          const int j = i / KK, o = i % KK, dy = o / k - R, dx = o % k - R;
          if (j + dx >= 0 && j + dx < W && rr + dy >= 0 && rr + dy < H)
            out[j] = fma2(pack2(cw[e], cw[e]), win[(rr + dy + k) % k][j + dx], out[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < W; ++j) {
      float lo, hi;
      unpack2(out[j], lo, hi);
      stx<T>(p0 + (rr * W + j) * ESZ, lo);
      stx<T>(p1 + (rr * W + j) * ESZ, hi);
    }
  }
}

template <typename T, class C, int MODE, int NW>
__global__ void __launch_bounds__(NW * 32, min_ctas<C>()) split_kernel(const SplitArgs a, const Tables<C>* __restrict__ gt) {
  constexpr int W = C::W, R = C::R, TW = C::TW, k = C::k, KK = C::KK, K = C::K, P = C::P;
  constexpr int NV = C::NV, PNV = C::PNV, NS = C::NS, NSX = C::NSX, CPW = C::CPW, LANES = C::LANES;
  constexpr int XW = C::XW, XOFF = C::XOFF;
  constexpr int NT = NW * 32;
  constexpr int ESZ = (int)sizeof(T);
  constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  constexpr bool POOLED = (MODE == MODE_POOL_FWD || MODE == MODE_POOL_BWD);
  constexpr int GSTRIDE = CPW * P * ESZ;  // bytes between consecutive channel groups
  constexpr int PSTRIDE = 2 * GSTRIDE;    // one work item = a pair of groups
  constexpr int GY_BYTES = K * P * ESZ;
  constexpr int HALOP = R * W + R;        // pixels a window reaches before / after its centre
  constexpr int NBUF = kNBuf;

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int S = a.S, Cs = a.Cs, NSUB = a.NSUB;
  const Lay<T, C, MODE, NW> L(Cs, a.lanech != 0);
  uint64_t* xfull = reinterpret_cast<uint64_t*>(smem_raw + L.bars);  // [NBUF][kMaxSub]
  uint64_t* gyfull = xfull + NBUF * kMaxSub;                           // [NBUF]
  uint64_t* empty = gyfull + NBUF;                                     // [NBUF]: every warp is done with the buffer
  uint64_t* tabfull = empty + NBUF;
  float* tfull = reinterpret_cast<float*>(smem_raw + L.tfull);
  float* tpart = reinterpret_cast<float*>(smem_raw + L.tpart);
  float* inv = reinterpret_cast<float*>(smem_raw + L.inv);
  float* wtab = reinterpret_cast<float*>(smem_raw + L.wtab);

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int rank = (S > 1) ? (int)cluster_ctarank() : 0;
  const int G = (int)gridDim.x / S, cid = (int)blockIdx.x / S;  // clusters in the grid, this cluster
  const int nmine = (a.B - cid + G - 1) / G;                    // images of this cluster: cid, cid + G, ...
  const int ch0 = rank * Cs;                                    // first channel of this CTA's units
  // the pixel slice whose per-pixel work (forward values / stencil coefficients) this CTA does, and the range of
  // table pixels that work reads
  const int p0 = rank * P / S, p1 = (rank + 1) * P / S, np = p1 - p0;
  const int plo = p0 - HALOP > 0 ? p0 - HALOP : 0, phi = p1 + HALOP < P ? p1 + HALOP : P;
  const uint32_t sub_bytes = (uint32_t)(a.sub_ch * P * ESZ);
  const bool x_early = BWD && a.x_early;

  if (tid == 0) {
    for (int j = 0; j < NBUF * kMaxSub; ++j) mbar_init(&xfull[j], 1);
    for (int j = 0; j < NBUF; ++j) {
      mbar_init(&gyfull[j], 1);
      mbar_init(&empty[j], NW);
    }
    mbar_init(tabfull, 1);
    fence_mbar_init();
  }
  __syncthreads();
  // loads of this cluster's i-th image into unit buffer i % NBUF (one elected thread)
  auto issue_x = [&](int i) {
    const int bb = cid + i * G, bf = i % NBUF;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(a.x) + ((size_t)bb * a.C + ch0) * P * ESZ;
    unsigned char* dst = smem_raw + L.xs + bf * L.x_stride;
    for (int j = 0; j < NSUB; ++j) {
      mbar_expect_tx(&xfull[bf * kMaxSub + j], sub_bytes);
      bulk_g2s(dst + (size_t)j * sub_bytes, src + (size_t)j * sub_bytes, sub_bytes, &xfull[bf * kMaxSub + j]);
    }
  };
  auto issue_gy = [&](int i) {
    if constexpr (MODE == MODE_BWD) {
      const int bb = cid + i * G, bf = i % NBUF;
      mbar_expect_tx(&gyfull[bf], (uint32_t)GY_BYTES);
      bulk_g2s(smem_raw + L.gyraw + bf * L.gy_stride, reinterpret_cast<const T*>(a.gy) + (size_t)bb * K * P,
               (uint32_t)GY_BYTES, &gyfull[bf]);
    }
  };
  const int npre = nmine < NBUF ? nmine : NBUF;
  if (tid == 0) {
    // the stencil tables are constants: fetch them before waiting for the preceding grid
    constexpr uint32_t TAB_BYTES = BWD ? Tables<C>::BWD_BYTES : Tables<C>::FWD_BYTES;
    mbar_expect_tx(tabfull, TAB_BYTES);
    bulk_g2s(smem_raw + L.tabs, reinterpret_cast<const unsigned char*>(gt) + (BWD ? Tables<C>::BWD_OFFSET : 0), TAB_BYTES,
             tabfull);
    // PDL: x (without the x-stable hint) and the upstream gradient are produced by the preceding grid.  Dependents
    // are released only AFTER this grid's own wait returned, so an early-starting dependent never overlaps the
    // grid BEFORE this one (the x-stable hint of include/nfp_b200.h stays safe in chains of any length).
    if (x_early) {
      for (int i = 0; i < npre; ++i) issue_x(i);
    } else {
      grid_dependency_wait();
      grid_launch_dependents();
      for (int i = 0; i < npre; ++i) {
        issue_gy(i);
        issue_x(i);
      }
    }
  }
  // zero the pads around the unit buffers: the strip-form pass B multiplies what it reads outside a channel plane by
  // zero coefficients, so those values only have to be finite (pass A never uses the accumulators they feed)
  if constexpr (BWD) {
    const int gapw = (L.x_stride - Cs * P * ESZ) / 4;  // words between the end of a unit buffer and the next one
    for (int i = tid; i < kLeadPad / 4; i += NT) reinterpret_cast<uint32_t*>(smem_raw + L.lead)[i] = 0u;
    for (int bf = 0; bf < NBUF; ++bf) {
      uint32_t* z = reinterpret_cast<uint32_t*>(smem_raw + L.xs + bf * L.x_stride + (size_t)Cs * P * ESZ);
      for (int i = tid; i < gapw; i += NT) z[i] = 0u;
    }
  }
  if (!x_early) grid_dependency_wait();

  const float sgn = a.similarity ? 1.f : -1.f;
  const bool lane_on = lane < LANES;
  const int chslot = lane_on ? lane / NS : 0;
  const int pos = lane_on ? lane % NS : 0;
  const int r = pos / NSX, c0 = (pos % NSX) * TW;
  const int toff = (chslot * P + r * W + c0) * ESZ;  // byte offset of this lane's strip inside a group
  const int nitems = Cs / (2 * CPW);                 // work items (group pairs) of a unit
  const int items_per_sub = a.sub_ch / (2 * CPW);
#define NFP_OFF(dy, jj) (((dy) * W + (jj) - XOFF) * ESZ)
#define NFP_ISTAMP(k) do { if (a.dbg && tid == 0 && it < 2) a.dbg[((size_t)blockIdx.x * 2 + it) * 8 + (k)] = globaltimer_ns(); } while (0)

  for (int it = 0; it < nmine; ++it) {
    const int b = cid + it * G;
    const int buf = it % NBUF;
    const uint32_t par = (uint32_t)((it / NBUF) & 1);
    unsigned char* xs = smem_raw + L.xs + buf * L.x_stride;
    uint64_t* xf = xfull + buf * kMaxSub;
    NFP_ISTAMP(0);

    // ---- backward: the gy-only part of the stencil, S[p][o] = sum of G over the taps of p that land on q = p + off(o),
    // plus the taps of q that land on p (o == ctr: the taps of p that land on p itself, replicate padding), for the
    // pixels of this CTA's slice.  Gather form: no atomics, fixed order.  Runs behind the x loads (first image with
    // the x-stable hint: after pass A, which then overlaps the tail of the preceding launch).
    auto stencil_part = [&]() {
      if constexpr (BWD) {
        const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
        const int16_t* fsrc = reinterpret_cast<const int16_t*>(smem_raw + L.t_fsrc);
        const int16_t* fdst = reinterpret_cast<const int16_t*>(smem_raw + L.t_fdst);
        const int16_t* fptr = reinterpret_cast<const int16_t*>(smem_raw + L.t_fptr);
        float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
        float* Gp = reinterpret_cast<float*>(smem_raw + L.gp);
        const unsigned char* g = smem_raw + L.gyraw + (POOLED ? 0 : buf * L.gy_stride);
        if constexpr (POOLED) {
          // d GAP(y) / dy: the same value on every pixel of a tap plane
          if (tid < K) reinterpret_cast<float*>(smem_raw + L.gyraw)[tid] = a.g_gap_nfp[(size_t)b * K + tid] * (1.f / (float)P);
          float* gs = reinterpret_cast<float*>(smem_raw + L.ggx);
          for (int i = tid; i < Cs; i += NT) gs[i] = a.g_gap_x[(size_t)b * a.C + ch0 + i];
          __syncthreads();
        } else {
          mbar_wait(&gyfull[buf], par);
        }
        if (it == 0) mbar_wait(tabfull, 0);
        auto Gv = [&](int flat) -> float {  // upstream gradient element n*P + p
          if constexpr (POOLED) return reinterpret_cast<const float*>(smem_raw + L.gyraw)[flat / P];
          else return ldx<T>(g + flat * ESZ);
        };
        // G'[p][o] = gradient of the taps of p that land on p + off(o): the direct tap ...
        for (int idx = plo * KK + tid; idx < phi * KK; idx += NT) {
          const int p = idx / KK, o = idx - p * KK;
          float v = 0.f;
          if (o != C::CTR && qt[idx] >= 0) v = Gv((o < C::CTR ? o : o - 1) * P + p);
          Gp[idx] = v;
        }
        __syncthreads();
        // ... plus, on border pixels, the taps folded back by the padding (one thread per entry, fixed order)
        const int nfd = fptr[Tables<C>::NFP - 1];
        for (int i = tid; i < nfd; i += NT) {
          const int dst = fdst[i];
          if (dst < plo * KK || dst >= phi * KK) continue;
          float v = Gp[dst];
          for (int j = fptr[i]; j < fptr[i + 1]; ++j) v += Gv(fsrc[j]);
          Gp[dst] = v;
        }
        __syncthreads();
        // S[p][o] = G'[p][o] + G'[q][-o]  (o == ctr: the taps of p that land on p itself, counted once)
        for (int idx = p0 * KK + tid; idx < p1 * KK; idx += NT) {
          const int p = idx / KK, o = idx - p * KK;
          const int q = (o == C::CTR) ? -1 : (int)qt[idx];
          float v = Gp[idx];
          if (q >= 0) v += Gp[q * KK + (KK - 1 - o)];
          Wd[C::widx(p, o)] = sgn * v;
        }
      }
    };
    const bool early_now = x_early && it == 0;
    if (!early_now) stencil_part();

    // ---- pass A: per-pixel |x|^2 and forward-direction dots over the unit's channels --------------------------------
    {
      float accs[TW][NV];
      int landed = 0;  // sub-chunks this thread has already waited for
      auto wait_sub = [&](int item) {
        const int need = item / items_per_sub + 1;
        while (landed < need) {
          mbar_wait(&xf[landed++], par);
          if (landed == 1) NFP_ISTAMP(5);  // first sub-chunk landed
        }
      };
      if constexpr (MODE == MODE_POOL_FWD) {
        // GAP(x) of the unit's channels (NFP_Pooling.py:27): one lane per channel plane
        for (int c = tid; c < Cs; c += NT) {
          wait_sub(c / (2 * CPW));
          const unsigned char* pl = xs + (size_t)c * P * ESZ;
          float s = 0.f;
#pragma unroll 7
          for (int e = 0; e < P; ++e) s += ldx<T>(pl + e * ESZ);
          a.gap_x[(size_t)b * a.C + ch0 + c] = s / (float)P;
        }
      }
      if constexpr (C::PACK) {
        uint64_t acc[TW][NV];
#pragma unroll
        for (int j = 0; j < TW; ++j)
#pragma unroll
          for (int v = 0; v < NV; ++v) acc[j][v] = 0ull;
        for (int item = warp; item < nitems; item += NW) {
          wait_sub(item);
          const unsigned char* pa = xs + (size_t)item * PSTRIDE + toff;
          if (lane_on) {
            uint64_t xr[R + 1][XW];
#pragma unroll
            for (int dy = 0; dy <= R; ++dy)
#pragma unroll
              for (int jj = 0; jj < XW; ++jj)
                xr[dy][jj] = pack2(ldx<T>(pa + NFP_OFF(dy, jj)), ldx<T>(pa + GSTRIDE + NFP_OFF(dy, jj)));
#pragma unroll
            for (int j = 0; j < TW; ++j) {
              const uint64_t c = xr[0][j + XOFF];
              acc[j][0] = fma2(c, c, acc[j][0]);
#pragma unroll
              for (int dx = 1; dx <= R; ++dx) {
                if (j + dx + XOFF < XW) acc[j][dx] = fma2(c, xr[0][j + dx + XOFF], acc[j][dx]);
              }
#pragma unroll
              for (int dy = 1; dy <= R; ++dy)
#pragma unroll
                for (int dx = -R; dx <= R; ++dx) {
                  if (j + dx + XOFF >= 0 && j + dx + XOFF < XW)
                    acc[j][dy * k + dx] = fma2(c, xr[dy][j + dx + XOFF], acc[j][dy * k + dx]);
                }
            }
          }
        }
#pragma unroll
        for (int j = 0; j < TW; ++j)
#pragma unroll
          for (int v = 0; v < NV; ++v) accs[j][v] = sum2(acc[j][v]);
      } else {
#pragma unroll
        for (int j = 0; j < TW; ++j)
#pragma unroll
          for (int v = 0; v < NV; ++v) accs[j][v] = 0.f;
        for (int item = warp; item < nitems; item += NW) {
          wait_sub(item);
          const unsigned char* pa = xs + (size_t)item * PSTRIDE + toff;
          if (lane_on) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const unsigned char* ph_ = pa + h * GSTRIDE;
              float xr[R + 1][XW];
#pragma unroll
              for (int dy = 0; dy <= R; ++dy)
#pragma unroll
                for (int jj = 0; jj < XW; ++jj) xr[dy][jj] = ldx<T>(ph_ + NFP_OFF(dy, jj));
#pragma unroll
              for (int j = 0; j < TW; ++j) {
                const float c = xr[0][j + XOFF];
                accs[j][0] = fmaf(c, c, accs[j][0]);
#pragma unroll
                for (int dx = 1; dx <= R; ++dx) {
                  if (j + dx + XOFF < XW) accs[j][dx] = fmaf(c, xr[0][j + dx + XOFF], accs[j][dx]);
                }
#pragma unroll
                for (int dy = 1; dy <= R; ++dy)
#pragma unroll
                  for (int dx = -R; dx <= R; ++dx) {
                    if (j + dx + XOFF >= 0 && j + dx + XOFF < XW)
                      accs[j][dy * k + dx] = fmaf(c, xr[dy][j + dx + XOFF], accs[j][dy * k + dx]);
                  }
              }
            }
          }
        }
      }
      // every thread observes every sub-chunk barrier of the unit (pass B reads all of them)
      while (landed < NSUB) mbar_wait(&xf[landed++], par);
      // sum over the channel slots of the warp (fixed shuffle tree: deterministic), then publish the warp's table
      if constexpr (CPW > 1) {
#pragma unroll
        for (int d = LANES / 2; d >= NS; d >>= 1)
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) accs[j][v] += __shfl_down_sync(0xffffffffu, accs[j][v], d);
      }
      if (lane < NS) {
        float* wt = wtab + warp * PNV + pos * (TW * NV);
#pragma unroll
        for (int j = 0; j < TW; ++j)
#pragma unroll
          for (int v = 0; v < NV; ++v) wt[j * NV + v] = accs[j][v];
      }
    }
    NFP_ISTAMP(1);  // pass A done
    // ---- refill: the unit buffer that has just become free takes this cluster's image NBUF ahead of its last user
    {
      // forward: pass A was the last reader of this image's buffer; backward: the previous image's buffer is free
      // once its pass B stores have read it (every warp arrives on `empty` when it is done with the buffer)
      const int done_it = BWD ? it - 1 : it;
      if constexpr (!BWD) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[buf]);
      }
      if (tid == 0 && done_it >= 0 && done_it + NBUF < nmine) {
        mbar_wait(&empty[done_it % NBUF], (uint32_t)((done_it / NBUF) & 1));
        issue_gy(done_it + NBUF);
        issue_x(done_it + NBUF);
      }
    }
    if (early_now) {
      grid_dependency_wait();
      if (tid == 0) {
        grid_launch_dependents();
        for (int i = 0; i < npre; ++i) issue_gy(i);
      }
      stencil_part();
    }
    __syncthreads();
    // the CTA's partial table (its channels): the warps' tables in a fixed order
    for (int i = tid; i < PNV; i += NT) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < NW; ++w) s += wtab[w * PNV + i];
      tpart[i] = s;
    }
    if (S > 1) {
      cluster_arrive();
      cluster_wait();
    } else {
      __syncthreads();
    }
    NFP_ISTAMP(6);  // partial tables exchanged
    // the image's table over all channels: the S partial tables in rank order (identical bits in every CTA), for the
    // pixels this CTA's slice needs
    {
      const uint32_t tp = smem_u32(tpart);
      for (int i = plo * NV + tid; i < phi * NV; i += NT) {
        float s;
        if (S > 1) {
          float part[kMaxS];
#pragma unroll
          for (int rr = 0; rr < kMaxS; ++rr)
            part[rr] = rr < S ? ld_dsmem_f32(dsmem_addr(tp + 4u * (uint32_t)i, (uint32_t)rr)) : 0.f;
          s = part[0];
#pragma unroll
          for (int rr = 1; rr < kMaxS; ++rr)
            if (rr < S) s += part[rr];
        } else {
          s = tpart[i];
        }
        tfull[i] = s;
        if (i % NV == 0) {  // |x_p|^2: the clamped inverse norm (and, backward, the 1/(N |x|) of the norm term)
          const int p = i / NV;
          const float nrm = sqrtf(s), N = fmaxf(nrm, a.eps);
          inv[p] = 1.f / N;
          if constexpr (BWD) reinterpret_cast<float*>(smem_raw + L.rn)[p] = nrm > 0.f ? 1.f / (N * nrm) : 0.f;
        }
      }
    }
    __syncthreads();
    NFP_ISTAMP(7);  // table reduced

    if constexpr (!BWD) {
      // ---- forward value for the CTA's pixel slice -----------------------------------------------------------
      if (it == 0) mbar_wait(tabfull, 0);
      const int16_t* fv = reinterpret_cast<const int16_t*>(smem_raw + L.t_fv);
      const int16_t* fd = reinterpret_cast<const int16_t*>(smem_raw + L.t_fd);
      float* ytab = reinterpret_cast<float*>(smem_raw + L.ytab);
      if constexpr (!POOLED) {
        if (S > 1) cluster_arrive();  // this CTA is done reading its peers' tables (wait: end of the image)
      }
      for (int idx = tid; idx < K * np; idx += NT) {
        const int n = idx / np, p = p0 + (idx - n * np);
        const int v = fv[n * P + p];
        float yv = 0.f;
        if (v >= 0) yv = tfull[fd[n * P + p]] * (inv[p] * inv[v]);
        if (!a.similarity) yv = 1.f - yv;
        if constexpr (POOLED) {
          ytab[idx] = yv;
        } else {
          if (a.y_f32) reinterpret_cast<float*>(a.y)[((size_t)b * K + n) * P + p] = yv;
          else reinterpret_cast<T*>(a.y)[((size_t)b * K + n) * P + p] = from_f32<T>(yv);
        }
      }
      if constexpr (POOLED) {
        // GAP over the plane of every tap (NFP_Pooling.py:31): the slice's partial sums go to rank 0
        __syncthreads();
        float* poolp = reinterpret_cast<float*>(smem_raw + L.poolp);
        for (int n = warp; n < K; n += NW) {
          float s = 0.f;
          for (int i = lane; i < np; i += 32) s += ytab[n * np + i];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lane == 0) {
            if (S > 1) st_dsmem_f32(dsmem_addr(smem_u32(poolp + rank * K + n), 0u), s);
            else a.gap_nfp[(size_t)b * K + n] = s / (float)P;
          }
        }
        if (S > 1) {
          cluster_arrive();
          cluster_wait();
          if (rank == 0 && tid < K) {
            float s = 0.f;
            for (int rr = 0; rr < S; ++rr) s += poolp[rr * K + tid];
            a.gap_nfp[(size_t)b * K + tid] = s / (float)P;
          }
        }
      } else {
        if (S > 1) cluster_wait();  // peers may still be reading this CTA's partial table
      }
      NFP_ISTAMP(2);  // forward outputs written
    } else {
      // ---- backward: stencil coefficients of the CTA's pixel slice.  Wd holds S[p][o] (the gy-only part); scale
      // by the inverse norms and close the centre tap:
      //   Wd[p][o]   = S[p][o] / (N_p N_q)
      //   Wd[p][ctr] = sw - (1/(N_p |x_p|)) * (sum_o Wd[p][o] dot(p, q_o) + sw |x_p|^2),  sw = 2 S[p][ctr] / N_p^2
      // and push them into the coefficient table of every CTA of the cluster.
      const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
      const float* rn = reinterpret_cast<const float*>(smem_raw + L.rn);
      float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
      const uint32_t wda = smem_u32(Wd);
      auto push = [&](int wi, float v) {
        if (S > 1) {
          for (int rr = 0; rr < S; ++rr) st_dsmem_f32(dsmem_addr(wda + 4u * (uint32_t)wi, (uint32_t)rr), v);
        } else {
          Wd[wi] = v;
        }
      };
      // eight lanes per pixel share the window offsets; fixed shuffle tree -> deterministic
      for (int i8 = tid; i8 < align_up(np * 8, 32); i8 += NT) {
        const int p = p0 + (i8 >> 3), g = i8 & 7;
        const bool valid = (i8 >> 3) < np;
        const float ip = valid ? inv[p] : 0.f;
        float s = 0.f;
        if (valid) {
#pragma unroll
          for (int t = 0; t < (K + 7) / 8; ++t) {
            const int n = g + 8 * t;          // neighbour number (window order, centre removed)
            if (n < K) {
              const int o = n < C::CTR ? n : n + 1;
              const int q = qt[p * KK + o];
              float w = 0.f;
              if (q >= 0) {
                w = Wd[C::widx(p, o)] * (ip * inv[q]);
                const float d = o > C::CTR ? tfull[p * NV + (o - C::CTR)] : tfull[q * NV + (C::CTR - o)];
                s = fmaf(w, d, s);
              }
              push(C::widx(p, o), w);
            }
          }
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if (valid && g == 0) {
          const float sw = 2.f * Wd[C::widx(p, C::CTR)] * (ip * ip);
          push(C::widx(p, C::CTR), sw - rn[p] * (s + sw * tfull[p * NV]));
        }
      }
      if (S > 1) {
        cluster_arrive();
        cluster_wait();
      } else {
        __syncthreads();
      }
      NFP_ISTAMP(2);  // coefficients ready
      // ---- pass B: gx = stencil(x) on the resident channels --------------------------------------------------------
      const float invP = 1.f / (float)P;
      unsigned char* gxb = reinterpret_cast<unsigned char*>(a.gx) + ((size_t)b * a.C + ch0) * P * ESZ;
      const float* ggx = reinterpret_cast<const float*>(smem_raw + L.ggx);
      bool lanech_done = false;
      if constexpr (C::LANECH) {
        if (a.lanech) {
          lanech_done = true;
          const int ntask = Cs / C::TASK;
          const float4* wd4 = reinterpret_cast<const float4*>(Wd);
          auto task_planes = [&](int t, unsigned char*& q0, unsigned char*& q1, uint64_t& gpair) {
            q0 = xs + (size_t)(t * C::TASK + lane) * P * ESZ;
            q1 = q0 + 32 * P * ESZ;
            float g0 = 0.f, g1 = 0.f;
            if constexpr (MODE == MODE_POOL_BWD) {
              g0 = ggx[t * C::TASK + lane] * invP;
              g1 = ggx[t * C::TASK + 32 + lane] * invP;
            }
            gpair = pack2(g0, g1);
          };
          auto store_task = [&](int t) {
            bulk_s2g(gxb + (size_t)t * C::TASK * P * ESZ, xs + (size_t)t * C::TASK * P * ESZ, (uint32_t)(C::TASK * P * ESZ));
            bulk_commit();
          };
          constexpr int HB = (C::H + 1) / 2;  // rows of the first band when a task is split in two
          if (NW == 4 && 2 * ntask <= NW && C::H >= 4) {
            // fewer tasks than warp pairs: two warps per task, one row band each
            const int t = warp >> 1, band = warp & 1;
            if (t < ntask) {
              unsigned char *q0, *q1;
              uint64_t gpair;
              task_planes(t, q0, q1, gpair);
              if (t == 0) {
                if (band == 0) lanech_rows<T, C, 0, HB, 2>(q0, q1, wd4, gpair);
                else lanech_rows<T, C, HB, C::H, 2>(q0, q1, wd4, gpair);
                fence_async_smem();
                named_sync<2, 64>();  // both bands of the task are written
              } else {
                if (band == 0) lanech_rows<T, C, 0, HB, 3>(q0, q1, wd4, gpair);
                else lanech_rows<T, C, HB, C::H, 3>(q0, q1, wd4, gpair);
                fence_async_smem();
                named_sync<3, 64>();
              }
              if (band == 0 && lane == 0) store_task(t);
            }
          } else {
            for (int t = warp; t < ntask; t += NW) {
              unsigned char *q0, *q1;
              uint64_t gpair;
              task_planes(t, q0, q1, gpair);
              lanech_rows<T, C, 0, C::H, 2>(q0, q1, wd4, gpair);
              fence_async_smem();
              __syncwarp();
              if (lane == 0) store_task(t);
            }
          }
          NFP_ISTAMP(3);  // pass B done
        }
      }
      if (!lanech_done) {
        unsigned char* mystg = smem_raw + L.stg + warp * L.stg_warp;
        const int stg_half = L.stg_warp / 2;
        int nstore = 0;
        const float* wdp = Wd + C::widx(r * W + c0, 0);
        float wr[(R == 1) ? TW : 1][(R == 1) ? KK : 1];
        if constexpr (R == 1) {
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int o = 0; o < KK; ++o) wr[j][o] = wdp[j * KK + o];
        }
        for (int item = warp; item < nitems; item += NW) {
          const unsigned char* pa = xs + (size_t)item * PSTRIDE + toff;
          unsigned char* sb = mystg + (nstore & 1) * stg_half;
          if (nstore >= 2) {
            if (lane == 0) bulk_wait_read<1>();  // the store that last used this buffer has read it
            __syncwarp();
          }
          if (lane_on) {
            // the two channel groups of the item share the coefficients, so the FMAs run on packed fp32 pairs (lo =
            // group 0, hi = group 1): ptxas folds the duplicated coefficient into FFMA2's scalar-broadcast operand
            float g0 = 0.f, g1 = 0.f;
            if constexpr (MODE == MODE_POOL_BWD) {
              const float* gp = ggx + 2 * item * CPW + chslot;
              g0 = gp[0] * invP;
              g1 = gp[CPW] * invP;
            }
            uint64_t out[TW];
#pragma unroll
            for (int j = 0; j < TW; ++j) out[j] = pack2(g0, g1);
#pragma unroll
            for (int dy = -R; dy <= R; ++dy) {
              // 3x3: all k*k coefficients of the strip live in registers; wider windows: one window row at a time
              float wrow[(R == 1) ? 1 : TW][(R == 1) ? 1 : k];
              if constexpr (R != 1) {
#pragma unroll
                for (int j = 0; j < TW; ++j)
#pragma unroll
                  for (int dx = 0; dx < k; ++dx) wrow[j][dx] = wdp[j * KK + (dy + R) * k + dx];
              }
              uint64_t xr[XW];
#pragma unroll
              for (int jj = 0; jj < XW; ++jj)
                xr[jj] = pack2(ldx<T>(pa + NFP_OFF(dy, jj)), ldx<T>(pa + GSTRIDE + NFP_OFF(dy, jj)));
              // dx outer, j inner: consecutive FMAs go to different accumulators (no 4-cycle chains)
#pragma unroll
              for (int dx = -R; dx <= R; ++dx)
#pragma unroll
                for (int j = 0; j < TW; ++j) {
                  if (j + dx + XOFF >= 0 && j + dx + XOFF < XW) {
                    float w;
                    if constexpr (R == 1) w = wr[j][(dy + R) * k + dx + R];
                    else w = wrow[j][dx + R];
                    out[j] = fma2(pack2(w, w), xr[j + dx + XOFF], out[j]);
                  }
                }
            }
#pragma unroll
            for (int j = 0; j < TW; ++j) {
              float lo, hi;
              unpack2(out[j], lo, hi);
              stx<T>(sb + toff + j * ESZ, lo);
              stx<T>(sb + GSTRIDE + toff + j * ESZ, hi);
            }
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            // the item's 2*CPW planes are contiguous in gx
            bulk_s2g(gxb + (size_t)item * PSTRIDE, sb, (uint32_t)PSTRIDE);
            bulk_commit();
          }
          ++nstore;
        }
        NFP_ISTAMP(3);  // pass B done
      }
      // this warp is done with the unit buffer (and with its staging) once its stores have read shared memory
      if (lane == 0) {
        bulk_wait_read<0>();
        mbar_arrive(&empty[buf]);
      }
      __syncwarp();
    }
    NFP_ISTAMP(4);
    // the per-image tables (Wd, Gp, tfull, wtab / staging, ...) are rewritten by the next image
    if (it + 1 < nmine) __syncthreads();
  }
#undef NFP_OFF
#undef NFP_ISTAMP
}

// ---- host side --------------------------------------------------------------------------------------

struct Plan {
  bool ok;
  int S, Cs, NSUB, sub_ch, lanech, ctas_per_sm;
  size_t smem;
};

// resident clusters of a kernel configuration (cluster placement accounts for GPC boundaries); cached per device
template <typename K>
int max_clusters(K kern, int S, size_t smem, int dev) {
  constexpr int kMaxDev = 64;
  static int cache[kMaxDev][kMaxS + 1] = {};
  if (cache[dev][S] > 0) return cache[dev][S];
  int n = 0;
  if (S > 1) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(S * 1024));
    cfg.blockDim = dim3(kNW * 32);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) n = 0;
  } else {
    int per_sm = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kNW * 32, smem) == cudaSuccess &&
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess)
      n = per_sm * sms;
  }
  if (n < 1) n = 1;
  cache[dev][S] = n;
  return n;
}

template <typename T, class C, int MODE>
Plan plan_for(const KParams& P) {
  Plan best{false, 0, 0, 0, 0, 0, 0, 0};
  constexpr int esz = (int)sizeof(T);
  constexpr bool bwd = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  constexpr int item = 2 * C::CPW;  // work item: a pair of channel groups
  constexpr int target_bytes = 25 * 1024 + 512;  // unit size
  constexpr int want_sub = 4;
  static_assert(want_sub <= kMaxSub, "sub-chunk barriers");
  if (((size_t)C::K * C::P * esz) % 16) return best;
  long best_cost = -1;
  for (int S = 1; S <= kMaxS; ++S) {
    if (P.C % S) continue;
    const int Cs = P.C / S;
    if (Cs % item) continue;
    const long bytes = (long)Cs * C::P * esz;
    if (bytes % 16) continue;
    if (((size_t)item * C::P * esz) % 16) continue;  // TMA bulk store granularity of the strip form
    const int lanech = (bwd && C::LANECH && Cs % C::TASK == 0) ? 1 : 0;
    Lay<T, C, MODE, kNW> L(Cs, lanech != 0);
    if (L.total > kSmemPerSM - 1024) continue;
    long cost = bytes > target_bytes ? 2 * (bytes - target_bytes) : (target_bytes - bytes);
    if (bwd && C::LANECH && !lanech) cost += 16 * 1024;
    if (best_cost >= 0 && cost >= best_cost) continue;
    // sub-chunks: as close to `want_sub` as the channel count allows (whole work items, 16-byte multiples)
    int nsub = 0;
    for (int n = want_sub; n >= 1; --n) {
      if (Cs % n) continue;
      const int sc = Cs / n;
      if (sc % item) continue;
      if (((size_t)sc * C::P * esz) % 16) continue;
      nsub = n;
      break;
    }
    if (!nsub) continue;
    best_cost = cost;
    best.ok = true;
    best.S = S;
    best.Cs = Cs;
    best.NSUB = nsub;
    best.sub_ch = Cs / nsub;
    best.lanech = lanech;
    best.smem = (size_t)L.total;
    int ctas = kSmemPerSM / (L.total + 1024);
    if (ctas > min_ctas<C>()) ctas = min_ctas<C>();
    best.ctas_per_sm = ctas;
  }
  return best;
}

template <typename T, class C, int MODE>
int launch_mode(const KParams& P, SplitArgs a, cudaStream_t stream) {
  const Plan pl = plan_for<T, C, MODE>(P);
  if (!pl.ok) return NFPB200_EUNSUPPORTED;
  a.S = pl.S;
  a.Cs = pl.Cs;
  a.NSUB = pl.NSUB;
  a.sub_ch = pl.sub_ch;
  a.lanech = pl.lanech;
  auto kern = split_kernel<T, C, MODE, kNW>;
  // per-device one-time setup (function attributes are per device; a process may drive several GPUs).
  // Idempotent, so a race between two host threads doing it at once is harmless.
  constexpr int kMaxDev = 64;
  static bool ready[kMaxDev] = {false};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < 0 || dev >= kMaxDev) return NFPB200_EDEVICE;
  if (!ready[dev]) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemPerSM);
    if (e != cudaSuccess) return (int)e;
    ready[dev] = true;
  }
  const Tables<C>* gt = tables_for<C>(a.pad_mode);
  if (!gt) return NFPB200_EINVAL;
  int G = max_clusters(kern, pl.S, pl.smem, dev);
  if (G > P.B) G = P.B;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(G * pl.S));
  cfg.blockDim = dim3(kNW * 32);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (pl.S > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)pl.S;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[na].val.programmaticStreamSerializationAllowed = 1;
  ++na;
  cfg.attrs = attr;
  cfg.numAttrs = na;
  cudaError_t lrc = cudaLaunchKernelEx(&cfg, kern, a, gt);
  if (lrc != cudaSuccess && getenv("NFPB200_VERBOSE")) {
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, kern);
    fprintf(stderr, "[nfpb200] split launch failed (%d): grid %d cluster %d dyn smem %zu static %zu regs %d\n", (int)lrc,
            G * pl.S, pl.S, pl.smem, fa.sharedSizeBytes, fa.numRegs);
  }
  return (int)lrc;
}

template <typename T, class C>
int launch_cfg(const KParams& P, int mode, const SplitArgs& a, cudaStream_t stream) {
  switch (mode) {
    case MODE_FWD: return launch_mode<T, C, MODE_FWD>(P, a, stream);
    case MODE_BWD: return launch_mode<T, C, MODE_BWD>(P, a, stream);
    case MODE_POOL_FWD: return launch_mode<T, C, MODE_POOL_FWD>(P, a, stream);
    default: return launch_mode<T, C, MODE_POOL_BWD>(P, a, stream);
  }
}
template <typename T, class C>
Plan plan_cfg(const KParams& P, int mode) {
  switch (mode) {
    case MODE_FWD: return plan_for<T, C, MODE_FWD>(P);
    case MODE_BWD: return plan_for<T, C, MODE_BWD>(P);
    case MODE_POOL_FWD: return plan_for<T, C, MODE_POOL_FWD>(P);
    default: return plan_for<T, C, MODE_POOL_BWD>(P);
  }
}

template <typename T>
int launch_dtype(const KParams& P, int mode, const SplitArgs& a, cudaStream_t stream) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return launch_cfg<T, Cfg<H_, W_, R_, TW_>>(P, mode, a, stream);
  NFP_STREAM_SHAPES(X)
#undef X
  return NFPB200_EUNSUPPORTED;
}
template <typename T>
Plan plan_dtype(const KParams& P, int mode) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return plan_cfg<T, Cfg<H_, W_, R_, TW_>>(P, mode);
  NFP_STREAM_SHAPES(X)
#undef X
  return Plan{false, 0, 0, 0, 0, 0, 0, 0};
}

}  // namespace split
}  // namespace nfp
