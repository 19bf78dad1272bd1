// Streaming fused NFP kernels for sm_100a: cosine measure, stride 1, dilation 1, padding = R
// (the configuration every live model path of the reference uses: models/NFP_Pooling.py:10-16,
// models/texture_pooling.py:232,302).  Included by nfp_stream_f32.cu / nfp_stream_bf16.cu / nfp_stream_f16.cu.
//
// One CTA owns one image at a time (persistent loop over b = blockIdx.x, += gridDim.x).  Inside
// the CTA one PRODUCER warp streams the image's x as chunks of CC channels (CC x H x W contiguous
// elements of the NCHW tensor) into a shared-memory ring with TMA bulk copies (cp.async.bulk +
// mbarrier complete_tx); NW CONSUMER warps work on the chunks as they land:
//
//   pass A   per-pixel |x_p|^2 and the dot products with the (k*k-1)/2 "forward" window
//            neighbours (dot(p,q) == dot(q,p): half the window suffices).  A lane owns a TW-pixel
//            row strip of TWO channels and keeps the strip's accumulators in registers as packed
//            fp32 pairs (fma.rn.f32x2 -> FFMA2: one issue slot per two FMAs); partial tables are
//            summed over lanes and warps through shared memory once per image, in a fixed order.
//   forward  y = dot / (max(|p|,eps) max(|q|,eps)) for the K taps -> the only HBM write;
//            pooled mode reduces y and x over the plane instead (nfp_pooling head).
//   backward the table + gy become a per-pixel k x k stencil of coefficients Wd[p][o] (closed form
//            of ATen's cosine_similarity backward, SURVEY.md 8 a3; gather form, no atomics): the gy-only part
//            S[p][o] is built from compile-time fold tables before pass A (behind the first loads), then
//            closed with the inverse norms after it; then
//   pass B   gx[c][p] = sum_o Wd[p][o] * x[c][p+o], chunk by chunk.  If the whole image fits in
//            the ring ("resident") the chunks of pass A are still there; otherwise the producer
//            streams them a second time -- they were read microseconds ago by the same SM, so
//            the second read is served by the 126 MB L2, not by HBM.  Two forms:
//            lane-per-channel (7x7 maps, C % 64 == 0): a warp owns 64 channels, a lane slides a k-row
//            window down its own two planes (each x element read from shared memory once, coefficients
//            as broadcast LDS.128, FFMA2), results in place, one TMA bulk store per task;
//            strip (everything else): lane = (row strip, channel slot), coefficients in registers,
//            results staged per warp and written with TMA bulk stores.
//
// The index arithmetic of the stencil (reflect / replicate / zero padding, tap order of
// nfp.py:64-67) is evaluated at COMPILE time into __device__ const tables.
// The (B, C*(k*k-1), H, W) neighbour tensor of the reference (nfp.py:153-154) never exists, x is
// read from HBM once per kernel, and no cluster / grid synchronisation is needed: images are
// independent and all resident CTAs have their loads in flight together.
#pragma once

#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "nfp_common.cuh"
#include "nfp_ptx.cuh"
#include "nfp_stream.h"

// pass B on packed fp32 pairs (FFMA2 with scalar-broadcast coefficients) vs scalar FFMA: A/B switch
#ifndef NFP_PASSB_FFMA2
#define NFP_PASSB_FFMA2 1
#endif

#include "nfp_tables.cuh"

// timing experiments (variant builds only -- `python -m neighbour_feature_pooling_b200.build --variant x -DNFP_DBG_...=1`,
// selected with NFPB200_LIB; results are wrong): compile out the arithmetic of pass A / everything after pass A in the
// forward / the forward's value loop, to see what the launch structure alone costs
// (profiles/r02_ubench_cold_read_floor.txt)
// forward: per-lane partial tables instead of the shuffle tree over the channel slots (A/B switch)
#ifndef NFP_FWD_DIRECT_PUBLISH
#define NFP_FWD_DIRECT_PUBLISH 1
#endif
#ifndef NFP_DBG_SKIP_PASSA
#define NFP_DBG_SKIP_PASSA 0
#endif
#ifndef NFP_DBG_SKIP_TAIL
#define NFP_DBG_SKIP_TAIL 0
#endif
#ifndef NFP_DBG_SKIP_EPI
#define NFP_DBG_SKIP_EPI 0
#endif
// same-tree baseline for the L2 prefetch before the dependency wait (results are unchanged either way)
#ifndef NFP_DBG_NO_L2_PREFETCH
#define NFP_DBG_NO_L2_PREFETCH 0
#endif

namespace nfp {
namespace stream {


using namespace ptx;
#define NFP_STAMP(k) do { if (a.dbg && tid == 0 && img == 0) a.dbg[(size_t)blockIdx.x * 8 + (k)] = globaltimer_ns(); } while (0)

constexpr int kMaxStages = 8;
// warps of a CTA: NW consumers and one producer (TMA issue)
__host__ __device__ constexpr int block_threads(int mode, int nw) {
  (void)mode;
  return (nw + 1) * 32;
}
constexpr int kNW = 8;                  // consumer warps
constexpr int kSmemPerSM = 227 * 1024;
constexpr int kLeadPad = 128;           // zeroed bytes in front of the ring (halo reads of the first plane)
// pause between two rounds of L2 prefetch lines (32 KB per CTA) before the dependency wait.  B200, 512x7x7 fp32 step
// at 128 / 256 / 512 ns: 21.05 / 20.95 / 20.79 us, but 512 slows the 2x2 and the 7x7 bf16 maps
constexpr unsigned kPrefetchPauseNs = 256;

// Shared-memory layout (byte offsets).  Fixed regions first, then a union: the per-warp partial
// tables of pass A are dead once the image's table is summed, the backward scratch / store staging
// and the pooled-forward y tile live after that.
template <typename T, class C, int MODE, int NW>
struct Smem {
  static constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  static constexpr int ESZ = (int)sizeof(T);
  int slot_stride, lead, ring, ggx, bars, tfull, inv, tabs, gyraw, uni, total;
  int t_fv, t_fd, t_q, t_fsrc, t_fdst, t_fptr;  // copies of the stencil tables
  int rn, wd, gp;                              // backward: 1/(N |x|) per pixel, stencil coefficients, stencil-warp scratch
  int wtab, stg, ytab;                         // inside the union
  int stg_warp;                                // staging bytes per warp (two buffers)
  int gyin, gyin_stride;                       // multi-radius backward: the inner radius' gradient block (two images in flight)
  // backward pass A publishes its per-warp tables in two rounds (upper half of the warps, then the lower half adds its
  // own on top): half the table space, one more barrier -- what lets a 512x7x7 fp32 image stay resident (below)
  static constexpr int NWT = BWD ? NW / 2 : NW;
  // forward: every lane publishes its own partial table (no shuffle tree over the channel slots; the table sum then
  // runs over NW * CPW tables) -- the forward has the shared memory for it, and its tail is latency-bound
  // (7x7 maps: 32 tables, -0.25 us; with 64 / 128 tables on 4x4 / 2x2 maps the longer sum costs more than the tree)
  static constexpr bool DIRECT = !BWD && (C::CPW > 1) && (C::CPW <= 4) && (NFP_FWD_DIRECT_PUBLISH != 0);
  static constexpr int NTAB = DIRECT ? NW * C::CPW : NWT;
  // lanech: the lane-per-channel pass B is in use -> no per-warp store staging, no pads between the ring slots (it
  // reads no halo; pass A's halo reads feed accumulators nobody uses, so they may land in the next slot);
  // gy_bufs: upstream-gradient buffers (1 when every CTA handles a single image)
  // bdirect: the BACKWARD publishes per-lane tables too (run-time choice: it costs 27 KB, i.e. the resident image)
  static constexpr bool BDIRECT_OK = BWD && (C::CPW > 1) && (C::CPW <= 4);
  __host__ __device__ Smem(int CC, int nst, int Cfull, int kin = 0, int lanech = 0, int gy_bufs = 2, int bdirect = 0) {
    int o = 0;
    auto take = [&](int n) { int r = o; o += (n + 127) & ~127; return r; };
    // everything whose size is known at compile time comes first (so its address is a constant in the
    // kernel); the ring, whose geometry depends on the run-time chunk size and stage count, comes last
    bars = take((2 * kMaxStages + 8) * 8);
    tfull = take(C::PNV * 4);
    inv = take(C::P * 4);
    rn = take(BWD ? C::P * 4 : 0);
    wd = take(BWD ? C::H * C::RS * 4 : 0);
    gp = take(BWD ? C::P * C::KK * 4 : 0);
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
    uni = o;
    wtab = take(((BDIRECT_OK && bdirect) ? NW * C::CPW : NTAB) * C::PNV * 4);  // partial tables of the warps / lanes
    const int u1 = o;
    o = uni;
    stg_warp = 2 * align_up(2 * C::CPW * C::P * ESZ, 16);
    stg = take(lanech ? 0 : NW * stg_warp);
    const int u2 = BWD ? o : uni;
    o = uni;
    ytab = take(C::K * C::P * 4);
    const int u3 = (MODE == MODE_POOL_FWD) ? o : uni;
    o = u1 > u2 ? (u1 > u3 ? u1 : u3) : (u2 > u3 ? u2 : u3);
    // (run-time sized regions from here on)
    gyraw = BWD ? take(gy_bufs * align_up(C::K * C::P * ESZ, 16)) : o;
    // each slot: chunk bytes, then >= HALO zeroed elements (shared with the next slot's "before" halo);
    // kLeadPad zeroed bytes in front of the first slot, one pad behind the last
    slot_stride = lanech ? align_up(CC * C::P * ESZ, 128) : align_up(CC * C::P * ESZ + C::HALO * ESZ, 128);
    lead = take(kLeadPad);
    ring = take(nst * slot_stride + (lanech ? 128 : 0));
    ggx = take(MODE == MODE_POOL_BWD ? 2 * Cfull * 4 : 0);  // pooled backward: d out / d GAP(x) of two images in flight
    gyin_stride = align_up(kin * C::P * ESZ, 16);
    gyin = take(MODE == MODE_BWD ? 2 * gyin_stride : 0);
    total = o;
  }
};

// register budget: 9 warps/CTA put up to 3 (1 CTA/SM) or 5 (2 CTAs/SM) warps on one SM sub-partition
// (16 K registers each) -> at most 96 registers per thread for 2 CTAs/SM, 168 for one
template <typename T, class C, int MODE, int NW>
__global__ void __launch_bounds__(block_threads(MODE, NW), C::MINB) stream_kernel(const StreamArgs a, const Tables<C>* __restrict__ gt) {
  constexpr int W = C::W, R = C::R, TW = C::TW, k = C::k, KK = C::KK, K = C::K, P = C::P;
  constexpr int NV = C::NV, PNV = C::PNV, NS = C::NS, NSX = C::NSX, CPW = C::CPW, LANES = C::LANES;
  constexpr int XW = C::XW, XOFF = C::XOFF;
  constexpr int NT = NW * 32;  // consumer threads
  constexpr int ESZ = (int)sizeof(T);
  constexpr bool BWD = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  constexpr bool POOLED = (MODE == MODE_POOL_FWD || MODE == MODE_POOL_BWD);
  constexpr int GSTRIDE = CPW * P * ESZ;  // bytes between consecutive channel groups
  constexpr int PSTRIDE = 2 * GSTRIDE;    // one work item = a pair of groups
  constexpr int GY_BYTES = K * P * ESZ;
  constexpr int GY_STRIDE = align_up(GY_BYTES, 16);

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int nst = a.nst, NCH = a.NCH, CC = a.CC;
  const Smem<T, C, MODE, NW> L(CC, nst, a.C, a.kin, BWD && a.lanech, a.gy_bufs, a.bdirect);
  unsigned char* ring = smem_raw + L.ring;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  uint64_t* empty = full + kMaxStages;
  uint64_t* gyfull = empty + kMaxStages;
  uint64_t* gyempty = gyfull + 2;
  uint64_t* tabfull = gyempty + 2;
  volatile uint32_t* dep_done = reinterpret_cast<volatile uint32_t*>(tabfull + 1);  // the producer's wait returned
  float* tfull = reinterpret_cast<float*>(smem_raw + L.tfull);
  float* inv = reinterpret_cast<float*>(smem_raw + L.inv);
  float* wtab = reinterpret_cast<float*>(smem_raw + L.wtab);

  // warp index through a shuffle: tells the compiler it is warp-uniform (uniform registers / datapath for the
  // per-warp address arithmetic)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const bool resident = BWD && a.resident;
  const uint32_t chunk_bytes = (uint32_t)(CC * P * ESZ);

  if (tid == 0) {
    for (int s = 0; s < nst; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], NW);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&gyfull[s], 1);
      mbar_init(&gyempty[s], 1);
    }
    mbar_init(tabfull, 1);
    *dep_done = 0u;
    fence_mbar_init();
  }
  __syncthreads();

  // ================================ producer warp ==================================================
  if (warp == NW) {
    if (lane == 0) {
      // the stencil tables are constants: fetch them before waiting for the preceding grid
      constexpr uint32_t TAB_BYTES = BWD ? Tables<C>::BWD_BYTES : Tables<C>::FWD_BYTES;
      mbar_expect_tx(tabfull, TAB_BYTES);
      bulk_g2s(smem_raw + L.tabs, reinterpret_cast<const unsigned char*>(gt) + (BWD ? Tables<C>::BWD_OFFSET : 0),
               TAB_BYTES, tabfull);
      // PDL: the upstream gradient (and, without the x-stable hint, x) is produced by the preceding grid.  With the
      // hint the first image's x chunks go out first (a ring-full of them), the wait comes before its gradient loads.
      // Dependents are released only AFTER this grid's own wait returned: an early-starting dependent then never
      // overlaps the grid BEFORE this one, so the x-stable hint is safe in launch chains of any length.
      bool dep_pending = BWD && a.x_early;
      if (!dep_pending) {
        grid_dependency_wait();
        *dep_done = 1u;
        grid_launch_dependents();
      }
      int slot = 0, img = 0;
      uint32_t phbits = 0;  // per-slot phase parity (every pass restarts at slot 0)
      const int npass = (BWD && !resident) ? 2 : 1;
      auto load_grads = [&](int b, int img) {
        if (MODE == MODE_BWD) {
          const int par = img & 1;
          mbar_wait(&gyempty[par], ((img >> 1) & 1) ^ 1);
          // multi-radius launch: the image's gradient is [kin inner-radius planes | K planes]; two copies, one barrier
          const uint32_t gin_bytes = (uint32_t)(a.kin * P * ESZ);
          const T* gb = reinterpret_cast<const T*>(a.gy) + (size_t)b * (K + a.kin) * P;
          mbar_expect_tx(&gyfull[par], (uint32_t)GY_BYTES + gin_bytes);
          bulk_g2s(smem_raw + L.gyraw + par * GY_STRIDE, gb + a.kin * P, (uint32_t)GY_BYTES, &gyfull[par]);
          if (gin_bytes) bulk_g2s(smem_raw + L.gyin + par * L.gyin_stride, gb, gin_bytes, &gyfull[par]);
        }
        if (MODE == MODE_POOL_BWD && a.ggx_tma) {  // the image's d out / d GAP(x): C floats, one bulk copy
          const int par = img & 1;
          mbar_wait(&gyempty[par], ((img >> 1) & 1) ^ 1);
          mbar_expect_tx(&gyfull[par], (uint32_t)a.C * 4u);
          bulk_g2s(smem_raw + L.ggx + par * a.C * 4, a.g_gap_x + (size_t)b * a.C, (uint32_t)a.C * 4u, &gyfull[par]);
        }
      };
      for (int b = blockIdx.x; b < a.B; b += gridDim.x, ++img) {
        if (!dep_pending) load_grads(b, img);
        const unsigned char* xb = reinterpret_cast<const unsigned char*>(a.x) + (size_t)b * a.C * P * ESZ;
        int issued = 0;
        for (int pass = 0; pass < npass; ++pass) {
          const unsigned char* src = xb;
          slot = 0;
          for (int ch = 0; ch < NCH; ++ch, src += chunk_bytes, ++issued) {
            if (dep_pending && issued == nst) {  // the ring is full of the first image's x: now wait, then its gradients
              grid_dependency_wait();
              grid_launch_dependents();
              dep_pending = false;
              load_grads(b, img);
            }
            mbar_wait(&empty[slot], ((phbits >> slot) & 1u) ^ 1u);
            mbar_expect_tx(&full[slot], chunk_bytes);
            bulk_g2s(ring + slot * L.slot_stride, src, chunk_bytes, &full[slot]);
            phbits ^= 1u << slot;
            if (++slot == nst) slot = 0;
          }
        }
        if (dep_pending) {  // fewer chunks than ring stages
          grid_dependency_wait();
          grid_launch_dependents();
          dep_pending = false;
          load_grads(b, img);
        }
      }
    }
    return;
  }

  // ================================ consumer warps =================================================
  // prologue (overlaps the first TMA loads): zero the halo pads.  Pass B multiplies the values read
  // outside a channel plane by zero coefficients, so they only have to be finite; pass A never
  // uses the accumulators they feed.
  if constexpr (BWD) {
    uint32_t* z = reinterpret_cast<uint32_t*>(smem_raw + L.lead);
    for (int i = tid; i < kLeadPad / 4; i += NT) z[i] = 0u;
    const int pad_words = (L.slot_stride - (int)chunk_bytes) / 4;
    for (int s = 0; s < nst; ++s) {
      uint32_t* zp = reinterpret_cast<uint32_t*>(ring + s * L.slot_stride + chunk_bytes);
      for (int i = tid; i < pad_words; i += NT) zp[i] = 0u;
    }
    if (a.lanech) {  // no pads between the slots: one behind the last
      uint32_t* zp = reinterpret_cast<uint32_t*>(ring + nst * L.slot_stride);
      for (int i = tid; i < 32; i += NT) zp[i] = 0u;
    }
  }
  // While the preceding grid still runs, warm L2 with the inputs of this CTA's first a.pf_imgs images, in the order
  // they are consumed, so that their HBM stream overlaps that grid's tail.  A prefetch moves no data into the SM:
  // everything this grid consumes is still read after griddepcontrol.wait, from L2 -- the point of coherence every
  // write of the preceding grid goes through -- so the data consumed is the same, also when x or gy is an output of
  // the preceding grid.  Every address is inside the caller's buffers.  The consumer threads issue one line each per
  // round and pause between rounds; they stop as soon as the producer's wait has returned: from then on the ring
  // loads stream the image in order, and prefetching further ahead would only make the first chunks land later (an
  // unpaced prefetch of the whole image costs 0.6 us per fp32 launch after a non-NFP kernel, where nothing overlaps;
  // a bulk prefetch from the producer, cp.async.bulk.prefetch.L2, queues ahead of the ring loads in the TMA unit and
  // costs 1.4 us).  With the x-stable hint the producer streams x before its wait itself.
  if (!NFP_DBG_NO_L2_PREFETCH && !(BWD && a.x_early)) {
    bool stop = false;
    auto prefetch_range = [&](const void* base, size_t bytes) {
      const unsigned char* p = reinterpret_cast<const unsigned char*>(base);
      for (size_t off = 0; off < bytes && !stop; off += (size_t)NT * 128) {
        if (*dep_done) {
          stop = true;
          break;
        }
        if (off + (size_t)tid * 128 < bytes) prefetch_l2(p + off + (size_t)tid * 128);
        if (tid == 0 && off + (size_t)NT * 128 >= bytes) prefetch_l2(p + bytes - 1);  // last line, base not 128-aligned
        __nanosleep(kPrefetchPauseNs);
      }
    };
    int n = 0;
    for (int b = blockIdx.x; b < a.B && n < a.pf_imgs && !stop; b += gridDim.x, ++n) {
      if (MODE == MODE_BWD)
        prefetch_range(reinterpret_cast<const unsigned char*>(a.gy) + (size_t)b * (K + a.kin) * P * ESZ,
                       (size_t)(K + a.kin) * P * ESZ);
      if (MODE == MODE_POOL_BWD && a.g_gap_x) prefetch_range(a.g_gap_x + (size_t)b * a.C, (size_t)a.C * 4);
      prefetch_range(reinterpret_cast<const unsigned char*>(a.x) + (size_t)b * a.C * P * ESZ, (size_t)a.C * P * ESZ);
    }
  }
  // PDL: nothing below may touch global memory the preceding grid still uses -- except, with the x-stable hint, the
  // ring (x only): then pass A of the first image runs first and the wait comes right after it
  const bool x_early = BWD && a.x_early;
  if (!x_early) grid_dependency_wait();
  consumer_sync<NT>();

  const float sgn = a.similarity ? 1.f : -1.f;
  const bool lane_on = lane < LANES;
  const int chslot = lane_on ? lane / NS : 0;
  const int pos = lane_on ? lane % NS : 0;
  const int r = pos / NSX, c0 = (pos % NSX) * TW;
  const int toff = (chslot * P + r * W + c0) * ESZ;  // byte offset of this lane's strip inside a group
  const int npairs = CC / (2 * CPW);                 // group pairs per chunk
  // byte offset of window element (dy, column jj of the loaded row) relative to the strip start
#define NFP_OFF(dy, jj) (((dy) * W + (jj) - XOFF) * ESZ)

  int slot = 0, img = 0;
  uint32_t phbits = 0;  // per-slot phase parity, in step with the producer's
  NFP_STAMP(0);  // consumers ready
  for (int b = blockIdx.x; b < a.B; b += gridDim.x, ++img) {
    const uint32_t phbits0 = phbits;
    slot = 0;

    // ---- backward, before pass A (overlaps the latency of the first chunk loads) or, with the x-stable hint,
    // right after it (pass A overlaps the tail of the preceding launch instead): the gy-only part of the
    // stencil, S[p][o] = sum of G over the taps of p that land on q = p + off(o), plus the taps of q that land on p
    // (o == ctr: the taps of p that land on p itself, replicate padding).  Gather form: no atomics, fixed order.
    auto stencil_part = [&]() {
    if constexpr (BWD) {
      const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
      const int16_t* fsrc = reinterpret_cast<const int16_t*>(smem_raw + L.t_fsrc);
      const int16_t* fdst = reinterpret_cast<const int16_t*>(smem_raw + L.t_fdst);
      const int16_t* fptr = reinterpret_cast<const int16_t*>(smem_raw + L.t_fptr);
      float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
      float* Gp = reinterpret_cast<float*>(smem_raw + L.gp);
      if (img == 0) mbar_wait(tabfull, 0);  // stencil tables (fetched by the producer at kernel start)
      const int par = img & 1;
      const unsigned char* g = smem_raw + L.gyraw + par * GY_STRIDE;
      if constexpr (POOLED) {
        bool head_done = false;
        if constexpr (MODE == MODE_POOL_BWD) {
          if (a.proj_w) {
            // fused head backward (NFP_Pooling.py:31-35): from d loss / d out, the forward's GAP(x) and GAP(NFP(x)):
            //   d/d GAP(x)[c]      = g_out[c] * (proj_w[c] . gnfp + proj_b[c])
            //   d/d GAP(NFP(x))[n] = sum_c g_out[c] * GAP(x)[c] * proj_w[c][n]      (fixed-order block reduction)
            head_done = true;
            float* gs = reinterpret_cast<float*>(smem_raw + L.ggx) + (img & 1) * a.C;
            float gn[K], part[K];
#pragma unroll
            for (int n = 0; n < K; ++n) {
              gn[n] = a.gap_nfp[(size_t)b * K + n];
              part[n] = 0.f;
            }
            for (int c = tid; c < a.C; c += NT) {
              const float go = a.head_gout[(size_t)b * a.C + c], gxv = a.gap_x[(size_t)b * a.C + c];
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
              gs[c] = go * proj;
            }
#pragma unroll
            for (int n = 0; n < K; ++n) {
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) part[n] += __shfl_xor_sync(0xffffffffu, part[n], o);
              if (lane == 0) Gp[warp * K + n] = part[n];   // Gp is free until the stencil loops below
            }
            consumer_sync<NT>();
            if (tid < K) {
              float sred = 0.f;
              for (int w = 0; w < NW; ++w) sred += Gp[w * K + tid];
              reinterpret_cast<float*>(smem_raw + L.gyraw)[tid] = sred * (1.f / (float)P);
            }
          }
        }
        if (!head_done) {
          // d GAP(y) / dy: the same value on every pixel of a tap plane
          if (tid < K) reinterpret_cast<float*>(smem_raw + L.gyraw)[tid] = a.g_gap_nfp[(size_t)b * K + tid] * (1.f / (float)P);
          if constexpr (MODE == MODE_POOL_BWD) {
            if (!a.ggx_tma) {  // rows not 16-byte aligned / sized: no bulk copy, stage them with plain loads
              float* gs = reinterpret_cast<float*>(smem_raw + L.ggx) + (img & 1) * a.C;
              for (int i = tid; i < a.C; i += NT) gs[i] = a.g_gap_x[(size_t)b * a.C + i];
            }
          }
        }
        consumer_sync<NT>();
      } else {
        mbar_wait(&gyfull[par], (img >> 1) & 1);
      }
      const unsigned char* gin = smem_raw + L.gyin + par * L.gyin_stride;
      auto G = [&](int flat) -> float {  // upstream gradient element n*P + p
        if constexpr (POOLED) {
          return reinterpret_cast<const float*>(smem_raw + L.gyraw)[flat / P];
        } else {
          float v = ldx<T>(g + flat * ESZ);
          if constexpr (R >= 2) {
            if (a.kin) {  // multi-radius launch: the same tap of the inner radius' map adds its gradient
              const int n = flat / P, n1 = inner_tap(n, R, a.rin);
              if (n1 >= 0) v += ldx<T>(gin + (n1 * P + flat - n * P) * ESZ);
            }
          }
          return v;
        }
      };
      // G'[p][o] = gradient of the taps of p that land on p + off(o): the direct tap ...
      for (int idx = tid; idx < P * KK; idx += NT) {
        const int p = idx / KK, o = idx - p * KK;
        float v = 0.f;
        if (o != C::CTR && qt[idx] >= 0) v = G((o < C::CTR ? o : o - 1) * P + p);
        Gp[idx] = v;
      }
      consumer_sync<NT>();
      // ... plus, on border pixels, the taps folded back by the padding (one thread per entry, fixed order)
      const int nfd = fptr[Tables<C>::NFP - 1];
      for (int i = tid; i < nfd; i += NT) {
        const int dst = fdst[i];
        float v = Gp[dst];
        for (int j = fptr[i]; j < fptr[i + 1]; ++j) v += G(fsrc[j]);
        Gp[dst] = v;
      }
      consumer_sync<NT>();
      if constexpr (!POOLED) {
        if (tid == 0) mbar_arrive(&gyempty[par]);  // every read of the raw gy happened before the barrier
      }
      // S[p][o] = G'[p][o] + G'[q][-o]  (o == ctr: the taps of p that land on p itself, counted once)
      for (int idx = tid; idx < P * KK; idx += NT) {
        const int p = idx / KK, o = idx - p * KK;
        const int q = (o == C::CTR) ? -1 : (int)qt[idx];
        float v = Gp[idx];
        if (q >= 0) v += Gp[q * KK + (KK - 1 - o)];
        Wd[C::widx(p, o)] = sgn * v;
      }
      // (Wd is next touched after the barriers that follow pass A; Gp is rewritten by the next image after them too)
    }
    };
    if (!x_early) stencil_part();

    // ---- pass A: per-pixel |x|^2 and forward-direction dots, streamed over the chunks -----------
    {
      float accs[TW][NV];
      if constexpr (C::PACK) {
        uint64_t acc[TW][NV];
#pragma unroll
        for (int j = 0; j < TW; ++j)
#pragma unroll
          for (int v = 0; v < NV; ++v) acc[j][v] = 0ull;
        for (int ch = 0; ch < NCH; ++ch) {
          mbar_wait(&full[slot], (phbits >> slot) & 1u);
          const unsigned char* sl = ring + slot * L.slot_stride;
          if constexpr (MODE == MODE_POOL_FWD) {
            // GAP(x) of this chunk's channels (NFP_Pooling.py:27): one lane per channel plane; the job rotates
            // over the warps chunk by chunk.  (Measured alternative, not kept: row sums from the strips pass A
            // already holds in registers + a shuffle tree over the strips -- 11.4 vs 8.7 us, shuffles share the
            // shared-memory data path and the extra live values spill.)
            const int w0 = (ch * 2) % NW;
            for (int c = ((warp - w0 + NW) % NW) * 32 + lane; c < CC; c += NT) {
              const unsigned char* pl = sl + c * P * ESZ;
              float s = 0.f;
#pragma unroll 7
              for (int e = 0; e < P; ++e) s += ldx<T>(pl + e * ESZ);
              a.gap_x[(size_t)b * a.C + ch * CC + c] = s / (float)P;
            }
          }
          const unsigned char* pa = sl + warp * PSTRIDE + toff;
          for (int it = warp; it < npairs; it += NW, pa += NW * PSTRIDE) {
            if (lane_on && !NFP_DBG_SKIP_PASSA) {
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
          if (!resident) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[slot]);
          }
          phbits ^= 1u << slot;
          if (++slot == nst) slot = 0;
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
        for (int ch = 0; ch < NCH; ++ch) {
          mbar_wait(&full[slot], (phbits >> slot) & 1u);
          const unsigned char* sl = ring + slot * L.slot_stride;
          if constexpr (MODE == MODE_POOL_FWD) {
            // GAP(x) of this chunk's channels (NFP_Pooling.py:27): one lane per channel plane; the job rotates
            // over the warps chunk by chunk.  (Measured alternative, not kept: row sums from the strips pass A
            // already holds in registers + a shuffle tree over the strips -- 11.4 vs 8.7 us, shuffles share the
            // shared-memory data path and the extra live values spill.)
            const int w0 = (ch * 2) % NW;
            for (int c = ((warp - w0 + NW) % NW) * 32 + lane; c < CC; c += NT) {
              const unsigned char* pl = sl + c * P * ESZ;
              float s = 0.f;
#pragma unroll 7
              for (int e = 0; e < P; ++e) s += ldx<T>(pl + e * ESZ);
              a.gap_x[(size_t)b * a.C + ch * CC + c] = s / (float)P;
            }
          }
          const unsigned char* pa = sl + warp * PSTRIDE + toff;
          for (int it = warp; it < npairs; it += NW, pa += NW * PSTRIDE) {
            if (lane_on && !NFP_DBG_SKIP_PASSA) {
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
          if (!resident) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[slot]);
          }
          phbits ^= 1u << slot;
          if (++slot == nst) slot = 0;
        }
      }
      if constexpr (NFP_DBG_SKIP_TAIL && !BWD) {
        consumer_sync<NT>();
        continue;
      }
      // sum over the channel slots of the warp (fixed shuffle tree: deterministic), then publish the warp's table
      constexpr bool DIRECT = Smem<T, C, MODE, NW>::DIRECT;
      const bool direct = DIRECT || (Smem<T, C, MODE, NW>::BDIRECT_OK && a.bdirect);
      if (direct) {
        if (lane_on) {
          float* wt = wtab + (warp * CPW + chslot) * PNV + pos * (TW * NV);
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) wt[j * NV + v] = accs[j][v];
        }
      }
      if (CPW > 1 && !direct) {
#pragma unroll
        for (int d = LANES / 2; d >= NS; d >>= 1)
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) accs[j][v] += __shfl_down_sync(0xffffffffu, accs[j][v], d);
      }
      constexpr int NWT = Smem<T, C, MODE, NW>::NWT;
      if (direct) {
      } else if constexpr (NWT == NW) {
        if (lane < NS) {
          float* wt = wtab + warp * PNV + pos * (TW * NV);
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) wt[j * NV + v] = accs[j][v];
        }
      } else {
        // two rounds over half the table space: the upper warps publish, the lower warps add their own on top
        // (each entry is touched by one lane of one warp per round: fixed order, deterministic)
        float* wt = wtab + (warp % NWT) * PNV + pos * (TW * NV);
        if (warp >= NWT && lane < NS) {
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) wt[j * NV + v] = accs[j][v];
        }
        consumer_sync<NT>();
        if (warp < NWT && lane < NS) {
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int v = 0; v < NV; ++v) wt[j * NV + v] += accs[j][v];
        }
      }
    }
    NFP_STAMP(1);  // pass A done (this warp)
    if (x_early) {
      if (img == 0) grid_dependency_wait();
      stencil_part();
    }
    consumer_sync<NT>();
    NFP_STAMP(5);  // every warp's partial tables are published
    if constexpr (!BWD) {
      if (img == 0) mbar_wait(tabfull, 0);  // stencil tables (fetched by the producer at kernel start)
    }
    for (int i = tid; i < PNV; i += NT) {
      const int ntab = (Smem<T, C, MODE, NW>::BDIRECT_OK && a.bdirect) ? NW * CPW : Smem<T, C, MODE, NW>::NTAB;
      float s = 0.f;
#pragma unroll 8
      for (int t = 0; t < ntab; ++t) s += wtab[t * PNV + i];  // fixed order: deterministic
      tfull[i] = s;
      if (i % NV == 0) {  // |x_p|^2: the clamped inverse norm (and, backward, the 1/(N |x|) of the norm term)
        const int p = i / NV;
        const float nrm = sqrtf(s), N = fmaxf(nrm, a.eps);
        inv[p] = 1.f / N;
        if constexpr (BWD) reinterpret_cast<float*>(smem_raw + L.rn)[p] = nrm > 0.f ? 1.f / (N * nrm) : 0.f;
      }
    }
    consumer_sync<NT>();
    NFP_STAMP(6);  // table summed, inverse norms ready

    // ---- forward value -----------------------------------------------------------------------------
    if constexpr (!BWD) {
      const int16_t* fv = reinterpret_cast<const int16_t*>(smem_raw + L.t_fv);
      const int16_t* fd = reinterpret_cast<const int16_t*>(smem_raw + L.t_fd);
      float* ytab = reinterpret_cast<float*>(smem_raw + L.ytab);
      for (int idx = tid; idx < (NFP_DBG_SKIP_EPI ? 0 : K * P); idx += NT) {
        const int p = idx % P;
        const int v = fv[idx];
        float yv = 0.f;
        if (v >= 0) yv = tfull[fd[idx]] * (inv[p] * inv[v]);
        if (!a.similarity) yv = 1.f - yv;
        if constexpr (POOLED) {
          ytab[idx] = yv;
        } else {
          // (multi-radius launch: kin planes of the inner radius in front; its taps are the inner taps of this window)
          const size_t yb = (size_t)b * (K + a.kin) * P;
          if (a.y_f32) reinterpret_cast<float*>(a.y)[yb + a.kin * P + idx] = yv;
          else reinterpret_cast<T*>(a.y)[yb + a.kin * P + idx] = from_f32<T>(yv);
          if constexpr (R >= 2) {
            if (a.kin) {
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
        // GAP over the plane of every tap (NFP_Pooling.py:31)
        consumer_sync<NT>();
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
        if constexpr (MODE == MODE_POOL_FWD) {
          if (a.proj_w) {
            // fused head (NFP_Pooling.py:31-35): out[c] = GAP(x)[c] * (proj_w[c] . GAP(NFP(x)) + proj_b[c])
            consumer_sync<NT>();   // tfull[0..K) and this CTA's gap_x stores are visible to the whole CTA
            for (int c = tid; c < a.C; c += NT) {
              const float4* wr4 = reinterpret_cast<const float4*>(a.proj_w + (size_t)c * K);
              float proj = a.proj_b ? a.proj_b[c] : 0.f;
#pragma unroll
              for (int n4 = 0; n4 < K / 4; ++n4) {
                const float4 w4 = wr4[n4];
                proj = fmaf(w4.x, tfull[4 * n4], proj); proj = fmaf(w4.y, tfull[4 * n4 + 1], proj);
                proj = fmaf(w4.z, tfull[4 * n4 + 2], proj); proj = fmaf(w4.w, tfull[4 * n4 + 3], proj);
              }
              a.head_out[(size_t)b * a.C + c] = a.gap_x[(size_t)b * a.C + c] * proj;
            }
          }
        }
      }
      NFP_STAMP(2);  // forward outputs written
      consumer_sync<NT>();  // tfull / inv / ytab / wtab are rewritten by the next image
      continue;
    } else {
      // ---- backward: stencil coefficients.  Wd currently holds S[p][o] (the gy-only part, computed
      // before pass A); scale by the inverse norms and close the centre tap:
      //   Wd[p][o]   = S[p][o] / (N_p N_q)
      //   Wd[p][ctr] = sw - (1/(N_p |x_p|)) * (sum_o Wd[p][o] dot(p, q_o) + sw |x_p|^2),  sw = 2 S[p][ctr] / N_p^2
      const int16_t* qt = reinterpret_cast<const int16_t*>(smem_raw + L.t_q);
      const float* rn = reinterpret_cast<const float*>(smem_raw + L.rn);
      float* Wd = reinterpret_cast<float*>(smem_raw + L.wd);
      // eight lanes per pixel share the window offsets; fixed shuffle tree -> deterministic
      for (int it = tid; it < align_up(P * 8, 32); it += NT) {
        const int p = it >> 3, g = it & 7;
        const bool valid = p < P;
        const float ip = valid ? inv[p] : 0.f;
        float s = 0.f;
        if (valid) {
#pragma unroll
          for (int t = 0; t < (K + 7) / 8; ++t) {
            const int n = g + 8 * t;          // neighbour number (window order, centre removed)
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
      consumer_sync<NT>();
      NFP_STAMP(2);  // coefficients ready
      // ---- pass B: gx = stencil(x), chunk by chunk ------------------------------------------------------
      {
        unsigned char* mystg = smem_raw + L.stg + warp * L.stg_warp;
        const int stg_half = L.stg_warp / 2;
        const float invP = 1.f / (float)P;
        unsigned char* gxb = reinterpret_cast<unsigned char*>(a.gx) + (size_t)b * a.C * P * ESZ;
        slot = 0;
        if (resident) phbits = phbits0;  // re-walk the slots pass A left in place
        const float* ggx = nullptr;
        if constexpr (MODE == MODE_POOL_BWD) {
          if (a.ggx_tma) mbar_wait(&gyfull[img & 1], (img >> 1) & 1);  // bulk copy issued by the producer
          ggx = reinterpret_cast<const float*>(smem_raw + L.ggx) + (img & 1) * a.C;
        }
        bool lanech_done = false;
        if constexpr (C::LANECH) {
          if (a.lanech) {
            // ---- lane-per-channel form: a warp owns a task of 64 channels of the chunk, lane = 2 channels (packed
            // fp32 pair), and slides a k-row window down ITS planes: every x element is read from shared memory once
            // (the strip form reads it k times), the map row's coefficients arrive as broadcast LDS.128, the
            // results overwrite the plane in place (a plane is private to its lane) and one TMA bulk store per task
            // writes them back.  Shared-memory wavefronts per image 5152 -> 4024, instructions per channel 31 -> 12.
            lanech_done = true;
            const int ntask = CC / C::TASK;
            const float4* wd4 = reinterpret_cast<const float4*>(Wd);
            for (int ch = 0; ch < NCH; ++ch) {
              mbar_wait(&full[slot], (phbits >> slot) & 1u);
              unsigned char* sl = ring + slot * L.slot_stride;
              bool stored = false;
              for (int t = 0; t < ntask; ++t) {
                if ((ch * ntask + t) % NW != warp) continue;
                unsigned char* p0 = sl + (size_t)(t * C::TASK + lane) * P * ESZ;
                unsigned char* p1 = p0 + 32 * P * ESZ;
                float g0 = 0.f, g1 = 0.f;
                if constexpr (MODE == MODE_POOL_BWD) {
                  g0 = ggx[ch * CC + t * C::TASK + lane] * invP;
                  g1 = ggx[ch * CC + t * C::TASK + 32 + lane] * invP;
                }
                const uint64_t gpair = pack2(g0, g1);
                // rows rr-R .. rr+R of the two planes, rotating: map row q lives in win[q mod k]; rows outside the
                // map are zero
                uint64_t win[k][W];
#pragma unroll
                for (int q = 0; q < k; ++q)
#pragma unroll
                  for (int j = 0; j < W; ++j)
                    win[q][j] = (q < R && q < C::H) ? pack2(ldx<T>(p0 + (q * W + j) * ESZ), ldx<T>(p1 + (q * W + j) * ESZ))
                                                    : 0ull;
#pragma unroll
                for (int rr = 0; rr < C::H; ++rr) {
#pragma unroll
                  for (int j = 0; j < W; ++j)
                    win[(rr + R) % k][j] = (rr + R < C::H) ? pack2(ldx<T>(p0 + ((rr + R) * W + j) * ESZ),
                                                                   ldx<T>(p1 + ((rr + R) * W + j) * ESZ))
                                                           : 0ull;
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
                        if (j + dx >= 0 && j + dx < W && rr + dy >= 0 && rr + dy < C::H)
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
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                  bulk_s2g(gxb + ((size_t)ch * CC + (size_t)t * C::TASK) * P * ESZ, sl + (size_t)t * C::TASK * P * ESZ,
                           (uint32_t)(C::TASK * P * ESZ));
                  bulk_commit();
                }
                stored = true;
              }
              if (stored && lane == 0) bulk_wait_read<0>();  // the slot goes back to the producer: the store has read it
              __syncwarp();
              if (lane == 0) mbar_arrive(&empty[slot]);
              phbits ^= 1u << slot;
              if (++slot == nst) slot = 0;
            }
            NFP_STAMP(3);  // pass B done (this warp)
          }
        }
        if (!lanech_done) {
        int nstore = 0;
        const float* wdp = Wd + C::widx(r * W + c0, 0);
        float wr[(R == 1) ? TW : 1][(R == 1) ? KK : 1];
        if constexpr (R == 1) {
#pragma unroll
          for (int j = 0; j < TW; ++j)
#pragma unroll
            for (int o = 0; o < KK; ++o) wr[j][o] = wdp[j * KK + o];
        }
        for (int ch = 0; ch < NCH; ++ch) {
          mbar_wait(&full[slot], (phbits >> slot) & 1u);
          const unsigned char* sl = ring + slot * L.slot_stride;
          const unsigned char* pa = sl + warp * PSTRIDE + toff;
          for (int it = warp; it < npairs; it += NW, pa += NW * PSTRIDE) {
            unsigned char* sb = mystg + (nstore & 1) * stg_half;
            if (nstore >= 2) {
              if (lane == 0) bulk_wait_read<1>();  // the store that last used this buffer has read it
              __syncwarp();
            }
            if (lane_on) {
              if constexpr (R == 1) {
#if NFP_PASSB_FFMA2
                // 3x3: all k*k coefficients of the strip live in registers.  The two channel groups of the pair
                // share them, so the FMAs run on packed fp32 pairs (lo = group 0, hi = group 1): ptxas folds the
                // duplicated coefficient into FFMA2's scalar-broadcast operand form (`FFMA2 Rd, Rw.F32, Rx.F32x2,
                // Rd.F32x2`), i.e. one issue slot per two FMAs and no extra registers for the coefficients.
                float g0 = 0.f, g1 = 0.f;
                if constexpr (MODE == MODE_POOL_BWD) {
                  const float* gp = ggx + ch * CC + 2 * it * CPW + chslot;
                  g0 = gp[0] * invP;
                  g1 = gp[CPW] * invP;
                }
                uint64_t out[TW];
#pragma unroll
                for (int j = 0; j < TW; ++j) out[j] = pack2(g0, g1);
#pragma unroll
                for (int dy = -R; dy <= R; ++dy) {
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
                        const float w = wr[j][(dy + R) * k + dx + R];
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
#else
                // 3x3: all k*k coefficients of the strip live in registers
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  const unsigned char* ph_ = pa + h * GSTRIDE;
                  float out[TW];
                  float g0 = 0.f;
                  if constexpr (MODE == MODE_POOL_BWD)
                    g0 = ggx[ch * CC + (2 * it + h) * CPW + chslot] * invP;
#pragma unroll
                  for (int j = 0; j < TW; ++j) out[j] = g0;
#pragma unroll
                  for (int dy = -R; dy <= R; ++dy) {
                    float xr[XW];
#pragma unroll
                    for (int jj = 0; jj < XW; ++jj) xr[jj] = ldx<T>(ph_ + NFP_OFF(dy, jj));
                    // dx outer, j inner: consecutive FMAs go to different accumulators (no 4-cycle chains)
#pragma unroll
                    for (int dx = -R; dx <= R; ++dx)
#pragma unroll
                      for (int j = 0; j < TW; ++j) {
                        if (j + dx + XOFF >= 0 && j + dx + XOFF < XW)
                          out[j] = fmaf(wr[j][(dy + R) * k + dx + R], xr[j + dx + XOFF], out[j]);
                      }
                  }
#pragma unroll
                  for (int j = 0; j < TW; ++j) stx<T>(sb + h * GSTRIDE + toff + j * ESZ, out[j]);
                }
#endif
              } else {
#if NFP_PASSB_FFMA2
                // wider windows: the coefficients of ONE window row at a time (register budget), each row
                // loaded once and applied to both channel groups of the pair as packed fp32 pairs (FFMA2 with
                // the coefficient as scalar-broadcast operand, see the 3x3 branch)
                float g0 = 0.f, g1 = 0.f;
                if constexpr (MODE == MODE_POOL_BWD) {
                  const float* gp = ggx + ch * CC + 2 * it * CPW + chslot;
                  g0 = gp[0] * invP;
                  g1 = gp[CPW] * invP;
                }
                uint64_t out[TW];
#pragma unroll
                for (int j = 0; j < TW; ++j) out[j] = pack2(g0, g1);
#pragma unroll
                for (int dy = -R; dy <= R; ++dy) {
                  float wrow[TW][k];
#pragma unroll
                  for (int j = 0; j < TW; ++j)
#pragma unroll
                    for (int dx = 0; dx < k; ++dx) wrow[j][dx] = wdp[j * KK + (dy + R) * k + dx];
                  uint64_t xr[XW];
#pragma unroll
                  for (int jj = 0; jj < XW; ++jj)
                    xr[jj] = pack2(ldx<T>(pa + NFP_OFF(dy, jj)), ldx<T>(pa + GSTRIDE + NFP_OFF(dy, jj)));
#pragma unroll
                  for (int dx = -R; dx <= R; ++dx)
#pragma unroll
                    for (int j = 0; j < TW; ++j) {
                      if (j + dx + XOFF >= 0 && j + dx + XOFF < XW) {
                        const float w = wrow[j][dx + R];
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
#else
                // wider windows: the coefficients of ONE window row at a time (register budget), each row
                // loaded once and applied to both channel groups of the pair
                float out[2][TW];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  float g0 = 0.f;
                  if constexpr (MODE == MODE_POOL_BWD)
                    g0 = ggx[ch * CC + (2 * it + h) * CPW + chslot] * invP;
#pragma unroll
                  for (int j = 0; j < TW; ++j) out[h][j] = g0;
                }
#pragma unroll
                for (int dy = -R; dy <= R; ++dy) {
                  float wrow[TW][k];
#pragma unroll
                  for (int j = 0; j < TW; ++j)
#pragma unroll
                    for (int dx = 0; dx < k; ++dx) wrow[j][dx] = wdp[j * KK + (dy + R) * k + dx];
#pragma unroll
                  for (int h = 0; h < 2; ++h) {
                    float xr[XW];
#pragma unroll
                    for (int jj = 0; jj < XW; ++jj) xr[jj] = ldx<T>(pa + h * GSTRIDE + NFP_OFF(dy, jj));
#pragma unroll
                    for (int dx = -R; dx <= R; ++dx)
#pragma unroll
                      for (int j = 0; j < TW; ++j) {
                        if (j + dx + XOFF >= 0 && j + dx + XOFF < XW)
                          out[h][j] = fmaf(wrow[j][dx + R], xr[j + dx + XOFF], out[h][j]);
                      }
                  }
                }
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                  for (int j = 0; j < TW; ++j) stx<T>(sb + h * GSTRIDE + toff + j * ESZ, out[h][j]);
#endif
              }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
              // the pair's 2*CPW planes are contiguous in gx
              bulk_s2g(gxb + ((size_t)ch * CC + (size_t)2 * it * CPW) * P * ESZ, sb, (uint32_t)PSTRIDE);
              bulk_commit();
            }
            ++nstore;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[slot]);
          phbits ^= 1u << slot;
          if (++slot == nst) slot = 0;
        }
        NFP_STAMP(3);  // pass B done (this warp)
        if (lane == 0) bulk_wait_read<0>();  // staging is part of the union the next image overwrites
        }
      }
      consumer_sync<NT>();
      if constexpr (MODE == MODE_POOL_BWD) {
        // every warp is past its last read of this image's g_gap_x
        if (tid == 0 && a.ggx_tma) mbar_arrive(&gyempty[img & 1]);
      }
    }
  }
  // shared memory must outlive the bulk stores' READS only; their global writes are complete (and visible to the
  // next grid) when this grid completes
  if (BWD && lane == 0) bulk_wait_read<0>();
  img = 0;
  NFP_STAMP(4);  // stores drained
#undef NFP_OFF
}

// ---- host side --------------------------------------------------------------------------------------

struct Plan {
  bool ok;
  int CC, NCH, nst, resident, ctas_per_sm, lanech, gy_bufs, bdirect;
  size_t smem;
};

template <typename T, class C, int MODE>
Plan plan_for(const KParams& P, int num_sms = 148) {
  Plan pl{false, 0, 0, 0, 0, 0, 0, 2, 0, 0};
  constexpr int esz = (int)sizeof(T);
  constexpr bool bwd = (MODE == MODE_BWD || MODE == MODE_POOL_BWD);
  constexpr int target_bytes = 16 * 1024;  // chunk size
  constexpr int pair = 2 * C::CPW;  // work item: a pair of channel groups
  if (((size_t)pair * C::P * esz) % 16) return pl;   // TMA bulk store / load granularity
  if (((size_t)C::K * C::P * esz) % 16) return pl;
  if (P.Kin && (C::R < 2 || ((size_t)P.Kin * C::P * esz) % 16)) return pl;  // multi-radius: the blocks of gy are bulk-copied
  if (P.C % pair) return pl;
  // backward of the full-row-strip 3x3 shapes: lane-per-channel pass B when C is a whole number of 64-channel tasks
  pl.lanech = (bwd && C::LANECH && P.C % C::TASK == 0) ? 1 : 0;
  // chunk: the largest CC <= target that divides C and is a whole number of group pairs (of tasks)
  const int step = pl.lanech ? C::TASK : pair;
  int best = 0;
  for (int cc = step; cc <= P.C; cc += step) {
    if (P.C % cc) continue;
    if ((size_t)cc * C::P * esz > (size_t)target_bytes && best) break;
    best = cc;
    if ((size_t)cc * C::P * esz >= (size_t)target_bytes) break;
  }
  if (!best) return pl;
  pl.CC = best;
  pl.NCH = P.C / best;
  for (int ctas = C::MINB; ctas >= 1 && !pl.ok; --ctas) {
    // one image per CTA (the whole batch fits the resident CTAs): a single upstream-gradient buffer suffices
    const int gy_bufs = (bwd && P.B <= num_sms * ctas) ? 1 : 2;
    const int budget = (kSmemPerSM + 1024) / ctas - 1024 - 256;  // 228 KB per SM, 1 KB reserved per CTA; 256 B slack
    int first = 5;  // measured: 4-5 stages beat 6-8 at B = 256
    // one image per CTA, lane-per-channel pass B: per-lane partial tables (no shuffle tree, one publish round) with the
    // image streamed twice, instead of the resident image with the two-round publish
    if (Smem<T, C, MODE, kNW>::BDIRECT_OK && pl.lanech && gy_bufs == 1) {
      for (int nst = first; nst >= 3 && !pl.ok; --nst) {
        Smem<T, C, MODE, kNW> L(pl.CC, nst, P.C, P.Kin, pl.lanech, gy_bufs, 1);
        if (L.total > budget) continue;
        pl.gy_bufs = gy_bufs;
        pl.bdirect = 1;
        pl.nst = nst;
        pl.smem = (size_t)L.total;
        pl.ctas_per_sm = ctas;
        pl.ok = true;
      }
      if (pl.ok) break;
    }
    // backward with the lane-per-channel pass B: if the WHOLE image fits (512x7x7 fp32: 8 slots, 98 KB), keep it -- a
    // warp owns a whole chunk in pass B, so with fewer slots than chunks the last warps wait for a slot to drain and
    // for its refill (an L2 round trip) before they can start
    if (pl.lanech && pl.NCH <= kMaxStages && pl.NCH > first) {
      Smem<T, C, MODE, kNW> L(pl.CC, pl.NCH, P.C, P.Kin, pl.lanech, gy_bufs);
      if (L.total <= budget) first = pl.NCH;
    }
    for (int nst = first; nst >= 2; --nst) {  // as many stages as fit
      Smem<T, C, MODE, kNW> L(pl.CC, nst, P.C, P.Kin, pl.lanech, gy_bufs);
      if (L.total > budget) continue;
      pl.gy_bufs = gy_bufs;
      pl.nst = nst;
      pl.smem = (size_t)L.total;
      pl.ctas_per_sm = ctas;
      pl.ok = true;
      break;
    }
  }
  if (!pl.ok) return pl;
  pl.resident = (bwd && pl.NCH <= pl.nst) ? 1 : 0;
  return pl;
}

template <typename T, class C, int MODE>
int launch_mode(const KParams& P, StreamArgs a, cudaStream_t stream) {
  constexpr int kMaxDev = 64;
  static int sm_count[kMaxDev] = {0};
  static int l2_bytes[kMaxDev] = {0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < 0 || dev >= kMaxDev) return NFPB200_EDEVICE;
  auto kern = stream_kernel<T, C, MODE, kNW>;
  // per-device one-time setup (function attributes are per device; a process may drive several GPUs).
  // Idempotent, so a race between two host threads doing it at once is harmless.
  if (sm_count[dev] == 0) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemPerSM);
    if (e != cudaSuccess) return (int)e;
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return (int)e;
    int l2 = 0;
    e = cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
    if (e != cudaSuccess) return (int)e;
    l2_bytes[dev] = l2;
    sm_count[dev] = n;
  }
  const int num_sms = sm_count[dev];
  const Plan pl = plan_for<T, C, MODE>(P, num_sms);
  if (!pl.ok) return NFPB200_EUNSUPPORTED;
  a.gy_bufs = pl.gy_bufs;
  a.bdirect = pl.bdirect;
  a.CC = pl.CC;
  a.NCH = pl.NCH;
  a.nst = pl.nst;
  a.resident = pl.resident;
  a.lanech = pl.lanech;
  const Tables<C>* gt = tables_for<C>(a.pad_mode);
  if (!gt) return NFPB200_EINVAL;
  const int slots = num_sms * pl.ctas_per_sm;
  const int grid = P.B < slots ? P.B : slots;
  // L2 prefetch before the dependency wait (stream_kernel's consumer prologue): at most the leading images of every
  // CTA whose inputs fit in half the L2 over the whole grid -- all of them at B = 256 on 512x7x7 -- so that a large
  // batch does not flush the working set of the launch it overlaps
  size_t pf_bytes = (size_t)P.C * C::P * sizeof(T);
  if (MODE == MODE_BWD) pf_bytes += (size_t)(C::K + P.Kin) * C::P * sizeof(T);
  if (MODE == MODE_POOL_BWD && a.g_gap_x) pf_bytes += (size_t)P.C * 4;
  const size_t pf_fit = (size_t)l2_bytes[dev] / 2 / ((size_t)grid * pf_bytes);
  const int per_cta = (P.B + grid - 1) / grid;
  a.pf_imgs = pf_fit < (size_t)per_cta ? (int)pf_fit : per_cta;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(block_threads(MODE, kNW));
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t lrc = cudaLaunchKernelEx(&cfg, kern, a, gt);
  if (lrc != cudaSuccess && getenv("NFPB200_VERBOSE")) {
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, kern);
    fprintf(stderr, "[nfpb200] launch failed (%d): grid %d block %d dyn smem %zu static %zu regs %d maxThreads %d\n",
            (int)lrc, grid, block_threads(MODE, kNW), pl.smem, fa.sharedSizeBytes, fa.numRegs, fa.maxThreadsPerBlock);
  }
  return (int)lrc;
}

template <typename T, class C>
int launch_cfg(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream) {
  switch (mode) {
    case MODE_FWD: return launch_mode<T, C, MODE_FWD>(P, a, stream);
    case MODE_BWD: return launch_mode<T, C, MODE_BWD>(P, a, stream);
    case MODE_POOL_FWD: return launch_mode<T, C, MODE_POOL_FWD>(P, a, stream);
    default: return launch_mode<T, C, MODE_POOL_BWD>(P, a, stream);
  }
}
template <typename T, class C>
bool plan_ok_cfg(const KParams& P, int mode) {
  switch (mode) {
    case MODE_FWD: return plan_for<T, C, MODE_FWD>(P).ok;
    case MODE_BWD: return plan_for<T, C, MODE_BWD>(P).ok;
    case MODE_POOL_FWD: return plan_for<T, C, MODE_POOL_FWD>(P).ok;
    default: return plan_for<T, C, MODE_POOL_BWD>(P).ok;
  }
}

template <typename T>
int launch_dtype(const KParams& P, int mode, const StreamArgs& a, cudaStream_t stream) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return launch_cfg<T, Cfg<H_, W_, R_, TW_>>(P, mode, a, stream);
  NFP_STREAM_SHAPES(X)
#undef X
  return NFPB200_EUNSUPPORTED;
}
template <typename T>
bool plan_ok_dtype(const KParams& P, int mode) {
#define X(H_, W_, R_, TW_) \
  if (P.H == H_ && P.W == W_ && P.R == R_) return plan_ok_cfg<T, Cfg<H_, W_, R_, TW_>>(P, mode);
  NFP_STREAM_SHAPES(X)
#undef X
  return false;
}

}  // namespace stream
}  // namespace nfp
