/*
 * nfp_b200.h -- C ABI of the B200-native Neighbourhood Feature Pooling operator.
 *
 * This is the drop-in boundary for the NFP hot path.  The reference has no
 * FFI layer of its own (it is pure PyTorch); the entry points below replace,
 * one for one, the Python-level operator surface a binding would wrap:
 *
 *   nfpb200_forward        <- NFPPooling.forward            (models/pooling/nfp.py:132-134)
 *                             and the measure it dispatches to (nfp.py:141-374)
 *   nfpb200_backward       <- autograd through that forward (the reference stores the
 *                             (B, C*(k*k-1), H', W') neighbour tensor; we recompute)
 *   nfpb200_pool_forward   <- nfp_pooling.forward up to the projection: GAP(x) and
 *                             GAP(NFP(x))                   (models/NFP_Pooling.py:27-31)
 *   nfpb200_pool_backward  <- autograd through those two lines
 *   nfpb200_pooled_map_forward  <- adaptive_avg_pool2d(NFPPooling(x), (1, 1)).view(B, -1): every stage of
 *                             MobileNetV3_MultiStageNFP   (models/texture_pooling.py:249-256)
 *   nfpb200_pooled_map_backward <- autograd through those lines
 *   nfpb200_output_shape   <- Conv2d output-size rule behind NFPPooling.output_size
 *                                                           (nfp.py:125-130, 42-47)
 *   nfpb200_desc_t         <- the constructor arguments     (nfp.py:16-18); inner_R: the two NFP layers of
 *                             MultiRadiusNFPHead evaluated together (models/nfp_heads.py:86-93,111-112)
 *
 * Conventions
 *   - plain C types only; every buffer is caller-owned DEVICE memory (NCHW
 *     contiguous unless desc->layout says otherwise), the library keeps no
 *     pointer after a call returns and never allocates on the hot path;
 *   - alignment, checked before any CUDA call (NFPB200_EALIGN below it):
 *       16 bytes: x, y, gy, gx, proj_w and a non-null workspace (bulk copies
 *                 and 16-byte vector accesses);
 *        4 bytes: the fp32 vectors gap_x, gap_nfp, g_gap_x, g_gap_nfp, out,
 *                 g_out and proj_b (read and written one float at a time);
 *     nothing else is assumed: no buffer needs more than its own size;
 *   - the library reads only the bytes its inputs span and writes only the
 *     bytes its outputs span, never an input, and never an element of the
 *     workspace beyond nfpb200_workspace_bytes; the workspace's contents on
 *     entry do not affect any result;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 on success, a negative NFPB200_E* code for argument
 *     errors, a positive cudaError_t for CUDA failures.  No C++ exception
 *     crosses the boundary.  nfpb200_status_string() renders either.
 *   - re-entrant and thread-safe: no global mutable state besides one-time
 *     cudaFuncSetAttribute calls, the (atomic) diagnostics pointer of
 *     nfpb200_debug_phase_timing, and the NFPB200_* tuning environment variables
 *     (INTEGRATION.md section 5), which are read ONCE, at the first launch that
 *     consults them, and never change behaviour afterwards.
 *   - sm_100a only.  There is no CPU path in this library.
 */
#ifndef NFP_B200_H_
#define NFP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFPB200_ABI_VERSION 5

/* element type of x / y / gy / gx.  Accumulation is always fp32; every GAP and head vector is fp32 whatever the dtype.
 * NFPB200_F16 (IEEE half, ABI v5) is served by two kernel families only: the NCHW streaming-ring kernels ("fused/stream_*")
 * and the channels-last token kernels ("fused/token_*"), for every op they carry (map, pooled, fused head, inner_R,
 * pooled map), on exactly the problems a bf16 descriptor sends to them.  Any other fp16 problem -- what bf16 sends to the
 * planar, generic or cluster-split kernels, and NFPB200_PATH_GENERIC -- returns NFPB200_EUNSUPPORTED: the caller widens
 * to fp32.  fp16 results are rounded to nearest: a gradient beyond 65504 is +-inf, as a narrowing copy makes it. */
enum { NFPB200_F32 = 0, NFPB200_BF16 = 1, NFPB200_F16 = 2 };

/* torch.nn.Conv2d padding_mode (nfp.py:17, default 'reflect') */
enum { NFPB200_PAD_ZEROS = 0, NFPB200_PAD_REFLECT = 1, NFPB200_PAD_REPLICATE = 2, NFPB200_PAD_CIRCULAR = 3 };

/* the measures NFPPooling.__init__ accepts (nfp.py:85-118), lower-cased */
enum {
  NFPB200_NORM = 0,        /* nfp.py:141-148 */
  NFPB200_COSINE = 1,      /* nfp.py:150-159  -- the only measure on the live model paths */
  NFPB200_DOT = 2,         /* nfp.py:161-170 */
  NFPB200_RMSE = 3,        /* nfp.py:172-179 */
  NFPB200_GEMAN = 4,       /* nfp.py:181-193 */
  NFPB200_ATTENTION = 5,   /* nfp.py:195-205 */
  NFPB200_EMD = 6,         /* nfp.py:207-216 */
  NFPB200_CANBERRA = 7,    /* nfp.py:218-227 */
  NFPB200_HELLINGER = 8,   /* nfp.py:229-241 */
  NFPB200_CHISQUARED1 = 9, /* nfp.py:243-252 */
  NFPB200_CHISQUARED2 = 10,/* nfp.py:254-263 */
  NFPB200_GFC = 11,        /* nfp.py:265-276 */
  NFPB200_PEARSON = 12,    /* nfp.py:278-293 */
  NFPB200_JEFFREY = 13,    /* nfp.py:295-308 */
  NFPB200_SQUAREDCHORD = 14,/* nfp.py:310-324 */
  NFPB200_SMITH = 15,      /* nfp.py:326-342 */
  NFPB200_SCS = 16,        /* nfp.py:344-374 ('scs' / 'sharpened_cosine'), batch-coupled as in the reference */
  NFPB200_NUM_MEASURES = 17
};

/* memory layout of x and gx.  y / gy are always (B, K, H', W') contiguous, the layout the reference returns. */
enum {
  NFPB200_LAYOUT_NCHW = 0,  /* (B, C, H, W) contiguous */
  NFPB200_LAYOUT_NHWC = 1   /* x[b][h][w][c]: channels of a pixel contiguous, pixels dense, batch stride free.  This is a
                               torch channels_last map and the ViT head's token view (models/texture_pooling.py:181-188:
                               feats[:, 1:].transpose(1, 2).reshape(B, C, H, W), strides (197*C, 1, W*C, C)); served by
                               the tensor-core "fused/token" kernels (bf16 / fp16, cosine, pad = R, stride 1) -- anything else
                               returns NFPB200_EUNSUPPORTED and the caller repacks to NCHW */
};

/* which implementation to use */
enum {
  NFPB200_PATH_AUTO = 0,    /* fused kernels when the problem qualifies, else the planar, else the generic kernels */
  NFPB200_PATH_GENERIC = 1, /* force the geometry-/measure-generic kernels */
  NFPB200_PATH_FUSED = 2,   /* force the fused kernels; NFPB200_EUNSUPPORTED when the problem does not qualify */
  NFPB200_PATH_SPLIT = 3    /* the cluster-split fused kernels (one thread-block cluster per image, DSMEM table exchange):
                               a measured experiment kept selectable for A/B runs and tests; same results, slower at B = 256.
                               NFPB200_EUNSUPPORTED when the problem does not qualify */
};

/* Optional hint, OR-ed into nfpb200_desc_t.path, for nfpb200_backward / nfpb200_pool_backward: `x` was NOT written by
 * the launch that immediately precedes this call on the stream (it is a saved forward activation, as under autograd).
 * The fused backward kernels are launched with programmatic dependent launch; with the hint they start streaming x
 * while the preceding kernel is still draining and only wait for it before touching the upstream gradient and gx.
 * Every fused kernel releases its dependents only after its own dependency wait has returned, so the early reads can
 * overlap nothing older than the immediately preceding launch: x may be the output of any EARLIER launch (stacked NFP
 * layers, recomputation under activation checkpointing).  Do not set it when x is written by the immediately
 * preceding launch itself. */
#define NFPB200_HINT_X_STABLE 0x100

/* Optional flag, OR-ed into nfpb200_desc_t.path, for nfpb200_forward with dtype = NFPB200_BF16 or NFPB200_F16: y is
 * written as fp32 (what the reference produces under torch.autocast on CUDA, where F.cosine_similarity runs in fp32 on
 * the bf16 / fp16 neighbours, nfp.py:152-156).  Honoured by the fused kernels; other paths return NFPB200_EUNSUPPORTED. */
#define NFPB200_FLAG_Y_F32 0x200

/* operations, for nfpb200_workspace_bytes / nfpb200_describe_path / nfpb200_launch_count */
enum {
  NFPB200_OP_FORWARD = 0,
  NFPB200_OP_BACKWARD = 1,
  NFPB200_OP_POOL_FORWARD = 2,
  NFPB200_OP_POOL_BACKWARD = 3,
  NFPB200_OP_POOLED_MAP_FORWARD = 4,  /* ABI v4 */
  NFPB200_OP_POOLED_MAP_BACKWARD = 5  /* ABI v4 */
};

/* error codes (negative); positive return values are cudaError_t */
enum {
  NFPB200_OK = 0,
  NFPB200_EINVAL = -1,       /* null pointer / non-positive size / unknown enum */
  NFPB200_EPADDING = -2,     /* reflect padding >= input dim, or circular padding > input dim (ATen's check) */
  NFPB200_ESHAPE = -3,       /* kernel window larger than the padded input */
  NFPB200_EWORKSPACE = -4,   /* workspace too small / null */
  NFPB200_EUNSUPPORTED = -5, /* e.g. NFPB200_PATH_FUSED on a problem the fused kernels do not cover */
  NFPB200_EDEVICE = -6,      /* the current device is not sm_100 */
  NFPB200_EALIGN = -7        /* a pointer below its alignment (Conventions above), or a batch stride not a multiple of 8 */
};

/* Constructor arguments of NFPPooling (nfp.py:16-18) plus the tensor shape. */
typedef struct nfpb200_desc {
  int32_t struct_bytes;     /* = sizeof(nfpb200_desc_t); ABI guard */
  int32_t dtype;            /* NFPB200_F32 | NFPB200_BF16 | NFPB200_F16 */
  int32_t B, C, H, W;       /* x is (B, C, H, W) contiguous */
  int32_t R;                /* radius; kernel_size = 2R+1, out_channels K = (2R+1)^2 - 1 (nfp.py:38-39) */
  int32_t stride;
  int32_t padding;
  int32_t dilation;
  int32_t padding_mode;     /* NFPB200_PAD_* */
  int32_t measure;          /* NFPB200_<MEASURE> */
  int32_t similarity;       /* bool (nfp.py:29) */
  int32_t difference_taps;  /* bool: neighbour taps emit centre - neighbour (nfp.py:74-76); only read by NORM / RMSE */
  float eps;                /* nfp.py:33 */
  float p;                  /* nfp.py:30: ord of NORM (INFINITY allowed), exponent of SCS */
  float q_scs;              /* nfp.py:34 */
  int32_t path;             /* NFPB200_PATH_* [| NFPB200_HINT_X_STABLE] [| NFPB200_FLAG_Y_F32] */
  int32_t layout;           /* NFPB200_LAYOUT_*; 0 = NCHW */
  int32_t inner_R;          /* multi-radius maps in one launch (models/nfp_heads.py:80-118, MultiRadiusNFPHead with
                               R_list = (1, 2)): 0 = off; r in [1, R) = y / gy carry K_r + K channels per image, the map
                               of radius r (padding r, K_r = (2r+1)^2 - 1 taps) FIRST, then the map of radius R -- the
                               layout of torch.cat([NFP_r(x), NFP_R(x)], dim=1).  With padding = R (and r) the window of
                               radius r is the inner part of the window of radius R under reflect / replicate / zero
                               padding alike, so both maps come out of ONE pass over x, and the backward folds both
                               gradient blocks into one stencil.  nfpb200_forward / nfpb200_backward on the fused
                               (NCHW ring, channels-last token) kernels and, for other map sizes with 16-byte aligned
                               planes, the planar row-band kernels; anything else: NFPB200_EUNSUPPORTED, and the caller
                               issues one launch per radius */
  int64_t x_batch_stride;   /* NHWC only: elements between consecutive images of x; 0 = dense (H*W*C); multiple of 8 */
  int64_t gx_batch_stride;  /* NHWC only: the same for gx.  Above the dense stride, nothing is written between images:
                               the elements from H*W*C to gx_batch_stride of each image keep their contents */
} nfpb200_desc_t;

int nfpb200_abi_version(void);

/* Human-readable text for a status returned by any entry point (static storage). */
const char* nfpb200_status_string(int status);

/* Diagnostics: when `device_stamps` is non-null, every fused-kernel CTA records 8 x uint64 nanosecond
 * timestamps (%globaltimer) of its phase boundaries for its first image at device_stamps[8 * blockIdx.x + k]
 * (k = 0 consumers ready, 1 pass A done, 2 forward written / coefficients ready, 3 pass B done, 4 stores
 * drained; the cluster-split and token kernels stamp two work items per CTA: 16 entries per CTA).  The buffer must hold
 * 16 * (number of CTAs) entries; pass NULL to switch it off.  Diagnostics only: the pointer is process-wide (atomic). */
int nfpb200_debug_phase_timing(unsigned long long* device_stamps);

/* (H', W') = Conv2d output size for the descriptor's geometry; validates the descriptor. */
int nfpb200_output_shape(const nfpb200_desc_t* desc, int32_t* Ho, int32_t* Wo);

/* Device scratch the given op needs (0 for the fused kernels' map and pool ops; per-pixel tables for the planar kernels,
 * pair coefficients for the generic ones; for the pooled-map ops see nfpb200_pooled_map_forward).  The caller allocates
 * it and passes it in. */
int nfpb200_workspace_bytes(const nfpb200_desc_t* desc, int32_t op, size_t* bytes);

/* Writes the name of the kernel path the op would take ("fused/...", "planar/..." or "generic/...") into buf. */
int nfpb200_describe_path(const nfpb200_desc_t* desc, int32_t op, char* buf, size_t buf_bytes);

/* Number of kernel launches the op issues on `stream` (bench.py's gpu_launches), counting a cudaMemsetAsync as one. */
int nfpb200_launch_count(const nfpb200_desc_t* desc, int32_t op, int32_t* launches);

/* y (B, K, H', W') = NFP(x)   (desc->inner_R = r > 0: (B, K_r + K, H, W), see nfpb200_desc_t).
 * Alignment: x, y, workspace 16 bytes. */
int nfpb200_forward(const nfpb200_desc_t* desc, const void* x, void* y,
                    void* workspace, size_t workspace_bytes, void* stream);

/* gx (B, C, H, W) = d<gy, NFP(x)>/dx ; similarities are recomputed from x, nothing is saved by forward.
 * (desc->inner_R = r > 0: gy is (B, K_r + K, H, W) and gx the sum of both layers' input gradients.)
 * Alignment: x, gy, gx, workspace 16 bytes. */
int nfpb200_backward(const nfpb200_desc_t* desc, const void* x, const void* gy, void* gx,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Fused head of nfp_pooling (NFP_Pooling.py:27-31): gap_x (B, C) = mean_hw x, gap_nfp (B, K) = mean_hw NFP(x).
 * Both outputs are fp32 regardless of desc->dtype.  Alignment: x, workspace 16 bytes; gap_x, gap_nfp 4 bytes. */
int nfpb200_pool_forward(const nfpb200_desc_t* desc, const void* x, float* gap_x, float* gap_nfp,
                         void* workspace, size_t workspace_bytes, void* stream);

/* gx = d(<g_gap_x, GAP(x)> + <g_gap_nfp, GAP(NFP(x))>)/dx ; g_* are fp32 (B, C) and (B, K).
 * Alignment: x, gx, workspace 16 bytes; g_gap_x, g_gap_nfp 4 bytes. */
int nfpb200_pool_backward(const nfpb200_desc_t* desc, const void* x, const float* g_gap_x,
                          const float* g_gap_nfp, void* gx,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- pooled similarity map (ABI v4) ----------------------------------------------------------------------------
 * The reference's multi-stage head pools every NFP map right away (models/texture_pooling.py:249-256:
 * adaptive_avg_pool2d(nfp(x), (1, 1)).view(B, -1)); these entry points compute only that, without writing the map:
 *   gap_nfp (B, K) fp32 = mean over the H' x W' output pixels of NFP(x), whatever desc->dtype.
 * desc->inner_R != 0 returns NFPB200_EUNSUPPORTED.  What each problem takes (nfpb200_describe_path names it):
 *   - NHWC bf16 / fp16 covered by the token kernels: their pooled mode ("fused/token_*"); GAP(x) goes to the workspace;
 *   - NCHW covered by the ring kernels: their pooled mode ("fused/stream_*"); GAP(x) goes to the workspace;
 *   - NCHW cosine, stride 1, dilation 1, padding = R <= 2, not circular, whose map mode takes "planar/band": the row-band
 *     kernels' pooled mode ("planar/band").  Forward: 2 launches (per-band partial sums (B, n_bands, K) fp32 in the
 *     workspace, then a kernel that sums them in band order and divides by H' W'); backward: 1 launch, no workspace;
 *   - anything else, and NFPB200_PATH_GENERIC: the generic kernels' pooled mode ("generic/pairs") without its GAP(x) part.
 * NFPB200_PATH_FUSED: the ring / token kernels or NFPB200_EUNSUPPORTED.  No float atomics on any path: results are
 * bit-identical from run to run.  Alignment: x, workspace 16 bytes; gap_nfp 4 bytes. */
int nfpb200_pooled_map_forward(const nfpb200_desc_t* desc, const void* x, float* gap_nfp,
                               void* workspace, size_t workspace_bytes, void* stream);

/* gx = d<g_gap_nfp, GAP(NFP(x))>/dx ; g_gap_nfp is fp32 (B, K).  Same paths as the forward.  The ring and token kernels
 * read a zero (B, C) g_gap_x from the workspace, which this call clears first with one cudaMemsetAsync (2 launches in
 * all); the row-band kernels (1 launch) keep g_gap_nfp / (H' W') in fp32 registers and shared memory and read no per-pixel
 * gradient; the generic kernels expand it to an fp32 map in the workspace.
 * Alignment: x, gx, workspace 16 bytes; g_gap_nfp 4 bytes. */
int nfpb200_pooled_map_backward(const nfpb200_desc_t* desc, const void* x, const float* g_gap_nfp, void* gx,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ---- fused nfp_pooling head (NFP_Pooling.py:25-36), one launch each way ---------------------------------------
 *   out (B, C) = GAP(x) * (proj_w . GAP(NFP(x)) + proj_b)        proj_w (C, K) fp32 row-major = nfp_proj.weight,
 *                                                                 proj_b (C) fp32 = nfp_proj.bias (NULL = none)
 * The forward also returns gap_x (B, C) and gap_nfp (B, K) (fp32): the backward reads them back, and the caller needs
 * them for the parameter gradients (d proj_w = (g_out * gap_x)^T gap_nfp, d proj_b = sum_b g_out * gap_x), which stay
 * on the caller's side.  Served by the fused NCHW ring kernels and the channels-last token kernels (cosine, pad = R, stride 1);
 * nfpb200_head_supported() returns NFPB200_OK when both directions are, NFPB200_EUNSUPPORTED otherwise -- then compose
 * nfpb200_pool_forward / _backward with the projection on the caller's side.
 * Alignment: x, gx, proj_w 16 bytes; proj_b, out, gap_x, gap_nfp, g_out 4 bytes. */
int nfpb200_head_supported(const nfpb200_desc_t* desc);
int nfpb200_head_forward(const nfpb200_desc_t* desc, const void* x, const float* proj_w, const float* proj_b, float* out,
                         float* gap_x, float* gap_nfp, void* stream);
/* gx = d loss / dx given g_out = d loss / d out (B, C) fp32 and the forward's gap_x / gap_nfp. */
int nfpb200_head_backward(const nfpb200_desc_t* desc, const void* x, const float* proj_w, const float* proj_b,
                          const float* gap_x, const float* gap_nfp, const float* g_out, void* gx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NFP_B200_H_ */
