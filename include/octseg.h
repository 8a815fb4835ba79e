/*
 * octseg.h — C-ABI of the B200-native hot path of oct_segmentation's hybrid-ensemble
 * inference (src/predict.py + OCTSegmentationModel.predict + smp network forward).
 *
 * The reference has no FFI of its own: its hot path is Python calling torch library ops
 * (SURVEY.md §8b).  Each entry point below names the reference call it replaces.  Rules:
 *   - plain C: pointers, sizes, POD structs; no torch / C++ types cross this boundary;
 *   - every pointer is a DEVICE pointer unless the parameter name starts with `h_`;
 *   - nothing here allocates device memory, takes ownership or synchronises: work is
 *     enqueued on the `stream` argument (a cudaStream_t passed as void*);
 *   - return 0 on success, a negative OCTSEG_E* code otherwise; octseg_last_error()
 *     returns a thread-local message for the last failure;
 *   - activations are dense NHWC bf16, channel pitch a multiple of 8 (16-byte pixels).
 */
#ifndef OCTSEG_H_
#define OCTSEG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCTSEG_ABI_VERSION 4

enum {
  OCTSEG_OK = 0,
  OCTSEG_EINVAL = -1,   /* bad argument / unsupported shape */
  OCTSEG_ECUDA = -2,    /* CUDA runtime or driver error     */
  OCTSEG_ENODEV = -3    /* no sm_100 device                 */
};

enum { OCTSEG_ACT_NONE = 0, OCTSEG_ACT_RELU = 1, OCTSEG_ACT_SWISH = 2, OCTSEG_ACT_SIGMOID = 3 };
enum { OCTSEG_RES_NONE = 0, OCTSEG_RES_BEFORE_ACT = 1, OCTSEG_RES_AFTER_ACT = 2 };
enum {
  OCTSEG_OUT_BF16_NHWC = 0, /* activation tensor                                      */
  OCTSEG_OUT_F32_NCHW = 1,  /* logits, the dtype/layout smp's forward() returns       */
  OCTSEG_OUT_U8_NCHW = 2    /* fused `sigmoid(y) > 0.5` (== y > 0): {0,1} bytes       */
};

#define OCTSEG_MAX_SEG 6

const char* octseg_last_error(void);
int octseg_abi_version(void);
/* Number of SMs of the current device (grid sizing); negative on error. */
int octseg_sm_count(void);

/* ------------------------------------------------------------------------------------------
 * Tensor-core implicit-GEMM convolution (tcgen05 + TMEM + TMA), one launch per fused op.
 * Replaces torch's conv2d / conv_transpose2d + batch_norm + relu|silu + interpolate(nearest)
 * + cat + residual add as issued by smp 0.3.3 decoders and the three encoders
 * (reference call sites: src/models/smp/model.py:70,192 `self.model(x)`).
 *
 * GEMM view:  D[pixel, cout] = sum over K-segments/taps/channels  A[pixel+tap, cin] * B[cout, k].
 * One K-segment = one source tensor of a fused channel concat.  Tiles are TH x TW output
 * pixels (TH*TW <= 128) by BN output channels; in 4-phase mode (fused nearest-x2 upsample or
 * ConvTranspose k4 s2 p1) tiles live on the half-resolution grid and each phase (ph,pw) writes
 * output pixels (2i+ph, 2j+pw).
 * ------------------------------------------------------------------------------------------ */
typedef struct octseg_conv_seg {
  const void* ptr;    /* bf16 NHWC source, first channel of the slice (16-byte aligned)      */
  int32_t N, H, W;    /* source extent                                                       */
  int32_t C;          /* channels visible to this segment (tensor-map extent)                */
  int32_t ldc;        /* channel pitch of the source in elements (multiple of 8)             */
  int32_t kh, kw;     /* taps                                                                */
  int32_t mul;        /* source coordinate = mul * tile_origin + off[parity] + tap           */
  int32_t off_h[2];   /* per row-phase parity (index 0 used when phases == 1)                */
  int32_t off_w[2];
  int32_t c_per_tile; /* 0: all tiles read channels [0,C); >0 (grouped conv): tile n reads
                         channels starting at n*c_per_tile                                   */
  int32_t cchunks;    /* kc-channel chunks per tap                                           */
  int32_t kc;         /* chunk width 16 | 32 | 64 (32B / 64B / 128B swizzle); 64/kc consecutive
                         (tap, chunk) sub-blocks of a segment share one pipeline stage          */
  int32_t wide;       /* 1 (needs kc=64, mul=1, TH=1): load one (TW+kw-1)-pixel box per tap row and
                         run the kw taps as shifted views of it (kw x less activation traffic)  */
} octseg_conv_seg;

typedef struct octseg_conv_desc {
  int32_t nseg;
  octseg_conv_seg seg[OCTSEG_MAX_SEG];
  int32_t phases;      /* 1 or 4                                                             */
  int32_t N, Hq, Wq;   /* tile-space extent (output grid, or half of it when phases == 4)    */
  int32_t TH, TW;      /* tile extent, TH*TW <= 128                                          */
  int32_t BN;          /* UMMA N: multiple of 16, 16..256                                    */
  int32_t n_tiles_n;   /* channel tiles (== groups for a grouped conv)                       */
  int32_t cout_per_tile; /* real output channels each channel tile stores (<= BN, mult. of 8
                            for bf16 output)                                                 */
  int32_t Cout;        /* total real output channels                                         */
  /* packed weights, bf16 [Z][n_tiles_n*BN][Ktot], Ktot = sum over segments of kh*kw*cchunks*kc;
     Z = phases * (per_image_weights ? N : 1), z = phase + phases*image                      */
  const void* weight;
  int32_t Ktot;
  int32_t per_image_weights;
  const float* bias;   /* fp32 [n_tiles_n*BN + 64] (zero padded)                             */
  int32_t act;         /* OCTSEG_ACT_*                                                       */
  int32_t res_mode;    /* OCTSEG_RES_*                                                       */
  const void* res;     /* bf16 NHWC residual at output resolution, or NULL                   */
  int32_t res_ldc;
  void* out;
  int32_t out_mode;    /* OCTSEG_OUT_*                                                       */
  int32_t out_H, out_W;/* output extent in pixels                                            */
  int32_t out_ldc;     /* NHWC: channel pitch; NCHW: number of channel planes                */
  int32_t out_c_off;   /* first output channel written                                       */
  int32_t out_pack;    /* NCHW outputs of a pixel-packed problem: GEMM column c is plane c % out_ldc
                          of pixel x*out_pack + c / out_ldc (rows are out_W*out_pack wide); 0/1 = off */
  int32_t d2s;         /* depth-to-space bf16 output: > 0 = channels per output pixel; GEMM column c is
                          channel c % d2s of pixel (2y + (c/d2s)/2, 2x + (c/d2s)%2) of a tensor twice as
                          large as the tile grid (fused upsample / ConvTranspose in one pass)        */
  int32_t halo;        /* 1 = halo-tile mode (needs nseg=1, phases=1, mul=1, TH=16, TW=8, no per-image
                          weights): one (TW+kw-1) x (TH+kh-1) halo box of A per channel chunk, the kh*kw taps are
                          shifted views of it, and the channel tile's weights (kh*kw*cchunks*BN*kc*2 bytes) stay
                          resident in shared memory; tiles are ordered channel tile slowest                */
  /* Fused 1x1 segmentation head (smp SegmentationHead with kernel_size 1: LinkNet, SURVEY.md N4) applied to this
     conv's activated output in the epilogue, so the conv's own (wide, full-resolution) output never reaches memory:
       logit[pixel][j] = head_bias[j] + sum_c act(conv[pixel][c] + bias[c]) * head_weight[j][c],  j < head_classes.
     Needs an NCHW out_mode (out_ldc = head_classes planes, written as logits or thresholded y > 0), n_tiles_n = 1,
     no residual, phases = 1, and GEMM columns = out_pack (1 | 2 | 4) packed pixels x head_cmid channels
     (Cout = out_pack * head_cmid <= BN, head_cmid in {16, 32, 48, 64}).  The three arrays are HOST pointers, read at
     plan creation: the head's operands travel in the kernel's parameter block (constant-bank FFMA operands), and
     `bias` (device) is not read by the fused epilogue.  0 = off.                                            */
  int32_t head_classes;         /* 1..4 */
  int32_t head_cmid;            /* channels of the conv per pixel */
  const float* head_weight;     /* host fp32 [head_classes][head_cmid] */
  const float* head_bias;       /* host fp32 [head_classes] */
  const float* head_conv_bias;  /* host fp32 [head_cmid]: the conv's own bias per channel */
} octseg_conv_desc;

typedef struct octseg_conv_plan octseg_conv_plan;

/* Builds TMA descriptors + launch geometry.  `*plan` is host memory owned by the library
   until octseg_conv_plan_destroy. */
int octseg_conv_plan_create(const octseg_conv_desc* desc, octseg_conv_plan** plan);
int octseg_conv_plan_destroy(octseg_conv_plan* plan);
int octseg_conv_run(const octseg_conv_plan* plan, void* stream);

/* What octseg_conv_plan_create decided for a plan (read-only; for tests and diagnostics).  The struct is used
   through its tag: the function below has the same name. */
struct octseg_conv_plan_info {
  int32_t grid;          /* persistent CTAs launched: min(total_tiles, SMs)                           */
  int32_t total_tiles;   /* phases * N * tiles_h * tiles_w * n_tiles_n                                */
  int32_t n_acc;         /* accumulators in the TMEM ring: min(8, 512 / BN)                           */
  int32_t nstages;       /* shared-memory pipeline stages                                             */
  int32_t use_tma_store; /* bf16 output leaves through TMA stores (else direct stores)                */
  int32_t out_grouped;   /* grouped conv stored through the 5-D (c, group, w, h, n) map              */
  int32_t d2s_tma;       /* depth-to-space output stored through TMA                                  */
  int32_t own_spatial;   /* a CTA takes whole spatial tiles, all their channel tiles back to back     */
  int32_t halo;          /* halo-tile mode                                                            */
  int32_t wide;          /* some segment loads wide (one box per tap row) A boxes                     */
};
int octseg_conv_plan_info(const octseg_conv_plan* plan, struct octseg_conv_plan_info* info);

/* ------------------------------------------------------------------------------------------
 * CUDA-core kernels for the HBM-bound / tiny-K layers.
 * ------------------------------------------------------------------------------------------ */

/* Network stem input (torch conv2d on `images_tensor`, model.py:189-192): space-to-depth packing of
   the 3-channel network input for the tensor-core stem conv.  The stride-2 k x k stem conv becomes a
   stride-1 conv (octseg_conv_*) over  out[n][y][x][(dy*2+dx)*3 + c] = norm(in[n][c][2y+dy][2x+dx]),
   bf16 NHWC [N][H/2][W/2][16] (channels 12..15 zero).
   Input is addressed by element strides so the NHWC-strided float tensor produced by
   `torch.Tensor(images.transpose(0,3,1,2))` (model.py:189) and uint8 NHWC frames are read in
   place.  in_dtype: 0 = f32, 1 = u8.  `mean`/`inv_std` (3 floats each, HOST pointers, may be
   NULL) apply OCTSegmentationModel.forward's normalisation (model.py:69) on the fly. */
int octseg_stem_pack(const void* in, int32_t in_dtype, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                     int32_t N, int32_t H, int32_t W, const float* h_mean, const float* h_inv_std,
                     void* out /* bf16 NHWC [N][H/2][W/2][16] */, void* stream);

/* torch max_pool2d(kernel 3, stride 2, padding 1) of torchvision ResNet (bf16 NHWC). */
int octseg_maxpool3x3s2(const void* in, void* out, int32_t N, int32_t H, int32_t W, int32_t C,
                        int32_t Ho, int32_t Wo, void* stream);

/* Depthwise kxk conv (efficientnet_pytorch MBConvBlock._depthwise_conv with static "same"
   padding, k in {3,5}, stride in {1,2}) + folded BN + swish; optionally writes the squeeze-excite channel sums
   (adaptive_avg_pool2d numerator) as partial sums `pool_sum` fp32 [N][pool_slots][C]: one slot per row group of
   tiles, each written exactly once (plain stores: no zeroing, no atomics, bit-reproducible);
   pool_slots = octseg_dwconv_pool_slots(C, Ho, Wo); octseg_se_hidden adds the slots in order. */
int octseg_dwconv(const void* in, const void* weight /* bf16 [kh][kw][C] */, const float* bias,
                  void* out, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k, int32_t stride,
                  int32_t pad_t, int32_t pad_l, int32_t Ho, int32_t Wo, int32_t act,
                  float* pool_sum, int32_t pool_slots, void* stream);
int octseg_dwconv_pool_slots(int32_t C, int32_t Ho, int32_t Wo);

/* Squeeze-excite (efficientnet_pytorch MBConvBlock: adaptive_avg_pool2d -> _se_reduce -> swish ->
   _se_expand -> sigmoid -> gate * x), folded into the projection 1x1 conv's weights:
   hidden[n][r] = swish(w1[r,:] . (sum_s pool_sum[n,s,:] * inv_hw) + b1[r])          fp32 [N][Cr]
   pool_sum: fp32 [N][slots][C] partial sums (octseg_dwconv), added in slot order into
   sums_scratch fp32 [N][C] first (a second tiny launch; may be NULL when slots == 1). */
int octseg_se_hidden(const float* pool_sum, int32_t slots, float* sums_scratch, float inv_hw,
                     const float* w1 /* [Cr][C] */, const float* b1, float* hidden, int32_t N, int32_t C, int32_t Cr,
                     void* stream);

/* gate[n][k] = sigmoid(w2[k,:] . hidden[n,:] + b2[k])                               fp32 [N][C]
   `pool_clear` (may be NULL): fp32 [N][C] buffer set to zero on the way (unused since the pool sums became
   write-once slots; kept for callers that accumulate into a buffer of their own). */
int octseg_se_gate(const float* hidden, const float* w2t /* fp32 [Cr][C] */, const float* b2, float* gate,
                   float* pool_clear, int32_t N, int32_t C, int32_t Cr, void* stream);

/* out[n][row][k] = bf16(w[row][k] * gate[n][k % gate_period]) for k < C and 0 for the K padding: per-image weights
   of the projection conv (B tensor map z = n), i.e. `gate * x` folded into `_project_conv`.  gate: fp32
   [N][gate_period]; gate_period = C for a plain conv (0 means C), the channel count of one pixel when the conv runs on
   a pixel-packed view (K = packed pixels x channels). */
int octseg_se_scale_weights(const float* gate, const float* w /* fp32 [rows][Ktot] */,
                            void* out /* bf16 [N][rows][Ktot] */, int32_t N, int32_t rows, int32_t Ktot,
                            int32_t C, int32_t gate_period, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pre-processing: preprocessing_img (src/data/utils.py:159-166): RGB->BGR + cv2.resize
 * INTER_LINEAR (uint8, 11-bit fixed point) of a uint8 HWC frame, written as the uint8 NHWC
 * network input (N,S,S,3).  Bit-exact vs cv2.
 * ------------------------------------------------------------------------------------------ */
/* xofs/yofs: int32 [S] left/top source index; xalpha/ybeta: int16 [S][2] 11-bit coefficients,
   computed by the caller with cv2's float32 rule (fx=(float)((dx+0.5)*scale-0.5); see
   oct_segmentation_b200/prepost.py).  All four are DEVICE pointers. */
int octseg_preprocess_resize_bgr(const uint8_t* src /* [N][Hs][Ws][3] RGB */, int32_t N, int32_t Hs,
                                 int32_t Ws, uint8_t* dst /* [N][S][S][3] BGR */, int32_t S,
                                 const int32_t* xofs, const int16_t* xalpha, const int32_t* yofs,
                                 const int16_t* ybeta, int32_t area_fast_2x, void* stream);

/* The same resize written straight into the stem's input format (what octseg_stem_pack produces for a uint8 frame
   without normalisation): dst = bf16 [N][S/2][S/2][16], channel (dy*2 + dx)*3 + c = pixel (2y+dy, 2x+dx), channel c of
   the BGR frame preprocessing_img returns (src/data/utils.py:159-166), channels 12..15 zero.  uint8 -> bf16 is exact, so
   this is octseg_preprocess_resize_bgr + octseg_stem_pack in one pass over the frame (predict path, model.py:192).
   channels: 3 (RGB source) or 1 (grayscale, replicated).  S even, dst 16-byte aligned. */
int octseg_preprocess_resize_s2d(const uint8_t* src, int32_t channels, int32_t N, int32_t Hs, int32_t Ws, void* dst,
                                 int32_t S, const int32_t* xofs, const int16_t* xalpha, const int32_t* yofs,
                                 const int16_t* ybeta, int32_t area_fast_2x, void* stream);

/* Grayscale extension (SURVEY.md section 8a, "grayscale-to-3ch"; the reference replicates channels only in
   dataset prep, src/data/utils.py:111): src is uint8 [N][Hs][Ws] and the resized plane is written to all three
   channels of dst -- identical to octseg_preprocess_resize_bgr on the channel-replicated frame. */
int octseg_preprocess_resize_gray(const uint8_t* src /* [N][Hs][Ws] */, int32_t N, int32_t Hs,
                                 int32_t Ws, uint8_t* dst /* [N][S][S][3] BGR */, int32_t S,
                                 const int32_t* xofs, const int16_t* xalpha, const int32_t* yofs,
                                 const int16_t* ybeta, int32_t area_fast_2x, void* stream);

/* ------------------------------------------------------------------------------------------
 * Post-processing: threshold (model.py:195) + cv2.resize INTER_NEAREST (predict.py:92-96) +
 * class routing (predict.py:97-100, MODELS_META) + priority label map (data/utils.py:231-233)
 * + per-class pixel count (analysis.py:199) in one pass over the output grid.
 *   chan[c]: pointer to the {0,1} uint8 planes [N][S_c][S_c] feeding mask channel c (or NULL:
 *            class absent -> zeros), c = class id - 1 (LM, FC, LC, VV); h_img_stride[c] = bytes
 *            between consecutive frames' planes (S_c*S_c when dense; C*S_c*S_c when the plane is
 *            one channel of a network's NCHW output).
 *   h_lut[c]: DEVICE int32 [Ho + Wo]: source row for each output row, then source column for
 *            each output column (cv2 rule sx = min(floor(x * (1/(dst/src))), src-1))
 *   mask   : uint8 [N][Ho][Wo][4] {0,1}      (the reference's float64 HxWx4 array, as bytes)
 *   label  : uint8 [N][Ho][Wo] 0 = background, else highest-priority class id (later class in
 *            `order` wins), or NULL
 *   counts : int32 [N][4] non-zero pixels per class (zeroed by caller)
 * ------------------------------------------------------------------------------------------ */
int octseg_postprocess(const uint8_t* const* h_chan, const int32_t* h_S, const int64_t* h_img_stride,
                       const int32_t* const* h_lut, const int32_t* h_order,
                       int32_t n_order, int32_t N, int32_t Ho, int32_t Wo, uint8_t* mask,
                       uint8_t* label, int32_t* counts, void* stream);

/* calculate_object_thickness (src/app/tools/analysis.py:60-130): 360 rays from the image
   centre; per ray the last radius inside the object before the first exit.
   mask: uint8 [N][H][W][4] (non-zero = object); radii: int32 [N][4][360] (0 = ray missed). */
/* cos_sin: DEVICE double [720] = cos(radians(a)) for a in 0..359, then sin(...) (host libm
   values, so x = int(cx + r*cos) truncates exactly like the reference's Python floats). */
int octseg_radial_thickness(const uint8_t* mask, int32_t N, int32_t H, int32_t W, const double* cos_sin,
                            int32_t* radii, void* stream);

/* Overlay cosmetics of save_results (src/data/utils.py:209-230 + get_img_mask_union_pil,
   src/models/smp/utils.py:203-213), one pass, bit-exact vs the reference's cv2 + PIL output:
   per class in paint order: CLOSE(ellipse 5x5) -> rim = dilate7 & ~erode7 -> 5x5 binomial blur ->
   two PIL alpha pastes (fill alpha = h_fill_lut[k], k = 256 * blur in 0..256; rim alpha = rim_alpha).
   img, out: DEVICE uint8 [N][H][W][3] RGB; mask: DEVICE uint8 [N][H][W][4] (non-zero = class present,
   4-byte aligned - the mask octseg_postprocess writes); h_order: HOST class channels (0..3) in
   cfg.classes order; h_colors: HOST uint8 [4][3] RGB per class channel; h_fill_lut: HOST uint8 [257].
   H, W >= 3. */
int octseg_overlay(const uint8_t* img, const uint8_t* mask, uint8_t* out, int32_t N, int32_t H, int32_t W,
                   const int32_t* h_order, int32_t n_order, const uint8_t* h_colors,
                   const uint8_t* h_fill_lut, int32_t rim_alpha, void* stream);

/* K-way probability averaging (north-star "ensemble averaging"; opt-in generalisation of the reference's
   per-class routing, SURVEY.md section 8a): out[i] = (1/K * sum_k sigmoid(logits[k][i])) > 0.5 ? 1 : 0 in fp32.
   K = 1 is `y.sigmoid() > 0.5` (src/models/smp/model.py:195).  h_logits: HOST array of K (1..8) DEVICE
   pointers to fp32 tensors of n elements each (16-byte aligned); out: DEVICE uint8 [n] (4-byte aligned). */
int octseg_fold_average_threshold(const float* const* h_logits, int32_t K, int64_t n, uint8_t* out, void* stream);

/* calculate_thickness_contour (src/app/tools/analysis.py:21-57), device part: per (frame, class) the largest outer
   border of cv2.findContours(mask, RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) (== max(contours, key=contourArea)), same
   points in the same order.  mask: DEVICE uint8 [N][H][W][4] (non-zero = object).  Outputs (DEVICE):
   sums int64 [N][4][4] = a00, a10, a01 (the integer accumulators of cv2's polygon moments: m00 = |a00|/2, ...)
   and the start pixel index y*W+x (-1: no border with non-zero area); nverts int32 [N][4] = kept points of that
   border (may exceed cap: only the first cap are stored); verts int16 [N][4][cap][2] = x, y.
   The host finishes centroid (int-truncated), distances, median / min / max.  (H+2)*(ceil((W+1)/32)+1)*4 bytes of
   shared memory must fit 226 KB (1000 x 1000: 132 KB). */
int octseg_contour_largest(const uint8_t* mask, int32_t N, int32_t H, int32_t W, int64_t* sums, int32_t* nverts,
                           int16_t* verts, int32_t cap, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OCTSEG_H_ */
