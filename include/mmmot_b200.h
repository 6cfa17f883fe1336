/*
 * mmmot_b200.h — C ABI of libmmmot_sm100a.so
 *
 * B200-native (sm_100a) implementation of mmMOT's per-frame-pair association forward.
 * The reference (ZwwWayne/mmMOT) has no FFI of its own: its boundary is the Python class
 * modules/tracking_net.py:15 `TrackingNet` and the function solvers.py:9 `ortools_solve`.
 * Each entry point below replaces one group of ATen/OR-tools calls behind that boundary; the
 * reference lines replaced are cited per function.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - plain pointers + sizes only; every pointer is a DEVICE pointer unless marked host.
 *   - no allocation, no ownership transfer, stateless, stream-ordered (last argument is a
 *     cudaStream_t passed as void*), thread-safe across streams.
 *   - return 0 on success, a negative MMMOT_E_* on a bad argument, or a positive cudaError_t.
 *   - every `workspace` starts with a 256-byte STATUS BLOCK (included in the mmmot_*_workspace sizes): stages raise
 *     flags in it while they run and never clear it.  Protocol: mmmot_status_reset(ws) -> stages ... -> mmmot_status_check(ws).
 *   - all real data is fp32; `stats` scratch is fp64.
 *   - "group" = one GroupNorm domain.  A frame-pair with N previous / M next detections has
 *     L = N + M detections; all pairs of one call share N, M, crop size H x W.
 *   - feature tensors are channel-major: feats[pair][stack 0..2][512][L]
 *     (stack 0 = image, 1 = LiDAR, 2 = fused; reference: modules/tracking_net.py:40,131-145).
 */
#ifndef MMMOT_B200_H
#define MMMOT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMMOT_ABI_VERSION 2

enum {
  MMMOT_E_ARG = -1,        /* null pointer / non-positive size / unsupported enum */
  MMMOT_E_WORKSPACE = -2,  /* workspace too small */
  MMMOT_E_SHAPE = -3,      /* shape constraint violated (see function comment) */
  MMMOT_E_RANGE = -4       /* an activation left FP16's range (|x| >= 65504) on the tensor-core path: the result
                              of the stage that raised it is clamped, i.e. WRONG (mmmot_status_check) */
};

/* fusion_module_{A,B,C}: reference modules/fusion_net.py:73,45,6 */
enum { MMMOT_FUSION_A = 0, MMMOT_FUSION_B = 1, MMMOT_FUSION_C = 2 };
/* batch_multiply / batch_minus_abs / batch_minus: reference modules/gcn.py:6,17,32 */
enum { MMMOT_AFF_MULTIPLY = 0, MMMOT_AFF_MINUS_ABS = 1, MMMOT_AFF_MINUS = 2 };
/* softmax_mode: reference modules/tracking_net.py:109-124 */
enum { MMMOT_SM_NONE = 0, MMMOT_SM_SINGLE = 1, MMMOT_SM_DUAL = 2, MMMOT_SM_DUAL_ADD = 3, MMMOT_SM_DUAL_MAX = 4 };
/* NewEndIndicator_v2 mode: reference modules/new_end.py:69-74 (mean / max of the normalised map over the other frame) */
enum { MMMOT_END_AVG = 0, MMMOT_END_MAX = 1 };

/*
 * Prepared weights.  Produced once per checkpoint by the host (mmmot_b200/weights.py) from the
 * reference state_dict: eval-mode BatchNorm folded into the preceding conv, the two constant
 * STN transforms (SURVEY F4) folded into the PointNet convs they feed, every matrix stored
 * TRANSPOSED as Wt[K][Cout] (K-major rows, Cout contiguous).
 */
enum mmmot_weight_id {
  /* VGG16-BN trunk, 13 convs: Wt[(ky*3+kx)*Cin + ci][Cout], bias[Cout]  (appear_net.py:166-172) */
  MMMOT_W_VGG_WT0 = 0,            /* .. +12 */
  MMMOT_W_VGG_B0 = 13,            /* .. +12 */
  /* SkipPool heads s=0..3, 10 tensors each (appear_net.py:18-32):
     +0 gn0_w[C] +1 gn0_b[C] +2 w1t[C][mid] +3 b1[mid] +4 gn1_w +5 gn1_b +6 w2t[mid][128] +7 b2 +8 gn2_w +9 gn2_b */
  MMMOT_W_SKIP0 = 26,             /* .. +39 */
  /* PointNet trunk (point_net.py:115-138), layer i=1..5: +0 wt[Cin][Cout] +1 b +2 gn_w +3 gn_b */
  MMMOT_W_PN_L1 = 66,             /* .. 5 layers x 4 = 20 */
  /* PointNet head (point_net.py:25-41) */
  MMMOT_W_PN_WHAT = 86,           /* [64][512]   local-feature part of conv1, T2 folded in   */
  MMMOT_W_PN_WHGT = 87,           /* [1024][512] global-feature part of conv1                */
  MMMOT_W_PN_BH = 88, MMMOT_W_PN_GHW = 89, MMMOT_W_PN_GHB = 90,
  MMMOT_W_PN_WOT = 91,            /* [512][512] conv2 */
  MMMOT_W_PN_BO = 92, MMMOT_W_PN_GOW = 93, MMMOT_W_PN_GOB = 94,
  /* fusion (fusion_net.py): A uses WPT as the [1024][512] matrix; B uses WPT/WIT; C adds gates */
  MMMOT_W_FU_WPT = 95, MMMOT_W_FU_BP = 96, MMMOT_W_FU_GPW = 97, MMMOT_W_FU_GPB = 98,
  MMMOT_W_FU_WIT = 99, MMMOT_W_FU_BI = 100, MMMOT_W_FU_GIW = 101, MMMOT_W_FU_GIB = 102,
  MMMOT_W_FU_GATE_PT = 103, MMMOT_W_FU_GATE_PB = 104, MMMOT_W_FU_GATE_IT = 105, MMMOT_W_FU_GATE_IB = 106,
  /* w_det (tracking_net.py:92-100), BN folded */
  MMMOT_W_WD_W1T = 107, MMMOT_W_WD_B1 = 108, MMMOT_W_WD_W2T = 109, MMMOT_W_WD_B2 = 110,
  MMMOT_W_WD_W3 = 111, MMMOT_W_WD_B3 = 112,
  /* affinity (gcn.py:59-66) + new/end conv0 (new_end.py:48-52) stacked as one [512][1024] matrix */
  MMMOT_W_AF_W01T = 113, MMMOT_W_AF_B01 = 114,
  MMMOT_W_AF_G1W = 115, MMMOT_W_AF_G1B = 116,   /* conv1.1  GN(512,512) */
  MMMOT_W_AF_G0W = 117, MMMOT_W_AF_G0B = 118,   /* w_new_end.conv0.1  GN(1,512) */
  MMMOT_W_AF_W2T = 119, MMMOT_W_AF_B2 = 120, MMMOT_W_AF_G2W = 121, MMMOT_W_AF_G2B = 122,
  MMMOT_W_AF_W3T = 123, MMMOT_W_AF_B3 = 124, MMMOT_W_AF_G3W = 125, MMMOT_W_AF_G3B = 126,
  MMMOT_W_AF_W4 = 127, MMMOT_W_AF_B4 = 128,
  /* new/end 1-D MLP (new_end.py:53-60) */
  MMMOT_W_NE_W1T = 129, MMMOT_W_NE_B1 = 130, MMMOT_W_NE_G1W = 131, MMMOT_W_NE_G1B = 132,
  MMMOT_W_NE_W2T = 133, MMMOT_W_NE_B2 = 134, MMMOT_W_NE_G2W = 135, MMMOT_W_NE_G2B = 136,
  MMMOT_W_NE_W3 = 137, MMMOT_W_NE_B3 = 138,
  /* ---- tensor-core operands: the same matrices split into FP16 hi/lo and pre-tiled in the UMMA
     canonical K-major core-matrix layout  [k chunk 32][m tile 128][hi|lo][k group 4][m group 16][8][8]
     (zero padded to multiples of 128 rows / 32 k); see csrc/tc_common.cuh.  VGG layer 0 (fp32 NCHW crops) uses
     the K order k = ci*9 + (ky*3+kx); layers 1..12 (packed FP16 NHWC activations) use k = (ky*3+kx)*Cin + ci. */
  MMMOT_W_VGG_WP0 = 139,          /* .. +12 */
  MMMOT_W_PN_WP1 = 152,           /* .. +4 : PointNet trunk layers 1..5 */
  MMMOT_W_PN_WHAP = 157,
  MMMOT_W_AF_W01P = 158, MMMOT_W_AF_W2P = 159, MMMOT_W_AF_W3P = 160,
  /* ---- training-mode operands (SURVEY 8f N4): the UNFOLDED conv weights / biases and the BatchNorm affines of the
     layers whose BatchNorm uses batch statistics in .train() */
  MMMOT_W_VGG_RAWW0 = 161,        /* .. +12 : Wt[(ky*3+kx)*Cin + ci][Cout], not folded */
  MMMOT_W_VGG_RAWB0 = 174,        /* .. +12 */
  MMMOT_W_VGG_BNW0 = 187,         /* .. +12 : BatchNorm2d weight */
  MMMOT_W_VGG_BNB0 = 200,         /* .. +12 : BatchNorm2d bias */
  MMMOT_W_WD_RAW0 = 213,          /* .. +7  : w_det w1t b1 bn1_w bn1_b w2t b2 bn2_w bn2_b */
  /* ---- packed tensor-core tiles of the per-detection contractions (fusion linears, gates, w_det; BN folded) */
  MMMOT_W_FU_WPP = 221, MMMOT_W_FU_WIP = 222, MMMOT_W_FU_GATE_PP = 223, MMMOT_W_FU_GATE_IP = 224,
  MMMOT_W_WD_W1P = 225, MMMOT_W_WD_W2P = 226,
  /* the two 64-output VGG layers again, compact for the pixel-major kernel: [k chunk][hi|lo][k group 4][row group 8][8][8] */
  MMMOT_W_VGG_WPX0 = 227,         /* .. +1 */
  /* packed tiles of the remaining small contractions: new/end MLP, PointNet per-detection parts */
  MMMOT_W_NE_W1P = 229, MMMOT_W_NE_W2P = 230, MMMOT_W_PN_WHGP = 231, MMMOT_W_PN_WOP = 232,
  MMMOT_W_COUNT = 233
};

typedef struct mmmot_weights {
  const float* w[MMMOT_W_COUNT];
  /* for the packed tensor-core operands (ids >= MMMOT_W_VGG_WP0): 2^-s, where the packed FP16 tiles
     hold W * 2^s (power-of-two pre-scaling keeps the lo terms in FP16's normal range) */
  float tc_scale[MMMOT_W_COUNT];
} mmmot_weights;

int mmmot_abi_version(void);

/* Status block of a workspace (see Conventions).  reset: stream-ordered clear.  check: copies the status word back,
 * SYNCHRONISES the stream and returns 0 or MMMOT_E_RANGE.  The tensor-core engines feed activations to the MMA units
 * as FP16 hi/lo pairs; a value with |x| >= 65504 saturates in that conversion, which these calls make loud. */
int mmmot_status_reset(void* workspace, void* stream);
int mmmot_status_check(const void* workspace, void* stream);
/* Small stream-ordered host -> device transfer that uses NEITHER the copy engine NOR a host synchronisation: a kernel
 * reads `count` int32 words straight from PINNED (page-locked, mapped) host memory.  For the CSR offsets that accompany
 * a sub-batch: a cudaMemcpyAsync of them would queue on the copy engine behind the bulk input copies of the NEXT
 * sub-batch (stalling the compute stream for milliseconds), a pageable copy blocks the calling thread.  The source
 * must stay untouched until the stream has passed this call.  MMMOT_E_ARG if `src_pinned_host` is not pinned. */
int mmmot_fetch_pinned_i32(int* dst_device, const int* src_pinned_host, long count, void* stream);
/* number of SMs / name of the current device: lets the host fail loudly when no sm_100 GPU is present */
int mmmot_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------------------------
 * Appearance: VGG16-BN trunk + 4 SkipPool heads -> stack 0 of feats.
 * Replaces AppearanceNet.forward, reference modules/appear_net.py:166-190 (+ vgg.py:67-80).
 *   crops  [n_img][3][H][W]   (H, W multiples of 32), n_img = pairs*L
 *   feats  [pairs][3][512][L] ; writes feats[p][0][:][l] for image p*L + l
 * workspace: mmmot_appearance_workspace(n_img, H, W) bytes.
 */
size_t mmmot_appearance_workspace(int n_img, int H, int W);
int mmmot_appearance_fwd(const mmmot_weights* wts, const float* crops, int n_img, int H, int W,
                         int L, float* feats, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * PointNet encoder over ragged per-detection point sets -> stack 1 of feats.
 * Replaces PointNet_v1.forward, reference modules/point_net.py:25-44,115-153.
 *   points     [P_total][3]  xyz, detections concatenated in order
 *   det_split  [pairs*L + 1] int32 CSR offsets into points (device)
 *   h_det_split same array on the HOST (used only to size the launch; the reference reads it
 *               with .item() per detection, point_net.py:33-35,140-142)
 * Every pair is one GroupNorm domain (all points of its L detections).
 */
size_t mmmot_pointnet_workspace(int pairs, int L, long p_total);
int mmmot_pointnet_fwd(const mmmot_weights* wts, const float* points, const int* det_split,
                       const int* h_det_split, int pairs, int L, float* feats,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fusion A/B/C -> stack 2 of feats, then the detection-score branch on all 3 stacks.
 * Replaces fusion_module_{A,B,C}.forward (modules/fusion_net.py:31-42,62-70,85-92) and
 * TrackingNet.determine_det eval branch (modules/tracking_net.py:149-163).
 *   det_scores [pairs][3][L]   = s - [s < neg_threshold],  s = sigmoid(w_det(feats)) if score_flags & MMMOT_SCORE_SIGMOID
 *                                ('cls' in score_arch, tracking_net.py:153-156) else w_det(feats);
 *                                the threshold step is skipped without MMMOT_SCORE_THRESHOLD.
 */
enum { MMMOT_SCORE_SIGMOID = 1, MMMOT_SCORE_THRESHOLD = 2 };
size_t mmmot_fusion_det_workspace(int pairs, int L);
int mmmot_fusion_det_fwd(const mmmot_weights* wts, int fusion_arch, int score_flags, float neg_threshold,
                         int pairs, int L, float* feats, float* det_scores,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training-mode variants (SURVEY.md 8f row N4) of the two stages that contain BatchNorm: in .train() the reference's
 * BatchNorm2d layers of the VGG trunk (modules/vgg.py:67-80) and BatchNorm1d layers of w_det (modules/tracking_net.py:
 * 92-100) use the statistics of the current batch, and det_scores stay raw logits (tracking_net.py:152-162).  FP32 FFMA
 * engine; one frame-pair = one batch (the reference trains on one sample per step, tracking_model.py:50-66).
 *   mmmot_appearance_train_fwd: as mmmot_appearance_fwd; bn_stats [13][2][512] = per layer (batch mean | biased batch
 *     variance) per channel, for the caller's running-average update.
 *   mmmot_w_det_train_fwd: feats [3][512][L] of one pair -> det_scores [3][L] raw logits; bn_stats [2][2][512].
 *     drop_mask2 / drop_mask3 (NULL = none): DropBlock2D weights of the two deepest SkipPool heads
 *     (modules/appear_net.py:27-30,143-152; modules/dropblock.py:28-55), [n_img][H/16][W/16] and [n_img][H/32][W/32] =
 *     block_mask * numel / sum.  The caller draws the Bernoulli seeds (the reference draws them with torch's CPU generator,
 *     which a bit-matching run has to share) and max-pools them into blocks; the library applies them before the mean.
 *   mmmot_pointnet_train_fwd: as mmmot_pointnet_fwd on the FP32 engine, with the optional nn.Dropout mask of the head
 *     activation (modules/point_net.py:29-30): head_drop_mask [512][P], values {0, 1/(1-p)}, NULL = none.
 * Fusion and affinity have neither BatchNorm nor dropout: the eval entry points serve both modes
 * (mmmot_fusion_det_fwd's det_scores are simply overwritten by mmmot_w_det_train_fwd's).  Forward only: no gradients.
 */
size_t mmmot_appearance_train_workspace(int n_img, int H, int W);
int mmmot_appearance_train_fwd(const mmmot_weights* wts, const float* crops, int n_img, int H, int W, int L,
                               float* feats, float* bn_stats, const float* drop_mask2, const float* drop_mask3,
                               void* workspace, size_t workspace_bytes, void* stream);
size_t mmmot_pointnet_train_workspace(int pairs, int L, long p_total);
int mmmot_pointnet_train_fwd(const mmmot_weights* wts, const float* points, const int* det_split, const int* h_det_split,
                             int pairs, int L, const float* head_drop_mask, float* feats, void* workspace,
                             size_t workspace_bytes, void* stream);
size_t mmmot_w_det_train_workspace(int L);
int mmmot_w_det_train_fwd(const mmmot_weights* wts, int L, const float* feats, float* det_scores, float* bn_stats,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pairwise affinity + start/end indicator + softmax mode.
 * Replaces affinity_module.forward (modules/gcn.py:68-82), NewEndIndicator_v2.forward
 * (modules/new_end.py:62-82, modes 'avg' and 'max') and TrackingNet.associate (tracking_net.py:106-126).
 * The 3 x 512 x N x M pairwise tensor is generated tile by tile inside the first contraction's operand producers
 * (csrc/gemm_gen.cuh) and never stored; GroupNorm + ReLU between the MLP layers is applied by the next layer's
 * producers, so each layer output crosses HBM once as fp32.
 *   link  [pairs][3][N][M]
 *   new_s [pairs][3][M]   end_s [pairs][3][N]   (un-padded; the host pads with zeros as
 *                                                tracking_net.py:183-189 does)
 */
size_t mmmot_affinity_workspace(int pairs, int n, int m);
int mmmot_affinity_fwd(const mmmot_weights* wts, int affinity_op, int softmax_mode, int end_mode,
                       int pairs, int n, int m, const float* feats,
                       float* link, float* new_s, float* end_s,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Association integer programme for 2-frame pairs, solved exactly as a rectangular
 * assignment problem (SURVEY F9).  Replaces ortools_solve, reference solvers.py:9-138.
 *   det [pairs][L], link [pairs][N][M], new_s/end_s [pairs][L] (zero-padded like the reference's
 *   forward output); strides in floats between consecutive pairs are given explicitly so the
 *   solver can read the test_mode stack straight out of the forward outputs.
 *   outputs (fp32 0/1, same layout as solvers.py:116-131):
 *   a_det [pairs][L], a_link [pairs][N][M], a_new [pairs][L], a_end [pairs][L]
 *   match [pairs][N] int32: column matched to previous detection j, or -1.
 */
size_t mmmot_lp_workspace(int pairs, int n, int m);
int mmmot_lp_assign(const float* det, long det_stride, const float* link, long link_stride,
                    const float* new_s, long new_stride, const float* end_s, long end_stride,
                    int pairs, int n, int m,
                    float* a_det, float* a_link, float* a_new, float* a_end, int* match,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-detection LiDAR cropping (SURVEY.md 8f row N1 — the step right before the hot path).
 * Replaces the host loop of reference point_cloud/preprocess.py:72-81 / box_np_ops.py:688-699 /
 * geometry.py:96-114.  planes[n_boxes][6][4]: inward plane equations (nx, ny, nz, d) of each rotated box,
 * prepared by the host exactly as the reference's numpy code does (mmmot_b200/lidar_crop.py), float64 when
 * planes_f64 != 0 (the reference's real pipeline: box_camera_to_lidar yields float64 boxes) else float32; a point is
 * inside iff x*nx + y*ny + z*nz + d < 0 for all six (evaluated in that precision, in the reference's operation
 * order, unfused).
 * Two steps because the output size is data dependent:
 *   mmmot_crop_count   -> split[n_boxes + 1] (device) CSR offsets; an empty box counts one (zero) point
 *   mmmot_crop_scatter -> out_points[split[n_boxes]][out_channels], scene order preserved inside a box
 * Both need the same workspace (mmmot_crop_workspace bytes) and the count step's contents are consumed by scatter.
 */
size_t mmmot_crop_workspace(int n_points, int n_boxes);
int mmmot_crop_count(const float* points, int n_points, int stride, const void* planes, int planes_f64, int n_boxes,
                     int* split, void* workspace, size_t workspace_bytes, void* stream);
int mmmot_crop_scatter(const float* points, int n_points, int stride, const void* planes, int planes_f64, int n_boxes,
                       const int* split, int out_channels, float* out_points, void* workspace,
                       size_t workspace_bytes, void* stream);

/*
 * Per-detection image crop-and-resize (SURVEY.md 8f row N2 — the image-side step right before the hot path).
 * Replaces reference dataset/test_seq_dataset.py:212-218 (PIL crop + 224x224 BILINEAR resize per detection) and
 * utils/build_util.py:137-142 (ToTensor + Normalize): image uint8 [img_h][img_w][3] (device), boxes int32
 * [n_det][4] = (x1, y1, x2, y2) integer crop boxes (floor/ceil of the detection boxes, taken on the host like the
 * reference; may reach outside the image: PIL pads with 0), row_off int64 [n_det + 1] = prefix sum of the crop
 * heights (y2 - y1), total_rows = row_off[n_det], max_crop_h = largest crop height, mean_std = 6 host floats
 * (mean r,g,b then std r,g,b).  out fp32 [n_det][3][out_size][out_size], bit-identical to the reference's PIL +
 * torchvision result (Pillow 8-bit two-pass resampler reproduced in fixed point).  taps = the filter-tap stride:
 * max over boxes and axes of ceil(max(crop side / out_size, 1)) * 2 + 1, at most mmmot_crop_resize_max_taps().
 */
int mmmot_crop_resize_max_taps(void);
size_t mmmot_crop_resize_workspace(int n_det, long total_rows, int out_size, int taps);
int mmmot_crop_resize(const unsigned char* image, int img_h, int img_w, const int* boxes, const long long* row_off,
                      int n_det, long total_rows, int max_crop_h, int out_size, int taps, const float* mean_std,
                      float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Contraction engine selection: 0 = auto (tcgen05 tensor-core engine for large problems, FP32 FFMA
 * engine for tiny ones), 1 = force the FP32 FFMA engine, 2 = force the tcgen05 engine.  Both engines
 * implement the same contraction; the switch exists for A/B parity tests and profiling. */
int mmmot_set_engine(int engine);

/* Accuracy / speed knob of the tcgen05 conv engine.  The tensor core's fp32 accumulator rounds toward zero at
 * every K=16 step (bias ~ steps * 2^-25), so K chains longer than `chunks` x 32 are accumulated in several
 * TMEM passes whose partial sums are added in fp32 round-to-nearest.  0 = single pass (fastest, end-to-end link
 * error up to 7.9e-5 on the test cases), 36 (default) splits the K >= 2304 layers (error <= 3.9e-5; bound 1e-4),
 * 72 only the K = 4608 layers (6.8e-5). */
int mmmot_set_kseg(int chunks);

/* Profiling experiments on the tcgen05 kernels (tools/stage_times.py, TC_DBG=...): each bit removes one part of
 * the work to show what bounds a kernel, so results are WRONG with any bit set.  Default 0.
 *   bit 0 (1)    skip epilogue work          bit 1 (2)   skip weight loads
 *   bit 2 (4)    skip operand loads          bit 3 (8)   skip MMA issue
 * Returns MMMOT_E_ARG, leaving the flags unchanged, if any other bit is set. */
int mmmot_set_debug(int flags);

/* Test hook: Y[M][S] = W X + bias through the FP32 FFMA engine (engine must be 1); Wt is [K][M] fp32, X is [K][S],
 * all device pointers (Wp / wp_scale are ignored; the tcgen05 engines have the planar / gen hooks below). */
int mmmot_debug_linear(const float* Wt, const void* Wp, float wp_scale, const float* bias, const float* X,
                       float* Y, int M, int K, int S, int engine, void* stream);

/* Test hook of the generated-operand tcgen05 engine (csrc/gemm_gen.cuh, GroupNorm+ReLU producer): with X [S][K] and
 * Y [S][M] fp32 channels-last, Y = relu(X*sc + sh) W^T + bias, sc/sh [K] per input channel (K a multiple of 32,
 * <= 512).  Wp = packed FP16 hi/lo tiles of W [M][K]. */
int mmmot_debug_linear_gen(const void* Wp, float wp_scale, const float* bias, const float* X, const float* sc,
                           const float* sh, float* Y, int M, int K, int S, void* stream);

/* Test hooks of the TMA-fed tcgen05 engine: operands are two FP16 planes (hi, lo), channels-last.
 * linear: Y[rows][M] fp32 = X W^T + bias, X planes [2][rows][K].  conv: 3x3 pad 1 + bias + ReLU on NHWC planes
 * [2][n][H][W][C] -> [2][n][H][W][M] (weights packed with K order (ky*3+kx)*C + ci). */
int mmmot_debug_linear_planar(const void* Wp, float wp_scale, const float* bias, const void* Xhi, float* Y,
                              int M, int K, long rows, void* stream);
int mmmot_debug_conv_planar(const void* Wp, float wp_scale, const float* bias, const void* Xhi, void* Yhi,
                            int n_img, int H, int W, int C, int M, float* kseg_scratch /* fp32 [n*H*W][M] or NULL */,
                            void* stream);

/* Per-launch timing of the hot kernels with CUDA events on the launching stream; used by bench.py's roofline
 * figures.  Every timed launch carries a tag = (stage, layer) — mmmot_timing_tag_count() tags, named by
 * mmmot_timing_tag_name() — and its ALGORITHMIC work (FLOPs; compulsory HBM bytes of that launch).
 * collect_tags() fills arrays of tag_count entries (any may be NULL) with the summed duration (ms), FLOPs, bytes and
 * launch count per tag since the last collect; collect() returns the totals over the 3x3-conv contractions of the
 * VGG trunk (layers 1..12, FLOPs = 2*Cout*9Cin*pixels), the dominant kernels. */
int mmmot_timing_enable(int on);
int mmmot_timing_tag_count(void);
const char* mmmot_timing_tag_name(int tag);
int mmmot_timing_collect_tags(double* ms, double* flop, double* bytes, long* launches);
int mmmot_timing_collect(double* total_ms, double* total_flop, long* launches);

/* counts kernel launches made through this library since process start (bench.py gpu_launches) */
unsigned long long mmmot_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MMMOT_B200_H */
