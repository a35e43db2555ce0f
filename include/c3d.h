/*
 * c3d.h — C ABI of libc3d.so, the B200-native (sm_100a) kernels behind the Cube R-CNN hot path.
 *
 * The reference (facebookresearch/omni3d) is pure Python and has no FFI of its own; every entry
 * point below replaces the third-party native op the reference reaches at the cited call site.
 *
 * Conventions (all entry points):
 *   - plain pointers + sizes; every pointer is DEVICE memory unless the name ends in _host;
 *   - the caller owns every buffer including the workspace (size from the matching
 *     *_workspace_bytes query); kernels never allocate, free or synchronise;
 *   - work is enqueued on `stream` (a cudaStream_t / CUstream handle passed as void*);
 *   - return 0 (C3D_OK) or a negative c3d_status; c3d_last_error() gives a thread-local string.
 */
#ifndef C3D_H_
#define C3D_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  C3D_OK = 0,
  C3D_EINVAL = -1,     /* bad argument (null pointer, negative size, misalignment) */
  C3D_EWORKSPACE = -2, /* workspace too small */
  C3D_ECUDA = -3       /* CUDA launch/runtime error, see c3d_last_error() */
} c3d_status;

const char* c3d_last_error(void);
/* library/ABI version, bumped when a signature changes */
int32_t c3d_abi_version(void);

/* ------------------------------------------------------------------------------------------
 * Oriented-box 3D IoU.
 * Replaces pytorch3d._C.iou_box3d as called at cubercnn/evaluation/omni3d_evaluation.py:155 and
 * the wrapper cubercnn/evaluation/omni3d_evaluation.py:106-166 (box3d_overlap) with its row
 * checks :65-104.  Boxes are (n,8,3) fp32 contiguous, corner order of DATA.md:109-131.
 * ------------------------------------------------------------------------------------------ */

/* workspace for n1 x n2 (cross) or n1 pairs (paired: pass n2 = 0) */
size_t c3d_iou_box3d_workspace_bytes(int64_t n1, int64_t n2);

/* == pytorch3d._C.iou_box3d(boxes1, boxes2) -> (vol, iou), both (n1, n2) fp32 row-major.
 * vol and nfaces may be NULL.  nfaces (int32) = number of triangles of the intersection
 * polyhedron per pair (debug/parity quantity; -1 if the pair exceeded every capacity). */
int32_t c3d_iou_box3d(const float* boxes1, int64_t n1, const float* boxes2, int64_t n2,
                      float* vol, float* iou, int32_t* nfaces,
                      void* workspace, size_t workspace_bytes, void* stream);

/* paired variant: pair k = (boxes1[k], boxes2[k]), outputs (n,) */
int32_t c3d_iou_box3d_paired(const float* boxes1, const float* boxes2, int64_t n,
                             float* vol, float* iou, int32_t* nfaces,
                             void* workspace, size_t workspace_bytes, void* stream);

/* == box3d_overlap(boxes_dt, boxes_gt, eps_coplanar, eps_nonzero) -> iou (n_dt, n_gt) with rows of
 * non-coplanar / zero-area dt boxes zeroed (the reference prints a warning instead of raising,
 * omni3d_evaluation.py:158-164).  n_bad (device int32[2], may be NULL) receives the number of
 * non-coplanar and zero-area dt boxes so the host mirror can print the same warnings. */
int32_t c3d_box3d_overlap(const float* boxes_dt, int64_t n_dt, const float* boxes_gt, int64_t n_gt,
                          float eps_coplanar, float eps_nonzero, float* iou, int32_t* n_bad,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Segmented (CSR) box3d_overlap: `num_groups` independent (detections x ground truths) blocks in ONE launch — replaces the
 * per-(image, category) calls of Omni3Deval.computeIoU (cubercnn/evaluation/omni3d_evaluation.py:1339-1343, 1359-1431,
 * call site :1401-1412).  boxes_dt [n_dt][8][3] / boxes_gt [n_gt][8][3] hold all groups back to back; group g owns dt rows
 * [dt_off[g], dt_off[g+1]) and gt rows [gt_off[g], gt_off[g+1]) (int32 device arrays of num_groups+1 entries); its IoU
 * matrix is written row-major at iou + pair_off[g] (int64 device array, pair_off[g+1]-pair_off[g] = rows x cols,
 * pair_off[num_groups] = total_pairs).  Row checks / n_bad as in c3d_box3d_overlap (over all dt boxes). */
size_t c3d_box3d_overlap_segmented_workspace_bytes(int64_t n_dt, int64_t n_gt, int64_t total_pairs);
int32_t c3d_box3d_overlap_segmented(const float* boxes_dt, int64_t n_dt, const float* boxes_gt, int64_t n_gt,
                                    const int32_t* dt_off, const int32_t* gt_off, const int64_t* pair_off,
                                    int32_t num_groups, int64_t total_pairs, float eps_coplanar, float eps_nonzero,
                                    float* iou, int32_t* n_bad, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * NHWC bf16 implicit-GEMM convolution on tcgen05 tensor cores (TMA-staged, fp32 accumulate in TMEM).
 * Replaces the cuDNN calls behind nn.Conv2d in cubercnn/modeling/backbone/dla.py:43-51,159-161,
 * 211-214,241-243,287-297, the detectron2 FPN convs built at dla.py:500-506 / resnet.py:88-95 and
 * the StandardRPNHead convs (configs/Base.yaml:49).  Data-gradient = the same entry point with
 * flipped/transposed weights; weight-gradient = c3d_conv2d_wgrad.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t N, H, W, Cin;      /* input  (N,H,W,Cin)  bf16, pixel stride x_pix_stride elements (0 => Cin) */
  int32_t Cout, KH, KW;      /* weight (Cout,KH,KW,Cin) bf16 contiguous */
  int32_t stride, pad;       /* stride 1 or 2 (same in h and w), symmetric zero padding */
  int32_t relu;              /* epilogue: max(.,0) after bias/addend */
  int32_t out_fp32;          /* output fp32 instead of bf16 */
  int32_t add_mode;          /* 0 none; 1 addend (N,Ho,Wo,Cout); 2 addend (N,Ho/2,Wo/2,Cout) nearest-up x2 (FPN);
                                3 accumulate in place: y (bf16) += result at the output's own (possibly strided) position */
  int64_t x_pix_stride, y_pix_stride, add_pix_stride;   /* elements; 0 => dense */
  /* optional strided output placement (in pixels): y pixel index = n*y_img_stride + ho*y_h_stride + wo*y_w_stride +
   * y_offset; all 0 => dense (N,Ho,Wo).  Used by the phase-decomposed stride-2 data gradient. */
  int64_t y_img_stride, y_h_stride, y_w_stride, y_offset;
  /* optional explicit output size (0 => (H + 2*pad - KH)/stride + 1): lets a conv pad only on the high side
   * (taps that run past H/W read TMA zero fill) */
  int32_t out_h, out_w;
  /* optional distance between consecutive input images in PIXELS (0 => dense H*W): lets a batch of row blocks of a
   * larger matrix be read in place (the cube head's RoIs are the first Fc of every image's S pooled RoIs) */
  int64_t x_img_stride;
  /* optional split of the output channels over two places of the output tensor: channels >= y_split_c (a multiple of 16)
   * are written y_split_off ELEMENTS further than their position inside the pixel.  Used by the merged stride-2 data
   * gradient: ONE 2x2 convolution of dy produces the 2x2 block of dx pixels of every dy pixel as 4*Cin output channels —
   * (row parity a, column parity b, ci) — the b halves are adjacent pixels, the a halves are W*Cin elements apart.  0 => off */
  int32_t y_split_c, pad_;
  int64_t y_split_off;
} c3d_conv_desc;

/* number of 128-pixel output tiles (= rows of the BatchNorm partial-statistics buffer) and tile shape */
int32_t c3d_conv2d_tiles(const c3d_conv_desc* d, int32_t* tiles_m, int32_t* tile_h, int32_t* tile_w);

/* y = conv(x, w) [+ bias] [+ addend] [relu].  stats (may be NULL): fp32 [tiles_m][2][Cout] per-tile
 * partial (sum, sum of squares) of the raw fp32 conv output, for train-mode BatchNorm. */
int32_t c3d_conv2d_fwd(const c3d_conv_desc* d, const void* x, const void* w, const float* bias,
                       const void* addend, void* y, float* stats, void* stream);

/* dw[Cout][KH][KW][Cin] (fp32) += the weight gradient of the convolution described by d, from the
 * forward input x (N,H,W,Cin) and the output gradient dy (N,Ho,Wo,Cout), both bf16 NHWC.
 * Split-K over pixels with fp32 atomics: the caller zeroes (or pre-loads) dw. */
int32_t c3d_conv2d_wgrad(const c3d_conv_desc* d, const void* x, const void* dy, float* dw, void* stream);
/* same, oihw != 0: dw is the fp32 master-layout gradient [Cout][Cin][KH][KW] (accumulate straight into the
 * optimizer's gradient arena, no layout conversion pass) */
int32_t c3d_conv2d_wgrad_ex(const c3d_conv_desc* d, const void* x, const void* dy, float* dw, int32_t oihw,
                            void* stream);
/* fp32 master weight (OIHW, or OHWI = torch channels_last storage when src_is_ohwi != 0) -> bf16 (Cout,KH,KW,Cin)
 * forward pack and/or bf16 (Cin,KH,KW,Cout) 180-degree-rotated data-gradient pack (either output may be NULL) */
int32_t c3d_pack_conv_weight(const float* w, int32_t Cout, int32_t Cin, int32_t KH, int32_t KW, int32_t src_is_ohwi,
                             void* fwd_ohwi, void* dgrad_ihwo, void* stream);

/* every conv weight of a model in one launch: descs_dev = device array of n c3d_pack_desc (forward pack, rotated /
 * transposed data-gradient pack and, for 3x3 stride-2 layers, the four phase sub-kernels of the phase-decomposed data
 * gradient: (Cin, KH', KW', Cout) with parity 0 -> tap [1], parity 1 -> taps [2, 0]); `start` = prefix sum of elements */
typedef struct {
  const float* src; void* fwd; void* dgrad; void* phase[4];
  int64_t start;
  int32_t Cout, Cin, KH, KW, src_is_ohwi, pad_;
} c3d_pack_desc;
int32_t c3d_pack_conv_weights_batched(const void* descs_dev, int32_t n, int64_t total_elems, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fully-connected layers on the same tcgen05 kernels (bf16 operands, fp32 accumulate in TMEM, bias + ReLU fused).
 * Replace the cuBLAS GEMMs behind nn.Linear in detectron2 FastRCNNConvFCHead / FastRCNNOutputLayers
 * (configs/Base.yaml:67-70, cubercnn/modeling/roi_heads/fast_rcnn.py:119-143) and in CubeHead
 * (cubercnn/modeling/roi_heads/cube_head.py:63-73,108-144,146-197).
 *   x  (rows, K) bf16 row-major; w (N, K) bf16 = nn.Linear.weight; wt (K, N) bf16 = its transpose;
 *   K % 16 == 0, N % 16 == 0 (callers zero-pad the predictors).
 * c3d_pack_linear_weight: fp32 master (N, K) -> bf16 w (N, K') and (optional) wt (K', N).  C * PP == K with PP > 1
 *   re-orders the input features from (c, p) [NCHW-flattened RoI, the reference's layout] to (p, c) [NHWC-flattened RoI].
 * c3d_linear_wgrad: dw (fp32, += with atomics) = dy^T x.  master_chw != 0: dw is addressed in the master's (c, p)
 *   feature order (accumulate straight into the optimizer's gradient arena), else in the packed (p, c) order.
 * ------------------------------------------------------------------------------------------ */
int32_t c3d_pack_linear_weight(const float* w, int32_t N, int32_t K, int32_t C, int32_t PP, void* w_bf16, void* wt_bf16,
                               void* stream);
int32_t c3d_linear_fwd(const void* x, const void* w, const float* bias, void* y, int64_t rows, int32_t K, int32_t N,
                       int32_t relu, int32_t out_fp32, void* stream);
int32_t c3d_linear_dgrad(const void* dy, const void* wt, void* dx, int64_t rows, int32_t N, int32_t K, void* stream);
int32_t c3d_linear_wgrad(const void* x, const void* dy, float* dw, int64_t rows, int32_t K, int32_t N, int32_t C,
                         int32_t PP, int32_t master_chw, void* stream);
/* Row-block variants: the `rows` = nseg * seg_rows feature vectors are nseg blocks of seg_rows consecutive rows that start
 * every seg_stride rows inside a larger (.., K) matrix (x for fwd / wgrad, dx for dgrad); the other operand is dense.
 * The cube head reads the first Fc of every image's S pooled RoIs in place, and its data gradient is ACCUMULATED
 * (accumulate != 0: dx += dy . W) into the box head's — no gather copy, no zero-padded scatter, no add pass. */
int32_t c3d_linear_fwd_blocks(const void* x, const void* w, const float* bias, void* y, int32_t nseg, int32_t seg_rows,
                              int64_t seg_stride, int32_t K, int32_t N, int32_t relu, int32_t out_fp32, void* stream);
int32_t c3d_linear_dgrad_blocks(const void* dy, const void* wt, void* dx, int32_t nseg, int32_t seg_rows, int64_t seg_stride,
                                int32_t N, int32_t K, int32_t accumulate, void* stream);
int32_t c3d_linear_wgrad_blocks(const void* x, const void* dy, float* dw, int32_t nseg, int32_t seg_rows, int64_t seg_stride,
                                int32_t K, int32_t N, int32_t C, int32_t PP, int32_t master_chw, void* stream);

/* ------------------------------------------------------------------------------------------
 * HBM-bound NHWC bf16 kernels around the convolutions.
 * Replace nn.BatchNorm2d(train) + ReLU + residual add (cubercnn/modeling/backbone/dla.py:17,58-66,
 * 168-172), nn.MaxPool2d(2,2) (dla.py:209), GeneralizedRCNN.preprocess_image (rcnn3d.py:46,87) and the
 * SGD step + per-parameter finite check (tools/train_net.py:226-252, cubercnn/solver/build.py:47-56).
 * ------------------------------------------------------------------------------------------ */
/* per-channel batch statistics from the conv epilogue partials [rows][2][C] -> mean, rstd (+ running stats) */
/* scratch (fp64 slab sums) needed by c3d_bn_finalize / c3d_bn_bwd */
size_t c3d_bn_scratch_bytes(int32_t C);
int32_t c3d_bn_finalize(const float* partial, int32_t rows, int32_t C, double count, float eps, float momentum,
                        float* running_mean, float* running_var, float* mean_out, float* rstd_out, void* scratch,
                        void* stream);
/* out = [relu]((y-mean)*rstd*gamma+beta [+ residual]); y,out,residual bf16 (P pixels x C) */
int32_t c3d_bn_apply(const void* y, const float* mean, const float* rstd, const float* gamma, const float* beta,
                     const void* residual, int32_t relu, void* out, int64_t P, int32_t C, int64_t res_stride,
                     int64_t out_stride, void* stream);
/* rows of the `partial` scratch needed by c3d_bn_bwd */
int32_t c3d_bn_bwd_blocks(int64_t P, int32_t C);
/* BatchNorm(+ReLU,+residual) backward: dy (bf16) w.r.t. the conv output, dgamma/dbeta accumulated (+=),
 * optional dres = masked dout for the residual branch. partial: fp32 [blocks][2][C]; coef: fp32 [3][C].
 * frozen_stats != 0: mean/rstd are running statistics (eval mode / freeze_bn, cubercnn/solver/build.py:71-76).
 * out may be NULL for a ReLU layer WITHOUT residual when beta is given: the mask is then recomputed from y exactly as
 * c3d_bn_apply produced it (saves re-reading `out` in both passes).
 * `relu` is a flag word: bit 0 = the layer has a ReLU, bit 1 = dres ACCUMULATES (dres += masked dout, fp32 add): the
 * residual tensor's gradient buffer already holds its other consumers' contributions (what autograd's AccumulateGrad /
 * add of dla.py:58-66's `out += residual` does with a separate pass). */
int32_t c3d_bn_bwd(const void* dout, const void* out, const void* y, const float* mean, const float* rstd,
                   const float* gamma, const float* beta, int32_t relu, int32_t frozen_stats, float* partial, float* coef, float* dgamma,
                   float* dbeta,
                   void* dy, void* dres, int64_t P, int32_t C, int64_t dout_stride, int64_t out_stride,
                   int64_t dres_stride, void* scratch, void* stream);
/* backward of the bias(+ReLU) epilogue of the bias convs (FPN / RPN head): dz (bf16) = dout * (out > 0 if relu),
 * dbias (fp32 [C]) += sum over pixels.  dtype_flags: bit 0 = dout is fp32 (else bf16), bit 1 = out is fp32 (else bf16).
 * partial: fp32 [c3d_bn_bwd_blocks(P,C)][C]; scratch: c3d_bn_scratch_bytes(C).
 * dz may be NULL when relu == 0 and dout is bf16: dz would equal dout (the FPN convs have no activation) and only the
 * bias gradient is computed — half of the pass's HBM traffic. */
int32_t c3d_bias_act_bwd(const void* dout, const void* out, int32_t relu, int32_t dtype_flags, void* dz, float* partial,
                         float* dbias, int64_t P, int32_t C, void* scratch, void* stream);
/* y (N,H/2,W/2,C) = 2x2 block sums of x: gradient of the FPN nearest-x2 upsampling */
int32_t c3d_sumpool2(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
/* z (N,H,W,C) = dy (N,Ho,Wo,C) at even positions, zero elsewhere: input of a stride-2 conv's data gradient */
int32_t c3d_zero_stuff2(const void* dy, void* z, int32_t N, int32_t Ho, int32_t Wo, int32_t H, int32_t W, int32_t C,
                        void* stream);
int32_t c3d_maxpool2_fwd(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, int64_t x_stride,
                         int64_t y_stride, void* stream);
int32_t c3d_maxpool2_bwd(const void* x, const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C,
                         int64_t x_stride, int64_t dy_stride, void* stream);
/* same, accumulating: dx (pixel stride dx_stride, 0 => C) += routed dy — x feeds the pool AND a strided convolution
 * (dla.py:209-214), the pool's share is added into the convolution's data gradient in place */
int32_t c3d_maxpool2_bwd_acc(const void* x, const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C,
                             int64_t x_stride, int64_t dy_stride, int64_t dx_stride, void* stream);
/* 3x3 / stride 2 / pad 1 max pool of the torchvision ResNet stem (cubercnn/modeling/backbone/resnet.py:17-27,45-50):
 * y (N,(H-1)/2+1,(W-1)/2+1,C); the backward routes dy to the first maximal element of every window (ATen tie order). */
int32_t c3d_maxpool3s2_fwd(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int32_t c3d_maxpool3s2_bwd(const void* x, const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C,
                           int64_t dy_stride, void* stream);
/* (3,H,W) fp32 BGR image -> (Hp,Wp,Cp) bf16 NHWC slot: (x-mean)/std in channels 0..2, zeros elsewhere */
int32_t c3d_preprocess_image(const float* img, int32_t H, int32_t W, void* out_slot, int32_t Hp, int32_t Wp,
                             int32_t Cp, const float* mean3_host, const float* std3_host, void* stream);
/* all N images of a batch in one launch: imgs_host / H_host / W_host are HOST arrays (device pointers, sizes) that travel in
 * the kernel parameters; out = (N,Hp,Wp,Cp) bf16; is_u8 selects uint8 or fp32 (3,H,W) inputs */
int32_t c3d_preprocess_batch(const void* const* imgs_host, const int32_t* H_host, const int32_t* W_host, int32_t N,
                             int32_t is_u8, void* out, int32_t Hp, int32_t Wp, int32_t Cp, const float* mean3_host,
                             const float* std3_host, void* stream);
/* same for the uint8 (3,H,W) image tensor detectron2's DatasetMapper produces (dataset_mapper.py: image as uint8) */
int32_t c3d_preprocess_image_u8(const uint8_t* img, int32_t H, int32_t W, void* out_slot, int32_t Hp, int32_t Wp,
                                int32_t Cp, const float* mean3_host, const float* std3_host, void* stream);
/* flag |= 1 if any gradient element is NaN/Inf */
int32_t c3d_grad_finite(const float* g, int64_t n, int32_t* flag, void* stream);
/* torch.optim.SGD(momentum, weight_decay) over a flat arena; no-op if *skip_flag != 0 */
int32_t c3d_sgd_momentum(float* p, const float* g, float* mom, int64_t n, float lr, float momentum,
                         float weight_decay, float grad_scale, const int32_t* skip_flag, void* stream);
/* same update with the learning rate read from device memory at run time (schedule changes without re-recording a
 * captured CUDA graph of the step) */
int32_t c3d_sgd_momentum_dev(float* p, const float* g, float* mom, int64_t n, const float* lr_dev, float momentum,
                             float weight_decay, float grad_scale, const int32_t* skip_flag, void* stream);

/* ------------------------------------------------------------------------------------------
 * Multi-level ROIAlign (aligned=True, sampling_ratio 0) on NHWC bf16 FPN maps.
 * Replaces detectron2 ROIPooler/ROIAlignV2 at cubercnn/modeling/roi_heads/roi_heads.py:267,362.
 * rois: fp32 [R][6] = (batch index, level index, x1, y1, x2, y2).  out: bf16 [R][ph][pw][C].
 * RoIs with a non-finite coordinate, a level outside [0, num_levels) or (when num_images > 0) an image index
 * outside [0, num_images) pool zeros / contribute no gradient instead of indexing out of bounds.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  const void* feat[5];   /* level l: bf16 (N,H[l],W[l],C) */
  void* grad[5];         /* backward only: fp32 (N,H[l],W[l],C), accumulated with atomics */
  int32_t H[5], W[5];
  float scale[5];
  int32_t num_levels;
  int32_t num_images;    /* N of the maps (0 = do not check the image index) */
} c3d_roi_levels;
int32_t c3d_roi_align_fwd(const c3d_roi_levels* levels, const float* rois, int32_t R, int32_t C, int32_t pooled_h,
                          int32_t pooled_w, void* out, void* stream);
int32_t c3d_roi_align_bwd(const c3d_roi_levels* levels, const float* rois, int32_t R, int32_t C, int32_t pooled_h,
                          int32_t pooled_w, const void* dout, void* stream);

/* ------------------------------------------------------------------------------------------
 * Batched greedy NMS (all images, two launches, no host sync).
 * Replaces torchvision nms behind detectron2 batched_nms in find_top_rpn_proposals (SURVEY A.3;
 * configs/Base.yaml:51-54).  boxes: fp32 [B][n][4] sorted by score desc per image (already shifted by the
 * per-level coordinate-trick offsets), nvalid[B] valid candidates.  keep_idx: int32 [B][max_keep] indices
 * into the sorted list in score order (-1 padded); keep_cnt[B].  n <= 8192.
 * cats (fp32 [B][n], may be NULL) = per-box category (FPN level); maxc (fp32 [B]) = per-image max coordinate:
 * images with 4*nvalid <= trick_max_numel use torchvision's coordinate trick (shift by cat*(maxc+1)),
 * larger ones plain same-category suppression — the two code paths of torchvision.ops.batched_nms.
 * ------------------------------------------------------------------------------------------ */
size_t c3d_nms_workspace_bytes(int32_t B, int32_t n);
int32_t c3d_nms_batched(const float* boxes, const int32_t* nvalid, const float* cats, const float* maxc,
                        int32_t trick_max_numel, int32_t B, int32_t n, float iou_thresh,
                        int32_t max_keep, int32_t* keep_idx, int32_t* keep_cnt, void* workspace,
                        size_t workspace_bytes, void* stream);
/* same result when the caller knows the categories are the integers 0..ncat-1 (ncat <= 16; boxes with another value are
 * dropped): candidates are split per category first, so suppression tiles and the greedy scans run inside a category
 * only.  max_per_cat_hint (0 = unknown) sizes the tile grid (performance only). */
int32_t c3d_nms_batched_grouped(const float* boxes, const int32_t* nvalid, const float* cats, const float* maxc,
                                int32_t trick_max_numel, int32_t B, int32_t n, float iou_thresh, int32_t max_keep,
                                int32_t ncat, int32_t max_per_cat_hint, int32_t* keep_idx, int32_t* keep_cnt,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * RPN anchor <-> ground-truth matching for a whole batch (two passes, GT boxes of an image in shared memory).
 * Replaces detectron2 pairwise_iou + Matcher(thresholds, allow_low_quality_matches=True) and the ignore-region IoA
 * of cubercnn/modeling/proposal_generator/rpn.py:93-105 (label_and_sample_anchors), :286-330.
 *   anchors [A][4], gt_boxes [B][G][4] (x1,y1,x2,y2 fp32, padded), gt_valid / gt_ign [B][G] (0/1 bytes)
 *   matched_idx [B][A] int64: first GT of maximal IoU among valid ones (0 if none)
 *   matched_iou [B][A]: that IoU (0 if none);  max_ioa [B][A]: max over ignore regions of inter / anchor area
 *   labels [B][A] int8: 1 if IoU >= fg_thresh or the anchor attains the maximum IoU of some valid GT, else 0
 *   best_idx [B][G] int32: first anchor attaining that GT's maximum (A for non-valid GTs)
 *   rowmax_ws [B][G] int32 scratch.  Bit-identical to the fp32 torch formulation (explicit rn arithmetic).
 * ------------------------------------------------------------------------------------------ */
int32_t c3d_anchor_match(const float* anchors, int64_t A, const float* gt_boxes, const uint8_t* gt_valid,
                         const uint8_t* gt_ign, int32_t B, int32_t G, float fg_thresh, int64_t* matched_idx,
                         float* matched_iou, int8_t* labels, float* max_ioa, int32_t* best_idx, int32_t* rowmax_ws,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * RPN objectness + localisation losses over all B*A anchors, one pass forward and one backward
 * (cubercnn/modeling/proposal_generator/rpn.py:108-218: IoU-ness objectness targets, both terms weighted by the target
 * and restricted to positive anchors).  logits [B][A], deltas [B][A][4], labels int8 [B][A] in {-1,0,1},
 * matched_idx int64 [B][A], gt_boxes [B][G][4], anchors [A][4], weights4_host = BBOX_REG_WEIGHTS.
 *   fwd: acc6 = {sum cls, sum loc, #pos, #neg, sum sigmoid(pos), sum sigmoid(non-pos)} (un-normalised)
 *   bwd: dlogits / ddeltas (dense, zero off the positives) scaled by the device scalars *g_cls / *g_loc
 * ------------------------------------------------------------------------------------------ */
int32_t c3d_rpn_loss_fwd(const float* logits, const float* deltas, const int8_t* labels, const int64_t* matched_idx,
                         const float* gt_boxes, const float* anchors, int32_t B, int64_t A, int32_t G,
                         const float* weights4_host, float* acc6, void* stream);
int32_t c3d_rpn_loss_bwd(const float* logits, const float* deltas, const int8_t* labels, const int64_t* matched_idx,
                         const float* gt_boxes, const float* anchors, int32_t B, int64_t A, int32_t G,
                         const float* weights4_host, const float* g_cls, const float* g_loc, float* dlogits,
                         float* ddeltas, void* stream);

/* RPN proposal decoding of one FPN level's top-k candidates for all images (apply_deltas, clip, finite / min-size
 * filter; detectron2 find_top_rpn_proposals via rpn.py:221-284).  topk_idx / topk_score [B][K] (rows in_stride elements
 * apart; 0 => K) index the level's anchors [A][4] and deltas [B][A][4]; image_hw [B][2] = (h, w).  Results go to columns col0..col0+K-1 of the
 * concatenated [B][Ktot] arrays: boxes (xyxy), key (score, or -inf when filtered), lvl (= level as float); nvalid[b] and
 * maxc[b] (max kept coordinate, fp32 bits; both zero-initialised by the caller) are accumulated with atomics. */
int32_t c3d_rpn_decode_level(const int64_t* topk_idx, const float* topk_score, int64_t in_stride, const float* deltas,
                             const float* anchors, const float* image_hw, int32_t B, int32_t K, int64_t A, const float* weights4_host,
                             float scale_clamp, float min_size, int32_t level, int32_t col0, int32_t Ktot, float* boxes,
                             float* key, float* lvl, int32_t* nvalid, float* maxc, void* stream);

/* ------------------------------------------------------------------------------------------
 * CubeHead decode + disentangled 3D corner losses, fused forward / backward (one thread per RoI).
 * Replaces the ATen micro-kernels of cubercnn/modeling/roi_heads/roi_heads.py:409-525 (decode) and :527-740
 * (xy / z / dims L1 corner losses, chamfer pose + joint losses, sqrt(2)*exp(-u) weighting), with
 * math_util.py:116-219,651-679 and pytorch3d rotation_6d_to_matrix inlined.
 *   raw  fp32 [n][13]: delta x,y | z | dims W,H,L | pose6 | uncertainty   (per-class-gathered head outputs)
 *   aux  fp32 [n][28]: box x1,y1,x2,y2 | fx,fy,px,py | virtual->real | prior W,H,L | gt u,v,z,W,H,L | gt R (9) | pad
 *   out  fp32 [n][10]: u, l_dims*sf, l_xy*sf, l_z*sf, l_pose*sf, l_joint*sf, |z-gz|, mean|dims-gt|, mean|xy-gt|, exp(-u)
 *   dout fp32 [n][6] : upstream gradient of out[:, 0:6];  draw fp32 [n][13]
 * ------------------------------------------------------------------------------------------ */
int32_t c3d_cube_loss_fwd(const float* raw, const float* aux, int32_t n, float* out, void* stream);
int32_t c3d_cube_loss_bwd(const float* raw, const float* aux, const float* dout, int32_t n, float* draw, void* stream);

/* ------------------------------------------------------------------------------------------
 * Selection / sampling kernels of the RPN and ROI-head glue (omni3d_b200/csrc/select_ops.cu).
 * ------------------------------------------------------------------------------------------ */
/* Sorted (descending) top-k of `nseg` row segments per image in ONE launch (grid B x nseg): the per-level pre-NMS top-k
 * of detectron2 find_top_rpn_proposals (via cubercnn/modeling/proposal_generator/rpn.py:221-284, configs/Base.yaml:51-54),
 * the score sort of the concatenated candidates (k == n), the top-M of the inference candidates (fast_rcnn.py:57-116).
 * Segment s of image b reads vals + b*row_stride [0, n) and writes its k results (value, index inside the segment) to
 * columns [out_col, out_col + k) of row b of out_vals / out_idx / out_idx64 (row length out_stride); k <= 8192.
 * Ties: equal values come out in ascending index order; WHICH of more-than-needed equal values are taken is unspecified
 * (as for torch.topk).  out_count [B][nseg] (may be NULL) = number of selected values > -inf. */
typedef struct {
  const float* vals;
  int64_t row_stride;
  int32_t n, k, out_col;
} c3d_topk_seg;
int32_t c3d_topk_segments(const c3d_topk_seg* segs, int32_t nseg, int32_t B, int32_t out_stride, float* out_vals,
                          int32_t* out_idx, int64_t* out_idx64, int32_t* out_count, void* stream);

/* ROIHeads3D.label_and_sample_proposals (cubercnn/modeling/roi_heads/roi_heads.py:826-929), one image per block:
 * matcher ([IOU_THRESHOLD] / labels [0,1]) over [proposals | appended valid GT], ignore-region rule (background proposals
 * with IoA >= ignore_thresh become -1 when the image has > 1 background proposals), IoU-weighted sampling WITHOUT
 * replacement of <= Fcap foreground and the remaining background proposals (Gumbel top-k on a Philox stream: the same
 * distribution as torch.multinomial(iou + 1e-4), rpn.py:275-328), foreground-first compaction into S slots and the gather
 * of the matched GT fields.  P + G <= 2048, G <= 256.  rng = {seed, step counter} on the device (bump_rng != 0: the
 * counter is incremented afterwards, so a replayed CUDA graph draws fresh noise every step).
 * Pre-sampling outputs (all three or none) are [B][P+G]: matched GT index, matched IoU (>= 0), class label
 * (K = background, -1 = ignore / padding).  Sampled outputs are [B][S]. */
typedef struct {
  const float* prop_boxes;      /* [B][P][4] */
  const int32_t* prop_count;    /* [B] */
  const float* gt_boxes;        /* [B][G][4] */
  const int64_t* gt_classes;    /* [B][G], < 0 = ignore region */
  const uint8_t* gt_present;    /* [B][G] */
  const float* gt_boxes3D;      /* [B][G][9] */
  const float* gt_poses;        /* [B][G][9] */
  int32_t B, P, G, K, S, Fcap, append_gt;
  float iou_thresh, ignore_thresh;
  const uint64_t* rng;
  int32_t bump_rng;
  int64_t* matched_idx; float* matched_iou; int64_t* labels;
  float* s_boxes; uint8_t* s_valid; int64_t* s_classes; float* s_gt_boxes; float* s_gt_boxes3D; float* s_gt_poses;
  int64_t* s_index;             /* index into [proposals | GT] of every slot (may be NULL) */
  float* stats;                 /* [2] += (#foreground, #background samples) over the batch (may be NULL) */
} c3d_label_sample_args;
int32_t c3d_label_sample_proposals(const c3d_label_sample_args* args, void* stream);

/* RPNWithIgnore.label_and_sample_anchors, sampling part (rpn.py:62-105, 275-328), around c3d_topk_segments:
 *   keys   [B][2][A]: Gumbel keys of the positive (labels01 == 1) / negative (== 0) anchors, -inf elsewhere;
 *          counts [B][2] = number of positive / negative candidates
 *   finish: out_labels [B][A] int8 = -1, sampled negatives 0 (-1 when inside an ignore region and > 1 negatives were
 *          sampled), sampled positives 1, the best anchor of every valid GT 1.  topk_idx [B][2][k] from the top-k of keys. */
int32_t c3d_anchor_sample_keys(const int8_t* labels01, const float* matched_iou, int32_t B, int64_t A, const uint64_t* rng,
                               float* keys, int32_t* counts, void* stream);
int32_t c3d_anchor_sample_finish(const int8_t* labels01, const float* max_ioa, const int32_t* topk_idx, const int32_t* counts,
                                 const int32_t* best_idx, const uint8_t* gt_valid, const uint8_t* gt_ign, int32_t B, int32_t G,
                                 int64_t A, int32_t k, int32_t cap_pos, int32_t n_total, float ignore_thresh,
                                 int8_t* out_labels, uint64_t* rng_bump, void* stream);

/* Inference post-processing before the NMS (cubercnn/modeling/roi_heads/fast_rcnn.py:76-100) for all images of a batch:
 * probs [B][P][K+1] (softmax scores, last = background), boxes [B][P][K][4] (per-class decoded boxes, unclipped),
 * prop_count [B], image_hw [B][2].  Proposals with any non-finite score / coordinate are dropped, boxes are clipped to
 * the image, (proposal p, class k) pairs with score > score_thresh become candidates at index p*K + k:
 * cand_score [B][P*K] (-inf = not a candidate), cand_boxes [B][P*K][4], maxc [B] = max candidate coordinate,
 * total [B] = number of candidates.  Followed by c3d_topk_segments + c3d_nms_batched (per-class) + top-100. */
int32_t c3d_det_candidates(const float* probs, const float* boxes, const int32_t* prop_count, const float* image_hw,
                           int32_t B, int32_t P, int32_t K, float score_thresh, float* cand_score, float* cand_boxes,
                           float* maxc, int32_t* total, void* stream);

/* ------------------------------------------------------------------------------------------
 * Loss assembly of the ROI heads (omni3d_b200/csrc/head_loss_ops.cu).
 * ------------------------------------------------------------------------------------------ */
/* FastRCNNOutputs.losses (cubercnn/modeling/roi_heads/fast_rcnn.py:145-194, box_reg_loss :196-260) on the fused predictor
 * rows pred [R][ld] fp32 = [K+1 class scores | 4K class-specific deltas | pad]: classes int64 [R] (K = background, -1 =
 * ignored), valid uint8 [R], boxes / gt_boxes [R][4], Box2BoxTransform weights (host, 4 floats).
 * acc [8] = sum CE(valid), sum L1(fg), #valid, #fg, #argmax==class (valid), #argmax==class (fg), #argmax==K (fg), 0.
 * bwd: dpred [R][ld] from g2 = {dL/dloss_cls, dL/dloss_box_reg} (both losses are normalised by #valid). */
int32_t c3d_box_loss_fwd(const float* pred, int32_t ld, const int64_t* classes, const uint8_t* valid, const float* boxes,
                         const float* gt_boxes, int32_t R, int32_t K, const float* weights4_host, float* acc8, void* stream);
int32_t c3d_box_loss_bwd(const float* pred, int32_t ld, const int64_t* classes, const uint8_t* valid, const float* boxes,
                         const float* gt_boxes, int32_t R, int32_t K, const float* weights4_host, const float* acc8,
                         const float* g2, float* dpred, void* stream);
/* Glue around c3d_cube_loss_fwd/bwd (cubercnn/modeling/roi_heads/roi_heads.py:372-461, 690-743, 932-941):
 *  gather : pred [n][ld] fp32 = [deltas 2K | dims 3K | pose 6K | z K | uncertainty K | pad] -> the predicted class's raw13
 *           rows and the aux28 constants (box, K / ratio, virtual->real depth, dims prior, GT) ; meta12 [B][12] = h, w,
 *           height/h, K (9); RoI i belongs to image i / per_image; priors [K][3]
 *  reduce : rows10 [n][10] -> sums12 (11 used: 6 finite-masked loss sums, |dz|, dims err, xy err, #(|dz|<0.2), conf) and
 *           cnts8 (6 finite counts + #valid); its backward gives d rows [n][6]
 *  scatter: d raw13 -> the class's columns of d pred [n][ld] (zero elsewhere) */
int32_t c3d_cube_gather(const float* pred, int32_t ld, const int64_t* classes, const float* boxes, const float* meta12,
                        const float* priors, const float* gt3, const float* gtR, int32_t n, int32_t per_image, int32_t K,
                        float virtual_focal, float* raw13, float* aux28, void* stream);
int32_t c3d_cube_reduce_fwd(const float* rows10, const uint8_t* valid, int32_t n, float* sums12, float* cnts8, void* stream);
int32_t c3d_cube_reduce_bwd(const float* rows10, const uint8_t* valid, int32_t n, const float* cnts8, const float* g6,
                            float* drows6, void* stream);
int32_t c3d_cube_scatter(const float* draw13, const int64_t* classes, int32_t n, int32_t K, int32_t ld, float* dpred,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * Input pipeline, image part (omni3d_b200/csrc/augment_ops.cu): Pillow-exact 8-bit bilinear resize + horizontal flip +
 * HWC -> CHW — what detectron2's ResizeShortestEdge / RandomFlip do on the CPU inside DatasetMapper3D
 * (cubercnn/data/dataset_mapper.py:22-35).  img_hwc [H][W][C] uint8 -> out_chw [C][new_h][new_w] uint8.
 * bounds_* [out][2] = (first input index, tap count), kk_* [out][ksize] = 22-bit fixed-point weights, computed on the host
 * like Pillow's precompute_coeffs / normalize_coeffs_8bpc; row_first/row_last = input rows the vertical pass reads;
 * tmp_hwc [H][new_w][C] scratch.  Bit-identical to Image.resize((new_w,new_h), BILINEAR) (+ [:, ::-1] when flip). */
int32_t c3d_resize_bilinear_u8(const uint8_t* img_hwc, int32_t H, int32_t W, int32_t C, const int32_t* bounds_h,
                               const int32_t* kk_h, int32_t ksize_h, const int32_t* bounds_v, const int32_t* kk_v,
                               int32_t ksize_v, int32_t new_h, int32_t new_w, int32_t row_first, int32_t row_last,
                               int32_t flip, uint8_t* tmp_hwc, uint8_t* out_chw, void* stream);

/* ------------------------------------------------------------------------------------------
 * Omni3D AP evaluation (omni3d_b200/csrc/eval_ops.cu): Omni3Deval.evaluate / accumulate of
 * cubercnn/evaluation/omni3d_evaluation.py:1172-1313, 1315-1357, 1433-1551 for every (image, category) group at once.
 * ------------------------------------------------------------------------------------------ */
/* Greedy matching, replacing the per-(category, range, image) evaluateImg calls (:1347-1352, loop :1489-1536).
 * Groups are back to back: group g owns detections [dt_off[g], dt_off[g+1]) — already sorted by -score (stable) and
 * truncated to maxDets[-1] — and ground truths [gt_off[g], gt_off[g+1]) in annotation order (int32 [num_groups+1]).
 *   dt_box / gt_box [n][4] fp64 XYWH; dt_rng / gt_rng [n] fp64 = area (2D) or depth (3D); gt_ignore [n_gt] (0/1);
 *   gt_id [n_gt] int64 annotation ids.  mode3d != 0: IoU = (double) iou3d[pair_off[g] + d * ng + j], the packed fp32
 *   matrices of c3d_box3d_overlap_segmented over the same groups; else pycocotools bbIou (iscrowd 0) in fp64.
 *   eval_prox != 0: a GT is a candidate only if bbIou(dt, gt) > prox_thresh, a detection with no such GT is ignored.
 *   iou_start_host [T] = min(iouThrs[t], 1 - 1e-10); ranges_host [A][2] = inclusive bounds (HOST arrays; A <= 8, T <= 16).
 * Outputs, chain c = a * T + t:  match [A*T][n_dt] int32 = matched GT row (global index) or -1;
 *   flags [A*T][n_dt] uint8 = bit 0 dtIgnore, bit 1 dtMatches != 0 (the matched GT's id is non-zero);
 *   npig [num_groups][A] int32 = number of non-ignored GTs.  Workspace: c3d_eval_match_workspace_bytes(n_gt, A, T). */
size_t c3d_eval_match_workspace_bytes(int64_t n_gt, int32_t A, int32_t T);
int32_t c3d_eval_match(int32_t mode3d, int32_t eval_prox, int32_t num_groups, int32_t A, int32_t T,
                       const int32_t* dt_off, const int32_t* gt_off, const double* dt_box, const double* dt_rng,
                       const double* gt_box, const double* gt_rng, const uint8_t* gt_ignore, const int64_t* gt_id,
                       const float* iou3d, const int64_t* pair_off, int64_t n_dt, int64_t n_gt,
                       const double* iou_start_host, const double* ranges_host, double prox_thresh, int32_t* match,
                       uint8_t* flags, int32_t* npig, void* workspace, size_t workspace_bytes, void* stream);
/* Precision / recall / score tables, replacing the (category, range, maxDet, threshold) loops of accumulate (:1227-1299).
 * Category k sums npig over the groups [grp_off[k], grp_off[k+1]) (rows of npig [.][A]) and owns the entries
 * [ent_off[k], ent_off[k+1]) (int32 [K+1]), sorted by -score (stable over image order, then per-group rank): entry e is
 * column ent_idx[e] of flags [A*T][n_dt] (as c3d_eval_match writes it), with per-group rank ent_rank[e] and score
 * ent_score[e] (fp64).  rec_thrs [R] fp64 and max_dets [M] int32 are device arrays; T * M <= 64.
 * precision / scores [T][R][K][A][M] and recall [T][K][A][M] (fp64) are written in full, -1 where npig == 0.  No workspace. */
int32_t c3d_eval_accumulate(int32_t K, int32_t A, int32_t T, int32_t M, int32_t R, const int32_t* grp_off,
                            const int32_t* npig, const int32_t* ent_off, const int32_t* ent_idx, const int32_t* ent_rank,
                            const double* ent_score, const uint8_t* flags, int64_t n_dt, const double* rec_thrs,
                            const int32_t* max_dets, double* precision, double* recall, double* scores, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* C3D_H_ */
