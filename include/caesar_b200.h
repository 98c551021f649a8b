/* caesar_b200.h — C ABI of libcaesar_b200.so, the B200 (sm_100a) implementation of caesar-yolo's tiled
 * source-finding hot path.  Plain pointers and sizes only; every pointer is a DEVICE pointer owned by the
 * caller unless the parameter name ends in _host.  Every function returns CY_OK (0) or a negative status and
 * never throws; cy_last_error() returns the message for the calling thread.  `stream` is a cudaStream_t
 * passed as uintptr_t (0 = legacy default stream).
 *
 * The reference (SKA-INAF/caesar-yolo) is pure Python and has no FFI; each entry point cites the reference
 * Python interface it replaces (file:line relative to the reference tree).
 */
#ifndef CAESAR_B200_H
#define CAESAR_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CY_OK 0
#define CY_ERR_INVALID (-1)
#define CY_ERR_CUDA (-2)
#define CY_ERR_NOMEM (-3)
#define CY_ERR_STATE (-4)

/* ------------------------------------------------------------------------------------------------ types */

/* One tile of utils.generate_tiles (caesar_yolo/utils.py:622-697): xmax/ymax are EXCLUSIVE. */
typedef struct { int32_t xmin, xmax, ymin, ymax; } cy_tile;

/* Per-tile detection after Analyzer.make_json_results (caesar_yolo/evaluation.py:418-469): integer-truncated
 * coordinates + tile origin (stored as float like the reference), flags bit0 = edge.  32 bytes: this is the
 * fixed record exchanged between GPUs (replaces the pickled dicts of inference.py:936-984). */
typedef struct { float x1, y1, x2, y2, score; int32_t cls, tile_id, flags; } cy_det_record;

/* Final catalog entry (SFinder.merge_edge_sources, caesar_yolo/inference.py:731-931).
 * flags bit0 = edge, bit1 = merged; tile_id = -1 for merged sources. */
typedef struct { float x1, y1, x2, y2, score; int32_t cls, flags, tile_id; } cy_source;

/* ultralytics LetterBox / scale_boxes geometry of one tile (SURVEY App. A.4/A.6). */
typedef struct { float gain, pad_x, pad_y; int32_t w0, h0; } cy_letterbox;

/* Preprocessing stage list = scripts/run.py:272-293 (fixed order), parameters = run.py:80-107 options. */
typedef struct {
    int32_t subtract_bkg;        double sigma_bkg;  int32_t use_box_mask_in_bkg;  double bkg_box_mask_fract;
    int32_t bkg_chid;
    int32_t clip_shift_data;     double sigma_clip; int32_t clip_chid;
    int32_t clip_data;           double sigma_clip_low, sigma_clip_up;
    int32_t nchannels;           /* ChanResizer target (input cube always has 3 identical channels) */
    int32_t zscale_stretch;      double zscale_contrasts[3];
    int32_t chan3_preproc;       double sigma_clip_baseline;
    int32_t normalize_minmax;    double norm_min, norm_max;
    int32_t enabled;             /* --preprocessing: 0 => the whole chain is skipped (dp = None) */
    int32_t out_f16;             /* model_in format: 0 = bf16, 1 = fp16 (must match cy_model_set_precision) */
} cy_pp_config;

/* General preprocessing chain = caesar_yolo/preprocessing.py's DataPreprocessor(stages) for ANY stage order
 * (preprocessing.py:47-67): a list of stage records interpreted by the chain kernel.  Stage parameters:
 *   BKG_SUB          p0 sigma, flag use_mask_box, p1 mask_fract, chid                          (:591-658)
 *   CLIP_SHIFT       p0 sigma, chid                                                            (:664-717)
 *   SIGMA_CLIP       p0 sigma_low, p1 sigma_up, chid                                           (:723-771)
 *   CHAN_RESIZE      n nchans (1 or 3: the cube Analyzer.predict builds already has 3 channels) (:1077-1133)
 *   ZSCALE           p0..p2 contrasts, n = number of contrasts given (< 3 => every tile rejected, :955-957) (:934-971)
 *   CHAN3            p0 sigma_clip_baseline, p1 sigma_clip_low, p2 sigma_clip_up, p3 zscale_contrast (:1020-1072)
 *   MINMAX           p0 norm_min, p1 norm_max                                                  (:75-111)
 *   ABS_MINMAX       p0 norm_min, p1 norm_max                                                  (:116-146)
 *   MAX_SCALE        -                                                                         (:152-176)
 *   ABS_MAX_SCALE    flag use_mask_box, p0 mask_fract                                          (:182-226)
 *   CHAN_MAX_SCALE   n chref, flag use_mask_box, p0 mask_fract                                 (:232-288)
 *   MIN_SHIFT        chid                                                                      (:294-327)
 *   SHIFT            p0..p2 offsets, n = number given (!= 3 => every tile rejected)            (:333-363)
 *   STANDARDIZE      p0..p2 means, p3..p5 sigmas, n = min(len(means), len(sigmas)) (!= 3 => rejected) (:369-402)
 *   NEG_FIX          -                                                                         (:408-440)
 *   LOG_STRETCH      chid = EXCLUDED channel (-1 none), flag bit0 minmaxnorm (required), bit1 clip_neg,
 *                    p0 data_norm_min, p1 data_norm_max                                        (:480-538)
 *   BORDER_MASK      p0 mask_fract; only before any stage that computes statistics             (:544-586)
 *   HISTEQ           - (non-adaptive)                                                          (:977-1012)
 * chid = -1: all channels. */
enum {
    CY_PP_BKG_SUB = 1, CY_PP_CLIP_SHIFT = 2, CY_PP_SIGMA_CLIP = 3, CY_PP_CHAN_RESIZE = 4, CY_PP_ZSCALE = 5,
    CY_PP_CHAN3 = 6, CY_PP_MINMAX = 7, CY_PP_ABS_MINMAX = 8, CY_PP_MAX_SCALE = 9, CY_PP_ABS_MAX_SCALE = 10,
    CY_PP_CHAN_MAX_SCALE = 11, CY_PP_MIN_SHIFT = 12, CY_PP_SHIFT = 13, CY_PP_STANDARDIZE = 14, CY_PP_NEG_FIX = 15,
    CY_PP_LOG_STRETCH = 16, CY_PP_BORDER_MASK = 17, CY_PP_HISTEQ = 18
};
#define CY_PP_MAX_STAGES 16
typedef struct { int32_t type, chid, flag, n; double p[8]; } cy_pp_stage;
typedef struct {
    int32_t nstages;
    int32_t out_f16;       /* model_in format: 0 = bf16, 1 = fp16 */
    int32_t reject_all;    /* set by cy_pp_chain_validate: the reference returns None for every image */
    int32_t reserved;
    cy_pp_stage st[CY_PP_MAX_STAGES];
} cy_pp_chain;

const char* cy_last_error(void);
int cy_version(void);
/* CY_OK iff the current device is sm_100. */
int cy_device_check(void);
/* cudaMemcpyAsync device->device on `stream` (lets hosts without a CUDA binding read library-owned buffers). */
int cy_memcpy_d2d(void* dst, const void* src, size_t nbytes, uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ tiling (host)
 * utils.generate_tiles (caesar_yolo/utils.py:622-697).  tiles_host == NULL: size query (ntiles only). */
int cy_generate_tiles(int img_xmin, int img_xmax, int img_ymin, int img_ymax, int tile_x, int tile_y, double step_x,
                      double step_y, cy_tile* tiles_host, int capacity, int* ntiles_host);
/* Neighbour lists of SFinder.create_tile_tasks (caesar_yolo/inference.py:1034-1071, predicates :123-163) as CSR,
 * ascending tile id, self excluded; nb_off_host has T+1 entries; nb_idx_host == NULL: size query. */
int cy_tile_neighbors(const cy_tile* tiles_host, int T, int* nb_off_host, int* nb_idx_host, int capacity,
                      int* total_host);

/* ------------------------------------------------------------------------------------------------ preprocessing
 * DataPreprocessor chain of caesar_yolo/preprocessing.py (BkgSubtractor :591-658, SigmaClipShifter :664-717,
 * SigmaClipper :723-771, ChanResizer :1077-1133, ZScaleTransformer :934-971, Chan3Trasformer :1020-1072 with
 * HistEqualizer :977-1012, MinMaxNormalizer :75-111) + Analyzer.predict's front part (evaluation.py:146-176) +
 * the ultralytics predictor preprocess (LetterBox, channel reversal, /255; SURVEY App. A.4).
 *
 * img: fp32 image in device memory, row-major with row_stride elements per row; big_endian != 0 means raw FITS
 * byte order (byte-swapped on load); non-finite pixels become 0 (utils.py:219,394).  Tile b covers
 * img[tile_y0[b] .. +Ty, tile_x0[b] .. +Tx].
 * chain_out  [B,Ty,Tx,3] fp32  : OPTIONAL (NULL: skipped) chain output before the resize — the parity surface; the
 *                                production path never materialises it (the final maps are evaluated per pixel inside
 *                                the fused letterbox kernel)
 * model_in   [B,Sh,Sw,4] bf16  : OPTIONAL letterboxed, channel-reversed, /255, NHWC (4th channel 0) — cy_model_forward
 *                                input (fp16 when cfg->out_f16)
 * model_in_f32 (optional) [B,3,Sh,Sw] fp32 NCHW: the same before bf16 rounding (parity entry)
 * status [B]: 0 ok, -1 tile rejected like the reference (preprocess returned None / constant rows,
 *             evaluation.py:164-176), -3 degenerate statistics (empty clip set), -6 a stage met data this build does
 *             not handle (order-reversing scale: non-positive maximum / sigma). */
int cy_letterbox_shape(int Ty, int Tx, int imgsz, int* Sh_host, int* Sw_host, cy_letterbox* lb_host);
/* run.py's option set -> stage list in run.py's order (scripts/run.py:272-293).  cfg->enabled == 0: empty chain. */
int cy_pp_chain_from_config(const cy_pp_config* cfg_host, cy_pp_chain* chain_host);
/* Checks a stage list (unknown types, stage combinations this build does not implement: CY_ERR_INVALID with the
 * reason in cy_last_error) and fills chain->reject_all. */
int cy_pp_chain_validate(cy_pp_chain* chain_host);
size_t cy_preprocess_chain_scratch_bytes(const cy_pp_chain* chain_host, int B, int Ty, int Tx);
/* cy_preprocess for a general stage list (same buffers and semantics). */
int cy_preprocess_chain(const cy_pp_chain* chain_host, const void* img, long long row_stride, int big_endian,
                        const int32_t* tile_x0, const int32_t* tile_y0, int B, int Ty, int Tx, int imgsz,
                        float* chain_out, void* model_in, float* model_in_f32, int32_t* status, void* scratch,
                        uintptr_t stream);
size_t cy_preprocess_scratch_bytes(const cy_pp_config* cfg_host, int B, int Ty, int Tx);
int cy_preprocess(const cy_pp_config* cfg_host, const void* img, long long row_stride, int big_endian,
                  const int32_t* tile_x0, const int32_t* tile_y0, int B, int Ty, int Tx, int imgsz, float* chain_out,
                  void* model_in, float* model_in_f32, int32_t* status, void* scratch, uintptr_t stream);
/* The predictor-preprocess part alone (LetterBox bilinear resize + pad 114 + channel reversal + /255, App. A.4) for
 * an already preprocessed HWC image: chain [B,Ty,Tx,3] fp32 -> model_in / model_in_f32 as above.  This is what the
 * `model(image, imgsz=...)` call of the reference does before the forward (caesar_yolo/evaluation.py:181-193). */
int cy_letterbox_resize(const float* chain, int B, int Ty, int Tx, int imgsz, void* model_in, float* model_in_f32,
                        uintptr_t stream);
/* Same with the 16-bit output format selectable: out_f16 = 0 bf16, 1 fp16. */
int cy_letterbox_resize_fmt(const float* chain, int B, int Ty, int Tx, int imgsz, void* model_in, float* model_in_f32,
                            int out_f16, uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ convolution
 * Layer primitive (ultralytics Conv = Conv2d+BN+SiLU fused; reference model call at
 * caesar_yolo/evaluation.py:181-193).  NHWC bf16 in, weights [cout_pad, k*k*cin] bf16 (K-major, BN folded),
 * bias fp32[cout_pad]; optional residual added after the activation; output bf16 or fp32 written into a
 * channel slice [out_coff, out_coff+cout) of an NHWC buffer with out_ctot channels. */
int cy_conv_block_n(int cout);
/* Diagnostics (tools/conv_probe.py): per-CTA clock64 timeline buffer for the conv kernel (NULL disables); the plan the
 * kernel would use for a shape: info8 = {mode, halves, units, block_n, a_stages, b_stages, acc_bufs, grid}. */
int cy_conv_set_debug(void* dev_buf, int units_per_cta);
int cy_conv_plan_info(int B, int Hin, int Win, int cin, int cout, int ksize, int stride, int* info8);
int cy_conv2d_nhwc(const void* in, int B, int Hin, int Win, int in_ctot, int in_coff, int cin, const void* w,
                   const float* bias, int cout, int cout_pad, int ksize, int stride, void* out, int out_ctot,
                   int out_coff, int out_f32, const void* res, int res_ctot, int res_coff, int act,
                   uintptr_t stream);

/* Stem layer primitive (model.0 of yolov8.yaml: Conv(3, c1, k=3, s=2) + BN + SiLU; same reference call site): the
 * model input [B,H,W,4] bf16 NHWC (4th channel ignored) -> [B,H/2,W/2,cout] bf16 in one fused kernel.  w_host is the
 * HOST fp32 OIHW weight [cout,3,3,3] with BN folded, bias_host HOST fp32 [cout]; cout in {16,32,48,64,80}; act: 0 none,
 * 1 SiLU (tanh form), 2 SiLU (ex2 + rcp).  Synchronises the stream (parity-test entry; the model plan keeps the
 * packed weights resident). */
int cy_stem_conv_nhwc4(const void* in, int B, int H, int W, const float* w_host, const float* bias_host, int cout,
                       int act, void* out, uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ model
 * Replaces `YOLO(weights)` (scripts/run.py:347) and `model(image, ...)` (caesar_yolo/evaluation.py:181-193):
 * YOLOv8 (variant "n" "s" "m" "l" "x"; yolov8.yaml, SURVEY App. A.5) or YOLO11 (variant "11n" ... "11x"; yolo11.yaml:
 * C3k2 / C2PSA / depthwise-separable Detect; the reference README lists yolo11 weights, README.md:200-207)
 * DetectionModel.forward with Conv+BN folded.  Tensors are given under their ultralytics state-dict names
 * (model.0.conv.weight, model.0.bn.running_var, ..., model.22.cv3.2.2.bias / model.23... for YOLO11), fp32, host memory.  forward: in = [B,Sh,Sw,4] bf16 NHWC (cy_preprocess output); heads_host receives three DEVICE
 * pointers (owned by the model, valid until the next forward of the same shape) to the raw Detect maps
 * [B, Sh/s, Sw/s, 80] fp32, s = 8,16,32: 64 DFL logits + nc class logits per anchor. */
int cy_model_create(const char* variant, int nc, void** model_host);
int cy_model_set_tensor(void* model, const char* name, const float* data_host, long long numel);
/* Storage format of weights and activations (call before cy_model_finalize): 0 = bf16 (default), 1 = fp16.  Both run
 * on the same tcgen05 kind::f16 instruction at the same rate with fp32 accumulation; fp16 keeps 11 significand bits
 * instead of 8 (ultralytics' own `half=True` inference type).  The model input (cy_preprocess out_f16) must match. */
int cy_model_set_precision(void* model, int fp16);
int cy_model_finalize(void* model);
/* info_host[0..7] of the plan for (B,Sh,Sw): conv launches, CTA-pair launches, launches in tap modes 0..3,
 * 256-wide-tile launches, two-half-tile launches (what the planner chose; parity tests assert on it). */
int cy_model_plan_summary(void* model, int B, int Sh, int Sw, int* info_host);
int cy_model_forward(void* model, const void* in, int B, int Sh, int Sw, const float** heads_host, uintptr_t stream);
/* info_host[0..7] = nparams, flops per forward of the last planned shape, #kernel launches per forward,
 * activation bytes, c3, c4, c5, #convs */
int cy_model_info(void* model, int B, int Sh, int Sw, double* info_host);
/* Per-layer timing of one forward (CUDA events, after a warm-up): names_host receives up to cap pointers to
 * internal strings, ms_host / flops_host the per-op numbers. Returns the number of ops in *nops_host. */
int cy_model_profile(void* model, const void* in, int B, int Sh, int Sw, int cap, const char** names_host,
                     float* ms_host, double* flops_host, int* nops_host, uintptr_t stream);
/* Sum over the conv launches of one forward of the algorithmic HBM bytes (input slice + weights + output slice +
 * residual, each once) -- the denominator for the ncu dram traffic in bench.py's roofline. */
int cy_model_conv_bytes(void* model, int B, int Sh, int Sw, double* bytes_host, int* nconv_host);
int cy_model_destroy(void* model);

/* ------------------------------------------------------------------------------------------------ detect / NMS
 * Detect._inference (DFL softmax + dist2bbox + sigmoid; SURVEY App. A.6): pred [B, 4+nc, A] fp32 (parity entry). */
int cy_num_anchors(int Sh, int Sw);
int cy_decode_pred(const float* h0, const float* h1, const float* h2, int B, int Sh, int Sw, int nc, float* pred,
                   uintptr_t stream);
/* Fused decode + ops.non_max_suppression (conf filter, best class, class-offset boxes, torchvision.ops.nms, max_det)
 * + ops.scale_boxes/clip_boxes.  dets [B,max_det,6] = x1,y1,x2,y2,conf,cls in descending score order. */
size_t cy_postprocess_scratch_bytes(int B, int Sh, int Sw, int max_det);
int cy_postprocess(const float* h0, const float* h1, const float* h2, int B, int Sh, int Sw, int nc, float conf,
                   float iou, int max_det, const cy_letterbox* lb, float* dets, int32_t* ndets, void* scratch,
                   uintptr_t stream);
/* == torchvision.ops.nms on each of B segments (boxes [B,N,4] xyxy, scores [B,N], counts [B] or NULL => N each):
 * keep [B,N] int64 original indices in descending score order (ties: lower index first), nkeep [B]. */
size_t cy_nms_scratch_bytes(int B, int N);
int cy_nms_batched(const float* boxes, const float* scores, const int32_t* counts, int B, int N, double iou_thr,
                   int max_keep, int64_t* keep, int32_t* nkeep, void* scratch, uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ merges
 * Analyzer.process_detections (caesar_yolo/evaluation.py:252-346) with utils.get_iou (utils.py:54-107) and Graph
 * (graph.py:2-41).  dets [B,det_stride,6]; keep_idx [B,det_stride] indices into the tile's dets in the
 * reference's output order; status[b] = -2 if get_iou would assert (degenerate box). det_stride <= 320.
 * pre_status (optional, [B]): tiles with a non-zero entry were rejected upstream (cy_preprocess status; the
 * reference's predict() returned -1) and yield no detections; their status is passed through. */
int cy_merge_tile(const float* dets, const int32_t* ndets, int B, int det_stride, float thr_score, float thr_soft,
                  float thr_hard, const int32_t* pre_status, int32_t* keep_idx, int32_t* nkeep, int32_t* status,
                  uintptr_t stream);
/* Analyzer.make_json_results (evaluation.py:418-469): records written at recs[tile_id*det_stride + i], nrec[tile_id]. */
int cy_make_records(const float* dets, const int32_t* keep_idx, const int32_t* nkeep, const int32_t* status,
                    int det_stride, const cy_tile* tiles, const int32_t* tile_ids, int B, cy_det_record* recs,
                    int32_t* nrec, uintptr_t stream);
size_t cy_compact_scratch_bytes(int T);
int cy_compact_records(const cy_det_record* slots, const int32_t* counts, int T, int slot_stride,
                       cy_det_record* out, int32_t* total, void* scratch, uintptr_t stream);
/* SFinder.find_sources_at_edge (inference.py:663-726) + merge_edge_sources (:731-931): recs = n records in gathered
 * order (tile-id major), tiles [T], CSR neighbour lists; out [>= n] sources in the reference's catalog order,
 * nout (device int64).  Synchronises the stream (component count is data dependent). */
int cy_merge_global(cy_det_record* recs, int n, const cy_tile* tiles, int T, const int32_t* nb_off,
                    const int32_t* nb_idx, cy_source* out, int64_t* nout, uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ source measurements
 * Per-source numbers the reference catalog does not carry (not part of the reference).  Pixel (x, y) belongs to source
 * s when x1 <= x <= x2 and y1 <= y <= y2 (catalog coordinates, inclusive), the pixel lies inside the image and the
 * owned rows, and its value is finite and non-zero (0 = masked, utils.py:219,394).  w = max(v, 0).
 *
 * Partial record of one source over one row range.  Every field combines by addition, the peak by max on the key
 * (peak, -peak_idx), so partials of disjoint row ranges fold into the partial of their union.  The first and second
 * moments are taken about the box corner (cx, cy) = (ceil(x1), ceil(y1)) — dx = x - cx, dy = y - cy — which is the
 * same on every rank and keeps fp64 free of the cancellation that absolute mosaic coordinates (~1e4 px) would bring
 * into the central moments.  peak_idx = y * ncols + x of the first pixel (row-major) that reaches the peak;
 * npix = 0: peak = -inf, peak_idx = INT64_MAX.  80 bytes. */
typedef struct {
    int64_t npix, peak_idx;
    double peak;
    double sum;                        /* sum of v */
    double sw, swx, swy;               /* sum of w, w*dx, w*dy */
    double swxx, swyy, swxy;           /* sum of w*dx^2, w*dy^2, w*dx*dy */
} cy_src_partial;
/* Final values.  xc, yc: w-weighted centroid (NaN when sum w = 0); a >= b: square roots of the eigenvalues of the
 * w-weighted central second-moment matrix (for a Gaussian source, its sigmas along the major / minor axis); theta: angle
 * of the major axis in degrees, in (-90, 90], measured from the +x (column) axis towards the +y (row) axis of the pixel
 * grid — counter-clockwise on the usual FITS display with row 0 at the bottom; it is not a sky position angle.  peak_x,
 * peak_y: pixel of the peak (NaN when npix = 0).  80 bytes. */
typedef struct {
    int64_t npix;
    double sum, peak, peak_x, peak_y, xc, yc, a, b, theta;
} cy_src_meas;
/* img: 4-byte pixels as for cy_preprocess (row_stride elements per row, big_endian = raw FITS byte order); the buffer
 * holds image rows from row0 on and columns [0, ncols).  Reads rows [row_begin, row_end) (row_begin >= row0, all inside
 * the buffer) for the nsrc sources src[] (device) and writes partials[nsrc].  Work units are up to 32 rows of one box;
 * the unit partials of a source are folded in unit order (deterministic for a given row range).  Synchronises the
 * stream (the unit count is data dependent). */
int cy_measure_sources(const void* img, long long row_stride, int big_endian, int row0, int ncols, const cy_source* src,
                       int nsrc, int row_begin, int row_end, cy_src_partial* partials, uintptr_t stream);
/* partials [world][nsrc] (e.g. all-gathered from `world` ranks that own disjoint row ranges) folded in rank order ->
 * meas[nsrc].  src and ncols as given to cy_measure_sources. */
int cy_measure_combine(const cy_src_partial* partials, int world, const cy_source* src, int nsrc, int ncols,
                       cy_src_meas* meas, uintptr_t stream);

/* Local background and noise of every source (not part of the reference).  The box of s is the integer rectangle
 * [ceil x1, floor x2] x [ceil y1, floor y2] of the measurements above (a source whose box is empty has no frame).  Its
 * frame is the box grown by F = `frame` pixels on every side, minus the box, clipped to columns [0, ncols) and to the
 * rows the run measures; membership is decided in absolute pixel coordinates, so it does not depend on the row split.
 * Non-finite pixels and 0 are masked, as for the box.  Mean-centred iterative sigma clipping, kappa = 3, at most 5
 * iterations (astropy's sigma_clip with cenfunc = 'mean', ddof = 0; astropy's default centre, the median, is the
 * median estimator below):
 *   pass 0 takes the mean mu_0 and standard deviation sigma_0 of all unmasked frame pixels;
 *   pass k >= 1 takes those of the pixels inside the intersection of [mu_j - 3 sigma_j, mu_j + 3 sigma_j], j < k
 *   (inclusive bounds: astropy's nested rejection, restated as one interval per source, so a pass needs no per-pixel
 *   state);
 *   a source stops when pass k >= 1 keeps as many pixels as pass k - 1, after pass 5, or when pass 0 finds no pixel.
 * bkg, rms: mean and standard deviation of the last kept set, nbkg its size, iters = k of the last pass (astropy's
 * niterations; 0 for an empty frame).  The mean is the default centre: it is a sum, so it adds up over row ranges and
 * ranks.  Pass k sums v - c and (v - c)^2 with c = 0 in pass 0 and c = mu_{k-1} after that, so the variance
 * does not cancel on a pedestal: mu = c + s1 / n, sigma^2 = max(s2 / n - (s1 / n)^2, 0).
 *
 * Partial record of one source over one row range and one pass: every field adds.  24 bytes. */
typedef struct {
    int64_t n;                         /* kept frame pixels */
    double s1, s2;                     /* sum of (v - c), (v - c)^2 */
} cy_noise_partial;
/* Clipping state of one source, the same on every rank.  While done = 0: [lo, hi] is the interval pass `iters` keeps
 * (-inf, +inf before the first clip), c its shift, nbkg the pixels the previous pass kept.  Once done = 1: bkg, rms,
 * nbkg, iters are final (bkg = rms = NaN when nbkg = 0).  56 bytes. */
typedef struct {
    double lo, hi, c;
    double bkg, rms;
    int64_t nbkg;
    int32_t iters, done;
} cy_noise_state;
/* Sets state[nsrc] to pass 0 and writes the exclusive offsets unit_off[nsrc + 1] of the work units (up to 32 rows of one
 * grown box inside [row_begin, row_end)), *units their count; the offsets serve every pass.  frame >= 1.  Synchronises
 * the stream (the unit count is data dependent). */
int cy_noise_init(const cy_source* src, int nsrc, int ncols, int row_begin, int row_end, int frame,
                  cy_noise_state* state, long long* unit_off, long long* units, uintptr_t stream);
/* One pass over rows [row_begin, row_end) of img (layout and row arguments as for cy_measure_sources; src, ncols, the
 * rows, frame, unit_off and units as given to cy_noise_init): partials[nsrc] for the sources that are not done (the
 * others are neither read nor written).  Rows inside the box's row span read the two side segments, other rows the
 * full grown width; the unit partials of a source are folded in unit order. */
int cy_noise_pass(const void* img, long long row_stride, int big_endian, int row0, int ncols, const cy_source* src,
                  int nsrc, int row_begin, int row_end, int frame, const long long* unit_off, long long units,
                  const cy_noise_state* state, cy_noise_partial* partials, uintptr_t stream);
/* partials [world][nsrc] of one pass (all-gathered from `world` ranks that own disjoint row ranges) folded in rank order
 * -> state advanced by one pass; *active: sources not yet done (the same on every rank, so every rank runs the same
 * number of passes: at most 6).  Synchronises the stream. */
int cy_noise_update(const cy_noise_partial* partials, int world, int nsrc, cy_noise_state* state, int* active,
                    uintptr_t stream);

/* Median estimator (opt-in, bkg_estimator = 'median'; not part of the reference).  The same pixel sets, frames, node
 * boxes and mask rules as above, clipped around the median: astropy's sigma_clipped_stats defaults (cenfunc = 'median',
 * stdfunc = 'std', ddof = 0, sigma = 3, maxiters = 5).
 *   Set 0 is all unmasked pixels.  Pass k takes n_k, the median m_k and the standard deviation sigma_k of set k; set
 *   k + 1 = set k intersected with [m_k - 3 sigma_k, m_k + 3 sigma_k] (inclusive bounds, one interval per source).
 *   A source stops when n_k = n_{k-1} for k >= 1 (the set did not change: m_k = m_{k-1}), after pass 5, or when set k
 *   is empty.  bkg = m of the last set, rms = sigma of the last set, nbkg its size, iters as above.
 *   Median of n values x_(0) <= ... <= x_(n-1): x_((n-1)/2) for odd n, (x_(n/2-1) + x_(n/2)) / 2 in fp64 for even n,
 *   which is np.median of the float64 values.  sigma is summed about the shift c = m_{k-1} (0 in pass 0), as above.
 * The median is selected exactly by radix select on the order-preserving key of the float32 bits (negative values:
 * every bit flipped; positive values: the sign bit set).  A pass is 4 digit rounds of 8 bits.  Round 0 reads set k and
 * writes the moment partials of the mean path together with the 256-bin histogram of the top key byte; round r >= 1
 * counts byte r of the kept keys whose top 8r bits equal the prefix of a middle rank.  The two middle ranks of an even
 * n may part at some digit; both prefixes are followed, in slots [0, 256) and [256, 512).  The histograms are uint32
 * counts, so they add exactly in any order over work units, row ranges and ranks (sum them across ranks, e.g. with an
 * all-reduce): the median does not depend on the row split.  A set of 2^32 pixels or more is refused.
 * Select state of one source or node, the same on every rank.  40 bytes. */
typedef struct {
    uint32_t prefix[2];                /* top 8 (round + 1) key bits of the lower / upper middle rank */
    int64_t rank[2];                   /* their ranks among the kept keys that share the prefix */
    int64_t n;                         /* n_k, the size of set k */
    int32_t split;                     /* the two prefixes differ */
    int32_t round;                     /* last round picked */
} cy_select_state;
/* Round `round` (0..3) of a median pass: hist[nsrc * 512] (uint32, device) is zeroed and filled with this range's
 * counts; in round 0 partials[nsrc] are written as by cy_noise_pass (the other rounds leave them).  The other arguments
 * as for cy_noise_pass; sel as left by cy_median_update. */
int cy_noise_pass_median(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                         const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                         const long long* unit_off, long long units, const cy_noise_state* state,
                         const cy_select_state* sel, int round, cy_noise_partial* partials, uint32_t* hist,
                         uintptr_t stream);
/* round r of a pass, after the histograms of all ranks are summed into hist[n * 512] (and, in round 0, the partials
 * [world][n] all-gathered): round 0 folds the partials in rank order and stops the sources whose set is empty or
 * unchanged; every round picks the bins of the middle ranks; round 3 finalises m_k and advances the states (as
 * cy_noise_update does for the mean), synchronises the stream and sets *active (rounds 0..2 do not synchronise and
 * leave *active alone; active may be NULL there).  n: sources, or the Nx * Ny nodes of a lattice. */
int cy_median_update(const cy_noise_partial* partials, int world, const uint32_t* hist, int n, cy_noise_state* state,
                     cy_select_state* sel, int round, int* active, uintptr_t stream);

/* Source mask (opt-in, not part of the reference).  M is the union over all sources of the integer boxes [ceil x1,
 * floor x2] x [ceil y1, floor y2], the rule of the box measurements; an empty box or NaN coordinates add nothing, and
 * the boxes are not dilated.  Membership is decided in absolute pixel coordinates, so M does not depend on the row
 * split.  With the mask, a frame pixel (cy_noise_pass_masked) or a node-box pixel (cy_bkg_grid_pass_masked) in M is
 * masked exactly like a non-finite or 0 pixel.  A frame already excludes its own box, so the mask removes the boxes of
 * its neighbours; a frame left empty gives nbkg = 0 and NaN bkg / rms, as above.  The per-source statistics and the
 * maps of one run use the same M, so they still compare directly.
 * Layout: rows [row_begin, row_end) of the image, (row_end - row_begin) x ceil(ncols / 32) uint32 words, row-major;
 * bit (x & 31) of word (x >> 5) of mask row y - row_begin is set when pixel (x, y) is in M; bits past ncols are 0.
 * Writes the mask of columns [0, ncols) and rows [row_begin, row_end) for the nsrc sources src[] (device): zeroed first,
 * then the bits of every box ORed in (work units of up to 32 rows of one box, so the result does not depend on the
 * order).  Synchronises the stream (the unit count is data dependent). */
int cy_source_mask(const cy_source* src, int nsrc, int ncols, int row_begin, int row_end, uint32_t* mask,
                   uintptr_t stream);
/* cy_noise_pass with the frame pixels in M masked; mask: cy_source_mask of the same src, ncols and rows. */
int cy_noise_pass_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                         const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                         const long long* unit_off, long long units, const cy_noise_state* state,
                         cy_noise_partial* partials, const uint32_t* mask, uintptr_t stream);

/* cy_noise_pass_median with the frame pixels in M masked. */
int cy_noise_pass_median_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                                const long long* unit_off, long long units, const cy_noise_state* state,
                                const cy_select_state* sel, int round, cy_noise_partial* partials, uint32_t* hist,
                                const uint32_t* mask, uintptr_t stream);

/* Background and rms maps of an image region (not part of the reference).  The region is W = ncols columns (columns
 * [0, ncols) of the buffer) by H = R1 - R0 rows (rows [R0, R1)); a run maps the pixels it read.
 * Grid nodes: with step g = grid, node column i sits at x_i = min(i g, W - 1), i = 0 .. Nx - 1, Nx = ceil((W - 1) / g)
 * + 1, and node row j at y_j = R0 + min(j g, H - 1), Ny alike from H: the first and last nodes lie on the region's
 * edges, and W = 1 (H = 1) gives one node along that axis.  Node n = j Nx + i.  The box of a node is [x_i - h, x_i + h]
 * x [y_j - h, y_j + h], h = box / 2, clipped to the region; box is odd and >= 3, grid >= 1.  Membership is decided in
 * absolute pixel coordinates, so it does not depend on the row split.
 * Node statistic: the one of cy_noise_state above, unchanged (unmasked box pixels, mean-centred sigma clipping, kappa =
 * 3, at most 5 iterations; passes, partials and cy_noise_update as for the sources).  A node whose box has no unmasked
 * pixel gets bkg = rms = NaN, like an empty frame.
 * Map pixel (x, y): bilinear in fp64 between the nodes i, i + 1 and j, j + 1, where i is the largest index with x_i <= x
 * clamped to Nx - 2 (0 when Nx = 1), t = (x - x_i) / (x_{i+1} - x_i) (0 when Nx = 1), and j, u alike along rows.  A
 * corner whose value is NaN is dropped and the weights of the others renormalised; the pixel is NaN when the finite
 * corners carry no weight.  The rms map interpolates the node rms (not the variance).  Stored as float32 in FITS byte
 * order (big-endian, BITPIX -32).
 * Background-subtracted and S/N maps (opt-in): at map pixel (x, y), v is the image pixel decoded as for the noise
 * statistics (byte order applied; non-finite and 0 are masked), fb and fr the float32 values of the bkg and rms maps
 * at that pixel, to the bit (same interpolation, NaN corners dropped alike).
 *   res = (float)((double)v - (double)fb),  snr = (float)(((double)v - (double)fb) / (double)fr).
 * A masked v or a NaN fb gives NaN in both maps; a NaN fr or fr <= 0 gives NaN in snr only.  The source mask M is not
 * applied to these maps (sources show in them; M only shaped the nodes).  Stored like the bkg and rms maps. */

/* Sets state[Nx * Ny] to pass 0 and writes the exclusive offsets unit_off[Ny + 1] of the work units of rows [row_begin,
 * row_end) (R0 <= row_begin <= row_end <= R1; a unit is one chunk of <= 32 rows of one node row and 16 adjacent node
 * columns), *units their count; the offsets serve every pass.  Synchronises the stream (for the unit count). */
int cy_bkg_grid_init(int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid, cy_noise_state* state,
                     long long* unit_off, long long* units, uintptr_t stream);
/* One clipping pass over rows [row_begin, row_end) of img (layout and row0 as for cy_measure_sources; the other
 * arguments as given to cy_bkg_grid_init): partials[Nx * Ny] for the nodes that are not done.  Rank partials are folded
 * with cy_noise_update(partials, world, Nx * Ny, state, &active, stream) until active = 0 (at most 6 passes). */
int cy_bkg_grid_pass(const void* img, long long row_stride, int big_endian, int row0, int ncols, int R0, int R1,
                     int row_begin, int row_end, int box, int grid, const long long* unit_off, long long units,
                     const cy_noise_state* state, cy_noise_partial* partials, uintptr_t stream);
/* cy_bkg_grid_pass with the node-box pixels in M masked.  mask: cy_source_mask of rows [row_begin, row_end) over
 * mask_ncols columns; region column x is mask column x + mask_col0 (0 <= mask_col0, mask_col0 + ncols <= mask_ncols), so
 * a region that starts at column X0 of a wider mask passes mask_col0 = X0. */
int cy_bkg_grid_pass_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols, int R0, int R1,
                            int row_begin, int row_end, int box, int grid, const long long* unit_off, long long units,
                            const cy_noise_state* state, cy_noise_partial* partials, const uint32_t* mask,
                            int mask_ncols, int mask_col0, uintptr_t stream);
/* Round `round` of a median pass of the lattice (median estimator above): hist[Nx * Ny * 512] as for
 * cy_noise_pass_median, the other arguments as for cy_bkg_grid_pass; rounds are folded with cy_median_update(partials,
 * world, hist, Nx * Ny, state, sel, round, &active, stream).  The hole probe and fill run unchanged on the median
 * states (the probe is an unmasked cy_bkg_grid_pass: it only counts). */
int cy_bkg_grid_pass_median(const void* img, long long row_stride, int big_endian, int row0, int ncols, int R0, int R1,
                            int row_begin, int row_end, int box, int grid, const long long* unit_off, long long units,
                            const cy_noise_state* state, const cy_select_state* sel, int round,
                            cy_noise_partial* partials, uint32_t* hist, uintptr_t stream);
int cy_bkg_grid_pass_median_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols, int R0,
                                   int R1, int row_begin, int row_end, int box, int grid, const long long* unit_off,
                                   long long units, const cy_noise_state* state, const cy_select_state* sel,
                                   int round, cy_noise_partial* partials, uint32_t* hist, const uint32_t* mask,
                                   int mask_ncols, int mask_col0, uintptr_t stream);
/* Hole fill of a masked lattice.  After the masked passes every node is one of:
 *   finite: nbkg > 0;
 *   hole:   nbkg = 0, but its box holds at least one data pixel (finite and non-zero) when M is ignored;
 *   blank:  its box holds no data pixel (the NaN borders of a mosaic).
 * Ring k fills every unfilled hole that has a finite or already-filled node among its 8 lattice neighbours with the fp64
 * mean of those neighbours' bkg and, separately, rms as they stood after ring k - 1, summed in row-major neighbour order
 * (deterministic).  Rings repeat until no node changes.  Blank nodes are never filled and never feed the fill, so NaN
 * borders do not spread; holes with no path to a finite node stay NaN; a filled node keeps nbkg = 0.  The map
 * interpolation above is unchanged.  Catalog bkg / rms are never filled.
 * Probe: sets probe[nodes] to pass 0 for the nodes with nbkg = 0 of the final states `state` and to done for the
 * others, *nprobe the count of the former (the same on every rank).  When it is not 0, one unmasked cy_bkg_grid_pass
 * of the probe (same arguments and unit plan as the passes; only the boxes of the probed nodes are read) gives each
 * probed node's data-pixel count n; the partials are all-gathered like those of a pass.  Synchronises the stream. */
int cy_bkg_grid_probe_init(const cy_noise_state* state, int nodes, cy_noise_state* probe, int* nprobe,
                           uintptr_t stream);
/* Fill: probe partials [world][Nx * Ny] folded in rank order (n > 0: hole) -> the holes of state[Nx * Ny] filled in
 * rings; *filled: the nodes filled.  Every rank fills the same replicated states identically.  Synchronises the stream
 * once per ring. */
int cy_bkg_grid_fill(const cy_noise_partial* probe_partials, int world, int nx, int ny, cy_noise_state* state,
                     int* filled, uintptr_t stream);
/* Final node states -> rows [row_begin, row_end) of the bkg and rms maps: (row_end - row_begin) x ncols 4-byte words
 * each, row-major, big-endian float32.  No pixel of the image is read. */
int cy_bkg_grid_maps(const cy_noise_state* state, int ncols, int R0, int R1, int row_begin, int row_end, int box,
                     int grid, void* bkg, void* rms, uintptr_t stream);
/* Final node states and rows [row_begin, row_end) of img (layout, row0 and region columns as for cy_bkg_grid_pass)
 * -> the same rows of the background-subtracted (res) and S/N (snr) maps above: (row_end - row_begin) x ncols 4-byte
 * words each, row-major, big-endian float32.  One pass: every image pixel of the rows is read once; no collective (each
 * rank maps its own rows).  The other arguments as for cy_bkg_grid_maps. */
int cy_bkg_grid_snr_maps(const cy_noise_state* state, const void* img, long long row_stride, int big_endian, int row0,
                         int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid, void* res, void* snr,
                         uintptr_t stream);

/* ------------------------------------------------------------------------------------------------ whole path
 * FITS file -> merged catalog with no host-language orchestration: SFinder.run_parallel (caesar_yolo/inference.py:
 * 578-658; the serial SFinder.run :485-552 is the tile_x <= 0 case: the whole region is one tile), TileTask.find_sources
 * (:173-275) incl. the per-tile file read (utils.read_fits_crop, utils.py:340-418), gather_task_data_from_workers
 * (:936-984), find_sources_at_edge + merge_edge_sources (:663-931).  One context per GPU / process; rank r of `world`
 * owns a contiguous band of tile rows (replaces the tile -> worker map of :1008-1029, max_ntasks_per_worker).  The
 * payload rows of the band are read with pread (read_threads threads) into two pinned staging buffers and uploaded
 * in ~64 MB pieces on a copy stream that overlaps the compute of earlier tile groups. */
typedef struct {
    int32_t imgsz;                       /* --imgsize */
    float score_thr, iou_thr;            /* --scoreThr, --iouThr */
    float thr_soft, thr_hard;            /* --merge_overlap_iou_thr_soft / _hard */
    int32_t tile_x, tile_y;              /* --tile_xsize / --tile_ysize; <= 0: no tiling (one tile = the region) */
    double step_x, step_y;               /* --tile_xstep / --tile_ystep */
    int32_t xmin, xmax, ymin, ymax;      /* --xmin ...: region of the image (inclusive), -1 = full axis */
    int32_t batch_tiles;                 /* tiles per preprocessing group / conv batch (0: 296 = two per SM) */
    int32_t read_threads;                /* file reader threads (0: 8) */
    int32_t rank, world;
} cy_run_config;
/* All-gather of `bytes_per_rank` bytes per rank between device buffers, enqueued on `stream` (e.g. a wrapper of
 * ncclAllGather(send, recv, bytes, ncclUint8, comm, stream)); returns 0 on success. */
typedef int (*cy_allgather_fn)(void* user, const void* send_dev, void* recv_dev, size_t bytes_per_rank, uintptr_t stream);

/* chain_host == NULL: no preprocessing (empty stage list).  The model must be finalized; its storage format decides
 * the model-input format. */
int cy_ctx_create(void* model, const cy_pp_chain* chain_host, const cy_run_config* cfg_host, void** ctx_host);
int cy_ctx_set_allgather(void* ctx, cy_allgather_fn fn, void* user);
int cy_ctx_destroy(void* ctx);
/* This rank's share: file -> records of its tiles (device, tile-id order).  Only unscaled BITPIX = -32 images with 2 or 4
 * axes are read in place (the reference takes plane [0,0] of a 4-D cube); other payloads: convert on the host and use the
 * _payload form (rows of 4-byte pixels in host memory, big_endian = raw FITS byte order, pinned != 0: page-locked). */
int cy_run_local(void* ctx, const char* fits_path, int* nrecords_host);
int cy_run_local_payload(void* ctx, const void* payload_host, int ny, int nx, int big_endian, int pinned,
                         int* nrecords_host);
int cy_ctx_records(void* ctx, const cy_det_record** recs_dev, int* n_host);
/* Exchange helpers: the all-gather slot of this rank = 32-byte header (record count) + the first `cap` records;
 * unpack: `world` gathered slots -> records of all ranks in rank (= tile-id) order; *max_count_host > cap means a
 * slot overflowed (redo with a larger cap). */
int cy_ctx_pack_slot(void* ctx, int cap, const void** slot_dev);
int cy_ctx_unpack_slots(void* ctx, const void* slots_dev, int world, int cap, const cy_det_record** recs_dev,
                        int* n_host, int* max_count_host);
/* Edge flags + cross-tile merge of a gathered record list -> sources in the reference's catalog order, copied to the
 * host (sources_host may be NULL: count only). */
int cy_run_merge(void* ctx, const cy_det_record* recs_dev, int n, cy_source* sources_host, int capacity,
                 int* nsources_host);
/* cy_run_local + exchange (the registered all-gather when world > 1) + cy_run_merge. */
int cy_run_mosaic(void* ctx, const char* fits_path, cy_source* sources_host, int capacity, int* nsources_host,
                  int* nrecords_host);
int cy_run_payload(void* ctx, const void* payload_host, int ny, int nx, int big_endian, int pinned,
                   cy_source* sources_host, int capacity, int* nsources_host, int* nrecords_host);
/* info_host[8]: tiles of the grid, tiles processed by this rank, payload bytes uploaded (cumulative), first / last
 * (exclusive) tile id of this rank, records of this rank. */
int cy_ctx_info(void* ctx, double* info_host);

#ifdef __cplusplus
}
#endif
#endif
