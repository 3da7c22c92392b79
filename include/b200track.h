/* b200track.h -- C ABI of libb200track.so (B200 / sm_100a).
 *
 * The reference (JackWoo0831/Yolov7-tracker) has no FFI: its "operator API" is the Python module
 * surface of tracker/{kalman_filter,matching,basetrack,bytetrack,botsort}.py.  Each entry point
 * below names the reference function it replaces (file:line relative to /root/reference); the
 * Python drop-in modules under yolov7-tracker_b200/tracker bind them through ctypes
 * (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, a negative B2T_E* code on failure;
 *     b2t_last_error() returns a thread-local message for the last failure.
 *   - pointers are DEVICE pointers unless the name ends in _host / the parameter says host.
 *   - dtype: B2T_F32 (all-float32 tracker arithmetic) or B2T_F64 (the reference's float64).
 *   - `stream` is a cudaStream_t passed as void*; device-pointer entry points never allocate
 *     and never synchronise.  *_host entry points copy H2D, launch, copy D2H and synchronise
 *     the stream before returning.
 *   - fmt: Kalman state parametrisation, B2T_FMT_XYAH ('default', KalmanFilter),
 *     B2T_FMT_XYWH ('botsort', BoTSORTKalmanFilter), B2T_FMT_NSA ('strongsort', NSAKalmanFilter).
 */
#ifndef B200TRACK_H
#define B200TRACK_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { B2T_F32 = 0, B2T_F64 = 1 };
enum { B2T_FMT_XYAH = 0, B2T_FMT_XYWH = 1, B2T_FMT_NSA = 2 };
enum { B2T_SORT = 0, B2T_BYTETRACK = 1, B2T_BOTSORT = 2, B2T_CBIOU = 3 };
enum { B2T_OK = 0, B2T_EINVAL = -1, B2T_ECUDA = -2, B2T_ECAPACITY = -3, B2T_ENOTBUILT = -4 };
/* 16-bit activation / weight type of the detector branch.  Both feed tcgen05 kind::f16 at the same rate with fp32
 * accumulation; fp16 (the reference's own GPU half mode, detect.py:41) carries 3 more mantissa bits than bf16. */
enum { B2T_ACT_BF16 = 0, B2T_ACT_F16 = 1 };

/* per-track flag bits used by the Kalman entry points */
enum { B2T_FLAG_MEAN_F32 = 1,   /* the reference still holds this mean as float32 (SURVEY q12) */
       B2T_FLAG_NOT_TRACKED = 2 /* state != Tracked: multi_predict zeroes mean[7] first (basetrack.py:263-265) */ };

const char* b2t_last_error(void);
int b2t_version(void);
/* number of kernel launches issued by this library in this process (bench.py's gpu_launches) */
long long b2t_launch_count(void);

/* ---------------------------------------------------------------- Kalman (tracker/kalman_filter.py) */
/* KalmanFilter.initiate :190-221 / BoTSORTKalmanFilter.initiate :435-466.
 * meas [k][4] (dtype), mean [k][8], cov [k][64] outputs. */
int b2t_kalman_initiate(int dtype, int fmt, const void* meas, void* mean, void* cov, int k, void* stream);
/* KalmanFilter.multi_predict :289-329 (BoT-SORT :534-571) incl. the STrack.multi_predict preamble
 * basetrack.py:253-271.  In place.  flags [n] int32 or NULL; q_f32 != 0 -> process noise in float32. */
int b2t_kalman_predict(int dtype, int fmt, void* mean, void* cov, const int* flags, int n, int q_f32, void* stream);
/* KalmanFilter.project :260-287 (+ NSA :617-631).  out_mean [n][4], out_cov [n][16]; conf [n] float or NULL. */
int b2t_kalman_project(int dtype, int fmt, const void* mean, const void* cov, const int* flags, const float* conf,
                       void* out_mean, void* out_cov, int n, void* stream);
/* KalmanFilter.update :331-363 (BoT-SORT :573-605, NSA :633-646).  In place on rows idx[0..k) of
 * mean/cov (idx NULL -> rows 0..k).  meas [k][4] (dtype); conf [k] float or NULL. */
int b2t_kalman_update(int dtype, int fmt, void* mean, void* cov, const int* idx, const void* meas,
                      const float* conf, const int* flags, int k, void* stream);
/* KalmanFilter.gating_distance :365-411 (metric 'maha' = 0, 'gaussian' = 1).  One state vs m
 * measurements: mean [8], cov [64], meas [m][4] -> out [m]. */
int b2t_kalman_gating(int dtype, int fmt, const void* mean, const void* cov, const void* meas, int m,
                      int only_position, int metric, void* out, void* stream);
/* botsort.multi_gmc, tracker/botsort.py:250-269.  warp_host: 6 doubles {a00,a01,tx,a10,a11,ty} on the HOST. */
int b2t_gmc_apply(int dtype, void* mean, void* cov, int n, const double* warp_host, void* stream);

/* ---------------------------------------------------------------- cost + assignment (tracker/matching.py) */
/* matching.ious / iou_distance :44-82 (cython_bbox "+1" IoU).  a [batch][n][4], b [batch][m][4] tlbr,
 * cost [batch][n][ld] = 1 - IoU (as_distance != 0) or IoU. */
int b2t_iou_cost(int dtype, const void* a, int n, const void* b, int m, void* cost, int ld, int batch,
                 int as_distance, void* stream);
/* matching.linear_assignment :30-41 == lap.lapjv(cost, extend_cost=True, cost_limit=thresh).
 * cost [batch][n][ld]; x [batch][n], y [batch][m] int32 outputs (-1 = unmatched).
 * workspace: b2t_lap_workspace_bytes(dtype, n, m, batch) bytes of device memory. */
size_t b2t_lap_workspace_bytes(int dtype, int n, int m, int batch);
int b2t_lap_solve(int dtype, const void* cost, int n, int m, int ld, double thresh, int* x, int* y,
                  void* workspace, size_t workspace_bytes, int batch, void* stream);

/* ---------------------------------------------------------------- fused trackers
 * One object = S independent video sequences advanced together, one CTA per sequence per frame:
 *   BaseTracker.update tracker/basetrack.py:368-487, ByteTrack.update tracker/bytetrack.py:41-204,
 *   BoTSORT.update tracker/botsort.py:313-493, C_BIoUTracker.update tracker/c_biou_tracker.py:218-353.
 * B2T_CBIOU (cascaded buffered IoU, no Kalman filter) reads conf_thresh, track_buffer and frame_rate and ignores fmt, iou_thresh and
 * use_gmc.  It needs dtype = B2T_F64 (B2T_EINVAL otherwise: the reference's IoU is float64 and there is no Kalman state to shrink) and
 * rejects predict_only (the reference's update_without_detection needs a Kalman filter).  Its lost tracks are never pruned (as in the
 * reference), so cap bounds the tracks a sequence can ever hold at once, lost ones included: an overflow is the sticky capacity
 * error, never a dropped track.  The per-slot record it keeps is documented with b2t_tracker_read_slot. */
typedef struct b2t_tracker b2t_tracker;

typedef struct b2t_tracker_config {
    int kind;          /* B2T_SORT / B2T_BYTETRACK / B2T_BOTSORT / B2T_CBIOU */
    int dtype;         /* B2T_F32 / B2T_F64 */
    int fmt;           /* Kalman format */
    int n_seq;         /* sequences per launch */
    int cap;           /* track slots per sequence (tracked + lost + births of one frame) */
    int dmax;          /* detections per sequence per frame, <= 1024 */
    int ecap;          /* sub-threshold (track, detection) pairs per association per sequence */
    int use_gmc;       /* BoT-SORT: apply the per-frame warp */
    int track_buffer;  /* opts.track_buffer */
    double conf_thresh; /* opts.conf_thresh (basetrack.py:354), a Python float in the reference */
    double iou_thresh;  /* opts.iou_thresh, SORT only (basetrack.py:414,438) */
    double frame_rate;  /* tracker ctor frame_rate */
} b2t_tracker_config;

size_t b2t_tracker_state_bytes(const b2t_tracker_config* cfg);
/* state_mem: b2t_tracker_state_bytes() bytes of device memory owned by the caller (256-B aligned). */
int b2t_tracker_create(const b2t_tracker_config* cfg, void* state_mem, void* stream, b2t_tracker** out);
int b2t_tracker_reset(b2t_tracker* t, void* stream);
void b2t_tracker_destroy(b2t_tracker* t);
int b2t_tracker_out_cols(void);   /* 8: id, x, y, w, h, cls, score, slot */
int b2t_tracker_stat_words(void); /* 64: [0..16) counters, [16..32) per-phase SM cycles, [32..64) sub-phase cycles */
/* One frame for every sequence.
 *   dets      [S][dmax][6] float32  x1,y1,x2,y2,score,cls (what track.py:149 hands to tracker.update)
 *   det_count [S] int32
 *   warps     [S][6] float64 or NULL (BoT-SORT camera motion, botsort.py:380)
 *   id_base   [S] int32 or NULL: overrides the sequence's id counter before births (BaseTrack._count)
 *   out       [S][out_rows][8] float64, stat [S][64] int32
 *   predict_only != 0 -> update_without_detection (basetrack.py:489-537) */
int b2t_tracker_step(b2t_tracker* t, const float* dets, const int* det_count, const double* warps,
                     const int* id_base, double* out, int out_rows, int* stat, int predict_only, void* stream);
/* Same with HOST buffers (pinned recommended); device staging lives inside the state block. */
int b2t_tracker_step_host(b2t_tracker* t, const float* dets_host, const int* det_count_host,
                          const double* warps_host, const int* id_base_host, double* out_host, int out_rows,
                          int* stat_host, int predict_only, void* stream);
/* One sequence's ordered list of tracked (which = 0) or lost (which = 1) tracks -- BaseTracker.tracked_stracks / .lost_stracks,
 * basetrack.py:358-360 -- as rows of b2t_tracker_list_cols() = 13 doubles on the HOST: id, tlwh[4] (STrack.tlwh of the Kalman mean;
 * B2T_CBIOU: the last matched detection box, C_BIoUSTrack.tlwh),
 * cls, score, slot, state, is_activated, tracklet_len, start_frame, frame_id.  *n_host = list length (rows beyond max_rows are not copied).
 * Synchronises the stream. */
int b2t_tracker_list_cols(void);
int b2t_tracker_read_list(b2t_tracker* t, int seq, int which, double* rows_host, int max_rows, int* n_host, void* stream);
/* Copies one slot's Kalman state to the host as float64: mean[8], cov[64] (lazy STrack.mean/.cov).
 * B2T_CBIOU keeps another record in the same 72 doubles r = mean[0..8) ++ cov[0..64): r[0] history length n (1..6), r[1]
 * time_since_update, r[8..32) the last n matched tlwh boxes oldest first, r[32..36) motion_state1, r[36..40) motion_state2 (tlwh);
 * the rest is unused.  Box values are float32 numbers. */
int b2t_tracker_read_slot(b2t_tracker* t, int seq, int slot, double* mean_host, double* cov_host, void* stream);

/* ---------------------------------------------------------------- detector: conv + bias + SiLU (tcgen05 / TMA)
 * Replaces Conv.fuseforward (models/common.py:110-111, BN folded as utils/torch_utils.py:181-201) and the
 * linear 1x1 convs of Detect (models/yolo.py:44).  Activations NHWC bf16, possibly a channel slice of a wider
 * (concat) buffer; weights [cout_rows][kh][kw][cin] bf16; bias fp32 [cout]; output bf16 or fp32 written at
 * channel offset out_coff of a buffer with out_pitch channels per pixel (concat-by-address).  Outputs leave through TMA
 * tensor stores, which clip at 16-byte granularity: a slice with cout % 8 (bf16) / % 4 (fp32) != 0 owns its padding.
 * A plan owns the three TMA tensor maps, a zero-padded snapshot of the bias (taken at plan time) and its tile counters;
 * pointers are fixed at plan time; b2t_conv_run only launches (with programmatic stream serialization, so the next conv's
 * prologue overlaps this one's tail).  At most one launch of a given plan may be in flight at a time. */
typedef struct b2t_conv_desc {
    const void* x;        /* input buffer base (bf16) */
    const void* w_packed; /* [cout_rows][kh*kw*cin] bf16 */
    const float* bias;    /* [cout] */
    void* y;              /* output buffer base */
    int n, h, w;          /* input batch / height / width */
    int cin;              /* channels read (multiple of 16) */
    int in_pitch;         /* channels per pixel of the input buffer (>= in_coff + cin, multiple of 8) */
    int in_coff;          /* first channel read (multiple of 8) */
    int cout;             /* output channels */
    int cout_rows;        /* rows of w_packed (>= cout, padded with zeros to a multiple of 16) */
    int kh, kw, stride;   /* k in {1,3}, stride in {1,2}, padding k/2 */
    int out_pitch, out_coff;
    int act;              /* 1 = SiLU, 0 = linear, 2 = ReLU (the ReID extractor, tracker/reid_models/deepsort_reid.py), 3 = LeakyReLU(0.1) (YOLOv7-tiny) */
    int out_f32;          /* 1 = fp32 output, 0 = bf16 */
    int block_n;          /* 0 = automatic; else output channels per CTA (multiple of 16, <= 256) */
    int tile_w;           /* 0 = automatic; else spatial tile width (4, 8 or 16) */
    int stages;           /* 0 = automatic (as deep as shared memory allows); else shared-memory ring depth (1..8) */
    int in_row_pixels;    /* 0 = w; else pixels per input row in memory (rows padded on the right; x points at column 0) */
    int rowpack;          /* 1 = "row-packed" 3x3 / stride 1 / cin 16 layer (the w6 stem after ReOrg): the three kw taps of a
                           * kernel row are ONE 64-channel K chunk read through an overlapping-stride tensor map (pixels
                           * x-1, x, x+1 and a dummy pixel with zero weights) -- 3 MMA chunks per tile instead of 9 quarter
                           * chunks.  Needs in_row_pixels >= w + 3, x pointing at a ZERO pixel that precedes column 0 of
                           * every row (and zeros after column w-1), w_packed = [cout_rows][3][64] with k = kw*16 + c. */
    int io_dtype;         /* B2T_ACT_BF16 / B2T_ACT_F16: type of x, w_packed and (unless out_f32) y */
    int halo;             /* 1 = halo-tile mode for a 3x3 / stride 1 / cin % 64 == 0 layer: one (16+2) x (8*mt+2) pixel input tile per
                           * 64-channel chunk is loaded once and read by all nine taps through shifted shared-memory windows
                           * (6.4x less activation traffic into shared memory than one tile per tap).  Same results up to fp32
                           * accumulation order. */
    int halo_bufs;        /* halo mode: 0 / 2 = two input-tile buffers, 3 = three (if shared memory allows) */
    int tps;              /* halo mode: filter taps per weight-ring stage: 0 = automatic (3 = one kernel row per 3-D TMA box when
                           * BLOCK_N <= 128, else 1; 9 = the CTA's nine weight tiles stay RESIDENT when the layer has one K chunk and
                           * one N tile, e.g. 64 -> 64), or 1 / 3 / 9 */
    int kpair;            /* 1x1 / stride 1 layers: 0 = automatic (two 64-channel K chunks per ring stage, each operand ONE 3-D TMA box, when
                           * the chunk count is even), 1 = one chunk per stage, 2 = require pairs */
    int out_bufs;         /* epilogue staging boxes (128 pixels x 128 B) per sub-tile: 0 = automatic, 1 or 2 */
    int mt;               /* 0 / 1 = one 128-pixel tile per CTA tile; 2 = two 128-pixel sub-tiles per tile (256 pixels), each weight
                           * tile that reaches shared memory feeds both: half the weight traffic per flop.  2 x mt x BLOCK_N <= 512. */
    int producers;        /* TMA producer warps per CTA: 0 = default (2), 1 or 2.  A thread's bulk-tensor copies complete one after the
                           * other, so a CTA that owns its SM needs several issuing threads to keep the operand ring full. */
    int splits;           /* 0 / 1 = off; k > 1 = split-K: k work units per tile accumulate disjoint K ranges, park fp32 partial sums
                           * in a plan-owned workspace, and the last unit to arrive reduces them in split order (deterministic) and
                           * runs the epilogue -- for the 20 x 20 / 40 x 40 maps whose tile count cannot fill 148 SMs. */
} b2t_conv_desc;
typedef struct b2t_conv_plan b2t_conv_plan;
const char* b2t_conv_last_error(void);
int b2t_conv_plan_create(const b2t_conv_desc* d, b2t_conv_plan** out_plan);
void b2t_conv_plan_destroy(b2t_conv_plan* plan);
double b2t_conv_plan_flops(const b2t_conv_plan* plan);
/* launch geometry chosen at plan time: out[0..17) = grid, threads, dynamic smem bytes, BLOCK_N, ring stages, mt, splits, halo,
 * halo buffers, tiles_m, tiles_n, TMEM columns, producer warps, taps per stage, resident weights, staging boxes, K chunks per stage (diagnostics for the autotuner and the per-layer tables in profiles/). */
int b2t_conv_plan_info(const b2t_conv_plan* plan, int* out, int n);
int b2t_conv_run(const b2t_conv_plan* plan, void* stream);
/* diagnostic builds (-DB2T_CONV_TRACE): per-CTA cycle counters of the MMA warp [total, ring wait, TMEM wait, halo wait, operand wait,
 * issue] and of the epilogue groups; returns the number of CTAs copied, 0 in normal builds */
int b2t_conv_plan_trace(const b2t_conv_plan* plan, long long* out_host, int max_ctas);

/* ---------------------------------------------------------------- detector glue + NMS (csrc/b2t_detect.cu) */
const char* b2t_detect_last_error(void);
/* ReOrg (models/common.py:48-53) fused with NCHW fp32 -> NHWC bf16 / fp16 (act_dtype); out [B][H/2][W/2][16] (12 used, 4 zero). */
int b2t_image_reorg(const float* img, void* out, int B, int H, int W, int act_dtype, void* stream);
/* same, into rows of row_pixels (>= W/2 + x0) pixels starting at pixel x0: the other pixels are not written (the caller
 * zeroes the buffer once) -- the padded layout the row-packed stem conv reads. */
/* float image [B][3][H][W] in [0, 1] -> NHWC 16-bit, 3 channels padded to 16: the input of a first convolution that reads the image
 * itself (YOLOv7-tiny, cfg/deploy/yolov7-tiny.yaml:15; w6 starts with ReOrg instead) */
int b2t_image_nhwc16(const float* img, void* out, int B, int H, int W, int act_dtype, void* stream);
int b2t_image_reorg_padded(const float* img, void* out, int B, int H, int W, int row_pixels, int x0, int act_dtype, void* stream);
/* nn.Upsample(None, 2, 'nearest'): src [B][H][W] slice (pitch, coff) -> dst [B][2H][2W] slice, C channels (bf16). */
int b2t_upsample2x(const void* src, int src_pitch, int src_coff, void* dst, int dst_pitch, int dst_coff, int B, int H, int W,
                   int C, void* stream);
/* SPPCSPC max-pools (models/common.py:271,278): reads channels [0,C) of buf, writes pool5 / 9 / 13 to [C,2C) [2C,3C) [3C,4C). */
int b2t_spp_pool(void* buf, int pitch, int C, int B, int H, int W, int act_dtype, void* stream);
/* Detect.forward inference decode (models/yolo.py:44-55) of one level: raw [B][H][W][raw_pitch] fp32 (channel a*no+o)
 * -> rows level_off + (a*H + y)*W + x of pred [B][n_total][no].  anchors_host: 6 floats (w,h) x 3 in pixels. */
int b2t_detect_decode(const float* raw, int raw_pitch, float* pred, int B, int H, int W, int na, int no, long long level_off,
                      long long n_total, float stride, const float* anchors_host, void* stream);
/* utils/general.py:607-695 non_max_suppression (best-class path, class-offset boxes, torchvision.ops.nms greedy rule,
 * max_nms cap, max_det cap; csrc/b2t_nms.cu).  pred [B][N][no] fp32 -> out [B][max_det][6] (x1 y1 x2 y2 conf cls),
 * out_count [B]; rows >= out_count[b] are not written.  post != 0 also applies scale_coords (gain, pad) + clip to
 * (img_w, img_h) + round (tracker/track.py:239-240).  0 <= conf_thres, max_det <= 2048, max_cand bounds the rows
 * that may pass the filter (extra ones are dropped: size it N to be exact). */
size_t b2t_nms_workspace_bytes(int B, int max_cand, int max_nms);
int b2t_nms(const float* pred, int B, int N, int no, float conf_thres, float iou_thres, int max_det, int max_nms, int max_cand,
            int post, float gain, float padw, float padh, float img_w, float img_h, void* workspace, size_t workspace_bytes,
            float* out, int* out_count, void* stream);
/* Detect.forward's inference decode (models/yolo.py:44-55) fused with non_max_suppression (utils/general.py:607-695):
 * what `non_max_suppression(model(img)[0], conf_thres, iou_thres)` returns, computed from the raw head maps without
 * materialising the (B, N, no) prediction tensor.  Level k: raw [B][h][w][raw_pitch] fp32 (channel a*no + o, 3 anchors),
 * anchors = (w,h) x 3 in pixels, level_off = first prediction row of the level (rows (a*h + y)*w + x follow).  Same
 * workspace, outputs and limits as b2t_nms. */
typedef struct b2t_head_level {
    const float* raw;
    int raw_pitch, h, w;
    float stride;
    float anchors[6];
    long long level_off;
} b2t_head_level;
int b2t_detect_nms(const b2t_head_level* levels, int n_levels, int B, int no, float conf_thres, float iou_thres, int max_det,
                   int max_nms, int max_cand, int post, float gain, float padw, float padh, float img_w, float img_h,
                   void* workspace, size_t workspace_bytes, float* out, int* out_count, void* stream);

/* ---------------------------------------------------------------- pre-processing (csrc/b2t_preproc.cu, SURVEY 8f row 2)
 * TrackerLoader._letterbox + __getitem__ (tracker/tracker_dataloader.py:64-130, 'v5' / 'v7' branch) for B uint8 BGR frames
 * of the same size already in device memory: cv2.resize(INTER_LINEAR) to (unpad_w, unpad_h) -- bit-exact 8-bit fixed-point
 * arithmetic, incl. OpenCV's 2 x 2 INTER_AREA shortcut -- placed at (top, left) of an (out_h, out_w) canvas filled with
 * pad_value (114), BGR -> RGB, HWC -> CHW, float32 / 255.  bgr: [B][src_h][src_pitch bytes]; out_chw: [B][3][out_h][out_w].
 * The geometry is the host arithmetic of :105-126 (b200track/preprocess.py: letterbox_geometry). */
int b2t_letterbox(const unsigned char* bgr, int B, int src_h, int src_w, int src_pitch, int unpad_w, int unpad_h, int top, int left,
                  int out_h, int out_w, int pad_value, float* out_chw, void* stream);
/* The same canvas written straight in the detector's input layout -- ReOrg (models/common.py:52-53) + NHWC bf16 padded to 16
 * channels, rows of row_pixels pixels starting at pixel x0 (what b2t_image_reorg_padded makes of the float tensor):
 * out_nhwc16 [B][out_h/2][row_pixels][16] bf16.  Same values as b2t_letterbox followed by b2t_image_reorg_padded. */
int b2t_letterbox_reorg(const unsigned char* bgr, int B, int src_h, int src_w, int src_pitch, int unpad_w, int unpad_h, int top, int left,
                        int out_h, int out_w, int pad_value, void* out_nhwc16, int row_pixels, int x0, int act_dtype, void* stream);

/* ---------------------------------------------------------------- camera-motion estimation (csrc/b2t_gmc.cu, SURVEY 8f row 1)
 * GMC.applyFeaures, method 'orb' (tracker/botsort.py:111-235; built by BoTSORT.__init__ :286 with downscale 2), for n_seq
 * sequences at once: BGR2GRAY + 1/downscale resize (:114-121), key-point mask = central 96 % of the frame minus the boxes of the
 * detections with score >= det_thresh (:123-130, what BoTSORT.update :380 passes), FAST(20) corners (:132), ORB descriptors of
 * those corners (:135), 2-NN Hamming matching against the previous frame (:149), ratio / spatial / 2.5 sigma filters (:158-198),
 * RANSAC partial affine (:221) -> warps_out[n_seq][6] = the 2 x 3 matrix in row-major order, translation at full resolution
 * (:224-226); identity on a sequence's first frame and when fewer than five matches survive (:221, :228).
 * frames_bgr: [n_seq][height][pitch bytes] uint8 BGR in device memory; dets: [n_seq][dmax][6] float (x1 y1 x2 y2 score cls, the NMS
 * output) with det_counts[n_seq], or NULL; the workspace (b2t_gmc_workspace_bytes, caller-owned, zeroed once by b2t_gmc_reset)
 * carries each sequence's previous key points and descriptors; max_kp caps the key points per frame (B2T_GMC_TRUNCATED in stat
 * when hit -- the reference has no cap).  stat: [n_seq][B2T_GMC_STAT_WORDS] ints (key points now / before, matches after the
 * ratio+spatial tests, after the sigma test, inliers of the best model, flags, best hypothesis, frame index) or NULL.
 * Never allocates, never synchronises; everything is enqueued on `stream`. */
#define B2T_GMC_STAT_WORDS 8
#define B2T_GMC_FIRST_FRAME 1
#define B2T_GMC_FEW_POINTS 2
#define B2T_GMC_TRUNCATED 4
size_t b2t_gmc_workspace_bytes(int n_seq, int height, int width, int downscale, int max_kp);
int b2t_gmc_reset(void* workspace, int n_seq, int height, int width, int downscale, int max_kp, void* stream);
int b2t_gmc_estimate(const unsigned char* frames_bgr, int n_seq, int height, int width, int pitch, int downscale, const float* dets,
                     const int* det_counts, int dmax, float det_thresh, void* workspace, int max_kp, double* warps_out, int* stat,
                     void* stream);
/* The same in two calls for pipelined callers: b2t_gmc_prepare needs only the frames (gray image, FAST scores, ORB's smoothed image
 * into plane set `slot`, 0 or 1), b2t_gmc_estimate_prepared needs only the detections; frame t + 1 may be prepared (other slot, other
 * stream) before frame t has been estimated.  Estimates must be enqueued in frame order. */
int b2t_gmc_prepare(const unsigned char* frames_bgr, int n_seq, int height, int width, int pitch, int downscale, void* workspace, int max_kp,
                    int slot, void* stream);
int b2t_gmc_estimate_prepared(int n_seq, int height, int width, int downscale, const float* dets, const int* det_counts, int dmax,
                              float det_thresh, void* workspace, int max_kp, int slot, double* warps_out, int* stat, void* stream);
/* tests / tools: byte offsets inside one sequence's workspace slice: out[0..9] = slice stride, state, gray, blurred, FAST score,
 * key points [2][max_kp] (x | y << 16), descriptors [2][max_kp][8 words], working height, working width, matched points */
int b2t_gmc_workspace_layout(int n_seq, int height, int width, int downscale, int max_kp, size_t* out, int n);

/* ---------------------------------------------------------------- appearance branch glue (csrc/b2t_reid.cu, SURVEY 8f row 3)
 * The reference's ReID extractor (tracker/reid_models/deepsort_reid.py:63-153: a ResNet-style net on 64 x 128 crops -> 512-d unit
 * vectors) runs as plans of the conv kernel above -- BatchNorm folded, act = 2 for ReLU -- plus these element-wise kernels; the cosine GEMM
 * of matching.embedding_distance (tracker/matching.py:84-103) is one more 1 x 1 plan.  All NHWC, 16-bit (act_dtype).
 * b2t_reid_crops: Extractor._preprocess :134-146 for n crops.  crops[i] = {byte offset of the crop's first pixel inside `pixels`, row
 *   pitch in bytes, height, width} (uint8 BGR, e.g. a window ori_img[y1:y2, x1:x2] of a frame, :301-303 of botsort.py): float / 255,
 *   cv2.resize to 64 x 128 (bilinear), Normalize -> out [n][128][64][16] (3 channels used). */
int b2t_reid_crops(const unsigned char* pixels, const long long* crops, int n, void* out_nhwc16, int act_dtype, void* stream);
/* nn.MaxPool2d(3, 2, padding=1) (:72): in [n][h][w][c] -> out [n][(h+1)/2][(w+1)/2][c], c a multiple of 8 */
int b2t_maxpool3x3s2(const void* in, void* out, int n, int h, int w, int c, int act_dtype, void* stream);
/* MP = nn.MaxPool2d(2, 2) of YOLOv7-tiny (models/common.py:30-35): in [n][h][w][c] -> out [n][h/2][w/2][c], h, w even, c a multiple of 8 */
int b2t_maxpool2x2s2(const void* in, void* out, int n, int h, int w, int c, int act_dtype, void* stream);
/* BasicBlock's F.relu(x.add(y)) (:49) over n_elems 16-bit values */
int b2t_add_relu(const void* a, const void* b, void* out, long long n_elems, int act_dtype, void* stream);
/* nn.BatchNorm2d with BATCH statistics -- the reference's extractor is never switched to eval() (deepsort_reid.py:112-121, :148-153), so
 * every call normalises with the mean and biased variance of that call's crops: y = (x - mean) / sqrt(var + eps) * gamma + beta
 * (+ ReLU) over x [n_pix][c]; sums_ws: 1024 doubles of scratch.  In place (y == x) is allowed. */
int b2t_batchnorm_batch_stats(const void* x, void* y, long long n_pix, int c, const float* gamma, const float* beta, float eps, int relu,
                              double* sums_ws, int act_dtype, void* stream);
/* nn.AvgPool2d over the whole hw-position map (:83) + division by the L2 norm (:103-104): in [n][hw][512] -> out [n][512] fp32 */
int b2t_avgpool_l2norm(const void* in, float* out, int n, int hw, int c, int act_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif
