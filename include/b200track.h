/* b200track -- C ABI of the B200-native tracker hot path (libb200track.so).
 *
 * The reference (ImChouOWO/A-lightweight-Unsupervised-Feature-Extractor-) is pure
 * Python and has no FFI layer of its own; its boundary for this path is a set of
 * Python callables (SURVEY.md section 8b).  Each entry point below is what a binding
 * for one of those callables would call; the callable it replaces is cited as
 * reference file:line.  INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless its
 *     name ends in _host; buffers are caller-owned; nothing is retained after return
 *     except inside a b200_tracker handle.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     calls are asynchronous on that stream unless documented otherwise.
 *   - return value: B200_OK (0) or a negative B200_E* code; no exception crosses the
 *     ABI; b200_last_error() returns a thread-local message for the last failure.
 *   - all kernels are sm_100a only; there is no CPU path.
 */
#ifndef B200TRACK_H_
#define B200TRACK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK            0
#define B200_EINVAL      (-1)   /* bad argument (shape, null pointer, unsupported value) */
#define B200_ECUDA       (-2)   /* CUDA runtime error (launch, copy, allocation)          */
#define B200_ECAPACITY   (-3)   /* a fixed capacity of a tracker handle would be exceeded */
#define B200_ENUMERIC    (-4)   /* NaN / -inf in a cost matrix (scipy raises ValueError)  */
#define B200_EINFEASIBLE (-5)   /* assignment infeasible (scipy raises ValueError)        */

#define B200_LAYOUT_NCHW 0
#define B200_LAYOUT_NHWC 1      /* torch.channels_last storage of a [B,C,H,W] tensor */

#define B200_DTYPE_F32 0
#define B200_DTYPE_F16 1

#define B200_EMB_DIM 128        /* embedding width the reference validates (mainTracking.py:109,267) */

int         b200_version(void);
const char* b200_last_error(void);
/* Number of kernels this library has launched in the calling process (for bench.py). */
int64_t     b200_launch_count(void);

/* ---- ROI Align ---------------------------------------------------------------
 * Replaces torchvision.ops.roi_align as called at tracking.py:214,
 * tracking_win.py:260, model/utils/inferScr/infer.py:163 and
 * model/utils/trainingScr/trainingCard.py:71.
 * feat: [B,C,H,W] float32 stored NCHW or NHWC; rois: [K,5] = (batch, x1, y1, x2, y2);
 * out: [K,C,PH,PW] float32 (NCHW, contiguous).  sampling_ratio <= 0 = adaptive.
 * A ROI whose batch index is outside [0,B) produces zeros (torchvision: undefined). */
int b200_roi_align_fwd_f32(const float* feat, int layout, int B, int C, int H, int W,
                           const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                           int sampling_ratio, int aligned, float* out, void* stream);

/* Same operator for float16 storage (the reference's live CUDA deployment runs the map in half precision,
 * tracking.py:177-178): feat and out are IEEE half, rois stay float32 (pass the reference's half-rounded
 * boxes converted to float), all arithmetic is float32 and the result is rounded to half once. */
int b200_roi_align_fwd_f16(const void* feat, int layout, int B, int C, int H, int W,
                           const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                           int sampling_ratio, int aligned, void* out, void* stream);

/* Extended form: element type as an argument (B200_DTYPE_*) and a choice of output layout.
 * out_layout = B200_LAYOUT_NCHW is the operator above; B200_LAYOUT_NHWC writes the patches as [K,PH,PW,C]
 * (torch.channels_last storage of a [K,C,PH,PW] tensor) -- the hand-off a channels_last encoder
 * (model/utils/encoder/card.py:24-41, first layers 1x1 / 3x3 convolutions) consumes without a copy, and the
 * layout in which this kernel's lane-per-channel accumulators store whole cache lines directly.  Same values
 * as the NCHW form, element for element. */
int b200_roi_align_fwd_ex(const void* feat, int dtype, int layout, int B, int C, int H, int W,
                          const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                          int sampling_ratio, int aligned, void* out, int out_layout, void* stream);

/* Backward of b200_roi_align_fwd_ex (torchvision's _roi_align_backward): ADDS d(loss)/d(feat) into grad_in.
 * grad_out: [K,C,PH,PW] of element type `dtype` (B200_DTYPE_F32 / _F16), stored NCHW or NHWC (grad_out_layout);
 * rois, spatial_scale, sampling_ratio, aligned: exactly as given to the forward call;
 * grad_in: float32 [B,C,H,W] in `layout` (NCHW or NHWC), caller-zeroed or holding a gradient to add to.
 * ROIs with a batch index outside [0,B) contribute nothing.  The summation order is not deterministic.
 * Half grad_out is read as stored and all arithmetic and accumulation is float32 (torchvision's half backward
 * accumulates with half atomics, so its result differs). */
int b200_roi_align_bwd_ex(const void* grad_out, int dtype, int grad_out_layout, const float* rois, int64_t K,
                          int PH, int PW, float spatial_scale, int sampling_ratio, int aligned,
                          float* grad_in, int layout, int B, int C, int H, int W, void* stream);

/* Box preparation in front of ROI Align, one launch: boxes [n, box_stride >= 4] float32 (first four columns xyxy; the
 * detector's NMS rows [x1,y1,x2,y2,conf,cls] qualify, yoloDetects2.py:135-157) -> rois [n,5] = (batch, x1, y1, x2, y2).
 * batch_index: int32 [n] or NULL (= 0, what both reference wrappers use: one map per call).
 *   B200_BOXES_INPUT    MainInfer.roi_align_from_input_boxes (tracking.py:209-213): boxes copied as they are; the
 *                       image -> map scaling is roi_align's spatial_scale.
 *   B200_BOXES_TRAINING PreProcess._preprocess_roi (model/utils/trainingScr/trainingCard.py:38-69): corners sorted,
 *                       scaled by Wf/img_w and Hf/img_h, clamped to [0, Wf-1] x [0, Hf-1], x2 >= x1 + enforce_min_size
 *                       (skipped when <= 0), clamped again; float32 operation for operation, NaN propagating like torch. */
#define B200_BOXES_INPUT    0
#define B200_BOXES_TRAINING 1
int b200_roi_boxes_prep_f32(const float* boxes, int64_t n, int box_stride, const int32_t* batch_index, int mode,
                            int img_h, int img_w, int Hf, int Wf, float enforce_min_size, float* rois, void* stream);

/* ---- appearance cost -----------------------------------------------------------
 * Replaces Tracking.build_C_app_topk (model/mainTracking.py:141-211).
 * bank: [M,T,128] float32 history banks, bank_len[M] valid rows per track (0 = the row
 * of ones at :180-186 unless fallback != NULL, then fallback[M,128] stands in as a
 * one-row bank); det: [N,128].  Rows are re-normalised as at :167-168,:188-189.
 * C_app: [M,ldc] float32 = 1 - mean(top-k over t of <bank_t, det_j>), k = min(topk, len).
 * use_topk_mean == 0 selects the max-sim variant (:203-204). */
int b200_app_cost_topk_f32(const float* bank, const int32_t* bank_len, const float* fallback,
                           const float* det, int M, int N, int T, int topk, int use_topk_mean,
                           float* C_app, int ldc, void* stream);

/* ---- box / confidence / total cost ------------------------------------------------
 * Replaces bbox_cost (model/utils/costTool/costCard.py:109-174), conf_cost (:178-203)
 * and the weighted sum of cal_cost (:264-268).  boxes are [.,4] xyxy float32, confs
 * float32; any output pointer may be NULL.  All matrices are [M,ldc] float32. */
int b200_pair_cost_f32(const float* C_app, const float* boxes_prev, const float* boxes_cur,
                       const float* conf_prev, const float* conf_cur, int M, int N,
                       float w_app, float w_bbox, float w_conf, float alpha, float beta,
                       float conf_eps, float* C_total, float* C_bbox, float* C_center,
                       float* C_scale, float* C_conf, int ldc, void* stream);

/* ---- batched Kalman filter -------------------------------------------------------
 * 8-state constant-velocity filter of model/utils/costTool/KalmanFilter.py:36-101 with
 * filterpy 1.4.5 predict/update semantics (mainTracking.py:343,400).  State is stored
 * as float64 x[M,8], P[M,8,8] plus stage[M] (uint8: number of updates so far, saturating
 * at 2), which selects the float32/float64 arithmetic the reference's numpy code would
 * have used at that point of a track's life (SURVEY.md section 8 row K).
 * q_diag[8], r_diag[4]: diagonals of Q and R (float32 values, as float).            */
int b200_kalman_init(const double* boxes_xyxy, int M, double* x, double* P, uint8_t* stage,
                     void* stream);                                  /* KalmanFilter.py:36-101 */
int b200_kalman_predict(double* x, double* P, const uint8_t* stage, int M, const float* q_diag,
                        double* pred_boxes_xyxy /* [M,4] or NULL: KalmanFilter.py:19-33 */,
                        void* stream);                               /* mainTracking.py:340-345 */
/* det_of_track[M]: index into meas[N,4] (float64) or -1 = no update for that track.  meas rows
 * are xyxy boxes (meas_is_z == 0; converted by bbox_xyxy_to_z, KalmanFilter.py:5-16) or already
 * (cx, cy, a, h) measurements (meas_is_z != 0; rounded to float32 like the reference's z). */
int b200_kalman_update(double* x, double* P, uint8_t* stage, int M, const int32_t* det_of_track,
                       const double* meas, int meas_is_z, const float* r_diag, void* stream);
                                                                     /* mainTracking.py:400 */
/* d2[M,ldd] float64 = squared Mahalanobis distance of every (track, box) pair
 * (KalmanFilter.py:105-116); if C != NULL, C[i,j] = inf_value where d2 > maha_thr
 * (Tracking.apply_kalman_gating, mainTracking.py:306-338). */
int b200_maha_gate(const double* x, const double* P, const uint8_t* stage, int M,
                   const double* boxes_xyxy, int N, const float* r_diag, double maha_thr,
                   float inf_value, float* C, int ldc, double* d2, int ldd, void* stream);

/* ---- assignment ----------------------------------------------------------------------
 * Replaces hungarian_assign (model/utils/costTool/hung.py:5-45): scipy's rectangular
 * LSAP (shortest augmenting path, float64 duals) on each of `batch` float32 matrices
 * C[b] = C + b*batch_stride, [M,ldc], followed by the cost <= cost_max filter.
 * col_of_row[b,M]: assigned column BEFORE the filter (-1 if the row is unassigned, tall
 * case); matched[b,M]: 1 where the pair passes the filter.  status[b]: B200_OK,
 * B200_ENUMERIC or B200_EINFEASIBLE.  Tie-breaking follows scipy exactly. */
int b200_lsap_f32(const float* C, int batch, int64_t batch_stride, int M, int N, int ldc,
                  double cost_max, int32_t* col_of_row, uint8_t* matched, int32_t* status,
                  void* stream);

/* ---- GPU-resident tracker ---------------------------------------------------------------
 * Replaces Tracking (model/mainTracking.py:45-610) for `n_streams` independent video
 * streams stepped together; one step = Tracking.update(obj) for every stream. */
typedef struct b200_tracker b200_tracker;

typedef struct b200_tracker_conf {      /* model/conf/conf.yaml:2-24, mainTracking.py:55-96 */
    double init_conf_min, w_app, w_bbox, w_conf, alpha, beta;
    double cost_max, ema_alpha, conf_update_min, cost_update_max, maha_thr, reid_only_cost_max;
    int32_t hist_max, emb_top_k, max_age, lost_reid_after;
} b200_tracker_conf;

int  b200_tracker_create(b200_tracker** out, int n_streams, int max_tracks, int max_dets,
                         const b200_tracker_conf* conf);
void b200_tracker_destroy(b200_tracker* t);
int  b200_tracker_reset(b200_tracker* t, void* stream);
/* Ints per stream in the result table, and its layout:
 *   [0] n_matches [1] n_unmatched_tracks [2] n_unmatched_dets [3] n_live (after the step)
 *   [4] next_id   [5] status (0 ok, B200_E*) [6] n_rows_main [7] n_rows_reid
 *   then matches (tid, det) x max_dets, unmatched track ids x max_tracks,
 *   unmatched det indices x max_dets -- in the order Tracking.update returns them (:607-610). */
int  b200_tracker_result_stride(const b200_tracker* t);
/* Live-track count and next track id of every stream as of the work queued on `stream` so far (copies 8 ints per
 * stream and synchronises the stream).  Callers that step with device-resident inputs (b200_tracker_step) use it
 * to learn how full the handle is; either pointer may be NULL. */
int  b200_tracker_live_counts(b200_tracker* t, int32_t* n_live_host, int32_t* next_id_host, void* stream);
/* Device-resident inputs: n_det[S] (-1 = stream idle this step, 0 = empty frame, :467-471),
 * boxes [S,max_dets,4] float64 xyxy, confs [S,max_dets] float64, embs [S,max_dets,128]
 * float32, frame_id[S].  result: device int32 [S, stride].
 * Capacity precondition: for every stream n_live + n_det <= max_tracks (a birth that finds no free slot is
 * dropped and reported as B200_ECAPACITY in the stream's status column; b200_tracker_live_counts tells n_live). */
int  b200_tracker_step(b200_tracker* t, const int32_t* n_det, const double* boxes,
                       const double* confs, const float* embs, const int32_t* frame_id,
                       int32_t* result, void* stream);
/* The same step from detections in the detector's / encoder's own layout (device pointers), K detections in any
 * stream order -- no host round trip and no padding on the caller's side (tracking.py:315-324 rebuilds host lists):
 *   boxes  : K rows at a stride of box_stride (>= 4) elements, first four = x1,y1,x2,y2 (the detector's NMS rows
 *            [x1,y1,x2,y2,conf,cls] qualify, yoloDetects2.py:135-157)
 *   confs  : K values at a stride of conf_stride (>= 1) elements (for NMS rows: boxes + 4, same stride)
 *   det_dtype (B200_DTYPE_F32 / _F16) applies to boxes and confs; both are widened to float64 exactly
 *   embs   : [K,128] contiguous rows of emb_dtype (F32 / F16; 16- / 8-byte aligned), widened to float32 exactly
 *   stream_index : int32 [K] (e.g. the ROI batch index) or NULL = every detection belongs to stream 0;
 *                  detections with an index outside [0,S) are ignored
 *   active : int32 [S] or NULL = every stream steps (a stream with no detection gets an empty frame, :467-471);
 *            0 = stream idle this step (state untouched, like n_det = -1 in b200_tracker_step)
 *   frame_id : int32 [S];  result : int32 [S, stride], exactly what b200_tracker_step writes
 *   track_of_det : int32 [K] or NULL: the track id detection k was matched to in this step, -1 otherwise (unmatched,
 *                  ignored, or in a stream that did not step; births are not reported, as :607-610 does not)
 * A stream's detections are taken in input order: the j-th detection of stream s in the input is det_idx j of that
 * stream in the result table, as if the caller had compacted them in order and called b200_tracker_step.
 * A stream with more than max_dets detections is not stepped (state untouched) and gets B200_ECAPACITY in its status
 * column; the other streams step normally.  Same capacity precondition as b200_tracker_step.
 * Three launches (pack, step, finish) through an input block owned by the handle: no allocation and no
 * synchronisation, so the call can be captured in a CUDA graph. */
int  b200_tracker_step_packed(b200_tracker* t, int64_t K, const void* boxes, int box_stride,
                              const void* confs, int conf_stride, int det_dtype, const void* embs, int emb_dtype,
                              const int32_t* stream_index, const int32_t* active, const int32_t* frame_id,
                              int32_t* result, int32_t* track_of_det, void* stream);
/* Same step with HOST buffers (pinned or pageable): copies inputs up, runs the step, copies
 * the result table back into result_host and synchronises the stream. */
int  b200_tracker_step_host(b200_tracker* t, const int32_t* n_det_host, const double* boxes_host,
                            const double* confs_host, const float* embs_host,
                            const int32_t* frame_id_host, int32_t* result_host, void* stream);
/* ---- Tracking's methods one by one (mainTracking.py:340-448) ------------------------------------------------
 * The reference exposes the pieces of update() as methods a caller may drive itself; these entry points are
 * those methods on one stream of a handle.  Host arrays in, synchronous (they synchronise `stream`); the fused
 * b200_tracker_step does not go through them.
 *   predict_all   (:340-345)  Kalman predict of every live track, last_bbox <- predicted box
 *   mark_missed   (:347-355)  miss_count += 1 for the listed track ids (unknown ids are skipped)
 *   purge_dead    (:357-360)  drops tracks with miss_count > max_age
 *   create_tracks (:362-373)  births for det_ids (caller's order) whose confidence >= init_conf_min; boxes [n_det,4],
 *                             confs [n_det], embs [n_det,128] are the frame's detections; returns the number created,
 *                             B200_ECAPACITY if the handle is full
 *   update_matched(:375-448)  per match (track id, detection index, cost = C_total[row, det]): Kalman update, last box /
 *                             confidence / frame / cost, age, miss reset, then -- if confidence >= conf_update_min, cost <=
 *                             cost_update_max and the posterior squared Mahalanobis distance <= maha_thr -- EMA embedding and
 *                             history-bank push.  B200_EINVAL if a track id is not live (the reference: KeyError). */
int  b200_tracker_predict_all(b200_tracker* t, int stream_idx, void* stream);
int  b200_tracker_mark_missed(b200_tracker* t, int stream_idx, const int32_t* track_ids_host, int n, void* stream);
int  b200_tracker_purge_dead(b200_tracker* t, int stream_idx, void* stream);
int  b200_tracker_create_tracks(b200_tracker* t, int stream_idx, const int32_t* det_ids_host, int n_ids,
                                const double* boxes_host, const double* confs_host, const float* embs_host,
                                int n_det, int frame_id, void* stream);
int  b200_tracker_update_matched(b200_tracker* t, int stream_idx, const int32_t* match_tid_host,
                                 const int32_t* match_det_host, const float* match_cost_host, int n_matches,
                                 const double* boxes_host, const double* confs_host, const float* embs_host,
                                 int n_det, int frame_id, double ema_alpha, double conf_update_min,
                                 double cost_update_max, double maha_thr, void* stream);

/* The same step without the wait (the reference's consumer is a queue, tracking.py:329): stages the inputs in a
 * pinned ring inside the handle and returns a ticket; at most four steps may be in flight.  The kernels run on
 * `stream`; the upload and the download of the result table run on two private streams of the handle, ordered with
 * `stream` by events, so the DMA of step k+1 / k-1 overlaps the kernels of step k.  b200_tracker_step_result blocks until THAT step's result table is on the host and copies
 * it out.  b200_tracker_step_host is exactly step_host_async followed by step_result. */
int  b200_tracker_step_host_async(b200_tracker* t, const int32_t* n_det_host, const double* boxes_host,
                                  const double* confs_host, const float* embs_host,
                                  const int32_t* frame_id_host, int64_t* ticket, void* stream);
int  b200_tracker_step_result(b200_tracker* t, int64_t ticket, int32_t* result_host);
/* step_host_async for callers whose detection arrays already sit in PAGE-LOCKED host memory (cudaHostAlloc,
 * cudaHostRegister, torch pin_memory -- e.g. the buffer the encoder's device->host copy lands in, tracking.py:315-324):
 * boxes / confs / embs ([S,max_dets,...], full shape) are read by DMA from where they are, with no staging copy, so they
 * must stay unchanged until the step's result has been collected; n_det_host / frame_id_host may be reused at once.
 * B200_EINVAL if an array is not page-locked.  Same ticket / result protocol as step_host_async. */
int  b200_tracker_step_pinned_async(b200_tracker* t, const int32_t* n_det_host, const double* boxes_pinned,
                                    const double* confs_pinned, const float* embs_pinned,
                                    const int32_t* frame_id_host, int64_t* ticket, void* stream);
/* Copies one stream's live tracks (ascending track id) to host arrays sized for max_tracks;
 * any pointer may be NULL.  bank is [n, hist_max, 128] oldest-first.  Returns n_live or <0. */
int  b200_tracker_export(b200_tracker* t, int stream_idx, int32_t* ids, double* x, double* P,
                         uint8_t* stage, float* ema, float* bank, int32_t* bank_len, int32_t* miss,
                         int32_t* age, double* last_bbox, double* last_conf, double* last_cost,
                         int32_t* next_id, void* stream);

/* Inverse of b200_tracker_export: replaces one stream's state by `n` tracks given in ascending track-id
 * order (host arrays, same layouts as export).  The arrays go through b200_tracker_import_device below as a
 * one-row image, with its checks: a malformed row returns B200_EINVAL and leaves the stream untouched.
 * b200_tracker_import_device does the same for any set of streams from device memory without a
 * synchronisation. */
int  b200_tracker_import(b200_tracker* t, int stream_idx, int n, const int32_t* ids, const double* x,
                         const double* P, const uint8_t* stage, const float* ema, const float* bank,
                         const int32_t* bank_len, const int32_t* miss, const int32_t* age,
                         const double* last_bbox, const double* last_conf, const double* last_cost,
                         int32_t next_id, void* stream);

/* Device-side image of the state of any set of streams: the layout of b200_tracker_export with a leading row
 * dimension (n_rows rows of cap track slots; a row's live tracks first, ascending track id).  Every pointer is a
 * device pointer; x, P, ema, bank and last_bbox must be 16-byte aligned. */
typedef struct b200_tracker_state {
    int32_t* n_live;        /* [n_rows] */
    int32_t* next_id;       /* [n_rows] */
    int32_t* ids;           /* [n_rows, cap] */
    double*  x;             /* [n_rows, cap, 8] */
    double*  P;             /* [n_rows, cap, 8, 8] */
    uint8_t* stage;         /* [n_rows, cap] (0..2) */
    float*   ema;           /* [n_rows, cap, 128] */
    float*   bank;          /* [n_rows, cap, hist_max, 128], oldest row first */
    int32_t* bank_len;      /* [n_rows, cap] */
    int32_t* miss;          /* [n_rows, cap] */
    int32_t* age;           /* [n_rows, cap] */
    double*  last_bbox;     /* [n_rows, cap, 4] */
    double*  last_conf;     /* [n_rows, cap] */
    double*  last_cost;     /* [n_rows, cap] */
    int32_t  n_rows, cap, hist_max;
} b200_tracker_state;

/* Image row r <-> handle stream streams[r] (device int32 [n_rows]; NULL = rows 0..S-1, then n_rows must be S).
 * status: device int32 [n_rows] or NULL, B200_OK or why the row was skipped.  Both calls are asynchronous on
 * `stream`, allocate nothing and never synchronise (capturable in a CUDA graph).
 * export: writes n_live, next_id and the live tracks of each row, exactly what b200_tracker_export writes (bank rows
 *   past bank_len zeroed); slots >= n_live are not touched.  B200_EINVAL: stream index outside [0,S);
 *   B200_ECAPACITY: more than cap live tracks (nothing of the row is written).
 * import: replaces each row's stream by the image and leaves the slot layout b200_tracker_import leaves, so the next
 *   step is bit-identical to one after a host import.  A row is validated before anything is written and skipped,
 *   its stream untouched, on: stream index outside [0,S) or named by another row, n_live < 0, ids not strictly
 *   ascending or outside [0, next_id), bank_len outside [0, hist_max], stage > 2 (B200_EINVAL);
 *   n_live > min(cap, max_tracks) (B200_ECAPACITY).  The image carries state only: hyper-parameters are the
 *   handle's. */
int  b200_tracker_export_device(b200_tracker* t, const int32_t* streams, const b200_tracker_state* img,
                                int32_t* status, void* stream);
int  b200_tracker_import_device(b200_tracker* t, const int32_t* streams, const b200_tracker_state* img,
                                int32_t* status, void* stream);

/* ---- result tables of all GPUs in one place, over NVLink peer memory (SURVEY.md section 8e) --------------------
 * The reference runs one inference process and hands every frame's matches to one consumer queue
 * (tracking.py:329, :363); with streams sharded over the GPUs of a node (one process per GPU) the per-stream result
 * tables have to meet again.  Every rank owns a receive ring of n_slots cells x world sources that its peers map
 * through CUDA IPC.  push: one kernel stores `bytes` of this rank's tables into cell (seq % n_slots, rank) of EVERY
 * rank's ring (plain 16-byte stores over NVLink / NVSwitch) and raises that cell's flag; it never waits for a peer
 * unless the cell still holds tables the peer has not collected (n_slots pushes ago).  collect: one kernel waits until
 * the cells of `seq` from all ranks are flagged, copies them to dst as [world][bytes] and acknowledges the slot.
 * Sequence numbers count from 0 and every rank pushes every sequence number; pushes of one handle go to one stream.
 * handle / connect: exchange the B200_IPC_HANDLE_BYTES-byte handles of all ranks (rank order) by any means
 * (torch.distributed all_gather in dist.py) and connect once.  All ranks must synchronise before destroy. */
typedef struct b200_peer_gather b200_peer_gather;
#define B200_IPC_HANDLE_BYTES 64
int  b200_peer_gather_create(b200_peer_gather** out, int rank, int world, int64_t bytes_per_rank, int n_slots);
int  b200_peer_gather_handle(b200_peer_gather* g, void* handle_host);
int  b200_peer_gather_connect(b200_peer_gather* g, const void* handles_host);
int  b200_peer_gather_push(b200_peer_gather* g, const void* src, int64_t bytes, int64_t seq, void* stream);
int  b200_peer_gather_collect(b200_peer_gather* g, void* dst, int64_t bytes, int64_t seq, void* stream);
void b200_peer_gather_destroy(b200_peer_gather* g);

#ifdef __cplusplus
}
#endif
#endif /* B200TRACK_H_ */
