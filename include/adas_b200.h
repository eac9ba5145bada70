/*
 * adas_b200.h -- C ABI of libadas_b200.so: the B200-native (sm_100a) replacement for the
 * ONNXRuntime / TensorRT dispatch behind the reference's coreEngine.py, plus the fused
 * per-frame post-processing (YOLO decode + NMS, UFLDv2 row/col-anchor decode, ByteTrack
 * IoU cost + linear assignment).
 *
 * Conventions
 *   - every entry point returns an int status: 0 = ok, non-zero = error; the message is
 *     available (thread-local) through adas_last_error().
 *   - plain pointers and sizes only; no torch / numpy types.  "host" pointers are ordinary
 *     (pageable or pinned) CPU memory, "dev" pointers are CUDA device memory on the handle's
 *     device (e.g. a torch CUDA tensor's data_ptr()).
 *   - a handle owns one device + one private CUDA stream; calls on one handle are serialised
 *     and synchronous (results are on the host / complete on return) unless the function name
 *     ends in _async.  This mirrors TensorRTBase.inference (reference coreEngine.py:93-118:
 *     H2D memcpy -> execute -> D2H memcpy -> stream.synchronize()).
 *
 * Each entry point cites the reference interface it replaces (paths relative to the
 * reference repo root).
 */
#ifndef ADAS_B200_H
#define ADAS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct adas_engine adas_engine;   /* opaque: one plan (network) on one device */

/* model kinds stored in the plan header */
enum { ADAS_MODEL_YOLOV8 = 0, ADAS_MODEL_YOLOV5 = 1, ADAS_MODEL_UFLDV2 = 2,
       /* adas_yolo_postprocess only: `raw` is the sigmoid-only head of a YOLOv5-lite export; YoloLiteParameters.lite_postprocess
        * (ObjectDetector/yoloDetector.py:36-50, model_type == ObjectModelType.YOLOV5_LITE) runs on the device first.  A lite PLAN
        * is a YOLOV5 plan whose header meta[2] != 0 (adas_engine_meta). */
       ADAS_MODEL_YOLOV5_LITE = 3,
       ADAS_MODEL_UFLDV1 = 4 };   /* UFLD v1 plans (ultrafastLaneDetector.py): one head tensor [griding_num + 1, rows, 4] */

/* ---- errors ------------------------------------------------------------------------- */
/* replaces: Python `raise Exception(...)` in coreEngine.py:12-14,20,26 */
const char* adas_last_error(void);
int         adas_version(void);
/* number of CUDA kernels launched by this library in this process (all handles) */
int64_t     adas_launch_count(void);

/* ---- engine lifecycle ------------------------------------------------------------------
 * replaces: TensorRTEngine.__init__ / OnnxEngine.__init__ (coreEngine.py:122-142,161-170):
 * deserialize a plan file (.b200w, produced by the packer), allocate device buffers for
 * batches up to max_batch, create the stream.  `device` replaces the hard-coded
 * cuda.Device(0) (coreEngine.py:47).  conv_impl: 0 = tcgen05 implicit-GEMM (product path),
 * 1 = plain SIMT CUDA-core kernel (validation path for tests; same plan, same buffers). */
int adas_engine_create(const char* plan_path, int device, int max_batch, int conv_impl,
                       adas_engine** out);
int adas_engine_destroy(adas_engine* e);

/* replaces: get_engine_input_shape / get_engine_output_shape (coreEngine.py:144-148,178-182).
 * in_shape4 = [N(=1), C, H, W].  out_shapes: n_out rows of 4 int64 (unused dims = 0),
 * out_ranks[n_out].  Shapes are per batch-1 like the reference bindings. */
int adas_engine_model_kind(const adas_engine* e, int* kind);
/* plan header meta word `idx` (0..15): YOLO [0] = classes, [1] = anchors, [2] = lite head (YOLOV5_LITE);
 * UFLD [0..5] = grid / class-row / lane dims, [6] = dataset (0 CULane, 1 TuSimple), see csrc/plan.h */
int adas_engine_meta(const adas_engine* e, int idx, int* value);
int adas_engine_input_shape(const adas_engine* e, int64_t in_shape4[4]);
int adas_engine_num_outputs(const adas_engine* e, int* n_out);
int adas_engine_output_shape(const adas_engine* e, int idx, int64_t shape4[4], int* rank);

/* replaces: engine_inference(input_tensor) (coreEngine.py:150-157,184-186).
 * input: fp32 NCHW [batch,C,H,W] on the HOST; outs[i]: HOST fp32 buffers the caller
 * allocated with batch * prod(shape_i[1:]) elements.  H2D, the network, the head decode
 * (YOLOv8: DFL+dist2bbox+sigmoid -> [batch,84,8400]; YOLOv5: sigmoid/grid/anchor ->
 * [batch,25200,85]; UFLDv2: the 4 head tensors) and D2H all happen inside the call. */
int adas_engine_infer(adas_engine* e, const float* input_nchw_host, int batch,
                      float* const* outs_host);
/* same, but input and outputs are DEVICE pointers (no PCIe traffic; used by bench `value`) */
int adas_engine_infer_dev(adas_engine* e, const float* input_nchw_dev, int batch,
                          float* const* outs_dev);

/* ---- fused YOLO detect ------------------------------------------------------------------
 * replaces YoloDetector.DetectFrame up to (not including) RectInfo construction
 * (ObjectDetector/yoloDetector.py:96-168, ObjectDetector/utils.py:42-87,161-256):
 * letterbox (cv2-exact fixed-point bilinear, pad 114) + BGR->RGB/255 + network + head decode
 * + per-anchor argmax / strict score threshold / ordered compaction + box un-letterboxing
 * + the reference's class-agnostic "soft" NMS (hard suppression, +1 area convention,
 * duplicate-emitting swap) -- all on the device.
 *   frames: batch x H x W x 3 uint8 BGR (host or device per `frames_on_device`)
 *   outputs (host): for frame b, count[b] kept detections in NMS emission order;
 *     boxes_xywh[b*max_det*4 ...] float32 (x,y,w,h in source-image pixels),
 *     scores[b*max_det ...] float32, class_ids[b*max_det ...] int32,
 *     cand_index[b*max_det ...] int32 = index into the pre-NMS candidate list (may repeat).
 *   n_candidates[b] (optional, may be NULL): number of pre-NMS candidates.
 * box_score / nms_iou are doubles because the reference compares float32 scores against the
 * Python-float (float64) thresholds (yoloDetector.py:128, utils.py:249). */
int adas_yolo_detect(adas_engine* e, const uint8_t* frames, int frames_on_device, int batch,
                     int H, int W, double box_score, double nms_iou, int max_det,
                     float* boxes_xywh, float* scores, int32_t* class_ids,
                     int32_t* cand_index, int32_t* counts, int32_t* n_candidates);

/* post-processing only, from a raw head tensor already on the host (parity tests for
 * rows E,F,N of SURVEY 8a without the network): raw is [batch,84,A] (kind YOLOv8, channel
 * major) or [batch,A,5+nc] (kind YOLOv5).  Letterbox geometry as Scaler would record it. */
int adas_yolo_postprocess(int device, const float* raw_host, int model_kind, int batch,
                          int n_anchors, int n_classes, int in_h, int in_w, int src_h, int src_w,
                          double box_score, double nms_iou, int max_det, float* boxes_xywh,
                          float* scores, int32_t* class_ids, int32_t* cand_index,
                          int32_t* counts, int32_t* n_candidates);

/* letterbox pre-processing alone (rows A,B): frames u8 BGR host -> fp32 NCHW host blob */
int adas_yolo_preprocess(int device, const uint8_t* frames_host, int batch, int H, int W,
                         int in_h, int in_w, float* blob_nchw_host);

/* ---- fused UFLDv2 lane detect ------------------------------------------------------------
 * replaces UltrafastLaneDetectorV2.DetectFrame up to lanes_points / lanes_status
 * (TrafficLaneDetector/ufldDetector/ultrafastLaneDetectorV2.py:96-181).
 *   outputs (host): pts[b][lane(4)][max_pts(=max(num_cls_row,num_cls_col))][2] int32,
 *   npts[b][4] int32, status[b][4] uint8; lane order left-side, left-ego, right-ego,
 *   right-side (ultrafastLaneDetectorV2.py:143-145,181).  coords_f (optional) receives the
 *   pre-truncation float64 coordinate of the expectation axis for tolerance tests. */
int adas_ufld_detect(adas_engine* e, const uint8_t* frames, int frames_on_device, int batch,
                     int H, int W, int32_t* pts, int32_t* npts, uint8_t* status,
                     double* coords_f);

/* adas_detect_pair: one call = adas_yolo_detect followed by adas_ufld_detect on the same frames (demo.py:269,280 run
 * both detectors on every frame).  Exists so a host thread that pipelines the tracker needs the interpreter lock once
 * per batch; argument meaning as in the two functions above. */
int adas_detect_pair(adas_engine* yolo, adas_engine* ufld, const uint8_t* frames, int frames_on_device, int batch,
                     int H, int W, double box_score, double nms_iou, int max_det, float* boxes_xywh,
                     float* scores, int32_t* class_ids, int32_t* cand_index, int32_t* counts,
                     int32_t* n_candidates, int32_t* pts, int32_t* npts, uint8_t* status);

/* decode only, from the 4 head tensors concatenated per frame ([batch, total_dim] fp32 host,
 * order loc_row, loc_col, exist_row, exist_col) */
int adas_ufld_postprocess(int device, const float* heads_host, int batch, int num_grid_row,
                          int num_cls_row, int num_grid_col, int num_cls_col, int num_lanes,
                          int img_w, int img_h, const double* row_anchor,
                          const double* col_anchor, int32_t* pts, int32_t* npts,
                          uint8_t* status, double* coords_f);

/* ---- lane geometry downstream of the lane decode (SURVEY 8f rank 1) --------------------------------------------------------
 * Replaces, per frame: LaneDetectBase.__update_lanes_status / __update_lanes_area / __adjust_lanes_points
 * (TrafficLaneDetector/ufldDetector/core.py:102-158: ego-lane polygon, optional degree-2 np.polyfit resampling on
 * np.linspace(miny, maxy, image_height)), PerspectiveTransformation.transformToBirdViewPoints
 * (perspectiveTransformation.py:120-142) and the arithmetic of calcCurveAndOffset (perspectiveTransformation.py:145-208; the
 * arrows and text it draws on the bird-view image stay with the host drawing code). */
typedef struct adas_lane_geom {
    int32_t area_status;   /* LaneInfo.area_status: both ego lanes detected */
    int32_t n_area;        /* points of the ego-lane polygon: left ++ flipud(right) */
    int32_t n_bird[4];     /* bird-view points per lane (0 when no matrix was given) */
    int32_t direction;     /* curvature_direction: -1 "L", 0 "F", 1 "R", 2 = None (an ego lane is missing) */
    int32_t pad;
    double curvature;      /* metres; valid when direction != 2 */
    double offset;         /* distance_from_center, metres; valid when direction != 2 */
} adas_lane_geom;

/* From host arrays shaped like adas_ufld_detect's outputs: pts [batch,4,max_pts,2] int32, npts [batch,4], status [batch,4].
 * M: [batch,9] row-major float64 frontal->bird-view matrices (PerspectiveTransformation.M after updateTransformParams) or NULL to
 * skip the bird view.  area: [batch,cap_area,2] (cap_area >= 2*max_pts, and >= 2*img_h with adjust_lanes), bird: [batch,4,max_pts,2]. */
int adas_lane_geometry(int device, const int32_t* pts, const int32_t* npts, const uint8_t* status, int batch, int max_pts, int img_w,
                       int img_h, int adjust_lanes, const double* M, int bird_w, int bird_h, int32_t* area, int cap_area, int32_t* bird,
                       adas_lane_geom* out);
/* Same, on the lane points the engine's last adas_ufld_detect / adas_detect_pair left on the device (no upload of the points). */
int adas_ufld_lane_geometry(adas_engine* e, int batch, int img_w, int img_h, int adjust_lanes, const double* M, int bird_w, int bird_h,
                            int32_t* area, int cap_area, int32_t* bird, adas_lane_geom* out);

/* cv2.warpPerspective(frame, M, (out_w, out_h), flags=cv2.INTER_LINEAR) for a batch of BGR u8 frames, bit-exact (constant black
 * border): PerspectiveTransformation.transformToBirdView / transformToFrontalView (perspectiveTransformation.py:90-117).
 * M: [batch,9] row-major float64 forward matrices (the function inverts them as cv2 does); out: [batch,out_h,out_w,3]. */
int adas_warp_perspective(int device, const uint8_t* frames_host, int batch, int H, int W, const double* M, int out_h, int out_w,
                          uint8_t* out_host);
/* Same, on the frames the engine's last detect call processed (still on the device: staged by the call, or the caller's device
 * pointer when it passed frames_on_device = 1 and has not overwritten them). */
int adas_engine_warp_perspective(adas_engine* e, int batch, const double* M, int out_h, int out_w, uint8_t* out_host);

/* UFLD v1 decode only (UltrafastLaneDetector.__process_output, ultrafastLaneDetector.py:97-136): head [batch, (griding_num+1)*rows*4]
 * fp32 host; cfg_w / cfg_h = ModelConfig.img_w / img_h, row_anchor[rows] in input-row coordinates.  pts [batch,4,rows,2]. */
int adas_ufld_v1_postprocess(int device, const float* head_host, int batch, int griding_num, int rows, int in_w, int in_h, int cfg_w,
                             int cfg_h, int img_w, int img_h, const double* row_anchor, int32_t* pts, int32_t* npts, uint8_t* status,
                             double* coords_f);

/* UFLD pre-processing alone (row H): u8 BGR host -> fp32 NCHW host [batch,3,in_h,in_w] */
int adas_ufld_preprocess(int device, const uint8_t* frames_host, int batch, int H, int W,
                         int in_h, int in_w, double crop_ratio, float* blob_nchw_host);

/* ---- ByteTrack association kernels -------------------------------------------------------
 * adas_iou_cost replaces matching.iou_distance (+ optional fuse_score)
 * (ObjectTracker/byteTrack/matching.py:34-80,108-116): cost[t*D+d] = 1 - iou(a_t, b_d)
 * (no +1 convention), fused: 1 - iou * det_score[d].  float64 in/out, host pointers.
 * `problems` independent (T_i x D_i) problems are batched: offsets arrays have
 * problems+1 entries (box offsets in units of boxes; cost offsets in elements). */
int adas_iou_cost(int device, int problems, const double* a_tlbr, const int32_t* a_off,
                  const double* b_tlbr, const int32_t* b_off, const double* det_scores,
                  int fuse, double* cost, const int64_t* cost_off);

/* adas_lap replaces matching.linear_assignment -> lap.lapjv(cost, extend_cost=True,
 * cost_limit=thresh) (matching.py:20-31): exact minimum of
 *   sum(cost[matched]) + thresh/2 * (#unmatched rows + #unmatched cols).
 * x[t] = matched column or -1, y[d] = matched row or -1. One warp per problem. */
int adas_lap(int device, int problems, const double* cost, const int64_t* cost_off,
             const int32_t* T, const int32_t* D, const double* thresh, int32_t* x,
             const int32_t* x_off, int32_t* y, const int32_t* y_off);

/* adas_associate: one association stage of BYTETracker.update in a single call -- replaces the sequence
 * iou_distance -> [fuse_score] -> linear_assignment (ObjectTracker/byteTrack/byteTracker.py:105-108,129-130,
 * 149-152).  a_tlbr [T,4], b_tlbr [D,4], det_scores [D] (used when fuse != 0), float64 host pointers.
 * Outputs: x[T], y[D] as adas_lap; cost_out (optional, may be NULL) receives the T*D cost matrix. */
int adas_associate(int device, int T, int D, const double* a_tlbr, const double* b_tlbr,
                   const double* det_scores, int fuse, double thresh, int32_t* x, int32_t* y,
                   double* cost_out);

/* ---- native ByteTrack --------------------------------------------------------------------------------------------------
 * adas_tracker_* replace BYTETracker.__init__/update/reset and the STrack / KalmanFilter records
 * (ObjectTracker/byteTrack/byteTracker.py:31-60,62-185,187-200; dtypes/strack.py; dtypes/kalman_filter.py:55-226;
 * utils.py:9-69).  The three association stages of update() run on the device (iou_cost + lap kernels); Kalman
 * algebra (float64) and list bookkeeping run in host C++.  class ids are ints (the Python wrapper maps labels).
 * The track-id counter is process-global like BaseTrack._count (base_track.py:12); adas_tracker_reset zeroes it. */
typedef struct adas_tracker adas_tracker;
typedef struct adas_track {
    int32_t track_id, state /* 0 new 1 tracked 2 lost 3 removed */, is_activated, class_id;
    int32_t start_frame, frame_id, tracklet_len, pad /* BaseTrack._count when the record was written */;
    double score;
    double tlwh[4];      /* current box (Kalman state), top-left x, y, w, h */
    double mean[8];      /* Kalman mean (cx, cy, a, h, velocities) */
    double det_tlbr[4];  /* detection matched in the last update() of a tracked track (STrack.trajectories entry) */
    int32_t traj_frame;  /* frame_id at which det_tlbr was recorded (0 = never) */
    int32_t pad2;
} adas_track;
int adas_tracker_create(int device, double track_thresh, int track_buffer, double match_thresh, int frame_rate,
                        adas_tracker** out);
int adas_tracker_destroy(adas_tracker* t);
int adas_tracker_reset(adas_tracker* t);
/* one frame: boxes_xyxy [n,4] float64 (demo.py feeds int-truncated RectInfo.tolist("xyxy")), scores [n], class_ids [n];
 * writes up to max_out tracked tracks (tracked_stracks order) and their count */
int adas_tracker_update(adas_tracker* t, int n, const double* boxes_xyxy, const double* scores,
                        const int32_t* class_ids, int max_out, adas_track* out, int* n_out);
/* all frames of one pipeline step in one call (no interpreter work between frames): counts[n_frames] detections per frame,
 * boxes / scores / class ids concatenated in frame order; out holds n_frames * max_out records, n_out[f] the tracked-track count
 * of frame f (records beyond max_out are dropped from `out`, never from the tracker). */
int adas_tracker_update_batch(adas_tracker* t, int n_frames, const int32_t* counts, const double* boxes_xyxy,
                              const double* scores, const int32_t* class_ids, int max_out, adas_track* out, int32_t* n_out);
int adas_tracker_get(adas_tracker* t, int which /* 0 tracked, 1 lost, 2 removed */, int max_out, adas_track* out, int* n_out);
int adas_tracker_count(void);    /* BaseTrack._count */
/* Wall-clock accounting of adas_tracker_update_batch since the tracker was created: out4 = {frames, total ms, ms spent between the
 * association launch and its result (the device round trip), association launches}.  Diagnostic; no reference counterpart. */
int adas_tracker_stats(adas_tracker* t, double* out4);

/* ---- test hooks (no reference counterpart): raw access to the plan's activation buffers so single kernels can be
 * parity-tested.  Buffers are [batch * rows_per_img, C] matrices (fp16 or fp32) as described in csrc/plan.h. */
int adas_engine_num_buffers(const adas_engine* e, int* n);
int adas_engine_buffer_info(const adas_engine* e, int idx, int64_t info[5] /* rows_per_img, C, dtype, H, W */);
int adas_engine_write_buffer(adas_engine* e, int idx, const void* host, int64_t bytes);
int adas_engine_read_buffer(adas_engine* e, int idx, void* host, int64_t bytes);
int adas_engine_run(adas_engine* e, int batch);   /* replay the plan on whatever buffer 0 holds; synchronous */

/* ---- timing hooks (bench.py): CUDA events on the handle's own stream (torch.cuda.Event only sees torch's stream).
 * adas_engine_event_record records event `slot` (0..3) on e's stream; adas_event_elapsed_ms synchronises on both
 * events and returns the time between (ea, slot_a) and (eb, slot_b).  adas_engine_time_ops replays, `iters` times and
 * back to back between two events, only the plan ops whose type bit (1 << PlanOpType) is set in type_mask, and
 * returns the average milliseconds per replay plus the number of kernel launches per replay. */
int adas_engine_event_record(adas_engine* e, int slot);
int adas_event_elapsed_ms(adas_engine* ea, int slot_a, adas_engine* eb, int slot_b, float* ms);
int adas_engine_time_ops(adas_engine* e, int batch, unsigned type_mask, int iters, float* ms_per_iter, int* launches);
/* per-layer table: adas_engine_num_steps = launches of one plan replay at `batch`; adas_engine_time_step replays launch
 * `step` alone, `iters` times back to back between two events (operands L2-warm), and returns its plan op type and a
 * description of the GEMM shape / tile choice (empty for non-GEMM steps). */
int adas_engine_num_steps(adas_engine* e, int batch, int* n);
int adas_engine_time_step(adas_engine* e, int batch, int step, int iters, float* ms_per_iter, int* op_type, char* desc, int desc_cap);
/* adas_engine_step_tiles: the (BN, MT) tiles the tcgen05 GEMM of launch `step` could have run with at `batch` -- every candidate
 * the program build prepared and launched without error while timing, in cost-model order (with ADAS_B200_AUTOTUNE=0 or a
 * plan-forced tile: the one tile in use).  *chosen = index of the tile the program runs (-1 when *n = 0).  Writes at most `cap` entries; *n is
 * the full count, 0 for a step that is not a tcgen05 GEMM (FC weight stream, im2col, stem conv, SIMT kernel, chain steps). */
int adas_engine_step_tiles(adas_engine* e, int batch, int step, int cap, int* bn, int* mt, int* n, int* chosen);

/* ---- optional multi-GPU gather -------------------------------------------------------------
 * (no reference counterpart: the reference is single-GPU, SURVEY 8e; BASELINE configs[4] asks for an NCCL gather of boxes.)
 * One communicator per process (one process per GPU): rank 0 makes the id with adas_comm_unique_id and hands its 128 bytes to the
 * other ranks by any means (bench.py: torch.distributed broadcast at start-up); adas_comm_create joins (ncclCommInitRank) and owns a
 * private stream.  adas_comm_all_gather takes this rank's record block of one batch (host memory, bytes_per_rank bytes), returns
 * immediately and runs upload + ncclAllGather on that stream; adas_comm_sync waits for everything enqueued so far; adas_comm_read
 * copies the last gathered [world, bytes_per_rank] block to the host.  NCCL is bound with dlopen at the first call. */
typedef struct adas_comm adas_comm;
int adas_comm_unique_id(uint8_t id[128]);
int adas_comm_create(int device, int rank, int world, const uint8_t id[128], int64_t bytes_per_rank, adas_comm** out);
int adas_comm_destroy(adas_comm* c);
int adas_comm_all_gather(adas_comm* c, const void* host_src);
int adas_comm_sync(adas_comm* c);
int adas_comm_read(adas_comm* c, void* host_dst);
int adas_comm_info(adas_comm* c, int* nranks, int64_t* gathers);
int adas_engine_stream(const adas_engine* e, void** cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* ADAS_B200_H */
