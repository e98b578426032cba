/* vnect_b200 -- C ABI of the B200-native VNect per-frame hot path.
 *
 * The reference (XinArkh/VNect) has no FFI of its own: its seam is the Python class `VNectEstimator`
 * (src/estimator.py:16-142) on top of a TensorFlow session looked up by tensor name (src/estimator.py:62-66).
 * Each entry point below names the reference interface it replaces.  Plain pointers and sizes only; every buffer
 * passed in or out is owned by the caller, the handle owns device weights, workspaces and per-stream filter state.
 * All functions return 0 on success or a negative VNECT_E_* code; vnect_last_error() gives the message.
 * One handle = one device + one CUDA stream; a handle is not thread-safe (neither is the reference object).  A process
 * may hold handles on several devices: every entry point switches to its handle's device and restores the caller's.
 */
#ifndef VNECT_B200_H
#define VNECT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VNECT_OK 0
#define VNECT_E_INVALID (-1)      /* bad argument / wrong call order */
#define VNECT_E_CUDA (-2)         /* CUDA runtime or driver error, incl. no usable sm_100 device */
#define VNECT_E_WEIGHT (-3)       /* unknown variable name, wrong shape, or missing variable at finalize */
#define VNECT_E_ZERO_DT (-4)      /* repeated timestamp for a stream: the reference raises ZeroDivisionError
                                     (src/OneEuroFilter.py:66) */
#define VNECT_E_UNSUPPORTED (-5)
#define VNECT_E_NUMERIC (-6)      /* NaN / Inf in the CNN output maps: fp16 activations overflowed (un-normalised weights?) */

#define VNECT_JOINTS 21
#define VNECT_MAX_SCALES 4

typedef struct vnect_handle vnect_t;

typedef struct vnect_config {
  int32_t device;       /* CUDA device ordinal */
  int32_t box_size;     /* CNN input side, 368 in the reference (src/estimator.py:19); multiple of 16 */
  int32_t n_scales;     /* 1..VNECT_MAX_SCALES */
  double scales[VNECT_MAX_SCALES]; /* pyramid scales, each in (0, 1]; reference default {1, 0.85, 0.7}
                                      (src/estimator.py:32) */
  int32_t max_frames;   /* largest n_frames of one vnect_estimate call (forward batch = max_frames * n_scales) */
  int32_t max_streams;  /* number of independent temporal-filter slots (video streams) */
  int32_t max_input_h;  /* largest raw frame accepted by vnect_estimate; 0 = box_size */
  int32_t max_input_w;
  int32_t filters;      /* 1 = OneEuroFilter smoothing on (reference behaviour), 0 = raw joints */
} vnect_config;

/* replaces VNectEstimator.__init__ (src/estimator.py:27-68): allocates the device context; weights come next */
int vnect_create(vnect_t** out, const vnect_config* cfg);

/* replaces VNect.load_weights / assign_weights_from_dict (src/vnect_model.py:219-236): one call per TF variable, names
 * and layouts of src/caffe2pkl.py:57-76 ("<scope>/weights" HWIO, "<scope>/biases", "<scope>/kernel",
 * "bn5c_branch2a/{gamma,beta,moving_mean,moving_variance}").  Host pointer, copied.  res2c_branch2a/* is accepted
 * and ignored (dead in the reference graph, src/vnect_model.py:54-56). */
int vnect_set_weight(vnect_t* h, const char* tf_name, const float* data, const int64_t* shape, int32_t rank);

/* weight-file helper: CRC32C (Castagnoli) of a host buffer -- the per-tensor / per-block checksum of the TensorFlow
 * checkpoint the reference restores (src/estimator.py:55-60); used by vnect_b200/tf_checkpoint.py */
uint32_t vnect_crc32c(const void* data, uint64_t n);

/* folds batch norm, converts to fp16, packs for the tensor cores, builds the launch plan (what saver.restore +
 * graph import do in src/estimator.py:54-60) */
int vnect_finalize(vnect_t* h);

/* replaces sess.run([split_2:0..3], {Placeholder:0: batch}) (src/estimator.py:100-104):
 * nhwc float32 [n, S, S, 3] -> four float32 [n, S/8, S/8, 21] maps (heat-map, x, y, z).  Host pointers. */
int vnect_forward(vnect_t* h, const float* nhwc, int32_t n, float* hm, float* xm, float* ym, float* zm);

/* replaces VNectEstimator.__call__ (src/estimator.py:97-142) for n_frames independent frames of identical size:
 * bgr uint8 [n_frames][H][W][3] with row pitch `pitch` and frame stride `frame_stride` (bytes);
 * stream_ids[n_frames] select the filter slot of each frame (distinct within one call);
 * t2d / t3d [n_frames] are the two clock readings the reference takes per frame (src/estimator.py:84);
 * joints2d float64 [n_frames][21][2] = (row, col) in input-image pixels, joints3d float32 [n_frames][21][3] in mm,
 * root-relative.  All pointers are HOST pointers; copies are part of the call. */
int vnect_estimate(vnect_t* h, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                   int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d,
                   double* joints2d, float* joints3d);

/* pipelined form of vnect_estimate: enqueue one batch on submission lane 0 or 1 and return immediately; the H2D copy
 * of a lane overlaps the kernels of the other one.  bgr / joints2d / joints3d are HOST pointers that must stay valid
 * (pinned memory recommended) until vnect_wait(h, lane) returns.  Batches execute in submission order, so frames of one
 * stream may alternate between lanes.  vnect_estimate == vnect_submit(lane 0) + vnect_wait(lane 0). */
int vnect_submit(vnect_t* h, int32_t lane, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                 int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                 float* joints3d);
int vnect_wait(vnect_t* h, int32_t lane);

/* Tracked video streams: replaces the loop body of run_estimator.py:98-119 for n streams at once.  Every stream keeps a
 * crop box on the device; vnect_track crops each FULL frame by its stream's box (run_estimator.py:100), runs
 * VNectEstimator.__call__ on the crop, shifts joints_2d to full-frame coordinates (:104-105) and updates the box from the
 * joints (:110-119) -- no host round trip between frames.  vnect_track_set_box seeds a stream's box (what HOGBox does in
 * run_estimator.py:66-83).  frames: HOST uint8 [n][FH][FW][3]; joints2d are full-frame (row, col); boxes_used (optional)
 * int32 [n][4] = the (x, y, w, h) each frame was cropped with. */
int vnect_track_set_box(vnect_t* h, int32_t stream_id, int32_t x, int32_t y, int32_t w, int32_t hh);
int vnect_track_get_box(vnect_t* h, int32_t stream_id, int32_t* xywh);
int vnect_track(vnect_t* h, const uint8_t* frames, int32_t n_frames, int32_t FH, int32_t FW, int64_t pitch,
                int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                float* joints3d, int32_t* boxes_used);

/* same computation with the frames and the results resident in device memory (dev_bgr, dev_joints2d, dev_joints3d are
 * DEVICE pointers; stream_ids / t2d / t3d stay host arrays).  Asynchronous on the handle's stream. */
int vnect_estimate_device(vnect_t* h, const uint8_t* dev_bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                          int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d,
                          double* dev_joints2d, float* dev_joints3d);

/* YUV 4:2:0 frames, as video decoders write them.  A YUV frame gives exactly the results of the BGR frame
 * cv2.cvtColor(frame, COLOR_YUV2BGR_NV12) (or COLOR_YUV2BGR_I420) fed to the BGR entry point: BT.601 limited range,
 * one chroma pair per 2x2 luma block, no chroma interpolation.  The conversion is fused into the pre-processing; no
 * BGR copy of the frame is ever made.  H and W must be even.  All offsets are in bytes from the start of each frame
 * (frame i starts at frames + i * frame_stride); planes may carry row padding and the chroma plane may start after
 * padding rows, as in a hardware decoder's surface (u_offset = y_pitch * aligned_height).
 * cv2's contiguous layout of a [3H/2][W] array:
 *   NV12: y_pitch = uv_pitch = W, u_offset = H*W, v_offset = H*W + 1 (U and V interleaved)
 *   I420: y_pitch = W, uv_pitch = W/2, u_offset = H*W, v_offset = H*W + (H/2)*(W/2)
 * Refused with VNECT_E_INVALID before anything runs: an unknown format, reserved != 0, odd or too small / large H or W,
 * pitches smaller than a row, a negative offset, a chroma plane that starts inside the luma plane, NV12 with
 * v_offset != u_offset + 1. */
#define VNECT_FMT_NV12 1
#define VNECT_FMT_I420 2
typedef struct vnect_yuv_layout {
  int32_t format;        /* VNECT_FMT_NV12 or VNECT_FMT_I420 */
  int32_t reserved;      /* 0 */
  int64_t y_pitch;       /* bytes between luma rows, >= W */
  int64_t uv_pitch;      /* bytes between chroma rows: >= W (NV12), >= W/2 (I420) */
  int64_t u_offset;      /* bytes from a frame's start to its first U sample */
  int64_t v_offset;      /* bytes from a frame's start to its first V sample (NV12: u_offset + 1) */
  int64_t frame_stride;  /* bytes between frames */
} vnect_yuv_layout;

/* replaces cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) followed by VNectEstimator.__call__: vnect_submit for
 * HOST YUV frames (H x W pixels each; staged to the device at 1.5 bytes per pixel).  Completes with vnect_wait. */
int vnect_submit_yuv(vnect_t* h, int32_t lane, const uint8_t* frames, int32_t n_frames, int32_t H, int32_t W,
                     const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d, const double* t3d,
                     double* joints2d, float* joints3d);
/* replaces cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) followed by VNectEstimator.__call__, like
 * vnect_estimate_device: DEVICE frames (e.g. a decoder's output surfaces) and DEVICE results, asynchronous. */
int vnect_estimate_device_yuv(vnect_t* h, const uint8_t* dev_frames, int32_t n_frames, int32_t H, int32_t W,
                              const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d,
                              const double* t3d, double* dev_joints2d, float* dev_joints3d);
/* replaces cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) followed by the loop body of run_estimator.py:98-119, like
 * vnect_track: HOST full frames of FH x FW pixels, cropped by each stream's tracked box. */
int vnect_track_yuv(vnect_t* h, const uint8_t* frames, int32_t n_frames, int32_t FH, int32_t FW,
                    const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d, const double* t3d,
                    double* joints2d, float* joints3d, int32_t* boxes_used);

/* Mixed-size batches: frames of different sizes, pitches and addresses in one call, one vnect_frame each (a HOST
 * array, copied by the call).  One pixel format per call: VNECT_FMT_BGR, VNECT_FMT_NV12 or VNECT_FMT_I420.  Frame i
 * gives bit-for-bit what the uniform entry point gives for that frame alone (joints, raw argmax, tracked box, filter
 * state), so a multi-camera server can fill one batch from cameras of any resolution, and device frames need not be
 * gathered into one strided buffer.  CUDA graphs are keyed by the frame count and format only: every composition of
 * a batch replays the same graph.
 * Refused with VNECT_E_INVALID before anything is staged or launched and before any filter state is touched: n_frames
 * outside [1, max_frames], a null table or null data, an unknown format, a side below 2, a BGR pitch below 3 * width,
 * a YUV entry that fails the vnect_yuv_layout rules above (frame_stride does not apply), and for the HOST entry points
 * a frame larger than max_input.  Duplicate stream ids and repeated or earlier timestamps are refused as elsewhere. */
#define VNECT_FMT_BGR 0
typedef struct vnect_frame {
  const uint8_t* data;                   /* first byte of the frame (BGR) or of its luma plane (YUV) */
  int32_t height, width;                 /* this frame's size (the FULL frame for vnect_track_frames) */
  int64_t pitch;                         /* BGR row pitch, or luma pitch */
  int64_t uv_pitch, u_offset, v_offset;  /* YUV only, bytes relative to data, as in vnect_yuv_layout; 0 for BGR */
} vnect_frame;                           /* 48 bytes */

/* replaces VNectEstimator.__call__ (src/estimator.py:97-142), or cv2.cvtColor(YUV2BGR) followed by it, for n_frames
 * frames of any sizes: vnect_submit(_yuv) with one descriptor per HOST frame.  The frames are staged one after another
 * into the lane's device buffer.  Completes with vnect_wait. */
int vnect_submit_frames(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                        const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                        float* joints3d);
/* the same on DEVICE frames (e.g. one decoder surface or one tensor per camera) with DEVICE results, like
 * vnect_estimate_device(_yuv); asynchronous on the handle's stream.  The frames' pointers are used as they are. */
int vnect_estimate_device_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                                 const int32_t* stream_ids, const double* t2d, const double* t3d,
                                 double* dev_joints2d, float* dev_joints3d);
/* replaces the loop body of run_estimator.py:98-119 for streams whose full frames differ in size, like
 * vnect_track(_yuv): HOST full frames, each cropped by its stream's box clipped to that frame. */
int vnect_track_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                       const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                       float* joints3d, int32_t* boxes_used);

/* Pipelined and device-resident tracking: the loop body of run_estimator.py:98-119 without waiting for the GPU.
 * vnect_track / vnect_track_frames synchronise, so the upload of the next step's full frames cannot overlap this
 * step's kernels, and frames already in device memory would have to round-trip through the host.  The calls below
 * take the vnect_frame table of vnect_track_frames (same validation, same errors, in the same order) and return
 * once the work is enqueued.  Every tracked call runs on the handle's stream in submission order, so frame i of an
 * asynchronous call gives bit for bit what vnect_track_frames gives for the same submission order -- joints_2d,
 * joints_3d, boxes_used, the raw argmax, the box left behind, the filter state, the timestamps and the packed
 * results -- also when consecutive frames of one stream go to different lanes and when lane 1 is submitted before
 * lane 0 has been waited on.  A refused call stages and launches nothing and touches no box, filter state or
 * timestamp.  CUDA graphs are keyed by lane, frame count, format and output pointers, as for the other table calls:
 * a moving crop, a decoder's rotating surfaces and changing camera sizes replay the same graph.
 * vnect_track_set_box, vnect_track_get_box, vnect_reset_stream, vnect_get_raw_argmax and vnect_export /
 * import_stream_state keep their synchronous meaning: they act after everything already submitted.  Waiting for
 * the GPU there does not complete a lane: NaN / Inf maps of its batch are still reported by its vnect_wait. */

/* vnect_track_frames on submission lane 0 or 1, completed by vnect_wait(h, lane) like vnect_submit: HOST frames
 * (staged into the lane's buffer), HOST results (boxes_used optional).  frames' pixels, joints2d, joints3d and
 * boxes_used must stay valid until the wait (pinned memory makes the copies truly asynchronous); NaN / Inf maps are
 * reported by the wait or by the next use of the lane. */
int vnect_submit_track_frames(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                              const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                              float* joints3d, int32_t* boxes_used);
/* vnect_track_frames on DEVICE full frames (e.g. a decoder's surfaces or one tensor per camera, pointers used as they
 * are) with DEVICE results: dev_joints2d float64 [n][21][2], dev_joints3d float32 [n][21][3], dev_boxes_used
 * (optional) int32 [n][4].  Asynchronous on the handle's stream, like vnect_estimate_device_frames. */
int vnect_track_device_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                              const int32_t* stream_ids, const double* t2d, const double* t3d, double* dev_joints2d,
                              float* dev_joints3d, int32_t* dev_boxes_used);
/* vnect_track_set_box for n streams at once, in submission order: after every call already submitted and before
 * every later one, without the host waiting for the GPU.  stream_ids int32 [n] and xywh int32 [n][4] are HOST arrays,
 * copied by the call; n = 0 does nothing.  Refused before anything is enqueued: n below 0, a null array, and as
 * vnect_track_set_box refuses one box, an id outside [0, max_streams), an id given twice, x or y below 0, w or h
 * below 2. */
int vnect_track_set_boxes(vnect_t* h, int32_t n, const int32_t* stream_ids, const int32_t* xywh);

/* Frame orientation of a stream: a camera mounted sideways, upside down or mirrored.  A stream with orientation o
 * that is given stored frame F produces bit for bit what a stream with VNECT_ORIENT_IDENTITY produces for the
 * materialised frame orient(F, o): joints2d, joints3d, the raw argmax, the packed results, boxes_used, the box left
 * behind, the filter state and the timestamp mirror.  Every coordinate the caller sees is in the oriented frame
 * (joints2d, boxes of vnect_track_set_box(es) / vnect_track_get_box, boxes_used, frame_hw of vnect_track_postprocess);
 * a frame's data, height, width, pitches and chroma layout describe it as stored, and max_input and the YUV layout
 * rules apply to the stored frame.  The tracked box is clamped to the oriented frame's sides.
 * The codes, with the numpy definition that is the contract, for a stored frame f of H x W and oriented pixel (yo, xo)
 * read from stored pixel (ys, xs).  Codes 1, 3, 6 and 7 swap the frame's sides.  A YUV 4:2:0 frame is oriented as
 * the BGR image cv2.cvtColor gives (the same as converting oriented planes, H and W being even). */
#define VNECT_ORIENT_IDENTITY 0   /* f                                     (ys, xs) = (yo, xo)             */
#define VNECT_ORIENT_ROT90_CW 1   /* np.rot90(f, 3)                        (ys, xs) = (H-1-xo, yo)         */
#define VNECT_ORIENT_ROT180 2     /* np.rot90(f, 2)                        (ys, xs) = (H-1-yo, W-1-xo)     */
#define VNECT_ORIENT_ROT90_CCW 3  /* np.rot90(f, 1)                        (ys, xs) = (xo, W-1-yo)         */
#define VNECT_ORIENT_FLIP_H 4     /* f[:, ::-1] (mirror)                   (ys, xs) = (yo, W-1-xo)         */
#define VNECT_ORIENT_FLIP_V 5     /* f[::-1]                               (ys, xs) = (H-1-yo, xo)         */
#define VNECT_ORIENT_TRANSPOSE 6  /* f.transpose(1, 0, 2)                  (ys, xs) = (xo, yo)             */
#define VNECT_ORIENT_TRANSVERSE 7 /* np.rot90(f, 2).transpose(1, 0, 2)     (ys, xs) = (H-1-xo, W-1-yo)     */
/* Sets the orientation of n streams (HOST arrays stream_ids int32 [n] and codes int32 [n], copied by the call;
 * n = 0 does nothing).  Host-only, nothing is enqueued: every call submitted after it, on either lane, uses the new
 * codes, and calls already submitted keep the ones they were submitted with.  Orientation is configuration, not
 * temporal state: vnect_reset_stream keeps it and vnect_export / import_stream_state do not carry it, so a stream
 * moved to another handle needs its orientation set there too.  A call in which every frame's stream has
 * VNECT_ORIENT_IDENTITY runs exactly as before (same launches, graphs and kernels).
 * Refused with VNECT_E_INVALID, changing nothing: n below 0, a null array, an id outside [0, max_streams), an id
 * given twice, a code outside [0, 8). */
int vnect_set_orientations(vnect_t* h, int32_t n, const int32_t* stream_ids, const int32_t* codes);
/* the orientation of one stream */
int vnect_get_orientation(vnect_t* h, int32_t stream_id, int32_t* code);

/* Joint confidence.  score[f][j] of frame f and joint j is the float64 value the reference takes its argmax of in
 * utils.extract_2d_joints (src/utils.py:153-175): up = cv2.resize(hm_avg[:, :, j], (0, 0), fx=8, fy=8, INTER_LINEAR)
 * on the multi-scale float64 average hm_avg of src/estimator.py:105-129, score = up.flat[np.argmax(up)] == up.max().
 * Bit for bit the reference's value, unfiltered, in heat-map units; it depends only on the CNN maps, not on filters,
 * orientation, tracking or the order of a sequence.  A confidence, not a probability.
 * The NEXT call of vnect_estimate, vnect_submit(_yuv), vnect_estimate_device(_yuv), vnect_track(_yuv),
 * vnect_submit_frames, vnect_estimate_device_frames, vnect_track_frames, vnect_submit_track_frames,
 * vnect_track_device_frames, vnect_submit_sequence, vnect_estimate_device_sequence, vnect_postprocess,
 * vnect_postprocess_sequence or vnect_track_postprocess also writes float64 [n_frames][21] scores to `scores`: a HOST
 * pointer, filled when the call completes (vnect_wait for the submit calls), except for the *_device* calls, where it
 * is a DEVICE pointer written in stream order.  That call consumes the request whether it is accepted or refused; a
 * refused call writes nothing.  NULL cancels a pending request.  Each call carries its own buffer, so two lanes in
 * flight never share one, and a rotating pool of buffers replays the same CUDA graphs.  A call with no pending request
 * (and no recovering stream, below) runs exactly as before: same launches, graphs and kernels. */
int vnect_request_scores(vnect_t* h, double* scores);
/* Lost-person recovery of tracked streams.  Sets the least mean score min_mean_score[i] (HOST arrays, copied; n = 0
 * does nothing) of n streams; 0 = off, the default and the reference's behaviour.  When a tracked call processes
 * frame f of a stream whose threshold tau > 0, it computes m = (((s0 + s1) + s2) + ... + s20) / 21 over the frame's
 * scores in float64 without FMA (Python's sum(scores[f]) / 21).  If m < tau, the box left behind is the one
 * vnect_reset_stream leaves, (0, 0, 1 << 30, 1 << 30), so the stream's next frame is cropped to its whole (oriented)
 * frame; otherwise the box update of run_estimator.py:110-119 runs unchanged.  Frame f's joints, filters and
 * timestamps are untouched.  Configuration like the orientation: host-only, a call reads its streams' thresholds at
 * submission, vnect_reset_stream keeps them and the stream-state export / import does not carry them.  A tracked call
 * with a recovering stream runs the table pipeline (uniform calls build their frame table on the host).
 * Refused with VNECT_E_INVALID, changing nothing: n below 0, a null array, an id outside [0, max_streams), an id
 * given twice, a threshold that is negative, NaN or infinite. */
int vnect_set_track_recovery(vnect_t* h, int32_t n, const int32_t* stream_ids, const double* min_mean_score);
/* the recovery threshold of one stream (0 = off) */
int vnect_get_track_recovery(vnect_t* h, int32_t stream_id, double* min_mean_score);

/* Sequence calls: consecutive frames of one stream in one batch (offline video: annotating a dataset, re-processing a
 * recording, motion capture from footage).  Up to max_frames frames in which a stream id may appear more than once;
 * the frames of one stream are consecutive in time in the order they appear in the call, and may be interleaved with
 * other streams' frames.  Frame i gets bit for bit what the untracked entry points give when the frames go in one
 * at a time in call order: joints2d, joints3d, the raw argmax, the packed results, and afterwards every stream's
 * filter state and timestamp mirror.  The CNN runs over the whole call at batch size; each stream's 2D filters, the
 * location-map gather at the filtered points and the 3D filters are then walked in frame order on the GPU.  Tracked
 * streams cannot be batched this way: frame k+1's crop depends on frame k's joints.
 * stream_ids is required; with filters on, so are t2d and t3d (one reading per frame).  Validation runs before
 * anything is staged or launched: the vnect_frame table as for vnect_submit_frames, ids in [0, max_streams), and each
 * stream's readings walked in call order against its previous reading (before the call, then the call's own earlier
 * frames) with the rules of the other calls -- a repeated 2D or 3D reading is VNECT_E_ZERO_DT, an earlier one
 * VNECT_E_INVALID, a reading of 0 is never compared.  A refused call touches no filter state and no timestamp mirror:
 * unlike a frame-by-frame loop, which would already have processed the frames before the bad one, it processes none.
 * A stream may continue across sequence calls on either lane and across ordinary calls, in submission order.  CUDA
 * graphs are keyed by lane, frame count, format and output pointers: every composition of a batch replays the same
 * graph. */
/* vnect_submit_frames with repeated stream ids: HOST frames of any sizes (BGR, NV12 or I420), HOST results;
 * completes with vnect_wait(h, lane). */
int vnect_submit_sequence(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                          const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                          float* joints3d);
/* vnect_estimate_device_frames with repeated stream ids: DEVICE frames, DEVICE results, asynchronous on the handle's
 * stream. */
int vnect_estimate_device_sequence(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                                   const int32_t* stream_ids, const double* t2d, const double* t3d,
                                   double* dev_joints2d, float* dev_joints3d);
/* vnect_postprocess with repeated stream ids, a diagnostic on given maps (same layout and arguments as
 * vnect_postprocess, same validation as the sequence calls above).  Not graphed; synchronises before returning. */
int vnect_postprocess_sequence(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm,
                               int32_t n_frames, const int32_t* stream_ids, const double* t2d, const double* t3d,
                               double scaler, int32_t offset_x, int32_t offset_y, double* joints2d, float* joints3d,
                               int32_t* raw_argmax);

/* replaces VNectEstimator.gen_input_batch (src/estimator.py:70-81): out float32 [n_frames*n_scales][S][S][3]
 * (fp16-rounded values of the network input), scaler_offsets float64 [3] = {scaler, offset_x, offset_y} */
int vnect_preprocess(vnect_t* h, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                     int64_t frame_stride, float* out_nhwc, double* scaler_offsets);

/* replaces src/estimator.py:105-142 fed with given maps (host float32 NHWC [n_frames*n_scales][S/8][S/8][21] each);
 * scaler / offset_x / offset_y as returned by gen_input_batch.  raw_argmax (optional, may be NULL): int32
 * [n_frames][21][2] unfiltered (row, col) in box pixels. */
int vnect_postprocess(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm, int32_t n_frames,
                      const int32_t* stream_ids, const double* t2d, const double* t3d, double scaler, int32_t offset_x,
                      int32_t offset_y, double* joints2d, float* joints3d, int32_t* raw_argmax);
/* the tracked tail of vnect_track_frames (src/estimator.py:105-142 and run_estimator.py:100-119 after the CNN) fed
 * with given maps, laid out as for vnect_postprocess: each frame's geometry from its stream's box clipped to the frame,
 * the post-process with that geometry (joints2d in full-frame pixels), then the box update.  frame_hw: host int32
 * [n_frames][2] full-frame (height, width); boxes_used (optional): int32 [n_frames][4].  Validated like
 * vnect_track_frames (sides below 2, ids, duplicate ids, repeated or earlier timestamps); a refused call touches no
 * box, filter state or timestamp.  Not graphed; synchronises before returning.  The raw argmax is read with
 * vnect_get_raw_argmax. */
int vnect_track_postprocess(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm,
                            int32_t n_frames, const int32_t* frame_hw, const int32_t* stream_ids, const double* t2d,
                            const double* t3d, double* joints2d, float* joints3d, int32_t* boxes_used);

/* replaces VNectEstimator.joint_filter (src/estimator.py:83-95) on explicit values: one step of the 21*dim scalar
 * filters of a stream at clock reading t.  values: host float64 [21*dim], filtered in place.  values_are_f32 = 1 when
 * the caller's array is float32 (the reference's joints_3d, src/utils.py:186): the raw difference is then taken in
 * float32 and the results are rounded to float32; 0 for a float64 array (joints_2d).
 * Errors like the reference: a repeated timestamp is VNECT_E_ZERO_DT (ZeroDivisionError, src/OneEuroFilter.py:66), an
 * earlier one VNECT_E_INVALID (ValueError "alpha ... should be in (0.0, 1.0]", src/OneEuroFilter.py:21-22); both are
 * detected before the stream's state is touched.  The same checks guard vnect_estimate / vnect_submit / vnect_track. */
int vnect_filter(vnect_t* h, int32_t stream_id, int32_t dim, int32_t values_are_f32, double t, double* values);

/* replaces Joints2Angles.__call__ / joints2angles (src/joints2angles.py:44-110): the eight arm angles (radians:
 * s0_l, s1_l, e0_l, e1_l, s0_r, s1_r, e0_r, e1_r) of n frames from their 3D joints (host float32 [n][21][3], as
 * returned by vnect_estimate), smoothed per stream by the eight OneEuroFilters of joints2angles.py:35-42 when t
 * (host float64 [n] clock readings) is not NULL.  angles: host float64 [n][8]. */
int vnect_joints2angles(vnect_t* h, const float* joints3d, int32_t n, const int32_t* stream_ids, const double* t,
                        double* angles);

/* forget the temporal-filter state of one stream (a new VNectEstimator() in the reference); -1 = all streams */
int vnect_reset_stream(vnect_t* h, int32_t stream_id);

/* Temporal state of one stream as VNECT_STREAM_STATE_DOUBLES plain doubles: the 42 + 63 OneEuroFilter objects of
 * src/estimator.py:46-53 ({prev, s_x, s_dx, lasttime, freq, has_prev, has_time} each), the two last clock readings and
 * the tracked crop box.  Lets a caller move a stream to another handle / GPU or keep it across a rebuild of the device
 * context (the reference keeps one filter set for the lifetime of its estimator object). */
#define VNECT_STREAM_STATE_DOUBLES (7 * 21 * 5 + 6)
int vnect_export_stream_state(vnect_t* h, int32_t stream_id, double* state);
int vnect_import_stream_state(vnect_t* h, int32_t stream_id, const double* state);

/* Multi-GPU gather layout: when dev_packed (DEVICE pointer, float64 [max_frames][21][5]) is set, every later
 * estimate / submit / track call also writes (row, col, x, y, z) per joint there, straight from the post-process
 * kernel -- the buffer a caller hands to ncclAllGather (SURVEY.md section 8e).  NULL turns it off. */
int vnect_set_packed_results(vnect_t* h, void* dev_packed);

/* run on a caller-provided cudaStream_t (e.g. torch's current stream) instead of the handle's own */
int vnect_set_stream(vnect_t* h, void* cuda_stream);
int vnect_synchronize(vnect_t* h);

/* introspection for tests and benchmarks */
int vnect_get_tap(vnect_t* h, const char* name, int32_t n, float* out_nhwc, int64_t capacity_elems,
                  int32_t* dims4 /* n, H, W, C */);
/* the network input of the most recent call, as the stem reads it: the raw fp16 bits of the first n forwards,
 * uint16 [n][2 parities][S/2 + 3 rows][(S + 6) * 4], zero border and 4th channel included (pixel (y, x) of forward f
 * is at parity (y + 2) & 1, row (y + 2) >> 1, column (x + 2) * 4).  Synchronises the handle's stream.  A null `out`
 * only fills dims4. */
int vnect_get_input(vnect_t* h, int32_t n, uint16_t* out, int64_t capacity, int32_t* dims4 /* n, 2, rows, halves */);
/* the CNN output maps of the most recent call (or the maps vnect_postprocess / vnect_track_postprocess were given) as
 * the post-process reads them: planar float32 [n_frames*n_scales][84][S/8][S/8], channels hm 0..20, xm 21..41, ym
 * 42..62, zm 63..83.  Synchronises the handle's stream.  A null `out` only fills dims4. */
int vnect_get_maps(vnect_t* h, int32_t n_frames, float* out, int64_t capacity, int32_t* dims4 /* n, 84, hs, hs */);
/* unfiltered (row, col) argmax in box pixels of the frames of the most recent estimate / submit / track call
 * (what utils.extract_2d_joints returns, src/utils.py:153-175, before joint_filter): int32 [n_frames][21][2].
 * Waits for that call to complete.  Parity tests use it to prove that an argmax difference is a near-tie. */
int vnect_get_raw_argmax(vnect_t* h, int32_t n_frames, int32_t* raw_argmax);
/* fp16 safety net.  Every estimate / submit / track call counts NaN / Inf values met in the CNN's output maps and the
 * call that synchronises with that batch (vnect_wait, vnect_estimate, vnect_track, the next use of the lane) fails
 * with VNECT_E_NUMERIC instead of returning joints computed from garbage.  vnect_check_finite then scans the
 * activations of the last forward: counts[i] = values of launch i's output (first n forwards) that are NaN / Inf or
 * saturated (|x| >= 65504); counts has one entry per launch (vnect_step_name order). */
int vnect_check_finite(vnect_t* h, int32_t n, int64_t* counts);
int64_t vnect_launch_count(vnect_t* h);      /* kernels launched by this handle so far */
double vnect_info(vnect_t* h, const char* key); /* "flops_per_forward", "num_sms", "conv_launches_per_forward", ...,
                                                   "cached_graphs" (live CUDA-graph cache entries) */
/* device time of `reps` back-to-back forwards of n images already in device memory (CUDA events on the handle's
 * stream); per_layer_ms may be NULL or float[conv_launches_per_forward + 1] (pool is the last entry) */
int vnect_time_forward(vnect_t* h, int32_t n, int32_t reps, float* total_ms, float* per_layer_ms);
/* device time (ms, CUDA events on the handle's stream) of the pre-processing kernels and of the post-process kernel for
 * n_frames S x S frames: whatever the lane-0 frame buffer and the CNN output maps currently hold; the filter state
 * of streams 0..n_frames-1 advances by one step per repetition */
int vnect_time_prepost(vnect_t* h, int32_t n_frames, int32_t reps, float* pre_ms, float* post_ms);
const char* vnect_step_name(vnect_t* h, int32_t i); /* name of launch i of one forward, NULL past the end */
/* how launch i of one forward runs, as the plan built it (tests check their coverage with it): out = int32[12].
 * Implicit-GEMM conv: {block_n, epilogue, cg (CTAs per MMA), b_resident, halo, im2col, mode (0 flat rows, 1 spatial
 * tiles), n2 (second conv of a fused block tail, 0 = none), tw, th (pixel tile), H, W (GEMM-row grid)}.
 * conv1 + pool1 (the step named "conv1+pool1"): {cg, n_xt (x tiles per row segment), 0, ...}. */
int vnect_step_path(vnect_t* h, int32_t i, int32_t* out);

const char* vnect_last_error(vnect_t* h);
const char* vnect_version(void);
void vnect_destroy(vnect_t* h);

#ifdef __cplusplus
}
#endif
#endif
