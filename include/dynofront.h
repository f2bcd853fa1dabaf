/*
 * dynofront.h -- C ABI of libdynofront: the front-end half of the DynOSAM hot path on sm_100a
 * (SURVEY.md section 8 rows a13 "dense-flow warp / label correlate" and a14 "pyramidal KLT").
 *
 * Replaces, with the same inputs / outputs and the same ordering semantics:
 *   dynofront_track_dynamic     FeatureTracker::trackDynamic        dynosam/src/frontend/vision/FeatureTracker.cc:339-498
 *   dynofront_sample_candidates FeatureTracker::sampleDynamic scan  FeatureTracker.cc:864-953
 *   dynofront_sample_dynamic    FeatureTracker::sampleDynamic: scan, ANMS (RangeTree), new features  FeatureTracker.cc:864-1015
 *   dynofront_anms_range_tree   AdaptiveNonMaximumSuppression(RangeTree)::suppressNonMax on equal responses
 *                               (NonMaximumSupression.cc:45-93, anms.cc:278-362), as trackDynamicKLT calls it (:818-834)
 *   dynofront_propagate_mask    FeatureTracker::propogateMask       FeatureTracker.cc:1212-1359
 *   dynofront_track_static_flow ExternalFlowFeatureTracker::trackStatic / constructStaticFeature  StaticFeatureTracker.cc:70-220
 *   dynofront_klt_track_fb      KltFeatureTracker::trackPoints: forward + backward LK, round-trip test, label / border / age checks (:486-592)
 *   dynofront_stereo_track      FeatureTracker::stereoTrack: left -> right LK + disparity / depth test  FeatureTracker.cc:194-337
 *   dynofront_klt_track         cv::calcOpticalFlowPyrLK as called by KltFeatureTracker::trackPoints
 *                               (StaticFeatureTracker.cc:420-625) and FeatureTracker::trackDynamicKLT (FeatureTracker.cc:500-862)
 * Images are row-major, tightly packed: flow float32[H][W][2] (CV_32FC2), masks int32[H][W] (CV_32S, ObjectId),
 * detection / tracking masks uint8[H][W], gray uint8[H][W]  (reference image types: dynosam README.md:199-202).
 * Plain C types only; 0 = ok, < 0 = error (same codes as dynoba.h).  No CPU fallback.
 */
#ifndef DYNOFRONT_H
#define DYNOFRONT_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct dynofront_ctx* dynofront_handle;

typedef struct {
  int32_t max_dynamic_feature_age;   /* params/FrontendParams.yaml:66 (20) */
  int32_t min_distance;              /* min_distance_btw_tracked_and_detected_dynamic_features (2) */
  int32_t shrink_row, shrink_col;    /* isWithinShrunkenImage margins (0) */
} dynofront_track_params;

int dynofront_create(int device, int width, int height, dynofront_handle* out);
int dynofront_destroy(dynofront_handle h);
const char* dynofront_last_error(dynofront_handle h);

/* Upload the current frame's dense inputs (any pointer may be NULL to keep the previous upload). */
int dynofront_set_frame(dynofront_handle h, const float* flow, const int32_t* motion_mask, const uint8_t* detection_mask);

/* Streaming mode: makes the frame that was current the previous one without moving it (device buffers swap roles) and
 * uploads ONLY the new frame: gray (its pyramid and Scharr derivatives are built at once), flow, motion mask, optional
 * detection mask.  Returns without synchronising; copies are asynchronous when the host buffers were registered with
 * dynofront_pin_host (they must then stay untouched until the next dynofront call returns).  After two frames
 * dynofront_propagate_mask and dynofront_klt_track_fb accept NULL images and work on the resident pair
 * (reference: the frame loop of FeatureTracker::track, FeatureTracker.cc:73-192, which re-uploads both images per call). */
int dynofront_next_frame(dynofront_handle h, const uint8_t* gray, const float* flow, const int32_t* motion_mask, const uint8_t* detection_mask);
int dynofront_pin_host(dynofront_handle h, void* ptr, size_t bytes);     /* cudaHostRegister / Unregister of a caller buffer */
int dynofront_unpin_host(dynofront_handle h, void* ptr);
int dynofront_get_motion_mask(dynofront_handle h, int32_t* out);          /* the current frame's motion mask as it is on the device */

/* trackDynamic: n previous dynamic features (predicted key-point at this frame, object label, age, tracklet id),
 * iterated in array order.  Outputs are per input feature (rows of rejected features are zero); new tracklet ids
 * are handed out in iteration order starting at *next_tracklet_id, which is updated.  detection_mask_out /
 * tracking_mask_out (may be NULL) receive the masks after the cv::circle side effects. */
int dynofront_track_dynamic(dynofront_handle h, int32_t n, const double* prev_pred_kp, const int32_t* prev_label,
                            const int32_t* prev_age, const int64_t* prev_tracklet, const dynofront_track_params* prm,
                            int64_t* next_tracklet_id, uint8_t* accepted, double* pred_kp, double* flow_out,
                            int32_t* age, int64_t* tracklet, int32_t* label, uint8_t* detection_mask_out,
                            uint8_t* tracking_mask_out);

/* sampleDynamic candidate scan over the whole image, using the detection mask left on the device by
 * dynofront_track_dynamic (or the uploaded one).  For each of the n_objects labels: counts[o] candidates whose
 * linear pixel indices (row*W + col, ascending) are written to indices + offsets[o]; zero_flow[o] = pixels of the
 * object skipped because a flow component is exactly 0.  capacity = size of indices. */
int dynofront_sample_candidates(dynofront_handle h, int32_t n_objects, const int32_t* objects, const dynofront_track_params* prm,
                                int32_t* counts, int32_t* offsets, int32_t* zero_flow, int32_t* indices, int64_t capacity);

/* sampleDynamic as ONE call: the candidate scan above, then per object AdaptiveNonMaximumSuppression(RangeTree) with
 * K = max(max_features - num_track[o], 0) and the given tolerance (0.01 in the reference) over the candidate list in
 * ascending pixel order, then the new features (FeatureTracker.cc:955-1015).  Uses the detection mask left on the device
 * by dynofront_track_dynamic (or the uploaded one); synchronises once, and only the selected features cross PCIe.
 * Per object: candidates[o] (the scan's count), zero_flow[o] (may be NULL), selected[o] and selected_offset[o] (first
 * row of the object's features; objects follow each other in the order of objects[]).  Per feature, in selection order:
 * keypoint[f][2] = (col, row), flow[f][2] (float -> double), predicted_keypoint[f][2] = keypoint + flow and tracklet[f],
 * counting up from *next_tracklet_id, which is updated.  New features have age 0.  K = 0 gives no features (the
 * reference's K = 0 is undefined behaviour, DESIGN.md section 8f-4).  If more than `capacity` features are selected the
 * call returns -1 with the per-object outputs filled in and *next_tracklet_id unchanged.  ms_device (may be NULL) = device
 * time from the first to the last operation of the call. */
int dynofront_sample_dynamic(dynofront_handle h, int32_t n_objects, const int32_t* objects, const int32_t* num_track, int32_t max_features,
                             float tolerance, const dynofront_track_params* prm, int64_t* next_tracklet_id, int32_t* candidates,
                             int32_t* zero_flow, int32_t* selected, int32_t* selected_offset, double* keypoint, double* flow,
                             double* predicted_keypoint, int64_t* tracklet, int64_t capacity, float* ms_device);

/* AdaptiveNonMaximumSuppression(RangeTree) on n_lists lists in one launch.  List l holds counts[l] points, stored one
 * list after the other in xy[][2] (float, in the caller's order; all responses equal, so the walk order is cv::sortIdx's
 * tie order, dynofront_anms_tie_order).  Coordinates must lie in [0, 65536) and cols / rows in [1, 65535]: the reference
 * keeps u16 cells.  num_ret_points[l] = K (<= 0: nothing selected).  Writes n_selected[l] and, at the list's own offset in
 * indices[], the selected points' indices within the list in selection order.  Bit-exact with the reference, including
 * its binary search ending on the previous width's selection (which need not hold K points) and K = 1 selecting nothing.
 * (Search boxes are not wrapped at 65536, where the reference's u16 bounds would.) */
int dynofront_anms_range_tree(dynofront_handle h, int32_t n_lists, const int32_t* counts, const float* xy, const int32_t* num_ret_points,
                              float tolerance, int32_t cols, int32_t rows, int32_t* indices, int32_t* n_selected);
/* parity hook, host only (no device needed): the walk order of n equal responses, out[k] = input index of the k-th point
 * = cv::sortIdx(zeros(1, n), SORT_EVERY_ROW | SORT_DESCENDING) */
int dynofront_anms_tie_order(int32_t n, int32_t* out);

/* propogateMask: previous-frame features (predicted key-point, label), previous mask / flow, current mask (in/out).
 * All three images NULL: streaming mode, the resident previous frame votes into the resident current motion mask in place. */
int dynofront_propagate_mask(dynofront_handle h, int32_t n, const double* prev_pred_kp, const int32_t* prev_label,
                             const int32_t* prev_mask, const float* prev_flow, const dynofront_track_params* prm,
                             int32_t min_votes, int32_t* current_mask);

/* Pyramidal Lucas-Kanade, OpenCV semantics (fixed-point bilinear weights, int16 Scharr derivatives).
 * next_pts is in/out when use_initial_flow != 0.  err may be NULL. */
int dynofront_klt_track(dynofront_handle h, const uint8_t* prev_gray, const uint8_t* cur_gray, int32_t n,
                        const float* prev_pts, float* next_pts, uint8_t* status, float* err, int32_t win,
                        int32_t max_level, int32_t max_count, double epsilon, int32_t use_initial_flow,
                        double min_eig_threshold, float* ms_device);
/* KltFeatureTracker::trackPoints as ONE call (StaticFeatureTracker.cc:486-534,575-592): forward LK, the reference's
 * retry without the initial flow when fewer than 10 points survive, backward LK from the forward result, the
 * forward-backward test (both statuses good and the backward track within max_fb_distance of the start, float
 * arithmetic) and, with check_static, the per-point checks that follow the (host-side, out of scope) RANSAC:
 * background label at the truncated key-point of the motion mask given to dynofront_set_frame, inside the image and the
 * shrunken image, age + 1 <= max_feature_track_age.  Nothing returns to the host between the stages.
 * prev_gray == cur_gray == NULL: streaming mode, the two resident pyramids are used (nothing is uploaded or rebuilt).
 * status[n] = forward-backward result, keep[n] = status && checks (may be NULL without check_static),
 * back_pts[n][2] (may be NULL) = where the backward pass landed. */
typedef struct {
  int32_t win, max_level, max_count; double epsilon;                 /* forward: (21, 3, 30, 0.03), StaticFeatureTracker.cc:440-446 */
  int32_t win_back, max_level_back, max_count_back; double epsilon_back;   /* backward: (21, 5, 30, 0.01), :510-512 (OpenCV defaults) */
  int32_t use_initial_flow; double min_eig_threshold; double max_fb_distance;   /* 1e-4, 0.5 */
  int32_t check_static, max_feature_track_age;                       /* params/FrontendParams.yaml max_feature_track_age */
  dynofront_track_params track;                                      /* shrink margins */
} dynofront_klt_fb_params;
int dynofront_klt_track_fb(dynofront_handle h, const uint8_t* prev_gray, const uint8_t* cur_gray, int32_t n, const float* prev_pts,
                           float* next_pts, uint8_t* status, float* back_pts, const dynofront_klt_fb_params* prm,
                           const int32_t* prev_age, uint8_t* keep, int32_t* n_status, int32_t* n_keep, float* ms_device);
/* FeatureTracker::stereoTrack (FeatureTracker.cc:194-337): LK from the left to the right image (21x21, 5 levels, OpenCV default
 * criteria) and the per-point disparity test: valid[i] = status[i] && !(uL - uR <= 1 || uR < 0), depth[i] = fx * baseline /
 * (uL - uR) (0 where invalid).  The fundamental-matrix RANSAC the reference runs between the two is host code:
 * final = status & ransac_mask & valid. */
int dynofront_stereo_track(dynofront_handle h, const uint8_t* left_gray, const uint8_t* right_gray, int32_t n, const float* left_pts,
                           float* right_pts, uint8_t* status, double fx, double baseline, double* depth, uint8_t* valid, float* ms_device);
/* parity hook: (min eigenvalue, trace/(2 win^2)) of the level-0 spatial gradient matrix of the last forward pass, [n][2] */
int dynofront_klt_last_min_eig(dynofront_handle h, int32_t n, float* out);

/* ExternalFlowFeatureTracker::trackStatic + constructStaticFeature (StaticFeatureTracker.cc:70-220) on the flow / motion
 * mask given to dynofront_set_frame.  Previous static features (predicted key-point, age, usable flag) are walked in
 * array order: the first one per grid cell (cell_size px, OccupancyGrid2D.hpp:96-101) that is contained, usable, on the
 * background, has a non-zero flow and a predicted key-point inside the image is kept with age + 1.  Then the detections
 * det_xy[n_det][2] (integer pixel positions, e.g. the ORB key-points, in detector order) fill the still empty cells
 * until the frame holds max_features; their tracklet ids count up from *next_tracklet_id (updated).  Rows of rejected
 * features are zero. */
int dynofront_track_static_flow(dynofront_handle h, int32_t n_prev, const double* prev_pred_kp, const int32_t* prev_age,
                                const uint8_t* prev_usable, int32_t n_det, const int32_t* det_xy, int32_t cell_size,
                                int32_t max_features, int64_t* next_tracklet_id, uint8_t* acc_prev, double* flow_prev,
                                double* pred_prev, int32_t* age_out, uint8_t* acc_det, double* flow_det, double* pred_det,
                                int64_t* tracklet_det, int32_t* n_tracked, int32_t* n_detected);

/* parity hooks: pyramid level / Scharr derivative of the last prev image (level l): sizes via w,h out */
int dynofront_get_pyramid_level(dynofront_handle h, int32_t which /*0 prev,1 cur*/, int32_t level, int32_t* w, int32_t* hgt,
                                uint8_t* img, int16_t* deriv);

#ifdef __cplusplus
}
#endif
#endif
