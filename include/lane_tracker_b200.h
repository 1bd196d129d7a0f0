/*
 * lane_tracker_b200 -- C ABI of the B200-native lane-tracking hot path.
 *
 * The reference (pierluigiferrari/lane_tracker) has no FFI: its boundary is the
 * Python class `LaneTracker` (lane_tracker.py:85-1209) called once per frame by
 * moviepy (process_video.py:43).  This header is the boundary a maintainer would
 * bind instead (ctypes stub in INTEGRATION.md): every entry point cites the
 * reference method it replaces.  Conventions:
 *   - plain C types only; every pointer named d_* is DEVICE memory owned by the
 *     caller, every h_* is HOST memory owned by the caller;
 *   - all work is enqueued on the caller's CUDA stream (`stream` is a
 *     cudaStream_t passed as void*); nothing synchronises unless documented;
 *   - int return: 0 = ok, <0 = error (see lt_last_error); no exceptions;
 *   - one handle per GPU; a handle is not thread-safe (the reference object is
 *     not re-entrant either: it carries tracking state);
 *   - images are uint8, RGB, row-major HWC, tightly packed.
 *   - a handle serves `max_streams` independent video streams; per-stream
 *     tracking state (lane_tracker.py:139-176) lives in device memory.
 */
#ifndef LANE_TRACKER_B200_H
#define LANE_TRACKER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LT_ABI_VERSION 4
#define LT_MAX_AVERAGE 8          /* capacity of the n_average rings */

typedef struct lt_handle lt_handle;

/* Constructor arguments of LaneTracker.__init__ (lane_tracker.py:101-137) plus the
 * calibration read by utils.load_camera_calib / load_warp_params (utils.py:13-55). */
typedef struct lt_config {
    int32_t img_w, img_h;         /* img_size    (width, height) */
    int32_t bv_w, bv_h;           /* warped_size (width, height); bv_w must be even */
    double  cam_matrix[9];        /* row-major 3x3 */
    double  dist_coeffs[5];       /* k1 k2 p1 p2 k3 */
    double  M[9];                 /* warp_matrices[0] */
    double  Minv[9];              /* warp_matrices[1] */
    double  mppv, mpph;           /* mpp_conversion */
    int32_t n_fail, n_reset, n_average, print_frame_count;
    int32_t max_streams;          /* independent streams served by this handle */
    int32_t device;               /* CUDA device ordinal */
} lt_config;

/* Keyword options of LaneTracker.process (lane_tracker.py:876-900). */
typedef struct lt_params {
    int32_t ksize_r, C_r, ksize_b, C_b;
    int32_t filter_type;          /* 0 = 'bilateral', 1 = 'neighborhood' */
    int32_t mask_noise, noise_thresh, ksize_noise, C_noise;
    int32_t window_width, window_height, search_range;
    double  mu;
    int32_t no_success_limit;
    double  start_slice;
    int32_t ignore_sides, ignore_bottom;
    int32_t bandwidth;
    double  partial;
    int32_t n_tries;
} lt_params;

/* Per-stream, per-frame result of lt_process (what process() leaves in the
 * tracker's attributes, lane_tracker.py:1142-1209). */
typedef struct lt_result {
    int32_t counter;              /* frames processed by this stream so far */
    int32_t attempts;             /* 1 or 2 (lane_tracker.py:1071) */
    int32_t search_mode;          /* of the last attempt: 0 sliding window, 1 band */
    int32_t detected_pixels;
    int32_t valid_lane_lines;
    int32_t last_detection;
    int32_t drew_lane;            /* 1: lane polygon blended, 0: failure frame */
    int32_t n_left, n_right;      /* lane pixels of the last attempt */
    int32_t n_left_avg, n_right_avg; /* vertices of the averaged polylines */
    int32_t success;
    int32_t fit_rank_deficient;   /* bit0 left, bit1 right: <3 distinct rows */
    int32_t first_detected, first_valid;      /* outcome of attempt 1 (== final when attempts == 1) */
    int32_t first_n_left, first_n_right;
    int32_t reserved0;
    /* radii are Python ints in the reference (int() of an unbounded float, lane_tracker.py:539-549): 64 bits here,
     * saturated at +-2^63 */
    int64_t left_curve_radius, right_curve_radius, average_curve_radius;
    double  left_fit[3], right_fit[3];   /* last attempt's np.polyfit equivalents */
    double  left_avg[3], right_avg[3];
    double  eccentricity;
    double  validity_d[3];        /* x1_diff, x2_diff, x3_diff of check_validity */
    double  first_left_fit[3], first_right_fit[3];
} lt_result;

/* Snapshot of one stream's tracking state (lane_tracker.py:139-176); used by
 * tests (teacher forcing) and for checkpoint/restore. */
typedef struct lt_state {
    int32_t last_detection, counter, success;
    int32_t ring_len;                             /* len(left_fit_coeffs) */
    int32_t ring_empty[LT_MAX_AVERAGE];           /* 1 = np.array([]) marker */
    double  ring_left[LT_MAX_AVERAGE][3], ring_right[LT_MAX_AVERAGE][3];
    int32_t has_last;
    double  last_left[3], last_right[3];
    int32_t has_avg;
    double  left_avg[3], right_avg[3];
    int32_t n_left_avg, n_right_avg;              /* polyline vertex counts */
    int32_t radii_len;
    int64_t radii[LT_MAX_AVERAGE];
    int64_t average_curve_radius;
    double  eccentricity;
} lt_state;

/* Acceptance windows of check_validity (lane_tracker.py:588-593, 617).  The reference hard-codes them as local
 * constants and documents other sets per demo video (tracker_settings.md); lt_create installs the shipped ones
 * (150/230, 110/230, 80/200, 0.25). */
typedef struct lt_validity {
    double min_dist_y1, max_dist_y1, min_dist_y2, max_dist_y2, min_dist_y3, max_dist_y3, tangent_thresh;
} lt_validity;

/* ---- lifetime ------------------------------------------------------------ */

/* LaneTracker.__init__ (lane_tracker.py:101-176) for `max_streams` streams.
 * Builds the fixed-point remap tables on the device.  Synchronous. */
int lt_create(const lt_config* cfg, lt_handle** out);
int lt_destroy(lt_handle* h);
/* Re-zero the state of the listed streams (ids == NULL: all). Synchronous. */
int lt_reset(lt_handle* h, const int32_t* ids, int32_t n);
int lt_set_validity(lt_handle* h, const lt_validity* v);     /* NULL restores the shipped constants */
int lt_get_validity(lt_handle* h, lt_validity* v);
const char* lt_last_error(void);
int lt_abi_version(void);
void lt_default_params(lt_params* p);            /* lane_tracker.py:876-900 */
/* Number of kernels this library has launched since load (bench bookkeeping). */
int64_t lt_launch_count(void);

/* ---- the per-frame hot path ---------------------------------------------- */

/* Frame buffers.  Every full-size frame buffer the caller passes -- d_frames and d_out of lt_process,
 * lt_process_front, lt_process_back and lt_draw_lane, d_frames of lt_remap, lt_warp_frame and lt_draw_text -- must
 * start at a 4-byte aligned address: the kernels read and write frames as 32-bit words.  A buffer that is not is
 * refused with an error before anything is launched.  (Frames are contiguous [n][img_h][img_w][3] and img_w is a
 * multiple of 4, so every row and every frame of an aligned buffer is aligned too.)  The bird's-eye images
 * (d_bv_rgb), masks, debug views and resize buffers are accessed byte by byte and need no alignment. */

/* LaneTracker.process (lane_tracker.py:876-1209) for streams 0..n_streams-1.
 *   d_frames : [n_streams][img_h][img_w][3]
 *   d_out    : same shape, NULL for fits-only mode (no overlay rendered), or == d_frames to annotate in place
 *              (only the rows the lane overlay can reach are rewritten)
 *   params   : one lt_params for all streams (the reference's defaults-are-the-
 *              config convention, README.md:34)
 *   d_results: [n_streams] lt_result, device memory (copy back asynchronously)
 * Stream s uses and updates state slot s (lt_process_streams below serves any subset of streams).  The putText overlays (lane_tracker.py:653-659, 668-672) are drawn
 * when glyph sprites are installed (lt_set_text_sprites). */
int lt_process(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n_streams,
               const lt_params* params, lt_result* d_results, void* stream);

/* lt_process in two halves, for callers that keep two batches in flight on two CUDA streams:
 *   lt_process_front: undistort + warp + first-attempt filter (find_lane_points 795-874 up to the binary mask).
 *                     Stateless; writes the handle's intermediate buffer set `set` (0 or 1; set 1 is allocated on
 *                     first use and doubles the intermediate memory).
 *   lt_process_back : searches, second attempt for the streams that failed, state machine, overlay and text
 *                     (lane_tracker.py:1040-1209) from buffer set `set`; advances the per-stream state.
 * lt_process(...) == lt_process_front(..., 0, stream) followed by lt_process_back(..., 0, ..., stream).
 * The caller orders things with its own events: back(k) after front(k); back(k) after back(k-1) (tracking state);
 * front(k+2) after back(k) (they share a buffer set).  lane_tracker_b200.DevicePipeline does exactly that. */
int lt_process_front(lt_handle* h, const uint8_t* d_frames, int32_t n_streams, const lt_params* params,
                     int32_t set, void* stream);
int lt_process_back(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n_streams,
                    const lt_params* params, int32_t set, lt_result* d_results, void* stream);

/* lt_process for an arbitrary set of streams, in any order: frame i of d_frames (and d_out[i], d_results[i]) belongs
 * to stream h_ids[i].
 *   h_ids: HOST int32 [n], 1 <= n <= max_streams, every id in [0, max_streams), pairwise distinct (two frames of
 *          one stream in one batch would race on its state).  The ids are copied when the call is enqueued: h_ids
 *          may be reused as soon as the call returns.  Nothing synchronises; the call is capturable in a CUDA graph.
 * Addressing rule: frames, out frames, result records, masks and the other intermediate buffers are indexed by batch
 * position i; the tracking state, averaged polylines, cached lane polygon and captured pixel lists by stream id
 * h_ids[i] (lt_get_state, lt_read_capture and lt_debug_read item 9 take a stream id; lt_debug_read items 3-8 a batch
 * position).  Streams not listed keep their tracking state, cached lane polygon and captured pixel lists byte for
 * byte.  With h_ids = {0, 1, ..., n-1} the results equal those of lt_process bit for bit.
 * A null h_ids, n outside [1, max_streams], an id out of range or a repeated id is refused with an error that names
 * the id, before anything is enqueued; every check of lt_process applies as well.
 * lt_process_streams(...) == lt_process_front(..., 0, stream) followed by lt_process_back_streams(..., 0, ..., stream)
 * (the front half is stateless and takes no ids).  lt_process_back_streams is ordered like lt_process_back: back(k)
 * after front(k) and after back(k-1), front(k+2) after back(k). */
int lt_process_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                       const lt_params* params, lt_result* d_results, void* stream);
int lt_process_back_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                            const lt_params* params, int32_t set, lt_result* d_results, void* stream);

/* Keep the ordered lane-pixel sets and window centroids of every lt_process call so that
 * lt_read_capture can return them (the reference exposes them as the attributes left_x/left_y/
 * right_x/right_y/left_window_centroids, lane_tracker.py:159-166).  Off by default: the
 * throughput path needs only the moment sums. */
int lt_set_capture(lt_handle* h, int32_t enable);
/* Capacity (entries per stream and side) of the ordered pixel lists kept for lt_read_capture.  Default:
 * max(65536, 64 * bv_h), enough for the sliding-window search (window_width <= 64) and for band searches with
 * bandwidth <= 32; a band-search row can hold 2 * bandwidth - 1 pixels, and lt_process rejects a bandwidth whose
 * lists could overflow while capture is on.  Synchronous; reallocates the capture buffers. */
int lt_set_pixel_capacity(lt_handle* h, int32_t capacity);
/* attempt: 0 first, 1 second.  h_pixels: (y<<16 | x+32768), up to `capacity` entries;
 * h_count: true count; h_centroids: LT_MAX_LEVELS ints (sliding-window search only). Synchronous. */
int lt_read_capture(lt_handle* h, int32_t stream_id, int32_t attempt, int32_t side, uint32_t* h_pixels,
                    int32_t capacity, int32_t* h_count, int32_t* h_centroids, int32_t* h_ncentroids);

/* Text overlays of draw_lane / print_failure (cv2.putText, FONT_HERSHEY_SIMPLEX, scale 1, white, thickness 2,
 * LINE_AA; lane_tracker.py:653-659, 668-672).  The glyph data (per-character pixel lists and 256-entry
 * background->output tables, tools/make_text_sprites.py) is supplied by the host, like the calibration; all
 * pointers are HOST memory and are copied.  Without sprites (or with h_tables == NULL) no text is drawn.
 * Strings are formatted on the device from the per-stream state. */
int lt_set_text_sprites(lt_handle* h, const uint8_t* h_tables, int32_t n_tables, const int32_t* h_char_start,
                        int32_t n_chars, const int16_t* h_dy, const int16_t* h_dx, const uint16_t* h_lut,
                        int32_t n_pixels, const int32_t* h_advance, int32_t first_char);

/* Remap variant.  0 (default): exact two-stage cv2.undistort + cv2.warpPerspective, bit-exact bird's-eye view.
 * 1: fused single resample (lens distortion and homography composed in fp64, one bilinear interpolation from the
 * raw frame).  Mode 1 is NOT bit-exact; its stated tolerance against mode 0 on the reference's bundled frames is
 * mask IoU >= 0.6 per frame and >= 0.8 on average (measured: tests/test_gpu_parity.py::test_fused_remap_variant). */
int lt_set_remap_mode(lt_handle* h, int32_t mode);

/* Copy frame rows [row0, row1) of n_frames frames between a host (pinned) and a device batch of full frames
 * (one cudaMemcpy2DAsync: pitch = frame size).  to_device: 1 host->device, 0 device->host.  Used to move only
 * the rows the tracker reads / the overlay can change (lt_debug_read geometry) across PCIe. */
int lt_memcpy_rows(lt_handle* h, void* dst, const void* src, int32_t n_frames, int32_t row0, int32_t row1,
                   int32_t to_device, void* stream);

/* ---- in-stream stage timing (bench.py's roofline figures) --------------------
 * lt_profile_begin arms CUDA-event recording at every stage boundary of the next `max_calls`
 * lt_process calls (events are recorded on the caller's stream, no synchronisation);
 * lt_profile_read synchronises, sums the per-stage durations [ms] over the recorded calls,
 * and disarms.  Stage ids: lt_stage_name(0..LT_NSTAGES-1). */
#define LT_NSTAGES 16
int lt_profile_begin(lt_handle* h, int32_t max_calls);
int lt_profile_read(lt_handle* h, double* h_stage_ms, int32_t* h_calls);
/* Restrict the marks to the stage boundaries whose bit (1 << stage index, see lt_stage_name) is set; 0 = all.
 * The time reported for a selected stage then runs from the previous SELECTED boundary of the same call, so select
 * the boundary before a stage as well (e.g. warp | erode55 | tophat55 to time the two morphology launches with three
 * events per call instead of a dozen). */
int lt_profile_select(lt_handle* h, uint32_t stage_mask);
const char* lt_stage_name(int32_t stage);

/* ---- stage entry points (mirror the reference's public methods) ----------- */

/* cv2.undistort + cv2.warpPerspective of find_lane_points (lane_tracker.py:832-834).
 *   d_bv_rgb : [n][bv_h][bv_w][3] (may be NULL: only the internal planes are kept) */
int lt_remap(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int32_t n_streams, void* stream);

/* LaneTracker.filter_lane_points (lane_tracker.py:183-240) on caller-supplied
 * bird's-eye RGB images.  d_mask: [n][bv_h][bv_w] uint8 {0,255}. */
int lt_filter_lane_points(lt_handle* h, const uint8_t* d_bv_rgb, uint8_t* d_mask, int32_t n_streams,
                          int32_t filter_type, int32_t ksize_r, int32_t C_r, int32_t ksize_b, int32_t C_b,
                          int32_t mask_noise, int32_t ksize_noise, int32_t C_noise, int32_t noise_thresh,
                          void* stream);

/* Pixel-set outputs of the two searches.  Pixels are (y<<16 | x) in the
 * reference's order; x is stored with a +32768 bias because NumPy slice
 * wrap-around can report negative x (lane_tracker.py:299-303).
 *   d_pixels : [n][2][capacity] uint32   (left, right)
 *   d_counts : [n][2] int32 (true counts, may exceed capacity)
 *   d_centroids: [n][2][LT_MAX_LEVELS] int32, d_ncentroids: [n][2] (SWS only; may be NULL) */
#define LT_MAX_LEVELS 128
int lt_sliding_window_search(lt_handle* h, const uint8_t* d_mask, int32_t n_streams,
                             int32_t window_width, int32_t window_height, int32_t search_range, double mu,
                             int32_t no_success_limit, double start_slice, int32_t ignore_sides,
                             int32_t ignore_bottom, double partial,
                             uint32_t* d_pixels, int32_t capacity, int32_t* d_counts,
                             int32_t* d_centroids, int32_t* d_ncentroids, int32_t* d_detected, void* stream);

/* LaneTracker.band_search (lane_tracker.py:449-500); coefficients per stream:
 * d_coeffs [n][2][3] (left, right) = last_left_coeffs / last_right_coeffs. */
int lt_band_search(lt_handle* h, const uint8_t* d_mask, int32_t n_streams, const double* d_coeffs,
                   int32_t bandwidth, int32_t ignore_bottom, double partial,
                   uint32_t* d_pixels, int32_t capacity, int32_t* d_counts, int32_t* d_detected, void* stream);

/* LaneTracker.fit_poly (lane_tracker.py:502-509): np.polyfit(y, x, 2) per side.
 *   d_pixels/d_counts as produced above; d_fits [n][2][3]. */
int lt_fit_poly(lt_handle* h, const uint32_t* d_pixels, int32_t capacity, const int32_t* d_counts,
                int32_t n_streams, double* d_fits, void* stream);

/* LaneTracker.check_validity (lane_tracker.py:561-627). d_valid [n] int32,
 * d_diffs [n][3] (may be NULL). */
int lt_check_validity(lt_handle* h, const double* d_fits, int32_t n_streams, int32_t* d_valid,
                      double* d_diffs, void* stream);

/* LaneTracker.get_poly_points (lane_tracker.py:511-528).
 *   d_fits [n][2][3]; d_x [n][2][bv_h] int32 (x of the kept points, re-stacked so
 *   entry i belongs to row bv_h - count + i); d_counts [n][2]. */
int lt_get_poly_points(lt_handle* h, const double* d_fits, int32_t n_streams, double partial,
                       int32_t* d_x, int32_t* d_counts, void* stream);

/* LaneTracker.draw_lane (lane_tracker.py:629-662) without putText: fills the lane
 * polygon of the given polylines, un-warps and blends it.  d_x/d_counts as above. */
int lt_draw_lane(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n_streams,
                 const int32_t* d_x, const int32_t* d_counts, void* stream);

/* LaneTracker.get_curve_radius / get_eccentricity (lane_tracker.py:530-559): per stream the left / right curve radius
 * in metres at the bottom row (int() truncation, saturated at 2^63 - 1) from the pixel-space fits d_fits [n][2][3], and
 * the lateral offset from the lane centre in metres from the last vertices of the polylines d_x / d_counts (layout of
 * lt_get_poly_points).  d_radii [n][2] int64; d_eccentricity [n] double, may be NULL (then d_x / d_counts may be too).
 * The running mean over n_average frames (:544-549) is bookkeeping of the caller, as in the reference. */
int lt_lane_metrics(lt_handle* h, const double* d_fits, const int32_t* d_x, const int32_t* d_counts, int32_t n_streams,
                    int64_t* d_radii, double* d_eccentricity, void* stream);

/* bilateral_adaptive_threshold (lane_tracker.py:14-83) on any single-channel uint8 device image (pitches in bytes):
 * mode 0 = 'floor', 1 = 'ceil'; true_value / false_value in [0, 255].  Runs on the current device. */
int lt_bilateral_adaptive_threshold(const uint8_t* d_img, int32_t width, int32_t height, int64_t pitch_in, uint8_t* d_out,
                                    int64_t pitch_out, int32_t ksize, int32_t C, int32_t mode, int32_t true_value,
                                    int32_t false_value, void* stream);

/* The cv2.putText overlays of draw_lane (kind 0) / print_failure (kind 1) (lane_tracker.py:653-659, 668-672) drawn in
 * place on device frames from HOST arrays of per-frame values (radius and eccentricity only read for kind 0; "Frame: n"
 * shows h_counter - 1 when the handle was created with print_frame_count).  Needs lt_set_text_sprites.  Synchronises
 * the stream once (staging of the small host arrays). */
int lt_draw_text(lt_handle* h, uint8_t* d_frames, int32_t n_frames, const int32_t* h_kind, const int64_t* h_radius,
                 const double* h_eccentricity, const int32_t* h_counter, void* stream);

/* ---- ingest (process_video.py:42-44: the reference receives RGB frames from moviepy / ffmpeg) ---- */

/* Decoder output -> the RGB frames lt_process consumes: cv2.cvtColor(nv12, COLOR_YUV2RGB_NV12) (ITU-R BT.601 limited
 * range, OpenCV's Q20 fixed point, chroma not interpolated), bit-exact.  d_nv12 [n][height * 3 / 2][width] uint8 (luma
 * plane, then interleaved U, V rows), d_rgb [n][height][width][3].  width % 4 == 0, height even, 4-byte aligned
 * buffers.  Runs on the current device. */
int lt_nv12_to_rgb(const uint8_t* d_nv12, uint8_t* d_rgb, int32_t n_frames, int32_t width, int32_t height, void* stream);

/* ---- debug views (lane_tracker.py:675-793, utils.py:57-103; not on the per-frame path) ---- */

/* cv2.warpPerspective(img, M, warped_size) of the RAW frames (lane_tracker.py:1035, the middle panel of the
 * split view): d_frames [n][img_h][img_w][3] -> d_bv_rgb [n][bv_h][bv_w][3]. */
int lt_warp_frame(lt_handle* h, const uint8_t* d_frames, int32_t n_streams, uint8_t* d_bv_rgb, void* stream);

typedef struct lt_vis {
    int32_t mode;               /* 0: visualize_sliding_window_search (:689-729), 1: visualize_band_search (:731-771) */
    int32_t n_left, n_right;    /* lane pixels of the search (left_y/left_x, right_y/right_x) */
    int32_t n_rects;            /* mode 0: search windows, <= 2 * LT_MAX_LEVELS */
    int32_t bandwidth;          /* mode 1 */
    int32_t reserved0;
    double  partial;            /* mode 1: `partial` of the band polylines */
    double  band_left[3], band_right[3];   /* mode 1: last_left_coeffs / last_right_coeffs the band was built on */
    double  left_fit[3], right_fit[3];     /* the new fit, drawn as graph points in (255, 235, 0) */
} lt_vis;

/* One search visualisation image, d_vis [bv_h][bv_w][3], from the binary image d_mask u8 [bv_h][bv_w], the lane
 * pixel lists (device, packed y << 16 | (x + 32768) as produced by lt_sliding_window_search / lt_band_search) and,
 * in mode 0, the search windows as HOST int32 [n_rects][5] = {row0, row1, col0, col1, side (0 left, 1 right)},
 * half-open, i.e. window_mask (:675-687) with Python's slice rules already applied. */
int lt_visualize_search(lt_handle* h, const lt_vis* v, const uint8_t* d_mask, const uint32_t* d_left,
                        const uint32_t* d_right, const int32_t* h_rects, uint8_t* d_vis, void* stream);

/* cv2.resize(img, dsize) as called by utils.create_split_view (utils.py:88): uint8, INTER_LINEAR, 1 or 3 channels.
 * Pitches in bytes, so that the destination can be a panel of a larger canvas. Runs on the current device. */
int lt_resize_linear(const uint8_t* d_src, int32_t src_w, int32_t src_h, int32_t channels, int64_t src_pitch,
                     uint8_t* d_dst, int32_t dst_w, int32_t dst_h, int64_t dst_pitch, void* stream);

/* ---- state access (tests, checkpoint/restore) ------------------------------ */
int lt_get_state(lt_handle* h, int32_t stream_id, lt_state* h_state, int32_t* h_left_avg_x,
                 int32_t* h_right_avg_x);   /* polylines: bv_h ints each, may be NULL. Synchronous. */
int lt_set_state(lt_handle* h, int32_t stream_id, const lt_state* h_state, const int32_t* h_left_avg_x,
                 const int32_t* h_right_avg_x);

/* Debug/test access to internal buffers of the last lt_process / stage call.  stream_id is a batch position for
 * items 3-8 (buffers of the last batch) and a stream id for item 9 (per-stream cache); the two coincide for lt_process.
 * what:0 undistort map (int32 [img_h][img_w][2]), 1 bird's-eye map (int32 [bv_h][bv_w][2]),
 *       2 overlay map (int32 [img_h][img_w][2]), 3 R plane u8 [bv_h][bv_w], 4 LAB-b plane,
 *       5 R top-hat, 6 b top-hat, 7 mask u8 {0,255}, 8 merged (pre-open) mask,
 *       9 lane row spans int32 [bv_h][2], 10 geometry int32[9] = {undistorted ROI first,last+1, overlay rows
 *       first,last+1, pair-plane width, mask words per row, pixel-list capacity of lt_read_capture, frame rows the
 *       tracker reads first,last+1}, 11 int32[3] = {row bands of the 55x55 and of the 29x29 morphology jobs in the
 *       last filter launch, SM count of the device}, 12 lane row spans of the last lt_draw_lane call (int32 [bv_h][2];
 *       9 is the per-stream cache that lt_process re-draws on failing frames).
 * Copies to HOST memory; synchronous. Returns bytes written or <0. */
int64_t lt_debug_read(lt_handle* h, int32_t what, int32_t stream_id, void* h_dst, int64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* LANE_TRACKER_B200_H */
