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
 *   - images are uint8, RGB, row-major HWC, tightly packed; the input frames of the
 *     hot path may be NV12 instead (lt_set_frame_format).
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
#define LT_MAX_PROFILES 16        /* parameter profiles per handle (lt_set_profile) */

typedef struct lt_handle lt_handle;

/* Constructor arguments of LaneTracker.__init__ (lane_tracker.py:101-137) plus the
 * calibration read by utils.load_camera_calib / load_warp_params (utils.py:13-55). */
typedef struct lt_config {
    int32_t img_w, img_h;         /* img_size    (width, height) */
    int32_t bv_w, bv_h;           /* warped_size (width, height); bv_w must be even (see lt_create) */
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
 * Builds the fixed-point remap tables on the device.  Synchronous.
 * Accepted geometry: img_w in [64, 32767] and a multiple of 4, img_h in [16, 32767], bv_w even and in [66, 32767],
 * bv_h in [16, 65535].  A bv_w at which a threshold kernel could not launch with some parameter set the process calls
 * accept (shared memory beyond the device's per-block opt-in limit) is refused as well: on a B200 (227 KB) the widest
 * accepted bird's-eye view is 3614 columns. */
int lt_create(const lt_config* cfg, lt_handle** out);
int lt_destroy(lt_handle* h);
/* Re-zero the state of the listed streams (ids == NULL: all): one cudaMemcpy per id from host memory on the legacy
 * default stream.  It is NOT ordered against work enqueued on other CUDA streams (non-blocking streams, such as the ones
 * the pipelines run their back halves on, do not wait for it): use it only with no work of the handle in flight.  To
 * start a new video on a stream while batches are in flight, use lt_reset_async on the stream of the back halves. */
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
 *   d_frames : [n_streams][img_h][img_w][3], or NV12 [n_streams][img_h * 3 / 2][img_w] (lt_set_frame_format)
 *   d_out    : [n_streams][img_h][img_w][3], NULL for fits-only mode (no overlay rendered), or, for RGB frames,
 *              == d_frames to annotate in place (only the rows the lane overlay can reach are rewritten)
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

/* Frame sequences: lt_process_streams in which ids may repeat.  The frames of one stream in the batch are consecutive
 * frames of that stream, in batch-position order, so one batch can carry many frames of a single video.  The results
 * equal, bit for bit, a series of lt_process_streams calls that feed each stream its frames one at a time.
 *   h_ids: HOST int32 [n], 1 <= n <= max_streams, every id in [0, max_streams); repeats allowed.
 * Addressing is that of lt_process_streams: frames, out frames, result records and masks by batch position, state by
 * stream id.  After the call a stream's state, averaged polylines, cached lane polygon and captured pixel lists are
 * those after its last frame in the batch; each out frame is drawn with the polygon and text of its own frame.
 * The front half is lt_process_front, unchanged.  The back half runs in rounds: round r holds the positions that are
 * the (r+1)-th frame of their stream in the batch, and the searches, second attempt and state update run round after
 * round; the overlay and text then run once over the batch.  A batch without a repeated id enqueues exactly the
 * launches of lt_process_streams.
 * Refused before anything is enqueued, naming the position: n outside [1, max_streams], a null h_ids, an id out of
 * range, and every other check of lt_process_streams except distinctness.  Nothing synchronises and the calls are
 * capturable in a CUDA graph (the first sequence call with a repeated id allocates the handle's per-position snapshot
 * buffers: make it before a capture).  Profiles and cameras are not available in these calls.
 * lt_process_sequence(...) == lt_process_front(..., 0, stream) followed by lt_process_back_sequence(..., 0, ..., stream);
 * lt_process_back_sequence is ordered like lt_process_back. */
int lt_process_sequence(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                        const lt_params* params, lt_result* d_results, void* stream);
int lt_process_back_sequence(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                             const lt_params* params, int32_t set, lt_result* d_results, void* stream);

/* Parameter profiles: one batch whose frames use different lt_params and check_validity windows (cameras on different
 * roads or mounted differently; tracker_settings.md of the reference documents one set per demo video).
 * lt_set_profile stores profile `profile` (0 <= profile < LT_MAX_PROFILES) on the handle: `params`, checked like the
 * lt_params of lt_process (same messages), and the windows `validity` (NULL: the shipped ones).  Synchronous; a profile
 * never set is "unset".  It may be called with work in flight: a batch uses the profile table as it stood when its
 * front half was enqueued (the front half copies the profiles into its intermediate buffer set, the back half reads
 * that copy only). */
int lt_set_profile(lt_handle* h, int32_t profile, const lt_params* params, const lt_validity* validity);

/* lt_process_streams / lt_process_front / lt_process_back_streams with a profile per batch position:
 *   h_profiles: HOST int32 [n], position i uses profile h_profiles[i] (its filter, searches, validity windows and
 *               n_tries; the second attempt keeps the reference's hard-coded parameters and uses the profile's
 *               windows).  Profiles belong to batch positions, like frames: a caller that keeps a profile per camera
 *               passes profile_of[ids], and a stream may change profile from one frame to the next.  Copied when the
 *               call is enqueued (kernel arguments): nothing synchronises and the calls are capturable in a CUDA graph.
 *   h_ids     : as lt_process_streams; NULL means the identity 0..n-1.
 * The front half filters each group of positions that share a filter configuration (filter_type, ksize_r, C_r,
 * ksize_b, C_b, mask_noise, and noise_thresh, ksize_noise, C_noise under mask_noise) with one launch sequence; with a
 * single group the launches are those of lt_process.  Refused before anything is enqueued, naming the position: a NULL
 * h_profiles, an index outside [0, LT_MAX_PROFILES), an unset profile; every check of lt_process_streams applies as
 * well (the pixel-capacity check of capture mode takes the widest bandwidth of the profiles used).
 * lt_process_back_profiles refuses a buffer set whose last front half was not lt_process_front_profiles, or had
 * another n or other profile indices (naming the first position that differs).  Ordering as lt_process_back.
 * lt_process_profiles(...) == lt_process_front_profiles(..., 0, stream) + lt_process_back_profiles(..., 0, ..., stream). */
int lt_process_profiles(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                        const int32_t* h_profiles, int32_t n, lt_result* d_results, void* stream);
int lt_process_front_profiles(lt_handle* h, const uint8_t* d_frames, const int32_t* h_profiles, int32_t n, int32_t set,
                              void* stream);
int lt_process_back_profiles(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                             const int32_t* h_profiles, int32_t n, int32_t set, lt_result* d_results, void* stream);

/* Cameras: one batch whose frames come from differently calibrated cameras (another mounting: its own warp M / Minv;
 * another lens: its own cam_matrix / dist_coeffs; and the metres per pixel of its bird's-eye view).  Image size,
 * bird's-eye size, n_fail / n_reset / n_average and print_frame_count stay those of the handle.
 * A handle holds up to LT_MAX_CAMERAS cameras.  Camera 0 is the calibration given to lt_create and cannot be changed;
 * lt_set_camera sets camera `camera` (1 <= camera < LT_MAX_CAMERAS) to `cam`, the same fields lt_config carries (taken
 * as given, like lt_create takes them).  It builds the camera's remap tables on the device and is synchronous (it
 * synchronises the device and may reallocate the intermediate buffer the camera calls undistort into).  A camera
 * cannot be unset.  Refused: camera 0, an index out of range, a NULL cam, and a call while a buffer set holds the front
 * half of a camera call whose back half has not been enqueued yet (the back half would draw with tables its front half
 * did not see). */
#define LT_MAX_CAMERAS 64
typedef struct lt_camera {
    double cam_matrix[9];         /* row-major 3x3 */
    double dist_coeffs[5];        /* k1 k2 p1 p2 k3 */
    double M[9];                  /* warp_matrices[0] */
    double Minv[9];               /* warp_matrices[1] */
    double mppv, mpph;            /* mpp_conversion */
} lt_camera;
int lt_set_camera(lt_handle* h, int32_t camera, const lt_camera* cam);

/* lt_process_streams / lt_process_profiles and their halves with a camera per batch position:
 *   h_cameras : HOST int32 [n], position i was filmed by camera h_cameras[i] (its undistort, warp, overlay and the
 *               metres per pixel of its curve radii and eccentricity).  Cameras belong to batch positions, like
 *               profiles: a caller that keeps one camera per stream passes camera_of[ids].  A stream may change camera
 *               between frames; its tracking state carries over (start a re-mounted camera's stream afresh with
 *               lt_reset_async, enqueued before the back half of the batch that carries its first new frame).
 *               Copied when the call is enqueued: nothing synchronises and the calls are capturable in a CUDA graph.
 *   params / h_profiles: exactly one is non-NULL (lt_process_streams or lt_process_profiles semantics).
 *   h_ids     : as lt_process_streams; NULL means the identity 0..n-1.
 * A batch whose positions all use camera 0 runs exactly the launches of the call without cameras.  Otherwise the front
 * half undistorts into a buffer of its own whose slots are grouped by camera; everything after the warp is indexed by
 * batch position as before.  Every check of lt_process_streams / lt_process_profiles applies, in the same order; then,
 * before anything is enqueued and naming the position: a NULL h_cameras, an index outside [0, LT_MAX_CAMERAS), a
 * camera never set, and remap mode 1 (the fused variant has camera 0's calibration baked in).
 * lt_process_back_cameras refuses a buffer set whose last front half was not lt_process_front_cameras, or had another
 * n or other camera indices.  Ordering as lt_process_back.
 * lt_process_cameras(...) == lt_process_front_cameras(..., 0, stream) + lt_process_back_cameras(..., 0, ..., stream). */
int lt_process_cameras(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                       const int32_t* h_cameras, int32_t n, const lt_params* params, const int32_t* h_profiles,
                       lt_result* d_results, void* stream);
int lt_process_front_cameras(lt_handle* h, const uint8_t* d_frames, const int32_t* h_cameras, int32_t n,
                             const lt_params* params, const int32_t* h_profiles, int32_t set, void* stream);
int lt_process_back_cameras(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                            const int32_t* h_cameras, int32_t n, const lt_params* params, const int32_t* h_profiles,
                            int32_t set, lt_result* d_results, void* stream);

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

/* Layout of the input frames d_frames.  LT_FRAME_RGB (default): [n][img_h][img_w][3].  LT_FRAME_NV12: what video
 * decoders deliver, [n][img_h * 3 / 2][img_w] uint8 per frame (the luma plane, then img_h / 2 rows of interleaved U, V
 * pairs), converted as cv2.cvtColor(COLOR_YUV2RGB_NV12) (ITU-R BT.601 limited range, chroma not interpolated) inside
 * the kernels that read the frames, with no RGB copy of the frame in between.  The results are bit for bit those of
 * the RGB path fed lt_nv12_to_rgb of the same frames.
 *   - The format applies to d_frames of lt_process, lt_process_front, lt_process_back, lt_process_streams,
 *     lt_process_back_streams and lt_remap, and to lt_memcpy_rows.  lt_draw_lane, lt_warp_frame and lt_draw_text
 *     always take RGB frames.  d_out stays RGB [n][img_h][img_w][3]: every row of it is written (the annotation cannot
 *     happen in place), and a d_out whose bytes overlap the NV12 input is refused.
 *   - NV12 buffers must be 4-byte aligned, like RGB frames.
 *   - The format is read when a call is enqueued, so it may change between calls with work in flight.
 *   - Refused with an error: an unknown format, NV12 on a handle with odd img_h, and NV12 together with remap mode 1
 *     (the fused variant samples raw RGB), whichever of lt_set_frame_format / lt_set_remap_mode comes second. */
#define LT_FRAME_RGB 0
#define LT_FRAME_NV12 1
int lt_set_frame_format(lt_handle* h, int32_t format);

/* Copy frame rows [row0, row1) of n_frames frames between a host (pinned) and a device batch of full frames
 * (one cudaMemcpy2DAsync: pitch = frame size).  to_device: 1 host->device, 0 device->host.  Used to move only
 * the rows the tracker reads / the overlay can change (lt_debug_read geometry) across PCIe.  Under LT_FRAME_NV12
 * the frames are NV12 and the copy moves luma rows [row0, row1) plus the chroma rows that cover them
 * ([row0 / 2, (row1 + 1) / 2) of the chroma plane): two cudaMemcpy2DAsync. */
int lt_memcpy_rows(lt_handle* h, void* dst, const void* src, int32_t n_frames, int32_t row0, int32_t row1,
                   int32_t to_device, void* stream);

/* ---- in-stream stage timing (bench.py's roofline figures) --------------------
 * lt_profile_begin arms CUDA-event recording at every stage boundary of the next `max_calls`
 * lt_process calls (events are recorded on the caller's stream, no synchronisation);
 * lt_profile_read synchronises, sums the per-stage durations [ms] over the recorded calls,
 * and disarms.  Stage ids: lt_stage_name(0..LT_NSTAGES-1).  A call with parameter profiles marks the threshold stages
 * once per filter group; their times add up. */
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

/* ---- stream starts and state records (stream-ordered) ----------------------
 * lt_reset_async: what lt_reset writes for the streams h_ids[0..n) (h_ids == NULL: every stream, n ignored), enqueued
 *   on `stream`: the initial state of lt_create (last_detection = n_reset + 1, everything else zero).  The ids travel
 *   as kernel arguments (one single-CTA launch per 1000 ids): h_ids may be reused when the call returns, nothing
 *   synchronises, and the call is capturable in a CUDA graph.  Like lt_reset it writes the tracking state only: the
 *   averaged polylines and the cached lane polygon of the old video stay in place but are not read again (nothing is
 *   drawn on a failing frame before a valid one rebuilds them).
 *   Usage: to start a new video on stream s in the batch you are about to enqueue, enqueue lt_reset_async({s}) on that
 *   batch's back-half stream, after the previous back half and before this one (lane_tracker_b200 does this for
 *   `starts=`).  Refused before anything is enqueued, naming the position: n outside [1, max_streams], an id out of
 *   range, a repeated id.
 *
 * State records move streams between slots, handles and GPUs without stopping the device.  A record is
 * lt_state_record_bytes(h) bytes (a multiple of 16: 18320 bytes at the shipped 1080x1100 bird's-eye view) and holds
 * everything a later frame of the stream reads:
 *   [0, 64)            header, int32 words: LT_RECORD_MAGIC, LT_ABI_VERSION, sizeof(lt_state), bv_w, bv_h, n_average,
 *                      n_fail, n_reset, then zeros;
 *   [64, A)            the tracking state (lt_state), zero-padded to 16 bytes: A = 64 + round_up(sizeof(lt_state), 16);
 *   [A, A + 8 bv_h)    the averaged polylines, int32 [2][bv_h] (left, right; vertex i of side k on row
 *                      bv_h - n_k_avg + i);
 *   [R = A + 8 bv_h, R + 8 bv_h)   the cached lane polygon rows, int32 [bv_h][2] (first, last column; empty: first > last);
 *   [B = round_up(R + 8 bv_h, 16), B + 16)   their bounding box, int32 [4] (min first, max last, first row, last row);
 *   zeros to the end.
 * Captured pixel lists (lt_set_capture) and per-batch outputs (result records, draw flags) are not state: they are not
 * carried.
 * lt_export_states gathers the records of streams h_ids[i] into d_dst + i * record_bytes; lt_import_states scatters the
 *   records d_src + i * record_bytes into slots h_ids[i].  Both on `stream`, ordered like the back halves they sit
 *   between; nothing synchronises and both are capturable.  h_ids: HOST int32 [n], 1 <= n <= max_streams, distinct ids
 *   in [0, max_streams) (refused before anything is enqueued, naming the position).  d_dst / d_src: device memory of
 *   the handle's GPU, 16-byte aligned.
 * lt_import_states checks every record on the device before it writes any of it: the header against the handle's
 *   (LT_RECORD_BAD_HEADER), and every field a kernel later uses as an index or a loop bound (LT_RECORD_BAD_STATE):
 *   ring_len and radii_len in [0, n_average], n_left_avg and n_right_avg in [0, bv_h], every non-empty polygon row and
 *   a non-empty bounding box inside the bird's-eye view.  A refused record is not applied: the slot keeps its bytes.
 *   d_status (device int32 [n], may be NULL) receives LT_RECORD_OK or the code of each record. */
#define LT_RECORD_MAGIC 0x5253544CU    /* "LTSR" */
#define LT_RECORD_OK 0
#define LT_RECORD_BAD_HEADER 1
#define LT_RECORD_BAD_STATE 2
int lt_reset_async(lt_handle* h, const int32_t* h_ids, int32_t n, void* stream);
int64_t lt_state_record_bytes(lt_handle* h);
int lt_export_states(lt_handle* h, const int32_t* h_ids, int32_t n, void* d_dst, void* stream);
int lt_import_states(lt_handle* h, const int32_t* h_ids, int32_t n, const void* d_src, int32_t* d_status, void* stream);

/* Debug/test access to internal buffers of the last lt_process / stage call.  stream_id is a batch position for
 * items 3-8 (buffers of the last batch) and a stream id for item 9 (per-stream cache); the two coincide for lt_process.
 * what:0 undistort map (int32 [img_h][img_w][2]), 1 bird's-eye map (int32 [bv_h][bv_w][2]),
 *       2 overlay map (int32 [img_h][img_w][2]), 3 R plane u8 [bv_h][bv_w], 4 LAB-b plane,
 *       5 R top-hat, 6 b top-hat, 7 mask u8 {0,255}, 8 merged (pre-open) mask,
 *       9 lane row spans int32 [bv_h][2], 10 geometry int32[9] = {undistorted ROI first,last+1, overlay rows
 *       first,last+1, pair-plane width, mask words per row, pixel-list capacity of lt_read_capture, frame rows the
 *       tracker reads first,last+1}, 11 int32[3] = {row bands of the 55x55 and of the 29x29 morphology jobs in the
 *       last filter launch, SM count of the device}, 12 lane row spans of the last lt_draw_lane call (int32 [bv_h][2];
 *       9 is the per-stream cache that lt_process re-draws on failing frames), 13 int32[6] = {undistorted ROI
 *       first,last+1, overlay rows first,last+1, frame rows the tracker reads first,last+1} of camera stream_id
 *       (lt_set_camera; stream_id in [0, LT_MAX_CAMERAS)).  Items 0-2 and 10 describe camera 0.
 * Copies to HOST memory; synchronous. Returns bytes written or <0. */
int64_t lt_debug_read(lt_handle* h, int32_t what, int32_t stream_id, void* h_dst, int64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* LANE_TRACKER_B200_H */
