// Shared declarations of the lane_tracker_b200 CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/lane_tracker_b200.h"

// ---------------------------------------------------------------------------
// Plane layout ("pair-packed"): a bird's-eye plane of width W is held as
// P2 = 32*ceil(W/64) uint32 entries per row; entry x carries pixel (y, x) in its
// low 16 bits and pixel (y, x + P2) in its high 16 bits.  Two independent image
// strips ride in the two u16 lanes of every register, which is what
// VIMNMX.U16x2 / packed adds want, and 32 consecutive entries of either lane
// are exactly one word of the bit-packed mask.
// Bit mask layout: row of 2*P2/32 uint32 words, bit (x & 31) of word (x >> 5).
// ---------------------------------------------------------------------------

#define LT_PIX_CAP_DEFAULT 65536

struct LtDims {
    int img_w, img_h, bv_w, bv_h;
    int p2;        // pair-plane width in entries (multiple of 32)
    int mwords;    // mask words per row = 2*p2/32
    int roi0, roi1;   // undistorted rows materialised: [roi0, roi1)
    int ov0, ov1;     // frame rows whose overlay taps can hit the bird's-eye view: [ov0, ov1), [0, 0) if none
    int pp;           // row pitch of the PADDED pair planes (morphology inputs) = p2 + 2*LT_HALO_X
};

// Padded pair planes (all six of them): every row carries LT_HALO_X extra entries on either side that hold
// the seam-stitched neighbour columns (the two strips of a pair plane are adjacent in the image) or the pad value
// of the morphological pass that reads the plane, and every stream carries LT_HALO_Y pad rows above and below.
// The plane pointers in lt_handle address (stream 0, row 0, column 0); negative offsets reach the halo.
constexpr int LT_HALO_X = 32;     // multiple of 4 (16-byte staging) >= 28
constexpr int LT_HALO_Y = 56;     // >= 27 + MORPH_RB - 1; the row-padded fast path of k_cross_v needs k + 16

// Undistorted ROI buffer (lt_remap.cu): groups of LT_UND_GROUP streams, stream-minor, zero-bordered; words per group.
constexpr int LT_UND_GROUP = 16;
static inline size_t lt_und_group_words(const LtDims& d) {
    return ((size_t)(d.roi1 - d.roi0 + 3) * (d.img_w + 1) + 2) * LT_UND_GROUP;
}

// Per-stream tracking state on the device (lane_tracker.py:139-176).
struct LtDevState {
    lt_state s;
};

struct LtAttemptParams {   // parameters of one attempt, device-visible
    int filter_type, ksize_r, C_r, ksize_b, C_b, mask_noise, noise_thresh, ksize_noise, C_noise;
    int window_width, window_height, search_range, no_success_limit, ignore_sides, ignore_bottom, bandwidth;
    double mu, start_slice, partial;
};

// One parameter profile (lt_set_profile) as the kernels read it.
struct LtProfile {
    LtAttemptParams p;
    lt_validity val;
    int n_tries;
};

// One camera of a handle (lt_set_camera; camera 0 is the calibration of lt_create and uses the handle's tables).
struct LtCamera {
    lt_camera cal;
    int2* und_map; int2* bv_map; int2* ov_map;    // [img_h][img_w], [bv_h][bv_w], [img_h][img_w]
    int2* und_desc;              // [roi rows][img_w] tap descriptors of the undistort
    int2* bv_desc;               // [bv_h][bv_w] tap descriptors of the warp (rows of this camera's ROI)
    int roi0, roi1, ov0, ov1, src0, src1;         // as LtDims / lt_handle::src0, src1
};

// What the camera kernels read of one camera (a snapshot per front set, lt_process_front_cameras).
struct LtCamDev {
    const int2* und_desc; const int2* bv_desc; const int2* ov_map;
    int roi_px;                  // undistorted ROI pixels: (roi1 - roi0) * img_w
    int ov0, ov1;                // frame rows the overlay can reach
    double mppv, mpph;
};

// Scratch result of one search+fit+validity pass for one stream.
struct LtAttemptOut {
    int detected, valid, mode, rank_def;
    int n[2];
    double fit[2][3];
    double diffs[3];
    double partial;   // the partial that get_poly_points() will see on success
};

// The buffers the stateless front half of a frame (undistort, warp, filter) produces and the stateful back half
// (search, second attempt, state update, overlay) consumes.  A handle owns two sets so that the front half of batch
// k+1 can run on one CUDA stream while the back half of batch k runs on another (lt_process_front / lt_process_back).
// A front half with profiles (lt_process_front_profiles) also leaves the batch's profile snapshot in its set: the
// back half reads the snapshot, never the live table, so lt_set_profile may run with work in flight.
struct LtFrontSet {
    uint32_t* und_roi;
    uint32_t* pad_alloc[6];
    uint32_t* merged; uint32_t* mask;
    int* group_pos;              // [S] batch positions ordered by filter group (bilateral groups first)
    int* pos_profile;            // [S] profile index of each batch position
    LtProfile* profiles;         // [LT_MAX_PROFILES] copy of the profile table
    // host copy of the snapshot: lt_process_back_profiles checks its arguments against it
    int* h_pos_profile;          // [S]
    int snap_n;                  // batch size of the last front half with profiles; 0: the last front half took lt_params
    LtProfile snap[LT_MAX_PROFILES];
    // Camera calls (lt_process_front_cameras): the undistorted ROI of such a batch goes to und_cam, whose slots are
    // grouped by camera (runs of whole 16-byte chunks of four slots).  und_cam is separate from und_roi: the plain path
    // relies on und_roi's zero rows below camera 0's ROI, which a taller camera would overwrite.
    uint32_t* und_cam;           // [und_cam_slots / 16][lt_und_group_words of und_cam_rows rows]
    int* slot_pos;               // [und_cam_slots] batch position of each slot, -1: pad
    int* chunk_cam;              // [und_cam_slots / 4] camera of each chunk of four slots
    int* pos_cam;                // [S] camera of each batch position
    LtCamDev* cams;              // [LT_MAX_CAMERAS] snapshot of the camera tables
    int* h_pos_cam;              // [S] host copy: lt_process_back_cameras checks its arguments against it
    int cam_n;                   // batch size of the last front half with cameras; 0: the last front half took none
    int cam_plain;               // that front half used camera 0 only (it ran the launches without cameras)
    int cam_pending;             // a camera front half was enqueued alone and its back half not yet (lt_set_camera waits)
    int cam_ov0, cam_ov1;        // union of the overlay rows of its cameras
};

struct lt_handle {
    lt_config cfg;
    LtDims d;
    int S;                       // max streams
    lt_validity val;             // check_validity windows
    LtProfile profiles[LT_MAX_PROFILES];   // lt_set_profile
    unsigned profiles_set;       // bit k: profile k was set
    int bands_key[3], bands_val[2];   // cached band split of the paired morphology launch (n, height, slots)
    int sm_count;
    int src0, src1;              // frame rows the undistort of the ROI reads: [src0, src1)
    LtCamera cams[LT_MAX_CAMERAS];   // [0] mirrors the tables above; [k] set by lt_set_camera (und_map != NULL)
    int und_cam_rows, und_cam_slots; // stride (tallest ROI of the cameras set) and slot capacity of LtFrontSet::und_cam
    // shared tables
    int2* und_map;               // [img_h][img_w]
    int2* bv_map;                // [bv_h][bv_w]
    int2* ov_map;                // [img_h][img_w]
    int2* bv_desc;               // [bv_h][bv_w] tap descriptors derived from bv_map and the ROI
    int2* fused_desc;            // [bv_h][bv_w] single-resample variant (lazily built by lt_set_remap_mode)
    int remap_mode;              // 0 exact two-stage (default), 1 fused single resample
    int frame_format;            // LT_FRAME_RGB (default) or LT_FRAME_NV12: layout of d_frames, read when a call is enqueued
    unsigned short* lab_gamma;   // [256]
    unsigned short* lab_cbrt;    // [3072]
    uint2* lab_yz;               // [3][256] Lab partial sums per channel value (lt_remap.cu)
    int2* und_desc;              // [roi rows][img_w] tap descriptors of the undistort (byte offset, fx | fy << 5 | flags << 10)
    // per-stream buffers
    uint32_t* und_roi;           // [ceil(S / 16)][lt_und_group_words]: RGBX, stream-minor, zero-bordered (lt_remap.cu)
    uint32_t* planeR; uint32_t* planeB;     // padded [S][bv_h + 2*LT_HALO_Y][pp]; lanes beyond the image / halo: 0xFFFF
    uint32_t* tmpR;   uint32_t* tmpB;       // padded eroded planes; lanes beyond the image / halo: 0
    uint32_t* topR;   uint32_t* topB;       // padded top-hat planes / box row sums; halo and pad rows: 0
    LtFrontSet fs[2];                       // [0] always allocated, [1] on first use; the fields above mirror the selected one
    uint32_t* merged; uint32_t* mask;       // [S][bv_h][mwords]
    int pix_cap;                 // entries per stream and side of the captured pixel lists
    int2* lane_rows;             // [S][bv_h]
    int4* lane_bbox;             // [S] bounding box of the polygon rows: (min lo, max hi, first row, last row); empty: (W, -1, H, -1)
    int* avg_x;                  // [S][2][bv_h]   averaged polylines (state)
    LtDevState* state;           // [S]
    LtDevState* init;            // [1] the initial state (init_state), written at lt_create: what lt_reset_async copies
    LtAttemptOut* att;           // [S]
    int* retry_list; int* retry_count;      // streams that need attempt 2
    int* draw_flags;             // [S]
    int* stream_ids;             // [S] state slot of each batch position of the last call with stream ids (lt_process_streams)
    // sequence batches (lt_process_sequence), allocated on first use: the positions grouped by round, and per batch
    // position what the overlay and the text of that frame read (k_update_state writes them, round by round)
    int* seq_pos;                // [S]
    int2* seq_rows;              // [S][bv_h]
    int4* seq_bbox;              // [S]
    LtDevState* seq_state;       // [S]
    int capture;                 // lt_set_capture
    uint32_t* cap_pixels;        // [2 attempts][S][2][pix_cap]
    int* cap_counts;             // [2][S][2]
    int* cap_cents;              // [2][S][2][LT_MAX_LEVELS]
    int* cap_ncents;             // [2][S][2]
    // text sprites (lt_set_text_sprites)
    uint8_t* txt_tables; int* txt_char_start; short* txt_dy; short* txt_dx; unsigned short* txt_lut; int* txt_advance;
    int txt_nchars, txt_first, txt_parallel_lines;
    int txt_row0, txt_row1;            // frame rows the text lines can touch: [txt_row0, txt_row1)
    int2* dl_rows; int* dl_flags; int4* dl_bbox;   // lazily allocated polygon rows / flags / bounding boxes of the lt_draw_lane stage call
    LtDevState* txt_state; int* txt_flags;   // lazily allocated state / flags the lt_draw_text stage call formats from
    unsigned long long* txt_bitmaps;   // [nchars][64] rows of 64 bits: glyph pixel (dy + 32, dx + 8)
    unsigned char* txt_pair_overlap;   // [nchars][nchars]: glyph b drawn right after glyph a shares pixels with it
    cudaEvent_t* prof_ev; int* prof_stage; int prof_cap, prof_n, prof_active, prof_calls, prof_max_calls;
    uint32_t prof_mask;          // 0: every stage boundary is marked; else only the boundaries whose bit is set
    unsigned char* vis_scratch;  // lazily allocated work area of lt_visualize_search
    cudaStream_t side;           // carries the horizontal threshold halves next to the vertical ones (lt_launch_filter)
    cudaEvent_t ev_fork, ev_join;
    size_t stream_pad;           // entries per stream in a padded pair plane
    size_t stream_mask;          // words per stream in a bit mask
};

// words per group of 16 slots of LtFrontSet::und_cam: the und layout at the stride of the tallest ROI of the cameras set
static inline size_t lt_und_cam_group_words(const lt_handle* h) {
    LtDims e = h->d;
    e.roi0 = 0; e.roi1 = h->und_cam_rows;
    return lt_und_group_words(e);
}

extern "C" int64_t lt_launch_count(void);
void lt_count_launch(int n = 1);
void lt_set_error(const char* fmt, ...);
// Raise the dynamic shared-memory limit of kernel `func` on the CURRENT device if `bytes` exceeds what this process
// has already requested there (per device: handles may live on different GPUs of one process). Thread-safe.
int lt_ensure_smem(const void* func, size_t bytes);

#define LT_CUDA(call)                                                                 \
    do {                                                                              \
        cudaError_t _e = (call);                                                      \
        if (_e != cudaSuccess) {                                                      \
            lt_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return -2;                                                                \
        }                                                                             \
    } while (0)

#define LT_LAUNCH_CHECK()                                                             \
    do {                                                                              \
        lt_count_launch();                                                            \
        cudaError_t _e = cudaGetLastError();                                          \
        if (_e != cudaSuccess) {                                                      \
            lt_set_error("%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return -3;                                                                \
        }                                                                             \
    } while (0)

// ---- stage launchers (defined in the .cu files) -----------------------------
// `list`/`count` (device pointers, may be NULL) restrict a launch to the streams
// list[0..*count): CTAs whose stream slot is >= *count exit immediately.
// `ids` (device pointer, may be NULL = identity) maps a batch position to the state slot of its stream: frames,
// masks, attempt outputs, draw flags and result records are indexed by batch position, the per-stream state
// (tracking state, averaged polylines, cached lane polygon, captured pixel lists) by ids[position].

// remap tables of one calibration; d: the handle's sizes and the calibration's ROI (roi0, roi1) for the descriptors
int lt_launch_build_maps(const lt_camera& c, const LtDims& d, int2* und_map, int2* bv_map, int2* ov_map, cudaStream_t st);
int lt_launch_build_desc(const int2* bv_map, int2* bv_desc, const LtDims& d, cudaStream_t st);
int lt_launch_build_lab_yz(lt_handle* h, cudaStream_t st);
int lt_launch_build_und_desc(const int2* und_map, int2* und_desc, const LtDims& d, cudaStream_t st);
int lt_launch_build_fused_desc(lt_handle* h, cudaStream_t st);
int lt_launch_warp_fused(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int n, cudaStream_t st);
int lt_launch_undistort(lt_handle* h, const uint8_t* d_frames, int n, cudaStream_t st);   // RGB or NV12 (h->frame_format)
int lt_launch_warp(lt_handle* h, uint8_t* d_bv_rgb, int n, cudaStream_t st);
// The front half of a camera batch in buffer set f: nslots slots of f->und_cam (slot_pos / chunk_cam / cams uploaded),
// max_rows: the tallest ROI of the cameras in the batch.
int lt_launch_undistort_cams(lt_handle* h, const LtFrontSet& f, const uint8_t* d_frames, int nslots, int max_rows,
                             cudaStream_t st);
int lt_launch_warp_cams(lt_handle* h, const LtFrontSet& f, int nslots, cudaStream_t st);
int lt_launch_planes_from_bv(lt_handle* h, const uint8_t* d_bv_rgb, int n, cudaStream_t st);
// cf (may be NULL): the buffer set of a camera batch; position s then takes its overlay map and rows from
// cf->cams[cf->pos_cam[s]], and the launch covers the union cf->cam_ov0 .. cam_ov1 of their rows
int lt_launch_overlay(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, const int* d_draw,
                      const int* ids, cudaStream_t st, const LtFrontSet* cf = nullptr);
// NV12 frames -> overlay-annotated RGB frames (every row of d_out written; d_out cannot alias d_frames)
int lt_launch_overlay_nv12(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, const int* d_draw,
                           const int* ids, cudaStream_t st, const LtFrontSet* cf = nullptr);
// rows [r0, r1) of NV12 frames -> RGB (nothing outside those rows is written)
int lt_launch_nv12_to_rgb(const uint8_t* d_nv12, uint8_t* d_rgb, int n, int w, int h, int r0, int r1, cudaStream_t st);

// The filter of one attempt over the whole batch, or over list[0..*count) when count != NULL (the retry list).
int lt_launch_filter(lt_handle* h, int n, const LtAttemptParams& p, const int* list, const int* count,
                     cudaStream_t st);
// One filter group of a batch: the positions list[0..n) (list == NULL: positions 0..n-1) filtered with p.
struct LtFilterGroup {
    LtAttemptParams p;
    const int* list;
    int n;
};
// The filter of a batch of n positions split into disjoint groups g[0..ng) that cover it.  The bilateral groups come
// first and their lists are consecutive in one device array, so that g[0].list covers all their positions (the
// morphology runs once over them).  count != NULL (device count of a retry list) only with ng == 1.
int lt_launch_filter_groups(lt_handle* h, int n, const LtFilterGroup* g, int ng, const int* count, cudaStream_t st);
// Largest dynamic shared memory a threshold launch takes at warped width bv_w, over every kernel size the parameter
// checks accept (lt_create refuses widths at which this exceeds the device's opt-in limit).
size_t lt_filter_smem_bytes(int bv_w);
int lt_launch_morph_pair(lt_handle* h, bool tophat, int n, const int* list, const int* count, cudaStream_t st);
int lt_launch_mask_to_u8(lt_handle* h, const uint32_t* bits, uint8_t* d_mask, int n, cudaStream_t st);
int lt_launch_u8_to_mask(lt_handle* h, const uint8_t* d_mask, uint32_t* bits, int n, cudaStream_t st);
int lt_launch_plane_to_u8(lt_handle* h, const uint32_t* plane, int pitch, uint8_t* d_dst, int n, cudaStream_t st);

struct LtSearchArgs {
    const uint32_t* mask;        // [n][bv_h][mwords]
    int mode;                    // 0: per-stream from state, 1: force SWS, 2: force band with `coeffs`
    const double* coeffs;        // [n][2][3] for mode 2
    uint32_t* pixels; int pix_cap; int* pix_counts;   // optional ordered pixel lists
    int* centroids; int* ncentroids;                  // optional, SWS
    LtAttemptOut* att;           // [n] out
    int do_fit;                  // also fit + validity
    int by_stream;               // index pixel/centroid outputs by stream id instead of launch slot
    const int* ids;              // [n] state slot per batch position (NULL: identity): state reads, by_stream outputs
};
// prof / pos_prof (device, may be NULL): position s takes its validity windows -- and, with prof_params, its attempt
// parameters instead of p -- from prof[pos_prof[s]]; its n_tries in lt_launch_select_retry.
int lt_launch_search(lt_handle* h, int n, const LtAttemptParams& p, const LtSearchArgs& a, const int* list,
                     const int* count, cudaStream_t st, const LtProfile* prof = nullptr, const int* pos_prof = nullptr,
                     int prof_params = 0);
// order (device, may be NULL; not with prof): the launch covers the batch positions order[0..n) instead of 0..n-1
int lt_launch_select_retry(lt_handle* h, int n, int n_tries, cudaStream_t st, const LtProfile* prof = nullptr,
                           const int* pos_prof = nullptr, const int* order = nullptr);
// cf (may be NULL): the buffer set of a camera batch; position s then takes mppv / mpph from cf->cams[cf->pos_cam[s]].
// order (device, may be NULL; not with cf): CTA b updates batch position order[b] and also writes the position's
// polygon rows, bounding box and state to h->seq_rows / seq_bbox / seq_state.
int lt_launch_update_state(lt_handle* h, int n, const int* ids, lt_result* d_results, int attempts_allowed,
                           cudaStream_t st, const LtFrontSet* cf = nullptr, const int* order = nullptr);
int lt_launch_fit_pixels(lt_handle* h, const uint32_t* d_pixels, int cap, const int* d_counts, int n,
                         double* d_fits, cudaStream_t st);
int lt_launch_validity(lt_handle* h, const double* d_fits, int n, int* d_valid, double* d_diffs, cudaStream_t st);
int lt_launch_poly_points(lt_handle* h, const double* d_fits, int n, double partial, int* d_x, int* d_counts,
                          cudaStream_t st);
int lt_launch_lane_rows(lt_handle* h, const int* d_x, const int* d_counts, int n, cudaStream_t st);
int lt_launch_text(lt_handle* h, uint8_t* d_out, int n, const int* ids, cudaStream_t st);
// debug views (lt_vis.cu, and the two helpers that live next to the code they reuse)
int lt_launch_warp_frame(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int n, cudaStream_t st);
int lt_launch_band_rows(lt_handle* h, const int* d_x, const int* d_counts, int bandwidth, int2* rows_l, int2* rows_r,
                        cudaStream_t st);
int lt_launch_vis_base(const uint8_t* d_mask, const int* d_rects, int nrect, int W, int H, uint8_t* d_out, cudaStream_t st);
int lt_launch_vis_scatter(const uint32_t* d_px, int n, int W, int H, uint32_t rgb, uint8_t* d_out, cudaStream_t st);
int lt_launch_vis_scatter_poly(const int* d_xs, const int* d_count, int W, int H, uint32_t rgb, uint8_t* d_out, cudaStream_t st);
int lt_launch_vis_band_blend(const int2* rows_l, const int2* rows_r, int W, int H, uint8_t* d_out, cudaStream_t st);
int lt_launch_resize_linear(const uint8_t* d_src, int sw, int sh, int cn, size_t src_pitch, uint8_t* d_dst, int dw, int dh,
                            size_t dst_pitch, cudaStream_t st);

enum LtStage { ST_BEGIN = 0, ST_UNDISTORT, ST_WARP, ST_ERODE55, ST_ERODE29, ST_TOPHAT55, ST_TOPHAT29, ST_CROSS_R,
               ST_CROSS_B, ST_BOX, ST_NOISE, ST_OPEN5, ST_SEARCH, ST_RETRY_SELECT, ST_UPDATE, ST_OVERLAY };
void lt_prof_mark(lt_handle* h, int stage, cudaStream_t st);   // "stage just finished being enqueued"

static inline int lt_div_up(int a, int b) { return (a + b - 1) / b; }
