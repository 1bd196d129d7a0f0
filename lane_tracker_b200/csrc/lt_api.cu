// C ABI of lane_tracker_b200 (include/lane_tracker_b200.h): handle lifetime, the batched
// process() pipeline and the per-method stage entry points.
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <vector>
#include "lt_common.cuh"
#include "lab_tables.inc"

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void lt_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void lt_count_launch(int n) { g_launches += n; }

int lt_ensure_smem(const void* func, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> granted;
    if (bytes <= 48 * 1024) return 0;
    int dev = 0;
    LT_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t& cur = granted[std::make_pair(dev, func)];
    if (bytes > cur) {
        LT_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    return 0;
}

extern "C" const char* lt_last_error(void) { return g_err; }
extern "C" int lt_abi_version(void) { return LT_ABI_VERSION; }
extern "C" int64_t lt_launch_count(void) { return (int64_t)g_launches.load(); }

extern "C" void lt_default_params(lt_params* p) {
    // lane_tracker.py:876-900
    p->ksize_r = 15; p->C_r = 8; p->ksize_b = 35; p->C_b = 5; p->filter_type = 0; p->mask_noise = 0;
    p->noise_thresh = 140; p->ksize_noise = 65; p->C_noise = 10; p->window_width = 30; p->window_height = 40;
    p->search_range = 20; p->mu = 0.1; p->no_success_limit = 8; p->start_slice = 0.25; p->ignore_sides = 360;
    p->ignore_bottom = 30; p->bandwidth = 25; p->partial = 1.0; p->n_tries = 2;
}

static LtAttemptParams attempt_from(const lt_params& p) {
    LtAttemptParams a;
    a.filter_type = p.filter_type; a.ksize_r = p.ksize_r; a.C_r = p.C_r; a.ksize_b = p.ksize_b; a.C_b = p.C_b;
    a.mask_noise = p.mask_noise; a.noise_thresh = p.noise_thresh; a.ksize_noise = p.ksize_noise; a.C_noise = p.C_noise;
    a.window_width = p.window_width; a.window_height = p.window_height; a.search_range = p.search_range;
    a.no_success_limit = p.no_success_limit; a.ignore_sides = p.ignore_sides; a.ignore_bottom = p.ignore_bottom;
    a.bandwidth = p.bandwidth; a.mu = p.mu; a.start_slice = p.start_slice; a.partial = p.partial;
    return a;
}

static LtAttemptParams second_attempt() {
    // hard-coded second attempt, lane_tracker.py:1081-1099
    lt_params p;
    lt_default_params(&p);
    p.C_r = 5; p.filter_type = 1; p.no_success_limit = 50; p.bandwidth = 30; p.partial = 1.0;
    return attempt_from(p);
}

static int check_params(const lt_handle* h, const LtAttemptParams& a) {
    if (a.filter_type != 0 && a.filter_type != 1) {
        lt_set_error("Unexpected filter mode. Expected modes are 'bilateral' or 'neighborhood'.");
        return -1;
    }
    int kmax = a.filter_type == 0 ? 255 : 255;
    if (a.ksize_r < 1 || a.ksize_b < 1 || a.ksize_r > kmax || a.ksize_b > kmax || a.ksize_noise < 1 || a.ksize_noise > 255) {
        lt_set_error("threshold kernel sizes must lie in [1, 255]");
        return -1;
    }
    if (a.filter_type == 1 && ((a.ksize_r & 1) == 0 || (a.ksize_b & 1) == 0 || a.ksize_r < 3 || a.ksize_b < 3)) {
        lt_set_error("'neighborhood' block sizes must be odd and >= 3 (cv2.adaptiveThreshold)");
        return -1;
    }
    if (a.window_width < 1 || a.window_width > 64 || a.window_height < 1 || a.window_height > h->d.bv_h) {
        lt_set_error("window_width must lie in [1, 64] and window_height in [1, warped height]");
        return -1;
    }
    if (!(a.partial >= 0.0 && a.partial <= 1.0) || a.ignore_bottom < 0 || a.ignore_bottom > h->d.bv_h) {
        lt_set_error("partial must lie in [0, 1] and ignore_bottom in [0, warped height]");
        return -1;
    }
    // the sliding-window walk keeps one centroid / one window per level in fixed-size arrays (LT_MAX_LEVELS): a
    // parameter set that needs more levels is rejected instead of being searched short (lane_tracker.py:346)
    const long long nlev = (long long)(a.partial * (double)(h->d.bv_h - a.ignore_bottom) / (double)a.window_height);
    if (nlev > LT_MAX_LEVELS) {
        lt_set_error("window_height %d gives %lld search levels; at most %d are supported", a.window_height, nlev, LT_MAX_LEVELS);
        return -1;
    }
    if (a.search_range < 0 || a.search_range > h->d.bv_w || a.ignore_sides < 0 || a.ignore_sides > h->d.bv_w ||
        a.no_success_limit < 0 || a.bandwidth < 0 || a.bandwidth > h->d.bv_w || !(a.mu == a.mu) ||
        !(a.start_slice >= 0.0 && a.start_slice <= 1.0)) {
        lt_set_error("search_range, ignore_sides and bandwidth must lie in [0, warped width], no_success_limit >= 0, "
                     "start_slice in [0, 1]");
        return -1;
    }
    return 0;
}

template <typename T> static int dev_alloc(T** p, size_t n) {
    cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
    if (e != cudaSuccess) { lt_set_error("cudaMalloc(%zu bytes) -> %s", n * sizeof(T), cudaGetErrorString(e)); return -2; }
    return 0;
}

static const lt_validity SHIPPED_VALIDITY = {150.0, 230.0, 110.0, 230.0, 80.0, 200.0, 0.25};   // lane_tracker.py:588-593, 617

extern "C" int lt_set_validity(lt_handle* h, const lt_validity* v) {
    if (!h) { lt_set_error("null handle"); return -1; }
    h->val = v ? *v : SHIPPED_VALIDITY;
    return 0;
}
extern "C" int lt_get_validity(lt_handle* h, lt_validity* v) {
    if (!h || !v) { lt_set_error("null argument"); return -1; }
    *v = h->val;
    return 0;
}

static void init_state(lt_handle* h, lt_state* s) {
    memset(s, 0, sizeof(*s));
    s->last_detection = h->cfg.n_reset + 1;     // lane_tracker.py:140
}

extern "C" int lt_destroy(lt_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->cfg.device);
    for (int k = 0; k < 2; ++k) {
        const LtFrontSet& f = h->fs[k];
        void* fp[] = {f.und_roi, f.pad_alloc[0], f.pad_alloc[1], f.pad_alloc[2], f.pad_alloc[3], f.pad_alloc[4], f.pad_alloc[5],
                      f.merged, f.mask};
        for (void* p : fp) if (p) cudaFree(p);
    }
    void* ptrs[] = {h->und_map, h->bv_map, h->ov_map, h->bv_desc, h->und_desc, h->lab_yz, h->fused_desc, h->lab_gamma, h->lab_cbrt, h->pixels, h->pix_counts, h->lane_rows, h->lane_bbox, h->dl_bbox,
                    h->avg_x, h->state, h->att, h->retry_list, h->retry_count, h->draw_flags, h->stream_ids, h->scratch_bv, h->vis_scratch,
                    h->cap_pixels, h->cap_counts, h->cap_cents, h->cap_ncents, h->dl_rows, h->dl_flags, h->txt_state, h->txt_flags,
                    h->txt_tables, h->txt_char_start, h->txt_dy, h->txt_dx, h->txt_lut, h->txt_advance, h->txt_pair_overlap,
                    h->txt_bitmaps};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (int i = 0; i < h->prof_cap; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev; delete[] h->prof_stage;
    if (h->side) cudaStreamDestroy(h->side);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    delete h;
    return 0;
}

// allocate one set of front-half buffers (LtFrontSet) and give its padded planes their pad values
static int alloc_front_set(lt_handle* h, int k) {
    LtFrontSet& f = h->fs[k];
    if (f.mask) return 0;
    const LtDims& d = h->d;
    const size_t S = h->S;
    const size_t und_words = (size_t)lt_div_up((int)S, LT_UND_GROUP) * lt_und_group_words(d);
    int rc = dev_alloc(&f.und_roi, und_words);
    if (!rc) cudaMemset(f.und_roi, 0, und_words * sizeof(uint32_t));      // the zero border is never written again
    // padded planes: + one row of slack (the last tile of a row block stages a few entries past the row end)
    const size_t n = S * h->stream_pad + d.pp;
    for (int i = 0; i < 6 && !rc; ++i) {
        rc = dev_alloc(&f.pad_alloc[i], n);
        if (!rc) cudaMemset(f.pad_alloc[i], i < 2 ? 0xFF : 0x00, n * sizeof(uint32_t));   // pad of erode / dilate
    }
    if (!rc) rc = dev_alloc(&f.merged, S * h->stream_mask);
    if (!rc) rc = dev_alloc(&f.mask, S * h->stream_mask);
    return rc;
}

// make set k the one the launchers see (kernel arguments are captured at launch, so switching between calls is safe)
static void select_set(lt_handle* h, int k) {
    const LtFrontSet& f = h->fs[k];
    const size_t origin = (size_t)LT_HALO_Y * h->d.pp + LT_HALO_X;
    h->und_roi = f.und_roi;
    for (int i = 0; i < 6; ++i) h->pad_alloc[i] = f.pad_alloc[i];
    h->planeR = f.pad_alloc[0] + origin; h->planeB = f.pad_alloc[1] + origin;
    h->tmpR = f.pad_alloc[2] + origin;   h->tmpB = f.pad_alloc[3] + origin;
    h->topR = f.pad_alloc[4] + origin;   h->topB = f.pad_alloc[5] + origin;
    h->merged = f.merged; h->mask = f.mask;
    h->cur_set = k;
}

extern "C" int lt_create(const lt_config* cfg, lt_handle** out) {
    if (!cfg || !out) { lt_set_error("null argument"); return -1; }
    if (cfg->img_w < 64 || cfg->img_h < 16 || cfg->bv_w < 64 || cfg->bv_h < 16 || (cfg->img_w & 3) || cfg->bv_h > 65535 ||
        cfg->bv_w > 32767 || cfg->img_w > 32767 || cfg->img_h > 32767) {
        lt_set_error("unsupported geometry: img %dx%d (width must be a multiple of 4), warped %dx%d", cfg->img_w,
                     cfg->img_h, cfg->bv_w, cfg->bv_h);
        return -1;
    }
    if (cfg->max_streams < 1 || cfg->n_average < 1 || cfg->n_average > LT_MAX_AVERAGE) {
        lt_set_error("max_streams must be >= 1 and n_average in [1, %d]", LT_MAX_AVERAGE);
        return -1;
    }
    LT_CUDA(cudaSetDevice(cfg->device));
    lt_handle* h = new lt_handle();
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    h->S = cfg->max_streams;
    h->val = SHIPPED_VALIDITY;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
    LtDims& d = h->d;
    d.img_w = cfg->img_w; d.img_h = cfg->img_h; d.bv_w = cfg->bv_w; d.bv_h = cfg->bv_h;
    d.p2 = 32 * ((cfg->bv_w + 63) / 64);
    d.mwords = 2 * d.p2 / 32;
    d.pp = d.p2 + 2 * LT_HALO_X;
    h->stream_pad = (size_t)(d.bv_h + 2 * LT_HALO_Y) * d.pp;
    h->stream_mask = (size_t)d.bv_h * d.mwords;
    h->pix_cap = LT_PIX_CAP_DEFAULT > 64 * d.bv_h ? LT_PIX_CAP_DEFAULT : 64 * d.bv_h;   // >= rows x widest window
    const size_t S = h->S, npx = (size_t)d.img_w * d.img_h, nbv = (size_t)d.bv_w * d.bv_h;
    int rc = 0;
#define A(ptr, n) if (!rc) rc = dev_alloc(&h->ptr, (n))
    A(und_map, npx); A(bv_map, nbv); A(ov_map, npx); A(lab_gamma, 256); A(lab_cbrt, 3072);
    if (rc) { lt_destroy(h); return rc; }
    cudaStream_t st = 0;
    if ((rc = lt_launch_build_maps(h, st))) { lt_destroy(h); return rc; }
    cudaMemcpy(h->lab_gamma, LT_LAB_GAMMA, sizeof(LT_LAB_GAMMA), cudaMemcpyHostToDevice);
    cudaMemcpy(h->lab_cbrt, LT_LAB_CBRT, sizeof(LT_LAB_CBRT), cudaMemcpyHostToDevice);
    // rows of the undistorted frame that the bird's-eye view can touch / frame rows the overlay can touch
    {
        std::vector<int2> m(nbv);
        cudaError_t e = cudaMemcpy(m.data(), h->bv_map, nbv * sizeof(int2), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { lt_set_error("map build failed: %s", cudaGetErrorString(e)); lt_destroy(h); return -2; }
        int r0 = d.img_h, r1 = 0;
        for (size_t i = 0; i < nbv; ++i) {
            int sx = m[i].x >> 5, sy = m[i].y >> 5;
            if (sx + 1 < 0 || sx >= d.img_w) continue;
            for (int yy = sy; yy <= sy + 1; ++yy)
                if (yy >= 0 && yy < d.img_h) { r0 = yy < r0 ? yy : r0; r1 = yy + 1 > r1 ? yy + 1 : r1; }
        }
        if (r0 >= r1) { r0 = 0; r1 = 1; }
        d.roi0 = r0; d.roi1 = r1;
        {   // frame rows read by the undistort of the ROI rows (for partial host->device transfers)
            std::vector<int2> u((size_t)(r1 - r0) * d.img_w);
            cudaMemcpy(u.data(), h->und_map + (size_t)r0 * d.img_w, u.size() * sizeof(int2), cudaMemcpyDeviceToHost);
            int s0 = d.img_h, s1 = 0;
            for (size_t i = 0; i < u.size(); ++i) {
                int sy = u[i].y >> 5;
                for (int yy = sy; yy <= sy + 1; ++yy)
                    if (yy >= 0 && yy < d.img_h) { s0 = yy < s0 ? yy : s0; s1 = yy + 1 > s1 ? yy + 1 : s1; }
            }
            if (s0 >= s1) { s0 = 0; s1 = d.img_h; }
            h->src0 = s0; h->src1 = s1;
        }
        std::vector<int2> o(npx);
        cudaMemcpy(o.data(), h->ov_map, npx * sizeof(int2), cudaMemcpyDeviceToHost);
        int o0 = d.img_h, o1 = 0;
        for (int y = 0; y < d.img_h; ++y)
            for (int x = 0; x < d.img_w; ++x) {
                int2 q = o[(size_t)y * d.img_w + x];
                int sx = q.x >> 5, sy = q.y >> 5;
                if (sx + 1 >= 0 && sx < d.bv_w && sy + 1 >= 0 && sy < d.bv_h) { o0 = y < o0 ? y : o0; o1 = y + 1 > o1 ? y + 1 : o1; }
            }
        if (o0 >= o1) { o0 = 0; o1 = 0; }
        d.ov0 = o0; d.ov1 = o1;
    }
    A(bv_desc, nbv);
    if (!rc) rc = lt_launch_build_desc(h, st);
    A(und_desc, (size_t)(d.roi1 - d.roi0) * d.img_w);
    if (!rc) rc = lt_launch_build_und_desc(h, st);
    A(lab_yz, 768);
    if (!rc) rc = lt_launch_build_lab_yz(h, st);
    if (!rc) rc = alloc_front_set(h, 0);
    if (!rc) select_set(h, 0);
    A(pixels, S * 2 * (size_t)h->pix_cap); A(pix_counts, S * 2);
    A(lane_rows, S * (size_t)d.bv_h); A(lane_bbox, S); A(avg_x, S * 2 * (size_t)d.bv_h);
    A(state, S); A(att, 2 * S); A(retry_list, S); A(retry_count, 1); A(draw_flags, 2 * S); A(stream_ids, S);
#undef A
    if (rc) { lt_destroy(h); return rc; }
    if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) {
        lt_set_error("cannot create the side stream"); lt_destroy(h); return -2;
    }
    cudaMemset(h->avg_x, 0, S * 2 * (size_t)d.bv_h * sizeof(int));
    cudaMemset(h->lane_rows, 0, S * (size_t)d.bv_h * sizeof(int2));
    cudaMemset(h->lane_bbox, 0, S * sizeof(int4));                 // (rows of zeros = column 0 of every row: box (0, 0, 0, 0) never drawn, draw flag 0)
    cudaMemset(h->draw_flags, 0, 2 * S * sizeof(int));
    cudaMemset(h->retry_count, 0, sizeof(int));
    cudaMemset(h->att, 0, 2 * S * sizeof(LtAttemptOut));
    *out = h;
    rc = lt_reset(h, nullptr, 0);
    if (rc) { lt_destroy(h); *out = nullptr; return rc; }
    LT_CUDA(cudaDeviceSynchronize());
    return 0;
}

extern "C" int lt_reset(lt_handle* h, const int32_t* ids, int32_t n) {
    if (!h) { lt_set_error("null handle"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LtDevState z;
    init_state(h, &z.s);
    if (!ids) {
        std::vector<LtDevState> all(h->S, z);
        LT_CUDA(cudaMemcpy(h->state, all.data(), all.size() * sizeof(LtDevState), cudaMemcpyHostToDevice));
        return 0;
    }
    for (int i = 0; i < n; ++i) {
        if (ids[i] < 0 || ids[i] >= h->S) { lt_set_error("stream id %d out of range", ids[i]); return -1; }
        LT_CUDA(cudaMemcpy(h->state + ids[i], &z, sizeof(z), cudaMemcpyHostToDevice));
    }
    return 0;
}

static int check_any_n(lt_handle* h, int n) {   // stage calls that touch no per-stream buffer of the handle
    if (!h) { lt_set_error("null handle"); return -1; }
    if (n < 1) { lt_set_error("n_streams must be positive"); return -1; }
    return 0;
}

static int check_n(lt_handle* h, int n) {
    if (!h) { lt_set_error("null handle"); return -1; }
    if (n < 1 || n > h->S) { lt_set_error("n_streams %d outside [1, %d]", n, h->S); return -1; }
    return 0;
}

// ---------------------------------------------------------------------------
// process()
// ---------------------------------------------------------------------------

// find_lane_points (lane_tracker.py:795-874) of the first attempt up to the binary mask, all streams: stateless
static int process_front(lt_handle* h, const uint8_t* d_frames, int n, const LtAttemptParams& p1, cudaStream_t st) {
    int rc;
    if (h->prof_active && h->prof_calls >= h->prof_max_calls) h->prof_active = 0;
    lt_prof_mark(h, ST_BEGIN, st);
    if (h->remap_mode == 1) {
        if ((rc = lt_launch_warp_fused(h, d_frames, nullptr, n, st))) return rc;
    } else {
        if ((rc = lt_launch_undistort(h, d_frames, n, st))) return rc;
        lt_prof_mark(h, ST_UNDISTORT, st);
        if ((rc = lt_launch_warp(h, nullptr, n, st))) return rc;
    }
    lt_prof_mark(h, ST_WARP, st);
    return lt_launch_filter(h, n, p1, nullptr, nullptr, st);
}

// The stream ids of a batch travel to the device as kernel arguments: a launch copies its arguments when it is
// enqueued, so the caller's host array may be reused as soon as the call returns, nothing synchronises, and the call
// stays capturable in a CUDA graph (a pageable cudaMemcpyAsync is neither).  One chunk holds LT_IDS_CHUNK ids (4 KB
// of arguments); larger batches take several launches.
#define LT_IDS_CHUNK 1000
struct LtIdsChunk {
    int offset, count;
    int ids[LT_IDS_CHUNK];
};

__global__ void k_set_stream_ids(LtIdsChunk c, int* __restrict__ dst) {
    for (int i = threadIdx.x; i < c.count; i += blockDim.x) dst[c.offset + i] = c.ids[i];
}

// Writes h_ids to the handle's one device id array on the stream of the back half that reads it.  One array per
// handle is enough: every kernel that reads it is a back-half kernel enqueued on that same stream after this write,
// and the back half of batch k must follow the back half of batch k-1 (lt_process_back), so a write for batch k
// cannot overtake a read of batch k-1, and no later write can overtake a read of batch k.
static int upload_stream_ids(lt_handle* h, const int32_t* h_ids, int n, cudaStream_t st) {
    LtIdsChunk c;
    for (int off = 0; off < n; off += LT_IDS_CHUNK) {
        c.offset = off;
        c.count = n - off < LT_IDS_CHUNK ? n - off : LT_IDS_CHUNK;
        memcpy(c.ids, h_ids + off, (size_t)c.count * sizeof(int32_t));
        k_set_stream_ids<<<1, 256, 0, st>>>(c, h->stream_ids);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

// searches, second attempt of the streams that failed, state machine, overlay: advances the per-stream state.
// h_ids (host, validated by check_ids) maps batch position i to state slot h_ids[i]; NULL: the identity.
static int process_back(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, const lt_params* params,
                        const LtAttemptParams& p1, lt_result* d_results, cudaStream_t st, bool own_begin,
                        const int32_t* h_ids = nullptr) {
    int rc;
    const LtAttemptParams p2 = second_attempt();
    const bool two = (params->n_tries >= 2) || (params->n_tries == -1);
    if (own_begin) lt_prof_mark(h, ST_BEGIN, st);       // stage times are differences of marks on ONE stream
    const int* ids = nullptr;
    if (h_ids) {
        if ((rc = upload_stream_ids(h, h_ids, n, st))) return rc;
        ids = h->stream_ids;
    }
    LtSearchArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.mask = h->mask; sa.mode = 0; sa.att = h->att; sa.do_fit = 1; sa.ids = ids;
    const size_t S = h->S;
    if (h->capture) {
        sa.by_stream = 1; sa.pixels = h->cap_pixels; sa.pix_cap = h->pix_cap; sa.pix_counts = h->cap_counts;
        sa.centroids = h->cap_cents; sa.ncentroids = h->cap_ncents;
    }
    if ((rc = lt_launch_search(h, n, p1, sa, nullptr, nullptr, st))) return rc;
    lt_prof_mark(h, ST_SEARCH, st);
    if (two) {
        // second attempt only for the streams whose first attempt failed (lane_tracker.py:1071-1128).
        // The reference re-runs undistort + warp here; their outputs are unchanged, so the planes are reused.
        if ((rc = lt_launch_select_retry(h, n, params->n_tries, st))) return rc;
        lt_prof_mark(h, ST_RETRY_SELECT, st);
        if ((rc = lt_launch_filter(h, n, p2, h->retry_list, h->retry_count, st))) return rc;
        sa.att = h->att + h->S;
        if (h->capture) {
            sa.pixels = h->cap_pixels + S * 2 * (size_t)h->pix_cap; sa.pix_counts = h->cap_counts + S * 2;
            sa.centroids = h->cap_cents + S * 2 * LT_MAX_LEVELS; sa.ncentroids = h->cap_ncents + S * 2;
        }
        if ((rc = lt_launch_search(h, n, p2, sa, h->retry_list, h->retry_count, st))) return rc;
        lt_prof_mark(h, ST_SEARCH, st);
    }
    if ((rc = lt_launch_update_state(h, n, ids, d_results, two ? 2 : 1, st))) return rc;
    lt_prof_mark(h, ST_UPDATE, st);
    if (d_out) {
        // (copying the untouched rows on a side stream under the search kernels was measured: the copy saturates HBM
        // and slows the search by what it saves -- the plain in-order copy stays)
        // draw_lane writes its text into the frame BEFORE the blend (lane_tracker.py:653-662).  With the shipped
        // geometry the text rows and the rows the lane overlay can reach are disjoint and the order is immaterial;
        // when they overlap (other calibrations) the text goes first and the blend runs in place over it.
        const bool text_under_blend = h->txt_nchars > 0 && h->txt_row0 < h->d.ov1 && h->d.ov0 < h->txt_row1;
        if (text_under_blend) {
            if (d_out != d_frames)
                LT_CUDA(cudaMemcpyAsync(d_out, d_frames, (size_t)n * h->d.img_w * h->d.img_h * 3, cudaMemcpyDeviceToDevice, st));
            if ((rc = lt_launch_text(h, d_out, n, ids, st))) return rc;
            if ((rc = lt_launch_overlay(h, d_out, d_out, n, h->draw_flags, ids, st))) return rc;
        } else {
            if ((rc = lt_launch_overlay(h, d_frames, d_out, n, h->draw_flags, ids, st))) return rc;
            if ((rc = lt_launch_text(h, d_out, n, ids, st))) return rc;
        }
        lt_prof_mark(h, ST_OVERLAY, st);
    }
    if (h->prof_active) h->prof_calls++;
    return 0;
}

// Full-size frame buffers (the caller's frames and annotated output) are read and written as 32-bit words: by the
// undistort (three words per tap pair) and by the overlay (three words per four pixels, in place when out == frames).
// A buffer that is not 4-byte aligned is refused here, before anything is launched.
static int check_frame_buffer(const void* p, const char* what) {
    if ((uintptr_t)p & 3) {
        lt_set_error("%s must be 4-byte aligned (got address %p)", what, p);
        return -1;
    }
    return 0;
}

static int process_args(lt_handle* h, const uint8_t* d_frames, int n, const lt_params* params, int set, LtAttemptParams* p1) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_frames || !params) { lt_set_error("null argument"); return -1; }
    if ((rc = check_frame_buffer(d_frames, "d_frames"))) return rc;
    if (set != 0 && set != 1) { lt_set_error("buffer set must be 0 or 1"); return -1; }
    *p1 = attempt_from(*params);
    if ((rc = check_params(h, *p1))) return rc;
    // captured pixel lists: a band-search row holds up to 2*bandwidth - 1 pixels (attempt 2 uses bandwidth 30)
    const int bw = p1->bandwidth > 30 ? p1->bandwidth : 30;
    if (h->capture && (long long)(2 * bw - 1) * h->d.bv_h > (long long)h->pix_cap) {
        lt_set_error("bandwidth %d can overflow the captured pixel lists (capacity %d): raise it with lt_set_pixel_capacity",
                     p1->bandwidth, h->pix_cap);
        return -1;
    }
    if ((rc = alloc_front_set(h, set))) return rc;
    select_set(h, set);
    return 0;
}

extern "C" int lt_process(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n, const lt_params* params,
                          lt_result* d_results, void* stream) {
    int rc;
    LtAttemptParams p1;
    if ((rc = check_frame_buffer(d_out, "d_out"))) return rc;
    if ((rc = process_args(h, d_frames, n, params, 0, &p1))) return rc;
    if (!d_results) { lt_set_error("null argument"); return -1; }
    if ((rc = process_front(h, d_frames, n, p1, (cudaStream_t)stream))) return rc;
    return process_back(h, d_frames, d_out, n, params, p1, d_results, (cudaStream_t)stream, false);
}

extern "C" int lt_process_front(lt_handle* h, const uint8_t* d_frames, int32_t n, const lt_params* params, int32_t set,
                                void* stream) {
    int rc;
    LtAttemptParams p1;
    if ((rc = process_args(h, d_frames, n, params, set, &p1))) return rc;
    return process_front(h, d_frames, n, p1, (cudaStream_t)stream);
}

extern "C" int lt_process_back(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n, const lt_params* params,
                               int32_t set, lt_result* d_results, void* stream) {
    int rc;
    LtAttemptParams p1;
    if ((rc = check_frame_buffer(d_out, "d_out"))) return rc;
    if ((rc = process_args(h, d_frames, n, params, set, &p1))) return rc;
    if (!d_results) { lt_set_error("null argument"); return -1; }
    return process_back(h, d_frames, d_out, n, params, p1, d_results, (cudaStream_t)stream, true);
}

// Stream ids of lt_process_streams / lt_process_back_streams: 1 <= n <= S ids in [0, S), pairwise distinct (two
// frames of one stream in a batch would race on its state).  Checked before anything is enqueued.
static int check_ids(lt_handle* h, const int32_t* h_ids, int n) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!h_ids) { lt_set_error("null stream id list"); return -1; }
    std::vector<unsigned char> seen(h->S, 0);
    for (int i = 0; i < n; ++i) {
        const int id = h_ids[i];
        if (id < 0 || id >= h->S) { lt_set_error("stream id %d at batch position %d outside [0, %d)", id, i, h->S); return -1; }
        if (seen[id]) { lt_set_error("stream id %d appears twice in the batch (position %d)", id, i); return -1; }
        seen[id] = 1;
    }
    return 0;
}

extern "C" int lt_process_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                                  const lt_params* params, lt_result* d_results, void* stream) {
    int rc;
    LtAttemptParams p1;
    if ((rc = check_ids(h, h_ids, n))) return rc;
    if ((rc = check_frame_buffer(d_out, "d_out"))) return rc;
    if ((rc = process_args(h, d_frames, n, params, 0, &p1))) return rc;
    if (!d_results) { lt_set_error("null argument"); return -1; }
    if ((rc = process_front(h, d_frames, n, p1, (cudaStream_t)stream))) return rc;
    return process_back(h, d_frames, d_out, n, params, p1, d_results, (cudaStream_t)stream, false, h_ids);
}

extern "C" int lt_process_back_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                       int32_t n, const lt_params* params, int32_t set, lt_result* d_results, void* stream) {
    int rc;
    LtAttemptParams p1;
    if ((rc = check_ids(h, h_ids, n))) return rc;
    if ((rc = check_frame_buffer(d_out, "d_out"))) return rc;
    if ((rc = process_args(h, d_frames, n, params, set, &p1))) return rc;
    if (!d_results) { lt_set_error("null argument"); return -1; }
    return process_back(h, d_frames, d_out, n, params, p1, d_results, (cudaStream_t)stream, true, h_ids);
}

static const char* STAGE_NAMES[LT_NSTAGES] = {"begin", "undistort", "warp", "erode55", "erode29", "tophat55", "tophat29",
                                               "cross_r", "cross_b", "box", "noise", "open5", "search", "retry_select",
                                               "update_state", "overlay"};
extern "C" const char* lt_stage_name(int32_t s) { return (s >= 0 && s < LT_NSTAGES) ? STAGE_NAMES[s] : "?"; }

void lt_prof_mark(lt_handle* h, int stage, cudaStream_t st) {
    if (!h->prof_active || h->prof_n >= h->prof_cap) return;
    if (h->prof_mask && !((h->prof_mask >> stage) & 1u)) return;
    h->prof_stage[h->prof_n] = stage;
    cudaEventRecord(h->prof_ev[h->prof_n], st);
    h->prof_n++;
}

extern "C" int lt_profile_begin(lt_handle* h, int32_t max_calls) {
    if (!h || max_calls < 1 || max_calls > 4096) { lt_set_error("bad argument"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    int need = max_calls * 32;
    if (need > h->prof_cap) {
        cudaEvent_t* ev = new cudaEvent_t[need];
        for (int i = 0; i < need; ++i) LT_CUDA(cudaEventCreate(&ev[i]));
        for (int i = 0; i < h->prof_cap; ++i) cudaEventDestroy(h->prof_ev[i]);
        delete[] h->prof_ev; delete[] h->prof_stage;
        h->prof_ev = ev; h->prof_stage = new int[need]; h->prof_cap = need;
    }
    h->prof_n = 0; h->prof_calls = 0; h->prof_max_calls = max_calls; h->prof_active = 1;
    return 0;
}

extern "C" int lt_profile_select(lt_handle* h, uint32_t stage_mask) {
    if (!h) { lt_set_error("bad argument"); return -1; }
    h->prof_mask = stage_mask ? (stage_mask | 1u) : 0u;       // stage 0 (begin) always marks
    return 0;
}

extern "C" int lt_profile_read(lt_handle* h, double* ms, int32_t* calls) {
    if (!h || !ms || !calls) { lt_set_error("bad argument"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    for (int i = 0; i < LT_NSTAGES; ++i) ms[i] = 0.0;
    for (int i = 1; i < h->prof_n; ++i) {
        if (h->prof_stage[i] == ST_BEGIN) continue;
        float t = 0.f;
        LT_CUDA(cudaEventElapsedTime(&t, h->prof_ev[i - 1], h->prof_ev[i]));
        ms[h->prof_stage[i]] += t;
    }
    *calls = h->prof_calls;
    h->prof_active = 0;
    return 0;
}

extern "C" int lt_set_text_sprites(lt_handle* h, const uint8_t* tables, int32_t n_tables, const int32_t* char_start,
                                   int32_t n_chars, const int16_t* dy, const int16_t* dx, const uint16_t* lut,
                                   int32_t n_pixels, const int32_t* advance, int32_t first_char) {
    if (!h) { lt_set_error("null handle"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    void* old[] = {h->txt_tables, h->txt_char_start, h->txt_dy, h->txt_dx, h->txt_lut, h->txt_advance, h->txt_pair_overlap, h->txt_bitmaps};
    for (void* p : old) if (p) cudaFree(p);
    h->txt_pair_overlap = nullptr; h->txt_bitmaps = nullptr;
    h->txt_tables = nullptr; h->txt_char_start = nullptr; h->txt_dy = nullptr; h->txt_dx = nullptr;
    h->txt_lut = nullptr; h->txt_advance = nullptr; h->txt_nchars = 0; h->txt_row0 = h->txt_row1 = 0;
    if (!tables) return 0;
    if (n_tables < 1 || n_chars < 1 || n_pixels < 0 || !char_start || !dy || !dx || !lut || !advance ||
        first_char > '?' || first_char + n_chars <= '?') { lt_set_error("bad sprite data"); return -1; }
    for (int i = 0; i < n_chars; ++i)
        if (char_start[i] > char_start[i + 1] || char_start[i + 1] > n_pixels) { lt_set_error("bad sprite index"); return -1; }
    for (int i = 0; i < n_pixels; ++i)
        if (lut[i] >= n_tables) { lt_set_error("bad sprite table index"); return -1; }
    int rc = 0;
    if (!rc) rc = dev_alloc(&h->txt_tables, (size_t)n_tables * 256);
    if (!rc) rc = dev_alloc(&h->txt_char_start, (size_t)n_chars + 1);
    if (!rc) rc = dev_alloc(&h->txt_dy, (size_t)(n_pixels > 0 ? n_pixels : 1));
    if (!rc) rc = dev_alloc(&h->txt_dx, (size_t)(n_pixels > 0 ? n_pixels : 1));
    if (!rc) rc = dev_alloc(&h->txt_lut, (size_t)(n_pixels > 0 ? n_pixels : 1));
    if (!rc) rc = dev_alloc(&h->txt_advance, (size_t)n_chars);
    if (rc) return rc;
    LT_CUDA(cudaMemcpy(h->txt_tables, tables, (size_t)n_tables * 256, cudaMemcpyHostToDevice));
    LT_CUDA(cudaMemcpy(h->txt_char_start, char_start, ((size_t)n_chars + 1) * sizeof(int), cudaMemcpyHostToDevice));
    LT_CUDA(cudaMemcpy(h->txt_dy, dy, (size_t)n_pixels * sizeof(short), cudaMemcpyHostToDevice));
    LT_CUDA(cudaMemcpy(h->txt_dx, dx, (size_t)n_pixels * sizeof(short), cudaMemcpyHostToDevice));
    LT_CUDA(cudaMemcpy(h->txt_lut, lut, (size_t)n_pixels * sizeof(unsigned short), cudaMemcpyHostToDevice));
    LT_CUDA(cudaMemcpy(h->txt_advance, advance, (size_t)n_chars * sizeof(int), cudaMemcpyHostToDevice));
    h->txt_nchars = n_chars; h->txt_first = first_char;
    // The three text lines (baselines 35 rows apart) may be drawn concurrently iff no glyph of the strings this
    // library formats reaches the rows of the neighbouring line.
    {
        const char* alphabet = "Curve Radius: -0123456789mEccentricity.FrameLaneLineDetectionFailed";
        int lo = 0, hi = 0;
        for (const char* p = alphabet; *p; ++p) {
            int c = *p - first_char;
            if (c < 0 || c >= n_chars) continue;
            for (int i = char_start[c]; i < char_start[c + 1]; ++i) { lo = dy[i] < lo ? dy[i] : lo; hi = dy[i] > hi ? dy[i] : hi; }
        }
        h->txt_parallel_lines = (hi - lo) < 35 ? 1 : 0;
        // frame rows the three text lines (baselines 35, 70, 105: lane_tracker.py:653-659) can touch
        h->txt_row0 = 35 + lo < 0 ? 0 : 35 + lo;
        h->txt_row1 = 105 + hi + 1 > h->d.img_h ? h->d.img_h : 105 + hi + 1;
    }
    {   // ordered glyph pairs that share pixels, and whether a glyph can reach beyond its immediate neighbour
        std::vector<unsigned char> ov((size_t)n_chars * n_chars, 0);
        int min_dx = 0, max_reach = 0, min_adv = 1 << 30;
        std::vector<std::vector<unsigned long long>> bm(n_chars, std::vector<unsigned long long>(64, 0ull));   // dy+32 rows, dx+8 bits
        bool fits = true;
        for (int c = 0; c < n_chars; ++c) {
            min_adv = advance[c] < min_adv ? advance[c] : min_adv;
            for (int i = char_start[c]; i < char_start[c + 1]; ++i) {
                int yy = dy[i] + 32, xx = dx[i] + 8;
                if (yy < 0 || yy >= 64 || xx < 0 || xx >= 64) { fits = false; continue; }
                bm[c][yy] |= 1ull << xx;
                min_dx = dx[i] < min_dx ? dx[i] : min_dx;
                int reach = dx[i] - advance[c];
                max_reach = reach > max_reach ? reach : max_reach;
            }
        }
        for (int a = 0; a < n_chars && fits; ++a)
            for (int b = 0; b < n_chars; ++b)
                for (int i = char_start[b]; i < char_start[b + 1]; ++i) {
                    int yy = dy[i] + 32, xx = dx[i] + advance[a] + 8;
                    if (yy >= 0 && yy < 64 && xx >= 0 && xx < 64 && ((bm[a][yy] >> xx) & 1ull)) { ov[(size_t)a * n_chars + b] = 1; break; }
                }
        const bool neighbours_only = fits && (max_reach - min_dx) < min_adv;
        if (h->txt_pair_overlap) { cudaFree(h->txt_pair_overlap); h->txt_pair_overlap = nullptr; }
        if (h->txt_bitmaps) { cudaFree(h->txt_bitmaps); h->txt_bitmaps = nullptr; }
        if (neighbours_only) {
            if (dev_alloc(&h->txt_pair_overlap, ov.size())) return -2;
            LT_CUDA(cudaMemcpy(h->txt_pair_overlap, ov.data(), ov.size(), cudaMemcpyHostToDevice));
            std::vector<unsigned long long> flat((size_t)n_chars * 64);
            for (int c = 0; c < n_chars; ++c) for (int r = 0; r < 64; ++r) flat[(size_t)c * 64 + r] = bm[c][r];
            if (dev_alloc(&h->txt_bitmaps, flat.size())) return -2;
            LT_CUDA(cudaMemcpy(h->txt_bitmaps, flat.data(), flat.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice));
        }
    }
    return 0;
}

extern "C" int lt_set_remap_mode(lt_handle* h, int32_t mode) {
    if (!h || (mode != 0 && mode != 1)) { lt_set_error("remap mode must be 0 (exact) or 1 (fused single resample)"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    if (mode == 1 && !h->fused_desc) {
        int rc = dev_alloc(&h->fused_desc, (size_t)h->d.bv_w * h->d.bv_h);
        if (rc) return rc;
        if ((rc = lt_launch_build_fused_desc(h, 0))) return rc;
        LT_CUDA(cudaDeviceSynchronize());
    }
    h->remap_mode = mode;
    return 0;
}

extern "C" int lt_memcpy_rows(lt_handle* h, void* dst, const void* src, int32_t n, int32_t row0, int32_t row1,
                              int32_t to_device, void* stream) {
    if (!h || !dst || !src || n < 1 || row0 < 0 || row1 > h->d.img_h || row0 >= row1) { lt_set_error("bad argument"); return -1; }
    const size_t row_bytes = (size_t)h->d.img_w * 3, frame_bytes = row_bytes * h->d.img_h;
    const char* s = (const char*)src + (size_t)row0 * row_bytes;
    char* d = (char*)dst + (size_t)row0 * row_bytes;
    LT_CUDA(cudaMemcpy2DAsync(d, frame_bytes, s, frame_bytes, (size_t)(row1 - row0) * row_bytes, (size_t)n,
                              to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return 0;
}

extern "C" int lt_set_capture(lt_handle* h, int32_t enable) {
    if (!h) { lt_set_error("null handle"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    if (enable && !h->cap_pixels) {
        const size_t S = h->S;
        int rc = 0;
        if (!rc) rc = dev_alloc(&h->cap_pixels, 2 * S * 2 * (size_t)h->pix_cap);
        if (!rc) rc = dev_alloc(&h->cap_counts, 2 * S * 2);
        if (!rc) rc = dev_alloc(&h->cap_cents, 2 * S * 2 * (size_t)LT_MAX_LEVELS);
        if (!rc) rc = dev_alloc(&h->cap_ncents, 2 * S * 2);
        if (rc) return rc;
        cudaMemset(h->cap_counts, 0, 2 * S * 2 * sizeof(int));
        cudaMemset(h->cap_ncents, 0, 2 * S * 2 * sizeof(int));
    }
    h->capture = enable ? 1 : 0;
    return 0;
}

extern "C" int lt_set_pixel_capacity(lt_handle* h, int32_t capacity) {
    if (!h || capacity < 1) { lt_set_error("bad argument"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    if (capacity == h->pix_cap) return 0;
    h->pix_cap = capacity;
    if (h->cap_pixels) {
        cudaFree(h->cap_pixels);
        h->cap_pixels = nullptr;
        int rc = dev_alloc(&h->cap_pixels, 2 * (size_t)h->S * 2 * (size_t)h->pix_cap);
        if (rc) { h->capture = 0; return rc; }
    }
    return 0;
}

extern "C" int lt_read_capture(lt_handle* h, int32_t id, int32_t attempt, int32_t side, uint32_t* h_pixels,
                               int32_t capacity, int32_t* h_count, int32_t* h_centroids, int32_t* h_ncentroids) {
    if (!h || id < 0 || id >= h->S || attempt < 0 || attempt > 1 || side < 0 || side > 1 || !h_count) {
        lt_set_error("bad argument");
        return -1;
    }
    if (!h->cap_pixels) { lt_set_error("capture is not enabled (lt_set_capture)"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    const size_t S = h->S, slot = ((size_t)attempt * S + id) * 2 + side;
    LT_CUDA(cudaMemcpy(h_count, h->cap_counts + slot, sizeof(int), cudaMemcpyDeviceToHost));
    int n = *h_count < h->pix_cap ? *h_count : h->pix_cap;
    if (n > capacity) n = capacity;
    if (h_pixels && n > 0)
        LT_CUDA(cudaMemcpy(h_pixels, h->cap_pixels + slot * (size_t)h->pix_cap, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (h_centroids && h_ncentroids) {
        LT_CUDA(cudaMemcpy(h_ncentroids, h->cap_ncents + slot, sizeof(int), cudaMemcpyDeviceToHost));
        LT_CUDA(cudaMemcpy(h_centroids, h->cap_cents + slot * LT_MAX_LEVELS, LT_MAX_LEVELS * sizeof(int), cudaMemcpyDeviceToHost));
    }
    return 0;
}

// ---------------------------------------------------------------------------
// stage entry points
// ---------------------------------------------------------------------------

extern "C" int lt_remap(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int32_t n, void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_frames) { lt_set_error("null argument"); return -1; }
    if ((rc = check_frame_buffer(d_frames, "d_frames"))) return rc;     // (the bird's-eye output is written byte by byte)
    cudaStream_t st = (cudaStream_t)stream;
    if (h->remap_mode == 1) return lt_launch_warp_fused(h, d_frames, d_bv_rgb, n, st);
    if ((rc = lt_launch_undistort(h, d_frames, n, st))) return rc;
    return lt_launch_warp(h, d_bv_rgb, n, st);
}

extern "C" int lt_nv12_to_rgb(const uint8_t* d_nv12, uint8_t* d_rgb, int32_t n, int32_t width, int32_t height, void* stream) {
    if (!d_nv12 || !d_rgb) { lt_set_error("null argument"); return -1; }
    if (n < 1 || width < 4 || height < 2 || (width & 3) || (height & 1) || (((uintptr_t)d_nv12 | (uintptr_t)d_rgb) & 3)) {
        lt_set_error("lt_nv12_to_rgb: width must be a multiple of 4, height even, buffers 4-byte aligned");
        return -1;
    }
    return lt_launch_nv12_to_rgb(d_nv12, d_rgb, n, width, height, (cudaStream_t)stream);
}

extern "C" int lt_filter_lane_points(lt_handle* h, const uint8_t* d_bv_rgb, uint8_t* d_mask, int32_t n,
                                     int32_t filter_type, int32_t ksize_r, int32_t C_r, int32_t ksize_b, int32_t C_b,
                                     int32_t mask_noise, int32_t ksize_noise, int32_t C_noise, int32_t noise_thresh,
                                     void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_mask) { lt_set_error("null argument"); return -1; }
    lt_params dp;
    lt_default_params(&dp);
    LtAttemptParams p = attempt_from(dp);
    p.filter_type = filter_type; p.ksize_r = ksize_r; p.C_r = C_r; p.ksize_b = ksize_b; p.C_b = C_b;
    p.mask_noise = mask_noise; p.ksize_noise = ksize_noise; p.C_noise = C_noise; p.noise_thresh = noise_thresh;
    if ((rc = check_params(h, p))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (d_bv_rgb) {   // NULL: reuse the planes left by the last lt_remap / lt_process
        if ((rc = lt_launch_planes_from_bv(h, d_bv_rgb, n, st))) return rc;
    }
    if ((rc = lt_launch_filter(h, n, p, nullptr, nullptr, st))) return rc;
    return lt_launch_mask_to_u8(h, h->mask, d_mask, n, st);
}

__global__ void k_detected_from_counts(const int* counts, int n, int* detected) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) detected[s] = (counts[2 * s] > 0 && counts[2 * s + 1] > 0) ? 1 : 0;
}

static int run_search_api(lt_handle* h, const uint8_t* d_mask, int n, const LtAttemptParams& p, int mode,
                          const double* d_coeffs, uint32_t* d_pixels, int cap, int* d_counts, int* d_centroids,
                          int* d_ncentroids, int* d_detected, cudaStream_t st) {
    int rc;
    if (!d_counts || (d_pixels && cap < 1)) { lt_set_error("d_counts is required; capacity must be positive"); return -1; }
    if (d_mask) {   // NULL: search the mask left by the last filter call
        if ((rc = lt_launch_u8_to_mask(h, d_mask, h->mask, n, st))) return rc;
    }
    LtSearchArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.mask = h->mask; sa.mode = mode; sa.coeffs = d_coeffs; sa.pixels = d_pixels; sa.pix_cap = cap;
    sa.pix_counts = d_counts; sa.centroids = d_centroids; sa.ncentroids = d_ncentroids; sa.att = h->att; sa.do_fit = 1;
    if ((rc = lt_launch_search(h, n, p, sa, nullptr, nullptr, st))) return rc;
    if (d_detected) {
        k_detected_from_counts<<<lt_div_up(n, 128), 128, 0, st>>>(d_counts, n, d_detected);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int lt_sliding_window_search(lt_handle* h, const uint8_t* d_mask, int32_t n, int32_t window_width,
                                        int32_t window_height, int32_t search_range, double mu,
                                        int32_t no_success_limit, double start_slice, int32_t ignore_sides,
                                        int32_t ignore_bottom, double partial, uint32_t* d_pixels, int32_t capacity,
                                        int32_t* d_counts, int32_t* d_centroids, int32_t* d_ncentroids,
                                        int32_t* d_detected, void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    lt_params dp;
    lt_default_params(&dp);
    LtAttemptParams p = attempt_from(dp);
    p.window_width = window_width; p.window_height = window_height; p.search_range = search_range; p.mu = mu;
    p.no_success_limit = no_success_limit; p.start_slice = start_slice; p.ignore_sides = ignore_sides;
    p.ignore_bottom = ignore_bottom; p.partial = partial;
    if ((rc = check_params(h, p))) return rc;
    if ((d_centroids == nullptr) != (d_ncentroids == nullptr)) { lt_set_error("centroid outputs come in pairs"); return -1; }
    return run_search_api(h, d_mask, n, p, 1, nullptr, d_pixels, capacity, d_counts, d_centroids, d_ncentroids,
                          d_detected, (cudaStream_t)stream);
}

extern "C" int lt_band_search(lt_handle* h, const uint8_t* d_mask, int32_t n, const double* d_coeffs,
                              int32_t bandwidth, int32_t ignore_bottom, double partial, uint32_t* d_pixels,
                              int32_t capacity, int32_t* d_counts, int32_t* d_detected, void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_coeffs) { lt_set_error("band_search needs the previous fit coefficients"); return -1; }
    lt_params dp;
    lt_default_params(&dp);
    LtAttemptParams p = attempt_from(dp);
    p.bandwidth = bandwidth; p.ignore_bottom = ignore_bottom; p.partial = partial;
    if ((rc = check_params(h, p))) return rc;
    return run_search_api(h, d_mask, n, p, 2, d_coeffs, d_pixels, capacity, d_counts, nullptr, nullptr, d_detected,
                          (cudaStream_t)stream);
}

extern "C" int lt_fit_poly(lt_handle* h, const uint32_t* d_pixels, int32_t capacity, const int32_t* d_counts,
                           int32_t n, double* d_fits, void* stream) {
    int rc;
    if ((rc = check_any_n(h, n))) return rc;
    if (!d_pixels || !d_counts || !d_fits) { lt_set_error("null argument"); return -1; }
    return lt_launch_fit_pixels(h, d_pixels, capacity, d_counts, n, d_fits, (cudaStream_t)stream);
}

extern "C" int lt_check_validity(lt_handle* h, const double* d_fits, int32_t n, int32_t* d_valid, double* d_diffs,
                                 void* stream) {
    int rc;
    if ((rc = check_any_n(h, n))) return rc;
    if (!d_fits || !d_valid) { lt_set_error("null argument"); return -1; }
    return lt_launch_validity(h, d_fits, n, d_valid, d_diffs, (cudaStream_t)stream);
}

extern "C" int lt_get_poly_points(lt_handle* h, const double* d_fits, int32_t n, double partial, int32_t* d_x,
                                  int32_t* d_counts, void* stream) {
    int rc;
    if ((rc = check_any_n(h, n))) return rc;
    if (!d_fits || !d_x || !d_counts) { lt_set_error("null argument"); return -1; }
    if (!(partial >= 0.0 && partial <= 1.0)) { lt_set_error("partial must lie in [0, 1]"); return -1; }
    return lt_launch_poly_points(h, d_fits, n, partial, d_x, d_counts, (cudaStream_t)stream);
}

extern "C" int lt_draw_lane(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n, const int32_t* d_x,
                            const int32_t* d_counts, void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_frames || !d_out || !d_x || !d_counts) { lt_set_error("null argument"); return -1; }
    if ((rc = check_frame_buffer(d_frames, "d_frames")) || (rc = check_frame_buffer(d_out, "d_out"))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // own polygon rows and draw flags: the per-stream ones cache the last valid lane of process() (the polygon a
    // failing frame re-draws, lane_tracker.py:1160-1166) and must survive a stage call
    LT_CUDA(cudaSetDevice(h->cfg.device));
    if (!h->dl_rows) {
        if ((rc = dev_alloc(&h->dl_rows, (size_t)h->S * h->d.bv_h))) return rc;
        if ((rc = dev_alloc(&h->dl_flags, (size_t)h->S))) return rc;
        if ((rc = dev_alloc(&h->dl_bbox, (size_t)h->S))) return rc;
    }
    lt_handle view = *h;
    view.lane_rows = h->dl_rows;
    view.lane_bbox = h->dl_bbox;
    view.draw_flags = h->dl_flags;
    if ((rc = lt_launch_lane_rows(&view, d_x, d_counts, n, st))) return rc;
    return lt_launch_overlay(&view, d_frames, d_out, n, view.draw_flags, nullptr, st);
}

// get_curve_radius / get_eccentricity (lane_tracker.py:530-559) for caller-supplied fits and polylines.
// The metric refit of the same pixels is the analytic rescaling of the pixel-space fit (a' = a*mpph/mppv^2,
// b' = b*mpph/mppv), exactly as k_update_state computes it inside lt_process.
__global__ void k_lane_metrics(const double* __restrict__ fits, const int* __restrict__ xs, const int* __restrict__ counts, int n,
                               int W, int H, double mppv, double mpph, long long* __restrict__ radii, double* __restrict__ ecc) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    for (int side = 0; side < 2; ++side) {
        const double a = fits[(size_t)s * 6 + side * 3], b = fits[(size_t)s * 6 + side * 3 + 1];
        const double am = a * mpph / (mppv * mppv), bm = b * mpph / mppv;
        const double g = 2.0 * am * (double)H * mppv + bm;
        const double r = pow(1.0 + g * g, 1.5) / fabs(2.0 * am);
        radii[s * 2 + side] = (!(r == r) || r >= 9.2233720368547758e18) ? 0x7FFFFFFFFFFFFFFFLL : (long long)r;   // int(float)
    }
    if (ecc) {
        const int nl = counts ? counts[s * 2] : 0, nr = counts ? counts[s * 2 + 1] : 0;
        double e = 0.0;
        if (xs && nl > 0 && nr > 0) {
            const int mid = W / 2, left = xs[(size_t)s * 2 * H + nl - 1], right = xs[(size_t)s * 2 * H + H + nr - 1];
            e = __dmul_rn((double)((mid - left) - (right - mid)) / 2.0, mpph);
        }
        ecc[s] = e;
    }
}

extern "C" int lt_lane_metrics(lt_handle* h, const double* d_fits, const int32_t* d_x, const int32_t* d_counts, int32_t n,
                               int64_t* d_radii, double* d_eccentricity, void* stream) {
    int rc;
    if ((rc = check_any_n(h, n))) return rc;
    if (!d_fits || !d_radii || (d_eccentricity && (!d_x || !d_counts))) { lt_set_error("null argument"); return -1; }
    k_lane_metrics<<<lt_div_up(n, 64), 64, 0, (cudaStream_t)stream>>>(d_fits, d_x, d_counts, n, h->d.bv_w, h->d.bv_h, h->cfg.mppv,
                                                                     h->cfg.mpph, (long long*)d_radii, d_eccentricity);
    LT_LAUNCH_CHECK();
    return 0;
}

// bilateral_adaptive_threshold (lane_tracker.py:14-83) on an arbitrary single-channel image: four zero-padded side sums
// of k neighbours against k*p -/+ C*k.  (filter2D's CV_16S saturation cannot change the sign the reference tests.)
__global__ void __launch_bounds__(256)
k_bilateral_threshold(const uint8_t* __restrict__ img, uint8_t* __restrict__ out, int w, int h, size_t pitch_in, size_t pitch_out,
                      int k, int C, int ceil_mode, int true_value, int false_value) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const uint8_t* row = img + (size_t)y * pitch_in;
    int L = 0, R = 0, U = 0, D = 0;
    for (int i = 1; i <= k; ++i) {
        if (x - i >= 0) L += __ldg(&row[x - i]);
        if (x + i < w) R += __ldg(&row[x + i]);
        if (y - i >= 0) U += __ldg(&img[(size_t)(y - i) * pitch_in + x]);
        if (y + i < h) D += __ldg(&img[(size_t)(y + i) * pitch_in + x]);
    }
    const int kp = k * (int)__ldg(&row[x]), delta = ceil_mode ? -C * k : C * k;
    bool pass;
    if (!ceil_mode) pass = ((L - kp + delta < 0) && (R - kp + delta < 0)) || ((U - kp + delta < 0) && (D - kp + delta < 0));
    else pass = ((L - kp + delta > 0) && (R - kp + delta > 0)) || ((U - kp + delta > 0) && (D - kp + delta > 0));
    out[(size_t)y * pitch_out + x] = (uint8_t)(pass ? true_value : false_value);
}

extern "C" int lt_bilateral_adaptive_threshold(const uint8_t* d_img, int32_t width, int32_t height, int64_t pitch_in, uint8_t* d_out,
                                               int64_t pitch_out, int32_t ksize, int32_t C, int32_t mode, int32_t true_value,
                                               int32_t false_value, void* stream) {
    if (!d_img || !d_out) { lt_set_error("null argument"); return -1; }
    if (width < 1 || height < 1 || pitch_in < width || pitch_out < width || ksize < 1 || ksize > 32767 / 255 * 64) {
        lt_set_error("lt_bilateral_adaptive_threshold: bad geometry or ksize");
        return -1;
    }
    if (mode != 0 && mode != 1) { lt_set_error("Unexpected mode value. Expected value is 'floor' or 'ceil'."); return -1; }
    if (true_value < 0 || true_value > 255 || false_value < 0 || false_value > 255) { lt_set_error("mask values must lie in [0, 255]"); return -1; }
    k_bilateral_threshold<<<dim3(lt_div_up(width, 256), height), 256, 0, (cudaStream_t)stream>>>(
        d_img, d_out, width, height, (size_t)pitch_in, (size_t)pitch_out, ksize, C, mode, true_value, false_value);
    LT_LAUNCH_CHECK();
    return 0;
}

// The putText overlays of draw_lane (kind 0: "Curve Radius: .. m", "Eccentricity: .. m") and print_failure (kind 1:
// "Lane Line Detection Failed"), plus "Frame: n" when the tracker was created with print_frame_count
// (lane_tracker.py:653-659, 668-672), drawn in place on device frames from caller-supplied values.
extern "C" int lt_draw_text(lt_handle* h, uint8_t* d_frames, int32_t n, const int32_t* h_kind, const int64_t* h_radius,
                            const double* h_eccentricity, const int32_t* h_counter, void* stream) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_frames || !h_kind || !h_counter) { lt_set_error("null argument"); return -1; }
    if ((rc = check_frame_buffer(d_frames, "d_frames"))) return rc;
    if (!h->txt_tables) { lt_set_error("no text sprites installed (lt_set_text_sprites)"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    if (!h->txt_state) {
        if ((rc = dev_alloc(&h->txt_state, (size_t)h->S))) return rc;
        if ((rc = dev_alloc(&h->txt_flags, (size_t)h->S))) return rc;
    }
    std::vector<LtDevState> st(n);
    std::vector<int> flags(n);
    for (int i = 0; i < n; ++i) {
        memset(&st[i], 0, sizeof(LtDevState));
        if (h_kind[i] != 0 && h_kind[i] != 1) { lt_set_error("text kind must be 0 (lane) or 1 (failure)"); return -1; }
        flags[i] = h_kind[i] == 0 ? 1 : 0;
        if (h_kind[i] == 0) {
            if (!h_radius || !h_eccentricity) { lt_set_error("lane text needs the radius and the eccentricity"); return -1; }
            st[i].s.average_curve_radius = h_radius[i];
            st[i].s.eccentricity = h_eccentricity[i];
        }
        st[i].s.counter = h_counter[i];
    }
    cudaStream_t s = (cudaStream_t)stream;
    LT_CUDA(cudaMemcpyAsync(h->txt_state, st.data(), (size_t)n * sizeof(LtDevState), cudaMemcpyHostToDevice, s));
    LT_CUDA(cudaMemcpyAsync(h->txt_flags, flags.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    LT_CUDA(cudaStreamSynchronize(s));                 // the staging vectors are pageable host memory
    lt_handle view = *h;
    view.state = h->txt_state;
    view.draw_flags = h->txt_flags;
    return lt_launch_text(&view, d_frames, n, nullptr, s);
}

// ---------------------------------------------------------------------------
// state and debug access (synchronous)
// ---------------------------------------------------------------------------

// ---------------------------------------------------------------------------
// debug views
// ---------------------------------------------------------------------------

extern "C" int lt_warp_frame(lt_handle* h, const uint8_t* d_frames, int32_t n, uint8_t* d_bv_rgb, void* stream) {
    if (!h || !d_frames || !d_bv_rgb) { lt_set_error("null argument"); return -1; }
    int rc;
    if ((rc = check_frame_buffer(d_frames, "d_frames"))) return rc;
    LT_CUDA(cudaSetDevice(h->cfg.device));
    if ((rc = check_any_n(h, n))) return rc;
    return lt_launch_warp_frame(h, d_frames, d_bv_rgb, n, (cudaStream_t)stream);
}

extern "C" int lt_visualize_search(lt_handle* h, const lt_vis* v, const uint8_t* d_mask, const uint32_t* d_left,
                                   const uint32_t* d_right, const int32_t* h_rects, uint8_t* d_vis, void* stream) {
    if (!h || !v || !d_mask || !d_vis) { lt_set_error("null argument"); return -1; }
    if (v->mode != 0 && v->mode != 1) { lt_set_error("lt_vis.mode must be 0 (sliding window) or 1 (band)"); return -1; }
    if (v->n_left < 0 || v->n_right < 0 || (v->n_left && !d_left) || (v->n_right && !d_right)) { lt_set_error("bad pixel lists"); return -1; }
    if (v->n_rects < 0 || v->n_rects > 2 * LT_MAX_LEVELS || (v->n_rects && !h_rects)) { lt_set_error("n_rects outside [0, %d]", 2 * LT_MAX_LEVELS); return -1; }
    if (v->mode == 1 && !(v->partial >= 0.0 && v->partial <= 1.0)) { lt_set_error("partial must lie in [0, 1]"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const LtDims& d = h->d;
    const int W = d.bv_w, H = d.bv_h;
    // work area: rects | fits [2][2][3] | xs [2 calls][2][H] | counts [2][2] | rows [2][H]
    const size_t o_fits = (size_t)5 * 2 * LT_MAX_LEVELS * sizeof(int), o_xs = o_fits + 12 * sizeof(double),
                 o_cnt = o_xs + (size_t)4 * H * sizeof(int), o_rows = o_cnt + 4 * sizeof(int),
                 total = o_rows + (size_t)2 * H * sizeof(int2);
    if (!h->vis_scratch) LT_CUDA(cudaMalloc((void**)&h->vis_scratch, total));
    int* d_rects = reinterpret_cast<int*>(h->vis_scratch);
    double* d_fits = reinterpret_cast<double*>(h->vis_scratch + o_fits);
    int* d_xs = reinterpret_cast<int*>(h->vis_scratch + o_xs);
    int* d_cnt = reinterpret_cast<int*>(h->vis_scratch + o_cnt);
    int2* d_rows = reinterpret_cast<int2*>(h->vis_scratch + o_rows);
    double fits[12];
    for (int j = 0; j < 3; ++j) {
        fits[j] = v->left_fit[j]; fits[3 + j] = v->right_fit[j];
        fits[6 + j] = v->band_left[j]; fits[9 + j] = v->band_right[j];
    }
    LT_CUDA(cudaMemcpyAsync(d_fits, fits, sizeof(fits), cudaMemcpyHostToDevice, st));
    const int nrect = v->mode == 0 ? v->n_rects : 0;
    if (nrect) LT_CUDA(cudaMemcpyAsync(d_rects, h_rects, (size_t)nrect * 5 * sizeof(int), cudaMemcpyHostToDevice, st));
    LT_CUDA(cudaStreamSynchronize(st));                       // fits / rects came from pageable host memory
    const uint32_t RED = 255u, BLUE = 255u << 16, YELLOW = 255u | (235u << 8);
    int rc;
    if ((rc = lt_launch_vis_base(d_mask, d_rects, nrect, W, H, d_vis, st))) return rc;
    // later writes win: left pixels, then right pixels (lane_tracker.py:720-721 / :745-746)
    if ((rc = lt_launch_vis_scatter(d_left, v->n_left, W, H, RED, d_vis, st))) return rc;
    if ((rc = lt_launch_vis_scatter(d_right, v->n_right, W, H, BLUE, d_vis, st))) return rc;
    if (v->mode == 1) {
        if ((rc = lt_launch_poly_points(h, d_fits + 6, 1, v->partial, d_xs + 2 * H, d_cnt + 2, st))) return rc;
        if ((rc = lt_launch_band_rows(h, d_xs + 2 * H, d_cnt + 2, v->bandwidth, d_rows, d_rows + H, st))) return rc;
        if ((rc = lt_launch_vis_band_blend(d_rows, d_rows + H, W, H, d_vis, st))) return rc;
    }
    if ((rc = lt_launch_poly_points(h, d_fits, 1, 1.0, d_xs, d_cnt, st))) return rc;
    if ((rc = lt_launch_vis_scatter_poly(d_xs, d_cnt, W, H, YELLOW, d_vis, st))) return rc;
    if ((rc = lt_launch_vis_scatter_poly(d_xs + H, d_cnt + 1, W, H, YELLOW, d_vis, st))) return rc;
    return 0;
}

extern "C" int lt_resize_linear(const uint8_t* d_src, int32_t sw, int32_t sh, int32_t cn, int64_t src_pitch, uint8_t* d_dst,
                                int32_t dw, int32_t dh, int64_t dst_pitch, void* stream) {
    if (!d_src || !d_dst) { lt_set_error("null argument"); return -1; }
    if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || (cn != 1 && cn != 3) || src_pitch < (int64_t)sw * cn || dst_pitch < (int64_t)dw * cn) {
        lt_set_error("lt_resize_linear: sizes must be positive, channels 1 or 3, pitches >= row bytes");
        return -1;
    }
    return lt_launch_resize_linear(d_src, sw, sh, cn, (size_t)src_pitch, d_dst, dw, dh, (size_t)dst_pitch, (cudaStream_t)stream);
}

extern "C" int lt_get_state(lt_handle* h, int32_t id, lt_state* hs, int32_t* h_lx, int32_t* h_rx) {
    if (!h || !hs || id < 0 || id >= h->S) { lt_set_error("bad argument"); return -1; }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    LT_CUDA(cudaMemcpy(hs, &h->state[id].s, sizeof(lt_state), cudaMemcpyDeviceToHost));
    size_t H = h->d.bv_h;
    if (h_lx) LT_CUDA(cudaMemcpy(h_lx, h->avg_x + (size_t)id * 2 * H, H * sizeof(int), cudaMemcpyDeviceToHost));
    if (h_rx) LT_CUDA(cudaMemcpy(h_rx, h->avg_x + (size_t)id * 2 * H + H, H * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int lt_set_state(lt_handle* h, int32_t id, const lt_state* hs, const int32_t* h_lx, const int32_t* h_rx) {
    if (!h || !hs || id < 0 || id >= h->S) { lt_set_error("bad argument"); return -1; }
    if (hs->ring_len < 0 || hs->ring_len > LT_MAX_AVERAGE || hs->radii_len < 0 || hs->radii_len > LT_MAX_AVERAGE ||
        hs->n_left_avg < 0 || hs->n_left_avg > h->d.bv_h || hs->n_right_avg < 0 || hs->n_right_avg > h->d.bv_h) {
        lt_set_error("inconsistent lt_state");
        return -1;
    }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());
    LT_CUDA(cudaMemcpy(&h->state[id].s, hs, sizeof(lt_state), cudaMemcpyHostToDevice));
    size_t H = h->d.bv_h;
    if (h_lx) LT_CUDA(cudaMemcpy(h->avg_x + (size_t)id * 2 * H, h_lx, H * sizeof(int), cudaMemcpyHostToDevice));
    if (h_rx) LT_CUDA(cudaMemcpy(h->avg_x + (size_t)id * 2 * H + H, h_rx, H * sizeof(int), cudaMemcpyHostToDevice));
    if (hs->has_avg && h_lx && h_rx) {
        // rebuild the cached polygon rows of this stream
        int counts[2] = {hs->n_left_avg, hs->n_right_avg};
        int* d_counts = nullptr;
        LT_CUDA(cudaMalloc((void**)&d_counts, 2 * sizeof(int)));
        cudaMemcpy(d_counts, counts, sizeof(counts), cudaMemcpyHostToDevice);
        // lt_launch_lane_rows works on slot 0..n-1; shift the base pointers to this stream
        lt_handle tmp = *h;
        tmp.lane_rows = h->lane_rows + (size_t)id * H;
        tmp.lane_bbox = h->lane_bbox + id;
        tmp.draw_flags = h->draw_flags + id;
        int rc = lt_launch_lane_rows(&tmp, h->avg_x + (size_t)id * 2 * H, d_counts, 1, 0);
        cudaDeviceSynchronize();
        cudaFree(d_counts);
        if (rc) return rc;
    }
    return 0;
}

extern "C" int64_t lt_debug_read(lt_handle* h, int32_t what, int32_t id, void* dst, int64_t cap) {
    if (!h || !dst || id < 0 || id >= h->S) { lt_set_error("bad argument"); return -1; }
    if (cudaSetDevice(h->cfg.device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
        lt_set_error("device error: %s", cudaGetErrorString(cudaGetLastError()));
        return -2;
    }
    const LtDims& d = h->d;
    const size_t npx = (size_t)d.img_w * d.img_h, nbv = (size_t)d.bv_w * d.bv_h;
    const void* src = nullptr;
    size_t bytes = 0;
    uint8_t* tmp = nullptr;
    int rc = 0;
    switch (what) {
        case 0: src = h->und_map; bytes = npx * sizeof(int2); break;
        case 1: src = h->bv_map; bytes = nbv * sizeof(int2); break;
        case 2: src = h->ov_map; bytes = npx * sizeof(int2); break;
        case 3: case 4: case 5: case 6: case 7: case 8: {
            bytes = nbv;
            if (cudaMalloc((void**)&tmp, nbv) != cudaSuccess) { lt_set_error("cudaMalloc failed"); return -2; }
            lt_handle one = *h;     // view of this stream as slot 0
            if (what <= 6) {
                const uint32_t* pl = what == 3 ? h->planeR : what == 4 ? h->planeB : what == 5 ? h->topR : h->topB;
                rc = lt_launch_plane_to_u8(&one, pl + (size_t)id * h->stream_pad, d.pp, tmp, 1, 0);
            } else {
                const uint32_t* bits = what == 7 ? h->mask : h->merged;
                rc = lt_launch_mask_to_u8(&one, bits + (size_t)id * h->stream_mask, tmp, 1, 0);
            }
            src = tmp;
            break;
        }
        case 9: src = h->lane_rows + (size_t)id * d.bv_h; bytes = (size_t)d.bv_h * sizeof(int2); break;
        case 12:    // polygon rows of the last lt_draw_lane stage call (its own scratch, not the per-stream cache)
            if (!h->dl_rows) { lt_set_error("lt_draw_lane has not been called"); return -1; }
            src = h->dl_rows + (size_t)id * d.bv_h; bytes = (size_t)d.bv_h * sizeof(int2); break;
        case 10: {
            int v[9] = {d.roi0, d.roi1, d.ov0, d.ov1, d.p2, d.mwords, h->pix_cap, h->src0, h->src1};
            if (cap < (int64_t)sizeof(v)) { lt_set_error("buffer too small"); return -1; }
            memcpy(dst, v, sizeof(v));
            return sizeof(v);
        }
        case 11: {   // launch geometry of the last paired morphology launch: bands of the 55x55 / 29x29 jobs, SM count
            int v[3] = {h->bands_val[0], h->bands_val[1], h->sm_count};
            if (cap < (int64_t)sizeof(v)) { lt_set_error("buffer too small"); return -1; }
            memcpy(dst, v, sizeof(v));
            return sizeof(v);
        }
        default: lt_set_error("unknown debug buffer %d", what); return -1;
    }
    if (rc) { if (tmp) cudaFree(tmp); return rc; }
    if ((int64_t)bytes > cap) { if (tmp) cudaFree(tmp); lt_set_error("buffer too small: need %zu bytes", bytes); return -1; }
    cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) { lt_set_error("copy failed: %s", cudaGetErrorString(e)); return -2; }
    return (int64_t)bytes;
}
