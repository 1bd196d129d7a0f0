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

// The filter options alone: lt_filter_lane_points takes no search options, so a view narrower or shorter than the
// default search windows must not refuse it.
static int check_filter_params(const LtAttemptParams& a) {
    if (a.filter_type != 0 && a.filter_type != 1) {
        lt_set_error("Unexpected filter mode. Expected modes are 'bilateral' or 'neighborhood'.");
        return -1;
    }
    if (a.ksize_r < 1 || a.ksize_b < 1 || a.ksize_r > 255 || a.ksize_b > 255 || a.ksize_noise < 1 || a.ksize_noise > 255) {
        lt_set_error("threshold kernel sizes must lie in [1, 255]");
        return -1;
    }
    if (a.filter_type == 1 && ((a.ksize_r & 1) == 0 || (a.ksize_b & 1) == 0 || a.ksize_r < 3 || a.ksize_b < 3)) {
        lt_set_error("'neighborhood' block sizes must be odd and >= 3 (cv2.adaptiveThreshold)");
        return -1;
    }
    return 0;
}

static int check_params(const lt_handle* h, const LtAttemptParams& a) {
    int rc;
    if ((rc = check_filter_params(a))) return rc;
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

static int check_params(const lt_handle* h, const LtAttemptParams& a);

extern "C" int lt_set_profile(lt_handle* h, int32_t profile, const lt_params* params, const lt_validity* validity) {
    if (!h) { lt_set_error("null handle"); return -1; }
    if (profile < 0 || profile >= LT_MAX_PROFILES) {
        lt_set_error("profile %d outside [0, %d)", profile, LT_MAX_PROFILES);
        return -1;
    }
    if (!params) { lt_set_error("null params"); return -1; }
    LtProfile q;
    memset(&q, 0, sizeof(q));
    q.p = attempt_from(*params);
    int rc;
    if ((rc = check_params(h, q.p))) return rc;
    q.val = validity ? *validity : SHIPPED_VALIDITY;
    q.n_tries = params->n_tries;
    h->profiles[profile] = q;
    h->profiles_set |= 1u << profile;
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
                      f.merged, f.mask, f.group_pos, f.pos_profile, f.profiles, f.und_cam, f.slot_pos, f.chunk_cam,
                      f.pos_cam, f.cams};
        for (void* p : fp) if (p) cudaFree(p);
        delete[] f.h_pos_profile;
        delete[] f.h_pos_cam;
    }
    for (int k = 1; k < LT_MAX_CAMERAS; ++k) {     // camera 0's tables are the handle's own, freed below
        const LtCamera& c = h->cams[k];
        void* cp[] = {c.und_map, c.bv_map, c.ov_map, c.und_desc, c.bv_desc};
        for (void* p : cp) if (p) cudaFree(p);
    }
    void* ptrs[] = {h->und_map, h->bv_map, h->ov_map, h->bv_desc, h->und_desc, h->lab_yz, h->fused_desc, h->lab_gamma, h->lab_cbrt, h->lane_rows, h->lane_bbox, h->dl_bbox,
                    h->avg_x, h->state, h->init, h->att, h->retry_list, h->retry_count, h->draw_flags, h->stream_ids, h->seq_pos,
                    h->seq_rows, h->seq_bbox, h->seq_state, h->vis_scratch,
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

// (re)allocate the camera undistort buffer of a front set at the handle's stride and capacity, zeroed: its row 0 and
// column 0 are the zero border of the und layout and are never written
static int alloc_und_cam(lt_handle* h, LtFrontSet& f) {
    if (f.und_cam) cudaFree(f.und_cam);
    f.und_cam = nullptr;
    const size_t words = (size_t)(h->und_cam_slots / LT_UND_GROUP) * lt_und_cam_group_words(h);
    int rc = dev_alloc(&f.und_cam, words);
    if (!rc) LT_CUDA(cudaMemset(f.und_cam, 0, words * sizeof(uint32_t)));
    return rc;
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
    if (!rc) rc = dev_alloc(&f.group_pos, S);
    if (!rc) rc = dev_alloc(&f.pos_profile, S);
    if (!rc) rc = dev_alloc(&f.profiles, LT_MAX_PROFILES);
    if (!rc) f.h_pos_profile = new int[S];
    // camera batches: at most S + 3 S slots (a run of one camera pads to a multiple of four)
    if (!rc) rc = dev_alloc(&f.slot_pos, 4 * S);
    if (!rc) rc = dev_alloc(&f.chunk_cam, S);
    if (!rc) rc = dev_alloc(&f.pos_cam, S);
    if (!rc) rc = dev_alloc(&f.cams, LT_MAX_CAMERAS);
    if (!rc) f.h_pos_cam = new int[S];
    if (!rc && h->und_cam_slots) rc = alloc_und_cam(h, f);
    return rc;
}

// make set k the one the launchers see (kernel arguments are captured at launch, so switching between calls is safe)
static void select_set(lt_handle* h, int k) {
    const LtFrontSet& f = h->fs[k];
    const size_t origin = (size_t)LT_HALO_Y * h->d.pp + LT_HALO_X;
    h->und_roi = f.und_roi;
    h->planeR = f.pad_alloc[0] + origin; h->planeB = f.pad_alloc[1] + origin;
    h->tmpR = f.pad_alloc[2] + origin;   h->tmpB = f.pad_alloc[3] + origin;
    h->topR = f.pad_alloc[4] + origin;   h->topB = f.pad_alloc[5] + origin;
    h->merged = f.merged; h->mask = f.mask;
}

// The rows of a calibration, from its maps: rows of the undistorted frame that the bird's-eye view can touch (the ROI),
// frame rows the undistort of the ROI reads (for partial host->device transfers), frame rows the overlay can touch.
static int camera_rows(const lt_handle* h, LtCamera& c) {
    const LtDims& d = h->d;
    const size_t npx = (size_t)d.img_w * d.img_h, nbv = (size_t)d.bv_w * d.bv_h;
    std::vector<int2> m(nbv);
    cudaError_t e = cudaMemcpy(m.data(), c.bv_map, nbv * sizeof(int2), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { lt_set_error("map build failed: %s", cudaGetErrorString(e)); return -2; }
    int r0 = d.img_h, r1 = 0;
    for (size_t i = 0; i < nbv; ++i) {
        int sx = m[i].x >> 5, sy = m[i].y >> 5;
        if (sx + 1 < 0 || sx >= d.img_w) continue;
        for (int yy = sy; yy <= sy + 1; ++yy)
            if (yy >= 0 && yy < d.img_h) { r0 = yy < r0 ? yy : r0; r1 = yy + 1 > r1 ? yy + 1 : r1; }
    }
    if (r0 >= r1) { r0 = 0; r1 = 1; }
    c.roi0 = r0; c.roi1 = r1;
    {   // frame rows read by the undistort of the ROI rows (for partial host->device transfers)
        std::vector<int2> u((size_t)(r1 - r0) * d.img_w);
        cudaMemcpy(u.data(), c.und_map + (size_t)r0 * d.img_w, u.size() * sizeof(int2), cudaMemcpyDeviceToHost);
        int s0 = d.img_h, s1 = 0;
        for (size_t i = 0; i < u.size(); ++i) {
            int sy = u[i].y >> 5;
            for (int yy = sy; yy <= sy + 1; ++yy)
                if (yy >= 0 && yy < d.img_h) { s0 = yy < s0 ? yy : s0; s1 = yy + 1 > s1 ? yy + 1 : s1; }
        }
        if (s0 >= s1) { s0 = 0; s1 = d.img_h; }
        c.src0 = s0; c.src1 = s1;
    }
    std::vector<int2> o(npx);
    cudaMemcpy(o.data(), c.ov_map, npx * sizeof(int2), cudaMemcpyDeviceToHost);
    int o0 = d.img_h, o1 = 0;
    for (int y = 0; y < d.img_h; ++y)
        for (int x = 0; x < d.img_w; ++x) {
            int2 q = o[(size_t)y * d.img_w + x];
            int sx = q.x >> 5, sy = q.y >> 5;
            if (sx + 1 >= 0 && sx < d.bv_w && sy + 1 >= 0 && sy < d.bv_h) { o0 = y < o0 ? y : o0; o1 = y + 1 > o1 ? y + 1 : o1; }
        }
    if (o0 >= o1) { o0 = 0; o1 = 0; }
    c.ov0 = o0; c.ov1 = o1;
    return 0;
}

// The tables of calibration c.cal on the device (synchronous): maps, rows, then the tap descriptors of its ROI.
// On failure, what was allocated is left in c for the caller to free.
static int build_camera(lt_handle* h, LtCamera& c) {
    const size_t npx = (size_t)h->d.img_w * h->d.img_h, nbv = (size_t)h->d.bv_w * h->d.bv_h;
    int rc = 0;
    if (!rc) rc = dev_alloc(&c.und_map, npx);
    if (!rc) rc = dev_alloc(&c.bv_map, nbv);
    if (!rc) rc = dev_alloc(&c.ov_map, npx);
    if (!rc) rc = lt_launch_build_maps(c.cal, h->d, c.und_map, c.bv_map, c.ov_map, 0);
    if (!rc) rc = camera_rows(h, c);
    if (rc) return rc;
    LtDims d = h->d;
    d.roi0 = c.roi0; d.roi1 = c.roi1; d.ov0 = c.ov0; d.ov1 = c.ov1;
    if (!rc) rc = dev_alloc(&c.bv_desc, nbv);
    if (!rc) rc = lt_launch_build_desc(c.bv_map, c.bv_desc, d, 0);
    if (!rc) rc = dev_alloc(&c.und_desc, (size_t)(d.roi1 - d.roi0) * d.img_w);
    if (!rc) rc = lt_launch_build_und_desc(c.und_map, c.und_desc, d, 0);
    return rc;
}

extern "C" int lt_create(const lt_config* cfg, lt_handle** out) {
    if (!cfg || !out) { lt_set_error("null argument"); return -1; }
    // bv_w >= 66: pair planes at least 2 * LT_HALO_X wide, so that every packed column feeds at most one of the two
    // seam halos the erosion epilogue of the morphology writes
    if (cfg->img_w < 64 || cfg->img_h < 16 || cfg->bv_w < 66 || cfg->bv_h < 16 || (cfg->img_w & 3) || (cfg->bv_w & 1) ||
        cfg->bv_h > 65535 || cfg->bv_w > 32767 || cfg->img_w > 32767 || cfg->img_h > 32767) {
        lt_set_error("unsupported geometry: img %dx%d (width must be a multiple of 4), warped %dx%d (width must be even and "
                     "at least 66)", cfg->img_w, cfg->img_h, cfg->bv_w, cfg->bv_h);
        return -1;
    }
    if (cfg->max_streams < 1 || cfg->n_average < 1 || cfg->n_average > LT_MAX_AVERAGE) {
        lt_set_error("max_streams must be >= 1 and n_average in [1, %d]", LT_MAX_AVERAGE);
        return -1;
    }
    LT_CUDA(cudaSetDevice(cfg->device));
    {
        // a view so wide that a threshold kernel could not launch would fail in the middle of a batch: refuse it here
        int optin = 0;
        LT_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device));
        if (lt_filter_smem_bytes(cfg->bv_w) > (size_t)optin) {
            int widest = 66;
            while (lt_filter_smem_bytes(widest + 2) <= (size_t)optin) widest += 2;
            lt_set_error("unsupported geometry: img %dx%d (width must be a multiple of 4), warped %dx%d (width must be "
                         "even and at most %d on this device)", cfg->img_w, cfg->img_h, cfg->bv_w, cfg->bv_h, widest);
            return -1;
        }
    }
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
    A(lab_gamma, 256); A(lab_cbrt, 3072);
    if (rc) { lt_destroy(h); return rc; }
    LtCamera& c0 = h->cams[0];
    memcpy(c0.cal.cam_matrix, cfg->cam_matrix, sizeof(c0.cal.cam_matrix));
    memcpy(c0.cal.dist_coeffs, cfg->dist_coeffs, sizeof(c0.cal.dist_coeffs));
    memcpy(c0.cal.M, cfg->M, sizeof(c0.cal.M));
    memcpy(c0.cal.Minv, cfg->Minv, sizeof(c0.cal.Minv));
    c0.cal.mppv = cfg->mppv; c0.cal.mpph = cfg->mpph;
    rc = build_camera(h, c0);
    h->und_map = c0.und_map; h->bv_map = c0.bv_map; h->ov_map = c0.ov_map; h->und_desc = c0.und_desc; h->bv_desc = c0.bv_desc;
    if (rc) { lt_destroy(h); return rc; }
    d.roi0 = c0.roi0; d.roi1 = c0.roi1; d.ov0 = c0.ov0; d.ov1 = c0.ov1;
    h->src0 = c0.src0; h->src1 = c0.src1;
    cudaStream_t st = 0;
    cudaMemcpy(h->lab_gamma, LT_LAB_GAMMA, sizeof(LT_LAB_GAMMA), cudaMemcpyHostToDevice);
    cudaMemcpy(h->lab_cbrt, LT_LAB_CBRT, sizeof(LT_LAB_CBRT), cudaMemcpyHostToDevice);
    A(lab_yz, 768);
    if (!rc) rc = lt_launch_build_lab_yz(h, st);
    if (!rc) rc = alloc_front_set(h, 0);
    if (!rc) select_set(h, 0);
    A(lane_rows, S * (size_t)d.bv_h); A(lane_bbox, S); A(avg_x, S * 2 * (size_t)d.bv_h);
    A(state, S); A(init, 1); A(att, 2 * S); A(retry_list, S); A(retry_count, 1); A(draw_flags, 2 * S); A(stream_ids, S);
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
    {
        LtDevState z;
        init_state(h, &z.s);
        if (cudaMemcpy(h->init, &z, sizeof(z), cudaMemcpyHostToDevice) != cudaSuccess) {
            lt_set_error("cannot write the initial state"); lt_destroy(h); return -2;
        }
    }
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

extern "C" int lt_set_camera(lt_handle* h, int32_t camera, const lt_camera* cam) {
    if (!h) { lt_set_error("null handle"); return -1; }
    if (camera == 0) { lt_set_error("camera 0 is the calibration given to lt_create and cannot be changed"); return -1; }
    if (camera < 1 || camera >= LT_MAX_CAMERAS) { lt_set_error("camera %d outside [1, %d)", camera, LT_MAX_CAMERAS); return -1; }
    if (!cam) { lt_set_error("null camera"); return -1; }
    for (int k = 0; k < 2; ++k)
        if (h->fs[k].cam_pending) {
            lt_set_error("buffer set %d holds the front half of a camera batch whose back half has not been enqueued: "
                         "enqueue it before lt_set_camera", k);
            return -1;
        }
    LT_CUDA(cudaSetDevice(h->cfg.device));
    LT_CUDA(cudaDeviceSynchronize());        // no work in flight reads the tables replaced below
    LtCamera c;
    memset(&c, 0, sizeof(c));
    c.cal = *cam;
    int rc = build_camera(h, c);
    if (!rc && cudaDeviceSynchronize() != cudaSuccess) {
        lt_set_error("camera tables: %s", cudaGetErrorString(cudaGetLastError()));
        rc = -2;
    }
    LtCamera& old = rc ? c : h->cams[camera];      // on failure the camera keeps its previous tables
    void* cp[] = {old.und_map, old.bv_map, old.ov_map, old.und_desc, old.bv_desc};
    for (void* p : cp) if (p) cudaFree(p);
    if (rc) return rc;
    h->cams[camera] = c;
    // the camera undistort buffer: the stride of the tallest ROI, S + 3 min(S, cameras) slots in groups of 16
    int rows = 0, ncams = 0;
    for (int k = 0; k < LT_MAX_CAMERAS; ++k)
        if (h->cams[k].und_map) {
            ++ncams;
            rows = h->cams[k].roi1 - h->cams[k].roi0 > rows ? h->cams[k].roi1 - h->cams[k].roi0 : rows;
        }
    const int slots = (h->S + 3 * (h->S < ncams ? h->S : ncams) + LT_UND_GROUP - 1) / LT_UND_GROUP * LT_UND_GROUP;
    if (rows > h->und_cam_rows || slots > h->und_cam_slots) {
        h->und_cam_rows = rows > h->und_cam_rows ? rows : h->und_cam_rows;
        h->und_cam_slots = slots > h->und_cam_slots ? slots : h->und_cam_slots;
        for (int k = 0; k < 2; ++k)
            if (h->fs[k].mask && (rc = alloc_und_cam(h, h->fs[k]))) return rc;
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

// The undistort and warp of a camera batch: nslots slots of f.und_cam, max_rows the tallest ROI of its cameras.
struct LtCamBatch {
    const LtFrontSet* f;
    int nslots, max_rows;
};

// find_lane_points (lane_tracker.py:795-874) of the first attempt up to the binary mask, all streams: stateless.
// The filter groups g[0..ng) cover the batch (one group {p1, NULL, n} without profiles).  cb: a camera batch (NULL:
// every position uses camera 0).
static int process_front(lt_handle* h, const uint8_t* d_frames, int n, const LtFilterGroup* g, int ng, cudaStream_t st,
                         const LtCamBatch* cb) {
    int rc;
    if (h->prof_active && h->prof_calls >= h->prof_max_calls) h->prof_active = 0;
    lt_prof_mark(h, ST_BEGIN, st);
    if (cb) {
        if ((rc = lt_launch_undistort_cams(h, *cb->f, d_frames, cb->nslots, cb->max_rows, st))) return rc;
        lt_prof_mark(h, ST_UNDISTORT, st);
        if ((rc = lt_launch_warp_cams(h, *cb->f, cb->nslots, st))) return rc;
    } else if (h->remap_mode == 1) {
        if ((rc = lt_launch_warp_fused(h, d_frames, nullptr, n, st))) return rc;
    } else {
        if ((rc = lt_launch_undistort(h, d_frames, n, st))) return rc;
        lt_prof_mark(h, ST_UNDISTORT, st);
        if ((rc = lt_launch_warp(h, nullptr, n, st))) return rc;
    }
    lt_prof_mark(h, ST_WARP, st);
    return lt_launch_filter_groups(h, n, g, ng, nullptr, st);
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

// Writes the host ints h_src[0..n) to the device array dst on stream st, as kernel arguments.
static int upload_ints(const int32_t* h_src, int n, int* dst, cudaStream_t st) {
    LtIdsChunk c;
    for (int off = 0; off < n; off += LT_IDS_CHUNK) {
        c.offset = off;
        c.count = n - off < LT_IDS_CHUNK ? n - off : LT_IDS_CHUNK;
        memcpy(c.ids, h_src + off, (size_t)c.count * sizeof(int32_t));
        k_set_stream_ids<<<1, 256, 0, st>>>(c, dst);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

// Writes h_ids to the handle's one device id array on the stream of the back half that reads it.  One array per
// handle is enough: every kernel that reads it is a back-half kernel enqueued on that same stream after this write,
// and the back half of batch k must follow the back half of batch k-1 (lt_process_back), so a write for batch k
// cannot overtake a read of batch k-1, and no later write can overtake a read of batch k.
static int upload_stream_ids(lt_handle* h, const int32_t* h_ids, int n, cudaStream_t st) {
    return upload_ints(h_ids, n, h->stream_ids, st);
}

struct LtProfileTable {
    LtProfile e[LT_MAX_PROFILES];
};

__global__ void k_set_profiles(LtProfileTable t, LtProfile* __restrict__ dst) {
    if (threadIdx.x < LT_MAX_PROFILES) dst[threadIdx.x] = t.e[threadIdx.x];
}

static bool same_filter(const LtAttemptParams& a, const LtAttemptParams& b) {
    if (a.filter_type != b.filter_type || a.ksize_r != b.ksize_r || a.C_r != b.C_r || a.ksize_b != b.ksize_b ||
        a.C_b != b.C_b || a.mask_noise != b.mask_noise)
        return false;
    return !a.mask_noise || (a.noise_thresh == b.noise_thresh && a.ksize_noise == b.ksize_noise && a.C_noise == b.C_noise);
}

// Front half with profiles: snapshot the profile table and the batch's profile indices into buffer set `set` (on the
// front stream: the back half of this batch runs after it, the front half of batch k+2 after that back half), group
// the positions by filter configuration, and run the front half over the groups.
static int process_front_profiles(lt_handle* h, const uint8_t* d_frames, const int32_t* h_prof, int n, int set,
                                  cudaStream_t st, const LtCamBatch* cb) {
    LtFrontSet& f = h->fs[set];
    LtProfileTable t;
    memcpy(t.e, h->profiles, sizeof(t.e));
    int rc;
    if ((rc = upload_ints(h_prof, n, f.pos_profile, st))) return rc;
    k_set_profiles<<<1, 32, 0, st>>>(t, f.profiles);
    LT_LAUNCH_CHECK();
    memcpy(f.snap, h->profiles, sizeof(f.snap));
    memcpy(f.h_pos_profile, h_prof, (size_t)n * sizeof(int32_t));
    f.snap_n = n;
    // one representative profile per filter configuration, bilateral configurations first
    int rep[LT_MAX_PROFILES], nrep = 0, group_of[LT_MAX_PROFILES];
    for (int pass = 0; pass < 2; ++pass)
        for (int k = 0; k < LT_MAX_PROFILES; ++k) {
            if (!((h->profiles_set >> k) & 1u) || (h->profiles[k].p.filter_type == 0) != (pass == 0)) continue;
            bool used = false;
            for (int i = 0; i < n && !used; ++i) used = h_prof[i] == k;
            if (!used) continue;
            int r = 0;
            while (r < nrep && !same_filter(h->profiles[rep[r]].p, h->profiles[k].p)) ++r;
            if (r == nrep) rep[nrep++] = k;
            group_of[k] = r;
        }
    LtFilterGroup g[LT_MAX_PROFILES];
    if (nrep == 1) {
        g[0] = {h->profiles[rep[0]].p, nullptr, n};
    } else {
        std::vector<int> pos;
        pos.reserve(n);
        for (int r = 0; r < nrep; ++r) {
            const size_t first = pos.size();
            for (int i = 0; i < n; ++i) if (group_of[h_prof[i]] == r) pos.push_back(i);
            g[r] = {h->profiles[rep[r]].p, f.group_pos + first, (int)(pos.size() - first)};
        }
        if ((rc = upload_ints(pos.data(), n, f.group_pos, st))) return rc;
    }
    return process_front(h, d_frames, n, g, nrep, st, cb);
}

struct LtCamTable {
    LtCamDev e[LT_MAX_CAMERAS];
};

__global__ void k_set_cameras(LtCamTable t, LtCamDev* __restrict__ dst) {
    if (threadIdx.x < LT_MAX_CAMERAS) dst[threadIdx.x] = t.e[threadIdx.x];
}

// Front half with cameras, first step: record the batch's cameras in buffer set `set`.  A batch on camera 0 alone
// leaves it at that (it runs the launches without cameras).  Otherwise the slots of und_cam are laid out -- positions
// stably sorted by camera, each camera's run padded to whole chunks of four slots -- and the slot positions, chunk
// cameras, position cameras and the camera snapshot are uploaded on the front stream (kernel arguments, as the
// profiles: the back half of this batch runs after them, the front half of batch k+2 after that back half).
static int prepare_cameras(lt_handle* h, const int32_t* h_cams, int n, int set, cudaStream_t st, LtCamBatch* cb) {
    LtFrontSet& f = h->fs[set];
    memcpy(f.h_pos_cam, h_cams, (size_t)n * sizeof(int32_t));
    f.cam_n = n;
    int count[LT_MAX_CAMERAS] = {0};
    for (int i = 0; i < n; ++i) count[h_cams[i]]++;
    f.cam_plain = count[0] == n;
    if (f.cam_plain) return 0;
    int next[LT_MAX_CAMERAS], nslots = 0, max_rows = 0, ov0 = h->d.img_h, ov1 = 0;
    LtCamTable t;
    memset(&t, 0, sizeof(t));
    for (int k = 0; k < LT_MAX_CAMERAS; ++k) {
        const LtCamera& c = h->cams[k];
        if (c.und_map) t.e[k] = {c.und_desc, c.bv_desc, c.ov_map, (c.roi1 - c.roi0) * h->d.img_w, c.ov0, c.ov1, c.cal.mppv, c.cal.mpph};
        next[k] = nslots;
        if (!count[k]) continue;
        nslots += (count[k] + 3) & ~3;
        max_rows = c.roi1 - c.roi0 > max_rows ? c.roi1 - c.roi0 : max_rows;
        if (c.ov1 > c.ov0) { ov0 = c.ov0 < ov0 ? c.ov0 : ov0; ov1 = c.ov1 > ov1 ? c.ov1 : ov1; }
    }
    std::vector<int> slot_pos(nslots, -1), chunk_cam(nslots / 4);
    for (int k = 0; k < LT_MAX_CAMERAS; ++k)
        for (int s = next[k]; s < next[k] + ((count[k] + 3) & ~3); s += 4) chunk_cam[s / 4] = k;
    for (int i = 0; i < n; ++i) slot_pos[next[h_cams[i]]++] = i;
    int rc;
    if ((rc = upload_ints(slot_pos.data(), nslots, f.slot_pos, st))) return rc;
    if ((rc = upload_ints(chunk_cam.data(), nslots / 4, f.chunk_cam, st))) return rc;
    if ((rc = upload_ints(h_cams, n, f.pos_cam, st))) return rc;
    k_set_cameras<<<1, LT_MAX_CAMERAS, 0, st>>>(t, f.cams);
    LT_LAUNCH_CHECK();
    f.cam_ov0 = ov1 > ov0 ? ov0 : 0;
    f.cam_ov1 = ov1 > ov0 ? ov1 : 0;
    *cb = {&f, nslots, max_rows};
    return 0;
}

static bool allows_retry(int n_tries) { return n_tries >= 2 || n_tries == -1; }

// The rounds of a sequence batch (lt_process_sequence): round r holds the positions that are the (r+1)-th occurrence
// of their stream, in position order; pos[off[r] .. off[r+1]) are its positions.
struct LtRounds {
    std::vector<int> pos, off;
};

// Rounds of the ids h_ids[0..n) (in [0, S)); false when no id repeats (one round: the batch itself).
static bool make_rounds(const int32_t* h_ids, int n, int S, LtRounds* r) {
    std::vector<int> occ(n), seen(S, 0);
    int R = 0;
    for (int i = 0; i < n; ++i) {
        occ[i] = seen[h_ids[i]]++;
        R = occ[i] + 1 > R ? occ[i] + 1 : R;
    }
    if (R < 2) return false;
    r->off.assign(R + 1, 0);
    for (int i = 0; i < n; ++i) r->off[occ[i] + 1]++;
    for (int k = 0; k < R; ++k) r->off[k + 1] += r->off[k];
    std::vector<int> next(r->off.begin(), r->off.end() - 1);
    r->pos.resize(n);
    for (int i = 0; i < n; ++i) r->pos[next[occ[i]]++] = i;
    return true;
}

// searches, second attempt of the streams that failed, state machine, overlay: advances the per-stream state.
// h_ids (host, validated by check_ids) maps batch position i to state slot h_ids[i]; NULL: the identity.
// fs: the buffer set whose profile snapshot the batch uses (NULL: p1 and the handle's windows for every position);
// n_tries: of the batch (with profiles: 2 when some position may take a second attempt, else 1).
// cf: the buffer set of a camera batch that is not on camera 0 alone (NULL otherwise).
// rounds (NULL: every id distinct): a sequence batch, without profiles or cameras.  The searches, the second attempt
// and the state update run round after round, each over its positions only, so that a frame sees the state its
// stream's previous frame left; the update snapshots what the overlay and the text of each position read, and the
// overlay and the text then run once over the batch from those snapshots.
static int process_back(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, int n_tries,
                        const LtAttemptParams& p1, lt_result* d_results, cudaStream_t st, bool own_begin,
                        const int32_t* h_ids, const LtFrontSet* fs, const LtFrontSet* cf, const LtRounds* rounds = nullptr) {
    int rc;
    const LtAttemptParams p2 = second_attempt();
    const LtProfile* prof = fs ? fs->profiles : nullptr;
    const int* pos_prof = fs ? fs->pos_profile : nullptr;
    const bool two = allows_retry(n_tries);
    if (own_begin) lt_prof_mark(h, ST_BEGIN, st);       // stage times are differences of marks on ONE stream
    const int* ids = nullptr;
    if (h_ids) {
        if ((rc = upload_stream_ids(h, h_ids, n, st))) return rc;
        ids = h->stream_ids;
    }
    // (h->seq_pos has one writer and its readers on this stream, as the stream ids: upload_stream_ids)
    if (rounds && (rc = upload_ints(rounds->pos.data(), n, h->seq_pos, st))) return rc;
    const int nr = rounds ? (int)rounds->off.size() - 1 : 1;
    const size_t S = h->S;
    for (int r = 0; r < nr; ++r) {
        const int* order = rounds ? h->seq_pos + rounds->off[r] : nullptr;
        const int m = rounds ? rounds->off[r + 1] - rounds->off[r] : n;
        LtSearchArgs sa;
        memset(&sa, 0, sizeof(sa));
        sa.mask = h->mask; sa.mode = 0; sa.att = h->att; sa.do_fit = 1; sa.ids = ids;
        if (h->capture) {
            sa.by_stream = 1; sa.pixels = h->cap_pixels; sa.pix_cap = h->pix_cap; sa.pix_counts = h->cap_counts;
            sa.centroids = h->cap_cents; sa.ncentroids = h->cap_ncents;
        }
        if ((rc = lt_launch_search(h, m, p1, sa, order, nullptr, st, prof, pos_prof, 1))) return rc;
        lt_prof_mark(h, ST_SEARCH, st);
        if (two) {
            // second attempt only for the streams whose first attempt failed (lane_tracker.py:1071-1128).
            // The reference re-runs undistort + warp here; their outputs are unchanged, so the planes are reused.
            if ((rc = lt_launch_select_retry(h, m, n_tries, st, prof, pos_prof, order))) return rc;
            lt_prof_mark(h, ST_RETRY_SELECT, st);
            if ((rc = lt_launch_filter(h, m, p2, h->retry_list, h->retry_count, st))) return rc;
            sa.att = h->att + h->S;
            if (h->capture) {
                sa.pixels = h->cap_pixels + S * 2 * (size_t)h->pix_cap; sa.pix_counts = h->cap_counts + S * 2;
                sa.centroids = h->cap_cents + S * 2 * LT_MAX_LEVELS; sa.ncentroids = h->cap_ncents + S * 2;
            }
            if ((rc = lt_launch_search(h, m, p2, sa, h->retry_list, h->retry_count, st, prof, pos_prof, 0))) return rc;
            lt_prof_mark(h, ST_SEARCH, st);
        }
        if ((rc = lt_launch_update_state(h, m, ids, d_results, two ? 2 : 1, st, cf, order))) return rc;
        lt_prof_mark(h, ST_UPDATE, st);
    }
    if (d_out) {
        // a sequence batch draws every position from its snapshot: a view of the handle whose polygon rows, boxes and
        // states are the snapshots, indexed by position (ids NULL), as lt_draw_lane and lt_draw_text draw
        lt_handle view;
        lt_handle* oh = h;
        if (rounds) {
            view = *h;
            view.lane_rows = h->seq_rows; view.lane_bbox = h->seq_bbox; view.state = h->seq_state;
            oh = &view;
            ids = nullptr;
        }
        // (copying the untouched rows on a side stream under the search kernels was measured: the copy saturates HBM
        // and slows the search by what it saves -- the plain in-order copy stays)
        // draw_lane writes its text into the frame BEFORE the blend (lane_tracker.py:653-662).  With the shipped
        // geometry the text rows and the rows the lane overlay can reach are disjoint and the order is immaterial;
        // when they overlap (other calibrations) the text goes first and the blend runs in place over it.
        // (a camera batch: the union of its cameras' overlay rows; for a camera whose rows miss the text rows, the
        // order of text and blend does not matter)
        const int ov0 = cf ? cf->cam_ov0 : h->d.ov0, ov1 = cf ? cf->cam_ov1 : h->d.ov1;
        const bool text_under_blend = h->txt_nchars > 0 && h->txt_row0 < ov1 && ov0 < h->txt_row1;
        // NV12 input: the frame is converted where it is read; with text under the blend, the whole frame is converted
        // into d_out first and the text and the blend then run on d_out as for RGB.
        const bool nv12 = h->frame_format == LT_FRAME_NV12;
        if (text_under_blend) {
            if (nv12) {
                if ((rc = lt_launch_nv12_to_rgb(d_frames, d_out, n, h->d.img_w, h->d.img_h, 0, h->d.img_h, st))) return rc;
            } else if (d_out != d_frames) {
                LT_CUDA(cudaMemcpyAsync(d_out, d_frames, (size_t)n * h->d.img_w * h->d.img_h * 3, cudaMemcpyDeviceToDevice, st));
            }
            if ((rc = lt_launch_text(oh, d_out, n, ids, st))) return rc;
            if ((rc = lt_launch_overlay(oh, d_out, d_out, n, h->draw_flags, ids, st, cf))) return rc;
        } else {
            if (nv12) rc = lt_launch_overlay_nv12(oh, d_frames, d_out, n, h->draw_flags, ids, st, cf);
            else rc = lt_launch_overlay(oh, d_frames, d_out, n, h->draw_flags, ids, st, cf);
            if (rc) return rc;
            if ((rc = lt_launch_text(oh, d_out, n, ids, st))) return rc;
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

// d_out of the process calls: 4-byte aligned; under LT_FRAME_NV12 it is a separate RGB buffer, so its bytes may not
// overlap the NV12 input (the annotation cannot happen in place).
static int check_out(const lt_handle* h, const uint8_t* d_frames, const uint8_t* d_out, int n) {
    int rc;
    if ((rc = check_frame_buffer(d_out, "d_out"))) return rc;
    if (h && d_out && d_frames && n > 0 && h->frame_format == LT_FRAME_NV12) {
        const size_t fb = (size_t)h->d.img_w * h->d.img_h;
        const uintptr_t o0 = (uintptr_t)d_out, o1 = o0 + (size_t)n * fb * 3;
        const uintptr_t f0 = (uintptr_t)d_frames, f1 = f0 + (size_t)n * (fb + fb / 2);
        if (o0 < f1 && f0 < o1) {
            lt_set_error("d_out overlaps the NV12 input frames: NV12 frames are annotated into a separate RGB buffer");
            return -1;
        }
    }
    return 0;
}

// The checks every process call makes on its batch size, frames and buffer set (has_params: params or the profile
// list is not NULL).
static int process_args(lt_handle* h, const uint8_t* d_frames, int n, bool has_params, int set) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!d_frames || !has_params) { lt_set_error("null argument"); return -1; }
    if ((rc = check_frame_buffer(d_frames, "d_frames"))) return rc;
    if (set != 0 && set != 1) { lt_set_error("buffer set must be 0 or 1"); return -1; }
    return 0;
}

// bandwidth: the widest band-search bandwidth the batch uses.  Then selects buffer set `set`.
static int process_set(lt_handle* h, int set, int bandwidth) {
    int rc;
    // captured pixel lists: a band-search row holds up to 2*bandwidth - 1 pixels (attempt 2 uses bandwidth 30)
    const int bw = bandwidth > 30 ? bandwidth : 30;
    if (h->capture && (long long)(2 * bw - 1) * h->d.bv_h > (long long)h->pix_cap) {
        lt_set_error("bandwidth %d can overflow the captured pixel lists (capacity %d): raise it with lt_set_pixel_capacity",
                     bandwidth, h->pix_cap);
        return -1;
    }
    if ((rc = alloc_front_set(h, set))) return rc;
    select_set(h, set);
    return 0;
}

// Stream ids of lt_process_streams / lt_process_back_streams: 1 <= n <= S ids in [0, S), pairwise distinct (two
// frames of one stream in a batch would race on its state) unless `repeats` (lt_process_sequence, whose back half
// runs the frames of a stream in rounds).  Checked before anything is enqueued.
static int check_ids(lt_handle* h, const int32_t* h_ids, int n, bool repeats = false) {
    int rc;
    if ((rc = check_n(h, n))) return rc;
    if (!h_ids) { lt_set_error("null stream id list"); return -1; }
    std::vector<unsigned char> seen(h->S, 0);
    for (int i = 0; i < n; ++i) {
        const int id = h_ids[i];
        if (id < 0 || id >= h->S) { lt_set_error("stream id %d at batch position %d outside [0, %d)", id, i, h->S); return -1; }
        if (seen[id] && !repeats) { lt_set_error("stream id %d appears twice in the batch (position %d)", id, i); return -1; }
        seen[id] = 1;
    }
    return 0;
}

// Profile indices of lt_process_*_profiles: every entry names a profile that is set.  Returns the widest bandwidth
// and the batch's n_tries (2 when a profile used allows a second attempt, else 1).
static int check_profiles(lt_handle* h, const int32_t* h_prof, int n, int* bandwidth, int* n_tries) {
    if (!h_prof) { lt_set_error("null profile list"); return -1; }
    *bandwidth = 0;
    *n_tries = 1;
    for (int i = 0; i < n; ++i) {
        const int k = h_prof[i];
        if (k < 0 || k >= LT_MAX_PROFILES) {
            lt_set_error("profile %d at batch position %d outside [0, %d)", k, i, LT_MAX_PROFILES);
            return -1;
        }
        if (!((h->profiles_set >> k) & 1u)) { lt_set_error("profile %d at batch position %d is unset", k, i); return -1; }
        const LtProfile& q = h->profiles[k];
        if (q.p.bandwidth > *bandwidth) *bandwidth = q.p.bandwidth;
        if (allows_retry(q.n_tries)) *n_tries = 2;
    }
    return 0;
}

// Camera indices of lt_process_*_cameras: every entry names a camera that is set; remap mode 1 (whose fused table
// holds camera 0's calibration) takes camera 0 only.
static int check_cameras(lt_handle* h, const int32_t* h_cams, int n) {
    if (!h_cams) { lt_set_error("null camera list"); return -1; }
    for (int i = 0; i < n; ++i) {
        const int k = h_cams[i];
        if (k < 0 || k >= LT_MAX_CAMERAS) {
            lt_set_error("camera %d at batch position %d outside [0, %d)", k, i, LT_MAX_CAMERAS);
            return -1;
        }
        if (!h->cams[k].und_map) { lt_set_error("camera %d at batch position %d is unset", k, i); return -1; }
        if (k && h->remap_mode == 1) {
            lt_set_error("camera %d at batch position %d: remap mode 1 (fused single resample) has camera 0's calibration "
                         "built in; camera calls need remap mode 0", k, i);
            return -1;
        }
    }
    return 0;
}

// What one process entry point does: the front half, the back half or both, with or without a stream id list, with
// one lt_params or with a parameter profile per batch position, and with or without a camera per batch position.
// PROC_SEQ (with PROC_IDS): ids may repeat, the frames of a stream being its consecutive frames (lt_process_sequence).
enum { PROC_FRONT = 1, PROC_BACK = 2, PROC_IDS = 4, PROC_PROFILES = 8, PROC_CAMERAS = 16, PROC_SEQ = 32 };

// Grow the stage-timing event pool, keeping the events already recorded, so that `marks` more marks fit.
static int prof_reserve(lt_handle* h, int marks) {
    if (!h->prof_active || h->prof_n + marks <= h->prof_cap) return 0;
    const int need = h->prof_n + marks, cap = need > 2 * h->prof_cap ? need : 2 * h->prof_cap;
    cudaEvent_t* ev = new cudaEvent_t[cap];
    int* stage = new int[cap];
    for (int i = 0; i < h->prof_cap; ++i) { ev[i] = h->prof_ev[i]; stage[i] = h->prof_stage[i]; }
    for (int i = h->prof_cap; i < cap; ++i)
        if (cudaEventCreate(&ev[i]) != cudaSuccess) {
            for (int k = h->prof_cap; k < i; ++k) cudaEventDestroy(ev[k]);
            delete[] ev; delete[] stage;
            lt_set_error("cannot create the stage-timing events");
            return -2;
        }
    delete[] h->prof_ev; delete[] h->prof_stage;
    h->prof_ev = ev; h->prof_stage = stage; h->prof_cap = cap;
    return 0;
}

// Buffers of the sequence back half (LtRounds), allocated on first use like buffer set 1.
static int alloc_sequence(lt_handle* h) {
    if (h->seq_state) return 0;
    LT_CUDA(cudaSetDevice(h->cfg.device));
    const size_t S = h->S;
    int rc = dev_alloc(&h->seq_pos, S);
    if (!rc) rc = dev_alloc(&h->seq_rows, S * (size_t)h->d.bv_h);
    if (!rc) rc = dev_alloc(&h->seq_bbox, S);
    if (!rc) rc = dev_alloc(&h->seq_state, S);
    return rc;
}

// The checks of the process entry points, in this order and all before anything is enqueued, then the halves.
static int process_call(lt_handle* h, int what, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int n,
                        const lt_params* params, const int32_t* h_prof, int set, lt_result* d_results, void* stream,
                        const int32_t* h_cams = nullptr) {
    int rc;
    LtAttemptParams p1;
    const bool front = what & PROC_FRONT, back = what & PROC_BACK, profiles = what & PROC_PROFILES;
    const cudaStream_t st = (cudaStream_t)stream;
    if ((what & PROC_IDS) && (rc = check_ids(h, h_ids, n, what & PROC_SEQ))) return rc;
    if (back && (rc = check_out(h, d_frames, d_out, n))) return rc;
    if ((rc = process_args(h, d_frames, n, profiles || params, set))) return rc;
    int bandwidth, n_tries;
    if (profiles) {
        if ((rc = check_profiles(h, h_prof, n, &bandwidth, &n_tries))) return rc;
        if (back && !front) {    // the front half of this set must have taken these profiles
            const LtFrontSet& f = h->fs[set];
            if (f.snap_n == 0) {
                lt_set_error("buffer set %d was last filled by a front half without profiles", set);
                return -1;
            }
            if (f.snap_n != n) {
                lt_set_error("buffer set %d holds a front half of %d frames, not %d", set, f.snap_n, n);
                return -1;
            }
            for (int i = 0; i < n; ++i)
                if (f.h_pos_profile[i] != h_prof[i]) {
                    lt_set_error("profile %d at batch position %d differs from the front half's profile %d", h_prof[i], i,
                                 f.h_pos_profile[i]);
                    return -1;
                }
            // the back half uses the snapshot of the front half: its bandwidths and n_tries
            bandwidth = 0; n_tries = 1;
            for (int i = 0; i < n; ++i) {
                const LtProfile& q = f.snap[h_prof[i]];
                if (q.p.bandwidth > bandwidth) bandwidth = q.p.bandwidth;
                if (allows_retry(q.n_tries)) n_tries = 2;
            }
        }
        // the launchers' own checks see a valid parameter set; every kernel reads its position's profile instead
        p1 = ((back && !front) ? h->fs[set].snap : h->profiles)[h_prof[0]].p;
    } else {
        p1 = attempt_from(*params);
        if ((rc = check_params(h, p1))) return rc;
        bandwidth = p1.bandwidth;
        n_tries = params->n_tries;
    }
    const bool cameras = what & PROC_CAMERAS;
    if (cameras) {
        if (profiles && params) { lt_set_error("params and h_profiles are exclusive: pass one of them"); return -1; }
        if ((rc = check_cameras(h, h_cams, n))) return rc;
        if (back && !front) {    // the front half of this set must have taken these cameras
            const LtFrontSet& f = h->fs[set];
            if (f.cam_n == 0) {
                lt_set_error("buffer set %d was last filled by a front half without cameras", set);
                return -1;
            }
            if (f.cam_n != n) {
                lt_set_error("buffer set %d holds a camera front half of %d frames, not %d", set, f.cam_n, n);
                return -1;
            }
            for (int i = 0; i < n; ++i)
                if (f.h_pos_cam[i] != h_cams[i]) {
                    lt_set_error("camera %d at batch position %d differs from the front half's camera %d", h_cams[i], i,
                                 f.h_pos_cam[i]);
                    return -1;
                }
        }
    }
    if ((rc = process_set(h, set, bandwidth))) return rc;
    if (back && !d_results) { lt_set_error("null argument"); return -1; }
    // a sequence batch with a repeated id: its rounds, buffers and stage marks (a batch without one runs as
    // lt_process_streams)
    LtRounds rounds;
    const bool seq = back && (what & PROC_SEQ) && make_rounds(h_ids, n, h->S, &rounds);
    if (seq) {
        if ((rc = alloc_sequence(h))) return rc;
        // lt_profile_begin leaves room for the marks of its calls; a round adds up to six (search, retry selection,
        // box, open5, search, update)
        const int left = h->prof_max_calls - h->prof_calls;
        if ((rc = prof_reserve(h, (32 + 2 * LT_MAX_PROFILES) * (left > 1 ? left : 1) + 6 * (int)rounds.off.size()))) return rc;
    }
    LtFrontSet& fset = h->fs[set];
    if (front) {
        LtCamBatch cb = {nullptr, 0, 0};
        fset.cam_n = 0;
        if (cameras && (rc = prepare_cameras(h, h_cams, n, set, st, &cb))) return rc;
        const LtCamBatch* cbp = cb.f ? &cb : nullptr;
        if (profiles) {
            rc = process_front_profiles(h, d_frames, h_prof, n, set, st, cbp);
        } else {
            fset.snap_n = 0;
            const LtFilterGroup g = {p1, nullptr, n};
            rc = process_front(h, d_frames, n, &g, 1, st, cbp);
        }
        if (rc) return rc;
        fset.cam_pending = cameras && !back;
    }
    if (!back) return 0;
    fset.cam_pending = 0;
    const LtFrontSet* cf = (cameras && !fset.cam_plain) ? &fset : nullptr;
    return process_back(h, d_frames, d_out, n, n_tries, p1, d_results, st, !front, h_ids, profiles ? &fset : nullptr, cf,
                        seq ? &rounds : nullptr);
}

extern "C" int lt_process(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n, const lt_params* params,
                          lt_result* d_results, void* stream) {
    return process_call(h, PROC_FRONT | PROC_BACK, d_frames, d_out, nullptr, n, params, nullptr, 0, d_results, stream);
}

extern "C" int lt_process_front(lt_handle* h, const uint8_t* d_frames, int32_t n, const lt_params* params, int32_t set,
                                void* stream) {
    return process_call(h, PROC_FRONT, d_frames, nullptr, nullptr, n, params, nullptr, set, nullptr, stream);
}

extern "C" int lt_process_back(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int32_t n, const lt_params* params,
                               int32_t set, lt_result* d_results, void* stream) {
    return process_call(h, PROC_BACK, d_frames, d_out, nullptr, n, params, nullptr, set, d_results, stream);
}

extern "C" int lt_process_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                                  const lt_params* params, lt_result* d_results, void* stream) {
    return process_call(h, PROC_FRONT | PROC_BACK | PROC_IDS, d_frames, d_out, h_ids, n, params, nullptr, 0, d_results, stream);
}

extern "C" int lt_process_back_streams(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                       int32_t n, const lt_params* params, int32_t set, lt_result* d_results, void* stream) {
    return process_call(h, PROC_BACK | PROC_IDS, d_frames, d_out, h_ids, n, params, nullptr, set, d_results, stream);
}

extern "C" int lt_process_sequence(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids, int32_t n,
                                   const lt_params* params, lt_result* d_results, void* stream) {
    return process_call(h, PROC_FRONT | PROC_BACK | PROC_IDS | PROC_SEQ, d_frames, d_out, h_ids, n, params, nullptr, 0,
                        d_results, stream);
}

extern "C" int lt_process_back_sequence(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                        int32_t n, const lt_params* params, int32_t set, lt_result* d_results, void* stream) {
    return process_call(h, PROC_BACK | PROC_IDS | PROC_SEQ, d_frames, d_out, h_ids, n, params, nullptr, set, d_results,
                        stream);
}

extern "C" int lt_process_profiles(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                   const int32_t* h_profiles, int32_t n, lt_result* d_results, void* stream) {
    return process_call(h, PROC_FRONT | PROC_BACK | PROC_PROFILES | (h_ids ? PROC_IDS : 0), d_frames, d_out, h_ids, n,
                        nullptr, h_profiles, 0, d_results, stream);
}

extern "C" int lt_process_front_profiles(lt_handle* h, const uint8_t* d_frames, const int32_t* h_profiles, int32_t n,
                                         int32_t set, void* stream) {
    return process_call(h, PROC_FRONT | PROC_PROFILES, d_frames, nullptr, nullptr, n, nullptr, h_profiles, set, nullptr,
                        stream);
}

extern "C" int lt_process_back_profiles(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                        const int32_t* h_profiles, int32_t n, int32_t set, lt_result* d_results,
                                        void* stream) {
    return process_call(h, PROC_BACK | PROC_PROFILES | (h_ids ? PROC_IDS : 0), d_frames, d_out, h_ids, n, nullptr,
                        h_profiles, set, d_results, stream);
}

extern "C" int lt_process_cameras(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                  const int32_t* h_cameras, int32_t n, const lt_params* params, const int32_t* h_profiles,
                                  lt_result* d_results, void* stream) {
    return process_call(h, PROC_FRONT | PROC_BACK | PROC_CAMERAS | (h_profiles ? PROC_PROFILES : 0) | (h_ids ? PROC_IDS : 0),
                        d_frames, d_out, h_ids, n, params, h_profiles, 0, d_results, stream, h_cameras);
}

extern "C" int lt_process_front_cameras(lt_handle* h, const uint8_t* d_frames, const int32_t* h_cameras, int32_t n,
                                        const lt_params* params, const int32_t* h_profiles, int32_t set, void* stream) {
    return process_call(h, PROC_FRONT | PROC_CAMERAS | (h_profiles ? PROC_PROFILES : 0), d_frames, nullptr, nullptr, n,
                        params, h_profiles, set, nullptr, stream, h_cameras);
}

extern "C" int lt_process_back_cameras(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, const int32_t* h_ids,
                                       const int32_t* h_cameras, int32_t n, const lt_params* params,
                                       const int32_t* h_profiles, int32_t set, lt_result* d_results, void* stream) {
    return process_call(h, PROC_BACK | PROC_CAMERAS | (h_profiles ? PROC_PROFILES : 0) | (h_ids ? PROC_IDS : 0), d_frames,
                        d_out, h_ids, n, params, h_profiles, set, d_results, stream, h_cameras);
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
    // a call marks at most about 20 boundaries, plus the threshold and noise stages once per filter group (a sequence
    // call with several rounds grows the pool before it enqueues: prof_reserve)
    int need = max_calls * (32 + 2 * LT_MAX_PROFILES);
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
    if (mode == 1 && h->frame_format == LT_FRAME_NV12) {
        lt_set_error("remap mode 1 (fused single resample) samples RGB frames: not available with NV12 frames");
        return -1;
    }
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

extern "C" int lt_set_frame_format(lt_handle* h, int32_t format) {
    if (!h) { lt_set_error("null handle"); return -1; }
    if (format != LT_FRAME_RGB && format != LT_FRAME_NV12) {
        lt_set_error("frame format must be %d (RGB) or %d (NV12), got %d", LT_FRAME_RGB, LT_FRAME_NV12, format);
        return -1;
    }
    if (format == LT_FRAME_NV12 && (h->d.img_h & 1)) {
        lt_set_error("NV12 frames need an even image height (got %d)", h->d.img_h);
        return -1;
    }
    if (format == LT_FRAME_NV12 && h->remap_mode == 1) {
        lt_set_error("NV12 frames are not available with remap mode 1 (fused single resample), which samples RGB frames");
        return -1;
    }
    h->frame_format = format;
    return 0;
}

extern "C" int lt_memcpy_rows(lt_handle* h, void* dst, const void* src, int32_t n, int32_t row0, int32_t row1,
                              int32_t to_device, void* stream) {
    if (!h || !dst || !src || n < 1 || row0 < 0 || row1 > h->d.img_h || row0 >= row1) { lt_set_error("bad argument"); return -1; }
    const cudaMemcpyKind kind = to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    if (h->frame_format == LT_FRAME_NV12) {     // luma rows [row0, row1), then the chroma rows that cover them
        const size_t W = (size_t)h->d.img_w, H = (size_t)h->d.img_h, frame_bytes = W * (H + H / 2);
        const size_t c0 = H + (size_t)row0 / 2, c1 = H + (size_t)(row1 + 1) / 2;
        LT_CUDA(cudaMemcpy2DAsync((char*)dst + row0 * W, frame_bytes, (const char*)src + row0 * W, frame_bytes,
                                  (size_t)(row1 - row0) * W, (size_t)n, kind, (cudaStream_t)stream));
        LT_CUDA(cudaMemcpy2DAsync((char*)dst + c0 * W, frame_bytes, (const char*)src + c0 * W, frame_bytes, (c1 - c0) * W,
                                  (size_t)n, kind, (cudaStream_t)stream));
        return 0;
    }
    const size_t row_bytes = (size_t)h->d.img_w * 3, frame_bytes = row_bytes * h->d.img_h;
    const char* s = (const char*)src + (size_t)row0 * row_bytes;
    char* d = (char*)dst + (size_t)row0 * row_bytes;
    LT_CUDA(cudaMemcpy2DAsync(d, frame_bytes, s, frame_bytes, (size_t)(row1 - row0) * row_bytes, (size_t)n, kind,
                              (cudaStream_t)stream));
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
    return lt_launch_nv12_to_rgb(d_nv12, d_rgb, n, width, height, 0, height, (cudaStream_t)stream);
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
    if ((rc = check_filter_params(p))) return rc;
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

// ---------------------------------------------------------------------------
// stream starts (lt_reset_async) and state records (lt_export_states / lt_import_states)
// ---------------------------------------------------------------------------

// lt_reset_async: the initial state h->init copied into the slots of a chunk of ids, one word per thread and step.
__global__ void __launch_bounds__(256) k_reset_states(const __grid_constant__ LtIdsChunk c, const LtDevState* __restrict__ init,
                                                      LtDevState* __restrict__ state) {
    constexpr int W = sizeof(LtDevState) / sizeof(int);
    static_assert(sizeof(LtDevState) % sizeof(int) == 0, "LtDevState is copied as words");
    const int* src = reinterpret_cast<const int*>(init);
    for (int i = threadIdx.x; i < c.count * W; i += blockDim.x)
        reinterpret_cast<int*>(state + c.ids[i / W])[i % W] = __ldg(&src[i % W]);
}

// Byte offsets of the parts of one state record (include/lane_tracker_b200.h), from the bird's-eye height.
struct LtRecordLayout {
    int state, avg, rows, bbox, bytes;
};
static constexpr int LT_RECORD_HEADER_BYTES = 64;
__host__ __device__ static inline int lt_align16(int v) { return (v + 15) & ~15; }
__host__ __device__ static inline LtRecordLayout lt_record_layout(int H) {
    LtRecordLayout r;
    r.state = LT_RECORD_HEADER_BYTES;
    r.avg = r.state + lt_align16((int)sizeof(LtDevState));
    r.rows = r.avg + 2 * H * (int)sizeof(int);
    r.bbox = lt_align16(r.rows + H * (int)sizeof(int2));
    r.bytes = r.bbox + (int)sizeof(int4);
    return r;
}

struct LtRecordHeader {          // the 64-byte header, int32 words
    uint32_t magic;
    int abi, state_bytes, bv_w, bv_h, n_average, n_fail, n_reset;
    int zero[8];
};
static_assert(sizeof(LtRecordHeader) == LT_RECORD_HEADER_BYTES, "record header is 64 bytes");

// What the record kernels read and write of a handle: its header and its per-stream arrays.
struct LtRecordDev {
    LtRecordHeader hdr;
    LtDevState* state; int* avg_x; int2* rows; int4* bbox;
};

// The ids of a record launch.  Kept at 512 so that they and LtRecordDev fit the classic 4 KB of kernel arguments.
#define LT_RECORD_CHUNK 512
struct LtRecordIds {
    int offset, count;
    int ids[LT_RECORD_CHUNK];
};

__device__ static inline void zero_bytes(uint8_t* p, int a, int b) {
    for (int i = a + (int)threadIdx.x; i < b; i += blockDim.x) p[i] = 0;
}

// One CTA per record: record offset + blockIdx.x of dst <- stream ids[blockIdx.x] (16-byte aligned records).
__global__ void __launch_bounds__(256) k_export_states(const __grid_constant__ LtRecordIds c, const __grid_constant__ LtRecordDev r,
                                                       uint8_t* __restrict__ dst) {
    const int H = r.hdr.bv_h, sid = c.ids[blockIdx.x], tid = threadIdx.x;
    const LtRecordLayout L = lt_record_layout(H);
    uint8_t* rec = dst + (size_t)(c.offset + blockIdx.x) * L.bytes;
    if (tid < LT_RECORD_HEADER_BYTES / 4)
        reinterpret_cast<int*>(rec)[tid] = reinterpret_cast<const int*>(&r.hdr)[tid];
    const int* st = reinterpret_cast<const int*>(r.state + sid);
    for (int i = tid; i < (int)(sizeof(LtDevState) / 4); i += blockDim.x) reinterpret_cast<int*>(rec + L.state)[i] = st[i];
    zero_bytes(rec, L.state + (int)sizeof(LtDevState), L.avg);
    const int* ax = r.avg_x + (size_t)sid * 2 * H;
    for (int i = tid; i < 2 * H; i += blockDim.x) reinterpret_cast<int*>(rec + L.avg)[i] = ax[i];
    const int2* rows = r.rows + (size_t)sid * H;
    for (int i = tid; i < H; i += blockDim.x) reinterpret_cast<int2*>(rec + L.rows)[i] = rows[i];
    zero_bytes(rec, L.rows + H * (int)sizeof(int2), L.bbox);
    if (tid == 0) *reinterpret_cast<int4*>(rec + L.bbox) = r.bbox[sid];
}

// One CTA per record: checks record offset + blockIdx.x of src, and applies it to slot ids[blockIdx.x] only if it
// passes (status: LT_RECORD_OK / LT_RECORD_BAD_HEADER / LT_RECORD_BAD_STATE).
__global__ void __launch_bounds__(256) k_import_states(const __grid_constant__ LtRecordIds c, const __grid_constant__ LtRecordDev r,
                                                       const uint8_t* __restrict__ src, int* __restrict__ status) {
    const int H = r.hdr.bv_h, W = r.hdr.bv_w, sid = c.ids[blockIdx.x], tid = threadIdx.x;
    const LtRecordLayout L = lt_record_layout(H);
    const int i = c.offset + blockIdx.x;
    const uint8_t* rec = src + (size_t)i * L.bytes;
    __shared__ int code;
    if (tid == 0) {
        const LtRecordHeader& g = *reinterpret_cast<const LtRecordHeader*>(rec);
        int k = LT_RECORD_OK;
        if (g.magic != r.hdr.magic || g.abi != r.hdr.abi || g.state_bytes != r.hdr.state_bytes || g.bv_w != W ||
            g.bv_h != H || g.n_average != r.hdr.n_average || g.n_fail != r.hdr.n_fail || g.n_reset != r.hdr.n_reset) {
            k = LT_RECORD_BAD_HEADER;
        } else {
            const lt_state& s = reinterpret_cast<const LtDevState*>(rec + L.state)->s;
            const int nav = r.hdr.n_average;
            const int4 b = *reinterpret_cast<const int4*>(rec + L.bbox);
            if (s.ring_len < 0 || s.ring_len > nav || s.radii_len < 0 || s.radii_len > nav || s.n_left_avg < 0 ||
                s.n_left_avg > H || s.n_right_avg < 0 || s.n_right_avg > H ||
                (b.x <= b.y && (b.x < 0 || b.y >= W || b.z < 0 || b.z > b.w || b.w >= H)))
                k = LT_RECORD_BAD_STATE;
        }
        code = k;
    }
    __syncthreads();
    int bad_row = 0;
    if (code == LT_RECORD_OK) {
        const int2* rows = reinterpret_cast<const int2*>(rec + L.rows);
        for (int y = tid; y < H; y += blockDim.x) {
            const int2 q = rows[y];
            bad_row |= q.x <= q.y && (q.x < 0 || q.y >= W);
        }
    }
    bad_row = __syncthreads_or(bad_row);
    const int k = code != LT_RECORD_OK ? code : (bad_row ? LT_RECORD_BAD_STATE : LT_RECORD_OK);
    if (tid == 0 && status) status[i] = k;
    if (k != LT_RECORD_OK) return;
    const int* st = reinterpret_cast<const int*>(rec + L.state);
    for (int j = tid; j < (int)(sizeof(LtDevState) / 4); j += blockDim.x) reinterpret_cast<int*>(r.state + sid)[j] = st[j];
    const int* ax = reinterpret_cast<const int*>(rec + L.avg);
    for (int j = tid; j < 2 * H; j += blockDim.x) r.avg_x[(size_t)sid * 2 * H + j] = ax[j];
    const int2* rows = reinterpret_cast<const int2*>(rec + L.rows);
    for (int j = tid; j < H; j += blockDim.x) r.rows[(size_t)sid * H + j] = rows[j];
    if (tid == 0) r.bbox[sid] = *reinterpret_cast<const int4*>(rec + L.bbox);
}

extern "C" int lt_reset_async(lt_handle* h, const int32_t* h_ids, int32_t n, void* stream) {
    int rc;
    if (!h) { lt_set_error("null handle"); return -1; }
    std::vector<int32_t> all;
    if (!h_ids) {
        all.resize(h->S);
        for (int i = 0; i < h->S; ++i) all[i] = i;
        h_ids = all.data();
        n = h->S;
    } else if ((rc = check_ids(h, h_ids, n))) {
        return rc;
    }
    const cudaStream_t st = (cudaStream_t)stream;
    LtIdsChunk c;
    for (int off = 0; off < n; off += LT_IDS_CHUNK) {
        c.offset = off;
        c.count = n - off < LT_IDS_CHUNK ? n - off : LT_IDS_CHUNK;
        memcpy(c.ids, h_ids + off, (size_t)c.count * sizeof(int32_t));
        k_reset_states<<<1, 256, 0, st>>>(c, h->init, h->state);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int64_t lt_state_record_bytes(lt_handle* h) {
    if (!h) { lt_set_error("null handle"); return -1; }
    return lt_record_layout(h->d.bv_h).bytes;
}

static LtRecordDev record_dev(const lt_handle* h) {
    LtRecordDev r;
    memset(&r, 0, sizeof(r));
    r.hdr.magic = LT_RECORD_MAGIC; r.hdr.abi = LT_ABI_VERSION; r.hdr.state_bytes = (int)sizeof(lt_state);
    r.hdr.bv_w = h->d.bv_w; r.hdr.bv_h = h->d.bv_h;
    r.hdr.n_average = h->cfg.n_average; r.hdr.n_fail = h->cfg.n_fail; r.hdr.n_reset = h->cfg.n_reset;
    r.state = h->state; r.avg_x = h->avg_x; r.rows = h->lane_rows; r.bbox = h->lane_bbox;
    return r;
}

// export (d_status unused) or import of the records of streams h_ids[0..n), all checks before anything is enqueued
static int move_states(lt_handle* h, bool to_handle, const int32_t* h_ids, int n, const void* d_rec, int32_t* d_status,
                       void* stream) {
    int rc;
    if ((rc = check_ids(h, h_ids, n))) return rc;
    if (!d_rec) { lt_set_error("null record buffer"); return -1; }
    if ((uintptr_t)d_rec & 15) { lt_set_error("the record buffer must be 16-byte aligned (got address %p)", d_rec); return -1; }
    if ((uintptr_t)d_status & 3) { lt_set_error("d_status must be 4-byte aligned (got address %p)", (void*)d_status); return -1; }
    const cudaStream_t st = (cudaStream_t)stream;
    const LtRecordDev r = record_dev(h);
    LtRecordIds c;
    for (int off = 0; off < n; off += LT_RECORD_CHUNK) {
        c.offset = off;
        c.count = n - off < LT_RECORD_CHUNK ? n - off : LT_RECORD_CHUNK;
        memcpy(c.ids, h_ids + off, (size_t)c.count * sizeof(int32_t));
        if (to_handle) k_import_states<<<c.count, 256, 0, st>>>(c, r, (const uint8_t*)d_rec, d_status);
        else k_export_states<<<c.count, 256, 0, st>>>(c, r, (uint8_t*)d_rec);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int lt_export_states(lt_handle* h, const int32_t* h_ids, int32_t n, void* d_dst, void* stream) {
    return move_states(h, false, h_ids, n, d_dst, nullptr, stream);
}

extern "C" int lt_import_states(lt_handle* h, const int32_t* h_ids, int32_t n, const void* d_src, int32_t* d_status,
                                void* stream) {
    return move_states(h, true, h_ids, n, d_src, d_status, stream);
}

extern "C" int64_t lt_debug_read(lt_handle* h, int32_t what, int32_t id, void* dst, int64_t cap) {
    if (h && what == 13) {     // rows of camera `id` (host data, no synchronisation)
        if (!dst || id < 0 || id >= LT_MAX_CAMERAS) { lt_set_error("bad argument"); return -1; }
        const LtCamera& c = h->cams[id];
        if (!c.und_map) { lt_set_error("camera %d is unset", id); return -1; }
        int v[6] = {c.roi0, c.roi1, c.ov0, c.ov1, c.src0, c.src1};
        if (cap < (int64_t)sizeof(v)) { lt_set_error("buffer too small"); return -1; }
        memcpy(dst, v, sizeof(v));
        return sizeof(v);
    }
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
