// Remap stage: cv2.undistort + cv2.warpPerspective (lane_tracker.py:832-834) and the
// overlay of draw_lane (lane_tracker.py:629-662), as fixed-point gather kernels.
//
// OpenCV evaluates the source coordinates in fp64, rounds them to 1/32 px (Q5) and
// interpolates with a Q15 weight table; the coordinate tables depend only on the
// calibration, so they are built once per handle (kernels below, fp64 with explicit
// round-to-nearest intrinsics: no FMA contraction, same operation order as OpenCV)
// and shared by every stream.  Compiled with -fmad=false.
#include "lt_common.cuh"

// ---------------------------------------------------------------------------
// coordinate tables
// ---------------------------------------------------------------------------

__device__ __forceinline__ double mul64(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add64(double a, double b) { return __dadd_rn(a, b); }

__device__ __forceinline__ int round_sat_i32(double v) {
    v = fmax(-2147483648.0, fmin(2147483647.0, v));
    return (int)rint(v);
}

struct UndistortCoef {
    double iR[9];
    double k1, k2, p1, p2, k3, fx, fy, cx, cy;
};

// cv2.undistort(src, K, D, None, K): Q5 source coordinates of every destination pixel.
__global__ void k_build_undistort_map(int2* __restrict__ map, int w, int h, UndistortCoef c) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= w || i >= h) return;
    double di = (double)i, dj = (double)j;
    double _x = add64(add64(mul64(di, c.iR[1]), c.iR[2]), mul64(dj, c.iR[0]));
    double _y = add64(add64(mul64(di, c.iR[4]), c.iR[5]), mul64(dj, c.iR[3]));
    double _w = add64(add64(mul64(di, c.iR[7]), c.iR[8]), mul64(dj, c.iR[6]));
    double x = __ddiv_rn(_x, _w), y = __ddiv_rn(_y, _w);
    double x2 = mul64(x, x), y2 = mul64(y, y);
    double r2 = add64(x2, y2);
    double _2xy = mul64(mul64(2.0, x), y);
    double kr = add64(1.0, mul64(add64(mul64(add64(mul64(c.k3, r2), c.k2), r2), c.k1), r2));
    double xd = add64(add64(mul64(x, kr), mul64(c.p1, _2xy)), mul64(c.p2, add64(r2, mul64(2.0, x2))));
    double yd = add64(add64(mul64(y, kr), mul64(c.p1, add64(r2, mul64(2.0, y2)))), mul64(c.p2, _2xy));
    double u = add64(mul64(c.fx, xd), c.cx);
    double v = add64(mul64(c.fy, yd), c.cy);
    map[(size_t)i * w + j] = make_int2(round_sat_i32(mul64(u, 32.0)), round_sat_i32(mul64(v, 32.0)));
}

struct Mat9 { double m[9]; };

// cv2.warpPerspective(src, M, (dw, dh)): `m` is inv(M); 64-column block origin as in OpenCV.
__global__ void k_build_perspective_map(int2* __restrict__ map, int dw, int dh, Mat9 mm) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= dw || y >= dh) return;
    const double* m = mm.m;
    double xb = (double)((x >> 6) << 6), x1 = (double)(x & 63), dy = (double)y;
    double X0 = add64(add64(mul64(m[0], xb), mul64(m[1], dy)), m[2]);
    double Y0 = add64(add64(mul64(m[3], xb), mul64(m[4], dy)), m[5]);
    double W0 = add64(add64(mul64(m[6], xb), mul64(m[7], dy)), m[8]);
    double W = add64(W0, mul64(m[6], x1));
    W = (W != 0.0) ? __ddiv_rn(32.0, W) : 0.0;
    double fX = mul64(add64(X0, mul64(m[0], x1)), W);
    double fY = mul64(add64(Y0, mul64(m[3], x1)), W);
    map[(size_t)y * dw + x] = make_int2(round_sat_i32(fX), round_sat_i32(fY));
}

static void invert3x3(const double* a, double* o) {
    // adjugate / determinant (what cv::invert does for 3x3)
    double d = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) +
               a[2] * (a[3] * a[7] - a[4] * a[6]);
    d = (d != 0.0) ? 1.0 / d : 0.0;
    o[0] = (a[4] * a[8] - a[5] * a[7]) * d;
    o[1] = (a[2] * a[7] - a[1] * a[8]) * d;
    o[2] = (a[1] * a[5] - a[2] * a[4]) * d;
    o[3] = (a[5] * a[6] - a[3] * a[8]) * d;
    o[4] = (a[0] * a[8] - a[2] * a[6]) * d;
    o[5] = (a[2] * a[3] - a[0] * a[5]) * d;
    o[6] = (a[3] * a[7] - a[4] * a[6]) * d;
    o[7] = (a[1] * a[6] - a[0] * a[7]) * d;
    o[8] = (a[0] * a[4] - a[1] * a[3]) * d;
}

int lt_launch_build_maps(const lt_camera& c, const LtDims& d, int2* und_map, int2* bv_map, int2* ov_map, cudaStream_t st) {
    UndistortCoef uc;
    invert3x3(c.cam_matrix, uc.iR);
    uc.k1 = c.dist_coeffs[0]; uc.k2 = c.dist_coeffs[1]; uc.p1 = c.dist_coeffs[2];
    uc.p2 = c.dist_coeffs[3]; uc.k3 = c.dist_coeffs[4];
    uc.fx = c.cam_matrix[0]; uc.fy = c.cam_matrix[4]; uc.cx = c.cam_matrix[2]; uc.cy = c.cam_matrix[5];
    dim3 b(256), g1(lt_div_up(d.img_w, 256), d.img_h), g2(lt_div_up(d.bv_w, 256), d.bv_h);
    k_build_undistort_map<<<g1, b, 0, st>>>(und_map, d.img_w, d.img_h, uc);
    LT_LAUNCH_CHECK();
    Mat9 mi;
    invert3x3(c.M, mi.m);
    k_build_perspective_map<<<g2, b, 0, st>>>(bv_map, d.bv_w, d.bv_h, mi);
    LT_LAUNCH_CHECK();
    invert3x3(c.Minv, mi.m);
    k_build_perspective_map<<<g1, b, 0, st>>>(ov_map, d.img_w, d.img_h, mi);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// bilinear sampling helpers (OpenCV remap, INTER_LINEAR, BORDER_CONSTANT 0)
// ---------------------------------------------------------------------------

struct Tap4 {
    int sx, sy, w00, w01, w10, w11;
};

__device__ __forceinline__ Tap4 make_taps(int2 q) {
    Tap4 t;
    int sx = q.x >> 5, sy = q.y >> 5;
    t.sx = max(-32768, min(32767, sx));
    t.sy = max(-32768, min(32767, sy));
    int fx = q.x & 31, fy = q.y & 31;
    t.w00 = (32 - fx) * (32 - fy);
    t.w01 = fx * (32 - fy);
    t.w10 = (32 - fx) * fy;
    t.w11 = fx * fy;
    return t;
}

// ---------------------------------------------------------------------------
// NV12 sampling: cv::cvtColor(COLOR_YUV2RGB_NV12) restated (SURVEY section 8 (f) #2: the reference gets RGB frames from
// moviepy / ffmpeg, process_video.py:42-44; a hardware decoder delivers NV12).  ITU-R BT.601 limited range in Q20 fixed
// point, one chroma sample per 2x2 block, no interpolation (oracle.cvops.yuv2rgb_nv12, pinned against cv2 in
// tests/test_oracle_cvops.py).  Frame layout [img_h * 3 / 2][img_w]: luma plane, then rows of interleaved U, V pairs;
// pixel (y, x) takes luma byte y * W + x and the pair at (H + (y >> 1)) * W + (x & ~1).
// ---------------------------------------------------------------------------

__device__ __forceinline__ uint32_t sat_q20(int v) { return (uint32_t)min(255, max(0, v >> 20)); }

// one luma byte and one chroma pair (U in bits 0-7, V in bits 8-15; higher bits ignored) -> R | G << 8 | B << 16
__device__ __forceinline__ uint32_t yuv_to_rgb(uint32_t luma, uint32_t uv) {
    const int u = (int)(uv & 255u) - 128, v = (int)((uv >> 8) & 255u) - 128;
    const int y = max(0, (int)luma - 16) * 1220542 + (1 << 19);
    return sat_q20(y + 1673527 * v) | (sat_q20(y - 852492 * v - 409993 * u) << 8) | (sat_q20(y + 2116026 * u) << 16);
}

// four pixels of one row: one aligned luma word and the chroma word under it (two U,V pairs) -> the three words of
// their 12 RGB bytes
__device__ __forceinline__ void nv12_to_rgb_words(uint32_t luma, uint32_t uv, uint32_t& w0, uint32_t& w1, uint32_t& w2) {
    uint32_t px[4];                                                    // R | G << 8 | B << 16
#pragma unroll
    for (int i = 0; i < 4; ++i) px[i] = yuv_to_rgb((luma >> (8 * i)) & 255u, uv >> (16 * (i >> 1)));
    w0 = px[0] | (px[1] << 24);
    w1 = (px[1] >> 8) | (px[2] << 16);
    w2 = (px[2] >> 16) | (px[3] << 8);
}

// ---------------------------------------------------------------------------
// undistort: frame rows -> undistorted ROI rows [roi0, roi1), RGBX
// ---------------------------------------------------------------------------

__device__ __forceinline__ uint32_t load_rgb(const uint8_t* __restrict__ img, int w, int h, int y, int x) {
    if ((unsigned)y >= (unsigned)h || (unsigned)x >= (unsigned)w) return 0u;
    const uint8_t* p = img + ((size_t)y * w + x) * 3;
    return (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16);
}

__device__ __forceinline__ uint32_t blend_rgb(uint32_t a, uint32_t b, uint32_t c, uint32_t d, const Tap4& t) {
    uint32_t out = 0;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        int s = 8 * ch;
        int v = (int)((a >> s) & 255) * t.w00 + (int)((b >> s) & 255) * t.w01 +
                (int)((c >> s) & 255) * t.w10 + (int)((d >> s) & 255) * t.w11;
        out |= (uint32_t)((v + 512) >> 10) << s;
    }
    return out;
}

__device__ __forceinline__ uint32_t blend_rgbx(uint32_t t00, uint32_t t01, uint32_t t10, uint32_t t11, uint32_t f);
__device__ __forceinline__ uint32_t blend_taps(uint32_t t00, uint32_t t01, uint32_t t10, uint32_t t11, uint32_t wA, uint32_t wB);
__device__ __forceinline__ void blend_weights(uint32_t f, uint32_t& wA, uint32_t& wB);

// Tap descriptor of every pixel of the undistorted ROI, built once from und_map:
//   x = BYTE offset of tap (sy, sx) in a frame, y = fx | fy << 5 | in-image flags of the four taps << 10 | "fast" << 14.
// fast: all four taps are inside the frame and the three aligned 32-bit words that cover a tap pair lie inside it too.
__global__ void k_build_und_desc(const int2* __restrict__ map, int2* __restrict__ desc, LtDims d) {
    int j = blockIdx.x * blockDim.x + threadIdx.x, i = d.roi0 + blockIdx.y;
    if (j >= d.img_w) return;
    const int2 q = map[(size_t)i * d.img_w + j];
    Tap4 t = make_taps(q);
    auto ok = [&](int yy, int xx) { return (unsigned)yy < (unsigned)d.img_h && (unsigned)xx < (unsigned)d.img_w; };
    uint32_t f = (uint32_t)(q.x & 31) | ((uint32_t)(q.y & 31) << 5);
    const uint32_t m = (ok(t.sy, t.sx) ? 1u : 0u) | (ok(t.sy, t.sx + 1) ? 2u : 0u) | (ok(t.sy + 1, t.sx) ? 4u : 0u) |
                       (ok(t.sy + 1, t.sx + 1) ? 8u : 0u);
    f |= m << 10;
    long long off = ((long long)t.sy * d.img_w + t.sx) * 3;
    const long long frame_bytes = (long long)d.img_w * d.img_h * 3;
    if (m == 15u && ((off + 3LL * d.img_w) & ~3LL) + 12 <= frame_bytes) f |= 1u << 14;
    if (!m) off = 0;
    desc[(size_t)(i - d.roi0) * d.img_w + j] = make_int2((int)off, (int)f);
}

int lt_launch_build_und_desc(const int2* und_map, int2* und_desc, const LtDims& d, cudaStream_t st) {
    dim3 g(lt_div_up(d.img_w, 256), d.roi1 - d.roi0);
    k_build_und_desc<<<g, 256, 0, st>>>(und_map, und_desc, d);
    LT_LAUNCH_CHECK();
    return 0;
}

// Layout of the undistorted ROI ("und") buffer, per group of NSW = 16 streams:
//     word ((r * UP + c) * NSW + s)     r = row - roi0 + 1,  c = column + 1,  UP = img_w + 1,  s = stream within the group
// i.e. STREAM-MINOR (the 16 streams of one pixel are 64 contiguous bytes: a thread that handles one pixel of all the
// streams of a group moves them with 16-byte vectors) and ZERO-BORDERED: column c = 0 of every row (which is also
// column img_w + 1 of the row above), row r = 0 and the two rows below the ROI are never written and stay 0 from the
// allocation.  They are cv2.warpPerspective's BORDER_CONSTANT: a tap outside the frame reads a zero word, so the warp
// needs neither in-image flags nor branches; a pixel with no tap inside the frame points at the two zero rows.
constexpr int NSW = LT_UND_GROUP;      // streams per group

// cv2.undistort of the ROI rows: one thread = one ROI pixel of UND_SPC streams (descriptor decoded once; the 32 lanes of
// a warp read 32 neighbouring pixels of one frame: whole sectors).  The stream-minor output goes through shared memory
// so that a warp stores whole 32-byte sectors.  Fast path: the six bytes of a tap pair come from three aligned 32-bit
// words and two funnel shifts.
constexpr int UND_SPC = 8;             // streams per CTA: 4, 8 or 16 (a CTA covers UND_SPC / 4 of the four 16-byte chunks of a pixel)
constexpr int UND_CH = UND_SPC / 4;
constexpr int UND_MINB = 6;            // resident CTAs per SM the undistort is compiled for
static_assert(UND_SPC == 4 || UND_SPC == 8 || UND_SPC == 16, "streams per CTA");

// rotate the chunk slot with the pixel index: the 16-byte accesses of a quarter warp land in distinct banks
__device__ __forceinline__ int und_slot(int px, int c) { return px * UND_CH + ((c + (px * UND_CH >> 3)) & (UND_CH - 1)); }

// Second half of the undistort kernels: the blended pixels of the CTA (tile, [pixel][chunk of four streams]) go to the
// stream-minor und layout.  The UND_CH chunks of this CTA inside the pixel's 64 bytes: streams s0 .. s0 + UND_SPC - 1
// of group s0 / NSW.
__device__ __forceinline__ void und_store_tile(const uint4* tile, uint32_t* __restrict__ und, int p0, int roi_px, int s0,
                                               const LtDims& d, size_t group_words) {
    uint32_t* const base = und + (size_t)(s0 / NSW) * group_words + (s0 % NSW);
#pragma unroll
    for (int r = 0; r < UND_CH; ++r) {
        const int e = r * 256 + threadIdx.x;           // (pixel, chunk) in output order
        const int px = e / UND_CH, c = e % UND_CH, pp = p0 + px;
        if (pp >= roi_px) break;
        const int i = pp / d.img_w, j = pp - i * d.img_w;
        uint4* out = reinterpret_cast<uint4*>(base + ((size_t)(i + 1) * (d.img_w + 1) + (j + 1)) * NSW);
        out[c] = tile[und_slot(px, c)];
    }
}

// Slots of a camera batch (lt_process_front_cameras): the und buffer (LtFrontSet::und_cam) holds the batch positions
// grouped by camera, each camera's run starting at a multiple of four slots, so that every chunk of four slots (one
// 16-byte vector of a pixel) belongs to one camera.  slot_pos: batch position of each slot (-1: pad, only at the end of
// a run); chunk_cam: camera of each chunk; cams: the snapshot of the camera tables.  Unused by the forms without cameras.
struct LtCamSlots {
    const int* slot_pos;
    const int* chunk_cam;
    const LtCamDev* cams;
};

// The four slots of chunk c of a CTA whose first slot is s0, in a camera batch: the batch positions of their frames and
// the number of slots of the CTA up to the last real one of the chunk (pads are skipped like slots beyond the batch).
__device__ __forceinline__ int cam_chunk_slots(const LtCamSlots& cs, int s0, int c, int ns, int4& pos) {
    pos = __ldg(reinterpret_cast<const int4*>(cs.slot_pos + s0 + 4 * c));
    const int real = (pos.x >= 0) + (pos.y >= 0) + (pos.z >= 0) + (pos.w >= 0);
    return min(ns, 4 * c + real);
}

__device__ __forceinline__ int i4_at(const int4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

// One ROI pixel's tap descriptor q, decoded once for every chunk of streams.
struct UndTap {
    int2 q;
    uint32_t wA, wB, m;
    bool fast;
    int pitch, wi, sh, wpitch;
};

__device__ __forceinline__ UndTap und_tap(int2 q, const LtDims& d) {
    UndTap t;
    t.q = q;
    const uint32_t f = (uint32_t)q.y;
    blend_weights(f, t.wA, t.wB);
    t.m = (f >> 10) & 15u;
    t.fast = f >> 14;                   // word loads: the API refuses frames that are not 4-byte aligned
    t.pitch = d.img_w * 3;
    t.wi = q.x >> 2; t.sh = (q.x & 3) * 8; t.wpitch = t.pitch >> 2;
    return t;
}

// The blended RGBX words of the four streams of chunk c at one ROI pixel (RGB frames): stream k reads the frame at
// frame(k); streams 4c + k >= ns give 0.
template <typename Frame>
__device__ __forceinline__ uint4 und_chunk_rgb(const UndTap& t, int c, int ns, Frame frame) {
    const int2 q = t.q;
    const uint32_t wA = t.wA, wB = t.wB, m = t.m;
    const bool fast = t.fast;
    const int pitch = t.pitch, wi = t.wi, sh = t.sh, wpitch = t.wpitch;
    uint32_t o[4] = {0u, 0u, 0u, 0u};
    if (4 * c < ns) {
        if (fast) {
            // all 24 words of the four streams are requested before the first blend needs one
            uint32_t a[4][3], b[4][3];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                const uint32_t* w = reinterpret_cast<const uint32_t*>(frame(k)) + wi;
                a[k][0] = __ldg(w); a[k][1] = __ldg(w + 1); a[k][2] = __ldg(w + 2);
                b[k][0] = __ldg(w + wpitch); b[k][1] = __ldg(w + wpitch + 1); b[k][2] = __ldg(w + wpitch + 2);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                const uint32_t qa0 = __funnelshift_r(a[k][0], a[k][1], sh), qa1 = __funnelshift_r(a[k][1], a[k][2], sh);     // bytes o..o+3, o+4..o+7
                const uint32_t qb0 = __funnelshift_r(b[k][0], b[k][1], sh), qb1 = __funnelshift_r(b[k][1], b[k][2], sh);
                o[k] = blend_taps(qa0, __funnelshift_r(qa0, qa1, 24), qb0, __funnelshift_r(qb0, qb1, 24), wA, wB);
            }
        } else if (m) {
#pragma unroll 1
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                const uint8_t* img = frame(k);
                auto tap = [&](uint32_t bit, int off) -> uint32_t {     // BORDER_CONSTANT 0
                    if (!(m & bit)) return 0u;
                    const uint8_t* tp = img + q.x + off;
                    return (uint32_t)__ldg(tp) | ((uint32_t)__ldg(tp + 1) << 8) | ((uint32_t)__ldg(tp + 2) << 16);
                };
                o[k] = blend_taps(tap(1u, 0), tap(2u, 3), tap(4u, pitch), tap(8u, pitch + 3), wA, wB);
            }
        }
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// The camera form of both undistort kernels: chunk c of the CTA takes the descriptors and ROI of its own camera.  Its
// pixels below that ROI, down to two rows past it, are written as zeros: the warp reads them (the no-tap index and the
// bottom taps of the last ROI row) and a slot may have held a taller camera's ROI in an earlier batch.  -> the number of
// pixels the store of this thread's chunk (threadIdx.x % UND_CH) covers.
template <typename Chunk>
__device__ __forceinline__ int und_cams_tile(uint4* tile, int p, int s0, int ns, const LtCamSlots& cs, const LtDims& d,
                                             Chunk chunk) {
    int lim_mine = 0;
#pragma unroll
    for (int c = 0; c < UND_CH; ++c) {
        int lim = 0;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (4 * c < ns) {
            const LtCamDev* cd = cs.cams + __ldg(&cs.chunk_cam[s0 / 4 + c]);
            const int roi_px = cd->roi_px;
            lim = roi_px + 2 * d.img_w;
            if (p < roi_px) {
                int4 pos;
                const int nsc = cam_chunk_slots(cs, s0, c, ns, pos);
                o = chunk(__ldg(&cd->und_desc[p]), c, nsc, pos);
            }
        }
        if (c == (int)(threadIdx.x % UND_CH)) lim_mine = lim;
        if (p < lim) tile[und_slot(threadIdx.x, c)] = o;
    }
    return lim_mine;
}

// CAMS: a camera batch (n slots of LtFrontSet::und_cam, tables per chunk from `cs`; `desc` unused).
template <bool CAMS>
__global__ void __launch_bounds__(256, UND_MINB)
k_undistort_roi(const uint8_t* __restrict__ frames, uint32_t* __restrict__ und, const int2* __restrict__ desc, LtDims d, int n,
                size_t group_words, LtCamSlots cs) {
    __shared__ uint4 tile[256 * UND_CH];               // [pixel][chunk of four streams], chunk slot rotated by the pixel
    const int p0 = blockIdx.x * blockDim.x, p = p0 + threadIdx.x;
    if (CAMS) {
        const int s0 = blockIdx.y * UND_SPC, ns = min(UND_SPC, n - s0);
        const size_t frame_bytes = (size_t)d.img_w * d.img_h * 3;
        const int lim = und_cams_tile(tile, p, s0, ns, cs, d, [&](int2 q, int c, int nsc, const int4& pos) {
            return und_chunk_rgb(und_tap(q, d), c, nsc, [&](int k) { return frames + (size_t)i4_at(pos, k) * frame_bytes; });
        });
        __syncthreads();
        und_store_tile(tile, und, p0, lim, s0, d, group_words);
        return;
    }
    const int roi_px = (d.roi1 - d.roi0) * d.img_w;
    const int s0 = blockIdx.y * UND_SPC, ns = min(UND_SPC, n - s0);
    // (the form without cameras keeps its own copy of the tap fetch of und_chunk_rgb: through the helper, ptxas lays
    // out its branches differently, and this form is meant to stay the code it was before cameras)
    if (p < roi_px) {
        const int2 q = __ldg(&desc[p]);
        const uint32_t f = (uint32_t)q.y;
        uint32_t wA, wB;
        blend_weights(f, wA, wB);
        const uint32_t m = (f >> 10) & 15u;
        const bool fast = f >> 14;          // word loads: the API refuses frames that are not 4-byte aligned
        const size_t frame_bytes = (size_t)d.img_w * d.img_h * 3;
        const int pitch = d.img_w * 3;
        const int wi = q.x >> 2, sh = (q.x & 3) * 8, wpitch = pitch >> 2;
#pragma unroll
        for (int c = 0; c < UND_CH; ++c) {
            uint32_t o[4] = {0u, 0u, 0u, 0u};
            if (4 * c < ns) {
                if (fast) {
                    // all 24 words of the four streams are requested before the first blend needs one
                    uint32_t a[4][3], b[4][3];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        const uint32_t* w = reinterpret_cast<const uint32_t*>(frames + (size_t)(s0 + 4 * c + k) * frame_bytes) + wi;
                        a[k][0] = __ldg(w); a[k][1] = __ldg(w + 1); a[k][2] = __ldg(w + 2);
                        b[k][0] = __ldg(w + wpitch); b[k][1] = __ldg(w + wpitch + 1); b[k][2] = __ldg(w + wpitch + 2);
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        const uint32_t qa0 = __funnelshift_r(a[k][0], a[k][1], sh), qa1 = __funnelshift_r(a[k][1], a[k][2], sh);     // bytes o..o+3, o+4..o+7
                        const uint32_t qb0 = __funnelshift_r(b[k][0], b[k][1], sh), qb1 = __funnelshift_r(b[k][1], b[k][2], sh);
                        o[k] = blend_taps(qa0, __funnelshift_r(qa0, qa1, 24), qb0, __funnelshift_r(qb0, qb1, 24), wA, wB);
                    }
                } else if (m) {
#pragma unroll 1
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        const uint8_t* img = frames + (size_t)(s0 + 4 * c + k) * frame_bytes;
                        auto tap = [&](uint32_t bit, int off) -> uint32_t {     // BORDER_CONSTANT 0
                            if (!(m & bit)) return 0u;
                            const uint8_t* tp = img + q.x + off;
                            return (uint32_t)__ldg(tp) | ((uint32_t)__ldg(tp + 1) << 8) | ((uint32_t)__ldg(tp + 2) << 16);
                        };
                        o[k] = blend_taps(tap(1u, 0), tap(2u, 3), tap(4u, pitch), tap(8u, pitch + 3), wA, wB);
                    }
                }
            }
            tile[und_slot(threadIdx.x, c)] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();
    und_store_tile(tile, und, p0, roi_px, s0, d, group_words);
}

// k_undistort_roi of NV12 frames: same descriptor, blend and store; only the tap fetch differs.  The descriptor's byte
// offset 3 (sy W + sx) gives the tap (sy, sx) back (sx = -1 when the left tap column lies outside the frame).  A tap
// outside the frame is RGB 0 (BORDER_CONSTANT applies to the RGB image), not the conversion of YUV (0, 0, 0).
// With all four taps inside, each needed byte or U,V pair comes from an aligned word of its own row (img_w % 4 == 0):
// two luma words and two chroma words per tap row, all requested before the first conversion.  The 32 words of four
// streams in flight need 64 registers: 4 resident CTAs per SM (at the 6 of k_undistort_roi they spill).
constexpr int UND_NV12_MINB = 4;

template <typename Frame>
__device__ __forceinline__ uint4 und_chunk_nv12(int2 q, uint32_t wA, uint32_t wB, int c, int ns, Frame frame, const LtDims& d) {
    const uint32_t f = (uint32_t)q.y;
    const uint32_t m = (f >> 10) & 15u;
    const int W = d.img_w, H = d.img_h;
    const int lo = (m & 5u) ? 0 : 1;                 // left tap column outside the frame: sx = -1
    const int t = q.x / 3 + lo + W;                  // (sy + 1) W + sx + lo >= 0
    const int sy = t / W - 1, sx = t - (sy + 1) * W - lo;
    const int ly = sy * W, cy0 = (H + (sy >> 1)) * W, cy1 = (H + ((sy + 1) >> 1)) * W;     // luma row, chroma rows
    const int xa = sx, xb = sx + 1, ca = sx & ~1, cb = (sx + 1) & ~1;
    uint32_t o[4] = {0u, 0u, 0u, 0u};
    if (4 * c < ns) {
        if (m == 15u) {
            const int sa = 8 * (xa & 3), sb = 8 * (xb & 3), ua = 8 * (ca & 2), ub = 8 * (cb & 2);
            uint32_t y[4][4], uv[4][4];          // [stream][tap], taps 00 01 10 11
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                const uint32_t* w = reinterpret_cast<const uint32_t*>(frame(k));
                y[k][0] = __ldg(w + ((ly + xa) >> 2));     y[k][1] = __ldg(w + ((ly + xb) >> 2));
                y[k][2] = __ldg(w + ((ly + W + xa) >> 2)); y[k][3] = __ldg(w + ((ly + W + xb) >> 2));
                uv[k][0] = __ldg(w + ((cy0 + ca) >> 2));   uv[k][1] = __ldg(w + ((cy0 + cb) >> 2));
                uv[k][2] = __ldg(w + ((cy1 + ca) >> 2));   uv[k][3] = __ldg(w + ((cy1 + cb) >> 2));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                o[k] = blend_taps(yuv_to_rgb((y[k][0] >> sa) & 255u, uv[k][0] >> ua),
                                  yuv_to_rgb((y[k][1] >> sb) & 255u, uv[k][1] >> ub),
                                  yuv_to_rgb((y[k][2] >> sa) & 255u, uv[k][2] >> ua),
                                  yuv_to_rgb((y[k][3] >> sb) & 255u, uv[k][3] >> ub), wA, wB);
            }
        } else if (m) {
#pragma unroll 1
            for (int k = 0; k < 4; ++k) {
                if (4 * c + k >= ns) break;
                const uint8_t* img = frame(k);
                auto tap = [&](uint32_t bit, int lrow, int crow, int x, int cx) -> uint32_t {     // BORDER_CONSTANT 0
                    if (!(m & bit)) return 0u;
                    return yuv_to_rgb(__ldg(img + lrow + x), __ldg(reinterpret_cast<const unsigned short*>(img + crow + cx)));
                };
                o[k] = blend_taps(tap(1u, ly, cy0, xa, ca), tap(2u, ly, cy0, xb, cb), tap(4u, ly + W, cy1, xa, ca),
                                  tap(8u, ly + W, cy1, xb, cb), wA, wB);
            }
        }
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// (the camera form: 3 CTAs per SM; with the chunk's camera and slot positions live as well, 64 registers spill)
template <bool CAMS>
__global__ void __launch_bounds__(256, CAMS ? UND_NV12_MINB - 1 : UND_NV12_MINB)
k_undistort_roi_nv12(const uint8_t* __restrict__ frames, uint32_t* __restrict__ und, const int2* __restrict__ desc, LtDims d,
                     int n, size_t group_words, LtCamSlots cs) {
    __shared__ uint4 tile[256 * UND_CH];
    const int p0 = blockIdx.x * blockDim.x, p = p0 + threadIdx.x;
    if (CAMS) {
        const int s0 = blockIdx.y * UND_SPC, ns = min(UND_SPC, n - s0);
        const size_t frame_bytes = (size_t)d.img_w * (d.img_h + d.img_h / 2);
        const int lim = und_cams_tile(tile, p, s0, ns, cs, d, [&](int2 q, int c, int nsc, const int4& pos) {
            uint32_t wA, wB;
            blend_weights((uint32_t)q.y, wA, wB);
            return und_chunk_nv12(q, wA, wB, c, nsc, [&](int k) { return frames + (size_t)i4_at(pos, k) * frame_bytes; }, d);
        });
        __syncthreads();
        und_store_tile(tile, und, p0, lim, s0, d, group_words);
        return;
    }
    const int roi_px = (d.roi1 - d.roi0) * d.img_w;
    const int s0 = blockIdx.y * UND_SPC, ns = min(UND_SPC, n - s0);
    // (the form without cameras keeps its own copy of the tap fetch of und_chunk_nv12, as k_undistort_roi does)
    if (p < roi_px) {
        const int2 q = __ldg(&desc[p]);
        const uint32_t f = (uint32_t)q.y;
        uint32_t wA, wB;
        blend_weights(f, wA, wB);
        const uint32_t m = (f >> 10) & 15u;
        const int W = d.img_w, H = d.img_h;
        const size_t frame_bytes = (size_t)W * (H + H / 2);
        const int lo = (m & 5u) ? 0 : 1;                 // left tap column outside the frame: sx = -1
        const int t = q.x / 3 + lo + W;                  // (sy + 1) W + sx + lo >= 0
        const int sy = t / W - 1, sx = t - (sy + 1) * W - lo;
        const int ly = sy * W, cy0 = (H + (sy >> 1)) * W, cy1 = (H + ((sy + 1) >> 1)) * W;     // luma row, chroma rows
        const int xa = sx, xb = sx + 1, ca = sx & ~1, cb = (sx + 1) & ~1;
#pragma unroll
        for (int c = 0; c < UND_CH; ++c) {
            uint32_t o[4] = {0u, 0u, 0u, 0u};
            if (4 * c < ns) {
                if (m == 15u) {
                    const int sa = 8 * (xa & 3), sb = 8 * (xb & 3), ua = 8 * (ca & 2), ub = 8 * (cb & 2);
                    uint32_t y[4][4], uv[4][4];          // [stream][tap], taps 00 01 10 11
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        const uint32_t* w = reinterpret_cast<const uint32_t*>(frames + (size_t)(s0 + 4 * c + k) * frame_bytes);
                        y[k][0] = __ldg(w + ((ly + xa) >> 2));     y[k][1] = __ldg(w + ((ly + xb) >> 2));
                        y[k][2] = __ldg(w + ((ly + W + xa) >> 2)); y[k][3] = __ldg(w + ((ly + W + xb) >> 2));
                        uv[k][0] = __ldg(w + ((cy0 + ca) >> 2));   uv[k][1] = __ldg(w + ((cy0 + cb) >> 2));
                        uv[k][2] = __ldg(w + ((cy1 + ca) >> 2));   uv[k][3] = __ldg(w + ((cy1 + cb) >> 2));
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        o[k] = blend_taps(yuv_to_rgb((y[k][0] >> sa) & 255u, uv[k][0] >> ua),
                                          yuv_to_rgb((y[k][1] >> sb) & 255u, uv[k][1] >> ub),
                                          yuv_to_rgb((y[k][2] >> sa) & 255u, uv[k][2] >> ua),
                                          yuv_to_rgb((y[k][3] >> sb) & 255u, uv[k][3] >> ub), wA, wB);
                    }
                } else if (m) {
#pragma unroll 1
                    for (int k = 0; k < 4; ++k) {
                        if (4 * c + k >= ns) break;
                        const uint8_t* img = frames + (size_t)(s0 + 4 * c + k) * frame_bytes;
                        auto tap = [&](uint32_t bit, int lrow, int crow, int x, int cx) -> uint32_t {     // BORDER_CONSTANT 0
                            if (!(m & bit)) return 0u;
                            return yuv_to_rgb(__ldg(img + lrow + x), __ldg(reinterpret_cast<const unsigned short*>(img + crow + cx)));
                        };
                        o[k] = blend_taps(tap(1u, ly, cy0, xa, ca), tap(2u, ly, cy0, xb, cb), tap(4u, ly + W, cy1, xa, ca),
                                          tap(8u, ly + W, cy1, xb, cb), wA, wB);
                    }
                }
            }
            tile[und_slot(threadIdx.x, c)] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();
    und_store_tile(tile, und, p0, roi_px, s0, d, group_words);
}

// cv2.warpPerspective(img, M, warped_size) of the RAW frame (lane_tracker.py:1035, the split view's middle panel)
__global__ void __launch_bounds__(256)
k_warp_frame(const uint8_t* __restrict__ frames, uint8_t* __restrict__ bv_rgb, const int2* __restrict__ map, LtDims d) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, s = blockIdx.z;
    if (x >= d.bv_w) return;
    const uint8_t* img = frames + (size_t)s * d.img_w * d.img_h * 3;
    Tap4 t = make_taps(__ldg(&map[(size_t)y * d.bv_w + x]));
    uint32_t o = blend_rgb(load_rgb(img, d.img_w, d.img_h, t.sy, t.sx), load_rgb(img, d.img_w, d.img_h, t.sy, t.sx + 1),
                           load_rgb(img, d.img_w, d.img_h, t.sy + 1, t.sx), load_rgb(img, d.img_w, d.img_h, t.sy + 1, t.sx + 1), t);
    uint8_t* p = bv_rgb + (((size_t)s * d.bv_h + y) * d.bv_w + x) * 3;
    p[0] = o & 255; p[1] = (o >> 8) & 255; p[2] = (o >> 16) & 255;
}

int lt_launch_warp_frame(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int n, cudaStream_t st) {
    const LtDims& d = h->d;
    k_warp_frame<<<dim3(lt_div_up(d.bv_w, 256), d.bv_h, n), 256, 0, st>>>(d_frames, d_bv_rgb, h->bv_map, d);
    LT_LAUNCH_CHECK();
    return 0;
}

int lt_launch_undistort(lt_handle* h, const uint8_t* d_frames, int n, cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up((d.roi1 - d.roi0) * d.img_w, 256), lt_div_up(n, UND_SPC));
    const LtCamSlots none = {nullptr, nullptr, nullptr};
    // the word loads of the fast path need 4-byte aligned rows: the frames are (lt_api.cu) and img_w % 4 == 0 (lt_create)
    if (h->frame_format == LT_FRAME_NV12)
        k_undistort_roi_nv12<false><<<g, 256, 0, st>>>(d_frames, h->und_roi, h->und_desc, d, n, lt_und_group_words(d), none);
    else
        k_undistort_roi<false><<<g, 256, 0, st>>>(d_frames, h->und_roi, h->und_desc, d, n, lt_und_group_words(d), none);
    LT_LAUNCH_CHECK();
    return 0;
}

// The camera batch: the grid covers the tallest ROI of its cameras plus the two zero rows below it.
int lt_launch_undistort_cams(lt_handle* h, const LtFrontSet& f, const uint8_t* d_frames, int nslots, int max_rows,
                             cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up((max_rows + 2) * d.img_w, 256), lt_div_up(nslots, UND_SPC));
    const LtCamSlots cs = {f.slot_pos, f.chunk_cam, f.cams};
    if (h->frame_format == LT_FRAME_NV12)
        k_undistort_roi_nv12<true><<<g, 256, 0, st>>>(d_frames, f.und_cam, nullptr, d, nslots, lt_und_cam_group_words(h), cs);
    else
        k_undistort_roi<true><<<g, 256, 0, st>>>(d_frames, f.und_cam, nullptr, d, nslots, lt_und_cam_group_words(h), cs);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// warp to the bird's-eye view, emitting the two planes the filter consumes:
// RGB R and CIE-Lab b (lane_tracker.py:207-208), pair-packed
// ---------------------------------------------------------------------------

__device__ __forceinline__ int lab_b(uint32_t rgb, const unsigned short* __restrict__ g,
                                     const unsigned short* __restrict__ cb) {
    int R = __ldg(&g[rgb & 255]), G = __ldg(&g[(rgb >> 8) & 255]), B = __ldg(&g[(rgb >> 16) & 255]);
    int fY = __ldg(&cb[(871 * R + 2929 * G + 296 * B + 2048) >> 12]);
    int fZ = __ldg(&cb[(73 * R + 448 * G + 3575 * B + 2048) >> 12]);
    int b = (200 * (fY - fZ) + 128 * 32768 + 16384) >> 15;
    return max(0, min(255, b));
}

// Per bird's-eye pixel tap descriptor, built once from bv_map: x = pixel index (r * UP + c) of tap (sy, sx) in the
// zero-bordered und layout above, y = fx | fy << 5.  Taps outside the frame fall on zero words of that layout (column 0 /
// row 0 / the rows below the ROI); a pixel without any tap inside the frame points at the two all-zero rows.
__global__ void k_build_bv_desc(const int2* __restrict__ map, int2* __restrict__ desc, LtDims d) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= d.bv_w) return;
    const int2 q = map[(size_t)y * d.bv_w + x];
    Tap4 t = make_taps(q);
    auto ok = [&](int yy, int xx) {
        return (unsigned)yy < (unsigned)d.img_h && (unsigned)xx < (unsigned)d.img_w && yy >= d.roi0 && yy < d.roi1;
    };
    const bool any = ok(t.sy, t.sx) || ok(t.sy, t.sx + 1) || ok(t.sy + 1, t.sx) || ok(t.sy + 1, t.sx + 1);
    const int up = d.img_w + 1, rows = d.roi1 - d.roi0;
    // with a tap inside the frame: sy in [roi0 - 1, roi1 - 1] and sx in [-1, img_w - 1] (the ROI is the hull of such taps)
    const int idx = any ? (t.sy - d.roi0 + 1) * up + (t.sx + 1) : (rows + 1) * up;
    desc[(size_t)y * d.bv_w + x] = make_int2(idx, (int)((uint32_t)(q.x & 31) | ((uint32_t)(q.y & 31) << 5)));
}

int lt_launch_build_desc(const int2* bv_map, int2* bv_desc, const LtDims& d, cudaStream_t st) {
    dim3 g(lt_div_up(d.bv_w, 256), d.bv_h);
    k_build_bv_desc<<<g, 256, 0, st>>>(bv_map, bv_desc, d);
    LT_LAUNCH_CHECK();
    return 0;
}

// bilinear blend of four RGBX taps, separable form: (t00*gx + t01*fx)*gy + (t10*gx + t11*fx)*fy, which is the
// same integer as sum(tap * w) with OpenCV's weights; R and B ride in the two 16-bit halves for the x pass.
__device__ __forceinline__ uint32_t blend_rgbx(uint32_t t00, uint32_t t01, uint32_t t10, uint32_t t11, uint32_t f) {
    const uint32_t fx = f & 31u, fy = (f >> 5) & 31u, gx = 32u - fx, gy = 32u - fy;
    uint32_t rb0 = (t00 & 0x00FF00FFu) * gx + (t01 & 0x00FF00FFu) * fx;      // lanes <= 255*32
    uint32_t rb1 = (t10 & 0x00FF00FFu) * gx + (t11 & 0x00FF00FFu) * fx;
    // G of the two tap rows rides in two 16-bit halves as well (byte 3 of every tap is 0: RGBX / 24-bit values)
    uint32_t g01 = __byte_perm(t00, t10, 0x3531) * gx + __byte_perm(t01, t11, 0x3531) * fx;
    uint32_t R = ((rb0 & 0xFFFFu) * gy + (rb1 & 0xFFFFu) * fy + 512u) >> 10;
    uint32_t B = ((rb0 >> 16) * gy + (rb1 >> 16) * fy + 512u) >> 10;
    uint32_t G = ((g01 & 0xFFFFu) * gy + (g01 >> 16) * fy + 512u) >> 10;
    return R | (G << 8) | (B << 16);
}

// Store one packed column of the two morphology input planes (padded layout, lt_common.cuh): lanes beyond the image
// carry the erosion pad 0xFFFF, and the columns next to the seam are mirrored into the halo of the other strip
// (column -j holds pixel p2 - j in its hi lane, column p2 + j holds pixel p2 + j in its lo lane).
__device__ __forceinline__ void store_padded(uint32_t* __restrict__ planeR, uint32_t* __restrict__ planeB, uint32_t r2,
                                             uint32_t b2, int x, int y, int s, unsigned stream_pad, const LtDims& d) {
    const bool hi_real = x + d.p2 < d.bv_w;
    if (!hi_real) { r2 |= 0xFFFF0000u; b2 |= 0xFFFF0000u; }
    uint32_t* pr = planeR + (size_t)((unsigned)s) * stream_pad;  // per-stream base (one 32x32->64 multiply); offsets below fit 32 bits
    uint32_t* pb = planeB + (size_t)((unsigned)s) * stream_pad;
    const int o = y * d.pp + x;
    pr[o] = r2;
    pb[o] = b2;
    if (x >= d.p2 - LT_HALO_X) {
        pr[o - d.p2] = (r2 << 16) | 0xFFFFu;
        pb[o - d.p2] = (b2 << 16) | 0xFFFFu;
    }
    if (x < LT_HALO_X) {
        pr[o + d.p2] = (r2 >> 16) | 0xFFFF0000u;                // hi lane of a halo column lies beyond the image
        pb[o + d.p2] = (b2 >> 16) | 0xFFFF0000u;
    }
}

// ---- the per-frame warp: one thread = one packed column (two bird's-eye pixels) of the NSW streams of a group -----
// The tap descriptors of the two pixels (8 bytes each from the shared table) are decoded once; the four taps of a pixel
// are fetched for four streams at a time with 16-byte loads from the stream-minor und layout (no flags, no branches:
// out-of-frame taps read its zero border).  The Lab look-up tables live in shared memory in a form that needs two
// 3-input adds instead of six multiplies:
//   YZ[c][v] = { coefY[c] * g[v] (+ 2048 for c = 0),  coefZ[c] * g[v] (+ 2048) }      (lane_tracker.py:208, SURVEY A.3)
struct LabSmem {
    uint2 yz[3][256];
    unsigned short cb[3072];
};

__device__ __forceinline__ void lab_smem_load(LabSmem& L, const uint2* __restrict__ yz, const unsigned short* __restrict__ cb) {
    for (int i = threadIdx.x; i < 768; i += blockDim.x) (&L.yz[0][0])[i] = __ldg(&yz[i]);
    const uint32_t* c32 = reinterpret_cast<const uint32_t*>(cb);
    for (int i = threadIdx.x; i < 1536; i += blockDim.x) reinterpret_cast<uint32_t*>(L.cb)[i] = __ldg(&c32[i]);
}

__device__ __forceinline__ uint32_t lab_b_smem(uint32_t R, uint32_t G, uint32_t B, const LabSmem& L) {
    const uint2 a = L.yz[0][R], b = L.yz[1][G], c = L.yz[2][B];
    const int fY = L.cb[(a.x + b.x + c.x) >> 12], fZ = L.cb[(a.y + b.y + c.y) >> 12];
    // OpenCV saturates this value to 8 bits; over all 2^24 RGB inputs it lies in [20, 223]
    // (tests/test_oracle_cvops.py::test_lab_b_never_saturates), so the clamp is dead code and is not executed here
    return (uint32_t)((200 * (fY - fZ) + 128 * 32768 + 16384) >> 15);
}

__global__ void k_build_lab_yz(const unsigned short* __restrict__ g, uint2* __restrict__ yz) {
    const int v = threadIdx.x;                      // 256 threads
    const uint32_t G = g[v];
    yz[v] = make_uint2(871u * G + 2048u, 73u * G + 2048u);
    yz[256 + v] = make_uint2(2929u * G, 448u * G);
    yz[512 + v] = make_uint2(296u * G, 3575u * G);
}

// bilinear blend of four RGB taps (byte 3 of a tap may hold anything), OpenCV's fixed point (SURVEY A.2):
//   out = (t00*w00 + t01*w01 + t10*w10 + t11*w11 + 512) >> 10,   w = (32-fx)(32-fy), fx(32-fy), (32-fx)fy, fx*fy
// as two IDP.2A (two 16-bit weights x two 8-bit taps + accumulator, FMA pipe) per channel: wA = w00 | w01 << 16 for the
// upper tap row, wB = w10 | w11 << 16 for the lower one; the tap bytes of a row are paired per channel by two PRMT.
__device__ __forceinline__ void blend_taps3(uint32_t t00, uint32_t t01, uint32_t t10, uint32_t t11, uint32_t wA, uint32_t wB,
                                            uint32_t& R, uint32_t& G, uint32_t& B) {
    const uint32_t p0 = __byte_perm(t00, t01, 0x5140), q0 = __byte_perm(t00, t01, 0x0062);    // {R,R',G,G'}, {B,B',.,.}
    const uint32_t p1 = __byte_perm(t10, t11, 0x5140), q1 = __byte_perm(t10, t11, 0x0062);
    R = __dp2a_lo(wB, p1, __dp2a_lo(wA, p0, 512u)) >> 10;
    G = __dp2a_hi(wB, p1, __dp2a_hi(wA, p0, 512u)) >> 10;
    B = __dp2a_lo(wB, q1, __dp2a_lo(wA, q0, 512u)) >> 10;
}

__device__ __forceinline__ uint32_t blend_taps(uint32_t t00, uint32_t t01, uint32_t t10, uint32_t t11, uint32_t wA, uint32_t wB) {
    uint32_t R, G, B;
    blend_taps3(t00, t01, t10, t11, wA, wB, R, G, B);
    return R | (G << 8) | (B << 16);
}

__device__ __forceinline__ void blend_weights(uint32_t f, uint32_t& wA, uint32_t& wB) {
    const uint32_t fx = f & 31u, fy = (f >> 5) & 31u, gx = 32u - fx, gy = 32u - fy;
    wA = gx * gy | (fx * gy) << 16;
    wB = gx * fy | (fx * fy) << 16;
}

__device__ __forceinline__ uint32_t u4_at(const uint4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

constexpr int WARP_ITEMS = 64;        // packed columns per pass of a CTA (x 4 stream chunks = 256 threads)
constexpr int WARP_NB = 8;            // passes per CTA (the Lab tables are loaded once per CTA)
constexpr int WARP_MINB = 4;          // resident CTAs per SM the warp is compiled for

// CAMS: a camera batch, n slots of LtFrontSet::und_cam: the chunk of a thread takes the descriptors of its camera and
// stream k of the chunk writes the planes of batch position slot_pos[s0 + k] (`desc` unused).  Where two cameras meet
// inside a group of 16 slots, the four threads of a column gather from different pixels.  The camera form runs at 3 CTAs
// per SM: with its camera's descriptor pointer and the slot positions, 64 registers spill.
template <bool RGB_OUT, bool CAMS>
__global__ void __launch_bounds__(256, CAMS ? WARP_MINB - 1 : WARP_MINB)
k_warp_planes(const uint32_t* __restrict__ und_all, const int2* __restrict__ desc, uint32_t* __restrict__ planeR,
              uint32_t* __restrict__ planeB, uint8_t* __restrict__ bv_rgb, const uint2* __restrict__ yz,
              const unsigned short* __restrict__ cb, LtDims d, unsigned stream_pad, int n, size_t group_words,
              LtCamSlots cs) {
    __shared__ LabSmem L;
    lab_smem_load(L, yz, cb);
    __syncthreads();
    // thread = (packed column, chunk of four streams): the four threads of a column are neighbours in the warp, so a warp
    // gathers 8 columns x 64 contiguous bytes per tap (every fetched sector fully used) and stores 32 contiguous bytes
    // per stream
    const int c = threadIdx.x & 3, il = threadIdx.x >> 2;
    const int s0 = blockIdx.y * NSW + 4 * c, ns = min(4, n - s0);
    if (ns <= 0) return;
    if (CAMS) desc = cs.cams[__ldg(&cs.chunk_cam[s0 / 4])].bv_desc;
    const int up4 = (d.img_w + 1) * (NSW / 4);                      // one und row in 16-byte units
    const uint4* und = reinterpret_cast<const uint4*>(und_all + (size_t)blockIdx.y * group_words) + c;
    const int total = d.bv_h * d.p2;
    // the descriptors of the next pass are requested while this pass computes (one dependent load less per pass)
    auto load_desc = [&](int item, int2& a, int2& c) {
        if (item >= total) return;
        const int y = item / d.p2, x = item - y * d.p2;
        a = __ldg(&desc[y * d.bv_w + x]);
        c = __ldg(&desc[y * d.bv_w + (x + d.p2 < d.bv_w ? x + d.p2 : x)]);
    };
    int2 nq0 = make_int2(0, 0), nq1 = make_int2(0, 0);
    load_desc(blockIdx.x * WARP_NB * WARP_ITEMS + il, nq0, nq1);
#pragma unroll 1
    for (int b = 0; b < WARP_NB; ++b) {
        const int item = (blockIdx.x * WARP_NB + b) * WARP_ITEMS + il;  // flat (row, packed column)
        if (item >= total) return;
        const int y = item / d.p2, x = item - y * d.p2;
        const bool hi_real = x + d.p2 < d.bv_w;
        const int2 q0 = nq0, q1 = nq1;
        if (b + 1 < WARP_NB) load_desc(item + WARP_ITEMS, nq0, nq1);
        const uint4* t0 = und + (size_t)(unsigned)q0.x * (NSW / 4);
        const uint4* t1 = und + (size_t)(unsigned)q1.x * (NSW / 4);
        // four streams of the four taps of both pixels: 8 x 16 bytes in flight
        const uint4 a00 = __ldg(t0), a01 = __ldg(t0 + NSW / 4), a10 = __ldg(t0 + up4), a11 = __ldg(t0 + up4 + NSW / 4);
        const uint4 b00 = __ldg(t1), b01 = __ldg(t1 + NSW / 4), b10 = __ldg(t1 + up4), b11 = __ldg(t1 + up4 + NSW / 4);
        uint32_t wA0, wB0, wA1, wB1;
        blend_weights((uint32_t)q0.y, wA0, wB0);
        blend_weights((uint32_t)q1.y, wA1, wB1);
        const unsigned o = (unsigned)(y * d.pp + x);
        const bool halo_l = x >= d.p2 - LT_HALO_X, halo_r = x < LT_HALO_X;
        const uint32_t beyond = hi_real ? 0u : 0xFFFF0000u;         // lanes beyond the image: the erosion pad
        uint32_t* pr = planeR + (size_t)(unsigned)s0 * stream_pad + o;
        uint32_t* pb = planeB + (size_t)(unsigned)s0 * stream_pad + o;
#pragma unroll
        for (int k = 0; k < 4; ++k, pr += stream_pad, pb += stream_pad) {
            if (k >= ns) break;
            const int pk = CAMS ? __ldg(&cs.slot_pos[s0 + k]) : 0;
            if (CAMS) {
                if (pk < 0) break;                                      // pads end a camera's run
                pr = planeR + (size_t)(unsigned)pk * stream_pad + o;
                pb = planeB + (size_t)(unsigned)pk * stream_pad + o;
            }
            uint32_t R0, G0, B0, R1, G1, B1;
            blend_taps3(u4_at(a00, k), u4_at(a01, k), u4_at(a10, k), u4_at(a11, k), wA0, wB0, R0, G0, B0);
            blend_taps3(u4_at(b00, k), u4_at(b01, k), u4_at(b10, k), u4_at(b11, k), wA1, wB1, R1, G1, B1);
            // (a pixel without a tap inside the frame is black; Lab b of black = 128 comes out of the tables)
            const uint32_t r2 = R0 | (R1 << 16) | beyond;
            const uint32_t b2 = lab_b_smem(R0, G0, B0, L) | (lab_b_smem(R1, G1, B1, L) << 16) | beyond;
            pr[0] = r2;
            pb[0] = b2;
            if (halo_l) { pr[-d.p2] = (r2 << 16) | 0xFFFFu; pb[-d.p2] = (b2 << 16) | 0xFFFFu; }      // seam-stitched halo columns
            if (halo_r) { pr[d.p2] = (r2 >> 16) | 0xFFFF0000u; pb[d.p2] = (b2 >> 16) | 0xFFFF0000u; }
            if (RGB_OUT) {
                uint8_t* p = bv_rgb + (((size_t)(CAMS ? pk : s0 + k) * d.bv_h + y) * d.bv_w + x) * 3;
                p[0] = R0; p[1] = G0; p[2] = B0;
                if (hi_real) { p += (size_t)d.p2 * 3; p[0] = R1; p[1] = G1; p[2] = B1; }
            }
        }
    }
}

int lt_launch_build_lab_yz(lt_handle* h, cudaStream_t st) {
    k_build_lab_yz<<<1, 256, 0, st>>>(h->lab_gamma, h->lab_yz);
    LT_LAUNCH_CHECK();
    return 0;
}

int lt_launch_warp(lt_handle* h, uint8_t* d_bv_rgb, int n, cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up(d.bv_h * d.p2, WARP_ITEMS * WARP_NB), lt_div_up(n, NSW));
    const LtCamSlots none = {nullptr, nullptr, nullptr};
    if (d_bv_rgb)
        k_warp_planes<true, false><<<g, 256, 0, st>>>(h->und_roi, h->bv_desc, h->planeR, h->planeB, d_bv_rgb, h->lab_yz,
                                                      h->lab_cbrt, d, (unsigned)h->stream_pad, n, lt_und_group_words(d), none);
    else
        k_warp_planes<false, false><<<g, 256, 0, st>>>(h->und_roi, h->bv_desc, h->planeR, h->planeB, nullptr, h->lab_yz,
                                                       h->lab_cbrt, d, (unsigned)h->stream_pad, n, lt_und_group_words(d), none);
    LT_LAUNCH_CHECK();
    return 0;
}

int lt_launch_warp_cams(lt_handle* h, const LtFrontSet& f, int nslots, cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up(d.bv_h * d.p2, WARP_ITEMS * WARP_NB), lt_div_up(nslots, NSW));
    const LtCamSlots cs = {f.slot_pos, f.chunk_cam, f.cams};
    k_warp_planes<false, true><<<g, 256, 0, st>>>(f.und_cam, nullptr, h->planeR, h->planeB, nullptr, h->lab_yz, h->lab_cbrt, d,
                                                  (unsigned)h->stream_pad, nslots, lt_und_cam_group_words(h), cs);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// Fused single-resample variant (BASELINE.json north_star (1), SURVEY.md A.2 (ii)): homography and lens
// distortion composed in fp64, ONE bilinear interpolation straight from the raw frame.  Not bit-exact with the
// two-stage OpenCV pipeline (no intermediate 8-bit rounding); reported separately under a mask-IoU tolerance.
// fused_desc: x = byte index of tap (sy, sx) in the raw frame / 3 (pixel index), y = fx | fy<<5 | flags<<10.
// ---------------------------------------------------------------------------

__global__ void k_build_fused_desc(int2* __restrict__ desc, LtDims d, Mat9 mm, UndistortCoef c) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= d.bv_w) return;
    const double* m = mm.m;
    // undistorted-image coordinates of this bird's-eye pixel (same arithmetic as k_build_perspective_map, unrounded)
    double xb = (double)((x >> 6) << 6), x1 = (double)(x & 63), dy = (double)y;
    double X0 = add64(add64(mul64(m[0], xb), mul64(m[1], dy)), m[2]);
    double Y0 = add64(add64(mul64(m[3], xb), mul64(m[4], dy)), m[5]);
    double W0 = add64(add64(mul64(m[6], xb), mul64(m[7], dy)), m[8]);
    double W = add64(W0, mul64(m[6], x1));
    W = (W != 0.0) ? __ddiv_rn(1.0, W) : 0.0;
    double xu = mul64(add64(X0, mul64(m[0], x1)), W), yu = mul64(add64(Y0, mul64(m[3], x1)), W);
    uint32_t f = 0;
    long long idx = 0;
    if (xu > -1.0 && xu < (double)d.img_w && yu > -1.0 && yu < (double)d.img_h) {
        // distorted (raw-frame) coordinates of that point: the undistort model at a non-integer position
        double _x = add64(add64(mul64(yu, c.iR[1]), c.iR[2]), mul64(xu, c.iR[0]));
        double _y = add64(add64(mul64(yu, c.iR[4]), c.iR[5]), mul64(xu, c.iR[3]));
        double _w = add64(add64(mul64(yu, c.iR[7]), c.iR[8]), mul64(xu, c.iR[6]));
        double px = __ddiv_rn(_x, _w), py = __ddiv_rn(_y, _w);
        double x2 = mul64(px, px), y2 = mul64(py, py), r2 = add64(x2, y2), _2xy = mul64(mul64(2.0, px), py);
        double kr = add64(1.0, mul64(add64(mul64(add64(mul64(c.k3, r2), c.k2), r2), c.k1), r2));
        double xd = add64(add64(mul64(px, kr), mul64(c.p1, _2xy)), mul64(c.p2, add64(r2, mul64(2.0, x2))));
        double yd = add64(add64(mul64(py, kr), mul64(c.p1, add64(r2, mul64(2.0, y2)))), mul64(c.p2, _2xy));
        int U = round_sat_i32(mul64(add64(mul64(c.fx, xd), c.cx), 32.0));
        int V = round_sat_i32(mul64(add64(mul64(c.fy, yd), c.cy), 32.0));
        Tap4 t = make_taps(make_int2(U, V));
        auto ok = [&](int yy, int xx) { return (unsigned)yy < (unsigned)d.img_h && (unsigned)xx < (unsigned)d.img_w; };
        f = (uint32_t)(U & 31) | ((uint32_t)(V & 31) << 5);
        f |= (ok(t.sy, t.sx) ? 1u : 0u) << 10 | (ok(t.sy, t.sx + 1) ? 1u : 0u) << 11 |
             (ok(t.sy + 1, t.sx) ? 1u : 0u) << 12 | (ok(t.sy + 1, t.sx + 1) ? 1u : 0u) << 13;
        if (f >> 10) idx = (long long)t.sy * d.img_w + t.sx;
        else f = 0;
    }
    desc[(size_t)y * d.bv_w + x] = make_int2((int)idx, (int)f);
}

int lt_launch_build_fused_desc(lt_handle* h, cudaStream_t st) {
    const lt_config& c = h->cfg;
    UndistortCoef uc;
    invert3x3(c.cam_matrix, uc.iR);
    uc.k1 = c.dist_coeffs[0]; uc.k2 = c.dist_coeffs[1]; uc.p1 = c.dist_coeffs[2];
    uc.p2 = c.dist_coeffs[3]; uc.k3 = c.dist_coeffs[4];
    uc.fx = c.cam_matrix[0]; uc.fy = c.cam_matrix[4]; uc.cx = c.cam_matrix[2]; uc.cy = c.cam_matrix[5];
    Mat9 mi;
    invert3x3(c.M, mi.m);
    dim3 g(lt_div_up(c.bv_w, 256), c.bv_h);
    k_build_fused_desc<<<g, 256, 0, st>>>(h->fused_desc, h->d, mi, uc);
    LT_LAUNCH_CHECK();
    return 0;
}

__global__ void __launch_bounds__(256)
k_warp_planes_fused(const uint8_t* __restrict__ frames, const int2* __restrict__ desc, uint32_t* __restrict__ planeR,
                    uint32_t* __restrict__ planeB, uint8_t* __restrict__ bv_rgb,
                    const unsigned short* __restrict__ g, const unsigned short* __restrict__ cb, LtDims d, unsigned stream_pad) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y, s = blockIdx.z;
    if (x >= d.p2) return;
    const uint8_t* img = frames + (size_t)s * d.img_w * d.img_h * 3;
    uint32_t r2 = 0, b2 = 0;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        int px = x + half * d.p2;
        if (px < d.bv_w) {
            int2 q = __ldg(&desc[(size_t)y * d.bv_w + px]);
            const uint32_t f = (uint32_t)q.y;
            auto tap = [&](int bit, int off) -> uint32_t {
                if (!(f & (1u << bit))) return 0u;
                const uint8_t* p = img + ((size_t)q.x + off) * 3;
                return (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16);
            };
            uint32_t o = blend_rgbx(tap(10, 0), tap(11, 1), tap(12, d.img_w), tap(13, d.img_w + 1), f);
            r2 |= (o & 255u) << (16 * half);
            b2 |= (uint32_t)lab_b(o, g, cb) << (16 * half);
            if (bv_rgb) {
                uint8_t* p = bv_rgb + (((size_t)s * d.bv_h + y) * d.bv_w + px) * 3;
                p[0] = o & 255; p[1] = (o >> 8) & 255; p[2] = (o >> 16) & 255;
            }
        }
    }
    store_padded(planeR, planeB, r2, b2, x, y, s, stream_pad, d);
}

int lt_launch_warp_fused(lt_handle* h, const uint8_t* d_frames, uint8_t* d_bv_rgb, int n, cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up(d.p2, 256), d.bv_h, n);
    k_warp_planes_fused<<<g, 256, 0, st>>>(d_frames, h->fused_desc, h->planeR, h->planeB, d_bv_rgb, h->lab_gamma,
                                           h->lab_cbrt, d, (unsigned)h->stream_pad);
    LT_LAUNCH_CHECK();
    return 0;
}

// planes from a caller-supplied bird's-eye RGB image (filter_lane_points API, lane_tracker.py:207-208)
__global__ void __launch_bounds__(256)
k_planes_from_bv(const uint8_t* __restrict__ bv_rgb, uint32_t* __restrict__ planeR, uint32_t* __restrict__ planeB,
                 const unsigned short* __restrict__ g, const unsigned short* __restrict__ cb, LtDims d, unsigned stream_pad) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y, s = blockIdx.z;
    if (x >= d.p2) return;
    uint32_t r2 = 0, b2 = 0;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        int px = x + half * d.p2;
        if (px < d.bv_w) {
            const uint8_t* p = bv_rgb + (((size_t)s * d.bv_h + y) * d.bv_w + px) * 3;
            uint32_t o = (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16);
            r2 |= (o & 255) << (16 * half);
            b2 |= (uint32_t)lab_b(o, g, cb) << (16 * half);
        }
    }
    store_padded(planeR, planeB, r2, b2, x, y, s, stream_pad, d);
}

int lt_launch_planes_from_bv(lt_handle* h, const uint8_t* d_bv_rgb, int n, cudaStream_t st) {
    const LtDims& d = h->d;
    dim3 g(lt_div_up(d.p2, 256), d.bv_h, n);
    k_planes_from_bv<<<g, 256, 0, st>>>(d_bv_rgb, h->planeR, h->planeB, h->lab_gamma, h->lab_cbrt, d, (unsigned)h->stream_pad);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// overlay: fillPoly canvas (row spans) -> warpPerspective(Minv) -> addWeighted(1, 0.3)
// Only the G channel can change: the canvas is (0,255,0) (lane_tracker.py:647).
// ---------------------------------------------------------------------------

__device__ __forceinline__ int lane_tap(const int2* __restrict__ rows, const LtDims& d, int y, int x) {
    if ((unsigned)y >= (unsigned)d.bv_h || (unsigned)x >= (unsigned)d.bv_w) return 0;
    int2 r = __ldg(&rows[y]);
    return (x >= r.x && x <= r.y) ? 255 : 0;
}

// Lane overlay of four pixels of frame row y, columns 4q .. 4q + 3, held as three RGB words (12 bytes): only G changes.
// CAMS: position s takes its overlay map and rows from its camera, cams[pos_cam[s]] (`map` unused).
template <bool CAMS>
__device__ __forceinline__ void overlay_words(uint32_t& w0, uint32_t& w1, uint32_t& w2, const int2* __restrict__ map,
                                              const int2* __restrict__ lane_rows, const int4* __restrict__ lane_bbox,
                                              const int* __restrict__ draw, const LtDims& d, int y, int q, int s,
                                              const int* __restrict__ ids, const LtCamDev* __restrict__ cams,
                                              const int* __restrict__ pos_cam) {
    int ov0 = d.ov0, ov1 = d.ov1;
    if (CAMS && draw[s]) {
        const LtCamDev* cd = cams + __ldg(&pos_cam[s]);
        map = cd->ov_map; ov0 = cd->ov0; ov1 = cd->ov1;
    }
    if (draw[s] && y >= ov0 && y < ov1) {
        // Q5 canvas coordinates of the four pixels; most of them cannot reach the polygon: one test against its
        // bounding box (taps of a pixel: columns sx, sx + 1, rows sy, sy + 1) skips the span look-ups
        const int4* mp = reinterpret_cast<const int4*>(map + (size_t)y * d.img_w + q * 4);
        const int4 m01 = __ldg(mp), m23 = __ldg(mp + 1);
        const int sid = ids ? __ldg(&ids[s]) : s;        // the cached polygon belongs to the stream, not the position
        const int4 bb = __ldg(&lane_bbox[sid]);
        const int qx[4] = {m01.x, m01.z, m23.x, m23.z}, qy[4] = {m01.y, m01.w, m23.y, m23.w};
        const int sx_lo = min(min(qx[0], qx[1]), min(qx[2], qx[3])) >> 5, sx_hi = max(max(qx[0], qx[1]), max(qx[2], qx[3])) >> 5;
        const int sy_lo = min(min(qy[0], qy[1]), min(qy[2], qy[3])) >> 5, sy_hi = max(max(qy[0], qy[1]), max(qy[2], qy[3])) >> 5;
        if (sx_hi + 1 >= bb.x && sx_lo <= bb.y && sy_hi + 1 >= bb.z && sy_lo <= bb.w) {
            const int2* rows = lane_rows + (size_t)sid * d.bv_h;
            uint32_t gch[4] = {(w0 >> 8) & 255, w1 & 255, (w1 >> 24) & 255, (w2 >> 16) & 255};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                Tap4 t = make_taps(make_int2(qx[k], qy[k]));
                // the two taps of a canvas row share its [lo, hi] span: two span loads instead of four
                const int2 none = make_int2(1, 0);
                const int2 s0 = ((unsigned)t.sy < (unsigned)d.bv_h) ? __ldg(&rows[t.sy]) : none;
                const int2 s1 = ((unsigned)(t.sy + 1) < (unsigned)d.bv_h) ? __ldg(&rows[t.sy + 1]) : none;
                const int xa = t.sx, xb = t.sx + 1;
                const bool ina = (unsigned)xa < (unsigned)d.bv_w, inb = (unsigned)xb < (unsigned)d.bv_w;
                int v = ((ina && xa >= s0.x && xa <= s0.y) ? t.w00 : 0) + ((inb && xb >= s0.x && xb <= s0.y) ? t.w01 : 0) +
                        ((ina && xa >= s1.x && xa <= s1.y) ? t.w10 : 0) + ((inb && xb >= s1.x && xb <= s1.y) ? t.w11 : 0);
                v = (v * 255 + 512) >> 10;
                if (v) {
                    // cv2.addWeighted(img,1,lane,0.3,0): float32 a + b*0.3f, round half to even, saturate
                    float f = __fadd_rn((float)gch[k], __fmul_rn((float)v, 0.3f));
                    gch[k] = (uint32_t)min(255, __float2int_rn(f));
                }
            }
            w0 = (w0 & 0xFFFF00FFu) | (gch[0] << 8);
            w1 = (w1 & 0x00FFFF00u) | gch[1] | (gch[2] << 24);
            w2 = (w2 & 0xFF00FFFFu) | (gch[3] << 16);
        }
    }
}

template <bool CAMS>
__global__ void __launch_bounds__(256)
k_overlay(const uint8_t* frames, uint8_t* out, const int2* __restrict__ map,
          const int2* __restrict__ lane_rows, const int4* __restrict__ lane_bbox, const int* __restrict__ draw, LtDims d, int row0,
          const int* __restrict__ ids, const LtCamDev* __restrict__ cams, const int* __restrict__ pos_cam) {
    // one thread = 4 pixels = 12 bytes (three aligned 32-bit words); img_w % 4 == 0 is checked at create.
    // `out` may alias `frames` (in-place annotation): every thread reads and writes only its own 12 bytes.
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    int y = row0 + blockIdx.y, s = blockIdx.z;
    int qw = d.img_w >> 2;
    if (q >= qw) return;
    size_t base = (((size_t)s * d.img_h + y) * d.img_w + (size_t)q * 4) * 3;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(frames + base);
    uint32_t w0 = src[0], w1 = src[1], w2 = src[2];
    overlay_words<CAMS>(w0, w1, w2, map, lane_rows, lane_bbox, draw, d, y, q, s, ids, cams, pos_cam);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + base);
    dst[0] = w0; dst[1] = w1; dst[2] = w2;
}

// k_overlay of NV12 frames: one thread converts 4 pixels (one luma word, one chroma word = two U,V pairs) to the three
// RGB words k_overlay reads, blends them the same way and writes them to the RGB output (which cannot alias the input).
template <bool CAMS>
__global__ void __launch_bounds__(256)
k_overlay_nv12(const uint8_t* __restrict__ frames, uint8_t* __restrict__ out, const int2* __restrict__ map,
               const int2* __restrict__ lane_rows, const int4* __restrict__ lane_bbox, const int* __restrict__ draw, LtDims d,
               int row0, const int* __restrict__ ids, const LtCamDev* __restrict__ cams, const int* __restrict__ pos_cam) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = row0 + blockIdx.y, s = blockIdx.z;
    if (q >= (d.img_w >> 2)) return;
    const uint8_t* f = frames + (size_t)s * d.img_w * (d.img_h + d.img_h / 2);
    const uint32_t luma = __ldg(reinterpret_cast<const uint32_t*>(f + (size_t)y * d.img_w) + q);
    const uint32_t uv = __ldg(reinterpret_cast<const uint32_t*>(f + (size_t)(d.img_h + (y >> 1)) * d.img_w) + q);
    uint32_t w0, w1, w2;
    nv12_to_rgb_words(luma, uv, w0, w1, w2);
    overlay_words<CAMS>(w0, w1, w2, map, lane_rows, lane_bbox, draw, d, y, q, s, ids, cams, pos_cam);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + (((size_t)s * d.img_h + y) * d.img_w + (size_t)q * 4) * 3);
    dst[0] = w0; dst[1] = w1; dst[2] = w2;
}

// rows the overlay cannot touch are a plain copy: 16-byte vectors, four in flight per thread
__global__ void __launch_bounds__(256)
k_copy_rows(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t frame_vec, size_t a_vec, size_t b_off,
            size_t b_vec) {
    const size_t total = a_vec + b_vec;
    const uint4* fs = src + (size_t)blockIdx.y * frame_vec;
    uint4* fd = dst + (size_t)blockIdx.y * frame_vec;
    size_t i0 = ((size_t)blockIdx.x * blockDim.x) * 4 + threadIdx.x;
    uint4 v[4];
    size_t idx[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        size_t i = i0 + (size_t)u * blockDim.x;
        idx[u] = i < a_vec ? i : b_off + (i - a_vec);
        if (i < total) v[u] = __ldg(&fs[idx[u]]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
        if (i0 + (size_t)u * blockDim.x < total) fd[idx[u]] = v[u];
}

// k_overlay runs on the rows [ov0, ov1) that the lane overlay can reach (a camera batch: the union over its cameras);
// out of place, the other rows of the output frame are a plain copy of the input.
int lt_launch_overlay(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, const int* d_draw,
                      const int* ids, cudaStream_t st, const LtFrontSet* cf) {
    const LtDims& d = h->d;
    const size_t row_bytes = (size_t)d.img_w * 3, frame_bytes = row_bytes * d.img_h;
    int r0 = cf ? cf->cam_ov0 : d.ov0, r1 = cf ? cf->cam_ov1 : d.ov1;
    if (d_out != d_frames) {
        if (row_bytes % 16 || ((uintptr_t)d_frames | (uintptr_t)d_out) % 16) {
            r0 = 0; r1 = d.img_h;                       // generic path: k_overlay copies every row itself
        } else if (r0 > 0 || r1 < d.img_h) {
            const size_t a_vec = (size_t)r0 * row_bytes / 16, b_off = (size_t)r1 * row_bytes / 16;
            const size_t b_vec = (size_t)(d.img_h - r1) * row_bytes / 16;
            dim3 g((unsigned)((a_vec + b_vec + 1023) / 1024), n);
            k_copy_rows<<<g, 256, 0, st>>>(reinterpret_cast<const uint4*>(d_frames), reinterpret_cast<uint4*>(d_out),
                                            frame_bytes / 16, a_vec, b_off, b_vec);
            LT_LAUNCH_CHECK();
        }
    }
    if (r1 > r0) {
        dim3 g(lt_div_up(d.img_w / 4, 256), r1 - r0, n);
        if (cf)
            k_overlay<true><<<g, 256, 0, st>>>(d_frames, d_out, nullptr, h->lane_rows, h->lane_bbox, d_draw, d, r0, ids, cf->cams,
                                               cf->pos_cam);
        else
            k_overlay<false><<<g, 256, 0, st>>>(d_frames, d_out, h->ov_map, h->lane_rows, h->lane_bbox, d_draw, d, r0, ids,
                                                nullptr, nullptr);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

// ---------------------------------------------------------------------------
// Decoder output -> RGB frames (lt_nv12_to_rgb), and the rows of an NV12 frame that the lane overlay cannot reach.
// HBM-bound: 1.5 bytes in, 3 bytes out per pixel.  One thread = 4 x 2 pixels: two aligned luma words, one chroma word
// (two U,V pairs), six RGB words out.  Only rows [r0, r1) are written: a row range may start or end in the middle of
// a chroma row pair, and the rows outside it belong to another kernel.
// ---------------------------------------------------------------------------

__global__ void __launch_bounds__(256)
k_nv12_to_rgb(const uint8_t* __restrict__ nv12, uint8_t* __restrict__ rgb, int w, int h, int r0, int r1) {
    const int qx = blockIdx.x * blockDim.x + threadIdx.x;            // group of four columns
    const int yp = (r0 >> 1) + blockIdx.y, s = blockIdx.z;             // row pair
    if (qx * 4 >= w) return;
    const uint8_t* f = nv12 + (size_t)s * w * (h + h / 2);
    const uint32_t y0 = __ldg(reinterpret_cast<const uint32_t*>(f + (size_t)(2 * yp) * w) + qx);
    const uint32_t y1 = __ldg(reinterpret_cast<const uint32_t*>(f + (size_t)(2 * yp + 1) * w) + qx);
    const uint32_t uv = __ldg(reinterpret_cast<const uint32_t*>(f + (size_t)(h + yp) * w) + qx);   // U0 V0 U1 V1
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int row = 2 * yp + r;
        if (row < r0 || row >= r1) continue;
        uint32_t* o = reinterpret_cast<uint32_t*>(rgb + (((size_t)s * h + row) * w + (size_t)qx * 4) * 3);
        nv12_to_rgb_words(r ? y1 : y0, uv, o[0], o[1], o[2]);
    }
}

int lt_launch_nv12_to_rgb(const uint8_t* d_nv12, uint8_t* d_rgb, int n, int w, int h, int r0, int r1, cudaStream_t st) {
    if (r1 <= r0) return 0;
    dim3 g(lt_div_up(w / 4, 256), (r1 + 1) / 2 - r0 / 2, n);
    k_nv12_to_rgb<<<g, 256, 0, st>>>(d_nv12, d_rgb, w, h, r0, r1);
    LT_LAUNCH_CHECK();
    return 0;
}

// The annotated RGB frames of NV12 input: k_overlay_nv12 on the rows the overlay can reach, the converter on the others.
int lt_launch_overlay_nv12(lt_handle* h, const uint8_t* d_frames, uint8_t* d_out, int n, const int* d_draw,
                           const int* ids, cudaStream_t st, const LtFrontSet* cf) {
    const LtDims& d = h->d;
    const int r0 = cf ? cf->cam_ov0 : d.ov0, r1 = cf ? cf->cam_ov1 : d.ov1;
    int rc;
    if ((rc = lt_launch_nv12_to_rgb(d_frames, d_out, n, d.img_w, d.img_h, 0, r0, st))) return rc;
    if ((rc = lt_launch_nv12_to_rgb(d_frames, d_out, n, d.img_w, d.img_h, r1, d.img_h, st))) return rc;
    if (r1 > r0) {
        dim3 g(lt_div_up(d.img_w / 4, 256), r1 - r0, n);
        if (cf)
            k_overlay_nv12<true><<<g, 256, 0, st>>>(d_frames, d_out, nullptr, h->lane_rows, h->lane_bbox, d_draw, d, r0, ids,
                                                    cf->cams, cf->pos_cam);
        else
            k_overlay_nv12<false><<<g, 256, 0, st>>>(d_frames, d_out, h->ov_map, h->lane_rows, h->lane_bbox, d_draw, d, r0, ids,
                                                     nullptr, nullptr);
        LT_LAUNCH_CHECK();
    }
    return 0;
}
