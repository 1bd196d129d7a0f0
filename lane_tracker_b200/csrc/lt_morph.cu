// Ellipse erosion / dilation / top-hat (cv2.morphologyEx with cv2.getStructuringElement(MORPH_ELLIPSE), lane_tracker.py:203-211)
// on pair-packed planes: the dominant cost of the whole path.
//
//   out(y, x) = op_{dy in [-R, R]} Hop_{hw[dy]}(y + dy, x)          (row-span decomposition, SURVEY.md A.4)
//
// Hop_w = horizontal window min/max of half-width w, taken from power-of-two window tables (T8, T16, T32) with two
// look-ups; the vertical combination is a K-deep register pipeline that advances two rows per step with one
// VIMNMX3.U16x2 per stage.  Measured on B200 (tools/pipe_probe.cu): VIMNMX(3).U16x2, HMNMX2 and PRMT share ONE
// half-rate pipe (2 warp-instructions / clock / SM), shared memory delivers one 128-byte wavefront per clock per SM,
// and this kernel needs about as many cycles of either -- so its speed is decided by how densely those two are kept
// busy.  Hence the WARP-SPECIALISED layout of this file:
//
//   * CTA = 6 consumer warps (192 packed columns, one per thread) + 2 producer warps, one tile x one row band.
//   * Producers stage 8 source rows at a time (one TMA bulk-tensor copy per block from the padded plane's tensor map),
//     build the byte-packed window tables of the 4 row pairs (T1 = the rows themselves, T4 -> T8, T16, T32) into one
//     of TWO table buffers and signal "full"; consumers walk a buffer and signal "empty".  Named barriers (bar.sync /
//     bar.arrive) only: a consumer never waits at a CTA-wide barrier and never executes a table build, a producer
//     never walks.
//   * The 55x55 (Lab-b) and the 29x29 (R) structuring elements are separate kernels with their own register budgets
//     (2 resp. 3 CTAs per SM) launched on two streams, so the lighter one fills the SM slots the heavy one leaves.
//   * A consumer derives the distinct Hop_w lazily in width order and feeds stages j and K-2-j (the ellipse is
//     symmetric: they need the same two widths) right away, ping-ponging between two register copies of the pipeline,
//     so only ~4 window values are live next to the K accumulators: no spills (round 1: 92 bytes of spill stores).
//
// Table words are byte packed {a.lo, b.lo, a.hi, b.hi} (a, b = the two rows of a pair; lo, hi = the two image strips
// of the pair plane): one LDS.32 serves 2 rows x 2 pixels.  Arithmetic runs on 16-bit lanes at "scale 256": a lane is
// value << 8 | junk, ordered by its value byte; row b's lanes are the table word as loaded, row a's the word shifted
// left by 8 (IMAD.SHL, on the FMA pipe); the junk byte is dropped when a result is stored.
#include <cstdlib>
#include <cstdio>
#include <algorithm>
#include <functional>
#include <vector>
#include <map>
#include <mutex>
#include <tuple>
#include "lt_common.cuh"
#include "lt_ellipse.cuh"
#include "lt_tma.cuh"

namespace {

constexpr int TW = 192;             // packed columns per CTA = consumer threads
constexpr int NPW = 2;              // producer warps
constexpr int UNROLL4 = 4, UNROLL8 = 4;   // unroll factors of the producers' task loops
constexpr int NPROD = 32 * NPW;
constexpr int NTHREADS = TW + NPROD;
constexpr int RB = 8, RP = RB / 2;  // source rows / row pairs per table build

// named barriers (0 is __syncthreads)
constexpr int BAR_FULL = 1, BAR_EMPTY = 3, BAR_PROD = 5;

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

template <bool IS_MAX> __device__ __forceinline__ uint32_t op2(uint32_t a, uint32_t b) { return IS_MAX ? __vmaxu2(a, b) : __vminu2(a, b); }
template <bool IS_MAX> __device__ __forceinline__ uint32_t op3(uint32_t a, uint32_t b, uint32_t c) {
    return IS_MAX ? __vimax3_u16x2(a, b, c) : __vimin3_u16x2(a, b, c);
}

template <int K> struct Geo {
    using E = Ellipse<K>;
    static constexpr int R = E::R;
    static constexpr int HA = (R + 3) & ~3;            // staged halo columns per side (16-byte granular)
    static constexpr int TE = TW + 2 * HA;             // staged / tabulated columns; column i <-> packed column x0 - HA + i
    static constexpr int TEA = TE + 32;                // table row pitch: slack for the window reads of the last columns
    static constexpr bool HAS32 = (2 * R + 1) >= 32;
    static constexpr int NCT = HAS32 ? 4 : 3;          // consumer-visible tables: T1, T8, T16 (, T32)
    static constexpr int CH = TE / 4;                  // 16-byte chunks (4 columns) per row
    static constexpr int TBUF = NCT * RP * TEA;        // words per table buffer
    static constexpr int TEP = TE + 4;                 // raw row pitch: slack read by the last T4 chunk
    static constexpr int PRIV = RP * TEA + 2 * RB * TEP;   // producer-private words: T4[RP][TEA], RAW[2][RB][TEP]
    static constexpr int OGW = 2 * RB * TW;            // words of the two original-row buffers of the top-hat epilogue
    static constexpr size_t smem(bool tophat) { return (size_t)(2 * TBUF + PRIV + (tophat ? OGW : 0)) * sizeof(uint32_t) + 32; }   // + four mbarriers
    static_assert((2 * TBUF + RP * TEA) % 32 == 0 && (RB * TEP) % 32 == 0 && TE <= 256, "the raw row buffers must be 128-byte aligned for the TMA copies");
    static_assert((2 * TBUF + PRIV) % 32 == 0 && (RB * TW) % 32 == 0, "so must the original-row buffers");
    static_assert(HA >= R && HA <= LT_HALO_X && R + RB <= LT_HALO_Y && TE % 4 == 0, "staging must be 16-byte granular and inside the plane padding");
};

// One pair step of the vertical pipeline, out of place (S -> D): the caller ping-pongs two register arrays, so the
// stages can be visited in ANY order -- here (0, K-2), (1, K-3), ... which needs the distinct widths one after the other.
//   D[j]   = op3(S[j+2], Ha[hw(j+1)], Hb[hw(j)])      j = 0 .. K-3
//   D[K-2] = op2(Ha[hw(K-1)], Hb[hw(K-2)]),  D[K-1] = Hb[hw(K-1)],  out_a = op2(S[1], Ha[hw(0)])
// After the step, out_a and D[0] are the finished output rows (source row a - R) and (source row b - R).
template <int K, bool IS_MAX>
__device__ __forceinline__ void pair_step(const uint32_t (&S)[K], uint32_t (&D)[K], uint32_t& out_a, const uint32_t* __restrict__ T,
                                          int base) {
    using G = Geo<K>;
    using E = Ellipse<K>;
    constexpr int TS = RP * G::TEA;                    // words between the tables of one buffer
    auto H = [&](int w, uint32_t& ha, uint32_t& hb) {  // Hop_w of rows a (ha) and b (hb) at this thread's column, scale 256
        const int len = 2 * w + 1;
        if (w == 0) { const uint32_t t = T[base]; ha = t << 8; hb = t; return; }
        const uint32_t* tab = len >= 32 ? T + 3 * TS : (len >= 16 ? T + 2 * TS : T + TS);
        const int k = len >= 32 ? 32 : (len >= 16 ? 16 : 8);
        const uint32_t l = tab[base - w], r = tab[base + w - k + 1];
        ha = op2<IS_MAX>(l << 8, r << 8);
        hb = op2<IS_MAX>(l, r);
    };
    uint32_t a0, b0, a1, b1;                           // widths hw(j) and hw(j+1)
    H(E::hw(0), a0, b0);
    out_a = op2<IS_MAX>(S[1], a0);
    D[K - 1] = b0;
#pragma unroll
    for (int j = 0; j <= (K - 3) / 2; ++j) {
        if (E::hw(j + 1) != E::hw(j)) H(E::hw(j + 1), a1, b1); else { a1 = a0; b1 = b0; }
        D[j] = op3<IS_MAX>(S[j + 2], a1, b0);
        const int q = K - 2 - j;                       // mirror stage: widths hw(q+1) = hw(j), hw(q) = hw(j+1)
        if (q != j) {
            if (q + 2 < K) D[q] = op3<IS_MAX>(S[q + 2], a0, b1);
            else D[q] = op2<IS_MAX>(a0, b1);
        }
        a0 = a1; b0 = b1;
    }
}

struct MorphArgs {
    uint32_t* dst;                                                // padded plane (pitch d.pp), stream 0; the sources come as tensor maps
    int bands, band_rows, tiles, n;
    size_t stride;                                                // words per stream
    const int* list; const int* count;
};

// Resident CTAs per SM each kernel is compiled for (register budget): two for 55x55, three for 29x29; three / four were
// measured slower (spills, DESIGN.md section 4).
template <int K, bool IS_MAX, bool TOPHAT>
__global__ void __launch_bounds__(NTHREADS, K == 55 ? 2 : 3)
k_morph(MorphArgs a, LtDims d, const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap omap) {
    using G = Geo<K>;
    using E = Ellipse<K>;
    constexpr int R = G::R, HA = G::HA, TEA = G::TEA;
    constexpr uint32_t PADL = IS_MAX ? 0u : 0xFFFFu, PAD2 = PADL | (PADL << 16);

    int item = blockIdx.x;
    const int slot = item % a.n;               // stream slot fastest: neighbouring CTAs read neighbouring rows of the shared maps
    item /= a.n;
    const int tile = item % a.tiles, band = item / a.tiles;
    if (a.count != nullptr && slot >= *a.count) return;
    const int s = a.list ? a.list[slot] : slot;
    uint32_t* dst = a.dst + (size_t)s * a.stride;
    const int pitch = d.pp;

    extern __shared__ __align__(128) uint32_t smem[];
    uint32_t* const TB = smem;                          // [2 buffers][NCT tables][RP pairs][TEA]
    uint32_t* const T4 = smem + 2 * G::TBUF;            // [RP][TEA]            producer private
    uint32_t* const RAW = T4 + RP * TEA;                // [2 buffers][RB][TEP] producer private
    uint32_t* const OG = RAW + 2 * RB * G::TEP;         // [2 buffers][RB][TW]  original rows of the top-hat epilogue
    uint64_t* const mbar = reinterpret_cast<uint64_t*>(smem + 2 * G::TBUF + G::PRIV + (TOPHAT ? G::OGW : 0));   // [4]: raw rows, original rows

    const int x0 = tile * TW;
    const int yb0 = band * a.band_rows;
    const int yb1 = min(yb0 + a.band_rows, d.bv_h);
    // source rows r_begin, r_begin + 1 complete output rows r_begin - R, r_begin - R + 1: with an even band start the
    // output rows come out in aligned pairs (yb0, yb0 + 1), (yb0 + 2, ...) after R warm-up steps
    const int r_begin = yb0 - R;
    const int r_end = yb1 + R;                          // exclusive
    const int nblk = (r_end - r_begin + RB - 1) / RB;

    // Roles: warps 0-5 (threads 0 .. TW - 1) are the consumers, thread = packed column within the tile; warps 6-7 are
    // the producers.
    const int tid = threadIdx.x;

    if (tid >= TW) {
        // ================================================================= producers
        const int pt = tid - TW;
        // ONE producer thread requests the whole 8-row block (box TE x RB of the plane's tensor map, rows dense in shared
        // memory, TE apart) and every producer waits on the buffer's mbarrier
        constexpr int TE = G::TE;
        constexpr unsigned BLOCK_BYTES = RB * TE * sizeof(uint32_t);
        const int tx = LT_HALO_X + x0 - HA;              // box origin in the padded plane: column ...
        int ty = s * (d.bv_h + 2 * LT_HALO_Y) + LT_HALO_Y + r_begin;     // ... and row (advances RB per block)
        auto stage = [&](int buf) {
            if (pt == 0) {
                fence_proxy_async();                     // the generic-proxy reads of this buffer are ordered before the bulk copy
                mbar_expect_tx(&mbar[buf], BLOCK_BYTES);
                tma_load_2d(RAW + buf * RB * G::TEP, &tmap, tx, ty, &mbar[buf]);
            }
            ty += RB;
        };
        // ... and the original rows of the block's OUTPUT rows (source rows - R) for the top-hat epilogue (box TW x RB of
        // the original plane's map, columns of the tile itself; rows outside the plane are pad rows of the layout and
        // are never emitted)
        const int ox = LT_HALO_X + x0;
        int oyt = s * (d.bv_h + 2 * LT_HALO_Y) + LT_HALO_Y + r_begin - R;
        auto stage_orig = [&](int buf) {
            if (pt == 0) {
                fence_proxy_async();
                mbar_expect_tx(&mbar[2 + buf], (unsigned)(RB * TW * sizeof(uint32_t)));
                tma_load_2d(OG + buf * RB * TW, &omap, ox, oyt, &mbar[2 + buf]);
            }
            oyt += RB;
        };
        if (pt == 0) {
            mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); mbar_init(&mbar[2], 1); mbar_init(&mbar[3], 1);
            mbar_init_fence();
        }
        bar_sync(BAR_PROD, NPROD);
        stage(0);
        for (int blk = 0; blk < nblk; ++blk) {
            const int b = blk & 1;
            mbar_wait(&mbar[b], (unsigned)(blk >> 1) & 1u);
            bar_sync(BAR_PROD, NPROD);                   // rows of this block landed; everybody is done with T4 and RAW[b ^ 1]
            if (blk + 1 < nblk) stage(b ^ 1);            // next block's rows: in flight during the whole build
            if (blk >= 2) bar_sync(BAR_EMPTY + b, NTHREADS);     // the consumers have left table buffer b (and OG[b])
            if (TOPHAT) stage_orig(b);                   // lands during the build (waited for before "full" is signalled)
            uint32_t* const Tb = TB + b * G::TBUF;
            const uint32_t* const Rw = RAW + b * RB * G::TEP;
            // ---- T1 (the rows themselves) and T4, four consecutive columns per task
            constexpr int NTASK = RP * G::CH, NIT = (NTASK + NPROD - 1) / NPROD;
#pragma unroll UNROLL4
            for (int it = 0; it < NIT; ++it) {
                const int q = pt + it * NPROD;
                if (q >= NTASK) break;
                const int pr = q / G::CH, c = (q - pr * G::CH) * 4;
                const uint4* ra = reinterpret_cast<const uint4*>(Rw + (2 * pr) * TE + c);
                const uint4* rb = reinterpret_cast<const uint4*>(Rw + (2 * pr + 1) * TE + c);
                const uint4 a0 = ra[0], a1 = ra[1], b0 = rb[0], b1 = rb[1];
                // raw lanes are plain values (or the 16-bit pad): their low bytes are the table bytes
                uint4 t1;
                t1.x = __byte_perm(a0.x, b0.x, 0x6240); t1.y = __byte_perm(a0.y, b0.y, 0x6240);
                t1.z = __byte_perm(a0.z, b0.z, 0x6240); t1.w = __byte_perm(a0.w, b0.w, 0x6240);
                *reinterpret_cast<uint4*>(Tb + pr * TEA + c) = t1;
                auto win4 = [](const uint4& u, const uint4& v, uint32_t (&e)[4]) {      // min/max over 4 consecutive columns
                    const uint32_t m01 = op2<IS_MAX>(u.x, u.y), m23 = op2<IS_MAX>(u.z, u.w), m45 = op2<IS_MAX>(v.x, v.y);
                    e[0] = op2<IS_MAX>(m01, m23);
                    e[1] = op3<IS_MAX>(u.y, m23, v.x);
                    e[2] = op2<IS_MAX>(m23, m45);
                    e[3] = op3<IS_MAX>(u.w, m45, v.z);
                };
                uint32_t ea[4], eb[4];
                win4(a0, a1, ea);
                win4(b0, b1, eb);
                uint4 t4;
                t4.x = __byte_perm(ea[0], eb[0], 0x6240); t4.y = __byte_perm(ea[1], eb[1], 0x6240);
                t4.z = __byte_perm(ea[2], eb[2], 0x6240); t4.w = __byte_perm(ea[3], eb[3], 0x6240);
                *reinterpret_cast<uint4*>(T4 + pr * TEA + c) = t4;
            }
            bar_sync(BAR_PROD, NPROD);
            // ---- T8, T16 and (HAS32) T32 from T4: entry i = op over T4[i + 4k]; T32 takes 8 vector loads and 13 min/max-pipe
            // operations per entry
#pragma unroll UNROLL8
            for (int it = 0; it < NIT; ++it) {
                const int q = pt + it * NPROD;
                if (q >= NTASK) break;
                const int pr = q / G::CH, c = (q - pr * G::CH) * 4;
                const uint4* t = reinterpret_cast<const uint4*>(T4 + pr * TEA + c);
                uint4 v[G::HAS32 ? 8 : 4];
#pragma unroll
                for (int k = 0; k < (G::HAS32 ? 8 : 4); ++k) v[k] = t[k];
                uint32_t o8[4], o16[4], o32[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    auto w = [&](int k) { const uint4& u = v[k]; return e == 0 ? u.x : (e == 1 ? u.y : (e == 2 ? u.z : u.w)); };
                    const uint32_t a8 = op2<IS_MAX>(w(0) << 8, w(1) << 8), b8 = op2<IS_MAX>(w(0), w(1));
                    const uint32_t a16 = op3<IS_MAX>(a8, w(2) << 8, w(3) << 8), b16 = op3<IS_MAX>(b8, w(2), w(3));
                    o8[e] = __byte_perm(a8, b8, 0x7351);          // value bytes back to {a.lo, b.lo, a.hi, b.hi}
                    o16[e] = __byte_perm(a16, b16, 0x7351);
                    if (G::HAS32) {
                        const uint32_t a32 = op3<IS_MAX>(a16, op2<IS_MAX>(w(4) << 8, w(5) << 8), op2<IS_MAX>(w(6) << 8, w(7) << 8));
                        const uint32_t b32 = op3<IS_MAX>(b16, op2<IS_MAX>(w(4), w(5)), op2<IS_MAX>(w(6), w(7)));
                        o32[e] = __byte_perm(a32, b32, 0x7351);
                    }
                }
                uint32_t* o = Tb + RP * TEA + pr * TEA + c;
                *reinterpret_cast<uint4*>(o) = make_uint4(o8[0], o8[1], o8[2], o8[3]);
                *reinterpret_cast<uint4*>(o + RP * TEA) = make_uint4(o16[0], o16[1], o16[2], o16[3]);
                if (G::HAS32) *reinterpret_cast<uint4*>(o + 2 * RP * TEA) = make_uint4(o32[0], o32[1], o32[2], o32[3]);
            }
            if (TOPHAT) mbar_wait(&mbar[2 + b], (unsigned)(blk >> 1) & 1u);     // OG[b] has landed
            bar_arrive(BAR_FULL + b, NTHREADS);
        }
        return;
    }

    // ===================================================================== consumers
    const int gx = x0 + tid;                       // this thread's packed column
    const bool col_ok = gx < d.p2;
    // scale 256 -> plain values; the hi lane of columns beyond the image is forced to 0 (the pad of the dilation that
    // consumes an eroded plane / a top-hat of nothing)
    const bool hi_real = gx + d.p2 < d.bv_w;
    const uint32_t sel_out = hi_real ? 0x4341u : 0x4441u;
    const uint32_t lane_mask = hi_real ? 0xFFFFFFFFu : 0x0000FFFFu;
    // halo copy for the pass that reads a padded dst (pad 0): column gx - p2 = {0, v.lo}, column gx + p2 = {v.hi, 0}
    int hoff = 0;
    uint32_t hsel = 0;
    if (!TOPHAT && col_ok) {
        if (gx >= d.p2 - LT_HALO_X) { hoff = -d.p2; hsel = 0x1044u; }
        else if (gx < LT_HALO_X) { hoff = d.p2; hsel = 0x4432u; }
    }
    uint32_t* dp = dst + (ptrdiff_t)(r_begin - R) * pitch + gx;            // output row of the first pair step

    uint32_t A[K], B[K];
#pragma unroll
    for (int j = 0; j < K; ++j) A[j] = PAD2;

    int ya = r_begin - R;                          // output row of the next pair step (row a)
    for (int blk = 0; blk < nblk; ++blk) {
        const int b = blk & 1;
        bar_sync(BAR_FULL + b, NTHREADS);
        const uint32_t* const Tb = TB + b * G::TBUF;
        if (col_ok) {
            int base = tid + HA;
            const uint32_t* ogp = OG + b * RB * TW + tid;
#pragma unroll
            for (int m = 0; m < RP; m += 2) {
#pragma unroll
                for (int h = 0; h < 2; ++h, base += TEA, ya += 2, dp += 2 * (ptrdiff_t)pitch, ogp += 2 * TW) {
                    uint32_t out_a, out_b;
                    if (h == 0) { pair_step<K, IS_MAX>(A, B, out_a, Tb, base); out_b = B[0]; }
                    else { pair_step<K, IS_MAX>(B, A, out_a, Tb, base); out_b = A[0]; }
                    if (ya < yb0 || ya >= yb1) continue;
                    uint32_t va = __byte_perm(out_a, 0, sel_out), vb = __byte_perm(out_b, 0, sel_out);
                    if (TOPHAT) { va = (ogp[0] - va) & lane_mask; vb = (ogp[TW] - vb) & lane_mask; }   // open <= src per lane: no borrow
                    const bool eb = ya + 1 < yb1;
                    dp[0] = va;
                    if (eb) dp[pitch] = vb;
                    if (!TOPHAT && hsel) {                                 // seam-stitched halo copies for the next pass
                        dp[hoff] = __byte_perm(va, 0, hsel);
                        if (eb) dp[hoff + pitch] = __byte_perm(vb, 0, hsel);
                    }
                }
            }
        } else {
            ya += 2 * RP;
        }
        if (blk + 2 < nblk) bar_arrive(BAR_EMPTY + b, NTHREADS);
    }
}

template <int K, bool IS_MAX, bool TOPHAT>
int launch_one(lt_handle* h, const uint32_t* src, uint32_t* dst, const uint32_t* orig, int bands, int n, const int* list,
               const int* count, cudaStream_t st) {
    const LtDims& d = h->d;
    MorphArgs a;
    a.dst = dst;
    a.band_rows = (lt_div_up(d.bv_h, bands) + 1) & ~1;          // even: output rows come out in aligned pairs
    a.bands = lt_div_up(d.bv_h, a.band_rows);
    a.tiles = lt_div_up(d.p2, TW);
    a.n = n; a.stride = h->stream_pad; a.list = list; a.count = count;
    CUtensorMap tm, om = {};                                     // om: original rows, top-hat only
    int rc;
    if ((rc = lt_plane_tensor_map(h, src, Geo<K>::TE, &tm))) return rc;
    if (TOPHAT && (rc = lt_plane_tensor_map(h, orig, TW, &om))) return rc;
    if ((rc = lt_ensure_smem((const void*)k_morph<K, IS_MAX, TOPHAT>, Geo<K>::smem(TOPHAT)))) return rc;
    k_morph<K, IS_MAX, TOPHAT><<<n * a.tiles * a.bands, NTHREADS, Geo<K>::smem(TOPHAT), st>>>(a, d, tm, om);
    LT_LAUNCH_CHECK();
    return 0;
}

}  // namespace

// The encoder comes from the driver through cudaGetDriverEntryPoint (no -lcuda).
int lt_plane_tensor_map(lt_handle* h, const uint32_t* plane, int box_w, CUtensorMap* out) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    static std::mutex mu;
    static std::map<std::tuple<int, const void*, int, long long, int>, CUtensorMap> cache;
    std::lock_guard<std::mutex> lock(mu);
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
            lt_set_error("cuTensorMapEncodeTiled is not available");
            return -2;
        }
        encode = (EncodeFn)fn;
    }
    const LtDims& d = h->d;
    const uint32_t* base = plane - ((size_t)LT_HALO_Y * d.pp + LT_HALO_X);          // start of the allocation
    const long long rows = (long long)h->S * (d.bv_h + 2 * LT_HALO_Y) + 1;
    const auto key = std::make_tuple(h->cfg.device, (const void*)base, d.pp, rows, box_w);
    auto it = cache.find(key);
    if (it == cache.end()) {
        CUtensorMap m;
        const cuuint64_t dims[2] = {(cuuint64_t)d.pp, (cuuint64_t)rows};
        const cuuint64_t strides[1] = {(cuuint64_t)d.pp * sizeof(uint32_t)};
        const cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)RB}, estr[2] = {1, 1};
        CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { lt_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return -2; }
        it = cache.emplace(key, m).first;
    }
    *out = it->second;
    return 0;
}

// Band counts of the two jobs: simulate list scheduling of both grids (55x55 CTAs first, they are the long ones) on
// the CTA slots of the device.  Per-row costs: measured relative walk costs of the two structuring elements.
static void choose_bands(lt_handle* h, int n, int tiles, int H, int* b55, int* b29) {
    const int sms = h->sm_count > 0 ? h->sm_count : 148;
    if (h->bands_key[0] == n && h->bands_key[1] == H && h->bands_key[2] == sms) { *b55 = h->bands_val[0]; *b29 = h->bands_val[1]; return; }
    int c55 = 1, c29 = 1;
    bool fixed = false;
    if (const char* ov = getenv("LT_MORPH_BANDS")) {      // tuning knob: "b55,b29"
        if (sscanf(ov, "%d,%d", &c55, &c29) == 2 && c55 >= 1 && c29 >= 1) fixed = true;
        else c55 = c29 = 1;
    }
    if (!fixed) {
        // a cost model, not the hardware's CTA counts: every CTA takes one of 3.5 slots per SM for (band rows + warm-up
        // rows) x the relative walk cost of its structuring element, scheduled greedily in launch order
        double best = 1e300;
        std::vector<double> freeat;
        for (int a = 1; a <= 16; ++a)
            for (int b = 1; b <= 16; ++b) {
                const int ra = (lt_div_up(H, a) + 1) & ~1, rb = (lt_div_up(H, b) + 1) & ~1;
                const int na = n * tiles * lt_div_up(H, ra), nb = n * tiles * lt_div_up(H, rb);
                const double ta = (ra + 56) * 1.0, tb = (rb + 30) * 0.55;
                const int slots = (7 * sms) / 2;
                freeat.assign(slots, 0.0);
                std::make_heap(freeat.begin(), freeat.end(), std::greater<double>());
                double makespan = 0.0;
                for (int i = 0; i < na + nb; ++i) {
                    std::pop_heap(freeat.begin(), freeat.end(), std::greater<double>());
                    const double t = freeat.back() + (i < na ? ta : tb);
                    freeat.back() = t;
                    std::push_heap(freeat.begin(), freeat.end(), std::greater<double>());
                    if (t > makespan) makespan = t;
                }
                if (makespan < best - 1e-9) { best = makespan; c55 = a; c29 = b; }
            }
    }
    h->bands_key[0] = n; h->bands_key[1] = H; h->bands_key[2] = sms;
    h->bands_val[0] = c55; h->bands_val[1] = c29;
    *b55 = c55; *b29 = c29;
}

// Both erosions (tophat = false: 55x55 on Lab-b, 29x29 on R, into the tmp planes) or both dilations with the top-hat
// epilogue (src - open, into the top planes).  The 29x29 job runs on the handle's side stream next to the 55x55 job.
int lt_launch_morph_pair(lt_handle* h, bool tophat, int n, const int* list, const int* count, cudaStream_t st) {
    const LtDims& d = h->d;
    int b55, b29, rc;
    choose_bands(h, n, lt_div_up(d.p2, TW), d.bv_h, &b55, &b29);
    cudaStream_t s2 = h->side;
    LT_CUDA(cudaEventRecord(h->ev_fork, st));
    LT_CUDA(cudaStreamWaitEvent(s2, h->ev_fork, 0));
    if (!tophat) {
        if ((rc = launch_one<55, false, false>(h, h->planeB, h->tmpB, nullptr, b55, n, list, count, st))) return rc;
        if ((rc = launch_one<29, false, false>(h, h->planeR, h->tmpR, nullptr, b29, n, list, count, s2))) return rc;
    } else {
        if ((rc = launch_one<55, true, true>(h, h->tmpB, h->topB, h->planeB, b55, n, list, count, st))) return rc;
        if ((rc = launch_one<29, true, true>(h, h->tmpR, h->topR, h->planeR, b29, n, list, count, s2))) return rc;
    }
    LT_CUDA(cudaEventRecord(h->ev_join, s2));
    LT_CUDA(cudaStreamWaitEvent(st, h->ev_join, 0));
    return 0;
}
