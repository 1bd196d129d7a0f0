// filter_lane_points (lane_tracker.py:183-240) on pair-packed planes:
//   ellipse top-hat 29 (R) / 55 (Lab b)  -> cross ("bilateral") threshold  \
//   or box-mean adaptive threshold on the raw planes                        > OR -> open 5x5 -> bit mask
// The ellipse erosion / dilation / top-hat kernels live in lt_morph.cu; this file holds the thresholds, the 5x5 opening
// of the bit mask, the layout converters and the launcher of one filter attempt.
#include <cstdio>
#include "lt_common.cuh"
#include "lt_tma.cuh"

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// ---------------------------------------------------------------------------
// cross ("bilateral") threshold, bilateral_adaptive_threshold (lane_tracker.py:14-83)
//   pass <=> (L < t and R < t) or (U < t and D < t),  t = k*p - C*k, zero-padded side sums
// horizontal half: one warp per row, exclusive prefix sums of the linearised row in smem
// vertical half:   one thread per packed column, running sums in packed u16x2 registers
// ---------------------------------------------------------------------------

constexpr int ROWK_WARPS = 8;

// exclusive prefix sums E[0..W] of one image row into shared memory (one warp)
__device__ __forceinline__ void warp_row_prefix(const uint32_t* __restrict__ prow, const LtDims& d,
                                                uint32_t* lin, uint32_t* E, int lane) {
    for (int x = lane; x < d.p2; x += 32) {
        uint32_t v = __ldg(&prow[x]);
        lin[x] = v & 0xFFFFu;
        if (x + d.p2 < d.bv_w) lin[x + d.p2] = v >> 16;
    }
    __syncwarp();
    uint32_t carry = 0;
    for (int b = 0; b < d.bv_w; b += 32) {
        int x = b + lane;
        uint32_t v = (x < d.bv_w) ? lin[x] : 0u, inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, o);
            if (lane >= o) inc += n;
        }
        if (x < d.bv_w) E[x] = carry + inc - v;
        carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    if (lane == 0) E[d.bv_w] = carry;
    __syncwarp();
}

// Horizontal half of the cross threshold.  A CTA stages 32 rows of a padded plane in shared memory as (lo, hi) BYTE
// pairs (top-hat values are bytes: half the footprint of the 32-bit pair entries, so five CTAs fit an SM): 16-byte loads,
// two PRMT and two 32-bit stores per four columns.  The K halo entries either side of a row are then built from the row
// itself -- the two strips of a pair plane are neighbours in the image: column -q = {0, entry[p2 - q].lo}, column
// p2 + q = {entry[q].hi, 0} -- and the high lanes that lie beyond the image are zeroed.  Thread (row = lane,
// segment = warp) walks its column segment with running window sums L, R in packed u16x2 registers and emits finished
// 32-column mask words from two shift registers.  Rows sit in different banks (the row pitch is 2 * odd half-words), so
// the walk is conflict-free.
constexpr int CROSSH_ROWS = 32;
constexpr int CROSSH_WARPS = 8;
static_assert(CROSSH_ROWS <= LT_HALO_Y && CROSSH_ROWS % CROSSH_WARPS == 0, "a tile may run into the pad rows below the plane");

__device__ __forceinline__ uint32_t unpack_pair(uint32_t v16) {            // (hi<<8 | lo) -> hi<<16 | lo
    return __byte_perm(v16, 0, 0x4140);
}

// One launch thresholds up to two planes (blockIdx.z): plane 0 with (k0, C0), plane 1 with (k1, C1).
__global__ void __launch_bounds__(CROSSH_WARPS * 32)
k_cross_h(const uint32_t* __restrict__ plane0, const uint32_t* __restrict__ plane1, uint32_t* __restrict__ bits_all, LtDims d,
          int k0, int C0, int k1, int C1, int accumulate, int pitch0, int pitch1, int ppitch, size_t plane_stride,
          size_t bits_stride, const int* __restrict__ list, const int* __restrict__ count) {
    int slot = blockIdx.y;
    if (count != nullptr && slot >= *count) return;
    int s = list ? list[slot] : slot;
    const uint32_t* __restrict__ plane_all = blockIdx.z ? plane1 : plane0;
    const int k = blockIdx.z ? k1 : k0, C = blockIdx.z ? C1 : C0, pitch = blockIdx.z ? pitch1 : pitch0;
    const int K = (k + 1) & ~1;                                          // even: packed column 0 starts a 32-bit word
    extern __shared__ uint32_t smem[];
    unsigned short* tile = reinterpret_cast<unsigned short*>(smem);     // [32][pitch], entry i <-> packed column i - K
    const int y0 = blockIdx.x * CROSSH_ROWS;
    const uint32_t* src = plane_all + (size_t)s * plane_stride + y0 * ppitch;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        // warp w stages rows w, w + 8, ...: one 16-byte chunk of each of its rows in flight per lane.  Rows below the
        // plane are pad rows of the padded layout: every address is valid, their verdicts are dropped.
        constexpr int RPW = CROSSH_ROWS / CROSSH_WARPS;
        for (int g0 = lane * 4; g0 < d.p2; g0 += 128) {
            uint4 v[RPW];
#pragma unroll
            for (int j = 0; j < RPW; ++j) v[j] = __ldg(reinterpret_cast<const uint4*>(src + (warp + j * CROSSH_WARPS) * ppitch + g0));
#pragma unroll
            for (int j = 0; j < RPW; ++j) {
                uint32_t* o = reinterpret_cast<uint32_t*>(tile + (warp + j * CROSSH_WARPS) * pitch + K + g0);
                o[0] = __byte_perm(v[j].x, v[j].y, 0x6420);             // {lo0, hi0, lo1, hi1}
                o[1] = __byte_perm(v[j].z, v[j].w, 0x6420);
            }
        }
    }
    __syncwarp();
    {
        // every warp finishes the rows it staged itself: high lanes beyond the image, then the two halos
        const int xint = d.bv_w - d.p2;                                  // high lanes of columns >= xint lie beyond the image
        const int nfix = d.p2 - xint;
        for (int r = warp; r < CROSSH_ROWS; r += CROSSH_WARPS) {
            unsigned short* t = tile + r * pitch + K;
            for (int j = lane; j < nfix; j += 32) t[xint + j] &= 0x00FFu;
            __syncwarp();
            for (int q = lane + 1; q <= k; q += 32) t[-q] = (unsigned short)((t[d.p2 - q] & 0xFFu) << 8);          // column -q
            for (int q = lane; q <= k; q += 32) t[d.p2 + q] = (unsigned short)(q < xint ? t[q] >> 8 : 0u);          // column p2 + q
        }
    }
    __syncthreads();
    const int y = y0 + lane;
    const int nw = d.p2 >> 5;                                            // words per strip
    const int w0 = (warp * nw) / CROSSH_WARPS, w1 = ((warp + 1) * nw) / CROSSH_WARPS;
    if (w0 >= w1) return;
    const unsigned short* trow = tile + lane * pitch + K;                // trow[x] = packed column x
    const uint32_t kk = (uint32_t)k;
    const uint32_t bias = ((uint32_t)(C * k + 1)) * 0x00010001u;         // pass <=> k*p >= side + C*k + 1
    int x = w0 * 32;
    uint32_t L = bias, Rs = bias;                                        // the running sums carry the compare bias
    for (int i = 1; i <= k; ++i) { L += unpack_pair(trow[x - i]); Rs += unpack_pair(trow[x + i]); }
    uint32_t p = unpack_pair(trow[x]);
    uint32_t* brow = bits_all + (size_t)s * bits_stride + (size_t)min(y, d.bv_h - 1) * d.mwords;
    for (int w = w0; w < w1; ++w) {
        uint32_t wl = 0, wh = 0;
#pragma unroll 8
        for (int b = 0; b < 32; ++b, ++x) {
            // lanes hold values < 2^15 (k <= 127): bit 15 of ((A | 0x8000) - B) is set iff A >= B, per lane
            const uint32_t T = p * kk + 0x80008000u;
            const uint32_t ok = (T - L) & (T - Rs);
            wl = __funnelshift_l(ok * 0x10000u, wl, 1);                  // newest column in bit 0 (reversed below)
            wh = __funnelshift_l(ok, wh, 1);
            const uint32_t pn = unpack_pair(trow[x + 1]);
            L = L + p - unpack_pair(trow[x - k]);
            Rs = Rs + unpack_pair(trow[x + k + 1]) - pn;
            p = pn;
        }
        if (y < d.bv_h) {
            wl = __brev(wl); wh = __brev(wh);
            // bits of columns >= bv_w in the high strip are forced to 0
            int hbase = (d.p2 + w * 32);
            uint32_t valid = hbase + 32 <= d.bv_w ? 0xFFFFFFFFu : (hbase >= d.bv_w ? 0u : ((1u << (d.bv_w - hbase)) - 1u));
            wh &= valid;
            if (accumulate) {
                if (wl) atomicOr(&brow[w], wl);
                if (wh) atomicOr(&brow[w + nw], wh);
            } else {
                brow[w] = wl;
                brow[w + nw] = wh;
            }
        }
    }
}

// generic fallback of the horizontal half for k > 127 (packed lanes would overflow 15 bits): prefix sums
__global__ void __launch_bounds__(ROWK_WARPS * 32)
k_cross_h_wide(const uint32_t* __restrict__ plane_all, uint32_t* __restrict__ bits_all, LtDims d, int k, int C,
               int accumulate, int ppitch, size_t plane_stride, size_t bits_stride, const int* __restrict__ list,
               const int* __restrict__ count) {
    int slot = blockIdx.y;
    if (count != nullptr && slot >= *count) return;
    int s = list ? list[slot] : slot;
    extern __shared__ uint32_t smem[];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int y = blockIdx.x * ROWK_WARPS + warp;
    if (y >= d.bv_h) return;
    int wpad = (d.bv_w + 32) & ~31;
    uint32_t* lin = smem + (size_t)warp * 2 * wpad;
    uint32_t* E = lin + wpad;
    warp_row_prefix(plane_all + (size_t)s * plane_stride + (size_t)y * ppitch, d, lin, E, lane);
    uint32_t* brow = bits_all + (size_t)s * bits_stride + (size_t)y * d.mwords;
    const int Ck = C * k;
    for (int wd = 0; wd < d.mwords; ++wd) {
        int c = wd * 32 + lane;
        bool pass = false;
        if (c < d.bv_w) {
            int t = k * (int)lin[c] - Ck;
            int L = (int)(E[c] - E[max(c - k, 0)]);
            int Rs = (int)(E[min(c + k + 1, d.bv_w)] - E[c + 1]);
            pass = (L < t) && (Rs < t);
        }
        uint32_t b = __ballot_sync(0xFFFFFFFFu, pass);
        // accumulate: the vertical half may be OR-ing into the same words from another stream -> atomic
        if (lane == 0) { if (!accumulate) brow[wd] = b; else if (b) atomicOr(&brow[wd], b); }
    }
}

// Vertical half: one thread per packed column walks a band of rows with running sums U, D (packed u16x2).  The rows a
// step needs (y + k + 1 to add, y + 1 as the next centre, y - k to drop) come from a per-warp ring of plane rows in
// shared memory that is filled CV_PF chunks of CV_CHUNK rows ahead of the walk -- by TMA for packed, row-padded planes
// (k_cross_v_tma, the hot path), by 4-byte cp.async otherwise (k_cross_v).
// PACKED: k*255 + C*k + 1 < 2^15, the compare is done on both lanes at once with a guard bit.
// ROWPAD: k + 2 * CV_CHUNK <= LT_HALO_Y, every row the walk touches or prefetches exists in the padded plane (pad rows are zero, which
//         is the filter's border), so loads carry no bounds logic.
// Every lane shifts the pass bits of its own column into two registers (one per strip); after 32 rows the warp holds
// two 32x32 bit matrices column-major, transposes them with five shuffle stages each, and lane r flushes the two
// mask words of row r with one RED.OR each -- no per-row ballot.
constexpr int CV_CHUNK = 8;
constexpr int CV_BAND = 288;         // rows per CTA (multiple of 32)
constexpr int CV_BAND_FEW = 96;      // ... when fewer than 16 streams are processed (latency, not throughput)
static_assert(CV_BAND % 32 == 0 && CV_BAND % CV_CHUNK == 0 && 32 % CV_CHUNK == 0, "band geometry");

// w[lane r] bit c  ->  w[lane c] bit r
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t w, int lane) {
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        const uint32_t m = j == 16 ? 0x0000FFFFu : j == 8 ? 0x00FF00FFu : j == 4 ? 0x0F0F0F0Fu : j == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, w, j);
        const bool up = (lane & j) != 0;
        const uint32_t sh = up ? (o >> j) : (o << j);
        const uint32_t keep = up ? ~m : m;
        w = (w & keep) | (sh & ~keep);
    }
    return w;
}

// Each warp keeps the rows its walk needs in a shared-memory RING (one 128-byte slot per row, lane = column:
// conflict-free, and a thread only ever reads what it fetched itself, so no barrier is needed).  Rows enter the ring
// by 4-byte cp.async CV_PF chunks ahead of the walk: every plane row is fetched from L2/HBM once per band (instead of
// three times, as p[y+k+1], p[y+1] and p[y-k]) and 8 * (CV_PF + 1) rows per warp are in flight without holding registers.
constexpr int CV_PF = 3;             // prefetch distance in chunks

__device__ __forceinline__ void cp_async4_zfill(void* smem_dst, const void* gsrc, bool valid) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(sa), "l"(gsrc), "r"(valid ? 4 : 0) : "memory");
}
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

static int crossv_ring_rows(int k) {                  // rows y - k .. y + k + 1 of a chunk + the chunks in flight, whole chunks
    return (2 * k + 1 + CV_CHUNK * (CV_PF + 1) + CV_CHUNK - 1) / CV_CHUNK * CV_CHUNK;
}

template <bool PACKED, bool ROWPAD>
__global__ void __launch_bounds__(32)
k_cross_v(const uint32_t* __restrict__ plane0, const uint32_t* __restrict__ plane1, uint32_t* __restrict__ bits_all, LtDims d,
          int k0, int C0, int k1, int C1, int nslots, int ppitch, size_t plane_stride, size_t bits_stride,
          const int* __restrict__ list, const int* __restrict__ count, int ring_rows, int band) {
    // blockIdx.z = plane * nslots + stream slot (two planes in one launch when plane1 != nullptr)
    const int which = blockIdx.z >= nslots ? 1 : 0;
    int slot = blockIdx.z - which * nslots;
    if (count != nullptr && slot >= *count) return;
    int s = list ? list[slot] : slot;
    const uint32_t* __restrict__ plane_all = which ? plane1 : plane0;
    const int k = which ? k1 : k0, C = which ? C1 : C0;
    const int lane = threadIdx.x;
    const int x = blockIdx.x * 32 + lane;              // packed column; p2 is a multiple of 32
    const int yb0 = blockIdx.y * band, yb1 = min(yb0 + band, d.bv_h);      // band: a multiple of 32
    const uint32_t* __restrict__ P = plane_all + (size_t)s * plane_stride + x;
    uint32_t* bits = bits_all + (size_t)s * bits_stride;
    const bool hi_ok = x + d.p2 < d.bv_w;
    extern __shared__ uint32_t ring[];                 // [ring_rows + CV_CHUNK][32]
    // Ring geometry: ring_rows (R) is a multiple of CV_CHUNK, plane row r lives in slot (r - (yb0 + k + 1)) mod R, so the
    // rows a chunk ADDS (y + k + 1) start at slot 0 and stay chunk-aligned: they never wrap inside a chunk.  The two other
    // read pointers are not aligned; CV_CHUNK mirror slots behind the ring repeat slots 0 .. CV_CHUNK - 1 (fetched
    // together with them), so reading `pointer + j` never needs a wrap test.
    const int R = ring_rows;
    uint32_t* const rl = ring + lane;
    // row offsets are taken from the lowest row the band touches as UNSIGNED 32-bit numbers (IMAD.WIDE.U32 on the FMA
    // pipe; a stream of a padded plane is far below 2^32 bytes)
    const int rbase = yb0 - k;
    const uint32_t* Pb = P + rbase * ppitch;
    asm volatile("" : "+l"(Pb));                       // opaque base: keeps the per-row address a single IMAD.WIDE.U32
    const int r_last = yb1 + k + CV_CHUNK;             // rows >= r_last are never read by the walk
    auto fetch = [&](int slot_row, int r) {            // plane row r -> ring slot
        const bool ok = ROWPAD || (unsigned)r < (unsigned)d.bv_h;
        cp_async4_zfill(rl + slot_row * 32, Pb + (unsigned)((ok ? r - rbase : 0) * ppitch), ok);
    };
    auto fetch_chunk = [&](int slot_row, int r0) {     // the CV_CHUNK rows a chunk adds, slot_row is chunk-aligned
        if (r0 >= r_last) return;
#pragma unroll
        for (int j = 0; j < CV_CHUNK; ++j) fetch(slot_row + j, r0 + j);
        if (__all_sync(0xFFFFFFFFu, slot_row == 0)) {  // (uniform: a real branch instead of eight predicated copies)
#pragma unroll
            for (int j = 0; j < CV_CHUNK; ++j) fetch(R + j, r0 + j);                 // mirror of slots 0 .. CV_CHUNK - 1
        }
    };
    // prologue: rows yb0 - k .. yb0 + k go to slots R - 2k - 1 .. R - 1, then the new rows of the first CV_PF chunks
    for (int i = 0; i <= 2 * k; ++i) fetch(R - 2 * k - 1 + i, yb0 - k + i);
    int r_pf = 0;                                      // slot of the next chunk to fetch
    int y_pf = yb0 + k + 1;                            // its first plane row
#pragma unroll
    for (int c = 0; c < CV_PF; ++c) {
        fetch_chunk(r_pf, y_pf);
        cp_async_commit();
        r_pf += CV_CHUNK; if (r_pf >= R) r_pf -= R;
        y_pf += CV_CHUNK;
    }
    const int Ck = C * k;
    const uint32_t kk = (uint32_t)k, bias = (uint32_t)(Ck + 1) * 0x00010001u;
    // running sums carry the compare bias: pass <=> k*p >= U + C*k + 1 (and the same for D), per lane
    uint32_t U = PACKED ? bias : 0u, D = U, p = 0;
    int r_new = 0, r_cur = R - k, r_old = R - 2 * k - 1;   // slots of rows y + k + 1, y + 1, y - k   (y = yc + j)
    uint32_t wl = 0, wh = 0;                           // pass bits of this column, newest row in bit 0
    for (int yc = yb0; yc < yb1; yc += CV_CHUNK) {
        fetch_chunk(r_pf, y_pf);                       // (rows beyond the band are fetched and never used)
        cp_async_commit();
        r_pf += CV_CHUNK; if (r_pf >= R) r_pf -= R;
        y_pf += CV_CHUNK;
        cp_async_wait_group<CV_PF>();                  // the rows this chunk adds (and everything older) have landed
        if (yc == yb0) {
            // initial window sums from the ring: rows yb0 - k .. yb0 - 1 above, yb0 + 1 .. yb0 + k below
            const uint32_t* f = rl + (R - 2 * k - 1) * 32;
            for (int i = 0; i < k; ++i) { U += f[i * 32]; D += f[(k + 1 + i) * 32]; }
            p = f[k * 32];
        }
        const uint32_t* const pn = rl + r_new * 32;
        const uint32_t* const pcur = rl + r_cur * 32;
        const uint32_t* const pold = rl + r_old * 32;
#pragma unroll
        for (int j = 0; j < CV_CHUNK; ++j) {
            const uint32_t pc = pcur[j * 32], pu = pold[j * 32], pd = pn[j * 32];
            if (PACKED) {
                // lanes hold values < 2^15: bit 15 of ((A | 0x8000) - B) is set iff A >= B, per lane
                const uint32_t T = p * kk + 0x80008000u;
                const uint32_t ok = (T - U) & (T - D);
                wl = __funnelshift_l(ok * 0x10000u, wl, 1);        // bit 15 (IMAD.SHL on the FMA pipe) -> bit 0 of wl << 1
                wh = __funnelshift_l(ok, wh, 1);                   // bit 31
            } else {
                const int tl = k * (int)(p & 0xFFFFu) - Ck, th = k * (int)(p >> 16) - Ck;
                const bool pl = ((int)(U & 0xFFFFu) < tl) && ((int)(D & 0xFFFFu) < tl);
                const bool ph = ((int)(U >> 16) < th) && ((int)(D >> 16) < th);
                wl = (wl << 1) | (pl ? 1u : 0u);
                wh = (wh << 1) | (ph ? 1u : 0u);
            }
            U = U + p - pu;                       // lanes stay in [0, 65535]: add first, then subtract
            D = D + pd - pc;
            p = pc;
        }
        r_new += CV_CHUNK; if (r_new >= R) r_new -= R;
        r_cur += CV_CHUNK; if (r_cur >= R) r_cur -= R;
        r_old += CV_CHUNK; if (r_old >= R) r_old -= R;
        const int ynext = yc + CV_CHUNK;
        if ((ynext & 31) == 0 || ynext >= yb1) {
            // rows [ybase, ynext) are in the low (ynext - ybase) bits, newest first: bit (ynext - 1 - y) <-> row y
            const int ybase = (ynext - 1) & ~31;
            const int sh = 32 - (ynext - ybase);                   // 0 for a full group
            uint32_t ml = __brev(wl << sh), mh = hi_ok ? __brev(wh << sh) : 0u;      // bit r <-> row ybase + r
            ml = warp_transpose32(ml, lane);                       // lane r: bit c <-> column blockIdx.x * 32 + c of row ybase + r
            mh = warp_transpose32(mh, lane);
            const int y = ybase + lane;
            if (y < yb1) {
                uint32_t* brow = bits + (size_t)y * d.mwords;     // fire-and-forget RED.OR: no load to wait for
                if (ml) atomicOr(&brow[blockIdx.x], ml);
                if (mh) atomicOr(&brow[blockIdx.x + (d.p2 >> 5)], mh);
            }
            wl = wh = 0;
        }
    }
    cp_async_wait_all();
}

// ---- the same walk with the ring filled by TMA (row-padded planes only: the pad rows are the filter's border) ------
// One lane requests a whole chunk -- a box of 32 columns x 8 rows of the plane's tensor map lands as eight consecutive
// ring slots -- and the warp waits on the chunk's mbarrier: the eight cp.async per chunk, their address arithmetic and
// the group bookkeeping leave the instruction stream (the walk is issue-bound).
constexpr int CV_NST = CV_PF + 1;    // chunk mbarriers (chunks in flight)
static_assert(CV_CHUNK == 8, "lt_plane_tensor_map builds boxes of 8 rows");

static int crossv_tma_ring_rows(int k) {              // fill boxes + the chunks in flight, whole chunks
    return CV_CHUNK * ((2 * k + 1 + CV_CHUNK - 1) / CV_CHUNK + CV_PF + 1);
}

__global__ void __launch_bounds__(32)
k_cross_v_tma(const __grid_constant__ CUtensorMap tmap0, const __grid_constant__ CUtensorMap tmap1, uint32_t* __restrict__ bits_all,
              LtDims d, int k0, int C0, int k1, int C1, int nslots, size_t bits_stride, const int* __restrict__ list,
              const int* __restrict__ count, int ring_rows, int band) {
    const int which = blockIdx.z >= nslots ? 1 : 0;
    int slot = blockIdx.z - which * nslots;
    if (count != nullptr && slot >= *count) return;
    const int s = list ? list[slot] : slot;
    const CUtensorMap* const tm = which ? &tmap1 : &tmap0;
    const int k = which ? k1 : k0, C = which ? C1 : C0;
    const int lane = threadIdx.x;
    const int x = blockIdx.x * 32 + lane;
    const int yb0 = blockIdx.y * band, yb1 = min(yb0 + band, d.bv_h);
    uint32_t* bits = bits_all + (size_t)s * bits_stride;
    const bool hi_ok = x + d.p2 < d.bv_w;
    extern __shared__ __align__(128) uint32_t ring[];  // [ring_rows + CV_CHUNK][32], then the mbarriers
    const int R = ring_rows;
    uint32_t* const rl = ring + lane;
    uint64_t* const bar = reinterpret_cast<uint64_t*>(ring + (R + CV_CHUNK) * 32);     // [CV_NST] chunks, [CV_NST] = fill
    const int tx = LT_HALO_X + blockIdx.x * 32;                                        // box origin: column ...
    const int ty0 = s * (d.bv_h + 2 * LT_HALO_Y) + LT_HALO_Y;                          // ... and row of image row 0
    constexpr unsigned BOX = CV_CHUNK * 32 * sizeof(uint32_t);
    const int nbox = (2 * k + 1 + CV_CHUNK - 1) / CV_CHUNK;                            // fill boxes: they end at row yb0 + k
    const int r_last = yb1 + k + CV_CHUNK;                                             // rows >= r_last are never read
    if (lane == 0) {
        for (int i = 0; i <= CV_NST; ++i) mbar_init(&bar[i], 1);
        mbar_init_fence();
        mbar_expect_tx(&bar[CV_NST], BOX * nbox);
        for (int j = 0; j < nbox; ++j)
            tma_load_2d(ring + (R - CV_CHUNK * (nbox - j)) * 32, tm, tx, ty0 + yb0 + k + 1 - CV_CHUNK * (nbox - j), &bar[CV_NST]);
    }
    __syncwarp();
    // chunk c adds rows yb0 + k + 1 + 8c .. + 7 to slots (8c) mod R (and their mirror when that is slot 0)
    auto fetch_chunk = [&](int c) {
        const int r0 = yb0 + k + 1 + CV_CHUNK * c;
        if (r0 >= r_last) return;
        const int slot_row = (CV_CHUNK * c) % R;
        if (lane == 0) {
            fence_proxy_async();
            uint64_t* b = &bar[c % CV_NST];
            mbar_expect_tx(b, slot_row == 0 ? 2 * BOX : BOX);
            tma_load_2d(ring + slot_row * 32, tm, tx, ty0 + r0, b);
            if (slot_row == 0) tma_load_2d(ring + R * 32, tm, tx, ty0 + r0, b);
        }
    };
#pragma unroll
    for (int c = 0; c < CV_PF; ++c) fetch_chunk(c);
    const int Ck = C * k;
    const uint32_t kk = (uint32_t)k, bias = (uint32_t)(Ck + 1) * 0x00010001u;
    uint32_t U = bias, D = bias, p = 0;
    int r_new = 0, r_cur = R - k, r_old = R - 2 * k - 1;
    uint32_t wl = 0, wh = 0;
    int c = 0;
    for (int yc = yb0; yc < yb1; yc += CV_CHUNK, ++c) {
        __syncwarp();                                  // every lane has finished reading the slots the next copy overwrites
        fetch_chunk(c + CV_PF);
        if (yc == yb0) {
            mbar_wait(&bar[CV_NST], 0u);
            const uint32_t* f = rl + (R - 2 * k - 1) * 32;
            for (int i = 0; i < k; ++i) { U += f[i * 32]; D += f[(k + 1 + i) * 32]; }
            p = f[k * 32];
        }
        mbar_wait(&bar[c % CV_NST], (unsigned)(c / CV_NST) & 1u);
        const uint32_t* const pn = rl + r_new * 32;
        const uint32_t* const pcur = rl + r_cur * 32;
        const uint32_t* const pold = rl + r_old * 32;
#pragma unroll
        for (int j = 0; j < CV_CHUNK; ++j) {
            const uint32_t pc = pcur[j * 32], pu = pold[j * 32], pd = pn[j * 32];
            const uint32_t T = p * kk + 0x80008000u;
            const uint32_t ok = (T - U) & (T - D);
            wl = __funnelshift_l(ok * 0x10000u, wl, 1);
            wh = __funnelshift_l(ok, wh, 1);
            U = U + p - pu;
            D = D + pd - pc;
            p = pc;
        }
        r_new += CV_CHUNK; if (r_new >= R) r_new -= R;
        r_cur += CV_CHUNK; if (r_cur >= R) r_cur -= R;
        r_old += CV_CHUNK; if (r_old >= R) r_old -= R;
        const int ynext = yc + CV_CHUNK;
        if ((ynext & 31) == 0 || ynext >= yb1) {
            const int ybase = (ynext - 1) & ~31;
            const int sh = 32 - (ynext - ybase);
            uint32_t ml = __brev(wl << sh), mh = hi_ok ? __brev(wh << sh) : 0u;
            ml = warp_transpose32(ml, lane);
            mh = warp_transpose32(mh, lane);
            const int y = ybase + lane;
            if (y < yb1) {
                uint32_t* brow = bits + (size_t)y * d.mwords;
                if (ml) atomicOr(&brow[blockIdx.x], ml);
                if (mh) atomicOr(&brow[blockIdx.x + (d.p2 >> 5)], mh);
            }
            wl = wh = 0;
        }
    }
}

// ---------------------------------------------------------------------------
// cv2.adaptiveThreshold(MEAN_C, THRESH_BINARY, block, -c) (lane_tracker.py:217-218)
// box sum with replicated border = row sums (k_box_h) then running column sums (k_box_v)
// ---------------------------------------------------------------------------

// Row sums: the tile scheme of k_cross_h.  A CTA stages 32 rows of a raw plane as (lo, hi) byte pairs, builds the
// `half` halo entries either side of a row in shared memory -- BORDER_REPLICATE at the image edges (the first / last
// pixel of the row), the neighbouring strip at the seam -- and thread (row = lane, segment = warp) walks its segment
// with ONE running window sum per lane (packed u16x2: <= 255 * 255 fits), storing four sums per 16-byte store.
__global__ void __launch_bounds__(CROSSH_WARPS * 32)
k_box_h(const uint32_t* __restrict__ plane0, const uint32_t* __restrict__ plane1, uint32_t* __restrict__ hs0,
        uint32_t* __restrict__ hs1, LtDims d, int half0, int half1, int pitch0, int pitch1,
        int ppitch, size_t plane_stride, size_t hs_stride, const int* __restrict__ list, const int* __restrict__ count, int nslots) {
    extern __shared__ uint32_t smem[];
    unsigned short* tile = reinterpret_cast<unsigned short*>(smem);     // [32][pitch], entry i <-> packed column i - K
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nsl = count ? *count : nslots;          // attempt-2 launches loop over the (usually empty) retry list
    const uint32_t* plane_all = blockIdx.z ? plane1 : plane0;      // both planes (R, Lab-b) in one launch
    uint32_t* hs_all = blockIdx.z ? hs1 : hs0;
    const int half = blockIdx.z ? half1 : half0, pitch = blockIdx.z ? pitch1 : pitch0;
    const int K = (half + 2) & ~1;                    // even and > half: packed column 0 starts a 32-bit word
    const int y0 = blockIdx.x * CROSSH_ROWS;
    const int xint = d.bv_w - d.p2;                   // high lanes of columns >= xint lie beyond the image
    const int nw = d.p2 >> 5;
    const int w0 = (warp * nw) / CROSSH_WARPS, w1 = ((warp + 1) * nw) / CROSSH_WARPS;
    for (int slot = blockIdx.y; slot < nsl; slot += gridDim.y) {
        const int s = list ? list[slot] : slot;
        const uint32_t* src = plane_all + (size_t)s * plane_stride + y0 * ppitch;
        {
            // rows below the plane are pad rows of the padded layout: valid addresses, results dropped
            constexpr int RPW = CROSSH_ROWS / CROSSH_WARPS;
            for (int g0 = lane * 4; g0 < d.p2; g0 += 128) {
                uint4 v[RPW];
#pragma unroll
                for (int j = 0; j < RPW; ++j) v[j] = __ldg(reinterpret_cast<const uint4*>(src + (warp + j * CROSSH_WARPS) * ppitch + g0));
#pragma unroll
                for (int j = 0; j < RPW; ++j) {
                    uint32_t* o = reinterpret_cast<uint32_t*>(tile + (warp + j * CROSSH_WARPS) * pitch + K + g0);
                    o[0] = __byte_perm(v[j].x, v[j].y, 0x6420);             // {lo0, hi0, lo1, hi1}
                    o[1] = __byte_perm(v[j].z, v[j].w, 0x6420);
                }
            }
        }
        __syncwarp();
        {
            // every warp finishes the rows it staged itself: the high lanes beyond the image, then the two halos
            const int nfix = d.p2 - xint;
            for (int r = warp; r < CROSSH_ROWS; r += CROSSH_WARPS) {
                unsigned short* t = tile + r * pitch + K;
                const uint32_t first = t[0] & 0xFFu, last = t[xint - 1] >> 8;         // image columns 0 and bv_w - 1
                for (int j = lane; j < nfix; j += 32) t[xint + j] = (unsigned short)((t[xint + j] & 0xFFu) | (last << 8));
                __syncwarp();
                for (int q = lane + 1; q <= half; q += 32) t[-q] = (unsigned short)(first | ((t[d.p2 - q] & 0xFFu) << 8));
                for (int q = lane; q <= half; q += 32) t[d.p2 + q] = (unsigned short)((q < xint ? t[q] >> 8 : last) | (last << 8));
            }
        }
        __syncthreads();
        if (w0 < w1 && y0 + lane < d.bv_h) {
            const unsigned short* trow = tile + lane * pitch + K;
            uint32_t* hrow = hs_all + (size_t)s * hs_stride + (size_t)(y0 + lane) * ppitch;
            int x = w0 * 32;
            uint32_t S = 0;
            for (int i = -half; i <= half; ++i) S += unpack_pair(trow[x + i]);
            for (; x < w1 * 32; x += 4) {
                uint32_t o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    o[k] = S;
                    S = S + unpack_pair(trow[x + k + half + 1]) - unpack_pair(trow[x + k - half]);
                }
                *reinterpret_cast<uint4*>(hrow + x) = make_uint4(o[0], o[1], o[2], o[3]);
            }
        }
        __syncthreads();                              // the tile is reused by the next slot
    }
}

constexpr int BOXV_BAND = 64;        // rows per CTA (two 32-row groups)
constexpr int BOXV_CHUNK = 8;        // rows whose loads are in flight together

__global__ void __launch_bounds__(32)
k_box_v(const uint32_t* __restrict__ plane0, const uint32_t* __restrict__ plane1, const uint32_t* __restrict__ hs0,
        const uint32_t* __restrict__ hs1, uint32_t* __restrict__ bits_all, LtDims d, int half0, int half1, int c0, int c1,
        int ppitch, size_t plane_stride, size_t hs_stride, size_t bits_stride,
        const int* __restrict__ list, const int* __restrict__ count, int nslots) {
    // one thread per packed column; the thresholds of the R and the Lab-b plane are OR-ed in registers (lane r keeps
    // the mask words of rows yb0 + r and yb0 + 32 + r) and every mask word is written exactly once
    // (lane_tracker.py:217-218 + the OR at :233)
    const int nsl = count ? *count : nslots;
    for (int slot = blockIdx.z; slot < nsl; slot += gridDim.z) {
        const int s = list ? list[slot] : slot;
        const int lane = threadIdx.x;
        const int x = blockIdx.x * 32 + lane;
        const int yb0 = blockIdx.y * BOXV_BAND, yb1 = min(yb0 + BOXV_BAND, d.bv_h);
        uint32_t* bits = bits_all + (size_t)s * bits_stride;
        const bool hi_ok = x + d.p2 < d.bv_w;
        uint32_t kl[2] = {0u, 0u}, kh[2] = {0u, 0u};
        for (int pl = 0; pl < 2; ++pl) {
            const uint32_t* P = (pl ? plane1 : plane0) + (size_t)s * plane_stride + x;
            const uint32_t* Hs = (pl ? hs1 : hs0) + (size_t)s * hs_stride + x;
            const int half = pl ? half1 : half0, c = pl ? c1 : c0;
            auto ldh = [&](int r) -> uint32_t { r = max(0, min(d.bv_h - 1, r)); return __ldg(&Hs[r * ppitch]); };   // BORDER_REPLICATE
            uint32_t Sl = 0, Sh = 0;
            for (int dy0 = -half; dy0 <= half; dy0 += BOXV_CHUNK) {
                uint32_t v[BOXV_CHUNK];
#pragma unroll
                for (int j = 0; j < BOXV_CHUNK; ++j) v[j] = (dy0 + j <= half) ? ldh(yb0 + dy0 + j) : 0u;
#pragma unroll
                for (int j = 0; j < BOXV_CHUNK; ++j) { Sl += v[j] & 0xFFFFu; Sh += v[j] >> 16; }
            }
            const uint32_t n = (uint32_t)(2 * half + 1) * (uint32_t)(2 * half + 1);
            for (int yc = yb0; yc < yb1; yc += BOXV_CHUNK) {
                uint32_t p[BOXV_CHUNK], a[BOXV_CHUNK], b[BOXV_CHUNK];
#pragma unroll
                for (int j = 0; j < BOXV_CHUNK; ++j) {
                    p[j] = __ldg(&P[min(yc + j, d.bv_h - 1) * ppitch]);
                    a[j] = ldh(yc + j + half + 1);
                    b[j] = ldh(yc + j - half);
                }
#pragma unroll
                for (int j = 0; j < BOXV_CHUNK; ++j) {
                    const int y = yc + j;
                    // mean = floor((2S + n) / 2n) (rounded box mean); p - mean > c  <=>  2S + n < 2n (p - c): no division
                    const bool ok = y < yb1;
                    bool pl_ = ok && (int)(2u * Sl + n) < (int)(2u * n) * ((int)(p[j] & 0xFFFFu) - c);
                    bool ph = ok && hi_ok && ((int)(2u * Sh + n) < (int)(2u * n) * ((int)(p[j] >> 16) - c));
                    uint32_t bl = __ballot_sync(0xFFFFFFFFu, pl_), bh = __ballot_sync(0xFFFFFFFFu, ph);
                    const int g = (y - yb0) >> 5;             // (BOXV_BAND = 64: g is 0 or 1 for rows of the band)
                    if (lane == ((y - yb0) & 31)) { kl[g & 1] |= bl; kh[g & 1] |= bh; }
                    Sl += (a[j] & 0xFFFFu) - (b[j] & 0xFFFFu);
                    Sh += (a[j] >> 16) - (b[j] >> 16);
                }
            }
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) {
            const int y = yb0 + 32 * g + lane;
            if (y < yb1) {
                uint32_t* brow = bits + (size_t)y * d.mwords;
                brow[blockIdx.x] = kl[g];
                brow[blockIdx.x + (d.p2 >> 5)] = kh[g];
            }
        }
    }
}

// mask_noise (lane_tracker.py:221-231): merged &= ~inRange(b, thresh, 255) | cross(b, k_noise, C_noise)
__global__ void __launch_bounds__(32)
k_noise_combine(const uint32_t* __restrict__ planeB_all, const uint32_t* __restrict__ noise_bits_all,
                uint32_t* __restrict__ merged_all, LtDims d, int thresh, int ppitch, size_t plane_stride, size_t bits_stride,
                const int* __restrict__ list, const int* __restrict__ count) {
    int slot = blockIdx.z;
    if (count != nullptr && slot >= *count) return;
    int s = list ? list[slot] : slot;
    int lane = threadIdx.x, x = blockIdx.x * 32 + lane, y = blockIdx.y;
    uint32_t p = __ldg(&planeB_all[(size_t)s * plane_stride + (size_t)y * ppitch + x]);
    uint32_t il = __ballot_sync(0xFFFFFFFFu, (int)(p & 0xFFFFu) >= thresh);
    uint32_t ih = __ballot_sync(0xFFFFFFFFu, (int)(p >> 16) >= thresh);
    if (lane == 0) {
        size_t o = (size_t)s * bits_stride + (size_t)y * d.mwords;
        int wl = blockIdx.x, wh = blockIdx.x + (d.p2 >> 5);
        merged_all[o + wl] &= (~il | noise_bits_all[o + wl]);
        merged_all[o + wh] &= (~ih | noise_bits_all[o + wh]);
    }
}

// ---------------------------------------------------------------------------
// open 5x5 ellipse on the bit mask (lane_tracker.py:238): rows [0,2,2,2,0]
// ---------------------------------------------------------------------------

// One lane = one mask word (32 columns), walking down a band of rows with the last rows in registers; the neighbour
// words come from the adjacent lanes by shuffle.  A warp carries 28 output words and two halo words either side (the
// erosion of a halo word feeds the dilation of an output word), so nothing goes through shared memory:
//   A5(y) = AND of the five horizontal shifts of row y            E(y) = M(y-2) & M(y+2) & A5(y-1) & A5(y) & A5(y+1)
//   O5(y) = OR  of the five horizontal shifts of E(y)           out(y) = E(y-2) | E(y+2) | O5(y-1) | O5(y) | O5(y+1)
// Outside the image: ones for the erosion (never blocks), zeros for the dilation (cv2.morphologyEx's default border).
constexpr int OPEN_BAND = 32;   // output rows per CTA (+ 8 warm-up rows: short bands keep enough warps in flight);
constexpr int OPEN_BAND_FEW = 8;   // with only a few streams the walk is pure latency: shorter bands, more warps
constexpr int OPEN_CORE = 28;   // output words per warp

__device__ __forceinline__ uint32_t shl_bits(uint32_t prev, uint32_t cur, int n) {   // bit x <- bit x-n
    return __funnelshift_l(prev, cur, n);
}
__device__ __forceinline__ uint32_t shr_bits(uint32_t cur, uint32_t next, int n) {   // bit x <- bit x+n
    return __funnelshift_r(cur, next, n);
}

__global__ void __launch_bounds__(64)
k_open5(const uint32_t* __restrict__ in_all, uint32_t* __restrict__ out_all, LtDims d, size_t bits_stride,
        const int* __restrict__ list, const int* __restrict__ count, int nslots, int band) {
    const int nsl = count ? *count : nslots;
    const int lane = threadIdx.x & 31, warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int mw = d.mwords;
    const int wd = warp * OPEN_CORE + lane - 2;                         // this lane's mask word
    if (warp * OPEN_CORE >= mw) return;
    const bool w_in = wd >= 0 && wd < mw;
    const uint32_t valid = !w_in ? 0u : (wd * 32 + 32 <= d.bv_w) ? 0xFFFFFFFFu : (wd * 32 >= d.bv_w ? 0u : ((1u << (d.bv_w - wd * 32)) - 1u));
    const bool emit = lane >= 2 && lane < 2 + OPEN_CORE && w_in;
    const int y0 = blockIdx.y * band, y1 = min(y0 + band, d.bv_h);
    for (int slot = blockIdx.z; slot < nsl; slot += gridDim.z) {
        const int s = list ? list[slot] : slot;
        const uint32_t* in = in_all + (size_t)s * bits_stride + (w_in ? wd : 0);
        uint32_t* out = out_all + (size_t)s * bits_stride + (w_in ? wd : 0);
        // rows r = y0 - 4 .. y1 + 3 enter one by one; row r completes E(r - 2) and out(r - 4)
        uint32_t m1 = ~0u, m2 = ~0u, m3 = ~0u, m4 = ~0u;                // M(r-1) .. M(r-4)
        uint32_t a1 = ~0u, a2 = ~0u, a3 = ~0u;                          // A5(r-1) .. A5(r-3)
        uint32_t e1 = 0u, e2 = 0u, e3 = 0u, e4 = 0u;                    // E(r-3) .. E(r-6)
        uint32_t o1 = 0u, o2 = 0u, o3 = 0u;                             // O5(r-3) .. O5(r-5)
        uint32_t nxt = ((unsigned)(y0 - 4) < (unsigned)d.bv_h && w_in) ? __ldg(in + (size_t)(y0 - 4) * mw) : 0u;
#pragma unroll 4
        for (int r = y0 - 4; r < y1 + 4; ++r) {
            const bool row_in = (unsigned)r < (unsigned)d.bv_h;
            const uint32_t m0 = row_in ? ((nxt & valid) | ~valid) : ~0u;
            nxt = ((unsigned)(r + 1) < (unsigned)d.bv_h && w_in) ? __ldg(in + (size_t)(r + 1) * mw) : 0u;      // one row ahead
            uint32_t pv = __shfl_up_sync(0xFFFFFFFFu, m0, 1), nx = __shfl_down_sync(0xFFFFFFFFu, m0, 1);
            const uint32_t a0 = m0 & shl_bits(pv, m0, 1) & shl_bits(pv, m0, 2) & shr_bits(m0, nx, 1) & shr_bits(m0, nx, 2);
            // E(r - 2): zero on rows outside the image and on columns beyond it
            const bool e_in = (unsigned)(r - 2) < (unsigned)d.bv_h;
            const uint32_t e0 = e_in ? (m4 & m0 & a3 & a2 & a1 & valid) : 0u;
            pv = __shfl_up_sync(0xFFFFFFFFu, e0, 1); nx = __shfl_down_sync(0xFFFFFFFFu, e0, 1);
            const uint32_t o0 = e0 | shl_bits(pv, e0, 1) | shl_bits(pv, e0, 2) | shr_bits(e0, nx, 1) | shr_bits(e0, nx, 2);
            // out(r - 4) = E(r-6) | E(r-2) | O5(r-5) | O5(r-4) | O5(r-3)
            const int yo = r - 4;
            if (emit && yo >= y0 && yo < y1) out[(size_t)yo * mw] = (e4 | e0 | o3 | o2 | o1) & valid;
            m4 = m3; m3 = m2; m2 = m1; m1 = m0;
            a3 = a2; a2 = a1; a1 = a0;
            e4 = e3; e3 = e2; e2 = e1; e1 = e0;
            o3 = o2; o2 = o1; o1 = o0;
        }
    }
}

// ---------------------------------------------------------------------------
// layout converters (API boundary / tests)
// ---------------------------------------------------------------------------

__global__ void k_mask_to_u8(const uint32_t* __restrict__ bits, uint8_t* __restrict__ out, LtDims d, size_t bits_stride) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, s = blockIdx.z;
    if (x >= d.bv_w) return;
    uint32_t w = __ldg(&bits[(size_t)s * bits_stride + (size_t)y * d.mwords + (x >> 5)]);
    out[((size_t)s * d.bv_h + y) * d.bv_w + x] = ((w >> (x & 31)) & 1u) ? 255 : 0;
}

__global__ void k_u8_to_mask(const uint8_t* __restrict__ in, uint32_t* __restrict__ bits, LtDims d, size_t bits_stride) {
    int wd = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    int y = blockIdx.y, s = blockIdx.z;
    if (wd >= d.mwords) return;
    int x = wd * 32 + lane;
    bool on = x < d.bv_w && __ldg(&in[((size_t)s * d.bv_h + y) * d.bv_w + x]) != 0;
    uint32_t b = __ballot_sync(0xFFFFFFFFu, on);
    if (lane == 0) bits[(size_t)s * bits_stride + (size_t)y * d.mwords + wd] = b;
}

__global__ void k_plane_to_u8(const uint32_t* __restrict__ plane, uint8_t* __restrict__ out, LtDims d, int ppitch,
                              size_t plane_stride) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, s = blockIdx.z;
    if (x >= d.bv_w) return;
    uint32_t v = __ldg(&plane[(size_t)s * plane_stride + (size_t)y * ppitch + (x >= d.p2 ? x - d.p2 : x)]);
    out[((size_t)s * d.bv_h + y) * d.bv_w + x] = (uint8_t)((x >= d.p2 ? (v >> 16) : v) & 255u);
}

int lt_launch_mask_to_u8(lt_handle* h, const uint32_t* bits, uint8_t* d_mask, int n, cudaStream_t st) {
    dim3 g(lt_div_up(h->d.bv_w, 256), h->d.bv_h, n);
    k_mask_to_u8<<<g, 256, 0, st>>>(bits, d_mask, h->d, h->stream_mask);
    LT_LAUNCH_CHECK();
    return 0;
}
int lt_launch_u8_to_mask(lt_handle* h, const uint8_t* d_mask, uint32_t* bits, int n, cudaStream_t st) {
    dim3 g(lt_div_up(h->d.mwords, 8), h->d.bv_h, n);
    k_u8_to_mask<<<g, 256, 0, st>>>(d_mask, bits, h->d, h->stream_mask);
    LT_LAUNCH_CHECK();
    return 0;
}
int lt_launch_plane_to_u8(lt_handle* h, const uint32_t* plane, int pitch, uint8_t* d_dst, int n, cudaStream_t st) {
    dim3 g(lt_div_up(h->d.bv_w, 256), h->d.bv_h, n);
    k_plane_to_u8<<<g, 256, 0, st>>>(plane, d_dst, h->d, pitch, h->stream_pad);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// the whole filter for one attempt
// ---------------------------------------------------------------------------

static bool cross_packed(int k, int C) { return k <= 127 && C >= 0 && k * 255 + C * k + 1 < 32768; }   // packed u16 lanes stay below 2^15

static int crossh_pitch(const LtDims& d, int k) {                  // in half-words
    int pitch = d.p2 + 2 * ((k + 1) & ~1) + 4;
    while (((pitch >> 1) & 1) == 0 || (pitch & 1)) ++pitch;       // pitch = 2 * odd: rows are word aligned and land in distinct banks
    return pitch;
}
constexpr size_t CROSSH_SMEM_MAX = 200 * 1024;

static int box_pitch(const LtDims& d, int half) {                  // in half-words: 2 * odd, like crossh_pitch
    int pitch = d.p2 + 2 * ((half + 2) & ~1) + 4;
    while (((pitch >> 1) & 1) == 0 || (pitch & 1)) ++pitch;
    return pitch;
}

// The row kernels are the only threshold kernels whose shared memory grows with the width: the packed one while its
// tile fits CROSSH_SMEM_MAX (k <= 127), the prefix-sum one (k > 127 or unpacked lanes, at any width) and the box one
// (block 255).  The column kernels, the morphology and the opening stage fixed-width strips, independent of
// bv_w.
size_t lt_filter_smem_bytes(int bv_w) {
    LtDims d;
    memset(&d, 0, sizeof(d));
    d.bv_w = bv_w;
    d.p2 = 32 * ((bv_w + 63) / 64);
    const size_t packed = (size_t)CROSSH_ROWS * crossh_pitch(d, 127) * sizeof(unsigned short);
    const size_t wide = (size_t)ROWK_WARPS * 2 * ((bv_w + 32) & ~31) * sizeof(uint32_t);
    const size_t box = (size_t)CROSSH_ROWS * box_pitch(d, 255 / 2) * sizeof(unsigned short);
    size_t m = wide > box ? wide : box;
    if (packed <= CROSSH_SMEM_MAX && packed > m) m = packed;
    return m;
}

// horizontal half of one plane, or of two planes in one launch (plane1 != nullptr; both must take the packed kernel)
static int launch_cross_h(lt_handle* h, const uint32_t* plane, uint32_t* bits, int k, int C, int accumulate, int n,
                          const int* list, const int* count, cudaStream_t st, const uint32_t* plane1 = nullptr, int k1 = 0,
                          int C1 = 0) {
    const LtDims& d = h->d;
    const int ppitch = d.pp;
    const size_t pstride = h->stream_pad;
    const size_t tile0 = (size_t)CROSSH_ROWS * crossh_pitch(d, k) * sizeof(unsigned short);
    const size_t tile1 = plane1 ? (size_t)CROSSH_ROWS * crossh_pitch(d, k1) * sizeof(unsigned short) : 0;
    if (cross_packed(k, C) && (!plane1 || cross_packed(k1, C1)) && tile0 <= CROSSH_SMEM_MAX && tile1 <= CROSSH_SMEM_MAX) {
        const int pitch0 = crossh_pitch(d, k), pitch1 = plane1 ? crossh_pitch(d, k1) : pitch0;
        size_t smem = tile0 > tile1 ? tile0 : tile1;
        int rc = lt_ensure_smem((const void*)k_cross_h, smem);
        if (rc) return rc;
        dim3 gh(lt_div_up(d.bv_h, CROSSH_ROWS), n, plane1 ? 2 : 1);
        k_cross_h<<<gh, CROSSH_WARPS * 32, smem, st>>>(plane, plane1, bits, d, k, C, k1, C1, accumulate, pitch0, pitch1, ppitch,
                                                         pstride, h->stream_mask, list, count);
        LT_LAUNCH_CHECK();
        return 0;
    }
    if (plane1) {        // mixed: one plane at a time
        int rc = launch_cross_h(h, plane, bits, k, C, accumulate, n, list, count, st);
        if (rc) return rc;
        return launch_cross_h(h, plane1, bits, k1, C1, 1, n, list, count, st);
    }
    {
        int wpad = (d.bv_w + 32) & ~31;
        size_t smem = (size_t)ROWK_WARPS * 2 * wpad * sizeof(uint32_t);
        int rc = lt_ensure_smem((const void*)k_cross_h_wide, smem);
        if (rc) return rc;
        dim3 gh(lt_div_up(d.bv_h, ROWK_WARPS), n);
        k_cross_h_wide<<<gh, ROWK_WARPS * 32, smem, st>>>(plane, bits, d, k, C, accumulate, ppitch, pstride,
                                                            h->stream_mask, list, count);
        LT_LAUNCH_CHECK();
    }
    return 0;
}

// pad_rows_zero: the pad rows of `plane` hold 0 (top-hat planes), i.e. they ARE the filter's BORDER_CONSTANT border and
// the row-padded fast path may read them; the raw planes carry the erosion pad 0xFFFF there and must be bounds-checked.
static int launch_cross_v(lt_handle* h, const uint32_t* plane, uint32_t* bits, int k, int C, int n,
                          const int* list, const int* count, cudaStream_t st, bool pad_rows_zero, const uint32_t* plane1 = nullptr,
                          int k1 = 0, int C1 = 0) {
    const LtDims& d = h->d;
    const int ppitch = d.pp;
    const size_t pstride = h->stream_pad;
    const bool packed = cross_packed(k, C), rowpad = pad_rows_zero && k + 2 * CV_CHUNK <= LT_HALO_Y;
    if (plane1 && (cross_packed(k1, C1) != packed || (pad_rows_zero && k1 + 2 * CV_CHUNK <= LT_HALO_Y) != rowpad)) {
        int rc = launch_cross_v(h, plane, bits, k, C, n, list, count, st, pad_rows_zero);     // different kernel variants
        if (rc) return rc;
        return launch_cross_v(h, plane1, bits, k1, C1, n, list, count, st, pad_rows_zero);
    }
    const int band = n >= 16 ? CV_BAND : CV_BAND_FEW;               // few streams: shorter sequential walks, more warps
    dim3 gv(d.p2 / 32, lt_div_up(d.bv_h, band), plane1 ? 2 * n : n);
    const int kmax = (plane1 && k1 > k) ? k1 : k;
    if (packed && rowpad) {
        CUtensorMap tm0, tm1;
        int rc_ = lt_plane_tensor_map(h, plane, 32, &tm0);
        if (!rc_) { if (plane1) rc_ = lt_plane_tensor_map(h, plane1, 32, &tm1); else tm1 = tm0; }
        if (rc_) return rc_;
        const int rr = crossv_tma_ring_rows(kmax);
        const size_t bytes = (size_t)(rr + CV_CHUNK) * 32 * sizeof(uint32_t) + (CV_NST + 1) * sizeof(uint64_t);
        if ((rc_ = lt_ensure_smem((const void*)k_cross_v_tma, bytes))) return rc_;
        k_cross_v_tma<<<gv, 32, bytes, st>>>(tm0, tm1, bits, d, k, C, k1, C1, n, h->stream_mask, list, count, rr, band);
        LT_LAUNCH_CHECK();
        return 0;
    }
    // the cp.async ring serves what TMA cannot: unpacked lanes, a plane whose pad rows are not zero (the raw plane of
    // mask_noise) and k > 40
    const int ring_rows = crossv_ring_rows(kmax);
    const size_t ring_bytes = (size_t)(ring_rows + CV_CHUNK) * 32 * sizeof(uint32_t);      // + the mirror slots
#define LT_CROSS_V(PK, RP) do { int rc_ = lt_ensure_smem((const void*)k_cross_v<PK, RP>, ring_bytes); if (rc_) return rc_; \
        k_cross_v<PK, RP><<<gv, 32, ring_bytes, st>>>(plane, plane1, bits, d, k, C, k1, C1, n, ppitch, pstride, h->stream_mask, list, count, ring_rows, band); } while (0)
    if (packed) LT_CROSS_V(true, false);
    else if (rowpad) LT_CROSS_V(false, true);
    else LT_CROSS_V(false, false);
#undef LT_CROSS_V
    LT_LAUNCH_CHECK();
    return 0;
}

// horizontal half writes (or ORs) the words, vertical half ORs into them
static int launch_cross(lt_handle* h, const uint32_t* plane, uint32_t* bits, int k, int C, int accumulate, int n,
                        const int* list, const int* count, cudaStream_t st, bool pad_rows_zero) {
    int rc = launch_cross_h(h, plane, bits, k, C, accumulate, n, list, count, st);
    if (rc) return rc;
    return launch_cross_v(h, plane, bits, k, C, n, list, count, st, pad_rows_zero);
}

static int launch_box_pair(lt_handle* h, int block_r, int c_r, int block_b, int c_b, int n, const int* list,
                           const int* count, cudaStream_t st) {
    // adaptiveThreshold of the R and the Lab-b plane in two launches (row sums of both, then columns + OR);
    // the top-hat planes, unused by this filter type, hold the row sums
    const LtDims& d = h->d;
    const int half_r = block_r / 2, half_b = block_b / 2;
    const int pitch_r = box_pitch(d, half_r), pitch_b = box_pitch(d, half_b);
    size_t smem = (size_t)CROSSH_ROWS * (pitch_r > pitch_b ? pitch_r : pitch_b) * sizeof(unsigned short);
    { int rc = lt_ensure_smem((const void*)k_box_h, smem); if (rc) return rc; }
    const int zs = count ? (n < 8 ? n : 8) : n;     // retry-list launches: few slots, each CTA loops over the list
    dim3 gh(lt_div_up(d.bv_h, CROSSH_ROWS), zs, 2);
    k_box_h<<<gh, CROSSH_WARPS * 32, smem, st>>>(h->planeR, h->planeB, h->topR, h->topB, d, half_r, half_b, pitch_r, pitch_b, d.pp,
                                                 h->stream_pad, h->stream_pad, list, count, n);
    LT_LAUNCH_CHECK();
    dim3 gv(d.p2 / 32, lt_div_up(d.bv_h, BOXV_BAND), zs);
    k_box_v<<<gv, 32, 0, st>>>(h->planeR, h->planeB, h->topR, h->topB, h->merged, d, block_r / 2, block_b / 2, c_r, c_b,
                               d.pp, h->stream_pad, h->stream_pad, h->stream_mask, list, count, n);
    LT_LAUNCH_CHECK();
    return 0;
}

int lt_launch_filter(lt_handle* h, int n, const LtAttemptParams& p, const int* list, const int* count,
                     cudaStream_t st) {
    const LtFilterGroup g = {p, list, n};
    return lt_launch_filter_groups(h, n, &g, 1, count, st);
}

int lt_launch_filter_groups(lt_handle* h, int n, const LtFilterGroup* g, int ng, const int* count, cudaStream_t st) {
    const LtDims& d = h->d;
    int rc;
    // the morphology has no parameters: one pair of launches over the positions of every bilateral group
    int n_morph = 0;
    for (int i = 0; i < ng && g[i].p.filter_type == 0; ++i) n_morph += g[i].n;
    if (n_morph > 0) {
        const int* ml = (n_morph == n && count == nullptr) ? nullptr : g[0].list;
        if ((rc = lt_launch_morph_pair(h, false, n_morph, ml, count, st))) return rc;
        lt_prof_mark(h, ST_ERODE55, st);            // both erosions (55x55 on Lab-b, 29x29 on R), two concurrent kernels
        if ((rc = lt_launch_morph_pair(h, true, n_morph, ml, count, st))) return rc;
        lt_prof_mark(h, ST_TOPHAT55, st);           // both dilations + top-hat epilogues
    }
    bool zeroed = false;
    for (int i = 0; i < ng; ++i) {
        const LtAttemptParams& p = g[i].p;
        const int* list = g[i].list;
        const int gn = g[i].n;
        if (p.filter_type == 0) {
            if (count == nullptr) {
                // The four threshold halves (R/Lab-b x horizontal/vertical) only OR bits into the merged mask and each
                // of them fills about half of the issue slots: the horizontal pair runs on a side stream, the vertical
                // pair on the caller's stream.  (Stage "cross_b" then reports both planes.)  The merged masks of the
                // whole batch are cleared once: the box threshold of a neighbourhood group rewrites every word.
                if (!zeroed) LT_CUDA(cudaMemsetAsync(h->merged, 0, (size_t)n * h->stream_mask * sizeof(uint32_t), st));
                zeroed = true;
                LT_CUDA(cudaEventRecord(h->ev_fork, st));
                LT_CUDA(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
                if ((rc = launch_cross_h(h, h->topR, h->merged, p.ksize_r, p.C_r, 1, gn, list, nullptr, h->side, h->topB, p.ksize_b, p.C_b))) return rc;
                LT_CUDA(cudaEventRecord(h->ev_join, h->side));
                if ((rc = launch_cross_v(h, h->topR, h->merged, p.ksize_r, p.C_r, gn, list, nullptr, st, true, h->topB, p.ksize_b, p.C_b))) return rc;
                LT_CUDA(cudaStreamWaitEvent(st, h->ev_join, 0));
                lt_prof_mark(h, ST_CROSS_B, st);
            } else {
                if ((rc = launch_cross(h, h->topR, h->merged, p.ksize_r, p.C_r, 0, gn, list, count, st, true))) return rc;
                lt_prof_mark(h, ST_CROSS_R, st);
                if ((rc = launch_cross(h, h->topB, h->merged, p.ksize_b, p.C_b, 1, gn, list, count, st, true))) return rc;
                lt_prof_mark(h, ST_CROSS_B, st);
            }
        } else {
            if ((rc = launch_box_pair(h, p.ksize_r, p.C_r, p.ksize_b, p.C_b, gn, list, count, st))) return rc;
            lt_prof_mark(h, ST_BOX, st);
        }
        if (p.mask_noise) {
            // h->mask of the group's own positions holds the noise bits until k_open5 overwrites it
            if ((rc = launch_cross(h, h->planeB, h->mask, p.ksize_noise, p.C_noise, 0, gn, list, count, st, false))) return rc;
            dim3 gz(d.p2 / 32, d.bv_h, gn);
            k_noise_combine<<<gz, 32, 0, st>>>(h->planeB, h->mask, h->merged, d, p.noise_thresh, d.pp, h->stream_pad,
                                               h->stream_mask, list, count);
            LT_LAUNCH_CHECK();
            lt_prof_mark(h, ST_NOISE, st);
        }
    }
    const int* list = ng == 1 ? g[0].list : nullptr;
    const int zs = count ? (n < 8 ? n : 8) : n;
    const int band = zs >= 16 ? OPEN_BAND : OPEN_BAND_FEW;
    dim3 go(lt_div_up(lt_div_up(d.mwords, OPEN_CORE), 2), lt_div_up(d.bv_h, band), zs);
    k_open5<<<go, 64, 0, st>>>(h->merged, h->mask, d, h->stream_mask, list, count, n, band);
    LT_LAUNCH_CHECK();
    lt_prof_mark(h, ST_OPEN5, st);
    return 0;
}
