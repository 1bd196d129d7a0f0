// Lane-pixel search, polynomial fit, validity check and per-stream state machine:
// sliding_window_search (lane_tracker.py:242-447), band_search (449-500), fit_poly (502-509),
// get_poly_points (511-528), check_validity (561-627), get_curve_radius / get_eccentricity
// (530-559) and the success / failure bookkeeping of process() (1142-1209).
//
// One CTA per stream.  Both searches reduce to "for an ordered list of mask rows, take the
// set bits inside a per-row column window"; the sliding-window search first walks its window
// centroids (sequential, but it only needs windowed column counts, which the CTA evaluates on
// demand from the bit mask with popc), the band search derives the window from the previous
// fit.  Counting, ordered compaction and the exact int64 moment sums then run over that row
// list in parallel.  Compiled with -fmad=false; every fp64 expression whose rounding matters
// for parity is written with explicit round-to-nearest intrinsics in the reference's order.
#include "lt_common.cuh"

#define SEARCH_THREADS 256
#define MAX_ROIS (2 * LT_MAX_LEVELS)

__device__ __forceinline__ double mul64(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add64(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub64(double a, double b) { return __dsub_rn(a, b); }

// a*y^2 + b*y + c exactly as NumPy evaluates  cf[0]*y**2 + cf[1]*y + cf[2]
__device__ __forceinline__ double poly_eval(const double* cf, double y) {
    return add64(add64(mul64(cf[0], mul64(y, y)), mul64(cf[1], y)), cf[2]);
}

// Python slice resolution of a[start:stop] on an axis of length n
__device__ __forceinline__ void pyslice(int start, int stop, int n, int& a, int& b) {
    a = start < 0 ? max(start + n, 0) : min(start, n);
    b = stop < 0 ? max(stop + n, 0) : min(stop, n);
    if (b < a) b = a;
}

// number of set bits / sum of their column indices in columns [xa, xb] of one mask row
__device__ __forceinline__ int row_bits(const uint32_t* __restrict__ row, int xa, int xb, int* sumx) {
    int n = 0, sx = 0;
    for (int w = xa >> 5; w <= (xb >> 5); ++w) {
        uint32_t v = __ldg(&row[w]);
        int lo = max(xa - w * 32, 0), hi = min(xb - w * 32, 31);
        uint32_t m = (hi == 31 ? 0xFFFFFFFFu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
        v &= m;
        int c = __popc(v);
        n += c;
        if (sumx) {
            sx += w * 32 * c + __popc(v & 0xAAAAAAAAu) + 2 * __popc(v & 0xCCCCCCCCu) + 4 * __popc(v & 0xF0F0F0F0u) +
                  8 * __popc(v & 0xFF00FF00u) + 16 * __popc(v & 0xFFFF0000u);
        }
    }
    if (sumx) *sumx = sx;
    return n;
}

template <typename T> __device__ T block_sum(T v, T* scratch) {
    // scratch: SEARCH_THREADS/32 entries
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    T r = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += scratch[i];
    __syncthreads();
    return r;
}

// In-place exclusive scan of a[0..n) in shared memory; returns the total. All threads call.
__device__ int block_excl_scan(int* a, int n, int* scratch) {
    int per = (n + blockDim.x - 1) / blockDim.x;
    int b = threadIdx.x * per, e = min(b + per, n);
    int s = 0;
    for (int i = b; i < e; ++i) s += a[i];
    scratch[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int i = 0; i < (int)blockDim.x; ++i) { int t = scratch[i]; scratch[i] = run; run += t; }
        scratch[blockDim.x] = run;
    }
    __syncthreads();
    int run = scratch[threadIdx.x];
    for (int i = b; i < e; ++i) { int t = a[i]; a[i] = run; run += t; }
    int total = scratch[blockDim.x];
    __syncthreads();
    return total;
}

struct Roi { int r0, r1, c0, c1, xoff; };

struct SearchShared {
    int s_max, s_first, s_last;
    int nroi[2];
    int ncent[2];
    int nvisit[2];
    int total[2];
    int detected;
    int nkeep[2];
    double coeffs[2][3];
    long long mom[2][8];
    int distinct[2];
    int ry[2][2], rn[2][2], rsx[2][2];
};

// Column histogram of mask rows [r0, r1) for the 32 columns of mask word `w`, written to out[0..31] (int):
// the rows are added bit-sliced (six carry-save bit planes hold up to 63 rows, then the planes are flushed).
// Only the first `nvalid` columns of the word are stored (the last mask word runs past the image: storing all 32
// counts would spill into the prefix-sum row of the next level, which another thread is filling).
__device__ void hist_word(const uint32_t* __restrict__ mask, int mwords, int r0, int r1, int w, int nvalid, int* __restrict__ out) {
    int cnt[32];
#pragma unroll
    for (int b = 0; b < 32; ++b) cnt[b] = 0;
    for (int g0 = r0; g0 < r1; g0 += 63) {
        uint32_t p0 = 0, p1 = 0, p2 = 0, p3 = 0, p4 = 0, p5 = 0;
        const int g1 = min(g0 + 63, r1);
        for (int y = g0; y < g1; ++y) {
            uint32_t c = __ldg(&mask[(size_t)y * mwords + w]), t;
            t = p0 & c; p0 ^= c; c = t;
            t = p1 & c; p1 ^= c; c = t;
            t = p2 & c; p2 ^= c; c = t;
            t = p3 & c; p3 ^= c; c = t;
            t = p4 & c; p4 ^= c; c = t;
            p5 ^= c;
        }
#pragma unroll
        for (int b = 0; b < 32; ++b)
            cnt[b] += (int)(((p0 >> b) & 1u) | (((p1 >> b) & 1u) << 1) | (((p2 >> b) & 1u) << 2) | (((p3 >> b) & 1u) << 3) |
                            (((p4 >> b) & 1u) << 4) | (((p5 >> b) & 1u) << 5));
    }
#pragma unroll
    for (int b = 0; b < 32; ++b)
        if (b < nvalid) out[b] = cnt[b];
}

// In-place: P[0] = 0, P[x + 1] = cnt[0] + ... + cnt[x] for the counts stored at P[1..W]; one warp.
__device__ void warp_prefix_inplace(int* P, int W, int lane) {
    const int per = (W + 31) / 32, b = min(lane * per, W), e = min(b + per, W);
    int s = 0;
    for (int x = b; x < e; ++x) s += P[1 + x];
    int inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += n;
    }
    int run = inc - s;
    for (int x = b; x < e; ++x) { run += P[1 + x]; P[1 + x] = run; }
    if (lane == 0) P[0] = 0;
    __syncwarp();
}

// Windowed column counts (np.convolve(ones(ww), colsum) 'full') of the columns [c0, c0 + nc) from the prefix sums P:
//   S[i] = sum col[max(0, i - ww + 1) .. min(i, nc - 1)],  col[j] = count of column c0 + j
__device__ __forceinline__ int window_sum(const int* P, int c0, int nc, int ww, int i) {
    const int a = max(0, i - ww + 1), b = min(i, nc - 1);
    return a <= b ? P[c0 + b + 1] - P[c0 + a] : 0;
}

// max of S[sa..sb) and the first / last index (relative to sa) attaining it; one warp, result uniform over the lanes
__device__ void warp_argmax(const int* P, int c0, int nc, int ww, int sa, int sb, int lane, int& smax, int& sfirst, int& slast) {
    int m = -1, f = 0x7FFFFFFF, l = -1;
    for (int i = sa + lane; i < sb; i += 32) {
        const int v = window_sum(P, c0, nc, ww, i);
        if (v > m) { m = v; f = i - sa; l = i - sa; }
        else if (v == m) l = i - sa;
    }
    smax = __reduce_max_sync(0xFFFFFFFFu, m);
    sfirst = __reduce_min_sync(0xFFFFFFFFu, m == smax ? f : 0x7FFFFFFF);
    slast = __reduce_max_sync(0xFFFFFFFFu, m == smax ? l : -1);
}

// Solve the 3x3 normal equations (Gaussian elimination, partial pivoting).
__device__ bool solve3(double A[3][3], double b[3], double x[3]) {
    int p[3] = {0, 1, 2};
    for (int c = 0; c < 3; ++c) {
        int best = c;
        for (int r = c + 1; r < 3; ++r)
            if (fabs(A[p[r]][c]) > fabs(A[p[best]][c])) best = r;
        int t = p[c]; p[c] = p[best]; p[best] = t;
        double piv = A[p[c]][c];
        if (piv == 0.0) return false;
        for (int r = c + 1; r < 3; ++r) {
            double f = A[p[r]][c] / piv;
            for (int k = c; k < 3; ++k) A[p[r]][k] -= f * A[p[c]][k];
            b[p[r]] -= f * b[p[c]];
        }
    }
    for (int c = 2; c >= 0; --c) {
        double s = b[p[c]];
        for (int k = c + 1; k < 3; ++k) s -= A[p[c]][k] * x[k];
        x[c] = s / A[p[c]][c];
    }
    return true;
}

// np.polyfit(y, x, 2) from exact integer moments about yc (t = y - yc):
//   mom = {S0, S1, S2, S3, S4, X0, X1, X2},  Sk = sum t^k,  Xj = sum x t^j
__device__ void fit_from_moments(const long long* mom, double yc, double sc, int distinct, const int* ry,
                                 const int* rn, const int* rsx, double* cf, int* rank_def) {
    *rank_def = 0;
    if (distinct >= 3) {
        double s1 = sc, s2 = sc * sc, s3 = s2 * sc, s4 = s2 * s2;
        double S0 = (double)mom[0], S1 = (double)mom[1] / s1, S2 = (double)mom[2] / s2,
               S3 = (double)mom[3] / s3, S4 = (double)mom[4] / s4;
        double X0 = (double)mom[5], X1 = (double)mom[6] / s1, X2 = (double)mom[7] / s2;
        double A[3][3] = {{S4, S3, S2}, {S3, S2, S1}, {S2, S1, S0}};
        double b[3] = {X2, X1, X0}, q[3];
        if (solve3(A, b, q)) {
            double a = q[0] / s2;
            double bb = q[1] / s1 - 2.0 * a * yc;
            double c = q[2] - q[1] * yc / s1 + a * yc * yc;
            cf[0] = a; cf[1] = bb; cf[2] = c;
            return;
        }
    }
    // Rank-deficient input (pixels on fewer than 3 distinct rows): np.polyfit returns the
    // minimum-norm least-squares solution in its column-scaled basis [y^2, y, 1].
    *rank_def = 1;
    if (distinct <= 1) {
        double y0 = (double)ry[0], xm = (double)rsx[0] / (double)rn[0];
        double v[3] = {y0 * y0, y0, 1.0};
        for (int j = 0; j < 3; ++j) cf[j] = (v[j] != 0.0) ? xm / (3.0 * v[j]) : 0.0;
        if (y0 == 0.0) { cf[0] = 0.0; cf[1] = 0.0; cf[2] = xm; }
        return;
    }
    double y1 = (double)ry[0], y2 = (double)ry[1];
    double n1 = (double)rn[0], n2 = (double)rn[1];
    double m1 = (double)rsx[0] / n1, m2 = (double)rsx[1] / n2;
    double v1[3] = {y1 * y1, y1, 1.0}, v2[3] = {y2 * y2, y2, 1.0}, sc3[3], B1[3], B2[3];
    for (int j = 0; j < 3; ++j) {
        sc3[j] = sqrt(n1 * v1[j] * v1[j] + n2 * v2[j] * v2[j]);
        if (sc3[j] == 0.0) sc3[j] = 1.0;
        B1[j] = v1[j] / sc3[j];
        B2[j] = v2[j] / sc3[j];
    }
    double g11 = 0, g12 = 0, g22 = 0;
    for (int j = 0; j < 3; ++j) { g11 += B1[j] * B1[j]; g12 += B1[j] * B2[j]; g22 += B2[j] * B2[j]; }
    double det = g11 * g22 - g12 * g12;
    double l1 = (g22 * m1 - g12 * m2) / det, l2 = (g11 * m2 - g12 * m1) / det;
    for (int j = 0; j < 3; ++j) cf[j] = (B1[j] * l1 + B2[j] * l2) / sc3[j];
}

// check_validity (lane_tracker.py:561-627); nL/nR = lengths returned by get_poly_points(l, r, 1)
__device__ int validity(const double* l, const double* r, int nL, int nR, int W, double* diffs, const lt_validity& V) {
    int n = min(nL, nR);
    int y1 = W - 1, y2 = W - (int)mul64((double)n, 0.35), y3 = W - (int)mul64((double)n, 0.75);
    auto f = [&](const double* c, int y) {
        return add64(add64(mul64(c[0], (double)((long long)y * y)), mul64(c[1], (double)y)), c[2]);
    };
    double d1 = fabs(sub64(f(l, y1), f(r, y1))), d2 = fabs(sub64(f(l, y2), f(r, y2))), d3 = fabs(sub64(f(l, y3), f(r, y3)));
    diffs[0] = d1; diffs[1] = d2; diffs[2] = d3;
    if ((d1 < V.min_dist_y1) | (d1 > V.max_dist_y1) | (d2 < V.min_dist_y2) | (d2 > V.max_dist_y2) |
        (d3 < V.min_dist_y3) | (d3 > V.max_dist_y3)) return 0;
    auto g = [&](const double* c, int y) { return add64(mul64(mul64(2.0, c[0]), (double)y), c[1]); };
    double t1 = fabs(sub64(g(l, y1), g(r, y1))), t3 = fabs(sub64(g(l, y3), g(r, y3)));
    if ((t1 >= V.tangent_thresh) | (t3 >= V.tangent_thresh)) return 0;
    return 1;
}

// count of rows y in linspace(H(1-partial), H-1, int(H*partial)) with 0 <= f(y) <= W-1; optionally
// writes the kept x (truncated) in order to xs (ordered compaction).  All threads call.
__device__ int poly_points(const double* cf, double partial, int W, int H, int* xs, int* flags, int* scratch) {
    int num = (int)mul64((double)H, partial);
    double start = mul64((double)H, sub64(1.0, partial)), stop = (double)(H - 1);
    double step = (num > 1) ? __ddiv_rn(sub64(stop, start), (double)(num - 1)) : 0.0;
    for (int i = threadIdx.x; i < num; i += blockDim.x) {
        double y = add64(mul64((double)i, step), start);
        if (num > 1 && i == num - 1) y = stop;
        double fx = poly_eval(cf, y);
        flags[i] = (fx <= (double)(W - 1)) & (fx >= 0.0);
    }
    __syncthreads();
    if (!xs) {
        int c = 0;
        for (int i = threadIdx.x; i < num; i += blockDim.x) c += flags[i];
        return block_sum<int>(c, scratch);
    }
    // ordered compaction: remember flags, scan, scatter
    for (int i = threadIdx.x; i < num; i += blockDim.x) {
        if (flags[i]) {
            double y = add64(mul64((double)i, step), start);
            if (num > 1 && i == num - 1) y = stop;
            xs[H + i] = (int)poly_eval(cf, y);      // staging area behind the output (xs has 2*H ints)
        }
    }
    __syncthreads();
    int total = block_excl_scan(flags, num, scratch);
    for (int i = threadIdx.x; i < num; i += blockDim.x) {
        bool keep = (i + 1 < num ? flags[i + 1] : total) != flags[i];
        if (keep) xs[flags[i]] = xs[H + i];
    }
    __syncthreads();
    return total;
}

// ---------------------------------------------------------------------------
// search + fit + validity for one attempt
// ---------------------------------------------------------------------------

// PROF: position s takes its validity windows, and with prof_params its attempt parameters, from prof[pos_prof[s]]
// (the parameter profiles of the batch) instead of V and p.
template <bool PROF>
__global__ void __launch_bounds__(SEARCH_THREADS)
k_search(LtDims d, LtAttemptParams p, LtSearchArgs a, const LtDevState* __restrict__ state, int n_reset, lt_validity V,
         size_t bits_stride, const int* __restrict__ list, const int* __restrict__ count, int lev_chunk,
         const LtProfile* __restrict__ prof, const int* __restrict__ pos_prof, int prof_params) {
    int slot = blockIdx.x;
    if (count != nullptr && slot >= *count) return;
    const int s = list ? list[slot] : slot;              // batch position: mask, att, coeffs
    if (PROF) {
        const LtProfile& q = prof[pos_prof[s]];
        V = q.val;
        if (prof_params) p = q.p;
    }
    const int sid = a.ids ? a.ids[s] : s;                // state slot of its stream: state, by_stream outputs
    const int W = d.bv_w, H = d.bv_h, tid = threadIdx.x;
    const uint32_t* mask = a.mask + (size_t)s * bits_stride;
    const int oidx = a.by_stream ? sid : slot;

    extern __shared__ unsigned char smem_raw[];
    __shared__ SearchShared sh;
    __shared__ Roi rois[2][LT_MAX_LEVELS];
    __shared__ int cents[2][LT_MAX_LEVELS + 1];
    __shared__ int scratch[SEARCH_THREADS + 1];
    __shared__ long long scratch64[SEARCH_THREADS / 32];
    // per-row tables for both sides
    int* win_c0 = reinterpret_cast<int*>(smem_raw);     // [2][H]
    int* win_len = win_c0 + 2 * H;                      // [2][H]
    int* win_xoff = win_len + 2 * H;                    // [2][H]
    int* visit = win_xoff + 2 * H;                      // [2][H]  row visited v-th
    int* cnt = visit + 2 * H;                           // [2][H]  per visit: count -> offset
    int* Sbuf = cnt + 2 * H;                            // [W + 64]

    int mode = a.mode;
    if (mode == 0) mode = (state[sid].s.last_detection > n_reset) ? 1 : 2;
    if (tid == 0) {
        sh.nroi[0] = sh.nroi[1] = 0; sh.ncent[0] = sh.ncent[1] = 0; sh.nvisit[0] = sh.nvisit[1] = 0;
        if (mode == 2) {
            const double* cf = a.coeffs ? a.coeffs + (size_t)s * 6 : nullptr;
            for (int j = 0; j < 3; ++j) {
                sh.coeffs[0][j] = cf ? cf[j] : state[sid].s.last_left[j];
                sh.coeffs[1][j] = cf ? cf[3 + j] : state[sid].s.last_right[j];
            }
        }
    }
    __syncthreads();

    if (mode == 1) {
        // ------------------------------------------------------ sliding window search
        // Column histograms of every level are built by the whole CTA (bit-sliced, one task per level x mask word) and
        // turned into prefix sums; the walk itself -- sequential by nature: every level's search range depends on the
        // centroids found below it -- then needs two prefix-sum reads per candidate position and is done by warp 0
        // alone with shuffle reductions, without any CTA barrier.
        const int ww = p.window_width, wh = p.window_height, hw = ww / 2;
        const int Hh = H - p.ignore_bottom;
        const int cxi = W / 2;
        const int y0 = (int)mul64(sub64(1.0, p.start_slice), (double)Hh);
        const int nlev = min((int)__ddiv_rn(mul64(p.partial, (double)Hh), (double)wh), LT_MAX_LEVELS);
        const int warp = tid >> 5, lane = tid & 31, nwarp = blockDim.x >> 5;
        const int PW = W + 1;                                   // prefix-sum row: P[0..W]
        int* Pbuf = Sbuf + (W + 64);                            // [levels_per_chunk][PW]
        // walk state: replicated in the registers of every lane of warp 0 (all lanes compute the same values)
        int c[2] = {0, 0}, miss[2] = {0, 0}, rmin[2] = {-p.search_range, -p.search_range};
        int rmax[2] = {p.search_range, p.search_range}, ndiff[2] = {0, 0}, lastdiff[2] = {0, 0};
        int nroi[2] = {0, 0}, ncent[2] = {0, 0};
        {   // ---- level 0: one histogram of rows [y0, Hh) serves both sides
            int r0, r1;
            pyslice(y0, Hh, H, r0, r1);
            for (int w = tid; w < d.mwords; w += blockDim.x) hist_word(mask, d.mwords, r0, r1, w, min(32, W - w * 32), Pbuf + 1 + w * 32);
            __syncthreads();
            if (warp == 0) {
                warp_prefix_inplace(Pbuf, W, lane);
                for (int side = 0; side < 2; ++side) {
                    const int lo0 = side == 0 ? p.ignore_sides : cxi, hi0 = side == 0 ? cxi : W - p.ignore_sides;
                    int c0, c1;
                    pyslice(lo0, hi0, W, c0, c1);
                    const int nc = c1 - c0, nS = nc > 0 ? nc + ww - 1 : 0;
                    int smax, sfirst, slast;
                    warp_argmax(Pbuf, c0, nc, ww, 0, nS, lane, smax, sfirst, slast);
                    if (nS > 0 && smax > 0) {
                        c[side] = (sfirst + slast) / 2 - hw + lo0;
                        Roi r; const int ra = Hh - wh;
                        pyslice(ra, Hh, H, r.r0, r.r1);
                        pyslice(c[side] - hw, c[side] + hw, W, r.c0, r.c1);
                        r.xoff = (c[side] - hw) - r.c0;
                        if (lane == 0) rois[side][nroi[side]] = r;
                        nroi[side]++;
                    } else {
                        c[side] = (int)mul64((double)W, side == 0 ? 0.4 : 0.6);
                    }
                    if (lane == 0) cents[side][0] = c[side];
                    ncent[side] = 1;
                }
            }
            __syncthreads();
        }
        const int nS = W + ww - 1;
        for (int l0 = 1; l0 < nlev; l0 += lev_chunk) {
            const int nl = min(lev_chunk, nlev - l0);
            // histograms of the chunk's levels: task = (level, mask word)
            for (int t = tid; t < nl * d.mwords; t += blockDim.x) {
                const int lv = t / d.mwords, w = t - lv * d.mwords, level = l0 + lv;
                int r0, r1;
                pyslice(Hh - (1 + level) * wh, Hh - level * wh, H, r0, r1);
                hist_word(mask, d.mwords, r0, r1, w, min(32, W - w * 32), Pbuf + (size_t)lv * PW + 1 + w * 32);
            }
            __syncthreads();
            for (int lv = warp; lv < nl; lv += nwarp) warp_prefix_inplace(Pbuf + (size_t)lv * PW, W, lane);
            __syncthreads();
            if (warp == 0) {
                for (int lv = 0; lv < nl; ++lv) {
                    const int level = l0 + lv;
                    const int* P = Pbuf + (size_t)lv * PW;
                    int r0, r1;
                    pyslice(Hh - (1 + level) * wh, Hh - level * wh, H, r0, r1);
                    for (int side = 0; side < 2; ++side) {
                        if (miss[side] >= p.no_success_limit) continue;
                        const int lo = max(c[side] + rmin[side] + hw, 0), hi = min(c[side] + rmax[side] + hw, W);
                        int sa, sb;
                        pyslice(lo, hi, nS, sa, sb);
                        int smax, sfirst, slast;
                        warp_argmax(P, 0, W, ww, sa, sb, lane, smax, sfirst, slast);
                        const int o = 1 - side;
                        if (sb > sa && smax > 0) {
                            const int mc = (sfirst + slast + 1) / 2;            // ceil of the midpoint
                            const int prev = c[side];                           // == cents[side][ncent - 1]
                            c[side] = mc + lo - hw;
                            if (lane == 0) cents[side][ncent[side]] = c[side];
                            ncent[side]++;
                            lastdiff[side] = c[side] - prev;
                            ndiff[side]++;
                            miss[side] = 0;
                            Roi r;
                            r.r0 = r0; r.r1 = r1;
                            pyslice(c[side] - hw, c[side] + hw, W, r.c0, r.c1);
                            r.xoff = (c[side] - hw) - r.c0;
                            if (nroi[side] < LT_MAX_LEVELS) { if (lane == 0) rois[side][nroi[side]] = r; nroi[side]++; }
                            const int dd = (int)mul64(p.mu, (double)lastdiff[side]);
                            rmin[side] += dd; rmax[side] += dd;
                        } else {
                            if (ndiff[o] > 0 && miss[o] == 0) c[side] += lastdiff[o];
                            if (lane == 0) cents[side][ncent[side]] = c[side];
                            ncent[side]++;
                            miss[side]++;
                            if (miss[side] >= p.no_success_limit) ncent[side] = max(ncent[side] - p.no_success_limit, 0);
                        }
                    }
                }
            }
            __syncthreads();
        }
        if (tid == 0) { sh.nroi[0] = nroi[0]; sh.nroi[1] = nroi[1]; sh.ncent[0] = ncent[0]; sh.ncent[1] = ncent[1]; }
        __syncthreads();
        // expand the ROI lists into per-row windows in visiting order
        if (tid < 2) {
            int side = tid, v = 0;
            for (int k = 0; k < sh.nroi[side]; ++k) {
                Roi r = rois[side][k];
                for (int y = r.r0; y < r.r1; ++y) {
                    win_c0[side * H + y] = r.c0; win_len[side * H + y] = r.c1 - r.c0; win_xoff[side * H + y] = r.xoff;
                    visit[side * H + v++] = y;
                }
            }
            sh.nvisit[side] = v;
        }
        __syncthreads();
        if (a.centroids) {
            for (int side = 0; side < 2; ++side) {
                for (int i = tid; i < sh.ncent[side]; i += blockDim.x)
                    a.centroids[((size_t)oidx * 2 + side) * LT_MAX_LEVELS + i] = cents[side][i];
                if (tid == 0) a.ncentroids[oidx * 2 + side] = sh.ncent[side];
            }
        }
    } else {
        if (a.ncentroids && tid < 2) a.ncentroids[oidx * 2 + tid] = 0;
        // ------------------------------------------------------------------ band search
        int ystart = (int)mul64((double)H, sub64(1.0, p.partial));
        ystart = max(0, min(ystart, H));
        int yend = max(ystart, H - p.ignore_bottom);
        const double bw = (double)p.bandwidth;
        for (int side = 0; side < 2; ++side) {
            for (int v = tid; v < yend - ystart; v += blockDim.x) {
                int y = ystart + v;
                double f = poly_eval(sh.coeffs[side], (double)y);          // y**2 is exact in int64 and fp64 alike
                double lo = sub64(f, bw), hi = add64(f, bw);
                // integers x with lo < x < hi
                double xa_d = floor(lo) + 1.0, xb_d = ceil(hi) - 1.0;
                int xa = (int)fmax(xa_d, 0.0), xb = (int)fmin(xb_d, (double)(W - 1));
                if (!(xa_d <= xb_d) || xa > xb || !(lo == lo) || !(hi == hi)) { xa = 0; xb = -1; }
                win_c0[side * H + y] = xa; win_len[side * H + y] = xb - xa + 1; win_xoff[side * H + y] = 0;
                visit[side * H + v] = y;
            }
            if (tid == 0) sh.nvisit[side] = yend - ystart;
        }
        __syncthreads();
    }

    // ------------------------------------------------ counts, offsets, moments, pixel lists
    const double yc = (double)(H / 2);
    for (int side = 0; side < 2; ++side) {
        const int nv = sh.nvisit[side];
        long long m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        int dist = 0;
        for (int v = tid; v < nv; v += blockDim.x) {
            int y = visit[side * H + v];
            int c0 = win_c0[side * H + y], len = win_len[side * H + y];
            int sx = 0, n = 0;
            if (len > 0) n = row_bits(mask + (size_t)y * d.mwords, c0, c0 + len - 1, &sx);
            cnt[side * H + v] = n;
            if (n > 0) {
                long long sxr = (long long)sx + (long long)n * win_xoff[side * H + y];   // reported x
                long long t = y - (int)yc, t2 = t * t;
                m[0] += n; m[1] += n * t; m[2] += n * t2; m[3] += n * t2 * t; m[4] += n * t2 * t2;
                m[5] += sxr; m[6] += sxr * t; m[7] += sxr * t2;
                dist++;
            }
        }
        __syncthreads();
        for (int k = 0; k < 8; ++k) {
            long long r = block_sum<long long>(m[k], scratch64);
            if (tid == 0) sh.mom[side][k] = r;
        }
        int dtot = block_sum<int>(dist, scratch);
        if (tid == 0) sh.distinct[side] = dtot;
        __syncthreads();
        if (dtot > 0 && dtot <= 2 && tid == 0) {
            // remember the (at most two) populated rows for the rank-deficient fit
            int k = 0;
            for (int v = 0; v < nv && k < 2; ++v) {
                if (cnt[side * H + v] > 0) {
                    int y = visit[side * H + v], sx = 0;
                    int n = row_bits(mask + (size_t)y * d.mwords, win_c0[side * H + y],
                                     win_c0[side * H + y] + win_len[side * H + y] - 1, &sx);
                    sh.ry[side][k] = y; sh.rn[side][k] = n; sh.rsx[side][k] = sx + n * win_xoff[side * H + y];
                    ++k;
                }
            }
        }
        __syncthreads();
        int total = block_excl_scan(cnt + side * H, nv, scratch);
        if (tid == 0) sh.total[side] = total;
        if (a.pixels) {
            uint32_t* out = a.pixels + ((size_t)oidx * 2 + side) * a.pix_cap;
            for (int v = tid; v < nv; v += blockDim.x) {
                int y = visit[side * H + v];
                int c0 = win_c0[side * H + y], len = win_len[side * H + y], xo = win_xoff[side * H + y];
                int off = cnt[side * H + v];
                if (len <= 0) continue;
                const uint32_t* row = mask + (size_t)y * d.mwords;
                for (int w = c0 >> 5; w <= ((c0 + len - 1) >> 5); ++w) {
                    uint32_t bits = __ldg(&row[w]);
                    int lo = max(c0 - w * 32, 0), hi = min(c0 + len - 1 - w * 32, 31);
                    bits &= (hi == 31 ? 0xFFFFFFFFu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                    while (bits) {
                        int bpos = __ffs(bits) - 1;
                        bits &= bits - 1;
                        if (off < a.pix_cap) out[off] = ((uint32_t)y << 16) | (uint32_t)(w * 32 + bpos + xo + 32768);
                        ++off;
                    }
                }
            }
        }
        __syncthreads();
    }
    if (a.pix_counts && tid < 2) a.pix_counts[oidx * 2 + tid] = sh.total[tid];

    // ----------------------------------------------------------------- fit + validity
    const bool detected = sh.total[0] > 0 && sh.total[1] > 0;
    LtAttemptOut* out = a.att ? &a.att[s] : nullptr;
    __shared__ double fit[2][3];
    __shared__ int rankdef[2];
    if (detected && a.do_fit) {
        if (tid < 2)
            fit_from_moments(sh.mom[tid], yc, (double)H * 0.5, sh.distinct[tid], sh.ry[tid], sh.rn[tid], sh.rsx[tid],
                             fit[tid], &rankdef[tid]);
        __syncthreads();
        int* flags = cnt;   // reuse
        int nL = poly_points(fit[0], 1.0, W, H, nullptr, flags, scratch);
        int nR = poly_points(fit[1], 1.0, W, H, nullptr, flags, scratch);
        if (tid == 0 && out) {
            double diffs[3] = {0, 0, 0};
            out->valid = validity(fit[0], fit[1], nL, nR, W, diffs, V);
            for (int j = 0; j < 3; ++j) { out->fit[0][j] = fit[0][j]; out->fit[1][j] = fit[1][j]; out->diffs[j] = diffs[j]; }
            out->rank_def = rankdef[0] | (rankdef[1] << 1);
        }
    } else if (tid == 0 && out) {
        out->valid = 0; out->rank_def = 0;
        for (int j = 0; j < 3; ++j) { out->fit[0][j] = out->fit[1][j] = 0.0; out->diffs[j] = 0.0; }
    }
    if (tid == 0 && out) {
        out->detected = detected ? 1 : 0;
        out->mode = mode - 1;
        out->n[0] = sh.total[0]; out->n[1] = sh.total[1];
        out->partial = p.partial;
    }
}

static size_t search_smem(const LtDims& d) { return (size_t)(10 * d.bv_h + d.bv_w + 64 + 2 * d.bv_h) * sizeof(int); }

int lt_launch_search(lt_handle* h, int n, const LtAttemptParams& p, const LtSearchArgs& a, const int* list,
                     const int* count, cudaStream_t st, const LtProfile* prof, const int* pos_prof, int prof_params) {
    if (p.window_width < 1 || p.window_height < 1) { lt_set_error("window size must be positive"); return -1; }
    // + prefix-sum rows of the sliding-window levels: as many levels per chunk as fit next to the per-row tables
    const size_t base = search_smem(h->d), per_level = (size_t)(h->d.bv_w + 1) * sizeof(int), budget = 200 * 1024;
    int lev_chunk = base + per_level < budget ? (int)((budget - base) / per_level) : 1;
    lev_chunk = lev_chunk < 1 ? 1 : (lev_chunk > LT_MAX_LEVELS ? LT_MAX_LEVELS : lev_chunk);
    const size_t smem = base + (size_t)lev_chunk * per_level;
    if (prof) {
        { int rc = lt_ensure_smem((const void*)k_search<true>, smem); if (rc) return rc; }
        k_search<true><<<n, SEARCH_THREADS, smem, st>>>(h->d, p, a, h->state, h->cfg.n_reset, h->val, h->stream_mask, list, count,
                                                        lev_chunk, prof, pos_prof, prof_params);
    } else {
        { int rc = lt_ensure_smem((const void*)k_search<false>, smem); if (rc) return rc; }
        k_search<false><<<n, SEARCH_THREADS, smem, st>>>(h->d, p, a, h->state, h->cfg.n_reset, h->val, h->stream_mask, list, count,
                                                         lev_chunk, nullptr, nullptr, 0);
    }
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// attempt-2 selection (lane_tracker.py:1071)
// ---------------------------------------------------------------------------

// PROF: n_tries of position s is prof[pos_prof[s]].n_tries.  ORDER: the batch positions are order[0..n) (one round
// of a sequence batch) instead of 0..n-1.
template <bool PROF, bool ORDER>
__global__ void k_select_retry(const LtAttemptOut* __restrict__ att, int n, int n_tries, int* list, int* count,
                               int* flags, const LtProfile* __restrict__ prof, const int* __restrict__ pos_prof,
                               const int* __restrict__ order) {
    // single CTA, ordered compaction so that the retry list is deterministic
    if (threadIdx.x == 0) {
        int c = 0;
        for (int i = 0; i < n; ++i) {
            const int s = ORDER ? order[i] : i;
            if (PROF) n_tries = prof[pos_prof[s]].n_tries;
            bool retry = ((!att[s].detected) | (!att[s].valid)) & ((n_tries >= 2) | (n_tries == -1));
            flags[s] = retry;
            if (retry) list[c++] = s;
        }
        *count = c;
    }
}

int lt_launch_select_retry(lt_handle* h, int n, int n_tries, cudaStream_t st, const LtProfile* prof, const int* pos_prof,
                           const int* order) {
    if (prof)
        k_select_retry<true, false><<<1, 32, 0, st>>>(h->att, n, n_tries, h->retry_list, h->retry_count, h->draw_flags + h->S,
                                                      prof, pos_prof, nullptr);
    else if (order)
        k_select_retry<false, true><<<1, 32, 0, st>>>(h->att, n, n_tries, h->retry_list, h->retry_count, h->draw_flags + h->S,
                                                      nullptr, nullptr, order);
    else
        k_select_retry<false, false><<<1, 32, 0, st>>>(h->att, n, n_tries, h->retry_list, h->retry_count, h->draw_flags + h->S,
                                                       nullptr, nullptr, nullptr);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// lane polygon rows (cv2.fillPoly at lane_tracker.py:642-647) from the averaged polylines
// ---------------------------------------------------------------------------

__device__ void lane_rows_from_polylines(const int* xl, int nl, const int* xr, int nr, int W, int H, int2* rows,
                                         int4* bbox = nullptr) {
    // all threads of the CTA call; xl[i] is the vertex on row H-nl+i.  bbox (optional): bounding box of the non-empty
    // rows, (min lo, max hi, first row, last row) -- lets the overlay skip the frame pixels whose taps cannot hit the polygon.
    for (int y = threadIdx.x; y < H; y += blockDim.x) {
        int lo = W, hi = -1;
        auto cover = [&](int a, int b) { lo = min(lo, max(min(a, b), 0)); hi = max(hi, min(max(a, b), W - 1)); };
        int il = y - (H - nl), ir = y - (H - nr);
        bool hl = nl > 0 && nr > 0 && il >= 0, hr = nl > 0 && nr > 0 && ir >= 0;
        if (hl) cover(xl[il], xl[il]);
        if (hr) cover(xr[ir], xr[ir]);
        if (hl && hr) cover(xl[il], xr[ir]);
        // 8-connected outline between consecutive vertices of one polyline (cv::Line walks left to right):
        // for |dx| >= 2 the first floor(|dx|/2)+1 pixels stay on the row of the LEFT end point.
        auto edge = [&](const int* xs, int i, int nn) {      // vertex i on this row, neighbours i-1 and i+1
            for (int dlt = -1; dlt <= 1; dlt += 2) {
                int j = i + dlt;
                if (j < 0 || j >= nn) continue;
                int xa = min(max(xs[i], 0), W - 1), xb = min(max(xs[j], 0), W - 1);   // cv::clipLine, rows one apart
                int adx = abs(xb - xa);
                if (adx < 2) continue;
                int xleft = min(xa, xb), half = adx / 2;
                if (xa < xb) cover(xleft, xleft + half);                 // this row holds the left end
                else cover(xleft + half + 1, xleft + adx);               // this row holds the right end
            }
        };
        if (hl) edge(xl, il, nl);
        if (hr) edge(xr, ir, nr);
        rows[y] = make_int2(lo, hi);
    }
    __syncthreads();
    if (threadIdx.x == 0 && nl > 0 && nr > 0 && nl != nr) {
        // closing edge between the two top vertices: outline + 16.16 fixed-point scanline fill
        auto cover = [&](int y, int a, int b) {
            if (y < 0 || y >= H) return;
            int a2 = max(min(a, b), 0), b2 = min(max(a, b), W - 1);
            if (a2 > b2) return;
            rows[y].x = min(rows[y].x, a2); rows[y].y = max(rows[y].y, b2);
        };
        int xlt = xl[0], ylt = H - nl, xrt = xr[0], yrt = H - nr;
        {   // cv::LineIterator, left to right
            int x0 = xrt, y0 = yrt, x1 = xlt, y1 = ylt;
            if (x1 < x0) { int t = x0; x0 = x1; x1 = t; t = y0; y0 = y1; y1 = t; }
            int dx = x1 - x0, dy = y1 - y0, sy = dy >= 0 ? 1 : -1, ady = abs(dy);
            int x = x0, y = y0;
            if (dx >= ady) {
                int err = dx - 2 * ady;
                for (int i = 0; i <= dx; ++i) {
                    cover(y, x, x);
                    bool m = err < 0;
                    err += -2 * ady + (m ? 2 * dx : 0);
                    if (m) y += sy;
                    x += 1;
                }
            } else {
                int err = ady - 2 * dx;
                for (int i = 0; i <= ady; ++i) {
                    cover(y, x, x);
                    bool m = err < 0;
                    err += -2 * dx + (m ? 2 * ady : 0);
                    if (m) x += 1;
                    y += sy;
                }
            }
        }
        int tx, ty, bx, by; const int* side; int nside;
        if (ylt > yrt) { tx = xrt; ty = yrt; bx = xlt; by = ylt; side = xr; nside = nr; }
        else { tx = xlt; ty = ylt; bx = xrt; by = yrt; side = xl; nside = nl; }
        long long x = (long long)tx << 16, num = ((long long)bx - tx) << 16, den = by - ty;
        long long dxx = (num >= 0 ? num / den : -((-num) / den));
        for (int y = ty; y < by; ++y) {
            long long e = x, sv = (long long)side[y - (H - nside)] << 16;
            long long lo = min(e, sv), hi = max(e, sv);
            int xs = (int)((lo + 65535) >> 16), xe = (int)(hi >> 16);
            if (xs <= xe) cover(y, xs, xe);
            x += dxx;
        }
    }
    __syncthreads();
    if (bbox) {
        __shared__ int sb[4];
        if (threadIdx.x == 0) { sb[0] = W; sb[1] = -1; sb[2] = H; sb[3] = -1; }
        __syncthreads();
        int lo = W, hi = -1, y0 = H, y1 = -1;
        for (int y = threadIdx.x; y < H; y += blockDim.x) {
            const int2 r = rows[y];
            if (r.x <= r.y) { lo = min(lo, r.x); hi = max(hi, r.y); y0 = min(y0, y); y1 = max(y1, y); }
        }
        if (hi >= 0) { atomicMin(&sb[0], lo); atomicMax(&sb[1], hi); atomicMin(&sb[2], y0); atomicMax(&sb[3], y1); }
        __syncthreads();
        if (threadIdx.x == 0) *bbox = make_int4(sb[0], sb[1], sb[2], sb[3]);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// per-frame state update (lane_tracker.py:1142-1209)
// ---------------------------------------------------------------------------

// What the overlay and the text of one frame read, per batch position (LtSeqSnap): the update of a round of a sequence
// batch copies them out of the stream's slot before a later frame of the stream overwrites it.
struct LtSeqSnap {
    int2* rows;                  // [S][bv_h] lane polygon rows: this frame's on a valid frame, the stream's cache otherwise
    int4* bbox;                  // [S] their bounding box
    LtDevState* state;           // [S] the stream's state after this frame (k_text formats from it)
};

// CAMS: position s takes mppv / mpph from its camera, cams[pos_cam[s]] (the handle's cfg otherwise).
// SEQ: CTA b updates batch position order[b] (one round of a sequence batch) and writes its snapshot to snap.
template <bool CAMS, bool SEQ>
__global__ void __launch_bounds__(SEARCH_THREADS)
k_update_state(LtDims d, lt_config cfg, LtDevState* __restrict__ state, const LtAttemptOut* __restrict__ att1,
               const LtAttemptOut* __restrict__ att2, const int* __restrict__ retry, int* __restrict__ avg_x,
               int2* __restrict__ lane_rows, int4* __restrict__ lane_bbox, int* __restrict__ draw, lt_result* __restrict__ results,
               const int* __restrict__ ids, const LtCamDev* __restrict__ cams, const int* __restrict__ pos_cam,
               const int* __restrict__ order, LtSeqSnap snap) {
    // s: batch position (attempt outputs, retry and draw flags, result record); sid: state slot of its stream
    const int s = SEQ ? order[blockIdx.x] : blockIdx.x, sid = ids ? ids[s] : s, tid = threadIdx.x, W = d.bv_w, H = d.bv_h;
    extern __shared__ unsigned char smem_raw[];
    int* flags = reinterpret_cast<int*>(smem_raw);        // [H]
    int* stage = flags + H;                               // [2*H]
    __shared__ int scratch[SEARCH_THREADS + 1];
    __shared__ double avg[2][3];
    __shared__ int nkeep[2];
    lt_state& st = state[sid].s;
    const bool second = retry && retry[s];
    const LtAttemptOut& a = second ? att2[s] : att1[s];
    const bool valid = a.detected && a.valid;
    const int nav = min(max(cfg.n_average, 1), LT_MAX_AVERAGE);
    int* xl = avg_x + (size_t)sid * 2 * H;
    int* xr = xl + H;

    if (tid == 0) {
        st.counter += 1;
        // ring append + trim (lane_tracker.py:1145-1156 / 1180-1188)
        if (st.ring_len == nav) {
            for (int i = 1; i < nav; ++i) {
                st.ring_empty[i - 1] = st.ring_empty[i];
                for (int j = 0; j < 3; ++j) { st.ring_left[i - 1][j] = st.ring_left[i][j]; st.ring_right[i - 1][j] = st.ring_right[i][j]; }
            }
            st.ring_len = nav - 1;
        }
        int k = st.ring_len++;
        st.ring_empty[k] = valid ? 0 : 1;
        for (int j = 0; j < 3; ++j) { st.ring_left[k][j] = valid ? a.fit[0][j] : 0.0; st.ring_right[k][j] = valid ? a.fit[1][j] : 0.0; }
        if (!valid) {
            if (st.radii_len == nav) { for (int i = 1; i < nav; ++i) st.radii[i - 1] = st.radii[i]; st.radii_len = nav - 1; }
            st.radii[st.radii_len++] = -1;
            st.last_detection += 1;
        } else {
            for (int j = 0; j < 3; ++j) { st.last_left[j] = a.fit[0][j]; st.last_right[j] = a.fit[1][j]; }
            st.has_last = 1;
            st.last_detection = 0;
            st.success += 1;
            // np.average over the non-empty ring entries, in order
            double sl[3] = {0, 0, 0}, sr[3] = {0, 0, 0}; int c = 0;
            for (int i = 0; i < st.ring_len; ++i) {
                if (st.ring_empty[i]) continue;
                for (int j = 0; j < 3; ++j) {
                    sl[j] = c ? add64(sl[j], st.ring_left[i][j]) : st.ring_left[i][j];
                    sr[j] = c ? add64(sr[j], st.ring_right[i][j]) : st.ring_right[i][j];
                }
                ++c;
            }
            for (int j = 0; j < 3; ++j) {
                st.left_avg[j] = __ddiv_rn(sl[j], (double)c); st.right_avg[j] = __ddiv_rn(sr[j], (double)c);
                avg[0][j] = st.left_avg[j]; avg[1][j] = st.right_avg[j];
            }
            st.has_avg = 1;
        }
    }
    __syncthreads();
    if (valid) {
        // averaged polylines (get_poly_points with the attempt's `partial`, lane_tracker.py:1199)
        for (int side = 0; side < 2; ++side) {
            int* xs = side == 0 ? xl : xr;
            int n = poly_points(avg[side], a.partial, W, H, stage, flags, scratch);
            for (int i = tid; i < n; i += blockDim.x) xs[i] = stage[i];
            if (tid == 0) nkeep[side] = n;
            __syncthreads();
        }
        if (tid == 0) {
            st.n_left_avg = nkeep[0]; st.n_right_avg = nkeep[1];
            // get_curve_radius (lane_tracker.py:530-549): the metric refit of the same pixels is the
            // analytic rescaling a' = a*mpph/mppv^2, b' = b*mpph/mppv of this frame's fit
            long long rad[2];
            double mppv = cfg.mppv, mpph = cfg.mpph;
            if (CAMS) {
                const LtCamDev& cd = cams[pos_cam[s]];
                mppv = cd.mppv; mpph = cd.mpph;
            }
            for (int side = 0; side < 2; ++side) {
                double am = a.fit[side][0] * mpph / (mppv * mppv), bm = a.fit[side][1] * mpph / mppv;
                double g = 2.0 * am * (double)H * mppv + bm;
                double r = pow(1.0 + g * g, 1.5) / fabs(2.0 * am);
                rad[side] = (!(r == r) || r >= 9.2233720368547758e18) ? 0x7FFFFFFFFFFFFFFFLL : (long long)r;   // int(float)
            }
            long long avr = (long long)(0.5 * (double)(rad[0] + rad[1]));           // int(0.5 * (l + r))
            if (st.radii_len == nav) { for (int i = 1; i < nav; ++i) st.radii[i - 1] = st.radii[i]; st.radii_len = nav - 1; }
            st.radii[st.radii_len++] = avr;
            // int(np.average(radii > 0)): float64 accumulation in NumPy's order (pairwise unrolled by 8 for n == 8)
            double v[LT_MAX_AVERAGE]; int c = 0;
            for (int i = 0; i < st.radii_len; ++i) if (st.radii[i] > 0) v[c++] = (double)st.radii[i];
            double sum = 0.0;
            if (c == 8) sum = add64(add64(add64(v[0], v[1]), add64(v[2], v[3])), add64(add64(v[4], v[5]), add64(v[6], v[7])));
            else for (int i = 0; i < c; ++i) sum = i ? add64(sum, v[i]) : v[0];
            st.average_curve_radius = c ? (long long)__ddiv_rn(sum, (double)c) : -1;
            results[s].left_curve_radius = rad[0]; results[s].right_curve_radius = rad[1];
            // get_eccentricity (lane_tracker.py:551-559)
            if (nkeep[0] > 0 && nkeep[1] > 0) {
                int mid = W / 2, left = xl[nkeep[0] - 1], right = xr[nkeep[1] - 1];
                st.eccentricity = mul64((double)((mid - left) - (right - mid)) / 2.0, mpph);
            }
        }
        __syncthreads();
        lane_rows_from_polylines(xl, st.n_left_avg, xr, st.n_right_avg, W, H, lane_rows + (size_t)sid * H, lane_bbox + sid);
    }
    if (tid == 0) {
        int drew = valid ? 1 : ((st.has_avg && st.n_left_avg != 0 && st.last_detection <= cfg.n_fail) ? 1 : 0);
        draw[s] = drew;
        lt_result& r = results[s];
        r.counter = st.counter; r.attempts = second ? 2 : 1; r.search_mode = a.mode; r.detected_pixels = a.detected;
        r.valid_lane_lines = valid ? 1 : 0; r.last_detection = st.last_detection; r.drew_lane = drew;
        r.n_left = a.n[0]; r.n_right = a.n[1]; r.n_left_avg = st.n_left_avg; r.n_right_avg = st.n_right_avg;
        if (!valid) { r.left_curve_radius = 0; r.right_curve_radius = 0; }
        r.average_curve_radius = st.average_curve_radius; r.success = st.success; r.fit_rank_deficient = a.rank_def;
        for (int j = 0; j < 3; ++j) {
            r.left_fit[j] = a.fit[0][j]; r.right_fit[j] = a.fit[1][j];
            r.left_avg[j] = st.left_avg[j]; r.right_avg[j] = st.right_avg[j]; r.validity_d[j] = a.diffs[j];
        }
        r.eccentricity = st.eccentricity;
        const LtAttemptOut& f1 = att1[s];
        r.first_detected = f1.detected; r.first_valid = (f1.detected && f1.valid) ? 1 : 0;
        r.first_n_left = f1.n[0]; r.first_n_right = f1.n[1];
        for (int j = 0; j < 3; ++j) { r.first_left_fit[j] = f1.fit[0][j]; r.first_right_fit[j] = f1.fit[1][j]; }
    }
    if (SEQ) {
        static_assert(sizeof(LtDevState) % sizeof(int) == 0, "LtDevState is copied as words");
        __syncthreads();                                  // the rows, box and state of this frame are complete
        for (int y = tid; y < H; y += blockDim.x) snap.rows[(size_t)s * H + y] = lane_rows[(size_t)sid * H + y];
        if (tid == 0) snap.bbox[s] = lane_bbox[sid];
        const int* src = reinterpret_cast<const int*>(state + sid);
        int* dst = reinterpret_cast<int*>(snap.state + s);
        for (int i = tid; i < (int)(sizeof(LtDevState) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
    }
}

int lt_launch_update_state(lt_handle* h, int n, const int* ids, lt_result* d_results, int attempts_allowed,
                           cudaStream_t st, const LtFrontSet* cf, const int* order) {
    size_t smem = (size_t)3 * h->d.bv_h * sizeof(int);
    const int* retry = attempts_allowed >= 2 ? h->draw_flags + h->S : nullptr;
    const LtSeqSnap none = {nullptr, nullptr, nullptr};
    if (cf)
        k_update_state<true, false><<<n, SEARCH_THREADS, smem, st>>>(h->d, h->cfg, h->state, h->att, h->att + h->S, retry,
                                                                     h->avg_x, h->lane_rows, h->lane_bbox, h->draw_flags,
                                                                     d_results, ids, cf->cams, cf->pos_cam, nullptr, none);
    else if (order)
        k_update_state<false, true><<<n, SEARCH_THREADS, smem, st>>>(h->d, h->cfg, h->state, h->att, h->att + h->S, retry,
                                                                     h->avg_x, h->lane_rows, h->lane_bbox, h->draw_flags,
                                                                     d_results, ids, nullptr, nullptr, order,
                                                                     {h->seq_rows, h->seq_bbox, h->seq_state});
    else
        k_update_state<false, false><<<n, SEARCH_THREADS, smem, st>>>(h->d, h->cfg, h->state, h->att, h->att + h->S, retry,
                                                                      h->avg_x, h->lane_rows, h->lane_bbox, h->draw_flags,
                                                                      d_results, ids, nullptr, nullptr, nullptr, none);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// stand-alone stage kernels behind the API methods
// ---------------------------------------------------------------------------

// fit_poly on explicit pixel lists (lane_tracker.py:502-509)
__global__ void __launch_bounds__(SEARCH_THREADS)
k_fit_pixels(const uint32_t* __restrict__ pixels, int cap, const int* __restrict__ counts, int H, double* __restrict__ fits) {
    const int s = blockIdx.x, side = blockIdx.y, tid = threadIdx.x;
    __shared__ long long scratch64[SEARCH_THREADS / 32];
    __shared__ long long mom[8];
    __shared__ int ymin, ymax, ymid_flag;
    const uint32_t* px = pixels + ((size_t)s * 2 + side) * cap;
    const int n = min(counts[s * 2 + side], cap);
    const int yc = H / 2;
    if (tid == 0) { ymin = 0x7FFFFFFF; ymax = -1; ymid_flag = 0; }
    __syncthreads();
    long long m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int lmin = 0x7FFFFFFF, lmax = -1;
    for (int i = tid; i < n; i += blockDim.x) {
        uint32_t v = px[i];
        int y = (int)(v >> 16), x = (int)(v & 0xFFFFu) - 32768;
        long long t = y - yc, t2 = t * t;
        m[0] += 1; m[1] += t; m[2] += t2; m[3] += t2 * t; m[4] += t2 * t2;
        m[5] += x; m[6] += x * t; m[7] += x * t2;
        lmin = min(lmin, y); lmax = max(lmax, y);
    }
    if (lmax >= 0) { atomicMin(&ymin, lmin); atomicMax(&ymax, lmax); }
    for (int k = 0; k < 8; ++k) {
        long long r = block_sum<long long>(m[k], scratch64);
        if (tid == 0) mom[k] = r;
    }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        int y = (int)(px[i] >> 16);
        if (y != ymin && y != ymax) ymid_flag = 1;
    }
    __syncthreads();
    if (tid == 0) {
        double* cf = fits + ((size_t)s * 2 + side) * 3;
        if (n == 0) { cf[0] = cf[1] = cf[2] = 0.0; return; }
        int distinct = ymid_flag ? 3 : (ymin == ymax ? 1 : 2);
        int ry[2] = {ymin, ymax}, rn[2] = {0, 0}, rsx[2] = {0, 0};
        if (distinct < 3)
            for (int i = 0; i < n; ++i) {
                int y = (int)(px[i] >> 16), x = (int)(px[i] & 0xFFFFu) - 32768;
                int k = (y == ymin) ? 0 : 1;
                rn[k]++; rsx[k] += x;
            }
        int rd;
        fit_from_moments(mom, (double)yc, (double)H * 0.5, distinct, ry, rn, rsx, cf, &rd);
    }
}

int lt_launch_fit_pixels(lt_handle* h, const uint32_t* d_pixels, int cap, const int* d_counts, int n, double* d_fits,
                         cudaStream_t st) {
    k_fit_pixels<<<dim3(n, 2), SEARCH_THREADS, 0, st>>>(d_pixels, cap, d_counts, h->d.bv_h, d_fits);
    LT_LAUNCH_CHECK();
    return 0;
}

__global__ void __launch_bounds__(SEARCH_THREADS)
k_validity(LtDims d, const double* __restrict__ fits, int* __restrict__ valid, double* __restrict__ diffs, lt_validity V) {
    const int s = blockIdx.x;
    extern __shared__ unsigned char smem_raw[];
    int* flags = reinterpret_cast<int*>(smem_raw);
    __shared__ int scratch[SEARCH_THREADS + 1];
    __shared__ double cf[2][3];
    if (threadIdx.x < 6) cf[threadIdx.x / 3][threadIdx.x % 3] = fits[(size_t)s * 6 + threadIdx.x];
    __syncthreads();
    int nL = poly_points(cf[0], 1.0, d.bv_w, d.bv_h, nullptr, flags, scratch);
    int nR = poly_points(cf[1], 1.0, d.bv_w, d.bv_h, nullptr, flags, scratch);
    if (threadIdx.x == 0) {
        double dd[3];
        valid[s] = validity(cf[0], cf[1], nL, nR, d.bv_w, dd, V);
        if (diffs) for (int j = 0; j < 3; ++j) diffs[(size_t)s * 3 + j] = dd[j];
    }
}

int lt_launch_validity(lt_handle* h, const double* d_fits, int n, int* d_valid, double* d_diffs, cudaStream_t st) {
    k_validity<<<n, SEARCH_THREADS, (size_t)h->d.bv_h * sizeof(int), st>>>(h->d, d_fits, d_valid, d_diffs, h->val);
    LT_LAUNCH_CHECK();
    return 0;
}

__global__ void __launch_bounds__(SEARCH_THREADS)
k_poly_points(LtDims d, const double* __restrict__ fits, double partial, int* __restrict__ xs_out, int* __restrict__ counts) {
    const int s = blockIdx.x, side = blockIdx.y, H = d.bv_h;
    extern __shared__ unsigned char smem_raw[];
    int* flags = reinterpret_cast<int*>(smem_raw);
    int* stage = flags + H;
    __shared__ int scratch[SEARCH_THREADS + 1];
    __shared__ double cf[3];
    if (threadIdx.x < 3) cf[threadIdx.x] = fits[((size_t)s * 2 + side) * 3 + threadIdx.x];
    __syncthreads();
    int n = poly_points(cf, partial, d.bv_w, H, stage, flags, scratch);
    int* out = xs_out + ((size_t)s * 2 + side) * H;
    for (int i = threadIdx.x; i < H; i += blockDim.x) out[i] = i < n ? stage[i] : 0;
    if (threadIdx.x == 0) counts[s * 2 + side] = n;
}

int lt_launch_poly_points(lt_handle* h, const double* d_fits, int n, double partial, int* d_x, int* d_counts,
                          cudaStream_t st) {
    k_poly_points<<<dim3(n, 2), SEARCH_THREADS, (size_t)3 * h->d.bv_h * sizeof(int), st>>>(h->d, d_fits, partial, d_x,
                                                                                          d_counts);
    LT_LAUNCH_CHECK();
    return 0;
}

__global__ void __launch_bounds__(SEARCH_THREADS)
k_lane_rows(LtDims d, const int* __restrict__ xs, const int* __restrict__ counts, int2* __restrict__ lane_rows,
            int4* __restrict__ lane_bbox, int* __restrict__ draw) {
    const int s = blockIdx.x, H = d.bv_h;
    const int* xl = xs + (size_t)s * 2 * H;
    lane_rows_from_polylines(xl, counts[s * 2], xl + H, counts[s * 2 + 1], d.bv_w, H, lane_rows + (size_t)s * H, lane_bbox + s);
    if (threadIdx.x == 0) draw[s] = 1;
}

int lt_launch_lane_rows(lt_handle* h, const int* d_x, const int* d_counts, int n, cudaStream_t st) {
    k_lane_rows<<<n, SEARCH_THREADS, 0, st>>>(h->d, d_x, d_counts, h->lane_rows, h->lane_bbox, h->draw_flags);
    LT_LAUNCH_CHECK();
    return 0;
}

// Row spans of the two search-band polygons of visualize_band_search (lane_tracker.py:749-760): the polylines of
// get_poly_points(last coeffs, partial) shifted by -/+ bandwidth.  Vertices may leave the canvas; cv::Line clips an edge
// before it rasterises it, which for one-row-apart vertices equals clamping x (lane_rows_from_polylines).
__global__ void __launch_bounds__(SEARCH_THREADS)
k_band_rows(LtDims d, const int* __restrict__ xs, const int* __restrict__ counts, int bandwidth, int2* __restrict__ rows_l,
            int2* __restrict__ rows_r) {
    const int H = d.bv_h;
    extern __shared__ unsigned char smem_raw[];
    int* lo = reinterpret_cast<int*>(smem_raw);
    int* hi = lo + H;
    for (int side = 0; side < 2; ++side) {
        const int n = counts[side];
        for (int i = threadIdx.x; i < n; i += blockDim.x) { int x = xs[side * H + i]; lo[i] = x - bandwidth; hi[i] = x + bandwidth; }
        __syncthreads();
        lane_rows_from_polylines(lo, n, hi, n, d.bv_w, H, side ? rows_r : rows_l);
        __syncthreads();
    }
}

int lt_launch_band_rows(lt_handle* h, const int* d_x, const int* d_counts, int bandwidth, int2* rows_l, int2* rows_r,
                        cudaStream_t st) {
    k_band_rows<<<1, SEARCH_THREADS, (size_t)2 * h->d.bv_h * sizeof(int), st>>>(h->d, d_x, d_counts, bandwidth, rows_l, rows_r);
    LT_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// text overlays (cv2.putText at lane_tracker.py:653-659, 668-672) from glyph sprites
// ---------------------------------------------------------------------------

struct TextLine { int x0, y0, len; unsigned char ch[56]; };

__device__ void put_str(TextLine& l, const char* s) { while (*s && l.len < 55) l.ch[l.len++] = (unsigned char)*s++; }
__device__ void put_int(TextLine& l, long long v) {                    // "{}".format(int)
    char buf[24]; int n = 0;
    unsigned long long u = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
    while (u > 0xFFFFFFFFull) { buf[n++] = (char)('0' + (int)(u % 10ull)); u /= 10ull; }   // rare: 64-bit digits
    unsigned int w = (unsigned int)u;                                                      // common: 32-bit digits
    do { buf[n++] = (char)('0' + (int)(w % 10u)); w /= 10u; } while (w);
    if (v < 0 && l.len < 55) l.ch[l.len++] = '-';
    while (n && l.len < 55) l.ch[l.len++] = (unsigned char)buf[--n];
}
__device__ void put_fixed2(TextLine& l, double x) {                    // "{:.2f}".format(float): exact half-even
    if (!(x == x)) { put_str(l, "nan"); return; }
    if (signbit(x)) put_str(l, "-");
    double v = fabs(x);
    if (!(v < 1e15)) { put_str(l, "inf"); return; }
    double t = mul64(v, 100.0), e = fma(v, 100.0, -t);                 // t + e == v * 100 exactly
    double r = floor(t), frac = add64(sub64(t, r), e);
    if (frac > 0.5 || (frac == 0.5 && fmod(r, 2.0) != 0.0)) r += 1.0;
    if (frac < 0.0) {                                                    // product rounded up across an integer
        double fr2 = add64(1.0, frac);
        r -= 1.0;
        if (fr2 > 0.5 || (fr2 == 0.5 && fmod(r, 2.0) != 0.0)) r += 1.0;
    }
    long long cents = (long long)r;
    put_int(l, cents / 100);
    put_str(l, ".");
    char d2[3] = {(char)('0' + (int)((cents / 10) % 10)), (char)('0' + (int)(cents % 10)), 0};
    put_str(l, d2);
}

// Sequential reference form: glyph after glyph (string order matters where neighbouring glyphs overlap).
__global__ void __launch_bounds__(128)
k_text_seq(uint8_t* out, LtDims d, const LtDevState* __restrict__ state, const int* __restrict__ draw, int print_frame_count,
           const uint8_t* __restrict__ tables, const int* __restrict__ char_start, const short* __restrict__ dy,
           const short* __restrict__ dx, const unsigned short* __restrict__ lut, const int* __restrict__ advance,
           int nchars, int first_char, const int* __restrict__ ids);

__device__ int format_lines(TextLine* lines, const lt_state& st, int drew, int print_frame_count) {
    for (int i = 0; i < 3; ++i) { lines[i].len = 0; lines[i].x0 = 20; lines[i].y0 = 35 + 35 * i; }
    int n = 0;
    if (drew) {                                                         // draw_lane, lane_tracker.py:653-659
        put_str(lines[0], "Curve Radius: "); put_int(lines[0], st.average_curve_radius); put_str(lines[0], " m");
        put_str(lines[1], "Eccentricity: "); put_fixed2(lines[1], st.eccentricity); put_str(lines[1], " m");
        n = 2;
    } else {                                                            // print_failure, lane_tracker.py:668-672
        put_str(lines[0], "Lane Line Detection Failed");
        n = 1;
    }
    if (print_frame_count) { put_str(lines[n], "Frame: "); put_int(lines[n], (long long)st.counter - 1); ++n; }
    return n;
}

__global__ void __launch_bounds__(128)
k_text_seq(uint8_t* out, LtDims d, const LtDevState* __restrict__ state, const int* __restrict__ draw, int print_frame_count,
           const uint8_t* __restrict__ tables, const int* __restrict__ char_start, const short* __restrict__ dy,
           const short* __restrict__ dx, const unsigned short* __restrict__ lut, const int* __restrict__ advance,
           int nchars, int first_char, const int* __restrict__ ids) {
    const int s = blockIdx.x;                       // batch position: frame, draw flag; the strings from the stream's state
    __shared__ TextLine lines[3];
    __shared__ int nlines;
    if (threadIdx.x == 0) nlines = format_lines(lines, state[ids ? ids[s] : s].s, draw[s], print_frame_count);
    __syncthreads();
    uint8_t* img = out + (size_t)s * d.img_w * d.img_h * 3;
    for (int li = 0; li < nlines; ++li) {
        int x = lines[li].x0;
        const int y0 = lines[li].y0;
        for (int ci = 0; ci < lines[li].len; ++ci) {
            int c = (int)lines[li].ch[ci] - first_char;
            if (c < 0 || c >= nchars) c = '?' - first_char;
            const int a = char_start[c], b = char_start[c + 1];
            for (int p = a + threadIdx.x; p < b; p += blockDim.x) {
                const int yy = y0 + dy[p], xx = x + dx[p];
                if ((unsigned)yy < (unsigned)d.img_h && (unsigned)xx < (unsigned)d.img_w) {
                    uint8_t* px = img + ((size_t)yy * d.img_w + xx) * 3;
                    const uint8_t* t = tables + (size_t)lut[p] * 256;
                    px[0] = t[px[0]]; px[1] = t[px[1]]; px[2] = t[px[2]];
                }
            }
            x += advance[c];
            __syncthreads();
        }
    }
}

// Parallel form: one CTA per (stream, line); every (glyph, pixel) of the line is an independent work item, except the
// pixels a glyph shares with its predecessor (flagged pairs only): those are applied in a second phase, on top of
// the predecessor's result.  Preconditions (checked on the host when the sprites are installed): the three lines
// occupy disjoint rows and a glyph can only overlap its immediate neighbour.
__global__ void __launch_bounds__(1024)
k_text(uint8_t* out, LtDims d, const LtDevState* __restrict__ state, const int* __restrict__ draw, int print_frame_count,
       const uint8_t* __restrict__ tables, const int* __restrict__ char_start, const short* __restrict__ dy,
       const short* __restrict__ dx, const unsigned short* __restrict__ lut, const int* __restrict__ advance,
       const unsigned char* __restrict__ pair_overlap, const unsigned long long* __restrict__ bitmaps, int nchars,
       int first_char, const int* __restrict__ ids) {
    const int s = blockIdx.x, li = blockIdx.y;      // batch position: frame, draw flag; the strings from the stream's state
    __shared__ TextLine lines[3];
    __shared__ int nlines;
    __shared__ int cx[56], cc[56], cstart[57], cflag[56];
    __shared__ int s_start[130], s_adv[129];                       // glyph index tables (<= 128 glyphs), off the
    const int ng = min(nchars, 128);                               // serial path of thread 0
    for (int i = threadIdx.x; i <= ng; i += blockDim.x) s_start[i] = char_start[i];
    for (int i = threadIdx.x; i < ng; i += blockDim.x) s_adv[i] = advance[i];
    if (threadIdx.x == 0) nlines = format_lines(lines, state[ids ? ids[s] : s].s, draw[s], print_frame_count);
    __syncthreads();
    if (li >= nlines) return;
    if (threadIdx.x == 0) {
        int x = lines[li].x0, tot = 0;
        for (int ci = 0; ci < lines[li].len; ++ci) {
            int c = (int)lines[li].ch[ci] - first_char;
            if (c < 0 || c >= ng) c = '?' - first_char;
            cc[ci] = c; cx[ci] = x; cstart[ci] = tot;
            tot += s_start[c + 1] - s_start[c];
            x += s_adv[c];
        }
        cstart[lines[li].len] = tot;
    }
    __syncthreads();
    for (int ci = threadIdx.x; ci < lines[li].len; ci += blockDim.x)
        cflag[ci] = ci > 0 ? (int)pair_overlap[cc[ci - 1] * nchars + cc[ci]] : 0;
    __syncthreads();
    uint8_t* img = out + (size_t)s * d.img_w * d.img_h * 3;
    const int nch = lines[li].len, y0 = lines[li].y0, total = cstart[nch];
    for (int phase = 0; phase < 2; ++phase) {
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int ci = 0;
            while (cstart[ci + 1] <= w) ++ci;                              // <= 56 glyphs: linear search
            const int c = cc[ci], p = s_start[c] + (w - cstart[ci]);
            const int yy = y0 + dy[p], xx = cx[ci] + dx[p];
            bool shared_px = false;
            if (cflag[ci]) {                                                // is this pixel also in the previous glyph?
                const int pc = cc[ci - 1], ry = dy[p] + 32, rx = xx - cx[ci - 1] + 8;      // 64x64 glyph bitmaps
                if ((unsigned)ry < 64u && (unsigned)rx < 64u) shared_px = (bitmaps[pc * 64 + ry] >> rx) & 1ull;
            }
            if ((int)shared_px != phase) continue;
            if ((unsigned)yy < (unsigned)d.img_h && (unsigned)xx < (unsigned)d.img_w) {
                uint8_t* px = img + ((size_t)yy * d.img_w + xx) * 3;
                const uint8_t* t = tables + (size_t)lut[p] * 256;
                px[0] = t[px[0]]; px[1] = t[px[1]]; px[2] = t[px[2]];
            }
        }
        __syncthreads();
    }
}

int lt_launch_text(lt_handle* h, uint8_t* d_out, int n, const int* ids, cudaStream_t st) {
    if (!h->txt_tables || !d_out) return 0;
    if (h->txt_parallel_lines && h->txt_pair_overlap && h->txt_bitmaps)
        k_text<<<dim3(n, 3), 1024, 0, st>>>(d_out, h->d, h->state, h->draw_flags, h->cfg.print_frame_count, h->txt_tables,
                                           h->txt_char_start, h->txt_dy, h->txt_dx, h->txt_lut, h->txt_advance,
                                           h->txt_pair_overlap, h->txt_bitmaps, h->txt_nchars, h->txt_first, ids);
    else
        k_text_seq<<<n, 128, 0, st>>>(d_out, h->d, h->state, h->draw_flags, h->cfg.print_frame_count, h->txt_tables,
                                      h->txt_char_start, h->txt_dy, h->txt_dx, h->txt_lut, h->txt_advance, h->txt_nchars,
                                      h->txt_first, ids);
    LT_LAUNCH_CHECK();
    return 0;
}
