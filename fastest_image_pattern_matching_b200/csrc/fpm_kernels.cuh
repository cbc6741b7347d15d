// fpm_kernels.cuh -- hand-written sm_100a kernels for every stage of TemplateMatcher::match
// (/root/reference/src/TemplateMatcher.cpp:97-437).  One kernel per reference stage:
//
//   fpm_pyrdown_kernel        cv::buildPyramid / pyrDown, 1 or 2 levels/launch (:55, :124)   [fpm_pyrdown.cuh]
//   fpm_warp_kernel           cv::warpAffine INTER_LINEAR, BORDER_CONSTANT    (:175, :1089)
//   fpm_top_score_kernel      matchTemplate(TM_CCORR) + CCOEFF_Denominator    (:177, :514, :527-598)
//   fpm_top_peaks_kernel      minMaxLoc / s_BlockMax / getNextMaxLoc          (:179-210, :1196-1221)
//   fpm_collect_sort_kernel   candidate list + std::sort                      (:186-214, :265-266)
//   fpm_refine_prep_kernel    getRotatedROI matrix                            (:1074-1088)
//   fpm_corr_rows_kernel      IM_Conv_SIMD row dot products (dp4a)            (:461-483, :496-510)
//   fpm_refine_finalize_kernel float row chain + CCOEFF_Denominator + argmax + pose update (:304-367)
//   fpm_final_kernel          filterWithScore / RotatedRect / NMS / output    (:373-432)
//   fpm_ingest_*_kernel       cv::imread(IMREAD_GRAYSCALE) of a BMP / JPEG (dequantisation + ISLOW IDCT), camera RGB32 -> gray (MatchToolDialog.cpp:314, :1557)
//   fpm_jpeg_*_kernel         Huffman decoding of a JPEG scan (self-synchronising sub-sequences)   [fpm_jpeg_par.cuh]
// and, in fpm_mma.cuh / fpm_fused.cuh, the tcgen05 versions of the row dot products (fpm_corr_mma_kernel,
// fpm_corr_fused_kernel, fpm_corr_warp_kernel).
//
// All integer work is exact; all double/float epilogues are written op-by-op (the library is
// compiled with -fmad=false) so they round like the reference's x86-64 (no FMA) build.
#pragma once
#include "fpm_common.cuh"
#include "fpm_geometry.cuh"
#include "fpm_pyrdown.cuh"
#include "fpm_jpeg_par.cuh"

// =====================================================================================
// K1  pyrDown: fpm_pyrdown.cuh (one or two pyramid levels per launch)
// =====================================================================================
// =====================================================================================
// K2/K3  warpAffine, u8 C1, INTER_LINEAR, BORDER_CONSTANT -- OpenCV's fixed-point path:
//   AB_BITS=10, INTER_BITS=5, adelta/bdelta = cvRound(M*x*1024), X0 = cvRound((M01*y+M02)*1024)+16,
//   X = (X0+adelta)>>5, sx = X>>5, ax = X&31, weights (32-ax)(32-ay)*32 ..., (sum + 16384) >> 15
//   == ((top<<5) + ay*(bot-top) + 512) >> 10 with top = (p00<<5) + ax*(p01-p00)   (same integers).
// One job per output image (top-layer angle or refinement ROI).  One CTA = one 128x64 output tile of a
// GROUP of jobs: the 3 angles of a refinement candidate are anchored at the same source point and differ by
// less than ~4 px over the tile, so they share one staged source box.  The fixed-point map is separable and
// monotone in x and y, so the exact source bounding box of a tile follows from its 4 corners; the union box
// (<= 160x160 px) is staged in shared memory with cp.async (odd word pitch: conflict-free gathers) and the
// 4 bilinear taps of every pixel are gathered from shared memory -- a diagonal walk through global memory
// would cost one L1 wavefront per lane.  32 pixels per thread and angle; padding columns up to dpitch are
// written as zero.
// =====================================================================================
#define WA_TW 128
#define WA_TH 64
#define WA_PX (WA_TW / 32)   // pixels per lane and tile row
#define WA_THREADS 256
#define WA_BW 160     // staged box: max bytes per row actually used (40 words)
#define WA_SW 260     // staged box pitch capacity in bytes.  The pitch in use is 65 or 63 words = +-1 (mod 32 banks), see below
#define WA_SH 160     // staged box: rows
#define WA_MAXG 3     // jobs per group

// getRotatedROI matrix of eval j of a candidate (src/TemplateMatcher.cpp:1074-1088), inverted like warpAffine does
// n_tpl: templates of the group (candidate image v reads source frame v / n_tpl)
// Scale-tolerant matching: eval e = k * n_ang + j of a candidate of scale s has angle index j and scale
// fpm_eval_scale(s, k, n_sc, scale_step): {s / (1 + ds), s, s * (1 + ds)} when a scale range is matched (n_sc == 3), {s}
// otherwise.  At a scale s != 1 the source is resampled by 1/s around the level centre c: matrix getRotationMatrix2D(c, angle,
// 1/s), and the anchor becomes c + (1/s) * (rotated anchor - c).
struct FpmRefineGeom { const FpmCand* cands; int n_ang, n_sc; double angle_step, scale_step; int lvl_w, lvl_h, tpl_w, tpl_h, n_tpl; };

FPM_HD double fpm_eval_scale(double s, int k, int n_sc, double ds)
{
    return n_sc == 1 ? s : (k == 0 ? s / (1 + ds) : (k == 1 ? s : s * (1 + ds)));
}

__device__ __forceinline__ FpmWarpJob fpm_refine_job(const FpmCand& c, int e, int n_ang, int n_sc, double angle_step, double scale_step,
                                                     int lvl_w, int lvl_h, int tpl_w, int tpl_h, int n_tpl)
{
    const int k = e / n_ang, j = e - k * n_ang;
    const double scale = fpm_eval_scale(c.scale, k, n_sc, scale_step);
    double angle = (n_ang == 1) ? 0.0 : c.angle + angle_step * (double)(j - 1);
    float ptcx = (float)(lvl_w - 1) / 2.0f, ptcy = (float)(lvl_h - 1) / 2.0f;
    float ltx = c.ptx * 2, lty = c.pty * 2;
    float rx, ry;
    fpm_pt_rotate(ltx, lty, ptcx, ptcy, angle * FPM_D2R, &rx, &ry);
    if (scale != 1.0) fpm_scale_about(rx, ry, ptcx, ptcy, 1.0 / scale, &rx, &ry);
    FpmWarpJob jb;
    fpm_rotation_matrix(ptcx, ptcy, angle, jb.m, 1.0 / scale);
    jb.m[2] -= (double)(rx - 3);
    jb.m[5] -= (double)(ry - 3);
    fpm_invert_affine(jb.m);
    jb.src_img = n_tpl > 1 ? c.img / n_tpl : c.img;
    jb.dw = tpl_w + FPM_ROI_PAD; jb.dh = tpl_h + FPM_ROI_PAD;
    jb.valid = 1;
    return jb;
}

// hot loop of fpm_warp_kernel: the rows warp, warp + 8, ... of one job's tile; SWC = pitch of the staged box in bytes
template <int SWC>
__device__ __forceinline__ void fpm_warp_rows(uint32_t sbase, const int (&adj)[WA_PX], const int (&bdj)[WA_PX], const int* pX0,
                                              const int* pY0, uint8_t* __restrict__ drow, size_t dstep, int warp, int nrows)
{
#pragma unroll 2
    for (int row = warp; row < nrows; row += WA_THREADS / 32, drow += dstep, pX0 += WA_THREADS / 32, pY0 += WA_THREADS / 32) {
        const int X0 = *pX0, Y0 = *pY0;
        int v[WA_PX];
#pragma unroll
        for (int k = 0; k < WA_PX; k++) {
            const int XX = X0 + adj[k], YY = Y0 + bdj[k];
            const int fx = XX & 0x3e0, fy = YY & 0x3e0;
            const uint32_t a = sbase + (uint32_t)((YY >> 10) * SWC + (XX >> 10));
            int p00, p01, p10, p11;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(p00) : "r"(a));
            asm volatile("ld.shared.u8 %0, [%1+1];" : "=r"(p01) : "r"(a));
            asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(p10) : "r"(a), "n"(SWC));
            asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(p11) : "r"(a), "n"(SWC + 1));
            const int top = (p00 << 10) + fx * (p01 - p00);
            const int dif = (p10 << 10) - top + fx * (p11 - p10);
            v[k] = ((top << 10) + (512 << 10) + fy * dif) >> 20;
        }
#pragma unroll
        for (int k = 0; k < WA_PX; k++) drow[32 * k] = (uint8_t)v[k];
    }
}

__global__ void __launch_bounds__(WA_THREADS)
fpm_warp_kernel(const FpmWarpJob* __restrict__ jobs_g, int group, FpmLevel src, uint8_t* __restrict__ dst,
                int dpitch, size_t dst_job_stride, int border, int tiles_x, int vec_ok, const int* __restrict__ n_groups_dev,
                FpmRefineGeom geom)
{
    // n_groups_dev (optional): number of live job groups, known only on the device (descent without a host round trip per layer:
    // the grid covers an upper bound, the surplus CTAs leave at once)
    // refinement: blockIdx.y = candidate * n_sc + scale index k, the n_ang ROIs of one scale share a staged box
    if (n_groups_dev && (int)blockIdx.y >= *n_groups_dev * (geom.cands ? geom.n_sc : 1)) return;
    const int g0 = blockIdx.y * group;
    // jobs: given (top-layer sweep, tests), or the ROI matrices of candidate blockIdx.y computed here from its record
    // (geom.cands != null: one launch less per pyramid layer than a separate preparation kernel)
    __shared__ FpmWarpJob jobs_s[WA_MAXG];
    if (threadIdx.x < group)
        jobs_s[threadIdx.x] = geom.cands ? fpm_refine_job(geom.cands[blockIdx.y / geom.n_sc], (blockIdx.y % geom.n_sc) * geom.n_ang + threadIdx.x,
                                                          geom.n_ang, geom.n_sc, geom.angle_step, geom.scale_step, geom.lvl_w,
                                                          geom.lvl_h, geom.tpl_w, geom.tpl_h, geom.n_tpl)
                                         : jobs_g[g0 + threadIdx.x];
    __syncthreads();
    const FpmWarpJob* jobs = jobs_s - g0;              // jobs[g0 + j] below
    const FpmWarpJob& jb0 = jobs[g0];
    const int dw = jb0.dw, dh = jb0.dh;
    const int tile_y = blockIdx.x / tiles_x, tile_x = blockIdx.x - tile_y * tiles_x;
    const int tx0 = tile_x * WA_TW, ty0 = tile_y * WA_TH;
    if (!jb0.valid || ty0 >= dh || tx0 >= dpitch) return;
    __shared__ int s_ad[WA_MAXG][WA_TW], s_bd[WA_MAXG][WA_TW], s_X0[WA_MAXG][WA_TH], s_Y0[WA_MAXG][WA_TH];
    __shared__ __align__(16) uint8_t s_src[WA_SH * WA_SW];
    // Bank of a staged byte = (row * pitch_words + x / 4) mod 32.  The 32 lanes of a gather walk a straight line through the
    // box; with pitch_words = +1 (mod 32) the bank is row + x/4, strictly monotone along any line whose row and column move
    // in the SAME direction, with -1 (mod 32) along any line where they move in opposite directions: no two lanes share a
    // bank unless they share the word.  (41 words, the first choice, left 42 % of the wavefronts to bank conflicts and the
    // kernel bound by the shared-memory pipe.)  The direction of the lanes' line is (m[0], m[3]) of the inverse matrix.
    const int SW = (jb0.m[0] * jb0.m[3] >= 0) ? 260 : 252;
    const int tid = threadIdx.x;
    for (int i = tid; i < group * (WA_TW + WA_TH); i += WA_THREADS) {
        const int j = i / (WA_TW + WA_TH), k = i - j * (WA_TW + WA_TH);
        const FpmWarpJob& jb = jobs[g0 + j];
        if (k < WA_TW) {
            double x = (double)(tx0 + k);
            s_ad[j][k] = fpm_cvround(jb.m[0] * x * 1024.0);
            s_bd[j][k] = fpm_cvround(jb.m[3] * x * 1024.0);
        } else {
            const int r = k - WA_TW;
            double y = (double)(ty0 + r);
            s_X0[j][r] = fpm_cvround((jb.m[1] * y + jb.m[2]) * 1024.0) + 16;
            s_Y0[j][r] = fpm_cvround((jb.m[4] * y + jb.m[5]) * 1024.0) + 16;
        }
    }
    __syncthreads();
    const int ncols = min(WA_TW, dw - tx0);            // real pixels in this tile (<= 0 for pad-only tiles)
    const int nrows = min(WA_TH, dh - ty0);
    const uint8_t* __restrict__ s = src.ptr + (size_t)jb0.src_img * src.img_stride;
    const int sw = src.w, sh = src.h, sp = src.pitch;

    // exact source box of the tile for every job of the group from the tile corners (X and Y are sums of
    // monotone functions of x and y), then the union
    int bx0 = 0, by0 = 0;
    bool staged = false, inside = false;
    if (ncols > 0) {
        int Xmin = 0x7fffffff, Xmax = -0x7fffffff, Ymin = 0x7fffffff, Ymax = -0x7fffffff;
        for (int j = 0; j < group; j++) {
            const int xa = s_ad[j][0], xb = s_ad[j][ncols - 1], ya = s_bd[j][0], yb = s_bd[j][ncols - 1];
            const int X0a = s_X0[j][0], X0b = s_X0[j][nrows - 1], Y0a = s_Y0[j][0], Y0b = s_Y0[j][nrows - 1];
            Xmin = min(Xmin, min(min(X0a + xa, X0a + xb), min(X0b + xa, X0b + xb)));
            Xmax = max(Xmax, max(max(X0a + xa, X0a + xb), max(X0b + xa, X0b + xb)));
            Ymin = min(Ymin, min(min(Y0a + ya, Y0a + yb), min(Y0b + ya, Y0b + yb)));
            Ymax = max(Ymax, max(max(Y0a + ya, Y0a + yb), max(Y0b + ya, Y0b + yb)));
        }
        const int sx0 = Xmin >> 10, sx1 = (Xmax >> 10) + 1, sy0 = Ymin >> 10, sy1 = (Ymax >> 10) + 1;
        inside = sx0 >= 0 && sy0 >= 0 && sx1 < sw && sy1 < sh;
        bx0 = max(sx0, 0) & ~3;
        by0 = max(sy0, 0);
        const int bx1 = min(sx1, sw - 1), by1 = min(sy1, sh - 1);
        staged = (bx1 - bx0 + 1 <= WA_BW) && (by1 - by0 + 1 <= WA_SH);
        if (staged && bx1 >= bx0 && by1 >= by0) {
            const int nwr = (bx1 - bx0) / 4 + 1, nr = by1 - by0 + 1;      // nwr <= 40
            const int wc = tid & 63;
            if (wc < nwr) {
                const int x = bx0 + 4 * wc;
                const uint8_t* rowp = s + (size_t)(by0 + (tid >> 6)) * sp + x;
                uint8_t* sp_out = s_src + (tid >> 6) * SW + 4 * wc;
                if (vec_ok && x + 3 < sw) {
                    for (int r = tid >> 6; r < nr; r += WA_THREADS / 64, rowp += (size_t)(WA_THREADS / 64) * sp,
                             sp_out += (WA_THREADS / 64) * SW)
                        fpm_cp_async4(sp_out, rowp, true);
                } else {
                    for (int r = tid >> 6; r < nr; r += WA_THREADS / 64, rowp += (size_t)(WA_THREADS / 64) * sp,
                             sp_out += (WA_THREADS / 64) * SW) {
                        uint32_t v = 0;
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            if (x + k < sw) v |= (uint32_t)__ldg(rowp + k) << (8 * k);
                        *reinterpret_cast<uint32_t*>(sp_out) = v;
                    }
                }
            }
        }
    }
    fpm_cp_async_commit();
    fpm_cp_async_wait<0>();
    __syncthreads();
    // Gather.  A warp owns one output row at a time and lane l the pixels l, l+32, l+64, l+96 of the tile row: neighbouring
    // lanes read neighbouring source pixels (same word -> broadcast) or, for steep angles, neighbouring source rows
    // (odd word pitch -> different banks), so the byte gathers are close to conflict-free at every angle.
    const int lane = tid & 31, warp = tid >> 5;
    const bool fastw = staged && inside && ncols == WA_TW;     // whole tile row inside the image and the ROI: no predicates
    if (fastw) {
        // Hot path, kept free of everything that is not per-pixel work (it was 46 instructions per pixel with the path
        // dispatch, the generic->shared address conversion and the 64-bit row pointer inside the row loop):
        //   XX = X0 + adelta, YY = Y0 + bdelta;  fx = XX & 0x3e0 = 32*ax, fy = YY & 0x3e0 = 32*ay (one LOP each instead of
        //   shift + mask);  top' = (p00 << 10) + fx*(p01 - p00) = 32*top, bot' likewise;
        //   v = ((top' << 10) + fy*(bot' - top') + (512 << 10)) >> 20   -- the same integer as ((top<<5) + ay*(bot-top) + 512) >> 10
        //   (all terms < 2^29).
        const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_src);
        for (int j = 0; j < group; j++) {
            if (!jobs[g0 + j].valid) continue;
            int adj[WA_PX], bdj[WA_PX];
#pragma unroll
            for (int k = 0; k < WA_PX; k++) {
                adj[k] = s_ad[j][lane + 32 * k] - (bx0 << 10);
                bdj[k] = s_bd[j][lane + 32 * k] - (by0 << 10);
            }
            uint8_t* __restrict__ drow = dst + (size_t)(g0 + j) * dst_job_stride + tx0 + (size_t)(ty0 + warp) * dpitch + lane;
            const size_t dstep = (size_t)(WA_THREADS / 32) * dpitch;
            const int* pX0 = &s_X0[j][warp];
            const int* pY0 = &s_Y0[j][warp];
            // the pitch as a compile-time constant: the second row's taps become immediate offsets of the first row's address
            if (SW == 260) fpm_warp_rows<260>(sbase, adj, bdj, pX0, pY0, drow, dstep, warp, nrows);
            else fpm_warp_rows<252>(sbase, adj, bdj, pX0, pY0, drow, dstep, warp, nrows);
        }
        return;
    }
    for (int j = 0; j < group; j++) {
        if (!jobs[g0 + j].valid) continue;
        uint8_t* __restrict__ d = dst + (size_t)(g0 + j) * dst_job_stride + tx0;
        int adj[WA_PX], bdj[WA_PX];
#pragma unroll
        for (int k = 0; k < WA_PX; k++) {
            adj[k] = s_ad[j][lane + 32 * k] - (bx0 << 10);
            bdj[k] = s_bd[j][lane + 32 * k] - (by0 << 10);
        }
        for (int row = warp; row < nrows; row += WA_THREADS / 32) {
            const int X0 = s_X0[j][row], Y0 = s_Y0[j][row];
            uint8_t* drow = d + (size_t)(ty0 + row) * dpitch;
            if (staged && inside) {
                // partial-width tile (the last tile column of a ROI, or a ROI narrower than a tile) whose taps all lie
                // inside the image: the fast arithmetic with a column predicate; padding columns are written as zero
#pragma unroll
                for (int k = 0; k < WA_PX; k++) {
                    const int col = lane + 32 * k;
                    if (tx0 + col >= dpitch) continue;
                    int v = 0;
                    if (col < ncols) {
                        const int XX = X0 + adj[k], YY = Y0 + bdj[k];
                        const int ax = (XX >> 5) & 31, ay = (YY >> 5) & 31;
                        const uint8_t* p = s_src + (YY >> 10) * SW + (XX >> 10);
                        const int p00 = p[0], p01 = p[1], p10 = p[SW], p11 = p[SW + 1];
                        const int top = (p00 << 5) + ax * (p01 - p00);
                        const int bot = (p10 << 5) + ax * (p11 - p10);
                        v = ((top << 5) + ay * (bot - top) + 512) >> 10;
                    }
                    drow[col] = (uint8_t)v;
                }
            } else {
#pragma unroll
                for (int k = 0; k < WA_PX; k++) {
                    const int col = lane + 32 * k;
                    if (tx0 + col >= dpitch) continue;
                    int v = 0;
                    if (col < ncols) {
                        const int XX = X0 + adj[k], YY = Y0 + bdj[k];
                        const int ax = (XX >> 5) & 31, ay = (YY >> 5) & 31;
                        const int lx = XX >> 10, ly = YY >> 10;              // relative to (bx0, by0)
                        const int sx = lx + bx0, sy = ly + by0;
                        const bool x0in = (unsigned)sx < (unsigned)sw, x1in = (unsigned)(sx + 1) < (unsigned)sw;
                        const bool y0in = (unsigned)sy < (unsigned)sh, y1in = (unsigned)(sy + 1) < (unsigned)sh;
                        int p00, p01, p10, p11;
                        if (staged) {
                            const uint8_t* p = s_src + ly * SW + lx;
                            p00 = (x0in && y0in) ? p[0] : border;
                            p01 = (x1in && y0in) ? p[1] : border;
                            p10 = (x0in && y1in) ? p[SW] : border;
                            p11 = (x1in && y1in) ? p[SW + 1] : border;
                        } else {
                            const uint8_t* p = s + (ptrdiff_t)sy * sp + sx;
                            p00 = (x0in && y0in) ? __ldg(p) : border;
                            p01 = (x1in && y0in) ? __ldg(p + 1) : border;
                            p10 = (x0in && y1in) ? __ldg(p + sp) : border;
                            p11 = (x1in && y1in) ? __ldg(p + sp + 1) : border;
                        }
                        const int top = (p00 << 5) + ax * (p01 - p00);
                        const int bot = (p10 << 5) + ax * (p11 - p10);
                        v = ((top << 5) + ay * (bot - top) + 512) >> 10;
                    }
                    drow[col] = (uint8_t)v;                                  // padding columns are written as zero
                }
            }
        }
    }
}

// =====================================================================================
// shared CCOEFF_NORMED epilogue (CCOEFF_Denominator, src/TemplateMatcher.cpp:567-595)
// =====================================================================================
__device__ __forceinline__ float fpm_ccoeff_epilogue(float numerator, double wsum, double wsqsum,
                                                     double tmean, double tnorm, double inv_area)
{
    double num = (double)numerator, t;
    double wndMean2 = 0, wndSum2 = 0;
    t = wsum;
    wndMean2 += t * t;
    num -= t * tmean;
    wndMean2 *= inv_area;
    t = wsqsum;
    wndSum2 += t;
    double diff2 = fmax(wndSum2 - wndMean2, 0.0);
    if (diff2 <= fmin(0.5, (double)(10 * FLT_EPSILON) * wndSum2))
        t = 0;
    else
        t = sqrt(diff2) * tnorm;
    if (fabs(num) < t)
        num /= t;
    else if (fabs(num) < t * 1.125)
        num = num > 0 ? 1 : -1;
    else
        num = 0;
    return (float)num;
}

// Top-layer variant with an early out.  The score map is only ever consumed by the greedy peak search, which
// observes nothing below its threshold (a pick is taken only if value >= thresh and the search stops at the first
// maximum below it), so a score that is certainly below the threshold may be stored as a float32 estimate instead
// of the exact double-precision quotient: that skips the fp64 sqrt and division (about half of the kernel's
// instructions for a 14x14 template).  The integer sums and the variance term stay exact; the estimate's error
// (~1e-6) is far inside the 0.01 margin of reject_below.  reject_below = -inf gives the exact map everywhere.
__device__ __forceinline__ float fpm_ccoeff_epilogue_top(float numerator, double wsum, double wsqsum, double tmean, double tnorm,
                                                         double inv_area, float reject_below, float inv_tnorm_f)
{
    const double num = (double)numerator - wsum * tmean;
    const double diff2 = wsqsum - (wsum * wsum) * inv_area;
    if (diff2 > 1.0) {                                       // away from the degenerate-variance guard of :575-577
        const float est = (float)num * rsqrtf((float)diff2) * inv_tnorm_f;
        if (est < reject_below) return est;
    }
    return fpm_ccoeff_epilogue(numerator, wsum, wsqsum, tmean, tnorm, inv_area);
}

// =====================================================================================
// K4+K7  top-layer dense score map: exact integer TM_CCORR numerator, exact window sum / sqsum,
// CCOEFF_NORMED epilogue.  One CTA = 64x16 scores, 4 horizontally adjacent scores per thread; image
// patch + template in shared memory as 32-bit words (rows zero padded).  Per template word a thread
// loads one patch word and one template word and feeds the 4 byte-shifted windows (funnel shifts by
// 0/8/16/24 bits) to dp4a: numerator, window sum and window sum of squares, all exact.
// =====================================================================================
#define TS_TW 64
#define TS_TH 16
#define TS_THREADS 256

// Template groups (tpl.n_tpl > 1): the CTA stages its canvas patch and its row-window sums once and scores the patch
// against every template of the group in turn; map k of job z is written to score + (z * n_tpl + k) * score_job_stride.
// GROUP = false (a single template) compiles to the one-template kernel.
// MASKED (a masked template or group, tpl.mrun set): the window sums run over the kept pixels only.  Instead of one row-window
// sum per patch row the CTA keeps row prefix sums of the patch and of its squares, ph x (TS_TW + tw) each, and every score adds
// P[x + e] - P[x + b] over the runs [b, e) of each row of the scored template's own mask: exact integers, the same ones a full
// mask gives through the row-window sums.  The prefix sums do not depend on the template: a group builds them once.
template <bool GROUP, bool MASKED = false>
__global__ void __launch_bounds__(TS_THREADS)
fpm_top_score_kernel(const FpmWarpJob* __restrict__ jobs, const uint8_t* __restrict__ rot, int rpitch,
                     size_t rot_job_stride, FpmTplLevel tpl, float* __restrict__ score, int spitch,
                     size_t score_job_stride, float reject_below)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const FpmWarpJob& jb = jobs[blockIdx.z];
    const int tw = tpl.w, th = tpl.h;
    const int RW = jb.dw - tw + 1, RH = jb.dh - th + 1;
    const int x0 = blockIdx.x * TS_TW, y0 = blockIdx.y * TS_TH;
    if (!jb.valid || RW <= 0 || RH <= 0 || x0 >= RW || y0 >= RH) return;
    const int nwt = (tw + 3) / 4;                          // template words per row
    const int ph = TS_TH + th - 1;
    const int pww = TS_TW / 4 + nwt + 1;                   // patch words per row
    uint32_t* s_t = reinterpret_cast<uint32_t*>(smem);     // th * nwt
    uint32_t* s_p = s_t + th * nwt;                        // ph * pww
    const int tid = threadIdx.x;
    const uint8_t* __restrict__ r = rot + (size_t)blockIdx.z * rot_job_stride;
    const bool word_ok = ((rpitch & 3) == 0) && ((reinterpret_cast<uintptr_t>(r) & 3) == 0);    // x0 is a multiple of 64
    auto stage_template = [&](const FpmTplLevel& t) {
        for (int i = tid; i < th * nwt; i += TS_THREADS) {
            int yy = i / nwt, xw = i - yy * nwt;
            uint32_t v = 0;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (4 * xw + k < tw) v |= (uint32_t)t.ptr[yy * t.pitch + 4 * xw + k] << (8 * k);
            s_t[i] = v;
        }
    };
    stage_template(tpl);
    for (int i = tid; i < ph * pww; i += TS_THREADS) {
        int yy = i / pww, xw = i - yy * pww;
        int gy = y0 + yy;
        uint32_t v = 0;
        if (gy < jb.dh) {
            const int gx0 = x0 + 4 * xw;
            if (word_ok && gx0 + 3 < jb.dw) {
                v = __ldg(reinterpret_cast<const uint32_t*>(r + (size_t)gy * rpitch + gx0));
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (gx0 + k < jb.dw) v |= (uint32_t)r[(size_t)gy * rpitch + gx0 + k] << (8 * k);
            }
        }
        s_p[i] = v;
    }
    __syncthreads();
    const int tail = tw & 3;
    const uint32_t tailbm = tail ? (0xffffffffu >> (8 * (4 - tail))) : 0xffffffffu;
    // Row-window sums of the patch, once per CTA: s_rs/s_rq[yy][x] = sum_{j<tw} P[yy][x+j] (^2).  Every score row
    // that covers patch row yy reuses them, so the main loop only multiplies by the template (the zero padding of
    // the template's last word masks the patch bytes beyond tw there).  The same for every template of a group; not
    // needed when all of them are flat.
    const int rs_w = MASKED ? TS_TW + tw : TS_TW;              // prefix entries P[0 .. TS_TW + tw - 1] per patch row when MASKED
    uint32_t* s_rs = s_t + ((th * nwt + ph * pww + 3) & ~3);   // ph * rs_w, 16-byte aligned
    uint32_t* s_rq = s_rs + ph * rs_w;
    bool need_sums = !tpl.result_equal1;
    if (GROUP)
        for (int k = 1; k < tpl.n_tpl; k++) need_sums |= !tpl.stats[k].result_equal1;
    if (MASKED && need_sums) {
        // one warp per patch row: each lane takes a word (4 pixels), an inclusive warp scan of the word sums gives the
        // prefix in front of every word; P[x] = sum of the pixels left of column x
        const int warp = tid >> 5, lane = tid & 31;
        for (int yy = warp; yy < ph; yy += TS_THREADS / 32) {
            uint32_t cs = 0, cq = 0;
            for (int w0 = 0; 4 * w0 < rs_w; w0 += 32) {
                const int xw = w0 + lane;
                const uint32_t v = xw < pww ? s_p[yy * pww + xw] : 0u;
                const uint32_t b0 = v & 255u, b1 = (v >> 8) & 255u, b2 = (v >> 16) & 255u, b3 = v >> 24;
                const uint32_t ws = b0 + b1 + b2 + b3, wq = b0 * b0 + b1 * b1 + b2 * b2 + b3 * b3;
                uint32_t is = ws, iq = wq;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t us = __shfl_up_sync(0xffffffffu, is, o), uq = __shfl_up_sync(0xffffffffu, iq, o);
                    if (lane >= o) { is += us; iq += uq; }
                }
                uint32_t ps = cs + is - ws, pq = cq + iq - wq;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    if (4 * xw + k < rs_w) { s_rs[yy * rs_w + 4 * xw + k] = ps; s_rq[yy * rs_w + 4 * xw + k] = pq; }
                    const uint32_t bk = (v >> (8 * k)) & 255u;
                    ps += bk; pq += bk * bk;
                }
                cs += __shfl_sync(0xffffffffu, is, 31);
                cq += __shfl_sync(0xffffffffu, iq, 31);
            }
        }
        __syncthreads();
    } else if (need_sums) {
        for (int i = tid; i < ph * (TS_TW / 4); i += TS_THREADS) {
            const int yy = i / (TS_TW / 4), xq = i - yy * (TS_TW / 4);
            const uint32_t* prow = s_p + yy * pww + xq;
            uint32_t b[4] = {0, 0, 0, 0}, c[4] = {0, 0, 0, 0};
            uint32_t lo = prow[0];
            for (int xw = 0; xw < nwt; xw++) {
                const uint32_t hi = prow[xw + 1];
                const uint32_t m = (xw == nwt - 1) ? tailbm : 0xffffffffu;
                uint32_t p[4];
                p[0] = lo & m;
                p[1] = __funnelshift_r(lo, hi, 8) & m;
                p[2] = __funnelshift_r(lo, hi, 16) & m;
                p[3] = __funnelshift_r(lo, hi, 24) & m;
#pragma unroll
                for (int k = 0; k < 4; k++) { b[k] = __dp4a(p[k], 0x01010101u, b[k]); c[k] = __dp4a(p[k], p[k], c[k]); }
                lo = hi;
            }
            *reinterpret_cast<uint4*>(s_rs + yy * TS_TW + 4 * xq) = make_uint4(b[0], b[1], b[2], b[3]);
            *reinterpret_cast<uint4*>(s_rq + yy * TS_TW + 4 * xq) = make_uint4(c[0], c[1], c[2], c[3]);
        }
        __syncthreads();
    }
    const int tx = tid & 15, ty = tid >> 4;
    const int ox = x0 + 4 * tx, oy = y0 + ty;
    const bool live = ox < RW && oy < RH;
    // window sum / square sum of the 4 scores' windows in row yy of template t
    auto window_rows = [&](const FpmTplLevel& t, int yy, uint4& rs, uint4& rq) {
        const uint32_t* ps = s_rs + (ty + yy) * rs_w + 4 * tx;
        const uint32_t* pq = s_rq + (ty + yy) * rs_w + 4 * tx;
        if (!MASKED) {
            rs = *reinterpret_cast<const uint4*>(ps);
            rq = *reinterpret_cast<const uint4*>(pq);
            return;
        }
        rs = make_uint4(0, 0, 0, 0); rq = make_uint4(0, 0, 0, 0);
        for (int k = __ldg(t.mrow + yy), ke = __ldg(t.mrow + yy + 1); k < ke; k++) {
            const int2 be = __ldg(t.mrun + k);
            rs.x += ps[be.y] - ps[be.x]; rs.y += ps[be.y + 1] - ps[be.x + 1];
            rs.z += ps[be.y + 2] - ps[be.x + 2]; rs.w += ps[be.y + 3] - ps[be.x + 3];
            rq.x += pq[be.y] - pq[be.x]; rq.y += pq[be.y + 1] - pq[be.x + 1];
            rq.z += pq[be.y + 2] - pq[be.x + 2]; rq.w += pq[be.y + 3] - pq[be.x + 3];
        }
    };
    if (!GROUP && !live) return;
    const int n_tpl = GROUP ? tpl.n_tpl : 1;
    for (int kt = 0; kt < n_tpl; kt++) {
        const FpmTplLevel tk = GROUP ? fpm_tpl_member(tpl, kt) : tpl;
        if (GROUP && kt > 0) {                                      // every thread is past the previous template's words
            __syncthreads();
            stage_template(tk);
            __syncthreads();
        }
        if (!live) continue;
        float* out = score + ((size_t)blockIdx.z * n_tpl + kt) * score_job_stride + (size_t)oy * spitch + ox;
        if (tk.result_equal1) {
            for (int k = 0; k < 4 && ox + k < RW; k++) out[k] = 1.0f;
            continue;
        }
        unsigned long long num[4], wsum[4], wsq[4];
        if ((long long)tw * th <= 66000) {
            // every sum is at most 255^2 * w * h < 2^32: plain 32-bit accumulators across all template rows (the 64-bit
            // adds of the general path cost as many instructions as the dp4a loop itself for a 14x14 template)
            uint32_t a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0}, c[4] = {0, 0, 0, 0};
            for (int yy = 0; yy < th; yy++) {
                const uint32_t* prow = s_p + (ty + yy) * pww + tx;
                const uint32_t* trow = s_t + yy * nwt;
                uint32_t lo = prow[0];
                for (int xw = 0; xw < nwt; xw++) {
                    const uint32_t hi = prow[xw + 1];
                    const uint32_t t = trow[xw];           // bytes beyond tw are 0 in the staged template
                    a[0] = __dp4a(lo, t, a[0]);
                    a[1] = __dp4a(__funnelshift_r(lo, hi, 8), t, a[1]);
                    a[2] = __dp4a(__funnelshift_r(lo, hi, 16), t, a[2]);
                    a[3] = __dp4a(__funnelshift_r(lo, hi, 24), t, a[3]);
                    lo = hi;
                }
                uint4 rs, rq;
                window_rows(tk, yy, rs, rq);
                b[0] += rs.x; b[1] += rs.y; b[2] += rs.z; b[3] += rs.w;
                c[0] += rq.x; c[1] += rq.y; c[2] += rq.z; c[3] += rq.w;
            }
#pragma unroll
            for (int k = 0; k < 4; k++) { num[k] = a[k]; wsum[k] = b[k]; wsq[k] = c[k]; }
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) { num[k] = 0; wsum[k] = 0; wsq[k] = 0; }
            for (int yy = 0; yy < th; yy++) {
                const uint32_t* prow = s_p + (ty + yy) * pww + tx;
                const uint32_t* trow = s_t + yy * nwt;
                uint32_t a[4] = {0, 0, 0, 0};
                uint32_t lo = prow[0];
                for (int xw = 0; xw < nwt; xw++) {
                    const uint32_t hi = prow[xw + 1];
                    const uint32_t t = trow[xw];
                    a[0] = __dp4a(lo, t, a[0]);
                    a[1] = __dp4a(__funnelshift_r(lo, hi, 8), t, a[1]);
                    a[2] = __dp4a(__funnelshift_r(lo, hi, 16), t, a[2]);
                    a[3] = __dp4a(__funnelshift_r(lo, hi, 24), t, a[3]);
                    lo = hi;
                }
                uint4 rs, rq;
                window_rows(tk, yy, rs, rq);
                num[0] += a[0]; num[1] += a[1]; num[2] += a[2]; num[3] += a[3];   // per-row s32, s64 across rows
                wsum[0] += rs.x; wsum[1] += rs.y; wsum[2] += rs.z; wsum[3] += rs.w;
                wsq[0] += rq.x; wsq[1] += rq.y; wsq[2] += rq.z; wsq[3] += rq.w;
            }
        }
        // TM_CCORR result cell is a float32 (cv::matchTemplate output depth), here the rounded exact sum
        const float inv_tnorm_f = 1.0f / (float)tk.norm;
        for (int k = 0; k < 4 && ox + k < RW; k++)
            out[k] = fpm_ccoeff_epilogue_top((float)num[k], (double)wsum[k], (double)wsq[k], tk.mean, tk.norm, tk.inv_area,
                                             reject_below, inv_tnorm_f);
    }
}

// =====================================================================================
// K8  greedy peak extraction per (image, angle): minMaxLoc / s_BlockMax + getNextMaxLoc.
// One CTA per score map.  A table of (max, location) per block is kept in global scratch;
// every pick is an argmax over the table, a paint of the suppression rectangle with -1 and a
// rescan of the blocks the rectangle touches.
//   mode 0 (plain minMaxLoc path): own square tiles; ties -> first in row-major scan order
//   mode 1 (Qt s_BlockMax path, DataStructures.h:150-245): template-sized blocks + right strip +
//          bottom strip + corner; ties -> first block in construction order
// =====================================================================================
struct FpmPick { int x, y; float v; };

struct FpmBlockGeom { int mode, bw, bh, ncol, nrow, nblocks, has_right, has_bottom, has_corner, bottom_w; };

// mode 0: plain tiles of `tile` x `tile` (whole-map minMaxLoc semantics); mode 1: Qt s_BlockMax
// (DataStructures.h:150-211: template-sized blocks, right strip, bottom strip, corner); mode 2: MFC s_BlockMax
// (MatchTool/MatchToolDlg.h:109-175: 2x template blocks, right strip when the width has a residue, bottom strip
// over the regular columns when both have one, over the full width when only the height has one; no corner; an
// empty table -- fewer than one block in a dimension -- falls back to the whole-map search, :196-200)
__device__ __forceinline__ FpmBlockGeom fpm_block_geom(int mode, int cols, int rows, int tw, int th, int tile)
{
    FpmBlockGeom g;
    if (mode == 2 && (cols / (2 * tw) == 0 || rows / (2 * th) == 0)) mode = 0;
    g.mode = mode;
    if (mode == 0) {
        g.bw = g.bh = tile;
        g.ncol = (cols + tile - 1) / tile; g.nrow = (rows + tile - 1) / tile;
        g.has_right = g.has_bottom = g.has_corner = 0;
        g.bottom_w = 0;
        g.nblocks = g.ncol * g.nrow;
    } else if (mode == 1) {
        g.bw = tw; g.bh = th;
        g.ncol = cols / g.bw; g.nrow = rows / g.bh;
        g.has_right = g.ncol * g.bw < cols;
        g.has_bottom = (g.nrow * g.bh < rows) && (g.ncol * g.bw > 0);
        g.has_corner = (g.ncol * g.bw < cols) && (g.nrow * g.bh < rows);
        g.bottom_w = g.ncol * g.bw;
        g.nblocks = g.ncol * g.nrow + g.has_right + g.has_bottom + g.has_corner;
    } else {
        g.bw = 2 * tw; g.bh = 2 * th;
        g.ncol = cols / g.bw; g.nrow = rows / g.bh;
        const int hres = g.ncol * g.bw < cols, vres = g.nrow * g.bh < rows;
        g.has_right = hres;
        g.has_bottom = vres;                     // (the upstream else-branch would scan an empty Mat when !vres: absent here)
        g.has_corner = 0;
        g.bottom_w = (hres && vres) ? g.ncol * g.bw : cols;
        g.nblocks = g.ncol * g.nrow + g.has_right + g.has_bottom;
    }
    return g;
}

__device__ __forceinline__ void fpm_block_rect(const FpmBlockGeom& g, int k, int cols, int rows,
                                               int& x, int& y, int& w, int& h)
{
    int regular = g.ncol * g.nrow;
    if (k < regular) {
        int by = k / g.ncol, bx = k - by * g.ncol;
        x = bx * g.bw; y = by * g.bh;
        w = min(g.bw, cols - x); h = min(g.bh, rows - y);
        return;
    }
    k -= regular;
    if (g.has_right) { if (k == 0) { x = g.ncol * g.bw; y = 0; w = cols - x; h = rows; return; } k--; }
    if (g.has_bottom) { if (k == 0) { x = 0; y = g.nrow * g.bh; w = g.bottom_w; h = rows - y; return; } k--; }
    x = g.ncol * g.bw; y = g.nrow * g.bh; w = cols - x; h = rows - y;
}

// n / d for 0 <= n, n * d < 2^32, through one multiply-high (the pick loop is a latency chain: no IDIV on it)
struct FpmFastDiv { uint32_t m; int d; };
__device__ __forceinline__ FpmFastDiv fpm_fastdiv_make(int d)
{
    FpmFastDiv f; f.d = d;
    f.m = d > 1 ? (uint32_t)((0x100000000ull + (unsigned)d - 1) / (unsigned)d) : 0u;
    return f;
}
__device__ __forceinline__ int fpm_fastdiv(int n, const FpmFastDiv& f) { return f.d > 1 ? (int)__umulhi((uint32_t)n, f.m) : n; }

// per-lane walk over a w-wide block in steps of 32 elements: start (yy0, xx0) and step (q, r) with one carry;
// dv.m != 0: multiply-high division by w is available (the regular block width), else a plain division is used
struct FpmScanStep { int w, q, r, yy0, xx0; FpmFastDiv dv; };
__device__ __forceinline__ FpmScanStep fpm_scan_step(int w, int lane, bool with_fastdiv)
{
    FpmScanStep s; s.w = w; s.q = 32 / w; s.r = 32 - s.q * w; s.yy0 = lane / w; s.xx0 = lane - s.yy0 * w;
    if (with_fastdiv) s.dv = fpm_fastdiv_make(w); else { s.dv.m = 0; s.dv.d = w; }
    return s;
}

// warp-cooperative scan of one block: max value, first location in row-major order.  The picks are a latency
// chain (one CTA per map, hundreds of sequential picks), so the loads of a batch of NB x 32 elements are all
// issued before the first comparison and nothing divides per element.
// Elements inside the rectangle [px0, px1) x [py0, py1) count as -1: that is the suppression rectangle of the pick in
// flight, whose stores may not have landed yet (no barrier between painting and rescanning); pass an empty
// rectangle to read the map as it is.
template <int NB>
__device__ __forceinline__ void fpm_scan_block(const float* __restrict__ map, int pitch, int x, int y,
                                               int w, int h, int lane, const FpmScanStep& st,
                                               int px0, int py0, int px1, int py1, float& bv, int& bx, int& by)
{
    float best = -INFINITY; int bidx = 0x7fffffff;
    const int n = w * h;
    int yy = st.yy0, xx = st.xx0;
    for (int i0 = lane; i0 < n; i0 += 32 * NB) {
        float v[NB];
#pragma unroll
        for (int k = 0; k < NB; k++) {
            const int gx = x + xx, gy = y + yy;
            const bool painted = gx >= px0 && gx < px1 && gy >= py0 && gy < py1;
            v[k] = (i0 + 32 * k < n) ? (painted ? -1.0f : map[(size_t)gy * pitch + gx]) : -INFINITY;
            xx += st.r; yy += st.q;
            if (xx >= w) { xx -= w; yy++; }
        }
#pragma unroll
        for (int k = 0; k < NB; k++)
            if (v[k] > best) { best = v[k]; bidx = i0 + 32 * k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
    }
    bv = best;
    if (bidx == 0x7fffffff) bidx = 0;
    const int byy = st.dv.m ? fpm_fastdiv(bidx, st.dv) : bidx / w;
    by = y + byy; bx = x + (bidx - byy * w);
}

#define PK_THREADS 512
#define PK_SUP_MAX 2048                 // super-table entries (32 blocks each) -> at most 65536 blocks per map

// (value, block index, location) ordering of the greedy pick: larger value first; ties go to the
// first block in table order (s_BlockMax::GetMaxValueLoc, mode 1) or to the first location in scan
// order (cv::minMaxLoc, mode 0).  Locations are packed (y << 16 | x): same order as y * cols + x.
__device__ __forceinline__ bool fpm_pick_better(int mode, float v, int k, int l, float bv, int bk, int bl)
{
    // MFC GetMaxValueLoc (MatchToolDlg.h:202-212) keeps the LAST maximal block (>=)
    return (v > bv) || (v == bv && (mode == 0 ? (l < bl) : (mode == 1 ? (k < bk) : (k > bk && k != 0x7fffffff))));
}

__device__ __forceinline__ void fpm_pick_warp_reduce(int mode, float& v, int& k, int& l)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, v, o);
        int ok = __shfl_xor_sync(0xffffffffu, k, o);
        int ol = __shfl_xor_sync(0xffffffffu, l, o);
        if (fpm_pick_better(mode, ov, ok, ol, v, k, l)) { v = ov; k = ok; l = ol; }
    }
}

// Greedy peak picking of one score map by one CTA.  Two-level maximum table: per block (shared memory, or
// global scratch for very large maps) and per 32 consecutive blocks (shared).  A pick repaints a rectangle,
// rescans only the blocks that rectangle touches (found by index arithmetic, not by testing every block),
// refreshes their super-entries and takes the argmax over the super-table with one warp.
__global__ void __launch_bounds__(PK_THREADS)
fpm_top_peaks_kernel(const FpmWarpJob* __restrict__ jobs, float* __restrict__ score, int spitch,
                     size_t score_job_stride, int tw, int th, int mode, int tile,
                     float* __restrict__ blk_val, int* __restrict__ blk_loc, int blk_stride,
                     double thresh, double max_overlap, int max_picks,
                     FpmPick* __restrict__ picks, int* __restrict__ pick_count, int smem_blocks, int j0, int n_tpl, int n_ang)
{
    // map blockIdx.x = (canvas j0 + blockIdx.x / n_tpl) x (template blockIdx.x % n_tpl), the score kernel's order; its picks go
    // to (virtual image, angle) slot job: canvas j = frame * n_ang + angle, virtual image = frame * n_tpl + template.  The
    // angle-sharded sweep of one frame passes its chunk of the schedule as n_ang (jobs relative to the chunk's first angle), so
    // the picks land in its rank block as [template][chunk angle]
    const int mi = blockIdx.x;
    const int wj = j0 + mi / n_tpl;
    const int job = n_tpl == 1 ? wj : ((wj / n_ang) * n_tpl + mi % n_tpl) * n_ang + wj % n_ang;
    const FpmWarpJob& jb = jobs[wj];
    const int cols = jb.dw - tw + 1, rows = jb.dh - th + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x, nwarps = nthreads >> 5;
    if (!jb.valid || cols <= 0 || rows <= 0) { if (tid == 0) pick_count[job] = 0; return; }
    float* __restrict__ map = score + (size_t)mi * score_job_stride;
    const FpmBlockGeom g = fpm_block_geom(mode, cols, rows, tw, th, tile);
    mode = g.mode;                                                // MFC tables that come out empty use the plain search
    // block table: in shared memory when the launch reserved room for it (smem_blocks), else in global scratch
    extern __shared__ float pk_dyn[];
    const bool tbl_smem = g.nblocks <= smem_blocks;
    float* bval = tbl_smem ? pk_dyn : blk_val + (size_t)mi * blk_stride;
    int* bloc = tbl_smem ? reinterpret_cast<int*>(pk_dyn + smem_blocks) : blk_loc + (size_t)mi * blk_stride;
    const int regular = g.ncol * g.nrow;
    const int nsup = (g.nblocks + 31) >> 5;
    const FpmFastDiv div_bw = fpm_fastdiv_make(g.bw), div_bh = fpm_fastdiv_make(g.bh);
    const FpmScanStep step_reg = fpm_scan_step(g.bw, lane, true);  // full-width blocks share one walk
    __shared__ float s_sv[PK_SUP_MAX];
    __shared__ int s_sk[PK_SUP_MAX], s_sl[PK_SUP_MAX];
    __shared__ float s_best_v[2];
    __shared__ int s_best_loc[2];

    auto scan_to_table = [&](int k, int x, int y, int w, int h, int px0, int py0, int px1, int py1) {
        float v; int bx, by;
        const FpmScanStep st = (w == g.bw) ? step_reg : fpm_scan_step(w, lane, false);
        if (w * h <= 64) fpm_scan_block<2>(map, spitch, x, y, w, h, lane, st, px0, py0, px1, py1, v, bx, by);   // small tiles (mode 0)
        else fpm_scan_block<8>(map, spitch, x, y, w, h, lane, st, px0, py0, px1, py1, v, bx, by);
        if (lane == 0) { bval[k] = v; bloc[k] = (by << 16) | bx; }
    };
    // table build: one THREAD per regular block (a sequential scan needs ~4 instructions per element and no
    // cross-lane reduction; the warp-cooperative scan is kept for the picks, where latency counts, and for the
    // big irregular strips)
    const int regular_seq = (g.bw * g.bh <= 256) ? regular : 0;   // big tiles stay warp-cooperative
    for (int k = tid; k < regular_seq; k += nthreads) {
        const int gy = k / g.ncol, gx = k - gy * g.ncol;
        const int x = gx * g.bw, y = gy * g.bh;
        const int w = min(g.bw, cols - x), h = min(g.bh, rows - y);
        float best = -INFINITY; int bx = 0, by = 0;
        for (int yy = 0; yy < h; yy++) {
            const float* rowp = map + (size_t)(y + yy) * spitch + x;
            for (int xx = 0; xx < w; xx++) {
                const float v = rowp[xx];
                if (v > best) { best = v; bx = xx; by = yy; }
            }
        }
        bval[k] = best; bloc[k] = ((y + by) << 16) | (x + bx);
    }
    for (int k = regular_seq + warp; k < g.nblocks; k += nwarps) {
        int x, y, w, h;
        fpm_block_rect(g, k, cols, rows, x, y, w, h);
        scan_to_table(k, x, y, w, h, 0, 0, 0, 0);
    }
    __syncthreads();
    auto refresh_sup = [&](int s) {
        int k = (s << 5) + lane;
        float v = -INFINITY; int kk = 0x7fffffff, l = 0x7fffffff;
        if (k < g.nblocks) { v = bval[k]; kk = k; l = bloc[k]; }
        fpm_pick_warp_reduce(mode, v, kk, l);
        if (lane == 0) { s_sv[s] = v; s_sk[s] = kk; s_sl[s] = l; }
    };
    for (int s = warp; s < nsup; s += nwarps) refresh_sup(s);
    __syncthreads();

    // getNextMaxLoc's rectangle (:1184-1222): constant size, origin follows the last pick
    const double off_x = (double)tw * (1 - max_overlap), off_y = (double)th * (1 - max_overlap);
    const int rw = (int)(2 * (double)tw * (1 - max_overlap));
    const int rh = (int)(2 * (double)th * (1 - max_overlap));
    const int RX = g.ncol * g.bw, RY = g.nrow * g.bh;
    int npicks = 0;
    int lastx = 0, lasty = 0;
    for (int it = 0; it < max_picks; it++) {
        if (it > 0) {
            // paint the suppression rectangle, refresh the touched blocks
            const int sx = (int)((double)lastx - off_x);
            const int sy = (int)((double)lasty - off_y);
            const int px0 = max(sx, 0), py0 = max(sy, 0), px1 = min(sx + rw, cols), py1 = min(sy + rh, rows);
            const int pw = px1 - px0, ph = py1 - py0;
            if (rw > 0 && rh > 0 && pw > 0 && ph > 0) {
                for (int yy = warp; yy < ph; yy += nwarps)
                    for (int xx = lane; xx < pw; xx += 32) map[(size_t)(py0 + yy) * spitch + px0 + xx] = -1.0f;
                // (no barrier: the rescans below treat the rectangle as painted without reading it)
                // blocks of the regular grid under the rectangle, plus the strips of mode 1
                const int bx0 = fpm_fastdiv(px0, div_bw), bx1 = min(fpm_fastdiv(px1 - 1, div_bw), g.ncol - 1);
                const int by0 = fpm_fastdiv(py0, div_bh), by1 = min(fpm_fastdiv(py1 - 1, div_bh), g.nrow - 1);
                int nbx = max(bx1 - bx0 + 1, 0), nby = max(by1 - by0 + 1, 0);
                if (nbx == 0 || nby == 0) nbx = nby = 0;
                const int nreg = nbx * nby;
                const int hit_right = g.has_right && px1 > RX;
                const int hit_bottom = g.has_bottom && py1 > RY && px0 < g.bottom_w;
                const int hit_corner = g.has_corner && px1 > RX && py1 > RY;
                for (int idx = warp; idx < nreg + 3; idx += nwarps) {
                    if (idx < nreg) {
                        int r = 0, c = idx;
                        while (c >= nbx) { c -= nbx; r++; }
                        const int gx = bx0 + c, gy = by0 + r;
                        const int x = gx * g.bw, y = gy * g.bh;
                        scan_to_table(gy * g.ncol + gx, x, y, min(g.bw, cols - x), min(g.bh, rows - y), px0, py0, px1, py1);
                    } else {
                        const int e = idx - nreg;
                        int k;
                        if (e == 0) { if (!hit_right) continue; k = regular; }
                        else if (e == 1) { if (!hit_bottom) continue; k = regular + g.has_right; }
                        else { if (!hit_corner) continue; k = regular + g.has_right + g.has_bottom; }
                        int x, y, w, h;
                        fpm_block_rect(g, k, cols, rows, x, y, w, h);
                        scan_to_table(k, x, y, w, h, px0, py0, px1, py1);
                    }
                }
                __syncthreads();
                // super-entries over the touched block runs (a run of nbx blocks per grid row)
                const int span = (nbx + 62) >> 5;
                for (int idx = warp; idx < nby * span + 3; idx += nwarps) {
                    int s;
                    if (idx < nby * span) {
                        int r = 0, j = idx;
                        while (j >= span) { j -= span; r++; }
                        const int k0 = (by0 + r) * g.ncol + bx0;
                        s = (k0 >> 5) + j;
                        if (s > ((k0 + nbx - 1) >> 5)) continue;
                    } else {
                        const int k = regular + (idx - nby * span);
                        if (k >= g.nblocks) continue;
                        s = k >> 5;
                    }
                    refresh_sup(s);
                }
                __syncthreads();
            }
        }
        // argmax over the super-table
        if (warp == 0) {
            float best = -INFINITY; int bk = 0x7fffffff, bl = 0x7fffffff;
            for (int s = lane; s < nsup; s += 32)
                if (fpm_pick_better(mode, s_sv[s], s_sk[s], s_sl[s], best, bk, bl)) { best = s_sv[s]; bk = s_sk[s]; bl = s_sl[s]; }
            fpm_pick_warp_reduce(mode, best, bk, bl);
            if (lane == 0) {
                if (g.nblocks == 0) { best = -1.0f; bl = -1; }      // s_BlockMax::GetMaxValueLoc on empty
                s_best_v[it & 1] = best; s_best_loc[it & 1] = bl;   // double-buffered: the next write is two barriers away
            }
        }
        __syncthreads();
        const float v = s_best_v[it & 1]; const int loc = s_best_loc[it & 1];
        if ((double)v < thresh) break;
        lastx = loc >= 0 ? (loc & 0xffff) : -1; lasty = loc >= 0 ? (loc >> 16) : -1;
        if (tid == 0) { FpmPick p; p.x = lastx; p.y = lasty; p.v = v; picks[(size_t)job * max_picks + npicks] = p; }
        npicks++;
    }
    if (tid == 0) pick_count[job] = npicks;
}

// =====================================================================================
// bitonic sort of 64-bit keys held in shared or global memory by one CTA (n_pad power of two)
// =====================================================================================
__device__ __forceinline__ void fpm_bitonic_sort(unsigned long long* keys, int n_pad, int tid, int nthreads)
{
    for (int k = 2; k <= n_pad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n_pad; i += nthreads) {
                int ixj = i ^ j;
                if (ixj > i) {
                    unsigned long long a = keys[i], b = keys[ixj];
                    bool up = (i & k) == 0;
                    if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
}

// float -> uint32 whose unsigned order is the DESCENDING float order
__device__ __forceinline__ uint32_t fpm_desc_key(float f)
{
    uint32_t u = __float_as_uint(f);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);   // ascending-order key
    return ~u;
}

// =====================================================================================
// candidate list of one image: gather the picks of all angles (angle-major, pick order), sort by
// score descending (ties keep gather order, like the oracle's stable sort), undo the canvas
// translation (:186) and rotate back into the un-rotated top layer (:265-266).
// =====================================================================================
#define CS_THREADS 1024
#define CS_MAX_SMEM_ANGLES 1024     // angle sweeps up to this size keep their pick-count prefix in shared memory

// Where the picks of (image, angle) live.  Contiguous: picks[(img*n_angles + a)*max_picks], count[img*n_angles + a].
// Segmented (angle-sharded mode, one frame, images = the templates of a group): the buffer is the result of an allgather
// of one fixed-size block per rank; rank r swept angles [r*seg_angles, (r+1)*seg_angles) of the schedule, and in its block
// the group's picks of (img, local angle l) sit at picks[(img*seg_angles + l)*max_picks] and their count at
// count[img*seg_angles + l], both pointers shifted by r*seg_stride bytes.  The gathered buffer is consumed in place.
struct FpmPickView {
    const FpmPick* picks;       // segmented: the group's picks in rank block 0
    const int* count;           // segmented: the group's counts in rank block 0
    int seg_angles;             // 0 = contiguous
    size_t seg_stride;          // bytes per rank block
};
__device__ __forceinline__ const FpmPick* fpm_pick_row(const FpmPickView& v, int img, int n_angles, int max_picks, int a)
{
    if (v.seg_angles == 0) return v.picks + ((size_t)img * n_angles + a) * max_picks;
    const int r = a / v.seg_angles, l = a - r * v.seg_angles;
    return reinterpret_cast<const FpmPick*>(reinterpret_cast<const char*>(v.picks) + (size_t)r * v.seg_stride) +
           ((size_t)img * v.seg_angles + l) * max_picks;
}
__device__ __forceinline__ int fpm_pick_count(const FpmPickView& v, int img, int n_angles, int max_picks, int a)
{
    if (v.seg_angles == 0) return v.count[img * n_angles + a];
    const int r = a / v.seg_angles, l = a - r * v.seg_angles;
    return reinterpret_cast<const int*>(reinterpret_cast<const char*>(v.count) + (size_t)r * v.seg_stride)[img * v.seg_angles + l];
}

// shard_n > 1 (angle-sharded mode): every rank sorts the identical global list and keeps candidates
// id % shard_n == shard_rank (candidate k -> rank k mod N); cand_count still reports the global count.
__global__ void __launch_bounds__(CS_THREADS)
fpm_collect_sort_kernel(FpmPickView pv,
                        int n_angles, int max_picks, const double* __restrict__ angles,
                        const float* __restrict__ ftx, const float* __restrict__ fty,
                        float centre_x, float centre_y,
                        unsigned long long* __restrict__ key_scratch, int key_stride, int use_smem,
                        int* __restrict__ off_scratch,
                        FpmCand* __restrict__ cands_flat, int* __restrict__ flat_counter,
                        float* __restrict__ top_pt, int cand_stride,
                        int* __restrict__ cand_count, int angle_idx_base, int shard_rank, int shard_n,
                        const double* __restrict__ scales)
{
    // pose slot a = scale index * n_angles_of_the_schedule + angle index (angles[a], scales[a]; scales null: every slot at scale 1).
    // At scale s != 1 the canvas resampled the level by 1/s around the centre: a pick maps back by centre + s * (p - centre)
    // before the un-rotation
    extern __shared__ unsigned long long s_keys[];
    const int img = blockIdx.x, tid = threadIdx.x;
    __shared__ int s_n, s_base;
    __shared__ int s_cnt[CS_MAX_SMEM_ANGLES], s_offs[CS_MAX_SMEM_ANGLES];
    // prefix of the pick counts per angle: in shared memory (counts loaded in parallel, a short serial scan over
    // shared memory) unless the sweep has more angles than fit; a serial loop over GLOBAL memory here and in the
    // fill loop below used to be most of this kernel's time (one L2 round trip per angle)
    const bool offs_smem = n_angles <= CS_MAX_SMEM_ANGLES;
    int* s_off = offs_smem ? s_offs : off_scratch + (size_t)img * n_angles;
    if (offs_smem) {
        for (int a = tid; a < n_angles; a += CS_THREADS) s_cnt[a] = fpm_pick_count(pv, img, n_angles, max_picks, a);
        __syncthreads();
    }
    if (tid == 0) {
        int n = 0;
        for (int a = 0; a < n_angles; a++) { s_off[a] = n; n += offs_smem ? s_cnt[a] : fpm_pick_count(pv, img, n_angles, max_picks, a); }
        s_n = n;
        const int mine = n > shard_rank ? (n - shard_rank + shard_n - 1) / shard_n : 0;
        s_base = atomicAdd(flat_counter, mine);
    }
    __syncthreads();
    const int n = s_n;
    const int base = s_base;
    int n_pad = 1;
    while (n_pad < n) n_pad <<= 1;
    unsigned long long* keys = use_smem ? s_keys : key_scratch + (size_t)img * key_stride;
    for (int i = tid; i < n_pad; i += CS_THREADS) keys[i] = ~0ull;
    __syncthreads();
    if (offs_smem) {
        // one thread per (angle, pick slot): the few picks of all angles are fetched in parallel
        for (int i = tid; i < n_angles * max_picks; i += CS_THREADS) {
            const int a = i / max_picks, j = i - a * max_picks;
            if (j < s_cnt[a]) {
                const FpmPick& p = fpm_pick_row(pv, img, n_angles, max_picks, a)[j];
                keys[s_off[a] + j] = ((unsigned long long)fpm_desc_key(p.v) << 32) | (uint32_t)i;
            }
        }
    } else {
        for (int a = 0; a < n_angles; a++) {
            int c = fpm_pick_count(pv, img, n_angles, max_picks, a);
            for (int j = tid; j < c; j += CS_THREADS) {
                const FpmPick& p = fpm_pick_row(pv, img, n_angles, max_picks, a)[j];
                uint32_t order = (uint32_t)(a * max_picks + j);
                keys[s_off[a] + j] = ((unsigned long long)fpm_desc_key(p.v) << 32) | order;
            }
        }
    }
    __syncthreads();
    fpm_bitonic_sort(keys, n_pad, tid, CS_THREADS);
    for (int i = tid; i < n; i += CS_THREADS) {
        uint32_t order = (uint32_t)(keys[i] & 0xffffffffu);
        int a = order / max_picks, j = order - a * max_picks;
        const FpmPick& p = fpm_pick_row(pv, img, n_angles, max_picks, a)[j];
        float ptx = (float)p.x - ftx[a], pty = (float)p.y - fty[a];
        if (i % shard_n == shard_rank) {
            FpmCand c;
            c.angle = angles[a];
            c.score = (double)p.v;
            c.img = img; c.id = i;
            c.scale = scales ? scales[a] : 1.0;
            double dRAngle = -c.angle * FPM_D2R;
            float qx = ptx, qy = pty;
            if (c.scale != 1.0) fpm_scale_about(ptx, pty, centre_x, centre_y, c.scale, &qx, &qy);
            fpm_pt_rotate(qx, qy, centre_x, centre_y, dRAngle, &c.ptx, &c.pty);
            cands_flat[base + i / shard_n] = c;
        }
        if (top_pt) {
            float* t = top_pt + ((size_t)img * cand_stride + i) * 4;
            t[0] = ptx; t[1] = pty; t[2] = p.v; t[3] = (float)(a + angle_idx_base);
        }
    }
    if (tid == 0) cand_count[img] = n;
}

// =====================================================================================
// refinement, per layer.  Eval e = candidate * n_ang + j.
// prep: rotation matrix of getRotatedROI (src/TemplateMatcher.cpp:1074-1088), inverted like warpAffine
// =====================================================================================
__global__ void fpm_refine_prep_kernel(const FpmCand* __restrict__ cands, int n_cands, int n_ang,
                                       double angle_step, int lvl_w, int lvl_h, int tpl_w, int tpl_h,
                                       FpmWarpJob* __restrict__ jobs, const int* __restrict__ n_cands_dev, int n_tpl)
{
    if (n_cands_dev) n_cands = min(n_cands, *n_cands_dev);
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_cands * n_ang) return;
    int ci = e / n_ang, j = e - ci * n_ang;
    jobs[e] = fpm_refine_job(cands[ci], j, n_ang, 1, angle_step, 0.0, lvl_w, lvl_h, tpl_w, tpl_h, n_tpl);
}

// =====================================================================================
// K5  correlation row sums (replaces IM_Conv_SIMD, src/TemplateMatcher.cpp:461-483):
//   rowsum[e][tr][r*7+c] = sum_x T[tr][x] * S_e[tr + r][x + c]      exact s32, dp4a
//   rowS[e][y][c] = sum_{x<w} S_e[y][x+c],  rowQ[e][y][c] = sum_{x<w} S_e[y][x+c]^2
//
// One THREAD owns one ROI row y of one eval and keeps all 49 sums (7 template rows y-6..y x 7
// column shifts) in registers, so no cross-lane reduction is needed at any template width.
// The CTA walks the row in slabs of 32 words (128 px): the slab of its ROI rows and of the
// template rows y0-6 .. y0+RB-1 is staged in shared memory with coalesced loads (odd word pitch:
// lanes read different rows conflict-free).  Per word: 1 new ROI word + 7 template words from
// shared memory, 5 funnel shifts, 49 dp4a.  Window sums are kept for shift 0 only and the other
// six follow exactly from the 6 head / 6 tail bytes of the row.  Results leave through a shared
// memory transpose so the global stores are coalesced.
//   CTA layout: evals_per_cta x rb threads; thread (el, yl) -> eval blockIdx.y*evals_per_cta+el,
//   row y = blockIdx.x*rb + yl.
//   Template groups (tpl.n_tpl > 1): the evals of a CTA may belong to different templates (template of eval e =
//   cands[e / n_ang].img % n_tpl), so every eval stages its own template rows.
// =====================================================================================
#define CR_SLAB 32                // template words per slab (128 px)
#define CR_PW 36                  // slab row pitch in words: 32 + 4 look-ahead; 36 = 4 (mod 32), so a
                                  // warp of lanes reading 16 B each from consecutive rows is conflict-free
#define CR_MAX_THREADS 256

__device__ __forceinline__ uint32_t fpm_shift_bytes(uint32_t lo, uint32_t hi, int c)
{
    return __funnelshift_r(lo, hi, 8 * c);
}

__device__ __forceinline__ uint32_t fpm_u4(const uint4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

__global__ void __launch_bounds__(CR_MAX_THREADS)
fpm_corr_rows_kernel(const uint8_t* __restrict__ roi, int rpitch, size_t roi_stride, FpmTplLevel tpl,
                     int n_evals, int rb, int evals_per_cta, int32_t* __restrict__ rowsum,
                     int32_t* __restrict__ rowS, int32_t* __restrict__ rowQ, const int* __restrict__ n_evals_dev, int n_ang,
                     const FpmCand* __restrict__ cands)
{
    extern __shared__ __align__(16) uint32_t smem_w[];
    if (n_evals_dev) {                                       // live evals known only on the device (n_ang per candidate)
        n_evals = min(n_evals, *n_evals_dev * n_ang);
        if ((int)blockIdx.y * evals_per_cta >= n_evals) return;
    }
    const int tw = tpl.w, th = tpl.h;
    const int rh = th + FPM_ROI_PAD;                       // ROI rows per eval
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int el = tid / rb, yl = tid - el * rb;
    const int e0 = blockIdx.y * evals_per_cta;
    const int e = e0 + el;
    const int y0 = blockIdx.x * rb;
    const int y = y0 + yl;
    const bool active = (el < evals_per_cta) && (e < n_evals) && (y < rh);
    const int n_srow = evals_per_cta * rb;                 // staged ROI rows
    const int n_trow = rb + FPM_ROI_PAD;                   // staged template rows: tr = y0-6 .. y0+rb-1
    const int n_tblk = tpl.n_tpl > 1 ? evals_per_cta : 1;  // staged templates: one per eval in a group
    const int stage_words = (n_srow + n_tblk * n_trow) * CR_PW;   // one slab buffer: ROI rows then template rows
    const int nw = (tw + 3) / 4;                           // template words per row
    const int tail = tw & 3;
    const uint32_t tailbm = tail ? (0xffffffffu >> (8 * (4 - tail))) : 0xffffffffu;
    const int nslabs = (nw + CR_SLAB - 1) / CR_SLAB;

    // stage slab `si` into buffer si&1 with 16-byte cp.async:
    //   ROI words xs .. xs+35 of every row (9 chunks), template words xs .. xs+31 (8 chunks)
    auto stage = [&](int si) {
        const int xb = si * CR_SLAB * 4;                     // byte offset of the slab in a row
        uint32_t* b_s = smem_w + (size_t)(si & 1) * stage_words;
        uint32_t* b_t = b_s + (size_t)n_srow * CR_PW;
        for (int i = tid; i < n_srow * 9; i += nthreads) {
            const int r = i / 9, c = i - r * 9;
            int rel = 0, ry = r;
            if (evals_per_cta > 1) { rel = r / rb; ry = r - rel * rb; }
            ry += y0;
            const int re = e0 + rel;
            const bool ok = re < n_evals && ry < rh && xb + 16 * c < rpitch;
            const uint8_t* g = ok ? roi + (size_t)re * roi_stride + (size_t)ry * rpitch + xb + 16 * c : roi;
            fpm_cp_async16z(b_s + r * CR_PW + 4 * c, g, ok);
        }
        for (int i = tid; i < n_tblk * n_trow * 8; i += nthreads) {
            const int rr = i >> 3, c = i & 7;
            const int tb = rr / n_trow, r = rr - tb * n_trow;
            const int tr = y0 - FPM_ROI_PAD + r;
            const uint8_t* tp = tpl.ptr;
            if (tpl.n_tpl > 1 && e0 + tb < n_evals) tp += (size_t)(cands[(e0 + tb) / n_ang].img % tpl.n_tpl) * tpl.tpl_stride;
            const bool ok = tr >= 0 && tr < th && xb + 16 * c < tpl.pitch;
            const uint8_t* g = ok ? tp + (size_t)tr * tpl.pitch + xb + 16 * c : tpl.ptr;
            fpm_cp_async16z(b_t + rr * CR_PW + 4 * c, g, ok);
        }
        fpm_cp_async_commit();
    };

    uint32_t acc[FPM_NSHIFT][FPM_NSHIFT];
#pragma unroll
    for (int j = 0; j < FPM_NSHIFT; j++)
#pragma unroll
        for (int c = 0; c < FPM_NSHIFT; c++) acc[j][c] = 0;
    uint32_t sS = 0, sQ = 0, head0 = 0, head1 = 0;
    uint32_t tailb[6];
#pragma unroll
    for (int k = 0; k < 6; k++) tailb[k] = 0;

    stage(0);
    for (int si = 0; si < nslabs; si++) {
        const int xs = si * CR_SLAB;
        if (si + 1 < nslabs) {
            stage(si + 1);                 // buffer (si+1)&1 was last read in iteration si-1: all threads are past it
            fpm_cp_async_wait<1>();        // slab si has landed (this thread's copies)
        } else {
            fpm_cp_async_wait<0>();
        }
        __syncthreads();
        if (active) {
            const uint32_t* s_s = smem_w + (size_t)(si & 1) * stage_words;
            const uint32_t* s_t = s_s + (size_t)(n_srow + (tpl.n_tpl > 1 ? el * n_trow : 0)) * CR_PW;
            const uint4* srow4 = reinterpret_cast<const uint4*>(s_s + (size_t)tid * CR_PW);
            const uint4* trow4 = reinterpret_cast<const uint4*>(s_t + (size_t)(yl + FPM_ROI_PAD) * CR_PW);   // row tr = y
            const int nx = min(CR_SLAB, nw - xs);
            const int ngroups = (nx + 3) >> 2;
            uint4 cur = srow4[0];
            if (xs == 0) { head0 = cur.x; head1 = cur.y; }
            for (int g = 0; g < ngroups; g++) {
                const uint4 nxt = srow4[g + 1];
                uint4 t4[FPM_NSHIFT];
#pragma unroll
                for (int j = 0; j < FPM_NSHIFT; j++) t4[j] = trow4[g - j * (CR_PW / 4)];        // template row y - j
                const uint32_t w[6] = {cur.x, cur.y, cur.z, cur.w, nxt.x, nxt.y};
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const uint32_t w0 = w[u], w1 = w[u + 1], w2 = w[u + 2];
                    uint32_t sh[FPM_NSHIFT];
                    sh[0] = w0;
                    sh[1] = fpm_shift_bytes(w0, w1, 1);
                    sh[2] = fpm_shift_bytes(w0, w1, 2);
                    sh[3] = fpm_shift_bytes(w0, w1, 3);
                    sh[4] = w1;
                    sh[5] = fpm_shift_bytes(w1, w2, 1);
                    sh[6] = fpm_shift_bytes(w1, w2, 2);
#pragma unroll
                    for (int j = 0; j < FPM_NSHIFT; j++) {
                        const uint32_t t = fpm_u4(t4[j], u);             // zero beyond the template width
#pragma unroll
                        for (int c = 0; c < FPM_NSHIFT; c++) acc[j][c] = __dp4a(t, sh[c], acc[j][c]);
                    }
                    const int idx = xs + 4 * g + u;
                    const uint32_t m0 = idx < nw - 1 ? w0 : (idx == nw - 1 ? (w0 & tailbm) : 0u);
                    sS = __dp4a(m0, 0x01010101u, sS);
                    sQ = __dp4a(m0, m0, sQ);
                }
                cur = nxt;
            }
            if (si == nslabs - 1) {
                // the 6 bytes that follow the template width: S[y][tw .. tw+5]
                const uint8_t* sb = reinterpret_cast<const uint8_t*>(srow4);
#pragma unroll
                for (int k = 0; k < 6; k++) tailb[k] = sb[tw + k - 4 * xs];
            }
        }
        __syncthreads();                   // everyone is done with buffer si&1 before it is refilled
    }
    // ---- window sums of the 7 shifts from shift 0 + head/tail bytes (exact)
    if (active) {
        uint32_t hb[6];
        hb[0] = head0 & 255; hb[1] = (head0 >> 8) & 255; hb[2] = (head0 >> 16) & 255; hb[3] = head0 >> 24;
        hb[4] = head1 & 255; hb[5] = (head1 >> 8) & 255;
        size_t base = ((size_t)e * rh + y) * FPM_WSTRIDE;
        uint32_t cs = sS, cq = sQ;
        int vs[FPM_WSTRIDE], vq[FPM_WSTRIDE];
        vs[0] = (int)cs; vq[0] = (int)cq; vs[FPM_NSHIFT] = 0; vq[FPM_NSHIFT] = 0;
#pragma unroll
        for (int c = 1; c < FPM_NSHIFT; c++) {
            cs = cs - hb[c - 1] + tailb[c - 1];
            cq = cq - hb[c - 1] * hb[c - 1] + tailb[c - 1] * tailb[c - 1];
            vs[c] = (int)cs; vq[c] = (int)cq;
        }
        int4* ps = reinterpret_cast<int4*>(rowS + base);                // one aligned 32-byte record per (eval, row)
        int4* pq = reinterpret_cast<int4*>(rowQ + base);
        ps[0] = make_int4(vs[0], vs[1], vs[2], vs[3]); ps[1] = make_int4(vs[4], vs[5], vs[6], vs[7]);
        pq[0] = make_int4(vq[0], vq[1], vq[2], vq[3]); pq[1] = make_int4(vq[4], vq[5], vq[6], vq[7]);
    }
    // ---- transpose through shared memory: out[el][tr_local][cell], then coalesced global stores
    uint32_t* s_o = smem_w;                                // [evals_per_cta][n_trow][49]
    if (active) {
#pragma unroll
        for (int j = 0; j < FPM_NSHIFT; j++) {
            uint32_t* o = s_o + ((size_t)el * n_trow + (yl + FPM_ROI_PAD - j)) * FPM_NCELL + j * FPM_NSHIFT;
#pragma unroll
            for (int c = 0; c < FPM_NSHIFT; c++) o[c] = acc[j][c];
        }
    }
    __syncthreads();
    const int per_eval = n_trow * FPM_NCELL;
    for (int i = tid; i < evals_per_cta * per_eval; i += nthreads) {
        int oel = i / per_eval, rem = i - oel * per_eval;
        int trl = rem / FPM_NCELL, cell = rem - trl * FPM_NCELL;
        int tr = y0 - FPM_ROI_PAD + trl, oe = e0 + oel;
        int j = cell / FPM_NSHIFT;
        int oy = tr + j;                                     // the ROI row (thread) that produced this cell
        if (oe < n_evals && tr >= 0 && tr < th && oy >= y0 && oy < y0 + rb && oy < rh)
            rowsum[((size_t)oe * th + tr) * FPM_NCELL + cell] = (int32_t)s_o[i];
    }
}

// =====================================================================================
// sub-pixel / sub-angle fit (subPixEstimation, src/TemplateMatcher.cpp:1002-1072):
// Z = (A^T A)^-1 A^T s via LU with partial pivoting (cv::Mat::inv DECOMP_LU for n > 3),
// optimum = K1^-1 K2 with the closed-form 3x3 inverse.
// =====================================================================================
__device__ int fpm_lu_inverse10(double* A /*10x10, destroyed*/, double* B /*10x10 out*/)
{
    const int m = 10;
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) B[i * m + j] = (i == j) ? 1.0 : 0.0;
    const double eps = DBL_EPSILON * 100;
    for (int i = 0; i < m; i++) {
        int k = i;
        for (int j = i + 1; j < m; j++)
            if (fabs(A[j * m + i]) > fabs(A[k * m + i])) k = j;
        if (fabs(A[k * m + i]) < eps) return 0;
        if (k != i) {
            for (int j = i; j < m; j++) { double t = A[i * m + j]; A[i * m + j] = A[k * m + j]; A[k * m + j] = t; }
            for (int j = 0; j < m; j++) { double t = B[i * m + j]; B[i * m + j] = B[k * m + j]; B[k * m + j] = t; }
        }
        double d = -1 / A[i * m + i];
        for (int j = i + 1; j < m; j++) {
            double alpha = A[j * m + i] * d;
            for (int kk = i + 1; kk < m; kk++) A[j * m + kk] += alpha * A[i * m + kk];
            for (int kk = 0; kk < m; kk++) B[j * m + kk] += alpha * B[i * m + kk];
        }
    }
    for (int i = m - 1; i >= 0; i--)
        for (int j = 0; j < m; j++) {
            double s = B[i * m + j];
            for (int k = i + 1; k < m; k++) s -= A[i * m + k] * B[k * m + j];
            B[i * m + j] = s / A[i * m + i];
        }
    return 1;
}

__device__ void fpm_subpix(const double* sc27 /* [theta][y][x] */, double xm, double ym, double tm,
                           double angle_step, double* outx, double* outy, double* outa,
                           double* scratch /* >= 27*10 + 100 + 100 + 270 doubles */)
{
    double* A = scratch;             // 27x10
    double* AtA = A + 270;           // 10x10
    double* Inv = AtA + 100;         // 10x10
    double* P = Inv + 100;           // 10x27
    int row = 0;
    for (int theta = 0; theta <= 2; theta++)
        for (int y = -1; y <= 1; y++)
            for (int x = -1; x <= 1; x++) {
                double dX = xm + x, dY = ym + y;
                double dT = (tm + (theta - 1) * angle_step) * FPM_D2R;
                double* a = A + row * 10;
                a[0] = dX * dX; a[1] = dY * dY; a[2] = dT * dT; a[3] = dX * dY; a[4] = dX * dT;
                a[5] = dY * dT; a[6] = dX; a[7] = dY; a[8] = dT; a[9] = 1.0;
                row++;
            }
    for (int i = 0; i < 10; i++)
        for (int j = 0; j < 10; j++) {
            double s = 0;
            for (int k = 0; k < 27; k++) s += A[k * 10 + i] * A[k * 10 + j];
            AtA[i * 10 + j] = s;
        }
    double Z[10];
    if (!fpm_lu_inverse10(AtA, Inv)) {
        for (int i = 0; i < 100; i++) Inv[i] = 0;   // cv::invert returns a zero matrix when singular
    }
    for (int i = 0; i < 10; i++)
        for (int j = 0; j < 27; j++) {
            double s = 0;
            for (int k = 0; k < 10; k++) s += Inv[i * 10 + k] * A[j * 10 + k];
            P[i * 27 + j] = s;
        }
    for (int i = 0; i < 10; i++) {
        double s = 0;
        for (int k = 0; k < 27; k++) s += P[i * 27 + k] * sc27[k];
        Z[i] = s;
    }
    // matK1.inv() * matK2 (:1066): OpenCV's matrix-expression layer evaluates inv(A) * B as cv::solve(A, B, DECOMP_LU)
    // (MatOp_Invert::matmul), which for a 3x3 double system is this closed form (adjugate rows times b, then * 1/det);
    // pinned bit-for-bit against cv2.solve on 2000 random systems (tests/test_oracle.py)
    const double S00 = 2 * Z[0], S01 = Z[3], S02 = Z[4];
    const double S10 = Z[3], S11 = 2 * Z[1], S12 = Z[5];
    const double S20 = Z[4], S21 = Z[5], S22 = 2 * Z[2];
    const double b0 = -Z[6], b1 = -Z[7], b2 = -Z[8];
    double d = S00 * (S11 * S22 - S12 * S21) - S01 * (S10 * S22 - S12 * S20) + S02 * (S10 * S21 - S11 * S20);
    if (d != 0.) {
        d = 1. / d;
        *outx = ((S11 * S22 - S12 * S21) * b0 + (S02 * S21 - S01 * S22) * b1 + (S01 * S12 - S02 * S11) * b2) * d;
        *outy = ((S12 * S20 - S10 * S22) * b0 + (S00 * S22 - S02 * S20) * b1 + (S02 * S10 - S00 * S12) * b2) * d;
        *outa = (((S10 * S21 - S11 * S20) * b0 + (S01 * S20 - S00 * S21) * b1 + (S00 * S11 - S01 * S10) * b2) * d) * FPM_R2D;
    } else {
        *outx = 0; *outy = 0; *outa = 0;
    }
}

// =====================================================================================
// masked refinement window sums (masked templates and groups): for every eval and every cell (r, c) of its 7x7 patch the exact sums
// of the ROI pixels and of their squares under the KEPT template pixels, t = sum M*S and t2 = sum M*S^2, as int64
// [eval][49] for fpm_refine_finalize_kernel.  One CTA per eval, one warp per ROI row at a time (rows y = warp, warp + nw,
// ...), no block-wide barrier until the end: the warp turns its row into prefix sums P[x] (the pixels left of column x;
// u32 is exact, (tw + 6) * 255^2 < 2^32) with one scan of the lanes' 4-pixel words, then each lane adds
// P[c + e] - P[c + b] over the runs [b, e) of template row y - r for its items of the 98 (cell, sum or square) totals,
// which it keeps in registers across its rows.  The warps' totals meet in shared memory at the end.  About 49 * (sum of
// runs) adds per eval against the 49 * w * h MACs of the numerator; a full mask gives the same integers as the row-window
// sums of the unmasked path.
// =====================================================================================
#define MW_MAX_WARPS 8

__global__ void __launch_bounds__(MW_MAX_WARPS * 32)
fpm_mask_window_kernel(const uint8_t* __restrict__ roi, int rpitch, size_t roi_stride, FpmTplLevel tpl, int ne, int pstride,
                       long long* __restrict__ totS, long long* __restrict__ totQ, const int* __restrict__ n_cands_dev, int n_ang,
                       const FpmCand* __restrict__ cands)
{
    extern __shared__ __align__(16) uint32_t s_pre[];        // per warp: pstride pixel prefix sums, then pstride square ones
    __shared__ unsigned long long s_tot[2 * FPM_NCELL];
    const int e = blockIdx.x;
    if (e >= ne || (n_cands_dev && e >= *n_cands_dev * n_ang)) return;
    if (tpl.n_tpl > 1) {                                     // a group: the eval's own template (CTA-uniform)
        tpl = fpm_tpl_member(tpl, cands[e / n_ang].img % tpl.n_tpl);
        if (tpl.result_equal1) return;                       // finalize scores a flat template 1 without its sums
    }
    const int th = tpl.h, rw = tpl.w + FPM_ROI_PAD, rh = th + FPM_ROI_PAD, pl = rw + 1;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
    for (int i = tid; i < 2 * FPM_NCELL; i += blockDim.x) s_tot[i] = 0;
    uint32_t* s_ps = s_pre + (size_t)warp * 2 * pstride;
    uint32_t* s_pq = s_ps + pstride;
    const uint8_t* __restrict__ base = roi + (size_t)e * roi_stride;
    long long acc[4] = {0, 0, 0, 0};                         // items j = lane + 32 k: j < 49 pixel sums of cell j, else squares
    for (int y = warp; y < rh; y += nw) {
        const uint32_t* row = reinterpret_cast<const uint32_t*>(base + (size_t)y * rpitch);   // rpitch % 16 == 0
        uint32_t cs = 0, cq = 0;
        for (int w0 = 0; 4 * w0 < pl; w0 += 32) {
            const int xw = w0 + lane;
            uint32_t v = 4 * xw < rw ? __ldg(row + xw) : 0u;
            if (4 * xw < rw && 4 * xw + 4 > rw) v &= 0xffffffffu >> (8 * (4 * xw + 4 - rw));
            const uint32_t b0 = v & 255u, b1 = (v >> 8) & 255u, b2 = (v >> 16) & 255u, b3 = v >> 24;
            const uint32_t ws = b0 + b1 + b2 + b3, wq = b0 * b0 + b1 * b1 + b2 * b2 + b3 * b3;
            uint32_t is = ws, iq = wq;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t us = __shfl_up_sync(0xffffffffu, is, o), uq = __shfl_up_sync(0xffffffffu, iq, o);
                if (lane >= o) { is += us; iq += uq; }
            }
            const uint32_t ps = cs + is - ws, pq = cq + iq - wq;  // in front of this word
            if (4 * xw < pl) {                                    // pstride % 4 == 0: the word's 4 entries fit
                *reinterpret_cast<uint4*>(s_ps + 4 * xw) = make_uint4(ps, ps + b0, ps + b0 + b1, ps + b0 + b1 + b2);
                *reinterpret_cast<uint4*>(s_pq + 4 * xw) = make_uint4(pq, pq + b0 * b0, pq + b0 * b0 + b1 * b1,
                                                                      pq + b0 * b0 + b1 * b1 + b2 * b2);
            }
            cs += __shfl_sync(0xffffffffu, is, 31);
            cq += __shfl_sync(0xffffffffu, iq, 31);
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int j = lane + 32 * k;
            if (j >= 2 * FPM_NCELL) continue;
            const int cell = j < FPM_NCELL ? j : j - FPM_NCELL;
            const int r = cell / FPM_NSHIFT, c = cell - r * FPM_NSHIFT, tr = y - r;   // template row over ROI row y in window (r, c)
            if (tr < 0 || tr >= th) continue;
            const uint32_t* p = (j < FPM_NCELL ? s_ps : s_pq) + c;
            uint32_t s = 0;
            for (int q = __ldg(tpl.mrow + tr), qe = __ldg(tpl.mrow + tr + 1); q < qe; q++) {
                const int2 be = __ldg(tpl.mrun + q);
                s += p[be.y] - p[be.x];
            }
            acc[k] += s;
        }
        __syncwarp();                                        // the next row overwrites this warp's prefix sums
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int j = lane + 32 * k;
        if (j < 2 * FPM_NCELL && acc[k]) atomicAdd(&s_tot[j], (unsigned long long)acc[k]);
    }
    __syncthreads();
    for (int i = tid; i < 2 * FPM_NCELL; i += blockDim.x)
        (i < FPM_NCELL ? totS[(size_t)e * FPM_NCELL + i] : totQ[(size_t)e * FPM_NCELL + i - FPM_NCELL]) = (long long)s_tot[i];
}

// =====================================================================================
// refine_finalize: one CTA per candidate, 64 threads per angle.
//   numerator  = float32 chain over template rows of the exact s32 row sums (reference order,
//                src/TemplateMatcher.cpp:505-508) or exact s64 total when use_chain == 0
//   window sums from rowS/rowQ (exact), CCOEFF_NORMED epilogue, minMaxLoc over the 7x7 patch,
//   best of the 3 angles, layer threshold, pose update (src/TemplateMatcher.cpp:331-367)
// =====================================================================================
#define RF_THREADS 192
#define RF_MAXEV 9         // evals per candidate: 3 angles x 3 scales

// GROUP: the candidates are virtual images of a template group (statistics of template img % n_tpl)
template <bool GROUP>
__global__ void __launch_bounds__(RF_THREADS, 6)
fpm_refine_finalize_kernel(const FpmCand* __restrict__ cands, int n_ang, double angle_step,
                           const int32_t* __restrict__ rowsum, int raw_epad, const int32_t* __restrict__ rowS,
                           const int32_t* __restrict__ rowQ, FpmTplLevel tpl, int lvl_w, int lvl_h,
                           double layer_score, int use_chain, int is_last, int out_scale, int subpixel,
                           FpmCand* __restrict__ next, int* __restrict__ next_count,
                           FpmRefined* __restrict__ refined, int* __restrict__ refined_count,
                           FpmEvalTrace* __restrict__ trace, float* __restrict__ trace_scores,
                           const float* __restrict__ numer, const long long* __restrict__ totS,
                           const long long* __restrict__ totQ, int raw_tile_evals, const int* __restrict__ n_cands_dev,
                           int n_sc, double scale_step)
{
    const int ci = blockIdx.x;
    if (n_cands_dev && ci >= *n_cands_dev) return;
    if (GROUP) tpl = fpm_tpl_member(tpl, cands[ci].img % tpl.n_tpl);    // one candidate per CTA: CTA-uniform statistics
    // n_ev = n_sc * n_ang evals per candidate (eval k * n_ang + j: scale index k, angle index j); the 64-thread eval slots
    // j0 = 0, 1, 2 take the evals j0, j0 + 3, j0 + 6
    const int tid = threadIdx.x, j0 = tid >> 6, cell = tid & 63, n_ev = n_sc * n_ang;
    __shared__ float s_sc[RF_MAXEV][FPM_NCELL];
    __shared__ float s_best[RF_MAXEV];
    __shared__ int s_loc[RF_MAXEV];
    __shared__ double s_scratch[27 + 270 + 100 + 100 + 270];
    __shared__ unsigned long long s_totS[RF_MAXEV][FPM_NSHIFT], s_totQ[RF_MAXEV][FPM_NSHIFT];      // sums over ALL ROI rows per shift
    __shared__ int s_edgeS[RF_MAXEV][2 * FPM_ROI_PAD][FPM_NSHIFT], s_edgeQ[RF_MAXEV][2 * FPM_ROI_PAD][FPM_NSHIFT];   // rows 0..5 and th..th+5
    const int th = tpl.h;
    // Window sums of CCOEFF_Denominator.  The 49 windows of an eval share their rows: window (r, c) = total of column c over
    // all th + 6 ROI rows minus the r rows above and the 6 - r rows below it.  The totals are gathered by all 64 threads of
    // the eval (every thread a strided share of the rows, 14 loads per row in flight) instead of a 2*th-load serial loop
    // per cell, which was most of this kernel's time at single-frame latency.
    // A masked template (tpl.mrun set) takes its 49 window sums per eval from totS / totQ [e][49] (fpm_mask_window_kernel).
    const bool masked = tpl.mrun != nullptr;
    const bool coop_window = !tpl.result_equal1 && !numer && !masked;
    if (coop_window) {
        for (int i = tid; i < n_ev * FPM_NSHIFT; i += RF_THREADS) { s_totS[i / FPM_NSHIFT][i % FPM_NSHIFT] = 0; s_totQ[i / FPM_NSHIFT][i % FPM_NSHIFT] = 0; }
        __syncthreads();
        for (int j = j0; j < n_ev; j += 3) {
            const int e = ci * n_ev + j;
            const int rh = th + FPM_ROI_PAD;
            const int32_t* ps = rowS + (size_t)e * rh * FPM_WSTRIDE;
            const int32_t* pq = rowQ + (size_t)e * rh * FPM_WSTRIDE;
            long long ts[FPM_NSHIFT], tq[FPM_NSHIFT];
#pragma unroll
            for (int c = 0; c < FPM_NSHIFT; c++) { ts[c] = 0; tq[c] = 0; }
#pragma unroll 2
            for (int y = cell; y < rh; y += 64) {
                int a[FPM_WSTRIDE], b[FPM_WSTRIDE];
                {                                                        // one 32-byte record per row: two 128-bit loads each
                    const int4 a0 = __ldg(reinterpret_cast<const int4*>(ps + (size_t)y * FPM_WSTRIDE)), a1 = __ldg(reinterpret_cast<const int4*>(ps + (size_t)y * FPM_WSTRIDE) + 1);
                    const int4 b0 = __ldg(reinterpret_cast<const int4*>(pq + (size_t)y * FPM_WSTRIDE)), b1 = __ldg(reinterpret_cast<const int4*>(pq + (size_t)y * FPM_WSTRIDE) + 1);
                    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
                    b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
                }
#pragma unroll
                for (int c = 0; c < FPM_NSHIFT; c++) { ts[c] += a[c]; tq[c] += b[c]; }
                if (y < FPM_ROI_PAD) {
#pragma unroll
                    for (int c = 0; c < FPM_NSHIFT; c++) { s_edgeS[j][y][c] = a[c]; s_edgeQ[j][y][c] = b[c]; }
                }
                if (y >= th) {
#pragma unroll
                    for (int c = 0; c < FPM_NSHIFT; c++) { s_edgeS[j][FPM_ROI_PAD + y - th][c] = a[c]; s_edgeQ[j][FPM_ROI_PAD + y - th][c] = b[c]; }
                }
            }
#pragma unroll
            for (int c = 0; c < FPM_NSHIFT; c++) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    ts[c] += __shfl_xor_sync(0xffffffffu, ts[c], o);
                    tq[c] += __shfl_xor_sync(0xffffffffu, tq[c], o);
                }
                if ((tid & 31) == 0) {
                    atomicAdd(&s_totS[j][c], (unsigned long long)ts[c]);
                    atomicAdd(&s_totQ[j][c], (unsigned long long)tq[c]);
                }
            }
        }
        __syncthreads();
    }
    for (int j = j0; j < n_ev && cell < FPM_NCELL; j += 3) {
        const int e = ci * n_ev + j;
        const int r = cell / FPM_NSHIFT, c = cell - r * FPM_NSHIFT;
        float sc;
        if (tpl.result_equal1) {
            sc = 1.0f;
        } else if (numer) {
            // fused tensor-core kernel: the float chain is already folded (column 8c + 7 - r), the window sums are
            // the totals over all ROI rows minus the r rows above and the 6 - r rows below the window
            const float numf = numer[(size_t)e * 64 + c * 8 + (7 - r)];
            long long ws, wq;
            if (masked) {
                ws = totS[(size_t)e * FPM_NCELL + cell]; wq = totQ[(size_t)e * FPM_NCELL + cell];
            } else {
                const int rh = th + FPM_ROI_PAD;
                ws = totS[(size_t)e * FPM_NSHIFT + c]; wq = totQ[(size_t)e * FPM_NSHIFT + c];
                const int32_t* ps = rowS + (size_t)e * rh * FPM_WSTRIDE + c;
                const int32_t* pq = rowQ + (size_t)e * rh * FPM_WSTRIDE + c;
                for (int y = 0; y < r; y++) { ws -= ps[(size_t)y * FPM_WSTRIDE]; wq -= pq[(size_t)y * FPM_WSTRIDE]; }
                for (int y = r + th; y < rh; y++) { ws -= ps[(size_t)y * FPM_WSTRIDE]; wq -= pq[(size_t)y * FPM_WSTRIDE]; }
            }
            sc = fpm_ccoeff_epilogue(numf, (double)ws, (double)wq, tpl.mean, tpl.norm, tpl.inv_area);
        } else {
            // row sums either as [e][tr][49] (dp4a kernel) or as raw[y][e_pad][64] with y = tr + r and
            // column 8c + 7 - r (tensor-core kernel); both walked in template-row order
            const int32_t* rs;
            size_t rstride;
            if (raw_epad) {
                // eval -> row of the raw buffer: contiguous, or 128-row tiles that hold raw_tile_evals evals each (fpm_corr_warp_kernel)
                const int slot = raw_tile_evals ? (e / raw_tile_evals) * 128 + e % raw_tile_evals : e;
                rs = rowsum + ((size_t)r * raw_epad + slot) * 64 + c * 8 + (7 - r);
                rstride = (size_t)raw_epad * 64;
            } else {
                rs = rowsum + (size_t)e * th * FPM_NCELL + cell;
                rstride = FPM_NCELL;
            }
            float numf;
            // loads are issued 32 at a time (independent), the additions stay in template-row order
            if (use_chain) {
                float acc = 0.0f;
                int tr = 0;
                for (; tr + 32 <= th; tr += 32) {
                    int v[32];
#pragma unroll
                    for (int k = 0; k < 32; k++) v[k] = rs[(size_t)(tr + k) * rstride];
#pragma unroll
                    for (int k = 0; k < 32; k++) acc = __fadd_rn(acc, __int2float_rn(v[k]));
                }
                for (; tr + 8 <= th; tr += 8) {
                    int v[8];
#pragma unroll
                    for (int k = 0; k < 8; k++) v[k] = rs[(size_t)(tr + k) * rstride];
#pragma unroll
                    for (int k = 0; k < 8; k++) acc = __fadd_rn(acc, __int2float_rn(v[k]));
                }
                for (; tr < th; tr++) acc = __fadd_rn(acc, __int2float_rn(rs[(size_t)tr * rstride]));
                numf = acc;
            } else {
                long long acc = 0;
#pragma unroll 8
                for (int tr = 0; tr < th; tr++) acc += rs[(size_t)tr * rstride];
                numf = (float)acc;
            }
            long long ws, wq;
            if (masked) {
                ws = totS[(size_t)e * FPM_NCELL + cell]; wq = totQ[(size_t)e * FPM_NCELL + cell];
            } else {
                ws = (long long)s_totS[j][c]; wq = (long long)s_totQ[j][c];
                for (int y = 0; y < r; y++) { ws -= s_edgeS[j][y][c]; wq -= s_edgeQ[j][y][c]; }
                for (int y = r; y < FPM_ROI_PAD; y++) { ws -= s_edgeS[j][FPM_ROI_PAD + y][c]; wq -= s_edgeQ[j][FPM_ROI_PAD + y][c]; }   // ROI rows th + r .. th + 5
            }
            sc = fpm_ccoeff_epilogue(numf, (double)ws, (double)wq, tpl.mean, tpl.norm, tpl.inv_area);
        }
        s_sc[j][cell] = sc;
        if (trace_scores) trace_scores[(size_t)e * FPM_NCELL + cell] = sc;
    }
    __syncthreads();
    for (int j = j0; j < n_ev && cell == 0; j += 3) {
        float best = s_sc[j][0]; int loc = 0;
        for (int i = 1; i < FPM_NCELL; i++) if (s_sc[j][i] > best) { best = s_sc[j][i]; loc = i; }
        s_best[j] = best; s_loc[j] = loc;
    }
    __syncthreads();
    if (tid != 0) return;
    const FpmCand c = cands[ci];
    int bi = 0; double big = -1;
    for (int k = 0; k < n_ev; k++) {                                   // the first strict maximum in eval order
        const int ja = k % n_ang;
        double ang = (n_ang == 1) ? 0.0 : c.angle + angle_step * (double)(ja - 1);
        if ((double)s_best[k] > big) { bi = k; big = (double)s_best[k]; }
        if (trace) {
            FpmEvalTrace t; t.angle = ang; t.score = s_best[k]; t.locx = s_loc[k] % FPM_NSHIFT; t.locy = s_loc[k] / FPM_NSHIFT;
            trace[ci * n_ev + k] = t;
        }
    }
    if ((double)s_best[bi] < layer_score) return;                      // :331-332
    const int bj = bi % n_ang, b0 = bi - bj;                           // angle index of the best eval, first eval of its scale
    const double scale = fpm_eval_scale(c.scale, bi / n_ang, n_sc, scale_step);
    double new_angle = (n_ang == 1) ? 0.0 : c.angle + angle_step * (double)(bj - 1);
    int lx = s_loc[bi] % FPM_NSHIFT, ly = s_loc[bi] / FPM_NSHIFT;
    double ptx = (double)lx, pty = (double)ly;
    bool on_border = (lx == 0 || ly == 0 || lx == FPM_NSHIFT - 1 || ly == FPM_NSHIFT - 1);
    if (subpixel && is_last && !on_border && bj == 1 && n_ang == 3) {    // :334-344 (the three angle evals of the best scale)
        // neighbours of the other two angles are taken around THEIR OWN maxima (vecResult, :323-328);
        // an angle whose maximum sits on the border leaves vecResult unset in the reference -> 0 here
        double* sc27 = s_scratch;
        for (int t = 0; t < 3; t++) {
            int tx = s_loc[b0 + t] % FPM_NSHIFT, ty = s_loc[b0 + t] / FPM_NSHIFT;
            bool tb = (tx == 0 || ty == 0 || tx == FPM_NSHIFT - 1 || ty == FPM_NSHIFT - 1);
            for (int y = -1; y <= 1; y++)
                for (int x = -1; x <= 1; x++)
                    sc27[t * 9 + (y + 1) * 3 + (x + 1)] = tb ? 0.0 : (double)s_sc[b0 + t][(ty + y) * FPM_NSHIFT + tx + x];
        }
        double nx, ny, na;
        fpm_subpix(sc27, ptx, pty, new_angle, angle_step, &nx, &ny, &na, s_scratch + 27);
        ptx = nx; pty = ny; new_angle = na;
    }
    float ptcx = (float)(lvl_w - 1) / 2.0f, ptcy = (float)(lvl_h - 1) / 2.0f;
    float ltx = c.ptx * 2, lty = c.pty * 2;
    float padx, pady;
    fpm_pt_rotate(ltx, lty, ptcx, ptcy, new_angle * FPM_D2R, &padx, &pady);      // :350
    if (scale != 1.0) fpm_scale_about(padx, pady, ptcx, ptcy, 1.0 / scale, &padx, &pady);   // the ROI's anchor (fpm_refine_job)
    padx = padx - 3.0f; pady = pady - 3.0f;
    float qx = (float)(ptx + (double)padx), qy = (float)(pty + (double)pady);    // :351
    if (scale != 1.0) fpm_scale_about(qx, qy, ptcx, ptcy, scale, &qx, &qy);
    float rx, ry;
    fpm_pt_rotate(qx, qy, ptcx, ptcy, -new_angle * FPM_D2R, &rx, &ry);           // :353
    if (is_last) {
        FpmRefined o;
        o.angle = new_angle; o.score = (double)s_best[bi];
        o.ptx = (double)(rx * (float)out_scale); o.pty = (double)(ry * (float)out_scale);   // pt * (iStopLayer == 0 ? 1 : 2), :357
        o.img = c.img; o.id = c.id; o.scale = scale;
        refined[atomicAdd(refined_count, 1)] = o;
    } else {
        FpmCand o = c;
        o.angle = new_angle;
        o.scale = scale;
        o.score = (double)s_best[bi];
        o.ptx = rx; o.pty = ry;
        next[atomicAdd(next_count, 1)] = o;
    }
}

// m_ckBitwiseNot (MatchTool/MatchToolDlg.cpp:788-794): the match runs on 255 - src
__global__ void fpm_invert_kernel(const uint8_t* __restrict__ src, int w, int h, int spitch, size_t simg,
                                  uint8_t* __restrict__ dst, int dpitch, size_t dimg)
{
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x >= w) return;
    const uint8_t* s = src + (size_t)blockIdx.z * simg + (size_t)y * spitch + x;
    uint8_t* d = dst + (size_t)blockIdx.z * dimg + (size_t)y * dpitch + x;
    uint32_t v = 0;
    for (int k = 0; k < 4 && x + k < w; k++) v |= (uint32_t)(255 - s[k]) << (8 * k);
    *reinterpret_cast<uint32_t*>(d) = v;                 // dpitch is a multiple of 128: the padded tail is ours
}

// ---- image ingest (SURVEY 8f rank 4): decode on the device -------------------------------------------------
// Uncompressed Windows BMP rows -> u8 grayscale like cv::imread(path, IMREAD_GRAYSCALE) (src/MatchToolDialog.cpp:314,341):
// 8-bit indices go through a gray look-up table built from the palette, 24-bit BGR pixels through OpenCV's fixed-point
// weights (B*1868 + G*9617 + R*4899 + 8192) >> 14 (both pinned against cv2.imdecode in tests/test_ingest.py).
struct FpmBmpLut { uint8_t g[256]; };

__global__ void fpm_ingest_bmp_kernel(const uint8_t* __restrict__ file, size_t data_off, size_t row_stride, int bpp,
                                      int top_down, FpmBmpLut lut, int w, int h, uint8_t* __restrict__ dst, int dpitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const uint8_t* row = file + data_off + (size_t)(top_down ? y : h - 1 - y) * row_stride;
    uint8_t v;
    if (bpp == 8) {
        v = lut.g[row[x]];
    } else {
        const uint32_t b = row[3 * x], g = row[3 * x + 1], r = row[3 * x + 2];
        v = (uint8_t)((b * 1868u + g * 9617u + r * 4899u + 8192u) >> 14);
    }
    dst[(size_t)y * dpitch + x] = v;
}

// Camera frame hand-off (src/MatchToolDialog.cpp:1557-1575: QImage::convertToFormat(Format_Grayscale8) of an RGB32 frame):
// 0xAARRGGBB pixels -> qGray = (R*11 + G*16 + B*5) / 32 (Qt's documented integer formula; no Qt here to pin it against)
__global__ void fpm_ingest_rgb32_kernel(const uint32_t* __restrict__ px, int spitch_words, int w, int h,
                                        uint8_t* __restrict__ dst, int dpitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const uint32_t p = px[(size_t)y * spitch_words + x];
    const uint32_t r = (p >> 16) & 255u, g = (p >> 8) & 255u, b = p & 255u;
    dst[(size_t)y * dpitch + x] = (uint8_t)((r * 11u + g * 16u + b * 5u) >> 5);
}

// JPEG luma blocks -> u8 pixels: dequantisation + libjpeg's accurate integer IDCT (JDCT_ISLOW, jidctint.c: the decoder
// behind cv::imread, 13-bit constants, 2 extra bits after the column pass, descale by 18 after the row pass) + the
// post-IDCT range limit (10-bit wrap, +128, clamp).  One thread per 8x8 block; integer-exact, so the frame is bit-identical
// to cv2.imdecode(IMREAD_GRAYSCALE) (tests/test_ingest.py).  The Huffman decoding happened on the device (fpm_jpeg_par.cuh)
// or on the host (fpm_jpeg.h).

__device__ __forceinline__ void fpm_idct_islow_1d(const int (&in)[8], int (&out)[8], int shift)
{
    // even part
    int z2 = in[2], z3 = in[6];
    int z1 = (z2 + z3) * 4433;                                       // FIX(0.541196100)
    int tmp2 = z1 + z3 * -15137;                                     // FIX(1.847759065)
    int tmp3 = z1 + z2 * 6270;                                       // FIX(0.765366865)
    int tmp0 = (in[0] + in[4]) << 13, tmp1 = (in[0] - in[4]) << 13;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    // odd part
    tmp0 = in[7]; tmp1 = in[5]; tmp2 = in[3]; tmp3 = in[1];
    z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
    int z4 = tmp1 + tmp3;
    const int z5 = (z3 + z4) * 9633;                                 // FIX(1.175875602)
    tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;       // FIX(0.298631336, 2.053119869, 3.072711026, 1.501321110)
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;            // FIX(0.899976223, 2.562915447, 1.961570560, 0.390180644)
    z3 += z5; z4 += z5;
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
    const int r = 1 << (shift - 1);
    out[0] = (tmp10 + tmp3 + r) >> shift; out[7] = (tmp10 - tmp3 + r) >> shift;
    out[1] = (tmp11 + tmp2 + r) >> shift; out[6] = (tmp11 - tmp2 + r) >> shift;
    out[2] = (tmp12 + tmp1 + r) >> shift; out[5] = (tmp12 - tmp1 + r) >> shift;
    out[3] = (tmp13 + tmp0 + r) >> shift; out[4] = (tmp13 - tmp0 + r) >> shift;
}

// One file of the wave per grid row (blockIdx.y).  Files decoded on the device take their DC values from dcval (luma blocks in
// scan order from f.luma0, each still short of its tile's offset dc_tile_off[L / 4096], fpm_jpeg_par.cuh); files decoded on
// the host from coef[b][0].  Frame of file f at frames + f.frame.
__global__ void __launch_bounds__(128)
fpm_ingest_jpeg_idct_kernel(const JpFile* __restrict__ files, const int16_t* __restrict__ coef, const int* __restrict__ dcval,
                            const int* __restrict__ dc_tile_off, uint8_t* __restrict__ frames, int dpitch)
{
    const JpFile& f = files[blockIdx.y];
    const JpScan& sc = f.sc;
    const int bw = sc.bw, bh = sc.mcuy * sc.luma_v, w = f.width, h = f.height;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= bw * bh) return;
    const uint16_t* q = f.quant;
    uint8_t* dst = frames + f.frame;
    coef += f.coef;
    const int by = b / bw, bx = b - by * bw;
    const uint4* c4 = reinterpret_cast<const uint4*>(coef + (size_t)b * 64);
    int ws[8][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {                                       // row r of the block: 8 coefficients = one 16-byte load
        const uint4 v = __ldg(c4 + r);
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            ws[r][2 * k] = (int)(int16_t)(u[k] & 0xffffu) * (int)q[8 * r + 2 * k];
            ws[r][2 * k + 1] = (int)(int16_t)(u[k] >> 16) * (int)q[8 * r + 2 * k + 1];
        }
    }
    if (f.device_huffman) {
        dcval += f.luma0;
        dc_tile_off += f.luma0 / JP_DC_TILE;
        const unsigned L = jp_luma_scan_index(sc, by, bx);
        int dc = dcval[L] + dc_tile_off[L / JP_DC_TILE];
        if (sc.restart_blocks) {                                        // the DC prediction restarts with every interval
            const unsigned seg = sc.restart_blocks / sc.nslots * sc.luma_slots, s0 = L / seg * seg;
            if (s0) dc -= dcval[s0 - 1] + dc_tile_off[(s0 - 1) / JP_DC_TILE];
        }
        ws[0][0] = (int)(int16_t)dc * (int)q[0];
    }
#pragma unroll
    for (int c = 0; c < 8; c++) {                                       // pass 1: columns, results scaled up by 4
        int in[8], out[8];
#pragma unroll
        for (int r = 0; r < 8; r++) in[r] = ws[r][c];
        fpm_idct_islow_1d(in, out, 13 - 2);
#pragma unroll
        for (int r = 0; r < 8; r++) ws[r][c] = out[r];
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {                                       // pass 2: rows, descale, range limit
        int out[8];
        fpm_idct_islow_1d(ws[r], out, 13 + 2 + 3);
        const int y = 8 * by + r;
        if (y >= h) continue;
        uint32_t px[2] = {0, 0};
#pragma unroll
        for (int c = 0; c < 8; c++) {
            int v = out[c] & 1023;                                      // libjpeg's range_limit table: 10-bit wrap,
            v = v >= 512 ? v - 1024 : v;                                // signed, centre 128, clamp
            v = min(255, max(0, v + 128));
            px[c >> 2] |= (uint32_t)v << (8 * (c & 3));
        }
        uint8_t* o = dst + (size_t)y * dpitch + 8 * bx;
        if (8 * bx + 8 <= w) {
            *reinterpret_cast<uint2*>(o) = make_uint2(px[0], px[1]);    // dpitch is a multiple of 128
        } else {
            for (int c = 0; c < 8 && 8 * bx + c < w; c++) o[c] = (uint8_t)(px[c >> 2] >> (8 * (c & 3)));
        }
    }
}

// top <= stop layer: the top-layer picks are final (src/TemplateMatcher.cpp:272-276)
__global__ void fpm_cands_to_refined_kernel(const FpmCand* __restrict__ cands, int n, int top,
                                            FpmRefined* __restrict__ refined, int* __restrict__ refined_count)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const FpmCand c = cands[i];
    FpmRefined o;
    float k = (top == 0) ? 1.0f : 2.0f;
    o.angle = c.angle; o.score = c.score;
    o.ptx = (double)(c.ptx * k); o.pty = (double)(c.pty * k);
    o.img = c.img; o.id = c.id; o.scale = c.scale;
    refined[i] = o;
    if (i == 0) *refined_count = n;
}

// =====================================================================================
// K9  final stage per image: filterWithScore (:984-1000), corner construction + RotatedRect
// (:380-390), filterWithRotatedRect (:1133-1194), result conversion (:407-432).
// =====================================================================================
struct FpmResultDev {
    double score, angle, cx, cy, ltx, lty, rtx, rty, rbx, rby, lbx, lby;
    double scale;           // match scale of the target (fpm_match_scaled)
};

// wd, hd: the rectangle's size, the template's times the match scale (exact integers at scale 1), narrowed to float here like
// the reference's float corner math
__device__ __forceinline__ void fpm_corners(double ptx, double pty, double angle, double wd, double hd, float* lt,
                                            float* rt, float* lb, float* rb)
{
    double dRAngle = -angle * FPM_D2R;
    float c = (float)cos(dRAngle), s = (float)sin(dRAngle);
    const float w = (float)wd, h = (float)hd;
    lt[0] = (float)ptx; lt[1] = (float)pty;
    rt[0] = lt[0] + w * c; rt[1] = lt[1] - w * s;
    lb[0] = lt[0] + h * s; lb[1] = lt[1] + h * c;
    rb[0] = rt[0] + h * s; rb[1] = rt[1] + h * c;
}

#define FN_THREADS 256
#define FN_PAIR_MAX 512      // survivors per frame handled by the all-pairs bit matrix
#define FN_KEYS_SMEM 1024    // sort keys per frame kept in shared memory

// two rotated rects whose centres are farther apart than the sum of their half diagonals (plus a margin that
// dwarfs float rounding) cannot touch: rotatedRectangleIntersection would return INTERSECT_NONE -> keep both
__device__ __forceinline__ bool fpm_rrect_far(const FpmRRect& a, const FpmRRect& b)
{
    const float dx = a.cx - b.cx, dy = a.cy - b.cy;
    const float ra = 0.5f * sqrtf(a.w * a.w + a.h * a.h), rb = 0.5f * sqrtf(b.w * b.w + b.h * b.h);
    const float lim = (ra + rb) * 1.001f + 1.0f;
    return dx * dx + dy * dy > lim * lim;
}

// Refined records of a call.  Contiguous: recs[0 .. *count).  Segmented (angle-sharded mode): the allgathered buffer of
// one block per rank, consumed in place; recs points at the group's segment { FpmRefined[seg_cap]; int count; int pad } in
// rank block 0, and rank r's segment is seg_stride bytes further per rank.
struct FpmRefinedView {
    const FpmRefined* recs;
    const int* count;
    int seg_cap;                // 0 = contiguous
    int nseg;
    size_t seg_stride;          // bytes per rank block
};
__device__ __forceinline__ int fpm_refined_slots(const FpmRefinedView& v) { return v.seg_cap ? v.seg_cap * v.nseg : *v.count; }
__device__ __forceinline__ const FpmRefined& fpm_refined_at(const FpmRefinedView& v, int i)
{
    if (v.seg_cap == 0) return v.recs[i];
    const int r = i / v.seg_cap, k = i - r * v.seg_cap;
    return reinterpret_cast<const FpmRefined*>(reinterpret_cast<const char*>(v.recs) + (size_t)r * v.seg_stride)[k];
}
__device__ __forceinline__ bool fpm_refined_valid(const FpmRefinedView& v, int i)
{
    if (v.seg_cap == 0) return true;
    const int r = i / v.seg_cap, k = i - r * v.seg_cap;
    const char* blk = reinterpret_cast<const char*>(v.recs) + (size_t)r * v.seg_stride;
    return k < *reinterpret_cast<const int*>(blk + (size_t)v.seg_cap * sizeof(FpmRefined));
}

struct FpmNoGroup { __device__ __forceinline__ int operator()(int) const { return -1; } };

// Greedy rotated-rectangle NMS of one CTA over rects[0, m), sorted by score descending: entry k is dropped when an earlier
// kept entry i gives fpm_rrect_overlap_decision(rects[i], rects[k], max_overlap) (the ratio over the kept rectangle's area);
// entries of one group (group(i) >= 0, the same for both) are never decided against each other.  bits (m <= FN_PAIR_MAX): the kept entries are left as bit words,
// s_kept[w] with s_base[w] survivors before word w and s_base[FN_PAIR_MAX / 32] survivors in all; otherwise del[k] = 1 marks
// the dropped entries (del[0, m) zero on entry).  Ends with the CTA synchronised.
template <class Group>
__device__ __forceinline__ void fpm_greedy_nms(const FpmRRect* __restrict__ rects, int* __restrict__ del, int m, bool bits,
                                               double max_overlap, Group group, unsigned* s_bits, unsigned* s_kept, int* s_base)
{
    const int tid = threadIdx.x;
    // Small sets: all pair decisions are evaluated in parallel first (the geometry is the expensive,
    // latency-bound part), then the greedy pass only reads the byte matrix.
    if (bits) {
        // Pair decisions as bit rows in shared memory (row i, bit k = "k must go if i stays"): a warp per row, one
        // ballot per 32 columns.  The greedy pass is then a chain of register / shared-memory operations in ONE warp
        // (lane l keeps the deletion bits of survivors 32 l .. 32 l + 31) instead of a chain of global-memory round trips.
        const int nw = (m + 31) >> 5;
        const int lane = tid & 31;
        for (int i = tid >> 5; i < m; i += FN_THREADS / 32) {
            const FpmRRect ri = rects[i];
            const int gi = group(i);
            for (int j = 0; j < nw; j++) {
                bool hit = false;
                const int k = 32 * j + lane;
                if (k > i && k < m) {
                    const FpmRRect rk = rects[k];
                    hit = !(gi >= 0 && group(k) == gi) && !fpm_rrect_far(ri, rk) && fpm_rrect_overlap_decision(ri, rk, max_overlap, nullptr, nullptr);
                }
                const unsigned w = __ballot_sync(0xffffffffu, hit);
                if (lane == 0) s_bits[i * (FN_PAIR_MAX / 32) + j] = w;
            }
        }
        __syncthreads();
        if (tid < 32) {
            unsigned dw = 0;
            for (int i = 0; i < m - 1; i++) {
                const unsigned wi = __shfl_sync(0xffffffffu, dw, i >> 5);
                if (!((wi >> (i & 31)) & 1u) && lane < nw) dw |= s_bits[i * (FN_PAIR_MAX / 32) + lane];
            }
            // survivors and their ranks straight from the bit words: exclusive prefix of the per-word counts
            const int left = m - 32 * lane;
            const unsigned valid = lane < nw ? (left >= 32 ? 0xffffffffu : ((1u << left) - 1u)) : 0u;
            const unsigned kept = ~dw & valid;
            int incl = __popc(kept);
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane < FN_PAIR_MAX / 32) { s_kept[lane] = kept; s_base[lane] = incl - __popc(kept); }
            if (lane == 31) s_base[FN_PAIR_MAX / 32] = incl;          // total survivors
        }
        __syncthreads();
    } else {
        for (int i = 0; i < m - 1; i++) {
            if (!del[i]) {
                const FpmRRect ri = rects[i];
                const int gi = group(i);
                for (int k = i + 1 + tid; k < m; k += FN_THREADS)
                    if (!del[k] && !(gi >= 0 && group(k) == gi) && !fpm_rrect_far(ri, rects[k]) &&
                        fpm_rrect_overlap_decision(ri, rects[k], max_overlap, nullptr, nullptr))
                        del[k] = 1;
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(FN_THREADS)
fpm_final_kernel(FpmRefinedView rv,
                 double score_thresh, double max_overlap, double nms_w, double nms_h, double tpl_w, double tpl_h,
                 unsigned long long* __restrict__ key_scratch, int key_stride,
                 FpmRRect* __restrict__ rect_scratch, int* __restrict__ del_scratch,
                 int* __restrict__ idmap_scratch, unsigned char* __restrict__ pair_scratch, int pair_cap,
                 int mfc_compat, int max_pos, FpmResultDev* __restrict__ results, int result_cap, int* __restrict__ result_count,
                 const int* __restrict__ row_members, int n_tpl, int n_set)
{
    const int img = blockIdx.x, tid = threadIdx.x;
    // output row of the image: itself, or (row_members: a group of a template set) frame img / n_tpl x set index
    const int row = row_members ? (img / n_tpl) * n_set + row_members[img % n_tpl] : img;
    const int n_total = fpm_refined_slots(rv);
    // sort keys in shared memory when the per-frame capacity allows (a bitonic sort in global memory pays one L2 round
    // trip per stage)
    __shared__ unsigned long long s_keys[FN_KEYS_SMEM];
    unsigned long long* keys = key_stride <= FN_KEYS_SMEM ? s_keys : key_scratch + (size_t)img * key_stride;
    FpmRRect* rects = rect_scratch + (size_t)img * key_stride;
    int* del = del_scratch + (size_t)img * key_stride;
    int* idmap = idmap_scratch + (size_t)img * key_stride;
    __shared__ int s_n, s_cut;
    __shared__ unsigned s_bits[FN_PAIR_MAX * (FN_PAIR_MAX / 32)];     // 32 KB: pair-decision bit rows of the NMS
    __shared__ unsigned s_kept[FN_PAIR_MAX / 32];
    __shared__ int s_base[FN_PAIR_MAX / 32 + 1];
    if (tid == 0) s_n = 0;
    __syncthreads();
    for (int i = tid; i < n_total; i += FN_THREADS)
        if (fpm_refined_valid(rv, i) && fpm_refined_at(rv, i).img == img) {
            // ties: lower candidate id first (the oracle's stable sort order); id is unique per image
            const FpmRefined& ri = fpm_refined_at(rv, i);
            int slot = atomicAdd(&s_n, 1);
            keys[slot] = ((unsigned long long)fpm_desc_key((float)ri.score) << 32) | (unsigned long long)(uint32_t)ri.id;
            idmap[ri.id] = i;
        }
    __syncthreads();
    const int n = s_n;
    int n_pad = 1;
    while (n_pad < n) n_pad <<= 1;
    for (int i = n + tid; i < n_pad; i += FN_THREADS) keys[i] = ~0ull;
    if (tid == 0) s_cut = n;
    __syncthreads();
    fpm_bitonic_sort(keys, n_pad, tid, FN_THREADS);
    // replace the id by the record index; filterWithScore: cut at the first score < Score
    for (int i = tid; i < n; i += FN_THREADS) {
        int idx = idmap[(uint32_t)(keys[i] & 0xffffffffu)];
        keys[i] = (keys[i] & 0xffffffff00000000ull) | (unsigned long long)(uint32_t)idx;
        if (fpm_refined_at(rv, idx).score < score_thresh) atomicMin(&s_cut, i);
    }
    __syncthreads();
    const int m = s_cut;
    for (int i = tid; i < m; i += FN_THREADS) {
        const FpmRefined& r = fpm_refined_at(rv, (int)(uint32_t)(keys[i] & 0xffffffffu));
        float lt[2], rt[2], lb[2], rb[2];
        fpm_corners(r.ptx, r.pty, r.angle, nms_w * r.scale, nms_h * r.scale, lt, rt, lb, rb);   // the scaled rectangle
        rects[i] = fpm_rrect_from3(lt[0], lt[1], rt[0], rt[1], rb[0], rb[1]);
        del[i] = 0;
    }
    __syncthreads();
    // filterWithRotatedRect: scores are sorted descending so the later index always loses.
    const bool bit_path = m <= pair_cap && m <= FN_PAIR_MAX;
    fpm_greedy_nms(rects, del, m, bit_path, max_overlap, FpmNoGroup(), s_bits, s_kept, s_base);
    // survivor ranks (from the bit words, or by one thread on the large-set path: idmap is free again and holds
    // the rank of record i, or -1), conversion by all threads
    if (!bit_path) {
        if (tid == 0) {
            int cnt = 0;
            for (int i = 0; i < m; i++) {
                const bool keep = !del[i] && !(mfc_compat && cnt >= max_pos);     // MatchToolDlg.cpp:1115-1116
                idmap[i] = keep ? cnt : -1;
                if (keep) cnt++;
            }
            result_count[row] = cnt;
        }
        __syncthreads();
    } else if (tid == 0) {
        const int total = s_base[FN_PAIR_MAX / 32];
        result_count[row] = (mfc_compat && total > max_pos) ? max_pos : total;
    }
    for (int i = tid; i < m; i += FN_THREADS) {
        int rank;
        if (bit_path) {
            const unsigned kw = s_kept[i >> 5];
            rank = ((kw >> (i & 31)) & 1u) ? s_base[i >> 5] + __popc(kw & ((1u << (i & 31)) - 1u)) : -1;
            if (mfc_compat && rank >= max_pos) rank = -1;                         // MatchToolDlg.cpp:1115-1116
        } else {
            rank = idmap[i];
        }
        if (rank < 0 || rank >= result_cap) continue;
        const FpmRefined& r = fpm_refined_at(rv, (int)(uint32_t)(keys[i] & 0xffffffffu));
        FpmResultDev o;
        o.score = r.score;
        o.scale = r.scale;
        const double tw = tpl_w * r.scale, th = tpl_h * r.scale;
        if (!mfc_compat) {
            // Qt TemplateMatcher conversion (src/TemplateMatcher.cpp:407-432): float corner math
            float lt[2], rt[2], lb[2], rb[2];
            fpm_corners(r.ptx, r.pty, r.angle, tw, th, lt, rt, lb, rb);
            o.angle = r.angle;
            o.cx = (double)((lt[0] + rt[0] + lb[0] + rb[0]) / 4.0f);
            o.cy = (double)((lt[1] + rt[1] + lb[1] + rb[1]) / 4.0f);
            o.ltx = lt[0]; o.lty = lt[1]; o.rtx = rt[0]; o.rty = rt[1];
            o.rbx = rb[0]; o.rby = rb[1]; o.lbx = lb[0]; o.lby = lb[1];
        } else {
            // MFC CMatchToolDlg conversion (MatchTool/MatchToolDlg.cpp:1085-1099): double corner math,
            // angle negated and wrapped to [-180, 180]
            const double a = -r.angle * FPM_D2R, c = cos(a), sn = sin(a);
            o.ltx = r.ptx; o.lty = r.pty;
            o.rtx = o.ltx + tw * c; o.rty = o.lty - tw * sn;
            o.lbx = o.ltx + th * sn; o.lby = o.lty + th * c;
            o.rbx = o.rtx + th * sn; o.rby = o.rty + th * c;
            o.cx = (o.ltx + o.rtx + o.rbx + o.lbx) / 4;
            o.cy = (o.lty + o.rty + o.rby + o.lby) / 4;
            double ang = -r.angle;
            if (ang < -180) ang += 360;
            if (ang > 180) ang -= 360;
            o.angle = ang;
        }
        results[(size_t)row * result_cap + rank] = o;
    }
}

// =====================================================================================
// K10  template sets, merged results: one CTA per frame b merges the frame's n_set per-template lists (template t: the
// first min(counts[b*n_set + t], lcap) records of lists + (b*n_set + t)*lcap) into one list.  Order: score descending,
// ties to the lower template, then the lower position (the sort key's low word t*lcap + i).  Greedy NMS across
// templates only (pairs of one template were decided by its own NMS): rectangles from three corners of the records.
// The kept records go to out[b*out_cap + k] unchanged, their set index to out_labels, their number to out_count[b].
// =====================================================================================
struct FpmLabelOf {
    const int* lab;
    __device__ __forceinline__ int operator()(int i) const { return lab[i]; }
};

// one frame of fpm_set_merge_kernel, m entries; inlined once with keys in shared and once in global memory, so that every
// key access has a known address space
__device__ __forceinline__ void fpm_set_merge_frame(unsigned long long* __restrict__ keys, int m, const FpmResultDev* __restrict__ fl,
                                                    const int* __restrict__ fc, int n_set, int lcap, double max_overlap,
                                                    FpmRRect* __restrict__ rects, int* __restrict__ del, int* __restrict__ lab,
                                                    unsigned* s_bits, unsigned* s_kept, int* s_base, FpmResultDev* __restrict__ out,
                                                    int* __restrict__ out_labels, int out_cap, int* __restrict__ out_count)
{
    const int tid = threadIdx.x;
    int n_pad = 1;
    while (n_pad < m) n_pad <<= 1;
    for (int t = 0, off = 0; t < n_set; t++) {
        const int take = min(fc[t], lcap);
        for (int i = tid; i < take; i += FN_THREADS) {
            const uint32_t e = (uint32_t)(t * lcap + i);
            keys[off + i] = ((unsigned long long)fpm_desc_key((float)fl[e].score) << 32) | e;
        }
        off += take;
    }
    for (int i = m + tid; i < n_pad; i += FN_THREADS) keys[i] = ~0ull;
    __syncthreads();
    fpm_bitonic_sort(keys, n_pad, tid, FN_THREADS);
    for (int i = tid; i < m; i += FN_THREADS) {
        const uint32_t e = (uint32_t)keys[i];
        const FpmResultDev& r = fl[e];
        rects[i] = fpm_rrect_from3((float)r.ltx, (float)r.lty, (float)r.rtx, (float)r.rty, (float)r.rbx, (float)r.rby);
        lab[i] = (int)(e / (uint32_t)lcap);
        del[i] = 0;
    }
    __syncthreads();
    const bool bits = m <= FN_PAIR_MAX;
    fpm_greedy_nms(rects, del, m, bits, max_overlap, FpmLabelOf{lab}, s_bits, s_kept, s_base);
    if (!bits) {
        if (tid == 0) {                                         // del[i] becomes the rank of entry i, or -1
            int cnt = 0;
            for (int i = 0; i < m; i++) del[i] = del[i] ? -1 : cnt++;
            *out_count = cnt;
        }
        __syncthreads();
    } else if (tid == 0) {
        *out_count = s_base[FN_PAIR_MAX / 32];
    }
    for (int i = tid; i < m; i += FN_THREADS) {
        int rank;
        if (bits) {
            const unsigned kw = s_kept[i >> 5];
            rank = ((kw >> (i & 31)) & 1u) ? s_base[i >> 5] + __popc(kw & ((1u << (i & 31)) - 1u)) : -1;
        } else {
            rank = del[i];
        }
        if (rank < 0 || rank >= out_cap) continue;
        out[rank] = fl[(uint32_t)keys[i]];
        out_labels[rank] = lab[i];
    }
}

__global__ void __launch_bounds__(FN_THREADS)
fpm_set_merge_kernel(const FpmResultDev* __restrict__ lists, const int* __restrict__ counts, int n_set, int lcap, double max_overlap,
                     unsigned long long* __restrict__ key_scratch, int key_stride, FpmRRect* __restrict__ rect_scratch,
                     int* __restrict__ del_scratch, int* __restrict__ lab_scratch,
                     FpmResultDev* __restrict__ out, int* __restrict__ out_labels, int out_cap, int* __restrict__ out_count)
{
    const int b = blockIdx.x;
    __shared__ unsigned long long s_keys[FN_KEYS_SMEM];
    __shared__ unsigned s_bits[FN_PAIR_MAX * (FN_PAIR_MAX / 32)];
    __shared__ unsigned s_kept[FN_PAIR_MAX / 32];
    __shared__ int s_base[FN_PAIR_MAX / 32 + 1];
    const FpmResultDev* fl = lists + (size_t)b * n_set * lcap;
    const int* fc = counts + (size_t)b * n_set;
    int m = 0;
    for (int t = 0; t < n_set; t++) m += min(fc[t], lcap);
    FpmRRect* rects = rect_scratch + (size_t)b * key_stride;
    int* del = del_scratch + (size_t)b * key_stride;
    int* lab = lab_scratch + (size_t)b * key_stride;
    if (m <= FN_KEYS_SMEM)
        fpm_set_merge_frame(s_keys, m, fl, fc, n_set, lcap, max_overlap, rects, del, lab, s_bits, s_kept, s_base,
                            out + (size_t)b * out_cap, out_labels + (size_t)b * out_cap, out_cap, out_count + b);
    else
        fpm_set_merge_frame(key_scratch + (size_t)b * key_stride, m, fl, fc, n_set, lcap, max_overlap, rects, del, lab, s_bits,
                            s_kept, s_base, out + (size_t)b * out_cap, out_labels + (size_t)b * out_cap, out_cap, out_count + b);
}
