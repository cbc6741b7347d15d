// fpm_common.cuh -- shared device/host records for the B200 NCC matcher.
//
// Domain vocabulary follows the reference (/root/reference/include/DataStructures.h):
//   template pyramid level, candidate (s_MatchParameter), target (s_SingleTargetMatch).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#define FPM_VISION_TOLERANCE 0.0000001              // DataStructures.h:10
#define FPM_PI 3.1415926535897932384626433832795    // CV_PI
#define FPM_D2R (FPM_PI / 180.0)                    // DataStructures.h:11
#define FPM_R2D (180.0 / FPM_PI)                    // DataStructures.h:12
#define FPM_MATCH_CANDIDATE_NUM 5                   // DataStructures.h:13
#define FPM_MAX_LEVELS 16
#define FPM_ROI_PAD 6                               // getRotatedROI: size + 6 (TemplateMatcher.cpp:1079)
#define FPM_NSHIFT 7                                // 7x7 score patch per refinement eval
#define FPM_NCELL 49
#define FPM_WSTRIDE 8                               // ints per (eval, ROI row) record of the window row sums rowS / rowQ: the 7 shifts + 1 pad
                                                    // = one aligned 32-byte sector, written and read with two 128-bit accesses

#define FPM_HD __host__ __device__ __forceinline__

// One pyramid level of a batch of images: [batch][h][pitch] u8
struct FpmLevel {
    uint8_t* ptr;
    int w, h, pitch;
    size_t img_stride;
};

// Per-level template statistics (s_TemplData, DataStructures.h:16-55)
struct FpmTplStat {
    double mean, norm, inv_area;
    int result_equal1;
};

// One level of a template group: n_tpl templates of one size, template k at ptr + k * tpl_stride with statistics
// stats[k].  The inline statistics are template 0's.  Virtual image v of a group = frame v / n_tpl x template v % n_tpl.
struct FpmTplLevel {
    const uint8_t* ptr;     // [h][pitch] u8, rows zero padded to pitch (pitch % 16 == 0)
    int w, h, pitch;
    double mean, norm, inv_area;
    int result_equal1;
    int n_tpl;              // templates in the group (1: a single template, stats unused)
    size_t tpl_stride;
    const FpmTplStat* stats;
    // masked template or group: the kept pixels of row y of template k are the column ranges [b, e) of
    // mrun[mrow[k * (h + 1) + y] .. mrow[k * (h + 1) + y + 1]) (fpm_tpl_member moves mrow to template k's h + 1 offsets);
    // the pixels at ptr are already multiplied by the mask.  null: every pixel is kept.
    const int* mrow;
    const int2* mrun;
};

// template k of a group level
FPM_HD FpmTplLevel fpm_tpl_member(FpmTplLevel t, int k)
{
    if (t.n_tpl > 1) {
        t.ptr += (size_t)k * t.tpl_stride;
        const FpmTplStat s = t.stats[k];
        t.mean = s.mean; t.norm = s.norm; t.inv_area = s.inv_area; t.result_equal1 = s.result_equal1;
        if (t.mrow) t.mrow += (size_t)k * (t.h + 1);
    }
    return t;
}

// One warpAffine job (dst <- src), matrix already inverted the way cv::warpAffine does it.
struct FpmWarpJob {
    double m[6];            // dst->src: x_s = m0*x + m1*y + m2 ; y_s = m3*x + m4*y + m5
    int src_img;            // image index in the batch
    int dw, dh;             // output size
    int valid;
};

// Candidate carried through the refinement (s_MatchParameter, DataStructures.h:58-94)
struct FpmCand {
    double angle;           // dMatchAngle
    double score;           // dMatchScore
    float ptx, pty;         // top layer: pt ; refinement: ptLT (cv::Point2f)
    int img;                // image index in the batch (virtual image of a template group)
    int id;                 // rank in the score-sorted top-layer list of its image
    double scale;           // match scale s: the source is resampled by 1/s (FPM_PARAM_SCALE_MIN / MAX; 1 = unscaled)
};

// Refined target before NMS
struct FpmRefined {
    double angle, score;
    double ptx, pty;        // cv::Point2d pt
    int img, id;
    double scale;           // match scale of the record (FpmCand::scale)
};

// per-eval record written by refine_finalize for tracing (parity ladder T6)
struct FpmEvalTrace {
    double angle;
    float score;
    int locx, locy;
};

// ---- cp.async (LDGSTS) helpers: global -> shared copies that bypass registers, so a thread can
// keep many copies in flight (deep memory-level parallelism for the staging loops) ----
__device__ __forceinline__ void fpm_cp_async4(void* smem, const void* gmem, bool valid)
{
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    int sz = valid ? 4 : 0;                                   // src-size 0 -> zero fill, no global read
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(sa), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void fpm_cp_async16(void* smem, const void* gmem)
{
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void fpm_cp_async16z(void* smem, const void* gmem, bool valid)
{
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    int sz = valid ? 16 : 0;                                  // src-size 0 -> 16 zero bytes
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sa), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void fpm_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void fpm_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Round-half-to-even of a double, like cvRound / saturate_cast<int>(double) (lrint).
__device__ __forceinline__ int fpm_cvround(double v) { return __double2int_rn(v); }

FPM_HD int fpm_reflect101(int i, int n)
{
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
    return i;
}

// ptRotatePt2f, src/TemplateMatcher.cpp:971-982 (double math, float result)
FPM_HD void fpm_pt_rotate(float px, float py, float ox, float oy, double ang, float* rx, float* ry)
{
    double dHeight = (double)(oy * 2);
    double dY1 = dHeight - (double)py, dY2 = dHeight - (double)oy;
    double c = cos(ang), s = sin(ang);
    double dX = ((double)px - (double)ox) * c - (dY1 - (double)oy) * s + (double)ox;
    double dY = ((double)px - (double)ox) * s + (dY1 - (double)oy) * c + dY2;
    dY = -dY + dHeight;
    *rx = (float)dX;
    *ry = (float)dY;
}

// Scale-tolerant matching: p -> c + k * (p - c), evaluated in double and stored as float.  k = s maps a point of a source
// resampled by 1/s back to the source, k = 1/s maps a source point into the resampled source.  Callers skip it at s == 1,
// which keeps the unscaled float path bit for bit.
FPM_HD void fpm_scale_about(float px, float py, float cx, float cy, double k, float* rx, float* ry)
{
    *rx = (float)((double)cx + k * ((double)px - (double)cx));
    *ry = (float)((double)cy + k * ((double)py - (double)cy));
}

// cv::getRotationMatrix2D(center, angle, scale) followed by the inversion cv::warpAffine applies
// when WARP_INVERSE_MAP is not set (OpenCV imgproc imgwarp.cpp; model pinned in SURVEY 8c).
// alpha = cos * scale, beta = sin * scale as OpenCV computes them, so scale 1 gives the unscaled matrix bit for bit.
FPM_HD void fpm_rotation_matrix(float cx, float cy, double angle_deg, double* m, double scale = 1.0)
{
    double a = angle_deg * (FPM_PI / 180);
    double alpha = cos(a) * scale, beta = sin(a) * scale;
    m[0] = alpha; m[1] = beta;  m[2] = (1 - alpha) * (double)cx - beta * (double)cy;
    m[3] = -beta; m[4] = alpha; m[5] = beta * (double)cx + (1 - alpha) * (double)cy;
}

FPM_HD void fpm_invert_affine(double* M)
{
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11; M[1] *= -D;
    M[3] *= -D; M[4] = A22;
    double b1 = -M[0] * M[2] - M[1] * M[5];
    double b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1; M[5] = b2;
}
