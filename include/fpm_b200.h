/* fpm_b200.h -- C ABI of the B200-native NCC template matcher (libfpm_b200.so).
 *
 * Drop-in boundary for the reference's `TemplateMatcher` class
 * (/root/reference/include/TemplateMatcher.h:9-52): every public method of that class has
 * one entry point here (plain pointers and sizes, no C++/torch/OpenCV types), so a binding for
 * the Qt app (include/fpm_template_matcher.hpp), pybind11 or ctypes is a thin wrapper.
 *
 * All functions return 0 on success and a negative FPM_ERR_* code on failure; they never
 * throw.  "No match" is n == 0, not an error (the reference returns an empty vector,
 * src/TemplateMatcher.cpp:99-114, :398-399).  A handle owns one CUDA device, one stream and all
 * device memory; it is not thread-safe, distinct handles are independent.
 */
#ifndef FPM_B200_H
#define FPM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fpm_handle fpm_handle;

/* POD mirror of s_SingleTargetMatch (/root/reference/include/DataStructures.h:97-115). */
typedef struct fpm_result {
    double score;            /* dMatchScore   */
    double angle;            /* dMatchedAngle (degrees, Qt sign convention) */
    double cx, cy;           /* ptCenter      */
    double ltx, lty;         /* ptLT          */
    double rtx, rty;         /* ptRT          */
    double rbx, rby;         /* ptRB          */
    double lbx, lby;         /* ptLB          */
} fpm_result;

/* Parameters = the setters of TemplateMatcher (include/TemplateMatcher.h:22-28). */
enum fpm_param {
    FPM_PARAM_MAX_POSITIONS = 0,   /* setMaxPositions  (TargetNum), default 70   */
    FPM_PARAM_MAX_OVERLAP = 1,     /* setMaxOverlap,               default 0.0  */
    FPM_PARAM_SCORE = 2,           /* setScore,                    default 0.7  */
    FPM_PARAM_TOLERANCE_ANGLE = 3, /* setToleranceAngle,           default 0.0  */
    FPM_PARAM_MIN_REDUCE_AREA = 4, /* setMinReduceArea,            default 256  */
    FPM_PARAM_USE_SIMD = 5,        /* setUseSIMD,                  default 1    */
    FPM_PARAM_SUBPIXEL = 6,        /* setSubPixelEstimation,       default 0    */
    FPM_PARAM_TRACE = 7,           /* keep per-stage records for fpm_trace_*   (tests) */
    FPM_PARAM_WORKSPACE_MB = 8,    /* refinement workspace budget per wave, default 4096 */
    FPM_PARAM_PROFILE = 9,         /* bracket every kernel launch with CUDA events (bench.py roofline) */
    FPM_PARAM_H2D_CHUNK = 10,      /* frames per host->device chunk in fpm_match_batch (0 = auto)      */
    FPM_PARAM_TENSOR_CORES = 11,   /* correlation: 0 = dp4a only, 1 = tcgen05 for template width >= 64, and for width >= 16 when a level has
                                      enough evals for the fused kernel (default), 2 = always,
                                      3 = like 1 but never the fused kernel (row dots to HBM, separate row sums), 4 = always fused,
                                      5 = same as 1 (kept for A/B runs), 6 = like 1 with fpm_corr_warp_kernel on the large levels:
                                      the rotated ROI rows are computed inside the tcgen05 producer and never reach HBM (bit-identical,
                                      1.45 GB/step less DRAM traffic on cfg1, but slower than warp + MMA today: DESIGN.md section 3) */
    FPM_PARAM_MFC_COMPAT = 12,     /* 1: upstream MFC conventions: result (MatchTool/MatchToolDlg.cpp:1085-1116: angle = -theta wrapped
                                      to [-180,180], results truncated to TargetNum, corners in double) and s_BlockMax
                                      (MatchToolDlg.h:109-213: 2x template blocks, last maximal block wins); default 0 = Qt port */
    /* MFC-only modes of the upstream dialog, off by default (the Qt TemplateMatcher has none of them) */
    FPM_PARAM_STOP_LAYER1 = 13,    /* m_bStopLayer1 (MatchToolDlg.cpp:936): stop the descent at layer 1, coordinates x2 */
    FPM_PARAM_BITWISE_NOT = 14,    /* m_ckBitwiseNot (:788-794): match on 255 - source                                */
    FPM_PARAM_TOLERANCE_RANGE = 15,/* m_bToleranceRange (:805-816): sweep [TOLERANCE1,TOLERANCE2] and [TOLERANCE3,TOLERANCE4] */
    FPM_PARAM_TOLERANCE1 = 16, FPM_PARAM_TOLERANCE2 = 17, FPM_PARAM_TOLERANCE3 = 18, FPM_PARAM_TOLERANCE4 = 19,
    FPM_PARAM_SPLIT_BATCH = 20,    /* fpm_match_batch_device: batches of at least this many frames run as two concurrent
                                      half-batches on two internal handles (default 8, 0 = never) */
    FPM_PARAM_SHARD_UPLOAD = 21,   /* fpm_match_sharded with a HOST frame: 1 (default) = every rank uploads 1/N of the rows over its own
                                      PCIe link and the slices are allgathered over NVLink; 0 = every rank uploads the whole frame */
    FPM_PARAM_ASYNC_DESCENT = 22,  /* pyramid descent without a host round trip per layer (grids sized to the top-layer candidate count, live
                                      counts read on the device): -1 = automatic (batches of fewer than 8 frames), 0 = never, 1 = always */
    FPM_PARAM_JPEG_DEVICE_HUFFMAN = 23, /* fpm_ingest_jpeg: 1 (default) = the scan is Huffman-decoded on the device (the compressed scan is the
                                           only H2D traffic), 0 = on the host (sequential; its coefficients are uploaded) */
    FPM_PARAM_JPEG_PASSES = 24,    /* read-only: synchronisation passes of the last JPEG ingest (0 = decoded on the host); a batch iterates
                                      as one, so this is the count of its slowest file */
    FPM_PARAM_SCALE_MIN = 25,
    FPM_PARAM_SCALE_MAX = 26,      /* match scale range [SCALE_MIN, SCALE_MAX], default [1, 1]: an instance s times the template's size is
                                      found by resampling the source by 1/s around each level's centre (getRotationMatrix2D(c, angle, 1/s))
                                      with the same template pyramid.  Values outside [0.5, 2] or not finite are refused (FPM_ERR_INVALID);
                                      min > max is refused at match time (the setters run in either order).
                                      Schedule: ds = 2 / max(w, h) of the top template level; {min} when min == max (a fixed
                                      magnification), else n = ceil(log(max/min) / log1p(ds)) + 1 scales min * exp(k log(max/min) / (n-1)),
                                      the last exactly max.  Top-layer pose slot k * n_angles + a (scale-major).  Descent: scales
                                      s / (1 + ds_L), s, s * (1 + ds_L) (range) or s (fixed) x the usual angles, best = first strict
                                      maximum; sub-pixel uses the three angle evals of the best scale.  Results are the rectangles of the
                                      scaled size (w * s, h * s) in every result convention; [1, 1] is the unscaled matcher bit for bit.
                                      fpm_match_scaled reports each record's scale; for template sets fpm_match_set_scaled*,
                                      fpm_match_ingested_set_scaled* and fpm_match_set_sharded_scaled* do.  fpm_match_set_batch*
                                      and fpm_match_ingested_set_batch* on sets of more than one template, fpm_match_sharded*, the
                                      fpm_match_set_sharded* calls without _scaled and fpm_stage_* refuse any range other than [1, 1].
                                      FPM_PARAM_TENSOR_CORES = 6 takes the mode-1 route at any range other than [1, 1]. */
    FPM_PARAM_COUNT_
};

enum fpm_error {
    FPM_OK = 0,
    FPM_ERR_INVALID = -1,      /* bad argument                                   */
    FPM_ERR_CUDA = -2,         /* CUDA runtime error, see fpm_last_error         */
    FPM_ERR_NOT_LEARNED = -3,
    FPM_ERR_NO_DEVICE = -4,    /* no CUDA device: there is NO CPU fallback       */
    FPM_ERR_LIMIT = -5         /* a documented capacity limit was exceeded       */
};

/* TemplateMatcher::TemplateMatcher / ~TemplateMatcher (src/TemplateMatcher.cpp:28-43). */
fpm_handle* fpm_create(int device);
void fpm_destroy(fpm_handle* h);
const char* fpm_last_error(const fpm_handle* h);
const char* fpm_version(void);

/* setX / getX (include/TemplateMatcher.h:22-37). */
int fpm_set_param(fpm_handle* h, int param, double value);
double fpm_get_param(const fpm_handle* h, int param);

/* learnPattern (src/TemplateMatcher.cpp:45-95).  tpl: host pointer, u8, `stride` bytes per row. */
int fpm_learn(fpm_handle* h, const uint8_t* tpl, int width, int height, int stride);
/* Template sets (the upstream OCR loop, MatchTool/MatchToolDlg.cpp:718-770: one LoadDst + Match per glyph): n templates
 * (template i: tpls[i], widths[i] x heights[i], strides[i] bytes per row) replace the handle's pattern, all with the handle's
 * parameters.  FPM_ERR_INVALID (the message names the index) for n < 1, null pointers or an empty template; the handle then
 * holds none.  fpm_learn is a set of one.  Templates of one level-0 size, border colour and masked-ness (fpm_learn_set_masked)
 * form a group that shares every launch of the pipeline (the template is a kernel dimension); groups run one after another.
 * There is no NMS across templates.
 * A handle holding more than one template refuses every single-template entry point with FPM_ERR_INVALID and a message:
 * fpm_match*, fpm_match_ingested*, fpm_learn_ingested, fpm_match_multi, fpm_match_sharded*, fpm_stage_*, fpm_tpl_* (and
 * fpm_match_set_batch with FPM_PARAM_TRACE on).  fpm_match_set_sharded* run a set in the angle-sharded mode.  FPM_PARAM_MIN_REDUCE_AREA changed after learning re-learns the whole set.
 * A scale range other than [1, 1] (FPM_PARAM_SCALE_MIN / MAX) is matched on a set by the calls that return each record's scale:
 * fpm_match_set_scaled, fpm_match_ingested_set_scaled, their _merged twins and fpm_match_set_sharded_scaled*. */
int fpm_learn_set(fpm_handle* h, int n, const uint8_t* const* tpls, const int* widths, const int* heights, const int* strides);
/* fpm_learn_set with a don't-care mask per template: masks[i] (u8, template i's size, mask_strides[i] bytes per row,
 * nonzero = kept) or NULL for an unmasked member; masks == NULL is fpm_learn_set.  Each masked member is learned exactly as
 * fpm_learn_masked learns it, and every set entry point returns for it the lists of a handle holding only that template.
 * Masked and unmasked members never share a group.  FPM_ERR_INVALID (the message names the template index, and the level
 * for the last case) for mask_strides == NULL with masks, mask_strides[i] < widths[i], a mask that keeps no pixel, or one that
 * keeps none at some pyramid level; the handle then holds none.  A FPM_PARAM_MIN_REDUCE_AREA change re-learns with the masks. */
int fpm_learn_set_masked(fpm_handle* h, int n, const uint8_t* const* tpls, const int* widths, const int* heights,
                         const int* strides, const uint8_t* const* masks, const int* mask_strides);
int fpm_set_size(const fpm_handle* h);              /* 0 = nothing learned, 1 after fpm_learn */
/* Masked template (a don't-care mask, like cv::matchTemplate(..., mask) with TM_CCOEFF_NORMED): mask is u8 of the template's
 * size, `mask_stride` bytes per row, a nonzero byte keeps the pixel.  M_0 = (mask != 0); M_{L+1} = (pyrDown(255 * M_L) >= 128).
 * The template pyramid T_L is built from the whole template as fpm_learn builds it.  Every level's mean / norm / inv_area come
 * from the exact sums over the kept pixels (n_L = sum M_L, inv_area = 1 / n_L), the border colour from the kept mean of level 0.
 * At every placement the numerator is the one of the template M_L * T_L and the window sums t, t2 run over the kept pixels only;
 * rectangles, corners, NMS and sub-pixel fitting use the template rectangle.  A full mask gives bit for bit fpm_learn's results.
 * Works on every single-template entry point; fpm_learn_set_masked learns masked templates into a set.
 * FPM_PARAM_TENSOR_CORES = 6 takes the mode-1 route on a masked handle (its window sums need the ROI patches in memory).  FPM_ERR_INVALID with a message for a null mask, a mask that keeps no
 * pixel, or one that keeps none at some pyramid level (the message names it); the handle then holds no template.
 * fpm_learn, fpm_learn_set and fpm_learn_ingested learn unmasked templates; a FPM_PARAM_MIN_REDUCE_AREA change re-learns with
 * the mask. */
int fpm_learn_masked(fpm_handle* h, const uint8_t* tpl, int width, int height, int stride, const uint8_t* mask, int mask_stride);
/* batch frames (HOST memory, or device memory with src_on_device = 1; frame i at src + i*frame_stride) x the set: frame b /
 * template t at out + (b*n + t)*cap, its total in counts[b*n + t].  For every (b, t) exactly the list a handle holding only
 * template t returns for frame b through fpm_match_batch_device.  Host frames use the chunked H2D pipeline of fpm_match_batch. */
int fpm_match_set_batch(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                        size_t frame_stride, fpm_result* out, int cap, int* counts);
/* the frames left by the last ingest (fpm_ingest_jpeg_batch etc.) x the set */
int fpm_match_ingested_set_batch(fpm_handle* h, fpm_result* out, int cap, int* counts);
/* The same match with one labelled list per frame: the n lists L(b, t) fpm_match_set_batch writes for frame b with the same
 * cap (their first min(count, cap) records) merged by score descending (ties: lower set index t, then lower position in
 * L(b, t)) and greedy rotated-rectangle NMS across templates: an entry of template t is dropped when an earlier kept entry of
 * a template t' != t overlaps it by more than max_overlap of the kept rectangle's area, or contains it (the rectangles come
 * from the records' lt, rt and rb corners).  Entries of one template never suppress each other: a set of one merges to its
 * own list.  max_overlap is this call's own threshold (any finite value; FPM_PARAM_MAX_OVERLAP stays the per-template one).
 * Frame b's kept records, bit-identical to the per-template ones, go to out + b*cap and their set index to labels + b*cap
 * (the first min(counts[b], cap)); counts[b] is their total.  set_counts (NULL: not written) gets the per-template totals
 * fpm_match_set_batch reports, [b*n + t], so a caller can tell when cap cut an input list.  labels may be NULL only when
 * cap = 0.  Refusals as fpm_match_set_batch's, and FPM_ERR_INVALID for a NaN or infinite max_overlap. */
int fpm_match_set_batch_merged(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                               size_t frame_stride, double max_overlap, fpm_result* out, int* labels, int cap, int* counts,
                               int* set_counts);
/* the frames left by the last ingest x the set, merged as in fpm_match_set_batch_merged */
int fpm_match_ingested_set_batch_merged(fpm_handle* h, double max_overlap, fpm_result* out, int* labels, int cap, int* counts,
                                        int* set_counts);
/* Scale-tolerant template sets: each call is its twin above (fpm_match_set_batch, fpm_match_ingested_set_batch and the two
 * _merged calls) at any scale range (FPM_PARAM_SCALE_MIN / MAX, [1, 1] included), plus the scale of each record in scales[] at
 * the same index as in out (scales may be NULL).  For every (b, t) the records and scales are bit for bit those a handle
 * holding only template t returns through fpm_match_scaled with the same parameters and range; the merged calls merge those
 * lists as fpm_match_set_batch_merged does, so the NMS across templates compares the scaled rectangles.  Each group of the set
 * runs its own scale schedule (ds = 2 / max of its top level).  Refusals as the twin's, and min > max. */
int fpm_match_set_scaled(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                         size_t frame_stride, fpm_result* out, double* scales, int cap, int* counts);
int fpm_match_ingested_set_scaled(fpm_handle* h, fpm_result* out, double* scales, int cap, int* counts);
int fpm_match_set_scaled_merged(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                                size_t frame_stride, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                int* counts, int* set_counts);
int fpm_match_ingested_set_scaled_merged(fpm_handle* h, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                         int* counts, int* set_counts);

/* isPatternLearned / clearPattern (include/TemplateMatcher.h:43-46). */
int fpm_is_learned(const fpm_handle* h);
void fpm_clear(fpm_handle* h);

/* match (src/TemplateMatcher.cpp:97-437).  src: HOST pointer, u8.  Writes up to `cap` results sorted
 * by score descending and the total number found to *n (which may exceed cap). */
int fpm_match(fpm_handle* h, const uint8_t* src, int width, int height, int stride,
              fpm_result* out, int cap, int* n);

/* Batch of equally sized frames in HOST memory (frame i at src + i*frame_stride).  out holds
 * batch*cap records, n holds batch counts.  Host->device copies are pipelined with the matching. */
int fpm_match_batch(fpm_handle* h, const uint8_t* src, int batch, int width, int height, int stride,
                    size_t frame_stride, fpm_result* out, int cap, int* n);

/* Same, frames already resident in DEVICE memory of the handle's device. */
int fpm_match_batch_device(fpm_handle* h, const uint8_t* d_src, int batch, int width, int height,
                           int stride, size_t frame_stride, fpm_result* out, int cap, int* n);

/* Multi-template matching (SURVEY 8f rank 3; the upstream "NCC-based OCR" loop, MatchTool/MatchToolDlg.cpp:727-750:
 * one LoadDst + Match per glyph template): the same HOST image matched by n_handles learned handles of one
 * device, concurrently.  out holds n_handles*cap records (handle i at out + i*cap), counts n_handles totals.
 * Handles may differ in parameters; templates with one set of parameters are better served by fpm_learn_set. */
int fpm_match_multi(fpm_handle* const* hs, int n_handles, const uint8_t* src, int width, int height, int stride,
                    fpm_result* out, int cap, int* counts);
/* Text assembly of that loop (MatchToolDlg.cpp:752-771): centres + one label each -> lines (sorted by y, split where
 * neighbours differ by more than line_tol (upstream: 10 px), each line sorted by x), '\n' between lines.
 * Returns the text length, or FPM_ERR_LIMIT if out_cap is too small. */
int fpm_ocr_assemble(const double* cx, const double* cy, const char* labels, int n, double line_tol, char* out, int out_cap);

/* Image ingest (SURVEY 8f rank 4): decode on the device, match the device-resident frame without a pixel copy.
 * fpm_ingest_bmp: an uncompressed Windows BMP file image (8-bit palettized or 24-bit BGR, bottom-up or top-down) in a
 *   HOST buffer -> u8 grayscale frame owned by the handle, bit-identical to cv::imread(path, IMREAD_GRAYSCALE)
 *   (src/MatchToolDialog.cpp:314 source, :341 template): (B*1868 + G*9617 + R*4899 + 8192) >> 14 on pixels / palette entries.
 * fpm_ingest_rgb32: camera frame hand-off (src/MatchToolDialog.cpp:1557-1575, QImage::convertToFormat(Format_Grayscale8)):
 *   0xAARRGGBB pixels -> (R*11 + G*16 + B*5) / 32.
 * fpm_match_ingested / fpm_learn_ingested use the last ingested frame as source / template;
 * fpm_ingested_pixels copies it back (width*height bytes). */
int fpm_ingest_bmp(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height);
/* fpm_ingest_jpeg: a baseline / extended-sequential Huffman JPEG file image (8-bit, one scan, grayscale or YCbCr with any chroma
 * subsampling, restart intervals) -> the frame cv::imread(path, IMREAD_GRAYSCALE) returns, bit for bit (luma only, libjpeg's
 * ISLOW integer IDCT): Huffman decoding, dequantisation, IDCT and range limit run on the device, the compressed scan is the
 * only host-to-device traffic.  Progressive,
 * arithmetic, 12-bit, CMYK / RGB-coded and multi-scan files are rejected with FPM_ERR_INVALID and a message.
 * fpm_ingest_image: BMP or JPEG by the file's signature, like cv::imread. */
int fpm_ingest_jpeg(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height);
int fpm_ingest_image(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height);
int fpm_ingest_rgb32(fpm_handle* h, const uint32_t* pixels, int width, int height, int stride_bytes);
int fpm_ingested_pixels(fpm_handle* h, uint8_t* out);
int fpm_match_ingested(fpm_handle* h, fpm_result* out, int cap, int* n);
int fpm_learn_ingested(fpm_handle* h);
/* Batched JPEG ingest: n JPEG file images packed back to back in ONE host buffer, file i = data[offsets[i], offsets[i+1]) (offsets
 * has n+1 entries).  All files must decode to frames of one width x height.  Result: n device-resident frames [n][height][pitch]
 * owned by the handle, frame i bit-identical to cv::imread(IMREAD_GRAYSCALE) of file i (what fpm_ingest_jpeg gives for that file
 * alone).  The host reads only the marker segments in front of each scan; the bytes data[offsets[0], offsets[n]) go to the device
 * in one cudaMemcpyAsync (pinned memory: PCIe rate), where the stuffing is removed and all files are Huffman-decoded by the same
 * launches, in waves of consecutive files that fit FPM_PARAM_WORKSPACE_MB.  FPM_ERR_INVALID (the message names the file) for an
 * empty batch, null pointers, decreasing offsets, a file fpm_ingest_jpeg rejects, or a frame size that differs from file 0's;
 * FPM_ERR_LIMIT above 2^30 pixels per frame.
 * Every ingest leaves fpm_ingested_count frames (1 for the single-file calls, 0 after an error).  fpm_ingested_pixels,
 * fpm_match_ingested and fpm_learn_ingested need exactly one; fpm_ingested_frame_pixels copies frame `index` (width*height
 * bytes), fpm_match_ingested_batch matches all of them (= fpm_match_batch_device on the frames: out holds count*cap records,
 * counts holds count totals). */
int fpm_ingest_jpeg_batch(fpm_handle* h, const uint8_t* data, const size_t* offsets, int n, int* width, int* height);
int fpm_ingested_count(const fpm_handle* h);
int fpm_ingested_frame_pixels(fpm_handle* h, int index, uint8_t* out);
int fpm_match_ingested_batch(fpm_handle* h, fpm_result* out, int cap, int* counts);

/* Scale-tolerant matching (FPM_PARAM_SCALE_MIN / MAX): the records of fpm_match_batch (src_on_device = 0) /
 * fpm_match_batch_device (1) / fpm_match_ingested_batch, plus the scale of each record in scales[] at the same index as in out
 * (frame b's record i at b * cap + i): the exact schedule / descent value, 1.0 at the range [1, 1].  scales may be NULL.
 * Refused like the single-template entry points on a set of more than one template. */
int fpm_match_scaled(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                     size_t frame_stride, fpm_result* out, double* scales, int cap, int* counts);
int fpm_match_ingested_scaled(fpm_handle* h, fpm_result* out, double* scales, int cap, int* counts);

/* getLastExecutionTime (include/TemplateMatcher.h:40), milliseconds of the last match call. */
double fpm_last_time_ms(const fpm_handle* h);

/* setUserDefinedRect / getUserDefinedRect / hasUserDefinedRect (src/TemplateMatcher.cpp:1224-1238):
 * pure storage, kept for API completeness. */
void fpm_set_user_rect(fpm_handle* h, int x, int y, int w, int hgt);
int fpm_get_user_rect(const fpm_handle* h, int* x, int* y, int* w, int* hgt); /* returns hasUserRect */

/* Number of kernel launches issued by this handle since creation (bench.py's gpu_launches). */
long long fpm_launch_count(const fpm_handle* h);

/* CUDA events on the handle's stream: record(0) before / record(1) after a region, then elapsed. */
int fpm_timer_record(fpm_handle* h, int which);
double fpm_timer_elapsed_ms(fpm_handle* h);

/* Per-kernel device time (CUDA events around every launch while FPM_PARAM_PROFILE = 1), launch
 * count and algorithmic work (bytes, or MACs for the correlation kernels) accumulated since reset. */
int fpm_profile_num_kernels(void);
const char* fpm_profile_name(int kernel);
int fpm_profile_get(fpm_handle* h, int kernel, double* ms, long long* launches, double* work);
void fpm_profile_reset(fpm_handle* h);

/* ---- learned-template introspection (s_TemplData, DataStructures.h:16-55) ---- */
int fpm_tpl_levels(const fpm_handle* h);                 /* pyramid size (top layer + 1) */
int fpm_tpl_level_info(const fpm_handle* h, int level, int* w, int* hgt, double* mean, double* norm,
                       double* inv_area, int* result_equal1);
int fpm_tpl_level_pixels(const fpm_handle* h, int level, uint8_t* out /* w*h */);
/* M_L of a masked template as 0/1 bytes (out may be NULL); returns n_L, its kept count.  Unmasked: all ones, w*h. */
int fpm_tpl_level_mask(const fpm_handle* h, int level, uint8_t* out /* w*h */);
int fpm_tpl_border_color(const fpm_handle* h);

/* ---- angle-sharded (multi-GPU latency mode) stage API; records are plain doubles ----
 * top:    run the top-layer sweep for angle indices [a0, a1) of the schedule; returns raw picks
 *         as rows of 5 doubles {angle_index, x, y, score, angle_deg} in (angle, pick) order.
 * refine: descend the pyramid for the given globally sorted candidate rows
 *         {id, ptx, pty, score, angle_deg} (pt already un-rotated, src/TemplateMatcher.cpp:265-266);
 *         returns rows of 5 doubles {id, ptx, pty, score, angle_deg}.
 * final:  filterWithScore + NMS + conversion over the union of refined rows. */
int fpm_stage_num_angles(fpm_handle* h, int width, int height);
int fpm_stage_top(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                  int a0, int a1, double* rows, int cap, int* n);
int fpm_stage_sort_candidates(fpm_handle* h, const double* picks, int n, double* cands /* n*5 */);
int fpm_stage_refine(fpm_handle* h, const double* cands, int n, double* rows, int cap, int* n_out);
int fpm_stage_final(fpm_handle* h, const double* refined, int n, fpm_result* out, int cap, int* n_out);

/* ---- angle-sharded latency mode across the GPUs of one box (SURVEY 8e) ----
 * One process (or thread) per GPU, each with its own handle, same template and parameters on every rank.  The work of
 * TemplateMatcher::match shards in two places -- the top-layer angle sweep (src/TemplateMatcher.cpp:162-211) and the
 * per-candidate descent (:262-371) -- joined by two ncclAllGather calls on device buffers (pick lists, refined records)
 * that the sort / NMS kernels consume in place; the result list is identical on every rank and bit-identical to
 * fpm_match on one GPU.  NCCL is loaded at run time (dlopen libnccl.so.2): the library has no link-time dependency.
 *   fpm_comm_get_unique_id: rank 0 creates the 128-byte ncclUniqueId; the caller distributes it (MPI, torch.distributed, a file...)
 *   fpm_comm_init:          collective over all ranks: ncclCommInitRank on the handle's device
 *   fpm_comm_attach:        use an existing ncclComm_t (borrowed, not destroyed by the handle)
 *   fpm_match_sharded:      collective; src is this rank's copy of the SAME frame (host pointer, or a device pointer with
 *                           src_on_device = 1).  A host frame is uploaded as 1/N row slices + one allgather (FPM_PARAM_SHARD_UPLOAD).
 *   fpm_match_sharded_virtual: the same pipeline with nranks handles of ONE device as the ranks and device-to-device block
 *                           copies as the exchange (tests the partitioning where a single GPU is available). */
#define FPM_COMM_ID_BYTES 128
int fpm_comm_available(void);
int fpm_comm_get_unique_id(void* id /* FPM_COMM_ID_BYTES */);
int fpm_comm_init(fpm_handle* h, int nranks, int rank, const void* id /* FPM_COMM_ID_BYTES */);
int fpm_comm_attach(fpm_handle* h, void* nccl_comm /* ncclComm_t */, int nranks, int rank);
void fpm_comm_destroy(fpm_handle* h);
int fpm_match_sharded(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                      fpm_result* out, int cap, int* n);
int fpm_match_sharded_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                              fpm_result* out /* nranks*cap */, int cap, int* n /* nranks */);
/* ---- template sets in the angle-sharded latency mode: one frame against the whole set across the ranks ----
 * fpm_match_set_sharded: collective; src is this rank's copy of the SAME frame (host, or device with src_on_device = 1).
 *   Template t's list goes to out + t*cap and its total to counts[t] (n = fpm_set_size).  On every rank the lists are
 *   bit-identical to what fpm_match_set_batch returns for the frame on one GPU (batch of 1, same cap).  Every group of the set
 *   sweeps this rank's chunk of its angle schedule (fpm_shard_angle_range) for all its templates, and the call issues the
 *   collectives of a one-template call however many groups the set has: two allgathers, plus one when a host frame is uploaded
 *   in slices (FPM_PARAM_SHARD_UPLOAD).  Refuses (FPM_ERR_INVALID, with a message) what fpm_match_set_batch refuses, and more
 *   than one rank without a communicator.  A handle with nothing learned returns empty lists.
 * fpm_match_set_sharded_merged: the same, merged as fpm_match_set_batch_merged does for one frame: one labelled list at out /
 *   labels, its total in *count, the per-template totals in set_counts (NULL: not written).  Also refuses a NaN or infinite
 *   max_overlap, and NULL labels while cap > 0.
 * The _virtual calls: nranks handles of ONE device play the ranks (none may have a communicator, all hold sets of one size);
 *   the exchanges are device-to-device block copies, each round counted as one collective in fpm_collective_count of every
 *   handle.  Rank r's lists go to out + r*n*cap and counts + r*n; merged, to out + r*cap, labels + r*cap, count[r] and
 *   set_counts + r*n. */
int fpm_match_set_sharded(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                          fpm_result* out, int cap, int* counts);
int fpm_match_set_sharded_merged(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                 double max_overlap, fpm_result* out, int* labels, int cap, int* count, int* set_counts);
int fpm_match_set_sharded_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                                  fpm_result* out, int cap, int* counts);
int fpm_match_set_sharded_merged_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height,
                                         int stride, double max_overlap, fpm_result* out, int* labels, int cap, int* count,
                                         int* set_counts);
/* The _scaled twins of the four calls above: any scale range, and each record's scale in scales[] at the same index as in out
 * (NULL: not written).  On every rank the lists and scales are bit-identical to what fpm_match_set_scaled (_merged) returns for
 * the frame on one GPU.  The ranks shard the pose slots (angle x scale, scale-major) of every group's schedule; the collectives
 * are those of the unscaled call.  Refusals as the twin's, and min > max.  On a set of one, fpm_match_set_sharded_scaled is the
 * angle-sharded single-template scaled match (fpm_match_sharded itself keeps refusing ranges). */
int fpm_match_set_sharded_scaled(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                 fpm_result* out, double* scales, int cap, int* counts);
int fpm_match_set_sharded_scaled_merged(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                        double max_overlap, fpm_result* out, double* scales, int* labels, int cap, int* count,
                                        int* set_counts);
int fpm_match_set_sharded_scaled_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                                         fpm_result* out, double* scales, int cap, int* counts);
int fpm_match_set_sharded_scaled_merged_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height,
                                                int stride, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                                int* count, int* set_counts);
/* contiguous chunk [a0, a1) of an n_angles schedule swept by `rank` (host arithmetic, no device needed) */
int fpm_shard_angle_range(int n_angles, int nranks, int rank, int* a0, int* a1);
/* number of NCCL collectives issued by this handle since creation */
long long fpm_collective_count(const fpm_handle* h);

/* ---- stage kernels exposed for bit-exact parity tests (host pointers in and out) ---- */
int fpm_dbg_pyrdown(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, uint8_t* dst /* ((w+1)/2)*((h+1)/2) */);
/* host half of fpm_ingest_jpeg alone (no device needed): quantised luma coefficients [bh*bw][64] in natural order + the luma
   quantisation table; coef may be NULL to query the sizes */
int fpm_dbg_jpeg_luma(const uint8_t* file, size_t nbytes, int* width, int* height, int* bw, int* bh, uint16_t* quant /* 64 */,
                      int16_t* coef, size_t coef_capacity, char* err, int err_capacity);
/* the parallel (device) Huffman decoder of fpm_ingest_jpeg run thread by thread on the CPU: same coefficients as fpm_dbg_jpeg_luma */
int fpm_dbg_jpeg_luma_parallel(const uint8_t* file, size_t nbytes, int16_t* coef, size_t coef_capacity, int* passes, char* err,
                               int err_capacity);
/* CPU emulation of the whole batched device decoder (unstuffing + passes + scans), thread by thread, no device: quantised luma
   coefficients of every file, file i's [bh*bw][64] blocks at coef + coef_offsets[i] (coef_offsets has n+1 entries: file i owns
   [coef_offsets[i], coef_offsets[i+1])); passes[i] = the synchronisation passes of file i.  Files may differ in size. */
int fpm_dbg_jpeg_luma_parallel_batch(const uint8_t* data, const size_t* offsets, int n, int16_t* coef, const size_t* coef_offsets,
                                     int* passes, char* err, int err_capacity);
/* unstuffing of one file's entropy-coded segment, no device: emulated = 1 runs the device phase functions thread by thread, 0 the
   sequential host reference.  out (out_cap >= file size - scan start + 20): the bytes + 16 zero bytes; rst: first bit of every
   restart interval, rst[nint] = nbits (0, nbits without restart intervals); *tile = the compaction tile size in bytes */
int fpm_dbg_jpeg_unstuff(const uint8_t* file, size_t nbytes, int emulated, uint8_t* out, size_t out_cap, unsigned* rst, int rst_cap,
                         unsigned* nbits, int* nint, int* tile);
/* one launch of the two-level pyramid kernel: dst1 = pyrDown(src), dst2 = pyrDown(dst1) (dst2 may be NULL: one level).
   misalign: byte offset of the device copy of src past a 128-byte boundary, also added to its pitch (0 / 8 / 4 / odd select
   the 16- / 8- / 4-byte cp.async and the byte staging paths). */
int fpm_dbg_pyrdown2(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, int misalign, uint8_t* dst1, uint8_t* dst2);
int fpm_dbg_warp_affine(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, const double m[6] /* forward 2x3 */,
                        int dw, int dh, int border, uint8_t* dst /* dw*dh */);
int fpm_dbg_corr_rows(fpm_handle* h, const uint8_t* roi /* (th+6)x(tw+6) */, const uint8_t* tpl, int tw, int th,
                      int32_t* rowsum /* th*49 */, int32_t* rowS /* (th+6)*7 */, int32_t* rowQ /* (th+6)*7 */);
int fpm_dbg_corr_rows_mma(fpm_handle* h, const uint8_t* rois /* ne x (th+6)x(tw+6) */, int ne, const uint8_t* tpl, int tw, int th,
                          int32_t* rowsum /* ne*th*49 */, int32_t* rowS /* ne*(th+6)*7 */, int32_t* rowQ);
/* fused tensor-core kernel: numer[ne*49] = float32 row-ordered accumulation of the row dots per (r,c) cell,
 * winS/winQ[ne*49] = window sum / square sum of the ROI under the template at shift (r,c) */
int fpm_dbg_corr_fused(fpm_handle* h, const uint8_t* rois, int ne, const uint8_t* tpl, int tw, int th,
                       float* numer, long long* winS, long long* winQ,
                       int32_t* edge_rowS /* optional, ne*(th+6)*7: the stored first/last 6 rows, others -1 */);
int fpm_dbg_top_score(fpm_handle* h, const uint8_t* img, int w, int hgt, float* score /* (h-th+1)*(w-tw+1) */);
/* the map exactly as match() computes it: scores certainly below reject_below = Score*0.9^top - 0.01 may be float32
 * estimates (the peak search cannot observe them); *reject_below returns the bound in use (-inf: exact everywhere) */
int fpm_dbg_top_score_production(fpm_handle* h, const uint8_t* img, int w, int hgt, float* score, float* reject_below);
/* block_mode: 0 = whole-map minMaxLoc, 1 = Qt s_BlockMax (DataStructures.h:150-245), 2 = MFC s_BlockMax (MatchToolDlg.h:109-213) */
int fpm_dbg_peaks(fpm_handle* h, const float* score, int cols, int rows, int tw, int th, int block_mode,
                  double thresh, double max_overlap, int max_picks, double* picks /* max_picks*3: x,y,v */, int* n);
/* host-side (CPU) evaluation of the NMS pair decision -- geometry code shared with the device */
int fpm_dbg_rrect_overlap(const float r1[5], const float r2[5], double max_overlap, int* type, double* ratio);
int fpm_dbg_rrect_from3(const float pts[6], float out[5]);

/* ---- trace access after a match with FPM_PARAM_TRACE = 1 (single image) ---- */
int fpm_trace_num_candidates(const fpm_handle* h);
int fpm_trace_candidates(const fpm_handle* h, double* rows /* n*4: x, y, score, angle_index */);
int fpm_trace_num_evals(const fpm_handle* h, int level);
int fpm_trace_evals(const fpm_handle* h, int level, double* rows /* n*5: cand id, angle, score, locx, locy */);
int fpm_trace_level(const fpm_handle* h, int level, uint8_t* out /* w*h of the source pyramid */, int* w, int* hgt);
/* the 7x7 float32 score patch of every refinement eval of `level`, in the row order of fpm_trace_evals */
int fpm_trace_eval_scores(const fpm_handle* h, int level, float* out /* n*49, row-major per eval */);
/* the ROI patch of every refinement eval of `level` (getRotatedROI: template size + 6), in the row order of fpm_trace_evals,
 * at the device pitch: out (may be null) receives n * hgt * pitch bytes, columns w .. pitch-1 as the device holds them.
 * Returns n (>= 0); 0 on levels whose ROIs are warped inside the correlation kernel (FPM_PARAM_TENSOR_CORES = 6). */
int fpm_trace_eval_rois(const fpm_handle* h, int level, uint8_t* out, int* w, int* hgt, int* pitch);

#ifdef __cplusplus
}
#endif
#endif /* FPM_B200_H */
