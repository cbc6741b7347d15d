// fpm_host.cu -- host driver + C ABI (include/fpm_b200.h) of the B200 NCC matcher.
//
// Mirrors TemplateMatcher::learnPattern / match (/root/reference/src/TemplateMatcher.cpp:45-437)
// as a sequence of batched kernel launches; all pixel work happens on the device, the host only
// computes the angle schedule and the per-angle top-layer geometry (a few dozen doubles) and reads
// back one counter per pyramid layer.  There is no CPU fallback: without a CUDA device
// fpm_create() fails.
#include "../../include/fpm_b200.h"
#include "fpm_kernels.cuh"
#include "fpm_mma.cuh"
#include "fpm_fused.cuh"
#include "fpm_jpeg.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

namespace {

// cudaFuncAttributeMaxDynamicSharedMemorySize is per-device state of a kernel, shared by every handle and host
// thread (fpm_match_multi runs handles concurrently): the opt-in is only ever RAISED, under a lock, so one
// thread can never shrink it below what another is about to launch with.
cudaError_t ensure_dyn_smem(const void* func, int device, size_t bytes)
{
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> granted;
    if (bytes <= 48 * 1024) return cudaSuccess;
    std::lock_guard<std::mutex> lock(mu);
    size_t& cur = granted[std::make_pair(func, device)];
    if (bytes <= cur) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// getTopLayer, src/TemplateMatcher.cpp:445-455
int get_top_layer(int w, int h, int min_dst_length)
{
    int top = 0;
    int min_area = min_dst_length * min_dst_length;
    int area = w * h;
    while (area > min_area) { area /= 4; top++; }
    return top;
}

// getBestRotationSize, src/TemplateMatcher.cpp:901-969
void best_rotation_size(int sw, int sh, int dw, int dh, double dRAngle, int* ow, int* oh)
{
    double rad = dRAngle * FPM_D2R;
    float cx = (sw - 1) / 2.0f, cy = (sh - 1) / 2.0f;
    float x[4], y[4];
    fpm_pt_rotate(0.f, 0.f, cx, cy, rad, &x[0], &y[0]);
    fpm_pt_rotate(0.f, (float)(sh - 1), cx, cy, rad, &x[1], &y[1]);
    fpm_pt_rotate((float)(sw - 1), (float)(sh - 1), cx, cy, rad, &x[2], &y[2]);
    fpm_pt_rotate((float)(sw - 1), 0.f, cx, cy, rad, &x[3], &y[3]);
    float fTopY = std::max(std::max(y[0], y[1]), std::max(y[2], y[3]));
    float fBottomY = std::min(std::min(y[0], y[1]), std::min(y[2], y[3]));
    float fRightX = std::max(std::max(x[0], x[1]), std::max(x[2], x[3]));
    float fLeftX = std::min(std::min(x[0], x[1]), std::min(x[2], x[3]));
    if (dRAngle > 360) dRAngle -= 360;
    else if (dRAngle < 0) dRAngle += 360;
    if (fabs(fabs(dRAngle) - 90) < FPM_VISION_TOLERANCE || fabs(fabs(dRAngle) - 270) < FPM_VISION_TOLERANCE) {
        *ow = sh; *oh = sw; return;
    } else if (fabs(dRAngle) < FPM_VISION_TOLERANCE || fabs(fabs(dRAngle) - 180) < FPM_VISION_TOLERANCE) {
        *ow = sw; *oh = sh; return;
    }
    double dAngle = dRAngle;
    if (dAngle > 0 && dAngle < 90) {}
    else if (dAngle > 90 && dAngle < 180) dAngle -= 90;
    else if (dAngle > 180 && dAngle < 270) dAngle -= 180;
    else if (dAngle > 270 && dAngle < 360) dAngle -= 270;
    float fH1 = (float)(dw * sin(dAngle * FPM_D2R) * cos(dAngle * FPM_D2R));
    float fH2 = (float)(dh * sin(dAngle * FPM_D2R) * cos(dAngle * FPM_D2R));
    int iHalfHeight = (int)ceilf(fTopY - cy - fH1);
    int iHalfWidth = (int)ceilf(fRightX - cx - fH2);
    int rw = iHalfWidth * 2, rh = iHalfHeight * 2;
    bool wrong = (dw < rw && dh > rh) || (dw > rw && dh < rh) || ((long long)dw * dh > (long long)rw * rh);
    if (wrong) {
        rw = (int)((double)(fRightX - fLeftX) + 0.5);
        rh = (int)((double)(fTopY - fBottomY) + 0.5);
    }
    *ow = rw; *oh = rh;
}

struct TplLevelHost {
    int w = 0, h = 0, pitch = 0;
    size_t dev_off = 0;
    size_t tsh_off = 0;          // 8 pre-shifted copies for the tensor-core path
    int bpitch = 0;
    double mean = 0, norm = 0, inv_area = 1;
    int equal1 = 0;
    std::vector<uint8_t> pix;    // w*h
    size_t tpl_stride = 0;       // template groups: bytes from one member's level to the next one's
    size_t stat_off = 0;         // template groups: index of member 0's FpmTplStat of this level in d_tstat
    bool all_flat = false;       // every member's result_equal1 is set
    // masked group: member 0's M_L as 0/1 bytes (w*h) and its kept count, and where the level's run table starts in d_mruns
    // (n_tpl x (h + 1) int offsets, member k's at k * (h + 1), then the int2 runs of all members); empty mask = unmasked group
    std::vector<uint8_t> mask;
    long long n_kept = 0;
    size_t run_off = 0, run_data_off = 0;
};

struct TopPlan {                  // cached per (source size, parameters); always the WHOLE angle schedule
    int sw = 0, sh = 0, top = -1, batch = 0;
    double tol = -1, scale_min = 0, scale_max = 0;
    // pose slots k * n_angles + a of scale k and angle a (scale-major; one scale: slot == angle)
    std::vector<double> angles;   // angle per slot: the full angle schedule once per scale
    std::vector<double> scales;   // scale per slot
    std::vector<float> ftx, fty;  // canvas translation per slot
    int maxW = 0, maxH = 0;
    int n_ang = 0;                // slots: angles.size()
    bool valid = false;
};

// Templates of a set with the same level-0 size, border colour and masked-ness: they share the top layer, the angle schedule, the
// canvases, the ROI sizes and the NMS rectangle, and run through the pipeline together as virtual images
// v = frame * n + member.  The group being matched lives in the handle's fields (tpl, border, tpl0_w/h, members, plan,
// d_jobs_top, d_angles, d_ftx, d_fty, d_scales); group 0 is there at rest, the others are swapped in for their pass.  Groups of
// different top-level sizes have different scale schedules, so the slot scales belong to the group like its plan.
struct TplGroup {
    std::vector<int> members;      // set indices, ascending
    std::vector<TplLevelHost> tpl; // levels (statistics and pixels of members[0])
    int border = 0, w0 = 0, h0 = 0;
    bool masked = false;           // its members carry masks (a group is all masked or all unmasked)
    TopPlan plan;
    DevBuf d_jobs_top, d_angles, d_ftx, d_fty, d_scales;
    void release() { d_jobs_top.release(); d_angles.release(); d_ftx.release(); d_fty.release(); d_scales.release(); }
};

struct SetTpl { std::vector<uint8_t> px, mask; int w = 0, h = 0; };   // mask: 0/1 bytes (w*h), empty = unmasked

}  // namespace

struct fpm_handle {
    int device = 0;
    int num_sms = 148;             // cudaDevAttrMultiProcessorCount of the device (B200: 148); sizes the wave arithmetic
    cudaStream_t stream = nullptr, copy_stream = nullptr, aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    // parameters (src/TemplateMatcher.cpp:28-39)
    int max_pos = 70;
    double max_overlap = 0.0, score = 0.7, tol_angle = 0.0;
    int min_reduce_area = 256;
    int use_simd = 1, subpixel = 0, trace = 0;
    double workspace_mb = 4096;
    int h2d_chunk = 0;             // frames per H2D chunk in fpm_match_batch (0 = auto)
    bool mma_attr_set = false, fused_attr_set = false, peaks_attr_set = false, warpmma_attr_set = false;
    // concurrent half-batches (fpm_match_batch_device): a second handle with the same template and parameters
    fpm_handle* twin = nullptr;
    int split_batch = 8;           // FPM_PARAM_SPLIT_BATCH: smallest batch that is split in two (0 = never)
    unsigned learn_gen = 0, twin_gen = 0;
    int stop_layer1 = 0, bitwise_not = 0, tol_range = 0;   // MFC-only modes (MatchTool/MatchToolDlg.cpp:788-816, :936)
    double tol_r[4] = {0, 0, 0, 0};
    double scale_min = 1.0, scale_max = 1.0;   // FPM_PARAM_SCALE_MIN / MAX: the match scale range
    int mfc_compat = 0;            // 1: MFC result convention (angle sign/wrap, TargetNum truncation, double corners)
    int async_descent = -1;        // FPM_PARAM_ASYNC_DESCENT: -1 auto (batches < 8 frames), 0 never, 1 always
    int jpeg_device_huffman = 1;   // FPM_PARAM_JPEG_DEVICE_HUFFMAN
    int jpeg_passes = 0;           // synchronisation passes of the last JPEG ingest (0: decoded on the host)
    DevBuf d_jpeg_scan;            // JPEG ingest: the uploaded files, their unstuffed scans, restart positions
    DevBuf d_jpeg;                 // JPEG ingest: file descriptors, decoder states, DC values of a decode wave
    int cur_batch = 1;             // frames of the match in flight
    bool err_check_pending = false;
    int use_tc = 1;                // 0 = dp4a only, 1 = tcgen05 for large levels, 2 = tcgen05 wherever possible
    // template
    bool learned = false;
    int learned_mra = -1;
    int border = 0;
    std::vector<SetTpl> set;       // the learned templates (fpm_learn: one), kept for re-learning when MinReduceArea changes
    bool masked_set = false;       // learned by fpm_learn_set_masked: learn refusals name the template index
    DevBuf d_mruns, d_mpyr, d_mwS, d_mwQ;   // masked templates: run tables, mask pyramids at learn time, refinement window sums
    std::vector<TplGroup> groups;  // their groups; groups[0]'s state is in the fields below (see TplGroup)
    DevBuf d_tstat;                // FpmTplStat of every (group, level, member)
    DevBuf d_members;              // the members of every group, group after group (merged set results: output rows)
    DevBuf d_mlists, d_merged;     // merged set results: per-template lists of a sub-batch, the merge's outputs
    std::vector<int> members;      // current group: its set indices
    int tpl0_w = 0, tpl0_h = 0;    // current group: level-0 size
    std::vector<TplLevelHost> tpl;
    DevBuf d_tpl, d_tsh, d_raw, d_inv, d_numer, d_totS, d_totQ, d_ingest_raw, d_ingest;
    int ingest_w = 0, ingest_h = 0, ingest_pitch = 0;      // last ingested frames (device resident, [count][h][pitch])
    int ingest_count = 0;
    // user rect (pure storage)
    int ur[4] = {0, 0, 0, 0};
    int has_ur = 0;
    // workspace
    DevBuf d_src, d_pyr, d_rot, d_score, d_blkv, d_blkl, d_picks, d_pickcnt, d_jobs_top, d_angles, d_ftx, d_fty, d_scales;
    DevBuf d_off, d_keys, d_cand[2], d_candcnt, d_toppt, d_counters, d_jobs_ref, d_roi, d_rowsum, d_rowS, d_rowQ;
    DevBuf d_pairs, d_refined, d_rects, d_del, d_idmap, d_results, d_rescnt, d_trace, d_trace_sc, d_dbg[4];
    PinnedBuf h_counts, h_results, h_stage;
    // angle-sharded latency mode (fpm_match_sharded): this handle is rank sh_rank of sh_nranks
    int sh_nranks = 1, sh_rank = 0;
    void* nccl_comm = nullptr;     // ncclComm_t (created by fpm_comm_init or borrowed through fpm_comm_attach)
    bool nccl_owned = false;
    int shard_upload = 1;          // FPM_PARAM_SHARD_UPLOAD: host frame uploaded as 1/N row slices + NVLink allgather
    DevBuf d_gpicks, d_grefined;   // allgather buffers: one fixed-size block per rank, consumed in place by the kernels
    FpmRefined* ref_out = nullptr; // where run_refine appends (null: d_refined / counters[CNT_REFINED])
    // fpm_match_scaled and the scaled set calls: run_final / run_set_merge write the scale of the record written at out_base[i]
    // to scales_out[i] (out_base: the caller's whole output array, so chunks, split halves, their twin handle and the ranks of
    // the virtual angle-sharded calls all index it the same way)
    double* scales_out = nullptr;
    const fpm_result* scales_base = nullptr;
    const char* scaled_fn = nullptr;   // the call in flight returns scales: a set matches at any range, refusals name this call
    int* ref_cnt = nullptr;
    // one call's layout of the rank blocks, the same on every rank: block = picks of every group that runs
    // [group][template][chunk angle][MaxPos+5], then their counts [group][template][chunk angle]; refined block = one
    // segment { FpmRefined[seg_cap]; int count; int pad } per group
    struct ShardGroup { int chunk = 0, n_tpl = 0, seg_cap = 0, n_local = 0, key_stride = 1; size_t pick_off = 0, cnt_off = 0, ref_off = 0; };
    struct ShardState {
        int empty = 1;
        size_t pick_blk = 0, cnt_off = 0, n_cnt = 0, ref_blk = 0;   // cnt_off: bytes to the counts; n_cnt: ints of counts
        std::vector<char> run;
        std::vector<ShardGroup> g;
    } sh;
    std::vector<FpmLevel> levels; // source pyramid of the current batch
    const std::vector<FpmLevel>* shared_levels = nullptr;   // fpm_match_multi: the pyramid built once by the first handle
    TopPlan plan;
    mutable std::string err;       // also set by the const accessors that refuse a template set
    double last_ms = 0;
    long long launches = 0, collectives = 0;
    // per-kernel profiling (CUDA events on the launch stream)
    int profile = 0;
    std::vector<cudaEvent_t> ev_pool;
    struct ProfRec { int kid; cudaEvent_t a, b; double work; };
    std::vector<ProfRec> prof_pending;
    double prof_ms[24] = {0}, prof_work[24] = {0};
    long long prof_launches[24] = {0};
    cudaEvent_t prof_cur = nullptr;
    // trace
    std::vector<double> tr_cands;                 // n*4
    std::vector<std::vector<double>> tr_evals;    // per level, n*5
    std::vector<std::vector<float>> tr_scores;    // per level, n*49: the 7x7 score patch of every row of tr_evals
    struct TraceRois { int w = 0, h = 0, pitch = 0; std::vector<uint8_t> px; };
    std::vector<TraceRois> tr_rois;               // per level, n ROI patches of h rows at full pitch (none on warp-fused levels)
};

namespace {

#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                \
            return FPM_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

#define CKL()                                                                            \
    do {                                                                                 \
        h->launches++;                                                                   \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) {                                                        \
            h->err = std::string("kernel launch: ") + cudaGetErrorString(e__);           \
            return FPM_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

// CNT_LAYER + l: candidates entering pyramid layer l (descent without host round trips)
enum { CNT_FLAT = 0, CNT_NEXT = 1, CNT_REFINED = 2, CNT_TOTAL = 3, CNT_ERR = 4, CNT_LAYER = 8, CNT_N = 8 + FPM_MAX_LEVELS };
enum { K_PYRDOWN = 0, K_WARP_TOP, K_TOP_SCORE, K_TOP_PEAKS, K_COLLECT, K_PREP, K_WARP_ROI, K_CORR, K_FINALIZE, K_FINAL, K_CORR_MMA, K_CORR_FUSED, K_CORR_WARP,
       K_JPEG_UPLOAD, K_JPEG_UNSTUFF, K_JPEG_PASSES, K_JPEG_SCAN, K_JPEG_WRITE, K_JPEG_IDCT, K_SET_MERGE, K_TOP_SCORE_MASKED,
       K_MASK_WINDOW, K_COUNT };
const char* const kKernelNames[K_COUNT] = {"fpm_pyrdown_kernel", "fpm_warp_kernel(top)", "fpm_top_score_kernel", "fpm_top_peaks_kernel",
                                           "fpm_collect_sort_kernel", "fpm_refine_prep_kernel", "fpm_warp_kernel(roi)",
                                           "fpm_corr_rows_kernel", "fpm_refine_finalize_kernel", "fpm_final_kernel",
                                           "fpm_corr_mma_kernel", "fpm_corr_fused_kernel", "fpm_corr_warp_kernel",
                                           "jpeg_upload(H2D copy)", "fpm_jpeg_unstuff_count/write_kernel", "fpm_jpeg_cold/sync_kernel(passes)",
                                           "fpm_jpeg_block_tile/dc_tile/offsets_kernel(scans)", "fpm_jpeg_write_kernel", "fpm_ingest_jpeg_idct_kernel",
                                           "fpm_set_merge_kernel", "fpm_top_score_kernel(masked)", "fpm_mask_window_kernel"};
static_assert(K_COUNT <= 24, "profile arrays");

cudaEvent_t prof_event(fpm_handle* h)
{
    if (!h->ev_pool.empty()) { cudaEvent_t e = h->ev_pool.back(); h->ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

inline void prof_begin(fpm_handle* h, cudaStream_t st = nullptr)
{
    if (!h->profile) return;
    h->prof_cur = prof_event(h);
    cudaEventRecord(h->prof_cur, st ? st : h->stream);
}

inline void prof_end(fpm_handle* h, int kid, double work, cudaStream_t st = nullptr)
{
    if (!h->profile) return;
    cudaEvent_t b = prof_event(h);
    cudaEventRecord(b, st ? st : h->stream);
    h->prof_pending.push_back({kid, h->prof_cur, b, work});
}

void prof_collect(fpm_handle* h)
{
    if (h->prof_pending.empty()) return;
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->aux_stream);
    for (auto& r : h->prof_pending) {
        float ms = 0;
        cudaEventElapsedTime(&ms, r.a, r.b);
        h->prof_ms[r.kid] += ms; h->prof_work[r.kid] += r.work; h->prof_launches[r.kid]++;
        h->ev_pool.push_back(r.a); h->ev_pool.push_back(r.b);
    }
    h->prof_pending.clear();
}

// launch wrapper: KL(kernel id, algorithmic work of this launch, <<<launch>>> statement)
#define KL(kid, work, ...)                 \
    do {                                   \
        prof_begin(h);                     \
        __VA_ARGS__;                       \
        prof_end(h, kid, (double)(work));  \
        CKL();                             \
    } while (0)

FpmTplLevel tpl_level_dev(const fpm_handle* h, int l)
{
    const TplLevelHost& t = h->tpl[l];
    FpmTplLevel d;
    d.ptr = h->d_tpl.as<uint8_t>() + t.dev_off;
    d.w = t.w; d.h = t.h; d.pitch = t.pitch;
    d.mean = t.mean; d.norm = t.norm; d.inv_area = t.inv_area; d.result_equal1 = t.equal1;
    d.n_tpl = std::max((int)h->members.size(), 1);
    d.tpl_stride = t.tpl_stride;
    d.stats = d.n_tpl > 1 ? h->d_tstat.as<FpmTplStat>() + t.stat_off : nullptr;
    d.mrow = t.mask.empty() ? nullptr : reinterpret_cast<const int*>(h->d_mruns.as<uint8_t>() + t.run_off);
    d.mrun = t.mask.empty() ? nullptr : reinterpret_cast<const int2*>(h->d_mruns.as<uint8_t>() + t.run_data_off);
    return d;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_tiled();

// One launch of the pyramid kernel: d1 = pyrDown(src) and, when d2 is given, d2 = pyrDown(d1) from the level-1 tile that is
// still in shared memory (fpm_pyrdown.cuh).
int launch_pyrdown(fpm_handle* h, const FpmLevel& src, const FpmLevel& d1, const FpmLevel* d2, int batch)
{
    auto aligned = [](const FpmLevel& L, int a) {
        return ((reinterpret_cast<uintptr_t>(L.ptr) % a) == 0) && (L.pitch % a == 0) && (L.img_stride % a == 0);
    };
    Pd2Args a;
    a.src = src; a.d1 = d1; a.d2 = d2 ? *d2 : FpmLevel{nullptr, 0, 0, 0, 0};
    a.vec = aligned(src, 16) ? 16 : (aligned(src, 8) ? 8 : (aligned(src, 4) ? 4 : 1));
    a.st1_vec = aligned(d1, 8) ? 1 : 0;
    a.st2_vec = (d2 && aligned(*d2, 8)) ? 1 : 0;
    dim3 grid((d1.w + PD2_TW - 1) / PD2_TW, (d1.h + PD2_TH - 1) / PD2_TH, batch);
    // 16-byte aligned source: the staged tile of a CTA is one TMA load of the [batch][h][pitch/4] u32 view of the level
    // (the row padding belongs to the tensor; the kernel never uses what it holds)
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    if (a.vec >= 16) {
        EncodeTiledFn enc = get_encode_tiled();
        if (!enc) { h->err = "cuTensorMapEncodeTiled not available"; return FPM_ERR_CUDA; }
        const cuuint64_t img = src.img_stride ? (cuuint64_t)src.img_stride : (cuuint64_t)src.pitch * src.h;
        cuuint64_t dims[3] = {(cuuint64_t)src.pitch / 4, (cuuint64_t)src.h, (cuuint64_t)batch};
        cuuint64_t strides[2] = {(cuuint64_t)src.pitch, img};
        cuuint32_t box[3] = {(cuuint32_t)((d2 ? Pd2Cfg<true>::IP : Pd2Cfg<false>::IP) / 4), (cuuint32_t)(d2 ? Pd2Cfg<true>::IH : Pd2Cfg<false>::IH), 1};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, src.ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) a.vec = 8;                   // e.g. a stride beyond the descriptor's range: cp.async staging instead
    }
    // algorithmic bytes (SURVEY 8d): every level of the chain read once and written once, also the level that stays on chip
    double work = (double)batch * ((double)src.w * src.h + (double)d1.w * d1.h);
    if (d2) {
        work += (double)batch * ((double)d1.w * d1.h + (double)d2->w * d2->h);
        CK(ensure_dyn_smem((const void*)fpm_pyrdown_kernel<true>, h->device, Pd2Cfg<true>::SMEM));
        KL(K_PYRDOWN, work, fpm_pyrdown_kernel<true><<<grid, Pd2Cfg<true>::NT, Pd2Cfg<true>::SMEM, h->stream>>>(a, tmap));
    } else {
        CK(ensure_dyn_smem((const void*)fpm_pyrdown_kernel<false>, h->device, Pd2Cfg<false>::SMEM));
        KL(K_PYRDOWN, work, fpm_pyrdown_kernel<false><<<grid, Pd2Cfg<false>::NT, Pd2Cfg<false>::SMEM, h->stream>>>(a, tmap));
    }
    return FPM_OK;
}

// levels[1..top] from levels[0], two levels per launch
int launch_pyramid_chain(fpm_handle* h, const std::vector<FpmLevel>& lv, int top, int batch)
{
    for (int l = 1; l <= top;) {
        const bool two = l + 1 <= top;
        int rc = launch_pyrdown(h, lv[l - 1], lv[l], two ? &lv[l + 1] : nullptr, batch);
        if (rc) return rc;
        l += two ? 2 : 1;
    }
    return FPM_OK;
}

// launch geometry of fpm_corr_rows_kernel for a template level (per_eval_tpl: every eval stages its own template rows,
// the evals of a CTA may belong to different templates of a group)
struct CorrCfg { int rb, evals_per_cta, threads; size_t smem; int blocks_y_rows; };

CorrCfg corr_config(int tpl_h, bool per_eval_tpl = false)
{
    CorrCfg c;
    const int rh = tpl_h + FPM_ROI_PAD;
    if (rh > 128) {
        int nblk = (rh + CR_MAX_THREADS - 1) / CR_MAX_THREADS;
        c.rb = (int)align_up((size_t)(rh + nblk - 1) / nblk, 32);
        c.evals_per_cta = 1;
        c.blocks_y_rows = (rh + c.rb - 1) / c.rb;
    } else {
        c.rb = rh;
        c.evals_per_cta = CR_MAX_THREADS / rh;
        c.blocks_y_rows = 1;
    }
    c.threads = (int)align_up((size_t)c.rb * c.evals_per_cta, 32);
    const size_t n_srow = (size_t)c.evals_per_cta * c.rb, n_trow = (size_t)c.rb + FPM_ROI_PAD;
    size_t stage = (n_srow + (per_eval_tpl ? c.evals_per_cta : 1) * n_trow) * CR_PW * 4;
    size_t outb = (size_t)c.evals_per_cta * n_trow * FPM_NCELL * 4;
    c.smem = std::max(2 * stage, outb);      // two slab buffers (cp.async double buffering)
    return c;
}

// masked: row prefix sums of TS_TW + tw entries in place of the TS_TW row-window sums
inline size_t top_score_smem(int tw, int th, bool masked = false)
{
    size_t nwt = (tw + 3) / 4, pww = TS_TW / 4 + nwt + 1, rs_w = masked ? TS_TW + tw : TS_TW;
    return 4 * ((size_t)th * nwt + (size_t)(TS_TH + th - 1) * (pww + 2 * rs_w)) + 16;   // template, patch, row-window sums
}

inline int level_vec_ok(const FpmLevel& L)
{
    return ((reinterpret_cast<uintptr_t>(L.ptr) & 3) == 0) && (L.pitch % 4 == 0) && (L.img_stride % 4 == 0);
}

// room for the peak kernel's block table in shared memory (value + location per block); 0 = keep it in global scratch
int peaks_smem_blocks(fpm_handle* h, int blk_stride)
{
    const int cap = 16384;                                   // 128 KB of dynamic shared memory next to the 24 KB static
    if (blk_stride > cap) return 0;
    if (!h->peaks_attr_set) {
        if (ensure_dyn_smem((const void*)fpm_top_peaks_kernel, h->device, (size_t)cap * 8) != cudaSuccess) {
            h->err = "cudaFuncSetAttribute(fpm_top_peaks_kernel) failed";
            return -1;
        }
        h->peaks_attr_set = true;
    }
    return blk_stride;
}

// ---- tensor-core correlation (fpm_mma.cuh): TMA descriptors + launch -----------------------
EncodeTiledFn get_encode_tiled()
{
    // function-local static: initialised once, thread-safe (handles may run on several host threads)
    static const EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<EncodeTiledFn>(p);
        return nullptr;
    }();
    return fn;
}

// 3-D u8 tensor [d2][d1][d0 bytes] with byte strides s1, s2; box (b0, b1, b2); 128-byte swizzle, zero OOB fill
int make_map_3d(fpm_handle* h, CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2,
                uint32_t b0, uint32_t b1, uint32_t b2)
{
    EncodeTiledFn enc = get_encode_tiled();
    if (!enc) { h->err = "cuTensorMapEncodeTiled not available"; return FPM_ERR_CUDA; }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {s1, s2};
    cuuint32_t box[3] = {b0, b1, b2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { h->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"; return FPM_ERR_CUDA; }
    return FPM_OK;
}

// which correlation path a template level takes: 0 = dp4a (fpm_corr_rows_kernel), 1 = tensor cores
// The tensor-core kernels share one B operand (the pre-shifted template) across the 128 evals of a tile: groups of
// more than one template take dp4a (bit-identical results).
bool mma_usable(const fpm_handle* h, int tw)
{
    if (h->use_tc == 0 || h->members.size() > 1) return false;
    if (!get_encode_tiled()) return false;
    return (h->use_tc == 2 || h->use_tc == 4) ? true : tw >= 64;     // modes 1, 3, 5, 6: large levels
}

// narrow levels (16 <= width < 64): the row-split tensor-core kernel does not beat dp4a there (256 B of row dots per
// 22..70-byte ROI row), the fused kernel does as soon as the level has enough evals to fill the SMs
bool mma_narrow_fused(const fpm_handle* h, int tw)
{
    return (h->use_tc == 1 || h->use_tc == 6) && h->use_simd && h->members.size() <= 1 && get_encode_tiled() && tw >= 16 && tw < 64;
}

// The fused kernel keeps one CTA on 128 evals for all ROI rows: it wins when the evals fill the SMs and the rows are
// short (then the row-split kernel is dominated by the 256 B of row dots per (eval, row) that it writes and the
// finalize kernel reads back), and loses when a level has few evals and long rows.  Measured on B200: a fused CTA
// streams its ROI patches at ~27 GB/s from HBM; the row-split path moves ~(row + 568) bytes per (eval, row) at ~5 TB/s.
bool fused_pays(int ne, int rh, int rpitch, int k_bytes, int use_tc, int num_sms)
{
    (void)rh; (void)k_bytes;
    if (use_tc == 4) return true;                                     // forced (tests)
    const double m_tiles = (ne + MM_M - 1) / MM_M;
    const double rounds = ceil(m_tiles / (double)num_sms);
    return m_tiles / rounds > 185.0 * rpitch / (rpitch + 568.0);
}

// fused tensor-core correlation: numerators (float chain), window totals and edge rows for `ne` ROI patches
int launch_corr_fused(fpm_handle* h, const uint8_t* roi, int rpitch, size_t roi_stride, const uint8_t* tsh, int bpitch, int tw, int th,
                      int ne, int32_t* rowS, int32_t* rowQ, const int* n_cands_dev = nullptr, int n_ang = 1)
{
    const int rh = th + FPM_ROI_PAD;
    const int m_tiles = (ne + MM_M - 1) / MM_M;
    CK(h->d_numer.ensure((size_t)ne * MM_N * sizeof(float)));
    CK(h->d_totS.ensure((size_t)ne * FPM_NSHIFT * sizeof(long long)));
    CK(h->d_totQ.ensure((size_t)ne * FPM_NSHIFT * sizeof(long long)));
    CUtensorMap map_a, map_b;
    int rc = make_map_3d(h, &map_a, roi, (uint64_t)rpitch, (uint64_t)rh, (uint64_t)ne, (uint64_t)rpitch, (uint64_t)roi_stride, MM_KCHUNK, 1, MM_M);
    if (rc) return rc;
    rc = make_map_3d(h, &map_b, tsh, (uint64_t)bpitch, (uint64_t)th, 8, (uint64_t)bpitch, (uint64_t)bpitch * th, MM_KCHUNK, 8, 8);
    if (rc) return rc;
    if (!h->fused_attr_set) {
        CK(ensure_dyn_smem((const void*)fpm_corr_fused_kernel, h->device, FM_SMEM_BYTES));
        h->fused_attr_set = true;
    }
    KL(K_CORR_FUSED, (double)ne * FPM_NCELL * (double)tw * th,
       fpm_corr_fused_kernel<<<m_tiles, FM_THREADS, FM_SMEM_BYTES, h->stream>>>(map_a, map_b, ne, rh, tw, th, tw + FPM_ROI_PAD,
                                                                               h->d_numer.as<float>(), rowS, rowQ,
                                                                               h->d_totS.as<long long>(), h->d_totQ.as<long long>(),
                                                                               n_cands_dev, n_ang));
    return FPM_OK;
}

// raw[y][e_pad][64] s32 + rowS/rowQ for `ne` ROI patches of one template level
int launch_corr_mma(fpm_handle* h, const uint8_t* roi, int rpitch, size_t roi_stride, const uint8_t* tsh, int bpitch, int tw, int th,
                    int ne, int* e_pad_out, int32_t* rowS, int32_t* rowQ, const int* n_cands_dev = nullptr, int n_ang = 1)
{
    const int rh = th + FPM_ROI_PAD;
    const int m_tiles = (ne + MM_M - 1) / MM_M;
    const int e_pad = m_tiles * MM_M;
    *e_pad_out = e_pad;
    CK(h->d_raw.ensure((size_t)rh * e_pad * MM_N * sizeof(int32_t)));
    CUtensorMap map_a, map_b;
    int rc = make_map_3d(h, &map_a, roi, (uint64_t)rpitch, (uint64_t)rh, (uint64_t)ne, (uint64_t)rpitch, (uint64_t)roi_stride, MM_KCHUNK, 1, MM_M);
    if (rc) return rc;
    rc = make_map_3d(h, &map_b, tsh, (uint64_t)bpitch, (uint64_t)th, 8, (uint64_t)bpitch, (uint64_t)bpitch * th, MM_KCHUNK, 8, 8);
    if (rc) return rc;
    // at most 2 full waves of the SMs (148 on B200; one CTA per SM): a third, nearly empty wave would cost a whole CTA time;
    // at least 2 ROI rows per CTA.  With the live count only known on the device (n_cands_dev) `ne` is the top-layer upper
    // bound and nearly all tiles leave at once: the rows are split as if one tile were live.
    int chunks = std::max(1, (2 * h->num_sms) / (n_cands_dev ? 1 : m_tiles));
    int rows_per_cta = std::max(2, (rh + chunks - 1) / chunks);
    chunks = (rh + rows_per_cta - 1) / rows_per_cta;
    if (!h->mma_attr_set) {                                  // per handle: the attribute is per device
        CK(ensure_dyn_smem((const void*)fpm_corr_mma_kernel, h->device, MM_SMEM_BYTES));
        h->mma_attr_set = true;
    }
    dim3 grid(chunks, m_tiles);
    KL(K_CORR_MMA, (double)ne * FPM_NCELL * (double)tw * th,
       fpm_corr_mma_kernel<<<grid, MM_THREADS, MM_SMEM_BYTES, h->stream>>>(map_a, map_b, ne, e_pad, rh, tw, th, tw + FPM_ROI_PAD,
                                                                           rows_per_cta, h->d_raw.as<int32_t>(), rowS, rowQ,
                                                                           n_cands_dev, n_ang));
    return FPM_OK;
}

// ---- ROI warp fused into the tensor-core correlation's producer (fpm_fused.cuh) ----------------------------------
// copy width the source level allows for the box staging (0 = not even word aligned: the kernel is not used)
inline int level_copy_vec(const FpmLevel& L)
{
    const uintptr_t p = reinterpret_cast<uintptr_t>(L.ptr);
    for (int v = 16; v >= 4; v >>= 1)
        if (p % v == 0 && L.pitch % v == 0 && L.img_stride % v == 0) return v;
    return 0;
}

// worst-case bytes of the source box of one visit (8 ROI rows x 128 columns, the 3 angles of a candidate, which are anchored
// at the same point and at most ~6 px apart anywhere in the ROI) over all rotation angles
bool fw_box_fits(int vec)
{
    static int worst[17] = {0};
    if (!worst[vec]) {
        double mx = 0;
        for (int i = 0; i <= 360; i++) {
            const double a = i * 0.25 * FPM_D2R, c = fabs(cos(a)), s = fabs(sin(a));
            const double W = 127 * c + (FW_R - 1) * s + 3 + 8, H = 127 * s + (FW_R - 1) * c + 3 + 8;
            const double pitch = floor((W + 2 * vec) / vec) * vec + 4;
            mx = std::max(mx, pitch * (H + 1));
        }
        worst[vec] = (int)mx;
    }
    return worst[vec] <= FW_BOX_BYTES;
}

// A masked template takes the mode-1 route: its window sums are computed from the ROI patches in HBM, which this kernel
// never writes.
bool corr_warp_usable(const fpm_handle* h, int tw, int n_ang, const FpmLevel& L)
{
    if (h->use_tc != 6 || h->members.size() > 1 || !h->tpl[0].mask.empty()) return false;   // opt-in: bit-identical, less DRAM traffic, but slower than warp + MMA today
    if (h->scale_min != 1.0 || h->scale_max != 1.0) return false;   // scaled ROIs: source boxes this kernel's staging is not sized for
    if (n_ang != 3 || tw < 64 || !get_encode_tiled()) return false;
    return level_copy_vec(L) >= 4 && fw_box_fits(4);       // the box is staged with 4-byte copies
}

// raw[y][tile*128 + slot][64] s32 + rowS/rowQ for the 3 angles of `nc` candidates, straight from the source level
int launch_corr_warp(fpm_handle* h, const FpmLevel& L, const FpmWarpJob* jobs, const uint8_t* tsh, int bpitch, int tw, int th,
                     int nc, int* e_pad_out, int32_t* rowS, int32_t* rowQ, const int* n_cands_dev = nullptr)
{
    const int rh = th + FPM_ROI_PAD;
    const int m_tiles = (nc + FW_CANDS - 1) / FW_CANDS;
    const int e_pad = m_tiles * FW_M;
    *e_pad_out = e_pad;
    CK(h->d_raw.ensure((size_t)rh * e_pad * MM_N * sizeof(int32_t)));
    CUtensorMap map_b;
    int rc = make_map_3d(h, &map_b, tsh, (uint64_t)bpitch, (uint64_t)th, 8, (uint64_t)bpitch, (uint64_t)bpitch * th, MM_KCHUNK, 8, 8);
    if (rc) return rc;
    if (!h->warpmma_attr_set) {
        CK(ensure_dyn_smem((const void*)fpm_corr_warp_kernel, h->device, FW_SMEM_BYTES));
        h->warpmma_attr_set = true;
    }
    dim3 grid((rh + FW_R - 1) / FW_R, m_tiles);
    KL(K_CORR_WARP, (double)nc * 3 * FPM_NCELL * (double)tw * th,
       fpm_corr_warp_kernel<<<grid, FW_THREADS, FW_SMEM_BYTES, h->stream>>>(jobs, nc, L, level_copy_vec(L), map_b, rh, tw, th,
                                                                            tw + FPM_ROI_PAD, e_pad, h->d_raw.as<int32_t>(), rowS, rowQ,
                                                                            h->d_counters.as<int>() + CNT_ERR, n_cands_dev));
    return FPM_OK;
}

// masked group: the 49 window sums of every eval, int64 [e][49] in d_mwS / d_mwQ, from the ROI patches in d_roi (eval e of
// candidate cands[e / n_ang], whose template is cands[e / n_ang].img % td.n_tpl)
int launch_mask_window(fpm_handle* h, int rpitch, size_t roi_stride, const FpmTplLevel& td, int ne, const int* n_cands_dev, int n_ang,
                       const FpmCand* cands)
{
    const int pstride = (int)align_up(td.w + FPM_ROI_PAD + 1, 4);                 // prefix entries of one ROI row
    const size_t per_warp = 2 * sizeof(uint32_t) * (size_t)pstride;
    if (per_warp > 200 * 1024) { h->err = "masked template too wide for the window-sum kernel"; return FPM_ERR_LIMIT; }
    const int warps = (int)std::min<size_t>(MW_MAX_WARPS, std::max<size_t>(1, 64 * 1024 / per_warp));   // <= 64 KB per CTA
    const size_t smem = warps * per_warp;
    CK(ensure_dyn_smem((const void*)fpm_mask_window_kernel, h->device, smem));
    CK(h->d_mwS.ensure((size_t)ne * FPM_NCELL * sizeof(long long)));
    CK(h->d_mwQ.ensure((size_t)ne * FPM_NCELL * sizeof(long long)));
    // algorithmic work: one pass over the ROI patch (bytes)
    KL(K_MASK_WINDOW, (double)ne * (td.w + FPM_ROI_PAD) * (td.h + FPM_ROI_PAD),
       fpm_mask_window_kernel<<<ne, warps * 32, smem, h->stream>>>(h->d_roi.as<uint8_t>(), rpitch, roi_stride, td, ne, pstride,
                                                                   h->d_mwS.as<long long>(), h->d_mwQ.as<long long>(), n_cands_dev, n_ang,
                                                                   cands));
    return FPM_OK;
}

// ---- learnPattern, src/TemplateMatcher.cpp:45-95, for every template of the set ---------------------
// Device layout: group by group and level by level, the members of a group level back to back (a set of one: today's
// single-template layout).  Each group's template pyramids are built by one pyramid chain over its members.
int do_learn(fpm_handle* h)
{
    CK(cudaSetDevice(h->device));
    h->learned = false;
    for (size_t g = 1; g < h->groups.size(); g++) h->groups[g].release();
    h->groups.clear();
    std::vector<TplGroup> gs;
    // masked and unmasked templates never share a group: unmasked groups keep the kernels without run walks
    for (int i = 0; i < (int)h->set.size(); i++) {
        const SetTpl& st = h->set[i];
        const bool masked = !st.mask.empty();
        unsigned long long S = 0, N = 0;
        for (size_t k = 0; k < st.px.size(); k++)
            if (!masked || st.mask[k]) { S += st.px[k]; N++; }
        const int border = ((double)S / (double)N) < 128 ? 255 : 0;     // iBorderColor (:58-59), over the kept pixels
        size_t g = 0;
        while (g < gs.size() && !(gs[g].w0 == st.w && gs[g].h0 == st.h && gs[g].border == border && gs[g].masked == masked)) g++;
        if (g == gs.size()) { gs.emplace_back(); gs[g].w0 = st.w; gs[g].h0 = st.h; gs[g].border = border; gs[g].masked = masked; }
        gs[g].members.push_back(i);
    }
    size_t off = 0, toff = 0, n_stat = 0;
    for (TplGroup& G : gs) {
        const int top = get_top_layer(G.w0, G.h0, (int)sqrt((double)h->min_reduce_area));
        if (top + 1 > FPM_MAX_LEVELS) { h->err = "too many pyramid levels"; return FPM_ERR_LIMIT; }
        const int T = (int)G.members.size();
        G.tpl.assign(top + 1, TplLevelHost());
        int w = G.w0, hh = G.h0;
        for (int l = 0; l <= top; l++) {
            TplLevelHost& t = G.tpl[l];
            t.w = w; t.h = hh; t.pitch = (int)align_up(w, 16);
            t.dev_off = off;
            t.tpl_stride = align_up((size_t)t.pitch * hh, 256);
            off += t.tpl_stride * T;
            t.stat_off = n_stat;
            n_stat += T;
            if (T == 1) {                                          // 8 pre-shifted copies for the tensor-core path
                t.bpitch = (int)align_up(t.w + 8, 16);
                t.tsh_off = toff;
                toff += align_up((size_t)8 * t.h * t.bpitch, 256);
            }
            w = (w + 1) / 2; hh = (hh + 1) / 2;
        }
    }
    CK(h->d_tpl.ensure(off));
    CK(cudaMemsetAsync(h->d_tpl.p, 0, off, h->stream));
    for (const TplGroup& G : gs) {
        const TplLevelHost& t0 = G.tpl[0];
        for (size_t k = 0; k < G.members.size(); k++)
            CK(cudaMemcpy2DAsync(h->d_tpl.as<uint8_t>() + t0.dev_off + k * t0.tpl_stride, t0.pitch, h->set[G.members[k]].px.data(), G.w0,
                                 G.w0, G.h0, cudaMemcpyHostToDevice, h->stream));
        const int top = (int)G.tpl.size() - 1, T = (int)G.members.size();
        std::vector<FpmLevel> lv(top + 1);
        for (int l = 0; l <= top; l++)
            lv[l] = FpmLevel{h->d_tpl.as<uint8_t>() + G.tpl[l].dev_off, G.tpl[l].w, G.tpl[l].h, G.tpl[l].pitch, T > 1 ? G.tpl[l].tpl_stride : 0};
        int rc = launch_pyramid_chain(h, lv, top, T);
        if (rc) return rc;
    }
    // mask pyramids of the masked groups: M_{L+1} = (pyrDown(255 * M_L) >= 128), per level one launch of the pyramid kernel
    // over the group's members (at k * tpl_stride, as their templates) and one read-back.  mk[g][l]: the members' M_l, w*h each.
    std::vector<std::vector<std::vector<uint8_t>>> mk(gs.size());
    for (size_t gi = 0; gi < gs.size(); gi++) {
        const TplGroup& G = gs[gi];
        if (!G.masked) continue;
        const std::vector<TplLevelHost>& tl = G.tpl;
        const int T = (int)G.members.size();
        mk[gi].assign(tl.size(), std::vector<uint8_t>());
        for (int k = 0; k < T; k++) mk[gi][0].insert(mk[gi][0].end(), h->set[G.members[k]].mask.begin(), h->set[G.members[k]].mask.end());
        CK(h->d_mpyr.ensure(off));
        uint8_t* mb = h->d_mpyr.as<uint8_t>();
        for (size_t l = 1; l < tl.size(); l++) {
            const TplLevelHost &a = tl[l - 1], &b = tl[l];
            const size_t na = (size_t)a.w * a.h, nb = (size_t)b.w * b.h;
            std::vector<uint8_t> up(a.tpl_stride * T, 0), dn(b.tpl_stride * T);
            for (int k = 0; k < T; k++)
                for (int y = 0; y < a.h; y++)
                    for (int x = 0; x < a.w; x++) up[k * a.tpl_stride + (size_t)y * a.pitch + x] = mk[gi][l - 1][k * na + (size_t)y * a.w + x] ? 255 : 0;
            CK(cudaMemcpyAsync(mb + a.dev_off, up.data(), up.size(), cudaMemcpyHostToDevice, h->stream));
            int rc = launch_pyrdown(h, FpmLevel{mb + a.dev_off, a.w, a.h, a.pitch, a.tpl_stride},
                                    FpmLevel{mb + b.dev_off, b.w, b.h, b.pitch, b.tpl_stride}, nullptr, T);
            if (rc) return rc;
            CK(cudaMemcpyAsync(dn.data(), mb + b.dev_off, dn.size(), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            std::vector<uint8_t>& m = mk[gi][l];
            m.resize(nb * T);
            for (int k = 0; k < T; k++) {
                size_t n = 0;
                for (int y = 0; y < b.h; y++)
                    for (int x = 0; x < b.w; x++) n += m[k * nb + (size_t)y * b.w + x] = dn[k * b.tpl_stride + (size_t)y * b.pitch + x] >= 128 ? 1 : 0;
                if (n == 0) {
                    const std::string lv = " keeps no pixel at pyramid level " + std::to_string(l) + " (" + std::to_string(b.w) + "x" +
                                           std::to_string(b.h) + "); enlarge the kept region or lower FPM_PARAM_MIN_REDUCE_AREA";
                    h->err = h->masked_set ? "fpm_learn_set_masked: the mask of template " + std::to_string(G.members[k]) + lv
                                           : "fpm_learn_masked: the mask" + lv;
                    return FPM_ERR_INVALID;
                }
            }
        }
    }
    std::vector<uint8_t> all(off);
    CK(cudaMemcpyAsync(all.data(), h->d_tpl.p, off, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::vector<FpmTplStat> stats(n_stat);
    for (size_t gi = 0; gi < gs.size(); gi++)
        for (size_t l = 0; l < gs[gi].tpl.size(); l++)
            for (size_t k = 0; k < gs[gi].members.size(); k++) {
                TplLevelHost& t = gs[gi].tpl[l];
                const uint8_t* base = all.data() + t.dev_off + k * t.tpl_stride;
                const uint8_t* m = gs[gi].masked ? mk[gi][l].data() + k * t.w * t.h : nullptr;
                unsigned long long S = 0, Q = 0, n = 0;
                for (int y = 0; y < t.h; y++)
                    for (int x = 0; x < t.w; x++) {
                        if (m && !m[(size_t)y * t.w + x]) continue;
                        const unsigned v = base[(size_t)y * t.pitch + x]; S += v; Q += (unsigned long long)v * v; n++;
                    }
                double N = (double)n;                              // the kept pixels (all of them without a mask)
                // cv::meanStdDev (u8): scale = 1/N; mean = S*scale; var = max(Q*scale - mean^2, 0); sdv = sqrt(var)
                double scale = 1.0 / N;
                double mean = (double)S * scale;
                double var = std::max((double)Q * scale - mean * mean, 0.0);
                double sdv = sqrt(var);
                double invArea = 1.0 / N;
                double templNorm = sdv * sdv;                       // :74
                const int equal1 = templNorm < DBL_EPSILON ? 1 : 0; // :77
                templNorm = sqrt(templNorm);                        // :85
                templNorm /= sqrt(invArea);                         // :86
                stats[t.stat_off + k] = FpmTplStat{mean, templNorm, invArea, equal1};
                t.all_flat = (k == 0 || t.all_flat) && equal1;
                if (k == 0) {
                    t.mean = mean; t.norm = templNorm; t.inv_area = invArea; t.equal1 = equal1;
                    t.pix.resize((size_t)t.w * t.h);
                    for (int y = 0; y < t.h; y++) memcpy(t.pix.data() + (size_t)y * t.w, base + (size_t)y * t.pitch, t.w);
                }
            }
    // masked groups: the correlation kernels see M_L * T_L of every member; the window sums walk the runs of kept pixels of
    // every row of the member's own mask
    std::vector<uint8_t> runs;
    for (size_t gi = 0; gi < gs.size(); gi++) {
        if (!gs[gi].masked) continue;
        for (size_t l = 0; l < gs[gi].tpl.size(); l++) {
            TplLevelHost& t = gs[gi].tpl[l];
            const size_t n = (size_t)t.w * t.h;
            t.mask.assign(mk[gi][l].begin(), mk[gi][l].begin() + n);
            t.n_kept = 0;
            std::vector<int> rows(1, 0), rr;
            for (size_t k = 0; k < gs[gi].members.size(); k++) {
                if (k) rows.push_back(rows.back());                // member k's h + 1 offsets start where member k - 1's end
                for (int y = 0; y < t.h; y++) {
                    const uint8_t* m = mk[gi][l].data() + k * n + (size_t)y * t.w;
                    uint8_t* px = all.data() + t.dev_off + k * t.tpl_stride + (size_t)y * t.pitch;
                    for (int x = 0; x < t.w; x++) {
                        if (!m[x]) px[x] = 0;
                        if (k == 0) t.n_kept += m[x];
                        if (m[x] && (x == 0 || !m[x - 1])) rr.push_back(x);
                        if (m[x] && (x == t.w - 1 || !m[x + 1])) rr.push_back(x + 1);
                    }
                    rows.push_back((int)rr.size() / 2);
                }
            }
            t.run_off = align_up(runs.size(), 16);
            t.run_data_off = align_up(t.run_off + rows.size() * sizeof(int), 16);
            runs.resize(t.run_data_off + rr.size() * sizeof(int));
            memcpy(runs.data() + t.run_off, rows.data(), rows.size() * sizeof(int));
            memcpy(runs.data() + t.run_data_off, rr.data(), rr.size() * sizeof(int));
        }
    }
    if (!runs.empty()) {
        CK(cudaMemcpy(h->d_tpl.p, all.data(), off, cudaMemcpyHostToDevice));
        CK(h->d_mruns.ensure(runs.size()));
        CK(cudaMemcpy(h->d_mruns.p, runs.data(), runs.size(), cudaMemcpyHostToDevice));
    }
    CK(h->d_tsh.ensure(toff));
    for (const TplGroup& G : gs) {
        if (G.members.size() != 1) continue;
        for (const TplLevelHost& t : G.tpl) {
            dim3 g((t.bpitch + 127) / 128, t.h, 8);
            fpm_shift_template_kernel<<<g, 128, 0, h->stream>>>(h->d_tpl.as<uint8_t>() + t.dev_off, t.w, t.h, t.pitch,
                                                                h->d_tsh.as<uint8_t>() + t.tsh_off, t.bpitch);
            CKL();
        }
    }
    CK(h->d_tstat.ensure(n_stat * sizeof(FpmTplStat)));
    CK(cudaMemcpy(h->d_tstat.p, stats.data(), n_stat * sizeof(FpmTplStat), cudaMemcpyHostToDevice));
    std::vector<int> members;
    for (const TplGroup& G : gs) members.insert(members.end(), G.members.begin(), G.members.end());
    CK(h->d_members.ensure(members.size() * sizeof(int)));
    CK(cudaMemcpy(h->d_members.p, members.data(), members.size() * sizeof(int), cudaMemcpyHostToDevice));
    // group 0 goes into the handle's fields (its plan buffers stay the handle's), the others wait in groups[1..]
    TplGroup& G0 = gs[0];
    h->tpl.swap(G0.tpl); h->members.swap(G0.members);
    h->border = G0.border; h->tpl0_w = G0.w0; h->tpl0_h = G0.h0;
    h->groups.swap(gs);
    h->learned = true;
    h->learned_mra = h->min_reduce_area;
    h->plan.valid = false;
    return FPM_OK;
}

// runs group g's pass with its state in the handle's fields, then puts it back
struct GroupScope {
    fpm_handle* h; size_t g;
    static void swap(fpm_handle* h, TplGroup& G)
    {
        std::swap(h->tpl, G.tpl); std::swap(h->members, G.members); std::swap(h->border, G.border);
        std::swap(h->tpl0_w, G.w0); std::swap(h->tpl0_h, G.h0); std::swap(h->plan, G.plan);
        std::swap(h->d_jobs_top, G.d_jobs_top); std::swap(h->d_angles, G.d_angles);
        std::swap(h->d_ftx, G.d_ftx); std::swap(h->d_fty, G.d_fty); std::swap(h->d_scales, G.d_scales);
    }
    GroupScope(fpm_handle* hh, size_t gg) : h(hh), g(gg) { if (g) swap(h, h->groups[g]); }
    ~GroupScope() { if (g) swap(h, h->groups[g]); }
};

// ---- source pyramid -----------------------------------------------------------------
int build_pyramid(fpm_handle* h, const uint8_t* d_src, int batch, int w, int hgt, int stride, size_t frame_stride, int top)
{
    if (h->shared_levels) {                                    // multi-template matching: one upload, one pyramid for all handles
        if (h->shared_levels != &h->levels) h->levels.assign(h->shared_levels->begin(), h->shared_levels->begin() + top + 1);
        return FPM_OK;
    }
    h->levels.assign(top + 1, FpmLevel());
    h->levels[0] = FpmLevel{const_cast<uint8_t*>(d_src), w, hgt, stride, frame_stride};
    size_t off = 0;
    int lw = w, lh = hgt;
    std::vector<size_t> offs(top + 1, 0);
    for (int l = 1; l <= top; l++) {
        lw = (lw + 1) / 2; lh = (lh + 1) / 2;
        int pitch = (int)align_up(lw, 128);
        size_t img = align_up((size_t)pitch * lh, 256);
        h->levels[l] = FpmLevel{nullptr, lw, lh, pitch, img};
        offs[l] = off;
        off += img * batch;
    }
    CK(h->d_pyr.ensure(off + 256));
    for (int l = 1; l <= top; l++) h->levels[l].ptr = h->d_pyr.as<uint8_t>() + offs[l];
    return launch_pyramid_chain(h, h->levels, top, batch);
}

// ---- angle schedule + per-angle top-layer geometry (src/TemplateMatcher.cpp:130-173) -----
void angle_schedule(const fpm_handle* h, int top, std::vector<double>& angles)
{
    const TplLevelHost& t = h->tpl[top];
    double dAngleStep = atan(2.0 / std::max(t.w, t.h)) * FPM_R2D;
    angles.clear();
    if (h->tol_range) {                                       // MatchTool/MatchToolDlg.cpp:805-816
        for (double a = h->tol_r[0]; a < h->tol_r[1] + dAngleStep; a += dAngleStep) angles.push_back(a);
        for (double a = h->tol_r[2]; a < h->tol_r[3] + dAngleStep; a += dAngleStep) angles.push_back(a);
    } else if (h->tol_angle < FPM_VISION_TOLERANCE) {
        angles.push_back(0.0);
    } else {
        for (double a = 0; a < h->tol_angle + dAngleStep; a += dAngleStep) angles.push_back(a);
        for (double a = -dAngleStep; a > -h->tol_angle - dAngleStep; a -= dAngleStep) angles.push_back(a);
    }
}

// Scale schedule of the range [lo, hi] for a top template level of w x h: {lo} when lo == hi, else n geometric steps of at most
// 1 + ds, ds = 2 / max(w, h) (the template's far edge moves by about 2 px, like the angle step atan(2 / max(w, h))), ending
// exactly at hi
void scale_schedule(double lo, double hi, int w, int h, std::vector<double>& out)
{
    out.clear();
    if (lo == hi) { out.push_back(lo); return; }
    const double ds = 2.0 / std::max(w, h), r = log(hi / lo);
    const int n = (int)ceil(r / log1p(ds)) + 1;
    for (int k = 0; k < n - 1; k++) out.push_back(lo * exp(k * r / (n - 1)));
    out.push_back(hi);
}

// The plan always covers the whole schedule (a few dozen doubles per angle); a partial sweep (stage API, angle-sharded
// mode) runs a sub-range of its job list, so a cached plan can never truncate a later full sweep.
int make_top_plan(fpm_handle* h, int top, int batch)
{
    const FpmLevel& L = h->levels[top];
    TopPlan& p = h->plan;
    if (p.valid && p.sw == L.w && p.sh == L.h && p.top == top && p.batch == batch && p.tol == h->tol_angle &&
        p.scale_min == h->scale_min && p.scale_max == h->scale_max)
        return FPM_OK;
    p.valid = false;
    const TplLevelHost& t = h->tpl[top];
    std::vector<double> ang1, sc;
    angle_schedule(h, top, ang1);
    scale_schedule(h->scale_min, h->scale_max, t.w, t.h, sc);
    p.angles.clear(); p.scales.clear();
    for (double s : sc)
        for (double a : ang1) { p.angles.push_back(a); p.scales.push_back(s); }
    p.sw = L.w; p.sh = L.h; p.top = top; p.batch = batch; p.tol = h->tol_angle; p.scale_min = h->scale_min; p.scale_max = h->scale_max;
    p.n_ang = (int)p.angles.size();
    float cx = (L.w - 1) / 2.0f, cy = (L.h - 1) / 2.0f;
    std::vector<FpmWarpJob> jobs((size_t)batch * std::max(p.n_ang, 1));
    p.ftx.assign(p.n_ang, 0.f); p.fty.assign(p.n_ang, 0.f);
    p.maxW = p.maxH = 1;
    for (int a = 0; a < p.n_ang; a++) {
        // scale s: the canvas resamples the level by 1/s around its centre (getRotationMatrix2D(c, angle, 1/s)) and is sized for
        // the resampled level, cvRound(w / s) x cvRound(h / s)
        const double s = p.scales[a];
        const int rsw = s == 1.0 ? L.w : (int)lrint(L.w / s), rsh = s == 1.0 ? L.h : (int)lrint(L.h / s);
        FpmWarpJob jb;
        fpm_rotation_matrix(cx, cy, p.angles[a], jb.m, 1.0 / s);
        int bw, bh;
        best_rotation_size(rsw, rsh, t.w, t.h, p.angles[a], &bw, &bh);
        float fTx = (bw - 1) / 2.0f - cx, fTy = (bh - 1) / 2.0f - cy;
        jb.m[2] += (double)fTx; jb.m[5] += (double)fTy;
        fpm_invert_affine(jb.m);
        jb.dw = bw; jb.dh = bh; jb.valid = (bw > 0 && bh > 0) ? 1 : 0;
        p.ftx[a] = fTx; p.fty[a] = fTy;
        p.maxW = std::max(p.maxW, bw); p.maxH = std::max(p.maxH, bh);
        for (int b = 0; b < batch; b++) { jb.src_img = b; jobs[(size_t)b * p.n_ang + a] = jb; }
    }
    if (p.n_ang > 0) {
        CK(h->d_jobs_top.ensure(jobs.size() * sizeof(FpmWarpJob)));
        CK(cudaMemcpyAsync(h->d_jobs_top.p, jobs.data(), jobs.size() * sizeof(FpmWarpJob), cudaMemcpyHostToDevice, h->stream));
        CK(h->d_angles.ensure(p.n_ang * sizeof(double)));
        CK(cudaMemcpyAsync(h->d_angles.p, p.angles.data(), p.n_ang * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(h->d_scales.ensure(p.n_ang * sizeof(double)));
        CK(cudaMemcpyAsync(h->d_scales.p, p.scales.data(), p.n_ang * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(h->d_ftx.ensure(p.n_ang * sizeof(float)));
        CK(h->d_fty.ensure(p.n_ang * sizeof(float)));
        CK(cudaMemcpyAsync(h->d_ftx.p, p.ftx.data(), p.n_ang * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_fty.p, p.fty.data(), p.n_ang * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));   // jobs is a local vector
    }
    p.valid = true;
    return FPM_OK;
}

// threshold of the top layer, vecLayerScore[top] = Score * 0.9^top (src/TemplateMatcher.cpp:153-156)
double top_layer_threshold(const fpm_handle* h, int top)
{
    double t = h->score;
    for (int l = 0; l < top; l++) t *= 0.9;
    return t;
}

// Scores certainly below the top-layer threshold may be stored as estimates (fpm_ccoeff_epilogue_top): the peak
// search cannot observe them.  Off (exact everywhere) when the threshold is not comfortably positive.
float top_reject_below(const fpm_handle* h, int top)
{
    const double t = top_layer_threshold(h, top);
    return t > 0.05 ? (float)(t - 0.01) : -INFINITY;
}

// ---- top-layer sweep: warp + score + peaks for jobs [j0, j0 + nj) of the plan's (frame, angle) list -----
// Each (frame, angle) canvas is warped once and scored against every template of the group.  picks go to
// picks_out[slot][max_picks], counts to cnt_out[slot]: slot = job - j0 for one template, (frame * n_tpl + template) *
// row_angles + angle for a group, with row_angles = the whole schedule (0) for whole sweeps and the chunk for the
// angle-sharded sweep of one frame (jobs [j0, j0 + nj), nj <= row_angles).  The sweep runs in chunks of canvases whose n_tpl
// score maps each fit FPM_PARAM_WORKSPACE_MB and whose jobs fit gridDim.y / gridDim.z.
int run_top(fpm_handle* h, int top, int j0, int nj, FpmPick* picks_out, int* cnt_out, int row_angles = 0)
{
    TopPlan& p = h->plan;
    const int max_picks = h->max_pos + FPM_MATCH_CANDIDATE_NUM;
    if (nj <= 0) return FPM_OK;
    const TplLevelHost& t = h->tpl[top];
    const int n_tpl = std::max((int)h->members.size(), 1);
    const int rpitch = (int)align_up(p.maxW, 16);
    const size_t rot_stride = (size_t)rpitch * p.maxH;
    const int maxRW = std::max(p.maxW - t.w + 1, 1), maxRH = std::max(p.maxH - t.h + 1, 1);
    const int spitch = (int)align_up(maxRW, 4);
    const size_t score_stride = (size_t)spitch * maxRH;
    const FpmWarpJob* jobs = h->d_jobs_top.as<FpmWarpJob>() + j0;
    const int kMaxGridYZ = 65535;                              // gridDim.y / gridDim.z limit: larger sweeps run in chunks
    const size_t budget = (size_t)(h->workspace_mb * 1024.0 * 1024.0);
    const int chunk = (int)std::min<size_t>({(size_t)kMaxGridYZ, (size_t)nj,
                                             std::max<size_t>(1, budget / ((size_t)n_tpl * score_stride * sizeof(float)))});
    CK(h->d_rot.ensure(rot_stride * chunk));
    CK(h->d_score.ensure(score_stride * chunk * n_tpl * sizeof(float)));
    const bool masked = !t.mask.empty();
    const size_t smem_ts = top_score_smem(t.w, t.h, masked);
    if (smem_ts > 200 * 1024) { h->err = "top-layer template too large for the score kernel"; return FPM_ERR_LIMIT; }
    const auto score_kernel = n_tpl > 1 ? (masked ? fpm_top_score_kernel<true, true> : fpm_top_score_kernel<true>)
                                        : (masked ? fpm_top_score_kernel<false, true> : fpm_top_score_kernel<false>);
    if (smem_ts > 48 * 1024) CK(ensure_dyn_smem((const void*)score_kernel, h->device, smem_ts));
    // bCalMaxByBlock, src/TemplateMatcher.cpp:158-159
    const FpmLevel& L = h->levels[top];
    const bool by_block = ((L.w * L.h) / (t.w * t.h) > 500) && h->max_pos > 10;
    const int mode = by_block ? (h->mfc_compat ? 2 : 1) : 0;    // MFC s_BlockMax differs from the Qt port's (MatchToolDlg.h:109-213)
    int tile = 8;
    while ((long long)((maxRW + tile - 1) / tile) * ((maxRH + tile - 1) / tile) > 1024 && tile < 256) tile *= 2;
    int blk_stride;
    const int tiles0 = ((maxRW + tile - 1) / tile) * ((maxRH + tile - 1) / tile);
    if (mode == 1) blk_stride = (maxRW / t.w) * (maxRH / t.h) + 3;
    else if (mode == 2) blk_stride = std::max((maxRW / (2 * t.w)) * (maxRH / (2 * t.h)) + 2, tiles0);   // an empty MFC table falls back to tiles
    else blk_stride = tiles0;
    blk_stride = std::max(blk_stride, 1);
    if (blk_stride > PK_SUP_MAX * 32) { h->err = "top-layer score map has too many blocks for the peak table"; return FPM_ERR_LIMIT; }
    CK(h->d_blkv.ensure((size_t)chunk * n_tpl * blk_stride * sizeof(float)));
    CK(h->d_blkl.ensure((size_t)chunk * n_tpl * blk_stride * sizeof(int)));
    const double thresh = top_layer_threshold(h, top);
    const int smem_blocks = peaks_smem_blocks(h, blk_stride);
    if (smem_blocks < 0) return FPM_ERR_CUDA;
    for (int c0 = 0; c0 < nj; c0 += chunk) {
        const int nc = std::min(chunk, nj - c0);
        const int tiles_x = (rpitch + WA_TW - 1) / WA_TW;
        dim3 wgrid(tiles_x * ((p.maxH + WA_TH - 1) / WA_TH), nc);
        KL(K_WARP_TOP, 2.0 * nc * (double)p.maxW * p.maxH,
           fpm_warp_kernel<<<wgrid, WA_THREADS, 0, h->stream>>>(jobs + c0, 1, h->levels[top], h->d_rot.as<uint8_t>(), rpitch, rot_stride,
                                                                h->border, tiles_x, level_vec_ok(h->levels[top]), nullptr, FpmRefineGeom{}));
        dim3 grid((maxRW + TS_TW - 1) / TS_TW, (maxRH + TS_TH - 1) / TS_TH, nc);
        dim3 block(TS_THREADS);
        KL(masked ? K_TOP_SCORE_MASKED : K_TOP_SCORE, (double)nc * n_tpl * maxRW * maxRH * t.w * t.h,      // MACs
           score_kernel<<<grid, block, smem_ts, h->stream>>>(jobs + c0, h->d_rot.as<uint8_t>(), rpitch, rot_stride,
                                                                     tpl_level_dev(h, top), h->d_score.as<float>(), spitch,
                                                                     score_stride, top_reject_below(h, top)));
        KL(K_TOP_PEAKS, 4.0 * nc * n_tpl * maxRW * maxRH,
           fpm_top_peaks_kernel<<<nc * n_tpl, (maxRW * maxRH <= 16384) ? 128 : PK_THREADS, (size_t)smem_blocks * 8, h->stream>>>(
               jobs, h->d_score.as<float>(), spitch, score_stride, t.w, t.h, mode, tile,
               h->d_blkv.as<float>(), h->d_blkl.as<int>(), blk_stride, thresh, h->max_overlap, max_picks,
               picks_out, cnt_out, smem_blocks, c0, n_tpl, row_angles ? row_angles : p.n_ang));
    }
    return FPM_OK;
}

// ---- refinement of a flat candidate list held in d_cand[0] ------------------------------
// per-layer geometry and workspace of the refinement
struct RefineLayer {
    int rpitch; size_t roi_stride; bool warp_fused; size_t per_eval; double step;
};
RefineLayer refine_layer(const fpm_handle* h, int layer, int n_ang)
{
    const TplLevelHost& t = h->tpl[layer];
    const FpmLevel& L = h->levels[layer];
    RefineLayer r;
    r.step = atan(2.0 / std::max(t.w, t.h)) * FPM_R2D;
    r.rpitch = (int)align_up(t.w + FPM_ROI_PAD, 16) + 16;
    r.roi_stride = (size_t)r.rpitch * (t.h + FPM_ROI_PAD);
    // bytes per eval of one wave: ROI patch, window row sums, job record, and the row dots in the layout of the
    // correlation path this level can take (dp4a [h][49], row-split tensor-core raw[h+6][64], or the fused kernel's
    // 64 numerators + 14 window totals)
    r.warp_fused = corr_warp_usable(h, t.w, n_ang, L);
    r.per_eval = (r.warp_fused ? 0 : r.roi_stride) + 2 * (size_t)(t.h + FPM_ROI_PAD) * FPM_WSTRIDE * 4 + sizeof(FpmWarpJob);
    if (mma_usable(h, t.w) || mma_narrow_fused(h, t.w))
        r.per_eval += std::max((size_t)(t.h + FPM_ROI_PAD) * MM_N * 4, (size_t)MM_N * 4 + 2 * FPM_NSHIFT * 8);
    if (!mma_usable(h, t.w)) r.per_eval += (size_t)t.h * FPM_NCELL * 4;
    if (!t.mask.empty()) r.per_eval += 2 * FPM_NCELL * sizeof(long long);   // masked window sums
    return r;
}

// ---- refinement of a flat candidate list held in d_cand[0] ------------------------------
// Two ways to walk down the pyramid (src/TemplateMatcher.cpp:279-368):
//   * with a counter read-back per layer (grids sized to the live candidates; workspace waves; tracing), or
//   * without any host round trip (single-frame latency): every layer is enqueued at once with grids sized to the
//     TOP-layer candidate count -- the list can only shrink -- and every kernel reads the live count of its layer from
//     device memory (counters[CNT_LAYER + layer]); surplus CTAs leave at once.
int run_refine(fpm_handle* h, int top, int n_cands, int* n_refined_out)
{
    int* counters = h->d_counters.as<int>();
    int* hc = h->h_counts.as<int>();
    FpmRefined* ref_out = h->ref_out;
    int* ref_cnt = h->ref_cnt ? h->ref_cnt : counters + CNT_REFINED;
    if (!ref_out) {
        CK(h->d_refined.ensure((size_t)std::max(n_cands, 1) * sizeof(FpmRefined)));
        ref_out = h->d_refined.as<FpmRefined>();
    }
    CK(cudaMemsetAsync(ref_cnt, 0, sizeof(int), h->stream));
    *n_refined_out = 0;
    if (n_cands == 0) return FPM_OK;
    const int stop = h->stop_layer1 ? 1 : 0;                  // iStopLayer, MatchToolDlg.cpp:936
    if (top <= stop) {
        fpm_cands_to_refined_kernel<<<(n_cands + 255) / 256, 256, 0, h->stream>>>(h->d_cand[0].as<FpmCand>(), n_cands, top,
                                                                               ref_out, ref_cnt);
        CKL();
        *n_refined_out = n_cands;
        return FPM_OK;
    }
    const int n_ang = (!h->tol_range && h->tol_angle < FPM_VISION_TOLERANCE) ? 1 : 3;
    // a scale range refines the scale too: evals k * n_ang + j over the scales s / (1 + ds_L), s, s * (1 + ds_L)
    const int n_sc = h->scale_min != h->scale_max ? 3 : 1, n_ev = n_sc * n_ang;
    CK(h->d_cand[1].ensure((size_t)n_cands * sizeof(FpmCand)));
    int cur = 0, n = n_cands;
    double layer_score[FPM_MAX_LEVELS + 1];
    layer_score[0] = h->score;
    for (int l = 1; l <= top; l++) layer_score[l] = layer_score[l - 1] * 0.9;
    if (h->trace) {
        h->tr_evals.assign(top + 1, std::vector<double>());
        h->tr_scores.assign(top + 1, std::vector<float>());
        h->tr_rois.assign(top + 1, fpm_handle::TraceRois());
    }
    const size_t budget = (size_t)(h->workspace_mb * 1024.0 * 1024.0);
    // the descent without host round trips needs every layer to fit one workspace wave at the top-layer count
    bool async = !h->trace && n_cands * n_sc <= 65535 && (h->async_descent == 1 || (h->async_descent < 0 && h->cur_batch < 8));
    for (int layer = top - 1; layer >= stop && async; layer--)
        if (refine_layer(h, layer, n_ang).per_eval * n_ev * (size_t)n_cands > budget) async = false;
    if (async) CK(cudaMemsetAsync(counters + CNT_LAYER, 0, FPM_MAX_LEVELS * sizeof(int), h->stream));
    for (int layer = top - 1; layer >= stop && n > 0; layer--) {
        const TplLevelHost& t = h->tpl[layer];
        const FpmLevel& L = h->levels[layer];
        const RefineLayer rl = refine_layer(h, layer, n_ang);
        const double step = rl.step;
        const int rpitch = rl.rpitch;
        const size_t roi_stride = rl.roi_stride;
        const bool warp_fused = rl.warp_fused;
        const double scale_step = 2.0 / std::max(t.w, t.h);
        int wave_cands = (int)std::max<size_t>(1, budget / (rl.per_eval * n_ev));
        wave_cands = std::min(wave_cands, n);
        wave_cands = std::min(wave_cands, 65535 / n_sc);      // one (candidate, scale) per gridDim.y slot of the ROI warp
        const int wave_evals = wave_cands * n_ev;
        CK(h->d_jobs_ref.ensure((size_t)wave_evals * sizeof(FpmWarpJob)));
        if (!warp_fused) CK(h->d_roi.ensure(roi_stride * wave_evals));
        if (!mma_usable(h, t.w)) CK(h->d_rowsum.ensure((size_t)wave_evals * t.h * FPM_NCELL * 4));
        CK(h->d_rowS.ensure((size_t)wave_evals * (t.h + FPM_ROI_PAD) * FPM_WSTRIDE * 4));
        CK(h->d_rowQ.ensure((size_t)wave_evals * (t.h + FPM_ROI_PAD) * FPM_WSTRIDE * 4));
        if (h->trace) {
            CK(h->d_trace.ensure((size_t)n * n_ev * sizeof(FpmEvalTrace)));
            CK(cudaMemsetAsync(h->d_trace.p, 0, (size_t)n * n_ev * sizeof(FpmEvalTrace), h->stream));
            // all-ones bytes are NaN: a score cell the finalize kernel does not write cannot pass for a result
            CK(h->d_trace_sc.ensure((size_t)n * n_ev * FPM_NCELL * sizeof(float)));
            CK(cudaMemsetAsync(h->d_trace_sc.p, 0xff, (size_t)n * n_ev * FPM_NCELL * sizeof(float), h->stream));
            fpm_handle::TraceRois& tr = h->tr_rois[layer];
            tr.w = t.w + FPM_ROI_PAD; tr.h = t.h + FPM_ROI_PAD; tr.pitch = rpitch;
            tr.px.assign(warp_fused ? 0 : (size_t)n * n_ev * roi_stride, 0);
        }
        // live candidates of this layer / where the survivors are counted
        const int* n_dev = !async ? nullptr : (layer == top - 1 ? counters + CNT_FLAT : counters + CNT_LAYER + layer);
        int* next_cnt = !async ? counters + CNT_NEXT : counters + CNT_LAYER + std::max(layer - 1, 0);
        if (!async) CK(cudaMemsetAsync(counters + CNT_NEXT, 0, sizeof(int), h->stream));
        const int n_tpl = std::max((int)h->members.size(), 1);
        const CorrCfg cc = corr_config(t.h, n_tpl > 1);
        const size_t smem = cc.smem;
        if (smem > 200 * 1024) { h->err = "correlation kernel shared memory limit"; return FPM_ERR_LIMIT; }
        if (smem > 48 * 1024)
            CK(ensure_dyn_smem((const void*)fpm_corr_rows_kernel, h->device, smem));
        const FpmTplLevel td = tpl_level_dev(h, layer);
        const FpmCand* cands = h->d_cand[cur].as<FpmCand>();
        for (int c0 = 0; c0 < n; c0 += wave_cands) {
            const int nc = std::min(wave_cands, n - c0);
            const int ne = nc * n_ev;
            if (warp_fused)                                 // the warp-fused kernel stages the job matrices of its 42 candidates itself
                KL(K_PREP, (double)ne * sizeof(FpmWarpJob),
                   fpm_refine_prep_kernel<<<(ne + 127) / 128, 128, 0, h->stream>>>(cands + c0, nc, n_ang, step, L.w, L.h, t.w, t.h,
                                                                                 h->d_jobs_ref.as<FpmWarpJob>(), n_dev, n_tpl));
            int raw_epad = 0;                               // 0 = [e][tr][49] row sums, else raw[y][e_pad][64] from the tensor cores
            int raw_tile_evals = 0;                         // evals per 128-row tile of raw (0 = contiguous)
            bool fused = false;                             // numerators + window totals straight from the fused tensor-core kernel
            if (warp_fused) {
                // the ROI patches are produced inside the correlation kernel and never reach HBM
                int rcm = launch_corr_warp(h, L, h->d_jobs_ref.as<FpmWarpJob>(), h->d_tsh.as<uint8_t>() + t.tsh_off, t.bpitch, t.w, t.h, nc,
                                           &raw_epad, h->d_rowS.as<int32_t>(), h->d_rowQ.as<int32_t>(), n_dev);
                if (rcm) return rcm;
                raw_tile_evals = FW_TILE_EVALS;
            } else {
                const int wtiles_x = (rpitch + WA_TW - 1) / WA_TW;
                dim3 wgrid(wtiles_x * ((t.h + FPM_ROI_PAD + WA_TH - 1) / WA_TH), nc * n_sc);   // one CTA = one tile of the n_ang ROIs of a (candidate, scale)
                // algorithmic bytes: 1 B gathered + 1 B written per ROI pixel (SURVEY 8d)
                // which correlation kernel will read the patches (the one-CTA-per-128-evals kernel only pays for many LIVE evals:
                // never with an upper-bound count)
                const bool go_fused = (mma_narrow_fused(h, t.w) || (mma_usable(h, t.w) && h->use_simd && h->use_tc != 3)) &&
                                      (!async || h->use_tc == 4) &&
                                      fused_pays(ne, t.h + FPM_ROI_PAD, rpitch, t.w + FPM_ROI_PAD, h->use_tc, h->num_sms);
                KL(K_WARP_ROI, 2.0 * ne * (double)(t.w + FPM_ROI_PAD) * (t.h + FPM_ROI_PAD),
                   fpm_warp_kernel<<<wgrid, WA_THREADS, 0, h->stream>>>(nullptr, n_ang, L,
                                                                        h->d_roi.as<uint8_t>(), rpitch, roi_stride, 0, wtiles_x,
                                                                        level_vec_ok(L), n_dev,
                                                                        FpmRefineGeom{cands + c0, n_ang, n_sc, step, scale_step, L.w, L.h, t.w, t.h, n_tpl}));
                if (go_fused) {
                    int rcm = launch_corr_fused(h, h->d_roi.as<uint8_t>(), rpitch, roi_stride, h->d_tsh.as<uint8_t>() + t.tsh_off, t.bpitch,
                                                t.w, t.h, ne, h->d_rowS.as<int32_t>(), h->d_rowQ.as<int32_t>(), n_dev, n_ev);
                    if (rcm) return rcm;
                    fused = true;
                } else if (mma_usable(h, t.w)) {
                    int rcm = launch_corr_mma(h, h->d_roi.as<uint8_t>(), rpitch, roi_stride, h->d_tsh.as<uint8_t>() + t.tsh_off, t.bpitch,
                                              t.w, t.h, ne, &raw_epad, h->d_rowS.as<int32_t>(), h->d_rowQ.as<int32_t>(), n_dev, n_ev);
                    if (rcm) return rcm;
                } else {
                    dim3 cgrid(cc.blocks_y_rows, (ne + cc.evals_per_cta - 1) / cc.evals_per_cta);
                    // algorithmic MACs: 49 * w * h per eval (SURVEY 8d)
                    KL(K_CORR, (double)ne * FPM_NCELL * (double)t.w * t.h,
                       fpm_corr_rows_kernel<<<cgrid, cc.threads, smem, h->stream>>>(h->d_roi.as<uint8_t>(), rpitch, roi_stride, td, ne,
                                                                                    cc.rb, cc.evals_per_cta, h->d_rowsum.as<int32_t>(),
                                                                                    h->d_rowS.as<int32_t>(), h->d_rowQ.as<int32_t>(), n_dev, n_ev,
                                                                                    cands + c0));
                }
            }
            const bool masked = td.mrun && !t.all_flat;      // finalize reads the sums of the members that are not flat
            if (masked) {
                int rcm = launch_mask_window(h, rpitch, roi_stride, td, ne, n_dev, n_ev, cands + c0);
                if (rcm) return rcm;
            }
            {
                auto fin = n_tpl > 1 ? fpm_refine_finalize_kernel<true> : fpm_refine_finalize_kernel<false>;
                KL(K_FINALIZE, (double)ne * ((double)t.h * FPM_NCELL * 4 + 2.0 * (t.h + FPM_ROI_PAD) * FPM_NSHIFT * 4),
                   fin<<<nc, RF_THREADS, 0, h->stream>>>(
                       cands + c0, n_ang, step, raw_epad ? h->d_raw.as<int32_t>() : h->d_rowsum.as<int32_t>(), raw_epad,
                       h->d_rowS.as<int32_t>(), h->d_rowQ.as<int32_t>(), td, L.w,
                       L.h, layer_score[layer], h->use_simd, layer == stop ? 1 : 0, stop ? 2 : 1, (h->subpixel && layer == 0) ? 1 : 0,
                       h->d_cand[cur ^ 1].as<FpmCand>(),
                       next_cnt, ref_out, ref_cnt,
                       h->trace ? h->d_trace.as<FpmEvalTrace>() + (size_t)c0 * n_ev : nullptr,
                       h->trace ? h->d_trace_sc.as<float>() + (size_t)c0 * n_ev * FPM_NCELL : nullptr,
                       fused ? h->d_numer.as<float>() : nullptr, (masked ? h->d_mwS : h->d_totS).as<long long>(),
                       (masked ? h->d_mwQ : h->d_totQ).as<long long>(), raw_tile_evals, n_dev, n_sc, scale_step));
            }
            if (h->trace && !warp_fused)                    // this wave's ROI patches, before the next wave overwrites them
                CK(cudaMemcpyAsync(h->tr_rois[layer].px.data() + (size_t)c0 * n_ev * roi_stride, h->d_roi.p, (size_t)ne * roi_stride,
                                   cudaMemcpyDeviceToHost, h->stream));
        }
        cur ^= 1;
        if (async) continue;                                  // n stays the top-layer count: an upper bound of every layer's list
        CK(cudaMemcpyAsync(hc, counters, CNT_N * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (h->trace) {
            const FpmCand* cands_done = h->d_cand[cur ^ 1].as<FpmCand>();
            std::vector<FpmEvalTrace> tr((size_t)n * n_ev);
            std::vector<FpmCand> cc2(n);
            CK(cudaMemcpy(tr.data(), h->d_trace.p, tr.size() * sizeof(FpmEvalTrace), cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(cc2.data(), cands_done, cc2.size() * sizeof(FpmCand), cudaMemcpyDeviceToHost));
            std::vector<double>& rows = h->tr_evals[layer];
            for (int i = 0; i < n; i++)
                for (int j = 0; j < n_ev; j++) {
                    const FpmEvalTrace& e = tr[(size_t)i * n_ev + j];
                    rows.push_back(cc2[i].id); rows.push_back(e.angle); rows.push_back(e.score);
                    rows.push_back(e.locx); rows.push_back(e.locy);
                }
            std::vector<float>& sc = h->tr_scores[layer];
            sc.resize((size_t)n * n_ev * FPM_NCELL);
            CK(cudaMemcpy(sc.data(), h->d_trace_sc.p, sc.size() * sizeof(float), cudaMemcpyDeviceToHost));
        }
        if (hc[CNT_ERR]) { h->err = "fpm_corr_warp_kernel: source box larger than its staging buffer"; return FPM_ERR_LIMIT; }
        n = (layer == stop) ? 0 : hc[CNT_NEXT];
        *n_refined_out = hc[CNT_REFINED];
    }
    if (async) h->err_check_pending = true;                   // CNT_ERR is read back together with the results
    return FPM_OK;
}

// merged set results of one sub-batch (fpm_match_set_batch_merged): every group's fpm_final_kernel leaves its lists on the
// device, frame b / set index t at lists + (b * n_set + t) * lcap with its count at counts[b * n_set + t], for
// fpm_set_merge_kernel
struct MergeDev {
    FpmResultDev* lists = nullptr;
    int* counts = nullptr;
    int lcap = 0;
    int ocap = 0;                  // merged records per frame in d_merged: min(cap, n_set * lcap), a merged list never exceeds its inputs
    const int* rows = nullptr;     // the current group's members (d_members)
    int* err = nullptr;            // the current group's slot for CNT_ERR (read back with the merged results)
};

// ---- final stage: filterWithScore + NMS + conversion, results to host ---------------------
// n_set > 1: image v of the batch is frame v / n_tpl x member v % n_tpl of the current group, written to the caller's
// [frame][set index][cap] layout, or (md) to the device lists of the merge
int run_final(fpm_handle* h, int batch, const FpmRefinedView& rv, int key_stride, fpm_result* out, int cap, int* n_out, int n_set = 1,
              const MergeDev* md = nullptr)
{
    key_stride = std::max(key_stride, 1);
    int ks = 1;
    while (ks < key_stride) ks <<= 1;
    CK(h->d_keys.ensure((size_t)batch * ks * sizeof(unsigned long long)));
    CK(h->d_rects.ensure((size_t)batch * ks * sizeof(FpmRRect)));
    CK(h->d_del.ensure((size_t)batch * ks * sizeof(int)));
    CK(h->d_idmap.ensure((size_t)batch * ks * sizeof(int)));
    const int pair_cap = std::min(ks, 512);                 // all-pairs NMS matrix for up to 512 survivors per frame
    CK(h->d_pairs.ensure((size_t)batch * pair_cap * pair_cap));
    const int rcap = std::max(cap, 1);
    if (!md) {
        CK(h->d_results.ensure((size_t)batch * rcap * sizeof(FpmResultDev)));
        CK(h->d_rescnt.ensure((size_t)batch * sizeof(int)));
        CK(h->h_results.ensure((size_t)batch * rcap * sizeof(FpmResultDev) + (size_t)batch * sizeof(int)));
    }
    const int n_tpl = std::max((int)h->members.size(), 1);
    // NMS rectangle size: pyramid[iStopLayer] * (iStopLayer == 0 ? 1 : 2)  (src/TemplateMatcher.cpp:376-377)
    const int stop_l = std::min(h->stop_layer1 ? 1 : 0, (int)h->tpl.size() - 1);
    const int nms_w = h->tpl[stop_l].w * (h->stop_layer1 ? 2 : 1), nms_h = h->tpl[stop_l].h * (h->stop_layer1 ? 2 : 1);
    KL(K_FINAL, 0,
       fpm_final_kernel<<<batch, FN_THREADS, 0, h->stream>>>(rv, h->score,
                                                             h->max_overlap, nms_w, nms_h, h->tpl[0].w, h->tpl[0].h,
                                                             h->d_keys.as<unsigned long long>(), ks, h->d_rects.as<FpmRRect>(),
                                                             h->d_del.as<int>(), h->d_idmap.as<int>(),
                                                             h->d_pairs.as<unsigned char>(), pair_cap, h->mfc_compat, h->max_pos,
                                                             md ? md->lists : h->d_results.as<FpmResultDev>(),
                                                             md ? md->lcap : rcap, md ? md->counts : h->d_rescnt.as<int>(),
                                                             md ? md->rows : nullptr, n_tpl, n_set));
    if (md) {                                                 // no copy, no synchronise: the merge reads the lists
        if (h->err_check_pending)
            CK(cudaMemcpyAsync(md->err, h->d_counters.as<int>() + CNT_ERR, sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
        h->err_check_pending = false;
        return FPM_OK;
    }
    FpmResultDev* hr = h->h_results.as<FpmResultDev>();
    int* hn = reinterpret_cast<int*>(hr + (size_t)batch * rcap);
    int* hc = h->h_counts.as<int>();
    const bool check_err = h->err_check_pending && hc;
    h->err_check_pending = false;
    if (check_err) CK(cudaMemcpyAsync(hc + CNT_ERR, h->d_counters.as<int>() + CNT_ERR, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(hn, h->d_rescnt.p, (size_t)batch * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(hr, h->d_results.p, (size_t)batch * rcap * sizeof(FpmResultDev), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (check_err && hc[CNT_ERR]) { h->err = "fpm_corr_warp_kernel: source box larger than its staging buffer"; return FPM_ERR_LIMIT; }
    for (int b = 0; b < batch; b++) {
        const size_t slot = n_set == 1 ? (size_t)b : (size_t)(b / n_tpl) * n_set + h->members[b % n_tpl];
        n_out[slot] = hn[b];
        int m = std::min(hn[b], cap);
        for (int i = 0; i < m; i++) {
            const FpmResultDev& r = hr[(size_t)b * rcap + i];
            fpm_result& o = out[slot * cap + i];
            if (h->scales_out) h->scales_out[&o - h->scales_base] = r.scale;
            o.score = r.score; o.angle = r.angle; o.cx = r.cx; o.cy = r.cy;
            o.ltx = r.ltx; o.lty = r.lty; o.rtx = r.rtx; o.rty = r.rty;
            o.rbx = r.rbx; o.rby = r.rby; o.lbx = r.lbx; o.lby = r.lby;
        }
    }
    return FPM_OK;
}

// candidate list: gather the picks of all angles, std::sort by score (:214), un-rotation (:265-266).  Leaves this
// rank's candidates (all of them when shard_n == 1) in d_cand[0] and, unless n_cands is null (the angle-sharded mode knows
// its counts from the gathered pick counts), reads their number back.
int collect_candidates(fpm_handle* h, int top, int batch, const FpmPickView& pv, int n_angles, int shard_rank, int shard_n,
                       int* n_cands, int* cand_stride_out)
{
    const int max_picks = h->max_pos + FPM_MATCH_CANDIDATE_NUM;
    const int cand_stride = std::max(n_angles * max_picks, 1);
    *cand_stride_out = cand_stride;
    int n_pad = 1;
    while (n_pad < cand_stride) n_pad <<= 1;
    CK(h->d_cand[0].ensure((size_t)batch * cand_stride * sizeof(FpmCand)));
    CK(h->d_candcnt.ensure((size_t)batch * sizeof(int)));
    CK(h->d_off.ensure((size_t)batch * std::max(n_angles, 1) * sizeof(int)));
    const int use_smem = (size_t)n_pad * 8 <= 96 * 1024;
    if (!use_smem) CK(h->d_keys.ensure((size_t)batch * n_pad * sizeof(unsigned long long)));
    if (h->trace) CK(h->d_toppt.ensure((size_t)batch * cand_stride * 4 * sizeof(float)));
    int* counters = h->d_counters.as<int>();
    {
        const FpmLevel& L = h->levels[top];
        size_t smem = use_smem ? (size_t)n_pad * 8 : 0;
        if (smem > 48 * 1024)
            CK(ensure_dyn_smem((const void*)fpm_collect_sort_kernel, h->device, smem));
        KL(K_COLLECT, 0,
           fpm_collect_sort_kernel<<<batch, CS_THREADS, smem, h->stream>>>(
               pv, n_angles, max_picks, h->d_angles.as<double>(),
               h->d_ftx.as<float>(), h->d_fty.as<float>(), (L.w - 1) / 2.0f, (L.h - 1) / 2.0f,
               h->d_keys.as<unsigned long long>(), n_pad, use_smem, h->d_off.as<int>(), h->d_cand[0].as<FpmCand>(),
               counters + CNT_FLAT, h->trace ? h->d_toppt.as<float>() : nullptr, cand_stride,
               h->d_candcnt.as<int>(), 0, shard_rank, shard_n,
               (h->scale_min == 1.0 && h->scale_max == 1.0) ? nullptr : h->d_scales.as<double>()));
    }
    if (!n_cands) return FPM_OK;
    int* hc = h->h_counts.as<int>();
    CK(cudaMemcpyAsync(hc, h->d_counters.p, CNT_N * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *n_cands = hc[CNT_FLAT];
    if (h->trace) {
        std::vector<float> tp((size_t)cand_stride * 4);
        int n0 = 0;
        CK(cudaMemcpy(&n0, h->d_candcnt.p, sizeof(int), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(tp.data(), h->d_toppt.p, (size_t)n0 * 4 * sizeof(float), cudaMemcpyDeviceToHost));
        h->tr_cands.clear();
        for (int i = 0; i < n0 * 4; i++) h->tr_cands.push_back(tp[i]);
    }
    return FPM_OK;
}

// guards of match(), src/TemplateMatcher.cpp:99-114; returns 1 when the match must return empty
int match_guards(const fpm_handle* h, int w, int hgt, int tw, int th)
{
    if (h->tol_range && (h->tol_r[0] >= h->tol_r[1] || h->tol_r[2] >= h->tol_r[3])) return 1;   // "left value must be smaller"
    if ((tw < w && th > hgt) || (tw > w && th < hgt)) return 1;
    if ((long long)tw * th > (long long)w * hgt) return 1;
    return 0;
}

int ensure_learned_for_mra(fpm_handle* h)
{
    if (!h->learned) return FPM_ERR_NOT_LEARNED;
    if (h->learned_mra != h->min_reduce_area) return do_learn(h);   // SURVEY 8a hazard: re-learn
    return FPM_OK;
}

// one group's pass over the pyramid of the batch: virtual images v = frame * n_tpl + member
int match_group(fpm_handle* h, int batch, fpm_result* out, int cap, int* n_out, int n_set, const MergeDev* md)
{
    const int top = (int)h->tpl.size() - 1;
    const int n_tpl = std::max((int)h->members.size(), 1), vbatch = batch * n_tpl;
    CK(cudaMemsetAsync(h->d_counters.p, 0, CNT_N * sizeof(int), h->stream));
    int rc = make_top_plan(h, top, batch);
    if (rc) return rc;
    const TopPlan& p = h->plan;
    const int max_picks = h->max_pos + FPM_MATCH_CANDIDATE_NUM;
    const int njobs = batch * p.n_ang;
    CK(h->d_picks.ensure((size_t)std::max(njobs * n_tpl, 1) * max_picks * sizeof(FpmPick)));
    CK(h->d_pickcnt.ensure((size_t)std::max(njobs * n_tpl, 1) * sizeof(int)));
    rc = run_top(h, top, 0, njobs, h->d_picks.as<FpmPick>(), h->d_pickcnt.as<int>());
    if (rc) return rc;
    FpmPickView pv{h->d_picks.as<FpmPick>(), h->d_pickcnt.as<int>(), 0, 0};
    int n_cands = 0, cand_stride = 0;
    rc = collect_candidates(h, top, vbatch, pv, p.n_ang, 0, 1, &n_cands, &cand_stride);
    if (rc) return rc;
    int n_refined = 0;
    h->ref_out = nullptr; h->ref_cnt = nullptr;
    rc = run_refine(h, top, n_cands, &n_refined);
    if (rc) return rc;
    FpmRefinedView rv{h->d_refined.as<FpmRefined>(), h->d_counters.as<int>() + CNT_REFINED, 0, 1, 0};
    return run_final(h, vbatch, rv, cand_stride, out, cap, n_out, n_set, md);
}

// merged set results (fpm_match_set_batch_merged): the caller's outputs besides out / counts, which then hold one list and
// one count per frame
struct SetMerge {
    double max_overlap;
    int* labels;                   // [frame][cap]
    int* set_counts;               // [frame][n_set], or nullptr
    SetMerge shifted(int frames, int cap, int n_set) const
    {
        return SetMerge{max_overlap, labels + (size_t)frames * cap, set_counts ? set_counts + (size_t)frames * n_set : nullptr};
    }
};

// d_merged, read back in one copy: int counts[batch] | int set_counts[batch][n_set] | int labels[batch][ocap] |
// int err[n_groups] (CNT_ERR of each group) | FpmResultDev records[batch][ocap] at a 256-byte aligned offset
struct MergedLayout {
    size_t set_counts, labels, err;   // int offsets
    size_t header_bytes, rec_off, bytes;
    MergedLayout(int batch, int n_set, int ocap, int n_groups)
    {
        set_counts = (size_t)batch;
        labels = set_counts + (size_t)batch * n_set;
        err = labels + (size_t)batch * ocap;
        header_bytes = (err + n_groups) * sizeof(int);
        rec_off = align_up(header_bytes, 256);
        bytes = rec_off + (size_t)batch * ocap * sizeof(FpmResultDev);
    }
};

// fpm_set_merge_kernel over the lists the groups left in d_mlists, then ONE read-back of everything (merged counts, the
// per-template totals, labels, CNT_ERR slots, records) and one synchronise
int run_set_merge(fpm_handle* h, int batch, int n_set, int n_groups, const MergeDev& md, const SetMerge* mg, fpm_result* out,
                  int cap, int* n_out)
{
    const int ocap = md.ocap;
    const MergedLayout lay(batch, n_set, ocap, n_groups);
    int ks = 1;
    while (ks < n_set * md.lcap) ks <<= 1;
    CK(h->d_keys.ensure((size_t)batch * ks * sizeof(unsigned long long)));
    CK(h->d_rects.ensure((size_t)batch * ks * sizeof(FpmRRect)));
    CK(h->d_del.ensure((size_t)batch * ks * sizeof(int)));
    CK(h->d_idmap.ensure((size_t)batch * ks * sizeof(int)));
    int* d_counts = h->d_merged.as<int>();
    int* d_labels = d_counts + lay.labels;
    FpmResultDev* d_rec = reinterpret_cast<FpmResultDev*>(h->d_merged.as<char>() + lay.rec_off);
    KL(K_SET_MERGE, (double)batch * n_set * md.lcap,
       fpm_set_merge_kernel<<<batch, FN_THREADS, 0, h->stream>>>(md.lists, md.counts, n_set, md.lcap, mg->max_overlap,
                                                                  h->d_keys.as<unsigned long long>(), ks, h->d_rects.as<FpmRRect>(),
                                                                  h->d_del.as<int>(), h->d_idmap.as<int>(), d_rec, d_labels, ocap,
                                                                  d_counts));
    CK(h->h_results.ensure(lay.bytes));
    CK(cudaMemcpyAsync(h->h_results.p, h->d_merged.p, lay.bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const int* hh = h->h_results.as<int>();
    const int* h_labels = hh + lay.labels;
    for (int g = 0; g < n_groups; g++)
        if (hh[lay.err + g]) { h->err = "fpm_corr_warp_kernel: source box larger than its staging buffer"; return FPM_ERR_LIMIT; }
    const FpmResultDev* h_rec = reinterpret_cast<const FpmResultDev*>(h->h_results.as<char>() + lay.rec_off);
    for (int b = 0; b < batch; b++) {
        n_out[b] = hh[b];
        if (mg->set_counts)
            for (int t = 0; t < n_set; t++) mg->set_counts[(size_t)b * n_set + t] = hh[lay.set_counts + (size_t)b * n_set + t];
        const int m = std::min(hh[b], cap);
        for (int i = 0; i < m; i++) {
            const FpmResultDev& r = h_rec[(size_t)b * ocap + i];
            fpm_result& o = out[(size_t)b * cap + i];
            if (h->scales_out) h->scales_out[&o - h->scales_base] = r.scale;
            o.score = r.score; o.angle = r.angle; o.cx = r.cx; o.cy = r.cy;
            o.ltx = r.ltx; o.lty = r.lty; o.rtx = r.rtx; o.rty = r.rty;
            o.rbx = r.rbx; o.rby = r.rby; o.lbx = r.lbx; o.lby = r.lby;
            mg->labels[(size_t)b * cap + i] = h_labels[(size_t)b * ocap + i];
        }
    }
    return FPM_OK;
}

// run[g] = 1 for the groups the size guards let run on a w x hgt source; returns the deepest top layer among them (-1: none)
int runnable_groups(const fpm_handle* h, int w, int hgt, std::vector<char>& run)
{
    const size_t n_groups = h->groups.size();
    run.assign(n_groups, 0);
    int max_top = -1;
    for (size_t g = 0; g < n_groups; g++) {
        const TplGroup& G = h->groups[g];
        const bool cur = g == 0;                             // group 0's state is in the handle's fields
        if (match_guards(h, w, hgt, cur ? h->tpl0_w : G.w0, cur ? h->tpl0_h : G.h0)) continue;
        run[g] = 1;
        max_top = std::max(max_top, (int)(cur ? h->tpl.size() : G.tpl.size()) - 1);
    }
    return max_top;
}

// device lists of the merge for the groups that run (run[g]) over `batch` frames, header zeroed on the stream
int merge_setup(fpm_handle* h, int batch, int cap, int n_set, const std::vector<char>& run, MergeDev* md)
{
    // list capacity: a group's list of a frame never exceeds its candidate list, (MaxPos + 5) entries per pose slot (angle x
    // scale of the schedule)
    const size_t n_groups = h->groups.size();
    int longest = 0;
    for (size_t g = 0; g < n_groups; g++) {
        if (!run[g]) continue;
        GroupScope scope(h, g);
        if (int rc = make_top_plan(h, (int)h->tpl.size() - 1, batch)) return rc;
        longest = std::max(longest, h->plan.n_ang * (h->max_pos + FPM_MATCH_CANDIDATE_NUM));
    }
    md->lcap = std::min(cap, longest);
    if ((long long)n_set * md->lcap >= (1ll << 30)) {
        h->err = "merged set results: n_set * list capacity (min(cap, pose slots x (MaxPos + 5))) too large";
        return FPM_ERR_LIMIT;
    }
    md->ocap = std::min(cap, n_set * md->lcap);
    const MergedLayout lay(batch, n_set, md->ocap, (int)n_groups);
    CK(h->d_mlists.ensure((size_t)batch * n_set * std::max(md->lcap, 1) * sizeof(FpmResultDev)));
    CK(h->d_merged.ensure(lay.bytes));
    CK(cudaMemsetAsync(h->d_merged.p, 0, lay.header_bytes, h->stream));   // the totals of groups that do not run, the CNT_ERR slots
    md->lists = h->d_mlists.as<FpmResultDev>();
    md->counts = h->d_merged.as<int>() + lay.set_counts;
    md->err = h->d_merged.as<int>() + lay.err;
    return FPM_OK;
}

// The match scale range (FPM_PARAM_SCALE_MIN / MAX), checked at match time because the two setters may run in either order:
// min <= max, and [1, 1] on the calls that do not carry a scale (scaled_ok = false: fpm_match_set_batch* and
// fpm_match_ingested_set_batch* on sets of more than one template, fpm_match_sharded*, fpm_match_set_sharded* without _scaled,
// fpm_stage_*).  The calls that return each record's scale accept any range: fpm_match_scaled, fpm_match_ingested_scaled,
// fpm_match_set_scaled*, fpm_match_ingested_set_scaled* and fpm_match_set_sharded_scaled*.
int refuse_scale(const fpm_handle* h, const char* fn, bool scaled_ok)
{
    if (h->scale_min == 1.0 && h->scale_max == 1.0) return FPM_OK;
    if (h->scale_min > h->scale_max)
        h->err = std::string(fn) + ": FPM_PARAM_SCALE_MIN (" + std::to_string(h->scale_min) + ") > FPM_PARAM_SCALE_MAX (" +
                 std::to_string(h->scale_max) + ")";
    else if (!scaled_ok)
        h->err = std::string(fn) + ": this call matches at scale 1 only (set FPM_PARAM_SCALE_MIN = FPM_PARAM_SCALE_MAX = 1)";
    else
        return FPM_OK;
    return FPM_ERR_INVALID;
}

// whole match() over a device-resident batch, for every template of the set: frame b / template t at out + (b * n + t) * cap,
// or (mg) the merged list of frame b at out + b * cap.
// The source pyramid (and bitwise_not) is built once, down to the deepest top layer of any group; the groups run one
// after another on the handle's stream.
int match_device(fpm_handle* h, const uint8_t* d_src, int batch, int w, int hgt, int stride, size_t frame_stride,
                 fpm_result* out, int cap, int* n_out, const SetMerge* mg = nullptr)
{
    const int n_set = std::max((int)h->set.size(), 1);
    for (int b = 0; b < batch * (mg ? 1 : n_set); b++) n_out[b] = 0;
    if (mg && mg->set_counts) std::fill(mg->set_counts, mg->set_counts + (size_t)batch * n_set, 0);
    if (!h->learned) return FPM_OK;                          // :99-101 -> empty
    const bool is_set = fpm_set_size(h) > 1;
    int rc = refuse_scale(h, h->scaled_fn ? h->scaled_fn : is_set ? "fpm_match_set_batch" : "fpm_match", !is_set || h->scaled_fn);
    if (rc) return rc;
    rc = ensure_learned_for_mra(h);
    if (rc) return rc;
    const size_t n_groups = h->groups.size();
    std::vector<char> run;
    const int max_top = runnable_groups(h, w, hgt, run);
    if (max_top < 0) return FPM_OK;
    h->cur_batch = batch;
    CK(h->d_counters.ensure(CNT_N * sizeof(int)));
    CK(h->h_counts.ensure((CNT_N + (size_t)batch * n_set) * sizeof(int)));
    if (h->bitwise_not) {
        const int ipitch = (int)align_up(w, 128);
        const size_t iimg = (size_t)ipitch * hgt;
        CK(h->d_inv.ensure(iimg * batch));
        dim3 ig((w / 4 + 128) / 128, hgt, batch);
        fpm_invert_kernel<<<ig, 128, 0, h->stream>>>(d_src, w, hgt, stride, frame_stride, h->d_inv.as<uint8_t>(), ipitch, iimg);
        CKL();
        d_src = h->d_inv.as<uint8_t>(); stride = ipitch; frame_stride = iimg;
    }
    rc = build_pyramid(h, d_src, batch, w, hgt, stride, frame_stride, max_top);
    if (rc) return rc;
    MergeDev md;
    if (mg && (rc = merge_setup(h, batch, cap, n_set, run, &md))) return rc;
    int* err_slots = md.err;
    size_t member_off = 0;
    for (size_t g = 0; g < n_groups && rc == FPM_OK; g++) {
        const size_t n_members = g == 0 ? h->members.size() : h->groups[g].members.size();
        md.rows = h->d_members.as<int>() + member_off;
        md.err = err_slots ? err_slots + g : nullptr;
        member_off += n_members;
        if (!run[g]) continue;
        GroupScope scope(h, g);
        rc = match_group(h, batch, out, cap, n_out, n_set, mg ? &md : nullptr);
    }
    if (rc == FPM_OK && mg) rc = run_set_merge(h, batch, n_set, (int)n_groups, md, mg, out, cap, n_out);
    return rc;
}

// ---- angle-sharded latency mode (SURVEY 8e): one frame, nranks GPUs -------------------------------------------
// The work of TemplateMatcher::match shards in two places: the top-layer angle sweep (src/TemplateMatcher.cpp:162-211)
// and the per-candidate descent (:262-371).  Each rank runs a contiguous chunk of the angle schedule, the pick lists are
// exchanged with ONE allgather of fixed-size blocks (picks + counts), every rank sorts the identical global list
// (:214) and refines candidates id % nranks == rank, the refined records are exchanged with a second allgather and
// every rank runs the identical filter / NMS (:373-395).  Both gathered buffers are consumed in place by the kernels
// (FpmPickView / FpmRefinedView): nothing but the final results and two counters ever reaches the host.
struct NcclApi {
    typedef struct { char internal[128]; } UniqueId;           // ncclUniqueId (ABI-stable: 128 opaque bytes)
    int (*GetUniqueId)(UniqueId*) = nullptr;
    int (*CommInitRank)(void**, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int /*ncclDataType_t*/, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int*) = nullptr;
    bool ok = false;
};

const NcclApi& nccl_api()
{
    // resolved at run time: the library must load (and every single-GPU entry point must work) on a box without NCCL;
    // in a torch process "libnccl.so.2" resolves to the copy torch has already loaded
    static const NcclApi api = []() {
        NcclApi a;
        void* lib = nullptr;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
        if (!lib) return a;
        a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
        a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
        a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
        a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(lib, "ncclAllGather"));
        a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
        a.GetVersion = reinterpret_cast<decltype(a.GetVersion)>(dlsym(lib, "ncclGetVersion"));
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllGather && a.GetErrorString;
        return a;
    }();
    return api;
}

// in-place allgather of one `bytes`-sized block per rank (own block already at buf + rank*bytes), on the handle's stream
int shard_allgather(fpm_handle* h, void* buf, size_t bytes)
{
    if (h->sh_nranks <= 1) return FPM_OK;
    if (!h->nccl_comm) { h->err = "angle-sharded match: no communicator (fpm_comm_init / fpm_comm_attach)"; return FPM_ERR_INVALID; }
    const NcclApi& a = nccl_api();
    const int r = a.AllGather(static_cast<const char*>(buf) + (size_t)h->sh_rank * bytes, buf, bytes, 0 /*ncclInt8*/, h->nccl_comm, h->stream);
    if (r != 0) { h->err = std::string("ncclAllGather: ") + a.GetErrorString(r); return FPM_ERR_CUDA; }
    h->collectives++;
    return FPM_OK;
}

// contiguous chunk of the angle schedule per rank: rank r sweeps [r*chunk, min(A, (r+1)*chunk))
inline int shard_chunk(int n_angles, int nranks) { return std::max(1, (n_angles + nranks - 1) / nranks); }

// candidates of a global list of n entries that rank R of N refines (candidate k -> rank k mod N)
inline int shard_share(int n, int R, int N) { return n > R ? (n - R + N - 1) / N : 0; }

// phase 1: source on the device (uploaded in 1/N row slices + allgather when it comes from the host), pyramid down to the
// deepest top layer of the groups that run, then for every such group the top-layer sweep of this rank's chunk of its angle
// schedule for all its templates, into the group's place in this rank's block of the gather buffer
int shard_begin(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, int src_on_device)
{
    h->sh = fpm_handle::ShardState();
    if (!h->learned) return FPM_OK;                          // :99-101 -> empty
    int rc = ensure_learned_for_mra(h);
    if (rc) return rc;
    if (!src || w <= 0 || hgt <= 0) return FPM_OK;
    if (stride < w) { h->err = "stride < width"; return FPM_ERR_INVALID; }
    std::vector<char> run;
    const int max_top = runnable_groups(h, w, hgt, run);
    if (max_top < 0) return FPM_OK;
    const int N = h->sh_nranks, R = h->sh_rank;
    const uint8_t* d_src = src;
    int pitch = stride;
    size_t img = (size_t)stride * hgt;
    if (!src_on_device) {
        const bool linear = (stride == w) && (w % 4 == 0);
        pitch = linear ? w : (int)align_up(w, 128);
        const int rows_per = (hgt + N - 1) / N;
        img = (size_t)pitch * rows_per * N;                   // room for N equal row slices
        CK(h->d_src.ensure(img));
        const bool sliced = N > 1 && h->shard_upload && h->nccl_comm;
        const int y0 = sliced ? std::min(hgt, R * rows_per) : 0, y1 = sliced ? std::min(hgt, y0 + rows_per) : hgt;
        if (y1 > y0) {
            if (linear)
                CK(cudaMemcpyAsync(h->d_src.as<uint8_t>() + (size_t)y0 * pitch, src + (size_t)y0 * stride, (size_t)(y1 - y0) * pitch,
                                   cudaMemcpyHostToDevice, h->stream));
            else
                CK(cudaMemcpy2DAsync(h->d_src.as<uint8_t>() + (size_t)y0 * pitch, pitch, src + (size_t)y0 * stride, stride, w, y1 - y0,
                                     cudaMemcpyHostToDevice, h->stream));
        }
        if (sliced) {
            rc = shard_allgather(h, h->d_src.p, (size_t)pitch * rows_per);
            if (rc) return rc;
        }
        d_src = h->d_src.as<uint8_t>();
    }
    h->cur_batch = 1;
    CK(h->d_counters.ensure(CNT_N * sizeof(int)));
    CK(h->h_counts.ensure((CNT_N + 1) * sizeof(int)));
    CK(cudaMemsetAsync(h->d_counters.p, 0, CNT_N * sizeof(int), h->stream));
    if (h->bitwise_not) {
        const int ipitch = (int)align_up(w, 128);
        const size_t iimg = (size_t)ipitch * hgt;
        CK(h->d_inv.ensure(iimg));
        dim3 ig((w / 4 + 128) / 128, hgt, 1);
        fpm_invert_kernel<<<ig, 128, 0, h->stream>>>(d_src, w, hgt, pitch, img, h->d_inv.as<uint8_t>(), ipitch, iimg);
        CKL();
        d_src = h->d_inv.as<uint8_t>(); pitch = ipitch; img = iimg;
    }
    rc = build_pyramid(h, d_src, 1, w, hgt, pitch, img, max_top);
    if (rc) return rc;
    // the block layout, from the plans (the same on every rank)
    fpm_handle::ShardState& S = h->sh;
    const int max_picks = h->max_pos + FPM_MATCH_CANDIDATE_NUM;
    const size_t n_groups = h->groups.size();
    S.g.assign(n_groups, fpm_handle::ShardGroup());
    size_t pick_bytes = 0, n_cnt = 0;
    for (size_t g = 0; g < n_groups; g++) {
        if (!run[g]) continue;
        GroupScope scope(h, g);
        if ((rc = make_top_plan(h, (int)h->tpl.size() - 1, 1))) return rc;
        fpm_handle::ShardGroup& sg = S.g[g];
        sg.n_tpl = std::max((int)h->members.size(), 1);
        sg.chunk = shard_chunk(h->plan.n_ang, N);
        sg.pick_off = pick_bytes;
        sg.cnt_off = n_cnt;
        pick_bytes += (size_t)sg.n_tpl * sg.chunk * max_picks * sizeof(FpmPick);
        n_cnt += (size_t)sg.n_tpl * sg.chunk;
    }
    S.cnt_off = pick_bytes; S.n_cnt = n_cnt;
    S.pick_blk = align_up(pick_bytes + n_cnt * sizeof(int), 16);
    CK(h->d_gpicks.ensure(S.pick_blk * N));
    uint8_t* mine = h->d_gpicks.as<uint8_t>() + (size_t)R * S.pick_blk;
    int* cnt = reinterpret_cast<int*>(mine + S.cnt_off);
    CK(cudaMemsetAsync(cnt, 0, n_cnt * sizeof(int), h->stream));   // angles past a schedule's end stay empty
    for (size_t g = 0; g < n_groups; g++) {
        if (!run[g]) continue;
        GroupScope scope(h, g);
        const fpm_handle::ShardGroup& sg = S.g[g];
        const int n_ang = h->plan.n_ang;
        const int a0 = std::min(n_ang, R * sg.chunk), a1 = std::min(n_ang, a0 + sg.chunk);
        rc = run_top(h, (int)h->tpl.size() - 1, a0, a1 - a0, reinterpret_cast<FpmPick*>(mine + sg.pick_off), cnt + sg.cnt_off, sg.chunk);
        if (rc) return rc;
    }
    S.run.swap(run);
    S.empty = 0;
    return FPM_OK;
}

int shard_exchange_picks(fpm_handle* h)
{
    if (h->sh.empty) return FPM_OK;
    return shard_allgather(h, h->d_gpicks.p, h->sh.pick_blk);
}

// phase 2: one read-back of the gathered pick counts gives every rank the global list size of every (group, template) and
// so the layout of the refined blocks; per group, every rank sorts the identical global lists in place and refines its share
// into the group's segment of its refined block
int shard_mid(fpm_handle* h)
{
    if (h->sh.empty) return FPM_OK;
    fpm_handle::ShardState& S = h->sh;
    const int N = h->sh_nranks, R = h->sh_rank;
    const size_t cnt_bytes = S.n_cnt * sizeof(int);
    CK(h->h_counts.ensure(std::max(cnt_bytes * N, (CNT_N + 1) * sizeof(int))));
    if (cnt_bytes)
        CK(cudaMemcpy2DAsync(h->h_counts.p, cnt_bytes, h->d_gpicks.as<uint8_t>() + S.cnt_off, S.pick_blk, cnt_bytes, N,
                             cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const int* hc = h->h_counts.as<int>();
    const size_t n_groups = S.g.size();
    size_t ref_bytes = 0;
    for (size_t g = 0; g < n_groups; g++) {
        if (!S.run[g]) continue;
        fpm_handle::ShardGroup& sg = S.g[g];
        int seg = 0;
        for (int t = 0; t < sg.n_tpl; t++) {
            int n = 0;
            for (int r = 0; r < N; r++)
                for (int l = 0; l < sg.chunk; l++) n += hc[(size_t)r * S.n_cnt + sg.cnt_off + (size_t)t * sg.chunk + l];
            sg.n_local += shard_share(n, R, N);
            seg += (n + N - 1) / N;                          // the largest share any rank gets of this list
            sg.key_stride = std::max(sg.key_stride, n);
        }
        sg.seg_cap = std::max(1, seg);
        sg.ref_off = ref_bytes;
        ref_bytes += align_up((size_t)sg.seg_cap * sizeof(FpmRefined) + 8, 16);
    }
    S.ref_blk = std::max<size_t>(ref_bytes, 16);
    CK(h->d_grefined.ensure(S.ref_blk * N));
    uint8_t* base = h->d_gpicks.as<uint8_t>();
    uint8_t* mine = h->d_grefined.as<uint8_t>() + (size_t)R * S.ref_blk;
    for (size_t g = 0; g < n_groups; g++) {
        if (!S.run[g]) continue;
        GroupScope scope(h, g);
        const fpm_handle::ShardGroup& sg = S.g[g];
        const int top = (int)h->tpl.size() - 1;
        CK(cudaMemsetAsync(h->d_counters.as<int>() + CNT_FLAT, 0, sizeof(int), h->stream));
        const FpmPickView pv{reinterpret_cast<const FpmPick*>(base + sg.pick_off), reinterpret_cast<const int*>(base + S.cnt_off) + sg.cnt_off,
                             sg.chunk, S.pick_blk};
        int cand_stride = 0;
        int rc = collect_candidates(h, top, sg.n_tpl, pv, sg.chunk * N, R, N, nullptr, &cand_stride);
        if (rc) return rc;
        h->ref_out = reinterpret_cast<FpmRefined*>(mine + sg.ref_off);
        h->ref_cnt = reinterpret_cast<int*>(mine + sg.ref_off + (size_t)sg.seg_cap * sizeof(FpmRefined));
        int n_refined = 0;
        rc = run_refine(h, top, sg.n_local, &n_refined);
        h->ref_out = nullptr; h->ref_cnt = nullptr;
        if (rc) return rc;
    }
    return FPM_OK;
}

int shard_exchange_refined(fpm_handle* h)
{
    if (h->sh.empty) return FPM_OK;
    return shard_allgather(h, h->d_grefined.p, h->sh.ref_blk);
}

// phase 3: per group, the replicated filterWithScore + NMS + conversion straight from the gathered blocks, to the caller's
// [template][cap] lists or (mg) the device lists of the merge, then one merge launch
int shard_end(fpm_handle* h, fpm_result* out, int cap, int* n_out, const SetMerge* mg)
{
    const fpm_handle::ShardState& S = h->sh;
    if (S.empty) return FPM_OK;
    const int n_set = std::max((int)h->set.size(), 1);
    const size_t n_groups = S.g.size();
    MergeDev md;
    if (mg) if (int rc = merge_setup(h, 1, cap, n_set, S.run, &md)) return rc;
    int* err_slots = md.err;
    size_t member_off = 0;
    for (size_t g = 0; g < n_groups; g++) {
        const size_t n_members = g == 0 ? h->members.size() : h->groups[g].members.size();
        md.rows = h->d_members.as<int>() + member_off;
        md.err = err_slots ? err_slots + g : nullptr;
        member_off += n_members;
        if (!S.run[g]) continue;
        GroupScope scope(h, g);
        const fpm_handle::ShardGroup& sg = S.g[g];
        const FpmRefinedView rv{reinterpret_cast<const FpmRefined*>(h->d_grefined.as<uint8_t>() + sg.ref_off), nullptr, sg.seg_cap,
                                h->sh_nranks, S.ref_blk};
        if (int rc = run_final(h, sg.n_tpl, rv, sg.key_stride, out, cap, n_out, n_set, mg ? &md : nullptr)) return rc;
    }
    return mg ? run_set_merge(h, 1, n_set, (int)n_groups, md, mg, out, cap, n_out) : FPM_OK;
}

// one frame against the whole set across the communicator's ranks (fpm_match_set_sharded*): every rank gets the lists
// fpm_match_set_batch (mg: fpm_match_set_batch_merged) returns for the frame on one GPU
int match_set_sharded(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device, fpm_result* out,
                      int cap, int* n, const SetMerge* mg)
{
    CK(cudaSetDevice(h->device));
    auto t0 = std::chrono::high_resolution_clock::now();
    int rc = shard_begin(h, src, width, height, stride, src_on_device);
    if (!rc) rc = shard_exchange_picks(h);
    if (!rc) rc = shard_mid(h);
    if (!rc) rc = shard_exchange_refined(h);
    if (!rc) rc = shard_end(h, out, cap, n, mg);
    prof_collect(h);
    if (rc) cudaStreamSynchronize(h->stream);
    h->last_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    return rc;
}

// The same pipeline with `nranks` handles of ONE device playing the ranks and the two exchanges done as device-to-device
// block copies: exercises the partitioning and the in-place consumption of the gathered buffers where only one GPU (and no
// NCCL peer) is available.  Rank r's lists go to out + r * n_rows * cap and n + r * n_rows (n_rows = 1 merged, else the set
// size); mg[r] is rank r's merge.  count_exchanges: every exchange round adds one to each handle's collective count.
int match_set_sharded_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                              fpm_result* out, int cap, int* n, int n_rows, const SetMerge* mg, bool count_exchanges)
{
    for (int r = 0; r < nranks; r++) { hs[r]->sh_nranks = nranks; hs[r]->sh_rank = r; }
    auto exchange = [&](DevBuf fpm_handle::*buf, size_t fpm_handle::ShardState::*blk) -> int {
        for (int r = 0; r < nranks; r++) {
            fpm_handle* h = hs[r];
            CK(cudaStreamSynchronize(h->stream));
        }
        for (int q = 0; q < nranks; q++) {
            fpm_handle* h = hs[q];
            if (h->sh.empty) continue;
            const size_t b = h->sh.*blk;
            for (int r = 0; r < nranks; r++)
                if (r != q && !hs[r]->sh.empty)
                    CK(cudaMemcpyAsync((h->*buf).as<uint8_t>() + (size_t)r * b, (hs[r]->*buf).as<uint8_t>() + (size_t)r * b, b,
                                       cudaMemcpyDeviceToDevice, h->stream));
            if (count_exchanges) h->collectives++;
        }
        return FPM_OK;
    };
    int rc = FPM_OK;
    for (int r = 0; r < nranks && !rc; r++) { cudaSetDevice(hs[r]->device); rc = shard_begin(hs[r], src, width, height, stride, 0); }
    if (!rc) rc = exchange(&fpm_handle::d_gpicks, &fpm_handle::ShardState::pick_blk);
    for (int r = 0; r < nranks && !rc; r++) rc = shard_mid(hs[r]);
    if (!rc) rc = exchange(&fpm_handle::d_grefined, &fpm_handle::ShardState::ref_blk);
    for (int r = 0; r < nranks && !rc; r++)
        rc = shard_end(hs[r], out + (size_t)r * n_rows * cap, cap, n + (size_t)r * n_rows, mg ? mg + r : nullptr);
    for (int r = 0; r < nranks; r++) {
        prof_collect(hs[r]);
        if (rc) cudaStreamSynchronize(hs[r]->stream);
        hs[r]->sh_nranks = 1; hs[r]->sh_rank = 0;
    }
    return rc;
}

}  // namespace

// =====================================================================================
// C ABI
// =====================================================================================
extern "C" {

const char* fpm_version(void) { return "fpm-b200 0.1 (sm_100a)"; }

fpm_handle* fpm_create(int device)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return nullptr;                       // no CPU fallback
    }
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    fpm_handle* h = new fpm_handle();
    h->device = device;
    if (cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || h->num_sms <= 0) h->num_sms = 148;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return nullptr;
    }
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&h->ev_copy[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming);
    }
    cudaEventCreate(&h->ev_t0);
    cudaEventCreate(&h->ev_t1);
    cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    return h;
}

void fpm_destroy(fpm_handle* h)
{
    if (!h) return;
    if (h->twin) { fpm_destroy(h->twin); h->twin = nullptr; }
    fpm_comm_destroy(h);
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->copy_stream);
    cudaStreamSynchronize(h->aux_stream);
    DevBuf* bufs[] = {&h->d_gpicks, &h->d_grefined, &h->d_tpl, &h->d_tsh, &h->d_raw, &h->d_inv, &h->d_numer, &h->d_totS, &h->d_totQ, &h->d_ingest_raw, &h->d_ingest, &h->d_src, &h->d_pyr, &h->d_rot, &h->d_score, &h->d_blkv, &h->d_blkl, &h->d_picks, &h->d_pickcnt,
                      &h->d_jobs_top, &h->d_angles, &h->d_ftx, &h->d_fty, &h->d_scales, &h->d_off, &h->d_keys, &h->d_cand[0], &h->d_cand[1],
                      &h->d_candcnt, &h->d_toppt, &h->d_counters, &h->d_jobs_ref, &h->d_roi, &h->d_rowsum, &h->d_rowS, &h->d_rowQ,
                      &h->d_pairs, &h->d_refined, &h->d_rects, &h->d_del, &h->d_idmap, &h->d_results, &h->d_rescnt, &h->d_trace, &h->d_trace_sc,
                      &h->d_dbg[0], &h->d_dbg[1], &h->d_dbg[2], &h->d_dbg[3], &h->d_members, &h->d_mlists, &h->d_merged};
    for (DevBuf* b : bufs) b->release();
    for (size_t g = 1; g < h->groups.size(); g++) h->groups[g].release();
    h->d_tstat.release();
    h->h_counts.release(); h->h_results.release(); h->h_stage.release();
    h->d_jpeg.release();
    h->d_jpeg_scan.release();
    for (int i = 0; i < 2; i++) { cudaEventDestroy(h->ev_copy[i]); cudaEventDestroy(h->ev_done[i]); }
    cudaEventDestroy(h->ev_t0); cudaEventDestroy(h->ev_t1);
    prof_collect(h);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    cudaEventDestroy(h->ev_fork); cudaEventDestroy(h->ev_join);
    cudaStreamDestroy(h->stream);
    cudaStreamDestroy(h->copy_stream);
    cudaStreamDestroy(h->aux_stream);
    delete h;
}

const char* fpm_last_error(const fpm_handle* h) { return h ? h->err.c_str() : "null handle (no CUDA device?)"; }

int fpm_set_param(fpm_handle* h, int param, double v)
{
    if (!h) return FPM_ERR_INVALID;
    switch (param) {
    case FPM_PARAM_MAX_POSITIONS: h->max_pos = (int)v; break;
    case FPM_PARAM_MAX_OVERLAP: h->max_overlap = v; break;
    case FPM_PARAM_SCORE: h->score = v; break;
    case FPM_PARAM_TOLERANCE_ANGLE: h->tol_angle = v; break;
    case FPM_PARAM_MIN_REDUCE_AREA: h->min_reduce_area = (int)v; break;
    case FPM_PARAM_USE_SIMD: h->use_simd = v != 0; break;
    case FPM_PARAM_SUBPIXEL: h->subpixel = v != 0; break;
    case FPM_PARAM_TRACE: h->trace = v != 0; break;
    case FPM_PARAM_WORKSPACE_MB: h->workspace_mb = v; break;
    case FPM_PARAM_PROFILE: prof_collect(h); h->profile = v != 0; break;
    case FPM_PARAM_H2D_CHUNK: h->h2d_chunk = (int)v; break;
    case FPM_PARAM_TENSOR_CORES: h->use_tc = (int)v; break;
    case FPM_PARAM_MFC_COMPAT: h->mfc_compat = v != 0; break;
    case FPM_PARAM_STOP_LAYER1: h->stop_layer1 = v != 0; break;
    case FPM_PARAM_BITWISE_NOT: h->bitwise_not = v != 0; break;
    case FPM_PARAM_SPLIT_BATCH: h->split_batch = (int)v; break;
    case FPM_PARAM_SHARD_UPLOAD: h->shard_upload = v != 0; break;
    case FPM_PARAM_ASYNC_DESCENT: h->async_descent = (int)v; break;
    case FPM_PARAM_JPEG_DEVICE_HUFFMAN: h->jpeg_device_huffman = v != 0; break;
    case FPM_PARAM_TOLERANCE_RANGE: h->tol_range = v != 0; break;
    case FPM_PARAM_TOLERANCE1: case FPM_PARAM_TOLERANCE2: case FPM_PARAM_TOLERANCE3: case FPM_PARAM_TOLERANCE4:
        h->tol_r[param - FPM_PARAM_TOLERANCE1] = v; break;
    case FPM_PARAM_SCALE_MIN: case FPM_PARAM_SCALE_MAX:
        // beyond 2 the bilinear resampling (no prefilter) aliases; below 0.5 the top-layer canvases grow by 4x or more
        if (!std::isfinite(v) || v < 0.5 || v > 2.0) {
            h->err = std::string(param == FPM_PARAM_SCALE_MIN ? "FPM_PARAM_SCALE_MIN" : "FPM_PARAM_SCALE_MAX") + " must lie in [0.5, 2], got " +
                     std::to_string(v);
            return FPM_ERR_INVALID;
        }
        (param == FPM_PARAM_SCALE_MIN ? h->scale_min : h->scale_max) = v; break;
    default: h->err = "unknown parameter"; return FPM_ERR_INVALID;
    }
    if (param == FPM_PARAM_TOLERANCE_RANGE || (param >= FPM_PARAM_TOLERANCE1 && param <= FPM_PARAM_TOLERANCE4)) {
        h->plan.valid = false;                                 // the angle schedule of every group
        for (TplGroup& g : h->groups) g.plan.valid = false;
    }
    return FPM_OK;
}

double fpm_get_param(const fpm_handle* h, int param)
{
    if (!h) return 0;
    switch (param) {
    case FPM_PARAM_MAX_POSITIONS: return h->max_pos;
    case FPM_PARAM_MAX_OVERLAP: return h->max_overlap;
    case FPM_PARAM_SCORE: return h->score;
    case FPM_PARAM_TOLERANCE_ANGLE: return h->tol_angle;
    case FPM_PARAM_MIN_REDUCE_AREA: return h->min_reduce_area;
    case FPM_PARAM_USE_SIMD: return h->use_simd;
    case FPM_PARAM_SUBPIXEL: return h->subpixel;
    case FPM_PARAM_TRACE: return h->trace;
    case FPM_PARAM_WORKSPACE_MB: return h->workspace_mb;
    case FPM_PARAM_PROFILE: return h->profile;
    case FPM_PARAM_H2D_CHUNK: return h->h2d_chunk;
    case FPM_PARAM_TENSOR_CORES: return h->use_tc;
    case FPM_PARAM_MFC_COMPAT: return h->mfc_compat;
    case FPM_PARAM_STOP_LAYER1: return h->stop_layer1;
    case FPM_PARAM_BITWISE_NOT: return h->bitwise_not;
    case FPM_PARAM_SPLIT_BATCH: return h->split_batch;
    case FPM_PARAM_SHARD_UPLOAD: return h->shard_upload;
    case FPM_PARAM_ASYNC_DESCENT: return h->async_descent;
    case FPM_PARAM_JPEG_DEVICE_HUFFMAN: return h->jpeg_device_huffman;
    case FPM_PARAM_JPEG_PASSES: return h->jpeg_passes;
    case FPM_PARAM_TOLERANCE_RANGE: return h->tol_range;
    case FPM_PARAM_TOLERANCE1: case FPM_PARAM_TOLERANCE2: case FPM_PARAM_TOLERANCE3: case FPM_PARAM_TOLERANCE4:
        return h->tol_r[param - FPM_PARAM_TOLERANCE1];
    case FPM_PARAM_SCALE_MIN: return h->scale_min;
    case FPM_PARAM_SCALE_MAX: return h->scale_max;
    default: return 0;
    }
}

int fpm_learn(fpm_handle* h, const uint8_t* tpl, int width, int height, int stride)
{
    if (!h) return FPM_ERR_INVALID;
    if (!tpl || width <= 0 || height <= 0 || stride < width) { h->err = "empty template"; return FPM_ERR_INVALID; }   // :47-49
    return fpm_learn_set(h, 1, &tpl, &width, &height, &stride);
}

namespace {
// fpm_learn_set, with the 0/1 level-0 mask of every template (empty: unmasked) or none (masks empty: all unmasked);
// masked_set: refusals name the template index (fpm_learn_set_masked)
int learn_set(fpm_handle* h, int n, const uint8_t* const* tpls, const int* widths, const int* heights, const int* strides,
              std::vector<std::vector<uint8_t>> masks, bool masked_set)
{
    h->learned = false;
    h->set.clear();
    h->learn_gen++;
    if (n < 1 || !tpls || !widths || !heights || !strides) { h->err = "template set: n < 1 or null arrays"; return FPM_ERR_INVALID; }
    for (int i = 0; i < n; i++)
        if (!tpls[i] || widths[i] <= 0 || heights[i] <= 0 || strides[i] < widths[i]) {
            h->err = "template set: template " + std::to_string(i) + " is empty (null, a size <= 0 or stride < width)";
            return FPM_ERR_INVALID;
        }
    std::vector<SetTpl> set(n);
    for (int i = 0; i < n; i++) {
        set[i].w = widths[i]; set[i].h = heights[i];
        set[i].px.resize((size_t)widths[i] * heights[i]);
        for (int y = 0; y < heights[i]; y++) memcpy(set[i].px.data() + (size_t)y * widths[i], tpls[i] + (size_t)y * strides[i], widths[i]);
        if (!masks.empty()) set[i].mask.swap(masks[i]);
    }
    h->set.swap(set);
    h->masked_set = masked_set;
    int rc = do_learn(h);
    if (rc) h->set.clear();
    return rc;
}

// the 0/1 copy of a caller's mask (w x h, mask_stride bytes per row) and its kept count
size_t copy_mask(const uint8_t* mask, int mask_stride, int w, int hgt, std::vector<uint8_t>& m)
{
    m.resize((size_t)w * hgt);
    size_t kept = 0;
    for (int y = 0; y < hgt; y++)
        for (int x = 0; x < w; x++) kept += m[(size_t)y * w + x] = mask[(size_t)y * mask_stride + x] ? 1 : 0;
    return kept;
}

int refuse_learn(fpm_handle* h, const std::string& why)
{
    h->learned = false; h->set.clear(); h->learn_gen++;
    h->err = why;
    return FPM_ERR_INVALID;
}
}  // namespace

int fpm_learn_set(fpm_handle* h, int n, const uint8_t* const* tpls, const int* widths, const int* heights, const int* strides)
{
    if (!h) return FPM_ERR_INVALID;
    return learn_set(h, n, tpls, widths, heights, strides, {}, false);
}

int fpm_learn_set_masked(fpm_handle* h, int n, const uint8_t* const* tpls, const int* widths, const int* heights,
                         const int* strides, const uint8_t* const* masks, const int* mask_strides)
{
    if (!h) return FPM_ERR_INVALID;
    if (!masks) return learn_set(h, n, tpls, widths, heights, strides, {}, false);
    if (!mask_strides) return refuse_learn(h, "fpm_learn_set_masked: null mask_strides with masks");
    if (n < 1 || !tpls || !widths || !heights || !strides) return learn_set(h, n, tpls, widths, heights, strides, {}, true);
    std::vector<std::vector<uint8_t>> ms(n);
    for (int i = 0; i < n; i++) {
        if (!masks[i]) continue;
        if (!tpls[i] || widths[i] <= 0 || heights[i] <= 0 || strides[i] < widths[i]) break;   // learn_set names the empty template
        const std::string ti = "fpm_learn_set_masked: template " + std::to_string(i);
        if (mask_strides[i] < widths[i]) return refuse_learn(h, ti + ": mask stride smaller than the template width");
        if (!copy_mask(masks[i], mask_strides[i], widths[i], heights[i], ms[i])) return refuse_learn(h, ti + ": the mask keeps no pixel");
    }
    return learn_set(h, n, tpls, widths, heights, strides, std::move(ms), true);
}

int fpm_learn_masked(fpm_handle* h, const uint8_t* tpl, int width, int height, int stride, const uint8_t* mask, int mask_stride)
{
    if (!h) return FPM_ERR_INVALID;
    const char* why = nullptr;
    if (!tpl || width <= 0 || height <= 0 || stride < width) why = "empty template";
    else if (!mask) why = "fpm_learn_masked: null mask";
    else if (mask_stride < width) why = "fpm_learn_masked: mask stride smaller than the template width";
    std::vector<std::vector<uint8_t>> m(1);
    if (!why && !copy_mask(mask, mask_stride, width, height, m[0])) why = "fpm_learn_masked: the mask keeps no pixel";
    if (why) return refuse_learn(h, why);
    return learn_set(h, 1, &tpl, &width, &height, &stride, std::move(m), false);
}

int fpm_set_size(const fpm_handle* h) { return h && h->learned ? (int)h->set.size() : 0; }

int fpm_is_learned(const fpm_handle* h) { return h && h->learned ? 1 : 0; }

void fpm_clear(fpm_handle* h)
{
    if (!h) return;
    h->learned = false; h->tpl.clear(); h->set.clear(); h->members.clear(); h->has_ur = 0;
    for (size_t g = 1; g < h->groups.size(); g++) h->groups[g].release();
    h->groups.clear();
    h->ur[0] = h->ur[1] = h->ur[2] = h->ur[3] = 0;
}

namespace {
// the single-template entry points on a handle that holds a set of more than one: refused, never template 0 alone
int refuse_set(const fpm_handle* h, const char* fn)
{
    if (fpm_set_size(h) <= 1) return FPM_OK;
    h->err = std::string(fn) + ": the handle holds a set of " + std::to_string(h->set.size()) +
             " templates (use fpm_match_set_batch / fpm_match_ingested_set_batch)";
    return FPM_ERR_INVALID;
}
}  // namespace

// second handle for the concurrent half-batches: same device, parameters and template set as h
int ensure_twin(fpm_handle* h)
{
    if (!h->twin) {
        h->twin = fpm_create(h->device);
        if (!h->twin) { h->err = "could not create the twin handle"; return FPM_ERR_CUDA; }
        h->twin->split_batch = 0;
        h->twin_gen = 0;
    }
    fpm_handle* t = h->twin;
    for (int p = 0; p < FPM_PARAM_COUNT_; p++)
        if (p != FPM_PARAM_TRACE && p != FPM_PARAM_SPLIT_BATCH && fpm_get_param(t, p) != fpm_get_param(h, p))
            fpm_set_param(t, p, fpm_get_param(h, p));
    if (h->twin_gen != h->learn_gen || !t->learned) {
        const int n = (int)h->set.size();
        std::vector<const uint8_t*> px(n);
        std::vector<int> ws(n), hs(n);
        std::vector<std::vector<uint8_t>> ms(n);
        for (int i = 0; i < n; i++) { px[i] = h->set[i].px.data(); ws[i] = h->set[i].w; hs[i] = h->set[i].h; ms[i] = h->set[i].mask; }
        int rc = learn_set(t, n, px.data(), ws.data(), hs.data(), ws.data(), std::move(ms), h->masked_set);
        if (rc) { h->err = t->err; return rc; }
        h->twin_gen = h->learn_gen;
    }
    return FPM_OK;
}

namespace {
// fpm_match_batch_device for the whole set: frame b / template t at out + (b * n_set + t) * cap, or (mg) frame b's merged
// list at out + b * cap
int match_batch_device(fpm_handle* h, const uint8_t* d_src, int batch, int width, int height, int stride,
                       size_t frame_stride, fpm_result* out, int cap, int* n, const SetMerge* mg = nullptr)
{
    const int n_set = std::max((int)h->set.size(), 1), n_rows = mg ? 1 : n_set;
    if (!n || batch < 0 || cap < 0 || (cap > 0 && !out)) { h->err = "bad output arguments"; return FPM_ERR_INVALID; }
    for (int b = 0; b < batch * n_rows; b++) n[b] = 0;
    if (!d_src || width <= 0 || height <= 0 || batch == 0) return FPM_OK;       // empty source -> empty result
    if (stride < width) { h->err = "stride < width"; return FPM_ERR_INVALID; }
    CK(cudaSetDevice(h->device));
    auto t0 = std::chrono::high_resolution_clock::now();
    int rc;
    if (h->split_batch > 0 && batch >= h->split_batch && !h->trace && h->learned &&
        (h->tol_range || h->tol_angle >= FPM_VISION_TOLERANCE)) {       // single-angle workloads gain nothing from it
        // Two half-batches on two handles (own streams and buffers), issued from two host threads: while one half
        // sits in a latency-bound stage (peak picking, the small pyramid levels, the per-layer counter read-back)
        // the other half's kernels fill the device.
        rc = ensure_twin(h);
        if (rc) return rc;
        h->twin->scales_out = h->scales_out; h->twin->scales_base = h->scales_base; h->twin->scaled_fn = h->scaled_fn;
        const int b0 = batch / 2;
        int rc2 = FPM_OK;
        const SetMerge mg2 = mg ? mg->shifted(b0, cap, n_set) : SetMerge{};
        std::thread second([&]() {
            rc2 = match_batch_device(h->twin, d_src + (size_t)b0 * frame_stride, batch - b0, width, height, stride, frame_stride,
                                     out + (size_t)b0 * n_rows * cap, cap, n + (size_t)b0 * n_rows, mg ? &mg2 : nullptr);
        });
        rc = match_device(h, d_src, b0, width, height, stride, frame_stride, out, cap, n, mg);
        second.join();
        if (rc == FPM_OK && rc2 != FPM_OK) { rc = rc2; h->err = h->twin->err; }
    } else {
        rc = match_device(h, d_src, batch, width, height, stride, frame_stride, out, cap, n, mg);
    }
    prof_collect(h);
    auto t1 = std::chrono::high_resolution_clock::now();
    h->last_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    return rc;
}

// fpm_match_batch for the whole set (mg: merged, as in match_batch_device)
int match_batch_host(fpm_handle* h, const uint8_t* src, int batch, int width, int height, int stride, size_t frame_stride,
                     fpm_result* out, int cap, int* n, const SetMerge* mg = nullptr)
{
    const int n_set = std::max((int)h->set.size(), 1), n_rows = mg ? 1 : n_set;
    if (!n || batch < 0 || cap < 0 || (cap > 0 && !out)) { h->err = "bad output arguments"; return FPM_ERR_INVALID; }
    for (int b = 0; b < batch * n_rows; b++) n[b] = 0;
    if (!src || width <= 0 || height <= 0 || batch == 0) return FPM_OK;
    if (stride < width) { h->err = "stride < width"; return FPM_ERR_INVALID; }
    CK(cudaSetDevice(h->device));
    auto t0 = std::chrono::high_resolution_clock::now();
    // double-buffered chunks: the H2D copy of chunk k+1 overlaps the matching of chunk k.
    // Contiguous frames whose width is a multiple of 4 keep their host layout on the device so that a
    // chunk is ONE linear copy (2D pitched copies from pinned memory run well below PCIe speed).
    const bool linear = (stride == width) && (width % 4 == 0) && (frame_stride == (size_t)stride * height) &&
                        (frame_stride % 4 == 0);
    const int pitch = linear ? width : (int)align_up(width, 128);
    const size_t img = linear ? frame_stride : align_up((size_t)pitch * height, 256);
    int chunk = std::max(1, std::min(batch, (int)std::max<size_t>(1, (size_t)(512ull << 20) / img)));
    // Chunk size by BYTES: about 96 MB = 1.7 ms of copy at the 55 GB/s of a PCIe 5 x16 link.  Measured on B200: matching c
    // cfg1 frames takes 0.63 + 0.073c ms, so from ~96 MB on the pipeline is copy-bound while the fill (the first chunk's
    // copy) and the drain (the last chunk's match) stay short -- 8 frames of 12 MB (cfg1..cfg4), ONE frame of 67 MB
    // (cfg5: +10 % against chunks of 4)
    const int by_bytes = (int)std::max<size_t>(1, ((size_t)(96ull << 20) + img / 2) / img);
    chunk = std::min(chunk, by_bytes);
    if (batch > 1) chunk = std::min(chunk, (batch + 1) / 2);
    if (h->h2d_chunk > 0) chunk = std::min(batch, h->h2d_chunk);
    const size_t buf_bytes = align_up(img * chunk, 256);
    CK(h->d_src.ensure(buf_bytes * 2));
    const int nchunks = (batch + chunk - 1) / chunk;
    auto enqueue_copy = [&](int k) -> cudaError_t {
        int b0 = k * chunk, nb = std::min(chunk, batch - b0);
        uint8_t* dst = h->d_src.as<uint8_t>() + (size_t)(k & 1) * buf_bytes;
        if (k >= 2) {
            cudaError_t e = cudaStreamWaitEvent(h->copy_stream, h->ev_done[k & 1], 0);
            if (e != cudaSuccess) return e;
        }
        if (linear) {
            cudaError_t e = cudaMemcpyAsync(dst, src + (size_t)b0 * frame_stride, (size_t)nb * frame_stride, cudaMemcpyHostToDevice,
                                            h->copy_stream);
            if (e != cudaSuccess) return e;
        } else {
            for (int b = 0; b < nb; b++) {
                cudaError_t e = cudaMemcpy2DAsync(dst + (size_t)b * img, pitch, src + (size_t)(b0 + b) * frame_stride, stride, width,
                                                  height, cudaMemcpyHostToDevice, h->copy_stream);
                if (e != cudaSuccess) return e;
            }
        }
        return cudaEventRecord(h->ev_copy[k & 1], h->copy_stream);
    };
    // every exit drains both streams: an H2D copy still in flight reads the caller's buffer
    auto fail_cuda = [&](const char* what, cudaError_t e) {
        h->err = std::string(what) + ": " + cudaGetErrorString(e);
        cudaStreamSynchronize(h->copy_stream);
        cudaStreamSynchronize(h->stream);
        return FPM_ERR_CUDA;
    };
    cudaError_t ce = enqueue_copy(0);
    if (ce != cudaSuccess) return fail_cuda("host->device copy", ce);
    int rc = FPM_OK;
    for (int k = 0; k < nchunks && rc == FPM_OK; k++) {
        if (k + 1 < nchunks && (ce = enqueue_copy(k + 1)) != cudaSuccess) return fail_cuda("host->device copy", ce);
        if ((ce = cudaStreamWaitEvent(h->stream, h->ev_copy[k & 1], 0)) != cudaSuccess) return fail_cuda("cudaStreamWaitEvent", ce);
        int b0 = k * chunk, nb = std::min(chunk, batch - b0);
        const SetMerge mgk = mg ? mg->shifted(b0, cap, n_set) : SetMerge{};
        rc = match_device(h, h->d_src.as<uint8_t>() + (size_t)(k & 1) * buf_bytes, nb, width, height, pitch, img,
                          out + (size_t)b0 * n_rows * cap, cap, n + (size_t)b0 * n_rows, mg ? &mgk : nullptr);
        if (rc == FPM_OK && (ce = cudaEventRecord(h->ev_done[k & 1], h->stream)) != cudaSuccess) return fail_cuda("cudaEventRecord", ce);
        prof_collect(h);
    }
    cudaStreamSynchronize(h->copy_stream);
    if (rc != FPM_OK) cudaStreamSynchronize(h->stream);
    auto t1 = std::chrono::high_resolution_clock::now();
    h->last_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    return rc;
}
}  // namespace

int fpm_match_batch_device(fpm_handle* h, const uint8_t* d_src, int batch, int width, int height, int stride,
                           size_t frame_stride, fpm_result* out, int cap, int* n)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_batch_device")) return rc;
    return match_batch_device(h, d_src, batch, width, height, stride, frame_stride, out, cap, n);
}

int fpm_match_batch(fpm_handle* h, const uint8_t* src, int batch, int width, int height, int stride, size_t frame_stride,
                    fpm_result* out, int cap, int* n)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_batch")) return rc;
    return match_batch_host(h, src, batch, width, height, stride, frame_stride, out, cap, n);
}

namespace {
int check_merge_args(fpm_handle* h, const char* fn, double max_overlap, int cap, const int* labels)
{
    if (!std::isfinite(max_overlap)) { h->err = std::string(fn) + ": max_overlap must be finite"; return FPM_ERR_INVALID; }
    if (cap > 0 && !labels) { h->err = std::string(fn) + ": labels is NULL while cap > 0"; return FPM_ERR_INVALID; }
    return FPM_OK;
}

// fpm_match_set_batch / fpm_match_set_batch_merged (mg) and their scaled twins; fn names the call in the refusals
int match_set(fpm_handle* h, const char* fn, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
              size_t frame_stride, fpm_result* out, int cap, int* counts, const SetMerge* mg)
{
    if (h->trace && fpm_set_size(h) > 1) {
        h->err = std::string(fn) + ": FPM_PARAM_TRACE is not supported for a set of more than one template";
        return FPM_ERR_INVALID;
    }
    if (mg) {
        if (int rc = check_merge_args(h, fn, mg->max_overlap, cap, mg->labels)) return rc;
        if (mg->set_counts && batch > 0) std::fill(mg->set_counts, mg->set_counts + (size_t)batch * std::max(fpm_set_size(h), 1), 0);
    }
    return src_on_device ? match_batch_device(h, src, batch, width, height, stride, frame_stride, out, cap, counts, mg)
                         : match_batch_host(h, src, batch, width, height, stride, frame_stride, out, cap, counts, mg);
}
}  // namespace

int fpm_match_set_batch(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                        size_t frame_stride, fpm_result* out, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    return match_set(h, "fpm_match_set_batch", src, src_on_device, batch, width, height, stride, frame_stride, out, cap, counts, nullptr);
}

int fpm_match_set_batch_merged(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                               size_t frame_stride, double max_overlap, fpm_result* out, int* labels, int cap, int* counts,
                               int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    const SetMerge mg{max_overlap, labels, set_counts};
    return match_set(h, "fpm_match_set_batch_merged", src, src_on_device, batch, width, height, stride, frame_stride, out, cap,
                     counts, &mg);
}

int fpm_match(fpm_handle* h, const uint8_t* src, int width, int height, int stride, fpm_result* out, int cap, int* n)
{
    if (h) if (int rc = refuse_set(h, "fpm_match")) return rc;
    return fpm_match_batch(h, src, 1, width, height, stride, (size_t)stride * (size_t)std::max(height, 0), out, cap, n);
}

// Multi-template matching ("NCC-based OCR", MatchTool/MatchToolDlg.cpp:727-750: LoadDst + Match per glyph).  Every
// handle owns its stream and buffers, so the matches are independent: they are issued from a small pool of host
// threads and overlap on the device (each single match is launch-latency bound, not throughput bound).
int fpm_match_multi(fpm_handle* const* hs, int n_handles, const uint8_t* src, int width, int height, int stride,
                    fpm_result* out, int cap, int* counts)
{
    if (!hs || n_handles <= 0 || !src || !out || !counts || cap < 0) return FPM_ERR_INVALID;
    for (int i = 0; i < n_handles; i++)
        if (!hs[i]) return FPM_ERR_INVALID;
    for (int i = 0; i < n_handles; i++)
        if (int rc = refuse_set(hs[i], "fpm_match_multi")) return rc;
    for (int i = 0; i < n_handles; i++) counts[i] = 0;
    if (width <= 0 || height <= 0) return FPM_OK;
    if (stride < width) return FPM_ERR_INVALID;
    // One upload and ONE source pyramid for all templates (the upstream loop re-reads the same image for every glyph,
    // MatchToolDlg.cpp:727-750): the first handle uploads the frame and builds the pyramid down to the deepest top layer
    // any template needs; the other handles' streams wait on its event and match against the shared levels.
    bool share = true;
    int max_top = 0;
    for (int i = 0; i < n_handles; i++) {
        fpm_handle* h = hs[i];
        if (!h->learned || h->device != hs[0]->device || h->bitwise_not || h->trace) { share = false; break; }
        if (ensure_learned_for_mra(h) != FPM_OK) { share = false; break; }
        max_top = std::max(max_top, (int)h->tpl.size() - 1);
    }
    fpm_handle* lead = hs[0];
    int pitch = 0;
    size_t img = 0;
    if (share) {
        fpm_handle* h = lead;
        CK(cudaSetDevice(h->device));
        pitch = (int)align_up(width, 128);
        img = align_up((size_t)pitch * height, 256);
        CK(h->d_src.ensure(img));
        CK(cudaMemcpy2DAsync(h->d_src.p, pitch, src, stride, width, height, cudaMemcpyHostToDevice, h->stream));
        h->shared_levels = nullptr;
        int rc = build_pyramid(h, h->d_src.as<uint8_t>(), 1, width, height, pitch, img, max_top);
        if (rc) return rc;
        CK(cudaEventRecord(h->ev_fork, h->stream));
    }
    const int n_threads = std::min(n_handles, 12);
    std::vector<int> rc(n_handles, FPM_OK);
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++)
        pool.emplace_back([&, t]() {
            for (int i = t; i < n_handles; i += n_threads) {
                fpm_handle* h = hs[i];
                if (!share) {
                    rc[i] = fpm_match(h, src, width, height, stride, out + (size_t)i * cap, cap, counts + i);
                    continue;
                }
                cudaSetDevice(h->device);
                if (h != lead && cudaStreamWaitEvent(h->stream, lead->ev_fork, 0) != cudaSuccess) { rc[i] = FPM_ERR_CUDA; continue; }
                h->shared_levels = &lead->levels;
                rc[i] = match_device(h, lead->d_src.as<uint8_t>(), 1, width, height, pitch, img, out + (size_t)i * cap, cap, counts + i);
                h->shared_levels = nullptr;
                prof_collect(h);
            }
        });
    for (std::thread& th : pool) th.join();
    for (int i = 0; i < n_handles; i++)
        if (rc[i] != FPM_OK) return rc[i];
    return FPM_OK;
}

// Text assembly of the OCR loop (MatchToolDlg.cpp:752-771): sort by y, every run of neighbours closer than
// line_tol in y is a line sorted by x, newline where consecutive entries are farther apart than line_tol.
// (std::sort there leaves ties unspecified; stable sorts here, like the oracle.)
int fpm_ocr_assemble(const double* cx, const double* cy, const char* labels, int n, double line_tol, char* out, int out_cap)
{
    if (n < 0 || !out || out_cap <= 0 || (n > 0 && (!cx || !cy || !labels))) return FPM_ERR_INVALID;
    std::vector<int> idx(n);
    for (int i = 0; i < n; i++) idx[i] = i;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return cy[a] < cy[b]; });
    auto by_x = [&](int a, int b) { return cx[a] < cx[b]; };
    int start = 0;
    for (int i = 0; i + 1 < n; i++) {
        if (fabs(cy[idx[i + 1]] - cy[idx[i]]) < line_tol) continue;
        std::stable_sort(idx.begin() + start, idx.begin() + i + 1, by_x);
        start = i + 1;
    }
    if (n > 0) std::stable_sort(idx.begin() + start, idx.end(), by_x);
    std::string text;
    for (int i = 0; i < n; i++) {
        if (i > 0 && fabs(cy[idx[i]] - cy[idx[i - 1]]) > line_tol) text += '\n';
        text += labels[idx[i]];
    }
    if ((int)text.size() + 1 > out_cap) return FPM_ERR_LIMIT;
    memcpy(out, text.c_str(), text.size() + 1);
    return (int)text.size();
}

// ---- image ingest (SURVEY 8f rank 4) ---------------------------------------------------------------------
namespace {
uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
uint32_t rd16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
}  // namespace

int fpm_ingest_bmp(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height)
{
    if (!h) return FPM_ERR_INVALID;
    h->ingest_count = 0;
    if (!file || nbytes < 54 || file[0] != 'B' || file[1] != 'M') { h->err = "not a BMP file"; return FPM_ERR_INVALID; }
    const uint32_t off = rd32(file + 10), dib = rd32(file + 14);
    if (dib < 40) { h->err = "unsupported BMP header (OS/2 core header)"; return FPM_ERR_INVALID; }
    // untrusted header fields: everything is range-checked in 64 bits before it sizes a buffer or a kernel
    const int64_t w64 = (int32_t)rd32(file + 18), hs64 = (int32_t)rd32(file + 22);
    const int bpp = (int)rd16(file + 28);
    const uint32_t comp = rd32(file + 30), clr_used = rd32(file + 46);
    const int top_down = hs64 < 0;
    const int64_t hh64 = top_down ? -hs64 : hs64;
    if (w64 <= 0 || hh64 <= 0 || comp != 0 || (bpp != 8 && bpp != 24)) {
        h->err = "unsupported BMP (only uncompressed 8-bit palettized and 24-bit BGR)";
        return FPM_ERR_INVALID;
    }
    if (w64 > (1 << 20) || hh64 > 65535 || w64 * hh64 > (1ll << 30)) {          // OpenCV's CV_IO_MAX_IMAGE_PIXELS = 2^30; one grid row per image row
        h->err = "BMP dimensions out of range";
        return FPM_ERR_INVALID;
    }
    const int w = (int)w64, hh = (int)hh64;
    const size_t row_stride = ((size_t)w * bpp + 31) / 32 * 4;
    const size_t pal_end = 14 + (size_t)dib + (bpp == 8 ? (size_t)(clr_used ? std::min<uint32_t>(clr_used, 256) : 256) * 4 : 0);
    if ((size_t)off < 14 + (size_t)dib || (size_t)off > nbytes || row_stride * (size_t)hh > nbytes - off) {
        h->err = "truncated BMP";
        return FPM_ERR_INVALID;
    }
    (void)pal_end;
    FpmBmpLut lut;
    memset(&lut, 0, sizeof(lut));
    if (bpp == 8) {
        const uint32_t n_pal = clr_used ? std::min<uint32_t>(clr_used, 256) : 256;
        const size_t pal_off = 14 + (size_t)dib;
        if (pal_off + (size_t)n_pal * 4 > nbytes) { h->err = "truncated BMP palette"; return FPM_ERR_INVALID; }
        for (uint32_t i = 0; i < n_pal; i++) {                       // CvtPaletteToGray: same weights as the 24-bit path
            const uint8_t* e = file + pal_off + (size_t)i * 4;
            lut.g[i] = (uint8_t)(((uint32_t)e[0] * 1868u + (uint32_t)e[1] * 9617u + (uint32_t)e[2] * 4899u + 8192u) >> 14);
        }
    }
    CK(cudaSetDevice(h->device));
    CK(h->d_ingest_raw.ensure(nbytes));
    const int pitch = (int)align_up(w, 128);
    CK(h->d_ingest.ensure((size_t)pitch * hh));
    CK(cudaMemcpyAsync(h->d_ingest_raw.p, file, nbytes, cudaMemcpyHostToDevice, h->stream));
    dim3 grid((w + 255) / 256, hh);
    fpm_ingest_bmp_kernel<<<grid, 256, 0, h->stream>>>(h->d_ingest_raw.as<uint8_t>(), (size_t)off, row_stride, bpp, top_down, lut, w, hh,
                                                       h->d_ingest.as<uint8_t>(), pitch);
    CKL();
    CK(cudaStreamSynchronize(h->stream));                             // the caller's file buffer is free again
    h->ingest_w = w; h->ingest_h = hh; h->ingest_pitch = pitch; h->ingest_count = 1;
    if (width) *width = w;
    if (height) *height = hh;
    return FPM_OK;
}

// ---- JPEG ingest ------------------------------------------------------------------------------------------------------
// entropy-coded segment without the 0xFF00 stuffing and without the RSTn markers (their positions go to rst_bits: first bit of
// every restart interval + a final sentinel); stops at the first other marker (EOI).  out needs n - begin + 16 bytes; the 16
// bytes after the data are zero (the device reader looks a few bytes ahead).  Returns the number of data bytes.  The sequential
// reference of the device unstuffing (jp_unstuff_*, fpm_jpeg_par.cuh): fpm_dbg_jpeg_unstuff runs both.
size_t jpeg_unstuff(const uint8_t* d, size_t n, size_t begin, uint8_t* out, std::vector<unsigned>* rst_bits)
{
    size_t i = begin, o = 0;
    if (rst_bits) { rst_bits->clear(); rst_bits->push_back(0); }
    while (i < n) {
        const uint8_t* ff = static_cast<const uint8_t*>(memchr(d + i, 0xFF, n - i));
        const size_t run = ff ? (size_t)(ff - (d + i)) : n - i;
        memcpy(out + o, d + i, run);
        o += run; i += run;
        if (!ff || i + 1 >= n) break;
        if (d[i + 1] == 0x00) { out[o++] = 0xFF; i += 2; }
        else if (d[i + 1] == 0xFF) { i++; }                              // fill byte
        else if (rst_bits && d[i + 1] >= 0xD0 && d[i + 1] <= 0xD7) { rst_bits->push_back((unsigned)(o * 8)); i += 2; }   // RSTn: next interval
        else break;                                                     // a marker: end of the scan
    }
    memset(out + o, 0, 16);
    if (rst_bits) rst_bits->push_back((unsigned)(o * 8));               // sentinel: rst[nint] = nbits
    return o;
}

// device tables and scan geometry of a parsed frame (fpm_jpeg_par.cuh)
void jpeg_device_tables(const fpm_jpeg::Frame& fr, JpTable* tabs /* 8 */, JpScan* sc, size_t scan_bytes)
{
    for (int t = 0; t < 8; t++) {
        JpTable& T = tabs[t];
        memset(&T, 0, sizeof(T));
        const uint8_t* counts = t < 4 ? fr.dc_counts[t] : fr.ac_counts[t - 4];
        const uint8_t* syms = t < 4 ? fr.dc_syms[t] : fr.ac_syms[t - 4];
        if (!(t < 4 ? fr.dc[t].defined : fr.ac[t - 4].defined)) continue;
        uint32_t code = 0;
        int k = 0;
        for (int l = 1; l <= 16; l++) {
            T.valoff[l] = k - (int)code;
            for (int i = 0; i < counts[l - 1] && k < 256; i++, k++, code++) {
                T.sym[k] = syms[k];
                if (l <= 9 && code < (1u << l))
                    for (uint32_t j = 0; j < (1u << (9 - l)); j++) T.fast[(code << (9 - l)) + j] = (uint16_t)((l << 8) | syms[k]);
            }
            T.limit[l] = std::min<uint32_t>(code, 1u << l) << (16 - l);
            code <<= 1;
        }
    }
    memset(sc, 0, sizeof(*sc));
    int slot = 0;
    for (size_t c = 0; c < fr.comp.size(); c++)
        for (int b = 0; b < fr.comp[c].h * fr.comp[c].v; b++, slot++) {
            sc->dc_tab[slot] = fr.comp[c].td;
            sc->ac_tab[slot] = 4 + fr.comp[c].ta;
        }
    sc->nslots = slot;
    sc->luma_h = fr.comp[0].h; sc->luma_v = fr.comp[0].v; sc->luma_slots = sc->luma_h * sc->luma_v;
    sc->mcux = fr.mcux; sc->mcuy = fr.mcuy; sc->bw = fr.mcux * fr.comp[0].h;
    sc->total_blocks = (unsigned)fr.mcux * fr.mcuy * slot;
    sc->nbits = (unsigned)(scan_bytes * 8);
    sc->nsub = (int)((sc->nbits + JP_SUB_BITS - 1) / JP_SUB_BITS);
    sc->restart_blocks = (unsigned)fr.restart_interval * slot;
    sc->nint = 1;
    sc->rst = nullptr;
}

// number of restart intervals the frame header promises
int jpeg_expected_intervals(const fpm_jpeg::Frame& fr)
{
    if (!fr.restart_interval) return 1;
    const long long mcus = (long long)fr.mcux * fr.mcuy;
    return (int)((mcus + fr.restart_interval - 1) / fr.restart_interval);
}

// can the scan be decoded by the parallel decoder?  (sizes inside its 32-bit bit positions)
bool jpeg_device_ok(const fpm_jpeg::Frame& fr, size_t file_bytes)
{
    int slots = 0;
    for (auto& c : fr.comp) slots += c.h * c.v;
    return slots <= JP_MAX_SLOTS && file_bytes < (400u << 20);
}

// ---- batches: the files of one fpm_ingest_jpeg_batch call (one file for fpm_ingest_jpeg) --------------------------------
struct JpegBatchFile {
    fpm_jpeg::Frame fr;
    size_t off = 0, nbytes = 0;    // the file is data[off, off + nbytes)
    bool device = false;           // Huffman decoding on the device (else on the host, fpm_jpeg.h)
};

std::string jpeg_file_prefix(int i, int n) { return n > 1 ? "JPEG file " + std::to_string(i) + " of the batch: " : std::string(); }

// headers of every file (the host reads nothing past them); same_size: all frames must have file 0's size
int jpeg_batch_parse(const uint8_t* data, const size_t* offsets, int n, bool same_size, std::vector<JpegBatchFile>* fs, std::string* err)
{
    if (n <= 0) { *err = "empty JPEG batch"; return FPM_ERR_INVALID; }
    if (!data || !offsets) { *err = "null JPEG batch buffer or offsets"; return FPM_ERR_INVALID; }
    for (int i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) { *err = "JPEG batch offsets decrease at file " + std::to_string(i); return FPM_ERR_INVALID; }
    fs->resize(n);
    for (int i = 0; i < n; i++) {
        JpegBatchFile& f = (*fs)[i];
        f.off = offsets[i];
        f.nbytes = offsets[i + 1] - offsets[i];
        const std::string why = fpm_jpeg::parse(data + f.off, f.nbytes, &f.fr);
        if (!why.empty()) { *err = jpeg_file_prefix(i, n) + why; return FPM_ERR_INVALID; }
        if ((size_t)f.fr.height * f.fr.width > ((size_t)1 << 30)) {
            *err = jpeg_file_prefix(i, n) + "JPEG too large (more than 2^30 pixels, OpenCV's own limit)";
            return FPM_ERR_LIMIT;
        }
        const fpm_jpeg::Frame& f0 = (*fs)[0].fr;
        if (same_size && (f.fr.width != f0.width || f.fr.height != f0.height)) {
            *err = "JPEG file " + std::to_string(i) + " of the batch is " + std::to_string(f.fr.width) + "x" + std::to_string(f.fr.height) +
                   ", file 0 is " + std::to_string(f0.width) + "x" + std::to_string(f0.height) + ": the frames of a batch must have one size";
            return FPM_ERR_INVALID;
        }
    }
    return FPM_OK;
}

// where every file's unstuffing reads and writes (offsets relative to data[offsets[0]]); files decoded on the host get no tiles
struct JpUnstuffPlan {
    std::vector<JpUnstuff> u;
    std::vector<int> tile_first;   // n + 1
    size_t out_bytes = 0, rst_entries = 0;
};

void jpeg_unstuff_plan(const std::vector<JpegBatchFile>& fs, size_t base, JpUnstuffPlan* p)
{
    const int n = (int)fs.size();
    p->u.assign(n, JpUnstuff{});
    p->tile_first.assign(n + 1, 0);
    int tiles = 0;
    for (int i = 0; i < n; i++) {
        JpUnstuff& u = p->u[i];
        p->tile_first[i] = tiles;
        if (!fs[i].device) continue;
        u.begin = fs[i].off - base + fs[i].fr.scan_begin;
        u.end = fs[i].off - base + fs[i].nbytes;
        u.stop = u.end;
        u.out = p->out_bytes;
        p->out_bytes += align_up(u.end - u.begin, 4) + 16;
        u.restart = fs[i].fr.restart_interval != 0;
        u.rst = p->rst_entries;
        u.rst_cap = u.restart ? jpeg_expected_intervals(fs[i].fr) + 2 : 0;     // more markers than that: the host decoder takes it
        p->rst_entries += u.rst_cap;
        tiles += (int)((u.end - u.begin + 1 + JP_UNSTUFF_TILE - 1) / JP_UNSTUFF_TILE);
    }
    p->tile_first[n] = tiles;
}

// the unstuffing kernels run tile by tile, thread by thread on the CPU (d = data[offsets[0]])
void jpeg_unstuff_emulate(const uint8_t* d, JpUnstuffPlan* p, uint8_t* out, unsigned* rst)
{
    const int n = (int)p->u.size(), ntiles = p->tile_first[n];
    std::vector<unsigned long long> tile_sum(ntiles);
    for (int t = 0; t < ntiles; t++) {                                  // fpm_jpeg_unstuff_count_kernel
        const int fi = jp_file_of(p->tile_first.data(), n, t);
        JpUnstuff& f = p->u[fi];
        unsigned long long sum = 0;
        for (int k = 0; k < JP_UNSTUFF_THREADS; k++) {
            unsigned long long a, b, s = ~0ull;
            unsigned e = 0, r = 0;
            jp_unstuff_chunk(f, t - p->tile_first[fi], k, &a, &b);
            if (a < b) jp_unstuff_count(d, f, a, b, &e, &r, &s);
            f.stop = std::min(f.stop, s);
            sum += ((unsigned long long)e << 32) | r;
        }
        tile_sum[t] = sum;
    }
    for (int fi = 0; fi < n; fi++) {                                    // fpm_jpeg_offsets_kernel
        unsigned long long run = 0;
        for (int t = p->tile_first[fi]; t < p->tile_first[fi + 1]; t++) { const unsigned long long v = tile_sum[t]; tile_sum[t] = run; run += v; }
    }
    for (int t = 0; t < ntiles; t++) {                                  // fpm_jpeg_unstuff_write_kernel
        const int fi = jp_file_of(p->tile_first.data(), n, t);
        JpUnstuff& f = p->u[fi];
        unsigned long long x = tile_sum[t];
        for (int k = 0; k < JP_UNSTUFF_THREADS; k++) {
            unsigned long long a, b, s;
            unsigned e = 0, r = 0;
            jp_unstuff_chunk(f, t - p->tile_first[fi], k, &a, &b);
            if (a < b) jp_unstuff_count(d, f, a, b, &e, &r, &s);
            if (a < b && a <= f.stop) jp_unstuff_write(d, f, a, b, (unsigned)(x >> 32), (unsigned)x, out, rst);
            x += ((unsigned long long)e << 32) | r;
        }
    }
}

// decoder descriptors of the files [f0, f1) of a batch (after the unstuffing); rst_base: the rst array the decoder reads
struct JpWave {
    std::vector<JpFile> files;
    std::vector<int> cta_first, bseg, dseg;        // f1 - f0 + 1 entries each
    size_t coef_elems = 0;
    int nsub = 0, nluma = 0, max_nsub = 0;         // state / DC array lengths (padded per file)
};

void jpeg_wave_plan(const std::vector<JpegBatchFile>& fs, const JpUnstuffPlan& up, int f0, int f1, const unsigned* rst_base, int pitch, JpWave* w)
{
    const int m = f1 - f0;
    w->files.assign(m, JpFile{});
    w->cta_first.assign(m + 1, 0); w->bseg.assign(m + 1, 0); w->dseg.assign(m + 1, 0);
    int ctas = 0;
    for (int k = 0; k < m; k++) {
        const JpegBatchFile& b = fs[f0 + k];
        const JpUnstuff& u = up.u[f0 + k];
        JpFile& f = w->files[k];
        memset(&f, 0, sizeof(f));
        jpeg_device_tables(b.fr, f.tabs, &f.sc, b.device ? u.nbits / 8 : 0);
        if (!b.device) f.sc.nsub = 0;
        else if (b.fr.restart_interval) { f.sc.nint = u.nint; f.sc.rst = rst_base + u.rst; }
        memcpy(f.quant, b.fr.qt[b.fr.comp[0].tq], sizeof(f.quant));
        f.bits = u.out;
        f.coef = w->coef_elems;
        w->coef_elems += (size_t)f.sc.bw * f.sc.mcuy * f.sc.luma_v * 64;
        f.frame = (size_t)(f0 + k) * pitch * b.fr.height;
        f.sub0 = w->nsub;
        f.luma0 = w->nluma;
        f.width = b.fr.width; f.height = b.fr.height;
        f.device_huffman = b.device;
        w->cta_first[k] = ctas; w->bseg[k] = f.sub0 / 4096; w->dseg[k] = f.luma0 / JP_DC_TILE;
        ctas += (f.sc.nsub + JP_THREADS - 1) / JP_THREADS;
        w->nsub += (int)align_up(f.sc.nsub, 4096);
        if (b.device) w->nluma += (int)align_up((size_t)f.sc.mcux * f.sc.mcuy * f.sc.luma_slots, JP_DC_TILE);
        w->max_nsub = std::max(w->max_nsub, f.sc.nsub);
    }
    w->cta_first[m] = ctas; w->bseg[m] = w->nsub / 4096; w->dseg[m] = w->nluma / JP_DC_TILE;
}

// device bytes one file needs in a decode wave: coefficients (2 B per luma pixel), decoder states, DC values
size_t jpeg_wave_bytes(const JpegBatchFile& b, const JpUnstuff& u)
{
    const size_t luma = (size_t)b.fr.mcux * b.fr.comp[0].h * b.fr.mcuy * b.fr.comp[0].v;
    size_t bytes = luma * 64 * sizeof(int16_t);
    if (b.device) {
        const size_t nsub = (u.nbits + JP_SUB_BITS - 1) / JP_SUB_BITS;
        bytes += align_up(nsub, 4096) * (3 * sizeof(JpState) + 4) + align_up(luma, JP_DC_TILE) * 4 * 2;
    }
    return bytes;
}

// Huffman decoding of the device files of a wave + dequantisation / IDCT of all its files into their frame slots
int jpeg_decode_wave(fpm_handle* h, const std::vector<JpegBatchFile>& fs, const uint8_t* data, const JpUnstuffPlan& up, int f0, int f1,
                     const uint8_t* bits, const unsigned* rst, int pitch, int* passes_out)
{
    const int m = f1 - f0;
    JpWave w;
    jpeg_wave_plan(fs, up, f0, f1, rst, pitch, &w);
    std::vector<fpm_jpeg::Luma> host(m);
    for (int k = 0; k < m; k++)
        if (!fs[f0 + k].device) {
            const JpegBatchFile& b = fs[f0 + k];
            const std::string why = fpm_jpeg::decode_scan_host(b.fr, data + b.off, b.nbytes, &host[k]);
            if (!why.empty()) { h->err = jpeg_file_prefix(f0 + k, (int)fs.size()) + why; return FPM_ERR_INVALID; }
        }
    // d_jpeg: [descriptors | cta_first | bseg | dseg] [3 state arrays | first-block index | block tile offsets | DC values |
    // DC tile offsets | flag]
    const size_t o_cta = align_up((size_t)m * sizeof(JpFile), 256), o_bseg = o_cta + align_up((m + 1) * 4, 256);
    const size_t o_dseg = o_bseg + align_up((m + 1) * 4, 256), desc_bytes = o_dseg + (m + 1) * 4;
    const size_t S = (size_t)w.nsub, L = (size_t)w.nluma, st_bytes = align_up(S * sizeof(JpState), 256);
    const size_t o_st = align_up(desc_bytes, 256), o_first = o_st + 3 * st_bytes, o_btile = o_first + align_up(S * 4, 256);
    const size_t o_dc = o_btile + align_up(S / 4096 * 4 + 4, 256), o_dtile = o_dc + align_up(L * 4, 256);
    const size_t o_flag = o_dtile + align_up(L / JP_DC_TILE * 4 + 4, 256);
    CK(h->d_jpeg.ensure(o_flag + 256));
    const size_t cbytes = w.coef_elems * sizeof(int16_t);
    CK(h->d_ingest_raw.ensure(cbytes));
    CK(h->h_stage.ensure(desc_bytes));
    uint8_t* hs = h->h_stage.as<uint8_t>();
    memcpy(hs, w.files.data(), (size_t)m * sizeof(JpFile));
    memcpy(hs + o_cta, w.cta_first.data(), (m + 1) * 4);
    memcpy(hs + o_bseg, w.bseg.data(), (m + 1) * 4);
    memcpy(hs + o_dseg, w.dseg.data(), (m + 1) * 4);
    uint8_t* base = h->d_jpeg.as<uint8_t>();
    CK(cudaMemcpyAsync(base, hs, desc_bytes, cudaMemcpyHostToDevice, h->stream));
    const JpFile* files = reinterpret_cast<const JpFile*>(base);
    const int* cta_first = reinterpret_cast<const int*>(base + o_cta);
    int16_t* coef = h->d_ingest_raw.as<int16_t>();
    CK(cudaMemsetAsync(coef, 0, cbytes, h->stream));
    for (int k = 0; k < m; k++)
        if (!fs[f0 + k].device)
            CK(cudaMemcpyAsync(coef + w.files[k].coef, host[k].coef.data(), host[k].coef.size() * sizeof(int16_t), cudaMemcpyHostToDevice, h->stream));
    JpState* st[2] = {reinterpret_cast<JpState*>(base + o_st), reinterpret_cast<JpState*>(base + o_st + st_bytes)};
    JpState* used = reinterpret_cast<JpState*>(base + o_st + 2 * st_bytes);
    unsigned* first = reinterpret_cast<unsigned*>(base + o_first);
    int* btile_off = reinterpret_cast<int*>(base + o_btile);
    int* dcval = reinterpret_cast<int*>(base + o_dc);
    int* dtile_off = reinterpret_cast<int*>(base + o_dtile);
    int* flag = reinterpret_cast<int*>(base + o_flag);
    const int nb = w.cta_first[m];
    int passes = 0;
    if (nb > 0) {
        KL(K_JPEG_PASSES, S, fpm_jpeg_cold_kernel<<<nb, JP_THREADS, 0, h->stream>>>(files, cta_first, m, bits, st[0], used));
        // synchronisation passes, two per flag read-back (a pass in which no entry state moved costs a few microseconds: its
        // CTAs leave before they stage anything)
        int cur = 0;
        CK(h->h_counts.ensure(256));
        int* hflag = h->h_counts.as<int>();
        for (;;) {
            if (passes > w.max_nsub + 2) { h->err = "JPEG scan did not synchronise"; return FPM_ERR_INVALID; }
            CK(cudaMemsetAsync(flag, 0, 8, h->stream));
            for (int k = 0; k < 2; k++) {
                KL(K_JPEG_PASSES, S, fpm_jpeg_sync_kernel<<<nb, JP_THREADS, 0, h->stream>>>(files, cta_first, m, bits, st[cur], st[cur ^ 1], used, flag + k));
                cur ^= 1;
            }
            CK(cudaMemcpyAsync(hflag, flag, 8, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            passes += hflag[0] ? 2 : 1;                               // passes that did work (+ the one that found the fixed point)
            if (!hflag[1]) break;
        }
        const int* bseg = reinterpret_cast<const int*>(base + o_bseg);
        const int* dseg = reinterpret_cast<const int*>(base + o_dseg);
        KL(K_JPEG_SCAN, S * 16, fpm_jpeg_block_tile_kernel<<<(int)(S / 4096), 256, 0, h->stream>>>(st[cur], (int)S, first, btile_off));
        KL(K_JPEG_SCAN, S / 4096 * 4, fpm_jpeg_offsets_kernel<int><<<m, 1024, 0, h->stream>>>(bseg, btile_off));
        KL(K_JPEG_WRITE, cbytes, fpm_jpeg_write_kernel<<<nb, JP_THREADS, 0, h->stream>>>(files, cta_first, m, bits, st[cur], first, btile_off, coef, dcval));
        if (L > 0) {
            KL(K_JPEG_SCAN, L * 8, fpm_jpeg_dc_tile_kernel<<<(int)(L / JP_DC_TILE), 256, 0, h->stream>>>((int)L, dcval, dtile_off));
            KL(K_JPEG_SCAN, L / JP_DC_TILE * 4, fpm_jpeg_offsets_kernel<int><<<m, 1024, 0, h->stream>>>(dseg, dtile_off));
        }
    }
    int max_blocks = 0;
    for (const JpFile& f : w.files) max_blocks = std::max(max_blocks, f.sc.bw * f.sc.mcuy * f.sc.luma_v);
    KL(K_JPEG_IDCT, cbytes, fpm_ingest_jpeg_idct_kernel<<<dim3((max_blocks + 127) / 128, m), 128, 0, h->stream>>>(
                                files, coef, dcval, dtile_off, h->d_ingest.as<uint8_t>(), pitch));
    CK(cudaStreamSynchronize(h->stream));                             // the stage buffer and the host coefficients are free again
    *passes_out = passes;
    return FPM_OK;
}

// n JPEG file images -> n device-resident frames [n][height][pitch].  The host reads the headers only: the span of all files
// goes to the device in one copy, the unstuffing kernels read back one record per file (nbits, nint), and the files are
// decoded in waves that fit FPM_PARAM_WORKSPACE_MB.  A file whose restart markers do not match its header (damaged) is
// Huffman-decoded on the host, like every file with FPM_PARAM_JPEG_DEVICE_HUFFMAN = 0; dequantisation + IDCT + range limit
// run on the device for all.
static int ingest_jpeg_batch_impl(fpm_handle* h, const uint8_t* data, const size_t* offsets, int n, int* width, int* height)
{
    std::vector<JpegBatchFile> fs;
    int rc = jpeg_batch_parse(data, offsets, n, true, &fs, &h->err);
    if (rc) return rc;
    for (JpegBatchFile& f : fs) f.device = h->jpeg_device_huffman && jpeg_device_ok(f.fr, f.nbytes);
    CK(cudaSetDevice(h->device));
    const size_t base = offsets[0], span = offsets[n] - base;
    JpUnstuffPlan up;
    jpeg_unstuff_plan(fs, base, &up);
    const int ntiles = up.tile_first[n];
    // d_jpeg_scan: [the files | unstuffed scans | rst | unstuffing records | tile_first | tile sums]
    const size_t o_out = align_up(span, 256), o_rst = o_out + align_up(up.out_bytes, 256), o_u = o_rst + align_up(up.rst_entries * 4, 256);
    const size_t o_tf = o_u + align_up((size_t)n * sizeof(JpUnstuff), 256), o_ts = o_tf + align_up((size_t)(n + 1) * 4, 256);
    CK(h->d_jpeg_scan.ensure(o_ts + (size_t)ntiles * 8 + 256));
    uint8_t* sb = h->d_jpeg_scan.as<uint8_t>();
    if (ntiles > 0) {
        prof_begin(h);
        CK(cudaMemcpyAsync(sb, data + base, span, cudaMemcpyHostToDevice, h->stream));
        prof_end(h, K_JPEG_UPLOAD, (double)span);
        const size_t rec_bytes = o_ts - o_u;
        CK(h->h_stage.ensure(rec_bytes));
        uint8_t* hs = h->h_stage.as<uint8_t>();
        memcpy(hs, up.u.data(), (size_t)n * sizeof(JpUnstuff));
        memcpy(hs + (o_tf - o_u), up.tile_first.data(), (size_t)(n + 1) * 4);
        CK(cudaMemcpyAsync(sb + o_u, hs, rec_bytes, cudaMemcpyHostToDevice, h->stream));
        JpUnstuff* u_dev = reinterpret_cast<JpUnstuff*>(sb + o_u);
        const int* tf_dev = reinterpret_cast<const int*>(sb + o_tf);
        unsigned long long* ts_dev = reinterpret_cast<unsigned long long*>(sb + o_ts);
        KL(K_JPEG_UNSTUFF, span, fpm_jpeg_unstuff_count_kernel<<<ntiles, JP_UNSTUFF_THREADS, 0, h->stream>>>(sb, u_dev, tf_dev, n, ts_dev));
        KL(K_JPEG_SCAN, ntiles * 8, fpm_jpeg_offsets_kernel<unsigned long long><<<n, 1024, 0, h->stream>>>(tf_dev, ts_dev));
        KL(K_JPEG_UNSTUFF, span, fpm_jpeg_unstuff_write_kernel<<<ntiles, JP_UNSTUFF_THREADS, 0, h->stream>>>(sb, u_dev, tf_dev, n, ts_dev, sb + o_out,
                                                                                                     reinterpret_cast<unsigned*>(sb + o_rst)));
        CK(cudaMemcpyAsync(hs, u_dev, (size_t)n * sizeof(JpUnstuff), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(up.u.data(), hs, (size_t)n * sizeof(JpUnstuff));
    }
    for (int i = 0; i < n; i++) {
        if (!fs[i].device) continue;
        if (up.u[i].nbits == 0) { h->err = jpeg_file_prefix(i, n) + "JPEG without image data"; return FPM_ERR_INVALID; }
        if (fs[i].fr.restart_interval && up.u[i].nint != jpeg_expected_intervals(fs[i].fr))
            fs[i].device = false;                                   // e.g. a restart marker is missing: the host decoder says what is wrong
    }
    const int W = fs[0].fr.width, H = fs[0].fr.height, pitch = (int)align_up(W, 128);
    CK(h->d_ingest.ensure((size_t)n * pitch * H));
    const size_t budget = (size_t)std::max(0.0, h->workspace_mb * 1024.0 * 1024.0);
    int max_passes = 0;
    for (int f0 = 0; f0 < n;) {
        size_t need = 0;
        int f1 = f0;
        while (f1 < n && f1 - f0 < 65535) {                         // grid rows of the IDCT kernel
            const size_t c = jpeg_wave_bytes(fs[f1], up.u[f1]);
            if (f1 > f0 && need + c > budget) break;
            need += c;
            f1++;
        }
        int passes = 0;
        rc = jpeg_decode_wave(h, fs, data, up, f0, f1, sb + o_out, reinterpret_cast<const unsigned*>(sb + o_rst), pitch, &passes);
        if (rc) return rc;
        max_passes = std::max(max_passes, passes);
        f0 = f1;
    }
    h->jpeg_passes = max_passes;
    h->ingest_w = W; h->ingest_h = H; h->ingest_pitch = pitch; h->ingest_count = n;
    if (width) *width = W;
    if (height) *height = H;
    return FPM_OK;
}

// nothing may be thrown across the C ABI; an error leaves no frame and nothing in flight
static int ingest_jpeg_batch(fpm_handle* h, const uint8_t* data, const size_t* offsets, int n, int* width, int* height)
{
    h->ingest_count = 0;
    int rc;
    try {
        rc = ingest_jpeg_batch_impl(h, data, offsets, n, width, height);
    } catch (const std::bad_alloc&) {
        h->err = "out of host memory while decoding the JPEG";
        rc = FPM_ERR_LIMIT;
    }
    if (rc != FPM_OK) {
        cudaStreamSynchronize(h->stream);
        h->ingest_count = 0;
    }
    return rc;
}

// JPEG file image -> grayscale frame like cv::imread(path, IMREAD_GRAYSCALE): luma only, libjpeg's ISLOW IDCT.  A batch of one.
int fpm_ingest_jpeg(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height)
{
    if (!h) return FPM_ERR_INVALID;
    if (!file) { h->ingest_count = 0; h->err = "null JPEG buffer"; return FPM_ERR_INVALID; }
    const size_t offsets[2] = {0, nbytes};
    return ingest_jpeg_batch(h, file, offsets, 1, width, height);
}

int fpm_ingest_jpeg_batch(fpm_handle* h, const uint8_t* data, const size_t* offsets, int n, int* width, int* height)
{
    if (!h) return FPM_ERR_INVALID;
    return ingest_jpeg_batch(h, data, offsets, n, width, height);
}

// what cv::imread does first: pick the decoder by the file's signature (two of the reference's "*.jpg" Test Images are BMP data)
int fpm_ingest_image(fpm_handle* h, const uint8_t* file, size_t nbytes, int* width, int* height)
{
    if (!h) return FPM_ERR_INVALID;
    h->ingest_count = 0;
    if (!file || nbytes < 2) { h->err = "empty image file"; return FPM_ERR_INVALID; }
    if (file[0] == 'B' && file[1] == 'M') return fpm_ingest_bmp(h, file, nbytes, width, height);
    if (file[0] == 0xFF && file[1] == 0xD8) return fpm_ingest_jpeg(h, file, nbytes, width, height);
    h->err = "unsupported image file (not BMP or JPEG)";
    return FPM_ERR_INVALID;
}

// host half of the JPEG ingest alone (no device): quantised luma coefficients [bh*bw][64] + the luma quantisation table, for
// the CPU-side pin of the Huffman decoder against cv2 (tests/test_ingest.py).  coef may be NULL to query the sizes.
int fpm_dbg_jpeg_luma(const uint8_t* file, size_t nbytes, int* width, int* height, int* bw, int* bh, uint16_t* quant /* 64 */,
                      int16_t* coef, size_t coef_capacity, char* err, int err_capacity)
try {
    fpm_jpeg::Luma im;
    const std::string why = fpm_jpeg::decode_luma(file, nbytes, &im);
    if (!why.empty()) {
        if (err && err_capacity > 0) { strncpy(err, why.c_str(), err_capacity - 1); err[err_capacity - 1] = 0; }
        return FPM_ERR_INVALID;
    }
    if (width) *width = im.width;
    if (height) *height = im.height;
    if (bw) *bw = im.bw;
    if (bh) *bh = im.bh;
    if (quant) memcpy(quant, im.quant, sizeof(im.quant));
    if (coef) {
        if (coef_capacity < im.coef.size()) return FPM_ERR_LIMIT;
        memcpy(coef, im.coef.data(), im.coef.size() * sizeof(int16_t));
    }
    return FPM_OK;
} catch (const std::bad_alloc&) {
    return FPM_ERR_LIMIT;
}

// the PARALLEL decoder of a batch (unstuffing + passes + scans, fpm_jpeg_par.cuh) run CTA by CTA, thread by thread on the CPU,
// no device: file i's coefficients go to coef + coef_offsets[i] (n + 1 entries: file i owns [coef_offsets[i], coef_offsets[i+1])),
// passes[i] = the synchronisation passes file i took (the pass in which it last moved + 1)
int fpm_dbg_jpeg_luma_parallel_batch(const uint8_t* data, const size_t* offsets, int n, int16_t* coef, const size_t* coef_offsets,
                                     int* passes, char* err, int err_capacity)
try {
    auto fail = [&](const std::string& why, int rc = FPM_ERR_INVALID) {
        if (err && err_capacity > 0) { strncpy(err, why.c_str(), err_capacity - 1); err[err_capacity - 1] = 0; }
        return rc;
    };
    std::vector<JpegBatchFile> fs;
    std::string why;
    const int rc = jpeg_batch_parse(data, offsets, n, false, &fs, &why);
    if (rc) return fail(why, rc);
    if (!coef || !coef_offsets) return fail("null coefficient buffer");
    for (int i = 0; i < n; i++) {
        if (!jpeg_device_ok(fs[i].fr, fs[i].nbytes)) return fail(jpeg_file_prefix(i, n) + "scan not eligible for the parallel decoder");
        fs[i].device = true;
    }
    JpUnstuffPlan up;
    jpeg_unstuff_plan(fs, offsets[0], &up);
    std::vector<uint8_t> bits(up.out_bytes);
    std::vector<unsigned> rst(up.rst_entries);
    jpeg_unstuff_emulate(data + offsets[0], &up, bits.data(), rst.data());
    for (int i = 0; i < n; i++)
        if (fs[i].fr.restart_interval && up.u[i].nint != jpeg_expected_intervals(fs[i].fr))
            return fail(jpeg_file_prefix(i, n) + "restart markers do not match the frame header");
    JpWave w;
    jpeg_wave_plan(fs, up, 0, n, rst.data(), 0, &w);
    for (int i = 0; i < n; i++) {
        const JpScan& sc = w.files[i].sc;
        const size_t need = (size_t)sc.mcux * sc.mcuy * sc.luma_slots * 64;
        if (coef_offsets[i + 1] < coef_offsets[i] || coef_offsets[i + 1] - coef_offsets[i] < need) return FPM_ERR_LIMIT;
        memset(coef + coef_offsets[i], 0, need * sizeof(int16_t));
    }
    std::vector<JpState> st[2] = {std::vector<JpState>(w.nsub), std::vector<JpState>(w.nsub)}, used(w.nsub);
    const int nb = w.cta_first[n];
    auto each_thread = [&](auto fn) {                                 // blockIdx.x -> file by the same search as the kernels
        for (int b = 0; b < nb; b++) {
            const int fi = jp_file_of(w.cta_first.data(), n, b), cta = b - w.cta_first[fi];
            const JpFile& f = w.files[fi];
            for (int t = 0; t < JP_THREADS; t++) fn(fi, f, JpBytes{bits.data() + f.bits}, cta * JP_THREADS + t);
        }
    };
    each_thread([&](int, const JpFile& f, const JpBytes& src, int i) { jp_pass_cold(i, src, f.tabs, f.sc, st[0].data() + f.sub0, used.data() + f.sub0); });
    int cur = 0, np = 0;
    std::vector<int> last(n, 0), changed(n);
    for (;;) {
        if (++np > w.max_nsub + 1) return fail("JPEG scan did not synchronise");
        std::fill(changed.begin(), changed.end(), 0);
        each_thread([&](int fi, const JpFile& f, const JpBytes& src, int i) {
            jp_pass_sync(i, src, f.tabs, f.sc, st[cur].data() + f.sub0, st[cur ^ 1].data() + f.sub0, used.data() + f.sub0, &changed[fi]);
        });
        cur ^= 1;
        bool any = false;
        for (int i = 0; i < n; i++)
            if (changed[i]) { last[i] = np; any = true; }
        if (!any) break;
    }
    std::vector<unsigned> first(w.nsub);
    std::vector<int> dcval(w.nluma, 0);
    for (const JpFile& f : w.files) {
        unsigned run = 0;
        for (int i = 0; i < f.sc.nsub; i++) { first[f.sub0 + i] = run; run += st[cur][f.sub0 + i].nblk; }
    }
    each_thread([&](int fi, const JpFile& f, const JpBytes& src, int i) {
        jp_pass_write(i, src, f.tabs, f.sc, st[cur].data() + f.sub0, first.data() + f.sub0, nullptr, coef + coef_offsets[fi], dcval.data() + f.luma0);
    });
    for (int fi = 0; fi < n; fi++) {
        const JpScan& sc = w.files[fi].sc;
        int* dc = dcval.data() + w.files[fi].luma0;
        int16_t* c = coef + coef_offsets[fi];
        const size_t nluma = (size_t)sc.mcux * sc.mcuy * sc.luma_slots;
        const size_t seg = sc.restart_blocks ? (size_t)sc.restart_blocks / sc.nslots * sc.luma_slots : 0;
        int acc = 0;
        for (size_t L = 0; L < nluma; L++) {
            if (seg && L % seg == 0) acc = 0;                           // the DC prediction restarts with every interval
            acc += dc[L];
            dc[L] = acc;
        }
        const int bh = sc.mcuy * sc.luma_v;
        for (int r = 0; r < bh; r++)
            for (int col = 0; col < sc.bw; col++) c[((size_t)r * sc.bw + col) * 64] = (int16_t)dc[jp_luma_scan_index(sc, r, col)];
        if (passes) passes[fi] = last[fi] + 1;
    }
    return FPM_OK;
} catch (const std::bad_alloc&) {
    return FPM_ERR_LIMIT;
}

// the same for one file
int fpm_dbg_jpeg_luma_parallel(const uint8_t* file, size_t nbytes, int16_t* coef, size_t coef_capacity, int* passes, char* err, int err_capacity)
{
    const size_t offsets[2] = {0, nbytes}, coef_offsets[2] = {0, coef_capacity};
    return fpm_dbg_jpeg_luma_parallel_batch(file, offsets, 1, coef, coef_offsets, passes, err, err_capacity);
}

// unstuffing of one file without a device: emulated = 1 runs the phase functions of the unstuffing kernels, 0 the sequential
// jpeg_unstuff.  out: the unstuffed bytes + 16 zero bytes (out_cap >= file size - scan start + 20); rst: the first bit of every
// restart interval and rst[nint] = nbits (0, nbits without restart intervals), up to rst_cap entries
int fpm_dbg_jpeg_unstuff(const uint8_t* file, size_t nbytes, int emulated, uint8_t* out, size_t out_cap, unsigned* rst, int rst_cap,
                         unsigned* nbits, int* nint, int* tile)
try {
    if (tile) *tile = JP_UNSTUFF_TILE;
    if (!file || !out) return FPM_ERR_INVALID;
    fpm_jpeg::Frame fr;
    if (!fpm_jpeg::parse(file, nbytes, &fr).empty()) return FPM_ERR_INVALID;
    const size_t cap = align_up(nbytes - fr.scan_begin, 4) + 16;
    if (out_cap < cap) return FPM_ERR_LIMIT;
    std::vector<unsigned> rv;
    unsigned nb;
    int ni;
    if (!emulated) {
        std::vector<uint8_t> tmp(cap);
        const size_t o = jpeg_unstuff(file, nbytes, fr.scan_begin, tmp.data(), fr.restart_interval ? &rv : nullptr);
        memcpy(out, tmp.data(), o + 16);
        nb = (unsigned)(o * 8);
        ni = fr.restart_interval ? (int)rv.size() - 1 : 1;
    } else {
        std::vector<JpegBatchFile> fs(1);
        fs[0].fr = fr;
        fs[0].nbytes = nbytes;
        fs[0].device = true;
        JpUnstuffPlan up;
        jpeg_unstuff_plan(fs, 0, &up);
        if (fr.restart_interval) up.u[0].rst_cap = std::max(rst_cap, 0);
        std::vector<uint8_t> tmp(up.out_bytes);
        rv.assign(up.u[0].rst_cap, 0);
        jpeg_unstuff_emulate(file, &up, tmp.data(), rv.data());
        nb = up.u[0].nbits;
        ni = up.u[0].nint;
        memcpy(out, tmp.data(), nb / 8 + 16);
        if (fr.restart_interval) rv.resize(std::min<size_t>(rv.size(), (size_t)ni + 1));
    }
    if (!fr.restart_interval) rv = {0u, nb};
    for (int i = 0; i < rst_cap && i < (int)rv.size(); i++) rst[i] = rv[i];
    if (nbits) *nbits = nb;
    if (nint) *nint = ni;
    return FPM_OK;
} catch (const std::bad_alloc&) {
    return FPM_ERR_LIMIT;
}

int fpm_ingest_rgb32(fpm_handle* h, const uint32_t* pixels, int width, int height, int stride_bytes)
{
    if (!h) return FPM_ERR_INVALID;
    h->ingest_count = 0;
    if (!pixels || width <= 0 || height <= 0 || height > 65535 || width > (1 << 20) || stride_bytes < 4 * width || (stride_bytes & 3)) {
        h->err = "bad RGB32 frame";
        return FPM_ERR_INVALID;
    }
    CK(cudaSetDevice(h->device));
    const size_t nbytes = (size_t)stride_bytes * height;
    CK(h->d_ingest_raw.ensure(nbytes));
    const int pitch = (int)align_up(width, 128);
    CK(h->d_ingest.ensure((size_t)pitch * height));
    CK(cudaMemcpyAsync(h->d_ingest_raw.p, pixels, nbytes, cudaMemcpyHostToDevice, h->stream));
    dim3 grid((width + 255) / 256, height);
    fpm_ingest_rgb32_kernel<<<grid, 256, 0, h->stream>>>(h->d_ingest_raw.as<uint32_t>(), stride_bytes / 4, width, height,
                                                         h->d_ingest.as<uint8_t>(), pitch);
    CKL();
    CK(cudaStreamSynchronize(h->stream));
    h->ingest_w = width; h->ingest_h = height; h->ingest_pitch = pitch; h->ingest_count = 1;
    return FPM_OK;
}

namespace {
// the single-frame accessors: exactly one ingested frame (a batch goes through the _batch / _frame_ functions)
int ingest_single(fpm_handle* h)
{
    if (h->ingest_count == 1) return FPM_OK;
    h->err = h->ingest_count == 0 ? std::string("no ingested frame")
                                  : "the last ingest left " + std::to_string(h->ingest_count) +
                                        " frames: use fpm_ingested_frame_pixels / fpm_match_ingested_batch";
    return FPM_ERR_INVALID;
}
}  // namespace

int fpm_ingested_count(const fpm_handle* h) { return h ? h->ingest_count : 0; }

int fpm_ingested_frame_pixels(fpm_handle* h, int index, uint8_t* out)
{
    if (!h) return FPM_ERR_INVALID;
    if (!out) { h->err = "null output buffer"; return FPM_ERR_INVALID; }
    if (index < 0 || index >= h->ingest_count) {
        h->err = "ingested frame " + std::to_string(index) + " out of range (" + std::to_string(h->ingest_count) + " frames)";
        return FPM_ERR_INVALID;
    }
    CK(cudaSetDevice(h->device));
    const uint8_t* src = h->d_ingest.as<uint8_t>() + (size_t)index * h->ingest_pitch * h->ingest_h;
    CK(cudaMemcpy2D(out, (size_t)h->ingest_w, src, (size_t)h->ingest_pitch, (size_t)h->ingest_w, h->ingest_h, cudaMemcpyDeviceToHost));
    return FPM_OK;
}

int fpm_ingested_pixels(fpm_handle* h, uint8_t* out)
{
    if (!h || !out) return FPM_ERR_INVALID;
    if (int rc = ingest_single(h)) return rc;
    return fpm_ingested_frame_pixels(h, 0, out);
}

namespace {
// the calls that return scales: the scale of every record written during the call goes to scales; fn (the scaled set calls)
// lets a set of more than one template match at any range
struct ScalesOut {
    fpm_handle* h;
    ScalesOut(fpm_handle* hh, fpm_result* out, double* scales, const char* fn = nullptr) : h(hh)
    {
        h->scales_out = scales; h->scales_base = out; h->scaled_fn = fn;
    }
    ~ScalesOut()
    {
        h->scales_out = nullptr; h->scales_base = nullptr; h->scaled_fn = nullptr;
        if (h->twin) { h->twin->scales_out = nullptr; h->twin->scales_base = nullptr; h->twin->scaled_fn = nullptr; }
    }
};

// the frames of the last ingest x the set, through match_set
int match_ingested_set(fpm_handle* h, const char* fn, fpm_result* out, int cap, int* counts, const SetMerge* mg)
{
    if (h->ingest_count <= 0) { h->err = "no ingested frame"; return FPM_ERR_INVALID; }
    return match_set(h, fn, h->d_ingest.as<uint8_t>(), 1, h->ingest_count, h->ingest_w, h->ingest_h, h->ingest_pitch,
                     (size_t)h->ingest_pitch * h->ingest_h, out, cap, counts, mg);
}
}  // namespace

int fpm_match_scaled(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                     size_t frame_stride, fpm_result* out, double* scales, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_scaled")) return rc;
    ScalesOut so(h, out, scales);
    return src_on_device ? match_batch_device(h, src, batch, width, height, stride, frame_stride, out, cap, counts)
                         : match_batch_host(h, src, batch, width, height, stride, frame_stride, out, cap, counts);
}

int fpm_match_ingested_scaled(fpm_handle* h, fpm_result* out, double* scales, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_ingested_scaled")) return rc;
    ScalesOut so(h, out, scales);
    return fpm_match_ingested_set_batch(h, out, cap, counts);
}

int fpm_match_set_scaled(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                         size_t frame_stride, fpm_result* out, double* scales, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    const char* fn = "fpm_match_set_scaled";
    ScalesOut so(h, out, scales, fn);
    return match_set(h, fn, src, src_on_device, batch, width, height, stride, frame_stride, out, cap, counts, nullptr);
}

int fpm_match_ingested_set_scaled(fpm_handle* h, fpm_result* out, double* scales, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    const char* fn = "fpm_match_ingested_set_scaled";
    ScalesOut so(h, out, scales, fn);
    return match_ingested_set(h, fn, out, cap, counts, nullptr);
}

int fpm_match_set_scaled_merged(fpm_handle* h, const uint8_t* src, int src_on_device, int batch, int width, int height, int stride,
                                size_t frame_stride, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                int* counts, int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    const char* fn = "fpm_match_set_scaled_merged";
    const SetMerge mg{max_overlap, labels, set_counts};
    ScalesOut so(h, out, scales, fn);
    return match_set(h, fn, src, src_on_device, batch, width, height, stride, frame_stride, out, cap, counts, &mg);
}

int fpm_match_ingested_set_scaled_merged(fpm_handle* h, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                         int* counts, int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    const char* fn = "fpm_match_ingested_set_scaled_merged";
    const SetMerge mg{max_overlap, labels, set_counts};
    ScalesOut so(h, out, scales, fn);
    return match_ingested_set(h, fn, out, cap, counts, &mg);
}

int fpm_match_ingested(fpm_handle* h, fpm_result* out, int cap, int* n)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_ingested")) return rc;
    if (int rc = ingest_single(h)) return rc;
    return fpm_match_ingested_batch(h, out, cap, n);
}

int fpm_match_ingested_batch(fpm_handle* h, fpm_result* out, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_ingested_batch")) return rc;
    return fpm_match_ingested_set_batch(h, out, cap, counts);
}

int fpm_match_ingested_set_batch(fpm_handle* h, fpm_result* out, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    if (h->ingest_count <= 0) { h->err = "no ingested frame"; return FPM_ERR_INVALID; }
    return fpm_match_set_batch(h, h->d_ingest.as<uint8_t>(), 1, h->ingest_count, h->ingest_w, h->ingest_h, h->ingest_pitch,
                               (size_t)h->ingest_pitch * h->ingest_h, out, cap, counts);
}

int fpm_match_ingested_set_batch_merged(fpm_handle* h, double max_overlap, fpm_result* out, int* labels, int cap, int* counts,
                                        int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    if (h->ingest_count <= 0) { h->err = "no ingested frame"; return FPM_ERR_INVALID; }
    return fpm_match_set_batch_merged(h, h->d_ingest.as<uint8_t>(), 1, h->ingest_count, h->ingest_w, h->ingest_h, h->ingest_pitch,
                                      (size_t)h->ingest_pitch * h->ingest_h, max_overlap, out, labels, cap, counts, set_counts);
}

int fpm_learn_ingested(fpm_handle* h)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_learn_ingested")) return rc;
    if (int rc = ingest_single(h)) return rc;
    std::vector<uint8_t> px((size_t)h->ingest_w * h->ingest_h);
    int rc = fpm_ingested_pixels(h, px.data());
    if (rc) return rc;
    return fpm_learn(h, px.data(), h->ingest_w, h->ingest_h, h->ingest_w);
}

double fpm_last_time_ms(const fpm_handle* h) { return h ? h->last_ms : 0; }

void fpm_set_user_rect(fpm_handle* h, int x, int y, int w, int hgt)
{
    if (!h) return;
    h->ur[0] = x; h->ur[1] = y; h->ur[2] = w; h->ur[3] = hgt; h->has_ur = 1;
}

int fpm_get_user_rect(const fpm_handle* h, int* x, int* y, int* w, int* hgt)
{
    if (!h) return 0;
    if (x) *x = h->ur[0];
    if (y) *y = h->ur[1];
    if (w) *w = h->ur[2];
    if (hgt) *hgt = h->ur[3];
    return h->has_ur;
}

long long fpm_launch_count(const fpm_handle* h) { return h ? h->launches + (h->twin ? h->twin->launches : 0) : 0; }

int fpm_tpl_levels(const fpm_handle* h)
{
    if (h) if (int rc = refuse_set(h, "fpm_tpl_levels")) return rc;
    return (h && h->learned) ? (int)h->tpl.size() : 0;
}

int fpm_tpl_level_info(const fpm_handle* h, int level, int* w, int* hgt, double* mean, double* norm, double* inv_area,
                       int* result_equal1)
{
    if (h) if (int rc = refuse_set(h, "fpm_tpl_level_info")) return rc;
    if (!h || !h->learned || level < 0 || level >= (int)h->tpl.size()) return FPM_ERR_INVALID;
    const TplLevelHost& t = h->tpl[level];
    if (w) *w = t.w;
    if (hgt) *hgt = t.h;
    if (mean) *mean = t.mean;
    if (norm) *norm = t.norm;
    if (inv_area) *inv_area = t.inv_area;
    if (result_equal1) *result_equal1 = t.equal1;
    return FPM_OK;
}

int fpm_tpl_level_mask(const fpm_handle* h, int level, uint8_t* out)
{
    if (h) if (int rc = refuse_set(h, "fpm_tpl_level_mask")) return rc;
    if (!h || !h->learned || level < 0 || level >= (int)h->tpl.size()) return FPM_ERR_INVALID;
    const TplLevelHost& t = h->tpl[level];
    const size_t n = (size_t)t.w * t.h;
    if (out) {
        if (t.mask.empty()) memset(out, 1, n);
        else memcpy(out, t.mask.data(), n);
    }
    return t.mask.empty() ? (int)n : (int)t.n_kept;
}

int fpm_tpl_level_pixels(const fpm_handle* h, int level, uint8_t* out)
{
    if (h) if (int rc = refuse_set(h, "fpm_tpl_level_pixels")) return rc;
    if (!h || !h->learned || level < 0 || level >= (int)h->tpl.size() || !out) return FPM_ERR_INVALID;
    memcpy(out, h->tpl[level].pix.data(), h->tpl[level].pix.size());
    return FPM_OK;
}

int fpm_tpl_border_color(const fpm_handle* h)
{
    if (h) if (int rc = refuse_set(h, "fpm_tpl_border_color")) return rc;
    return h ? h->border : 0;
}

// ---- stage API (angle-sharded latency mode) -------------------------------------------
int fpm_stage_num_angles(fpm_handle* h, int width, int height)
{
    (void)width; (void)height;
    if (h) if (int rc = refuse_set(h, "fpm_stage_num_angles")) return rc;
    if (!h || !h->learned) return 0;
    if (ensure_learned_for_mra(h)) return 0;
    std::vector<double> a;
    angle_schedule(h, (int)h->tpl.size() - 1, a);
    return (int)a.size();
}

int fpm_stage_top(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device, int a0, int a1,
                  double* rows, int cap, int* n)
{
    if (!h || !n) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_stage_top")) return rc;
    if (int rc = refuse_scale(h, "fpm_stage_top", false)) return rc;
    *n = 0;
    if (!h->learned) return FPM_ERR_NOT_LEARNED;
    int rc = ensure_learned_for_mra(h);
    if (rc) return rc;
    if (!src || width <= 0 || height <= 0) return FPM_OK;
    CK(cudaSetDevice(h->device));
    h->levels.clear();
    if (match_guards(h, width, height, h->tpl0_w, h->tpl0_h)) return FPM_OK;
    const uint8_t* d_src = src;
    int pitch = stride;
    size_t img = (size_t)stride * height;
    if (!src_on_device) {
        pitch = (int)align_up(width, 128);
        img = align_up((size_t)pitch * height, 256);
        CK(h->d_src.ensure(img));
        CK(cudaMemcpy2DAsync(h->d_src.p, pitch, src, stride, width, height, cudaMemcpyHostToDevice, h->stream));
        d_src = h->d_src.as<uint8_t>();
    }
    const int top = (int)h->tpl.size() - 1;
    h->cur_batch = 1;
    CK(h->d_counters.ensure(CNT_N * sizeof(int)));
    CK(h->h_counts.ensure((CNT_N + 1) * sizeof(int)));
    if (h->bitwise_not) {
        const int ipitch = (int)align_up(width, 128);
        const size_t iimg = (size_t)ipitch * height;
        CK(h->d_inv.ensure(iimg));
        dim3 ig((width / 4 + 128) / 128, height, 1);
        fpm_invert_kernel<<<ig, 128, 0, h->stream>>>(d_src, width, height, pitch, img, h->d_inv.as<uint8_t>(), ipitch, iimg);
        CKL();
        d_src = h->d_inv.as<uint8_t>(); pitch = ipitch; img = iimg;
    }
    rc = build_pyramid(h, d_src, 1, width, height, pitch, img, top);
    if (rc) return rc;
    rc = make_top_plan(h, top, 1);
    if (rc) return rc;
    const TopPlan& p = h->plan;
    if (a1 < 0) a1 = p.n_ang;
    a0 = std::max(0, std::min(a0, p.n_ang));
    a1 = std::max(a0, std::min(a1, p.n_ang));
    const int n_loc = a1 - a0;
    if (n_loc == 0) return FPM_OK;
    const int max_picks = h->max_pos + FPM_MATCH_CANDIDATE_NUM;
    CK(h->d_picks.ensure((size_t)n_loc * max_picks * sizeof(FpmPick)));
    CK(h->d_pickcnt.ensure((size_t)n_loc * sizeof(int)));
    rc = run_top(h, top, a0, n_loc, h->d_picks.as<FpmPick>(), h->d_pickcnt.as<int>());
    if (rc) return rc;
    std::vector<FpmPick> picks((size_t)n_loc * max_picks);
    std::vector<int> cnt(n_loc);
    CK(cudaMemcpyAsync(picks.data(), h->d_picks.p, picks.size() * sizeof(FpmPick), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(cnt.data(), h->d_pickcnt.p, cnt.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int k = 0;
    for (int a = 0; a < n_loc; a++)
        for (int j = 0; j < cnt[a]; j++) {
            if (k < cap) {
                const FpmPick& pk = picks[(size_t)a * max_picks + j];
                double* r = rows + (size_t)k * 5;
                // translation removed here like :186 (float arithmetic)
                r[0] = a0 + a;
                r[1] = (double)((float)pk.x - p.ftx[a0 + a]);
                r[2] = (double)((float)pk.y - p.fty[a0 + a]);
                r[3] = pk.v;
                r[4] = p.angles[a0 + a];
            }
            k++;
        }
    *n = k;
    return FPM_OK;
}

// picks rows {angle_index, x, y, score, angle} in global (angle, pick) order -> candidate rows
// {id, ptLT.x, ptLT.y, score, angle}: stable sort by score descending (:214) and the un-rotation of
// :265-266.  Host side on purpose: it runs on the allgathered list, a few hundred rows.
int fpm_stage_sort_candidates(fpm_handle* h, const double* picks, int n, double* cands)
{
    if (!h || n < 0) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_stage_sort_candidates")) return rc;
    if (int rc = refuse_scale(h, "fpm_stage_sort_candidates", false)) return rc;
    if (h->levels.empty()) { h->err = "fpm_stage_top must run first"; return FPM_ERR_INVALID; }
    std::vector<int> idx(n);
    for (int i = 0; i < n; i++) idx[i] = i;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return (float)picks[a * 5 + 3] > (float)picks[b * 5 + 3]; });
    const FpmLevel& L = h->levels.back();
    float cx = (L.w - 1) / 2.0f, cy = (L.h - 1) / 2.0f;
    for (int i = 0; i < n; i++) {
        const double* p = picks + (size_t)idx[i] * 5;
        float rx, ry;
        fpm_pt_rotate((float)p[1], (float)p[2], cx, cy, -p[4] * FPM_D2R, &rx, &ry);
        double* c = cands + (size_t)i * 5;
        c[0] = i; c[1] = rx; c[2] = ry; c[3] = p[3]; c[4] = p[4];
    }
    return FPM_OK;
}

int fpm_stage_refine(fpm_handle* h, const double* cands, int n, double* rows, int cap, int* n_out)
{
    if (!h || !n_out) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_stage_refine")) return rc;
    if (int rc = refuse_scale(h, "fpm_stage_refine", false)) return rc;
    *n_out = 0;
    if (h->levels.empty()) { h->err = "fpm_stage_top must run first"; return FPM_ERR_INVALID; }
    CK(cudaSetDevice(h->device));
    const int top = (int)h->tpl.size() - 1;
    std::vector<FpmCand> cc(std::max(n, 1));
    for (int i = 0; i < n; i++) {
        const double* c = cands + (size_t)i * 5;
        cc[i].id = (int)c[0]; cc[i].ptx = (float)c[1]; cc[i].pty = (float)c[2]; cc[i].score = c[3]; cc[i].angle = c[4];
        cc[i].img = 0; cc[i].scale = 1.0;
    }
    CK(h->d_cand[0].ensure(cc.size() * sizeof(FpmCand)));
    CK(cudaMemcpyAsync(h->d_cand[0].p, cc.data(), cc.size() * sizeof(FpmCand), cudaMemcpyHostToDevice, h->stream));
    CK(h->d_counters.ensure(CNT_N * sizeof(int)));
    CK(h->h_counts.ensure((CNT_N + 1) * sizeof(int)));
    CK(cudaMemsetAsync(h->d_counters.p, 0, CNT_N * sizeof(int), h->stream));
    CK(cudaMemcpyAsync(h->d_counters.as<int>() + CNT_FLAT, &n, sizeof(int), cudaMemcpyHostToDevice, h->stream));   // live count of the first layer
    CK(cudaStreamSynchronize(h->stream));
    int n_ref = 0;
    h->ref_out = nullptr; h->ref_cnt = nullptr;
    h->cur_batch = 1;
    int rc = run_refine(h, top, n, &n_ref);
    if (rc) return rc;
    h->err_check_pending = false;
    CK(cudaMemcpyAsync(h->h_counts.p, h->d_counters.p, CNT_N * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_counts.as<int>()[CNT_ERR]) { h->err = "fpm_corr_warp_kernel: source box larger than its staging buffer"; return FPM_ERR_LIMIT; }
    n_ref = h->h_counts.as<int>()[CNT_REFINED];
    std::vector<FpmRefined> rr(std::max(n_ref, 1));
    if (n_ref) {
        CK(cudaMemcpyAsync(rr.data(), h->d_refined.p, (size_t)n_ref * sizeof(FpmRefined), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    std::sort(rr.begin(), rr.begin() + n_ref, [](const FpmRefined& a, const FpmRefined& b) { return a.id < b.id; });
    for (int i = 0; i < n_ref && i < cap; i++) {
        double* r = rows + (size_t)i * 5;
        r[0] = rr[i].id; r[1] = rr[i].ptx; r[2] = rr[i].pty; r[3] = rr[i].score; r[4] = rr[i].angle;
    }
    *n_out = n_ref;
    return FPM_OK;
}

int fpm_stage_final(fpm_handle* h, const double* refined, int n, fpm_result* out, int cap, int* n_out)
{
    if (!h || !n_out) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_stage_final")) return rc;
    if (int rc = refuse_scale(h, "fpm_stage_final", false)) return rc;
    *n_out = 0;
    if (!h->learned) return FPM_ERR_NOT_LEARNED;
    CK(cudaSetDevice(h->device));
    std::vector<FpmRefined> rr(std::max(n, 1));
    int max_id = 0;
    for (int i = 0; i < n; i++) {
        const double* r = refined + (size_t)i * 5;
        rr[i].id = (int)r[0]; rr[i].ptx = r[1]; rr[i].pty = r[2]; rr[i].score = r[3]; rr[i].angle = r[4]; rr[i].img = 0; rr[i].scale = 1.0;
        max_id = std::max(max_id, rr[i].id);
    }
    CK(h->d_counters.ensure(CNT_N * sizeof(int)));
    CK(h->d_refined.ensure(rr.size() * sizeof(FpmRefined)));
    CK(cudaMemcpyAsync(h->d_refined.p, rr.data(), rr.size() * sizeof(FpmRefined), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_counters.as<int>() + CNT_REFINED, &n, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    FpmRefinedView rv{h->d_refined.as<FpmRefined>(), h->d_counters.as<int>() + CNT_REFINED, 0, 1, 0};
    return run_final(h, 1, rv, std::max(max_id + 1, n), out, cap, n_out);
}

// ---- angle-sharded latency mode: communicator + whole-match entry points ---------------------------------
int fpm_comm_available(void) { return nccl_api().ok ? 1 : 0; }

int fpm_comm_get_unique_id(void* id)
{
    if (!id || !nccl_api().ok) return FPM_ERR_INVALID;
    NcclApi::UniqueId u;
    if (nccl_api().GetUniqueId(&u) != 0) return FPM_ERR_CUDA;
    memcpy(id, &u, sizeof(u));
    return FPM_OK;
}

void fpm_comm_destroy(fpm_handle* h)
{
    if (!h) return;
    if (h->nccl_comm && h->nccl_owned) {
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->stream);
        nccl_api().CommDestroy(h->nccl_comm);
    }
    h->nccl_comm = nullptr; h->nccl_owned = false; h->sh_nranks = 1; h->sh_rank = 0;
}

int fpm_comm_init(fpm_handle* h, int nranks, int rank, const void* id)
{
    if (!h) return FPM_ERR_INVALID;
    if (nranks < 1 || rank < 0 || rank >= nranks || !id) { h->err = "bad communicator arguments"; return FPM_ERR_INVALID; }
    const NcclApi& a = nccl_api();
    if (!a.ok) { h->err = "libnccl.so.2 could not be loaded"; return FPM_ERR_INVALID; }
    fpm_comm_destroy(h);
    CK(cudaSetDevice(h->device));
    NcclApi::UniqueId u;
    memcpy(&u, id, sizeof(u));
    void* comm = nullptr;
    const int r = a.CommInitRank(&comm, nranks, u, rank);
    if (r != 0) { h->err = std::string("ncclCommInitRank: ") + a.GetErrorString(r); return FPM_ERR_CUDA; }
    h->nccl_comm = comm; h->nccl_owned = true; h->sh_nranks = nranks; h->sh_rank = rank;
    return FPM_OK;
}

int fpm_comm_attach(fpm_handle* h, void* nccl_comm, int nranks, int rank)
{
    if (!h) return FPM_ERR_INVALID;
    if (nranks < 1 || rank < 0 || rank >= nranks || (nranks > 1 && !nccl_comm)) { h->err = "bad communicator arguments"; return FPM_ERR_INVALID; }
    if (nranks > 1 && !nccl_api().ok) { h->err = "libnccl.so.2 could not be loaded"; return FPM_ERR_INVALID; }
    fpm_comm_destroy(h);
    h->nccl_comm = nccl_comm; h->nccl_owned = false; h->sh_nranks = nranks; h->sh_rank = rank;
    return FPM_OK;
}

int fpm_shard_angle_range(int n_angles, int nranks, int rank, int* a0, int* a1)
{
    if (n_angles < 0 || nranks < 1 || rank < 0 || rank >= nranks || !a0 || !a1) return FPM_ERR_INVALID;
    const int chunk = shard_chunk(n_angles, nranks);
    *a0 = std::min(n_angles, rank * chunk);
    *a1 = std::min(n_angles, *a0 + chunk);
    return FPM_OK;
}

long long fpm_collective_count(const fpm_handle* h) { return h ? h->collectives : 0; }

namespace {
// refusals shared by the whole-set sharded calls (fpm_match_set_batch's, plus a missing communicator); scaled: the _scaled
// calls, which accept any scale range
int check_set_sharded(fpm_handle* h, const char* fn, int cap, const void* out, const int* n, bool scaled = false)
{
    if (int rc = refuse_scale(h, fn, scaled)) return rc;
    if (h->trace && fpm_set_size(h) > 1) {
        h->err = std::string(fn) + ": FPM_PARAM_TRACE is not supported for a set of more than one template";
        return FPM_ERR_INVALID;
    }
    if (!n || cap < 0 || (cap > 0 && !out)) { h->err = std::string(fn) + ": bad output arguments"; return FPM_ERR_INVALID; }
    if (h->sh_nranks > 1 && !h->nccl_comm) {
        h->err = std::string(fn) + ": " + std::to_string(h->sh_nranks) + " ranks without a communicator (fpm_comm_init / fpm_comm_attach)";
        return FPM_ERR_INVALID;
    }
    return FPM_OK;
}

// refusals of the virtual-rank drivers: every handle present, none with a communicator, one set size on all of them
int check_virtual(fpm_handle* const* hs, int nranks, const char* fn, bool whole_set, bool scaled = false)
{
    if (!hs || nranks < 1) return FPM_ERR_INVALID;
    for (int r = 0; r < nranks; r++)
        if (!hs[r]) return FPM_ERR_INVALID;
    auto refuse = [&](const std::string& msg) {
        for (int r = 0; r < nranks; r++) hs[r]->err = std::string(fn) + ": " + msg;
        return FPM_ERR_INVALID;
    };
    for (int r = 0; r < nranks; r++)
        if (int rc = refuse_scale(hs[r], fn, scaled)) return rc;
    for (int r = 0; r < nranks; r++) {
        if (hs[r]->nccl_comm) return whole_set ? refuse("the handle of rank " + std::to_string(r) + " has a communicator") : FPM_ERR_INVALID;
        if (!whole_set) {
            if (int rc = refuse_set(hs[r], fn)) return rc;
        } else if (fpm_set_size(hs[r]) != fpm_set_size(hs[0])) {
            return refuse("rank " + std::to_string(r) + " holds a set of " + std::to_string(fpm_set_size(hs[r])) + " templates, rank 0 one of " +
                          std::to_string(fpm_set_size(hs[0])));
        }
    }
    return FPM_OK;
}
}  // namespace

int fpm_match_sharded(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                      fpm_result* out, int cap, int* n)
{
    if (!h) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_match_sharded")) return rc;
    if (int rc = refuse_scale(h, "fpm_match_sharded", false)) return rc;
    if (!n || cap < 0 || (cap > 0 && !out)) { h->err = "bad output arguments"; return FPM_ERR_INVALID; }
    *n = 0;
    return match_set_sharded(h, src, width, height, stride, src_on_device, out, cap, n, nullptr);
}

// rank r's result list at out + r*cap, n[r]; the block copies are not counted as collectives
int fpm_match_sharded_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                              fpm_result* out, int cap, int* n)
{
    if (!n || cap < 0 || (cap > 0 && !out)) return FPM_ERR_INVALID;
    if (int rc = check_virtual(hs, nranks, "fpm_match_sharded_virtual", false)) return rc;
    for (int r = 0; r < nranks; r++) n[r] = 0;
    return match_set_sharded_virtual(hs, nranks, src, width, height, stride, out, cap, n, 1, nullptr, false);
}

namespace {
// fpm_match_set_sharded* (mg: merged; scaled: the _scaled calls, which accept any range and write each record's scale)
int set_sharded(fpm_handle* h, const char* fn, bool scaled, const uint8_t* src, int width, int height, int stride, int src_on_device,
                fpm_result* out, double* scales, int cap, int* counts, const SetMerge* mg)
{
    if (int rc = check_set_sharded(h, fn, cap, out, counts, scaled)) return rc;
    if (mg) if (int rc = check_merge_args(h, fn, mg->max_overlap, cap, mg->labels)) return rc;
    const int n_set = std::max(fpm_set_size(h), 1);
    std::fill(counts, counts + (mg ? 1 : n_set), 0);
    if (mg && mg->set_counts) std::fill(mg->set_counts, mg->set_counts + n_set, 0);
    ScalesOut so(h, out, scales, scaled ? fn : nullptr);
    return match_set_sharded(h, src, width, height, stride, src_on_device, out, cap, counts, mg);
}

// fpm_match_set_sharded*_virtual: mg holds the caller's whole labels / set_counts arrays, split here into the ranks' merges
int set_sharded_virtual(fpm_handle* const* hs, int nranks, const char* fn, bool scaled, const uint8_t* src, int width, int height,
                        int stride, fpm_result* out, double* scales, int cap, int* counts, const SetMerge* mg)
{
    if (int rc = check_virtual(hs, nranks, fn, true, scaled)) return rc;
    for (int r = 0; r < nranks; r++) {
        if (int rc = check_set_sharded(hs[r], fn, cap, out, counts, scaled)) return rc;
        if (mg) if (int rc = check_merge_args(hs[r], fn, mg->max_overlap, cap, mg->labels)) return rc;
    }
    const int n_set = std::max(fpm_set_size(hs[0]), 1), n_rows = mg ? 1 : n_set;
    std::fill(counts, counts + (size_t)nranks * n_rows, 0);
    if (mg && mg->set_counts) std::fill(mg->set_counts, mg->set_counts + (size_t)nranks * n_set, 0);
    std::vector<SetMerge> mgs;
    for (int r = 0; mg && r < nranks; r++)
        mgs.push_back(SetMerge{mg->max_overlap, mg->labels ? mg->labels + (size_t)r * cap : nullptr,
                               mg->set_counts ? mg->set_counts + (size_t)r * n_set : nullptr});
    std::vector<std::unique_ptr<ScalesOut>> so;            // every rank indexes the whole out / scales arrays
    for (int r = 0; r < nranks; r++) so.emplace_back(new ScalesOut(hs[r], out, scales, scaled ? fn : nullptr));
    return match_set_sharded_virtual(hs, nranks, src, width, height, stride, out, cap, counts, n_rows, mg ? mgs.data() : nullptr, true);
}
}  // namespace

int fpm_match_set_sharded(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                          fpm_result* out, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    return set_sharded(h, "fpm_match_set_sharded", false, src, width, height, stride, src_on_device, out, nullptr, cap, counts, nullptr);
}

int fpm_match_set_sharded_merged(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                 double max_overlap, fpm_result* out, int* labels, int cap, int* count, int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    const SetMerge mg{max_overlap, labels, set_counts};
    return set_sharded(h, "fpm_match_set_sharded_merged", false, src, width, height, stride, src_on_device, out, nullptr, cap, count, &mg);
}

int fpm_match_set_sharded_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                                  fpm_result* out, int cap, int* counts)
{
    return set_sharded_virtual(hs, nranks, "fpm_match_set_sharded_virtual", false, src, width, height, stride, out, nullptr, cap,
                               counts, nullptr);
}

int fpm_match_set_sharded_merged_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height,
                                         int stride, double max_overlap, fpm_result* out, int* labels, int cap, int* count,
                                         int* set_counts)
{
    const SetMerge mg{max_overlap, labels, set_counts};
    return set_sharded_virtual(hs, nranks, "fpm_match_set_sharded_merged_virtual", false, src, width, height, stride, out, nullptr,
                               cap, count, &mg);
}

int fpm_match_set_sharded_scaled(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                 fpm_result* out, double* scales, int cap, int* counts)
{
    if (!h) return FPM_ERR_INVALID;
    return set_sharded(h, "fpm_match_set_sharded_scaled", true, src, width, height, stride, src_on_device, out, scales, cap, counts,
                       nullptr);
}

int fpm_match_set_sharded_scaled_merged(fpm_handle* h, const uint8_t* src, int width, int height, int stride, int src_on_device,
                                        double max_overlap, fpm_result* out, double* scales, int* labels, int cap, int* count,
                                        int* set_counts)
{
    if (!h) return FPM_ERR_INVALID;
    const SetMerge mg{max_overlap, labels, set_counts};
    return set_sharded(h, "fpm_match_set_sharded_scaled_merged", true, src, width, height, stride, src_on_device, out, scales, cap,
                       count, &mg);
}

int fpm_match_set_sharded_scaled_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height, int stride,
                                         fpm_result* out, double* scales, int cap, int* counts)
{
    return set_sharded_virtual(hs, nranks, "fpm_match_set_sharded_scaled_virtual", true, src, width, height, stride, out, scales,
                               cap, counts, nullptr);
}

int fpm_match_set_sharded_scaled_merged_virtual(fpm_handle* const* hs, int nranks, const uint8_t* src, int width, int height,
                                                int stride, double max_overlap, fpm_result* out, double* scales, int* labels, int cap,
                                                int* count, int* set_counts)
{
    const SetMerge mg{max_overlap, labels, set_counts};
    return set_sharded_virtual(hs, nranks, "fpm_match_set_sharded_scaled_merged_virtual", true, src, width, height, stride, out,
                               scales, cap, count, &mg);
}

// ---- stage kernels for parity tests ----------------------------------------------------
int fpm_dbg_pyrdown(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, uint8_t* dst)
{
    return fpm_dbg_pyrdown2(h, src, w, hgt, stride, 0, dst, nullptr);
}

// one launch: dst1 = pyrDown(src) and (dst2 != NULL) dst2 = pyrDown(dst1).  The device copy of src starts `misalign` bytes
// past a 128-byte boundary and its pitch is a multiple of 128 plus `misalign`: 0 -> 16-byte cp.async, 8 -> 8-byte,
// 4 -> 4-byte, odd -> byte loads.
int fpm_dbg_pyrdown2(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, int misalign, uint8_t* dst1, uint8_t* dst2)
{
    if (!h || !src || !dst1 || w <= 0 || hgt <= 0 || misalign < 0 || misalign > 127) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int w1 = (w + 1) / 2, h1 = (hgt + 1) / 2, w2 = (w1 + 1) / 2, h2 = (h1 + 1) / 2;
    const int sp = (int)align_up(w, 128) + misalign, p1 = (int)align_up(w1, 128), p2 = (int)align_up(w2, 128);
    CK(h->d_dbg[0].ensure((size_t)sp * hgt + 128));
    CK(h->d_dbg[1].ensure((size_t)p1 * h1));
    CK(h->d_dbg[2].ensure((size_t)p2 * h2));
    uint8_t* ds = h->d_dbg[0].as<uint8_t>() + misalign;
    CK(cudaMemcpy2DAsync(ds, sp, src, stride, w, hgt, cudaMemcpyHostToDevice, h->stream));
    FpmLevel s{ds, w, hgt, sp, 0}, d1{h->d_dbg[1].as<uint8_t>(), w1, h1, p1, 0}, d2{h->d_dbg[2].as<uint8_t>(), w2, h2, p2, 0};
    int rc = launch_pyrdown(h, s, d1, dst2 ? &d2 : nullptr, 1);
    if (rc) return rc;
    CK(cudaMemcpy2DAsync(dst1, w1, d1.ptr, p1, w1, h1, cudaMemcpyDeviceToHost, h->stream));
    if (dst2) CK(cudaMemcpy2DAsync(dst2, w2, d2.ptr, p2, w2, h2, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FPM_OK;
}

int fpm_dbg_warp_affine(fpm_handle* h, const uint8_t* src, int w, int hgt, int stride, const double m[6], int dw, int dh,
                        int border, uint8_t* dst)
{
    if (!h || !src || !dst || w <= 0 || hgt <= 0 || dw <= 0 || dh <= 0) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    int sp = (int)align_up(w, 128), dp = (int)align_up(dw, 16);
    CK(h->d_dbg[0].ensure((size_t)sp * hgt));
    CK(h->d_dbg[1].ensure((size_t)dp * dh));
    CK(h->d_dbg[2].ensure(sizeof(FpmWarpJob)));
    FpmWarpJob jb;
    for (int i = 0; i < 6; i++) jb.m[i] = m[i];
    fpm_invert_affine(jb.m);
    jb.src_img = 0; jb.dw = dw; jb.dh = dh; jb.valid = 1;
    CK(cudaMemcpy2DAsync(h->d_dbg[0].p, sp, src, stride, w, hgt, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_dbg[2].p, &jb, sizeof(jb), cudaMemcpyHostToDevice, h->stream));
    FpmLevel s{h->d_dbg[0].as<uint8_t>(), w, hgt, sp, 0};
    const int tiles_x = (dp + WA_TW - 1) / WA_TW;
    dim3 grid(tiles_x * ((dh + WA_TH - 1) / WA_TH), 1);
    fpm_warp_kernel<<<grid, WA_THREADS, 0, h->stream>>>(h->d_dbg[2].as<FpmWarpJob>(), 1, s, h->d_dbg[1].as<uint8_t>(), dp, 0, border,
                                                        tiles_x, level_vec_ok(s), nullptr, FpmRefineGeom{});
    CKL();
    CK(cudaMemcpy2DAsync(dst, dw, h->d_dbg[1].p, dp, dw, dh, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FPM_OK;
}

int fpm_dbg_corr_rows(fpm_handle* h, const uint8_t* roi, const uint8_t* tpl, int tw, int th, int32_t* rowsum, int32_t* rowS,
                      int32_t* rowQ)
{
    if (!h || !roi || !tpl || tw <= 0 || th <= 0) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int rpitch = (int)align_up(tw + FPM_ROI_PAD, 16) + 16, tp = (int)align_up(tw, 16);
    const size_t roi_bytes = (size_t)rpitch * (th + FPM_ROI_PAD), t_bytes = (size_t)tp * th;
    CK(h->d_dbg[0].ensure(roi_bytes));
    CK(h->d_dbg[1].ensure(t_bytes));
    CK(h->d_dbg[2].ensure((size_t)th * FPM_NCELL * 4));
    CK(h->d_dbg[3].ensure(2 * (size_t)(th + FPM_ROI_PAD) * FPM_WSTRIDE * 4));
    CK(cudaMemsetAsync(h->d_dbg[0].p, 0, roi_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_dbg[1].p, 0, t_bytes, h->stream));
    CK(cudaMemcpy2DAsync(h->d_dbg[0].p, rpitch, roi, tw + FPM_ROI_PAD, tw + FPM_ROI_PAD, th + FPM_ROI_PAD, cudaMemcpyHostToDevice,
                         h->stream));
    CK(cudaMemcpy2DAsync(h->d_dbg[1].p, tp, tpl, tw, tw, th, cudaMemcpyHostToDevice, h->stream));
    FpmTplLevel td;
    td.ptr = h->d_dbg[1].as<uint8_t>(); td.w = tw; td.h = th; td.pitch = tp;
    td.mean = 0; td.norm = 1; td.inv_area = 1; td.result_equal1 = 0;
    td.n_tpl = 1; td.tpl_stride = 0; td.stats = nullptr; td.mrow = nullptr; td.mrun = nullptr;
    const CorrCfg cc = corr_config(th);
    if (cc.smem > 200 * 1024) { h->err = "correlation kernel shared memory limit"; return FPM_ERR_LIMIT; }
    if (cc.smem > 48 * 1024)
        CK(ensure_dyn_smem((const void*)fpm_corr_rows_kernel, h->device, cc.smem));
    int32_t* dS = h->d_dbg[3].as<int32_t>();
    int32_t* dQ = dS + (size_t)(th + FPM_ROI_PAD) * FPM_WSTRIDE;
    dim3 grid(cc.blocks_y_rows, 1);
    fpm_corr_rows_kernel<<<grid, cc.threads, cc.smem, h->stream>>>(h->d_dbg[0].as<uint8_t>(), rpitch, roi_bytes, td, 1, cc.rb,
                                                                    cc.evals_per_cta, h->d_dbg[2].as<int32_t>(), dS, dQ, nullptr, 1, nullptr);
    CKL();
    CK(cudaMemcpyAsync(rowsum, h->d_dbg[2].p, (size_t)th * FPM_NCELL * 4, cudaMemcpyDeviceToHost, h->stream));
    // the device records are 8 ints per (eval, row); the caller gets the 7 window sums of each
    CK(cudaMemcpy2DAsync(rowS, FPM_NSHIFT * 4, dS, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)(th + FPM_ROI_PAD), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(rowQ, FPM_NSHIFT * 4, dQ, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)(th + FPM_ROI_PAD), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FPM_OK;
}

// tensor-core path on `ne` ROI patches (each (th+6)x(tw+6), contiguous); results converted to the [e][tr][49] layout
int fpm_dbg_corr_rows_mma(fpm_handle* h, const uint8_t* rois, int ne, const uint8_t* tpl, int tw, int th, int32_t* rowsum,
                          int32_t* rowS, int32_t* rowQ)
{
    if (!h || !rois || !tpl || tw <= 0 || th <= 0 || ne <= 0) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (!get_encode_tiled()) { h->err = "cuTensorMapEncodeTiled not available"; return FPM_ERR_CUDA; }
    const int rh = th + FPM_ROI_PAD, rw = tw + FPM_ROI_PAD;
    const int rpitch = (int)align_up(rw, 16) + 16, tp = (int)align_up(tw, 16), bpitch = (int)align_up(tw + 8, 16);
    const size_t roi_stride = (size_t)rpitch * rh;
    CK(h->d_dbg[0].ensure(roi_stride * ne));
    CK(h->d_dbg[1].ensure((size_t)tp * th + (size_t)8 * th * bpitch + 256));
    CK(h->d_dbg[3].ensure(2 * (size_t)ne * rh * FPM_WSTRIDE * 4));
    CK(cudaMemsetAsync(h->d_dbg[0].p, 0, roi_stride * ne, h->stream));
    CK(cudaMemsetAsync(h->d_dbg[1].p, 0, (size_t)tp * th, h->stream));
    for (int e = 0; e < ne; e++)
        CK(cudaMemcpy2DAsync(h->d_dbg[0].as<uint8_t>() + e * roi_stride, rpitch, rois + (size_t)e * rh * rw, rw, rw, rh,
                             cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpy2DAsync(h->d_dbg[1].p, tp, tpl, tw, tw, th, cudaMemcpyHostToDevice, h->stream));
    uint8_t* tsh = h->d_dbg[1].as<uint8_t>() + align_up((size_t)tp * th, 256);
    dim3 g((bpitch + 127) / 128, th, 8);
    fpm_shift_template_kernel<<<g, 128, 0, h->stream>>>(h->d_dbg[1].as<uint8_t>(), tw, th, tp, tsh, bpitch);
    CKL();
    int32_t* dS = h->d_dbg[3].as<int32_t>();
    int32_t* dQ = dS + (size_t)ne * rh * FPM_WSTRIDE;
    int e_pad = 0;
    int rc = launch_corr_mma(h, h->d_dbg[0].as<uint8_t>(), rpitch, roi_stride, tsh, bpitch, tw, th, ne, &e_pad, dS, dQ);
    if (rc) return rc;
    std::vector<int32_t> raw((size_t)rh * e_pad * MM_N);
    CK(cudaMemcpyAsync(raw.data(), h->d_raw.p, raw.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(rowS, FPM_NSHIFT * 4, dS, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)ne * rh, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(rowQ, FPM_NSHIFT * 4, dQ, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)ne * rh, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int e = 0; e < ne; e++)
        for (int tr = 0; tr < th; tr++)
            for (int r = 0; r < FPM_NSHIFT; r++)
                for (int c = 0; c < FPM_NSHIFT; c++)
                    rowsum[((size_t)e * th + tr) * FPM_NCELL + r * FPM_NSHIFT + c] =
                        raw[((size_t)(tr + r) * e_pad + e) * MM_N + c * 8 + (7 - r)];
    return FPM_OK;
}

int fpm_dbg_corr_fused(fpm_handle* h, const uint8_t* rois, int ne, const uint8_t* tpl, int tw, int th, float* numer,
                       long long* winS, long long* winQ, int32_t* edge_rowS)
{
    if (!h || !rois || !tpl || !numer || !winS || !winQ || tw <= 0 || th <= 0 || ne <= 0) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (!get_encode_tiled()) { h->err = "cuTensorMapEncodeTiled not available"; return FPM_ERR_CUDA; }
    const int rh = th + FPM_ROI_PAD, rw = tw + FPM_ROI_PAD;
    const int rpitch = (int)align_up(rw, 16) + 16, tp = (int)align_up(tw, 16), bpitch = (int)align_up(tw + 8, 16);
    const size_t roi_stride = (size_t)rpitch * rh;
    CK(h->d_dbg[0].ensure(roi_stride * ne));
    CK(h->d_dbg[1].ensure((size_t)tp * th + (size_t)8 * th * bpitch + 256));
    CK(h->d_dbg[3].ensure(2 * (size_t)ne * rh * FPM_WSTRIDE * 4));
    CK(cudaMemsetAsync(h->d_dbg[0].p, 0, roi_stride * ne, h->stream));
    CK(cudaMemsetAsync(h->d_dbg[1].p, 0, (size_t)tp * th, h->stream));
    CK(cudaMemsetAsync(h->d_dbg[3].p, 0xff, 2 * (size_t)ne * rh * FPM_WSTRIDE * 4, h->stream));   // rows the kernel must not need stay poisoned
    for (int e = 0; e < ne; e++)
        CK(cudaMemcpy2DAsync(h->d_dbg[0].as<uint8_t>() + e * roi_stride, rpitch, rois + (size_t)e * rh * rw, rw, rw, rh,
                             cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpy2DAsync(h->d_dbg[1].p, tp, tpl, tw, tw, th, cudaMemcpyHostToDevice, h->stream));
    uint8_t* tsh = h->d_dbg[1].as<uint8_t>() + align_up((size_t)tp * th, 256);
    dim3 g((bpitch + 127) / 128, th, 8);
    fpm_shift_template_kernel<<<g, 128, 0, h->stream>>>(h->d_dbg[1].as<uint8_t>(), tw, th, tp, tsh, bpitch);
    CKL();
    int32_t* dS = h->d_dbg[3].as<int32_t>();
    int32_t* dQ = dS + (size_t)ne * rh * FPM_WSTRIDE;
    int rc = launch_corr_fused(h, h->d_dbg[0].as<uint8_t>(), rpitch, roi_stride, tsh, bpitch, tw, th, ne, dS, dQ);
    if (rc) return rc;
    std::vector<float> hn((size_t)ne * MM_N);
    std::vector<long long> tS((size_t)ne * FPM_NSHIFT), tQ((size_t)ne * FPM_NSHIFT);
    std::vector<int32_t> rS((size_t)ne * rh * FPM_NSHIFT), rQ((size_t)ne * rh * FPM_NSHIFT);
    CK(cudaMemcpyAsync(hn.data(), h->d_numer.p, hn.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(tS.data(), h->d_totS.p, tS.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(tQ.data(), h->d_totQ.p, tQ.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(rS.data(), FPM_NSHIFT * 4, dS, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)ne * rh, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(rQ.data(), FPM_NSHIFT * 4, dQ, FPM_WSTRIDE * 4, FPM_NSHIFT * 4, (size_t)ne * rh, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (edge_rowS) memcpy(edge_rowS, rS.data(), rS.size() * 4);
    // same window arithmetic as fpm_refine_finalize_kernel's fused branch
    for (int e = 0; e < ne; e++)
        for (int r = 0; r < FPM_NSHIFT; r++)
            for (int c = 0; c < FPM_NSHIFT; c++) {
                long long ws = tS[(size_t)e * FPM_NSHIFT + c], wq = tQ[(size_t)e * FPM_NSHIFT + c];
                for (int y = 0; y < rh; y++)
                    if (y < r || y >= r + th) {
                        ws -= rS[((size_t)e * rh + y) * FPM_NSHIFT + c];
                        wq -= rQ[((size_t)e * rh + y) * FPM_NSHIFT + c];
                    }
                const size_t o = (size_t)e * FPM_NCELL + r * FPM_NSHIFT + c;
                numer[o] = hn[(size_t)e * MM_N + c * 8 + (7 - r)];
                winS[o] = ws; winQ[o] = wq;
            }
    return FPM_OK;
}

// dense NCC map of `img` against the learned TOP-layer template
int fpm_dbg_top_score_production(fpm_handle* h, const uint8_t* img, int w, int hgt, float* score, float* reject_below);
int fpm_dbg_top_score(fpm_handle* h, const uint8_t* img, int w, int hgt, float* score)
{
    return fpm_dbg_top_score_production(h, img, w, hgt, score, nullptr);
}

// reject_below == null: the exact map everywhere.  Otherwise the kernel runs exactly as inside match() (scores certainly
// below Score*0.9^top - 0.01 may be float32 estimates) and the bound in use is returned.
int fpm_dbg_top_score_production(fpm_handle* h, const uint8_t* img, int w, int hgt, float* score, float* reject_below)
{
    if (!h || !img || !score) return FPM_ERR_INVALID;
    if (int rc = refuse_set(h, "fpm_dbg_top_score_production")) return rc;
    if (!h->learned) return FPM_ERR_NOT_LEARNED;
    CK(cudaSetDevice(h->device));
    const int top = (int)h->tpl.size() - 1;
    const TplLevelHost& t = h->tpl[top];
    const int RW = w - t.w + 1, RH = hgt - t.h + 1;
    if (RW <= 0 || RH <= 0) return FPM_ERR_INVALID;
    const int rp = (int)align_up(w, 16), sp = (int)align_up(RW, 4);
    CK(h->d_dbg[0].ensure((size_t)rp * hgt));
    CK(h->d_dbg[1].ensure((size_t)sp * RH * 4));
    CK(h->d_dbg[2].ensure(sizeof(FpmWarpJob)));
    FpmWarpJob jb;
    memset(&jb, 0, sizeof(jb));
    jb.dw = w; jb.dh = hgt; jb.valid = 1;
    CK(cudaMemcpy2DAsync(h->d_dbg[0].p, rp, img, w, w, hgt, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_dbg[2].p, &jb, sizeof(jb), cudaMemcpyHostToDevice, h->stream));
    const bool masked = !t.mask.empty();
    size_t smem = top_score_smem(t.w, t.h, masked);
    if (smem > 200 * 1024) { h->err = "top-layer template too large for the score kernel"; return FPM_ERR_LIMIT; }
    const auto kern = masked ? fpm_top_score_kernel<false, true> : fpm_top_score_kernel<false>;
    CK(ensure_dyn_smem((const void*)kern, h->device, smem));
    dim3 grid((RW + TS_TW - 1) / TS_TW, (RH + TS_TH - 1) / TS_TH, 1), block(TS_THREADS);
    kern<<<grid, block, smem, h->stream>>>(h->d_dbg[2].as<FpmWarpJob>(), h->d_dbg[0].as<uint8_t>(), rp, 0,
                                                           tpl_level_dev(h, top), h->d_dbg[1].as<float>(), sp, 0,
                                                           reject_below ? top_reject_below(h, top) : -INFINITY);
    CKL();
    if (reject_below) *reject_below = top_reject_below(h, top);
    CK(cudaMemcpy2DAsync(score, (size_t)RW * 4, h->d_dbg[1].p, (size_t)sp * 4, (size_t)RW * 4, RH, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FPM_OK;
}

int fpm_dbg_peaks(fpm_handle* h, const float* score, int cols, int rows, int tw, int th, int block_mode, double thresh,
                  double max_overlap, int max_picks, double* picks, int* n)
{
    if (!h || !score || !picks || !n || cols <= 0 || rows <= 0 || max_picks <= 0) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int sp = (int)align_up(cols, 4);
    CK(h->d_dbg[0].ensure((size_t)sp * rows * 4));
    CK(h->d_dbg[2].ensure(sizeof(FpmWarpJob)));
    FpmWarpJob jb;
    memset(&jb, 0, sizeof(jb));
    jb.dw = cols + tw - 1; jb.dh = rows + th - 1; jb.valid = 1;
    int tile = 8;
    while ((long long)((cols + tile - 1) / tile) * ((rows + tile - 1) / tile) > 1024 && tile < 256) tile *= 2;
    const int tiles0 = ((cols + tile - 1) / tile) * ((rows + tile - 1) / tile);
    int blk_stride = block_mode == 1 ? (cols / tw) * (rows / th) + 3 : (block_mode == 2 ? std::max((cols / (2 * tw)) * (rows / (2 * th)) + 2, tiles0) : tiles0);
    if (blk_stride > PK_SUP_MAX * 32) { h->err = "score map has too many blocks for the peak table"; return FPM_ERR_LIMIT; }
    CK(h->d_dbg[1].ensure((size_t)blk_stride * 8));
    CK(h->d_dbg[3].ensure((size_t)max_picks * sizeof(FpmPick) + 16));
    CK(cudaMemcpy2DAsync(h->d_dbg[0].p, (size_t)sp * 4, score, (size_t)cols * 4, (size_t)cols * 4, rows, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_dbg[2].p, &jb, sizeof(jb), cudaMemcpyHostToDevice, h->stream));
    float* bv = h->d_dbg[1].as<float>();
    int* bl = reinterpret_cast<int*>(bv + blk_stride);
    FpmPick* dp = h->d_dbg[3].as<FpmPick>();
    int* dn = reinterpret_cast<int*>(dp + max_picks);
    const int smem_blocks = peaks_smem_blocks(h, blk_stride);
    if (smem_blocks < 0) return FPM_ERR_CUDA;
    fpm_top_peaks_kernel<<<1, PK_THREADS, (size_t)smem_blocks * 8, h->stream>>>(h->d_dbg[2].as<FpmWarpJob>(), h->d_dbg[0].as<float>(), sp, 0, tw, th,
                                                                              block_mode, tile, bv, bl, blk_stride, thresh, max_overlap,
                                                                              max_picks, dp, dn, smem_blocks, 0, 1, 1);
    CKL();
    std::vector<FpmPick> hp(max_picks);
    int hn = 0;
    CK(cudaMemcpyAsync(hp.data(), dp, (size_t)max_picks * sizeof(FpmPick), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&hn, dn, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < hn; i++) { picks[i * 3] = hp[i].x; picks[i * 3 + 1] = hp[i].y; picks[i * 3 + 2] = hp[i].v; }
    *n = hn;
    return FPM_OK;
}

int fpm_dbg_rrect_overlap(const float r1[5], const float r2[5], double max_overlap, int* type, double* ratio)
{
    FpmRRect a{r1[0], r1[1], r1[2], r1[3], r1[4]}, b{r2[0], r2[1], r2[2], r2[3], r2[4]};
    return fpm_rrect_overlap_decision(a, b, max_overlap, type, ratio);
}

int fpm_dbg_rrect_from3(const float pts[6], float out[5])
{
    FpmRRect r = fpm_rrect_from3(pts[0], pts[1], pts[2], pts[3], pts[4], pts[5]);
    out[0] = r.cx; out[1] = r.cy; out[2] = r.w; out[3] = r.h; out[4] = r.angle;
    return 0;
}

// ---- timing / profiling -----------------------------------------------------------------
int fpm_timer_record(fpm_handle* h, int which)
{
    if (!h || which < 0 || which > 1) return FPM_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(which ? h->ev_t1 : h->ev_t0, h->stream));
    return FPM_OK;
}

double fpm_timer_elapsed_ms(fpm_handle* h)
{
    if (!h) return -1;
    float ms = -1;
    if (cudaEventSynchronize(h->ev_t1) != cudaSuccess) return -1;
    if (cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1) != cudaSuccess) return -1;
    return ms;
}

int fpm_profile_num_kernels(void) { return K_COUNT; }
const char* fpm_profile_name(int kid) { return (kid >= 0 && kid < K_COUNT) ? kKernelNames[kid] : ""; }

int fpm_profile_get(fpm_handle* h, int kid, double* ms, long long* launches, double* work)
{
    if (!h || kid < 0 || kid >= K_COUNT) return FPM_ERR_INVALID;
    prof_collect(h);
    if (ms) *ms = h->prof_ms[kid];
    if (launches) *launches = h->prof_launches[kid];
    if (work) *work = h->prof_work[kid];
    if (h->twin) {                                           // the half-batches of the twin handle count too
        prof_collect(h->twin);
        if (ms) *ms += h->twin->prof_ms[kid];
        if (launches) *launches += h->twin->prof_launches[kid];
        if (work) *work += h->twin->prof_work[kid];
    }
    return FPM_OK;
}

void fpm_profile_reset(fpm_handle* h)
{
    if (!h) return;
    prof_collect(h);
    for (int i = 0; i < 24; i++) { h->prof_ms[i] = 0; h->prof_work[i] = 0; h->prof_launches[i] = 0; }
    if (h->twin) fpm_profile_reset(h->twin);
}

// ---- trace access -----------------------------------------------------------------------
int fpm_trace_num_candidates(const fpm_handle* h) { return h ? (int)(h->tr_cands.size() / 4) : 0; }

int fpm_trace_candidates(const fpm_handle* h, double* rows)
{
    if (!h || !rows) return FPM_ERR_INVALID;
    for (size_t i = 0; i < h->tr_cands.size(); i++) rows[i] = h->tr_cands[i];
    return FPM_OK;
}

int fpm_trace_num_evals(const fpm_handle* h, int level)
{
    if (!h || level < 0 || level >= (int)h->tr_evals.size()) return 0;
    return (int)(h->tr_evals[level].size() / 5);
}

int fpm_trace_evals(const fpm_handle* h, int level, double* rows)
{
    if (!h || !rows || level < 0 || level >= (int)h->tr_evals.size()) return FPM_ERR_INVALID;
    for (size_t i = 0; i < h->tr_evals[level].size(); i++) rows[i] = h->tr_evals[level][i];
    return FPM_OK;
}

int fpm_trace_eval_scores(const fpm_handle* h, int level, float* out)
{
    if (!h || !out || level < 0 || level >= (int)h->tr_scores.size()) return FPM_ERR_INVALID;
    std::copy(h->tr_scores[level].begin(), h->tr_scores[level].end(), out);
    return FPM_OK;
}

int fpm_trace_eval_rois(const fpm_handle* h, int level, uint8_t* out, int* w, int* hgt, int* pitch)
{
    if (!h || level < 0 || level >= (int)h->tr_rois.size()) return FPM_ERR_INVALID;
    const fpm_handle::TraceRois& r = h->tr_rois[level];
    if (w) *w = r.w;
    if (hgt) *hgt = r.h;
    if (pitch) *pitch = r.pitch;
    if (out) std::copy(r.px.begin(), r.px.end(), out);
    const size_t per = (size_t)r.h * r.pitch;
    return per ? (int)(r.px.size() / per) : 0;
}

int fpm_trace_level(const fpm_handle* hc, int level, uint8_t* out, int* w, int* hgt)
{
    fpm_handle* h = const_cast<fpm_handle*>(hc);
    if (!h || level < 0 || level >= (int)h->levels.size()) return FPM_ERR_INVALID;
    const FpmLevel& L = h->levels[level];
    if (w) *w = L.w;
    if (hgt) *hgt = L.h;
    if (out) {
        CK(cudaMemcpy2D(out, L.w, L.ptr, L.pitch, L.w, L.h, cudaMemcpyDeviceToHost));
    }
    return FPM_OK;
}

}  // extern "C"
