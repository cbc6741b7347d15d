// fpm_template_matcher.hpp -- header-only C++ shim with the reference's `TemplateMatcher` surface
// (/root/reference/include/TemplateMatcher.h:9-52) on top of the C ABI in fpm_b200.h.
//
// With FPM_WITH_OPENCV defined (and OpenCV headers available, as in the Qt app) the cv::Mat overloads
// are compiled and `src/MatchToolDialog.cpp` builds against this class unchanged:
//     m_matcher.setMaxPositions(..); ... m_matcher.learnPattern(cv::Mat); m_matcher.match(cv::Mat)
// Without it the raw-pointer overloads are available (used by tests/test_cpp_shim.py).
#pragma once
#include "fpm_b200.h"

#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#ifdef FPM_WITH_OPENCV
#include <opencv2/core.hpp>
#endif

namespace fpm {

struct Point2d { double x, y; };

// s_SingleTargetMatch (/root/reference/include/DataStructures.h:97-115)
struct SingleTargetMatch {
#ifdef FPM_WITH_OPENCV
    cv::Point2d ptLT, ptRT, ptRB, ptLB, ptCenter;
#else
    Point2d ptLT, ptRT, ptRB, ptLB, ptCenter;
#endif
    double dMatchedAngle;
    double dMatchScore;
    double dScale = 1.0;     // match scale (setScaleRange): the instance is dScale times the template's size
};

class TemplateMatcher {
public:
    explicit TemplateMatcher(int device = 0, int resultCapacity = 4096) : cap_(resultCapacity)
    {
        h_ = fpm_create(device);
        if (!h_) throw std::runtime_error("fpm_create failed: no usable CUDA device (no CPU fallback)");
    }
    ~TemplateMatcher() { fpm_destroy(h_); }
    TemplateMatcher(const TemplateMatcher&) = delete;
    TemplateMatcher& operator=(const TemplateMatcher&) = delete;

    // include/TemplateMatcher.h:22-37
    void setMaxPositions(int v) { fpm_set_param(h_, FPM_PARAM_MAX_POSITIONS, v); }
    void setMaxOverlap(double v) { fpm_set_param(h_, FPM_PARAM_MAX_OVERLAP, v); }
    void setScore(double v) { fpm_set_param(h_, FPM_PARAM_SCORE, v); }
    void setToleranceAngle(double v) { fpm_set_param(h_, FPM_PARAM_TOLERANCE_ANGLE, v); }
    void setMinReduceArea(int v) { fpm_set_param(h_, FPM_PARAM_MIN_REDUCE_AREA, v); }
    void setUseSIMD(bool v) { fpm_set_param(h_, FPM_PARAM_USE_SIMD, v ? 1 : 0); }
    void setSubPixelEstimation(bool v) { fpm_set_param(h_, FPM_PARAM_SUBPIXEL, v ? 1 : 0); }
    // match instances lo..hi times the template's size (each in [0.5, 2]); false when refused, and then the range is unchanged
    bool setScaleRange(double lo, double hi)
    {
        const double old = fpm_get_param(h_, FPM_PARAM_SCALE_MIN);
        if (fpm_set_param(h_, FPM_PARAM_SCALE_MIN, lo) != 0) return false;
        if (fpm_set_param(h_, FPM_PARAM_SCALE_MAX, hi) != 0) { fpm_set_param(h_, FPM_PARAM_SCALE_MIN, old); return false; }
        return true;
    }
    std::pair<double, double> getScaleRange() const
    {
        return {fpm_get_param(h_, FPM_PARAM_SCALE_MIN), fpm_get_param(h_, FPM_PARAM_SCALE_MAX)};
    }
    int getMaxPositions() const { return (int)fpm_get_param(h_, FPM_PARAM_MAX_POSITIONS); }
    double getMaxOverlap() const { return fpm_get_param(h_, FPM_PARAM_MAX_OVERLAP); }
    double getScore() const { return fpm_get_param(h_, FPM_PARAM_SCORE); }
    double getToleranceAngle() const { return fpm_get_param(h_, FPM_PARAM_TOLERANCE_ANGLE); }
    int getMinReduceArea() const { return (int)fpm_get_param(h_, FPM_PARAM_MIN_REDUCE_AREA); }
    bool getUseSIMD() const { return fpm_get_param(h_, FPM_PARAM_USE_SIMD) != 0; }
    bool getSubPixelEstimation() const { return fpm_get_param(h_, FPM_PARAM_SUBPIXEL) != 0; }
    double getLastExecutionTime() const { return fpm_last_time_ms(h_) / 1000.0; }   // seconds (:40)
    bool isPatternLearned() const { return fpm_is_learned(h_) != 0; }
    void clearPattern() { fpm_clear(h_); }

    // raw-pointer surface (single-channel 8-bit, `stride` bytes per row)
    bool learnPattern(const unsigned char* tpl, int w, int h, int stride)
    {
        if (!tpl || w <= 0 || h <= 0) return false;                       // src/TemplateMatcher.cpp:47-49
        return fpm_learn(h_, tpl, w, h, stride) == FPM_OK;
    }
    // masked template: `mask` (same size, `mask_stride` bytes per row), nonzero = kept; false when fpm_learn_masked refuses it
    bool learnPattern(const unsigned char* tpl, int w, int h, int stride, const unsigned char* mask, int mask_stride)
    {
        if (!tpl || w <= 0 || h <= 0) return false;
        return fpm_learn_masked(h_, tpl, w, h, stride, mask, mask_stride) == FPM_OK;
    }
    std::vector<SingleTargetMatch> match(const unsigned char* src, int w, int h, int stride)
    {
        std::vector<SingleTargetMatch> out;
        if (!src || w <= 0 || h <= 0) return out;
        std::vector<fpm_result> r((size_t)cap_);
        std::vector<double> sc((size_t)cap_);
        int n = 0;
        if (fpm_match_scaled(h_, src, 0, 1, w, h, stride, (size_t)stride * h, r.data(), sc.data(), cap_, &n) != FPM_OK)
            throw std::runtime_error(fpm_last_error(h_));
        if (n > cap_) n = cap_;
        out.resize((size_t)n);
        for (int i = 0; i < n; i++) {
            out[i].ptLT = {r[i].ltx, r[i].lty}; out[i].ptRT = {r[i].rtx, r[i].rty};
            out[i].ptRB = {r[i].rbx, r[i].rby}; out[i].ptLB = {r[i].lbx, r[i].lby};
            out[i].ptCenter = {r[i].cx, r[i].cy};
            out[i].dMatchedAngle = r[i].angle; out[i].dMatchScore = r[i].score; out[i].dScale = sc[i];
        }
        return out;
    }

#ifdef FPM_WITH_OPENCV
    bool learnPattern(const cv::Mat& t)
    {
        if (t.empty() || t.type() != CV_8UC1) return false;
        return learnPattern(t.data, t.cols, t.rows, (int)t.step);
    }
    bool learnPattern(const cv::Mat& t, const cv::Mat& mask)
    {
        if (mask.empty()) return learnPattern(t);
        if (t.empty() || t.type() != CV_8UC1 || mask.type() != CV_8UC1 || mask.size() != t.size()) return false;
        return learnPattern(t.data, t.cols, t.rows, (int)t.step, mask.data, (int)mask.step);
    }
    std::vector<SingleTargetMatch> match(const cv::Mat& s)
    {
        if (s.empty() || s.type() != CV_8UC1) return {};
        return match(s.data, s.cols, s.rows, (int)s.step);
    }
    void setUserDefinedRect(const cv::Rect& r) { fpm_set_user_rect(h_, r.x, r.y, r.width, r.height); }
    cv::Rect getUserDefinedRect() const { int x, y, w, hh; fpm_get_user_rect(h_, &x, &y, &w, &hh); return cv::Rect(x, y, w, hh); }
#endif
    bool hasUserDefinedRect() const { return fpm_get_user_rect(h_, nullptr, nullptr, nullptr, nullptr) != 0; }

    fpm_handle* handle() { return h_; }

private:
    fpm_handle* h_;
    int cap_;
};

}  // namespace fpm
