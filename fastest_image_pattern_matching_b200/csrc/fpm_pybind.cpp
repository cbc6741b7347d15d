// fpm_pybind.cpp -- pybind11 module `fpm_b200_pybind`: the "C++ .so with Pybind11 for Python" the reference
// README advertises (README.md:11-13; its source is not in the reference repo).  Thin wrapper over the
// C++ shim (include/fpm_template_matcher.hpp), i.e. over the C ABI; numpy uint8 2-D arrays in, result objects out.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "../../include/fpm_template_matcher.hpp"

namespace py = pybind11;
using Img = py::array_t<unsigned char, py::array::c_style | py::array::forcecast>;

PYBIND11_MODULE(fpm_b200_pybind, m)
{
    m.doc() = "B200-native rotation-invariant NCC template matcher (TemplateMatcher surface of lrm2017/Fastest_Image_Pattern_Matching)";
    py::class_<fpm::SingleTargetMatch>(m, "SingleTargetMatch")
        .def_property_readonly("ptLT", [](const fpm::SingleTargetMatch& r) { return py::make_tuple(r.ptLT.x, r.ptLT.y); })
        .def_property_readonly("ptRT", [](const fpm::SingleTargetMatch& r) { return py::make_tuple(r.ptRT.x, r.ptRT.y); })
        .def_property_readonly("ptRB", [](const fpm::SingleTargetMatch& r) { return py::make_tuple(r.ptRB.x, r.ptRB.y); })
        .def_property_readonly("ptLB", [](const fpm::SingleTargetMatch& r) { return py::make_tuple(r.ptLB.x, r.ptLB.y); })
        .def_property_readonly("ptCenter", [](const fpm::SingleTargetMatch& r) { return py::make_tuple(r.ptCenter.x, r.ptCenter.y); })
        .def_readonly("dMatchedAngle", &fpm::SingleTargetMatch::dMatchedAngle)
        .def_readonly("dMatchScore", &fpm::SingleTargetMatch::dMatchScore)
        .def_readonly("dScale", &fpm::SingleTargetMatch::dScale);
    py::class_<fpm::TemplateMatcher>(m, "TemplateMatcher")
        .def(py::init<int, int>(), py::arg("device") = 0, py::arg("result_capacity") = 4096)
        .def("setMaxPositions", &fpm::TemplateMatcher::setMaxPositions)
        .def("setMaxOverlap", &fpm::TemplateMatcher::setMaxOverlap)
        .def("setScore", &fpm::TemplateMatcher::setScore)
        .def("setToleranceAngle", &fpm::TemplateMatcher::setToleranceAngle)
        .def("setMinReduceArea", &fpm::TemplateMatcher::setMinReduceArea)
        .def("setUseSIMD", &fpm::TemplateMatcher::setUseSIMD)
        .def("setSubPixelEstimation", &fpm::TemplateMatcher::setSubPixelEstimation)
        .def("setScaleRange", &fpm::TemplateMatcher::setScaleRange)
        .def("getScaleRange", &fpm::TemplateMatcher::getScaleRange)
        .def("getMaxPositions", &fpm::TemplateMatcher::getMaxPositions)
        .def("getMaxOverlap", &fpm::TemplateMatcher::getMaxOverlap)
        .def("getScore", &fpm::TemplateMatcher::getScore)
        .def("getToleranceAngle", &fpm::TemplateMatcher::getToleranceAngle)
        .def("getMinReduceArea", &fpm::TemplateMatcher::getMinReduceArea)
        .def("getUseSIMD", &fpm::TemplateMatcher::getUseSIMD)
        .def("getSubPixelEstimation", &fpm::TemplateMatcher::getSubPixelEstimation)
        .def("getLastExecutionTime", &fpm::TemplateMatcher::getLastExecutionTime)
        .def("isPatternLearned", &fpm::TemplateMatcher::isPatternLearned)
        .def("clearPattern", &fpm::TemplateMatcher::clearPattern)
        .def("hasUserDefinedRect", &fpm::TemplateMatcher::hasUserDefinedRect)
        .def("learnPattern",
             [](fpm::TemplateMatcher& self, Img t, py::object mask) {
                 if (t.ndim() != 2 || t.size() == 0) return false;
                 if (mask.is_none()) return self.learnPattern(t.data(), (int)t.shape(1), (int)t.shape(0), (int)t.strides(0));
                 Img m = mask.cast<Img>();
                 if (m.ndim() != 2 || m.shape(0) != t.shape(0) || m.shape(1) != t.shape(1))
                     throw std::invalid_argument("mask must be a 2-D array of the template's shape");
                 return self.learnPattern(t.data(), (int)t.shape(1), (int)t.shape(0), (int)t.strides(0), m.data(), (int)m.strides(0));
             },
             py::arg("tpl"), py::arg("mask") = py::none())
        .def("match", [](fpm::TemplateMatcher& self, Img s) {
            if (s.ndim() != 2 || s.size() == 0) return std::vector<fpm::SingleTargetMatch>();
            const unsigned char* p = s.data();
            int w = (int)s.shape(1), h = (int)s.shape(0), st = (int)s.strides(0);
            py::gil_scoped_release rel;
            return self.match(p, w, h, st);
        });
}
