// lib_python.cpp -- pybind11 module `lib_python`, the reference's drop-in boundary
// (reference lib/PythonBindings.cpp:170-555): same module, class, method and field names for
// everything pose_optimization.py / process.py / params.py / loaders/video_dataset.py touch, so
// those files run unchanged with `sys.path` pointing at this directory instead of lib/build.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "model.h"
#include <cstring>

namespace py = pybind11;
using namespace rcvdh;

static py::array_t<float> vec3ToNp(const Vec3f& v) { py::array_t<float> a(3); auto m = a.mutable_unchecked<1>(); m(0) = v.x; m(1) = v.y; m(2) = v.z; return a; }
static Vec3f npToVec3(const py::object& o) { auto a = py::cast<py::array_t<float, py::array::c_style | py::array::forcecast>>(o); if (a.size() != 3) throw std::runtime_error("Expected 3 values."); return {a.data()[0], a.data()[1], a.data()[2]}; }
static py::object imageToNp(const Image* img) {
  if (!img) return py::none();
  const int cn = cvChannels(img->type);
  std::vector<py::ssize_t> shape = {img->rows, img->cols}; if (cn > 1) shape.push_back(cn);
  py::array out;
  switch (cvDepth(img->type)) {
    case CV_8U: out = py::array_t<uint8_t>(shape); break;
    case CV_32S: out = py::array_t<int32_t>(shape); break;
    case CV_32F: out = py::array_t<float>(shape); break;
    case CV_64F: out = py::array_t<double>(shape); break;
    default: throw std::runtime_error("Can only convert byte, int, float, double images to numpy.ndarray.");
  }
  std::memcpy(out.mutable_data(), img->data.data(), img->data.size());   // owning copy, like the reference casters
  return std::move(out);
}

PYBIND11_MODULE(lib_python, m) {
  m.doc() = "B200-native drop-in for robust_cvd's lib_python (pose / depth-deformation optimizer on CUDA).";
  m.def("initLib", []() {});
  m.def("logToStdout", []() { setLogToStdout(true); });

  py::class_<Quatf>(m, "Quaternionf")
      .def("x", [](const Quatf& q) { return q.x; }).def("y", [](const Quatf& q) { return q.y; })
      .def("z", [](const Quatf& q) { return q.z; }).def("w", [](const Quatf& q) { return q.w; });
  py::class_<Extrinsics>(m, "Extrinsics")
      .def(py::init<>())
      .def_property("position", [](const Extrinsics& e) { return vec3ToNp(e.position); }, [](Extrinsics& e, const py::object& o) { e.position = npToVec3(o); })
      .def_readwrite("orientation", &Extrinsics::orientation)
      .def("left", [](const Extrinsics& e) { return vec3ToNp(e.left()); }).def("right", [](const Extrinsics& e) { return vec3ToNp(e.right()); })
      .def("down", [](const Extrinsics& e) { return vec3ToNp(e.down()); }).def("up", [](const Extrinsics& e) { return vec3ToNp(e.up()); })
      .def("forward", [](const Extrinsics& e) { return vec3ToNp(e.forward()); }).def("backward", [](const Extrinsics& e) { return vec3ToNp(e.backward()); });
  py::class_<Intrinsics>(m, "Intrinsics")
      .def(py::init<>())
      .def_readwrite("vFov", &Intrinsics::vFov).def_readwrite("hFov", &Intrinsics::hFov)
      .def_readwrite("centerLat", &Intrinsics::centerLat).def_readwrite("centerLon", &Intrinsics::centerLon);

  py::enum_<ValueXformType>(m, "ValueXformType").value("None", ValueXformType::None).value("Scale", ValueXformType::Scale).value("ScaleShift", ValueXformType::ScaleShift);
  py::enum_<XformType>(m, "XformType").value("Depth", XformType::Depth).value("Spatial", XformType::Spatial);
  py::enum_<DepthXformType>(m, "DepthXformType").value("None", DepthXformType::None).value("Identity", DepthXformType::Identity).value("Global", DepthXformType::Global).value("Grid", DepthXformType::Grid);
  py::enum_<SpatialXformType>(m, "SpatialXformType").value("None", SpatialXformType::None).value("Identity", SpatialXformType::Identity)
      .value("VerticalLinear", SpatialXformType::VerticalLinear).value("CornersBilinear", SpatialXformType::CornersBilinear)
      .value("BilinearGrid", SpatialXformType::BilinearGrid).value("BicubicGrid", SpatialXformType::BicubicGrid);

  py::class_<XformDescriptor>(m, "XformDescriptor")
      .def(py::init<>())
      .def_readwrite("type", &XformDescriptor::type).def_readwrite("depthType", &XformDescriptor::depthType)
      .def_readwrite("spatialType", &XformDescriptor::spatialType).def_readwrite("valueXform", &XformDescriptor::valueXform)
      .def_property("gridSize", [](const XformDescriptor& d) { py::array_t<int> a(3); for (int i = 0; i < 3; ++i) a.mutable_data()[i] = d.gridSize[i]; return a; },
                    [](XformDescriptor& d, const std::vector<int>& v) { if (v.size() != 3) throw std::runtime_error("gridSize needs 3 values."); for (int i = 0; i < 3; ++i) d.gridSize[i] = v[i]; })
      .def_property("depthMinMax", [](const XformDescriptor& d) { py::array_t<double> a(2); a.mutable_data()[0] = d.depthMinMax[0]; a.mutable_data()[1] = d.depthMinMax[1]; return a; },
                    [](XformDescriptor& d, const std::vector<double>& v) { if (v.size() != 2) throw std::runtime_error("depthMinMax needs 2 values."); d.depthMinMax = {{v[0], v[1]}}; })
      .def("reset", &XformDescriptor::reset, py::arg("type") = XformType::Depth)
      .def("str", &XformDescriptor::str).def("parse", &XformDescriptor::parse);

  py::class_<Xform>(m, "Xform")
      .def("clone", [](const Xform& x) { return x.clone(); }).def("copyFrom", &Xform::copyFrom)
      .def("desc", [](const Xform& x) { return x.desc(); }).def("str", &Xform::str)
      .def("params", [](const Xform& x) { return x.params(); }).def("numParams", &Xform::numParams)
      // DepthXform / SpatialXform methods (one native class serves both)
      .def("paramMap", [](const Xform& x, DepthFrame& df) { Image im = x.paramMap(df); return imageToNp(&im); })
      .def("warp", [](const Xform& x, int h, int w) { Image im = x.warp(h, w); return imageToNp(&im); });
  m.attr("DepthXform") = m.attr("Xform");
  m.attr("SpatialXform") = m.attr("Xform");

  py::class_<ColorFrame>(m, "ColorFrame").def("image", [](ColorFrame& f) { return imageToNp(f.image()); });
  py::class_<ColorStream>(m, "ColorStream")
      .def("frame", &ColorStream::frame, py::return_value_policy::reference)
      .def("name", &ColorStream::name).def("path", &ColorStream::path).def("extension", &ColorStream::extension)
      .def("width", &ColorStream::width).def("height", &ColorStream::height).def("setDir", &ColorStream::setDir);
  py::class_<DepthFrame>(m, "DepthFrame")
      .def("depth", [](DepthFrame& f) { return imageToNp(f.depth()); })
      .def("sourceDepth", [](DepthFrame& f) { return imageToNp(f.sourceDepth()); })
      .def("setDepth", [](DepthFrame& f, py::array_t<float, py::array::c_style | py::array::forcecast> a) {
        if (a.ndim() != 2) throw std::runtime_error("Depth image must be a 2-D float32 array.");
        Image img; img.create(int(a.shape(0)), int(a.shape(1)), cvMakeType(CV_32F, 1));
        std::memcpy(img.ptr<float>(), a.data(), size_t(a.shape(0)) * a.shape(1) * sizeof(float));
        f.setDepth(img);
      })
      .def("clear", &DepthFrame::clear)
      .def("clearCache", &DepthFrame::clearCache).def("clearXformedCache", &DepthFrame::clearXformedCache)
      .def("depthXform", [](DepthFrame& f) -> Xform& { return f.depthXform(); }, py::return_value_policy::reference)
      .def("resetDepthXform", &DepthFrame::resetDepthXform)
      .def("spatialXform", [](DepthFrame& f) -> Xform& { return f.spatialXform(); }, py::return_value_policy::reference)
      .def("resetSpatialXform", &DepthFrame::resetSpatialXform)
      .def_readwrite("intrinsics", &DepthFrame::intrinsics).def_readwrite("extrinsics", &DepthFrame::extrinsics);
  py::class_<DepthStream>(m, "DepthStream")
      .def("frame", &DepthStream::frame, py::return_value_policy::reference)
      .def("name", &DepthStream::name).def("path", &DepthStream::path)
      .def("depthXformDesc", [](const DepthStream& s) { return s.depthXformDesc(); }).def("spatialXformDesc", [](const DepthStream& s) { return s.spatialXformDesc(); })
      .def("width", &DepthStream::width).def("height", &DepthStream::height).def("setDir", &DepthStream::setDir)
      .def("resetDepthXforms", &DepthStream::resetDepthXforms).def("resetSpatialXforms", &DepthStream::resetSpatialXforms).def("clearCache", &DepthStream::clearCache);

  py::class_<DepthVideo>(m, "DepthVideo")
      .def(py::init<>())
      .def("printInfo", &DepthVideo::printInfo).def("save", &DepthVideo::save).def("load", &DepthVideo::load).def("saveDepth", &DepthVideo::saveDepth)
      .def("width", &DepthVideo::width).def("height", &DepthVideo::height).def("aspect", &DepthVideo::aspect).def("invAspect", &DepthVideo::invAspect)
      .def("path", &DepthVideo::path).def("numFrames", &DepthVideo::numFrames)
      .def("numColorStreams", &DepthVideo::numColorStreams).def("hasColorStream", &DepthVideo::hasColorStream).def("colorStreamIndex", &DepthVideo::colorStreamIndex)
      .def("colorStream", [](DepthVideo& v, int i) -> ColorStream& { return v.colorStream(i); }, py::return_value_policy::reference)
      .def("colorStream", [](DepthVideo& v, const std::string& n) -> ColorStream& { return v.colorStream(n); }, py::return_value_policy::reference)
      .def("createColorStream", &DepthVideo::createColorStream, py::arg("name"), py::arg("dir"), py::arg("extension"), py::arg("type"), py::arg("size") = std::pair<int, int>{-1, -1})
      .def("numDepthStreams", &DepthVideo::numDepthStreams).def("hasDepthStream", &DepthVideo::hasDepthStream).def("depthStreamIndex", &DepthVideo::depthStreamIndex)
      .def("depthStream", [](DepthVideo& v, int i) -> DepthStream& { return v.depthStream(i); }, py::return_value_policy::reference)
      .def("depthStream", [](DepthVideo& v, const std::string& n) -> DepthStream& { return v.depthStream(n); }, py::return_value_policy::reference)
      .def("createDepthStream", &DepthVideo::createDepthStream, py::arg("name"), py::arg("dir"), py::arg("size") = std::pair<int, int>{-1, -1})
      .def("depthFrame", &DepthVideo::depthFrame, py::return_value_policy::reference)
      .def("clearDepthCaches", &DepthVideo::clearDepthCaches);

  py::class_<FrameRange>(m, "FrameRange")
      .def(py::init<>())
      .def("fromString", &FrameRange::fromString).def("toString", &FrameRange::toString)
      .def("resolve", &FrameRange::resolve, py::arg("numFrames"), py::arg("clip") = false)
      .def("isEmpty", &FrameRange::isEmpty).def("firstFrame", &FrameRange::firstFrame).def("lastFrame", &FrameRange::lastFrame)
      .def("count", &FrameRange::count).def("isConsecutive", &FrameRange::isConsecutive).def("inRange", &FrameRange::inRange).def("checkEmpty", &FrameRange::checkEmpty);

  py::class_<FlowConstraintsParams>(m, "FlowConstraintsParams")
      .def(py::init<>())
      .def_readwrite("matchSeparation", &FlowConstraintsParams::matchSeparation).def_readwrite("minDynamicDistance", &FlowConstraintsParams::minDynamicDistance)
      .def_readwrite("frameRange", &FlowConstraintsParams::frameRange).def_readwrite("doNotUseCache", &FlowConstraintsParams::doNotUseCache);
  py::class_<FlowConstraintsCollection>(m, "FlowConstraintsCollection")
      .def(py::init<DepthVideo&, const FlowConstraintsParams&>(), py::keep_alive<1, 2>())
      .def("load", &FlowConstraintsCollection::load).def("save", &FlowConstraintsCollection::save)
      .def("resetStaticFlag", &FlowConstraintsCollection::resetStaticFlag)
      .def("setStaticFlagFromDynamicMask", &FlowConstraintsCollection::setStaticFlagFromDynamicMask)
      .def("pruneStaticFlag", &FlowConstraintsCollection::pruneStaticFlag)
      // test/debug accessor (not in the reference): (pair keys, per-pair arrays [n,4] float32 + static flags)
      .def("_pairs", [](const FlowConstraintsCollection& c) {
        py::dict d;
        for (const auto& kv : c.pairs()) {
          py::array_t<float> a({(py::ssize_t)kv.second.size(), (py::ssize_t)4}); py::array_t<bool> s((py::ssize_t)kv.second.size());
          for (size_t i = 0; i < kv.second.size(); ++i) { std::memcpy(a.mutable_data() + 4 * i, kv.second[i].loc, 16); s.mutable_data()[i] = kv.second[i].isStatic; }
          d[py::make_tuple(kv.first.first, kv.first.second)] = py::make_tuple(a, s);
        }
        return d; })
      .def("_triplets", [](const FlowConstraintsCollection& c) {
        py::dict d;
        for (const auto& kv : c.triplets()) {
          py::array_t<float> a({(py::ssize_t)kv.second.size(), (py::ssize_t)6}); py::array_t<bool> s((py::ssize_t)kv.second.size());
          for (size_t i = 0; i < kv.second.size(); ++i) { std::memcpy(a.mutable_data() + 6 * i, kv.second[i].loc, 24); s.mutable_data()[i] = kv.second[i].isStatic; }
          d[py::int_(kv.first)] = py::make_tuple(a, s);
        }
        return d; });

  struct DepthVideoImporter {};
  py::class_<DepthVideoImporter>(m, "DepthVideoImporter")
      .def_static("importVideo", [](DepthVideo& v, const std::string& path, bool discover) { importVideo(v, path, discover); })
      .def_static("importPoses", [](DepthVideo&, const std::string&, int) { throw std::runtime_error("importPoses (ground-truth pose import) is outside the pose-optimization path and not implemented in this build."); })
      .def_static("importColmapDepth", [](DepthVideo&) { throw std::runtime_error("COLMAP import is not implemented in this build."); })
      .def_static("importColmapRecon", [](DepthVideo&, const std::string&, int, bool) { throw std::runtime_error("COLMAP import is not implemented in this build."); });

  py::enum_<StaticLossType>(m, "StaticLossType").value("Euclidean", StaticLossType::Euclidean).value("ReproDisparity", StaticLossType::ReproDisparity)
      .value("ReproDepthRatio", StaticLossType::ReproDepthRatio).value("ReproLogDepth", StaticLossType::ReproLogDepth);
  py::enum_<SmoothLossType>(m, "SmoothLossType").value("EuclideanLaplacian", SmoothLossType::EuclideanLaplacian).value("ReproDisparityLaplacian", SmoothLossType::ReproDisparityLaplacian)
      .value("ReproDepthRatioConsistency", SmoothLossType::ReproDepthRatioConsistency).value("ReproLogDepthConsistency", SmoothLossType::ReproLogDepthConsistency);
  py::enum_<IntrinsicsOptimization>(m, "IntrinsicsOptimization").value("Fixed", IntrinsicsOptimization::Fixed).value("Shared", IntrinsicsOptimization::Shared).value("PerFrame", IntrinsicsOptimization::PerFrame);

  py::class_<DepthVideoPoseOptimizer> dvpo(m, "DepthVideoPoseOptimizer");
  using P = DepthVideoPoseOptimizer::Params;
  py::class_<P>(dvpo, "Params")
      .def(py::init<>())
      .def_readwrite("frameRange", &P::frameRange).def_readwrite("maxIterations", &P::maxIterations).def_readwrite("numThreads", &P::numThreads)
      .def_readwrite("numSteps", &P::numSteps).def_readwrite("robustness", &P::robustness).def_readwrite("staticLossType", &P::staticLossType)
      .def_readwrite("staticSpatialWeight", &P::staticSpatialWeight).def_readwrite("staticDepthWeight", &P::staticDepthWeight)
      .def_readwrite("smoothLossType", &P::smoothLossType).def_readwrite("smoothStaticWeight", &P::smoothStaticWeight).def_readwrite("smoothDynamicWeight", &P::smoothDynamicWeight)
      .def_readwrite("positionReg", &P::positionReg).def_readwrite("scaleReg", &P::scaleReg).def_readwrite("scaleRegGridSize", &P::scaleRegGridSize)
      .def_readwrite("depthDeformRegInitial", &P::depthDeformRegInitial).def_readwrite("depthDeformRegFinal", &P::depthDeformRegFinal)
      .def_readwrite("adaptiveDeformationCost", &P::adaptiveDeformationCost).def_readwrite("spatialDeformReg", &P::spatialDeformReg)
      .def_readwrite("graduateDepthDeformReg", &P::graduateDepthDeformReg).def_readwrite("focalReg", &P::focalReg)
      .def_readwrite("coarseToFine", &P::coarseToFine).def_readwrite("ctfLong", &P::ctfLong).def_readwrite("ctfShort", &P::ctfShort)
      .def_readwrite("deferredSpatialOpt", &P::deferredSpatialOpt).def_readwrite("dsoLong", &P::dsoLong).def_readwrite("dsoShort", &P::dsoShort)
      .def_readwrite("focalLong", &P::focalLong).def_readwrite("intrOpt", &P::intrOpt)
      .def_readwrite("fixPoses", &P::fixPoses).def_readwrite("fixDepthXforms", &P::fixDepthXforms).def_readwrite("fixSpatialXforms", &P::fixSpatialXforms);
  dvpo.def(py::init<DepthVideo*, int>(), py::keep_alive<1, 2>())
      .def("poseOptimization", &DepthVideoPoseOptimizer::poseOptimization)
      .def("normalizeDepth", &DepthVideoPoseOptimizer::normalizeDepth)
      // test/debug accessor (not in the reference): the arrays one optimisation step hands to the C ABI
      .def("_buildProblem", [](DepthVideoPoseOptimizer& o, const P& params, const FlowConstraintsCollection* c, double deformReg, bool normalize) {
        auto pa = o.buildProblem(params, c, deformReg, normalize);
        py::dict d;
        d["config"] = py::bytes(reinterpret_cast<const char*>(&pa.cfg), sizeof(pa.cfg));
        d["in_range"] = py::array_t<uint8_t>(pa.inRange.size(), pa.inRange.data());
        d["median"] = py::array_t<double>(pa.median.size(), pa.median.data());
        d["adaptive"] = py::array_t<double>(pa.adaptive.size(), pa.adaptive.data());
        d["state"] = py::array_t<double>(pa.state.size(), pa.state.data());
        d["pair_frames"] = py::array_t<int32_t>(pa.pairFrames.size(), pa.pairFrames.data());
        d["offsets"] = py::array_t<int64_t>(pa.offsets.size(), pa.offsets.data());
        d["records"] = py::array_t<float>(pa.records.size(), pa.records.data());
        d["trip_centers"] = py::array_t<int32_t>(pa.tripCenters.size(), pa.tripCenters.data());
        d["trip_offsets"] = py::array_t<int64_t>(pa.tripOffsets.size(), pa.tripOffsets.data());
        d["trip_records"] = py::array_t<float>(pa.tripRecords.size(), pa.tripRecords.data());
        return d; }, py::arg("params"), py::arg("constraints"), py::arg("depthDeformReg") = 0.1, py::arg("normalize") = false);

  py::class_<DepthVideoProcessor> dvp(m, "DepthVideoProcessor");
  using Q = DepthVideoProcessor::Params;
  py::class_<Q>(dvp, "Params")
      .def(py::init<>())
      .def_readwrite("op", &Q::op).def_readwrite("frameRange", &Q::frameRange).def_readwrite("colorStream", &Q::colorStream)
      .def_readwrite("depthStream", &Q::depthStream).def_readwrite("sourceDepthStream", &Q::sourceDepthStream)
      .def_readwrite("spatialRadius", &Q::spatialRadius).def_readwrite("frameRadius", &Q::frameRadius).def_readwrite("depthSigma", &Q::depthSigma)
      .def_readwrite("colorSigma", &Q::colorSigma).def_readwrite("median", &Q::median).def_readwrite("farConnections", &Q::farConnections)
      .def_readwrite("matchSeparation", &Q::matchSeparation).def_readwrite("flowConsistancyThresh", &Q::flowConsistancyThresh)
      .def_readwrite("trackSpawnDistance", &Q::trackSpawnDistance).def_readwrite("trackPruneDistance", &Q::trackPruneDistance)
      .def_readwrite("minDynamicDistance", &Q::minDynamicDistance).def_readwrite("minTrackLength", &Q::minTrackLength)
      .def_readwrite("depthXformDesc", &Q::depthXformDesc).def_readwrite("spatialXformDesc", &Q::spatialXformDesc).def_readwrite("poseOptimizer", &Q::poseOptimizer);
  using Op = DepthVideoProcessor::Op;
  py::enum_<Op>(dvp, "Op")
      .value("None", Op::None).value("Reset", Op::Reset).value("Copy", Op::Copy).value("BilateralFilter", Op::BilateralFilter).value("FlowGuidedFilter", Op::FlowGuidedFilter)
      .value("ComputeConstraints", Op::ComputeConstraints).value("ResetConstraintStaticFlag", Op::ResetConstraintStaticFlag)
      .value("SetConstraintStaticFlagFromDynamicMask", Op::SetConstraintStaticFlagFromDynamicMask).value("ComputeTracks", Op::ComputeTracks)
      .value("GridXformSplit", Op::GridXformSplit).value("ResetPoses", Op::ResetPoses).value("ResetDepthXforms", Op::ResetDepthXforms)
      .value("ResetSpatialXforms", Op::ResetSpatialXforms).value("NormalizeDepth", Op::NormalizeDepth).value("OptimizePoses", Op::OptimizePoses)
      .value("ResetNormalizeOptimize", Op::ResetNormalizeOptimize);
  dvp.def(py::init<DepthVideo*>(), py::keep_alive<1, 2>())
      .def("process", &DepthVideoProcessor::process).def("gridXformSplit", &DepthVideoProcessor::gridXformSplit)
      .def("reset", &DepthVideoProcessor::reset).def("copy", &DepthVideoProcessor::copy).def("flowGuidedFilter", &DepthVideoProcessor::flowGuidedFilter)
      .def("bilateralFilter", &DepthVideoProcessor::bilateralFilter)
      .def("resetPoses", &DepthVideoProcessor::resetPoses).def("resetDepthXforms", &DepthVideoProcessor::resetDepthXforms)
      .def("resetSpatialXforms", &DepthVideoProcessor::resetSpatialXforms)
      .def("normalizeDepth", &DepthVideoProcessor::normalizeDepth).def("optimizePoses", &DepthVideoProcessor::optimizePoses);

  // image-operator restatements, exposed for the CPU parity tests against cv2
  m.def("_cornerMinEigenVal3", [](py::array_t<float, py::array::c_style | py::array::forcecast> bgr) {
    Image im; im.create((int)bgr.shape(0), (int)bgr.shape(1), cvMakeType(CV_32F, 3)); std::memcpy(im.data.data(), bgr.data(), im.data.size());
    Image r = cornerMinEigenVal3(bgr2gray32f(im)); return imageToNp(&r); });
  m.def("_distanceTransformL2_5", [](py::array_t<uint8_t, py::array::c_style | py::array::forcecast> b) {
    Image im; im.create((int)b.shape(0), (int)b.shape(1), cvMakeType(CV_8U, 1)); std::memcpy(im.data.data(), b.data(), im.data.size());
    Image r = distanceTransformL2_5(im); return imageToNp(&r); });
  m.def("_imreadPng", [](const std::string& f, bool gray) { Image im = imreadPng(f, gray); return imageToNp(im.empty() ? nullptr : &im); });
  m.def("_makeQuat", [](float x, float y, float z, float w) { Quatf q; q.x = x; q.y = y; q.z = z; q.w = w; return q; });   // tests: the reference binds no quaternion constructor
  m.def("_quatToAngleAxis", [](float x, float y, float z, float w) { Quatf q; q.x = x; q.y = y; q.z = z; q.w = w; double aa[3]; quatToAngleAxis(q, aa); return py::make_tuple(aa[0], aa[1], aa[2]); });
  m.def("_angleAxisToQuat", [](double a, double b, double c) { const double aa[3] = {a, b, c}; Quatf q = angleAxisToQuat(aa); return py::make_tuple(q.x, q.y, q.z, q.w); });
}
