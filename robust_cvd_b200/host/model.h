// model.h -- minimal native data model behind the `lib_python` module.
//
// Mirrors the subset of the reference's C++ API that pose_optimization.py, process.py,
// params.py and loaders/video_dataset.py use (reference lib/PythonBindings.cpp:170-555;
// SURVEY.md section 8b).  Same class / method / field names and error behaviour
// (std::runtime_error -> Python RuntimeError); the Ceres solve is replaced by the CUDA
// library behind include/rcvd.h.  Eigen / OpenCV / Boost are not available in this image,
// so small value types and image containers are defined here.
#pragma once
#include <array>
#include <atomic>
#include <cstdlib>
#include <exception>
#include <functional>
#include <thread>
#include <cstdint>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <system_error>
#include <utility>
#include <vector>

#include "../../include/rcvd.h"

namespace rcvdh {
// CUDA device of every device call of the host layer: the caller's current device (or RCVD_DEVICE); 0 when no device is usable so that
// the entry point itself reports RCVD_ERR_NO_DEVICE.
inline int currentDevice() { const int d = rcvd_current_device(); return d < 0 ? 0 : d; }
// Host-side loops over independent frames / pairs (depth files, medians, observation records): a few threads, results written to
// per-item slots so that the outcome does not depend on the schedule.  RCVD_HOST_THREADS overrides the count (1 = sequential).
inline int hostThreads() {
  if (const char* e = std::getenv("RCVD_HOST_THREADS")) { const int v = std::atoi(e); if (v > 0) return v; }
  const unsigned hw = std::thread::hardware_concurrency();
  return int(hw == 0 ? 1 : (hw > 16 ? 16 : hw));
}
inline void parallelFor(size_t n, const std::function<void(size_t)>& fn) {
  const size_t nt = std::min<size_t>(size_t(hostThreads()), n);
  if (nt <= 1) { for (size_t i = 0; i < n; ++i) fn(i); return; }
  std::atomic<size_t> next{0}; std::exception_ptr err; std::atomic<bool> failed{false};
  auto work = [&]() {
    for (;;) {
      const size_t i = next.fetch_add(1);
      if (i >= n || failed.load()) return;
      try { fn(i); } catch (...) { if (!failed.exchange(true)) err = std::current_exception(); return; }
    }
  };
  std::vector<std::thread> th;
  for (size_t t = 1; t < nt; ++t) { try { th.emplace_back(work); } catch (const std::system_error&) { break; } }   // no thread to be had: the caller works alone
  work();
  for (auto& t : th) t.join();
  if (err) std::rethrow_exception(err);
}
}

namespace rcvdh {

// OpenCV type codes used on the Python side (cv2.CV_8UC1 ...): depth + ((cn-1) << 3)
constexpr int CV_8U = 0, CV_32S = 4, CV_32F = 5, CV_64F = 6;
inline int cvMakeType(int depth, int cn) { return depth + ((cn - 1) << 3); }
inline int cvDepth(int type) { return type & 7; }
inline int cvChannels(int type) { return (type >> 3) + 1; }

struct Vec3f { float x = 0, y = 0, z = 0; };
struct Quatf {   // Eigen::Quaternionf coefficient order x, y, z, w
  float x = 0, y = 0, z = 0, w = 1;
  Vec3f rotate(const Vec3f& v) const;   // Eigen: operator*(Vector3f)
};

struct Image {   // row-major interleaved, like cv::Mat (continuous)
  int rows = 0, cols = 0, type = 0;
  std::vector<uint8_t> data;
  bool empty() const { return rows == 0 || cols == 0; }
  size_t elemSize() const { static const int ds[8] = {1, 1, 2, 2, 4, 4, 8, 2}; return size_t(ds[cvDepth(type)]) * cvChannels(type); }
  void create(int r, int c, int t) { rows = r; cols = c; type = t; data.assign(size_t(r) * c * elemSize(), 0); }
  template <class T> T* ptr(int y = 0) { return reinterpret_cast<T*>(data.data() + size_t(y) * cols * elemSize()); }
  template <class T> const T* ptr(int y = 0) const { return reinterpret_cast<const T*>(data.data() + size_t(y) * cols * elemSize()); }
};
void freadim(const std::string& fileName, Image& dst);        // lib/core/CvUtil.cpp:25-42
void fwriteim(const std::string& fileName, const Image& src); // :98-113
Image imreadPng(const std::string& fileName, bool grayscale); // cv::imread subset (8-bit PNG)

// --- FrameRange (lib/FrameRange.{h,cpp}) ---
struct FrameRange {
  std::set<int> frames;
  void fromString(const std::string& str);
  std::string toString() const;
  void resolve(int numFrames, bool clip = false);
  bool isEmpty() const { return frames.empty(); }
  void checkEmpty() const;
  int firstFrame() const;
  int lastFrame() const;
  int count() const { return int(frames.size()); }
  bool isConsecutive() const;
  bool inRange(int frame) const { return frames.count(frame) > 0; }
};

// --- transforms (lib/DepthMapTransform.h, lib/ValueTransform.h) ---
enum class ValueXformType { None, Scale, ScaleShift };
enum class XformType { Depth, Spatial };
enum class DepthXformType { None, Identity, Global, Grid };
enum class SpatialXformType { None, Identity, VerticalLinear, CornersBilinear, BilinearGrid, BicubicGrid };

struct XformDescriptor {
  XformType type = XformType::Depth;
  DepthXformType depthType = DepthXformType::Identity;
  SpatialXformType spatialType = SpatialXformType::None;
  ValueXformType valueXform = ValueXformType::None;
  bool cubicInterpolation = false;
  std::array<int, 3> gridSize{{0, 0, 0}};
  std::array<double, 2> depthMinMax{{0.0, 0.0}};
  void reset(XformType t = XformType::Depth);
  std::string str() const;
  void parse(const std::string& s);
  bool operator==(const XformDescriptor& o) const {
    return type == o.type && depthType == o.depthType && spatialType == o.spatialType && valueXform == o.valueXform && gridSize == o.gridSize;
  }
  bool operator!=(const XformDescriptor& o) const { return !(*this == o); }
};

class DepthFrame;
// One class for all transforms: descriptor + flat parameter vector with the reference's layout
// (grid node x + y*gx, k values per node; spatial 2 per node).
class Xform {
 public:
  explicit Xform(const XformDescriptor& desc);
  Xform(const Xform&) = delete;
  std::unique_ptr<Xform> clone() const;
  void copyFrom(const Xform& other);
  const XformDescriptor& desc() const { return desc_; }
  std::string str() const;
  std::vector<double>& params() { return params_; }
  const std::vector<double>& params() const { return params_; }
  int numParams() const { return int(params_.size()); }
  int valueParams() const { return desc_.valueXform == ValueXformType::ScaleShift ? 2 : 1; }
  // DepthXform::paramMap (lib/DepthMapTransform.cpp:950-994), SpatialXform::warp (:428-449),
  // DepthXform::apply (:394-415) -- evaluated by the CUDA dense kernels (rcvd_depth_param_map etc.).
  Image paramMap(const DepthFrame& df) const;
  Image warp(int h, int w) const;
  Image apply(const Image& src) const;
  void fillConfig(rcvd_config& cfg) const;   // descriptor -> C ABI fields
 private:
  XformDescriptor desc_;
  std::vector<double> params_;
};
void fillDepthConfig(const XformDescriptor& d, rcvd_config& cfg);
void fillSpatialConfig(const XformDescriptor& d, rcvd_config& cfg);
// the one-frame rcvd_config the dense kernels (rcvd_depth_apply, rcvd_depth_param_map, rcvd_spatial_warp) take for a transform
void denseConfig(const XformDescriptor& d, rcvd_config& cfg);

// --- DepthPhoto::Intrinsics / Extrinsics (lib/DepthPhoto.{h,cpp}) ---
struct Extrinsics {
  Vec3f position;
  Quatf orientation;
  Vec3f left() const { return orientation.rotate({-1, 0, 0}); }
  Vec3f right() const { return orientation.rotate({1, 0, 0}); }
  Vec3f down() const { return orientation.rotate({0, -1, 0}); }
  Vec3f up() const { return orientation.rotate({0, 1, 0}); }
  Vec3f forward() const { return orientation.rotate({0, 0, -1}); }
  Vec3f backward() const { return orientation.rotate({0, 0, 1}); }
};
struct Intrinsics {
  float vFov = 0.f, hFov = 0.f, centerLat = 0.f, centerLon = 0.f;
  void resolveMissingFov(float aspect);   // lib/DepthPhoto.cpp:114-158
};

class DepthVideo;
class DepthStream;
class ColorStream;

class ColorFrame {
 public:
  ColorFrame(ColorStream& s, int index) : stream_(s), index_(index) {}
  ColorFrame(const ColorFrame&) = delete;
  const Image* image();    // lazily loaded, cached; nullptr if the file does not exist
  void clearCache() { img_.reset(); loaded_ = false; }
 private:
  ColorStream& stream_; int index_; std::unique_ptr<Image> img_; bool loaded_ = false;
};
class ColorStream {
 public:
  explicit ColorStream(DepthVideo& v) : video_(v) {}
  ColorStream(const ColorStream&) = delete;
  ColorFrame& frame(int i);
  const std::string& name() const { return name_; }
  const std::string& path() const { return path_; }
  const std::string& extension() const { return extension_; }
  int type() const { return type_; }
  int width();
  int height();
  void setDir(const std::string& dir);
  std::string name_, dir_, path_, extension_; int type_ = 0; int width_ = -1, height_ = -1;
  std::vector<std::unique_ptr<ColorFrame>> frames_;
  DepthVideo& video_;
};

class DepthFrame {
 public:
  DepthFrame(DepthVideo& v, DepthStream& s, int index);
  DepthFrame(const DepthFrame&) = delete;
  const Image* sourceDepth();          // depth = 1/disparity from depth/frame_%06d.raw (lib/DepthStream.cpp:193-216)
  const Image* depth();                // transformed depth (lib/DepthStream.cpp:266-290)
  void setDepth(const Image& depth);   // becomes the new source depth; transformed caches dropped (lib/DepthStream.cpp:102-116)
  void clear();                        // caches + default intrinsics / extrinsics (:145-149)
  void clearCache() { source_.reset(); sourceLoaded_ = false; xformed_.reset(); medianValid_ = false; }
  // median of ALL source depth samples incl. zeros, nth_element at size/2 (lib/PoseOptimizer.cpp:1363-1375); cached: the source
  // depth does not change between the optimisation steps that ask for it
  float sourceDepthMedian();
  void clearXformedCache() { xformed_.reset(); }
  Xform& depthXform() { return *depthXform_; }
  const Xform& depthXform() const { return *depthXform_; }
  Xform& spatialXform() { return *spatialXform_; }
  const Xform& spatialXform() const { return *spatialXform_; }
  void resetDepthXform();
  void resetSpatialXform();
  int width() const;
  int height() const;
  float invAspect() const;
  Intrinsics intrinsics;
  Extrinsics extrinsics;
  bool enabled = true;
 private:
  DepthVideo& video_; DepthStream& stream_; int index_;
  std::unique_ptr<Image> source_, xformed_; bool sourceLoaded_ = false; bool medianValid_ = false; float median_ = 0.f;
  XformDescriptor appliedDesc_; std::vector<double> appliedParams_;   // what xformed_ was computed with
  std::unique_ptr<Xform> depthXform_, spatialXform_;
};
class DepthStream {
 public:
  explicit DepthStream(DepthVideo& v) : video_(v) {}
  DepthStream(const DepthStream&) = delete;
  DepthFrame& frame(int i);
  const std::string& name() const { return name_; }
  const std::string& path() const { return path_; }
  const XformDescriptor& depthXformDesc() const { return depthXformDesc_; }
  const XformDescriptor& spatialXformDesc() const { return spatialXformDesc_; }
  int width();
  int height();
  void setDir(const std::string& dir);
  void resetDepthXforms(const XformDescriptor& desc);
  void resetSpatialXforms(const XformDescriptor& desc);
  void clearCache() { for (auto& f : frames_) f->clearCache(); }
  // Loads the source depth (and, if asked, the medians) of the given frames on several threads; the first one is loaded alone because it
  // fixes the stream's dimensions, which the others only compare against.
  void preloadSourceDepth(const std::vector<int>& frames, bool medians);
  std::string name_, dir_, path_; int width_ = -1, height_ = -1;
  XformDescriptor depthXformDesc_, spatialXformDesc_;
  std::vector<std::unique_ptr<DepthFrame>> frames_;
  DepthVideo& video_;
};

class DepthVideo {
 public:
  DepthVideo() = default;
  DepthVideo(const DepthVideo&) = delete;
  void init(const std::string& path, int width, int height, const std::vector<float>& pts);   // lib/DepthVideo.cpp:103-119
  void save();                                                                                 // :300-385 (video.dat)
  void load(const std::string& path);                                                          // :120-298 (video.dat as written by save())
  void saveDepth(int stream);                                                                  // :597-635 (depth/frame_%06d.raw as disparity)
  void printInfo() const;
  int width() const { return width_; }
  int height() const { return height_; }
  float aspect() const { return aspect_; }
  float invAspect() const { return invAspect_; }
  const std::string& path() const { return path_; }
  int numFrames() const { return int(pts_.size()); }
  int numColorStreams() const { return int(colorStreams_.size()); }
  bool hasColorStream(const std::string& name) const;
  int colorStreamIndex(const std::string& name) const;
  ColorStream& colorStream(int i);
  ColorStream& colorStream(const std::string& name) { return colorStream(colorStreamIndex(name)); }
  void createColorStream(const std::string& name, const std::string& dir, const std::string& ext, int type, std::pair<int, int> size);
  int numDepthStreams() const { return int(depthStreams_.size()); }
  bool hasDepthStream(const std::string& name) const;
  int depthStreamIndex(const std::string& name) const;
  DepthStream& depthStream(int i);
  DepthStream& depthStream(const std::string& name) { return depthStream(depthStreamIndex(name)); }
  void createDepthStream(const std::string& name, const std::string& dir, std::pair<int, int> size);
  DepthFrame& depthFrame(int stream, int frame) { return depthStream(stream).frame(frame); }
  void clearDepthCaches() { for (auto& s : depthStreams_) s->clearCache(); }
  std::vector<float> pts_;
 private:
  std::string path_; int width_ = 0, height_ = 0; float aspect_ = 0.f, invAspect_ = 0.f, duration_ = 0.f;
  std::vector<std::unique_ptr<ColorStream>> colorStreams_;
  std::vector<std::unique_ptr<DepthStream>> depthStreams_;
};
void importVideo(DepthVideo& video, const std::string& path, bool discoverStreams);   // lib/Importer.cpp:25-37, :197-238

// --- flow constraints (lib/FlowConstraints.{h,cpp}) ---
struct FlowConstraintsParams {
  int matchSeparation = 10;
  float minDynamicDistance = -1.f;
  FrameRange frameRange;
  bool doNotUseCache = false;
};
struct PairConstraint { float loc[2][2]; bool isStatic = true; };       // [obs][x,y], float32 like Vector2fna
struct TripletConstraint { float loc[3][2]; bool isStatic = true; };
using PairKey = std::pair<int, int>;

class FlowConstraintsCollection {
 public:
  FlowConstraintsCollection(DepthVideo& video, const FlowConstraintsParams& params);
  bool load();
  void save();
  void resetStaticFlag();
  void setStaticFlagFromDynamicMask(int distance);
  void pruneStaticFlag(int distance);
  const std::map<PairKey, std::vector<PairConstraint>>& pairs() const { return pairs_; }
  const std::map<int, std::vector<TripletConstraint>>& triplets() const { return triplets_; }
  void compute();                       // GPU builder (rcvd_build_constraints) unless RCVD_CONSTRAINT_BUILDER=host
  void computeOnDevice();
  void compute(const PairKey& pair);
  void computeTriplet(int triplet);
 private:
  Image dynamicDistance(int frame);
  DepthVideo* video_; std::string path_; FlowConstraintsParams params_;
  std::map<PairKey, std::vector<PairConstraint>> pairs_;
  std::map<int, std::vector<TripletConstraint>> triplets_;
};
// image ops restating the OpenCV calls of lib/FlowConstraints.cpp:249,279,419,423
Image bgr2gray32f(const Image& bgr);
Image cornerMinEigenVal3(const Image& gray32f);
Image distanceTransformL2_5(const Image& bin8u);

// --- optimizer (lib/PoseOptimizer.{h,cpp}) ---
enum class StaticLossType { Euclidean, ReproDisparity, ReproDepthRatio, ReproLogDepth };
enum class SmoothLossType { EuclideanLaplacian, ReproDisparityLaplacian, ReproDepthRatioConsistency, ReproLogDepthConsistency };
enum class IntrinsicsOptimization { Fixed, Shared, PerFrame };

class DepthVideoPoseOptimizer {
 public:
  struct Params {   // lib/PoseOptimizer.h:54-108
    FrameRange frameRange;
    int maxIterations = 1000; int numThreads = 12; int numSteps = 4; double robustness = 0.5;
    StaticLossType staticLossType = StaticLossType::ReproDisparity; double staticSpatialWeight = 1.0, staticDepthWeight = 1.0;
    SmoothLossType smoothLossType = SmoothLossType::ReproDisparityLaplacian; double smoothStaticWeight = 0.0, smoothDynamicWeight = 0.0;
    double positionReg = 0.0, scaleReg = 1.0; int scaleRegGridSize = 10;
    double depthDeformRegInitial = 1.0, depthDeformRegFinal = 0.1, adaptiveDeformationCost = 0.0, spatialDeformReg = 1.0;
    bool graduateDepthDeformReg = false; double focalReg = 1.0;
    bool coarseToFine = true; int ctfLong = 17, ctfShort = 10;
    bool deferredSpatialOpt = false; int dsoLong = 4, dsoShort = 3;
    double focalLong = 0.3461538376301239; IntrinsicsOptimization intrOpt = IntrinsicsOptimization::PerFrame;
    bool fixPoses = false, fixDepthXforms = false, fixSpatialXforms = false;
    bool normalizeDepthFromFirstFrame = true;
  };
  DepthVideoPoseOptimizer(DepthVideo* video, int depthStream);
  void poseOptimization(const Params& params, const FlowConstraintsCollection& constraints);
  void poseOptimizationStep(const Params& params, const FlowConstraintsCollection& constraints, double depthDeformReg);
  void normalizeDepth(const Params& params, const FlowConstraintsCollection& constraints);
  // exposed for tests: the exact arrays handed to the C ABI for one step
  struct ProblemArrays {
    rcvd_config cfg; std::vector<uint8_t> inRange; std::vector<double> median, adaptive, state;
    std::vector<int32_t> pairFrames; std::vector<int64_t> offsets; std::vector<float> records;
    std::vector<int32_t> tripCenters; std::vector<int64_t> tripOffsets; std::vector<float> tripRecords;   // smoothness triplets, 10 floats each
    int pairCount = 0; int64_t constraintCount = 0;
  };
  ProblemArrays buildProblem(const Params& params, const FlowConstraintsCollection* constraints, double depthDeformReg, bool normalize);
  // record cache of one poseOptimization() call (see buildProblem)
  bool recordCacheOn_ = false, recordCacheValid_ = false; std::vector<int32_t> cachedPairFrames_; std::vector<int64_t> cachedOffsets_; std::vector<float> cachedRecords_;
  int cachedPairCount_ = 0; int64_t cachedConstraintCount_ = 0;
  const std::vector<std::array<double, 7>>& poseParams() const { return poseParams_; }
 private:
  void solveAndWriteBack(ProblemArrays& pa, const Params& params, bool writePoses);
  DepthVideo* video_; int depthStream_; int numFrames_ = 0;
  std::vector<std::array<double, 7>> poseParams_;
};

class DepthVideoProcessor {
 public:
  enum class Op { None, Reset, Copy, BilateralFilter, FlowGuidedFilter, ComputeConstraints, ResetConstraintStaticFlag,
                  SetConstraintStaticFlagFromDynamicMask, ComputeTracks, GridXformSplit, ResetPoses, ResetDepthXforms,
                  ResetSpatialXforms, NormalizeDepth, OptimizePoses, ResetNormalizeOptimize };
  struct Params {   // lib/Processor.h:60-90
    Op op = Op::None; FrameRange frameRange; int colorStream = 0, depthStream = 0, sourceDepthStream = 0;
    int spatialRadius = 0, frameRadius = 2; float depthSigma = 0.3f, colorSigma = 0.0f; bool median = false; bool farConnections = false;
    float maxDepth = 1000.f;
    int matchSeparation = 10; float flowConsistancyThresh = 0.05f; int trackSpawnDistance = 20, trackPruneDistance = 5;
    int minDynamicDistance = 3; int minTrackLength = 4;
    XformDescriptor depthXformDesc, spatialXformDesc; DepthVideoPoseOptimizer::Params poseOptimizer;
  };
  explicit DepthVideoProcessor(DepthVideo* video) : video_(video) {}
  void process(const Params& params);
  void reset(const Params& params);               // lib/Processor.cpp:146-150
  void copy(const Params& params);                // :152-180
  void bilateralFilter(const Params& params);     // :183-313, on the GPU (rcvd_bilateral_filter)
  void flowGuidedFilter(const Params& params);    // :315-590, on the GPU (rcvd_flow_guided_filter)
  void gridXformSplit(const Params& params);      // lib/Processor.cpp:888-985
  void resetPoses(const Params& params);          // :987-1003
  void resetDepthXforms(const Params& params);    // :1005-1008
  void resetSpatialXforms(const Params& params);  // :1010-1013
  void normalizeDepth(const Params& params, const FlowConstraintsCollection& constraints);   // :1015-1019
  void optimizePoses(const Params& params, const FlowConstraintsCollection& constraints);    // :1021-1025
 private:
  DepthVideo* video_;
};

// Conversions restated from Ceres / Eigen (host side of lib/PoseOptimizer.cpp:748-783, :964-987)
void quatToAngleAxis(const Quatf& q, double aa[3]);          // Eigen q -> rotation(right, up, -front) -> ceres::RotationMatrixToAngleAxis
Quatf angleAxisToQuat(const double aa[3]);                   // ceres::AngleAxisToRotationMatrix -> Eigen::Quaterniond(R).cast<float>()

void logInfo(const std::string& s);
void setLogToStdout(bool v);

}  // namespace rcvdh
