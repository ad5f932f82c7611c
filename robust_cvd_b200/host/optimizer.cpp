// optimizer.cpp -- DepthVideoPoseOptimizer / DepthVideoProcessor host logic.
//
// Same control flow as the reference (lib/PoseOptimizer.cpp:788-1147, lib/Processor.cpp:888-1034):
// problem assembly from the DepthVideo + FlowConstraintsCollection, coarse-to-fine schedule, pose
// write-back -- but "ceres::Solve" is the CUDA library behind include/rcvd.h.  No CPU solver here.
#include "model.h"
#include <dirent.h>
#include <cstring>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <stdexcept>

namespace rcvdh {

DepthVideoPoseOptimizer::DepthVideoPoseOptimizer(DepthVideo* video, int depthStream) : video_(video), depthStream_(depthStream) {
  numFrames_ = video_->numFrames();
  poseParams_.resize(numFrames_);
  for (int f = 0; f < numFrames_; ++f) {   // lib/PoseOptimizer.cpp:755-782
    DepthFrame& df = video_->depthFrame(depthStream_, f);
    auto& pose = poseParams_[f];
    pose[0] = df.extrinsics.position.x; pose[1] = df.extrinsics.position.y; pose[2] = df.extrinsics.position.z;
    quatToAngleAxis(df.extrinsics.orientation, &pose[3]);
    pose[6] = std::tan(df.intrinsics.vFov / 2.0);
  }
}

static void checkStatus(int rc) { if (rc != RCVD_OK) throw std::runtime_error(std::string("rcvd: ") + rcvd_last_error()); }

DepthVideoPoseOptimizer::ProblemArrays DepthVideoPoseOptimizer::buildProblem(const Params& params, const FlowConstraintsCollection* constraints,
                                                                             double depthDeformReg, bool normalize) {
  ProblemArrays pa;
  DepthStream& ds = video_->depthStream(depthStream_);
  rcvd_config& cfg = pa.cfg; memset(&cfg, 0, sizeof(cfg));
  cfg.num_frames = numFrames_;
  fillDepthConfig(ds.depthXformDesc(), cfg); fillSpatialConfig(ds.spatialXformDesc(), cfg);
  if (cfg.value_xform == RCVD_VALUE_NONE) cfg.value_xform = RCVD_VALUE_SCALE;
  if (ds.depthXformDesc().depthType == DepthXformType::Grid && ds.depthXformDesc().gridSize[2] > 1) throw std::runtime_error("Bilateral depth grids are not supported.");
  const double aspect = video_->aspect();                                        // float -> double (:1155)
  const double vFocal = (aspect >= 1.f ? params.focalLong / aspect : params.focalLong);   // :1156-1157
  cfg.aspect = aspect; cfg.fixed_vfocal = vFocal; cfg.focal_target = vFocal;
  cfg.intr_opt = int(params.intrOpt); cfg.static_loss_type = int(params.staticLossType);
  cfg.robust_type = RCVD_ROBUST_CAUCHY; cfg.robustness = params.robustness;       // ceres::CauchyLoss(robustness), :1219-1220
  cfg.static_spatial_weight = params.staticSpatialWeight; cfg.static_depth_weight = params.staticDepthWeight;
  // scale-regulariser lattice (:1346-1351)
  int gx = params.scaleRegGridSize; int gy = int(std::round(float(gx) * video_->invAspect()));
  if (video_->aspect() <= 1.f) std::swap(gx, gy);
  cfg.scale_grid_x = gx; cfg.scale_grid_y = gy;
  cfg.smooth_loss_type = int(params.smoothLossType);
  FrameRange range = params.frameRange;
  if (range.isEmpty()) range.resolve(numFrames_);
  pa.inRange.assign(numFrames_, 0);
  for (int f : range.frames) { if (f < 0 || f >= numFrames_) throw std::runtime_error("Frame range contains out-of-range frame indices."); pa.inRange[f] = 1; }
  if (normalize) {   // normalizeDepth, :992-1147
    cfg.scale_reg = params.scaleReg > 0.0 ? params.scaleReg : 0.0;
    cfg.depth_deform_reg = params.depthDeformRegInitial > 0.0 ? params.depthDeformRegInitial : 0.0;
    cfg.depth_lower_bound = 1;
  } else {           // poseOptimizationStep, :890-953
    cfg.position_reg = params.positionReg > 0.0 ? params.positionReg : 0.0;
    cfg.depth_deform_reg = depthDeformReg > 0.0 ? depthDeformReg : 0.0;
    cfg.spatial_deform_reg = params.spatialDeformReg > 0.0 ? params.spatialDeformReg : 0.0;
    cfg.fix_poses = params.fixPoses; cfg.fix_depth_xforms = params.fixDepthXforms; cfg.fix_spatial_xforms = params.fixSpatialXforms;
    cfg.scale_reg = (!params.fixDepthXforms && params.scaleReg > 0.0) ? params.scaleReg : 0.0;
    cfg.focal_reg = params.focalReg > 0.0 ? params.focalReg : 0.0;
  }
  cfg.adaptive_deform = (params.adaptiveDeformationCost > 0.0 && cfg.depth_deform_reg > 0.0 && cfg.depth_type == RCVD_DEPTH_GRID) ? params.adaptiveDeformationCost : 0.0;
  const int stride = rcvd_frame_stride(&cfg);
  if (stride < 0) throw std::runtime_error("Unsupported transform configuration for the optimizer.");
  const int offD = rcvd_depth_param_offset(&cfg), offS = rcvd_spatial_param_offset(&cfg);
  // medians (:1363-1375): over ALL depth samples including zeros, nth_element at size/2
  pa.median.assign(numFrames_, 1.0);
  if (cfg.scale_reg > 0.0) {
    ds.preloadSourceDepth(std::vector<int>(range.frames.begin(), range.frames.end()), true);   // files + nth_element of every frame, in parallel
    for (int f : range.frames) pa.median[f] = ds.frame(f).sourceDepthMedian();
  }
  // adaptive deformation weights (AdaptiveDeformationCost ctor, :559-619)
  if (cfg.adaptive_deform > 0.0) {
    if (!video_->hasColorStream("dynamic_mask")) throw std::runtime_error("Adaptive smoothness requires a dynamic mask stream.");
    const int gw = cfg.depth_grid_x, gh = cfg.depth_grid_y;
    pa.adaptive.assign(size_t(numFrames_) * gw * gh, 0.0);
    for (int f : range.frames) {
      const Image* m = video_->colorStream("dynamic_mask").frame(f).image();
      if (!m) throw std::runtime_error("Dynamic mask stream is missing a frame.");
      std::vector<double> dyn(size_t(gw) * gh, 0.0), sta(size_t(gw) * gh, 0.0);
      for (int y = 0; y < m->rows; ++y) { const double fy = double(y) * (gh - 1) / m->rows; const int iy = int(fy); const double ry = fy - iy;
        for (int x = 0; x < m->cols; ++x) { const double fx = double(x) * (gw - 1) / m->cols; const int ix = int(fx); const double rx = fx - ix;
          std::vector<double>& w = m->data[size_t(y) * m->cols + x] > 127 ? sta : dyn;
          w[size_t(iy) * gw + ix] += (1.0 - rx) * (1.0 - ry); w[size_t(iy) * gw + ix + 1] += rx * (1.0 - ry);
          w[size_t(iy + 1) * gw + ix] += (1.0 - rx) * ry; w[size_t(iy + 1) * gw + ix + 1] += rx * ry; } }
      for (int i = 0; i < gw * gh; ++i) pa.adaptive[size_t(f) * gw * gh + i] = dyn[i] / (dyn[i] + sta[i]);
    }
  }
  // static-scene constraints (addStaticSceneLoss :1149-1240, Observation :104-117)
  pa.offsets.assign(1, 0);
  if (!normalize && constraints && recordCacheOn_ && recordCacheValid_) {
    // the coarse-to-fine steps of one poseOptimization() call see the same constraints and source depths: the records are assembled once
    pa.pairFrames = cachedPairFrames_; pa.offsets = cachedOffsets_; pa.records = cachedRecords_; pa.pairCount = cachedPairCount_; pa.constraintCount = cachedConstraintCount_;
  } else if (!normalize && constraints) {
    const float invAspect = video_->invAspect();
    // pairs with both ends in range, in map order; their records are assembled in parallel into per-pair slots and concatenated in order
    struct PairJob { int f0, f1; const std::vector<PairConstraint>* list; const Image* d0; const Image* d1; std::vector<float> rec; };
    std::vector<PairJob> jobs;
    { std::set<int> touched;
      for (const auto& kv : constraints->pairs()) if (range.inRange(kv.first.first) && range.inRange(kv.first.second)) { touched.insert(kv.first.first); touched.insert(kv.first.second); }
      ds.preloadSourceDepth(std::vector<int>(touched.begin(), touched.end()), false); }
    for (const auto& kv : constraints->pairs()) {
      const int f0 = kv.first.first, f1 = kv.first.second;
      if (!range.inRange(f0) || !range.inRange(f1)) continue;
      const Image* d0 = ds.frame(f0).sourceDepth(); const Image* d1 = ds.frame(f1).sourceDepth();
      if (!d0 || !d1) throw std::runtime_error("Missing depth image.");
      jobs.push_back({f0, f1, &kv.second, d0, d1, {}});
    }
    parallelFor(jobs.size(), [&](size_t j) {
      PairJob& job = jobs[j];
      job.rec.reserve(job.list->size() * 6);
      for (const PairConstraint& c : *job.list) {
        if (!c.isStatic) continue;
        float rec[6];
        bool ok = true;
        for (int o = 0; o < 2; ++o) {
          const Image* d = o ? job.d1 : job.d0;
          const float lx = c.loc[o][0], ly = c.loc[o][1];
          rec[o * 3] = -1.f + 2.f * lx; rec[o * 3 + 1] = 1.f - 2.f * ly / invAspect;
          int px = int(lx * d->cols), py = int(ly / invAspect * d->rows);
          // the reference indexes the Mat unchecked (SURVEY A1 quirk for targets in (-1.5,-0.5]); clamp instead of reading out of bounds
          px = std::min(std::max(px, 0), d->cols - 1); py = std::min(std::max(py, 0), d->rows - 1);
          const float sd = d->ptr<float>(py)[px];
          rec[o * 3 + 2] = sd;
          if (!std::isfinite(sd) || sd <= 0) ok = false;
        }
        if (!ok) continue;
        job.rec.insert(job.rec.end(), rec, rec + 6);
      }
    });
    size_t total = 0; for (const PairJob& job : jobs) total += job.rec.size();
    pa.records.reserve(total);
    for (const PairJob& job : jobs) {
      ++pa.pairCount;
      pa.records.insert(pa.records.end(), job.rec.begin(), job.rec.end());
      const int64_t n = int64_t(job.rec.size()) / 6;
      pa.pairFrames.push_back(job.f0); pa.pairFrames.push_back(job.f1);
      pa.offsets.push_back(pa.offsets.back() + n);
      pa.constraintCount += n;
    }
    if (recordCacheOn_) { cachedPairFrames_ = pa.pairFrames; cachedOffsets_ = pa.offsets; cachedRecords_ = pa.records; cachedPairCount_ = pa.pairCount; cachedConstraintCount_ = pa.constraintCount; recordCacheValid_ = true; }
  }
  // scene-flow smoothness constraints (addSceneFlowSmoothnessLoss :1242-1339): only if either weight is positive (:899-901)
  pa.tripOffsets.assign(1, 0);
  if (!normalize && constraints && (params.smoothStaticWeight > 0.0 || params.smoothDynamicWeight > 0.0)) {
    const float invAspect = video_->invAspect();
    for (int frame = range.firstFrame(); frame < range.lastFrame() - 1; ++frame) {
      if (!range.inRange(frame) || !range.inRange(frame + 1) || !range.inRange(frame + 2)) continue;
      const int triplet = frame + 1;
      auto it = constraints->triplets().find(triplet);
      if (it == constraints->triplets().end()) throw std::runtime_error("Missing triplet constraints.");
      const Image* dimg[3];
      for (int o = 0; o < 3; ++o) { dimg[o] = ds.frame(frame + o).sourceDepth(); if (!dimg[o]) throw std::runtime_error("Missing depth image."); }
      const size_t before = pa.tripRecords.size();
      for (const TripletConstraint& c : it->second) {
        float rec[10]; bool ok = true;
        for (int o = 0; o < 3; ++o) {
          const Image* d = dimg[o];
          const float lx = c.loc[o][0], ly = c.loc[o][1];
          rec[o * 3] = -1.f + 2.f * lx; rec[o * 3 + 1] = 1.f - 2.f * ly / invAspect;
          int px = int(lx * d->cols), py = int(ly / invAspect * d->rows);
          px = std::min(std::max(px, 0), d->cols - 1); py = std::min(std::max(py, 0), d->rows - 1);
          const float sd = d->ptr<float>(py)[px];
          rec[o * 3 + 2] = sd;
          if (!std::isfinite(sd) || sd <= 0) ok = false;
        }
        if (!ok) continue;
        rec[9] = float(c.isStatic ? params.smoothStaticWeight : params.smoothDynamicWeight);   // ScaledLoss weight (:1314-1317)
        pa.tripRecords.insert(pa.tripRecords.end(), rec, rec + 10);
      }
      pa.tripCenters.push_back(triplet);
      pa.tripOffsets.push_back(pa.tripOffsets.back() + int64_t(pa.tripRecords.size() - before) / 10);
    }
  }
  // state
  pa.state.assign(size_t(numFrames_) * stride, 0.0);
  for (int f = 0; f < numFrames_; ++f) {
    double* x = &pa.state[size_t(f) * stride];
    for (int i = 0; i < 7; ++i) x[i] = poseParams_[f][i];
    const auto& dp = ds.frame(f).depthXform().params(); const auto& sp = ds.frame(f).spatialXform().params();
    if (int(dp.size()) != offS - offD || int(sp.size()) != stride - offS) throw std::runtime_error("Transform parameter count does not match the stream descriptor.");
    std::copy(dp.begin(), dp.end(), x + offD); std::copy(sp.begin(), sp.end(), x + offS);
  }
  return pa;
}

void DepthVideoPoseOptimizer::solveAndWriteBack(ProblemArrays& pa, const Params& params, bool writePoses) {
  logInfo("Solving...");
  rcvd_problem* p = nullptr;
  checkStatus(rcvd_problem_create(&pa.cfg, currentDevice(), &p));
  try {
    checkStatus(rcvd_problem_set_frames(p, pa.inRange.data(), pa.median.data(), pa.adaptive.empty() ? nullptr : pa.adaptive.data()));
    checkStatus(rcvd_problem_set_constraints(p, int(pa.pairFrames.size() / 2), pa.pairFrames.data(), pa.offsets.data(), pa.records.data()));
    if (!pa.tripCenters.empty()) checkStatus(rcvd_problem_set_triplets(p, int(pa.tripCenters.size()), pa.tripCenters.data(), pa.tripOffsets.data(), pa.tripRecords.data()));
    checkStatus(rcvd_problem_set_state(p, pa.state.data()));
    rcvd_solve_options opt; rcvd_default_solve_options(&opt);
    opt.max_iterations = params.maxIterations; opt.verbose = 1;   // minimizer_progress_to_stdout = true (:957)
    rcvd_solve_summary sum;
    checkStatus(rcvd_solve(p, &opt, &sum));
    char b[320];
    snprintf(b, sizeof(b), "rcvd Solver Report: Iterations: %d, Initial cost: %e, Final cost: %e, Termination: %s (%s) [%.1f ms, %lld kernel launches]",
             sum.iterations, sum.initial_cost, sum.final_cost, sum.termination == RCVD_TERM_CONVERGENCE ? "CONVERGENCE" : sum.termination == RCVD_TERM_NO_CONVERGENCE ? "NO_CONVERGENCE" : "FAILURE",
             sum.message, sum.total_ms, (long long)sum.gpu_launches);
    logInfo(b);
    checkStatus(rcvd_problem_get_state(p, pa.state.data()));
  } catch (...) { rcvd_problem_destroy(p); throw; }
  rcvd_problem_destroy(p);
  const int stride = rcvd_frame_stride(&pa.cfg), offD = rcvd_depth_param_offset(&pa.cfg), offS = rcvd_spatial_param_offset(&pa.cfg);
  DepthStream& ds = video_->depthStream(depthStream_);
  for (int f = 0; f < numFrames_; ++f) {
    const double* x = &pa.state[size_t(f) * stride];
    for (int i = 0; i < 7; ++i) poseParams_[f][i] = x[i];
    auto& dp = ds.frame(f).depthXform().params(); auto& sp = ds.frame(f).spatialXform().params();
    std::copy(x + offD, x + offS, dp.begin()); std::copy(x + offS, x + stride, sp.begin());
  }
  if (!writePoses) return;
  FrameRange range = params.frameRange; if (range.isEmpty()) range.resolve(numFrames_);
  for (int f : range.frames) {   // :964-987
    const auto& pose = poseParams_[f];
    DepthFrame& df = ds.frame(f);
    df.extrinsics.position = {float(pose[0]), float(pose[1]), float(pose[2])};
    df.extrinsics.orientation = angleAxisToQuat(&pose[3]);
    df.clearXformedCache();
    const double phi = (params.intrOpt == IntrinsicsOptimization::Shared) ? poseParams_[0][6] : pose[6];
    df.intrinsics.vFov = float(std::atan(phi) * 2.f);
    df.intrinsics.hFov = float(std::atan(phi * video_->aspect()) * 2.f);
  }
}

void DepthVideoPoseOptimizer::poseOptimizationStep(const Params& params, const FlowConstraintsCollection& constraints, double depthDeformReg) {
  logInfo("Building problem...");
  ProblemArrays pa = buildProblem(params, &constraints, depthDeformReg, false);
  logInfo("    Using " + std::to_string(pa.pairCount) + " frame pairs.");
  logInfo("    Added " + std::to_string(pa.constraintCount) + " constraints.");
  solveAndWriteBack(pa, params, true);
}

void DepthVideoPoseOptimizer::normalizeDepth(const Params& params, const FlowConstraintsCollection& constraints) {
  logInfo("------------------------");
  logInfo("Depth Normalization (depth stream " + std::to_string(depthStream_) + ")...");
  if (!params.normalizeDepthFromFirstFrame) throw std::runtime_error("normalizeDepthFromFirstFrame = false is not supported (it is not reachable from Python in the reference either).");
  (void)constraints;
  ProblemArrays pa = buildProblem(params, nullptr, 0.0, true);
  solveAndWriteBack(pa, params, false);
  FrameRange range = params.frameRange; if (range.isEmpty()) range.resolve(numFrames_);
  DepthStream& ds = video_->depthStream(depthStream_);
  const int first = range.firstFrame();   // copy the first frame's transform to all others (:1127-1138)
  for (int f : range.frames) { if (f != first) ds.frame(f).depthXform().copyFrom(ds.frame(first).depthXform()); }
  for (int f : range.frames) ds.frame(f).clearXformedCache();
}

void DepthVideoPoseOptimizer::poseOptimization(const Params& params, const FlowConstraintsCollection& constraints) {   // :788-888
  logInfo("------------------------");
  logInfo("Pose optimization (depth stream " + std::to_string(depthStream_) + ")...");
  int ctfRows = params.ctfLong, ctfCols = params.ctfShort, dsoRows = params.dsoLong, dsoCols = params.dsoShort;
  if (video_->aspect() >= 1.f) { std::swap(ctfCols, ctfRows); std::swap(dsoCols, dsoRows); }
  auto gridSize = [](const XformDescriptor& d) { return d.depthType == DepthXformType::Grid ? d.gridSize : std::array<int, 3>{{1, 1, 1}}; };
  DepthStream& ds = video_->depthStream(depthStream_);
  const std::array<int, 3> initGrid = gridSize(ds.depthXformDesc());
  DepthVideoProcessor processor(video_);
  struct CacheScope {   // observation records (constraint locations + source depths) do not change between the steps of this call
    DepthVideoPoseOptimizer* o;
    explicit CacheScope(DepthVideoPoseOptimizer* o_) : o(o_) { o->recordCacheOn_ = true; o->recordCacheValid_ = false; }
    ~CacheScope() { o->recordCacheOn_ = false; o->recordCacheValid_ = false; std::vector<float>().swap(o->cachedRecords_); }
  } cacheScope(this);
  if (params.deferredSpatialOpt) {
    DepthVideoProcessor::Params pp; pp.depthStream = depthStream_; pp.spatialXformDesc.type = XformType::Spatial; pp.spatialXformDesc.depthType = DepthXformType::None; pp.spatialXformDesc.spatialType = SpatialXformType::Identity;
    processor.resetSpatialXforms(pp);
  }
  for (int step = 0; step < params.numSteps; ++step) {
    logInfo("----------------");
    logInfo("Step " + std::to_string(step + 1) + " / " + std::to_string(params.numSteps) + "...");
    const double stepIter = (params.numSteps > 1 ? step / double(params.numSteps - 1) : 0.0);
    double depthDeformReg = params.depthDeformRegFinal;
    if (params.graduateDepthDeformReg) { const double a = std::log(params.depthDeformRegInitial), b = std::log(params.depthDeformRegFinal); depthDeformReg = std::exp(a + (b - a) * stepIter); }
    poseOptimizationStep(params, constraints, depthDeformReg);
    if (params.coarseToFine && step < params.numSteps - 1) {
      const double ctfIter = (step + 1) / double(params.numSteps - 1);
      DepthVideoProcessor::Params sp; sp.depthStream = depthStream_; sp.depthXformDesc = ds.depthXformDesc();
      if (sp.depthXformDesc.depthType == DepthXformType::Global) sp.depthXformDesc.depthType = DepthXformType::Grid;
      sp.depthXformDesc.gridSize[0] = int(initGrid[0] + (ctfCols - initGrid[0]) * ctfIter + 0.5);
      sp.depthXformDesc.gridSize[1] = int(initGrid[1] + (ctfRows - initGrid[1]) * ctfIter + 0.5);
      sp.depthXformDesc.gridSize[2] = initGrid[2];
      logInfo("Splitting grid --> " + std::to_string(sp.depthXformDesc.gridSize[0]) + " x " + std::to_string(sp.depthXformDesc.gridSize[1]) + " x " + std::to_string(sp.depthXformDesc.gridSize[2]) + "...");
      processor.gridXformSplit(sp);
    }
  }
  if (params.deferredSpatialOpt) {
    DepthVideoProcessor::Params pp; pp.depthStream = depthStream_; pp.spatialXformDesc.type = XformType::Spatial; pp.spatialXformDesc.depthType = DepthXformType::None; pp.spatialXformDesc.spatialType = SpatialXformType::BicubicGrid;
    pp.spatialXformDesc.gridSize[1] = dsoRows; pp.spatialXformDesc.gridSize[0] = dsoCols;
    processor.resetSpatialXforms(pp);
    poseOptimizationStep(params, constraints, params.depthDeformRegFinal);
  }
}

// ---------------------------------------------------------------------------
void DepthVideoProcessor::process(const Params& params) {   // lib/Processor.cpp:115-144
  struct Trim { ~Trim() { rcvd_trim_device_memory(currentDevice()); } } trimAtExit;   // hand the cached device memory back (PyTorch shares the GPU)
  switch (params.op) {
    case Op::None: break;
    case Op::GridXformSplit: gridXformSplit(params); break;
    case Op::ResetPoses: resetPoses(params); break;
    case Op::ResetDepthXforms: resetDepthXforms(params); break;
    case Op::ResetSpatialXforms: resetSpatialXforms(params); break;
    case Op::Reset: reset(params); break;
    case Op::Copy: copy(params); break;
    case Op::FlowGuidedFilter: flowGuidedFilter(params); break;
    case Op::BilateralFilter: bilateralFilter(params); break;
    default: throw std::runtime_error("Unsupported operation selected.");
  }
}
void DepthVideoProcessor::reset(const Params& params) {   // :146-150
  for (int frame : params.frameRange.frames) video_->depthFrame(params.depthStream, frame).clear();
}
void DepthVideoProcessor::copy(const Params& params) {   // :152-180
  if (params.sourceDepthStream < 0 || params.sourceDepthStream >= video_->numDepthStreams()) throw std::runtime_error("Source depth stream out of range.");
  if (params.sourceDepthStream == params.depthStream) throw std::runtime_error("Source and destination depth stream cannot be identical.");
  DepthStream& srcDs = video_->depthStream(params.sourceDepthStream);
  DepthStream& dstDs = video_->depthStream(params.depthStream);
  for (int frame : params.frameRange.frames) {
    DepthFrame& src = srcDs.frame(frame); DepthFrame& dst = dstDs.frame(frame);
    const Image* depth = src.depth();
    if (!depth) throw std::runtime_error("Source depth frame " + std::to_string(frame) + " has no depth image.");
    dst.setDepth(*depth);
    dst.intrinsics = src.intrinsics; dst.extrinsics = src.extrinsics;
  }
}
// Bilateral filter (:183-313).  The reference filters frame by frame on the CPU, reading depth stream 0 and the "down" colour
// stream whatever params.sourceDepthStream / colorStream say.  Here the host gathers the transformed depth of every frame a
// temporal window reaches (and the colour only when the colour term is on) and rcvd_bilateral_filter (csrc/rcvd_bilateral.cuh)
// filters the whole range.  With depthStream == 0 the reference's write-back between frames is honoured on the device: a later
// window reads the depth transform applied to an earlier filtered frame, exactly what depth() returns after setDepth.
void DepthVideoProcessor::bilateralFilter(const Params& params) {
  logInfo("Applying bilateral filter...");
  // every argument is checked before the first depth() call: depth() applies the transform on the GPU
  if (params.spatialRadius < 0 || params.frameRadius < 0) throw std::runtime_error("Spatial and frame radius must be non-negative.");
  params.frameRange.checkEmpty();
  const int numFrames = video_->numFrames(), R = params.frameRadius;
  const int first = params.frameRange.firstFrame(), last = params.frameRange.lastFrame();
  if (first < 0 || last >= numFrames) throw std::runtime_error("Frame index out of range.");
  DepthStream& ds = video_->depthStream(0);
  DepthStream& dstDs = video_->depthStream(params.depthStream);
  ColorStream& cs = video_->colorStream("down");
  if (cs.type() != cvMakeType(CV_32F, 3)) throw std::runtime_error("Image has incorrect type.");   // ColorFrame::image3f
  const bool useColor = params.colorSigma > 0.f, inPlace = params.depthStream == 0;
  const int base = std::max(0, first - R), F = std::min(numFrames - 1, last + R) - base + 1;
  std::vector<char> reached(F, 0);
  for (int f : params.frameRange.frames) for (int g = std::max(0, f - R); g <= std::min(numFrames - 1, f + R); ++g) reached[g - base] = 1;
  const int w = ds.width(), h = ds.height();
  if (w <= 0 || h <= 0) throw std::runtime_error("Depth stream 0 has no depth frames.");
  for (int i = 0; i < F; ++i) {
    if (!reached[i]) continue;
    if (!ds.frame(base + i).sourceDepth()) throw std::runtime_error("Depth frame " + std::to_string(base + i) + " has no depth image.");
    if (useColor) {
      const Image* c = cs.frame(base + i).image();
      if (!c) throw std::runtime_error("Color frame " + std::to_string(base + i) + " has no image.");
      if (c->cols != w || c->rows != h) throw std::runtime_error("Color frame " + std::to_string(base + i) + " does not have the depth frame's size.");
    }
  }
  std::vector<int32_t> outFrames;
  for (int f : params.frameRange.frames) outFrames.push_back(f - base);
  // in place: the depth transform of every output frame, applied again to its filtered image on the device
  rcvd_config cfg{}; std::vector<double> xp(1, 0.0);
  const bool chain = inPlace && R > 0;
  if (chain) {
    const XformDescriptor& desc = ds.frame(first).depthXform().desc();
    denseConfig(desc, cfg);
    const int nd = rcvd_spatial_param_offset(&cfg) - rcvd_depth_param_offset(&cfg);
    if (nd < 0) throw std::runtime_error("Unsupported depth transform for in-place filtering.");
    xp.assign(std::max<size_t>(1, size_t(outFrames.size()) * nd), 0.0);
    for (size_t k = 0; k < outFrames.size(); ++k) {
      const Xform& x = ds.frame(base + outFrames[k]).depthXform();
      if (x.desc() != desc || x.numParams() != nd) throw std::runtime_error("Depth transforms of the frame range differ.");
      std::copy(x.params().begin(), x.params().end(), xp.begin() + k * nd);
    }
  }
  std::vector<float> depth(size_t(F) * w * h, 0.f), color(useColor ? size_t(F) * w * h * 3 : 0);
  for (int i = 0; i < F; ++i) {
    if (!reached[i]) continue;
    const Image* d = ds.frame(base + i).depth();
    std::memcpy(depth.data() + size_t(i) * w * h, d->ptr<float>(), size_t(w) * h * sizeof(float));
    if (useColor) std::memcpy(color.data() + size_t(i) * w * h * 3, cs.frame(base + i).image()->ptr<float>(), size_t(w) * h * 3 * sizeof(float));
  }
  rcvd_bilateral_params prm{};
  prm.num_frames = F; prm.num_out = int(outFrames.size()); prm.width = w; prm.height = h;
  prm.spatial_radius = params.spatialRadius; prm.frame_radius = R; prm.median = params.median ? 1 : 0; prm.in_place = inPlace ? 1 : 0;
  prm.depth_sigma = params.depthSigma; prm.color_sigma = params.colorSigma;
  std::vector<float> out(size_t(prm.num_out) * w * h);
  const int rc = rcvd_bilateral_filter(&prm, currentDevice(), depth.data(), useColor ? color.data() : nullptr, outFrames.data(),
                                       chain ? &cfg : nullptr, chain ? xp.data() : nullptr, out.data());
  if (rc != RCVD_OK) throw std::runtime_error(std::string("bilateral filter failed: ") + rcvd_last_error());
  for (size_t k = 0; k < outFrames.size(); ++k) {   // range order, as the reference writes
    Image img; img.create(h, w, cvMakeType(CV_32F, 1));
    std::memcpy(img.ptr<float>(), out.data() + k * w * h, size_t(w) * h * sizeof(float));
    dstDs.frame(base + outFrames[k]).setDepth(img);
  }
}

// Flow-guided temporal filter (:315-590).  The reference walks frame by frame and pixel by pixel on the CPU; here the host
// gathers the depth images, cameras and consecutive-frame flows of the whole range once and one kernel launch
// (rcvd_flow_guided_filter, csrc/rcvd_filter.cuh) filters every frame.
void DepthVideoProcessor::flowGuidedFilter(const Params& params) {
  logInfo("Applying flow guided filter...");
  if (!params.frameRange.isConsecutive()) throw std::runtime_error("Frame range must be consecutive.");
  params.frameRange.checkEmpty();
  ColorStream& cs = video_->colorStream("down");
  const int w = cs.width(), h = cs.height();
  if (w <= 0 || h <= 0) throw std::runtime_error("Color stream 'down' has no frames.");
  DepthStream& srcDs = video_->depthStream(params.sourceDepthStream);
  DepthStream& dstDs = video_->depthStream(params.depthStream);
  const int first = params.frameRange.firstFrame(), last = params.frameRange.lastFrame();
  if (params.sourceDepthStream == params.depthStream)   // the reference would then read frames it has already filtered (order dependent)
    throw std::runtime_error("Source and destination depth stream cannot be identical.");
  // frames held on the device: the temporal windows of the range, or the whole video when far connections may point anywhere
  const int winBase = std::max(0, first - params.frameRadius);
  const int base = params.farConnections ? 0 : winBase, F = (params.farConnections ? video_->numFrames() - 1 : last) - base + 1;
  const size_t plane = size_t(w) * h;
  auto flowFile = [&](int a, int b) { char buf[64]; snprintf(buf, sizeof(buf), "/flow/flow_%06d_%06d.raw", a, b); return video_->path() + buf; };
  auto maskFile = [&](int a, int b) { char buf[64]; snprintf(buf, sizeof(buf), "/flow_mask/mask_%06d_%06d.png", a, b); return video_->path() + buf; };
  auto loadPair = [&](int a, int b, float* flowDst, uint8_t* maskDst, bool required) -> bool {
    Image flow, mask;
    bool ok = false;
    try {
      freadim(flowFile(a, b), flow); mask = imreadPng(maskFile(a, b), true);
      ok = flow.cols == w && flow.rows == h && flow.type == cvMakeType(CV_32F, 2) && mask.cols == w && mask.rows == h;
    } catch (const std::exception&) { ok = false; }
    if (!ok) { if (required) throw std::runtime_error("Missing or mismatched flow / flow mask for frames " + std::to_string(a) + " -> " + std::to_string(b) + "."); return false; }
    std::memcpy(flowDst, flow.ptr<float>(), plane * 2 * sizeof(float)); std::memcpy(maskDst, mask.ptr<uint8_t>(), plane);
    return true;
  };
  // depth + cameras of frames base .. last
  int wd = -1, hd = -1;
  std::vector<float> depth, cams(size_t(F) * 9);
  for (int i = 0; i < F; ++i) {
    DepthFrame& df = srcDs.frame(base + i);
    const Image* d = df.depth();
    if (!d) throw std::runtime_error("Source depth frame " + std::to_string(base + i) + " has no depth image.");
    if (wd < 0) { wd = d->cols; hd = d->rows; depth.resize(size_t(F) * wd * hd); }
    if (d->cols != wd || d->rows != hd) throw std::runtime_error("Depth frame has inconsistent dimensions.");
    std::memcpy(depth.data() + size_t(i) * wd * hd, d->ptr<float>(), size_t(wd) * hd * sizeof(float));
    float* c = cams.data() + size_t(i) * 9;
    c[0] = df.extrinsics.position.x; c[1] = df.extrinsics.position.y; c[2] = df.extrinsics.position.z;
    c[3] = df.extrinsics.orientation.x; c[4] = df.extrinsics.orientation.y; c[5] = df.extrinsics.orientation.z; c[6] = df.extrinsics.orientation.w;
    c[7] = df.intrinsics.hFov; c[8] = df.intrinsics.vFov;
  }
  // consecutive-frame flows: slot i holds (base+i -> base+i+1) resp. (base+i -> base+i-1); every slot a chain can reach is required (:405-413 CHECKs)
  std::vector<float> fwd, bwd; std::vector<uint8_t> fwdMask, bwdMask;
  if (params.frameRadius > 0 && F > 1) {
    fwd.assign(size_t(F) * plane * 2, 0.f); bwd.assign(size_t(F) * plane * 2, 0.f); fwdMask.assign(size_t(F) * plane, 0); bwdMask.assign(size_t(F) * plane, 0);
    for (int f = winBase; f < last; ++f) {
      const int i = f - base;
      if (f >= first) loadPair(f, f + 1, fwd.data() + size_t(i) * plane * 2, fwdMask.data() + size_t(i) * plane, true);    // forward chains start at frames >= first
      loadPair(f + 1, f, bwd.data() + size_t(i + 1) * plane * 2, bwdMask.data() + size_t(i + 1) * plane, true);
    }
  }
  // far connections (:415-427): every flow file (frame, fi) with fi outside the temporal window of `frame`
  std::vector<int32_t> farPairs; std::vector<float> farFlow; std::vector<uint8_t> farMask;
  if (params.farConnections) {
    std::vector<std::pair<int, int>> flowPairs;
    if (DIR* dir = opendir((video_->path() + "/flow").c_str())) {
      while (dirent* e = readdir(dir)) {
        const std::string name = e->d_name; const size_t dot = name.rfind('.');
        const std::string stem = dot == std::string::npos ? name : name.substr(0, dot);
        if (stem.size() != 18 || stem.substr(0, 5) != "flow_") continue;
        flowPairs.emplace_back(std::stoi(stem.substr(5, 6)), std::stoi(stem.substr(12, 6)));
      }
      closedir(dir);
    }
    std::sort(flowPairs.begin(), flowPairs.end());   // directory order is unspecified in the reference; sorted here
    for (const auto& pr : flowPairs) {
      const int frame = pr.first, fi = pr.second;
      if (frame < first || frame > last || fi < 0 || fi >= video_->numFrames()) continue;
      const int f0 = std::max(0, frame - params.frameRadius), f1 = std::min(last, frame + params.frameRadius);
      if (!(fi < f0 || fi > f1)) continue;
      const size_t k = farPairs.size() / 2;
      farFlow.resize((k + 1) * plane * 2); farMask.resize((k + 1) * plane);
      if (!loadPair(frame, fi, farFlow.data() + k * plane * 2, farMask.data() + k * plane, false)) { farFlow.resize(k * plane * 2); farMask.resize(k * plane); continue; }
      farPairs.push_back(frame - base); farPairs.push_back(fi - base);
    }
  }
  rcvd_filter_params prm{};
  prm.num_frames = F; prm.first_out = first - base; prm.num_out = last - first + 1; prm.width = w; prm.height = h; prm.depth_width = wd; prm.depth_height = hd;
  prm.frame_radius = params.frameRadius; prm.spatial_radius = params.spatialRadius; prm.median = params.median ? 1 : 0; prm.num_far = int(farPairs.size() / 2);
  prm.inv_aspect = video_->invAspect();
  std::vector<float> out(size_t(prm.num_out) * plane);
  const int rc = rcvd_flow_guided_filter(&prm, currentDevice(), depth.data(), cams.data(), fwd.empty() ? nullptr : fwd.data(), fwdMask.empty() ? nullptr : fwdMask.data(),
                                         bwd.empty() ? nullptr : bwd.data(), bwdMask.empty() ? nullptr : bwdMask.data(),
                                         farPairs.empty() ? nullptr : farPairs.data(), farFlow.empty() ? nullptr : farFlow.data(), farMask.empty() ? nullptr : farMask.data(), out.data());
  if (rc != RCVD_OK) throw std::runtime_error(std::string("flow guided filter failed: ") + rcvd_last_error());
  for (int i = 0; i < prm.num_out; ++i) {
    Image img; img.create(h, w, cvMakeType(CV_32F, 1));
    std::memcpy(img.ptr<float>(), out.data() + size_t(i) * plane, plane * sizeof(float));
    dstDs.frame(first + i).setDepth(img);
  }
}
void DepthVideoProcessor::gridXformSplit(const Params& params) {   // :888-985
  if (params.depthXformDesc.depthType != DepthXformType::Grid) throw std::runtime_error("Transform type must be a grid type.");
  DepthStream& ds = video_->depthStream(params.depthStream);
  const XformDescriptor prev = ds.depthXformDesc();
  if (prev.depthType != DepthXformType::Global && prev.depthType != DepthXformType::Grid) throw std::runtime_error("Can only split global or grid type transforms.");
  if (params.depthXformDesc.valueXform != prev.valueXform) throw std::runtime_error("Old and new transforms must use same value transform.");
  if (prev.depthType != DepthXformType::Global && (prev.gridSize[0] > params.depthXformDesc.gridSize[0] || prev.gridSize[1] > params.depthXformDesc.gridSize[1]))
    throw std::runtime_error("New transform must have at least the same number of rows and columns as the old transform.");
  std::vector<std::unique_ptr<Xform>> prevX;
  for (int f = 0; f < video_->numFrames(); ++f) prevX.push_back(ds.frame(f).depthXform().clone());
  ds.resetDepthXforms(params.depthXformDesc);
  const int newCols = params.depthXformDesc.gridSize[0], newRows = params.depthXformDesc.gridSize[1];
  for (int f = 0; f < video_->numFrames(); ++f) {
    const std::vector<double>& pp = prevX[f]->params();
    std::vector<double>& np = ds.frame(f).depthXform().params();
    const int N = prevX[f]->valueParams();
    for (int row = 0; row < newRows; ++row) for (int col = 0; col < newCols; ++col) {
      const int idx = col + row * newCols;
      if (prev.depthType == DepthXformType::Global) { for (int i = 0; i < N; ++i) np[size_t(idx) * N + i] = pp[i]; continue; }
      const int prevRows = prev.gridSize[1], prevCols = prev.gridSize[0];
      const double maxx = std::nextafter(double(prevCols - 1), 0.0), maxy = std::nextafter(double(prevRows - 1), 0.0);
      const double sx = std::min(col / double(newCols - 1) * (prevCols - 1), maxx), sy = std::min(row / double(newRows - 1) * (prevRows - 1), maxy);
      const int ix = int(sx), iy = int(sy);
      const double rx = sx - ix, ry = sy - iy;
      const double w0 = (1.f - rx) * (1.f - ry), w1 = rx * (1.f - ry), w2 = (1.f - rx) * ry, w3 = rx * ry;
      const double* b0 = &pp[size_t(ix + iy * prevCols) * N]; const double* b1 = &pp[size_t(ix + 1 + iy * prevCols) * N];
      const double* b2 = &pp[size_t(ix + (iy + 1) * prevCols) * N]; const double* b3 = &pp[size_t(ix + 1 + (iy + 1) * prevCols) * N];
      for (int i = 0; i < N; ++i) np[size_t(idx) * N + i] = b0[i] * w0 + b1[i] * w1 + b2[i] * w2 + b3[i] * w3;
    }
  }
}
void DepthVideoProcessor::resetPoses(const Params& params) {   // :987-1003
  DepthStream& ds = video_->depthStream(params.depthStream);
  for (int f = 0; f < video_->numFrames(); ++f) {
    DepthFrame& df = ds.frame(f);
    df.extrinsics.position = Vec3f(); df.extrinsics.orientation = Quatf();
    const float focal = float(params.poseOptimizer.focalLong);
    if (video_->aspect() >= 1.f) { df.intrinsics.hFov = std::atan(focal) * 2.f; df.intrinsics.vFov = std::atan(focal / video_->aspect()) * 2.f; }
    else { df.intrinsics.hFov = std::atan(focal * video_->aspect()) * 2.f; df.intrinsics.vFov = std::atan(focal) * 2.f; }
  }
}
void DepthVideoProcessor::resetDepthXforms(const Params& params) { video_->depthStream(params.depthStream).resetDepthXforms(params.depthXformDesc); }
void DepthVideoProcessor::resetSpatialXforms(const Params& params) { video_->depthStream(params.depthStream).resetSpatialXforms(params.spatialXformDesc); }
void DepthVideoProcessor::normalizeDepth(const Params& params, const FlowConstraintsCollection& constraints) {
  DepthVideoPoseOptimizer optimizer(video_, params.depthStream); optimizer.normalizeDepth(params.poseOptimizer, constraints);
  rcvd_trim_device_memory(currentDevice());
}
void DepthVideoProcessor::optimizePoses(const Params& params, const FlowConstraintsCollection& constraints) {
  DepthVideoPoseOptimizer optimizer(video_, params.depthStream); optimizer.poseOptimization(params.poseOptimizer, constraints);
  rcvd_trim_device_memory(currentDevice());   // the solver's cached device memory goes back to the driver: the fine-tuning stage (PyTorch) runs next on this GPU
}

}  // namespace rcvdh
