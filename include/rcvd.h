/*
 * rcvd.h -- C ABI of the B200-native temporal-consistency optimizer.
 *
 * This is the drop-in boundary beneath the reference's `lib_python` module
 * (reference: lib/PythonBindings.cpp:170-555).  Everything the reference does
 * inside `DepthVideoPoseOptimizer::poseOptimizationStep` and
 * `DepthVideoPoseOptimizer::normalizeDepth` between "Building problem..." and
 * the pose write-back (lib/PoseOptimizer.cpp:890-990, :992-1147) is replaced
 * by one `rcvd_problem_*` object:
 *
 *   reference                                   | this ABI
 *   --------------------------------------------+------------------------------
 *   problem_ = make_unique<ceres::Problem>()    | rcvd_problem_create
 *     (lib/PoseOptimizer.cpp:895, :1000)        |
 *   addStaticSceneLoss (:1149-1240)             | rcvd_problem_set_constraints
 *   addScaleRegularization (:1341-1415),        | rcvd_problem_set_frames
 *   addDepthDeformRegularization (:1449-1495),  |   (+ weights in rcvd_config)
 *   addSpatialDeformRegularization (:1497-1522),|
 *   addFocalRegularization (:1524-1549),        |
 *   addPositionRegularization (:1417-1447)      |
 *   addSceneFlowSmoothnessLoss (:1242-1339)     | rcvd_problem_set_triplets
 *   poseParams_ / xform params_ (:748-783)      | rcvd_problem_set_state / get_state
 *   ceres::Solve (:954-962, :1117-1125)         | rcvd_solve
 *
 * Plain structs, caller-owned host buffers, int status codes, no exceptions
 * and no torch types cross this boundary.  One CUDA stream (and optionally one
 * NCCL communicator) is owned by the handle.  Thread-compatible, not
 * thread-safe.
 */
#ifndef RCVD_H_
#define RCVD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Enum values follow the reference's enum order so that the pybind layer can
 * cast directly (lib/DepthMapTransform.h:24-46, lib/ValueTransform.h:16-20,
 * lib/PoseOptimizer.h:22-50). */
enum { RCVD_DEPTH_NONE = 0, RCVD_DEPTH_IDENTITY = 1, RCVD_DEPTH_GLOBAL = 2, RCVD_DEPTH_GRID = 3 };
enum { RCVD_VALUE_NONE = 0, RCVD_VALUE_SCALE = 1, RCVD_VALUE_SCALESHIFT = 2 };
enum {
  RCVD_SPATIAL_NONE = 0, RCVD_SPATIAL_IDENTITY = 1, RCVD_SPATIAL_VERTICAL_LINEAR = 2,
  RCVD_SPATIAL_CORNERS_BILINEAR = 3, RCVD_SPATIAL_BILINEAR_GRID = 4, RCVD_SPATIAL_BICUBIC_GRID = 5
};
enum { RCVD_INTR_FIXED = 0, RCVD_INTR_SHARED = 1, RCVD_INTR_PER_FRAME = 2 };
enum { RCVD_LOSS_EUCLIDEAN = 0, RCVD_LOSS_REPRO_DISPARITY = 1, RCVD_LOSS_REPRO_DEPTH_RATIO = 2, RCVD_LOSS_REPRO_LOG_DEPTH = 3 };
/* Robustifier on the static-scene residual blocks.  The reference uses
 * ceres::CauchyLoss(robustness) (lib/PoseOptimizer.cpp:1219-1220).  Huber is an
 * extension (BASELINE.json config 4) with no reference behaviour. */
enum { RCVD_ROBUST_TRIVIAL = 0, RCVD_ROBUST_CAUCHY = 1, RCVD_ROBUST_HUBER = 2 };
/* SmoothLossType of the scene-flow smoothness loss (lib/PoseOptimizer.h:37-42) */
enum { RCVD_SMOOTH_EUCLIDEAN_LAPLACIAN = 0, RCVD_SMOOTH_REPRO_DISPARITY_LAPLACIAN = 1, RCVD_SMOOTH_REPRO_DEPTH_RATIO_CONSISTENCY = 2, RCVD_SMOOTH_REPRO_LOG_DEPTH_CONSISTENCY = 3 };

enum {
  RCVD_OK = 0,
  RCVD_ERR_INVALID = 1,     /* bad argument / unsupported configuration */
  RCVD_ERR_CUDA = 2,        /* CUDA runtime error (see rcvd_last_error) */
  RCVD_ERR_NCCL = 3,
  RCVD_ERR_NUMERIC = 4,     /* factorisation failed beyond recovery */
  RCVD_ERR_NO_DEVICE = 5    /* no usable CUDA device: there is NO CPU fallback */
};

/* Per-frame parameter vector layout (all double):
 *   [0..2] camera position, [3..5] angle-axis rotation, [6] tan(vFov/2)
 *   (reference poseParams_, lib/PoseOptimizer.h:145-149),
 *   then the frame's depth-transform params (row-major grid x + y*gx, k values per
 *   node; lib/DepthMapTransform.cpp:733-736), then its spatial-transform params
 *   (2 per node; :1359-1362).  Stride = rcvd_frame_stride(cfg). */
typedef struct rcvd_config {
  int32_t num_frames;
  int32_t depth_type;        /* RCVD_DEPTH_* */
  int32_t value_xform;       /* RCVD_VALUE_* */
  int32_t depth_cubic;       /* XformDescriptor::cubicInterpolation */
  int32_t depth_grid_x, depth_grid_y;     /* gridSize.x/.y (gz must be 1) */
  int32_t spatial_type;      /* RCVD_SPATIAL_* */
  int32_t spatial_grid_x, spatial_grid_y;
  int32_t intr_opt;          /* RCVD_INTR_* */
  int32_t static_loss_type;  /* RCVD_LOSS_* */
  int32_t robust_type;       /* RCVD_ROBUST_* */
  int32_t fix_poses, fix_depth_xforms, fix_spatial_xforms;  /* lib/PoseOptimizer.cpp:915-948 */
  int32_t depth_lower_bound; /* normalizeDepth: lower bound 0 on param 0 of every depth block (:1108-1115) */
  int32_t scale_grid_x, scale_grid_y;     /* scale-regulariser lattice (:1346-1351) */
  int32_t smooth_loss_type;  /* RCVD_SMOOTH_* (only read when triplet constraints are set) */
  double aspect;             /* double(video.aspect()) (float -> double, :1155) */
  double fixed_vfocal;       /* focalLong/aspect for landscape (:1156-1157) */
  double robustness;         /* Cauchy/Huber scale a */
  double static_spatial_weight, static_depth_weight;
  double scale_reg;          /* <=0: term absent */
  double depth_deform_reg;   /* <=0: term absent */
  double adaptive_deform;    /* >0: needs adaptive node weights in rcvd_problem_set_frames */
  double spatial_deform_reg;
  double focal_reg;
  double focal_target;       /* vFocal target of TargetFocalCost (:1531-1533) */
  double position_reg;
} rcvd_config;

/* Ceres-default trust-region options restated (SURVEY.md section 8c). */
typedef struct rcvd_solve_options {
  int32_t max_iterations;         /* Params::maxIterations (default 1000) */
  int32_t verbose;                /* 1: per-iteration progress line on stderr */
  double function_tolerance;      /* 1e-6 */
  double gradient_tolerance;      /* 1e-10 */
  double parameter_tolerance;     /* 1e-8 */
  double initial_radius;          /* 1e4 */
  double max_radius;              /* 1e16 */
  double min_radius;              /* 1e-32 */
  double min_relative_decrease;   /* 1e-3 */
  double min_lm_diagonal;         /* 1e-6 */
  double max_lm_diagonal;         /* 1e32 */
  int32_t max_consecutive_invalid_steps; /* 5 */
  int32_t jacobi_scaling;         /* 1 */
} rcvd_solve_options;

enum { RCVD_TERM_CONVERGENCE = 0, RCVD_TERM_NO_CONVERGENCE = 1, RCVD_TERM_FAILURE = 2 };

typedef struct rcvd_solve_summary {
  int32_t termination;            /* RCVD_TERM_* */
  int32_t iterations;             /* LM iterations run (excluding iteration 0) */
  int32_t num_successful_steps;
  int32_t num_unsuccessful_steps;
  double initial_cost;
  double final_cost;
  double total_ms;                /* wall clock of the solve call */
  double eval_ms;                 /* device time: residual+Jacobian+accumulate launches */
  double linear_ms;               /* device time: factor + solve launches */
  double cost_ms;                 /* device time: cost-only launches */
  int64_t num_constraints;
  int64_t gpu_launches;           /* kernels launched by this call */
  char message[128];
} rcvd_solve_summary;

typedef struct rcvd_problem rcvd_problem;

/* Last error message of the calling thread (never NULL). */
const char* rcvd_last_error(void);
/* Library/ABI version; bumps when a struct above changes. */
int32_t rcvd_abi_version(void);
/* Number of doubles per frame for this configuration, or -1 if unsupported. */
int32_t rcvd_frame_stride(const rcvd_config* cfg);
/* Offsets inside a frame's parameter vector. */
int32_t rcvd_depth_param_offset(const rcvd_config* cfg);
int32_t rcvd_spatial_param_offset(const rcvd_config* cfg);
void rcvd_default_solve_options(rcvd_solve_options* opt);

/* Creates the device-side problem on CUDA device `device` (cudaSetDevice
 * ordinal).  Fails with RCVD_ERR_NO_DEVICE when no GPU is usable. */
int32_t rcvd_problem_create(const rcvd_config* cfg, int32_t device, rcvd_problem** out);
void rcvd_problem_destroy(rcvd_problem* p);

/* Per-frame inputs.  in_range[N]: frame participates (Params::frameRange).
 * median_depth[N]: median of the frame's source depth incl. zeros
 * (lib/PoseOptimizer.cpp:1363-1375), only read if scale_reg > 0.
 * adaptive_weights[N * gx * gy] (nullable): AdaptiveDeformationCost node
 * weights (:612-618), only read if adaptive_deform > 0. */
int32_t rcvd_problem_set_frames(rcvd_problem* p, const uint8_t* in_range,
                                const double* median_depth, const double* adaptive_weights);

/* Static-scene constraints, already filtered exactly as the reference does
 * (isStatic, both frames in range, finite positive source depths,
 * lib/PoseOptimizer.cpp:1167-1193), grouped by directed frame pair.
 * pair_frames[P][2], offsets[P+1], records[C][6] = {ndc0.x, ndc0.y, depth0,
 * ndc1.x, ndc1.y, depth1} as float32 (Observation, :104-117). */
int32_t rcvd_problem_set_constraints(rcvd_problem* p, int32_t num_pairs, const int32_t* pair_frames,
                                     const int64_t* offsets, const float* records);

/* Scene-flow smoothness constraints (addSceneFlowSmoothnessLoss, lib/PoseOptimizer.cpp:1242-1339), grouped by the centre
 * frame f of the triplet (f-1, f, f+1): centers[T], offsets[T+1], records[n][10] float32 =
 * {ndc.x, ndc.y, depth} for the three observations + the ScaledLoss weight (smoothStaticWeight or
 * smoothDynamicWeight, :1314-1317).  Optional; absent by default as in the reference (both weights 0). */
int32_t rcvd_problem_set_triplets(rcvd_problem* p, int32_t num_groups, const int32_t* centers,
                                  const int64_t* offsets, const float* records);

/* Multi-GPU: this rank only holds a shard of the pairs; accumulated normal
 * equations and costs are all-reduced over `nranks` ranks with NCCL.
 * unique_id is the 128-byte ncclUniqueId (rcvd_nccl_unique_id on rank 0). */
int32_t rcvd_nccl_unique_id(uint8_t out[128]);
int32_t rcvd_problem_init_comm(rcvd_problem* p, int32_t nranks, int32_t rank, const uint8_t unique_id[128]);
/* Multi-GPU: the GLOBAL list of directed frame pairs [num_pairs][2] (all ranks pass the same list) so that every rank builds
 * the identical block structure / elimination order although it only holds a shard of the constraints. */
int32_t rcvd_problem_set_structure(rcvd_problem* p, int32_t num_pairs, const int32_t* pair_frames);
/* regulariser terms are evaluated by the rank that owns frame f: f % nranks == rank */

/* State: params[N * stride] host doubles. */
int32_t rcvd_problem_set_state(rcvd_problem* p, const double* params);
int32_t rcvd_problem_get_state(rcvd_problem* p, double* params);

/* Robustified cost 1/2 sum rho(|r|^2) at the current state (ceres cost), and
 * optionally the gradient J^T r (length N*stride, nullable). */
int32_t rcvd_evaluate(rcvd_problem* p, double* cost, double* gradient);
/* Dense copy of the Gauss-Newton normal matrix J^T J at the current state
 * (row-major (N*stride)^2 doubles) -- test/debug entry point for small problems. */
int32_t rcvd_normal_matrix_dense(rcvd_problem* p, double* H);
/* Runs `iters` residual+Jacobian+accumulate passes (no solve) and returns the
 * mean device time per pass in ms -- the hot kernel in isolation (bench). */
int32_t rcvd_time_accumulate(rcvd_problem* p, int32_t iters, double* ms_per_pass);
/* Runs `iters` fixed-radius Gauss-Newton/LM iterations worth of device work
 * (accumulate + factor + solve + candidate cost) without host decisions,
 * state left unchanged; mean device ms per iteration. */
int32_t rcvd_time_iteration(rcvd_problem* p, int32_t iters, double radius, double* ms_per_iter,
                            double* ms_accumulate, double* ms_linear, double* ms_cost);

/* Levenberg-Marquardt with Ceres semantics (TrustRegionMinimizer +
 * LevenbergMarquardtStrategy + exact sparse Cholesky), replacing
 * ceres::Solve at lib/PoseOptimizer.cpp:954-962 and :1117-1125. */
int32_t rcvd_solve(rcvd_problem* p, const rcvd_solve_options* opt, rcvd_solve_summary* summary);

/* ---- next-row kernels (SURVEY.md section 8f-1): dense transform application ---- */
/* DepthXform::apply (lib/DepthMapTransform.cpp:394-415): dst = xform(src) per pixel.
 * depth_params: the frame's depth-transform params (host). src/dst: h*w float32 host. */
int32_t rcvd_depth_apply(const rcvd_config* cfg, int32_t device, const double* depth_params,
                         const float* src, float* dst, int32_t h, int32_t w);
/* GridDepthXform::paramMap (:950-994): out h*w*k doubles. */
int32_t rcvd_depth_param_map(const rcvd_config* cfg, int32_t device, const double* depth_params,
                             double* out, int32_t h, int32_t w);
/* SpatialXform::warp (:428-449): out h*w*2 float32. */
int32_t rcvd_spatial_warp(const rcvd_config* cfg, int32_t device, const double* spatial_params,
                          float* out, int32_t h, int32_t w);

/* Device memory: handles and the one-shot entry points allocate from the device's stream-ordered pool and keep freed blocks
 * cached (a solve call per schedule step re-uses gigabytes of factor storage).  A host application that shares the GPU with
 * another allocator (the reference's fine-tuning stage runs PyTorch on it) returns the cache to the driver with this call;
 * robust_cvd_b200/host does so at the end of every DepthVideoProcessor operation. */
int32_t rcvd_trim_device_memory(int32_t device);
/* device ordinal the host layer should use: RCVD_DEVICE if set, else the caller's current CUDA device; -1 without a device.
 * Every entry point restores the caller's current device on return. */
int32_t rcvd_current_device(void);

/* ---- flow-guided temporal depth filter (SURVEY.md section 8f-4) ----
 * Replaces DepthVideoProcessor::flowGuidedFilter (lib/Processor.cpp:315-590) for a consecutive frame range in one call.
 * Arrays are indexed by a local frame index 0..num_frames-1 where index 0 is the absolute frame
 * max(0, rangeFirst - frame_radius) (the reference reaches back that far, :395) and the range's last frame is
 * first_out + num_out - 1 (no frame after it is read, :396-397).
 *   depth     [num_frames][depth_height][depth_width] f32  transformed depth of the source stream (DepthFrame::depth())
 *   cams      [num_frames][9] f32  extrinsics position xyz, orientation quaternion x,y,z,w, hFov, vFov (radians)
 *   fwd_flow  [num_frames][height][width][2] f32, fwd_mask [num_frames][height][width] u8: slot i = flow/mask i -> i+1
 *   bwd_flow / bwd_mask: slot i = flow/mask i -> i-1        (slots never reached by a chain may hold anything)
 *   far_pairs [num_far][2] i32 local (source, target) indices, far_flow [num_far][height][width][2], far_mask [num_far][height][width]
 *             (Params::farConnections, :415-427; may be NULL when num_far = 0)
 *   out       [num_out][height][width] f32  filtered depth of frames first_out .. first_out + num_out - 1
 * Float32 arithmetic in the reference's operation order; parity tolerance 1e-5 relative (libm expf/tanf, FMA contraction
 * of the reference build are not pinned). */
typedef struct rcvd_filter_params {
  int32_t num_frames, first_out, num_out;
  int32_t width, height, depth_width, depth_height;
  int32_t frame_radius;   /* Params::frameRadius (lib/Processor.h:68) */
  int32_t spatial_radius; /* Params::spatialRadius */
  int32_t median;         /* Params::median: 0 weighted mean, 1 weighted median */
  int32_t num_far;
  float inv_aspect;       /* DepthVideo::invAspect() */
} rcvd_filter_params;
int32_t rcvd_flow_guided_filter(const rcvd_filter_params* prm, int32_t device, const float* depth, const float* cams,
                                const float* fwd_flow, const uint8_t* fwd_mask, const float* bwd_flow, const uint8_t* bwd_mask,
                                const int32_t* far_pairs, const float* far_flow, const uint8_t* far_mask, float* out);

/* ---- bilateral depth filter ----
 * Replaces DepthVideoProcessor::bilateralFilter (lib/Processor.cpp:183-313).  Arrays are indexed by a local frame index
 * 0..num_frames-1 over a consecutive block of the video that holds every temporal window, i.e. from
 * max(0, first - frame_radius) to min(numFrames - 1, last + frame_radius); frames no window reaches may hold anything.
 *   depth        [num_frames][height][width] f32     transformed depth of depth stream 0 (DepthFrame::depth())
 *   color        [num_frames][height][width][3] f32  "down" colour stream (CV_32FC3); only read, and may be NULL, when color_sigma <= 0
 *   out_frames   [num_out] strictly ascending local indices of the frames to filter (Params::frameRange)
 *   xform_cfg    depth transform of stream 0 and xform_params [num_out][depth params] of each output frame: only read with
 *                in_place and frame_radius > 0
 *   out          [num_out][height][width] f32
 * in_place (depthStream == 0): the reference writes each filtered frame back to stream 0 before the next one, so a later
 * window reads the depth transform applied to the filtered image; frames are then filtered one launch at a time in order.
 * Float32 arithmetic in the reference's operation order; weights use the accurate expf (1 ulp from libm's).  A median pixel
 * whose cumulative weight never reaches half the total (NaN weights) is 0, where the reference leaves it uninitialised.
 * spatial_radius is limited by the TMA box (256 elements) and the shared memory of one CTA: at most 24 with the colour term,
 * about 70 without; a larger radius returns RCVD_ERR_INVALID. */
typedef struct rcvd_bilateral_params {
  int32_t num_frames, num_out;
  int32_t width, height;
  int32_t spatial_radius; /* Params::spatialRadius (lib/Processor.h:66) */
  int32_t frame_radius;   /* Params::frameRadius */
  int32_t median;         /* Params::median: 0 weighted mean, 1 weighted median */
  int32_t in_place;       /* 1: outputs replace the filtered frames' depth before later windows read them (depthStream == 0) */
  float depth_sigma;      /* Params::depthSigma; <= 0 switches the depth term off */
  float color_sigma;      /* Params::colorSigma; <= 0 switches the colour term off */
} rcvd_bilateral_params;
int32_t rcvd_bilateral_filter(const rcvd_bilateral_params* prm, int32_t device, const float* depth, const float* color,
                              const int32_t* out_frames, const rcvd_config* xform_cfg, const double* xform_params, float* out);

/* ---- GPU flow-constraint builder (SURVEY.md section 8f-2) ----
 * Replaces FlowConstraintsCollection::compute (lib/FlowConstraints.cpp:401-550: admission tests, cv::cornerMinEigenVal
 * priorities) and sampleConstraints (:352-397: greedy disc sampler) for a batch of frame pairs and frame triplets.
 * Frames are local indices 0..num_frames-1 into color_bgr / dyn_dist.
 *   color_bgr    [num_frames][height][width][3] f32   "down" colour stream (BGR, as cv::Mat CV_32FC3)
 *   dyn_dist     [num_frames][dyn_height][dyn_width] f32  dynamicDistance() images (:257-286), or NULL when the video has no
 *                dynamic_mask stream (distance = FLT_MAX)
 *   pair_frames  [num_pairs][2], pair_flow [num_pairs][height][width][2] f32, pair_mask [num_pairs][height][width] u8
 *   trip_frames  [num_triplets] centre frame t, trip_flow [num_triplets][2][height][width][2] (t -> t-1, t -> t+1), trip_mask likewise
 * Outputs, in the reference's order (descending corner score; ties, which std::sort leaves unspecified, by scan index):
 *   pair_offsets [num_pairs+1], pair_out [.][4] f32 = scaled (loc0.xy, loc1.xy)  (what flow_constraints.dat stores, :116-224)
 *   trip_offsets [num_triplets+1], trip_out [.][6] f32 = scaled (loc0.xy, loc1.xy, loc2.xy)
 * If a capacity (in constraints) is too small the offsets are still filled (so the caller can size the buffers) and
 * RCVD_ERR_INVALID is returned.  Results are bit-identical to the host builder (robust_cvd_b200/host/constraints.cpp). */
typedef struct rcvd_builder_params {
  int32_t num_frames, width, height, dyn_width, dyn_height;
  int32_t match_separation;        /* FlowConstraintsParams::matchSeparation */
  int32_t num_pairs, num_triplets;
  float min_dynamic_distance;      /* FlowConstraintsParams::minDynamicDistance */
  float inv_aspect;                /* DepthVideo::invAspect() */
} rcvd_builder_params;
int32_t rcvd_build_constraints(const rcvd_builder_params* prm, int32_t device, const float* color_bgr, const float* dyn_dist,
                               const int32_t* pair_frames, const float* pair_flow, const uint8_t* pair_mask,
                               const int32_t* trip_frames, const float* trip_flow, const uint8_t* trip_mask,
                               int64_t* pair_offsets, float* pair_out, int64_t pair_capacity,
                               int64_t* trip_offsets, float* trip_out, int64_t trip_capacity);

/* Static flags of flow constraints on the device: replaces FlowConstraintsCollection::setStaticFlagFromDynamicMask
 * (reference lib/FlowConstraints.cpp:573-660) and the distance images of ::dynamicDistance (:257-286).
 * masks [F][h][w] u8 (dynamic-mask frames: < 127 = dynamic); a constraint is static when
 * cv::distanceTransform(mask >= 127, DIST_L2, 5) > distance at every end, the end's pixel being
 * (int(loc.x * w), int(loc.y * w)) -- y scaled by the WIDTH, as the reference does.
 * pair_locs [n][4] / trip_locs [n][6] float32 in the builder's output layout; *_static one byte per constraint (out);
 * dist_out optional [F][h][w] float32 distance images. */
int32_t rcvd_static_flags(int32_t device, const uint8_t* masks, int32_t num_frames, int32_t height, int32_t width, float distance,
                          int32_t num_pairs, const int32_t* pair_frames, const int64_t* pair_offsets, const float* pair_locs, uint8_t* pair_static,
                          int32_t num_triplets, const int32_t* trip_frames, const int64_t* trip_offsets, const float* trip_locs, uint8_t* trip_static,
                          float* dist_out);

#ifdef __cplusplus
}
#endif
#endif /* RCVD_H_ */
