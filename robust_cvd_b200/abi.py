"""ctypes mirror of include/rcvd.h (the C ABI of the B200 solver).

Struct layouts must match include/rcvd.h exactly; `tests/test_abi.py` checks
sizes against the compiled library (`rcvd_abi_version`, `rcvd_frame_stride`).
Enum values follow the reference (lib/DepthMapTransform.h:24-46,
lib/ValueTransform.h:16-20, lib/PoseOptimizer.h:22-50).
"""
import ctypes as C

DEPTH_NONE, DEPTH_IDENTITY, DEPTH_GLOBAL, DEPTH_GRID = 0, 1, 2, 3
VALUE_NONE, VALUE_SCALE, VALUE_SCALESHIFT = 0, 1, 2
(SPATIAL_NONE, SPATIAL_IDENTITY, SPATIAL_VERTICAL_LINEAR, SPATIAL_CORNERS_BILINEAR,
 SPATIAL_BILINEAR_GRID, SPATIAL_BICUBIC_GRID) = range(6)
INTR_FIXED, INTR_SHARED, INTR_PER_FRAME = 0, 1, 2
LOSS_EUCLIDEAN, LOSS_REPRO_DISPARITY, LOSS_REPRO_DEPTH_RATIO, LOSS_REPRO_LOG_DEPTH = 0, 1, 2, 3
ROBUST_TRIVIAL, ROBUST_CAUCHY, ROBUST_HUBER = 0, 1, 2
TERM_CONVERGENCE, TERM_NO_CONVERGENCE, TERM_FAILURE = 0, 1, 2
OK, ERR_INVALID, ERR_CUDA, ERR_NCCL, ERR_NUMERIC, ERR_NO_DEVICE = range(6)


class Config(C.Structure):
    _fields_ = [
        ("num_frames", C.c_int32), ("depth_type", C.c_int32), ("value_xform", C.c_int32),
        ("depth_cubic", C.c_int32), ("depth_grid_x", C.c_int32), ("depth_grid_y", C.c_int32),
        ("spatial_type", C.c_int32), ("spatial_grid_x", C.c_int32), ("spatial_grid_y", C.c_int32),
        ("intr_opt", C.c_int32), ("static_loss_type", C.c_int32), ("robust_type", C.c_int32),
        ("fix_poses", C.c_int32), ("fix_depth_xforms", C.c_int32), ("fix_spatial_xforms", C.c_int32),
        ("depth_lower_bound", C.c_int32), ("scale_grid_x", C.c_int32), ("scale_grid_y", C.c_int32),
        ("smooth_loss_type", C.c_int32),
        ("aspect", C.c_double), ("fixed_vfocal", C.c_double), ("robustness", C.c_double),
        ("static_spatial_weight", C.c_double), ("static_depth_weight", C.c_double),
        ("scale_reg", C.c_double), ("depth_deform_reg", C.c_double), ("adaptive_deform", C.c_double),
        ("spatial_deform_reg", C.c_double), ("focal_reg", C.c_double), ("focal_target", C.c_double),
        ("position_reg", C.c_double),
    ]


class SolveOptions(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int32), ("verbose", C.c_int32),
        ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
        ("parameter_tolerance", C.c_double), ("initial_radius", C.c_double),
        ("max_radius", C.c_double), ("min_radius", C.c_double),
        ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
        ("max_lm_diagonal", C.c_double),
        ("max_consecutive_invalid_steps", C.c_int32), ("jacobi_scaling", C.c_int32),
    ]


class SolveSummary(C.Structure):
    _fields_ = [
        ("termination", C.c_int32), ("iterations", C.c_int32),
        ("num_successful_steps", C.c_int32), ("num_unsuccessful_steps", C.c_int32),
        ("initial_cost", C.c_double), ("final_cost", C.c_double),
        ("total_ms", C.c_double), ("eval_ms", C.c_double), ("linear_ms", C.c_double), ("cost_ms", C.c_double),
        ("num_constraints", C.c_int64), ("gpu_launches", C.c_int64),
        ("message", C.c_char * 128),
    ]


def default_solve_options(max_iterations=1000, verbose=0):
    """Ceres defaults as used by the reference (lib/PoseOptimizer.cpp:955-961)."""
    return SolveOptions(
        max_iterations=max_iterations, verbose=verbose, function_tolerance=1e-6,
        gradient_tolerance=1e-10, parameter_tolerance=1e-8, initial_radius=1e4,
        max_radius=1e16, min_radius=1e-32, min_relative_decrease=1e-3,
        min_lm_diagonal=1e-6, max_lm_diagonal=1e32, max_consecutive_invalid_steps=5,
        jacobi_scaling=1)


class FilterParams(C.Structure):
    """rcvd_filter_params (include/rcvd.h)."""
    _fields_ = [(n, C.c_int32) for n in ("num_frames", "first_out", "num_out", "width", "height", "depth_width", "depth_height",
                                         "frame_radius", "spatial_radius", "median", "num_far")] + [("inv_aspect", C.c_float)]


class BilateralParams(C.Structure):
    """rcvd_bilateral_params (include/rcvd.h)."""
    _fields_ = [(n, C.c_int32) for n in ("num_frames", "num_out", "width", "height", "spatial_radius", "frame_radius", "median", "in_place")] + \
               [("depth_sigma", C.c_float), ("color_sigma", C.c_float)]


class BuilderParams(C.Structure):
    """rcvd_builder_params (include/rcvd.h)."""
    _fields_ = [(n, C.c_int32) for n in ("num_frames", "width", "height", "dyn_width", "dyn_height", "match_separation", "num_pairs", "num_triplets")] + \
               [("min_dynamic_distance", C.c_float), ("inv_aspect", C.c_float)]


def default_config(num_frames, aspect, **kw):
    """Config with the reference's Params defaults (lib/PoseOptimizer.h:55-103)."""
    focal_long = kw.pop("focal_long", 0.3461538376301239)
    vfocal = focal_long / aspect if aspect >= 1.0 else focal_long
    cfg = Config(
        num_frames=num_frames, depth_type=DEPTH_GLOBAL, value_xform=VALUE_SCALE, depth_cubic=0,
        depth_grid_x=0, depth_grid_y=0, spatial_type=SPATIAL_IDENTITY, spatial_grid_x=0, spatial_grid_y=0,
        intr_opt=INTR_PER_FRAME, static_loss_type=LOSS_REPRO_DISPARITY, robust_type=ROBUST_CAUCHY,
        fix_poses=0, fix_depth_xforms=0, fix_spatial_xforms=0, depth_lower_bound=0,
        scale_grid_x=0, scale_grid_y=0, smooth_loss_type=0,
        aspect=aspect, fixed_vfocal=vfocal, robustness=0.5,
        static_spatial_weight=1.0, static_depth_weight=1.0, scale_reg=1.0,
        depth_deform_reg=0.1, adaptive_deform=0.0, spatial_deform_reg=1.0, focal_reg=1.0,
        focal_target=vfocal, position_reg=0.0)
    # scale-regulariser lattice, lib/PoseOptimizer.cpp:1346-1351 (float32 arithmetic)
    import numpy as np
    gx = 10
    inv_aspect = np.float32(1.0) / np.float32(aspect)
    gy = int(np.floor(float(np.float32(gx) * inv_aspect) + 0.5))  # std::round, half away from zero
    if aspect <= 1.0:
        gx, gy = gy, gx
    cfg.scale_grid_x, cfg.scale_grid_y = gx, gy
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg
