"""Python binding (ctypes) of the C ABI in include/rcvd.h -- the B200 solver.

`Problem` is the array-level equivalent of the reference's
DepthVideoPoseOptimizer::poseOptimizationStep / normalizeDepth
(lib/PoseOptimizer.cpp:890-990, :992-1147): one non-linear least-squares
problem over per-frame [pose(6), focal, depth-transform params, spatial params].

There is no CPU fallback: if librcvd_b200.so is missing or no CUDA device is
usable, construction raises RuntimeError.
"""
import ctypes as C
import os
import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "librcvd_b200.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(the CUDA extension is mandatory, there is no CPU fallback)")
        L = C.CDLL(path)
        L.rcvd_last_error.restype = C.c_char_p
        L.rcvd_launch_count.restype = C.c_int64
        L.rcvd_problem_create.argtypes = [C.POINTER(abi.Config), C.c_int32, C.POINTER(C.c_void_p)]
        L.rcvd_problem_destroy.argtypes = [C.c_void_p]
        for name in ("rcvd_frame_stride", "rcvd_depth_param_offset", "rcvd_spatial_param_offset"):
            getattr(L, name).argtypes = [C.POINTER(abi.Config)]
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def _check(rc):
    if rc != 0:
        raise RuntimeError(f"rcvd error {rc}: {lib().rcvd_last_error().decode()}")


def frame_stride(cfg):
    return lib().rcvd_frame_stride(C.byref(cfg))


def depth_param_offset(cfg):
    return lib().rcvd_depth_param_offset(C.byref(cfg))


def spatial_param_offset(cfg):
    return lib().rcvd_spatial_param_offset(C.byref(cfg))


class Problem:
    def __init__(self, cfg, device=0):
        self.cfg = cfg
        self.L = lib()
        self.h = C.c_void_p()
        _check(self.L.rcvd_problem_create(C.byref(cfg), C.c_int32(device), C.byref(self.h)))
        self.N = cfg.num_frames
        self.stride = frame_stride(cfg)
        self.U = self.N * self.stride
        self.num_constraints = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.rcvd_problem_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frames(self, in_range=None, median_depth=None, adaptive_weights=None):
        ir = None if in_range is None else np.ascontiguousarray(in_range, np.uint8)
        md = None if median_depth is None else np.ascontiguousarray(median_depth, np.float64)
        aw = None if adaptive_weights is None else np.ascontiguousarray(adaptive_weights, np.float64)
        _check(self.L.rcvd_problem_set_frames(self.h, _p(ir, C.c_uint8), _p(md, C.c_double), _p(aw, C.c_double)))

    def set_constraints(self, pair_frames, offsets, records):
        pf = np.ascontiguousarray(pair_frames, np.int32).reshape(-1, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        rec = np.ascontiguousarray(records, np.float32).reshape(-1, 6)
        assert off.shape[0] == pf.shape[0] + 1 and off[-1] == rec.shape[0]
        self.num_constraints = int(rec.shape[0])
        _check(self.L.rcvd_problem_set_constraints(self.h, C.c_int32(pf.shape[0]), _p(pf, C.c_int32), _p(off, C.c_int64), _p(rec, C.c_float)))

    def set_triplets(self, centers, offsets, records):
        """Scene-flow smoothness constraints (addSceneFlowSmoothnessLoss): centers[T], offsets[T+1], records[n][10]."""
        ce = np.ascontiguousarray(centers, np.int32); off = np.ascontiguousarray(offsets, np.int64)
        rec = np.ascontiguousarray(records, np.float32).reshape(-1, 10)
        assert off.shape[0] == ce.shape[0] + 1 and off[-1] == rec.shape[0]
        _check(self.L.rcvd_problem_set_triplets(self.h, C.c_int32(ce.shape[0]), _p(ce, C.c_int32), _p(off, C.c_int64), _p(rec, C.c_float)))

    def set_structure(self, pair_frames):
        pf = np.ascontiguousarray(pair_frames, np.int32).reshape(-1, 2)
        _check(self.L.rcvd_problem_set_structure(self.h, C.c_int32(pf.shape[0]), _p(pf, C.c_int32)))

    def init_comm(self, nranks, rank, unique_id):
        uid = np.ascontiguousarray(unique_id, np.uint8)
        assert uid.size == 128
        _check(self.L.rcvd_problem_init_comm(self.h, C.c_int32(nranks), C.c_int32(rank), _p(uid, C.c_uint8)))

    def set_state(self, x):
        x = np.ascontiguousarray(x, np.float64).reshape(-1)
        assert x.size == self.U
        _check(self.L.rcvd_problem_set_state(self.h, _p(x, C.c_double)))

    def get_state(self):
        x = np.empty(self.U, np.float64)
        _check(self.L.rcvd_problem_get_state(self.h, _p(x, C.c_double)))
        return x.reshape(self.N, self.stride)

    def evaluate(self, gradient=False):
        cost = C.c_double()
        g = np.zeros(self.U, np.float64) if gradient else None
        _check(self.L.rcvd_evaluate(self.h, C.byref(cost), _p(g, C.c_double)))
        return (cost.value, g) if gradient else cost.value

    def normal_matrix_dense(self):
        H = np.zeros((self.U, self.U), np.float64)
        _check(self.L.rcvd_normal_matrix_dense(self.h, _p(H, C.c_double)))
        return H

    def debug_linear_solve(self, S, D2, b):
        S = np.ascontiguousarray(S, np.float64); D2 = np.ascontiguousarray(D2, np.float64)
        b = np.ascontiguousarray(b, np.float64); y = np.zeros_like(b)
        _check(self.L.rcvd_debug_linear_solve(self.h, _p(S, C.c_double), _p(D2, C.c_double), _p(b, C.c_double), _p(y, C.c_double)))
        return y

    def solve(self, options=None):
        opt = options or abi.default_solve_options()
        s = abi.SolveSummary()
        _check(self.L.rcvd_solve(self.h, C.byref(opt), C.byref(s)))
        return s

    def time_accumulate(self, iters=10):
        ms = C.c_double()
        _check(self.L.rcvd_time_accumulate(self.h, C.c_int32(iters), C.byref(ms)))
        return ms.value

    def time_iteration(self, iters=5, radius=1e4):
        a, b, c, d = C.c_double(), C.c_double(), C.c_double(), C.c_double()
        _check(self.L.rcvd_time_iteration(self.h, C.c_int32(iters), C.c_double(radius), C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"iter_ms": a.value, "accumulate_ms": b.value, "linear_ms": c.value, "cost_ms": d.value}

    def iteration_outputs(self):
        """Bench hook: gradient, LM step and candidate state ([N, stride] each) and {cost, candidate cost} of the last
        time_iteration step."""
        g, step, xc = (np.empty((self.N, self.stride), np.float64) for _ in range(3))
        costs = np.empty(2, np.float64)
        _check(self.L.rcvd_debug_iteration_outputs(self.h, _p(g, C.c_double), _p(step, C.c_double), _p(xc, C.c_double), _p(costs, C.c_double)))
        return {"gradient": g, "step": step, "candidate_state": xc, "costs": costs}

    def structure_info(self):
        out = (C.c_int32 * 8)()
        _check(self.L.rcvd_structure_info(self.h, out))
        keys = ["frames", "offdiag_factor_blocks", "levels", "h_blocks", "npad", "stride", "tiles", "update_tasks"]
        return dict(zip(keys, list(out)))

    def linear_residual(self, radius=1e4):
        """Bench / test hook: one damped LM step at the current state; device-side residual of the linear system and checksums."""
        out = (C.c_double * 6)()
        _check(self.L.rcvd_debug_linear_residual(self.h, C.c_double(radius), out))
        keys = ["rel_residual", "rhs_norm", "cost", "grad_norm", "step_norm", "pivot_fail"]
        return dict(zip(keys, list(out)))

    def profile_linear(self, reps=3):
        """Bench hook: per-kernel-class device time of one factorisation + solve (serialised on one stream, CUDA events per launch)."""
        out = (C.c_double * 8)()
        _check(self.L.rcvd_debug_profile_linear(self.h, C.c_int32(reps), out))
        keys = ["load_ms", "potrf_ms", "trinv_ms", "trsm_ms", "gemm_ms", "solve_ms", "gemm_launches", "gemm_flops"]
        return dict(zip(keys, list(out)))

    def set_fast_path(self, on=True):
        """Test hook: False / 0 forces the generic accumulate kernel, 2 the round-1 specialised kernel without the run path."""
        _check(self.L.rcvd_debug_set_fast_path(self.h, C.c_int32(int(on))))

    def set_update_kernel(self, tma=True, side_items_per_cta=0):
        """Test / bench hook: persistent TMA-fed update kernel (default) or the round-1 cp.async kernel."""
        _check(self.L.rcvd_debug_set_update_kernel(self.h, C.c_int32(1 if tma else 0), C.c_int32(side_items_per_cta)))

    def set_eval_only(self, on=True):
        """Test / bench hook: the handle only evaluates cost / gradient; no matrix storage is allocated."""
        _check(self.L.rcvd_debug_set_eval_only(self.h, C.c_int32(1 if on else 0)))

    def set_distributed(self, on=True):
        """Test / bench hook (nranks > 1): distributed factorisation (default) or the round-1 replicated scheme."""
        _check(self.L.rcvd_debug_set_distributed(self.h, C.c_int32(1 if on else 0)))

    def distribution_info(self):
        out = (C.c_int32 * 4)()
        _check(self.L.rcvd_distribution_info(self.h, out))
        return dict(zip(["distributed", "first_replicated_level", "levels", "frames_owned"], list(out)))

    def set_side_slice(self, ctas):
        _check(self.L.rcvd_debug_set_side_slice(self.h, C.c_int32(ctas)))

    def set_trim_gemm(self, on=True):
        _check(self.L.rcvd_debug_set_trim_gemm(self.h, C.c_int32(1 if on else 0)))

    def set_fused_substitution(self, on=True):
        _check(self.L.rcvd_debug_set_fused_substitution(self.h, C.c_int32(int(on))))

    def set_trsm_ll(self, on=True):
        _check(self.L.rcvd_debug_set_trsm_ll(self.h, C.c_int32(1 if on else 0)))

    def set_order_slack(self, slack):
        _check(self.L.rcvd_debug_set_order_slack(self.h, C.c_int32(slack)))

    def set_overlap(self, on=True):
        _check(self.L.rcvd_debug_set_overlap(self.h, C.c_int32(1 if on else 0)))

    def launch_count(self):
        return int(self.L.rcvd_launch_count(self.h))


def nccl_unique_id():
    out = np.zeros(128, np.uint8)
    _check(lib().rcvd_nccl_unique_id(_p(out, C.c_uint8)))
    return out


def depth_apply(cfg, depth_params, src, device=0):
    """DepthXform::apply (reference lib/DepthMapTransform.cpp:394-415) on the GPU."""
    src = np.ascontiguousarray(src, np.float32); h, w = src.shape
    dp = np.ascontiguousarray(depth_params, np.float64); dst = np.empty_like(src)
    _check(lib().rcvd_depth_apply(C.byref(cfg), C.c_int32(device), _p(dp, C.c_double), _p(src, C.c_float), _p(dst, C.c_float), C.c_int32(h), C.c_int32(w)))
    return dst


def depth_param_map(cfg, depth_params, h, w, device=0):
    """GridDepthXform::paramMap (reference lib/DepthMapTransform.cpp:950-994) on the GPU."""
    k = 2 if cfg.value_xform == abi.VALUE_SCALESHIFT else 1
    dp = np.ascontiguousarray(depth_params, np.float64); out = np.empty((h, w, k), np.float64)
    _check(lib().rcvd_depth_param_map(C.byref(cfg), C.c_int32(device), _p(dp, C.c_double), _p(out, C.c_double), C.c_int32(h), C.c_int32(w)))
    return out[:, :, 0] if k == 1 else out


def spatial_warp(cfg, spatial_params, h, w, device=0):
    """SpatialXform::warp (reference lib/DepthMapTransform.cpp:428-449) on the GPU."""
    sp = np.ascontiguousarray(spatial_params, np.float64); out = np.empty((h, w, 2), np.float32)
    _check(lib().rcvd_spatial_warp(C.byref(cfg), C.c_int32(device), _p(sp, C.c_double), _p(out, C.c_float), C.c_int32(h), C.c_int32(w)))
    return out


def flow_guided_filter(depth, cams, fwd_flow, fwd_mask, bwd_flow, bwd_mask, first_out, num_out, frame_radius, spatial_radius=0, median=False,
                       inv_aspect=1.0, far_pairs=None, far_flow=None, far_mask=None, device=0):
    """rcvd_flow_guided_filter (DepthVideoProcessor::flowGuidedFilter, reference lib/Processor.cpp:315-590) on the GPU.
    depth [F,hd,wd] f32, cams [F,9] f32, flows [F,h,w,2] f32, masks [F,h,w] u8 -> filtered depth [num_out,h,w] f32."""
    depth = np.ascontiguousarray(depth, np.float32); cams = np.ascontiguousarray(cams, np.float32)
    F, hd, wd = depth.shape
    arrs = []
    for a, dt in ((fwd_flow, np.float32), (fwd_mask, np.uint8), (bwd_flow, np.float32), (bwd_mask, np.uint8), (far_flow, np.float32), (far_mask, np.uint8)):
        arrs.append(None if a is None else np.ascontiguousarray(a, dt))
    ff, fm, bf, bm, rf, rm = arrs
    ref_mask = fm if fm is not None else rm
    if ref_mask is None:
        raise ValueError("flow masks are needed to define the output resolution")
    h, w = ref_mask.shape[1:3]
    nfar = 0 if far_pairs is None else len(far_pairs)
    fp = None if nfar == 0 else np.ascontiguousarray(far_pairs, np.int32).reshape(-1, 2)
    prm = abi.FilterParams(num_frames=F, first_out=first_out, num_out=num_out, width=w, height=h, depth_width=wd, depth_height=hd,
                           frame_radius=frame_radius, spatial_radius=spatial_radius, median=1 if median else 0, num_far=nfar, inv_aspect=inv_aspect)
    out = np.zeros((num_out, h, w), np.float32)
    _check(lib().rcvd_flow_guided_filter(C.byref(prm), C.c_int32(device), _p(depth, C.c_float), _p(cams, C.c_float),
                                         _p(ff, C.c_float), _p(fm, C.c_uint8), _p(bf, C.c_float), _p(bm, C.c_uint8),
                                         _p(fp, C.c_int32), _p(rf, C.c_float), _p(rm, C.c_uint8), _p(out, C.c_float)))
    return out


def bilateral_filter(depth, out_frames, frame_radius=2, spatial_radius=0, depth_sigma=0.3, color_sigma=0.0, median=False, color=None,
                     in_place=False, xform_cfg=None, xform_params=None, device=0):
    """rcvd_bilateral_filter (DepthVideoProcessor::bilateralFilter, reference lib/Processor.cpp:183-313) on the GPU.
    depth [F,h,w] f32 (transformed depth of stream 0), color [F,h,w,3] f32 or None, out_frames ascending frame indices
    -> filtered depth [len(out_frames),h,w] f32.  in_place: each filtered frame replaces its depth, with the transform
    (xform_cfg, xform_params [len(out_frames), depth params]) applied again, before later windows read it."""
    depth = np.ascontiguousarray(depth, np.float32); F, h, w = depth.shape
    col = None if color is None else np.ascontiguousarray(color, np.float32)
    of = np.ascontiguousarray(out_frames, np.int32).reshape(-1)
    xp = None if xform_params is None else np.ascontiguousarray(xform_params, np.float64)
    if xp is not None and xp.size == 0:
        xp = np.zeros(1, np.float64)        # a transform without parameters (identity)
    prm = abi.BilateralParams(num_frames=F, num_out=len(of), width=w, height=h, spatial_radius=spatial_radius, frame_radius=frame_radius,
                              median=1 if median else 0, in_place=1 if in_place else 0, depth_sigma=depth_sigma, color_sigma=color_sigma)
    out = np.zeros((len(of), h, w), np.float32)
    _check(lib().rcvd_bilateral_filter(C.byref(prm), C.c_int32(device), _p(depth, C.c_float), _p(col, C.c_float), _p(of, C.c_int32),
                                       C.byref(xform_cfg) if xform_cfg is not None else None, _p(xp, C.c_double), _p(out, C.c_float)))
    return out


def build_constraints(color_bgr, pair_frames, pair_flow, pair_mask, match_separation, inv_aspect, dyn_dist=None, min_dynamic_distance=-1.0,
                      trip_frames=None, trip_flow=None, trip_mask=None, device=0):
    """rcvd_build_constraints (FlowConstraintsCollection::compute + sampleConstraints, reference lib/FlowConstraints.cpp:352-550) on the GPU.
    Returns (pair_offsets, pair_constraints [n,4], trip_offsets, trip_constraints [m,6])."""
    color = np.ascontiguousarray(color_bgr, np.float32)
    F, h, w = color.shape[:3]
    pf = np.ascontiguousarray(pair_frames, np.int32).reshape(-1, 2); P = len(pf)
    pfl = np.ascontiguousarray(pair_flow, np.float32) if P else None; pm = np.ascontiguousarray(pair_mask, np.uint8) if P else None
    T = 0 if trip_frames is None else len(trip_frames)
    tf = np.ascontiguousarray(trip_frames, np.int32) if T else None
    tfl = np.ascontiguousarray(trip_flow, np.float32) if T else None; tm = np.ascontiguousarray(trip_mask, np.uint8) if T else None
    dd = None if dyn_dist is None else np.ascontiguousarray(dyn_dist, np.float32)
    prm = abi.BuilderParams(num_frames=F, width=w, height=h, dyn_width=0 if dd is None else dd.shape[2], dyn_height=0 if dd is None else dd.shape[1],
                            match_separation=match_separation, num_pairs=P, num_triplets=T, min_dynamic_distance=min_dynamic_distance, inv_aspect=inv_aspect)
    poff = np.zeros(P + 1, np.int64); toff = np.zeros(T + 1, np.int64)
    pcap, tcap = 0, 0
    for attempt in range(2):
        pout = np.zeros((max(pcap, 1), 4), np.float32); tout = np.zeros((max(tcap, 1), 6), np.float32)
        rc = lib().rcvd_build_constraints(C.byref(prm), C.c_int32(device), _p(color, C.c_float), _p(dd, C.c_float), _p(pf if P else None, C.c_int32), _p(pfl, C.c_float), _p(pm, C.c_uint8),
                                          _p(tf, C.c_int32), _p(tfl, C.c_float), _p(tm, C.c_uint8), _p(poff, C.c_int64), _p(pout, C.c_float), C.c_int64(pcap),
                                          _p(toff, C.c_int64), _p(tout, C.c_float), C.c_int64(tcap))
        if rc == 0:
            break
        if attempt == 0 and (poff[P] > pcap or toff[T] > tcap):
            pcap, tcap = int(poff[P]), int(toff[T])      # the first call reports the sizes
            continue
        _check(rc)
    return poff, pout[:poff[P]], toff, tout[:toff[T]]


def static_flags(masks, distance, pair_frames=None, pair_offsets=None, pair_locs=None, trip_frames=None, trip_offsets=None, trip_locs=None, want_distance=False, device=0):
    """rcvd_static_flags (FlowConstraintsCollection::setStaticFlagFromDynamicMask + dynamicDistance, reference lib/FlowConstraints.cpp:573-660,
    :257-286) on the GPU.  masks [F,h,w] u8.  Returns (pair_static u8[n], trip_static u8[m], distance images [F,h,w] f32 or None)."""
    m = np.ascontiguousarray(masks, np.uint8); F, h, w = m.shape
    P = 0 if pair_frames is None else len(pair_frames); T = 0 if trip_frames is None else len(trip_frames)
    pf = np.ascontiguousarray(pair_frames, np.int32).reshape(-1, 2) if P else None
    po = np.ascontiguousarray(pair_offsets, np.int64) if P else None
    pl = np.ascontiguousarray(pair_locs, np.float32).reshape(-1, 4) if P else None
    tf = np.ascontiguousarray(trip_frames, np.int32) if T else None
    to = np.ascontiguousarray(trip_offsets, np.int64) if T else None
    tl = np.ascontiguousarray(trip_locs, np.float32).reshape(-1, 6) if T else None
    ps = np.zeros(int(po[-1]) if P else 0, np.uint8); ts = np.zeros(int(to[-1]) if T else 0, np.uint8)
    dist = np.zeros((F, h, w), np.float32) if want_distance else None
    _check(lib().rcvd_static_flags(C.c_int32(device), _p(m, C.c_uint8), C.c_int32(F), C.c_int32(h), C.c_int32(w), C.c_float(distance),
                                   C.c_int32(P), _p(pf, C.c_int32), _p(po, C.c_int64), _p(pl, C.c_float), _p(ps if P else None, C.c_uint8),
                                   C.c_int32(T), _p(tf, C.c_int32), _p(to, C.c_int64), _p(tl, C.c_float), _p(ts if T else None, C.c_uint8), _p(dist, C.c_float)))
    return ps, ts, dist


def fp64_tensor_peak(device=0):
    """Bench hook: live-measured fp64 tensor-core (DMMA) peak of `device` in TFLOP/s."""
    v = C.c_double()
    _check(lib().rcvd_debug_fp64_tensor_peak(C.c_int32(device), C.byref(v)))
    return v.value
