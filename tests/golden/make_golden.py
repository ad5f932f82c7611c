"""Generates the committed golden fixtures: `python tests/golden/make_golden.py <robust_cvd checkout>` (the reference's
pure-Python pieces are imported from that checkout; the solver goldens come from the CPU oracle because the reference's
C++ path cannot be built without its dependencies -- see DESIGN.md "Oracle")."""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REFERENCE = None          # path of a robust_cvd checkout (command line)


def golden_pairs():
    sys.path.insert(0, REFERENCE)
    from utils import frame_sampling as fs
    from utils.frame_range import FrameRange, OptionalSet
    out = {}
    for n in (2, 3, 8, 17, 64, 300):
        fr = FrameRange(frame_range=OptionalSet(), num_frames=n)
        pairs = fs.SamplePairs.sample([fs.SamplePairsOptions(mode=fs.SamplePairsMode.HIERARCHICAL2)], frame_range=fr, two_way=True)
        out[str(n)] = [[int(p[0]), int(p[1])] for p in pairs]
    json.dump(out, open(os.path.join(HERE, "hierarchical2_pairs.json"), "w"))


def golden_solver():
    from robust_cvd_b200 import abi
    from oracle import oracle
    from tests import helpers
    out = {}
    for name in ("bilinear_perframe_disp", "bicubic_shared_ratio_bicubicwarp", "global_fixed_log_bilinearwarp"):
        ov = dict(helpers.VARIANTS)[name]
        sc, cfg, pairs, offs, rec, med = helpers.make_case(**ov)
        off_d, nd = helpers.layout_numbers(cfg)
        O = oracle.OracleProblem(cfg)
        x = helpers.initial_state(sc, cfg, O.stride, off_d, nd)
        helpers.setup_problem(O, cfg, pairs, offs, rec, med, x)
        cost, g = O.evaluate(True)
        Hd = np.diag(O.normal_matrix_dense()).copy()
        s = O.solve(abi.default_solve_options(max_iterations=60))
        out[name + "/x0"] = x; out[name + "/cost"] = np.array(cost); out[name + "/grad"] = g; out[name + "/hdiag"] = Hd
        out[name + "/final_cost"] = np.array(s.final_cost); out[name + "/iterations"] = np.array(s.iterations); out[name + "/x_final"] = O.get_state()
    np.savez_compressed(os.path.join(HERE, "oracle_solver_golden.npz"), **out)


def golden_raw_images():
    """.raw wire format: files written by the reference's own utils/image_io.py::save_raw_float32_image (imported unchanged)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_image_io", os.path.join(REFERENCE, "utils", "image_io.py"))
    io = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(io)
    except Exception:      # the module imports cv2 / other helpers at the top; only the two raw functions are needed
        src = open(os.path.join(REFERENCE, "utils", "image_io.py")).read()
        a = src.index("def load_raw_float32_image"); b = src.index("def save_raw_float32_image")
        end = src.find("\ndef ", b + 10)
        ns = {"np": np, "struct": __import__("struct")}
        exec(compile(src[a:end if end > 0 else len(src)], os.path.join(REFERENCE, "utils", "image_io.py"), "exec"), ns)      # executed in place, not copied
        io = type("io", (), {k: staticmethod(v) for k, v in ns.items() if callable(v)})
    rng = np.random.default_rng(4)
    disp = (rng.random((5, 7)) * 2 + 0.1).astype(np.float32); disp[1, 2] = 0.0; disp[3, 3] = np.inf
    flow = rng.normal(0, 1.5, (5, 7, 2)).astype(np.float32)
    color = rng.random((5, 7, 3)).astype(np.float32)
    io.save_raw_float32_image(os.path.join(HERE, "ref_writer_disparity_5x7.raw"), disp)
    io.save_raw_float32_image(os.path.join(HERE, "ref_writer_flow_5x7x2.raw"), flow)
    io.save_raw_float32_image(os.path.join(HERE, "ref_writer_color_5x7x3.raw"), color)
    np.savez_compressed(os.path.join(HERE, "ref_writer_arrays.npz"), disp=disp, flow=flow, color=color)


def golden_host_restatements():
    """Outputs of the float32 restatements of the post-filter and the disc sampler (oracle/host_ref.py) on fixed inputs:
    pins the restatements against silent edits (the reference's C++ for these cannot be built here)."""
    from oracle import host_ref
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from tests.test_gpu_filter import make_filter_case
    case, far_pairs, ff, fm = make_filter_case(F=5, w=20, h=12, seed=9, far=((2, 0), (2, 4)))
    out = {}
    for name, kw in (("mean_r0", dict(spatial_radius=0, median=False)), ("median_r1_far", dict(spatial_radius=1, median=True, far_pairs=far_pairs, far_flow=ff, far_mask=fm))):
        out["filter_" + name] = host_ref.flow_guided_filter(**case, first_out=1, num_out=3, frame_radius=2, **kw)
    rng = np.random.default_rng(12)
    iy, ix = np.mgrid[0:24, 0:32]
    color = (np.sin(ix * 0.9)[..., None] * np.cos(iy * 0.7)[..., None] * 0.4 + 0.5 + rng.normal(0, 0.08, (24, 32, 3))).astype(np.float32)
    flow = rng.normal(0, 2.0, (24, 32, 2)).astype(np.float32); mask = (rng.random((24, 32)) > 0.1).astype(np.uint8) * 255
    for sep in (1, 4):
        c, score = host_ref.pair_constraints(color, flow, mask, sep, np.float32(0.75))
        out[f"sampler_sep{sep}"] = c
    out["sampler_color"] = color; out["sampler_flow"] = flow; out["sampler_mask"] = mask; out["sampler_score"] = score
    np.savez_compressed(os.path.join(HERE, "host_restatement_golden.npz"), **out)


def golden_geometry():
    """Reprojection vectors from the reference's OWN camera model in Python (utils/geometry.py, imported unchanged) with
    intrinsics / extrinsics assembled exactly like loaders/video_dataset.py:177-189 does from the C++ pose state:
    extrinsics = [right, up, backward | position], fx = (W/2)/tan(hFov/2), fy = (H/2)/tan(vFov/2), c = (W/2, H/2).
    The fine-tuning loss consumes the poses the C++ optimiser produced with this model, so StaticSceneCost's geometry
    (sign conventions, NDC mapping, aspect handling, focal definition) must reproduce it: tests/test_oracle.py checks that the
    oracle's residuals vanish on these correspondences."""
    sys.path.insert(0, REFERENCE)
    import torch
    from utils import geometry as G
    from robust_cvd_b200.synthetic import rodrigues
    rng = np.random.default_rng(21)
    W, H, K = 64, 48, 160
    aspect = np.float32(W) / np.float32(H)
    out = {"W": np.array(W), "H": np.array(H)}
    aa = rng.normal(0, 0.15, (2, 3)); t = rng.normal(0, 0.3, (2, 3)); phi = np.array([0.26, 0.31])       # tan(vFov/2) per frame
    extr = np.zeros((2, 3, 4)); intr = np.zeros((2, 4))
    for f in range(2):
        extr[f, :, :3] = rodrigues(aa[f]); extr[f, :, 3] = t[f]                                             # columns right, up, backward
        intr[f] = [(W / 2.0) / (phi[f] * float(aspect)), (H / 2.0) / phi[f], W / 2.0, H / 2.0]
    px = rng.integers(0, W, K).astype(np.float64); py = rng.integers(0, H, K).astype(np.float64); depth = rng.uniform(1.0, 4.0, K)
    pixels = torch.tensor(np.stack([px, py])[None, :, None, :]); depths = torch.tensor(depth[None, None, None, :])
    E = torch.tensor(extr); I = torch.tensor(intr)
    pc0 = G.pixels_to_points(I[0:1], depths, pixels.clone())
    pc1 = G.reproject_points(pc0, E[0:1], E[1:2])
    pix1 = G.project(pc1.clone(), I[1:2])
    out.update(angle_axis=aa, position=t, tan_half_vfov=phi, px0=px, py0=py, depth0=depth,
               px1=pix1[0, 0, 0].numpy(), py1=pix1[0, 1, 0].numpy(), depth1=(-pc1[0, 2, 0]).numpy(),
               world=G.points_cam_to_world(pc0, E[0:1])[0, :, 0].numpy().T)
    np.savez_compressed(os.path.join(HERE, "ref_python_geometry.npz"), **out)


def golden_pose_optimization_trace():
    """Every lib_python attribute read, call and assignment that the reference's own pose_optimization.py (imported unchanged)
    makes in PoseOptimizer(...) and optimize_poses() on the 8-frame scene of tests/test_host.py, with what each returned, recorded
    on a machine without a GPU: optimize_poses() ends with the call that refuses to run without one.  Objects are numbered in
    order of appearance (0 = the module), paths inside the scene directory are written relative to "{root}".
    tests/test_host.py replays the sequence against lib_python."""
    import importlib
    import shutil
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "robust_cvd_b200", "host"))
    import lib_python
    from tests.test_host import write_scene8
    root = tempfile.mkdtemp(prefix="rcvd_trace_")
    write_scene8(root)
    trace = {"init": [], "optimize_poses": []}
    phase = ["init"]
    primitive = (bool, int, float, str, type(None))

    def enc(v):
        if isinstance(v, Recorder):
            return {"ref": object.__getattribute__(v, "_id")}
        if isinstance(v, (list, tuple)):
            return [enc(x) for x in v]
        assert isinstance(v, primitive), type(v)
        return v.replace(root, "{root}") if isinstance(v, str) else v

    def raw(v):
        if isinstance(v, Recorder):
            return object.__getattribute__(v, "_obj")
        return [raw(x) for x in v] if isinstance(v, list) else v

    def result(op, v):
        trace[phase[0]].append(op)
        if isinstance(v, primitive) or (isinstance(v, (list, tuple)) and all(isinstance(x, primitive) for x in v)):
            op["out"] = enc(v)
            return v
        r = Recorder(v)
        op["out"] = enc(r)
        return r

    class Recorder:
        count = [0]

        def __init__(self, obj):
            object.__setattr__(self, "_obj", obj)
            object.__setattr__(self, "_id", Recorder.count[0])
            Recorder.count[0] += 1

        def __getattr__(self, name):
            v = getattr(object.__getattribute__(self, "_obj"), name)
            if name.startswith("__"):          # import machinery
                return v
            return result({"op": "get", "obj": object.__getattribute__(self, "_id"), "name": name}, v)

        def __setattr__(self, name, value):
            trace[phase[0]].append({"op": "set", "obj": object.__getattribute__(self, "_id"), "name": name, "value": enc(value)})
            setattr(object.__getattribute__(self, "_obj"), name, raw(value))

        def __call__(self, *args, **kwargs):
            assert not kwargs
            op = {"op": "call", "obj": object.__getattribute__(self, "_id"), "args": enc(list(args))}
            try:
                v = object.__getattribute__(self, "_obj")(*[raw(a) for a in args])
            except Exception as e:
                op["raises"] = {"type": type(e).__name__, "message": str(e)}
                trace[phase[0]].append(op)
                raise
            return result(op, v)

    dflt = lib_python.DepthVideoPoseOptimizer.Params()
    sys.modules["lib_python"] = Recorder(lib_python)
    sys.path.insert(0, REFERENCE)
    try:
        po = importlib.import_module("pose_optimization")
        from utils.helpers import Nestedspace
        o = Nestedspace()
        for k, v in dict(max_iterations=50, num_threads=12, num_steps=4, robustness=0.5, static_loss_type="ReproDisparity", static_spatial_weight=1.0,
                         static_depth_weight=1.0, smooth_loss_type="ReproDisparityLaplacian", smooth_static_weight=0.0, smooth_dynamic_weight=0.0,
                         position_regularization=0.0, scale_regularization=1.0, scale_regularization_grid_size=10, deformation_regularization_initial=1.0,
                         deformation_regularization_final=0.1, adaptive_deformation_cost=0.0, spatial_deformation_regularization=1.0,
                         graduate_deformation_regularization=False, focal_regularization=1.0, coarse_to_fine=True, ctf_long=dflt.ctfLong, ctf_short=dflt.ctfShort,
                         deferred_spatial_opt=False, dso_long=4, dso_short=3, focal_long=dflt.focalLong, intr_opt="PerFrame", fix_poses=False,
                         fix_depth_transforms=False, fix_spatial_transforms=False, use_global_scale=False, dynamic_constraints="Mask").items():
            setattr(o, k, v)
        os.environ["RCVD_CONSTRAINT_BUILDER"] = "host"          # as in tests/test_host.py
        opt = po.PoseOptimizer(root, "midas2", list(range(8)), o)
        phase[0] = "optimize_poses"
        try:
            opt.optimize_poses()
            raise AssertionError("optimize_poses() ran: record the trace on a machine without a GPU")
        except RuntimeError:
            pass
    finally:
        sys.modules["lib_python"] = lib_python
        shutil.rmtree(root, ignore_errors=True)
    with open(os.path.join(HERE, "ref_pose_optimization_trace.json"), "w") as f:       # one operation per line
        f.write("{\n" + ",\n".join(f'"{k}": [\n' + ",\n".join(json.dumps(op) for op in ops) + "\n]" for k, ops in trace.items()) + "\n}\n")


if __name__ == "__main__":
    REFERENCE = sys.argv[1]
    golden_geometry()
    golden_pairs()
    golden_solver()
    golden_raw_images()
    golden_host_restatements()
    golden_pose_optimization_trace()
    print("golden fixtures written")
