"""Host-side (lib_python) logic on CPU: wire formats, constraint generation against the numpy/cv2
restatement, problem assembly arrays, pose conversions, coarse-to-fine split -- everything of the
drop-in boundary that does not need the GPU."""
import os
import re
import shutil
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "robust_cvd_b200", "host"))

lp = pytest.importorskip("lib_python")
from robust_cvd_b200 import abi, synthetic, synthetic_files  # noqa: E402
from oracle import host_ref  # noqa: E402

CV_32FC3, CV_8UC1 = 21, 0


@pytest.fixture(autouse=True)
def _host_constraint_builder(monkeypatch):
    """These tests run without a GPU: select the sequential host builder explicitly (the default is the GPU builder,
    tests/test_gpu_builder.py checks that both produce identical lists)."""
    monkeypatch.setenv("RCVD_CONSTRAINT_BUILDER", "host")


def write_scene8(root):
    sc = synthetic.Scene(8, 128, 96, seed=3)
    rng = np.random.default_rng(5)
    masks = []
    for i in range(sc.N):           # a dynamic blob (0 = dynamic, 255 = static) so that the static flag matters
        m = np.full((96, 128), 255, np.uint8); cx, cy = rng.integers(30, 100), rng.integers(30, 70); m[cy - 8:cy + 8, cx - 10:cx + 10] = 0; masks.append(m)
    pairs = synthetic_files.write_scene(sc, root, dynamic_masks=masks)
    return sc, root, pairs, masks


@pytest.fixture(scope="module")
def scene_dir(tmp_path_factory):
    return write_scene8(str(tmp_path_factory.mktemp("scene8")))


def _open(root):
    v = lp.DepthVideo()
    lp.DepthVideoImporter.importVideo(v, root, False)
    v.createColorStream("full", "color_full", ".png", CV_32FC3)
    v.createColorStream("down", "color_down", ".raw", CV_32FC3)
    v.createColorStream("dynamic_mask", "dynamic_mask", ".png", CV_8UC1)
    v.createDepthStream("depth_midas2", "depth_midas2", [-1, -1])
    return v


def test_video_and_streams(scene_dir):
    sc, root, pairs, masks = scene_dir
    v = _open(root)
    assert (v.numFrames(), v.width(), v.height()) == (8, 128, 96)
    assert v.aspect() == np.float32(128) / np.float32(96) and v.invAspect() == np.float32(1) / v.aspect()
    ds = v.depthStream(v.numDepthStreams() - 1)
    assert ds.depthXformDesc().str() == "Identity()" and ds.spatialXformDesc().str() == "Identity"
    f = ds.frame(0)
    np.testing.assert_array_equal(f.extrinsics.position, np.zeros(3, np.float32))
    assert (f.extrinsics.orientation.w(), f.extrinsics.orientation.x()) == (1.0, 0.0)
    assert abs(f.intrinsics.vFov - 0.666488587) < 1e-7 and f.intrinsics.hFov > f.intrinsics.vFov   # resolveMissingFov, landscape
    src = f.sourceDepth()
    disp = synthetic_files.read_raw(f"{root}/depth_midas2/depth/frame_000000.raw")
    np.testing.assert_array_equal(src, np.float32(1.0) / disp)
    assert (ds.width(), ds.height()) == (128, 96)
    np.testing.assert_array_equal(v.colorStream("dynamic_mask").frame(2).image(), masks[2])
    v.save()
    raw = open(f"{root}/video.dat", "rb").read()
    assert struct.unpack("<III", raw[:12]) == (0xDEADBEEF, 13, 3) and struct.unpack("<I", raw[-4:])[0] == 0xDEADBEEF
    with pytest.raises(RuntimeError):
        lp.DepthVideoImporter.importVideo(lp.DepthVideo(), root + "/nope", False)


def test_video_dat_round_trip_and_processor_defaults(scene_dir, tmp_path):
    """video.dat written by save() (byte layout of lib/DepthVideo.cpp:300-385) is read back by load(); setDepth replaces
    the source depth; DepthVideoProcessor.Params defaults are the reference's (lib/Processor.h:60-80)."""
    sc, root, pairs, masks = scene_dir
    root2 = str(tmp_path / "copy"); shutil.copytree(root, root2)
    v = _open(root2)
    ds = v.depthStream(0)
    rp = lp.DepthVideoProcessor.Params(); rp.depthStream = 0; rp.depthXformDesc.parse("Grid(Scale, Linear, 4, 3, 1)")
    lp.DepthVideoProcessor(v).resetDepthXforms(rp)
    for f in range(8):
        df = ds.frame(f); e = df.extrinsics; e.position = np.array([f, -f, 0.5 * f], np.float32); e.orientation = lp._makeQuat(0.0, np.sin(0.1 * f), 0.0, np.cos(0.1 * f)); df.extrinsics = e
        df.depthXform().params()[:] = list(1.0 + 0.01 * f + 0.001 * np.arange(12))
    v.save()
    v2 = lp.DepthVideo(); v2.load(root2)
    assert (v2.numFrames(), v2.numColorStreams(), v2.numDepthStreams(), v2.width(), v2.height()) == (8, 3, 1, 128, 96)
    assert v2.aspect() == v.aspect() and v2.colorStream("down").extension() == ".raw" and v2.depthStream(0).depthXformDesc().str() == "Grid(Scale, Linear, 4, 3, 1)"
    for f in range(8):
        a, b = v2.depthStream(0).frame(f), ds.frame(f)
        np.testing.assert_array_equal(a.extrinsics.position, b.extrinsics.position)
        assert (a.extrinsics.orientation.y(), a.extrinsics.orientation.w()) == (b.extrinsics.orientation.y(), b.extrinsics.orientation.w())
        assert (a.intrinsics.vFov, a.intrinsics.hFov) == (b.intrinsics.vFov, b.intrinsics.hFov)
        assert list(a.depthXform().params()) == list(b.depthXform().params())
    np.testing.assert_array_equal(v2.depthStream(0).frame(1).sourceDepth(), ds.frame(1).sourceDepth())
    open(root2 + "/video.dat", "r+b").write(b"\x00\x00\x00\x00")
    with pytest.raises(RuntimeError, match="magic marker"):
        lp.DepthVideo().load(root2)
    img = np.full((96, 128), 2.5, np.float32); ds.frame(3).setDepth(img)
    np.testing.assert_array_equal(ds.frame(3).sourceDepth(), img)
    with pytest.raises(RuntimeError, match="inconsistent dimensions"):
        ds.frame(4).setDepth(np.zeros((10, 10), np.float32))
    p = lp.DepthVideoProcessor.Params()
    assert (p.colorStream, p.depthStream, p.sourceDepthStream, p.spatialRadius, p.frameRadius, p.median, p.farConnections) == (0, 0, 0, 0, 2, False, False)
    assert (p.depthSigma, p.colorSigma, p.matchSeparation, p.trackSpawnDistance, p.trackPruneDistance, p.minDynamicDistance, p.minTrackLength) == (np.float32(0.3), 0.0, 10, 20, 5, 3, 4)
    assert p.flowConsistancyThresh == np.float32(0.05)


GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_raw_files_written_by_the_reference_python_writer(tmp_path):
    """tests/golden/ref_writer_*.raw were written by the reference's own utils/image_io.py::save_raw_float32_image
    (tests/golden/make_golden.py imports it unchanged): the C++ reader must decode them, and our writers must produce the
    same bytes."""
    arrs = np.load(os.path.join(GOLDEN, "ref_writer_arrays.npz"))
    root = str(tmp_path / "v"); os.makedirs(root + "/d/depth"); os.makedirs(root + "/color_down")
    open(root + "/frames.txt", "w").write("1\n7\n5\n0.0\n")
    shutil.copy(os.path.join(GOLDEN, "ref_writer_disparity_5x7.raw"), root + "/d/depth/frame_000000.raw")
    shutil.copy(os.path.join(GOLDEN, "ref_writer_color_5x7x3.raw"), root + "/color_down/frame_000000.raw")
    v = lp.DepthVideo(); lp.DepthVideoImporter.importVideo(v, root, False)
    v.createColorStream("down", "color_down", ".raw", CV_32FC3); v.createDepthStream("d", "d", [-1, -1])
    src = np.asarray(v.depthStream(0).frame(0).sourceDepth())
    disp = arrs["disp"]
    with np.errstate(divide="ignore"):
        want = np.where(np.isfinite(disp) & (disp > 0), np.float32(1.0) / disp, np.float32(0.0)).astype(np.float32)   # lib/DepthStream.cpp:200-211
    np.testing.assert_array_equal(src, want)
    np.testing.assert_array_equal(np.asarray(v.colorStream("down").frame(0).image()), arrs["color"])
    # our Python and C++ writers emit the reference writer's bytes
    synthetic_files.write_raw(str(tmp_path / "flow.raw"), arrs["flow"])
    assert open(str(tmp_path / "flow.raw"), "rb").read() == open(os.path.join(GOLDEN, "ref_writer_flow_5x7x2.raw"), "rb").read()
    np.testing.assert_array_equal(synthetic_files.read_raw(os.path.join(GOLDEN, "ref_writer_flow_5x7x2.raw")), arrs["flow"])


def test_host_restatements_reproduce_their_goldens():
    """oracle/host_ref.py (post-filter loop, disc sampler) against tests/golden/host_restatement_golden.npz."""
    from tests.test_gpu_filter import make_filter_case
    g = np.load(os.path.join(GOLDEN, "host_restatement_golden.npz"))
    case, far_pairs, ff, fm = make_filter_case(F=5, w=20, h=12, seed=9, far=((2, 0), (2, 4)))
    got = host_ref.flow_guided_filter(**case, first_out=1, num_out=3, frame_radius=2, spatial_radius=0, median=False)
    np.testing.assert_array_equal(got, g["filter_mean_r0"])
    got = host_ref.flow_guided_filter(**case, first_out=1, num_out=3, frame_radius=2, spatial_radius=1, median=True, far_pairs=far_pairs, far_flow=ff, far_mask=fm)
    np.testing.assert_array_equal(got, g["filter_median_r1_far"])
    for sep in (1, 4):
        c, score = host_ref.pair_constraints(g["sampler_color"], g["sampler_flow"], g["sampler_mask"], sep, np.float32(0.75), score=g["sampler_score"])
        np.testing.assert_array_equal(c, g[f"sampler_sep{sep}"])


def test_constraints_match_numpy_cv2_restatement(scene_dir):
    import cv2
    sc, root, pairs, masks = scene_dir
    if os.path.exists(f"{root}/flow_constraints.dat"):
        os.remove(f"{root}/flow_constraints.dat")
    v = _open(root)
    fp = lp.FlowConstraintsParams(); fp.frameRange.resolve(v.numFrames(), True)
    assert (fp.matchSeparation, fp.minDynamicDistance, fp.doNotUseCache) == (10, -1.0, False)
    fc = lp.FlowConstraintsCollection(v, fp)
    P = fc._pairs()
    assert sorted(P.keys()) == sorted(map(tuple, pairs))
    total = 0
    for (a, b), (loc, st) in P.items():
        color = synthetic_files.read_raw(f"{root}/color_down/frame_{a:06d}.raw")
        flow = synthetic_files.read_raw(f"{root}/flow/flow_{a:06d}_{b:06d}.raw")
        mask = cv2.imread(f"{root}/flow_mask/mask_{a:06d}_{b:06d}.png", cv2.IMREAD_GRAYSCALE)
        ref, _ = host_ref.pair_constraints(color, flow, mask, 10, v.invAspect())
        np.testing.assert_array_equal(loc, ref)       # bit-exact selection, order and float32 locations
        assert st.all()
        total += len(ref)
    assert total > 2000
    # cache round trip: flow_constraints.dat
    raw = open(f"{root}/flow_constraints.dat", "rb").read()
    assert struct.unpack("<IIi", raw[:12]) == (0xDEADBEEF, 3, 10)
    fc2 = lp.FlowConstraintsCollection(v, fp)          # loads the cache
    for k, (loc, st) in fc2._pairs().items():
        np.testing.assert_array_equal(loc, P[k][0])
    # static flag from dynamic masks (distance > 8 at both ends; y scaled by the mask WIDTH as in the reference)
    fc.setStaticFlagFromDynamicMask(8)
    n_dyn = 0
    for (a, b), (loc, st) in fc._pairs().items():
        d0 = cv2.distanceTransform(np.where(masks[a] < 127, 0, 255).astype(np.uint8), cv2.DIST_L2, 5)
        d1 = cv2.distanceTransform(np.where(masks[b] < 127, 0, 255).astype(np.uint8), cv2.DIST_L2, 5)
        w = 128
        exp = (d0[(loc[:, 1] * np.float32(w)).astype(int), (loc[:, 0] * np.float32(w)).astype(int)] > 8) & \
              (d1[(loc[:, 3] * np.float32(w)).astype(int), (loc[:, 2] * np.float32(w)).astype(int)] > 8)
        np.testing.assert_array_equal(st, exp)
        n_dyn += int((~st).sum())
    assert n_dyn > 0


def test_image_operators_against_cv2(scene_dir):
    import cv2
    sc, root, pairs, masks = scene_dir
    color = synthetic_files.read_raw(f"{root}/color_down/frame_000003.raw")
    ref = cv2.cornerMinEigenVal(cv2.cvtColor(color, cv2.COLOR_BGR2GRAY), 3)
    mine = lp._cornerMinEigenVal3(color)
    np.testing.assert_array_equal(np.asarray(mine), ref)        # bit-exact: OpenCV's fused / double-accumulated operation order restated
    # ... at the BASELINE image sizes and at a width that exercises OpenCV's scalar tail (w % 4 != 0)
    rng = np.random.default_rng(11)
    for (hh, ww) in ((224, 384), (384, 640), (37, 53)):
        img = rng.uniform(0, 1, (hh, ww, 3)).astype(np.float32)
        img = (cv2.GaussianBlur(img, (0, 0), 1.5) + 0.2 * rng.uniform(0, 1, (hh, ww, 3)).astype(np.float32)).astype(np.float32)
        np.testing.assert_array_equal(np.asarray(lp._cornerMinEigenVal3(img)), cv2.cornerMinEigenVal(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), 3))
    b = np.where(masks[1] < 127, 0, 255).astype(np.uint8)
    # OpenCV's own fixed-point 5x5 chamfer vs the IPP float variant that pip-built cv2 dispatches to: metric 1.4 is
    # 91750/65536 in the former, float(1.4) in the latter -> differences of a few 1e-6 per step, irrelevant for the '> 8' test
    np.testing.assert_allclose(lp._distanceTransformL2_5(b), cv2.distanceTransform(b, cv2.DIST_L2, 5), rtol=1e-5, atol=1e-3)
    np.testing.assert_array_equal(lp._imreadPng(f"{root}/dynamic_mask/frame_000001.png", True), cv2.imread(f"{root}/dynamic_mask/frame_000001.png", cv2.IMREAD_GRAYSCALE))


def test_problem_assembly_records(scene_dir):
    sc, root, pairs, masks = scene_dir
    v = _open(root)
    fp = lp.FlowConstraintsParams(); fp.frameRange.resolve(v.numFrames(), True)
    fc = lp.FlowConstraintsCollection(v, fp)
    fc.setStaticFlagFromDynamicMask(8)
    proc = lp.DepthVideoProcessor(v)
    pp = lp.DepthVideoProcessor.Params(); pp.depthStream = v.numDepthStreams() - 1
    pp.depthXformDesc.type = lp.XformType.Depth; pp.depthXformDesc.depthType = lp.DepthXformType.Global; pp.depthXformDesc.valueXform = lp.ValueXformType.Scale
    pp.op = lp.DepthVideoProcessor.Op.ResetDepthXforms; proc.process(pp)
    opt = lp.DepthVideoPoseOptimizer(v, pp.depthStream)
    params = lp.DepthVideoPoseOptimizer.Params(); params.frameRange.fromString("0-7")
    d = opt._buildProblem(params, fc, 0.1, False)
    ds = v.depthStream(pp.depthStream)
    recs, offs, pf = [], [0], []
    for (a, b), (loc, st) in sorted(fc._pairs().items()):
        r = host_ref.observation_records(loc[st], ds.frame(a).sourceDepth(), ds.frame(b).sourceDepth(), v.invAspect())
        recs.append(r); offs.append(offs[-1] + len(r)); pf += [a, b]
    np.testing.assert_array_equal(d["records"].reshape(-1, 6), np.concatenate(recs))
    np.testing.assert_array_equal(d["offsets"], offs); np.testing.assert_array_equal(d["pair_frames"], pf)
    st = d["state"].reshape(8, -1)
    assert st.shape[1] == 8 and np.all(st[:, 7] == 1.0) and np.all(st[:, :6] == 0.0)
    np.testing.assert_allclose(st[:, 6], np.tan(np.float32(0.666488587) / 2.0), rtol=1e-7)
    for f in range(8):   # median over all depth pixels, nth_element at size/2
        s = np.sort(ds.frame(f).sourceDepth().ravel()); assert d["median"][f] == s[s.size // 2]
    # frame-range filtering: pairs need both ends in range
    params.frameRange.fromString("0-3")
    d2 = opt._buildProblem(params, fc, 0.1, False)
    assert set(map(tuple, d2["pair_frames"].reshape(-1, 2))) == {k for k in fc._pairs() if k[0] <= 3 and k[1] <= 3}
    assert d2["in_range"].tolist() == [1, 1, 1, 1, 0, 0, 0, 0]


def test_threaded_assembly_equals_sequential(scene_dir, monkeypatch):
    """Depth files / medians / observation records are assembled on host threads into per-item slots (model.h parallelFor): the arrays
    must not depend on the thread count, and a failure inside a worker (missing depth file) must surface as the same RuntimeError."""
    sc, root, pairs, masks = scene_dir

    def build(threads):
        monkeypatch.setenv("RCVD_HOST_THREADS", str(threads))
        v = _open(root)
        fp = lp.FlowConstraintsParams(); fp.frameRange.resolve(v.numFrames(), True)
        fc = lp.FlowConstraintsCollection(v, fp); fc.setStaticFlagFromDynamicMask(8)
        opt = lp.DepthVideoPoseOptimizer(v, v.numDepthStreams() - 1)
        params = lp.DepthVideoPoseOptimizer.Params(); params.frameRange.fromString("0-7")
        return opt._buildProblem(params, fc, 0.0, True), opt._buildProblem(params, fc, 0.1, False)
    (n1, s1), (n4, s4) = build(1), build(4)
    for a, b in ((n1, n4), (s1, s4)):
        for k in a:
            np.testing.assert_array_equal(np.asarray(a[k]), np.asarray(b[k]), err_msg=k)
    assert s4["records"].size > 0 and np.all(n4["median"] > 0)
    # a worker's exception is rethrown on the calling thread
    import shutil, tempfile
    broken = tempfile.mkdtemp(prefix="rcvd_broken_"); shutil.rmtree(broken); shutil.copytree(root, broken)
    try:
        os.remove(f"{broken}/depth_midas2/depth/frame_000005.raw")
        monkeypatch.setenv("RCVD_HOST_THREADS", "4")
        v = _open(broken)
        opt = lp.DepthVideoPoseOptimizer(v, v.numDepthStreams() - 1)
        params = lp.DepthVideoPoseOptimizer.Params(); params.frameRange.fromString("0-7")
        with pytest.raises(RuntimeError, match="Missing depth image"):
            opt._buildProblem(params, None, 0.0, True)
    finally:
        shutil.rmtree(broken, ignore_errors=True)


def test_adaptive_deformation_node_weights_follow_reference_splat(scene_dir):
    """AdaptiveDeformationCost constructor (reference lib/PoseOptimizer.cpp:559-619): every dynamic-mask pixel is splatted bilinearly onto
    the depth grid into a static or a dynamic accumulator; node weight = dynamic / (dynamic + static).  Restated here in numpy."""
    sc, root, pairs, masks = scene_dir
    v = _open(root)
    fp = lp.FlowConstraintsParams(); fp.frameRange.resolve(v.numFrames(), True)
    fc = lp.FlowConstraintsCollection(v, fp)
    proc = lp.DepthVideoProcessor(v)
    pp = lp.DepthVideoProcessor.Params(); pp.depthStream = v.numDepthStreams() - 1
    pp.depthXformDesc.type = lp.XformType.Depth; pp.depthXformDesc.parse("Grid(Scale, Linear, 6, 4, 1)")
    pp.op = lp.DepthVideoProcessor.Op.ResetDepthXforms; proc.process(pp)
    opt = lp.DepthVideoPoseOptimizer(v, pp.depthStream)
    params = lp.DepthVideoPoseOptimizer.Params(); params.frameRange.fromString("0-7"); params.adaptiveDeformationCost = 2.5
    d = opt._buildProblem(params, fc, 0.1, False)
    gw, gh = 6, 4
    got = d["adaptive"].reshape(8, gh, gw)
    for f in range(8):
        m = masks[f]; dh, dw = m.shape
        dyn = np.zeros((gh, gw)); sta = np.zeros((gh, gw))
        fy = np.arange(dh, dtype=np.float64) * (gh - 1) / dh; iy = fy.astype(int); ry = fy - iy
        fx = np.arange(dw, dtype=np.float64) * (gw - 1) / dw; ix = fx.astype(int); rx = fx - ix
        for y in range(dh):          # same accumulation order as the reference loop (row-major), so the sums agree to the last bit
            for x in range(dw):
                w = sta if m[y, x] > 127 else dyn
                w[iy[y], ix[x]] += (1.0 - rx[x]) * (1.0 - ry[y]); w[iy[y], ix[x] + 1] += rx[x] * (1.0 - ry[y])
                w[iy[y] + 1, ix[x]] += (1.0 - rx[x]) * ry[y]; w[iy[y] + 1, ix[x] + 1] += rx[x] * ry[y]
        np.testing.assert_array_equal(got[f], dyn / (dyn + sta))
    assert got.max() > 0.05 and got.min() == 0.0            # the blobs really reach some nodes
    cfg = abi.Config.from_buffer_copy(d["config"])
    assert cfg.adaptive_deform == 2.5 and cfg.depth_deform_reg == 0.1


def test_descriptor_strings_and_frame_range():
    d = lp.XformDescriptor(); d.type = lp.XformType.Depth
    d.parse("Grid(Scale, Linear, 17, 10, 1)")
    assert (d.depthType, d.valueXform, d.gridSize.tolist(), d.str()) == (lp.DepthXformType.Grid, lp.ValueXformType.Scale, [17, 10, 1], "Grid(Scale, Linear, 17, 10, 1)")
    d.parse("BicubicGrid(ScaleShift, 4, 3)"); assert d.str() == "Grid(ScaleShift, Cubic, 4, 3, 1)"
    d.parse("Global(Scale)"); assert d.str() == "Global(Scale)"
    s = lp.XformDescriptor(); s.reset(lp.XformType.Spatial); assert s.str() == "Identity"
    s.parse("BicubicGrid(4, 3)"); assert s.str() == "BicubicGrid(4, 3)" and s.spatialType == lp.SpatialXformType.BicubicGrid
    with pytest.raises(RuntimeError):
        d.parse("Grid(Scale, Quartic, 2, 2, 1)")
    r = lp.FrameRange(); r.fromString("0-3,7,9-10")
    assert (r.count(), r.firstFrame(), r.lastFrame(), r.toString(), r.isConsecutive(), r.inRange(5), r.inRange(9)) == (7, 0, 10, "0-3,7,9-10", False, False, True)
    r.resolve(8, True); assert r.toString() == "0-3,7"
    with pytest.raises(RuntimeError):
        q = lp.FrameRange(); q.fromString("5-9"); q.resolve(8)
    e = lp.FrameRange(); e.resolve(4); assert e.toString() == "0-3"


def test_pose_conversions_round_trip():
    from scipy.spatial.transform import Rotation as R
    rng = np.random.default_rng(0)
    for _ in range(50):
        aa = rng.normal(size=3) * rng.uniform(0.01, 3.0)
        q = lp._angleAxisToQuat(*aa)
        qr = R.from_rotvec(aa).as_quat()
        if np.dot(q, qr) < 0: qr = -qr
        np.testing.assert_allclose(q, qr, atol=2e-7)
        aa2 = np.array(lp._quatToAngleAxis(*q))
        np.testing.assert_allclose(R.from_rotvec(aa2).as_matrix(), R.from_rotvec(aa).as_matrix(), atol=5e-7)
    assert lp._quatToAngleAxis(0, 0, 0, 1) == (0.0, 0.0, 0.0)          # identity -> Taylor branch of the rotation
    assert lp._angleAxisToQuat(0, 0, 0) == (0.0, 0.0, 0.0, 1.0)


def test_grid_split_resamples_bilinearly(scene_dir):
    sc, root, pairs, masks = scene_dir
    v = _open(root)
    proc = lp.DepthVideoProcessor(v)
    pp = lp.DepthVideoProcessor.Params(); pp.depthStream = v.numDepthStreams() - 1
    pp.depthXformDesc.parse("Global(Scale)"); proc.resetDepthXforms(pp)
    pp.depthXformDesc.parse("Grid(Scale, Linear, 6, 4, 1)"); proc.gridXformSplit(pp)
    x = v.depthStream(pp.depthStream).frame(0).depthXform()
    assert x.numParams() == 24 and x.params() == [1.0] * 24 and x.desc().str() == "Grid(Scale, Linear, 6, 4, 1)"
    pp.depthXformDesc.parse("Grid(Scale, Linear, 12, 7, 1)"); proc.gridXformSplit(pp)
    assert v.depthStream(pp.depthStream).frame(3).depthXform().numParams() == 84
    with pytest.raises(RuntimeError):
        pp.depthXformDesc.parse("Grid(Scale, Linear, 4, 4, 1)"); proc.gridXformSplit(pp)   # fewer columns than before
    pr = lp.DepthVideoProcessor.Params(); pr.depthStream = pp.depthStream; proc.resetPoses(pr)
    f = v.depthStream(pp.depthStream).frame(1)
    assert abs(f.intrinsics.hFov - 2 * np.arctan(np.float32(0.3461538376301239))) < 1e-6


NO_CPU_FALLBACK = "no CPU fallback|no usable CUDA device"


def _replay(ops, objs, root):
    """Replays a recorded lib_python call sequence (tests/golden/make_golden.py records it): every attribute read, call and
    assignment, each primitive result checked against the recorded one.  A recorded failure may only end the sequence and must be
    the refusal to run without a GPU; returns whether the sequence ended in it."""
    def dec(v):
        if isinstance(v, dict):
            return objs[v["ref"]]
        if isinstance(v, list):
            return [dec(x) for x in v]
        return v.replace("{root}", root) if isinstance(v, str) else v
    for i, op in enumerate(ops):
        o = objs[op["obj"]]
        if op["op"] == "set":
            setattr(o, op["name"], dec(op["value"]))
            continue
        if "raises" in op:
            assert i == len(ops) - 1 and op["raises"]["type"] == "RuntimeError" and re.search(NO_CPU_FALLBACK, op["raises"]["message"]), op
            with pytest.raises(RuntimeError, match=NO_CPU_FALLBACK):
                o(*dec(op["args"]))
            return True
        out = getattr(o, op["name"]) if op["op"] == "get" else o(*dec(op["args"]))
        if isinstance(op["out"], dict):
            objs[op["out"]["ref"]] = out
        else:
            assert (list(out) if isinstance(out, tuple) else out) == dec(op["out"]), (i, op)
    return False


def test_reference_pose_optimization_py_runs_unchanged_up_to_the_solve(tmp_path):
    """The calls the reference's own pose_optimization.py makes into lib_python (PoseOptimizer(...) and optimize_poses() on
    this module's 8-frame scene, recorded from the unmodified script into tests/golden/ref_pose_optimization_trace.json) run
    against our lib_python with the same results: everything up to the device solve runs here; the solve itself must refuse to
    run without a GPU (no CPU fallback)."""
    import json
    trace = json.load(open(os.path.join(GOLDEN, "ref_pose_optimization_trace.json")))
    root = str(tmp_path / "scene8")
    write_scene8(root)
    objs = {0: lp}
    assert not _replay(trace["init"], objs, root)
    assert os.path.exists(f"{root}/flow_constraints.dat") and os.path.exists(f"{root}/video.dat")
    import torch
    if not torch.cuda.is_available():
        assert _replay(trace["optimize_poses"], objs, root)
