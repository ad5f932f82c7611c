"""Bilateral depth filter on the GPU (rcvd_bilateral_filter, csrc/rcvd_bilateral.cuh) against the float32 restatement of
the reference loop (tests/bilateral_ref.py, lib/Processor.cpp:183-313): through the C ABI, in place with a
depth transform, through lib_python, and at size."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "robust_cvd_b200", "host"))

from tests import bilateral_ref  # noqa: E402
from robust_cvd_b200 import abi, solver, synthetic, synthetic_files  # noqa: E402

pytestmark = pytest.mark.gpu
CV_32FC3 = 21


def _case(F=6, h=20, w=37, seed=0):
    """w = 37: rows that are not a multiple of 16 bytes (the device planes are pitched)."""
    rng = np.random.default_rng(seed)
    depth = rng.uniform(0.5, 2.0, (F, h, w)).astype(np.float32)
    depth[:, 3:9, 5:20] = 1.25                      # a flat patch: exact ties in the median
    color = rng.uniform(0.0, 1.0, (F, h, w, 3)).astype(np.float32)
    return depth, color


def _launches():
    return solver.lib().rcvd_filter_launch_count()


def _compare(got, want, median):
    assert got.shape == want.shape and np.isfinite(got).all()
    close = np.isclose(got, want, rtol=1e-5, atol=0)
    # the weighted median picks one sample: a last-ulp difference of expf may move the pick at a near-tie
    assert close.mean() >= (0.995 if median else 1.0), (close.mean(), np.abs(got - want).max())


def _grid_cfg():
    return abi.default_config(1, 1.0, depth_type=abi.DEPTH_GRID, value_xform=abi.VALUE_SCALE, depth_grid_x=4, depth_grid_y=3)


@pytest.mark.parametrize("median", [False, True])
@pytest.mark.parametrize("ds,cs", [(0.3, 0.0), (0.3, 0.15), (0.0, 0.15)])
@pytest.mark.parametrize("R", [0, 1, 2])
@pytest.mark.parametrize("r", [0, 1, 3])
def test_c_abi_matches_restatement(r, R, ds, cs, median):
    depth, color = _case()
    frames = [0, 2, 3, 5]          # first and last video frames; frames 1 and 4 are read by windows only
    want = bilateral_ref.bilateral_filter(depth, frames, R, r, ds, cs, median, color=color)
    l0 = _launches()
    got = solver.bilateral_filter(depth, frames, R, r, ds, cs, median, color=color if cs > 0 else None)
    assert _launches() > l0
    _compare(got, want, median)
    if cs == 0 and (r, R) != (0, 0):   # a strong colour term can leave the centre sample dominant: output = input
        assert np.abs(got - depth[frames]).max() > 1e-3


@pytest.mark.parametrize("median", [False, True])
@pytest.mark.parametrize("r", [0, 1, 3])
def test_bit_exact_without_range_weights(r, median):
    """depthSigma = colorSigma = 0: every weight is 1, so the output pins the summation order, the sort and the tie rule."""
    depth, _ = _case(F=7, seed=1)
    frames = [1, 3, 4, 5]          # the range "1,3-5"
    want = bilateral_ref.bilateral_filter(depth, frames, 2, r, 0.0, 0.0, median)
    got = solver.bilateral_filter(depth, frames, 2, r, 0.0, 0.0, median)
    assert np.array_equal(got, want)


def test_launch_count_and_bad_arguments():
    depth, color = _case()
    l0 = _launches()
    solver.bilateral_filter(depth, [0, 1, 2, 3, 4, 5], 2, 1, 0.3, 0.1, False, color=color)
    assert _launches() == l0 + 1
    with pytest.raises(RuntimeError, match="ascending"):
        solver.bilateral_filter(depth, [2, 1], 2, 1, 0.3, 0.0, False)
    with pytest.raises(RuntimeError, match="colour"):
        solver.bilateral_filter(depth, [1], 2, 1, 0.3, 0.1, False)
    with pytest.raises(RuntimeError, match="too large"):
        solver.bilateral_filter(depth, [1], 2, 40, 0.3, 0.1, False, color=color)


def _grid_inputs(F, h, w, seed):
    rng = np.random.default_rng(seed)
    cfg = _grid_cfg()
    xp = rng.uniform(0.6, 1.6, (F, 12))
    src = rng.uniform(0.5, 2.0, (F, h, w)).astype(np.float32)
    depth = np.stack([solver.depth_apply(cfg, xp[f], src[f]) for f in range(F)])
    return cfg, xp, depth


@pytest.mark.parametrize("median", [False, True])
def test_in_place_chain_with_grid_transform(median):
    F, h, w = 8, 18, 29
    cfg, xp, depth = _grid_inputs(F, h, w, seed=7)
    _, color = _case(F, h, w, seed=8)
    frames = [0, 1, 2, 4, 5, 7]
    l0 = _launches()
    got = solver.bilateral_filter(depth, frames, 2, 1, 0.0, 0.0, median, in_place=True, xform_cfg=cfg, xform_params=xp[frames])
    assert _launches() == l0 + len(frames)          # one launch per frame, in range order
    want = bilateral_ref.bilateral_filter(depth, frames, 2, 1, 0.0, 0.0, median, in_place=True,
                                          retransform=lambda k, img: solver.depth_apply(cfg, xp[frames[k]], img))
    assert np.array_equal(got, want)
    plain = solver.bilateral_filter(depth, frames, 2, 1, 0.0, 0.0, median)
    assert np.array_equal(got[0], plain[0])
    assert all(not np.array_equal(got[k], plain[k]) for k in range(1, len(frames)))
    # with range weights (mean): close to the chained restatement
    if not median:
        got = solver.bilateral_filter(depth, frames, 2, 1, 0.3, 0.1, False, color=color, in_place=True, xform_cfg=cfg, xform_params=xp[frames])
        want = bilateral_ref.bilateral_filter(depth, frames, 2, 1, 0.3, 0.1, False, color=color, in_place=True,
                                              retransform=lambda k, img: solver.depth_apply(cfg, xp[frames[k]], img))
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=0)


def test_through_lib_python(tmp_path):
    """Op.BilateralFilter out of place into a created stream, then saveDepth / load; then bilateralFilter in place on stream 0
    with a grid depth transform: afterwards depth() of each frame is the transform applied to the filtered image, bit for bit."""
    import lib_python as lp
    root = str(tmp_path / "scene")
    N, W, H = 7, 40, 24
    sc = synthetic.Scene(N, W, H, seed=4)
    synthetic_files.write_scene(sc, root)
    v = lp.DepthVideo(); lp.DepthVideoImporter.importVideo(v, root, False)
    v.createColorStream("down", "color_down", ".raw", CV_32FC3)
    v.createDepthStream("depth_midas2", "depth_midas2", [-1, -1])
    src = v.depthStream(0)
    proc = lp.DepthVideoProcessor(v)
    rp = lp.DepthVideoProcessor.Params(); rp.depthStream = 0
    rp.depthXformDesc.type = lp.XformType.Depth; rp.depthXformDesc.depthType = lp.DepthXformType.Grid
    rp.depthXformDesc.valueXform = lp.ValueXformType.Scale; rp.depthXformDesc.gridSize = [4, 3, 1]
    proc.resetDepthXforms(rp)
    # Xform.params() returns a copy, as in the reference: the frames keep the reset parameters (random grid parameters are
    # covered through the C ABI by test_in_place_chain_with_grid_transform)
    xp = np.stack([np.asarray(src.frame(f).depthXform().params(), np.float64) for f in range(N)])
    assert xp.shape == (N, 12)
    depth = np.stack([np.array(src.frame(f).depth()) for f in range(N)])
    color = np.stack([synthetic_files.read_raw(os.path.join(root, "color_down", f"frame_{f:06d}.raw")) for f in range(N)]).astype(np.float32)
    # --- out of place, through process() ---
    dst_id = v.numDepthStreams()
    v.createDepthStream("depth_bilateral", "depth_bilateral", [W, H])
    params = lp.DepthVideoProcessor.Params()
    assert (params.spatialRadius, params.frameRadius, params.median) == (0, 2, False)
    assert abs(params.depthSigma - 0.3) < 1e-7 and params.colorSigma == 0.0   # lib/Processor.h defaults
    params.op = lp.DepthVideoProcessor.Op.BilateralFilter; params.depthStream = dst_id
    params.frameRange.fromString("1-4"); params.spatialRadius = 1; params.colorSigma = 0.1
    l0 = _launches()
    proc.process(params)
    assert _launches() == l0 + 1
    got = np.stack([np.array(v.depthStream(dst_id).frame(f).depth()) for f in range(1, 5)])
    want = bilateral_ref.bilateral_filter(depth, [1, 2, 3, 4], 2, 1, 0.3, 0.1, False, color=color)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=0)
    v.saveDepth(dst_id); v.save()
    v2 = lp.DepthVideo(); v2.load(root)
    np.testing.assert_allclose(np.array(v2.depthStream(dst_id).frame(2).depth()), got[1], rtol=2e-6)   # disparity round trip
    # --- in place on stream 0, through bilateralFilter() ---
    params = lp.DepthVideoProcessor.Params()
    params.frameRange.fromString("0,2-5"); params.depthSigma = 0.0; params.spatialRadius = 1; params.frameRadius = 2; params.median = True
    frames = [0, 2, 3, 4, 5]
    l0 = _launches()
    proc.bilateralFilter(params)
    assert _launches() == l0 + len(frames)
    cfg = _grid_cfg()
    want = bilateral_ref.bilateral_filter(depth, frames, 2, 1, 0.0, 0.0, True, in_place=True,
                                          retransform=lambda k, img: solver.depth_apply(cfg, xp[frames[k]], img))
    for k, f in enumerate(frames):
        filtered = np.array(src.frame(f).sourceDepth())
        assert np.array_equal(filtered, want[k])
        assert np.array_equal(np.array(src.frame(f).depth()), solver.depth_apply(cfg, xp[f], filtered))
    assert np.array_equal(np.array(src.frame(1).depth()), depth[1])   # outside the range: untouched


def test_at_size_against_sampled_pixels():
    """300 frames of 384 x 224, r = 2, R = 2, depthSigma 0.3, colorSigma 0.1: 2 000 sampled pixels (100 in each of 20 frames,
    including the first and the last) against the restatement, mean and median; in place against the restatement fed the GPU's
    own earlier outputs, re-transformed."""
    F, h, w = 300, 224, 384
    rng = np.random.default_rng(21)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = (1.0 + 0.3 * np.sin(xx / 23.0) * np.cos(yy / 17.0)).astype(np.float32)
    depth = (base[None] * rng.uniform(0.9, 1.1, (F, 1, 1)) + rng.normal(0, 0.05, (F, h, w))).astype(np.float32)
    color = rng.uniform(0.0, 1.0, (F, h, w, 3)).astype(np.float32)
    sample_frames = np.unique(np.concatenate([[0, F - 1], rng.choice(F, 18, replace=False)]))[:20]
    ys, xs = rng.integers(0, h, 100), rng.integers(0, w, 100)
    ys[:4] = [0, h - 1, 0, h - 1]; xs[:4] = [0, w - 1, w - 1, 0]          # corners
    for median in (False, True):
        got = solver.bilateral_filter(depth, np.arange(F), 2, 2, 0.3, 0.1, median, color=color)
        want = bilateral_ref.bilateral_filter(depth, sample_frames, 2, 2, 0.3, 0.1, median, color=color, pixels=(ys, xs))
        _compare(got[sample_frames][:, ys, xs], want, median)
    cfg = abi.default_config(1, w / h, depth_type=abi.DEPTH_GRID, value_xform=abi.VALUE_SCALE, depth_grid_x=5, depth_grid_y=4)
    xp = rng.uniform(0.8, 1.25, (F, 20))
    got = solver.bilateral_filter(depth, np.arange(F), 2, 2, 0.3, 0.1, False, color=color, in_place=True, xform_cfg=cfg, xform_params=xp)
    for f in (0, 1, 150, F - 1):
        fed = depth.copy()
        for g in range(max(0, f - 2), f):
            fed[g] = solver.depth_apply(cfg, xp[g], got[g])
        want = bilateral_ref.bilateral_filter(fed, [f], 2, 2, 0.3, 0.1, False, color=color, pixels=(ys, xs))
        _compare(got[f][ys, xs][None], want, False)
