"""Bilateral depth filter (DepthVideoProcessor::bilateralFilter, reference lib/Processor.cpp:183-313) without a GPU: the
float32 restatement in tests/bilateral_ref.py against an independent float64 formulation, its in-place mode, and the host
argument checks of lib_python, which all run before the first device call."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "robust_cvd_b200", "host"))

from tests import bilateral_ref  # noqa: E402
from robust_cvd_b200 import synthetic, synthetic_files  # noqa: E402

CV_8UC3, CV_32FC3 = 16, 21


def _case(F=5, h=12, w=16, seed=0):
    rng = np.random.default_rng(seed)
    depth = rng.uniform(0.5, 2.0, (F, h, w)).astype(np.float32)
    color = rng.uniform(0.0, 1.0, (F, h, w, 3)).astype(np.float32)
    return depth, color


def _mean_float64(depth, color, frame, R, r, ds, cs):
    """Whole-window formulation: NaN-padded sliding windows of every window frame, weights in float64."""
    F, h, w = depth.shape
    d = np.pad(depth.astype(np.float64), ((0, 0), (r, r), (r, r)), constant_values=np.nan)
    c = np.pad(color.astype(np.float64), ((0, 0), (r, r), (r, r), (0, 0)), constant_values=np.nan)
    frames = range(max(0, frame - R), min(F - 1, frame + R) + 1)
    dw = np.stack([np.lib.stride_tricks.sliding_window_view(d[g], (2 * r + 1, 2 * r + 1)) for g in frames])        # [T,h,w,k,k]
    cw = np.stack([np.lib.stride_tricks.sliding_window_view(c[g], (2 * r + 1, 2 * r + 1), axis=(0, 1)) for g in frames])  # [T,h,w,3,k,k]
    e = np.zeros(dw.shape)
    if ds > 0:
        e -= (dw - depth[frame].astype(np.float64)[None, :, :, None, None]) ** 2 / np.float64(np.float32(ds) * np.float32(ds))
    if cs > 0:
        diff = cw - color[frame].astype(np.float64)[None, :, :, :, None, None]
        e -= (diff ** 2).sum(3) / np.float64(np.float32(cs) * np.float32(cs))
    wt = np.where(np.isnan(dw), 0.0, np.exp(e))
    return np.nansum(dw * wt, axis=(0, 3, 4)) / wt.sum(axis=(0, 3, 4))


@pytest.mark.parametrize("r", [0, 1, 3])
@pytest.mark.parametrize("ds,cs", [(0.0, 0.0), (0.3, 0.0), (0.0, 0.2), (0.3, 0.2)])
def test_restatement_mean_matches_float64(r, ds, cs):
    depth, color = _case()
    frames = [0, 2, 4]
    got = bilateral_ref.bilateral_filter(depth, frames, 2, r, ds, cs, False, color=color)
    for k, f in enumerate(frames):
        want = _mean_float64(depth, color, f, 2, r, ds, cs)
        np.testing.assert_allclose(got[k], want, rtol=1e-5, atol=0)


def test_restatement_median_picks_a_window_sample():
    depth, color = _case(seed=1)
    got = bilateral_ref.bilateral_filter(depth, [1, 3], 1, 1, 0.3, 0.2, True, color=color)
    for k, f in enumerate([1, 3]):
        window = depth[f - 1:f + 2]
        for y in (0, 5, 11):
            for x in (0, 7, 15):
                near = window[:, max(0, y - 1):y + 2, max(0, x - 1):x + 2]
                assert got[k, y, x] in near
    # equal weights: the weighted median is the lower median of the window
    got = bilateral_ref.bilateral_filter(depth, [2], 1, 1, 0.0, 0.0, True)
    y, x = 6, 8
    s = np.sort(depth[1:4, y - 1:y + 2, x - 1:x + 2].ravel())
    assert got[0, y, x] == s[(s.size - 1) // 2]


def test_restatement_pixel_subset():
    depth, color = _case(seed=2)
    full = bilateral_ref.bilateral_filter(depth, [1, 4], 2, 1, 0.3, 0.1, True, color=color)
    ys, xs = np.array([0, 3, 11, 11]), np.array([0, 9, 15, 2])
    sub = bilateral_ref.bilateral_filter(depth, [1, 4], 2, 1, 0.3, 0.1, True, color=color, pixels=(ys, xs))
    np.testing.assert_array_equal(sub, full[:, ys, xs])


def test_in_place_restatement_chains_frames():
    """In place = out of place one frame at a time, each filtered frame re-transformed before the next frame's window."""
    depth, color = _case(F=7, seed=4)
    frames = [1, 2, 3, 5]
    scale = np.float32([1.5, 0.75, 2.0, 1.25])

    def retransform(k, img):
        return (img * scale[k]).astype(np.float32)
    got = bilateral_ref.bilateral_filter(depth, frames, 2, 1, 0.3, 0.2, False, color=color, in_place=True, retransform=retransform)
    cur = depth.copy()
    for k, f in enumerate(frames):
        res = bilateral_ref.bilateral_filter(cur, [f], 2, 1, 0.3, 0.2, False, color=color)[0]
        np.testing.assert_array_equal(got[k], res)
        cur[f] = retransform(k, res)
    plain = bilateral_ref.bilateral_filter(depth, frames, 2, 1, 0.3, 0.2, False, color=color)
    np.testing.assert_array_equal(got[0], plain[0])
    assert not np.array_equal(got[1], plain[1])


# ---- lib_python ----
@pytest.fixture(scope="module")
def lp():
    return pytest.importorskip("lib_python")


def _has_device():
    from robust_cvd_b200 import solver
    return solver.lib().rcvd_current_device() >= 0


@pytest.fixture
def scene(tmp_path):
    root = str(tmp_path / "scene")
    sc = synthetic.Scene(5, 24, 16, seed=2)
    synthetic_files.write_scene(sc, root)
    return root


def _video(lp, root, color_type=CV_32FC3, color_dir="color_down", ext=".raw"):
    v = lp.DepthVideo(); lp.DepthVideoImporter.importVideo(v, root, False)
    if color_type is not None:
        v.createColorStream("down", color_dir, ext, color_type)
    v.createDepthStream("depth_midas2", "depth_midas2", [-1, -1])
    return v


def _params(lp, frames="0-4", **kw):
    p = lp.DepthVideoProcessor.Params()
    p.op = lp.DepthVideoProcessor.Op.BilateralFilter
    p.frameRange.fromString(frames)
    for k, val in kw.items():
        setattr(p, k, val)
    return p


def test_lib_python_binds_bilateral_filter(lp):
    assert hasattr(lp.DepthVideoProcessor, "bilateralFilter")
    assert hasattr(lp.DepthVideoProcessor.Op, "BilateralFilter")


def test_host_argument_errors_before_any_device_call(lp, scene):
    v = _video(lp, scene)
    proc = lp.DepthVideoProcessor(v)
    cases = [
        (_params(lp, spatialRadius=-1), "non-negative"),
        (_params(lp, frameRadius=-2), "non-negative"),
        (_params(lp, frames="3-9"), "out of range"),
        (_params(lp, depthStream=4), "Depth stream index out of range"),
    ]
    for p, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            proc.bilateralFilter(p)
        with pytest.raises(RuntimeError, match=msg):
            proc.process(p)
    # no "down" colour stream
    with pytest.raises(RuntimeError, match="not found"):
        lp.DepthVideoProcessor(_video(lp, scene, color_type=None)).bilateralFilter(_params(lp))
    # "down" is not CV_32FC3 (ColorFrame::image3f)
    with pytest.raises(RuntimeError, match="incorrect type"):
        lp.DepthVideoProcessor(_video(lp, scene, color_type=CV_8UC3, ext=".png")).bilateralFilter(_params(lp))
    # colour of another size than the depth (read only when the colour term is on)
    other = os.path.join(scene, "color_small")
    os.makedirs(other)
    for f in range(5):
        synthetic_files.write_raw(os.path.join(other, f"frame_{f:06d}.raw"), np.zeros((8, 12, 3), np.float32))
    with pytest.raises(RuntimeError, match="size"):
        lp.DepthVideoProcessor(_video(lp, scene, color_dir="color_small")).bilateralFilter(_params(lp, colorSigma=0.1))
    # a depth frame some window reaches is missing
    os.remove(os.path.join(scene, "depth_midas2", "depth", "frame_000004.raw"))
    with pytest.raises(RuntimeError, match="frame 4 has no depth"):
        lp.DepthVideoProcessor(_video(lp, scene)).bilateralFilter(_params(lp, frames="2", frameRadius=2))


@pytest.mark.skipif("_has_device()")
def test_without_device_reports_no_device(lp, scene):
    from robust_cvd_b200 import solver
    depth, color = _case()
    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        solver.bilateral_filter(depth, [0, 1], color=color, color_sigma=0.1)
    v = _video(lp, scene)
    for call in (lambda p: lp.DepthVideoProcessor(v).process(p), lambda p: lp.DepthVideoProcessor(v).bilateralFilter(p)):
        with pytest.raises(RuntimeError) as e:
            call(_params(lp))
        assert "no usable CUDA device" in str(e.value) and "not implemented" not in str(e.value)
