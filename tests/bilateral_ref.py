"""Float32 restatement of the reference's bilateral depth filter (TEST INFRASTRUCTURE; checks rcvd_bilateral_filter and
DepthVideoProcessor::bilateralFilter in robust_cvd_b200/host/optimizer.cpp against lib/Processor.cpp:183-313)."""
import numpy as np

f32 = np.float32


# Vectorised over pixels only: every pixel visits its window in the reference's order (window frame, row, column) and every
# operation is one float32 rounding, as in the reference loop.
def _bilateral_frame(depth, color, frame, frame_radius, spatial_radius, depth_sigma, color_sigma, median, ys, xs):
    F, h, w = depth.shape
    ds2, cs2 = f32(depth_sigma) * f32(depth_sigma), f32(color_sigma) * f32(color_sigma)
    use_d, use_c = f32(depth_sigma) > 0, f32(color_sigma) > 0
    dref = depth[frame, ys, xs]
    cref = color[frame, ys, xs] if use_c else None
    P = ys.size
    dsum = np.zeros(P, f32); wsum = np.zeros(P, f32)
    samples = []                                    # (depth, weight, valid) in scan order, for the median
    r = spatial_radius
    for g in range(max(0, frame - frame_radius), min(F - 1, frame + frame_radius) + 1):
        for dy in range(-r, r + 1):
            yy = ys + dy; vy = (yy >= 0) & (yy < h); yc = np.clip(yy, 0, h - 1)
            for dx in range(-r, r + 1):
                xx = xs + dx; valid = vy & (xx >= 0) & (xx < w); xc = np.clip(xx, 0, w - 1)
                d = depth[g, yc, xc]
                e = np.zeros(P, f32)
                if use_d:
                    diff = (d - dref).astype(f32)
                    e = (e + (-(diff * diff).astype(f32)) / ds2).astype(f32)
                if use_c:
                    c = (color[g, yc, xc] - cref).astype(f32)
                    s = ((c[:, 0] * c[:, 0]).astype(f32) + (c[:, 1] * c[:, 1]).astype(f32)).astype(f32)
                    s = (s + (c[:, 2] * c[:, 2]).astype(f32)).astype(f32)
                    e = (e + (-s) / cs2).astype(f32)
                wt = np.where(e != 0, np.exp(e), f32(1)).astype(f32)
                if median:
                    samples.append((d, wt, valid))
                else:
                    dsum = np.where(valid, dsum + (d * wt).astype(f32), dsum).astype(f32)
                wsum = np.where(valid, wsum + wt, wsum).astype(f32)
    if not median:
        return np.where(wsum > 0, dsum / np.where(wsum > 0, wsum, f32(1)), f32(0)).astype(f32)
    sd = np.stack([s[0] for s in samples], 1); sw = np.stack([s[1] for s in samples], 1); sv = np.stack([s[2] for s in samples], 1)
    order = np.lexsort((sw, sd, ~sv), axis=1)       # (depth, weight) ascending, samples outside the image last
    sd = np.take_along_axis(sd, order, 1); sw = np.take_along_axis(np.where(sv, sw, f32(0)), order, 1); sv = np.take_along_axis(sv, order, 1)
    cum = np.add.accumulate(sw, axis=1, dtype=f32)   # sequential float32 running sum in sorted order
    hit = (cum >= (wsum / f32(2)).astype(f32)[:, None]) & sv
    first = np.argmax(hit, axis=1)
    return np.where(hit.any(1), sd[np.arange(P), first], f32(0)).astype(f32)


def bilateral_filter(depth, out_frames, frame_radius, spatial_radius, depth_sigma, color_sigma, median, color=None,
                     in_place=False, retransform=None, pixels=None):
    """depth [F,h,w] f32 (every frame of the video), color [F,h,w,3] f32 (read when color_sigma > 0), out_frames ascending.
    Returns [len(out_frames),h,w] f32, or [len(out_frames),n] for pixels=(ys, xs).  in_place: after frame out_frames[k] is
    filtered, its depth becomes retransform(k, filtered) for the windows of later frames (depthStream == 0 in the reference)."""
    depth = np.array(depth, f32, copy=True)
    F, h, w = depth.shape
    if pixels is None:
        ys, xs = (a.ravel() for a in np.mgrid[0:h, 0:w])
    else:
        ys, xs = np.asarray(pixels[0], np.int64), np.asarray(pixels[1], np.int64)
    if in_place and (pixels is not None or retransform is None):
        raise ValueError("in_place needs whole frames and a retransform callable")
    with np.errstate(all="ignore"):
        out = []
        for k, f in enumerate(out_frames):
            res = _bilateral_frame(depth, color, int(f), frame_radius, spatial_radius, depth_sigma, color_sigma, median, ys, xs)
            out.append(res if pixels is not None else res.reshape(h, w))
            if in_place:
                depth[int(f)] = np.asarray(retransform(k, out[-1]), f32)
    return np.stack(out)
