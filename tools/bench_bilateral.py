"""Bilateral depth filter benchmark (rcvd_bilateral_filter / DepthVideoProcessor::bilateralFilter) on a synthetic
300-frame 384 x 224 video.  Prints one JSON document (and writes it to --out):

  * per case: kernel time per frame from CUDA events-backed profiler records of k_bilateral (warmed, repeated), samples/s,
    algorithmic bytes/s (every depth / colour frame read once, every output written once) against the 7.7 TB/s of HBM3e,
    H2D and D2H copy time of the C ABI call, and its wall-clock;
  * lib_python wall-clock of bilateralFilter on files written to a temporary directory, with the depth() gathering timed
    on its own and the C ABI call (H2D, kernel, D2H) timed on the same inputs; the remainder is colour reads, host copies
    and setDepth;
  * the GPU name and power limit, read in the same run.

Cases: the Params defaults (spatialRadius 0, frameRadius 2, depthSigma 0.3, mean), spatialRadius 2 with colour
(colorSigma 0.1), the median with spatialRadius 2; each out of place and in place (depthStream 0: one launch per frame)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "robust_cvd_b200", "host"))

from robust_cvd_b200 import abi, solver, synthetic, synthetic_files  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
CASES = [
    dict(name="defaults_r0_R2_mean", r=0, R=2, ds=0.3, cs=0.0, median=False),
    dict(name="r2_R2_color_mean", r=2, R=2, ds=0.3, cs=0.1, median=False),
    dict(name="r2_R2_color_median", r=2, R=2, ds=0.3, cs=0.1, median=True),
]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def count_samples(F, h, w, r, R):
    rows = sum(min(h - 1, y + r) - max(0, y - r) + 1 for y in range(h))
    cols = sum(min(w - 1, x + r) - max(0, x - r) + 1 for x in range(w))
    frames = sum(min(F - 1, f + R) - max(0, f - R) + 1 for f in range(F))
    return rows * cols * frames


def profile_call(fn, reps):
    """Kernel / H2D / D2H device time per call from torch.profiler CUDA activity records."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    kern = h2d = d2h = 0.0
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        n = e.name
        if "k_bilateral" in n:
            kern += us
        elif "HtoD" in n:
            h2d += us
        elif "DtoH" in n:
            d2h += us
    return kern / reps / 1e3, h2d / reps / 1e3, d2h / reps / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--width", type=int, default=384)
    ap.add_argument("--height", type=int, default=224)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    F, w, h = args.frames, args.width, args.height
    sc = synthetic.Scene(F, w, h, seed=1)
    depth = np.stack([sc.depth_image(f) for f in range(F)]).astype(np.float32)
    color = np.stack([synthetic_files.texture(sc, f) for f in range(F)]).astype(np.float32)
    cfg = abi.default_config(1, w / h, depth_type=abi.DEPTH_GRID, value_xform=abi.VALUE_SCALE, depth_grid_x=5, depth_grid_y=4)
    xp = np.random.default_rng(2).uniform(0.8, 1.25, (F, 20))
    frames = np.arange(F)
    result = {"workload": f"{F} frames of {w} x {h}", **gpu_info(), "cases": []}
    for c in CASES:
        for in_place in (False, True):
            kw = dict(frame_radius=c["R"], spatial_radius=c["r"], depth_sigma=c["ds"], color_sigma=c["cs"], median=c["median"],
                      color=color if c["cs"] > 0 else None, in_place=in_place, xform_cfg=cfg if in_place else None, xform_params=xp if in_place else None)
            call = lambda: solver.bilateral_filter(depth, frames, **kw)  # noqa: E731
            call()                                   # warm-up: module load, pool growth
            t0 = time.perf_counter()
            for _ in range(args.reps):
                call()
            wall = (time.perf_counter() - t0) / args.reps * 1e3
            kern, h2d, d2h = profile_call(call, args.reps)
            samples = count_samples(F, h, w, c["r"], c["R"])
            nbytes = F * h * w * 4 * (2 + (3 if c["cs"] > 0 else 0)) + (F * h * w * 4 if in_place else 0)
            result["cases"].append({
                "case": c["name"], "in_place": in_place, "launches": F if in_place else "1 (median: frame chunks of <= 1 GiB scratch)" if c["median"] else 1,
                "kernel_ms": round(kern, 3), "kernel_us_per_frame": round(kern / F * 1e3, 2),
                "h2d_ms": round(h2d, 3), "d2h_ms": round(d2h, 3), "abi_call_wall_ms": round(wall, 2),
                "samples": samples, "samples_per_s": float(f"{samples / (kern / 1e3):.4g}"),
                "algorithmic_bytes": nbytes, "algorithmic_bytes_per_s": float(f"{nbytes / (kern / 1e3):.4g}"),
                "share_of_hbm_bandwidth": round(nbytes / (kern / 1e3) / HBM_BYTES_PER_S, 4)})
            print(json.dumps(result["cases"][-1]), file=sys.stderr)
    # ---- lib_python wall-clock ----
    import lib_python as lp
    CV_32FC3 = 21
    with tempfile.TemporaryDirectory() as tmp:
        root = os.path.join(tmp, "scene")
        synthetic_files.write_scene(sc, root, pairs=[])
        lib_rows = []
        for c in CASES[:2]:
            for in_place in (False, True):
                v = lp.DepthVideo(); lp.DepthVideoImporter.importVideo(v, root, False)
                v.createColorStream("down", "color_down", ".raw", CV_32FC3)
                v.createDepthStream("depth_midas2", "depth_midas2", [-1, -1])
                proc = lp.DepthVideoProcessor(v)
                rp = lp.DepthVideoProcessor.Params(); rp.depthStream = 0
                rp.depthXformDesc.type = lp.XformType.Depth; rp.depthXformDesc.depthType = lp.DepthXformType.Grid
                rp.depthXformDesc.valueXform = lp.ValueXformType.Scale; rp.depthXformDesc.gridSize = [5, 4, 1]
                proc.resetDepthXforms(rp)
                src = v.depthStream(0)
                xp_lp = np.stack([np.asarray(src.frame(f).depthXform().params(), np.float64) for f in range(F)])   # params() is a copy
                if not in_place:
                    v.createDepthStream("depth_bilateral", "depth_bilateral", [w, h])
                params = lp.DepthVideoProcessor.Params()
                params.op = lp.DepthVideoProcessor.Op.BilateralFilter; params.frameRange.fromString(f"0-{F - 1}")
                params.spatialRadius = c["r"]; params.frameRadius = c["R"]; params.depthSigma = c["ds"]; params.colorSigma = c["cs"]
                params.depthStream = 0 if in_place else 1
                for f in range(F):                   # source depth files read once, outside the timed region
                    src.frame(f).sourceDepth()
                t0 = time.perf_counter()
                depth_lp = [np.array(src.frame(f).depth()) for f in range(F)]
                t_depth = (time.perf_counter() - t0) * 1e3
                for f in range(F):
                    src.frame(f).clearXformedCache()
                t0 = time.perf_counter()
                proc.bilateralFilter(params)
                total = (time.perf_counter() - t0) * 1e3
                dl = np.stack(depth_lp)
                kw = dict(frame_radius=c["R"], spatial_radius=c["r"], depth_sigma=c["ds"], color_sigma=c["cs"], median=False,
                          color=color if c["cs"] > 0 else None, in_place=in_place, xform_cfg=cfg if in_place else None, xform_params=xp_lp if in_place else None)
                t0 = time.perf_counter()
                solver.bilateral_filter(dl, frames, **kw)
                t_abi = (time.perf_counter() - t0) * 1e3
                lib_rows.append({"case": c["name"], "in_place": in_place, "bilateralFilter_wall_ms": round(total, 1),
                                 "depth_gather_ms": round(t_depth, 1), "abi_call_ms": round(t_abi, 1),
                                 "colour_reads_copies_setDepth_ms": round(total - t_depth - t_abi, 1)})
                print(json.dumps(lib_rows[-1]), file=sys.stderr)
        result["lib_python"] = lib_rows
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
