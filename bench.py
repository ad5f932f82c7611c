#!/usr/bin/env python3
"""bench.py -- flow-residual-constraints/sec per Gauss-Newton (LM) iteration (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W                (our arm: CUDA path through the C ABI)
  python bench.py --impl reference --gpus N --steps K --warmup W   (reference arm: CPU restatement, host cores)
  python bench.py ... --dump-outputs DIR                        (also writes what the last timed step computed, DIR/<name>.npy)

Workload (config.workload): BASELINE.json configs[1] -- 300 frames, 384x224, 16x12 bilinear depth-scale
grid, hierarchical2 frame pairs, matchSeparation 10 (reference default), Cauchy 0.5, PerFrame intrinsics,
synthetic scene (robust_cvd_b200/synthetic.py: MiDaS / RAFT weights are not in the image, their outputs are
emulated).  A "step" is one full LM iteration's device work at a fixed state: residual + Jacobian +
normal-equation accumulation, damped block-Cholesky factor + solve, candidate-cost evaluation.
value = constraints / step time, inputs resident in HBM.  e2e = the same through the C ABI with host
buffers (create + upload + K-iteration solve + download), host<->device copies inside the timed region.

The reference (Ceres/Eigen/OpenCV C++) cannot be built in this image, so --impl reference times the
repo's CPU restatement of it (oracle/, "port") on the box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from robust_cvd_b200 import abi, synthetic  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs.  scene: synthetic.Scene keyword arguments; cfg: rcvd_config overrides; mask_ratio: overlap filter of the
    # pair schedule (loaders/video_dataset.py:129-136, `--flow_min_mask_ratio`-style score > ratio on flow_list.json)
    "config2_300f_384x224_grid16x12_sep10": dict(frames=300, w=384, h=224, gx=16, gy=12, sep=10),
    "config1_8f_128x96_grid4x4_sep10": dict(frames=8, w=128, h=96, gx=4, gy=4, sep=10),
    # config 3: the same video with a faster camera so that the 0.20 overlap filter actually removes long-range pairs
    "config3_300f_384x224_grid16x12_sep10_maskratio0.20": dict(frames=300, w=384, h=224, gx=16, gy=12, sep=10, mask_ratio=0.20,
                                                               scene=dict(rot_deg=1.2, motion=0.04)),
    # config 4: Huber robustifier (an extension: the reference only has Cauchy, SURVEY fact 1)
    "config4_1000f_640x384_grid32x24_sep10": dict(frames=1000, w=640, h=384, gx=32, gy=24, sep=10),
    "config4_1000f_640x384_grid32x24_sep10_huber": dict(frames=1000, w=640, h=384, gx=32, gy=24, sep=10, cfg=dict(robust_type=abi.ROBUST_HUBER, robustness=0.05)),
    # config 5: dynamic-mask holes (29 % of every frame => ~50 % of the pixels of a pair keep both ends visible) and a dolly-in
    # (divergent flow field)
    "config5_300f_384x224_grid16x12_sep10_holes50_dolly": dict(frames=300, w=384, h=224, gx=16, gy=12, sep=10, scene=dict(hole_fraction=0.29, dolly=0.008)),
}
METRIC = "flow_residual_constraints_per_sec_per_gn_iteration"
def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the two roofline kernels, from the `ncu --set full` captures of THIS
    round's kernels (profiles/r2_ncu_traffic.json, written by tools/round_profiles_post.sh together with the kernel names and the capture
    command); null when the file is missing or was captured for other kernels."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))
        return {"update": t["k_update_tma"]["dram_bytes_per_launch"], "accumulate": t["k_accumulate_runs"]["dram_bytes_per_launch"], "source": t["source"]}
    except Exception:
        return {"update": None, "accumulate": None, "source": None}


def build_case(wl, frames=None, sep=None, seed=2, valid_fraction=1.0):
    spec = dict(WORKLOADS[wl])
    if frames:
        spec["frames"] = frames
    if sep is not None:
        spec["sep"] = sep
    sc = synthetic.Scene(spec["frames"], spec["w"], spec["h"], seed=seed, **spec.get("scene", {}))
    cfg = abi.default_config(spec["frames"], sc.aspect, depth_type=abi.DEPTH_GRID, depth_grid_x=spec["gx"], depth_grid_y=spec["gy"], **spec.get("cfg", {}))
    pair_list = sc.filtered_pairs(spec["mask_ratio"]) if spec.get("mask_ratio") else None
    pairs, offs, rec = sc.constraints(pairs=pair_list, sep=spec["sep"], valid_fraction=valid_fraction)
    med = sc.median_depths(stride=8)
    return spec, sc, cfg, pairs, offs, rec, med


def initial_state(sc, cfg, stride):
    nd = cfg.depth_grid_x * cfg.depth_grid_y
    x = sc.gt_state(stride, 7, nd)
    rng = np.random.default_rng(7)
    return x + rng.normal(0, 0.005, x.shape)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes float64 arrays as out_dir/<name>.npy so that two builds can be compared output for output.  Arrays of one row per
    frame that would exceed DUMP_LIMIT_BYTES together keep a fixed, seeded sample of frames; sampled_frames.npy lists them."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    per_frame = [k for k, v in arrays.items() if v.ndim == 2]
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES and per_frame:
        n = arrays[per_frame[0]].shape[0]
        row_bytes = sum(arrays[k][0].nbytes for k in per_frame) + 8      # + the entry of sampled_frames
        keep = (DUMP_LIMIT_BYTES - 4096 - (total - n * (row_bytes - 8))) // row_bytes   # 4 KiB for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: (v[rows] if k in per_frame else v) for k, v in arrays.items()}
        arrays["sampled_frames"] = rows.astype(np.float64)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def shard_pairs(pairs, offs, rec, rank, nranks):
    """Longest-processing-time partition of directed pairs by constraint count (SURVEY.md 8e)."""
    from robust_cvd_b200 import sharding
    sel = sharding.lpt_partition(np.diff(offs), nranks)[rank]
    return sharding.take_pairs(pairs, offs, rec, sel)


class ClockSampler:
    def __init__(self, device=0):
        self.samples, self.reasons, self.proc, self.thread = [], set(), None, None
        self.device = device

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def run():
            for line in self.proc.stdout:
                parts = [s.strip() for s in line.split(",")]
                try:
                    self.samples.append((float(parts[0]), float(parts[1])))
                    for n, v in zip(names, parts[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(n)
                except Exception:
                    pass
        self.thread = threading.Thread(target=run, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples), "reasons": sorted(self.reasons), "samples": len(sm)}


class CpuBaseline:
    """One LM iteration of the CPU restatement (oracle 'port': analytic Jacobian + level-parallel block Cholesky, OpenMP over
    the CPUs the cgroup grants) on the same workload; `frames` < workload frames takes a frame-prefix sample."""

    def __init__(self, wl, frames=None):
        from oracle import oracle
        self.threads = oracle.effective_cpus()
        oracle.set_threads(self.threads)
        total = WORKLOADS[wl]["frames"]
        nf = min(frames or total, total)
        spec, sc, cfg, pairs, offs, rec, med = build_case(wl, frames=nf)
        self.O = oracle.OracleProblem(cfg)
        self.O.set_frames(np.ones(cfg.num_frames, np.uint8), med)
        self.O.set_constraints(pairs, offs, rec)
        self.O.set_state(initial_state(sc, cfg, self.O.stride))
        self.C = int(rec.shape[0]); self.npairs = len(pairs)
        self.what = ("all" if nf == total else f"first {nf} of") + f" {total} frames ({self.npairs} pairs, {self.C} constraints)"

    def step(self):
        ev, li, co = self.O.time_iteration()
        return ev, li, co

    def describe(self, times):
        ev, li, co = np.median(np.array(times), axis=0)
        tot = (ev + li + co) / 1e3
        return {"value": float(self.C / tot), "unit": "constraints/s", "cores": self.threads, "kind": "port",
                "sample": f"{self.what}, one LM iteration: eval {ev:.1f} ms + factor/solve {li:.1f} ms + cost {co:.1f} ms, median of {len(times)}",
                "ms_per_step": float(tot * 1e3)}


def cpu_baseline_sample(wl, seconds_budget=25.0, frames=None):
    cb = CpuBaseline(wl, frames)
    cb.step()    # warm-up
    t0 = time.time(); times = []
    while (time.time() - t0 < seconds_budget and len(times) < 5) or not times:
        times.append(cb.step())
    return cb.describe(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = CpuBaseline(args.workload, args.ref_frames)
    for _ in range(args.warmup):
        cb.step()
    t0 = time.perf_counter()
    times = [cb.step() for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    d = cb.describe(times)
    v = float(cb.C * args.steps / wall)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "constraints/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": wall * 1e3 / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "note": "CPU restatement of the reference (Ceres semantics restated, not Ceres; the reference's C++ needs Ceres/Eigen/OpenCV "
                       "which are not in this image) on the box's host cores; step = one LM iteration's work (evaluate+accumulate, factor+solve, candidate cost)"},
            "cpu_baseline": {"value": v, "unit": "constraints/s", "cores": d["cores"], "kind": d["kind"], "sample": d["sample"]},
            "e2e": {"value": v, "unit": "constraints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    from robust_cvd_b200 import solver
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    spec, sc, cfg, pairs, offs, rec, med = build_case(args.workload, frames=args.frames, sep=args.sep)
    C_total = int(rec.shape[0])
    P = solver.Problem(cfg, device=local)
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.from_numpy(solver.nccl_unique_id()).cuda()
        dist.broadcast(uid, 0)
        P.init_comm(world, rank, uid.cpu().numpy())
        P.set_structure(pairs)
        lp, lo, lr = shard_pairs(pairs, offs, rec, rank, world)
    else:
        lp, lo, lr = pairs, offs, rec
    P.set_frames(np.ones(cfg.num_frames, np.uint8), med)
    P.set_constraints(lp, lo, lr)
    x0 = initial_state(sc, cfg, P.stride)
    P.set_state(x0)
    if args.legacy_update or args.side_ipc:
        P.set_update_kernel(not args.legacy_update, args.side_ipc)
    if world > 1 and args.no_dist:
        P.set_distributed(False)
    info = P.structure_info()
    dinfo = P.distribution_info()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (also builds the structure, uploads, instantiates the CUDA graph)
    t_w = P.time_iteration(iters=max(args.warmup, 3))
    sampler = ClockSampler(local); sampler.start()
    sync_all()
    l0 = P.launch_count()
    t0 = time.perf_counter()
    tm = P.time_iteration(iters=args.steps)     # device-timed (CUDA events on the solver stream), K steps
    sync_all()
    wall = time.perf_counter() - t0
    launches = P.launch_count() - l0
    clocks = sampler.stop()
    outputs = P.iteration_outputs() if args.dump_outputs else None      # before the calls below overwrite the device buffers
    ms = tm["iter_ms"]
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    acc_ms = P.time_accumulate(iters=max(args.steps, 5))
    # ---- parity evidence at the size that was just timed (outside the timed region) ----
    # (a) device-side residual of the damped normal equations of one LM step (SpMV over the assembled H, independent of the
    #     factorisation kernels) + cost / |g| checksums; (b) N > 1: the all-reduced cost / gradient of every rank against a
    #     single-GPU evaluation of the whole problem on rank 0.
    lr_ = P.linear_residual(1e4)
    parity = {"linear_rel_residual": lr_["rel_residual"], "pivot_fail": int(lr_["pivot_fail"]), "cost": lr_["cost"], "grad_norm": lr_["grad_norm"],
              "step_norm": lr_["step_norm"], "bar": "rel_residual < 1e-8; N>1: cost/gradient of every rank vs rank-0 full evaluation <= 1e-9 relative",
              "tests": "tests/test_gpu_parity_at_size.py compares this workload with the CPU oracle (cost, gradient, linear solve, LM iterations)"}
    if world > 1:
        c_sh, g_sh = P.evaluate(True)
        chk = torch.tensor([c_sh, float(np.linalg.norm(g_sh)), float(np.abs(g_sh).sum())], dtype=torch.float64, device="cuda")
        allchk = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allchk, chk)
        if rank == 0:
            Q = solver.Problem(cfg, device=local)
            Q.set_eval_only(True)        # cost / gradient only: no second copy of the matrices next to the sharded problem
            Q.set_frames(np.ones(cfg.num_frames, np.uint8), med); Q.set_constraints(pairs, offs, rec); Q.set_state(x0)
            c_full, g_full = Q.evaluate(True)
            Q.close()
            ref = np.array([c_full, np.linalg.norm(g_full), np.abs(g_full).sum()])
            parity["multi_gpu"] = {"ranks": world, "max_rel_diff_cost_gradnorm_gradl1_vs_rank0_full_evaluation": float(max(np.max(np.abs(a.cpu().numpy() - ref) / np.abs(ref)) for a in allchk)),
                                   "max_abs_grad_diff_rank0": float(np.abs(g_sh - g_full).max()), "grad_max": float(np.abs(g_full).max())}
    lin_prof = P.profile_linear(reps=3)            # per-kernel-class device time, serialised (CUDA events around every launch)
    peak64 = solver.fp64_tensor_peak(local)        # live DMMA peak (TFLOP/s) of this GPU
    # ---- e2e: C ABI with host buffers, copies inside the timed region ----
    e2e_iters = args.e2e_iters
    opt = abi.default_solve_options(max_iterations=e2e_iters)
    opt.function_tolerance = 0.0; opt.parameter_tolerance = 0.0; opt.gradient_tolerance = 0.0   # run exactly e2e_iters iterations
    pinned = [torch.from_numpy(a).pin_memory().numpy() for a in (lr, x0)]
    def e2e_once():
        Q = solver.Problem(cfg, device=local)
        if world > 1:
            Q.init_comm_from(P) if hasattr(Q, "init_comm_from") else None
        Q.set_frames(np.ones(cfg.num_frames, np.uint8), med)
        Q.set_constraints(lp, lo, pinned[0])
        Q.set_state(pinned[1])
        s = Q.solve(opt)
        xs = Q.get_state()
        Q.close()
        return s, xs
    def e2e_once_multi():
        # N > 1: the handle (and its NCCL communicator) is kept, everything else of a call is redone: host shard -> device,
        # structure, LM solve with the per-evaluation all-reduces, state back to the host
        P.set_frames(np.ones(cfg.num_frames, np.uint8), med)
        P.set_constraints(lp, lo, pinned[0])
        P.set_state(pinned[1])
        s = P.solve(opt)
        return s, P.get_state()
    e2e = None
    if world == 1:
        P.close()          # the e2e calls create their own handle; two resident copies of a large problem (config 4: ~107 GB) do not fit
    if not args.skip_e2e:
        call = e2e_once if world == 1 else e2e_once_multi
        call()
        sync_all(); t1 = time.perf_counter(); its = 0
        for _ in range(args.e2e_steps):
            s, xs = call(); its += s.iterations
        sync_all(); dt = time.perf_counter() - t1
        if outputs is not None:
            outputs.update(e2e_state=xs, e2e_costs=np.array([s.initial_cost, s.final_cost]))
        h2d = float(lr.nbytes + lp.nbytes + lo.nbytes + x0.nbytes + med.nbytes + cfg.num_frames)
        if world > 1:
            tt = torch.tensor([dt, -h2d], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX); dt = float(tt[0].item())
            hh = torch.tensor([h2d], dtype=torch.float64, device="cuda"); dist.all_reduce(hh, op=dist.ReduceOp.SUM); h2d = float(hh.item())
        e2e = {"value": C_total * its / dt, "unit": "constraints/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(x0.nbytes) * world, "lm_iterations_per_call": its // max(args.e2e_steps, 1), "ms_per_call": dt * 1e3 / args.e2e_steps,
               "note": ("rcvd_problem_create + set_frames/constraints/state (pinned host) + rcvd_solve + get_state + destroy per call" if world == 1 else
                        "per rank: set_frames/constraints/state of its pair shard (pinned host) + rcvd_solve (NCCL all-reduces inside) + get_state on a kept handle/communicator; max over ranks")}
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = ncu_traffic()
    # algorithmic bytes of the residual/Jacobian/accumulate pass (SURVEY 8d): 24 B per constraint + per pair
    # ids + 2 parameter vectors + the outputs (gradient + H blocks of the original structure)
    nf, npad = info["stride"], info["npad"]
    alg_bytes = 24.0 * C_total + len(pairs) * (8 + 16 * nf) + 8.0 * cfg.num_frames * nf + 8.0 * info["h_blocks"] * nf * nf
    roof_acc = {"bound": "hbm", "kernel": "gn_accumulate (memset of H + k_accumulate_runs + k_regularisers + cost reduction)", "achieved": alg_bytes / (acc_ms * 1e-3) / 1e9,
                "peak": hbm_peak, "unit": "GB/s", "frac": alg_bytes / (acc_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback 6650 GB/s",
                "traffic": traffic["accumulate"], "traffic_source": traffic["source"], "ms": acc_ms,
                "note": "latency / fp64-issue bound at matchSeparation 10 (22 MB of records, L2 resident), not HBM bound: see DESIGN.md section 4"}
    traffic_note = None
    # dominant kernel of the step: k_update_tma, the fp64 tensor-core block updates of the sparse Cholesky
    n_g = max(lin_prof["gemm_launches"], 1.0)
    g_tf = lin_prof["gemm_flops"] / max(lin_prof["gemm_ms"] * 1e-3, 1e-12) / 1e12
    roof = {"bound": "tensor", "kernel": "k_update_tma (TMA-fed fp64 DMMA Schur updates of the block Cholesky)" if not args.legacy_update else "k_gemm_nt (round-1 cp.async kernel)", "achieved": g_tf, "peak": peak64, "unit": "TFLOP/s",
            "frac": g_tf / peak64, "peak_source": "fp64 DMMA.8x8x4 register loop measured live (rcvd_debug_fp64_tensor_peak); MEASURED_PEAKS.json has no fp64 figure",
            "traffic": traffic["update"], "traffic_source": traffic["source"], "launches_per_step": int(n_g), "avg_launch_us": lin_prof["gemm_ms"] * 1e3 / n_g,
            "flops_per_launch": lin_prof["gemm_flops"] / n_g, "share_of_step_serialised": lin_prof["gemm_ms"] / max(sum(lin_prof[k] for k in ("load_ms", "potrf_ms", "trinv_ms", "trsm_ms", "gemm_ms", "solve_ms")) + acc_ms, 1e-9)}
    line = {"metric": METRIC, "value": C_total / (ms * 1e-3), "unit": "constraints/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload if not args.frames else f"{args.workload}[frames={args.frames}]", "frames": spec["frames"], "image": [spec["w"], spec["h"]],
                       "depth_grid": [spec["gx"], spec["gy"]], "match_separation": spec["sep"], "pairs": int(len(pairs)), "constraints": C_total,
                       "unknowns": int(cfg.num_frames * nf), "parallelism": (f"pair-sharded x{world}; " + ("H reduced to block owners, wide elimination levels factored by frame owners (one fused NCCL broadcast of the new factor blocks per level), narrow tail + substitution replicated" if dinfo["distributed"] else "H all-reduced, factorisation replicated")) if world > 1 else "single GPU",
                       "distribution": dinfo, "l2_note": "H/L working set >> L2 (126 MB)",
                       "structure": info},
            "breakdown_ms": {"accumulate": tm["accumulate_ms"], "factor_solve": tm["linear_ms"], "candidate_cost": tm["cost_ms"], "accumulate_isolated": acc_ms},
            "linear_kernels_ms_serialised": {k: lin_prof[k] for k in ("load_ms", "potrf_ms", "trinv_ms", "trsm_ms", "gemm_ms", "solve_ms")},
            "roofline": roof, "roofline_accumulate": roof_acc, "parity": parity, "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall}
    if e2e:
        line["e2e"] = e2e
    if world == 1 and not args.skip_cpu:
        try:
            line["cpu_baseline"] = {k: v for k, v in cpu_baseline_sample(args.workload, seconds_budget=25.0, frames=args.ref_frames).items() if k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:  # the oracle is a checker; its absence must not hide the GPU number
            line["cpu_baseline"] = {"error": str(e)}
    if world == 1 and not args.skip_pose_opt:
        # metric (ii): pose-optimisation wall-clock through the reference-facing module (lib_python) on a 300-frame directory on disk
        # (own process: a fresh CUDA context and allocator, as a pose_optimization.py run has -- inside this process the same call
        # measured 2-3x slower after the bench's other work)
        try:
            cmd = [sys.executable, os.path.join(ROOT, "tools", "bench_pose_opt.py"), "--frames", str(args.pose_opt_frames), "--max-iterations", str(args.pose_opt_iterations), "--autodiff-iterations", "1"]
            if args.skip_cpu:
                cmd.append("--skip-cpu")
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
            line["pose_opt_wallclock"] = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1]) if out.returncode == 0 else {"error": out.stderr[-600:]}
        except Exception as e:
            line["pose_opt_wallclock"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2_300f_384x224_grid16x12_sep10", choices=list(WORKLOADS))
    ap.add_argument("--frames", type=int, default=None, help="override frame count (debug)")
    ap.add_argument("--sep", type=int, default=None, help="override matchSeparation (0 = dense)")
    ap.add_argument("--ref-frames", type=int, default=None, help="frame-prefix size of the CPU sample (default: the whole workload)")
    ap.add_argument("--e2e-iters", type=int, default=20)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-pose-opt", action="store_true", help="skip metric (ii), the lib_python normalizeDepth + optimizePoses wall-clock on a directory on disk")
    ap.add_argument("--pose-opt-frames", type=int, default=300)
    ap.add_argument("--pose-opt-iterations", type=int, default=10, help="LM iteration cap per solve of the pose-opt wall-clock run (GPU and CPU replay alike)")
    ap.add_argument("--no-dist", action="store_true", help="A/B at N > 1: round-1 scheme (all-reduce of H, factorisation replicated on every rank)")
    ap.add_argument("--legacy-update", action="store_true", help="A/B: round-1 cp.async update GEMM instead of the TMA-fed persistent kernel")
    ap.add_argument("--side-ipc", type=int, default=0, help="A/B: items-per-CTA cap of the overlapped (side-stream) update launches")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (gradient, LM step, candidate state, costs; and the last e2e call's final "
                         "state and costs) as DIR/<name>.npy, float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        try:
            run_ours(args)
        except BaseException:
            import traceback
            traceback.print_exc()
            sys.stderr.flush()
            os._exit(1)          # a rank that failed must not linger in a collective: the launcher then tears the job down at once


if __name__ == "__main__":
    main()
