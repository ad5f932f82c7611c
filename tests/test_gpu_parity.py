"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.
Run on the B200 box with `pytest -m gpu`."""
import numpy as np
import pytest

from robust_cvd_b200 import abi
from tests import helpers

pytestmark = pytest.mark.gpu


def _both(overrides, num_frames=8, **kw):
    from oracle import oracle
    from robust_cvd_b200 import solver
    sc, cfg, pairs, offs, rec, med = helpers.make_case(num_frames=num_frames, **overrides, **kw)
    off_d, nd = helpers.layout_numbers(cfg)
    O = oracle.OracleProblem(cfg)
    G = solver.Problem(cfg)
    assert O.stride == G.stride
    x = helpers.initial_state(sc, cfg, G.stride, off_d, nd)
    helpers.setup_problem(O, cfg, pairs, offs, rec, med, x)
    helpers.setup_problem(G, cfg, pairs, offs, rec, med, x)
    return sc, cfg, O, G, x


@pytest.mark.parametrize("name,overrides", helpers.VARIANTS, ids=[v[0] for v in helpers.VARIANTS])
def test_cost_gradient_normal_matrix(name, overrides):
    sc, cfg, O, G, x = _both(overrides)
    co, go = O.evaluate(True)
    cg, gg = G.evaluate(True)
    assert abs(co - cg) <= 1e-11 * abs(co), (co, cg)
    assert np.abs(go - gg).max() <= 1e-9 * max(1.0, np.abs(go).max())
    Ho = O.normal_matrix_dense()
    Hg = G.normal_matrix_dense()
    assert np.abs(Ho - Hg).max() <= 1e-9 * np.abs(Ho).max()


@pytest.mark.parametrize("name,overrides", helpers.VARIANTS[:4], ids=[v[0] for v in helpers.VARIANTS[:4]])
def test_linear_solve(name, overrides):
    sc, cfg, O, G, x = _both(overrides)
    Ho = O.normal_matrix_dense()
    U = Ho.shape[0]
    rng = np.random.default_rng(3)
    S = 1.0 / (1.0 + np.sqrt(np.diag(Ho)))
    D2 = np.clip(S * S * np.diag(Ho), 1e-6, 1e32) / 1e4
    b = rng.normal(size=U)
    A = Ho * S[:, None] * S[None, :] + np.diag(D2)
    y_ref = np.linalg.solve(A, b)
    y = G.debug_linear_solve(S, D2, b)
    res = np.linalg.norm(A @ y - b) / np.linalg.norm(b)
    assert res < 1e-8, res
    assert np.linalg.norm(y - y_ref) / np.linalg.norm(y_ref) < 1e-6
    # solver variants must agree to round-off: level-scheduled substitution launches (instead of the persistent dataflow kernel),
    # round-1 pivot-tile Cholesky, untrimmed update GEMMs, single-stream graph, explicit-inverse TRSM
    for setter in (lambda: G.set_fused_substitution(False), lambda: G.L.rcvd_debug_set_potrf_chain_warp(G.h, 3), lambda: G.set_trim_gemm(False),
                   lambda: G.set_overlap(False), lambda: G.set_trsm_ll(False)):
        setter()
        y2 = G.debug_linear_solve(S, D2, b)
        assert np.linalg.norm(y2 - y) / np.linalg.norm(y) < 1e-9


def test_iteration_outputs_are_one_lm_step():
    """Problem.iteration_outputs (what bench.py --dump-outputs writes) after time_iteration: cost and gradient at the state, the
    Jacobi-scaled LM step of trust radius 1e4 on the oracle's normal matrix, and the cost at the candidate state."""
    sc, cfg, O, G, x = _both(helpers.VARIANTS[0][1])
    G.time_iteration(iters=2, radius=1e4)
    out = G.iteration_outputs()
    co, go = O.evaluate(True)
    assert abs(out["costs"][0] - co) <= 1e-11 * abs(co), (out["costs"], co)
    assert np.abs(out["gradient"].ravel() - go).max() <= 1e-9 * max(1.0, np.abs(go).max())
    H = O.normal_matrix_dense()
    S = 1.0 / (1.0 + np.sqrt(np.diag(H)))
    D2 = np.clip(S * S * np.diag(H), 1e-6, 1e32) / 1e4
    step = -S * np.linalg.solve(H * S[:, None] * S[None, :] + np.diag(D2), S * go)
    assert np.linalg.norm(out["step"].ravel() - step) <= 1e-6 * np.linalg.norm(step)
    G.set_state(out["candidate_state"])
    assert abs(G.evaluate() - out["costs"][1]) <= 1e-11 * abs(out["costs"][1])


@pytest.mark.parametrize("name,overrides", helpers.VARIANTS, ids=[v[0] for v in helpers.VARIANTS])
def test_lm_solve_matches_oracle(name, overrides):
    sc, cfg, O, G, x = _both(overrides)
    # the Euclidean world-space loss is singular in practice (the reference notes it 'does not produce good results',
    # lib/PoseOptimizer.cpp:268-269): once the trust radius saturates round-off decides individual steps, so compare early
    opt = abi.default_solve_options(max_iterations=25 if cfg.static_loss_type == abi.LOSS_EUCLIDEAN else 60)
    so = O.solve(opt)
    sg = G.solve(opt)
    assert sg.gpu_launches > 0
    assert so.termination == sg.termination, (so.message, sg.message)
    assert abs(so.final_cost - sg.final_cost) <= 1e-6 * abs(so.final_cost), (so.final_cost, sg.final_cost)
    assert abs(so.iterations - sg.iterations) <= 2
    xo, xg = O.get_state(), G.get_state()
    # same trajectory up to round-off: parameters agree well inside the 1e-4 relative target
    rel = np.linalg.norm(xo - xg) / np.linalg.norm(xo)
    assert rel < 1e-4, rel


@pytest.mark.parametrize("cubic", [0, 1])
def test_adaptive_deformation_cost_with_node_weights(cubic):
    """AdaptiveDeformationCost (reference lib/PoseOptimizer.cpp:559-656, :1470-1481) with non-zero per-node weights: residual of a grid
    edge x (base + max(w_i, w_j) adaptive).  CUDA regulariser kernel vs the oracle: cost, gradient, normal matrix, LM trajectory."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    ov = dict(depth_type=abi.DEPTH_GRID, depth_grid_x=6, depth_grid_y=4, depth_cubic=cubic, depth_deform_reg=0.07, adaptive_deform=3.0)
    sc, cfg, pairs, offs, rec, med = helpers.make_case(num_frames=8, **ov)
    off_d, nd = helpers.layout_numbers(cfg)
    rng = np.random.default_rng(21)
    aw = rng.uniform(0.0, 1.0, (8, 4, 6)); aw[rng.uniform(size=aw.shape) < 0.4] = 0.0          # static regions have weight 0
    O = oracle.OracleProblem(cfg); G = solver.Problem(cfg)
    x = helpers.initial_state(sc, cfg, G.stride, off_d, nd, perturb=0.03)
    helpers.setup_problem(O, cfg, pairs, offs, rec, med, x, adaptive=aw)
    helpers.setup_problem(G, cfg, pairs, offs, rec, med, x, adaptive=aw)
    co, go = O.evaluate(True); cg, gg = G.evaluate(True)
    assert abs(co - cg) <= 1e-11 * abs(co) and np.abs(go - gg).max() <= 1e-9 * max(1.0, np.abs(go).max())
    Ho, Hg = O.normal_matrix_dense(), G.normal_matrix_dense()
    assert np.abs(Ho - Hg).max() <= 1e-9 * np.abs(Ho).max()
    # the weights matter: the same problem without them has a different cost
    cfg0 = abi.default_config(8, sc.aspect, **dict(ov, adaptive_deform=0.0))
    G0 = solver.Problem(cfg0); helpers.setup_problem(G0, cfg0, pairs, offs, rec, med, x)
    assert abs(G0.evaluate() - cg) > 1e-6 * abs(cg)
    opt = abi.default_solve_options(max_iterations=40)
    so, sg = O.solve(opt), G.solve(opt)
    assert so.termination == sg.termination and abs(so.iterations - sg.iterations) <= 2
    assert abs(so.final_cost - sg.final_cost) <= 1e-6 * abs(so.final_cost)
    assert np.linalg.norm(O.get_state() - G.get_state()) <= 1e-4 * np.linalg.norm(O.get_state())


@pytest.mark.parametrize("name", ["bilinear_perframe_disp", "global_perframe_disp", "bilinear_fixedintr_ratio", "global_euclid", "identitydepth_perframe"])
def test_fast_kernel_matches_generic(name):
    overrides = dict(helpers.VARIANTS)[name]
    sc, cfg, O, G, x = _both(overrides)
    Hf = G.normal_matrix_dense(); cf, gf = G.evaluate(True)      # default: run path on bilinear grids (records sorted by cell pair), else k_accumulate_fast
    G.set_fast_path(2)
    Hr = G.normal_matrix_dense(); cr, gr = G.evaluate(True)      # round-1 specialised kernel, unsorted records
    G.set_fast_path(0)
    Hg = G.normal_matrix_dense(); cg, gg = G.evaluate(True)      # generic kernel
    for Hs, cs_, gs_ in ((Hf, cf, gf), (Hr, cr, gr)):
        assert np.abs(Hs - Hg).max() <= 1e-10 * np.abs(Hg).max()
        assert np.abs(gs_ - gg).max() <= 1e-10 * max(1.0, np.abs(gg).max())
        assert abs(cs_ - cg) <= 1e-12 * abs(cg)


def test_run_path_dense_and_ragged_runs():
    """Run path of the accumulate kernel on dense constraints (matchSeparation 0: runs longer than a warp, split at warp and tile
    boundaries) and on a coarse 3x2 grid (few cell pairs, very long runs) against the generic kernel and the oracle."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    for gx, gy, sep, frames in ((5, 4, 0, 3), (3, 2, 4, 5), (16, 12, 10, 6)):
        sc, cfg, pairs, offs, rec, med = helpers.make_case(num_frames=frames, w=64, h=48, sep=sep, depth_type=abi.DEPTH_GRID, depth_grid_x=gx, depth_grid_y=gy)
        off_d, nd = helpers.layout_numbers(cfg)
        G = solver.Problem(cfg); O = oracle.OracleProblem(cfg)
        x = helpers.initial_state(sc, cfg, G.stride, off_d, nd)
        helpers.setup_problem(G, cfg, pairs, offs, rec, med, x); helpers.setup_problem(O, cfg, pairs, offs, rec, med, x)
        Hf = G.normal_matrix_dense(); cf, gf = G.evaluate(True)
        Ho = O.normal_matrix_dense(); co, go = O.evaluate(True)
        assert np.abs(Hf - Ho).max() <= 1e-9 * np.abs(Ho).max()
        assert np.abs(gf - go).max() <= 1e-9 * max(1.0, np.abs(go).max()) and abs(cf - co) <= 1e-11 * abs(co)
        G.set_fast_path(0)
        Hg = G.normal_matrix_dense()
        assert np.abs(Hf - Hg).max() <= 1e-10 * np.abs(Hg).max()


SMOOTH_CASES = [
    (abi_smooth, ov) for abi_smooth, ov in [
        (1, dict(depth_type=abi.DEPTH_GRID, depth_grid_x=4, depth_grid_y=4)),
        (0, dict(depth_type=abi.DEPTH_GLOBAL, intr_opt=abi.INTR_SHARED)),
        (2, dict(depth_type=abi.DEPTH_GRID, depth_cubic=1, depth_grid_x=4, depth_grid_y=3, spatial_type=abi.SPATIAL_BILINEAR_GRID, spatial_grid_x=3, spatial_grid_y=2)),
        (3, dict(depth_type=abi.DEPTH_GLOBAL, intr_opt=abi.INTR_FIXED)),
    ]]


@pytest.mark.parametrize("smooth_type,overrides", SMOOTH_CASES, ids=["disparity_laplacian", "euclid_shared", "ratio_bicubic_warp", "log_fixed"])
def test_scene_flow_smoothness_loss(smooth_type, overrides):
    """SceneFlowSmoothnessLoss triplets (lib/PoseOptimizer.cpp:321-423, :1242-1339): CUDA analytic Jacobian vs the oracle's
    literal Jet evaluation, and the LM result with the term enabled."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    sc, cfg, pairs, offs, rec, med = helpers.make_case(smooth_loss_type=smooth_type, **overrides)
    ce, to, tr = sc.triplets(sep=14)
    off_d, nd = helpers.layout_numbers(cfg)
    O = oracle.OracleProblem(cfg); G = solver.Problem(cfg)
    x = helpers.initial_state(sc, cfg, G.stride, off_d, nd)
    for P in (O, G):
        helpers.setup_problem(P, cfg, pairs, offs, rec, med, x); P.set_triplets(ce, to, tr)
    co, go = O.evaluate(True); cg, gg = G.evaluate(True)
    assert abs(co - cg) <= 1e-11 * abs(co)
    assert np.abs(go - gg).max() <= 1e-9 * max(1.0, np.abs(go).max())
    Ho, Hg = O.normal_matrix_dense(), G.normal_matrix_dense()
    assert np.abs(Ho - Hg).max() <= 1e-9 * np.abs(Ho).max()
    opt = abi.default_solve_options(max_iterations=25 if smooth_type == 0 else 50)
    so, sg = O.solve(opt), G.solve(opt)
    assert so.termination == sg.termination and abs(so.final_cost - sg.final_cost) <= 1e-6 * so.final_cost
    assert np.linalg.norm(O.get_state() - G.get_state()) <= 1e-4 * np.linalg.norm(O.get_state())


def test_normalize_depth_bounded():
    """normalizeDepth problem (lib/PoseOptimizer.cpp:992-1147): scale regulariser only, lower bound 0,
    Armijo line search along the projected path."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    sc, cfg, pairs, offs, rec, med = helpers.make_case(depth_type=abi.DEPTH_GLOBAL, depth_lower_bound=1, depth_deform_reg=1.0, focal_reg=0.0)
    res = []
    for cls in (oracle.OracleProblem, solver.Problem):
        P = cls(cfg)
        P.set_frames(np.ones(8, np.uint8), med)
        P.set_constraints(np.zeros((0, 2), np.int32), np.zeros(1, np.int64), np.zeros((0, 6), np.float32))
        P.set_state(sc.identity_state(P.stride, 7, 1))
        s = P.solve(abi.default_solve_options())
        res.append((s.termination, s.iterations, s.final_cost, P.get_state()[:, 7].copy()))
    assert res[0][0] == res[1][0]
    assert abs(res[0][1] - res[1][1]) <= 1
    np.testing.assert_allclose(res[1][3], res[0][3], rtol=1e-6)
    np.testing.assert_allclose(res[1][3], 1.0 / med, rtol=1e-5)


def test_no_cpu_fallback_symbol():
    from robust_cvd_b200 import solver
    L = solver.lib()
    assert L.rcvd_abi_version() == 1


def test_large_grid_uses_global_factor_kernel():
    """npad > 224 takes the non-shared-memory potrf path (config 4's 32x24 grid is npad 784)."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    sc, cfg, pairs, offs, rec, med = helpers.make_case(num_frames=5, sep=6, depth_type=abi.DEPTH_GRID, depth_grid_x=20, depth_grid_y=14)
    O = oracle.OracleProblem(cfg); G = solver.Problem(cfg)
    assert G.stride == 287
    x = helpers.initial_state(sc, cfg, G.stride, 7, 280)
    helpers.setup_problem(O, cfg, pairs, offs, rec, med, x); helpers.setup_problem(G, cfg, pairs, offs, rec, med, x)
    assert G.structure_info()["npad"] == 288
    co, go = O.evaluate(True); cg, gg = G.evaluate(True)
    assert abs(co - cg) <= 1e-11 * abs(co) and np.abs(go - gg).max() <= 1e-9 * max(1.0, np.abs(go).max())
    opt = abi.default_solve_options(max_iterations=30)
    so, sg = O.solve(opt), G.solve(opt)
    assert so.termination == sg.termination and abs(so.final_cost - sg.final_cost) <= 1e-6 * so.final_cost
    assert np.linalg.norm(O.get_state() - G.get_state()) <= 1e-4 * np.linalg.norm(O.get_state())


def test_ragged_and_empty_inputs():
    """Edge cases of BASELINE config 5 (holes: ~50 % valid pixels): ragged pair sizes, pairs without any constraint,
    frames outside the range, a frame that no constraint touches."""
    from oracle import oracle
    from robust_cvd_b200 import solver, synthetic
    sc = synthetic.Scene(8, 128, 96, seed=9)
    cfg = abi.default_config(8, sc.aspect, depth_type=abi.DEPTH_GRID, depth_grid_x=4, depth_grid_y=4)
    pairs, offs, rec = sc.constraints(sep=10, valid_fraction=0.5)
    # drop every constraint of three pairs and of everything touching frame 7; keep the (now empty) pairs in the list
    keep = np.ones(rec.shape[0], bool)
    for p, (a, b) in enumerate(pairs):
        if p in (0, 5, 11) or a == 7 or b == 7:
            keep[offs[p]:offs[p + 1]] = False
        elif p % 4 == 1:                      # ragged: thin some pairs to a handful of constraints
            keep[offs[p] + 3:offs[p + 1]] = False
    counts = np.array([keep[offs[p]:offs[p + 1]].sum() for p in range(len(pairs))]); rec = rec[keep]; offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    assert (counts == 0).sum() >= 5 and counts.max() > 2 * counts[counts > 0].min()
    in_range = np.array([1, 1, 1, 1, 1, 1, 0, 1], np.uint8)       # frame 6 out of range (its pairs are simply not passed by the host)
    sel = np.array([i for i, (a, b) in enumerate(pairs) if a != 6 and b != 6])
    from robust_cvd_b200 import sharding
    pairs2, offs2, rec2 = sharding.take_pairs(pairs, offs, rec, sel)
    med = sc.median_depths()
    res = []
    for cls in (oracle.OracleProblem, solver.Problem):
        P = cls(cfg)
        P.set_frames(in_range, med); P.set_constraints(pairs2, offs2, rec2)
        P.set_state(helpers.initial_state(sc, cfg, P.stride, 7, 16))
        c, g = P.evaluate(True)
        s = P.solve(abi.default_solve_options(max_iterations=40))
        res.append((c, g, s.final_cost, s.termination, P.get_state()))
    assert abs(res[0][0] - res[1][0]) <= 1e-11 * abs(res[0][0])
    assert np.abs(res[0][1] - res[1][1]).max() <= 1e-9 * max(1.0, np.abs(res[0][1]).max())
    assert res[0][3] == res[1][3] and abs(res[0][2] - res[1][2]) <= 1e-6 * res[0][2]
    np.testing.assert_allclose(res[1][4], res[0][4], rtol=1e-4, atol=1e-9)
    x0 = helpers.initial_state(sc, cfg, 23, 7, 16)
    np.testing.assert_array_equal(res[1][4][6], x0[6])               # out-of-range frame untouched
    np.testing.assert_array_equal(res[1][4][7][:6], x0[7][:6])       # pose of the unconstrained frame is not in the problem


def test_dense_constraints_small():
    """matchSeparation = 0 (every valid pixel): 0.3 M constraints on 8 frames, fast kernel vs oracle."""
    from oracle import oracle
    from robust_cvd_b200 import solver
    sc, cfg, pairs, offs, rec, med = helpers.make_case(num_frames=4, sep=0, depth_type=abi.DEPTH_GRID, depth_grid_x=6, depth_grid_y=4)
    assert rec.shape[0] > 100000
    O = oracle.OracleProblem(cfg); G = solver.Problem(cfg)
    x = helpers.initial_state(sc, cfg, G.stride, 7, 24)
    helpers.setup_problem(O, cfg, pairs, offs, rec, med, x); helpers.setup_problem(G, cfg, pairs, offs, rec, med, x)
    co, go = O.evaluate(True); cg, gg = G.evaluate(True)
    assert abs(co - cg) <= 1e-10 * abs(co) and np.abs(go - gg).max() <= 1e-8 * max(1.0, np.abs(go).max())
    Ho, Hg = O.normal_matrix_dense(), G.normal_matrix_dense()
    assert np.abs(Ho - Hg).max() <= 1e-9 * np.abs(Ho).max()


def test_cuda_residuals_vanish_on_reference_python_correspondences():
    """tests/golden/ref_python_geometry.npz (reference utils/geometry.py, see tests/test_oracle.py): the CUDA cost of these exact
    correspondences is zero up to the float32 wire format, for every loss type."""
    import os
    from robust_cvd_b200 import solver
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_python_geometry.npz"))
    W, H = int(g["W"]), int(g["H"]); aspect = float(np.float32(W) / np.float32(H)); n = len(g["px0"])
    x0, y0 = -1.0 + 2.0 * g["px0"] / W, 1.0 - 2.0 * g["py0"] / H
    x1, y1 = -1.0 + 2.0 * g["px1"] / W, 1.0 - 2.0 * g["py1"] / H
    rec = np.concatenate([np.stack([x0, y0, g["depth0"], x1, y1, g["depth1"]], 1), np.stack([x1, y1, g["depth1"], x0, y0, g["depth0"]], 1)]).astype(np.float32)
    for loss in (abi.LOSS_EUCLIDEAN, abi.LOSS_REPRO_DISPARITY, abi.LOSS_REPRO_DEPTH_RATIO, abi.LOSS_REPRO_LOG_DEPTH):
        cfg = abi.default_config(2, aspect, depth_type=abi.DEPTH_IDENTITY, static_loss_type=loss, intr_opt=abi.INTR_PER_FRAME,
                                 scale_reg=0.0, focal_reg=0.0, depth_deform_reg=0.0, spatial_deform_reg=0.0)
        G = solver.Problem(cfg)
        G.set_frames(np.ones(2, np.uint8), np.ones(2))
        G.set_constraints(np.array([[0, 1], [1, 0]], np.int32), np.array([0, n, 2 * n], np.int64), rec)
        x = np.zeros((2, G.stride)); x[:, 0:3] = g["position"]; x[:, 3:6] = g["angle_axis"]; x[:, 6] = g["tan_half_vfov"]
        G.set_state(x.ravel())
        cost = G.evaluate()
        cost = cost[0] if isinstance(cost, tuple) else cost
        assert 0.0 <= cost < 2 * n * 3 * (5e-6) ** 2, (loss, cost)
        G.close()
