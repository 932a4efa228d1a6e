"""The drop-in test: the UNMODIFIED reference LM solver (oracle/_ref/ref_driver_dropin, compiled from
/root/reference in the build container) with CLinearSolver_Schur_B200 (include/slam_b200/) plugged into its
linear-solver slot -- i.e. the reference's own edges, Jacobians and LM loop, our Schur / Cholesky / back-substitution
through the C ABI. Since the linearisation is the reference's own, the whole LM trace must reproduce the
pure-reference golden run to the accuracy of the linear solves (1e-9)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden, rel_err

pytestmark = pytest.mark.gpu

BIN = os.path.join(ROOT, "oracle", "_ref", "ref_driver_dropin")


REF = os.path.join(ROOT, "oracle", "_ref", "ref_driver_ba")


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    return oracle


def _schur_slot(ctx, g):
    """The B200 Schur solver in the linear-solver slot of the oracle's LM loop (the reference's loop restated in C,
    oracle/spp_oracle.c): the damped lambda in the reference's block layout and eta in vertex order go through
    spp_schur_symbolic / spp_schur_solve, as CLinearSolver_Schur_B200 hands them over."""
    from slam_plus_plus_b200 import capi
    oracle = _oracle()
    loc, cam = g.vertex_local_index(), g.vtype == 0
    state = {}

    def solve(U, V, W, gc, gp, alpha):
        Ud = (U.reshape(-1, 6, 6) + alpha * np.eye(6)).reshape(-1, 36)
        Vd = (V.reshape(-1, 3, 3) + alpha * np.eye(3)).reshape(-1, 9)
        col_dims, col_ptr, row_idx, vals = oracle.lambda_blocks_to_reference_layout(g, Ud, Vd, W)
        if "pattern" not in state:
            ctx.schur_symbolic(col_dims, col_ptr, row_idx)
            state["pattern"] = True
        eta = np.concatenate([gc[loc[v]] if cam[v] else gp[loc[v]] for v in range(g.n_vertices)])
        try:
            dx = ctx.schur_solve(vals, eta)
        except capi.NotPositiveDefinite:
            return 1, None, None
        off = np.concatenate([[0], np.cumsum(np.where(cam, 6, 3))])
        dxc = np.stack([dx[off[v]:off[v + 1]] for v in np.flatnonzero(cam)])
        dxp = np.stack([dx[off[v]:off[v + 1]] for v in np.flatnonzero(~cam)])
        return 0, dxc[np.argsort(loc[cam])], dxp[np.argsort(loc[~cam])]
    return solve


def _compare_traces(tr, tg, tol_chi2, tol_first=None):
    """LM traces [alpha, chi2_last, chi2, ., accepted, .] of two runs; tg is the reference one. tol_first, if given,
    is the (tighter) chi2 tolerance of the first step, where both runs linearise at the same state."""
    # damping history: alpha_{k+1} = alpha_k * max(1/3, 1 - (2 rho - 1)^3) with rho = (chi2_last - chi2) / denominator
    # (LM.h:204-223). chi2 is reproduced to tol_chi2 RELATIVE TO CHI2, so rho carries a relative error of
    # tol_chi2 * chi2 / |chi2_last - chi2| (large once the steps stop reducing chi2), and |d factor / d rho| <= 6 with
    # factor >= 1/3 turns that into <= 18x as much in alpha. The tolerance accumulates over the steps.
    tol_alpha = 100 * tol_chi2
    for k in range(min(len(tr), len(tg))):
        if abs(tg[k, 1] - tg[k, 2]) <= max(tol_chi2, 1e-9) * tg[k, 1]:
            break  # chi2 no longer changes: the accept / reject decision is rounding noise from here on
        assert int(tr[k, 4]) == int(tg[k, 4])
        assert abs(tr[k, 2] - tg[k, 2]) <= (tol_first if (k == 0 and tol_first) else tol_chi2) * tg[k, 2]
        assert abs(tr[k, 0] - tg[k, 0]) <= tol_alpha * tg[k, 0]
        tol_alpha += 20 * tol_chi2 * tg[k, 1] / abs(tg[k, 1] - tg[k, 2])


@pytest.mark.parametrize("name", ["ba_tiny", "ba_tiny_interleaved", "ba_small", "ba_small_hard"])
def test_reference_lm_with_b200_linear_solver(name, tmp_path):
    g, d = load_golden(name)
    if not os.path.exists(BIN) or not os.path.exists(REF):
        # without the reference's drivers: its LM loop as the oracle restates it, the B200 Schur solver in its slot,
        # against the committed golden run of the reference on this graph (the same bounds as below)
        from slam_plus_plus_b200 import capi
        ctx = capi.Context(0)
        try:
            r = _oracle().ba_optimize(g, int(d["max_iter"][0]), 0.0, linear_solver=_schur_slot(ctx, g))
        finally:
            ctx.close()
        assert r["status"] == 0
        assert abs(r["chi2_initial"] - d["chi2_0"][0]) <= 1e-11 * d["chi2_0"][0]
        _compare_traces(r["trace"], d["lm_trace"].reshape(-1, 6), 2e-5)
        assert abs(r["chi2_final"] - d["chi2"][0]) <= 1e-6 * d["chi2"][0]
        loc = g.vertex_local_index()
        states = np.concatenate([r["cams"][loc[v]] if g.vtype[v] == 0 else r["pts"][loc[v]] for v in range(g.n_vertices)])
        assert rel_err(states, d["states"]) < 1e-4
        return
    from slam_plus_plus_b200 import sppio
    gp, dp, rp = str(tmp_path / "g.bin"), str(tmp_path / "d.dump"), str(tmp_path / "r.dump")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    n_it = str(int(d["max_iter"][0]))
    subprocess.run([BIN, gp, dp, n_it, "0"], check=True, stdout=subprocess.DEVNULL, env=env)
    # the pure reference on THIS machine: its forward-difference Jacobians (delta = 1e-9) amplify last-bit libm
    # differences between host CPUs to ~1e-6 (SURVEY F3), so the 1e-9 comparison must not cross machines
    subprocess.run([REF, "dump", gp, rp, n_it, "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
    r, ref = sppio.read_dump(dp), sppio.read_dump(rp)
    assert abs(r["chi2_0"][0] - ref["chi2_0"][0]) <= 1e-13 * ref["chi2_0"][0]
    # First step: same state, same Jacobians, so chi2 after the step shows the accuracy of the linear solve alone
    # (1e-9). From the second step on the two runs linearise at states that differ in the last bits (our increment
    # agrees with the reference's to ~1e-13, not bitwise), and the reference's forward-difference Jacobians turn
    # that into ~1e-7 relative noise in J (rounding of h(x) over delta = 1e-9, SURVEY F3): the intermediate chi2 of
    # far-from-converged steps then agree at that noise floor (2e-5, as in test_ba_gpu.py; measured 1.5e-6 on
    # ba_small_hard, whose chi2 falls from 1e9 to 2.5e3), the final chi2 within the north-star bound of 1e-6.
    _compare_traces(r["lm_trace"].reshape(-1, 6), ref["lm_trace"].reshape(-1, 6), 2e-5, tol_first=1e-9)
    assert abs(r["chi2"][0] - ref["chi2"][0]) <= 1e-6 * ref["chi2"][0]
    # converged problems end with noise-decided accept / reject steps along nearly flat directions: the states
    # agree less tightly than chi2 does
    assert rel_err(r["states"], ref["states"]) < 1e-4
    # and against the committed golden run (another machine): FD noise floor
    assert abs(r["chi2_0"][0] - d["chi2_0"][0]) <= 1e-11 * d["chi2_0"][0]
    _compare_traces(r["lm_trace"].reshape(-1, 6), d["lm_trace"].reshape(-1, 6), 2e-5)
    assert abs(r["chi2"][0] - d["chi2"][0]) <= 1e-6 * d["chi2"][0]


# ---- pose graphs: CLinearSolver_UberBlock_B200 in the reference's Gauss-Newton solver --------------------------------

BIN_POSE = os.path.join(ROOT, "oracle", "_ref", "ref_driver_dropin_pose")
REF_POSE = os.path.join(ROOT, "oracle", "_ref", "ref_driver_pose")


def _block_cholesky_slot(ctx, B):
    """The B200 block Cholesky in the linear-solver slot of the oracle's Gauss-Newton loop: lambda as upper
    block-triangular CSC of B x B column-major blocks (the reference's layout) through spp_chol_symbolic /
    spp_chol_solve, as CLinearSolver_UberBlock_B200 hands it over."""
    from slam_plus_plus_b200 import capi
    state = {}

    def solve(lam, eta):
        n = lam.shape[0] // B
        blocks = lam.reshape(n, B, n, B).transpose(0, 2, 1, 3)  # [row block, column block]
        nz = np.triu(np.abs(blocks).max(axis=(2, 3)) > 0)
        rows, cols = np.nonzero(nz.T)  # column-major traversal: (column, row) pairs, rows ascending per column
        col_ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.uint64)
        row_idx = cols.astype(np.uint64)
        if state.get("pattern") is None or not np.array_equal(state["pattern"], nz):
            ctx.chol_symbolic(B, col_ptr, row_idx)
            state["pattern"] = nz
        vals = blocks[cols, rows].transpose(0, 2, 1).ravel()  # column-major blocks
        try:
            return 0, ctx.chol_solve(vals, eta)
        except capi.NotPositiveDefinite:
            return 1, None
    return solve


@pytest.mark.parametrize("name", ["se2_tiny", "se2_small", "se3_tiny", "se3_small"])
def test_reference_gauss_newton_with_b200_block_cholesky(name, tmp_path):
    """the UNMODIFIED reference (its vertices, edges, Jacobians, GN loop and AMD ordering) with the GPU block Cholesky
    in its linear-solver slot reproduces the pure-reference run on the same machine"""
    from test_pose_cpu import load_pose_golden
    g, d = load_pose_golden(name)
    tol = 1e-9 if name.startswith("se2") else 1e-5  # see below
    if not os.path.exists(BIN_POSE) or not os.path.exists(REF_POSE):
        # without the reference's drivers: its Gauss-Newton loop as the oracle restates it, the B200 block Cholesky in
        # its slot, against the committed golden run of the reference on this graph
        from slam_plus_plus_b200 import capi
        ctx = capi.Context(0)
        try:
            r = _oracle().pose_optimize(g, int(d["max_iter"][0]), 0.0, linear_solver=_block_cholesky_slot(ctx, g.dim))
        finally:
            ctx.close()
        assert r["status"] == 0
        assert abs(r["chi2_initial"] - d["chi2_0"][0]) <= 1e-12 * d["chi2_0"][0]
        assert abs(r["chi2_final"] - d["chi2"][0]) <= tol * d["chi2"][0]
        return
    from slam_plus_plus_b200 import sppio
    gp, dp, rp = str(tmp_path / "g.bin"), str(tmp_path / "d.dump"), str(tmp_path / "r.dump")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    n_it = str(int(d["max_iter"][0]))
    subprocess.run([BIN_POSE, gp, dp, n_it, "0"], check=True, stdout=subprocess.DEVNULL, env=env)
    subprocess.run([REF_POSE, "time", gp, rp, n_it, "0"], check=True, stdout=subprocess.DEVNULL, env=env)
    r, ref = sppio.read_dump(dp), sppio.read_dump(rp)
    assert abs(r["chi2_0"][0] - d["chi2_0"][0]) <= 1e-12 * d["chi2_0"][0]
    # SE(2): analytic Jacobians, the whole trajectory follows to the accuracy of the linear solves; SE(3): the
    # reference's forward-difference Jacobians amplify the last-bit differences of the increments (see test_pose_gpu.py)
    assert abs(r["chi2"][0] - ref["chi2"][0]) <= tol * ref["chi2"][0]
    assert abs(r["chi2"][0] - d["chi2"][0]) <= tol * d["chi2"][0]


# ---- slot 3: CNonlinearSolver_Lambda_LM_B200 in place of the reference's nonlinear solver ----------------------------

BIN_LM = os.path.join(ROOT, "oracle", "_ref", "ref_driver_dropin_lm")


def _batch_b200_and_oracle(g, with_marginals=False):
    """Optimize(5, 0) on the whole graph by the library's own LM solver (what CNonlinearSolver_Lambda_LM_B200 forwards
    to) and by the oracle's restatement of the reference's CNonlinearSolver_Lambda_LM; states in vertex order"""
    from slam_plus_plus_b200 import capi
    loc, cam = g.vertex_local_index(), g.vtype == 0
    ctx = capi.Context(0)
    try:
        ctx.ba_set_graph(g)
        rep = ctx.ba_optimize(5, 0.0)
        cams, pts = ctx.ba_get_states()
        margs = ctx.ba_marginals(0.0) if with_marginals else None
    finally:
        ctx.close()
    r = _oracle().ba_optimize(g, 5, 0.0)
    b = {"chi2_trace": [rep["chi2_initial"], rep["chi2_final"]],
         "states": np.concatenate([cams[loc[v]] if cam[v] else pts[loc[v]] for v in range(g.n_vertices)]), "margs": margs}
    o = {"chi2_trace": [r["chi2_initial"], r["chi2_final"]],
         "states": np.concatenate([r["cams"][loc[v]] if cam[v] else r["pts"][loc[v]] for v in range(g.n_vertices)])}
    return b, o


@pytest.mark.parametrize("mode,name", [("batch", "ba_tiny_interleaved"), ("batch", "ba_small"), ("incremental", "ba_small"),
                                       ("incremental", "ba_small_hard")])
def test_reference_system_with_b200_nonlinear_solver(mode, name, tmp_path):
    """the UNMODIFIED reference's CFlatSystem / vertices / edges with the solver TYPE swapped for
    CNonlinearSolver_Lambda_LM_B200 (everything from the linearisation on runs on the GPU), against the reference's own
    CNonlinearSolver_Lambda_LM on the same machine; "incremental" = Optimize() at a marker every 6 cameras on a growing,
    append-only system (the application's CParseLoop_ConsistencyMarker behaviour). Without the reference's drivers
    neither the adapter nor the reference's system can be built: the batch cases then compare only the solver underneath
    the adapter (spp_ba_optimize) with the oracle's restatement of the reference's solver."""
    if not os.path.exists(BIN_LM) and mode == "batch":
        # without the reference's drivers: the library's solver against the oracle's restatement of the reference's
        # LM solver on the same graph, with the bounds below
        b, r = _batch_b200_and_oracle(load_golden(name)[0])
        tb, tr = b["chi2_trace"], r["chi2_trace"]
        assert abs(tb[0] - tr[0]) <= 1e-11 * tr[0]
        assert abs(tb[-1] - tr[-1]) <= 1e-6 * tr[-1]
        assert len(b["states"]) == len(r["states"]) > 6
        assert rel_err(b["states"], r["states"]) < 1e-4
        return
    if not os.path.exists(BIN_LM):
        pytest.skip("oracle/_ref/ref_driver_dropin_lm not built (it needs the reference's sources in SPP_REFERENCE at build time)")
    from slam_plus_plus_b200 import sppio
    g, d = load_golden(name)
    gp = str(tmp_path / "g.bin")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = {}
    for impl in ("b200", "ref"):
        dp = str(tmp_path / (impl + ".dump"))
        subprocess.run([BIN_LM, impl, mode, gp, dp, "5", "0", "6"], check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL, env=env)
        out[impl] = sppio.read_dump(dp)
    b, r = out["b200"], out["ref"]
    assert int(b["n_vertices"][0]) == int(r["n_vertices"][0]) and int(b["n_edges"][0]) == int(r["n_edges"][0])
    tb, tr = b["chi2_trace"], r["chi2_trace"]
    assert len(tb) == len(tr)
    if mode == "batch":
        assert abs(tb[0] - tr[0]) <= 1e-11 * tr[0]  # chi2 of the untouched system: no Jacobians involved
    # chi2 after every Optimize(): FD-noise floor in between (the two runs linearise with forward differences on
    # different libm implementations), north-star bound on the final value
    for a, c in zip(tb[:-1], tr[:-1]):
        assert abs(a - c) <= 2e-5 * max(c, 1.0)
    assert abs(tb[-1] - tr[-1]) <= 1e-6 * tr[-1]
    assert len(b["states"]) == len(r["states"]) > 6
    assert rel_err(b["states"], r["states"]) < 1e-4


@pytest.mark.parametrize("name,period", [("ba_small", 6), ("ba_small_hard", 4)])
def test_b200_nonlinear_solver_incremental_policy(name, period, tmp_path):
    """no markers: both solver types are built with TIncrementalSolveSetting(solve::nonlinear, frequency::Every(period))
    and decide inside Incremental_Step() when to solve -- the adapter inherits the reference's own t_Incremental_Step
    (NonlinearSolver_Base.h:557-622: vertex-counted periods, a solve only after a loop closure). The solves must happen
    after the same edges, and the final chi2 must agree to the north-star bound."""
    if not os.path.exists(BIN_LM):
        pytest.skip("oracle/_ref/ref_driver_dropin_lm not built (it needs the reference's sources in SPP_REFERENCE at build time)")
    from slam_plus_plus_b200 import sppio
    g, d = load_golden(name)
    gp = str(tmp_path / "g.bin")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = {}
    for impl in ("b200", "ref"):
        dp = str(tmp_path / (impl + ".dump"))
        subprocess.run([BIN_LM, impl, "periodic", gp, dp, "5", "0", str(period)], check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL, env=env)
        out[impl] = sppio.read_dump(dp)
    b, r = out["b200"], out["ref"]
    assert len(r["solve_edges"]) >= 3
    assert list(b["solve_edges"]) == list(r["solve_edges"])  # the same solves, after the same edges
    assert abs(b["chi2_trace"][-1] - r["chi2_trace"][-1]) <= 1e-6 * r["chi2_trace"][-1]
    assert rel_err(b["states"], r["states"]) < 1e-4


@pytest.mark.parametrize("name", ["ba_tiny", "ba_small"])
def test_b200_nonlinear_solver_marginals(name, tmp_path):
    """the marginals policy of the reference's solver interface (TMarginalsComputationPolicy, mpart_Diagonal) on the
    swapped-in solver type: r_MarginalCovariance().r_SparseMatrix() after Optimize() against the reference's own, up to
    the variance of the unobservable scale (tests/test_marginals_cpu.py explains the one-scalar fit). Without the
    reference's drivers only the solver and marginals underneath the adapter (spp_ba_optimize, spp_ba_marginals) are
    compared, with the oracle's restatement of the reference's solver and marginals."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    from conftest import gauge_fit_residual, weakest_modes
    from slam_plus_plus_b200 import sppio
    g, d = load_golden(name)
    assert g.vtype[0] == 0  # the unary factor sits on a camera: one gauge mode
    if not os.path.exists(BIN_LM):
        # without the reference's drivers: the library's solver and marginals against the oracle's restatement of the
        # reference's LM solver and of its block-diagonal marginals, with the bounds below
        b, r = _batch_b200_and_oracle(g, with_marginals=True)
        assert rel_err(b["states"], r["states"]) < 1e-4
        cb, pb = b["margs"]
        loc, off = g.vertex_local_index(), 0
        for v in range(g.n_vertices):  # the graph at the oracle's final states: its marginals and the gauge mode
            k = 6 if g.vtype[v] == 0 else 3
            (g.cams if k == 6 else g.pts)[loc[v], :k] = r["states"][off:off + k]
            off += k
        cr, pr, L = oracle.ba_marginals(g)
        assert cb.shape == cr.shape == (g.n_cams, 6, 6) and pb.shape == pr.shape == (g.n_pts, 3, 3)
        rc, rp, _ = gauge_fit_residual(g.n_cams, cb, pb, cr, pr, weakest_modes(L, 1))
        print(f"{name}: marginals after the gauge fit: cameras {rc:.3g}, points {rp:.3g}")
        assert rc < 1e-4 and rp < 1e-3
        return
    gp = str(tmp_path / "g.bin")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1", SPP_DROPIN_MARGS="1")
    out = {}
    for impl in ("b200", "ref"):
        dp = str(tmp_path / (impl + ".dump"))
        subprocess.run([BIN_LM, impl, "batch", gp, dp, "5", "0", "6"], check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL, env=env, cwd=str(tmp_path))  # the reference writes marginals.txt
        out[impl] = sppio.read_dump(dp)
    b, r = out["b200"], out["ref"]
    assert len(b["states"]) == len(r["states"]) == 6 * g.n_cams + 3 * g.n_pts
    assert rel_err(b["states"], r["states"]) < 1e-4
    cb, pb = b["cam_cov"].reshape(-1, 6, 6), b["pt_cov"].reshape(-1, 3, 3)
    cr, pr = r["cam_cov"].reshape(-1, 6, 6), r["pt_cov"].reshape(-1, 3, 3)
    assert cb.shape == cr.shape == (g.n_cams, 6, 6) and pb.shape == pr.shape == (g.n_pts, 3, 3)
    loc, off = g.vertex_local_index(), 0
    for v in range(g.n_vertices):  # the graph at the final states, for the gauge mode of its lambda
        k = 6 if g.vtype[v] == 0 else 3
        (g.cams if k == 6 else g.pts)[loc[v], :k] = b["states"][off:off + k]
        off += k
    _, _, L = oracle.ba_marginals(g)
    rc, rp, _ = gauge_fit_residual(g.n_cams, cb, pb, cr, pr, weakest_modes(L, 1))
    print(f"{name}: marginals after the gauge fit: cameras {rc:.3g}, points {rp:.3g}")
    assert rc < 1e-4 and rp < 1e-3  # measured 8e-6 / 1.3e-5


# ---- slot 3 for pose graphs: CNonlinearSolver_Lambda_B200 in place of the reference's Gauss-Newton solver ------------

BIN_GN = os.path.join(ROOT, "oracle", "_ref", "ref_driver_dropin_gn")


@pytest.mark.parametrize("kind,mode", [("se2", "batch"), ("se2", "incremental"), ("se3", "batch"), ("se3", "incremental")])
def test_reference_pose_system_with_b200_nonlinear_solver(kind, mode, tmp_path):
    """the UNMODIFIED reference's CFlatSystem of CVertexPose2D/3D + CEdgePose2D/3D with the solver TYPE swapped for
    CNonlinearSolver_Lambda_B200, against the reference's own CNonlinearSolver_Lambda on the same machine. "incremental"
    = slam_app's feeding order: edges sorted by their later pose, new poses initialised by the edge constructors on the
    host, Incremental_Step() after every edge with a nonlinear solve every 10 new vertices once a loop has closed. The
    marginals policy (mpart_Diagonal) is on: r_MarginalCovariance() is compared as well."""
    if not os.path.exists(BIN_GN):
        pytest.skip("oracle/_ref/ref_driver_dropin_gn not built (it needs the reference's sources in SPP_REFERENCE at build time)")
    from slam_plus_plus_b200 import graphs, sppio
    # SE(3): the graph of the golden se3_tiny (tests/golden/make_golden.py) -- the reference's robust SE(3) Gauss-Newton
    # does not settle (w^2 / w gradient weights, BaseTypes_Binary.h:820-843): on a sphere with small noise its chi2 after
    # 5 / 10 / 20 / 40 iterations is 352.4 / 347.5 / 346.6 / 349.1, so only graphs on which it converges can be compared
    g = (graphs.make_manhattan(300, 150, seed=21) if kind == "se2" else
         graphs.make_sphere(n_rings=5, n_per_ring=8, seed=3, sigma_t=0.03, sigma_r=0.005, radius=5.0))
    gp = str(tmp_path / "g.bin")
    sppio.write_graph(gp, g)
    env = dict(os.environ, OMP_NUM_THREADS="1", SPP_DROPIN_MARGS="1")
    out = {}
    for impl in ("b200", "ref"):
        dp = str(tmp_path / (impl + ".dump"))
        subprocess.run([BIN_GN, impl, mode, gp, dp, "5", "0", "10"], check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL, env=env, cwd=str(tmp_path))
        out[impl] = sppio.read_dump(dp)
    b, r = out["b200"], out["ref"]
    n, dim = g.poses.shape
    assert int(b["n_vertices"][0]) == int(r["n_vertices"][0]) == n and int(b["n_edges"][0]) == int(r["n_edges"][0])
    assert len(b["states"]) == len(r["states"]) == n * dim
    # SE(2): analytic Jacobians, the two runs differ by rounding times the conditioning of the solves; SE(3): forward
    # differences (delta = 1e-9) on two libm implementations -- the FD noise floor of the other SE(3) tests
    tol_chi2, tol_state, tol_cov = (1e-9, 1e-7, 1e-6) if kind == "se2" else (1e-5, 1e-4, 1e-3)
    print(f"{kind} {mode}: chi2 {b['chi2_trace']} vs {r['chi2_trace']}, states {rel_err(b['states'], r['states']):.3g}, "
          f"cov {rel_err(b['cov'], r['cov']):.3g}")
    for a, c in zip(b["chi2_trace"], r["chi2_trace"]):
        assert abs(a - c) <= tol_chi2 * max(c, 1.0)
    if kind == "se2":
        assert rel_err(b["states"], r["states"]) < tol_state
    else:
        # SE(3): the identity prior on pose 0 against edge information of 1e3 .. 4e4 leaves a rigid motion of the whole
        # graph almost free (cond 1e10), and an axis-angle vector near pi has two representations: compare what the
        # edges see, the relative poses of consecutive vertices
        def relative_poses(st):
            st = st.reshape(n, 6)
            R = graphs._axis_angle_to_rotmat(st[:, 3:])
            return (np.einsum("nji,njk->nik", R[:-1], R[1:]), np.einsum("nji,nj->ni", R[:-1], st[1:, :3] - st[:-1, :3]))
        (Rb, tb), (Rr, tr) = relative_poses(b["states"]), relative_poses(r["states"])
        assert np.abs(Rb - Rr).max() < 1e-5 and np.abs(tb - tr).max() < 1e-4  # measured 1e-7 / 1.1e-5 (FD noise floor)
        print(f"   relative poses: rotation {np.abs(Rb - Rr).max():.3g}, translation {np.abs(tb - tr).max():.3g}")
    assert b["cov"].shape == r["cov"].shape == (n * dim * dim,)
    assert rel_err(b["cov"], r["cov"]) < tol_cov


def test_incremental_manhattan3500_matches_reference_solve_for_solve(tmp_path):
    """BASELINE.json configs[0] shape fed edge by edge (slam_app's policy: a nonlinear solve of at most 5 iterations with
    the 0.01 step-norm threshold every 10 new vertices once a loop has closed): with the threshold in play every early
    exit is a decision, so the adapter must reproduce the reference's SEQUENCE of linear solves -- the printed step norms
    of all of them (4 decimals, the reference's verbose output) -- and the final chi2 to 1e-9 (analytic SE(2) Jacobians:
    no forward-difference noise). Round 1 lost two solves here: a root front covering the whole (still small) matrix read
    factor blocks that are never formed for root columns (sparse_chol.cu, block_update)."""
    if not os.path.exists(BIN_GN):
        pytest.skip("oracle/_ref/ref_driver_dropin_gn not built (it needs the reference's sources in SPP_REFERENCE at build time)")
    from slam_plus_plus_b200 import graphs, sppio
    g = graphs.make_manhattan(fill_loops=True)
    gp = str(tmp_path / "g.bin")
    sppio.write_graph(gp, g)
    norms, chi2 = {}, {}
    for impl in ("b200", "ref"):
        dp = str(tmp_path / (impl + ".dump"))
        r = subprocess.run([BIN_GN, impl, "incremental", gp, dp, "5", "0.01", "10"], check=True, capture_output=True, text=True,
                           env=dict(os.environ, OMP_NUM_THREADS="1", SPP_REF_VERBOSE="1"), cwd=str(tmp_path))
        norms[impl] = [l.split(":")[1].strip() for l in r.stdout.splitlines() if l.startswith("residual norm:")]
        chi2[impl] = float(sppio.read_dump(dp)["chi2_trace"][-1])
        assert "Cholesky failed" not in r.stderr
    assert len(norms["b200"]) == len(norms["ref"]) > 500
    assert norms["b200"] == norms["ref"]
    assert abs(chi2["b200"] - chi2["ref"]) <= 1e-9 * chi2["ref"]
