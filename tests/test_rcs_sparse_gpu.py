"""GPU parity tests of the block-sparse (supernodal) solver of the reduced camera system -- the path the reference
takes when its dense solver cannot allocate S and it falls back to CLinearSolver_UberBlock with AMD
(LinearSolver_Schur.h:1836-1847). All calls go through the C ABI."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden, rel_err

pytestmark = pytest.mark.gpu

CASES = ["ba_tiny", "ba_tiny_interleaved", "ba_small", "ba_small_hard"]


@pytest.fixture()
def sparse_ctx(ctx):
    from slam_plus_plus_b200 import capi
    ctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    ctx.schur_set_rcs_ordering(None)
    yield ctx
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.schur_set_rcs_ordering(None)


@pytest.mark.parametrize("name", CASES)
def test_slot_increment_vs_reference_1e9(sparse_ctx, name):
    """P1 on the sparse path: the reference's lambda / eta through slot 1 -> dx within 1e-9 of the reference's dx"""
    g, d = load_golden(name)
    sparse_ctx.schur_symbolic(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"])
    dx = sparse_ctx.schur_solve(d["L0.vals"], d["L0.eta"])
    assert rel_err(dx, d["L0.dx"]) < 1e-9
    info = sparse_ctx.schur_get_rcs_info()
    assert info["cameras"] == int((d["L0.col_dims"] == 6).sum())


def test_reference_ordering_is_used_bit_exact(sparse_ctx):
    """the reference's AMD permutation of the Schur complement (golden, made by the reference's own
    CMatrixOrdering::p_BlockOrdering) goes in through spp_schur_set_rcs_ordering and is the elimination order in use"""
    g, d = load_golden("ba_small")
    o = np.load(os.path.join(GOLDEN, "order_ref.npz"))
    ref_order = o["rcs_small.order"]
    sparse_ctx.schur_symbolic(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"])
    # the pattern the golden ordering was computed for is the pattern the library derives
    _, _, pattern = sparse_ctx.schur_get_reduced_system(want_values=False)
    C = pattern.shape[0]
    cp, ri = o["rcs_small.col_ptr"], o["rcs_small.row_idx"]
    ref_pattern = np.zeros((C, C), np.uint8)
    for c in range(C):
        ref_pattern[ri[int(cp[c]):int(cp[c + 1])].astype(np.int64), c] = 1
    assert np.array_equal(pattern, ref_pattern)
    sparse_ctx.schur_set_rcs_ordering(ref_order)
    dx = sparse_ctx.schur_solve(d["L0.vals"], d["L0.eta"])
    info = sparse_ctx.schur_get_rcs_info()
    assert np.array_equal(info["order"], ref_order)
    assert rel_err(dx, d["L0.dx"]) < 1e-9
    with pytest.raises(Exception):
        sparse_ctx.schur_set_rcs_ordering(np.zeros(C, np.uint64))  # not a permutation


@pytest.mark.parametrize("shape,kw", [("mid", {}), ("mid", dict(interleave_ids=True, shuffle_edges=True)),
                                      ("seq", {})])
def test_sparse_vs_dense_step_and_lm(sparse_ctx, shape, kw):
    """same graph, same linearisation: the supernodal path and the dense path give the same increment (1e-10) and the
    same LM trajectory; several supernodes and supernode updates are exercised"""
    from slam_plus_plus_b200 import capi, graphs
    if shape == "seq":
        g = graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    else:
        g = graphs.ba_shape(shape, **kw)
    ctx = sparse_ctx
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    dx_s = ctx.ba_solve_step(10.0)
    info = ctx.schur_get_rcs_info()
    rep_s = ctx.ba_optimize(4, 0.0)
    ctx.schur_set_rcs_solver(capi.RCS_DENSE)
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    dx_d = ctx.ba_solve_step(10.0)
    rep_d = ctx.ba_optimize(4, 0.0)
    assert rel_err(dx_s, dx_d) < 1e-10
    assert rep_s["trace_accepted"] == rep_d["trace_accepted"]
    # two factorisations with different summation orders: the 1e-13 difference of the increments goes through forward-
    # difference Jacobians (delta = 1e-9) at every relinearisation, so the chi2 of later iterations agrees to ~1e-8, not to
    # rounding (SURVEY F3: the reference differs from itself by 1.2e-6 between two builds); north_star asks for 1e-6
    assert abs(rep_s["chi2_final"] - rep_d["chi2_final"]) <= 1e-7 * rep_d["chi2_final"]
    if shape == "seq":
        assert info["supernodes"] > 3 and info["updates"] > 3
        assert info["factor_blocks_stored"] < 0.8 * (400 * 401 // 2)  # it really is sparse


def test_not_positive_definite(sparse_ctx):
    """a non-positive pivot is reported the way the reference's solvers report it (false -> SPP_NOT_POSDEF)"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("small")
    sparse_ctx.ba_set_graph(g)
    sparse_ctx.ba_linearise()
    with pytest.raises(capi.NotPositiveDefinite):
        sparse_ctx.ba_solve_step(-1e9)


def test_full_size_venice_sparse_vs_dense(sparse_ctx):
    """Venice-871 shape: 5226 unknowns through both solvers of the reduced camera system"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("venice871")
    ctx = sparse_ctx
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    dx_s = ctx.ba_solve_step(1.0)
    ctx.schur_set_rcs_solver(capi.RCS_DENSE)
    dx_d = ctx.ba_solve_step(1.0)
    assert rel_err(dx_s, dx_d) < 1e-9


def test_residual_check_small(sparse_ctx):
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("mid")
    sparse_ctx.ba_set_graph(g)
    sparse_ctx.ba_linearise()
    sparse_ctx.ba_solve_step(5.0)
    assert sparse_ctx.schur_get_rcs_residual() < 1e-12
    sparse_ctx.schur_set_rcs_solver(capi.RCS_DENSE)
    sparse_ctx.ba_solve_step(5.0)
    with pytest.raises(capi.SppError):  # only defined for the block-sparse path
        sparse_ctx.schur_get_rcs_residual()


def test_full_size_bal13682_properties(ctx):
    """BASELINE.json configs[3] shape at full size (13 682 cameras, 4.46 M points, 29 M observations; 82 092 unknowns in
    the reduced camera system, factored block-sparse): size-independent properties -- the reduced system is solved to
    rounding (residual on the device), the landmark back-substitution satisfies its block equations on a sample of
    landmarks, and LM steps reduce chi2."""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("bal13682")
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    alpha = 50.0
    dx = ctx.ba_solve_step(alpha)
    info = ctx.schur_get_rcs_info()
    assert info["cameras"] == g.n_cams and info["supernodes"] > 50
    assert info["factor_blocks_stored"] < 0.2 * g.n_cams * (g.n_cams + 1) / 2  # never formed densely
    assert ctx.schur_get_rcs_residual() < 1e-10
    assert np.all(np.isfinite(dx))
    rep = ctx.ba_optimize(3, 0.0)
    assert rep["n_accepted"] >= 1 and rep["chi2_final"] < 0.5 * rep["chi2_initial"]


def test_sparse_path_is_bit_reproducible(sparse_ctx):
    """side streams carry the supernode updates, but all updates into one panel stay on one stream in elimination
    order: two solves of the same system give the same bits (no floating-point atomics anywhere on the path)"""
    from slam_plus_plus_b200 import graphs
    g = graphs.make_ba(600, 40000, 600, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    sparse_ctx.ba_set_graph(g)
    sparse_ctx.ba_linearise()
    a = sparse_ctx.ba_solve_step(3.0)
    b = sparse_ctx.ba_solve_step(3.0)
    info = sparse_ctx.schur_get_rcs_info()
    assert info["supernodes"] > 10 and info["updates"] > 20
    assert np.array_equal(a, b)
    assert sparse_ctx.schur_get_rcs_residual() < 1e-13


def test_bal_sixteenth_against_the_reference_itself(tmp_path):
    """The 1/16 sub-sequence of the BAL-13682 shape that bench.py times the reference on (855 cameras; the full shape
    does not finish on the CPU): the UNMODIFIED reference (oracle/_ref/ref_driver_ba, its dense Schur path) against this
    library with the block-sparse (supernodal) reduced-camera-system solver forced, and with the dense one -- the final
    chi2 of Optimize(2, 0) within the north-star 1e-6, the two device paths within 1e-7 of each other (measured 2e-9:
    their increments differ in the 13th digit, and the second linearisation -- forward differences with delta = 1e-9 --
    amplifies that by 1e9 eps in the Jacobians). The reference's result is taken from its drivers where they are built,
    and from tests/golden/oracle_runs.json where that file records it ("reference_chi2_final"). The same Optimize(2, 0)
    by the CPU oracle (the reference's plain-C restatement), stored there as well, is held to the same bounds on every
    run, so that the test also checks something where neither is available."""
    import json
    import subprocess
    from slam_plus_plus_b200 import capi, graphs, sppio
    g = graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
    with open(os.path.join(GOLDEN, "oracle_runs.json")) as f:
        stored = json.load(f)["bal_sixteenth"]
    chi2_refs = [stored["chi2_final"]] + ([stored["reference_chi2_final"]] if "reference_chi2_final" in stored else [])
    ref_bin = os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "_ref", "ref_driver_ba")
    if os.path.exists(ref_bin):
        gp, dp = str(tmp_path / "g.bin"), str(tmp_path / "ref.dump")
        sppio.write_graph(gp, g)
        subprocess.run([ref_bin, "time", gp, dp, "2", "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        chi2_refs.append(float(sppio.read_dump(dp)["chi2"][0]))
    chi2 = {}
    for mode in (capi.RCS_SPARSE, capi.RCS_DENSE):
        ctx = capi.Context(0)
        ctx.schur_set_rcs_solver(mode)
        ctx.ba_set_graph(g)
        rep = ctx.ba_optimize(2, 0.0)
        chi2[mode] = rep["chi2_final"]
        if mode == capi.RCS_SPARSE:
            info = ctx.schur_get_rcs_info()
            assert info["cameras"] == g.n_cams and info["supernodes"] >= 1
        ctx.close()
    for chi2_ref in chi2_refs:
        assert abs(chi2[capi.RCS_SPARSE] - chi2_ref) <= 1e-6 * chi2_ref, (chi2, chi2_ref)
        assert abs(chi2[capi.RCS_DENSE] - chi2_ref) <= 1e-6 * chi2_ref, (chi2, chi2_ref)
        assert abs(chi2[capi.RCS_SPARSE] - chi2[capi.RCS_DENSE]) <= 1e-7 * chi2_ref
