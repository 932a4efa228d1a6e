"""Marginal covariances through the block-sparse (supernodal) reduced camera system and its selected inversion
(spp_ba_marginals_sparse / spp_schur_marginals_sparse, csrc/selinv.cu + csrc/marginals.cu): against a float64 dense
inverse of the same lambda, against the reference's own marginals, against the dense-path marginals on systems with
many supernodes, and on the full BAL-13682 shape, which has no dense path. All calls go through the C ABI."""
import numpy as np
import pytest

from conftest import gauge_fit_residual, lambda_to_dense, load_golden, load_margs_golden, rel_err, weakest_modes

pytestmark = pytest.mark.gpu

CASES = ["ba_tiny", "ba_tiny_interleaved", "ba_small", "ba_small_hard"]


@pytest.fixture()
def sctx(ctx):
    from slam_plus_plus_b200 import capi
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.schur_set_rcs_ordering(None)
    yield ctx
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.schur_set_rcs_ordering(None)


def _blocks_of_inverse(A, dims):
    Ai = np.linalg.inv(A)
    base = np.concatenate([[0], np.cumsum(dims)])
    six = [Ai[base[i]:base[i] + 6, base[i]:base[i] + 6] for i in range(len(dims)) if dims[i] == 6]
    three = [Ai[base[i]:base[i] + 3, base[i]:base[i] + 3] for i in range(len(dims)) if dims[i] == 3]
    return np.stack(six), np.stack(three)


def _max_lambda_diag(ctx):
    """max of the diagonal of lambda from its block list (the diagonal block is the last of every block column)"""
    col_dims, col_ptr, row_idx, vals, _ = ctx.ba_get_lambda()
    dims = col_dims.astype(np.int64)
    ptr = col_ptr.astype(np.int64)
    col_of = np.repeat(np.arange(len(dims)), np.diff(ptr))
    sizes = dims[row_idx.astype(np.int64)] * dims[col_of]
    off = np.concatenate([[0], np.cumsum(sizes)])
    m = 0.0
    for c in range(len(dims)):
        k = ptr[c + 1] - 1
        d = dims[c]
        blk = vals[off[k]:off[k] + d * d].reshape(d, d)
        m = max(m, float(np.diag(blk).max()))
    return m


@pytest.mark.parametrize("name", CASES)
def test_slot_sparse_marginals_vs_dense_inverse(sctx, name):
    """the reference's own lambda through slot 1, alpha = 0 and 0.5: block diagonal of the inverse to 1e-9"""
    g, d = load_golden(name)
    dims = d["L0.col_dims"].astype(np.int64)
    sctx.schur_symbolic(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"])
    sctx.schur_solve(d["L0.vals"], d["L0.eta"])
    A = lambda_to_dense(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"], d["L0.vals"])
    for alpha in (0.0, 0.5):
        cc, pc = sctx.schur_marginals_sparse(alpha)
        rc, rp = _blocks_of_inverse(A + alpha * np.eye(A.shape[0]), dims)
        assert rel_err(cc, rc) < 1e-9 and rel_err(pc, rp) < 1e-9, (alpha, rel_err(cc, rc), rel_err(pc, rp))
        assert np.array_equal(cc, cc.transpose(0, 2, 1))  # read through the upper triangle: exactly symmetric


@pytest.mark.parametrize("name", ["margs_tiny", "margs_tiny_interleaved", "margs_small"])
def test_ba_sparse_marginals_vs_reference(sctx, name):
    """alpha = 0 at the reference's final states against the reference's Schur_Marginals output (gauge fitted)"""
    g, d = load_margs_golden(name)
    sctx.ba_set_graph(g)
    cc, pc = sctx.ba_marginals_sparse(0.0)
    assert cc.shape == d["cam_cov"].shape and pc.shape == d["pt_cov"].shape
    col_dims, col_ptr, row_idx, vals, _ = sctx.ba_get_lambda()
    A = lambda_to_dense(col_dims, col_ptr, row_idx, vals)
    dims = np.asarray(col_dims, np.int64)
    base = np.concatenate([[0], np.cumsum(dims)])
    perm = np.concatenate([np.arange(base[i], base[i + 1]) for i in np.flatnonzero(dims == 6)] +
                          [np.arange(base[i], base[i + 1]) for i in np.flatnonzero(dims == 3)])
    L = A[np.ix_(perm, perm)]
    m = 1 if g.vtype[0] == 0 else 4
    rc, rp, k = gauge_fit_residual(g.n_cams, cc, pc, d["cam_cov"], d["pt_cov"], weakest_modes(L, m))
    assert rc < 1e-4 and rp < 1e-3, (rc, rp, k)
    assert np.all(np.einsum("kii->ki", cc) > 0) and np.all(np.einsum("kii->ki", pc) > 0)


def _many_supernode_graph(shape):
    from slam_plus_plus_b200 import graphs
    if shape == "seq":
        return graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    if shape == "bal16":  # the 1/16 sub-sequence of the BAL-13682 shape (855 cameras)
        return graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
    if shape == "mid_interleaved":
        return graphs.ba_shape("mid", interleave_ids=True, shuffle_edges=True)
    return graphs.ba_shape(shape)


@pytest.mark.parametrize("shape", ["mid", "mid_interleaved", "seq", "bal16"])
def test_sparse_vs_dense_marginals_many_supernodes(sctx, shape):
    """the supernodal selected inversion against the dense inverse path on the same linearisation"""
    g = _many_supernode_graph(shape)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    cs, ps = sctx.ba_marginals_sparse(alpha)
    info = sctx.schur_get_rcs_info()
    cd, pd = sctx.ba_marginals(alpha)
    assert rel_err(cs, cd) < 1e-9 and rel_err(ps, pd) < 1e-9, (rel_err(cs, cd), rel_err(ps, pd))
    if shape == "seq":
        assert info["supernodes"] > 3 and info["updates"] > 3, info
    if shape == "bal16":  # a few wide supernodes: the widest (>= 6C / supernodes >= 1024 columns) is factored by k_chol_dataflow
        assert info["supernodes"] >= 2 and info["updates"] >= 1, info
        assert 6 * info["cameras"] / info["supernodes"] >= 1024, info


def test_venice_sparse_vs_dense_marginals(sctx):
    from slam_plus_plus_b200 import graphs
    g = graphs.ba_shape("venice871")
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    cs, ps = sctx.ba_marginals_sparse(alpha)
    cd, pd = sctx.ba_marginals(alpha)
    assert rel_err(cs, cd) < 1e-9 and rel_err(ps, pd) < 1e-9, (rel_err(cs, cd), rel_err(ps, pd))


def test_sparse_marginals_reproducible_and_state(sctx):
    """two calls give the same bits; solves and LM after the marginals give the bits they give without them; a negative
    damping is reported as a non-positive pivot; the residual check of the last solve is refused after the marginals"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    sctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    # without the marginals
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    max_diag = _max_lambda_diag(sctx)
    dx0 = sctx.ba_solve_step(3.0)
    rep0 = sctx.ba_optimize(3, 0.0)
    # with them
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    a = sctx.ba_marginals_sparse(1.0)
    b = sctx.ba_marginals_sparse(1.0)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    with pytest.raises(capi.SppError):
        sctx.schur_get_rcs_residual()  # the panels and the block list are the marginals', not a solve's
    dx1 = sctx.ba_solve_step(3.0)
    assert np.array_equal(dx0, dx1)
    assert sctx.schur_get_rcs_residual() < 1e-12
    sctx.ba_marginals_sparse(1.0)
    with pytest.raises(capi.SppError):
        sctx.schur_get_rcs_residual()
    rep1 = sctx.ba_optimize(3, 0.0)
    assert rep0["trace_chi2"] == rep1["trace_chi2"] and rep0["chi2_final"] == rep1["chi2_final"]
    with pytest.raises(capi.NotPositiveDefinite):
        sctx.ba_marginals_sparse(-10.0 * max_diag)


def test_full_size_bal13682_marginals(sctx):
    """BAL-13682 shape (82 092 unknowns in the reduced camera system): finite, symmetric, positive definite blocks, and
    Sigma_pp - C_p^-1 positive semidefinite on a seeded sample of landmarks"""
    from slam_plus_plus_b200 import graphs
    g = graphs.ba_shape("bal13682")
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 50.0
    cc, pc = sctx.ba_marginals_sparse(alpha)
    assert np.all(np.isfinite(cc)) and np.all(np.isfinite(pc))
    assert np.array_equal(cc, cc.transpose(0, 2, 1))
    assert np.max(np.abs(pc - pc.transpose(0, 2, 1))) <= 1e-12 * np.abs(pc).max()
    np.linalg.cholesky(cc)
    np.linalg.cholesky(0.5 * (pc + pc.transpose(0, 2, 1)))
    # C_p^-1 = (V_p + alpha I)^-1 from the device's own landmark blocks
    _, V, _, _, _ = sctx.ba_get_blocks()
    rng = np.random.default_rng(13682)
    sample = rng.choice(pc.shape[0], 2000, replace=False)
    Cinv = np.linalg.inv(V[sample].reshape(-1, 3, 3) + alpha * np.eye(3))
    D = pc[sample] - Cinv
    ev = np.linalg.eigvalsh(0.5 * (D + D.transpose(0, 2, 1)))
    assert np.all(ev >= -1e-9 * np.abs(pc[sample]).max(axis=(1, 2))[:, None]), ev.min()
