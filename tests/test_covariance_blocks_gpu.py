"""Off-diagonal blocks of the covariance (lambda + alpha I)^-1 (spp_ba_covariance_blocks / spp_schur_covariance_pattern,
csrc/marginals.cu): camera pairs that share a landmark and the camera-landmark block of every observation, on the dense
and on the supernodal reduced camera system. Against a float64 dense inverse of the same lambda, path against path, the
identity Sigma_pp = C_p^-1 - C_p^-1 sum_a W_a^T Sigma_{c_a p}, reproducibility and state, refusals, and the full
BAL-13682 shape. All calls go through the C ABI."""
import numpy as np
import pytest

from conftest import lambda_to_dense, load_golden, rel_err

pytestmark = pytest.mark.gpu

CASES = ["ba_tiny", "ba_tiny_interleaved", "ba_small", "ba_small_hard"]
PATHS = ["dense", "sparse"]


@pytest.fixture()
def sctx(ctx):
    from slam_plus_plus_b200 import capi
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.schur_set_rcs_ordering(None)
    yield ctx
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.schur_set_rcs_ordering(None)


def _set_path(ctx, path):
    from slam_plus_plus_b200 import capi
    ctx.schur_set_rcs_solver(capi.RCS_DENSE if path == "dense" else capi.RCS_SPARSE)


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
        m = max(m, float(np.diag(vals[off[k]:off[k] + d * d].reshape(d, d)).max()))
    return m


def _edge_indices(g):
    """local camera and point index of every edge (edge insertion order)"""
    loc = np.asarray(g.vertex_local_index(), np.int64)
    return loc[np.asarray(g.obs_cam, np.int64)], loc[np.asarray(g.obs_pt, np.int64)]


def _covisible_pairs(g):
    """off-diagonal upper blocks (i < j) of the reduced camera system, through the library's host helper"""
    from slam_plus_plus_b200 import capi
    oc, op = _edge_indices(g)
    r, c = capi.rcs_block_pattern(g.n_cams, g.n_pts, oc, op)
    off = r != c
    return np.stack([r[off], c[off]], 1).astype(np.int64)


def _request(g):
    """every covisible pair, each reversed, and every diagonal pair"""
    up = _covisible_pairs(g)
    diag = np.stack([np.arange(g.n_cams)] * 2, 1)
    return np.concatenate([up, up[:, ::-1], diag])


def _identity_points(ctx, g, alpha, obs_cov):
    """C_p^-1 - C_p^-1 sum_a W_a^T Sigma_{c_a p}, C_p = V_p + alpha I, from the device's own W and V (all observations)"""
    _, V, W, _, _ = ctx.ba_get_blocks()
    _, op = _edge_indices(g)
    W = W.reshape(-1, 3, 6).transpose(0, 2, 1)  # column-major 6 x 3
    Cinv = np.linalg.inv(V.reshape(-1, 3, 3).transpose(0, 2, 1) + alpha * np.eye(3))
    acc = np.zeros((g.n_pts, 3, 3))
    np.add.at(acc, op, np.einsum("eji,ejk->eik", W, obs_cov))
    return Cinv - Cinv @ acc


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", CASES)
def test_slot_covariance_pattern_vs_dense_inverse(sctx, name, path):
    """the reference's own lambda through slot 1, alpha = 0 and 0.5: (lambda + alpha I)^-1 on the pattern of lambda, in
    its value layout, to 1e-9"""
    g, d = load_golden(name)
    _set_path(sctx, path)
    dims = d["L0.col_dims"].astype(np.int64)
    col_ptr, row_idx = d["L0.col_ptr"].astype(np.int64), d["L0.row_idx"].astype(np.int64)
    sctx.schur_symbolic(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"])
    sctx.schur_solve(d["L0.vals"], d["L0.eta"])
    A = lambda_to_dense(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"], d["L0.vals"])
    base = np.concatenate([[0], np.cumsum(dims)])
    for alpha in (0.0, 0.5):
        cov = sctx.schur_covariance_pattern(alpha)
        assert cov.shape == d["L0.vals"].shape
        Ai = np.linalg.inv(A + alpha * np.eye(A.shape[0]))
        ref, off = np.empty_like(cov), 0
        for c in range(len(dims)):
            for k in range(col_ptr[c], col_ptr[c + 1]):
                r = row_idx[k]
                h, w = dims[r], dims[c]
                ref[off:off + h * w] = Ai[base[r]:base[r] + h, base[c]:base[c] + w].T.ravel()  # column-major
                off += h * w
        assert off == len(cov)
        assert rel_err(cov, ref) < 1e-9, (alpha, rel_err(cov, ref))


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", CASES)
def test_ba_covariance_blocks_vs_dense_inverse(sctx, name, path):
    """every covisible pair (both orders), every diagonal pair and every observation against the inverse of the dense,
    permuted lambda at alpha = 1e-4 max diag; the identity for the landmark blocks"""
    g, _ = load_golden(name)
    _set_path(sctx, path)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    col_dims, col_ptr, row_idx, vals, _ = sctx.ba_get_lambda()
    A = lambda_to_dense(col_dims, col_ptr, row_idx, vals)
    dims = np.asarray(col_dims, np.int64)
    base = np.concatenate([[0], np.cumsum(dims)])
    perm = np.concatenate([np.arange(base[i], base[i + 1]) for i in np.flatnonzero(dims == 6)] +
                          [np.arange(base[i], base[i + 1]) for i in np.flatnonzero(dims == 3)])
    Ai = np.linalg.inv(A[np.ix_(perm, perm)] + alpha * np.eye(A.shape[0]))
    pairs = _request(g)
    oc, op = _edge_indices(g)
    out = sctx.ba_covariance_blocks(alpha, pairs, np.arange(g.n_obs), diagonal=True)
    o = 6 * g.n_cams
    ref_pairs = np.stack([Ai[6 * i:6 * i + 6, 6 * j:6 * j + 6] for i, j in pairs])
    ref_obs = np.stack([Ai[6 * c:6 * c + 6, o + 3 * p:o + 3 * p + 3] for c, p in zip(oc, op)])
    assert out["pairs"].shape == (len(pairs), 6, 6) and out["observations"].shape == (g.n_obs, 6, 3)
    assert rel_err(out["pairs"], ref_pairs) < 1e-9, rel_err(out["pairs"], ref_pairs)
    assert rel_err(out["observations"], ref_obs) < 1e-9, rel_err(out["observations"], ref_obs)
    ident = _identity_points(sctx, g, alpha, out["observations"])
    assert rel_err(ident, out["points"]) < 1e-9, rel_err(ident, out["points"])


def _shape_graph(shape):
    from slam_plus_plus_b200 import graphs
    if shape == "seq":
        return graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    if shape == "bal16":  # the 1/16 sub-sequence of the BAL-13682 shape (855 cameras)
        return graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
    if shape == "mid_interleaved":
        return graphs.ba_shape("mid", interleave_ids=True, shuffle_edges=True)
    return graphs.ba_shape(shape)


@pytest.mark.parametrize("shape", ["mid", "mid_interleaved", "seq", "bal16", "venice871"])
def test_dense_and_supernodal_paths_agree(sctx, shape):
    """the two paths agree to 1e-9; on each, the block diagonal and the (i, i) pairs are the bits of that path's
    marginals, (j, i) is the exact transpose of (i, j), and the identity for the landmark blocks holds"""
    g = _shape_graph(shape)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    pairs = _request(g)
    n_up = (len(pairs) - g.n_cams) // 2
    obs = np.arange(g.n_obs)
    res = {}
    for path in PATHS:
        _set_path(sctx, path)
        out = sctx.ba_covariance_blocks(alpha, pairs, obs, diagonal=True)
        cc, pc = sctx.ba_marginals(alpha) if path == "dense" else sctx.ba_marginals_sparse(alpha)
        assert np.array_equal(out["cameras"], cc) and np.array_equal(out["points"], pc), path
        assert np.array_equal(out["pairs"][2 * n_up:], cc), path
        assert np.array_equal(out["pairs"][n_up:2 * n_up], out["pairs"][:n_up].transpose(0, 2, 1)), path
        ident = _identity_points(sctx, g, alpha, out["observations"])
        assert rel_err(ident, pc) < 1e-9, (path, rel_err(ident, pc))
        res[path] = out
    for key in ("pairs", "observations", "cameras", "points"):
        e = rel_err(res["sparse"][key], res["dense"][key])
        assert e < 1e-9, (key, e)


def test_covariance_blocks_reproducible_and_state(sctx):
    """two calls give the same bits; after the call on the supernodal path the residual check of the last solve is
    refused, solves and LM give the bits they give without the call, and a negative damping is reported as a
    non-positive pivot"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    sctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    max_diag = _max_lambda_diag(sctx)
    dx0 = sctx.ba_solve_step(3.0)
    rep0 = sctx.ba_optimize(3, 0.0)
    pairs = _request(g)
    obs = np.random.default_rng(400).choice(g.n_obs, 5000, replace=False)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    a = sctx.ba_covariance_blocks(1.0, pairs, obs, diagonal=True)
    b = sctx.ba_covariance_blocks(1.0, pairs, obs, diagonal=True)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    with pytest.raises(capi.SppError):
        sctx.schur_get_rcs_residual()  # the panels and the block list hold the covariance, not a solve
    dx1 = sctx.ba_solve_step(3.0)
    assert np.array_equal(dx0, dx1)
    assert sctx.schur_get_rcs_residual() < 1e-12
    sctx.ba_covariance_blocks(1.0, pairs, obs)
    with pytest.raises(capi.SppError):
        sctx.schur_get_rcs_residual()
    rep1 = sctx.ba_optimize(3, 0.0)
    assert rep0["trace_chi2"] == rep1["trace_chi2"] and rep0["chi2_final"] == rep1["chi2_final"]
    with pytest.raises(capi.NotPositiveDefinite):
        sctx.ba_covariance_blocks(-10.0 * max_diag, pairs, obs)


@pytest.mark.parametrize("path", PATHS)
def test_covariance_blocks_refusals(sctx, path):
    """a pair that shares no landmark, a camera index and an observation index out of range are refused; the context
    still solves afterwards, with the same bits"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("mid")
    _set_path(sctx, path)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    dx0 = sctx.ba_solve_step(1.0)
    up = _covisible_pairs(g)
    covisible = set(map(tuple, up))
    far = next((i, j) for i in range(g.n_cams) for j in range(i + 1, g.n_cams) if (i, j) not in covisible)
    good = up[:3]
    for pairs, obs in (([far], None), ([far[::-1]], None), (np.concatenate([good, [far]]), [0]), ([[0, g.n_cams]], None),
                       (good, [g.n_obs]), (None, [0, g.n_obs + 5])):
        with pytest.raises(capi.SppError):
            sctx.ba_covariance_blocks(1.0, pairs, obs)
    assert np.array_equal(sctx.ba_solve_step(1.0), dx0)
    out = sctx.ba_covariance_blocks(1.0, good, [0, 1])
    assert np.all(np.isfinite(out["pairs"])) and np.all(np.isfinite(out["observations"]))


def test_covariance_pattern_needs_a_slot_system():
    """slot 1 on a context that has no system of the caller's: the library's refusal, not a binding error"""
    from slam_plus_plus_b200 import capi
    c = capi.Context(0)
    try:
        with pytest.raises(capi.SppError):
            c.schur_covariance_pattern(1.0)
    finally:
        c.close()


def test_full_size_bal13682_covariance_blocks(sctx):
    """BAL-13682 shape, alpha = 50, supernodal path: a seeded sample of 20 000 covisible pairs and the observations of
    2 000 landmarks; finite, every 12 x 12 joint covariance of a pair positive definite, the identity against
    ba_marginals_sparse on the sampled landmarks"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("bal13682")
    sctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 50.0
    rng = np.random.default_rng(13682)
    up = _covisible_pairs(g)
    pairs = up[rng.choice(len(up), 20000, replace=False)]
    oc, op = _edge_indices(g)
    pts = rng.choice(g.n_pts, 2000, replace=False)
    obs = np.flatnonzero(np.isin(op, pts))
    out = sctx.ba_covariance_blocks(alpha, pairs, obs, diagonal=True)
    for key in out:
        assert np.all(np.isfinite(out[key])), key
    cc, pc = sctx.ba_marginals_sparse(alpha)
    assert np.array_equal(out["cameras"], cc) and np.array_equal(out["points"], pc)
    i, j = pairs[:, 0], pairs[:, 1]
    joint = np.block([[cc[i], out["pairs"]], [out["pairs"].transpose(0, 2, 1), cc[j]]])
    np.linalg.cholesky(joint)
    # the identity on the sampled landmarks, with the device's own W and V
    _, V, W, _, _ = sctx.ba_get_blocks()
    Wo = W[obs].reshape(-1, 3, 6).transpose(0, 2, 1)
    sp = np.sort(pts)
    acc = np.zeros((len(sp), 3, 3))
    np.add.at(acc, np.searchsorted(sp, op[obs]), np.einsum("eji,ejk->eik", Wo, out["observations"]))
    Cinv = np.linalg.inv(V[sp].reshape(-1, 3, 3).transpose(0, 2, 1) + alpha * np.eye(3))
    ident = Cinv - Cinv @ acc
    assert rel_err(ident, pc[sp]) < 1e-9, rel_err(ident, pc[sp])
