"""Joint marginal covariance of any set of vertices (spp_ba_joint_marginals / spp_schur_joint_marginals,
csrc/joint_marginals.cu): against a float64 dense inverse of the same lambda on both paths, off-pattern blocks on medium
shapes against an oracle built from the library's own U, V, W, agreement with the covariance blocks and the marginals,
reproducibility, independence of the batching, state, refusals, and the full BAL-13682 shape. All calls go through the
C ABI."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import lambda_to_dense, load_golden, rel_err

pytestmark = pytest.mark.gpu

CASES = ["ba_tiny", "ba_tiny_interleaved", "ba_small", "ba_small_hard"]
PATHS = ["dense", "sparse"]
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _scalar_index(dims, cols):
    """scalar rows of the given block columns, in the order given"""
    base = np.concatenate([[0], np.cumsum(dims)])
    return np.concatenate([np.arange(base[c], base[c] + dims[c]) for c in cols])


def _random_sets(rng, n_cols, n_sets, max_size):
    return [rng.choice(n_cols, rng.integers(1, max_size + 1), replace=False) for _ in range(n_sets)]


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", CASES)
def test_slot_joint_marginals_vs_dense_inverse(sctx, name, path):
    """the reference's own lambda through slot 1 at alpha = 0 and 0.5: the whole inverse as one set and seeded random
    mixed subsets, to 1e-9"""
    g, d = load_golden(name)
    _set_path(sctx, path)
    dims = d["L0.col_dims"].astype(np.int64)
    sctx.schur_symbolic(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"])
    sctx.schur_solve(d["L0.vals"], d["L0.eta"])
    A = lambda_to_dense(d["L0.col_dims"], d["L0.col_ptr"], d["L0.row_idx"], d["L0.vals"])
    rng = np.random.default_rng(len(dims))
    sets = [np.arange(len(dims))] + _random_sets(rng, len(dims), 12, min(8, len(dims)))
    for alpha in (0.0, 0.5):
        out = sctx.schur_joint_marginals(alpha, sets)
        Ai = np.linalg.inv(A + alpha * np.eye(A.shape[0]))
        for s, cov in zip(sets, out):
            idx = _scalar_index(dims, s)
            assert cov.shape == (len(idx), len(idx))
            assert rel_err(cov, Ai[np.ix_(idx, idx)]) < 1e-9, (alpha, list(s), rel_err(cov, Ai[np.ix_(idx, idx)]))


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", CASES)
def test_ba_joint_marginals_vs_dense_inverse(sctx, name, path):
    """the BA entry point at alpha = 1e-4 max diag: sets of vertex ids, cameras and points mixed in arbitrary order,
    against the inverse of lambda (whose block columns are the vertex ids)"""
    g, _ = load_golden(name)
    _set_path(sctx, path)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    col_dims, col_ptr, row_idx, vals, _ = sctx.ba_get_lambda()
    A = lambda_to_dense(col_dims, col_ptr, row_idx, vals)
    dims = np.asarray(col_dims, np.int64)
    Ai = np.linalg.inv(A + alpha * np.eye(A.shape[0]))
    rng = np.random.default_rng(7 + len(dims))
    nv = len(dims)
    cams, pts = np.flatnonzero(dims == 6), np.flatnonzero(dims == 3)
    sets = _random_sets(rng, nv, 16, min(10, nv)) + [np.concatenate([pts[:2], cams[-2:], pts[-1:], cams[:1]]), rng.permutation(nv)]
    out = sctx.ba_joint_marginals(alpha, sets)
    for s, cov in zip(sets, out):
        idx = _scalar_index(dims, s)
        assert rel_err(cov, Ai[np.ix_(idx, idx)]) < 1e-9, (list(s), rel_err(cov, Ai[np.ix_(idx, idx)]))


# ---- medium shapes ---------------------------------------------------------------------------------------------------

def _shape_graph(shape):
    from slam_plus_plus_b200 import graphs
    if shape == "seq":
        return graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    if shape == "bal16":  # the 1/16 sub-sequence of the BAL-13682 shape (855 cameras)
        return graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
    if shape == "mid_interleaved":
        return graphs.ba_shape("mid", interleave_ids=True, shuffle_edges=True)
    return graphs.ba_shape(shape)


class _Oracle:
    """float64 numpy from the library's own exports: S at alpha from U, V, W, its inverse, and
    Sigma_uv = delta C^-1 + b_u^T S^-1 b_v"""

    def __init__(self, ctx, g, alpha):
        import scipy.sparse as sp
        U, V, W, _, _ = ctx.ba_get_blocks()
        loc = np.asarray(g.vertex_local_index(), np.int64)
        oc, op = loc[np.asarray(g.obs_cam, np.int64)], loc[np.asarray(g.obs_pt, np.int64)]
        self.C, self.P = g.n_cams, g.n_pts
        self.vtype, self.loc = np.asarray(g.vtype), loc
        self.Cinv = np.linalg.inv(V.reshape(-1, 3, 3).transpose(0, 2, 1) + alpha * np.eye(3))
        Wc = W.reshape(-1, 3, 6).transpose(0, 2, 1)  # column-major 6 x 3, edge order
        r = (6 * oc[:, None, None] + np.arange(6)[None, :, None]).repeat(3, 2)
        c = (3 * op[:, None, None] + np.arange(3)[None, None, :]).repeat(6, 1)
        Wm = sp.csr_matrix((Wc.ravel(), (r.ravel(), c.ravel())), shape=(6 * self.C, 3 * self.P))
        Cb = sp.block_diag(list(self.Cinv), format="csr")
        self.Y = (Wm @ Cb).tocsc()
        S = sp.block_diag([u.reshape(6, 6).T for u in U]).toarray() + alpha * np.eye(6 * self.C)
        S -= (self.Y @ Wm.T).toarray()
        self.Sinv = np.linalg.inv(S)

    def rhs(self, v):
        """b_v (6C x d) of vertex id v"""
        i = self.loc[v]
        if self.vtype[v] == 0:
            B = np.zeros((6 * self.C, 6))
            B[6 * i:6 * i + 6] = np.eye(6)
            return B
        return -self.Y[:, 3 * i:3 * i + 3].toarray()

    def joint(self, s):
        B = np.concatenate([self.rhs(v) for v in s], 1)
        J = B.T @ self.Sinv @ B
        off = np.concatenate([[0], np.cumsum([6 if self.vtype[v] == 0 else 3 for v in s])])
        for x, u in enumerate(s):
            for y, v in enumerate(s):
                if self.vtype[u] == 1 and u == v:
                    J[off[x]:off[x + 1], off[y]:off[y + 1]] += self.Cinv[self.loc[u]]
        return J


def _vertex_ids(g):
    vt = np.asarray(g.vtype)
    return np.flatnonzero(vt == 0), np.flatnonzero(vt == 1)  # local index -> vertex id, cameras / points


class _Tracks:
    """cameras of every landmark, and the covisible camera pairs (the block pattern of S) as sorted keys"""

    def __init__(self, g):
        from slam_plus_plus_b200 import capi
        loc = np.asarray(g.vertex_local_index(), np.int64)
        self.oc, self.op = loc[np.asarray(g.obs_cam, np.int64)], loc[np.asarray(g.obs_pt, np.int64)]
        self.order = np.argsort(self.op, kind="stable")
        self.bounds = np.searchsorted(self.op[self.order], np.arange(g.n_pts + 1))
        r, c = capi.rcs_block_pattern(g.n_cams, g.n_pts, self.oc, self.op)
        self.C = g.n_cams
        self.keys = np.sort(np.asarray(r, np.int64) * g.n_cams + np.asarray(c, np.int64))

    def edges(self, p):
        return self.order[self.bounds[p]:self.bounds[p + 1]]

    def cams(self, p):
        return set(self.oc[self.edges(p)].tolist())

    def covisible(self, a, b):
        k = min(a, b) * self.C + max(a, b)
        i = np.searchsorted(self.keys, k)
        return i < len(self.keys) and self.keys[i] == k


def _shape_sets(g, rng):
    """camera pairs that share no landmark, landmark pairs with disjoint tracks, camera-landmark pairs with no
    observation, covisible pairs, singles and one mixed window"""
    cam_id, pt_id = _vertex_ids(g)
    tr = _Tracks(g)
    far, near, pts_far, cam_pt = [], [], [], []
    while len(far) < 12:
        a, b = rng.choice(g.n_cams, 2, replace=False)
        if not tr.covisible(a, b):
            far.append([cam_id[a], cam_id[b]])
    while len(near) < 8:
        p = rng.integers(g.n_pts)
        cs = sorted(tr.cams(p))
        if len(cs) >= 2:
            near.append([cam_id[cs[-1]], cam_id[cs[0]]])
    while len(pts_far) < 12:
        p, q = rng.choice(g.n_pts, 2, replace=False)
        if not tr.cams(p) & tr.cams(q):
            pts_far.append([pt_id[p], pt_id[q]])
    while len(cam_pt) < 12:
        c, p = rng.integers(g.n_cams), rng.integers(g.n_pts)
        if c not in tr.cams(p):
            cam_pt.append([pt_id[p], cam_id[c]] if len(cam_pt) % 2 else [cam_id[c], pt_id[p]])
    singles = [[cam_id[c]] for c in rng.choice(g.n_cams, 4, replace=False)] + [[pt_id[p]] for p in rng.choice(g.n_pts, 4, replace=False)]
    window = list(cam_id[5:13]) + list(pt_id[rng.choice(g.n_pts, 4, replace=False)])
    return dict(far=far, near=near, pts_far=pts_far, cam_pt=cam_pt, singles=singles, window=[window])


@pytest.mark.parametrize("shape", ["mid", "mid_interleaved", "seq", "bal16", "venice871"])
def test_off_pattern_blocks_on_medium_shapes(sctx, shape):
    """off-pattern blocks against the oracle to 1e-9 on both paths; on-pattern blocks against ba_covariance_blocks and
    single vertices against the marginals of the same path; the two paths against each other; exact transposes"""
    g = _shape_graph(shape)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 1e-4 * _max_lambda_diag(sctx)
    rng = np.random.default_rng(sum(map(ord, shape)))
    groups = _shape_sets(g, rng)
    names = [k for k in groups for _ in groups[k]]
    sets = [np.asarray(s, np.int64) for k in groups for s in groups[k]]
    oracle = _Oracle(sctx, g, alpha)
    loc = np.asarray(g.vertex_local_index(), np.int64)
    res = {}
    for path in PATHS:
        _set_path(sctx, path)
        out = sctx.ba_joint_marginals(alpha, sets)
        for name, s, cov in zip(names, sets, out):
            e = rel_err(cov, oracle.joint(s))
            assert e < 1e-9, (path, name, list(s), e)
            assert np.array_equal(cov, cov.T), (path, name)
        near = np.array([[loc[a], loc[b]] for a, b in groups["near"]])
        cb = sctx.ba_covariance_blocks(alpha, near)
        for k, cov in enumerate(out[names.index("near"):names.index("near") + len(near)]):
            assert rel_err(cov[:6, 6:], cb["pairs"][k]) < 1e-9, (path, k)
        cc, pc = sctx.ba_marginals(alpha) if path == "dense" else sctx.ba_marginals_sparse(alpha)
        for s, cov in zip(sets, out):
            if len(s) == 1:
                ref = cc[loc[s[0]]] if g.vtype[s[0]] == 0 else pc[loc[s[0]]]
                assert rel_err(cov, ref) < 1e-9, (path, int(s[0]), rel_err(cov, ref))
        res[path] = out
    for a, b in zip(res["dense"], res["sparse"]):
        assert rel_err(b, a) < 1e-9, rel_err(b, a)


# ---- reproducibility, batching, state ------------------------------------------------------------------------------

_BATCH_SCRIPT = r"""
import sys, numpy as np
from slam_plus_plus_b200 import capi, graphs
g = graphs.ba_shape("mid")
c = capi.Context(0)
c.schur_set_rcs_solver(capi.RCS_DENSE if sys.argv[2] == "dense" else capi.RCS_SPARSE)
c.ba_set_graph(g)
c.ba_linearise()
sets = [np.asarray(s) for s in np.load(sys.argv[1], allow_pickle=True)["sets"]]
out = c.ba_joint_marginals(1.0, sets)
np.savez(sys.argv[1] + ".out.npz", *out)
c.close()
"""


@pytest.mark.parametrize("path", PATHS)
def test_joint_marginals_independent_of_batching(sctx, path, tmp_path):
    """two calls give the same bits; a set alone gives the bits it gets among 300 other sets in batches of at most 64
    columns (SPP_JOINT_BATCH_COLS, read once per process: in a subprocess)"""
    from slam_plus_plus_b200 import graphs
    g = graphs.ba_shape("mid")
    _set_path(sctx, path)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    rng = np.random.default_rng(64)
    nv = len(g.vtype)
    target = rng.choice(nv, 6, replace=False)
    others = _random_sets(rng, nv, 300, 5)
    alone = sctx.ba_joint_marginals(1.0, [target])[0]
    again = sctx.ba_joint_marginals(1.0, [target])[0]
    assert np.array_equal(alone, again)
    many = sctx.ba_joint_marginals(1.0, others[:150] + [target] + others[150:])
    assert np.array_equal(many[150], alone)
    f = str(tmp_path / "sets.npz")
    sets = np.empty(301, object)
    sets[:] = others[:150] + [target] + others[150:]
    np.savez(f, sets=sets)
    env = dict(os.environ, SPP_JOINT_BATCH_COLS="64", PYTHONPATH=REPO + os.pathsep + os.environ.get("PYTHONPATH", ""))
    subprocess.run([sys.executable, "-c", _BATCH_SCRIPT, f, path], check=True, env=env, cwd=REPO, timeout=600)
    sub = np.load(f + ".out.npz")
    assert np.array_equal(sub["arr_150"], alone)
    for k in range(301):
        assert np.array_equal(sub[f"arr_{k}"], many[k]), k


def test_joint_marginals_state(sctx):
    """after a supernodal call the residual check of the last solve is refused, and solves and LM give the bits they
    give without the call; a strongly negative damping is reported as a non-positive pivot"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.make_ba(400, 30000, 400, mean_extra_track=3.0, max_track=20, max_stride=4, loops=2)
    sctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    max_diag = _max_lambda_diag(sctx)
    dx0 = sctx.ba_solve_step(3.0)
    rep0 = sctx.ba_optimize(3, 0.0)
    sets = _random_sets(np.random.default_rng(400), len(g.vtype), 50, 6)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    sctx.ba_joint_marginals(1.0, sets)
    with pytest.raises(capi.SppError):
        sctx.schur_get_rcs_residual()
    dx1 = sctx.ba_solve_step(3.0)
    assert np.array_equal(dx0, dx1)
    assert sctx.schur_get_rcs_residual() < 1e-12
    sctx.ba_joint_marginals(1.0, sets)
    rep1 = sctx.ba_optimize(3, 0.0)
    assert rep0["trace_chi2"] == rep1["trace_chi2"] and rep0["chi2_final"] == rep1["chi2_final"]
    for path in PATHS:
        _set_path(sctx, path)
        with pytest.raises(capi.NotPositiveDefinite):
            sctx.ba_joint_marginals(-10.0 * max_diag, sets)


@pytest.mark.parametrize("path", PATHS)
def test_joint_marginals_refusals(sctx, path):
    """an id out of range, an empty set and a set wider than 16 384 columns are refused; the context still solves
    afterwards, with the same bits"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("mid")
    _set_path(sctx, path)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    dx0 = sctx.ba_solve_step(1.0)
    nv = len(g.vtype)
    cam0 = int(np.flatnonzero(np.asarray(g.vtype) == 0)[0])
    for sets in ([[0, nv]], [[0, 1], []], [[0], np.full(2731, cam0)]):
        with pytest.raises(capi.SppError):
            sctx.ba_joint_marginals(1.0, sets)
    assert np.array_equal(sctx.ba_solve_step(1.0), dx0)
    out = sctx.ba_joint_marginals(1.0, [[0, 1], [nv - 1]])
    assert np.all(np.isfinite(out[0])) and np.all(np.isfinite(out[1]))


def test_schur_joint_marginals_needs_a_slot_system():
    """slot 1 on a context that has no system of the caller's: the library's refusal, not a binding error"""
    from slam_plus_plus_b200 import capi
    c = capi.Context(0)
    try:
        with pytest.raises(capi.SppError):
            c.schur_joint_marginals(1.0, [[0, 1]])
    finally:
        c.close()


# ---- full BAL-13682 shape ------------------------------------------------------------------------------------------

def test_full_size_bal13682_joint_marginals(sctx):
    """alpha = 50, supernodal path: 200 seeded camera pairs that share no landmark (positive definite, diagonal blocks
    as ba_marginals_sparse), a window of 100 consecutive cameras (positive definite, covisible blocks as
    ba_covariance_blocks), and the row identity of lambda Sigma = I for 100 seeded landmark pairs"""
    from slam_plus_plus_b200 import capi, graphs
    g = graphs.ba_shape("bal13682")
    sctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    sctx.ba_set_graph(g)
    sctx.ba_linearise()
    alpha = 50.0
    rng = np.random.default_rng(13682)
    cam_id, pt_id = _vertex_ids(g)
    tr = _Tracks(g)
    oc = tr.oc
    pairs = []
    while len(pairs) < 200:
        a, b = sorted(rng.choice(g.n_cams, 2, replace=False).tolist())
        if not tr.covisible(a, b):
            pairs.append((a, b))
    cc, _ = sctx.ba_marginals_sparse(alpha)
    out = sctx.ba_joint_marginals(alpha, [[cam_id[a], cam_id[b]] for a, b in pairs])
    for (a, b), J in zip(pairs, out):
        np.linalg.cholesky(J)
        assert rel_err(J[:6, :6], cc[a]) < 1e-9 and rel_err(J[6:, 6:], cc[b]) < 1e-9
    w0 = int(rng.integers(0, g.n_cams - 100))
    win = sctx.ba_joint_marginals(alpha, [cam_id[w0:w0 + 100]])[0]
    np.linalg.cholesky(win)
    near = np.array([(i, j) for i in range(w0, w0 + 100) for j in range(i + 1, w0 + 100) if tr.covisible(i, j)])
    cb = sctx.ba_covariance_blocks(alpha, near)["pairs"]
    got = np.stack([win[6 * (i - w0):6 * (i - w0) + 6, 6 * (j - w0):6 * (j - w0) + 6] for i, j in near])
    assert rel_err(got, cb) < 1e-9, rel_err(got, cb)
    # (V_p + alpha I) Sigma_pq + sum_{a in track(p)} W_a^T Sigma_{c_a q} = delta_pq I, the device's own V and W
    _, V, W, _, _ = sctx.ba_get_blocks()
    sets, meta = [], []
    for k in range(100):
        p = int(rng.integers(g.n_pts))
        q = p if k % 10 == 0 else int(rng.integers(g.n_pts))
        edges = tr.edges(p)
        sets.append([pt_id[p]] + [cam_id[c] for c in oc[edges]] + [pt_id[q]])
        meta.append((p, q, edges))
    worst = 0.0
    for (p, q, edges), J in zip(meta, sctx.ba_joint_marginals(alpha, sets)):
        n_e = len(edges)
        lhs = (V[p].reshape(3, 3).T + alpha * np.eye(3)) @ J[:3, -3:]
        for k, a in enumerate(edges):
            Wa = W[a].reshape(3, 6).T  # column-major 6 x 3
            lhs += Wa.T @ J[3 + 6 * k:9 + 6 * k, -3:]
        ref = np.eye(3) if p == q else np.zeros((3, 3))
        assert n_e > 0
        worst = max(worst, float(np.abs(lhs - ref).max()))
    assert worst < 1e-9, worst
