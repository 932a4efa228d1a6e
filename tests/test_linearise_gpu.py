"""GPU tests of the linearisation (k_linearise_cams, k_sum_point_records) and of the landmark inverse of the Schur stage
(k_landmark_inverse):
  * two linearisations give bit-identical U, V, W, eta_c, eta_p;
  * V and eta_p are the insertion-order sums of the per-observation landmark records. The records are read back from
    an "exploded" copy of the graph in which every observation has a landmark of its own (same position, same
    measurement), so numpy restates the sums without restating the Jacobians; U, eta_c and W are checked against the
    same copy;
  * Cinv = (V + alpha I)^-1 and Y = W Cinv, which are not exposed, through the reduced camera system and the increment
    of ba_solve_step against a numpy Schur complement built from the library's own blocks;
on the `mid` shape, on a graph with landmarks of track length 1 and 50+, and on a graph whose cameras all see fewer
observations than one CTA trip (256) and whose unary factor sits on a landmark."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

ALPHA = 10.0


def graph_mid():
    from slam_plus_plus_b200 import graphs
    return graphs.ba_shape("mid")


def graph_long_and_single():
    """tracks of length 1 (every third landmark keeps only its first observation) next to tracks of 50-60"""
    from slam_plus_plus_b200 import graphs
    from slam_plus_plus_b200.sppio import BAGraph
    g = graphs.make_ba(64, 600, 5, mean_extra_track=40.0, max_track=60, max_stride=1)
    op = np.asarray(g.obs_pt, np.int64)
    first = np.r_[True, op[1:] != op[:-1]]  # make_ba lists each track's edges together
    keep = first | ((op - 64) % 3 != 0)
    return BAGraph(g.vtype, g.cams, g.pts, g.obs_pt[keep], g.obs_cam[keep], g.z[keep], g.info[keep])


def graph_short_cams_point_unary():
    """every camera sees fewer than 256 observations; vertex 0, which carries the unary factor, is a landmark"""
    from slam_plus_plus_b200 import graphs
    return graphs.make_ba(40, 1500, 1, interleave_ids=True, mean_extra_track=3.0, max_track=12, max_stride=2)


GRAPHS = {"mid": graph_mid, "long_and_single": graph_long_and_single, "short_cams_point_unary": graph_short_cams_point_unary}


def exploded(g):
    """the same cameras, one landmark per observation (at the position of the observation's landmark)"""
    from slam_plus_plus_b200.sppio import BAGraph
    loc = np.asarray(g.vertex_local_index(), np.int64)
    O, C = len(g.obs_pt), g.n_cams
    vtype = np.r_[np.zeros(C, np.int64), np.ones(O, np.int64)]
    pts = np.asarray(g.pts)[loc[np.asarray(g.obs_pt, np.int64)]]
    obs_cam = loc[np.asarray(g.obs_cam, np.int64)]
    return BAGraph(vtype, g.cams, pts, C + np.arange(O, dtype=np.int64), obs_cam, g.z, g.info)


@pytest.fixture(scope="module", params=list(GRAPHS))
def case(request):
    g = GRAPHS[request.param]()
    track = np.bincount(np.asarray(g.vertex_local_index())[np.asarray(g.obs_pt, np.int64)], minlength=g.n_pts)
    cam_obs = np.bincount(np.asarray(g.vertex_local_index())[np.asarray(g.obs_cam, np.int64)], minlength=g.n_cams)
    if request.param == "long_and_single":
        assert track.min() == 1 and track.max() >= 50
    if request.param == "short_cams_point_unary":
        assert cam_obs.max() < 256 and g.vtype[0] == 1
    return request.param, g


def test_linearise_bit_reproducible(ctx, case):
    _, g = case
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    a = ctx.ba_get_blocks()
    ctx.ba_linearise()
    b = ctx.ba_get_blocks()
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint64), y.view(np.uint64))


def test_point_sums_vs_records(ctx, case):
    """V_p, eta_p = sum of the observation records along the track in insertion order (+ I for the unary factor)"""
    _, g = case
    loc = np.asarray(g.vertex_local_index(), np.int64)
    op, oc = loc[np.asarray(g.obs_pt, np.int64)], loc[np.asarray(g.obs_cam, np.int64)]
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    U, V, W, gc, gp = ctx.ba_get_blocks()
    ctx.ba_set_graph(exploded(g))
    ctx.ba_linearise()
    Ux, Vx, Wx, gcx, gpx = ctx.ba_get_blocks()
    # per-observation blocks are the same expressions of the same inputs
    assert np.array_equal(W, Wx)
    V_ref, gp_ref = np.zeros_like(V), np.zeros_like(gp)
    np.add.at(V_ref, op, Vx)  # unbuffered, in index order: edge insertion order within each track
    np.add.at(gp_ref, op, gpx)
    eye3, eye6 = np.eye(3).ravel(), np.eye(6).ravel()
    Ux[0] -= eye6  # the exploded graph's vertex 0 is camera 0
    if g.vtype[0] == 1:
        V_ref[loc[0]] += eye3
    else:
        Ux[loc[0]] += eye6
    assert rel_err(V, V_ref) < 1e-14, rel_err(V, V_ref)
    assert rel_err(gp, gp_ref) < 1e-14, rel_err(gp, gp_ref)
    # U_c, eta_c sum the same observation terms in another order (the camera's list is in track order)
    assert rel_err(U, Ux) < 1e-12, rel_err(U, Ux)
    assert rel_err(gc, gcx) < 1e-12, rel_err(gc, gcx)
    assert np.array_equal(np.bincount(oc, minlength=g.n_cams) > 0, np.ones(g.n_cams, bool))


def test_landmark_inverse_through_schur(ctx, case):
    """reduced camera system, its right-hand side and the increment against numpy from the library's U, V, W, eta"""
    import scipy.sparse as sp
    _, g = case
    loc = np.asarray(g.vertex_local_index(), np.int64)
    op, oc = loc[np.asarray(g.obs_pt, np.int64)], loc[np.asarray(g.obs_cam, np.int64)]
    C, P = g.n_cams, g.n_pts
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    U, V, W, gc, gp = ctx.ba_get_blocks()
    ctx.schur_get_reduced_system(want_values=False)  # arms the copy
    dx = ctx.ba_solve_step(ALPHA)
    S, rhs, _ = ctx.schur_get_reduced_system()

    Cinv = np.linalg.inv(V.reshape(-1, 3, 3).transpose(0, 2, 1) + ALPHA * np.eye(3))
    Wc = W.reshape(-1, 3, 6).transpose(0, 2, 1)  # column-major 6 x 3, edge order
    r = (6 * oc[:, None, None] + np.arange(6)[None, :, None]).repeat(3, 2)
    c = (3 * op[:, None, None] + np.arange(3)[None, None, :]).repeat(6, 1)
    Wm = sp.csr_matrix((Wc.ravel(), (r.ravel(), c.ravel())), shape=(6 * C, 3 * P))
    Cb = sp.block_diag(list(Cinv), format="csr")
    Y = Wm @ Cb
    S_ref = sp.block_diag([u.reshape(6, 6).T for u in U]).toarray() + ALPHA * np.eye(6 * C) - (Y @ Wm.T).toarray()
    rhs_ref = gc.ravel() - Y @ gp.ravel()
    iu = np.triu_indices(6 * C)
    assert rel_err(S[iu], S_ref[iu]) < 1e-11, rel_err(S[iu], S_ref[iu])
    assert rel_err(rhs, rhs_ref) < 1e-11, rel_err(rhs, rhs_ref)

    dxc = np.linalg.solve(S_ref, rhs_ref)
    dxp = np.einsum("pij,pj->pi", Cinv, gp - (Wm.T @ dxc).reshape(-1, 3))
    dx_ref = np.concatenate([dxc.reshape(-1, 6)[loc[v]] if g.vtype[v] == 0 else dxp[loc[v]] for v in range(len(g.vtype))])
    assert rel_err(dx, dx_ref) < 1e-9, rel_err(dx, dx_ref)
