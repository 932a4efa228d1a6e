"""ctypes access to the CPU oracle (oracle/spp_oracle.c). TEST INFRASTRUCTURE ONLY: imported by tests/,
__graft_entry__.smoke() and the cpu_baseline leg of bench.py -- never by the product package."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_build", "libspp_oracle.so")
_lib = None


def build():
    subprocess.run(["make", "-C", _HERE, "CC=gcc"], check=True, stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(os.path.join(_HERE, "spp_oracle.c")):
            build()
        _lib = C.CDLL(_LIB)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _graph_args(g):
    vt = np.ascontiguousarray(g.vtype, np.uint8)
    cams = np.ascontiguousarray(g.cams, np.float64)
    pts = np.ascontiguousarray(g.pts, np.float64)
    op = np.ascontiguousarray(g.obs_pt, np.uint64)
    oc = np.ascontiguousarray(g.obs_cam, np.uint64)
    z = np.ascontiguousarray(g.z, np.float64)
    info = np.ascontiguousarray(g.info, np.float64)
    keep = (vt, cams, pts, op, oc, z, info)
    args = [C.c_size_t(len(vt)), _p(vt, C.c_uint8), _p(cams, C.c_double), _p(pts, C.c_double), C.c_size_t(len(op)),
            _p(op, C.c_uint64), _p(oc, C.c_uint64), _p(z, C.c_double), _p(info, C.c_double)]
    return args, keep


def ba_chi2(g) -> float:
    args, keep = _graph_args(g)
    v = C.c_double()
    assert lib().spo_ba_chi2(*args, C.byref(v)) == 0
    return v.value


def ba_linearise(g):
    """Returns U (C,36), V (P,9), W (O,18; edge order), gc (C,6), gp (P,3), max per-edge diagonal."""
    args, keep = _graph_args(g)
    c, p, o = g.n_cams, g.n_pts, g.n_obs
    U, V, W = np.zeros((c, 36)), np.zeros((p, 9)), np.zeros((o, 18))
    gc, gp = np.zeros((c, 6)), np.zeros((p, 3))
    md = C.c_double()
    assert lib().spo_ba_linearise(*args, _p(U, C.c_double), _p(V, C.c_double), _p(W, C.c_double), _p(gc, C.c_double),
                                  _p(gp, C.c_double), C.byref(md)) == 0
    return U, V, W, gc, gp, md.value


def schur_solve(obs_c, obs_p, U, V, W, gc, gp, alpha, want_reduced=False):
    """Returns (status, dxc, dxp[, S, rhs]); status 1 = not positive definite."""
    c, p, o = U.shape[0], V.shape[0], W.shape[0]
    oc = np.ascontiguousarray(obs_c, np.uint32)
    op = np.ascontiguousarray(obs_p, np.uint32)
    arrs = [np.ascontiguousarray(a, np.float64) for a in (U, V, W, gc, gp)]
    dxc, dxp = np.zeros((c, 6)), np.zeros((p, 3))
    S = np.zeros((6 * c, 6 * c)) if want_reduced else None
    rhs = np.zeros(6 * c) if want_reduced else None
    rc = lib().spo_schur_solve(C.c_size_t(c), C.c_size_t(p), C.c_size_t(o), _p(oc, C.c_uint32), _p(op, C.c_uint32),
                               *[_p(a, C.c_double) for a in arrs], C.c_double(alpha), _p(dxc, C.c_double), _p(dxp, C.c_double),
                               _p(S, C.c_double) if want_reduced else None, _p(rhs, C.c_double) if want_reduced else None)
    if want_reduced:
        return rc, dxc, dxp, S.T.copy(), rhs  # the C side writes column-major
    return rc, dxc, dxp


def dense_llt_solve(A, b):
    Af = np.asfortranarray(A, np.float64).copy(order="F")
    x = np.array(b, np.float64, copy=True)
    rc = lib().spo_dense_llt_solve(C.c_size_t(A.shape[0]), Af.ctypes.data_as(C.POINTER(C.c_double)), _p(x, C.c_double))
    return rc, x


def relative_to_absolute(v1, v2):
    a = np.ascontiguousarray(v1, np.float64)
    b = np.ascontiguousarray(v2, np.float64)
    d = np.zeros(6)
    lib().spo_relative_to_absolute.restype = None
    lib().spo_relative_to_absolute(_p(a, C.c_double), _p(b, C.c_double), _p(d, C.c_double))
    return d


_BA_SOLVER = C.CFUNCTYPE(C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, *([C.POINTER(C.c_double)] * 5), C.c_double,
                         C.POINTER(C.c_double), C.POINTER(C.c_double))
_POSE_SOLVER = C.CFUNCTYPE(C.c_int, C.c_size_t, C.POINTER(C.c_double), C.POINTER(C.c_double))


def _arr(p, n):
    return np.ctypeslib.as_array(p, shape=(n,))


def ba_optimize(g, max_iter=5, min_dx=0.0, max_trace=64, linear_solver=None):
    """The reference's LM loop. linear_solver(U, V, W, gc, gp, alpha) -> (status, dxc, dxp), if given, takes the place of
    the oracle's own Schur solve (the reference's linear-solver slot)."""
    if linear_solver is not None:
        errors = []

        def cb(c, p, o, U, V, W, gc, gp, alpha, dxc, dxp):
            try:
                rc, xc, xp = linear_solver(_arr(U, c * 36).reshape(c, 36), _arr(V, p * 9).reshape(p, 9),
                                           _arr(W, o * 18).reshape(o, 18), _arr(gc, c * 6).reshape(c, 6),
                                           _arr(gp, p * 3).reshape(p, 3), alpha)
                if rc == 0:
                    _arr(dxc, c * 6)[:] = np.ravel(xc)
                    _arr(dxp, p * 3)[:] = np.ravel(xp)
                return rc
            except BaseException as ex:  # stops the C loop; raised again once it has returned
                errors.append(ex)
                return -1
        fn = _BA_SOLVER(cb)
        lib().spo_set_ba_linear_solver(fn)
        try:
            r = ba_optimize(g, max_iter, min_dx, max_trace)
        finally:
            lib().spo_set_ba_linear_solver(None)
        if errors:
            raise errors[0]
        return r
    args, keep = _graph_args(g)
    cam_out, pts_out = np.zeros((g.n_cams, 6)), np.zeros((g.n_pts, 3))
    trace = np.zeros((max_trace, 6))
    sc = np.zeros(5)
    assert lib().spo_ba_optimize(*args, C.c_size_t(max_iter), C.c_double(min_dx), _p(cam_out, C.c_double),
                                 _p(pts_out, C.c_double), _p(trace, C.c_double), C.c_size_t(max_trace), _p(sc, C.c_double)) == 0
    n = int(sc[3])
    return dict(chi2_initial=sc[0], chi2_final=sc[1], alpha_initial=sc[2], n_solves=n, status=int(sc[4]),
                trace=trace[:min(n, max_trace)], cams=cam_out, pts=pts_out)


def ba_dense_lambda(g, U, V, W):
    """(U, V, W) -> dense lambda with the cameras first, then the points (each group in vertex id order)."""
    c, p = g.n_cams, g.n_pts
    loc = g.vertex_local_index()
    L = np.zeros((6 * c + 3 * p, 6 * c + 3 * p))
    for i in range(c):
        L[6 * i:6 * i + 6, 6 * i:6 * i + 6] = U[i].reshape(6, 6)
    for j in range(p):
        L[6 * c + 3 * j:6 * c + 3 * j + 3, 6 * c + 3 * j:6 * c + 3 * j + 3] = V[j].reshape(3, 3)
    for e in range(g.n_obs):
        i, j = int(loc[g.obs_cam[e]]), int(loc[g.obs_pt[e]])
        w = W[e].reshape(3, 6).T
        L[6 * i:6 * i + 6, 6 * c + 3 * j:6 * c + 3 * j + 3] = w
        L[6 * c + 3 * j:6 * c + 3 * j + 3, 6 * i:6 * i + 6] = w.T
    return L


def ba_marginals(g, alpha=0.0):
    """Block diagonal of (lambda + alpha I)^-1 at the states of g, the quantity the reference recovers from the
    Schur-complemented system (CSchurComplement_Marginals::Schur_Marginals, include/slam/BAMarginals.h:579-760, called
    from NonlinearSolver_Lambda_LM.h:1118-1350 with alpha = 0), here by a plain dense inverse (small cases only).
    Returns cam_cov (C, 6, 6), pt_cov (P, 3, 3) and the dense lambda."""
    U, V, W, _, _, _ = ba_linearise(g)
    L = ba_dense_lambda(g, U, V, W)
    S = np.linalg.inv(L + alpha * np.eye(L.shape[0]))
    c, p = g.n_cams, g.n_pts
    cc = np.stack([S[6 * i:6 * i + 6, 6 * i:6 * i + 6] for i in range(c)])
    pc = np.stack([S[6 * c + 3 * j:6 * c + 3 * j + 3, 6 * c + 3 * j:6 * c + 3 * j + 3] for j in range(p)])
    return cc, pc, L


def lambda_blocks_to_reference_layout(g, U, V, W):
    """(U, V, W) -> the reference's block layout of lambda (upper block-triangular, vertex id order, column-major
    blocks): col_dims, col_ptr, row_idx, vals -- what CUberBlockMatrix accessors enumerate."""
    nv = g.n_vertices
    loc = g.vertex_local_index()
    cols = [[] for _ in range(nv)]
    for e in range(g.n_obs):
        vc, vp = int(g.obs_cam[e]), int(g.obs_pt[e])
        r, c = min(vc, vp), max(vc, vp)
        cols[c].append((r, e))
    col_dims = np.where(g.vtype == 0, 6, 3).astype(np.uint64)
    col_ptr = [0]
    row_idx, vals = [], []
    for v in range(nv):
        for r, e in sorted(cols[v]):
            row_idx.append(r)
            w = W[e].reshape(3, 6).T  # 6x3
            blk = w if g.vtype[v] == 1 else w.T  # column vertex is the point -> 6x3, else 3x6
            vals.append(blk.T.ravel())  # column-major
        row_idx.append(v)
        d = U[loc[v]].reshape(6, 6) if g.vtype[v] == 0 else V[loc[v]].reshape(3, 3)
        vals.append(d.ravel())  # symmetric: row/column-major agree
        col_ptr.append(len(row_idx))
    return col_dims, np.array(col_ptr, np.uint64), np.array(row_idx, np.uint64), np.concatenate(vals)


# ---- SE(2) pose graphs ------------------------------------------------------------------------------------------

def _pose_args(g, poses=None):
    st = np.ascontiguousarray(g.poses if poses is None else poses, np.float64).copy()
    ef = np.ascontiguousarray(g.e_from, np.uint64)
    et = np.ascontiguousarray(g.e_to, np.uint64)
    z = np.ascontiguousarray(g.z, np.float64)
    info = np.ascontiguousarray(g.info, np.float64)
    keep = (st, ef, et, z, info)
    args = [C.c_size_t(st.shape[0]), _p(st, C.c_double), C.c_size_t(ef.shape[0]), _p(ef, C.c_uint64), _p(et, C.c_uint64),
            _p(z, C.c_double), _p(info, C.c_double)]
    return args, keep


def _fn(g, name):
    return getattr(lib(), ("spo_se2_" if g.dim == 3 else "spo_se3_") + name)


def pose_chi2(g, poses=None) -> float:
    args, keep = _pose_args(g, poses)
    v = C.c_double()
    assert _fn(g, "chi2")(*args, C.byref(v)) == 0
    return v.value


def pose_linearise_dense(g, poses=None):
    """Dense lambda (n x n, symmetric) and eta of the SE(2) / SE(3) graph at the given poses."""
    args, keep = _pose_args(g, poses)
    n = keep[0].shape[0] * g.dim
    lam, eta = np.zeros((n, n)), np.zeros(n)
    assert _fn(g, "linearise_dense")(*args, _p(lam, C.c_double), _p(eta, C.c_double)) == 0
    return lam, eta  # symmetric: row/column-major agree


def pose_optimize(g, max_iter=5, min_dx=0.0, linear_solver=None):
    """The reference's Gauss-Newton loop. linear_solver(lambda, eta) -> (status, dx), if given, takes the place of the
    oracle's own dense solve (the reference's linear-solver slot); lambda is dense and symmetric."""
    if linear_solver is not None:
        errors = []

        def cb(n, lam, eta):
            try:
                rc, dx = linear_solver(_arr(lam, n * n).reshape(n, n), _arr(eta, n).copy())
                if rc == 0:
                    _arr(eta, n)[:] = dx
                return rc
            except BaseException as ex:  # stops the C loop; raised again once it has returned
                errors.append(ex)
                return -1
        fn = _POSE_SOLVER(cb)
        lib().spo_set_pose_linear_solver(fn)
        try:
            r = pose_optimize(g, max_iter, min_dx)
        finally:
            lib().spo_set_pose_linear_solver(None)
        if errors:
            raise errors[0]
        return r
    args, keep = _pose_args(g)
    out, norms = np.zeros(3), np.zeros(max(max_iter, 1))
    rc = _fn(g, "optimize")(*args, C.c_size_t(max_iter), C.c_double(min_dx), _p(out, C.c_double), _p(norms, C.c_double))
    return dict(status=rc, chi2_initial=out[0], chi2_final=out[1], n_solves=int(out[2]), dx_norms=norms[:int(out[2])],
                poses=keep[0])


se2_chi2, se2_linearise_dense, se2_optimize = pose_chi2, pose_linearise_dense, pose_optimize
