"""The block-sparse Cholesky (sparse_chol.cu) against a dense LAPACK reference, in each of its three execution regimes:
levels of the elimination tree on a cooperative grid, the narrow tail of the levels on a single CTA, and the dense root
front factored by the dense Cholesky. The regime a case runs is read from the SPP_SPARSE_VERBOSE line of the symbolic
analysis, so a case fails when it no longer runs the code path it was built for.

Every case checks, against the dense matrix: the factor R (R^T R = P A P^T) entry by entry, that the reference factor has
nothing outside the returned block pattern (the symbolic fill is complete), the forward error of the solution and its
backward error in extended precision. It also covers the spp_chol_* slot and the pose path sharing one analysis."""
import functools
import re

import numpy as np
import pytest
import scipy.linalg

from slam_plus_plus_b200 import capi, graphs

pytestmark = pytest.mark.gpu

ROOT_MAX_SCALARS = 6144  # SC_ROOT_MAX_SCALARS: the widest dense root front


# ---- block patterns: upper block CSC, rows ascending, diagonal present (the layout spp_chol_symbolic takes) -----------

def pattern(cols):
    """cols[c] = the rows of block column c (including c) -> (col_ptr, row_idx)"""
    cols = [sorted(set(r) | {c}) for c, r in enumerate(cols)]
    cp = np.concatenate([[0], np.cumsum([len(r) for r in cols])]).astype(np.uint64)
    return cp, np.array([r for rs in cols for r in rs], np.uint64)


def chain(n):
    return pattern([[c - 1] if c else [] for c in range(n)])


def arrow(n_leaves):
    """n_leaves diagonal-only columns and a hub coupled to all of them, ordered last"""
    return pattern([[] for _ in range(n_leaves)] + [list(range(n_leaves))])


def grid(w, h):
    """2D 4-neighbour grid, vertex x + w y"""
    return pattern([([c - 1] if c % w else []) + ([c - w] if c >= w else []) for c in range(w * h)])


def full(n):
    return pattern([list(range(c)) for c in range(n)])


def block_diagonal(*parts):
    cols, off = [], 0
    for cp, ri in parts:
        n = len(cp) - 1
        cols += [[int(r) + off for r in ri[cp[c]:cp[c + 1]]] for c in range(n)]
        off += n
    return pattern(cols)


def forest():
    """several elimination trees side by side: two chains, an arrow and diagonal-only columns"""
    return block_diagonal(chain(40), chain(60), arrow(100), pattern([[] for _ in range(20)]))


def random_order(n, seed=7):
    return np.random.default_rng(seed).permutation(n)


# ---- values, dense form, references -----------------------------------------------------------------------------------

def block_cols(cp):
    return np.repeat(np.arange(len(cp) - 1), np.diff(cp.astype(np.int64)))


def make_values(cp, ri, B, seed=0):
    """Values in the slot's layout (column-major B x B blocks in structure order, full symmetric diagonal blocks):
    random off-diagonal blocks; every diagonal entry exceeds the absolute sum of the other entries of its row by
    c = 1 + max row sum / 100, so the eigenvalues lie in [c, 2 max row sum + c] (Gershgorin) and cond < 201 for
    large row sums."""
    rng = np.random.default_rng(seed)
    ri = ri.astype(np.int64)
    col = block_cols(cp)
    ar = np.arange(B)
    blk = rng.uniform(-1, 1, (len(ri), B, B))  # blk[k, r, c] = element (r, c) of block k
    diag = ri == col
    blk[diag] = (blk[diag] + blk[diag].transpose(0, 2, 1)) / 2
    a = np.abs(blk)
    rs = np.zeros(B * (len(cp) - 1))
    np.add.at(rs, ri[~diag, None] * B + ar, a[~diag].sum(2))
    np.add.at(rs, col[~diag, None] * B + ar, a[~diag].sum(1))
    kd = np.nonzero(diag)[0]
    sd = ri[kd, None] * B + ar
    rs[sd] += a[kd].sum(2) - a[kd][:, ar, ar]
    blk[kd[:, None], ar, ar] = rs[sd] + 1 + rs.max() / 100
    return blk.transpose(0, 2, 1).ravel()


def blocks_of(cp, ri, vals, B):
    """(rows, cols, blocks[k, r, c]) of the upper structure; diagonal blocks are read from their upper triangle"""
    blk = np.asarray(vals, np.float64).reshape(-1, B, B).transpose(0, 2, 1).copy()
    ri, col = ri.astype(np.int64), block_cols(cp)
    d = ri == col
    blk[d] = np.triu(blk[d]) + np.triu(blk[d], 1).transpose(0, 2, 1)
    return ri, col, blk


def dense(col_ptr, row_idx, vals, B):
    ri, col, blk = blocks_of(col_ptr, row_idx, vals, B)
    ar = np.arange(B)
    n = (len(col_ptr) - 1) * B
    A = np.zeros((n, n))
    rr, cc = ri[:, None, None] * B + ar[None, :, None], col[:, None, None] * B + ar[None, None, :]
    A[rr, cc] = blk
    A[cc, rr] = blk
    return A


def cond(cp, ri, vals, B):
    """2-norm condition number of the SPD matrix; above 2000 scalars the two extreme eigenvalues by Lanczos on the
    sparse matrix (a dense eigensolver takes seconds there)"""
    if (len(cp) - 1) * B <= 2000:
        w = np.linalg.eigvalsh(dense(cp, ri, vals, B))
        lo, hi = w[0], w[-1]
    else:
        import scipy.sparse
        import scipy.sparse.linalg
        rows, col, blk = blocks_of(cp, ri, vals, B)
        ar = np.arange(B)
        rr = np.broadcast_to(rows[:, None, None] * B + ar[:, None], blk.shape)
        cc = np.broadcast_to(col[:, None, None] * B + ar, blk.shape)
        off = rows != col
        A = scipy.sparse.csr_matrix((np.concatenate([blk.ravel(), blk[off].ravel()]),
                                     (np.concatenate([rr.ravel(), cc[off].ravel()]),
                                      np.concatenate([cc.ravel(), rr[off].ravel()]))), shape=(len(ar) * (len(cp) - 1),) * 2)
        hi = scipy.sparse.linalg.eigsh(A, 1, which="LA", tol=1e-10, return_eigenvectors=False)[0]
        lo = scipy.sparse.linalg.eigsh(A, 1, which="SA", tol=1e-10, return_eigenvectors=False)[0]
    assert lo > 0
    return hi / lo


def backward_error(cp, ri, vals, B, x, b):
    """||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf), the product and the residual in extended precision"""
    rows, col, blk = blocks_of(cp, ri, vals, B)
    ar = np.arange(B)
    xl, bl = np.asarray(x, np.longdouble), np.asarray(b, np.longdouble)
    bk = blk.astype(np.longdouble)
    y = np.zeros(len(xl), np.longdouble)
    ir, ic = rows[:, None] * B + ar, col[:, None] * B + ar
    np.add.at(y, ir, np.matmul(bk, xl[ic][:, :, None])[:, :, 0])
    off = rows != col
    np.add.at(y, ic[off], np.matmul(bk[off].transpose(0, 2, 1), xl[ir[off]][:, :, None])[:, :, 0])
    rs = np.zeros(len(xl))
    np.add.at(rs, ir, np.abs(blk).sum(2))
    np.add.at(rs, ic[off], np.abs(blk[off]).sum(1))
    den = np.longdouble(rs.max()) * np.max(np.abs(xl)) + np.max(np.abs(bl))
    return float(np.max(np.abs(bl - y)) / den)


def factor_blocks(R_cp, R_ri, R_vals, B):
    """the block CSC of chol_get_factor -> rows, cols, blocks[k, r, c]"""
    return R_ri.astype(np.int64), block_cols(R_cp), R_vals.reshape(-1, B, B).transpose(0, 2, 1)


def scalar_perm(order, B):
    return (np.asarray(order, np.int64)[:, None] * B + np.arange(B)).ravel()


def check_against_dense(ctx, cp, ri, vals, B, order, x, b):
    """factor entry by entry, fill of the pattern, forward and backward error of x"""
    n = len(cp) - 1
    A = dense(cp, ri, vals, B)
    p = scalar_perm(order, B)
    R_ref = np.linalg.cholesky(A[np.ix_(p, p)]).T
    del A
    x_ref = np.empty_like(x)  # the dense Cholesky of the same permuted matrix (a third of numpy.linalg.solve's time)
    x_ref[p] = scipy.linalg.cho_solve((R_ref, False), b[p])
    assert np.linalg.norm(x - x_ref) <= 1e-12 * np.linalg.norm(x_ref)
    assert backward_error(cp, ri, vals, B, x, b) <= 1e-13
    rows, cols, Rb = factor_blocks(*ctx.chol_get_factor(n, B), B)
    assert np.all(rows <= cols)
    ar = np.arange(B)
    rr, cc = rows[:, None, None] * B + ar[None, :, None], cols[:, None, None] * B + ar[None, None, :]
    scale = np.abs(R_ref).max()
    assert np.abs(Rb - R_ref[rr, cc]).max() <= 1e-12 * scale
    R_ref[rr, cc] = 0  # what is left lies outside the block pattern of the factor: must be zero
    assert np.abs(R_ref).max() <= 1e-14 * scale


# ---- regime: the SPP_SPARSE_VERBOSE line of the analysis ----------------------------------------------------------------

VERBOSE_RE = re.compile(r"\[spp sparse chol\] n (\d+) \(B = (\d+)\), A blocks \d+, L blocks (\d+), levels (\d+) "
                        r"\(cooperative 0\.\.(\d+), single CTA \.\.(\d+)\), dense root front (\d+) columns")


def last_regime(capfd):
    lines = VERBOSE_RE.findall(capfd.readouterr().err)
    assert lines, "no SPP_SPARSE_VERBOSE line: the analysis did not run"
    n, B, nl, levels, T, N, m = map(int, lines[-1])
    return dict(n=n, B=B, L_blocks=nl, levels=levels, T=T, N=N, m=m)


def assert_regime(rg, coop, single, root):
    """root: 0 (none), "all" (the whole matrix is the root front) or "part" (0 < m < n)"""
    assert (rg["T"] > 0) == coop, rg
    assert (rg["T"] < rg["N"]) == single, rg
    if root == "all":
        assert rg["m"] == rg["n"] and rg["N"] == 0, rg
    elif root == "part":
        assert 0 < rg["m"] < rg["n"], rg
    else:
        assert rg["m"] == 0, rg


@pytest.fixture
def verbose(monkeypatch):
    monkeypatch.setenv("SPP_SPARSE_VERBOSE", "1")
    monkeypatch.delenv("SPP_SPARSE_NO_ROOT", raising=False)
    return monkeypatch


@pytest.fixture(scope="module")
def sctx():
    c = capi.Context(0)
    yield c
    c.close()


# ---- cases: structure, ordering and the regime each must run ---------------------------------------------------------

MIXED_GRID = (32, 32)  # n B <= 6144 at B = 6: the dense reference and its condition number stay cheap
BAD_GRID = (20, 20)    # a bad ordering makes the factor nearly dense: the update lists grow with the cube of n


def identity(cp):
    return np.arange(len(cp) - 1)


def case_structure(name, B):
    """-> (col_ptr, row_idx, order passed to chol_symbolic (None: the library's AMD), expected regime)"""
    if name == "whole_root":
        cp, ri = chain(300)
        return cp, ri, identity(cp), (False, False, "all")
    if name == "root_boundary":  # the root front at its widest
        cp, ri = chain(ROOT_MAX_SCALARS // B)
        return cp, ri, identity(cp), (False, False, "all")
    if name == "root_boundary_plus_one":  # one block column more: no root, every level on the single CTA
        cp, ri = chain(ROOT_MAX_SCALARS // B + 1)
        return cp, ri, identity(cp), (False, True, 0)
    if name == "unpadded_root":  # 606 scalars: the dense solver pads the front to a multiple of 128
        cp, ri = chain(101)
        return cp, ri, identity(cp), (False, False, "all")
    if name == "levels_only":  # the leaves on the cooperative grid, the hub on the single CTA
        cp, ri = arrow(500)
        return cp, ri, identity(cp), (True, True, 0)
    if name == "mixed":
        # the root front takes the top levels down to the first one wider than 16 columns, and the single CTA only
        # levels of at most 8: next to a root front every level runs on the cooperative grid
        cp, ri = grid(*MIXED_GRID)
        return cp, ri, None, (True, False, "part")
    if name == "mixed_no_root":  # SPP_SPARSE_NO_ROOT: the narrow top of the tree goes to the single CTA instead
        cp, ri = grid(*MIXED_GRID)
        return cp, ri, None, (True, True, 0)
    if name == "forest":  # the root front holds the tops of several trees; level 0 is wide
        cp, ri = forest()
        return cp, ri, identity(cp), (True, False, "part")
    if name == "dense":
        cp, ri = full(64)
        return cp, ri, identity(cp), (False, False, "all")
    if name == "random_order":
        cp, ri = grid(*BAD_GRID)
        return cp, ri, random_order(len(cp) - 1), (True, False, "part")
    if name == "reversed_amd":
        cp, ri = grid(*BAD_GRID)
        return cp, ri, capi.block_ordering(cp, ri).astype(np.int64)[::-1].copy(), (True, False, "part")
    raise KeyError(name)


CASES = [(name, B) for name in ("whole_root", "root_boundary", "root_boundary_plus_one", "levels_only", "forest",
                                "random_order", "reversed_amd") for B in (2, 3, 6)]
CASES += [("unpadded_root", 6), ("dense", 6)]
CASES += [(name, B) for name in ("mixed", "mixed_no_root") for B in (3, 6)]


@functools.lru_cache(maxsize=None)
def system(name, B):
    """structure, values and right-hand side of a case; the condition number is asserted once per matrix"""
    cp, ri, order, expect = case_structure(name, B)
    vals = make_values(cp, ri, B, seed=B)
    n = len(cp) - 1
    if n * B <= 6200:
        assert cond(cp, ri, vals, B) <= 1e4
    b = np.random.default_rng(100 + B).standard_normal(n * B)
    return cp, ri, order, expect, vals, b


def run_case(ctx, monkeypatch, capfd, name, B):
    if name.endswith("no_root"):
        monkeypatch.setenv("SPP_SPARSE_NO_ROOT", "1")
    cp, ri, order, expect, vals, b = system(name, B)
    capfd.readouterr()
    p = ctx.chol_symbolic(B, cp, ri, order)
    rg = last_regime(capfd)
    assert (rg["n"], rg["B"]) == (len(cp) - 1, B)
    assert_regime(rg, *expect)
    if order is not None:
        assert np.array_equal(p, order)
    x = ctx.chol_solve(vals, b)
    return p, x, rg


@pytest.mark.parametrize("name,B", CASES)
def test_factor_and_solve_against_dense(sctx, verbose, capfd, name, B):
    p, x, rg = run_case(sctx, verbose, capfd, name, B)
    cp, ri, _, _, vals, b = system(name, B)
    check_against_dense(sctx, cp, ri, vals, B, p, x, b)
    if name == "forest":
        assert rg["m"] == 39 + 59 + 1  # all chain columns but the first of each, and the hub
    if name in ("random_order", "reversed_amd"):
        assert rg["L_blocks"] >= 4 * len(ri)  # heavy fill


@pytest.mark.parametrize("B", [3, 6])
def test_no_root_equals_root_run(sctx, verbose, capfd, B):
    """the same system with and without the dense root front: factor and solution within 1e-12"""
    p1, x1, _ = run_case(sctx, verbose, capfd, "mixed", B)
    R1 = sctx.chol_get_factor(len(p1), B)
    p2, x2, _ = run_case(sctx, verbose, capfd, "mixed_no_root", B)
    R2 = sctx.chol_get_factor(len(p2), B)
    assert np.array_equal(p1, p2)
    assert np.array_equal(R1[0], R2[0]) and np.array_equal(R1[1], R2[1])
    assert np.abs(R1[2] - R2[2]).max() <= 1e-12 * np.abs(R1[2]).max()
    assert np.abs(x1 - x2).max() <= 1e-12 * np.abs(x1).max()


@pytest.mark.parametrize("B", [3, 6])
def test_reproducible(sctx, verbose, capfd, B):
    """two solves of the mixed system: bit-identical solution and factor"""
    n = len(system("mixed", B)[0]) - 1
    _, x1, _ = run_case(sctx, verbose, capfd, "mixed", B)
    R1 = sctx.chol_get_factor(n, B)
    cp, ri, _, _, vals, b = system("mixed", B)
    x2 = sctx.chol_solve(vals, b)
    R2 = sctx.chol_get_factor(n, B)
    assert np.array_equal(x1, x2)
    assert all(np.array_equal(u, v) for u, v in zip(R1, R2))


# ---- not positive definite, in each regime ------------------------------------------------------------------------------

def set_diagonal_entry(cp, ri, vals, B, col, value):
    """vals with the first diagonal entry of block column col set to value"""
    v = vals.copy()
    k = int(cp[col + 1]) - 1  # the diagonal block is the last of its column
    assert int(ri[k]) == col
    v[k * B * B] = value
    return v


NOT_POSDEF = {  # case -> (block column made indefinite, regime)
    "levels_only_leaf": ("levels_only", 7, (True, True, 0)),
    "levels_only_hub": ("levels_only", 500, (True, True, 0)),
    "single_cta_chain": ("root_boundary_plus_one", None, (False, True, 0)),
    "whole_root": ("whole_root", 150, (False, False, "all")),
}


@pytest.mark.parametrize("B", [2, 3, 6])
@pytest.mark.parametrize("which", list(NOT_POSDEF))
def test_not_posdef_then_good_solves(verbose, capfd, which, B):
    name, col, expect = NOT_POSDEF[which]
    cp, ri, order, _, vals, b = system(name, B)
    n = len(cp) - 1
    col = n // 2 if col is None else col
    ctx = capi.Context(0)
    capfd.readouterr()
    ctx.chol_symbolic(B, cp, ri, order)
    assert_regime(last_regime(capfd), *expect)
    with pytest.raises(capi.NotPositiveDefinite):
        ctx.chol_solve(set_diagonal_entry(cp, ri, vals, B, col, -1e6), b)
    # the same analysis, good values
    x = ctx.chol_solve(vals, b)
    assert backward_error(cp, ri, vals, B, x, b) <= 1e-13
    # a new analysis of another structure on the same context
    cp2, ri2, _, _, vals2, b2 = system("forest", B)
    p2 = ctx.chol_symbolic(B, cp2, ri2)
    x2 = ctx.chol_solve(vals2, b2)
    check_against_dense(ctx, cp2, ri2, vals2, B, p2, x2, b2)
    ctx.close()


def test_block_size_changes_on_one_context(verbose, capfd):
    """analyses of B = 2, 6, 3, 2 on one context, each on the cooperative grid and the single CTA"""
    ctx = capi.Context(0)
    for B in (2, 6, 3, 2):
        p, x, _ = run_case(ctx, verbose, capfd, "levels_only", B)
        cp, ri, _, _, vals, b = system("levels_only", B)
        check_against_dense(ctx, cp, ri, vals, B, p, x, b)
    ctx.close()


# ---- the pose path ------------------------------------------------------------------------------------------------------

POSE_CASES = {  # graph, regime with the root front, regime under SPP_SPARSE_NO_ROOT
    "manhattan_1000_300": (lambda: graphs.make_manhattan(1000, 300), (True, False, "part"), (True, True, 0)),
    "odometry_chain_400": (lambda: graphs.make_manhattan(400, 0), (False, False, "all"), (False, True, 0)),
    "sphere_12x12": (lambda: graphs.make_sphere(12, 12), (True, False, "part"), (True, True, 0)),
}


def pose_solve_checked(ctx, dim):
    """one linearisation and solve; the increment against the pose path's own lambda: backward error in extended
    precision (pose systems have cond 1e8 .. 1e10, so the forward error says little)"""
    ctx.pose_linearise()
    cp, ri, vals, eta = ctx.pose_get_lambda()
    dx = ctx.pose_solve_step()
    assert backward_error(cp, ri, vals, dim, dx, eta) <= 1e-13
    return cp, ri, vals, dx


@pytest.mark.parametrize("no_root", [False, True])
@pytest.mark.parametrize("name", list(POSE_CASES))
def test_pose_solve_against_its_lambda(sctx, verbose, capfd, name, no_root):
    make, expect, expect_no_root = POSE_CASES[name]
    if no_root:
        verbose.setenv("SPP_SPARSE_NO_ROOT", "1")
    g = make()
    dim = g.poses.shape[1]
    sctx.pose_set_graph(g)
    capfd.readouterr()
    pose_solve_checked(sctx, dim)
    rg = last_regime(capfd)
    assert (rg["n"], rg["B"]) == g.poses.shape
    assert_regime(rg, *(expect_no_root if no_root else expect))


# ---- the slot and the pose path on one context ------------------------------------------------------------------------

def assert_pose_factor(ctx, cp, ri, vals, dim):
    """chol_get_factor holds the factor of the pose solve: R^T R = P lambda P^T for the library's ordering of lambda"""
    n = len(cp) - 1
    rows, cols, Rb = factor_blocks(*ctx.chol_get_factor(n, dim), dim)
    ar = np.arange(dim)
    R = np.zeros((n * dim, n * dim))
    R[rows[:, None, None] * dim + ar[:, None], cols[:, None, None] * dim + ar] = Rb
    p = scalar_perm(capi.block_ordering(cp, ri).astype(np.int64), dim)
    A = dense(cp, ri, vals, dim)[np.ix_(p, p)]
    assert np.abs(R.T @ R - A).max() <= 1e-13 * np.abs(A).max()


def solve_or_error(f, *args):
    """the result of f, or the library's refusal: on a wrong analysis a solve may also meet a non-positive pivot"""
    try:
        return f(*args)
    except (capi.SppError, capi.NotPositiveDefinite) as e:
        return e


def test_pose_solve_after_slot_analysis():
    """pose solve, spp_chol_symbolic of another structure, pose solve again: the second pose solve must analyse the
    pose graph again, not factor its values with the slot's structure. The slot structure is smaller than the pose
    graph in blocks and in scalars."""
    ctx = capi.Context(0)
    g = graphs.make_manhattan(300, 80)
    ctx.pose_set_graph(g)
    cp, ri, vals, dx1 = pose_solve_checked(ctx, 3)
    s_cp, s_ri = chain(100)
    s_vals, s_b = make_values(s_cp, s_ri, 2), np.random.default_rng(1).standard_normal(200)
    assert len(s_ri) * 4 < len(ri) * 9 and 200 < 900
    ctx.chol_symbolic(2, s_cp, s_ri, identity(s_cp))
    dx2 = solve_or_error(ctx.pose_solve_step)
    assert isinstance(dx2, np.ndarray) and np.array_equal(dx2, dx1), dx2
    assert_pose_factor(ctx, cp, ri, vals, 3)
    # the slot does not keep its structure: its analysis has to be made again
    r = solve_or_error(ctx.chol_solve, s_vals, s_b)
    assert isinstance(r, capi.SppError) and "spp_chol_symbolic" in str(r), r
    p = ctx.chol_symbolic(2, s_cp, s_ri, identity(s_cp))
    check_against_dense(ctx, s_cp, s_ri, s_vals, 2, p, ctx.chol_solve(s_vals, s_b), s_b)
    ctx.close()


def test_slot_solve_after_pose_solve():
    """spp_chol_symbolic, a pose solve, spp_chol_solve with the values of the slot's structure: the slot must refuse
    rather than solve with the pose graph's analysis. The pose graph is smaller than the slot's arrays."""
    ctx = capi.Context(0)
    a_cp, a_ri = arrow(200)
    a_vals, a_b = make_values(a_cp, a_ri, 6), np.random.default_rng(2).standard_normal(201 * 6)
    ctx.chol_symbolic(6, a_cp, a_ri, identity(a_cp))
    g = graphs.make_manhattan(60, 15)
    ctx.pose_set_graph(g)
    cp, ri, vals, dx1 = pose_solve_checked(ctx, 3)
    assert len(ri) * 9 < len(a_ri) * 36 and 60 * 3 < 201 * 6
    r = solve_or_error(ctx.chol_solve, a_vals, a_b)
    assert isinstance(r, capi.SppError) and "spp_chol_symbolic" in str(r), r
    assert_pose_factor(ctx, cp, ri, vals, 3)  # the refused call left the pose solve's factor in place
    p = ctx.chol_symbolic(6, a_cp, a_ri, identity(a_cp))
    check_against_dense(ctx, a_cp, a_ri, a_vals, 6, p, ctx.chol_solve(a_vals, a_b), a_b)
    dx2 = ctx.pose_solve_step()
    assert np.array_equal(dx2, dx1)
    assert_pose_factor(ctx, cp, ri, vals, 3)
    ctx.close()
