"""The supernodal Cholesky of the reduced camera system (supernodal_chol.cu, selinv.cu) against a float64 dense
reference, in each of its execution regimes. One factorisation picks its code path per supernode and per update from
the panel shape: the factorisation of a panel of one diagonal block (ld = 128) on a side stream, the look-ahead panel
factorisation for 128 < ld < 1024, the dataflow kernel for ld >= 1024; the 128 x 64 or the 64 x 64 tile for an update;
the selected inversion on a side lane or on the main stream. Every case states the counts of these it must produce and
reads them from the SPP_SNODE_VERBOSE line of the analysis, so a case fails when it no longer runs the paths it was
built for.

A case is a list of landmarks, each with the cameras that see it (a landmark seen by cameras K makes K a clique of the
reduced camera system S), and a camera ordering (None: the library's AMD). Everything goes through slot 1
(spp_schur_symbolic / spp_schur_solve) on a lambda built here. Checks: the increment against a LAPACK solve of the
dense lambda (forward error) and in extended precision (backward error), the residual of the reduced system, the
block diagonal of (lambda + alpha I)^-1 by the selected inversion against a dense inverse, bit reproducibility (a second
solve, a solve after the marginals, the same pattern uploaded again, a solve after a failed factorisation), the
dataflow supernodes with the look-ahead factorisation instead, and a non-positive pivot in each regime."""
import functools
import re

import numpy as np
import pytest
import scipy.linalg

from slam_plus_plus_b200 import capi

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
KAPPA_MAX = 300.0  # every lambda below is asserted to have a 2-norm condition number at most this


def tol_forward(n):
    """relative forward error of a solve, and of the blocks of an inverse, against LAPACK: two backward-stable
    factorisations of a matrix with condition number kappa differ by about kappa eps times a slowly growing function
    of the size; 4 sqrt(n) kappa eps is 1.1e-11 at n = 3600 and the largest kappa allowed"""
    return 4 * np.sqrt(n) * KAPPA_MAX * EPS


def tol_backward(n):
    """normwise backward error ||eta - lambda dx||_inf / (||lambda||_inf ||dx||_inf + ||eta||_inf) in extended precision"""
    return 8 * np.sqrt(n) * EPS


# ---- cases ------------------------------------------------------------------------------------------------------------

class Cams:
    """hands out consecutive camera indices"""

    def __init__(self):
        self.n = 0

    def __call__(self, k):
        r = list(range(self.n, self.n + k))
        self.n += k
        return r


def sequence(n=160, seed=3):
    """a camera sequence: landmarks seen by 2 .. 5 consecutive cameras, a few loop closures"""
    rng = np.random.default_rng(seed)
    lms = []
    for c in range(n):
        for _ in range(2):
            w = int(rng.integers(2, 6))
            lms.append(list(range(c, min(n, c + w))))
    for _ in range(6):
        a = int(rng.integers(0, n - 20))
        b = int(rng.integers(a + 15, n))
        lms.append([a, a + 1, b, b - 1])
    return n, lms


def case_structure(name):
    """-> (cameras, landmarks, camera ordering or None, expected regime counts, cameras of one supernode).

    Counts: supernodes (ns), on the side streams / look-ahead / dataflow, largest ld and h (scalars), updates on the
    128 x 64 / 64 x 64 tiles, selected inversions on the side lanes. They were worked out on the host analysis with the
    solver's relaxed amalgamation (a supernode merges into its parent while the merge adds at most 5 % explicit zeros
    or stays within 16 block columns); an explicit ordering puts a leaf that must stay a supernode of its own away from
    its parent."""
    cams = Cams()
    if name == "lone":  # 12 roots with h = 0: the side streams are reused round-robin, no updates
        cams(12)
        return cams.n, [], None, dict(ns=12, side=12, look=0, flow=0, ld=128, h=0, t128=0, t64=0, lane=12), [5]
    m = re.fullmatch(r"clique(\d+)", name)
    if m:  # 21 / 22 cameras: ld 128 / 256 (side stream / look-ahead); 149 / 150: ld 896 / 1024 (look-ahead / dataflow)
        k = int(m.group(1))
        c = cams(k)
        ld = -(-6 * k // 128) * 128
        side, flow = ld == 128, ld >= 1024
        return cams.n, [c], None, dict(ns=1, side=int(side), look=int(not side and not flow), flow=int(flow), ld=ld, h=0,
                                       t128=0, t64=0, lane=int(side)), c
    if name == "arrow":  # 20 leaf groups of 4 on the side streams, each tied to 3 cameras of a look-ahead hub of 30
        hub = cams(30)
        lms = [hub]
        leaves = []
        for g in range(20):
            leaf = cams(4)
            leaves.append(leaf)
            lms.append(leaf + [hub[(3 * g + k) % 30] for k in range(3)])
        return cams.n, lms, None, dict(ns=21, side=20, look=1, flow=0, ld=256, h=18, t128=0, t64=20, lane=20), leaves[5]
    if name == "wide":
        # A (150 cameras, dataflow) -> P (137, look-ahead) -> G (30, look-ahead root). A's update into P: M = 6 x 129,
        # N = 6 x 129 + 1: 7 x 7 = 49 tiles (128 x 64). E (2 cameras, a structure 75 times as wide as its columns):
        # 128 rows in P and 22 in G, M = 768, N = 901: 6 x 8 = 48 tiles (128 x 64), and 2 x 2 into G (64 x 64).
        # D: 128 rows in P, 6 x 7 = 42 tiles (64 x 64). F merges into P. P -> G: 64 x 64, h = 132.
        A, E, D, F, P, G = cams(150), cams(2), cams(2), cams(2), cams(135), cams(30)
        lms = [G, P + G[:10], A + P[:129], E + P[:128] + G[:22], D + P[:128], F + P[:5]]
        return cams.n, lms, A + E + D + F + P + G, dict(ns=5, side=2, look=2, flow=1, ld=1024, h=900, t128=2, t64=3,
                                                        lane=2), E
    if name == "tall":
        # leaves of 20 cameras (ld 128, side streams) under a root of 342 (+ the third leaf, merged: dataflow, ld 2176):
        # the first leaf's structure is 342 cameras (h = 2052, padded 2112 > 2048: selected inversion on the main
        # stream), the second's 341 (h = 2046, padded 2048: on a side lane)
        P = cams(342)
        lms, leaves = [P], []
        for hh in (342, 341, 342):
            leaf = cams(20)
            leaves.append(leaf)
            lms.append(leaf + P[:hh])
        return cams.n, lms, sum(leaves, []) + P, dict(ns=3, side=2, look=0, flow=1, ld=2176, h=2052, t128=2, t64=0,
                                                      lane=1), leaves[0]
    if name == "edges":
        # leaves of 4 cameras tied to 21, 22 and 23 cameras of a look-ahead root: h = 126, 132, 138 (k_snode_gemv: two
        # chunks with a tail, three chunks with a tail of 4, ...); the panel has ld + round_up(h + 1, 128) columns, so
        # the rhs column at ld + h is the last of its tile at h = 126 and opens a new tile at h = 132
        P = cams(24)
        lms, leaves = [P], []
        for hh in (21, 22, 23, 24):
            leaf = cams(4)
            leaves.append(leaf)
            lms.append(leaf + P[:hh])
        return cams.n, lms, sum(leaves, []) + P, dict(ns=4, side=3, look=1, flow=0, ld=256, h=138, t128=0, t64=3,
                                                      lane=3), leaves[0]
    if name == "sequence_amd":
        n, lms = sequence()
        return n, lms, None, dict(ns=18, side=18, look=0, flow=0, ld=128, h=36, t128=0, t64=31, lane=18), \
            [3, 4] + list(range(6, 15))
    if name == "sequence_random":  # a random ordering: heavy fill, 576 updates
        n, lms = sequence()
        return n, lms, np.random.default_rng(11).permutation(n), dict(ns=99, side=98, look=1, flow=0, ld=256, h=252,
                                                                      t128=0, t64=576, lane=98), [128]
    raise KeyError(name)


CASES = ["lone", "clique21", "clique22", "clique149", "clique150", "arrow", "wide", "tall", "edges", "sequence_amd",
         "sequence_random"]
DATAFLOW_CASES = ["clique150", "wide", "tall"]


# ---- lambda in the slot's layout ---------------------------------------------------------------------------------------

class System:
    """lambda of a case: cameras are block columns 0 .. C-1 (6 wide), landmarks C .. C+P-1 (3 wide); every camera also
    sees a landmark of its own and camera 0 two more, so that the cameras are fewer than half the block columns, as the
    slot's guided ordering requires"""

    def __init__(self, name, seed=0):
        self.name = name
        C, lms, order, self.expect, self.focus = case_structure(name)
        lms = [sorted(set(k)) for k in lms] + [[c] for c in range(C)] + [[0], [0]]
        self.C, self.P, self.lms = C, len(lms), lms
        self.order = None if order is None else np.asarray(order, np.int64)
        self.col_dims = np.array([6] * C + [3] * self.P, np.uint64)
        base = np.concatenate([[0], np.cumsum(self.col_dims.astype(np.int64))])
        self.base, self.N = base, int(base[-1])
        cols = [[c] for c in range(C)] + [k + [C + p] for p, k in enumerate(lms)]  # rows ascending, diagonal last
        self.col_ptr = np.concatenate([[0], np.cumsum([len(r) for r in cols])]).astype(np.uint64)
        self.row_idx = np.array([r for rs in cols for r in rs], np.uint64)
        self.cols = cols
        self.A = self.make_dense(seed)
        self.vals = self.values(self.A)

    def make_dense(self, seed):
        """random blocks on the pattern; every diagonal entry exceeds the absolute sum of the other entries of its row
        by c = 1 + max row sum / 100, so the eigenvalues lie in [c, 2 max row sum + c] (Gershgorin): cond < 201"""
        rng = np.random.default_rng(seed)
        A = np.zeros((self.N, self.N))
        b = self.base
        for c, rows in enumerate(self.cols):
            for r in rows:
                blk = rng.uniform(-1, 1, (b[r + 1] - b[r], b[c + 1] - b[c]))
                if r == c:
                    blk = (blk + blk.T) / 2
                A[b[r]:b[r + 1], b[c]:b[c + 1]] = blk
                A[b[c]:b[c + 1], b[r]:b[r + 1]] = blk.T
        np.fill_diagonal(A, 0)
        rs = np.abs(A).sum(1)
        np.fill_diagonal(A, rs + 1 + rs.max() / 100)
        return A

    def values(self, A):
        """the slot's value array: the blocks of the upper structure, column-major, in structure order"""
        b = self.base
        return np.concatenate([A[b[r]:b[r + 1], b[c]:b[c + 1]].ravel(order="F") for c, rows in enumerate(self.cols)
                               for r in rows])

    def diag_index(self, cam):
        """index in the value array of the first diagonal entry of camera cam (its column holds only the diagonal)"""
        return 36 * cam

    def rhs(self, kind):
        rng = np.random.default_rng(17)
        if kind == "random":
            return rng.standard_normal(self.N)
        eta = np.zeros(self.N)  # non-zero only on the cameras of one supernode
        for c in self.focus:
            eta[6 * c:6 * c + 6] = rng.standard_normal(6)
        return eta


@functools.lru_cache(maxsize=None)
def system(name, seed=0):
    return System(name, seed)


@functools.lru_cache(maxsize=None)
def kappa(name, seed=0):
    A = system(name, seed).A
    if A.shape[0] <= 1500:
        w = np.linalg.eigvalsh(A)
        lo, hi = w[0], w[-1]
    else:  # the two extreme eigenvalues by Lanczos on the sparse matrix
        import scipy.sparse
        import scipy.sparse.linalg
        S = scipy.sparse.csr_matrix(A)
        hi = scipy.sparse.linalg.eigsh(S, 1, which="LA", tol=1e-10, return_eigenvectors=False)[0]
        lo = scipy.sparse.linalg.eigsh(S, 1, which="SA", tol=1e-10, return_eigenvectors=False)[0]
    assert lo > 0
    return hi / lo


def backward_error(A, x, b):
    Al, xl, bl = A.astype(np.longdouble), np.asarray(x, np.longdouble), np.asarray(b, np.longdouble)
    r = bl - Al @ xl
    den = np.longdouble(np.abs(A).sum(1).max()) * np.max(np.abs(xl)) + np.max(np.abs(bl))
    return float(np.max(np.abs(r)) / den)


def marginal_blocks(sy, alpha):
    """block diagonal of (lambda + alpha I)^-1 from a float64 dense inverse: (C, 6, 6), (P, 3, 3)"""
    Z = scipy.linalg.cho_solve(scipy.linalg.cho_factor(sy.A + alpha * np.eye(sy.N)), np.eye(sy.N))
    b = sy.base
    cc = np.stack([Z[b[i]:b[i + 1], b[i]:b[i + 1]] for i in range(sy.C)])
    pc = np.stack([Z[b[i]:b[i + 1], b[i]:b[i + 1]] for i in range(sy.C, sy.C + sy.P)])
    return cc, pc


# ---- regime: the SPP_SNODE_VERBOSE line of the analysis ----------------------------------------------------------------

VERBOSE_RE = re.compile(r"\[spp snode\] n (\d+), S blocks \d+, supernodes (\d+), .*?, (\d+) updates; supernodes on the "
                        r"side streams (\d+), look-ahead (\d+), dataflow (\d+) \(ld >= \d+\); largest ld (\d+), largest "
                        r"h (\d+); updates on 128x64 tiles (\d+), on 64x64 tiles (\d+); selected inversion on the side "
                        r"lanes (\d+)")


def regime_lines(capfd):
    return [dict(zip(("n", "ns", "upd", "side", "look", "flow", "ld", "h", "t128", "t64", "lane"), map(int, m)))
            for m in VERBOSE_RE.findall(capfd.readouterr().err)]


def assert_regime(capfd, sy):
    lines = regime_lines(capfd)
    assert len(lines) == 1, "expected one SPP_SNODE_VERBOSE line: the analysis ran %d times" % len(lines)
    rg = lines[0]
    assert rg["n"] == sy.C and rg["upd"] == rg["t128"] + rg["t64"], rg
    got = {k: rg[k] for k in sy.expect}
    assert got == sy.expect, (got, sy.expect)


@pytest.fixture
def verbose(monkeypatch):
    monkeypatch.setenv("SPP_SNODE_VERBOSE", "1")
    monkeypatch.setenv("SPP_SNODE_NO_REUSE", "1")
    monkeypatch.delenv("SPP_CHOL_DATAFLOW", raising=False)
    return monkeypatch


def new_context(sy):
    """a context with slot 1 set up for the case: block-sparse reduced camera system, the case's ordering"""
    ctx = capi.Context(0)
    order, cut = ctx.schur_symbolic(sy.col_dims, sy.col_ptr, sy.row_idx)
    assert cut == sy.C and np.array_equal(order, np.arange(sy.C + sy.P))
    ctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    ctx.schur_set_rcs_ordering(sy.order)
    return ctx


def solve(ctx, sy, vals=None, eta=None):
    return ctx.schur_solve(sy.vals if vals is None else vals, sy.rhs("random") if eta is None else eta)


# ---- solve and marginals against the dense reference, bit reproducibility -------------------------------------------

@pytest.mark.parametrize("name", CASES)
def test_solve_and_marginals_against_dense(verbose, capfd, name):
    sy = system(name)
    assert kappa(name) <= KAPPA_MAX
    tf, tb = tol_forward(sy.N), tol_backward(sy.N)
    cho = scipy.linalg.cho_factor(sy.A)
    ctx = new_context(sy)
    capfd.readouterr()
    first = {}
    for kind in ("random", "one_supernode"):
        eta = sy.rhs(kind)
        dx = solve(ctx, sy, eta=eta)
        if kind == "random":
            assert_regime(capfd, sy)
            info = ctx.schur_get_rcs_info()
            if sy.order is not None:
                assert np.array_equal(info["order"].astype(np.int64), sy.order)
        ref = scipy.linalg.cho_solve(cho, eta)
        err = np.linalg.norm(dx - ref) / np.linalg.norm(ref)
        assert err <= tf, (kind, err, tf)
        be = backward_error(sy.A, dx, eta)
        assert be <= tb, (kind, be, tb)
        assert ctx.schur_get_rcs_residual() < 1e-13
        first[kind] = dx
        assert np.array_equal(solve(ctx, sy, eta=eta), dx)  # a second solve: the same bits
    for alpha in (0.0, 10.0):
        cc, pc = ctx.schur_marginals_sparse(alpha)
        rc, rp = marginal_blocks(sy, alpha)
        ec, ep = np.abs(cc - rc).max() / np.abs(rc).max(), np.abs(pc - rp).max() / np.abs(rp).max()
        assert ec <= tf and ep <= tf, (alpha, ec, ep, tf)
        assert np.array_equal(cc, cc.transpose(0, 2, 1))
    # the marginals overwrote the panels: a solve after them gives the bits of a solve without them
    for kind in ("random", "one_supernode"):
        assert np.array_equal(solve(ctx, sy, eta=sy.rhs(kind)), first[kind])
    assert regime_lines(capfd) == []  # the same context kept its analysis
    ctx.close()


@pytest.mark.parametrize("name", ["lone", "clique22", "arrow", "wide", "edges", "sequence_random"])
def test_same_pattern_again_equals_fresh_context(monkeypatch, capfd, name):
    """the same block pattern uploaded again keeps the ordering, supernodes and panel layout; new values on it give the
    bits of a fresh context's analysis"""
    monkeypatch.setenv("SPP_SNODE_VERBOSE", "1")
    monkeypatch.delenv("SPP_SNODE_NO_REUSE", raising=False)
    monkeypatch.delenv("SPP_CHOL_DATAFLOW", raising=False)
    sy, sy2 = system(name), system(name, 1)
    assert kappa(name, 1) <= KAPPA_MAX
    eta = sy.rhs("random")
    capfd.readouterr()
    ctx = new_context(sy)
    solve(ctx, sy)
    assert len(regime_lines(capfd)) == 1
    ctx.schur_symbolic(sy.col_dims, sy.col_ptr, sy.row_idx)  # the same pattern again
    x_kept = solve(ctx, sy, sy2.vals, eta)
    assert regime_lines(capfd) == []  # the analysis was kept
    ctx.close()
    fresh = new_context(sy2)
    x_fresh = solve(fresh, sy2, sy2.vals, eta)
    assert len(regime_lines(capfd)) == 1
    fresh.close()
    assert np.array_equal(x_kept, x_fresh)
    ref = np.linalg.solve(sy2.A, eta)
    assert np.linalg.norm(x_fresh - ref) <= tol_forward(sy2.N) * np.linalg.norm(ref)


@pytest.mark.parametrize("name", DATAFLOW_CASES)
def test_dataflow_off_agrees_to_rounding(verbose, capfd, name):
    """SPP_CHOL_DATAFLOW=0 factors the dataflow supernodes with the look-ahead panel factorisation: another summation
    order, the same result to rounding (solve and marginals)"""
    sy = system(name)
    assert sy.expect["flow"] >= 1 and kappa(name) <= KAPPA_MAX
    tf = tol_forward(sy.N)
    out = {}
    for flag in ("1", "0"):
        verbose.setenv("SPP_CHOL_DATAFLOW", flag)
        ctx = new_context(sy)
        capfd.readouterr()
        x = solve(ctx, sy)
        assert_regime(capfd, sy)
        assert ctx.schur_get_rcs_residual() < 1e-13
        out[flag] = (x,) + ctx.schur_marginals_sparse(1.0)
        ctx.close()
    for a, b in zip(out["1"], out["0"]):
        assert np.abs(a - b).max() <= 2 * tf * np.abs(a).max()


# ---- a non-positive pivot in each regime ------------------------------------------------------------------------------

NOT_POSDEF = {  # which -> (case, camera made indefinite: the first failing pivot lies in its supernode)
    "side_stream_leaf": ("arrow", 30 + 4 * 5 + 1),
    "look_ahead_panel": ("wide", 150 + 6 + 40),     # P
    "dataflow_panel": ("wide", 100),                # A
    "look_ahead_root": ("arrow", 10),               # the hub
    "dataflow_root": ("tall", 200),
}


@pytest.mark.parametrize("which", list(NOT_POSDEF))
def test_not_posdef_then_good_solve(verbose, capfd, which):
    """one diagonal entry of a camera's U made very negative changes only that diagonal block of S, and the leading
    part of S before it stays positive definite: the factorisation meets its first non-positive pivot in that camera's
    supernode. The solve raises; the next solve with good values on the same context gives a fresh context's bits,
    whatever the failed factorisation left in the panels and in the inverses of the diagonal blocks."""
    name, cam = NOT_POSDEF[which]
    sy = system(name)
    bad = sy.vals.copy()
    bad[sy.diag_index(cam)] = -1e6
    eta = sy.rhs("random")
    ctx = new_context(sy)
    capfd.readouterr()
    with pytest.raises(capi.NotPositiveDefinite):
        ctx.schur_solve(bad, eta)
    assert_regime(capfd, sy)
    with pytest.raises(capi.SppError):
        ctx.schur_get_rcs_residual()  # nothing solved to check
    x = solve(ctx, sy, eta=eta)
    assert ctx.schur_get_rcs_residual() < 1e-13
    # the marginals of an indefinite lambda fail in the same place, then a good solve again
    with pytest.raises(capi.NotPositiveDefinite):
        ctx.schur_solve(bad, eta)
    with pytest.raises(capi.NotPositiveDefinite):
        ctx.schur_marginals_sparse(1.0)
    x_again = solve(ctx, sy, eta=eta)
    ctx.close()
    fresh = new_context(sy)
    x_fresh = solve(fresh, sy, eta=eta)
    fresh.close()
    assert np.array_equal(x, x_fresh) and np.array_equal(x_again, x_fresh)
    ref = scipy.linalg.cho_solve(scipy.linalg.cho_factor(sy.A), eta)
    assert np.linalg.norm(x - ref) <= tol_forward(sy.N) * np.linalg.norm(ref)
