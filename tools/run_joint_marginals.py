#!/usr/bin/env python
"""Development helper: joint marginals (spp_ba_joint_marginals), timed by phase in one process:
  - BAL-13682 shape after ba_linearise, supernodal path, alpha = 50: 1 000 seeded camera pairs that share no landmark,
    1 000 seeded landmark pairs from different tracks, one window of 200 consecutive cameras; ba_covariance_blocks and
    ba_marginals_sparse on the same system beside them;
  - Venice-871 shape, alpha = 1: the same scenarios on the dense and on the supernodal path, and their agreement.
The phases come from CUDA events inside the library (SPP_MARGINALS_TIMING): forming + factorisation, host plan,
right-hand side, forward solve (flops from the plan, TFLOP/s), Gram, copy to host, batches and columns. Prints the device
name and power limit with the numbers. Usage: python tools/run_joint_marginals.py [out.jsonl]"""
import json
import os
import re
import sys

os.environ["SPP_MARGINALS_TIMING"] = "1"
import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from run_covariance_blocks import MARG_RE, captured, cov_phases, covisible, edge_indices, gpu_info  # noqa: E402
from slam_plus_plus_b200 import capi, graphs  # noqa: E402

NUM = r"([\d.e+-]+)"
JOINT_RE = re.compile(r"\[spp joint marginals\] (supernodal|dense) path: schur \+ factor " + NUM + r" ms, plan " + NUM +
                      r" ms \(host\), rhs " + NUM + r" ms, forward solve " + NUM + r" ms \(" + NUM + r" flops, " + NUM +
                      r" TFLOP/s\), gram " + NUM + r" ms, copy to host " + NUM + r" ms; (\d+) sets, (\d+) batches, (\d+) columns")
KEYS = ("path", "schur_factor_ms", "plan_ms", "rhs_ms", "forward_ms", "forward_flops", "forward_tflops", "gram_ms", "copy_ms",
        "sets", "batches", "columns")
out_lines = []


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    out_lines.append(line)


def joint_phases(text):
    m = JOINT_RE.search(text)
    if not m:
        return None
    v = m.groups()
    return dict(zip(KEYS, [v[0]] + [float(x) for x in v[1:9]] + [int(x) for x in v[9:]]))


def scenarios(g, rng, window=200):
    """far camera pairs, landmark pairs from different tracks, one window of consecutive cameras (vertex ids)"""
    vt = np.asarray(g.vtype)
    cam_id, pt_id = np.flatnonzero(vt == 0), np.flatnonzero(vt == 1)
    up = covisible(g)
    keys = set((up[:, 0] * g.n_cams + up[:, 1]).tolist())
    far = []
    while len(far) < 1000:
        a, b = sorted(rng.choice(g.n_cams, 2, replace=False).tolist())
        if a * g.n_cams + b not in keys:
            far.append([cam_id[a], cam_id[b]])
    oc, op = edge_indices(g)
    order = np.argsort(op, kind="stable")
    bounds = np.searchsorted(op[order], np.arange(g.n_pts + 1))
    cams = lambda p: set(oc[order[bounds[p]:bounds[p + 1]]].tolist())  # noqa: E731
    pts = []
    while len(pts) < 1000:
        p, q = rng.choice(g.n_pts, 2, replace=False)
        if not cams(p) & cams(q):
            pts.append([pt_id[p], pt_id[q]])
    w0 = int(rng.integers(0, g.n_cams - window))
    return dict(far_camera_pairs=far, far_landmark_pairs=pts, camera_window=[list(cam_id[w0:w0 + window])])


def run_case(ctx, case, alpha, sets_by_name, runs, path):
    for r in range(runs):
        for name, sets in sets_by_name.items():
            out, wall, text = captured(lambda: ctx.ba_joint_marginals(alpha, sets))
            emit(dict(case=case, run=r, path=path, scenario=name, wall_ms=round(wall, 2), phases=joint_phases(text),
                      finite=bool(all(np.all(np.isfinite(o)) for o in out))))
    return {name: ctx.ba_joint_marginals(alpha, sets) for name, sets in sets_by_name.items()}


def main():
    emit(dict(device=gpu_info()))
    ctx = capi.Context(0)

    g = graphs.ba_shape("bal13682")
    ctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    alpha = 50.0
    sets = scenarios(g, np.random.default_rng(13682))
    emit(dict(case="bal13682", C=g.n_cams, P=g.n_pts, O=g.n_obs))
    captured(lambda: ctx.ba_joint_marginals(alpha, sets["far_camera_pairs"][:10]))  # warm-up: first launches, scratch
    run_case(ctx, "bal13682", alpha, sets, 2, "sparse")
    up = covisible(g)
    pairs = up[np.random.default_rng(1).choice(len(up), 20000, replace=False)]
    _, wall, text = captured(lambda: ctx.ba_covariance_blocks(alpha, pairs))
    emit(dict(case="bal13682", call="ba_covariance_blocks", n_pairs=len(pairs), wall_ms=round(wall, 2), phases=cov_phases(text)))
    _, wall, text = captured(lambda: ctx.ba_marginals_sparse(alpha))
    m = MARG_RE.search(text)
    emit(dict(case="bal13682", call="ba_marginals_sparse", wall_ms=round(wall, 2),
              phases=None if not m else dict(zip(("schur_ms", "factor_ms", "selinv_ms", "cameras_ms", "points_ms"), map(float, m.groups())))))

    g = graphs.ba_shape("venice871")
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    sets = scenarios(g, np.random.default_rng(871))
    res = {}
    for path, mode in (("dense", capi.RCS_DENSE), ("sparse", capi.RCS_SPARSE)):
        ctx.schur_set_rcs_solver(mode)
        res[path] = run_case(ctx, "venice871", 1.0, sets, 2, path)
        for call, fn in (("ba_covariance_blocks", lambda: ctx.ba_covariance_blocks(1.0, covisible(g))),
                         ("ba_marginals", lambda: ctx.ba_marginals(1.0) if path == "dense" else ctx.ba_marginals_sparse(1.0))):
            _, wall, text = captured(fn)
            emit(dict(case="venice871", path=path, call=call, wall_ms=round(wall, 2)))
    for name in sets:
        err = max(float(np.linalg.norm(a - b) / np.linalg.norm(a)) for a, b in zip(res["dense"][name], res["sparse"][name]))
        emit(dict(case="venice871", scenario=name, max_rel_err_sparse_vs_dense=err))
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.close()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
