#!/usr/bin/env python
"""Development helper: off-diagonal covariance blocks (spp_ba_covariance_blocks), timed by phase in one process:
  - BAL-13682 shape after ba_linearise, supernodal path, alpha = 50: the call for a seeded sample (20 000 covisible pairs,
    the observations of 2 000 landmarks), for every observation, and ba_marginals_sparse beside them. The phases come
    from CUDA events inside the library (SPP_MARGINALS_TIMING): forming, factorisation, selected inversion, block
    diagonal, the pair kernel, the observation kernel; the host copy is timed on its own;
  - Venice-871 shape, alpha = 1: every covisible pair and every observation on the dense and the supernodal path, time
    and agreement.
Prints the device name and power limit with the numbers. Usage: python tools/run_covariance_blocks.py [out.jsonl]"""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

os.environ["SPP_MARGINALS_TIMING"] = "1"
import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from slam_plus_plus_b200 import capi, graphs  # noqa: E402

NUM = r"([\d.]+)"
COV_RE = re.compile(r"\[spp covariance blocks\] (supernodal|dense) path " + NUM + r" ms.*?pairs " + NUM + r" ms \((\d+)\), observations " +
                    NUM + r" ms \((\d+)\); pattern check " + NUM + r" ms, copy to host " + NUM + r" ms \(" + NUM + r" GB\)")
SPARSE_RE = re.compile(r"schur " + NUM + r" ms, factor " + NUM + r" ms, selected inversion " + NUM + r" ms, cameras " + NUM +
                       r" ms, points " + NUM + r" ms;")
MARG_RE = re.compile(r"\[spp marginals sparse\] schur " + NUM + r" ms, factor " + NUM + r" ms, selected inversion " + NUM +
                     r" ms .*?cameras " + NUM + r" ms, points " + NUM + r" ms")
out_lines = []


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    out_lines.append(line)


def captured(fn):
    """fn() with stderr captured: (result, wall ms, stderr text)"""
    sys.stderr.flush()
    with tempfile.TemporaryFile(mode="w+b") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            t = time.perf_counter()
            r = fn()
            wall = (time.perf_counter() - t) * 1e3
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode(errors="replace")
    return r, wall, text


def cov_phases(text):
    m = COV_RE.search(text)
    if not m:
        return None
    v = m.groups()
    ph = dict(path=v[0], path_ms=float(v[1]), pairs_ms=float(v[2]), n_pairs=int(v[3]), observations_ms=float(v[4]), n_obs=int(v[5]),
              pattern_check_ms=float(v[6]), copy_ms=float(v[7]), copy_gb=float(v[8]))
    s = SPARSE_RE.search(text)
    if s:
        ph.update(zip(("schur_ms", "factor_ms", "selinv_ms", "cameras_ms", "points_ms"), map(float, s.groups())))
    return ph


def rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return q


def edge_indices(g):
    loc = np.asarray(g.vertex_local_index(), np.int64)
    return loc[np.asarray(g.obs_cam, np.int64)], loc[np.asarray(g.obs_pt, np.int64)]


def covisible(g):
    oc, op = edge_indices(g)
    r, c = capi.rcs_block_pattern(g.n_cams, g.n_pts, oc, op)
    return np.stack([r[r != c], c[r != c]], 1).astype(np.int64)


def main():
    emit(dict(device=gpu_info()))
    ctx = capi.Context(0)

    g = graphs.ba_shape("bal13682")
    ctx.schur_set_rcs_solver(capi.RCS_SPARSE)
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    alpha = 50.0
    rng = np.random.default_rng(13682)
    up = covisible(g)
    pairs = up[rng.choice(len(up), 20000, replace=False)]
    _, op = edge_indices(g)
    obs_sample = np.flatnonzero(np.isin(op, rng.choice(g.n_pts, 2000, replace=False)))
    obs_all = np.arange(g.n_obs)
    emit(dict(case="bal13682", C=g.n_cams, P=g.n_pts, O=g.n_obs, covisible_pairs=len(up), sample_pairs=len(pairs),
              sample_obs=len(obs_sample)))
    captured(lambda: ctx.ba_covariance_blocks(alpha, pairs, obs_sample))  # warm-up: first launches, scratch
    for r in range(3):
        _, wall, text = captured(lambda: ctx.ba_marginals_sparse(alpha))
        m = MARG_RE.search(text)
        emit(dict(case="bal13682", run=r, call="ba_marginals_sparse", wall_ms=round(wall, 2),
                  phases=None if not m else dict(zip(("schur_ms", "factor_ms", "selinv_ms", "cameras_ms", "points_ms"), map(float, m.groups())))))
        _, wall, text = captured(lambda: ctx.ba_covariance_blocks(alpha, pairs, obs_sample))
        emit(dict(case="bal13682", run=r, call="sample", wall_ms=round(wall, 2), phases=cov_phases(text)))
        out, wall, text = captured(lambda: ctx.ba_covariance_blocks(alpha, None, obs_all))
        emit(dict(case="bal13682", run=r, call="all_observations", wall_ms=round(wall, 2), phases=cov_phases(text),
                  finite=bool(np.all(np.isfinite(out["observations"])))))
        del out
    a = ctx.ba_covariance_blocks(alpha, pairs, obs_sample, diagonal=True)
    b = ctx.ba_covariance_blocks(alpha, pairs, obs_sample, diagonal=True)
    emit(dict(case="bal13682", bitwise_reproducible=all(np.array_equal(a[k], b[k]) for k in a)))
    del a, b

    g = graphs.ba_shape("venice871")
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    up = covisible(g)
    pairs = np.concatenate([up, np.stack([np.arange(g.n_cams)] * 2, 1)])
    obs_all = np.arange(g.n_obs)
    res = {}
    for r in range(3):
        for path, mode in (("dense", capi.RCS_DENSE), ("sparse", capi.RCS_SPARSE)):
            ctx.schur_set_rcs_solver(mode)
            res[path], wall, text = captured(lambda: ctx.ba_covariance_blocks(1.0, pairs, obs_all, diagonal=True))
            emit(dict(case="venice871", run=r, path=path, C=g.n_cams, P=g.n_pts, O=g.n_obs, n_pairs=len(pairs), wall_ms=round(wall, 2),
                      phases=cov_phases(text)))
        emit(dict(case="venice871", run=r, **{f"rel_err_{k}": rel(res["sparse"][k], res["dense"][k]) for k in res["dense"]}))
    ctx.schur_set_rcs_solver(capi.RCS_AUTO)
    ctx.close()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
