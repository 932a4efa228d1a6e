#!/usr/bin/env python
"""Development helper: marginal covariances through the block-sparse reduced camera system (spp_ba_marginals_sparse:
supernodal factorisation + selected inversion), in one process:
  - BAL-13682 shape after ba_linearise: the call timed by phase (Schur forming, factorisation, selected inversion,
    cameras, points; CUDA events inside the library, SPP_MARGINALS_TIMING), the selected inversion's flops from the
    symbolic analysis and its rate against an in-run cuBLAS DGEMM 4096^3 (as bench.py measures the FP64 peak);
  - Venice-871 shape: sparse against dense marginals, time and agreement;
  - the 1/16 sub-sequence of the BAL-13682 shape (855 cameras): the same.
Prints the device name and power limit with the numbers. Usage: python tools/run_marginals_sparse.py [out.jsonl]"""
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

PHASE_RE = re.compile(r"schur ([\d.]+) ms, factor ([\d.]+) ms, selected inversion ([\d.]+) ms \(([\d.e+]+) flops, ([\d.]+) TFLOP/s\), "
                      r"cameras ([\d.]+) ms, points ([\d.]+) ms; scratch ([\d.]+) GB \(main\) \+ (\d+) x ([\d.]+) GB \(lanes\), panels ([\d.]+) GB")
out_lines = []


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    out_lines.append(line)


def timed_sparse(ctx, alpha):
    """one ba_marginals_sparse call: wall time and the library's phase line (stderr captured around the call)"""
    sys.stderr.flush()
    with tempfile.TemporaryFile(mode="w+b") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            t = time.perf_counter()
            cc, pc = ctx.ba_marginals_sparse(alpha)
            wall = time.perf_counter() - t
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode(errors="replace")
    m = PHASE_RE.search(text)
    ph = None
    if m:
        v = [float(x) for x in m.groups()]
        ph = dict(schur_ms=v[0], factor_ms=v[1], selinv_ms=v[2], selinv_flops=v[3], selinv_tflops=v[4], cameras_ms=v[5],
                  points_ms=v[6], scratch_main_gb=v[7], lanes=int(v[8]), scratch_lane_gb=v[9], panels_gb=v[10])
    return cc, pc, wall * 1e3, ph


def rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return q


def fp64_dgemm_tflops():
    import torch
    dev = torch.device("cuda:0")
    n = 4096
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize(dev)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    torch.cuda.empty_cache()
    return best


def main():
    emit(dict(device=gpu_info(), fp64_dgemm_tflops=round(fp64_dgemm_tflops(), 2)))
    ctx = capi.Context(0)

    # BAL-13682: one warm-up call (first launches, scratch allocation), then timed calls
    g = graphs.ba_shape("bal13682")
    ctx.ba_set_graph(g)
    ctx.ba_linearise()
    for r in range(3):
        cc, pc, wall, ph = timed_sparse(ctx, 50.0)
        info = ctx.schur_get_rcs_info()
        emit(dict(case="bal13682", run=r, C=g.n_cams, P=g.n_pts, alpha=50.0, wall_ms=round(wall, 2), phases=ph,
                  supernodes=info["supernodes"], updates=info["updates"], factor_flops=info["factor_flops"],
                  finite=bool(np.all(np.isfinite(cc)) and np.all(np.isfinite(pc))),
                  cam_var_max=float(np.einsum("kii->ki", cc).max()), pt_var_max=float(np.einsum("kii->ki", pc).max())))
    cc2, pc2, _, _ = timed_sparse(ctx, 50.0)
    emit(dict(case="bal13682", bitwise_reproducible=bool(np.array_equal(cc, cc2) and np.array_equal(pc, pc2))))
    del cc, pc, cc2, pc2

    for name, g in (("venice871", graphs.ba_shape("venice871")),
                    ("bal13682_sixteenth", graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120,
                                                          max_stride=12, loops=1))):
        ctx.ba_set_graph(g)
        ctx.ba_linearise()
        alpha = 1.0
        for r in range(3):
            cs, ps, wall_s, ph = timed_sparse(ctx, alpha)
            t = time.perf_counter()
            cd, pd = ctx.ba_marginals(alpha)
            wall_d = (time.perf_counter() - t) * 1e3
            info = ctx.schur_get_rcs_info()
            emit(dict(case=name, run=r, C=g.n_cams, P=g.n_pts, alpha=alpha, sparse_wall_ms=round(wall_s, 2), dense_wall_ms=round(wall_d, 2),
                      phases=ph, supernodes=info["supernodes"], updates=info["updates"], rel_err_cameras=rel(cs, cd),
                      rel_err_points=rel(ps, pd)))
    ctx.close()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
