#!/usr/bin/env python3
"""Robust losses on a contaminated bundle adjustment problem: the Venice-871 shape with a fraction (default 5 %) of its
measurements replaced by uniform pixels (graphs.add_outliers), optimised with SPP_LOSS_NONE, HUBER and CAUCHY.

For each loss it reports the reprojection RMS over the inliers after Optimize (and, for reference, that of the clean
graph with the outliers removed) and the LM iteration time split into the report's phases. The three losses run on one
resident graph (the loss is context state; ba_restore_initial puts the states back), alternating over --rounds rounds
after one warm-up run each; the median round is reported. The card's name and power limit are read in the same run.
Output: JSON lines on stdout, and with --out appended to that file (profiles/r6_robust.jsonl)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from time_linearise import card  # noqa: E402

PHASES = ("linearise", "schur", "factor", "backsubst", "update", "chi2", "total")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shape", default="venice871")
    ap.add_argument("--outliers", type=float, default=0.05)
    ap.add_argument("--scale", type=float, default=2.0, help="scale k of HUBER and CAUCHY (pixels)")
    ap.add_argument("--iterations", type=int, default=20, help="LM iterations per Optimize")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1, help="seed of the outliers")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these numbers can only be measured on the GPU")
    from slam_plus_plus_b200 import capi, graphs
    from slam_plus_plus_b200.sppio import BAGraph

    dev = card()
    lines = [json.dumps({"card": dev})]
    print(lines[-1], flush=True)
    clean = graphs.ba_shape(args.shape)
    g, idx = graphs.add_outliers(clean, args.outliers, args.seed)
    inl = np.ones(len(g.obs_pt), bool)
    inl[idx] = False
    losses = {"none": capi.LOSS_NONE, "huber": capi.LOSS_HUBER, "cauchy": capi.LOSS_CAUCHY}

    ctx = capi.Context(0)

    def inlier_rms(mask):
        ctx.ba_set_robust_loss(capi.LOSS_NONE)
        s2, _ = ctx.ba_observation_errors()  # identity information: squared pixel errors
        return float(np.sqrt(s2[mask].mean()))

    ctx.ba_set_graph(g)
    runs = {name: [] for name in losses}
    result = {}
    for r in range(args.rounds + 1):  # round 0 warms every loss up
        for name, kind in losses.items():
            ctx.ba_set_robust_loss(kind, args.scale)
            ctx.ba_restore_initial()
            rep = ctx.ba_optimize(args.iterations, 0.0)
            if r == 0:
                continue
            n = max(rep["n_iterations"], 1)
            runs[name].append({p: rep["ms"][p] / n for p in PHASES})
            if r == 1:
                result[name] = {"n_iterations": rep["n_iterations"], "n_accepted": rep["n_accepted"],
                                "cost_initial": rep["chi2_initial"], "cost_final": rep["chi2_final"],
                                "inlier_rms_px": inlier_rms(inl)}
    for name in losses:
        per_it = sorted(runs[name], key=lambda x: x["total"])[len(runs[name]) // 2]
        result[name]["ms_per_iteration"] = {p: round(v, 4) for p, v in per_it.items()}
        result[name]["ms_per_iteration_total_rounds"] = [round(x["total"], 4) for x in runs[name]]

    ctx.ba_set_robust_loss(capi.LOSS_NONE)
    ctx.ba_set_graph(BAGraph(clean.vtype, clean.cams, clean.pts, clean.obs_pt[inl], clean.obs_cam[inl], clean.z[inl],
                             clean.info[inl]))
    rep = ctx.ba_optimize(args.iterations, 0.0)
    clean_rms = inlier_rms(np.ones(int(inl.sum()), bool))
    ctx.close()

    base = result["none"]["ms_per_iteration"]["total"]
    for name in losses:
        r = dict(shape=args.shape, outliers=args.outliers, n_outliers=int(len(idx)), loss=name,
                 scale=args.scale if name != "none" else None, iterations=args.iterations, **result[name])
        r["inlier_rms_vs_clean"] = round(r["inlier_rms_px"] / clean_rms, 4)
        r["iteration_vs_none"] = round(r["ms_per_iteration"]["total"] / base, 4)
        r["card"] = dev
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    lines.append(json.dumps({"shape": args.shape, "loss": "none", "graph": "clean (outliers removed)",
                             "n_iterations": rep["n_iterations"], "inlier_rms_px": clean_rms, "card": dev}))
    print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
