#!/usr/bin/env python3
"""Times the observation-bound kernels of an LM iteration -- the linearisation (k_cam_prepare, k_linearise_cams,
k_sum_point_records) and the landmark inverse of the Schur stage (k_landmark_inverse) -- at the bench shapes, and
reports each kernel's achieved bandwidth against the bytes the algorithm has to move (computed from O, P and C).

Per-kernel device times come from torch.profiler (CUDA activities) over --reps calls of ba_linearise() and
ba_solve_step(); the whole ba_linearise() call is also timed with CUDA events on the library's stream. Every working
set here is larger than the 126 MB L2, so repeated calls do not run from cache. The card's name and power limit are
read in the same run and printed with the numbers. Output: one JSON line per shape (and with --out, the same lines
appended to that file).

--loss none,huber,cauchy times the robust-loss variants of the linearisation on the same resident graph in the same
run: the event-timed ba_linearise() calls alternate between the losses in --rounds rounds, then each loss is profiled on
its own. One JSON line per (shape, loss); --outliers replaces that fraction of the measurements by uniform pixels
(graphs.add_outliers), so that the robust branches see gross errors."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK_GBS = 6454.0  # measured HBM bandwidth of the B200 (DESIGN.md §4)

# algorithmic bytes (read + write) of each kernel, DESIGN.md §4
KERNEL_BYTES = {
    "k_cam_prepare": lambda O, P, C: 88 * C + 7 * 96 * C + 40 * C,
    "k_linearise_cams": lambda O, P, C: 84 * O + 224 * O + 336 * C,
    "k_sum_point_records": lambda O, P, C: 80 * O + 96 * P,
    "k_landmark_inverse": lambda O, P, C: 2 * (72 * P + 144 * O),
}
LINEARISE_BYTES = lambda O, P, C: 200 * O + 120 * P + 424 * C  # noqa: E731  (bench.py's roofline.hbm_stage)


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"] = float(q[0])
        out["sm_max_mhz"] = float(q[1])
    except Exception as e:  # the numbers are still printed; the line says the power limit could not be read
        out["power_limit_w"] = None
        out["power_limit_error"] = str(e)
    return out


def kernel_times(prof, names):
    """Mean device time (us) and launch count of each kernel whose name contains one of `names`."""
    acc = {n: [0.0, 0] for n in names}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        for n in names:
            if n in ev.key and t:
                acc[n][0] += t
                acc[n][1] += ev.count
    return {n: (v[0] / v[1] if v[1] else None, v[1]) for n, v in acc.items()}


LOSSES = {"none": 0, "huber": 1, "cauchy": 2}  # capi.LOSS_*


def time_shape(shape, reps, alpha, losses=("none",), scale=2.0, outliers=0.0, rounds=5):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from slam_plus_plus_b200 import capi, graphs

    g = graphs.ba_shape(shape)
    if outliers > 0:
        g, _ = graphs.add_outliers(g, outliers, 1)
    C, P, O = int(g.cams.shape[0]), int(g.pts.shape[0]), int(g.obs_pt.shape[0])
    ctx = capi.Context(0)
    ctx.ba_set_graph(g)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    for loss in losses:
        ctx.ba_set_robust_loss(LOSSES[loss], scale)
        for _ in range(3):  # first launches load the modules; the Schur / factor buffers are sized here
            ctx.ba_linearise()
            ctx.ba_solve_step(alpha)
    ctx.synchronize()

    # event-timed calls, the losses alternating round by round
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_round = max(reps // rounds, 1)
    lin_ms = {loss: [] for loss in losses}
    for _ in range(rounds):
        for loss in losses:
            ctx.ba_set_robust_loss(LOSSES[loss], scale)
            e0.record(stream)
            for _ in range(per_round):
                ctx.ba_linearise()
            e1.record(stream)
            ctx.synchronize()
            e1.synchronize()
            lin_ms[loss].append(e0.elapsed_time(e1) / per_round)

    out = []
    for loss in losses:
        ctx.ba_set_robust_loss(LOSSES[loss], scale)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                ctx.ba_linearise()
                ctx.ba_solve_step(alpha)
            ctx.synchronize()
            torch.cuda.synchronize()
        kt = kernel_times(prof, list(KERNEL_BYTES))
        kernels = {}
        for name, (us, n) in kt.items():
            if us is None:
                raise RuntimeError(f"{name} was not seen in the profile of {shape}")
            b = KERNEL_BYTES[name](O, P, C)
            kernels[name] = {"us": round(us, 2), "launches": n, "algorithmic_mb": round(b / 1e6, 1),
                             "achieved_gbs": round(b / (us * 1e-6) / 1e9, 1),
                             "frac_of_hbm": round(b / (us * 1e-6) / 1e9 / HBM_PEAK_GBS, 3)}
        ms = sorted(lin_ms[loss])[len(lin_ms[loss]) // 2]
        lb = LINEARISE_BYTES(O, P, C)
        r = {"shape": shape, "C": C, "P": P, "O": O, "reps": reps, "alpha": alpha,
             "linearise_call": {"ms": round(ms, 4), "ms_rounds": [round(x, 4) for x in lin_ms[loss]],
                                "algorithmic_mb": round(lb / 1e6, 1), "achieved_gbs": round(lb / (ms * 1e-3) / 1e9, 1)},
             "kernels": kernels}
        if losses != ("none",):
            r.update(loss=loss, loss_scale=scale if loss != "none" else None, outliers=outliers)
        out.append(r)
    ctx.close()
    if "none" in losses:  # cost of each loss against the plain kernel of the same run
        base = next(r for r in out if r.get("loss", "none") == "none")
        for r in out:
            r["vs_none"] = {"k_linearise_cams": round(r["kernels"]["k_linearise_cams"]["us"] / base["kernels"]["k_linearise_cams"]["us"], 4),
                            "linearise_call": round(r["linearise_call"]["ms"] / base["linearise_call"]["ms"], 4)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shapes", default="venice871,bal13682")
    ap.add_argument("--reps", type=int, default=50, help="timed calls per shape")
    ap.add_argument("--alpha", type=float, default=1.0, help="damping of the Schur stage's landmark inverse")
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    ap.add_argument("--loss", default="none", help="comma-separated robust losses to time in the same run: none,huber,cauchy")
    ap.add_argument("--loss-scale", type=float, default=2.0, help="scale k of the robust losses (pixels)")
    ap.add_argument("--outliers", type=float, default=0.0, help="fraction of measurements replaced by uniform pixels")
    ap.add_argument("--rounds", type=int, default=5, help="rounds of alternating event-timed calls")
    args = ap.parse_args()
    losses = tuple(args.loss.split(","))
    for loss in losses:
        if loss not in LOSSES:
            raise SystemExit(f"unknown loss {loss!r}: choose from {','.join(LOSSES)}")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these numbers can only be measured on the GPU")
    dev = card()
    print(json.dumps({"card": dev}), flush=True)
    lines = [json.dumps({"card": dev})]
    for shape in args.shapes.split(","):
        for r in time_shape(shape, args.reps if shape != "bal13682" else max(args.reps // 5, 3), args.alpha, losses,
                            args.loss_scale, args.outliers, args.rounds):
            r["card"] = dev
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
