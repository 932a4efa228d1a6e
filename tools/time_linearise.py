#!/usr/bin/env python3
"""Times the observation-bound kernels of an LM iteration -- the linearisation (k_cam_prepare, k_linearise_cams,
k_sum_point_records) and the landmark inverse of the Schur stage (k_landmark_inverse) -- at the bench shapes, and
reports each kernel's achieved bandwidth against the bytes the algorithm has to move (computed from O, P and C).

Per-kernel device times come from torch.profiler (CUDA activities) over --reps calls of ba_linearise() and
ba_solve_step(); the whole ba_linearise() call is also timed with CUDA events on the library's stream. Every working
set here is larger than the 126 MB L2, so repeated calls do not run from cache. The card's name and power limit are
read in the same run and printed with the numbers. Output: one JSON line per shape (and with --out, the same lines
appended to that file)."""
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


def time_shape(shape, reps, alpha):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from slam_plus_plus_b200 import capi, graphs

    g = graphs.ba_shape(shape)
    C, P, O = int(g.cams.shape[0]), int(g.pts.shape[0]), int(g.obs_pt.shape[0])
    ctx = capi.Context(0)
    ctx.ba_set_graph(g)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    for _ in range(3):  # first launches load the modules; the Schur / factor buffers are sized here
        ctx.ba_linearise()
        ctx.ba_solve_step(alpha)
    ctx.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        ctx.ba_linearise()
    e1.record(stream)
    ctx.synchronize()
    e1.synchronize()
    lin_ms = e0.elapsed_time(e1) / reps

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.ba_linearise()
            ctx.ba_solve_step(alpha)
        ctx.synchronize()
        torch.cuda.synchronize()
    ctx.close()

    kt = kernel_times(prof, list(KERNEL_BYTES))
    kernels = {}
    for name, (us, n) in kt.items():
        if us is None:
            raise RuntimeError(f"{name} was not seen in the profile of {shape}")
        b = KERNEL_BYTES[name](O, P, C)
        kernels[name] = {"us": round(us, 2), "launches": n, "algorithmic_mb": round(b / 1e6, 1),
                         "achieved_gbs": round(b / (us * 1e-6) / 1e9, 1),
                         "frac_of_hbm": round(b / (us * 1e-6) / 1e9 / HBM_PEAK_GBS, 3)}
    lb = LINEARISE_BYTES(O, P, C)
    return {"shape": shape, "C": C, "P": P, "O": O, "reps": reps, "alpha": alpha,
            "linearise_call": {"ms": round(lin_ms, 4), "algorithmic_mb": round(lb / 1e6, 1),
                               "achieved_gbs": round(lb / (lin_ms * 1e-3) / 1e9, 1)},
            "kernels": kernels}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shapes", default="venice871,bal13682")
    ap.add_argument("--reps", type=int, default=50, help="timed calls per shape")
    ap.add_argument("--alpha", type=float, default=1.0, help="damping of the Schur stage's landmark inverse")
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these numbers can only be measured on the GPU")
    dev = card()
    print(json.dumps({"card": dev}), flush=True)
    lines = [json.dumps({"card": dev})]
    for shape in args.shapes.split(","):
        r = time_shape(shape, args.reps if shape != "bal13682" else max(args.reps // 5, 3), args.alpha)
        r["card"] = dev
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
