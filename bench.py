#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 NLS hot path (BASELINE.json: BA LM iterations/s, Venice-871 shape).

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the reference's own CPU solver (oracle/_ref)

One "step" = one CNonlinearSolver_Lambda_LM::Optimize(max_iter = 5, min_dx = 0) on the synthetic Venice-871-shape
graph (871 cameras, 530 304 points, 2 837 687 observations; slam_plus_plus_b200/graphs.py, seed 871):
linearise -> landmark Schur complement -> dense FP64 Cholesky of the 5226 x 5226 reduced camera system ->
back-substitution -> update -> chi2, five times, with the reference's LM control flow. `value` counts linear
solves (LM iterations) per second with the graph resident in HBM (vertex states are restored from a device
snapshot at the start of every step); `e2e` times the full public call sequence with HOST buffers:
spp_ba_set_graph (H2D + symbolic analysis) + spp_ba_optimize + spp_ba_get_states (D2H).

Rank 0 prints ONE JSON line. Timing: CUDA events on the context's stream, barrier + synchronize on both sides,
max over ranks. The working set (W, Y: 2 x 409 MB; S: 220 MB) is far larger than the 126 MB L2, so consecutive
steps do not find their inputs in cache ("inputs larger than L2").

--dump-outputs DIR writes what the last timed step handed its caller as DIR/<name>.npy (float64): the optimised
camera states and landmark positions (spp_ba_get_states; `poses` on the pose-graph shapes) and the LM trace of the
report, with the prefix `bal13682_` for the second block of the headline line. The graphs are seeded, so two builds
run with the same arguments can be compared array for array. Landmark arrays above DUMP_MAX_ROWS rows are replaced by
a fixed, seeded sample of rows (`<name>_rows.npy` holds their indices), which keeps a dump under 64 MB.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "ba_lm_iterations_per_s"
UNIT = "LM iterations/s"
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "ref_driver_ba")
DUMP_MAX_ROWS = 1 << 20  # Venice-871 (530 304 landmarks) is dumped whole, BAL-13682 (4.46 M) as a sample


def dump_outputs(out_dir, prefix, rep, arrays):
    """Writes the report's LM trace and the given (name -> 2-D float64 array) outputs as out_dir/<prefix><name>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"chi2_trace": rep["trace_chi2"], "alpha_trace": rep["trace_alpha"], "dx_norm_trace": rep["trace_dx_norm"],
           "accepted_trace": rep["trace_accepted"], "chi2": [rep["chi2_initial"], rep["chi2_final"]]}
    for name, a in arrays.items():
        if a.shape[0] > DUMP_MAX_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_MAX_ROWS, replace=False))
            out[name + "_rows"], a = rows, a[rows]
        out[name] = a
    for name, a in out.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, np.float64))


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE JSON line: anything a native library prints to file descriptor 1 (NCCL's version banner
    from ncclCommInitRank, for one) is sent to stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi samples"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples)}


def measure_fp64_peak(torch, dev):
    """FP64 matrix-pipe peak of this GPU: cuBLAS DGEMM 4096^3 through torch.matmul, best of 5 (TFLOP/s).
    MEASURED_PEAKS.json carries no FP64 entry (SURVEY 7 'hard parts'), so the denominator is measured in-run."""
    n = 4096
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize(dev)
    best = 0.0
    for _ in range(5):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    return best


def write_graph_file(g):
    from slam_plus_plus_b200 import sppio
    path = os.path.join(tempfile.gettempdir(), f"spp_bench_{os.getpid()}.bin")
    sppio.write_graph(path, g)
    return path


def run_reference_steps(graph_path, warmup, steps, threads=None):
    """Runs the reference's own LM solver (oracle/_ref, compiled from the unmodified reference sources) and returns
    the per-step seconds of Optimize(1, 0) calls on the resident system."""
    from slam_plus_plus_b200 import sppio
    if not os.path.exists(REF_BIN):
        raise RuntimeError("oracle/_ref/ref_driver_ba is missing (built by __graft_entry__.build() where the reference's "
                           "sources are present, see oracle/build_ref.sh)")
    out = os.path.join(tempfile.gettempdir(), f"spp_bench_ref_{os.getpid()}.dump")
    env = dict(os.environ)
    if threads:
        env["OMP_NUM_THREADS"] = str(threads)
    subprocess.run([REF_BIN, "steps", graph_path, out, str(warmup), str(steps)], check=True, env=env,
                   stdout=subprocess.DEVNULL)
    d = sppio.read_dump(out)
    os.unlink(out)
    return d["step_seconds"], int(d["omp_threads"][0]), d


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from slam_plus_plus_b200 import graphs
    g = graphs.ba_shape(args.shape)
    path = write_graph_file(g)
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: the reference gets all the host cores whatever N is
    n_threads = (os.cpu_count() or 1) if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None
    try:
        secs, threads, d = run_reference_steps(path, args.warmup, args.steps, threads=n_threads)
    finally:
        os.unlink(path)
    timed = secs[args.warmup:]
    total = float(np.sum(timed))
    value = len(timed) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / max(len(timed), 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.shape}-shape BA, reference CNonlinearSolver_Lambda_LM + CLinearSolver_Schur (dense LLT), "
                               "one LM iteration (Optimize(1, 0)) per step on the resident system",
                   "cameras": g.n_cams, "points": g.n_pts, "observations": g.n_obs},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                         "sample": "each step = Optimize(max_iter=1) of the unmodified reference on the full graph "
                                   "(structure build excluded: it happens in the first warm-up step)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def check_chi2(args, rep):
    """chi2 after the last LM iteration of the last timed step against profiles/chi2_trace.json (written by a single-GPU
    run with --write-chi2-trace). FD Jacobians amplify the rounding differences of another summation order (NCCL, the
    rank count) to ~1e-8 after five iterations; the bound asserted is 1e-6 (north_star)."""
    path = os.path.join(ROOT, "profiles", "chi2_trace.json")
    key = f"{args.shape}/lm{args.lm_iters}"
    if args.jacobians != "fd":
        return {"checked": False, "why": "the committed trace is that of the forward-difference (parity) mode"}
    if args.write_chi2_trace:  # a path: gpurun only brings gpurun_out/ back, the file is then committed as profiles/chi2_trace.json
        out = args.write_chi2_trace
        d = json.load(open(out)) if os.path.exists(out) else (json.load(open(path)) if os.path.exists(path) else {})
        d[key] = {"chi2_final": rep["chi2_final"], "trace_chi2": rep["trace_chi2"], "trace_accepted": [int(x) for x in rep["trace_accepted"]]}
        if int(os.environ.get("RANK", "0")) == 0:
            json.dump(d, open(out, "w"), indent=1)
        return {"checked": False, "why": "this run wrote the trace"}
    if not os.path.exists(path):
        return {"checked": False, "why": "no committed trace"}
    d = json.load(open(path)).get(key)
    if d is None:
        return {"checked": False, "why": "no committed trace for " + key}
    rel = abs(rep["chi2_final"] - d["chi2_final"]) / d["chi2_final"]
    ok = rel <= 1e-6 and [int(x) for x in rep["trace_accepted"]] == [int(x) for x in d["trace_accepted"]]
    if not ok:
        raise SystemExit(f"chi2 check failed: {rep['chi2_final']!r} vs committed {d['chi2_final']!r} (rel {rel:.3e}), accepted "
                         f"{rep['trace_accepted']} vs {d['trace_accepted']}")
    return {"checked": True, "chi2_final": rep["chi2_final"], "committed": d["chi2_final"], "rel_diff": rel, "bound": 1e-6}


def gpu_arm(args):
    """The headline line (Venice-871 shape, LM iterations/s) and, inside the same line, the second metric BASELINE.json
    names: Schur-solve ms per LM iteration on the BAL-13682 shape ("bal13682" block; --no-bal skips it)."""
    import copy
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    line = measure_ba(args, torch, dist, dev, rank, world, local)
    if args.shape == "venice871" and not args.no_bal:
        a2 = copy.copy(args)
        a2.shape = "bal13682"
        try:
            bal = measure_ba(a2, torch, dist, dev, rank, world, local, dump_prefix="bal13682_")
        except Exception as ex:  # the headline line must still be printed
            bal = {"failed": repr(ex)}
        if rank == 0:
            for k in ("n_gpus", "warmup", "scaling", "vs_baseline", "dtype", "data", "clocks"):
                bal.pop(k, None)
            line["bal13682"] = bal
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_ba(args, torch, dist, dev, rank, world, local, dump_prefix=""):
    """One BA shape on the rank's GPU; returns the bench line (rank 0) or None."""
    from slam_plus_plus_b200 import capi, graphs

    g = graphs.ba_shape(args.shape)
    ctx = capi.Context(local)
    if world > 1:
        from slam_plus_plus_b200.parallel import attach_nccl
        attach_nccl(ctx, rank, world)  # ncclAllReduce inside libspp_b200.so; torch.distributed only carries the unique id
    if args.jacobians == "analytic":  # the production variant; the default (forward differences) is the reference's parity mode
        ctx.ba_set_jacobian_mode(capi.JAC_ANALYTIC)
    t0 = time.time()
    ctx.ba_set_graph(g)
    setup_s = time.time() - t0
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def one_step():
        ctx.ba_restore_initial()
        return ctx.ba_optimize(args.lm_iters, 0.0)

    for _ in range(max(args.warmup, 3)):
        rep = one_step()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    launches0 = ctx.kernel_launches
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    n_iters = 0
    phase = {}
    for _ in range(args.steps):
        rep = one_step()
        n_iters += rep["n_iterations"]
        for k, v in rep["ms"].items():
            phase[k] = phase.get(k, 0.0) + v
    e1.record(stream)
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches - launches0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n_iters / (ms * 1e-3)
    if world > 1:  # phase times: max over ranks as well
        keys = sorted(phase)
        t = torch.tensor([phase[k] for k in keys], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        phase = {k: float(v) for k, v in zip(keys, t.tolist())}
    if args.dump_outputs:  # the states the last timed step left on the device, read back outside the timed window
        cams, pts = ctx.ba_gather_states() if world > 1 else ctx.ba_get_states()
        if rank == 0:
            dump_outputs(args.dump_outputs, dump_prefix, rep, {"cams": cams, "points": pts})
    sparse_rcs = 6 * g.n_cams > 16384  # SPP_RCS_AUTO: block-sparse (supernodal) reduced camera system above 16 384 unknowns
    rcs_info = ctx.schur_get_rcs_info() if sparse_rcs else None

    # ---- end to end through the public API with host buffers (pinned), every step: H2D graph, optimise, D2H states
    vtype = np.ascontiguousarray(g.vtype, np.uint8)
    host = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in
            (g.cams, g.pts, g.obs_pt.astype(np.uint64).view(np.int64), g.obs_cam.astype(np.uint64).view(np.int64), g.z, g.info)]
    h2d = int(vtype.nbytes + sum(t.numel() * t.element_size() for t in host))
    d2h = int(g.n_cams * 6 * 8 + g.n_pts * 3 * 8)
    from slam_plus_plus_b200.sppio import BAGraph
    gh = BAGraph(vtype, host[0].numpy(), host[1].numpy(), host[2].numpy().view(np.uint64), host[3].numpy().view(np.uint64),
                 host[4].numpy(), host[5].numpy())
    e2e_steps = max(1, min(args.steps, 5 if not sparse_rcs else 2))
    out_c, out_p = torch.empty((g.n_cams, 6), dtype=torch.float64).pin_memory(), torch.zeros((g.n_pts, 3), dtype=torch.float64).pin_memory()
    barrier()
    t0 = time.perf_counter()
    e2e_iters = 0
    for _ in range(e2e_steps):
        ctx.ba_set_graph(gh)
        r = ctx.ba_optimize(args.lm_iters, 0.0)
        ctx.ba_get_states(out_c.numpy(), out_p.numpy())  # the result lands in the caller's page-locked buffers
        e2e_iters += r["n_iterations"]
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = e2e_iters / e2e_s

    # numerical evidence at every N: the final chi2 of the last timed step against the committed single-GPU trace
    chi2_check = check_chi2(args, rep)

    barrier()
    ctx.close()  # every rank leaves the same way: the library's communicator (and the device memory of this shape) first
    if world > 1:
        dist.barrier()
    if rank != 0:
        return None
    # ---- roofline of the dominant kernel: the Cholesky factorisation of the reduced camera system.
    # dense (Venice): ONE kernel, k_chol_dataflow -- achieved = n^3 / 3 flops / its own launch duration (CUDA events around the
    # launch on the context's stream, recorded inside the LM loop of the timed region: report field ms_factor_kernel);
    # block-sparse (BAL): the kernel group of the supernodal factorisation, flops of the numeric phase as executed.
    n = 6 * g.n_cams
    chol_flops = rcs_info["factor_flops"] if sparse_rcs else n ** 3 / 3.0
    phase_ms = phase["factor"] / max(n_iters, 1)
    chol_ms = phase_ms if sparse_rcs else phase["factor_kernel"] / max(n_iters, 1)
    fp64_peak = measure_fp64_peak(torch, dev)
    achieved = chol_flops / (chol_ms * 1e-3) / 1e12
    hbm_peak, hbm_src = load_peaks()
    O, P, Cn = g.n_obs, g.n_pts, g.n_cams
    bytes_lin = 200 * O + 120 * P + 424 * Cn
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "chol_traffic.json")  # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
    if os.path.exists(tpath) and not sparse_rcs:
        td = json.load(open(tpath)).get(args.shape)
        if td:
            traffic, traffic_src = td["dram_bytes_per_launch"], td["source"]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.shape}-shape BA, LM Optimize({args.lm_iters}, 0) per step, Schur + dense FP64 Cholesky",
                   "cameras": Cn, "points": P, "observations": O, "lm_iterations_per_step": n_iters / args.steps,
                   "jacobians": "forward differences, delta=1e-9 (reference parity mode)" if args.jacobians == "fd" else
                                "analytic (closed-form derivatives; agrees with the forward differences at their noise floor)",
                   "l2_policy": "inputs larger than L2 (W+Y 817 MB, S 220 MB vs 126 MB L2)",
                   "parallelism": f"landmark-sharded x{world}" if world > 1 else "single GPU",
                   "symbolic_setup_s": setup_s},
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "note": "spp_ba_set_graph(host, incl. symbolic analysis) + spp_ba_optimize + spp_ba_get_states"},
        "gpu_launches": int(launches),
        "chi2_check": chi2_check,
        "phase_ms_per_lm_iteration": {k: v / max(n_iters, 1) for k, v in phase.items()},
        "roofline": {"bound": "tensor", "kernel": ("supernodal block Cholesky of the %d^2 reduced camera system, %d supernodes (k_snode_update + k_gemm_tn DMMA, k_potrf128)"
                                                   % (n, rcs_info["supernodes"])) if sparse_rcs else
                     "k_chol_dataflow: dense FP64 Cholesky %d^2 as one persistent dataflow kernel (TMA-fed mma.sync.m8n8k4.f64 tile tasks, chain / helper / worker CTAs)" % n,
                     "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                     "kernel_ms": chol_ms, "traffic": traffic, "traffic_source": traffic_src,
                     "factor_phase": {"ms": phase_ms, "tflops": chol_flops / (phase_ms * 1e-3) / 1e12, "frac": chol_flops / (phase_ms * 1e-3) / 1e12 / fp64_peak,
                                      "note": "the whole factor phase of an LM iteration: flag reset, padding, right-hand side copies, the factorisation kernel, the backward solve"},
                     "flops_per_launch": chol_flops,
                     "peak_source": "FP64: cuBLAS DGEMM 4096^3 via torch.matmul measured in this run (no FP64 entry in MEASURED_PEAKS.json)",
                     "hbm_stage": {"kernel": "linearise (k_cam_prepare + k_linearise_cams + k_sum_point_records)",
                                   "achieved_gbs": bytes_lin / (phase["linearise"] / max(n_iters, 1) * 1e-3) / 1e9,
                                   "peak_gbs": hbm_peak, "peak_source": hbm_src}},
    }
    if sparse_rcs:
        # second headline metric (BASELINE.json): Schur-solve ms / LM iteration = reduced system + factor + solve + back-substitution
        it = max(n_iters, 1)
        solve_ms = (phase["schur"] + phase["factor"] + phase["backsubst"]) / it
        line.update({"metric": "schur_solve_ms_per_iteration", "unit": "ms", "value": solve_ms, "higher_is_better": False,
                     "lm_iterations_per_s": value})
        line["config"]["workload"] = (f"{args.shape}-shape BA, LM Optimize({args.lm_iters}, 0) per step, Schur complement + supernodal block-sparse "
                                      "FP64 Cholesky of the reduced camera system (the reference's sparse fallback, LinearSolver_Schur.h:1836-1847)")
        line["config"]["l2_policy"] = "inputs larger than L2 (W+Y %.1f GB, factor %.1f GB vs 126 MB L2)" % (2 * 144e-9 * O, rcs_info["factor_bytes"] * 1e-9)
        line["config"]["rcs"] = {k: v for k, v in rcs_info.items() if k != "order"}
        line["e2e"] = {"value": 1e3 * e2e_s / max(e2e_iters, 1), "unit": "ms per LM iteration (whole call sequence)", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                       "note": "spp_ba_set_graph(host, incl. the device-side structure analysis) + spp_ba_optimize + spp_ba_get_states; the ordering and "
                               "symbolic analysis of the block-sparse factorisation are reused when the same block pattern is uploaded again "
                               "(as the reference reuses its symbolic decomposition while the structure is unchanged)"}
    if world == 1 and not args.no_cpu_baseline and sparse_rcs:
        # the reference cannot finish this shape in bounded time (sparse block Cholesky of ~3e12 flop on one thread): bounded sample
        try:
            gs = graphs.make_ba(g.n_cams // 16, g.n_pts // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
            path = write_graph_file(gs)
            secs, threads, dd = run_reference_steps(path, 1, 1)
            os.unlink(path)
            line["cpu_baseline"] = {"value": 1e3 * float(secs[1]), "unit": "ms per LM iteration (whole iteration, sample)", "cores": threads,
                                    "kind": "reference",
                                    "sample": "unmodified reference (oracle/_ref) on a 1/16 sub-sequence of the same shape: %d cameras, %d points, "
                                              "%d observations; second Optimize(max_iter=1) call" % (gs.n_cams, gs.n_pts, gs.n_obs)}
        except Exception as ex:
            line["cpu_baseline"] = {"value": None, "unit": "ms", "cores": 0, "kind": "reference", "sample": f"failed: {ex}"}
    elif world == 1 and not args.no_cpu_baseline:
        try:
            path = write_graph_file(g)
            secs, threads, _ = run_reference_steps(path, 1, 1)
            os.unlink(path)
            line["cpu_baseline"] = {"value": 1.0 / float(secs[1]), "unit": UNIT, "cores": threads, "kind": "reference",
                                    "sample": "unmodified reference (oracle/_ref), full graph, second Optimize(max_iter=1) call "
                                              "(the first call, which also builds the structure, took %.1f s)" % float(secs[0])}
        except Exception as ex:  # the bench line must still be printed
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {ex}"}
    return line


POSE_SHAPES = {
    # BASELINE.json configs[0] and configs[2] shapes (replicas only: pose graphs do not shard, SURVEY 8(e))
    "manhattan3500": ("make_manhattan", dict(fill_loops=True)),
    "sphere2500": ("make_sphere", dict(n_rings=50, n_per_ring=50, seed=2500, sigma_t=0.004, sigma_r=0.0004, radius=5.0)),
}


def pose_arm(args):
    """Gauss-Newton batch time on a pose-graph shape: one step = CNonlinearSolver_Lambda::Optimize(5, 0) on the resident
    graph (linearise -> block-sparse Cholesky -> update, five times). N > 1 runs N independent replicas."""
    import torch
    from slam_plus_plus_b200 import capi, graphs, sppio
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    gen, kw = POSE_SHAPES[args.shape]
    g = getattr(graphs, gen)(**kw)
    ctx = capi.Context(local)
    ctx.pose_set_graph(g)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    for _ in range(max(args.warmup, 3)):
        ctx.pose_restore_initial()
        rep = ctx.pose_optimize(args.lm_iters, 0.0)
    sampler = ClockSampler(local)
    sampler.start()
    ctx.synchronize()
    if world > 1:
        dist.barrier()
    l0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    phase = {}
    for _ in range(args.steps):
        ctx.pose_restore_initial()
        rep = ctx.pose_optimize(args.lm_iters, 0.0)
        for k, v in rep["ms"].items():
            phase[k] = phase.get(k, 0.0) + v
    e1.record(stream)
    ctx.synchronize()
    torch.cuda.synchronize(dev)
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "", rep, {"poses": ctx.pose_get_states()})
    t0 = time.perf_counter()
    for _ in range(args.steps):  # end to end with host buffers: upload + structure + optimise + download
        ctx.pose_set_graph(g)
        ctx.pose_optimize(args.lm_iters, 0.0)
        ctx.pose_get_states()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        return
    dim, N, E = g.dim, g.poses.shape[0], g.e_from.shape[0]
    line = {
        "metric": "gn_optimize_ms", "value": ms / args.steps, "unit": "ms per Optimize(%d)" % args.lm_iters, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": False,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.shape}-shape pose graph, Gauss-Newton Optimize({args.lm_iters}, 0) per step, block-sparse FP64 Cholesky "
                               f"({dim} x {dim} blocks)", "poses": N, "edges": E, "parallelism": "replicas only" if world > 1 else "single GPU",
                   "l2_policy": "working set (%.1f MB) is L2 resident by nature of the shape" % ((E * (3 * dim * dim + 2 * dim) + N * dim) * 8e-6)},
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_ms, "unit": "ms per set_graph + Optimize + get_states", "h2d_bytes_per_step": int(8 * (N * dim + E * (dim + dim * dim)) + 16 * E),
                "d2h_bytes_per_step": int(8 * N * dim)},
        "gpu_launches": int(launches),
        "phase_ms_per_step": {k: v / args.steps for k, v in phase.items()},
        "roofline": {"bound": "latency", "kernel": "k_sparse_chol (level-scheduled cooperative block Cholesky) + dense root front",
                     "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None,
                     "note": "a %d-pose graph holds ~1e7 flops per factorisation: the step is bound by the dependency depth of the "
                             "elimination tree (grid barriers / kernel launches), not by HBM or the FP64 pipes" % N},
    }
    ref = os.path.join(ROOT, "oracle", "_ref", "ref_driver_pose")
    if not args.no_cpu_baseline and os.path.exists(ref):
        path = os.path.join(tempfile.gettempdir(), f"spp_bench_pose_{os.getpid()}.bin")
        sppio.write_graph(path, g)
        out = subprocess.run([ref, "time", path, path + ".dump", str(args.lm_iters), "0"], capture_output=True, text=True).stdout
        d = sppio.read_dump(path + ".dump")
        os.unlink(path)
        os.unlink(path + ".dump")
        line["cpu_baseline"] = {"value": 1e3 * float(d["optimize_time"][0]), "unit": line["unit"], "cores": int(d["omp_threads"][0]),
                                "kind": "reference", "sample": "unmodified reference (oracle/_ref/ref_driver_pose), the same graph, one Optimize(%d, 0): %s"
                                                               % (args.lm_iters, out.strip())}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every shape measured (the BAL-13682 block included)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--shape", default="venice871")
    ap.add_argument("--lm-iters", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--jacobians", choices=["fd", "analytic"], default="fd",
                    help="fd: forward differences with delta = 1e-9, the reference's own Jacobians (parity mode, the default and "
                         "the configuration of the headline number); analytic: closed-form derivatives")
    ap.add_argument("--no-bal", action="store_true", help="skip the BAL-13682-shape block of the headline line")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write what the last timed step computed (optimised states, "
                    "LM trace) to DIR/<name>.npy, float64, under 64 MB in all")
    ap.add_argument("--write-chi2-trace", default="", metavar="PATH", help="single-GPU run: record the final chi2 of each shape in this "
                    "JSON file (committed as profiles/chi2_trace.json, which every later run is checked against)")
    args = ap.parse_args()
    guard_stdout()
    if args.shape in POSE_SHAPES and args.impl == "b200":
        pose_arm(args)
    elif args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs dumps the outputs of this repository's GPU path (--impl b200)")
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
