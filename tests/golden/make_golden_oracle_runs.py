#!/usr/bin/env python
"""Generates tests/golden/oracle_runs.json: results of the CPU oracle (oracle/spp_oracle.c, the plain-C restatement of
the reference's solvers, pinned against the reference's own golden vectors by tests/test_oracle_cpu.py) on seeded graphs
too large for the .npz goldens, and, where the reference's drivers are built (oracle/build_ref.sh), the reference's own
result beside each ("reference_chi2_final"). The GPU tests compare with these numbers, so they need neither the
reference's sources nor minutes of CPU time at test time.

    python tests/golden/make_golden_oracle_runs.py        # about a minute on one core
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import oracle  # noqa: E402
from slam_plus_plus_b200 import graphs, sppio  # noqa: E402

REF_BA = os.path.join(ROOT, "oracle", "_ref", "ref_driver_ba")


def bal_sixteenth():
    """Optimize(2, 0) on the 1/16 sub-sequence of the BAL-13682 shape (tests/test_rcs_sparse_gpu.py::test_bal_sixteenth_*)"""
    g = graphs.make_ba(13682 // 16, 4456117 // 16, 13682, mean_extra_track=4.5, max_track=120, max_stride=12, loops=1)
    r = oracle.ba_optimize(g, 2, 0.0)
    assert r["status"] == 0
    out = {"max_iter": 2, "chi2_initial": float(r["chi2_initial"]), "chi2_final": float(r["chi2_final"]),
           "alpha_initial": float(r["alpha_initial"]), "n_solves": int(r["n_solves"]), "lm_trace": r["trace"].tolist()}
    if os.path.exists(REF_BA):  # the reference's own Optimize(2, 0) on the same graph
        with tempfile.TemporaryDirectory() as td:
            gp, dp = os.path.join(td, "g.bin"), os.path.join(td, "d.dump")
            sppio.write_graph(gp, g)
            subprocess.run([REF_BA, "time", gp, dp, "2", "0"], check=True, stdout=subprocess.DEVNULL)
            out["reference_chi2_final"] = float(sppio.read_dump(dp)["chi2"][0])
    return out


def main():
    out = {"_about": "CPU oracle (oracle/spp_oracle.c) runs, made by tests/golden/make_golden_oracle_runs.py; "
                     "lm_trace: one row per linear solve, in the layout of the reference drivers' lm_trace",
           "bal_sixteenth": bal_sixteenth()}
    with open(os.path.join(HERE, "oracle_runs.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
