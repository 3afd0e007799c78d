"""Jacobi-PCG against Galerkin GMG-PCG on the weighted heat operators (curvilinear tools, cylinder, composite core).

One JSON line per case: iterations per solve, device ms per call (CUDA events of pde_wheat_solve: initial state, every
solve and the snapshot copies), ms per iteration, multigrid set-up ms, and for the GMG run the fine-level k_wsweep
kernels by mode (torch.profiler, a separate run): time per launch, algorithmic bytes per dof, achieved GB/s and the
fraction of the HBM figure bench.py uses (MEASURED_PEAKS.json when present, its fallback otherwise).  The first line
names the GPU and its power limit.

    python scripts/wheat_bench.py [--cases 2d_spherical_4096,...] [--out profiles/wheat_bench.jsonl]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
import pde_solver_b200 as P  # noqa: E402

# Sizes a user of the tools would run; every axis even so that the GMG hierarchy coarsens.
CASES = {
    "2d_spherical_4096": dict(fn="_solve_heat_2d_spherical_raw", nodes=4097 ** 2, nh=4,
                              kw=dict(r_inner=0.0, r_outer=1.0, nr=4096, ntheta=4096, diffusivity=1.0,
                                      T_boundary=35.0, T_initial=0.0, dt=0.01, num_steps=1, steady=True,
                                      source_type="constant", source_value=40.0)),
    "3d_spherical_256x128x256": dict(fn="_solve_heat_3d_spherical_raw", nodes=257 * 129 * 257, nh=8,
                                     kw=dict(r_inner=0.2, r_outer=1.0, nr=256, ntheta=128, nphi=256, diffusivity=1.0,
                                             T_boundary=35.0, T_initial=0.0, dt=0.01, num_steps=1, steady=True,
                                             source_type="constant", source_value=40.0)),
    "core_box_512_5steps": dict(fn="_solve_heat_3d_raw", nodes=513 ** 3, nh=8,
                                kw=dict(Lx=1.0, Ly=1.0, Lz=1.0, nx=512, ny=512, nz=512, diffusivity=1.0,
                                        T_boundary=0.0, T_initial=20.0, dt=0.01, num_steps=5, core_radius=0.3,
                                        core_diffusivity=25.0, snapshot_stride=5)),
    "cylinder_256": dict(fn="_solve_heat_3d_raw", nodes=257 ** 3, nh=8,
                         kw=dict(Lx=1.0, Ly=1.0, Lz=1.0, nx=256, ny=256, nz=256, diffusivity=1.0, T_boundary=0.0,
                                 T_initial=0.0, dt=0.01, num_steps=1, steady=True, source_type="constant",
                                 source_value=40.0, geometry_type="cylinder", cylinder_radius=0.5)),
}
MODES = ("first", "apply", "resid", "cheby")


def run(case, precond):
    c = CASES[case]
    f = getattr(P, c["fn"])(**c["kw"], precond=precond, as_arrays=True)
    return np.asarray(f.values[-1]), P.last_stats()


def sweep_bytes(mode, nh, with_prev):
    """Algorithmic bytes per dof of one k_wsweep launch: every plane and vector once."""
    planes = {"first": 3, "apply": nh + 2, "resid": nh + 3, "cheby": nh + 3 + (1 if with_prev else 0)}[mode]
    return 8.0 * planes


def profile_sweeps(case):
    """Fine-level k_wsweep launches of one GMG call, by mode.  Per V-cycle the sweeps run in a fixed order: level 0
    first/cheby/resid, the coarser levels, level 0 cheby (restart)/cheby (with x_prev) last."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(case, "gmg")
    st_p = P.last_stats()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            ev = json.load(fh)["traceEvents"]
    k = sorted((e for e in ev if e.get("cat") == "kernel" and "k_wsweep" in e.get("name", "")), key=lambda e: e["ts"])

    def mode(e):
        return MODES[int(re.search(r"k_wsweep<\s*\d+\s*,\s*(\d+)\s*>", e["name"]).group(1))]

    apply_ = [e for e in k if mode(e) == "apply"]
    rest = [e for e in k if mode(e) != "apply"]
    cycles = st_p["iters_total"] + st_p["solves"]
    per = len(rest) // cycles if cycles else 0
    fine = {m: [] for m in MODES}
    fine["apply"] = [(e["dur"], False) for e in apply_]
    for cyc in range(cycles):
        seg = rest[cyc * per:(cyc + 1) * per]
        for pos, with_prev in ((0, False), (1, False), (2, False), (per - 2, False), (per - 1, True)):
            fine[mode(seg[pos])].append((seg[pos]["dur"], with_prev))
    peaks, kind = bench.measured_peaks()
    out = {}
    nodes, nh = CASES[case]["nodes"], CASES[case]["nh"]
    for m in MODES:
        if not fine[m]:
            continue
        us = sum(d for d, _ in fine[m]) / len(fine[m])
        bpd = sum(sweep_bytes(m, nh, w) for _, w in fine[m]) / len(fine[m])
        gbs = nodes * bpd / (us * 1e-6) / 1e9
        out[m] = {"launches": len(fine[m]), "us_per_launch": round(us, 1), "bytes_per_dof": bpd,
                  "achieved_gbs": round(gbs, 1), "frac_of_peak": round(gbs / peaks["hbm_gbs"], 3)}
    return out, {"hbm_gbs": peaks["hbm_gbs"], "source": f"MEASURED_PEAKS.json ({kind})" if kind == "measured"
                 else "bench.py fallback"}


def summary(st):
    it = st["iters_total"] / max(1, st["solves"])
    return {"levels": st["levels"], "solves": st["solves"], "iters_per_solve": round(it, 1),
            "ms_per_call": round(st["solve_ms"], 2), "ms_per_solve": round(st["solve_ms"] / max(1, st["solves"]), 2),
            "ms_per_iter": round(st["solve_ms"] / max(1, st["iters_total"]), 4), "setup_ms": round(st["setup_ms"], 1),
            "true_relres": st["true_relres"], "final_relres": st["final_relres"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    lines = []
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines.append({"gpu": gpu[0] if gpu else "unknown"})
    # warm-up: module load and first launches of every kernel family, both paths
    for pre in ("jacobi", "gmg"):
        P._solve_heat_2d_spherical_raw(0.0, 1.0, 32, 32, 1.0, 35.0, 0.0, 0.01, 1, steady=True, precond=pre)
        P._solve_heat_3d_raw(1, 1, 1, 8, 8, 8, 1.0, 0.0, 0.0, 0.01, 1, steady=True, core_radius=0.3,
                             core_diffusivity=25.0, precond=pre)
    for case in a.cases.split(","):
        vj, sj = run(case, "jacobi")
        vg, sg = run(case, "gmg")
        rel = float(np.linalg.norm(vg - vj) / max(np.linalg.norm(vj), 1e-300))
        sweeps, peak = profile_sweeps(case)
        lines.append({"case": case, "jacobi": summary(sj), "gmg": summary(sg),
                      "speedup_per_call": round(sj["solve_ms"] / sg["solve_ms"], 2), "rel_l2_gmg_vs_jacobi": rel,
                      "k_wsweep_fine_level": sweeps, "hbm_peak": peak})
        print(json.dumps(lines[-1]), flush=True)
    print(json.dumps(lines[0]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as fh:
            for ln in lines:
                fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
