"""Streamed against in-memory snapshots for the weighted heat solves (composite core, GMG-PCG).

Each case runs in a process of its own, so that its peak host RSS (resource.getrusage, ru_maxrss) belongs to that case
alone.  One JSON line per case: device ms per step (sum of the per-step solve_ms of the resident stepper, or
pde_wheat_solve's solve_ms for the in-memory path, over the steps), wall ms per step (host clock around the whole
call, set-up included), peak RSS, bytes written, iterations, and the card's name and power limit read in the same run.
The 256^3 in-memory case also reports whether its snapshots equal the streamed file bit for bit.

    python scripts/wheat_stream_bench.py [--out-dir DIR] [--cases core_512_stream,...] [--jsonl FILE]

The streamed files go to --out-dir (default: a temporary directory, removed at the end); 512^3 with 20 steps writes
21 x 1.08 GB."""
import argparse
import json
import os
import resource
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# composite core on the unit box, as in scripts/wheat_bench.py; 20 backward-Euler steps, every state kept
CASES = {
    "core_512_stream": dict(n=512, stream=True),
    "core_256_stream": dict(n=256, stream=True),
    "core_256_memory": dict(n=256, stream=False, compare="core_256_stream"),
}
STEPS = 20


def _npz(out_dir, case):
    return os.path.join(out_dir, case + ".npz")


def run_case(case, out_dir):
    sys.path.insert(0, ROOT)
    import numpy as np
    import pde_solver_b200 as P
    from pde_solver_b200 import io

    c = CASES[case]
    n = c["n"]
    kw = dict(core_radius=0.3, core_diffusivity=25.0, precond="gmg", snapshot_stride=1, as_arrays=True)
    args = (1.0, 1.0, 1.0, n, n, n, 1.0, 0.0, 20.0, 0.01, STEPS)
    # warm-up: module load and the first launch of every kernel of both paths
    small = (1.0, 1.0, 1.0, 16, 16, 16, 1.0, 0.0, 20.0, 0.01, 2)
    P._solve_heat_3d_raw(*small, **kw)
    with tempfile.TemporaryDirectory() as d:
        with io.open_writer("npz", os.path.join(d, "w.npz"), 3, [16] * 3, [1.0] * 3) as w:
            P._solve_heat_3d_raw(*small, stream_to=w, **kw)
    written = 0
    t0 = time.perf_counter()
    if c["stream"]:
        path = _npz(out_dir, case)
        with io.open_writer("npz", path, 3, [n] * 3, [1.0] * 3) as w:
            f = P._solve_heat_3d_raw(*args, stream_to=w, **kw)
        wall = time.perf_counter() - t0
        written = os.path.getsize(path)
    else:
        f = P._solve_heat_3d_raw(*args, **kw)
        wall = time.perf_counter() - t0
    st = P.last_stats()
    rss_gb = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024 / 1e9
    out = {"case": case, "nodes": (n + 1) ** 3, "steps": STEPS, "snapshots_kept": STEPS + 1,
           "mode": "streamed to npz" if c["stream"] else "in memory",
           "device_ms_per_step": round(st["solve_ms"] / STEPS, 2), "wall_ms_per_step": round(1e3 * wall / STEPS, 2),
           "wall_s_total": round(wall, 2), "peak_rss_gb": round(rss_gb, 3), "bytes_written": written,
           "snapshot_gb": round((n + 1) ** 3 * 8 / 1e9, 3), "levels": st["levels"],
           "iters_per_step": round(st["iters_total"] / max(1, st["solves"]), 2), "setup_ms": round(st["setup_ms"], 1),
           "true_relres": st["true_relres"], "converged": st["converged"]}
    if c.get("compare"):
        ref = _npz(out_dir, c["compare"])
        same = os.path.exists(ref)
        if same:
            with np.load(ref) as z:
                same = len(z["times"]) == f.values.shape[0] and all(
                    np.array_equal(z[f"t{k:06d}"], f.values[k]) for k in range(f.values.shape[0]))
        out["bitwise_equal_to"] = {c["compare"]: bool(same)}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out-dir", default=None, help="where the streamed files go (kept when given)")
    ap.add_argument("--jsonl", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.one:
        run_case(a.one, a.out_dir)
        return
    smi = shutil.which("nvidia-smi")
    q = smi and subprocess.run([smi, "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True)
    if not q or q.returncode != 0 or not q.stdout.strip():
        sys.exit("nvidia-smi found no GPU: this benchmark measures the GPU and has no CPU mode")
    name, power = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    out_dir = a.out_dir or tempfile.mkdtemp(prefix="wheat_stream_")
    os.makedirs(out_dir, exist_ok=True)
    lines = []
    try:
        for case in a.cases.split(","):
            free_gb = shutil.disk_usage(out_dir).free / 1e9
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", case, "--out-dir", out_dir],
                               capture_output=True, text=True)
            if r.returncode != 0:
                line = {"case": case, "error": r.stderr.strip().splitlines()[-1:] or ["exit %d" % r.returncode]}
            else:
                line = json.loads(r.stdout.strip().splitlines()[-1])
            line.update(gpu=name, power_limit=power, disk_free_gb_before=round(free_gb, 1))
            lines.append(line)
            print(json.dumps(line), flush=True)
            if a.out_dir is None and case not in {c.get("compare") for c in CASES.values()} \
                    and os.path.exists(_npz(out_dir, case)):
                os.remove(_npz(out_dir, case))
    finally:
        if a.out_dir is None:
            shutil.rmtree(out_dir, ignore_errors=True)
    if a.jsonl:
        os.makedirs(os.path.dirname(os.path.abspath(a.jsonl)), exist_ok=True)
        with open(a.jsonl, "a") as fh:
            for ln in lines:
                fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
