#!/usr/bin/env python
"""Headline benchmark of the hot path (BASELINE.json): 3D P1 heat, backward Euler, config 4 - plus the other half of
the metric (3D elasticity, config 5), strong scaling of both, and the smaller configs.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (SciPy port)
    python bench.py ... --dump-outputs DIR                   # also save a fixed sample of the computed field

--dump-outputs DIR writes the temperature field the timed steps left in HBM (the state a caller of the stepper reads
back), sampled at fixed, seeded vertex indices, as DIR/heat_temperature.npy (float64), so that two builds can be
compared output for output: with the same arguments the inputs and the sampled indices are the same on every run.

One "step" = one backward-Euler time step (a full linear solve to rtol 1e-10) of the heat equation on the
unit-cube-per-GPU 512^3 P1 mesh (135 M dofs per GPU; weak scaling stacks slabs along z).
`value` = dofs advanced one time step per second (GDOF/s = dofs x time steps / s; NOT dofs x CG iterations: that
figure is `gdof_iters_per_s`), state resident in HBM, timed with CUDA events on the library's stream, max over ranks.
Extra keys (same JSON line): CG iterations/s, the whole-step roofline fraction with its stated bytes per dof, the
sweep-kernel rooflines of both operators measured live, the kernel share table of the committed ncu launch list,
3D elasticity (weak and strong), strong scaling of config 4, configs 1-3, the halo path the library actually took with
its exchange / all-reduce counts per iteration, the end-to-end number through the C ABI with host buffers, a bounded
CPU baseline and the clocks seen during the timed region.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: cells per GPU (weak scaling stacks these blocks along z), matching elasticity block
    "heat3d_512": dict(n=(512, 512, 512), kappa=1.0, dt=0.01, T_initial=20.0, T_boundary=0.0, elast=(1280, 256, 256)),
    "heat3d_256": dict(n=(256, 256, 256), kappa=1.0, dt=0.01, T_initial=20.0, T_boundary=0.0, elast=(640, 128, 128)),
    "heat3d_128": dict(n=(128, 128, 128), kappa=1.0, dt=0.01, T_initial=20.0, T_boundary=0.0, elast=(320, 64, 64)),
}

# Bytes per dof and PCG iteration on the fine level, by the kernels that actually run (DESIGN.md §5):
#   CG part  : apply 16 + r update 24 + p / deferred x update 40                                   = 80
#   V-cycle  : fused first two sweeps 16 + fused residual-and-restriction 17 + prolongation 17 + fused post sweeps 24 = 74
#              (round 1, before the residual / restriction fusion: 24 + 9 instead of 17 = 90)
#   coarser levels repeat the V-cycle part on 1/8 of the dofs each: x 8/7
HEAT_STEP_BYTES = 80.0 + 74.0 * 8.0 / 7.0
HEAT_STEP_BYTES_R1 = 80.0 + 90.0 * 8.0 / 7.0      # the round-1 accounting VERDICT r1 quotes (183 B): kept for comparison
#   elasticity (natural faces): fused first two sweeps 16 + residual 24 + restriction 9 + prolongation 17 + restart sweep 24
#   + sweep with x_prev 32 = 122   (round 1, before the first-sweeps fusion: 16 + 24 instead of 16 = 146)
ELAST_STEP_BYTES = 80.0 + 122.0 * 8.0 / 7.0
ELAST_STEP_BYTES_R1 = 80.0 + 146.0 * 8.0 / 7.0
SWEEP_BYTES = {0: 16, 1: 24, 2: 24, 3: 32}
SWEEP_NAME = {0: "apply (+fused dots)", 1: "residual", 2: "chebyshev sweep (restart)", 3: "chebyshev sweep (with x_prev)"}
DUMP_SAMPLES = 1 << 21          # --dump-outputs: vertices kept of the 135 M of heat3d_512 (16 MB of float64)
DUMP_SEED = 20261020


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def profile_json(name):
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            with open(p) as f:
                return json.load(f)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
LU_SECONDS_PER_STEP = {24: 1.1, 32: 5.0, 40: 21.0}     # measured on the 8-core container host (SuperLU, one thread)


def run_reference(args):
    """The reference's own per-step work on the host cores: assemble + row-wise BC + sparse LU (what DOLFIN's
    solve() does every step), at the largest size whose K+W steps finish in about a minute; plus a Krylov leg
    (assembled CSR, Jacobi-PCG, rtol 1e-10) at 128^3.  SciPy restatement (FEniCS is not installable), one thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle.reference_arm import HeatCsrCg3D, HeatReference3D
    total = args.steps + args.warmup
    n = max([k for k, s in LU_SECONDS_PER_STEP.items() if s * total <= 75.0] or [24])
    ref = HeatReference3D(n)
    cpu0, w0 = time.process_time(), time.perf_counter()
    sec = ref.run(args.steps, args.warmup)
    busy = (time.process_time() - cpu0) / max(1e-9, time.perf_counter() - w0)      # BLAS threads inside SuperLU / NumPy count
    cores = max(1, int(round(busy)))
    val = ref.ndofs * args.steps / sec / 1e9
    cg = None
    if not args.no_cg_leg:
        cn = args.cg_cells
        t0 = time.perf_counter()
        kr = HeatCsrCg3D(cn)
        setup = time.perf_counter() - t0
        cpu1 = time.process_time()
        t0 = time.perf_counter()
        kr.step()
        csec = time.perf_counter() - t0
        kbusy = (time.process_time() - cpu1) / max(1e-9, csec)
        cg = {"sample": f"3D heat {cn}^3 cells ({kr.ndofs} dofs), 1 backward-Euler step, CSR assembled once "
                        f"({setup:.1f} s, not timed), Jacobi-PCG rtol 1e-10 from the warm start",
              "value": kr.ndofs / csec / 1e9, "unit": "GDOF/s", "seconds_per_step": csec, "cg_iters": kr.iters,
              "gdof_iters_per_s": kr.ndofs * kr.iters / csec / 1e9, "cores": max(1, int(round(kbusy))),
              "cores_busy": round(kbusy, 2), "kind": "port"}
    sample = (f"3D heat {n}^3 cells ({ref.ndofs} dofs; the largest size whose {total} steps fit in about a minute of "
              f"the reference's O(n^6) sparse LU - the GPU arm runs 512^3), same kappa/dt/IC/BC; per step: assemble A and b, "
              "row-wise Dirichlet, SuperLU factorise+solve (what DOLFIN solve() does each step); SciPy restatement: "
              "assembly and SuperLU are serial, its BLAS calls may use more threads - `cores` is the measured CPU time / wall time")
    out = {
        "impl": "reference", "metric": "GDOF/s", "value": val, "unit": "GDOF/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "sample": f"{n}^3 cells ({ref.ndofs} dofs), same kappa/dt/IC/BC",
                   "same_config": False},
        "cpu_baseline": {"value": val, "unit": "GDOF/s", "cores": cores, "cores_busy": round(busy, 2),
                         "cores_available": os.cpu_count(), "kind": "port", "sample": sample},
        "krylov_leg": cg,
        "e2e": {"value": val, "unit": "GDOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    args.emit_restore()
    print(json.dumps(out), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ native arm
def run_native(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    import numpy as np
    from pde_solver_b200 import _lib

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.Context(local_rank)
    if world > 1:
        path = _lib.nccl_library_path()
        uid = [_lib.nccl_unique_id(path) if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0], path)

    def barrier():
        ctx.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def reduce_ranks(x, op):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    def max_over_ranks(x):
        return reduce_ranks(x, "MAX")

    def sum_over_ranks(x):
        return reduce_ranks(x, "SUM")

    peaks, peak_kind = measured_peaks()
    peak = peaks["hbm_gbs"]
    w = WORKLOADS[args.workload]
    bc = _lib.make_bc({f: w["T_boundary"] for f in range(6)})
    opts = _lib.make_opts(rtol=args.rtol, precond=args.precond)

    def heat_run(n, L, steps, warmup):
        """`steps` timed backward-Euler steps on the global grid n (slab-partitioned over the ranks)."""
        hs = _lib.HeatStepper(ctx, 3, n, L, w["kappa"], w["dt"], T_initial=w["T_initial"], bc=bc, opts=opts)
        for _ in range(warmup):
            hs.step(1)
        barrier()
        c0 = _lib.comm_info(ctx)
        st = hs.step(steps)
        barrier()
        c1 = _lib.comm_info(ctx)
        ms = max_over_ranks(st["solve_ms"])
        nd = (n[0] + 1) * (n[1] + 1) * (n[2] + 1)
        it = max(1, st["iters_total"])
        return hs, {"cells": list(n), "dofs": nd, "ms_per_step": ms / steps, "value_gdofs": nd * steps / (ms / 1e3) / 1e9,
                    "cg_iters_per_step": st["iters_total"] / steps, "ms_per_iter": ms / it,
                    "gdof_iters_per_s": nd * st["iters_total"] / (ms / 1e3) / 1e9, "levels": st["levels"],
                    "converged": bool(st["converged"]), "final_relres": st["final_relres"],
                    "true_relres": st["true_relres"], "launches": int(st["launches"]),
                    "halo_exchanges_per_iter": (c1["halo_exchanges"] - c0["halo_exchanges"]) / it,
                    "allreduces_per_iter": (c1["allreduces"] - c0["allreduces"]) / it, "_st": st, "_ms": ms}

    def elast_run(n, L, reps=2):
        """Cantilever under gravity on the global grid n (z-slabs over the ranks): GMG-PCG + von Mises projection
        through pde_elasticity_solve (the C ABI behind solve_elasticity_3D_static); best of `reps`."""
        z0, nzl, nzg = _lib.slab_partition(3, n, rank, world)
        nloc = (n[0] + 1) * (n[1] + 1) * nzl
        ep = _lib.ElastParams()
        ep.dim = 3
        ep.n = _lib.i3(n)
        ep.L = _lib.d3(L)
        ep.E, ep.nu = 210e9, 0.3
        ep.body = _lib.d3([0.0, 0.0, -76518.0], 0.0)
        ep.quantity, ep.plane_stress, ep.area = 0, 0, 1.0
        vm = _lib.PinnedArray(nloc)
        o = _lib.make_opts(rtol=args.rtol, precond="gmg")
        best = None
        for _ in range(reps):
            st, sp = _lib.Stats(), _lib.Stats()
            barrier()
            c0 = _lib.comm_info(ctx)
            t0 = time.perf_counter()
            _lib.check(_lib.lib().pde_elasticity_solve(ctx.handle, C.byref(ep), C.byref(o), _lib.ptr(vm.array), None,
                                                       C.byref(st), C.byref(sp)))
            barrier()
            wall = max_over_ranks(time.perf_counter() - t0)
            c1 = _lib.comm_info(ctx)
            ms = max_over_ranks(st.solve_ms)
            if best is None or ms < best["solve_ms"]:
                nd = 3 * (n[0] + 1) * (n[1] + 1) * (n[2] + 1)
                it = max(1, st.iters_total)
                best = {"cells": list(n), "dofs": nd, "cg_iters": int(st.iters_total), "solve_ms": ms,
                        "ms_per_iter": ms / it, "setup_ms": max_over_ranks(st.setup_ms),
                        "projection_ms": max_over_ranks(sp.solve_ms), "gdofs_per_s": nd / (ms / 1e3) / 1e9,
                        "cg_iters_per_s": st.iters_total / (ms / 1e3),
                        "gdof_iters_per_s": nd * st.iters_total / (ms / 1e3) / 1e9, "converged": bool(st.converged),
                        "final_relres": st.final_relres, "true_relres": st.true_relres, "levels": int(st.levels),
                        "e2e_wall_s": wall, "launches": int(st.launches),
                        "halo_exchanges_per_iter": (c1["halo_exchanges"] - c0["halo_exchanges"]) / it,
                        "allreduces_per_iter": (c1["allreduces"] - c0["allreduces"]) / it}
        vm.free()
        best["roofline_step"] = step_roofline(best["dofs"], best["cg_iters"], best["solve_ms"], ELAST_STEP_BYTES)
        best["roofline_step"]["frac_by_round1_accounting_247B"] = step_roofline(best["dofs"], best["cg_iters"], best["solve_ms"],
                                                                              ELAST_STEP_BYTES_R1)["frac"]
        return best

    def step_roofline(dofs, iters, ms, bpd):
        ach = dofs * iters * bpd / (ms / 1e3) / 1e9 / world          # per GPU
        return {"bound": "hbm", "bytes_per_dof_iter": round(bpd, 1), "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "note": "whole solve: fine-level kernels by their own traffic, coarser levels x 8/7"}

    def sweep_rooflines(kind, n, L, faces, modes=(0, 1, 2, 3)):
        """Every sweep mode of one operator on this rank's slab, timed with CUDA events on the library's stream."""
        lam, mu = 121.15e9, 80.77e9
        p = _lib.op_params(kind, 3, n, L, 1.0, w["dt"] * w["kappa"], lam, mu, bc=_lib.make_bc(faces))
        out = []
        for m in modes:
            barrier()
            ms, nd = _lib.op_bench_mode(ctx, p, m, reps=10, warmup=3)
            ms = max_over_ranks(ms)
            ach = SWEEP_BYTES[m] * nd / (ms / 1e3) / 1e9
            out.append({"kernel": SWEEP_NAME[m], "bytes_per_dof": SWEEP_BYTES[m], "ms_per_launch": ms, "achieved": ach,
                        "frac": ach / peak})
        return out, nd

    def dump_field(name, local, n):
        """Sample a nodal field held as z-slabs (this rank's part of the natural vertex order) at fixed, seeded global
        vertex indices; rank 0 writes the sample as DIR/<name>.npy."""
        plane = (n[0] + 1) * (n[1] + 1)
        nglob = plane * (n[2] + 1)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(nglob, min(DUMP_SAMPLES, nglob), replace=False))
        z0, nzl, _ = _lib.slab_partition(3, n, rank, world)
        if local.size != nzl * plane:
            raise RuntimeError(f"rank {rank} holds {local.size} vertices, its slab has {nzl * plane}")
        lo = z0 * plane
        mine = (idx >= lo) & (idx < lo + local.size)
        vals = np.zeros(idx.size)
        vals[mine] = local[idx[mine] - lo]
        if dist is not None:          # each index lies in exactly one slab, so the sum over ranks is exact
            import torch
            t = torch.from_numpy(vals).cuda()
            dist.all_reduce(t)
            vals = t.cpu().numpy()
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, name + ".npy"), vals)

    # ---- 1. headline: heat, weak scaling (inputs resident in HBM) ----
    n_w = [w["n"][0], w["n"][1], w["n"][2] * world]
    L_w = [1.0, 1.0, 1.0 * world]
    sampler = ClockSampler(local_rank)
    hs = _lib.HeatStepper(ctx, 3, n_w, L_w, w["kappa"], w["dt"], T_initial=w["T_initial"], bc=bc, opts=opts)
    for _ in range(args.warmup):
        hs.step(1)
    barrier()
    if rank == 0:
        sampler.start()
    c0 = _lib.comm_info(ctx)
    st = hs.step(args.steps)
    barrier()
    c1 = _lib.comm_info(ctx)
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(st["solve_ms"])
    ndofs = (n_w[0] + 1) * (n_w[1] + 1) * (n_w[2] + 1)
    value = ndofs * args.steps / (ms / 1e3) / 1e9
    iters = st["iters_total"]

    # ---- 2. end to end through the C ABI with pinned HOST buffers (H2D + step + D2H per step) ----
    # every step: H2D copy of that step's input field from pinned host memory, one backward-Euler solve, D2H read of
    # the result into pinned host memory.  (1) pipelined: pde_heat_advance_batch over e_steps independent requests;
    # the upload of request k+1 and the download of result k-1 run on copy streams while request k is solved.
    # (2) serial, for comparison: set_state / step / get_state, the result being the next step's input.
    hbuf = _lib.PinnedArray(hs.nloc)
    hs.get_state(hbuf.array)                            # the state after the timed steps
    if args.dump_outputs:
        dump_field("heat_temperature", hbuf.array, n_w)
    e_steps = max(1, args.steps)
    h_in = [_lib.PinnedArray(hs.nloc) for _ in range(2)]
    h_out = [_lib.PinnedArray(hs.nloc) for _ in range(2)]
    for b in h_in:
        b.array[:] = hbuf.array
    ins = [h_in[k % 2].array for k in range(e_steps)]
    outs = [h_out[k % 2].array for k in range(e_steps)]
    hs.advance_batch(ins[:2], outs[:2])                 # untimed: allocates the staging buffers and streams
    barrier()
    t0 = time.perf_counter()
    hs.advance_batch(ins, outs)
    barrier()
    e_sec = max_over_ranks(time.perf_counter() - t0)
    e2e = ndofs * e_steps / e_sec / 1e9
    s_steps = max(1, min(args.steps, 3))
    barrier()
    t0 = time.perf_counter()
    for _ in range(s_steps):
        hs.set_state(hbuf.array)
        hs.step(1)
        hs.get_state(hbuf.array)
    barrier()
    s_sec = max_over_ranks(time.perf_counter() - t0)
    e2e_serial = ndofs * s_steps / s_sec / 1e9
    bytes_dir = int(sum_over_ranks(hs.nloc * 8))
    for b in h_in + h_out:
        b.free()
    hs.close()
    hbuf.free()

    # ---- 3. kernel rooflines measured live: the sweep modes of both operators on this rank's slab ----
    heat_sweeps, op_nd = sweep_rooflines("heat", n_w, L_w, {f: 0.0 for f in range(6)})
    op_ms = heat_sweeps[0]["ms_per_launch"]
    traffic = profile_json("traffic.json") or {}
    roofline = {"bound": "hbm", "achieved": heat_sweeps[0]["achieved"], "peak": peak, "unit": "GB/s",
                "frac": heat_sweeps[0]["frac"], "traffic": (traffic.get(args.workload) or {}).get("dram_bytes_per_launch"),
                "kernel": "heat operator apply k_sweep3d<1,4,APPLY> (+fused dots)",
                "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})", "ms_per_launch": op_ms,
                "per_gpu_dofs": op_nd, "nominal_8TBs_frac": heat_sweeps[0]["achieved"] / 8000.0}
    roofline_step = step_roofline(ndofs, iters, ms, HEAT_STEP_BYTES)
    roofline_step["frac_by_round1_accounting_183B"] = step_roofline(ndofs, iters, ms, HEAT_STEP_BYTES_R1)["frac"]

    # ---- 4. halo exchange (N > 1): one 513x513 plane each way per z-neighbour over NVLink ----
    halo = None
    if world > 1:
        barrier()
        h_ms, h_bytes = _lib.halo_bench(ctx, 3, n_w, 1, reps=50)
        h_ms = max_over_ranks(h_ms)
        plane_bytes = (((n_w[0] + 2 + 3) // 4) * 4) * (n_w[1] + 2) * 8      # one padded vertex plane
        gbs = plane_bytes / (h_ms / 1e3) / 1e9 if h_ms > 0 else None
        halo = {"us_per_exchange": 1e3 * h_ms, "plane_bytes": plane_bytes,
                "bytes_sent_per_rank_max": int(max_over_ranks(h_bytes)), "gbs_per_direction": gbs,
                "nvlink_peer_copy_peak_gbs": 770.0, "frac_of_nvlink": gbs / 770.0 if gbs else None,
                "path": _lib.comm_info(ctx)["halo_path"],
                "exchanges_per_iter": (c1["halo_exchanges"] - c0["halo_exchanges"]) / max(1, iters),
                "allreduces_per_iter": (c1["allreduces"] - c0["allreduces"]) / max(1, iters),
                "note": "one contiguous plane per neighbour; latency-bound at this size (flag round trips, not bytes)"}

    # ---- 5. strong scaling of config 4: the SAME global grid split over the ranks ----
    strong = None
    if world > 1 and not args.no_strong:
        hs2, strong_heat = heat_run(list(w["n"]), [1.0, 1.0, 1.0], max(3, args.steps // 2), 3)
        hs2.close()
        strong_heat = {k: v for k, v in strong_heat.items() if not k.startswith("_")}
        strong_heat["roofline_step"] = step_roofline(strong_heat["dofs"], strong_heat["cg_iters_per_step"],
                                                     strong_heat["ms_per_step"], HEAT_STEP_BYTES)
        strong = {"heat": strong_heat}

    # ---- 6. the other half of the headline metric: 3D elasticity (config 5 block per GPU, weak; and config 5 strong) ----
    elast = None
    if not args.no_elasticity:
        en = w["elast"]
        sc = en[0] / 1280.0
        e_sweeps, e_nd = sweep_rooflines("elasticity", [en[0], en[1], en[2] * world], [1.0 * sc, 0.2 * sc, 0.2 * sc * world],
                                         {0: 0.0})
        elast = elast_run([en[0], en[1], en[2] * world], [1.0 * sc, 0.2 * sc, 0.2 * sc * world])
        elast["workload"] = (f"elast3d cantilever {en[0]}x{en[1]}x{en[2]} cells per GPU (z-slabs x{world}), gravity, "
                             f"GMG-PCG rtol {args.rtol:g}; 16 B/dof apply incl. the face-row kernel")
        etr = (traffic.get("elast3d_1280x256x256") or {}).get("dram_bytes_per_launch") if en[0] == 1280 else None
        elast["roofline"] = {"bound": "hbm", "kernel": "elasticity operator apply k_elast3d<APPLY> + k_face_rows (+fused dots)",
                             "achieved": e_sweeps[0]["achieved"], "peak": peak, "unit": "GB/s", "frac": e_sweeps[0]["frac"],
                             "ms_per_launch": e_sweeps[0]["ms_per_launch"], "per_gpu_dofs": e_nd, "traffic": etr,
                             "nominal_8TBs_frac": e_sweeps[0]["achieved"] / 8000.0}
        elast["sweeps"] = e_sweeps
        if world > 1 and not args.no_strong:
            es = elast_run(list(en), [1.0 * sc, 0.2 * sc, 0.2 * sc], reps=2)
            strong["elasticity"] = es

    # ---- 7. the smaller BASELINE configs (N = 1 only; device-resident steppers / the host API) ----
    configs = None
    if world == 1 and not args.no_configs:
        import pde_solver_b200 as P
        configs = {}
        t0 = time.perf_counter()
        P._solve_heat_1d_raw(2.0, 100, 1.0, 20.0, 0.0, 0.0, 0.01, 200, as_arrays=True)
        s1 = P.last_stats()
        configs["cfg1_heat1d_100"] = {"steps": 200, "solve_ms": s1["solve_ms"], "wall_s": time.perf_counter() - t0,
                                      "cg_iters": s1["iters_total"]}
        n2 = [4096, 4096]
        h2 = _lib.HeatStepper(ctx, 2, n2, [1.0, 1.0], 1.0, 0.01, T_initial=20.0, bc=_lib.make_bc({f: 0.0 for f in range(4)}),
                              opts=opts)
        h2.step(3)
        s2 = h2.step(20)
        h2.close()
        nd2 = 4097 * 4097
        configs["cfg2_heat2d_4096"] = {"dofs": nd2, "steps": 20, "ms_per_step": s2["solve_ms"] / 20,
                                       "cg_iters_per_step": s2["iters_total"] / 20,
                                       "value_gdofs": nd2 * 20 / (s2["solve_ms"] / 1e3) / 1e9, "levels": s2["levels"],
                                       "true_relres": s2["true_relres"]}
        e3 = elast_run([320, 64, 64], [1.0, 0.2, 0.2], reps=2)
        configs["cfg3_elast3d_320x64x64"] = {k: e3[k] for k in ("dofs", "cg_iters", "solve_ms", "projection_ms", "gdofs_per_s",
                                                                "gdof_iters_per_s", "true_relres", "levels")}
        configs["cfg3_elast3d_320x64x64"]["note"] = "31 MiB per vector: largely L2-resident, not an HBM-roofline case"

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- 8. bounded CPU baseline (rank 0, N=1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle.reference_arm import HeatReference3D
        cn, csteps = 32, 3
        ref = HeatReference3D(cn)
        cpu0, w0 = time.process_time(), time.perf_counter()
        csec = ref.run(csteps, 0)
        busy = (time.process_time() - cpu0) / max(1e-9, time.perf_counter() - w0)
        cpu = {"value": ref.ndofs * csteps / csec / 1e9, "unit": "GDOF/s", "cores": max(1, int(round(busy))),
               "cores_busy": round(busy, 2), "cores_available": os.cpu_count(), "kind": "port",
               "sample": f"3D heat {cn}^3 cells ({ref.ndofs} dofs), {csteps} steps of assemble + row-wise BC + SuperLU "
                         "factorise/solve per step (SciPy restatement of the FEniCS path; cores = measured CPU time / wall time; "
                         "`--impl reference` adds an assembled-CSR Jacobi-PCG leg at 128^3)"}

    kernel_table = profile_json("r02_kernel_table.json")
    out = {
        "metric": "GDOF/s", "value": value, "unit": "GDOF/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "cells": n_w, "dofs": ndofs, "dt": w["dt"], "kappa": w["kappa"],
                   "rtol": args.rtol, "precond": "gmg" if st["levels"] > 1 else "jacobi", "mg_levels": st["levels"],
                   "partition": f"z-slabs x{world}", "l2": "vectors (>=1 GiB each) exceed the 126 MB L2",
                   "value_definition": "dofs x backward-Euler time steps / s (one step = one full PCG solve to rtol); "
                                       "dofs x CG iterations / s is gdof_iters_per_s"},
        "cg_iters": iters, "cg_iters_per_s": iters / (ms / 1e3), "cg_iters_per_step": iters / args.steps,
        "ms_per_iter": ms / max(1, iters), "gdof_iters_per_s": ndofs * iters / (ms / 1e3) / 1e9,
        "converged": bool(st["converged"]), "final_relres": st["final_relres"], "true_relres": st["true_relres"],
        "operator_gdofs": op_nd * world / (op_ms / 1e3) / 1e9,
        "roofline": roofline, "roofline_step": roofline_step, "sweeps": heat_sweeps, "kernel_table": kernel_table,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e, "unit": "GDOF/s", "h2d_bytes_per_step": bytes_dir, "d2h_bytes_per_step": bytes_dir,
                "steps": e_steps, "api": "pde_heat_advance_batch (3-stream pipeline, pinned host buffers)",
                "serial_value": e2e_serial, "serial_steps": s_steps,
                "host_gbs_each_direction": bytes_dir * e_steps / e_sec / 1e9,
                "note": "a time stepper keeps its state in HBM (value); this leg moves the whole field both ways every step"},
        "gpu_launches": int(st["launches"]), "clocks": clocks, "elasticity": elast, "strong": strong, "configs": configs,
        "halo": halo,
    }
    args.emit_restore()
    print(json.dumps(out), flush=True)
    os.dup2(2, 1)          # anything printed during teardown goes to stderr again
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    # stdout carries exactly ONE JSON line: libraries that chat on stdout (NCCL prints its version / debug lines there)
    # are sent to stderr for the duration of the run, the result goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit_restore():
        sys.stdout.flush()
        os.dup2(real_stdout, 1)

    rc = 1
    try:
        rc = _main(emit_restore)
    finally:
        sys.stdout.flush()
    return rc


def _main(emit_restore):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="heat3d_512", choices=sorted(WORKLOADS))
    ap.add_argument("--precond", default="auto", choices=["auto", "gmg", "jacobi"])
    ap.add_argument("--rtol", type=float, default=1e-10)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-elasticity", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-cg-leg", action="store_true")
    ap.add_argument("--cg-cells", type=int, default=128)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of the field the timed steps computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3
    args.emit_restore = emit_restore
    if args.impl == "reference":
        return run_reference(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
