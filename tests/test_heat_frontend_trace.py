"""What the heat front end hands the C ABI, call by call (CPU, no GPU).

A fake library stands in for libpde_b200.so.  It records every call (name, scalar arguments, the bytes of every
parameter / options struct passed by reference, the contents of every host field it is given), answers the mesh
counts and pinned allocations truthfully, fills every values, coordinates and state buffer with a pattern of the call
counter and the entry index, and reports chosen statistics.  Each case runs one public heat function (or a bare
HeatStepper) against it and compares the call trace, the returned field, last_stats() and what the snapshot writer
received with tests/golden/heat_frontend_trace.json, which keeps a digest of each run (see _summary).  The pure
queries pde_mesh_counts, pde_solver_opts_default and pde_*_local_nverts are left out of the trace and do not advance
the counter.

    python tests/test_heat_frontend_trace.py      rewrites the golden file from the current package"""
import ctypes as C
import functools
import hashlib
import json
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pde_solver_b200 import _lib, io, solvers  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "heat_frontend_trace.json")
CELLS_PER_BOX = {1: 1, 2: 2, 3: 6}


def _nv(dim, n):
    return int(np.prod([int(n[q]) + 1 for q in range(int(dim))]))


def _doubles(p, size):
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(size,))


class FakeLib:
    def __init__(self, converged=1):
        self.converged = converged
        self.trace = []
        self.nv = {}                    # stepper handle -> vertices
        self.names = {}                 # fake handle value -> name in the trace
        self.pinned = {}

    def __getattr__(self, name):
        if not name.startswith("pde_"):
            raise AttributeError(name)
        return lambda *args: self._call(name, args)

    def _arg(self, a):
        if a is None or isinstance(a, (int, float)):
            return a
        if isinstance(a, C.c_void_p):
            return self.names.get(a.value, "ptr") if a.value else None
        if isinstance(a, C.Array):
            return list(a)
        if isinstance(a, C._SimpleCData):
            return a.value
        obj = a._obj                    # by reference
        if isinstance(obj, C.Structure) and not isinstance(obj, _lib.Stats):
            return type(obj).__name__ + ":" + bytes(obj).hex()
        return "out"

    def _handle(self, ref, name):
        ref._obj.value = 16 * (len(self.names) + 1)
        self.names[ref._obj.value] = name
        return ref._obj.value

    def _fill(self, p, size, scale=1.0):
        _doubles(p, size)[:] = (1000.0 * len(self.trace) + np.arange(size)) * scale

    def _stats(self, ref, nv):
        k = len(self.trace)
        st = ref._obj
        st.ndofs, st.iters_total, st.solves, st.converged, st.levels = nv, 3 * k, 1 + k % 2, self.converged, 1 + k % 3
        st.final_relres, st.true_relres, st.solve_ms, st.setup_ms, st.launches = k * 2.0 ** -40, k * 2.0 ** -41, \
            k * 0.25, k * 0.5, 7 * k

    def _call(self, name, args):
        if name == "pde_mesh_counts":
            dim, n = args[0], args[1]
            args[2]._obj.value = _nv(dim, n)
            args[3]._obj.value = int(np.prod([n[q] for q in range(dim)])) * CELLS_PER_BOX[dim]
            return 0
        if name == "pde_solver_opts_default":
            return 0
        if name.endswith("_local_nverts"):
            return self.nv[args[0].value]
        rec = [name] + [self._arg(a) for a in args]
        self.trace.append(rec)
        if name == "pde_ctx_create":
            self._handle(args[1], "ctx")
        elif name == "pde_host_alloc":
            buf = C.create_string_buffer(args[0].value)
            args[1]._obj.value = C.addressof(buf)
            self.pinned[C.addressof(buf)] = buf
        elif name == "pde_host_free":
            del self.pinned[args[0].value]
        elif name in ("pde_mesh_coords", "pde_mesh_coords_box"):
            dim, n = args[1], args[2]
            self._fill(args[-1], _nv(dim, n) * dim)
        elif name in ("pde_heat_solve", "pde_wheat_solve"):
            p = args[1]._obj
            nv = _nv(p.dim, p.n)
            nsnap = 1 if p.steady else 1 + p.num_steps // max(1, p.snapshot_stride)
            u0, values, times = (args[3], args[4], args[5]) if name == "pde_heat_solve" else (None, args[3], args[4])
            if u0:
                rec[4] = _doubles(u0, nv).tolist()
            self._fill(values, nsnap * nv)
            self._fill(times, nsnap, 1.0 / 64)
            self._stats(args[-1], nv)
        elif name.endswith("_open"):
            p = args[1]._obj
            self.nv[self._handle(args[3], "h%d" % len(self.names))] = _nv(p.dim, p.n)
        elif name.endswith("_set_state"):
            rec[2] = _doubles(args[1], self.nv[args[0].value]).tolist()
        elif name.endswith("_get_state"):
            self._fill(args[1], self.nv[args[0].value])
        elif name.endswith("_step"):
            self._stats(args[2], self.nv[args[0].value])
        return 0


# ------------------------------------------------------------------------------------------------------------ cases
PHYS = dict(diffusivity=0.75, T_initial=20.0, dt=0.125, num_steps=3, source_type="constant", source_value=3.0,
            initial_type="cosine", initial_amplitude=2.0)
RAW = {
    "1d": ("_solve_heat_1d_raw", dict(length=2.0, nx=4, T_left=5.0, T_right=1.0, initial_wavenumber=3.0), [4]),
    "2d": ("_solve_heat_2d_raw", dict(Lx=1.0, Ly=2.0, nx=2, ny=3, T_boundary=4.0, initial_wavenumber=3.0), [2, 3]),
    "3d": ("_solve_heat_3d_raw", dict(Lx=1.0, Ly=0.5, Lz=0.75, nx=2, ny=2, nz=3, T_boundary=4.0,
                                      initial_wavenumber=3.0), [2, 2, 3]),
    "1d_cylindrical": ("_solve_heat_1d_cylindrical_raw", dict(r_inner=0.25, r_outer=1.0, nr=4, T_inner=9.0,
                                                              T_outer=2.0), [4]),
    "1d_spherical": ("_solve_heat_1d_spherical_raw", dict(r_inner=0.0, r_outer=1.0, nr=4, T_inner=9.0,
                                                          T_outer=2.0), [4]),
    "2d_cylindrical": ("_solve_heat_2d_cylindrical_raw", dict(r_inner=0.25, r_outer=1.0, z_length=2.0, nr=2, nz=3,
                                                              T_boundary=6.0), [2, 3]),
    "2d_spherical": ("_solve_heat_2d_spherical_raw", dict(r_inner=0.25, r_outer=1.0, nr=2, ntheta=3,
                                                          T_boundary=6.0), [2, 3]),
    "3d_spherical": ("_solve_heat_3d_spherical_raw", dict(r_inner=0.0, r_outer=1.0, nr=2, ntheta=2, nphi=2,
                                                          T_boundary=6.0), [2, 2, 2]),
}
SPECIAL = {  # extra arguments of _solve_heat_3d_raw on the "3d" case; (ny, nz) = (2, 3) -> cylinder grid [2, 2, 2]
    "3d_directional": dict(T_left=7.0, T_right=1.0, T_side=3.0),
    "3d_left_only": dict(T_left=7.0, geometry_type="cylinder"),
    "3d_cylinder": dict(geometry_type="cylinder", cylinder_radius=0.5),
    "3d_cylinder_directional": dict(geometry_type="cylinder", cylinder_radius=0.5, T_left=7.0, T_side=3.0),
    "3d_core": dict(core_radius=0.25, core_diffusivity=8.0),
    "3d_core_directional": dict(core_radius=0.25, core_diffusivity=8.0, T_right=1.0, T_side=3.0),
    "3d_cylinder_core": dict(geometry_type="cylinder", cylinder_radius=0.5, core_radius=0.25, core_diffusivity=8.0),
}
MODES = {
    "plain": {}, "stride2": dict(snapshot_stride=2), "stream": dict(snapshot_stride=2, stream_to=True),
    "stream_stride1": dict(stream_to=True), "stream_u0": dict(u0=True, stream_to=True), "u0": dict(u0=True),
    "steady": dict(steady=True), "steady_u0": dict(steady=True, u0=True),
    "steady_stream": dict(steady=True, stream_to=True), "jacobi": dict(precond="jacobi"),
    "auto": dict(precond="auto"), "gmg": dict(precond="gmg"),
}
FEW_MODES = ("plain", "stream", "u0", "steady_u0", "gmg")     # for the variants of the cylinder / core branch
NOT_CONVERGED = {"3d_box_streaming": ("3d", "stream"), "2d_spherical_in_memory": ("2d_spherical", "plain"),
                 "2d_spherical_stepper": ("2d_spherical", "u0"), "3d_core_stepper": ("3d_core", "stream")}


def _cases():
    out = {}
    for geo in list(RAW) + list(SPECIAL):
        for mode in MODES if geo in RAW or geo in ("3d_cylinder", "3d_cylinder_core") else FEW_MODES:
            out[f"{geo}/{mode}"] = (geo, mode, 1)
    for name, (geo, mode) in NOT_CONVERGED.items():
        out[f"not_converged/{name}"] = (geo, mode, 0)
    return out


CASES = _cases()


def _grid(geo):
    if geo in SPECIAL:
        kw = dict(RAW["3d"][1], **SPECIAL[geo])
        return solvers.heat_3d_grid(kw["Lx"], kw["Ly"], kw["Lz"], kw["nx"], kw["ny"], kw["nz"],
                                    kw.get("geometry_type", "box"), kw.get("cylinder_radius"))[0]
    return RAW[geo][2]


def _install(monkeypatch, converged):
    fake = FakeLib(converged)
    monkeypatch.setattr(_lib, "_lib", fake)
    monkeypatch.setattr(_lib, "_ctx", None)
    monkeypatch.delenv("PDE_B200_GPUS", raising=False)
    return fake


def _run_case(name, monkeypatch, tmp_path):
    geo, mode, converged = CASES[name]
    fake = _install(monkeypatch, converged)
    fn, kw, _ = RAW["3d" if geo in SPECIAL else geo]
    kw = dict(kw, **SPECIAL.get(geo, {}), **PHYS, **MODES[mode])
    n = _grid(geo)
    if kw.get("u0"):
        kw["u0"] = 7.0 + 0.5 * np.arange(_nv(len(n), n))
    writer = None
    if kw.get("stream_to"):
        writer = kw["stream_to"] = io.open_writer("npz", tmp_path / "s.npz", len(n), n, [1.0] * len(n))
    out = {}
    try:
        f = getattr(solvers, fn)(**kw)
        out.update(coords=np.asarray(f.coords).tolist(), values=np.asarray(f.values).tolist(),
                   times=np.asarray(f.times).tolist(), meta=f.meta)
    except _lib.PdeError as e:
        out["error"] = str(e)
    if writer is not None:
        writer.close()
        with np.load(tmp_path / "s.npz") as z:
            t = z["times"].tolist()
            out["writer"] = {"times": t, "values": [z[f"t{k:06d}"].tolist() for k in range(len(t))]}
    out.update(stats=solvers.last_stats(), trace=fake.trace)
    return out


def _run_stepper(monkeypatch):
    """HeatStepper as bench.py builds and drives it."""
    fake = _install(monkeypatch, 1)
    ctx = _lib.default_context()
    n = [2, 2, 3]
    bc = _lib.make_bc({f: 4.0 for f in range(6)})
    hs = _lib.HeatStepper(ctx, 3, n, [1.0, 1.0, 1.0], 0.75, 0.125, T_initial=20.0, bc=bc,
                          opts=_lib.make_opts(rtol=1e-9, precond="gmg"))
    st = hs.step(2)
    hs.set_state(np.arange(hs.nloc, dtype=np.float64))
    state = hs.get_state(np.empty(hs.nloc)).tolist()
    hs.close()
    return {"nloc": hs.nloc, "step": st, "state": state, "trace": fake.trace}


def _summary(rec):
    """What the golden file keeps of a run: 64 bits of the SHA-256 of everything but the coordinates, and three
    weighted sums of the coordinates, which pass through sin / cos, whose last bit may differ between CPUs."""
    rec = json.loads(json.dumps(rec))
    x = np.asarray(rec.pop("coords", []), dtype=float).ravel()
    w = np.arange(1.0, x.size + 1)
    return {"sha256": hashlib.sha256(json.dumps(rec, sort_keys=True, separators=(",", ":")).encode()).hexdigest()[:16],
            "coords": [float(x.sum()), float(x @ w), float(x @ w ** 2)]}


def _check(rec, want):
    got = _summary(rec)
    assert got["sha256"] == want["sha256"], ("calls or results differ", [c[0] for c in rec["trace"]],
                                             rec.get("stats"), rec.get("error"))
    assert np.allclose(got["coords"], want["coords"], rtol=1e-12, atol=1e-9), (got["coords"], want["coords"])


@functools.lru_cache(maxsize=None)
def _golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


@pytest.mark.parametrize("name", sorted(CASES))
def test_heat_call_matches_golden(name, monkeypatch, tmp_path):
    rec = _run_case(name, monkeypatch, tmp_path)
    _check(rec, _golden()["cases"][name])
    if CASES[name][2] == 0:
        assert "did not converge" in rec["error"]


def test_heat_stepper_matches_golden(monkeypatch):
    _check(_run_stepper(monkeypatch), _golden()["heat_stepper"])


def _record_golden():
    import tempfile
    mp = pytest.MonkeyPatch()
    cases = {}
    with tempfile.TemporaryDirectory() as d:
        for k in sorted(CASES):
            os.makedirs(os.path.join(d, k))
            cases[k] = _summary(_run_case(k, mp, Path(d, k)))
            mp.undo()
    stepper = _summary(_run_stepper(mp))
    mp.undo()
    with open(GOLDEN, "w") as fh:       # one case per line
        fh.write('{"heat_stepper": ' + json.dumps(stepper) + ',\n"cases": {\n' +
                 ",\n".join(json.dumps(k) + ": " + json.dumps(v) for k, v in cases.items()) + "}}\n")
    print(f"wrote {GOLDEN}: {len(cases)} cases")


if __name__ == "__main__":
    _record_golden()
