"""Host-side mirror of the reference's raw solvers (same names, arguments and result type).

Reference: /root/reference/fenics_mcp_server.py
  _solve_heat_1d_raw :204-338      _solve_heat_2d_raw :345-468      _solve_heat_3d_raw :475-762
  _solve_elasticity_1d_static :1470-1587   _2d_ :1593-1743   _3d_ :1749-1892
Each function only marshals arguments into the C ABI (include/pde_b200.h) and wraps the result;
all arithmetic runs in hand-written CUDA.  Extra keyword-only arguments (rtol, precond,
snapshot_stride, as_arrays, u0, stream_to) are additions the reference does not have; their defaults reproduce
the reference's behaviour."""
import ctypes as C
import os
from typing import Optional

import numpy as np

from . import _lib, mesh, multi
from .fields import TimeSeriesField

# above this many stored values the result keeps NumPy arrays instead of nested Python lists
LIST_LIMIT = int(os.environ.get("PDE_B200_LIST_LIMIT", "4000000"))

_last_stats = {}


def last_stats():
    """Solver statistics (iterations, residuals, device time, launches) of the most recent call."""
    return dict(_last_stats)


def _record(stats, what, **extra):
    """Publish the statistics of a finished solve and refuse to hand out an unconverged field: the reference
    solves with sparse LU (fenics_mcp_server.py:265, 1838), so a PCG that stopped at max_iters is an error here."""
    _last_stats.clear()
    _last_stats.update(stats)
    _last_stats.update(extra)
    bad = [k for k, d in (("solve", stats), *extra.items()) if isinstance(d, dict) and not d.get("converged", 1)]
    if bad:
        d = stats if "solve" in bad else extra[bad[0]]
        raise _lib.PdeError(f"{what}: PCG did not converge ({', '.join(bad)}; {d.get('iters_total')} iterations, "
                            f"relative residual {d.get('final_relres'):.3e})")


def _embed3(coords, dim):
    out = np.zeros((coords.shape[0], 3), dtype=np.float64)
    out[:, :dim] = coords
    return out


def _finish(coords3, values, times, dim, meta, as_arrays, n=None):
    if n is not None and mesh.dof_permutation(dim, n) is not None:
        # plugged dof numbering (mesh.set_dof_permutation): coordinates and values leave in that order, paired exactly
        # as the reference pairs tabulate_dof_coordinates() with get_local()
        coords3 = mesh.to_dof_order(dim, n, coords3, axis=0)
        values = mesh.to_dof_order(dim, n, values, axis=-1)
    if as_arrays is None:
        as_arrays = values.size > LIST_LIMIT
    if as_arrays:
        return TimeSeriesField(coords=coords3, values=values, times=np.asarray(times), dim=dim, meta=meta)
    return TimeSeriesField(coords=coords3.tolist(), values=values.tolist(), times=[float(t) for t in times],
                           dim=dim, meta=meta)


def _heat(dim, L, n, diffusivity, T_initial, dt, num_steps, steady, source_type, source_value, initial_type,
          initial_amplitude, initial_wavenumber, bc, rtol, precond, snapshot_stride, u0=None, ctx=None, stream_to=None):
    """stream_to: an io.*SnapshotWriter.  Snapshots then go to the writer one at a time (device-resident
    stepper, one pinned host buffer) and only the first and last are returned."""
    ctx = ctx or _lib.default_context()
    p = _lib.heat_params(dim, n, L, diffusivity, dt, T_initial=T_initial, bc=bc,
                         source_value=source_value if source_type == "constant" else 0.0, steady=steady,
                         num_steps=num_steps, snapshot_stride=snapshot_stride,
                         initial_type="array" if u0 is not None else initial_type,
                         initial_amplitude=initial_amplitude, initial_wavenumber=initial_wavenumber)
    nv, _ = _lib.mesh_counts(dim, n)
    o = _lib.make_opts(rtol=rtol, precond=precond)
    u0a = np.ascontiguousarray(u0, dtype=np.float64) if u0 is not None else None
    if stream_to is not None and not steady:
        values, times = _run_stepper(_lib.Stepper("heat", ctx, p, o), p, u0a, stream_to, "heat solve")
        return mesh.coordinates(dim, n, L, ctx), values, times
    if dim == 3 and u0 is None and multi.usable(int(n[2])):
        # PDE_B200_GPUS=N: the same call on N z-slabs, one worker process per GPU (multi.py)
        stats, values, times = multi.heat_solve(p, o, _nsnap(p), nv)
        _record(stats, "heat solve")
    else:
        values, times = _solve_in_memory(_lib.lib().pde_heat_solve, ctx, p, o, nv, "heat solve", _lib.ptr(u0a))
    return mesh.coordinates(dim, n, L, ctx), values, times


def _nsnap(p):
    return 1 if p.steady else 1 + int(p.num_steps) // max(1, int(p.snapshot_stride))


def _solve_in_memory(fn, ctx, p, o, nv, what, *u0):
    """(values, times) of one pde_heat_solve / pde_wheat_solve call, every kept snapshot in host memory."""
    values = np.empty((_nsnap(p), nv), dtype=np.float64)
    times = np.empty(_nsnap(p), dtype=np.float64)
    st = _lib.Stats()
    _lib.check(fn(ctx.handle, C.byref(p), C.byref(o), *u0, _lib.ptr(values), _lib.ptr(times), C.byref(st)))
    _record(st.as_dict(), what)
    return values, times


def _run_stepper(stepper, p, u0, writer, what):
    """(values, times) of the solve p on a resident stepper, which it closes.  u0 (natural vertex order) replaces
    the initial field.  A transient run keeps the state at t = 0 and after every snapshot_stride-th step: with a
    writer every kept state goes through one pinned buffer to the writer and only the first and last are returned
    (host memory use is one snapshot); without one every kept state is returned.  A steady run (never with a writer)
    takes its one solve, u0 being the starting guess, and keeps the result at t = 0."""
    steady, stride = bool(p.steady), max(1, int(p.snapshot_stride))
    acc = {"iters_total": 0, "solves": 0, "converged": 1, "solve_ms": 0.0, "launches": 0}
    kept, times, buf = [], [], None

    def keep(t):
        out = buf.array if buf is not None else np.empty(stepper.nloc, dtype=np.float64)
        stepper.get_state(out)
        times.append(t)
        if writer is not None:
            writer.append(t, out)
        kept.append(out.copy() if writer is not None and not kept else out)

    try:
        if writer is not None:
            buf = _lib.PinnedArray(stepper.nloc)
        if u0 is not None:
            stepper.set_state(u0)
        if not steady:
            keep(0.0)
        for step in range(1 if steady else int(p.num_steps)):
            d = stepper.step(1)
            for k in ("iters_total", "solves", "solve_ms", "launches"):
                acc[k] += d[k]
            acc["converged"] &= d["converged"]
            acc.update({k: d[k] for k in ("ndofs", "levels", "final_relres", "setup_ms", "true_relres")})
            if steady or (step + 1) % stride == 0:
                keep(0.0 if steady else (step + 1) * p.dt)
        if writer is not None:      # the first kept state and the pinned buffer, which holds the last
            kept, times = [kept[0], kept[-1].copy()], [times[0], times[-1]]
    finally:
        stepper.close()
        if buf is not None:
            buf.free()
    _record(acc, what + (" (streaming)" if writer is not None else ""))
    return np.stack(kept), np.array(times)


def _solve_heat_1d_raw(length: float, nx: int, diffusivity: float, T_left: float, T_right: float,
                       T_initial: float, dt: float, num_steps: int, steady: bool = False,
                       source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                       initial_amplitude: float = 1.0, initial_wavenumber: float = 1.0, *, rtol: float = 1e-10,
                       precond: str = "auto", snapshot_stride: int = 1, as_arrays: Optional[bool] = None,
                       u0=None, stream_to=None) -> TimeSeriesField:
    """1D heat equation on [0, length], Dirichlet T_left / T_right, backward Euler or steady."""
    bc = mesh.heat_bc(1, T_left=T_left, T_right=T_right)
    coords, values, times = _heat(1, [length], [nx], diffusivity, T_initial, dt, num_steps, steady, source_type,
                                  source_value, initial_type, initial_amplitude, initial_wavenumber, bc, rtol,
                                  precond, snapshot_stride, u0, stream_to=stream_to)
    # the reference sorts dofs by x (:252-254); natural order is already sorted
    order = np.argsort(coords[:, 0], kind="stable")
    meta = {"name": "temperature", "unit": "°C", "pde": "heat", "coordinate_system": "cartesian",
            "length": length, "source_type": source_type, "source_value": source_value, "steady": steady}
    return _finish(_embed3(coords[order], 1), values[:, order], times, 1, meta, as_arrays)


def _solve_heat_2d_raw(Lx: float, Ly: float, nx: int, ny: int, diffusivity: float, T_boundary: float,
                       T_initial: float, dt: float, num_steps: int, steady: bool = False,
                       source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                       initial_amplitude: float = 1.0, initial_wavenumber: float = 1.0, *, rtol: float = 1e-10,
                       precond: str = "auto", snapshot_stride: int = 1, as_arrays: Optional[bool] = None,
                       u0=None, stream_to=None) -> TimeSeriesField:
    """2D heat equation on [0,Lx]x[0,Ly], constant Dirichlet value on the whole boundary."""
    bc = mesh.heat_bc(2, T_boundary=T_boundary)
    coords, values, times = _heat(2, [Lx, Ly], [nx, ny], diffusivity, T_initial, dt, num_steps, steady,
                                  source_type, source_value, initial_type, initial_amplitude, initial_wavenumber,
                                  bc, rtol, precond, snapshot_stride, u0, stream_to=stream_to)
    meta = {"name": "temperature", "unit": "°C", "pde": "heat", "coordinate_system": "cartesian", "Lx": Lx,
            "Ly": Ly, "source_type": source_type, "source_value": source_value, "steady": steady}
    return _finish(_embed3(coords, 2), values, times, 2, meta, as_arrays, n=[nx, ny])


def _solve_heat_3d_raw(Lx: float, Ly: float, Lz: float, nx: int, ny: int, nz: int, diffusivity: float,
                       T_boundary: float, T_initial: float, dt: float, num_steps: int, steady: bool = False,
                       source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                       initial_amplitude: float = 1.0, initial_wavenumber: float = 1.0,
                       geometry_type: str = "box", cylinder_radius: Optional[float] = None,
                       T_left: Optional[float] = None, T_right: Optional[float] = None,
                       T_side: Optional[float] = None, core_radius: Optional[float] = None,
                       core_diffusivity: Optional[float] = None, *, rtol: float = 1e-10, precond: str = "auto",
                       snapshot_stride: int = 1, as_arrays: Optional[bool] = None, u0=None,
                       stream_to=None) -> TimeSeriesField:
    """3D heat equation on the box [0,Lx]x[0,Ly]x[0,Lz]; uniform or directional Dirichlet values."""
    cyl = geometry_type == "cylinder" and cylinder_radius is not None
    core = (core_radius, core_diffusivity) if core_radius is not None and core_diffusivity is not None else None
    special = cyl or core is not None
    directional = T_left is not None or T_right is not None or T_side is not None
    if special and directional and geometry_type == "cylinder":
        # side_boundary_cylinder (:594-598) asks for near(r, R) on boundary facets away from the x ends; on the
        # BoxMesh no facet has all vertices and its midpoint at r == R, so DOLFIN's topological search finds none
        # and T_side constrains nothing; left / right are the x-end faces
        bc = _lib.make_bc({f: v for f, v in ((0, T_left), (1, T_right)) if v is not None})
    else:
        bc = mesh.heat_bc(3, T_boundary=T_boundary, T_left=T_left, T_right=T_right, T_side=T_side)
    if special:
        coords, values, times = _heat_3d_special(
            Lx=Lx, Ly=Ly, Lz=Lz, nx=nx, ny=ny, nz=nz, geometry_type=geometry_type, cylinder_radius=cylinder_radius,
            cyl=cyl, core=core, bc=bc, diffusivity=diffusivity, T_initial=T_initial, dt=dt, num_steps=num_steps,
            steady=steady, source_type=source_type, source_value=source_value, initial_type=initial_type,
            initial_amplitude=initial_amplitude, initial_wavenumber=initial_wavenumber, rtol=rtol, precond=precond,
            snapshot_stride=snapshot_stride, u0=u0, stream_to=stream_to)
    else:
        coords, values, times = _heat(3, [Lx, Ly, Lz], [nx, ny, nz], diffusivity, T_initial, dt, num_steps, steady,
                                      source_type, source_value, initial_type, initial_amplitude, initial_wavenumber,
                                      bc, rtol, precond, snapshot_stride, u0, stream_to=stream_to)
    box = geometry_type == "box"
    # the cylinder / core branch reports the cylinder's diameter as Ly and Lz whenever a radius is given
    D = cylinder_radius * 2 if special and not box and cylinder_radius else None
    meta = {"name": "temperature", "unit": "°C", "pde": "heat",
            "coordinate_system": "cartesian" if box else "cylindrical", "Lx": Lx, "Ly": Ly if D is None else D,
            "Lz": Lz if D is None else D, "geometry_type": geometry_type, "source_type": source_type,
            "source_value": source_value, "steady": steady}
    if cyl:
        meta["cylinder_radius"] = cylinder_radius
    if directional:
        meta.update({k: v for k, v in (("T_left", T_left), ("T_right", T_right), ("T_side", T_side)) if v is not None})
    else:
        meta["T_boundary"] = T_boundary
    if core is not None:
        meta.update(core_radius=core_radius, core_diffusivity=core_diffusivity, base_diffusivity=diffusivity)
    else:
        meta["diffusivity"] = diffusivity
    return _finish(coords, values, times, 3, meta, as_arrays, n=None if special else [nx, ny, nz])


def heat_3d_grid(Lx, Ly, Lz, nx, ny, nz, geometry_type="box", cylinder_radius=None):
    """(n, lo, hi) of the mesh a _solve_heat_3d_raw call builds: the cylinder is BoxMesh((0,-R,-R), (Lx,R,R), nx,
    int(ny*2R), int(nz*2R)) (the reference without mshr), every other geometry the box [0,Lx]x[0,Ly]x[0,Lz]."""
    if geometry_type == "cylinder" and cylinder_radius is not None:
        R = float(cylinder_radius)
        return [int(nx), int(ny * R * 2), int(nz * R * 2)], [0.0, -R, -R], [float(Lx), R, R]
    return [int(nx), int(ny), int(nz)], [0.0, 0.0, 0.0], [float(Lx), float(Ly), float(Lz)]


def _heat_3d_special(*, Lx, Ly, Lz, nx, ny, nz, geometry_type, cylinder_radius, cyl, core, bc, diffusivity, T_initial,
                     dt, num_steps, steady, source_type, source_value, initial_type, initial_amplitude,
                     initial_wavenumber, rtol, precond, snapshot_stride, u0, stream_to):
    """Cylinder / composite-core branches of _solve_heat_3d_raw (:512-572, 576-605, 642-645) as the reference's
    deployment runs them (no mshr in Dockerfile / requirements.txt, so MSHR_AVAILABLE is False): the "cylinder" is
    BoxMesh((0,-R,-R),(Lx,R,R), nx, int(ny*2R), int(nz*2R)) with every term weighted by
    Expression("sqrt(x[1]^2+x[2]^2)", degree=2); the core is a DG0 diffusivity marked by SubDomain.mark.
    core: (radius, diffusivity) or None.  Returns (coords, values, times)."""
    n, lo, hi = heat_3d_grid(Lx, Ly, Lz, nx, ny, nz, geometry_type, cylinder_radius)
    if min(n) < 1:
        raise ValueError(f"BoxMesh needs at least one cell per axis, got {n}")
    p = _wheat_params(3, n, lo, hi, bc, diffusivity, T_initial, dt, num_steps, steady, source_type, source_value,
                      snapshot_stride, weight=(0, 0, 2 if cyl else 1), weight_kind=1 if cyl else 0, core=core,
                      initial_type=initial_type, initial_amplitude=initial_amplitude,
                      initial_wavenumber=initial_wavenumber)
    values, times = _wheat(p, rtol, precond, u0, stream_to, "heat solve (weighted box)")
    return mesh.coordinates_box(3, n, lo, hi), values, times


def _wheat_params(dim, n, lo, hi, bc, diffusivity, T_initial, dt, num_steps, steady, source_type, source_value,
                  snapshot_stride, weight=(0, 0, 1), weight_kind=0, core=None, initial_type="constant",
                  initial_amplitude=0.0, initial_wavenumber=0.0):
    """WheatParams (pde_wheat_params).  weight: (r-power, sin(x1) factor, Expression degree) of a curvilinear
    weight; weight_kind 1 is the cylinder's sqrt(x1^2 + x2^2); core: (radius, diffusivity) of a DG0 core or None."""
    p = _lib.WheatParams()
    p.dim = dim
    p.n = _lib.i3(n)
    p.lo = _lib.d3(lo, 0.0)
    p.hi = _lib.d3(hi, 1.0)
    p.weight_rpow, p.weight_sin_axis1, p.weight_degree = weight
    p.weight_kind = weight_kind
    p.has_core = 1 if core is not None else 0
    p.core_radius, p.core_diffusivity = (float(core[0]), float(core[1])) if core is not None else (0.0, 0.0)
    p.steady = 1 if steady else 0
    p.diffusivity = float(diffusivity)
    p.dt = float(dt)
    p.num_steps = int(num_steps)
    p.snapshot_stride = int(snapshot_stride)
    p.source_value = float(source_value) if source_type == "constant" else 0.0
    p.T_initial = float(T_initial)
    p.initial_type = _lib.IC.get(initial_type, _lib.IC["constant"])
    p.initial_amplitude = float(initial_amplitude)
    p.initial_wavenumber = float(initial_wavenumber)
    p.bc = bc
    return p


def _elasticity(dim, L, n, E, nu, body, quantity, plane_stress=True, area=1.0, rtol=1e-10, precond="auto",
                want_displacement=False, ctx=None):
    ctx = ctx or _lib.default_context()
    p = _lib.ElastParams()
    p.dim = dim
    p.n = _lib.i3(n)
    p.L = _lib.d3(L)
    p.E = float(E)
    p.nu = float(nu)
    p.body = _lib.d3(body, 0.0)
    p.quantity = 1 if quantity == "strain" else 0
    p.plane_stress = 1 if plane_stress else 0
    p.area = float(area)
    nv, _ = _lib.mesh_counts(dim, n)
    o = _lib.make_opts(rtol=rtol, precond=precond)
    if dim == 3 and multi.usable(int(n[2])):
        stats, pstats, out, disp = multi.elasticity_solve(p, o, nv, want_displacement)
        _record(stats, "elasticity solve", projection=pstats)
        return mesh.coordinates(dim, n, L, ctx), out, disp
    out = np.empty(nv, dtype=np.float64)
    disp = np.empty((nv, dim), dtype=np.float64) if want_displacement else None
    st, sp = _lib.Stats(), _lib.Stats()
    _lib.check(_lib.lib().pde_elasticity_solve(ctx.handle, C.byref(p), C.byref(o), _lib.ptr(out), _lib.ptr(disp),
                                               C.byref(st), C.byref(sp)))
    _record(st.as_dict(), "elasticity solve", projection=sp.as_dict())
    coords = mesh.coordinates(dim, n, L, ctx)
    return coords, out, disp


def _solve_elasticity_1d_static(L: float, nx: int, E: float, area: float, body_force: float,
                                quantity: str = "stress", *, rtol: float = 1e-10, precond: str = "auto",
                                as_arrays: Optional[bool] = None) -> TimeSeriesField:
    """Axial bar -(EA u')' = body_force, u(0) = 0; output the projected axial stress or strain."""
    coords, val, _ = _elasticity(1, [L], [nx], E, 0.0, [body_force], quantity, area=area, rtol=rtol,
                                 precond=precond)
    order = np.argsort(coords[:, 0], kind="stable")
    if quantity == "strain":
        name, unit = "axial_strain", "-"
    else:
        name, unit = "axial_stress", "Pa"
    meta = {"name": name, "unit": unit, "pde": "elasticity_1d", "L": L, "E": E, "area": area,
            "body_force": body_force, "quantity": quantity}
    return _finish(_embed3(coords[order], 1), val[order][None, :], [0.0], 1, meta, as_arrays)


def _solve_elasticity_2d_static(Lx: float, Ly: float, nx: int, ny: int, E: float, nu: float, body_fx: float = 0.0,
                                body_fy: float = 0.0, quantity: str = "stress", plane_stress: bool = True, *,
                                rtol: float = 1e-10, precond: str = "auto",
                                as_arrays: Optional[bool] = None) -> TimeSeriesField:
    """Plane stress/strain static elasticity clamped at x = 0; projected von Mises stress or strain."""
    coords, val, _ = _elasticity(2, [Lx, Ly], [nx, ny], E, nu, [body_fx, body_fy], quantity,
                                 plane_stress=plane_stress, rtol=rtol, precond=precond)
    name, unit = ("von_mises_strain", "-") if quantity == "strain" else ("von_mises_stress", "Pa")
    meta = {"name": name, "unit": unit, "pde": "elasticity_2d", "Lx": Lx, "Ly": Ly, "E": E, "nu": nu,
            "body_fx": body_fx, "body_fy": body_fy, "quantity": quantity, "plane_stress": plane_stress}
    return _finish(_embed3(coords, 2), val[None, :], [0.0], 2, meta, as_arrays, n=[nx, ny])


def _solve_elasticity_3d_static(Lx: float, Ly: float, Lz: float, nx: int, ny: int, nz: int, E: float, nu: float,
                                body_fx: float = 0.0, body_fy: float = 0.0, body_fz: float = 0.0,
                                quantity: str = "stress", *, rtol: float = 1e-10, precond: str = "auto",
                                as_arrays: Optional[bool] = None) -> TimeSeriesField:
    """3D static elasticity on a box clamped at x = 0; projected von Mises stress or strain."""
    coords, val, _ = _elasticity(3, [Lx, Ly, Lz], [nx, ny, nz], E, nu, [body_fx, body_fy, body_fz], quantity,
                                 rtol=rtol, precond=precond)
    name, unit = ("von_mises_strain", "-") if quantity == "strain" else ("von_mises_stress", "Pa")
    meta = {"name": name, "unit": unit, "pde": "elasticity_3d", "Lx": Lx, "Ly": Ly, "Lz": Lz, "E": E, "nu": nu,
            "body_fx": body_fx, "body_fy": body_fy, "body_fz": body_fz, "quantity": quantity}
    return _finish(coords, val[None, :], [0.0], 3, meta, as_arrays, n=[nx, ny, nz])


# ----------------------------------------------------------------------------------------------------------
# Curvilinear heat tools (reference :769-1464): the same loop on the coordinate-space mesh with one scalar weight
# ----------------------------------------------------------------------------------------------------------
def _cylindrical_rz(X):
    coords = np.zeros((X.shape[0], 3))
    coords[:, 0], coords[:, 2] = X[:, 0], X[:, 1]                 # (r, 0, z)
    return coords


def _spherical_xyz(X):
    coords = np.zeros((X.shape[0], 3))
    if X.shape[1] == 2:                                           # phi = 0: (r sin(theta), 0, r cos(theta))
        coords[:, 0] = X[:, 0] * np.sin(X[:, 1])
    else:
        coords[:, 0] = X[:, 0] * np.sin(X[:, 1]) * np.cos(X[:, 2])
        coords[:, 1] = X[:, 0] * np.sin(X[:, 1]) * np.sin(X[:, 2])
    coords[:, 2] = X[:, 0] * np.cos(X[:, 1])
    return coords


_CURVI = {
    # kind: (dim, weight r-power, sin(x1) factor, weight Expression degree, coordinate system, geometry_type without
    #        and with an inner radius, map of the coordinate-space vertices to (x, y, z))
    "1d_cylindrical": (1, 1, 0, 1, "cylindrical", "cylinder", "annulus", lambda X: _embed3(X, 1)),
    "1d_spherical": (1, 2, 0, 2, "spherical", "sphere", "spherical_shell", lambda X: _embed3(X, 1)),
    "2d_cylindrical": (2, 1, 0, 1, "cylindrical", "cylinder", "annular_cylinder", _cylindrical_rz),
    "2d_spherical": (2, 2, 1, 2, "spherical", "sphere", "spherical_shell", _spherical_xyz),
    "3d_spherical": (3, 2, 1, 2, "spherical", "sphere", "spherical_shell", _spherical_xyz),
}


def curvilinear_grid(kind, r_inner, r_outer, n, z_length=None):
    """(n, lo, hi) of the coordinate-space mesh of a curvilinear tool: IntervalMesh(nr, r_inner, r_outer),
    RectangleMesh to (r_outer, z_length) / (r_outer, pi), BoxMesh to (r_outer, pi, 2 pi)."""
    rest = {"2d_cylindrical": [z_length], "2d_spherical": [float(np.pi)],
            "3d_spherical": [float(np.pi), float(2.0 * np.pi)]}.get(kind, [])
    return [int(k) for k in n], [r_inner] + [0.0] * len(rest), [r_outer] + rest


def _wheat(p, rtol, precond, u0, writer, what):
    """(values, times) of the weighted solve p.  A plain call is one pde_wheat_solve.  With a host initial field u0
    (natural vertex order) or a snapshot writer it runs on the resident stepper (_run_stepper).  Steady solves never
    stream; u0 is their starting guess."""
    nv = int(np.prod([int(p.n[q]) + 1 for q in range(int(p.dim))]))
    if u0 is not None:
        u0 = np.ascontiguousarray(u0, dtype=np.float64)
        if u0.shape != (nv,):
            raise ValueError(f"u0 must hold one value per mesh vertex ({nv}), got shape {u0.shape}")
    ctx = _lib.default_context()
    if p.steady:
        writer = None
    if precond not in _lib.PRECOND:
        raise ValueError(f"precond must be one of {sorted(_lib.PRECOND)}, got {precond!r}")
    # "gmg" selects Galerkin multigrid; "auto" still means Jacobi-PCG for the weighted operators
    o = _lib.make_opts(rtol=rtol, precond="gmg" if precond == "gmg" else "jacobi")
    if u0 is not None or writer is not None:
        return _run_stepper(_lib.WheatStepper(ctx, p, o), p, u0, writer, what)
    return _solve_in_memory(_lib.lib().pde_wheat_solve, ctx, p, o, nv, what)


def _curvilinear(kind, r_inner, r_outer, n, bc, diffusivity, T_initial, dt, num_steps, steady, source_type,
                 source_value, *, rtol, precond, snapshot_stride, as_arrays, u0, stream_to, z_length=None):
    """One curvilinear tool: the weighted solve on the coordinate-space mesh of curvilinear_grid, its vertices mapped
    to (x, y, z); the 1-D tools sort the vertices by r as the reference does."""
    dim, rpow, wsin, wdeg, system, solid, hollow, to_xyz = _CURVI[kind]
    n, lo, hi = curvilinear_grid(kind, r_inner, r_outer, n, z_length)
    p = _wheat_params(dim, n, lo, hi, bc, diffusivity, T_initial, dt, num_steps, steady, source_type, source_value,
                      snapshot_stride, weight=(rpow, wsin, wdeg))
    values, times = _wheat(p, rtol, precond, u0, stream_to, "curvilinear heat solve")
    X = mesh.coordinates_box(dim, n, lo, hi)
    if dim == 1:
        order = np.argsort(X[:, 0], kind="stable")
        X, values = X[order], values[:, order]
    meta = {"name": "temperature", "unit": "°C", "pde": "heat", "coordinate_system": system,
            "geometry_type": solid if r_inner < 1e-10 else hollow, "r_inner": r_inner, "r_outer": r_outer}
    if z_length is not None:
        meta["z_length"] = z_length
    meta.update({"source_type": source_type, "source_value": source_value, "steady": steady})
    return _finish(to_xyz(X), values, times, dim, meta, as_arrays)


def _radial_bc(r_inner, T_inner, T_outer):
    faces = {1: T_outer}
    if r_inner > 1e-10:          # the inner condition is only imposed on an annulus / shell (:811-815, 967-972)
        faces[0] = T_inner
    return _lib.make_bc(faces)


def _solve_heat_1d_cylindrical_raw(r_inner: float, r_outer: float, nr: int, diffusivity: float, T_inner: float,
                                   T_outer: float, T_initial: float, dt: float, num_steps: int, steady: bool = False,
                                   source_type: str = "none", source_value: float = 0.0,
                                   initial_type: str = "constant", initial_amplitude: float = 1.0, *,
                                   rtol: float = 1e-10, precond: str = "jacobi", snapshot_stride: int = 1,
                                   as_arrays: Optional[bool] = None, u0=None, stream_to=None) -> TimeSeriesField:
    """1D radial heat equation in cylindrical coordinates, weight r (:769-920)."""
    return _curvilinear("1d_cylindrical", r_inner, r_outer, [nr], _radial_bc(r_inner, T_inner, T_outer), diffusivity,
                        T_initial, dt, num_steps, steady, source_type, source_value, rtol=rtol, precond=precond,
                        snapshot_stride=snapshot_stride, as_arrays=as_arrays, u0=u0, stream_to=stream_to)


def _solve_heat_1d_spherical_raw(r_inner: float, r_outer: float, nr: int, diffusivity: float, T_inner: float,
                                 T_outer: float, T_initial: float, dt: float, num_steps: int, steady: bool = False,
                                 source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                                 initial_amplitude: float = 1.0, *, rtol: float = 1e-10, precond: str = "jacobi",
                                 snapshot_stride: int = 1, as_arrays: Optional[bool] = None, u0=None,
                                 stream_to=None) -> TimeSeriesField:
    """1D radial heat equation in spherical coordinates, weight r^2 (:926-1057)."""
    return _curvilinear("1d_spherical", r_inner, r_outer, [nr], _radial_bc(r_inner, T_inner, T_outer), diffusivity,
                        T_initial, dt, num_steps, steady, source_type, source_value, rtol=rtol, precond=precond,
                        snapshot_stride=snapshot_stride, as_arrays=as_arrays, u0=u0, stream_to=stream_to)


def _solve_heat_2d_cylindrical_raw(r_inner: float, r_outer: float, z_length: float, nr: int, nz: int,
                                   diffusivity: float, T_boundary: float, T_initial: float, dt: float, num_steps: int,
                                   steady: bool = False, source_type: str = "none", source_value: float = 0.0,
                                   initial_type: str = "constant", initial_amplitude: float = 1.0, *,
                                   rtol: float = 1e-10, precond: str = "jacobi", snapshot_stride: int = 1,
                                   as_arrays: Optional[bool] = None, u0=None, stream_to=None) -> TimeSeriesField:
    """2D axisymmetric heat equation in the (r, z) plane, weight r (:1063-1185)."""
    return _curvilinear("2d_cylindrical", r_inner, r_outer, [nr, nz], _lib.make_bc({f: T_boundary for f in range(4)}),
                        diffusivity, T_initial, dt, num_steps, steady, source_type, source_value, rtol=rtol,
                        precond=precond, snapshot_stride=snapshot_stride, as_arrays=as_arrays, u0=u0,
                        stream_to=stream_to, z_length=z_length)


def _solve_heat_2d_spherical_raw(r_inner: float, r_outer: float, nr: int, ntheta: int, diffusivity: float,
                                 T_boundary: float, T_initial: float, dt: float, num_steps: int, steady: bool = False,
                                 source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                                 initial_amplitude: float = 1.0, *, rtol: float = 1e-10, precond: str = "jacobi",
                                 snapshot_stride: int = 1, as_arrays: Optional[bool] = None, u0=None,
                                 stream_to=None) -> TimeSeriesField:
    """2D axisymmetric heat equation in the (r, theta) plane, weight r^2 sin(theta) (:1191-1320)."""
    return _curvilinear("2d_spherical", r_inner, r_outer, [nr, ntheta], _lib.make_bc({f: T_boundary for f in range(4)}),
                        diffusivity, T_initial, dt, num_steps, steady, source_type, source_value, rtol=rtol,
                        precond=precond, snapshot_stride=snapshot_stride, as_arrays=as_arrays, u0=u0,
                        stream_to=stream_to)


def _solve_heat_3d_spherical_raw(r_inner: float, r_outer: float, nr: int, ntheta: int, nphi: int, diffusivity: float,
                                 T_boundary: float, T_initial: float, dt: float, num_steps: int, steady: bool = False,
                                 source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
                                 initial_amplitude: float = 1.0, *, rtol: float = 1e-10, precond: str = "jacobi",
                                 snapshot_stride: int = 1, as_arrays: Optional[bool] = None, u0=None,
                                 stream_to=None) -> TimeSeriesField:
    """3D heat equation in (r, theta, phi), weight r^2 sin(theta) (:1326-1464)."""
    return _curvilinear("3d_spherical", r_inner, r_outer, [nr, ntheta, nphi],
                        _lib.make_bc({f: T_boundary for f in range(6)}), diffusivity, T_initial, dt, num_steps, steady,
                        source_type, source_value, rtol=rtol, precond=precond, snapshot_stride=snapshot_stride,
                        as_arrays=as_arrays, u0=u0, stream_to=stream_to)
