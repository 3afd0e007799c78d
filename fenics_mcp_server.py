#!/usr/bin/env python
"""Drop-in MCP tool server: same file name, server name, tool names, keyword arguments, defaults and
result types as the reference's `fenics_mcp_server.py`, with the structured-mesh P1 heat and
linear-elasticity solves running on hand-written sm_100a CUDA (libpde_b200.so) instead of
FEniCS/PETSc.

Reference boundary (file:line under /root/reference/fenics_mcp_server.py):
  FastMCP("FEniCS-Heat") :1899            mcp.run(transport="stdio") :4554-4555
  solve_heat_1D :1902-1974   solve_heat_2D :1977-2041   solve_heat_3D :2122-2213
  solve_elasticity_1D_static :2523-2588   _2D_ :2590-2678   _3D_ :2680-2761
  SolveResult / TimeSeriesField / PlotResult :168-197 (defined in pde_solver_b200.fields)
  file contract: pickle of a TimeSeriesField at <data_dir>/<kind>_<uuid8>.pkl (:1961-1968 and siblings)
The orchestrator launches this file as a stdio child (multi_agent_orchestrator.py:27, 70-78); stdout is
the JSON-RPC channel, so nothing here or in the CUDA library prints to it.

All eleven solve tools run on the GPU: the six Cartesian ones (box geometry, uniform diffusivity) and the five
curvilinear heat tools (:2044-2119, 2220-2520; same loop with one scalar weight, SURVEY.md §8f n3).  The cylinder
and composite-core branches of solve_heat_3D (:512-572) run as in the reference's deployment, which has no mshr:
BoxMesh((0,-R,-R),(Lx,R,R)) with the radial weight sqrt(y^2+z^2), DG0 core diffusivity (n4).

Solver knobs the reference does not have come from the environment so existing callers are
unaffected: PDE_B200_RTOL (default 1e-10), PDE_B200_PRECOND (auto|gmg|jacobi),
PDE_B200_SNAPSHOT_STRIDE (default 1 = every step, as the reference), PDE_B200_STREAM (npz|xdmf: stream the
snapshots to a file beside the pickle instead of holding them all in memory).  All eight heat tools honour the
stride and streaming; the curvilinear tools write their coordinate-space lattice (e.g. (r, theta, phi)) and the
cylinder branch of solve_heat_3D the BoxMesh (0,-R,-R)-(Lx,R,R) it solves on.  Steady solves do not stream."""
import json
import os
import pickle
import sys
import uuid
from pathlib import Path
from typing import Dict, List, Optional

_ROOT = os.path.dirname(os.path.abspath(__file__))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

import numpy as np  # noqa: E402
from mcp.server.fastmcp import FastMCP  # noqa: E402

import pde_solver_b200 as _p  # noqa: E402
from pde_solver_b200.fields import PlotResult, SolveResult, TimeSeriesField  # noqa: E402,F401
from pde_solver_b200.solvers import curvilinear_grid, heat_3d_grid  # noqa: E402

mcp = FastMCP("FEniCS-Heat")


def _knobs():
    return dict(rtol=float(os.environ.get("PDE_B200_RTOL", "1e-10")),
                precond=os.environ.get("PDE_B200_PRECOND", "auto"))


def _stride():
    return max(1, int(os.environ.get("PDE_B200_SNAPSHOT_STRIDE", "1")))


def _stream(data_dir: str, stem: str, dim: int, n, L, origin=None, meta=None):
    """PDE_B200_STREAM=npz|xdmf: snapshots go to <data_dir>/<stem>_<uuid8>.<ext> one at a time (the pickle
    then keeps only the first and last one).  Returns (writer or None, uuid8)."""
    tag = uuid.uuid4().hex[:8]
    fmt = os.environ.get("PDE_B200_STREAM", "").lower()
    if fmt not in ("npz", "xdmf"):
        return None, tag
    from pde_solver_b200 import io as _io
    Path(data_dir).mkdir(parents=True, exist_ok=True)
    return _io.open_writer(fmt, str(Path(data_dir) / f"{stem}_{tag}.{fmt}"), dim, n, L, name="temperature",
                           meta=meta, origin=origin), tag


def _stream_grid(data_dir: str, stem: str, grid, system=None):
    """_stream for the lattice grid = (n, lo, hi) a solver builds: L = hi - lo, origin = lo."""
    n, lo, hi = grid
    meta = {"coordinate_system": system} if system else None
    return _stream(data_dir, stem, len(n), n, [h - l for l, h in zip(lo, hi)], origin=lo, meta=meta)


def _save(field: TimeSeriesField, data_dir: str, stem: str, tag: Optional[str] = None, writer=None) -> SolveResult:
    """mkdir data_dir, pickle the field to <stem>_<uuid8>.pkl, return SolveResult (:1956-1974)."""
    data_path = Path(data_dir)
    data_path.mkdir(parents=True, exist_ok=True)
    if writer is not None:
        # steady solves never stream: do not publish an empty series
        written = len(writer.times)
        path = writer.close()
        if written > 0:
            field.meta["snapshots_file"] = path
        else:
            for leftover in (path, os.path.splitext(path)[0] + ".bin"):
                if os.path.exists(leftover):
                    os.remove(leftover)
    filepath = data_path / f"{stem}_{tag or uuid.uuid4().hex[:8]}.pkl"
    with open(filepath, "wb") as f:
        pickle.dump(field, f, protocol=pickle.HIGHEST_PROTOCOL)
    return SolveResult(data_file=str(filepath), dim=field.dim, meta=field.meta)


# ─────────────────────────────── heat (Cartesian, in scope) ───────────────────────────────
@mcp.tool()
def solve_heat_1D(
    length: float = 2.0,
    nx: int = 50,
    diffusivity: float = 1.0,
    T_left: float = 20.0,
    T_right: float = 0.0,
    T_initial: float = 0.0,
    dt: float = 0.01,
    num_steps: int = 50,
    data_dir: str = "data",
    steady: bool = False,
    source_type: str = "none",
    source_value: float = 0.0,
    initial_type: str = "constant",
    initial_amplitude: float = 1.0,
    initial_wavenumber: float = 1.0,
) -> SolveResult:
    """1D heat equation u_t - k u_xx = f on (0, length), Dirichlet T_left / T_right, backward Euler
    (or steady when steady=True).  Returns the path of the pickled TimeSeriesField."""
    writer, tag = _stream(data_dir, "heat_1d", 1, [nx], [length])
    field = _p._solve_heat_1d_raw(
        length=length, nx=nx, diffusivity=diffusivity, T_left=T_left, T_right=T_right, T_initial=T_initial,
        dt=dt, num_steps=num_steps, steady=steady, source_type=source_type, source_value=source_value,
        initial_type=initial_type, initial_amplitude=initial_amplitude, initial_wavenumber=initial_wavenumber,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_1d", tag, writer)


@mcp.tool()
def solve_heat_2D(
    Lx: float = 1.0,
    Ly: float = 1.0,
    nx: int = 30,
    ny: int = 30,
    diffusivity: float = 1.0,
    T_boundary: float = 0.0,
    T_initial: float = 20.0,
    dt: float = 0.01,
    num_steps: int = 50,
    data_dir: str = "data",
    steady: bool = False,
    source_type: str = "none",
    source_value: float = 0.0,
    initial_type: str = "constant",
    initial_amplitude: float = 1.0,
    initial_wavenumber: float = 1.0,
) -> SolveResult:
    """2D heat equation on [0,Lx]x[0,Ly] with the constant Dirichlet value T_boundary on the whole boundary."""
    writer, tag = _stream(data_dir, "heat_2d", 2, [nx, ny], [Lx, Ly])
    field = _p._solve_heat_2d_raw(
        Lx=Lx, Ly=Ly, nx=nx, ny=ny, diffusivity=diffusivity, T_boundary=T_boundary, T_initial=T_initial, dt=dt,
        num_steps=num_steps, steady=steady, source_type=source_type, source_value=source_value,
        initial_type=initial_type, initial_amplitude=initial_amplitude, initial_wavenumber=initial_wavenumber,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_2d", tag, writer)


@mcp.tool()
def solve_heat_3D(
    Lx: float = 1.0,
    Ly: float = 1.0,
    Lz: float = 1.0,
    nx: int = 10,
    ny: int = 10,
    nz: int = 10,
    diffusivity: float = 1.0,
    T_boundary: float = 0.0,
    T_initial: float = 20.0,
    dt: float = 0.01,
    num_steps: int = 20,
    data_dir: str = "data",
    steady: bool = False,
    source_type: str = "none",
    source_value: float = 0.0,
    initial_type: str = "constant",
    initial_amplitude: float = 1.0,
    initial_wavenumber: float = 1.0,
    geometry_type: str = "box",
    cylinder_radius: Optional[float] = None,
    T_left: Optional[float] = None,
    T_right: Optional[float] = None,
    T_side: Optional[float] = None,
    core_radius: Optional[float] = None,
    core_diffusivity: Optional[float] = None,
) -> SolveResult:
    """3D heat equation on the box [0,Lx]x[0,Ly]x[0,Lz]: uniform Dirichlet value T_boundary, or the
    directional values T_left (x=0) / T_right (x=Lx) / T_side (remaining faces)."""
    # the cylinder branch solves on BoxMesh (0,-R,-R)-(Lx,R,R) with its own node counts
    writer, tag = _stream_grid(data_dir, "heat_3d", heat_3d_grid(Lx, Ly, Lz, nx, ny, nz, geometry_type,
                                                                 cylinder_radius))
    field = _p._solve_heat_3d_raw(
        Lx=Lx, Ly=Ly, Lz=Lz, nx=nx, ny=ny, nz=nz, diffusivity=diffusivity, T_boundary=T_boundary,
        T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        initial_wavenumber=initial_wavenumber, geometry_type=geometry_type, cylinder_radius=cylinder_radius,
        T_left=T_left, T_right=T_right, T_side=T_side, core_radius=core_radius,
        core_diffusivity=core_diffusivity, snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_3d", tag, writer)


# ─────────────────────────────── elasticity (in scope) ───────────────────────────────
@mcp.tool()
def solve_elasticity_1D_static(
    L: float = 1.0,
    nx: int = 50,
    E: float = 210e9,
    area: float = 1.0,
    body_force: float = 0.0,
    quantity: str = "stress",
    data_dir: str = "data",
) -> SolveResult:
    """1D axial bar, static: -(E A u')' = body_force, u(0)=0; outputs axial stress or strain (P1-projected)."""
    field = _p._solve_elasticity_1d_static(L=L, nx=nx, E=E, area=area, body_force=body_force, quantity=quantity,
                                           **_knobs())
    return _save(field, data_dir, f"elasticity_1d_{quantity}")


@mcp.tool()
def solve_elasticity_2D_static(
    Lx: float = 1.0,
    Ly: float = 1.0,
    nx: int = 30,
    ny: int = 30,
    E: float = 210e9,
    nu: float = 0.3,
    body_fx: float = 0.0,
    body_fy: float = 0.0,
    quantity: str = "stress",
    plane_stress: bool = True,
    data_dir: str = "data",
) -> SolveResult:
    """2D static linear elasticity on a rectangle clamped at x=0; outputs von Mises stress or strain."""
    field = _p._solve_elasticity_2d_static(Lx=Lx, Ly=Ly, nx=nx, ny=ny, E=E, nu=nu, body_fx=body_fx, body_fy=body_fy,
                                           quantity=quantity, plane_stress=plane_stress, **_knobs())
    return _save(field, data_dir, f"elasticity_2d_{quantity}")


@mcp.tool()
def solve_elasticity_3D_static(
    Lx: float = 1.0,
    Ly: float = 1.0,
    Lz: float = 1.0,
    nx: int = 10,
    ny: int = 10,
    nz: int = 10,
    E: float = 210e9,
    nu: float = 0.3,
    body_fx: float = 0.0,
    body_fy: float = 0.0,
    body_fz: float = 0.0,
    quantity: str = "stress",
    data_dir: str = "data",
) -> SolveResult:
    """3D static linear elasticity on a box clamped at x=0; outputs von Mises stress or strain."""
    field = _p._solve_elasticity_3d_static(Lx=Lx, Ly=Ly, Lz=Lz, nx=nx, ny=ny, nz=nz, E=E, nu=nu, body_fx=body_fx,
                                           body_fy=body_fy, body_fz=body_fz, quantity=quantity, **_knobs())
    return _save(field, data_dir, f"elasticity_3d_{quantity}")


# ─────────────────── curvilinear heat tools (reference :2044-2119, 2220-2520) ───────────────────
@mcp.tool()
def solve_heat_3D_spherical(
    r_inner: float = 0.1, r_outer: float = 1.0, nr: int = 20, ntheta: int = 20, nphi: int = 20,
    diffusivity: float = 1.0, T_boundary: float = 20.0, T_initial: float = 20.0, dt: float = 0.01,
    num_steps: int = 50, data_dir: str = "data", steady: bool = False, source_type: str = "none",
    source_value: float = 0.0, initial_type: str = "constant", initial_amplitude: float = 1.0,
) -> SolveResult:
    """3D heat equation in spherical coordinates (r, theta, phi) on [r_inner, r_outer] x [0, pi] x [0, 2 pi]."""
    writer, tag = _stream_grid(data_dir, "heat_3d_spherical",
                               curvilinear_grid("3d_spherical", r_inner, r_outer, [nr, ntheta, nphi]),
                               "spherical (r, theta, phi)")
    field = _p._solve_heat_3d_spherical_raw(
        r_inner=r_inner, r_outer=r_outer, nr=nr, ntheta=ntheta, nphi=nphi, diffusivity=diffusivity,
        T_boundary=T_boundary, T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_3d_spherical", tag, writer)


@mcp.tool()
def solve_heat_1D_cylindrical(
    r_inner: float = 0.1, r_outer: float = 1.0, nr: int = 50, diffusivity: float = 1.0, T_inner: float = 100.0,
    T_outer: float = 20.0, T_initial: float = 20.0, dt: float = 0.01, num_steps: int = 50, data_dir: str = "data",
    steady: bool = False, source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
    initial_amplitude: float = 1.0,
) -> SolveResult:
    """1D radial heat equation in cylindrical coordinates on (r_inner, r_outer)."""
    writer, tag = _stream_grid(data_dir, "heat_1d_cylindrical",
                               curvilinear_grid("1d_cylindrical", r_inner, r_outer, [nr]), "cylindrical (r)")
    field = _p._solve_heat_1d_cylindrical_raw(
        r_inner=r_inner, r_outer=r_outer, nr=nr, diffusivity=diffusivity, T_inner=T_inner, T_outer=T_outer,
        T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_1d_cylindrical", tag, writer)


@mcp.tool()
def solve_heat_1D_spherical(
    r_inner: float = 0.1, r_outer: float = 1.0, nr: int = 50, diffusivity: float = 1.0, T_inner: float = 100.0,
    T_outer: float = 20.0, T_initial: float = 20.0, dt: float = 0.01, num_steps: int = 50, data_dir: str = "data",
    steady: bool = False, source_type: str = "none", source_value: float = 0.0, initial_type: str = "constant",
    initial_amplitude: float = 1.0,
) -> SolveResult:
    """1D radial heat equation in spherical coordinates on (r_inner, r_outer)."""
    writer, tag = _stream_grid(data_dir, "heat_1d_spherical", curvilinear_grid("1d_spherical", r_inner, r_outer, [nr]),
                               "spherical (r)")
    field = _p._solve_heat_1d_spherical_raw(
        r_inner=r_inner, r_outer=r_outer, nr=nr, diffusivity=diffusivity, T_inner=T_inner, T_outer=T_outer,
        T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_1d_spherical", tag, writer)


@mcp.tool()
def solve_heat_2D_cylindrical(
    r_inner: float = 0.1, r_outer: float = 1.0, z_length: float = 2.0, nr: int = 30, nz: int = 30,
    diffusivity: float = 1.0, T_boundary: float = 20.0, T_initial: float = 20.0, dt: float = 0.01,
    num_steps: int = 50, data_dir: str = "data", steady: bool = False, source_type: str = "none",
    source_value: float = 0.0, initial_type: str = "constant", initial_amplitude: float = 1.0,
) -> SolveResult:
    """2D axisymmetric heat equation in cylindrical coordinates (r, z)."""
    writer, tag = _stream_grid(data_dir, "heat_2d_cylindrical",
                               curvilinear_grid("2d_cylindrical", r_inner, r_outer, [nr, nz], z_length),
                               "cylindrical (r, z)")
    field = _p._solve_heat_2d_cylindrical_raw(
        r_inner=r_inner, r_outer=r_outer, z_length=z_length, nr=nr, nz=nz, diffusivity=diffusivity,
        T_boundary=T_boundary, T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_2d_cylindrical", tag, writer)


@mcp.tool()
def solve_heat_2D_spherical(
    r_inner: float = 0.1, r_outer: float = 1.0, nr: int = 30, ntheta: int = 30, diffusivity: float = 1.0,
    T_boundary: float = 20.0, T_initial: float = 20.0, dt: float = 0.01, num_steps: int = 50,
    data_dir: str = "data", steady: bool = False, source_type: str = "none", source_value: float = 0.0,
    initial_type: str = "constant", initial_amplitude: float = 1.0,
) -> SolveResult:
    """2D axisymmetric heat equation in spherical coordinates (r, theta)."""
    writer, tag = _stream_grid(data_dir, "heat_2d_spherical",
                               curvilinear_grid("2d_spherical", r_inner, r_outer, [nr, ntheta]), "spherical (r, theta)")
    field = _p._solve_heat_2d_spherical_raw(
        r_inner=r_inner, r_outer=r_outer, nr=nr, ntheta=ntheta, diffusivity=diffusivity, T_boundary=T_boundary,
        T_initial=T_initial, dt=dt, num_steps=num_steps, steady=steady, source_type=source_type,
        source_value=source_value, initial_type=initial_type, initial_amplitude=initial_amplitude,
        snapshot_stride=_stride(), stream_to=writer, **_knobs())
    return _save(field, data_dir, "heat_2d_spherical", tag, writer)


# ─────────────────────────────── plot tools (consumers of the .pkl) ───────────────────────────────
def _check_field(coords, values, times):
    """Shape contract the reference's plot tool enforces (:3453-3466)."""
    coords = np.asarray(coords, dtype=float)
    values = np.asarray(values, dtype=float)
    times = np.asarray(times, dtype=float)
    if values.ndim != 2:
        raise ValueError("values must be 2-D [Nt][N]")
    if coords.ndim != 2 or coords.shape[1] != 3:
        raise ValueError("coords must be [N][3]")
    if coords.shape[0] != values.shape[1]:
        raise ValueError("coords and values disagree on the number of points")
    if times.shape[0] != values.shape[0]:
        raise ValueError("times and values disagree on the number of frames")
    if values.size == 0:
        raise ValueError("empty field")
    return coords, values, times


def _render(coords, values, times, dim, field_name, unit, output_dir, filename) -> PlotResult:
    """Minimal HTML rendering of a scalar time series.  The reference's 1 800-line Plotly/griddata
    visualiser (:2764-4551) is out of scope; this keeps the dispatcher's solve -> plot flow working
    (dispatcher_agent.py:248-283).  Plotly is used when importable, otherwise a dependency-free page."""
    coords, values, times = _check_field(coords, values, times)
    out = Path(output_dir)
    out.mkdir(parents=True, exist_ok=True)
    path = out / filename
    label = f"{field_name} [{unit}]" if unit else field_name
    try:
        import plotly.graph_objects as go  # type: ignore
    except Exception:
        go = None
    if go is not None:
        n = coords.shape[0]
        pick = np.arange(n) if n <= 20000 else np.linspace(0, n - 1, 20000).astype(int)
        last = values[-1]
        if dim == 1:
            fig = go.Figure([go.Scatter(x=coords[pick, 0], y=values[k, pick], name=f"t={times[k]:.4g}")
                             for k in np.unique(np.linspace(0, len(times) - 1, 6).astype(int))])
            fig.update_layout(xaxis_title="x", yaxis_title=label)
        elif dim == 2:
            fig = go.Figure(go.Scatter(x=coords[pick, 0], y=coords[pick, 1], mode="markers",
                                       marker=dict(color=last[pick], colorscale="Inferno", showscale=True,
                                                   colorbar=dict(title=label))))
        else:
            fig = go.Figure(go.Scatter3d(x=coords[pick, 0], y=coords[pick, 1], z=coords[pick, 2], mode="markers",
                                         marker=dict(size=2, color=last[pick], colorscale="Inferno",
                                                     showscale=True, colorbar=dict(title=label))))
        fig.update_layout(title=f"{label}, t = {times[-1]:.4g}")
        fig.write_html(str(path), include_plotlyjs="cdn")
    else:
        rows = "".join(f"<tr><td>{t:.6g}</td><td>{v.min():.6g}</td><td>{v.max():.6g}</td><td>{v.mean():.6g}</td></tr>"
                       for t, v in zip(times, values))
        summary = {"dim": int(dim), "points": int(coords.shape[0]), "frames": int(len(times)), "field": label}
        path.write_text(
            "<!doctype html><html><head><meta charset='utf-8'><title>" + label + "</title></head><body>"
            "<h3>" + label + "</h3><pre>" + json.dumps(summary) + "</pre>"
            "<table border='1'><tr><th>t</th><th>min</th><th>max</th><th>mean</th></tr>" + rows +
            "</table><p>plotly is not installed: summary table only.</p></body></html>", encoding="utf-8")
    return PlotResult(html_path=str(path))


@mcp.tool()
def plot_time_series_field_from_file(
    data_file: str,
    field_name: Optional[str] = None,
    unit: Optional[str] = None,
    output_dir: str = "plots",
    filename: Optional[str] = None,
) -> PlotResult:
    """Load a pickled TimeSeriesField written by a solve_* tool and render it to HTML (:2764-2936)."""
    with open(data_file, "rb") as f:
        field = pickle.load(f)
    meta = getattr(field, "meta", {}) or {}
    name = field_name or meta.get("name", "u")
    un = unit if unit is not None else meta.get("unit", "")
    if filename is None:
        filename = Path(data_file).stem + ".html"
    return _render(field.coords, field.values, field.times, field.dim, name, un, output_dir, filename)


@mcp.tool()
def plot_time_series_field(
    coords: List[List[float]],
    values: List[List[float]],
    times: List[float],
    dim: int = 1,
    field_name: str = "u",
    unit: str = "",
    output_dir: str = "plots",
    filename: str = "field_timeseries_3d.html",
    domain_bounds: Optional[Dict[str, float]] = None,
    geometry_type: Optional[str] = None,
    geometry_params: Optional[Dict[str, float]] = None,
) -> PlotResult:
    """Render a scalar field time series given in memory (:3409-3466)."""
    return _render(coords, values, times, dim, field_name, unit, output_dir, filename)


@mcp.tool()
def plot_time_series_field_old(
    coords: List[List[float]],
    values: List[List[float]],
    times: List[float],
    dim: int = 1,
    field_name: str = "u",
    unit: str = "",
    output_dir: str = "plots",
    filename: str = "field_timeseries_3d.html",
) -> PlotResult:
    """Older entry point kept for name compatibility (:4143-4551)."""
    return _render(coords, values, times, dim, field_name, unit, output_dir, filename)


if __name__ == "__main__":
    mcp.run(transport="stdio")
