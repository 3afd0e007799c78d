"""Resident stepper of the weighted heat solves (pde_wheat_open / set_state / step / get_state / close): snapshot
streaming, snapshot stride and host initial fields for the curvilinear tools and the cylinder / composite-core
branches of _solve_heat_3d_raw.

CPU: the writers' origin, the cylinder mesh rule shared by the solver and the MCP tool, u0 validation.  GPU
(pytest.mark.gpu): streamed runs against the in-memory path bit for bit, runs from u0 against an LU reference built
from the oracle's weighted assembly, restarts through the C ABI, statistics, the MCP tools and one large grid."""
import ctypes as C
import os
import pickle
import re

import numpy as np
import pytest

from oracle import fem_oracle as fo

TOL = 1e-8


# ---------------------------------------------------------------- CPU
# written by the XdmfSnapshotWriter before it took an origin: without one the file must not change
XDMF_1D = """<?xml version="1.0" ?>
<Xdmf Version="3.0">
 <Domain>
  <Grid Name="series" GridType="Collection" CollectionType="Temporal">
   <Grid Name="step0" GridType="Uniform">
    <Time Value="0.5"/>
    <Topology TopologyType="2DCoRectMesh" Dimensions="1 4"/>
    <Geometry GeometryType="ORIGIN_DXDY">
     <DataItem Dimensions="2" NumberType="Float" Precision="8" Format="XML">0 0</DataItem>
     <DataItem Dimensions="2" NumberType="Float" Precision="8" Format="XML">1 0.5</DataItem>
    </Geometry>
    <Attribute Name="temperature" AttributeType="Scalar" Center="Node">
     <DataItem Dimensions="1 4" NumberType="Float" Precision="8" Format="Binary" Endian="Little" Seek="0">g1.bin</DataItem>
    </Attribute>
   </Grid>
  </Grid>
 </Domain>
</Xdmf>
"""
XDMF_3D = """<?xml version="1.0" ?>
<Xdmf Version="3.0">
 <Domain>
  <Grid Name="series" GridType="Collection" CollectionType="Temporal">
   <Grid Name="step0" GridType="Uniform">
    <Time Value="0.5"/>
    <Topology TopologyType="3DCoRectMesh" Dimensions="2 2 3"/>
    <Geometry GeometryType="ORIGIN_DXDYDZ">
     <DataItem Dimensions="3" NumberType="Float" Precision="8" Format="XML">0 0 0</DataItem>
     <DataItem Dimensions="3" NumberType="Float" Precision="8" Format="XML">0.25 0.5 0.5</DataItem>
    </Geometry>
    <Attribute Name="temperature" AttributeType="Scalar" Center="Node">
     <DataItem Dimensions="2 2 3" NumberType="Float" Precision="8" Format="Binary" Endian="Little" Seek="0">g3.bin</DataItem>
    </Attribute>
   </Grid>
  </Grid>
 </Domain>
</Xdmf>
"""


def _origin_item(xml):
    return re.search(r'GeometryType="ORIGIN_DXDY(?:DZ)?">\s*<DataItem[^>]*>([^<]*)<', xml).group(1)


def test_xdmf_without_origin_is_unchanged(tmp_path):
    from pde_solver_b200 import io
    for stem, dim, n, L, want in (("g1", 1, [3], [1.5], XDMF_1D), ("g3", 3, [2, 1, 1], [1.0, 0.5, 0.25], XDMF_3D)):
        for origin in (None, [0.0] * dim):
            with io.open_writer("xdmf", tmp_path / stem, dim, n, L, name="temperature", origin=origin) as w:
                w.append(0.5, np.arange(int(np.prod([k + 1 for k in n])), dtype=float))
            assert open(tmp_path / f"{stem}.xdmf").read() == want, (stem, origin)


def test_writer_origin_round_trips(tmp_path):
    import json
    import zipfile
    from pde_solver_b200 import io
    for dim, n, lo, hi in ((1, [4], [0.1], [1.0]), (2, [3, 2], [0.25, 0.0], [1.0, np.pi]),
                           (3, [2, 3, 4], [0.0, -0.5, -0.5], [1.0, 0.5, 0.5])):
        L = [h - l for l, h in zip(lo, hi)]
        nv = int(np.prod([k + 1 for k in n]))
        snaps = [np.arange(nv, dtype=float) * (k + 1) for k in range(2)]
        meta = {"coordinate_system": "test"}
        for fmt in ("npz", "xdmf"):
            with io.open_writer(fmt, tmp_path / f"o{dim}.{fmt}", dim, n, L, meta=meta, origin=lo) as w:
                for k, v in enumerate(snaps):
                    w.append(0.1 * k, v)
        with np.load(tmp_path / f"o{dim}.npz") as z:
            assert np.array_equal(z["origin"], lo) and np.array_equal(z["extent"], L)
        with zipfile.ZipFile(tmp_path / f"o{dim}.npz") as z:
            m = json.loads(z.read("meta.json"))
        assert m["origin"] == lo and m["coordinate_system"] == "test"
        t, v = io.read_npz_series(tmp_path / f"o{dim}.npz")
        assert np.array_equal(v, np.stack(snaps))
        xml = open(tmp_path / f"o{dim}.xdmf").read()
        # XDMF lists the slowest axis first; a 1-D lattice is padded with a leading axis at 0
        want = ([0.0] + lo) if dim == 1 else lo[::-1]
        assert [float(x) for x in _origin_item(xml).split()] == want
        t, v = io.read_xdmf_series(str(tmp_path / f"o{dim}.xdmf"))
        assert np.array_equal(v, np.stack(snaps)) and np.allclose(t, [0.0, 0.1])


@pytest.mark.parametrize("R,ny,nz,Lx,nx", [(0.5, 8, 8, 1.0, 4), (0.75, 8, 6, 2.0, 3), (0.3, 10, 7, 1.0, 5),
                                          (1.25, 4, 4, 0.5, 2)])
def test_cylinder_grid_is_the_mesh_the_solver_builds(R, ny, nz, Lx, nx):
    from pde_solver_b200.solvers import heat_3d_grid
    n, lo, hi = heat_3d_grid(Lx, 9.0, 9.0, nx, ny, nz, "cylinder", R)
    mesh = fo.box_mesh((0.0, -R, -R), (Lx, R, R), nx, int(ny * 2 * R), int(nz * 2 * R))
    assert int(np.prod([k + 1 for k in n])) == mesh.nv
    assert np.array_equal(mesh.coords.min(axis=0), lo) and np.array_equal(mesh.coords.max(axis=0), hi)
    # without a radius (and for every other geometry) the box itself
    assert heat_3d_grid(Lx, 2.0, 3.0, nx, ny, nz, "cylinder", None) == ([nx, ny, nz], [0.0] * 3, [Lx, 2.0, 3.0])
    assert heat_3d_grid(Lx, 2.0, 3.0, nx, ny, nz, "box", R) == ([nx, ny, nz], [0.0] * 3, [Lx, 2.0, 3.0])


def test_u0_of_the_wrong_length_is_rejected_before_the_library():
    import pde_solver_b200 as P
    with pytest.raises(ValueError, match="u0"):
        P._solve_heat_2d_spherical_raw(0.1, 1.0, 8, 8, 1.0, 35.0, 20.0, 0.01, 2, u0=np.zeros(80))
    with pytest.raises(ValueError, match="u0"):
        P._solve_heat_1d_cylindrical_raw(0.1, 1.0, 8, 1.0, 100.0, 20.0, 20.0, 0.01, 2, u0=np.zeros((1, 9)))
    with pytest.raises(ValueError, match="u0"):
        P._solve_heat_3d_raw(1, 1, 1, 4, 4, 4, 1.0, 0.0, 20.0, 0.01, 1, geometry_type="cylinder", cylinder_radius=1.0,
                             u0=np.zeros(125))


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def P():
    import pde_solver_b200 as p
    return p


# the curvilinear cases of tests/test_weighted_gmg.py (every axis even, so GMG coarsens)
CURVI = [
    ("1d_cylindrical", [64], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("1d_cylindrical", [64], dict(r_inner=0.0, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("1d_spherical", [64], dict(r_inner=0.1, r_outer=1.0, T_inner=100.0, T_outer=20.0)),
    ("2d_cylindrical", [32, 32], dict(r_inner=0.1, r_outer=1.0, z_length=2.0, T_boundary=35.0)),
    ("2d_spherical", [32, 32], dict(r_inner=0.1, r_outer=1.0, T_boundary=35.0)),
    ("3d_spherical", [16, 8, 16], dict(r_inner=0.2, r_outer=1.0, T_boundary=35.0)),
]
NAMES = {"1d_cylindrical": ["nr"], "1d_spherical": ["nr"], "2d_cylindrical": ["nr", "nz"],
         "2d_spherical": ["nr", "ntheta"], "3d_spherical": ["nr", "ntheta", "nphi"]}
SPECIAL = [
    dict(geometry_type="cylinder", cylinder_radius=0.5, T_boundary=1.0, T_initial=5.0, source_type="constant",
         source_value=3.0),
    dict(core_radius=0.3, core_diffusivity=25.0, T_left=1.0, T_side=2.0, T_initial=3.0),
    dict(core_radius=0.3, core_diffusivity=4.0, T_boundary=0.5, initial_type="cosine", initial_amplitude=2.0,
         initial_wavenumber=3.0),
]
COMMON = dict(diffusivity=0.8, T_initial=20.0, dt=0.02, num_steps=4, source_type="constant", source_value=40.0)


def _curvi(P, kind, n, kw, **extra):
    args = dict(COMMON)
    args.update(extra)
    return getattr(P, f"_solve_heat_{kind}_raw")(**kw, **dict(zip(NAMES[kind], n)), **args, as_arrays=True)


def _special(P, case, **extra):
    kw = dict(T_boundary=0.0, T_initial=0.0, dt=0.02, num_steps=4)
    kw.update(case)
    kw.update(extra)
    return P._solve_heat_3d_raw(1.0, 0.5, 0.5, 8, 16, 16, 0.8, kw.pop("T_boundary"), kw.pop("T_initial"),
                                kw.pop("dt"), kw.pop("num_steps"), as_arrays=True, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
@pytest.mark.parametrize("case", [c[0] + "_" + str(i) for i, c in enumerate(CURVI)] +
                         ["special_" + str(i) for i in range(len(SPECIAL))])
def test_streaming_matches_in_memory_bitwise(P, case, precond, tmp_path):
    from pde_solver_b200 import io
    kind, idx = case.rsplit("_", 1)
    idx = int(idx)
    if kind == "special":
        run = lambda **kw: _special(P, SPECIAL[idx], precond=precond, **kw)  # noqa: E731
        n = _special_n(SPECIAL[idx])
        dim = 3
    else:
        kind, n, kw0 = CURVI[idx]
        run = lambda **kw: _curvi(P, kind, n, kw0, precond=precond, **kw)  # noqa: E731
        dim = len(n)
    full = run()
    assert full.values.shape[0] == 5
    with io.open_writer("npz", tmp_path / "s.npz", dim, n, [1.0] * dim) as w:
        part = run(snapshot_stride=2, stream_to=w)
    t, v = io.read_npz_series(tmp_path / "s.npz")
    assert np.array_equal(v, full.values[::2])
    assert np.array_equal(t, full.times[::2])
    assert np.array_equal(part.values, full.values[[0, -1]]) and np.array_equal(part.times, full.times[[0, -1]])
    # stride without a writer: the in-memory path keeps every second state
    strided = run(snapshot_stride=2)
    assert np.array_equal(strided.values, full.values[::2])


def _special_n(case):
    from pde_solver_b200.solvers import heat_3d_grid
    return heat_3d_grid(1.0, 0.5, 0.5, 8, 16, 16, case.get("geometry_type", "box"), case.get("cylinder_radius"))[0]


def _reference_from(u0, K, Mw, mw, bc_dofs, bc_vals, dt, f, num_steps):
    """Backward Euler of the oracle (rowwise Dirichlet elimination, sparse LU) from the host field u0."""
    u = np.array(u0, dtype=float)
    u[bc_dofs] = bc_vals
    snaps = [u.copy()]
    A, _ = fo.apply_bc_rowwise((Mw + dt * K).tocsr(), np.zeros(u.size), bc_dofs, bc_vals)
    for _ in range(num_steps):
        b = Mw @ u + (dt * f) * mw
        b[bc_dofs] = bc_vals
        u = fo.lu_solve(A.tocsr(), b)
        snaps.append(u.copy())
    return np.array(snaps)


def _system(name, kappa):
    """(K with kappa, Mw, mw, Dirichlet dofs, values) of the u0 cases; every boundary vertex carries T_boundary."""
    if name == "cylinder_core":
        R, core, kcore = 0.5, 0.3, 25.0
        mesh = fo.box_mesh((0.0, -R, -R), (1.0, R, R), 8, 16, 16)
        X = mesh.coords[mesh.cells]
        rv = np.sqrt(X[:, :, 1] ** 2 + X[:, :, 2] ** 2)
        mid = X.mean(axis=1)
        inside = (rv < core).all(axis=1) & (np.sqrt(mid[:, 1] ** 2 + mid[:, 2] ** 2) < core)
        K, Mw, mw = fo.assemble_weighted(mesh, lambda x: np.sqrt(x[:, 1] ** 2 + x[:, 2] ** 2), 2,
                                         cell_scale=np.where(inside, kcore, kappa))
    else:
        r_inner = 0.2 if name == "3d_spherical" else 0.1
        n = [16, 8, 16] if name == "3d_spherical" else [32, 32]
        dim, degree, wfun = fo.CURVILINEAR[name]
        mesh = fo.curvilinear_mesh(name, r_inner, 1.0, n)
        K, Mw, mw = fo.assemble_weighted(mesh, wfun, degree)
        K = kappa * K
    dofs = fo.dirichlet_dofs(mesh, lambda x, ob: ob)
    return K, Mw, mw, dofs, mesh.nv


U0_CASES = ["2d_spherical", "3d_spherical", "cylinder_core"]


def _run_u0(P, name, u0, precond, **kw):
    common = dict(diffusivity=0.8, T_initial=20.0, dt=0.02, num_steps=4, source_type="constant", source_value=40.0,
                  precond=precond, as_arrays=True, u0=u0)
    common.update(kw)
    if name == "2d_spherical":
        return P._solve_heat_2d_spherical_raw(0.1, 1.0, 32, 32, T_boundary=35.0, **common)
    if name == "3d_spherical":
        return P._solve_heat_3d_spherical_raw(0.2, 1.0, 16, 8, 16, T_boundary=35.0, **common)
    kappa = common.pop("diffusivity")
    return P._solve_heat_3d_raw(1.0, 1.0, 1.0, 8, 16, 16, kappa, 35.0, common.pop("T_initial"), common.pop("dt"),
                                common.pop("num_steps"), geometry_type="cylinder", cylinder_radius=0.5, core_radius=0.3,
                                core_diffusivity=25.0, **common)


@pytest.mark.gpu
@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
@pytest.mark.parametrize("name", U0_CASES)
def test_u0_matches_oracle(P, name, precond):
    K, Mw, mw, dofs, nv = _system(name, 0.8)
    u0 = 20.0 + 10.0 * np.random.default_rng(7).standard_normal(nv)
    f = _run_u0(P, name, u0, precond)
    ref = _reference_from(u0, K, Mw, mw, dofs, np.full(dofs.size, 35.0), 0.02, 40.0, 4)
    assert f.values.shape == ref.shape
    free = np.ones(nv, dtype=bool)
    free[dofs] = False
    assert np.array_equal(f.values[0][dofs], np.full(dofs.size, 35.0))       # Dirichlet values re-applied
    assert np.array_equal(f.values[0][free], u0[free])
    for k in range(ref.shape[0]):
        assert fo.rel_l2(f.values[k], ref[k]) <= TOL, (k, fo.rel_l2(f.values[k], ref[k]))
    st = P.last_stats()
    assert st["converged"] == 1 and st["solves"] == 4
    if precond == "gmg":
        assert st["levels"] >= 2 and st["true_relres"] <= 1e-9, st


@pytest.mark.gpu
@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
def test_steady_u0_is_only_the_starting_guess(P, precond):
    u0 = np.full(33 * 33, 30.0)
    f = _run_u0(P, "2d_spherical", u0, precond, steady=True)
    ref = fo.solve_heat_curvilinear("2d_spherical", 0.1, 1.0, [32, 32], 0.8, steady=True, source_type="constant",
                                    source_value=40.0, T_boundary=35.0)
    assert f.values.shape == (1, 33 * 33) and fo.rel_l2(f.values[0], ref.values[0]) <= TOL
    assert P.last_stats()["solves"] == 1


def _params(P, name):
    """WheatParams of a transient U0 case, as the public functions fill them."""
    L = P._lib
    p = L.WheatParams()
    if name == "2d_spherical":
        p.dim, p.n, p.lo, p.hi = 2, L.i3([32, 32]), L.d3([0.1, 0.0], 0.0), L.d3([1.0, np.pi], 1.0)
        p.weight_rpow, p.weight_sin_axis1, p.weight_degree = 2, 1, 2
        p.bc = L.make_bc({f: 35.0 for f in range(4)})
    else:
        p.dim, p.n, p.lo, p.hi = 3, L.i3([8, 16, 16]), L.d3([0.0, -0.5, -0.5]), L.d3([1.0, 0.5, 0.5])
        p.weight_degree, p.weight_kind = 2, 1
        p.has_core, p.core_radius, p.core_diffusivity = 1, 0.3, 25.0
        p.bc = L.make_bc({f: 35.0 for f in range(6)})
    p.diffusivity, p.dt, p.num_steps, p.snapshot_stride = 0.8, 0.02, 0, 1
    p.source_value, p.T_initial = 40.0, 20.0
    return p


def _stepper(P, p, precond):
    return P._lib.WheatStepper(P._lib.default_context(), p, P._lib.make_opts(precond=precond))


@pytest.mark.gpu
@pytest.mark.parametrize("precond", ["jacobi", "gmg"])
@pytest.mark.parametrize("name", ["2d_spherical", "cylinder_core"])
def test_set_state_restarts_cleanly(P, name, precond):
    p = _params(P, name)
    a = _stepper(P, p, precond)
    b = _stepper(P, p, precond)
    try:
        assert a.nloc == (33 * 33 if name == "2d_spherical" else 9 * 17 * 17)
        u0 = np.random.default_rng(11).standard_normal(a.nloc)
        a.step(3)
        a.set_state(u0)
        a.step(2)
        b.set_state(u0)
        b.step(2)
        assert np.array_equal(a.get_state(np.empty(a.nloc)), b.get_state(np.empty(b.nloc)))
    finally:
        a.close()
        b.close()
    # a host initial field only enters through set_state
    p.initial_type = P._lib.IC["array"]
    h = C.c_void_p()
    o = P._lib.make_opts(precond=precond)
    assert P._lib.lib().pde_wheat_open(P._lib.default_context().handle, C.byref(p), C.byref(o), C.byref(h)) != 0
    vals, times = np.empty((1, 33 * 33 if name == "2d_spherical" else 9 * 17 * 17)), np.empty(1)
    assert P._lib.lib().pde_wheat_solve(P._lib.default_context().handle, C.byref(p), C.byref(o), P._lib.ptr(vals),
                                        P._lib.ptr(times), None) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d_spherical", "cylinder_core"])
def test_streamed_gmg_stats(P, name, tmp_path):
    from pde_solver_b200 import io
    s = _stepper(P, _params(P, name), "gmg")
    try:
        per_step = [s.step(1)["iters_total"] for _ in range(6)]
    finally:
        s.close()
    with io.open_writer("npz", tmp_path / "s.npz", 3, [1, 1, 1], [1, 1, 1]) as w:
        if name == "2d_spherical":
            P._solve_heat_2d_spherical_raw(0.1, 1.0, 32, 32, 0.8, 35.0, 20.0, 0.02, 6, source_type="constant",
                                           source_value=40.0, precond="gmg", stream_to=w)
        else:
            P._solve_heat_3d_raw(1.0, 1.0, 1.0, 8, 16, 16, 0.8, 35.0, 20.0, 0.02, 6, source_type="constant",
                                 source_value=40.0, geometry_type="cylinder", cylinder_radius=0.5, core_radius=0.3,
                                 core_diffusivity=25.0, precond="gmg", stream_to=w)
    st = P.last_stats()
    assert st["converged"] == 1 and st["levels"] >= 2 and st["true_relres"] <= 1e-9, st
    assert st["solves"] == 6 and st["iters_total"] == sum(per_step), (st, per_step)
    assert st["solve_ms"] > 0 and st["launches"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("R,ny", [(0.5, 8), (0.75, 8)])
def test_mcp_tools_stream_the_mesh_they_solve_on(P, R, ny, tmp_path, monkeypatch):
    import fenics_mcp_server as server
    from pde_solver_b200 import io
    kw2 = dict(r_inner=0.1, r_outer=1.0, z_length=2.0, nr=8, nz=ny, num_steps=4)
    kw3 = dict(Lx=1.0, Ly=1.0, Lz=1.0, nx=4, ny=ny, nz=ny, num_steps=4, geometry_type="cylinder",
               cylinder_radius=R, T_initial=20.0)
    raw2 = P._solve_heat_2d_cylindrical_raw(diffusivity=1.0, T_boundary=20.0, T_initial=20.0, dt=0.01,
                                            as_arrays=True, **kw2)
    raw3 = P._solve_heat_3d_raw(diffusivity=1.0, T_boundary=0.0, dt=0.01, as_arrays=True, **kw3)
    n3 = [4, int(ny * 2 * R), int(ny * 2 * R)]
    assert raw3.values.shape[1] == int(np.prod([k + 1 for k in n3]))
    # defaults: the pickles hold exactly the raw calls
    for tool, kw, raw in ((server.solve_heat_2D_cylindrical, kw2, raw2), (server.solve_heat_3D, kw3, raw3)):
        res = tool(data_dir=str(tmp_path / "plain"), **kw)
        field = pickle.load(open(res.data_file, "rb"))
        assert "snapshots_file" not in res.meta
        assert np.array_equal(np.asarray(field.values), raw.values)
    monkeypatch.setenv("PDE_B200_STREAM", "xdmf")
    monkeypatch.setenv("PDE_B200_SNAPSHOT_STRIDE", "2")
    for tool, kw, raw, origin in ((server.solve_heat_2D_cylindrical, kw2, raw2, [0.0, 0.1]),
                                  (server.solve_heat_3D, kw3, raw3, [-R, -R, 0.0])):
        res = tool(data_dir=str(tmp_path / "stream"), **kw)
        path = res.meta["snapshots_file"]
        t, v = io.read_xdmf_series(path)
        assert v.shape == (3, raw.values.shape[1])
        assert np.array_equal(v, raw.values[::2]) and np.array_equal(t, raw.times[::2])
        assert [float(x) for x in _origin_item(open(path).read()).split()] == origin
        field = pickle.load(open(res.data_file, "rb"))
        assert np.array_equal(np.asarray(field.values), raw.values[[0, -1]])


@pytest.mark.gpu
def test_core_256_streams_bitwise(P, tmp_path):
    from pde_solver_b200 import io
    kw = dict(core_radius=0.3, core_diffusivity=25.0, precond="gmg", snapshot_stride=5, as_arrays=True)
    args = (1.0, 1.0, 1.0, 256, 256, 256, 1.0, 0.0, 20.0, 0.01, 10)
    full = P._solve_heat_3d_raw(*args, **kw)
    with io.open_writer("npz", tmp_path / "core.npz", 3, [256] * 3, [1.0] * 3) as w:
        part = P._solve_heat_3d_raw(*args, stream_to=w, **kw)
    st = P.last_stats()
    assert st["converged"] == 1 and st["levels"] >= 6 and st["solves"] == 10, st
    assert np.array_equal(part.values[-1], full.values[-1])
    with np.load(tmp_path / "core.npz") as z:
        assert np.array_equal(z["t000002"], full.values[-1])
    assert os.path.getsize(tmp_path / "core.npz") > 3 * 257 ** 3 * 8
