"""Drop-in boundary: tool names / keyword arguments / defaults equal the reference's (golden JSON made by
tests/golden/make_golden_signatures.py from /root/reference/fenics_mcp_server.py), the C-ABI library
exports every symbol include/pde_b200.h declares, and (GPU) the tools work through MCP."""
import asyncio
import inspect
import json
import os
import pickle
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_signatures.json")))
IN_SCOPE = ["solve_heat_1D", "solve_heat_2D", "solve_heat_3D", "solve_elasticity_1D_static",
            "solve_elasticity_2D_static", "solve_elasticity_3D_static"]


@pytest.fixture(scope="module")
def server():
    import fenics_mcp_server as s
    return s


def test_server_and_tool_names(server):
    assert server.mcp.name == GOLD["server_name"] == "FEniCS-Heat"
    tools = asyncio.run(server.mcp.list_tools())
    assert sorted(t.name for t in tools) == sorted(GOLD["tools"])


@pytest.mark.parametrize("name", sorted(GOLD["tools"]))
def test_tool_signature_matches_reference(server, name):
    fn = getattr(server, name)
    ours = inspect.signature(fn)
    ref = GOLD["tools"][name]["args"]
    assert [p for p in ours.parameters] == [a["name"] for a in ref]
    for a in ref:
        p = ours.parameters[a["name"]]
        if a["has_default"]:
            assert p.default == a["default"], (name, a["name"])
        else:
            assert p.default is inspect.Parameter.empty
    assert ours.return_annotation.__name__ == GOLD["tools"][name]["returns"]


@pytest.mark.parametrize("name", ["_solve_heat_1d_raw", "_solve_heat_2d_raw", "_solve_heat_3d_raw",
                                  "_solve_elasticity_1d_static", "_solve_elasticity_2d_static",
                                  "_solve_elasticity_3d_static", "_solve_heat_1d_cylindrical_raw",
                                  "_solve_heat_1d_spherical_raw", "_solve_heat_2d_cylindrical_raw",
                                  "_solve_heat_2d_spherical_raw", "_solve_heat_3d_spherical_raw"])
def test_raw_solver_signature_is_a_superset(name):
    import pde_solver_b200 as P
    ours = inspect.signature(getattr(P, name))
    ref = GOLD["raw"][name]["args"]
    positional = [p.name for p in ours.parameters.values() if p.kind == p.POSITIONAL_OR_KEYWORD]
    assert positional == [a["name"] for a in ref]          # same names, same order
    for a in ref:
        if a["has_default"]:
            assert ours.parameters[a["name"]].default == a["default"]
    extra = [p for p in ours.parameters.values() if p.kind == p.KEYWORD_ONLY]
    assert all(p.default is not inspect.Parameter.empty for p in extra)   # additions are optional


def test_result_dataclasses_have_reference_fields():
    from pde_solver_b200.fields import PlotResult, SolveResult, TimeSeriesField
    assert list(TimeSeriesField.__dataclass_fields__) == ["coords", "values", "times", "dim", "meta"]
    assert list(SolveResult.__dataclass_fields__) == ["data_file", "dim", "meta"]
    assert list(PlotResult.__dataclass_fields__) == ["html_path"]


def test_cabi_exports_every_declared_symbol():
    import ctypes
    hdr = open(os.path.join(ROOT, "include", "pde_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(pde_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 25
    from pde_solver_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing


def test_cylinder_and_composite_branches_reach_the_cuda_library():
    """geometry_type='cylinder' and core_radius/core_diffusivity are served (reference :512-572 without mshr); on a
    box without a GPU they must fail in the CUDA layer, never fall back to a CPU path."""
    import pde_solver_b200 as P
    from pde_solver_b200 import _lib
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("covered by the gpu parity tests")
    with pytest.raises(_lib.PdeError):
        P._solve_heat_3d_raw(1, 1, 1, 4, 4, 4, 1.0, 0.0, 20.0, 0.01, 1, geometry_type="cylinder", cylinder_radius=0.5)
    with pytest.raises(_lib.PdeError):
        P._solve_heat_3d_raw(1, 1, 1, 4, 4, 4, 1.0, 0.0, 20.0, 0.01, 1, core_radius=0.2, core_diffusivity=5.0)


def test_plot_tool_accepts_solver_pickles(server, tmp_path):
    from pde_solver_b200.fields import TimeSeriesField
    f = TimeSeriesField(coords=[[0, 0, 0], [1, 0, 0], [2, 0, 0]], values=[[0, 1, 2], [1, 2, 3]], times=[0.0, 0.1],
                        dim=1, meta={"name": "temperature", "unit": "°C"})
    p = tmp_path / "heat_1d_deadbeef.pkl"
    pickle.dump(f, open(p, "wb"))
    r = server.plot_time_series_field_from_file(str(p), output_dir=str(tmp_path / "plots"))
    assert os.path.exists(r.html_path) and r.html_path.endswith("heat_1d_deadbeef.html")
    with pytest.raises(ValueError):
        server.plot_time_series_field([[0, 0, 0]], [[1, 2]], [0.0], output_dir=str(tmp_path))


def test_product_path_does_not_import_the_oracle():
    # the oracle is test infrastructure: nothing under the package or the server may reference it
    for base in (os.path.join(ROOT, "pde_solver_b200"), ROOT):
        for fn in os.listdir(base):
            if fn.endswith(".py") and fn not in ("bench.py", "__graft_entry__.py"):
                src = open(os.path.join(base, fn)).read()
                assert "oracle" not in src.replace("# oracle", ""), fn


def test_library_reads_only_the_multi_gpu_and_cell_rhs_switches():
    # kernel variants are compared as separate library builds, not switched at run time: the CUDA library reads the
    # environment only for the multi-GPU halo / hierarchy settings and the cell right-hand-side pass count
    csrc = os.path.join(ROOT, "pde_solver_b200", "csrc")
    read = set()
    for fn in os.listdir(csrc):
        src = open(os.path.join(csrc, fn)).read()
        read |= set(re.findall(r"\b(?:getenv|env_int)\s*\(\s*\"(PDE_B200_\w+)\"", src))
    assert read == {"PDE_B200_HALO", "PDE_B200_HALO_BLOCKS", "PDE_B200_HALO_DEBUG", "PDE_B200_REP_NODES",
                    "PDE_B200_NO_LEAN_HALO", "PDE_B200_CELL_2PASS"}


# ------------------------------------------------------------------ GPU: through MCP
@pytest.mark.gpu
def test_call_tool_in_process(server, tmp_path):
    from oracle import fem_oracle as fo
    args = dict(Lx=1.0, Ly=1.0, Lz=1.0, nx=8, ny=8, nz=8, diffusivity=1.0, T_boundary=0.0, T_initial=20.0, dt=0.01,
                num_steps=4, data_dir=str(tmp_path))
    res = asyncio.run(server.mcp.call_tool("solve_heat_3D", args))
    payload = res[1] if isinstance(res, tuple) else json.loads(res[0].text)
    assert set(payload) == {"data_file", "dim", "meta"} and payload["dim"] == 3
    assert re.fullmatch(r"heat_3d_[0-9a-f]{8}\.pkl", os.path.basename(payload["data_file"]))
    field = pickle.load(open(payload["data_file"], "rb"))
    ref = fo.solve_heat(3, [1, 1, 1], [8, 8, 8], 1.0, T_initial=20.0, dt=0.01, num_steps=4)
    assert np.asarray(field.values).shape == (5, 729) and len(field.times) == 5
    assert isinstance(field.values, list) and isinstance(field.coords[0], list)      # reference layout
    assert fo.rel_l2(np.asarray(field.values)[-1], ref.values[-1]) <= 1e-8
    plot = server.plot_time_series_field_from_file(payload["data_file"], output_dir=str(tmp_path / "plots"))
    assert os.path.exists(plot.html_path)
    res = asyncio.run(server.mcp.call_tool("solve_elasticity_3D_static", dict(
        Lx=1.0, Ly=0.2, Lz=0.2, nx=10, ny=2, nz=2, body_fz=-76518.0, quantity="strain", data_dir=str(tmp_path))))
    payload = res[1] if isinstance(res, tuple) else json.loads(res[0].text)
    assert re.fullmatch(r"elasticity_3d_strain_[0-9a-f]{8}\.pkl", os.path.basename(payload["data_file"]))
    assert payload["meta"]["name"] == "von_mises_strain"


@pytest.mark.gpu
def test_stdio_round_trip(tmp_path):
    """Launch the server the way the orchestrator does (python fenics_mcp_server.py over stdio)."""
    from mcp import ClientSession, StdioServerParameters
    from mcp.client.stdio import stdio_client

    async def go():
        params = StdioServerParameters(command=sys.executable, args=[os.path.join(ROOT, "fenics_mcp_server.py")],
                                       cwd=str(tmp_path))
        async with stdio_client(params) as (r, w):
            async with ClientSession(r, w) as s:
                await s.initialize()
                names = sorted(t.name for t in (await s.list_tools()).tools)
                out = await s.call_tool("solve_heat_1D", dict(length=2.0, nx=100, T_left=20.0, T_right=0.0,
                                                              T_initial=0.0, dt=0.01, num_steps=10))
                return names, out
    names, out = asyncio.run(go())
    assert names == sorted(GOLD["tools"])
    assert not out.isError
    payload = json.loads(out.content[0].text)
    path = payload["data_file"] if os.path.isabs(payload["data_file"]) else os.path.join(str(tmp_path), payload["data_file"])
    field = pickle.load(open(path, "rb"))
    assert len(field.values) == 11 and len(field.values[0]) == 101 and field.meta["pde"] == "heat"


def test_snapshot_writers_round_trip(tmp_path):
    from pde_solver_b200 import io
    n, L = [3, 2, 1], [1.0, 0.5, 0.25]
    nv = 4 * 3 * 2
    snaps = [np.arange(nv, dtype=float) + 100 * k for k in range(3)]
    for fmt in ("npz", "xdmf"):
        with io.open_writer(fmt, tmp_path / f"s.{fmt}", 3, n, L, name="temperature", meta={"pde": "heat"}) as w:
            for k, v in enumerate(snaps):
                w.append(0.1 * k, v)
    t, v = io.read_npz_series(tmp_path / "s.npz")
    assert np.allclose(t, [0, 0.1, 0.2]) and np.array_equal(v, np.stack(snaps))
    t, v = io.read_xdmf_series(str(tmp_path / "s.xdmf"))
    assert np.allclose(t, [0, 0.1, 0.2]) and np.array_equal(v, np.stack(snaps))
    xml = open(tmp_path / "s.xdmf").read()
    from xml.dom import minidom
    minidom.parseString(xml)                                        # well-formed
    assert 'Dimensions="2 3 4"' in xml and 'TopologyType="3DCoRectMesh"' in xml and 'Seek="192"' in xml
    with pytest.raises(ValueError):
        io.XdmfSnapshotWriter(tmp_path / "bad", 3, n, L).append(0.0, np.zeros(5))


@pytest.mark.gpu
def test_streaming_solve_matches_in_memory(server, tmp_path, monkeypatch):
    import pde_solver_b200 as P
    from pde_solver_b200 import io
    full = P._solve_heat_3d_raw(1, 1, 1, 12, 10, 8, 1.0, 0.0, 20.0, 0.01, 6, as_arrays=True)
    with io.open_writer("npz", tmp_path / "a.npz", 3, [12, 10, 8], [1, 1, 1]) as w:
        part = P._solve_heat_3d_raw(1, 1, 1, 12, 10, 8, 1.0, 0.0, 20.0, 0.01, 6, as_arrays=True, stream_to=w,
                                    snapshot_stride=2)
    t, v = io.read_npz_series(tmp_path / "a.npz")
    assert np.allclose(t, [0, 0.02, 0.04, 0.06])
    assert np.array_equal(v, full.values[[0, 2, 4, 6]])            # same kernels, same arithmetic
    assert np.array_equal(part.values, full.values[[0, 6]]) and np.allclose(part.times, [0, 0.06])
    monkeypatch.setenv("PDE_B200_STREAM", "xdmf")
    res = server.solve_heat_2D(nx=8, ny=8, num_steps=3, data_dir=str(tmp_path))
    assert res.meta["snapshots_file"].endswith(".xdmf")
    t, v = io.read_xdmf_series(res.meta["snapshots_file"])
    assert v.shape == (4, 81)


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in _lib.py and the structs of include/pde_b200.h (compiled here as plain C99) agree in size
    and in the offsets of the fields behind which padding can hide."""
    import ctypes as C
    import shutil
    import subprocess
    from pde_solver_b200 import _lib as L
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    pairs = dict(pde_bc="Bc", pde_solver_opts="SolverOpts", pde_stats="Stats", pde_heat_params="HeatParams",
                 pde_wheat_params="WheatParams", pde_elast_params="ElastParams", pde_op_params="OpParams")
    offs = [("pde_wheat_params", "bc"), ("pde_wheat_params", "weight_kind"), ("pde_wheat_params", "core_radius"),
            ("pde_wheat_params", "initial_wavenumber"), ("pde_heat_params", "bc"), ("pde_heat_params", "T_initial"),
            ("pde_op_params", "variant"), ("pde_elast_params", "quantity"), ("pde_elast_params", "area"),
            ("pde_stats", "final_relres"), ("pde_solver_opts", "cheby_ratio")]
    src = ["#include <stdio.h>", "#include <stddef.h>", '#include "pde_b200.h"', "int main(void) {"]
    for cname in pairs:
        src.append(f'  printf("S {cname} %zu\\n", sizeof({cname}));')
    for cname, fld in offs:
        src.append(f'  printf("O {cname} {fld} %zu\\n", offsetof({cname}, {fld}));')
    src += ["  return 0;", "}"]
    cfile = tmp_path / "abi.c"
    cfile.write_text("\n".join(src))
    exe = tmp_path / "abi"
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(cfile), "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout.split("\n")
    for line in filter(None, out):
        t = line.split()
        if t[0] == "S":
            assert C.sizeof(getattr(L, pairs[t[1]])) == int(t[2]), line
        else:
            assert getattr(getattr(L, pairs[t[1]]), t[2]).offset == int(t[3]), line


def test_dof_permutation_hook_is_validated():
    """mesh.set_dof_permutation (SURVEY §8c(2), row a3): only true permutations of the mesh vertices are accepted; the
    arrays it reorders are exercised on the GPU (tests/test_gpu_parity.py::test_dof_permutation_reorders_exports)."""
    import pytest as _pt
    from pde_solver_b200 import mesh
    with _pt.raises(ValueError):
        mesh.set_dof_permutation(2, [2, 2], [0, 1, 2])
    with _pt.raises(ValueError):
        mesh.set_dof_permutation(2, [2, 2], [0] * 9)
    mesh.set_dof_permutation(2, [2, 2], list(range(9))[::-1])
    assert mesh.dof_permutation(2, [2, 2])[0] == 8
    a = np.arange(18).reshape(2, 9)
    assert np.array_equal(mesh.to_dof_order(2, [2, 2], a), a[:, ::-1])
    mesh.set_dof_permutation(2, [2, 2], None)
    assert mesh.dof_permutation(2, [2, 2]) is None
