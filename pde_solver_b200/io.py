"""Streaming snapshot writers (SURVEY §8f n1): the reference keeps every snapshot as nested Python lists and
pickles them at the end (fenics_mcp_server.py:712, 2200-2207), which is what breaks at 134 M dofs.  These
writers take one snapshot at a time (NumPy array in natural lattice order), so a run never holds more than
one snapshot on the host.

    npz   one standard .npz (zip) file, members  t000000.npy ... , times.npy, coords_*.npy, meta.json
    xdmf  <stem>.xdmf (temporal collection on a 3DCoRectMesh / 2DCoRectMesh, node-centred attribute)
          + <stem>.bin  (raw little-endian float64, one snapshot after another; XDMF "Binary" + Seek)

Both describe the structured grid by origin / spacing / node counts instead of a coordinate list.  The origin
defaults to zeros; the weighted heat solves write their coordinate-space lattice (origin = lo, L = hi - lo, e.g.
(r, theta, phi)) and name it in meta["coordinate_system"]."""
import json
import os
import zipfile

import numpy as np


def _origin(dim, origin):
    return [0.0] * int(dim) if origin is None else [float(v) for v in origin]


class NpzSnapshotWriter:
    def __init__(self, path, dim, n, L, meta=None, origin=None):
        self.path = str(path)
        self.dim, self.n, self.L = int(dim), [int(v) for v in n], [float(v) for v in L]
        self.origin = _origin(dim, origin)
        self.meta = dict(meta or {})
        self.times = []
        self._zip = zipfile.ZipFile(self.path, "w", compression=zipfile.ZIP_STORED, allowZip64=True)

    def _put(self, name, arr):
        with self._zip.open(name + ".npy", "w", force_zip64=True) as f:
            np.lib.format.write_array(f, np.ascontiguousarray(arr), allow_pickle=False)

    def append(self, t, values):
        self._put(f"t{len(self.times):06d}", np.asarray(values, dtype=np.float64))
        self.times.append(float(t))

    def close(self):
        if self._zip is None:
            return self.path
        self._put("times", np.asarray(self.times))
        self._put("shape_nodes", np.asarray([v + 1 for v in self.n], dtype=np.int64))
        self._put("extent", np.asarray(self.L))
        self._put("origin", np.asarray(self.origin))
        with self._zip.open("meta.json", "w") as f:
            f.write(json.dumps({"dim": self.dim, "n": self.n, "L": self.L, "origin": self.origin,
                                "order": "natural (x fastest)", **self.meta}, default=str).encode())
        self._zip.close()
        self._zip = None
        return self.path

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class XdmfSnapshotWriter:
    def __init__(self, path, dim, n, L, name="u", meta=None, origin=None):
        stem = str(path)
        stem = stem[:-5] if stem.endswith(".xdmf") else stem
        self.xdmf_path, self.bin_path = stem + ".xdmf", stem + ".bin"
        self.dim, self.n, self.L = int(dim), [int(v) for v in n], [float(v) for v in L]
        self.origin = _origin(dim, origin)
        self.name = name
        self.meta = dict(meta or {})
        self.times = []
        self._bin = open(self.bin_path, "wb")
        self.nv = int(np.prod([v + 1 for v in self.n]))

    def append(self, t, values):
        a = np.ascontiguousarray(values, dtype="<f8")
        if a.size != self.nv:
            raise ValueError(f"snapshot has {a.size} values, mesh has {self.nv} vertices")
        a.tofile(self._bin)
        self.times.append(float(t))

    def close(self):
        if self._bin is None:
            return self.xdmf_path
        self._bin.close()
        self._bin = None
        d = self.dim
        # XDMF lists the slowest axis first (z y x); pad to at least 2-D for readers
        nodes = [v + 1 for v in self.n][::-1]
        spacing = [l / c for l, c in zip(self.L, self.n)][::-1]
        origin = self.origin[::-1]
        if d == 1:
            nodes, spacing, origin = [1] + nodes, [1.0] + spacing, [0.0] + origin
        dd = max(d, 2)
        topo = "3DCoRectMesh" if dd == 3 else "2DCoRectMesh"
        geo = "ORIGIN_DXDYDZ" if dd == 3 else "ORIGIN_DXDY"
        dims = " ".join(str(v) for v in nodes)
        out = ['<?xml version="1.0" ?>', '<Xdmf Version="3.0">', " <Domain>",
               '  <Grid Name="series" GridType="Collection" CollectionType="Temporal">']
        base = os.path.basename(self.bin_path)
        for k, t in enumerate(self.times):
            out += [f'   <Grid Name="step{k}" GridType="Uniform">', f'    <Time Value="{t:.17g}"/>',
                    f'    <Topology TopologyType="{topo}" Dimensions="{dims}"/>',
                    f'    <Geometry GeometryType="{geo}">',
                    f'     <DataItem Dimensions="{dd}" NumberType="Float" Precision="8" Format="XML">'
                    + " ".join(f"{v:.17g}" for v in origin) + "</DataItem>",
                    f'     <DataItem Dimensions="{dd}" NumberType="Float" Precision="8" Format="XML">'
                    + " ".join(f"{v:.17g}" for v in spacing) + "</DataItem>", "    </Geometry>",
                    f'    <Attribute Name="{self.name}" AttributeType="Scalar" Center="Node">',
                    f'     <DataItem Dimensions="{dims}" NumberType="Float" Precision="8" Format="Binary" '
                    f'Endian="Little" Seek="{k * self.nv * 8}">{base}</DataItem>', "    </Attribute>", "   </Grid>"]
        out += ["  </Grid>", " </Domain>", "</Xdmf>"]
        with open(self.xdmf_path, "w") as f:
            f.write("\n".join(out) + "\n")
        return self.xdmf_path

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def open_writer(fmt, path, dim, n, L, name="u", meta=None, origin=None):
    if fmt == "npz":
        return NpzSnapshotWriter(path, dim, n, L, meta=meta, origin=origin)
    if fmt == "xdmf":
        return XdmfSnapshotWriter(path, dim, n, L, name=name, meta=meta, origin=origin)
    raise ValueError("snapshot format must be 'npz' or 'xdmf'")


def read_npz_series(path):
    """(times, values [Nt][N]) from a file written by NpzSnapshotWriter."""
    with np.load(path) as z:
        times = z["times"]
        vals = np.stack([z[f"t{k:06d}"] for k in range(len(times))])
    return times, vals


def read_xdmf_series(xdmf_path):
    """(times, values [Nt][N]) from the .xdmf/.bin pair written by XdmfSnapshotWriter."""
    import re
    txt = open(xdmf_path).read()
    times = np.array([float(v) for v in re.findall(r'<Time Value="([^"]+)"', txt)])
    m = re.search(r'Format="Binary"[^>]*>([^<]+)<', txt)
    raw = np.fromfile(os.path.join(os.path.dirname(os.path.abspath(xdmf_path)), m.group(1)), dtype="<f8")
    return times, raw.reshape(len(times), -1)
