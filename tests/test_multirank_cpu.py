"""N>1 host-side logic on CPU: slab partition arithmetic (C ABI, host only) and the torchrun plumbing of
bench.py, exercised with world_size-2 gloo process groups (no GPU needed)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("dim,n,world", [(3, [512, 512, 4096], 8), (3, [1280, 256, 256], 8), (3, [64, 64, 64], 2),
                                         (2, [4096, 4096], 4), (3, [16, 16, 33], 2)])
def test_slab_partition_tiles_and_nests(dim, n, world):
    from pde_solver_b200 import _lib
    level = 0
    while True:
        try:
            parts = [_lib.slab_partition(dim, n, r, world, level) for r in range(world)]
        except _lib.PdeError:
            assert level > 0          # level 0 always exists
            break
        nzg = parts[0][2]
        assert nzg == n[dim - 1] // 2 ** level + 1
        # disjoint cover of [0, nzg), rank order = plane order, every rank owns at least one plane
        z = 0
        for z0, nzl, g in parts:
            assert z0 == z and nzl >= 1 and g == nzg
            z += nzl
        assert z == nzg
        if level > 0:
            # nesting: rank r's coarse slab starts at half of its fine start, so restriction of owned fine planes
            # (plus one ghost plane) lands on owned coarse planes
            for (z0c, nzlc, _), (z0f, nzlf, _) in zip(parts, prev):
                assert 2 * z0c == z0f and 2 * (z0c + nzlc - 1) <= z0f + nzlf
        prev = parts
        level += 1
    assert level >= 1


def test_slab_partition_rejects_bad_arguments():
    from pde_solver_b200 import _lib
    with pytest.raises(_lib.PdeError):
        _lib.slab_partition(3, [8, 8, 4], 0, 8)        # fewer cell layers than ranks
    with pytest.raises(_lib.PdeError):
        _lib.slab_partition(3, [8, 8, 8], 2, 2)        # rank out of range
    with pytest.raises(_lib.PdeError):
        _lib.slab_partition(1, [100], 0, 4)            # 1-D rods are never slab-partitioned


WORKER = r"""
import os, sys, json
import numpy as np
import torch.distributed as dist
sys.path.insert(0, os.environ["REPO_ROOT"])
from pde_solver_b200 import _lib
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n = [6, 5, 8]
z0, nzl, nzg = _lib.slab_partition(3, n, rank, world)
plane = (n[0] + 1) * (n[1] + 1)
glob = np.arange(plane * nzg, dtype=np.float64)                 # a global nodal field, natural order
mine = glob[z0 * plane:(z0 + nzl) * plane].copy()
# halo exchange as the library does it (first/last owned plane to the z-neighbours), here over gloo
import torch
lo = torch.zeros(plane, dtype=torch.float64); hi = torch.zeros(plane, dtype=torch.float64)
reqs = []
if rank > 0:
    reqs += [dist.isend(torch.from_numpy(mine[:plane].copy()), rank - 1), dist.irecv(lo, rank - 1)]
if rank < world - 1:
    reqs += [dist.isend(torch.from_numpy(mine[-plane:].copy()), rank + 1), dist.irecv(hi, rank + 1)]
for r in reqs: r.wait()
ok = True
if rank > 0: ok = ok and np.array_equal(lo.numpy(), glob[(z0 - 1) * plane:z0 * plane])
if rank < world - 1: ok = ok and np.array_equal(hi.numpy(), glob[(z0 + nzl) * plane:(z0 + nzl + 1) * plane])
# gather the slabs in rank order: must reproduce the global field (what bench.py / mgpu_check.py rely on)
parts = [None] * world
dist.all_gather_object(parts, mine)
ok = ok and np.array_equal(np.concatenate(parts), glob)
flags = [None] * world
dist.all_gather_object(flags, bool(ok))
if rank == 0: print(json.dumps({"ok": all(flags), "world": world}))
dist.destroy_process_group()
"""


def _torchrun(args, env_extra=None, timeout=300):
    env = dict(os.environ, REPO_ROOT=ROOT, OMP_NUM_THREADS="1")
    env.update(env_extra or {})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(29600 + os.getpid() % 300)] + args
    return subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout,
                          cwd=ROOT)


def test_gloo_world2_slabs_and_halos(tmp_path):
    w = tmp_path / "worker.py"
    w.write_text(WORKER)
    r = _torchrun([str(w)])
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line) == {"ok": True, "world": 2}


def test_reference_arm_under_torchrun_prints_once():
    r = _torchrun(["bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                      # rank 0 alone runs and prints
    assert [l for l in r.stdout.splitlines() if l.strip()] == lines      # stdout carries the JSON line and nothing else
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0


def test_tool_pool_wire_format_and_slab_offsets():
    """pde_solver_b200/multi.py (PDE_B200_GPUS=N): length-prefixed pickle frames over pipes; every rank's slab is a
    contiguous range of the natural (z-slowest) vertex order and the ranges tile the global array exactly."""
    import io

    from pde_solver_b200 import _lib, multi
    buf = io.BytesIO()
    msgs = [{"kind": "heat", "p": b"\\x00" * 100, "nsnap": 3, "nv": 17, "shm": ["a"]}, ("ok", ({"iters_total": 5}, [0.0, 0.1]))]
    for m in msgs:
        multi._send(buf, m)
    buf.seek(0)
    assert [multi._recv(buf) for _ in msgs] == msgs
    with pytest.raises(EOFError):
        multi._recv(buf)
    for n, world in (([8, 6, 16], 2), ([5, 4, 24], 4), ([3, 3, 17], 8)):
        plane = (n[0] + 1) * (n[1] + 1)
        nxt = 0
        for r in range(world):
            off, nloc, nglob = multi._slab(n, r, world)
            assert off == nxt and nloc > 0 and nglob == plane * (n[2] + 1)
            z0, nzl, nzg = _lib.slab_partition(3, n, r, world)
            assert (off, nloc) == (z0 * plane, nzl * plane)
            nxt = off + nloc
        assert nxt == plane * (n[2] + 1)
    assert not multi.usable(16, world=1) and multi.usable(16, world=4) and not multi.usable(15, world=4)


def test_requested_gpus_beyond_the_visible_devices_is_refused(monkeypatch):
    """A worker that cannot open its GPU would leave rank 0 waiting in the communicator set-up: the tool layer refuses
    PDE_B200_GPUS > pde_device_count() up front (and never silently falls back to fewer GPUs or to the CPU)."""
    from pde_solver_b200 import _lib, multi
    have = _lib.device_count()
    assert have >= 0
    monkeypatch.setenv("PDE_B200_GPUS", str(have + 2))
    with pytest.raises(_lib.PdeError, match="PDE_B200_GPUS"):
        multi.usable(64)
    monkeypatch.setenv("PDE_B200_GPUS", "1")
    assert not multi.usable(64)
    monkeypatch.setenv("PDE_B200_GPUS", "not-a-number")
    assert multi.requested_gpus() == 1


def test_tool_pool_reports_a_rank_without_a_device_instead_of_hanging(monkeypatch):
    """Pool start-up handshake: every worker says whether it holds a device context BEFORE rank 0 enters the NCCL
    communicator set-up.  Here the spawned rank sees no GPU and cannot create its context: the pool must raise with the
    rank's own message and reap the worker - not block in the collective."""
    import time

    from pde_solver_b200 import _lib, multi
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")          # the worker inherits it, also on a machine with GPUs

    class FakeContext:                       # rank 0 'has' a device; its comm_init must never be reached
        def __init__(self, device):
            self.device = device

        def comm_init(self, *a):
            raise AssertionError("entered the collective although a rank reported no device")

    monkeypatch.setattr(_lib, "Context", FakeContext)
    monkeypatch.setattr(_lib, "nccl_unique_id", lambda path: b"\0" * 128)
    monkeypatch.setattr(_lib, "nccl_library_path", lambda: "libnccl.so.2")
    t0 = time.time()
    with pytest.raises(_lib.PdeError, match=r"rank 1 \(device 1\).*no CUDA device"):
        multi.Pool(2)
    assert time.time() - t0 < 120


def test_tool_pool_start_up_and_shutdown_handshake(monkeypatch, tmp_path):
    """The success path of the same handshake without a GPU: the spawned rank imports a stand-in device context (a
    sitecustomize on its PYTHONPATH patches _lib.Context before multi.py runs), so 'ctx' -> collective -> 'ready' ->
    'quit' runs over the real pipes and the worker exits cleanly."""
    from pde_solver_b200 import _lib, multi
    (tmp_path / "sitecustomize.py").write_text(
        "import pde_solver_b200._lib as L\n"
        "class C:\n"
        "    def __init__(self, device): self.device = device\n"
        "    def comm_init(self, rank, world, uid, path):\n"
        "        assert (rank, world, len(uid)) == (1, 2, 128)\n"
        "L.Context = C\n")
    calls = []

    class FakeContext:
        def __init__(self, device):
            calls.append(("ctx", device))

        def comm_init(self, rank, world, uid, path):
            calls.append(("comm", rank, world))

    monkeypatch.setattr(_lib, "Context", FakeContext)
    monkeypatch.setattr(_lib, "nccl_unique_id", lambda path: b"\1" * 128)
    monkeypatch.setattr(_lib, "nccl_library_path", lambda: "libnccl.so.2")
    monkeypatch.setenv("PYTHONPATH", str(tmp_path))
    p = multi.Pool(2)
    assert calls == [("ctx", 0), ("comm", 0, 2)] and len(p.procs) == 1 and not p.broken
    pr = p.procs[0]
    p.close()
    assert pr.returncode == 0 and p.procs == []
