"""ctypes binding of libpde_b200.so (C ABI: include/pde_b200.h).  Plumbing only."""
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PDE_B200_LIB") or os.path.join(_HERE, "libpde_b200.so")  # override: A/B kernel builds


class PdeError(RuntimeError):
    pass


class Bc(C.Structure):
    _fields_ = [("face_on", C.c_int32 * 6), ("face_val", C.c_double * 6), ("side_excludes_xends", C.c_int32)]


class SolverOpts(C.Structure):
    _fields_ = [("rtol", C.c_double), ("max_iters", C.c_int32), ("precond", C.c_int32),
                ("cheby_degree", C.c_int32), ("check_every", C.c_int32), ("cheby_ratio", C.c_double),
                ("verify_residual", C.c_int32), ("reserved", C.c_int32 * 3)]


class Stats(C.Structure):
    _fields_ = [("ndofs", C.c_int64), ("iters_total", C.c_int64), ("solves", C.c_int32),
                ("converged", C.c_int32), ("levels", C.c_int32), ("reserved", C.c_int32),
                ("final_relres", C.c_double), ("true_relres", C.c_double), ("solve_ms", C.c_double),
                ("setup_ms", C.c_double), ("launches", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class HeatParams(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n", C.c_int32 * 3), ("L", C.c_double * 3), ("diffusivity", C.c_double),
                ("dt", C.c_double), ("num_steps", C.c_int32), ("steady", C.c_int32),
                ("source_value", C.c_double), ("initial_type", C.c_int32), ("snapshot_stride", C.c_int32),
                ("T_initial", C.c_double), ("initial_amplitude", C.c_double),
                ("initial_wavenumber", C.c_double), ("bc", Bc)]


class ElastParams(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n", C.c_int32 * 3), ("L", C.c_double * 3), ("E", C.c_double),
                ("nu", C.c_double), ("body", C.c_double * 3), ("quantity", C.c_int32),
                ("plane_stress", C.c_int32), ("area", C.c_double)]


class WheatParams(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n", C.c_int32 * 3), ("lo", C.c_double * 3), ("hi", C.c_double * 3),
                ("weight_rpow", C.c_int32), ("weight_sin_axis1", C.c_int32), ("weight_degree", C.c_int32),
                ("steady", C.c_int32), ("diffusivity", C.c_double), ("dt", C.c_double), ("num_steps", C.c_int32),
                ("snapshot_stride", C.c_int32), ("source_value", C.c_double), ("T_initial", C.c_double), ("bc", Bc),
                ("weight_kind", C.c_int32), ("has_core", C.c_int32), ("core_radius", C.c_double),
                ("core_diffusivity", C.c_double), ("initial_type", C.c_int32), ("reserved0", C.c_int32),
                ("initial_amplitude", C.c_double), ("initial_wavenumber", C.c_double)]


class OpParams(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("n", C.c_int32 * 3), ("L", C.c_double * 3),
                ("alpha", C.c_double), ("beta", C.c_double), ("lam", C.c_double), ("mu", C.c_double),
                ("bc", Bc), ("variant", C.c_int32)]


MG_MAX_LEVELS = 16
MG_PATHS = {"first2": 1, "heat_post2": 2, "post2_r1": 4, "resid_restrict": 8}


class MgInfo(C.Structure):
    _fields_ = [("levels", C.c_int32), ("n_dense", C.c_int32), ("graph", C.c_int32), ("reserved", C.c_int32),
                ("n", (C.c_int32 * 3) * MG_MAX_LEVELS), ("lmax", C.c_double * MG_MAX_LEVELS),
                ("paths", C.c_uint32 * MG_MAX_LEVELS)]

    def as_dict(self):
        nl = self.levels
        return {"levels": nl, "n_dense": self.n_dense, "graph": self.graph,
                "n": [list(self.n[l]) for l in range(nl)], "lmax": [self.lmax[l] for l in range(nl)],
                "paths": [int(self.paths[l]) for l in range(nl)]}


PRECOND = {"jacobi": 0, "gmg": 1, "auto": 2}
IC = {"constant": 0, "zero": 1, "cosine": 2, "sine": 3, "array": 4}
OP = {"heat": 0, "mass": 1, "stiffness": 2, "elasticity": 3}

_lib = None
_lock = threading.Lock()


def lib():
    """Load the CUDA library; fail loudly if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise PdeError(
                f"{LIB_PATH} is missing: build it with `python pde_solver_b200/build.py` "
                "(this package has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.pde_last_error.restype = C.c_char_p
        L.pde_ctx_launch_count.restype = C.c_int64
        L.pde_heat_local_nverts.restype = C.c_int64
        L.pde_wheat_local_nverts.restype = C.c_int64
        L.pde_solver_opts_default.restype = None
        for name in ("pde_ctx_create", "pde_ctx_destroy", "pde_ctx_sync", "pde_timer_start", "pde_timer_stop",
                     "pde_nccl_unique_id", "pde_comm_init", "pde_mesh_counts", "pde_mesh_coords",
                     "pde_mesh_cells", "pde_dofmap_cells", "pde_boundary_mask", "pde_heat_solve",
                     "pde_heat_open", "pde_heat_set_state", "pde_heat_step", "pde_heat_get_state",
                     "pde_heat_advance_batch", "pde_halo_check",
                     "pde_heat_close", "pde_elasticity_solve", "pde_op_table", "pde_op_apply", "pde_op_bench", "pde_op_sweep", "pde_op_bench_mode", "pde_comm_info", "pde_device_count",
                     "pde_op_solve", "pde_version", "pde_host_alloc", "pde_host_free", "pde_slab_partition", "pde_op_manufactured", "pde_halo_bench", "pde_wheat_solve", "pde_wheat_level_coefs",
                     "pde_wheat_open", "pde_wheat_set_state", "pde_wheat_step", "pde_wheat_get_state", "pde_wheat_close",
                     "pde_mesh_coords_box", "pde_op_vcycle", "pde_wheat_vcycle"):
            getattr(L, name).restype = C.c_int
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise PdeError(lib().pde_last_error().decode("utf-8", "replace"))


def ptr(a, ctype=C.c_void_p):
    return a.ctypes.data_as(ctype) if a is not None else None


def i3(vals):
    v = list(vals) + [0] * (3 - len(vals))
    return (C.c_int32 * 3)(*[int(x) for x in v])


def d3(vals, fill=1.0):
    v = list(vals) + [fill] * (3 - len(vals))
    return (C.c_double * 3)(*[float(x) for x in v])


def make_bc(faces=None, side_excludes_xends=False):
    """faces: {face_index: value}, face order x0,x1,y0,y1,z0,z1 of the user's axes."""
    bc = Bc()
    for f, v in (faces or {}).items():
        bc.face_on[f] = 1
        bc.face_val[f] = float(v)
    bc.side_excludes_xends = 1 if side_excludes_xends else 0
    return bc


def make_opts(rtol=1e-10, precond="auto", max_iters=100000, cheby_degree=2, check_every=10, cheby_ratio=8.0,
              verify=True):
    o = SolverOpts()
    lib().pde_solver_opts_default(C.byref(o))
    o.rtol = float(rtol)
    o.precond = PRECOND[precond] if isinstance(precond, str) else int(precond)
    o.max_iters = int(max_iters)
    o.cheby_degree = int(cheby_degree)
    o.check_every = int(check_every)
    o.cheby_ratio = float(cheby_ratio)
    o.verify_residual = 0 if verify else -1     # recompute ||b - A x||/||b|| after the last solve of a call
    return o


class Context:
    """One GPU.  Under torchrun each rank creates one (device = LOCAL_RANK)."""

    def __init__(self, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", os.environ.get("PDE_B200_DEVICE", "0")))
        self.handle = C.c_void_p()
        check(lib().pde_ctx_create(int(device), C.byref(self.handle)))
        self.device = int(device)
        self.rank, self.world = 0, 1

    def comm_init(self, rank, world, uid_bytes, libnccl_path=None):
        buf = (C.c_char * 128).from_buffer_copy(uid_bytes)
        path = libnccl_path.encode() if libnccl_path else None
        check(lib().pde_comm_init(self.handle, int(rank), int(world), buf, path))
        self.rank, self.world = int(rank), int(world)

    def launches(self):
        return int(lib().pde_ctx_launch_count(self.handle))

    def sync(self):
        check(lib().pde_ctx_sync(self.handle))

    def timer_start(self):
        check(lib().pde_timer_start(self.handle))

    def timer_stop(self):
        ms = C.c_double()
        check(lib().pde_timer_stop(self.handle, C.byref(ms)))
        return ms.value

    def close(self):
        if self.handle:
            lib().pde_ctx_destroy(self.handle)
            self.handle = C.c_void_p()


_ctx = None


def default_context():
    global _ctx
    if _ctx is None:
        _ctx = Context()
    return _ctx


def device_count():
    """CUDA devices visible to this process (0 without a GPU)."""
    n = C.c_int32(0)
    check(lib().pde_device_count(C.byref(n)))
    return int(n.value)


def nccl_library_path():
    """torch's bundled libnccl.so.2 if present (the one torch.distributed itself uses)."""
    try:
        import nvidia.nccl as _n
        base = list(_n.__path__)[0]
        p = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(p):
            return p
    except Exception:
        pass
    return None


def nccl_unique_id(libnccl_path=None):
    buf = (C.c_char * 128)()
    path = libnccl_path.encode() if libnccl_path else None
    check(lib().pde_nccl_unique_id(path, buf))
    return bytes(buf)


def mesh_counts(dim, n):
    nv, nc = C.c_int64(), C.c_int64()
    check(lib().pde_mesh_counts(int(dim), i3(n), C.byref(nv), C.byref(nc)))
    return nv.value, nc.value


def slab_partition(dim, n, rank, world, level=0):
    """(z0, nzl, nzg): vertex planes [z0, z0+nzl) of nzg that `rank` owns on multigrid `level` (host only)."""
    z0, nzl, nzg = C.c_int32(), C.c_int32(), C.c_int32()
    check(lib().pde_slab_partition(int(dim), i3(n), int(rank), int(world), int(level), C.byref(z0), C.byref(nzl),
                                   C.byref(nzg)))
    return z0.value, nzl.value, nzg.value


def op_params(kind, dim, n, L, alpha=1.0, beta=1.0, lam=0.0, mu=0.0, bc=None, variant=0):
    p = OpParams()
    p.kind = OP[kind] if isinstance(kind, str) else int(kind)
    p.dim = int(dim)
    p.n = i3(n)
    p.L = d3(L)
    p.alpha, p.beta, p.lam, p.mu = float(alpha), float(beta), float(lam), float(mu)
    p.bc = bc if bc is not None else Bc()
    p.variant = int(variant)
    return p


def op_table(p):
    nc = C.c_int32()
    check(lib().pde_op_table(C.byref(p), None, C.byref(nc)))
    t = np.zeros((27, 15, nc.value, nc.value))
    check(lib().pde_op_table(C.byref(p), ptr(t), C.byref(nc)))
    return t


def op_apply(ctx, p, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty_like(x)
    check(lib().pde_op_apply(ctx.handle, C.byref(p), ptr(x), ptr(y)))
    return y


def op_sweep(ctx, p, mode, x, b=None, xprev=None, c1=0.0, c2=0.0):
    """One smoother / residual kernel (see pde_op_sweep in include/pde_b200.h); returns (y, dots)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
    xprev = None if xprev is None else np.ascontiguousarray(xprev, dtype=np.float64)
    y = np.empty_like(x)
    dots = np.zeros(2)
    check(lib().pde_op_sweep(ctx.handle, C.byref(p), int(mode), C.c_double(c1), C.c_double(c2), ptr(x),
                             ptr(b) if b is not None else None, ptr(xprev) if xprev is not None else None, ptr(y),
                             ptr(dots)))
    return y, dots


def op_bench_mode(ctx, p, mode, reps=20, warmup=3):
    ms, nd = C.c_double(), C.c_int64()
    check(lib().pde_op_bench_mode(ctx.handle, C.byref(p), int(mode), int(reps), int(warmup), C.byref(ms), C.byref(nd)))
    return ms.value, nd.value


def op_solve(ctx, p, b, opts=None):
    b = np.ascontiguousarray(b, dtype=np.float64)
    x = np.empty_like(b)
    st = Stats()
    o = opts if opts is not None else make_opts()
    check(lib().pde_op_solve(ctx.handle, C.byref(p), C.byref(o), ptr(b), ptr(x), C.byref(st)))
    return x, st.as_dict()


def _vcycle(fn, b, ncycles):
    b = np.ascontiguousarray(b, dtype=np.float64)
    z_first, z_last = np.empty_like(b), np.empty_like(b)
    bz = C.c_double()
    info = MgInfo()
    check(fn(int(ncycles), ptr(b), ptr(z_first), ptr(z_last), C.byref(bz), C.byref(info)))
    return z_first, z_last, bz.value, info.as_dict()


def op_vcycle(ctx, p, b, opts=None, ncycles=3):
    """The GMG V-cycle of op_solve applied `ncycles` times to b [ncomp][nverts] (see pde_op_vcycle in
    include/pde_b200.h); returns (z of cycle 1, z of the last cycle, fused b.z of the last cycle, info dict)."""
    o = C.byref(opts) if opts is not None else None
    return _vcycle(lambda *a: lib().pde_op_vcycle(ctx.handle, C.byref(p), o, *a), b, ncycles)


def wheat_vcycle(ctx, p, b, ncycles=3):
    """As op_vcycle for the weighted operators of WheatParams and their Galerkin hierarchy."""
    return _vcycle(lambda *a: lib().pde_wheat_vcycle(ctx.handle, C.byref(p), *a), b, ncycles)


def comm_info(ctx):
    """{"halo_path": none / nccl send-recv / peer-memory kernel, "halo_exchanges": n, "allreduces": n} so far."""
    hp, ne, na = C.c_int32(), C.c_int64(), C.c_int64()
    check(lib().pde_comm_info(ctx.handle, C.byref(hp), C.byref(ne), C.byref(na)))
    return {"halo_path": {0: "none", 1: "nccl send/recv", 2: "peer-memory mailbox kernel (cudaIpc over NVLink)"}[hp.value],
            "halo_exchanges": ne.value, "allreduces": na.value}


def halo_check(ctx, dim, n, ncomp=1, depth=1, reps=4):
    """Number of ghost entries that differ from the neighbours' values after `reps` exchanges (0 = correct)."""
    bad = C.c_int64(0)
    check(lib().pde_halo_check(ctx.handle, int(dim), i3(n), int(ncomp), int(depth), int(reps), C.byref(bad)))
    return int(bad.value)


def halo_bench(ctx, dim, n, ncomp=1, reps=50):
    """(ms per halo exchange, bytes this rank sends per exchange) over NCCL send/recv."""
    ms, nb = C.c_double(), C.c_int64()
    check(lib().pde_halo_bench(ctx.handle, int(dim), i3(n), int(ncomp), int(reps), C.byref(ms), C.byref(nb)))
    return ms.value, nb.value


def op_manufactured(ctx, p, opts=None):
    """Device-resident manufactured-solution check: (relative L2 error of the solve, stats)."""
    err = C.c_double()
    st = Stats()
    o = opts if opts is not None else make_opts()
    check(lib().pde_op_manufactured(ctx.handle, C.byref(p), C.byref(o), C.byref(err), C.byref(st)))
    return err.value, st.as_dict()


def op_bench(ctx, p, reps=20, warmup=3):
    ms, nd = C.c_double(), C.c_int64()
    check(lib().pde_op_bench(ctx.handle, C.byref(p), int(reps), int(warmup), C.byref(ms), C.byref(nd)))
    return ms.value, nd.value


class PinnedArray:
    """float64 NumPy view over cudaHostAlloc'ed memory (for the H2D/D2H legs of a step)."""

    def __init__(self, n):
        self.ptr = C.c_void_p()
        check(lib().pde_host_alloc(C.c_uint64(int(n) * 8), C.byref(self.ptr)))
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_double)), shape=(int(n),))

    def free(self):
        if self.ptr:
            self.array = None
            lib().pde_host_free(self.ptr)
            self.ptr = C.c_void_p()


def heat_params(dim, n, L, diffusivity, dt, T_initial=0.0, bc=None, source_value=0.0, steady=False, num_steps=0,
                snapshot_stride=1, initial_type="constant", initial_amplitude=0.0, initial_wavenumber=0.0):
    """HeatParams (pde_heat_params) of a box heat problem; the defaults are those of a bare HeatStepper."""
    p = HeatParams()
    p.dim = int(dim)
    p.n = i3(n)
    p.L = d3(L)
    p.diffusivity = float(diffusivity)
    p.dt = float(dt)
    p.num_steps = int(num_steps)
    p.steady = 1 if steady else 0
    p.source_value = float(source_value)
    p.initial_type = IC.get(initial_type, IC["constant"])
    p.snapshot_stride = int(snapshot_stride)
    p.T_initial = float(T_initial)
    p.initial_amplitude = float(initial_amplitude)
    p.initial_wavenumber = float(initial_wavenumber)
    p.bc = bc if bc is not None else Bc()
    return p


class Stepper:
    """Device-resident backward-Euler stepper of one solver family (pde_<kind>_open / set_state / step / get_state /
    close): the state stays in HBM between steps."""

    def __init__(self, kind, ctx, params, opts=None):
        self.kind = kind
        self.ctx = ctx
        self.handle = C.c_void_p()
        o = opts if opts is not None else make_opts()
        check(self._fn("open")(ctx.handle, C.byref(params), C.byref(o), C.byref(self.handle)))
        self.nloc = int(self._fn("local_nverts")(self.handle))

    def _fn(self, name):
        return getattr(lib(), f"pde_{self.kind}_{name}")

    def step(self, nsteps=1):
        st = Stats()
        check(self._fn("step")(self.handle, int(nsteps), C.byref(st)))
        return st.as_dict()

    def set_state(self, u):
        check(self._fn("set_state")(self.handle, ptr(u)))

    def get_state(self, out):
        check(self._fn("get_state")(self.handle, ptr(out)))
        return out

    def close(self):
        if self.handle:
            self._fn("close")(self.handle)
            self.handle = C.c_void_p()


class HeatStepper(Stepper):
    """Stepper of the box heat solve (pde_heat_*)."""

    def __init__(self, ctx, dim, n, L, diffusivity, dt, T_initial=0.0, bc=None, source_value=0.0, steady=False,
                 opts=None):
        super().__init__("heat", ctx, heat_params(dim, n, L, diffusivity, dt, T_initial=T_initial, bc=bc,
                                                  source_value=source_value, steady=steady), opts)

    def advance_batch(self, inputs, outputs):
        """Independent one-step advances inputs[k] -> outputs[k] (host arrays of nloc float64, ideally pinned):
        uploads, solves and downloads are pipelined on three streams (pde_heat_advance_batch)."""
        n = len(inputs)
        if len(outputs) != n:
            raise ValueError("inputs and outputs differ in length")
        pin = (C.c_void_p * max(1, n))(*[a.ctypes.data for a in inputs])
        pout = (C.c_void_p * max(1, n))(*[a.ctypes.data for a in outputs])
        st = Stats()
        check(lib().pde_heat_advance_batch(self.handle, n, pin, pout, C.byref(st)))
        return st.as_dict()


class WheatStepper(Stepper):
    """Stepper of the coordinate-weighted heat solve (pde_wheat_*) for a filled WheatParams."""

    def __init__(self, ctx, params, opts=None):
        super().__init__("wheat", ctx, params, opts)
