"""ctypes front-end over libpmg.so (the C ABI of include/pmg.h).

The product is the C/C++/CUDA library; this module is glue for the tests and bench.py.  It never
computes anything itself and has NO fallback: if libpmg.so is missing or no B200 is visible, calls
raise.  (The directory name contains hyphens, so import it through the repo-root shim `pmg_b200`.)

Reference surface mirrored here (see include/pmg.hpp for the C++ twin):
  Solver.cycle / Solver.solve   <- MultigridSolver::{v,w,f}_cycle + the runner loop
                                   (2_part_MG/MultiGrid.hpp:57-183, MultiGridTestRunner.hpp:190-212)
  jacobi / residual / restrict_fw / prolong_add / norm2
                                <- class Parallel + DynamicGridUtils
                                   (3_part_parallel/Parallel_Method.cu:144-199, DynamicGridUtils.hpp:21-69)
"""
import ctypes
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpmg.so")

V, W, F, FMG = 0, 1, 2, 3
PROLONG_REFERENCE, PROLONG_FULL = 0, 1
ENGINE_FUSED, ENGINE_OPERATOR = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
NORM_TREE, NORM_SEQUENTIAL = 0, 1
SMOOTHER_JACOBI, SMOOTHER_RBGS, SMOOTHER_GS_LEX, SMOOTHER_CHEBYSHEV = 0, 1, 2, 3
OK = 0
STATUS_NAMES = {0: "PMG_OK", 1: "PMG_ERR_INVALID", 2: "PMG_ERR_CUDA", 3: "PMG_ERR_NO_DEVICE",
                4: "PMG_ERR_ALLOC", 5: "PMG_ERR_COMM", 6: "PMG_ERR_UNSUPPORTED"}


class PmgError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))
        self.status = status


class Config(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int), ("nu1", ctypes.c_int), ("nu2", ctypes.c_int),
                ("omega", ctypes.c_double), ("gamma", ctypes.c_int), ("n_coarse", ctypes.c_int),
                ("coarse_sweeps", ctypes.c_int), ("fmg_sweeps", ctypes.c_int),
                ("prolong_mode", ctypes.c_int), ("engine", ctypes.c_int),
                ("smoother_eps", ctypes.c_double), ("device", ctypes.c_int), ("use_graph", ctypes.c_int),
                ("rank", ctypes.c_int), ("n_ranks", ctypes.c_int), ("agglomerate_below", ctypes.c_int),
                ("norm_mode", ctypes.c_int), ("smoother", ctypes.c_int), ("smoother_fp32", ctypes.c_int), ("reserved", ctypes.c_int * 5)]


# every symbol include/pmg.h declares (tests/test_abi.py checks the library exports all of them)
ABI_SYMBOLS = [
    "pmg_version", "pmg_last_error", "pmg_status_string", "pmg_config_default", "pmg_kernel_launches",
    "pmg_create", "pmg_destroy", "pmg_set_rhs", "pmg_set_guess", "pmg_get_solution", "pmg_zero_guess",
    "pmg_stage_rhs", "pmg_commit_rhs", "pmg_fetch_solution_begin", "pmg_fetch_solution_wait",
    "pmg_set_rhs_sine", "pmg_residual_norm", "pmg_cycle", "pmg_restrict_to_level", "pmg_f_cycle_from", "pmg_solve", "pmg_pcg", "pmg_last_device_ms", "pmg_stream",
    "pmg_jacobi", "pmg_gauss_seidel", "pmg_residual", "pmg_restrict_fw", "pmg_prolong_add", "pmg_diff_norm2", "pmg_norm2", "pmg_release_scratch",
    "pmg_device_alloc", "pmg_device_free", "pmg_host_alloc_pinned", "pmg_host_free_pinned", "pmg_memcpy",
    "pmg_device_synchronize", "pmg_device_count",
    "pmg_comm_unique_id", "pmg_comm_init", "pmg_comm_finalize", "pmg_partition_rows",
]

_lib = None


def build():
    """Compile libpmg.so for sm_100a with the package Makefile (nvcc cross-compiles without a GPU)."""
    subprocess.run(["make", "-s", "-C", _HERE, "-j4"], check=True)


def lib():
    """The loaded library.  Fails loudly when the CUDA build is missing -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libpmg.so is not built (%s): run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` or `make -C %s`; there is no CPU fallback" % (LIB_PATH, _HERE))
    L = ctypes.CDLL(LIB_PATH)
    vp, dp, i, d, sz = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t
    pd = ctypes.POINTER(ctypes.c_double)
    pi = ctypes.POINTER(ctypes.c_int)
    L.pmg_version.restype = ctypes.c_char_p
    L.pmg_last_error.restype = ctypes.c_char_p
    L.pmg_status_string.restype = ctypes.c_char_p
    L.pmg_status_string.argtypes = [i]
    L.pmg_config_default.restype = None
    L.pmg_config_default.argtypes = [ctypes.POINTER(Config), i]
    L.pmg_kernel_launches.restype = ctypes.c_ulonglong
    L.pmg_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(vp)]
    L.pmg_destroy.restype = None
    L.pmg_destroy.argtypes = [vp]
    for name in ("pmg_set_rhs", "pmg_set_guess", "pmg_get_solution"):
        getattr(L, name).argtypes = [vp, dp, i]
    L.pmg_zero_guess.argtypes = [vp]
    L.pmg_set_rhs_sine.argtypes = [vp]
    L.pmg_residual_norm.argtypes = [vp, pd]
    L.pmg_cycle.argtypes = [vp, i, pd]
    L.pmg_solve.argtypes = [vp, i, d, i, pd, pi]
    L.pmg_last_device_ms.argtypes = [vp, pd]
    L.pmg_stream.restype = vp
    L.pmg_stream.argtypes = [vp]
    L.pmg_jacobi.argtypes = [dp, dp, i, i, d, d, i, dp, vp]
    L.pmg_residual.argtypes = [dp, dp, dp, i, i, d, pd, vp]
    L.pmg_restrict_fw.argtypes = [dp, dp, i, i, vp]
    L.pmg_prolong_add.argtypes = [dp, dp, i, i, i, vp]
    L.pmg_norm2.argtypes = [dp, sz, pd, vp]
    L.pmg_device_alloc.argtypes = [ctypes.POINTER(vp), sz]
    L.pmg_device_free.argtypes = [vp]
    L.pmg_host_alloc_pinned.argtypes = [ctypes.POINTER(vp), sz]
    L.pmg_host_free_pinned.argtypes = [vp]
    L.pmg_memcpy.argtypes = [vp, vp, sz, i, i]
    L.pmg_partition_rows.argtypes = [i, i, i, pi, pi]
    L.pmg_comm_unique_id.argtypes = [ctypes.c_char_p]
    L.pmg_comm_init.argtypes = [ctypes.c_char_p, i, i, i]
    L.pmg_smooth.argtypes = [vp, i, i]
    L.pmg_bench_pass.argtypes = [vp, i, i, i, pd]
    L.pmg_fused_set_variant.restype = None
    L.pmg_fused_set_variant.argtypes = [i]
    L.pmg_fused_num_variants.restype = i
    L.pmg_fused_set_deep_prefetch_below.restype = None
    L.pmg_fused_set_deep_prefetch_below.argtypes = [i]
    L.pmg_fused_set_halo_prologue.restype = None
    L.pmg_fused_set_halo_prologue.argtypes = [i]
    L.pmg_small_vcycle_set_version.restype = None
    L.pmg_small_vcycle_set_version.argtypes = [i]
    L.pmg_small_vcycle_version.restype = i
    L.pmg_fused_set_min_chunk_rows.restype = None
    L.pmg_fused_set_min_chunk_rows.argtypes = [i]
    _lib = L
    return L


def check(status):
    if status != OK:
        raise PmgError(status, lib().pmg_last_error().decode())


def device_count():
    return lib().pmg_device_count()


def kernel_launches():
    return int(lib().pmg_kernel_launches())


def default_config(n, **overrides):
    cfg = Config()
    lib().pmg_config_default(ctypes.byref(cfg), n)
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise TypeError("unknown config field %r" % k)
        setattr(cfg, k, v)
    return cfg


def partition_rows(n, n_ranks, rank):
    y0, y1 = ctypes.c_int(), ctypes.c_int()
    check(lib().pmg_partition_rows(n, n_ranks, rank, ctypes.byref(y0), ctypes.byref(y1)))
    return y0.value, y1.value


COMM_ID_BYTES = 128


def comm_unique_id():
    """128 opaque bytes made by one rank; ship them to the others (e.g. torch.distributed.broadcast)."""
    buf = ctypes.create_string_buffer(COMM_ID_BYTES)
    check(lib().pmg_comm_unique_id(buf))
    return buf.raw


def comm_init(unique_id, rank, n_ranks, device):
    """Collective: creates this process's NCCL communicator (one process per GPU)."""
    assert len(unique_id) == COMM_ID_BYTES
    check(lib().pmg_comm_init(ctypes.create_string_buffer(unique_id, COMM_ID_BYTES), rank, n_ranks, device))


def comm_finalize():
    lib().pmg_comm_finalize()


def init_distributed_from_torch(device=None):
    """Bootstrap from an initialised torch.distributed process group (the plumbing only: the id travels
    over it once; all solver traffic then goes through libpmg's own NCCL communicator)."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", rank))
    ids = [comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    comm_init(ids[0], rank, world, device)
    return rank, world, device


class DeviceArray:
    """A device buffer of doubles owned through pmg_device_alloc (tests need no torch)."""

    def __init__(self, shape):
        self.shape = tuple(shape)
        self.size = int(np.prod(self.shape))
        p = ctypes.c_void_p()
        check(lib().pmg_device_alloc(ctypes.byref(p), max(self.size, 1) * 8))
        self.ptr = p.value

    @classmethod
    def from_numpy(cls, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        d = cls(a.shape)
        check(lib().pmg_memcpy(d.ptr, a.ctypes.data, a.size * 8, 1, 0))
        return d

    def numpy(self):
        out = np.empty(self.shape, dtype=np.float64)
        check(lib().pmg_memcpy(out.ctypes.data, self.ptr, self.size * 8, 0, 1))
        return out

    def free(self):
        if self.ptr:
            lib().pmg_device_free(self.ptr)
            self.ptr = None

    def __del__(self):
        # never call into CUDA while the interpreter is being torn down (the runtime may already be gone)
        if sys.is_finalizing():
            return
        try:
            self.free()
        except Exception:
            pass


def _ptr_and_mem(a):
    """(address, pmg_mem) of a numpy array, a DeviceArray or a torch tensor."""
    if isinstance(a, DeviceArray):
        return a.ptr, MEM_DEVICE
    if isinstance(a, np.ndarray):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        return a.ctypes.data, MEM_HOST
    if hasattr(a, "data_ptr"):  # torch tensor
        assert a.is_contiguous() and str(a.dtype) == "torch.float64"
        return a.data_ptr(), (MEM_DEVICE if a.is_cuda else MEM_HOST)
    raise TypeError(type(a))


class Solver:
    """One multigrid hierarchy resident in HBM (pmg_solver)."""

    def __init__(self, n, **cfg):
        self.cfg = default_config(n, **cfg)
        self.n = n
        h = ctypes.c_void_p()
        check(lib().pmg_create(ctypes.byref(self.cfg), ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().pmg_destroy(self._h)
            self._h = None

    def __del__(self):
        if sys.is_finalizing():
            return
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_rhs(self, f):
        p, m = _ptr_and_mem(f)
        check(lib().pmg_set_rhs(self._h, p, m))

    def set_rhs_sine(self):
        check(lib().pmg_set_rhs_sine(self._h))

    def set_guess(self, phi):
        if phi is None:  # the zero start
            check(lib().pmg_set_guess(self._h, None, MEM_HOST))
            return
        p, m = _ptr_and_mem(phi)
        check(lib().pmg_set_guess(self._h, p, m))

    # overlapped host transfers (pinned numpy buffers): see include/pmg.h
    def stage_rhs(self, f_pinned):
        check(lib().pmg_stage_rhs(self._h, ctypes.c_void_p(f_pinned.ctypes.data)))

    def commit_rhs(self):
        check(lib().pmg_commit_rhs(self._h))

    def fetch_solution_begin(self, out_pinned):
        check(lib().pmg_fetch_solution_begin(self._h, ctypes.c_void_p(out_pinned.ctypes.data)))

    def fetch_solution_wait(self):
        check(lib().pmg_fetch_solution_wait(self._h))

    def zero_guess(self):
        check(lib().pmg_zero_guess(self._h))

    @property
    def local_rows(self):
        """(y0, y1): the rows of the finest level this rank owns (the whole grid on one GPU)."""
        if self.cfg.n_ranks > 1:
            return partition_rows(self.n, self.cfg.n_ranks, self.cfg.rank)
        return 0, self.n

    def get_solution(self, out=None):
        if out is None:
            y0, y1 = self.local_rows
            out = np.empty((y1 - y0, self.n))
        p, m = _ptr_and_mem(out)
        check(lib().pmg_get_solution(self._h, p, m))
        return out

    def residual_norm(self):
        v = ctypes.c_double()
        check(lib().pmg_residual_norm(self._h, ctypes.byref(v)))
        return v.value

    def cycle(self, kind=V, want_norm=True):
        v = ctypes.c_double()
        check(lib().pmg_cycle(self._h, kind, ctypes.byref(v) if want_norm else None))
        return v.value if want_norm else None

    def solve(self, kind=V, rel_tol=1e-8, max_cycles=100):
        hist = (ctypes.c_double * (max_cycles + 1))()
        k = ctypes.c_int()
        check(lib().pmg_solve(self._h, kind, rel_tol, max_cycles, hist, ctypes.byref(k)))
        return k.value, np.array(hist[: k.value + 1])

    def pcg(self, precond=1, rel_tol=1e-8, max_iter=100):
        """Conjugate gradients from the current iterate, preconditioned by one cycle of this solver (precond = 1) or not
        at all (0); returns (iterations, history).  On row slabs every rank calls it and updates its own rows
        (local_rows, get_solution); the history is the global one, the same on every rank."""
        hist = (ctypes.c_double * (max_iter + 1))()
        k = ctypes.c_int()
        L = lib()
        L.pmg_pcg.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                              ctypes.POINTER(ctypes.c_int)]
        check(L.pmg_pcg(self._h, precond, rel_tol, max_iter, hist, ctypes.byref(k)))
        return k.value, np.array(hist[: k.value + 1])

    def smooth(self, sweeps, block=1):
        check(lib().pmg_smooth(self._h, sweeps, block))

    def bench_pass(self, which, level=0, reps=5):
        """Average device ms of one fused pass in isolation (0: Pass A, 1: Pass B + norm, 2: Pass B,
        3: Pass A from a zero iterate).  Clobbers the iterate."""
        v = ctypes.c_double()
        check(lib().pmg_bench_pass(self._h, which, level, reps, ctypes.byref(v)))
        return v.value

    @property
    def cross_cycle(self):
        """True if pmg_solve(V) on this handle takes the cross-cycle path (level 0: Pass B + next Pass A in one sweep)."""
        L = lib()
        L.pmg_cross_cycle_active.restype = ctypes.c_int
        L.pmg_cross_cycle_active.argtypes = [ctypes.c_void_p]
        return bool(L.pmg_cross_cycle_active(self._h))

    @property
    def cluster_top(self):
        """Level size from which one cluster launch runs the rest of the cycle (0: not in use)."""
        L = lib()
        L.pmg_cluster_top.restype = ctypes.c_int
        L.pmg_cluster_top.argtypes = [ctypes.c_void_p]
        return L.pmg_cluster_top(self._h)

    @property
    def last_ms(self):
        v = ctypes.c_double()
        check(lib().pmg_last_device_ms(self._h, ctypes.byref(v)))
        return v.value

    @property
    def stream(self):
        return lib().pmg_stream(self._h)


# ---- operator level (device pointers, dense reference layout) ----------------------------------------
def jacobi(x, f, h, omega=1.0, sweeps=1, scratch=None):
    check(lib().pmg_jacobi(x.ptr, f.ptr, x.shape[1], x.shape[0], h, omega, sweeps,
                           scratch.ptr if scratch is not None else None, None))


def residual(r, x, f, h, want_norm2=False):
    v = ctypes.c_double()
    check(lib().pmg_residual(r.ptr if r is not None else None, x.ptr, f.ptr, x.shape[1], x.shape[0], h,
                             ctypes.byref(v) if want_norm2 else None, None))
    return v.value if want_norm2 else None


def gauss_seidel(x, f, h, sweeps=1, ordering=0):
    """Gauss-Seidel sweeps in place: ordering 0 = lexicographic (the reference's GaussSeidelSmoother, exact), 1 = red-black."""
    L = lib()
    L.pmg_gauss_seidel.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                   ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    check(L.pmg_gauss_seidel(x.ptr, f.ptr, x.shape[1], x.shape[0], h, sweeps, ordering, None))


def restrict_fw(fine, coarse):
    check(lib().pmg_restrict_fw(fine.ptr, coarse.ptr, fine.shape[0], coarse.shape[0], None))


def prolong_add(coarse, fine, mode=PROLONG_REFERENCE):
    check(lib().pmg_prolong_add(coarse.ptr, fine.ptr, coarse.shape[0], fine.shape[0], mode, None))


def norm2(v):
    out = ctypes.c_double()
    check(lib().pmg_norm2(v.ptr, v.size, ctypes.byref(out), None))
    return out.value


def set_fused_variant(down, up=None):
    """Tuning: pick the kernel instantiation of the nu == 2 passes (Pass A, Pass B)."""
    lib().pmg_fused_set_variant(down if up is None else (down | (up << 8) | 0x10000))


def num_fused_variants():
    return lib().pmg_fused_num_variants()


def set_small_vcycle_version(v):
    """Which generation of the single-CTA kernel for the levels <= 65 new cycles use (1, 2; 0 = default)."""
    lib().pmg_small_vcycle_set_version(v)


def small_vcycle_version():
    return lib().pmg_small_vcycle_version()


def set_deep_prefetch_below(n):
    """Levels with n <= this use the 7-rows-in-flight variant of the nu == 2 fused passes (0: never, -1: default)."""
    lib().pmg_fused_set_deep_prefetch_below(n)


def set_cluster_top(n):
    """Top level of the 16-CTA cluster kernel (kernels_coarse.cu) for solvers created afterwards: 129 (default), 257,
    0 = off (streaming passes + single-CTA kernel), -1 = back to PMG_CLUSTER / the default."""
    L = lib()
    L.pmg_set_cluster_top.restype = None
    L.pmg_set_cluster_top.argtypes = [ctypes.c_int]
    L.pmg_set_cluster_top(n)


def set_cross_cycle(on, minb=None):
    """Cross-cycle solve on level 0 (Pass B of cycle k fused with Pass A of cycle k+1) for solvers created afterwards:
    True / False, or -1 = PMG_CROSS / the default (on).  minb: shape of the cross pass -- 2 = strips of 128 columns, 4 per
    lane, 8 warps per SM (default; 7 = the same with deeper prefetch); 3 .. 6 = strips of 64 columns with that many CTAs
    per SM; 0 = back to the default."""
    L = lib()
    L.pmg_set_cross_cycle.restype = None
    L.pmg_set_cross_cycle.argtypes = [ctypes.c_int]
    L.pmg_set_cross_cycle(-1 if on == -1 else (2 if on == 2 else (1 if on else 0)))
    if minb is not None:
        L.pmg_fused_set_cross_minb.restype = None
        L.pmg_fused_set_cross_minb.argtypes = [ctypes.c_int]
        L.pmg_fused_set_cross_minb(minb)


def set_pdl(on):
    """Programmatic dependent launch of the cycle kernels (default on; PMG_PDL=0 does the same as set_pdl(False)).
    Affects solvers created afterwards."""
    L = lib()
    L.pmg_set_pdl.restype = None
    L.pmg_set_pdl.argtypes = [ctypes.c_int]
    L.pmg_set_pdl(1 if on else 0)


def set_halo_prologue(on):
    """Multi-GPU Pass A: copy the neighbours' halo rows in a prologue (only boundary warps wait) instead of
    streaming them in place.  Default since round 2 (PMG_HALO_PROLOGUE=0 / set_halo_prologue(False) switch it off)."""
    lib().pmg_fused_set_halo_prologue(1 if on else 0)
