"""ctypes binding of ``csrc/libtruss_b200.so`` (the C ABI declared in ``include/truss_b200.h``).

The product has no CPU fallback: if the library has not been built, importing the solver
raises; if it is loaded on a machine without a CUDA device, every solve raises
``NoCudaDeviceError`` (``TB_ERR_NO_DEVICE``).  Build with ``python __graft_entry__.py`` or
``python -m python_stable_3d_truss_analysis_b200._lib``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.environ.get("TB_LIB_PATH") or os.path.join(CSRC, "libtruss_b200.so")   # TB_LIB_PATH: instrumented builds (tools/)
SOURCES = ["tb_plan.cu", "tb_tsplan.cu", "tb_small.cu", "tb_dense16.cu", "tb_large.cu", "tb_band.cu", "tb_bandts.cu", "tb_api.cu", "tb_adjoint.cu", "tb_peak.cu",
           "tb_ga.cu", "tb_augment.cu", "tb_json.cu", "tb_gencube.cu"]

TB_ERR_NO_DEVICE = -7
TB_ERR_TOO_LARGE = -6


class TrussLibError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"truss_b200 error {code}: {msg}")
        self.code = code


class NoCudaDeviceError(TrussLibError):
    pass


HEADERS = ("tb_common.cuh", "tb_blocks.cuh", "tb_ts.cuh")


def build(force: bool = False, verbose: bool = False, extra_flags=(), out: str | None = None) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU).

    Every source is compiled to an object file on its own (in parallel, rebuilt only when it or a header changed) and
    the objects are linked into ``csrc/libtruss_b200.so``; ``out`` builds a separate (e.g. instrumented) library from
    scratch with ``extra_flags``."""
    if out is not None:
        return _compile(out, verbose, list(extra_flags), objdir=None)
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(INCLUDE, "truss_b200.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    return _compile(LIB_PATH, verbose, list(extra_flags), objdir=os.path.join(CSRC, "build"), force=force)


def _compile(out_path: str, verbose: bool, extra_flags, objdir, force: bool = True) -> str:
    from concurrent.futures import ThreadPoolExecutor
    import tempfile

    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    base = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-Xcompiler", "-fPIC", "-I", INCLUDE] + list(extra_flags)
    if verbose:
        base.insert(1, "-Xptxas=-v")
    tmp = None
    if objdir is None:
        tmp = tempfile.TemporaryDirectory()
        objdir = tmp.name
    os.makedirs(objdir, exist_ok=True)
    hdr_time = max(os.path.getmtime(p) for p in [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(INCLUDE, "truss_b200.h")])

    def one(src):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        path = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(path), hdr_time):
            return obj, ""
        res = subprocess.run(base + ["-c", path, "-o", obj], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        done = list(ex.map(one, SOURCES))
    if verbose:
        print("".join(err for _, err in done))
    res = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out_path] + [o for o, _ in done],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    if tmp is not None:
        tmp.cleanup()
    return out_path


# --------------------------------------------------------------------------- ctypes mirrors
class TbTopology(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_joint", C.c_int32), ("n_member", C.c_int32),
                ("conn", C.c_void_p), ("support", C.c_void_p)]


class TbPlanInfo(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_joint", C.c_int32), ("n_member", C.c_int32), ("n_dof", C.c_int32),
                ("n_free", C.c_int32), ("n_support", C.c_int32), ("n_resist", C.c_int32), ("stable", C.c_int32),
                ("path", C.c_int32), ("n_pad", C.c_int32), ("nnz_lower", C.c_int64), ("n_contrib", C.c_int64),
                ("half_bandwidth", C.c_int64), ("n_tiles", C.c_int64), ("n_tiles_nonzero", C.c_int64),
                ("n_tile_products", C.c_int64), ("chol_flops", C.c_double), ("band_blocks", C.c_int32),
                ("envelope_size", C.c_int64), ("envelope_flops", C.c_double), ("reordered", C.c_int32),
                ("band_blocks_nonzero", C.c_int64), ("band_products", C.c_int64)]


class TbAugmentParams(C.Structure):
    _fields_ = [("move_to_centroid", C.c_int32), ("random_translation", C.c_int32), ("translate_lo", C.c_double),
                ("translate_hi", C.c_double), ("joint_noise", C.c_int32), ("noise_mean", C.c_double * 3),
                ("noise_std", C.c_double * 3), ("reset_pin", C.c_int32), ("min_pin", C.c_int32),
                ("max_pin_ratio", C.c_double), ("seed", C.c_uint64)]


class TbGencubeParams(C.Structure):
    _fields_ = [("grid", C.c_int32 * 3), ("ncube_lo", C.c_int32), ("ncube_hi", C.c_int32), ("method", C.c_int32),
                ("link_type", C.c_int32), ("add_pin", C.c_int32), ("allow_parallel", C.c_int32), ("nforce_lo", C.c_int32),
                ("nforce_hi", C.c_int32), ("n_type", C.c_int32), ("max_attempts", C.c_int32), ("length_lo", C.c_double),
                ("length_hi", C.c_double), ("force_lo", C.c_double * 3), ("force_hi", C.c_double * 3), ("seed", C.c_uint64)]


class TbGaParams(C.Structure):
    _fields_ = [("n_pop", C.c_int32), ("n_elite", C.c_int32), ("n_member", C.c_int32), ("n_type", C.c_int32),
                ("p_crossover", C.c_double), ("p_mutate", C.c_double), ("p_origin", C.c_double), ("seed", C.c_uint64)]


class TbGaReport(C.Structure):
    _fields_ = [("best_index", C.c_int32), ("feasible_index", C.c_int32), ("best_fitness", C.c_double),
                ("feasible_fitness", C.c_double), ("best_stress_ok", C.c_uint8), ("best_displace_ok", C.c_uint8),
                ("pad_", C.c_uint8 * 6)]


class TbBatchIn(C.Structure):
    _fields_ = [("batch", C.c_int32), ("joint_xyz", C.c_void_p), ("joint_stride", C.c_int64),
                ("member_aed", C.c_void_p), ("member_stride", C.c_int64), ("gene", C.c_void_p),
                ("gene_stride", C.c_int64), ("type_table", C.c_void_p), ("n_type", C.c_int32),
                ("force", C.c_void_p), ("force_stride", C.c_int64)]


class TbBatchOut(C.Structure):
    _fields_ = [("u", C.c_void_p), ("ext", C.c_void_p), ("axial", C.c_void_p), ("weight", C.c_void_p),
                ("info", C.c_void_p), ("u_free", C.c_void_p), ("react", C.c_void_p)]


class TbAdjIn(C.Structure):
    _fields_ = [("u", C.c_void_p), ("ext", C.c_void_p), ("axial", C.c_void_p), ("weight", C.c_void_p)]


class TbAdjOut(C.Structure):
    _fields_ = [("joint_xyz", C.c_void_p), ("member_aed", C.c_void_p), ("force", C.c_void_p), ("info", C.c_void_p)]


class TbFitOut(C.Structure):
    _fields_ = [("fitness", C.c_void_p), ("flags", C.c_void_p), ("info", C.c_void_p)]


class TbRaggedIn(C.Structure):
    _fields_ = [("dim", C.c_int32), ("batch", C.c_int32), ("joint_off", C.c_void_p), ("member_off", C.c_void_p),
                ("joint_xyz", C.c_void_p), ("support", C.c_void_p), ("conn", C.c_void_p), ("member_aed", C.c_void_p),
                ("force", C.c_void_p), ("max_joint", C.c_int32), ("max_member", C.c_int32)]


EXPORTS = ["tb_plan_create", "tb_plan_destroy", "tb_plan_query", "tb_plan_set_path", "tb_plan_get_maps",
           "tb_plan_get_scatter", "tb_solve", "tb_solve_host", "tb_solve_host_async", "tb_host_wait", "tb_solve_loadcases", "tb_solve_loadcases_host", "tb_adjoint", "tb_fitness", "tb_fitness_host", "tb_solve_ragged",
           "tb_solve_ragged_host", "tb_adjoint_ragged", "tb_ga_init", "tb_ga_step", "tb_augment_ragged", "tb_json_scan", "tb_json_fill", "tb_gencube_limits", "tb_gencube", "tb_gencube_pack", "tb_pinned_alloc", "tb_pinned_free", "tb_small_path_limits", "tb_fp64_peak", "tb_rsqrt_probe", "tb_div_probe", "tb_profile_enable", "tb_profile_read",
           "tb_launch_count", "tb_strerror", "tb_version", "tb_small_path_fits", "tb_debug_assemble_host", "tb_plan_ts_info", "tb_plan_ts_array", "tb_ts_phase_read"]

_lib = None


def lib():
    """Load the shared library (once).  Raises if it has not been built -- no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library has not been built and there is no CPU fallback. "
            "Run `python __graft_entry__.py` (needs nvcc).")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.tb_plan_create.argtypes = [C.POINTER(TbTopology), C.POINTER(vp)]
    L.tb_plan_destroy.argtypes = [vp]
    L.tb_plan_destroy.restype = None
    L.tb_plan_query.argtypes = [vp, C.POINTER(TbPlanInfo)]
    L.tb_plan_set_path.argtypes = [vp, i32]
    L.tb_plan_get_maps.argtypes = [vp, vp, vp, vp]
    L.tb_plan_get_scatter.argtypes = [vp, vp, vp, vp, vp, vp]
    L.tb_solve.argtypes = [vp, C.POINTER(TbBatchIn), C.POINTER(TbBatchOut), vp]
    L.tb_solve_host.argtypes = [vp, C.POINTER(TbBatchIn), C.POINTER(TbBatchOut)]
    L.tb_solve_host_async.argtypes = [vp, C.POINTER(TbBatchIn), C.POINTER(TbBatchOut), C.POINTER(C.c_uint64)]
    L.tb_host_wait.argtypes = [vp, C.c_uint64]
    L.tb_solve_loadcases.argtypes = [vp, C.POINTER(TbBatchIn), C.POINTER(TbBatchOut), vp]
    L.tb_solve_loadcases_host.argtypes = [vp, C.POINTER(TbBatchIn), C.POINTER(TbBatchOut)]
    L.tb_adjoint.argtypes = [vp, C.POINTER(TbBatchIn), vp, C.POINTER(TbAdjIn), C.POINTER(TbAdjOut), i32, vp]
    L.tb_fitness.argtypes = [vp, C.POINTER(TbBatchIn), dbl, dbl, C.POINTER(TbFitOut), C.POINTER(TbBatchOut), vp]
    L.tb_fitness_host.argtypes = [vp, C.POINTER(TbBatchIn), dbl, dbl, C.POINTER(TbFitOut), C.POINTER(TbBatchOut)]
    L.tb_solve_ragged.argtypes = [C.POINTER(TbRaggedIn), C.POINTER(TbBatchOut), vp]
    L.tb_solve_ragged_host.argtypes = [C.POINTER(TbRaggedIn), C.POINTER(TbBatchOut)]
    L.tb_adjoint_ragged.argtypes = [C.POINTER(TbRaggedIn), vp, C.POINTER(TbAdjIn), C.POINTER(TbAdjOut), vp, vp]
    L.tb_pinned_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.tb_pinned_free.argtypes = [vp]
    L.tb_small_path_limits.argtypes = [C.POINTER(i32), C.POINTER(i32)]
    L.tb_fp64_peak.argtypes = [i32, i32, C.POINTER(dbl), C.POINTER(C.c_float)]
    L.tb_rsqrt_probe.argtypes = [i32, C.POINTER(dbl)]
    L.tb_div_probe.argtypes = [i64, C.c_uint64, C.POINTER(C.c_uint64)]
    L.tb_augment_ragged.argtypes = [C.POINTER(TbRaggedIn), i32, vp, vp, vp, C.POINTER(TbAugmentParams), vp, vp, vp, vp, vp, vp]
    L.tb_gencube_limits.argtypes = [C.POINTER(TbGencubeParams), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.tb_gencube.argtypes = [C.POINTER(TbGencubeParams), i32] + [vp] * 13
    L.tb_gencube_pack.argtypes = [C.POINTER(TbGencubeParams), i32] + [vp] * 13
    L.tb_json_scan.argtypes = [i32, vp, vp, vp, vp, vp, i32]
    L.tb_json_fill.argtypes = [i32, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32]
    L.tb_ga_init.argtypes = [C.POINTER(TbGaParams), vp, vp, vp]
    L.tb_ga_step.argtypes = [C.POINTER(TbGaParams), C.c_uint64, vp, vp, vp, vp, vp, vp, vp]
    L.tb_profile_enable.argtypes = [i32]
    L.tb_profile_read.argtypes = [vp, vp]
    L.tb_launch_count.restype = i64
    L.tb_debug_assemble_host.argtypes = [vp, C.POINTER(TbBatchIn), vp]
    L.tb_plan_ts_info.argtypes = [vp, vp]
    L.tb_plan_ts_array.argtypes = [vp, i32, i32, vp]
    L.tb_plan_ts_array.restype = i64
    L.tb_ts_phase_read.argtypes = [vp]
    L.tb_strerror.argtypes = [C.c_int]
    L.tb_strerror.restype = C.c_char_p
    _lib = L
    return L


def strerror(rc: int) -> str:
    return lib().tb_strerror(int(rc)).decode()


def check(rc: int):
    if rc == 0:
        return
    msg = lib().tb_strerror(rc).decode()
    if rc == TB_ERR_NO_DEVICE:
        raise NoCudaDeviceError(rc, msg)
    raise TrussLibError(rc, msg)


def _ptr(a):
    """Address of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _np(a, dtype, shape=None):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None:
        a = a.reshape(shape)
    return a


class _PinnedOwner:
    """Frees a page-locked allocation when the last view of it is gone."""

    def __init__(self, addr):
        self.addr = addr

    def __del__(self):
        try:
            lib().tb_pinned_free(self.addr)
        except Exception:
            pass


def json_load_packed(texts, dim, is_output=False, threads=0):
    """Parse JSON documents of the reference's format (bytes objects) straight into packed arrays through the native
    loader (tb_json_scan / tb_json_fill, csrc/tb_json.cu).  Returns ``(arrays, err)``: the dict of packed arrays
    (joint_off, member_off, xyz, support, conn, aed, force [+ u, ext, axial, weight]) and the per-document status codes;
    raises TrussLibError on argument errors only (a malformed document is reported through ``err``)."""
    n = len(texts)
    bufs = [t if isinstance(t, bytes) else bytes(t) for t in texts]          # (bytes objects are NUL-terminated in memory)
    ptrs = (C.c_char_p * max(n, 1))(*bufs)
    lens = np.array([len(b) for b in bufs], np.int64)
    nj, nm, err = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int32)
    L = lib()
    rc = L.tb_json_scan(n, ptrs, _ptr(lens), _ptr(nj), _ptr(nm), _ptr(err), int(threads))
    if rc not in (0, -10):
        check(rc)
    nj[err != 0] = 0
    nm[err != 0] = 0
    jo, mo = np.zeros(n + 1, np.int64), np.zeros(n + 1, np.int64)
    jo[1:], mo[1:] = np.cumsum(nj), np.cumsum(nm)
    SJ, SM = int(jo[-1]), int(mo[-1])
    a = {"joint_off": jo, "member_off": mo, "xyz": np.empty(SJ * dim), "support": np.empty(SJ, np.uint8),
         "conn": np.empty(2 * SM, np.int32), "aed": np.empty(3 * SM), "force": np.empty(SJ * dim)}
    if is_output:
        a.update(u=np.empty(SJ * dim), ext=np.empty(SJ * dim), axial=np.empty(SM), weight=np.empty(n))
    # documents that failed the scan keep empty slices; the fill pass reports them again
    err2 = np.zeros(n, np.int32)
    rc = L.tb_json_fill(n, ptrs, _ptr(lens), int(dim), int(bool(is_output)), _ptr(jo), _ptr(mo), _ptr(a["xyz"]),
                        _ptr(a["support"]), _ptr(a["force"]), _ptr(a["conn"]), _ptr(a["aed"]), _ptr(a.get("u")),
                        _ptr(a.get("ext")), _ptr(a.get("axial")), _ptr(a.get("weight")), _ptr(err2), int(threads))
    if rc not in (0, -10):
        check(rc)
    err = np.where(err != 0, err, err2)
    return a, err


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by page-locked memory from the library.  The allocation is owned by the ctypes buffer at the
    bottom of the array's ``base`` chain, so it is freed when the array and every view of it have been collected."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    check(lib().tb_pinned_alloc(C.byref(p), max(n, 1)))
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    buf._owner = _PinnedOwner(p.value)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def fp64_peak(which: int, iters: int = 4096):
    t, ms = C.c_double(), C.c_float()
    check(lib().tb_fp64_peak(which, iters, C.byref(t), C.byref(ms)))
    return t.value, ms.value


def ga_init(params: TbGaParams, gene, type_cum=None, stream=None):
    """GA.Initialize on the device: fills the int32 CUDA tensor ``gene`` [n_pop, n_member]."""
    import torch
    st = torch.cuda.current_stream() if stream is None else stream
    check(lib().tb_ga_init(C.byref(params), _ptr(type_cum), _ptr(gene), C.c_void_p(st.cuda_stream)))


def ga_step(params: TbGaParams, generation: int, fitness, flags, gene_in, gene_out, order, report, stream=None):
    """GA.Select + GA.UpdatePop on the device (all arguments CUDA tensors; gene_out / report may be None)."""
    import torch
    st = torch.cuda.current_stream() if stream is None else stream
    check(lib().tb_ga_step(C.byref(params), int(generation), _ptr(fitness), _ptr(flags), _ptr(gene_in), _ptr(gene_out),
                           _ptr(order), _ptr(report), C.c_void_p(st.cuda_stream)))


def rsqrt_probe(n: int = 1 << 22) -> float:
    """Largest relative error of the pivot reciprocal square root against 1/sqrt(d) (see tb_rsqrt_probe)."""
    e = C.c_double()
    check(lib().tb_rsqrt_probe(n, C.byref(e)))
    return e.value


PROFILE_SLOTS = ("geom", "assemble", "chol", "recover", "small", "subst")


def profile_enable(on: bool):
    check(lib().tb_profile_enable(1 if on else 0))


def profile_read():
    """{slot: (total_ms, launches)} recorded since the last read."""
    ms = np.zeros(8, np.float32)
    cnt = np.zeros(8, np.int64)
    check(lib().tb_profile_read(ms.ctypes.data, cnt.ctypes.data))
    return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(PROFILE_SLOTS)}


def launch_count() -> int:
    return int(lib().tb_launch_count())


# --------------------------------------------------------------------------- Plan
class Plan:
    """One topology (dim, connectivity, supports) -> integer maps + device mirrors."""

    def __init__(self, dim, conn, support):
        L = lib()
        self.conn = _np(conn, np.int32).reshape(-1, 2)
        self.support = _np(support, np.uint8).reshape(-1)
        topo = TbTopology(int(dim), int(self.support.shape[0]), int(self.conn.shape[0]),
                          self.conn.ctypes.data, self.support.ctypes.data)
        h = C.c_void_p()
        check(L.tb_plan_create(C.byref(topo), C.byref(h)))
        self._h = h
        info = TbPlanInfo()
        check(L.tb_plan_query(self._h, C.byref(info)))
        self.info = info
        self.dim, self.nJ, self.M = info.dim, info.n_joint, info.n_member
        self.N, self.n, self.s = info.n_dof, info.n_free, info.n_support
        self.stable = bool(info.stable)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                lib().tb_plan_destroy(h)
            except Exception:
                pass
            self._h = None

    @property
    def path(self):
        info = TbPlanInfo()
        check(lib().tb_plan_query(self._h, C.byref(info)))
        return info.path

    def set_path(self, path: int):
        check(lib().tb_plan_set_path(self._h, int(path)))

    def maps(self):
        free_idx = np.empty(self.n, np.int32)
        dof2free = np.empty(self.N, np.int32)
        sup_idx = np.empty(self.s, np.int32)
        check(lib().tb_plan_get_maps(self._h, free_idx.ctypes.data, dof2free.ctypes.data, sup_idx.ctypes.data))
        return free_idx, dof2free, sup_idx

    def scatter(self):
        nnz, nc = self.info.nnz_lower, self.info.n_contrib
        row, col = np.empty(nnz, np.int32), np.empty(nnz, np.int32)
        ptr = np.empty(nnz + 1, np.int64)
        mem, loc = np.empty(nc, np.int32), np.empty(nc, np.int32)
        check(lib().tb_plan_get_scatter(self._h, row.ctypes.data, col.ctypes.data, ptr.ctypes.data,
                                        mem.ctypes.data, loc.ctypes.data))
        return row, col, ptr, mem, loc

    def assemble_host(self, B, xyz, aed):
        """Debug: the K_ff values the device assembles, [B, nnz_lower] in the entry order of ``scatter()``."""
        keep = []
        bi = self._batch_in(B, xyz, aed, None, None, np.zeros(self.N), keep)
        kv = np.empty((B, int(self.info.nnz_lower)), np.float64)
        check(lib().tb_debug_assemble_host(self._h, C.byref(bi), kv.ctypes.data))
        return kv

    TS_SIDE_ARRAYS = ("colmask", "srcmask", "xmask", "colent", "rowdof", "rownat", "lofs")
    TS_PROGRAM_ARRAYS = ("epos", "ent_src", "tq_first", "tq_multi", "tq_ptr", "tq_pack")

    def ts_program(self):
        """The two-sided band program of the band kernel as host arrays (None when the band is too wide for it):
        ``{"info": {...}, "side": [{name: int32 array}, {...}], "epos": ..., "tq_*": ...}`` -- replayed in numpy by
        the CPU tests."""
        L = lib()
        raw = np.zeros(16, np.int32)
        check(L.tb_plan_ts_info(self._h, raw.ctypes.data))
        if not raw[0]:
            return None
        keys = ("ok", "nblk", "n_pad", "bT", "nS", "nB", "nb_top", "nb_bottom", "chunk_max", "l_per_sys", "products", "solves",
                "entries", "contributions", "multi_entries")

        def fetch(side, which):
            cnt = L.tb_plan_ts_array(self._h, side, which, None)
            a = np.zeros(max(int(cnt), 0), np.int32)
            if cnt > 0:
                L.tb_plan_ts_array(self._h, side, which, a.ctypes.data)
            return a

        out = {"info": {k: int(raw[i]) for i, k in enumerate(keys)}, "side": []}
        for s in range(2):
            d = {name: fetch(s, w) for w, name in enumerate(self.TS_SIDE_ARRAYS)}
            d["colent"] = d["colent"].reshape(-1, 2)
            d["colrec"] = fetch(s, 13).reshape(-1, 4)
            out["side"].append(d)
        for w, name in enumerate(self.TS_PROGRAM_ARRAYS):
            out[name] = fetch(0, len(self.TS_SIDE_ARRAYS) + w)
        return out

    # ------------------------------------------------------------------ batch packing
    def _batch_in(self, B, xyz, aed, gene, type_table, force, keep):
        """Build tb_batch_in from arrays whose leading dim is B or is absent (shared, stride 0)."""
        def rows(a, row, dtype):
            a = _np(a, dtype) if isinstance(a, (np.ndarray, list, tuple)) else a
            total = int(np.prod(a.shape))
            if total == row:
                return a, 0
            if total == row * B:
                return a, row
            raise ValueError(f"array of {total} elements is neither [{row}] nor [{B},{row}]")
        bi = TbBatchIn()
        bi.batch = B
        x, sx = rows(xyz, self.nJ * self.dim, np.float64)
        f, sf = rows(force, self.N, np.float64)
        keep += [x, f]
        bi.joint_xyz, bi.joint_stride, bi.force, bi.force_stride = _ptr(x), sx, _ptr(f), sf
        if aed is not None:
            m, sm = rows(aed, self.M * 3, np.float64)
            keep.append(m)
            bi.member_aed, bi.member_stride = _ptr(m), sm
        else:
            g, sg = rows(gene, self.M, np.int32)
            t = _np(type_table, np.float64).reshape(-1, 3) if isinstance(type_table, (np.ndarray, list)) else type_table
            keep += [g, t]
            bi.gene, bi.gene_stride, bi.type_table, bi.n_type = _ptr(g), sg, _ptr(t), int(t.shape[0])
        return bi

    def solve_host(self, B, xyz, force, aed=None, gene=None, type_table=None, want=("u", "ext", "axial", "weight"),
                   out=None, shared_factor=False):
        """Truss.Solve() for B systems, host (numpy) buffers; H2D/D2H happen inside the library.
        ``shared_factor``: the B systems are load cases of one truss (tb_solve_loadcases_host)."""
        keep = []
        bi = self._batch_in(B, xyz, aed, gene, type_table, force, keep)
        out = {} if out is None else out
        shp = {"u": (B, self.N), "ext": (B, self.N), "axial": (B, self.M), "weight": (B,), "u_free": (B, self.n),
               "react": (B, self.s)}
        for k in want:
            if k not in out:
                out[k] = np.empty(shp[k], np.float64)
        if "info" not in out:
            out["info"] = np.empty(B, np.int32)
        bo = TbBatchOut(_ptr(out.get("u")), _ptr(out.get("ext")), _ptr(out.get("axial")), _ptr(out.get("weight")),
                        _ptr(out["info"]), _ptr(out.get("u_free")), _ptr(out.get("react")))
        fn = lib().tb_solve_loadcases_host if shared_factor else lib().tb_solve_host
        check(fn(self._h, C.byref(bi), C.byref(bo)))
        return out

    def expand_compact(self, u_free, react, force):
        """Dense ``u`` / ``ext`` ([B, N]) from the compact outputs: ``u`` is zero at supported DOFs, ``ext`` is the load
        vector with the supported DOFs overwritten by the reactions (truss.py:342-351)."""
        free_idx, _, sup_idx = self.maps()
        u_free = np.asarray(u_free, dtype=np.float64).reshape(-1, self.n)
        B = u_free.shape[0]
        u = np.zeros((B, self.N))
        u[:, free_idx] = u_free
        ext = np.broadcast_to(np.asarray(force, dtype=np.float64).reshape(-1, self.N), (B, self.N)).copy()
        ext[:, sup_idx] = np.asarray(react, dtype=np.float64).reshape(B, -1)
        return u, ext

    def solve_host_async(self, B, xyz, force, aed=None, gene=None, type_table=None, want=("u", "ext", "axial", "weight"),
                         out=None):
        """Pipelined tb_solve_host (tb_solve_host_async): enqueues the batch and returns ``(ticket, out)`` at once;
        ``host_wait(ticket)`` blocks until ``out`` holds the results.  Three calls may be in flight per plan.  Buffers should
        be page-locked (``pinned_empty``) and must not be touched before the wait."""
        keep = []
        bi = self._batch_in(B, xyz, aed, gene, type_table, force, keep)
        out = {} if out is None else out
        shp = {"u": (B, self.N), "ext": (B, self.N), "axial": (B, self.M), "weight": (B,), "u_free": (B, self.n),
               "react": (B, self.s)}
        for k in want:
            if k not in out:
                out[k] = pinned_empty(shp[k], np.float64)
        if "info" not in out:
            out["info"] = pinned_empty((B,), np.int32)
        bo = TbBatchOut(_ptr(out.get("u")), _ptr(out.get("ext")), _ptr(out.get("axial")), _ptr(out.get("weight")),
                        _ptr(out["info"]), _ptr(out.get("u_free")), _ptr(out.get("react")))
        ticket = C.c_uint64(0)
        check(lib().tb_solve_host_async(self._h, C.byref(bi), C.byref(bo), C.byref(ticket)))
        self._async_keep = getattr(self, "_async_keep", {})
        self._async_keep[ticket.value] = (keep, out, xyz, force, aed, gene, type_table)   # inputs stay alive until the wait
        return ticket.value, out

    def host_wait(self, ticket):
        check(lib().tb_host_wait(self._h, C.c_uint64(int(ticket))))
        keep = getattr(self, "_async_keep", {})
        for t in [t for t in keep if t <= ticket]:
            del keep[t]

    def fitness_host(self, B, xyz, force, gene, type_table, allow_stress, allow_displace, aed=None, full=False,
                     out=None):
        keep = []
        bi = self._batch_in(B, xyz, aed, gene, type_table, force, keep)
        out = {} if out is None else out
        out.setdefault("fitness", np.empty(B, np.float64))
        out.setdefault("flags", np.empty((B, 2), np.uint8))
        out.setdefault("info", np.empty(B, np.int32))
        fo = TbFitOut(_ptr(out["fitness"]), _ptr(out["flags"]), _ptr(out["info"]))
        bo = None
        if full:
            for k, s in (("u", (B, self.N)), ("ext", (B, self.N)), ("axial", (B, self.M)), ("weight", (B,))):
                out.setdefault(k, np.empty(s, np.float64))
            bo = C.byref(TbBatchOut(_ptr(out["u"]), _ptr(out["ext"]), _ptr(out["axial"]), _ptr(out["weight"]), None))
        check(lib().tb_fitness_host(self._h, C.byref(bi), float(allow_stress), float(allow_displace), C.byref(fo), bo))
        return out

    def solve_device(self, B, xyz, force, aed=None, gene=None, type_table=None, out=None, stream=None,
                     shared_factor=False):
        """Device pointers (torch CUDA tensors); enqueues on ``stream`` (a torch stream or None = current).
        ``shared_factor``: the B systems are load cases of one truss (tb_solve_loadcases)."""
        import torch

        keep = []
        bi = self._batch_in(B, xyz, aed, gene, type_table, force, keep)
        st = torch.cuda.current_stream() if stream is None else stream
        bo = TbBatchOut(_ptr(out.get("u")), _ptr(out.get("ext")), _ptr(out.get("axial")), _ptr(out.get("weight")),
                        _ptr(out.get("info")), _ptr(out.get("u_free")), _ptr(out.get("react")))
        fn = lib().tb_solve_loadcases if shared_factor else lib().tb_solve
        check(fn(self._h, C.byref(bi), C.byref(bo), C.c_void_p(st.cuda_stream)))
        return out

    def adjoint_device(self, B, xyz, force, aed, u, grads, out, stream=None, shared_factor=False):
        """Reverse mode of ``solve_device`` (tb_adjoint) on torch CUDA tensors.  ``u`` is the forward's dense [B, N]
        displacements of the same inputs; ``grads`` maps "u" / "ext" / "axial" / "weight" to cotangents (missing or
        None = 0); ``out`` maps "joint_xyz" [B, nJ, d], "member_aed" [B, M, 3] (required), "force" [B, N] and "info" [B]
        to preallocated tensors (missing or None = skipped).  Gradients are per system, also for shared inputs."""
        import torch

        keep = []
        bi = self._batch_in(B, xyz, aed, None, None, force, keep)
        st = torch.cuda.current_stream() if stream is None else stream
        gi = TbAdjIn(_ptr(grads.get("u")), _ptr(grads.get("ext")), _ptr(grads.get("axial")), _ptr(grads.get("weight")))
        go = TbAdjOut(_ptr(out.get("joint_xyz")), _ptr(out.get("member_aed")), _ptr(out.get("force")), _ptr(out.get("info")))
        check(lib().tb_adjoint(self._h, C.byref(bi), _ptr(u), C.byref(gi), C.byref(go), 1 if shared_factor else 0,
                               C.c_void_p(st.cuda_stream)))
        return out

    def fitness_device(self, B, xyz, force, gene, type_table, allow_stress, allow_displace, out, aed=None, stream=None):
        import torch

        keep = []
        bi = self._batch_in(B, xyz, aed, gene, type_table, force, keep)
        st = torch.cuda.current_stream() if stream is None else stream
        fo = TbFitOut(_ptr(out.get("fitness")), _ptr(out.get("flags")), _ptr(out.get("info")))
        bo = None
        if out.get("u") is not None or out.get("axial") is not None or out.get("ext") is not None:
            bo = C.byref(TbBatchOut(_ptr(out.get("u")), _ptr(out.get("ext")), _ptr(out.get("axial")),
                                    _ptr(out.get("weight")), None))
        check(lib().tb_fitness(self._h, C.byref(bi), float(allow_stress), float(allow_displace), C.byref(fo), bo,
                               C.c_void_p(st.cuda_stream)))
        return out


# --------------------------------------------------------------------------- ragged batches
def small_path_fits(dim: int, n_joint: int, n_member: int) -> bool:
    """Does a truss of this size fit the fused shared-memory kernels (the test tb_solve_ragged applies)?"""
    return bool(lib().tb_small_path_fits(int(dim), int(n_joint), int(n_member)))


def small_path_limits():
    a, b = C.c_int32(), C.c_int32()
    lib().tb_small_path_limits(C.byref(a), C.byref(b))
    return a.value, b.value


def solve_ragged_host(dim, joint_off, member_off, xyz, support, conn, aed, force, want=("u", "ext", "axial", "weight"),
                      out=None):
    """B independent trusses with their own topology (generate.py:354-357), packed back to back.  ``out`` may hold
    preallocated result arrays (page-locked ones from ``pinned_empty`` travel at full PCIe speed)."""
    joint_off = _np(joint_off, np.int64)
    member_off = _np(member_off, np.int64)
    B = joint_off.shape[0] - 1
    xyz, force = _np(xyz, np.float64), _np(force, np.float64)
    support, conn, aed = _np(support, np.uint8), _np(conn, np.int32), _np(aed, np.float64)
    SJ, SM = int(joint_off[-1]), int(member_off[-1])
    ri = TbRaggedIn(int(dim), int(B), joint_off.ctypes.data, member_off.ctypes.data, xyz.ctypes.data,
                    support.ctypes.data, conn.ctypes.data, aed.ctypes.data, force.ctypes.data,
                    int(np.diff(joint_off).max()) if B else 0, int(np.diff(member_off).max()) if B else 0)
    out = {} if out is None else out
    out.setdefault("info", np.empty(B, np.int32))
    shp = {"u": SJ * dim, "ext": SJ * dim, "axial": SM, "weight": B}
    for k in want:
        if k not in out:
            out[k] = np.empty(shp[k], np.float64)
        elif out[k].size != shp[k] or out[k].dtype != np.float64:
            raise ValueError(f"out[{k!r}] must be a float64 array of {shp[k]} elements")
    bo = TbBatchOut(_ptr(out.get("u")), _ptr(out.get("ext")), _ptr(out.get("axial")), _ptr(out.get("weight")),
                    _ptr(out["info"]))
    check(lib().tb_solve_ragged_host(C.byref(ri), C.byref(bo)))
    return out


def _ragged_in(dim, packed, max_joint=None, max_member=None):
    """tb_ragged_in over the CUDA tensors of a packed dict (joint_off, member_off, xyz, support, conn, aed, force).  The
    maxima come from the offsets (one device-to-host read) unless given."""
    import torch

    jo, mo = packed["joint_off"], packed["member_off"]
    B = int(jo.shape[0]) - 1
    if max_joint is None or max_member is None:
        mx = [0, 0]
        if B > 0:
            mx = torch.stack([(jo[1:] - jo[:-1]).max(), (mo[1:] - mo[:-1]).max()]).tolist()
        max_joint = mx[0] if max_joint is None else max_joint
        max_member = mx[1] if max_member is None else max_member
    return TbRaggedIn(int(dim), B, _ptr(jo), _ptr(mo), _ptr(packed["xyz"]), _ptr(packed["support"]), _ptr(packed["conn"]),
                      _ptr(packed["aed"]), _ptr(packed["force"]), int(max_joint), int(max_member))


def solve_ragged_device(dim, packed, out=None, stream=None, max_joint=None, max_member=None):
    """tb_solve_ragged on torch CUDA tensors: ``packed`` holds joint_off, member_off [B+1] (int64), xyz [d sum nJ],
    support [sum nJ] (uint8), conn [2 sum M] (int32, local joint ids), aed [3 sum M] and force [d sum nJ] (float64), as
    ``gencube_device`` / ``augment_and_solve_device`` return them.  ``out`` may hold preallocated u, ext [d sum nJ],
    axial [sum M], weight [B] and info [B] tensors; missing ones are allocated.  Enqueues on ``stream`` (None = current)
    and returns ``out``."""
    import torch

    ri = _ragged_in(dim, packed, max_joint, max_member)
    dev = packed["xyz"].device
    SJ, SM, B = int(packed["support"].numel()), int(packed["conn"].numel()) // 2, ri.batch
    out = {} if out is None else out
    for k, n, dt in (("u", SJ * dim, torch.float64), ("ext", SJ * dim, torch.float64), ("axial", SM, torch.float64),
                     ("weight", B, torch.float64), ("info", B, torch.int32)):
        if out.get(k) is None:
            out[k] = torch.empty(n, dtype=dt, device=dev)
    st = torch.cuda.current_stream() if stream is None else stream
    bo = TbBatchOut(_ptr(out["u"]), _ptr(out["ext"]), _ptr(out["axial"]), _ptr(out["weight"]), _ptr(out["info"]))
    check(lib().tb_solve_ragged(C.byref(ri), C.byref(bo), C.c_void_p(st.cuda_stream)))
    return out


def adjoint_ragged_device(dim, packed, u, grads, out, stream=None, max_joint=None, max_member=None, work=None):
    """Reverse mode of ``solve_ragged_device`` (tb_adjoint_ragged) on torch CUDA tensors.  ``u`` is the forward's
    displacements [d sum nJ] of the same inputs; ``grads`` maps "u" / "ext" / "axial" / "weight" to cotangents in the
    packed layout (missing or None = 0); ``out`` maps "joint_xyz" [d sum nJ], "member_aed" [3 sum M] (required),
    "force" [d sum nJ] and "info" [B] (required) to preallocated tensors.  ``work``: device scratch of d sum nJ doubles
    (allocated when None)."""
    import torch

    ri = _ragged_in(dim, packed, max_joint, max_member)
    if work is None:
        work = torch.empty(max(int(packed["support"].numel()) * dim, 1), dtype=torch.float64, device=packed["xyz"].device)
    st = torch.cuda.current_stream() if stream is None else stream
    gi = TbAdjIn(_ptr(grads.get("u")), _ptr(grads.get("ext")), _ptr(grads.get("axial")), _ptr(grads.get("weight")))
    go = TbAdjOut(_ptr(out.get("joint_xyz")), _ptr(out.get("member_aed")), _ptr(out.get("force")), _ptr(out.get("info")))
    check(lib().tb_adjoint_ragged(C.byref(ri), _ptr(u), C.byref(gi), C.byref(go), _ptr(work), C.c_void_p(st.cuda_stream)))
    return out


def augment_and_solve_device(dim, pool, n_out, params: "TbAugmentParams", src=None, solve=True, device=None):
    """Dataset generation on the device: expand the packed pool (dict of numpy arrays: joint_off, member_off, xyz,
    support, conn, aed, force) into ``n_out`` augmented trusses (tb_augment_ragged) and, if ``solve``, run
    tb_solve_ragged on them without leaving the GPU.  Returns a dict of torch CUDA tensors in the packed layout
    (joint_off, member_off, src, xyz, support, conn, aed, force [, u, ext, axial, weight, info])."""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    jo, mo = _np(pool["joint_off"], np.int64), _np(pool["member_off"], np.int64)
    P = jo.shape[0] - 1
    src = (np.arange(n_out) % P).astype(np.int32) if src is None else _np(src, np.int32)
    nj, nm = np.diff(jo), np.diff(mo)
    ojo = np.zeros(n_out + 1, np.int64)
    omo = np.zeros(n_out + 1, np.int64)
    ojo[1:] = np.cumsum(nj[src])
    omo[1:] = np.cumsum(nm[src])
    td = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)  # noqa: E731
    d = {"p_jo": td(jo, np.int64), "p_mo": td(mo, np.int64), "p_xyz": td(pool["xyz"], np.float64),
         "p_sup": td(pool["support"], np.uint8), "p_conn": td(pool["conn"], np.int32), "p_aed": td(pool["aed"], np.float64),
         "p_force": td(pool["force"], np.float64)}
    SJ, SM = int(ojo[-1]), int(omo[-1])
    out = {"joint_off": td(ojo, np.int64), "member_off": td(omo, np.int64), "src": td(src, np.int32),
           "xyz": torch.empty(SJ * dim, dtype=torch.float64, device=dev), "support": torch.empty(SJ, dtype=torch.uint8, device=dev),
           "conn": torch.empty(SM * 2, dtype=torch.int32, device=dev), "aed": torch.empty(SM * 3, dtype=torch.float64, device=dev),
           "force": torch.empty(SJ * dim, dtype=torch.float64, device=dev)}
    maxj, maxm = int(nj.max()), int(nm.max())
    ri = TbRaggedIn(int(dim), int(P), _ptr(d["p_jo"]), _ptr(d["p_mo"]), _ptr(d["p_xyz"]), _ptr(d["p_sup"]), _ptr(d["p_conn"]),
                    _ptr(d["p_aed"]), _ptr(d["p_force"]), maxj, maxm)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    check(lib().tb_augment_ragged(C.byref(ri), int(n_out), _ptr(out["src"]), _ptr(out["joint_off"]), _ptr(out["member_off"]),
                                  C.byref(params), _ptr(out["xyz"]), _ptr(out["support"]), _ptr(out["conn"]), _ptr(out["aed"]),
                                  _ptr(out["force"]), st))
    if solve:
        solve_ragged_device(dim, out, out=out, max_joint=maxj, max_member=maxm)
    out["_keep"] = d
    return out


def gencube_device(params: "TbGencubeParams", n, type_table, solve=True, export=False, device=None):
    """Random cube trusses generated on the device (tb_gencube), compacted into the packed ragged layout
    (tb_gencube_pack) and, if ``solve``, solved by tb_solve_ragged without leaving the GPU.  Returns a dict of torch CUDA
    tensors (joint_off, member_off, xyz, support, conn, aed, force, gen_info [, u, ext, axial, weight, info]); with
    ``export`` also the walk (``cells`` [n, max_cube], ``picks`` [n, max_cube, 6], ``length`` [n, 3]) for replay tests."""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    mj, mm, mc = C.c_int32(), C.c_int32(), C.c_int32()
    check(lib().tb_gencube_limits(C.byref(params), C.byref(mj), C.byref(mm), C.byref(mc)))
    mj, mm, mc = mj.value, mm.value, mc.value
    n = int(n)
    tt = torch.from_numpy(np.ascontiguousarray(type_table, dtype=np.float64).reshape(-1, 3)).to(dev)
    if tt.shape[0] != params.n_type:
        raise ValueError("type_table must hold params.n_type rows")
    f64, e = torch.float64, lambda *shape, dt=torch.float64: torch.empty(*shape, dtype=dt, device=dev)  # noqa: E731
    s = {"xyz": e(n, mj, 3), "support": e(n, mj, dt=torch.uint8), "force": e(n, mj, 3), "conn": e(n, mm, 2, dt=torch.int32),
         "aed": e(n, mm, 3), "nj": e(n, dt=torch.int32), "nm": e(n, dt=torch.int32), "info": e(n, dt=torch.int32)}
    ex = {"cells": e(n, mc, dt=torch.int16), "picks": e(n, mc, 6, dt=torch.uint8), "length": e(n, 3)} if export else {}
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    check(lib().tb_gencube(C.byref(params), n, _ptr(tt), _ptr(s["xyz"]), _ptr(s["support"]), _ptr(s["force"]), _ptr(s["conn"]),
                           _ptr(s["aed"]), _ptr(s["nj"]), _ptr(s["nm"]), _ptr(s["info"]), _ptr(ex.get("cells")),
                           _ptr(ex.get("picks")), _ptr(ex.get("length")), st))
    z = torch.zeros(1, dtype=torch.int64, device=dev)
    jo = torch.cat([z, torch.cumsum(s["nj"].to(torch.int64), 0)])
    mo = torch.cat([z, torch.cumsum(s["nm"].to(torch.int64), 0)])
    SJ, SM = int(jo[-1]), int(mo[-1])
    out = {"joint_off": jo, "member_off": mo, "xyz": e(SJ * 3), "support": e(SJ, dt=torch.uint8), "force": e(SJ * 3),
           "conn": e(SM * 2, dt=torch.int32), "aed": e(SM * 3), "gen_info": s["info"]}
    check(lib().tb_gencube_pack(C.byref(params), n, _ptr(s["xyz"]), _ptr(s["support"]), _ptr(s["force"]), _ptr(s["conn"]),
                                _ptr(s["aed"]), _ptr(jo), _ptr(mo), _ptr(out["xyz"]), _ptr(out["support"]), _ptr(out["force"]),
                                _ptr(out["conn"]), _ptr(out["aed"]), st))
    out.update(ex)
    if solve and n > 0:
        solve_ragged_device(3, out, out=out, max_joint=int(s["nj"].max()), max_member=int(s["nm"].max()))
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
