"""ctypes binding of libtcmcmc.so — the C ABI declared in include/tcmcmc.h.

There is NO CPU fallback: if the library is missing and cannot be built, or no CUDA device is
present, the compute entry points raise.  This module never imports anything from oracle/.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

MAX_SETS = 8
MAX_GPUS = 8
TC_EINVAL = -1        # bad argument (the message says which)
TC_EDIM = -4          # numel(t(1):dt:t(end)) != numel(t)
TC_ESTATE = -6        # ss(theta0) not finite for a chain
NCOUNTERS = 16
ALGO_PAIRS, ALGO_TOEPLITZ = 0, 1
CNT_SS_EVALS, CNT_ACC_STAGE1, CNT_ACC_STAGE2, CNT_OUT_OF_BOUNDS = 0, 1, 2, 3
CNT_ADAPTATIONS, CNT_CHOL_FAIL, CNT_DR_TRIES, CNT_STATUS = 4, 5, 6, 7
CNT_CYCLES0 = 8       # + 0..7: per-phase clock readings (include/tcmcmc.h)
FL_ACCEPT, FL_STAGE2, FL_OOB1, FL_DR, FL_OOB2 = 1, 2, 4, 8, 16
LAYOUT_AUTO, LAYOUT_BIG, LAYOUT_WARP, LAYOUT_CTA = 0, 1, 2, 3   # tc_mcmc_opts.layout (TC_LAYOUT_*)

EXPORTS = [
    "tc_version", "tc_last_error", "tc_device_count", "tc_device_info_get", "tc_opts_default",
    "tc_cells_create", "tc_cells_destroy", "tc_cells_t_interp", "tc_ss_batch", "tc_ss_batch_device",
    "tc_forward", "tc_mcmc_run", "tc_last_kernel_seconds", "tc_rng_dump", "tc_measure_fp64_peak",
    "tc_debug_subprof", "tc_last_drain_seconds", "tc_host_alloc", "tc_host_free",
]


class TcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libtcmcmc error %d: %s" % (code, msg))
        self.code = code


class Construct(C.Structure):
    """tc_construct — mirrors the table of GetFluorFromPolPos.m:18-30."""
    _fields_ = [("nsets", C.c_int32), ("_pad", C.c_int32), ("L_ms2", C.c_double), ("L_pp7", C.c_double)] + [
        (n, C.c_double * MAX_SETS)
        for n in ("ms2_start", "ms2_end", "ms2_loopn", "pp7_start", "pp7_end", "pp7_loopn")
    ]


class McmcOpts(C.Structure):
    _fields_ = [
        ("nsimu", C.c_int32), ("burnintime", C.c_int32), ("adaptint", C.c_int32), ("ntry", C.c_int32),
        ("updatesigma", C.c_int32), ("burnin_cumulative", C.c_int32), ("n_burn", C.c_int32),
        ("store_chain", C.c_int32), ("replay", C.c_int32), ("algo", C.c_int32), ("ngpus", C.c_int32),
        ("devices", C.c_int32 * MAX_GPUS),
        ("drscale", C.c_double), ("adascale", C.c_double), ("qcovadj", C.c_double),
        ("burnin_scale", C.c_double), ("N0", C.c_double), ("S20", C.c_double), ("sigma2_0", C.c_double),
        ("seed", C.c_uint64), ("layout", C.c_int32), ("qcovadj_always", C.c_int32),
    ]


class Replay(C.Structure):
    _fields_ = [("z1", C.c_void_p), ("u1", C.c_void_p), ("z2", C.c_void_p), ("u2", C.c_void_p),
                ("chi2", C.c_void_p), ("flags", C.c_void_p), ("sschain", C.c_void_p)]


class DeviceInfo(C.Structure):
    _fields_ = [("name", C.c_char * 128), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("sm_count", C.c_int32), ("_pad", C.c_int32), ("total_mem", C.c_int64),
                ("smem_per_block_optin", C.c_int64)]


_lib = None


def lib_path():
    return _build.LIB


def load():
    """Load (building in-tree if needed) libtcmcmc.so.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.is_stale():
        try:
            _build.build()
        except Exception as e:                                   # stale-but-present: keep going
            if not os.path.exists(_build.LIB):
                raise RuntimeError("libtcmcmc.so is missing and could not be built (%s); "
                                   "there is no CPU fallback" % e)
    L = C.CDLL(_build.LIB)
    vp, ip, dp = C.c_void_p, C.c_void_p, C.c_void_p
    L.tc_version.restype = C.c_int
    L.tc_last_error.restype = C.c_char_p
    L.tc_last_kernel_seconds.restype = C.c_double
    L.tc_last_drain_seconds.restype = C.c_double
    L.tc_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.tc_host_free.argtypes = [C.c_void_p]
    L.tc_host_free.restype = None
    L.tc_device_count.argtypes = [C.POINTER(C.c_int)]
    L.tc_device_info_get.argtypes = [C.c_int, C.POINTER(DeviceInfo)]
    L.tc_opts_default.argtypes = [C.POINTER(McmcOpts)]
    L.tc_opts_default.restype = None
    L.tc_cells_create.argtypes = [C.POINTER(Construct), C.c_int, ip, ip, dp, dp, dp, C.c_int, ip,
                                  C.POINTER(vp)]
    L.tc_cells_destroy.argtypes = [vp]
    L.tc_cells_destroy.restype = None
    L.tc_cells_t_interp.argtypes = [vp, C.c_int, dp, C.c_int]
    L.tc_ss_batch.argtypes = [vp, C.c_int64, ip, dp, C.c_int, C.c_int, dp]
    L.tc_ss_batch_device.argtypes = [vp, C.c_int, C.c_int64, vp, vp, C.c_int, C.c_int, vp, vp]
    L.tc_forward.argtypes = [vp, C.c_int64, ip, dp, C.c_int, C.c_int, dp, dp, C.c_int]
    L.tc_mcmc_run.argtypes = [vp, C.POINTER(McmcOpts), C.c_int, ip, vp, C.c_int] + [dp] * 6 + \
                             [vp, vp, vp, vp, vp, vp, C.POINTER(Replay)]
    L.tc_rng_dump.argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.c_double, C.c_int, dp, dp, dp, dp, dp,
                              C.c_int]
    L.tc_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.tc_debug_subprof.argtypes = [vp, C.c_int]
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise TcError(rc, load().tc_last_error().decode("utf-8", "replace"))
    return rc


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class _Pinned:
    """Owner of one tc_host_alloc block (freed when the last array viewing it goes away)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p(None)
        check(load().tc_host_alloc(nbytes, C.byref(self.ptr)))
        self.nbytes = nbytes

    def __del__(self):
        try:
            if self.ptr:
                load().tc_host_free(self.ptr)
                self.ptr = C.c_void_p(None)
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64):
    """ndarray in page-locked host memory (tc_host_alloc): the destination of large device -> host copies (raw chains)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    own = _Pinned(max(n, 1))
    buf = (C.c_char * max(n, 1)).from_address(own.ptr.value)
    buf._owner = own                                            # keeps the block alive as long as the buffer is referenced
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def device_count():
    n = C.c_int(0)
    try:
        load().tc_device_count(C.byref(n))
    except OSError:
        return 0
    return n.value


def device_info(device=0):
    info = DeviceInfo()
    check(load().tc_device_info_get(device, C.byref(info)))
    return dict(name=info.name.decode(), cc=(info.cc_major, info.cc_minor), sm_count=info.sm_count,
                total_mem=info.total_mem, smem_per_block_optin=info.smem_per_block_optin)


def default_opts(**kw):
    o = McmcOpts()
    load().tc_opts_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise AttributeError("tc_mcmc_opts has no field %r" % k)
        setattr(o, k, v)
    return o


def measure_fp64_peak(device=0):
    """(DFMA lane-ops/s, SM clock MHz during the micro-benchmark)."""
    a, b = C.c_double(0), C.c_double(0)
    check(load().tc_measure_fp64_peak(device, C.byref(a), C.byref(b)))
    return a.value, b.value


def rng_dump(seed, chain_uid, npar, chi2_dof, nsimu, device=0):
    z1 = np.zeros((nsimu, npar)); z2 = np.zeros((nsimu, npar))
    u1 = np.zeros(nsimu); u2 = np.zeros(nsimu); c2 = np.zeros(nsimu)
    check(load().tc_rng_dump(seed, chain_uid, npar, float(chi2_dof), nsimu, ptr(z1), ptr(u1), ptr(z2),
                             ptr(u2), ptr(c2), device))
    return dict(z1=z1, u1=u1, z2=z2, u2=u2, chi2=c2)


def debug_subprof():
    """Sub-phase cycle counters of chain 0 (zeros unless libtcmcmc was built with -DTC_SUBPROF)."""
    out = np.zeros(32, dtype=np.int64)
    load().tc_debug_subprof(ptr(out), 32)
    return out
