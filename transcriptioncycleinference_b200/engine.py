"""Thin object layer over the C ABI: a device-resident dataset and the three operators of the
hot path (ssfun batch, forward curves, DRAM fit).  All compute happens in libtcmcmc.so."""
import ctypes as C

import numpy as np

from . import _lib
from .constructs import DEFAULT_CONSTRUCT, to_c


class Cells:
    """Packed single-cell traces resident on one or more GPUs.

    Mirrors the reference's `data(cellNum).{time,MS2,PP7}` struct array after truncation
    (src/TranscriptionCycleMCMC.m:163-181).  `t`, `ms2`, `pp7` are lists of 1-D arrays (NaN =
    missing)."""

    def __init__(self, t, ms2, pp7, construct=DEFAULT_CONSTRUCT, devices=(0,)):
        self.ncells = len(t)
        self.N = np.array([len(x) for x in t], dtype=np.int32)
        self.off = np.zeros(self.ncells + 1, dtype=np.int64)
        self.off[1:] = np.cumsum(self.N)
        self.t = _lib.f64(np.concatenate([np.asarray(x, dtype=np.float64) for x in t]))
        self.ms2 = _lib.f64(np.concatenate([np.asarray(x, dtype=np.float64) for x in ms2]))
        self.pp7 = _lib.f64(np.concatenate([np.asarray(x, dtype=np.float64) for x in pp7]))
        self.Nmax = int(self.N.max())
        self.ld = 7 + self.Nmax
        self.construct = construct
        self.devices = list(devices)
        self._c = to_c(construct)
        self._h = C.c_void_p(None)
        L = _lib.load()
        dev = _lib.i32(self.devices)
        _lib.check(L.tc_cells_create(C.byref(self._c), self.ncells, _lib.ptr(self.N), _lib.ptr(self.off),
                                     _lib.ptr(self.t), _lib.ptr(self.ms2), _lib.ptr(self.pp7),
                                     len(self.devices), _lib.ptr(dev), C.byref(self._h)))

    @classmethod
    def from_packed(cls, N, off, t, ms2, pp7, **kw):
        sl = [slice(int(off[c]), int(off[c]) + int(N[c])) for c in range(len(N))]
        return cls([t[s] for s in sl], [ms2[s] for s in sl], [pp7[s] for s in sl], **kw)

    def close(self):
        if self._h:
            _lib.load().tc_cells_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def cell(self, c):
        s = slice(int(self.off[c]), int(self.off[c + 1]))
        return self.t[s], self.ms2[s], self.pp7[s]

    def t_interp(self, c):
        out = np.zeros(int(self.N[c]))
        _lib.check(_lib.load().tc_cells_t_interp(self._h, c, _lib.ptr(out), out.size))
        return out

    def pad_theta(self, thetas):
        """list of per-cell parameter vectors -> [n, ld] zero-padded array"""
        out = np.zeros((len(thetas), self.ld))
        for i, th in enumerate(thetas):
            out[i, :len(th)] = th
        return out

    # ---- ssfun(theta, data) for a batch: SumofSquaresFunction_TranscriptionCycleMCMC.m
    def ss_batch(self, cell_id, theta, algo=_lib.ALGO_TOEPLITZ):
        theta = _lib.f64(theta)
        cell_id = _lib.i32(cell_id)
        assert theta.ndim == 2 and theta.shape[0] == cell_id.size
        out = np.zeros(cell_id.size)
        _lib.check(_lib.load().tc_ss_batch(self._h, cell_id.size, _lib.ptr(cell_id), _lib.ptr(theta),
                                           theta.shape[1], algo, _lib.ptr(out)))
        return out

    def ss_batch_device(self, n, d_cell_id, d_theta, ld, d_out, algo=_lib.ALGO_TOEPLITZ, device=None, stream=0):
        """Device-pointer variant (ints are raw device addresses, e.g. torch .data_ptr())."""
        dev = self.devices[0] if device is None else device
        _lib.check(_lib.load().tc_ss_batch_device(self._h, dev, n, d_cell_id, d_theta, ld, algo, d_out, stream))

    # ---- model curves: ConstantElongationSim + GetFluorFromPolPos + A scaling
    def forward(self, cell_id, theta, on_raw_grid=True):
        theta = _lib.f64(theta)
        cell_id = _lib.i32(cell_id)
        a = np.zeros((cell_id.size, self.Nmax)); b = np.zeros((cell_id.size, self.Nmax))
        _lib.check(_lib.load().tc_forward(self._h, cell_id.size, _lib.ptr(cell_id), _lib.ptr(theta),
                                          theta.shape[1], 1 if on_raw_grid else 0, _lib.ptr(a), _lib.ptr(b),
                                          self.Nmax))
        return a, b

    # ---- the DRAM fit: mcmcrun(model,data,params,options) for many chains at once
    def mcmc_run(self, opts, chain_cell, theta0, qcov_diag, low, upp, prior_mu, prior_sig, chain_uid=None,
                 replay=None, want_flags=False, chain_out=None, s2chain_out=None):
        """chain_out / s2chain_out: optional caller-owned destinations of the raw chains ([nch, nkeep, ld] and [nch, ns2]
        float64, C-contiguous, with (nkeep, ns2) = _lib.stored_rows(opts): n_steps-n_burn+1 and n_steps at opts.thin = 1;
        ideally from _lib.pinned_empty, which a caller fitting repeatedly allocates once: page-locking GBs costs about as much
        as copying them)."""
        chain_cell = _lib.i32(chain_cell)
        nch = chain_cell.size
        arrs = [_lib.f64(x) for x in (theta0, qcov_diag, low, upp, prior_mu, prior_sig)]
        ld = arrs[0].shape[1]
        for x in arrs:
            assert x.shape == (nch, ld)
        mean = np.zeros((nch, ld)); std = np.zeros((nch, ld)); sig = np.zeros((nch, 2))
        cnt = np.zeros((nch, _lib.NCOUNTERS), dtype=np.int64)
        chain = s2 = None
        if opts.store_chain:
            nkeep, ns2 = _lib.stored_rows(opts)
            # raw chains are GBs: page-locked destinations, so that the device -> host copy runs at PCIe speed (every row is
            # written by the kernel: the buffers need no zero fill)
            chain = chain_out if chain_out is not None else _lib.pinned_empty((nch, nkeep, ld))
            s2 = s2chain_out if s2chain_out is not None else _lib.pinned_empty((nch, ns2))
            assert chain.shape == (nch, nkeep, ld) and s2.shape == (nch, ns2)
            assert chain.dtype == np.float64 and s2.dtype == np.float64 and chain.flags.c_contiguous and s2.flags.c_contiguous
        uid = None if chain_uid is None else np.ascontiguousarray(chain_uid, dtype=np.uint64)
        rp = None
        keep = []
        flags = sschain = None
        if replay is not None or want_flags:
            rp = _lib.Replay()
            if replay is not None:
                for k in ("z1", "u1", "z2", "u2", "chi2"):
                    a = _lib.f64(replay[k]); keep.append(a)
                    setattr(rp, k, a.ctypes.data)
                assert keep[0].shape == (nch, opts.nsimu, ld) and keep[1].shape == (nch, opts.nsimu)
            flags = np.zeros((nch, opts.nsimu), dtype=np.int32); sschain = np.zeros((nch, opts.nsimu))
            rp.flags = flags.ctypes.data
            rp.sschain = sschain.ctypes.data
        L = _lib.load()
        _lib.check(L.tc_mcmc_run(self._h, C.byref(opts), nch, _lib.ptr(chain_cell), _lib.ptr(uid), ld,
                                 *[_lib.ptr(x) for x in arrs], _lib.ptr(mean), _lib.ptr(std), _lib.ptr(sig),
                                 _lib.ptr(cnt), _lib.ptr(chain), _lib.ptr(s2),
                                 C.byref(rp) if rp is not None else None))
        return dict(mean=mean, std=std, sig=sig, counters=cnt, chain=chain, s2chain=s2, flags=flags,
                    sschain=sschain, kernel_seconds=L.tc_last_kernel_seconds(), drain_seconds=L.tc_last_drain_seconds())
