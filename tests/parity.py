"""The harness of the GPU parity tests: cells on synthetic series, the randomness a sampler run consumes, the C oracle's
chain for every device chain (oracle/tc_oracle.c: orc_dram), and the comparison of the two.  The test_gpu_* modules
import it; it holds no tests itself (no test_ prefix, so pytest does not collect it)."""
import concurrent.futures as cf
import ctypes as C

import numpy as np
import pytest

from transcriptioncycleinference_b200 import _lib

DTS = (0.1, 1.0 / 3.0, 0.3, 0.7)
LAYOUTS = [(_lib.LAYOUT_CTA, "cta"), (_lib.LAYOUT_WARP, "warp"), (_lib.LAYOUT_BIG, "big")]
# the oracle's counters (orc_dram): SS evaluations, stage-1 / stage-2 accepts, out-of-bounds proposals, adaptations,
# Cholesky failures
ORC_SS, ORC_ACC1, ORC_ACC2, ORC_OOB, ORC_ADAPT, ORC_CHOL_FAIL = range(6)


def need_gpu():
    """_lib, or skip the test when there is no CUDA device."""
    if _lib.device_count() < 1:
        pytest.skip("no CUDA device")
    return _lib


# ------------------------------------------------------------------------------------------------ cells
def _grid_ok(co, t):
    try:
        co.t_interp(t)
        return True
    except ValueError:
        return False


def series(co, rng, N, dt=None):
    """One cell: the irregular grid + NaN mask of test_series_length_extremes_replay, or the regular grid t = k dt (the first
    of DTS, starting at `dt`, whose t(1):dt:t(end) has N points).  Irregular grids are redrawn until that holds."""
    if dt is None:
        while True:
            t = np.concatenate([[0.0], np.cumsum(rng.uniform(0.15, 0.35, N - 1))])
            if _grid_ok(co, t):
                break
    else:
        k = DTS.index(dt)
        for d in DTS[k:] + DTS[:k]:
            t = np.arange(N) * d
            if _grid_ok(co, t):
                break
        else:
            raise AssertionError("no regular grid of %d points" % N)
    m2 = rng.uniform(0, 3, N); p7 = rng.uniform(0, 10, N)
    m2[rng.random(N) < 0.4] = np.nan; p7[rng.random(N) < 0.2] = np.nan
    return t, m2, p7


def make_cells(co, cols, construct=None):
    """Cells from (t, ms2, pp7) triples; t_interp of every cell must be the oracle's, bit for bit."""
    from transcriptioncycleinference_b200.engine import Cells
    kw = {} if construct is None else dict(construct=construct)
    cells = Cells([c[0] for c in cols], [c[1] for c in cols], [c[2] for c in cols], **kw)
    for c, col in enumerate(cols):
        assert np.array_equal(cells.t_interp(c), co.t_interp(col[0])), c
    return cells, dict(N=cells.N, off=cells.off, t=cells.t, ms2=cells.ms2, pp7=cells.pp7)


def cols(orc, lengths, seed):
    co, _ = orc
    rng = np.random.default_rng(seed)
    return [series(co, rng, N, DTS[k % 4] if k % 2 else None) for k, N in enumerate(lengths)]


# ------------------------------------------------------------------------------------------------ randomness
def replay_streams(N_of_chain, nsimu, ld, seed):
    """Injected randomness for one chain per entry of N_of_chain (its series length): z1, u1, z2, u2, chi2 with 1 + 2N
    degrees of freedom, drawn in that order.  z1, z2 [nch, nsimu, ld]; u1, u2, chi2 [nch, nsimu]."""
    g = np.random.default_rng(seed)
    nch = len(N_of_chain)
    return dict(z1=g.standard_normal((nch, nsimu, ld)), u1=g.random((nch, nsimu)), z2=g.standard_normal((nch, nsimu, ld)),
                u2=g.random((nch, nsimu)), chi2=np.stack([g.chisquare(1 + 2 * int(N), nsimu) for N in N_of_chain]))


def dumped_streams(N_of_chain, uid, seed, nsimu):
    """The Philox streams a production run with this seed draws for chain uid[i] (tc_rng_dump), per chain: z1, z2
    [nsimu, 7 + N_of_chain[i]]; u1, u2, chi2 [nsimu]."""
    per = [_lib.rng_dump(seed, int(u), 7 + int(N), 1 + 2 * int(N), nsimu) for N, u in zip(N_of_chain, uid)]
    return {k: [d[k] for d in per] for k in per[0]}


# ------------------------------------------------------------------------------------------------ oracle and checks
def oracle_chains(orc, packed, cc, opts, ins, streams):
    """The oracle's chain for every device chain i (cell cc[i], inputs x[i] of ins) on streams[k][i] (z1, z2 at least npar
    wide), with the oracle's options opts.  packed: N, off, t, ms2, pp7 of the cells."""
    co, cons = orc

    def one(i):
        c = int(cc[i]); N = int(packed["N"][c]); o = int(packed["off"][c]); npar = 7 + N
        sti = {k: v[i][:, :npar] if k in ("z1", "z2") else v[i] for k, v in streams.items()}
        return co.dram(cons, packed["t"][o:o + N], packed["ms2"][o:o + N], packed["pp7"][o:o + N], opts,
                       *[x[i, :npar] for x in ins], streams=sti)

    with cf.ThreadPoolExecutor() as ex:                            # the oracle releases the GIL
        return list(ex.map(one, range(len(cc))))


def _check_counters(tag, out, i, ref):
    cnt, rc = out["counters"][i], ref["counters"]
    want = {_lib.CNT_SS_EVALS: rc[ORC_SS], _lib.CNT_ACC_STAGE1: rc[ORC_ACC1], _lib.CNT_ACC_STAGE2: rc[ORC_ACC2],
            _lib.CNT_OUT_OF_BOUNDS: rc[ORC_OOB], _lib.CNT_ADAPTATIONS: rc[ORC_ADAPT], _lib.CNT_CHOL_FAIL: rc[ORC_CHOL_FAIL],
            _lib.CNT_DR_TRIES: int(np.sum((ref["flags"] & _lib.FL_DR) != 0)), _lib.CNT_STATUS: 0}
    got = {k: int(cnt[k]) for k in want}
    assert got == {k: int(v) for k, v in want.items()}, (tag, i, got, want)


def check_chain(tag, out, i, ref, npar, first_row=0, atol=1e-7):
    """Flags, rows (to atol), s2chain, sschain and all seven counters of device chain i against the oracle's chain."""
    assert np.array_equal(out["flags"][i], ref["flags"]), (tag, i, int(np.argmax(out["flags"][i] != ref["flags"])))
    np.testing.assert_allclose(out["chain"][i][:, :npar], ref["chain"][first_row:], rtol=0, atol=atol, err_msg=str((tag, i)))
    np.testing.assert_allclose(out["s2chain"][i], ref["s2chain"], rtol=1e-9, err_msg=str((tag, i)))
    np.testing.assert_allclose(out["sschain"][i], ref["sschain"], rtol=1e-9, err_msg=str((tag, i)))
    _check_counters(tag, out, i, ref)


def check_summaries(tag, out, i, ref, npar, n_burn=1, atol=None):
    """For a run that stored no rows: flags and sschain when the run returned them, all seven counters, and the summaries of
    device chain i against the oracle's chain — mean and population std of rows n_burn-1 ... (the rows a run with this
    n_burn stores), sqrt(mean(s2chain)) and std(sqrt(s2chain), 1).  Mean and std to 1e-7, check_chain's tolerance for the
    rows they summarise (after 7 adaptations in 1 000 steps the means differ from the oracle's by up to 6e-9: the
    factorisations sum in another order), std also to 1e-6 relative; sigma to 1e-9 and 1e-8 relative.  atol replaces them
    all by one absolute tolerance (long runs)."""
    if out["flags"] is not None:
        assert np.array_equal(out["flags"][i], ref["flags"]), (tag, i, int(np.argmax(out["flags"][i] != ref["flags"])))
    if out["sschain"] is not None:
        np.testing.assert_allclose(out["sschain"][i], ref["sschain"], rtol=1e-9, err_msg=str((tag, i)))
    _check_counters(tag, out, i, ref)
    rows = ref["chain"][n_burn - 1:]
    s2 = ref["s2chain"]
    got = (out["mean"][i][:npar], out["std"][i][:npar], out["sig"][i][0], out["sig"][i][1])
    want = (rows.mean(axis=0), rows.std(axis=0), np.sqrt(s2.mean()), np.sqrt(s2).std())
    tols = [(0, 1e-7), (1e-6, 1e-7), (1e-9, 0), (1e-8, 0)] if atol is None else [(0, atol)] * 4
    for what, g, w, (rt, at) in zip(("mean", "std", "sig0", "sig1"), got, want, tols):
        np.testing.assert_allclose(g, w, rtol=rt, atol=at, err_msg=str((tag, i, what)))


def check_recorded_ss(cells, cc, out, ld):
    """The SS the sampler recorded for every stored row (n_burn = 1: row r of the chain is step r) is tc_ss_batch's."""
    nsimu = out["sschain"].shape[1]
    rows = out["chain"].reshape(-1, ld)
    ss = cells.ss_batch(np.repeat(cc, nsimu), rows)
    ref = out["sschain"].reshape(-1)
    rel = np.abs(ss - ref) / np.abs(ref)
    assert rel.max() <= 1e-14, rel.max()


def ld_mean_std(x):
    """Long-double two-pass mean and population std of the columns of x."""
    xl = x.astype(np.longdouble)
    m = xl.sum(axis=0) / x.shape[0]
    d = xl - m
    return m, np.sqrt((d * d).sum(axis=0) / x.shape[0])


def raw_run(cells, opts, cc, ins, uid, counters=True):
    """tc_mcmc_run through ctypes: (return code, message, outputs) — Cells.mcmc_run raises on TC_ESTATE and drops them.
    counters=False passes no counters buffer (NULL)."""
    need_gpu()
    nch, ld = cc.size, cells.ld
    arrs = [_lib.f64(x) for x in ins]
    out = dict(mean=np.zeros((nch, ld)), std=np.zeros((nch, ld)), sig=np.zeros((nch, 2)),
               counters=np.zeros((nch, _lib.NCOUNTERS), dtype=np.int64) if counters else None,
               chain=np.zeros((nch, opts.nsimu - opts.n_burn + 1, ld)), s2chain=np.zeros((nch, opts.nsimu)),
               flags=np.zeros((nch, opts.nsimu), dtype=np.int32), sschain=np.zeros((nch, opts.nsimu)))
    rp = _lib.Replay()
    rp.flags = out["flags"].ctypes.data
    rp.sschain = out["sschain"].ctypes.data
    L = _lib.load()
    rc = L.tc_mcmc_run(cells._h, C.byref(opts), nch, _lib.ptr(_lib.i32(cc)), _lib.ptr(np.ascontiguousarray(uid, dtype=np.uint64)),
                       ld, *[_lib.ptr(x) for x in arrs], _lib.ptr(out["mean"]), _lib.ptr(out["std"]), _lib.ptr(out["sig"]),
                       _lib.ptr(out["counters"]), _lib.ptr(out["chain"]), _lib.ptr(out["s2chain"]), C.byref(rp))
    return rc, L.tc_last_error().decode(), out
