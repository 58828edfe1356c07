"""GPU parity along the step axis: the chain lengths, burn-in rows, adaptation intervals and time slices where the samplers'
loops change shape, against the C oracle (oracle/tc_oracle.c), on every sampler layout.

test_gpu_lengths.py pins the samplers along the series-length axis.  Along the step axis dram_kernel generates 8 steps at a
time into a ring of 16 slots (8 under the big layout) and never lets a round cross an adaptation; dram_warp_kernel
generates 8 steps at a time (4 in replay mode); both cut a fit into time slices that are a multiple of adaptint (of 2 when
adaptint = 1, of 1 when adaptation is off) and park the chain between them; n_burn decides which rows the summaries and the stored chain start at
(chain_consts, flush_run, wk_flush).  Here:

  * replays with injected randomness, flag for flag, at nsimu below one batch / one ring, adaptint below a batch, at and
    beside the batch and ring sizes, adaptint = 0 and adaptint > nsimu, every adaptation inside burn-in (no covariance
    buffers), the largest interval with a full distinct-row buffer, a chain whose factorisations all fail, and every
    counter compared with the oracle's;
  * n_burn = 1 ... nsimu against the n_burn = 1 run and a long-double reduction of its rows, and the production (Philox)
    path against the oracle on the device's own streams;
  * a chain whose ss(theta0) is not finite inside a 16-chain group, through time slices;
  * std(sqrt(s2chain),1) where it is exactly 0 and over 200 000 rows.

Every case runs on two cells, N = 12 on an irregular grid and N = 129 on a regular one."""
import numpy as np
import pytest

from parity import (LAYOUTS, ORC_ADAPT, ORC_CHOL_FAIL, ORC_OOB, check_chain, check_recorded_ss, cols, dumped_streams,
                    ld_mean_std, make_cells, need_gpu, oracle_chains, raw_run, replay_streams)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def two_cells(orc):
    """(cells, packed): N = 12 on an irregular grid, N = 129 on a regular grid."""
    need_gpu()
    cells, packed = make_cells(orc[0], cols(orc, (12, 129), 4242))
    assert cells.N.tolist() == [12, 129]
    yield cells, packed
    cells.close()


def _inputs(cells, cc, seed, v0_chains=()):
    """chain_inputs for the chains cc; the chains listed in v0_chains get the loadPrevious bounds v0 +- 1e-5."""
    from transcriptioncycleinference_b200 import setup_cell
    rng = np.random.default_rng(seed)
    ins = [x.copy() for x in setup_cell.chain_inputs(cells, cc, rng)]
    for i in v0_chains:
        one = setup_cell.chain_inputs(cells, cc[i:i + 1], rng, v0=np.array([1.0 + rng.random()]))
        for x, y in zip(ins, one):
            x[i] = y[0]
    return ins


# ------------------------------------------------------------------------------------------------ 1. schedule replays
# (nsimu, burnintime, adaptint, extra options)
SCHEDULES = ([(n, 0, 100, {}) for n in (1, 2, 3, 5, 8, 9)] +              # no step at all, or less than one batch
             [(n, 0, 100, {}) for n in (16, 17, 24, 25)] +                 # ring wrap (16 slots; 8 in the big layout)
             [(40, 0, 1, {}), (40, 20, 1, {})] +                           # adaptation after every step; burn-in scaling every step
             [(9, 0, 1, {}), (25, 0, 1, {}), (25, 10, 1, {})] +            # ... with slices of 2 steps: the first block is rows 0, 1
             [(100, 50, 3, {}), (100, 50, 7, {}), (100, 50, 7, dict(burnin_cumulative=0))] +   # interval shorter than a batch
             [(200, 64, m, {}) for m in (8, 9, 16, 17)] +                  # at and beside the batch and ring sizes
             [(300, 100, 100, {}),                                         # adaptation at isimu = nsimu
              (330, 301, 100, {}),                                         # every adaptation in burn-in: no covariance buffers
              (330, 0, 0, {}),                                             # no adaptation: slices of 11 steps, cut mid-batch
              (330, 0, 500, {}),                                           # adaptint > nsimu: one slice, no covariance buffers
              (4200, 0, 2048, dict(tiny_j0=True))])                        # largest block; one chain fills the distinct-row buffer


def _sid(s):
    n, b, m, x = s
    return "n%d-b%d-a%d%s" % (n, b, m, "".join("-" + k for k in sorted(x)))


def _replay_all_layouts(orc, cells, packed, cc, ins, nsimu, burn, adaptint, dev_kw, orc_kw, seed, extra_check=None):
    _lib = need_gpu()
    co, _ = orc
    ld = cells.ld
    st = replay_streams(cells.N[cc], nsimu, ld, seed)
    refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, adaptint=adaptint, **orc_kw), ins, st)
    for layout, name in LAYOUTS:
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, adaptint=adaptint, n_burn=1, store_chain=1, replay=1,
                                 layout=layout, **dev_kw)
        out = cells.mcmc_run(opts, cc, *ins, replay=st, want_flags=True)
        for i, ref in enumerate(refs):
            check_chain(name, out, i, ref, 7 + int(cells.N[cc[i]]))
        check_recorded_ss(cells, cc, out, ld)
        if extra_check is not None:
            extra_check(name, out, refs)
    return refs


@pytest.mark.parametrize("sched", SCHEDULES, ids=[_sid(s) for s in SCHEDULES])
def test_schedule_replay(orc, two_cells, sched):
    """Four chains (two per cell) replayed with injected randomness and qcovadj_always = 1 on every layout: flags, rows,
    s2chain, sschain, the seven counters, and the recorded SS of every row."""
    _lib = need_gpu()
    nsimu, burn, adaptint, extra = sched
    cells, packed = two_cells
    cc = np.array([0, 1, 0, 1], dtype=np.int32)
    ins = _inputs(cells, cc, 10 + nsimu + adaptint)
    kw = {k: v for k, v in extra.items() if k != "tiny_j0"}
    check = None
    if extra.get("tiny_j0"):
        # J0 ~ 1e-20: the proposals barely move the state, nearly every step accepts, and the 2048 rows of the first
        # covariance block are nearly all distinct (the distinct-row buffer holds adaptint rows)
        ins[1][1, :] = 1e-20

        def check(name, out, refs):
            acc = int(np.sum(out["flags"][1][1:adaptint] & 1))
            assert acc >= 0.95 * (adaptint - 1), (name, acc)
            assert out["counters"][1][_lib.CNT_ADAPTATIONS] == refs[1]["counters"][ORC_ADAPT] == 2
    _replay_all_layouts(orc, cells, packed, cc, ins, nsimu, burn, adaptint, dict(qcovadj_always=1, **kw),
                        dict(qcovadj_always=1, **kw), 20 + nsimu + adaptint, check)


def test_frozen_chain_every_factorisation_fails(orc, two_cells):
    """low = upp = theta0 with qcovadj = 0 on the default path: every proposal is out of bounds, the covariance is exactly
    zero, chol(cov) and chol(cov + 0 I) both fail at every adaptation, so the failure count is the oracle's (nonzero) and
    no adaptation is counted: the proposal factor stays the diagonal one."""
    cells, packed = two_cells
    cc = np.array([0, 1], dtype=np.int32)
    ins = _inputs(cells, cc, 77)
    ins[2] = ins[0].copy(); ins[3] = ins[0].copy()
    nsimu, burn = 330, 100
    refs = _replay_all_layouts(orc, cells, packed, cc, ins, nsimu, burn, 100, dict(qcovadj=0.0), dict(qcovadj=0.0), 78)
    for ref in refs:
        assert ref["counters"][ORC_CHOL_FAIL] == 3 and ref["counters"][ORC_ADAPT] == 0
        assert ref["counters"][ORC_OOB] == 2 * (nsimu - 1)


# ------------------------------------------------------------------------------------------------ 2. n_burn and Philox
@pytest.mark.parametrize("layout,name", LAYOUTS, ids=[n for _, n in LAYOUTS])
def test_n_burn_sweep_against_oracle(orc, two_cells, layout, name):
    """One production (Philox) run of nsimu = 100, adaptint = 3, burn-in 30: slices of a few steps on both kernels.  It is the
    oracle's chain on the device's dumped streams; then every n_burn = 1 ... 100 stores rows n_burn-1 ... of it bit for bit,
    leaves flags, s2chain, sig and the counters alone, and reports the mean / population std of those rows (long-double
    two-pass: mean within 1e-13 max|x|, std within 1e-10 relative + 1e-13 max|x|).  Chains 2 and 3 have v confined to
    v0 +- 1e-5 (loadPrevious), so their std / |mean| is ~1e-6."""
    _lib = need_gpu()
    co, _ = orc
    cells, packed = two_cells
    cc = np.array([0, 1, 0, 1], dtype=np.int32)
    uid = np.array([11, 12, 13, 1 << 40], dtype=np.uint64)
    ins = _inputs(cells, cc, 300, v0_chains=(2, 3))
    nsimu, burn, adaptint, seed = 100, 30, 3, 777
    kw = dict(nsimu=nsimu, burnintime=burn, adaptint=adaptint, store_chain=1, seed=seed, layout=layout, qcovadj_always=1)
    base = cells.mcmc_run(_lib.default_opts(n_burn=1, **kw), cc, *ins, chain_uid=uid, want_flags=True)
    refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, adaptint=adaptint, qcovadj_always=1), ins,
                         dumped_streams(cells.N[cc], uid, seed, nsimu))
    for i, ref in enumerate(refs):
        check_chain(name, base, i, ref, 7 + int(cells.N[cc[i]]))
    worst = [0.0, 0.0]
    for nb in range(1, nsimu + 1):
        out = cells.mcmc_run(_lib.default_opts(n_burn=nb, **kw), cc, *ins, chain_uid=uid, want_flags=True)
        assert np.array_equal(out["chain"], base["chain"][:, nb - 1:]), (name, nb)
        for k in ("flags", "s2chain", "sig"):
            assert np.array_equal(out[k], base[k]), (name, nb, k)
        assert np.array_equal(out["counters"][:, :8], base["counters"][:, :8]), (name, nb)
        for i, c in enumerate(cc):
            npar = 7 + int(cells.N[c])
            rows = base["chain"][i, nb - 1:, :npar]
            m, s = ld_mean_std(rows)
            scale = np.abs(rows).max(axis=0)
            em = np.abs(out["mean"][i, :npar] - m).astype(np.float64)
            es = np.abs(out["std"][i, :npar] - s).astype(np.float64)
            assert np.all(em <= 1e-13 * scale), (name, nb, i, int(np.argmax(em / scale)), float(np.max(em / scale)))
            assert np.all(es <= 1e-10 * s.astype(np.float64) + 1e-13 * scale), (name, nb, i, int(np.argmax(es / scale)))
            worst[0] = max(worst[0], float(np.max(em / scale))); worst[1] = max(worst[1], float(np.max(es / scale)))
            assert np.all(out["mean"][i, npar:] == 0) and np.all(out["std"][i, npar:] == 0)
    v = base["chain"][2:, :, 0]
    assert np.all(v.std(axis=1) / np.abs(v.mean(axis=1)) < 1e-5)
    print("%s: n_burn 1..%d, max |mean err| / max|x| %.3g, max |std err| / max|x| %.3g" % (name, nsimu, worst[0], worst[1]))


PHILOX_SCHEDULES = [(25, 0, 100), (9, 0, 1), (40, 20, 1), (100, 50, 7), (200, 64, 9), (330, 0, 0), (330, 301, 100)]


@pytest.mark.parametrize("sched", PHILOX_SCHEDULES, ids=["n%d-b%d-a%d" % s for s in PHILOX_SCHEDULES])
def test_production_schedule_against_oracle(orc, two_cells, sched):
    """The production path generates 8 steps per batch on both kernels (dram_warp_kernel's replay batch is 4): schedules of
    section 1 on the device's Philox streams, every layout, against the oracle on tc_rng_dump's streams, with n_burn = 1
    and n_burn in the middle of a slice."""
    _lib = need_gpu()
    co, _ = orc
    nsimu, burn, adaptint = sched
    cells, packed = two_cells
    cc = np.array([0, 1, 1, 0], dtype=np.int32)
    uid = np.array([5, 6, 7, 8], dtype=np.uint64) + np.uint64(nsimu * 1000 + adaptint)
    ins = _inputs(cells, cc, 40 + nsimu)
    seed = 31337
    refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, adaptint=adaptint, qcovadj_always=1), ins,
                         dumped_streams(cells.N[cc], uid, seed, nsimu))
    nb = max(1, (2 * nsimu) // 3 + 1)
    for layout, name in LAYOUTS:
        for n_burn in sorted({1, nb}):
            opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, adaptint=adaptint, n_burn=n_burn, store_chain=1,
                                     seed=seed, layout=layout, qcovadj_always=1)
            out = cells.mcmc_run(opts, cc, *ins, chain_uid=uid, want_flags=True)
            for i, ref in enumerate(refs):
                check_chain("%s n_burn=%d" % (name, n_burn), out, i, ref, 7 + int(cells.N[cc[i]]), first_row=n_burn - 1)


# ------------------------------------------------------------------------------------------------ 3. ss(theta0) not finite
@pytest.mark.parametrize("layout,name", LAYOUTS, ids=[n for _, n in LAYOUTS])
def test_nonfinite_ss0_chain_inside_a_group(orc, two_cells, layout, name):
    """Chain 7 of 16 (the middle of one chain-per-warp group) starts at A = 1e200 (upp = 1e300, flat prior on A): its squared
    residual overflows, so ss(theta0) = inf (checked with the oracle).  Over 32 time slices the call returns TC_ESTATE naming
    that chain, the chain reports zeros and status 1, and every other chain's outputs are bit-identical to a run of the
    other 15 chains alone with the same chain_uids."""
    _lib = need_gpu()
    co, cons = orc
    cells, packed = two_cells
    bad = 7
    cc = (np.arange(16) % 2).astype(np.int32)
    uid = np.arange(16, dtype=np.uint64) * np.uint64(97) + np.uint64(3)
    ins = _inputs(cells, cc, 500)
    ins[0][bad, 5] = 1e200; ins[3][bad, 5] = 1e300
    assert np.isinf(ins[5][bad, 5])
    c = int(cc[bad]); N = int(cells.N[c]); o = int(cells.off[c])
    assert co.ss(cons, packed["t"][o:o + N], packed["ms2"][o:o + N], packed["pp7"][o:o + N], ins[0][bad, :7 + N]) == np.inf
    opts = _lib.default_opts(nsimu=3200, burnintime=1000, n_burn=1000, store_chain=1, seed=99, layout=layout, qcovadj_always=1)
    rc, msg, out = raw_run(cells, opts, cc, ins, uid)
    assert rc == _lib.TC_ESTATE and ("chain %d" % bad) in msg, (rc, msg)
    assert np.all(out["mean"][bad] == 0) and np.all(out["std"][bad] == 0) and np.all(out["sig"][bad] == 0)
    assert out["counters"][bad, _lib.CNT_STATUS] == 1 and np.all(out["counters"][bad, _lib.CNT_ACC_STAGE1:_lib.CNT_STATUS] == 0), out["counters"][bad]
    keep = np.array([i for i in range(16) if i != bad])
    rc2, msg2, ref = raw_run(cells, opts, cc[keep], [x[keep] for x in ins], uid[keep])
    assert rc2 == 0, msg2
    for k in ("mean", "std", "sig", "chain", "s2chain", "flags", "sschain"):
        assert np.array_equal(out[k][keep], ref[k]), (name, k)
    assert np.array_equal(out["counters"][keep, :8], ref["counters"][:, :8])
    assert np.all(ref["counters"][:, _lib.CNT_STATUS] == 0) and np.all(ref["sig"][:, 0] > 0)


# ------------------------------------------------------------------------------------------------ 4. std(sqrt(s2chain),1)
@pytest.mark.parametrize("sigma2", [0.3, 123.4])
def test_sigma_sigma_is_zero_with_fixed_sigma2(two_cells, sigma2):
    """updatesigma = 0: every row of s2chain is sigma2_0, so std(sqrt(s2chain),1) is 0 and sqrt(mean(s2chain)) is
    sqrt(sigma2_0).  20 000 rows: sig[1] <= 1e-14 sig[0], sig[0] within 1e-11 relative."""
    _lib = need_gpu()
    cells, _ = two_cells
    cc = np.array([0, 1], dtype=np.int32)
    ins = _inputs(cells, cc, 600)
    for layout, name in LAYOUTS:
        opts = _lib.default_opts(nsimu=20000, burnintime=1000, n_burn=20000, updatesigma=0, sigma2_0=sigma2, seed=5,
                                 layout=layout, qcovadj_always=1)
        out = cells.mcmc_run(opts, cc, *ins)
        s0 = np.sqrt(sigma2)
        print("%s sigma2_0 = %g: sig[0] rel err %.3g, sig[1] / sig[0] %.3g" % (name, sigma2, np.max(np.abs(out["sig"][:, 0] - s0)) / s0,
                                                                        np.max(out["sig"][:, 1] / out["sig"][:, 0])))
        assert np.all(np.abs(out["sig"][:, 0] - s0) <= 1e-11 * s0), (name, out["sig"])
        assert np.all(out["sig"][:, 1] <= 1e-14 * out["sig"][:, 0]), (name, out["sig"])


@pytest.mark.parametrize("N0", [1.0, 1e6])
def test_sigma_sigma_long_run(two_cells, N0):
    """updatesigma = 1, 200 000 rows (s2chain stored, n_burn = nsimu so the chain is one row): sig[1] within 1e-12 relative of
    a long-double two-pass std of sqrt(s2chain), sig[0] of sqrt(mean(s2chain)).  N0 = 1e6 (a prior on sigma2 worth 1e6
    observations) makes s2chain narrow: std / mean of sqrt(s2) ~ 1e-3, where a difference of running moments cancels most."""
    _lib = need_gpu()
    cells, _ = two_cells
    cc = np.array([0, 1], dtype=np.int32)
    ins = _inputs(cells, cc, 700)
    nsimu = 200000
    for layout, name in LAYOUTS:
        opts = _lib.default_opts(nsimu=nsimu, burnintime=10000, n_burn=nsimu, store_chain=1, seed=6, layout=layout,
                                 qcovadj_always=1, N0=N0)
        out = cells.mcmc_run(opts, cc, *ins)
        for i in range(cc.size):
            s2 = out["s2chain"][i].astype(np.longdouble)
            m, s = ld_mean_std(np.sqrt(s2)[:, None])
            rel1 = float(abs(out["sig"][i, 1] - s[0]) / s[0])
            rel0 = float(abs(out["sig"][i, 0] - np.sqrt(s2.mean())) / np.sqrt(s2.mean()))
            print("%s N0 = %g chain %d: sig[1] = %.17g, reference %.17g, rel err %.3g; sig[0] rel err %.3g" % (name, N0, i, out["sig"][i, 1], float(s[0]), rel1, rel0))
            assert rel1 <= 1e-12, (name, i, rel1)
            assert rel0 <= 1e-12, (name, i, rel0)
