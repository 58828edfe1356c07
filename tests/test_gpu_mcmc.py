"""GPU parity of the device-resident DRAM sampler, through the C ABI, against the CPU oracle.

mcmcstat records no proposals and the reference sets no RNG seed (SURVEY 0.1 #16, 7.3 #2), so
"replaying the reference's recorded proposals" is realised as: the SAME randomness (z1,u1,z2,u2,
chi2 per step) is fed to the oracle's DRAM restatement and to the GPU kernel; accept/reject flags
must be identical and the chains equal to rounding.

Short replays (burn-in of a few hundred steps) factor covariances of fewer distinct rows than parameters.  Those
are singular, and whether chol(cov) "succeeds" on such a matrix is decided by rounding noise, so these tests set
qcovadj_always = 1 (always factor cov + qcovadj I) on both sides.  The default path (mcmcstat: chol(cov) first,
+ qcovadj I only when that fails) is replayed where the covariance is well conditioned
(test_replay_long_default_path) and where chol(cov) fails for certain (test_singular_covariance_falls_back)."""
import numpy as np
import pytest

from parity import LAYOUTS, check_chain, dumped_streams, oracle_chains, raw_run, replay_streams
from transcriptioncycleinference_b200 import _lib

pytestmark = pytest.mark.gpu
SHORT = dict(qcovadj_always=1)


def _setup(gpu_cells, chain_cell, seed):
    from transcriptioncycleinference_b200 import setup_cell
    rng = np.random.default_rng(seed)
    return setup_cell.chain_inputs(gpu_cells, chain_cell, rng)


@pytest.mark.parametrize("algo,layout", [(_lib.ALGO_TOEPLITZ, _lib.LAYOUT_AUTO), (_lib.ALGO_PAIRS, _lib.LAYOUT_AUTO),
                                         (_lib.ALGO_TOEPLITZ, _lib.LAYOUT_WARP), (_lib.ALGO_PAIRS, _lib.LAYOUT_WARP)])
def test_replay_accept_reject_identical(gpu_cells, cells_npz, orc, algo, layout):
    """600 steps with burn-in 300: covers burn-in, the first covariance adaptation (Cholesky of
    the 300-row covariance) and three later ones.  TC_LAYOUT_AUTO: one CTA per chain (dram_kernel), TC_LAYOUT_WARP: one warp
    per chain (dram_warp_kernel)."""
    co, _ = orc
    chain_cell = np.array([0, 5, 77, 150, 298, 42], dtype=np.int32)
    nsimu, burn = 600, 300
    inputs = _setup(gpu_cells, chain_cell, 11)
    st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 12)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, algo=algo, layout=layout, **SHORT)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, replay=st, want_flags=True)
    refs = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT), inputs, st)
    for i, ref in enumerate(refs):
        npar = 7 + int(cells_npz["N"][chain_cell[i]])
        check_chain("algo %d layout %d" % (algo, layout), out, i, ref, npar)
        assert out["counters"][i][_lib.CNT_ADAPTATIONS] == 4
        # summaries = mean / population std of the stored rows (TranscriptionCycleMCMC.m:286-303)
        np.testing.assert_allclose(out["mean"][i][:npar], ref["chain"].mean(axis=0), rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(out["std"][i][:npar], ref["chain"].std(axis=0), rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(out["sig"][i][0], np.sqrt(ref["s2chain"].mean()), rtol=1e-9)
        np.testing.assert_allclose(out["sig"][i][1], np.sqrt(ref["s2chain"]).std(), rtol=1e-8)


def test_production_rng_equals_replay_of_its_own_dump(gpu_cells, cells_npz, orc):
    """Philox path: dump the device's streams for (seed, uid), feed them to the ORACLE, compare with
    the production (non-replay) run."""
    co, _ = orc
    chain_cell = np.array([3, 200], dtype=np.int32)
    uid = np.array([1000003, 77], dtype=np.uint64)
    nsimu, burn, seed = 400, 200, 987654321
    inputs = _setup(gpu_cells, chain_cell, 21)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, seed=seed, **SHORT)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, chain_uid=uid, want_flags=True)
    Ns = cells_npz["N"][chain_cell]
    st = dumped_streams(Ns, uid, seed, nsimu)
    for i, N in enumerate(Ns):
        # sanity of the streams themselves
        assert abs(st["z1"][i][1:].mean()) < 0.02 and abs(st["z1"][i][1:].std() - 1) < 0.02
        assert 0 < st["u1"][i].min() and st["u1"][i].max() < 1
        assert abs(st["chi2"][i][1:].mean() / (1 + 2 * int(N)) - 1) < 0.02
    refs = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT), inputs, st)
    for i, ref in enumerate(refs):
        check_chain("philox", out, i, ref, 7 + int(Ns[i]))


def test_results_independent_of_partition(gpu_cells):
    """Philox draws are keyed by (seed, chain_uid): running a chain alone or inside a larger batch
    gives bit-identical output (this is what makes the output independent of the GPU count)."""
    cc = np.array([10, 20, 30, 40], dtype=np.int32)
    uid = np.array([10, 20, 30, 40], dtype=np.uint64)
    inputs = _setup(gpu_cells, cc, 31)
    opts = _lib.default_opts(nsimu=300, burnintime=100, n_burn=50)
    full = gpu_cells.mcmc_run(opts, cc, *inputs, chain_uid=uid)
    sub = gpu_cells.mcmc_run(opts, cc[2:3], *[x[2:3] for x in inputs], chain_uid=uid[2:3])
    assert np.array_equal(full["mean"][2], sub["mean"][0])
    assert np.array_equal(full["sig"][2], sub["sig"][0])


def test_solo_sm_scheduling_is_transparent(gpu_cells, monkeypatch):
    """With about as many chains as CTA slots the CTA-per-chain kernel lets a lagging chain take its SM (the neighbour CTA
    gives way at its next slice boundary, csrc/tc_mcmc.cu: smctl).  That is scheduling only: 299 chains x 6 000 steps give
    bit-identical summaries and counters with the rule off (TC_SOLO_LAG=0), at its default, and at its most eager setting
    with many short slices."""
    cc = np.arange(299, dtype=np.int32)
    inputs = _setup(gpu_cells, cc, 77)
    opts = _lib.default_opts(nsimu=6000, burnintime=1000, n_burn=1000)
    outs = []
    for lag, nseg in (("0", "32"), (None, None), ("1", "512")):
        for k, v in (("TC_SOLO_LAG", lag), ("TC_NSEG", nseg)):
            if v is None:
                monkeypatch.delenv(k, raising=False)
            else:
                monkeypatch.setenv(k, v)
        outs.append(gpu_cells.mcmc_run(opts, cc, *inputs))
    for o in outs[1:]:
        assert np.array_equal(o["mean"], outs[0]["mean"])
        assert np.array_equal(o["std"], outs[0]["std"])
        assert np.array_equal(o["sig"], outs[0]["sig"])
        assert np.array_equal(o["counters"][:, :8], outs[0]["counters"][:, :8])      # the rest are cycle counts


def test_chain_layout_and_bounds(gpu_cells, cells_npz):
    """Row 1 = x0, s2chain(1) = sigma2_0 = 1, n_steps - n_burn + 1 stored rows, samples inside the
    bounds (SURVEY 0.1 #7, 4.2)."""
    cc = np.arange(0, 299, 23, dtype=np.int32)
    inputs = _setup(gpu_cells, cc, 41)
    th0, q, lo, hi, mu, sg = inputs
    opts = _lib.default_opts(nsimu=500, burnintime=200, n_burn=200, store_chain=1)
    out = gpu_cells.mcmc_run(opts, cc, *inputs)
    assert out["chain"].shape == (len(cc), 301, gpu_cells.ld)
    assert np.all(out["s2chain"][:, 0] == 1.0)
    for i, c in enumerate(cc):
        npar = 7 + int(cells_npz["N"][c])
        ch = out["chain"][i][:, :npar]
        assert np.all(ch >= lo[i, :npar]) and np.all(ch <= hi[i, :npar])
        np.testing.assert_allclose(out["mean"][i][:npar], ch.mean(axis=0), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(out["std"][i][:npar], ch.std(axis=0), rtol=1e-8, atol=1e-10)
    opts1 = _lib.default_opts(nsimu=50, burnintime=10, n_burn=1, store_chain=1)
    out1 = gpu_cells.mcmc_run(opts1, cc, *inputs)
    for i, c in enumerate(cc):
        npar = 7 + int(cells_npz["N"][c])
        assert np.array_equal(out1["chain"][i][0, :npar], th0[i, :npar])
    acc = out["counters"][:, _lib.CNT_ACC_STAGE1] + out["counters"][:, _lib.CNT_ACC_STAGE2]
    assert np.all(acc > 0)


def test_time_slices_are_transparent(gpu_cells, cells_npz, orc):
    """Chains are time-sliced over the persistent CTAs (state parked in HBM between slices).  With
    nsimu = 3300 a slice is 200 steps = two adaptation intervals, and there are 17 park/resume
    cycles: the production run must still be the oracle's chain on the device's own Philox streams
    (regression: the parked phase clocks once overlapped x[0])."""
    co, _ = orc
    chain_cell = np.array([0, 250], dtype=np.int32)
    uid = np.array([0, 250 << 20], dtype=np.uint64)
    nsimu, burn, seed = 3300, 1000, 20201028
    inputs = _setup(gpu_cells, chain_cell, 51)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, seed=seed, **SHORT)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, chain_uid=uid, want_flags=True)
    assert np.all(out["counters"][:, [_lib.CNT_CYCLES0 + 3, _lib.CNT_CYCLES0 + 4, _lib.CNT_CYCLES0 + 6]] == 0)   # phases dram_kernel does not time
    Ns = cells_npz["N"][chain_cell]
    refs = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT), inputs,
                         dumped_streams(Ns, uid, seed, nsimu))
    for i, ref in enumerate(refs):
        check_chain("time slices", out, i, ref, 7 + int(Ns[i]))


@pytest.mark.parametrize("variant", [
    dict(ntry=1),                                   # plain adaptive Metropolis, no delayed rejection
    dict(updatesigma=0),                            # sigma2 fixed at sigma2_0
    dict(burnin_cumulative=0),                      # burn-in scaling on the rejection rate since the last adaptation
    dict(adaptint=64, drscale=3.0, qcovadj=1e-6),   # other adaptation interval / DR scale / regulariser
])
@pytest.mark.parametrize("layout", [l for l, _ in LAYOUTS], ids=[n for _, n in LAYOUTS])
def test_replay_option_variants(gpu_cells, cells_npz, orc, variant, layout):
    """Every tc_mcmc_opts field that changes the DRAM arithmetic, replayed against the oracle with the same
    injected randomness on every sampler layout: flags, rows, s2chain, sschain and every counter."""
    co, _ = orc
    chain_cell = np.array([7, 123, 250], dtype=np.int32)
    nsimu, burn = 420, 150
    inputs = _setup(gpu_cells, chain_cell, 61)
    st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 62)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, layout=layout, **SHORT, **variant)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, replay=st, want_flags=True)
    refs = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT, **variant), inputs, st)
    for i, ref in enumerate(refs):
        check_chain((variant, layout), out, i, ref, 7 + int(cells_npz["N"][chain_cell[i]]))


def test_posterior_means_agree_with_independent_cpu_chains(gpu_cells, cells_npz, orc):
    """north_star's second correctness criterion — posterior means of v, tau, t_on, R (and sigma) agree within Monte
    Carlo standard error — against the only long reference-algorithm chains that can exist here: the CPU oracle's,
    run with ITS OWN random numbers (xorshift, not Philox).  12 chains per side on each of 3 cells, same x0 per
    chain index; the standard error is the between-chain one, the bound is 4 combined standard errors."""
    co, cons = orc
    cells3 = np.array([12, 150, 270], dtype=np.int32)
    per = 12
    cc = np.repeat(cells3, per)
    nsimu, burn = 5000, 2500
    inputs = _setup(gpu_cells, cc, 71)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=burn, seed=4242)
    gpu = gpu_cells.mcmc_run(opts, cc, *inputs, chain_uid=np.arange(cc.size, dtype=np.uint64) + 900)
    cmean, _, csig, _ = co.run_chains(cons, cells_npz, co.default_opts(nsimu, burn), burn, cc, *inputs, seed=99, nthreads=0)
    for ci in range(cells3.size):
        s = slice(ci * per, (ci + 1) * per)
        for name, col in (("v", 0), ("tau", 1), ("ton", 2), ("R", 6)):
            g, c = gpu["mean"][s, col], cmean[s, col]
            se = np.sqrt(g.var(ddof=1) / per + c.var(ddof=1) / per)
            assert abs(g.mean() - c.mean()) <= 4.0 * se + 1e-9, (int(cells3[ci]), name, g.mean(), c.mean(), se)
        g, c = gpu["sig"][s, 0], csig[s, 0]
        se = np.sqrt(g.var(ddof=1) / per + c.var(ddof=1) / per)
        assert abs(g.mean() - c.mean()) <= 4.0 * se + 1e-9, (int(cells3[ci]), "sigma", g.mean(), c.mean(), se)


def test_big_layout_matches_oracle_and_regular_layout(gpu_cells, cells_npz, orc):
    """The large-series layout (TC_LAYOUT_BIG: what series with more than ~210 points get) forced onto TestData cells:
    (1) replay against the oracle over burn-in + 5 covariance adaptations, flags identical; (2) production Philox run,
    regular vs big layout: the two differ only in the rounding of the Cholesky factor (shared-memory right-looking vs
    left-looking through L2), so the accept/reject sequence and the counters must be identical and the means equal to rounding."""
    co, _ = orc
    chain_cell = np.array([0, 57, 130, 298], dtype=np.int32)
    inputs = _setup(gpu_cells, chain_cell, 21)
    nsimu, burn = 600, 200
    st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 22)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, layout=_lib.LAYOUT_BIG, **SHORT)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, replay=st, want_flags=True)
    refs = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT), inputs, st)
    for i, ref in enumerate(refs):
        check_chain("big", out, i, ref, 7 + int(cells_npz["N"][chain_cell[i]]))
        cnt = out["counters"][i]
        assert cnt[_lib.CNT_ADAPTATIONS] == 5 and cnt[_lib.CNT_CHOL_FAIL] == 0        # adaptations at 200..600, no Cholesky failure
    res = []
    for layout in (_lib.LAYOUT_AUTO, _lib.LAYOUT_BIG):
        opts = _lib.default_opts(nsimu=3000, burnintime=500, n_burn=500, layout=layout, seed=99, **SHORT)
        res.append(gpu_cells.mcmc_run(opts, chain_cell, *inputs, want_flags=True))
    assert np.array_equal(res[0]["flags"], res[1]["flags"])
    assert np.array_equal(res[0]["counters"][:, :8], res[1]["counters"][:, :8])
    np.testing.assert_allclose(res[0]["mean"], res[1]["mean"], rtol=0, atol=1e-6)


def test_replay_long_default_path(gpu_cells, cells_npz, orc):
    """One 20 000-step chain per layout against the C oracle with the same injected randomness, at the DEFAULT options
    (cumulative burn-in rule, chol(cov) first): burn-in of 5 000 steps (50 scaling decisions), then 150 covariance
    adaptations = 150 Cholesky factorisations of a well-conditioned covariance (>= 5 000 rows).  Flags identical over
    all 20 000 steps, chain equal to 1e-6 (150 factorisations in a different summation order), counters equal."""
    co, _ = orc
    nsimu, burn = 20000, 5000
    for c, layout in ((17, _lib.LAYOUT_AUTO), (211, _lib.LAYOUT_BIG), (250, _lib.LAYOUT_WARP)):
        chain_cell = np.array([c], dtype=np.int32)
        inputs = _setup(gpu_cells, chain_cell, 81 + layout)
        st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 82 + layout)
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, layout=layout)
        assert opts.burnin_cumulative == 1 and opts.qcovadj_always == 0
        out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, replay=st, want_flags=True)
        ref, = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn), inputs, st)
        check_chain("layout %d" % layout, out, 0, ref, 7 + int(cells_npz["N"][c]), atol=1e-6)
        cnt = out["counters"][0]
        assert cnt[_lib.CNT_ADAPTATIONS] == 151 and cnt[_lib.CNT_CHOL_FAIL] == 0


def test_replay_200_adaptations(gpu_cells, cells_npz, orc):
    """20 000 steps with a burn-in of 100: 199 covariance adaptations (VERDICT r1: nothing compared a long run with the
    oracle).  The early covariances are singular, so cov + qcovadj I is factored on both sides (see the module docstring)."""
    co, _ = orc
    nsimu, burn, c = 20000, 100, 123
    chain_cell = np.array([c], dtype=np.int32)
    inputs = _setup(gpu_cells, chain_cell, 91)
    st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 92)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, **SHORT)
    out = gpu_cells.mcmc_run(opts, chain_cell, *inputs, replay=st, want_flags=True)
    ref, = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn, **SHORT), inputs, st)
    check_chain("200 adaptations", out, 0, ref, 7 + int(cells_npz["N"][c]), atol=1e-6)
    assert out["counters"][0][_lib.CNT_ADAPTATIONS] == 200


def test_singular_covariance_falls_back(gpu_cells, cells_npz, orc):
    """A chain that cannot move (low = upp = theta0: every proposal is out of bounds) has an exactly zero covariance:
    chol(cov) fails for certain and the default path must fall back to chol(cov + qcovadj I) = sqrt(qcovadj) I, as
    mcmcstat's "try to blow it" branch does — not count a failed adaptation."""
    co, _ = orc
    chain_cell = np.array([5], dtype=np.int32)
    th0, q, lo, hi, mu, sg = _setup(gpu_cells, chain_cell, 95)
    ins = (th0, q, th0.copy(), th0.copy(), mu, sg)
    nsimu, burn = 400, 200
    st = replay_streams(cells_npz["N"][chain_cell], nsimu, gpu_cells.ld, 96)
    ref, = oracle_chains(orc, cells_npz, chain_cell, co.default_opts(nsimu, burn), ins, st)
    for layout in (_lib.LAYOUT_AUTO, _lib.LAYOUT_BIG, _lib.LAYOUT_WARP):
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, layout=layout)
        out = gpu_cells.mcmc_run(opts, chain_cell, *ins, replay=st, want_flags=True)
        check_chain("layout %d" % layout, out, 0, ref, 7 + int(cells_npz["N"][5]))
        assert out["counters"][0][_lib.CNT_ADAPTATIONS] == 3 and out["counters"][0][_lib.CNT_CHOL_FAIL] == 0


def test_input_validation_and_device_restored(gpu_cells):
    """mcmcstat refuses an initial value outside its bounds; a zero / NaN prior width would make the prior sum NaN and the
    chain would silently never accept: both are TC_EINVAL with the chain and parameter index.  ss(theta0) not finite is
    reported (TC_ESTATE) even when the caller does not ask for counters.  The caller's current device is left alone."""
    cc = np.array([1, 2], dtype=np.int32)
    th0, q, lo, hi, mu, sg = _setup(gpu_cells, cc, 5)
    opts = _lib.default_opts(nsimu=50, burnintime=20, n_burn=1)
    bad = th0.copy(); bad[1, 3] = hi[1, 3] + 1.0
    with pytest.raises(_lib.TcError, match=r"theta0 must lie inside \[low, upp\] \(chain 1, parameter 3\)"):
        gpu_cells.mcmc_run(opts, cc, bad, q, lo, hi, mu, sg)
    sg0 = sg.copy(); sg0[0, 9] = 0.0
    with pytest.raises(_lib.TcError, match=r"prior_sig must be > 0.*chain 0, parameter 9"):
        gpu_cells.mcmc_run(opts, cc, th0, q, lo, hi, mu, sg0)
    lo2 = lo.copy(); lo2[0, 0] = hi[0, 0] + 1.0
    with pytest.raises(_lib.TcError, match="low must be <= upp"):
        gpu_cells.mcmc_run(opts, cc, th0, q, lo2, hi, mu, sg)
    nan0 = th0.copy(); nan0[0, 6] = np.nan                      # NaN lies inside no bounds
    with pytest.raises(_lib.TcError, match=r"theta0 must lie inside"):
        gpu_cells.mcmc_run(opts, cc, nan0, q, lo, hi, mu, sg)
    # TC_ESTATE without a counters buffer (the ABI called directly with counters = NULL): chain 0 starts at A = 1e200
    # (upp = 1e300, flat prior on A), so its squared residual overflows and ss(theta0) = inf
    inf0 = th0.copy(); inf0[0, 5] = 1e200
    hi0 = hi.copy(); hi0[0, 5] = 1e300
    assert np.isinf(sg[0, 5])
    rc, msg, _ = raw_run(gpu_cells, opts, cc, (inf0, q, lo, hi0, mu, sg), np.arange(cc.size, dtype=np.uint64), counters=False)
    assert rc == _lib.TC_ESTATE and "chain 0" in msg, (rc, msg)
    try:
        import torch
        if torch.cuda.device_count() >= 1:
            torch.cuda.set_device(0)
            gpu_cells.mcmc_run(opts, cc, th0, q, lo, hi, mu, sg)
            assert torch.cuda.current_device() == 0
    except ImportError:
        pass


def test_warp_kernel_production_path(gpu_cells, cells_npz, orc):
    """dram_warp_kernel (one warp per chain: what thousands of chains get, BASELINE config 3) on its production path:
    (1) Philox streams: the chain is the oracle's on the device's dumped randomness, through 16 park/resume slices and with
    more chains than one CTA holds (two groups of 16 + a ragged one); (2) the same chains through dram_kernel: identical
    accept/reject sequence and counters, means equal to rounding (the two kernels factor the covariance in different orders);
    (3) option variants the warp kernel implements separately: ntry = 1, updatesigma = 0, a bounds vector without the
    reference's head + block structure (generic path)."""
    co, _ = orc
    cc = np.arange(0, 296, 8, dtype=np.int32)                     # 37 chains of different cells
    uid = cc.astype(np.uint64) * np.uint64(1 << 20) + np.uint64(3)
    nsimu, burn, seed = 3300, 1000, 20201028
    inputs = _setup(gpu_cells, cc, 101)
    res = {}
    for layout in (_lib.LAYOUT_WARP, _lib.LAYOUT_AUTO):
        # 1 000-row covariances of ~130 parameters are nearly singular: chol(cov) without the regulariser amplifies the
        # rounding differences between the kernels' factorisations to 1e-3 in the chain (measured), so: SHORT
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, seed=seed, layout=layout, **SHORT)
        res[layout] = gpu_cells.mcmc_run(opts, cc, *inputs, chain_uid=uid, want_flags=True)
    warp, auto = res[_lib.LAYOUT_WARP], res[_lib.LAYOUT_AUTO]
    assert np.array_equal(warp["flags"], auto["flags"])
    assert np.array_equal(warp["counters"][:, :8], auto["counters"][:, :8])
    assert np.array_equal(warp["counters"][:, _lib.CNT_CYCLES0 + 7], warp["counters"][:, _lib.CNT_SS_EVALS])
    np.testing.assert_allclose(warp["mean"], auto["mean"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(warp["sig"], auto["sig"], rtol=1e-9)
    sel = [0, 17, 36]
    refs = oracle_chains(orc, cells_npz, cc[sel], co.default_opts(nsimu, burn, **SHORT), [x[sel] for x in inputs],
                         dumped_streams(cells_npz["N"][cc[sel]], uid[sel], seed, nsimu))
    for i, ref in zip(sel, refs):
        check_chain("warp philox", warp, i, ref, 7 + int(cells_npz["N"][cc[i]]))
    th0, q, lo, hi, mu, sg = [x[:3].copy() for x in inputs]
    lo[:, 40] = -25.0; sg[:, 55] = 10.0                          # breaks the head + block structure
    for variant in (dict(ntry=1), dict(updatesigma=0), dict()):
        a = gpu_cells.mcmc_run(_lib.default_opts(nsimu=700, burnintime=300, n_burn=1, seed=5, layout=_lib.LAYOUT_WARP, **SHORT, **variant), cc[:3], th0, q, lo, hi, mu, sg, want_flags=True)
        b = gpu_cells.mcmc_run(_lib.default_opts(nsimu=700, burnintime=300, n_burn=1, seed=5, layout=_lib.LAYOUT_AUTO, **SHORT, **variant), cc[:3], th0, q, lo, hi, mu, sg, want_flags=True)
        assert np.array_equal(a["flags"], b["flags"]), variant
        np.testing.assert_allclose(a["mean"], b["mean"], rtol=0, atol=1e-6)


def test_philox_variates_pass_ks(gpu_cells):
    """The sampling variates are the one place single precision enters (DESIGN.md 2): the proposal normals and the normal
    inside Marsaglia-Tsang's chi-square are Box-Muller in FP32 (32-bit radius uniform => |z| <= 6.76, 24-bit angle) widened
    to FP64; u1, u2 are 53-bit uniforms.  Stated tolerance: indistinguishable from N(0,1) / U(0,1) / chi2(nu) by
    Kolmogorov-Smirnov at 2.5e5 - 5e6 draws (p > 1e-3), moments within 4 standard errors, tails present up to 4.5 sigma,
    and no correlation between the two stages or consecutive steps."""
    from scipy import stats
    npar, nsimu, nu = 127, 20000, 241.0
    d = _lib.rng_dump(20201028, 123456789, npar, nu, nsimu)
    for k in ("z1", "z2"):
        z = d[k][1:].reshape(-1)
        assert stats.kstest(z[:500000], "norm").pvalue > 1e-3
        se = 1.0 / np.sqrt(z.size)
        assert abs(z.mean()) < 4 * se and abs(z.var() - 1) < 4 * np.sqrt(2.0) * se
        assert abs(stats.skew(z)) < 4 * np.sqrt(6.0) * se and abs(stats.kurtosis(z)) < 4 * np.sqrt(24.0) * se
        # tail mass against the exact normal: P(|z| > 4.5) = 6.8e-6 -> ~17 of 2.5e6
        n45 = int((np.abs(z) > 4.5).sum())
        assert 2 <= n45 <= 45 and np.abs(z).max() <= 6.77
    z1, z2 = d["z1"][1:], d["z2"][1:]
    assert abs(np.corrcoef(z1.reshape(-1), z2.reshape(-1))[0, 1]) < 4 / np.sqrt(z1.size)
    assert abs(np.corrcoef(z1[:-1].reshape(-1), z1[1:].reshape(-1))[0, 1]) < 4 / np.sqrt(z1.size)
    assert abs(np.corrcoef(z1[:, :-1].reshape(-1), z1[:, 1:].reshape(-1))[0, 1]) < 4 / np.sqrt(z1.size)
    for k in ("u1", "u2"):
        assert stats.kstest(d[k][1:], "uniform").pvalue > 1e-3
    c2 = d["chi2"][1:]
    assert stats.kstest(c2, "chi2", args=(nu,)).pvalue > 1e-3
    assert abs(c2.mean() / nu - 1) < 4 * np.sqrt(2.0 / nu / c2.size) and abs(c2.var() / (2 * nu) - 1) < 0.06
    # a second degrees-of-freedom value (N = 400: nu = 801) and an independent chain identity
    d2 = _lib.rng_dump(7, 42, 16, 801.0, 50000)
    assert stats.kstest(d2["chi2"][1:], "chi2", args=(801.0,)).pvalue > 1e-3
    assert stats.kstest(d2["z1"][1:].reshape(-1), "norm").pvalue > 1e-3
