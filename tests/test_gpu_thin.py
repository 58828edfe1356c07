"""Thinned raw chains (tc_mcmc_opts.thin = k): a fit that stores every k-th row returns chain[:, ::k] and s2chain[:, ::k] of
the fit that stores every row, bit for bit, and the same summaries and counters, on every sampler, schedule and GPU count.

chain keeps the 0-based rows n_burn-1 + j k and s2chain the rows j k; the run writers of both samplers (flush_run in
dram_kernel, wk_flush in dram_warp_kernel) write the kept rows of each run of equal rows, and a run that straddles the end
of a time slice is flushed in pieces, so nsimu = 2000 with adaptint = 9 (slices of 63 steps, ~32 per chain) puts kept rows
on both sides of many slice ends."""
import numpy as np
import pytest

from parity import LAYOUTS, check_chain, cols, make_cells, need_gpu, oracle_chains, raw_run, replay_streams
from transcriptioncycleinference_b200 import _lib

pytestmark = pytest.mark.gpu

NSIMU, ADAPTINT, SEED = 2000, 9, 20261023
BURNS = (1, 2, 613)                    # 613: a multiple of no k below and of no adaptint
UNSLICED = 4 * 296                     # tc_mcmc_run: dram_kernel stops slicing from this many chains on (TC_UNSLICED_CHAINS)
SUMMARY_KEYS = ("mean", "std", "sig")


def ks(nsimu, n_burn):
    return (2, 3, 7, 13, 100, nsimu - n_burn, nsimu - n_burn + 1, 2 ** 31 - 1)


def fit(cells, cc, ins, uid, **kw):
    opts = _lib.default_opts(**dict(dict(nsimu=NSIMU, burnintime=300, adaptint=ADAPTINT, store_chain=1, seed=SEED), **kw))
    return cells.mcmc_run(opts, cc, *ins, chain_uid=uid)


def assert_thinned(tag, out, full, k):
    """out stores every k-th row of full's chain: rows, s2chain, summaries and the seven counters + status bit for bit."""
    nkeep, ns2 = out["chain"].shape[1], out["s2chain"].shape[1]
    assert nkeep == (full["chain"].shape[1] - 1) // k + 1 and ns2 == (full["s2chain"].shape[1] - 1) // k + 1, (tag, k)
    assert np.array_equal(out["chain"], full["chain"][:, ::k]), (tag, k, "chain")
    assert np.array_equal(out["s2chain"], full["s2chain"][:, ::k]), (tag, k, "s2chain")
    for key in SUMMARY_KEYS:
        assert np.array_equal(out[key], full[key]), (tag, k, key)
    assert np.array_equal(out["counters"][:, :8], full["counters"][:, :8]), (tag, k, "counters")


@pytest.fixture(scope="module")
def mixed(orc):
    """Cells of N = 12, 61, 129 and 144 (irregular and regular grids), two chains each, with fixed inputs and uids."""
    need_gpu()
    from transcriptioncycleinference_b200 import setup_cell
    cells, packed = make_cells(orc[0], cols(orc, (12, 61, 129, 144), 9101))
    cc = np.repeat(np.arange(4, dtype=np.int32), 2)
    ins = setup_cell.chain_inputs(cells, cc, np.random.default_rng(9102))
    uid = np.arange(cc.size, dtype=np.uint64) * np.uint64(1 << 20) + np.uint64(5)
    yield cells, packed, cc, ins, uid
    cells.close()


# ------------------------------------------------------------------------------------------------ 1. every layout, k, n_burn
@pytest.mark.parametrize("n_burn", BURNS)
@pytest.mark.parametrize("layout,name", LAYOUTS, ids=[n for _, n in LAYOUTS])
def test_thinned_is_every_kth_row(mixed, layout, name, n_burn):
    """Philox production runs (seed, no replay) of 8 chains on mixed series lengths: thin = 1, then every k of ks(); each
    thinned fit is the full fit's chain[:, ::k], s2chain[:, ::k], and the same mean, std, sig and counters."""
    cells, _, cc, ins, uid = mixed
    full = fit(cells, cc, ins, uid, n_burn=n_burn, layout=layout)
    assert full["chain"].shape[1] == NSIMU - n_burn + 1 and full["s2chain"].shape[1] == NSIMU
    for k in ks(NSIMU, n_burn):
        assert_thinned("%s n_burn=%d" % (name, n_burn), fit(cells, cc, ins, uid, n_burn=n_burn, layout=layout, thin=k), full, k)


# ------------------------------------------------------------------------------------------------ 2. scheduler shapes
@pytest.mark.parametrize("case", [("cta-unsliced-1185", _lib.LAYOUT_CTA, lambda S: UNSLICED + 1),
                                  ("auto-warp-13S+1", _lib.LAYOUT_AUTO, lambda S: 13 * S + 1)], ids=lambda c: c[0])
def test_thinned_at_scheduler_chain_counts(gpu_cells, case):
    """Above TC_UNSLICED_CHAINS (dram_kernel, nothing sliced, a CTA takes any free chain) and above 13 chains per SM under AUTO
    (dram_warp_kernel, 16-chain groups parked and resumed): thin = 7 and 50 against thin = 1 on the TestData cells."""
    from transcriptioncycleinference_b200 import setup_cell
    name, layout, nc_of = case
    nc = nc_of(_lib.device_info(0)["sm_count"])
    cc = (np.arange(nc) % gpu_cells.ncells).astype(np.int32)
    ins = setup_cell.chain_inputs(gpu_cells, cc, np.random.default_rng(nc))
    uid = np.arange(nc, dtype=np.uint64) * np.uint64(1 << 20) + np.uint64(9)
    kw = dict(nsimu=500, burnintime=100, adaptint=100, n_burn=101, layout=layout)
    full = fit(gpu_cells, cc, ins, uid, **kw)
    for k in (7, 50):
        assert_thinned(name, fit(gpu_cells, cc, ins, uid, thin=k, **kw), full, k)


# ------------------------------------------------------------------------------------------------ 3. replay against the oracle
@pytest.mark.parametrize("layout,name", LAYOUTS, ids=[n for _, n in LAYOUTS])
def test_thinned_replay_against_oracle(orc, mixed, layout, name):
    """Injected randomness, thin = 3, n_burn = 5: the stored rows are the oracle's rows 4, 7, 10, ... and s2chain its rows 0, 3,
    6, ... (check_chain's tolerances); flags and sschain keep every step and are the oracle's."""
    co, _ = orc
    cells, packed, cc, ins, _ = mixed
    nsimu, burn, n_burn, k = 300, 100, 5, 3
    st = replay_streams(cells.N[cc], nsimu, cells.ld, 9103)
    refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, qcovadj_always=1), ins, st)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=n_burn, store_chain=1, replay=1, layout=layout,
                             qcovadj_always=1, thin=k)
    out = cells.mcmc_run(opts, cc, *ins, replay=st, want_flags=True)
    assert out["flags"].shape == (cc.size, nsimu) and out["sschain"].shape == (cc.size, nsimu)
    for i, ref in enumerate(refs):
        thinned = dict(ref, chain=ref["chain"][n_burn - 1::k], s2chain=ref["s2chain"][::k])
        check_chain(name, out, i, thinned, 7 + int(cells.N[cc[i]]))


# ------------------------------------------------------------------------------------------------ 4. several GPUs
def test_thinned_two_gpus_same_bytes(orc, mixed):
    """ngpus = 2, thin = 7 on TC_LAYOUT_CTA: the same bytes as one GPU (each device writes its chains at its own offsets of
    the thinned outputs), and every 7th row of the one-GPU thin = 1 fit."""
    if need_gpu().device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    from transcriptioncycleinference_b200.engine import Cells
    _, packed, cc, ins, uid = mixed
    cells = Cells.from_packed(packed["N"], packed["off"], packed["t"], packed["ms2"], packed["pp7"], devices=(0, 1))
    try:
        full = fit(cells, cc, ins, uid, n_burn=613, layout=_lib.LAYOUT_CTA, ngpus=1)
        one = fit(cells, cc, ins, uid, n_burn=613, layout=_lib.LAYOUT_CTA, ngpus=1, thin=7)
        two = fit(cells, cc, ins, uid, n_burn=613, layout=_lib.LAYOUT_CTA, ngpus=2, thin=7)
        assert_thinned("1 GPU", one, full, 7)
        for key in ("chain", "s2chain", "counters") + SUMMARY_KEYS:
            x, y = (one[key][:, :8], two[key][:, :8]) if key == "counters" else (one[key], two[key])
            assert np.array_equal(x, y), key
    finally:
        cells.close()


# ------------------------------------------------------------------------------------------------ 5. errors and store_chain = 0
@pytest.mark.parametrize("thin", [0, -1])
def test_thin_below_one_is_refused(mixed, thin):
    """store_chain with thin < 1: TC_EINVAL naming thin, before any device work, and the caller's current device as it was."""
    import torch
    cells, _, cc, ins, uid = mixed
    dev = _lib.device_count() - 1
    torch.cuda.set_device(dev)
    try:
        opts = _lib.default_opts(nsimu=100, burnintime=50, n_burn=50, store_chain=1, thin=thin)
        rc, msg, _ = raw_run(cells, opts, cc, ins, uid)
        assert rc == _lib.TC_EINVAL and "thin" in msg, (rc, msg)
        assert torch.cuda.current_device() == dev
    finally:
        torch.cuda.set_device(0)


def test_thin_ignored_without_stored_rows(mixed):
    """store_chain = 0 with thin = 5 runs and returns the summaries and counters of thin = 1."""
    cells, _, cc, ins, uid = mixed
    a = fit(cells, cc, ins, uid, n_burn=613, store_chain=0)
    b = fit(cells, cc, ins, uid, n_burn=613, store_chain=0, thin=5)
    assert a["chain"] is None and b["chain"] is None
    for key in SUMMARY_KEYS:
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(a["counters"][:, :8], b["counters"][:, :8])


# ------------------------------------------------------------------------------------------------ 6. the driver
def test_driver_thin(tmp_path, cells_npz):
    """TranscriptionCycleMCMC(..., 'thin', 4, 'numChains', 2): MCMCchain is every 4th row of each chain of the thin = 1 fit
    (rows and s2chain); MCMCresults are those of the thin = 1 fit except mean_sigma / sigma_sigma, which come from the
    device's all-row sig and so are exactly the saveChains = False fit's; the raw-chain file carries thin = 4 (and the
    thin = 1 file no such variable); MCMCdiagnostics has split-Rhat and ESS from the stored rows."""
    import scipy.io as sio
    from transcriptioncycleinference_b200 import mcmc
    need_gpu()
    idx = [0, 9, 100]
    d = tmp_path / "in"; d.mkdir()
    data = np.zeros((1, len(idx)), dtype=[("time", "O"), ("MS2", "O"), ("PP7", "O"), ("name", "O")])
    for j, c in enumerate(idx):
        o, n = int(cells_npz["off"][c]), int(cells_npz["N"][c])
        data[0, j] = (cells_npz["t"][o:o + n].reshape(1, -1), cells_npz["ms2"][o:o + n].reshape(1, -1),
                      cells_npz["pp7"][o:o + n].reshape(1, -1), "TestData")
    sio.savemat(str(d / "TestData.mat"), dict(data=data))
    n_burn, n_steps, k = 100, 600, 4

    def run(where, *extra):
        return mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(tmp_path / where), "numParPools", 1,
                                           "n_burn", n_burn, "n_steps", n_steps, "seed", 5, "numChains", 2,
                                           "returnResults", True, *extra)[0]
    full, thin, nochain = run("full"), run("thin", "thin", k), run("nochain", "saveChains", False)
    base = "%s-TestData_RawChain.mat" % mcmc.matlab_date()
    assert "thin" not in sio.loadmat(str(tmp_path / "full" / base))
    assert float(np.asarray(sio.loadmat(str(tmp_path / "thin" / base))["thin"]).squeeze()) == k
    for c in range(len(idx)):
        f, t = full["MCMCchain"][c], thin["MCMCchain"][c]
        for field in mcmc.CHAIN_FIELDS:
            rows = n_steps if field == "s2chain" else n_steps - n_burn + 1
            want = f[field].reshape(2, rows, -1)[:, ::k].reshape(-1, f[field].shape[1])
            assert np.array_equal(t[field], want), (c, field)
        for field in mcmc.RESULT_FIELDS:
            assert np.array_equal(thin["MCMCresults"][c][field], nochain["MCMCresults"][c][field]), (c, field)
            if field not in ("mean_sigma", "sigma_sigma"):
                assert np.array_equal(thin["MCMCresults"][c][field], full["MCMCresults"][c][field]), (c, field)
        assert abs(thin["MCMCresults"][c]["mean_sigma"] - full["MCMCresults"][c]["mean_sigma"]) <= 1e-12 * full["MCMCresults"][c]["mean_sigma"]
        dg = thin["MCMCdiagnostics"][c]
        assert dg["split_Rhat"].shape == dg["ESS"].shape == (1, 7 + int(cells_npz["N"][idx[c]]))
        assert np.all(dg["ESS"] <= 2 * ((n_steps - n_burn) // k + 1))
