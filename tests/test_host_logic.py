"""CPU tests of the host-side mirror: option parsing, per-cell set-up constants, construct registry,
.mat layouts, and the world_size-2 (gloo) sharding logic."""
import os
import sys

import numpy as np
import pytest

from transcriptioncycleinference_b200 import constructs, distributed, mcmc, setup_cell


def test_defaults_match_reference_code_not_readme():
    # src/TranscriptionCycleMCMC.m:36-45 (README says numParPools=0, n_steps=200000, t_end=0: SURVEY 0.1 #1)
    o = mcmc.parse_varargin(())
    assert (o["numParPools"], o["n_burn"], o["n_steps"], o["ratePriorWidth"]) == (8, 10000, 20000, 50.0)
    assert o["t_start"] == 0 and o["t_end"] == np.inf and o["loadPrevious"] is False
    assert o["construct"] == "P2P-MS2v5-LacZ-PP7v4"


def test_varargin_case_insensitive_and_presence_only_loadprevious():
    o = mcmc.parse_varargin(("N_STEPS", 500, "n_Burn", 100, "LOADPREVIOUS", False, "bogus", 3, "t_end", 25.0))
    assert o["n_steps"] == 500 and o["n_burn"] == 100 and o["t_end"] == 25.0
    assert o["loadPrevious"] is True          # the value after the name is ignored (:72-74)
    with pytest.raises(IndexError):
        mcmc.parse_varargin(("n_steps",))


def test_truncate_semantics():
    t = np.array([0.0, 1.0, 2.0, 3.0, 4.0]); y = np.arange(5.0)
    a, b, c = setup_cell.truncate(t, y, y, 1.0, 3.0)       # t >= 1 first, t < 3 last
    assert list(a) == [1.0, 2.0] and list(b) == [1.0, 2.0]
    a, _, _ = setup_cell.truncate(t, y, y, 0.0, np.inf)
    assert a.size == 5
    a, _, _ = setup_cell.truncate(t, y, y, 10.0, np.inf)
    assert a.size == 0


def test_setup_constants_appendix_a():
    t = np.array([0.0, 0.3, 0.5, 0.9])
    rng = np.random.default_rng(0)
    x0 = setup_cell.initial_state(4, rng)
    assert x0.size == 11 and 1 <= x0[0] <= 3 and 0 <= x0[1] <= 4 and 0 <= x0[2] <= 4
    assert x0[3] == 10 and x0[4] == 5 and 0 <= x0[5] <= 1 and x0[6] == 15
    J0 = setup_cell.proposal_variances(t)
    np.testing.assert_allclose(J0, [0.05, 0.1, 0.4, 1, 1, 0.05, 0.5, 0.5, 0.5, 0.5, 0.5])
    assert setup_cell.proposal_variances(t, True)[0] == 1e-7
    lo, hi, mu, sg = setup_cell.bounds_and_priors(4, x0, 50.0)
    np.testing.assert_array_equal(lo, [0, 0, 0, 0, 0, 0, 0, -30, -30, -30, -30])
    np.testing.assert_array_equal(hi, [10, 20, 10, 50, 50, 1, 40, 30, 30, 30, 30])
    assert np.all(np.isinf(sg[:7])) and np.all(sg[7:] == 50) and np.all(mu == 0)
    lo, hi, _, _ = setup_cell.bounds_and_priors(4, x0, 50.0, load_previous=True)
    assert abs(lo[0] - (x0[0] - 1e-5)) < 1e-15 and abs(hi[0] - (x0[0] + 1e-5)) < 1e-15


def test_construct_registry():
    c = constructs.get_construct("P2P-MS2v5-LacZ-PP7v4")
    assert c["L_MS2"] == 6.626 and c["MS2_start"] == [0.024] and c["PP7_end"] == [5.758] and c["MS2_loopn"] == [24.0]
    with pytest.raises(NameError):
        constructs.get_construct("no-such-construct")
    constructs.register_construct("two-sets", 5.0, 5.5, [0.1, 2.0], [1.0, 3.0], [24, 12], [3.2, 4.0], [3.9, 4.9], [24, 24])
    cc = constructs.to_c("two-sets")
    assert cc.nsets == 2 and cc.ms2_loopn[1] == 12.0 and cc.L_pp7 == 5.5
    with pytest.raises(ValueError):
        constructs.register_construct("bad", 5.0, 5.0, [0.1, 2.0], [1.0], [24, 24], [3.0, 4.0], [3.9, 4.9], [24, 24])


def test_matlab_date_and_struct_layout(tmp_path):
    import datetime
    import scipy.io as sio
    assert mcmc.matlab_date(datetime.date(2020, 10, 28)) == "28-Oct-2020"
    recs = [{f: np.float64(i) for f in mcmc.RESULT_FIELDS} for i in range(3)]
    for r in recs:
        r["mean_dR"] = np.zeros((1, 5)); r["sigma_dR"] = np.ones((1, 5))
    p = tmp_path / "x.mat"
    sio.savemat(p, dict(MCMCresults=mcmc._struct_array(mcmc.RESULT_FIELDS, recs), DatasetName="TestData"))
    m = sio.loadmat(p, mat_dtype=True)
    assert m["MCMCresults"].shape == (1, 3)
    assert m["MCMCresults"].dtype.names == mcmc.RESULT_FIELDS       # field ORDER of :151-155
    assert m["MCMCresults"][0, 1]["mean_dR"].shape == (1, 5)
    assert str(m["DatasetName"][0]) == "TestData"


def test_output_field_order_matches_reference_fixture(results_npz, chains_npz):
    assert tuple(results_npz["field_order"]) == mcmc.RESULT_FIELDS
    assert tuple(results_npz["plot_field_order"]) == mcmc.PLOT_FIELDS
    assert tuple(chains_npz["chain_field_order"]) == mcmc.CHAIN_FIELDS


def test_partition_contiguous_and_balanced(cells_npz):
    N = cells_npz["N"]
    cc = np.repeat(np.arange(299), 64)
    w = distributed.chain_work(N[cc])
    for parts in (1, 2, 4, 8):
        p = distributed.partition(w, parts)
        assert p[0][0] == 0 and p[-1][1] == cc.size
        assert all(p[i][1] == p[i + 1][0] for i in range(parts - 1))
        loads = np.array([w[s:e].sum() for s, e in p])
        assert loads.max() / loads.mean() < 1.02
    p = distributed.partition(np.ones(3), 8)                 # fewer units than parts
    assert sum(e - s for s, e in p) == 3 and all(e - s in (0, 1) for s, e in p)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    N_of_cell = np.array([5, 9, 7, 12, 6])
    cc = np.array([0, 0, 1, 2, 3, 3, 4], dtype=np.int32)
    uid = np.arange(100, 107, dtype=np.uint64)
    arrays = [np.arange(7 * 3, dtype=np.float64).reshape(7, 3)]

    def run_local(c, arrs, u):           # stand-in for Cells.mcmc_run: results depend only on the chain identity
        return dict(mean=arrs[0] * 2 + u[:, None].astype(np.float64), counters=np.stack([c, u.astype(np.int64)], 1),
                    owner=np.full(len(c), rank))
    out = distributed.fit_sharded(run_local, cc, N_of_cell, arrays, uid, rank, world)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_fit_world2_gloo():
    """world_size 2 over gloo: every rank ends with the full, correctly ordered result, identical to
    the single-rank result (the data path has no collective; only the final gather)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    N_of_cell = np.array([5, 9, 7, 12, 6]); cc = np.array([0, 0, 1, 2, 3, 3, 4], dtype=np.int32)
    uid = np.arange(100, 107, dtype=np.uint64); arr = np.arange(21, dtype=np.float64).reshape(7, 3)
    expect = arr * 2 + uid[:, None].astype(np.float64)
    for r in (0, 1):
        np.testing.assert_array_equal(res[r]["mean"], expect)
        np.testing.assert_array_equal(res[r]["counters"][:, 0], cc)
        assert set(res[r]["owner"]) == {0, 1}               # both ranks did work
        assert np.all(np.diff(res[r]["owner"]) >= 0)         # contiguous blocks


def test_rhat_from_summaries_matches_raw_chain_formula():
    """Gelman-Rubin Rhat / n_eff computed from per-chain (mean, population std, n) == the textbook formula on raw chains."""
    from transcriptioncycleinference_b200 import diagnostics
    rng = np.random.default_rng(3)
    m, n, p = 6, 400, 5
    chains = rng.standard_normal((m, n, p)) + rng.standard_normal((m, 1, p)) * np.array([0.0, 0.05, 0.3, 1.0, 3.0])
    rh, ne = diagnostics.rhat_from_summaries(chains.mean(axis=1), chains.std(axis=1), n)
    W = chains.var(axis=1, ddof=1).mean(axis=0); B = n * chains.mean(axis=1).var(axis=0, ddof=1)
    Vp = (n - 1) / n * W + B / n
    np.testing.assert_allclose(rh, np.sqrt(Vp / W), rtol=1e-12)
    assert rh[0] < 1.02 and rh[-1] > 2.0 and np.all(np.diff(rh) > 0)
    assert np.all(ne <= m * n) and ne[-1] < 20
    with pytest.raises(ValueError):
        diagnostics.rhat_from_summaries(chains.mean(axis=1)[:1], chains.std(axis=1)[:1], n)


def test_synthetic_recovery_fraction():
    """synthetic.recovery: fraction of cells whose truth lies within mean +- 3 sigma, per parameter (config 5's check)."""
    from transcriptioncycleinference_b200 import synthetic
    truth = np.zeros((4, 10)); mean = np.zeros((4, 10)); std = np.ones((4, 10))
    mean[0, 0] = 2.9; mean[1, 0] = 3.1; mean[2, 1] = -4.0
    assert synthetic.recovery(truth, mean, std) == [0.75, 0.75, 1.0]


def test_mex_gateway_compiles_against_stub_header(tmp_path):
    """matlab/tcmcmc_mex.cu (the MATLAB side of the boundary) is syntax-checked against tests/stubs/mex.h and the real
    include/tcmcmc.h: every ABI call and struct field it uses exists with the types it assumes.  (MATLAB itself is
    not in this image; the gateway is host-only C++ despite the .cu suffix mexcuda wants.)"""
    import shutil, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    src = tmp_path / "tcmcmc_mex.cpp"
    shutil.copy(os.path.join(root, "matlab", "tcmcmc_mex.cu"), src)
    res = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(root, "tests", "stubs"),
                          "-I", os.path.join(root, "include"), str(src)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr


def test_raw_chains_beyond_the_mat5_limit_are_split_into_matlab_readable_parts(tmp_path):
    """Plain `save` (MAT v5) cannot hold a variable of 2 GiB and the reference's own defaults on TestData give a 3.1 GB
    MCMCchain (SURVEY 0.1 #17): below the limit the writer produces the reference's single file, above it parts of whole
    cells + an index, all of them MAT v5 files that scipy (and MATLAB) read back — never a non-MATLAB format."""
    import scipy.io as sio
    from transcriptioncycleinference_b200 import mcmc
    rng = np.random.default_rng(0)
    chain = []
    for c in range(7):
        N = 5 + c
        rec = {f: rng.standard_normal((11, 1)) for f in mcmc.CHAIN_FIELDS}
        rec["dR_chain"] = rng.standard_normal((11, N)); rec["s2chain"] = rng.random((20, 1))
        chain.append(rec)
    one = mcmc.save_raw_chains(str(tmp_path), "a", chain)                       # fits: the reference's file
    assert [os.path.basename(f) for f in one] == ["a_RawChain.mat"]
    m = sio.loadmat(one[0])["MCMCchain"]
    assert m.shape == (1, 7) and m.dtype.names == mcmc.CHAIN_FIELDS
    size = [sum(v.nbytes for v in c.values()) for c in chain]
    files = mcmc.save_raw_chains(str(tmp_path), "b", chain, limit=size[0] + size[1] + size[2] + 8)   # forces a split
    assert os.path.basename(files[0]) == "b_RawChain.mat" and len(files) >= 3
    idx = sio.loadmat(files[0])
    assert int(idx["nParts"].squeeze()) == len(files) - 1
    names = [str(x[0]) if isinstance(x, np.ndarray) else str(x) for x in idx["MCMCchainParts"].reshape(-1)]
    back = [None] * 7
    for k, nm in enumerate(names, start=1):
        with open(os.path.join(tmp_path, nm.strip()), "rb") as fh:
            assert fh.read(19) == b"MATLAB 5.0 MAT-file"
        p = sio.loadmat(os.path.join(tmp_path, nm.strip()))
        a, b = int(p["firstCell"].squeeze()), int(p["lastCell"].squeeze())
        assert np.all(idx["MCMCchainPartOfCell"][0, a - 1:b] == k) and p["MCMCchain"].shape == (1, b - a + 1)
        for j in range(a, b + 1):
            back[j - 1] = p["MCMCchain"][0, j - a]
    for c in range(7):
        for f in mcmc.CHAIN_FIELDS:
            np.testing.assert_array_equal(back[c][f], chain[c][f])
    with pytest.raises(ValueError):
        mcmc.save_raw_chains(str(tmp_path), "c", chain, limit=size[0] - 8)       # one cell alone is too large


def test_split_rhat_and_ess_from_raw_chains():
    """split-Rhat and the autocorrelation-based ESS (diagnostics.split_rhat / ess): AR(1) chains with known
    integrated autocorrelation time (1 + phi) / (1 - phi); a drifting single chain is caught by split-Rhat although plain
    Rhat cannot see it."""
    from transcriptioncycleinference_b200 import diagnostics
    rng = np.random.default_rng(11)
    m, n = 4, 20000
    phis = np.array([0.0, 0.5, 0.9, 0.98])
    x = np.zeros((m, n, phis.size))
    e = rng.standard_normal((m, n, phis.size))
    for t in range(1, n):
        x[:, t] = phis * x[:, t - 1] + np.sqrt(1 - phis ** 2) * e[:, t]
    es = diagnostics.ess(x)
    expect = m * n * (1 - phis) / (1 + phis)
    assert np.all(np.abs(es / expect - 1) < 0.25), (es, expect)
    sr = diagnostics.split_rhat(x)
    assert np.all(sr < 1.05)
    _, ne = diagnostics.rhat_from_summaries(x.mean(axis=1), x.std(axis=1), n)
    assert np.all(np.isfinite(ne)) and np.all(ne <= m * n)      # the summaries-only estimate: right order of magnitude, m - 1 degrees of freedom
    assert np.all(ne / expect < 20) and np.all(ne / expect > 0.05)
    drift = x[:1, :, :1] + np.linspace(0, 3, n)[None, :, None]
    assert diagnostics.split_rhat(drift)[0] > 1.3 and diagnostics.ess(drift)[0] < 0.05 * n


def test_headless_curation_writes_approvedfits_back(tmp_path):
    """curate.ApproveMCMCResults: the reference's ApprovedFits convention (1 / 0 / -1, stored in MCMCresults of the same file,
    src/ApproveMCMCResults.m:11-15,335) without a display — explicit lists, automatic rules on the fields the current driver
    writes, 'LoadPrevious' matched on cell_index; every other variable of the file survives."""
    import scipy.io as sio
    from transcriptioncycleinference_b200 import curate, mcmc
    def rec(ci, sigma, app=0.0):
        r = {f: np.float64(1.0) for f in mcmc.RESULT_FIELDS}
        r.update(mean_dR=np.zeros((1, 5)), sigma_dR=np.ones((1, 5)), mean_sigma=np.float64(sigma), cell_index=np.float64(ci), ApprovedFits=np.float64(app))
        return r
    results = [rec(1, 0.9), rec(2, 5.0), rec(4, 1.1), rec(7, 1.0)]
    diags = [dict(cell_index=float(c), numChains=4.0, Rhat=np.ones((1, 12)), n_eff=np.ones((1, 12)), Rhat_max=rm,
                  split_Rhat=np.zeros((0, 0)), ESS=np.zeros((0, 0))) for c, rm in ((1, 1.02), (2, 1.01), (4, 1.8), (7, 1.05))]
    f = str(tmp_path / "18-Oct-2026-X.mat")
    sio.savemat(f, dict(MCMCresults=mcmc._struct_array(mcmc.RESULT_FIELDS, results), DatasetName="X",
                        MCMCplot=np.zeros((1, 4)), MCMCdiagnostics=mcmc._struct_array(mcmc.DIAG_FIELDS, diags)))
    app = curate.ApproveMCMCResults("file", f, "reject", [4], "maxRhat", 1.1, "maxSigma", 3.0)
    assert app.tolist() == [1.0, -1.0, -1.0, -1.0]          # ok | noise too large | chains disagree | rejected by hand
    m = sio.loadmat(f, mat_dtype=True)
    assert [float(m["MCMCresults"][0, k]["ApprovedFits"].squeeze()) for k in range(4)] == [1.0, -1.0, -1.0, -1.0]
    assert m["MCMCresults"].dtype.names == mcmc.RESULT_FIELDS and str(m["DatasetName"][0]) == "X" and "MCMCdiagnostics" in m
    # a later fit of a subset: carry the curation over by cell_index
    f2 = str(tmp_path / "19-Oct-2026-X.mat")
    sio.savemat(f2, dict(MCMCresults=mcmc._struct_array(mcmc.RESULT_FIELDS, [rec(7, 1.0), rec(1, 1.0), rec(9, 1.0)]), DatasetName="X"))
    assert curate.ApproveMCMCResults("file", f2, "LoadPrevious", f, "approve", [3]).tolist() == [-1.0, 1.0, 1.0]


@pytest.mark.parametrize("width", [0.5, 2.0, 50.0])
def test_rate_prior_width_reaches_the_sampler(tmp_path, monkeypatch, width):
    """TranscriptionCycleMCMC(..., 'ratePriorWidth', w) hands the sampler prior_sig = w on every dR and Inf on the seven head
    parameters, prior_mu = 0 (TranscriptionCycleMCMC.m:242-255), for cells of different lengths in one padded call."""
    import scipy.io as sio
    from transcriptioncycleinference_b200 import engine
    seen = {}

    class FakeCells(engine.Cells):
        def __init__(self, t, ms2, pp7, construct=None, devices=(0,)):
            self.ncells = len(t); self.N = np.array([len(x) for x in t], dtype=np.int32)
            self.off = np.concatenate([[0], np.cumsum(self.N)]); self.t = np.concatenate(t)
            self.ms2 = np.concatenate(ms2); self.pp7 = np.concatenate(pp7)
            self.Nmax = int(self.N.max()); self.ld = 7 + self.Nmax

        def close(self):
            pass

        def mcmc_run(self, opts, chain_cell, theta0, qcov_diag, low, upp, prior_mu, prior_sig, chain_uid=None, **kw):
            seen.update(cc=np.array(chain_cell), mu=np.array(prior_mu), sig=np.array(prior_sig), N=self.N.copy())
            n = len(chain_cell)
            return dict(mean=np.array(theta0), std=np.ones((n, self.ld)), sig=np.ones((n, 2)))

        def forward(self, cell_id, theta, on_raw_grid=True):
            return np.zeros((len(cell_id), self.Nmax)), np.zeros((len(cell_id), self.Nmax))

    monkeypatch.setattr(mcmc, "Cells", FakeCells)
    monkeypatch.setattr(mcmc._lib, "device_count", lambda: 1)
    rng = np.random.default_rng(0)
    recs = []
    for n in (5, 9):
        t = np.arange(n) * 0.5
        recs.append(dict(time=t, MS2=rng.random(n), PP7=rng.random(n), name="X"))
    data = np.empty((1, 2), dtype=[("time", object), ("MS2", object), ("PP7", object), ("name", object)])
    for k, r in enumerate(recs):
        data[0, k] = (r["time"], r["MS2"], r["PP7"], r["name"])
    sio.savemat(str(tmp_path / "d.mat"), dict(data=data))
    mcmc.TranscriptionCycleMCMC("fileDir", str(tmp_path), "saveLoc", str(tmp_path / "out"), "ratePriorWidth", width,
                                "n_steps", 10, "n_burn", 5, "saveChains", False, "seed", 1, "numChains", 2)
    assert seen["N"].tolist() == [5, 9] and seen["cc"].tolist() == [0, 0, 1, 1]
    for i, c in enumerate(seen["cc"]):
        npar = 7 + int(seen["N"][c])
        assert np.all(np.isinf(seen["sig"][i, :7])) and np.all(seen["sig"][i, 7:npar] == width), seen["sig"][i]
        assert np.all(seen["mu"][i, :npar] == 0)
