"""End-to-end drop-in test: TranscriptionCycleMCMC(varargin) -> the reference's .mat layouts
(SURVEY Appendix C), plus the working loadPrevious mode and a custom construct (BASELINE config 4)."""
import glob
import os

import numpy as np
import pytest
import scipy.io as sio

from parity import need_gpu

pytestmark = pytest.mark.gpu


def _f(x):
    return float(np.asarray(x).squeeze())


def _write_dataset(path, cells_npz, idx, name="TestData"):
    data = np.zeros((1, len(idx)), dtype=[("time", "O"), ("MS2", "O"), ("PP7", "O"), ("name", "O")])
    for k, c in enumerate(idx):
        o, n = int(cells_npz["off"][c]), int(cells_npz["N"][c])
        data[0, k]["time"] = cells_npz["t"][o:o + n].reshape(1, -1)
        data[0, k]["MS2"] = cells_npz["ms2"][o:o + n].reshape(1, -1)
        data[0, k]["PP7"] = cells_npz["pp7"][o:o + n].reshape(1, -1)
        data[0, k]["name"] = name
    sio.savemat(path, dict(data=data))


def test_driver_outputs_reference_layout(tmp_path, cells_npz, orc):
    from transcriptioncycleinference_b200 import mcmc
    need_gpu()
    co, cons = orc
    idx = [0, 9, 100, 250, 298]
    d = tmp_path / "in"; s = tmp_path / "out"; d.mkdir()
    _write_dataset(str(d / "TestData.mat"), cells_npz, idx)
    mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(s), "numParPools", 1, "n_burn", 100, "N_STEPS", 300,
                                "seed", 3)
    base = "%s-TestData" % mcmc.matlab_date()
    res = sio.loadmat(str(s / (base + ".mat")), mat_dtype=True)
    raw = sio.loadmat(str(s / (base + "_RawChain.mat")), mat_dtype=True)
    assert res["MCMCresults"].shape == (1, 5) and res["MCMCresults"].dtype.names == mcmc.RESULT_FIELDS
    assert res["MCMCplot"].dtype.names == mcmc.PLOT_FIELDS and raw["MCMCchain"].dtype.names == mcmc.CHAIN_FIELDS
    assert str(res["DatasetName"][0]) == "TestData"
    for k, c in enumerate(idx):
        n = int(cells_npz["N"][c]); o = int(cells_npz["off"][c])
        ch, r, p = raw["MCMCchain"][0, k], res["MCMCresults"][0, k], res["MCMCplot"][0, k]
        assert ch["v_chain"].shape == (201, 1) and ch["dR_chain"].shape == (201, n) and ch["s2chain"].shape == (300, 1)
        assert r["mean_dR"].shape == (1, n) and r["sigma_dR"].shape == (1, n) and r["mean_v"].shape == (1, 1)
        assert _f(r["cell_index"]) == k + 1 and _f(r["ApprovedFits"]) == 0
        assert abs(_f(r["mean_v"]) - ch["v_chain"].mean()) < 1e-12
        assert abs(_f(r["sigma_tau"]) - ch["tau_chain"].std()) < 1e-9
        np.testing.assert_allclose(r["mean_dR"][0], ch["dR_chain"].mean(axis=0), atol=1e-12)
        assert abs(_f(r["mean_sigma"]) - np.sqrt(ch["s2chain"].mean())) < 1e-12
        assert abs(_f(r["sigma_sigma"]) - np.sqrt(ch["s2chain"]).std()) < 1e-10
        np.testing.assert_array_equal(p["t_plot"][0], cells_npz["t"][o:o + n])
        # best-fit curves = oracle forward model at the posterior means on the raw grid (:307-309)
        th = np.concatenate([[_f(r["mean_v"]), _f(r["mean_tau"]), _f(r["mean_ton"]), _f(r["mean_MS2_basal"]),
                              _f(r["mean_PP7_basal"]), _f(r["mean_A"]), _f(r["mean_R"])], r["mean_dR"][0]])
        m1, m2 = co.model_on_grid(cons, th, cells_npz["t"][o:o + n])
        np.testing.assert_allclose(p["simMS2"][0], m1, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(p["simPP7"][0], m2, rtol=1e-10, atol=1e-12)


def test_load_previous_and_custom_construct(tmp_path, cells_npz):
    from transcriptioncycleinference_b200 import mcmc, register_construct
    need_gpu()
    idx = [3, 4, 5, 6]
    d = tmp_path / "in"; s1 = tmp_path / "o1"; s2 = tmp_path / "o2"; d.mkdir()
    _write_dataset(str(d / "TestData.mat"), cells_npz, idx)
    first = mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(s1), "numParPools", 1, "n_burn", 50, "n_steps", 150,
                                        "seed", 1, "returnResults", True)[0]
    # drop cell 2 from the previous results and mark cell 3 as approved
    prev_path = glob.glob(str(s1 / "*-TestData.mat"))[0]
    m = sio.loadmat(prev_path, mat_dtype=True)
    keep = m["MCMCresults"][:, [0, 2, 3]].copy()
    keep[0, 1]["ApprovedFits"] = np.array([[1.0]])
    sio.savemat(prev_path, dict(MCMCresults=keep, MCMCplot=m["MCMCplot"][:, [0, 2, 3]], DatasetName="TestData"))
    register_construct("test-two-sets", 6.0, 6.3, [0.024, 2.0], [1.299, 2.6], [24, 12], [4.292, 5.8], [5.758, 6.0], [24, 6])
    out = mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(s2), "numParPools", 1, "n_burn", 50, "n_steps", 150,
                                      "loadPrevious", "previousResults", prev_path, "construct", "test-two-sets",
                                      "seed", 2, "returnResults", True)[0]
    assert [int(_f(r["cell_index"])) for r in out["MCMCresults"]] == [1, 3, 4]      # unmatched cell removed
    assert [int(_f(r["ApprovedFits"])) for r in out["MCMCresults"]] == [0, 1, 0]
    for r, ch in zip(out["MCMCresults"], out["MCMCchain"]):
        v0 = _f(first["MCMCresults"][int(_f(r["cell_index"])) - 1]["mean_v"])
        assert np.all(np.abs(ch["v_chain"] - v0) <= 1e-5 + 1e-15)                 # v in [v0 - 1e-5, v0 + 1e-5]
    with pytest.raises(NameError):
        mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(s2), "construct", "undefined-construct")


def test_multiple_chains_per_cell_pool_and_diagnose(tmp_path, cells_npz):
    """'numChains' > 1 (BASELINE config 3 through the drop-in driver): the chains of a cell are pooled into the
    reference's MCMCresults layout (pooled mean / population std = those of the concatenated chains) and the extra
    variable MCMCdiagnostics carries Rhat / n_eff per parameter."""
    from transcriptioncycleinference_b200 import mcmc
    need_gpu()
    idx = [3, 77, 200]
    d = tmp_path / "in"; s = tmp_path / "out"; d.mkdir()
    _write_dataset(str(d / "TestData.mat"), cells_npz, idx)
    mcmc.TranscriptionCycleMCMC("fileDir", str(d), "saveLoc", str(s), "numParPools", 1, "n_burn", 200, "n_steps", 600,
                                "numChains", 4, "seed", 5)
    base = "%s-TestData" % mcmc.matlab_date()
    res = sio.loadmat(str(s / (base + ".mat")), mat_dtype=True)
    raw = sio.loadmat(str(s / (base + "_RawChain.mat")), mat_dtype=True)
    assert res["MCMCresults"].shape == (1, 3) and res["MCMCresults"].dtype.names == mcmc.RESULT_FIELDS
    assert res["MCMCdiagnostics"].dtype.names == mcmc.DIAG_FIELDS and res["MCMCdiagnostics"].shape == (1, 3)
    for k, c in enumerate(idx):
        n = int(cells_npz["N"][c])
        ch, r, dg = raw["MCMCchain"][0, k], res["MCMCresults"][0, k], res["MCMCdiagnostics"][0, k]
        assert ch["v_chain"].shape == (4 * 401, 1) and ch["s2chain"].shape == (4 * 600, 1)
        assert abs(_f(r["mean_v"]) - ch["v_chain"].mean()) < 1e-10 and abs(_f(r["sigma_v"]) - ch["v_chain"].std()) < 1e-8
        np.testing.assert_allclose(r["sigma_dR"][0], ch["dR_chain"].std(axis=0), rtol=1e-7, atol=1e-9)
        assert dg["Rhat"].shape == (1, 7 + n) and _f(dg["numChains"]) == 4 and _f(dg["cell_index"]) == k + 1
        # recompute Rhat of v from the raw chains
        v = ch["v_chain"].reshape(4, 401)
        W = v.var(axis=1, ddof=1).mean(); B = 401 * v.mean(axis=1).var(ddof=1)
        assert abs(dg["Rhat"][0, 0] - np.sqrt((400 / 401 * W + B / 401) / W)) < 1e-8
        assert _f(dg["Rhat_max"]) >= 1.0 - 1e-12


def test_two_gpus_same_result_as_one(cells_npz):
    """numParPools = 2 -> two GPUs inside one process (tc_mcmc_opts.ngpus = 2: chains partitioned by cumulative N^2, one
    stream and one drain thread per device): bit-identical to the one-GPU fit, raw chains included (Philox is keyed by chain
    identity, never by device).  That holds for a given sampler: 43 chains run dram_kernel on one GPU and on two.  Under
    TC_LAYOUT_AUTO the sampler is chosen per device, so for 13 S <= nchains < 13 S * ngpus (S SMs per device) one GPU runs
    dram_warp_kernel and two run dram_kernel, and the fits agree to rounding only (test_gpu_chain_counts.py,
    DESIGN.md 5).  Skipped on a box with fewer than two devices."""
    from transcriptioncycleinference_b200 import _lib, setup_cell
    from transcriptioncycleinference_b200.engine import Cells
    if _lib.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    g = cells_npz
    cc = np.arange(0, 299, 7, dtype=np.int32)
    res = []
    for devs in ((0,), (0, 1)):
        cells = Cells.from_packed(g["N"], g["off"], g["t"], g["ms2"], g["pp7"], devices=devs)
        inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(3))
        opts = _lib.default_opts(nsimu=1200, burnintime=400, n_burn=400, store_chain=1, ngpus=len(devs), seed=11)
        res.append(cells.mcmc_run(opts, cc, *inputs, chain_uid=cc.astype(np.uint64)))
        cells.close()
    for k in ("mean", "std", "sig", "chain", "s2chain"):
        assert np.array_equal(res[0][k], res[1][k]), k
    assert np.array_equal(res[0]["counters"][:, :8], res[1]["counters"][:, :8])
