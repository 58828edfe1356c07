"""The 'thin' option on the host, without a GPU: its default, its parsing and validation in the driver, the row counts it
implies, and the raw-chain files it writes."""
import os

import numpy as np
import pytest
import scipy.io as sio

from transcriptioncycleinference_b200 import _lib, mcmc


def test_default_thin_is_one():
    o = _lib.default_opts()
    assert o.thin == 1
    assert _lib.stored_rows(o) == (o.nsimu - o.n_burn + 1, o.nsimu)


@pytest.mark.parametrize("nsimu,n_burn,thin,want", [
    (2000, 1, 1, (2000, 2000)), (2000, 613, 7, (199, 286)), (2000, 613, 1387, (2, 2)), (2000, 613, 1388, (1, 2)),
    (2000, 2000, 3, (1, 667)), (2 ** 31 - 1, 1, 2 ** 31 - 1, (1, 1)), (2 ** 31 - 1, 2, 2 ** 31 - 1, (1, 1))])
def test_stored_row_counts(nsimu, n_burn, thin, want):
    """nkeep = floor((nsimu - n_burn) / thin) + 1 chain rows, ns2 = ceil(nsimu / thin) s2chain rows: the lengths of
    range(n_burn - 1, nsimu, thin) and range(0, nsimu, thin)."""
    o = _lib.default_opts(nsimu=nsimu, n_burn=n_burn, thin=thin)
    assert _lib.stored_rows(o) == want == (len(range(n_burn - 1, nsimu, thin)), len(range(0, nsimu, thin)))


def test_varargin_thin_case_insensitive():
    assert mcmc.parse_varargin(())["thin"] == 1
    assert mcmc.parse_varargin(("THIN", 4))["thin"] == 4
    assert mcmc.parse_varargin(("n_steps", 10, "Thin", 20.0))["thin"] == 20.0


@pytest.mark.parametrize("bad", [0, -2, 2.5, float("nan"), "x", True])
def test_driver_rejects_bad_thin_before_any_work(tmp_path, monkeypatch, bad):
    def no_device():
        raise AssertionError("a device was queried")
    monkeypatch.setattr(mcmc._lib, "device_count", no_device)
    with pytest.raises(ValueError, match="thin"):
        mcmc.TranscriptionCycleMCMC("fileDir", str(tmp_path), "saveLoc", str(tmp_path), "thin", bad)


@pytest.mark.parametrize("good,want", [(1, 1), (3, 3), (4.0, 4), (np.int64(7), 7)])
def test_positive_int_accepts_whole_numbers(good, want):
    assert mcmc.positive_int(good, "thin") == want


def _chains(rng, n):
    out = []
    for c in range(n):
        rec = {f: rng.standard_normal((11, 1)) for f in mcmc.CHAIN_FIELDS}
        rec["dR_chain"] = rng.standard_normal((11, 5 + c)); rec["s2chain"] = rng.random((20, 1))
        out.append(rec)
    return out


def test_raw_chain_files_carry_thin_only_above_one(tmp_path):
    """One file: `thin` next to MCMCchain when thin > 1, the reference's variables alone at thin = 1.  Parts: `thin` in the
    index and next to MCMCchain in every part."""
    chain = _chains(np.random.default_rng(0), 5)
    one = sio.loadmat(mcmc.save_raw_chains(str(tmp_path), "a", chain)[0])
    assert [k for k in one if not k.startswith("__")] == ["MCMCchain"]
    assert [k for k in sio.loadmat(mcmc.save_raw_chains(str(tmp_path), "b", chain, thin=1)[0]) if not k.startswith("__")] == ["MCMCchain"]
    th = sio.loadmat(mcmc.save_raw_chains(str(tmp_path), "c", chain, thin=20)[0])
    assert float(th["thin"].squeeze()) == 20 and th["MCMCchain"].shape == (1, 5)
    size = sum(v.nbytes for v in chain[0].values())
    files = mcmc.save_raw_chains(str(tmp_path), "d", chain, limit=2 * size + 8, thin=20)
    assert len(files) >= 3
    for f in files:
        assert float(sio.loadmat(f)["thin"].squeeze()) == 20, os.path.basename(f)
    files = mcmc.save_raw_chains(str(tmp_path), "e", chain, limit=2 * size + 8)
    assert all("thin" not in sio.loadmat(f) for f in files)


def test_driver_passes_thin_and_takes_sigma_from_the_device(tmp_path, monkeypatch):
    """With thin > 1 the driver asks the engine for thinned rows, shapes MCMCchain from them, writes `thin` to the raw-chain
    file and takes mean_sigma / sigma_sigma from the device's all-row sig, not from the thinned s2chain."""
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

        def mcmc_run(self, opts, chain_cell, theta0, *a, chain_uid=None, **kw):
            seen["thin"] = opts.thin
            n = len(chain_cell)
            nkeep, ns2 = _lib.stored_rows(opts)
            return dict(mean=np.array(theta0), std=np.ones((n, self.ld)), sig=np.full((n, 2), 0.5),
                        chain=np.zeros((n, nkeep, self.ld)), s2chain=np.full((n, ns2), 9.0))

        def forward(self, cell_id, theta, on_raw_grid=True):
            return np.zeros((len(cell_id), self.Nmax)), np.zeros((len(cell_id), self.Nmax))

    monkeypatch.setattr(mcmc, "Cells", FakeCells)
    monkeypatch.setattr(mcmc._lib, "device_count", lambda: 1)
    data = np.empty((1, 1), dtype=[("time", object), ("MS2", object), ("PP7", object), ("name", object)])
    data[0, 0] = (np.arange(6) * 0.5, np.ones(6), np.ones(6), "X")
    sio.savemat(str(tmp_path / "d.mat"), dict(data=data))
    out = mcmc.TranscriptionCycleMCMC("fileDir", str(tmp_path), "saveLoc", str(tmp_path / "out"), "n_steps", 100, "n_burn",
                                      31, "thin", 7, "seed", 1, "returnResults", True)[0]
    assert seen["thin"] == 7
    assert out["MCMCchain"][0]["v_chain"].shape == (10, 1) and out["MCMCchain"][0]["s2chain"].shape == (15, 1)
    assert out["MCMCresults"][0]["mean_sigma"] == 0.5 and out["MCMCresults"][0]["sigma_sigma"] == 0.5
    raw = sio.loadmat(str(tmp_path / "out" / ("%s-X_RawChain.mat" % mcmc.matlab_date())))
    assert float(raw["thin"].squeeze()) == 7
