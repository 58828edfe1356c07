"""Multi-set constructs on the GPU vs the oracle (per-set basal clamp, SURVEY 0.1 #11) and t_start/t_end
windows (truncated cells have their own t_interp)."""
import numpy as np
import pytest

from conftest import random_theta
from parity import check_chain, make_cells, need_gpu, oracle_chains, replay_streams, series

pytestmark = pytest.mark.gpu


def test_two_set_construct_ss_and_forward(cells_npz, orc):
    from transcriptioncycleinference_b200 import register_construct
    from transcriptioncycleinference_b200.engine import Cells
    need_gpu()
    co, _ = orc
    d = dict(L_MS2=6.0, L_PP7=6.3, MS2_start=[0.024, 2.0], MS2_end=[1.299, 2.6], MS2_loopn=[24.0, 12.0],
             PP7_start=[4.292, 5.8], PP7_end=[5.758, 6.0], PP7_loopn=[24.0, 6.0])
    register_construct("gpu-two-sets", d["L_MS2"], d["L_PP7"], d["MS2_start"], d["MS2_end"], d["MS2_loopn"],
                       d["PP7_start"], d["PP7_end"], d["PP7_loopn"])
    cons2 = co.Construct.from_dict(d)
    sub = np.arange(0, 299, 10)
    N = cells_npz["N"][sub]; off = np.concatenate([[0], np.cumsum(N)]).astype(np.int64)
    t = np.concatenate([cells_npz["t"][cells_npz["off"][c]:cells_npz["off"][c + 1]] for c in sub])
    m2 = np.concatenate([cells_npz["ms2"][cells_npz["off"][c]:cells_npz["off"][c + 1]] for c in sub])
    p7 = np.concatenate([cells_npz["pp7"][cells_npz["off"][c]:cells_npz["off"][c + 1]] for c in sub])
    packed = dict(N=N.astype(np.int32), off=off, t=t, ms2=m2, pp7=p7)
    cells = Cells.from_packed(packed["N"], off, t, m2, p7, construct="gpu-two-sets")
    rng = np.random.default_rng(0)
    n = 4000
    cid = rng.integers(0, len(sub), n).astype(np.int32)
    th = np.zeros((n, cells.ld))
    for i, c in enumerate(cid):
        th[i, :7 + int(N[c])] = random_theta(rng, int(N[c]), i % 2 == 0)
        th[i, 3] = rng.uniform(0, 6); th[i, 4] = rng.uniform(0, 6)     # basal levels that actually clamp
    ref = co.ss_batch(cons2, packed, cid, th)
    for algo in (0, 1):
        got = cells.ss_batch(cid, th, algo=algo)
        rel = np.abs(got - ref) / np.abs(ref)
        assert (rel >= 1e-10).sum() <= 1, (algo, rel.max())
    f1, f2 = cells.forward(cid[:50], th[:50], on_raw_grid=True)
    for i in range(50):
        c = cid[i]; nn = int(N[c]); tt = t[off[c]:off[c] + nn]
        r1, r2 = co.model_on_grid(cons2, th[i, :7 + nn], tt)
        np.testing.assert_allclose(f1[i, :nn], r1, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(f2[i, :nn], r2, rtol=1e-10, atol=1e-12)
    cells.close()


def test_truncated_window_cells(cells_npz, orc):
    """t_start / t_end windows: shorter series, t(1) != 0, their own t_interp."""
    from transcriptioncycleinference_b200 import setup_cell
    from transcriptioncycleinference_b200.engine import Cells
    need_gpu()
    co, cons = orc
    ts, m2s, p7s = [], [], []
    for c in range(0, 299, 15):
        o, n = int(cells_npz["off"][c]), int(cells_npz["N"][c])
        a, b, d = setup_cell.truncate(cells_npz["t"][o:o + n], cells_npz["ms2"][o:o + n], cells_npz["pp7"][o:o + n], 3.0, 22.5)
        ts.append(a); m2s.append(b); p7s.append(d)
    cells = Cells(ts, m2s, p7s)
    packed = dict(N=cells.N, off=cells.off, t=cells.t, ms2=cells.ms2, pp7=cells.pp7)
    rng = np.random.default_rng(1)
    n = 3000
    cid = rng.integers(0, cells.ncells, n).astype(np.int32)
    th = np.zeros((n, cells.ld))
    for i, c in enumerate(cid):
        th[i, :7 + int(cells.N[c])] = random_theta(rng, int(cells.N[c]), False)
        th[i, 2] = rng.uniform(0, 8)                   # onset inside / before the window
    ref = co.ss_batch(cons, packed, cid, th)
    for algo in (0, 1):
        got = cells.ss_batch(cid, th, algo=algo)
        assert np.max(np.abs(got - ref) / np.abs(ref)) < 1e-10
    for c in range(cells.ncells):
        assert np.array_equal(cells.t_interp(c), co.t_interp(ts[c]))
    cells.close()


@pytest.mark.parametrize("N", [12, 200, 250, 400, 441])
def test_series_length_extremes_replay(orc, N):
    """Series much shorter / longer than TestData's 113-129 points: N = 12 (npar = 19: 3 column tiles, 5 Cholesky tile
    rows), N = 200 (npar = 207: one CTA per SM, 26 column tiles, several passes of the scatter update), and N = 250 /
    N = 400 (BASELINE config 5's length; npar = 257 / 407: the big layout — ring of 8 slots, bounds read from HBM/L2, proposal
    factor factorised through HBM/L2 by chol_global; 257 has an odd number of 4x4 tile rows), and N = 441, the longest series
    the engine takes (npar = 448: seven column tiles of 8 per warp in gen_increments_tma).  Synthetic irregular time
    grid with missing data; the DRAM replay must match the oracle: flags, rows, s2chain, sschain and every counter."""
    from transcriptioncycleinference_b200 import setup_cell
    _lib = need_gpu()
    co, _ = orc
    rng = np.random.default_rng(100 + N)
    cells, packed = make_cells(co, [series(co, rng, N) for _ in range(3)])
    cc = np.arange(3, dtype=np.int32)
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(7))
    nsimu, burn = 330, 100
    st = replay_streams(cells.N[cc], nsimu, cells.ld, 8)
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=1, store_chain=1, replay=1, qcovadj_always=1)   # singular covariances: see test_gpu_mcmc.py
    out = cells.mcmc_run(opts, cc, *inputs, replay=st, want_flags=True)
    refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, qcovadj_always=1), inputs, st)
    for i, ref in enumerate(refs):
        check_chain("N=%d" % N, out, i, ref, 7 + N)
    cells.close()


def test_series_longer_than_the_limit_are_rejected():
    """max(N) = 442 does not fit the one-CTA-per-chain layouts (include/tcmcmc.h): tc_mcmc_run returns TC_EINVAL, it does not
    run a kernel that would silently drop column tiles."""
    from transcriptioncycleinference_b200 import setup_cell
    from transcriptioncycleinference_b200.engine import Cells
    _lib = need_gpu()
    N = 442
    rng = np.random.default_rng(5)
    t = np.concatenate([[0.0], np.cumsum(rng.uniform(0.15, 0.35, N - 1))])
    cells = Cells([t], [rng.uniform(0, 3, N)], [rng.uniform(0, 10, N)])
    cc = np.zeros(1, dtype=np.int32)
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(7))
    with pytest.raises(Exception) as ei:
        cells.mcmc_run(_lib.default_opts(nsimu=200, burnintime=100, n_burn=100), cc, *inputs)
    assert "too large" in str(ei.value)
    cells.close()


def test_synthetic_config5_workload_big_layout():
    """BASELINE config 5 at a small scale: synthetic N = 400 cells from the forward model (synthetic.make_cells), production
    Philox run on the big layout.  Checks what does not depend on how well the reference's sampler mixes: every adaptation
    factorised (no Cholesky failure), the fit explains the data better than the start (posterior sigma below the initial
    one), chains independent of how they are batched (bit-identical), summaries inside the bounds."""
    from transcriptioncycleinference_b200 import setup_cell, synthetic
    _lib = need_gpu()
    cells, truth = synthetic.make_cells(12, 400)
    assert cells.Nmax == 400 and truth.shape == (12, 407)
    assert 0.35 < np.isnan(cells.ms2).mean() < 0.65 and 0.1 < np.isnan(cells.pp7).mean() < 0.3
    cc = np.arange(12, dtype=np.int32)
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(5))
    opts = _lib.default_opts(nsimu=1500, burnintime=500, n_burn=500)
    out = cells.mcmc_run(opts, cc, *inputs)
    cnt = out["counters"]
    assert np.all(cnt[:, 4] == 11) and np.all(cnt[:, 5] == 0)             # adaptations at 500, 600, .., 1500
    ss0 = cells.ss_batch(cc, inputs[0])
    n_obs = np.array([np.sum(~np.isnan(cells.cell(c)[1])) + np.sum(~np.isnan(cells.cell(c)[2])) for c in cc])
    assert np.all(out["sig"][:, 0] < np.sqrt(ss0 / n_obs))
    lo, hi = inputs[2], inputs[3]
    assert np.all(out["mean"] >= lo - 1e-12) and np.all(out["mean"] <= hi + 1e-12)
    sub = cells.mcmc_run(opts, cc[5:7], *[x[5:7] for x in inputs], chain_uid=np.array([5, 6], dtype=np.uint64))
    assert np.array_equal(sub["mean"], out["mean"][5:7]) and np.array_equal(sub["sig"], out["sig"][5:7])
    rec = synthetic.recovery(truth, out["mean"], out["std"])
    assert len(rec) == 3 and all(0.0 <= r <= 1.0 for r in rec)
    cells.close()
