"""GPU parity at the series lengths where the engine changes kernels or shared-memory layouts, and on loading-counter ties.

The engine picks its kernels from the dataset's max N: the batched Toeplitz SS runs in ss_stream_kernel (operands staged in
shared memory) up to N = 152 and in ss_batch_kernel (operands read from HBM/L2) from 153 on, for every cell of the dataset;
the CTA-per-chain sampler holds two CTAs per SM up to N = 141, one up to 213, and takes the big layout from 214; the
chain-per-warp sampler takes N <= 144.  TestData has 113-129 points, so the rest of that range is covered here, against the
C oracle (oracle/tc_oracle.c: the literal m x n restatement, sequential, bit-exact on the reference's golden vectors):

  * SS of both algorithms at N = 3 ... 441, each length its own dataset (so it selects its path), 1e-10 relative;
  * cross-path agreement of ss_stream_kernel, ss_batch_kernel and tc_ss_batch_device on the same (cell, theta), and
    independence of the leading dimension of theta;
  * forward curves on both grids, the config-5 generator, 3- and 8-set constructs;
  * the adversarial counter cases of test_counter_ties.py, whose floors need scan_counts' sequential redo;
  * DRAM replays flag for flag on every sampler layout at its edge lengths and on mixed-length datasets.

The ABI does not report which layout ran: at N = 213 a replay under TC_LAYOUT_CTA passes whether the regular layout or
(had it stopped fitting) the big one ran."""
import numpy as np
import pytest

from conftest import random_theta
from parity import DTS, check_chain, check_recorded_ss, cols, make_cells, need_gpu, oracle_chains, replay_streams, series
from test_counter_ties import COUNT_CONS, adversarial_cases, control_cases, count_theta, oracle_floors
from transcriptioncycleinference_b200 import _lib

pytestmark = pytest.mark.gpu
TOL = 1e-10
LENGTHS = list(range(3, 13)) + [31, 32, 33, 127, 128, 129, 130, 141, 142, 144, 145, 152, 153, 200, 211, 212, 213, 214,
                                255, 256, 257, 384, 400, 441]
STREAM_MAX_N = 152            # ss_stream_kernel: two CTAs of 8 warps per SM at max N <= 152 (launch_ss)


def model_cell(co, cons, rng, N):
    """A cell whose data are the oracle's own noise-free model at theta* (interpolated to t, with the NaN mask)."""
    t, m2, p7 = series(co, rng, N)
    thstar = random_theta(rng, N, False)
    tg = co.t_interp(t)
    a, b = co.model_on_grid(cons, thstar, tg)
    return (t, np.where(np.isnan(m2), np.nan, np.interp(t, tg, a)), np.where(np.isnan(p7), np.nan, np.interp(t, tg, b))), thstar


def theta_rows(rng, cells, n):
    """n rows over the cells: uniform in the wide bounds, uniform in the chain region, v -> 0 (long ramps), and t_on set to a
    t_interp value or one of its two neighbouring doubles."""
    tgs = [cells.t_interp(c) for c in range(cells.ncells)]
    cid = rng.integers(0, cells.ncells, n).astype(np.int32)
    th = np.zeros((n, cells.ld))
    for i, c in enumerate(cid):
        N = int(cells.N[c]); kind = i % 4
        th[i, :7 + N] = random_theta(rng, N, kind == 0)
        if kind == 2:
            th[i, 0] = 10.0 ** rng.uniform(-3.0, -0.3); th[i, 1] = rng.uniform(0.0, 20.0)
        if kind == 3:
            g = tgs[c][int(rng.integers(0, N))]
            th[i, 2] = (g, np.nextafter(g, -np.inf), np.nextafter(g, np.inf))[(i // 4) % 3]
    return cid, th


def _path(algo, nmax):
    return "pairs" if algo == 0 else ("toeplitz/stream" if nmax <= STREAM_MAX_N else "toeplitz/batch")


def _check_ss(tag, got, ref, nrows_cap=60000):
    """1e-10 relative; a polymerase within an ulp of L = L0 + tau v may flip (SURVEY 7.3 #4): at most 1 row per 60 000."""
    rel = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    flips = int((rel >= TOL).sum())
    print("%-28s rows %6d  max rel %.3g  median %.3g  beyond 1e-10: %d" % (tag, rel.size, rel.max(), np.median(rel), flips))
    assert flips <= max(1, rel.size // nrows_cap), (tag, flips, rel.max())
    assert np.median(rel) < 1e-13, tag
    return rel


@pytest.fixture(scope="module")
def length_sets(orc):
    """N -> (cells, packed, theta*): per length one dataset of 3 cells — irregular grid, regular grid, and the model cell."""
    need_gpu()
    co, cons = orc
    out = {}
    for N in LENGTHS:
        rng = np.random.default_rng(1000 + N)
        mc, thstar = model_cell(co, cons, rng, N)
        cells, packed = make_cells(co, [series(co, rng, N), series(co, rng, N, DTS[N % 4]), mc])
        out[N] = (cells, packed, thstar)
    yield out
    for cells, _, _ in out.values():
        cells.close()


@pytest.mark.parametrize("N", LENGTHS)
def test_ss_parity_per_length(length_sets, orc, N):
    """Each length as its own dataset, so that max N selects the path; both algorithms against the oracle.  At theta* the
    model cell's SS is rounding noise, so there the bound is absolute: |dSS| <= 1e-10 sum(y^2 + model^2)."""
    co, cons = orc
    cells, packed, thstar = length_sets[N]
    rng = np.random.default_rng(N)
    cid, th = theta_rows(rng, cells, 10000 if N < 200 else 2000)
    ref = co.ss_batch(cons, packed, cid, th)
    star = np.zeros((4, cells.ld)); star[:, :7 + N] = thstar
    sref = co.ss_batch(cons, packed, np.full(4, 2, np.int32), star)
    y = np.concatenate([cells.cell(2)[1], cells.cell(2)[2]])
    bound = 1e-10 * 2.0 * np.nansum(y * y)                    # y = model at theta* where not masked
    for algo in (1, 0):
        _check_ss("%s N=%d" % (_path(algo, N), N), cells.ss_batch(cid, th, algo=algo), ref)
        got = cells.ss_batch(np.full(4, 2, np.int32), star, algo=algo)
        assert np.all(np.abs(got - sref) <= bound), (algo, got, sref, bound)
        assert np.all(sref <= bound)


@pytest.mark.parametrize("N", LENGTHS)
def test_forward_curves_per_length(length_sets, orc, N):
    """tc_forward on the model grid (t_interp: what the likelihood and the config-5 generator use) and on the raw grid."""
    co, cons = orc
    cells, _, _ = length_sets[N]
    rng = np.random.default_rng(50 + N)
    cid, th = theta_rows(rng, cells, 12)
    for raw in (False, True):
        f1, f2 = cells.forward(cid, th, on_raw_grid=raw)
        for i, c in enumerate(cid):
            grid = cells.cell(c)[0] if raw else cells.t_interp(c)
            r1, r2 = co.model_on_grid(cons, th[i, :7 + N], grid)
            np.testing.assert_allclose(f1[i, :N], r1, rtol=1e-10, atol=1e-12, err_msg="raw=%s row %d" % (raw, i))
            np.testing.assert_allclose(f2[i, :N], r2, rtol=1e-10, atol=1e-12, err_msg="raw=%s row %d" % (raw, i))


def _short_plus(co, extra):
    rng = np.random.default_rng(7)
    short = [series(co, rng, N, DTS[N % 4] if N % 2 else None) for N in (3, 5, 8, 12, 33, 129)]
    return make_cells(co, short + [series(co, np.random.default_rng(extra), extra)])


def _device_ss(cells, cid, th, algo=1):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("torch has no CUDA")
    d_cid = torch.from_numpy(np.ascontiguousarray(cid, dtype=np.int32)).cuda()
    d_th = torch.from_numpy(np.ascontiguousarray(th)).cuda()
    d_out = torch.zeros(cid.size, dtype=torch.float64, device="cuda")
    cells.ss_batch_device(cid.size, d_cid.data_ptr(), d_th.data_ptr(), th.shape[1], d_out.data_ptr(), algo=algo)
    torch.cuda.synchronize()
    return d_out.cpu().numpy()


def test_stream_vs_batch_kernel_on_the_same_cells(orc):
    """The same short cells in a dataset with one cell of N = 152 (ss_stream_kernel) and one of N = 153 (ss_batch_kernel):
    both against the oracle; the Toeplitz SS of ss_stream_kernel, ss_batch_kernel and tc_ss_batch_device (torch device buffers)
    agree to 1e-14 (the same ss_eval on the same operands: a staging or permutation bug would be O(1)); theta with a padded
    leading dimension (7 + max N, +1, +8: ss_stream_kernel rounds it up and may stop fitting) gives identical results."""
    need_gpu()
    co, cons = orc
    (ca, pa), (cb, pb) = _short_plus(co, 152), _short_plus(co, 153)
    rng = np.random.default_rng(11)
    cid, th = theta_rows(rng, ca, 6000)
    thb = np.zeros((th.shape[0], cb.ld)); thb[:, :ca.ld] = th
    assert (cid == 6).any() and (cid < 6).any()             # the long cell / the short cells both datasets hold
    ra = co.ss_batch(cons, pa, cid, th); rb = co.ss_batch(cons, pb, cid, thb)
    res = {}
    for algo in (1, 0):
        res[("a", algo)] = ca.ss_batch(cid, th, algo=algo); res[("b", algo)] = cb.ss_batch(cid, thb, algo=algo)
        _check_ss("%s max N=152" % _path(algo, 152), res[("a", algo)], ra)
        _check_ss("%s max N=153" % _path(algo, 153), res[("b", algo)], rb)
    sh = cid < 6
    stream, batch = res[("a", 1)][sh], res[("b", 1)][sh]
    dev_a, dev_b = _device_ss(ca, cid, th), _device_ss(cb, cid, thb)
    for name, x in (("ss_batch_kernel", batch), ("tc_ss_batch_device (stream)", dev_a[sh]),
                    ("tc_ss_batch_device (batch)", dev_b[sh])):
        rel = np.abs(x - stream) / np.abs(stream)
        print("cross-path ss_stream_kernel vs %-28s rows %d  max rel %.3g  bit-identical %d" % (name, rel.size, rel.max(), int(np.sum(x == stream))))
        assert rel.max() <= 1e-14, (name, rel.max())
    for cells, t0, base in ((ca, th, res[("a", 1)]), (cb, thb, res[("b", 1)])):
        for pad in (1, 8):
            tp = np.zeros((t0.shape[0], t0.shape[1] + pad)); tp[:, :t0.shape[1]] = t0
            for algo in (1, 0):
                assert np.array_equal(cells.ss_batch(cid, tp, algo=algo), res[("a" if cells is ca else "b", algo)]), (cells.Nmax, pad, algo)
    ca.close(); cb.close()


def test_config5_generator_is_the_oracle_model(orc):
    """synthetic.make_cells(k, 400, noise=0): MS2 / PP7 = the oracle's model at the truth on t_interp, interpolated to t."""
    need_gpu()
    from transcriptioncycleinference_b200 import synthetic
    co, cons = orc
    cells, truth = synthetic.make_cells(4, 400, noise=0.0)
    for c in range(4):
        t, m2, p7 = cells.cell(c)
        tg = co.t_interp(t)
        assert np.array_equal(cells.t_interp(c), tg)
        a, b = co.model_on_grid(cons, truth[c], tg)
        for y, r in ((m2, np.interp(t, tg, a)), (p7, np.interp(t, tg, b))):
            ok = ~np.isnan(y)
            assert ok.sum() > 100
            np.testing.assert_allclose(y[ok], r[ok], rtol=1e-10, atol=1e-12)
    cells.close()


MULTI_SETS = {
    "lengths-3-sets": dict(L_MS2=6.626, L_PP7=6.9, MS2_start=[0.024, 2.0, 3.1], MS2_end=[1.299, 2.6, 3.5], MS2_loopn=[24.0, 12.0, 6.0],
                           PP7_start=[4.292, 5.8, 0.5], PP7_end=[5.758, 6.0, 0.9], PP7_loopn=[24.0, 6.0, 12.0]),
    "lengths-8-sets": dict(L_MS2=6.626, L_PP7=6.626,                  # TC_MAX_SETS, overlapping windows
                           MS2_start=[0.02, 0.5, 1.0, 1.2, 2.0, 2.1, 3.0, 4.0], MS2_end=[1.22, 1.3, 1.5, 2.7, 2.3, 3.0, 5.0, 5.0],
                           MS2_loopn=[24.0, 12.0, 6.0, 18.0, 3.0, 9.0, 24.0, 1.0],
                           PP7_start=[4.292, 4.0, 0.1, 5.0, 2.2, 2.5, 0.0, 6.0], PP7_end=[5.758, 6.0, 0.4, 5.5, 4.4, 2.6, 6.5, 6.2],
                           PP7_loopn=[24.0, 6.0, 12.0, 2.0, 20.0, 7.0, 1.0, 24.0]),
}


@pytest.mark.parametrize("name", sorted(MULTI_SETS))
@pytest.mark.parametrize("lengths", [(3, 7, 12, 129, 152), (130, 153, 213, 257)], ids=["stream", "batch"])
def test_multi_set_constructs(orc, name, lengths):
    """3- and 8-set constructs (the per-set basal clamp sits inside the loop over sets): SS of both algorithms and the curves
    on both grids against the oracle."""
    need_gpu()
    from transcriptioncycleinference_b200 import register_construct
    co, _ = orc
    d = MULTI_SETS[name]
    register_construct(name, d["L_MS2"], d["L_PP7"], d["MS2_start"], d["MS2_end"], d["MS2_loopn"], d["PP7_start"], d["PP7_end"], d["PP7_loopn"])
    cons = co.Construct.from_dict(d)
    rng = np.random.default_rng(len(name) + lengths[0])
    cells, packed = make_cells(co, [series(co, rng, N, DTS[N % 4] if N % 2 else None) for N in lengths], construct=name)
    cid, th = theta_rows(rng, cells, 1500)
    th[:, 3] = rng.uniform(0, 6, th.shape[0]); th[:, 4] = rng.uniform(0, 6, th.shape[0])     # basal levels that clamp
    ref = co.ss_batch(cons, packed, cid, th)
    for algo in (1, 0):
        _check_ss("%s %s %s" % (_path(algo, cells.Nmax), name, lengths), cells.ss_batch(cid, th, algo=algo), ref)
    for raw in (False, True):
        f1, f2 = cells.forward(cid[:30], th[:30], on_raw_grid=raw)
        for i, c in enumerate(cid[:30]):
            N = int(cells.N[c])
            r1, r2 = co.model_on_grid(cons, th[i, :7 + N], cells.cell(c)[0] if raw else cells.t_interp(c))
            np.testing.assert_allclose(f1[i, :N], r1, rtol=1e-10, atol=1e-12)
            np.testing.assert_allclose(f2[i, :N], r2, rtol=1e-10, atol=1e-12)
    cells.close()


def test_counter_ties_against_the_oracle(orc):
    """The adversarial cases of test_counter_ties.py (the fast path's floors differ from the sequential ones: the kernel must
    take its sequential redo) and the controls, one cell per case: SS of both algorithms on both SS kernels (all cases in one
    dataset, max N = 400: ss_batch_kernel; the N <= 129 cases alone: ss_stream_kernel) at 1e-10, the curves on t_interp at
    1e-10 / 1e-12 (a wrong floor moves a whole polymerase), and, under a construct whose curves are the loading counts, the
    counts themselves equal to the oracle's floors."""
    need_gpu()
    from transcriptioncycleinference_b200 import register_construct
    co, cons = orc
    cases = list(adversarial_cases()) + list(control_cases())
    rng = np.random.default_rng(3)
    cols = []
    for case in cases:
        N = case["N"]
        m2 = rng.uniform(0, 3, N); p7 = rng.uniform(0, 10, N)
        m2[rng.random(N) < 0.3] = np.nan
        cols.append((case["t"], m2, p7))
    short = [i for i, case in enumerate(cases) if case["N"] <= 129]
    for sel in (list(range(len(cases))), short):
        cells, packed = make_cells(co, [cols[i] for i in sel])
        for k, i in enumerate(sel):
            assert np.array_equal(cells.t_interp(k), cases[i]["tg"])
        th = cells.pad_theta([cases[i]["theta"] for i in sel])
        cid = np.arange(len(sel), dtype=np.int32)
        ref = co.ss_batch(cons, packed, cid, th)
        for algo in (1, 0):
            got = cells.ss_batch(cid, th, algo=algo)
            rel = np.abs(got - ref) / np.abs(ref)
            print("counter ties, %-16s %d cells: max rel %.3g" % (_path(algo, cells.Nmax), len(sel), rel.max()))
            assert rel.max() < TOL, (algo, cells.Nmax, [cases[sel[j]]["N"] for j in np.flatnonzero(rel >= TOL)])
        f1, f2 = cells.forward(cid, th, on_raw_grid=False)
        for k, i in enumerate(sel):
            N = cases[i]["N"]
            r1, r2 = co.model_on_grid(cons, cases[i]["theta"], cases[i]["tg"])
            np.testing.assert_allclose(f1[k, :N], r1, rtol=1e-10, atol=1e-12, err_msg="case %d" % i)
            np.testing.assert_allclose(f2[k, :N], r2, rtol=1e-10, atol=1e-12, err_msg="case %d" % i)
        cells.close()
    d = COUNT_CONS
    register_construct("loading-counts", d["L_MS2"], d["L_PP7"], d["MS2_start"], d["MS2_end"], d["MS2_loopn"], d["PP7_start"], d["PP7_end"], d["PP7_loopn"])
    cells, _ = make_cells(co, cols, construct="loading-counts")
    th = cells.pad_theta([count_theta(case["theta"]) for case in cases])
    f1, f2 = cells.forward(np.arange(len(cases), dtype=np.int32), th, on_raw_grid=False)
    for k, case in enumerate(cases):
        fc, _ = oracle_floors(co, case)
        N = case["N"]
        assert np.array_equal(f1[k, 1:N], fc) and np.array_equal(f2[k, 1:N], fc), (k, N, case["dt"], int(np.sum(f2[k, 1:N] != fc)))
    cells.close()


# ------------------------------------------------------------------------------------------------ sampler replays
NSIMU, BURN = 330, 100          # burn-in, the first covariance adaptation and two more
AUTO, BIG, WARP, CTA = _lib.LAYOUT_AUTO, _lib.LAYOUT_BIG, _lib.LAYOUT_WARP, _lib.LAYOUT_CTA
SMALL = tuple(range(3, 13))


def replay(orc, cols, layout, nch=None, ld_pad=0, seed=0):
    """Replay nch chains (chain i on cell i % ncells) with injected randomness and qcovadj_always = 1 against the oracle: flags,
    rows, s2chain, sschain and every counter; the SS the sampler recorded for every stored row must be tc_ss_batch's SS of
    that row (1e-14 relative)."""
    need_gpu()
    from transcriptioncycleinference_b200 import setup_cell
    co, _ = orc
    cells, packed = make_cells(co, cols)
    nch = nch or cells.ncells
    cc = (np.arange(nch) % cells.ncells).astype(np.int32)
    ins = setup_cell.chain_inputs(cells, cc, np.random.default_rng(seed))
    ld = cells.ld + ld_pad
    if ld_pad:
        fill = (0.0, 1.0, 0.0, 0.0, 0.0, np.inf)                  # chain_inputs' own padding
        ins = tuple(np.concatenate([x, np.full((nch, ld_pad), f)], axis=1) for x, f in zip(ins, fill))
    st = replay_streams(cells.N[cc], NSIMU, ld, seed + 1)
    opts = _lib.default_opts(nsimu=NSIMU, burnintime=BURN, n_burn=1, store_chain=1, replay=1, layout=layout, qcovadj_always=1)
    out = cells.mcmc_run(opts, cc, *ins, replay=st, want_flags=True)
    refs = oracle_chains(orc, packed, cc, co.default_opts(NSIMU, BURN, qcovadj_always=1), ins, st)
    for i, ref in enumerate(refs):
        check_chain("layout %d N=%d" % (layout, cells.N[cc[i]]), out, i, ref, 7 + int(cells.N[cc[i]]))
        cnt = out["counters"][i]
        assert cnt[_lib.CNT_ADAPTATIONS] == 3 and cnt[_lib.CNT_CHOL_FAIL] == 0
    check_recorded_ss(cells, cc, out, ld)
    cells.close()


REPLAYS = ([("cta", (N, N), CTA) for N in SMALL + (141, 142, 211, 212, 213)] +
           [("auto", (N, N), AUTO) for N in (213, 214)] +
           [("big", (N, N), BIG) for N in SMALL + (213,)] +
           [("warp", (N, N), WARP) for N in SMALL + (143, 144)] +
           [("mixed-cta", (3, 12, 61, 129, 144), CTA), ("mixed-big", (3, 12, 61, 129, 144), BIG),
            ("mixed-cta", (3, 12, 129, 213), CTA), ("mixed-auto", (3, 129, 214, 441), AUTO)])


@pytest.mark.parametrize("name,lengths,layout", REPLAYS, ids=["%s-%s" % (r[0], "-".join(map(str, sorted(set(r[1]))))) for r in REPLAYS])
def test_replay_at_layout_edges(orc, name, lengths, layout):
    """Each dataset holds these cells (a single length: two cells, one irregular and one regular grid); short chains in a
    mixed dataset run in a layout sized by the longest one."""
    replay(orc, cols(orc, lengths, sum(lengths) + layout), layout)


def test_replay_warp_mixed_lengths_ragged_groups(orc):
    """Chain-per-warp layout, 20 chains over cells of N = 3, 12, 61, 129, 144: the first 16-chain group mixes lengths, a ragged
    group of 4 follows."""
    replay(orc, cols(orc, (3, 12, 61, 129, 144), 5), WARP, nch=20)


def test_replay_padded_leading_dimension(orc):
    """ld = 7 + max N + 1 for every array of the run (theta0, bounds, priors, streams, chain)."""
    replay(orc, cols(orc, (5, 129, 141), 9), CTA, ld_pad=1)


@pytest.mark.parametrize("N", range(145, 151))
def test_warp_layout_limit(orc, N):
    """Past N = 144 (DESIGN 3: the chain-per-warp layout's promise) a length either runs and replays, or is refused with
    TC_EINVAL "too large for the chain-per-warp layout" — never a kernel that does not fit."""
    need_gpu()
    try:
        replay(orc, cols(orc, (N, N), N), WARP)
        print("chain-per-warp layout at N = %d: runs and replays" % N)
    except _lib.TcError as e:
        assert e.code == _lib.TC_EINVAL and "too large for the chain-per-warp layout" in str(e), str(e)
        print("chain-per-warp layout at N = %d: refused (TC_EINVAL)" % N)
