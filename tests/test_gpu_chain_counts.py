"""GPU parity along the chain-count axis: the chain counts per launch, and the GPU counts, at which tc_mcmc_run's schedulers
change shape, against the C oracle (oracle/tc_oracle.c) on the device's own Philox streams.

tc_mcmc_run schedules a launch by its per-device chain count nc (S = the device's SM count, 148 on a B200):
  * dram_kernel, regular layout (two CTAs per SM at N <= 129): one chain per CTA while nc <= S; above S the solo-SM rule
    (smctl: a lagging chain gets its SM to itself) with slices of nsimu/128; above 2S chains queue for the 2S persistent
    CTAs; from 4 * 296 = 1184 chains on (a literal of the host code) nothing is sliced and a CTA takes any free chain;
  * the big layout: one CTA per SM, the same thresholds at S and 1184;
  * dram_warp_kernel (16 chains per CTA, one CTA per SM): with more 16-chain groups than CTAs, groups are parked and resumed
    by other CTAs, in other per-warp L2 slots;
  * TC_LAYOUT_AUTO: dram_warp_kernel from 13 S chains per device on, dram_kernel below;
  * ngpus > 1: contiguous blocks of equal sum N^2, one per device, each scheduled by the rules above on its own count.

Sections 1 and 3 run nsimu = 1000, burn-in and n_burn 300, adaptint = 100 (slices of 100 steps: every chain is parked and
resumed about 10 times where the launch is sliced) with qcovadj_always = 1 (300-row covariances are singular: see
test_gpu_mcmc.py).  Chain i goes to TestData cell i mod 299, has chain_uid i * 2^20 + 3 (never its index) and the same inputs
in every launch, so the oracle's chain of i serves every launch that holds it.  Section 2 runs the two benchmarked
many-chain workloads as bench.py builds them."""
import numpy as np
import pytest

from parity import check_chain, check_summaries, cols, dumped_streams, ld_mean_std, make_cells, need_gpu, oracle_chains
from transcriptioncycleinference_b200 import _lib

pytestmark = pytest.mark.gpu

NSIMU, BURN, ADAPTINT, SEED = 1000, 300, 100, 20261022
UNSLICED = 4 * 296                     # tc_mcmc_run: dram_kernel stops slicing from this many chains on
GROUP = 16                             # chains per dram_warp_kernel CTA
CONFIG3 = 299 * 64
OUT_KEYS = ("flags", "sschain", "mean", "std", "sig")


def _opts(layout, **kw):
    kw = dict(dict(nsimu=NSIMU, burnintime=BURN, adaptint=ADAPTINT, n_burn=BURN, seed=SEED, qcovadj_always=1), **kw)
    return _lib.default_opts(layout=layout, **kw)


def sampler_of(counters):
    """Which sampler ran each chain, from its phase counters: dram_kernel never writes CYCLES0 + 3, + 4, + 6;
    dram_warp_kernel times the randomness in + 3 and counts its evaluations, all committed, in + 7."""
    c = counters
    cta = np.all(c[:, [_lib.CNT_CYCLES0 + 3, _lib.CNT_CYCLES0 + 4, _lib.CNT_CYCLES0 + 6]] == 0, axis=1)
    warp = (c[:, _lib.CNT_CYCLES0 + 3] > 0) & (c[:, _lib.CNT_CYCLES0 + 7] == c[:, _lib.CNT_SS_EVALS])
    assert not np.any(cta & warp) and np.all(cta | warp), "a chain's counters fit neither sampler"
    return np.where(warp, "warp", "cta")


def assert_same_chains(tag, a, b, keys=OUT_KEYS + ("chain", "s2chain")):
    """Every output of every chain bit-identical (counters: the seven results and the status, not the clocks); a failure
    names the first few chains that differ and, for the flags, the first step where they do."""
    for k in keys + ("counters",):
        x, y = a.get(k), b.get(k)
        if x is None and y is None:
            continue
        if k == "counters":
            x, y = x[:, :8], y[:, :8]
        bad = np.flatnonzero(np.any(x.reshape(x.shape[0], -1) != y.reshape(y.shape[0], -1), axis=1))
        step = [int(np.argmax(x[i] != y[i])) for i in bad[:4]] if k == "flags" else None
        assert bad.size == 0, (tag, k, "%d chains differ" % bad.size, bad[:8].tolist(), step)


def _take(out, idx):
    """The per-chain outputs of the chains idx of a launch."""
    return {k: v[idx] for k, v in out.items() if isinstance(v, np.ndarray)}


def assert_one_sampler(tag, out, want):
    got = sampler_of(out["counters"])
    assert np.all(got == want), (tag, want, np.unique(got, return_counts=True))


def _sample(nc, S, warp, seed, n=20):
    """First and last chain; both sides of the first chain (16-chain group) without a CTA of its own at the start, and of the
    last group; the ragged last group; random chains up to n."""
    if warp:
        last = GROUP * ((nc - 1) // GROUP)
        edges = [GROUP * S - 1, GROUP * S, last - 1, last] + (list(range(last, nc)) if nc % GROUP else [])
    else:
        edges = [S - 1, S, 2 * S - 1, 2 * S]
    pick = {i for i in [0, nc - 1] + edges if 0 <= i < nc}
    rng = np.random.default_rng(seed)
    while len(pick) < min(n, nc):
        pick.add(int(rng.integers(nc)))
    return np.array(sorted(pick))


class Workload:
    """nmax chains round-robin over the cells of a dataset with fixed inputs and uids; runs any subset of them in any order,
    and keeps the oracle's chain of every chain it has computed."""

    def __init__(self, orc, cells, packed, nmax, seed):
        from transcriptioncycleinference_b200 import setup_cell
        self.orc, self.cells, self.packed = orc, cells, packed
        self.cc = (np.arange(nmax) % cells.ncells).astype(np.int32)
        self.uid = np.arange(nmax, dtype=np.uint64) * np.uint64(1 << 20) + np.uint64(3)
        self.ins = setup_cell.chain_inputs(cells, self.cc, np.random.default_rng(seed))
        self._refs = {}

    def npar(self, i):
        return 7 + int(self.cells.N[self.cc[i]])

    def run(self, idx, layout, cells=None, **kw):
        idx = np.asarray(idx)
        return (cells or self.cells).mcmc_run(_opts(layout, **kw), self.cc[idx], *[x[idx] for x in self.ins],
                                              chain_uid=self.uid[idx], want_flags=True)

    def refs(self, idx):
        new = np.array(sorted({int(i) for i in idx} - set(self._refs)), dtype=np.int64)
        if new.size:
            co, _ = self.orc
            st = dumped_streams(self.cells.N[self.cc[new]], self.uid[new], SEED, NSIMU)
            got = oracle_chains(self.orc, self.packed, self.cc[new], co.default_opts(NSIMU, BURN, adaptint=ADAPTINT, qcovadj_always=1),
                                [x[new] for x in self.ins], st)
            self._refs.update(zip(new.tolist(), got))
        return [self._refs[int(i)] for i in idx]


@pytest.fixture(scope="module")
def S():
    return need_gpu().device_info(0)["sm_count"]


@pytest.fixture(scope="module")
def tdata(orc, gpu_cells, cells_npz, S):
    """Chains on the 299 TestData cells (max N = 129: regular layout, two CTAs per SM), enough for every count below."""
    return Workload(orc, gpu_cells, cells_npz, max(CONFIG3, GROUP * S + 1, 13 * S), 7001)


@pytest.fixture(scope="module")
def big257(orc, S):
    """Chains on 8 cells of N = 257 (irregular and regular grids): the big layout, one CTA per SM."""
    need_gpu()
    cells, packed = make_cells(orc[0], cols(orc, [257] * 8, 7002))
    yield Workload(orc, cells, packed, UNSLICED, 7003)
    cells.close()


# ------------------------------------------------------------------------------------------------ 1. chain-count sweep
# (test id, layout, nc from S).  The id names the regime the launch runs in on a B200 (S = 148).
SWEEP = [
    ("cta-one_chain_per_cta-S", _lib.LAYOUT_CTA, lambda S: S),
    ("cta-solo_sm-S+1", _lib.LAYOUT_CTA, lambda S: S + 1),
    ("cta-solo_sm_two_ctas_per_sm-2S", _lib.LAYOUT_CTA, lambda S: 2 * S),
    ("cta-queued-2S+1", _lib.LAYOUT_CTA, lambda S: 2 * S + 1),
    ("cta-queued_config2-299", _lib.LAYOUT_CTA, lambda S: 299),
    ("cta-queued_sliced-1183", _lib.LAYOUT_CTA, lambda S: UNSLICED - 1),
    ("cta-unsliced_any_free_chain-1184", _lib.LAYOUT_CTA, lambda S: UNSLICED),
    ("big-one_chain_per_cta-S", _lib.LAYOUT_BIG, lambda S: S),
    ("big-queued-S+1", _lib.LAYOUT_BIG, lambda S: S + 1),
    ("big-queued_sliced-1183", _lib.LAYOUT_BIG, lambda S: UNSLICED - 1),
    ("big-unsliced_any_free_chain-1184", _lib.LAYOUT_BIG, lambda S: UNSLICED),
    ("warp-one_group_per_cta_ragged-16S-1", _lib.LAYOUT_WARP, lambda S: GROUP * S - 1),
    ("warp-one_group_per_cta-16S", _lib.LAYOUT_WARP, lambda S: GROUP * S),
    ("warp-parked_groups_ragged-16S+1", _lib.LAYOUT_WARP, lambda S: GROUP * S + 1),
    ("warp-parked_groups_config3-19136", _lib.LAYOUT_WARP, lambda S: CONFIG3),
    ("auto-cta_below_13_per_sm-13S-1", _lib.LAYOUT_AUTO, lambda S: 13 * S - 1),
    ("auto-warp_from_13_per_sm-13S", _lib.LAYOUT_AUTO, lambda S: 13 * S),
]


@pytest.mark.parametrize("case", SWEEP, ids=[c[0] for c in SWEEP])
def test_chain_count_sweep(request, S, case):
    """One launch of nc chains on one GPU, then:
    (1) the same chains in a seeded random order, each uid moving with its chain: flags, sschain, mean, std, sig and the
        counters of every chain bit-identical;
    (2) the sample alone (16-24 chains), on the same sampler, with its rows stored: bit-identical to the launch; rows,
        flags, s2chain, sschain and the seven counters the oracle's on the dumped streams; mean and std those of its own
        rows (long-double two-pass, within 1e-13 max|x|);
    (3) the sample in the launch against the oracle: flags, sschain, the seven counters, the summaries;
    and which sampler ran, from the counters (under AUTO: dram_warp_kernel exactly from 13 S chains on)."""
    name, layout, nc_of = case
    wl = request.getfixturevalue("big257" if layout == _lib.LAYOUT_BIG else "tdata")
    nc = nc_of(S)
    out = wl.run(np.arange(nc), layout)
    warp = layout == _lib.LAYOUT_WARP or (layout == _lib.LAYOUT_AUTO and nc >= 13 * S)
    assert_one_sampler(name, out, "warp" if warp else "cta")

    perm = np.random.default_rng(nc).permutation(nc)
    pout = wl.run(perm, layout)
    assert_same_chains(name + " permuted", pout, _take(out, perm))

    smp = _sample(nc, S, warp, nc)
    refs = wl.refs(smp)
    alone = wl.run(smp, _lib.LAYOUT_WARP if warp else (_lib.LAYOUT_CTA if layout == _lib.LAYOUT_AUTO else layout), store_chain=1)
    assert_one_sampler(name + " alone", alone, "warp" if warp else "cta")
    assert_same_chains(name + " alone", alone, _take(out, smp), keys=OUT_KEYS)
    drow = dmean = 0.0
    for j, (i, ref) in enumerate(zip(smp, refs)):
        npar = wl.npar(i)
        check_chain(name + " alone", alone, j, ref, npar, first_row=BURN - 1)
        rows = alone["chain"][j, :, :npar]
        m, s = ld_mean_std(rows)
        scale = np.abs(rows).max(axis=0)
        assert np.all(np.abs(alone["mean"][j, :npar] - m) <= 1e-13 * scale), (name, int(i))
        assert np.all(np.abs(alone["std"][j, :npar] - s) <= 1e-10 * s + 1e-13 * scale), (name, int(i))
        drow = max(drow, float(np.max(np.abs(rows - ref["chain"][BURN - 1:]))))
        dmean = max(dmean, float(np.max(np.abs(out["mean"][i, :npar] - ref["chain"][BURN - 1:].mean(axis=0)))))
        check_summaries(name, out, i, ref, npar, n_burn=BURN)
    print("%s: nc = %d, %d chains against the oracle (max |row - oracle| %.2g, max |mean - oracle| %.2g), kernel %.3f s"
          % (name, nc, smp.size, drow, dmean, out["kernel_seconds"]))


# ------------------------------------------------------------------------------------------------ 2. benchmarked workloads
def test_config3_as_benched_against_oracle(orc, gpu_cells, cells_npz, S):
    """BASELINE config 3 as bench.py runs it on one GPU: 299 cells x 64 chains = 19 136 chains under AUTO (dram_warp_kernel,
    1 196 groups for S CTAs), 20 000 steps, burn-in and n_burn 10 000, default options (chol(cov) first), no flags.  Four
    chains — the first, the first of the first group without a CTA of its own, one at random, the last — against the oracle
    on the dumped streams: the seven counters exactly, mean / std / sig to 1e-6 (test_replay_long_default_path's rows)."""
    from transcriptioncycleinference_b200 import setup_cell
    co, _ = orc
    cc = np.repeat(np.arange(299, dtype=np.int32), 64)
    uid = cc.astype(np.uint64) * np.uint64(1 << 20) + np.tile(np.arange(64, dtype=np.uint64), 299)
    inputs = setup_cell.chain_inputs(gpu_cells, cc, np.random.default_rng(1000))
    nsimu, burn, seed = 20000, 10000, 20201028
    opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=burn, store_chain=0, seed=seed, ngpus=1)
    out = gpu_cells.mcmc_run(opts, cc, *inputs, chain_uid=uid)
    assert out["flags"] is None
    assert_one_sampler("config3", out, "warp")
    sel = np.array(sorted({0, GROUP * S, int(np.random.default_rng(3).integers(cc.size)), cc.size - 1}))
    refs = oracle_chains(orc, cells_npz, cc[sel], co.default_opts(nsimu, burn), [x[sel] for x in inputs],
                         dumped_streams(cells_npz["N"][cc[sel]], uid[sel], seed, nsimu))
    for i, ref in zip(sel, refs):
        check_summaries("config3", out, i, ref, 7 + int(cells_npz["N"][cc[i]]), n_burn=burn, atol=1e-6)
    print("config3: kernel %.3f s, chains %s against the oracle" % (out["kernel_seconds"], sel.tolist()))


def test_config5_as_benched_against_oracle(orc, S):
    """BASELINE config 5's shape as bench.py's config5_leg builds it: 1 184 synthetic cells of N = 400 (npar = 407: the big
    layout, one CTA per SM, 8 chains per CTA, unsliced), one chain each with chain_uid = NULL (the chain index), AUTO.
    600 steps with burn-in and n_burn 300 and qcovadj_always = 1: 300-row covariances of 407 parameters are singular.  Six
    chains — first, last, both sides of chain S, two at random — against the oracle on the dumped streams."""
    from transcriptioncycleinference_b200 import setup_cell, synthetic
    need_gpu()
    co, _ = orc
    cells, _ = synthetic.make_cells(UNSLICED, 400)
    try:
        cc = np.arange(UNSLICED, dtype=np.int32)
        inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(5))
        nsimu, burn = 600, 300
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, n_burn=burn, qcovadj_always=1, ngpus=1)
        out = cells.mcmc_run(opts, cc, *inputs, want_flags=True)
        assert_one_sampler("config5", out, "cta")
        rng = np.random.default_rng(5)
        sel = np.array(sorted({0, S - 1, S, UNSLICED - 1} | {int(x) for x in rng.choice(UNSLICED, 2, replace=False)}))
        packed = dict(N=cells.N, off=cells.off, t=cells.t, ms2=cells.ms2, pp7=cells.pp7)
        for c in sel:
            assert np.array_equal(cells.t_interp(c), co.t_interp(cells.cell(c)[0])), c
        refs = oracle_chains(orc, packed, cc[sel], co.default_opts(nsimu, burn, qcovadj_always=1), [x[sel] for x in inputs],
                             dumped_streams(cells.N[sel], sel.astype(np.uint64), opts.seed, nsimu))
        for i, ref in zip(sel, refs):
            check_summaries("config5", out, i, ref, 407, n_burn=burn)
        print("config5: kernel %.3f s, chains %s against the oracle" % (out["kernel_seconds"], sel.tolist()))
    finally:
        cells.close()


# ------------------------------------------------------------------------------------------------ 3. several GPUs
@pytest.fixture(scope="module")
def D():
    if need_gpu().device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    return min(_lib.MAX_GPUS, _lib.device_count())


@pytest.fixture(scope="module")
def tdata_multi(cells_npz, D):
    """The TestData cells resident on devices 0 .. D-1."""
    from transcriptioncycleinference_b200.engine import Cells
    g = cells_npz
    cells = Cells.from_packed(g["N"], g["off"], g["t"], g["ms2"], g["pp7"], devices=tuple(range(D)))
    yield cells
    cells.close()


@pytest.mark.parametrize("layout,name", [(_lib.LAYOUT_WARP, "warp"), (_lib.LAYOUT_AUTO, "auto")], ids=["warp", "auto"])
def test_partition_config3_size_any_gpu_count(tdata, tdata_multi, D, layout, name):
    """19 136 chains on 1, 2 and D GPUs: every device holds at least 13 S chains, so under AUTO too every device runs
    dram_warp_kernel, and every output of every chain is bit-identical to the one-GPU launch."""
    idx = np.arange(CONFIG3)
    base = tdata.run(idx, layout, cells=tdata_multi, ngpus=1)
    assert_one_sampler(name, base, "warp")
    for ng in sorted({2, D}):
        out = tdata.run(idx, layout, cells=tdata_multi, ngpus=ng)
        assert_one_sampler("%s ngpus=%d" % (name, ng), out, "warp")
        assert_same_chains("%s ngpus=%d" % (name, ng), out, base)


@pytest.fixture(scope="module")
def edge_cells(orc, D):
    """Cells of N = 12 (irregular grid), 129 (regular) and 200 (irregular), resident on devices 0 .. D-1."""
    cells, packed = make_cells(orc[0], cols(orc, (12, 129, 200), 7004))
    cells.close()
    from transcriptioncycleinference_b200.engine import Cells
    cells = Cells.from_packed(packed["N"], packed["off"], packed["t"], packed["ms2"], packed["pp7"], devices=tuple(range(D)))
    yield cells, packed
    cells.close()


@pytest.mark.parametrize("which", ["1", "D-1", "D", "D+1", "D+1-reversed"])
def test_partition_edges(orc, edge_cells, D, which):
    """ngpus = D with 1, D-1, D and D+1 chains (fewer chains than devices: one chain per device), on cells of N = 200, 12 and
    129 in turn, so that the cuts of sum N^2 are uneven; chain_uid = NULL (the uid of a chain is its global index, whichever
    device runs it); rows stored; once with devices[] in reverse order.  Every output, rows included, bit-identical to the
    one-GPU launch, and on D+1 chains every chain the oracle's."""
    from transcriptioncycleinference_b200 import setup_cell
    co, _ = orc
    cells, packed = edge_cells
    nch = {"1": 1, "D-1": D - 1, "D": D, "D+1": D + 1, "D+1-reversed": D + 1}[which]
    cc = np.array([2, 0, 1] * D, dtype=np.int32)[:nch]
    ins = setup_cell.chain_inputs(cells, cc, np.random.default_rng(7005))
    nsimu, burn, n_burn, seed = 600, 200, 100, 7006
    kw = dict(nsimu=nsimu, burnintime=burn, n_burn=n_burn, store_chain=1, seed=seed, qcovadj_always=1)
    base = cells.mcmc_run(_lib.default_opts(ngpus=1, **kw), cc, *ins, want_flags=True)
    opts = _lib.default_opts(ngpus=D, **kw)
    if which.endswith("reversed"):
        for g in range(D):
            opts.devices[g] = D - 1 - g
    out = cells.mcmc_run(opts, cc, *ins, want_flags=True)
    assert_same_chains("partition %s" % which, out, base)
    if nch == D + 1:
        refs = oracle_chains(orc, packed, cc, co.default_opts(nsimu, burn, qcovadj_always=1), ins,
                             dumped_streams(packed["N"][cc], np.arange(nch, dtype=np.uint64), seed, nsimu))
        for i, ref in enumerate(refs):
            check_chain("partition %s" % which, out, i, ref, 7 + int(packed["N"][cc[i]]), first_row=n_burn - 1)


def test_auto_window_gpu_count_picks_the_sampler(tdata, tdata_multi, S, D):
    """13 S chains under AUTO: one GPU runs dram_warp_kernel, two GPUs (13 S / 2 chains each) run dram_kernel.  The two-GPU
    fit is bit-identical to the one-GPU fit forced onto dram_kernel (TC_LAYOUT_CTA), and a sample of both fits is the oracle's
    chain; the two samplers agree with each other to the rounding of their Cholesky orders (DESIGN.md 2): the same flags and
    counters, means within 1e-6."""
    idx = np.arange(13 * S)
    one = tdata.run(idx, _lib.LAYOUT_AUTO, cells=tdata_multi, ngpus=1)
    two = tdata.run(idx, _lib.LAYOUT_AUTO, cells=tdata_multi, ngpus=2)
    cta = tdata.run(idx, _lib.LAYOUT_CTA, cells=tdata_multi, ngpus=1)
    assert_one_sampler("auto 1 GPU", one, "warp")
    assert_one_sampler("auto 2 GPUs", two, "cta")
    assert_same_chains("auto 2 GPUs vs CTA on 1", two, cta)
    smp = _sample(idx.size, S, True, 7007, n=12)
    for i, ref in zip(smp, tdata.refs(smp)):
        check_summaries("auto 1 GPU", one, i, ref, tdata.npar(i), n_burn=BURN)
        check_summaries("auto 2 GPUs", two, i, ref, tdata.npar(i), n_burn=BURN)
    _report_cross_sampler("auto 1 GPU vs 2 GPUs", one, two)


def test_auto_window_samplers_agree_to_rounding(tdata, S):
    """The one-GPU half of the window, on any box: 13 S chains under AUTO (dram_warp_kernel) against the same chains on
    TC_LAYOUT_CTA (dram_kernel: what each device of a multi-GPU fit of them runs).  Same flags and counters, means within
    1e-6; how many chains are bit-identical is printed."""
    idx = np.arange(13 * S)
    warp = tdata.run(idx, _lib.LAYOUT_AUTO)
    cta = tdata.run(idx, _lib.LAYOUT_CTA)
    assert_one_sampler("auto", warp, "warp")
    assert_one_sampler("cta", cta, "cta")
    _report_cross_sampler("warp vs cta", warp, cta)


def _report_cross_sampler(tag, a, b):
    assert_same_chains(tag, a, b, keys=("flags",))
    np.testing.assert_allclose(a["mean"], b["mean"], rtol=0, atol=1e-6, err_msg=tag)
    np.testing.assert_allclose(a["sig"], b["sig"], rtol=1e-9, err_msg=tag)
    same = np.all(a["mean"] == b["mean"], axis=1) & np.all(a["std"] == b["std"], axis=1) & np.all(a["sig"] == b["sig"], axis=1)
    print("%s: %d of %d chains bit-identical, max |mean difference| %.3g" % (tag, int(same.sum()), same.size,
                                                                            float(np.max(np.abs(a["mean"] - b["mean"])))))
