"""GPU parity along the third input of a fit: the bounds and the Gaussian prior (low, upp, prior_mu, prior_sig), against the
C oracle (oracle/tc_oracle.c: prior_ss, out_of_bounds, orc_dram), on every sampler layout.

test_gpu_lengths.py varies the series length and test_gpu_schedule.py the step axis; both build their bounds and priors
with setup_cell.chain_inputs, the reference's structure at its default ratePriorWidth of 50 (prior_mu = 0, prior_sig = Inf
on the seven head parameters, 50 on every dR), where the prior moves the log acceptance by ~1e-2 per step.  Both samplers
check once per time slice whether a chain's vectors have that structure — seven head parameters, then one block whose
entries all equal parameter 7 (`uni` in dram_kernel and dram_warp_kernel) — and then read entries j >= 8 from one
register copy; otherwise every entry is read per parameter (cand_bounds_t / wk_check, UNI and generic instances).  Here
each chain of a launch gets its own variant, so that both paths share one CTA and one 16-chain warp group:

  A. tight rate priors (width 0.5 and 2) around a non-zero common mean: the prior dominates the dR block;
  B. finite head priors with non-zero means, the block uniform;
  C. the structure broken at one position p (7, 8, 31-33, 63, 64, 127, 128, npar - 1) in each of the four vectors;
  D. infinite and one-sided bounds, a whole block at +-Inf, prior_sig = Inf on part of the block, -0.0 against 0.0;
  E. the stage-1 proposal of step 1 exactly on a bound (in bounds) and one ulp outside it (out of bounds).

Runs: replays with injected randomness (flag for flag, every counter, the recorded SS, mean / std), the production
Philox path over many time slices (the detection runs again on every slice), a padded leading dimension under the big
layout (bounds and prior means read from HBM at stride ld), and the two paths against each other bit for bit.

Cells: N = 12 on an irregular grid and N = 129 on a regular one (npar = 136: the chain-per-warp kernel's fifth parameter
iteration), on every layout; a dataset with N = 257 (where the big layout is chosen automatically) under the big layout."""
import numpy as np
import pytest

from parity import (LAYOUTS, ORC_OOB, check_chain, check_recorded_ss, cols, dumped_streams, ld_mean_std, make_cells, need_gpu,
                    oracle_chains, replay_streams)
from transcriptioncycleinference_b200 import _lib

pytestmark = pytest.mark.gpu
NSIMU, BURN, ADAPT = 600, 200, 100
POSITIONS = (7, 8, 31, 32, 33, 63, 64, 127, 128)       # and npar - 1
KEYS = ("th0", "q", "lo", "hi", "mu", "sg")              # the six chain inputs, in tc_mcmc_run's order
BLOCK_MU = 1.5


# ------------------------------------------------------------------------------------------------ input families
# A modifier edits one chain's rows in place: x maps KEYS (and "z1", the stage-1 normals of step 1, when known) to 1-D views
# of length ld; npar = 7 + N.  It returns True if the chain keeps the reference's structure (the UNI path).
def tight(w, m):
    def f(x, npar):
        x["sg"][7:npar] = w; x["mu"][7:npar] = m
        return True
    return f


HEAD_MU = np.array([2.0, 1.5, 2.5, 1.0, 0.8, 0.4, 14.0])
HEAD_SIG = np.array([0.3, 0.8, 0.6, 0.5, 0.5, 0.15, 2.0])


def head_priors(scale, block_mu, shift):
    def f(x, npar):
        x["mu"][:7] = HEAD_MU + shift * HEAD_SIG; x["sg"][:7] = HEAD_SIG * scale; x["mu"][7:npar] = block_mu
        return True
    return f


def broken(p, what):
    """The block of a tight prior (width 2 around BLOCK_MU) with one entry changed: p = 7 breaks its reference entry, p = -1
    stands for npar - 1."""
    def f(x, npar):
        q = npar - 1 if p < 0 else p
        tight(2.0, BLOCK_MU)(x, npar)
        if what == "lo":
            x["lo"][q] = min(x["th0"][q], BLOCK_MU) - 3.0
        elif what == "hi":
            x["hi"][q] = max(x["th0"][q], BLOCK_MU) + 3.0
        elif what == "mu":
            x["mu"][q] = -2.5
        else:
            x["sg"][q] = 0.6
        return False
    f.applies = lambda npar: p < npar
    return f


def head_inf(x, npar):
    """lower bounds of the basal levels at -Inf, upper bounds of v, tau and R at +Inf: the block is untouched."""
    x["lo"][[3, 4]] = -np.inf; x["hi"][[0, 1, 6]] = np.inf
    return True


def block_mixed_inf(x, npar):
    tight(2.0, BLOCK_MU)(x, npar)
    x["lo"][7:npar:3] = -np.inf; x["hi"][8:npar:4] = np.inf
    return False


def block_inf(x, npar):
    """the whole block at [-Inf, Inf]: the structure holds, with infinite block bounds."""
    tight(2.0, BLOCK_MU)(x, npar)
    x["lo"][7:npar] = -np.inf; x["hi"][7:npar] = np.inf
    return True


def sig_part_inf(first):
    def f(x, npar):
        tight(2.0, BLOCK_MU)(x, npar)
        if first:
            x["sg"][7] = np.inf                                      # the reference entry flat, the rest finite
        else:
            x["sg"][9:npar:2] = np.inf
        return False
    return f


def neg_zero(x, npar):
    """-0.0 against 0.0: head lower bounds, and a block bounded below at zero whose low and prior_mu alternate the sign of
    zero.  Compared with ==, the structure holds."""
    x["lo"][1:5] = -0.0
    x["th0"][7:npar] = np.abs(x["th0"][7:npar])
    x["lo"][7:npar] = 0.0; x["lo"][8:npar:2] = -0.0
    x["mu"][7:npar] = -0.0; x["mu"][9:npar:2] = 0.0
    x["sg"][7:npar] = 2.0
    return True


def on_bound(side, where, outside):
    """A bound at the stage-1 proposal of step 1, x0[j] + z1[j] sqrt(q[j]) (the factor is diag(sqrt(qcov_diag)) there, and
    that is the double both the oracle's propose and the samplers form), or one ulp beyond it."""
    def f(x, npar):
        prop = x["th0"][:npar] + x["z1"][:npar] * np.sqrt(x["q"][:npar])
        sgn = -1.0 if side == "lo" else 1.0
        js = range(7) if where == "head" else range(7, npar)
        ok = [j for j in js if sgn * x["z1"][j] > 0.3 and x["lo"][j] < prop[j] < x["hi"][j]]
        assert ok, (side, where)
        j = ok[len(ok) // 2]
        b = prop[j] if not outside else np.nextafter(prop[j], -sgn * np.inf)
        x[side][j] = b
        f.j = j
        return where == "head"
    return f


FAMILIES = {
    "A": [tight(0.5, BLOCK_MU), tight(2.0, BLOCK_MU), tight(0.5, -0.75), tight(2.0, -0.75)],
    "B": [head_priors(1.0, 0.0, 0.5), head_priors(3.0, -1.0, -1.0), head_priors(1.0, 0.7, 0.0)],
    "C": [broken(p, w) for p in POSITIONS + (-1,) for w in ("lo", "hi", "mu", "sg")],
    "D": [head_inf, block_mixed_inf, block_inf, sig_part_inf(True), sig_part_inf(False), neg_zero],
    "E": [on_bound(s, w, o) for s in ("lo", "hi") for w in ("head", "block") for o in (False, True)],
}


def _applies(f, npar):
    return getattr(f, "applies", lambda n: True)(npar)


def plan(cells, mods, nref=1, first_plain=False):
    """Chains over every cell: one per modifier (family, f) that applies to the cell's length, with nref unmodified chains
    (the reference's structure at width 50) before every fourth, so that variants of both paths and plain chains share
    CTAs and warp groups.  first_plain: chain 0 is a plain chain (the variants sit at indices > 0)."""
    rows = [(0, (None, None))] if first_plain else []
    for c in range(cells.ncells):
        npar = 7 + int(cells.N[c])
        ms = [m for m in mods if _applies(m[1], npar)]
        for k, m in enumerate(ms):
            if k % 4 == 0:
                rows += [(c, (None, None))] * nref
            rows.append((c, m))
    return np.array([c for c, _ in rows], dtype=np.int32), [m for _, m in rows]


def apply(cells, cc, mods, seed, z1=None, ld_pad=0):
    """chain_inputs for cc (padded by ld_pad columns, filled as chain_inputs pads), then every chain's modifier.  z1: the
    step-1 normals [nch, >= npar] (family E).  Returns (ins, base, info): base = the inputs before the modifiers, info[i] =
    (family, uni, j) with j the parameter family E put its bound on."""
    from transcriptioncycleinference_b200 import setup_cell
    ins = setup_cell.chain_inputs(cells, cc, np.random.default_rng(seed))
    if ld_pad:
        fill = (0.0, 1.0, 0.0, 0.0, 0.0, np.inf)
        ins = [np.concatenate([x, np.full((cc.size, ld_pad), v)], axis=1) for x, v in zip(ins, fill)]
    ins = [np.ascontiguousarray(x) for x in ins]
    base = [x.copy() for x in ins]
    info = []
    for i, (fam, f) in enumerate(mods):
        npar = 7 + int(cells.N[cc[i]])
        x = dict(zip(KEYS, (a[i] for a in ins)))
        if z1 is not None:
            x["z1"] = z1[i]
        uni = True if f is None else f(x, npar)
        info.append((fam, uni, getattr(f, "j", None)))
        assert np.all(x["lo"][:npar] <= x["th0"][:npar]) and np.all(x["th0"][:npar] <= x["hi"][:npar]), (fam, i)
    return ins, base, info


def _fam(*names):
    return [(n, f) for n in names for f in FAMILIES[n]]


def _check_run(tag, cells, cc, out, refs):
    """check_chain for every chain, the recorded SS of every row, and mean / population std of the stored rows against a
    long-double reduction of the oracle's rows (the rows agree to 1e-7)."""
    for i, ref in enumerate(refs):
        npar = 7 + int(cells.N[cc[i]])
        check_chain(tag, out, i, ref, npar)
        m, s = ld_mean_std(ref["chain"])
        np.testing.assert_allclose(out["mean"][i, :npar], m.astype(np.float64), rtol=0, atol=2e-7, err_msg=str((tag, i)))
        np.testing.assert_allclose(out["std"][i, :npar], s.astype(np.float64), rtol=0, atol=2e-7, err_msg=str((tag, i)))
    check_recorded_ss(cells, cc, out, out["chain"].shape[2])


def _replay_opts(layout, nsimu=NSIMU):
    return _lib.default_opts(nsimu=nsimu, burnintime=BURN, adaptint=ADAPT, n_burn=1, store_chain=1, replay=1, layout=layout,
                             qcovadj_always=1)


def _orc_opts(co, nsimu=NSIMU, burn=BURN):
    return co.default_opts(nsimu, burn, adaptint=ADAPT, qcovadj_always=1)


@pytest.fixture(scope="module")
def cells2(orc):
    """N = 12 on an irregular grid, N = 129 on a regular grid."""
    need_gpu()
    cells, packed = make_cells(orc[0], cols(orc, (12, 129), 4243))
    assert cells.N.tolist() == [12, 129]
    yield cells, packed
    cells.close()


@pytest.fixture(scope="module")
def cells3(orc):
    """N = 12, 129 and 257 in one dataset (ld = 264: the big layout is the one chosen automatically)."""
    need_gpu()
    cells, packed = make_cells(orc[0], cols(orc, (12, 129, 257), 4244))
    assert cells.N.tolist() == [12, 129, 257]
    yield cells, packed
    cells.close()


# ------------------------------------------------------------------------------------------------ 1. replays
def _family_replay(orc, cells, packed, names, layouts, seed):
    need_gpu()
    co, _ = orc
    cc, mods = plan(cells, _fam(*names))
    st = replay_streams(cells.N[cc], NSIMU, cells.ld, seed)
    ins, base, info = apply(cells, cc, mods, seed + 1, z1=st["z1"][:, 1])
    assert any(u for _, u, _ in info) and (names[0] in "AB" or not all(u for _, u, _ in info))
    refs = oracle_chains(orc, packed, cc, _orc_opts(co), ins, st)
    for layout, name in layouts:
        out = cells.mcmc_run(_replay_opts(layout), cc, *ins, replay=st, want_flags=True)
        _check_run("%s %s" % ("".join(names), name), cells, cc, out, refs)
    return cc, ins, base, info, st, refs


def _guard_tight_prior(orc, cells, packed, cc, base, info, st, refs):
    """Family A: on the same streams the oracle's flags at width 0.5 differ from its flags at the reference's width 50."""
    co, _ = orc
    idx = [i for i, (fam, _, _) in enumerate(info) if fam == "A"]
    wide = oracle_chains(orc, packed, cc[idx], _orc_opts(co), [x[idx] for x in base], {k: v[idx] for k, v in st.items()})
    diff = {}
    for k, i in enumerate(idx):
        sg = np.unique(base[5][i][7:7 + int(cells.N[cc[i]])])
        assert sg.tolist() == [50.0]
        diff[i] = int(np.sum(refs[i]["flags"] != wide[k]["flags"]))
    print("tight rate prior: flags changed against width 50 per chain (N, changed):",
          [(int(cells.N[cc[i]]), d) for i, d in diff.items()])
    assert all(d > 0 for d in diff.values()), diff
    return diff


def _check_on_bound(cells, cc, ins, info, st, refs):
    """Family E: the stage-1 proposal of step 1 is x0 + z1 sqrt(q); mcmcstat's rule (x < lower | x > upper) on it decides the
    oracle's (and so, flag for flag, every sampler's) TC_FL_OOB1 at step 1; exactly on the bound is inside, one ulp
    beyond is outside."""
    n = 0
    for i, (fam, _, j) in enumerate(info):
        if fam != "E":
            continue
        npar = 7 + int(cells.N[cc[i]])
        prop = ins[0][i, :npar] + st["z1"][i, 1, :npar] * np.sqrt(ins[1][i, :npar])
        lo, hi = ins[2][i, :npar], ins[3][i, :npar]
        on = prop[j] == lo[j] or prop[j] == hi[j]
        assert on or np.nextafter(prop[j], lo[j]) == lo[j] or np.nextafter(prop[j], hi[j]) == hi[j], (i, j)
        assert (prop[j] < lo[j] or prop[j] > hi[j]) == (not on), (i, j)
        oob = bool(np.any((prop < lo) | (prop > hi)))
        assert bool(refs[i]["flags"][1] & 4) == oob, (i, j, oob)
        if not on:
            assert oob and refs[i]["counters"][ORC_OOB] >= 1
        n += 1
    assert n >= 8


@pytest.mark.parametrize("fam", sorted(FAMILIES))
def test_family_replay(orc, cells2, fam):
    """600 steps, burn-in 200, adaptint 100, qcovadj_always = 1, every layout: flags, rows, s2chain, sschain, all counters
    (out-of-bounds proposals and delayed-rejection tries included), the recorded SS of every row, mean and std."""
    cells, packed = cells2
    cc, ins, base, info, st, refs = _family_replay(orc, cells, packed, (fam,), LAYOUTS, 100 + ord(fam))
    if fam == "A":
        _guard_tight_prior(orc, cells, packed, cc, base, info, st, refs)
    if fam == "E":
        _check_on_bound(cells, cc, ins, info, st, refs)


@pytest.mark.parametrize("fam", sorted(FAMILIES))
def test_family_replay_long_cell_big_layout(orc, cells3, fam):
    """The same with a cell of N = 257 in the dataset, under the big layout, where bounds and prior means are read from
    HBM at stride ld = 264 for every chain (npar = 19, 136, 264)."""
    cells, packed = cells3
    cc, ins, base, info, st, refs = _family_replay(orc, cells, packed, (fam,), [(_lib.LAYOUT_BIG, "big")], 200 + ord(fam))
    if fam == "E":
        _check_on_bound(cells, cc, ins, info, st, refs)


# ------------------------------------------------------------------------------------------------ 2. production Philox
PHILOX_C = [("C", broken(p, w)) for p in (7, 33, 128, -1) for w in ("lo", "mu")]


def test_production_families_against_oracle(orc, cells2):
    """Families A, B, D and part of C in one launch on the device's Philox streams, 3300 steps (burn-in 1000, adaptint
    100): many time slices, so the structure check runs again on every slice and dram_warp_kernel reuses the reciprocal
    widths it stored at slice 0.  Every layout against the oracle on tc_rng_dump's streams."""
    need_gpu()
    co, _ = orc
    cells, packed = cells2
    nsimu, burn, seed = 3300, 1000, 2718
    cc, mods = plan(cells, _fam("A", "B", "D") + PHILOX_C)
    ins, _, info = apply(cells, cc, mods, 300)
    uid = np.arange(cc.size, dtype=np.uint64) * np.uint64(31) + np.uint64(17)
    refs = oracle_chains(orc, packed, cc, _orc_opts(co, nsimu, burn), ins, dumped_streams(cells.N[cc], uid, seed, nsimu))
    for layout, name in LAYOUTS:
        opts = _lib.default_opts(nsimu=nsimu, burnintime=burn, adaptint=ADAPT, n_burn=1, store_chain=1, seed=seed,
                                 layout=layout, qcovadj_always=1)
        out = cells.mcmc_run(opts, cc, *ins, chain_uid=uid, want_flags=True)
        for i, ref in enumerate(refs):
            check_chain("philox %s %s" % (name, info[i][0]), out, i, ref, 7 + int(cells.N[cc[i]]))


# ------------------------------------------------------------------------------------------------ 3. padded ld, big layout
def test_padded_leading_dimension_big_layout(orc, cells2):
    """ld = 7 + max N + 5 for every array, chain 0 plain and the variants of every family at indices > 0: under the big
    layout each chain's bounds and prior means are read from HBM at ch * ld.  Replayed against the oracle on every layout.
    (This found dram_warp_kernel carving its per-warp shared-memory regions and increment slots for N = ld - 7 while the
    host had sized them for max N: with a padded ld the last warps ran past both.)"""
    need_gpu()
    co, _ = orc
    cells, packed = cells2
    fams = _fam("A", "B", "D", "E") + [m for m in _fam("C") if m[1] in FAMILIES["C"][::3]]
    cc, mods = plan(cells, fams, first_plain=True)
    ld = cells.ld + 5
    st = replay_streams(cells.N[cc], NSIMU, ld, 400)
    ins, _, info = apply(cells, cc, mods, 401, z1=st["z1"][:, 1], ld_pad=5)
    assert info[0][0] is None and ins[0].shape[1] == ld
    refs = oracle_chains(orc, packed, cc, _orc_opts(co), ins, st)
    for layout, name in [(_lib.LAYOUT_BIG, "big")] + [l for l in LAYOUTS if l[0] != _lib.LAYOUT_BIG]:
        out = cells.mcmc_run(_replay_opts(layout), cc, *ins, replay=st, want_flags=True)
        _check_run("ld+5 %s" % name, cells, cc, out, refs)
    _check_on_bound(cells, cc, ins, info, st, refs)


# ------------------------------------------------------------------------------------------------ 4. path against path
def test_uni_and_generic_paths_bit_for_bit(orc, cells2):
    """Pairs of chains on the same streams: one in the reference's structure, its copy with prior_mu changed at one position
    p of family C.  The block's prior is flat (prior_sig = Inf: the samplers' reciprocal width is 0), so (theta - mu) * 0
    is exactly 0 and only the path changes (a bound is never used for this: a bound moved out of reach can still be
    reached).  Finite head priors with non-zero means keep the prior sum non-trivial.  Replay and Philox (3300 steps, many
    time slices), every layout: flags, rows, s2chain, sschain, mean, std, sig and the counters are bit-identical."""
    need_gpu()
    cells, _ = cells2
    hp = head_priors(1.0, 0.75, 0.5)
    half = []
    for c in range(cells.ncells):
        npar = 7 + int(cells.N[c])
        half += [(c, p) for p in POSITIONS + (npar - 1,) if p < npar]
    cch = np.array([c for c, _ in half], dtype=np.int32)
    cc = np.repeat(cch, 2)
    from transcriptioncycleinference_b200 import setup_cell
    ins = [np.repeat(x, 2, axis=0) for x in setup_cell.chain_inputs(cells, cch, np.random.default_rng(500))]
    for i, (c, p) in enumerate(half):
        npar = 7 + int(cells.N[c])
        for r in (2 * i, 2 * i + 1):
            x = dict(zip(KEYS, (a[r] for a in ins)))
            assert hp(x, npar)
            x["sg"][7:npar] = np.inf
        ins[4][2 * i + 1, p] = 2.5
    sth = replay_streams(cells.N[cch], NSIMU, cells.ld, 501)
    st = {k: np.ascontiguousarray(np.repeat(v, 2, axis=0)) for k, v in sth.items()}
    uid = np.repeat(np.arange(cch.size, dtype=np.uint64) + np.uint64(900), 2)
    runs = [("replay", lambda layout: (_replay_opts(layout), dict(replay=st)))]
    runs.append(("philox", lambda layout: (_lib.default_opts(nsimu=3300, burnintime=1000, adaptint=ADAPT, n_burn=1,
                                                               store_chain=1, seed=77, layout=layout, qcovadj_always=1),
                                           dict(chain_uid=uid))))
    for rname, mk in runs:
        for layout, name in LAYOUTS:
            opts, kw = mk(layout)
            out = cells.mcmc_run(opts, cc, *ins, want_flags=True, **kw)
            a, b = slice(0, None, 2), slice(1, None, 2)
            for k in ("flags", "chain", "s2chain", "sschain", "mean", "std", "sig"):
                assert np.array_equal(out[k][a], out[k][b]), (rname, name, k, np.flatnonzero(np.any((out[k][a] != out[k][b]).reshape(cch.size, -1), axis=1)))
            assert np.array_equal(out["counters"][a, :8], out["counters"][b, :8]), (rname, name)
            acc = out["counters"][a, _lib.CNT_ACC_STAGE1] + out["counters"][a, _lib.CNT_ACC_STAGE2]
            assert np.all(acc > 0) and np.all(out["counters"][a, _lib.CNT_OUT_OF_BOUNDS] > 0), (rname, name)
