"""TranscriptionCycleMCMC — host-side mirror of the reference driver
(src/TranscriptionCycleMCMC.m, paths relative to the reference repo), same option names, same
defaults, same output .mat layouts; the MCMC itself runs in libtcmcmc.so on the GPU(s).

    TranscriptionCycleMCMC('fileDir', d, 'saveLoc', s, 'numParPools', 8, 'n_burn', 10000,
                           'n_steps', 20000, 'ratePriorWidth', 50, 't_start', 0, 't_end', inf,
                           'loadPrevious', True, 'construct', 'P2P-MS2v5-LacZ-PP7v4')

Differences that are deliberate and documented (DESIGN.md):
  * 'numParPools' is the number of GPUs (clamped to the devices present), not a MATLAB pool size.
  * no GUI: `listdlg` is replaced by "all *.mat files in fileDir that hold a `data` variable", or
    the optional 'files' list; `waitbar` by an optional 'verbose' print.  Paths are joined with
    os.path.join (the reference's hard-coded '\\' only works on Windows).
  * 'loadPrevious' works (the reference's branch is broken as shipped, SURVEY 0.1 #3): previous
    results are read from 'previousResults' (a results .mat in this same layout) or from the newest
    results file in fileDir whose DatasetName matches; cells are matched on cell_index, unmatched
    cells are skipped and removed, ApprovedFits is carried over.
  * raw chains beyond MAT v5's 2 GiB per variable (the reference's own defaults on TestData are 3.1 GB) are written as
    MATLAB-readable parts `<date>-<name>_RawChain_part<K>.mat` + an index (save_raw_chains, matlab/LoadRawChains.m).
  * new optional arguments: 'files', 'previousResults', 'numChains' (default 1), 'seed',
    'saveChains' (default True), 'thin' (default 1), 'verbose', 'returnResults'.  With numChains > 1 the chains of a
    cell are pooled in MCMCresults and an extra variable MCMCdiagnostics (Rhat, n_eff per parameter) is saved.
  * 'thin', k: MCMCchain keeps every k-th row — rows n_burn, n_burn + k, ... of the chain, and s2chain rows 1, 1 + k, ...
    (MATLAB numbering) — stored on the device as a regular subsample of the same chain, so raw chains fit in memory at
    sizes where every row would not; the raw-chain file then carries the scalar `thin`.  MCMCresults still summarise
    every row.
"""
import datetime
import glob
import os

import numpy as np

from . import _lib, diagnostics, setup_cell
from .constructs import DEFAULT_CONSTRUCT, get_construct
from .engine import Cells

RESULT_FIELDS = ("mean_v", "sigma_v", "mean_ton", "sigma_ton", "mean_A", "sigma_A", "mean_tau", "sigma_tau",
                 "mean_MS2_basal", "sigma_MS2_basal", "mean_PP7_basal", "sigma_PP7_basal", "mean_R", "sigma_R",
                 "mean_dR", "sigma_dR", "mean_sigma", "sigma_sigma", "cell_index", "ApprovedFits")  # :151-155
PLOT_FIELDS = ("t_plot", "MS2_plot", "PP7_plot", "simMS2", "simPP7")                                 # :156-157
DIAG_FIELDS = ("cell_index", "numChains", "Rhat", "n_eff", "Rhat_max", "split_Rhat", "ESS")   # extension, only with numChains > 1
# (Rhat, n_eff: from the device summaries, n_eff = the between-chain estimate; split_Rhat, ESS: from the raw chains — split
# halves, autocorrelation — empty unless saveChains; with 'thin' > 1 from the stored rows, so ESS counts stored draws)
CHAIN_FIELDS = ("v_chain", "ton_chain", "A_chain", "tau_chain", "MS2_basal_chain", "PP7_basal_chain", "R_chain",
                "dR_chain", "s2chain")                                                              # :149-150
_IDX = dict(v=0, tau=1, ton=2, MS2_basal=3, PP7_basal=4, A=5, R=6)


def parse_varargin(varargin):
    """The name/value scan of :36-78: case-insensitive names, every position is examined, unknown
    names are ignored, 'loadPrevious' is presence-only (its value, if any, is not read)."""
    o = dict(fileDir=os.getcwd(), saveLoc=os.getcwd(), numParPools=8, n_burn=10000, n_steps=20000,
             ratePriorWidth=50.0, t_start=0.0, t_end=np.inf, loadPrevious=False, construct=DEFAULT_CONSTRUCT,
             files=None, previousResults=None, numChains=1, seed=None, saveChains=True, thin=1, verbose=False,
             returnResults=False)
    names = {k.lower(): k for k in o}
    for i, v in enumerate(varargin):
        if not isinstance(v, str):
            continue
        key = names.get(v.lower())
        if key is None:
            continue
        if key == "loadPrevious":
            o["loadPrevious"] = True
        elif i + 1 < len(varargin):
            o[key] = varargin[i + 1]
        else:
            raise IndexError("Index exceeds the number of array elements (option %r has no value)" % v)
    return o


def matlab_date(d=None):
    """MATLAB `date`: dd-mmm-yyyy (:373)."""
    d = d or datetime.date.today()
    return "%02d-%s-%04d" % (d.day, ("Jan", "Feb", "Mar", "Apr", "May", "Jun", "Jul", "Aug", "Sep", "Oct", "Nov",
                                     "Dec")[d.month - 1], d.year)


def load_dataset(path):
    """`dat = load(file); dat.data` (:134-135): 1 x Ncells struct array with time, MS2, PP7, name."""
    import scipy.io as sio
    m = sio.loadmat(path, mat_dtype=True)
    if "data" not in m:
        raise KeyError("Reference to non-existent field 'data'. (%s)" % path)
    d = m["data"].reshape(-1)
    cells = []
    for c in d:
        cells.append(dict(time=np.asarray(c["time"], dtype=np.float64).reshape(-1),
                          MS2=np.asarray(c["MS2"], dtype=np.float64).reshape(-1),
                          PP7=np.asarray(c["PP7"], dtype=np.float64).reshape(-1),
                          name=str(np.asarray(c["name"]).reshape(-1)[0]) if np.asarray(c["name"]).size else ""))
    return cells


def load_previous_results(path):
    """mean_v / cell_index / ApprovedFits of an earlier fit (:101-106), keyed by cell_index."""
    import scipy.io as sio
    m = sio.loadmat(path, mat_dtype=True)
    r = m["MCMCresults"].reshape(-1)
    out = {}
    for c in r:
        out[int(np.asarray(c["cell_index"]).squeeze())] = (float(np.asarray(c["mean_v"]).squeeze()),
                                                           float(np.asarray(c["ApprovedFits"]).squeeze()))
    name = str(np.asarray(m.get("DatasetName", [""])).reshape(-1)[0]) if "DatasetName" in m else ""
    return out, name


def _find_previous(file_dir, dataset_name):
    import scipy.io as sio
    best = None
    for f in glob.glob(os.path.join(file_dir, "*.mat")):
        try:
            names = [n for n, _, _ in sio.whosmat(f)]
        except Exception:
            continue
        if "MCMCresults" not in names:
            continue
        try:
            nm = str(np.asarray(sio.loadmat(f, variable_names=["DatasetName"]).get("DatasetName", [""])).reshape(-1)[0])
        except Exception:
            nm = ""
        if nm == dataset_name and (best is None or os.path.getmtime(f) > os.path.getmtime(best)):
            best = f
    return best


def _struct_array(fields, records):
    arr = np.zeros((1, len(records)), dtype=[(f, "O") for f in fields])
    for i, r in enumerate(records):
        for f in fields:
            arr[0, i][f] = r[f]
    return arr


MAT5_LIMIT = 2 ** 31 - 2 ** 24          # bytes per MAT v5 variable (2 GiB), with room for the struct headers


def positive_int(value, name):
    """An option that must be a whole number >= 1 ('thin'): an int, or a float with an integral value as MATLAB passes it."""
    try:
        ok = not isinstance(value, (bool, np.bool_)) and float(value) == int(value) and int(value) >= 1
    except (TypeError, ValueError, OverflowError):
        ok = False
    if not ok:
        raise ValueError("'%s' must be an integer >= 1, got %r" % (name, value))
    return int(value)


def save_raw_chains(save_loc, base, chain, limit=MAT5_LIMIT, thin=1):
    """`save([saveLoc,'\',filename,'_RawChain.mat'],'MCMCchain')` (:377-378).  Plain `save` writes MAT v5, whose variables
    are limited to 2 GiB — the reference's own defaults on TestData (299 cells x 10 001 rows x ~128 doubles = 3.1 GB) already
    exceed that (SURVEY 0.1 #17).  Up to the limit: the reference's single file.  Beyond it: MATLAB-readable PARTS
    `<base>_RawChain_part<K>.mat`, each a v5 file below the limit holding `MCMCchain` for a run of whole cells
    (plus `firstCell`, `lastCell`: positions in the full 1 x Ncells array), and the index `<base>_RawChain.mat` with
    `MCMCchainParts` (file names), `MCMCchainPartOfCell` (1 x Ncells) and `nParts`; matlab/LoadRawChains.m puts them back
    together.  thin > 1 (rows thinned on the device, 'thin') adds the scalar `thin` next to `MCMCchain` in every file that
    holds it and in the index; thin = 1 writes the variables above and nothing else.  Returns the list of files written."""
    import scipy.io as sio
    sizes = [sum(np.asarray(v).nbytes for v in c.values()) for c in chain]
    if any(b > limit for b in sizes):
        raise ValueError("the raw chain of one cell (%d bytes) exceeds the MAT v5 variable limit: store fewer rows with the "
                         "option 'thin' or lower n_steps" % max(sizes))
    extra = dict(thin=float(thin)) if thin > 1 else {}
    path = os.path.join(save_loc, base + "_RawChain.mat")
    if sum(sizes) <= limit:
        sio.savemat(path, dict(MCMCchain=_struct_array(CHAIN_FIELDS, chain), **extra))
        return [path]
    groups, cur, cur_b = [], [], 0
    for i, b in enumerate(sizes):
        if cur and cur_b + b > limit:
            groups.append(cur); cur, cur_b = [], 0
        cur.append(i); cur_b += b
    groups.append(cur)
    files, part_of = [], np.zeros((1, len(chain)))
    for k, idx in enumerate(groups, start=1):
        fn = "%s_RawChain_part%d.mat" % (base, k)
        sio.savemat(os.path.join(save_loc, fn), dict(MCMCchain=_struct_array(CHAIN_FIELDS, [chain[i] for i in idx]),
                                                     firstCell=float(idx[0] + 1), lastCell=float(idx[-1] + 1), part=float(k),
                                                     **extra))
        files.append(fn); part_of[0, idx] = k
    sio.savemat(path, dict(MCMCchainParts=np.array(files, dtype=object).reshape(-1, 1), MCMCchainPartOfCell=part_of,
                           nParts=float(len(groups)), **extra))
    return [path] + [os.path.join(save_loc, f) for f in files]


def fit_dataset(cells_in, o, devices):
    """The parfor body (:161-357) for one dataset, all cells at once.  Returns (MCMCchain,
    MCMCresults, MCMCplot) as lists of dicts, already stripped of skipped cells (:360-369)."""
    n_burn, n_steps = int(o["n_burn"]), int(o["n_steps"])
    nchains = int(o["numChains"])
    thin = positive_int(o["thin"], "thin")
    rng = np.random.default_rng(o["seed"])
    prev = o.get("_prev")                                   # {cell_index: (mean_v, ApprovedFits)} or None
    kept, ts, m2s, p7s = [], [], [], []
    for ci, c in enumerate(cells_in):
        t, ms2, pp7 = setup_cell.truncate(c["time"], c["MS2"], c["PP7"], float(o["t_start"]), float(o["t_end"]))
        if o["loadPrevious"] and (prev is None or (ci + 1) not in prev):
            continue                                        # `continue` at :196-198 -> removed at :360-369
        if len(t) < 3:
            raise ValueError("cell %d has fewer than 3 timepoints in [t_start, t_end)" % (ci + 1))
        kept.append(ci); ts.append(t); m2s.append(ms2); p7s.append(pp7)
    if not kept:
        return [], [], []
    cells = Cells(ts, m2s, p7s, construct=o["construct"], devices=devices)
    try:
        cc = np.repeat(np.arange(len(kept), dtype=np.int32), nchains)
        v0 = None
        if o["loadPrevious"]:
            v0 = np.repeat([prev[ci + 1][0] for ci in kept], nchains)
        inputs = setup_cell.chain_inputs(cells, cc, rng, float(o["ratePriorWidth"]), v0)
        uid = (np.repeat(np.array(kept, dtype=np.uint64), nchains) << np.uint64(20)) + \
            np.tile(np.arange(nchains, dtype=np.uint64), len(kept))
        opts = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn,
                                 store_chain=1 if o["saveChains"] else 0, ngpus=len(devices),
                                 seed=int(rng.integers(0, 2 ** 63 - 1)), thin=thin)
        out = cells.mcmc_run(opts, cc, *inputs, chain_uid=uid)
        # pool the chains of a cell (numChains > 1 is an extension; with 1 chain this is the identity)
        MCMCchain, MCMCresults, MCMCplot = [], [], []
        means, diags = [], []
        for k, ci in enumerate(kept):
            N = len(ts[k]); npar = 7 + N
            sl = slice(k * nchains, (k + 1) * nchains)
            mu_c, sd_c = out["mean"][sl, :npar], out["std"][sl, :npar]
            mean = mu_c.mean(axis=0)
            # pooled population variance = mean of within-chain variances + variance of chain means
            std = np.sqrt((sd_c ** 2).mean(axis=0) + mu_c.var(axis=0))
            if o["saveChains"]:
                ch = out["chain"][sl, :, :npar].reshape(-1, npar)
                s2 = out["s2chain"][sl].reshape(-1)
                MCMCchain.append(dict(
                    v_chain=ch[:, [_IDX["v"]]], ton_chain=ch[:, [_IDX["ton"]]], A_chain=ch[:, [_IDX["A"]]],
                    tau_chain=ch[:, [_IDX["tau"]]], MS2_basal_chain=ch[:, [_IDX["MS2_basal"]]],
                    PP7_basal_chain=ch[:, [_IDX["PP7_basal"]]], R_chain=ch[:, [_IDX["R"]]], dR_chain=ch[:, 7:],
                    s2chain=s2.reshape(-1, 1)))
            else:
                MCMCchain.append({f: np.zeros((0, 0)) for f in CHAIN_FIELDS})
            if o["saveChains"] and thin == 1:
                mean_sigma, sigma_sigma = float(np.sqrt(s2.mean())), float(np.sqrt(s2).std())
            else:
                # sig of every row, from the device (a thinned s2chain holds only some of them)
                sg = out["sig"][sl]
                mean_sigma = float(np.sqrt((sg[:, 0] ** 2).mean()))
                sigma_sigma = float(sg[:, 1].mean()) if nchains == 1 else float(np.sqrt((sg[:, 1] ** 2).mean()))
            means.append(mean)
            if nchains > 1:
                # order of theta: [v, tau, ton, MS2_basal, PP7_basal, A, R, dR_1..dR_N]
                rh, ne = diagnostics.rhat_from_summaries(mu_c, sd_c, n_steps - n_burn + 1)
                d = dict(cell_index=float(ci + 1), numChains=float(nchains), Rhat=rh.reshape(1, -1),
                         n_eff=ne.reshape(1, -1), Rhat_max=float(np.nanmax(rh[:7])), split_Rhat=np.zeros((0, 0)), ESS=np.zeros((0, 0)))
                if o["saveChains"]:
                    raw = out["chain"][sl, :, :npar]
                    d["split_Rhat"] = diagnostics.split_rhat(raw).reshape(1, -1)
                    d["ESS"] = diagnostics.ess(raw).reshape(1, -1)
                diags.append(d)
            r = dict(mean_v=mean[0], sigma_v=std[0], mean_tau=mean[1], sigma_tau=std[1], mean_ton=mean[2],
                     sigma_ton=std[2], mean_MS2_basal=mean[3], sigma_MS2_basal=std[3], mean_PP7_basal=mean[4],
                     sigma_PP7_basal=std[4], mean_A=mean[5], sigma_A=std[5], mean_R=mean[6], sigma_R=std[6],
                     mean_dR=mean[7:].reshape(1, -1), sigma_dR=std[7:].reshape(1, -1), mean_sigma=mean_sigma,
                     sigma_sigma=sigma_sigma, cell_index=float(ci + 1),
                     ApprovedFits=float(prev[ci + 1][1]) if o["loadPrevious"] else 0.0)         # :343-350
            MCMCresults.append({f: (np.float64(r[f]) if np.ndim(r[f]) == 0 else r[f]) for f in RESULT_FIELDS})
        # best-fit curves at the posterior means on the RAW grid, no interp1 (:307-309)
        sim1, sim2 = cells.forward(np.arange(len(kept)), cells.pad_theta(means), on_raw_grid=True)
        for k in range(len(kept)):
            N = len(ts[k])
            MCMCplot.append(dict(t_plot=ts[k].reshape(1, -1), MS2_plot=m2s[k].reshape(1, -1),
                                 PP7_plot=p7s[k].reshape(1, -1), simMS2=sim1[k, :N].reshape(1, -1),
                                 simPP7=sim2[k, :N].reshape(1, -1)))
        o["_diagnostics"] = diags
        return MCMCchain, MCMCresults, MCMCplot
    finally:
        cells.close()


def TranscriptionCycleMCMC(*varargin):
    """See the module docstring.  Returns None like the reference (or the per-dataset results when
    'returnResults' is set)."""
    import scipy.io as sio
    o = parse_varargin(varargin)
    get_construct(o["construct"])                          # unknown construct: fail before any work
    positive_int(o["thin"], "thin")
    if int(o["n_burn"]) < 1 or int(o["n_burn"]) > int(o["n_steps"]):
        raise IndexError("n_burn must satisfy 1 <= n_burn <= n_steps (chain(n_burn:end,:))")
    ndev = _lib.device_count()
    if ndev < 1:
        raise RuntimeError("TranscriptionCycleMCMC: no CUDA device (libtcmcmc has no CPU fallback)")
    devices = list(range(max(1, min(int(o["numParPools"]), ndev))))
    file_dir, save_loc = o["fileDir"], o["saveLoc"]
    if o["files"] is not None:
        files = [f if os.path.isabs(f) else os.path.join(file_dir, f) for f in o["files"]]
    else:
        files = []
        for f in sorted(glob.glob(os.path.join(file_dir, "*.mat"))):
            try:
                if "data" in [n for n, _, _ in sio.whosmat(f)]:
                    files.append(f)
            except Exception:
                pass
    if not files:
        raise FileNotFoundError("no dataset (*.mat with a `data` variable) found in %s" % file_dir)
    ret = []
    for k, f in enumerate(files):
        if o["verbose"]:
            print("Analyzing dataset %d of %d" % (k + 1, len(files)))
        cells_in = load_dataset(f)
        name = cells_in[0]["name"]                           # :158
        oo = dict(o)
        if o["loadPrevious"]:
            pf = o["previousResults"] or _find_previous(file_dir, name)
            if pf is None:
                raise FileNotFoundError("loadPrevious: no previous results for dataset %r in %s" % (name, file_dir))
            oo["_prev"], _ = load_previous_results(pf)
        chain, results, plot = fit_dataset(cells_in, oo, devices)
        os.makedirs(save_loc, exist_ok=True)
        base = "%s-%s" % (matlab_date(), name)
        mat = dict(MCMCresults=_struct_array(RESULT_FIELDS, results), MCMCplot=_struct_array(PLOT_FIELDS, plot),
                   DatasetName=name)
        diags = oo.get("_diagnostics") or []
        if diags:
            mat["MCMCdiagnostics"] = _struct_array(DIAG_FIELDS, diags)
        sio.savemat(os.path.join(save_loc, base + ".mat"), mat)
        if o["saveChains"]:
            save_raw_chains(save_loc, base, chain, thin=int(o["thin"]))
        ret.append(dict(DatasetName=name, MCMCresults=results, MCMCplot=plot, MCMCchain=chain, MCMCdiagnostics=diags))
    print("MCMC analysis complete. Information stored in: %s" % save_loc)
    return ret if o["returnResults"] else None
