#!/usr/bin/env python
"""Generate the committed golden fixtures from the reference's own .mat files.

  python tests/golden/make_golden.py <checkout of the reference project>

The tests, smoke() and bench.py only ever read the .npz files this script writes
next to itself, so they need no copy of the reference.

Sources (all MAT v5, read with scipy.io.loadmat), relative to the reference checkout:
  TestScripts/TestData.mat                      -> cells.npz
  TestScripts/28-Oct-2020-TestData.mat          -> results.npz, results.1.npz
  TestScripts/28-Oct-2020-TestData_RawChain.mat -> chains.npz, chains.1.npz

A fixture larger than 1 MB is stored in parts, <stem>.npz, <stem>.1.npz, ...;
tests/conftest.py:load_golden merges them back, concatenating an array that is
split over several parts along its first axis.

Layout of the packed ("ragged") arrays: cell c owns [off[c], off[c]+N[c]) of
every per-timepoint array, off = exclusive cumulative sum of N.

  cells.npz    N[299] int32, off[300] int64, t/ms2/pp7 [sum N] f64 (NaN = missing),
               name (str)                                  (README.md:11-16)
  results.npz  the 18 scalar MCMCresults fields as [299] f64 arrays (field order of
               TranscriptionCycleMCMC.m:151-155), mean_dR/sigma_dR packed [sum N],
               cell_index, ApprovedFits [299]; MCMCplot fields t_plot, MS2_plot,
               PP7_plot, simMS2, simPP7 packed [sum N]; DatasetName
  chains.npz   theta[299,10,7+Nmax] f64 in the sampler's own parameter order
               [v,tau,ton,MS2_basal,PP7_basal,A,R,dR_1..dR_N] (NaN padded beyond
               7+N[c]), s2chain[299,10]   (the shipped fixtures are a 10-step run,
               SURVEY.md section 0.1 #15)
"""
import os
import sys

import numpy as np
import scipy.io as sio

HERE = os.path.dirname(os.path.abspath(__file__))
RESULTS_PART1 = ("MS2_plot", "PP7_plot", "simMS2", "simPP7")     # stored in results.1.npz
CHAINS_SPLIT = 150                                                # theta of cells [0, 150) in chains.npz, the rest in chains.1.npz

SCALAR_FIELDS = [
    "mean_v", "sigma_v", "mean_ton", "sigma_ton", "mean_A", "sigma_A", "mean_tau",
    "sigma_tau", "mean_MS2_basal", "sigma_MS2_basal", "mean_PP7_basal",
    "sigma_PP7_basal", "mean_R", "sigma_R", "mean_sigma", "sigma_sigma",
    "cell_index", "ApprovedFits",
]


def save_results(out):
    """results.npz + results.1.npz: the same arrays as one file would hold, each file under 1 MB."""
    np.savez_compressed(os.path.join(HERE, "results.npz"), **{k: v for k, v in out.items() if k not in RESULTS_PART1})
    np.savez_compressed(os.path.join(HERE, "results.1.npz"), **{k: out[k] for k in RESULTS_PART1})


def save_chains(out):
    """chains.npz + chains.1.npz: theta split by cell, each file under 1 MB."""
    first = dict(out, theta=out["theta"][:CHAINS_SPLIT])
    np.savez_compressed(os.path.join(HERE, "chains.npz"), **first)
    np.savez_compressed(os.path.join(HERE, "chains.1.npz"), theta=out["theta"][CHAINS_SPLIT:])


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "TestScripts")):
        sys.exit("usage: make_golden.py <checkout of the reference project (with TestScripts/)>")
    ref = os.path.join(sys.argv[1], "TestScripts")

    d = sio.loadmat(os.path.join(ref, "TestData.mat"), mat_dtype=True)["data"]
    nc = d.shape[1]
    N = np.array([d[0, c]["time"].shape[1] for c in range(nc)], dtype=np.int32)
    off = np.zeros(nc + 1, dtype=np.int64)
    off[1:] = np.cumsum(N)
    t = np.concatenate([d[0, c]["time"][0] for c in range(nc)])
    ms2 = np.concatenate([d[0, c]["MS2"][0] for c in range(nc)])
    pp7 = np.concatenate([d[0, c]["PP7"][0] for c in range(nc)])
    name = str(d[0, 0]["name"][0])
    np.savez_compressed(os.path.join(HERE, "cells.npz"), N=N, off=off, t=t, ms2=ms2,
                        pp7=pp7, name=name)

    r = sio.loadmat(os.path.join(ref, "28-Oct-2020-TestData.mat"), mat_dtype=True)
    res, plot = r["MCMCresults"], r["MCMCplot"]
    out = {}
    for f in SCALAR_FIELDS:
        out[f] = np.array([float(res[0, c][f].squeeze()) for c in range(nc)])
    for f in ("mean_dR", "sigma_dR"):
        out[f] = np.concatenate([res[0, c][f].reshape(-1) for c in range(nc)])
    for f in ("t_plot", "MS2_plot", "PP7_plot", "simMS2", "simPP7"):
        out[f] = np.concatenate([plot[0, c][f].reshape(-1) for c in range(nc)])
    out["DatasetName"] = str(r["DatasetName"][0])
    out["field_order"] = np.array(res.dtype.names)
    out["plot_field_order"] = np.array(plot.dtype.names)
    save_results(dict(N=N, off=off, **out))

    ch = sio.loadmat(os.path.join(ref, "28-Oct-2020-TestData_RawChain.mat"),
                     mat_dtype=True)["MCMCchain"]
    nrow = ch[0, 0]["v_chain"].shape[0]
    npmax = 7 + int(N.max())
    theta = np.full((nc, nrow, npmax), np.nan)
    s2 = np.zeros((nc, nrow))
    order = ["v_chain", "tau_chain", "ton_chain", "MS2_basal_chain", "PP7_basal_chain",
             "A_chain", "R_chain"]
    for c in range(nc):
        for k, f in enumerate(order):
            theta[c, :, k] = ch[0, c][f][:, 0]
        theta[c, :, 7:7 + N[c]] = ch[0, c]["dR_chain"]
        s2[c] = ch[0, c]["s2chain"][:, 0]
    save_chains(dict(N=N, theta=theta, s2chain=s2, chain_field_order=np.array(ch.dtype.names)))
    for f in ("cells.npz", "results.npz", "results.1.npz", "chains.npz", "chains.1.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")


if __name__ == "__main__":
    main()
