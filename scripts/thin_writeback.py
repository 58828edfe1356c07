"""Raw chains thinned on the device (tc_mcmc_opts.thin): what storing every k-th row costs at the benchmark's sizes.

    python scripts/thin_writeback.py [--out profiles/thin_writeback.json] [--parent DIR] [--rounds 3]

Prints one JSON line (also written to --out) with the card's name and power limit, read in the same run:
  (a) config 2 as benched (299 cells x 1 chain, n_burn 10 000, n_steps 200 000): store_chain = 0, then thin = 20 and 100;
  (b) config 3 on one GPU (299 cells x 64 chains, n_steps 20 000): store_chain = 0, then thin = 50;
  for each, the sampler kernel time and the drain time (tc_last_kernel_seconds / tc_last_drain_seconds, mean over the timed
  fits after one warm-up fit), the bytes stored, and the algorithmic bytes of the stored rows ((npar + 1) doubles a row)
  over kernel time;
  (c) with --parent DIR (a built checkout of another commit): bench.py's write-back leg size (config 2, n_steps 20 000,
  store_chain = 0 and 1 at thin = 1) run by that tree and by this one in turn, --rounds times each, in separate processes,
  so that a kernel-time difference can be read against the spread of repeated runs.
The inputs are bench.py's (seeded chain_inputs, uid = cell << 20 + replica, seed 20201028)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def workload(root, per_cell):
    sys.path.insert(0, root)
    from transcriptioncycleinference_b200 import setup_cell
    from transcriptioncycleinference_b200.engine import Cells
    g = dict(np.load(os.path.join(root, "tests", "golden", "cells.npz")))
    cells = Cells.from_packed(g["N"], g["off"], g["t"], g["ms2"], g["pp7"])
    cc = np.repeat(np.arange(299, dtype=np.int32), per_cell)
    uid = cc.astype(np.uint64) * np.uint64(1 << 20) + np.tile(np.arange(per_cell, dtype=np.uint64), 299)
    return g, cells, cc, uid, setup_cell.chain_inputs(cells, cc, np.random.default_rng(1000))


def timed(cells, cc, uid, inputs, opts, fits, **kw):
    """One warm-up fit, then `fits` timed ones: mean and spread of kernel and drain seconds."""
    ks, ds = [], []
    for it in range(fits + 1):
        out = cells.mcmc_run(opts, cc, *inputs, chain_uid=uid, **kw)
        if it:
            ks.append(out["kernel_seconds"]); ds.append(out["drain_seconds"])
    return dict(kernel_s=float(np.mean(ks)), kernel_s_min=float(np.min(ks)), kernel_s_max=float(np.max(ks)),
                drain_s=float(np.mean(ds)), fits=fits), out


def thinned_leg(name, per_cell, n_steps, n_burn, thins, fits):
    from transcriptioncycleinference_b200 import _lib
    g, cells, cc, uid, inputs = workload(ROOT, per_cell)
    npar = g["N"][cc].astype(np.float64) + 7
    res = dict(workload="%s: %d chains, n_burn=%d, n_steps=%d" % (name, cc.size, n_burn, n_steps))
    base = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn, store_chain=0, seed=20201028, ngpus=1)
    res["summaries_only"], _ = timed(cells, cc, uid, inputs, base, fits)
    for k in thins:
        opts = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn, store_chain=1, seed=20201028, ngpus=1, thin=k)
        nkeep, ns2 = _lib.stored_rows(opts)
        chain = _lib.pinned_empty((cc.size, nkeep, cells.ld)); s2 = _lib.pinned_empty((cc.size, ns2))
        r, _ = timed(cells, cc, uid, inputs, opts, fits, chain_out=chain, s2chain_out=s2)
        rows_bytes = float(np.sum(npar + 1) * 8.0 * nkeep)
        r.update(rows_kept=nkeep, stored_bytes=int(chain.nbytes + s2.nbytes),
                 row_bytes_per_kernel_s_gbs=rows_bytes / r["kernel_s"] / 1e9,
                 kernel_vs_summaries_only=r["kernel_s"] / res["summaries_only"]["kernel_s"],
                 d2h_gbs=(chain.nbytes + s2.nbytes) / r["drain_s"] / 1e9)
        res["thin_%d" % k] = r
        del chain, s2
    cells.close()
    return res


def writeback_worker(root, fits):
    """bench.py's write-back leg size at thin = 1 with the tree at root: store_chain = 0 and 1."""
    sys.path.insert(0, root)
    from transcriptioncycleinference_b200 import _lib
    _, cells, cc, uid, inputs = workload(root, 1)
    n_steps, n_burn = 20000, 10000
    chain = _lib.pinned_empty((cc.size, n_steps - n_burn + 1, cells.ld)); s2 = _lib.pinned_empty((cc.size, n_steps))
    out = {}
    for store in (0, 1):
        opts = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn, store_chain=store, seed=20201028, ngpus=1)
        kw = dict(chain_out=chain, s2chain_out=s2) if store else {}
        out["store_chain_%d" % store], last = timed(cells, cc, uid, inputs, opts, fits, **kw)
        out["store_chain_%d" % store]["mean_checksum"] = float(np.sum(last["mean"]))
    print(json.dumps(out))


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "thin_writeback.json"))
    ap.add_argument("--parent", help="a built checkout of another commit, for the thin = 1 write-back comparison")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--fits", type=int, default=3)
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return writeback_worker(a.worker, a.fits)
    sys.path.insert(0, ROOT)
    from transcriptioncycleinference_b200 import _lib
    if _lib.device_count() < 1:
        raise SystemExit("thin_writeback.py: no CUDA device (libtcmcmc has no CPU fallback)")
    t0 = time.time()
    line = dict(script="scripts/thin_writeback.py", device=_lib.device_info(0)["name"], nvidia_smi=device_line())
    line["a_config2_as_benched"] = thinned_leg("config2", 1, 200000, 10000, (20, 100), a.fits)
    line["b_config3_one_gpu"] = thinned_leg("config3", 64, 20000, 10000, (50,), max(1, a.fits - 1))
    if a.parent:
        runs = {"parent": [], "this": []}
        for _ in range(a.rounds):
            for tag, root in (("parent", os.path.abspath(a.parent)), ("this", ROOT)):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", root, "--fits", str(a.fits)],
                                   capture_output=True, text=True, cwd=root)
                if p.returncode:
                    raise SystemExit("worker %s failed:\n%s" % (tag, p.stderr))
                runs[tag].append(json.loads(p.stdout.strip().splitlines()[-1]))
        line["c_writeback_thin1_parent_vs_this"] = runs
    line["nvidia_smi_after"] = device_line()
    line["wall_s"] = time.time() - t0
    s = json.dumps(line)
    print(s)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
