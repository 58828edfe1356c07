#!/usr/bin/env python
"""bench.py — headline benchmark of the transcription-cycle MCMC hot path on B200.

Metric (BASELINE.json): MCMC chain-steps/s (and SS-likelihood evaluations/s) on the 299 cells of TestData.mat.
One bench "step" = one complete DRAM fit of the workload (all chains, n_steps MCMC steps each): ONE launch of the
device-resident sampler kernel per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload auto|config2|config3] [--scaling strong|weak] [--n-steps S] [--n-burn B]
                  [--dump-outputs DIR]

  --gpus 1 (default)  BASELINE configs[1] = "config 2": 299 cells x 1 chain, n_burn=10000, n_steps=200000 (dram_kernel: one
                      CTA per chain).  Secondary legs in the same line: config 3 on one GPU (the N > 1 workload, and one fit
                      at n_steps=200000), the raw-chain write-back leg, the batched ssfun kernel, N = 400, CPU baselines.
  --gpus N > 1        BASELINE configs[2] = "config 3": 299 cells x 64 chains = 19 136 chains, PARTITIONED over the ranks by
                      cumulative work (transcriptioncycleinference_b200.distributed.fit_sharded around Cells.mcmc_run: the
                      reference's `parfor (cellNum = 1:N, numParPools)`), summaries all-gathered over NCCL inside the e2e
                      region: strong scaling.  n_burn=10000, n_steps=20000 (the reference's code defaults,
                      src/TranscriptionCycleMCMC.m:38-40).  The one-GPU point of this series is `config3` in the --gpus 1
                      line (or: --gpus 1 --workload config3).  --scaling weak: every rank fits its own replica set instead.

The path has no data-path collective; Philox streams are keyed by chain identity, never by rank or GPU.
`value` = chain-steps of all ranks / max-over-ranks sampler-kernel time (CUDA events on the launching stream, inside
libtcmcmc); `e2e` = the same through the public call with HOST buffers, max-over-ranks host time around it.

--impl reference times the CPU restatement of the reference algorithm (oracle/, a C port: the reference is MATLAB +
un-vendored mcmcstat and cannot run here) on the box's host cores on a bounded sample of the same workload.

--dump-outputs DIR writes what the last timed fit returned to its caller as DIR/<name>.npy (float64): the per-chain
posterior means and standard deviations, the sigma summaries and the decision counters.  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)
GOLDEN = os.path.join(ROOT, "tests", "golden", "cells.npz")
CSRC = [os.path.join(ROOT, "transcriptioncycleinference_b200", "csrc", f) for f in ("tc_mcmc.cu", "tc_device.cuh", "tc_warp.cuh")]
METRIC = "mcmc_chain_steps_per_s"
UNIT = "chain-steps/s"


def w_flop(N):
    """Algorithmic flops of one SS evaluation (SURVEY.md 8d): 9 N(N-1)/2 + 30 N."""
    return 9.0 * N * (N - 1) / 2 + 30.0 * N


def w_op(N):
    """Algorithmic FP64-pipe instructions of one SS evaluation: 11 N(N-1)/2 + 20 N."""
    return 11.0 * N * (N - 1) / 2 + 20.0 * N


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "config2", "config3"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--n-steps", type=int, default=0, help="0: 200000 for config2, 20000 for config3")
    ap.add_argument("--n-burn", type=int, default=10000)
    ap.add_argument("--cpu-sample-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the secondary N = 400 leg")
    ap.add_argument("--no-config3", action="store_true", help="skip the secondary config-3 legs of the one-GPU line")
    ap.add_argument("--no-writeback", action="store_true", help="skip the raw-chain write-back leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed fit to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.workload == "auto":
        a.workload = "config2" if world == 1 else "config3"
    if a.n_steps == 0:
        a.n_steps = 200000 if a.workload == "config2" else 20000
    return a


def source_hash():
    h = hashlib.sha256()
    for f in CSRC:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def measured_traffic(kernel, workload, n_steps, n_burn):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel` on this workload, from the newest ncu capture
    that scripts/profile_gpu.sh committed under profiles/ (traffic_<kernel>_<tag>.json).  A capture made from other kernel
    sources than the ones benched is not quoted: -> (None, why)."""
    best = None
    for f in glob.glob(os.path.join(ROOT, "profiles", "traffic_%s_*.json" % kernel)):
        try:
            d = json.load(open(f))
        except Exception:
            continue
        if d.get("workload") == workload and d.get("n_steps") == n_steps and d.get("n_burn") == n_burn:
            if best is None or d.get("when", "") > best.get("when", ""):
                best = dict(d, file=os.path.relpath(f, ROOT))
    if best is None:
        return None, "no ncu capture of %s for %s (n_steps %d) under profiles/" % (kernel, workload, n_steps)
    if best.get("source_hash") != source_hash():
        return None, "%s was captured from other kernel sources (%s) than the ones benched (%s)" % (best["file"], best.get("source_hash"), source_hash())
    return best, None


# ------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(self.rows))


# ------------------------------------------------------------------------------- CPU baseline
def host_cores():
    """all the host cores this process may use (torchrun exports OMP_NUM_THREADS=1: ask the OS, not OpenMP)"""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class _HostCells:                             # the bits of engine.Cells that setup_cell.chain_inputs needs
    def __init__(self, g):
        self.g = g
        self.ld = 7 + int(g["N"].max())

    def cell(self, c):
        o = int(self.g["off"][c]); n = int(self.g["N"][c])
        return self.g["t"][o:o + n], self.g["ms2"][o:o + n], self.g["pp7"][o:o + n]


def cpu_baseline(g, target_seconds, with_config1=False):
    """Oracle (C port of the reference algorithm: literal m x n forward model + DRAM) on the host cores, OpenMP over chains
    (the parfor analogue).  Bounded sample: all 299 cells, one chain each, a reduced number of MCMC steps chosen to cost
    ~target_seconds on all cores.  with_config1: also BASELINE configs[0] in full (cell 1, n_burn 10000, n_steps 20000,
    ONE thread) and the one-thread rate of the 299-cell slice (SURVEY.md 8d)."""
    from oracle import c_oracle, forward_literal
    from transcriptioncycleinference_b200 import setup_cell

    cons = c_oracle.Construct.from_dict(forward_literal.CONSTRUCTS["P2P-MS2v5-LacZ-PP7v4"])
    cores = host_cores()
    cc = np.arange(299, dtype=np.int32)
    inputs = setup_cell.chain_inputs(_HostCells(g), cc, np.random.default_rng(1))
    opts = c_oracle.default_opts(40, 20)                                 # calibrate: 40 steps
    t0 = time.time()
    c_oracle.run_chains(cons, g, opts, 20, cc, *inputs, seed=1, nthreads=cores)
    per_step = (time.time() - t0) / (299 * 40)
    nsimu = int(max(100, min(20000, target_seconds / (per_step * 299))))
    nsimu = (nsimu // 100) * 100
    burn = nsimu // 2
    opts = c_oracle.default_opts(nsimu, burn)
    t0 = time.time()
    _, _, _, cnt = c_oracle.run_chains(cons, g, opts, burn, cc, *inputs, seed=2, nthreads=cores)
    dt = time.time() - t0
    out = dict(value=299 * nsimu / dt, unit=UNIT, cores=cores, kind="port",
               sample="299 cells x 1 chain x %d MCMC steps (burnintime %d), literal m x n forward model, "
                      "C port of the reference algorithm (oracle/tc_oracle.c), OpenMP over chains, %d threads" % (nsimu, burn, cores),
               seconds=dt, ss_evals_per_s=float(cnt[:, 0].sum()) / dt)
    if with_config1:
        o1 = c_oracle.default_opts(20000, 10000)
        one = [x[:1] for x in inputs]
        t0 = time.time()
        _, _, _, c1 = c_oracle.run_chains(cons, g, o1, 10000, cc[:1], *one, seed=3, nthreads=1)
        d1 = time.time() - t0
        out["config1"] = dict(value=20000 / d1, unit=UNIT, cores=1, seconds=d1, ss_evals_per_s=float(c1[:, 0].sum()) / d1,
                              sample="BASELINE configs[0] in full: TestData cell 1 (N = %d), n_burn 10000, n_steps 20000, one chain, one thread" % int(g["N"][0]))
        ns1 = max(100, (int(nsimu / max(cores, 1) * 1.5) // 100) * 100)
        o2 = c_oracle.default_opts(ns1, ns1 // 2)
        sub = np.arange(0, 299, 13, dtype=np.int32)                      # 23 cells spread over the six movies
        t0 = time.time()
        c_oracle.run_chains(cons, g, o2, ns1 // 2, sub, *[x[sub] for x in inputs], seed=4, nthreads=1)
        d2 = time.time() - t0
        out["one_thread"] = dict(value=sub.size * ns1 / d2, unit=UNIT, cores=1, seconds=d2,
                                 sample="%d of the 299 cells x %d MCMC steps (burnintime %d), one thread" % (sub.size, ns1, ns1 // 2))
    return out


def run_reference(args, g):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    last = None
    for i in range(args.warmup + args.steps):
        last = cpu_baseline(g, max(2.0, args.cpu_sample_seconds / 3))
        if i >= args.warmup:
            vals.append(last)
    v = float(np.mean([x["value"] for x in vals]))
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=float(np.mean([x["seconds"] for x in vals]) * 1e3), higher_is_better=True,
                scaling="strong" if (args.gpus > 1 and args.scaling == "strong") else "weak", vs_baseline=None, dtype="f64",
                data="TestData.mat cells (tests/golden/cells.npz), synthetic x0",
                impl="reference",
                config=dict(workload=args.workload + " (bounded sample: one chain per cell, reduced n_steps; chain-steps/s does not depend on the chain count on a CPU)",
                            cells=299, chains_per_cell=1),
                cpu_baseline=dict(value=v, unit=UNIT, cores=last["cores"], kind=last["kind"], sample=last["sample"]),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                ss_evals_per_s=float(np.mean([x["ss_evals_per_s"] for x in vals])), gpu_launches=0)
    return line


# ----------------------------------------------------------------------------------- GPU arm
def algorithmic_flops(g, cc, cnt, n_steps, n_burn, _lib):
    """SURVEY.md 8(d): SS evaluations x W_flop(N) + full-R proposal mat-vecs after burn-in (2 proposals: 2 npar^2/2 FMA) +
    covariance block updates (npar^2/2 FMA per row) + Cholesky (npar^3/6 FMA) per adaptation."""
    Ns = g["N"][cc].astype(np.float64)
    npar = Ns + 7
    ss_evals = cnt[:, _lib.CNT_SS_EVALS].astype(np.float64)
    post = max(0, n_steps - n_burn)
    flops_ss = float(np.sum(ss_evals * w_flop(Ns)))
    flops_dram = float(np.sum(2.0 * post * npar ** 2 * 2 / 2 + n_steps * npar ** 2 + cnt[:, _lib.CNT_ADAPTATIONS] * npar ** 3 / 3))
    ops_ss = float(np.sum(ss_evals * w_op(Ns)))
    return flops_ss, flops_dram, ops_ss


def run_ours(args, g):
    import torch
    import torch.distributed as dist
    from transcriptioncycleinference_b200 import _lib, distributed, setup_cell
    from transcriptioncycleinference_b200.engine import Cells

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (libtcmcmc has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cells = Cells.from_packed(g["N"], g["off"], g["t"], g["ms2"], g["pp7"], devices=(local,))
    ld = cells.ld
    per_cell = 1 if args.workload == "config2" else 64
    strong = world > 1 and args.scaling == "strong"
    cc = np.repeat(np.arange(299, dtype=np.int32), per_cell)
    # chain identity = (cell, chain replica); weak scaling: rank r owns replicas [r per_cell, (r+1) per_cell)
    rep = np.tile(np.arange(per_cell, dtype=np.uint64), 299) + np.uint64(0 if strong else rank * per_cell)
    uid = cc.astype(np.uint64) * np.uint64(1 << 20) + rep
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(1000 + (0 if strong else rank)))
    opts = _lib.default_opts(nsimu=args.n_steps, burnintime=args.n_burn, n_burn=args.n_burn, store_chain=0,
                             seed=20201028, ngpus=1)
    opts.devices[0] = local
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2
    peak_dfma, peak_clk = _lib.measure_fp64_peak(local)
    schema = distributed.summary_schema(ld, _lib.NCOUNTERS)

    def run_local(c, arrs, u):
        return cells.mcmc_run(opts, c, *arrs, chain_uid=u)               # host buffers in, summaries out

    def one_fit():
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if strong:
            out = distributed.fit_sharded(run_local, cc, g["N"], list(inputs), uid, rank, world, schema=schema)
            ks = out["local"].get("kernel_seconds", 0.0)
        else:
            out = run_local(cc, inputs, uid)
            ks = out["kernel_seconds"]
        return time.perf_counter() - t0, ks, out

    for _ in range(args.warmup):
        one_fit()
    barrier()
    kernel_s, e2e_s, out = [], [], None
    sampler = ClockSampler(local)
    with sampler:
        for _ in range(args.steps):
            dt, ks, out = one_fit()
            e2e_s.append(dt); kernel_s.append(ks)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs, _lib)
    tk, te = float(np.sum(kernel_s)), float(np.sum(e2e_s))
    if world > 1:
        tt = torch.tensor([tk, te], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        tk, te = float(tt[0]), float(tt[1])
    cnt = out["counters"]                                               # strong: gathered (all chains); else this rank's
    chains_total = cc.size if strong else world * cc.size
    nsteps_total = chains_total * args.n_steps * args.steps
    flops_ss, flops_dram, ops_ss = algorithmic_flops(g, cc, cnt, args.n_steps, args.n_burn, _lib)
    if not strong:
        flops_ss, flops_dram, ops_ss = world * flops_ss, world * flops_dram, world * ops_ss
    ss_evals = cnt[:, _lib.CNT_SS_EVALS].astype(np.float64)
    t_fit = tk / args.steps
    achieved = (flops_ss + flops_dram) / t_fit / 1e12
    peak_tf = 2 * peak_dfma / 1e12 * world
    if strong:
        parts = out["partition"]
        n_loc = [b - a for a, b in parts]
        h2d = int(sum(x.nbytes for x in inputs) / cc.size * max(n_loc) + max(n_loc) * 12)
        d2h = int(max(n_loc) * ((2 * ld + 2) * 8 + _lib.NCOUNTERS * 8))
        gather = int(cc.size * ((2 * ld + 2) * 8 + _lib.NCOUNTERS * 8))
    else:
        h2d = sum(x.nbytes for x in inputs) + cc.nbytes + uid.nbytes
        d2h = cc.size * (2 * ld + 2) * 8 + cc.size * _lib.NCOUNTERS * 8
        gather = 0
    chains_per_gpu = int(np.ceil(cc.size / world)) if strong else int(cc.size)
    sms = _lib.device_info(local)["sm_count"]
    kernel = "dram_warp_kernel" if chains_per_gpu >= 6 * sms else "dram_kernel"
    traffic, why = measured_traffic(kernel, args.workload, args.n_steps, args.n_burn) if world == 1 else (None, "captured on one GPU only")
    line = dict(
        metric=METRIC, value=nsteps_total / tk, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=tk / args.steps * 1e3, higher_is_better=True, scaling="strong" if strong else "weak", vs_baseline=None,
        dtype="f64",
        data="TestData.mat cells (tests/golden/cells.npz: the reference's 299-cell dataset), synthetic x0",
        config=dict(workload="%s: 299 cells x %d chain(s)/cell = %d chains %s, n_burn=%d, n_steps=%d, adaptint=100, DRAM, "
                             "construct P2P-MS2v5-LacZ-PP7v4" % (args.workload, per_cell, cc.size,
                                                                 "partitioned over %d GPU(s)" % world if strong else "per GPU",
                                                                 args.n_burn, args.n_steps),
                    chains_per_gpu=chains_per_gpu, kernel=kernel, l2="flushed between timed fits (256 MiB write)",
                    sharding=("chains partitioned over the ranks by cumulative N^2 + npar^2 (distributed.fit_sharded around "
                              "Cells.mcmc_run); no collective in the data path; summaries + counters all-gathered over NCCL "
                              "(%d bytes per fit) inside the e2e region" % gather) if strong else
                             "chains replicated per rank, no collective in the data path",
                    one_gpu_point="python bench.py --gpus 1: key config3.value (same workload, one GPU)" if strong else None),
        e2e=dict(value=nsteps_total / te, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                 gather_bytes_per_step=gather),
        gpu_launches=args.steps * world,
        ss_evals_per_s=float((1 if strong else world) * ss_evals.sum() * args.steps / tk),
        ss_evals_per_chain_step=float(ss_evals.sum() / (cc.size * args.n_steps)),
        accept_rate=float((cnt[:, _lib.CNT_ACC_STAGE1] + cnt[:, _lib.CNT_ACC_STAGE2]).sum() / (cc.size * args.n_steps)),
        roofline=dict(bound="fp64_pipe", kernel=kernel, achieved=achieved, peak=peak_tf, unit="TFLOP/s",
                      frac=achieved / peak_tf,
                      traffic=(traffic["bytes_read"] + traffic["bytes_write"]) if traffic else None,
                      traffic_source=(dict(file=traffic["file"], bytes_read=traffic["bytes_read"], bytes_write=traffic["bytes_write"],
                                           when=traffic.get("when"), source_hash=traffic.get("source_hash"))
                                      if traffic else why),
                      traffic_unit="bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum); the kernel is bound by "
                                   "FP64-pipe latency, not HBM",
                      peak_source="measured DFMA micro-benchmark on this GPU (tc_measure_fp64_peak) x %d GPU(s), SM clock %.0f MHz; "
                                  "MEASURED_PEAKS.json has no FP64 entry" % (world, peak_clk),
                      algorithmic_flops_per_launch=(flops_ss + flops_dram) / world, flops_ss=flops_ss, flops_dram=flops_dram,
                      frac_ops_ss_only=ops_ss / t_fit / (peak_dfma * world)),
        clocks=sampler.summary(),
    )
    if rank == 0 and world == 1:
        # secondary legs of the one-GPU line (each guarded: a secondary leg must not cost the headline)
        def leg(name, fn):
            try:
                line[name] = fn()
            except Exception as e:
                line[name] = dict(error=repr(e))
        leg("ss_kernel", lambda: ss_kernel_leg(cells, g, peak_dfma, torch))
        if args.workload == "config2" and not args.no_config3:
            leg("config3", lambda: config3_leg(cells, g, local, peak_dfma, flush, torch, 20000, args.n_burn, fits=2))
            leg("config3_n200000", lambda: config3_leg(cells, g, local, peak_dfma, flush, torch, 200000, args.n_burn, fits=1))
        if not args.no_writeback:
            leg("chain_writeback", lambda: writeback_leg(cells, g, local, flush, torch))
        if not args.no_config5:
            leg("config5_scale", lambda: config5_leg(local))
        if not args.no_cpu_baseline:
            leg("cpu_baseline", lambda: cpu_baseline(g, args.cpu_sample_seconds, with_config1=True))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line if rank == 0 else None


def dump_outputs(out, d, _lib):
    """The summaries Cells.mcmc_run returned for every chain of the fit (gathered over the ranks under strong scaling; rank
    0's own chains under weak scaling), as float64.  Counters past CNT_STATUS are SM cycle readings, not results, and are
    left out; the others are exact in float64.  The largest workload, config3, comes to about 42 MB."""
    os.makedirs(d, exist_ok=True)
    arrs = dict(mean=out["mean"], std=out["std"], sig=out["sig"], counters=out["counters"][:, :_lib.CNT_STATUS + 1])
    for name, a in arrs.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def config3_leg(cells, g, device, peak_dfma, flush, torch, n_steps, n_burn, fits):
    """BASELINE config 3 on ONE GPU: 299 cells x 64 chains = 19 136 chains (dram_warp_kernel: one warp per chain) — the
    one-GPU point of the partitioned --gpus N series (n_steps 20 000), and one fit at n_steps 200 000."""
    from transcriptioncycleinference_b200 import _lib, setup_cell
    cc = np.repeat(np.arange(299, dtype=np.int32), 64)
    uid = cc.astype(np.uint64) * np.uint64(1 << 20) + np.tile(np.arange(64, dtype=np.uint64), 299)
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(1000))
    opts = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn, store_chain=0, seed=20201028, ngpus=1)
    opts.devices[0] = device
    warm = _lib.default_opts(nsimu=min(n_steps, 2000), burnintime=1000, n_burn=1000, store_chain=0, seed=1, ngpus=1)
    warm.devices[0] = device
    cells.mcmc_run(warm, cc, *inputs, chain_uid=uid)                     # pools, code, clocks
    ks, es, out = [], [], None
    for _ in range(fits):
        flush.zero_(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = cells.mcmc_run(opts, cc, *inputs, chain_uid=uid)
        es.append(time.perf_counter() - t0); ks.append(out["kernel_seconds"])
    t, te = float(np.mean(ks)), float(np.mean(es))
    flops_ss, flops_dram, ops_ss = algorithmic_flops(g, cc, out["counters"], n_steps, n_burn, _lib)
    return dict(workload="config3: 299 cells x 64 chains = 19136 chains on one GPU, n_burn=%d, n_steps=%d" % (n_burn, n_steps),
                kernel="dram_warp_kernel", value=cc.size * n_steps / t, unit=UNIT, e2e_value=cc.size * n_steps / te, ms_per_fit=t * 1e3, fits=fits,
                ss_evals_per_s=float(out["counters"][:, _lib.CNT_SS_EVALS].sum()) / t,
                roofline_frac=(flops_ss + flops_dram) / t / (2 * peak_dfma), frac_ops_ss_only=ops_ss / t / peak_dfma)


def writeback_leg(cells, g, device, flush, torch, n_steps=20000, n_burn=10000):
    """The reference's default product is the raw chain (src/TranscriptionCycleMCMC.m:276-283,315-323,377-378): config 2 at the
    reference's code defaults (n_burn 10000, n_steps 20000) with store_chain = 1 — 299 x 10 001 rows x ld doubles + s2chain —
    against the same fit with summaries only.  Destinations are page-locked host buffers allocated once (tc_host_alloc)."""
    from transcriptioncycleinference_b200 import _lib, setup_cell
    cc = np.arange(299, dtype=np.int32)
    uid = cc.astype(np.uint64) * np.uint64(1 << 20)
    inputs = setup_cell.chain_inputs(cells, cc, np.random.default_rng(1000))
    ld = cells.ld
    res = {}
    nstore = n_steps - n_burn + 1
    chain = _lib.pinned_empty((cc.size, nstore, ld)); s2 = _lib.pinned_empty((cc.size, n_steps))
    for store in (0, 1):
        opts = _lib.default_opts(nsimu=n_steps, burnintime=n_burn, n_burn=n_burn, store_chain=store, seed=20201028, ngpus=1)
        opts.devices[0] = device
        ks, es, ds = [], [], []
        for it in range(4):
            flush.zero_(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = cells.mcmc_run(opts, cc, *inputs, chain_uid=uid, chain_out=chain if store else None, s2chain_out=s2 if store else None)
            if it >= 1:
                es.append(time.perf_counter() - t0); ks.append(out["kernel_seconds"]); ds.append(out["drain_seconds"])
        res[store] = (float(np.mean(ks)), float(np.mean(es)), float(np.mean(ds)))
    nbytes = chain.nbytes + s2.nbytes
    rows_bytes = float(np.sum((g["N"][cc] + 7 + 1) * 8.0) * nstore)     # algorithmic: (npar + 1) doubles per stored row
    (k0, e0, d0), (k1, e1, d1) = res[0], res[1]
    return dict(workload="config2, n_burn=%d, n_steps=%d, store_chain=1: %d rows x %d chains" % (n_burn, n_steps, nstore, cc.size),
                chain_bytes=int(nbytes), kernel_ms_summaries_only=k0 * 1e3, kernel_ms_with_chains=k1 * 1e3, kernel_slowdown=k1 / k0,
                hbm_row_write_gbs=rows_bytes / k1 / 1e9,
                hbm_note="algorithmic bytes of the stored rows / kernel time; ncu's dram__bytes_write.sum.per_second for this launch is in profiles/ (writeback capture)",
                d2h_seconds=d1, d2h_gbs=nbytes / d1 / 1e9, e2e_ms_summaries_only=e0 * 1e3, e2e_ms_with_chains=e1 * 1e3,
                e2e_slowdown=e1 / e0, chain_steps_per_s_e2e_with_chains=cc.size * n_steps / e1)


def config5_leg(device, ncells=1184, N=400, nsteps=2000):
    """Secondary: BASELINE config 5's series length (N = 400, npar = 407: the big layout of the sampler) at a single-GPU
    scale — synthetic cells from the forward model (transcriptioncycleinference_b200/synthetic.py), 8 chains per SM."""
    from transcriptioncycleinference_b200 import _lib, setup_cell, synthetic
    cells5, _ = synthetic.make_cells(ncells, N, devices=(device,))
    cc = np.arange(ncells, dtype=np.int32)
    inputs = setup_cell.chain_inputs(cells5, cc, np.random.default_rng(5))
    opts = _lib.default_opts(nsimu=nsteps, burnintime=nsteps // 2, n_burn=nsteps // 2, ngpus=1)
    opts.devices[0] = device
    ks = []
    for _ in range(3):
        ks.append(cells5.mcmc_run(opts, cc, *inputs)["kernel_seconds"])
    cells5.close()
    t = float(np.mean(ks[1:]))
    return dict(workload="%d synthetic cells x N=%d (npar=%d), 1 chain each, n_steps=%d, n_burn=%d" % (ncells, N, N + 7, nsteps, nsteps // 2),
                chain_steps_per_s=ncells * nsteps / t, ms=t * 1e3)


def ss_kernel_leg(cells, g, peak_dfma, torch):
    from transcriptioncycleinference_b200 import _lib
    rng = np.random.default_rng(0)
    per = 1024
    cid = np.repeat(np.arange(299, dtype=np.int32), per)
    th = np.zeros((cid.size, cells.ld))
    for c in range(299):
        N = int(g["N"][c]); m = slice(c * per, (c + 1) * per)
        lo = np.concatenate([[0.5, 0, 0, 0, 0, 0, 5], -8 * np.ones(N)])
        hi = np.concatenate([[4, 6, 6, 3, 3, 1, 25], 8 * np.ones(N)])
        th[m, :7 + N] = lo + (hi - lo) * rng.random((per, 7 + N))
    d_th = torch.from_numpy(th).cuda(); d_cid = torch.from_numpy(cid).cuda()
    d_out = torch.zeros(cid.size, dtype=torch.float64, device="cuda")
    res = {}
    for name, algo in (("toeplitz", _lib.ALGO_TOEPLITZ), ("pairs", _lib.ALGO_PAIRS)):
        ms = []
        for it in range(8):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            cells.ss_batch_device(cid.size, d_cid.data_ptr(), d_th.data_ptr(), cells.ld, d_out.data_ptr(), algo=algo)
            e1.record(); torch.cuda.synchronize()
            if it >= 3:
                ms.append(e0.elapsed_time(e1))
        t = float(np.mean(ms)) * 1e-3
        ops = float(np.sum(w_op(g["N"][cid].astype(np.float64))))
        res[name] = dict(evals_per_s=cid.size / t, ms=t * 1e3, batch=int(cid.size),
                         frac_of_fp64_peak_algorithmic_ops=ops / t / peak_dfma)
    res["note"] = ("device-resident inputs, %.0f MB of theta streamed from HBM per launch (> 126 MB L2); toeplitz = the O(N) "
                   "algorithm (ss_stream_kernel: operands staged in shared memory), pairs = the O(N^2) algorithm W_op counts "
                   "(ss_batch_kernel); frac = evals/s x W_op(N) / measured DFMA rate" % (th.nbytes / 1e6))
    return res


def main():
    args = parse()
    # ONE JSON line on stdout: whatever a library prints to file descriptor 1 while the bench runs (NCCL's version banner and
    # NCCL_DEBUG lines, torchrun notices) goes to stderr, where the driver can still read it
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    g = dict(np.load(GOLDEN))
    line = run_reference(args, g) if args.impl == "reference" else run_ours(args, g)
    sys.stdout.flush()
    if line is not None:
        os.write(out_fd, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    main()
