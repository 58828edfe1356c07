/*
 * tcmcmc.h — C ABI of libtcmcmc.so, the B200-native (sm_100a) engine for the per-cell DRAM fit of
 * the Liu et al. (2020) transcription-cycle model.
 *
 * This is the drop-in boundary for the ONE hot path of GarciaLab/TranscriptionCycleInference:
 *   TranscriptionCycleMCMC -> parfor over cells -> mcmcrun (DRAM) -> ssfun ->
 *   SumofSquaresFunction_TranscriptionCycleMCMC -> ConstantElongationSim -> GetFluorFromPolPos.
 * The reference is MATLAB; its FFI for this path would be a MEX gateway (matlab/tcmcmc_mex.cu) that
 * only marshals mxArrays into the plain buffers below.  The same symbols are bound from Python with
 * ctypes (transcriptioncycleinference_b200/_lib.py).  Citations are file:line in the reference
 * (paths relative to /root/reference).
 *
 * Conventions: extern "C"; every function returns 0 on success or a negative TC_E* code, with a
 * thread-local message in tc_last_error(); no exceptions cross the ABI; the caller owns every
 * buffer it passes; arrays are dense FP64, row-major, unless stated.  Functions whose name ends in
 * `_device` take DEVICE pointers (already resident in HBM) and a CUDA stream; all others take HOST
 * pointers and include the host<->device copies.  There is no CPU fallback: without a CUDA device
 * every compute entry point fails with TC_ENODEV.
 *
 * Parameter vector layout (everywhere): theta = [v, tau, ton, MS2_basal, PP7_basal, A, R,
 * dR_1..dR_N], npar = 7+N  (src/TranscriptionCycleMCMC.m:210,242-255;
 * src/SumofSquaresFunction_TranscriptionCycleMCMC.m:35-42).  Per-chain / per-evaluation vectors are
 * padded to a common leading dimension ld >= 7+max(N).
 */
#ifndef TCMCMC_H
#define TCMCMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TC_VERSION 100          /* 0.1.0 */
#define TC_MAX_SETS 8           /* stem-loop sets per colour in one construct */
#define TC_MAX_GPUS 8

enum {
    TC_OK = 0,
    TC_EINVAL = -1,    /* bad argument (message says which) */
    TC_ENODEV = -2,    /* no CUDA device / device index out of range */
    TC_ECUDA = -3,     /* CUDA runtime error (message carries cudaGetErrorString) */
    TC_EDIM = -4,      /* numel(t_interp) != N: MATLAB would raise a dimension error at
                          src/dependencies/ConstantElongationSim.m:47 */
    TC_ENOMEM = -5,
    TC_ESTATE = -6     /* ss(theta0) not finite etc. */
};

/* Construct table — replaces the if-block of src/GetFluorFromPolPos.m:18-45.
 * L_* are the BASE lengths (kb); the engine adds tau*v (:19-20).  One entry per loop set; the
 * reference indexes the PP7 vectors with the MS2 loop index (:47,60-69), so both colours have
 * nsets entries.  fluorval = loopn/24 (:48,60).  Requires start >= 0 (unloaded polymerases sit at
 * position 0 and must not light up), start < end. */
typedef struct tc_construct {
    int32_t nsets;
    int32_t _pad;
    double L_ms2, L_pp7;
    double ms2_start[TC_MAX_SETS], ms2_end[TC_MAX_SETS], ms2_loopn[TC_MAX_SETS];
    double pp7_start[TC_MAX_SETS], pp7_end[TC_MAX_SETS], pp7_loopn[TC_MAX_SETS];
} tc_construct;

/* Forward-model algorithm selector (results agree to ~1e-14 relative; tests/test_gpu_ss.py) */
enum {
    TC_ALGO_PAIRS = 0,     /* every (cohort i, time j) pair with position v*(t_j - t_i); any grid.
                              This is the W_op(N) = 11 N(N-1)/2 + 20 N algorithm of SURVEY.md 8(d). */
    TC_ALGO_TOEPLITZ = 1   /* uniform t_interp grid only: the response depends on the lag alone and is 0 / ramp /
                              plateau / 0 in the lag, so each time point is O(1) from two exact prefix sums of the
                              cohort sizes (counts K, first moments S): O(N) per evaluation (DESIGN.md 4.1) */
};

/* Options of the DRAM sampler — replaces the `model`/`options` structs handed to mcmcrun at
 * src/TranscriptionCycleMCMC.m:257-270 plus mcmcstat's own defaults (upstream, un-vendored; each
 * default's evidence level is in DESIGN.md). */
typedef struct tc_mcmc_opts {
    int32_t nsimu;            /* options.nsimu = n_steps (:264); rows of the chain incl. row 1 = x0 */
    int32_t burnintime;       /* options.burnintime = n_burn (:267) */
    int32_t adaptint;         /* options.adaptint = 100 (:268); 0 disables adaptation */
    int32_t ntry;             /* 'dram' => 2: one delayed-rejection retry; 1 => plain AM */
    int32_t updatesigma;      /* options.updatesigma = 1 (:265) */
    int32_t burnin_cumulative;/* burn-in scaling: 1 (default) the CUMULATIVE rejection rate, mcmcstat's
                                 `rejected > 0.95*isimu` (SURVEY.md 3.2 / B.3, [U]); 0: rejections since the last adaptation */
    int32_t n_burn;           /* summaries / stored rows start at MATLAB row n_burn: chain(n_burn:end,:)
                                 (:276-283); >= 1 */
    int32_t store_chain;      /* 0: summaries only; 1: also return rows n_burn..nsimu and s2chain (every thin-th of them) */
    int32_t replay;           /* 1: consume caller-supplied randomness instead of Philox */
    int32_t algo;             /* TC_ALGO_* used for ssfun inside the sampler */
    int32_t ngpus;            /* 'numParPools' reinterpreted: devices 0..ngpus-1 (or devices[]) */
    int32_t devices[TC_MAX_GPUS]; /* used when devices[0] >= 0 ... else 0..ngpus-1 */
    double drscale;           /* 5 */
    double adascale;          /* <= 0 => 2.4/sqrt(npar) */
    double qcovadj;           /* 1e-8 */
    double burnin_scale;      /* 10 */
    double N0;                /* 1 */
    double S20;               /* sigma2_0 */
    double sigma2_0;          /* model.sigma2 = 1 (:212,259) */
    uint64_t seed;            /* Philox key; draws are addressed by (seed, chain_uid, step, slot), never by device or place in
                                 the launch, so for a given sampler the results are bit-identical for every GPU count and
                                 partition.  Under TC_LAYOUT_AUTO the sampler is chosen per device (see layout) */
    int32_t layout;           /* TC_LAYOUT_AUTO (0): one CTA per chain (speculative rounds) for up to a few chains per SM, one
                                 WARP per chain beyond that (thousands of chains: BASELINE config 3), the large-series
                                 layout for series with more than ~210 points.  TC_LAYOUT_BIG forces the large-series layout
                                 (ring of 8 proposal slots, proposal factor factorised through HBM/L2), TC_LAYOUT_WARP the
                                 chain-per-warp kernel, TC_LAYOUT_CTA the CTA-per-chain kernel whatever the chain count.  The
                                 same chain whichever runs, to rounding: the kernels factor the covariance in different
                                 orders (DESIGN.md 2), so flags and counters agree, means to about 1e-9 after 1 000 steps
                                 (up to 1e-3 on near-singular covariances at qcovadj_always = 0), not bit for bit.  AUTO
                                 picks the chain-per-warp kernel from 13 chains per SM on, counted per DEVICE: with ngpus > 1 and 13 S <= nchains < 13 S ngpus
                                 (S SMs per device) one GPU runs it and several run the CTA-per-chain kernel, so there the
                                 GPU count changes the last bits of the output.  Force TC_LAYOUT_WARP or TC_LAYOUT_CTA for
                                 results bit-identical across GPU counts at every chain count */
    int32_t qcovadj_always;   /* 0 (default): R = chol(cov), and chol(cov + qcovadj I) only when that fails — mcmcstat's
                                 "try to blow it" branch [U]; 1: always factor cov + qcovadj I */
    int32_t thin;             /* store_chain: keep every thin-th row (>= 1; 1, the default: every row).  chain keeps the 0-based
                                 rows n_burn-1 + j*thin, j < nkeep = (nsimu-n_burn)/thin + 1; s2chain the rows j*thin,
                                 j < ns2 = (nsimu-1)/thin + 1: a regular subsample of the chain thin = 1 returns, bit for bit.
                                 mean, std, sig, the counters, flags and sschain still cover every row.  Ignored without
                                 store_chain */
} tc_mcmc_opts;
enum { TC_LAYOUT_AUTO = 0, TC_LAYOUT_BIG = 1, TC_LAYOUT_WARP = 2, TC_LAYOUT_CTA = 3 };

/* Per-chain counters returned by tc_mcmc_run (int64 each) */
enum {
    TC_CNT_SS_EVALS = 0, TC_CNT_ACC_STAGE1 = 1, TC_CNT_ACC_STAGE2 = 2, TC_CNT_OUT_OF_BOUNDS = 3,
    TC_CNT_ADAPTATIONS = 4, TC_CNT_CHOL_FAIL = 5, TC_CNT_DR_TRIES = 6, TC_CNT_STATUS = 7,
    /* TC_CNT_CYCLES0 + i: SM cycles the chain spent per phase (clock readings, not results), by sampler.
       One CTA per chain (TC_LAYOUT_CTA / _BIG), cycles of thread 0:
         +0 generation (randomness + proposal increments), +1 bounds checks + the speculative evaluations of a
         round, +2 decisions + commit of a round, +3 +4 +6 always 0, +5 adaptation (covariance update + Cholesky);
         +7 is a count: forward-model evaluations executed, including the discarded speculative ones
         (TC_CNT_SS_EVALS counts only the committed).
       One warp per chain (TC_LAYOUT_WARP), cycles of lane 0:
         +0 generation, +1 the step loop, +2 waits at the barriers that keep the CTA's warps in one phase,
         +3 the randomness part of +0, +4 the scatter-update part of +5, +5 adaptation, +6 the scatter-update +
         factorisation part of +5; +7 = TC_CNT_SS_EVALS (no speculation: every evaluation is committed; a
         -DWK_SUBPROF development build puts the cycles of the forward-model evaluations there instead). */
    TC_CNT_CYCLES0 = 8,
    TC_NCOUNTERS = 16
};
/* Per-step flag bits returned in `flags` (replay / parity harness) */
enum { TC_FL_ACCEPT = 1, TC_FL_STAGE2 = 2, TC_FL_OOB1 = 4, TC_FL_DR = 8, TC_FL_OOB2 = 16 };

typedef struct tc_cells tc_cells;   /* opaque: packed cells resident on one or more devices */

typedef struct tc_device_info {
    char name[128];
    int32_t cc_major, cc_minor, sm_count, _pad;
    int64_t total_mem, smem_per_block_optin;
} tc_device_info;

int tc_version(void);
const char *tc_last_error(void);
int tc_device_count(int *count);
int tc_device_info_get(int device, tc_device_info *out);
void tc_opts_default(tc_mcmc_opts *o);     /* mcmcstat defaults + reference configuration */

/* Upload a dataset — replaces the struct array `data(cellNum).{time,MS2,PP7}` after truncation to
 * [t_start,t_end) (src/TranscriptionCycleMCMC.m:163-181).  N[c] timepoints for cell c stored at
 * off[c].. (off has ncells+1 entries); NaN = missing sample.  Precomputes per cell, on the host,
 * dt = mean(diff(t)) and t_interp = t(1):dt:t(end) with MATLAB colon semantics
 * (src/SumofSquaresFunction_TranscriptionCycleMCMC.m:29-30) and the interp1 bracketing
 * index/weight of every experimental time (:55-56).  ndev devices (NULL => device 0). */
int tc_cells_create(const tc_construct *construct, int ncells, const int32_t *N, const int64_t *off,
                    const double *t, const double *ms2, const double *pp7, int ndev,
                    const int32_t *devices, tc_cells **out);
void tc_cells_destroy(tc_cells *cells);
/* t_interp of cell c as the engine computed it (host copy; for tests) */
int tc_cells_t_interp(const tc_cells *cells, int cell, double *out, int cap);

/* ss = ssfun(theta, data) for a batch of (cell, theta) pairs — replaces
 * src/SumofSquaresFunction_TranscriptionCycleMCMC.m:1-65 (called through the closure at
 * src/TranscriptionCycleMCMC.m:186).  theta is [nbatch x ld].  Runs on cells' first device. */
int tc_ss_batch(const tc_cells *cells, int64_t nbatch, const int32_t *cell_id, const double *theta,
                int ld, int algo, double *ss_out);
int tc_ss_batch_device(const tc_cells *cells, int device, int64_t nbatch, const int32_t *d_cell_id,
                       const double *d_theta, int ld, int algo, double *d_ss_out, void *stream);

/* [A*MS2, PP7] model curves — replaces ConstantElongationSim + GetFluorFromPolPos + the A scaling as
 * called at src/TranscriptionCycleMCMC.m:307-309 (on_raw_grid = 1: raw data.xdata, no interp1) or at
 * SumofSquares...m:49-51 (on_raw_grid = 0: on t_interp).  Outputs are [nbatch x ldo], ldo >= N. */
int tc_forward(const tc_cells *cells, int64_t nbatch, const int32_t *cell_id, const double *theta,
               int ld, int on_raw_grid, double *ms2_out, double *pp7_out, int ldo);

/* The DRAM fit — replaces [results,chain,s2chain] = mcmcrun(model,data,params,options) at
 * src/TranscriptionCycleMCMC.m:273 for nchains independent chains (one per parfor iteration, :161),
 * plus the slicing/summaries of :276-303.
 *   chain_cell[c]  cell index of chain c;  chain_uid[c]  RNG identity (NULL => c)
 *   theta0, qcov_diag (J0 diagonal = proposal VARIANCES, :230,266), low, upp, prior_mu, prior_sig
 *   (params cell array :242-255; prior_sig = Inf => flat):  [nchains x ld]
 * Outputs (any may be NULL):
 *   mean, std [nchains x ld]   mean / population std of rows n_burn..nsimu (:286-301)
 *   sig [nchains x 2]          sqrt(mean(s2chain)), std(sqrt(s2chain),1) over ALL rows (:302-303)
 *   counters [nchains x TC_NCOUNTERS] int64
 *   chain [nchains x nkeep x ld], s2chain [nchains x ns2]   (store_chain = 1; opts->thin = 1: nkeep = nsimu-n_burn+1,
 *                              ns2 = nsimu; larger thin: the counts of tc_mcmc_opts.thin)
 * Series length: max(N) <= 441 (one CTA per chain holds the cell, the chain state, the proposal slots and the
 * forward-model scratch in one SM; beyond ~210 points the large-series layout of opts->layout is used); longer series
 * return TC_EINVAL.
 * Replay harness (opts->replay = 1): z1,z2 [nchains x nsimu x ld], u1,u2,chi2 [nchains x nsimu]
 * (row k feeds MCMC step k; row 0 unused) and optional per-step outputs flags [nchains x nsimu]
 * int32 and sschain [nchains x nsimu]. */
typedef struct tc_replay {
    const double *z1, *u1, *z2, *u2, *chi2;
    int32_t *flags;
    double *sschain;
} tc_replay;

int tc_mcmc_run(const tc_cells *cells, const tc_mcmc_opts *opts, int nchains,
                const int32_t *chain_cell, const uint64_t *chain_uid, int ld, const double *theta0,
                const double *qcov_diag, const double *low, const double *upp,
                const double *prior_mu, const double *prior_sig, double *mean, double *std,
                double *sig, int64_t *counters, double *chain, double *s2chain,
                const tc_replay *replay);

/* Seconds spent in the sampler kernel(s) of the last tc_mcmc_run on this thread, measured with CUDA
 * events on the launching stream (max over devices). */
double tc_last_kernel_seconds(void);
/* Host seconds the last tc_mcmc_run on this thread spent draining its outputs (device -> host copies of summaries, counters
 * and, with store_chain, the raw chains) after the kernels had finished. */
double tc_last_drain_seconds(void);

/* Page-locked host memory for large outputs (the raw chains of src/TranscriptionCycleMCMC.m:276-283,315-323 are GBs): a
 * chain / s2chain buffer allocated here goes device -> host by DMA at PCIe speed and, with several GPUs, in parallel;
 * ordinary (pageable) buffers are accepted everywhere too, only slower.  Free with tc_host_free. */
int tc_host_alloc(size_t bytes, void **out);
void tc_host_free(void *p);

/* The randomness tc_mcmc_run would draw for (seed, chain_uid) at steps [0, nsimu): lets the CPU
 * oracle consume the device's Philox streams.  z1,z2 [nsimu x npar]; u1,u2,chi2 [nsimu]. */
int tc_rng_dump(uint64_t seed, uint64_t chain_uid, int npar, double chi2_dof, int nsimu, double *z1,
                double *u1, double *z2, double *u2, double *chi2, int device);

/* FP64 DFMA micro-benchmark on `device`: returns measured DFMA instructions/s (lane-ops/s) so the
 * roofline denominator is measured, not assumed (SURVEY.md 8d). */
int tc_measure_fp64_peak(int device, double *dfma_per_s, double *sm_clock_mhz);

/* Development aid: cycle counts of the sampler's sub-phases for chain 0 (read and reset).  Returns 1
 * and fills out[0..n) when the library was built with -DTC_SUBPROF, else returns 0 and zero-fills. */
int tc_debug_subprof(long long *out, int n);

#ifdef __cplusplus
}
#endif
#endif /* TCMCMC_H */
