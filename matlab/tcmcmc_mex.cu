// tcmcmc_mex.cu — MEX gateway: MATLAB <-> libtcmcmc C ABI (include/tcmcmc.h).
//
// Build (on a machine with MATLAB + CUDA; NOT buildable in the development container, which has no
// mex.h — everything testable lives behind the C ABI, this file only marshals):
//     mexcuda -I../include tcmcmc_mex.cu -L../transcriptioncycleinference_b200 -ltcmcmc
//
// MATLAB call (from matlab/TranscriptionCycleMCMC.m, replacing the parfor body of the reference,
// src/TranscriptionCycleMCMC.m:161-357):
//
//   out = tcmcmc_mex('fit', construct, cells, opts, x0, J0diag, low, upp, prior_mu, prior_sig)
//   sim = tcmcmc_mex('forward', construct, cells, theta)       % best-fit curves on the raw grid (:307-309)
//
//   construct  struct: L_MS2, L_PP7, MS2_start, MS2_end, MS2_loopn, PP7_start, PP7_end, PP7_loopn
//              (the quantities of src/GetFluorFromPolPos.m:18-30; vectors = one entry per loop set)
//   cells      1 x Ncells struct array with fields time, MS2, PP7 (already truncated to [t_start,t_end))
//   opts       struct: n_steps, n_burn, numGPUs, seed, saveChains  (+ optional mcmcstat overrides); chainCell: optional
//              1 x Nchains vector, the (1-based) cell of every chain ('numChains' > 1); default one chain per cell; thin:
//              optional, store every thin-th row of the raw chains (default 1: every row)
//   x0 .. prior_sig   npar_max x Nchains double (column c = chain c, zero padded)
//
//   out        struct: mean, std (npar_max x Nchains), sig (2 x Nchains), counters (16 x Nchains, int64),
//              chain (npar_max x nkeep x Nchains), s2chain (ns2 x Nchains) [chain/s2chain only when opts.saveChains; rows
//              n_burn, n_burn+thin, .. of the chain, nkeep = floor((n_steps-n_burn)/thin)+1, and rows 1, 1+thin, .. of
//              s2chain, ns2 = ceil(n_steps/thin)], simMS2/simPP7 (Nmax x Ncells; only with one chain per cell)
//   sim        struct: simMS2, simPP7 (Nmax x Ncells) for theta (npar_max x Ncells)
#include <cstring>
#include <vector>

#include "mex.h"
#include "tcmcmc.h"

static double field_scalar(const mxArray *s, const char *name, double dflt)
{
    const mxArray *f = mxGetField(s, 0, name);
    return f ? mxGetScalar(f) : dflt;
}

static void fill_vec(const mxArray *s, const char *name, double *dst, int &n)
{
    const mxArray *f = mxGetField(s, 0, name);
    if (!f) mexErrMsgIdAndTxt("tcmcmc:construct", "construct.%s is missing", name);
    n = (int)mxGetNumberOfElements(f);
    if (n < 1 || n > TC_MAX_SETS) mexErrMsgIdAndTxt("tcmcmc:construct", "construct.%s: 1..%d loop sets", name, TC_MAX_SETS);
    std::memcpy(dst, mxGetPr(f), sizeof(double) * n);
}

static void check(int rc)
{
    if (rc < 0) mexErrMsgIdAndTxt("tcmcmc:engine", "%s", tc_last_error());
}

static void read_construct(const mxArray *a, tc_construct &c)
{
    std::memset(&c, 0, sizeof(c));
    c.L_ms2 = field_scalar(a, "L_MS2", 0);
    c.L_pp7 = field_scalar(a, "L_PP7", 0);
    int n = 0, n2 = 0;
    fill_vec(a, "MS2_start", c.ms2_start, n);
    fill_vec(a, "MS2_end", c.ms2_end, n2);
    fill_vec(a, "MS2_loopn", c.ms2_loopn, n2);
    fill_vec(a, "PP7_start", c.pp7_start, n2);
    fill_vec(a, "PP7_end", c.pp7_end, n2);
    fill_vec(a, "PP7_loopn", c.pp7_loopn, n2);
    c.nsets = n;
}

struct Packed {
    int ncells = 0, Nmax = 0;
    std::vector<int32_t> N;
    std::vector<int64_t> off;
    std::vector<double> t, ms2, pp7;
};
static void read_cells(const mxArray *a, Packed &p)
{
    p.ncells = (int)mxGetNumberOfElements(a);
    p.N.resize(p.ncells);
    p.off.assign(p.ncells + 1, 0);
    for (int i = 0; i < p.ncells; ++i) {
        const mxArray *ft = mxGetField(a, i, "time"), *f1 = mxGetField(a, i, "MS2"), *f2 = mxGetField(a, i, "PP7");
        if (!ft || !f1 || !f2) mexErrMsgIdAndTxt("tcmcmc:cells", "cells need the fields time, MS2, PP7");
        p.N[i] = (int32_t)mxGetNumberOfElements(ft);
        p.off[i + 1] = p.off[i] + p.N[i];
        p.Nmax = p.N[i] > p.Nmax ? p.N[i] : p.Nmax;
        p.t.insert(p.t.end(), mxGetPr(ft), mxGetPr(ft) + p.N[i]);
        p.ms2.insert(p.ms2.end(), mxGetPr(f1), mxGetPr(f1) + p.N[i]);
        p.pp7.insert(p.pp7.end(), mxGetPr(f2), mxGetPr(f2) + p.N[i]);
    }
}

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    char cmd[16] = "";
    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], cmd, sizeof(cmd)))
        mexErrMsgIdAndTxt("tcmcmc:usage", "tcmcmc_mex('fit' | 'forward', ...)");
    tc_construct c;
    Packed p;
    if (!std::strcmp(cmd, "forward")) {
        if (nrhs != 4) mexErrMsgIdAndTxt("tcmcmc:usage", "tcmcmc_mex('forward', construct, cells, theta)");
        read_construct(prhs[1], c);
        read_cells(prhs[2], p);
        const int ld = (int)mxGetM(prhs[3]);
        if ((int)mxGetN(prhs[3]) != p.ncells || ld < 7 + p.Nmax) mexErrMsgIdAndTxt("tcmcmc:dims", "theta must be (7+max N) x Ncells");
        tc_cells *cells = nullptr;
        check(tc_cells_create(&c, p.ncells, p.N.data(), p.off.data(), p.t.data(), p.ms2.data(), p.pp7.data(), 1, nullptr, &cells));
        std::vector<int32_t> id(p.ncells);
        for (int i = 0; i < p.ncells; ++i) id[i] = i;
        const char *names[] = {"simMS2", "simPP7"};
        plhs[0] = mxCreateStructMatrix(1, 1, 2, names);
        mxArray *sim1 = mxCreateDoubleMatrix(p.Nmax, p.ncells, mxREAL), *sim2 = mxCreateDoubleMatrix(p.Nmax, p.ncells, mxREAL);
        const int rc = tc_forward(cells, p.ncells, id.data(), mxGetPr(prhs[3]), ld, 1, mxGetPr(sim1), mxGetPr(sim2), p.Nmax);
        tc_cells_destroy(cells);
        check(rc);
        mxSetField(plhs[0], 0, "simMS2", sim1); mxSetField(plhs[0], 0, "simPP7", sim2);
        return;
    }
    if (std::strcmp(cmd, "fit") || nrhs != 10) mexErrMsgIdAndTxt("tcmcmc:usage", "tcmcmc_mex('fit', construct, cells, opts, x0, J0, low, upp, mu, sig)");
    read_construct(prhs[1], c);
    read_cells(prhs[2], p);
    const int ncells = p.ncells, Nmax = p.Nmax;
    // ---- options: mcmcstat defaults + the reference's configuration, then the caller's values
    tc_mcmc_opts o;
    tc_opts_default(&o);
    o.nsimu = (int)field_scalar(prhs[3], "n_steps", o.nsimu);
    o.burnintime = o.n_burn = (int)field_scalar(prhs[3], "n_burn", o.n_burn);
    o.ngpus = (int)field_scalar(prhs[3], "numGPUs", 1);            // 'numParPools' reinterpreted
    o.seed = (uint64_t)field_scalar(prhs[3], "seed", (double)o.seed);
    o.store_chain = (int)field_scalar(prhs[3], "saveChains", 1);
    o.adaptint = (int)field_scalar(prhs[3], "adaptint", o.adaptint);
    o.drscale = field_scalar(prhs[3], "drscale", o.drscale);
    o.qcovadj = field_scalar(prhs[3], "qcovadj", o.qcovadj);
    o.qcovadj_always = (int32_t)field_scalar(prhs[3], "qcovadj_always", o.qcovadj_always);
    o.burnin_cumulative = (int32_t)field_scalar(prhs[3], "burnin_cumulative", o.burnin_cumulative);
    o.N0 = field_scalar(prhs[3], "N0", o.N0);
    o.layout = (int32_t)field_scalar(prhs[3], "layout", o.layout);   // TC_LAYOUT_AUTO; 1: large-series layout, 2: one warp per chain
    o.thin = (int32_t)field_scalar(prhs[3], "thin", 1);
    int ndev = 0;
    check(tc_device_count(&ndev));
    if (o.ngpus > ndev) o.ngpus = ndev;
    // ---- chains: one per cell, or opts.chainCell (1-based cell of every chain)
    const mxArray *cc = mxGetField(prhs[3], 0, "chainCell");
    const int nchains = cc ? (int)mxGetNumberOfElements(cc) : ncells;
    std::vector<int32_t> chain_cell(nchains);
    std::vector<uint64_t> uid(nchains);
    std::vector<int> seen(ncells, 0);
    for (int i = 0; i < nchains; ++i) {
        const int ci = cc ? (int)mxGetPr(cc)[i] - 1 : i;
        if (ci < 0 || ci >= ncells) mexErrMsgIdAndTxt("tcmcmc:dims", "opts.chainCell out of range");
        chain_cell[i] = ci;
        uid[i] = ((uint64_t)ci << 20) + (uint64_t)seen[ci]++;      // RNG identity = (cell, replica): independent of the order
    }
    const int ld = (int)mxGetM(prhs[4]);                             // npar_max rows, one column per chain
    if ((int)mxGetN(prhs[4]) != nchains || ld < 7 + Nmax) mexErrMsgIdAndTxt("tcmcmc:dims", "x0 must be (7+max N) x Nchains");
    // ---- run
    tc_cells *cells = nullptr;
    std::vector<int32_t> devs(o.ngpus);
    for (int d = 0; d < o.ngpus; ++d) devs[d] = d;
    check(tc_cells_create(&c, ncells, p.N.data(), p.off.data(), p.t.data(), p.ms2.data(), p.pp7.data(), o.ngpus, devs.data(), &cells));
    const char *names[] = {"mean", "std", "sig", "counters", "chain", "s2chain", "simMS2", "simPP7"};
    plhs[0] = mxCreateStructMatrix(1, 1, 8, names);
    mxArray *mean = mxCreateDoubleMatrix(ld, nchains, mxREAL), *sd = mxCreateDoubleMatrix(ld, nchains, mxREAL);
    mxArray *sig = mxCreateDoubleMatrix(2, nchains, mxREAL);
    mxArray *cnt = mxCreateNumericMatrix(TC_NCOUNTERS, nchains, mxINT64_CLASS, mxREAL);
    mxArray *chain = nullptr, *s2 = nullptr;
    if (o.store_chain) {
        if (o.thin < 1) mexErrMsgIdAndTxt("tcmcmc:opts", "opts.thin must be an integer >= 1");
        // MATLAB is column-major: [ld x nkeep x nchains] here is the engine's row-major [nchains][nkeep][ld]
        const mwSize dims[3] = {(mwSize)ld, (mwSize)((o.nsimu - o.n_burn) / o.thin + 1), (mwSize)nchains};
        chain = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);
        s2 = mxCreateDoubleMatrix((o.nsimu - 1) / o.thin + 1, nchains, mxREAL);
    }
    const int rc = tc_mcmc_run(cells, &o, nchains, chain_cell.data(), uid.data(), ld, mxGetPr(prhs[4]), mxGetPr(prhs[5]),
                               mxGetPr(prhs[6]), mxGetPr(prhs[7]), mxGetPr(prhs[8]), mxGetPr(prhs[9]), mxGetPr(mean),
                               mxGetPr(sd), mxGetPr(sig), (int64_t *)mxGetData(cnt), chain ? mxGetPr(chain) : nullptr,
                               s2 ? mxGetPr(s2) : nullptr, nullptr);
    // best-fit curves at the posterior means on the RAW grid (src/TranscriptionCycleMCMC.m:307-309); with several chains
    // per cell the caller pools the means first and asks for the curves with 'forward'
    mxArray *sim1 = nullptr, *sim2 = nullptr;
    int rc2 = rc;
    if (rc >= 0 && !cc) {
        sim1 = mxCreateDoubleMatrix(Nmax, ncells, mxREAL); sim2 = mxCreateDoubleMatrix(Nmax, ncells, mxREAL);
        rc2 = tc_forward(cells, ncells, chain_cell.data(), mxGetPr(mean), ld, 1, mxGetPr(sim1), mxGetPr(sim2), Nmax);
    }
    tc_cells_destroy(cells);
    check(rc2);
    mxSetField(plhs[0], 0, "mean", mean); mxSetField(plhs[0], 0, "std", sd); mxSetField(plhs[0], 0, "sig", sig);
    mxSetField(plhs[0], 0, "counters", cnt);
    if (chain) { mxSetField(plhs[0], 0, "chain", chain); mxSetField(plhs[0], 0, "s2chain", s2); }
    if (sim1) { mxSetField(plhs[0], 0, "simMS2", sim1); mxSetField(plhs[0], 0, "simPP7", sim2); }
}
