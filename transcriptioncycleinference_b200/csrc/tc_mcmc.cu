// tc_mcmc.cu — kernels and C ABI of libtcmcmc.so (sm_100a).  See include/tcmcmc.h for the boundary
// and DESIGN.md for the data layout and roofline of each kernel.
//
//   ss_batch_kernel   one warp per (cell, theta): the batched ssfun
//                     (replaces src/SumofSquaresFunction_TranscriptionCycleMCMC.m:1-65), and, with output
//                     pointers, the model curves for the best-fit plots (src/TranscriptionCycleMCMC.m:307-309)
//   dram_kernel       persistent CTAs time-slicing the chains: the whole mcmcrun DRAM loop device-resident
//                     (replaces the call at src/TranscriptionCycleMCMC.m:273 + summaries :276-303)
//   rng_dump_kernel   the Philox streams of a chain, for the parity harness
//   dfma_peak_kernel  FP64 pipe micro-benchmark (roofline denominator)
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "tc_device.cuh"

using namespace tc;

// ------------------------------------------------------------------------------------ utilities
static thread_local std::string g_err;
static thread_local double g_last_kernel_s = 0.0;
static thread_local double g_last_drain_s = 0.0;

static int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return fail(TC_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));       \
    } while (0)

// The library is loaded into host applications (MATLAB through MEX, a PyTorch process) that have their own notion of the
// current device: every entry point that calls cudaSetDevice restores the caller's device on return.
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define DRAM_THREADS 256   // 8 warps per chain
#define SPEC 8             // forward-model evaluations per speculative round (= warps per CTA)
#define RING 16            // ring of proposal increments: generated GEN_M steps at a time, ahead of use
#define SS_WARPS 8
#define SS_THREADS (32 * SS_WARPS)
#define SS_MIN_CTAS 4          // 64 registers: 32 warps per SM hide the latency of streaming theta (measured +12 % over 2)
#define TC_WARP_MIN_CHAINS_PER_SM 13  // chain-per-warp kernel from this many chains per SM on (measured crossover on B200: ~1 900 chains)
#define TC_SOLO_LAG 2       // dram_kernel: slices a chain must lag the mean progress by to get its SM to itself (0: never)
#define TC_SOLO_NSEG 128    // ... and the number of time slices per chain then
#define TC_UNSLICED_CHAINS (4 * 296)  // dram_kernel from this many chains on: many chains per CTA slot, imbalance averages out, no slicing
#define COV_CR 32          // weighted rows of the covariance block staged per pass of the scatter update

// development aid: cycle counts of sub-phases, chain 0 only (build with -DTC_SUBPROF; see scripts/subprof.py)
#ifdef TC_SUBPROF
__device__ long long tc_subprof[32];
#define SUBP_BEGIN long long sp_prev__ = clock64()
#define SUBP(i) do { if (threadIdx.x == 0 && cx.ch == 0) { const long long t__ = clock64(); tc_subprof[i] += t__ - sp_prev__; sp_prev__ = t__; } } while (0)
#else
#define SUBP_BEGIN
#define SUBP(i)
#endif

// --------------------------------------------------------------------------------- SS / forward
struct SsArgs {
    CellsDev cells;
    ConsX cons;
    long long nbatch;
    const int *cell_id;
    const double *theta;
    int ld, algo, raw_grid, ldo, wsz;
    int csz, ld2;                                       // ss_stream_kernel: per-warp cell area / theta buffer (doubles, even)
    double *ss_out, *out1, *out2;
};

// one warp per (cell, theta): no block barriers, cell data and theta read straight from HBM/L2
__global__ void __launch_bounds__(SS_THREADS, SS_MIN_CTAS) ss_batch_kernel(const __grid_constant__ SsArgs a)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int base = warp * a.wsz;                          // this warp's scratch (offset into tc_smem)
#pragma unroll 1
    for (long long b = (long long)blockIdx.x * SS_WARPS + warp; b < a.nbatch; b += (long long)gridDim.x * SS_WARPS) {
        const int cid = a.cell_id[b];
        const GlobCell cv = view_cell(a.cells, cid, a.raw_grid != 0);
        Work w;
        carve_work(base, cv.N, w);
        double *o1 = a.out1 ? a.out1 + b * a.ldo : nullptr;
        double *o2 = a.out2 ? a.out2 + b * a.ldo : nullptr;
        const double ss = ss_eval(a.cons, cv, GlobVec{a.theta + b * a.ld}, w, a.algo, false, o1, o2);
        if (lane == 0 && a.ss_out) a.ss_out[b] = ss;
    }
}

// The batched ssfun when only SS is wanted (tc_ss_batch, tc_ss_batch_device): every warp owns a CONTIGUOUS run of the
// batch and keeps its operands in shared memory, the way the sampler does — the cell's series are staged once and reused
// while consecutive items belong to the same cell (proposals for a cell arrive together), theta of item i+1 streams in
// with cp.async while item i is evaluated (double buffer) — so an evaluation never waits on a global load: the
// global-view kernel above spends half of its warp-cycles in long-scoreboard stalls (ncu, profiles/ncu_ss_r1w.txt).
// Per warp: [cell | theta x 2 | forward-model scratch] = 13 KB at N = 129, two CTAs per SM.
__global__ void __launch_bounds__(SS_THREADS, 2) ss_stream_kernel(const __grid_constant__ SsArgs a)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // theta buffers start at an ODD offset: element 7 (the first dR) is then 16-byte aligned and the loading scan fetches
    // the four steps of a lane with two 16-byte loads (SmemVecA)
    const int o_cell = warp * (a.csz + 2 * a.ld2 + 2 + a.wsz), o_th = o_cell + a.csz + 1, o_work = o_cell + a.csz + 2 + 2 * a.ld2;
    const long long nw = (long long)gridDim.x * SS_WARPS, wi = (long long)blockIdx.x * SS_WARPS + warp;
    const long long chunk = (a.nbatch + nw - 1) / nw, b0 = wi * chunk, b1 = min(a.nbatch, b0 + chunk);
    const unsigned sth = (unsigned)__cvta_generic_to_shared(tc_smem + o_th);
    int cur = -1;
    SmemCell cv{};
    Work w{};
#define SS_ISSUE_THETA(bb, buf)                                                                             \
    {                                                                                                       \
        const double *src__ = a.theta + (bb) * a.ld;                                                        \
        for (int i = lane; i < a.ld; i += 32)                                                               \
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sth + 8u * (unsigned)((buf) * a.ld2 + i)), "l"(src__ + i) : "memory"); \
        asm volatile("cp.async.commit_group;" ::: "memory");                                                \
    }
    if (b0 < b1) SS_ISSUE_THETA(b0, 0)
#pragma unroll 1
    for (long long b = b0; b < b1; ++b) {
        const int buf = (int)(b - b0) & 1;
        const bool more = b + 1 < b1;
        if (more) SS_ISSUE_THETA(b + 1, buf ^ 1)
        const int cid = a.cell_id[b];
        if (cid != cur) {                                       // warp-uniform
            const int N = a.cells.N[cid];
            carve_cell(o_cell, N, cv);
            carve_work(o_work, N, w);
            stage_cell(a.cells, cid, cv, lane, 32);
            cv.d = a.cells.dmean[cid];
            cur = cid;
        }
        if (more) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        const double ss = ss_eval(a.cons, cv, SmemVecA{o_th + buf * a.ld2}, w, a.algo, false, nullptr, nullptr);
        if (lane == 0) a.ss_out[b] = ss;
        __syncwarp();                                           // the buffer is free for the copy issued two items on
    }
#undef SS_ISSUE_THETA
}

// ------------------------------------------------------------------------------------- sampler
struct RunArgs {
    CellsDev cells;
    ConsX cons;
    // options
    int nsimu, burnintime, adaptint, ntry, updatesigma, burnin_cumulative, n_burn, store_chain, replay,
        algo, qcovadj_always;
    double drscale, adascale, qcovadj, burnin_scale, N0, S20, sigma2_0;
    unsigned long long seed;
    // chains
    int nchains, ld, ldR, do_cov, wsz, big;
    int nmax;                                           // max N over the dataset: sizes the chain-per-warp kernel's shared-memory
                                                        // regions and increment slots (ld may be larger: a caller's padding)
    int blk_rows;                                       // rows of the largest adaptation block: the distinct-row buffer of a chain
    const int *chain_cell;
    const unsigned long long *chain_uid;
    const double *theta0, *qcov_diag, *low, *upp, *pmu, *psig;
    double *mean, *std, *sig;
    long long *counters;
    double *chain, *s2chain;
    const double *z1, *u1, *z2, *u2, *chi2;
    int *flags;
    double *sschain;
    // scratch (global)
    double *gR, *gM2, *gRows, *gWts, *gCmean, *gState;
    double *gW;                                         // big layout: one Cholesky workspace (ldR doubles) per CTA; warp kernel: per warp
    // chain-per-warp kernel (tc_warp.cuh): reciprocal prior widths and block-mean accumulators per chain; per warp slot the
    // increments / scalars of the current batch of steps; the work-item counter
    double *gPinv, *gMb, *gInc, *gSc;
    unsigned long long *wq;
    // time slicing
    int seglen;
    int thin;                                           // store_chain: every thin-th row is stored.  (thin and nkeep fill the
                                                        // alignment holes before the pointers: the fields keep their offsets)
    int *cstate;
    // dram_kernel, two CTAs per SM: a chain that lags the mean progress by solo_lag slices or more gets its SM to itself
    // (smctl[%smid] = 1 + blockIdx of the owner; 0: shared); solo_lag <= 0: off
    int solo_lag;
    int nkeep;                                          // store_chain: chain rows stored per chain (thin_nkeep)
    int *smctl;
};

// Shared-memory budget of the sampler (doubles), N = max time points over the dataset.
//   cell constants | 10 per-parameter vectors | RING slots of interleaved proposal increments (+8 scalars)
//   | SPEC per-warp forward-model scratch areas.
// Ring + per-warp areas are contiguous: during adaptation (when both are idle) they are the workspace of
// the covariance update and of the Cholesky factorisation.
__host__ __device__ __forceinline__ int tidx(int nt4, int bi, int bj) { return bi * nt4 - (bi * (bi - 1)) / 2 + (bj - bi); }
// doubles of an n x n upper triangle in 4x4 tiles (the factor R, the scatter matrix M2, a Cholesky workspace)
__host__ __device__ __forceinline__ int tri_doubles(int n) { const int nt4 = (n + 3) >> 2; return 16 * (nt4 * (nt4 + 1) / 2); }
__host__ __device__ inline int chol_ws_doubles(int n)
{
    const int d = tri_doubles(n), T = d / 16;
    return d + (T + 3) / 4 + 2;                           // tiles + the u16 tile table
}

// one ring slot = [pad | increments of stage 1: s1 doubles | of stage 2: s1 | pad | 8 per-step scalars]; the two increment
// vectors start at ODD offsets (slot + 1, slot + 1 + s1, s1 even): element 7, the first dR, is then 16-byte aligned for the
// loading scan's vector loads (SumVec::get4)
__host__ __device__ inline int dram_s1(int N) { return (7 + N + 1) & ~1; }
__host__ __device__ inline int dram_slot(int N) { return 2 * dram_s1(N) + 2 + 8; }
// Two shared-memory layouts:
//   regular (big = 0): ring of RING = 16 slots, all 10 per-parameter vectors in shared memory, the Cholesky workspace
//                      of the proposal factor inside ring + per-warp areas (N up to ~210);
//   big     (big = 1): ring of 8 slots (randomness is generated when the ring is empty), bounds and prior means read
//                      from HBM/L2, the factorisation done through HBM/L2 by chol_global (N up to ~410, BASELINE config 5).
__host__ __device__ inline int dram_wsz(int N, int big)
{
    const int npar = 7 + N;
    int w = (work_doubles(N) + 1) & ~1;
    if (!big) {
        const int need = (chol_ws_doubles(npar) - RING * dram_slot(N) + SPEC - 1) / SPEC + 2;
        if (w < need) w = need;
    }
    const int need2 = 2 * ((npar + 3) & ~3) + 16 * 32;        // generate(): a row of Z + the warp's B staging (16 k-steps x 32 lanes)
    if (w < need2) w = need2;
    const int need3 = 4 * ((npar + 3) & ~3) + 48;              // gen_increments_tma(): one of the 8 ring stages (zero tile + tile row + slack)
    if (big && w < need3) w = need3;
    return (w + 1) & ~1;
}
__host__ __device__ inline int dram_smem_doubles(int N, int big)
{
    return cell_doubles(N) + (big ? 7 : 10) * (7 + N) + 4 + (big ? RING / 2 : RING) * dram_slot(N) + SPEC * dram_wsz(N, big) + 16;
}

// reciprocal pivots of the current diagonal block / failure flag of the factorisations (file scope: the out-of-line phases
// address them as shared memory, a pointer parameter would make every access generic)
__shared__ double tc_dinv[8];
__shared__ int tc_cholfail;
__shared__ int tc_genctr;                               // generate(): next unclaimed work item

// ---- Cholesky of the proposal covariance, in shared memory, by the whole CTA
// Storage: the upper triangle in 4x4 TILES (tile (bi, bj), bi <= bj, at index bi*nt4 - bi(bi-1)/2 + bj - bi, 16
// doubles row-major), padded to a multiple of 4 with an identity block, so that every tile operation is
// eight 16-byte shared-memory accesses with no index arithmetic; `tab[t]` = (bi << 8) | bj of tile t.
__device__ __forceinline__ void ld_tile(const double *p, double (&t)[16])
{
#pragma unroll
    for (int e = 0; e < 8; ++e) { const double2 v = reinterpret_cast<const double2 *>(p)[e]; t[2 * e] = v.x; t[2 * e + 1] = v.y; }
}
__device__ __forceinline__ void st_tile(double *p, const double (&t)[16])
{
#pragma unroll
    for (int e = 0; e < 8; ++e) reinterpret_cast<double2 *>(p)[e] = make_double2(t[2 * e], t[2 * e + 1]);
}

// Upper Cholesky of an 8x8 block held in registers (A[r][c], r <= c), in place; dinv = reciprocal pivots.  Returns true
// when a pivot is not positive.
__device__ __forceinline__ bool chol8(double (&A)[8][8], double (&dinv)[8])
{
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const double d = A[j][j];
        if (!(d > 0.0)) bad = true;
        // 1/sqrt(d): single-precision seed + two Newton steps in FP64 (full precision; the IEEE sqrt + divide pair is
        // ~60 dependent instructions per pivot, and the 8 pivots of a block are a serial chain on one warp)
        double ri = (double)rsqrtf((float)d);
        const double hd = 0.5 * d;
        ri = ri * fma(-hd * ri, ri, 1.5);
        ri = ri * fma(-hd * ri, ri, 1.5);
        dinv[j] = ri;
        A[j][j] = d * ri;
#pragma unroll
        for (int c = j + 1; c < 8; ++c) A[j][c] *= ri;
#pragma unroll
        for (int r = j + 1; r < 8; ++r)
#pragma unroll
            for (int c = r; c < 8; ++c) A[r][c] = fma(-A[j][r], A[j][c], A[r][c]);
    }
    return bad;
}
// (Measured and dropped: the root-free elimination U' D^-1 U — the next pivot then waits only for a reciprocal (MUFU.RCP64H seed +
// two Newton steps) and the reciprocal square roots are side chains: -2 % on the factorisation of dram_kernel, +4 % on the
// chain-per-warp kernel's, whose FP64 pipe is shared by 16 factorisations and sees the extra instructions.)

// The panel arithmetic of the three factorisations (chol_tiled, chol_global, wk_chol).  The matrix factorised is
// cov + adj I = M2 / (n - 1) + adj I inside npar; on the padding the diagonal is 1 and every other entry 0 (M2 is 0 there).
// (v by reference: adapt()'s diagonal loop then loads it only inside npar)
__device__ __forceinline__ double cov_diag(const double &v, int i, int npar, double adj) { return i < npar ? v + adj : 1.0; }
// columns col, col + 1 of matrix row `row`, from the scatter-matrix pair v; in = false (a tile outside the padded upper
// triangle): v as loaded.  (chol_global passes its tile test as `in`: tested at its call site instead, the diagonal tests
// compile to selects, and chol_global and dram_kernel spill differently.)
__device__ __forceinline__ double2 cov_entry(bool in, double2 v, int row, int col, int npar, double invn, double adj)
{
    if (in) {
        v.x *= invn; v.y *= invn;
        if (row == col) v.x = cov_diag(v.x, row, npar, adj);
        if (row == col + 1) v.y = cov_diag(v.y, row, npar, adj);
    }
    return v;
}
// the 8x8 diagonal block of the panel buffer S (row stride ldS); a one-tile-row panel (the last of an odd nt4) is filled out
// with the identity
__device__ __forceinline__ void diag_block(const double *S, int ldS, bool two, double (&A)[8][8])
{
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = r; c < 8; ++c) A[r][c] = (two || c < 4) ? S[r * ldS + c] : (r == c ? 1.0 : 0.0);
}
// forward substitution of one panel column xv against the factored diagonal block (r11[p][r], p < r; reciprocal pivots dinv)
__device__ __forceinline__ void solve_col(const double (&r11)[8][8], const double (&dinv)[8], double (&xv)[8])
{
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        double sacc = xv[r];
#pragma unroll
        for (int p_ = 0; p_ < r; ++p_) sacc = fma(-r11[p_][r], xv[p_], sacc);
        xv[r] = sacc * dinv[r];
    }
}
// the panel at tile rows b0, b0 + 1 (two: b0 + 1 < nt4; ntc = nt4 - b0 tile columns) from S to the tiled gW, zeros below the
// diagonal; thread i0 of NTHR, CG: __stcg stores
template <int NTHR, bool CG>
__device__ __forceinline__ void store_panel(const double *S, int ldS, double *gW, int nt4, int b0, int ntc, bool two, int i0)
{
    const int nT = ntc + (two ? ntc - 1 : 0);
#pragma unroll 1
    for (int e = i0; e < 8 * nT; e += NTHR) {
        const int u = e >> 3, r = (e >> 1) & 3, c2 = e & 1;
        const int h = u < ntc ? 0 : 1, tcl = h ? u - ntc + 1 : u;
        const double2 v = *reinterpret_cast<const double2 *>(S + (4 * h + r) * ldS + 4 * tcl + 2 * c2);
        const bool dg = tcl == h;
        const double2 o = make_double2((dg && 2 * c2 < r) ? 0.0 : v.x, (dg && 2 * c2 + 1 < r) ? 0.0 : v.y);
        double2 *dst = reinterpret_cast<double2 *>(gW + 16 * (size_t)tidx(nt4, b0 + h, b0 + tcl) + 4 * r + 2 * c2);
        if (CG) __stcg(dst, o); else *dst = o;
    }
}

// Factor the 8x8 diagonal block that starts at tile row b0 (one 4x4 tile when it is the last row of an odd nt4): every
// lane of the calling warp factors it redundantly in registers (a chain of 8 dependent rsqrt's, no communication),
// lanes 0-2 write the three tiles back, lane 0 the reciprocal pivots.
__device__ __forceinline__ void chol_diag(int nt4, double *W, int b0)
{
    const int lane = threadIdx.x & 31;
    const bool two = b0 + 1 < nt4;
    double *t00 = W + 16 * tidx(nt4, b0, b0);
    double *t01 = two ? W + 16 * tidx(nt4, b0, b0 + 1) : nullptr;
    double *t11 = two ? W + 16 * tidx(nt4, b0 + 1, b0 + 1) : nullptr;
    double A[8][8];                                       // upper triangle of the block, A[r][c], r <= c
    {
        double q[16];
        ld_tile(t00, q);
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = r; c < 4; ++c) A[r][c] = q[4 * r + c];
        if (two) {
            ld_tile(t01, q);
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) A[r][4 + c] = q[4 * r + c];
            ld_tile(t11, q);
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = r; c < 4; ++c) A[4 + r][4 + c] = q[4 * r + c];
        } else {
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = (r < 4 ? 4 : r); c < 8; ++c) A[r][c] = (r == c) ? 1.0 : 0.0;
        }
    }
    double dinv[8];
    const bool bad = chol8(A, dinv);
    if (lane == 0) {
        double q[16];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) q[4 * r + c] = c >= r ? A[r][c] : 0.0;
        st_tile(t00, q);
#pragma unroll
        for (int j = 0; j < 8; ++j) tc_dinv[j] = dinv[j];
        if (bad) tc_cholfail = 1;
    } else if (lane == 1 && two) {
        double q[16];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) q[4 * r + c] = A[r][4 + c];
        st_tile(t01, q);
    } else if (lane == 2 && two) {
        double q[16];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) q[4 * r + c] = c >= r ? A[4 + r][4 + c] : 0.0;
        st_tile(t11, q);
    }
}

// rank-8 update of trailing tile t = (bi, bj) by the panel at tile rows b0, b0+1: C -= R12(:,bi)' R12(:,bj)
__device__ __forceinline__ void chol_tile_update(int nt4, double *W, int b0, int t, int bi, int bj)
{
    double ai[16], aj[16], c[16];
    ld_tile(W + 16 * t, c);
    ld_tile(W + 16 * tidx(nt4, b0, bi), ai);
    ld_tile(W + 16 * tidx(nt4, b0, bj), aj);
#pragma unroll
    for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
        for (int ii = 0; ii < 4; ++ii)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) c[4 * ii + jj] = fma(-ai[4 * p_ + ii], aj[4 * p_ + jj], c[4 * ii + jj]);
    ld_tile(W + 16 * tidx(nt4, b0 + 1, bi), ai);
    ld_tile(W + 16 * tidx(nt4, b0 + 1, bj), aj);
#pragma unroll
    for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
        for (int ii = 0; ii < 4; ++ii)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) c[4 * ii + jj] = fma(-ai[4 * p_ + ii], aj[4 * p_ + jj], c[4 * ii + jj]);
    st_tile(W + 16 * t, c);
}

// In-place upper Cholesky (R'R = A) of the tiled matrix W (n padded to 4*nt4).  Right-looking, panels of two
// tile rows (8 matrix rows), with one panel of LOOK-AHEAD: per panel (1) the tiles to the right of the (already
// factored) diagonal block are solved column by column (one thread per column); (2) the trailing tiles get the
// rank-8 update in registers by warps 1-7 while warp 0 updates just the NEXT diagonal block and factors it — so
// the chain of dependent rsqrt's never sits on the critical path of the other warps.  Returns false when a
// pivot is not positive.
__device__ __noinline__ bool chol_tiled(int nt4, int oW, bool prof)
{
    double *W = tc_smem + oW;                             // (offset arithmetic on tc_smem compiles to LDS / STS)
    const unsigned short *tab = reinterpret_cast<const unsigned short *>(W + 16 * (nt4 * (nt4 + 1) / 2));
#ifdef TC_SUBPROF
    long long tq = clock64();
#define CHP(i) do { if (threadIdx.x == 0 && prof) { const long long t__ = clock64(); tc_subprof[i] += t__ - tq; tq = t__; } } while (0)
#else
#define CHP(i)
#endif
    const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5;
    const int T = nt4 * (nt4 + 1) / 2;
    if (tid == 0) tc_cholfail = 0;
    __syncthreads();
    if (warp == 0) chol_diag(nt4, W, 0);
    __syncthreads();
    if (tc_cholfail) return false;                        // uniform
#pragma unroll 1
    for (int b0 = 0; b0 + 2 < nt4; b0 += 2) {
        const int bnext = b0 + 2;
        double *t00 = W + 16 * tidx(nt4, b0, b0), *t01 = W + 16 * tidx(nt4, b0, b0 + 1), *t11 = W + 16 * tidx(nt4, b0 + 1, b0 + 1);
        // (1) panel solve R12 = R11^-T A12: thread = one matrix column of the panel (tile column bj, column c)
        {
            double r11[8][8];                             // R11[p][r], p < r (broadcast reads)
#pragma unroll
            for (int p_ = 0; p_ < 8; ++p_)
#pragma unroll
                for (int r = p_ + 1; r < 8; ++r)
                    r11[p_][r] = (p_ < 4) ? (r < 4 ? t00[4 * p_ + r] : t01[4 * p_ + (r - 4)]) : t11[4 * (p_ - 4) + (r - 4)];
            double di[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) di[j] = tc_dinv[j];
#pragma unroll 1
            for (int cc = tid; cc < 4 * (nt4 - bnext); cc += nthr) {
                const int bj = bnext + (cc >> 2), c = cc & 3;
                double *u0 = W + 16 * tidx(nt4, b0, bj) + c, *u1 = W + 16 * tidx(nt4, b0 + 1, bj) + c;
                double xv[8];
#pragma unroll
                for (int r = 0; r < 4; ++r) { xv[r] = u0[4 * r]; xv[4 + r] = u1[4 * r]; }
                solve_col(r11, di, xv);
#pragma unroll
                for (int r = 0; r < 4; ++r) { u0[4 * r] = xv[r]; u1[4 * r] = xv[4 + r]; }
            }
        }
        CHP(13);
        __syncthreads();
        CHP(14);
        // (2) trailing update, with the next diagonal block taken out and factored at once by warp 0
        const int tA = tidx(nt4, bnext, bnext);
        const bool two = bnext + 1 < nt4;
        const int tB = two ? tA + 1 : -1, tC = two ? tidx(nt4, bnext + 1, bnext + 1) : -1;
        // the three tiles of the next diagonal block first, by three warps: 48 outputs x 2 halves of the 8-term dot product
        // (thread pair = one output, combined with a shuffle), so that the serial factorisation below can start at once
        if (tid < 96) {
            const double *p0 = W + 16 * tidx(nt4, b0, bnext), *p1 = W + 16 * tidx(nt4, b0 + 1, bnext);   // panel rows x tile columns bnext, bnext+1:
            const int e = tid >> 1, half = tid & 1;                                                        // adjacent tiles, 16 doubles apart
            const bool on = e < (two ? 48 : 16);
            const int te = e >> 4, ii = (e >> 2) & 3, jj = e & 3;
            const int ci = 16 * (te >> 1) + ii, cj = 16 * ((te + 1) >> 1) + jj;        // (bi, bj) - bnext = (0,0), (0,1), (1,1)
            double *dst = W + 16 * (te == 0 ? tA : (te == 1 ? tB : tC)) + 4 * ii + jj;
            const double *ph = half ? p1 : p0;
            double acc = (on && !half) ? *dst : 0.0;
            if (on) {
#pragma unroll
                for (int p_ = 0; p_ < 4; ++p_) acc = fma(-ph[4 * p_ + ci], ph[4 * p_ + cj], acc);
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            if (on && !half) *dst = acc;
        }
        __syncthreads();
        CHP(6);
        if (warp == 0) {
            chol_diag(nt4, W, bnext);
            CHP(7);
        } else {
#pragma unroll 1
            for (int t = tA + 1 + (tid - 32); t < T; t += nthr - 32) {
                if (t == tB || t == tC) continue;
                chol_tile_update(nt4, W, b0, t, tab[t] >> 8, tab[t] & 0xff);
            }
        }
        CHP(15);
        __syncthreads();
        CHP(5);
        if (tc_cholfail) return false;                    // uniform
    }
    return true;
}

// D = A * B + D on the FP64 tensor cores: A 8x4 (row), B 4x8 (col), D 8x8.  Lane l holds
// A[l>>2][l&3], B[l&3][l>>2] and D[l>>2][2*(l&3) + {0,1}].
__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// ---- TMA bulk copies (cp.async.bulk, global -> shared, completion on an mbarrier) for the big layout.  A tile row of the
// tiled upper-triangular matrices (tiles (r, c0..nt4-1)) is ONE contiguous segment of 128 (nt4 - c0) bytes, so the
// factor streams through a ring of shared-memory stages with one bulk copy per tile row, issued by thread 0; the 8 warps
// consume a stage (full barrier) and release it (empty barrier, one arrival per warp).
#define TMA_MAXST 8
__shared__ __align__(8) unsigned long long tc_mbar[2 * TMA_MAXST];          // full[0..7], empty[0..7]
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *b, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(unsigned long long *b)
{
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *b, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *b)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *b, unsigned parity)
{
    const unsigned addr = smem_u32(b);
    unsigned ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// generic-proxy writes (st.global / st.shared) that a later bulk copy reads or overwrites: order them before the async proxy
__device__ __forceinline__ void fence_async_proxy() { asm volatile("fence.proxy.async;" ::: "memory"); }
// after mbarrier.init by one thread: make the initialised barriers visible to the async proxy (TMA complete_tx, cp.async arrive)
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async;" ::: "memory");
}
// ring bookkeeping: use number g of the ring -> stage g % NS (NS a power of two); producer side (thread 0) and consumer
// side (everyone)
template <int NS>
struct TmaRing {
    static_assert(NS <= TMA_MAXST && (NS & (NS - 1)) == 0, "ring size");
    int o0, sst;                                         // first stage (offset into tc_smem, doubles), stage stride
    __device__ __forceinline__ void init(int o0_, int sst_)
    {
        o0 = o0_; sst = sst_;
        fence_async_proxy();                             // the stages were last written by ordinary stores
        __syncthreads();
        if (threadIdx.x == 0)
        {
            for (int s_ = 0; s_ < NS; ++s_) { mbar_init(tc_mbar + s_, 1); mbar_init(tc_mbar + TMA_MAXST + s_, SPEC); }
            fence_mbar_init();                           // the generic-proxy inits, before the async proxy's complete_tx
        }
        __syncthreads();
    }
    // thread 0: arm use g for `total` bytes (waits until every warp has released the stage's previous use), then copy pieces
    __device__ __forceinline__ void begin(int g, unsigned total) const
    {
        const int s_ = g & (NS - 1);
        if (g >= NS) mbar_wait(tc_mbar + TMA_MAXST + s_, (unsigned)((g / NS - 1) & 1));
        mbar_expect_tx(tc_mbar + s_, total);
    }
    __device__ __forceinline__ void copy(int g, int off, const double *src, unsigned bytes) const
    {
        const int s_ = g & (NS - 1);
        bulk_g2s(tc_smem + o0 + s_ * sst + off, src, bytes, tc_mbar + s_);
    }
    __device__ __forceinline__ void issue(int g, const double *src, unsigned bytes) const { begin(g, bytes); copy(g, 0, src, bytes); }
    __device__ __forceinline__ int acquire(int g) const  // -> offset of the stage into tc_smem (doubles)
    {
        const int s_ = g & (NS - 1);
        mbar_wait(tc_mbar + s_, (unsigned)((g / NS) & 1));
        return o0 + s_ * sst;
    }
    __device__ __forceinline__ void release(int g) const
    {
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(tc_mbar + TMA_MAXST + (g & (NS - 1)));
    }
    __device__ __forceinline__ void fini() const         // after a __syncthreads that follows the last release
    {
        if (threadIdx.x == 0)
            for (int s_ = 0; s_ < NS; ++s_) { mbar_inval(tc_mbar + s_); mbar_inval(tc_mbar + TMA_MAXST + s_); }
    }
};

// The same ring filled COOPERATIVELY: every thread copies 16-byte pieces with cp.async.cg (LDGSTS) and its copies arrive on the
// stage's full barrier (cp.async.mbarrier.arrive.noinc; 256 arrivals complete a stage).  Used where a stage is made of many
// separate segments — chol_global's per-row pieces of a few KB: a bulk copy costs ~350-650 cycles EACH almost independently of
// its size (scripts/stream_bench.cu), LDGSTS has no per-copy cost.  (Measured: at equal stage sizes the two fill methods give
// the same factorisation time — what counts is the number of stage hand-overs, ~1 k cycles each; hence few, large stages.)
template <int NS>
struct CoopRing {
    static_assert(NS <= TMA_MAXST && (NS & (NS - 1)) == 0, "ring size");
    int o0, sst;
    __device__ __forceinline__ void init(int o0_, int sst_)
    {
        o0 = o0_; sst = sst_;
        __syncthreads();
        if (threadIdx.x == 0)
        {
            for (int s_ = 0; s_ < NS; ++s_) { mbar_init(tc_mbar + s_, DRAM_THREADS); mbar_init(tc_mbar + TMA_MAXST + s_, SPEC); }
            fence_mbar_init();
        }
        __syncthreads();
    }
    // every thread: wait until every warp has released the stage's previous use
    __device__ __forceinline__ void begin(int g) const
    {
        if (g >= NS) mbar_wait(tc_mbar + TMA_MAXST + (g & (NS - 1)), (unsigned)((g / NS - 1) & 1));
    }
    // every thread: its share of one contiguous segment of `n16` 16-byte pieces -> stage offset `off` (doubles)
    __device__ __forceinline__ void copy(int g, int off, const double *src, int n16) const
    {
        const unsigned dst = smem_u32(tc_smem + o0 + (g & (NS - 1)) * sst + off);
        for (int i = threadIdx.x; i < n16; i += DRAM_THREADS)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (unsigned)i), "l"(src + 2 * i) : "memory");
    }
    __device__ __forceinline__ void commit(int g) const
    {
        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(tc_mbar + (g & (NS - 1)))) : "memory");
    }
    __device__ __forceinline__ int acquire(int g) const  // -> offset of the stage into tc_smem (doubles)
    {
        const int s_ = g & (NS - 1);
        mbar_wait(tc_mbar + s_, (unsigned)((g / NS) & 1));
        return o0 + s_ * sst;
    }
    __device__ __forceinline__ void release(int g) const
    {
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(tc_mbar + TMA_MAXST + (g & (NS - 1)));
    }
    __device__ __forceinline__ void fini() const         // after a __syncthreads that follows the last release
    {
        if (threadIdx.x == 0)
            for (int s_ = 0; s_ < NS; ++s_) { mbar_inval(tc_mbar + s_); mbar_inval(tc_mbar + TMA_MAXST + s_); }
    }
};

// CALL with the compile-time constant N_ = n_ (1 .. 7; any other n_: nothing)
#define DISPATCH_1_7(n_, CALL)                                                                              \
    switch (n_) {                                                       /* warp-uniform */                  \
    case 7: { constexpr int N_ = 7; CALL; } break;                                                          \
    case 6: { constexpr int N_ = 6; CALL; } break;                                                          \
    case 5: { constexpr int N_ = 5; CALL; } break;                                                          \
    case 4: { constexpr int N_ = 4; CALL; } break;                                                          \
    case 3: { constexpr int N_ = 3; CALL; } break;                                                          \
    case 2: { constexpr int N_ = 2; CALL; } break;                                                          \
    case 1: { constexpr int N_ = 1; CALL; } break;                                                          \
    default: break;                                                                                         \
    }

// chol_global, accumulation over `nr` staged tile rows (stride `rs` doubles) for the NM column blocks of this warp: per row one
// A fragment and NM B fragments (constant offsets: block m sits 256 m doubles after the warp's first block) + NM MMAs.
// Lanes whose tile column lies beyond the matrix read whatever follows the row (finite or not): those are columns / rows
// of the 8x8 outputs that nobody reads.
template <int NM>
__device__ __forceinline__ void cg_accumulate(int oa, int ob, int nr, int rs, double (&acc)[7][2])
{
    // few column blocks = few independent MMA chains: split the rows over KS accumulator sets so that 4+ chains are in flight
    constexpr int KS = NM >= 4 ? 1 : (NM >= 2 ? 2 : 4);
    constexpr int U = KS > 1 ? KS : 2;
    double loc[KS][NM][2];
#pragma unroll
    for (int s_ = 0; s_ < KS; ++s_)
#pragma unroll
        for (int m = 0; m < NM; ++m) { loc[s_][m][0] = s_ == 0 ? acc[m][0] : 0.0; loc[s_][m][1] = s_ == 0 ? acc[m][1] : 0.0; }
#pragma unroll 1
    for (int q = 0; q < nr; q += U, oa += U * rs, ob += U * rs) {
        double av[U], bv[U][NM];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const bool on = q + u < nr;                                             // warp-uniform
            av[u] = on ? tc_smem[oa + u * rs] : 0.0;
#pragma unroll
            for (int m = 0; m < NM; ++m) bv[u][m] = on ? tc_smem[ob + u * rs + 256 * m] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int m = 0; m < NM; ++m) dmma_m8n8k4(loc[u % KS][m][0], loc[u % KS][m][1], av[u], bv[u][m]);   // unconditional: a
    }                                                                                                           // conditional mma.sync costs a WARPSYNC
#pragma unroll
    for (int m = 0; m < NM; ++m) {
        double s0 = loc[0][m][0], s1 = loc[0][m][1];
#pragma unroll
        for (int s_ = 1; s_ < KS; ++s_) { s0 += loc[s_][m][0]; s1 += loc[s_][m][1]; }
        acc[m][0] = s0; acc[m][1] = s1;
    }
}

// Left-looking blocked Cholesky THROUGH HBM/L2, for proposal factors too large for shared memory (big layout):
// R'R = gA * invn + qcovadj I (identity on the padding), gA and the result gW in the 4x4-tile layout of chol_tiled.
// Panels of two tile rows (8 matrix rows).  Per panel:
//  (1) S = A(panel rows, columns >= panel) - sum over the tile rows above of R(row, panel cols)' R(row, cols) on the FP64
//      tensor cores: one mma.sync m8n8k4 per tile row above per 8-column block.  The tile rows above stream through
//      the cooperative ring (a stage = up to CG_RPS tile rows of 128 (nt4 - b0) bytes each, two stages ahead); a warp owns the column
//      blocks w, w+8, .. (<= CG_MAXB), its accumulators stay in registers for the whole panel; fragment reads from
//      a stage are conflict-free (the 32 B elements of a warp are two adjacent tiles);
//  (2) warp 0 factors the 8x8 diagonal block in registers; (3) the rest of the panel is solved one column per thread
//      while the first tile rows of the NEXT panel are already in flight; (4) the panel is written to gW.
// S = shared-memory buffer [8][8 ceil(nt4 / 2) + 4] at `ws`, the ring stages after it (`ws_doubles` in all).  Returns
// false when a pivot is not positive (gW is then garbage; the caller keeps the old R).  Reads 11 MB from L2 at
// npar = 407 (a right-looking sweep would move 34 MB).
#define CG_MAXB 7          // column blocks per warp: npar <= 8 * 8 * 7 = 448
#define CG_NS 4            // ring stages (a power of two): few, large stages — the hand-over of a stage costs ~1 k cycles
#define CG_RPS 32          // tile rows per stage, at most
__device__ __noinline__ bool chol_global(int nt4, int npar, const double *gA, double invn, double qcovadj, double *gW,
                                         int o_ws, int ws_doubles)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ar = lane >> 2, ak = lane & 3;
    const int ldS = 8 * ((nt4 + 1) >> 1) + 4;
    const int th = ar >> 2, inner = 4 * ak + (ar & 3);
    double *S = tc_smem + o_ws;                        // (offset arithmetic on tc_smem compiles to LDS / STS)
    CoopRing<CG_NS> ring;
    {
        // CG_NS stages of equal capacity; a stage holds as many tile rows of the current panel as fit (<= CG_RPS); 32 doubles of
        // slack after the last one (cg_accumulate reads up to two tiles past a row)
        const int o = (8 * ldS + 1) & ~1;
        ring.init(o_ws + o, ((ws_doubles - o - 32) / CG_NS) & ~1);
    }
    if (tid == 0) tc_cholfail = 0;
#ifdef TC_SUBPROF
    long long tq = clock64();
#define CGP(i) do { if (tid == 0 && blockIdx.x == 0) { const long long t__ = clock64(); tc_subprof[i] += t__ - tq; tq = t__; } } while (0)
#else
#define CGP(i)
#endif
    int gi = 0, gc = 0, si = 0;        // ring uses issued / consumed; stages of the current panel already issued (uniform)
    bool ok = true;
    // every thread: its share of stage u of the panel at b0 (rows u rps .. of the tile rows above, each 16 ntc doubles)
#define CG_ISSUE(b0_, ntc_, rps_, u_)                                                                       \
    {                                                                                                       \
        const int r0__ = (u_) * (rps_), nr__ = min((rps_), (b0_) - r0__);                                     \
        ring.begin(gi);                                                                                     \
        for (int q__ = 0; q__ < nr__; ++q__)                                                                \
            ring.copy(gi, 16 * (ntc_) * q__, gW + 16 * (size_t)tidx(nt4, r0__ + q__, (b0_)), 8 * (ntc_));   \
        ring.commit(gi);                                                                                    \
        ++gi;                                                                                               \
    }
#pragma unroll 1
    for (int b0 = 0; b0 < nt4; b0 += 2) {
        const bool two = b0 + 1 < nt4;
        const int ntc = nt4 - b0, nb = (ntc + 1) >> 1;
        const int rps = max(1, min(CG_RPS, ring.sst / (16 * ntc))), nst = (b0 + rps - 1) / rps;
        // (1) accumulate over the tile rows 0 .. b0-1
        {
            double acc[CG_MAXB][2];
#pragma unroll
            for (int m = 0; m < CG_MAXB; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; }
            while (si < nst && si < CG_NS - 2) { CG_ISSUE(b0, ntc, rps, si) ++si; }
            const int nmine = nb > warp ? (nb - warp + SPEC - 1) / SPEC : 0;          // column blocks warp, warp + 8, .. < nb
            // the covariance entries of the panel are needed after the accumulation: pull them into L2 now
            if (lane < 2 * nmine) {
                const int j = warp + SPEC * (lane >> 1), tcn = b0 + 2 * j, trp = b0 + (lane & 1);
                if (trp < nt4 && trp <= tcn)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(gA + 16 * (size_t)tidx(nt4, trp, tcn)));
                if (trp < nt4 && tcn + 1 < nt4)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(gA + 16 * (size_t)tidx(nt4, trp, tcn + 1)));
            }
#pragma unroll 1
            for (int u = 0; u < nst; ++u) {
                // issued CG_NS - 2 uses ahead: the stage being re-armed was released an iteration ago, so thread 0 does not
                // hold the other warps in lock step
                if (si < nst) { CG_ISSUE(b0, ntc, rps, si) ++si; }
                const int nr = min(rps, b0 - u * rps);
                const int pa = ring.acquire(gc) + 16 * th + inner, pb = pa + 32 * warp;
                DISPATCH_1_7(nmine, cg_accumulate<N_>(pa, pb, nr, 16 * ntc, acc))
                ring.release(gc);
                ++gc;
            }
            CGP(13);
            // S = A - acc: lane holds row ar, columns 2 ak, 2 ak + 1 of each of its blocks (all loads first: one L2 round trip)
            const int tr = b0 + th, rin = ar & 3, row = 4 * tr + rin;
            double2 vin[CG_MAXB];
#pragma unroll
            for (int m = 0; m < CG_MAXB; ++m) {
                const int j = warp + SPEC * m, tcn = b0 + 2 * j + (ak >> 1);
                vin[m] = make_double2(0.0, 0.0);
                if (j < nb && tr <= tcn && tcn < nt4 && tr < nt4)
                    vin[m] = __ldcg(reinterpret_cast<const double2 *>(gA + 16 * (size_t)tidx(nt4, tr, tcn) + 4 * rin + 2 * (ak & 1)));
            }
#pragma unroll
            for (int m = 0; m < CG_MAXB; ++m) {
                const int j = warp + SPEC * m;
                if (j >= nb) continue;
                const int tcn = b0 + 2 * j + (ak >> 1), col = 4 * tcn + 2 * (ak & 1);
                const double2 v = cov_entry(tr <= tcn && tcn < nt4 && tr < nt4, vin[m], row, col, npar, invn, qcovadj);
                *reinterpret_cast<double2 *>(S + ar * ldS + 8 * j + 2 * ak) = make_double2(v.x - acc[m][0], v.y - acc[m][1]);
            }
        }
        __syncthreads();
        CGP(14);
        // (2) the diagonal block
        if (warp == 0) {
            double A[8][8], dinv[8];
            diag_block(S, ldS, two, A);
            const bool bad = chol8(A, dinv);
            if (lane == 0) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int c = r; c < 8; ++c) S[r * ldS + c] = A[r][c];
#pragma unroll
                for (int j = 0; j < 8; ++j) tc_dinv[j] = dinv[j];
                if (bad) tc_cholfail = 1;
            }
        }
        __syncthreads();
        CGP(7);
        if (tc_cholfail) { ok = false; break; }                       // uniform; nothing is in flight here
        // the first stages of the next panel that hold only final rows (< b0) start streaming now
        si = 0;
        if (b0 + 2 < nt4) {
            const int ntc2 = ntc - 2, rps2 = max(1, min(CG_RPS, ring.sst / (16 * ntc2)));
            while ((si + 1) * rps2 <= b0 && si < CG_NS - 2) { CG_ISSUE(b0 + 2, ntc2, rps2, si) ++si; }
        }
        // (3) panel solve R12 = R11^-T A12: thread = one matrix column
        if (4 * ntc > 8) {
            double r11[8][8], di[8];
#pragma unroll
            for (int p_ = 0; p_ < 8; ++p_)
#pragma unroll
                for (int r = p_ + 1; r < 8; ++r) r11[p_][r] = S[p_ * ldS + r];
#pragma unroll
            for (int j = 0; j < 8; ++j) di[j] = tc_dinv[j];
#pragma unroll 1
            for (int cc = 8 + tid; cc < 4 * ntc; cc += DRAM_THREADS) {
                double xv[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) xv[r] = S[r * ldS + cc];
                solve_col(r11, di, xv);
#pragma unroll
                for (int r = 0; r < 8; ++r) S[r * ldS + cc] = xv[r];
            }
            __syncthreads();
        }
        // (4) the panel goes to gW
        store_panel<DRAM_THREADS, false>(S, ldS, gW, nt4, b0, ntc, two, tid);
        __syncthreads();                                          // the next panels read these tiles back from L2 (cp.async.cg)
        CGP(15);
    }
#undef CG_ISSUE
#undef CGP
    __syncthreads();
    ring.fini();
    return ok;
}

// per-candidate-step record of a round: out-of-bounds bits and prior sums of the two proposals (shared memory)
struct Cand { double pr1, pr2; int oob, pad; };
// outcome of one step under the hypothesis "every earlier step of the round rejected" (registers of lane = step)
struct StepOut { double ssn, prin; int acc, fl, nev, noob; };

// ---- chain book-keeping shared by dram_kernel and dram_warp_kernel (tc_warp.cuh)

// Rows a fit stores with store_chain, keeping every thin-th: chain rows first_row + j thin (j < thin_nkeep), s2chain rows j thin
// (j < thin_ns2).  Ceilings as (x - 1) / thin + 1: no overflow at thin = 2^31 - 1.
static int thin_nkeep(int nsimu, int n_burn, int thin) { return (nsimu - n_burn) / thin + 1; }
__host__ __device__ inline int thin_ns2(int nsimu, int thin) { return (nsimu - 1) / thin + 1; }

// Constants of a chain that both samplers derive their per-step arithmetic from
struct ChainConsts {
    unsigned long long uid;                             // Philox identity
    int first_row, nkeep;                               // first row of the summaries and of the stored chain (n_burn - 1), rows stored
    double inv_dr, adascale, chi_d, chi_c;              // chi_d, chi_c: Marsaglia-Tsang constants of chi2(N0 + 2 N)
};
__device__ __forceinline__ ChainConsts chain_consts(const RunArgs &a, int ch, int N)
{
    ChainConsts k;
    k.uid = a.chain_uid ? a.chain_uid[ch] : (unsigned long long)ch;
    k.first_row = a.n_burn - 1;
    k.nkeep = a.nkeep;
    k.inv_dr = 1.0 / a.drscale;
    k.adascale = a.adascale > 0.0 ? a.adascale : 2.4 / sqrt((double)(7 + N));
    chi2_consts(a.N0 + 2.0 * N, k.chi_d, k.chi_c);
    return k;
}

// Phase clocks: pc[i] of the tally is returned as counter TC_CNT_CYCLES0 + i; include/tcmcmc.h says what each sampler times in
// each slot (PH_COMMIT: dram_kernel, PH_WAIT, PH_RAND, PH_SCATTER, PH_FACTOR: dram_warp_kernel, PH_EVAL: its WK_SUBPROF build)
enum { PH_GEN = 0, PH_STEPS = 1, PH_COMMIT = 2, PH_WAIT = 2, PH_RAND = 3, PH_SCATTER = 4, PH_ADAPT = 5, PH_FACTOR = 6, PH_EVAL = 7 };

// What a chain counts and sums, in shared memory (one thread writes each field); parked with the chain between slices
struct Tally {
    long long n_ss, n_acc1, n_acc2, n_oob, n_adapt, n_cholfail, n_dr;   // counters TC_CNT_SS_EVALS .. TC_CNT_DR_TRIES
    long long n_spec;                                   // dram_kernel: evaluations including the discarded speculative ones
    long long rej, reju;                                // rejected steps: in all, since the last adaptation
    double s2sum, s2cnt;                                // s2chain over ALL rows (TranscriptionCycleMCMC.m:302-303): sum s2, rows
    double sqmean, sqM2;                                // ... mean of sqrt(s2) and sum of squared deviations from it (tally_s2)
    double wcnt, cov_n;                                 // rows in the Welford summaries, rows in the covariance
    long long pc[8];                                    // phase clocks (PH_*)
};

// Fold nb more rows of s2chain into the tally: sum s2b of their s2, mean mb and sum of squared deviations M2b of their sqrt(s2),
// merged with Chan et al.'s update.  std(sqrt(s2chain),1) from two running sums, sqrt(E[s2] - E[sqrt(s2)]^2), cancels: with
// sigma2 fixed it is ~1e-6 sqrt(sigma2) after 2e5 rows instead of 0.  One thread.  Out of line: inlined, it costs
// dram_warp_kernel (at its 128-register cap) spill traffic on every step.
__device__ __noinline__ void tally_s2(Tally &t, double nb, double s2b, double mb, double M2b)
{
    const double n = t.s2cnt + nb, d = mb - t.sqmean, f = nb * tc_rcp(n);
    t.sqmean = fma(d, f, t.sqmean);
    t.sqM2 += fma(d * d, t.s2cnt * f, M2b);
    t.s2sum += s2b; t.s2cnt = n;
}

// The rules both samplers decide and count by, each written once.  They take and return scalars (a pointer into shared memory
// would make every access generic, §3 of DESIGN.md) and keep the association the replay tests pin bit for bit.

// reciprocal prior width: an infinite width is a flat prior
__device__ __forceinline__ double prior_inv(double sg) { return isinf(sg) ? 0.0 : 1.0 / sg; }

// Slice seg of a chain: steps [k, k_end) (row 0 is x0, no step), and the first step whose isimu is a multiple of adaptint,
// which triggers an adaptation (kept as a running value afterwards: an integer division per round is ~40 dependent instructions)
struct Slice { int k, k_end, next_adapt; bool last; };
__device__ __forceinline__ Slice slice_of(const RunArgs &a, int seg)
{
    Slice s;
    s.k = seg == 0 ? 1 : seg * a.seglen;
    s.k_end = min(a.nsimu, (seg + 1) * a.seglen);
    s.last = s.k_end >= a.nsimu;
    s.next_adapt = a.adaptint > 0 ? ((s.k + a.adaptint) / a.adaptint) * a.adaptint : 0x7fffffff;
    return s;
}

// 1 / (N0 S20 + ss): a step that sees sigma2 = (N0 S20 + ss) / chi2 uses 1 / sigma2 = chi2 * rden_of(ss)
__device__ __forceinline__ double rden_of(double n0s20, double ss) { return tc_rcp(n0s20 + ss); }
// sigma2 of a row (the draw made from the row's ss and chi2), or the fixed sigma2 without updatesigma
__device__ __forceinline__ double row_sigma2(int updatesigma, double n0s20, double ss, double chi2, double sig2)
{
    return updatesigma ? (n0s20 + ss) * tc_rcp(chi2) : sig2;
}
// Stage 1, decided in the log domain: a12 = exp(x12) > u1 <=> x12 >= 0 or x12 > log u1 (no exponential); x12 goes on to resolve_dr
__device__ __forceinline__ bool stage1_accepts(double ss1, double ss, double is2, double pr1, double pri, double logu, double &x12)
{
    x12 = -0.5 * ((ss1 - ss) * is2 + pr1 - pri);
    return x12 >= 0.0 || x12 > logu;
}

// A run (the rows [r0, r1), all equal to the state) closes: the rows it adds to the Welford summaries (those >= first_row),
// and whether it is one more distinct row of the covariance block
__device__ __forceinline__ int run_rows(int r0, int r1, int first_row) { return max(0, r1 - max(r0, first_row)); }
// The stored rows of a run's m_w summarised rows [rs, rs + m_w), rs >= first_row, when every thin-th row is stored: chain rows
// j0 .. j0 + return value - 1, the rows first_row + j thin among them.  Two divisions per run, computed before the run
// writer's per-parameter loop; none per row.
//
// The samplers are compiled twice, THIN = false (every row; thin = 1 or no stored rows) and THIN = true (thin > 1): the run
// writers sit on the path of every accept, and the code and registers of the thinned writes cost config 2 ~0.7 % of kernel
// time (B200) even where they never run.
__device__ __forceinline__ int kept_rows(int rs, int m_w, int first_row, int thin, int &j0)
{
    const int x = rs - first_row;
    j0 = x == 0 ? 0 : (x - 1) / thin + 1;
    return m_w > 0 ? (x + m_w - 1) / thin - j0 + 1 : 0;
}
__device__ __forceinline__ bool run_distinct(int do_cov, int r0, int r1) { return do_cov && r1 > r0; }
// Welford weights of m_w rows folded into wcnt rows (mean += d f1, M2 += d^2 f2) through ONE reciprocal (two quotients were
// ~300 cycles at the head of every accept)
__device__ __forceinline__ void welford_weights(double wcnt, int m_w, double &f1, double &f2)
{
    const double nn = wcnt + m_w, rnn = m_w > 0 ? tc_rcp(nn) : 0.0;
    f1 = m_w * rnn; f2 = wcnt * m_w * rnn;
}

// Rejection rate the burn-in scaling looks at after step k: since the start (burnin_cumulative) or since the last adaptation
__device__ __forceinline__ double adapt_rate(const RunArgs &a, long long rej, long long reju, int k)
{
    return a.burnin_cumulative ? (double)rej / k : (double)reju / a.adaptint;
}
// Burn-in scales R by this factor (1: R unchanged)
__device__ __forceinline__ double burnin_factor(double rate, double burnin_scale)
{
    double f = 1.0;
    if (rate > 0.95) f = 1.0 / burnin_scale;
    else if (rate < 0.05) f = burnin_scale;
    return f;
}
// The covariance block closed at isimu, when the covariance holds cov_n rows: its m rows (adaptint; rows 0 .. isimu-1 for the
// first block, which is 2 rows when adaptint = 1), the rows of its scatter update (ndist distinct rows + Chan's mean-shift row,
// once there is a covariance) with the weight fcorr of the mean-shift row, and the share `shift` of the block's mean in the new
// covariance mean
struct CovBlock { int m, nrows; double fcorr, shift; };
__device__ __forceinline__ CovBlock cov_block(int isimu, double cov_n, int ndist)
{
    CovBlock b;
    b.m = isimu - (int)cov_n;
    b.fcorr = cov_n * b.m / (cov_n + b.m);
    b.nrows = ndist + (cov_n > 0.0 ? 1 : 0);
    b.shift = b.m / (cov_n + b.m);
    return b;
}
// The tally after the adaptation at isimu = k that returned rc (1: new factor, 2: Cholesky failed); the caller starts a new
// run and block at k, and leaves the diagonal proposal when rc = 1
__device__ __forceinline__ void after_adapt(Tally &t, int do_cov, int k, int rc)
{
    if (do_cov) t.cov_n = k;
    if (rc == 1) ++t.n_adapt;
    else if (rc == 2) ++t.n_cholfail;
    t.reju = 0;
}

// A chain between two time slices: its slot of gState (state_doubles(ld) doubles) holds this record, then the vectors
// x | wmean | wM2 | rdiag, ld doubles each (dram_warp_kernel keeps the last three there all along).  16-byte aligned: the vectors
// after it stay aligned, and it moves through L2 as 16-byte words.
struct __align__(16) ParkedChain {
    double ss, pri, sigma2;
    double rsig;                                        // 1 / sigma2 as the next step sees it (chi2 of the last row * rden)
    int r_diag;
    int bad0;                                           // ss(x0) was not finite (dram_warp_kernel: the later slices skip the chain)
    Tally t;
};
constexpr int ST_VEC0 = sizeof(ParkedChain) / sizeof(double);
__host__ __device__ inline int state_doubles(int ld) { return ST_VEC0 + 4 * ld; }

// the next slice may run on another SM: past L1 both ways
__device__ __forceinline__ void park_chain(double *gst, const ParkedChain &p)
{
    const double2 *src = reinterpret_cast<const double2 *>(&p);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(ParkedChain) / 16); ++i) __stcg(reinterpret_cast<double2 *>(gst) + i, src[i]);
}
__device__ __forceinline__ ParkedChain resume_chain(const double *gst)
{
    ParkedChain p;
    double2 *dst = reinterpret_cast<double2 *>(&p);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(ParkedChain) / 16); ++i) dst[i] = __ldcg(reinterpret_cast<const double2 *>(gst) + i);
    return p;
}

// The optional per-row outputs of row r: s2chain (store_chain; THIN: rows 0, thin, 2 thin, ..), flags and sschain (replay /
// parity harness; every row)
template <bool THIN>
__device__ __forceinline__ void store_row(const RunArgs &a, int ch, int r, double s2, int fl, double ss)
{
    const size_t g = (size_t)ch * a.nsimu + r;
    if (THIN) {
        const int j = r / a.thin;
        if (a.store_chain && a.s2chain && j * a.thin == r) a.s2chain[(size_t)ch * thin_ns2(a.nsimu, a.thin) + j] = s2;
    } else if (a.store_chain && a.s2chain) {
        a.s2chain[g] = s2;
    }
    if (a.flags) a.flags[g] = fl;
    if (a.sschain) a.sschain[g] = ss;
}
// Row 0 = x0 with a finite ss0: s2 = sigma2_0 (TranscriptionCycleMCMC.m:259), no flags.  One thread.
template <bool THIN>
__device__ __forceinline__ void record_row0(const RunArgs &a, int ch, double ss0, Tally &t)
{
    tally_s2(t, 1.0, a.sigma2_0, sqrt(a.sigma2_0), 0.0);
    store_row<THIN>(a, ch, 0, a.sigma2_0, 0, ss0);
}

// a Welford vector: shared memory (dram_kernel) or L2 (dram_warp_kernel: written by other SMs, so past L1)
__device__ __forceinline__ double ld_welford(const double *p) { return __isGlobal(p) ? __ldcg(p) : *p; }
// Outputs of a finished chain (TranscriptionCycleMCMC.m:286-303): mean / std of the stored rows by the threads i0 = 0 .. nthr-1,
// sig and the counters by thread i0 = 0.  slot7 = counter TC_CNT_CYCLES0 + 7, the one slot whose meaning the caller decides.
// A chain whose ss(x0) is not finite (bad0) reports zeros and status 1.
__device__ void write_outputs(const RunArgs &a, int ch, int npar, const double *wmean, const double *wM2, const Tally &t,
                              long long slot7, bool bad0, int i0, int nthr)
{
    const double wcnt = t.wcnt;
#pragma unroll 1
    for (int i = i0; i < npar; i += nthr) {
        if (a.mean) a.mean[(size_t)ch * a.ld + i] = bad0 ? 0.0 : ld_welford(wmean + i);
        if (a.std) a.std[(size_t)ch * a.ld + i] = (!bad0 && wcnt > 0) ? sqrt(ld_welford(wM2 + i) / wcnt) : 0.0;
    }
    if (i0 != 0) return;
    if (a.sig) {
        // sqrt(mean(s2chain)); std(sqrt(s2chain),1) = sqrt(M2 / rows) of the running (mean, M2) of sqrt(s2)   (:302-303)
        a.sig[2 * (size_t)ch] = bad0 ? 0.0 : sqrt(t.s2sum / t.s2cnt);
        a.sig[2 * (size_t)ch + 1] = bad0 ? 0.0 : sqrt(t.sqM2 / t.s2cnt);
    }
    if (a.counters) {
        long long *c = a.counters + (size_t)ch * TC_NCOUNTERS;
        c[TC_CNT_SS_EVALS] = t.n_ss; c[TC_CNT_ACC_STAGE1] = t.n_acc1; c[TC_CNT_ACC_STAGE2] = t.n_acc2;
        c[TC_CNT_OUT_OF_BOUNDS] = t.n_oob; c[TC_CNT_ADAPTATIONS] = t.n_adapt;
        c[TC_CNT_CHOL_FAIL] = t.n_cholfail; c[TC_CNT_DR_TRIES] = t.n_dr; c[TC_CNT_STATUS] = bad0 ? 1 : 0;
        for (int i = 0; i < 7; ++i) c[TC_CNT_CYCLES0 + i] = t.pc[i];
        c[TC_CNT_CYCLES0 + 7] = slot7;
    }
}

// Mutable chain state (uniform across the CTA) in shared memory.  Written by thread 0 in the commit phase
// (between the post-speculation barrier and the end-of-round barrier), read by everyone at the top of a round.
// In the commit phase thread 0 and lane 0 of warp SPEC-1 write disjoint fields.
struct ChainState {
    double ss, pri, sigma2;
    double rden, rsig;                                  // 1 / (N0 S20 + ss) and 1 / sigma2 as the next step sees it (= chi2 of the last row * rden)
    int r_diag, bad0, run_r0, ndist;
    Tally t;
    long long tprev;
};

// Immutable per-chain context, built once in shared memory so that the out-of-line phases below
// (kept out of line to keep the hot loop inside the instruction cache) can share it.
struct ChainCtx {
    int N, npar, npad, ld, slot_sz, s1, wsz, ch, ring_mask, uni;
    double blk[4];                                      // uni: common lo, hi, mu, 1/sig of the parameters >= 7 (the dR block)
    ChainConsts cc;
    SmemCell cv;
    int o_x, o_ring, o_U;                               // offsets (doubles) into tc_smem
    int o_lo, o_pinv, o_wmean, o_wM2, o_mb;             // hot per-parameter vectors by offset (tc_smem + offset compiles to LDS/STS, the
                                                        // pointers below to generic accesses); o_lo < 0: bounds / prior means in HBM (big layout)
    double *ring, *x, *lo, *hi, *mu, *pinv, *wmean, *wM2, *rdiag, *mb, *dm, *U;
    double *gRb, *gM2, *gRows, *gWts, *cmean;
    __device__ __forceinline__ int slot_o(int step) const { return o_ring + (step & ring_mask) * slot_sz; }
    __device__ __forceinline__ int slot_i(int step) const { return o_ring + (step & ring_mask) * slot_sz + 1; }   // stage-1 increments (stage 2: + s1)
    __device__ __forceinline__ double *slot_d(int step) const { return tc_smem + o_ring + (step & ring_mask) * slot_sz; }
    __device__ __forceinline__ double *slot_sc(int step) const { return tc_smem + o_ring + (step & ring_mask) * slot_sz + (slot_sz - 8); }
};

// The chain rows [r0, r1) all equal the current state x (a run: the accept at row r0, then rejections).
// Fold the run into the summaries (Welford with multiplicity; rows >= n_burn-1 only), the optional chain
// storage, and the distinct-row buffer of the current covariance block (row + weight); then, when
// so >= 0, move the state: x += increment at tc_smem[so + i].  Every thread owns the indices i = tid, tid+256, ..
// so the whole thing is one pass.
template <bool THIN>
__device__ __noinline__ void flush_run(const RunArgs &a, const ChainCtx &cx, int r0, int r1, double wcnt, int ndist, int so, int t0)
{
    // threads t0 .. DRAM_THREADS-1 take part (t0 = 32 at an accept: warp 0 writes the per-row scalars meanwhile)
    const int tid = (int)threadIdx.x - t0, nthr = DRAM_THREADS - t0, npar = cx.npar;
    if (tid < 0) return;
    const int m_c = r1 - r0, rs = max(r0, cx.cc.first_row), m_w = run_rows(r0, r1, cx.cc.first_row);
    const bool cov = run_distinct(a.do_cov, r0, r1);
    double f1, f2;
    welford_weights(wcnt, m_w, f1, f2);
    double *grow = cov ? cx.gRows + (size_t)ndist * cx.ld : nullptr;
    int j0 = rs - cx.cc.first_row, nkr = m_w;
    if (THIN && a.store_chain && a.chain) nkr = kept_rows(rs, m_w, cx.cc.first_row, a.thin, j0);
    const int ox = cx.o_x, owm = cx.o_wmean, ow2 = cx.o_wM2, omb = cx.o_mb;
#pragma unroll 1
    for (int i = tid; i < npar; i += nthr) {
        const double xo = tc_smem[ox + i];
        if (m_w > 0) {
            const double wm = tc_smem[owm + i], d1 = xo - wm;
            tc_smem[owm + i] = fma(d1, f1, wm);
            tc_smem[ow2 + i] = fma(d1 * d1, f2, tc_smem[ow2 + i]);
            if (a.store_chain && a.chain) {
                double *dst = a.chain + ((size_t)cx.ch * cx.cc.nkeep + j0) * cx.ld + i;
#pragma unroll 1
                for (int r = 0; r < nkr; ++r) dst[(size_t)r * cx.ld] = xo;
            }
        }
        if (cov) {
            grow[i] = xo;
            tc_smem[omb + i] = fma((double)m_c, xo, tc_smem[omb + i]);
        }
        if (so >= 0) tc_smem[ox + i] = xo + tc_smem[so + i];
    }
    if (cov && tid == 0) cx.gWts[ndist] = (double)m_c;
}

#define GEN_M 8
// Big layout: the increments z1 R and z2 R/drscale of the GEN_M new steps (rows of Z = the ring slots) with R streamed through
// the TMA ring: one bulk copy per tile row kk of R (tiles (kk, kk..nt4-1), 128 (nt4 - kk) bytes), consecutive tile rows
// packed into a stage as long as they fit (<= GENB_RPS), so the mbarrier round trip (~90 cycles each way) is paid per stage
// of 2-8 rows.  Row kk is k-step kk of every column tile: warp w owns the column tiles w, w+8, .. (<= GENB_MAXT) and keeps
// their accumulators in registers for the whole pass (2 x GENB_MAXT independent MMA chains), so R crosses the SM once per
// call and no lane issues per-element copies; the B fragment of tile column bj sits 16 (bj - kk) doubles into the row.
#define GENB_MAXT 7        // column tiles per warp: npar <= 8 * 8 * 7 = 448
#define GENB_NS 4          // ring stages
#define GENB_RPS 32        // tile rows per stage, at most (the short rows at the bottom of the triangle pack many to a stage)
// one k-step for the NA column tiles that still have rows: accumulator j belongs to the j-th tile from the TOP (so the live
// ones are always a prefix and the code is straight-line: a conditional mma.sync costs a WARPSYNC each); `bt` = B fragment
// of the top tile, tile j sits 256 j doubles before it.  EDGE: the lowest live tile (j = NA-1) is in its last k-step,
// where the lanes of its first tile column have nothing stored (below the diagonal).
template <int NA, bool EDGE>
__device__ __forceinline__ void genb_row(int bt, bool lowhalf, double2 za, double (&acc)[GENB_MAXT][4])
{
    double bv[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) bv[j] = tc_smem[bt - 256 * j];
    if (EDGE && lowhalf) bv[NA - 1] = 0.0;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
        dmma_m8n8k4(acc[j][0], acc[j][1], za.x, bv[j]);
        dmma_m8n8k4(acc[j][2], acc[j][3], za.y, bv[j]);
    }
}
// k-steps [kk, kend) of the NA live tiles, none of them an edge row: a tight loop (the dispatch on NA is paid once per run
// of rows, not per row).  bt = B fragment of the top tile in row kk; it moves on by one tile row minus one tile per row.
template <int NA>
__device__ __forceinline__ void genb_rows(int kk, int kend, int &bt, int oa, int nt4, int npar, int ak, double (&acc)[GENB_MAXT][4])
{
    int dbt = 16 * (nt4 - kk - 1);
#pragma unroll 2
    for (; kk < kend; ++kk, bt += dbt, dbt -= 16) {
        double2 za = make_double2(0.0, 0.0);                            // rows of the padding carry no increment
        if (4 * kk + ak < npar) za = *reinterpret_cast<const double2 *>(tc_smem + oa + 8 * kk);
        genb_row<NA, false>(bt, false, za, acc);
    }
}
#ifdef TC_SUBPROF
#define GSP_T0 long long gt__ = clock64()
#define GSP(i) do { if (threadIdx.x == 0 && cx.ch == 0) { const long long t__ = clock64(); tc_subprof[i] += t__ - gt__; gt__ = t__; } } while (0)
#else
#define GSP_T0
#define GSP(i)
#endif
__device__ __noinline__ void gen_increments_tma(const ChainCtx &cx, int g0, int nnew)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, npar = cx.npar;
    const int nt4 = (npar + 3) >> 2, NT = (npar + 7) >> 3;
    const int ar = lane >> 2, ak = lane & 3, th = ar >> 2, inner = 4 * ak + (ar & 3);
    TmaRing<GENB_NS> ring;      // a bulk copy per stage (one contiguous 16-32 KB piece): cp.async.cg fills measured 12 % slower here
    // the stages fill the per-warp areas (Z lives in the ring slots); one tile of room before the first stage and two after
    // the last row of a stage: the fragment reads of a half-stored tile pair fall there and are discarded
    const int sst = ((SPEC * cx.wsz - 16) / GENB_NS) & ~1, cap = sst - 32;
    ring.init(cx.o_U + 16, sst);
    // thread 0: next tile row to issue / its address (tile (pk, pk); the next diagonal tile is (nt4 - pk) tiles further) / stages issued
    int pk = 0, pg = 0;
    const double *src = cx.gRb;
#define GENB_ISSUE()                                                                                        \
    {                                                                                                       \
        int kend__ = pk, used__ = 0;                                                                        \
        while (kend__ < nt4 && kend__ - pk < GENB_RPS && used__ + 16 * (nt4 - kend__) <= cap) { used__ += 16 * (nt4 - kend__); ++kend__; } \
        ring.issue(pg, src, 8u * (unsigned)used__);     /* consecutive tile rows are contiguous: ONE segment */ \
        src += used__; pk = kend__;                                                                         \
        ++pg;                                                                                               \
    }
    if (tid == 0)
        while (pk < nt4 && pg < GENB_NS - 2) GENB_ISSUE()
    double acc[GENB_MAXT][4];
#pragma unroll
    for (int m = 0; m < GENB_MAXT; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; acc[m][2] = 0.0; acc[m][3] = 0.0; }
    const int oa = cx.slot_o(g0 + ar) + 2 * ak;                     // A row of this lane = ring slot of step g0 + ar (slots of rows >= nnew
                                                                    // hold stale data: their results are dropped)
    const int mcnt = NT > warp ? (NT - warp + SPEC - 1) / SPEC : 0; // column tiles warp, warp + 8, .. < NT
    int na = mcnt;                                                  // column tiles that still have rows at kk: the top `na` ones
    int last = 2 * warp + 1;                                        // last tile row of the lowest live tile
    // B fragment of the top tile (warp + 8 (mcnt - 1)), row kk: row start + ob - 16 kk
    const int ob = 16 * (2 * (warp + SPEC * (mcnt - 1)) + th) + inner;
    const int kmax = min(nt4, 2 * (warp + SPEC * (mcnt - 1)) + 2);  // rows this warp has MMAs for
    int kk = 0;
#pragma unroll 1
    for (int g = 0; kk < nt4; ++g) {
        GSP_T0;
        if (tid == 0 && pk < nt4) GENB_ISSUE()
        GSP(28);
        int kend = kk, used = 0;                                    // the rows of stage g: the producer's packing rule
        while (kend < nt4 && kend - kk < GENB_RPS && used + 16 * (nt4 - kend) <= cap) { used += 16 * (nt4 - kend); ++kend; }
        int bt = ring.acquire(g) + ob - 16 * kk;                    // B fragment of the top tile in row kk (stage start = row kk)
        GSP(29);
        int k = kk;
#pragma unroll 1
        while (k < kend && k < kmax) {
            const int kto = min(kend, min(last, kmax));             // the rows before the next edge row
            if (k < kto) {
                DISPATCH_1_7(na, genb_rows<N_>(k, kto, bt, oa, nt4, npar, ak, acc))
                k = kto;
            }
            if (k < kend && k == last && k < kmax) {
                // the lowest live tile is in its last k-step: the lanes of its first tile column have nothing stored there
                double2 za = make_double2(0.0, 0.0);
                if (4 * k + ak < npar) za = *reinterpret_cast<const double2 *>(tc_smem + oa + 8 * k);
                DISPATCH_1_7(na, (genb_row<N_, true>(bt, th == 0, za, acc)))
                bt += 16 * (nt4 - k - 1);
                ++k; --na; last += 2 * SPEC;
            }
        }
        kk = kend;
        GSP(30);
        ring.release(g);
        GSP(31);
    }
#undef GENB_ISSUE
    __syncthreads();                                                // every warp is done reading Z: the increments overwrite it
    if (ar < nnew) {
        const int oo = cx.slot_i(g0 + ar), o2 = oo + cx.s1;
        const double inv_dr = cx.cc.inv_dr;
#pragma unroll
        for (int j = 0; j < GENB_MAXT; ++j) {
            const int jc = 8 * (warp + SPEC * (mcnt - 1 - j)) + 2 * ak;     // accumulator j = the j-th tile from the top
            if (j < mcnt && jc < npar) { tc_smem[oo + jc] = acc[j][0]; tc_smem[o2 + jc] = acc[j][2] * inv_dr; }
            if (j < mcnt && jc + 1 < npar) { tc_smem[oo + jc + 1] = acc[j][1]; tc_smem[o2 + jc + 1] = acc[j][3] * inv_dr; }
        }
    }
    __syncthreads();
    ring.fini();
}

// Randomness and proposal increments for steps [g0, g0+nnew), nnew <= GEN_M = 8 (one MMA row group).
//   1. Philox normals z1, z2 -> scratch Z (the idle per-warp areas; row = step - g0, (z1, z2) interleaved per
//      parameter); u1, u2, chi2 -> the scalars of the step's ring slot.
//   2. the two norms entering q1, from z.
//   3. increments z1 R and z2 R/drscale -> the ring slot.  With a full factor this is ONE pass over R on the
//      FP64 tensor cores ([8 x npar] x [npar x npar] as mma.sync m8n8k4, A rows = the new steps, 4 interleaved
//      accumulator sets).  Every element of R is needed exactly once per call, so R is not staged as a matrix:
//      each lane pulls its own B elements HBM/L2 -> shared memory with 8-byte cp.async into private staging slots,
//      two groups of 8 k-steps in flight.  (The big layout's TMA-staged version, gen_increments_tma, measured 5 % slower
//      here at N = 120: R is 76 KB, and the per-lane cp.async stream needs no CTA-wide stage hand-over.)
__device__ __forceinline__ void warp_sum2(double &p, double &q)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { p += __shfl_xor_sync(0xffffffffu, p, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
}
__device__ __noinline__ void generate(const RunArgs &a, const ChainCtx &cx, int g0, int nnew, bool r_diag)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, npar = cx.npar;
    const int zs = 2 * cx.npad;                                   // doubles per row of Z
    // big layout: row sidx of Z is the ring slot of step g0 + sidx itself (the increments overwrite it at the end), which
    // leaves the per-warp areas to the TMA stages of R
    const bool big = a.big != 0;
#define ZROW(sidx) (big ? cx.slot_d(g0 + (sidx)) : cx.U + (size_t)(sidx) * zs)
    SUBP_BEGIN;
#ifdef TC_SUBPROF
    if (tid == 0 && cx.ch == 0) { tc_subprof[26] += 1; tc_subprof[27] += nnew; }
#endif
    if (a.replay) {
#pragma unroll 1
        for (int sidx = 0; sidx < nnew; ++sidx) {
            const int st = g0 + sidx;
            double *dz = ZROW(sidx), *sc = cx.slot_sc(st);
            const size_t g = ((size_t)cx.ch * a.nsimu + st) * cx.ld;
#pragma unroll 1
            for (int i = tid; i < npar; i += DRAM_THREADS) { dz[2 * i] = a.z1[g + i]; dz[2 * i + 1] = a.z2[g + i]; }
            if (tid == 0) {
                sc[0] = a.u1[(size_t)cx.ch * a.nsimu + st]; sc[1] = a.u2[(size_t)cx.ch * a.nsimu + st];
                sc[2] = a.chi2[(size_t)cx.ch * a.nsimu + st];
                sc[5] = tc_log(sc[0]);
            }
        }
    } else {
        // (Measured and dropped: warp w owning step g0 + w — its row's normals with the two norms folded in on the way, its
        // uniforms and chi-square on lane 0.  The norms pass disappears (1.8 k -> 0.7 k cycles per call) but every warp then
        // pays the serial chi-square + log chain, ~4.5 k cycles: randomness 5.5 k -> 7.6 k per call.)
        // lanes 0..nnew-1 of warp 0: the uniforms and the chi-square of step g0 + lane (a long serial draw, one step
        // per lane); everybody: one work item = the 4 normals of a parameter pair.  The items are dealt from warp 1
        // on, so that the odd extra item round lands on warp 7, not on warp 0.
        if (warp == 0 && lane < nnew) {
            const int st = g0 + lane;
            double *sc = cx.slot_sc(st);
            const u32x4 ru = draw(a.seed, cx.cc.uid, st, RK_U, 0);
            sc[0] = u01(ru.x, ru.y);
            sc[1] = u01(ru.z, ru.w);
            sc[2] = a.updatesigma ? chi2_draw_dc(a.seed, cx.cc.uid, st, cx.cc.chi_d, cx.cc.chi_c) : 1.0;
            sc[5] = tc_log(sc[0]);                                  // stage 1 is decided in the log domain
        }
        __syncwarp();
        const int npairs = (npar + 1) >> 1, nitems = nnew * npairs;
        const float inv_np = 1.0f / (float)npairs;                  // it / npairs without an integer division: exact here
        // the items are handed out 32 at a time from a shared counter: warp 0 joins when its chi-square draws are done (the draws
        // are addressed by (step, parameter pair), so who computes which does not matter)
#pragma unroll 1                                                    // (it + 0.5 is >= 0.5/npairs away from a multiple of npairs)
        for (;;) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&tc_genctr, 32);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= nitems) break;
            const int it = base + lane;
            if (it < nitems) {
                const int sidx = (int)(((float)it + 0.5f) * inv_np), q2 = it - sidx * npairs;
                double *dz = ZROW(sidx);
                const double4 z = normal_quad(a.seed, cx.cc.uid, g0 + sidx, q2);
                *reinterpret_cast<double2 *>(dz + 4 * q2) = make_double2(z.x, z.z);          // (z1, z2) of parameter 2q
                if (2 * q2 + 1 < npar) *reinterpret_cast<double2 *>(dz + 4 * q2 + 2) = make_double2(z.y, z.w);
            }
        }
    }
    __syncthreads();
    if (tid == 0) tc_genctr = 0;                                    // for the next call (many barriers away)
    SUBP(0);
    // q1 = -1/2 (|(y1-y2) R^-1|^2 - |(y1-x) R^-1|^2) = -1/2 (|z1 - z2/drscale|^2 - |z1|^2)
    if (warp < nnew) {
        const double2 *dz = reinterpret_cast<const double2 *>(ZROW(warp));
        double n1 = 0.0, n0 = 0.0;
#pragma unroll 1
        for (int i = lane; i < npar; i += 32) {
            const double2 zz = dz[i];
            const double d = zz.x - zz.y * cx.cc.inv_dr;
            n1 = fma(d, d, n1);
            n0 = fma(zz.x, zz.x, n0);
        }
        warp_sum2(n1, n0);                                          // (the two butterflies side by side)
        if (lane == 0) { double *sc = cx.slot_sc(g0 + warp); sc[3] = n1; sc[4] = n0; }
    }
    SUBP(1);
    if (r_diag) {
        // big layout: Z lives in the ring slots and is scaled IN PLACE below, while the warps above may still be reading it
        // for the norms (the regular layout keeps Z apart, and gen_increments_tma starts with a barrier of its own)
        if (big) __syncthreads();
#pragma unroll 1
        for (int sidx = 0; sidx < nnew; ++sidx) {
            const double2 *dz = reinterpret_cast<const double2 *>(ZROW(sidx));
            const int o1 = cx.slot_i(g0 + sidx), o2 = o1 + cx.s1;
            // (big layout: Z is this very slot, interleaved; every thread reads all its pairs before anyone stores)
            double2 zz[(7 + 414 + DRAM_THREADS - 1) / DRAM_THREADS];
#pragma unroll
            for (int m = 0; m < (int)(sizeof(zz) / sizeof(zz[0])); ++m) { const int j = tid + m * DRAM_THREADS; if (j < npar) zz[m] = dz[j]; }
            if (big) __syncthreads();
#pragma unroll
            for (int m = 0; m < (int)(sizeof(zz) / sizeof(zz[0])); ++m) {
                const int j = tid + m * DRAM_THREADS;
                if (j < npar) {
                    const double r = cx.rdiag[j];
                    tc_smem[o1 + j] = zz[m].x * r; tc_smem[o2 + j] = zz[m].y * (r * cx.cc.inv_dr);
                }
            }
        }
    } else if (big) {
        gen_increments_tma(cx, g0, nnew);
        SUBP(2);
    } else {
        const int NT = (npar + 7) >> 3;                              // column tiles of 8
        const int ar = lane >> 2, ak = lane & 3;                     // A[row = step][k], B[k][col]
        const double *gR = cx.gRb;
        const double inv_dr = cx.cc.inv_dr;
        // Column tiles are dealt to the warps in serpentine order (longest k-range first: balances the triangle):
        // tile of round r = NT-1 - (8 r + (r odd ? 7-w : w)).
        const int oa = cx.o_U + ar * zs;                              // A row of this lane (offset into tc_smem); rows >= nnew hold
                                                                      // stale scratch: their results are dropped
        const int oo = cx.slot_i(g0 + ar), oo2 = oo + cx.s1;          // output vectors (stage 1, stage 2) of this lane's row
        const bool rowok = ar < nnew;
        const int nt4 = (npar + 3) >> 2;
        const int inner = 4 * ak + (ar & 3);                          // position of (row 4kk+ak, column 8nt+ar) inside its 4x4 tile
        const int ostg = cx.o_U + GEN_M * zs + warp * (16 * 32) + lane;   // staging slot s of this lane: ostg + 32 s
        const unsigned sstg = (unsigned)__cvta_generic_to_shared(tc_smem + ostg);
#pragma unroll 1
        for (int rnd = 0; rnd * SPEC < NT; ++rnd) {
            const int nt = NT - 1 - (rnd * SPEC + ((rnd & 1) ? SPEC - 1 - warp : warp));
            if (nt < 0) continue;
            const int ks = (min(8 * nt + 8, npar) + 3) >> 2;         // k-steps (= tile rows) of this column tile
            const int bj = (8 * nt + ar < npar) ? 2 * nt + (ar >> 2) : -1;   // 4x4 tile column of this lane (-1: nothing to load)
            // four interleaved accumulator sets (k-steps u mod 4): 8 independent MMA chains hide the MMA latency
            double acc[4][4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[q][e] = 0.0;
            // R is stored in 4x4 tiles (see chol_tiled): tile (kk, bj) sits 16 (nt4 - kk - 1) doubles after tile (kk-1, bj)
            int il = 0, dpl = 16 * (nt4 - 1), ic = ak;
            const double *pl = gR + 16 * bj + inner;
            // B fragments: 8-byte cp.async into this lane's private staging slots, two groups of 8 k-steps in flight
            // (commit / wait_group order the arrivals; a register pipeline would have to share the warp's 6 scoreboards)
#define GEN_ISSUE(slot, live)                                                                               \
    {                                                                                                       \
        if ((live) && il <= bj) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sstg + 256u * (unsigned)(slot)), "l"(pl) : "memory"); \
        else tc_smem[ostg + 32 * (slot)] = 0.0;                                                             \
        pl += dpl; dpl -= 16; il += 1;                                                                      \
    }
            // k-steps are consumed in groups of 8; the slots of a group past the last k-step are zero-filled, so that the MMAs
            // of a group are unconditional (an mma.sync under a condition costs a WARPSYNC + predicate each)
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                if (8 * g < ks) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) GEN_ISSUE(8 * g + u, 8 * g + u < ks)
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
#pragma unroll 1
            for (int kk = 0; kk < ks; kk += 8) {
                asm volatile("cp.async.wait_group 1;" ::: "memory");
                const int base = kk & 15;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const double bv = tc_smem[ostg + 32 * (base + u)];
                    double2 za = make_double2(0.0, 0.0);
                    if (ic < npar) za = *reinterpret_cast<const double2 *>(tc_smem + oa + 2 * ic);
                    dmma_m8n8k4(acc[u & 3][0], acc[u & 3][1], za.x, bv);
                    dmma_m8n8k4(acc[u & 3][2], acc[u & 3][3], za.y, bv);
                    ic += 4;
                }
                if (kk + 16 < ks) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) GEN_ISSUE(base + u, kk + 16 + u < ks)
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
#undef GEN_ISSUE
            const double acc0 = (acc[0][0] + acc[1][0]) + (acc[2][0] + acc[3][0]), acc1 = (acc[0][1] + acc[1][1]) + (acc[2][1] + acc[3][1]);
            const double acc2 = (acc[0][2] + acc[1][2]) + (acc[2][2] + acc[3][2]), acc3 = (acc[0][3] + acc[1][3]) + (acc[2][3] + acc[3][3]);
            const int jc = 8 * nt + 2 * ak;
            if (rowok) {
                if (jc < npar) { tc_smem[oo + jc] = acc0; tc_smem[oo2 + jc] = acc2 * inv_dr; }
                if (jc + 1 < npar) { tc_smem[oo + jc + 1] = acc1; tc_smem[oo2 + jc + 1] = acc3 * inv_dr; }
            }
        }
        SUBP(2);
    }
    __syncthreads();
    SUBP(3);
#undef ZROW
}


// Round phase A: bounds and prior of both proposals of the candidate steps k .. k+C-1 (warp w: candidates w, w+8).
// The proposals are never materialised: theta = x + ring increment, the very expression the forward model
// (SumVec) and the commit phase use.                    bounds/prior: TranscriptionCycleMCMC.m:235-255
// UNI: this chain's bounds / prior have the reference's structure (TranscriptionCycleMCMC.m:242-255) — seven head parameters with
// their own bounds, then one block (dR) with common bounds and prior (cx.blk) — so only the first pass (j < 32) reads the
// per-parameter vectors; SM: the vectors are in shared memory (regular layout) or in HBM/L2 (big layout).
template <bool SM, bool UNI>
__device__ __forceinline__ void cand_bounds_t(const ChainCtx &cx, int k, int C, Cand *cand)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, npar = cx.npar;
    const int ox = cx.o_x, ol = cx.o_lo, oh = ol + npar, om = oh + npar, op = cx.o_pinv;
    const double blo = cx.blk[0], bhi = cx.blk[1], bmu = cx.blk[2], bpinv = cx.blk[3];
#pragma unroll 1
    for (int c = warp; c < C; c += SPEC) {
        const int o1 = cx.slot_i(k + c), o2 = o1 + cx.s1;
        double pr1 = 0.0, pr2 = 0.0;
        unsigned oob = 0;
#pragma unroll 1                                                    // the smallest code: measured +1 % on config 2 against unroll 4
        for (int j = lane; j < npar; j += 32) {
            const double xj = tc_smem[ox + j], a1 = xj + tc_smem[o1 + j], a2 = xj + tc_smem[o2 + j];
            double lo, hi, mu, pinv;
            if (UNI && j >= 8) { lo = blo; hi = bhi; mu = bmu; pinv = bpinv; }
            else {
                lo = SM ? tc_smem[ol + j] : cx.lo[j]; hi = SM ? tc_smem[oh + j] : cx.hi[j];
                mu = SM ? tc_smem[om + j] : cx.mu[j]; pinv = tc_smem[op + j];
            }
            if (a1 < lo || a1 > hi) oob |= 1u;
            if (a2 < lo || a2 > hi) oob |= 2u;
            const double e1 = (a1 - mu) * pinv, e2 = (a2 - mu) * pinv;
            pr1 = fma(e1, e1, pr1);
            pr2 = fma(e2, e2, pr2);
        }
        warp_sum2(pr1, pr2);
        oob = __reduce_or_sync(0xffffffffu, oob);
        if (lane == 0) { cand[c].pr1 = pr1; cand[c].pr2 = pr2; cand[c].oob = (int)oob; }
    }
}
__device__ __noinline__ void cand_bounds(const ChainCtx &cx, int k, int C, Cand *cand)
{
    if (cx.o_lo >= 0) { if (cx.uni) cand_bounds_t<true, true>(cx, k, C, cand); else cand_bounds_t<true, false>(cx, k, C, cand); }
    else { if (cx.uni) cand_bounds_t<false, true>(cx, k, C, cand); else cand_bounds_t<false, false>(cx, k, C, cand); }
}

// The delayed-rejection decision of ONE step (one lane) whose first stage rejected, from state (ss, pri) seeing sigma2 = s2p;
// q1 = -1/2 (|z1 - z2/drscale|^2 - |z1|^2) and the uniform u2 are the step's (generate()).  Both samplers decide through it:
// dram_kernel in round phase D, dram_warp_kernel in its step loop.  The three exponentials are evaluated in one interleaved
// body (an unused one may see garbage or Inf: it is never read):
//   a12 = exp(-1/2 ((ss1-ss)/s2 + pr1-pri)), a32 = exp(-1/2 ((ss1-ss2)/s2 + pr1-pr2)), exp(l2 + q1)
//                                                                             mcmcstat DRAM: SURVEY.md 3.2
__device__ __noinline__ int resolve_dr(double q1, double u2, bool o1, double x12, double pr1, double pr2, double ss1, double ss2,
                                       double ss, double pri, double is2p)            // is2p = 1 / sigma2 of the step
{
    double e12, e32, e13;
    tc_exp3(x12, -0.5 * ((ss1 - ss2) * is2p + pr1 - pr2), -0.5 * ((ss2 - ss) * is2p + pr2 - pri) + q1, e12, e32, e13);
    const double a12 = o1 ? 0.0 : e12;
    double a32 = e32;
    a32 = a32 > 1.0 ? 1.0 : a32;
    if (!(a32 >= 0.0)) a32 = 0.0;
    // accept iff min(1, e13 (1 - a32) / (1 - a12)) > u2 (or = 1), decided without the quotient: 1 - a12 > 0 because stage 1
    // rejected (a12 < u1 < 1; an out-of-bounds first stage has a12 = 0), so the test is num > u2 den (or num >= den).  A
    // denominator that rounds to 0 keeps the quotient's answer: +Inf -> accept when num > 0, 0/0 -> reject.
    const double num = e13 * (1.0 - a32), den = 1.0 - a12;
    if (!(den > 0.0)) return num > 0.0 ? 1 : 0;
    return (num >= den || num > u2 * den) ? 1 : 0;
}

// dst[e] = src[e] * sc, e < n 16-byte units, src in HBM/L2: 8 independent loads in flight per thread (written as one loop
// the compiler keeps every load behind the previous store: dst may alias src for all it knows)
__device__ __forceinline__ void scaled_copy_cg(double2 *dst, const double2 *src, int n, double sc)
{
    int e = threadIdx.x;
#pragma unroll 1
    for (; e + 7 * DRAM_THREADS < n; e += 8 * DRAM_THREADS) {
        double2 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldcg(src + e + u * DRAM_THREADS);
#pragma unroll
        for (int u = 0; u < 8; ++u) dst[e + u * DRAM_THREADS] = make_double2(v[u].x * sc, v[u].y * sc);
    }
#pragma unroll 1
    for (; e < n; e += DRAM_THREADS) { const double2 v = __ldcg(src + e); dst[e] = make_double2(v.x * sc, v.y * sc); }
}

// Adaptation after the step with isimu (a multiple of adaptint).  The block of chain rows since the last adaptation (adaptint
// of them; the first block is rows 0 .. isimu-1, which is 2 rows when adaptint = 1) arrives as `ndist` DISTINCT rows with integer weights (a rejected step repeats the previous row): the
// scatter of the block is sum_d w_d (x_d - mb)(x_d - mb)', folded into the running scatter matrix with
// Chan's mean-shift term as one more weighted row, in 4x4 register tiles.  Then either burn-in scaling or
// R = chol(cov + qcovadj I) * adascale.  Returns 0: R unchanged / scaled, 1: new full factor, 2: Cholesky failed.
__device__ __noinline__ int adapt(const RunArgs &a, const ChainCtx &cx, int isimu, double cov_n, double rate, bool r_diag,
                                  int ndist)
{
    const int tid = threadIdx.x, npar = cx.npar, ld = cx.ld;
    double *sw = tc_smem + cx.o_ring;                  // workspace: ring + per-warp areas (idle now); sqrt(weight) per row first
                                                       // (offset arithmetic on tc_smem compiles to LDS / STS, cx.ring would be generic)
    SUBP_BEGIN;
    if (a.do_cov) {
        const CovBlock blk = cov_block(isimu, cov_n, ndist);
        const int m = blk.m, nrows = blk.nrows;
        const double fcorr = blk.fcorr;
#pragma unroll 1
        for (int i = tid; i < npar; i += DRAM_THREADS) {
            const double mbi = cx.mb[i] / m;
            cx.mb[i] = mbi;
            cx.dm[i] = mbi - __ldcg(cx.cmean + i);
        }
        // M2 += U'U on the FP64 tensor cores, U = the weighted, centred rows (COV_CR of them per pass, staged in shared
        // memory): per 8x8 block of M2 one mma.sync m8n8k4 per 4 rows (A = U' fragment, B = U fragment), two blocks
        // interleaved per warp; the block is then added to the scatter matrix in HBM/L2, which uses the same 4x4-tile
        // layout as the Cholesky workspace (a lane's two adjacent columns are one 16-byte access).
        const int warp = tid >> 5, lane = tid & 31, ar = lane >> 2, ak = lane & 3;
        const int nt4 = (npar + 3) >> 2, NT = (npar + 7) >> 3, NB = NT * (NT + 1) / 2;
        const int ldu = 8 * NT + 4;                                   // row stride of U (doubles); + 4: rows 0..3 of a k-step hit different banks
        double *U = tc_smem + cx.o_ring + COV_CR + 8;                 // after sw[COV_CR]
#pragma unroll 1
        for (int r0 = 0; r0 < nrows; r0 += COV_CR) {
            const int rc = min(COV_CR, nrows - r0), rc4 = (rc + 3) & ~3;
            __syncthreads();
            if (tid < rc) sw[tid] = r0 + tid < ndist ? sqrt(__ldcg(cx.gWts + r0 + tid)) : sqrt(fcorr);
            __syncthreads();
            // warp w stages rows w, w+8, ..: coalesced along the row, several rows' loads in flight
#pragma unroll 1
            for (int c = lane; c < 8 * NT; c += 32) {
                const double mbc = c < npar ? cx.mb[c] : 0.0, dmc = c < npar ? cx.dm[c] : 0.0;
                double v[COV_CR / SPEC];
#pragma unroll
                for (int q = 0; q < COV_CR / SPEC; ++q) {
                    const int r = warp + SPEC * q, rr = r0 + r;
                    v[q] = (c < npar && r < rc && rr < ndist) ? __ldcg(cx.gRows + (size_t)rr * ld + c) : 0.0;
                }
#pragma unroll
                for (int q = 0; q < COV_CR / SPEC; ++q) {
                    const int r = warp + SPEC * q, rr = r0 + r;
                    if (r < rc4) U[r * ldu + c] = (c < npar && r < rc) ? sw[r] * (rr < ndist ? v[q] - mbc : dmc) : 0.0;
                }
            }
            __syncthreads();
            // blocks b and b + SPEC (upper triangle of 8x8 blocks, row-major): (block row, position in the row) advance by
            // 2 SPEC blocks per iteration
            int bi0 = 0, rm0 = warp, bi1 = 0, rm1 = warp + SPEC;
            while (bi0 < NT && rm0 >= NT - bi0) { rm0 -= NT - bi0; ++bi0; }
            while (bi1 < NT && rm1 >= NT - bi1) { rm1 -= NT - bi1; ++bi1; }
#pragma unroll 1
            for (int b = warp; b < NB; b += 2 * SPEC) {
                const int bj0 = bi0 + rm0;
                const bool two = b + SPEC < NB;
                const int bi1u = two ? bi1 : 0, bj1 = two ? bi1 + rm1 : 0;      // no second block: block 0 again, result dropped
                // the old values of the two blocks: loaded first, so that their L2 latency overlaps with the MMAs
                double2 *g0 = nullptr, *g1 = nullptr;
                {
                    const int row = 8 * bi0 + ar, col = 8 * bj0 + 2 * ak, tr = row >> 2, tcn = col >> 2;
                    if (tr <= tcn && tcn < nt4)                       // the tile exists (upper triangle, inside the padded matrix)
                        g0 = reinterpret_cast<double2 *>(cx.gM2 + 16 * (size_t)tidx(nt4, tr, tcn) + 4 * (row & 3) + (col & 3));
                }
                if (two) {
                    const int row = 8 * bi1u + ar, col = 8 * bj1 + 2 * ak, tr = row >> 2, tcn = col >> 2;
                    if (tr <= tcn && tcn < nt4)
                        g1 = reinterpret_cast<double2 *>(cx.gM2 + 16 * (size_t)tidx(nt4, tr, tcn) + 4 * (row & 3) + (col & 3));
                }
                double2 o0 = make_double2(0.0, 0.0), o1 = o0;
                if (g0) o0 = __ldcg(g0);
                if (g1) o1 = __ldcg(g1);
                double d00 = 0.0, d01 = 0.0, d10 = 0.0, d11 = 0.0;
                const double *ua0 = U + ak * ldu + 8 * bi0 + ar, *ub0 = U + ak * ldu + 8 * bj0 + ar;
                const double *ua1 = U + ak * ldu + 8 * bi1u + ar, *ub1 = U + ak * ldu + 8 * bj1 + ar;
#pragma unroll 2
                for (int kk = 0; kk < rc4; kk += 4) {
                    dmma_m8n8k4(d00, d01, ua0[kk * ldu], ub0[kk * ldu]);
                    dmma_m8n8k4(d10, d11, ua1[kk * ldu], ub1[kk * ldu]);               // unconditional (no second block: block 0 again, dropped)
                }
                if (g0) *g0 = make_double2(o0.x + d00, o0.y + d01);
                if (g1) *g1 = make_double2(o1.x + d10, o1.y + d11);
                rm0 += 2 * SPEC; rm1 += 2 * SPEC;
                while (bi0 < NT && rm0 >= NT - bi0) { rm0 -= NT - bi0; ++bi0; }
                while (bi1 < NT && rm1 >= NT - bi1) { rm1 -= NT - bi1; ++bi1; }
            }
        }
        SUBP(8);
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < npar; i += DRAM_THREADS) { cx.cmean[i] = __ldcg(cx.cmean + i) + cx.dm[i] * blk.shift; cx.mb[i] = 0.0; }
        cov_n += m;
        __syncthreads();
        SUBP(9);
    }
    int ret = 0;
    if (isimu < a.burnintime) {
        const double f = burnin_factor(rate, a.burnin_scale);
        if (f != 1.0) {
            if (r_diag) {
#pragma unroll 1
                for (int i = tid; i < npar; i += DRAM_THREADS) cx.rdiag[i] *= f;
            } else {
#pragma unroll 1
                for (int i = tid; i < tri_doubles(npar); i += DRAM_THREADS) cx.gRb[i] = __ldcg(cx.gRb + i) * f;
                if (a.big) fence_async_proxy();
            }
        }
    } else {
        // R = chol(cov + qcovadj I) * adascale, factorised in shared memory (tiled layout), kept in HBM/L2
        const double invn = 1.0 / (cov_n - 1.0);
        const int nt4 = (npar + 3) >> 2, T4 = tri_doubles(npar) / 16;
        // mcmcstat: [Ra,is] = chol(cov); only when that fails ("try to blow it") chol(cov + qcovadj I)  [U]; qcovadj_always = 1
        // factors cov + qcovadj I at once
        if (a.big) {
            // the factor does not fit in shared memory: factorise through HBM/L2 into this CTA's workspace
            double *gW = a.gW + (size_t)blockIdx.x * a.ldR;
            const int o_ws = cx.o_ring, ws_d = (cx.ring_mask + 1) * cx.slot_sz + SPEC * cx.wsz;
            bool ok = chol_global(nt4, npar, cx.gM2, invn, a.qcovadj_always ? a.qcovadj : 0.0, gW, o_ws, ws_d);
            if (!ok && !a.qcovadj_always) ok = chol_global(nt4, npar, cx.gM2, invn, a.qcovadj, gW, o_ws, ws_d);
            SUBP(11);
            if (ok) {
                scaled_copy_cg(reinterpret_cast<double2 *>(cx.gRb), reinterpret_cast<const double2 *>(gW), 8 * T4, cx.cc.adascale);
                fence_async_proxy();                                // generate() reads R back with bulk copies
            }
            __syncthreads();
            SUBP(12);
            return ok ? 1 : 2;
        }
        double *W = tc_smem + cx.o_ring;
        unsigned short *tab = reinterpret_cast<unsigned short *>(W + 16 * T4);
#pragma unroll 1
        for (int t = tid; t < T4; t += DRAM_THREADS) {
            int rem = t, b = 0;
            while (rem >= nt4 - b) { rem -= nt4 - b; ++b; }
            tab[t] = (unsigned short)((b << 8) | (b + rem));
        }
        bool ok = false;
#pragma unroll 1
        for (int attempt = a.qcovadj_always ? 1 : 0; attempt < 2 && !ok; ++attempt) {
            const double adj = attempt ? a.qcovadj : 0.0;
            __syncthreads();
            scaled_copy_cg(reinterpret_cast<double2 *>(W), reinterpret_cast<const double2 *>(cx.gM2), 8 * T4, invn);
            __syncthreads();
            // the diagonal of cov_entry's matrix (the rest of the padding is zero: it only ever accumulated zeros)
#pragma unroll 1
            for (int i = tid; i < 4 * nt4; i += DRAM_THREADS) {
                double *d = W + 16 * tidx(nt4, i >> 2, i >> 2) + 5 * (i & 3);
                *d = cov_diag(*d, i, npar, adj);
            }
            __syncthreads();
            SUBP(10);
            ok = chol_tiled(nt4, cx.o_ring, cx.ch == 0);
            __syncthreads();
            SUBP(11);
        }
        if (ok) {
            {
                const double2 *src = reinterpret_cast<const double2 *>(W);
                double2 *dst = reinterpret_cast<double2 *>(cx.gRb);
                const double sc = cx.cc.adascale;
#pragma unroll 8
                for (int e = tid; e < 8 * T4; e += DRAM_THREADS) { const double2 v = src[e]; dst[e] = make_double2(v.x * sc, v.y * sc); }
            }
            ret = 1;
        } else {
            ret = 2;                                                // R unchanged
        }
    }
    __syncthreads();
    SUBP(12);
    return ret;
}

// The device-resident DRAM sampler: one CTA per chain slice, SPEC future steps per round.
//
// DRAM is sequential, but a step that rejects leaves the state untouched, and at the acceptance
// rates of this model (3-30 %) most do.  So the CTA simulates the next SPEC steps AT ONCE, warp w
// running step k+w in full (both proposal stages, forward model, accept/reject) under the
// hypothesis "nothing before me accepted"; the round is then cut after the first step that did
// accept, that prefix is committed, and the later warps' work is discarded.  The chain produced is
// exactly the sequential one (same Philox draws per step; the replay tests compare it flag by flag
// with the CPU oracle).  The randomness and the proposal increments z R do not depend on the state,
// so they are generated ahead of use, up to RING steps per call, into a ring of RING slots.
// Book-keeping works on RUNS (an accepted state and the rejections that follow it): a rejected step
// only lengthens the current run; summaries, chain storage and the covariance block see a run once,
// with its length as weight.
template <bool THIN>
__global__ void __launch_bounds__(DRAM_THREADS, 2) dram_kernel(const __grid_constant__ RunArgs ga)
{
    // The out-of-line phases take the launch arguments by reference: a reference to the kernel parameter
    // itself would turn every field access into a generic load from parameter memory, so they get a
    // shared-memory copy instead.
    __shared__ RunArgs a;
    {
        const int *src = reinterpret_cast<const int *>(&ga);
        int *dst = reinterpret_cast<int *>(&a);
        for (int i = threadIdx.x; i < (int)(sizeof(RunArgs) / sizeof(int)); i += DRAM_THREADS) dst[i] = src[i];
        if (threadIdx.x == 0) tc_genctr = 0;
    }
    __syncthreads();
    __shared__ Cand s_cand[RING];
    __shared__ double s_ssv[2 * RING];
    __shared__ ChainCtx cx;
    __shared__ int s_item, s_done, s_sum, s_own;
    __shared__ unsigned s_min;
    __shared__ ChainState st;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // Persistent CTAs time-slice the chains: a free CTA claims a chain that is not running and still
    // has slices left (a.cstate[c] = next slice, bit 30 = running) — the one that is furthest behind,
    // so that all chains finish together — runs one slice and releases it.  So any number of chains
    // shares the resident CTAs evenly (299 chains on 296 CTA slots would otherwise cost two full
    // waves).  A slice ends on an adaptation boundary, where the ring is empty, the current run is
    // closed and the factor R / covariance already live in HBM; the rest of the chain state is a few vectors.
    const int LOCK = 1 << 30;
    const int nseg = (a.nsimu + a.seglen - 1) / a.seglen;
    int start = (int)(((long long)blockIdx.x * a.nchains) / gridDim.x);
    // Two CTAs share an SM and slow each other down: a chain runs ~24 % faster with the SM to itself (scripts/solo_sm.py), and
    // the fit lasts as long as its slowest chain.  So a CTA whose chain lags the mean progress of all chains by solo_lag slices
    // takes the SM (smctl[%smid]); its neighbour finishes the slice it is in, claims nothing and sleeps until the SM is
    // shared again.  Chains that are ahead wait for a slot instead (the furthest-behind chain is always claimed first), so
    // the slots given up come out of the time the fast chains would have idled at the end of the fit.
    unsigned smid = 0;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    int *const smc = (a.solo_lag > 0 && nseg > 1) ? a.smctl + (smid & 1023) : nullptr;
    const int me = (int)blockIdx.x + 1;
    bool own = false;                                       // uniform: this CTA holds its SM
#pragma unroll 1
    for (;;) {
        // claim a chain: the whole CTA scans the state words in parallel; key = (slices done, distance from `start`)
#pragma unroll 1
        for (;;) {
            __syncthreads();
            if (tid == 0) { s_min = 0xffffffffu; s_sum = 0; }
            if (smc && !own && tid == 0) {
                // the neighbour holds the SM: stay out of its way
#pragma unroll 1
                while (*reinterpret_cast<volatile int *>(smc) != 0) __nanosleep(4000);
            }
            __syncthreads();
            int pending = 0, prog = 0;
#pragma unroll 1
            for (int base = 0; base < a.nchains; base += DRAM_THREADS) {
                const int i = base + tid;
                int hit = 0;
                if (i < a.nchains) {
                    const int v = *reinterpret_cast<volatile int *>(a.cstate + (start + i) % a.nchains);
                    prog += min(v & ~LOCK, nseg);
                    if (v & LOCK) pending = 1;
                    else if (v < nseg) { hit = 1; atomicMin(&s_min, ((unsigned)v << 24) | (unsigned)min(i, 0xffffff)); }
                }
                if (__syncthreads_or(hit) && nseg == 1) break;           // unsliced: any free chain will do
            }
            if (smc) { prog = __reduce_add_sync(0xffffffffu, prog); if (lane == 0) atomicAdd(&s_sum, prog); }
            pending = __syncthreads_or(pending);
            const unsigned kmin = s_min;
            if (kmin == 0xffffffffu) {
                if (own) { if (tid == 0) atomicExch(smc, 0); own = false; }   // nothing to run: the neighbour may
                if (!pending) { if (tid == 0) s_item = -1; break; }     // every chain is finished
                __nanosleep(50000);                                     // (a slice lasts milliseconds; the scan costs the neighbour issue slots)
                continue;
            }
            if (tid == 0) {
                const int c = (start + (int)(kmin & 0xffffffu)) % a.nchains;
                const int v = *reinterpret_cast<volatile int *>(a.cstate + c);
                const bool ok = !(v & LOCK) && v < nseg && atomicCAS(a.cstate + c, v, v | LOCK) == v;
                s_item = ok ? c : -2;
                s_done = v;
                s_own = own ? 1 : 0;
                if (ok && smc) {
                    const bool lagging = (long long)s_sum - (long long)v * a.nchains >= (long long)a.solo_lag * a.nchains;
                    if (lagging) {
                        if (!own) {
                            if (atomicCAS(smc, 0, me) == 0) s_own = 1;
                            else { atomicExch(a.cstate + c, v); s_item = -2; }      // the neighbour took the SM meanwhile: give the chain back
                        }
                    } else {
                        if (own) { atomicExch(smc, 0); s_own = 0; }
                        else if (*reinterpret_cast<volatile int *>(smc) != 0) { atomicExch(a.cstate + c, v); s_item = -2; }
                    }
                }
            }
            __syncthreads();
            own = s_own != 0;
            if (s_item != -2) break;
        }
        __syncthreads();
        const int ch = s_item, seg = s_done;
        if (ch < 0) break;                                  // every chain is finished (own is false here)
        start = (ch + 1) % a.nchains;
        __threadfence();
        const int cid = a.chain_cell[ch];
        const int N = a.cells.N[cid];
        const int npar = 7 + N;
        double *gst = a.gState + (size_t)ch * state_doubles(a.ld);

        // ---- carve shared memory (offsets in doubles into tc_smem), publish the context
        {
            SmemCell cv;
            int o = carve_cell(0, N, cv);
            o += o & 1;
            if (tid == 0) {
                cx.N = N; cx.npar = npar; cx.npad = (npar + 3) & ~3; cx.ld = a.ld;
                cx.slot_sz = dram_slot(N); cx.s1 = dram_s1(N); cx.wsz = a.wsz; cx.ch = ch;
                cx.cc = chain_consts(a, ch, N);
                cx.cv = cv; cx.cv.d = a.cells.dmean[cid];
                o |= 1;                                             // x at an ODD offset: x[7] is 16-byte aligned (SumVec::get4)
                cx.o_x = o;
                cx.x = tc_smem + o; o += npar;
                cx.o_lo = a.big ? -1 : o;                           // lo, hi, mu consecutive
                if (a.big) {
                    // bounds and prior means stay in HBM/L2 (read once per candidate step by cand_bounds)
                    cx.lo = const_cast<double *>(a.low) + (size_t)ch * a.ld; cx.hi = const_cast<double *>(a.upp) + (size_t)ch * a.ld;
                    cx.mu = const_cast<double *>(a.pmu) + (size_t)ch * a.ld;
                } else {
                    cx.lo = tc_smem + o; o += npar;    cx.hi = tc_smem + o; o += npar;    cx.mu = tc_smem + o; o += npar;
                }
                cx.o_pinv = o; cx.pinv = tc_smem + o; o += npar;  cx.o_wmean = o; cx.wmean = tc_smem + o; o += npar;
                cx.o_wM2 = o; cx.wM2 = tc_smem + o; o += npar;   cx.rdiag = tc_smem + o; o += npar; cx.o_mb = o; cx.mb = tc_smem + o; o += npar;
                cx.dm = tc_smem + o; o += npar;
                o += o & 1;
                cx.o_ring = o;
                cx.ring_mask = (a.big ? RING / 2 : RING) - 1;
                cx.ring = tc_smem + o; o += (cx.ring_mask + 1) * dram_slot(N);
                cx.o_U = o;
                cx.U = tc_smem + o;
                cx.gRb = a.gR + (size_t)ch * a.ldR;                 // the factor R lives in HBM/L2 (4x4 tiles)
                cx.gM2 = a.gM2 ? a.gM2 + (size_t)ch * a.ldR : nullptr;
                cx.gRows = a.gRows ? a.gRows + (size_t)ch * (size_t)a.blk_rows * a.ld : nullptr;
                cx.gWts = a.gWts ? a.gWts + (size_t)ch * (size_t)a.blk_rows : nullptr;
                cx.cmean = a.gCmean ? a.gCmean + (size_t)ch * a.ld : nullptr;
            }
            load_cell(a.cells, cid, cv);
        }
        __syncthreads();
        // this warp's private forward-model scratch
        Work w;
        carve_work(cx.o_U + warp * cx.wsz, N, w);
#pragma unroll 1
        for (int i = tid; i < npar; i += DRAM_THREADS) {
            const size_t g = (size_t)ch * a.ld + i;
            if (!a.big) {
                cx.lo[i] = a.low[g];
                cx.hi[i] = a.upp[g];
                cx.mu[i] = a.pmu[g];
            }
            cx.pinv[i] = prior_inv(a.psig[g]);
            cx.mb[i] = 0.0;
            if (seg == 0) {
                cx.x[i] = a.theta0[g];
                cx.rdiag[i] = sqrt(a.qcov_diag[g]);            // chol(diag(J0))
                cx.wmean[i] = 0.0;
                cx.wM2[i] = 0.0;
                if (a.do_cov) cx.cmean[i] = 0.0;
            } else {
                cx.x[i] = __ldcg(gst + ST_VEC0 + i);
                cx.wmean[i] = __ldcg(gst + ST_VEC0 + a.ld + i);
                cx.wM2[i] = __ldcg(gst + ST_VEC0 + 2 * a.ld + i);
                cx.rdiag[i] = __ldcg(gst + ST_VEC0 + 3 * a.ld + i);
            }
        }
        if (seg == 0) {
            if (a.do_cov) {
#pragma unroll 1
                for (int i = tid; i < tri_doubles(npar); i += DRAM_THREADS) cx.gM2[i] = 0.0;
            }
            // ring slot 0 = zero increments: row 0 evaluates ss(x0) through the same theta view as every step
#pragma unroll 1
            for (int i = tid; i < cx.slot_sz; i += DRAM_THREADS) cx.ring[i] = 0.0;
        }

        {
            // bounds / prior in the reference's head + block structure?  (four vectors read once per slice)
            int diff = 0;
#pragma unroll 1
            for (int i = 8 + tid; i < npar; i += DRAM_THREADS) {
                const size_t g = (size_t)ch * a.ld;
                const double s7 = a.psig[g + 7], si = a.psig[g + i];
                diff |= !(a.low[g + i] == a.low[g + 7] && a.upp[g + i] == a.upp[g + 7] && a.pmu[g + i] == a.pmu[g + 7] && si == s7);
            }
            diff = __syncthreads_or(diff);
            if (tid == 0) {
                const size_t g = (size_t)ch * a.ld + 7;
                cx.uni = diff ? 0 : 1;
                cx.blk[0] = a.low[g]; cx.blk[1] = a.upp[g]; cx.blk[2] = a.pmu[g]; cx.blk[3] = prior_inv(a.psig[g]);
            }
        }
        if (tid == 0) {
            if (seg == 0) {
                st.sigma2 = a.sigma2_0; st.r_diag = 1;              // (ss, pri, rden, rsig: row 0 below)
                st.t = Tally{};
                st.t.n_ss = 1;                                      // ss(x0)
                st.run_r0 = 0;
            } else {
                // (the tally's reju comes back as parked, which is 0: a slice ends on an adaptation boundary, or adaptation
                // is off and nothing reads it)
                const ParkedChain p = resume_chain(gst);
                st.ss = p.ss; st.pri = p.pri; st.sigma2 = p.sigma2; st.rsig = p.rsig; st.r_diag = p.r_diag;
                st.rden = rden_of(a.N0 * a.S20, p.ss);
                st.t = p.t;
                st.run_r0 = seg * a.seglen;
            }
            st.bad0 = 0;
            st.ndist = 0;
            st.tprev = clock64();
        }
        __syncthreads();
        // phase clocks (TC_CNT_CYCLES0..).  (Sampling them every 8th round was measured: no gain — 66.7 M against 67.5 M.)
#define TC_PHASE(i) do { if (tid == 0) { const long long tn__ = clock64(); st.t.pc[i] += tn__ - st.tprev; st.tprev = tn__; } } while (0)

        if (seg == 0) {
            // ---- row 0: x0 (opens the first run)
            const double ss0 = ss_eval(a.cons, cx.cv, SumVec{cx.o_x, cx.slot_i(0)}, w, a.algo, false, nullptr, nullptr);   // every warp, same value
            double sp = 0.0;
#pragma unroll 1
            for (int i = lane; i < npar; i += 32) { const double e = (cx.x[i] - cx.mu[i]) * cx.pinv[i]; sp += e * e; }
            sp = warp_sum(sp);
            const bool bad = !isfinite(ss0);
            if (tid == 0) {
                st.ss = ss0; st.pri = sp; st.bad0 = bad ? 1 : 0; st.rden = rden_of(a.N0 * a.S20, ss0); st.rsig = 1.0 / a.sigma2_0;
                if (!bad) record_row0<THIN>(a, ch, ss0, st.t);
            }
            __syncthreads();
        }

        const Slice slice = slice_of(a, seg);
        const int k_end = slice.k_end;
        int k = slice.k, next_adapt = slice.next_adapt;   // next step to decide, next adaptation
        int gen_upto = k;                           // increments are ready for steps [k, gen_upto)
        const bool bad0 = st.bad0 != 0;
#pragma unroll 1
        while (k < k_end && !bad0) {
            // the round never crosses an adaptation: the step whose isimu = st+1 is a multiple of adaptint
            // is the last one that may use the current R
            const int bound = min(k_end, next_adapt);                       // exclusive step bound
            // chain state of this round (thread 0 rewrites st only in the commit phase, after two barriers)
            const double ss = st.ss, pri = st.pri, sig2 = st.sigma2, wcnt = st.t.wcnt;
            const int run_r0 = st.run_r0, ndist = st.ndist;
            // 1 / sigma2 of the candidate steps, started here so that the divisions are off the critical path of phase D:
            // step k sees sig2, step k + w sees (N0 S20 + ss) / chi2_{k+w-1}, i.e. 1/sigma2 = chi2_{k+w-1} * rden.  (A product
            // with a rounded reciprocal instead of a quotient: the acceptance exponent moves by an ulp, like the log-domain
            // decision of stage 1.)
            const double rden = st.rden, rsig = st.rsig;

            if (gen_upto < bound && gen_upto - k < (a.big ? 1 : SPEC)) {
                // fewer than SPEC steps ready => at least GEN_M of the RING slots are free (big layout: ring of GEN_M
                // slots, refilled when empty)
                const int glim = min(gen_upto + GEN_M, bound);
                generate(a, cx, gen_upto, glim - gen_upto, st.r_diag != 0);
                gen_upto = glim;
            }
            TC_PHASE(PH_GEN);

            // ---- one round = SPEC forward-model evaluations, one per warp, over as many future steps as they cover.
            // A. bounds + prior of both proposals of every ready step (an out-of-bounds proposal needs no evaluation)
            const int C = min(gen_upto - k, SPEC);                          // candidates: one per warp (more are almost never covered)
            SUBP_BEGIN;
            cand_bounds(cx, k, C, s_cand);
            SUBP(16);
            __syncthreads();
            SUBP(17);
            // B. task list, in step order: stage 1 (if in bounds), stage 2 (if in bounds; needed unless stage 1 accepts,
            //    which is rare); the round covers the longest prefix of steps whose tasks fit in SPEC warps.  Every warp
            //    derives the same list (lane = candidate step).
            int c_oob = 3, c_nt = 2 * SPEC;
            if (lane < C) {
                c_oob = s_cand[lane].oob;
                c_nt = ((c_oob & 1) ? 0 : 1) + ((a.ntry >= 2 && !(c_oob & 2)) ? 1 : 0);
            }
            int inc = c_nt;
#pragma unroll
            for (int o = 1; o < RING; o <<= 1) { const int up = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += up; }
            const int exc = inc - c_nt;
            const bool covered = lane < C && inc <= SPEC;
            const int nsteps = __popc(__ballot_sync(0xffffffffu, covered));  // >= 1: a step has at most 2 tasks
            const unsigned tmask = __ballot_sync(0xffffffffu, covered && exc <= warp && warp < inc);
            // C. this warp's evaluation
            if (tmask) {
                const int mc = __ffs(tmask) - 1;
                const int e0 = __shfl_sync(0xffffffffu, exc, mc), ob = __shfl_sync(0xffffffffu, c_oob, mc);
                const int stage = (warp == e0 && !(ob & 1)) ? 0 : 1;
                const double v = ss_eval(a.cons, cx.cv, SumVec{cx.o_x, cx.slot_i(k + mc) + stage * cx.s1}, w, a.algo, false, nullptr, nullptr);
                if (lane == 0) s_ssv[2 * mc + stage] = v;
            }
            SUBP(18);
            __syncthreads();
            SUBP(19);
            TC_PHASE(PH_STEPS);
            // D. accept/reject of every covered step under the hypothesis "the steps before it rejected" (lane = step; the
            //    sigma2 a step sees is the draw made at the end of the previous step from the unchanged ss).  Every warp
            //    computes the same outcomes, so no barrier is needed before the commit (and a warp running this alone is
            //    no faster: measured).
            //    Stage 1 is decided in the log domain (a12 > u  <=>  x12 > log u, log u drawn with the step's randomness), so
            //    a step that accepts at once costs one division and no exponential; only the steps BEFORE the first such
            //    accept can matter, and only they run the delayed-rejection arithmetic.
            StepOut so_;
            so_.acc = 0; so_.fl = 0; so_.nev = 0; so_.noob = 0; so_.ssn = 0.0; so_.prin = 0.0;
            const bool act = lane < nsteps;
            const bool o1 = (c_oob & 1) != 0, o2 = (c_oob & 2) != 0;
            double is2p = rsig, x12 = 0.0, pr1 = 0.0, pr2 = 0.0, ss1 = INFINITY, ss2 = 0.0;
            const double *scp = cx.slot_sc(k + (act ? lane : 0));
            bool acc1 = false;
            if (act) {
                if (lane > 0 && a.updatesigma) is2p = cx.slot_sc(k + lane - 1)[2] * rden;
                pr2 = s_cand[lane].pr2; ss2 = s_ssv[2 * lane + 1];
                if (!o1) {
                    pr1 = s_cand[lane].pr1; ss1 = s_ssv[2 * lane];
                    acc1 = stage1_accepts(ss1, ss, is2p, pr1, pri, scp[5], x12);
                }
            }
            const unsigned m1 = __ballot_sync(0xffffffffu, act && acc1);
            const int f1 = m1 ? __ffs(m1) - 1 : nsteps;                      // first step accepting at stage 1
            if (act && lane <= f1) {
                so_.ssn = ss1; so_.prin = pr1;
                if (o1) { so_.fl |= TC_FL_OOB1; so_.noob = 1; } else so_.nev = 1;
                if (acc1) so_.acc = 1;
            }
            if (f1 > 0 && a.ntry >= 2) {                                    // warp-uniform: someone needs the second stage
                if (act && lane < f1) {
                    so_.fl |= TC_FL_DR;
                    if (o2) { so_.fl |= TC_FL_OOB2; ++so_.noob; }
                    else {
                        ++so_.nev;
                        if (resolve_dr(-0.5 * (scp[3] - scp[4]), scp[1], o1, x12, pr1, pr2, ss1, ss2, ss, pri, is2p)) { so_.acc = 2; so_.fl |= TC_FL_STAGE2; so_.ssn = ss2; so_.prin = pr2; }
                    }
                }
            }
            if (so_.acc) so_.fl |= TC_FL_ACCEPT;
            const unsigned amask = __ballot_sync(0xffffffffu, lane < nsteps && so_.acc != 0);
            const bool accd = amask != 0;
            const int first = accd ? __ffs(amask) - 1 : nsteps;
            const int ncommit = accd ? first + 1 : nsteps;
            const int r_acc = k + first;                                    // row of the accept
            const int src = accd ? first : 0;
            const int acc_t = __shfl_sync(0xffffffffu, so_.acc, src);
            const double ssn_a = __shfl_sync(0xffffffffu, so_.ssn, src), prin_a = __shfl_sync(0xffffffffu, so_.prin, src);
            SUBP(20);
            if (accd) {
                // close the run of the old state at row r_acc and move x by the accepted increment
                flush_run<THIN>(a, cx, run_r0, r_acc, wcnt, ndist, cx.slot_i(r_acc) + (acc_t == 2 ? cx.s1 : 0), 32);
            }
            SUBP(21);
            if (warp == 0) {
                // the chain state of the next round: only what the next round needs, one division (lane 0).  The sigma2 the
                // next step sees is the draw of the last committed row, made from that row's ss
                if (lane == 0) {
                    const double ss_new = accd ? ssn_a : ss;
                    if (accd) {
                        st.ss = ss_new; st.pri = prin_a;
                        st.t.wcnt = wcnt + run_rows(run_r0, r_acc, cx.cc.first_row);
                        if (run_distinct(a.do_cov, run_r0, r_acc)) st.ndist = ndist + 1;
                        st.run_r0 = r_acc;
                    }
                    // sigma2 of the next step = (N0 S20 + ss_new) / chi2 of the last committed row, kept as its reciprocal (the
                    // same product chi2 * rden the later steps of a round use: the chain does not depend on where rounds are cut)
                    const double rd = accd ? rden_of(a.N0 * a.S20, ss_new) : rden;
                    if (accd) st.rden = rd;
                    if (a.updatesigma) st.rsig = cx.slot_sc(k + ncommit - 1)[2] * rd;
                }
            } else if (warp == SPEC - 1) {
                // meanwhile: per-row scalars of the committed rows (lane = row) — sigma2 of the row (rows before the accept
                // keep ss), s2chain statistics, optional per-step outputs — and the counters
                const double ss_new = accd ? ssn_a : ss;
                double s2 = 0.0, sq = 0.0;
                if (lane < ncommit) {
                    const int r = k + lane;
                    const double ssr = lane < first ? ss : ss_new;
                    s2 = row_sigma2(a.updatesigma, a.N0 * a.S20, ssr, cx.slot_sc(r)[2], sig2);
                    sq = sqrt(s2);
                    store_row<THIN>(a, cx.ch, r, s2, so_.fl, ssr);
                }
                // the round's sum of s2, and mean of sqrt(s2) and squared deviations from it (rows = lanes < ncommit <= RING / 2)
                double s2b = s2, mb = sq;
#pragma unroll
                for (int o = RING / 2; o > 0; o >>= 1) { s2b += __shfl_xor_sync(0xffffffffu, s2b, o); mb += __shfl_xor_sync(0xffffffffu, mb, o); }
                mb *= tc_rcp((double)ncommit);
                double dq = lane < ncommit ? sq - mb : 0.0;
                dq *= dq;
#pragma unroll
                for (int o = RING / 2; o > 0; o >>= 1) dq += __shfl_xor_sync(0xffffffffu, dq, o);
                const int d_ss = __reduce_add_sync(0xffffffffu, lane < ncommit ? so_.nev : 0);
                const int d_oob = __reduce_add_sync(0xffffffffu, lane < ncommit ? so_.noob : 0);
                const int d_dr = __reduce_add_sync(0xffffffffu, (lane < ncommit && (so_.fl & TC_FL_DR)) ? 1 : 0);
                const int d_spec = __shfl_sync(0xffffffffu, inc, nsteps - 1);       // evaluations of this round
                if (lane == 0) {
                    tally_s2(st.t, ncommit, s2b, mb, dq);
                    const int nrej = accd ? first : nsteps;
                    st.t.n_ss += d_ss; st.t.n_oob += d_oob; st.t.n_dr += d_dr; st.t.n_spec += d_spec;
                    st.t.rej += nrej; st.t.reju += nrej;
                    if (accd) { if (acc_t == 1) ++st.t.n_acc1; else ++st.t.n_acc2; }
                }
            }
            SUBP(22);
            k += ncommit;
            __syncthreads();
            SUBP(23);
#ifdef TC_SUBPROF
            if (tid == 0 && cx.ch == 0) { tc_subprof[24] += 1; tc_subprof[25] += ncommit; }
#endif
            TC_PHASE(PH_COMMIT);

            // adaptation after the step with isimu = k, a multiple of adaptint
            if (k == next_adapt) {
                const int rr0 = st.run_r0, nd0 = st.ndist;
                const double wc0 = st.t.wcnt;
                flush_run<THIN>(a, cx, rr0, k, wc0, nd0, -1, 0);                     // close the run at the block boundary
                const int nd = nd0 + (run_distinct(a.do_cov, rr0, k) ? 1 : 0);
                const double rate = adapt_rate(a, st.t.rej, st.t.reju, k);
                const double cov_n = st.t.cov_n;
                const bool rdg = st.r_diag != 0;
                __syncthreads();
                const int rc = adapt(a, cx, k, cov_n, rate, rdg, nd);
                if (tid == 0) {
                    st.t.wcnt = wc0 + run_rows(rr0, k, cx.cc.first_row);
                    st.run_r0 = k; st.ndist = 0;
                    after_adapt(st.t, a.do_cov, k, rc);
                    if (rc == 1) st.r_diag = 0;
                }
                __syncthreads();
                next_adapt += a.adaptint;
                TC_PHASE(PH_ADAPT);
            }
        }

        __syncthreads();
        if (!bad0 && st.run_r0 < k) {
            // close the last run (the fit or the slice does not end on an adaptation boundary)
            const int rr0 = st.run_r0;
            const double wc0 = st.t.wcnt;
            flush_run<THIN>(a, cx, rr0, k, wc0, st.ndist, -1, 0);
            __syncthreads();
            if (tid == 0) { st.t.wcnt = wc0 + run_rows(rr0, k, cx.cc.first_row); st.run_r0 = k; }
            __syncthreads();
        }
        if (!slice.last && !bad0) {
            // ---- park the chain: the next slice may run on any CTA
#pragma unroll 1
            for (int i = tid; i < npar; i += DRAM_THREADS) {
                gst[ST_VEC0 + i] = cx.x[i];
                gst[ST_VEC0 + a.ld + i] = cx.wmean[i];
                gst[ST_VEC0 + 2 * a.ld + i] = cx.wM2[i];
                gst[ST_VEC0 + 3 * a.ld + i] = cx.rdiag[i];
            }
            if (tid == 0) park_chain(gst, ParkedChain{st.ss, st.pri, st.sigma2, st.rsig, st.r_diag, 0, st.t});
            __threadfence();
            __syncthreads();
            if (tid == 0) atomicExch(a.cstate + ch, seg + 1);      // release: next slice, not running
            continue;
        }

        // ---- summaries; a chain whose ss(x0) is not finite ends here
        write_outputs(a, ch, npar, cx.wmean, cx.wM2, st.t, st.t.n_spec, bad0, tid, DRAM_THREADS);
        if (tid == 0) {
            __threadfence();
            atomicExch(a.cstate + ch, nseg);                        // finished (also ends a chain whose ss(x0) failed)
        }
    }
}

#include "tc_warp.cuh"

// -------------------------------------------------------------------------- RNG dump / FP64 peak
__global__ void rng_dump_kernel(unsigned long long seed, unsigned long long uid, int npar, double dof,
                                int nsimu, double *z1, double *u1, double *z2, double *u2, double *chi2)
{
    for (int k = blockIdx.x; k < nsimu; k += gridDim.x) {
        for (int q = threadIdx.x; 2 * q < npar; q += blockDim.x) {
            const double4 z = normal_quad(seed, uid, k, q);
            z1[(size_t)k * npar + 2 * q] = z.x;
            z2[(size_t)k * npar + 2 * q] = z.z;
            if (2 * q + 1 < npar) { z1[(size_t)k * npar + 2 * q + 1] = z.y; z2[(size_t)k * npar + 2 * q + 1] = z.w; }
        }
        if (threadIdx.x == 0) {
            const u32x4 ru = draw(seed, uid, k, RK_U, 0);
            u1[k] = u01(ru.x, ru.y);
            u2[k] = u01(ru.z, ru.w);
            chi2[k] = chi2_draw(seed, uid, k, dof);
        }
    }
}

__global__ void dfma_peak_kernel(double *out, long long *clk, int iters)
{
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
           a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-7;
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const long long t1 = clock64();
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (threadIdx.x == 0) clk[blockIdx.x] = t1 - t0;
}

// ===================================================================================== host side
struct DevCells {
    int device = -1;
    CellsDev d{};
    std::vector<void *> allocs;
    // Scratch of the fits comes from a PRIVATE stream-ordered pool owned by the dataset (created on first use, destroyed
    // with it): consecutive fits recycle their tens of MB without cudaMalloc/cudaFree, and the host application's default
    // pool is never touched.
    mutable cudaMemPool_t pool = nullptr;
};

struct tc_cells {
    tc_construct cons;
    int ncells = 0, Nmax = 0;
    std::vector<int> N;
    std::vector<long long> off;
    std::vector<double> t, tg, dtraw, dtg, ms2, pp7, iw, dmean, tgp, dtgp;
    std::vector<int> ik;
    std::vector<DevCells> dev;
};

static double ml_round(double x) { return x >= 0 ? std::floor(x + 0.5) : -std::floor(-x + 0.5); }

// MATLAB a:d:b (Moler's colon algorithm) — t_interp = t(1):dt:t(end), SumofSquares...m:30
static std::vector<double> matlab_colon(double a, double d, double b)
{
    std::vector<double> out;
    if (d == 0 || (d > 0 && a > b) || (d < 0 && a < b) || std::isnan(a) || std::isnan(b) || std::isnan(d)) return out;
    const double tol = 2.0 * std::numeric_limits<double>::epsilon() * std::max(std::fabs(a), std::fabs(b));
    const double sig = d > 0 ? 1.0 : -1.0;
    long long n;
    if (a == std::floor(a) && d == 1) n = (long long)(std::floor(b) - a);
    else if (a == std::floor(a) && d == std::floor(d)) {
        const double q = std::floor(a / d), r = a - q * d;
        n = (long long)(std::floor((b - r) / d) - q);
    } else {
        n = (long long)ml_round((b - a) / d);
        if (sig * (a + n * d - b) > tol) n -= 1;
    }
    double c = a + n * d;
    if (sig * (c - b) > -tol) c = b;
    out.assign((size_t)n + 1, 0.0);
    for (long long k = 0; k <= n / 2; ++k) {
        out[(size_t)k] = a + k * d;
        out[(size_t)(n - k)] = c - k * d;
    }
    if (n % 2 == 0) out[(size_t)(n / 2)] = (a + c) / 2;
    return out;
}

template <typename T>
static int upload(DevCells &dc, const std::vector<T> &h, const T *&dptr)
{
    void *p = nullptr;
    CUDA_TRY(cudaMalloc(&p, std::max<size_t>(h.size(), 1) * sizeof(T)));
    dc.allocs.push_back(p);
    CUDA_TRY(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    dptr = static_cast<const T *>(p);
    return TC_OK;
}

static int validate_construct(const tc_construct *c)
{
    if (!c) return fail(TC_EINVAL, "construct is NULL");
    if (c->nsets < 1 || c->nsets > TC_MAX_SETS) return fail(TC_EINVAL, "construct.nsets out of range");
    for (int s = 0; s < c->nsets; ++s) {
        if (!(c->ms2_start[s] >= 0 && c->pp7_start[s] >= 0)) return fail(TC_EINVAL, "construct: loop start must be >= 0");
        if (!(c->ms2_start[s] < c->ms2_end[s] && c->pp7_start[s] < c->pp7_end[s]))
            return fail(TC_EINVAL, "construct: loop start must be < loop end");
    }
    return TC_OK;
}

extern "C" {

int tc_version(void) { return TC_VERSION; }
const char *tc_last_error(void) { return g_err.c_str(); }
double tc_last_kernel_seconds(void) { return g_last_kernel_s; }
double tc_last_drain_seconds(void) { return g_last_drain_s; }

int tc_host_alloc(size_t bytes, void **out)
{
    if (!out) return fail(TC_EINVAL, "out is NULL");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1) return fail(TC_ENODEV, "no CUDA device available (libtcmcmc has no CPU fallback)");
    CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return TC_OK;
}

void tc_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

int tc_device_count(int *count)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return fail(TC_ENODEV, cudaGetErrorString(e)); }
    *count = n;
    return TC_OK;
}

int tc_device_info_get(int device, tc_device_info *out)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return fail(TC_ENODEV, "no such CUDA device");
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, device));
    std::memset(out, 0, sizeof(*out));
    std::strncpy(out->name, p.name, sizeof(out->name) - 1);
    out->cc_major = p.major; out->cc_minor = p.minor; out->sm_count = p.multiProcessorCount;
    out->total_mem = (int64_t)p.totalGlobalMem; out->smem_per_block_optin = (int64_t)p.sharedMemPerBlockOptin;
    return TC_OK;
}

void tc_opts_default(tc_mcmc_opts *o)
{
    std::memset(o, 0, sizeof(*o));
    o->nsimu = 20000; o->burnintime = 10000; o->adaptint = 100; o->ntry = 2; o->updatesigma = 1;
    o->burnin_cumulative = 1; o->qcovadj_always = 0; o->n_burn = 10000; o->store_chain = 0; o->replay = 0; o->algo = TC_ALGO_TOEPLITZ;
    o->ngpus = 1; o->thin = 1;
    for (int i = 0; i < TC_MAX_GPUS; ++i) o->devices[i] = -1;
    o->drscale = 5.0; o->adascale = 0.0; o->qcovadj = 1e-8; o->burnin_scale = 10.0; o->N0 = 1.0; o->S20 = 1.0;
    o->sigma2_0 = 1.0; o->seed = 20201028ULL;
}

int tc_cells_create(const tc_construct *construct, int ncells, const int32_t *N, const int64_t *off,
                    const double *t, const double *ms2, const double *pp7, int ndev, const int32_t *devices,
                    tc_cells **out)
{
    if (!out) return fail(TC_EINVAL, "out is NULL");
    *out = nullptr;
    int rc = validate_construct(construct);
    if (rc) return rc;
    if (ncells < 1 || !N || !off || !t || !ms2 || !pp7) return fail(TC_EINVAL, "empty dataset or NULL array");
    int ndevs = 0;
    if (cudaGetDeviceCount(&ndevs) != cudaSuccess || ndevs < 1) return fail(TC_ENODEV, "no CUDA device available (libtcmcmc has no CPU fallback)");
    if (ndev < 1) ndev = 1;
    DeviceGuard guard;
    tc_cells *c = new tc_cells();
    c->cons = *construct;
    c->ncells = ncells;
    c->N.assign(N, N + ncells);
    c->off.resize(ncells + 1);
    long long tot = 0;
    for (int i = 0; i < ncells; ++i) {
        if (N[i] < 3) { delete c; return fail(TC_EINVAL, "cell with fewer than 3 timepoints"); }
        c->off[i] = tot; tot += N[i];
        c->Nmax = std::max(c->Nmax, (int)N[i]);
    }
    c->off[ncells] = tot;
    c->t.resize(tot); c->tg.resize(tot); c->dtraw.assign(tot, 0.0); c->dtg.assign(tot, 0.0);
    c->ms2.resize(tot); c->pp7.resize(tot); c->iw.assign(tot, 0.0); c->ik.assign(tot, -1); c->dmean.resize(ncells);
    for (int ci = 0; ci < ncells; ++ci) {
        const int n = N[ci];
        const double *ts = t + off[ci];
        double *T = c->t.data() + c->off[ci], *G = c->tg.data() + c->off[ci];
        std::copy(ts, ts + n, T);
        std::copy(ms2 + off[ci], ms2 + off[ci] + n, c->ms2.data() + c->off[ci]);
        std::copy(pp7 + off[ci], pp7 + off[ci] + n, c->pp7.data() + c->off[ci]);
        for (int i = 0; i + 1 < n; ++i)
            if (!(ts[i + 1] > ts[i])) { delete c; return fail(TC_EINVAL, "time vector must be strictly increasing"); }
        double s = 0;                                      // mean(t(2:end)-t(1:end-1))  SumofSquares...m:29
        for (int i = 0; i + 1 < n; ++i) s += ts[i + 1] - ts[i];
        const double dt = s / (n - 1);
        c->dmean[ci] = dt;
        std::vector<double> g = matlab_colon(ts[0], dt, ts[n - 1]);
        if ((int)g.size() != n) {
            delete c;
            return fail(TC_EDIM, "numel(t(1):dt:t(end)) != numel(t) for cell " + std::to_string(ci) +
                                     " (MATLAB: arrays have incompatible sizes in ConstantElongationSim R.*dt)");
        }
        std::copy(g.begin(), g.end(), G);
        for (int i = 0; i + 1 < n; ++i) {
            c->dtraw[c->off[ci] + i] = ts[i + 1] - ts[i];
            c->dtg[c->off[ci] + i] = G[i + 1] - G[i];
        }
        // interp1(t_interp, model, t): bracketing interval + weight per experimental time (:55-56)
        for (int j = 0; j < n; ++j) {
            const double z = ts[j];
            if (!(z >= G[0] && z <= G[n - 1])) continue;      // NaN outside the grid
            int k = (int)(std::upper_bound(G, G + n, z) - G) - 1;
            if (k > n - 2) k = n - 2;
            c->ik[c->off[ci] + j] = k;
            c->iw[c->off[ci] + j] = (z - G[k]) / (G[k + 1] - G[k]);
        }
    }
    // tg / dtg in the order the kernels keep them in shared memory (cell_perm): cell ci at off[ci] + 4 ci
    c->tgp.assign(tot + 4LL * ncells, 0.0); c->dtgp.assign(tot + 4LL * ncells, 0.0);
    for (int ci = 0; ci < ncells; ++ci)
        for (int i = 0; i < N[ci]; ++i) {
            const long long dst = c->off[ci] + 4LL * ci + cell_perm(N[ci], i);
            c->tgp[dst] = c->tg[c->off[ci] + i];
            c->dtgp[dst] = c->dtg[c->off[ci] + i];
        }
    c->dev.resize(ndev);
    for (int d = 0; d < ndev; ++d) {
        DevCells &dc = c->dev[d];
        dc.device = devices ? devices[d] : d;
        if (dc.device < 0 || dc.device >= ndevs) { tc_cells_destroy(c); return fail(TC_ENODEV, "device index out of range"); }
        cudaError_t e = cudaSetDevice(dc.device);
        if (e != cudaSuccess) { tc_cells_destroy(c); return fail(TC_ECUDA, cudaGetErrorString(e)); }
        dc.d.ncells = ncells;
        if ((rc = upload(dc, c->N, dc.d.N)) || (rc = upload(dc, c->off, dc.d.off)) || (rc = upload(dc, c->t, dc.d.t)) ||
            (rc = upload(dc, c->tg, dc.d.tg)) || (rc = upload(dc, c->dtraw, dc.d.dtraw)) ||
            (rc = upload(dc, c->dtg, dc.d.dtg)) || (rc = upload(dc, c->ms2, dc.d.ms2)) ||
            (rc = upload(dc, c->pp7, dc.d.pp7)) || (rc = upload(dc, c->iw, dc.d.iw)) ||
            (rc = upload(dc, c->dmean, dc.d.dmean)) || (rc = upload(dc, c->ik, dc.d.ik)) ||
            (rc = upload(dc, c->tgp, dc.d.tgp)) || (rc = upload(dc, c->dtgp, dc.d.dtgp))) {
            std::string m = g_err;
            tc_cells_destroy(c);
            return fail(rc, m);
        }
    }
    *out = c;
    return TC_OK;
}

void tc_cells_destroy(tc_cells *c)
{
    if (!c) return;
    DeviceGuard guard;
    for (auto &dc : c->dev) {
        if (dc.device >= 0) cudaSetDevice(dc.device);
        for (void *p : dc.allocs) cudaFree(p);
        if (dc.pool) { cudaDeviceSynchronize(); cudaMemPoolDestroy(dc.pool); dc.pool = nullptr; }
    }
    delete c;
}

int tc_cells_t_interp(const tc_cells *c, int cell, double *out, int cap)
{
    if (!c || cell < 0 || cell >= c->ncells) return fail(TC_EINVAL, "bad cell index");
    const int n = c->N[cell];
    if (cap < n) return fail(TC_EINVAL, "buffer too small");
    std::copy(c->tg.begin() + c->off[cell], c->tg.begin() + c->off[cell] + n, out);
    return n;
}

static const DevCells *find_dev(const tc_cells *c, int device)
{
    for (auto &d : c->dev) if (d.device == device) return &d;
    return nullptr;
}

// ss_stream_kernel stages per warp the cell (a.csz doubles, set here), two theta rows (a.ld2, set here) and the
// forward-model scratch (a.wsz).  It runs where two of its CTAs, each also holding 1 KB of reserved shared memory, fit one
// SM: returns its dynamic shared memory per CTA then, else 0.
static size_t ss_stream_smem(SsArgs &a, int Nmax, int ld, int optin)
{
    a.csz = (cell_doubles(Nmax) + 1) & ~1;
    a.ld2 = (ld + 1) & ~1;
    const size_t smem = sizeof(double) * (size_t)(a.csz + 2 * a.ld2 + 2 + a.wsz) * SS_WARPS;
    return 2 * (smem + 1024) <= (size_t)optin + 1024 ? smem : 0;
}

static int launch_ss(const tc_cells *c, const DevCells *dc, long long nbatch, const int *d_cell, const double *d_theta,
                     int ld, int algo, int raw, double *d_ss, double *d_o1, double *d_o2, int ldo, cudaStream_t st)
{
    if (algo != TC_ALGO_PAIRS && algo != TC_ALGO_TOEPLITZ) return fail(TC_EINVAL, "unknown algo");
    if (raw && algo != TC_ALGO_PAIRS) return fail(TC_EINVAL, "the raw (irregular) grid needs TC_ALGO_PAIRS");
    if (ld < 7 + c->Nmax) return fail(TC_EINVAL, "ld < 7 + max(N)");
    if (nbatch <= 0) return TC_OK;
    SsArgs a{};
    a.cells = dc->d; a.cons = make_consx(c->cons); a.nbatch = nbatch; a.cell_id = d_cell; a.theta = d_theta; a.ld = ld;
    a.algo = algo; a.raw_grid = raw; a.ldo = ldo; a.ss_out = d_ss; a.out1 = d_o1; a.out2 = d_o2;
    a.wsz = (work_doubles(c->Nmax) + 3) & ~1;
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dc->device));
    if (!raw && d_ss && !d_o1 && !d_o2 && algo == TC_ALGO_TOEPLITZ) {
        // SS only, O(N) algorithm (latency-bound): operands staged in shared memory (ss_stream_kernel) when two CTAs per SM
        // fit.  The pairs algorithm is FP64-pipe-bound and prefers the 32 warps/SM of the global-view kernel (measured:
        // 52.7 M evaluations/s there, 34.2 M with 16 warps/SM here).
        int optin = 0;
        CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dc->device));
        if (const size_t smem2 = ss_stream_smem(a, c->Nmax, ld, optin)) {
            CUDA_TRY(cudaFuncSetAttribute(ss_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            const long long want2 = (nbatch + SS_WARPS - 1) / SS_WARPS;
            const int grid2 = (int)std::min<long long>(want2, (long long)sms * 2);
            ss_stream_kernel<<<grid2, SS_THREADS, smem2, st>>>(a);
            CUDA_TRY(cudaGetLastError());
            return TC_OK;
        }
    }
    const size_t smem = sizeof(double) * (size_t)a.wsz * SS_WARPS;
    CUDA_TRY(cudaFuncSetAttribute(ss_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long want = (nbatch + SS_WARPS - 1) / SS_WARPS, maxgrid = (long long)sms * 16;
    const int grid = (int)std::min<long long>(want, maxgrid);
    ss_batch_kernel<<<grid, SS_THREADS, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return TC_OK;
}

int tc_ss_batch_device(const tc_cells *c, int device, int64_t nbatch, const int32_t *d_cell_id, const double *d_theta,
                       int ld, int algo, double *d_ss_out, void *stream)
{
    if (!c) return fail(TC_EINVAL, "cells is NULL");
    const DevCells *dc = find_dev(c, device);
    if (!dc) return fail(TC_EINVAL, "cells not resident on that device");
    DeviceGuard guard;
    CUDA_TRY(cudaSetDevice(device));
    return launch_ss(c, dc, nbatch, d_cell_id, d_theta, ld, algo, 0, d_ss_out, nullptr, nullptr, 0, (cudaStream_t)stream);
}

}  // extern "C"

struct DevBuf {                      // RAII for device scratch
    // With a pool: stream-ordered allocation from the dataset's private memory pool (DevCells::pool), so that the
    // scratch of one fit (tens of MB) is recycled by the next instead of going through cudaMalloc/cudaFree every call.
    std::vector<void *> ptrs;
    cudaStream_t st = nullptr;
    cudaMemPool_t pool = nullptr;
    bool pooled = false;
    void release()
    {
        for (void *p : ptrs) { if (pooled) cudaFreeAsync(p, st); else cudaFree(p); }
        ptrs.clear();
    }
    ~DevBuf() { release(); }
    template <typename T> cudaError_t alloc(T *&p, size_t n)
    {
        void *q = nullptr;
        const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
        cudaError_t e = pooled ? cudaMallocFromPoolAsync(&q, bytes, pool, st) : cudaMalloc(&q, bytes);
        if (e == cudaSuccess) { ptrs.push_back(q); p = static_cast<T *>(q); }
        return e;
    }
};

static int ss_host(const tc_cells *c, int64_t nbatch, const int32_t *cell_id, const double *theta, int ld, int algo,
                   int raw, double *ss_out, double *o1, double *o2, int ldo)
{
    if (!c) return fail(TC_EINVAL, "cells is NULL");
    if (nbatch < 0 || (nbatch > 0 && (!cell_id || !theta))) return fail(TC_EINVAL, "NULL batch arrays");
    if (nbatch == 0) return TC_OK;
    for (int64_t b = 0; b < nbatch; ++b)
        if (cell_id[b] < 0 || cell_id[b] >= c->ncells) return fail(TC_EINVAL, "cell_id out of range");
    if ((o1 || o2) && ldo < c->Nmax) return fail(TC_EINVAL, "ldo < max(N)");
    const DevCells *dc = &c->dev[0];
    DeviceGuard guard;
    CUDA_TRY(cudaSetDevice(dc->device));
    DevBuf buf;
    int *d_cell = nullptr; double *d_theta = nullptr, *d_ss = nullptr, *d_o1 = nullptr, *d_o2 = nullptr;
    CUDA_TRY(buf.alloc(d_cell, nbatch));
    CUDA_TRY(buf.alloc(d_theta, (size_t)nbatch * ld));
    if (ss_out) CUDA_TRY(buf.alloc(d_ss, nbatch));
    if (o1) { CUDA_TRY(buf.alloc(d_o1, (size_t)nbatch * ldo)); CUDA_TRY(buf.alloc(d_o2, (size_t)nbatch * ldo)); }
    CUDA_TRY(cudaMemcpy(d_cell, cell_id, nbatch * sizeof(int), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_theta, theta, (size_t)nbatch * ld * sizeof(double), cudaMemcpyHostToDevice));
    if (o1) { CUDA_TRY(cudaMemset(d_o1, 0, (size_t)nbatch * ldo * sizeof(double))); CUDA_TRY(cudaMemset(d_o2, 0, (size_t)nbatch * ldo * sizeof(double))); }
    int rc = launch_ss(c, dc, nbatch, d_cell, d_theta, ld, algo, raw, d_ss, d_o1, d_o2, ldo, 0);
    if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    if (ss_out) CUDA_TRY(cudaMemcpy(ss_out, d_ss, nbatch * sizeof(double), cudaMemcpyDeviceToHost));
    if (o1) {
        CUDA_TRY(cudaMemcpy(o1, d_o1, (size_t)nbatch * ldo * sizeof(double), cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(o2, d_o2, (size_t)nbatch * ldo * sizeof(double), cudaMemcpyDeviceToHost));
    }
    return TC_OK;
}

extern "C" {

int tc_ss_batch(const tc_cells *c, int64_t nbatch, const int32_t *cell_id, const double *theta, int ld, int algo,
                double *ss_out)
{
    if (!ss_out && nbatch > 0) return fail(TC_EINVAL, "ss_out is NULL");
    return ss_host(c, nbatch, cell_id, theta, ld, algo, 0, ss_out, nullptr, nullptr, 0);
}

int tc_forward(const tc_cells *c, int64_t nbatch, const int32_t *cell_id, const double *theta, int ld, int on_raw_grid,
               double *ms2_out, double *pp7_out, int ldo)
{
    if (!ms2_out || !pp7_out) return fail(TC_EINVAL, "output is NULL");
    return ss_host(c, nbatch, cell_id, theta, ld, TC_ALGO_PAIRS, on_raw_grid ? 1 : 0, nullptr, ms2_out, pp7_out, ldo);
}

}  // extern "C"

// ------------------------------------------------------------------------------------- mcmc run
// The launch plan of one device's share of a fit: sampler kernel, shared-memory layout and schedule.  Pure functions of
// the device's numbers decide it, so that the policy is checked on the host (tests/stubs/layout_check.cu).
struct LaunchPlan {
    bool warp = false;                    // dram_warp_kernel (one warp per chain), else dram_kernel (one CTA per chain)
    int big = 0, threads = 0, wsz = 0, grid = 0, seglen = 0, solo_lag = 0;
    size_t smem = 0, nslots = 0;          // dynamic shared memory per CTA; dram_warp_kernel: chain slots (per-warp gInc, gSc, gW)
    std::string err;                      // non-empty: max(N) fits no layout the options allow (TC_EINVAL)
};

// Kernel and layout for nc chains on cells of up to Nmax points, on a device of sms SMs with optin bytes of opt-in shared
// memory per block; static_cta / static_warp: the static shared memory of dram_kernel / dram_warp_kernel.
static LaunchPlan plan_layout(int Nmax, int nc, int layout, int sms, int optin, size_t static_cta, size_t static_warp)
{
    LaunchPlan p;
    const int npmax = 7 + Nmax;
    const size_t avail = (size_t)optin > static_cta ? (size_t)optin - static_cta : 0;
    // regular layout when the Cholesky workspace fits in one SM's shared memory, else the big one
    p.big = (sizeof(double) * (size_t)dram_smem_doubles(Nmax, 0) > avail || layout == TC_LAYOUT_BIG) ? 1 : 0;
    // Many chains per SM: one warp per chain (dram_warp_kernel, tc_warp.cuh) instead of one CTA per chain.  The CTA kernel
    // buys latency with speculation and wins while there are about as many chains as CTA slots (measured crossover on
    // B200: ~13 chains per SM); beyond that the warp kernel does no wasted evaluations and no CTA barriers.
    const size_t smem_w = sizeof(double) * (size_t)wk_region(Nmax) * WK_WARPS;
    const bool warp_fits = smem_w + static_warp <= (size_t)optin && npmax <= 32 * WK_PIT;
    if (layout == TC_LAYOUT_WARP && !warp_fits) {
        p.err = "max(N) = " + std::to_string(Nmax) + " is too large for the chain-per-warp layout";
        return p;
    }
    p.warp = layout == TC_LAYOUT_WARP || (layout == TC_LAYOUT_AUTO && warp_fits && !p.big && nc >= TC_WARP_MIN_CHAINS_PER_SM * sms);   // TC_LAYOUT_CTA / _BIG: never
    if (p.warp) { p.big = 0; p.threads = WK_THREADS; p.smem = smem_w; return p; }
    p.wsz = dram_wsz(Nmax, p.big);
    p.threads = DRAM_THREADS;
    p.smem = sizeof(double) * (size_t)dram_smem_doubles(Nmax, p.big);
    // (big layout: gen_increments_tma keeps at most GENB_MAXT column tiles of 8 per warp in registers)
    if (p.smem > avail || (npmax + 3) / 4 > 255 || (p.big && npmax > 8 * SPEC * GENB_MAXT))
        p.err = "max(N) = " + std::to_string(Nmax) + " is too large for the shared-memory layout of this build "
                "(one CTA per chain: the cell, the chain state, 8 proposal slots and 8 forward-model scratch areas must fit in one SM)";
    return p;
}

// Grid and time slices of the planned kernel for nc chains of nsimu steps, with per_sm of its CTAs resident per SM;
// solo_lag and nseg: the solo-SM rule's lag and slices per chain (TC_SOLO_LAG, TC_SOLO_NSEG).
static void plan_schedule(LaunchPlan &p, int nc, int nsimu, int adaptint, int sms, int per_sm, int solo_lag, int nseg)
{
    // time slices: ~32 per chain, each ending on an adaptation step (a slice parks no partial covariance block): a multiple
    // of adaptint, and of 2 when adaptint = 1 (the first adaptation is at isimu = 2, so k = 1 would split the first block)
    const int unit = adaptint > 1 ? adaptint : (adaptint == 1 ? 2 : 1);
    long long sl = ((long long)nsimu + 31) / 32;
    if (p.warp) {
        // persistent grid, one item = WK_WARPS consecutive chains.  (More, shorter slices were measured for the one-wave
        // case — 2 392 chains = 150 groups on 148 SMs — and change nothing: 0.589 s with 29 slices, 0.599 s with 200; what
        // bounds that case is its slowest group, whose slices are sequential.)
        p.grid = std::max(1, std::min(per_sm * sms, (nc + WK_WARPS - 1) / WK_WARPS));
        p.nslots = (size_t)p.grid * WK_WARPS;
    } else {
        if (nc >= TC_UNSLICED_CHAINS) sl = nsimu;
        else if (per_sm == 2 && nc > sms) {
            // about as many chains as CTA slots, two CTAs per SM: lagging chains get an SM to themselves (dram_kernel's
            // claim loop); finer slices, so that the neighbour of such a chain gives way soon
            p.solo_lag = solo_lag;
            if (solo_lag > 0) sl = std::max<long long>(((long long)nsimu + nseg - 1) / nseg, 4LL * unit);
        }
        p.grid = std::min(nc, per_sm * sms);             // persistent grid = resident CTA slots: slices may wait on each other
    }
    sl = ((sl + unit - 1) / unit) * unit;
    p.seglen = (int)std::max<long long>(sl, unit);
}

// Static partition over ngpus devices, at most one per chain: contiguous blocks of ~equal work (work ~ N^2 per step), none
// empty.  Device g runs chains [b[g], b[g + 1]).
static std::vector<int> partition_chains(const std::vector<int> &N, const int32_t *chain_cell, int nchains, int ngpus)
{
    ngpus = std::min(ngpus, nchains);
    std::vector<double> wk(nchains + 1, 0.0);
    for (int i = 0; i < nchains; ++i) { const double n = N[chain_cell[i]]; wk[i + 1] = wk[i] + n * n; }
    std::vector<int> b(ngpus + 1, nchains);
    b[0] = 0;
    for (int g = 0; g + 1 < ngpus; ++g) {
        const double target = wk[nchains] * (g + 1) / ngpus;
        const int end = (int)(std::lower_bound(wk.begin(), wk.end(), target) - wk.begin());
        b[g + 1] = std::min(std::max(end, b[g] + 1), nchains - (ngpus - 1 - g));
    }
    return b;
}

// does any adaptation with a covariance ever happen?
static bool cov_adaptations(const tc_mcmc_opts *o)
{
    if (o->adaptint > 0)
        for (long long m = o->adaptint; m <= o->nsimu; m += o->adaptint) if (m >= o->burnintime) return true;
    return false;
}

// The dataset's scratch pool on dc's device, created on first use; nullptr where the device has no stream-ordered pools.
static cudaMemPool_t scratch_pool(const DevCells *dc)
{
    int pools = 0;
    if (!dc->pool && cudaDeviceGetAttribute(&pools, cudaDevAttrMemoryPoolsSupported, dc->device) == cudaSuccess && pools) {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dc->device;
        cudaMemPool_t pool = nullptr;
        if (cudaMemPoolCreate(&pool, &props) == cudaSuccess) {
            unsigned long long keep = ~0ULL;                  // our own pool: keep the scratch between fits
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            dc->pool = pool;
        } else {
            (void)cudaGetLastError();
        }
    }
    return dc->pool;
}

struct DevRun {
    int device = -1, c0 = 0, c1 = 0;      // chains [c0, c1)
    LaunchPlan plan;
    DevBuf buf;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    RunArgs a{};
    ~DevRun()
    {
        if (device >= 0) cudaSetDevice(device);
        buf.release();                                  // stream-ordered frees need the stream
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    }
};

template <typename T>
static cudaError_t up(DevBuf &b, T *&d, const T *h, size_t n, cudaStream_t st)
{
    cudaError_t e = b.alloc(d, n);
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, st);
}

// params{i} = {name, init, lo, hi, mu, sig} (TranscriptionCycleMCMC.m:242-255): mcmcstat refuses an initial value outside
// its bounds; a prior width that is zero, negative or NaN would make the prior sum NaN and the chain would never accept
static int check_params(const tc_cells *c, int nchains, const int32_t *chain_cell, int ld, const double *theta0,
                        const double *qcov_diag, const double *low, const double *upp, const double *prior_mu,
                        const double *prior_sig)
{
    for (size_t i = 0; i < (size_t)nchains; ++i)
        for (int p = 0; p < 7 + c->N[chain_cell[i]]; ++p) {
            const size_t e = i * ld + p;
            const char *what = nullptr;
            if (!(qcov_diag[e] > 0)) what = "qcov_diag must be > 0";
            else if (!(low[e] <= upp[e])) what = "low must be <= upp";
            else if (!(theta0[e] >= low[e] && theta0[e] <= upp[e])) what = "theta0 must lie inside [low, upp]";
            else if (!(prior_sig[e] > 0)) what = "prior_sig must be > 0 (Inf = flat)";
            else if (std::isnan(prior_mu[e])) what = "prior_mu is NaN";
            if (what) return fail(TC_EINVAL, std::string(what) + " (chain " + std::to_string(i) + ", parameter " + std::to_string(p) + ")");
        }
    return TC_OK;
}

// The thinning of the stored rows: thin, validated by tc_mcmc_run when rows are stored, and ignored (1) when they are not
static int stored_thin(const tc_mcmc_opts *o) { return o->store_chain ? o->thin : 1; }

// The sampler of a launch: dram_warp_kernel or dram_kernel, compiled for thinned rows when thin > 1 is stored
static void (*sampler_kernel(bool warp, bool thin))(RunArgs)
{
    if (warp) return thin ? dram_warp_kernel<true> : dram_warp_kernel<false>;
    return thin ? dram_kernel<true> : dram_kernel<false>;
}

// One device's share of a fit, chains [r.c0, r.c1): its stream, events and scratch pool, RunArgs from the options and
// r.plan, the chains' inputs uploaded, outputs and scratch allocated.
static int setup_run(DevRun &r, const tc_cells *c, const tc_mcmc_opts *o, int ld, const int32_t *chain_cell,
                     const uint64_t *chain_uid, const double *theta0, const double *qcov_diag, const double *low,
                     const double *upp, const double *prior_mu, const double *prior_sig, const tc_replay *rp)
{
    const int nc = r.c1 - r.c0, Nmax = c->Nmax;
    const int thin = stored_thin(o);
    const size_t nkeep = thin_nkeep(o->nsimu, o->n_burn, thin), ns2 = thin_ns2(o->nsimu, thin);
    const size_t o0 = (size_t)r.c0;
    const int ldR = tri_doubles(7 + Nmax);               // proposal factor / scatter matrix in 4x4 tiles (chol_tiled)
    const bool do_cov = cov_adaptations(o);
    const LaunchPlan &p = r.plan;
    const DevCells *dc = find_dev(c, r.device);
    CUDA_TRY(cudaSetDevice(r.device));
    CUDA_TRY(cudaStreamCreateWithFlags(&r.st, cudaStreamNonBlocking));
    if (cudaMemPool_t pool = scratch_pool(dc)) { r.buf.st = r.st; r.buf.pool = pool; r.buf.pooled = true; }
    CUDA_TRY(cudaEventCreate(&r.e0));
    CUDA_TRY(cudaEventCreate(&r.e1));
    RunArgs &a = r.a;
    a.cells = dc->d; a.cons = make_consx(c->cons);
    a.nsimu = o->nsimu; a.burnintime = o->burnintime; a.adaptint = o->adaptint; a.ntry = o->ntry;
    a.updatesigma = o->updatesigma; a.burnin_cumulative = o->burnin_cumulative; a.n_burn = o->n_burn;
    a.store_chain = o->store_chain; a.replay = o->replay; a.algo = o->algo; a.qcovadj_always = o->qcovadj_always;
    a.thin = thin; a.nkeep = (int)nkeep;
    a.drscale = o->drscale; a.adascale = o->adascale; a.qcovadj = o->qcovadj; a.burnin_scale = o->burnin_scale;
    a.N0 = o->N0; a.S20 = o->S20; a.sigma2_0 = o->sigma2_0; a.seed = o->seed;
    a.nchains = nc; a.ld = ld; a.nmax = Nmax; a.ldR = ldR; a.do_cov = do_cov ? 1 : 0;
    a.big = p.big; a.wsz = p.wsz; a.seglen = p.seglen; a.solo_lag = p.solo_lag;
    // the first block is rows 0 .. isimu-1 of the first adaptation (row 0 is x0, no step): with adaptint = 1 that is 2 rows
    a.blk_rows = std::max(o->adaptint, 2);
    int *d_cell; unsigned long long *d_uid; double *d;
    CUDA_TRY(up(r.buf, d_cell, (const int *)chain_cell + o0, nc, r.st)); a.chain_cell = d_cell;
    std::vector<unsigned long long> uid(nc);
    for (int i = 0; i < nc; ++i) uid[i] = chain_uid ? chain_uid[o0 + i] : (unsigned long long)(o0 + i);
    CUDA_TRY(r.buf.alloc(d_uid, nc));
    CUDA_TRY(cudaMemcpyAsync(d_uid, uid.data(), nc * sizeof(unsigned long long), cudaMemcpyHostToDevice, r.st)); a.chain_uid = d_uid;   // pageable source: staged before the call returns
    CUDA_TRY(up(r.buf, d, theta0 + o0 * ld, (size_t)nc * ld, r.st)); a.theta0 = d;
    CUDA_TRY(up(r.buf, d, qcov_diag + o0 * ld, (size_t)nc * ld, r.st)); a.qcov_diag = d;
    CUDA_TRY(up(r.buf, d, low + o0 * ld, (size_t)nc * ld, r.st)); a.low = d;
    CUDA_TRY(up(r.buf, d, upp + o0 * ld, (size_t)nc * ld, r.st)); a.upp = d;
    CUDA_TRY(up(r.buf, d, prior_mu + o0 * ld, (size_t)nc * ld, r.st)); a.pmu = d;
    CUDA_TRY(up(r.buf, d, prior_sig + o0 * ld, (size_t)nc * ld, r.st)); a.psig = d;
    CUDA_TRY(r.buf.alloc(a.mean, (size_t)nc * ld)); CUDA_TRY(cudaMemsetAsync(a.mean, 0, (size_t)nc * ld * 8, r.st));
    CUDA_TRY(r.buf.alloc(a.std, (size_t)nc * ld)); CUDA_TRY(cudaMemsetAsync(a.std, 0, (size_t)nc * ld * 8, r.st));
    CUDA_TRY(r.buf.alloc(a.sig, (size_t)nc * 2));
    CUDA_TRY(r.buf.alloc(a.counters, (size_t)nc * TC_NCOUNTERS));
    if (o->store_chain) {
        CUDA_TRY(r.buf.alloc(a.chain, (size_t)nc * nkeep * ld));
        CUDA_TRY(cudaMemsetAsync(a.chain, 0, (size_t)nc * nkeep * ld * 8, r.st));
        CUDA_TRY(r.buf.alloc(a.s2chain, (size_t)nc * ns2));
        CUDA_TRY(cudaMemsetAsync(a.s2chain, 0, (size_t)nc * ns2 * 8, r.st));
    }
    if (o->replay) {
        const size_t nz = (size_t)nc * o->nsimu * ld, nu = (size_t)nc * o->nsimu;
        CUDA_TRY(up(r.buf, d, rp->z1 + o0 * o->nsimu * ld, nz, r.st)); a.z1 = d;
        CUDA_TRY(up(r.buf, d, rp->z2 + o0 * o->nsimu * ld, nz, r.st)); a.z2 = d;
        CUDA_TRY(up(r.buf, d, rp->u1 + o0 * o->nsimu, nu, r.st)); a.u1 = d;
        CUDA_TRY(up(r.buf, d, rp->u2 + o0 * o->nsimu, nu, r.st)); a.u2 = d;
        CUDA_TRY(up(r.buf, d, rp->chi2 + o0 * o->nsimu, nu, r.st)); a.chi2 = d;
    }
    if (rp && rp->flags) CUDA_TRY(r.buf.alloc(a.flags, (size_t)nc * o->nsimu));
    if (rp && rp->sschain) CUDA_TRY(r.buf.alloc(a.sschain, (size_t)nc * o->nsimu));
    // scratch
    CUDA_TRY(r.buf.alloc(a.gR, (size_t)nc * ldR));
    if (do_cov) {
        CUDA_TRY(r.buf.alloc(a.gM2, (size_t)nc * ldR));
        CUDA_TRY(r.buf.alloc(a.gRows, (size_t)nc * a.blk_rows * ld));
        CUDA_TRY(r.buf.alloc(a.gWts, (size_t)nc * a.blk_rows));
        CUDA_TRY(r.buf.alloc(a.gCmean, (size_t)nc * ld));
    }
    CUDA_TRY(r.buf.alloc(a.smctl, 1024));
    CUDA_TRY(cudaMemsetAsync(a.smctl, 0, sizeof(int) * 1024, r.st));
    CUDA_TRY(r.buf.alloc(a.gState, (size_t)nc * state_doubles(ld)));
    CUDA_TRY(r.buf.alloc(a.cstate, nc));
    CUDA_TRY(cudaMemsetAsync(a.cstate, 0, sizeof(int) * nc, r.st));
    if (p.warp) {
        const int ldp = wk_ldp(Nmax);
        CUDA_TRY(r.buf.alloc(a.gPinv, (size_t)nc * ld));
        CUDA_TRY(r.buf.alloc(a.gInc, p.nslots * 2 * WK_GEN * ldp));
        CUDA_TRY(r.buf.alloc(a.gSc, p.nslots * 8 * WK_GEN));
        CUDA_TRY(r.buf.alloc(a.wq, 1));
        CUDA_TRY(cudaMemsetAsync(a.wq, 0, sizeof(unsigned long long), r.st));
        if (do_cov) {
            CUDA_TRY(r.buf.alloc(a.gMb, (size_t)nc * ld));
            CUDA_TRY(r.buf.alloc(a.gW, p.nslots * ldR));
        }
    } else if (p.big && do_cov) {
        CUDA_TRY(r.buf.alloc(a.gW, (size_t)p.grid * ldR));
    }
    return TC_OK;
}

extern "C" {

int tc_mcmc_run(const tc_cells *c, const tc_mcmc_opts *o, int nchains, const int32_t *chain_cell,
                const uint64_t *chain_uid, int ld, const double *theta0, const double *qcov_diag, const double *low,
                const double *upp, const double *prior_mu, const double *prior_sig, double *mean, double *std,
                double *sig, int64_t *counters, double *chain, double *s2chain, const tc_replay *rp)
{
    if (!c || !o) return fail(TC_EINVAL, "cells/opts is NULL");
    if (nchains < 1) return fail(TC_EINVAL, "nchains < 1");
    if (!chain_cell || !theta0 || !qcov_diag || !low || !upp || !prior_mu || !prior_sig) return fail(TC_EINVAL, "NULL chain input");
    if (ld < 7 + c->Nmax) return fail(TC_EINVAL, "ld < 7 + max(N)");
    if (o->nsimu < 1) return fail(TC_EINVAL, "nsimu < 1");
    if (o->n_burn < 1 || o->n_burn > o->nsimu) return fail(TC_EINVAL, "n_burn must be in [1, nsimu]");
    if (o->store_chain && o->thin < 1) return fail(TC_EINVAL, "thin must be >= 1");
    if (o->ntry < 1 || o->ntry > 2) return fail(TC_EINVAL, "ntry must be 1 or 2");
    if (!(o->drscale > 0)) return fail(TC_EINVAL, "drscale must be > 0");
    if (o->algo != TC_ALGO_PAIRS && o->algo != TC_ALGO_TOEPLITZ) return fail(TC_EINVAL, "unknown algo");
    if (o->adaptint < 0 || o->adaptint > 2048) return fail(TC_EINVAL, "adaptint must be in [0, 2048]");
    if (o->replay && (!rp || !rp->z1 || !rp->u1 || !rp->z2 || !rp->u2 || !rp->chi2)) return fail(TC_EINVAL, "replay streams missing");
    if (o->store_chain && (!chain || !s2chain)) return fail(TC_EINVAL, "store_chain set but chain/s2chain is NULL");
    for (int i = 0; i < nchains; ++i)
        if (chain_cell[i] < 0 || chain_cell[i] >= c->ncells) return fail(TC_EINVAL, "chain_cell out of range");
    if (const int rc = check_params(c, nchains, chain_cell, ld, theta0, qcov_diag, low, upp, prior_mu, prior_sig)) return rc;
    DeviceGuard guard;                                    // declared before `runs`: restores the caller's device last

    // devices: 'numParPools' => GPU count
    const int ngpus = std::max(1, o->ngpus);
    std::vector<int> devs;
    for (int g = 0; g < ngpus; ++g) devs.push_back(o->devices[0] >= 0 ? o->devices[g] : c->dev[std::min<size_t>(g, c->dev.size() - 1)].device);
    if (o->devices[0] < 0 && ngpus > (int)c->dev.size()) return fail(TC_EINVAL, "ngpus exceeds the devices the cells were uploaded to");
    for (int d : devs) if (!find_dev(c, d)) return fail(TC_EINVAL, "cells not resident on a requested device");
    const std::vector<int> part = partition_chains(c->N, chain_cell, nchains, ngpus);
    std::vector<DevRun> runs(part.size() - 1);
    for (size_t g = 0; g < runs.size(); ++g) { runs[g].device = devs[g]; runs[g].c0 = part[g]; runs[g].c1 = part[g + 1]; }

    // every device's plan before any device work: a series length no allowed layout takes is refused here
    const char *e1 = getenv("TC_SOLO_LAG"), *e2 = getenv("TC_NSEG");          // development switches
    const int solo_lag = e1 ? atoi(e1) : TC_SOLO_LAG, nseg = e2 ? atoi(e2) : TC_SOLO_NSEG;
    for (auto &r : runs) {
        int optin = 0, sms = 0, per_sm = 0;
        cudaFuncAttributes fa, faw;
        CUDA_TRY(cudaSetDevice(r.device));
        CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, r.device));
        CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, r.device));
        CUDA_TRY(cudaFuncGetAttributes(&fa, dram_kernel<false>));
        CUDA_TRY(cudaFuncGetAttributes(&faw, dram_warp_kernel<false>));
        LaunchPlan &p = r.plan = plan_layout(c->Nmax, r.c1 - r.c0, o->layout, sms, optin, fa.sharedSizeBytes, faw.sharedSizeBytes);
        if (!p.err.empty()) return fail(TC_EINVAL, p.err);
        const auto kernel = sampler_kernel(p.warp, stored_thin(o) > 1);
        CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, p.threads, p.smem));
        if (per_sm < 1) return fail(TC_EINVAL, p.warp ? "chain-per-warp kernel does not fit on this device" : "sampler kernel does not fit on this device");
        plan_schedule(p, r.c1 - r.c0, o->nsimu, o->adaptint, sms, per_sm, solo_lag, nseg);
    }
    for (auto &r : runs) {
        const int rc = setup_run(r, c, o, ld, chain_cell, chain_uid, theta0, qcov_diag, low, upp, prior_mu, prior_sig, rp);
        if (rc) return rc;
        const auto kernel = sampler_kernel(r.plan.warp, stored_thin(o) > 1);
        CUDA_TRY(cudaEventRecord(r.e0, r.st));
        kernel<<<r.plan.grid, r.plan.threads, r.plan.smem, r.st>>>(r.a);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(r.e1, r.st));
    }
    // Drain: every device's outputs go back on its own stream; with several devices one host thread per device, so the
    // device -> host copies (raw chains: GBs) of the 8 GPUs overlap instead of queueing behind each other.
    const auto t_drain0 = std::chrono::steady_clock::now();
    const int thin = stored_thin(o);
    const size_t nkeep = thin_nkeep(o->nsimu, o->n_burn, thin), ns2 = thin_ns2(o->nsimu, thin);
    std::vector<int64_t> cnt_tmp;
    if (!counters) { cnt_tmp.assign((size_t)nchains * TC_NCOUNTERS, 0); counters = cnt_tmp.data(); }   // TC_CNT_STATUS is always checked
    std::vector<double> ksec(runs.size(), 0.0);
    std::vector<int> rcs(runs.size(), TC_OK);
    std::vector<std::string> errs(runs.size());
    auto drain = [&](size_t g) -> int {
        DevRun &r = runs[g];
        const int nc = r.c1 - r.c0;
        const size_t o0 = (size_t)r.c0;
        CUDA_TRY(cudaSetDevice(r.device));
        RunArgs &a = r.a;
        cudaStream_t st = r.st;
        if (mean) CUDA_TRY(cudaMemcpyAsync(mean + o0 * ld, a.mean, (size_t)nc * ld * 8, cudaMemcpyDeviceToHost, st));
        if (std) CUDA_TRY(cudaMemcpyAsync(std + o0 * ld, a.std, (size_t)nc * ld * 8, cudaMemcpyDeviceToHost, st));
        if (sig) CUDA_TRY(cudaMemcpyAsync(sig + o0 * 2, a.sig, (size_t)nc * 2 * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(counters + o0 * TC_NCOUNTERS, a.counters, (size_t)nc * TC_NCOUNTERS * 8, cudaMemcpyDeviceToHost, st));
        if (o->store_chain) {
            CUDA_TRY(cudaMemcpyAsync(chain + o0 * nkeep * ld, a.chain, (size_t)nc * nkeep * ld * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(s2chain + o0 * ns2, a.s2chain, (size_t)nc * ns2 * 8, cudaMemcpyDeviceToHost, st));
        }
        if (rp && rp->flags) CUDA_TRY(cudaMemcpyAsync(rp->flags + o0 * o->nsimu, a.flags, (size_t)nc * o->nsimu * 4, cudaMemcpyDeviceToHost, st));
        if (rp && rp->sschain) CUDA_TRY(cudaMemcpyAsync(rp->sschain + o0 * o->nsimu, a.sschain, (size_t)nc * o->nsimu * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, r.e0, r.e1));
        ksec[g] = (double)ms * 1e-3;
        return TC_OK;
    };
    if (runs.size() == 1) {
        rcs[0] = drain(0);
        if (rcs[0]) return rcs[0];
    } else {
        std::vector<std::thread> th;
        for (size_t g = 0; g < runs.size(); ++g)
            th.emplace_back([&, g]() { rcs[g] = drain(g); if (rcs[g]) errs[g] = g_err; });
        for (auto &t : th) t.join();
        for (size_t g = 0; g < runs.size(); ++g) if (rcs[g]) return fail(rcs[g], errs[g]);
    }
    double kmax = 0.0;
    for (double k : ksec) kmax = std::max(kmax, k);
    g_last_kernel_s = kmax;
    // host time from the last launch to the last byte on the host, minus the kernel: the device -> host copies
    g_last_drain_s = std::max(0.0, std::chrono::duration<double>(std::chrono::steady_clock::now() - t_drain0).count() - kmax);
    for (int i = 0; i < nchains; ++i)
        if (counters[(size_t)i * TC_NCOUNTERS + TC_CNT_STATUS] != 0)
            return fail(TC_ESTATE, "ss(theta0) is not finite for chain " + std::to_string(i));
    return TC_OK;
}

int tc_rng_dump(uint64_t seed, uint64_t chain_uid, int npar, double chi2_dof, int nsimu, double *z1, double *u1,
                double *z2, double *u2, double *chi2, int device)
{
    if (npar < 1 || nsimu < 1 || !z1 || !u1 || !z2 || !u2 || !chi2) return fail(TC_EINVAL, "bad argument");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return fail(TC_ENODEV, "no such CUDA device");
    DeviceGuard guard;
    CUDA_TRY(cudaSetDevice(device));
    DevBuf b;
    double *dz1, *dz2, *du1, *du2, *dc2;
    CUDA_TRY(b.alloc(dz1, (size_t)nsimu * npar)); CUDA_TRY(b.alloc(dz2, (size_t)nsimu * npar));
    CUDA_TRY(b.alloc(du1, nsimu)); CUDA_TRY(b.alloc(du2, nsimu)); CUDA_TRY(b.alloc(dc2, nsimu));
    rng_dump_kernel<<<std::min(nsimu, 1024), 128>>>(seed, chain_uid, npar, chi2_dof, nsimu, dz1, du1, dz2, du2, dc2);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(z1, dz1, (size_t)nsimu * npar * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(z2, dz2, (size_t)nsimu * npar * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(u1, du1, (size_t)nsimu * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(u2, du2, (size_t)nsimu * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(chi2, dc2, (size_t)nsimu * 8, cudaMemcpyDeviceToHost));
    return TC_OK;
}

int tc_debug_subprof(long long *out, int n)
{
#ifdef TC_SUBPROF
    long long h[32];
    CUDA_TRY(cudaMemcpyFromSymbol(h, tc_subprof, sizeof(h)));
    for (int i = 0; i < n && i < 32; ++i) out[i] = h[i];
    std::memset(h, 0, sizeof(h));
    CUDA_TRY(cudaMemcpyToSymbol(tc_subprof, h, sizeof(h)));
    return 1;
#else
    for (int i = 0; i < n; ++i) out[i] = 0;
    return 0;
#endif
}

int tc_measure_fp64_peak(int device, double *dfma_per_s, double *sm_clock_mhz)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return fail(TC_ENODEV, "no such CUDA device");
    DeviceGuard guard;
    CUDA_TRY(cudaSetDevice(device));
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    const int blocks = sms * 8, threads = 256, iters = 1 << 16;
    DevBuf b;
    double *out; long long *clk;
    CUDA_TRY(b.alloc(out, (size_t)blocks * threads));
    CUDA_TRY(b.alloc(clk, blocks));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    double best = 0, clk_mhz = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(cudaEventRecord(e0));
        dfma_peak_kernel<<<blocks, threads>>>(out, clk, iters);
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double rate = (double)blocks * threads * 8.0 * iters / (ms * 1e-3);
        if (rate > best) {
            best = rate;
            // one wave of 8 CTAs/SM runs concurrently: per-CTA cycles / kernel time ~ SM clock
            std::vector<long long> h(blocks);
            CUDA_TRY(cudaMemcpy(h.data(), clk, blocks * sizeof(long long), cudaMemcpyDeviceToHost));
            long long mx = 0;
            for (long long v : h) mx = std::max(mx, v);
            clk_mhz = (double)mx / (ms * 1e-3) * 1e-6;
        }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (dfma_per_s) *dfma_per_s = best;
    if (sm_clock_mhz) *sm_clock_mhz = clk_mhz;
    return TC_OK;
}

}  // extern "C"
