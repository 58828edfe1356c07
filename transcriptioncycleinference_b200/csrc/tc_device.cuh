// tc_device.cuh — device-side building blocks of libtcmcmc (sm_100a).
//
//  * Philox4x32-10 counter-based RNG, Box-Muller normals, Marsaglia-Tsang chi-square
//  * warp-shuffle reductions
//  * the forward model + residual sum of squares for one (cell, theta), evaluated by ONE WARP (no
//    block barriers), scratch in shared memory.  Behavioural spec: SURVEY.md Appendix B.2, i.e.
//      src/SumofSquaresFunction_TranscriptionCycleMCMC.m:28-64,
//      src/dependencies/ConstantElongationSim.m:33-67,
//      src/GetFluorFromPolPos.m:18-70            (paths relative to /root/reference).
//    Not a translation: the reference builds an m x n position matrix and makes ~10 masked passes
//    over it; here polymerases loaded in the same step form one cohort of integer size
//    n_i = floor(c_i) - floor(c_{i-1}) at position v*(t_j - t_i), so a row of the matrix collapses
//    to a (cohort, time) sum — evaluated either pair by pair (TC_ALGO_PAIRS) or, on the uniform
//    t_interp grid, through the banded structure of the per-lag response (TC_ALGO_TOEPLITZ).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/tcmcmc.h"

// The construct as the kernels see it: the caller's definition + what depends on it alone — the slope f / (e - s) of the ramp
// of every loop set, computed once on the host (an IEEE quotient, i.e. the very value the device's own division would give).
struct ConsX : tc_construct {
    double sc1[TC_MAX_SETS], sc2[TC_MAX_SETS];
};
inline ConsX make_consx(const tc_construct &c)
{
    ConsX x{};
    static_cast<tc_construct &>(x) = c;
    for (int s = 0; s < TC_MAX_SETS; ++s) {
        x.sc1[s] = s < c.nsets ? (c.ms2_loopn[s] * (1.0 / 24.0)) / (c.ms2_end[s] - c.ms2_start[s]) : 0.0;
        x.sc2[s] = s < c.nsets ? (c.pp7_loopn[s] * (1.0 / 24.0)) / (c.pp7_end[s] - c.pp7_start[s]) : 0.0;
    }
    return x;
}

namespace tc {
#ifdef TC_SS_PROFILE
__device__ long long tc_ss_prof[8];
#endif

// ------------------------------------------------------------------------------------------ RNG
__device__ double tc_exp(double x);
__device__ double tc_log(double x);
__device__ void tc_exp3(double x0, double x1, double x2, double &e0, double &e1, double &e2);
struct u32x4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ void philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2,
                                                      uint32_t &c3, uint32_t k0, uint32_t k1)
{
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__host__ __device__ __forceinline__ u32x4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                        uint32_t c3, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return u32x4{c0, c1, c2, c3};
}

// Stream kinds: which draw of MCMC step `step` a counter addresses.
enum { RK_Z1 = 0, RK_Z2 = 1, RK_U = 2, RK_CHI2 = 3 };

// counter = (slot, step, uid_lo, uid_hi[23:0] << 8 | kind); key = seed
__device__ __noinline__ u32x4 draw(uint64_t seed, uint64_t uid, uint32_t step, uint32_t kind,
                                      uint32_t slot)
{
    return philox4x32_10(slot, step, (uint32_t)uid, ((uint32_t)(uid >> 32) << 8) | kind,
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}

// 53-bit uniform in (0,1) from two 32-bit words
__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo)
{
    const uint64_t m = ((uint64_t)(hi >> 5) << 26) | (uint64_t)(lo >> 6);
    return ((double)m + 0.5) * (1.0 / 9007199254740992.0);
}

// two standard normals from one Philox block (Box-Muller, FP64)
__device__ __noinline__ void normal_pair(const u32x4 &r, double &z0, double &z1)
{
    const double ua = u01(r.x, r.y), ub = u01(r.z, r.w);
    const double rad = sqrt(-2.0 * log(ua));     // inlined here: overlaps with sincospi below
    double s, c;
    sincospi(2.0 * ub, &s, &c);
    z0 = rad * c;
    z1 = rad * s;
}

// The proposal normals (z1[2q], z1[2q+1], z2[2q], z2[2q+1]) of step `step`, parameters 2q and 2q+1, from ONE
// Philox block (kind RK_Z1, slot q): words (x, y) -> the stage-1 pair, (z, w) -> the stage-2 pair.
// Standard-normal VARIATES are a sampling device, not part of the likelihood arithmetic: they are drawn by
// Box-Muller in single precision (32-bit radius uniform => |z| <= 6.76, 24-bit angle) and widened to FP64;
// everything downstream (proposal, forward model, SS, acceptance) is FP64.  tc_rng_dump calls this very
// function, so the parity harness sees bit-identical draws.
__device__ __forceinline__ double4 normal_quad_inl(uint64_t seed, uint64_t uid, uint32_t step, uint32_t q)
{
    const u32x4 r = philox4x32_10(q, step, (uint32_t)uid, ((uint32_t)(uid >> 32) << 8) | RK_Z1, (uint32_t)seed, (uint32_t)(seed >> 32));
    const float ua1 = ((float)r.x + 0.5f) * 2.3283064365386963e-10f, ua2 = ((float)r.z + 0.5f) * 2.3283064365386963e-10f;   // (0, 1]
    const float ub1 = (float)(r.y >> 8) * 1.1920928955078125e-7f, ub2 = (float)(r.w >> 8) * 1.1920928955078125e-7f;       // [0, 2) turns / 2
    const float rad1 = sqrtf(-2.0f * logf(ua1)), rad2 = sqrtf(-2.0f * logf(ua2));
    float s1, c1, s2, c2;
    sincospif(ub1, &s1, &c1);
    sincospif(ub2, &s2, &c2);
    return make_double4((double)(rad1 * c1), (double)(rad1 * s1), (double)(rad2 * c2), (double)(rad2 * s2));
}
// one out-of-line copy for the callers that draw a block at a time (normal_quad_inl: callers that interleave several blocks)
__device__ __noinline__ double4 normal_quad(uint64_t seed, uint64_t uid, uint32_t step, uint32_t q) { return normal_quad_inl(seed, uid, step, q); }

// chi-square(dof) = 2*Gamma(dof/2) by Marsaglia-Tsang (dof >= 2); attempt t uses slots 2t (the normal: Box-Muller
// in single precision like the proposal normals, words x, y) and 2t+1 (the 53-bit uniform).
// d = dof/2 - 1/3 and c = 1/sqrt(9 d) are constants of a chain: chi2_consts() once, chi2_draw_dc() per draw
__device__ __forceinline__ void chi2_consts(double dof, double &d, double &c)
{
    d = 0.5 * dof - 1.0 / 3.0;
    c = 1.0 / sqrt(9.0 * d);
}
__device__ __noinline__ double chi2_draw_dc(uint64_t seed, uint64_t uid, uint32_t step, double d, double c)
{
    for (uint32_t t = 0; t < 64; ++t) {
        const u32x4 r0 = draw(seed, uid, step, RK_CHI2, 2 * t);
        const u32x4 r1 = draw(seed, uid, step, RK_CHI2, 2 * t + 1);
        const float ua = ((float)r0.x + 0.5f) * 2.3283064365386963e-10f, ub = (float)(r0.y >> 8) * 1.1920928955078125e-7f;
        const double x = (double)(sqrtf(-2.0f * logf(ua)) * cospif(ub));
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        const double u = u01(r1.x, r1.y);
        const double x2 = x * x;
        if (u < 1.0 - 0.0331 * x2 * x2) return 2.0 * d * v;
        if (tc_log(u) < 0.5 * x2 + d * (1.0 - v + tc_log(v))) return 2.0 * d * v;
    }
    return 2.0 * d;   // unreachable in practice (acceptance > 0.95 per attempt)
}
__device__ __forceinline__ double chi2_draw(uint64_t seed, uint64_t uid, uint32_t step, double dof)
{
    double d, c;
    chi2_consts(dof, d, c);
    return chi2_draw_dc(seed, uid, step, d, c);
}

// One out-of-line copy of the long libdevice sequences: the sampler's hot loop has to stay inside
// the instruction cache (ncu: icc hit rate 58 %, stall_no_instruction dominant before this).
__device__ __noinline__ double tc_exp(double x) { return exp(x); }
__device__ __noinline__ double tc_log(double x) { return log(x); }
// three independent exponentials in one body: their dependent chains interleave (the DRAM acceptance ratios)
__device__ __noinline__ void tc_exp3(double x0, double x1, double x2, double &e0, double &e1, double &e2)
{
    e0 = exp(x0); e1 = exp(x1); e2 = exp(x2);
}

// 1 / d to within an ulp or two: MUFU.RCP64H seed + two Newton steps (the IEEE quotient is ~25 dependent instructions with a
// slow-path branch; where this is used a product with the reciprocal replaces a quotient anyway)
__device__ __forceinline__ double tc_rcp(double d)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(fma(-d, r, 1.0), r, r);
    r = fma(fma(-d, r, 1.0), r, r);
    return r;
}

// ------------------------------------------------------------------------------- reductions
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------- shared-memory views
// All dynamic shared memory of the library's kernels is this one array.  The forward model addresses
// it by OFFSET (in doubles), never through generic pointers, so that every access compiles to
// LDS/STS with an immediate offset instead of a generic LD/ST plus pointer traffic through local
// memory (measured: ~2x on the latency of one evaluation).
extern __shared__ __align__(16) double tc_smem[];

// get4(i, ok, v): elements i .. i+3 (the four consecutive steps a lane owns in the loading scan); ok[e] says whether element
// e is wanted.  The aligned views fetch them as two 16-byte loads — a lane-stride of 32 bytes costs 2 shared-memory
// wavefronts per 8 lanes with 16-byte accesses, 4 with 8-byte ones (ncu: the 8-byte pattern was a quarter of all
// bank conflicts of the samplers) — and may read one element past the last wanted one (always inside the vector).
struct SmemVec {          // a vector in shared memory
    int off;
    __device__ __forceinline__ double operator[](int i) const { return tc_smem[off + i]; }
    __device__ __forceinline__ void get4(int i, const bool (&ok)[4], double (&v)[4]) const
    {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = ok[e] ? tc_smem[off + i + e] : 0.0;
    }
};
struct SmemVecA {         // ... whose element 7 (the first dR) is 16-byte aligned: off is ODD
    int off;
    __device__ __forceinline__ double operator[](int i) const { return tc_smem[off + i]; }
    __device__ __forceinline__ void get4(int i, const bool (&ok)[4], double (&v)[4]) const      // i - 7 a multiple of 4
    {
        double2 a = make_double2(0.0, 0.0), b = make_double2(0.0, 0.0);
        if (ok[0]) a = *reinterpret_cast<const double2 *>(tc_smem + off + i);
        if (ok[2]) b = *reinterpret_cast<const double2 *>(tc_smem + off + i + 2);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
};
struct SumVec {           // theta = state + proposal increment, both in shared memory (the increments of one stage are a plain
    int ox, os;           // vector); ox and os are ODD, like SmemVecA::off
    __device__ __forceinline__ double operator[](int i) const { return tc_smem[ox + i] + tc_smem[os + i]; }
    __device__ __forceinline__ void get4(int i, const bool (&ok)[4], double (&v)[4]) const      // i - 7 a multiple of 4
    {
        double2 xa = make_double2(0.0, 0.0), xb = xa, sa = xa, sb = xa;
        if (ok[0]) { xa = *reinterpret_cast<const double2 *>(tc_smem + ox + i); sa = *reinterpret_cast<const double2 *>(tc_smem + os + i); }
        if (ok[2]) { xb = *reinterpret_cast<const double2 *>(tc_smem + ox + i + 2); sb = *reinterpret_cast<const double2 *>(tc_smem + os + i + 2); }
        v[0] = xa.x + sa.x; v[1] = xa.y + sa.y; v[2] = xb.x + sb.x; v[3] = xb.y + sb.y;
    }
};
struct GlobVec {          // a vector in global memory
    const double *p;
    __device__ __forceinline__ double operator[](int i) const { return p[i]; }
    __device__ __forceinline__ void get4(int i, const bool (&ok)[4], double (&v)[4]) const
    {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = ok[e] ? p[i + e] : 0.0;
    }
};

// Where the loading scan reads the model grid and its steps: lane l of the warp owns the four consecutive steps
// 4l .. 4l+3 of a block of 128, so in shared memory tg / dtg are stored PERMUTED inside each block of 128 (a shorter last
// block: length blen, q = ceil(blen / 4)): step i sits at block + (i & 3) * q + ((i & 127) >> 2).  The four loads of a lane
// are then lane-contiguous (conflict-free) instead of 32 bytes apart (4 wavefronts per 8-byte load).  The dataset keeps
// permuted copies (CellsDev::tgp / dtgp, cell c at off[c] + 4 c, (N + 3) & ~3 entries), so staging a cell is a plain copy.
__host__ __device__ __forceinline__ int cell_perm(int N, int i)
{
    const int r0 = i & ~127, rem = N - r0, q = ((rem < 128 ? rem : 128) + 3) >> 2;
    return r0 + (i & 3) * q + ((i & 127) >> 2);
}
struct SmemCell {         // one cell's constants staged in shared memory (offsets into tc_smem)
    int N;
    double d;             // mean(diff(t))                       SumofSquares...m:29
    int o_tg, o_dtg, o_ms2, o_pp7, o_iw, o_ik;
    __device__ __forceinline__ double tg(int i) const { return tc_smem[o_tg + cell_perm(N, i)]; }     // model grid (permuted)
    __device__ __forceinline__ double dtg(int i) const { return tc_smem[o_dtg + cell_perm(N, i)]; }   // tg[i+1]-tg[i] (permuted)
    // steps r0 + 4 lane + e, e = 0..3, of the block of 128 starting at r0
    __device__ __forceinline__ void grid4(int r0, int lane, const bool (&ok)[4], double (&t)[4], double (&dt)[4]) const
    {
        const int q = (min(128, N - r0) + 3) >> 2, b = r0 + lane;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            t[e] = ok[e] ? tc_smem[o_tg + b + e * q] : 0.0;
            dt[e] = ok[e] ? tc_smem[o_dtg + b + e * q] : 0.0;
        }
    }
    __device__ __forceinline__ double ms2(int i) const { return tc_smem[o_ms2 + i]; }   // data, NaN = missing
    __device__ __forceinline__ double pp7(int i) const { return tc_smem[o_pp7 + i]; }
    __device__ __forceinline__ double iw(int i) const { return tc_smem[o_iw + i]; }     // interp1 weight
    __device__ __forceinline__ int ik(int i) const { return reinterpret_cast<const int *>(tc_smem + o_ik)[i]; }
};
struct GlobCell {         // the same view straight onto the device-resident dataset
    int N;
    double d;
    const double *p_tg, *p_dtg, *p_ms2, *p_pp7, *p_iw;
    const int *p_ik;
    __device__ __forceinline__ double tg(int i) const { return p_tg[i]; }
    __device__ __forceinline__ double dtg(int i) const { return p_dtg[i]; }
    __device__ __forceinline__ void grid4(int r0, int lane, const bool (&ok)[4], double (&t)[4], double (&dt)[4]) const
    {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            t[e] = ok[e] ? p_tg[r0 + 4 * lane + e] : 0.0;
            dt[e] = ok[e] ? p_dtg[r0 + 4 * lane + e] : 0.0;
        }
    }
    __device__ __forceinline__ double ms2(int i) const { return p_ms2[i]; }
    __device__ __forceinline__ double pp7(int i) const { return p_pp7[i]; }
    __device__ __forceinline__ double iw(int i) const { return p_iw[i]; }
    __device__ __forceinline__ int ik(int i) const { return p_ik[i]; }
};
// One warp's forward-model scratch.  n, F1, F2, thr: offsets in doubles into tc_smem, [N+2] each.  K and S (counts and first
// moments: integers) are kept as 32-BIT INTEGERS — half the shared-memory wavefronts of the per-time-point prefix differences,
// which are then exact integer subtractions — and are offsets in INTS into tc_smem_i(), = 3 mod 4: the scan stores
// K[4l+1 .. 4l+4] / S[...] of lane l as ONE aligned 16-byte store each.
struct Work {
    int K, n, S, F1, F2, thr;
};
__device__ __forceinline__ int *tc_smem_i() { return reinterpret_cast<int *>(tc_smem); }
__host__ __device__ inline int work_ks_doubles(int N) { return (((N + 9) >> 1) + 1) & ~1; }     // 3 + (N + 2) + 3 ints, even number of doubles
__host__ __device__ inline int work_doubles(int N) { return 3 * (N + 2) + 2 * work_ks_doubles(N) + 4 + 1; }
__host__ __device__ inline int cell_doubles(int N) { return 2 * ((N + 3) & ~3) + 3 * (N + 1) + (N + 2) / 2 + 1; }

// carve from offset `o` (doubles); returns the next free offset
__device__ inline int carve_cell(int o, int N, SmemCell &cv)
{
    cv.N = N;
    cv.o_tg = o; o += (N + 3) & ~3;
    cv.o_dtg = o; o += (N + 3) & ~3;
    cv.o_ms2 = o; o += N + 1;
    cv.o_pp7 = o; o += N + 1;
    cv.o_iw = o; o += N + 1;
    cv.o_ik = o; o += (N + 2) / 2 + 1;
    return o;
}
__device__ inline int carve_work(int o, int N, Work &w)
{
    o += o & 1;                                            // 16-byte align (thr is read as int4)
    w.thr = o; o += 4;
    w.K = 2 * o + 3; o += work_ks_doubles(N);              // ints; the 16-byte store of a lane may run up to three past K[n]
    w.S = 2 * o + 3; o += work_ks_doubles(N);
    w.n = o; o += N + 2;
    w.F1 = o; o += N + 2;
    w.F2 = o; o += N + 2;
    return o;
}

struct CellsDev {        // device-resident packed dataset (one per device)
    int ncells;
    const int *N;
    const long long *off;
    const double *t, *tg, *dtraw, *dtg, *ms2, *pp7, *iw, *dmean;
    const int *ik;
    const double *tgp, *dtgp;                      // tg / dtg in the shared-memory order (cell_perm), cell c at off[c] + 4 c
};

// copy cell `cid` (model grid) into its shared-memory view, by `nthr` threads of which this is thread `t`
__device__ __forceinline__ void stage_cell(const CellsDev &cd, int cid, const SmemCell &cv, int t, int nthr)
{
    const int N = cv.N, N4 = (N + 3) & ~3;
    const long long o = cd.off[cid], op = o + 4LL * cid;
    int *ikp = reinterpret_cast<int *>(tc_smem + cv.o_ik);
#pragma unroll 2
    for (int i = t; i < N4; i += nthr) {
        tc_smem[cv.o_tg + i] = cd.tgp[op + i];
        tc_smem[cv.o_dtg + i] = cd.dtgp[op + i];
        if (i < N) {
            tc_smem[cv.o_ms2 + i] = cd.ms2[o + i];
            tc_smem[cv.o_pp7 + i] = cd.pp7[o + i];
            tc_smem[cv.o_iw + i] = cd.iw[o + i];
            ikp[i] = cd.ik[o + i];
        }
    }
}

// stage cell `cid` (model grid) into shared memory (whole CTA)
__device__ inline void load_cell(const CellsDev &cd, int cid, SmemCell &cv)
{
    stage_cell(cd, cid, cv, threadIdx.x, blockDim.x);
    cv.d = cd.dmean[cid];
}
__device__ inline GlobCell view_cell(const CellsDev &cd, int cid, bool raw_grid)
{
    const long long o = cd.off[cid];
    GlobCell cv;
    cv.N = cd.N[cid];
    cv.d = cd.dmean[cid];
    cv.p_tg = (raw_grid ? cd.t : cd.tg) + o;
    cv.p_dtg = (raw_grid ? cd.dtraw : cd.dtg) + o;
    cv.p_ms2 = cd.ms2 + o;
    cv.p_pp7 = cd.pp7 + o;
    cv.p_iw = cd.iw + o;
    cv.p_ik = cd.ik + o;
    return cv;
}

// ------------------------------------------------------------------------- forward model pieces

// literal response of one loop set at position p  (GetFluorFromPolPos.m:49-52 / :61-64)
__device__ __forceinline__ double loop_response(double p, double s, double e, double L, double fv)
{
    double val = 0.0;
    if (p > e && p < L) val = fv;
    if (p > s && p < e) val = (p - s) * fv / (e - s);
    return val;
}

// per-step loading increment rho_i*delta_i; zero before onset (the reference `continue`s, which
// leaves the counter unchanged)                      ConstantElongationSim.m:33-36,57-60
template <class Cell, class Vec>
__device__ __forceinline__ double load_increment(const Cell &cv, const Vec &th, int i, double R, double ton)
{
    double r = R + th[7 + i];                                 // SumofSquares...m:45
    r = r < 0.0 ? 0.0 : r;
    return (cv.tg(i) < ton) ? 0.0 : __dmul_rn(r, cv.dtg(i));
}

// the reference's own order: one lane, sequential (rare fallback; kept out of line)
template <class Cell, class Vec>
__device__ __noinline__ void scan_counts_sequential(Cell cv, Vec th, double R, double ton, int oK)
{
    double c = 0.0;
    tc_smem_i()[oK] = 0;
#pragma unroll 1
    for (int i = 0; i < cv.N - 1; ++i) {
        c = __dadd_rn(c, load_increment(cv, th, i, R, ton));
        tc_smem_i()[oK + i + 1] = (int)floor(c);
    }
}

// Loaded-polymerase counts and their prefix sums by ONE warp:
//   K[0] = 0, K[i+1] = floor(counter after step i)   (= sum_{i'<=i} n_i')       ConstantElongationSim.m:53-61
//   n[i] = K[i+1] - K[i]                               cohort loaded in step i
//   S[m] = sum_{i<m} i n_i                             first moments (exact: integers, 32-bit integer shuffles)
// With K and S any ramp sum is O(1):  sum_{i=a}^{b} (j - i) n_i = j (K[b+1] - K[a]) - (S[b+1] - S[a]).
// floor() is discontinuous, so the running sum must give the same integers as the reference's sequential order
// with separately rounded products (no FMA contraction).  Fast path: every lane owns 4 consecutive steps (local
// prefix in the reference's own order), ONE warp scan of the lane totals per 128 steps; if any partial sum lands
// within 1e-7 of an integer — where a different association could flip a floor — lane 0 redoes the sum
// sequentially.  Error bound of either order: (N-1) * eps * max(c) < 400 * 1.1e-16 * 3e4 << 1e-7, so the two paths
// agree otherwise.
template <class Cell, class Vec>
__device__ __forceinline__ void scan_counts(const Cell &cv, const Vec &th, double R, double ton, const Work &w,
                                            bool force_sequential, bool want_n)
{
    const int lane = threadIdx.x & 31;
    const int n = cv.N - 1;                        // increments i = 0..n-1
    bool redo = force_sequential;
    if (!force_sequential) {
        double carry = 0.0;                        // running counter / its floor at the end of the previous block of 128
        int carryS = 0, fprev = 0;
        bool risky = false;
#pragma unroll 1
        for (int r0 = 0; r0 < n; r0 += 128) {
            const int i0 = r0 + 4 * lane;
            const bool ok[4] = {i0 < n, i0 + 1 < n, i0 + 2 < n, i0 + 3 < n};
            double p[4], thv[4], tgv[4], dtv[4];
            th.get4(7 + i0, ok, thv);
            cv.grid4(r0, lane, ok, tgv, dtv);
#pragma unroll
            for (int e = 0; e < 4; ++e) {                  // load_increment(), on the values fetched above
                double r = R + thv[e];
                r = r < 0.0 ? 0.0 : r;
                p[e] = (ok[e] && !(tgv[e] < ton)) ? __dmul_rn(r, dtv[e]) : 0.0;
            }
            p[1] = __dadd_rn(p[0], p[1]); p[2] = __dadd_rn(p[1], p[2]); p[3] = __dadd_rn(p[2], p[3]);
            double t = p[3];                       // inclusive scan of the lane totals
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double up = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t = __dadd_rn(t, up);
            }
            const double tot = __shfl_sync(0xffffffffu, t, 31);
            double excl = __shfl_up_sync(0xffffffffu, t, 1);
            if (lane == 0) excl = 0.0;
            const double base = __dadd_rn(carry, excl);
            double f[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double c = __dadd_rn(base, p[e]);
                f[e] = floor(c);
                const double fr = c - f[e];
                // c == 0: every increment so far is exactly 0 (they are all >= 0): exact in any order
                risky |= ok[e] && (c != 0.0) && (fr < 1e-7 || fr > 1.0 - 1e-7);
            }
            const int k0 = (int)f[0], k1 = (int)f[1], k2 = (int)f[2], k3 = (int)f[3];
            int fl = __shfl_up_sync(0xffffffffu, k3, 1);            // floor at the end of the previous lane
            if (lane == 0) fl = fprev;
            const int nn0 = k0 - fl, nn1 = k1 - k0, nn2 = k2 - k1, nn3 = k3 - k2;
            const int q0 = ok[0] ? i0 * nn0 : 0;
            const int q1 = q0 + (ok[1] ? (i0 + 1) * nn1 : 0);
            const int q2 = q1 + (ok[2] ? (i0 + 2) * nn2 : 0);
            const int q3 = q2 + (ok[3] ? (i0 + 3) * nn3 : 0);
            int ts = q3;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, ts, o);
                if (lane >= o) ts += up;
            }
            const int totS = __shfl_sync(0xffffffffu, ts, 31);
            int exS = __shfl_up_sync(0xffffffffu, ts, 1);
            if (lane == 0) exS = 0;
            exS += carryS;
            // K[i0+1 .. i0+4], S[...]: one aligned 16-byte store each; the elements past the last step repeat the last floor /
            // moment (steps beyond n add exactly 0) and nobody reads them
            if (ok[0]) {
                *reinterpret_cast<int4 *>(tc_smem_i() + w.K + i0 + 1) = make_int4(k0, k1, k2, k3);
                *reinterpret_cast<int4 *>(tc_smem_i() + w.S + i0 + 1) = make_int4(exS + q0, exS + q1, exS + q2, exS + q3);
            }
            if (want_n) {                                           // cohort sizes: only the pairs algorithm reads them
                if (ok[0]) tc_smem[w.n + i0] = (double)nn0;
                if (ok[1]) tc_smem[w.n + i0 + 1] = (double)nn1;
                if (ok[2]) tc_smem[w.n + i0 + 2] = (double)nn2;
                if (ok[3]) tc_smem[w.n + i0 + 3] = (double)nn3;
            }
            fprev = __shfl_sync(0xffffffffu, k3, 31);              // steps beyond n add exactly 0: lane 31 holds the block's last floor
            carry = __dadd_rn(carry, tot);
            carryS += totS;
        }
        if (lane == 0) { tc_smem_i()[w.K] = 0; tc_smem_i()[w.S] = 0; }
        redo = __any_sync(0xffffffffu, risky);
    }
    if (redo) {
        if (lane == 0) scan_counts_sequential(cv, th, R, ton, w.K);
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < n; i += 32) tc_smem[w.n + i] = (double)(tc_smem_i()[w.K + i + 1] - tc_smem_i()[w.K + i]);
        __syncwarp();
        if (lane == 0) {
            int sacc = 0;
            tc_smem_i()[w.S] = 0;
#pragma unroll 1
            for (int i = 0; i < n; ++i) { sacc += i * (tc_smem_i()[w.K + i + 1] - tc_smem_i()[w.K + i]); tc_smem_i()[w.S + i + 1] = sacc; }
        }
    }
}

// smallest lag in [1, N] with v*(d*lag) > x (strict) or >= x; N when none.  inv_vd = 1/(v d) only seeds
// the guess; membership is always decided by the exact predicate on p = v*(d*lag).
__device__ __forceinline__ int first_lag(double v, double d, double inv_vd, double x, int N, bool strict)
{
    if (!(v * d > 0.0)) return N;
    const double q = floor(x * inv_vd);
    int g = q < 1.0 ? 1 : (q > (double)N ? N : (int)q);
    auto pred = [&](int lag) {
        const double p = v * (d * (double)lag);
        return strict ? (p > x) : (p >= x);
    };
#pragma unroll 1
    while (g > 1 && pred(g - 1)) --g;
#pragma unroll 1
    while (g < N && !pred(g)) ++g;
    return g;
}

// TC_ALGO_PAIRS: every (cohort i, time j) pair with the literal response at p = v*(t_j - t_i); any grid
template <class Cell>
__device__ __noinline__ void rows_pairs(Cell cv, Work w, int s, double v, double s1, double e1, double L1,
                                        double f1, double b1, double s2, double e2, double L2, double f2, double b2)
{
    const int N = cv.N, lane = threadIdx.x & 31;
#pragma unroll 1
    for (int j = lane; j < N; j += 32) {
        double a1 = 0.0, a2 = 0.0;
        const double tj = cv.tg(j);
#pragma unroll 2
        for (int i = 0; i < j; ++i) {
            const double ni = tc_smem[w.n + i];
            if (ni > 0.0) {
                const double p = v * (tj - cv.tg(i));
                a1 = fma(ni, loop_response(p, s1, e1, L1, f1), a1);
                a2 = fma(ni, loop_response(p, s2, e2, L2, f2), a2);
            }
        }
        if (s > 0) { a1 += tc_smem[w.F1 + j]; a2 += tc_smem[w.F2 + j]; }
        tc_smem[w.F1 + j] = a1 < b1 ? b1 : a1;
        tc_smem[w.F2 + j] = a2 < b2 ? b2 : a2;
    }
}

#ifdef TC_SS_PROFILE
#define SS_MARK(i) do { const long long tn__ = clock64(); if (lane == 0) tc_ss_prof[i] += tn__ - tp__; tp__ = tn__; } while (0)
#else
#define SS_MARK(i)
#endif

// The residual sum of squares of one (cell, theta) — SumofSquares...m:1-65 — by ONE WARP.
// Cell / Vec say where the cell constants and theta live (shared memory in the sampler, global memory
// in the batched ssfun kernel); w is this warp's private scratch.  On return every lane holds SS.
// When out1/out2 != nullptr the model curves [A*MS2, PP7] on the model grid are also written there
// (tc_forward).  All 32 lanes must call this.
template <class Cell, class Vec>
__device__ __noinline__ double ss_eval(const ConsX &C, Cell cv, Vec th, Work w, int algo, bool seq_scan,
                                       double *out1, double *out2)
{
    const int N = cv.N, lane = threadIdx.x & 31;
    const double v = th[0], tau = th[1], ton = th[2], b1 = th[3], b2 = th[4], A = th[5], R = th[6];
#ifdef TC_SS_PROFILE
    long long tp__ = clock64();
#endif
    // 1 / (v d) only seeds the guesses of the lag thresholds (membership is decided by the exact predicate): the hardware's
    // approximate reciprocal (MUFU.RCP64H, ~20 bits) + one Newton step is plenty, and not the ~25 dependent instructions of a quotient
    const double vd = v * cv.d;
    double inv_vd;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(inv_vd) : "d"(vd));
    inv_vd = fma(fma(-vd, inv_vd, 1.0), inv_vd, inv_vd);
    // (a) loaded-polymerase counts K and cohort sizes n
    scan_counts(cv, th, R, ton, w, seq_scan, algo != TC_ALGO_TOEPLITZ);
    __syncwarp();
    SS_MARK(0);
    // (b) fluorescence per time point, one loop set at a time: the basal clamp sits inside the
    //     per-set loop in the reference (GetFluorFromPolPos.m:47,57,69)
    const double tv = tau * v;
    const double L1 = C.L_ms2 + tv, L2 = C.L_pp7 + tv;        // :19-20
#pragma unroll 1
    for (int s = 0; s < C.nsets; ++s) {
        const double s1 = C.ms2_start[s], e1 = C.ms2_end[s], f1 = C.ms2_loopn[s] * (1.0 / 24.0);
        const double s2 = C.pp7_start[s], e2 = C.pp7_end[s], f2 = C.pp7_loopn[s] * (1.0 / 24.0);
        if (algo == TC_ALGO_TOEPLITZ) {
            // lag thresholds of the piecewise response, by exact predicate on p = v*(d*lag):
            // ramp = [la, le), plateau = [lb, lL); lanes 0-3: MS2, lanes 4-7: PP7
            // (A straight-line version — all 32 lanes testing the four candidate lags around the guess of each threshold at once
            // — was measured: +0.8 % on the batched kernel, -3 % on both samplers, whose instruction footprint it enlarges.)
            int *thr = reinterpret_cast<int *>(tc_smem + w.thr);
            if (lane < 8) {
                const bool c2 = lane >= 4;
                const int q = lane & 3;
                const double x = q == 0 ? (c2 ? s2 : s1) : (q == 3 ? (c2 ? L2 : L1) : (c2 ? e2 : e1));
                thr[lane] = first_lag(v, cv.d, inv_vd, x, N, (q & 1) == 0);        // >s, >=e, >e, >=L
            }
            const double sc1 = C.sc1[s], sc2 = C.sc2[s];                 // f / (e - s), from the host
            __syncwarp();
            const int4 t1 = *reinterpret_cast<const int4 *>(thr), t2 = *reinterpret_cast<const int4 *>(thr + 4);
            const int la1 = t1.x, le1 = t1.y, lb1 = t1.z, lL1 = t1.w;
            const int la2 = t2.x, le2 = t2.y, lb2 = t2.z, lL2 = t2.w;
            SS_MARK(1);
            // Per time point j, both parts of the response in O(1) from the prefix sums K (counts) and S (first moments):
            //   ramp,    lags [la, min(le-1, j)]:  sc (v d sum lag n[j-lag] - s sum n[j-lag])   (cost independent of v: a chain
            //            that wanders to v -> 0, where the ramp spans every lag, is no slower than any other)
            //   plateau, lags [lb, min(lL-1, j)]:  whole polymerases -> exact count
            //   Branch-free: a part that is absent gets the index pair (0, 0), i.e. an empty prefix difference.
            //   One time point per lane per pass, for the instruction cache: two made ss_eval 18.6 KB of SASS instead of 13 KB,
            //   measured 2 % slower on config 2 and 1 % on config 3; four doubled the code for no gain.
#pragma unroll 1
            for (int j = lane; j < N; j += 32) {
                const double dj = (double)j;
                const int lh1 = min(le1 - 1, j), lh2 = min(le2 - 1, j);
                const bool r1ok = lh1 >= la1, r2ok = lh2 >= la2;
                const bool p1ok = j >= lb1 && lb1 < lL1, p2ok = j >= lb2 && lb2 < lL2;
                const int a1i = r1ok ? j - la1 + 1 : 0, b1i = r1ok ? j - lh1 : 0;
                const int a2i = r2ok ? j - la2 + 1 : 0, b2i = r2ok ? j - lh2 : 0;
                const int p1a = p1ok ? j - lb1 + 1 : 0, p1b = p1ok ? max(j - lL1 + 1, 0) : 0;
                const int p2a = p2ok ? j - lb2 + 1 : 0, p2b = p2ok ? max(j - lL2 + 1, 0) : 0;
                const int *ks = tc_smem_i();
                const double dK1 = (double)(ks[w.K + a1i] - ks[w.K + b1i]), dS1 = (double)(ks[w.S + a1i] - ks[w.S + b1i]);
                const double dK2 = (double)(ks[w.K + a2i] - ks[w.K + b2i]), dS2 = (double)(ks[w.S + a2i] - ks[w.S + b2i]);
                const double pl1 = (double)(ks[w.K + p1a] - ks[w.K + p1b]), pl2 = (double)(ks[w.K + p2a] - ks[w.K + p2b]);
                double c1 = fma(f1, pl1, sc1 * (vd * (dj * dK1 - dS1) - s1 * dK1));
                double c2 = fma(f2, pl2, sc2 * (vd * (dj * dK2 - dS2) - s2 * dK2));
                if (s > 0) { c1 += tc_smem[w.F1 + j]; c2 += tc_smem[w.F2 + j]; }
                tc_smem[w.F1 + j] = c1 < b1 ? b1 : c1;                          // :57
                tc_smem[w.F2 + j] = c2 < b2 ? b2 : c2;                          // :69
            }
        } else {
            SS_MARK(1);
            rows_pairs(cv, w, s, v, s1, e1, L1, f1, b1, s2, e2, L2, f2, b2);
        }
        __syncwarp();
        SS_MARK(2);
    }
    if (out1) {
#pragma unroll 1
        for (int j = lane; j < N; j += 32) { out1[j] = A * tc_smem[w.F1 + j]; out2[j] = tc_smem[w.F2 + j]; }
    }

    // (c) MS2 *= A, interp1 back to the experimental times, NaN-skipping residual sum of squares
    //     SumofSquares...m:51-64
    double acc = 0.0;
#pragma unroll 1
    for (int j = lane; j < N; j += 32) {
        const int k = cv.ik(j);                                                 // -1: outside the model grid (interp1 -> NaN)
        const int kk = k >= 0 ? k : 0;
        const double wj = cv.iw(j);
        const double m1 = A * tc_smem[w.F1 + kk], m1n = A * tc_smem[w.F1 + kk + 1];
        double r1 = cv.ms2(j) - (m1 + wj * (m1n - m1));
        const double f2k = tc_smem[w.F2 + kk];
        double r2 = cv.pp7(j) - (f2k + wj * (tc_smem[w.F2 + kk + 1] - f2k));
        r1 = (k >= 0 && r1 == r1) ? r1 : 0.0;                                   // nansum
        r2 = (k >= 0 && r2 == r2) ? r2 : 0.0;
        acc += fma(r2, r2, fma(r1, r1, 0.0));               // the point's two squares, then one add (folding acc into the fma rounds differently)
    }
    SS_MARK(3);
    acc = warp_sum(acc);
    SS_MARK(4);
    __syncwarp();
    return acc;
}

}  // namespace tc
