// tc_warp.cuh — dram_warp_kernel: the DRAM sampler with ONE WARP PER CHAIN (included by tc_mcmc.cu).
//
// dram_kernel gives a chain a whole CTA and buys latency with speculation: right when there are about as many chains as
// SMs (BASELINE config 2: 299 chains), wasteful when there are thousands (config 3: 19 136 chains; every GPU of an 8-GPU
// partition still holds 2 392) — a third of the speculative evaluations are thrown away and every round is three CTA-wide
// barriers.  Here every warp of the persistent grid owns a chain slice and runs mcmcrun's loop sequentially, step by step,
// with no CTA barrier anywhere: bounds + prior -> ssfun -> (delayed rejection: bounds + prior -> ssfun) -> accept/reject ->
// sigma2 draw, the warps of an SM covering each other's latencies (16 chains in flight per SM).  What a CTA did
// cooperatively becomes warp-local and streams through L2/HBM:
//   * proposal increments: every WK_GEN = 8 steps one pass over the chain's factor R on the FP64 tensor cores
//     ([8 steps x npar] x [npar x npar], mma.sync.m8n8k4.f64 = DMMA; A fragments from the normals in shared memory — stored as
//     the FP32 values they are —, B fragments straight from HBM/L2), results to an L2-resident scratch slot;
//   * adaptation: scatter update M2 += U'U (DMMA, 8 rows of the block at a time) and a left-looking blocked Cholesky through
//     L2 (8-row panels: DMMA accumulation over the rows above, the 8x8 diagonal block in registers, panel solve one column
//     per lane), all by the one warp.
// Same Philox addressing, same arithmetic per step as dram_kernel: the chain is the oracle's flag for flag (replay tests run
// both kernels).  Shared memory per warp: [slot 0 | slot 1 | cell | forward-model scratch]; the two slots hold the state x and
// the proposal under evaluation (an accept swaps them), cell + scratch double as the workspace of generation / adaptation
// (the cell is re-staged afterwards).
#pragma once

#define WK_WARPS 16         // one CTA per SM
#define WK_THREADS (32 * WK_WARPS)
#define WK_GEN 8           // steps per generation batch (one MMA row group)
#define WK_GENR 4          // ... in replay mode (the caller's normals are FP64: half the rows fit)

__host__ __device__ inline int wk_ldp(int N) { return (7 + N + 1) & ~1; }
// row stride of the normals Z (in elements) such that the A-fragment reads (lane -> row lane>>2, column 4 kk + (lane & 3)) are
// bank-conflict free: stride = 4 mod 8 elements
__host__ __device__ inline int wk_ldz(int N) { int n = (7 + N + 3) & ~3; while ((n & 7) != 4) n += 4; return n; }
__host__ __device__ inline int wk_ldu(int N) { return 8 * ((7 + N + 7) >> 3) + 4; }
__host__ __device__ inline int wk_cell_sz(int N) { return (cell_doubles(N) + 1) & ~1; }
__host__ __device__ inline int wk_overlay(int N)
{
    int need = wk_cell_sz(N) + ((work_doubles(N) + 3) & ~1);         // what the steps need: cell + forward-model scratch
    const int gen = 8 * wk_ldz(N);                                   // 2 stages x 8 rows of FP32 (= 2 x 4 rows of FP64 in replay)
    const int ad = 8 * wk_ldu(N) + 16;                               // 8 rows of the covariance block / the Cholesky panel
    if (need < gen) need = gen;
    if (need < ad) need = ad;
    return (need + 1) & ~1;
}
// the two theta slots start at ODD offsets (region + 1, region + 1 + ldp): element 7, the first dR, is 16-byte aligned (SmemVecA)
__host__ __device__ inline int wk_region(int N) { return 2 * wk_ldp(N) + 2 + wk_overlay(N); }

// per-warp mutable book-keeping in shared memory (lane 0 writes; everything hot lives in registers)
struct WkState {
    Tally t;
    long long tprev;
};
// per-warp chain context (written by lane 0 when a slice is claimed)
struct WkCtx {
    int N, npar, ld, ldp, ch, o_s0, o_ov, o_work;
    ChainConsts cc;
    const double *lo, *hi, *mu, *pinv;
    double *gInc, *gSc, *gWs;                                        // this warp slot's scratch
    double *gR, *gM2, *gRows, *gWts, *cmean, *mb, *wmean, *wM2, *rdiag;
    SmemCell cv;
    // bounds / prior in the reference's own structure (TranscriptionCycleMCMC.m:242-255): seven head parameters with their own
    // bounds, then one block (dR) with common bounds and prior.  uni = 1 when this chain's vectors have that structure: the
    // proposals are then checked against these few values instead of four vectors streamed from L2 every step.
    int uni;
    int nmax;                                                       // max N over the dataset: the layout of the warp's region
    double head[4][8];                                              // lo, hi, mu, 1/sig of parameters 0..7
    double blk[4];                                                  // ... of the block (parameters >= 7)
};
__shared__ WkCtx wk_cx[WK_WARPS];
__shared__ WkState wk_st[WK_WARPS];

__device__ __forceinline__ void wk_stage_cell(const CellsDev &cd, int cid, const SmemCell &cv)
{
    const int N = cv.N, lane = threadIdx.x & 31;
    const long long o = cd.off[cid], op = o + 4LL * cid;           // tgp / dtgp: the grid in its shared-memory order (cell_perm)
    int *ikp = reinterpret_cast<int *>(tc_smem + cv.o_ik);
#pragma unroll 5
    for (int i = lane; i < N; i += 32) {
        tc_smem[cv.o_tg + i] = cd.tgp[op + i];
        tc_smem[cv.o_dtg + i] = cd.dtgp[op + i];
        tc_smem[cv.o_ms2 + i] = cd.ms2[o + i];
        tc_smem[cv.o_pp7 + i] = cd.pp7[o + i];
        tc_smem[cv.o_iw + i] = cd.iw[o + i];
        ikp[i] = cd.ik[o + i];
    }
    if (lane < 3 && N + lane < ((N + 3) & ~3)) {                    // the permuted order spreads N entries over (N + 3) & ~3 places
        tc_smem[cv.o_tg + N + lane] = cd.tgp[op + N + lane];
        tc_smem[cv.o_dtg + N + lane] = cd.dtgp[op + N + lane];
    }
    __syncwarp();
}

// increments of the batch rows from the normals in shared memory: inc1 = z1 R, inc2 = z2 R / drscale -> gInc[row][j] (double2).
// ZT = float (production: the Box-Muller normals are FP32 values) or double (replay).  Column tiles of 8, k-steps of 4 rows of
// R in groups of 8 (8 B-fragment loads in flight), four interleaved accumulator sets — the summation order of dram_kernel's
// generate(), so the two kernels produce bit-identical increments.
// L2 residency: the proposal factors stream through once per batch (76 KB per chain, GBs per second in all) and must not
// evict the small per-warp scratch (increments / scalars of the current batch) that the step loop re-reads
__device__ __forceinline__ unsigned long long wk_policy_stream()
{
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long wk_policy_keep()
{
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ double wk_ld_stream(const double *p, unsigned long long pol)
{
    double v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void wk_st_keep(double2 *p, double2 v, unsigned long long pol)
{
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1,%2}, %3;" ::"l"(p), "d"(v.x), "d"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ double wk_ld_keep(const double *p, unsigned long long pol)
{
    double v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}

template <typename ZT>
__device__ __forceinline__ void wk_increments(const WkCtx &c, int nnew)
{
    const int lane = threadIdx.x & 31, npar = c.npar, ar = lane >> 2, ak = lane & 3;
    const int ldz = wk_ldz(c.nmax), rows = sizeof(ZT) == 4 ? WK_GEN : WK_GENR;
    const ZT *Z1 = reinterpret_cast<const ZT *>(tc_smem + c.o_ov), *Z2 = Z1 + rows * ldz;
    const int NT = (npar + 7) >> 3, nt4 = (npar + 3) >> 2, inner = 4 * ak + (ar & 3);
    const bool rowok = ar < nnew;
    const double inv_dr = c.cc.inv_dr;
    // rows >= nnew of Z hold stale data: their results are dropped; columns >= npar are zero (wk_generate)
    const ZT *za1p = Z1 + (ar < rows ? ar : 0) * ldz + ak, *za2p = Z2 + (ar < rows ? ar : 0) * ldz + ak;
    double2 *out = reinterpret_cast<double2 *>(c.gInc) + (size_t)ar * c.ldp;
    const unsigned long long pol_r = wk_policy_stream(), pol_k = wk_policy_keep();
    // The B fragments of one group (8 k-steps of one column tile) are loaded while the previous group is multiplied: the
    // loads of a warp never wait behind its own MMAs.  State of the group being loaded: column tile nt_n, first k-step
    // kk_n, pointer to this lane's element of tile (kk_n, bj_n) — tile (k+1, bj) sits 16 (nt4 - k - 1) doubles after (k, bj).
    int nt_n = NT - 1, kk_n = 0, ks_n, bj_n, dpl_n;
    const double *pl_n;
    double bvn[8];
#define WK_OPEN_TILE()                                                                                      \
    {                                                                                                       \
        ks_n = (min(8 * nt_n + 8, npar) + 3) >> 2;                                                          \
        bj_n = (8 * nt_n + ar < npar) ? 2 * nt_n + (ar >> 2) : -1;                                          \
        pl_n = c.gR + 16 * bj_n + inner; dpl_n = 16 * (nt4 - 1); kk_n = 0;                                  \
    }
#define WK_LOAD_GROUP()                                                                                     \
    {                                                                                                       \
        _Pragma("unroll") for (int u = 0; u < 8; ++u) {                                                     \
            /* (unconditional loads with a select were measured slower: the padded k-steps become real L2 transactions) */ \
            bvn[u] = (kk_n + u < ks_n && kk_n + u <= bj_n) ? wk_ld_stream(pl_n, pol_r) : 0.0;               \
            pl_n += dpl_n; dpl_n -= 16;                                                                     \
        }                                                                                                   \
        kk_n += 8;                                                                                          \
        if (kk_n >= ks_n) { --nt_n; if (nt_n >= 0) WK_OPEN_TILE() }                                         \
    }
    WK_OPEN_TILE()
    WK_LOAD_GROUP()
#pragma unroll 1
    for (int nt = NT - 1; nt >= 0; --nt) {
        const int ks = (min(8 * nt + 8, npar) + 3) >> 2;
        double acc[4][4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[q][e] = 0.0;
#pragma unroll 1
        for (int kk = 0; kk < ks; kk += 8) {
            double bv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) bv[u] = bvn[u];
            if (nt_n >= 0) WK_LOAD_GROUP()
            // k-steps past the last one of the tile multiply by B = 0; A is read unconditionally (finite: Z is padded)
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int kc = min(4 * (kk + u), ldz - 4);
                // FP32 Z widens exactly through F2F: integer-instruction widening measured no faster (28.2 k vs 27.0 k cycles per step)
                const double a1 = za1p[kc], a2 = za2p[kc];
                dmma_m8n8k4(acc[u & 3][0], acc[u & 3][1], a1, bv[u]);
                dmma_m8n8k4(acc[u & 3][2], acc[u & 3][3], a2, bv[u]);
            }
        }
        const double acc0 = (acc[0][0] + acc[1][0]) + (acc[2][0] + acc[3][0]), acc1 = (acc[0][1] + acc[1][1]) + (acc[2][1] + acc[3][1]);
        const double acc2 = (acc[0][2] + acc[1][2]) + (acc[2][2] + acc[3][2]), acc3 = (acc[0][3] + acc[1][3]) + (acc[2][3] + acc[3][3]);
        const int jc = 8 * nt + 2 * ak;
        if (rowok) {
            if (jc < npar) wk_st_keep(out + jc, make_double2(acc0, acc2 * inv_dr), pol_k);
            if (jc + 1 < npar) wk_st_keep(out + jc + 1, make_double2(acc1, acc3 * inv_dr), pol_k);
        }
    }
#undef WK_LOAD_GROUP
#undef WK_OPEN_TILE
}

__device__ __forceinline__ void wk_prefetch_l2(const double *p, int nlines)     // nlines x 128 B
{
    for (int i = threadIdx.x & 31; i < nlines; i += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + 16 * (size_t)i));
}

// Randomness and proposal increments of steps [g0, g0 + nnew) by one warp: scalars (u1, u2, chi2, the two q1 norms, log u1)
// -> gSc[row][0..5], increments -> gInc[row][j].  Overwrites the cell + scratch area (the caller re-stages the cell).
__device__ __noinline__ void wk_generate(const RunArgs &a, const WkCtx &c, int g0, int nnew, bool r_diag)
{
    const int lane = threadIdx.x & 31, npar = c.npar;
    const int ldz = wk_ldz(c.nmax);
    const bool rep = a.replay != 0;
    if (!r_diag) wk_prefetch_l2(c.gR, tri_doubles(npar) / 16);      // R: HBM -> L2 while the normals are drawn
    if (lane < nnew) {
        const int st = g0 + lane;
        double u1, u2, x2;
        if (rep) {
            const size_t g = (size_t)c.ch * a.nsimu + st;
            u1 = a.u1[g]; u2 = a.u2[g]; x2 = a.chi2[g];
        } else {
            const u32x4 ru = draw(a.seed, c.cc.uid, st, RK_U, 0);
            u1 = u01(ru.x, ru.y); u2 = u01(ru.z, ru.w);
            x2 = a.updatesigma ? chi2_draw_dc(a.seed, c.cc.uid, st, c.cc.chi_d, c.cc.chi_c) : 1.0;
        }
        double *sc = c.gSc + 8 * lane;
        __stcg(sc + 0, u1); __stcg(sc + 1, u2); __stcg(sc + 2, x2); __stcg(sc + 5, tc_log(u1));
    }
    __syncwarp();
    const double inv_dr = c.cc.inv_dr;
    if (rep) {
        double *Z1 = tc_smem + c.o_ov, *Z2 = Z1 + WK_GENR * ldz;
#pragma unroll 1
        for (int s = 0; s < nnew; ++s) {
            const size_t g = ((size_t)c.ch * a.nsimu + g0 + s) * c.ld;
            double n1 = 0.0, n0 = 0.0;
#pragma unroll 1
            for (int i = lane; i < npar; i += 32) {
                const double z1 = a.z1[g + i], z2 = a.z2[g + i];
                Z1[s * ldz + i] = z1; Z2[s * ldz + i] = z2;
                const double d = z1 - z2 * inv_dr;
                n1 = fma(d, d, n1); n0 = fma(z1, z1, n0);
            }
            if (lane < ldz - npar) { Z1[s * ldz + npar + lane] = 0.0; Z2[s * ldz + npar + lane] = 0.0; }     // padding columns (ldz - npar <= 11)
            warp_sum2(n1, n0);
            if (lane == 0) { __stcg(c.gSc + 8 * s + 3, n1); __stcg(c.gSc + 8 * s + 4, n0); }
        }
    } else {
        float *Z1 = reinterpret_cast<float *>(tc_smem + c.o_ov), *Z2 = Z1 + WK_GEN * ldz;
        const int npairs = (npar + 1) >> 1;
        // Two steps per pass: a lane draws the parameter pairs lane, lane + 32 of step s and of step s + 1 — four independent
        // Philox + Box-Muller chains in flight instead of two — and the norms of the two steps are reduced side by side.
        // (npairs <= 64 here: npar <= 128 + ...; the general case loops.)
#pragma unroll 1
        for (int s = 0; s < nnew; s += 2) {
            const bool two = s + 1 < nnew;
            double n1a = 0.0, n0a = 0.0, n1b = 0.0, n0b = 0.0;
#pragma unroll 1
            for (int q0 = 0; q0 < npairs; q0 += 64) {
                double4 z[4];
                bool on[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int q = q0 + lane + 32 * (u & 1), ss = s + (u >> 1);
                    on[u] = q < npairs && ss < nnew;
                    z[u] = normal_quad_inl(a.seed, c.cc.uid, g0 + ss, on[u] ? q : 0);   // (z1[2q], z1[2q+1], z2[2q], z2[2q+1]): FP32 values
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int q = q0 + lane + 32 * (u & 1), ss = s + (u >> 1);
                    if (on[u]) {
                        *reinterpret_cast<float2 *>(Z1 + ss * ldz + 2 * q) = make_float2((float)z[u].x, (float)z[u].y);
                        *reinterpret_cast<float2 *>(Z2 + ss * ldz + 2 * q) = make_float2((float)z[u].z, (float)z[u].w);
                        double &n1 = (u >> 1) ? n1b : n1a, &n0 = (u >> 1) ? n0b : n0a;      // (compile-time: the loop is unrolled)
                        const double d0 = z[u].x - z[u].z * inv_dr;
                        n1 = fma(d0, d0, n1); n0 = fma(z[u].x, z[u].x, n0);
                        if (2 * q + 1 < npar) { const double d1 = z[u].y - z[u].w * inv_dr; n1 = fma(d1, d1, n1); n0 = fma(z[u].y, z[u].y, n0); }
                    }
                }
            }
            __syncwarp();
            if (lane < ldz - npar) {                                                                        // padding columns (incl. the odd pair's spare)
                Z1[s * ldz + npar + lane] = 0.0f; Z2[s * ldz + npar + lane] = 0.0f;
                if (two) { Z1[(s + 1) * ldz + npar + lane] = 0.0f; Z2[(s + 1) * ldz + npar + lane] = 0.0f; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                n1a += __shfl_xor_sync(0xffffffffu, n1a, o); n0a += __shfl_xor_sync(0xffffffffu, n0a, o);
                n1b += __shfl_xor_sync(0xffffffffu, n1b, o); n0b += __shfl_xor_sync(0xffffffffu, n0b, o);
            }
            if (lane == 0) {
                __stcg(c.gSc + 8 * s + 3, n1a); __stcg(c.gSc + 8 * s + 4, n0a);
                if (two) { __stcg(c.gSc + 8 * (s + 1) + 3, n1b); __stcg(c.gSc + 8 * (s + 1) + 4, n0b); }
            }
        }
    }
    __syncwarp();
    if (lane == 0) { WkState &st = wk_st[threadIdx.x >> 5]; st.t.pc[PH_RAND] += clock64() - st.tprev; }    // sub-phase: randomness (tprev is not moved)
    if (r_diag) {
        double2 *out = reinterpret_cast<double2 *>(c.gInc);
        const unsigned long long pol_k = wk_policy_keep();
#pragma unroll 1
        for (int s = 0; s < nnew; ++s) {
#pragma unroll 1
            for (int j = lane; j < npar; j += 32) {
                const double r = __ldcg(c.rdiag + j);
                double z1, z2;
                if (rep) { z1 = tc_smem[c.o_ov + s * ldz + j]; z2 = tc_smem[c.o_ov + (WK_GENR + s) * ldz + j]; }
                else {
                    const float *Zf = reinterpret_cast<const float *>(tc_smem + c.o_ov);
                    z1 = (double)Zf[s * ldz + j]; z2 = (double)Zf[(WK_GEN + s) * ldz + j];
                }
                wk_st_keep(out + (size_t)s * c.ldp + j, make_double2(z1 * r, z2 * (r * inv_dr)), pol_k);
            }
        }
    } else if (rep) {
        wk_increments<double>(c, nnew);
    } else {
        wk_increments<float>(c, nnew);
    }
    __syncwarp();
}

// Bounds and prior of one proposal component (TranscriptionCycleMCMC.m:235-255): p += ((th - mu)/sig)^2, returns out-of-bounds.
// UNI: the structured form (head parameters + one block), it = iteration (j = lane + 32 it: only it = 0 can touch the head).
template <bool UNI>
__device__ __forceinline__ bool wk_check(const WkCtx &c, int it, int j, double th, double &p)
{
    double lo, hi, mu, pinv;
    if (UNI) {
        const bool head = it == 0 && j < 8;
        lo = head ? c.head[0][j & 7] : c.blk[0]; hi = head ? c.head[1][j & 7] : c.blk[1];
        mu = head ? c.head[2][j & 7] : c.blk[2]; pinv = head ? c.head[3][j & 7] : c.blk[3];
    } else {
        lo = __ldg(c.lo + j); hi = __ldg(c.hi + j); mu = __ldg(c.mu + j); pinv = __ldg(c.pinv + j);
    }
    const double e = (th - mu) * pinv;
    p = fma(e, e, p);
    return th < lo || th > hi;
}
#define WK_PIT 5           // parameter iterations per lane: npar <= 160 (tc_mcmc_run checks)
__device__ __forceinline__ double2 wk_ld_keep2(const double *p, unsigned long long pol)
{
    double2 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}
// stage 1: theta1 = x + inc1 -> slot ob, bounds + prior; the stage-2 increments of the row stay in registers (inc2)
template <bool UNI>
__device__ __forceinline__ bool wk_propose1(const WkCtx &c, int ox, int ob, int row, double &pr, double (&inc2)[WK_PIT])
{
    const int lane = threadIdx.x & 31, npar = c.npar;
    const double *inc = c.gInc + 2 * (size_t)row * c.ldp;
    const unsigned long long pol_k = wk_policy_keep();
    double2 d[WK_PIT];
#pragma unroll
    for (int it = 0; it < WK_PIT; ++it) {
        const int j = lane + 32 * it;
        d[it] = j < npar ? wk_ld_keep2(inc + 2 * j, pol_k) : make_double2(0.0, 0.0);
    }
    double p = 0.0;
    bool oob = false;
#pragma unroll
    for (int it = 0; it < WK_PIT; ++it) {
        const int j = lane + 32 * it;
        inc2[it] = d[it].y;
        if (j < npar) {
            const double th = tc_smem[ox + j] + d[it].x;
            oob |= wk_check<UNI>(c, it, j, th, p);
            tc_smem[ob + j] = th;
        }
    }
    pr = warp_sum(p);
    __syncwarp();
    return __any_sync(0xffffffffu, oob);
}
template <bool UNI>
__device__ __forceinline__ bool wk_propose2(const WkCtx &c, int ox, int ob, double &pr, const double (&inc2)[WK_PIT])
{
    const int lane = threadIdx.x & 31, npar = c.npar;
    double p = 0.0;
    bool oob = false;
#pragma unroll
    for (int it = 0; it < WK_PIT; ++it) {
        const int j = lane + 32 * it;
        if (j < npar) {
            const double th = tc_smem[ox + j] + inc2[it];
            oob |= wk_check<UNI>(c, it, j, th, p);
            tc_smem[ob + j] = th;
        }
    }
    pr = warp_sum(p);
    __syncwarp();
    return __any_sync(0xffffffffu, oob);
}

// The chain rows [r0, r1) all equal the state x (slot ox): Welford summaries with multiplicity (rows >= first_row), optional
// chain storage, and the distinct-row buffer of the current covariance block.  (flush_run of dram_kernel, warp-local, the
// summary vectors in L2.)
template <bool THIN>
__device__ __noinline__ void wk_flush(const RunArgs &a, const WkCtx &c, int ox, int r0, int r1, double wcnt, int ndist)
{
    const int lane = threadIdx.x & 31, npar = c.npar;
    const int m_c = r1 - r0, rs = max(r0, c.cc.first_row), m_w = run_rows(r0, r1, c.cc.first_row);
    const bool cov = run_distinct(a.do_cov, r0, r1);
    double f1, f2;
    welford_weights(wcnt, m_w, f1, f2);
    double *grow = cov ? c.gRows + (size_t)ndist * c.ld : nullptr;
    int j0 = rs - c.cc.first_row, nkr = m_w;
    if (THIN && a.store_chain && a.chain) nkr = kept_rows(rs, m_w, c.cc.first_row, a.thin, j0);
#pragma unroll 1
    for (int i = lane; i < npar; i += 32) {
        const double xo = tc_smem[ox + i];
        if (m_w > 0) {
            const double wm = __ldcg(c.wmean + i), d1 = xo - wm;
            __stcg(c.wmean + i, fma(d1, f1, wm));
            __stcg(c.wM2 + i, fma(d1 * d1, f2, __ldcg(c.wM2 + i)));
            if (a.store_chain && a.chain) {
                double *dst = a.chain + ((size_t)c.ch * c.cc.nkeep + j0) * c.ld + i;
#pragma unroll 1
                for (int r = 0; r < nkr; ++r) dst[(size_t)r * c.ld] = xo;
            }
        }
        if (cov) {
            __stcg(grow + i, xo);
            __stcg(c.mb + i, fma((double)m_c, xo, __ldcg(c.mb + i)));
        }
    }
    if (cov && lane == 0) __stcg(c.gWts + ndist, (double)m_c);
    __syncwarp();
}

// M2 += U'U for the covariance block (ndist distinct rows with weights + Chan's mean-shift row), 8 rows at a time: U staged in
// shared memory, one DMMA pair per 8x8 block of M2 (two blocks interleaved), read-modify-write of M2 in HBM/L2 (4x4-tile layout).
// mbar (the block mean) sits in shared memory at o_mb.
__device__ __noinline__ void wk_scatter(const WkCtx &c, int o_mb, int ndist, int nrows, double fcorr)
{
    const int lane = threadIdx.x & 31, npar = c.npar, ar = lane >> 2, ak = lane & 3;
    const int nt4 = (npar + 3) >> 2, NT = (npar + 7) >> 3, ldu = wk_ldu(c.nmax);
    const int oU = c.o_ov;
#pragma unroll 1
    for (int r0 = 0; r0 < nrows; r0 += 8) {
        const int rc = min(8, nrows - r0);
        double wr[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) wr[r] = r < rc ? (r0 + r < ndist ? __ldcg(c.gWts + r0 + r) : fcorr) : 0.0;
#pragma unroll
        for (int r = 0; r < 8; ++r) wr[r] = sqrt(wr[r]);
#pragma unroll 1
        for (int cc = lane; cc < 8 * NT; cc += 32) {
            const bool in = cc < npar;
            const double mbc = in ? tc_smem[o_mb + cc] : 0.0;
            double v[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) {                              // 8 rows in flight
                const int rr = r0 + r;
                v[r] = (in && r < rc) ? (rr < ndist ? __ldcg(c.gRows + (size_t)rr * c.ld + cc) : __ldcg(c.cmean + cc)) : mbc;
            }
#pragma unroll
            for (int r = 0; r < 8; ++r)                               // data rows: x - mean(block); the mean-shift row: mean(block) - cmean
                tc_smem[oU + r * ldu + cc] = wr[r] * (r0 + r < ndist ? v[r] - mbc : mbc - v[r]);
        }
        __syncwarp();
        // 8x8 blocks (bi <= bj) of M2, two per iteration; the old values of the NEXT pair are loaded before the MMAs of this one
        const int ua = oU + ak * ldu + ar;
        int bi = 0, bj = 0;
        double2 *g0 = nullptr, *g1 = nullptr;
        double2 o0 = make_double2(0.0, 0.0), o1 = o0;
#define WK_SC_PTRS(bi_, bj_, p0, p1, v0, v1)                                                                \
    {                                                                                                       \
        const int row__ = 8 * (bi_) + ar, tr__ = row__ >> 2, col0__ = 8 * (bj_) + 2 * ak, tc0__ = col0__ >> 2, tc1__ = tc0__ + 2; \
        p0 = ((bi_) < NT && tr__ <= tc0__ && tc0__ < nt4) ? reinterpret_cast<double2 *>(c.gM2 + 16 * (size_t)tidx(nt4, tr__, tc0__) + 4 * (row__ & 3) + (col0__ & 3)) : nullptr; \
        p1 = ((bi_) < NT && (bj_) + 1 < NT && tr__ <= tc1__ && tc1__ < nt4) ? reinterpret_cast<double2 *>(c.gM2 + 16 * (size_t)tidx(nt4, tr__, tc1__) + 4 * (row__ & 3) + (col0__ & 3)) : nullptr; \
        v0 = make_double2(0.0, 0.0); v1 = v0;                                                               \
        if (p0) v0 = __ldcg(p0);                                                                            \
        if (p1) v1 = __ldcg(p1);                                                                            \
    }
        WK_SC_PTRS(bi, bj, g0, g1, o0, o1)
#pragma unroll 1
        while (bi < NT) {
            int nbi = bi, nbj = bj + 2;
            if (nbj >= NT) { ++nbi; nbj = nbi; }
            double2 *n0, *n1;
            double2 on0, on1;
            WK_SC_PTRS(nbi, nbj, n0, n1, on0, on1)
            const int bj1 = bj + 1 < NT ? bj + 1 : bj;
            const double a0 = tc_smem[ua + 8 * bi], a1 = tc_smem[ua + 4 * ldu + 8 * bi];
            double d00 = 0.0, d01 = 0.0, d10 = 0.0, d11 = 0.0;
            dmma_m8n8k4(d00, d01, a0, tc_smem[ua + 8 * bj]);
            dmma_m8n8k4(d10, d11, a0, tc_smem[ua + 8 * bj1]);
            dmma_m8n8k4(d00, d01, a1, tc_smem[ua + 4 * ldu + 8 * bj]);
            dmma_m8n8k4(d10, d11, a1, tc_smem[ua + 4 * ldu + 8 * bj1]);
            if (g0) __stcg(g0, make_double2(o0.x + d00, o0.y + d01));
            if (g1) __stcg(g1, make_double2(o1.x + d10, o1.y + d11));
            bi = nbi; bj = nbj; g0 = n0; g1 = n1; o0 = on0; o1 = on1;
        }
#undef WK_SC_PTRS
        __syncwarp();
    }
}

// Upper Cholesky R'R = W of the tiled matrix in gW (HBM/L2, in place) by ONE warp: left-looking, panels of 8 rows.
// Per panel: S = W(panel, cols >= panel) - sum over the tile rows above of R(row, panel)' R(row, cols) on the FP64 tensor cores
// (four 8-column blocks share one A fragment), S -> shared memory; the 8x8 diagonal block is factored in registers by every
// lane (chol8), which leaves the factor where the panel solve needs it; one column per lane; the panel goes back to gW.
// Returns false when a pivot is not positive.
__device__ __noinline__ bool wk_chol(int nt4, int npar, const double *gA, double invn, double adj, double *gW, int oS)
{
    const int lane = threadIdx.x & 31, ar = lane >> 2, ak = lane & 3, th = ar >> 2, inner = 4 * ak + (ar & 3);
    const int ldS = 8 * ((nt4 + 1) >> 1) + 4;
    bool ok = true;
#pragma unroll 1
    for (int b0 = 0; b0 < nt4; b0 += 2) {
        const bool two = b0 + 1 < nt4;
        const int ntc = nt4 - b0, nb = (ntc + 1) >> 1;
        const int tr = b0 + th, rin = ar & 3;
#pragma unroll 1
        for (int j0 = 0; j0 < nb; j0 += 4) {
            double acc[4][2];
            bool bon[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; bon[m] = j0 + m < nb && b0 + 2 * (j0 + m) + th < nt4; }
            const bool aon = b0 + th < nt4;
            // the scatter-matrix entries of the panel: loaded before the accumulation so that their latency hides behind it
            double2 vin[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int j = j0 + m, tcn = b0 + 2 * j + (ak >> 1);
                vin[m] = make_double2(0.0, 0.0);
                if (j < nb && tr <= tcn && tcn < nt4 && tr < nt4)
                    vin[m] = __ldcg(reinterpret_cast<const double2 *>(gA + 16 * (size_t)tidx(nt4, tr, tcn) + 4 * rin + 2 * (ak & 1)));
            }
            const double *pa = gW + 16 * (b0 + th) + inner;          // tile (0, b0 + th); tile (r+1, c) is (nt4 - r - 1) tiles after (r, c)
            int dpa = 16 * (nt4 - 1);
#pragma unroll 4
            for (int r = 0; r < b0; ++r) {
                const double av = aon ? __ldcg(pa) : 0.0;
                double bv[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) bv[m] = bon[m] ? __ldcg(pa + 32 * (j0 + m)) : 0.0;
#pragma unroll
                for (int m = 0; m < 4; ++m) dmma_m8n8k4(acc[m][0], acc[m][1], av, bv[m]);
                pa += dpa; dpa -= 16;
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int j = j0 + m;
                if (j >= nb) continue;
                const int tcn = b0 + 2 * j + (ak >> 1), row = 4 * tr + rin, col = 4 * tcn + 2 * (ak & 1);
                // the tile test here, not through cov_entry's `in`: so the compiler shares it with the load loop's test above
                // (through `in`, config 3 measured 0.2 % slower on a B200 at 1000 W)
                double2 v = vin[m];
                if (tr <= tcn && tcn < nt4 && tr < nt4) v = cov_entry(true, v, row, col, npar, invn, adj);
                *reinterpret_cast<double2 *>(tc_smem + oS + ar * ldS + 8 * j + 2 * ak) = make_double2(v.x - acc[m][0], v.y - acc[m][1]);
            }
        }
        __syncwarp();
        double A[8][8], dinv[8];
        diag_block(tc_smem + oS, ldS, two, A);
        const bool bad = chol8(A, dinv);
        if (bad) { ok = false; break; }                                  // every lane computed the same
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int cc = r; cc < 8; ++cc) tc_smem[oS + r * ldS + cc] = A[r][cc];
        }
#pragma unroll 1
        for (int cc = 8 + lane; cc < 4 * ntc; cc += 32) {
            double xv[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) xv[r] = tc_smem[oS + r * ldS + cc];
            solve_col(A, dinv, xv);
#pragma unroll
            for (int r = 0; r < 8; ++r) tc_smem[oS + r * ldS + cc] = xv[r];
        }
        __syncwarp();
        store_panel<32, true>(tc_smem + oS, ldS, gW, nt4, b0, ntc, two, lane);
        __syncwarp();
    }
    __syncwarp();
    return ok;
}

// Adaptation after the step with isimu (a multiple of adaptint): adapt() of dram_kernel, warp-local, M2 and R in L2.
// Returns 0: R unchanged / scaled, 1: new full factor, 2: Cholesky failed.  o_mb: a free vector in shared memory (the idle slot).
__device__ __noinline__ int wk_adapt(const RunArgs &a, const WkCtx &c, int o_mb, int isimu, double cov_n, double rate, bool r_diag, int ndist)
{
    const int lane = threadIdx.x & 31, npar = c.npar;
    const int nt4 = (npar + 3) >> 2, T4 = tri_doubles(npar) / 16;
    if (a.do_cov) {
        const CovBlock blk = cov_block(isimu, cov_n, ndist);
        const int m = blk.m;
        wk_prefetch_l2(c.gM2, T4);                                  // the scatter matrix: HBM -> L2
#pragma unroll 1
        for (int i = lane; i < npar; i += 32) tc_smem[o_mb + i] = __ldcg(c.mb + i) / m;
        __syncwarp();
        wk_scatter(c, o_mb, ndist, blk.nrows, blk.fcorr);
#pragma unroll 1
        for (int i = lane; i < npar; i += 32) {
            const double cm = __ldcg(c.cmean + i), dm = tc_smem[o_mb + i] - cm;
            __stcg(c.cmean + i, cm + dm * blk.shift);
            __stcg(c.mb + i, 0.0);
        }
        cov_n += m;
        __syncwarp();
    }
    if (lane == 0) { WkState &st = wk_st[threadIdx.x >> 5]; st.t.pc[PH_SCATTER] += clock64() - st.tprev; }    // sub-phase: scatter update
    if (isimu < a.burnintime) {
        const double f = burnin_factor(rate, a.burnin_scale);
        if (f != 1.0) {
            if (r_diag) {
#pragma unroll 1
                for (int i = lane; i < npar; i += 32) __stcg(c.rdiag + i, __ldcg(c.rdiag + i) * f);
            } else {
#pragma unroll 1
                for (int i = lane; i < 16 * T4; i += 32) __stcg(c.gR + i, __ldcg(c.gR + i) * f);
            }
        }
        __syncwarp();
        return 0;
    }
    const double invn = 1.0 / (cov_n - 1.0);
    // mcmcstat: chol(cov) first, chol(cov + qcovadj I) only when that fails [U]; qcovadj_always = 1 adds it at once
    bool ok = wk_chol(nt4, npar, c.gM2, invn, a.qcovadj_always ? a.qcovadj : 0.0, c.gWs, c.o_ov);
    if (!ok && !a.qcovadj_always) ok = wk_chol(nt4, npar, c.gM2, invn, a.qcovadj, c.gWs, c.o_ov);
    if (lane == 0) { WkState &st = wk_st[threadIdx.x >> 5]; st.t.pc[PH_FACTOR] += clock64() - st.tprev; }    // sub-phase: scatter + factorisation
    if (ok) {
        const double2 *src = reinterpret_cast<const double2 *>(c.gWs);
        double2 *dst = reinterpret_cast<double2 *>(c.gR);
        const double sc = c.cc.adascale;
#pragma unroll 8
        for (int e = lane; e < 8 * T4; e += 32) { const double2 v = __ldcg(src + e); __stcg(dst + e, make_double2(v.x * sc, v.y * sc)); }
    }
    __syncwarp();
    return ok ? 1 : 2;
}

// Work items: (slice, group of WK_WARPS consecutive chains) in slice-major order from one global counter, one item per CTA; a
// slice of a chain waits for the previous slice of the same chain (claimed earlier, hence running or done: no deadlock).
// The warps of a CTA share nothing but the PHASE: every batch starts with a CTA barrier, so that all 16 warps of the SM are in
// generation, in the step loop or in adaptation at the same time — each phase's code fits the SM's instruction cache, the
// union does not (measured without the barriers: instruction-cache hit rate 61 %, 46 % of the stall cycles waiting for
// instructions).  Parked state between slices: scalars + counters + x in gState (the summary vectors live in L2 all along).
template <bool THIN>
__global__ void __launch_bounds__(WK_THREADS, 1) dram_warp_kernel(const __grid_constant__ RunArgs ga)
{
    __shared__ RunArgs a;
    __shared__ long long s_item;
    {
        const int *src = reinterpret_cast<const int *>(&ga);
        int *dst = reinterpret_cast<int *>(&a);
        for (int i = threadIdx.x; i < (int)(sizeof(RunArgs) / sizeof(int)); i += WK_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x * WK_WARPS + warp;
    const int nseg = (a.nsimu + a.seglen - 1) / a.seglen;
    const int ngroups = (a.nchains + WK_WARPS - 1) / WK_WARPS;
    const int regsz = wk_region(a.nmax), ldp = wk_ldp(a.nmax);     // as the host sized them (tc_mcmc_run)
    const int o_reg = warp * regsz;
    WkCtx &c = wk_cx[warp];
    WkState &st = wk_st[warp];
    const int genmax = a.replay ? WK_GENR : WK_GEN;
    const double n0s20 = a.N0 * a.S20;
    // Work items = (group of WK_WARPS consecutive chains, slice).  A free CTA claims the group that is furthest behind among
    // those nobody is running (a.cstate[g] = slices done, bit 30 = running): a group's slices are sequential, groups differ in
    // speed (series length, acceptance rate), and with about as many groups as CTAs — 2 392 chains of an 8-GPU partition are
    // 150 groups on 148 SMs — handing the items out in a fixed order makes the fast CTAs wait for the slices of the slow
    // ones (measured: 0.618 s against 0.518 s for 148 groups).
    const int LOCK = 1 << 30;
    int start = (int)(((long long)blockIdx.x * ngroups) / gridDim.x);
#pragma unroll 1
    for (;;) {
        __syncthreads();
        if (warp == 0) {
            long long got = -2;
#pragma unroll 1
            while (got == -2) {
                unsigned best = 0xffffffffu;
                int pending = 0;
#pragma unroll 1
                for (int i = lane; i < ngroups; i += 32) {
                    int gi = start + i; if (gi >= ngroups) gi -= ngroups;
                    const int v = *reinterpret_cast<volatile int *>(a.cstate + gi);
                    if (v & LOCK) pending = 1;
                    else if (v < nseg) best = min(best, ((unsigned)v << 20) | (unsigned)min(i, 0xfffff));
                }
                best = __reduce_min_sync(0xffffffffu, best);
                pending = __any_sync(0xffffffffu, pending);
                if (best == 0xffffffffu) {
                    if (!pending) { got = -1; break; }                  // every group is finished
                    __nanosleep(10000);
                    continue;
                }
                if (lane == 0) {
                    int gi = start + (int)(best & 0xfffffu); if (gi >= ngroups) gi -= ngroups;
                    const int v = (int)(best >> 20);
                    if (atomicCAS(a.cstate + gi, v, v | LOCK) == v) got = (long long)v * ngroups + gi;
                }
                got = __shfl_sync(0xffffffffu, got, 0);
            }
            if (lane == 0) s_item = got;
        }
        __syncthreads();
        const long long item = s_item;
        if (item < 0) break;
        const int seg = (int)(item / ngroups), grp = (int)(item - (long long)seg * ngroups), ch = grp * WK_WARPS + warp;
        start = grp + 1 < ngroups ? grp + 1 : 0;
        __threadfence();
        const bool valid = ch < a.nchains;
        const int k_end = min(a.nsimu, (seg + 1) * a.seglen);
        const bool last_seg = k_end >= a.nsimu;
        int cid = 0, N = 3, npar = 10;
        double *gst = nullptr;
        SmemCell cv{};
        Work w{};
        int ox = o_reg + 1, ob = o_reg + 1 + ldp;
        // is2 = 1 / sigma2 as the next step sees it, kept as the product chi2 * rden, rden = 1 / (N0 S20 + ss): the expression
        // dram_kernel uses at every position of a round, so the two kernels decide every step on the same bits
        double ss = 0.0, pri = 0.0, sig2 = a.sigma2_0, is2 = 1.0 / a.sigma2_0, rden = 0.0;
        int r_diag = 1, run_r0 = 0, ndist = 0;
        bool bad0 = false, uni = false;
        if (valid) {
            cid = a.chain_cell[ch];
            N = a.cells.N[cid]; npar = 7 + N;
            gst = a.gState + (size_t)ch * state_doubles(a.ld);
            if (lane == 0) {
                c.N = N; c.npar = npar; c.ld = a.ld; c.nmax = a.nmax; c.ldp = ldp; c.ch = ch;
                c.o_s0 = o_reg + 1; c.o_ov = o_reg + 2 * ldp + 2; c.o_work = c.o_ov + wk_cell_sz(a.nmax);
                c.cc = chain_consts(a, ch, N);
                c.lo = a.low + (size_t)ch * a.ld; c.hi = a.upp + (size_t)ch * a.ld; c.mu = a.pmu + (size_t)ch * a.ld;
                c.pinv = a.gPinv + (size_t)ch * a.ld;
                c.gInc = a.gInc + (size_t)slot * (2 * WK_GEN * ldp); c.gSc = a.gSc + (size_t)slot * (8 * WK_GEN);
                c.gWs = a.gW ? a.gW + (size_t)slot * a.ldR : nullptr;
                c.gR = a.gR + (size_t)ch * a.ldR;
                c.gM2 = a.gM2 ? a.gM2 + (size_t)ch * a.ldR : nullptr;
                c.gRows = a.gRows ? a.gRows + (size_t)ch * (size_t)a.blk_rows * a.ld : nullptr;
                c.gWts = a.gWts ? a.gWts + (size_t)ch * (size_t)a.blk_rows : nullptr;
                c.cmean = a.gCmean ? a.gCmean + (size_t)ch * a.ld : nullptr;
                c.mb = a.gMb ? a.gMb + (size_t)ch * a.ld : nullptr;
                c.wmean = gst + ST_VEC0 + a.ld; c.wM2 = gst + ST_VEC0 + 2 * a.ld; c.rdiag = gst + ST_VEC0 + 3 * a.ld;
                SmemCell cv0;
                carve_cell(c.o_ov, N, cv0);
                cv0.d = a.cells.dmean[cid];
                c.cv = cv0;
            }
            __syncwarp();
            cv = c.cv;
            carve_work(c.o_work, N, w);
            wk_stage_cell(a.cells, cid, cv);
            // ---- load or initialise the chain state
            if (seg == 0) {
#pragma unroll 1
                for (int i = lane; i < npar; i += 32) {
                    const size_t g = (size_t)ch * a.ld + i;
                    tc_smem[ox + i] = a.theta0[g];
                    a.gPinv[g] = prior_inv(a.psig[g]);
                    __stcg(c.rdiag + i, sqrt(a.qcov_diag[g]));
                    __stcg(c.wmean + i, 0.0); __stcg(c.wM2 + i, 0.0);
                    if (a.do_cov) { __stcg(c.cmean + i, 0.0); __stcg(c.mb + i, 0.0); }
                }
                if (a.do_cov) {
#pragma unroll 1
                    for (int i = lane; i < tri_doubles(npar); i += 32) __stcg(c.gM2 + i, 0.0);
                }
                if (lane == 0) {
                    st.t = Tally{};
                    st.t.n_ss = 1;                                      // ss(x0)
                }
                __syncwarp();
                // row 0: x0
                ss = ss_eval(a.cons, cv, SmemVecA{ox}, w, a.algo, false, nullptr, nullptr);
                double sp = 0.0;
#pragma unroll 1
                for (int i = lane; i < npar; i += 32) { const double e = (tc_smem[ox + i] - __ldg(c.mu + i)) * __ldcg(c.pinv + i); sp += e * e; }
                pri = warp_sum(sp);
                bad0 = !isfinite(ss);
                if (!bad0 && lane == 0) record_row0<THIN>(a, ch, ss, st.t);
            } else {
#pragma unroll 1
                for (int i = lane; i < npar; i += 32) tc_smem[ox + i] = __ldcg(gst + ST_VEC0 + i);
                const ParkedChain p = resume_chain(gst);
                ss = p.ss; pri = p.pri; sig2 = p.sigma2; is2 = p.rsig; r_diag = p.r_diag;
                bad0 = p.bad0 != 0;                                     // ss(x0) was not finite: reported at slice 0, nothing left to do
                run_r0 = seg * a.seglen;
                if (lane == 0) st.t = p.t;
            }
            // bounds / prior in the reference's structure?  (every slice: four vectors read once)
            {
                bool same = true;
                const double l7 = __ldg(c.lo + 7), h7 = __ldg(c.hi + 7), m7 = __ldg(c.mu + 7), p7 = __ldcg(c.pinv + 7);
#pragma unroll 1
                for (int i = 8 + lane; i < npar; i += 32)
                    same &= __ldg(c.lo + i) == l7 && __ldg(c.hi + i) == h7 && __ldg(c.mu + i) == m7 && __ldcg(c.pinv + i) == p7;
                same = __all_sync(0xffffffffu, same);
                if (lane < 8) {
                    c.head[0][lane] = __ldg(c.lo + lane); c.head[1][lane] = __ldg(c.hi + lane);
                    c.head[2][lane] = __ldg(c.mu + lane); c.head[3][lane] = __ldcg(c.pinv + lane);
                }
                if (lane == 0) { c.uni = same ? 1 : 0; c.blk[0] = l7; c.blk[1] = h7; c.blk[2] = m7; c.blk[3] = p7; }
            }
            if (lane == 0) st.tprev = clock64();
            __syncwarp();
            uni = c.uni != 0;
        }
        const bool active = valid && !bad0;
#ifdef WK_SUBPROF
#define WK_T0 const long long t0__ = clock64()
#define WK_T1(i) do { if (lane == 0) st.t.pc[i] += clock64() - t0__; } while (0)
#else
#define WK_T0
#define WK_T1(i)
#endif
#define WK_PHASE(i) do { if (lane == 0) { const long long tn__ = clock64(); st.t.pc[i] += tn__ - st.tprev; st.tprev = tn__; } } while (0)

        // the slice as slice_of() computes it, written out: through slice_of() this kernel spills more
        int k = seg == 0 ? 1 : seg * a.seglen;
        rden = tc_rcp(n0s20 + ss);                                  // (a function of ss alone: recomputed, not parked)
        int next_adapt = a.adaptint > 0 ? ((k + a.adaptint) / a.adaptint) * a.adaptint : 0x7fffffff;
#pragma unroll 1
        while (k < k_end) {                                             // the same trip count for every warp of the CTA
            const int g0 = k, gen_upto = min(k + genmax, min(k_end, next_adapt));
            // phase alignment: generation.  Every batch: aligning every 2nd / 4th measured 62.9 k / 72.7 k cycles per step
            // against 55.5 k (9 568 chains)
            __syncthreads();
            if (active) {
                WK_PHASE(PH_WAIT);
                wk_generate(a, c, g0, gen_upto - g0, r_diag != 0);
                wk_stage_cell(a.cells, cid, cv);
                WK_PHASE(PH_GEN);
            }
            __syncthreads();                                            // phase alignment: the step loop
            if (active) WK_PHASE(PH_WAIT);
#pragma unroll 1
            for (; k < gen_upto && active; ++k) {
                const int row = k - g0;
                const double *sc = c.gSc + 8 * row;
                // the step's scalars: one round trip to L2, overlapped with the proposal below
                const double s_u2 = __ldcg(sc + 1), s_chi = __ldcg(sc + 2), s_n1 = __ldcg(sc + 3), s_n0 = __ldcg(sc + 4), s_logu = __ldcg(sc + 5);
                // ---- stage 1
                int fl = 0, nev = 0, noob = 0, acc = 0;
                double pr1 = 0.0, ss1 = INFINITY, x12 = 0.0;
                double inc2[WK_PIT];
                const bool o1 = uni ? wk_propose1<true>(c, ox, ob, row, pr1, inc2) : wk_propose1<false>(c, ox, ob, row, pr1, inc2);
                if (o1) { fl |= TC_FL_OOB1; noob = 1; pr1 = 0.0; }
                else {
                    WK_T0;
                    ss1 = ss_eval(a.cons, cv, SmemVecA{ob}, w, a.algo, false, nullptr, nullptr);
                    WK_T1(PH_EVAL);
                    nev = 1;
                    if (stage1_accepts(ss1, ss, is2, pr1, pri, s_logu, x12)) acc = 1;
                }
                double ssn = ss1, prin = pr1;
                if (!acc && a.ntry >= 2) {
                    // ---- delayed rejection: one retry with R / drscale
                    fl |= TC_FL_DR;
                    double pr2 = 0.0;
                    const bool o2 = uni ? wk_propose2<true>(c, ox, ob, pr2, inc2) : wk_propose2<false>(c, ox, ob, pr2, inc2);
                    if (o2) { fl |= TC_FL_OOB2; ++noob; }
                    else {
                        WK_T0;
                        const double ss2 = ss_eval(a.cons, cv, SmemVecA{ob}, w, a.algo, false, nullptr, nullptr);
                        WK_T1(PH_EVAL);
                        ++nev;
                        if (resolve_dr(-0.5 * (s_n1 - s_n0), s_u2, o1, x12, pr1, pr2, ss1, ss2, ss, pri, is2)) { acc = 2; fl |= TC_FL_STAGE2; ssn = ss2; prin = pr2; }
                    }
                }
                // ---- commit
                if (acc) {
                    fl |= TC_FL_ACCEPT;
                    const double wcnt = st.t.wcnt;
                    wk_flush<THIN>(a, c, ox, run_r0, k, wcnt, ndist);          // close the run of the old state at row k
                    if (lane == 0) st.t.wcnt = wcnt + run_rows(run_r0, k, c.cc.first_row);
                    if (run_distinct(a.do_cov, run_r0, k)) ++ndist;
                    run_r0 = k;
                    const int t_ = ox; ox = ob; ob = t_;                 // the proposal becomes the state
                    ss = ssn; pri = prin;
                    rden = rden_of(n0s20, ss);
                }
                const double s2 = row_sigma2(a.updatesigma, n0s20, ss, s_chi, sig2);
                if (lane == 0) {
                    tally_s2(st.t, 1.0, s2, sqrt(s2), 0.0);                 // Welford: a batch of one row
                    st.t.n_ss += nev; st.t.n_oob += noob; if (fl & TC_FL_DR) ++st.t.n_dr;
                    if (acc == 1) ++st.t.n_acc1; else if (acc == 2) ++st.t.n_acc2; else { ++st.t.rej; ++st.t.reju; }
                    store_row<THIN>(a, ch, k, s2, fl, ss);
                }
                if (a.updatesigma) { sig2 = s2; is2 = s_chi * rden; }
                __syncwarp();
            }
            k = gen_upto;
            if (active) WK_PHASE(PH_STEPS);
            if (k == next_adapt) {
                __syncthreads();                                        // phase alignment: adaptation
                if (active) {
                    WK_PHASE(PH_WAIT);
                    const double wc0 = st.t.wcnt, cov_n = st.t.cov_n;
                    wk_flush<THIN>(a, c, ox, run_r0, k, wc0, ndist);           // close the run at the block boundary
                    const int nd = ndist + (run_distinct(a.do_cov, run_r0, k) ? 1 : 0);
                    const double rate = adapt_rate(a, st.t.rej, st.t.reju, k);
                    __syncwarp();
                    const int rc = wk_adapt(a, c, ob, k, cov_n, rate, r_diag != 0, nd);
                    if (lane == 0) {
                        st.t.wcnt = wc0 + run_rows(run_r0, k, c.cc.first_row);
                        after_adapt(st.t, a.do_cov, k, rc);
                    }
                    if (rc == 1) r_diag = 0;
                    run_r0 = k; ndist = 0;
                    __syncwarp();
                    wk_stage_cell(a.cells, cid, cv);
                    WK_PHASE(PH_ADAPT);
                }
                next_adapt += a.adaptint;
            }
        }
        if (valid) {
        __syncwarp();
        if (!bad0 && run_r0 < k) {
            const double wc0 = st.t.wcnt;
            wk_flush<THIN>(a, c, ox, run_r0, k, wc0, ndist);
            if (lane == 0) st.t.wcnt = wc0 + run_rows(run_r0, k, c.cc.first_row);
            run_r0 = k;
            __syncwarp();
        }
        if (bad0 && seg > 0) {
            // reported when slice 0 found ss(x0) not finite
        } else if (!last_seg && !bad0) {
            // ---- park
#pragma unroll 1
            for (int i = lane; i < npar; i += 32) __stcg(gst + ST_VEC0 + i, tc_smem[ox + i]);
            if (lane == 0) park_chain(gst, ParkedChain{ss, pri, sig2, is2, r_diag, 0, st.t});
            __syncwarp();
        } else {
            // ---- summaries
            if (bad0 && lane == 0) reinterpret_cast<ParkedChain *>(gst)->bad0 = 1;
#ifdef WK_SUBPROF
            const long long slot7 = st.t.pc[PH_EVAL];
#else
            const long long slot7 = st.t.n_ss;                          // no speculation: every evaluation is committed
#endif
            write_outputs(a, ch, npar, c.wmean, c.wM2, st.t, slot7, bad0, lane, 32);
        }
        }
        // ---- release the group: its next slice may run on any CTA
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) atomicExch(a.cstate + grp, seg + 1);
    }
#undef WK_PHASE
}
