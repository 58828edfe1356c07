// Host-side check of the shared-memory layouts the kernels rely on and of tc_mcmc_run's launch plan (compiled and run by
// tests/test_layout_invariants.py; needs nvcc, no GPU).  It includes the product's translation unit, so the formulas and
// plan functions checked are the ones the library uses.
#include <cstdio>
#include <cstring>
#include <set>
#include "../../transcriptioncycleinference_b200/csrc/tc_mcmc.cu"

static int fails = 0;
#define CHECK(cond, ...) do { if (!(cond)) { if (++fails < 20) { std::printf("FAIL: " __VA_ARGS__); std::printf("\n"); } } } while (0)

int main()
{
    const size_t optin = 232448;                      // 227 KB: B200's opt-in shared memory per block
    for (int N = 3; N <= 460; ++N) {
        // (1) the permuted model grid: a bijection of [0, N) into [0, (N + 3) & ~3), and the four loads of lane l in the block
        //     starting at r0 (steps r0 + 4 l + e) sit at r0 + e q + l
        const int N4 = (N + 3) & ~3;
        std::set<int> seen;
        for (int i = 0; i < N; ++i) {
            const int p = cell_perm(N, i);
            CHECK(p >= 0 && p < N4, "cell_perm(%d, %d) = %d outside [0, %d)", N, i, p, N4);
            CHECK(seen.insert(p).second, "cell_perm(%d, %d) = %d twice", N, i, p);
            const int r0 = i & ~127, rem = N - r0, q = ((rem < 128 ? rem : 128) + 3) >> 2, lane = (i & 127) >> 2, e = i & 3;
            CHECK(p == r0 + e * q + lane, "cell_perm(%d, %d) != block + e q + lane", N, i);
        }
        // (2) the forward-model scratch: thr (4) + alignment (1) + K, S as 32-bit integers with 3 leading pad ints and room for
        //     the 16-byte store of the last lane (index n + 3 = N + 2) + n, F1, F2 of N + 2 doubles
        const int ks = work_ks_doubles(N);
        CHECK(ks % 2 == 0 && 2 * ks >= 3 + (N + 3), "K/S area of %d doubles too small for N = %d", ks, N);
        CHECK(tc::work_doubles(N) >= 4 + 1 + 2 * ks + 3 * (N + 2), "work_doubles(%d)", N);
        CHECK(tc::cell_doubles(N) >= 2 * N4 + 3 * (N + 1) + (N + 2) / 2 + 1, "cell_doubles(%d)", N);
        // (3) a ring slot: two increment vectors of s1 >= npar doubles at odd offsets + 8 scalars, even size; Z (2 npar doubles
        //     from the slot base, big layout) must not reach the scalars
        const int s1 = dram_s1(N), slot = dram_slot(N), npar = 7 + N;
        CHECK(s1 % 2 == 0 && s1 >= npar && slot % 2 == 0 && slot == 2 * s1 + 10, "slot of N = %d", N);
        CHECK(2 * npar <= slot - 8, "Z overlaps the scalars at N = %d", N);
        // (4) budgets: what the kernel carves (cell, <= 3 alignment doubles, vectors, ring, per-warp areas) fits what the host asks for
        for (int big = 0; big < 2; ++big) {
            const int wsz = dram_wsz(N, big);
            CHECK(wsz % 2 == 0 && wsz >= ((tc::work_doubles(N) + 1) & ~1), "wsz(%d, %d)", N, big);
            const long long carved = tc::cell_doubles(N) + 3 + (long long)(big ? 7 : 10) * npar + (long long)(big ? RING / 2 : RING) * slot + (long long)SPEC * wsz;
            CHECK(carved <= dram_smem_doubles(N, big), "carve of N = %d (big %d) exceeds its budget", N, big);
            if (!big) CHECK((long long)(big ? RING / 2 : RING) * slot + (long long)SPEC * wsz >= chol_ws_doubles(npar) || sizeof(double) * (size_t)dram_smem_doubles(N, 0) > optin,
                            "Cholesky workspace does not fit ring + per-warp areas at N = %d", N);
        }
        // (5) chain-per-warp region: two slots of ldp >= npar at odd offsets, then the overlay (cell + scratch | normals | panel)
        CHECK(wk_ldp(N) % 2 == 0 && wk_ldp(N) >= npar && wk_region(N) % 2 == 0, "warp region of N = %d", N);
        CHECK(wk_overlay(N) >= wk_cell_sz(N) + ((tc::work_doubles(N) + 3) & ~1), "warp overlay of N = %d", N);
    }
    // tc_mcmc_run's launch plan on a B200: S = 148 SMs, static shared memory of dram_kernel / dram_warp_kernel taken as
    // 2.5 KB / 13 KB (ptxas: 2 544 / 13 008 bytes)
    const int S = 148, static_cta = 2560, static_warp = 13312;
    const auto plan = [&](int N, int nc, int layout) { return plan_layout(N, nc, layout, S, optin, static_cta, static_warp); };
    int max_reg = 0, max_two = 0, max_big = 0, max_warp = 0, max_stream = 0;
    for (int N = 3; N <= 460; ++N) {
        const LaunchPlan cta = plan(N, 1, TC_LAYOUT_CTA), big = plan(N, 1, TC_LAYOUT_BIG), warp = plan(N, 1, TC_LAYOUT_WARP);
        if (cta.err.empty() && !cta.big) max_reg = N;
        // two CTAs per SM: dynamic + static shared memory + 1 KB reserved each, out of optin + 1 KB
        if (cta.err.empty() && !cta.big && 2 * (cta.smem + static_cta + 1024) <= optin + 1024) max_two = N;
        if (big.err.empty() && big.big) max_big = N;
        if (warp.err.empty() && warp.warp) max_warp = N;
        CHECK(cta.err.empty() == (N <= 441) && cta.big == (N > 213) && !cta.warp, "TC_LAYOUT_CTA plan at N = %d", N);
        CHECK(big.err.empty() || big.err.find("too large for the shared-memory layout") != std::string::npos, "big layout refusal at N = %d", N);
        CHECK(warp.err.empty() || warp.err.find("too large for the chain-per-warp layout") != std::string::npos, "chain-per-warp refusal at N = %d", N);
        SsArgs a{};
        a.wsz = (tc::work_doubles(N) + 3) & ~1;               // launch_ss's forward-model scratch
        if (ss_stream_smem(a, N, 7 + N, optin)) max_stream = N;
    }
    std::printf("max N: regular %d (two CTAs per SM %d), big %d, chain-per-warp %d, ss_stream_kernel %d\n", max_reg, max_two,
                max_big, max_warp, max_stream);
    CHECK(max_reg == 213 && max_two == 141 && max_warp == 144 && max_stream == 152, "series-length limits");
    CHECK(max_big == 441, "big layout limit %d (include/tcmcmc.h says 441)", max_big);

    // schedules at the chain counts of tests/test_gpu_chain_counts.py: nsimu = 1000, adaptint = 100, per-SM occupancy of a
    // B200 (two CTAs of the regular layout at N = 129, one of the big layout or of dram_warp_kernel)
    struct Sched { int layout, N, nc; const char *kernel; int grid, seglen, solo_lag; };
    const Sched sched[] = {
        {TC_LAYOUT_CTA, 129, S, "cta", S, 100, 0},             {TC_LAYOUT_CTA, 129, S + 1, "cta", S + 1, 400, 2},
        {TC_LAYOUT_CTA, 129, 2 * S, "cta", 2 * S, 400, 2},     {TC_LAYOUT_CTA, 129, 2 * S + 1, "cta", 2 * S, 400, 2},
        {TC_LAYOUT_CTA, 129, 299, "cta", 2 * S, 400, 2},       {TC_LAYOUT_CTA, 129, 1183, "cta", 2 * S, 400, 2},
        {TC_LAYOUT_CTA, 129, 1184, "cta", 2 * S, 1000, 0},
        {TC_LAYOUT_BIG, 257, S, "big", S, 100, 0},             {TC_LAYOUT_BIG, 257, S + 1, "big", S, 100, 0},
        {TC_LAYOUT_BIG, 257, 2 * S, "big", S, 100, 0},         {TC_LAYOUT_BIG, 257, 2 * S + 1, "big", S, 100, 0},
        {TC_LAYOUT_BIG, 257, 299, "big", S, 100, 0},           {TC_LAYOUT_BIG, 257, 1183, "big", S, 100, 0},
        {TC_LAYOUT_BIG, 257, 1184, "big", S, 1000, 0},
        {TC_LAYOUT_WARP, 129, 16 * S - 1, "warp", S, 100, 0},  {TC_LAYOUT_WARP, 129, 16 * S, "warp", S, 100, 0},
        {TC_LAYOUT_WARP, 129, 16 * S + 1, "warp", S, 100, 0},  {TC_LAYOUT_WARP, 129, 19136, "warp", S, 100, 0},
        {TC_LAYOUT_AUTO, 129, 13 * S - 1, "cta", 2 * S, 1000, 0}, {TC_LAYOUT_AUTO, 129, 13 * S, "warp", 121, 100, 0},
    };
    for (const Sched &e : sched) {
        LaunchPlan p = plan(e.N, e.nc, e.layout);
        plan_schedule(p, e.nc, 1000, 100, S, p.warp || p.big ? 1 : 2, TC_SOLO_LAG, TC_SOLO_NSEG);
        const char *kernel = p.warp ? "warp" : (p.big ? "big" : "cta");
        CHECK(p.err.empty() && !std::strcmp(kernel, e.kernel) && p.grid == e.grid && p.seglen == e.seglen && p.solo_lag == e.solo_lag,
              "layout %d, N = %d, nc = %d: %s grid %d seglen %d solo_lag %d", e.layout, e.N, e.nc, kernel, p.grid, p.seglen, p.solo_lag);
        CHECK(!p.warp || p.nslots == (size_t)p.grid * WK_WARPS, "warp slots at nc = %d", e.nc);
    }
    std::printf("schedules: %d chain counts\n", (int)(sizeof(sched) / sizeof(sched[0])));

    // partitions of 1, D-1, D, D+1 and 19 136 chains over D = 1 ... 8 devices: contiguous blocks covering the chains, one
    // per device (per chain when there are fewer chains), none empty; of equal chains, blocks within one chain of nc / D.
    // Chains on cells of cycling lengths, one chain of N = 441 before chains of N = 3, or all of N = 129.
    const std::vector<int> Ncell = {200, 12, 441, 129, 3};
    for (int D = 1; D <= 8; ++D)
        for (int nc : {1, D - 1, D, D + 1, 19136})
            for (int mix = 0; nc >= 1 && mix < 3; ++mix) {
                std::vector<int32_t> cc(nc);
                for (int i = 0; i < nc; ++i) cc[i] = mix == 0 ? i % 5 : (mix == 1 ? (i == 0 ? 2 : 4) : 3);
                const std::vector<int> b = partition_chains(Ncell, cc.data(), nc, D);
                CHECK(b.size() == (size_t)std::min(D, nc) + 1 && b.front() == 0 && b.back() == nc, "partition of %d over %d", nc, D);
                for (size_t g = 0; g + 1 < b.size(); ++g) {
                    CHECK(b[g] < b[g + 1], "empty device %d: %d chains over %d (mix %d)", (int)g, nc, D, mix);
                    CHECK(mix != 2 || std::abs((b[g + 1] - b[g]) * D - nc) <= D, "unequal blocks: %d chains over %d", nc, D);
                }
            }
    std::printf("partitions: ok\n");
    std::printf(fails ? "layout check: %d failure(s)\n" : "layout check ok\n", fails);
    return fails ? 1 : 0;
}
