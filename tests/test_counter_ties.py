"""Ties in the loading counter, on the host: cases where the order of summation decides a floor.

The forward model loads floor(counter) polymerases, the counter being the SEQUENTIAL FP64 sum of rate x dt per step
(ConstantElongationSim.m:53-61).  scan_counts (csrc/tc_device.cuh) sums the steps in a warp-scan order instead — four
consecutive steps per lane, a Hillis-Steele scan of the 32 lane totals, a carry from one block of 128 steps to the next —
and redoes the sum sequentially when any partial sum lands within 1e-7 of an integer (`risky`), because there a different
association can move a floor.  Random data reach that branch only by chance; an exactly regular time grid (microscopes
produce them) with a rate that is a simple fraction of 1 / dt reaches it at every step.  This module builds such cases,
proves with a NumPy emulation of the fast path that each one needs the redo (its floors differ from the sequential ones and
the risky flag is set), and checks that the two oracles agree on the sequential floors, which are the specification.
Controls sit 1e-6 off the integers: outside the redo window, where both orders must give the same floors.
tests/test_gpu_lengths.py runs the same cases through the kernels."""
import functools

import numpy as np

from oracle import forward_literal as fl

DTS = (0.1, 1.0 / 3.0, 0.3, 0.7)           # regular frame intervals (min)
NS = (40, 129, 200, 400)                   # 129, 200 and 400 cross the carry between blocks of 128 steps
PER = 3                                    # adversarial cases per (N, dt)
RISK = 1e-7                                # scan_counts' redo window
# A construct whose curves ARE the loading counts: every polymerase past 1e-6 kb is on the plateau (1 per polymerase), none
# reaches L.  With the basal levels at 0 and A = 1, MS2 = PP7 = floor(counter after step j - 1) at time point j >= 1.
COUNT_CONS = dict(L_MS2=1e6, L_PP7=1e6, MS2_start=[0.0], MS2_end=[1e-6], MS2_loopn=[24.0],
                  PP7_start=[0.0], PP7_end=[1e-6], PP7_loopn=[24.0])


def regular_grid(N, dt):
    """t = k dt and its model grid t(1):mean(diff(t)):t(end), or None when that grid does not have N points (the
    reference rejects such a cell, and so does tc_cells_create)."""
    t = np.arange(N) * dt
    tg = fl.t_interp_of(t)
    return (t, tg) if tg.size == N else None


def increments(theta, tg):
    """rate x dt of every step, as the reference forms it: R + dR clamped at 0, times diff(t_interp); 0 before onset."""
    r = theta[6] + theta[7:6 + tg.size]
    r = np.where(r < 0.0, 0.0, r)
    return np.where(tg[:-1] < theta[2], 0.0, r * np.diff(tg))


def sequential_floors(p):
    return np.floor(np.add.accumulate(p))


def fast_path_floors(p):
    """NumPy emulation of scan_counts' fast path.  Per block of 128 steps, lane l sums its steps 4l..4l+3 in order, a
    Hillis-Steele inclusive scan combines the 32 lane totals, step i's counter is (carry + exclusive lane prefix) + local
    prefix, and the block total is added to the carry.  -> (floors, risky flag)"""
    n = p.size
    nb = -(-n // 128)
    q = np.zeros(nb * 128)
    q[:n] = p
    loc = np.add.accumulate(q.reshape(nb, 32, 4), axis=2)     # local inclusive prefix, the reference's own order
    t = loc[:, :, 3].copy()
    o = 1
    while o < 32:                                             # lane l adds lane l - o's value of the previous round
        t[:, o:] = t[:, o:] + t[:, :-o]
        o *= 2
    excl = np.concatenate([np.zeros((nb, 1)), t[:, :-1]], axis=1)
    c = np.empty_like(loc)
    carry = 0.0
    for b in range(nb):
        c[b] = (carry + excl[b])[:, None] + loc[b]
        carry = carry + t[b, 31]
    c = c.reshape(-1)[:n]
    f = np.floor(c)
    fr = c - f
    risky = bool(np.any((c != 0.0) & ((fr < RISK) | (fr > 1.0 - RISK))))
    return f, risky


def _theta(rng, N, tg, R, dR, ton):
    th = np.zeros(7 + N)
    th[:6] = [rng.uniform(0.5, 3.0), rng.uniform(0.0, 4.0), ton, rng.uniform(0.0, 3.0), rng.uniform(0.0, 3.0),
              rng.uniform(0.2, 1.0)]
    th[6] = R
    th[7:] = dR
    return th


@functools.lru_cache(maxsize=None)
def adversarial_cases():
    """PER cases per (N, dt): rate k / (m dt), dR = 0 or a constant, onset at 0 or exactly at a grid point.  Candidates are
    drawn (seed 0) from that family and kept when the fast path's floors differ from the sequential ones, so every case
    needs the redo.  -> list of dict(N, dt, t, tg, theta)"""
    rng = np.random.default_rng(0)
    out = []
    for N in NS:
        for dt in DTS:
            g = regular_grid(N, dt)
            assert g is not None, (N, dt)
            t, tg = g
            kept = 0
            for _ in range(400):
                m = int(rng.choice([1, 2, 3, 5, 10]))
                rate = float(rng.integers(1, 30)) / (m * dt)
                if rate > 70.0:                      # R + dR inside the sampler's bounds (R <= 40, dR <= 30)
                    continue
                c = float(rng.integers(-6, 7)) * 0.5 if rng.random() < 0.5 else 0.0
                ton = float(tg[int(rng.integers(1, N // 3))]) if rng.random() < 0.5 else 0.0
                th = _theta(rng, N, tg, rate - c, c, ton)
                p = increments(th, tg)
                if np.array_equal(fast_path_floors(p)[0], sequential_floors(p)):
                    continue
                out.append(dict(N=N, dt=dt, t=t, tg=tg, theta=th))
                kept += 1
                if kept == PER:
                    break
            assert kept == PER, (N, dt, kept)
    return tuple(out)


@functools.lru_cache(maxsize=None)
def control_cases():
    """One per (N, dt): the same rates with the first step's load raised by 1e-6, so that the partial sums land about 1e-6
    above the integers: close, but outside the redo window."""
    rng = np.random.default_rng(1)
    out = []
    for N in NS:
        for dt in DTS:
            t, tg = regular_grid(N, dt)
            m = int(rng.choice([1, 2, 5]))
            rate = float(rng.integers(1, 12)) / (m * dt)
            dR = np.zeros(N)
            dR[0] = 1e-6 / (tg[1] - tg[0])
            out.append(dict(N=N, dt=dt, t=t, tg=tg, theta=_theta(rng, N, tg, rate, dR, 0.0)))
    return tuple(out)


def count_theta(theta):
    """theta with the basal levels at 0 and A = 1: under COUNT_CONS the curves are then the loading counts."""
    th = np.array(theta, dtype=np.float64)
    th[3] = th[4] = 0.0
    th[5] = 1.0
    return th


def oracle_floors(co, case):
    """floor(counter) after steps 0..N-2 from both oracles (C, NumPy), read off the COUNT_CONS curves at time points 1..N-1."""
    th = count_theta(case["theta"])
    c_ms2, c_pp7 = co.model_on_grid(co.Construct.from_dict(COUNT_CONS), th, case["tg"])
    n_ms2, n_pp7 = fl.model_on_grid(COUNT_CONS, th, case["tg"])
    assert np.array_equal(c_ms2, c_pp7) and np.array_equal(n_ms2, n_pp7)
    return c_pp7[1:], n_pp7[1:]


def test_grids_match_the_c_oracle(orc):
    co, _ = orc
    for case in adversarial_cases() + control_cases():
        assert np.array_equal(co.t_interp(case["t"]), case["tg"])


def test_adversarial_cases_need_the_redo(orc):
    """Every case: the emulated fast path gives floors that differ from both oracles' sequential floors, and sets the risky
    flag, so the kernel's answer rests on the sequential redo.  The oracles agree with each other, and with a plain
    sequential sum of increments() (which is what the emulation is fed)."""
    co, _ = orc
    cases = adversarial_cases()
    assert {(c["N"], c["dt"]) for c in cases} == {(N, dt) for N in NS for dt in DTS}
    ndiff, past_first_block = [], 0
    for case in cases:
        p = increments(case["theta"], case["tg"])
        fc, fn = oracle_floors(co, case)
        assert np.array_equal(fc, fn), (case["N"], case["dt"])
        assert np.array_equal(fc, sequential_floors(p)), (case["N"], case["dt"])
        fast, risky = fast_path_floors(p)
        assert not np.array_equal(fast, fc), (case["N"], case["dt"])
        assert risky, (case["N"], case["dt"])
        ndiff.append(int(np.sum(fast != fc)))
        past_first_block += bool(np.any(fast[128:] != fc[128:]))        # differences that ride on the carry
    assert past_first_block >= 10, past_first_block
    print("%d adversarial cases, floors differing per case: min %d, median %d, max %d; %d differ past step 128"
          % (len(cases), min(ndiff), int(np.median(ndiff)), max(ndiff), past_first_block))


def test_controls_outside_the_redo_window(orc):
    """About 1e-6 off the integers both orders give the same floors and the fast path does not ask for the redo."""
    co, _ = orc
    for case in control_cases():
        p = increments(case["theta"], case["tg"])
        c = np.add.accumulate(p)
        fr = c - np.floor(c)
        assert 1e-7 < fr.min() < 2e-6, (case["N"], case["dt"], fr.min())          # near ties, but outside the window
        fc, fn = oracle_floors(co, case)
        assert np.array_equal(fc, fn) and np.array_equal(fc, sequential_floors(p))
        fast, risky = fast_path_floors(p)
        assert np.array_equal(fast, fc) and not risky, (case["N"], case["dt"])


def test_emulation_reproduces_random_sums():
    """The emulation itself: on random increments (no ties) it gives the sequential floors, and on a sum built to differ
    in association it differs (so a test above cannot pass through an emulation that silently sums sequentially)."""
    rng = np.random.default_rng(2)
    for n in (39, 128, 129, 399):
        p = rng.uniform(0.0, 3.0, n)
        f, risky = fast_path_floors(p)
        assert np.array_equal(f, sequential_floors(p)) or risky
    p = np.zeros(129)
    p[0], p[4:8] = 1.0 - 2.0 ** -53, 4e-17      # each 4e-17 alone rounds away; lane 1's total 1.6e-16 reaches 1
    assert np.add.accumulate(p)[7] < 1.0 <= fast_path_floors(p)[0][7]
    assert fast_path_floors(p)[1]
