"""Host-side planning of the radiation look-ahead (hc_plan.cpp) against a restatement of the reference's bracket
logic (TestHydro::AdvanceToBracket / InterpolateVelocity6D, src/hydro_forces.cpp:343-381,601-610).  CPU only."""
import math

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import synth


def reference_plan(times, rirf_t):
    """Per lag: None (no bracket) or the position of the query in history rows back from the step
    (bracket index + weight of the older row), from the reference's own arithmetic."""
    tm = list(times)
    out = []
    for ts in rirf_t:
        q = tm[0] - ts
        if not (tm[-1] <= q):
            out.append(None)
            continue
        i = 0
        while not (tm[i + 1] <= q):          # AdvanceToBracket: smallest i with time(i+1) <= q
            i += 1
        newer, older = tm[i], tm[i + 1]
        if q == older:
            out.append(float(i + 1))
        elif q == newer:
            out.append(float(i))
        else:
            out.append(i + (newer - q) / (newer - older))
    return out


def history(n, dt, window):
    """Time history at step n of a run t += dt from 0, newest first, pruned like PruneHistory (:327-340)."""
    t, ts = 0.0, [0.0]
    for _ in range(n):
        t += dt
        ts.append(t)
    tm = ts[::-1]
    t_min = tm[0] - window
    while len(tm) > 1 and tm[len(tm) - 2] < t_min:
        tm.pop()
    return tm


def expected(tm, rirf_t, pnom, snap, need_all):
    plan = reference_plan(tm, rirf_t)
    smax = -1
    for s, p in enumerate(plan):
        if p is None:
            break
        if abs(p - pnom[s]) > snap:
            return -1
        smax = s
    if need_all and smax != len(rirf_t) - 1:
        return -1
    return smax


@pytest.mark.parametrize("nb,steps,duration,dt,mode,m", [
    (2, 1001, 60.0, 0.01, 1, 6),       # the headline workload: lag spacing 0.06 = 6 dt
    (1, 401, 4.0, 0.01, 1, 1),         # lag spacing = dt
    (2, 601, 30.0, 0.03, 2, 1),        # OSWEC shape: ratio 5/3 -> row grid
    (3, 401, 20.0, 0.02, 2, 1),        # F3OF shape: ratio 5/2 -> row grid
])
def test_plan_and_step_check(nb, steps, duration, dt, mode, m):
    raw = synth.make_tables(num_bodies=nb, rirf_steps=steps, rirf_duration=duration)
    T = hc.Tables.from_raw(raw)
    rirf_t = np.linspace(0.0, duration, steps)
    got_mode, got_m, lk = T.rad_lookahead_plan(dt)
    assert (got_mode, got_m) == (mode, m)
    pnom = (m * np.arange(steps)).astype(float) if mode == 1 else rirf_t / dt
    assert lk == (steps if mode == 1 else math.floor(pnom[-1]) + 2)
    full = int(round(duration / dt))
    for n in (1, 2, 7, full // 3, full - 1, full, full + 1, full + 57):
        tm = history(n, dt, duration)
        for snap in (1e-8, 0.0):
            want = expected(tm, rirf_t, pnom, snap, need_all=(mode == 2))
            got = T.rad_lookahead_check_step(dt, snap, tm)
            # snap = 0 asks for exact hits: the device snaps nothing either, both sides must agree lag by lag
            assert got == want, (n, snap, got, want)
    # with the window full and snapped brackets every step is served
    assert T.rad_lookahead_check_step(dt, 1e-8, history(full + 5, dt, duration)) == steps - 1


def test_irregular_steps_are_rejected():
    raw = synth.rm3_like()
    T = hc.Tables.from_raw(raw)
    rng = np.random.default_rng(3)
    ts = np.concatenate([[0.0], np.cumsum(rng.uniform(0.004, 0.012, size=400))])
    assert T.rad_lookahead_check_step(0.01, 1e-8, ts[::-1].copy()) == -1
    # one perturbed row in an otherwise uniform history: the lags that land on it are off by 3e-3 rows
    tm = np.array(history(300, 0.01, 60.0))
    assert T.rad_lookahead_check_step(0.01, 1e-8, tm) >= 0
    tm[120] += 3e-5
    assert T.rad_lookahead_check_step(0.01, 1e-8, tm) == -1
    # a step size the plan was not made for
    assert T.rad_lookahead_check_step(0.02, 1e-8, np.array(history(300, 0.01, 60.0))) == -1
    assert T.rad_lookahead_plan(0.0007)[0] == 0          # 86 rows per lag: neither grid pays off


@pytest.mark.parametrize("nb,steps,duration,dt", [(2, 601, 30.0, 0.03), (1, 401, 4.0, 0.01), (2, 1001, 60.0, 0.01)])
def test_row_kernel_reproduces_the_reference_convolution(nb, steps, duration, dt):
    """sum_s K[:, :, s] w[s] lerp(v, t - t_s)  (hydro_forces.cpp:586-647)  ==  sum_i Krow[i] v[row i]  for a history on a
    uniform grid: the row-grid kernel folds the interpolation weights in, the lag-grid kernel is (K w) itself."""
    _check_row_kernel(synth.make_tables(num_bodies=nb, rirf_steps=steps, rirf_duration=duration), nb, steps, duration, dt)


@pytest.mark.parametrize("nb,steps,duration,dt", [(2, 601, 30.0, 0.03), (1, 401, 4.0, 0.01), (2, 1001, 60.0, 0.01)])
def test_row_kernel_reproduces_the_reference_convolution_asymmetric(nb, steps, duration, dt):
    """The same identity with non-symmetric K (common.asymmetric_tables): on symmetric K a row kernel applied
    transposed would pass it."""
    raw = common.asymmetric_tables(synth.make_tables(num_bodies=nb, rirf_steps=steps, rirf_duration=duration))
    _check_row_kernel(raw, nb, steps, duration, dt)


def _check_row_kernel(raw, nb, steps, duration, dt):
    T = hc.Tables.from_raw(raw)
    D = 6 * nb
    mode, m, lk = T.rad_lookahead_plan(dt)
    Krow = T.rad_lookahead_row_kernel(dt)
    assert Krow.shape == (lk, D, D)
    K = T.rirf()                      # [D][D][L], what GetRIRFval returns
    w = T.rirf_width()
    rirf_t = T.rirf_time()
    n = int(round(duration / dt)) + 9
    tm = np.array(history(n, dt, duration))
    rng = np.random.default_rng(8)
    v = rng.standard_normal((len(tm), D))              # row i = velocity sample at tm[i]
    plan = reference_plan(tm, rirf_t)
    ref = np.zeros(D)
    for s, p in enumerate(plan):
        assert p is not None
        i = int(math.floor(p))
        wo = p - i
        vq = v[i] if wo == 0.0 else (1.0 - wo) * v[i] + wo * v[i + 1]
        ref += K[:, :, s] @ (vq * w[s])
    rows = m * np.arange(lk) if mode == 1 else np.arange(lk)
    rows = rows[rows < len(tm)]
    got = np.einsum("irc,ic->r", Krow[: len(rows)], v[rows])
    # the reference gives the neighbouring row a weight of the size of the rounding noise of the accumulated times
    # (|p - p_nominal| ~ 1e-11 rows at t ~ 60 s); with white-noise rows that is the whole difference.  The block path
    # is only used when that offset is below bracket_snap (1e-8 in bench.py), the bound asserted here.
    dev = max(abs(p - q) for p, q in zip(plan, (m * np.arange(steps)).astype(float) if mode == 1 else rirf_t / dt))
    assert dev < 1e-8
    assert np.abs(got - ref).max() <= max(1e-12, 50 * dev) * np.abs(ref).max()


@pytest.mark.parametrize("nb,steps,duration,dt", [(2, 1001, 60.0, 0.01), (2, 601, 30.0, 0.03)])
@pytest.mark.parametrize("base_blocks", [0, 1])
def test_block_decomposition_is_the_full_convolution(nb, steps, duration, dt, base_blocks):
    """The identity k_rad_block<D> / k_step<D> are built on (DESIGN.md section 4), written out with numpy on the
    library's own row kernel: for a block whose snapshot of the history was taken `base` steps before its first step,
        F_j = sum_u Krow[u + g + 1] v_res[m u + m - 1 - rho]  +  sum_{l <= jj / m} Krow[l] v_young[jj - m l],
    jj = base + j = rho + m g, equals the convolution of all rows with the row kernel."""
    _check_block_decomposition(synth.make_tables(num_bodies=nb, rirf_steps=steps, rirf_duration=duration), nb, dt,
                               base_blocks)


@pytest.mark.parametrize("nb,steps,duration,dt", [(2, 1001, 60.0, 0.01), (2, 601, 30.0, 0.03)])
@pytest.mark.parametrize("base_blocks", [0, 1])
def test_block_decomposition_is_the_full_convolution_asymmetric(nb, steps, duration, dt, base_blocks):
    """The same identity with non-symmetric K (common.asymmetric_tables)."""
    raw = common.asymmetric_tables(synth.make_tables(num_bodies=nb, rirf_steps=steps, rirf_duration=duration))
    _check_block_decomposition(raw, nb, dt, base_blocks)


def _check_block_decomposition(raw, nb, dt, base_blocks):
    T = hc.Tables.from_raw(raw)
    D = 6 * nb
    mode, m, lk = T.rad_lookahead_plan(dt)
    K = T.rad_lookahead_row_kernel(dt)                      # [lk][D][D], one entry per lag (lag grid) or row (row grid)
    TT = 8 * m
    base = base_blocks * TT
    n0 = m * (lk - 1) + 40                                  # snapshot step: the window is full
    rng = np.random.default_rng(5)
    v = rng.standard_normal((n0 + 2 * TT + 1, D))           # v[n] = velocity sample of step n
    for j in (0, 1, m - 1 if m > 1 else 2, TT // 2, TT - 1):
        jj = base + j
        n = n0 + jj                                         # this step
        # direct: lag s (lag grid) or row i (row grid) reads the sample m s (or i) steps back
        direct = sum(K[s] @ v[n - m * s] for s in range(lk))
        rho, g = jj % m, jj // m
        # resident rows: r = 0 is the newest sample before the snapshot step, i.e. step n0 - 1 - r
        resident = np.zeros(D)
        u = 0
        while u + g + 1 < lk:
            r = m * u + (m - 1 - rho)
            resident += K[u + g + 1] @ v[n0 - 1 - r]
            u += 1
        # young rows: appended by the snapshot step and after it, k = jj - m l steps after the snapshot
        young = sum(K[l] @ v[n0 + jj - m * l] for l in range(min(g, lk - 1) + 1))
        assert np.abs(resident + young - direct).max() <= 1e-12 * np.abs(direct).max(), (j, jj)


def test_pass_slices_tile_the_work_items_whatever_the_policy():
    """The slices a look-ahead pass is launched in (hc_plan.cpp::rad_pass_next) cover [0, N) exactly once, also when
    the rounding of the boundaries (whole waves for device-resident stepping, equal slices for host-buffer stepping)
    changes in the middle of the pass."""
    import ctypes as C
    from hydrochrono_b200._capi import lib
    rng = np.random.default_rng(12)
    for N, nsl in ((27648, 48), (1536, 48), (59904, 8), (7, 48), (444 * 5, 16)):
        for trial in range(20):
            ns, ni = C.c_int(0), C.c_longlong(0)
            covered, launches = [], 0
            while ns.value < nsl:
                wave = int(rng.choice([1, 444, 296]))
                count = int(rng.choice([1, 1, 1, 4]))
                i0, i1 = C.c_longlong(), C.c_longlong()
                any_ = lib.hc_rad_pass_next(N, nsl, C.byref(ns), C.byref(ni), count, wave, C.byref(i0), C.byref(i1))
                if any_:
                    assert i1.value > i0.value
                    covered.append((i0.value, i1.value))
                    launches += 1
                else:
                    assert i1.value == i0.value
            assert covered[0][0] == 0 and covered[-1][1] == N
            assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
    # one policy throughout: wave-aligned boundaries (except the end), equal slices with wave = 1
    ns, ni = C.c_int(0), C.c_longlong(0)
    ends = []
    for _ in range(48):
        i0, i1 = C.c_longlong(), C.c_longlong()
        lib.hc_rad_pass_next(27648, 48, C.byref(ns), C.byref(ni), 1, 444, C.byref(i0), C.byref(i1))
        ends.append(i1.value)
    assert all(e % 444 == 0 for e in ends[:-1]) and ends[-1] == 27648
    ns, ni = C.c_int(0), C.c_longlong(0)
    ends = []
    for _ in range(48):
        i0, i1 = C.c_longlong(), C.c_longlong()
        lib.hc_rad_pass_next(27648, 48, C.byref(ns), C.byref(ni), 1, 1, C.byref(i0), C.byref(i1))
        ends.append(i1.value)
    assert ends == [576 * (k + 1) for k in range(48)]
