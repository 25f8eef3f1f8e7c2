"""Reuse of one ensemble: reset, new sea states, bracket-snap and kernel changes, chained simulate calls.

An hc_ensemble keeps state between calls that its kernels read: the history ring (capacity only grows), prev_time and
the cached force, the radiation and excitation look-ahead blocks (including a pending side-stream slice and the pending
second half of a split excitation build), the switch-off heuristics, the captured graphs, the staged kernel tables,
the wave buffers and the device-stepping buffers.  Sweeps larger than one batch reuse one ensemble, so every call that
starts a new run or changes the configuration must invalidate or re-arm the right parts.

Each case: some prior use of ensemble E, the action under test, then a probe with three checks:
1. a fresh ensemble F, built directly in E's new configuration and given the same probe, matches E bit for bit
   (DESIGN section 7: bitwise reproducibility for equal sizes and configurations) -- total and the three components of
   every instance and DoF at every step; for simulate the records, the energy and the final state;
2. sampled instances against oracle instances driven through the same sequence (1e-9, common.force_tol; 1e-11 where
   the brackets are bit-faithful);
3. which path served the probe: the steps served by radiation blocks (rad_block_stats) and by excitation blocks
   (exc_block_stats), and lookahead_state().  A stale snap or a look-ahead that was not re-armed moves the forces by
   less than the bar; only these counters show it.  They depend on the step times alone, so the check is
   deterministic.  Which kernel variant a block or a per-step evaluation uses is fixed when the ensemble is created
   and is checked by test_gpu_dispatch_coverage.
"""
import functools

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import synth
from oracle import hc_oracle as orc
from test_gpu_device_stepping import _oracle_force, np_simulate
from test_gpu_parity import _acc_times, _assert_parity, _motion

pytestmark = pytest.mark.gpu

G981 = (0.0, 0.0, -9.81)
DT = 0.01
BIG = 16384
BENCH = dict(bracket_snap=1e-8)                        # bench.py's options: both look-aheads automatic
SEA = dict(Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0, nfreq=48, ramp=0.3)
MASS, INERTIA = synth.RM3_MASSES, synth.RM3_INERTIAS
# tables: the RM3 shape with a +-6 s excitation IRF (test_gpu_dispatch_coverage's rm3_short: D = 12, 60 s RIRF, lag
# spacing 6 dt) and the sphere (D = 6: k_rad_block<6>, k_step<6>, the ND = 6 excitation blocks)
KIND_DT = {"rm3_short": DT, "sphere": 0.015}
LOOKAHEAD_CFGS = {"auto_16384": ("rm3_short", BIG, BENCH),
                  "sphere_16384": ("sphere", BIG, BENCH),
                  "dmma_2049": ("rm3_short", 2049, dict(bracket_snap=1e-8, exc_lookahead=5, rad_lookahead=2)),
                  "fma_2049": ("rm3_short", 2049, dict(bracket_snap=1e-8, exc_lookahead=2, rad_lookahead=2))}

_RAW = {}
_TABLES = {}


def _raw(kind="rm3_short"):
    if kind not in _RAW:
        _RAW[kind] = synth.rm3_like(exc_irf_steps=241, exc_half_window=6.0) if kind == "rm3_short" else common.sphere_raw()
    return _RAW[kind]


def _tables(kind="rm3_short"):
    """Shared (hc.Tables, orc.Tables); cases that change the convolution mode build their own."""
    if kind not in _TABLES:
        _TABLES[kind] = (hc.Tables.from_raw(_raw(kind)), orc.Tables(_raw(kind)))
    return _TABLES[kind]


def _sample(B):
    return sorted({0, min(1, B - 1), B // 2, B - 1})


# ---------------------------------------------------------------------------------------------
# wave specifications, applied alike to an ensemble, a multi-device ensemble and one oracle instance
# ---------------------------------------------------------------------------------------------
def _irr(duration, seed0=1, per_instance=False, nfreq=48, kind="rm3_short"):
    return dict(kind="irregular", tables=kind, kw=dict(SEA, dt=KIND_DT[kind], duration=duration, nfreq=nfreq),
                seed0=seed0, per_instance=per_instance)


def _regular_spec(kind="rm3_short"):
    return dict(kind="regular", tables=kind)


def _none_spec(kind="rm3_short"):
    return dict(kind="none", tables=kind)


def _series_spec(duration, kind="rm3_short"):
    return dict(kind="series", tables=kind, duration=duration)


REGULAR = _regular_spec()


def _hs_tp(B):
    b = np.arange(B)
    return 1.0 + 0.05 * (b % 40), 6.0 + 0.13 * (b % 31)


def _regular(B):
    b = np.arange(B)
    return 0.5 + 0.02 * (b % 25), 0.6 + 0.015 * (b % 40)


@functools.lru_cache(maxsize=2)
def _series(kind, B, duration):
    """Per-instance imported elevation on a 0.05 s grid covering the excitation IRF's window."""
    pad = float(np.abs(_raw(kind)["bodies"][0]["exc_irf_t"]).max()) + 2.0
    t = np.linspace(-pad, duration + pad, int(round((duration + 2 * pad) / 0.05)) + 1)
    b = np.arange(B)[:, None]
    return t, 0.6 * np.sin(0.8 * t + 0.3 * b) + 0.25 * np.sin(1.9 * t + 0.11 * b)


def _set_waves(ens, w):
    B = ens.batch
    if w["kind"] == "none":
        ens.set_waves_none()
    elif w["kind"] == "regular":
        ens.set_waves_regular(*_regular(B))
    elif w["kind"] == "series":
        ens.set_waves_series(KIND_DT[w["tables"]], *_series(w["tables"], B, w["duration"]))
    else:
        seeds = w["seed0"] + np.arange(B, dtype=np.int32)
        if w["per_instance"]:
            Hs, Tp = _hs_tp(B)
            ens.set_waves_irregular(seeds=seeds, Hs_per_instance=Hs, Tp_per_instance=Tp, **w["kw"])
        else:
            ens.set_waves_irregular(seeds=seeds, **w["kw"])


def _orc_waves(inst, w, b, B):
    if w["kind"] == "none":
        inst.set_nowave()
    elif w["kind"] == "regular":
        a, om = _regular(B)
        inst.set_regular(float(a[b]), float(om[b]))
    elif w["kind"] == "series":
        t, eta = _series(w["tables"], B, w["duration"])
        inst.set_irregular_series(KIND_DT[w["tables"]], t, eta[b])
    else:
        kw = dict(w["kw"])
        if w["per_instance"]:
            Hs, Tp = _hs_tp(B)
            kw.update(Hs=float(Hs[b]), Tp=float(Tp[b]))
        inst.set_irregular(seed=int(w["seed0"] + b), **kw)


def _oracle(w, sample, B, O=None):
    out = []
    for b in sample:
        i = orc.Instance(O or _tables(w["tables"])[1], omp_mode=0)
        _orc_waves(i, w, b, B)
        out.append(i)
    return out


def _ensemble(B, opts, w, T=None, dt_hint=None):
    e = hc.Ensemble(T or _tables(w["tables"])[0], batch=B, dt_hint=dt_hint or KIND_DT[w["tables"]], **opts)
    _set_waves(e, w)
    return e


def _exc_serves(w, opts, B):
    """Whether the excitation look-ahead is configured for these waves and options (hc_ensemble::setup_lookahead)."""
    if w["kind"] not in ("irregular", "series") or opts.get("exc_lookahead", 0) == 1:
        return False
    return opts.get("exc_lookahead", 0) != 0 or B >= BIG


# ---------------------------------------------------------------------------------------------
# the probe
# ---------------------------------------------------------------------------------------------
def _served(E):
    """(radiation, excitation) steps served by look-ahead blocks since the last call."""
    return E.rad_block_stats()["steps_served"], E.exc_block_stats()["steps_served"]


def _probe(E, F, times, sample=(), insts=(), tag=""):
    """Steps E, and the fresh ensemble F (None: none), through `times` with the prescribed motion; E and F must agree
    bit for bit in the total and in the three components at every step.  Returns (E's forces at `sample`, the oracle
    instances' forces)."""
    D, B = E.dofs, E.batch
    got, want = [], []
    for n, t in enumerate(times):
        pose, vel = _motion(D, B, t)
        a = E.step(t, pose, vel, G981)
        if F is not None:
            b = F.step(t, pose, vel, G981)
            np.testing.assert_array_equal(a, b, err_msg="%s: total, step %d" % (tag, n))
            for what, x, y in zip(("hydrostatic", "radiation", "wave"), E.components(), F.components()):
                np.testing.assert_array_equal(x, y, err_msg="%s: %s component, step %d" % (tag, what, n))
        if insts:
            got.append(a[sample])
            want.append([i.force(t, pose[b], vel[b], G981) for b, i in zip(sample, insts)])
    return np.array(got), np.array(want)


def _probe_fresh(E, opts, w, n, tag, rad_served, exc_served, T=None, dt_hint=None, dt=None):
    """Probe of E from t = 0 after a reset: against a fresh ensemble in the same configuration, against fresh oracle
    instances, and the path: E and F report the same look-ahead state and serve the same steps from blocks, namely
    rad_served radiation and exc_served excitation steps (None: some, as many as F)."""
    B = E.batch
    F = _ensemble(B, opts, w, T=T, dt_hint=dt_hint)
    # (the excitation state is reported only while the waves are irregular: E keeps its look-ahead buffers)
    keys = ("radiation", "excitation") if w["kind"] in ("irregular", "series") else ("radiation",)
    assert all(E.lookahead_state()[k] == F.lookahead_state()[k] for k in keys), (tag, E.lookahead_state(),
                                                                                 F.lookahead_state())
    _served(E)
    sample = _sample(B)
    got, want = _probe(E, F, _acc_times(n, dt or KIND_DT[w["tables"]]), sample, _oracle(w, sample, B), tag=tag)
    _assert_parity(got, want, tag)
    se, sf = _served(E), _served(F)
    assert se == sf, (tag, se, sf)
    assert se[0] == rad_served and (se[1] == exc_served if exc_served is not None else se[1] > 0), (tag, se)
    assert E.history_len() == F.history_len()
    F.close()


# ---------------------------------------------------------------------------------------------
# A. reset
# ---------------------------------------------------------------------------------------------
RESET_CASES = [("rm3_short", "mid_radiation_block"), ("rm3_short", "split_excitation_build"),
               ("rm3_short", "both_switched_off"), ("rm3_short", "ring_grew"), ("sphere", "mid_radiation_block"),
               ("sphere", "both_switched_off")]


@pytest.mark.parametrize("kind,point", RESET_CASES, ids=["%s-%s" % c for c in RESET_CASES])
def test_reset_at_scale(kind, point):
    """16384 instances, bench options.  Reset after 70 steps (inside a radiation block), after 44 steps (the second
    half of the background excitation build is pending: it is launched at the fifth step of a block), after jittered
    step times switched both look-aheads off, or after the history ring grew: dt_hint = 2 dt, 3100 steps of dt >
    the 3040 rows the hint sized the ring for.  Then 150 steps from t = 0 against a fresh ensemble (at 2 dt after the
    ring grew, so that both look-aheads serve the probe on the grown ring; the fresh ensemble's ring never grew)."""
    dt = KIND_DT[kind]
    hint = 2 * dt if point == "ring_grew" else dt
    w = _irr(33.0 if point == "ring_grew" else 8.0, kind=kind)
    E = _ensemble(BIG, BENCH, w, dt_hint=hint)
    D = E.dofs
    if point == "both_switched_off":
        t = 0.0
        for n in range(200):
            pose, vel = _motion(D, BIG, t)
            E.step(t, pose, vel, G981)
            t += dt * (1.0 + 0.37 * ((n * 7) % 5))
            if E.lookahead_state() == {"radiation": 0, "excitation": 0}:
                break
        assert E.lookahead_state() == {"radiation": 0, "excitation": 0}, E.lookahead_state()
    else:
        n0 = {"mid_radiation_block": 70, "split_excitation_build": 44, "ring_grew": 3100}[point]
        for t in _acc_times(n0, dt):
            E.step(t, *_motion(D, BIG, t), G981)
        if point == "ring_grew":
            assert E.history_len() == n0 > 60.0 / hint + 8 + 48
            assert _served(E)[0] <= 3                    # steps of dt on a 2 dt plan: the blocks do not serve
        else:
            assert E.lookahead_state() == {"radiation": 1, "excitation": 1}
            assert _served(E) == (n0 - 1, n0)
    E.reset()
    assert E.history_len() == 0
    assert E.lookahead_state() == {"radiation": 1, "excitation": 1}, E.lookahead_state()
    # after the ring grew the probe steps at 2 dt over an eta grid of dt: the excitation look-ahead serves only the first
    # blocks and then switches itself off (40 of 150 steps on a B200, the fresh ensemble alike); the forces still match
    # the oracle
    _probe_fresh(E, BENCH, w, 150, "reset at %s, %s" % (point, kind), 149, None if point == "ring_grew" else 150,
                 dt_hint=hint, dt=hint)
    if point != "ring_grew":             # (there the excitation look-ahead switches itself off, in F as well)
        assert E.lookahead_state() == {"radiation": 1, "excitation": 1}
    E.close()


@pytest.mark.parametrize("B,rk", [(1, 0), (513, 2), (513, 3)], ids=["compact_B1", "fork_B513_rk2", "fork_B513_rk3"])
def test_reset_per_step_paths(B, rk):
    """B = 1 on the compact graph; B = 513 on the per-step fork path with the DMMA / hybrid radiation kernels (no
    look-ahead at these sizes: no step is served from a block)."""
    opts = dict(rad_kernel=rk) if rk else {}
    w = _irr(6.0)
    E = _ensemble(B, opts, w)
    for t in _acc_times(70, DT):
        E.step(t, *_motion(E.dofs, B, t), G981)
    E.reset()
    assert E.lookahead_state() == {"radiation": -1, "excitation": -1}
    _probe_fresh(E, opts, w, 150, "reset, B = %d, rad_kernel %d" % (B, rk), 0, 0)
    E.close()


# ---------------------------------------------------------------------------------------------
# B. reset followed by new waves
# ---------------------------------------------------------------------------------------------
def _transitions(kind="rm3_short"):
    """irregular -> irregular (other seeds, per-instance Hs / Tp, other nfreq and duration: n_eta changes) -> regular
    (per-instance amplitude and omega) -> irregular -> imported series (per instance) -> irregular -> none ->
    irregular."""
    return [_irr(6.0, kind=kind), _irr(9.5, seed0=1000, per_instance=True, nfreq=64, kind=kind), _regular_spec(kind),
            _irr(6.0, kind=kind), _series_spec(6.0, kind), _irr(7.0, seed0=77, kind=kind), _none_spec(kind),
            _irr(6.0, kind=kind)]


@pytest.mark.parametrize("cfg", list(LOOKAHEAD_CFGS))
def test_reset_then_new_waves(cfg):
    """Each wave set after a reset, probed for 60 steps against a fresh ensemble built with that wave set only.  60
    steps leave E inside a radiation block with the second half of a split excitation build pending."""
    kind, B, opts = LOOKAHEAD_CFGS[cfg]
    seq = _transitions(kind)
    E = _ensemble(B, opts, seq[0])
    for t in _acc_times(60, KIND_DT[kind]):
        E.step(t, *_motion(E.dofs, B, t), G981)
    for k, w in enumerate(seq[1:]):
        E.reset()
        _set_waves(E, w)
        tag = "%s, transition %d to %s" % (cfg, k + 1, w["kind"])
        exc = _exc_serves(w, opts, B)
        if exc:
            assert E.lookahead_state() == {"radiation": 1, "excitation": 1}, (tag, E.lookahead_state())
        _probe_fresh(E, opts, w, 60, tag, 59, 60 if exc else 0)
    E.close()


# ---------------------------------------------------------------------------------------------
# C. new waves without a reset
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", list(LOOKAHEAD_CFGS))
def test_new_waves_mid_run(cfg):
    """The same switches every 29 steps of one run (never on an 8- or 48-step block boundary), the history kept; the
    oracle instances switch at the same step.  Every step is compared with the oracle, so a block built from the old
    elevation that served a step after the switch would show; in every segment with an irregular sea each step takes
    its wave force from a block, in the others none does, and the radiation blocks serve throughout."""
    kind, B, opts = LOOKAHEAD_CFGS[cfg]
    seq = _transitions(kind)
    E = _ensemble(B, opts, seq[0])
    sample = _sample(B)
    insts = _oracle(seq[0], sample, B)
    D, every = E.dofs, 29
    times = _acc_times(every * len(seq), KIND_DT[kind])
    got, ref = [], []
    prev = None
    _served(E)
    for n, t in enumerate(times):
        k = n // every
        if n and n % every == 0:
            w = seq[k]
            _set_waves(E, w)
            for b, i in zip(sample, insts):
                _orc_waves(i, w, b, B)
            if k == 1:
                # a step at the last time returns the cached totals of that time, new waves or not (as the reference)
                again = E.step(times[n - 1], *_motion(D, B, times[n - 1]), G981)
                assert E.last_recomputed is False
                np.testing.assert_array_equal(again, prev)
        pose, vel = _motion(D, B, t)
        F = E.step(t, pose, vel, G981)
        prev = F
        got.append(F[sample])
        ref.append([i.force(t, pose[b], vel[b], G981) for b, i in zip(sample, insts)])
        if n % every == every - 1:
            # every step of a segment with an irregular sea takes its wave force from a block built after the switch
            rad, exc = _served(E)
            assert rad == (every - 1 if k == 0 else every), (cfg, k, rad)
            assert exc == (every if _exc_serves(seq[k], opts, B) else 0), (cfg, k, seq[k]["kind"], exc)
    got, ref = np.array(got), np.array(ref)
    for k in range(len(seq)):
        sl = slice(k * every, (k + 1) * every)
        _assert_parity(got[sl], ref[sl], "%s, %s segment %d" % (cfg, seq[k]["kind"], k))
    E.close()


# ---------------------------------------------------------------------------------------------
# D. set_bracket_snap mid-run
# ---------------------------------------------------------------------------------------------
def test_set_bracket_snap_mid_block():
    """2304 instances (test_mixing_host_and_device_stepping_inside_a_block's size), rad_lookahead = 2, snap 1e-8.
    Invalid values leave everything as it was: the following steps equal a twin's that got no call, bit for bit.
    1e-8 -> 0 inside the second radiation block: no step is served from a block (the per-step kernels serve every
    step), 1e-11 bar.
    0 -> 1e-8 inside what would be the fourth block: the blocks serve again, 1e-9 bar."""
    B = 2304
    opts = dict(bracket_snap=1e-8, rad_lookahead=2)
    w = _irr(4.0)
    E, twin = _ensemble(B, opts, w), _ensemble(B, opts, w)
    assert E.rad_lookahead_steps() == 48 and E.lookahead_state()["excitation"] == -1
    sample = _sample(B)
    insts = _oracle(w, sample, B)
    times = _acc_times(270, DT)
    n_off, n_on = 70, 170
    got, ref, stats = [], [], {}
    for n, t in enumerate(times):
        if n == 30:
            for bad in (-1e-9, 0.5, float("nan")):
                with pytest.raises(hc.HydroError) as ei:
                    E.set_bracket_snap(bad)
                assert ei.value.status == 1, bad
        if n == n_off:
            stats["before"] = E.rad_block_stats(reset=True)
            twin.close()
            E.set_bracket_snap(0.0)
        if n == n_on:
            stats["off"] = E.rad_block_stats(reset=True)
            stats["off_state"] = E.lookahead_state()["radiation"]
            E.set_bracket_snap(1e-8)
            assert E.lookahead_state()["radiation"] == 1
        pose, vel = _motion(E.dofs, B, t)
        F = E.step(t, pose, vel, G981)
        if n < n_off:
            np.testing.assert_array_equal(F, twin.step(t, pose, vel, G981), err_msg="step %d" % n)
        got.append(F[sample])
        ref.append([i.force(t, pose[b], vel[b], G981) for b, i in zip(sample, insts)])
    stats["on"] = E.rad_block_stats(reset=True)
    got, ref = np.array(got), np.array(ref)
    assert stats["before"]["steps_served"] == n_off - 1, stats
    assert stats["off"]["steps_served"] == 0 and stats["off_state"] == 0, stats
    assert stats["on"]["steps_served"] == len(times) - n_on, stats
    _assert_parity(got[:n_off], ref[:n_off], "snap 1e-8")
    worst = _assert_parity(got[n_off:n_on], ref[n_off:n_on], "snap 0", rel=1e-11)
    _assert_parity(got[n_on:], ref[n_on:], "snap 1e-8 again")
    print("snap 0 segment: worst %.2e" % worst)
    E.close()


# ---------------------------------------------------------------------------------------------
# E. refresh_rirf while the look-aheads serve
# ---------------------------------------------------------------------------------------------
TAPER = dict(smoothing="sg", window_length=5, rirf_end_time=10.0, taper_start_percent=0.1, taper_end_percent=0.5,
             taper_final_amplitude=0.0)
ORC_TAPER = dict(smoothing="sg", window_length=5, rirf_end_time=10.0, start=0.1, end=0.5, final=0.0)
REFRESH_CFGS = {"auto_16384": (BIG, BENCH), "rk1_513": (513, dict(rad_kernel=1)),
                "rk2_513": (513, dict(rad_kernel=2)), "rk3_513": (513, dict(rad_kernel=3)), "compact_B1": (1, {})}


@pytest.mark.parametrize("cfg", list(REFRESH_CFGS))
def test_refresh_rirf_mid_block(cfg):
    """TaperedDirect (taper from 1 s to 5 s) + refresh_rirf after 130 steps (inside the third radiation block), back
    to Baseline after 230 steps (inside the fifth).  The oracle switches its tables at the same step; for the return
    to Baseline it is rebuilt on fresh tables and loaded with the history the GPU holds.  A Baseline oracle run next
    to it shows that the first step after the first switch moves by far more than the bar."""
    B, opts = REFRESH_CFGS[cfg]
    raw = _raw()
    T, O, O_base = hc.Tables.from_raw(raw), orc.Tables(raw), orc.Tables(raw)
    w = _irr(5.0)
    E = _ensemble(B, opts, w, T=T)
    sample = _sample(B)
    insts, base = _oracle(w, sample, B, O), _oracle(w, sample, B, O_base)
    n1, n2 = 130, 230
    times = _acc_times(330, DT)
    D = E.dofs
    got, ref, ref_base = [], [], []
    _served(E)
    for n, t in enumerate(times):
        if n == n1:
            T.set_convolution_mode("TaperedDirect", **TAPER)
            O.set_tapered(**ORC_TAPER)
            E.refresh_rirf()
        if n == n2:
            T.set_convolution_mode("Baseline")
            E.refresh_rirf()
            O = orc.Tables(raw)
            insts = _oracle(w, sample, B, O)
            hist = times[:n][::-1]
            vel = np.array([_motion(D, B, tt)[1][sample] for tt in hist])
            for j, i in enumerate(insts):
                i.set_history(hist, vel[:, j])
        pose, vel = _motion(D, B, t)
        F = E.step(t, pose, vel, G981)
        got.append(F[sample])
        ref.append([i.force(t, pose[b], vel[b], G981) for b, i in zip(sample, insts)])
        if n <= n1:
            ref_base.append([i.force(t, pose[b], vel[b], G981) for b, i in zip(sample, base)])
    got, ref = np.array(got), np.array(ref)
    moved = np.abs(ref[n1] - ref_base[n1]) / common.force_tol(np.array(ref_base))[n1]
    assert moved.max() > 1e3, moved.max()
    for lo, hi, what in ((0, n1, "Baseline"), (n1, n2, "TaperedDirect"), (n2, len(times), "Baseline again")):
        _assert_parity(got[lo:hi], ref[lo:hi], "%s, %s" % (cfg, what))
    # 16384: the blocks serve every step, the first one after each refresh rebuilt with the new kernel
    assert _served(E) == ((len(times) - 1, len(times)) if B == BIG else (0, 0)), (cfg, _served(E))
    E.close()


# ---------------------------------------------------------------------------------------------
# F. device stepping reused
# ---------------------------------------------------------------------------------------------
def _pose0(B):
    pose0 = np.zeros((B, 12))
    pose0[:, [3, 4, 9, 10]] = [0.03, -0.02, 0.01, 0.04]
    return pose0


def test_euler_split_into_three_calls_at_scale():
    """16384 instances, both look-aheads: 160 Euler steps as 52 + 48 + 60.  Both split points lie inside a radiation
    block and leave the second half of a split excitation build pending.  Records and final state equal one call's
    bit for bit; each call zeroes its energy, so the sum of the three equals one call's energy to rounding."""
    w = _irr(6.0)
    c = np.linspace(1e3, 1e5, BIG)[:, None] * np.ones(12)
    kw = dict(pto_damping=c, record_every=4)
    pose0 = _pose0(BIG)
    F = _ensemble(BIG, BENCH, w)
    one = F.simulate(pose0, 160, DT, MASS, INERTIA, **kw)
    f_served = _served(F)
    F.close()
    E = _ensemble(BIG, BENCH, w)
    parts, pose, vel, t0 = [], pose0, None, 0.0
    for m in (52, 48, 60):
        r = E.simulate(pose, m, DT, MASS, INERTIA, vel0=vel, t0=t0, **kw)
        parts.append(r)
        pose, vel, t0 = r.final_pose, r.final_vel, r[0][-1]
    assert E.lookahead_state() == {"radiation": 1, "excitation": 1}
    e_served = _served(E)
    assert e_served == f_served and e_served[0] >= 158 and e_served[1] == 160, (e_served, f_served)
    for k in range(3):
        np.testing.assert_array_equal(np.concatenate([p[k] for p in parts]), one[k])
    np.testing.assert_array_equal(pose, one.final_pose)
    np.testing.assert_array_equal(vel, one.final_vel)
    np.testing.assert_allclose(sum(p[3] for p in parts), one[3], rtol=1e-12, atol=0.0)
    assert np.abs(one[3]).max() > 0.0
    E.close()


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_simulate_reset_new_sea_matches_fresh(scheme):
    """simulate -> reset -> new sea state -> simulate equals a fresh ensemble's simulate, bit for bit.  The first call
    records every 50th step, so the record buffers start small and the second call must grow them.  The second call's
    initial angles equal the first call's final angles bit for bit for even instances (the continuation keep rule must
    not apply after a reset) and differ for odd ones."""
    B = 65
    opts = dict(bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=4)
    w1, w2 = _irr(4.0), _irr(5.0, seed0=500, per_instance=True)
    E = _ensemble(B, opts, w1)
    a = E.simulate(_pose0(B), 100, DT, MASS, INERTIA, scheme=scheme, pto_damping=1e4, record_every=50)
    assert np.abs(a.final_pose[:, [3, 4, 9, 10]] - _pose0(B)[:, [3, 4, 9, 10]]).min() > 0.0
    E.reset()
    _set_waves(E, w2)
    _served(E)
    pose1 = 1.5 * _pose0(B)
    pose1[::2] = a.final_pose[::2]
    vel1 = np.zeros((B, 12))
    vel1[::2] = a.final_vel[::2]
    kw = dict(vel0=vel1, scheme=scheme, pto_damping=2e4, pto_stiffness=1e3)
    r = E.simulate(pose1, 120, DT, MASS, INERTIA, **kw)
    F = _ensemble(B, opts, w2)
    f = F.simulate(pose1, 120, DT, MASS, INERTIA, **kw)
    for k, what in enumerate(("times", "pose", "vel", "energy")):
        np.testing.assert_array_equal(r[k], f[k], err_msg=what)
    np.testing.assert_array_equal(r.final_pose, f.final_pose)
    np.testing.assert_array_equal(r.final_vel, f.final_vel)
    se, sf = _served(E), _served(F)
    assert se == sf and se[0] > 100 and se[1] == 120 + (scheme == "hht"), (se, sf)       # HHT: n + 1 evaluations
    assert E.lookahead_state() == F.lookahead_state() == {"radiation": 1, "excitation": 1}
    E.close(); F.close()


def test_step_between_simulate_calls():
    """simulate, one hc_step at the next time, then simulate from the time after: against the numpy restatement of
    Euler driven by oracle instances that saw the same steps."""
    B, n1, n2 = 3, 80, 90
    T, O = _tables()
    E = _ensemble(B, {}, REGULAR)
    insts = _oracle(REGULAR, range(B), B)
    pose0, c = _pose0(B), 5e4
    a = E.simulate(pose0, n1, DT, MASS, INERTIA, pto_damping=c)
    t1 = a[0][-1]
    E.step(t1, a.final_pose, a.final_vel, G981)
    assert E.last_recomputed
    t2 = t1 + DT
    b = E.simulate(a.final_pose, n2, DT, MASS, INERTIA, vel0=a.final_vel, t0=t2, pto_damping=c)
    f = _oracle_force(insts)
    _, xr, vr = np_simulate(f, T.added_mass(), MASS, INERTIA, pose0, n1, DT, c=c)
    f(t1, xr[-1], vr[-1])
    tr2, xr2, _ = np_simulate(lambda t, p, v: f(t2 + t, p, v), T.added_mass(), MASS, INERTIA, xr[-1], n2, DT, c=c,
                              vel0=vr[-1])
    assert insts[0].history_len() == E.history_len()
    for j in range(B):
        amp = np.abs(xr2[:, j] - xr2[0, j]).max()
        assert amp > 1e-3
        assert np.abs(a[1][:, j] - xr[:, j]).max() <= 1e-8 * np.abs(xr[:, j] - xr[0, j]).max(), j
        assert np.abs(b[1][:, j] - xr2[:, j]).max() <= 1e-8 * amp, j
    E.close()


# ---------------------------------------------------------------------------------------------
# G. multi-device handle
# ---------------------------------------------------------------------------------------------
def test_multi_reset_then_new_waves():
    """MultiEnsemble on devices [0, 0] (shards of 4 and 3 instances): reset + new waves, then step and simulate, bit
    for bit a fresh MultiEnsemble's."""
    T, _ = _tables()
    B = 7
    opts = dict(dt_hint=DT, bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=4)
    w1, w2 = _irr(4.0), _irr(5.0, seed0=40, per_instance=True)
    E = hc.MultiEnsemble(T, B, devices=[0, 0], **opts)
    assert [s["count"] for s in E.shards()] == [4, 3]
    _set_waves(E, w1)
    for t in _acc_times(30, DT):
        E.step(t, *_motion(12, B, t), G981)
    E.reset()
    _set_waves(E, w2)
    F = hc.MultiEnsemble(T, B, devices=[0, 0], **opts)
    _set_waves(F, w2)
    times = _acc_times(41, DT)
    for t in times[:40]:
        pose, vel = _motion(12, B, t)
        np.testing.assert_array_equal(E.step(t, pose, vel, G981), F.step(t, pose, vel, G981))
        for x, y in zip(E.components(), F.components()):
            np.testing.assert_array_equal(x, y)
    pose0 = _pose0(B)
    r, f = (m.simulate(pose0, 60, DT, MASS, INERTIA, t0=times[40], scheme="hht", pto_damping=1e4) for m in (E, F))
    for k in range(4):
        np.testing.assert_array_equal(r[k], f[k])
    np.testing.assert_array_equal(r.final_pose, f.final_pose)
    E.close(); F.close()


# ---------------------------------------------------------------------------------------------
# H. end of the eta window on the look-ahead paths
# ---------------------------------------------------------------------------------------------
def _window_steps(duration):
    """Steps at t = 0, dt, 2 dt, ... (repeated addition) whose excitation window lies inside the eta grid of an
    irregular sea of this duration (the library's bounds test: eta_t[0] <= t - tau_last, t - tau_first <= eta_t[-1])."""
    e = hc.Ensemble(_tables()[0], batch=1, dt_hint=DT)
    _set_waves(e, _irr(duration))
    ir = e.irregular(0)
    e.close()
    lo, hi = ir["eta_t"][0], ir["eta_t"][-1]
    taus = [(g["t"][0], g["t"][-1]) for g in ir["irf"]]
    n, t = 0, 0.0
    while all(lo <= t - tl and t - tf <= hi for tf, tl in taus):
        n += 1
        t += DT
    return n


def _duration_for(last_block):
    """A sea duration whose final 8-step excitation block holds `last_block` (< 8) steps."""
    for d in np.arange(0.3, 0.5, 0.01):
        if _window_steps(float(d)) % 8 == last_block:
            return float(d)
    raise AssertionError("no duration gives a final block of %d steps" % last_block)


EDGE_CFGS = [(65, 2), (65, 4), (65, 5), (2049, 2), (2049, 4), (2049, 5), (BIG, 0)]


@pytest.mark.parametrize("B,xl", EDGE_CFGS, ids=["B%d_exc%d" % c for c in EDGE_CFGS])
def test_eta_window_end_on_lookahead_paths(B, xl):
    """Every step up to the last time inside the eta window against the oracle; the final excitation block holds 3 or
    5 steps (unused warps recompute the last time, eta rows clamp to n_eta - 1, no prefetch) and serves them: every
    step's wave force comes from a block.  The next step raises EtaWindowError and leaves the reference's state
    (sample pushed, cached zero totals at that time).  Then reset + a longer sea, probed against a fresh ensemble."""
    opts = dict(BENCH) if xl == 0 else dict(bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=xl)
    last = 3 if (B + xl) % 2 else 5
    dur = _duration_for(last)
    n_ok = _window_steps(dur)
    assert 0 < n_ok % 8 == last < 8
    w = _irr(dur)
    E = _ensemble(B, opts, w)
    sample = _sample(B)
    insts = _oracle(w, sample, B)
    times = _acc_times(n_ok + 1, DT)
    got, want = _probe(E, None, times[:n_ok], sample, insts, tag="B = %d, exc_lookahead %d" % (B, xl))
    _assert_parity(got, want, "up to the end of the eta window, B = %d, exc_lookahead %d" % (B, xl))
    # every step, those of the short final block included, took its wave force from a block
    assert _served(E) == (n_ok - 1, n_ok), (_served(E), n_ok)
    assert E.lookahead_state() == {"radiation": 1, "excitation": 1}
    t, D = times[n_ok], E.dofs
    pose, vel = _motion(D, B, t)
    with pytest.raises(orc.OracleError):
        insts[0].force(t, pose[0], vel[0], G981)
    hl = E.history_len()
    with pytest.raises(hc.EtaWindowError):
        E.step(t, pose, vel, G981)
    assert E.history_len() == hl + 1 == insts[0].history_len()
    F0 = E.step(t, pose, vel, G981)
    assert E.last_recomputed is False and np.all(F0 == 0.0)
    E.reset()
    w2 = _irr(dur + 2.0, seed0=9)
    _set_waves(E, w2)
    _probe_fresh(E, opts, w2, 60, "after the window error, B = %d, exc %d" % (B, xl), 59, 60)
    E.close()
