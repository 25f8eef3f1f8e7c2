"""Water kinematics of every ensemble instance on the device (hc_waves_kinematics_at_time, k_wave_kinematics): the
elevation, particle velocity and acceleration of WaveBase::GetElevation / GetVelocity / GetAcceleration
(src/wave_types.cpp:14-160,301-313,515-550) for each instance's own wave at its own points.

Bar: for each output component |got - ref| <= 1e-12 * sum_i |term_i|, the same sum with every cos / sin replaced by 1
(the scale the rounding error is proportional to; meaningful where the sum cancels).  References: the CPU oracle's
restatement of the reference (orc.Instance.kinematics), and, for whole populations, the vectorised numpy restatement
below, which also yields the bar.
"""
import os
import subprocess

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import _capi, h5io, synth
from oracle import hc_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "hydrochrono_b200", "host")
BAR = 1e-12
DT = 0.05
SEA = dict(dt=DT, duration=30.0, ramp=5.0, Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0)


@pytest.fixture(scope="module")
def host_build():
    subprocess.check_call(["make", "-C", HOST, "-j8"], stdout=subprocess.DEVNULL)
    return os.path.join(HOST, "build")


_RAW = {}


def _raw(depth):
    if depth not in _RAW:
        _RAW[depth] = synth.make_tables(num_bodies=1, rirf_steps=201, rirf_duration=10.0, exc_irf_steps=201,
                                        exc_half_window=5.0, water_depth=float(depth))
    return _RAW[depth]


def _points(B, P, seed=3):
    """[B][P][3]: x in +-50 m, z below, at and above the mean water level (first three points fixed)."""
    rng = np.random.default_rng(seed + 1000 * P + B)
    pts = np.empty((B, P, 3))
    pts[..., 0] = rng.uniform(-50.0, 50.0, (B, P))
    pts[..., 1] = rng.uniform(-5.0, 5.0, (B, P))
    pts[..., 2] = rng.uniform(-12.0, 1.0, (B, P))
    fixed = [(0.0, 0.0, -6.0), (-50.0, 1.0, 0.0), (50.0, 0.0, 0.7)]
    for p in range(min(P, 3)):
        pts[:, p] = fixed[p]
    return pts


def restate(om, k, A, ph, pts, t, depth, mwl, wheeler):
    """numpy restatement; om, k, A, ph broadcast to [B][nf], pts [B][P][3] -> ((eta, vel, acc), (bars))."""
    B = pts.shape[0]
    om, k, A, ph = (np.broadcast_to(np.asarray(v, dtype=np.float64), (B, np.shape(v)[-1]))[:, None, :]
                    for v in (om, k, A, ph))
    x = pts[..., 0:1]
    z = pts[..., 2:3] - mwl
    arg = (k * x - om * t) + ph
    c, s = np.cos(arg), np.sin(arg)
    eta = (A * c).sum(-1)
    eta_bar = np.broadcast_to(np.abs(A).sum(-1), eta.shape)
    if wheeler:
        z = depth * (z - eta[..., None]) / (depth + eta[..., None]) - mwl
    deep = (2 * np.pi / k > depth) | (k * depth > 500.0)
    with np.errstate(over="ignore", invalid="ignore"):
        e = np.exp(k * z)
        shkd = np.sinh(k * depth)
        fx = np.where(deep, e, np.cosh(k * (z + depth)) / shkd)
        fz = np.where(deep, e, np.sinh(k * (z + depth)) / shkd)
    oa, ooa = om * A, om * om * A
    zero = np.zeros_like(eta)
    vel = np.stack([(oa * fx * c).sum(-1), zero, (oa * fz * s).sum(-1)], -1)
    acc = np.stack([(ooa * fx * s).sum(-1), zero, -(ooa * fz * c).sum(-1)], -1)
    vbar = np.stack([np.abs(oa * fx).sum(-1), zero, np.abs(oa * fz).sum(-1)], -1)
    abar = np.stack([np.abs(ooa * fx).sum(-1), zero, np.abs(ooa * fz).sum(-1)], -1)
    return (eta, vel, acc), (eta_bar, vbar, abar)


def _assert_bar(got, ref, bars, what=""):
    for g, r, b, name in zip(got, ref, bars, ("eta", "vel", "acc")):
        err = np.abs(np.asarray(g) - np.asarray(r))
        bad = err > BAR * np.asarray(b)
        assert not bad.any(), (what, name, np.argwhere(bad)[:5], float((err / np.maximum(b, 1e-300)).max()))


def _components(ens, idx):
    """Components of the ensemble's current irregular waves for instances idx: om, k [nf]; A, ph [len(idx)][nf]."""
    d = ens.irregular(0)
    om, k, w = 2 * np.pi * d["freqs"], d["wavenumbers"], d["widths"]
    A, ph = np.empty((len(idx), om.size)), np.empty((len(idx), om.size))
    for j, b in enumerate(idx):
        S, p = np.empty(om.size), np.empty(om.size)
        hc._check(_capi.lib.hc_waves_irregular_spectrum(ens._h, int(b), None, hc._dp(S), None, hc._dp(p), None))
        A[j], ph[j] = np.sqrt(2 * S * w), p
    return om, k, A, ph


def _irregular_ensemble(T, B, kind, seeds, nfreq, **kw):
    ens = hc.Ensemble(T, batch=B, **kw)
    sea = dict(SEA, nfreq=nfreq)
    if kind == "per_instance":
        hs, tp = _hs_tp(B)
        ens.set_waves_irregular(seeds=seeds, Hs_per_instance=hs, Tp_per_instance=tp, **sea)
    else:
        ens.set_waves_irregular(seeds=seeds, **sea)
    return ens


def _hs_tp(B):
    b = np.arange(B)
    return 1.0 + 0.07 * (b % 23), 5.0 + 0.21 * (b % 29)


# ---------------------------------------------------------------------------------------------
# 1. oracle parity for each wave kind
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth", [200.0, 30.0])
@pytest.mark.parametrize("kind", ["regular", "irregular_shared", "per_instance"])
def test_oracle_parity_per_wave_kind(kind, depth):
    B, P = 5, 7
    raw = _raw(depth)
    T, O = hc.Tables.from_raw(raw), orc.Tables(raw)
    seeds = np.array([3, 17, 4242, 9, 123456], dtype=np.int32)
    insts = []
    if kind == "regular":
        amp = np.array([0.4, 1.1, 2.0, 0.05, 0.9])
        om = np.array([0.35, 0.9, 1.7, 3.1, 4.6])
        ph = np.array([0.0, 1.3, -2.2, 5.9, 0.7])
        ens = hc.Ensemble(T, batch=B)
        ens.set_waves_regular(amp, om, ph)
        for b in range(B):
            i = orc.Instance(O)
            i.set_regular(amp[b], om[b], ph[b])
            insts.append(i)
        comps = (om[:, None], np.array([[ens.regular_coeffs(b)[2]] for b in range(B)]), amp[:, None], ph[:, None])
    else:
        ens = _irregular_ensemble(T, B, kind, seeds, 200)
        hs, tp = _hs_tp(B)
        for b in range(B):
            i = orc.Instance(O)
            kw = dict(SEA, nfreq=200, seed=int(seeds[b]))
            if kind == "per_instance":
                kw.update(Hs=float(hs[b]), Tp=float(tp[b]))
            i.set_irregular(share_irf_from=insts[0] if insts else None, **kw)
            insts.append(i)
        comps = _components(ens, range(B))
        deep = (2 * np.pi / comps[1] > depth) | (comps[1] * depth > 500.0)
        if depth == 200.0:
            assert deep.any() and not deep.all()         # the sea state reaches both branches
    pts = _points(B, P)
    for t in (0.0, 2.3, 1000.37):
        for mwl, wheeler in ((0.0, False), (0.45, False), (0.0, True), (-0.3, True)):
            got = ens.wave_kinematics(t, pts, mwl=mwl, wheeler=wheeler)
            _, bars = restate(*comps, pts, t, depth, mwl, wheeler and kind != "regular")
            ref = [np.empty((B, P)), np.empty((B, P, 3)), np.empty((B, P, 3))]
            for b in range(B):
                for p in range(P):
                    e, v, a = insts[b].kinematics(pts[b, p], t, wave_stretching=wheeler, mwl=mwl)
                    ref[0][b, p], ref[1][b, p], ref[2][b, p] = e, v, a
            _assert_bar(got, ref, bars, (kind, depth, t, mwl, wheeler))


# ---------------------------------------------------------------------------------------------
# 2. the whole population at scale
# ---------------------------------------------------------------------------------------------
def test_whole_population_at_scale():
    B, P, nf, depth = 16384, 2, 1000, 200.0
    raw = _raw(depth)
    T, O = hc.Tables.from_raw(raw), orc.Tables(raw)
    seeds = np.arange(1, B + 1, dtype=np.int32)
    ens = _irregular_ensemble(T, B, "shared", seeds, nf)
    sp = ens.irregular(0)
    om, k = 2 * np.pi * sp["freqs"], sp["wavenumbers"]
    A = np.sqrt(2 * sp["S"] * sp["widths"])
    pts = _points(B, P)
    t, mwl = 417.25, 0.2
    for wheeler in (False, True):
        got = ens.wave_kinematics(t, pts, mwl=mwl, wheeler=wheeler)
        for b0 in range(0, B, 1024):
            sl = slice(b0, b0 + 1024)
            ph = np.stack([hc.random_phases(int(s), nf) for s in seeds[sl]])
            ref, bars = restate(om, k, A, ph, pts[sl], t, depth, mwl, wheeler)
            _assert_bar([g[sl] for g in got], ref, bars, (wheeler, b0))
        for b in (0, 1, 127, 128, 511, 512, 8191, 8192, 16383):
            i = orc.Instance(O)
            i.set_irregular(seed=int(seeds[b]), nfreq=nf, **SEA)
            ph = hc.random_phases(int(seeds[b]), nf)[None]
            _, bars = restate(om, k, A, ph, pts[b:b + 1], t, depth, mwl, wheeler)
            for p in range(P):
                e, v, a = i.kinematics(pts[b, p], t, wave_stretching=wheeler, mwl=mwl)
                _assert_bar([got[0][b, p], got[1][b, p], got[2][b, p]], [e, v, a],
                            [bars[0][0, p], bars[1][0, p], bars[2][0, p]], ("oracle", b, p, wheeler))


@pytest.mark.parametrize("P", [5, 9])
def test_points_per_thread_variants_at_scale(P):
    """At 16384 instances P = 5 runs two points per thread and P = 9 four (groups of 2 + 2 + 1 / 4 + 4 + 1)."""
    import torch
    B, nf, depth = 16384, 64, 30.0
    T = hc.Tables.from_raw(_raw(depth))
    seeds = 7 + np.arange(B, dtype=np.int32)
    ens = _irregular_ensemble(T, B, "per_instance", seeds, nf)
    pts = _points(B, P)
    got = ens.wave_kinematics(12.5, pts, mwl=-0.1, wheeler=True)
    dev = torch.device("cuda", 0)
    d_pts = torch.from_numpy(pts).to(dev)
    d_out = [torch.full((B, P), np.nan, dtype=torch.float64, device=dev),
             torch.full((B, P, 3), np.nan, dtype=torch.float64, device=dev),
             torch.full((B, P, 3), np.nan, dtype=torch.float64, device=dev)]
    torch.cuda.synchronize()
    ens.wave_kinematics_device(12.5, P, d_pts, *d_out, mwl=-0.1, wheeler=True)
    ens.sync()
    for g, d in zip(got, d_out):
        np.testing.assert_array_equal(g, d.cpu().numpy())
    sl = np.r_[0:300, B - 300:B]
    om, k, A, ph = _components(ens, sl)
    ref, bars = restate(om, k, A, ph, pts[sl], 12.5, depth, -0.1, True)
    _assert_bar([g[sl] for g in got], ref, bars)


# ---------------------------------------------------------------------------------------------
# 3. tie to k_eta
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["shared", "per_instance"])
def test_eta_at_origin_equals_synthesised_sample_bitwise(kind):
    B, nf = 300, 1000
    T = hc.Tables.from_raw(_raw(200.0))
    seeds = 11 + np.arange(B, dtype=np.int32)
    ens = _irregular_ensemble(T, B, kind, seeds, nf)
    eta_t = ens.irregular(0)["eta_t"]
    ks = [int(np.searchsorted(eta_t, SEA["ramp"])) + 3, len(eta_t) // 2, len(eta_t) - 1]
    samples = np.empty((B, len(eta_t)))
    for b in range(B):
        hc._check(_capi.lib.hc_waves_irregular_eta(ens._h, b, None, hc._dp(samples[b])))
    for kk in ks:
        assert eta_t[kk] > SEA["ramp"]
        pts = np.zeros((B, 2, 3))
        pts[:, 1, 2] = -3.0                     # y and z do not enter eta
        for wheeler in (False, True):
            eta, _, _ = ens.wave_kinematics(eta_t[kk], pts, wheeler=wheeler)
            np.testing.assert_array_equal(eta[:, 0], samples[:, kk])
            np.testing.assert_array_equal(eta[:, 1], samples[:, kk])


# ---------------------------------------------------------------------------------------------
# 4. batch and point edges, host and device entry points agree bitwise
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 31, 64, 65, 1000])
def test_batch_and_point_edges(B):
    import torch
    depth = 30.0
    T = hc.Tables.from_raw(_raw(depth))
    seeds = 5 + 3 * np.arange(B, dtype=np.int32)
    ens = _irregular_ensemble(T, B, "per_instance", seeds, 64)
    om, k, A, ph = _components(ens, range(B))
    dev = torch.device("cuda", 0)
    for P in (1, 4, 5, 9):
        pts = _points(B, P)
        for wheeler in (False, True):
            got = ens.wave_kinematics(3.3, pts, mwl=0.1, wheeler=wheeler)
            ref, bars = restate(om, k, A, ph, pts, 3.3, depth, 0.1, wheeler)
            _assert_bar(got, ref, bars, (B, P, wheeler))
            d_pts = torch.from_numpy(pts).to(dev)
            d_eta = torch.full((B, P), np.nan, dtype=torch.float64, device=dev)
            d_acc = torch.full((B, P, 3), np.nan, dtype=torch.float64, device=dev)
            torch.cuda.synchronize()
            ens.wave_kinematics_device(3.3, P, d_pts, d_eta, None, d_acc.data_ptr(), mwl=0.1, wheeler=wheeler)
            ens.sync()
            np.testing.assert_array_equal(d_eta.cpu().numpy(), got[0])
            np.testing.assert_array_equal(d_acc.cpu().numpy(), got[2])


# ---------------------------------------------------------------------------------------------
# 5. stepping is undisturbed
# ---------------------------------------------------------------------------------------------
def test_stepping_undisturbed_by_kinematics_calls():
    import torch
    raw = synth.make_tables(num_bodies=2, rirf_steps=201, rirf_duration=10.0, exc_irf_steps=201, exc_half_window=5.0)
    T = hc.Tables.from_raw(raw)
    B, D, n = 256, 12, 80
    opts = dict(dt_hint=DT, bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=5)
    seeds = np.arange(1, B + 1, dtype=np.int32)
    sea = dict(SEA, duration=(n + 20) * DT, nfreq=64)
    ens = [hc.Ensemble(T, batch=B, **opts) for _ in range(2)]
    for e in ens:
        e.set_waves_irregular(seeds=seeds, **sea)
    dev = torch.device("cuda", 0)
    amp, om = synth.prescribed_motion(D)
    ph = 0.01 * np.arange(B)[:, None]
    pts = _points(B, 3)
    d_pts = torch.from_numpy(pts).to(dev)
    d_eta = torch.empty((B, 3), dtype=torch.float64, device=dev)
    d_vel = torch.empty((B, 3, 3), dtype=torch.float64, device=dev)
    d_pose, d_v = torch.empty((B, D), dtype=torch.float64, device=dev), torch.empty((B, D), dtype=torch.float64, device=dev)
    d_f = [torch.empty((B, D), dtype=torch.float64, device=dev) for _ in range(2)]
    t = 0.0
    for step in range(n):
        d_pose.copy_(torch.from_numpy(amp * np.sin(om * t + ph)))
        d_v.copy_(torch.from_numpy(amp * om * np.cos(om * t + ph)))
        torch.cuda.synchronize()
        F = []
        for j, e in enumerate(ens):
            e.step_device(t, d_pose, d_v, d_f[j])
            if j == 1:
                e.wave_kinematics_device(t + 0.5 * DT, 3, d_pts, d_eta, d_vel, None, wheeler=True)
                if step % 9 == 0:
                    e.wave_kinematics(-7.0 + step, pts)
            e.sync()
            F.append(d_f[j].cpu().numpy())
        np.testing.assert_array_equal(F[0], F[1])
        t += DT
    assert ens[0].lookahead_state() == ens[1].lookahead_state() == {"radiation": 1, "excitation": 1}
    stats = [e.rad_block_stats() for e in ens]
    assert stats[0] == stats[1] and stats[0]["steps_served"] > 0
    for e in ens:
        e.close()


# ---------------------------------------------------------------------------------------------
# 6. zeros and reconfiguration
# ---------------------------------------------------------------------------------------------
def test_zeros_reconfiguration_and_errors():
    depth, B, P = 200.0, 40, 3
    raw = _raw(depth)
    T, O = hc.Tables.from_raw(raw), orc.Tables(raw)
    ens = hc.Ensemble(T, batch=B)
    pts = _points(B, P)

    def zeros():
        for wheeler in (False, True):
            for g in ens.wave_kinematics(5.0, pts, mwl=0.3, wheeler=wheeler):
                assert not np.any(g)

    zeros()                                                   # a fresh ensemble has no waves
    ens.set_waves_irregular(seeds=np.arange(B, dtype=np.int32) + 1, nfreq=80, **SEA)
    assert np.any(ens.wave_kinematics(5.0, pts)[0])
    ens.set_waves_none()
    zeros()
    tt = np.arange(0.0, 40.0, DT)
    ens.set_waves_series(DT, tt - 10.0, np.sin(0.7 * tt))     # imported eta series: no components
    zeros()

    def check(insts, comps, wheeler):
        got = ens.wave_kinematics(61.5, pts, mwl=-0.2, wheeler=wheeler)
        _, bars = restate(*comps, pts, 61.5, depth, -0.2, wheeler)
        ref = [np.empty((B, P)), np.empty((B, P, 3)), np.empty((B, P, 3))]
        for b in range(B):
            for p in range(P):
                e, v, a = insts[b].kinematics(pts[b, p], 61.5, wave_stretching=wheeler, mwl=-0.2)
                ref[0][b, p], ref[1][b, p], ref[2][b, p] = e, v, a
        _assert_bar(got, ref, bars)

    for seed0, wheeler in ((100, True), (None, False), (500, False)):
        if seed0 is None:                                     # irregular -> regular
            amp, om = 0.5 + 0.01 * np.arange(B), 0.4 + 0.05 * np.arange(B)
            phase = 0.1 * np.arange(B)
            ens.set_waves_regular(amp, om, phase)
            insts = []
            for b in range(B):
                i = orc.Instance(O)
                i.set_regular(amp[b], om[b], phase[b])
                insts.append(i)
            comps = (om[:, None], np.array([[ens.regular_coeffs(b)[2]] for b in range(B)]), amp[:, None], phase[:, None])
        else:                                                 # -> irregular with other seeds
            seeds = seed0 + np.arange(B, dtype=np.int32)
            ens.set_waves_irregular(seeds=seeds, nfreq=80, **SEA)
            insts = []
            for b in range(B):
                i = orc.Instance(O)
                i.set_irregular(seed=int(seeds[b]), nfreq=80, share_irf_from=insts[0] if insts else None, **SEA)
                insts.append(i)
            comps = _components(ens, range(B))
        check(insts, comps, wheeler)

    with pytest.raises(hc.HydroError) as ei:
        ens.wave_kinematics(0.0, np.zeros((B, 0, 3)))
    assert ei.value.status == 1
    st = _capi.lib.hc_waves_kinematics_at_time(ens._h, 0.0, 2, None, 0.0, 0, None, None, None)
    assert st == 1
    st = _capi.lib.hc_waves_kinematics_at_time_device(ens._h, 0.0, 2, None, 0.0, 0, None, None, None)
    assert st == 1
    st = _capi.lib.hc_waves_kinematics_at_time(ens._h, 0.0, -1, hc._dp(pts), 0.0, 0, None, None, None)
    assert st == 1
    ens.close()


# ---------------------------------------------------------------------------------------------
# 7. multi-device handle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("waves", ["irregular", "regular"])
def test_multi_device_handle_matches_single_ensemble_bitwise(waves):
    B, P = 1001, 3
    T = hc.Tables.from_raw(_raw(30.0))
    seeds = 2 + np.arange(B, dtype=np.int32)
    hs, tp = _hs_tp(B)
    single = hc.Ensemble(T, batch=B)
    multi = hc.MultiEnsemble(T, B, devices=[0, 0])
    amp, om, ph = 0.3 + 1e-3 * np.arange(B), 0.5 + 2e-3 * np.arange(B), 0.01 * np.arange(B)
    for e in (single, multi):
        if waves == "irregular":
            e.set_waves_irregular(seeds=seeds, Hs_per_instance=hs, Tp_per_instance=tp, nfreq=100, **SEA)
        else:
            e.set_waves_regular(amp, om, ph)
    pts = _points(B, P)
    for wheeler in (False, True):
        a = single.wave_kinematics(333.3, pts, mwl=0.05, wheeler=wheeler)
        b = multi.wave_kinematics(333.3, pts, mwl=0.05, wheeler=wheeler)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
        assert np.any(a[0])
    multi.close()
    single.close()


# ---------------------------------------------------------------------------------------------
# 8. C++ host layer: TestHydroEnsemble::GetWaveKinematics over a hydro.yaml sweep
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sphere_h5(tmp_path_factory):
    f = tmp_path_factory.mktemp("h5") / "sphere.h5"
    h5io.write_bemio(f, common.sphere_raw())
    return str(f)


@pytest.mark.parametrize("wave", ["irregular", "regular"])
def test_host_layer_sweep_kinematics(host_build, sphere_h5, tmp_path, wave):
    y = tmp_path / "sweep.hydro.yaml"
    if wave == "regular":
        y.write_text("hydrodynamics:\n  bodies:\n    - name: body1\n      h5_file: %s\n  waves:\n    type: regular\n"
                     "    height: 0.5\n    period:\n      values: [3.0, 4.4, 6.0]\n" % sphere_h5)
        seeds, periods = 1, [3.0, 4.4, 6.0]
    else:
        y.write_text("hydrodynamics:\n  bodies:\n    - name: body1\n      h5_file: %s\n  waves:\n    type: irregular\n"
                     "    height: 1.5\n    seed: 4\n    period:\n      linspace: { start: 8.0, stop: 12.0, num: 3 }\n"
                     % sphere_h5)
        seeds, periods = 2, [8.0, 10.0, 12.0]
    o = tmp_path / "kin.txt"
    duration, dt, ramp = 20.0, 0.015, 3.0
    out = subprocess.run([os.path.join(host_build, "test_ensemble_kinematics"), str(y), str(o), str(seeds),
                          str(duration)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    words = out.stdout.split()
    B = len(periods) * seeds
    assert int(words[words.index("instances") + 1]) == B
    assert int(words[words.index("device_evaluations") + 1]) == 0       # kinematics are not force evaluations
    O = orc.Tables(common.sphere_raw())
    depth = float(common.sphere_raw()["water_depth"])
    insts = []
    for i in range(B):                       # instance i: period i % P, seed base + i / P (SetupHydroSweepFromYAML)
        inst = orc.Instance(O)
        T_i = periods[i % len(periods)]
        if wave == "regular":
            inst.set_regular(0.5 / 2.0, 2.0 * np.pi / T_i)
        else:
            inst.set_irregular(dt=dt, duration=duration, ramp=ramp, Hs=1.5, Tp=T_i, seed=4 + i // len(periods))
        insts.append(inst)
    rows = np.loadtxt(o)
    assert rows.shape == (3 * B * 4, 12)
    seen = set()
    for r in rows:
        t, i, pos = r[0], int(r[1]), r[2:5]
        inst = insts[i]
        if wave == "regular":
            _, _, k = inst.regular()
            comps = ([2.0 * np.pi / periods[i % len(periods)]], [k], [0.25], [0.0])
        else:
            d = inst.irregular()
            comps = (2 * np.pi * d["freqs"], d["wavenumbers"], np.sqrt(2 * d["S"] * d["widths"]), d["phases"])
        wheeler = wave == "irregular"        # IrregularWaveParams::wave_stretching_ defaults to true
        _, bars = restate(*[np.asarray(c)[None] for c in comps], pos[None, None], t, depth, 0.0, wheeler)
        e, v, a = inst.kinematics(pos, t, wave_stretching=wheeler, mwl=0.0)
        _assert_bar([r[5], r[6:9], r[9:12]], [e, v, a], [bars[0][0, 0], bars[1][0, 0], bars[2][0, 0]], (wave, t, i))
        seen.add((t, i))
    assert len(seen) == 3 * B
