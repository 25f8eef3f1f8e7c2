"""Device-side stepping of the ensemble's bodies (hc_ensemble_simulate / Ensemble.simulate).

- The reference's regression cases run through the device loop, held to the gates of test_oracle_goldens.py.
- The same physics as the host loops: tests/stepper.py driven by hc_step, the chrono_compat lock-step run
  (host/tests/test_device_stepping.cpp), and a numpy restatement of both schemes (quaternions included) driven by
  oracle forces.
- At scale: 16384 RM3-shaped instances past the full history window, on the look-ahead paths.
- Bitwise properties, and the errors the call reports.
"""
import os
import subprocess

import numpy as np
import pytest

import common
import stepper
import hydrochrono_b200 as hc
from hydrochrono_b200 import h5io, synth
from oracle import hc_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "hydrochrono_b200", "host")
G981 = (0.0, 0.0, -9.81)
HEAVE = np.array([0, 0, 1, 0, 0, 0], bool)
RM3_LOCK = np.tile(np.array([0, 0, 1, 0, 1, 0], bool), 2)     # heave + pitch per body (see test_rm3_at_scale)


@pytest.fixture(scope="module")
def sphere():
    raw = common.sphere_raw()
    return hc.Tables.from_raw(raw), orc.Tables(raw)


@pytest.fixture(scope="module")
def rm3():
    raw = synth.rm3_like()
    return hc.Tables.from_raw(raw), orc.Tables(raw)


# ---------------------------------------------------------------------------------------------
# numpy restatement of the chrono_compat stepper (host/src/chrono_compat.cpp), batched over instances
# ---------------------------------------------------------------------------------------------
def _qmul(a, q):
    a0, a1, a2, a3 = np.moveaxis(a, -1, 0)
    q0, q1, q2, q3 = np.moveaxis(q, -1, 0)
    return np.stack([a0 * q0 - a1 * q1 - a2 * q2 - a3 * q3, a0 * q1 + a1 * q0 + a2 * q3 - a3 * q2,
                     a0 * q2 - a1 * q3 + a2 * q0 + a3 * q1, a0 * q3 + a1 * q2 - a2 * q1 + a3 * q0], -1)


def _angle_axis(angle, axis):
    h = 0.5 * angle
    s = np.sin(h)
    return np.concatenate([np.cos(h)[..., None], axis * s[..., None]], -1)


def _rotate_by(q, d):
    a = np.sqrt((d * d).sum(-1))
    safe = np.where(a > 0, a, 1.0)
    p = _qmul(_angle_axis(a, d * (1.0 / safe)[..., None]), q)
    p = p / np.sqrt((p * p).sum(-1))[..., None]
    return np.where((a > 0)[..., None], p, q)


def _cardan(q):
    e0, e1, e2, e3 = np.moveaxis(q, -1, 0)
    r00, r01 = 1 - 2 * (e2 * e2 + e3 * e3), 2 * (e1 * e2 - e0 * e3)
    r02, r12, r22 = 2 * (e1 * e3 + e0 * e2), 2 * (e2 * e3 - e0 * e1), 1 - 2 * (e1 * e1 + e2 * e2)
    return np.stack([np.arctan2(-r12, r22), np.arcsin(np.clip(r02, -1, 1)), np.arctan2(-r01, r00)], -1)


def _quat_from_cardan(ang):
    ex, ey, ez = np.eye(3)
    return _qmul(_qmul(_angle_axis(ang[..., 0], ex), _angle_axis(ang[..., 1], ey)), _angle_axis(ang[..., 2], ez))


def _minv(added_mass, mass, inertia, free):
    D = added_mass.shape[0]
    M = np.diag(np.concatenate([[m] * 3 + list(j) for m, j in zip(mass, inertia)])) + added_mass
    idx = np.where(free)[0]
    Minv = np.zeros((D, D))
    Minv[np.ix_(idx, idx)] = np.linalg.inv(M[np.ix_(idx, idx)])
    return Minv


def np_simulate(force_fn, added_mass, mass, inertia, pose0, n_steps, dt, scheme="euler", free=None, c=None, k=None,
                gvec=G981, vel0=None):
    """force_fn(t, pose [B][D], vel [B][D]) -> hydro force [B][D].  Returns (times, poses [n][B][D], vels)."""
    pose0 = np.array(pose0, dtype=np.float64)
    B, D = pose0.shape
    N = D // 6
    free = np.ones(D, bool) if free is None else np.asarray(free, bool)
    Minv = _minv(added_mass, mass, inertia, free)
    c = np.zeros((B, D)) if c is None else np.broadcast_to(c, (B, D))
    k = np.zeros((B, D)) if k is None else np.broadcast_to(k, (B, D))
    fg = np.zeros(D)
    for b in range(N):
        fg[6 * b:6 * b + 3] = mass[b] * np.asarray(gvec)
    q = _quat_from_cardan(pose0.reshape(B, N, 6)[..., 3:])
    pos = pose0.reshape(B, N, 6)[..., :3].copy()
    pose = np.concatenate([pos, _cardan(q)], -1).reshape(B, D)
    x0 = pose.copy()
    vel = np.zeros((B, D)) if vel0 is None else np.array(vel0, dtype=np.float64)

    def total(t, p, v):
        return force_fn(t, p, v) + fg - c * v - k * (p - x0)

    def assemble(pos, q):
        return np.concatenate([pos, _cardan(q)], -1).reshape(B, D)

    times, poses, vels = np.empty(n_steps), np.empty((n_steps, B, D)), np.empty((n_steps, B, D))
    t = 0.0
    if scheme == "euler":
        for n in range(n_steps):
            acc = total(t, pose, vel) @ Minv.T
            vel = np.where(free, vel + dt * acc, 0.0)
            v3 = vel.reshape(B, N, 6)
            pos = pos + v3[..., :3] * dt
            q = _rotate_by(q, v3[..., 3:] * dt)
            pose = assemble(pos, q)
            t += dt
            times[n], poses[n], vels[n] = t, pose, vel
        return times, poses, vels
    alpha = -0.2
    gamma, beta = 0.5 - alpha, 0.25 * (1.0 - alpha) * (1.0 - alpha)
    h = dt
    F = total(t, pose, vel)
    a = F @ Minv.T
    for n in range(n_steps):
        v3, a3 = vel.reshape(B, N, 6), a.reshape(B, N, 6)
        ppos = pos + v3[..., :3] * h + a3[..., :3] * (0.5 * h * h)
        pq = _rotate_by(q, v3[..., 3:] * h + a3[..., 3:] * (0.5 * h * h))
        pvel = vel + a * h
        t += h
        F1 = total(t, assemble(ppos, pq), pvel)
        a1 = ((1.0 + alpha) * F1 - alpha * F) @ Minv.T
        dx = h * vel + h * h * ((0.5 - beta) * a + beta * a1)
        dv = h * ((1.0 - gamma) * a + gamma * a1)
        dx3 = np.where(free, dx, 0.0).reshape(B, N, 6)
        pos = pos + dx3[..., :3]
        q = _rotate_by(q, dx3[..., 3:])
        vel = np.where(free, vel + dv, 0.0)
        pose = assemble(pos, q)
        F, a = F1, a1
        times[n], poses[n], vels[n] = t, pose, vel
    return times, poses, vels


def _oracle_force(insts, gvec=G981):
    return lambda t, p, v: np.array([i.force(t, p[b], v[b], gvec) for b, i in enumerate(insts)])


def _amplitude(poses, pose0):
    return np.abs(poses - pose0[None]).max()


# ---------------------------------------------------------------------------------------------
# 1. the reference's golden trajectories through the device loop
# ---------------------------------------------------------------------------------------------
def test_sphere_decay_golden(sphere):
    T, _ = sphere
    gold = common.sphere_goldens()["decay_um"] * 1e-6
    ens = hc.Ensemble(T, batch=1, dt_hint=common.SPHERE_DT)
    pose0 = np.zeros((1, 6))
    pose0[0, 2] = -1.0
    t, x, v, e, done = ens.simulate(pose0, gold.size, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]])
    assert done == gold.size
    n1, n2 = common.traj_norms(x[:, 0, 2], gold)
    assert n1 <= 1e-4 and n2 <= 1e-6, (n1, n2)
    assert np.abs(x[:, 0, [0, 1, 3, 4, 5]]).max() < 1e-9


def test_regular_wave_goldens_as_one_ensemble(sphere):
    """All ten regular-wave cases as ten instances: per-instance wave and per-instance PTO damper on heave."""
    T, _ = sphere
    golds = [common.sphere_goldens()["reg%d_um" % (k + 1)] * 1e-6 for k in range(10)]
    n = max(g.size for g in golds)
    ens = hc.Ensemble(T, batch=10, dt_hint=common.SPHERE_DT)
    ens.set_waves_regular(common.TASK10_AMPS, common.TASK10_OMEGAS)
    pose0 = np.zeros((10, 6))
    pose0[:, 2] = -2.0
    c = np.zeros((10, 6))
    c[:, 2] = common.TASK10_DAMPING
    t, x, v, e, done = ens.simulate(pose0, n, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]], free_dof=HEAVE,
                                    pto_damping=c)
    for k, g in enumerate(golds):
        n1, n2 = common.traj_norms(x[:g.size, k, 2], g)
        assert n1 <= 1e-4 and n2 <= 2e-6, (k, n1, n2)
    # absorbed energy = sum c v^2 dt of the heave velocities the force evaluations used (v_0 = 0, then v_1 .. v_{n-1})
    ve = np.concatenate([np.zeros((1, 10)), v[:-1, :, 2]])
    np.testing.assert_allclose(e[:, 2], (c[:, 2] * (ve * ve)).sum(0) * common.SPHERE_DT, rtol=1e-12)
    assert np.all(e[:, [0, 1, 3, 4, 5]] == 0.0)


def test_irregular_golden(sphere):
    T, _ = sphere
    ens = hc.Ensemble(T, batch=1, dt_hint=common.SPHERE_DT)
    ens.set_waves_irregular(dt=common.SPHERE_DT, duration=600.0, ramp=60.0, Hs=2.0, Tp=12.0, nfreq=1000, gamma=1.0, seed=1)
    nsteps = 6700
    gold = common.sphere_goldens()["irreg_um"][:nsteps] * 1e-6
    pose0 = np.zeros((1, 6))
    pose0[0, 2] = -2.0
    t, x, v, e, done = ens.simulate(pose0, nsteps, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]],
                                    free_dof=HEAVE)
    n1, n2 = common.traj_norms(x[:, 0, 2], gold)
    assert n1 <= 1e-4 and n2 <= 2e-4, (n1, n2)


def test_iea_sphere_decay_hht(sphere):
    T, _ = sphere
    g = common.sphere_goldens()
    ens = hc.Ensemble(T, batch=1, dt_hint=0.01)
    pose0 = np.zeros((1, 6))
    pose0[0, 2] = -1.0
    t, x, v, e, done = ens.simulate(pose0, 4000, 0.01, [261800.0], [[999.0, 999.0, 999.0]], scheme="hht",
                                    gvec=(0.0, 0.0, -9.8), free_dof=HEAVE)
    assert common.rms_relative_error(g["iea_decay_z"], np.interp(g["iea_decay_t"], t, x[:, 0, 2])) <= 2e-3
    assert ens.history_len() > 0


# ---------------------------------------------------------------------------------------------
# 2. the same physics as the host loops
# ---------------------------------------------------------------------------------------------
def test_heave_only_matches_host_stepper(sphere):
    """Euler, heave-only regular waves with a PTO damper: the device loop against tests/stepper.py driven by hc_step."""
    T, _ = sphere
    B, n = 3, 900
    amps, oms = common.TASK10_AMPS[2:2 + B], common.TASK10_OMEGAS[2:2 + B]
    ens = hc.Ensemble(T, batch=B, dt_hint=common.SPHERE_DT)
    ens.set_waves_regular(amps, oms)
    pose0 = np.zeros((B, 6))
    pose0[:, 2] = -2.0
    c = np.zeros((B, 6))
    c[:, 2] = common.TASK10_DAMPING[2:2 + B]
    t, x, _, _, _ = ens.simulate(pose0, n, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]], free_dof=HEAVE,
                                 pto_damping=c)
    for b in range(B):
        ref = hc.Ensemble(T, batch=1, dt_hint=common.SPHERE_DT)
        ref.set_waves_regular(amps[b], oms[b])
        tr, xr = stepper.run(lambda tt, p, v: ref.step(tt, p[None], v[None], G981)[0], T.added_mass(), [common.SPHERE_MASS],
                             [[1.0, 1.0, 1.0]], pose0[b], common.SPHERE_DT, n, free=HEAVE, damping=c[b])
        np.testing.assert_array_equal(t, tr)
        assert np.abs(x[:, b] - xr).max() <= 1e-9 * _amplitude(xr, pose0[b]), b
        assert ens.history_len() == ref.history_len()


@pytest.fixture(scope="module")
def host_build():
    subprocess.check_call(["make", "-C", HOST, "-j8"], stdout=subprocess.DEVNULL)
    return os.path.join(HOST, "build")


def test_matches_chrono_compat_lockstep(host_build, tmp_path):
    """host/tests/test_device_stepping.cpp: heave-only spheres (prismatic joint to ground) and the free RM3-shaped pair
    with initial roll / pitch, Euler and HHT, hc_ensemble_simulate against the lock-stepped chrono_compat systems."""
    sph, r3 = tmp_path / "sphere.h5", tmp_path / "rm3_like.h5"
    h5io.write_bemio(sph, common.sphere_raw())
    h5io.write_bemio(r3, synth.rm3_like())
    out = subprocess.run([os.path.join(host_build, "test_device_stepping"), str(sph), str(r3), "400"], capture_output=True,
                         text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = [ln.split() for ln in out.stdout.splitlines() if ln.startswith("case ")]
    assert sorted((w[1], w[3]) for w in lines) == [("rm3", "euler"), ("rm3", "hht"), ("sphere", "euler"), ("sphere", "hht")]
    for w in lines:
        steps, diff, amp = int(w[5]), float(w[7]), float(w[9])
        assert steps == 400 and amp > 1e-3, w
        assert diff <= 1e-9 * amp, w


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_matches_numpy_restatement_with_rotations(rm3, scheme):
    """Free RM3-shaped pair with initial roll / pitch / yaw, regular waves, PTO damper and spring on every DoF: the
    device loop against the numpy restatement of the scheme driven by oracle forces."""
    T, O = rm3
    B, n, dt = 3, 300, 0.01
    amps, oms = [0.5, 1.0, 1.5], [0.6, 0.9, 1.2]
    ens = hc.Ensemble(T, batch=B, dt_hint=dt)
    ens.set_waves_regular(amps, oms)
    insts = []
    for b in range(B):
        i = orc.Instance(O)
        i.set_regular(amps[b], oms[b])
        insts.append(i)
    rng = np.random.Generator(np.random.MT19937(5))
    pose0 = np.zeros((B, 12))
    pose0[:, [2, 8]] = [-0.1, 0.2]
    pose0[:, [3, 4, 5, 9, 10, 11]] = rng.uniform(-0.08, 0.08, (B, 6))
    vel0 = rng.uniform(-0.05, 0.05, (B, 12))
    c = rng.uniform(0.0, 1e5, (B, 12))
    k = rng.uniform(0.0, 1e5, (B, 12))
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    t, x, v, e, done = ens.simulate(pose0, n, dt, mass, inertia, vel0=vel0, scheme=scheme, pto_damping=c, pto_stiffness=k)
    tr, xr, vr = np_simulate(_oracle_force(insts), T.added_mass(), mass, inertia, pose0, n, dt, scheme=scheme, c=c, k=k,
                             vel0=vel0)
    np.testing.assert_array_equal(t, tr)
    for b in range(B):
        amp = _amplitude(xr[:, b], xr[0, b])
        assert amp > 1e-3
        assert np.abs(x[:, b] - xr[:, b]).max() <= 1e-8 * amp, b
    assert np.abs(x[:, :, [3, 4, 9, 10]]).max() > 0.01         # the orientation path is exercised


# ---------------------------------------------------------------------------------------------
# 3. at scale and on the fast paths
# ---------------------------------------------------------------------------------------------
def test_rm3_at_scale_window_full(rm3):
    """16384 RM3-shaped instances, irregular waves, snapped brackets, 6150 Euler steps (past the 6000-step history
    window).  The synthetic tables give no restoring force in surge, sway and yaw, so those DoFs are locked: each body
    heaves and pitches.  Eight sampled instances are re-stepped by the numpy restatement with oracle forces; the run
    with both look-aheads switched off agrees with the look-ahead run."""
    T, O = rm3
    B, n, dt, every = 16384, 6150, 0.01, 50
    irr = dict(dt=dt, duration=n * dt + 5.0, ramp=5.0, Hs=2.5, Tp=8.0, nfreq=64, gamma=3.3)
    seeds = np.arange(1, B + 1, dtype=np.int32)
    pose0 = np.zeros((B, 12))
    pose0[:, 2], pose0[:, 8] = -0.05, 0.05
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    c = np.zeros((B, 12))
    c[:, 2] = np.linspace(0.0, 2e5, B)
    runs = {}
    for name, opts in (("on", dict(rad_lookahead=2, exc_lookahead=4)), ("off", dict(rad_lookahead=1, exc_lookahead=1))):
        ens = hc.Ensemble(T, batch=B, dt_hint=dt, bracket_snap=1e-8, **opts)
        ens.set_waves_irregular(seeds=seeds, **irr)
        runs[name] = ens.simulate(pose0, n, dt, mass, inertia, free_dof=RM3_LOCK, pto_damping=c, record_every=every)
        if name == "on":
            assert ens.rad_block_stats()["steps_served"] >= n - 100
            assert 6000 <= ens.history_len() <= 6003
        ens.close()
    t, x, v, e, done = runs["on"]
    assert done == n and np.all(np.isfinite(x)) and np.all(np.isfinite(e))
    amp = np.abs(x - pose0[None]).max(axis=(0, 2))
    assert amp.min() > 1e-3
    xo = runs["off"][1]
    assert np.all(np.abs(xo - x).max(axis=(0, 2)) <= 1e-9 * amp)
    sample = [0, 1, 4095, 4096, 8191, 9000, 16382, 16383]
    insts = []
    for b in sample:
        i = orc.Instance(O)
        i.set_irregular(seed=int(seeds[b]), share_irf_from=insts[0] if insts else None, **irr)
        insts.append(i)
    tr, xr, _ = np_simulate(_oracle_force(insts), T.added_mass(), mass, inertia, pose0[sample], n, dt, free=RM3_LOCK,
                            c=c[sample])
    np.testing.assert_array_equal(t, tr[every - 1::every])
    for j, b in enumerate(sample):
        assert np.abs(x[:, b] - xr[every - 1::every, j]).max() <= 1e-8 * amp[b], b


# ---------------------------------------------------------------------------------------------
# 4. bitwise properties
# ---------------------------------------------------------------------------------------------
RM3_IRR = dict(dt=0.01, duration=12.0, ramp=2.0, Hs=2.5, Tp=8.0, nfreq=64, gamma=3.3)


def _rm3_ens(T, B, seeds, **kw):
    ens = hc.Ensemble(T, batch=B, dt_hint=0.01, **kw)
    ens.set_waves_irregular(seeds=seeds, **RM3_IRR)
    return ens


def _rm3_pose0(B):
    pose0 = np.zeros((B, 12))
    pose0[:, [3, 4, 9, 10]] = [0.03, -0.02, 0.01, 0.04]
    return pose0


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_bitwise_properties(rm3, scheme):
    T, _ = rm3
    B, n = 6, 240
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    seeds = [3, 4, 3, 5, 4, 3]
    pose0 = _rm3_pose0(B)
    kw = dict(scheme=scheme, pto_damping=1e4)
    one = _rm3_ens(T, B, seeds).simulate(pose0, n, 0.01, mass, inertia, **kw)
    t, x, v, e, done = one
    # replicated seeds, same initial state: equal trajectories
    assert np.array_equal(x[:, 0], x[:, 2]) and np.array_equal(x[:, 0], x[:, 5]) and np.array_equal(x[:, 1], x[:, 4])
    assert not np.array_equal(x[:, 0], x[:, 1])
    # record_every 7 = every 7th record of record_every 1
    t7, x7, v7, e7, _ = _rm3_ens(T, B, seeds).simulate(pose0, n, 0.01, mass, inertia, record_every=7, **kw)
    assert np.array_equal(t7, t[6::7]) and np.array_equal(x7, x[6::7]) and np.array_equal(v7, v[6::7])
    assert np.array_equal(e7, e)
    # host variant = device variant (torch buffers)
    import torch
    ens = _rm3_ens(T, B, seeds)
    dev = torch.device("cuda", 0)
    dp, dv = torch.tensor(pose0, device=dev), torch.zeros((B, 12), dtype=torch.float64, device=dev)
    rt = torch.empty(n, dtype=torch.float64, device=dev)
    rp, rv = (torch.empty((n, B, 12), dtype=torch.float64, device=dev) for _ in range(2))
    de = torch.empty((B, 12), dtype=torch.float64, device=dev)
    assert ens.simulate_device(dp, dv, n, 0.01, mass, inertia, d_rec_t=rt, d_rec_pose=rp, d_rec_vel=rv, d_pto_energy=de,
                               **kw) == n
    ens.sync()
    assert np.array_equal(rt.cpu().numpy(), t) and np.array_equal(rp.cpu().numpy(), x) and np.array_equal(rv.cpu().numpy(), v)
    assert np.array_equal(de.cpu().numpy(), e)
    assert np.array_equal(dp.cpu().numpy(), one.final_pose) and np.array_equal(dv.cpu().numpy(), one.final_vel)
    if scheme == "euler":
        # split into two calls = one call (the second starts at the first's end time and state)
        ens = _rm3_ens(T, B, seeds)
        m = 97
        a = ens.simulate(pose0, m, 0.01, mass, inertia, **kw)
        b = ens.simulate(a.final_pose, n - m, 0.01, mass, inertia, vel0=a.final_vel, t0=a[0][-1], **kw)
        assert np.array_equal(np.concatenate([a[0], b[0]]), t)
        assert np.array_equal(np.concatenate([a[1], b[1]]), x) and np.array_equal(np.concatenate([a[2], b[2]]), v)
        # after a run, hc_step at the next time works; the history is that of the host loop
        F = ens.step(b[0][-1], b.final_pose, b.final_vel)
        assert np.all(np.isfinite(F)) and ens.last_recomputed
        ref = _rm3_ens(T, B, seeds)
        tt = 0.0
        for _ in range(n + 1):
            ref.step(tt, pose0, np.zeros((B, 12)))
            tt += 0.01
        assert ens.history_len() == ref.history_len()


def test_multi_ensemble_matches_standalone_shards(rm3):
    T, _ = rm3
    B, n = 7, 150
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    seeds = np.arange(11, 11 + B, dtype=np.int32)
    pose0 = _rm3_pose0(B)
    c = np.linspace(0.0, 1e5, B)[:, None] * np.ones(12)
    me = hc.MultiEnsemble(T, B, devices=[0, 0], dt_hint=0.01)
    me.set_waves_irregular(seeds=seeds, **RM3_IRR)
    t, x, v, e, done = me.simulate(pose0, n, 0.01, mass, inertia, scheme="hht", pto_damping=c, record_every=3)
    assert done == n
    for sh in me.shards():
        f, k = sh["first"], sh["count"]
        s = _rm3_ens(T, k, seeds[f:f + k]).simulate(pose0[f:f + k], n, 0.01, mass, inertia, scheme="hht",
                                                    pto_damping=c[f:f + k], record_every=3)
        assert np.array_equal(s[0], t) and np.array_equal(s[1], x[:, f:f + k]) and np.array_equal(s[2], v[:, f:f + k])
        assert np.array_equal(s[3], e[f:f + k])


# ---------------------------------------------------------------------------------------------
# 5. errors
# ---------------------------------------------------------------------------------------------
def test_eta_window_error_ends_the_run():
    T = hc.Tables.from_raw(synth.rm3_like(exc_irf_steps=201, exc_half_window=5.0))   # eta window ends at t ~ 6 s
    B = 3
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    irr = dict(RM3_IRR, duration=1.0, ramp=0.5)
    pose0 = _rm3_pose0(B)

    def ens():
        e = hc.Ensemble(T, batch=B, dt_hint=0.01)
        e.set_waves_irregular(seeds=[1, 2, 3], **irr)
        return e

    for scheme in ("euler", "hht"):
        r = ens().simulate(pose0, 2000, 0.01, mass, inertia, scheme=scheme, check=False)
        assert r.status == 5 and 100 < r[4] < 2000, (scheme, r[4])
        ok = ens().simulate(pose0, r[4], 0.01, mass, inertia, scheme=scheme)
        assert np.array_equal(r.final_pose, ok.final_pose) and np.array_equal(r.final_vel, ok.final_vel)
        assert np.array_equal(r[1][:r[4]], ok[1]) and np.array_equal(r[3], ok[3])
        with pytest.raises(hc.EtaWindowError):
            ens().simulate(pose0, 2000, 0.01, mass, inertia, scheme=scheme)


def test_invalid_arguments(sphere):
    import ctypes as C
    from hydrochrono_b200 import _capi
    T, _ = sphere
    ens = hc.Ensemble(T, batch=2, dt_hint=0.01)
    pose = np.zeros((2, 6))
    good = dict(mass=[common.SPHERE_MASS], inertia=[[1.0, 1.0, 1.0]])
    for kw in (dict(n_steps=0), dict(record_every=0), dict(dt=0.0), dict(dt=-0.01)):
        args = dict(n_steps=10, dt=0.01, **good)
        args.update(kw)
        with pytest.raises(hc.HydroError) as ei:
            ens.simulate(pose, **args)
        assert ei.value.status == 1, kw
    # singular free-DoF mass matrix: heave mass cancels the heave added mass
    with pytest.raises(hc.HydroError) as ei:
        ens.simulate(pose, 10, 0.01, [-T.added_mass()[2, 2]], [[1.0, 1.0, 1.0]], free_dof=HEAVE)
    assert ei.value.status == 1
    # NULL where a pointer is required
    p, keep = hc._sim_params(6, 2, 10, 0.01, 0.0, "euler", 1, G981, good["mass"], good["inertia"], None, None, None)
    vel = np.zeros((2, 6))
    done = C.c_int()
    for field in ("mass", "inertia"):
        q = _capi.SimParams.from_buffer_copy(p)
        setattr(q, field, None)
        assert hc.lib.hc_ensemble_simulate(ens._h, C.byref(q), hc._dp(pose), hc._dp(vel), None, None, None, None,
                                           C.byref(done)) == 1, field
    assert hc.lib.hc_ensemble_simulate(ens._h, None, hc._dp(pose), hc._dp(vel), None, None, None, None, None) == 1
    assert hc.lib.hc_ensemble_simulate(ens._h, C.byref(p), None, hc._dp(vel), None, None, None, None, None) == 1
    assert hc.lib.hc_ensemble_simulate(ens._h, C.byref(p), hc._dp(pose), None, None, None, None, None, None) == 1
    assert hc.lib.hc_ensemble_simulate_device(ens._h, C.byref(p), None, None, None, None, None, None, None) == 1
    # nothing ran: the ensemble is untouched
    assert ens.history_len() == 0
