"""Device-side stepping with prismatic joints and translational spring-dampers (Ensemble.simulate with prismatic= /
tsda=, k_body_step_linked): the RM3 float on its moving spar with a PTO, and the sphere on a joint to ground.

- The chrono_compat lock-step run (host/tests/test_device_links.cpp) and a numpy restatement of SolveAccelerations /
  ProjectOntoJoints / the spring-damper force, driven by oracle forces.
- At scale: a 16384-instance RM3 power matrix past the full history window, on the look-ahead paths.
- Cross-checks against the unlinked device path, bitwise properties, the absorbed energy, and the errors of the call.
"""
import os
import subprocess

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import h5io, synth
from oracle import hc_oracle as orc
from test_gpu_device_stepping import G981, HEAVE, _cardan, _oracle_force, _qmul, _quat_from_cardan, _rotate_by

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "hydrochrono_b200", "host")
MASS, INERTIA = synth.RM3_MASSES, synth.RM3_INERTIAS
FLOAT_Z, SPAR_Z = -0.72, -21.29
JOINT = hc.Prismatic(0, 1, (0.0, 0.0, 1.0))                   # float (body 0) slides on the spar (body 1)


def _pto(damping=0.0, stiffness=0.0, rest_length=None):
    return hc.TSDA(0, 1, (0.0, 0.0, FLOAT_Z), (0.0, 0.0, SPAR_Z), damping=damping, stiffness=stiffness,
                   rest_length=rest_length)


@pytest.fixture(scope="module")
def sphere():
    return hc.Tables.from_raw(common.sphere_raw())


@pytest.fixture(scope="module")
def rm3():
    raw = synth.rm3_like()
    return hc.Tables.from_raw(raw), orc.Tables(raw)


# ---------------------------------------------------------------------------------------------
# numpy restatement of the chrono_compat stepper with joints and spring-dampers, batched over instances
# ---------------------------------------------------------------------------------------------
_CONJ = np.array([1.0, -1.0, -1.0, -1.0])


def _rot(q, v):                                   # ChQuaterniond::Rotate
    u = q[..., 1:]
    t = 2.0 * np.cross(u, v)
    return v + q[..., :1] * t + np.cross(u, t)


def _rot_back(q, v):
    return _rot(q * _CONJ, v)


def _normalize(q):
    return q / np.sqrt((q * q).sum(-1))[..., None]


def _assembly(pose0, prismatic, tsda):
    """Per-instance assembly data (ChLinkLockPrismatic / ChLinkTSDA::Initialize) at the initial pose."""
    B, D = pose0.shape
    p6 = pose0.reshape(B, D // 6, 6)
    pos, q = p6[..., :3], _quat_from_cardan(p6[..., 3:])

    def body(i):
        if i < 0:
            return np.zeros((B, 3)), np.tile([1.0, 0.0, 0.0, 0.0], (B, 1))
        return pos[:, i], q[:, i]

    joints = []
    for j in prismatic:
        xP, qP = body(j.parent)
        ax = np.asarray(j.axis) / np.linalg.norm(j.axis)
        joints.append(dict(child=j.child, parent=j.parent, off=_rot_back(qP, pos[:, j.child] - xP),
                           rel=_qmul(qP * _CONJ, q[:, j.child]), ax=_rot_back(qP, np.broadcast_to(ax, (B, 3)))))
    springs = []
    for s in tsda:
        (x1, q1), (x2, q2) = body(s.body1), body(s.body2)
        p1, p2 = np.asarray(s.point1), np.asarray(s.point2)
        rest = np.full(B, np.linalg.norm(p1 - p2) if s.rest_length is None else s.rest_length)
        springs.append(dict(b1=s.body1, b2=s.body2, loc1=_rot_back(q1, p1 - x1), loc2=_rot_back(q2, p2 - x2), rest=rest,
                            c=np.broadcast_to(np.asarray(s.damping, float), (B,)),
                            k=np.broadcast_to(np.asarray(s.stiffness, float), (B,))))
    return joints, springs


def _residual(poses, joints):
    """Largest joint residual (transverse offset in the parent frame, relative rotation) of poses [..., B, D]."""
    shp = poses.shape
    p6 = poses.reshape(shp[:-1] + (shp[-1] // 6, 6))
    pos, q = p6[..., :3], _quat_from_cardan(p6[..., 3:])
    r = 0.0
    for j in joints:
        c, p = j["child"], j["parent"]
        xP = pos[..., p, :] if p >= 0 else 0.0
        qP = q[..., p, :] if p >= 0 else np.array([1.0, 0.0, 0.0, 0.0])
        d = _rot_back(qP, pos[..., c, :] - xP) - j["off"]
        tr = d - j["ax"] * (d * j["ax"]).sum(-1)[..., None]
        rel = _qmul(qP * _CONJ, q[..., c, :])
        rel = rel * np.sign((rel * j["rel"]).sum(-1))[..., None]
        r = max(r, np.abs(tr).max(), np.abs(rel - j["rel"]).max())
    return r


def np_simulate_links(force_fn, added_mass, pose0, n_steps, dt, scheme="euler", free=None, vel0=None, prismatic=(),
                      tsda=(), mass=MASS, inertia=INERTIA, gvec=G981):
    """Returns (times, poses [n][B][D], vels, tsda energy [B][n_tsda])."""
    pose0 = np.array(pose0, dtype=np.float64)
    B, D = pose0.shape
    N = D // 6
    free = np.ones(D, bool) if free is None else np.asarray(free, bool)
    M = np.diag(np.concatenate([[m] * 3 + list(j) for m, j in zip(mass, inertia)])) + added_mass
    fg = np.zeros(D)
    for b in range(N):
        fg[6 * b:6 * b + 3] = mass[b] * np.asarray(gvec)
    joints, springs = _assembly(pose0, prismatic, tsda)
    child_of = {j["child"]: j for j in joints}
    cols = [(n, k) for n in range(N) if n not in child_of for k in range(6) if free[6 * n + k]]
    cols += [(n, 6) for n in range(N) if n in child_of]
    p6 = pose0.reshape(B, N, 6)
    pos, q = p6[..., :3].copy(), _quat_from_cardan(p6[..., 3:])
    vel = np.zeros((B, D)) if vel0 is None else np.array(vel0, dtype=np.float64)
    v, w = vel.reshape(B, N, 6)[..., :3].copy(), vel.reshape(B, N, 6)[..., 3:].copy()
    energy = np.zeros((B, len(springs)))

    def body(i, pos, q, v, w):
        if i < 0:
            z = np.zeros((B, 3))
            return z, np.tile([1.0, 0.0, 0.0, 0.0], (B, 1)), z, z
        return pos[:, i], q[:, i], v[:, i], w[:, i]

    def flat(a, b):
        return np.concatenate([a, b], -1).reshape(B, D)

    def force(t, pos, q, v, w, count):            # Assemble
        F = force_fn(t, flat(pos, _cardan(q)), flat(v, w)) + fg
        F = F.reshape(B, N, 6)
        for k, s in enumerate(springs):
            x1, q1, v1, w1 = body(s["b1"], pos, q, v, w)
            x2, q2, v2, w2 = body(s["b2"], pos, q, v, w)
            s1, s2 = _rot(q1, s["loc1"]), _rot(q2, s["loc2"])
            d = (x1 + s1) - (x2 + s2)
            ln = np.sqrt((d * d).sum(-1))
            u = d / ln[:, None]
            ld = ((v1 + np.cross(w1, s1) - v2 - np.cross(w2, s2)) * u).sum(-1)
            f = -(s["k"] * (ln - s["rest"]) + s["c"] * ld)
            if count:
                energy[:, k] += s["c"] * ld * ld * dt
            for i, sv, sign in ((s["b1"], s1, 1.0), (s["b2"], s2, -1.0)):
                if i >= 0:
                    fv = u * (sign * f)[:, None]
                    F[:, i, :3] += fv
                    F[:, i, 3:] += np.cross(sv, fv)
        return F.reshape(B, D)

    def accel(rhs, pos, q, v, w):                 # SolveAccelerations
        T, bias = np.zeros((B, D, len(cols))), np.zeros((B, D))
        nax, rho = {}, {}
        for c, j in child_of.items():
            xP, qP, vP, wP = body(j["parent"], pos, q, v, w)
            nax[c] = _rot(qP, j["ax"])
            if j["parent"] >= 0:
                rho[c] = pos[:, c] - xP
                sd = (nax[c] * (v[:, c] - vP - np.cross(wP, rho[c]))).sum(-1)
                bias[:, 6 * c:6 * c + 3] = np.cross(wP, np.cross(wP, rho[c])) + 2.0 * sd[:, None] * np.cross(wP, nax[c])
        for ci, (n, k) in enumerate(cols):
            if k == 6:
                T[:, 6 * n:6 * n + 3, ci] = nax[n]
                continue
            T[:, 6 * n + k, ci] = 1.0
            for c, j in child_of.items():
                if j["parent"] != n:
                    continue
                T[:, 6 * c + k, ci] = 1.0
                if k >= 3:
                    x, y, z = rho[c][:, 0], rho[c][:, 1], rho[c][:, 2]
                    sk = np.stack([np.stack([0 * x, z, -y], -1), np.stack([-z, 0 * x, x], -1),
                                   np.stack([y, -x, 0 * x], -1)], -2)
                    T[:, 6 * c:6 * c + 3, ci] = sk[:, :, k - 3]
        r = rhs - bias @ M.T
        A = np.einsum("bic,ij,bjd->bcd", T, M, T)
        qdd = np.linalg.solve(A, np.einsum("bic,bi->bc", T, r)[..., None])[..., 0]
        return bias + np.einsum("bic,bc->bi", T, qdd)

    def project(pos, q, v, w):                    # ProjectOntoJoints
        for c, j in child_of.items():
            xP, qP, vP, wP = body(j["parent"], pos, q, v, w)
            nax = _rot(qP, j["ax"])
            rho_b = _rot_back(qP, pos[:, c] - xP)
            s = ((rho_b - j["off"]) * j["ax"]).sum(-1)
            rho = _rot(qP, j["off"] + j["ax"] * s[:, None])
            sd = (nax * (v[:, c] - vP - np.cross(wP, rho))).sum(-1)
            q[:, c] = _normalize(_qmul(qP, j["rel"]))
            pos[:, c] = xP + rho
            w[:, c] = wP
            v[:, c] = vP + np.cross(wP, rho) + nax * sd[:, None]

    fr = free.reshape(N, 6)
    times, poses, vels = np.empty(n_steps), np.empty((n_steps, B, D)), np.empty((n_steps, B, D))
    t = 0.0
    if scheme == "euler":
        for n in range(n_steps):
            a = accel(force(t, pos, q, v, w, True), pos, q, v, w).reshape(B, N, 6)
            v = np.where(fr[:, :3], v + dt * a[..., :3], 0.0)
            w = np.where(fr[:, 3:], w + dt * a[..., 3:], 0.0)
            pos = pos + v * dt
            q = _rotate_by(q, w * dt)
            project(pos, q, v, w)
            t += dt
            times[n], poses[n], vels[n] = t, flat(pos, _cardan(q)), flat(v, w)
        return times, poses, vels, energy
    alpha = -0.2
    gamma, beta = 0.5 - alpha, 0.25 * (1.0 - alpha) * (1.0 - alpha)
    h = dt
    F = force(t, pos, q, v, w, False)
    a = accel(F, pos, q, v, w).reshape(B, N, 6)
    for n in range(n_steps):
        pp, pq = pos + v * h + a[..., :3] * (0.5 * h * h), _rotate_by(q, w * h + a[..., 3:] * (0.5 * h * h))
        pv, pw = v + a[..., :3] * h, w + a[..., 3:] * h
        project(pp, pq, pv, pw)
        t += h
        F1 = force(t, pp, pq, pv, pw, True)
        a1 = accel((1.0 + alpha) * F1 - alpha * F, pp, pq, pv, pw).reshape(B, N, 6)
        dx = h * flat(v, w).reshape(B, N, 6) + h * h * ((0.5 - beta) * a + beta * a1)
        dv = h * ((1.0 - gamma) * a + gamma * a1)
        dx = np.where(fr, dx, 0.0)
        pos = pos + dx[..., :3]
        q = _rotate_by(q, dx[..., 3:])
        v = np.where(fr[:, :3], v + dv[..., :3], 0.0)
        w = np.where(fr[:, 3:], w + dv[..., 3:], 0.0)
        project(pos, q, v, w)
        F, a = F1, a1
        times[n], poses[n], vels[n] = t, flat(pos, _cardan(q)), flat(v, w)
    return times, poses, vels, energy


def _amplitude(poses, pose0):
    return np.abs(poses - pose0[None]).max()


def _rm3_pose0(B, rng):
    pose0 = np.zeros((B, 12))
    pose0[:, 2], pose0[:, 8] = FLOAT_Z, SPAR_Z
    pose0[:, [3, 4, 5]] = rng.uniform(-0.05, 0.05, (B, 3))
    pose0[:, [9, 10, 11]] = rng.uniform(-0.04, 0.04, (B, 3))
    return pose0


def _rm3_vel0(B, rng):
    vel0 = np.zeros((B, 12))
    vel0[:, 6:12] = rng.uniform(-0.02, 0.02, (B, 6))
    return vel0


# ---------------------------------------------------------------------------------------------
# 1. the chrono_compat lock-step run and the numpy restatement
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_build():
    subprocess.check_call(["make", "-C", HOST, "-j8"], stdout=subprocess.DEVNULL)
    return os.path.join(HOST, "build")


def test_matches_chrono_compat_lockstep(host_build, tmp_path):
    """host/tests/test_device_links.cpp: the RM3 float on its all-free spar with a damper PTO (and with a spring PTO),
    the sphere on a joint and a damper to ground; Euler and HHT against the lock-stepped chrono_compat systems."""
    sph, r3 = tmp_path / "sphere.h5", tmp_path / "rm3_like.h5"
    h5io.write_bemio(sph, common.sphere_raw())
    h5io.write_bemio(r3, synth.rm3_like())
    out = subprocess.run([os.path.join(host_build, "test_device_links"), str(sph), str(r3), "400"], capture_output=True,
                         text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = [ln.split() for ln in out.stdout.splitlines() if ln.startswith("case ")]
    assert sorted((w[1], w[3]) for w in lines) == [(c, s) for c in ("rm3", "rm3_spring", "sphere") for s in ("euler", "hht")]
    for w in lines:
        steps, diff, amp, res = int(w[5]), float(w[7]), float(w[9]), float(w[11])
        assert steps == 400 and amp > 1e-3, w
        assert diff <= 1e-9 * amp, w
        assert res <= 1e-12, w


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_matches_numpy_restatement(rm3, scheme):
    """RM3 pair with rotations: float on a prismatic joint to the all-free spar, spring-damper PTO with per-instance
    damping, regular waves; the device loop against the numpy restatement driven by oracle forces."""
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
    rng = np.random.Generator(np.random.MT19937(7))
    pose0, vel0 = _rm3_pose0(B, rng), _rm3_vel0(B, rng)
    pto = _pto(damping=[0.0, 1e6, 3e6], stiffness=2e5, rest_length=20.0)
    r = ens.simulate(pose0, n, dt, MASS, INERTIA, vel0=vel0, scheme=scheme, prismatic=[JOINT], tsda=[pto])
    t, x = r[0], r[1]
    tr, xr, _, er = np_simulate_links(_oracle_force(insts), T.added_mass(), pose0, n, dt, scheme=scheme, vel0=vel0,
                                      prismatic=[JOINT], tsda=[pto])
    np.testing.assert_array_equal(t, tr)
    for b in range(B):
        amp = _amplitude(xr[:, b], xr[0, b])
        assert amp > 1e-3
        assert np.abs(x[:, b] - xr[:, b]).max() <= 1e-8 * amp, b
    np.testing.assert_allclose(r.tsda_energy, er, rtol=1e-7, atol=1e-12 * er.max())
    # the float's surge and roll move through the spar's rotation (rho x w), not on their own
    assert np.abs(x[:, :, 0] - pose0[None, :, 0]).max() > 1e-3
    assert np.abs(x[:, :, 3] - x[:1, :, 3]).max() > 1e-3
    joints, _ = _assembly(pose0, [JOINT], [])
    assert _residual(x, joints) <= 1e-12


# ---------------------------------------------------------------------------------------------
# 2. at scale: the RM3 power matrix
# ---------------------------------------------------------------------------------------------
SPAR_FREE = np.array([1, 1, 1, 1, 1, 1, 0, 0, 1, 1, 1, 0], bool)     # float all free (jointed); spar heave, roll, pitch


def test_rm3_power_matrix_at_scale(rm3):
    """16384 RM3 instances = 128 PTO dampings x 128 sea-state seeds, irregular waves, snapped brackets, 6150 Euler
    steps (past the 6000-step history window).  Joint residual of every record, look-ahead on against off, eight sampled
    instances against the numpy restatement with oracle forces, and the absorbed energy."""
    T, O = rm3
    B, n, dt, every = 16384, 6150, 0.01, 50
    irr = dict(dt=dt, duration=n * dt + 5.0, ramp=5.0, Hs=2.5, Tp=8.0, nfreq=64, gamma=3.3)
    damp = np.repeat(np.linspace(0.0, 4e6, 128), 128)
    seeds = np.tile(np.arange(1, 129, dtype=np.int32), 128)
    pose0 = np.zeros((B, 12))
    pose0[:, 2], pose0[:, 8] = FLOAT_Z - 0.05, SPAR_Z + 0.05
    pto = _pto(damping=damp, rest_length=None)
    kw = dict(free_dof=SPAR_FREE, prismatic=[JOINT], tsda=[pto], record_every=every)
    runs = {}
    for name, opts in (("on", dict(rad_lookahead=2, exc_lookahead=4)), ("off", dict(rad_lookahead=1, exc_lookahead=1))):
        ens = hc.Ensemble(T, batch=B, dt_hint=dt, bracket_snap=1e-8, **opts)
        ens.set_waves_irregular(seeds=seeds, **irr)
        runs[name] = ens.simulate(pose0, n, dt, MASS, INERTIA, **kw)
        if name == "on":
            assert ens.rad_block_stats()["steps_served"] >= n - 100
            assert 6000 <= ens.history_len() <= 6003
        ens.close()
    r = runs["on"]
    t, x, done = r[0], r[1], r[4]
    assert done == n and np.all(np.isfinite(x))
    amp = np.abs(x - pose0[None]).max(axis=(0, 2))
    assert amp.min() > 1e-3
    assert np.all(np.abs(runs["off"][1] - x).max(axis=(0, 2)) <= 1e-9 * amp)
    joints, _ = _assembly(pose0[:1], [JOINT], [])
    for k in range(0, x.shape[0], 8):
        assert _residual(x[k:k + 8], joints) <= 1e-10, k
    e = r.tsda_energy[:, 0]
    assert np.all(np.isfinite(e)) and np.all(e >= 0.0)
    assert np.all(e[damp == 0.0] == 0.0) and np.all(e[damp > 0.0] > 0.0)
    sample = [0, 1, 4095, 4096, 8191, 9000, 16382, 16383]
    insts = []
    for b in sample:
        i = orc.Instance(O)
        i.set_irregular(seed=int(seeds[b]), share_irf_from=insts[0] if insts else None, **irr)
        insts.append(i)
    tr, xr, _, er = np_simulate_links(_oracle_force(insts), T.added_mass(), pose0[sample], n, dt, free=SPAR_FREE,
                                      prismatic=[JOINT], tsda=[_pto(damping=damp[sample])])
    np.testing.assert_array_equal(t, tr[every - 1::every])
    for j, b in enumerate(sample):
        assert np.abs(x[:, b] - xr[every - 1::every, j]).max() <= 1e-8 * amp[b], b
    np.testing.assert_allclose(e[sample], er[:, 0], rtol=1e-6, atol=1e-9 * er.max())


# ---------------------------------------------------------------------------------------------
# 3. cross-checks against the unlinked device path
# ---------------------------------------------------------------------------------------------
def _sphere_run(T, B=3, n=600, **kw):
    ens = hc.Ensemble(T, batch=B, dt_hint=common.SPHERE_DT)
    ens.set_waves_regular(common.TASK10_AMPS[:B], common.TASK10_OMEGAS[:B])
    pose0 = np.zeros((B, 6))
    pose0[:, 2] = -2.0
    return ens.simulate(pose0, n, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]], **kw)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_joint_to_ground_equals_heave_only(sphere, scheme):
    a = _sphere_run(sphere, scheme=scheme, prismatic=[hc.Prismatic(0, -1, (0.0, 0.0, 1.0))])
    b = _sphere_run(sphere, scheme=scheme, free_dof=HEAVE)
    assert _rel(a[1][..., 2], b[1][..., 2]) <= 1e-12 and _rel(a[2], b[2]) <= 1e-12
    assert np.abs(a[1] - b[1]).max() <= 1e-12 * np.abs(b[1]).max()


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_spring_damper_to_ground_equals_heave_damper(sphere, scheme):
    c = np.array([0.0, 2e5, 4e5])
    a = _sphere_run(sphere, scheme=scheme, free_dof=HEAVE,
                    tsda=[hc.TSDA(0, -1, (0.0, 0.0, -2.0), (0.0, 0.0, -5.0), damping=c)])
    pc = np.zeros((3, 6))
    pc[:, 2] = c
    b = _sphere_run(sphere, scheme=scheme, free_dof=HEAVE, pto_damping=pc)
    assert _rel(a[1], b[1]) <= 1e-12 and _rel(a[2], b[2]) <= 1e-12
    assert _rel(a.tsda_energy[:, 0], b[3][:, 2]) <= 1e-12
    assert a.tsda_energy[0, 0] == 0.0 and np.all(a[3] == 0.0)


def test_empty_links_equal_no_links(rm3):
    import ctypes as C
    from hydrochrono_b200 import _capi
    T, _ = rm3
    B, n = 4, 120
    rng = np.random.Generator(np.random.MT19937(3))
    pose0, vel0 = _rm3_pose0(B, rng), _rm3_vel0(B, rng)
    out = []
    for empty in (False, True):
        ens = hc.Ensemble(T, batch=B, dt_hint=0.01)
        ens.set_waves_regular([0.5, 1.0, 1.5, 2.0], [0.6, 0.8, 1.0, 1.2])
        p, keep = hc._sim_params(12, B, n, 0.01, 0.0, "hht", 1, G981, MASS, INERTIA, None, 1e4, None)
        if empty:
            L = _capi.SimLinks()
            keep["links"] = L
            p.links = C.pointer(L)
        out.append(hc._simulate_host(hc.lib.hc_ensemble_simulate, ens._h, B, 12, pose0, vel0, n, 1, True, True, p, keep))
    (s0, r0), (s1, r1) = out
    assert s0 == s1 == 0
    for a, b in zip(r0[:4], r1[:4]):
        assert np.array_equal(a, b)
    assert np.array_equal(r0.final_pose, r1.final_pose) and np.array_equal(r0.final_vel, r1.final_vel)


# ---------------------------------------------------------------------------------------------
# 4. bitwise properties
# ---------------------------------------------------------------------------------------------
RM3_IRR = dict(dt=0.01, duration=12.0, ramp=2.0, Hs=2.5, Tp=8.0, nfreq=64, gamma=3.3)


def _rm3_ens(T, B, seeds, **kw):
    ens = hc.Ensemble(T, batch=B, dt_hint=0.01, **kw)
    ens.set_waves_irregular(seeds=seeds, **RM3_IRR)
    return ens


@pytest.mark.parametrize("scheme", ["euler", "hht"])
def test_bitwise_properties(rm3, scheme):
    T, _ = rm3
    B, n = 5, 240
    seeds = [3, 4, 3, 5, 4]
    rng = np.random.Generator(np.random.MT19937(11))
    pose0, vel0 = _rm3_pose0(B, rng), _rm3_vel0(B, rng)
    pose0[2], vel0[2] = pose0[0], vel0[0]
    links = dict(prismatic=[JOINT], tsda=[_pto(damping=np.linspace(0, 2e6, B), stiffness=1e5)])
    kw = dict(scheme=scheme, vel0=vel0, **links)
    one = _rm3_ens(T, B, seeds).simulate(pose0, n, 0.01, MASS, INERTIA, **kw)
    t, x, v = one[0], one[1], one[2]
    assert not np.array_equal(x[:, 0], x[:, 1])
    # reset, then a run = a fresh ensemble (after a run with other links and another initial state)
    ens = _rm3_ens(T, B, seeds)
    ens.simulate(pose0 + 0.01, 50, 0.01, MASS, INERTIA, scheme=scheme, prismatic=[JOINT], tsda=[_pto(damping=1e5)])
    ens.reset()
    again = ens.simulate(pose0, n, 0.01, MASS, INERTIA, **kw)
    for a, b in zip(one[:4], again[:4]):
        assert np.array_equal(a, b)
    assert np.array_equal(one.tsda_energy, again.tsda_energy)
    # host variant = device variant (torch buffers)
    import torch
    ens = _rm3_ens(T, B, seeds)
    dev = torch.device("cuda", 0)
    dp, dv = torch.tensor(pose0, device=dev), torch.tensor(vel0, device=dev)
    rt = torch.empty(n, dtype=torch.float64, device=dev)
    rp, rv = (torch.empty((n, B, 12), dtype=torch.float64, device=dev) for _ in range(2))
    de = torch.empty((B, 1), dtype=torch.float64, device=dev)
    assert ens.simulate_device(dp, dv, n, 0.01, MASS, INERTIA, scheme=scheme, d_rec_t=rt, d_rec_pose=rp, d_rec_vel=rv,
                               d_tsda_energy=de, **links) == n
    ens.sync()
    assert np.array_equal(rt.cpu().numpy(), t) and np.array_equal(rp.cpu().numpy(), x) and np.array_equal(rv.cpu().numpy(), v)
    assert np.array_equal(de.cpu().numpy(), one.tsda_energy)
    assert np.array_equal(dp.cpu().numpy(), one.final_pose) and np.array_equal(dv.cpu().numpy(), one.final_vel)
    if scheme == "euler":
        # split into two calls = one call (the second continues from the first's end state: assembly data kept)
        ens = _rm3_ens(T, B, seeds)
        m = 97
        a = ens.simulate(pose0, m, 0.01, MASS, INERTIA, **kw)
        b = ens.simulate(a.final_pose, n - m, 0.01, MASS, INERTIA, scheme=scheme, vel0=a.final_vel, t0=a[0][-1], **links)
        assert np.array_equal(np.concatenate([a[0], b[0]]), t)
        assert np.array_equal(np.concatenate([a[1], b[1]]), x) and np.array_equal(np.concatenate([a[2], b[2]]), v)
        assert np.array_equal(a.tsda_energy + b.tsda_energy, one.tsda_energy) or \
            np.allclose(a.tsda_energy + b.tsda_energy, one.tsda_energy, rtol=1e-14)


def test_multi_ensemble_matches_standalone_shards(rm3):
    T, _ = rm3
    B, n = 7, 150
    seeds = np.arange(11, 11 + B, dtype=np.int32)
    rng = np.random.Generator(np.random.MT19937(13))
    pose0 = _rm3_pose0(B, rng)
    damp, stiff = np.linspace(0.0, 2e6, B), np.linspace(1e5, 3e5, B)
    me = hc.MultiEnsemble(T, B, devices=[0, 0], dt_hint=0.01)
    me.set_waves_irregular(seeds=seeds, **RM3_IRR)
    r = me.simulate(pose0, n, 0.01, MASS, INERTIA, scheme="hht", prismatic=[JOINT],
                    tsda=[_pto(damping=damp, stiffness=stiff)], record_every=3)
    assert r[4] == n
    for sh in me.shards():
        f, k = sh["first"], sh["count"]
        s = _rm3_ens(T, k, seeds[f:f + k]).simulate(pose0[f:f + k], n, 0.01, MASS, INERTIA, scheme="hht", prismatic=[JOINT],
                                                    tsda=[_pto(damping=damp[f:f + k], stiffness=stiff[f:f + k])],
                                                    record_every=3)
        assert np.array_equal(s[0], r[0]) and np.array_equal(s[1], r[1][:, f:f + k]) and np.array_equal(s[2], r[2][:, f:f + k])
        assert np.array_equal(s.tsda_energy, r.tsda_energy[f:f + k])


# ---------------------------------------------------------------------------------------------
# 5. the absorbed energy, and errors
# ---------------------------------------------------------------------------------------------
def test_energy_equals_recorded_damping_work(rm3):
    """Euler: tsda_energy = sum c ldot^2 dt, ldot recomputed in numpy from the recorded states (each step's force is
    evaluated at the previous step's state)."""
    T, _ = rm3
    B, n, dt = 4, 400, 0.01
    ens = hc.Ensemble(T, batch=B, dt_hint=dt)
    ens.set_waves_regular([0.5, 1.0, 1.5, 2.0], [0.6, 0.8, 1.0, 1.2])
    rng = np.random.Generator(np.random.MT19937(17))
    pose0, vel0 = _rm3_pose0(B, rng), _rm3_vel0(B, rng)
    c = np.array([0.0, 5e5, 1e6, 2e6])
    pto = _pto(damping=c, stiffness=1e5)
    r = ens.simulate(pose0, n, dt, MASS, INERTIA, vel0=vel0, prismatic=[JOINT], tsda=[pto])
    _, springs = _assembly(pose0, [], [pto])
    s = springs[0]
    P = np.concatenate([pose0[None], r[1][:-1]])
    V = np.concatenate([vel0[None], r[2][:-1]])
    p6, v6 = P.reshape(n, B, 2, 6), V.reshape(n, B, 2, 6)
    q = _quat_from_cardan(p6[..., 3:])
    s1, s2 = _rot(q[:, :, 0], s["loc1"]), _rot(q[:, :, 1], s["loc2"])
    d = (p6[:, :, 0, :3] + s1) - (p6[:, :, 1, :3] + s2)
    u = d / np.linalg.norm(d, axis=-1)[..., None]
    ld = ((v6[:, :, 0, :3] + np.cross(v6[:, :, 0, 3:], s1) - v6[:, :, 1, :3] - np.cross(v6[:, :, 1, 3:], s2)) * u).sum(-1)
    e = (c * ld * ld * dt).sum(0)
    assert r.tsda_energy[0, 0] == 0.0 and np.all(r.tsda_energy[1:, 0] > 0.0)
    np.testing.assert_allclose(r.tsda_energy[:, 0], e, rtol=1e-9)


def test_invalid_arguments(rm3, sphere):
    T, _ = rm3
    ens = hc.Ensemble(T, batch=2, dt_hint=0.01)
    pose = _rm3_pose0(2, np.random.Generator(np.random.MT19937(1)))
    base = dict(n_steps=10, dt=0.01, mass=MASS, inertia=INERTIA)
    P, S = hc.Prismatic, hc.TSDA
    p0 = (0.0, 0.0, 0.0)
    cases = [
        dict(prismatic=[P(2, 1)]),                                   # child out of range
        dict(prismatic=[P(0, 2)]),                                   # parent out of range
        dict(prismatic=[P(0, -2)]),
        dict(prismatic=[P(0, 0)]),                                   # child == parent
        dict(prismatic=[P(0, 1), P(0, -1)]),                         # a second joint on one child
        dict(prismatic=[P(0, 1), P(1, -1)]),                         # chain
        dict(prismatic=[P(0, 1, (0.0, 0.0, 0.0))]),                  # zero axis
        dict(tsda=[S(0, 0, p0, p0)]),                                # body1 == body2
        dict(tsda=[S(-1, -1, p0, p0)]),                              # ground to ground
        dict(tsda=[S(2, 0, p0, p0)]),                                # index out of range
        dict(tsda=[S(0, -2, p0, p0)]),
        dict(tsda=[S(0, 1, p0, p0)] * 17),                           # more than HC_SIM_MAX_TSDA
        dict(prismatic=[P(0, 1)], free_dof=np.r_[np.ones(11), 0]),   # fine: the spar's yaw locked
        dict(prismatic=[P(0, 1)], free_dof=np.r_[0, np.ones(11)]),   # a jointed child with a locked DoF
        dict(prismatic=[P(0, 1)], mass=[-T.added_mass()[2, 2], MASS[1]]),   # mass matrix not positive definite
    ]
    for i, kw in enumerate(cases):
        args = dict(base)
        args.update(kw)
        if i == 12:
            ens.simulate(pose, **args)
            ens.reset()
            continue
        with pytest.raises(hc.HydroError) as ei:
            ens.simulate(pose, **args)
        assert ei.value.status == 1, (i, kw)
    hl = ens.history_len()
    ens2 = hc.Ensemble(T, batch=2, dt_hint=0.01)
    with pytest.raises(hc.HydroError):
        ens2.simulate(pose, prismatic=[P(0, 0)], **base)
    assert ens2.history_len() == 0 and hl >= 0
