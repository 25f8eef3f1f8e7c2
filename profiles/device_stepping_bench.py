"""Device-side stepping benchmark: hc_ensemble_simulate against hc_step plus a vectorised numpy Euler loop.

1. RM3-shaped tables (bench.py's workload: 16384 instances, dt = 0.01, irregular waves, snapped brackets, both
   look-aheads), linearised Euler.  The synthetic tables have no restoring force in surge, sway and yaw, so those DoFs
   are locked (heave + pitch per body).  The history window is filled first (6050 untimed steps); then K steps through
   Ensemble.simulate (host variant, no records) and K steps of the host loop (hc_step on the ensemble's pinned buffers
   + numpy Euler over all instances) are timed in alternating windows on two ensembles of the same set-up.
2. Sphere power matrix: 16384 instances = 128 PTO damping values x 128 seeds, heave only, irregular waves, Euler,
   simulate with the absorbed-energy output; instance-steps/s and the mean absorbed power range.
3. With 8 GPUs: the strong split (2048 instances per GPU) through hc_multi_ensemble_simulate against hc_multi_step +
   the same host loop.  Fewer GPUs: reported as not measured.
Every timed trajectory is checked to be finite.  The card's name and power limit are read in the same run.
usage: python profiles/device_stepping_bench.py [--out FILE] [--steps K] [--windows W]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

DT = 0.01
RM3_FREE = np.tile(np.array([0, 0, 1, 0, 1, 0], bool), 2)


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "device_count": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi_index_name_power_limit_max_sm_clock"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi_index_name_power_limit_max_sm_clock"] = "unavailable: %s" % e
    return info


def minv(added, mass, inertia, free):
    D = added.shape[0]
    M = np.diag(np.concatenate([[m] * 3 + list(j) for m, j in zip(mass, inertia)])) + added
    idx = np.where(free)[0]
    out = np.zeros((D, D))
    out[np.ix_(idx, idx)] = np.linalg.inv(M[np.ix_(idx, idx)])
    return out


class HostLoop:
    """hc_step (or hc_multi_step) + vectorised numpy linearised Euler over every instance (translations and Cardan
    angles integrated alike: the timing baseline, not a reference)."""

    def __init__(self, step, B, D, Mi, mass, free, pose0, g=(0.0, 0.0, -9.81), c=None):
        self.step, self.Mi, self.free = step, Mi, free
        self.pose, self.vel = pose0.copy(), np.zeros((B, D))
        self.force = np.empty((B, D))
        self.fg = np.zeros(D)
        for b, m in enumerate(mass):
            self.fg[6 * b:6 * b + 3] = m * np.asarray(g)
        self.c = np.zeros((B, D)) if c is None else c
        self.t = 0.0

    def run(self, n):
        for _ in range(n):
            self.step(self.t, self.pose, self.vel, self.force)
            F = self.force + self.fg - self.c * self.vel
            self.vel = np.where(self.free, self.vel + DT * (F @ self.Mi.T), 0.0)
            self.pose = self.pose + DT * self.vel
            self.t += DT


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def rm3_leg(hc, synth, K, W, B=16384):
    raw = synth.rm3_like()
    T = hc.Tables.from_raw(raw)
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    total = 6050 + (K + 1) * W + 10
    irr = dict(dt=DT, duration=total * DT + 10.0, ramp=20.0, Hs=2.5, Tp=8.0, nfreq=1000, gamma=3.3)
    seeds = np.arange(1, B + 1, dtype=np.int32)
    pose0 = np.zeros((B, 12))
    pose0[:, 2], pose0[:, 8] = -0.05, 0.05

    def make():
        e = hc.Ensemble(T, batch=B, dt_hint=DT, bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=4)
        e.set_waves_irregular(seeds=seeds, **irr)
        return e

    dev, host = make(), make()
    state = {"t": 0.0, "pose": pose0, "vel": np.zeros((B, 12))}

    def dev_run(n):
        r = dev.simulate(state["pose"], n, DT, mass, inertia, vel0=state["vel"], t0=state["t"], free_dof=RM3_FREE,
                         record=False, energy=False)
        state["pose"], state["vel"] = r.final_pose, r.final_vel
        for _ in range(n):
            state["t"] += DT
        assert r[4] == n

    pb, vb, fb = host.host_buffers()
    loop = HostLoop(lambda t, p, v, f: (pb.__setitem__(slice(None), p), vb.__setitem__(slice(None), v),
                                         host.step(t, pb, vb, out=f)),
                    B, 12, minv(T.added_mass(), mass, inertia, RM3_FREE), mass, RM3_FREE, pose0)
    t_fill = timed(lambda: dev_run(6050))
    loop.run(6050)
    assert abs(loop.t - state["t"]) < 1e-9
    dev_s, host_s = [], []
    for _ in range(W):
        dev_s.append(timed(lambda: dev_run(K)))
        host_s.append(timed(lambda: loop.run(K)))
    ok = bool(np.all(np.isfinite(state["pose"])) and np.all(np.isfinite(loop.pose)))
    served = dev.rad_block_stats()["steps_served"]
    hist = dev.history_len()
    dev.close(); host.close()
    return {
        "workload": "RM3-shaped, %d instances, dt %.2f, irregular nf 1000, bracket_snap 1e-8, rad_lookahead 2, "
                    "exc_lookahead 4, heave + pitch free per body, Euler, history window full (%d rows)" % (B, DT, hist),
        "fill_6050_steps_s": t_fill,
        "window_steps": K, "windows": W,
        "device_simulate_s_per_window": dev_s, "host_loop_s_per_window": host_s,
        "device_instance_steps_per_s_median": B * K / float(np.median(dev_s)),
        "host_loop_instance_steps_per_s_median": B * K / float(np.median(host_s)),
        "device_us_per_step_median": 1e6 * float(np.median(dev_s)) / K,
        "host_loop_us_per_step_median": 1e6 * float(np.median(host_s)) / K,
        "speedup_median": float(np.median(host_s)) / float(np.median(dev_s)),
        "radiation_steps_served_by_lookahead": served,
        "trajectories_finite": ok,
    }


def sphere_power_matrix(hc, common, K, B=16384):
    T = hc.Tables.from_raw(common.sphere_raw())
    nd, ns = 128, B // 128
    damping = np.repeat(np.linspace(0.0, 1.2e6, nd), ns)
    seeds = np.tile(np.arange(1, ns + 1, dtype=np.int32), nd)
    c = np.zeros((B, 6))
    c[:, 2] = damping
    n = K
    ens = hc.Ensemble(T, batch=B, dt_hint=common.SPHERE_DT, bracket_snap=1e-8)
    ens.set_waves_irregular(dt=common.SPHERE_DT, duration=n * common.SPHERE_DT + 70.0, ramp=20.0, Hs=2.0, Tp=8.0,
                            nfreq=1000, gamma=3.3, seeds=seeds)
    pose0 = np.zeros((B, 6))
    free = np.array([0, 0, 1, 0, 0, 0], bool)
    kw = dict(free_dof=free, pto_damping=c, record=False)
    ens.simulate(pose0, 100, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]], **kw)       # warm-up
    ens.reset()
    t0 = time.perf_counter()
    r = ens.simulate(pose0, n, common.SPHERE_DT, [common.SPHERE_MASS], [[1.0, 1.0, 1.0]], **kw)
    s = time.perf_counter() - t0
    P = r[3][:, 2] / (n * common.SPHERE_DT)
    ok = bool(np.all(np.isfinite(r.final_pose)) and np.all(np.isfinite(P)))
    ens.close()
    return {"workload": "sphere, %d instances = %d PTO damping values x %d seeds, heave only, irregular Hs 2 Tp 8 nf 1000, "
                        "dt %.3f, Euler, %d steps from rest (the 15 s history window is full after 1000)" % (B, nd, ns, common.SPHERE_DT, n),
            "simulate_s": s, "instance_steps_per_s": B * n / s, "us_per_step": 1e6 * s / n,
            "mean_absorbed_power_W_min_max": [float(P.min()), float(P.max())], "trajectories_finite": ok}


def strong_split(hc, synth, K, n_gpu=8, B=16384):
    if hc.device_count() < n_gpu:
        return {"status": "not measured: %d GPU(s) on this machine" % hc.device_count()}
    T = hc.Tables.from_raw(synth.rm3_like())
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    irr = dict(dt=DT, duration=(3 * K + 100) * DT + 10.0, ramp=20.0, Hs=2.5, Tp=8.0, nfreq=1000, gamma=3.3)
    seeds = np.arange(1, B + 1, dtype=np.int32)
    pose0 = np.zeros((B, 12))
    out = {}
    for name in ("device", "host_loop"):
        me = hc.MultiEnsemble(T, B, devices=list(range(n_gpu)), dt_hint=DT, bracket_snap=1e-8, rad_lookahead=2,
                              exc_lookahead=4)
        me.set_waves_irregular(seeds=seeds, **irr)
        if name == "device":
            me.simulate(pose0, 50, DT, mass, inertia, free_dof=RM3_FREE, record=False, energy=False)
            t0 = time.perf_counter()
            r = me.simulate(pose0, K, DT, mass, inertia, t0=50 * DT, free_dof=RM3_FREE, record=False, energy=False)
            s = time.perf_counter() - t0
            ok = bool(np.all(np.isfinite(r.final_pose)))
        else:
            loop = HostLoop(lambda t, p, v, f: me.step(t, p, v, out=f), B, 12, minv(T.added_mass(), mass, inertia, RM3_FREE),
                            mass, RM3_FREE, pose0)
            loop.run(50)
            s = timed(lambda: loop.run(K))
            ok = bool(np.all(np.isfinite(loop.pose)))
        out[name] = {"s": s, "instance_steps_per_s": B * K / s, "trajectories_finite": ok}
        me.close()
    out["workload"] = "RM3-shaped, %d instances over %d GPUs, Euler, %d steps (history window not full)" % (B, n_gpu, K)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "device_stepping_bench.json"))
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--windows", type=int, default=3)
    a = ap.parse_args()
    import torch  # noqa: F401
    import common
    import hydrochrono_b200 as hc
    from hydrochrono_b200 import synth
    res = {"card": card_info()}
    res["rm3_window_full"] = rm3_leg(hc, synth, a.steps, a.windows)
    print(json.dumps(res["rm3_window_full"]), flush=True)
    res["sphere_power_matrix"] = sphere_power_matrix(hc, common, 2000)
    print(json.dumps(res["sphere_power_matrix"]), flush=True)
    res["strong_split_8_gpus"] = strong_split(hc, synth, a.steps)
    print(json.dumps(res["strong_split_8_gpus"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
