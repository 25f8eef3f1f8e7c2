"""RM3 power matrix on the device: the float on a prismatic joint to its spar with a damper PTO between them
(k_body_step_linked), 16384 instances = 128 PTO dampings x 128 sea-state seeds, against the free-body leg of
device_stepping_bench.py (the same tables and waves, each body heaving and pitching on its own, k_body_step).

RM3-shaped tables, dt = 0.01, irregular waves (nf 1000), snapped brackets, both look-aheads, linearised Euler.  Both
ensembles first fill the history window (6050 untimed steps); then K steps of each are timed in alternating windows.
Jointed run: float all free (reduced to its slide), spar heave / roll / pitch free.  Then, in a run of its own under
torch.profiler (CUDA activities), the device time of the integrator kernels per launch.  The mean absorbed power per
damping value is the PTO energy of the timed windows over their duration, averaged over the 128 seeds.  The card's
name and power limit are read in the same run.
usage: python profiles/rm3_power_matrix_bench.py [--out FILE] [--steps K] [--windows W]
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402

from device_stepping_bench import DT, RM3_FREE, card_info, timed  # noqa: E402

FLOAT_Z, SPAR_Z = -0.72, -21.29
SPAR_FREE = np.array([1, 1, 1, 1, 1, 1, 0, 0, 1, 1, 1, 0], bool)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rm3_power_matrix_bench.json"))
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16384)
    a = ap.parse_args()
    import torch
    import hydrochrono_b200 as hc
    from hydrochrono_b200 import synth
    B, K, W = a.batch, a.steps, a.windows
    nd, ns = 128, max(B // 128, 1)
    T = hc.Tables.from_raw(synth.rm3_like())
    mass, inertia = synth.RM3_MASSES, synth.RM3_INERTIAS
    total = 6050 + (K + 1) * W + 200
    irr = dict(dt=DT, duration=total * DT + 10.0, ramp=20.0, Hs=2.5, Tp=8.0, nfreq=1000, gamma=3.3)
    damping = np.repeat(np.linspace(0.0, 4e6, nd), ns)[:B]
    seeds = np.tile(np.arange(1, ns + 1, dtype=np.int32), nd)[:B]
    joint = hc.Prismatic(0, 1, (0.0, 0.0, 1.0))
    pto = hc.TSDA(0, 1, (0.0, 0.0, FLOAT_Z), (0.0, 0.0, SPAR_Z), damping=damping)
    legs = {
        "jointed": dict(pose=np.tile([0, 0, FLOAT_Z, 0, 0, 0, 0, 0, SPAR_Z, 0, 0, 0], (B, 1)).astype(float),
                        kw=dict(free_dof=SPAR_FREE, prismatic=[joint], tsda=[pto], record=False, energy=True)),
        "free_body": dict(pose=np.tile([0, 0, -0.05, 0, 0, 0, 0, 0, 0.05, 0, 0, 0], (B, 1)).astype(float),
                          kw=dict(free_dof=RM3_FREE, record=False, energy=False)),
    }
    for leg in legs.values():
        e = hc.Ensemble(T, batch=B, dt_hint=DT, bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=4)
        e.set_waves_irregular(seeds=seeds, **irr)
        leg.update(ens=e, t=0.0, vel=np.zeros((B, 12)), energy=np.zeros(B), steps=0, s=[])

    def run(leg, n, count=True):
        r = leg["ens"].simulate(leg["pose"], n, DT, mass, inertia, vel0=leg["vel"], t0=leg["t"], **leg["kw"])
        assert r[4] == n
        leg["pose"], leg["vel"] = r.final_pose, r.final_vel
        for _ in range(n):
            leg["t"] += DT
        if count and r.tsda_energy is not None:
            leg["energy"] += r.tsda_energy[:, 0]
            leg["steps"] += n

    fill = {name: timed(lambda: run(leg, 6050, count=False)) for name, leg in legs.items()}
    for _ in range(W):
        for leg in legs.values():
            leg["s"].append(timed(lambda: run(leg, K)))
    res = {"card": card_info()}
    for name, leg in legs.items():
        med = float(np.median(leg["s"]))
        res[name] = {"fill_6050_steps_s": fill[name], "s_per_window": leg["s"], "window_steps": K, "windows": W,
                     "instance_steps_per_s_median": B * K / med, "us_per_step_median": 1e6 * med / K,
                     "history_rows": leg["ens"].history_len(),
                     "trajectories_finite": bool(np.all(np.isfinite(leg["pose"])))}
    res["jointed_over_free_body_time"] = float(np.median(legs["jointed"]["s"]) / np.median(legs["free_body"]["s"]))
    P = legs["jointed"]["energy"] / (legs["jointed"]["steps"] * DT)
    per_c = P.reshape(nd, -1).mean(axis=1) if B % nd == 0 else P
    res["mean_absorbed_power_W_per_damping"] = {"damping_Ns_per_m": [float(c) for c in np.linspace(0.0, 4e6, nd)],
                                                "power_W": [float(p) for p in per_c]}
    # integrator kernels' own device time: torch.profiler with CUDA activities, one window of each leg
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    with tempfile.TemporaryDirectory() as tmp:
        os.environ.setdefault("TMPDIR", tmp)
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for leg in legs.values():
                run(leg, 100, count=False)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if ev.key.startswith("_ZN2hc11k_body_step") or ev.key.startswith("_ZN2hc18k_body_step_linked") or \
                    "k_body_step" in ev.key:
                dev_us = getattr(ev, "device_time_total", None)
                if dev_us is None:
                    dev_us = ev.cuda_time_total
                kern[ev.key] = {"launches": ev.count, "device_us_total": float(dev_us),
                                "device_us_per_launch": float(dev_us) / max(ev.count, 1)}
    res["integrator_kernels_torch_profiler"] = kern
    res["workload"] = ("RM3-shaped tables, %d instances = %d PTO dampings (0 .. 4e6 N s/m) x %d seeds, dt %.2f, irregular "
                       "Hs 2.5 Tp 8 nf 1000, bracket_snap 1e-8, rad_lookahead 2, exc_lookahead 4, Euler, history window "
                       "full; jointed: float on a prismatic joint to the spar + damper PTO, spar heave / roll / pitch "
                       "free; free_body: heave + pitch per body, no joint" % (B, nd, ns, DT))
    for leg in legs.values():
        leg["ens"].close()
    print(json.dumps(res), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    t0 = time.perf_counter()
    main()
    print("total %.1f s" % (time.perf_counter() - t0))
