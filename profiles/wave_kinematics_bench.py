"""Water-kinematics benchmark: hc_waves_kinematics_at_time_device (k_wave_kinematics) on one GPU.

1. Device call time (CUDA events on the ensemble's stream, after warm-up) over B in {2048, 16384}, P in {1, 2, 8}
   points per instance, nf in {64, 1000} components, Wheeler stretching off and on; reported as ms per call and as
   component evaluations per second (B P nf per call; with Wheeler stretching the elevation pass runs in addition).
   At B = 16384, nf = 1000 the per-instance phases are 131 MB, just above the 126 MB L2, and are re-read every call;
   the smaller shapes run from L2 after the first call.
2. The host arithmetic for comparison: hc_wave_kinematics (one instance, one point, nf components) timed on a sample
   of calls and scaled to B P calls per query.
3. The cost of one call per step (P = 2, Wheeler off) on top of device-resident stepping at bench.py's workload
   (RM3-shaped tables, 16384 instances, dt = 0.01, nf = 1000, snapped brackets, both look-aheads), in alternating
   windows with and without the call.
The card's name and power limit are read in the same run.
usage: python profiles/wave_kinematics_bench.py [--out FILE] [--step-window K]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEA = dict(Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0, ramp=20.0)


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi_name_power_limit_max_sm_clock"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi_name_power_limit_max_sm_clock"] = "unavailable: %s" % e
    return info


def points(B, P):
    rng = np.random.default_rng(5)
    pts = np.empty((B, P, 3))
    pts[..., 0] = rng.uniform(-50.0, 50.0, (B, P))
    pts[..., 1] = 0.0
    pts[..., 2] = rng.uniform(-10.0, 0.5, (B, P))
    return pts


def time_device_calls(torch, ens, stream, P, d_pts, outs, wheeler, min_seconds=0.3):
    def window(n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(n):
            ens.wave_kinematics_device(100.0 + 0.01 * i, P, d_pts, *outs, wheeler=wheeler)
        ev1.record(stream)
        ens.sync()
        return ev0.elapsed_time(ev1) / n
    window(3)                                             # warm-up (first call stages the components)
    est = window(3)
    n = int(min(5000, max(5, min_seconds / max(est * 1e-3, 1e-9))))
    return min(window(n) for _ in range(3)), n


def kernel_grid(hc, torch, out):
    from hydrochrono_b200 import synth
    T = hc.Tables.from_raw(synth.rm3_like(rirf_steps=201, rirf_duration=10.0, exc_irf_steps=201, exc_half_window=5.0))
    dev = torch.device("cuda", 0)
    rows = []
    for B in (2048, 16384):
        for nf in (64, 1000):
            stream = torch.cuda.Stream(device=dev)
            ens = hc.Ensemble(T, batch=B, stream=stream.cuda_stream)
            ens.set_waves_irregular(dt=0.01, duration=10.0, nfreq=nf, seeds=np.arange(1, B + 1, dtype=np.int32), **SEA)
            for P in (1, 2, 8):
                d_pts = torch.from_numpy(points(B, P)).to(dev)
                outs = (torch.empty((B, P), dtype=torch.float64, device=dev),
                        torch.empty((B, P, 3), dtype=torch.float64, device=dev),
                        torch.empty((B, P, 3), dtype=torch.float64, device=dev))
                torch.cuda.synchronize()
                for wheeler in (False, True):
                    ms, n = time_device_calls(torch, ens, stream, P, d_pts, outs, wheeler)
                    evals = B * P * nf
                    rows.append({"B": B, "P": P, "nf": nf, "wheeler": wheeler, "ms_per_call": ms, "calls_timed": n,
                                 "component_evals_per_call": evals, "component_evals_per_s": evals / (ms * 1e-3)})
                    print("B %5d  P %d  nf %4d  wheeler %d  %.4f ms/call  %.3e comp/s" %
                          (B, P, nf, wheeler, ms, evals / (ms * 1e-3)), flush=True)
            ens.close()
    out["device_calls"] = rows


def host_sample(hc, out, nf=1000, calls=200):
    rng = np.random.default_rng(1)
    f = np.linspace(0.001, 1.0, nf)
    om = 2 * np.pi * f
    k = np.array([hc.compute_wave_number(w, 200.0, 9.81) for w in om])
    A = np.full(nf, 0.01)
    t0 = time.perf_counter()
    for _ in range(calls):
        ph = rng.uniform(0, 2 * np.pi, nf)
        hc.wave_kinematics(om, A, ph, k, (rng.uniform(-50, 50), 0.0, -2.0), 417.0, 200.0)
    per_call = (time.perf_counter() - t0) / calls
    out["host_hc_wave_kinematics"] = {
        "nf": nf, "calls_timed": calls, "seconds_per_instance_point": per_call,
        "seconds_per_query_B16384_P2_extrapolated": per_call * 16384 * 2,
        "note": "one host thread; phases drawn per call (as a loop over instances would fetch them); scaled linearly "
                "from the sample to 16384 x 2 calls"}
    print("host: %.3e s per (instance, point) at nf %d -> %.2f s per 16384 x 2 query" % (per_call, nf, per_call * 32768))


def step_overhead(hc, torch, out, K):
    from hydrochrono_b200 import synth
    B, dt, D = 16384, 0.01, 12
    prefill = 6010                                        # fills the 10 s radiation window (bench.py's PREFILL)
    total = prefill + 4 * K + 64
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev, priority=-1)
    T = hc.Tables.from_raw(synth.rm3_like())
    ens = hc.Ensemble(T, batch=B, dt_hint=dt, bracket_snap=1e-8, stream=stream.cuda_stream)
    ens.set_waves_irregular(dt=dt, duration=total * dt, nfreq=1000, seeds=np.arange(1, B + 1, dtype=np.int32), **SEA)
    amp, om = synth.prescribed_motion(D)
    ph = 0.01 * np.arange(B)[:, None]
    d_pose = [torch.from_numpy(amp * np.sin(om * (i * dt) + ph)).to(dev) for i in range(8)]
    d_vel = [torch.from_numpy(amp * om * np.cos(om * (i * dt) + ph)).to(dev) for i in range(8)]
    d_force = torch.empty((B, D), dtype=torch.float64, device=dev)
    d_pts = torch.from_numpy(points(B, 2)).to(dev)
    outs = (torch.empty((B, 2), dtype=torch.float64, device=dev), torch.empty((B, 2, 3), dtype=torch.float64, device=dev),
            torch.empty((B, 2, 3), dtype=torch.float64, device=dev))
    torch.cuda.synchronize()
    state = {"n": 0, "t": 0.0}

    def step(with_call):
        n = state["n"]
        ens.step_device(state["t"], d_pose[n % 8], d_vel[n % 8], d_force)
        if with_call:
            ens.wave_kinematics_device(state["t"], 2, d_pts, *outs)
        state["n"] += 1
        state["t"] += dt

    for _ in range(prefill):
        step(False)
    ens.sync()

    def window(with_call):
        while state["n"] % 8:
            step(False)
        ens.join(); ens.sync()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(K):
            step(with_call)
        ens.join()
        ev1.record(stream)
        ens.sync()
        return ev0.elapsed_time(ev1) / K

    res = {"without": [], "with": []}
    for _ in range(2):
        res["without"].append(window(False))
        res["with"].append(window(True))
    out["step_overhead"] = {
        "workload": "bench.py rm3_irregular_ensemble: 16384 instances, dt 0.01, nf 1000, bracket_snap 1e-8, look-aheads auto",
        "steps_per_window": K, "prefill_steps": prefill, "ms_per_step_without_call": res["without"],
        "ms_per_step_with_one_call_P2": res["with"],
        "added_ms_per_step": float(np.mean(res["with"]) - np.mean(res["without"])),
        "lookahead_state": ens.lookahead_state()}
    print("step: %s ms without, %s ms with one P = 2 call per step" % (res["without"], res["with"]))
    ens.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wave_kinematics_bench.json"))
    ap.add_argument("--step-window", type=int, default=500)
    args = ap.parse_args()
    import torch
    import hydrochrono_b200 as hc
    if not torch.cuda.is_available():
        raise SystemExit("wave_kinematics_bench: no CUDA device (the measurement needs the GPU)")
    out = {"card": card_info()}
    kernel_grid(hc, torch, out)
    host_sample(hc, out)
    step_overhead(hc, torch, out, args.step_window)
    out["card_after"] = card_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
