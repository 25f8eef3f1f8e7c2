#!/usr/bin/env python
"""bench.py -- batched sim-steps/s of the hydrodynamic force path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload = "rm3_irregular_ensemble"): SURVEY.md section 8(d) -- RM3-shaped two-body design
(D = 12, L = 1001 radiation lags over 60 s, dt = 0.01 s, excitation IRF +-30 s -> 6000 lags), JONSWAP
Hs 2.5 m / Tp 8 s / gamma 3.3, 1000 spectrum components, one random-phase realisation per instance
(seed 1 + global instance index).  A "step" is one lock-step force evaluation of every instance: hydrostatics +
radiation convolution + excitation convolution + total.  The velocity-history window is pre-filled (>= 6000 steps)
before anything is timed, so the timed steps are steady state.

The line's `value` / `e2e` are WEAK scaling: 16384 instances PER GPU (instances are independent, tables replicated, no
data-path collective).  For N > 1 the same run also measures the north-star split -- 16384 instances IN TOTAL
partitioned over the N GPUs -- and reports it under "strong".

value : instance-steps/s with the step's pose/velocity already resident in HBM (hc_step_device), CUDA events on the
        ensemble's stream; both events are recorded after hc_ensemble_join, so the interval holds every look-ahead
        pass the K steps gave rise to on the library's side streams.  Max over ranks.
e2e   : the same through the host-buffer C-ABI call (hc_step): pinned host pose/velocity -> H2D -> kernels -> D2H
        force, every step, wall clock around K synchronous calls + a device synchronize, max over ranks.
parity: after the timed legs the CPU oracle is loaded with the history of sampled instances and stepped next to the
        GPU for a few dozen more steps, at the benchmarked state (full batch, full window, ring wrapped).
--dump-outputs DIR: forces_device.npy / forces_host.npy = the [instances, D] forces of the last timed step of the
        `value` and `e2e` legs.  Every input is seeded, so two builds run with the same arguments can be compared
        element for element.

`--impl reference` times the reference's CPU path (the oracle port; the reference needs Chrono/Eigen/HDF5 and cannot be
compiled here) on the box's host cores: K real lock-steps of a bounded sample of the same workload.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# headline workload (BASELINE.json metric) -- module-level names are rebound by select_workload()
DT = 0.01
DOFS = 12
RIRF_STEPS = 1001
EXC_STEPS = 6000
SEA = dict(Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0, nfreq=1000, ramp=20.0)
SNAP = 1e-8
GVEC = (0.0, 0.0, -9.81)
WORKLOAD = "rm3_irregular_ensemble"
PREFILL = 6010
NBUF = 8                    # the synthetic state of step n is buffer n % NBUF
TOTAL_INSTANCES = 16384     # the north-star ensemble
METRIC = "batched sim-steps/sec (RM3 irregular ensemble)"


def load_plain(name):
    """hydrochrono_b200/<name>.py as a stand-alone module: the package __init__ (which maps the product .so) does not
    run, so the reference arm's process holds no product code."""
    spec = importlib.util.spec_from_file_location("hc_plain_" + name, os.path.join(ROOT, "hydrochrono_b200", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def workload_tables():
    if WORKLOAD == "sphere_irregular_ensemble":
        return sphere_tables()
    return load_plain("synth").rm3_like()


def sphere_tables():
    z = np.load(os.path.join(ROOT, "tests", "golden", "sphere_tables.npz"))
    body = {k: z[k] for k in ("cg", "cb", "lin_matrix", "inf_added_mass", "rirf_K", "rirf_t", "exc_mag", "exc_phase",
                              "exc_irf_f", "exc_irf_t")}
    body["disp_vol"] = float(z["disp_vol"])
    return {"rho": float(z["rho"]), "g": float(z["g"]), "water_depth": float(z["water_depth"]), "w": z["w"],
            "bodies": [body]}


def select_workload(name):
    """Secondary workload on the reference's real tables (SURVEY.md 8d): sphere x 16384, N = 1, D = 6, L = 1001 lags
    with rirf spacing == dt = 0.015, excitation IRF resampled to 8334 lags, Hs 2 / Tp 12 / gamma 1."""
    global DT, DOFS, RIRF_STEPS, EXC_STEPS, SEA, WORKLOAD, PREFILL
    WORKLOAD = name
    if name == "sphere_irregular_ensemble":
        DT, DOFS, RIRF_STEPS, EXC_STEPS, PREFILL = 0.015, 6, 1001, 8334, 1010
        SEA = dict(Hs=2.0, Tp=12.0, gamma=1.0, fmin=0.001, fmax=1.0, nfreq=1000, ramp=60.0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=TOTAL_INSTANCES, help="instances per GPU (weak-scaling leg)")
    ap.add_argument("--prefill", type=int, default=-1, help="untimed steps to fill the history window (-1 = auto)")
    ap.add_argument("--faithful", action="store_true", help="bracket_snap = 0 (bit-faithful bracketing) for the main legs")
    ap.add_argument("--rad-chunk", type=int, default=0)
    ap.add_argument("--exc-chunk", type=int, default=0)
    ap.add_argument("--cpu-instances", type=int, default=0, help="reference arm: instances in the sample (0 = 32 per core, <= 1024)")
    ap.add_argument("--cpu-steps", type=int, default=0, help="(kept for compatibility; the reference arm times --steps lock-steps)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check at the benchmarked state")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling (16384 in total) leg")
    ap.add_argument("--no-b1", action="store_true", help="skip the B = 1 drop-in latency leg")
    ap.add_argument("--no-faithful-leg", action="store_true", help="skip the short bracket_snap = 0 leg")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-lookahead", action="store_true", help="per-step excitation kernel only")
    ap.add_argument("--lookahead-mode", type=int, default=0, help="0 auto (= 5), 2 in-stream, 3 background, 4 in-stream DMMA, 5 background DMMA")
    ap.add_argument("--rad-lookahead", type=int, default=0, help="radiation look-ahead block: 0 auto (on, background), 1 off, 2 on (background), 3 on (in-stream)")
    ap.add_argument("--rad-pass-mode", type=int, default=0, help="pacing of the look-ahead pass: 0 auto, 1 gated slice per step, 2 ungated slice per step, 3 whole pass per block")
    ap.add_argument("--rad-kernel", type=int, default=0, help="0 auto (= 1), 1 FP64 FMA pipe, 2 FP64 tensor cores (DMMA, 12 DoF only), 3 tensor cores (rows 0-7) + FMA pipe (rows 8-11)")
    ap.add_argument("--multi-devices", default="", help="single-process hc_multi_* mode on this comma-separated device list "
                                                        "(a device may repeat: several shards on one GPU)")
    ap.add_argument("--workload", default="rm3_irregular_ensemble",
                    choices=["rm3_irregular_ensemble", "sphere_irregular_ensemble"])
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the forces of the last timed step of each timed leg as DIR/<name>.npy (float64, "
                         "[instances, dofs]; a fixed sample of rows when they would exceed 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm returns no forces")
    return args


DUMP_BYTES = 63 << 20          # under 64 MB with the .npy headers


def dump_outputs(directory, arrays):
    """arrays: {name: [rows, ...]} with equal row counts.  Beyond DUMP_BYTES in all, every array keeps the same seeded
    sample of rows (a function of the row count only), so runs with the same arguments write the same elements."""
    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    rows = None
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            if rows is None:
                rows = np.sort(np.random.default_rng(0).choice(len(a), len(a) * DUMP_BYTES // total, replace=False))
            a = a[rows]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------------
# synthetic inputs shared by both arms
# ------------------------------------------------------------------------------------------------------
def step_times(n):
    """t advanced as Chrono advances ChTime: repeated addition of dt."""
    out = np.empty(n)
    t = 0.0
    for i in range(n):
        out[i] = t
        t += DT
    return out


def motion_buffers(amp, om, nb, offset=0):
    """pose / vel [NBUF][nb][D]: the prescribed state of step n is buffer n % NBUF (instance i gets a phase 0.01 i)."""
    ph = 0.01 * (offset + np.arange(nb))[:, None]
    pose = np.stack([amp * np.sin(om * (i * DT) + ph) for i in range(NBUF)])
    vel = np.stack([amp * om * np.cos(om * (i * DT) + ph) for i in range(NBUF)])
    return np.ascontiguousarray(pose), np.ascontiguousarray(vel)


def base_config(batch, world):
    """Identical in both arms (the driver compares the key sets)."""
    hist_gb = 8e-9 * DOFS * batch * (RIRF_STEPS - 1) * round((60.0 if DOFS == 12 else 15.0) / (RIRF_STEPS - 1) / DT)
    return {"workload": WORKLOAD, "instances_per_gpu": batch, "instances_total": world * batch, "dofs": DOFS,
            "rirf_steps": RIRF_STEPS, "exc_irf_steps": EXC_STEPS, "dt": DT, "spectrum_components": SEA["nfreq"],
            "sea_state": SEA, "history_prefill_steps": PREFILL,
            "l2": "inputs larger than L2 (126 MB), no flush needed: the %.1f GB velocity-history window and the eta "
                  "table of a GPU's instances are streamed from HBM" % hist_gb}


class ClockSampler:
    """SM clock and throttle reasons of ONE GPU, sampled during the timed region by a thread of the rank that drives
    it (in-process NVML, ~0.1 ms per sample every 20 ms).  A single `nvidia-smi -lms` process polling all the GPUs of
    an 8-rank job stalls kernel launches of every rank while it walks the devices, so nvidia-smi is only the fallback
    when the NVML binding is missing."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.th, self.nvml, self.proc = index, [], False, None, None, None
        self.period = float(os.environ.get("HC_BENCH_CLOCK_PERIOD", "0.005"))

    def start(self):
        if os.environ.get("HC_BENCH_NO_CLOCKS"):       # experiment switch: no sampling at all
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            try:      # the CUDA ordinal need not be the NVML index: match by UUID when torch exposes it
                import torch
                self.h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(self.index).uuid))
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception:
            self.nvml = None
            try:
                q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                              "--format=csv,noheader,nounits", "-lms", "100"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.th = threading.Thread(target=self._read, daemon=True)
                self.th.start()
            except Exception:
                self.proc = None

    def _poll(self):
        n = self.nvml
        bits = [n.nvmlClocksThrottleReasonHwSlowdown, n.nvmlClocksThrottleReasonHwThermalSlowdown,
                n.nvmlClocksThrottleReasonSwThermalSlowdown, n.nvmlClocksThrottleReasonSwPowerCap]
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((sm, self.mx, [1.0 if (r & b) else 0.0 for b in bits]))
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            try:
                self.samples.append((float(p[0]), float(p[1]), [1.0 if v.lower().startswith("active") else 0.0 for v in p[2:6]]))
            except (ValueError, IndexError):
                continue

    def stop(self):
        """[median sm, min sm, max clock, 4 reason flags, samples] of this GPU (None when unavailable)."""
        self.stop_flag = True
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
        if self.th:
            self.th.join(timeout=2)
        if not self.samples:
            return None
        sm = [x[0] for x in self.samples]
        flags = [max(x[2][i] for x in self.samples) for i in range(4)]
        return [float(np.median(sm)), float(min(sm)), float(max(x[1] for x in self.samples))] + flags + [float(len(sm))]


def hbm_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernels from the committed ncu --set full capture, if any."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (line-faithful port of the reference's CPU path) on the host cores
# ------------------------------------------------------------------------------------------------------
def oracle_with_all_cores():
    """torchrun exports OMP_NUM_THREADS=1 to its children; the reference arm uses every host core it can."""
    os.environ.pop("OMP_NUM_THREADS", None)
    from oracle import hc_oracle as orc
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    orc.set_num_threads(cores)
    return orc, cores


def oracle_instances(orc, T, seeds, duration, threads):
    """Instances with their own eta realisation (the synthesis is the slow part of set-up: one thread per instance)."""
    from concurrent.futures import ThreadPoolExecutor
    kw = dict(dt=DT, duration=duration, ramp=SEA["ramp"], Hs=SEA["Hs"], Tp=SEA["Tp"], fmin=SEA["fmin"], fmax=SEA["fmax"],
              nfreq=SEA["nfreq"], gamma=SEA["gamma"])
    first = orc.Instance(T, omp_mode=0)
    first.set_irregular(seed=int(seeds[0]), **kw)

    def make(s):
        inst = orc.Instance(T, omp_mode=0)
        inst.set_irregular(seed=int(s), share_irf_from=first, **kw)      # ctypes releases the GIL
        return inst
    if len(seeds) == 1:
        return [first]
    with ThreadPoolExecutor(max_workers=max(1, threads)) as ex:
        return [first] + list(ex.map(make, seeds[1:]))


def window_rows(raw):
    """Rows of velocity history a full radiation window holds at the workload's step size (+ slack)."""
    return int(round(float(raw["bodies"][0]["rirf_t"][-1]) / DT)) + 4


def load_history(insts, times, vel_bufs, n_done, window_rows):
    """What stepping instance i through steps 0 .. n_done - 1 would have left in its velocity history."""
    rows = min(n_done, window_rows)
    idx = np.arange(n_done - 1, n_done - 1 - rows, -1)                   # newest first
    tnf = times[idx]
    for i, inst in enumerate(insts):
        inst.set_history(tnf, vel_bufs[idx % NBUF, i, :])


def cpu_reference(K, W, n_inst, prefill, instance_offset=0):
    """K timed lock-steps of a bounded sample (n_inst instances, one per thread across all cores) in steady state."""
    synth = load_plain("synth")
    orc, cores = oracle_with_all_cores()
    if n_inst <= 0:
        n_inst = min(1024, 32 * cores)
    raw = workload_tables()
    T = orc.Tables(raw)
    amp, om = synth.prescribed_motion(DOFS)
    n_total = prefill + W + K + 16
    times = step_times(n_total + 64)
    t_setup = time.time()
    seeds = 1 + instance_offset + np.arange(n_inst)
    insts = oracle_instances(orc, T, seeds, (n_total + 64) * DT, cores)
    pose, vel = motion_buffers(amp, om, n_inst, instance_offset)
    load_history(insts, times, vel, prefill, window_rows(raw))
    setup_s = time.time() - t_setup
    n = prefill
    if W > 0:
        orc.bench_lockstep(insts, times[n:n + W], pose, vel, buf0=n % NBUF, mode=1, gvec=GVEC)
        n += W
    sec, cs, _ = orc.bench_lockstep(insts, times[n:n + K], pose, vel, buf0=n % NBUF, mode=1, gvec=GVEC)
    n += K
    value = n_inst * K / sec
    # reference-style threading: instances one after another, OpenMP across radiation lags (hydro_forces.cpp:593-647)
    n_ref, k_ref = min(n_inst, 4), min(8, 16)
    sec_ref, _, _ = orc.bench_lockstep(insts[:n_ref], times[n:n + k_ref], pose[:, :n_ref].copy(), vel[:, :n_ref].copy(),
                                       buf0=n % NBUF, mode=0, gvec=GVEC)
    ref_style = n_ref * k_ref / sec_ref
    hist = insts[0].history_len()
    return {"value": value, "unit": "instance-steps/s", "cores": cores, "kind": "port",
            "sample": "%d instances (seeds %d..%d) x %d timed lock-steps after %d warm-up steps, history window loaded "
                      "with the %d rows of a %d-step prefill, one instance per thread over %d threads (best effort); "
                      "reference-style threading (OpenMP across lags, instances serial): %.1f instance-steps/s on %d "
                      "instances x %d steps" % (n_inst, seeds[0], seeds[-1], K, W, hist, prefill, cores, ref_style, n_ref,
                                                k_ref),
            "reference_style_value": ref_style, "sample_instances": n_inst, "seconds": sec, "setup_s": setup_s,
            "checksum": cs}


def run_reference(args, rank, world):
    if rank != 0:
        return
    prefill = args.prefill if args.prefill >= 0 else PREFILL
    t0 = time.time()
    K, W = args.steps, max(args.warmup, 0)
    res = cpu_reference(K, W, args.cpu_instances, prefill)
    v = res["value"]
    line = {
        "metric": METRIC, "value": v, "unit": "instance-steps/s",
        "impl": "reference", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * res["seconds"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": base_config(args.batch, world),
        "note": "reference CPU path (oracle port; the reference itself needs Chrono/Eigen/HDF5 and cannot be built "
                "here).  A step of this arm is one lock-step of the bounded sample named in cpu_baseline.sample "
                "(%d instances), ms_per_step is its measured duration; one lock-step of all instances_per_gpu "
                "instances would take %.0f ms at this rate" % (res["sample_instances"], 1e3 * args.batch / v),
        "cpu_baseline": res,
        "e2e": {"value": v, "unit": "instance-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class Leg:
    """One ensemble of `batch` instances on this rank's GPU, pre-filled to steady state, with the rotating synthetic
    state buffers on host (pinned) and device."""

    def __init__(self, hc, torch, T, args, dev, local_rank, batch, offset, snap, total_steps):
        self.torch, self.batch, self.offset, self.ens_snap = torch, batch, offset, snap
        self.stream = torch.cuda.Stream(device=dev, priority=-1)
        tiles = batch // 64
        # explicit look-ahead modes below the auto threshold (one CTA per SM): the strong-scaling split
        rad_la = args.rad_lookahead or (2 if tiles < 148 else 0)
        exc_la = 1 if args.no_lookahead else (args.lookahead_mode or (5 if tiles < 148 else 0))
        self.ens = hc.Ensemble(T, batch=batch, device=local_rank, dt_hint=DT, bracket_snap=snap, rad_chunk=args.rad_chunk,
                               exc_chunk=args.exc_chunk, use_graph=not args.no_graph, stream=self.stream.cuda_stream,
                               exc_lookahead=exc_la, rad_kernel=args.rad_kernel, rad_lookahead=rad_la,
                               rad_pass_mode=args.rad_pass_mode)
        from hydrochrono_b200 import shard
        self.seeds = shard.instance_seeds(offset, offset + batch)
        self.duration = total_steps * DT
        self.ens.set_waves_irregular(dt=DT, duration=self.duration, ramp=SEA["ramp"], Hs=SEA["Hs"], Tp=SEA["Tp"],
                                     fmin=SEA["fmin"], fmax=SEA["fmax"], nfreq=SEA["nfreq"], gamma=SEA["gamma"],
                                     seeds=self.seeds)
        self.nf, self.n_eta, le = self.ens.irregular_sizes()
        assert le == [EXC_STEPS] * (DOFS // 6), le
        synth = load_plain("synth")
        amp, om = synth.prescribed_motion(DOFS)
        self.pose_np, self.vel_np = motion_buffers(amp, om, batch, offset)
        # pinned host state, [vel, pose] of a step adjacent in memory (hc_step then uploads them in one copy)
        self.h_state = [torch.from_numpy(np.stack([self.vel_np[i], self.pose_np[i]])).pin_memory() for i in range(NBUF)]
        self.h_vel = [x[0] for x in self.h_state]
        self.h_pose = [x[1] for x in self.h_state]
        self.h_force = torch.empty((batch, DOFS), dtype=torch.float64).pin_memory()
        self.h_pose_np = [x.numpy() for x in self.h_pose]      # views of the pinned buffers, made once
        self.h_vel_np = [x.numpy() for x in self.h_vel]
        self.h_force_np = self.h_force.numpy()
        self.d_pose = [x.to(dev) for x in self.h_pose]
        self.d_vel = [x.to(dev) for x in self.h_vel]
        self.d_force = torch.empty((batch, DOFS), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        self.n = 0
        self.times = step_times(total_steps + 8)

    def dev_step(self):
        n = self.n
        self.ens.step_device(self.times[n], self.d_pose[n % NBUF], self.d_vel[n % NBUF], self.d_force, GVEC)
        self.n = n + 1

    def host_step(self):
        n = self.n
        self.ens.step(self.times[n], self.h_pose_np[n % NBUF], self.h_vel_np[n % NBUF], GVEC, out=self.h_force_np)
        self.n = n + 1

    def align(self, multiple=8):
        """Untimed steps up to the next multiple of the excitation look-ahead block: every timed window starts at
        the same phase of the look-ahead pipeline, whatever K and W are."""
        while self.n % multiple:
            self.dev_step()

    def timed_device(self, K, barrier):
        torch = self.torch
        self.ens.join()
        self.ens.sync()
        barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(self.stream)                          # CUDA events on the launching stream
        for _ in range(K):
            self.dev_step()
        t_enq = time.perf_counter() - t0                 # host time to enqueue the K steps (the GPU runs behind)
        self.ens.join()                                  # ... and every look-ahead pass they launched on side streams
        ev1.record(self.stream)
        self.ens.sync()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t0
        barrier()
        return ev0.elapsed_time(ev1) * 1e-3, t_enq, t_wall

    def timed_host(self, K, barrier):
        torch = self.torch
        self.ens.join()
        self.ens.sync()
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(K):
            self.host_step()
        torch.cuda.synchronize()                         # look-ahead passes of these steps included
        t = time.perf_counter() - t0
        barrier()
        return t


def parity_at_state(leg, orc, cores, n_check, n_steps):
    """The oracle, loaded with the history the GPU holds for `n_check` sampled instances, stepped next to the GPU for
    n_steps more steps (alternating hc_step_device / hc_step).  Reference: src/hydro_forces.cpp:537-691,742-767,
    src/wave_types.cpp:776-844."""
    torch = leg.torch
    B = leg.batch
    sample = sorted(set(int(x) for x in np.linspace(0, B - 1, n_check).round()))
    raw = workload_tables()
    T = orc.Tables(raw)
    insts = oracle_instances(orc, T, leg.seeds[sample], leg.duration, cores)
    n0 = leg.n
    load_history(insts, leg.times, leg.vel_np[:, sample, :], n0, window_rows(raw))
    hist_rows = leg.ens.history_len()
    assert insts[0].history_len() >= hist_rows, (insts[0].history_len(), hist_rows)
    gpu = np.empty((n_steps, len(sample), DOFS))
    for k in range(n_steps):
        if k % 2 == 0:
            leg.dev_step()
            leg.ens.sync()
            gpu[k] = leg.d_force[sample].cpu().numpy()
        else:
            leg.host_step()
            gpu[k] = leg.h_force.numpy()[sample]
    _, _, ref = orc.bench_lockstep(insts, leg.times[n0:n0 + n_steps], leg.pose_np[:, sample, :].copy(),
                                   leg.vel_np[:, sample, :].copy(), buf0=n0 % NBUF, mode=1, gvec=GVEC, want_forces=True)
    scale = np.maximum(np.abs(ref), 1e-3 * np.abs(ref).max(axis=0, keepdims=True))
    rel = np.abs(gpu - ref) / scale
    st = leg.ens.rad_block_stats(reset=False)
    return {"worst_rel": float(rel.max()), "tolerance": 1e-9, "ok": bool(rel.max() <= 1e-9), "instances": len(sample),
            "steps": n_steps, "first_step": n0, "history_rows": hist_rows, "batch": B,
            "what": "per force component and step: |F_gpu - F_oracle| <= 1e-9 max(|F_oracle|, 1e-3 max_t |F_oracle|); "
                    "oracle instances carry the same seeds and the same %d-row velocity history as the GPU's; steps "
                    "alternate hc_step_device / hc_step; bracket_snap %g" % (hist_rows, leg.ens_snap),
            "radiation_block_steps_served_total": st["steps_served"]}


def latency_b1(hc, orc, which):
    """Drop-in case: ONE system (B = 1) through hc_step with host buffers, default options (what the C++ TestHydro
    layer creates), next to the oracle's time for the same step."""
    if True:
        if which == "sphere":
            raw, dt, D, prefill = sphere_tables(), 0.015, 6, 1010
            sea = dict(Hs=2.0, Tp=12.0, gamma=1.0, fmin=0.001, fmax=1.0, nfreq=1000, ramp=60.0)
        else:
            raw, dt, D, prefill = load_plain("synth").rm3_like(), 0.01, 12, 6010
            sea = dict(SEA)
        n_time = 400
        total = prefill + 2 * n_time + 64
        T = hc.Tables.from_raw(raw)
        ens = hc.Ensemble(T, batch=1, device=0, dt_hint=dt)
        kw = dict(dt=dt, duration=total * dt, ramp=sea["ramp"], Hs=sea["Hs"], Tp=sea["Tp"], fmin=sea["fmin"], fmax=sea["fmax"],
                  nfreq=sea["nfreq"], gamma=sea["gamma"])
        ens.set_waves_irregular(seeds=np.array([1], dtype=np.int32), **kw)
        amp, om = load_plain("synth").prescribed_motion(D)
        t = 0.0
        tt, pp, vv = [], [], []
        for n in range(prefill + n_time):
            tt.append(t)
            pp.append((amp * np.sin(om * t))[None, :].copy())
            vv.append((amp * om * np.cos(om * t))[None, :].copy())
            t += dt
        out = np.empty((1, D))
        for n in range(prefill):
            ens.step(tt[n], pp[n], vv[n], GVEC, out=out)
        lat = []
        for n in range(prefill, prefill + n_time):
            t0 = time.perf_counter()
            ens.step(tt[n], pp[n], vv[n], GVEC, out=out)
            lat.append(time.perf_counter() - t0)
        ens.close()
        O = orc.Tables(raw)
        res = {"gpu_us": 1e6 * float(np.median(lat)), "gpu_us_p90": 1e6 * float(np.percentile(lat, 90))}
        for name, mode in (("oracle_serial_us", 0), ("oracle_openmp_lags_us", 1)):
            inst = orc.Instance(O, omp_mode=mode)
            inst.set_irregular(seed=1, **kw)
            for n in range(prefill):
                inst.force(tt[n], pp[n][0], vv[n][0], GVEC)
            cl = []
            for n in range(prefill, prefill + n_time):
                t0 = time.perf_counter()
                inst.force(tt[n], pp[n][0], vv[n][0], GVEC)
                cl.append(time.perf_counter() - t0)
            res[name] = 1e6 * float(np.median(cl))
        res["shape"] = "%s: D = %d, L = %d, Le = %d, dt = %g, history window full" % (
            which, D, len(raw["bodies"][0]["rirf_t"]), ens_le(raw, dt), dt)
        return res


def ens_le(raw, dt):
    te = raw["bodies"][0]["exc_irf_t"]
    return int(np.ceil((te[-1] - te[0]) / dt))


def run_multi(args):
    """`python bench.py --gpus N` WITHOUT torchrun: ONE process drives the N GPUs through the C ABI's multi-device
    handle (hc_multi_*: one host thread + one hc_ensemble per GPU, contiguous shards, the caller's [B][6N] host arrays
    partition without a copy).  Same metric; times are wall clock around the calls + a sync of every shard, since no
    single CUDA stream spans the devices."""
    import torch
    import hydrochrono_b200 as hc
    devs = [int(x) for x in args.multi_devices.split(",")] if args.multi_devices else list(range(args.gpus))
    N = len(devs)
    if torch.cuda.device_count() <= max(devs):
        raise SystemExit("bench.py: devices %s but only %d CUDA devices" % (devs, torch.cuda.device_count()))
    K, W = args.steps, max(args.warmup, 3)
    prefill = args.prefill if args.prefill >= 0 else PREFILL
    snap = 0.0 if args.faithful else SNAP
    total_steps = prefill + 4 * (W + K) + 512
    T = hc.Tables.from_raw(workload_tables())
    amp, om = load_plain("synth").prescribed_motion(DOFS)
    times = step_times(total_steps + 8)

    def leg(B_total, outputs=None):
        per = B_total // N
        small = per // 64 < 148
        m = hc.MultiEnsemble(T, batch=B_total, devices=devs, dt_hint=DT, bracket_snap=snap,
                             rad_lookahead=args.rad_lookahead or (2 if small else 0),
                             exc_lookahead=1 if args.no_lookahead else (args.lookahead_mode or (5 if small else 0)),
                             rad_pass_mode=args.rad_pass_mode)
        m.set_waves_irregular(dt=DT, duration=total_steps * DT, ramp=SEA["ramp"], Hs=SEA["Hs"], Tp=SEA["Tp"], fmin=SEA["fmin"],
                              fmax=SEA["fmax"], nfreq=SEA["nfreq"], gamma=SEA["gamma"],
                              seeds=(1 + np.arange(B_total)).astype(np.int32))
        pose, vel = motion_buffers(amp, om, B_total, 0)
        h_pose = [torch.from_numpy(pose[i]).pin_memory() for i in range(NBUF)]
        h_vel = [torch.from_numpy(vel[i]).pin_memory() for i in range(NBUF)]
        h_force = torch.empty((B_total, DOFS), dtype=torch.float64).pin_memory()
        sh = m.shards()
        d_pose = [[h_pose[i][s["first"]:s["first"] + s["count"]].to("cuda:%d" % s["device"]) for s in sh] for i in range(NBUF)]
        d_vel = [[h_vel[i][s["first"]:s["first"] + s["count"]].to("cuda:%d" % s["device"]) for s in sh] for i in range(NBUF)]
        d_force = [torch.empty((s["count"], DOFS), dtype=torch.float64, device="cuda:%d" % s["device"]) for s in sh]
        n = 0
        for _ in range(prefill + W):
            m.step_device(times[n], d_pose[n % NBUF], d_vel[n % NBUF], d_force, GVEC); n += 1
        while n % 8:
            m.step_device(times[n], d_pose[n % NBUF], d_vel[n % NBUF], d_force, GVEC); n += 1
        m.sync()
        for d in set(devs):
            torch.cuda.synchronize(d)
        t0 = time.perf_counter()
        for _ in range(K):
            m.step_device(times[n], d_pose[n % NBUF], d_vel[n % NBUF], d_force, GVEC); n += 1
        t_enq = time.perf_counter() - t0
        m.sync()
        for d in set(devs):
            torch.cuda.synchronize(d)
        t_dev = time.perf_counter() - t0
        if outputs is not None:
            outputs["forces_device"] = np.concatenate([f.cpu().numpy() for f in d_force])
        for _ in range(W):
            m.step(times[n], h_pose[n % NBUF].numpy(), h_vel[n % NBUF].numpy(), GVEC, out=h_force.numpy()); n += 1
        for d in set(devs):
            torch.cuda.synchronize(d)
        t0 = time.perf_counter()
        for _ in range(K):
            m.step(times[n], h_pose[n % NBUF].numpy(), h_vel[n % NBUF].numpy(), GVEC, out=h_force.numpy()); n += 1
        for d in set(devs):
            torch.cuda.synchronize(d)
        t_e2e = time.perf_counter() - t0
        if outputs is not None:
            outputs["forces_host"] = h_force.numpy().copy()
        # gather check: the instance of global index g on its shard equals a single-device run of the same seed
        comps = m.components()
        res = {"instances_total": B_total, "instances_per_gpu": per, "value": B_total * K / t_dev, "ms_per_step": 1e3 * t_dev / K,
               "enqueue_ms_per_step": 1e3 * t_enq / K,
               "e2e": {"value": B_total * K / t_e2e, "unit": "instance-steps/s", "ms_per_step": 1e3 * t_e2e / K,
                       "h2d_bytes_per_step": 2 * B_total * DOFS * 8, "d2h_bytes_per_step": B_total * DOFS * 8},
               "checksum": float(h_force.numpy()[:, 2].sum()), "components_gathered": [list(c.shape) for c in comps]}
        m.close()
        del d_pose, d_vel, d_force
        torch.cuda.empty_cache()
        return res

    outputs = {} if args.dump_outputs else None
    weak = leg(N * args.batch, outputs)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    strong = None if args.no_strong else leg(TOTAL_INSTANCES)
    line = {"metric": METRIC, "value": weak["value"], "unit": "instance-steps/s", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": weak["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": base_config(args.batch, N), "e2e": weak["e2e"],
            "launcher": "single process, hc_multi_* (one host thread + one hc_ensemble per GPU); value and e2e are wall "
                        "clock around K calls + a synchronize of every device",
            "weak": weak, "strong": dict(strong, scaling="strong") if strong else None,
            "gpu_launches": None, "cpu_baseline": {"value": None, "unit": "instance-steps/s", "cores": None, "kind": "port",
                                                   "sample": "not run at N > 1; see bench.py --impl reference"}}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    select_workload(args.workload)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if (args.gpus > 1 or args.multi_devices) and "WORLD_SIZE" not in os.environ:
        run_multi(args)
        return

    import torch
    import torch.distributed as dist
    import hydrochrono_b200 as hc

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hydro force path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.batch
    K, W = args.steps, max(args.warmup, 3)
    prefill = args.prefill if args.prefill >= 0 else PREFILL
    snap = 0.0 if args.faithful else SNAP
    n_parity = 0 if args.no_parity else 64
    total_steps = prefill + 4 * (W + K) + n_parity + 512
    raw = workload_tables()
    T = hc.Tables.from_raw(raw)

    # ================= weak-scaling leg: B instances per GPU =========================================
    t_setup = time.time()
    leg = Leg(hc, torch, T, args, dev, local_rank, B, rank * B, snap, total_steps)
    ens = leg.ens
    eta_s = ens.profile()["eta_synthesis_seconds"]
    for _ in range(prefill):                          # untimed: fill the radiation history window
        leg.dev_step()
    ens.sync()
    assert ens.history_len() >= min(prefill, RIRF_STEPS - 1), ens.history_len()
    hist_rows = ens.history_len()
    setup_s = time.time() - t_setup

    for _ in range(W):
        leg.dev_step()
    leg.align()
    sampler = ClockSampler(local_rank)              # every rank samples the GPU it drives
    if world > 1 and "HC_BENCH_CLOCK_PERIOD" not in os.environ:
        sampler.period = 0.02                       # eight processes polling NVML every 5 ms is more than the run needs
    launches0 = ens.profile()["kernel_launches"]
    ens.sync()
    barrier()
    sampler.start()
    t_dev, t_enq, t_wall = leg.timed_device(K, barrier)
    outputs = {"forces_device": leg.d_force.cpu().numpy()} if args.dump_outputs else None
    launches = ens.profile()["kernel_launches"] - launches0
    t_dev = max_over_ranks(t_dev)
    t_enq_max = max_over_ranks(t_enq)

    # ---- per-kernel device times (CUDA events on the ensemble's stream; graph off while profiling) ----
    ens.set_profiling(True)
    rb_T = ens.rad_lookahead_steps()                 # steps per radiation look-ahead block (0: per-step kernel)
    nprof = min(max(K // 4, 20), 100) if not rb_T else rb_T * max(2, round(100 / rb_T))   # whole blocks
    for _ in range(3):
        leg.dev_step()
    ens.sync()
    ens.kernel_ms(reset=True)
    ens.rad_block_stats(reset=True)
    for _ in range(nprof):
        leg.dev_step()
    ens.sync()
    kms = ens.kernel_ms(reset=True)
    rb_stats = ens.rad_block_stats(reset=True)
    rb_on = bool(rb_T) and rb_stats["steps_served"] == nprof
    ens.set_profiling(False)

    # ---- end-to-end leg (host buffers through hc_step) -----------------------------------------------
    for _ in range(W):
        leg.host_step()
    t_e2e = max_over_ranks(leg.timed_host(K, barrier))
    if outputs is not None:
        outputs["forces_host"] = leg.h_force.numpy().copy()
        dump_outputs(args.dump_outputs, {k + (".rank%d" % rank if world > 1 else ""): v for k, v in outputs.items()})
    checksum = float(leg.h_force.numpy()[:, 2].sum())
    # the final result gather of the north star (the only inter-GPU traffic of the whole run besides the timing
    # reductions): every rank's heave forces of the last step, in global instance order, on rank 0
    gathered = None
    if world > 1:
        from hydrochrono_b200 import shard
        full = shard.gather_results(leg.h_force.numpy()[:, 2:3].copy(), world * B, world, rank, dist=dist, device=dev)
        if rank == 0:
            gathered = {"instances": int(full.shape[0]), "checksum": float(full.sum()),
                        "rank0_block_matches": bool(np.array_equal(full[:B, 0], leg.h_force.numpy()[:, 2]))}
    mine = sampler.stop()          # sampled from the start of the device-resident leg to the end of the end-to-end leg
    # over the ranks: the slowest GPU's median and minimum SM clock, any throttle reason seen anywhere
    vec = torch.tensor(mine if mine else [0.0] * 8, dtype=torch.float64, device=dev)
    lo, hi = vec.clone(), vec.clone()
    if world > 1:
        if not mine:
            lo[:2] = float("inf")
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        tot = vec[7:8].clone()
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        nsamp = float(tot.item())
    else:
        nsamp = float(vec[7].item())
    lo, hi = lo.tolist(), hi.tolist()
    if nsamp > 0 and np.isfinite(lo[0]):
        clocks = {"sm_mhz": lo[0], "sm_min_mhz": lo[1], "sm_max_mhz": hi[2],
                  "reasons": [nm for nm, f in zip(ClockSampler.NAMES, hi[3:7]) if f > 0], "samples": int(nsamp), "gpus": world,
                  "source": "NVML, one sampling thread per rank (5 ms period at N = 1, 20 ms at N > 1) from the start of the device-resident timed "
                            "region to the end of the end-to-end timed region; sm_mhz = the slowest GPU's median"}
    else:
        clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "samples": 0, "gpus": world}

    # ---- parity at the benchmarked state ----------------------------------------------------------------
    parity = None
    if not args.no_parity:
        orc, cores = oracle_with_all_cores()
        parity = parity_at_state(leg, orc, max(1, cores // max(1, world)), 8 if world == 1 else 4, n_parity)
        parity["worst_rel"] = max_over_ranks(parity["worst_rel"])
        parity["ok"] = parity["worst_rel"] <= parity["tolerance"]
        parity["instances"] *= world
        lk = ens.lookahead_state()
        parity["lookahead_armed"] = lk

    # ---- the same device-resident leg with bit-faithful bracketing (bracket_snap = 0), short ----------------
    faithful = None
    if snap > 0 and not args.no_faithful_leg:
        ens.set_bracket_snap(0.0)
        kf = min(max(50, K // 5), 200)
        for _ in range(W):
            leg.dev_step()
        t_f, _, _ = leg.timed_device(kf, barrier)
        t_f = max_over_ranks(t_f)
        faithful = {"value": world * B * kf / t_f, "unit": "instance-steps/s", "steps": kf, "ms_per_step": 1e3 * t_f / kf,
                    "note": "bracket_snap = 0, the C-ABI default: every convolution query is bracketed with the "
                            "reference's == / lerp logic, a ~1e-9-weight second history row is read where the query "
                            "misses a sample by floating-point noise; served by the per-step kernels"}
        ens.set_bracket_snap(snap)

    fp64_peak = hc.measure_fp64_peak(local_rank) if rank == 0 else None
    mma_peak = hc.measure_fp64_mma_peak(local_rank) if rank == 0 else None
    weak_hist_gb = 8e-9 * DOFS * B * ens.history_len()
    weak_eta_gb = 8e-9 * B * leg.n_eta
    nf, n_eta = leg.nf, leg.n_eta

    # ================= strong-scaling leg: TOTAL_INSTANCES over the N GPUs (north star) =====================
    strong = None
    if world > 1 and not args.no_strong and TOTAL_INSTANCES % world == 0:
        del leg, ens
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        Bs = TOTAL_INSTANCES // world
        sl = Leg(hc, torch, T, args, dev, local_rank, Bs, rank * Bs, snap, total_steps)
        for _ in range(prefill):
            sl.dev_step()
        sl.ens.sync()
        Ks = max(K, 48)
        for _ in range(W):
            sl.dev_step()
        sl.align()
        s_dev, s_enq, _ = sl.timed_device(Ks, barrier)
        s_dev, s_enq = max_over_ranks(s_dev), max_over_ranks(s_enq)
        for _ in range(W):
            sl.host_step()
        s_e2e = max_over_ranks(sl.timed_host(Ks, barrier))
        sp = None
        if not args.no_parity:
            sp = parity_at_state(sl, orc, max(1, cores // world), 2, 32)
            sp = max_over_ranks(sp["worst_rel"])
        strong = {"scaling": "strong", "instances_total": TOTAL_INSTANCES, "instances_per_gpu": Bs, "steps": Ks,
                  "value": TOTAL_INSTANCES * Ks / s_dev, "ms_per_step": 1e3 * s_dev / Ks,
                  "enqueue_ms_per_step": 1e3 * s_enq / Ks,
                  "e2e": {"value": TOTAL_INSTANCES * Ks / s_e2e, "ms_per_step": 1e3 * s_e2e / Ks,
                          "h2d_bytes_per_step": 2 * Bs * DOFS * 8, "d2h_bytes_per_step": Bs * DOFS * 8},
                  "unit": "instance-steps/s", "parity_worst_rel": sp,
                  "radiation_lookahead_steps": sl.ens.rad_lookahead_steps(),
                  "limiter": "per-step latency, not bandwidth or flops: at %d instances per GPU a step is ~%.0f us of "
                             "tensor work; device-resident stepping is bound by max(that, host enqueue %.0f us/step), "
                             "the host-buffer path by the serial chain H2D -> k_step -> D2H -> host wake-up every step "
                             "(the integrator stays on the CPU, src/hydro_forces.cpp:742-767: one evaluation per time "
                             "value)" % (Bs, 229.0 * Bs / 16384, 1e3 * s_enq / Ks)}
        del sl

    if rank == 0:
        peak, peak_src = hbm_peak()
        # distinct history rows touched per step: one per lag with exact hits / snapping, up to two otherwise
        rows = RIRF_STEPS if snap > 0 else min(2 * RIRF_STEPS, hist_rows)
        rad_bytes = B * (8 * DOFS * rows + 8 * DOFS * 3) + 8 * DOFS * DOFS * RIRF_STEPS
        exc_bytes = B * 8 * (EXC_STEPS + 1) + 8 * (DOFS + 2) * EXC_STEPS
        ach = rad_bytes / (kms["radiation"] * 1e-3) / 1e9
        ach_exc = exc_bytes / (kms["excitation"] * 1e-3) / 1e9 if kms["excitation"] > 0 else None
        exc_flops = 2.0 * DOFS * EXC_STEPS * B                      # per step: 2 * D * Le per instance
        rad_flops = 2.0 * DOFS * DOFS * RIRF_STEPS * B
        exc_tf = exc_flops / (kms["excitation"] * 1e-3) / 1e12 if kms["excitation"] > 0 else None
        rad_tf = rad_flops / (kms["radiation"] * 1e-3) / 1e12
        traffic = ncu_traffic() if WORKLOAD == "rm3_irregular_ensemble" else None
        value = world * B * K / t_dev
        step_bytes = rad_bytes + (exc_bytes if args.no_lookahead else (B * 8 * (EXC_STEPS + 8) // 8))
        step_flops = rad_flops + exc_flops
        exc_mma = (not args.no_lookahead) and args.lookahead_mode in (0, 4, 5)
        exc_peak = mma_peak if exc_mma else fp64_peak
        rad_roof = {"bound": "hbm", "kernel": ("k_radiation_mma12 (DMMA m8n8k4)" if (DOFS == 12 and args.rad_kernel == 2)
                                               else "k_radiation_hybrid12 (DMMA + DFMA)" if (DOFS == 12 and args.rad_kernel == 3)
                                               else "k_radiation<%d>" % DOFS), "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": (traffic or {}).get("radiation_dram_bytes_per_launch"),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": rad_bytes,
                    "kernel_ms": kms["radiation"],
                    "fp64_tflops": rad_tf, "fp64_peak_tflops": fp64_peak,
                    "fp64_frac": rad_tf / fp64_peak if fp64_peak else None}
        if rb_on:
            # k_rad_block<12>: one launch = the resident rows' share of rb_T steps; lags served by the block at block
            # step j: (L - 1) - floor(j / m)  (the younger lags belong to k_step)
            m = rb_T // 8
            lag_steps = sum((RIRF_STEPS - 1) - (j // m) for j in range(rb_T))
            blk_flops = 2.0 * DOFS * DOFS * lag_steps * B
            blk_ms = rb_stats["avg_ms"]
            blk_tf = blk_flops / (blk_ms * 1e-3) / 1e12
            hist_bytes = 8.0 * DOFS * B * m * (RIRF_STEPS - 1)         # every resident row once per block
            rad_roof = {"bound": "tensor", "kernel": "k_rad_block<%d> (radiation look-ahead: %d steps per pass over the "
                                                     "history, FP64 tensor cores, DMMA m8n8k4)" % (DOFS, rb_T),
                        "achieved": blk_tf, "peak": mma_peak, "unit": "TFLOP/s", "frac": blk_tf / mma_peak,
                        "traffic": (traffic or {}).get("rad_block_dram_bytes_per_launch"),
                        "peak_source": "FP64 tensor-core peak measured in this run (hc_measure_fp64_mma_peak, DMMA m8n8k4 "
                                       "loop); MEASURED_PEAKS.json holds no FP64 figure (B200 nominal: 40 TFLOP/s)",
                        "algorithmic_flops_per_launch": blk_flops, "launch_ms": blk_ms, "steps_per_launch": rb_T,
                        "history_bytes_per_launch": hist_bytes,
                        "kernel_ms": kms["radiation"],
                        "kernel_ms_note": "launch_ms = one whole pass = the sum of its per-step slices, each timed with "
                                          "CUDA events on its stream in the profiling pass; radiation per step = "
                                          "launch_ms / %d + k_step<%d>" % (rb_T, DOFS),
                        "hbm_view": {"algorithmic_bytes_per_step": rad_bytes, "gbs": ach, "hbm_peak": peak, "frac": ach / peak,
                                     "note": "SURVEY 8(d) bytes of the per-step formulation over the measured radiation "
                                             "time per step: the block pass reads each history row once per %d steps, "
                                             "so the per-step HBM roofline no longer binds (frac > 1); "
                                             "--rad-lookahead 1 measures the per-step kernel k_radiation<%d> against "
                                             "that roofline" % (rb_T, DOFS)}}
            step_bytes = hist_bytes / rb_T + (B * 8 * (EXC_STEPS + 8) // 8)
        step_s = t_dev / K
        e2e = world * B * K / t_e2e
        line = {
            "metric": METRIC, "value": value, "unit": "instance-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * t_dev / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": base_config(B, world),
            "e2e": {"value": e2e, "unit": "instance-steps/s", "h2d_bytes_per_step": 2 * B * DOFS * 8,
                    "d2h_bytes_per_step": B * DOFS * 8, "ms_per_step": 1e3 * t_e2e / K},
            "gpu_launches": int(launches) * world,
            "clocks": clocks,
            "parity": parity,
            "faithful_bracketing": faithful,
            "strong": strong,
            "run": {"bracket_snap": snap, "cuda_graph": not args.no_graph,
                    "eta_samples": n_eta, "history_rows": hist_rows,
                    "resident_gb": {"history": weak_hist_gb, "eta": weak_eta_gb},
                    "excitation_lookahead_steps": 1 if args.no_lookahead else 8,
                    "radiation_lookahead_steps": rb_T if rb_on else 1,
                    "radiation_pass_mode": args.rad_pass_mode or 1,
                    "excitation_lookahead_mode": ("off" if args.no_lookahead else
                                                  {0: "background stream, DMMA", 2: "in-stream", 3: "background stream",
                                                   4: "in-stream, DMMA", 5: "background stream, DMMA"}
                                                  .get(args.lookahead_mode, str(args.lookahead_mode))),
                    "enqueue_ms_per_step": 1e3 * t_enq_max / K,
                    "timing": "value: CUDA events on the ensemble's stream, each recorded after hc_ensemble_join, around K "
                              "hc_step_device calls that start on an excitation-block boundary (wall %.4f s, of which "
                              "%.4f s to enqueue them); e2e: wall clock around K synchronous hc_step calls + device "
                              "synchronize; per-kernel ms: CUDA events inside the library on the kernels' own streams"
                              % (t_wall, t_enq),
                    "launches_before_timed_region": int(launches0)},
            "roofline": {**rad_roof,
                         "excitation": ({"kernel": ("k_exc_block_mma<%d> (look-ahead, 8 steps per eta pass, DMMA m8n8k4)" % DOFS
                                                    if args.lookahead_mode in (0, 4, 5) else
                                                    "k_exc_block<%d> (look-ahead, 8 steps per eta pass)" % DOFS), "bound": "fp64",
                                         "achieved": exc_tf, "peak": exc_peak, "unit": "TFLOP/s",
                                         "frac": exc_tf / exc_peak if (exc_tf and exc_peak) else None,
                                         "peak_source": "measured in this run (%s)" % ("hc_measure_fp64_mma_peak, DMMA loop" if exc_mma
                                                                                        else "hc_measure_fp64_peak, DFMA loop"),
                                         "flops_per_step": exc_flops, "kernel_ms_per_step": kms["excitation"],
                                         "traffic": (traffic or {}).get("exc_block_dram_bytes_per_launch"),
                                         "traffic_note": "dram bytes per k_exc_block launch (one launch per 8 steps)"}
                                        if not args.no_lookahead else
                                        {"kernel": "k_excitation<%d>" % DOFS, "bound": "hbm", "achieved": ach_exc, "peak": peak,
                                         "unit": "GB/s", "frac": (ach_exc / peak) if ach_exc else None,
                                         "algorithmic_bytes_per_launch": exc_bytes, "kernel_ms": kms["excitation"],
                                         "traffic": (traffic or {}).get("excitation_dram_bytes_per_launch")})},
            "step_roofline": {"hbm_gbs": step_bytes / step_s / 1e9, "hbm_frac": step_bytes / step_s / 1e9 / peak,
                              "fp64_tflops": step_flops / step_s / 1e12,
                              "fp64_frac": (step_flops / step_s / 1e12 / max(fp64_peak, mma_peak)) if fp64_peak else None,
                              "fp64_peaks_tflops": {"fma_pipe": fp64_peak, "tensor_dmma": mma_peak},
                              "note": "whole step (all kernels, overlapped): algorithmic bytes and flops per step over "
                                      "the measured step time; the step needs both resources at once"},
            "kernel_ms": kms,
            "kernel_ms_note": "isolated kernel durations (the profiling pass runs every kernel back-to-back in one "
                              "stream).  excitation = look-ahead block time / 8.  With the radiation look-ahead on: "
                              "radiation = this step's slice of the next block's k_rad_block<D> pass + k_step<D> (append, "
                              "block partials, rows appended since the snapshot AND finalize, fused), finalize ~ 0.  "
                              "In the timed region the excitation block of the next 8 steps and the slices of the next "
                              "radiation block run on side streams underneath the per-step kernels and the host <-> "
                              "device copies, so ms_per_step < sum(kernel_ms)",
            "setup": {"eta_synthesis_s": eta_s, "setup_and_prefill_s": setup_s},
            "checksum": checksum,
            "gathered": gathered,
        }
        if world == 1 and not args.no_b1 and WORKLOAD == "rm3_irregular_ensemble":
            try:
                orc_b1, _ = oracle_with_all_cores()
                line["latency_b1_us"] = {"rm3": latency_b1(hc, orc_b1, "rm3"), "sphere": latency_b1(hc, orc_b1, "sphere"),
                                         "what": "median wall time of one hc_step call (host buffers in, forces out, "
                                                 "synchronous) at B = 1 with the C-ABI's default options, irregular "
                                                 "waves, full history window; oracle_* = the CPU restatement's time for "
                                                 "the same step, serial and with the reference's OpenMP loop over lags"}
            except Exception as ex:
                line["latency_b1_us"] = {"error": repr(ex)}
        if args.no_cpu or world > 1:
            line["cpu_baseline"] = {"value": None, "unit": "instance-steps/s", "cores": None, "kind": "port",
                                    "sample": "not run (%s): the CPU leg runs on rank 0 at N = 1 only; see the reference "
                                              "arm (bench.py --impl reference)" % ("--no-cpu" if args.no_cpu else "N > 1")}
        else:
            # the CPU leg runs in a fresh interpreter (no torch / CUDA threads competing for the cores, no product
            # library mapped): the same code path as `bench.py --impl reference`
            try:
                env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS")}
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", WORKLOAD,
                                      "--cpu-instances", str(args.cpu_instances), "--steps", str(max(K if K <= 100 else 100, 10)),
                                      "--warmup", "3", "--prefill", str(prefill), "--batch", str(B)],
                                     capture_output=True, text=True, timeout=900, env=env)
                line["cpu_baseline"] = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as ex:   # never lose the GPU line because the CPU leg failed
                line["cpu_baseline"] = {"value": None, "unit": "instance-steps/s", "cores": None, "kind": "port",
                                        "sample": "cpu leg failed: %r" % (ex,)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
