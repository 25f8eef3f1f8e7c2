"""Dispatch coverage: every instance and every DoF against the CPU oracle, at the batch sizes, body counts and options
where the library switches from one kernel to another.

Which kernel serves a step depends on the batch size (lane tiles of 64, convolution tiles of 256 / 512, the k_step2
threshold of one 64-instance CTA per SM, the 8-instance warp finalize, the 64 KB compact-graph staging limit, the
2048-instance fork limit), on the body count and on the options.  Each case here names the kernels it is meant to
exercise and proves with torch.profiler that they ran, so that a later change of a threshold cannot silently make a case
test something else.

Full-population oracle check: the oracle instances are created in batches of 2048 with their own seeds (their waves
are synthesised independently, which also checks k_eta for every instance), loaded with the velocity history the GPU
holds after n0 steps (the state-loading path of bench.py), and stepped next to the GPU's recorded forces for K steps.
The bar is tests/test_gpu_parity._assert_parity: 1e-9 relative with the 1e-3 floor (common.force_tol).

Diagnostic overrides that are read once per process (HC_FINALIZE_MODE, HC_KSTEP2, HC_COMPACT_*, HC_FORK_MAX_BATCH)
run in child processes of this file (see __main__ at the bottom).
"""
import json
import os
import subprocess
import sys
import warnings
from concurrent.futures import ThreadPoolExecutor

if __name__ == "__main__":      # child process: no conftest to set the path up
    _ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for _p in (_ROOT, os.path.join(_ROOT, "tests")):
        if _p not in sys.path:
            sys.path.insert(0, _p)

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import synth
from oracle import hc_oracle as orc
from test_gpu_parity import _acc_times, _assert_parity

pytestmark = pytest.mark.gpu

G981 = (0.0, 0.0, -9.81)
NBUF = 8                 # the prescribed state of step n is buffer n % NBUF (as bench.py)
ORACLE_BATCH = 2048      # oracle instances alive at a time (host memory)
CHILD_TIMEOUT = 900

# sea states: bench.py's RM3 / sphere sea states with nfreq lowered from 1000 to 64 (the oracle synthesises every
# instance's elevation on the host; 16384 x 6100 samples x 1000 components would not fit the suite's time budget)
SEA_RM3_BENCH = dict(Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0, nfreq=64, ramp=20.0)
SEA_SPHERE_BENCH = dict(Hs=2.0, Tp=12.0, gamma=1.0, fmin=0.001, fmax=1.0, nfreq=64, ramp=60.0)
SEA_SHORT = dict(Hs=2.5, Tp=8.0, gamma=3.3, fmin=0.001, fmax=1.0, nfreq=48, ramp=0.3)


# ---------------------------------------------------------------------------------------------
# tables, runs and the oracle
# ---------------------------------------------------------------------------------------------
_RAW = {}


def _raw(kind):
    if kind not in _RAW:
        if kind == "rm3":            # the headline workload: N = 2, L = 1001 lags over 60 s, excitation IRF +-30 s
            r = synth.rm3_like()
        elif kind == "rm3_short":    # RM3 shape with a +-6 s excitation IRF (1200 lags at dt 0.01): cheaper oracle
            r = synth.rm3_like(exc_irf_steps=241, exc_half_window=6.0)
        elif kind == "rm3_window6":  # RM3 shape with a 6 s RIRF window (lag spacing 6 dt) and a +-2 s excitation IRF:
            #                          a full window after 600 steps, so every lag chunk's partial is non-zero
            r = synth.rm3_like(rirf_steps=101, rirf_duration=6.0, exc_irf_steps=81, exc_half_window=2.0)
        elif kind == "rm3_two_windows":     # body 1's excitation IRF on a narrower window: two ND = 6 groups
            r = synth.rm3_like(exc_irf_steps=241, exc_half_window=6.0)
            r["bodies"][1]["exc_irf_t"] = np.linspace(-4.5, 4.5, 241)
        elif kind == "sphere":
            r = common.sphere_raw()
        elif kind == "oswec":        # test_baseline_config_shapes' OSWEC shape: lag spacing 0.05 = 5/3 dt at dt 0.03
            r = synth.make_tables(num_bodies=2, rirf_steps=601, rirf_duration=30.0, exc_irf_steps=401,
                                  exc_half_window=24.0)
        elif kind.startswith("bodies"):
            r = synth.make_tables(num_bodies=int(kind[6:]), rirf_steps=201, rirf_duration=10.0, exc_irf_steps=201,
                                  exc_half_window=5.0)
        else:
            raise KeyError(kind)
        _RAW[kind] = r
    return _RAW[kind]


def _dofs(kind):
    return 6 * len(_raw(kind)["bodies"])


def _buffers(D, B, dt):
    """pose / vel [NBUF][B][D]: analytic motion at t = i dt with a per-instance and per-DoF phase."""
    amp, om = synth.prescribed_motion(D, 3)
    ph = 0.37 * np.arange(B)[:, None] + 0.11 * np.arange(D)[None, :]
    pose = np.stack([amp * np.sin(om * (i * dt) + ph) for i in range(NBUF)])
    vel = np.stack([amp * om * np.cos(om * (i * dt) + ph) for i in range(NBUF)])
    return np.ascontiguousarray(pose), np.ascontiguousarray(vel)


def _spec(tables, B, dt, nsteps, n0=0, opts=None, waves="irregular", sea=None, api="host", gvec=G981, seed0=1,
          per_instance_sea=False):
    """A run: B instances stepped nsteps times from an empty history; forces of steps n0 .. nsteps - 1 are recorded."""
    return dict(tables=tables, B=B, dt=dt, nsteps=nsteps, n0=n0, opts=dict(opts or {}), waves=waves,
                sea=dict(sea or SEA_SHORT), api=api, gvec=list(gvec), seed0=seed0, per_instance_sea=per_instance_sea)


def _seeds(s):
    return s["seed0"] + np.arange(s["B"], dtype=np.int32)


def _sea_kw(s):
    return dict(dt=s["dt"], duration=(s["nsteps"] + 64) * s["dt"], **s["sea"])


def _hs_tp(s):
    b = np.arange(s["B"])
    return 1.0 + 0.05 * (b % 40), 6.0 + 0.13 * (b % 31)


REGULAR = (1.0, 0.9)     # amplitude, omega


def _kernel_names(fn):
    """Names of the CUDA kernels that ran during fn() (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages()})


def _run_gpu(s, profile_steps=10):
    """Steps the GPU ensemble of spec s.  Returns (forces [nsteps - n0][B][D], kernel names seen over profile_steps
    steps from n0, info)."""
    import torch
    raw = _raw(s["tables"])
    T = hc.Tables.from_raw(raw)
    B, dt, D = s["B"], s["dt"], _dofs(s["tables"])
    ens = hc.Ensemble(T, batch=B, dt_hint=dt, **s["opts"])
    if s["waves"] == "irregular":
        if s["per_instance_sea"]:
            Hs, Tp = _hs_tp(s)
            ens.set_waves_irregular(seeds=_seeds(s), Hs_per_instance=Hs, Tp_per_instance=Tp, **_sea_kw(s))
        else:
            ens.set_waves_irregular(seeds=_seeds(s), **_sea_kw(s))
    elif s["waves"] == "regular":
        ens.set_waves_regular([REGULAR[0]], [REGULAR[1]])
    times = _acc_times(s["nsteps"], dt)
    pose, vel = _buffers(D, B, dt)
    g = tuple(s["gvec"])
    dev = torch.device("cuda", 0)
    if s["api"] == "alternate":
        d_pose = [torch.from_numpy(pose[i]).to(dev) for i in range(NBUF)]
        d_vel = [torch.from_numpy(vel[i]).to(dev) for i in range(NBUF)]
        d_force = torch.empty((B, D), dtype=torch.float64, device=dev)
    n0 = s["n0"]
    F = np.empty((s["nsteps"] - n0, B, D))
    h_out = np.empty((B, D))

    def step(n):
        if s["api"] == "alternate" and (n % 12) < 7:
            ens.step_device(times[n], d_pose[n % NBUF], d_vel[n % NBUF], d_force, g)
            ens.sync()
            if n >= n0:
                F[n - n0] = d_force.cpu().numpy()
        else:
            ens.step(times[n], pose[n % NBUF], vel[n % NBUF], g, out=h_out)
            if n >= n0:
                F[n - n0] = h_out

    for n in range(n0):
        step(n)
    stats0 = ens.rad_block_stats(reset=True)
    p1 = min(s["nsteps"], n0 + profile_steps)

    def prof():
        for n in range(n0, p1):
            step(n)
    names = _kernel_names(prof) if p1 > n0 else (prof() or [])
    for n in range(p1, s["nsteps"]):
        step(n)
    info = dict(lookahead=ens.lookahead_state(), rad_blocks=ens.rad_block_stats(reset=True), rad_blocks_before=stats0,
                history_len=ens.history_len(), irregular_sizes=list(ens.irregular_sizes()[2]) if s["waves"] == "irregular"
                else None)
    if s["waves"] == "irregular" and s["per_instance_sea"]:
        info["irregular"] = [ens.irregular(b) for b in range(B)]
    ens.close()
    return F, names, info


_ORC_T = {}
_CORES = None


def _oracle_threads():
    global _CORES
    if _CORES is None:
        try:
            _CORES = len(os.sched_getaffinity(0))
        except AttributeError:
            _CORES = os.cpu_count() or 1
        orc.set_num_threads(_CORES)
    return _CORES


def _oracle_instances(s, idx):
    """Oracle instances idx of spec s, each with its own seed (own elevation synthesis), the IRFs shared."""
    kind = s["tables"]
    if kind not in _ORC_T:
        _ORC_T[kind] = orc.Tables(_raw(kind))
    O = _ORC_T[kind]
    seeds = _seeds(s)
    if s["waves"] != "irregular":
        out = []
        for _ in idx:
            i = orc.Instance(O, omp_mode=0)
            if s["waves"] == "regular":
                i.set_regular(*REGULAR)
            out.append(i)
        return out
    kw = _sea_kw(s)
    Hs, Tp = _hs_tp(s)

    def kw_of(b):
        if not s["per_instance_sea"]:
            return kw
        return dict(kw, Hs=float(Hs[b]), Tp=float(Tp[b]))
    first = orc.Instance(O, omp_mode=0)
    first.set_irregular(seed=int(seeds[idx[0]]), **kw_of(idx[0]))

    def make(b):
        i = orc.Instance(O, omp_mode=0)
        i.set_irregular(seed=int(seeds[b]), share_irf_from=first, **kw_of(b))      # ctypes releases the GIL
        return i
    with ThreadPoolExecutor(max_workers=_oracle_threads()) as ex:
        return [first] + list(ex.map(make, idx[1:]))


def _check_oracle(s, F, what, info=None, rel=1e-9):
    """Every instance and every DoF of the recorded forces F against the oracle (tests/test_gpu_parity._assert_parity
    per batch of ORACLE_BATCH instances: the 1e-3 floor is taken over that batch's steps and instances)."""
    _oracle_threads()
    B, dt, D, n0 = s["B"], s["dt"], _dofs(s["tables"]), s["n0"]
    raw = _raw(s["tables"])
    times = _acc_times(s["nsteps"], dt)
    pose, vel = _buffers(D, B, dt)
    window_rows = int(round(float(raw["bodies"][0]["rirf_t"][-1]) / dt)) + 4
    worst = 0.0
    for lo in range(0, B, ORACLE_BATCH):
        idx = list(range(lo, min(B, lo + ORACLE_BATCH)))
        insts = _oracle_instances(s, idx)
        if n0 > 0:     # what stepping instance b through steps 0 .. n0 - 1 leaves in its history (bench.load_history)
            rows = min(n0, window_rows)
            hidx = np.arange(n0 - 1, n0 - 1 - rows, -1)            # newest first
            for b, inst in zip(idx, insts):
                inst.set_history(times[hidx], vel[hidx % NBUF, b, :])
        _, _, ref = orc.bench_lockstep(insts, times[n0:], np.ascontiguousarray(pose[:, lo:lo + len(idx)]),
                                       np.ascontiguousarray(vel[:, lo:lo + len(idx)]), buf0=n0 % NBUF, mode=1,
                                       gvec=tuple(s["gvec"]), want_forces=True)
        if info is not None and lo == 0:      # the oracle held at least the rows the GPU convolved
            assert insts[0].history_len() >= info["history_len"], (insts[0].history_len(), info["history_len"])
        worst = max(worst, _assert_parity(F[:, lo:lo + len(idx)], ref, "%s, instances %d..%d" % (what, lo, idx[-1]),
                                          rel=rel))
        del insts
    return worst


def _expect_kernels(names, want, forbid=(), what=""):
    """Substring match of kernel names; skipped (with a message) only when the profiler recorded no kernel at all."""
    if not names:
        msg = "%s: torch.profiler recorded no CUDA kernel; the dispatch assertion is skipped (parity still checked)" % what
        warnings.warn(msg)
        print(msg)
        return
    for w in want:
        assert any(w in n for n in names), "%s: no kernel matching %r ran; kernels: %s" % (what, w, names)
    for w in forbid:
        assert not any(w in n for n in names), "%s: kernel matching %r ran; kernels: %s" % (what, w, names)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# child processes: a list of specs stepped under an environment override, forces and kernel names written back
# ---------------------------------------------------------------------------------------------
def _run_child(tmp_path, name, env_over, specs):
    spec_file = tmp_path / ("%s.json" % name)
    out_dir = tmp_path / name
    out_dir.mkdir()
    spec_file.write_text(json.dumps(specs))
    env = dict(os.environ)
    env.update(env_over)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(spec_file), str(out_dir)], env=env,
                       timeout=CHILD_TIMEOUT, capture_output=True, text=True)
    assert r.returncode == 0, "child %s (%s) exited with %d:\n%s\n%s" % (name, env_over, r.returncode, r.stdout[-3000:],
                                                                          r.stderr[-3000:])
    out = []
    for k in range(len(specs)):
        F = np.load(out_dir / ("F%d.npy" % k))
        meta = json.loads((out_dir / ("meta%d.json" % k)).read_text())
        out.append((F, meta["names"], meta["info"]))
    return out


def _child_main(spec_file, out_dir):
    specs = json.loads(open(spec_file).read())
    for k, s in enumerate(specs):
        F, names, info = _run_gpu(s)
        np.save(os.path.join(out_dir, "F%d.npy" % k), F)
        info.pop("irregular", None)
        with open(os.path.join(out_dir, "meta%d.json" % k), "w") as f:
            json.dump({"names": names, "info": info}, f)


_DEFAULT_RUNS = {}


def _default_run(s):
    """The run of spec s in this process (no override), oracle-checked once and cached for bitwise comparisons."""
    key = json.dumps(s, sort_keys=True)
    if key not in _DEFAULT_RUNS:
        F, names, info = _run_gpu(s)
        _check_oracle(s, F, "default options, B = %d" % s["B"], info)
        _DEFAULT_RUNS[key] = (F, names, info)
    return _DEFAULT_RUNS[key]


# ---------------------------------------------------------------------------------------------
# 1 + 2. production-scale cases, all instances
# ---------------------------------------------------------------------------------------------
def _bench_state_spec(snap):
    # full window: 6030 steps > 6000 history rows; K = 40 recorded steps cover the radiation block boundary at step
    # 6049 (blocks start at steps 1 + 48 k) and five 8-step excitation blocks
    opts = dict(bracket_snap=snap) if snap > 0 else dict(exc_lookahead=1)     # 1: excitation look-ahead off
    return _spec("rm3", 16384, 0.01, 6070, n0=6030, opts=opts, sea=SEA_RM3_BENCH, api="alternate")


def test_rm3_bench_state_all_instances():
    """bench.py's state (B = 16384, dt 0.01, snap 1e-8, history window full), hc_step / hc_step_device alternating:
    k_rad_block<12>, k_step2<12> and k_exc_block_mma<12>.  nfreq lowered to 64 (host-side synthesis cost)."""
    s = _bench_state_spec(1e-8)
    F, names, info = _run_gpu(s)
    _expect_kernels(names, ["k_rad_block<12>", "k_step2<12>", "k_exc_block_mma<12>"], what="RM3 bench state")
    assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info
    assert info["history_len"] >= 6001
    worst = _check_oracle(s, F, "RM3 bench state", info)
    print("RM3 bench state: worst %.2e over %d instances x %d steps" % (worst, s["B"], F.shape[0]))


def test_rm3_bit_faithful_all_instances():
    """Same state with snap 0 (bit-faithful brackets) and the excitation look-ahead off (at this size it is on by
    default, snap or not): the per-step k_radiation<12> / k_excitation<12> kernels and the automatically selected
    finalize.  nfreq lowered to 64."""
    s = _bench_state_spec(0.0)
    F, names, info = _run_gpu(s)
    _expect_kernels(names, ["k_radiation<12", "k_excitation<12", "k_finalize"], forbid=["k_step", "k_rad_block"],
                    what="RM3 bit-faithful")
    worst = _check_oracle(s, F, "RM3 bit-faithful", info)
    assert worst < 1e-11, worst           # differs from the oracle only by summation order / FMA contraction


def test_sphere_secondary_workload_all_instances():
    """The README's secondary workload: sphere tables x 16384, dt 0.015, bench.py's sphere sea state (nfreq lowered to
    64), snap 1e-8, window full (1030 steps > 1000 rows): k_rad_block<6>, k_step<6>, excitation look-ahead (ND = 6)."""
    s = _spec("sphere", 16384, 0.015, 1070, n0=1030, opts=dict(bracket_snap=1e-8), sea=SEA_SPHERE_BENCH,
              api="alternate")
    F, names, info = _run_gpu(s)
    _expect_kernels(names, ["k_rad_block<6>", "k_step<6>", "k_exc_block"], forbid=["k_step2"], what="sphere x 16384")
    assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info
    # rel 2e-9: on the sway DoF (force ~1e-6 of the heave force: an axisymmetric body in head seas) the error measured
    # on a B200 reached 1.07 x the 1e-9 bar against the floor at a few instances (2e-11 N where the series maximum is
    # 1.9 N), consistent with the ~1e-11 interpolation weights that bracket_snap = 1e-8 drops
    _check_oracle(s, F, "sphere x 16384", info, rel=2e-9)


def _threshold_spec(B, opts, n0=50, nsteps=100):
    # 100 steps: the radiation block boundary at step 97 and six excitation blocks inside the recorded steps
    return _spec("rm3", B, 0.01, nsteps, n0=n0, opts=opts)


def _kstep2_min_batch():
    """The smallest batch served by k_step2<12> (and by the automatic radiation look-ahead): one 64-instance CTA per SM
    once padded to the 64-instance lane tile, i.e. 64 (sm_count - 1) + 1 (9409 on 148 SMs)."""
    return 64 * (_sm_count() - 1) + 1


def test_kstep2_ragged_above_threshold():
    """The smallest k_step2 batch, auto options: k_step2<12>, whose last 64-instance CTA holds one instance."""
    B = _kstep2_min_batch()
    s = _threshold_spec(B, dict(bracket_snap=1e-8))
    F, names, info = _default_run(s)
    _expect_kernels(names, ["k_step2<12>", "k_rad_block<12>"], what="B = %d" % B)
    assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info


def test_kstep_just_below_threshold():
    """One instance fewer (9408 on 148 SMs): below k_step2's threshold (and the automatic radiation look-ahead's);
    rad_lookahead = 2 forces the blocks: k_step<12>."""
    B = _kstep2_min_batch() - 1
    s = _threshold_spec(B, dict(bracket_snap=1e-8, rad_lookahead=2))
    F, names, info = _default_run(s)
    _expect_kernels(names, ["k_step<12>", "k_rad_block<12>"], forbid=["k_step2"], what="B = %d" % B)
    assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info


def test_row_grid_blocks_at_scale():
    """OSWEC-shaped tables (lag spacing 5/3 dt): once the history window is full (1000 steps) the look-ahead blocks
    convolve rows with the row-grid kernel (rb_general).  B = 4096, rad_lookahead = 2, snap 1e-8."""
    s = _spec("oswec", 4096, 0.03, 1080, n0=1040, opts=dict(bracket_snap=1e-8, rad_lookahead=2, exc_lookahead=4),
              sea=dict(SEA_SHORT, Hs=1.5, Tp=10.0))
    F, names, info = _run_gpu(s)
    _expect_kernels(names, ["k_rad_block<12>", "k_step<12>"], what="OSWEC row grid")
    assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info
    _check_oracle(s, F, "OSWEC row grid, B = 4096", info)


# ---------------------------------------------------------------------------------------------
# 3. batch-size boundaries, all instances
# ---------------------------------------------------------------------------------------------
BOUNDARY_B = [1, 8, 9, 63, 64, 65, 340, 341, 511, 512, 513, 2048, 2049]


@pytest.mark.parametrize("B", BOUNDARY_B)
@pytest.mark.parametrize("cfg", ["per_step", "lookahead"])
def test_batch_size_boundaries(B, cfg):
    """kFinalizeWarpMaxB (8/9), the 64-instance lane tile (63..65), the compact graph's 64 KB staging limit (340/341
    at D = 12), the 512-instance convolution tile (511..513), fork_max_batch (2048/2049).  Below 600 instances the
    oracle steps from an empty history; above, it is loaded with the GPU's history (full-population path)."""
    opts = {} if cfg == "per_step" else dict(bracket_snap=1e-8, exc_lookahead=4, rad_lookahead=2)
    if B < 600:
        s = _spec("rm3", B, 0.01, 110, opts=opts)
    else:
        s = _spec("rm3", B, 0.01, 110, n0=60, opts=opts)
    F, names, info = _run_gpu(s, profile_steps=0)
    if cfg == "lookahead":
        assert info["rad_blocks"]["steps_served"] == s["nsteps"] - max(s["n0"], 1), info
    _check_oracle(s, F, "B = %d, %s" % (B, cfg), info)


# ---------------------------------------------------------------------------------------------
# 4. variant matrix
# ---------------------------------------------------------------------------------------------
FINALIZE_KERNEL = {"1": "k_finalize(", "2": "k_finalize_warp<", "3": "k_finalize_split<"}


@pytest.mark.parametrize("mode", ["1", "2", "3"])
def test_finalize_modes(tmp_path, mode):
    """HC_FINALIZE_MODE = 1 / 2 / 3 (thread / warp / split) at B = 9, 513, 2049, on the per-step path and with the
    excitation look-ahead cache, with the history window full (every radiation and excitation partial is non-zero, so
    a finalize that skips one is seen).  The modes agree with each other only to rounding (different summation
    grouping of the partials), so oracle parity is the assertion."""
    specs = [_spec("rm3_window6", B, 0.01, 670, n0=640, opts=opts) for B in (9, 513, 2049)
             for opts in ({}, dict(exc_lookahead=4))]
    for s, (F, names, info) in zip(specs, _run_child(tmp_path, "finalize%s" % mode, {"HC_FINALIZE_MODE": mode}, specs)):
        what = "HC_FINALIZE_MODE=%s, B = %d, %s" % (mode, s["B"], s["opts"])
        _expect_kernels(names, [FINALIZE_KERNEL[mode]], [v for k, v in FINALIZE_KERNEL.items() if k != mode], what=what)
        _check_oracle(s, F, what, info)


def test_kstep2_off_is_bitwise_equal(tmp_path):
    """HC_KSTEP2 = 0 (k_step<12> instead of k_step2<12>) at B = 16384 and at the smallest k_step2 batch: k_step2 keeps
    k_step's summation order per item, so the forces are bit for bit the same."""
    specs = [_threshold_spec(B, dict(bracket_snap=1e-8)) for B in (16384, _kstep2_min_batch())]
    for s, (F, names, info) in zip(specs, _run_child(tmp_path, "kstep2", {"HC_KSTEP2": "0"}, specs)):
        _expect_kernels(names, ["k_step<12>"], forbid=["k_step2"], what="HC_KSTEP2=0, B = %d" % s["B"])
        F0, names0, _ = _default_run(s)
        _expect_kernels(names0, ["k_step2<12>"], what="default, B = %d" % s["B"])
        assert info["rad_blocks"]["steps_served"] == s["nsteps"] - s["n0"], info
        np.testing.assert_array_equal(F, F0, err_msg="k_step vs k_step2, B = %d" % s["B"])


COMPACT_ENVS = [{"HC_COMPACT_FORK": "0"}, {"HC_COMPACT_INLINE": "0"}, {"HC_COMPACT_DIRECT": "0"},
                {"HC_COMPACT_MAX_BYTES": "0"}]


@pytest.mark.parametrize("env", COMPACT_ENVS, ids=lambda e: "-".join("%s=%s" % kv for kv in e.items()))
def test_compact_graph_variants_bitwise(tmp_path, env):
    """The compact-graph variants change how a step is launched (fork, inline plans, direct write-back, whether the
    compact graph is used at all), not what the kernels compute: bit for bit the default's forces at B = 1, 65, 340."""
    specs = [_spec("rm3_short", B, 0.01, 60) for B in (1, 65, 340)]
    name = "compact_" + "_".join(k.lower() for k in env)
    for s, (F, names, info) in zip(specs, _run_child(tmp_path, name, env, specs)):
        _expect_kernels(names, ["k_radiation<12", "k_excitation<12", "k_finalize"], what="%s, B = %d" % (env, s["B"]))
        F0, _, _ = _default_run(s)
        np.testing.assert_array_equal(F, F0, err_msg="%s, B = %d" % (env, s["B"]))


def test_fork_max_batch_override_bitwise(tmp_path):
    """HC_FORK_MAX_BATCH = 0 at B = 513: the step graph without the forked excitation branch; same forces."""
    s = _spec("rm3_short", 513, 0.01, 60)
    (F, names, info), = _run_child(tmp_path, "forkmax", {"HC_FORK_MAX_BATCH": "0"}, [s])
    _expect_kernels(names, ["k_radiation<12", "k_excitation<12", "k_finalize"], what="HC_FORK_MAX_BATCH=0")
    np.testing.assert_array_equal(F, _default_run(s)[0])


@pytest.mark.parametrize("B", [1, 513, "ragged"])
def test_stream_path_without_graph_bitwise(B):
    """use_graph = False: every step's kernels launched on the stream; bit for bit the graph path's forces (at the
    ragged k_step2 size with the look-ahead blocks, else the per-step kernels)."""
    if B == "ragged":
        s = _threshold_spec(_kstep2_min_batch(), dict(bracket_snap=1e-8))
        want = ["k_step2<12>"]
    else:
        s = _spec("rm3_short", B, 0.01, 60)
        want = ["k_radiation<12", "k_excitation<12"]
    s2 = json.loads(json.dumps(s))
    s2["opts"]["use_graph"] = False
    F, names, info = _run_gpu(s2)
    _expect_kernels(names, want, what="use_graph=False, B = %d" % s["B"])
    np.testing.assert_array_equal(F, _default_run(s)[0])


RAD_KERNEL = {1: "k_radiation<12", 2: "k_radiation_mma12", 3: "k_radiation_hybrid12"}


@pytest.mark.parametrize("B", [513, 2049])
@pytest.mark.parametrize("rk", [1, 2, 3])
def test_radiation_kernels_beyond_one_tile(rk, B):
    """rad_kernel 1 / 2 / 3 (FMA / DMMA / hybrid) beyond one 512-instance tile, ragged against the hybrid kernel's
    256-instance tile."""
    s = _spec("rm3_short", B, 0.01, 60, opts=dict(rad_kernel=rk))
    F, names, info = _run_gpu(s)
    _expect_kernels(names, [RAD_KERNEL[rk]], [v for k, v in RAD_KERNEL.items() if k != rk],
                    what="rad_kernel %d, B = %d" % (rk, B))
    worst = _check_oracle(s, F, "rad_kernel %d, B = %d" % (rk, B), info)
    assert worst < 1e-11, worst


# ---------------------------------------------------------------------------------------------
# 5. chunk options
# ---------------------------------------------------------------------------------------------
def _chunk_case(kind, dt, opts):
    s = _spec(kind, 65, dt, 50, opts=opts)
    F, names, info = _run_gpu(s, profile_steps=0)
    _check_oracle(s, F, "%s %s" % (kind, opts), info)


CHUNK_TABLES = [("sphere", 0.015), ("rm3", 0.01)]


@pytest.mark.parametrize("kind,dt", CHUNK_TABLES, ids=["D6", "D12"])
def test_rad_chunk_options(kind, dt):
    """User rad_chunk: tiny, around the 8-lag groups, L - 1, L and 10 L (clamped to L, then halved to fit the 200 KB
    dynamic shared memory)."""
    L = _raw(kind)["bodies"][0]["rirf_t"].size
    for c in (1, 3, 7, 8, 9, L - 1, L, 10 * L):
        _chunk_case(kind, dt, dict(rad_chunk=c))


@pytest.mark.parametrize("kind,dt", CHUNK_TABLES, ids=["D6", "D12"])
def test_exc_chunk_options(kind, dt):
    """User exc_chunk up to the whole excitation IRF (Le = 8334 / 6000 lags): chunks whose staging exceeds the 200 KB
    of dynamic shared memory must be clamped when the ensemble is created, not fail to launch at the first step."""
    T = hc.Tables.from_raw(_raw(kind))
    e = hc.Ensemble(T, batch=1, dt_hint=dt)
    e.set_waves_irregular(dt=dt, duration=2.0, **SEA_SHORT)
    Le = max(e.irregular_sizes()[2])
    e.close()
    assert Le > 4096
    for c in (1, 5, 16, 17, Le, 4096):
        _chunk_case(kind, dt, dict(exc_chunk=c))


def test_dmma_radiation_chunk_clamp():
    """rad_kernel = 2 stages 16-row DMMA fragments (1568 B per lag at D = 12, against 1184 B for the FMA kernel):
    rad_chunk 131 .. 172 fit the FMA kernel's shared memory but not the DMMA kernel's."""
    for c in (130, 150, 172):
        _chunk_case("rm3", 0.01, dict(rad_kernel=2, rad_chunk=c))


# ---------------------------------------------------------------------------------------------
# 6. shapes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4, 8])
def test_many_bodies(N):
    """N = 4 / 8 bodies (D = 24 / 48): the run-time-D k_radiation_generic, one excitation group per body,
    kMaxBodies = 8 hydrostatics tables; irregular waves with tilted gravity, regular waves; rad_lookahead = 2 has no
    block kernel for these D and must fall back."""
    kind = "bodies%d" % N
    for waves, gvec, opts in (("irregular", (0.3, -0.2, -9.7), {}), ("regular", G981, {}),
                              ("irregular", G981, dict(rad_lookahead=2, bracket_snap=1e-8))):
        s = _spec(kind, 65, 0.05, 60, opts=opts, waves=waves, gvec=gvec)
        F, names, info = _run_gpu(s)
        what = "N = %d, %s, g = %s, %s" % (N, waves, gvec, opts)
        _expect_kernels(names, ["k_radiation_generic"], what=what)
        if opts:
            assert info["lookahead"]["radiation"] == -1, info
        _check_oracle(s, F, what, info)


def test_nine_bodies_rejected():
    raw = synth.make_tables(num_bodies=9, rirf_steps=21, rirf_duration=2.0, exc_irf_steps=21, exc_half_window=1.0)
    with pytest.raises(hc.HydroError):
        T = hc.Tables.from_raw(raw)
        hc.Ensemble(T, batch=2, dt_hint=0.05)


@pytest.mark.parametrize("opts", [{}, dict(exc_lookahead=4)], ids=["per_step", "lookahead"])
def test_two_excitation_windows(opts):
    """Bodies whose excitation IRFs sit on different windows cannot share one ND = 12 group: two ND = 6 groups."""
    s = _spec("rm3_two_windows", 65, 0.01, 70, opts=opts)
    F, names, info = _run_gpu(s)
    Le = info["irregular_sizes"]
    assert len(Le) == 2 and Le[0] != Le[1], Le
    _expect_kernels(names, ["k_excitation<6" if not opts else "k_exc_block"], forbid=["k_excitation<12"],
                    what="two windows %s" % opts)
    _check_oracle(s, F, "two excitation windows %s" % opts, info)


def test_per_instance_sea_states():
    """Hs_per_instance / Tp_per_instance (the per-instance amplitude branch of k_eta): spectrum, elevation and forces
    of every instance against oracle instances built with that instance's own Hs and Tp."""
    s = _spec("rm3_short", 65, 0.01, 80, per_instance_sea=True)
    F, names, info = _run_gpu(s)
    insts = _oracle_instances(s, list(range(s["B"])))
    for b, i in enumerate(insts):
        g, r = info["irregular"][b], i.irregular()
        for k in ("freqs", "S", "widths", "phases", "wavenumbers", "eta_t"):
            np.testing.assert_array_equal(g[k], r[k], err_msg="%s, instance %d" % (k, b))
        assert np.abs(g["eta"] - r["eta"]).max() <= 1e-12 * np.abs(r["eta"]).max(), b
    assert info["irregular"][0]["S"].max() != info["irregular"][1]["S"].max()
    _check_oracle(s, F, "per-instance sea states", info)


if __name__ == "__main__":
    _child_main(sys.argv[1], sys.argv[2])
