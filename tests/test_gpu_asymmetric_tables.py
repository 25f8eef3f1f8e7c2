"""Every matrix-indexed kernel path against the CPU oracle with hydro tables whose matrices are not symmetric.

The synthetic tables (synth.make_tables) have symmetric K, A_inf and hydrostatic stiffness, and the sphere's real
tables are nearly so: a row / column swap in any D x D path would pass every other parity test.  BEM output is not
exactly reciprocal and the reference never assumes symmetry (F_r = sum_c K_rc v_c), so the library must not either.
The tables here are common.asymmetric_tables of short synth.make_tables windows: K scaled per (row, column) by an
independent factor, a full non-symmetric hydrostatic stiffness, an asymmetric A_inf.

Each device layout of (K w) is reached by at least one case, named by the kernels torch.profiler sees it run:
d_K (k_radiation<6/12>, the INLINE compact-graph variants, k_radiation_generic, the leading-lag share in the
finalize / step kernels), d_Kfrag (k_radiation_mma12), d_Khyb (k_radiation_hybrid12), d_Kpad (k_rad_block<6/12/18>)
and d_Kyoung (k_step<6/12/18>, k_step2<12>); the hydrostatic stiffness through every finalize / step kernel; A_inf
through k_added_mass_mv and the inverse mass matrix of k_body_step.

The CPU cases (unmarked) prove that each GPU case can see a swap: the oracle run on that case's motion with every
matrix transposed differs from the plain run by at least 1e3 x the case's tolerance, on each compared quantity.
"""
import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import h5io, synth
from oracle import hc_oracle as orc
from test_gpu_device_stepping import np_simulate
from test_gpu_dispatch_coverage import NBUF, SEA_SHORT, _buffers, _expect_kernels, _kernel_names, _sm_count
from test_gpu_parity import _acc_times, _assert_parity

G981 = (0.0, 0.0, -9.81)
REL = 1e-9                   # force bar (test_gpu_parity._assert_parity, 1e-3 floor)
STEP_REL = 1e-8              # trajectory bar, x amplitude (test_gpu_device_stepping)
SENSITIVITY = 1e3            # a swap must move each compared quantity by this many tolerances

# short windows keep the oracle cheap; every case below runs past its full RIRF window
_SHAPES = {
    "n1_m1": dict(num_bodies=1, rirf_steps=101, rirf_duration=1.0),     # lag spacing = dt (0.01)
    "n1_m2": dict(num_bodies=1, rirf_steps=101, rirf_duration=2.0),     # 2 dt
    "n2_m6": dict(num_bodies=2, rirf_steps=101, rirf_duration=6.0),     # 6 dt, the headline workload's spacing
    "n2_oswec": dict(num_bodies=2, rirf_steps=121, rirf_duration=6.0),  # 0.05 = 5/3 dt at dt 0.03: row grid
    "n3_m2": dict(num_bodies=3, rirf_steps=101, rirf_duration=2.0),
    "n4": dict(num_bodies=4, rirf_steps=101, rirf_duration=5.0),        # dt 0.05
    "n8": dict(num_bodies=8, rirf_steps=101, rirf_duration=5.0),
}
_RAW = {}


def _raw(kind, transposed=False):
    key = (kind, transposed)
    if key not in _RAW:
        if transposed:
            _RAW[key] = common.transposed_tables(_raw(kind))
        else:
            base = synth.make_tables(exc_irf_steps=81, exc_half_window=2.0, num_freqs=64, **_SHAPES[kind])
            _RAW[key] = common.asymmetric_tables(base)
    return _RAW[key]


@pytest.fixture(scope="module", params=sorted(_SHAPES))
def asym(request):
    return request.param, _raw(request.param)


def test_fixture_is_asymmetric(asym):
    """The perturbation reaches every matrix: coupling blocks unrelated, every Kh entry non-zero."""
    kind, raw = asym
    D = 6 * len(raw["bodies"])
    K = np.concatenate([b["rirf_K"] for b in raw["bodies"]])
    A = np.concatenate([b["inf_added_mass"] for b in raw["bodies"]])
    off_diag = ~np.eye(D, dtype=bool)
    for s in (0, K.shape[2] // 3):
        assert np.abs(K - K.transpose(1, 0, 2))[:, :, s].max() > 0.1 * np.abs(K[:, :, s][off_diag]).max()
    assert np.abs(A - A.T).max() > 0.02 * np.abs(A).max()
    for b in raw["bodies"]:
        Kh = b["lin_matrix"]
        assert np.all(Kh != 0.0) and np.abs(Kh - Kh.T).max() > 1e-3 * np.abs(Kh).max()
        off = np.abs(Kh - np.diag(np.diag(Kh)))
        assert np.all(off.sum(axis=1) < 0.5 * np.abs(np.diag(Kh)))       # diagonally dominant: stepping stays stable
    assert A.shape == (D, D)


# ---------------------------------------------------------------------------------------------
# force cases: runs, GPU and oracle
# ---------------------------------------------------------------------------------------------
def _case(kind, B, dt, nsteps, want, forbid=(), opts=None, tapered=False, check=None, served=False):
    return dict(kind=kind, B=B, dt=dt, nsteps=nsteps, want=list(want), forbid=list(forbid), opts=dict(opts or {}),
                tapered=tapered, check=check, served=served)


BLOCKS = dict(bracket_snap=1e-8, rad_lookahead=2)     # look-ahead forced, snapped brackets
STREAM = dict(use_graph=False)                        # per-step kernels launched on the stream (no compact graph)


def _kstep2_batch():
    """The smallest batch served by k_step2<12> (test_gpu_dispatch_coverage._kstep2_min_batch), or its B200 value
    when no device is visible (the CPU sensitivity check only needs the instance indices)."""
    try:
        return 64 * (_sm_count() - 1) + 1
    except Exception:
        return 64 * 147 + 1


CASES = {
    # D = 6
    "d6_radiation": _case("n1_m2", 65, 0.01, 230, ["k_radiation<6, false", "k_finalize"], ["k_rad_block", "k_step"],
                          STREAM),
    "d6_compact_inline": _case("n1_m2", 4, 0.01, 230, ["k_radiation<6, true", "k_finalize_warp"]),
    "d6_blocks_lag_dt": _case("n1_m1", 8, 0.01, 140, ["k_rad_block<6>", "k_step<6>"], opts=BLOCKS, served=True),
    "d6_blocks_m2": _case("n1_m2", 8, 0.01, 230, ["k_rad_block<6>", "k_step<6>"], opts=BLOCKS, served=True),
    "d6_tapered": _case("n1_m2", 4, 0.01, 230, ["k_radiation<6"], tapered=True),
    # D = 12
    "d12_radiation": _case("n2_m6", 65, 0.01, 640, ["k_radiation<12, false", "k_finalize"],
                           ["k_rad_block", "k_step"], STREAM),
    "d12_dmma": _case("n2_m6", 65, 0.01, 640, ["k_radiation_mma12"], opts=dict(rad_kernel=2)),
    "d12_hybrid": _case("n2_m6", 65, 0.01, 640, ["k_radiation_hybrid12"], opts=dict(rad_kernel=3)),
    "d12_compact_inline": _case("n2_m6", 4, 0.01, 640, ["k_radiation<12, true", "k_finalize_warp"]),
    "d12_blocks_lag_grid": _case("n2_m6", 8, 0.01, 680, ["k_rad_block<12>", "k_step<12>"], opts=BLOCKS, served=True),
    "d12_blocks_row_grid": _case("n2_oswec", 8, 0.03, 240, ["k_rad_block<12>", "k_step<12>"], opts=BLOCKS,
                                 served=True),
    # orientation, not lane mapping, is the question: the oracle follows the first and the last two 64-instance tiles
    "d12_kstep2": _case("n2_m6", "kstep2", 0.01, 680, ["k_rad_block<12>", "k_step2<12>"],
                        opts=dict(bracket_snap=1e-8), check="tiles", served=True),
    "d12_tapered_blocks": _case("n2_m6", 8, 0.01, 680, ["k_rad_block<12>", "k_step<12>"], opts=BLOCKS, tapered=True,
                                served=True),
    # D = 18
    "d18_generic": _case("n3_m2", 65, 0.01, 230, ["k_radiation_generic"]),
    "d18_blocks": _case("n3_m2", 8, 0.01, 230, ["k_rad_block<18>", "k_step<18>"], opts=BLOCKS, served=True),
    # D = 24, 48
    "d24_generic": _case("n4", 65, 0.05, 110, ["k_radiation_generic"]),
    "d48_generic": _case("n8", 65, 0.05, 110, ["k_radiation_generic"]),
}


def _batch(c):
    return _kstep2_batch() if c["B"] == "kstep2" else c["B"]


def _check_idx(c):
    B = _batch(c)
    if c["check"] == "tiles":
        return list(range(64)) + list(range(B - 65, B))
    return list(range(B))


def _seeds(B):
    return 1 + np.arange(B, dtype=np.int32)


def _sea(c):
    return dict(dt=c["dt"], duration=(c["nsteps"] + 64) * c["dt"], **SEA_SHORT)


TAPER = dict(taper_start_percent=0.5, taper_end_percent=0.9)


def _oracle(c, idx, transposed=False):
    """Oracle forces of case c for instances idx: (total, hydrostatics, radiation, waves), each [nsteps][len(idx)][D]."""
    raw = _raw(c["kind"], transposed)
    O = orc.Tables(raw)
    if c["tapered"]:
        O.set_tapered(start=TAPER["taper_start_percent"], end=TAPER["taper_end_percent"])
    D = 6 * len(raw["bodies"])
    seeds = _seeds(_batch(c))
    insts = []
    for b in idx:
        i = orc.Instance(O, omp_mode=0)
        i.set_irregular(seed=int(seeds[b]), share_irf_from=insts[0] if insts else None, **_sea(c))
        insts.append(i)
    pose, vel = _buffers(D, _batch(c), c["dt"])
    times = _acc_times(c["nsteps"], c["dt"])
    out = np.empty((4, c["nsteps"], len(idx), D))
    for n, t in enumerate(times):
        p, v = pose[n % NBUF], vel[n % NBUF]
        for j, (b, inst) in enumerate(zip(idx, insts)):
            out[:, n, j] = inst.force(t, p[b], v[b], G981, components=True)
    return out


def _run_gpu(c, idx, profile_steps=10):
    """GPU forces of case c (recorded for instances idx, same layout as _oracle), the kernel names seen over the last
    profile_steps steps (history window full, look-ahead serving) and the look-ahead statistics."""
    raw = _raw(c["kind"])
    T = hc.Tables.from_raw(raw)
    if c["tapered"]:
        T.set_convolution_mode("TaperedDirect", **TAPER)
    B, dt, D = _batch(c), c["dt"], T.dofs
    ens = hc.Ensemble(T, batch=B, dt_hint=dt, **c["opts"])
    ens.set_waves_irregular(seeds=_seeds(B), **_sea(c))
    pose, vel = _buffers(D, B, dt)
    times = _acc_times(c["nsteps"], dt)
    out = np.empty((4, c["nsteps"], len(idx), D))
    h_out = np.empty((B, D))

    def step(n):
        ens.step(times[n], pose[n % NBUF], vel[n % NBUF], G981, out=h_out)
        hs, rad, wv = ens.components()
        out[0, n], out[1, n], out[2, n], out[3, n] = h_out[idx], hs[idx], rad[idx], wv[idx]

    p0 = c["nsteps"] - profile_steps
    for n in range(p0):
        step(n)

    def prof():
        for n in range(p0, c["nsteps"]):
            step(n)
    names = _kernel_names(prof)
    stats = ens.rad_block_stats()
    ens.close()
    return out, names, stats


def _sensitivity(ref, alt):
    """For each compared quantity (total, hydrostatics, radiation): the largest |alt - ref| in units of the tolerance
    the GPU case grants ref (the hydrostatics are compared bitwise; they are measured on the same 1e-9 scale)."""
    out = {}
    for k, name in ((0, "total"), (1, "hydrostatics"), (2, "radiation")):
        tol = common.force_tol(ref[k], rel=REL)
        out[name] = float((np.abs(alt[k] - ref[k]) / tol).max())
    return out


@pytest.mark.parametrize("name", sorted(CASES))
def test_force_case_sees_a_transposition(name):
    """The oracle on the case's motion, with every matrix transposed (K per lag, Kh, A_inf), differs from the plain
    oracle by >= 1e3 x the case's tolerance on the total, the hydrostatic and the radiation component.  The radiation
    component is checked on its own because it can be small next to the hydrostatics and the waves."""
    c = CASES[name]
    idx = _check_idx(c)
    idx = [idx[0], idx[-1]]                       # two instances are enough to show the case can see a swap
    ref, alt = _oracle(c, idx), _oracle(c, idx, transposed=True)
    sens = _sensitivity(ref, alt)
    assert min(sens.values()) >= SENSITIVITY, (name, sens)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_force_case_matches_oracle(name):
    """Every recorded instance, DoF and step against the oracle: the total, the radiation and the wave component at
    the 1e-9 bar, the hydrostatic component bit for bit."""
    c = CASES[name]
    idx = _check_idx(c)
    got, names, stats = _run_gpu(c, idx)
    _expect_kernels(names, c["want"], c["forbid"], what=name)
    if c["served"]:
        assert stats["steps_served"] > 0, stats
    ref = _oracle(c, idx)
    np.testing.assert_array_equal(got[1], ref[1], err_msg="%s: hydrostatics" % name)
    worst = _assert_parity(got[2], ref[2], "%s: radiation" % name, rel=REL)
    _assert_parity(got[3], ref[3], "%s: waves" % name, rel=REL)
    _assert_parity(got[0], ref[0], "%s: total" % name, rel=REL)
    print("%s: %d instances x %d steps, worst radiation error %.2e, kernels %s" % (
        name, len(idx), c["nsteps"], worst, [n for n in names if any(w.split("<")[0] in n for w in c["want"])]))


# ---------------------------------------------------------------------------------------------
# added mass
# ---------------------------------------------------------------------------------------------
AM_KINDS = {6: "n1_m2", 12: "n2_m6", 18: "n3_m2", 48: "n8"}


@pytest.mark.parametrize("D", sorted(AM_KINDS))
def test_added_mass_matrix_is_the_oracle_bitwise(D):
    raw = _raw(AM_KINDS[D])
    M = hc.Tables.from_raw(raw).added_mass()
    np.testing.assert_array_equal(M, orc.Tables(raw).added_mass())
    assert np.abs(M - M.T).max() > 1e-3 * np.abs(M).max()


def _am_inputs(B, D):
    rng = np.random.default_rng(100 + D + B)
    return 0.37, rng.standard_normal((B, D)), rng.standard_normal((B, D))


@pytest.mark.parametrize("D", sorted(AM_KINDS))
def test_added_mass_mv_sees_a_transposition(D):
    c, w, R = _am_inputs(2, D)
    O, Ot = orc.Tables(_raw(AM_KINDS[D])), orc.Tables(_raw(AM_KINDS[D], transposed=True))
    ref = np.array([O.added_mass_mv(c, w[b], R[b]) for b in range(2)])
    alt = np.array([Ot.added_mass_mv(c, w[b], R[b]) for b in range(2)])
    assert np.abs(alt - ref).max() >= SENSITIVITY * REL * np.abs(ref).max()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [127, 128, 129])
@pytest.mark.parametrize("D", sorted(AM_KINDS))
def test_added_mass_mv_is_the_oracle_bitwise(D, B):
    """Ensemble.added_mass_mv and added_mass_mv_device against the oracle, bit for bit; B straddles the kernel's
    128-thread CTA."""
    import torch
    raw = _raw(AM_KINDS[D])
    T, O = hc.Tables.from_raw(raw), orc.Tables(raw)
    ens = hc.Ensemble(T, batch=B, dt_hint=0.01)
    c, w, R = _am_inputs(B, D)
    ref = np.array([O.added_mass_mv(c, w[b], R[b]) for b in range(B)])
    names = _kernel_names(lambda: ens.added_mass_mv(c, w, R))
    _expect_kernels(names, ["k_added_mass_mv"], what="added_mass_mv D = %d, B = %d" % (D, B))
    np.testing.assert_array_equal(ens.added_mass_mv(c, w, R), ref)
    dev = torch.device("cuda", 0)
    dw, dR = torch.from_numpy(w).to(dev), torch.from_numpy(R).to(dev)
    ens.added_mass_mv_device(D, c, dw, dR)
    ens.sync()
    np.testing.assert_array_equal(dR.cpu().numpy(), ref)
    ens.close()


# ---------------------------------------------------------------------------------------------
# device stepping: asymmetric A_inf, so the inverse mass matrix of k_body_step is not symmetric
# ---------------------------------------------------------------------------------------------
STEP_KINDS = {1: "n1_m2", 2: "n2_m6", 3: "n3_m2", 8: "n8"}
STEP_B, STEP_N, STEP_DT = 65, 120, 0.01          # 65: two k_body_step CTAs of 64, the second holding one instance
REGULAR = (0.5, 0.9)


def _free_mask(N, mask):
    if mask == "all":
        return np.ones(6 * N, bool)
    heave_pitch = np.array([0, 0, 1, 0, 1, 0], bool)
    if N == 1:
        return heave_pitch
    # body 0 locked to ground, body 1 free in heave and pitch, any further body free
    return np.concatenate([np.zeros(6, bool), heave_pitch] + [np.ones(6, bool)] * (N - 2))


def _step_inputs(N, B):
    D = 6 * N
    rng = np.random.Generator(np.random.MT19937(40 + N))
    pose0 = np.zeros((B, D))
    pose0[:, 2::6] = rng.uniform(-0.1, 0.1, (B, N))
    for k in (3, 4, 5):
        pose0[:, k::6] = rng.uniform(-0.05, 0.05, (B, N))
    vel0 = rng.uniform(-0.05, 0.05, (B, D))
    pto_c = rng.uniform(0.0, 1e5, (B, D))
    pto_k = rng.uniform(0.0, 1e5, (B, D))
    mass = [synth.RM3_MASSES[b % 2] for b in range(N)]
    inertia = [synth.RM3_INERTIAS[b % 2] for b in range(N)]
    return pose0, vel0, pto_c, pto_k, mass, inertia


def _np_run(N, scheme, mask, idx, transposed=False):
    raw = _raw(STEP_KINDS[N], transposed)
    O = orc.Tables(raw)
    insts = []
    for _ in idx:
        i = orc.Instance(O, omp_mode=0)
        i.set_regular(*REGULAR)
        insts.append(i)
    pose0, vel0, c, k, mass, inertia = _step_inputs(N, STEP_B)

    def force(t, p, v):
        return np.array([i.force(t, p[j], v[j], G981) for j, i in enumerate(insts)])
    return np_simulate(force, O.added_mass(), mass, inertia, pose0[idx], STEP_N, STEP_DT, scheme=scheme,
                       free=_free_mask(N, mask), c=c[idx], k=k[idx], vel0=vel0[idx])


def _step_errors(x, xr, pose0):
    """Per instance: max |x - xr| over steps and DoFs, in units of the instance's amplitude max |xr - pose0|."""
    amp = np.abs(xr - pose0[None]).max(axis=(0, 2))
    assert amp.min() > 1e-3, amp.min()
    return np.abs(x - xr).max(axis=(0, 2)) / amp


STEP_PARAMS = [(N, s, m) for N in sorted(STEP_KINDS) for s in ("euler", "hht") for m in ("all", "mixed")]


@pytest.mark.parametrize("N,scheme,mask", STEP_PARAMS)
def test_stepping_case_sees_a_transposition(N, scheme, mask):
    """np_simulate with every matrix transposed (A_inf, so M^-1, and the force tables) differs from the plain run by
    >= 1e3 x the 1e-8 x amplitude bar."""
    idx = [0, STEP_B - 1]
    pose0 = _step_inputs(N, STEP_B)[0][idx]
    _, xr, _ = _np_run(N, scheme, mask, idx)
    _, xt, _ = _np_run(N, scheme, mask, idx, transposed=True)
    assert _step_errors(xt, xr, pose0).max() >= SENSITIVITY * STEP_REL


@pytest.mark.gpu
@pytest.mark.parametrize("N,scheme,mask", STEP_PARAMS)
def test_stepping_matches_numpy_restatement(N, scheme, mask):
    """Ensemble.simulate (k_body_step) with an asymmetric A_inf against np_simulate driven by oracle forces, every
    instance at 1e-8 x its amplitude."""
    raw = _raw(STEP_KINDS[N])
    T = hc.Tables.from_raw(raw)
    pose0, vel0, c, k, mass, inertia = _step_inputs(N, STEP_B)
    ens = hc.Ensemble(T, batch=STEP_B, dt_hint=STEP_DT)
    ens.set_waves_regular([REGULAR[0]], [REGULAR[1]])
    res = []
    names = _kernel_names(lambda: res.append(ens.simulate(pose0, STEP_N, STEP_DT, mass, inertia, vel0=vel0,
                                                          scheme=scheme, free_dof=_free_mask(N, mask), pto_damping=c,
                                                          pto_stiffness=k)))
    _expect_kernels(names, ["k_body_step"], what="N = %d, %s, %s" % (N, scheme, mask))
    t, x, v, e, done = res[0]
    ens.close()
    assert done == STEP_N
    idx = list(range(STEP_B))
    tr, xr, _ = _np_run(N, scheme, mask, idx)
    np.testing.assert_array_equal(t, tr)
    err = _step_errors(x, xr, pose0)
    assert err.max() <= STEP_REL, (err.max(), int(err.argmax()))


# ---------------------------------------------------------------------------------------------
# .h5 round trip
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["n1_m2", "n2_m6"])
def test_h5_round_trip_keeps_orientation(tmp_path, kind):
    """write_bemio of asymmetric tables, read back by Tables.from_h5: bit for bit Tables.from_raw."""
    raw = _raw(kind)
    N = len(raw["bodies"])
    f = tmp_path / "asym.h5"
    h5io.write_bemio(f, raw)
    A, B = hc.Tables.from_h5(f, N), hc.Tables.from_raw(raw)
    np.testing.assert_array_equal(A.rirf(), B.rirf())
    np.testing.assert_array_equal(A.rirf_time(), B.rirf_time())
    np.testing.assert_array_equal(A.added_mass(), B.added_mass())
    for b in range(N):
        np.testing.assert_array_equal(A.lin_matrix(b), B.lin_matrix(b))
        np.testing.assert_array_equal(A.lin_matrix(b), raw["bodies"][b]["lin_matrix"])
        np.testing.assert_array_equal(A.inf_added_mass(b), B.inf_added_mass(b))
