"""hydrochrono_b200 -- B200-native hydrodynamic force path for HydroChrono (Python host binding).

The product is the C-ABI library (include/hydrochrono_b200.h) and the C++ host layer that mirrors
HydroChrono's classes (hydrochrono_b200/host).  This module is the thin ctypes binding used by the
parity tests and bench.py; it adds nothing to the computation.
"""
import ctypes as C

import numpy as np

from . import _capi
from ._capi import lib

__all__ = ["Tables", "Ensemble", "HydroError", "DuplicateTimeError", "EtaWindowError", "version", "device_count"]


class HydroError(RuntimeError):
    """std::runtime_error on the reference side."""

    def __init__(self, status, msg):
        super().__init__("%s: %s" % (_capi.STATUS_NAMES.get(status, status), msg))
        self.status = status


class DuplicateTimeError(HydroError):
    pass


class EtaWindowError(HydroError):
    pass


def _check(status):
    if status == 0:
        return
    msg = lib.hc_last_error().decode(errors="replace")
    if status == 2:
        raise IndexError(msg)  # std::out_of_range
    if status == 4:
        raise DuplicateTimeError(status, msg)
    if status == 5:
        raise EtaWindowError(status, msg)
    raise HydroError(status, msg)


def version():
    return lib.hc_version().decode()


def device_count():
    return lib.hc_device_count()


def measure_fp64_peak(device=0):
    """Measured FP64 FMA peak of the device, TFLOP/s."""
    v = C.c_double()
    _check(lib.hc_measure_fp64_peak(device, C.byref(v)))
    return v.value


def measure_fp64_mma_peak(device=0):
    """Measured FP64 tensor-core (DMMA m8n8k4) peak of the device, TFLOP/s."""
    v = C.c_double()
    _check(lib.hc_measure_fp64_mma_peak(device, C.byref(v)))
    return v.value


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def wave_kinematics(omega, amplitude, phase, wavenumber, position, t, water_depth, mwl=0.0, wheeler_stretching=False):
    """(eta, velocity[3], acceleration[3]) at a point for a sum of Airy components travelling along +x: the
    arithmetic behind {RegularWave,IrregularWaves}::GetElevation / GetVelocity / GetAcceleration
    (src/wave_types.cpp:14-160,301-313,515-550).  Host code, off the step path."""
    om, am, ph, k = (_f64(np.atleast_1d(x)) for x in (omega, amplitude, phase, wavenumber))
    pos = _f64(position)
    eta = C.c_double()
    v, a = np.empty(3), np.empty(3)
    _check(lib.hc_wave_kinematics(om.size, _dp(om), _dp(am), _dp(ph), _dp(k), _dp(pos), float(t), float(water_depth),
                                  float(mwl), int(bool(wheeler_stretching)), C.byref(eta), _dp(v), _dp(a)))
    return eta.value, v, a


def jonswap_spectrum_hz(f, Hs, Tp, gamma=3.3, is_normalized=False):
    f = _f64(f)
    S = np.empty_like(f)
    _check(lib.hc_jonswap_spectrum_hz(f.size, _dp(f), Hs, Tp, gamma, int(is_normalized), _dp(S)))
    return S


def compute_wave_number(omega, water_depth, g):
    k = C.c_double()
    _check(lib.hc_compute_wave_number(omega, water_depth, g, C.byref(k)))
    return k.value


def random_phases(seed, n):
    out = np.empty(n)
    _check(lib.hc_random_phases(int(seed), int(n), _dp(out)))
    return out


def _dp(a):
    return a.ctypes.data_as(_capi.dp) if a is not None else None


def _kin_points(points, batch):
    pts = _f64(points)
    if pts.ndim != 3 or pts.shape[0] != batch or pts.shape[2] != 3:
        raise ValueError("points must be [batch][P][3]")
    return pts


def _kin_outputs(pts):
    B, P = pts.shape[:2]
    return np.empty((B, P)), np.empty((B, P, 3)), np.empty((B, P, 3))


def _ptr(x):
    """Address of a numpy array / torch tensor / raw integer pointer."""
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    return C.c_void_p(x.ctypes.data)


class Tables:
    """HydroData (reference include/hydroc/h5fileinfo.h:35-226)."""

    def __init__(self, handle):
        self._h = handle
        self.num_bodies = lib.hc_tables_num_bodies(handle)
        self.dofs = 6 * self.num_bodies
        self.rirf_steps = lib.hc_tables_rirf_steps(handle)

    @classmethod
    def from_h5(cls, path, num_bodies=1):
        h = C.c_void_p()
        _check(lib.hc_tables_load_h5(str(path).encode(), num_bodies, C.byref(h)))
        return cls(h)

    @classmethod
    def from_raw(cls, raw):
        """raw: dict in the layout of tests/h5lite.load_bemio / hydrochrono_b200.synth.make_tables."""
        bodies = raw["bodies"]
        N = len(bodies)
        L = int(np.asarray(bodies[0]["rirf_t"]).size)
        w = _f64(raw.get("w", np.zeros(0)))
        nw = w.size
        Le0 = int(np.asarray(bodies[0].get("exc_irf_t", np.zeros(0))).size)
        keep = {
            "rirf_t": _f64(np.stack([np.asarray(b["rirf_t"]).ravel() for b in bodies])),
            "rirf_K": _f64(np.stack([b["rirf_K"] for b in bodies])),
            "lin": _f64(np.stack([b["lin_matrix"] for b in bodies])),
            "ainf": _f64(np.stack([b["inf_added_mass"] for b in bodies])),
            "vol": _f64([b["disp_vol"] for b in bodies]),
            "cg": _f64(np.stack([np.asarray(b["cg"]).ravel() for b in bodies])),
            "cb": _f64(np.stack([np.asarray(b["cb"]).ravel() for b in bodies])),
            "w": w,
        }
        if keep["rirf_K"].shape != (N, 6, 6 * N, L):
            raise ValueError("rirf_K must be [N][6][6N][L], got %s" % (keep["rirf_K"].shape,))
        if nw:
            keep["mag"] = _f64(np.stack([np.asarray(b["exc_mag"]).reshape(6, -1, nw)[:, 0, :] for b in bodies]))
            keep["ph"] = _f64(np.stack([np.asarray(b["exc_phase"]).reshape(6, -1, nw)[:, 0, :] for b in bodies]))
        if Le0:
            keep["et"] = _f64(np.stack([np.asarray(b["exc_irf_t"]).ravel() for b in bodies]))
            keep["ef"] = _f64(np.stack([np.asarray(b["exc_irf_f"]).reshape(6, -1, Le0)[:, 0, :] for b in bodies]))
        d = _capi.TablesDesc(N, L, nw, Le0, float(raw["rho"]), float(raw["g"]), float(raw["water_depth"]),
                             _dp(keep["rirf_t"]), _dp(keep["rirf_K"]), _dp(keep["lin"]), _dp(keep["ainf"]),
                             _dp(keep["vol"]), _dp(keep["cg"]), _dp(keep["cb"]), _dp(w), _dp(keep.get("mag")),
                             _dp(keep.get("ph")), _dp(keep.get("et")), _dp(keep.get("ef")))
        h = C.c_void_p()
        _check(lib.hc_tables_create(C.byref(d), C.byref(h)))
        return cls(h)

    # -- HydroData getters ---------------------------------------------------
    @property
    def rho(self):
        return lib.hc_tables_rho(self._h)

    @property
    def g(self):
        return lib.hc_tables_g(self._h)

    @property
    def water_depth(self):
        return lib.hc_tables_water_depth(self._h)

    def rirf_time(self):
        out = np.empty(self.rirf_steps)
        _check(lib.hc_tables_rirf_time(self._h, _dp(out)))
        return out

    def rirf_width(self):
        out = np.empty(self.rirf_steps)
        _check(lib.hc_tables_rirf_width(self._h, _dp(out)))
        return out

    def rirf_val(self, row, col, st):
        v = C.c_double()
        _check(lib.hc_tables_rirf_val(self._h, row, col, st, C.byref(v)))
        return v.value

    def rirf(self):
        out = np.empty((self.dofs, self.dofs, self.rirf_steps))
        _check(lib.hc_tables_rirf_all(self._h, _dp(out)))
        return out

    def lin_matrix(self, b):
        out = np.empty((6, 6))
        _check(lib.hc_tables_lin_matrix(self._h, b, _dp(out)))
        return out

    def hydrostatic_stiffness(self, b, i, j):
        v = C.c_double()
        _check(lib.hc_tables_hydrostatic_stiffness(self._h, b, i, j, C.byref(v)))
        return v.value

    def inf_added_mass(self, b):
        out = np.empty((6, self.dofs))
        _check(lib.hc_tables_inf_added_mass(self._h, b, _dp(out)))
        return out

    def disp_vol(self, b):
        v = C.c_double()
        _check(lib.hc_tables_disp_vol(self._h, b, C.byref(v)))
        return v.value

    def cg(self, b):
        out = np.empty(3)
        _check(lib.hc_tables_cg(self._h, b, _dp(out)))
        return out

    def cb(self, b):
        out = np.empty(3)
        _check(lib.hc_tables_cb(self._h, b, _dp(out)))
        return out

    def set_convolution_mode(self, mode, smoothing="sg", window_length=5, rirf_end_time=-1.0, taper_start_percent=0.8,
                             taper_end_percent=1.0, taper_final_amplitude=0.0):
        """TestHydro::SetRadiationConvolutionMode / SetTaperedDirectOptions. mode: 'Baseline' | 'TaperedDirect'."""
        m = 1 if str(mode).lower() == "tapereddirect" else 0
        o = _capi.TaperedOpts(smoothing.encode(), window_length, rirf_end_time, taper_start_percent,
                              taper_end_percent, taper_final_amplitude)
        _check(lib.hc_tables_set_convolution_mode(self._h, m, C.byref(o)))

    def added_mass(self, n_sys=None):
        """ChLoadAddedMass system matrix (src/chloadaddedmass.cpp:12-52)."""
        n = n_sys or self.dofs
        M = np.empty((n, n))
        _check(lib.hc_added_mass(self._h, n, _dp(M)))
        return M

    def rad_lookahead_plan(self, dt_hint):
        """Host-side plan of the radiation look-ahead for a step size: (mode, rows_per_lag, kernel_lags); mode 0 =
        not usable, 1 = lag grid, 2 = row grid (hc_rad_lookahead_plan)."""
        mode, m, lk = C.c_int(), C.c_int(), C.c_int()
        _check(lib.hc_rad_lookahead_plan(self._h, float(dt_hint), C.byref(mode), C.byref(m), C.byref(lk)))
        return mode.value, m.value, lk.value

    def rad_lookahead_row_kernel(self, dt_hint):
        """[kernel_lags][6N][6N] kernel the look-ahead blocks convolve the history rows with."""
        _, _, lk = self.rad_lookahead_plan(dt_hint)
        D = 6 * self.num_bodies
        out = np.empty((lk, D, D))
        _check(lib.hc_rad_lookahead_row_kernel(self._h, float(dt_hint), _dp(out)))
        return out

    def rad_lookahead_check_step(self, dt_hint, bracket_snap, times_newest_first):
        """smax (largest bracketed lag) if the look-ahead could serve a step with this time history, else -1."""
        tm = _f64(times_newest_first)
        smax = C.c_int()
        _check(lib.hc_rad_lookahead_check_step(self._h, float(dt_hint), float(bracket_snap), _dp(tm), int(tm.size),
                                               C.byref(smax)))
        return smax.value

    def close(self):
        if getattr(self, "_h", None):
            lib.hc_tables_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


class Ensemble:
    """B lock-stepped TestHydro instances on one GPU."""

    def __init__(self, tables, batch=1, device=0, dt_hint=0.0, bracket_snap=0.0, rad_chunk=0, exc_chunk=0,
                 use_graph=True, stream=None, exc_lookahead=0, rad_kernel=0, rad_lookahead=0, rad_pass_mode=0):
        self.tables = tables  # keep alive
        o = _capi.EnsembleOpts()
        lib.hc_ensemble_default_opts(C.byref(o))
        o.device, o.batch, o.dt_hint, o.bracket_snap = device, batch, dt_hint, bracket_snap
        o.rad_chunk, o.exc_chunk, o.use_graph = rad_chunk, exc_chunk, int(use_graph)
        o.exc_lookahead = int(exc_lookahead)
        o.rad_kernel = int(rad_kernel)
        o.rad_lookahead = int(rad_lookahead)
        o.rad_pass_mode = int(rad_pass_mode)
        o.stream = stream
        h = C.c_void_p()
        _check(lib.hc_ensemble_create(tables._h, C.byref(o), C.byref(h)))
        self._h = h
        self.batch = batch
        self.dofs = tables.dofs
        self.device = device
        self._gcache = {}
        self._re_val = C.c_int()
        self._re = C.byref(self._re_val)

    # -- waves ---------------------------------------------------------------
    def set_waves_none(self):
        _check(lib.hc_waves_none(self._h))

    def set_waves_regular(self, amplitude, omega, phase=None):
        a, w = _f64(np.atleast_1d(amplitude)), _f64(np.atleast_1d(omega))
        p = _f64(np.atleast_1d(phase)) if phase is not None else None
        _check(lib.hc_waves_regular(self._h, a.size, _dp(a), _dp(w), _dp(p)))

    def set_waves_irregular(self, dt, duration, ramp=0.0, Hs=0.0, Tp=0.0, fmin=0.001, fmax=1.0, nfreq=0, gamma=1.0,
                            is_normalized=False, seed=1, seeds=None, Hs_per_instance=None, Tp_per_instance=None):
        p = _capi.IrregularParams(dt, duration, ramp, Hs, Tp, fmin, fmax, float(nfreq), gamma, int(is_normalized), seed)
        s = np.ascontiguousarray(seeds, dtype=np.int32) if seeds is not None else None
        hs = _f64(Hs_per_instance) if Hs_per_instance is not None else None
        tp = _f64(Tp_per_instance) if Tp_per_instance is not None else None
        _check(lib.hc_waves_irregular(self._h, C.byref(p), s.ctypes.data_as(_capi.ip) if s is not None else None,
                                      _dp(hs), _dp(tp)))

    def set_waves_series(self, dt, time, eta):
        """Imported free-surface elevation (IrregularWaveParams::eta_file_path_, wave_types.cpp:480-500): time [n] and eta
        [n] (shared) or [B][n] (per instance); dt = the spacing the excitation IRF is resampled to."""
        t, e = _f64(time), _f64(eta)
        if t.ndim != 1 or e.shape[-1] != t.size or e.ndim not in (1, 2) or (e.ndim == 2 and e.shape[0] != self.batch):
            raise ValueError("time must be [n] and eta [n] or [batch][n]")
        _check(lib.hc_waves_irregular_series(self._h, float(dt), t.size, _dp(t), _dp(e), int(e.ndim == 2)))

    def irregular_sizes(self):
        nf, ne = C.c_int(), C.c_int()
        le = (C.c_int * self.tables.num_bodies)()
        _check(lib.hc_waves_irregular_sizes(self._h, C.byref(nf), C.byref(ne), le))
        return nf.value, ne.value, list(le)

    def irregular(self, instance=0):
        nf, ne, le = self.irregular_sizes()
        out = {}
        if nf:
            for k in ("freqs", "S", "widths", "phases", "wavenumbers"):
                out[k] = np.empty(nf)
            _check(lib.hc_waves_irregular_spectrum(self._h, instance, _dp(out["freqs"]), _dp(out["S"]),
                                                   _dp(out["widths"]), _dp(out["phases"]), _dp(out["wavenumbers"])))
        out["eta_t"], out["eta"] = np.empty(ne), np.empty(ne)
        _check(lib.hc_waves_irregular_eta(self._h, instance, _dp(out["eta_t"]), _dp(out["eta"])))
        out["irf"] = []
        for b, n in enumerate(le):
            t, w, f = np.empty(n), np.empty(n), np.empty((6, n))
            _check(lib.hc_waves_irregular_irf(self._h, b, _dp(t), _dp(w), _dp(f)))
            out["irf"].append({"t": t, "w": w, "f": f})
        return out

    def regular_coeffs(self, instance=0):
        mag, ph = np.empty(self.dofs), np.empty(self.dofs)
        k = C.c_double()
        _check(lib.hc_waves_regular_coeffs(self._h, instance, _dp(mag), _dp(ph), C.byref(k)))
        return mag, ph, k.value

    # -- stepping ------------------------------------------------------------
    def host_buffers(self):
        """The ensemble's pinned staging buffers as numpy views [B][6N]: (pose, vel, force)."""
        p, v, f = _capi.dp(), _capi.dp(), _capi.dp()
        _check(lib.hc_ensemble_host_buffers(self._h, C.byref(p), C.byref(v), C.byref(f)))
        shape = (self.batch, self.dofs)
        return tuple(np.ctypeslib.as_array(x, shape=shape) for x in (p, v, f))

    def step(self, t, pose, vel, gvec=(0.0, 0.0, -9.81), out=None):
        """Host-buffer step: returns force [B][6N] (numpy)."""
        pose, vel = _f64(pose), _f64(vel)
        g = self._gvec(gvec)
        if pose.size != self.batch * self.dofs or vel.size != pose.size:
            raise ValueError("pose/vel must be [B][6N]")
        if out is None:
            out = np.empty((self.batch, self.dofs))
        re = self._re
        _check(lib.hc_step(self._h, t, pose.ctypes.data, vel.ctypes.data, g, out.ctypes.data, re))
        self.last_recomputed = bool(self._re_val.value)
        return out

    def _gvec(self, gvec):
        """ctypes pointer to the gravity vector; tuples are converted once (a step is tens of microseconds)."""
        if isinstance(gvec, tuple):
            hit = self._gcache.get(gvec)
            if hit is None:
                arr = _f64(gvec)
                hit = self._gcache[gvec] = (arr, _dp(arr))
            return hit[1]
        arr = _f64(gvec)
        self._gtmp = arr
        return _dp(arr)

    def step_device(self, t, d_pose, d_vel, d_force, gvec=(0.0, 0.0, -9.81)):
        """Device-pointer step (torch CUDA tensors or raw addresses); asynchronous on the ensemble stream."""
        g = _f64(gvec)
        re = C.c_int()
        _check(lib.hc_step_device(self._h, float(t), _ptr(d_pose), _ptr(d_vel), _dp(g), _ptr(d_force), C.byref(re)))
        self.last_recomputed = bool(re.value)

    def components(self):
        shape = (self.batch, self.dofs)
        hs, rad, wv = np.empty(shape), np.empty(shape), np.empty(shape)
        _check(lib.hc_get_components(self._h, _dp(hs), _dp(rad), _dp(wv)))
        return hs, rad, wv

    def wave_force_at_time(self, t):
        """WaveBase::GetForceAtTime(t) for every instance: [B][6N]."""
        out = np.empty((self.batch, self.dofs))
        _check(lib.hc_waves_force_at_time(self._h, float(t), _dp(out)))
        return out

    def wave_kinematics(self, t, points, mwl=0.0, wheeler=False):
        """Water elevation, particle velocity and acceleration of every instance's wave at its own points
        (WaveBase::GetElevation / GetVelocity / GetAcceleration, on the device): points [B][P][3] ->
        (eta [B][P], vel [B][P][3], acc [B][P][3]).  Irregular eta is not ramped; see hc_waves_kinematics_at_time."""
        pts = _kin_points(points, self.batch)
        eta, vel, acc = _kin_outputs(pts)
        _check(lib.hc_waves_kinematics_at_time(self._h, float(t), pts.shape[1], _dp(pts), float(mwl), int(bool(wheeler)),
                                               _dp(eta), _dp(vel), _dp(acc)))
        return eta, vel, acc

    def wave_kinematics_device(self, t, n_points, d_points, d_eta=None, d_vel=None, d_acc=None, mwl=0.0, wheeler=False):
        """wave_kinematics on device buffers (torch CUDA tensors or raw addresses; any output may be None):
        d_points [B][n_points][3], d_eta [B][n_points], d_vel / d_acc [B][n_points][3]; asynchronous on the
        ensemble stream."""
        _check(lib.hc_waves_kinematics_at_time_device(self._h, float(t), int(n_points), _ptr(d_points), float(mwl),
                                                      int(bool(wheeler)), _ptr(d_eta), _ptr(d_vel), _ptr(d_acc)))

    def refresh_rirf(self):
        _check(lib.hc_ensemble_refresh_rirf(self._h))

    def sync(self):
        _check(lib.hc_sync(self._h))

    def join(self):
        """Orders the ensemble's stream after all look-ahead work enqueued so far on the library's side streams."""
        _check(lib.hc_ensemble_join(self._h))

    def lookahead_state(self):
        r, x = C.c_int(), C.c_int()
        _check(lib.hc_ensemble_lookahead_state(self._h, C.byref(r), C.byref(x)))
        return {"radiation": r.value, "excitation": x.value}

    def reset(self):
        _check(lib.hc_ensemble_reset(self._h))

    def set_bracket_snap(self, snap):
        _check(lib.hc_ensemble_set_bracket_snap(self._h, float(snap)))

    def history_len(self):
        return lib.hc_ensemble_history_len(self._h)

    def added_mass_mv(self, c, w, R):
        w, R = _f64(w), _f64(R).copy()
        n_sys = w.shape[-1]
        _check(lib.hc_added_mass_mv(self._h, n_sys, float(c), _ptr(w), _ptr(R)))
        return R

    def added_mass_mv_device(self, n_sys, c, d_w, d_R):
        _check(lib.hc_added_mass_mv_device(self._h, n_sys, float(c), _ptr(d_w), _ptr(d_R)))

    # -- profiling -----------------------------------------------------------
    def set_profiling(self, on=True):
        _check(lib.hc_set_profiling(self._h, int(on)))

    def profile(self):
        s = _capi.ProfileStats()
        _check(lib.hc_get_profile(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in _capi.ProfileStats._fields_}

    def kernel_ms(self, reset=True):
        v = [C.c_double() for _ in range(4)]
        _check(lib.hc_get_kernel_ms(self._h, *[C.byref(x) for x in v], int(reset)))
        return dict(zip(("prestep", "radiation", "excitation", "finalize"), [x.value for x in v]))

    def rad_lookahead_steps(self):
        """Steps per radiation look-ahead block (0: not active)."""
        return lib.hc_ensemble_rad_lookahead_steps(self._h)

    def rad_block_stats(self, reset=True):
        n, served, ms = C.c_longlong(), C.c_longlong(), C.c_double()
        _check(lib.hc_get_rad_block_stats(self._h, C.byref(n), C.byref(served), C.byref(ms), int(reset)))
        return {"launches": n.value, "steps_served": served.value, "avg_ms": ms.value}

    def close(self):
        if getattr(self, "_h", None):
            lib.hc_ensemble_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def multi_shard_range(total, shards, index):
    """Contiguous block [first, first + count) of global instance indices owned by shard `index`."""
    f, c = C.c_int(), C.c_int()
    lib.hc_multi_shard_range(int(total), int(shards), int(index), C.byref(f), C.byref(c))
    return f.value, c.value


class MultiEnsemble:
    """The instances of one ensemble partitioned over several GPUs of one node (hc_multi_*): one hc_ensemble and one
    host thread per device, contiguous shards, no exchange between devices on the step path."""

    def __init__(self, tables, batch, devices=None, dt_hint=0.0, bracket_snap=0.0, use_graph=True, exc_lookahead=0,
                 rad_kernel=0, rad_lookahead=0, rad_pass_mode=0):
        self.tables = tables
        o = _capi.EnsembleOpts()
        lib.hc_ensemble_default_opts(C.byref(o))
        o.batch, o.dt_hint, o.bracket_snap, o.use_graph = int(batch), dt_hint, bracket_snap, int(use_graph)
        o.exc_lookahead, o.rad_kernel, o.rad_lookahead, o.rad_pass_mode = int(exc_lookahead), int(rad_kernel), int(rad_lookahead), int(rad_pass_mode)
        if devices is None:
            devices = list(range(device_count()))
        dv = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        _check(lib.hc_multi_ensemble_create(tables._h, C.byref(o), dv, len(devices), C.byref(h)))
        self._h = h
        self.batch, self.dofs, self.devices = int(batch), tables.dofs, list(devices)

    def shards(self):
        out = []
        for i in range(lib.hc_multi_ensemble_num_shards(self._h)):
            d, f, c = C.c_int(), C.c_int(), C.c_int()
            _check(lib.hc_multi_ensemble_shard(self._h, i, C.byref(d), C.byref(f), C.byref(c), None))
            out.append({"device": d.value, "first": f.value, "count": c.value})
        return out

    def set_waves_none(self):
        _check(lib.hc_multi_waves_none(self._h))

    def set_waves_regular(self, amplitude, omega, phase=None):
        a, w = _f64(np.atleast_1d(amplitude)), _f64(np.atleast_1d(omega))
        p = _f64(np.atleast_1d(phase)) if phase is not None else None
        _check(lib.hc_multi_waves_regular(self._h, a.size, _dp(a), _dp(w), _dp(p)))

    def set_waves_irregular(self, dt, duration, ramp=0.0, Hs=0.0, Tp=0.0, fmin=0.001, fmax=1.0, nfreq=0, gamma=1.0,
                            is_normalized=False, seed=1, seeds=None, Hs_per_instance=None, Tp_per_instance=None):
        p = _capi.IrregularParams()
        lib.hc_irregular_default_params(C.byref(p))
        p.simulation_dt, p.simulation_duration, p.ramp_duration = dt, duration, ramp
        p.wave_height, p.wave_period, p.frequency_min, p.frequency_max = Hs, Tp, fmin, fmax
        p.nfrequencies, p.peak_enhancement_factor, p.is_normalized, p.seed = float(nfreq), gamma, int(is_normalized), int(seed)
        sd = np.ascontiguousarray(seeds, dtype=np.int32) if seeds is not None else None
        hs = _f64(Hs_per_instance) if Hs_per_instance is not None else None
        tp = _f64(Tp_per_instance) if Tp_per_instance is not None else None
        for a in (sd, hs, tp):
            if a is not None and a.size != self.batch:
                raise ValueError("per-instance arrays must have one entry per (global) instance")
        _check(lib.hc_multi_waves_irregular(self._h, C.byref(p), sd.ctypes.data_as(_capi.ip) if sd is not None else None,
                                            _dp(hs), _dp(tp)))

    def set_waves_series(self, dt, time, eta):
        """Imported free-surface elevation: time [n], eta [n] (shared) or [B][n] in global instance order."""
        t, e = _f64(time), _f64(eta)
        if t.ndim != 1 or e.shape[-1] != t.size or e.ndim not in (1, 2) or (e.ndim == 2 and e.shape[0] != self.batch):
            raise ValueError("time must be [n] and eta [n] or [batch][n]")
        _check(lib.hc_multi_waves_irregular_series(self._h, float(dt), t.size, _dp(t), _dp(e), int(e.ndim == 2)))

    def step(self, t, pose, vel, gvec=(0.0, 0.0, -9.81), out=None):
        """One lock-step of every instance on every device; host [B][6N] arrays in global instance order."""
        pose, vel, g = _f64(pose), _f64(vel), _f64(gvec)
        if pose.size != self.batch * self.dofs or vel.size != pose.size:
            raise ValueError("pose/vel must be [B][6N]")
        if out is None:
            out = np.empty((self.batch, self.dofs))
        re = C.c_int()
        _check(lib.hc_multi_step(self._h, float(t), _ptr(pose), _ptr(vel), _dp(g), _ptr(out), C.byref(re)))
        self.last_recomputed = bool(re.value)
        return out

    def step_device(self, t, d_pose, d_vel, d_force, gvec=(0.0, 0.0, -9.81)):
        """Device-resident step: per shard one device buffer [count_i][6N] on that shard's device (torch CUDA tensors
        or raw addresses); asynchronous on the shards' streams."""
        g = _f64(gvec)
        n = len(d_pose)
        arr = [(C.c_void_p * n)(*[_ptr(x).value for x in lst]) for lst in (d_pose, d_vel, d_force)]
        _check(lib.hc_multi_step_device(self._h, float(t), arr[0], arr[1], _dp(g), arr[2]))

    def wave_kinematics(self, t, points, mwl=0.0, wheeler=False):
        """Ensemble.wave_kinematics over every shard: points [B][P][3] in global instance order."""
        pts = _kin_points(points, self.batch)
        eta, vel, acc = _kin_outputs(pts)
        _check(lib.hc_multi_waves_kinematics_at_time(self._h, float(t), pts.shape[1], _dp(pts), float(mwl),
                                                     int(bool(wheeler)), _dp(eta), _dp(vel), _dp(acc)))
        return eta, vel, acc

    def components(self):
        shape = (self.batch, self.dofs)
        hs, rad, wv = np.empty(shape), np.empty(shape), np.empty(shape)
        _check(lib.hc_multi_get_components(self._h, _dp(hs), _dp(rad), _dp(wv)))
        return hs, rad, wv

    def sync(self):
        _check(lib.hc_multi_sync(self._h))

    def reset(self):
        _check(lib.hc_multi_reset(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib.hc_multi_ensemble_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()
