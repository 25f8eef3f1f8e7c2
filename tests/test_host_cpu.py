"""CPU-side tests of the product's host layer (no GPU, no compute kernels).

* the C-ABI library loads and exports every symbol include/hydrochrono_b200.h declares
* table staging (scalings, widths, added mass, TaperedDirect preprocessing) agrees with the oracle
* setup-time wave maths (spectra, dispersion, phases, IRF resampling) agrees with the oracle
* the built-in classic-HDF5 reader agrees with the independent pure-Python reader
* compute entry points fail loudly without a CUDA device (no CPU fallback)
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

import common
import hydrochrono_b200 as hc
from hydrochrono_b200 import _capi, synth
from oracle import hc_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "hydrochrono_b200.h")).read()
    declared = set(re.findall(r"HC_API[^;(]*?\b(hc_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 50
    lib = C.CDLL(_capi.LIB_PATH)
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    assert "sm_100a" in hc.version()


@pytest.fixture(scope="module")
def sphere():
    raw = common.sphere_raw()
    return raw, hc.Tables.from_raw(raw), orc.Tables(raw)


@pytest.fixture(scope="module")
def rm3():
    raw = synth.rm3_like()
    return raw, hc.Tables.from_raw(raw), orc.Tables(raw)


@pytest.mark.parametrize("which", ["sphere", "rm3"])
def test_tables_match_oracle(which, sphere, rm3):
    raw, T, O = sphere if which == "sphere" else rm3
    assert T.num_bodies == O.N and T.rirf_steps == O.L
    np.testing.assert_array_equal(T.rirf(), O.rirf())                 # rho * K, bitwise
    np.testing.assert_array_equal(T.rirf_width(), O.rirf_width())
    np.testing.assert_array_equal(T.added_mass(), O.added_mass())
    n_sys = O.D + 6                                                    # a non-hydro body appended to the system
    M = T.added_mass(n_sys)
    np.testing.assert_array_equal(M, O.added_mass(n_sys))
    assert np.all(M[O.D:, :] == 0) and np.all(M[:, O.D:] == 0)
    b0 = raw["bodies"][0]
    np.testing.assert_array_equal(T.lin_matrix(0), b0["lin_matrix"])
    np.testing.assert_array_equal(T.inf_added_mass(0), np.asarray(b0["inf_added_mass"]) * raw["rho"])
    assert T.hydrostatic_stiffness(0, 2, 2) == b0["lin_matrix"][2, 2] * raw["rho"] * raw["g"]
    assert T.disp_vol(0) == b0["disp_vol"]
    np.testing.assert_array_equal(T.cg(0), b0["cg"])
    np.testing.assert_array_equal(T.cb(0), b0["cb"])
    assert T.rirf_val(2, 2, 5) == O.rirf()[2, 2, 5]
    with pytest.raises(IndexError):                                    # std::out_of_range, hydro_forces.cpp:694-697
        T.rirf_val(O.D, 0, 0)
    with pytest.raises(IndexError):
        T.rirf_val(0, 0, O.L)


def test_rirf_time_vectors_must_agree():
    raw = synth.rm3_like()
    raw["bodies"][1]["rirf_t"] = raw["bodies"][1]["rirf_t"] + 1e-6
    with pytest.raises(hc.HydroError):                                 # h5fileinfo.cpp:329-343
        hc.Tables.from_raw(raw)


@pytest.mark.parametrize("opts", [
    dict(),                                                            # defaults: SG, 80..100 %, final 0
    dict(smoothing="savitzky_golay", rirf_end_time=9.0, taper_start_percent=0.6, taper_end_percent=0.9,
         taper_final_amplitude=0.2),                                   # f3of decay_dt3 style options
    dict(smoothing="moving_average", window_length=7),
])
def test_tapered_direct_matches_oracle(opts, sphere):
    raw, _, _ = sphere
    T, O = hc.Tables.from_raw(raw), orc.Tables(raw)
    T.set_convolution_mode("TaperedDirect", **opts)
    O.set_tapered(smoothing=opts.get("smoothing", "sg"), window_length=opts.get("window_length", 5),
                  rirf_end_time=opts.get("rirf_end_time", -1.0), start=opts.get("taper_start_percent", 0.8),
                  end=opts.get("taper_end_percent", 1.0), final=opts.get("taper_final_amplitude", 0.0))
    a, b = T.rirf(), O.rirf()
    np.testing.assert_array_equal(a, b)
    assert np.any(a != orc.Tables(raw).rirf())
    T.set_convolution_mode("Baseline")
    np.testing.assert_array_equal(T.rirf(), orc.Tables(raw).rirf())


def test_spectra_and_dispersion_match_oracle():
    f = orc.linspaced(1000, 0.001, 1.0)
    for Hs, Tp, gamma, norm in [(2.0, 12.0, 1.0, 0), (2.5, 8.0, 3.3, 0), (1.0, 6.0, 2.0, 1)]:
        S = np.empty_like(f)
        assert _capi.lib.hc_jonswap_spectrum_hz(f.size, f.ctypes.data_as(_capi.dp), Hs, Tp, gamma, norm,
                                                S.ctypes.data_as(_capi.dp)) == 0
        np.testing.assert_array_equal(S, orc.jonswap(f, Hs, Tp, gamma, bool(norm)))
        assert _capi.lib.hc_pierson_moskowitz_spectrum_hz(f.size, f.ctypes.data_as(_capi.dp), Hs, Tp,
                                                          S.ctypes.data_as(_capi.dp)) == 0
        np.testing.assert_array_equal(S, orc.pierson_moskowitz(f, Hs, Tp))
    k = C.c_double()
    for om, h in [(0.5, 200.0), (2.1, 50.0), (1.0, 0.0), (1.0, 2000.0), (0.3, float("inf")), (6.28, 10.0)]:
        assert _capi.lib.hc_compute_wave_number(om, h, 9.81, C.byref(k)) == 0
        assert k.value == orc.wave_number(om, h, 9.81)
        if 0 < h <= 1000:
            assert abs(om * om - 9.81 * k.value * np.tanh(k.value * h)) < 1e-5
    assert _capi.lib.hc_compute_wave_number(-1.0, 10.0, 9.81, C.byref(k)) != 0
    assert "positive" in _capi.lib.hc_last_error().decode()


def test_random_phases_match_std_distribution():
    for seed in (1, 2, 12345):
        p = np.empty(1000)
        _capi.lib.hc_random_phases(seed, p.size, p.ctypes.data_as(_capi.dp))
        np.testing.assert_array_equal(p, orc.phases(seed, p.size))
        np.testing.assert_array_equal(p, orc.phases(seed, p.size, stdlib=True))  # std::uniform_real_distribution
        assert 0 <= p.min() and p.max() < 2 * np.pi
    # first phase of seed 1: mt19937(1) draws 1791095845, 4282876139 -> (x0 + x1 * 2^32) / 2^64 * 2 pi
    expect = (1791095845 + 4282876139 * 2.0**32) / 2.0**64 * (2 * np.pi)
    assert orc.phases(1, 1)[0] == expect


def _resample(T, dt, body=0):
    n = C.c_int()
    assert _capi.lib.hc_resample_excitation_irf(T._h, dt, body, C.byref(n), None, None, None) == 0
    t, w, f = np.empty(n.value), np.empty(n.value), np.empty((6, n.value))
    dp = _capi.dp
    assert _capi.lib.hc_resample_excitation_irf(T._h, dt, body, C.byref(n), t.ctypes.data_as(dp),
                                                w.ctypes.data_as(dp), f.ctypes.data_as(dp)) == 0
    return t, w, f


def test_excitation_irf_resampling(sphere):
    raw, T, O = sphere
    t, w, f = _resample(T, common.SPHERE_DT)
    assert t.size == 8334                                              # SURVEY.md Appendix C
    inst = orc.Instance(O)
    inst.set_irregular(dt=common.SPHERE_DT, duration=10.0)             # Hs = 0: IRF vectors only
    ref = inst.irregular()["irf"][0]
    np.testing.assert_array_equal(t, ref["t"])
    np.testing.assert_array_equal(w, ref["w"])
    scale = np.abs(ref["f"]).max(axis=1, keepdims=True)
    assert np.abs(f - ref["f"]).max() <= 1e-12 * scale.max()           # two independent solvers of one system
    # third opinion: scipy's interpolating cubic B-spline with the same averaged knot vector
    from scipy.interpolate import make_interp_spline
    n0 = raw["bodies"][0]["exc_irf_t"].size
    u = np.linspace(0, 1, n0)
    knots = np.concatenate([[0.0] * 4, [(u[j] + u[j + 1] + u[j + 2]) / 3 for j in range(1, n0 - 3)], [1.0] * 4])
    y = np.asarray(raw["bodies"][0]["exc_irf_f"]).reshape(6, n0) * (raw["rho"] * raw["g"])
    spl = make_interp_spline(u, y.T, k=3, t=knots)
    fs = spl(np.linspace(0, 1, t.size)).T
    assert np.abs(f - fs).max() <= 1e-11 * scale.max()


def test_excitation_irf_resampling_two_bodies(rm3):
    raw, T, O = rm3
    inst = orc.Instance(O)
    inst.set_irregular(dt=0.01, duration=10.0)
    for b in range(2):
        t, w, f = _resample(T, 0.01, b)
        ref = inst.irregular()["irf"][b]
        assert t.size == 6000
        np.testing.assert_array_equal(t, ref["t"])
        assert np.abs(f - ref["f"]).max() <= 1e-12 * np.abs(ref["f"]).max()


@pytest.fixture(scope="module")
def sphere_h5(tmp_path_factory):
    """sphere.h5 as a BEMIO-layout file, written from the committed fixture of its datasets."""
    from hydrochrono_b200 import h5io
    f = tmp_path_factory.mktemp("h5") / "sphere.h5"
    h5io.write_bemio(f, common.sphere_raw())
    return str(f)


def test_h5_reader_against_python_reader_and_fixture(sphere_h5):
    from h5lite import load_bemio
    T = hc.Tables.from_h5(sphere_h5, 1)
    raw = load_bemio(sphere_h5, 1)
    O = orc.Tables(raw)
    np.testing.assert_array_equal(T.rirf(), O.rirf())
    np.testing.assert_array_equal(T.added_mass(), O.added_mass())
    np.testing.assert_array_equal(T.rirf_time(), raw["bodies"][0]["rirf_t"])
    assert (T.rho, T.g, T.water_depth) == (1000.0, 9.81, 200.0)
    assert T.disp_vol(0) == 261.724
    # the committed fixture is the same data
    fx = common.sphere_raw()
    np.testing.assert_array_equal(fx["bodies"][0]["rirf_K"], raw["bodies"][0]["rirf_K"])
    t, w, f = _resample(T, common.SPHERE_DT)
    t2, w2, f2 = _resample(hc.Tables.from_raw(fx), common.SPHERE_DT)
    np.testing.assert_array_equal(f, f2)


def test_h5_reader_errors(tmp_path, sphere_h5):
    with pytest.raises(hc.HydroError) as ei:
        hc.Tables.from_h5(str(tmp_path / "missing.h5"), 1)
    assert "Unable to open/read HDF5 hydro data file" in str(ei.value)   # h5fileinfo.cpp:172-181
    bad = tmp_path / "bad.h5"
    bad.write_bytes(b"not an hdf5 file" * 10)
    with pytest.raises(hc.HydroError):
        hc.Tables.from_h5(str(bad), 1)
    with pytest.raises(hc.HydroError):                                    # file holds one body only
        hc.Tables.from_h5(sphere_h5, 2)
    data = open(sphere_h5, "rb").read()
    trunc = tmp_path / "trunc.h5"
    trunc.write_bytes(data[: len(data) // 3])
    with pytest.raises(hc.HydroError):
        hc.Tables.from_h5(str(trunc), 1)


def test_no_cpu_fallback(sphere):
    """Without a CUDA device every compute entry point must fail loudly, never fall back to the host."""
    if hc.device_count() > 0:
        pytest.skip("CUDA device present")
    _, T, _ = sphere
    with pytest.raises(hc.HydroError) as ei:
        hc.Ensemble(T, batch=4)
    assert ei.value.status == 3 and "no CPU fallback" in str(ei.value)


def test_product_does_not_reference_the_oracle():
    """The oracle is test infrastructure: nothing under hydrochrono_b200/ or include/ may mention it."""
    bad = []
    for base in ("hydrochrono_b200", "include"):
        for dp_, _, files in os.walk(os.path.join(ROOT, base)):
            if "build" in dp_ or "__pycache__" in dp_:
                continue
            for fn in files:
                if fn.endswith((".so", ".o", ".pyc")):
                    continue
                txt = open(os.path.join(dp_, fn), errors="replace").read()
                if re.search(r"hc_oracle|libhc_oracle|from oracle|import oracle|orc_", txt):
                    bad.append(os.path.join(dp_, fn))
    assert not bad, bad


def test_multi_shard_ranges_and_no_device():
    """hc_multi_*: contiguous shards that differ by at most one instance (the same rule as shard.shard_range, which
    the torchrun ranks of bench.py use), and no CPU fallback for the multi-device handle either."""
    import hydrochrono_b200 as hc
    from hydrochrono_b200 import shard, synth
    for total in (7, 16384, 16385):
        for n in (1, 2, 3, 8):
            blocks = [hc.multi_shard_range(total, n, i) for i in range(n)]
            assert blocks == [(lo, hi - lo) for lo, hi in (shard.shard_range(total, n, r) for r in range(n))]
    if hc.device_count() == 0:
        T = hc.Tables.from_raw(synth.make_tables(num_bodies=1, rirf_steps=21, rirf_duration=1.0, exc_irf_steps=21,
                                                 exc_half_window=1.0))
        with pytest.raises(hc.HydroError) as ei:
            hc.MultiEnsemble(T, batch=8, devices=[0, 1])
        assert "no CPU fallback" in str(ei.value)
