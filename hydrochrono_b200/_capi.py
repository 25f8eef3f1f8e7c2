"""ctypes binding of include/hydrochrono_b200.h (libhydrochrono_b200.so, built in-tree by csrc/Makefile).

There is no fallback: if the shared library is missing the import of this module fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhydrochrono_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "hydrochrono_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
        "`make -C hydrochrono_b200/csrc`. There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
vp = C.c_void_p

HC_OK = 0
STATUS_NAMES = {0: "HC_OK", 1: "HC_ERR_INVALID", 2: "HC_ERR_OUT_OF_RANGE", 3: "HC_ERR_CUDA", 4: "HC_ERR_DUPLICATE_TIME",
                5: "HC_ERR_ETA_WINDOW", 6: "HC_ERR_IO", 7: "HC_ERR_TIME_ORDER", 8: "HC_ERR_CAPACITY"}


class TablesDesc(C.Structure):
    _fields_ = [("num_bodies", C.c_int), ("rirf_steps", C.c_int), ("num_freqs", C.c_int), ("exc_irf_steps", C.c_int),
                ("rho", C.c_double), ("g", C.c_double), ("water_depth", C.c_double),
                ("rirf_t", dp), ("rirf_K", dp), ("lin_matrix", dp), ("inf_added_mass", dp), ("disp_vol", dp),
                ("cg", dp), ("cb", dp), ("w", dp), ("exc_mag", dp), ("exc_phase", dp), ("exc_irf_t", dp),
                ("exc_irf_f", dp)]


class TaperedOpts(C.Structure):
    _fields_ = [("smoothing", C.c_char_p), ("window_length", C.c_int), ("rirf_end_time", C.c_double),
                ("taper_start_percent", C.c_double), ("taper_end_percent", C.c_double),
                ("taper_final_amplitude", C.c_double)]


class EnsembleOpts(C.Structure):
    _fields_ = [("device", C.c_int), ("batch", C.c_int), ("dt_hint", C.c_double), ("bracket_snap", C.c_double),
                ("rad_chunk", C.c_int), ("exc_chunk", C.c_int), ("use_graph", C.c_int), ("exc_lookahead", C.c_int),
                ("rad_kernel", C.c_int), ("rad_lookahead", C.c_int), ("rad_pass_mode", C.c_int), ("stream", vp)]


class IrregularParams(C.Structure):
    _fields_ = [("simulation_dt", C.c_double), ("simulation_duration", C.c_double), ("ramp_duration", C.c_double),
                ("wave_height", C.c_double), ("wave_period", C.c_double), ("frequency_min", C.c_double),
                ("frequency_max", C.c_double), ("nfrequencies", C.c_double), ("peak_enhancement_factor", C.c_double),
                ("is_normalized", C.c_int), ("seed", C.c_int)]


class ProfileStats(C.Structure):
    _fields_ = [("hydrostatics_seconds", C.c_double), ("radiation_seconds", C.c_double), ("waves_seconds", C.c_double),
                ("hydrostatics_calls", C.c_int), ("radiation_calls", C.c_int), ("waves_calls", C.c_int),
                ("eta_synthesis_seconds", C.c_double), ("step_seconds", C.c_double), ("kernel_launches", C.c_longlong)]


class SimPrismatic(C.Structure):
    _fields_ = [("child", C.c_int), ("parent", C.c_int), ("axis", C.c_double * 3)]


class SimTSDA(C.Structure):
    _fields_ = [("body1", C.c_int), ("body2", C.c_int), ("point1", C.c_double * 3), ("point2", C.c_double * 3),
                ("rest_length", C.c_double)]


class SimLinks(C.Structure):
    _fields_ = [("n_prismatic", C.c_int), ("n_tsda", C.c_int), ("prismatic", C.POINTER(SimPrismatic)),
                ("tsda", C.POINTER(SimTSDA)), ("tsda_damping", dp), ("tsda_stiffness", dp), ("tsda_energy", vp)]


class SimParams(C.Structure):
    _fields_ = [("scheme", C.c_int), ("t0", C.c_double), ("dt", C.c_double), ("n_steps", C.c_int),
                ("record_every", C.c_int), ("g", C.c_double * 3), ("mass", dp), ("inertia", dp), ("free_dof", ip),
                ("pto_damping", dp), ("pto_stiffness", dp), ("links", C.POINTER(SimLinks))]


# every symbol include/hydrochrono_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "hc_last_error": (C.c_char_p, []),
    "hc_version": (C.c_char_p, []),
    "hc_device_count": (C.c_int, []),
    "hc_tables_create": (C.c_int, [C.POINTER(TablesDesc), C.POINTER(vp)]),
    "hc_tables_load_h5": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(vp)]),
    "hc_tables_destroy": (None, [vp]),
    "hc_tables_num_bodies": (C.c_int, [vp]),
    "hc_tables_rirf_steps": (C.c_int, [vp]),
    "hc_tables_num_freqs": (C.c_int, [vp]),
    "hc_tables_exc_irf_steps": (C.c_int, [vp]),
    "hc_tables_rho": (C.c_double, [vp]),
    "hc_tables_g": (C.c_double, [vp]),
    "hc_tables_water_depth": (C.c_double, [vp]),
    "hc_tables_rirf_time": (C.c_int, [vp, dp]),
    "hc_tables_rirf_width": (C.c_int, [vp, dp]),
    "hc_tables_rirf_val": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, dp]),
    "hc_tables_rirf_all": (C.c_int, [vp, dp]),
    "hc_tables_lin_matrix": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_hydrostatic_stiffness": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, dp]),
    "hc_tables_inf_added_mass": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_disp_vol": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_cg": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_cb": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_freq_list": (C.c_int, [vp, dp]),
    "hc_tables_excitation_mag": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_excitation_phase": (C.c_int, [vp, C.c_int, dp]),
    "hc_tables_excitation_irf": (C.c_int, [vp, C.c_int, dp, dp]),
    "hc_tables_set_convolution_mode": (C.c_int, [vp, C.c_int, C.POINTER(TaperedOpts)]),
    "hc_added_mass": (C.c_int, [vp, C.c_int, dp]),
    "hc_ensemble_default_opts": (None, [C.POINTER(EnsembleOpts)]),
    "hc_ensemble_create": (C.c_int, [vp, C.POINTER(EnsembleOpts), C.POINTER(vp)]),
    "hc_ensemble_destroy": (None, [vp]),
    "hc_ensemble_batch": (C.c_int, [vp]),
    "hc_ensemble_dofs": (C.c_int, [vp]),
    "hc_ensemble_reset": (C.c_int, [vp]),
    "hc_ensemble_set_bracket_snap": (C.c_int, [vp, C.c_double]),
    "hc_ensemble_host_buffers": (C.c_int, [vp, C.POINTER(dp), C.POINTER(dp), C.POINTER(dp)]),
    "hc_waves_none": (C.c_int, [vp]),
    "hc_waves_regular": (C.c_int, [vp, C.c_int, dp, dp, dp]),
    "hc_irregular_default_params": (None, [C.POINTER(IrregularParams)]),
    "hc_waves_irregular": (C.c_int, [vp, C.POINTER(IrregularParams), ip, dp, dp]),
    "hc_waves_irregular_series": (C.c_int, [vp, C.c_double, C.c_int, dp, dp, C.c_int]),
    "hc_waves_irregular_sizes": (C.c_int, [vp, ip, ip, ip]),
    "hc_waves_irregular_spectrum": (C.c_int, [vp, C.c_int, dp, dp, dp, dp, dp]),
    "hc_waves_irregular_eta": (C.c_int, [vp, C.c_int, dp, dp]),
    "hc_waves_irregular_irf": (C.c_int, [vp, C.c_int, dp, dp, dp]),
    "hc_waves_regular_coeffs": (C.c_int, [vp, C.c_int, dp, dp, dp]),
    "hc_step": (C.c_int, [vp, C.c_double, vp, vp, dp, vp, ip]),
    "hc_step_device": (C.c_int, [vp, C.c_double, vp, vp, dp, vp, ip]),
    "hc_get_components": (C.c_int, [vp, dp, dp, dp]),
    "hc_waves_force_at_time": (C.c_int, [vp, C.c_double, dp]),
    "hc_waves_kinematics_at_time": (C.c_int, [vp, C.c_double, C.c_int, dp, C.c_double, C.c_int, dp, dp, dp]),
    "hc_waves_kinematics_at_time_device": (C.c_int, [vp, C.c_double, C.c_int, vp, C.c_double, C.c_int, vp, vp, vp]),
    "hc_ensemble_simulate": (C.c_int, [vp, C.POINTER(SimParams), dp, dp, dp, dp, dp, dp, ip]),
    "hc_ensemble_simulate_device": (C.c_int, [vp, C.POINTER(SimParams), vp, vp, vp, vp, vp, vp, ip]),
    "hc_ensemble_refresh_rirf": (C.c_int, [vp]),
    "hc_sync": (C.c_int, [vp]),
    "hc_ensemble_join": (C.c_int, [vp]),
    "hc_ensemble_lookahead_state": (C.c_int, [vp, ip, ip]),
    "hc_ensemble_history_len": (C.c_int, [vp]),
    "hc_added_mass_mv": (C.c_int, [vp, C.c_int, C.c_double, vp, vp]),
    "hc_added_mass_mv_device": (C.c_int, [vp, C.c_int, C.c_double, vp, vp]),
    "hc_set_profiling": (C.c_int, [vp, C.c_int]),
    "hc_get_profile": (C.c_int, [vp, C.POINTER(ProfileStats)]),
    "hc_get_kernel_ms": (C.c_int, [vp, dp, dp, dp, dp, C.c_int]),
    "hc_measure_fp64_peak": (C.c_int, [C.c_int, dp]),
    "hc_measure_fp64_mma_peak": (C.c_int, [C.c_int, dp]),
    "hc_rad_lookahead_plan": (C.c_int, [vp, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hc_rad_pass_next": (C.c_int, [C.c_longlong, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.c_int, C.c_longlong,
                                   C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "hc_rad_lookahead_row_kernel": (C.c_int, [vp, C.c_double, dp]),
    "hc_rad_lookahead_check_step": (C.c_int, [vp, C.c_double, C.c_double, dp, C.c_int, C.POINTER(C.c_int)]),
    "hc_ensemble_rad_lookahead_steps": (C.c_int, [vp]),
    "hc_get_rad_block_stats": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), dp, C.c_int]),
    "hc_get_exc_block_stats": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.c_int]),
    "hc_multi_shard_range": (None, [C.c_int, C.c_int, C.c_int, ip, ip]),
    "hc_multi_ensemble_create": (C.c_int, [vp, C.POINTER(EnsembleOpts), ip, C.c_int, C.POINTER(vp)]),
    "hc_multi_ensemble_destroy": (None, [vp]),
    "hc_multi_ensemble_num_shards": (C.c_int, [vp]),
    "hc_multi_ensemble_batch": (C.c_int, [vp]),
    "hc_multi_ensemble_shard": (C.c_int, [vp, C.c_int, ip, ip, ip, C.POINTER(vp)]),
    "hc_multi_waves_none": (C.c_int, [vp]),
    "hc_multi_waves_regular": (C.c_int, [vp, C.c_int, dp, dp, dp]),
    "hc_multi_waves_irregular": (C.c_int, [vp, C.POINTER(IrregularParams), ip, dp, dp]),
    "hc_multi_waves_irregular_series": (C.c_int, [vp, C.c_double, C.c_int, dp, dp, C.c_int]),
    "hc_multi_step": (C.c_int, [vp, C.c_double, vp, vp, dp, vp, ip]),
    "hc_multi_step_device": (C.c_int, [vp, C.c_double, C.POINTER(vp), C.POINTER(vp), dp, C.POINTER(vp)]),
    "hc_multi_waves_kinematics_at_time": (C.c_int, [vp, C.c_double, C.c_int, dp, C.c_double, C.c_int, dp, dp, dp]),
    "hc_multi_ensemble_simulate": (C.c_int, [vp, C.POINTER(SimParams), dp, dp, dp, dp, dp, dp, ip]),
    "hc_multi_get_components": (C.c_int, [vp, dp, dp, dp]),
    "hc_multi_sync": (C.c_int, [vp]),
    "hc_multi_reset": (C.c_int, [vp]),
    "hc_host_alloc": (vp, [C.c_size_t]),
    "hc_host_free": (None, [vp]),
    "hc_pierson_moskowitz_spectrum_hz": (C.c_int, [C.c_int, dp, C.c_double, C.c_double, dp]),
    "hc_jonswap_spectrum_hz": (C.c_int, [C.c_int, dp, C.c_double, C.c_double, C.c_double, C.c_int, dp]),
    "hc_compute_wave_number": (C.c_int, [C.c_double, C.c_double, C.c_double, dp]),
    "hc_resample_excitation_irf": (C.c_int, [vp, C.c_double, C.c_int, ip, dp, dp, dp]),
    "hc_random_phases": (C.c_int, [C.c_int, C.c_int, dp]),
    "hc_wave_kinematics": (C.c_int, [C.c_int, dp, dp, dp, dp, dp, C.c_double, C.c_double, C.c_double, C.c_int, dp, dp, dp]),
    "hc_h5_writer_create": (C.c_int, [C.POINTER(vp)]),
    "hc_h5_writer_destroy": (None, [vp]),
    "hc_h5_writer_put_group": (C.c_int, [vp, C.c_char_p]),
    "hc_h5_writer_put_f64": (C.c_int, [vp, C.c_char_p, C.c_int, C.POINTER(C.c_uint64), dp]),
    "hc_h5_writer_put_string": (C.c_int, [vp, C.c_char_p, C.c_char_p]),
    "hc_h5_writer_put_string_array": (C.c_int, [vp, C.c_char_p, C.c_int, C.POINTER(C.c_char_p)]),
    "hc_h5_writer_attr_string": (C.c_int, [vp, C.c_char_p, C.c_char_p, C.c_char_p]),
    "hc_h5_writer_attr_f64": (C.c_int, [vp, C.c_char_p, C.c_char_p, C.c_double]),
    "hc_h5_writer_save": (C.c_int, [vp, C.c_char_p]),
    "hc_h5_read_f64": (C.c_int, [C.c_char_p, C.c_char_p, ip, C.POINTER(C.c_uint64), dp, C.c_size_t]),
    "hc_h5_read_string": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]),
    "hc_h5_list": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args
