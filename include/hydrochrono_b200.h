/* =====================================================================================
 * hydrochrono_b200.h -- C ABI of the B200-native hydrodynamic force path.
 *
 * Drop-in boundary for HydroChrono's per-timestep force computation (reference paths are
 * relative to the HydroChrono source tree):
 *
 *   hc_tables_*        replaces  H5FileInfo::ReadH5Data / HydroData          src/h5fileinfo.cpp:27-91,309-343
 *                                + TestHydro ctor tables (widths, equilibrium) src/hydro_forces.cpp:170-216
 *                                + TestHydro::EnsureProcessedRIRF             src/hydro_forces.cpp:385-535
 *   hc_ensemble_*      replaces  TestHydro state (velocity history, cache)    include/hydroc/hydro_forces.h:286-340
 *   hc_waves_*         replaces  NoWave / RegularWave / IrregularWaves setup  src/wave_types.cpp:257-352,432-459,
 *                                                                             572-774
 *   hc_step*           replaces  TestHydro::CoordinateFuncForBody recompute:  src/hydro_forces.cpp:727-767
 *                                ComputeForceHydrostatics (:263-322), ComputeForceRadiationDampingConv (:537-691),
 *                                ComputeForceWaves (:713-725) -> WaveBase::GetForceAtTime
 *                                (src/wave_types.cpp:257-264,315-327,552-570,776-844)
 *   hc_added_mass*     replaces  ChLoadAddedMass ctor / ComputeJacobian / LoadIntLoadResidual_Mv
 *                                                                             src/chloadaddedmass.cpp:12-71
 *   hc_get_profile     replaces  TestHydro::GetProfileStats                   include/hydroc/hydro_forces.h:153-160,284
 *
 * One ensemble = B independent copies ("instances") of one TestHydro: same hydro tables, own body
 * state, own velocity history, own wave realisation.  B = 1 is the reference's single system.
 * All instances are stepped in lockstep (same t).  Everything is FP64.
 *
 * Conventions: plain pointers and sizes only.  Every function returns an hc_status (0 = ok);
 * hc_last_error() gives the thread-local message.  Exceptions the reference would throw map to
 * status codes (see each function).  Handles are not thread-safe: one host thread per handle.
 * There is NO CPU fallback: every compute entry point requires a CUDA device and fails with
 * HC_ERR_CUDA otherwise.
 * ===================================================================================== */
#ifndef HYDROCHRONO_B200_H
#define HYDROCHRONO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HC_API __attribute__((visibility("default")))

typedef enum hc_status {
    HC_OK = 0,
    HC_ERR_INVALID = 1,       /* bad argument / bad table shape                     (std::runtime_error)   */
    HC_ERR_OUT_OF_RANGE = 2,  /* index / frequency outside tables                   (std::out_of_range)    */
    HC_ERR_CUDA = 3,          /* CUDA runtime failure or no device                                          */
    HC_ERR_DUPLICATE_TIME = 4,/* radiation convolution evaluated twice at one time  hydro_forces.cpp:555-557*/
    HC_ERR_ETA_WINDOW = 5,    /* t - tau outside the precomputed eta window         wave_types.cpp:833-840  */
    HC_ERR_IO = 6,            /* cannot open / parse HDF5 file                      h5fileinfo.cpp:172-181  */
    HC_ERR_TIME_ORDER = 7,    /* time went backwards (history no longer bracketed)  hydro_forces.cpp:370    */
    HC_ERR_CAPACITY = 8       /* velocity-history ring too small for this dt                               */
} hc_status;

typedef struct hc_tables hc_tables;
typedef struct hc_ensemble hc_ensemble;

HC_API const char* hc_last_error(void);
HC_API const char* hc_version(void);
HC_API int hc_device_count(void);

/* ---------------------------------------------------------------------------------------
 * Hydro tables (HydroData).  Arrays are the RAW values of the BEMIO .h5 datasets, row-major:
 *   rirf_t [N][L], rirf_K [N][6][6N][L], lin_matrix [N][6][6], inf_added_mass [N][6][6N],
 *   disp_vol [N], cg/cb [N][3], w [nw], exc_mag/exc_phase [N][6][nw] (wave direction 0),
 *   exc_irf_t [N][Le0], exc_irf_f [N][6][Le0].
 * Scalings (x rho, x rho*g) are applied inside exactly where the reference applies them.
 * nw or Le0 may be 0 (no regular / irregular wave data).
 * ------------------------------------------------------------------------------------- */
typedef struct hc_tables_desc {
    int num_bodies;
    int rirf_steps;          /* L   */
    int num_freqs;           /* nw  */
    int exc_irf_steps;       /* Le0 */
    double rho, g, water_depth;   /* water_depth may be +inf ("infinite" in the file) */
    const double* rirf_t;
    const double* rirf_K;
    const double* lin_matrix;
    const double* inf_added_mass;
    const double* disp_vol;
    const double* cg;
    const double* cb;
    const double* w;
    const double* exc_mag;
    const double* exc_phase;
    const double* exc_irf_t;
    const double* exc_irf_f;
} hc_tables_desc;

HC_API hc_status hc_tables_create(const hc_tables_desc* desc, hc_tables** out);
/* H5FileInfo(file, num_bodies).ReadH5Data(): built-in classic-HDF5 reader, no libhdf5. */
HC_API hc_status hc_tables_load_h5(const char* path, int num_bodies, hc_tables** out);
HC_API void hc_tables_destroy(hc_tables* t);

/* HydroData getters (include/hydroc/h5fileinfo.h:102-225) */
HC_API int hc_tables_num_bodies(const hc_tables* t);
HC_API int hc_tables_rirf_steps(const hc_tables* t);                 /* GetRIRFDims(2) */
HC_API int hc_tables_num_freqs(const hc_tables* t);
HC_API int hc_tables_exc_irf_steps(const hc_tables* t);
HC_API double hc_tables_rho(const hc_tables* t);                     /* GetRhoVal */
HC_API double hc_tables_g(const hc_tables* t);
HC_API double hc_tables_water_depth(const hc_tables* t);
HC_API hc_status hc_tables_rirf_time(const hc_tables* t, double* out /*[L]*/);       /* GetRIRFTimeVector */
HC_API hc_status hc_tables_rirf_width(const hc_tables* t, double* out /*[L]*/);      /* hydro_forces.cpp:181-190 */
/* TestHydro::GetRIRFval(row, col, st): rho-scaled (or TaperedDirect-processed) kernel value */
HC_API hc_status hc_tables_rirf_val(const hc_tables* t, int row, int col, int st, double* out);
HC_API hc_status hc_tables_rirf_all(const hc_tables* t, double* out /*[6N][6N][L]*/);
HC_API hc_status hc_tables_lin_matrix(const hc_tables* t, int body, double* out /*[36]*/);   /* GetLinMatrix */
HC_API hc_status hc_tables_hydrostatic_stiffness(const hc_tables* t, int body, int i, int j, double* out);
HC_API hc_status hc_tables_inf_added_mass(const hc_tables* t, int body, double* out /*[6][6N], x rho*/);
HC_API hc_status hc_tables_disp_vol(const hc_tables* t, int body, double* out);
HC_API hc_status hc_tables_cg(const hc_tables* t, int body, double* out /*[3]*/);
HC_API hc_status hc_tables_cb(const hc_tables* t, int body, double* out /*[3]*/);
/* HydroData::RegularWaveInfo / IrregularWaveInfo (include/hydroc/h5fileinfo.h:60-72), scaled as the reference
 * scales them at load time (mag x rho*g, IRF x rho*g). */
HC_API hc_status hc_tables_freq_list(const hc_tables* t, double* out /*[nw]*/);
HC_API hc_status hc_tables_excitation_mag(const hc_tables* t, int body, double* out /*[6][nw]*/);
HC_API hc_status hc_tables_excitation_phase(const hc_tables* t, int body, double* out /*[6][nw]*/);
HC_API hc_status hc_tables_excitation_irf(const hc_tables* t, int body, double* time /*[Le0]*/, double* f /*[6][Le0]*/);

/* TestHydro::SetRadiationConvolutionMode + SetTaperedDirectOptions (hydro_forces.h:233-265).
 * mode 0 = Baseline, 1 = TaperedDirect.  smoothing: "moving_average" selects the moving average, anything else
 * the 5-point Savitzky-Golay branch (hydro_forces.cpp:433-457).  Must be called before ensembles are created. */
typedef struct hc_tapered_opts {
    const char* smoothing;
    int window_length;
    double rirf_end_time;
    double taper_start_percent;
    double taper_end_percent;
    double taper_final_amplitude;
} hc_tapered_opts;
HC_API hc_status hc_tables_set_convolution_mode(hc_tables* t, int mode, const hc_tapered_opts* opts);

/* ChLoadAddedMass (src/chloadaddedmass.cpp:12-52): the 6N x 6N infinite-frequency added-mass matrix,
 * zero-padded to n_sys x n_sys with the block at (0,0).  n_sys >= 6N.  Host table op. */
HC_API hc_status hc_added_mass(const hc_tables* t, int n_sys, double* M_out /*[n_sys][n_sys]*/);

/* ---------------------------------------------------------------------------------------
 * Ensemble
 * ------------------------------------------------------------------------------------- */
typedef struct hc_ensemble_opts {
    int device;               /* CUDA device ordinal */
    int batch;                /* B, number of instances on this device */
    double dt_hint;           /* expected step size; sizes the velocity-history ring (rirf window / dt + slack).
                                 <= 0: ring sized for rirf_t spacing. The ring grows on demand.          */
    double bracket_snap;      /* 0 = bit-faithful bracketing (==, as the reference).  > 0: a convolution query
                                 time within snap*(t_newer - t_older) of a history sample is treated as an exact
                                 hit (skips reading the second, ~zero-weight row).  See DESIGN.md.      */
    int rad_chunk;            /* radiation lags per CTA (0 = auto)   */
    int exc_chunk;            /* excitation lags per CTA (0 = auto)  */
    int use_graph;            /* 1: capture the per-step kernel sequence in a CUDA graph (default 1) */
    int exc_lookahead;        /* irregular waves: 0 = auto (on when dt_hint > 0 and the batch fills the GPU), 1 = off,
                                 2 = on, blocks built in the step's stream (FMA-pipe kernel), 3 = next block built on a
                                 low-priority side stream, 4 / 5 = like 2 / 3 with the FP64 tensor-core (DMMA) kernel
                                 (5: the background build is launched in two halves, 4 steps apart, so that the
                                 look-ahead work is spread evenly over the steps).  The wave force is state-independent, so it is evaluated for the predicted
                                 times t, t+dt, ... of the next 8 steps in one pass over eta (t advanced by repeated
                                 addition of dt_hint, as Chrono advances ChTime); a step whose time is not bitwise
                                 equal to the prediction falls back to / rebuilds from the actual time, so results
                                 never depend on the prediction being right. */
    int rad_kernel;           /* radiation kernel for 6N = 12: 0 = auto (currently the FP64 FMA-pipe kernel), 1 = FMA pipe,
                                 2 = FP64 tensor cores (DMMA m8n8k4; 12 rows padded to 16: lower power, slower),
                                 3 = both engines: rows 0..7 on the tensor cores, rows 8..11 on the FMA pipe.
                                 Other body counts always use the FMA-pipe kernels. */
    int rad_lookahead;        /* radiation look-ahead for 6N = 6, 12, 18: the share of the resident history rows in the
                                 next (predicted) steps' convolutions is evaluated in one pass over the history on the
                                 FP64 tensor cores, 1/8 of the per-step HBM traffic.  RIRF lag spacing = m dt_hint with
                                 an integer m <= 8: blocks of 8 m steps on the lag grid.  Any other ratio: blocks of 8
                                 steps with a row-grid kernel (the velocity interpolation weights at the nominal lag
                                 positions t_rirf / dt_hint folded into K), used once the history window is full.
                                 A step is served from a block only if its time matches the prediction bitwise and
                                 every lag sits within bracket_snap (in rows) of its nominal position; other steps run
                                 the per-step kernel.  0 = auto (on for large ensembles with bracket_snap > 0), 1 = off,
                                 2 = on (each block is evaluated one block ahead, one slice per step on a side
                                 stream), 3 = on, whole pass in the main stream at the block's first step */
    int rad_pass_mode;        /* how the pass of the radiation block evaluated ahead is paced on its side stream: 0 = auto
                                 (= 1), 1 = one slice per step, each gated by its step's forces, 2 = one slice per step,
                                 not gated (two driver calls per step), 3 = the whole pass at the block's first step (one
                                 launch per block; k_step competes with resident pass CTAs for SM slots) */
    void* stream;             /* cudaStream_t to run on (NULL = ensemble creates its own non-blocking stream) */
} hc_ensemble_opts;

HC_API void hc_ensemble_default_opts(hc_ensemble_opts* o);
HC_API hc_status hc_ensemble_create(const hc_tables* t, const hc_ensemble_opts* opts, hc_ensemble** out);
HC_API void hc_ensemble_destroy(hc_ensemble* e);
HC_API int hc_ensemble_batch(const hc_ensemble* e);
HC_API int hc_ensemble_dofs(const hc_ensemble* e);      /* 6N */
/* Drops the velocity history, the time cache and the orientations kept by hc_ensemble_simulate (a fresh TestHydro),
 * keeps the waves. */
HC_API hc_status hc_ensemble_reset(hc_ensemble* e);
/* Changes hc_ensemble_opts.bracket_snap for the following steps (0 = bit-faithful bracketing). */
HC_API hc_status hc_ensemble_set_bracket_snap(hc_ensemble* e, double snap);
/* Pinned host staging owned by the ensemble ([B][6N] each).  Filling/reading these in place makes hc_step
 * copy-free on the host side. */
HC_API hc_status hc_ensemble_host_buffers(hc_ensemble* e, double** pose, double** vel, double** force);

/* ---- waves (TestHydro::AddWaves, src/hydro_forces.cpp:244-261) ---- */
HC_API hc_status hc_waves_none(hc_ensemble* e);                               /* NoWave */
/* RegularWave (src/wave_types.cpp:266-352).  Arrays have length B, or stride 0 semantics when count == 1
 * (one wave shared by all instances). */
HC_API hc_status hc_waves_regular(hc_ensemble* e, int count, const double* amplitude, const double* omega,
                                  const double* phase /* may be NULL -> 0 */);
/* IrregularWaves(IrregularWaveParams) (include/hydroc/wave_types.h:277-292, src/wave_types.cpp:430-459). */
typedef struct hc_irregular_params {
    double simulation_dt;
    double simulation_duration;
    double ramp_duration;
    double wave_height;              /* Hs */
    double wave_period;              /* Tp */
    double frequency_min;            /* default 0.001 */
    double frequency_max;            /* default 1.0   */
    double nfrequencies;             /* 0 = ceil((fmax-fmin)*duration) */
    double peak_enhancement_factor;  /* gamma, default 1.0 */
    int is_normalized;
    int seed;                        /* default 1; ignored when per-instance seeds are given */
} hc_irregular_params;
HC_API void hc_irregular_default_params(hc_irregular_params* p);
/* seeds: NULL (every instance uses p->seed) or [B] (instance b uses std::mt19937(seeds[b])).
 * wave_height / wave_period: NULL (shared p->...) or [B] per-instance sea states.
 * Synthesises eta for every instance on the device (src/wave_types.cpp:27-59,717-774). */
HC_API hc_status hc_waves_irregular(hc_ensemble* e, const hc_irregular_params* p, const int* seeds,
                                    const double* wave_height, const double* wave_period);
/* SURVEY a16 -- free-surface elevation imported as a (time, eta) series instead of synthesised from a spectrum
 * (IrregularWaves::ReadEtaFromFile, src/wave_types.cpp:480-500, called from InitializeIRFVectors :451-453 when
 * IrregularWaveParams::eta_file_path_ is set).  time[n] strictly increasing (the grid the excitation convolution
 * interpolates on; the reference snapshot leaves that grid empty on this branch, :784-785 -- the file's time column is
 * the intended one); eta is [n], shared by every instance, or [B][n] when per_instance != 0.  simulation_dt is the
 * spacing the excitation IRF is resampled to (ResampleIRF, :572-606).  hc_waves_irregular_spectrum then fails as
 * IrregularWaves::GetSpectrum does (:461-467); hc_waves_irregular_eta returns the series. */
HC_API hc_status hc_waves_irregular_series(hc_ensemble* e, double simulation_dt, int n, const double* time,
                                           const double* eta, int per_instance);
/* Introspection of the irregular-wave setup (IrregularWaves::GetSpectrum / GetFreeSurfaceElevation /
 * GetFreeSurfaceTime / GetFrequenciesHz, wave_types.h:300-309). */
HC_API hc_status hc_waves_irregular_sizes(const hc_ensemble* e, int* nfreq, int* n_eta, int* exc_steps /*[N]*/);
HC_API hc_status hc_waves_irregular_spectrum(const hc_ensemble* e, int instance, double* freqs_hz, double* S,
                                             double* widths, double* phases, double* wavenumbers); /* any NULL */
HC_API hc_status hc_waves_irregular_eta(const hc_ensemble* e, int instance, double* eta_t, double* eta); /* D2H */
HC_API hc_status hc_waves_irregular_irf(const hc_ensemble* e, int body, double* t, double* width,
                                        double* f /*[6][Le]*/);
HC_API hc_status hc_waves_regular_coeffs(const hc_ensemble* e, int instance, double* mag /*[6N]*/,
                                         double* phase /*[6N]*/, double* wavenumber);

/* ---- per-step force (TestHydro::CoordinateFuncForBody, src/hydro_forces.cpp:727-767) ----
 * pose  [B][6N]: per body (x, y, z, Cardan-XYZ roll, pitch, yaw)   -- GetPos(), GetRot().GetCardanAnglesXYZ()
 * vel   [B][6N]: per body (GetPosDt(), GetAngVelParent())
 * g_vec [3]    : system gravitational acceleration vector
 * force [B][6N]: total = hydrostatic - radiation + waves
 * Calling twice with the same t returns the cached forces (status HC_OK, *recomputed = 0), like the reference's
 * time-keyed cache; a new t appends (t, vel) to the history and recomputes.
 * Host-pointer version: H2D, kernels, D2H, synchronous at return.  Pinned buffers are recommended. */
HC_API hc_status hc_step(hc_ensemble* e, double t, const double* pose, const double* vel, const double g_vec[3],
                         double* force, int* recomputed /* may be NULL */);
/* Device-pointer version: pointers are device memory on the ensemble's device; asynchronous on the
 * ensemble's stream (use hc_sync or the caller's own stream ordering). */
HC_API hc_status hc_step_device(hc_ensemble* e, double t, const double* d_pose, const double* d_vel,
                                const double g_vec[3], double* d_force, int* recomputed);
/* Components of the last evaluation (ComputeForceHydrostatics / RadiationDampingConv / Waves), host [B][6N]
 * each; any may be NULL. */
HC_API hc_status hc_get_components(hc_ensemble* e, double* hydrostatic, double* radiation, double* waves);
/* WaveBase::GetForceAtTime(t) (src/wave_types.cpp:257-264,315-327,552-570) for every instance, host [B][6N]:
 * the wave excitation force alone at an arbitrary time; does not touch the velocity history or the force cache. */
HC_API hc_status hc_waves_force_at_time(hc_ensemble* e, double t, double* waves);
/* Water kinematics of every instance's own wave at its own points: WaveBase::GetElevation / GetVelocity /
 * GetAcceleration (src/wave_types.cpp:14-160,301-313,515-550) evaluated on the device (k_wave_kinematics).
 * points [B][P][3] (x, y, z) in, eta [B][P], velocity and acceleration [B][P][3] out; any output may be NULL.
 * - NoWave (hc_waves_none, a fresh ensemble), an imported eta series (hc_waves_irregular_series) or irregular waves
 *   without a sea state: every output is zero (the reference sums over empty component vectors).
 * - Regular waves: the instance's amplitude, omega, phase and wavenumber; Wheeler stretching is never applied.
 * - Irregular waves: the nf spectral components, amplitudes sqrt(2 S df) and phases of the instance.  eta is NOT
 *   ramped (GetEtaIrregular has no ramp), so during the ramp it differs from the synthesised series that
 *   hc_waves_irregular_eta returns; at x = 0 after the ramp it equals that series' samples bit for bit.  With
 *   wheeler_stretching != 0, velocity and acceleration are taken at z' = depth (z - mwl - eta) / (depth + eta).
 * - Deep-water branch per component when 2 pi / k > depth or k depth > 500, finite depth otherwise.
 * Any t is allowed: the call reads no eta window and no history, touches no force cache and is not a force
 * evaluation.  The first call after the waves were set stages the components on the device (irregular waves:
 * per-instance phases, and per-instance amplitudes when the sea state is per instance, 8 nf B bytes each); they are
 * released when the waves are set again or the ensemble is destroyed.
 * n_points < 1 or points == NULL: HC_ERR_INVALID.  Synchronous at return. */
HC_API hc_status hc_waves_kinematics_at_time(hc_ensemble* e, double t, int n_points, const double* points,
                                             double mwl, int wheeler_stretching,
                                             double* eta, double* velocity, double* acceleration);
/* The same with device pointers on the ensemble's device, asynchronous on the ensemble's stream. */
HC_API hc_status hc_waves_kinematics_at_time_device(hc_ensemble* e, double t, int n_points, const double* d_points,
                                                    double mwl, int wheeler_stretching,
                                                    double* d_eta, double* d_velocity, double* d_acceleration);
/* ---- device-side stepping of the ensemble's bodies ----
 * Advances every instance n_steps on the device: per step the force evaluation of hc_step_device, then one integrator
 * kernel (k_body_step), no host synchronisation inside the loop.  Rigid bodies with 6 DoF each, every DoF free or locked
 * to ground; forces = hydro + m g on translations + an optional linear PTO per instance and DoF,
 * -k (x - x_init) - c v.  Mass matrix = diag(m, m, m, Ixx, Iyy, Izz) per body + the infinite-frequency added mass
 * (hc_added_mass), restricted to the free DoFs, inverted once on the host per call.  Prismatic joints and translational
 * spring-dampers (the RM3 float / spar pair and its PTO) are covered through hc_sim_params.links (below).  Revolute
 * joints, rotational spring-dampers, chains of joints, contact and mooring are not covered: step those with Chrono.
 * The schemes follow the chrono_compat stepper (hydrochrono_b200/host/src/chrono_compat.cpp) operation for operation:
 *   scheme 0, linearised Euler (ChSystem::StepEnd): forces at (t_n, x_n, v_n); v += dt a (locked DoFs: v = 0);
 *     x += dt v; q <- normalize(QuatFromAngleAxis(|w dt|, w / |w|) q).
 *   scheme 1, HHT-alpha with alpha = -0.2 (StepHHTBegin / StepHHTEnd): initial accelerations from the force at t0; the
 *     force at t_{n+1} is evaluated at the predictor state (whose velocity enters the radiation history); the corrector
 *     balances (1 + alpha) F_{n+1} - alpha F_n.  F_n and a_n stay on the device.  HHT evaluates n_steps + 1 forces.
 * The device keeps one quaternion per body; the initial Cardan XYZ angles (roll, pitch, yaw) map to
 * q = qx(roll) qy(pitch) qz(yaw), and the pose given to the force path and returned is (pos, GetCardanAnglesXYZ(q)).
 * Times advance by repeated addition (t += dt), as Chrono advances ChTime.
 * A second call with t0 equal to the previous end time continues the run: the orientation of a body whose given angles
 * equal those of the ensemble's last quaternion bit for bit is kept, so Euler split into calls is bitwise identical to
 * one call (without PTO springs, whose rest pose is each call's initial pose).  The rule applies only to such a
 * continuation: after hc_ensemble_reset every orientation is built from the given angles, as in a fresh ensemble.
 * HHT restarts its acceleration history from the (time-cached) force at t0, as a freshly set-up ChSystem would.
 * Arrays of hc_sim_params are host memory (copied at the call).  pto_energy = sum over the call's steps of
 * c v_eval^2 dt per DoF, v_eval being the velocity of that step's force evaluation (the absorbed energy of a linear
 * damper PTO; / (n_steps dt) gives the mean absorbed power).  Any output may be NULL.
 * Errors of the force path (HC_ERR_ETA_WINDOW, HC_ERR_DUPLICATE_TIME, ...; all detected when a step is enqueued) end the
 * run with that status: *steps_done = completed steps, pose / vel hold the state after the last completed step, the
 * records and energy cover the completed steps.  HC_ERR_INVALID: n_steps < 1, record_every < 1, dt <= 0, mass or
 * inertia NULL, pose or vel NULL, a singular free-DoF mass matrix.
 *
 * Joints and spring-dampers (links != NULL with at least one joint or spring-damper; a NULL or empty links struct runs
 * the path above unchanged, bit for bit).  They follow the chrono_compat stepper's reduced coordinates
 * (ChSystem::Assemble / SolveAccelerations / ProjectOntoJoints) operation for operation, in one device kernel
 * (k_body_step_linked):
 *   - Prismatic joint to a moving parent B: the child A keeps one slide DoF along the joint axis n.  The columns of T
 *     are the free DoFs of every root body (a body that is nobody's child), then one slide per child;
 *     vA = vB + wB x rho + sd n, wA = wB (rho = xA - xB), with the bias wB x (wB x rho) + 2 sd wB x n.  Per step
 *     (T^T M T) qdd = T^T (rhs - M bias) is solved by partial-pivot Gaussian elimination and a = bias + T qdd, with
 *     M = diag(m, m, m, Ixx, Iyy, Izz) per body + A_inf over all 6N DoFs.
 *   - Prismatic joint to ground (parent = -1): vA = sd n, wA = 0 (the reference's sphere demos).
 *   - After every position / velocity update (the Euler update, the HHT predictor and the HHT corrector) each child is
 *     projected onto its joint: orientation q_parent rel_rot, transverse offset from the parent, slide kept, velocity
 *     vB + wB x rho + sd n.  The initial state is not projected.
 *   - Spring-damper: force -(k (l - rest) + c dl/dt) along the line between the two attachment points at the
 *     evaluation state, applied with its moment s x f to both bodies.  tsda_energy = sum over the call's steps of
 *     c (dl/dt)^2 dt with dl/dt of that step's force evaluation (the convention of pto_energy).
 *   - Assembly data (each joint's offset in the parent frame, relative rotation and axis in the parent frame; each
 *     spring-damper's body-frame points and rest length) are derived per instance from its initial pose.  They are
 *     kept by a continuation call -- the instance's given pose equals, bit for bit, the pose the previous call ended
 *     in, and the links are the same -- so that Euler with links split into calls is bitwise identical to one call;
 *     otherwise, and after hc_ensemble_reset, they are derived again.
 *   - free_dof selects the DoFs of root bodies; pto_damping / pto_stiffness and gravity add to the generalised force
 *     before it is projected through T^T.
 * HC_ERR_INVALID (checked on the host at the call, before anything runs): a body index out of range; child == parent;
 * a second joint on one child; a chain (a parent that is itself a child); a zero axis; more than HC_SIM_MAX_TSDA
 * spring-dampers; a spring-damper with body1 == body2 or between ground and ground; a jointed child with a locked DoF;
 * a mass matrix diag(m, I) + A_inf whose symmetric part is not positive definite (which keeps every T^T M T
 * nonsingular).
 * Callers must zero-initialise hc_sim_params (hc_sim_params p{} in C++, memset in C): fields added at its end read as
 * "absent" when zero. */
#define HC_SIM_MAX_TSDA 16
typedef struct hc_sim_prismatic {   /* ChLinkLockPrismatic */
    int child, parent;              /* body indices; parent = -1: ground */
    double axis[3];                 /* joint axis in the world frame at assembly (the z axis of the joint frame) */
} hc_sim_prismatic;
typedef struct hc_sim_tsda {        /* ChLinkTSDA */
    int body1, body2;               /* body index, -1: ground */
    double point1[3], point2[3];    /* attachment points, world frame at assembly */
    double rest_length;             /* < 0: the length at assembly (ChLinkTSDA::Initialize) */
} hc_sim_tsda;
typedef struct hc_sim_links {
    int n_prismatic, n_tsda;
    const hc_sim_prismatic* prismatic;
    const hc_sim_tsda* tsda;
    const double* tsda_damping;     /* [B][n_tsda] or NULL (0) */
    const double* tsda_stiffness;   /* [B][n_tsda] or NULL (0) */
    double* tsda_energy;            /* [B][n_tsda] out or NULL; host or device memory, matching the call variant */
} hc_sim_links;
typedef struct hc_sim_params {
    int scheme;                 /* 0 = linearised Euler, 1 = HHT-alpha (alpha = -0.2) */
    double t0, dt;
    int n_steps, record_every;  /* record k = state after step (k+1)*record_every, k < n_steps / record_every */
    double g[3];
    const double* mass;         /* [N] */
    const double* inertia;      /* [N][3], diagonal (ChBody::SetInertiaXX) */
    const int* free_dof;        /* [6N] 1 free / 0 locked to ground; NULL = all free */
    const double* pto_damping;  /* [B][6N] or NULL */
    const double* pto_stiffness;/* [B][6N] or NULL; spring about the instance's initial pose */
    const hc_sim_links* links;  /* NULL: free / ground-locked bodies only */
} hc_sim_params;
/* Host buffers: pose / vel [B][6N] (in: initial state, out: final state), rec_t [n_rec], rec_pose / rec_vel
 * [n_rec][B][6N], pto_energy [B][6N].  Records go through a device buffer of bounded size, copied out in chunks.
 * Synchronous at return. */
HC_API hc_status hc_ensemble_simulate(hc_ensemble* e, const hc_sim_params* p, double* pose, double* vel, double* rec_t,
                                      double* rec_pose, double* rec_vel, double* pto_energy, int* steps_done);
/* The same with pose, vel, rec_t, rec_pose, rec_vel and pto_energy as device pointers on the ensemble's device;
 * asynchronous on the ensemble's stream (hc_sync waits). */
HC_API hc_status hc_ensemble_simulate_device(hc_ensemble* e, const hc_sim_params* p, double* d_pose, double* d_vel,
                                             double* d_rec_t, double* d_rec_pose, double* d_rec_vel, double* d_pto_energy,
                                             int* steps_done);
/* Re-stage the radiation kernel after hc_tables_set_convolution_mode() changed the ensemble's tables. */
HC_API hc_status hc_ensemble_refresh_rirf(hc_ensemble* e);
HC_API hc_status hc_sync(hc_ensemble* e);
/* Orders the ensemble's stream after every look-ahead pass enqueued so far on the library's side streams (no host
 * wait).  A caller that times device-resident stepping with events on the ensemble's stream calls this before each
 * event so that the interval contains all the work the steps in between gave rise to. */
HC_API hc_status hc_ensemble_join(hc_ensemble* e);
/* Whether the radiation / excitation look-ahead paths are armed (1), configured but switched off by the misprediction
 * heuristic (0: irregular step sizes; hc_ensemble_reset or hc_ensemble_set_bracket_snap arm them again) or not
 * configured at all (-1). */
HC_API hc_status hc_ensemble_lookahead_state(const hc_ensemble* e, int* radiation, int* excitation);
HC_API int hc_ensemble_history_len(const hc_ensemble* e);

/* ChLoadAddedMass::LoadIntLoadResidual_Mv (src/chloadaddedmass.cpp:55-71), batched: R[b] += c * M_sys * w[b]
 * for every instance.  w, R host [B][n_sys]. */
HC_API hc_status hc_added_mass_mv(hc_ensemble* e, int n_sys, double c, const double* w, double* R);
HC_API hc_status hc_added_mass_mv_device(hc_ensemble* e, int n_sys, double c, const double* d_w, double* d_R);

/* HydroProfileStats (include/hydroc/hydro_forces.h:153-160), fed by CUDA events. */
typedef struct hc_profile_stats {
    double hydrostatics_seconds;
    double radiation_seconds;
    double waves_seconds;
    int hydrostatics_calls;
    int radiation_calls;
    int waves_calls;
    double eta_synthesis_seconds;   /* one-off, hc_waves_irregular */
    double step_seconds;            /* whole per-step kernel sequence */
    long long kernel_launches;      /* kernels of this library launched so far */
} hc_profile_stats;
/* enable = 1 inserts CUDA events around each kernel group (adds sync cost at read time only). */
HC_API hc_status hc_set_profiling(hc_ensemble* e, int enable);
HC_API hc_status hc_get_profile(hc_ensemble* e, hc_profile_stats* out);
/* Average device time (ms) of the radiation / excitation / finalize kernels since the last call (needs profiling). */
HC_API hc_status hc_get_kernel_ms(hc_ensemble* e, double* prestep_ms, double* radiation_ms, double* excitation_ms,
                                  double* finalize_ms, int reset);

/* Radiation look-ahead (hc_ensemble_opts.rad_lookahead): steps per block (8 m, m = RIRF lag spacing / dt_hint), 0 when
   the path is not configured or switched itself off.  hc_get_rad_block_stats: k_rad_block<12> launches so far, how many
   steps they served, and the average launch duration in ms over the launches timed while profiling was on. */
HC_API int hc_ensemble_rad_lookahead_steps(const hc_ensemble* e);
HC_API hc_status hc_get_rad_block_stats(hc_ensemble* e, long long* launches, long long* steps_served, double* avg_ms,
                                        int reset);
/* Excitation look-ahead (hc_ensemble_opts.exc_lookahead): blocks of wave forces built so far (a split build counts
   once) and how many steps took their wave force from a block instead of the per-step excitation kernels. */
HC_API hc_status hc_get_exc_block_stats(hc_ensemble* e, long long* blocks_built, long long* steps_served, int reset);

/* Host-side planning of the radiation look-ahead, exposed for testing (no device needed).
   hc_rad_lookahead_plan: mode = 0 (the look-ahead cannot serve this step size), 1 (lag grid: RIRF lag spacing =
   rows_per_lag * dt_hint) or 2 (row grid: interpolation weights folded into a kernel of kernel_lags rows).
   hc_rad_lookahead_check_step: times_newest_first[0 .. n) = the time history at a step (element 0 = the step's time);
   smax = the largest lag with a bracket when every bracketed lag sits within bracket_snap rows of its nominal
   position (and, for mode 2, all lags are bracketed), else -1: the step would run the per-step kernel. */
HC_API hc_status hc_rad_lookahead_plan(const hc_tables* t, double dt_hint, int* mode, int* rows_per_lag, int* kernel_lags);
/* Slicing of a look-ahead pass of `items` work items into `nslices` launches (test hook of the launcher's arithmetic):
   advances the cursor (next_slice, next_item) by `count` slices with boundaries rounded to multiples of `wave` and
   returns 1 with the range [i0, i1) to launch, 0 when the range is empty.  The ranges of a pass tile [0, items). */
HC_API int hc_rad_pass_next(long long items, int nslices, int* next_slice, long long* next_item, int count, long long wave,
                            long long* i0, long long* i1);
/* The kernel the block path convolves the history rows with: out[kernel_lags][6N][6N] (row, column). */
HC_API hc_status hc_rad_lookahead_row_kernel(const hc_tables* t, double dt_hint, double* out);
HC_API hc_status hc_rad_lookahead_check_step(const hc_tables* t, double dt_hint, double bracket_snap,
                                             const double* times_newest_first, int n, int* smax);

/* Measured FP64 FMA peak of the device in TFLOP/s (roofline denominator for the FP64-bound kernels). */
HC_API hc_status hc_measure_fp64_peak(int device, double* tflops);
/* The same on the FP64 tensor cores (DMMA m8n8k4 loop). */
HC_API hc_status hc_measure_fp64_mma_peak(int device, double* tflops);

/* Pinned host memory helpers for callers that keep their own buffers. */
HC_API void* hc_host_alloc(size_t bytes);
HC_API void hc_host_free(void* p);

/* -------------------------------------------------------------------------------------
 * Multi-device ensemble (SURVEY.md 8e): the B instances of one ensemble partitioned over several GPUs of one node.
 * Instances are independent and the tables are replicated, so there is no exchange between devices on the step
 * path; the reference has no counterpart (it steps one system on one CPU thread) -- the per-step contract kept is
 * "one evaluation per time value" (src/hydro_forces.cpp:742-767) for every shard.  Shard i owns the contiguous block
 * hc_multi_shard_range(B, n, i) of global instance indices, has its own hc_ensemble on devices[i] and its own host
 * thread.  opts->batch is the TOTAL number of instances, opts->device is ignored, opts->stream must be NULL; the
 * look-ahead "auto" thresholds apply per shard (pass explicit modes for small shards).  A device may be listed more
 * than once (several shards on one GPU).
 * ------------------------------------------------------------------------------------- */
typedef struct hc_multi_ensemble hc_multi_ensemble;
HC_API void hc_multi_shard_range(int total, int shards, int index, int* first, int* count);
HC_API hc_status hc_multi_ensemble_create(const hc_tables* t, const hc_ensemble_opts* opts, const int* devices /* NULL: 0..n-1 */,
                                          int n_devices, hc_multi_ensemble** out);
HC_API void hc_multi_ensemble_destroy(hc_multi_ensemble* m);
HC_API int hc_multi_ensemble_num_shards(const hc_multi_ensemble* m);
HC_API int hc_multi_ensemble_batch(const hc_multi_ensemble* m);          /* total instances */
/* Device, first global instance, instance count and the per-device handle of shard `index` (any out pointer may be
 * NULL).  The handle may be used with the single-device queries (hc_waves_irregular_eta, hc_get_profile, ...) from the
 * calling thread while no hc_multi_* call is in flight. */
HC_API hc_status hc_multi_ensemble_shard(const hc_multi_ensemble* m, int index, int* device, int* first, int* count,
                                         hc_ensemble** ens);
/* Wave set-up for all shards at once; per-instance arrays are indexed by GLOBAL instance ([B]). */
HC_API hc_status hc_multi_waves_none(hc_multi_ensemble* m);
HC_API hc_status hc_multi_waves_regular(hc_multi_ensemble* m, int count /* 1 or B */, const double* amplitude,
                                        const double* omega, const double* phase /* may be NULL */);
HC_API hc_status hc_multi_waves_irregular(hc_multi_ensemble* m, const hc_irregular_params* p, const int* seeds /* [B] or NULL */,
                                          const double* Hs /* [B] or NULL */, const double* Tp /* [B] or NULL */);
HC_API hc_status hc_multi_waves_irregular_series(hc_multi_ensemble* m, double simulation_dt, int n, const double* time,
                                                 const double* eta /* [n] or [B][n] */, int per_instance);
/* One lock-step of every instance on every device: host [B][6N] arrays in global instance order (pinned recommended);
 * each shard uploads, evaluates and downloads its own slice concurrently -- the result gather is the slices landing
 * in `force`.  Synchronous at return.  Same status codes and time-keyed cache as hc_step. */
HC_API hc_status hc_multi_step(hc_multi_ensemble* m, double t, const double* pose, const double* vel, const double g_vec[3],
                               double* force, int* recomputed /* may be NULL */);
/* Device-resident variant: per shard a device pointer on that shard's device ([count_i][6N]); asynchronous on the
 * shards' streams (hc_multi_sync waits). */
HC_API hc_status hc_multi_step_device(hc_multi_ensemble* m, double t, const double* const* d_pose, const double* const* d_vel,
                                      const double g_vec[3], double* const* d_force);
/* hc_waves_kinematics_at_time for every shard at once: host arrays in global instance order (points [B][P][3], eta
 * [B][P], velocity / acceleration [B][P][3]); each shard fills its slice concurrently.  Synchronous at return. */
HC_API hc_status hc_multi_waves_kinematics_at_time(hc_multi_ensemble* m, double t, int n_points, const double* points,
                                                   double mwl, int wheeler_stretching,
                                                   double* eta, double* velocity, double* acceleration);
/* hc_ensemble_simulate for every shard at once: host arrays in global instance order (pose / vel / pto_energy [B][6N],
 * rec_pose / rec_vel [n_rec][B][6N], pto_* of the params [B][6N], tsda_damping / tsda_stiffness / tsda_energy of the
 * links [B][n_tsda]).  Each shard runs its whole loop on its own worker
 * thread, with no cross-shard barrier per step.  *steps_done = the fewest steps any shard completed. */
HC_API hc_status hc_multi_ensemble_simulate(hc_multi_ensemble* m, const hc_sim_params* p, double* pose, double* vel,
                                            double* rec_t, double* rec_pose, double* rec_vel, double* pto_energy,
                                            int* steps_done);
/* Final gather of the three force components of the last evaluation, host [B][6N] each (may be NULL). */
HC_API hc_status hc_multi_get_components(hc_multi_ensemble* m, double* hydrostatic, double* radiation, double* waves);
HC_API hc_status hc_multi_sync(hc_multi_ensemble* m);
HC_API hc_status hc_multi_reset(hc_multi_ensemble* m);

/* ---- stand-alone wave helpers on the reference's public surface (host, setup-time) ---- */
HC_API hc_status hc_pierson_moskowitz_spectrum_hz(int n, const double* f, double Hs, double Tp, double* S);
HC_API hc_status hc_jonswap_spectrum_hz(int n, const double* f, double Hs, double Tp, double gamma,
                                        int is_normalized, double* S);
HC_API hc_status hc_compute_wave_number(double omega, double water_depth, double g, double* k);
/* IrregularWaves::ResampleIRF + CalculateWidthIRF (src/wave_types.cpp:572-628) for one body: excitation IRF resampled
 * to ceil((t1-t0)/dt) points with Eigen's cubic B-spline fit.  Call with t_out == NULL to query *n_out. */
HC_API hc_status hc_resample_excitation_irf(const hc_tables* t, double dt, int body, int* n_out, double* t_out,
                                            double* width_out, double* f_out /*[6][n]*/);
/* Random phases of CreateSpectrum (src/wave_types.cpp:663-669): std::mt19937(seed), uniform_real(0, 2 pi). */
HC_API hc_status hc_random_phases(int seed, int n, double* out);
/* Airy water kinematics at a point for a sum of n wave components travelling along +x (host arithmetic, off the step
 * path as in the reference): GetEta / GetEtaIrregular (src/wave_types.cpp:14-45), GetWaterVelocity /
 * GetWaterAcceleration (+Irregular) (:61-160, deep-water branch when 2 pi / k > depth or k depth > 500), and the Wheeler
 * stretching of IrregularWaves::GetVelocity / GetAcceleration (:515-545) when wheeler_stretching != 0:
 * z' = depth (z - mwl - eta) / (depth + eta).  Components are summed in ascending order.  n = 1 with
 * wheeler_stretching = 0 is RegularWave::GetElevation / GetVelocity / GetAcceleration (:301-313).
 * Any of eta / velocity / acceleration may be NULL. */
HC_API hc_status hc_wave_kinematics(int n, const double* omega, const double* amplitude, const double* phase,
                                    const double* wavenumber, const double position[3], double time, double water_depth,
                                    double mwl, int wheeler_stretching, double* eta, double velocity[3],
                                    double acceleration[3]);

/* ---------------------------------------------------------------------------------------
 * HDF5 output / generic input without libhdf5 (classic format: superblock v0, old-style groups, contiguous
 * little-endian float64 datasets, fixed-length strings, scalar attributes).  Replaces the HDF5 C++ calls of
 * H5Writer (src/h5_writer.cpp) used by SimulationExporter (src/simulation_exporter.cpp:181-199,373-391).
 * Paths are '/'-separated; intermediate groups are created on demand.  Nothing touches the disk before save.
 * ------------------------------------------------------------------------------------- */
typedef struct hc_h5_writer hc_h5_writer;
HC_API hc_status hc_h5_writer_create(hc_h5_writer** out);
HC_API void hc_h5_writer_destroy(hc_h5_writer* w);
HC_API hc_status hc_h5_writer_put_group(hc_h5_writer* w, const char* path);
HC_API hc_status hc_h5_writer_put_f64(hc_h5_writer* w, const char* path, int rank, const uint64_t* dims,
                                      const double* data);
HC_API hc_status hc_h5_writer_put_string(hc_h5_writer* w, const char* path, const char* value);
/* 1-D dataset of fixed-length, null-padded strings (names arrays of the results schema). */
HC_API hc_status hc_h5_writer_put_string_array(hc_h5_writer* w, const char* path, int count, const char* const* values);
HC_API hc_status hc_h5_writer_attr_string(hc_h5_writer* w, const char* path, const char* name, const char* value);
HC_API hc_status hc_h5_writer_attr_f64(hc_h5_writer* w, const char* path, const char* name, double value);
HC_API hc_status hc_h5_writer_save(hc_h5_writer* w, const char* file);
/* Reads: out may be NULL to query rank/dims (dims has room for 8 entries). */
HC_API hc_status hc_h5_read_f64(const char* file, const char* dataset, int* rank, uint64_t* dims, double* out,
                                size_t capacity);
HC_API hc_status hc_h5_read_string(const char* file, const char* dataset, char* out, size_t capacity);
HC_API hc_status hc_h5_list(const char* file, const char* group, char* out /* '\n'-separated */, size_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* HYDROCHRONO_B200_H */
