// TestHydroEnsemble -- B independent copies of one hydro system evaluated in lock-step by ONE device ensemble.
//
// The reference's hydro.yaml front end parses period sweeps (waves.period.values / linspace / range,
// src/hydro_yaml_parser.cpp:441-524 -> WaveSettings::period_values, src/hydro_types.h:49) but builds a single
// TestHydro from the first value.  Here every sweep point (x every seed) becomes one INSTANCE of a batched
// ensemble: each instance has its own Chrono system (bodies, joints, PTO) and its own wave, all share the BEMIO
// tables, and the first force query at a new time value gathers the state of ALL systems and runs one hc_step for
// the whole batch (the reference's once-per-time-value contract, src/hydro_forces.cpp:742-767, applied batch-wide).
// The systems must therefore be advanced in lock-step: chrono::ChSystem::DoStepDynamicsLockstep with the
// chrono_compat stand-in; with the real Chrono and an explicit-force stepper, one DoStepDynamics per system per step.
#ifndef HYDROC_B200_HYDRO_ENSEMBLE_H
#define HYDROC_B200_HYDRO_ENSEMBLE_H
#pragma once

#include <memory>
#include <string>
#include <vector>

#include <chrono_compat/chrono_compat.h>
#include <hydroc/h5fileinfo.h>
#include <hydroc/hydro_types.h>
#include <hydroc/wave_types.h>

class ChLoadAddedMass;

class TestHydroEnsemble {
  public:
    using BodyList = std::vector<std::shared_ptr<chrono::ChBody>>;
    // systems[i] = the hydro bodies ("body1", "body2", ...) of instance i, every list with the same body count
    TestHydroEnsemble(std::vector<BodyList> systems, const std::string& h5_file_name, double dt_hint = 0.0);
    TestHydroEnsemble(const TestHydroEnsemble&) = delete;
    TestHydroEnsemble& operator=(const TestHydroEnsemble&) = delete;
    ~TestHydroEnsemble();

    int Batch() const { return int(systems_.size()); }
    int NumBodies() const { return num_bodies_; }

    // one wave per instance (size 1 = shared by all instances)
    void AddWavesNone();
    void AddWavesRegular(const std::vector<double>& amplitude, const std::vector<double>& omega);
    void AddWavesIrregular(const IrregularWaveParams& base, const std::vector<int>& seeds, const std::vector<double>& Hs,
                           const std::vector<double>& Tp);

    // water elevation, particle velocity and acceleration of every instance's wave at its own points on the device
    // (WaveBase::GetElevation / GetVelocity / GetAcceleration, hc_waves_kinematics_at_time): points [B][n_points][3]
    // in, eta [B][n_points], vel / acc [B][n_points][3] out (resized; any may be null).  Wheeler stretching as the
    // IrregularWaveParams::wave_stretching_ given to AddWavesIrregular.  Irregular eta is not ramped.  Not a force
    // evaluation: the force cache and DeviceEvaluations() are untouched.
    void GetWaveKinematics(double t, int n_points, const std::vector<double>& points, std::vector<double>* eta,
                           std::vector<double>* vel, std::vector<double>* acc, double mwl = 0.0);

    // total force on body b (1-based) of instance inst in DoF i; one batched device evaluation per time value
    double CoordinateFuncForInstance(int inst, int b, int i);
    // the three components of the last evaluation, [B][6N] each
    void GetComponents(std::vector<double>& hydrostatic, std::vector<double>& radiation, std::vector<double>& waves);
    // R[i] += c * M_added * w[i] for every instance at once on the device (ChLoadAddedMass::LoadIntLoadResidual_Mv,
    // src/chloadaddedmass.cpp:55-71, batched: hc_added_mass_mv); w and R are [B][n_sys], n_sys >= 6 * bodies
    void AddedMassMvAll(int n_sys, double c, const std::vector<double>& w, std::vector<double>& R);
    long long DeviceEvaluations() const { return evaluations_; }
    hc_ensemble* ensemble() const { return ens_; }
    HydroData& GetHydroData() { return file_info_; }

  private:
    void EvaluateAtCurrentTime();
    std::vector<BodyList> systems_;
    int num_bodies_;
    HydroData file_info_;
    hc_ensemble* ens_ = nullptr;
    std::vector<double> pose_, vel_, force_;
    double prev_time_ = -1.0;
    bool wave_stretching_ = false;
    long long evaluations_ = 0;
    std::vector<std::shared_ptr<chrono::ChLoadContainer>> load_containers_;
    std::vector<std::shared_ptr<ChLoadAddedMass>> added_mass_;
};

// One instance per (period value x seed): instance i runs period_values[i % P] (P = max(1, #period_values); the single
// `period` when no sweep is given) and seed  base_seed + i / P  (irregular waves; base_seed = waves.seed or 1).
// systems.size() must be P * seeds_per_period.  Wave mapping as SetupHydroFromYAML: amplitude = height / 2,
// omega = 2 pi / period (src/setup_hydro_from_yaml.cpp:28-80).
std::unique_ptr<TestHydroEnsemble> SetupHydroSweepFromYAML(const YAMLHydroData& hydro_data,
                                                           const std::vector<TestHydroEnsemble::BodyList>& systems,
                                                           double timestep, double sim_duration, double ramp_duration,
                                                           int seeds_per_period = 1);

#endif
