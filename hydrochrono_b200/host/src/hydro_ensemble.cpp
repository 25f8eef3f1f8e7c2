// TestHydroEnsemble / SetupHydroSweepFromYAML (see hydroc/hydro_ensemble.h).
#include <hydroc/hydro_ensemble.h>

#include <algorithm>
#include <cmath>
#include <stdexcept>

#include <hydroc/chloadaddedmass.h>

#include "hc_check.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

using namespace chrono;

namespace {
constexpr int kDof = 6;

// ChFunction serving one force component of one body of one instance (the ensemble's ComponentFunc)
class InstanceComponentFunc : public ChFunction {
  public:
    InstanceComponentFunc(TestHydroEnsemble* e, int inst, int b, int dof) : e_(e), inst_(inst), b_(b), dof_(dof) {}
    ChFunction* Clone() const override { return new InstanceComponentFunc(*this); }
    double GetVal(double) const override { return e_->CoordinateFuncForInstance(inst_, b_, dof_); }

  private:
    TestHydroEnsemble* e_;
    int inst_, b_, dof_;
};

std::string lowercase(std::string s) {
    std::transform(s.begin(), s.end(), s.begin(), ::tolower);
    return s;
}
}  // namespace

TestHydroEnsemble::TestHydroEnsemble(std::vector<BodyList> systems, const std::string& h5_file_name, double dt_hint)
    : systems_(std::move(systems)), num_bodies_(systems_.empty() ? 0 : int(systems_[0].size())),
      file_info_(H5FileInfo(h5_file_name, num_bodies_).ReadH5Data()) {
    if (systems_.empty() || num_bodies_ == 0) throw std::runtime_error("TestHydroEnsemble: no systems / no bodies");
    for (const auto& s : systems_)
        if (int(s.size()) != num_bodies_) throw std::runtime_error("TestHydroEnsemble: every instance needs the same number of bodies");
    const int B = Batch(), D = kDof * num_bodies_;
    pose_.assign(size_t(B) * D, 0.0); vel_.assign(size_t(B) * D, 0.0); force_.assign(size_t(B) * D, 0.0);

    hc_ensemble_opts o;
    hc_ensemble_default_opts(&o);
    o.batch = B;
    o.dt_hint = dt_hint;
    hc_throw_on_error(hc_ensemble_create(file_info_.handle(), &o, &ens_));

    for (int i = 0; i < B; ++i) {
        ChSystem* sys = systems_[i][0]->GetSystem();
        for (int b = 0; b < num_bodies_; ++b) {
            // two world-aligned ChForces per body, as ForceFunc6d sets them up (src/hydro_forces.cpp:87-168);
            // body numbering from the name "bodyN" (:106-107)
            const auto& body = systems_[i][b];
            std::string name = body->GetName();
            const int b_num = std::stoi(name.erase(0, 4));
            auto f = chrono_types::make_shared<ChForce>();
            auto t = chrono_types::make_shared<ChForce>();
            f->SetAlign(ChForce::AlignmentFrame::WORLD_DIR); t->SetAlign(ChForce::AlignmentFrame::WORLD_DIR);
            f->SetName("hydroforce"); t->SetName("hydrotorque");
            f->SetF_x(std::make_shared<InstanceComponentFunc>(this, i, b_num, 0));
            f->SetF_y(std::make_shared<InstanceComponentFunc>(this, i, b_num, 1));
            f->SetF_z(std::make_shared<InstanceComponentFunc>(this, i, b_num, 2));
            t->SetF_x(std::make_shared<InstanceComponentFunc>(this, i, b_num, 3));
            t->SetF_y(std::make_shared<InstanceComponentFunc>(this, i, b_num, 4));
            t->SetF_z(std::make_shared<InstanceComponentFunc>(this, i, b_num, 5));
            t->SetMode(ChForce::ForceType::TORQUE);
            body->AddForce(f);
            body->AddForce(t);
        }
        // added mass of instance i: the same stiff load the single-system TestHydro attaches (:223-234)
        auto container = chrono_types::make_shared<ChLoadContainer>();
        std::vector<std::shared_ptr<ChLoadable>> loadables(systems_[i].begin(), systems_[i].end());
        auto load = chrono_types::make_shared<ChLoadAddedMass>(file_info_.GetBodyInfos(), loadables, sys);
        if (sys) sys->Add(container);
        container->Add(load);
        load_containers_.push_back(container);
        added_mass_.push_back(load);
    }
    AddWavesNone();
}

TestHydroEnsemble::~TestHydroEnsemble() {
    if (ens_) hc_ensemble_destroy(ens_);
}

void TestHydroEnsemble::AddWavesNone() {
    hc_throw_on_error(hc_waves_none(ens_));
    wave_stretching_ = false;
}

void TestHydroEnsemble::AddWavesRegular(const std::vector<double>& amplitude, const std::vector<double>& omega) {
    const size_t B = size_t(Batch());
    if (amplitude.size() != omega.size() || !(amplitude.size() == 1 || amplitude.size() == B))
        throw std::runtime_error("TestHydroEnsemble::AddWavesRegular: need 1 or B (amplitude, omega) pairs");
    hc_throw_on_error(hc_waves_regular(ens_, int(amplitude.size()), amplitude.data(), omega.data(), nullptr));
    wave_stretching_ = false;
}

void TestHydroEnsemble::AddWavesIrregular(const IrregularWaveParams& p, const std::vector<int>& seeds,
                                          const std::vector<double>& Hs, const std::vector<double>& Tp) {
    const size_t B = size_t(Batch());
    auto ok = [&](size_t n) { return n == 0 || n == B; };
    if (!ok(seeds.size()) || !ok(Hs.size()) || !ok(Tp.size()))
        throw std::runtime_error("TestHydroEnsemble::AddWavesIrregular: per-instance arrays must be empty or of size B");
    hc_irregular_params q;
    hc_irregular_default_params(&q);
    q.simulation_dt = p.simulation_dt_; q.simulation_duration = p.simulation_duration_; q.ramp_duration = p.ramp_duration_;
    q.wave_height = p.wave_height_; q.wave_period = p.wave_period_; q.frequency_min = p.frequency_min_;
    q.frequency_max = p.frequency_max_; q.nfrequencies = p.nfrequencies_; q.peak_enhancement_factor = p.peak_enhancement_factor_;
    q.is_normalized = p.is_normalized_ ? 1 : 0; q.seed = p.seed_;
    hc_throw_on_error(hc_waves_irregular(ens_, &q, seeds.empty() ? nullptr : seeds.data(), Hs.empty() ? nullptr : Hs.data(),
                                         Tp.empty() ? nullptr : Tp.data()));
    wave_stretching_ = p.wave_stretching_;
}

void TestHydroEnsemble::GetWaveKinematics(double t, int n_points, const std::vector<double>& points, std::vector<double>* eta,
                                          std::vector<double>* vel, std::vector<double>* acc, double mwl) {
    const size_t n = size_t(Batch()) * size_t(n_points > 0 ? n_points : 0);
    if (n_points < 1 || points.size() != 3 * n)
        throw std::runtime_error("TestHydroEnsemble::GetWaveKinematics: points must be [B][n_points][3], n_points >= 1");
    if (eta) eta->resize(n);
    if (vel) vel->resize(3 * n);
    if (acc) acc->resize(3 * n);
    hc_throw_on_error(hc_waves_kinematics_at_time(ens_, t, n_points, points.data(), mwl, wave_stretching_ ? 1 : 0,
                                                  eta ? eta->data() : nullptr, vel ? vel->data() : nullptr,
                                                  acc ? acc->data() : nullptr));
}

// One batched device step at the current Chrono time with the state every system holds at this moment.
void TestHydroEnsemble::EvaluateAtCurrentTime() {
    const int B = Batch(), D = kDof * num_bodies_;
    const double t = systems_[0][0]->GetChTime();
    for (int i = 0; i < B; ++i) {
        if (systems_[i][0]->GetChTime() != t)
            throw std::runtime_error("TestHydroEnsemble: the systems are not in lock-step (instance " + std::to_string(i) +
                                     " is at t = " + std::to_string(systems_[i][0]->GetChTime()) + ", instance 0 at t = " +
                                     std::to_string(t) + "); advance them with ChSystem::DoStepDynamicsLockstep");
        for (int b = 0; b < num_bodies_; ++b) {
            const auto& body = systems_[i][b];
            const ChVector3d p = body->GetPos(), a = body->GetRot().GetCardanAnglesXYZ();     // reference :279-280
            const ChVector3d v = body->GetPosDt(), w = body->GetAngVelParent();               // reference :567-568
            double* x = &pose_[size_t(i) * D + kDof * b];
            double* u = &vel_[size_t(i) * D + kDof * b];
            x[0] = p.x(); x[1] = p.y(); x[2] = p.z(); x[3] = a.x(); x[4] = a.y(); x[5] = a.z();
            u[0] = v.x(); u[1] = v.y(); u[2] = v.z(); u[3] = w.x(); u[4] = w.y(); u[5] = w.z();
        }
    }
    // gravity is a property of the (shared) environment: instance 0's system, as TestHydro reads its system's
    const ChVector3d g = systems_[0][0]->GetSystem()->GetGravitationalAcceleration();
    const double gv[3] = {g.x(), g.y(), g.z()};
    hc_throw_on_error(hc_step(ens_, t, pose_.data(), vel_.data(), gv, force_.data(), nullptr));
    prev_time_ = t;
    ++evaluations_;
}

double TestHydroEnsemble::CoordinateFuncForInstance(int inst, int b, int i) {
    if (i < 0 || i >= kDof || b < 1 || b > num_bodies_ || inst < 0 || inst >= Batch())
        throw std::out_of_range("Invalid index in CoordinateFuncForInstance");
    // cache keyed by the time of the system that asks (:742-744): within a lock-step all systems ask at the same time
    if (systems_[inst][0]->GetChTime() != prev_time_) EvaluateAtCurrentTime();
    return force_[size_t(inst) * kDof * num_bodies_ + kDof * (b - 1) + i];
}

void TestHydroEnsemble::AddedMassMvAll(int n_sys, double c, const std::vector<double>& w, std::vector<double>& R) {
    const size_t n = size_t(Batch()) * n_sys;
    if (w.size() != n || R.size() != n) throw std::runtime_error("AddedMassMvAll: w and R must be [B][n_sys]");
    hc_throw_on_error(hc_added_mass_mv(ens_, n_sys, c, w.data(), R.data()));
}

void TestHydroEnsemble::GetComponents(std::vector<double>& hs, std::vector<double>& rad, std::vector<double>& wv) {
    const size_t n = size_t(Batch()) * kDof * num_bodies_;
    hs.resize(n); rad.resize(n); wv.resize(n);
    hc_throw_on_error(hc_get_components(ens_, hs.data(), rad.data(), wv.data()));
}

std::unique_ptr<TestHydroEnsemble> SetupHydroSweepFromYAML(const YAMLHydroData& hydro_data,
                                                           const std::vector<TestHydroEnsemble::BodyList>& systems,
                                                           double timestep, double sim_duration, double ramp_duration,
                                                           int seeds_per_period) {
    const WaveSettings& ws = hydro_data.waves;
    std::vector<double> periods = ws.period_values;
    if (periods.empty()) periods.push_back(ws.period);
    const int P = int(periods.size());
    if (seeds_per_period < 1 || int(systems.size()) != P * seeds_per_period)
        throw std::runtime_error("SetupHydroSweepFromYAML: need one system per (period value x seed): " + std::to_string(P) +
                                 " x " + std::to_string(seeds_per_period) + ", got " + std::to_string(systems.size()));
    if (hydro_data.bodies.empty()) throw std::runtime_error("No hydrodynamic bodies found in Chrono system");
    // match hydro bodies to every system's Chrono bodies by name; the first body's h5_file is used (reference :91-95)
    std::vector<TestHydroEnsemble::BodyList> matched(systems.size());
    for (size_t i = 0; i < systems.size(); ++i) {
        for (const auto& hb : hydro_data.bodies)
            for (const auto& cb : systems[i])
                if (cb->GetName() == hb.name) { matched[i].push_back(cb); break; }
        if (matched[i].empty()) throw std::runtime_error("No hydrodynamic bodies found in Chrono system");
    }
    auto ens = std::make_unique<TestHydroEnsemble>(matched, hydro_data.bodies[0].h5_file, timestep);
    const int B = ens->Batch();
    const std::string type = lowercase(ws.type);
    if (type == "regular") {
        std::vector<double> amp(B), om(B);
        for (int i = 0; i < B; ++i) { amp[i] = ws.height / 2.0; om[i] = 2.0 * M_PI / periods[i % P]; }
        ens->AddWavesRegular(amp, om);
    } else if (type == "irregular") {
        IrregularWaveParams p;
        p.num_bodies_ = static_cast<unsigned int>(ens->NumBodies());
        p.simulation_dt_ = timestep; p.simulation_duration_ = sim_duration; p.ramp_duration_ = ramp_duration;
        p.wave_height_ = ws.height; p.wave_period_ = periods[0];
        const int base_seed = ws.seed > 0 ? ws.seed : 1;
        p.seed_ = base_seed;
        std::vector<int> seeds(B);
        std::vector<double> Tp(B);
        for (int i = 0; i < B; ++i) { seeds[i] = base_seed + i / P; Tp[i] = periods[i % P]; }
        ens->AddWavesIrregular(p, seeds, {}, Tp);
    } else if (type == "no_wave" || type == "still_ci" || type == "still") {
        ens->AddWavesNone();
    } else {
        throw std::runtime_error("Unsupported wave type: " + ws.type);
    }
    if (lowercase(hydro_data.radiation_convolution_mode) == "tapereddirect") {
        hc_tapered_opts o;
        const std::string sm = !hydro_data.td_smoothing.empty() ? hydro_data.td_smoothing : std::string("sg");
        o.smoothing = sm.c_str();
        o.window_length = std::max(3, hydro_data.td_window_length != 0 ? hydro_data.td_window_length : 5);
        if (o.window_length % 2 == 0) o.window_length += 1;
        o.rirf_end_time = hydro_data.td_rirf_end_time;
        o.taper_start_percent = hydro_data.td_taper_start_percent;
        o.taper_end_percent = hydro_data.td_taper_end_percent;
        o.taper_final_amplitude = hydro_data.td_taper_final_amplitude;
        hc_throw_on_error(hc_tables_set_convolution_mode(ens->GetHydroData().handle(), 1, &o));
        hc_throw_on_error(hc_ensemble_refresh_rirf(ens->ensemble()));
    }
    return ens;
}
