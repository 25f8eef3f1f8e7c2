// Device-side stepping (hc_ensemble_simulate) against the chrono_compat stepper: B systems advanced in lock-step around
// one TestHydroEnsemble (ChSystem::DoStepDynamicsLockstep), and the same B instances run by hc_ensemble_simulate on the
// handle of a second TestHydroEnsemble built the same way.  Two cases under linearised Euler and HHT:
//   sphere  heave-only spheres (prismatic joint to ground == free_dof {0,0,1,0,0,0}), one regular wave per instance
//   rm3     the free 12-DoF RM3-shaped pair, nonzero initial roll / pitch (quaternion path), regular waves
// usage: test_device_stepping <sphere.h5> <rm3_like.h5> [steps = 400]
// out: one line per (case, scheme): case <c> scheme <s> steps <n> max_diff <d> amplitude <a>
//      (largest |pose difference| over every step, instance and DoF, and the largest |pose - initial pose|)
#include <hydroc/hydro_ensemble.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <iomanip>
#include <iostream>

#include "../src/hc_check.h"

using namespace chrono;

namespace {

struct Case {
    std::string name, h5;
    int bodies;
    std::vector<double> mass;
    std::vector<ChVector3d> inertia, pos;
    std::vector<ChVector3d> rpy;      // initial roll, pitch, yaw per body (instance i adds 0.01 i to roll)
    bool heave_only;
    std::vector<double> amp, omega;   // per instance
    double dt;
};

struct Built {
    std::vector<std::unique_ptr<ChSystemNSC>> systems;
    std::vector<TestHydroEnsemble::BodyList> lists;
    std::unique_ptr<TestHydroEnsemble> ens;
};

Built build(const Case& c, bool hht) {
    Built r;
    const int B = int(c.amp.size());
    for (int i = 0; i < B; ++i) {
        r.systems.push_back(std::make_unique<ChSystemNSC>());
        ChSystemNSC& sys = *r.systems.back();
        sys.SetGravitationalAcceleration(ChVector3d(0, 0, -9.81));
        if (hht) sys.SetTimestepperType(ChTimestepper::Type::HHT);
        auto ground = chrono_types::make_shared<ChBody>();
        ground->SetFixed(true);
        sys.AddBody(ground);
        TestHydroEnsemble::BodyList list;
        for (int b = 0; b < c.bodies; ++b) {
            auto body = chrono_types::make_shared<ChBody>();
            body->SetName("body" + std::to_string(b + 1));
            body->SetMass(c.mass[b]);
            body->SetInertiaXX(c.inertia[b]);
            body->SetPos(c.pos[b]);
            const ChVector3d a = c.rpy[b] + ChVector3d(0.01 * i, 0, 0) * (c.heave_only ? 0.0 : 1.0);
            body->SetRot(QuatFromAngleX(a.x()) * QuatFromAngleY(a.y()) * QuatFromAngleZ(a.z()));
            sys.AddBody(body);
            if (c.heave_only) {
                auto joint = chrono_types::make_shared<ChLinkLockPrismatic>();
                joint->Initialize(body, ground, false, ChFramed(c.pos[b]), ChFramed(ChVector3d(0, 0, -5)));
                sys.AddLink(joint);
            }
            list.push_back(body);
        }
        r.lists.push_back(list);
    }
    r.ens = std::make_unique<TestHydroEnsemble>(r.lists, c.h5, c.dt);
    r.ens->AddWavesRegular(c.amp, c.omega);
    return r;
}

void pose_of(const TestHydroEnsemble::BodyList& l, double* x) {
    for (size_t b = 0; b < l.size(); ++b) {
        const ChVector3d p = l[b]->GetPos(), a = l[b]->GetRot().GetCardanAnglesXYZ();
        x[6 * b + 0] = p.x(); x[6 * b + 1] = p.y(); x[6 * b + 2] = p.z();
        x[6 * b + 3] = a.x(); x[6 * b + 4] = a.y(); x[6 * b + 5] = a.z();
    }
}

void run(const Case& c, bool hht, int steps) {
    const int B = int(c.amp.size()), D = 6 * c.bodies;
    const size_t bd = size_t(B) * D;
    // lock-step host run
    Built host = build(c, hht);
    std::vector<double> x0(bd), ref(size_t(steps) * bd);
    for (int i = 0; i < B; ++i) pose_of(host.lists[i], &x0[size_t(i) * D]);
    std::vector<ChSystem*> sys;
    for (auto& s : host.systems) sys.push_back(s.get());
    for (int n = 0; n < steps; ++n) {
        ChSystem::DoStepDynamicsLockstep(sys, c.dt);
        for (int i = 0; i < B; ++i) pose_of(host.lists[i], &ref[size_t(n) * bd + size_t(i) * D]);
    }
    // device run on a second ensemble built the same way
    Built dev = build(c, hht);
    std::vector<double> pose(bd), vel(bd, 0.0), rec(size_t(steps) * bd), inertia;
    for (int i = 0; i < B; ++i) pose_of(dev.lists[i], &pose[size_t(i) * D]);
    for (const auto& j : c.inertia) { inertia.push_back(j.x()); inertia.push_back(j.y()); inertia.push_back(j.z()); }
    std::vector<int> free_dof(D, 1);
    if (c.heave_only)
        for (int k = 0; k < D; ++k) free_dof[k] = (k % 6 == 2);
    hc_sim_params p{};
    p.scheme = hht ? 1 : 0;
    p.t0 = 0.0; p.dt = c.dt; p.n_steps = steps; p.record_every = 1;
    p.g[0] = 0.0; p.g[1] = 0.0; p.g[2] = -9.81;
    p.mass = c.mass.data(); p.inertia = inertia.data(); p.free_dof = free_dof.data();
    int done = 0;
    hc_throw_on_error(hc_ensemble_simulate(dev.ens->ensemble(), &p, pose.data(), vel.data(), nullptr, rec.data(), nullptr,
                                           nullptr, &done));
    double diff = 0.0, amp = 0.0;
    for (size_t n = 0; n < size_t(steps); ++n)
        for (size_t k = 0; k < bd; ++k) {
            diff = std::max(diff, std::fabs(rec[n * bd + k] - ref[n * bd + k]));
            amp = std::max(amp, std::fabs(ref[n * bd + k] - x0[k]));
        }
    std::cout << std::setprecision(6) << "case " << c.name << " scheme " << (hht ? "hht" : "euler") << " steps " << done
              << " max_diff " << diff << " amplitude " << amp << std::endl;
}

}  // namespace

int main(int argc, char* argv[]) {
    if (argc < 3) { std::cerr << "usage: test_device_stepping <sphere.h5> <rm3_like.h5> [steps]" << std::endl; return 2; }
    const int steps = argc > 3 ? std::atoi(argv[3]) : 400;
    try {
        Case sphere{"sphere", argv[1], 1, {261.8e3}, {ChVector3d(1, 1, 1)}, {ChVector3d(0, 0, -2)}, {ChVector3d(0, 0, 0)},
                    true, {0.177, 0.706, 2.374}, {2.094395102, 1.047197551, 0.571198664}, 0.015};
        Case rm3{"rm3", argv[2], 2, {725834.0, 886691.0},
                 {ChVector3d(20907301.0, 21306090.66, 37085481.11), ChVector3d(94419614.57, 94407091.24, 28542224.82)},
                 {ChVector3d(0, 0, -0.72), ChVector3d(0, 0, -21.29)}, {ChVector3d(0.05, -0.03, 0.0), ChVector3d(-0.02, 0.04, 0.01)},
                 false, {0.5, 1.0, 1.5, 2.0}, {0.6, 0.8, 1.0, 1.2}, 0.01};
        for (bool hht : {false, true}) {
            run(sphere, hht, steps);
            run(rm3, hht, steps);
        }
    } catch (const std::exception& e) {
        std::cerr << "error: " << e.what() << std::endl;
        return 1;
    }
    return 0;
}
