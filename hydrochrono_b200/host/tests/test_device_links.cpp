// Device-side stepping with joints and spring-dampers (hc_ensemble_simulate with hc_sim_params.links) against the
// chrono_compat stepper: B systems advanced in lock-step around one TestHydroEnsemble (ChSystem::DoStepDynamicsLockstep),
// and the same B instances run by hc_ensemble_simulate on the handle of a second TestHydroEnsemble built the same way,
// with hc_sim_links built from the systems' ChLinkLockPrismatic / ChLinkTSDA.  Under linearised Euler and HHT:
//   rm3         float on a prismatic joint to an all-free spar (initial roll / pitch and angular velocity), a damper PTO
//               between them with per-instance damping, regular waves per instance
//   rm3_spring  the same with a spring-damper PTO and an explicit rest length
//   sphere      heave sphere on a prismatic joint to ground with a damper PTO to ground (the reference's
//               sphere_reg_waves arrangement)
// usage: test_device_links <sphere.h5> <rm3_like.h5> [steps = 400]
// out: one line per (case, scheme): case <c> scheme <s> steps <n> max_diff <d> amplitude <a> residual <r>
//      (largest |pose difference| over every step, instance and DoF; the largest |pose - initial pose|; the largest
//      joint residual of the device states: transverse offset in the parent frame and relative rotation)
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
    std::vector<ChVector3d> rpy;      // initial roll, pitch, yaw per body (instance i adds 0.01 i to the parent's roll)
    ChVector3d w_parent;              // initial angular velocity of the parent (rm3)
    bool to_ground;                   // sphere: joint and PTO to ground; else float (0) on spar (1)
    std::vector<double> amp, omega;   // per instance
    std::vector<double> damping;      // per instance
    double stiffness, rest;           // rest < 0: the length at assembly
    double dt;
};

struct Built {
    std::vector<std::unique_ptr<ChSystemNSC>> systems;
    std::vector<TestHydroEnsemble::BodyList> lists;
    std::vector<std::shared_ptr<ChLinkLockPrismatic>> joints;   // one per instance
    std::vector<std::shared_ptr<ChLinkTSDA>> ptos;
    std::unique_ptr<TestHydroEnsemble> ens;
};

ChQuaterniond rot_of(const ChVector3d& a) { return QuatFromAngleX(a.x()) * QuatFromAngleY(a.y()) * QuatFromAngleZ(a.z()); }

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
            const bool parent = !c.to_ground && b == 1;
            body->SetRot(rot_of(c.rpy[b] + ChVector3d(parent ? 0.01 * i : 0.0, 0, 0)));
            sys.AddBody(body);
            list.push_back(body);
        }
        auto joint = chrono_types::make_shared<ChLinkLockPrismatic>();
        auto pto = chrono_types::make_shared<ChLinkTSDA>();
        if (c.to_ground) {
            joint->Initialize(list[0], ground, false, ChFramed(c.pos[0]), ChFramed(ChVector3d(0, 0, -5)));
            pto->Initialize(list[0], ground, false, c.pos[0], ChVector3d(0, 0, -5));
        } else {
            // the spar moves: its angular velocity, and the float moving with it (vA = vB + wB x rho)
            list[1]->SetAngVelParent(c.w_parent);
            list[0]->SetPosDt(c.w_parent % (list[0]->GetPos() - list[1]->GetPos()));
            // the slide runs along the world z axis at assembly (tilted in the frame of the rolled / pitched spar)
            joint->Initialize(list[0], list[1], false, ChFramed(c.pos[0]), ChFramed(c.pos[1]));
            pto->Initialize(list[0], list[1], false, c.pos[0], c.pos[1]);
        }
        pto->SetDampingCoefficient(c.damping[i]);
        pto->SetSpringCoefficient(c.stiffness);
        if (c.rest >= 0) pto->SetRestLength(c.rest);
        sys.AddLink(joint);
        sys.AddLink(pto);
        r.joints.push_back(joint);
        r.ptos.push_back(pto);
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

void vel_of(const TestHydroEnsemble::BodyList& l, double* v) {
    for (size_t b = 0; b < l.size(); ++b) {
        const ChVector3d p = l[b]->GetPosDt(), w = l[b]->GetAngVelParent();
        for (int k = 0; k < 3; ++k) { v[6 * b + k] = p[k]; v[6 * b + 3 + k] = w[k]; }
    }
}

// joint residual of a device pose: transverse offset of the child in the parent frame and the deviation of its
// relative rotation from the assembly's (quaternions rebuilt from the Cardan angles)
double residual(const double* x, int child, int parent, const ChLinkLockPrismatic& J) {
    const ChVector3d xA(x[6 * child], x[6 * child + 1], x[6 * child + 2]);
    const ChQuaterniond qA = rot_of(ChVector3d(x[6 * child + 3], x[6 * child + 4], x[6 * child + 5]));
    ChVector3d xB;
    ChQuaterniond qB;
    if (parent >= 0) {
        xB = ChVector3d(x[6 * parent], x[6 * parent + 1], x[6 * parent + 2]);
        qB = rot_of(ChVector3d(x[6 * parent + 3], x[6 * parent + 4], x[6 * parent + 5]));
    }
    const ChVector3d d = qB.RotateBack(xA - xB) - J.offset_in_parent;
    const ChVector3d tr = d - J.axis_in_parent * d.Dot(J.axis_in_parent);
    const ChQuaterniond rel = qB.GetConjugate() * qA;
    const double s = rel.e0 * J.rel_rot.e0 < 0 ? -1.0 : 1.0;
    double r = tr.Length();
    r = std::max(r, std::fabs(s * rel.e0 - J.rel_rot.e0));
    r = std::max(r, std::fabs(s * rel.e1 - J.rel_rot.e1));
    r = std::max(r, std::fabs(s * rel.e2 - J.rel_rot.e2));
    r = std::max(r, std::fabs(s * rel.e3 - J.rel_rot.e3));
    return r;
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
    // device run on a second ensemble built the same way; the links as the systems hold them
    Built dev = build(c, hht);
    std::vector<double> pose(bd), vel(bd), rec(size_t(steps) * bd), inertia;
    for (int i = 0; i < B; ++i) { pose_of(dev.lists[i], &pose[size_t(i) * D]); vel_of(dev.lists[i], &vel[size_t(i) * D]); }
    for (const auto& j : c.inertia) { inertia.push_back(j.x()); inertia.push_back(j.y()); inertia.push_back(j.z()); }
    const int child = 0, parent = c.to_ground ? -1 : 1;
    hc_sim_prismatic pr{child, parent, {0.0, 0.0, 1.0}};
    const ChVector3d p2 = c.to_ground ? ChVector3d(0, 0, -5) : c.pos[1];
    hc_sim_tsda ts{child, parent, {c.pos[0].x(), c.pos[0].y(), c.pos[0].z()}, {p2.x(), p2.y(), p2.z()}, c.rest};
    std::vector<double> damping(c.damping), stiffness(size_t(B), c.stiffness), energy(size_t(B), 0.0);
    hc_sim_links links{};
    links.n_prismatic = 1; links.n_tsda = 1;
    links.prismatic = &pr; links.tsda = &ts;
    links.tsda_damping = damping.data(); links.tsda_stiffness = stiffness.data(); links.tsda_energy = energy.data();
    hc_sim_params p{};
    p.scheme = hht ? 1 : 0;
    p.t0 = 0.0; p.dt = c.dt; p.n_steps = steps; p.record_every = 1;
    p.g[0] = 0.0; p.g[1] = 0.0; p.g[2] = -9.81;
    p.mass = c.mass.data(); p.inertia = inertia.data();
    p.links = &links;
    int done = 0;
    hc_throw_on_error(hc_ensemble_simulate(dev.ens->ensemble(), &p, pose.data(), vel.data(), nullptr, rec.data(), nullptr,
                                           nullptr, &done));
    double diff = 0.0, amp = 0.0, res = 0.0;
    for (size_t n = 0; n < size_t(steps); ++n) {
        for (size_t k = 0; k < bd; ++k) {
            diff = std::max(diff, std::fabs(rec[n * bd + k] - ref[n * bd + k]));
            amp = std::max(amp, std::fabs(ref[n * bd + k] - x0[k]));
        }
        for (int i = 0; i < B; ++i) res = std::max(res, residual(&rec[n * bd + size_t(i) * D], child, parent, *dev.joints[i]));
    }
    for (double e : energy)
        if (!(e >= 0.0) || !std::isfinite(e)) throw std::runtime_error("spring-damper energy not finite and >= 0");
    std::cout << std::setprecision(6) << "case " << c.name << " scheme " << (hht ? "hht" : "euler") << " steps " << done
              << " max_diff " << diff << " amplitude " << amp << " residual " << res << std::endl;
}

}  // namespace

int main(int argc, char* argv[]) {
    if (argc < 3) { std::cerr << "usage: test_device_links <sphere.h5> <rm3_like.h5> [steps]" << std::endl; return 2; }
    const int steps = argc > 3 ? std::atoi(argv[3]) : 400;
    try {
        Case sphere{"sphere", argv[1], 1, {261.8e3}, {ChVector3d(1, 1, 1)}, {ChVector3d(0, 0, -2)}, {ChVector3d(0, 0, 0)},
                    ChVector3d(0, 0, 0), true, {0.177, 0.706, 2.374}, {2.094395102, 1.047197551, 0.571198664},
                    {0.0, 2.0e5, 4.0e5}, 0.0, -1.0, 0.015};
        Case rm3{"rm3", argv[2], 2, {725834.0, 886691.0},
                 {ChVector3d(20907301.0, 21306090.66, 37085481.11), ChVector3d(94419614.57, 94407091.24, 28542224.82)},
                 {ChVector3d(0, 0, -0.72), ChVector3d(0, 0, -21.29)}, {ChVector3d(0.05, -0.03, 0.0), ChVector3d(-0.02, 0.04, 0.01)},
                 ChVector3d(0.01, -0.02, 0.005), false, {0.5, 1.0, 1.5, 2.0}, {0.6, 0.8, 1.0, 1.2},
                 {0.0, 1.0e6, 2.0e6, 4.0e6}, 0.0, -1.0, 0.01};
        Case rm3s = rm3;
        rm3s.name = "rm3_spring";
        rm3s.stiffness = 5.0e5;
        rm3s.rest = 20.0;
        for (bool hht : {false, true}) {
            run(sphere, hht, steps);
            run(rm3, hht, steps);
            run(rm3s, hht, steps);
        }
    } catch (const std::exception& e) {
        std::cerr << "error: " << e.what() << std::endl;
        return 1;
    }
    return 0;
}
