// Water kinematics of every instance of a hydro.yaml sweep ensemble (TestHydroEnsemble::GetWaveKinematics): one
// sphere system per (period value x seed), set up by SetupHydroSweepFromYAML, then elevation, velocity and acceleration
// at fixed points and times for the whole batch in one device call per time.
// usage: test_ensemble_kinematics <hydro.yaml> <out.txt> [seeds per period = 1] [duration = 20]
// out: one line per (time, instance, point): t instance x y z eta vx vy vz ax ay az
#include <hydroc/hydro_ensemble.h>
#include <hydroc/hydro_yaml_parser.h>

#include <cstdlib>
#include <fstream>
#include <iomanip>
#include <iostream>

using namespace chrono;

int main(int argc, char* argv[]) {
    if (argc < 3) { std::cerr << "usage: test_ensemble_kinematics <hydro.yaml> <out.txt> [seeds] [duration]" << std::endl; return 2; }
    const int seeds_per_period = argc > 3 ? std::atoi(argv[3]) : 1;
    const double duration = argc > 4 ? std::atof(argv[4]) : 20.0;
    const double dt = 0.015, ramp = 3.0;
    try {
        YAMLHydroData y = ReadHydroYAML(argv[1]);
        const int P = std::max<size_t>(1, y.waves.period_values.size());
        const int B = P * seeds_per_period;
        std::vector<std::unique_ptr<ChSystemNSC>> systems;
        std::vector<TestHydroEnsemble::BodyList> lists;
        for (int i = 0; i < B; ++i) {
            systems.push_back(std::make_unique<ChSystemNSC>());
            auto body = chrono_types::make_shared<ChBody>();
            body->SetName("body1");
            systems.back()->AddBody(body);
            lists.push_back({body});
        }
        std::unique_ptr<TestHydroEnsemble> ens = SetupHydroSweepFromYAML(y, lists, dt, duration, ramp, seeds_per_period);
        // below, at and above the mean water level, x across +-40 m
        const double pts[][3] = {{0.0, 0.0, -2.0}, {12.5, 1.0, 0.0}, {-37.0, -2.0, 0.4}, {40.0, 0.0, -25.0}};
        const int np = 4;
        std::vector<double> points(size_t(B) * np * 3);
        for (int i = 0; i < B; ++i)
            for (int p = 0; p < np; ++p)
                for (int c = 0; c < 3; ++c) points[(size_t(i) * np + p) * 3 + c] = pts[p][c];
        std::ofstream out(argv[2]);
        out << std::setprecision(17);
        std::vector<double> eta, vel, acc;
        for (double t : {0.0, 1.7, 250.3}) {
            ens->GetWaveKinematics(t, np, points, &eta, &vel, &acc);
            for (int i = 0; i < B; ++i)
                for (int p = 0; p < np; ++p) {
                    const size_t o = size_t(i) * np + p;
                    out << t << ' ' << i << ' ' << pts[p][0] << ' ' << pts[p][1] << ' ' << pts[p][2] << ' ' << eta[o];
                    for (int c = 0; c < 3; ++c) out << ' ' << vel[3 * o + c];
                    for (int c = 0; c < 3; ++c) out << ' ' << acc[3 * o + c];
                    out << '\n';
                }
        }
        std::cout << "instances " << B << " device_evaluations " << ens->DeviceEvaluations() << std::endl;
    } catch (const std::exception& e) {
        std::cerr << "error: " << e.what() << std::endl;
        return 1;
    }
    return 0;
}
