// Internal host-side structures shared by the C-ABI translation units.
#pragma once
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "hydrochrono_b200.h"

namespace hc {

using dvec = std::vector<double>;

struct StatusError : std::exception {
    hc_status code;
    std::string msg;
    StatusError(hc_status c, std::string m) : code(c), msg(std::move(m)) {}
    const char* what() const noexcept override { return msg.c_str(); }
};
[[noreturn]] inline void fail(hc_status c, const std::string& m) { throw StatusError(c, m); }

void set_last_error(const std::string& m);

// ---- hydro tables on the host (HydroData, src/h5fileinfo.cpp:27-91) -------------------------
struct BodyTables {
    double disp_vol = 0;
    dvec rirf_t;       // [L]
    dvec cg, cb;       // [3]
    dvec lin;          // [36]    unscaled K_h
    dvec ainf;         // [6][D]  x rho
    dvec K;            // [6][D][L] raw
    dvec exc_mag;      // [6][nw] x rho*g
    dvec exc_phase;    // [6][nw]
    dvec exc_irf_t;    // [Le0]
    dvec exc_irf_f;    // [6][Le0] x rho*g
};

struct TaperOpts {
    bool moving_average = false;
    int window_length = 5;
    double rirf_end_time = -1.0;
    double start_percent = 0.8, end_percent = 1.0, final_amplitude = 0.0;
};

}  // namespace hc

struct hc_tables {
    int N = 0, D = 0, L = 0, nw = 0, Le0 = 0;
    double rho = 0, g = 0, depth = 0;
    std::vector<hc::BodyTables> body;
    hc::dvec w_list;
    hc::dvec rirf_t, rirf_w;   // shared time vector + trapezoid widths (hydro_forces.cpp:179-190)
    hc::dvec equilibrium;      // [D]
    hc::dvec cb_minus_cg;      // [3N]
    int conv_mode = 0;         // 0 Baseline, 1 TaperedDirect
    hc::dvec Keff;             // [D][D][L] effective kernel = rho*K or processed (what GetRIRFval returns)
    void rebuild_effective_kernel(const hc::TaperOpts* taper);
};

namespace hc {

// ---- setup-time wave maths (host), src/wave_types.cpp ---------------------------------------
dvec linspaced(int n, double lo, double hi);                       // Eigen LinSpaced semantics
dvec trapezoid_widths(const dvec& x);                              // GetWidthArray, :608-620
double wave_number(double omega, double depth, double g);          // ComputeWaveNumber, :178-255
dvec pierson_moskowitz(dvec f, double Hs, double Tp);              // :679-693
dvec jonswap(dvec f, double Hs, double Tp, double gamma, bool normalized);  // :695-715
dvec random_phases(int seed, int n);                               // :663-669 (std::mt19937 + uniform_real)
// cubic interpolating B-spline with knot averaging through rows of pts [dim][n] at u = LinSpaced(n,0,1),
// evaluated at LinSpaced(m,0,1)  (Eigen SplineFitting::Interpolate as used by ResampleIRF, :594-602)
void bspline_resample(const double* pts, int dim, int n, int m, double* out);

struct ExcIrfBody {       // resampled excitation IRF for one body (:572-628)
    dvec t, w, f;         // [Le], [Le], [6][Le]
};
std::vector<ExcIrfBody> resample_excitation_irf(const hc_tables& T, double dt);

// Radiation look-ahead planning (hc_plan.cpp): positions of the RIRF lags on the history-row grid
struct RadPlan {
    bool usable = false;
    bool general = false;     // lag spacing is not a multiple of dt: row-grid kernel with the lerp weights folded in
    int m = 1;                // history rows per lag (lag-grid path), 1 on the row grid
    int Lk = 0;               // lags of the kernel the block path convolves with (L, or rows of the row grid)
    dvec pnom;                // [L] nominal position of every lag, in rows back from the step
    std::vector<int> pi;      // [L] its integer part (bracket index)
    dvec pw;                  // [L] its fraction (weight of the older row)
};
RadPlan make_rad_plan(const hc_tables& T, double dt, int max_m, int min_lags);
bool rad_plan_step(const hc_tables& T, const RadPlan& P, const double* tm, int len, double snap, int& smax);
dvec rad_plan_row_kernel(const hc_tables& T, const RadPlan& P);
bool rad_pass_next(long long N, int nslices, int& next_slice, long long& next_item, int count, long long wave,
                   long long& i0, long long& i1);

// H5 reader (hc_h5.cpp)
hc_tables* load_bemio_h5(const char* path, int num_bodies);
hc_tables* tables_from_desc(const hc_tables_desc& d);

}  // namespace hc

// hc_multi_ensemble_simulate's per-shard call (hc_ensemble.cu): hc_ensemble_simulate on host arrays whose record k
// starts at element k * rec_stride (a shard's slice of global-order records)
extern "C" hc_status hc_ensemble_simulate_strided(hc_ensemble* e, const hc_sim_params* p, double* pose, double* vel,
                                                  double* rec_t, double* rec_pose, double* rec_vel, size_t rec_stride,
                                                  double* pto_energy, int* steps_done);
