// Ensemble: device-resident state of B lock-stepped TestHydro instances and the per-step driver.
//
// Host-side logic restated from TestHydro (src/hydro_forces.cpp): the time-keyed force cache (:742-755), the
// duplicate-evaluation guard (:555-557), history push + pruning (:559-577, :327-340) -- all functions of the
// time values alone, which are shared by every instance, so they run once on the host; everything that touches
// per-instance data runs in the kernels of hc_kernels.cu.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>

#include "hc_internal.h"
#include "hc_kernels.cuh"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace hc {

#define CUDA_CHECK(expr)                                                                            \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            fail(HC_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #expr); \
    } while (0)

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    // The ensemble's streams are non-blocking: they do NOT order against the legacy default stream that cudaMemset /
    // cudaMemcpy run on, and both may return before the device has finished (memset is asynchronous; a pageable H2D
    // returns once the data is staged).  Every fill therefore ends with a wait on that stream -- otherwise a kernel or
    // copy enqueued right afterwards on the ensemble's stream can be overtaken by the fill (seen as a history ring
    // zeroed AFTER grow_ring had copied the rows into it, once in ~15 runs).
    void alloc(size_t count, bool zero = true) {
        release();
        if (count == 0) return;
        CUDA_CHECK(cudaMalloc(&p, count * sizeof(T)));
        n = count;
        if (zero) {
            CUDA_CHECK(cudaMemset(p, 0, count * sizeof(T)));
            CUDA_CHECK(cudaStreamSynchronize(cudaStreamLegacy));
        }
    }
    void upload(const T* src, size_t count) {
        alloc(count, false);
        CUDA_CHECK(cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaStreamSynchronize(cudaStreamLegacy));
    }
    void upload(const std::vector<T>& v) { upload(v.data(), v.size()); }
};

struct PinBuf {
    void* p = nullptr;
    ~PinBuf() { if (p) cudaFreeHost(p); }
    void alloc(size_t bytes) {
        if (p) cudaFreeHost(p);
        p = nullptr;
        CUDA_CHECK(cudaMallocHost(&p, bytes));
        std::memset(p, 0, bytes);
    }
};

enum { EV_BEGIN = 0, EV_PLAN, EV_EXC, EV_RAD, EV_APPEND, EV_END, EV_COUNT };

}  // namespace hc

using namespace hc;

struct hc_ensemble {
    const hc_tables* T = nullptr;
    hc_ensemble_opts opts{};
    int dev = 0, B = 0, Bp = 0, D = 0, N = 0, L = 0, sm_count = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = false;

    // static tables on the device
    DevBuf<double> d_K, d_Kfrag, d_Khyb, d_rirf_t, d_rirf_w, d_ainf;
    bool rad_mma = false;             // D = 12: FP64 tensor-core (DMMA) radiation kernel
    bool rad_hybrid = false;          // D = 12: rows 0..7 on the tensor cores + rows 8..11 on the FMA pipe
    HydrostaticTables hs{};

    // history ring
    DevBuf<double> d_hist, d_times;
    int cap = 0, head = -1;
    std::deque<double> times;         // newest first, mirrors TestHydro::time_history_
    double prev_time = -1.0;          // hydro_forces.cpp:176
    bool force_valid = false;

    // radiation plan + partials
    DevBuf<int> d_pr_new, d_pr_old;
    DevBuf<double> d_pr_wn, d_pr_wo, d_pr_wd, d_pr_head, d_rad_partial;
    DevBuf<int> d_pr_lead;
    int rad_chunk = 0, rad_nchunk = 0;

    // radiation look-ahead (D = 12): resident rows' share of the next kRbT steps in one pass (k_rad_block<12>)
    bool rb_enabled = false, rb_use = false;      // configured / serving the current step
    int rb_R = 0, rb_nchunk = 0, rb_m = 1;        // rows per chunk, chunks, history rows per RIRF lag
    int rb_occ = 3;
    bool rb_general = false;                      // RIRF lag spacing is not a multiple of dt: row-grid kernel (below)
    int rb_Lk = 0;                                // lags of the kernel the block path convolves with (L, or row grid)
    std::vector<double> rb_pnom;                  // [L] nominal position of every lag in history rows (rirf_t / dt)
    RadPlan rb_plan;                              // the same + bracket index / older-row weight per lag (hc_plan.cpp)
    DevBuf<double> d_Kyoung;                      // first 2 kRbT lags of that kernel, [lag][col][row] (k_step)
    DevBuf<double> d_Kpad, d_rb_partial[2];
    DevBuf<int> d_rb_smax[2];
    std::vector<double> rb_scratch;
    struct RbBlock {
        double times[kRbT * kRbMaxM]; int smax[kRbT * kRbMaxM];
        int len = 0, nchunk_used = 0, base = 0; bool valid = false;
    } rbk[2];                                     // double-buffered: the block being served / the one evaluated ahead
    int rb_cur = 0, rb_pos = 0;
    bool rb_ahead = false;                        // next block evaluated one block ahead, one slice after every step
    struct RbPass {
        RadBlockArgs args{};
        int items = 0, next_slice = 0, nslices = 0;
        long long next_item = 0;                  // where the next slice starts
        bool active = false;
    } rb_pass;
    cudaStream_t rb_stream = nullptr;             // the pass of the block evaluated ahead runs here
    cudaEvent_t ev_rb_side = nullptr;             // last slice enqueued on rb_stream
    cudaEvent_t ev_rb_snap = nullptr;             // main stream at the block's snapshot of the history
    bool rb_side_pending = false;
    int rb_pass_mode = 1;                         // 1 slice per step gated by the step's forces, 2 slice per step
                                                  // ungated, 3 whole pass at the block's first step
    bool last_step_fast = false;                  // the previous step had an empty phase 1 (both look-aheads served it)
    bool inputs_on_copy_stream = false;           // hc_step: the state upload of this step is on copy_stream (ev_inputs)
    StepHeader hdr_h{};                           // header of the step being enqueued (k_step takes it by value)
    bool hdr_on_device = false;                   // ... and whether this step also needs it in d_hdr
    bool host_stepping = false;                   // the current step came through hc_step (host buffers)
    int rb_builds = 0, rb_hits_this_block = 0, rb_poor_blocks = 0;
    long long rb_launches = 0, rb_steps_served = 0, rb_items_timed = 0;
    int rb_items_pending = 0, rb_items_per_pass = 0;
    double rb_ms_sum = 0.0;
    cudaEvent_t ev_rb[2] = {nullptr, nullptr};
    bool rb_events_pending = false;
    int graph_key[3] = {-1, -1, -1};
    // HC_TRACE=1: device-side timeline of hc_step (H2D, wait for phase 2 to start, phase 2, D2H), printed at destroy
    bool trace = false;
    cudaEvent_t ev_tr[6] = {};
    double tr_ms[6] = {0, 0, 0, 0, 0, 0};
    long long tr_n = 0;              // what the captured graph of each phase contains

    // step I/O
    // the step's inputs live in ONE device block [header (256 B) | vel [B][D] | pose [B][D]] so that a small ensemble can
    // receive all of them in a single copy (compact host path, below)
    DevBuf<unsigned char> d_stage;
    struct Ptr { StepHeader* p = nullptr; } d_hdr;
    struct DPtr { double* p = nullptr; } d_pose, d_vel;
    DevBuf<double> d_force, d_comp, d_wave_tmp;
    // compact host path (hc_step on a small ensemble served by the per-step kernels -- the drop-in B = 1 case): inputs
    // staged in one pinned block, ONE captured graph per step = H2D of the block + every kernel of the step + D2H of
    // the forces; one driver call + one synchronise instead of nine calls
    PinBuf h_stage;
    size_t stage_bytes = 0;
    bool compact_ok = false, defer_launch = false;
    double* h_force_dev = nullptr;                // device-side address of the pinned force buffer (compact graph writes it directly)
    bool compact_fork = true;                     // HC_COMPACT_FORK=0: excitation and radiation convolutions in sequence (diagnostic)
    bool compact_inline = true;                   // HC_COMPACT_INLINE=0: keep the plan kernel in the compact graph (diagnostic)
    bool compact_capture = false;                 // enqueue_phase is recording the compact graph (state already on the device)
    cudaEvent_t ev_cfork = nullptr, ev_cjoin = nullptr;
    cudaStream_t fork_stream = nullptr;           // second branch of a captured graph (never runs work outside a capture)
    bool phase1_capture = false;                  // enqueue_phase is recording the phase-1 graph of the per-step path
    int fork_max_batch = 2048;                    // phase-1 graph: parallel convolution branches up to this ensemble size
    void ensure_fork_objects();
    cudaGraph_t graph_c = nullptr;
    cudaGraphExec_t graph_c_exec = nullptr;
    int graph_c_key = -1;
    bool graph_c_inline = false;                  // the captured compact graph has no plan kernel
    void run_compact();

    PinBuf h_pose, h_vel, h_force;

    // device-side stepping (hc_ensemble_simulate).  d_sim holds [B][D] slots: evaluation pose / velocity ping-pong pairs
    // (what the force path reads), HHT state and history, the spring rest pose and the energy of the host variant;
    // d_simq the state and predictor orientations [B][N][4] each.  The force path's kernels read the evaluation state
    // through the step header on the ensemble's stream only (the look-ahead passes on the side streams read the history
    // ring), so a buffer is free again once the next step's k_body_step has read it.
    enum { kSimPose0 = 0, kSimPose1, kSimVel0, kSimVel1, kSimX, kSimV, kSimFn, kSimAn, kSimX0, kSimEnergy, kSimSlots };
    DevBuf<double> d_sim, d_simq, d_minv, d_pto, d_rec;
    PinBuf h_rec;
    size_t h_rec_bytes = 0;
    bool sim_q_valid = false;                     // d_simq holds the orientations of the last run's final state
    double* sim(int slot) { return d_sim.p + size_t(slot) * B * D; }
    // runs with joints / spring-dampers (k_body_step_linked): full mass matrix, per-instance assembly data, the pose the
    // last linked run ended in (continuation test), spring-damper coefficients [2][B][n_tsda] and the host variant's energy
    DevBuf<double> d_link_M, d_link_asm, d_link_end, d_link_coef, d_link_energy;
    bool link_asm_valid = false;                  // d_link_asm / d_link_end belong to the last run, which had links link_key
    std::vector<double> link_key;

    // waves
    int wave_mode = 0;
    DevBuf<double> d_reg_amp, d_reg_omega, d_reg_mag, d_reg_phase;
    std::vector<double> reg_mag_h, reg_phase_h, reg_k_h;   // [count][D], [count][D], [count]
    std::vector<double> reg_amp_h, reg_omega_h, reg_wave_phase_h;   // [count] each (the wave itself: kinematics)
    int reg_count = 0;
    // irregular
    hc_irregular_params ip{};
    std::vector<ExcIrfBody> irf;      // per body, host
    struct Group {
        int dof0, nd, Le, chunk0, nchunk;
        DevBuf<double> tau, fw, w1, w2;
        DevBuf<int> idx;
        double tau_first, tau_last;
        // look-ahead block: per-(time, lag) brackets and per-row taps
        DevBuf<int> la_idx;
        DevBuf<double> la_w1, la_w2, la_taps;
        int la_rows_cap = 0;
        int la_row0 = 0, la_nrows = 0;    // eta rows of the block being built (second half of a split build)
    };
    std::vector<std::unique_ptr<Group>> groups;
    int exc_chunk = 0, exc_total_chunks = 0, exc_ndmax = 0;
    DevBuf<double> d_exc_partial, d_eta, d_eta_t, d_omega, d_amp, d_phase;
    std::vector<double> eta_t_h, freqs_h, widths_h, wavenumbers_h;
    double eta_grid_dt = 0.0;                     // nominal spacing of the eta grid (index guess of the excitation plans)
    void setup_excitation_groups(double simulation_dt);
    std::vector<double> S_h;          // [nS][nf]  (nS = 1 shared or B)
    std::vector<double> phases_h;     // [B][nf]
    bool per_instance_spectrum = false;
    int n_eta = 0, nf = 0;
    void pack_irregular(std::vector<double>& amp, std::vector<double>& ph) const;
    // water kinematics (hc_waves_kinematics_at_time): the wave's components staged on the first call (per-instance
    // phases and amplitudes [nf][Bp], 8 B x nf x Bp each), released whenever the waves are set again
    DevBuf<double> d_kin_comp, d_kin_amp, d_kin_phase, d_kin_io;
    bool kin_staged = false;
    void stage_kinematics();
    void release_kinematics() {
        d_kin_comp.release(); d_kin_amp.release(); d_kin_phase.release(); d_kin_io.release();
        kin_staged = false;
    }
    void enqueue_kinematics(double t, int n_points, const double* d_points, double mwl, int wheeler, double* d_eta,
                            double* d_vel, double* d_acc);
    // excitation look-ahead (state-independent wave force evaluated kLaT predicted steps at a time)
    bool la_enabled = false;
    double la_dt = 0.0;
    struct LaBlock { std::vector<double> times; int len = 0; bool valid = false; };
    LaBlock la_blk[2];                // double-buffered blocks of predicted times / cached wave forces
    int la_cur = 0, la_pos = 0;       // block being consumed / next slot expected
    bool la_background = false;       // next block evaluated on a side stream under the current block's steps
    bool la_mma = false;              // look-ahead block on the FP64 tensor cores (DMMA)
    int la_S = 1;                     // eta-row segments of the DMMA block kernel (partials summed by k_finalize)
    cudaStream_t la_stream = nullptr;
    cudaEvent_t ev_la_done[2] = {nullptr, nullptr}, ev_la_free[2] = {nullptr, nullptr}, ev_la_build = nullptr;
    cudaEvent_t ev_la_join = nullptr;
    int la_builds = 0, la_hits_this_block = 0, la_poor_blocks = 0;
    long long la_blocks_built = 0, la_steps_served = 0;   // hc_get_exc_block_stats (never cleared by a reset)
    DevBuf<double> d_la_cache, d_la_times;
    cudaEvent_t ev_la[2] = {nullptr, nullptr};
    bool la_events_pending = false;

    // graph + profiling
    cudaGraph_t graph = nullptr, graph1 = nullptr;          // phase 2 / phase 1
    cudaGraphExec_t graph_exec = nullptr, graph1_exec = nullptr;
    bool graph_valid = false, graph1_valid = false;
    cudaStream_t copy_stream = nullptr;                     // H2D of pose/vel overlaps phase 1
    cudaEvent_t ev_inputs = nullptr, ev_force = nullptr;   // state uploaded / forces of the step ready
    bool profiling = false;
    int phase1_launches = 0;
    bool phase_uses_lookahead = false;    // set per step: phase 1 skips the per-step excitation kernels
    bool skip_radiation = false;          // wave-only evaluation (hc_waves_force_at_time)
    cudaEvent_t ev[EV_COUNT] = {};
    hc_profile_stats prof{};
    double acc_ms[4] = {0, 0, 0, 0};
    long long ms_steps = 0;
    bool events_pending = false;

    ~hc_ensemble() {
        cudaSetDevice(dev);
        if (trace && tr_n > 0)
            fprintf(stderr, "[hc trace] steps %lld  h2d %.1f us  h2d_end->phase2_start %.1f us  phase2 %.1f us  d2h %.1f us  "
                            "device total %.1f us  host call %.1f us\n", tr_n, 1e3 * tr_ms[0] / tr_n, 1e3 * tr_ms[1] / tr_n,
                    1e3 * tr_ms[2] / tr_n, 1e3 * tr_ms[3] / tr_n, 1e3 * tr_ms[4] / tr_n, 1e3 * tr_ms[5] / tr_n);
        for (auto& x : ev_tr) if (x) cudaEventDestroy(x);
        drop_graph();
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        if (own_stream && stream) cudaStreamDestroy(stream);
        if (ev_cfork) cudaEventDestroy(ev_cfork);
        if (ev_cjoin) cudaEventDestroy(ev_cjoin);
        if (fork_stream) cudaStreamDestroy(fork_stream);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (ev_inputs) cudaEventDestroy(ev_inputs);
        if (ev_force) cudaEventDestroy(ev_force);
        if (la_stream) { cudaStreamSynchronize(la_stream); cudaStreamDestroy(la_stream); }
        for (auto& x : ev_la) if (x) cudaEventDestroy(x);
        for (auto& x : ev_la_done) if (x) cudaEventDestroy(x);
        for (auto& x : ev_la_free) if (x) cudaEventDestroy(x);
        if (ev_la_build) cudaEventDestroy(ev_la_build);
        if (ev_la_join) cudaEventDestroy(ev_la_join);
        for (auto& x : ev_rb) if (x) cudaEventDestroy(x);
        if (rb_stream) { cudaStreamSynchronize(rb_stream); cudaStreamDestroy(rb_stream); }
        if (ev_rb_side) cudaEventDestroy(ev_rb_side);
        if (ev_rb_snap) cudaEventDestroy(ev_rb_snap);
    }
    void drop_graph() {
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        if (graph) cudaGraphDestroy(graph);
        if (graph1_exec) cudaGraphExecDestroy(graph1_exec);
        if (graph1) cudaGraphDestroy(graph1);
        graph_exec = nullptr; graph = nullptr; graph_valid = false;
        graph1_exec = nullptr; graph1 = nullptr; graph1_valid = false;
        if (graph_c_exec) cudaGraphExecDestroy(graph_c_exec);
        if (graph_c) cudaGraphDestroy(graph_c);
        graph_c_exec = nullptr; graph_c = nullptr; graph_c_key = -1;
    }
    void use_device() const { CUDA_CHECK(cudaSetDevice(dev)); }

    void stage_kernel();
    void alloc_ring(int new_cap);
    void grow_ring();
    void setup_radiation_chunks();
    void setup_radiation_block();
    bool rb_step_plan(const double* tm, int len, double snap, int& smax) const;
    int radiation_block_slot(double t, StepHeader& hh);
    int rb_plan_block(RbBlock& Bk, double t, int base);
    void rb_setup_pass(int buf);
    void rb_launch_slices(int count, bool side);
    void rb_join_side();
    void rb_begin_ahead(int buf, double t);
    void rb_invalidate() { rbk[0].valid = rbk[1].valid = false; rb_pos = 0; rb_pass.active = false; }
    void enqueue_phase(int phase, bool with_events);
    void launch_phase(int phase);
    void begin_step(double t, const double* g, const double* d_pose_in, const double* d_vel_in, double* d_force_out);
    void setup_lookahead();
    int lookahead_slot(double t);
    int enqueue_lookahead_block(int buf, double t0, cudaStream_t st, int part = -1);
    void finish_split_build();
    int la_half_pending = -1;         // buffer whose block still lacks the second half of its segments
    void prefetch_lookahead(int buf);
    void finish_step(double t);
    void collect_events();
};

// (K w) staged as [lag][col][row] (one lag's D x D block contiguous, rows fastest) and, for D = 12, additionally in
// DMMA A-fragment order [lag][M-tile 0..1][k-step 0..2][lane]: element (row = mt*8 + lane/4, col = ks*4 + lane%4),
// rows 12..15 zero.
void hc_ensemble::stage_kernel() {
    const hc_tables* t = T;
    std::vector<double> Kdev(size_t(L) * D * D);
    for (int r = 0; r < D; ++r)
        for (int c = 0; c < D; ++c)
            for (int s = 0; s < L; ++s) Kdev[(size_t(s) * D + c) * D + r] = t->Keff[(size_t(r) * D + c) * L + s] * t->rirf_w[s];
    d_K.upload(Kdev);
    if (rad_mma) {
        std::vector<double> Kf(size_t(L) * 192, 0.0);
        for (int s = 0; s < L; ++s)
            for (int mt = 0; mt < 2; ++mt)
                for (int ks = 0; ks < 3; ++ks)
                    for (int lane = 0; lane < 32; ++lane) {
                        const int r = mt * 8 + lane / 4, c = ks * 4 + lane % 4;
                        if (r < D) Kf[(size_t(s) * 6 + mt * 3 + ks) * 32 + lane] = t->Keff[(size_t(r) * D + c) * L + s] * t->rirf_w[s];
                    }
        d_Kfrag.upload(Kf);
    }
    if (rad_hybrid) {
        std::vector<double> Kh(size_t(L) * 144, 0.0);
        for (int s = 0; s < L; ++s) {
            double* o = &Kh[size_t(s) * 144];
            auto kw = [&](int r, int c) { return t->Keff[(size_t(r) * D + c) * L + s] * t->rirf_w[s]; };
            for (int ks = 0; ks < 3; ++ks)
                for (int lane = 0; lane < 32; ++lane) o[ks * 32 + lane] = kw(lane / 4, ks * 4 + lane % 4);
            for (int q = 0; q < 4; ++q)
                for (int ks = 0; ks < 3; ++ks)
                    for (int r = 0; r < 4; ++r) o[96 + q * 12 + ks * 4 + r] = kw(8 + r, ks * 4 + q);
        }
        d_Khyb.upload(Kh);
    }
    if (rb_plan.usable && rb_nchunk > 0) {        // look-ahead CONFIGURED (it may be switched off at run time and back on)
        // The kernel the block path convolves the history ROWS with, Krow[i][r][c], i = rows back.  Lag spacing a
        // multiple of dt: Krow = (K w) on the lag grid (row m s <-> lag s).  Otherwise the linear interpolation of the
        // velocity between rows i and i + 1 at the nominal position x_s = t_rirf[s] / dt = i + wo is folded into the
        // kernel:  (K w)[s] (wn v_i + wo v_{i+1})  ->  Krow[i] += wn (K w)[s],  Krow[i + 1] += wo (K w)[s].
        const std::vector<double> Krow = rad_plan_row_kernel(*t, rb_plan);     // hc_plan.cpp, [rb_Lk][D][D]
        // device copies: [lag][row][col padded to a multiple of 4] with lag stride rb_stride(D), zero beyond the last
        // lag (rows older than the kernel's support), and the first lags as [lag][col][row] for k_step
        const int lags = rb_nchunk * rb_R + 2 * kRbT + 1;
        const int stride = rb_stride(D), dp = rb_dp(D);
        std::vector<double> Kp(size_t(lags) * stride, 0.0);
        for (int i = 0; i < rb_Lk; ++i)
            for (int r = 0; r < D; ++r)
                for (int c = 0; c < D; ++c) Kp[size_t(i) * stride + r * dp + c] = Krow[(size_t(i) * D + r) * D + c];
        d_Kpad.upload(Kp);
        const int ny = 2 * kRbT;
        std::vector<double> Ky(size_t(ny) * D * D, 0.0);
        for (int i = 0; i < std::min(ny, rb_Lk); ++i)
            for (int r = 0; r < D; ++r)
                for (int c = 0; c < D; ++c) Ky[(size_t(i) * D + c) * D + r] = Krow[(size_t(i) * D + r) * D + c];
        d_Kyoung.upload(Ky);
    }
}

// ---------------------------------------------------------------------------------------
void hc_ensemble::alloc_ring(int new_cap) {
    d_hist.alloc(size_t(new_cap) * D * Bp);
    d_times.alloc(new_cap);
    cap = new_cap;
    head = -1;
}

// Ring too small for the step size actually used: double it, keeping the live entries in order.
void hc_ensemble::grow_ring() {
    const int old_cap = cap, len = int(times.size());
    const int new_cap = old_cap * 2;
    DevBuf<double> nh, nt;
    nh.alloc(size_t(new_cap) * D * Bp);
    nt.alloc(new_cap);
    const size_t row = size_t(D) * Bp;
    CUDA_CHECK(cudaStreamSynchronize(stream));
    // history index i (0 = newest) moves from slot (head - i) mod old_cap to slot len-1-i
    for (int i = 0; i < len; ++i) {
        int s = head - i;
        if (s < 0) s += old_cap;
        CUDA_CHECK(cudaMemcpyAsync(nh.p + size_t(len - 1 - i) * row, d_hist.p + size_t(s) * row, row * sizeof(double),
                                   cudaMemcpyDeviceToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(nt.p + (len - 1 - i), d_times.p + s, sizeof(double), cudaMemcpyDeviceToDevice, stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
    std::swap(d_hist.p, nh.p); std::swap(d_hist.n, nh.n);
    std::swap(d_times.p, nt.p); std::swap(d_times.n, nt.n);
    cap = new_cap;
    head = len - 1;
    drop_graph();
}

// Lag-chunk size such that the grid (instance tiles x chunks) fills an integer number of waves of resident CTAs:
// the smallest wave count whose chunk fits the shared-memory budget for `occ_target` CTAs per SM.
static int pick_chunk(int n_lags, int tiles, int sm_count, int occ_target, size_t smem_budget,
                      size_t (*smem_of)(int, int), int width, int min_chunk) {
    const int slots = sm_count * occ_target;
    for (int waves = 1; waves <= 64; ++waves) {
        const int n = (waves * slots) / tiles;
        if (n < 1) continue;
        int chunk = (n_lags + n - 1) / n;
        if (chunk < min_chunk) return std::min(min_chunk, n_lags);
        if (smem_of(width, chunk) <= smem_budget) return chunk;
    }
    return std::min(std::max(min_chunk, 8), n_lags);
}

void hc_ensemble::setup_radiation_chunks() {
    const int tile_inst = rad_hybrid ? kHybTileInst : kTileInst;
    const int tiles = (Bp + tile_inst - 1) / tile_inst;
    int chunk = opts.rad_chunk;
    if (chunk <= 0 && rad_hybrid) chunk = pick_chunk(L, tiles, sm_count, 3, size_t(72) * 1024, radiation_smem_bytes, D, 4);
    if (chunk <= 0) {
        const bool templated = (D == 6 || D == 12);
        const int occ = templated ? 2 : 4;
        auto smem_of = rad_mma ? +[](int, int chunk) -> size_t { return radiation_mma_smem_bytes(chunk); }
                       : (templated ? radiation_smem_bytes : +[](int, int) -> size_t { return 0; });
        chunk = pick_chunk(L, tiles * (templated ? 1 : D / 6), sm_count, occ, size_t(110) * 1024, smem_of, D, 4);
    }
    chunk = std::max(1, std::min(chunk, L));
    // clamp with the shared memory of the kernel that launch_radiation will pick (a user rad_chunk is not checked
    // elsewhere): the DMMA kernel stages 16-row fragments, more per lag than the FMA and hybrid kernels
    auto launch_smem = [&](int c) -> size_t {
        if (rad_mma) return radiation_mma_smem_bytes(c);
        return (D == 6 || D == 12) ? radiation_smem_bytes(D, c) : 0;
    };
    while (chunk > 1 && launch_smem(chunk) > 200 * 1024) chunk /= 2;
    rad_chunk = chunk;
    rad_nchunk = (L + chunk - 1) / chunk;
    d_rad_partial.alloc(size_t(rad_nchunk) * D * Bp);
}

// Radiation look-ahead configuration.  RIRF lag spacing = m dt with an integer m: the block works on the lag grid,
// one residue class of history rows per step (rb_m = m).  Any other ratio: the block works on a row-grid kernel with
// the interpolation weights folded in (rb_general, rb_m = 1; stage_kernel).  Row chunks of R rows per residue class
// such that (instance tiles x chunks x m) fills whole waves of resident CTAs.
void hc_ensemble::setup_radiation_block() {
    rb_enabled = false; rb_invalidate();
    rb_plan = RadPlan{}; rb_nchunk = 0;
    const int want = opts.rad_lookahead;
    if (want == 1 || (D != 6 && D != 12 && D != 18) || opts.dt_hint <= 0.0) return;
    const int tiles = Bp / kRbTileInst;
    if (want == 0 && (tiles < sm_count || !(opts.bracket_snap > 0.0))) return;       // auto: large ensembles only
    rb_plan = make_rad_plan(*T, opts.dt_hint, kRbMaxM, 2 * kRbT);      // hc_plan.cpp
    if (!rb_plan.usable) return;
    rb_general = rb_plan.general; rb_m = rb_plan.m; rb_Lk = rb_plan.Lk; rb_pnom = rb_plan.pnom;
    rb_occ = (D <= 12) ? 3 : 2;                                    // resident CTAs per SM of k_rad_block<D> (registers)
    rb_R = pick_chunk(rb_Lk - 1, tiles * rb_m, sm_count, rb_occ, size_t(rb_occ == 3 ? 74 : 110) * 1024,
                      rad_block_smem_bytes, D, 8);
    rb_nchunk = (rb_Lk - 1 + rb_R - 1) / rb_R;
    rb_ahead = (want != 3);                                        // 3 = whole pass at the block's first step
    for (int i = 0; i < (rb_ahead ? 2 : 1); ++i) {
        d_rb_partial[i].alloc(size_t(kRbT) * rb_m * rb_nchunk * D * Bp, false);
        d_rb_smax[i].alloc(kRbT * kRbMaxM);
    }
    rb_pass_mode = opts.rad_pass_mode >= 1 && opts.rad_pass_mode <= 3 ? opts.rad_pass_mode : 1;
    if (!ev_rb[0]) { CUDA_CHECK(cudaEventCreate(&ev_rb[0])); CUDA_CHECK(cudaEventCreate(&ev_rb[1])); }
    if (rb_ahead && !rb_stream) {
        int lo = 0, hi = 0;
        CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));     // lo = least priority (numerically largest)
        // gated slices: above the excitation block's stream (they are held back by the steps); ungated / whole pass:
        // below it, or the pass would starve the excitation block that the steps need sooner
        const int prio = rb_pass_mode == 1 ? (lo + hi) / 2 : lo;
        CUDA_CHECK(cudaStreamCreateWithPriority(&rb_stream, cudaStreamNonBlocking, prio));
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_rb_side, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_rb_snap, cudaEventDisableTiming));
    }
    rb_builds = 0; rb_hits_this_block = 0; rb_poor_blocks = 0;
    rb_enabled = true;
}

// The radiation plan of one step (k_prestep's bracket arithmetic, same IEEE operations) reduced to the question the
// block kernel needs answered: does every lag s that has a bracket sit at its nominal position rb_pnom[s] (in history
// rows back from the step, bracket index + weight of the older row) to within bracket_snap?  tm[0 .. len) = the time
// history as it will be at that step, newest first.  smax = the largest lag with a bracket; the row-grid kernel
// needs all of them (full window).
bool hc_ensemble::rb_step_plan(const double* tm, int len, double snap, int& smax) const {
    return rad_plan_step(*T, rb_plan, tm, len, snap, smax);                // hc_plan.cpp
}

// Plans the block whose first step comes `base` steps after the current one (time t, already on `times`): predicted
// times, PruneHistory and plan purity are simulated on the host.  all[] = predicted times newest first, then the
// current history; the step jj after the current one sees all[n - 1 - jj ...].  Returns the number of block steps
// that can be served (every one before the first step that needs a true interpolation).
int hc_ensemble::rb_plan_block(RbBlock& Bk, double t, int base) {
    const int TT = kRbT * rb_m, n = base + TT;
    const double snap = opts.bracket_snap;
    const double window = T->rirf_t.back();
    rb_scratch.resize(size_t(n - 1) + times.size());
    double* all = rb_scratch.data();
    std::copy(times.begin(), times.end(), all + (n - 1));
    double tp = t;
    int len = int(times.size());
    Bk.len = 0; Bk.base = base; Bk.valid = false;
    for (int jj = 0; jj < n; ++jj) {
        double* tm = all + (n - 1 - jj);
        if (jj > 0) {
            tp = tp + opts.dt_hint;                                         // as Chrono advances ChTime
            tm[0] = tp;
            ++len;
            const double t_min = tp - window;                               // PruneHistory
            while (len > 1 && tm[len - 2] < t_min) --len;
        }
        if (jj < base) continue;                                            // steps of the block being served
        int smax = -1;
        if (!rb_step_plan(tm, len, snap, smax)) break;
        Bk.times[jj - base] = tp; Bk.smax[jj - base] = rb_general ? rb_Lk - 1 : smax; Bk.len = jj - base + 1;
    }
    for (int j = Bk.len; j < TT; ++j) { Bk.times[j] = Bk.len ? Bk.times[Bk.len - 1] : t; Bk.smax[j] = -1; }
    const int n_res = std::min(int(times.size()) - 1, rb_m * (rb_Lk - 1));  // rows resident before this step's append
    const int nu = (n_res + rb_m - 1) / rb_m;                               // rows of the fullest residue class
    Bk.nchunk_used = std::max(1, std::min(rb_nchunk, (nu + rb_R - 1) / rb_R));
    return Bk.len;
}

// Prepares the pass that evaluates block `buf` from the current snapshot of the history (head, resident rows).
void hc_ensemble::rb_setup_pass(int buf) {
    RbBlock& Bk = rbk[buf];
    const int TT = kRbT * rb_m;
    // (one small copy per pass of 8 m steps; pageable source, staged at call time)
    CUDA_CHECK(cudaMemcpyAsync(d_rb_smax[buf].p, Bk.smax, TT * sizeof(int), cudaMemcpyHostToDevice, stream));
    RadBlockArgs& ba = rb_pass.args;
    ba = RadBlockArgs{};
    ba.hist = d_hist.p; ba.Kpad = d_Kpad.p; ba.partial = d_rb_partial[buf].p; ba.smax = d_rb_smax[buf].p;
    ba.head0 = head; ba.cap = cap; ba.n_res = std::min(int(times.size()) - 1, rb_m * (rb_Lk - 1));
    ba.D = D; ba.Bp = Bp; ba.R = rb_R; ba.nchunk = rb_nchunk; ba.m = rb_m; ba.g0 = Bk.base / rb_m;
    ba.nchunk_used = Bk.nchunk_used; ba.item0 = 0;
    rb_pass.items = rad_block_items(ba);
    rb_items_per_pass = rb_pass.items;
    rb_pass.next_slice = 0; rb_pass.next_item = 0; rb_pass.nslices = TT; rb_pass.active = true;
    ++rb_launches;
    Bk.valid = true;
}

// Launches the next `count` slices of the pending pass (slice i = items [N i / n, N (i + 1) / n)) on the main stream
// (side = false: a block that must be complete before the step that asked for it) or on the side stream.  There the
// pass of the block evaluated ahead is paced in one of three ways (rb_pass_mode):
//   1  one slice per step, each gated by its step's forces (ev_force): the pass never runs ahead of the steps it is
//      interleaved with, the steps never queue behind it (what a caller that synchronises every step wants);
//   2  one slice per step, not gated: two driver calls per step instead of five;
//   3  the whole pass at the block's first step: one launch per block.
// In modes 2 and 3 the side stream ranks below the excitation block's stream.  Every pass is ordered after the main
// stream's position at the block's snapshot (ev_rb_snap: the rows it reads, the partial buffer it overwrites).
void hc_ensemble::rb_launch_slices(int count, bool side) {
    if (!rb_pass.active) return;
    side = side && !profiling && rb_stream;
    cudaStream_t st = side ? rb_stream : stream;
    const bool gated = side && rb_pass_mode == 1;
    // Back-to-back stepping (hc_step_device): slice boundaries on whole waves of resident CTAs (3 per SM), so that no
    // slice ends in a nearly empty wave.  Host-buffer stepping (hc_step) leaves the GPU a window of copies + caller
    // turnaround after every step: equal slices fit that window best.  A range always starts where the previous one
    // ended (hc_plan.cpp), so a caller may mix the two inside a block.
    const long long wave = host_stepping ? 1 : (long long)sm_count * rb_occ;
    long long i0 = 0, i1 = 0;
    const bool first = rb_pass.next_slice == 0;
    const bool any = rad_pass_next(rb_pass.items, rb_pass.nslices, rb_pass.next_slice, rb_pass.next_item, count, wave, i0, i1);
    const bool last = rb_pass.next_slice >= rb_pass.nslices;
    if (last) rb_pass.active = false;
    if (side && first && !gated) CUDA_CHECK(cudaStreamWaitEvent(rb_stream, ev_rb_snap, 0));
    if (any) {
        RadBlockArgs ba = rb_pass.args;
        ba.item0 = int(i0);
        if (gated) {
            CUDA_CHECK(cudaEventRecord(ev_force, stream));
            CUDA_CHECK(cudaStreamWaitEvent(rb_stream, ev_force, 0));
        }
        if (profiling) CUDA_CHECK(cudaEventRecord(ev_rb[0], st));
        CUDA_CHECK(launch_rad_block(ba, int(i1 - i0), st));
        if (profiling) { CUDA_CHECK(cudaEventRecord(ev_rb[1], st)); rb_events_pending = true; rb_items_pending = int(i1 - i0); }
        prof.kernel_launches += 1;
        if (side) rb_side_pending = true;
    }
}

// Main stream waits for everything enqueued on the side stream (block switch, or a miss that abandons a pass).
void hc_ensemble::rb_join_side() {
    if (!rb_side_pending) return;
    CUDA_CHECK(cudaEventRecord(ev_rb_side, rb_stream));
    CUDA_CHECK(cudaStreamWaitEvent(stream, ev_rb_side, 0));
    rb_side_pending = false;
}

// Look-ahead by one block: at the first step of a block, the NEXT block is planned from the same snapshot of the
// history (g0 = 8) and its pass is cut into one slice per step of the current block, launched on the main stream
// right after each step's phase 2 -- underneath the device -> host copy of the step's forces, the caller's turnaround
// and the next step's host -> device copies.  The ring must not wrap into the snapshot's rows before the pass ends.
void hc_ensemble::rb_begin_ahead(int buf, double t) {
    rbk[buf].valid = false;
    const int TT = kRbT * rb_m;
    RbBlock& Cur = rbk[buf ^ 1];
    if (!rb_ahead || !Cur.valid || Cur.len < TT) return;
    if (int(times.size()) + TT + 2 > cap) return;
    if (rb_plan_block(rbk[buf], t, TT) < TT / 2) return;
    rb_setup_pass(buf);
    if (rb_stream && !profiling && rb_pass_mode != 1) {
        // everything the pass reads (rows appended by earlier steps) or overwrites (partials of the block before the
        // current one) is ordered before this point of the main stream
        CUDA_CHECK(cudaEventRecord(ev_rb_snap, stream));
        if (rb_pass_mode == 3) rb_launch_slices(TT, true);
    }
}

// Position of the step at time t inside the current radiation block, switching to the block evaluated ahead or
// starting a new one (whole pass on the main stream) when needed; -1: the per-step kernels serve this step.  Called
// after the step's time was pushed onto `times`.
int hc_ensemble::radiation_block_slot(double t, StepHeader& hh) {
    const int TT = kRbT * rb_m;
    auto fill = [&](int j) {
        const RbBlock& Bk = rbk[rb_cur];
        ++rb_steps_served; ++rb_hits_this_block;
        hh.rad_src = 1; hh.rb_j = j; hh.rb_jj = Bk.base + j; hh.rb_smax = Bk.smax[j]; hh.rb_nchunk = Bk.nchunk_used;
        hh.rb_buf = rb_cur;
        return j;
    };
    RbBlock& Cur = rbk[rb_cur];
    if (Cur.valid && rb_pos < Cur.len && Cur.times[rb_pos] == t) return fill(rb_pos++);
    RbBlock& Nxt = rbk[rb_cur ^ 1];
    if (rb_ahead && Cur.valid && rb_pos == TT && Nxt.valid && !rb_pass.active && Nxt.len > 0 && Nxt.times[0] == t) {
        rb_cur ^= 1; rb_pos = 0; rb_hits_this_block = 0; rb_poor_blocks = 0;
        rb_join_side();
        rb_begin_ahead(rb_cur ^ 1, t);
        return fill(rb_pos++);
    }
    // miss: first steps, end of a block that has no successor, or a time the prediction did not foresee
    rb_invalidate();
    // row-grid kernel: needs the full window, i.e. a bracket for the oldest lag (k_prestep's test)
    if (rb_general && !(times.back() <= t - T->rirf_t.back())) return -1;
    if (rb_builds > 0 && rb_hits_this_block < 2) {
        if (++rb_poor_blocks >= 3) { rb_enabled = false; return -1; }      // unpredictable stepping: stop trying
    } else {
        rb_poor_blocks = 0;
    }
    rb_hits_this_block = 0;
    if (times.size() < 2) return -1;
    ++rb_builds;
    if (rb_plan_block(rbk[rb_cur], t, 0) < TT / 2) return -1;              // not worth a block pass
    rb_join_side();
    rb_setup_pass(rb_cur);
    rb_launch_slices(TT, false);                                           // the whole pass, now
    rb_pos = 0;
    rb_begin_ahead(rb_cur ^ 1, t);
    return fill(rb_pos++);
}

// The per-step kernel sequence in two phases.  Phase 1 needs only the step header (time): interpolation plans +
// excitation convolution.  Phase 2 needs the step's state: history append, radiation convolution, finalize.
// hc_step overlaps the pose/velocity H2D copy with phase 1.
void hc_ensemble::enqueue_phase(int phase, bool with_events) {
    PrestepArgs pa{};
    pa.hdr = d_hdr.p; pa.hist = d_hist.p; pa.times = d_times.p;
    pa.rirf_t = d_rirf_t.p; pa.rirf_w = d_rirf_w.p;
    pa.pr_new = d_pr_new.p; pa.pr_old = d_pr_old.p; pa.pr_wn = d_pr_wn.p; pa.pr_wo = d_pr_wo.p; pa.pr_wd = d_pr_wd.p;
    pa.pr_head = d_pr_head.p; pa.pr_lead = d_pr_lead.p;
    pa.B = B; pa.Bp = Bp; pa.D = D; pa.L = L;
    pa.ngroups = 0;
    const bool per_step_exc = (wave_mode == 2) && !(la_enabled && phase_uses_lookahead);
    if (per_step_exc) {
        pa.ngroups = int(groups.size());
        for (size_t g = 0; g < groups.size(); ++g) {
            pa.tau[g] = groups[g]->tau.p; pa.Le[g] = groups[g]->Le;
            pa.pe_idx[g] = groups[g]->idx.p; pa.pe_w1[g] = groups[g]->w1.p; pa.pe_w2[g] = groups[g]->w2.p;
        }
        pa.eta_t = d_eta_t.p; pa.n_eta = n_eta; pa.eta_dt = eta_grid_dt;
    }
    if (phase == 1) {
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_BEGIN], stream));
        // convolution over the history that is already resident: every row except this step's own sample
        RadiationArgs ra{};
        ra.hdr = d_hdr.p; ra.K = d_K.p; ra.Kfrag = rad_mma ? d_Kfrag.p : nullptr;
        ra.Khyb = rad_hybrid ? d_Khyb.p : nullptr;
        ra.rirf_t = d_rirf_t.p; ra.rirf_w = d_rirf_w.p; ra.hist = d_hist.p;
        ra.times = d_times.p; ra.partial = d_rad_partial.p;
        ra.L = L; ra.D = D; ra.Bp = Bp; ra.chunk = rad_chunk; ra.nchunk = rad_nchunk;
        const bool run_rad = !skip_radiation && !rb_use;
        // Compact graph: the state is on the device before anything runs.  The convolution kernels plan their own
        // lags / taps and the radiation kernel appends the sample (no k_prestep level); the excitation convolution,
        // independent of the radiation convolution, is a parallel branch of the graph.  Without a radiation kernel
        // that can do so, the append at least rides in the plan kernel.
        // (inline plans in the phase-1 graph of the two-phase path, append left to phase 2, were measured: 91 vs 95 us per
        //  step at 512 instances, no difference at 1024 and 2048 -- the plan kernel hides under the state upload; not kept)
        const bool plan_inline = compact_capture && compact_inline && run_rad && radiation_plans_inline(ra);
        if (compact_capture) graph_c_inline = plan_inline;
        if (!plan_inline && (!rb_use || per_step_exc)) CUDA_CHECK(launch_prestep(pa, compact_capture ? 3 : 2, stream));
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_PLAN], stream));
        // (the same fork in the phase-1 graph of an ensemble small enough for the two kernels to be latency-bound
        //  rather than HBM-bound: measured in DESIGN.md section 4)
        const bool fork = (compact_capture || (phase1_capture && B <= fork_max_batch)) && compact_fork && per_step_exc && run_rad;
        cudaStream_t es = fork ? fork_stream : stream;
        if (fork) {
            CUDA_CHECK(cudaEventRecord(ev_cfork, stream));
            CUDA_CHECK(cudaStreamWaitEvent(fork_stream, ev_cfork, 0));
        }
        if (per_step_exc) {
            ExcitationArgs ea{};
            ea.hdr = d_hdr.p; ea.eta = d_eta.p; ea.eta_t = d_eta_t.p; ea.partial = d_exc_partial.p;
            ea.eta_dt = eta_grid_dt; ea.n_eta = n_eta; ea.Bp = Bp; ea.chunk = exc_chunk; ea.ndmax = exc_ndmax;
            for (size_t g = 0; g < groups.size(); ++g) {
                Group& G = *groups[g];
                ExcGroup eg{G.tau.p, G.fw.p, G.Le, G.nd, G.dof0, G.chunk0, G.nchunk};
                CUDA_CHECK(launch_excitation(ea, eg, G.idx.p, G.w1.p, G.w2.p, es, plan_inline));
            }
        }
        if (fork) CUDA_CHECK(cudaEventRecord(ev_cjoin, fork_stream));
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_EXC], stream));
        if (run_rad) {
            const InlinePlan ipl{d_pr_wd.p, d_pr_head.p, d_pr_lead.p, B};
            CUDA_CHECK(launch_radiation(ra, d_pr_new.p, d_pr_old.p, d_pr_wn.p, d_pr_wo.p, d_pr_wd.p, stream,
                                        plan_inline ? &ipl : nullptr));
        }
        if (fork) CUDA_CHECK(cudaStreamWaitEvent(stream, ev_cjoin, 0));
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_RAD], stream));
        return;
    }
    if (!rb_use && !compact_capture) {
        CUDA_CHECK(launch_prestep(pa, 1, stream));
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_APPEND], stream));
    }

    FinalizeGroups fg{};
    if (wave_mode == 2)
        for (size_t g = 0; g < groups.size(); ++g) {
            Group& G = *groups[g];
            fg.dof0[g] = G.dof0; fg.nd[g] = G.nd; fg.chunk0[g] = G.chunk0; fg.nchunk[g] = G.nchunk;
        }
    FinalizeArgs fa{};
    fa.hdr = d_hdr.p; fa.rad_partial = d_rad_partial.p; fa.exc_partial = d_exc_partial.p;
    fa.comp = d_comp.p;
    fa.reg_amp = d_reg_amp.p; fa.reg_omega = d_reg_omega.p; fa.reg_mag = d_reg_mag.p; fa.reg_phase = d_reg_phase.p;
    fa.B = B; fa.Bp = Bp; fa.D = D; fa.N = N; fa.rad_nchunk = rad_nchunk; fa.wave_mode = wave_mode;
    fa.exc_ngroups = (wave_mode == 2) ? int(groups.size()) : 0; fa.exc_ndmax = exc_ndmax;
    fa.exc_cache = d_la_cache.p; fa.exc_S = la_S;
    fa.K = d_K.p; fa.pr_lead = d_pr_lead.p; fa.pr_wd = d_pr_wd.p; fa.pr_head = d_pr_head.p; fa.L = L;
    if (rb_use) {
        // served by the radiation look-ahead: append + block partials + young rows + finalize in one kernel that
        // takes the step header by value (launched directly, never part of a captured graph)
        RadStepArgs sa{};
        sa.hist = d_hist.p; sa.times = d_times.p; sa.K = d_Kyoung.p;
        sa.partial[0] = d_rb_partial[0].p; sa.partial[1] = d_rb_partial[1].p; sa.D = D;
        sa.B = B; sa.Bp = Bp; sa.nchunk = rb_nchunk; sa.L = rb_Lk; sa.m = rb_m;
        CUDA_CHECK(launch_step(sa, fa, hs, fg, hdr_h, stream));
        if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_APPEND], stream));
    } else {
        CUDA_CHECK(launch_finalize(fa, hs, fg, stream));
    }
    if (with_events) CUDA_CHECK(cudaEventRecord(ev[EV_END], stream));
}

void hc_ensemble::collect_events() {
    // called after a stream synchronisation
    float plan = 0, exc = 0, app = 0, rad = 0, fin = 0;
    cudaEventElapsedTime(&plan, ev[EV_BEGIN], ev[EV_PLAN]);
    cudaEventElapsedTime(&exc, ev[EV_PLAN], ev[EV_EXC]);
    cudaEventElapsedTime(&rad, ev[EV_EXC], ev[EV_RAD]);
    cudaEventElapsedTime(&app, ev[EV_RAD], ev[EV_APPEND]);
    cudaEventElapsedTime(&fin, ev[EV_APPEND], ev[EV_END]);
    if (la_events_pending) {
        float la = 0;
        cudaEventSynchronize(ev_la[1]);           // may have been recorded on the side stream
        cudaEventElapsedTime(&la, ev_la[0], ev_la[1]);
        exc += la;
        la_events_pending = false;
    }
    if (rb_events_pending) {
        float rbm = 0;
        cudaEventElapsedTime(&rbm, ev_rb[0], ev_rb[1]);
        rad += rbm;
        rb_ms_sum += rbm; rb_items_timed += rb_items_pending;
        rb_events_pending = false;
    }
    if (rb_use) { rad += app; app = 0; }      // k_rad_step: append + the block's per-step share
    acc_ms[0] += plan + app; acc_ms[1] += rad; acc_ms[2] += exc; acc_ms[3] += fin;
    ms_steps++;
    events_pending = false;
    prof.radiation_seconds += 1e-3 * (plan + app + rad);
    prof.waves_seconds += 1e-3 * exc;
    prof.hydrostatics_seconds += 1e-3 * fin;
    prof.step_seconds += 1e-3 * (plan + app + rad + exc + fin);
}

void hc_ensemble::launch_phase(int phase) {
    // phase 2 of a step served by the radiation look-ahead is the single kernel k_step: launched directly
    const bool want_graph = opts.use_graph && !profiling && !(phase == 2 && rb_use);
    if (!want_graph) {
        enqueue_phase(phase, profiling);
        if (phase == 2) events_pending = profiling;
        return;
    }
    cudaGraph_t& g = phase == 1 ? graph1 : graph;
    cudaGraphExec_t& ge = phase == 1 ? graph1_exec : graph_exec;
    const int key = (phase_uses_lookahead ? 1 : 0) | (rb_use ? 2 : 0) | (skip_radiation ? 4 : 0);
    // (the step's pose / velocity / force pointers travel in the header, so the graphs do not depend on them)
    const bool valid = (phase == 1 ? graph1_valid : graph_valid) && graph_key[phase] == key;
    if (!valid) {
        if (ge) cudaGraphExecDestroy(ge);
        if (g) cudaGraphDestroy(g);
        ge = nullptr; g = nullptr;
        ensure_fork_objects();
        CUDA_CHECK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        phase1_capture = (phase == 1);
        try {
            enqueue_phase(phase, false);
        } catch (...) {
            phase1_capture = false;
            cudaGraph_t tmp = nullptr;
            cudaStreamEndCapture(stream, &tmp);
            if (tmp) cudaGraphDestroy(tmp);
            throw;
        }
        phase1_capture = false;
        CUDA_CHECK(cudaStreamEndCapture(stream, &g));
        CUDA_CHECK(cudaGraphInstantiate(&ge, g, 0));
        graph_key[phase] = key;
        if (phase == 1) graph1_valid = true; else graph_valid = true;
    }
    CUDA_CHECK(cudaGraphLaunch(ge, stream));
}

// Host-side bookkeeping of one recompute (hydro_forces.cpp:746-760) + phase 1 launch.
void hc_ensemble::begin_step(double t, const double* g, const double* d_pose_in, const double* d_vel_in, double* d_force_out) {
    // --- ComputeForceRadiationDampingConv's host-side bookkeeping ---
    if (!times.empty() && t == times.front())
        fail(HC_ERR_DUPLICATE_TIME, "Tried to compute the radiation damping convolution twice within the same time step!");
    if (!times.empty() && t < times.front())
        fail(HC_ERR_TIME_ORDER, "Radiation convolution: interpolation error; query_time not bracketed by history.");
    std::string eta_error;
    if (wave_mode == 2) {
        // ExcitationConvolution bounds (wave_types.cpp:800,833-840): every t - tau_j must lie inside the eta window
        const double tmin = eta_t_h.front(), tmax = eta_t_h.back();
        for (auto& G : groups) {
            const double hi = t - G->tau_first, lo = t - G->tau_last;
            if (!(tmin <= lo && hi <= tmax)) {
                eta_error = "Excitation convolution: trying to find free surface elevation at a time out of bounds from the "
                            "precomputed free surface elevation (" + std::to_string(hi > tmax ? hi : lo) + "not in [" +
                            std::to_string(tmin) + ", " + std::to_string(tmax) + "]). Excitation force ignored at this time step.";
                break;
            }
        }
    }
    if (int(times.size()) >= cap) {
        if (rb_stream) CUDA_CHECK(cudaStreamSynchronize(rb_stream));
        grow_ring();
        rb_invalidate();
    }
    times.push_front(t);
    head = (head + 1) % cap;
    const double t_min = t - T->rirf_t.back();                        // history_min_time (:552)
    while (times.size() > 1 && times[times.size() - 2] < t_min) times.pop_back();   // PruneHistory (:327-340)

    if (events_pending) {   // the profiling events are about to be re-recorded
        CUDA_CHECK(cudaStreamSynchronize(stream));
        collect_events();
    }
    StepHeader& hh = hdr_h;
    hh = StepHeader{};
    hh.t = t; hh.g[0] = g[0]; hh.g[1] = g[1]; hh.g[2] = g[2];
    hh.snap = opts.bracket_snap; hh.head = head; hh.len = int(times.size()); hh.cap = cap; hh.flags = 0;
    hh.pose = d_pose_in; hh.vel = d_vel_in; hh.force = d_force.p;
    hh.force2 = (d_force_out != d_force.p) ? d_force_out : nullptr;   // the caller's buffer + the time-keyed cache
    phase_uses_lookahead = false;
    rb_use = false;
    if (!eta_error.empty()) {
        // The reference throws from ComputeForceWaves (wave_types.cpp:833-840) AFTER ComputeForceRadiationDampingConv
        // has pushed the step's sample and after prev_time was set (hydro_forces.cpp:747-756): the history keeps the
        // sample, the force cache of this time holds the zeros it was reset to, and the caller sees the exception.
        rb_invalidate();
        la_blk[0].valid = la_blk[1].valid = false; la_half_pending = -1;
        last_step_fast = false;
        if (inputs_on_copy_stream) CUDA_CHECK(cudaStreamWaitEvent(stream, ev_inputs, 0));
        if (defer_launch)       // compact host path: the state is still in the pinned staging block
            CUDA_CHECK(cudaMemcpyAsync(d_stage.p + 256, static_cast<unsigned char*>(h_stage.p) + 256, stage_bytes - 256,
                                       cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(d_hdr.p, &hh, sizeof(StepHeader), cudaMemcpyHostToDevice, stream));
        PrestepArgs pa{};
        pa.hdr = d_hdr.p; pa.hist = d_hist.p; pa.times = d_times.p; pa.B = B; pa.Bp = Bp; pa.D = D; pa.L = L;
        CUDA_CHECK(launch_prestep(pa, 1, stream));
        CUDA_CHECK(cudaMemsetAsync(d_force.p, 0, d_force.n * sizeof(double), stream));
        CUDA_CHECK(cudaMemsetAsync(d_comp.p, 0, d_comp.n * sizeof(double), stream));
        prof.kernel_launches += 1;
        prev_time = t;
        force_valid = true;
        fail(HC_ERR_ETA_WINDOW, eta_error);
    }
    if (wave_mode == 2 && la_enabled) {
        const int slot = lookahead_slot(t);
        if (slot >= 0) { hh.exc_src = 1; hh.exc_slot = slot; phase_uses_lookahead = true; }
    }
    if (rb_enabled && !skip_radiation) rb_use = radiation_block_slot(t, hh) >= 0;
    phase1_launches = 0;
    const bool per_step_exc = (wave_mode == 2) && !(la_enabled && phase_uses_lookahead);
    // k_step takes the header by value; every other kernel of a step reads it from d_hdr.  Pageable source: the runtime
    // stages small copies at call time, so hdr_h can be rewritten by the next step at once.
    hdr_on_device = !(rb_use && !per_step_exc) || profiling;
    last_step_fast = rb_use && !per_step_exc && !profiling;
    phase1_launches = last_step_fast ? 0 : (rb_use ? 0 : 1) + ((rb_use && !per_step_exc) ? 0 : 1) + (per_step_exc ? int(groups.size()) : 0);
    if (defer_launch && !rb_use) return;                        // compact host path: header + both phases go in one graph
    defer_launch = false;
    if (hdr_on_device) CUDA_CHECK(cudaMemcpyAsync(d_hdr.p, &hh, sizeof(StepHeader), cudaMemcpyHostToDevice, stream));
    if (last_step_fast) return;                                 // phase 1 is empty
    launch_phase(1);
}

// ---- excitation look-ahead ---------------------------------------------------------------------
void hc_ensemble::setup_lookahead() {
    la_enabled = false; la_pos = 0; la_cur = 0; la_builds = 0; la_hits_this_block = 0; la_poor_blocks = 0;
    la_blk[0].valid = la_blk[1].valid = false; la_half_pending = -1;
    if (la_stream) CUDA_CHECK(cudaStreamSynchronize(la_stream));
    if (wave_mode != 2 || n_eta == 0) return;
    const int want = opts.exc_lookahead;
    if (want == 1 || opts.dt_hint <= 0.0) return;
    for (auto& G : groups) if (G->nd != 6 && G->nd != 12) return;
    const int tiles = (Bp + 32 * kIPT - 1) / (32 * kIPT);
    if (want == 0 && tiles < sm_count) return;             // auto: only when one CTA per instance tile fills the GPU
    la_dt = opts.dt_hint;
    la_background = (want == 0 || want == 3 || want == 5);
    la_mma = (want == 0 || want == 4 || want == 5);
    for (auto& b : la_blk) b.times.assign(kLaT, 0.0);
    // DMMA kernel: (instance tiles x segments) should fill whole waves of 3 resident CTAs per SM, >= 8 stages each
    la_S = 1;
    if (la_mma) {
        const int mtiles = (Bp + 63) / 64, slots = sm_count * 3;
        int min_stages = 1 << 30;
        for (auto& G : groups) min_stages = std::min(min_stages, (G->Le + kLaT + 8) / kLaRows + 1);
        double best = 0.0;
        for (int S = 1; S <= 24 && min_stages / S >= 8; ++S) {
            const double w = double(mtiles) * S / slots, eff = w / std::ceil(w);
            if (eff > best + 0.02) { best = eff; la_S = S; }
        }
    }
    d_la_cache.alloc(size_t(2) * la_S * kLaT * D * Bp);
    d_la_times.alloc(2 * kLaT);
    if (!la_stream) {
        int lo = 0, hi = 0;
        CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));     // lo = least priority
        // below the per-step kernels; above the radiation pass when that pass is not held back by the steps (ungated
        // slices / whole pass), because the steps need the excitation block sooner (8 steps) than the radiation block
        const int rpm = opts.rad_pass_mode >= 1 && opts.rad_pass_mode <= 3 ? opts.rad_pass_mode : 1;
        CUDA_CHECK(cudaStreamCreateWithPriority(&la_stream, cudaStreamNonBlocking, rpm == 1 ? lo : (lo + hi) / 2));
        for (auto& x : ev_la_done) CUDA_CHECK(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
        for (auto& x : ev_la_free) CUDA_CHECK(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_la_build, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_la_join, cudaEventDisableTiming));
    }
    for (auto& G : groups) {
        G->la_idx.alloc(size_t(kLaT) * G->Le);
        G->la_w1.alloc(size_t(kLaT) * G->Le);
        G->la_w2.alloc(size_t(kLaT) * G->Le);
        G->la_rows_cap = ((G->Le + kLaT + 8 + kLaRows - 1) / kLaRows + 1) * kLaRows;
        G->la_taps.alloc(size_t(G->la_rows_cap) * kLaT * G->nd);
    }
    if (!ev_la[0]) { CUDA_CHECK(cudaEventCreate(&ev_la[0])); CUDA_CHECK(cudaEventCreate(&ev_la[1])); }
    la_enabled = true;
}

// Builds the block of wave forces for the predicted times t0, t0+dt, ... into cache buffer `buf` on stream `st`.
// Returns the number of valid block times (0: t0 is outside the eta window).  The per-group scratch (brackets,
// taps) is shared by all builds, which are therefore chained through ev_la_build.
// part = -1: the whole block; 0: plan + the first half of the eta-row segments; 1: the second half (same plan, same
// taps).  A background build is split like that, the halves launched 4 steps apart, so that the excitation work the
// steps give rise to is spread evenly over them (and a timing window of any multiple of 4 steps holds its exact share).
int hc_ensemble::enqueue_lookahead_block(int buf, double t0, cudaStream_t st, int part) {
    LaBlock& Bk = la_blk[buf];
    if (part == 1) {
        for (size_t gi = 0; gi < groups.size(); ++gi) {
            Group& G = *groups[gi];
            LookaheadArgs la{};
            la.eta = d_eta.p; la.taps = G.la_taps.p; la.cache = d_la_cache.p + size_t(buf) * la_S * kLaT * D * Bp;
            la.S = la_S; la.seg0 = la_S / 2; la.nseg = la_S - la_S / 2;
            la.n_eta = n_eta; la.Bp = Bp; la.D = D; la.dof0 = G.dof0; la.nd = G.nd; la.row0 = G.la_row0;
            la.nchunk = (G.la_nrows + kLaRows - 1) / kLaRows; la.use_mma = 1;
            CUDA_CHECK(launch_lookahead(la, st));
            prof.kernel_launches += 1;
        }
        CUDA_CHECK(cudaEventRecord(ev_la_build, st));
        return Bk.len;
    }
    Bk.valid = false; Bk.len = 0;
    const double tmin = eta_t_h.front(), tmax = eta_t_h.back();
    int T = 0;
    double tp = t0;                                          // repeated addition of dt, as Chrono advances ChTime
    for (int i = 0; i < kLaT; ++i) {
        bool ok = true;
        for (auto& G : groups) ok = ok && (tmin <= tp - G->tau_last) && (tp - G->tau_first <= tmax);
        if (!ok) break;
        Bk.times[i] = tp; ++T;
        tp = tp + la_dt;
    }
    if (T == 0) return 0;
    for (int i = T; i < kLaT; ++i) Bk.times[i] = Bk.times[T - 1];    // unused warps recompute the last time
    auto row_of = [&](double tt) {                            // largest i with eta_t[i] <= tt
        auto it = std::upper_bound(eta_t_h.begin(), eta_t_h.end(), tt);
        return int(it - eta_t_h.begin()) - 1;
    };
    // eta rows each group's taps cover; the capacity check for ALL groups comes before anything is enqueued
    int row0s[kMaxBodies], nrowss[kMaxBodies];
    for (size_t gi = 0; gi < groups.size(); ++gi) {
        Group& G = *groups[gi];
        int row0 = row_of(Bk.times[0] - G.tau_last) - 1;
        if (row0 < 0) row0 = 0;
        const int row_hi = std::min(n_eta - 1, row_of(Bk.times[T - 1] - G.tau_first) + 1);
        row0s[gi] = row0; nrowss[gi] = row_hi - row0 + 1;
        if (nrowss[gi] > G.la_rows_cap - kLaRows) return 0;
    }
    CUDA_CHECK(cudaStreamWaitEvent(st, ev_la_build, 0));
    double* d_times = d_la_times.p + size_t(buf) * kLaT;
    CUDA_CHECK(cudaMemcpyAsync(d_times, Bk.times.data(), kLaT * sizeof(double), cudaMemcpyHostToDevice, st));
    const bool timed = profiling;
    if (timed) CUDA_CHECK(cudaEventRecord(ev_la[0], st));
    for (size_t gi = 0; gi < groups.size(); ++gi) {
        Group& G = *groups[gi];
        const int row0 = row0s[gi], nrows = nrowss[gi];
        LookaheadPlanArgs pa{};
        pa.times = d_times; pa.tau = G.tau.p; pa.fw = G.fw.p; pa.eta_t = d_eta_t.p;
        pa.idx = G.la_idx.p; pa.w1 = G.la_w1.p; pa.w2 = G.la_w2.p; pa.taps = G.la_taps.p;
        pa.eta_dt = eta_grid_dt; pa.n_eta = n_eta; pa.Le = G.Le; pa.nd = G.nd; pa.T = kLaT;
        pa.row0 = row0; pa.nrows = nrows; pa.frag_order = la_mma ? 1 : 0;
        CUDA_CHECK(launch_lookahead_plan(pa, st));
        LookaheadArgs la{};
        la.eta = d_eta.p; la.taps = G.la_taps.p; la.cache = d_la_cache.p + size_t(buf) * la_S * kLaT * D * Bp;
        la.S = la_mma ? la_S : 1;
        la.seg0 = 0; la.nseg = (part == 0) ? la_S / 2 : la.S;
        la.n_eta = n_eta; la.Bp = Bp; la.D = D; la.dof0 = G.dof0; la.nd = G.nd; la.row0 = row0;
        la.nchunk = (nrows + kLaRows - 1) / kLaRows; la.use_mma = la_mma ? 1 : 0;
        G.la_row0 = row0; G.la_nrows = nrows;
        CUDA_CHECK(launch_lookahead(la, st));
        prof.kernel_launches += 3;
    }
    if (timed) { CUDA_CHECK(cudaEventRecord(ev_la[1], st)); la_events_pending = true; }
    CUDA_CHECK(cudaEventRecord(ev_la_build, st));
    Bk.len = T; Bk.valid = true;
    ++la_builds; ++la_blocks_built;
    return T;
}

// Background mode: the block after the current one is evaluated on a low-priority side stream while the main stream
// runs the steps of the current block (FP64-bound look-ahead kernel under the HBM-bound radiation kernel).
void hc_ensemble::prefetch_lookahead(int buf) {
    LaBlock& Cur = la_blk[la_cur];
    la_blk[buf].valid = false;
    // (profiling runs every kernel back-to-back in the main stream so that per-kernel event times are meaningful)
    if (!la_background || profiling || !Cur.valid || Cur.len < kLaT) return;   // short block: end of the eta window
    CUDA_CHECK(cudaStreamWaitEvent(la_stream, ev_la_free[buf], 0));
    const bool split = la_mma && la_S >= 2;
    if (enqueue_lookahead_block(buf, Cur.times[kLaT - 1] + la_dt, la_stream, split ? 0 : -1) > 0) {
        if (split) la_half_pending = buf;                 // second half: 4 steps from now (lookahead_slot)
        else CUDA_CHECK(cudaEventRecord(ev_la_done[buf], la_stream));
    }
}

// Second half of a split background build (no-op when none is pending).
void hc_ensemble::finish_split_build() {
    if (la_half_pending < 0) return;
    const int buf = la_half_pending;
    la_half_pending = -1;
    enqueue_lookahead_block(buf, 0.0, la_stream, 1);
    CUDA_CHECK(cudaEventRecord(ev_la_done[buf], la_stream));
}

// Cache slot holding the wave force for time t (bitwise match with a predicted time), building / switching blocks as
// needed; -1 when look-ahead cannot serve this step (the per-step kernels run instead).
int hc_ensemble::lookahead_slot(double t) {
    LaBlock& Cur = la_blk[la_cur];
    if (Cur.valid && la_pos < Cur.len && Cur.times[la_pos] == t) {
        if (la_pos >= kLaT / 2) finish_split_build();
        ++la_hits_this_block; ++la_steps_served;
        return la_cur * kLaT + la_pos++;
    }
    finish_split_build();             // a switch or a rebuild follows: the build in flight must be complete (its scratch
                                      // is reused by the next one, and the switch waits for its event)
    LaBlock& Nxt = la_blk[la_cur ^ 1];
    if (la_background && !profiling && Nxt.valid && Nxt.len > 0 && Nxt.times[0] == t) {
        const int old = la_cur;
        la_cur ^= 1; la_pos = 0; la_hits_this_block = 1; la_poor_blocks = 0;
        CUDA_CHECK(cudaStreamWaitEvent(stream, ev_la_done[la_cur], 0));
        CUDA_CHECK(cudaEventRecord(ev_la_free[old], stream));     // every reader of `old` is already enqueued
        prefetch_lookahead(old);
        ++la_steps_served;
        return la_cur * kLaT + la_pos++;
    }
    // miss: first step, end of a block without prefetch, or a time the prediction did not foresee
    if (la_builds > 0 && la_hits_this_block < 2) {                // a block that served < 2 steps was wasted work
        if (++la_poor_blocks >= 3) { la_enabled = false; la_blk[0].valid = la_blk[1].valid = false; la_half_pending = -1; drop_graph(); return -1; }
    } else {
        la_poor_blocks = 0;
    }
    la_pos = 0; la_hits_this_block = 0;
    if (enqueue_lookahead_block(la_cur, t, stream) == 0) return -1;
    if (la_background) {
        CUDA_CHECK(cudaEventRecord(ev_la_free[la_cur ^ 1], stream));
        prefetch_lookahead(la_cur ^ 1);
    }
    ++la_hits_this_block; ++la_steps_served;
    return la_cur * kLaT + la_pos++;
}

// Compact host path: the staged inputs (header, velocities, pose: one pinned block) go up in ONE copy, every kernel of
// the step runs, the forces come back into the pinned force buffer -- all nodes of one captured graph.
void hc_ensemble::ensure_fork_objects() {
    if (fork_stream) return;
    CUDA_CHECK(cudaStreamCreateWithFlags(&fork_stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_cfork, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_cjoin, cudaEventDisableTiming));
}

void hc_ensemble::run_compact() {
    const int key = (phase_uses_lookahead ? 1 : 0) | (skip_radiation ? 4 : 0);
    if (!graph_c_exec || graph_c_key != key) {
        if (graph_c_exec) cudaGraphExecDestroy(graph_c_exec);
        if (graph_c) cudaGraphDestroy(graph_c);
        graph_c_exec = nullptr; graph_c = nullptr;
        ensure_fork_objects();
        CUDA_CHECK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        compact_capture = true;
        try {
            CUDA_CHECK(cudaMemcpyAsync(d_stage.p, h_stage.p, stage_bytes, cudaMemcpyHostToDevice, stream));
            enqueue_phase(1, false);
            enqueue_phase(2, false);
            // (no D2H node when the finalize kernel stores its second copy of the totals straight into the pinned buffer)
            if (!h_force_dev)
                CUDA_CHECK(cudaMemcpyAsync(h_force.p, d_force.p, size_t(B) * D * sizeof(double), cudaMemcpyDeviceToHost, stream));
        } catch (...) {
            compact_capture = false;
            cudaGraph_t tmp = nullptr;
            cudaStreamEndCapture(stream, &tmp);
            if (tmp) cudaGraphDestroy(tmp);
            throw;
        }
        compact_capture = false;
        CUDA_CHECK(cudaStreamEndCapture(stream, &graph_c));
        CUDA_CHECK(cudaGraphInstantiate(&graph_c_exec, graph_c, 0));
        graph_c_key = key;
    }
    CUDA_CHECK(cudaGraphLaunch(graph_c_exec, stream));
}

void hc_ensemble::finish_step(double t) {
    launch_phase(2);
    if (rb_use && rb_pass_mode != 3) rb_launch_slices(1, true);    // this step's share of the next block's pass
    prof.kernel_launches += phase1_launches + (rb_use ? 1 : 2);
    prof.hydrostatics_calls++; prof.radiation_calls++; prof.waves_calls++;
    prev_time = t;
    force_valid = true;
}

// =====================================================================================
// C ABI
// =====================================================================================
#define HC_GUARD_BEGIN try {
#define HC_GUARD_END                                                                                 \
    }                                                                                                \
    catch (const hc::StatusError& e) { hc::set_last_error(e.msg); return e.code; }                   \
    catch (const std::out_of_range& e) { hc::set_last_error(e.what()); return HC_ERR_OUT_OF_RANGE; } \
    catch (const std::exception& e) { hc::set_last_error(e.what()); return HC_ERR_INVALID; }

extern "C" {

int hc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void hc_ensemble_default_opts(hc_ensemble_opts* o) {
    std::memset(o, 0, sizeof(*o));
    o->device = 0; o->batch = 1; o->dt_hint = 0.0; o->bracket_snap = 0.0;
    o->rad_chunk = 0; o->exc_chunk = 0; o->use_graph = 1; o->exc_lookahead = 0; o->rad_kernel = 0; o->rad_lookahead = 0;
    o->rad_pass_mode = 0;
    o->stream = nullptr;
}

hc_status hc_ensemble_create(const hc_tables* t, const hc_ensemble_opts* opts, hc_ensemble** out) {
    HC_GUARD_BEGIN
    if (!t || !opts || !out) fail(HC_ERR_INVALID, "null argument");
    if (opts->batch < 1) fail(HC_ERR_INVALID, "batch must be >= 1");
    if (t->N > kMaxBodies) fail(HC_ERR_INVALID, "too many bodies (max " + std::to_string(kMaxBodies) + ")");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        fail(HC_ERR_CUDA, "no CUDA device available: hydrochrono_b200 has no CPU fallback");
    }
    if (opts->device < 0 || opts->device >= ndev) fail(HC_ERR_INVALID, "bad device ordinal");
    std::unique_ptr<hc_ensemble> e(new hc_ensemble());
    e->T = t; e->opts = *opts; e->dev = opts->device;
    e->use_device();
    e->B = opts->batch; e->N = t->N; e->D = t->D; e->L = t->L;
    CUDA_CHECK(cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, e->dev));
    const int lane_tile = 32 * kIPT;
    e->Bp = ((e->B + lane_tile - 1) / lane_tile) * lane_tile;
    if (opts->stream) { e->stream = static_cast<cudaStream_t>(opts->stream); }
    else {
        int lo = 0, hi = 0;                      // per-step kernels outrank the look-ahead passes on the side streams
        CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, hi));
        e->own_stream = true;
    }
    for (auto& ev : e->ev) CUDA_CHECK(cudaEventCreate(&ev));
    if (const char* tr = std::getenv("HC_TRACE")) e->trace = std::atoi(tr) != 0;
    if (e->trace) for (auto& ev : e->ev_tr) CUDA_CHECK(cudaEventCreate(&ev));
    CUDA_CHECK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_inputs, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_force, cudaEventDisableTiming));

    const int D = e->D, L = e->L;
    // measured on B200 (profiles/README.md): the DMMA kernel runs below the power cap but pads 12 rows to 16 and ends
    // up slower (0.319 ms vs 0.274 ms), so auto selects the FMA-pipe kernel
    e->rad_mma = (D == 12) && (opts->rad_kernel == 2);
    e->rad_hybrid = (D == 12) && (opts->rad_kernel == 3);
    e->setup_radiation_block();
    e->stage_kernel();
    e->d_rirf_t.upload(t->rirf_t);
    e->d_rirf_w.upload(t->rirf_w);
    std::vector<double> A(size_t(D) * D);
    for (int b = 0; b < t->N; ++b)
        for (int r = 0; r < 6; ++r)
            for (int c = 0; c < D; ++c) A[size_t(6 * b + r) * D + c] = t->body[b].ainf[size_t(r) * D + c];
    e->d_ainf.upload(A);
    e->hs.rho = t->rho;
    for (int b = 0; b < t->N; ++b) {
        std::copy(t->body[b].lin.begin(), t->body[b].lin.end(), e->hs.Kh[b]);
        e->hs.disp_vol[b] = t->body[b].disp_vol;
        for (int i = 0; i < 3; ++i) e->hs.cb_minus_cg[b][i] = t->cb_minus_cg[3 * b + i];
        for (int i = 0; i < 6; ++i) e->hs.equilibrium[b][i] = t->equilibrium[6 * b + i];
    }
    // history ring: window / dt + slack
    const double window = t->rirf_t.back() - t->rirf_t.front();
    double dt = opts->dt_hint > 0.0 ? opts->dt_hint : (t->rirf_t[1] - t->rirf_t[0]);
    int cap = int(std::ceil(window / dt)) + 8;
    if (e->rb_enabled && e->rb_ahead) cap += kRbT * e->rb_m + 8;   // a pass spread over a block's steps must not be lapped
    cap = std::max(cap, 16);
    e->alloc_ring(cap);
    e->d_pr_new.alloc(L); e->d_pr_old.alloc(L); e->d_pr_wn.alloc(L); e->d_pr_wo.alloc(L); e->d_pr_wd.alloc(L);
    e->d_pr_head.alloc(L); e->d_pr_lead.alloc(L);
    e->setup_radiation_chunks();
    const size_t bd = size_t(e->B) * D;
    e->stage_bytes = 256 + 2 * bd * sizeof(double);
    e->d_stage.alloc(e->stage_bytes);
    e->d_hdr.p = reinterpret_cast<StepHeader*>(e->d_stage.p);
    e->d_vel.p = reinterpret_cast<double*>(e->d_stage.p + 256);
    e->d_pose.p = e->d_vel.p + bd;
    static_assert(sizeof(StepHeader) <= 256, "step header must fit its slot of the staging block");
    size_t compact_max = 64 * 1024;
    if (const char* v = std::getenv("HC_COMPACT_MAX_BYTES")) compact_max = size_t(std::atoll(v));   // diagnostic override
    e->compact_ok = e->stage_bytes <= compact_max && opts->use_graph;
    if (e->compact_ok) e->h_stage.alloc(e->stage_bytes);
    e->d_force.alloc(bd); e->d_comp.alloc(3 * bd);
    e->h_pose.alloc(bd * sizeof(double)); e->h_vel.alloc(bd * sizeof(double)); e->h_force.alloc(bd * sizeof(double));
    {
        const char* vf = std::getenv("HC_COMPACT_FORK");
        if (vf && std::atoi(vf) == 0) e->compact_fork = false;
        const char* vi = std::getenv("HC_COMPACT_INLINE");
        if (vi && std::atoi(vi) == 0) e->compact_inline = false;
        const char* vm = std::getenv("HC_FORK_MAX_BATCH");         // diagnostic override
        if (vm) e->fork_max_batch = std::atoi(vm);
    }
    if (e->compact_ok) {
        const char* v = std::getenv("HC_COMPACT_DIRECT");            // diagnostic: 0 = forces come back through a copy node
        if (!(v && std::atoi(v) == 0)) {
            void* dp = nullptr;
            if (cudaHostGetDevicePointer(&dp, e->h_force.p, 0) == cudaSuccess) e->h_force_dev = static_cast<double*>(dp);
            else cudaGetLastError();
        }
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    *out = e.release();
    return HC_OK;
    HC_GUARD_END
}

void hc_ensemble_destroy(hc_ensemble* e) { delete e; }
int hc_ensemble_batch(const hc_ensemble* e) { return e->B; }
int hc_ensemble_dofs(const hc_ensemble* e) { return e->D; }
int hc_ensemble_history_len(const hc_ensemble* e) { return int(e->times.size()); }

hc_status hc_ensemble_reset(hc_ensemble* e) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->times.clear();
    e->head = -1;
    if (e->la_stream) CUDA_CHECK(cudaStreamSynchronize(e->la_stream));
    e->la_blk[0].valid = e->la_blk[1].valid = false; e->la_pos = 0; e->la_half_pending = -1;
    if (e->rb_stream) CUDA_CHECK(cudaStreamSynchronize(e->rb_stream));
    e->rb_invalidate(); e->rb_hits_this_block = 0; e->rb_builds = 0; e->rb_poor_blocks = 0;
    // a new run: look-aheads that the misprediction heuristics switched off are armed again
    if (e->d_Kpad.p && e->rb_plan.usable) e->rb_enabled = true;
    e->rb_side_pending = false;
    if (e->wave_mode == 2 && e->d_la_cache.p && !e->la_enabled) { e->la_enabled = true; e->drop_graph(); }
    e->la_cur = 0; e->la_builds = 0; e->la_hits_this_block = 0; e->la_poor_blocks = 0;
    e->last_step_fast = false;
    e->prev_time = -1.0;
    e->force_valid = false;
    // a new run builds its orientations from the given angles, as a fresh ensemble does: no quaternion is kept
    e->sim_q_valid = false;
    e->link_asm_valid = false;                    // ... and every joint / spring-damper is assembled again
    CUDA_CHECK(cudaMemsetAsync(e->d_force.p, 0, e->d_force.n * sizeof(double), e->stream));
    CUDA_CHECK(cudaMemsetAsync(e->d_comp.p, 0, e->d_comp.n * sizeof(double), e->stream));
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_ensemble_set_bracket_snap(hc_ensemble* e, double snap) {
    if (!(snap >= 0.0) || snap >= 0.5) { set_last_error("bracket_snap must be in [0, 0.5)"); return HC_ERR_INVALID; }
    e->opts.bracket_snap = snap;     // travels in the per-step header: takes effect at the next step
    e->rb_invalidate();
    if (e->d_Kpad.p) { e->rb_enabled = true; e->rb_builds = 0; e->rb_hits_this_block = 0; e->rb_poor_blocks = 0; }
    return HC_OK;
}

hc_status hc_ensemble_host_buffers(hc_ensemble* e, double** pose, double** vel, double** force) {
    if (pose) *pose = static_cast<double*>(e->h_pose.p);
    if (vel) *vel = static_cast<double*>(e->h_vel.p);
    if (force) *force = static_cast<double*>(e->h_force.p);
    return HC_OK;
}

// ---- waves ---------------------------------------------------------------------------
hc_status hc_waves_none(hc_ensemble* e) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->wave_mode = 0;
    e->release_kinematics();
    e->drop_graph();
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_regular(hc_ensemble* e, int count, const double* amplitude, const double* omega, const double* phase) {
    HC_GUARD_BEGIN
    const hc_tables& T = *e->T;
    if (!(count == 1 || count == e->B)) fail(HC_ERR_INVALID, "count must be 1 or the batch size");
    if (!amplitude || !omega) fail(HC_ERR_INVALID, "null argument");
    if (T.nw < 2) fail(HC_ERR_INVALID, "tables hold no excitation magnitude/phase data");
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    const int D = e->D, Bp = e->Bp;
    // RegularWave::AddH5Data (wave_types.cpp:278-299) per distinct wave
    e->reg_count = count;
    e->reg_mag_h.assign(size_t(count) * D, 0.0);
    e->reg_phase_h.assign(size_t(count) * D, 0.0);
    e->reg_k_h.assign(count, 0.0);
    const double omega_max = T.w_list.back();
    const double num_freqs = double(T.w_list.size());
    const double domega = omega_max / num_freqs;                       // GetOmegaDelta (:329-333)
    for (int i = 0; i < count; ++i) {
        const double pos = (omega[i] / domega) - 1;                    // freq_index_des (:290)
        const double fl = std::floor(pos);
        const int i0 = int(fl);
        if (i0 < 0 || i0 + 1 >= T.nw)
            throw std::out_of_range("regular wave omega outside the excitation frequency table");
        const double frac = pos - fl;
        for (int b = 0; b < T.N; ++b)
            for (int r = 0; r < 6; ++r) {
                const double* m = &T.body[b].exc_mag[size_t(r) * T.nw];
                const double* p = &T.body[b].exc_phase[size_t(r) * T.nw];
                e->reg_mag_h[size_t(i) * D + 6 * b + r] = (frac * (m[i0 + 1] - m[i0])) + m[i0];
                e->reg_phase_h[size_t(i) * D + 6 * b + r] = (frac * (p[i0 + 1] - p[i0])) + p[i0];
            }
        e->reg_k_h[i] = wave_number(omega[i], T.depth, T.g);           // RegularWave::Initialize (:274-276)
    }
    std::vector<double> amp(Bp, 0.0), om(Bp, 0.0), mag(size_t(D) * Bp, 0.0), ph(size_t(6) * Bp, 0.0);
    for (int b = 0; b < e->B; ++b) {
        const int i = count == 1 ? 0 : b;
        amp[b] = amplitude[i]; om[b] = omega[i];
        for (int d = 0; d < D; ++d) mag[size_t(d) * Bp + b] = e->reg_mag_h[size_t(i) * D + d];
        for (int r = 0; r < 6; ++r) ph[size_t(r) * Bp + b] = e->reg_phase_h[size_t(i) * D + r];   // body 0 (quirk, :323)
    }
    // regular_wave_phase_ is not used by the force, only by eta / kinematics
    e->reg_amp_h.assign(amplitude, amplitude + count);
    e->reg_omega_h.assign(omega, omega + count);
    if (phase) e->reg_wave_phase_h.assign(phase, phase + count); else e->reg_wave_phase_h.assign(count, 0.0);
    e->release_kinematics();
    e->d_reg_amp.upload(amp); e->d_reg_omega.upload(om); e->d_reg_mag.upload(mag); e->d_reg_phase.upload(ph);
    e->wave_mode = 1;
    e->drop_graph();
    return HC_OK;
    HC_GUARD_END
}

void hc_irregular_default_params(hc_irregular_params* p) {
    std::memset(p, 0, sizeof(*p));
    p->frequency_min = 0.001; p->frequency_max = 1.0; p->nfrequencies = 0;
    p->peak_enhancement_factor = 1.0; p->is_normalized = 0; p->seed = 1;
}

// InitializeIRFVectors / ResampleIRF (wave_types.cpp:432-449,572-606) + the excitation groups' device tables; leaves the
// ensemble in irregular-wave mode with an empty eta.
void hc_ensemble::setup_excitation_groups(double simulation_dt) {
    hc_ensemble* e = this;
    const hc_tables& T = *e->T;
    release_kinematics();
    irf = resample_excitation_irf(T, simulation_dt);
    // group bodies that share one IRF time grid bit-for-bit (the usual case: one BEMIO run)
    groups.clear();
    bool all_same = true;
    for (int b = 1; b < T.N; ++b)
        if (e->irf[b].t != e->irf[0].t) all_same = false;
    const bool merged = all_same && (D == 6 || D == 12);
    const int ngroups = merged ? 1 : T.N;
    if (ngroups > kMaxBodies) fail(HC_ERR_INVALID, "too many excitation groups");
    e->exc_ndmax = merged ? D : 6;
    int max_Le = 0;
    for (int g = 0; g < ngroups; ++g) max_Le = std::max(max_Le, int(e->irf[g].t.size()));
    {
        const int tiles = (Bp + kTileInst - 1) / kTileInst;
        int chunk = e->opts.exc_chunk;
        if (chunk <= 0)
            chunk = pick_chunk(max_Le, tiles * ngroups, e->sm_count, 2, size_t(110) * 1024, excitation_smem_bytes,
                               e->exc_ndmax, 16);
        chunk = std::min(chunk, std::max(1, max_Le));
        // a user exc_chunk must still fit k_excitation's dynamic shared memory (200 KB attribute), as the radiation
        // chunk does
        while (chunk > 1 && excitation_smem_bytes(e->exc_ndmax, chunk) > 200 * 1024) chunk /= 2;
        e->exc_chunk = chunk;
    }
    int chunk0 = 0;
    for (int g = 0; g < ngroups; ++g) {
        auto G = std::make_unique<hc_ensemble::Group>();
        const ExcIrfBody& I0 = e->irf[g];
        G->Le = int(I0.t.size());
        G->dof0 = merged ? 0 : 6 * g;
        G->nd = merged ? D : 6;
        G->tau_first = I0.t.front(); G->tau_last = I0.t.back();
        std::vector<double> fw(size_t(G->Le) * G->nd);
        for (int d = 0; d < G->nd; ++d) {
            const int body = (G->dof0 + d) / 6, r = (G->dof0 + d) % 6;
            const ExcIrfBody& I = e->irf[body];
            for (int j = 0; j < G->Le; ++j) fw[size_t(j) * G->nd + d] = I.f[size_t(r) * G->Le + j] * I.w[j];
        }
        G->tau.upload(I0.t); G->fw.upload(fw);
        G->idx.alloc(G->Le); G->w1.alloc(G->Le); G->w2.alloc(G->Le);
        G->chunk0 = chunk0;
        G->nchunk = (G->Le + e->exc_chunk - 1) / e->exc_chunk;
        chunk0 += G->nchunk;
        e->groups.push_back(std::move(G));
    }
    e->exc_total_chunks = chunk0;
    e->d_exc_partial.alloc(size_t(chunk0) * e->exc_ndmax * Bp);

    e->n_eta = 0; e->nf = 0;
    e->wave_mode = 2;
    e->la_enabled = false; e->la_blk[0].valid = e->la_blk[1].valid = false; e->la_half_pending = -1;
    if (e->la_stream) CUDA_CHECK(cudaStreamSynchronize(e->la_stream));
    e->drop_graph();
}

// Device layout of the irregular components (k_eta, k_wave_kinematics): phases [nf][Bp], amplitudes sqrt(2 S df)
// [nf][Bp] when the spectrum is per instance, else [nf]; padded lanes zero.
void hc_ensemble::pack_irregular(std::vector<double>& amp, std::vector<double>& ph) const {
    amp.assign(per_instance_spectrum ? size_t(nf) * Bp : size_t(nf), 0.0);
    ph.assign(size_t(nf) * Bp, 0.0);
    const int nS = per_instance_spectrum ? B : 1;
    for (int s = 0; s < nS; ++s)
        for (int i = 0; i < nf; ++i) {
            const double a = std::sqrt(2 * S_h[size_t(s) * nf + i] * widths_h[i]);     // GetEtaIrregular (:39)
            if (per_instance_spectrum) amp[size_t(i) * Bp + s] = a; else amp[i] = a;
        }
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < nf; ++i) ph[size_t(i) * Bp + b] = phases_h[size_t(b) * nf + i];
}

hc_status hc_waves_irregular(hc_ensemble* e, const hc_irregular_params* p, const int* seeds, const double* Hs_arr,
                             const double* Tp_arr) {
    HC_GUARD_BEGIN
    if (!p) fail(HC_ERR_INVALID, "null argument");
    const hc_tables& T = *e->T;
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (p->simulation_dt <= 0.0) fail(HC_ERR_INVALID, "simulation_dt must be positive for irregular waves");
    const int B = e->B, Bp = e->Bp;
    e->ip = *p;
    e->eta_grid_dt = p->simulation_dt;
    e->setup_excitation_groups(p->simulation_dt);
    const bool have_sea = (Hs_arr || p->wave_height != 0.0) && (Tp_arr || p->wave_period != 0.0);
    // --- eta time grid (CreateFreeSurfaceElevation, wave_types.cpp:717-744) ---
    double t_irf_min = 0.0, t_irf_max = 0.0;
    for (const ExcIrfBody& I : e->irf) {
        t_irf_min = std::min({t_irf_min, I.t.front(), I.t.back()});
        t_irf_max = std::max({t_irf_max, I.t.front(), I.t.back()});
    }
    const double duration = p->simulation_duration + 2 * (t_irf_max - t_irf_min);
    const int num_timesteps = static_cast<int>(std::ceil(duration / p->simulation_dt));
    e->eta_t_h = linspaced(num_timesteps + 1, 0, num_timesteps * p->simulation_dt);
    for (double& x : e->eta_t_h) x += -t_irf_max;
    e->n_eta = int(e->eta_t_h.size());
    e->d_eta_t.upload(e->eta_t_h);
    e->d_eta.alloc(size_t(e->n_eta) * Bp);   // zero: wave_height == 0 leaves eta empty in the reference
    if (!have_sea) return HC_OK;             // wave_types.cpp:454 (no spectrum, no elevation)

    // --- CreateSpectrum (wave_types.cpp:643-676) ---
    int nf;
    if (p->nfrequencies == 0) {
        const double df = 1.0 / p->simulation_duration;
        nf = std::ceil((p->frequency_max - p->frequency_min) / df);
    } else {
        nf = p->nfrequencies;
    }
    if (nf < 1) fail(HC_ERR_INVALID, "no spectrum frequencies");
    e->nf = nf;
    e->freqs_h = linspaced(nf, p->frequency_min, p->frequency_max);
    e->widths_h = trapezoid_widths(e->freqs_h);
    e->wavenumbers_h.resize(nf);
    std::vector<double> omega(nf);
    for (int i = 0; i < nf; ++i) {
        omega[i] = 2 * M_PI * e->freqs_h[i];
        e->wavenumbers_h[i] = wave_number(omega[i], T.depth, T.g);
    }
    e->per_instance_spectrum = (Hs_arr != nullptr) || (Tp_arr != nullptr);
    const int nS = e->per_instance_spectrum ? B : 1;
    e->S_h.resize(size_t(nS) * nf);
    for (int s = 0; s < nS; ++s) {
        const double Hs = Hs_arr ? Hs_arr[s] : p->wave_height;
        const double Tp = Tp_arr ? Tp_arr[s] : p->wave_period;
        dvec S = jonswap(e->freqs_h, Hs, Tp, p->peak_enhancement_factor, p->is_normalized != 0);
        std::copy(S.begin(), S.end(), e->S_h.begin() + size_t(s) * nf);
    }
    e->phases_h.resize(size_t(B) * nf);
    for (int b = 0; b < B; ++b) {
        dvec v = random_phases(seeds ? seeds[b] : p->seed, nf);
        std::copy(v.begin(), v.end(), e->phases_h.begin() + size_t(b) * nf);
    }
    {
        std::vector<double> amp, ph;
        e->pack_irregular(amp, ph);
        e->d_omega.upload(omega); e->d_amp.upload(amp); e->d_phase.upload(ph);
    }

    // --- eta synthesis on the device (wave_types.cpp:27-59,750-769) ---
    EtaArgs ea{};
    ea.eta_t = e->d_eta_t.p; ea.omega = e->d_omega.p; ea.amp = e->d_amp.p; ea.phase = e->d_phase.p; ea.eta = e->d_eta.p;
    ea.ramp = p->ramp_duration; ea.n_eta = e->n_eta; ea.nf = nf; ea.Bp = Bp; ea.amp_per_instance = e->per_instance_spectrum;
    CUDA_CHECK(cudaEventRecord(e->ev[EV_BEGIN], e->stream));
    CUDA_CHECK(launch_eta(ea, e->stream));
    CUDA_CHECK(cudaEventRecord(e->ev[EV_END], e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev[EV_BEGIN], e->ev[EV_END]);
    e->prof.eta_synthesis_seconds += 1e-3 * ms;
    e->prof.kernel_launches += 1;
    e->setup_lookahead();
    // phases/amplitudes are only needed for the synthesis; keep omega/amp small arrays, free the big ones
    e->d_phase.release();
    if (e->per_instance_spectrum) e->d_amp.release();
    return HC_OK;
    HC_GUARD_END
}

// SURVEY a16: the free-surface elevation imported as a (time, eta) series instead of synthesised from a spectrum
// (IrregularWaves::ReadEtaFromFile, src/wave_types.cpp:480-500, from InitializeIRFVectors :451-453).  The reference
// snapshot never fills free_surface_time_sampled_ on this branch although ExcitationConvolution reads it (:784-785);
// the grid used here is the intended one, the series' own time column.
hc_status hc_waves_irregular_series(hc_ensemble* e, double simulation_dt, int n, const double* time, const double* eta,
                                    int per_instance) {
    HC_GUARD_BEGIN
    if (!time || !eta) fail(HC_ERR_INVALID, "null argument");
    if (simulation_dt <= 0.0) fail(HC_ERR_INVALID, "simulation_dt must be positive for irregular waves");
    if (n < 2) fail(HC_ERR_INVALID, "an eta series needs at least two samples");
    for (int k = 1; k < n; ++k)
        if (!(time[k] > time[k - 1])) fail(HC_ERR_INVALID, "eta series: time must be strictly increasing (line " + std::to_string(k + 1) + ")");
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    const int B = e->B, Bp = e->Bp;
    hc_irregular_default_params(&e->ip);
    e->ip.simulation_dt = simulation_dt;
    e->ip.simulation_duration = time[n - 1] - time[0];
    e->ip.wave_height = 0.0; e->ip.wave_period = 0.0;
    e->setup_excitation_groups(simulation_dt);
    e->eta_t_h.assign(time, time + n);
    e->eta_grid_dt = (time[n - 1] - time[0]) / double(n - 1);
    e->n_eta = n;
    e->d_eta_t.upload(e->eta_t_h);
    e->d_eta.alloc(size_t(n) * Bp);                            // zero-filled; padded lanes stay zero
    // eta[sample][instance] on the device: transposed through a bounded pinned staging block
    const int rows = std::max(1, std::min(n, int((size_t(8) << 20) / (size_t(Bp) * sizeof(double)))));
    PinBuf stage;
    stage.alloc(size_t(rows) * Bp * sizeof(double));
    double* hs = static_cast<double*>(stage.p);
    for (int k0 = 0; k0 < n; k0 += rows) {
        const int nk = std::min(rows, n - k0);
        for (int k = 0; k < nk; ++k) {
            double* row = hs + size_t(k) * Bp;
            if (per_instance) for (int b = 0; b < B; ++b) row[b] = eta[size_t(b) * n + k0 + k];
            else for (int b = 0; b < B; ++b) row[b] = eta[k0 + k];
        }
        CUDA_CHECK(cudaMemcpyAsync(e->d_eta.p + size_t(k0) * Bp, hs, size_t(nk) * Bp * sizeof(double), cudaMemcpyHostToDevice,
                                   e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
    }
    e->per_instance_spectrum = false;
    e->freqs_h.clear(); e->widths_h.clear(); e->wavenumbers_h.clear(); e->S_h.clear(); e->phases_h.clear();
    e->setup_lookahead();
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_irregular_sizes(const hc_ensemble* e, int* nfreq, int* n_eta, int* exc_steps) {
    if (e->wave_mode != 2) { set_last_error("ensemble has no irregular waves"); return HC_ERR_INVALID; }
    if (nfreq) *nfreq = e->nf;
    if (n_eta) *n_eta = e->n_eta;
    if (exc_steps) for (int b = 0; b < e->N; ++b) exc_steps[b] = int(e->irf[b].t.size());
    return HC_OK;
}

hc_status hc_waves_irregular_spectrum(const hc_ensemble* e, int inst, double* freqs, double* S, double* widths,
                                      double* phases, double* wavenumbers) {
    HC_GUARD_BEGIN
    if (e->wave_mode != 2 || e->nf == 0)   // IrregularWaves::GetSpectrum (wave_types.cpp:461-467)
        fail(HC_ERR_INVALID, "Spectrum has not been created. Initialize with wave height and period to create spectrum.");
    if (inst < 0 || inst >= e->B) throw std::out_of_range("instance index out of range");
    const int nf = e->nf;
    if (freqs) std::copy(e->freqs_h.begin(), e->freqs_h.end(), freqs);
    if (widths) std::copy(e->widths_h.begin(), e->widths_h.end(), widths);
    if (wavenumbers) std::copy(e->wavenumbers_h.begin(), e->wavenumbers_h.end(), wavenumbers);
    if (S) {
        const size_t s = e->per_instance_spectrum ? inst : 0;
        std::copy(e->S_h.begin() + s * nf, e->S_h.begin() + (s + 1) * nf, S);
    }
    if (phases) std::copy(e->phases_h.begin() + size_t(inst) * nf, e->phases_h.begin() + size_t(inst + 1) * nf, phases);
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_irregular_eta(const hc_ensemble* e, int inst, double* eta_t, double* eta) {
    HC_GUARD_BEGIN
    if (e->wave_mode != 2) fail(HC_ERR_INVALID, "ensemble has no irregular waves");
    if (inst < 0 || inst >= e->B) throw std::out_of_range("instance index out of range");
    e->use_device();
    if (eta_t) std::copy(e->eta_t_h.begin(), e->eta_t_h.end(), eta_t);
    if (eta) {
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        CUDA_CHECK(cudaMemcpy2D(eta, sizeof(double), e->d_eta.p + inst, size_t(e->Bp) * sizeof(double), sizeof(double),
                                e->n_eta, cudaMemcpyDeviceToHost));
    }
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_irregular_irf(const hc_ensemble* e, int body, double* t, double* width, double* f) {
    HC_GUARD_BEGIN
    if (e->wave_mode != 2) fail(HC_ERR_INVALID, "ensemble has no irregular waves");
    if (body < 0 || body >= e->N) throw std::out_of_range("body index out of range");
    const ExcIrfBody& I = e->irf[body];
    if (t) std::copy(I.t.begin(), I.t.end(), t);
    if (width) std::copy(I.w.begin(), I.w.end(), width);
    if (f) std::copy(I.f.begin(), I.f.end(), f);
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_regular_coeffs(const hc_ensemble* e, int inst, double* mag, double* phase, double* wavenumber) {
    HC_GUARD_BEGIN
    if (e->wave_mode != 1) fail(HC_ERR_INVALID, "ensemble has no regular waves");
    if (inst < 0 || inst >= e->B) throw std::out_of_range("instance index out of range");
    const int i = e->reg_count == 1 ? 0 : inst;
    if (mag) std::copy(e->reg_mag_h.begin() + size_t(i) * e->D, e->reg_mag_h.begin() + size_t(i + 1) * e->D, mag);
    if (phase) std::copy(e->reg_phase_h.begin() + size_t(i) * e->D, e->reg_phase_h.begin() + size_t(i + 1) * e->D, phase);
    if (wavenumber) *wavenumber = e->reg_k_h[i];
    return HC_OK;
    HC_GUARD_END
}

// ---- step ----------------------------------------------------------------------------
hc_status hc_step_device(hc_ensemble* e, double t, const double* d_pose, const double* d_vel, const double g[3],
                         double* d_force, int* recomputed) {
    HC_GUARD_BEGIN
    if (!d_pose || !d_vel || !g || !d_force) fail(HC_ERR_INVALID, "null argument");
    e->use_device();
    const size_t bytes = size_t(e->B) * e->D * sizeof(double);
    if (t == e->prev_time) {                                           // time-keyed cache (hydro_forces.cpp:742-744)
        if (d_force != e->d_force.p)
            CUDA_CHECK(cudaMemcpyAsync(d_force, e->d_force.p, bytes, cudaMemcpyDeviceToDevice, e->stream));
        if (recomputed) *recomputed = 0;
        return HC_OK;
    }
    e->host_stepping = false;
    e->inputs_on_copy_stream = false;
    // the kernels write the forces to the caller's buffer and to the ensemble's time-keyed cache
    e->begin_step(t, g, d_pose, d_vel, d_force);
    e->finish_step(t);
    if (recomputed) *recomputed = 1;
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_step(hc_ensemble* e, double t, const double* pose, const double* vel, const double g[3], double* force,
                  int* recomputed) {
    HC_GUARD_BEGIN
    if (!pose || !vel || !g || !force) fail(HC_ERR_INVALID, "null argument");
    e->use_device();
    const size_t bytes = size_t(e->B) * e->D * sizeof(double);
    int re = 0;
    const bool tr = e->trace && t != e->prev_time;
    const auto h0 = std::chrono::steady_clock::now();
    bool compact_done = false;
    if (t != e->prev_time) {
        e->host_stepping = true;
        const bool try_compact = e->compact_ok && !e->profiling && !tr && e->opts.use_graph;
        if (try_compact) {
            // small ensemble (the drop-in B = 1 case): stage the inputs in the pinned block; if the per-step kernels serve
            // this step the whole step is ONE graph launch
            unsigned char* hs = static_cast<unsigned char*>(e->h_stage.p);
            std::memcpy(hs + 256, vel, bytes);
            std::memcpy(hs + 256 + bytes, pose, bytes);
            e->defer_launch = true;
            e->inputs_on_copy_stream = false;
            bool began = false;
            try {
                e->begin_step(t, g, e->d_pose.p, e->d_vel.p, e->d_force.p);
                began = true;
            } catch (...) {
                e->defer_launch = false;
                cudaStreamSynchronize(e->stream);
                throw;
            }
            if (began && e->defer_launch) {              // per-step kernels: one graph
                e->defer_launch = false;
                if (e->h_force_dev) e->hdr_h.force2 = e->h_force_dev;
                std::memcpy(hs, &e->hdr_h, sizeof(StepHeader));
                e->run_compact();
                e->prof.kernel_launches += e->phase1_launches + (e->graph_c_inline ? 0 : 1);   // (no append kernel; no plan kernel either when the convolutions plan inline)
                e->prof.hydrostatics_calls++; e->prof.radiation_calls++; e->prof.waves_calls++;
                e->prev_time = t;
                e->force_valid = true;
                CUDA_CHECK(cudaStreamSynchronize(e->stream));
                std::memcpy(force, e->h_force.p, bytes);
                compact_done = true;
            } else {                                     // a look-ahead block serves the step: upload, then as usual
                CUDA_CHECK(cudaMemcpyAsync(e->d_stage.p + 256, hs + 256, 2 * bytes, cudaMemcpyHostToDevice, e->stream));
                e->finish_step(t);
            }
            re = 1;
        } else {
        // State upload.  A step served by both look-aheads has nothing to run before its state arrives (phase 1 is
        // empty): everything goes down the main stream, no cross-stream events.  Otherwise the upload runs on the copy
        // stream underneath the state-independent phase 1 (plans, per-step convolutions).  Which of the two this step
        // will be is known only inside begin_step, so the previous step's answer decides where the copies go.
        const bool on_copy = !e->last_step_fast;
        cudaStream_t cs = on_copy ? e->copy_stream : e->stream;
        if (tr) CUDA_CHECK(cudaEventRecord(e->ev_tr[0], cs));
        CUDA_CHECK(cudaMemcpyAsync(e->d_vel.p, vel, bytes, cudaMemcpyHostToDevice, cs));
        CUDA_CHECK(cudaMemcpyAsync(e->d_pose.p, pose, bytes, cudaMemcpyHostToDevice, cs));
        if (tr) CUDA_CHECK(cudaEventRecord(e->ev_tr[1], cs));
        if (on_copy) CUDA_CHECK(cudaEventRecord(e->ev_inputs, e->copy_stream));
        e->inputs_on_copy_stream = on_copy;
        // (Measured and not kept, 2048 instances per GPU: k_step reading the state straight from pinned host memory
        //  -- SM-issued PCIe reads of 0.4 MB take ~50 us against 11 us for the copy engine; k_step writing the totals
        //  straight into a pinned result buffer, and one merged upload of adjacent arrays -- no gain, 65.7 vs 65.2 us per
        //  step: the chain is k_step's own ~26 us latency plus host wake-up, not the copies.)
        try {
            e->begin_step(t, g, e->d_pose.p, e->d_vel.p, e->d_force.p);
        } catch (...) {
            cudaStreamSynchronize(e->copy_stream);
            cudaStreamSynchronize(e->stream);
            throw;
        }
        if (on_copy) CUDA_CHECK(cudaStreamWaitEvent(e->stream, e->ev_inputs, 0));
        e->inputs_on_copy_stream = false;
        if (tr) CUDA_CHECK(cudaEventRecord(e->ev_tr[2], e->stream));
        e->finish_step(t);
        re = 1;
        }
    }
    if (!compact_done) {
        if (tr) CUDA_CHECK(cudaEventRecord(e->ev_tr[3], e->stream));
        CUDA_CHECK(cudaMemcpyAsync(force, e->d_force.p, bytes, cudaMemcpyDeviceToHost, e->stream));
        if (tr) CUDA_CHECK(cudaEventRecord(e->ev_tr[4], e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
    }
    if (tr) {
        float a = 0, b = 0, c = 0, d = 0, f = 0;
        cudaEventElapsedTime(&a, e->ev_tr[0], e->ev_tr[1]);
        cudaEventElapsedTime(&b, e->ev_tr[1], e->ev_tr[2]);
        cudaEventElapsedTime(&c, e->ev_tr[2], e->ev_tr[3]);
        cudaEventElapsedTime(&d, e->ev_tr[3], e->ev_tr[4]);
        cudaEventElapsedTime(&f, e->ev_tr[0], e->ev_tr[4]);
        e->tr_ms[0] += a; e->tr_ms[1] += b; e->tr_ms[2] += c; e->tr_ms[3] += d; e->tr_ms[4] += f;
        e->tr_ms[5] += 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - h0).count();
        ++e->tr_n;
    }
    if (e->events_pending) e->collect_events();
    if (recomputed) *recomputed = re;
    return HC_OK;
    HC_GUARD_END
}

// WaveBase::GetForceAtTime(t) for every instance (src/wave_types.cpp:257-264,315-327,552-570): state-independent,
// does not touch the velocity history or the force cache.
hc_status hc_waves_force_at_time(hc_ensemble* e, double t, double* out) {
    HC_GUARD_BEGIN
    if (!out) fail(HC_ERR_INVALID, "null argument");
    e->use_device();
    const size_t n = size_t(e->B) * e->D;
    if (e->wave_mode == 0) { std::fill(out, out + n, 0.0); return HC_OK; }
    if (e->wave_mode == 2) {
        const double tmin = e->eta_t_h.front(), tmax = e->eta_t_h.back();
        for (auto& G : e->groups) {
            const double hi = t - G->tau_first, lo = t - G->tau_last;
            if (!(tmin <= lo && hi <= tmax))
                fail(HC_ERR_ETA_WINDOW,
                     "Excitation convolution: trying to find free surface elevation at a time out of bounds from the "
                     "precomputed free surface elevation (" + std::to_string(hi > tmax ? hi : lo) + "not in [" +
                     std::to_string(tmin) + ", " + std::to_string(tmax) + "]). Excitation force ignored at this time step.");
        }
    }
    if (e->events_pending) { CUDA_CHECK(cudaStreamSynchronize(e->stream)); e->collect_events(); }
    if (e->d_wave_tmp.n < n) e->d_wave_tmp.alloc(n);
    StepHeader hh{};
    hh.t = t; hh.snap = e->opts.bracket_snap; hh.head = e->head < 0 ? 0 : e->head; hh.len = 0; hh.cap = e->cap;
    hh.force = e->d_wave_tmp.p;
    CUDA_CHECK(cudaMemcpyAsync(e->d_hdr.p, &hh, sizeof(StepHeader), cudaMemcpyHostToDevice, e->stream));
    const bool saved_la = e->phase_uses_lookahead;
    const bool saved_rb = e->rb_use;
    e->phase_uses_lookahead = false;                 // always the per-step kernels here
    e->rb_use = false;
    e->skip_radiation = true;
    e->enqueue_phase(1, false);
    e->skip_radiation = false;
    e->phase_uses_lookahead = saved_la;
    e->rb_use = saved_rb;
    FinalizeGroups fg{};
    if (e->wave_mode == 2)
        for (size_t g = 0; g < e->groups.size(); ++g) {
            auto& G = *e->groups[g];
            fg.dof0[g] = G.dof0; fg.nd[g] = G.nd; fg.chunk0[g] = G.chunk0; fg.nchunk[g] = G.nchunk;
        }
    FinalizeArgs fa{};
    fa.hdr = e->d_hdr.p; fa.exc_partial = e->d_exc_partial.p; fa.comp = nullptr;
    fa.reg_amp = e->d_reg_amp.p; fa.reg_omega = e->d_reg_omega.p; fa.reg_mag = e->d_reg_mag.p; fa.reg_phase = e->d_reg_phase.p;
    fa.B = e->B; fa.Bp = e->Bp; fa.D = e->D; fa.N = e->N; fa.rad_nchunk = 0; fa.wave_mode = e->wave_mode;
    fa.exc_ngroups = (e->wave_mode == 2) ? int(e->groups.size()) : 0; fa.exc_ndmax = e->exc_ndmax; fa.waves_only = 1;
    fa.pr_lead = e->d_pr_lead.p; fa.pr_wd = e->d_pr_wd.p; fa.pr_head = e->d_pr_head.p; fa.K = e->d_K.p; fa.L = 0;
    CUDA_CHECK(launch_finalize(fa, e->hs, fg, e->stream));
    CUDA_CHECK(cudaMemcpyAsync(out, e->d_wave_tmp.p, n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->prof.kernel_launches += 2 + (e->wave_mode == 2 ? (long long)e->groups.size() : 0);
    return HC_OK;
    HC_GUARD_END
}

// WaveBase::GetElevation / GetVelocity / GetAcceleration for every instance at its own points; like
// hc_waves_force_at_time it reads no eta window or history and touches no force cache.
hc_status hc_waves_kinematics_at_time_device(hc_ensemble* e, double t, int n_points, const double* d_points, double mwl,
                                             int wheeler_stretching, double* d_eta, double* d_velocity,
                                             double* d_acceleration) {
    HC_GUARD_BEGIN
    if (n_points < 1 || !d_points) fail(HC_ERR_INVALID, "n_points must be positive and points non-null");
    e->use_device();
    e->enqueue_kinematics(t, n_points, d_points, mwl, wheeler_stretching, d_eta, d_velocity, d_acceleration);
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_waves_kinematics_at_time(hc_ensemble* e, double t, int n_points, const double* points, double mwl,
                                      int wheeler_stretching, double* eta, double* velocity, double* acceleration) {
    HC_GUARD_BEGIN
    if (n_points < 1 || !points) fail(HC_ERR_INVALID, "n_points must be positive and points non-null");
    e->use_device();
    const size_t n = size_t(e->B) * n_points;
    // one device block: points [n][3] | eta [n] | velocity [n][3] | acceleration [n][3]
    if (e->d_kin_io.n < 10 * n) e->d_kin_io.alloc(10 * n, false);
    double* dp = e->d_kin_io.p;
    double* de = dp + 3 * n;
    double* dv = de + n;
    double* da = dv + 3 * n;
    CUDA_CHECK(cudaMemcpyAsync(dp, points, 3 * n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    e->enqueue_kinematics(t, n_points, dp, mwl, wheeler_stretching, eta ? de : nullptr, velocity ? dv : nullptr,
                          acceleration ? da : nullptr);
    if (eta) CUDA_CHECK(cudaMemcpyAsync(eta, de, n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (velocity) CUDA_CHECK(cudaMemcpyAsync(velocity, dv, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    if (acceleration)
        CUDA_CHECK(cudaMemcpyAsync(acceleration, da, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    return HC_OK;
    HC_GUARD_END
}

// Components of the current waves for k_wave_kinematics.  omega, k, the branch flag and sinh(k depth) are computed here
// with the reference's expressions (wave_types.cpp:66-83): the same doubles the host arithmetic uses.
void hc_ensemble::stage_kinematics() {
    const double depth = T->depth;
    auto deep = [depth](double k) { return (2 * M_PI / k > depth || k * depth > 500.0) ? 1.0 : 0.0; };
    auto put = [](std::vector<double>& c, size_t stride, size_t j, double om, double k, double dp, double shkd, double A,
                  double ph) {
        c[kKinOmega * stride + j] = om; c[kKinK * stride + j] = k; c[kKinDeep * stride + j] = dp;
        c[kKinSinhKd * stride + j] = shkd; c[kKinAmp * stride + j] = A; c[kKinPhase * stride + j] = ph;
    };
    if (wave_mode == 1) {
        std::vector<double> c(size_t(kKinFields) * Bp, 0.0);
        for (int b = 0; b < B; ++b) {
            const int i = reg_count == 1 ? 0 : b;
            const double k = reg_k_h[i];
            put(c, Bp, b, reg_omega_h[i], k, deep(k), std::sinh(k * depth), reg_amp_h[i], reg_wave_phase_h[i]);
        }
        d_kin_comp.upload(c);
    } else {
        std::vector<double> amp, ph;
        pack_irregular(amp, ph);
        std::vector<double> c(size_t(kKinFields) * nf, 0.0);
        for (int i = 0; i < nf; ++i) {
            const double k = wavenumbers_h[i];
            put(c, nf, i, 2 * M_PI * freqs_h[i], k, deep(k), std::sinh(k * depth), per_instance_spectrum ? 0.0 : amp[i],
                0.0);
        }
        d_kin_comp.upload(c);
        d_kin_phase.upload(ph);
        if (per_instance_spectrum) d_kin_amp.upload(amp);
    }
    kin_staged = true;
}

void hc_ensemble::enqueue_kinematics(double t, int n_points, const double* d_points, double mwl, int wheeler,
                                     double* d_eta, double* d_vel, double* d_acc) {
    const size_t n = size_t(B) * n_points;
    if (wave_mode == 0 || (wave_mode == 2 && nf == 0)) {
        // NoWave, an imported eta series, or no sea state: the reference sums over empty component vectors
        if (d_eta) CUDA_CHECK(cudaMemsetAsync(d_eta, 0, n * sizeof(double), stream));
        if (d_vel) CUDA_CHECK(cudaMemsetAsync(d_vel, 0, 3 * n * sizeof(double), stream));
        if (d_acc) CUDA_CHECK(cudaMemsetAsync(d_acc, 0, 3 * n * sizeof(double), stream));
        return;
    }
    if (!kin_staged) stage_kinematics();
    KinArgs a{};
    a.points = d_points; a.eta = d_eta; a.vel = d_vel; a.acc = d_acc;
    a.comp = d_kin_comp.p; a.amp = d_kin_amp.p; a.phase = d_kin_phase.p;
    a.t = t; a.depth = T->depth; a.mwl = mwl;
    a.B = B; a.Bp = Bp; a.P = n_points; a.nf = nf;
    a.regular = wave_mode == 1;
    a.wheeler = (wave_mode == 2 && wheeler) ? 1 : 0;
    CUDA_CHECK(launch_wave_kinematics(a, sm_count, stream));
    prof.kernel_launches += 1;
}

// ---- device-side stepping ----------------------------------------------------------------
// Inverse of diag(m, m, m, Ixx, Iyy, Izz) + A_inf restricted to the free DoFs (Gauss-Jordan, partial pivoting), zero
// rows and columns at locked DoFs.
static std::vector<double> sim_inverse_mass(const hc_tables* T, const hc_sim_params& p, unsigned long long free_mask) {
    const int D = T->D;
    std::vector<int> idx;
    for (int i = 0; i < D; ++i) if ((free_mask >> i) & 1ull) idx.push_back(i);
    const int n = int(idx.size());
    std::vector<double> A(size_t(n) * 2 * n, 0.0);
    for (int r = 0; r < n; ++r) {
        const int i = idx[r], b = i / 6, k = i % 6;
        for (int c = 0; c < n; ++c) {
            const int j = idx[c];
            double m = (i == j) ? (k < 3 ? p.mass[b] : p.inertia[3 * b + k - 3]) : 0.0;
            m += T->body[b].ainf[size_t(k) * D + j];
            A[size_t(r) * 2 * n + c] = m;
        }
        A[size_t(r) * 2 * n + n + r] = 1.0;
    }
    for (int c = 0; c < n; ++c) {
        int piv = c;
        for (int r = c + 1; r < n; ++r)
            if (std::fabs(A[size_t(r) * 2 * n + c]) > std::fabs(A[size_t(piv) * 2 * n + c])) piv = r;
        const double d = A[size_t(piv) * 2 * n + c];
        if (d == 0.0 || !std::isfinite(d)) fail(HC_ERR_INVALID, "hc_ensemble_simulate: singular free-DoF mass matrix");
        if (piv != c) for (int k = 0; k < 2 * n; ++k) std::swap(A[size_t(c) * 2 * n + k], A[size_t(piv) * 2 * n + k]);
        for (int k = 0; k < 2 * n; ++k) A[size_t(c) * 2 * n + k] /= d;
        for (int r = 0; r < n; ++r) {
            const double f = A[size_t(r) * 2 * n + c];
            if (r == c || f == 0.0) continue;
            for (int k = 0; k < 2 * n; ++k) A[size_t(r) * 2 * n + k] -= f * A[size_t(c) * 2 * n + k];
        }
    }
    std::vector<double> Minv(size_t(D) * D, 0.0);
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) {
            const double v = A[size_t(r) * 2 * n + n + c];
            if (!std::isfinite(v)) fail(HC_ERR_INVALID, "hc_ensemble_simulate: singular free-DoF mass matrix");
            Minv[size_t(idx[r]) * D + idx[c]] = v;
        }
    return Minv;
}

// Validation and descriptors of a run with joints / spring-dampers (k_body_step_linked): fills the link fields of la,
// the full mass matrix M = diag(m, m, m, Ixx, Iyy, Izz) + A_inf and the key that identifies the links (continuation).
static void sim_links_setup(const hc_tables* T, const hc_sim_params& p, unsigned long long free_mask, LinkStepArgs& la,
                            std::vector<double>& M, std::vector<double>& key) {
    const hc_sim_links& L = *p.links;
    const int N = T->N, D = T->D;
    auto bad = [](const std::string& m) { fail(HC_ERR_INVALID, "hc_ensemble_simulate: " + m); };
    if (L.n_prismatic < 0 || L.n_tsda < 0) bad("negative joint or spring-damper count");
    if ((L.n_prismatic > 0 && !L.prismatic) || (L.n_tsda > 0 && !L.tsda)) bad("null joint or spring-damper array");
    if (L.n_tsda > kMaxLinkTsda) bad("more than " + std::to_string(kMaxLinkTsda) + " spring-dampers");
    if (L.n_prismatic > N) bad("more joints than bodies (a body is the child of one joint at most)");
    for (int n = 0; n < kMaxBodies; ++n) { la.parent_of[n] = -2; la.joint_of[n] = -1; }
    for (int j = 0; j < L.n_prismatic; ++j) {
        const hc_sim_prismatic& J = L.prismatic[j];
        if (J.child < 0 || J.child >= N || J.parent < -1 || J.parent >= N) bad("joint body index out of range");
        if (J.child == J.parent) bad("joint child == parent");
        if (la.joint_of[J.child] >= 0) bad("a second joint on one child");
        const double n2 = J.axis[0] * J.axis[0] + J.axis[1] * J.axis[1] + J.axis[2] * J.axis[2];
        if (!(n2 > 0.0) || !std::isfinite(n2)) bad("zero or non-finite joint axis");
        const double n = std::sqrt(n2);
        la.joint_of[J.child] = j;
        la.parent_of[J.child] = J.parent;
        la.pr_child[j] = J.child; la.pr_parent[j] = J.parent;
        for (int k = 0; k < 3; ++k) la.pr_axis[j][k] = J.axis[k] / n;
        for (int k = 0; k < 6; ++k)
            if (!((free_mask >> (6 * J.child + k)) & 1ull)) bad("a jointed child must have every DoF free");
    }
    for (int j = 0; j < L.n_prismatic; ++j)
        if (la.pr_parent[j] >= 0 && la.joint_of[la.pr_parent[j]] >= 0) bad("chains of joints are not supported");
    for (int t = 0; t < L.n_tsda; ++t) {
        const hc_sim_tsda& S = L.tsda[t];
        if (S.body1 < -1 || S.body1 >= N || S.body2 < -1 || S.body2 >= N) bad("spring-damper body index out of range");
        if (S.body1 == S.body2) bad(S.body1 < 0 ? "spring-damper between ground and ground" : "spring-damper body1 == body2");
        la.ts_b1[t] = S.body1; la.ts_b2[t] = S.body2; la.ts_rest[t] = S.rest_length;
        for (int k = 0; k < 3; ++k) { la.ts_p1[t][k] = S.point1[k]; la.ts_p2[t][k] = S.point2[k]; }
    }
    la.n_pr = L.n_prismatic; la.n_tsda = L.n_tsda;
    // columns of T: the free DoFs of every root body in body order, then one slide per child in body order
    int nq = 0;
    for (int n = 0; n < N; ++n)
        if (la.joint_of[n] < 0)
            for (int k = 0; k < 6; ++k)
                if ((free_mask >> (6 * n + k)) & 1ull) { la.col_body[nq] = (signed char)n; la.col_dof[nq] = (signed char)k; ++nq; }
    for (int n = 0; n < N; ++n)
        if (la.joint_of[n] >= 0) { la.col_body[nq] = (signed char)n; la.col_dof[nq] = 6; ++nq; }
    la.nq = nq;
    M.assign(size_t(D) * D, 0.0);
    for (int i = 0; i < D; ++i) {
        const int b = i / 6, k = i % 6;
        M[size_t(i) * D + i] = k < 3 ? p.mass[b] : p.inertia[3 * b + k - 3];
    }
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) M[size_t(i) * D + j] += T->body[i / 6].ainf[size_t(i % 6) * D + j];
    // Cholesky of the symmetric part: positive definite => T^T M T is nonsingular for every full-column-rank T
    std::vector<double> C(size_t(D) * D);
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) C[size_t(i) * D + j] = 0.5 * (M[size_t(i) * D + j] + M[size_t(j) * D + i]);
    for (int j = 0; j < D; ++j) {
        double d = C[size_t(j) * D + j];
        for (int k = 0; k < j; ++k) d -= C[size_t(j) * D + k] * C[size_t(j) * D + k];
        if (!(d > 0.0) || !std::isfinite(d)) bad("the mass matrix diag(m, I) + A_inf is not positive definite");
        const double r = std::sqrt(d);
        C[size_t(j) * D + j] = r;
        for (int i = j + 1; i < D; ++i) {
            double s = C[size_t(i) * D + j];
            for (int k = 0; k < j; ++k) s -= C[size_t(i) * D + k] * C[size_t(j) * D + k];
            C[size_t(i) * D + j] = s / r;
        }
    }
    key.clear();
    for (int j = 0; j < la.n_pr; ++j) {
        key.push_back(la.pr_child[j]); key.push_back(la.pr_parent[j]);
        for (int k = 0; k < 3; ++k) key.push_back(la.pr_axis[j][k]);
    }
    key.push_back(-1.0);
    for (int t = 0; t < la.n_tsda; ++t) {
        key.push_back(la.ts_b1[t]); key.push_back(la.ts_b2[t]); key.push_back(la.ts_rest[t]);
        for (int k = 0; k < 3; ++k) { key.push_back(la.ts_p1[t][k]); key.push_back(la.ts_p2[t][k]); }
    }
}

// host = true: pose, vel, rec_*, energy are host memory (records through a bounded device buffer, copied out in chunks;
// record k of rec_pose / rec_vel starts at element k * rec_stride).  host = false: device memory, rec_stride = B D.
static hc_status sim_run(hc_ensemble* e, const hc_sim_params* p, bool host, double* pose, double* vel, double* rec_t,
                         double* rec_pose, double* rec_vel, size_t rec_stride, double* energy, int* steps_done) {
    HC_GUARD_BEGIN
    if (steps_done) *steps_done = 0;
    if (!p || !pose || !vel) fail(HC_ERR_INVALID, "hc_ensemble_simulate: null params, pose or vel");
    if (p->n_steps < 1 || p->record_every < 1) fail(HC_ERR_INVALID, "hc_ensemble_simulate: n_steps and record_every must be >= 1");
    if (!(p->dt > 0.0)) fail(HC_ERR_INVALID, "hc_ensemble_simulate: dt must be > 0");
    if (!p->mass || !p->inertia) fail(HC_ERR_INVALID, "hc_ensemble_simulate: mass and inertia are required");
    if (p->scheme != 0 && p->scheme != 1) fail(HC_ERR_INVALID, "hc_ensemble_simulate: scheme must be 0 (Euler) or 1 (HHT)");
    e->use_device();
    const int B = e->B, D = e->D, N = e->N;
    const size_t bd = size_t(B) * D, bytes = bd * sizeof(double);
    unsigned long long free_mask = 0;
    for (int i = 0; i < D; ++i) if (!p->free_dof || p->free_dof[i]) free_mask |= 1ull << i;
    // links: a non-empty hc_sim_links runs k_body_step_linked; NULL or empty runs k_body_step as before
    const bool linked = p->links && (p->links->n_prismatic != 0 || p->links->n_tsda != 0);
    LinkStepArgs la{};
    std::vector<double> link_M, link_key;
    if (linked) sim_links_setup(e->T, *p, free_mask, la, link_M, link_key);
    const std::vector<double> Minv = linked ? std::vector<double>() : sim_inverse_mass(e->T, *p, free_mask);
    cudaStream_t st = e->stream;
    if (e->d_sim.n != size_t(hc_ensemble::kSimSlots) * bd) { e->d_sim.alloc(size_t(hc_ensemble::kSimSlots) * bd); e->sim_q_valid = false; }
    if (e->d_simq.n != size_t(8) * B * N) { e->d_simq.alloc(size_t(8) * B * N); e->sim_q_valid = false; }
    if (e->d_minv.n != size_t(D) * D) e->d_minv.alloc(size_t(D) * D);
    // pageable sources: the runtime stages them at the call, so the host vectors may go out of scope at once
    if (!linked) CUDA_CHECK(cudaMemcpyAsync(e->d_minv.p, Minv.data(), Minv.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    const hc_sim_links* L = p->links;
    double* d_tsda_energy = nullptr;
    if (linked) {
        const size_t asm_n = size_t(B) * (la.n_pr * kLinkAsmJoint + la.n_tsda * kLinkAsmTsda);
        const size_t bt = size_t(B) * la.n_tsda;
        if (e->d_link_M.n != size_t(D) * D) e->d_link_M.alloc(size_t(D) * D);
        if (e->d_link_asm.n != asm_n) { e->d_link_asm.alloc(asm_n); e->link_asm_valid = false; }
        if (e->d_link_end.n != bd) { e->d_link_end.alloc(bd); e->link_asm_valid = false; }
        if (bt > 0 && e->d_link_coef.n < 2 * bt) e->d_link_coef.alloc(2 * bt);
        if (host && bt > 0 && L->tsda_energy && e->d_link_energy.n < bt) e->d_link_energy.alloc(bt);
        CUDA_CHECK(cudaMemcpyAsync(e->d_link_M.p, link_M.data(), link_M.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        if (bt > 0 && L->tsda_damping)
            CUDA_CHECK(cudaMemcpyAsync(e->d_link_coef.p, L->tsda_damping, bt * sizeof(double), cudaMemcpyHostToDevice, st));
        if (bt > 0 && L->tsda_stiffness)
            CUDA_CHECK(cudaMemcpyAsync(e->d_link_coef.p + bt, L->tsda_stiffness, bt * sizeof(double), cudaMemcpyHostToDevice, st));
        la.M = e->d_link_M.p;
        la.asm_data = e->d_link_asm.p;
        la.end_pose = e->d_link_end.p;
        la.tsda_c = bt > 0 && L->tsda_damping ? e->d_link_coef.p : nullptr;
        la.tsda_k = bt > 0 && L->tsda_stiffness ? e->d_link_coef.p + bt : nullptr;
        d_tsda_energy = bt > 0 && L->tsda_energy ? (host ? e->d_link_energy.p : L->tsda_energy) : nullptr;
        if (d_tsda_energy) CUDA_CHECK(cudaMemsetAsync(d_tsda_energy, 0, bt * sizeof(double), st));
        la.tsda_energy = d_tsda_energy;
        la.keep_asm = e->link_asm_valid && link_key == e->link_key ? 1 : 0;
    }
    const bool has_c = p->pto_damping != nullptr, has_k = p->pto_stiffness != nullptr;
    if ((has_c || has_k) && e->d_pto.n != 2 * bd) e->d_pto.alloc(2 * bd);
    if (has_c) CUDA_CHECK(cudaMemcpyAsync(e->d_pto.p, p->pto_damping, bytes, cudaMemcpyHostToDevice, st));
    if (has_k) CUDA_CHECK(cudaMemcpyAsync(e->d_pto.p + bd, p->pto_stiffness, bytes, cudaMemcpyHostToDevice, st));
    const cudaMemcpyKind in = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const cudaMemcpyKind out = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CUDA_CHECK(cudaMemcpyAsync(e->sim(hc_ensemble::kSimPose0), pose, bytes, in, st));
    CUDA_CHECK(cudaMemcpyAsync(e->sim(hc_ensemble::kSimVel0), vel, bytes, in, st));
    double* d_energy = energy ? (host ? e->sim(hc_ensemble::kSimEnergy) : energy) : nullptr;
    if (d_energy) CUDA_CHECK(cudaMemsetAsync(d_energy, 0, bytes, st));

    // records: device variant straight into the caller's arrays, host variant through a chunk of R records
    const int n_rec = p->n_steps / p->record_every;
    const bool want_rec = (rec_pose || rec_vel) && n_rec > 0;
    int R = n_rec;
    if (host && want_rec) {
        R = int(std::max<size_t>(1, std::min<size_t>(size_t(n_rec), (size_t(64) << 20) / (2 * bytes))));
        if (e->d_rec.n < 2 * size_t(R) * bd) e->d_rec.alloc(2 * size_t(R) * bd, false);
        if (e->h_rec_bytes < 2 * size_t(R) * bytes) { e->h_rec.alloc(2 * size_t(R) * bytes); e->h_rec_bytes = 2 * size_t(R) * bytes; }
    }
    int chunk_first = 0, chunk_len = 0;
    auto flush = [&]() {
        if (!host || chunk_len == 0) return;
        double* hp = static_cast<double*>(e->h_rec.p);
        CUDA_CHECK(cudaMemcpyAsync(hp, e->d_rec.p, size_t(chunk_len) * bytes, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(hp + size_t(R) * bd, e->d_rec.p + size_t(R) * bd, size_t(chunk_len) * bytes,
                                   cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (int k = 0; k < chunk_len; ++k) {
            if (rec_pose) std::memcpy(rec_pose + size_t(chunk_first + k) * rec_stride, hp + size_t(k) * bd, bytes);
            if (rec_vel) std::memcpy(rec_vel + size_t(chunk_first + k) * rec_stride, hp + size_t(R + k) * bd, bytes);
        }
        chunk_first += chunk_len;
        chunk_len = 0;
    };

    BodyStepArgs a{};
    a.force = e->d_force.p;
    a.q = e->d_simq.p; a.qe = e->d_simq.p + size_t(4) * B * N;
    a.Minv = e->d_minv.p;
    a.pto_c = has_c ? e->d_pto.p : nullptr;
    a.pto_k = has_k ? e->d_pto.p + bd : nullptr;
    a.x0 = has_k ? e->sim(hc_ensemble::kSimX0) : nullptr;
    for (int k = 0; k < 3; ++k) a.g[k] = p->g[k];
    for (int b = 0; b < N; ++b) a.mass[b] = p->mass[b];
    a.dt = p->dt; a.free_mask = free_mask; a.B = B; a.N = N; a.D = D;
    const bool hht = p->scheme == 1;
    if (hht) {
        a.sx = e->sim(hc_ensemble::kSimX); a.sv = e->sim(hc_ensemble::kSimV);
        a.Fn = e->sim(hc_ensemble::kSimFn); a.an = e->sim(hc_ensemble::kSimAn);
    }
    auto evp = [&](int i) { return e->sim(hc_ensemble::kSimPose0 + i); };
    auto evv = [&](int i) { return e->sim(hc_ensemble::kSimVel0 + i); };
    auto launch = [&](int mode, int cur) {
        a.pose_in = evp(cur); a.vel_in = evv(cur);
        a.pose_out = evp(mode == kBodyInit ? cur : cur ^ 1); a.vel_out = evv(mode == kBodyInit ? cur : cur ^ 1);
        if (linked) {
            la.s = a;
            CUDA_CHECK(launch_body_step_linked(la, mode, st));
        } else {
            CUDA_CHECK(launch_body_step(a, mode, st));
        }
        e->prof.kernel_launches += 1;
    };
    a.keep_q = e->sim_q_valid ? 1 : 0;
    launch(kBodyInit, 0);
    e->sim_q_valid = true;
    a.keep_q = 0;
    la.keep_asm = 0;
    // the assembly data now belong to this run (a run without links leaves none behind)
    e->link_asm_valid = linked;
    if (linked) e->link_key = link_key;

    std::vector<double> times(static_cast<size_t>(n_rec), 0.0);
    double t = p->t0;
    int cur = 0, done = 0;
    hc_status status = HC_OK;
    if (hht) {
        status = hc_step_device(e, t, evp(0), evv(0), p->g, e->d_force.p, nullptr);     // StepHHTBegin's F_0
        if (status == HC_OK) { launch(kBodyHHTStart, 0); cur = 1; }
    }
    for (int n = 0; status == HC_OK && n < p->n_steps; ++n) {
        if (hht) t += p->dt;
        status = hc_step_device(e, t, evp(cur), evv(cur), p->g, e->d_force.p, nullptr);
        if (status != HC_OK) break;
        if (!hht) t += p->dt;
        const bool rec_step = n_rec > 0 && (n + 1) % p->record_every == 0;
        const int k = (n + 1) / p->record_every - 1;
        if (rec_step) times[size_t(k)] = t;
        const bool rec = want_rec && rec_step;
        a.energy = d_energy;
        a.rec_pose = a.rec_vel = nullptr;
        if (rec) {
            if (host) {
                a.rec_pose = e->d_rec.p + size_t(chunk_len) * bd;
                a.rec_vel = e->d_rec.p + size_t(R + chunk_len) * bd;
            } else {
                a.rec_pose = rec_pose ? rec_pose + size_t(k) * rec_stride : nullptr;
                a.rec_vel = rec_vel ? rec_vel + size_t(k) * rec_stride : nullptr;
            }
        }
        launch(hht ? kBodyHHTStep : kBodyEuler, cur);
        cur ^= 1;
        done = n + 1;
        if (rec && host && ++chunk_len == R) flush();
    }
    const std::string msg = status == HC_OK ? std::string() : std::string(hc_last_error());
    flush();
    // final state: Euler = the evaluation buffer of the next step; HHT = the state slots (the evaluation buffer holds
    // the predictor)
    CUDA_CHECK(cudaMemcpyAsync(pose, hht ? e->sim(hc_ensemble::kSimX) : evp(cur), bytes, out, st));
    CUDA_CHECK(cudaMemcpyAsync(vel, hht ? e->sim(hc_ensemble::kSimV) : evv(cur), bytes, out, st));
    if (energy && host) CUDA_CHECK(cudaMemcpyAsync(energy, d_energy, bytes, cudaMemcpyDeviceToHost, st));
    if (linked) {
        // the pose this run ended in: a continuation call that starts from it keeps the assembly data
        CUDA_CHECK(cudaMemcpyAsync(e->d_link_end.p, hht ? e->sim(hc_ensemble::kSimX) : evp(cur), bytes,
                                   cudaMemcpyDeviceToDevice, st));
        if (d_tsda_energy && host)
            CUDA_CHECK(cudaMemcpyAsync(L->tsda_energy, d_tsda_energy, size_t(B) * la.n_tsda * sizeof(double),
                                       cudaMemcpyDeviceToHost, st));
    }
    const size_t n_done_rec = size_t(done / p->record_every);
    if (rec_t && n_done_rec > 0) {
        if (host) std::memcpy(rec_t, times.data(), n_done_rec * sizeof(double));
        else CUDA_CHECK(cudaMemcpyAsync(rec_t, times.data(), n_done_rec * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if (host) CUDA_CHECK(cudaStreamSynchronize(st));
    if (steps_done) *steps_done = done;
    if (status != HC_OK) fail(status, msg);
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_ensemble_simulate(hc_ensemble* e, const hc_sim_params* p, double* pose, double* vel, double* rec_t,
                               double* rec_pose, double* rec_vel, double* pto_energy, int* steps_done) {
    return sim_run(e, p, true, pose, vel, rec_t, rec_pose, rec_vel, size_t(e->B) * e->D, pto_energy, steps_done);
}

hc_status hc_ensemble_simulate_device(hc_ensemble* e, const hc_sim_params* p, double* d_pose, double* d_vel,
                                      double* d_rec_t, double* d_rec_pose, double* d_rec_vel, double* d_pto_energy,
                                      int* steps_done) {
    return sim_run(e, p, false, d_pose, d_vel, d_rec_t, d_rec_pose, d_rec_vel, size_t(e->B) * e->D, d_pto_energy,
                   steps_done);
}

// hc_multi_ensemble_simulate: a shard's slice of global-order host arrays (records keep the global record stride)
hc_status hc_ensemble_simulate_strided(hc_ensemble* e, const hc_sim_params* p, double* pose, double* vel, double* rec_t,
                                       double* rec_pose, double* rec_vel, size_t rec_stride, double* pto_energy,
                                       int* steps_done) {
    return sim_run(e, p, true, pose, vel, rec_t, rec_pose, rec_vel, rec_stride, pto_energy, steps_done);
}

// Re-stages the radiation kernel after hc_tables_set_convolution_mode was called on the ensemble's tables.
hc_status hc_ensemble_refresh_rirf(hc_ensemble* e) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (e->rb_stream) CUDA_CHECK(cudaStreamSynchronize(e->rb_stream));
    e->rb_invalidate();              // blocks evaluated with the old kernel
    e->drop_graph();                 // the captured kernels hold the addresses of the old tables
    e->stage_kernel();
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_get_components(hc_ensemble* e, double* hs, double* rad, double* waves) {
    HC_GUARD_BEGIN
    e->use_device();
    const size_t n = size_t(e->B) * e->D;
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (hs) CUDA_CHECK(cudaMemcpy(hs, e->d_comp.p, n * sizeof(double), cudaMemcpyDeviceToHost));
    if (rad) CUDA_CHECK(cudaMemcpy(rad, e->d_comp.p + n, n * sizeof(double), cudaMemcpyDeviceToHost));
    if (waves) CUDA_CHECK(cudaMemcpy(waves, e->d_comp.p + 2 * n, n * sizeof(double), cudaMemcpyDeviceToHost));
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_sync(hc_ensemble* e) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (e->events_pending) e->collect_events();
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_ensemble_join(hc_ensemble* e) {
    HC_GUARD_BEGIN
    e->use_device();
    if (e->rb_stream) {
        CUDA_CHECK(cudaEventRecord(e->ev_rb_side, e->rb_stream));
        CUDA_CHECK(cudaStreamWaitEvent(e->stream, e->ev_rb_side, 0));
        if (!e->rb_pass.active) e->rb_side_pending = false;
    }
    if (e->la_stream) {
        CUDA_CHECK(cudaEventRecord(e->ev_la_join, e->la_stream));
        CUDA_CHECK(cudaStreamWaitEvent(e->stream, e->ev_la_join, 0));
    }
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_ensemble_lookahead_state(const hc_ensemble* e, int* radiation, int* excitation) {
    if (radiation) *radiation = (e->d_Kpad.p && e->rb_plan.usable) ? (e->rb_enabled ? 1 : 0) : -1;
    if (excitation) *excitation = e->d_la_cache.p ? (e->la_enabled ? 1 : 0) : -1;
    return HC_OK;
}

// ---- added mass ----------------------------------------------------------------------
hc_status hc_added_mass_mv_device(hc_ensemble* e, int n_sys, double c, const double* d_w, double* d_R) {
    HC_GUARD_BEGIN
    if (n_sys < e->D) fail(HC_ERR_INVALID, "n_sys must be >= 6 * num_bodies");
    e->use_device();
    CUDA_CHECK(launch_added_mass_mv(e->d_ainf.p, n_sys, e->D, c, d_w, d_R, e->B, e->stream));
    e->prof.kernel_launches += 1;
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_added_mass_mv(hc_ensemble* e, int n_sys, double c, const double* w, double* R) {
    HC_GUARD_BEGIN
    if (n_sys < e->D) fail(HC_ERR_INVALID, "n_sys must be >= 6 * num_bodies");
    e->use_device();
    const size_t n = size_t(e->B) * n_sys;
    DevBuf<double> dw, dR;
    dw.alloc(n, false); dR.alloc(n, false);
    CUDA_CHECK(cudaMemcpyAsync(dw.p, w, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CUDA_CHECK(cudaMemcpyAsync(dR.p, R, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CUDA_CHECK(launch_added_mass_mv(e->d_ainf.p, n_sys, e->D, c, dw.p, dR.p, e->B, e->stream));
    CUDA_CHECK(cudaMemcpyAsync(R, dR.p, n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->prof.kernel_launches += 1;
    return HC_OK;
    HC_GUARD_END
}

// ---- profiling -----------------------------------------------------------------------
hc_status hc_set_profiling(hc_ensemble* e, int enable) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (e->events_pending) e->collect_events();
    if (e->la_stream) CUDA_CHECK(cudaStreamSynchronize(e->la_stream));
    e->profiling = enable != 0;
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_get_profile(hc_ensemble* e, hc_profile_stats* out) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (e->events_pending) e->collect_events();
    *out = e->prof;
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_get_kernel_ms(hc_ensemble* e, double* pre, double* rad, double* exc, double* fin, int reset) {
    HC_GUARD_BEGIN
    e->use_device();
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    if (e->events_pending) e->collect_events();
    const double cnt = e->ms_steps > 0 ? double(e->ms_steps) : 1.0;
    if (pre) *pre = e->acc_ms[0] / cnt;
    if (rad) *rad = e->acc_ms[1] / cnt;
    if (exc) *exc = e->acc_ms[2] / cnt;
    if (fin) *fin = e->acc_ms[3] / cnt;
    if (reset) { for (double& v : e->acc_ms) v = 0.0; e->ms_steps = 0; }
    return HC_OK;
    HC_GUARD_END
}

// FP64 FMA throughput of the device (TFLOP/s), best of a few launches of a register-resident DFMA loop.
int hc_ensemble_rad_lookahead_steps(const hc_ensemble* e) { return e->rb_enabled ? kRbT * e->rb_m : 0; }

hc_status hc_get_rad_block_stats(hc_ensemble* e, long long* launches, long long* steps_served, double* avg_ms, int reset) {
    HC_GUARD_BEGIN
    e->use_device();
    if (e->events_pending) { CUDA_CHECK(cudaStreamSynchronize(e->stream)); e->collect_events(); }
    if (launches) *launches = e->rb_launches;
    if (steps_served) *steps_served = e->rb_steps_served;
    // duration of one whole pass, extrapolated from the slices timed while profiling was on
    if (avg_ms) *avg_ms = e->rb_items_timed ? e->rb_ms_sum / double(e->rb_items_timed) * e->rb_items_per_pass : 0.0;
    if (reset) { e->rb_launches = 0; e->rb_steps_served = 0; e->rb_items_timed = 0; e->rb_ms_sum = 0.0; }
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_get_exc_block_stats(hc_ensemble* e, long long* blocks_built, long long* steps_served, int reset) {
    if (blocks_built) *blocks_built = e->la_blocks_built;
    if (steps_served) *steps_served = e->la_steps_served;
    if (reset) { e->la_blocks_built = 0; e->la_steps_served = 0; }
    return HC_OK;
}

hc_status hc_measure_fp64_mma_peak(int device, double* tflops) {
    HC_GUARD_BEGIN
    if (!tflops) fail(HC_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(device));
    CUDA_CHECK(measure_dmma_peak(0.5, tflops));
    return HC_OK;
    HC_GUARD_END
}

hc_status hc_measure_fp64_peak(int device, double* tflops) {
    HC_GUARD_BEGIN
    if (!tflops) fail(HC_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(device));
    CUDA_CHECK(measure_dfma_peak(0.5, tflops));
    return HC_OK;
    HC_GUARD_END
}

void* hc_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void hc_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
