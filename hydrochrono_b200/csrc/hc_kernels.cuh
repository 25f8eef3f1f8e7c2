// Device-side data structures and kernel launch wrappers (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hc {

constexpr int kMaxBodies = 8;        // static hydrostatics tables live in kernel-parameter space
constexpr int kThreads = 256;        // CTA size of the convolution kernels
constexpr int kIPT = 2;              // instances per thread (one 16-byte load per history value pair)
constexpr int kTileInst = kThreads * kIPT;
constexpr int kHybTileInst = 256;  // instances per CTA of k_radiation_hybrid12 (4 warps x 64)

// Written by the host for every step (pinned -> device copy), read by every kernel of the step so that the
// captured CUDA graph is static.
struct StepHeader {
    double t;
    double g[3];
    double snap;       // bracket snap tolerance (0 = faithful)
    int head;          // ring slot of the newest history entry
    int len;           // history entries after pruning (newest first)
    int cap;           // ring capacity
    int flags;
    int exc_src;       // 0: irregular wave force = sum of this step's lag-chunk partials; 1: look-ahead cache slot
    int exc_slot;
    int rad_src;       // 0: radiation = this step's lag-chunk partials + head-row share; 1: radiation block (k_step)
    int rb_j;          // position of this step inside the radiation block
    int rb_smax;       // largest lag with a bracket at this step
    int rb_nchunk;     // row chunks of the block that hold data
    int rb_jj;         // steps since the block's snapshot of the history (rb_j, or rb_j + block length for a
                       // block that was evaluated in the background one block ahead)
    int rb_buf;        // which of the two partial buffers holds the block
    // the step's state and result buffers travel in the header so that the captured graphs and the directly launched
    // k_step stay valid when a caller rotates its device buffers from step to step
    const double* pose;   // [B][D]
    const double* vel;    // [B][D]
    double* force;        // [B][D]
    double* force2;       // second copy of the total (the caller's buffer when `force` is the ensemble's cache), or null
};

struct HydrostaticTables {
    double rho;
    double Kh[kMaxBodies][36];
    double disp_vol[kMaxBodies];
    double cb_minus_cg[kMaxBodies][3];
    double equilibrium[kMaxBodies][6];
};

struct RadiationArgs {
    const StepHeader* hdr;
    const double* K;          // [L][D col][D row]  (K w)
    const double* Kfrag;      // D = 12 only: [L][2][3][32] the same in DMMA A-fragment order (rows padded to 16); or null
    const double* Khyb;       // D = 12 only: [L][144] rows 0..7 as A fragments [3][32] + rows 8..11 as [q][k-step][row]; or null
    const double* rirf_t;     // [L]
    const double* rirf_w;     // [L]
    const double* hist;       // [cap][D][Bp]
    const double* times;      // [cap]
    double* partial;          // [nchunk][D][Bp]
    int L, D, Bp, chunk, nchunk;
};

struct ExcGroup {             // bodies sharing one excitation-IRF time grid
    const double* tau;        // [Le]
    const double* fw;         // [Le][nd]   f * width, dof fastest
    int Le, nd, dof0;         // dofs [dof0, dof0+nd) of the 6N vector
    int chunk0;               // first partial chunk index of this group
    int nchunk;
};

struct ExcitationArgs {
    const StepHeader* hdr;
    const double* eta;        // [n_eta][Bp]
    const double* eta_t;      // [n_eta]
    double* partial;          // [total chunks][ndmax][Bp]
    double eta_dt;            // nominal grid spacing (index guess only)
    int n_eta, Bp, chunk, ndmax;
};

struct FinalizeArgs {
    const StepHeader* hdr;    // pose / vel / force of the step come from the header
    const double* rad_partial;
    const double* exc_partial;
    double* comp;             // [3][B][D] hydrostatic, radiation, waves
    // regular waves (SoA over instances)
    const double* reg_amp;    // [Bp]
    const double* reg_omega;  // [Bp]
    const double* reg_mag;    // [D][Bp]
    const double* reg_phase;  // [6][Bp]  (body 0's phases, reference quirk wave_types.cpp:323)
    int B, Bp, D, N;
    int rad_nchunk;
    int wave_mode;            // 0 none, 1 regular, 2 irregular
    int exc_ngroups;
    int exc_ndmax;
    const double* exc_cache;  // [2][S][T][D][Bp] look-ahead blocks of wave forces (hdr->exc_src == 1), S row segments
    int exc_S;
    // share of this step's own velocity sample in the radiation convolution
    const double* K;          // [L][D][D]  (K w)
    const int* pr_lead;
    const double* pr_wd;
    const double* pr_head;
    int L;
    int waves_only;           // 1: write only the wave force (WaveBase::GetForceAtTime), no state needed
};

struct EtaArgs {
    const double* eta_t;      // [n_eta]
    const double* omega;      // [nf]    2*pi*f
    const double* amp;        // [nf] shared, or [nf][Bp] per instance
    const double* phase;      // [nf][Bp]
    double* eta;              // [n_eta][Bp]
    double ramp;
    int n_eta, nf, Bp, amp_per_instance;
};

// Water kinematics at caller-given points for every instance (k_wave_kinematics).  Lanes map to instances; each thread
// evaluates up to kKinPts points of its instance, further points go to blockIdx.y.
constexpr int kKinPts = 4;
constexpr int kKinChunk = 128;        // components staged in shared memory at a time
// rows of KinArgs::comp: omega, wavenumber, deep-water flag (1.0 / 0.0), sinh(k depth), amplitude, phase
enum { kKinOmega = 0, kKinK, kKinDeep, kKinSinhKd, kKinAmp, kKinPhase, kKinFields };
struct KinArgs {
    const double* points;     // [B][P][3]
    double* eta;              // [B][P]    or null
    double* vel;              // [B][P][3] or null
    double* acc;              // [B][P][3] or null
    // irregular waves: comp = [kKinFields][nf] per component (amplitude row = the shared spectrum's, phase row unused),
    // phase = [nf][Bp] per instance, amp = [nf][Bp] per instance or null when the spectrum is shared.
    // regular waves: comp = [kKinFields][Bp], one component per instance; amp and phase unused.
    const double* comp;
    const double* amp;
    const double* phase;
    double t, depth, mwl;
    int B, Bp, P, nf;
    int regular;
    int wheeler;              // irregular only: z' = depth (z - mwl - eta) / (depth + eta)
};

struct PrestepArgs {
    const StepHeader* hdr;
    double* hist;          // [cap][D][Bp]
    double* times;         // [cap]
    const double* rirf_t;  // [L]
    const double* rirf_w;  // [L]
    int* pr_new;           // [L] ring slot of the newer bracket sample
    int* pr_old;           // [L]
    double* pr_wn;         // [L] weight of the newer sample
    double* pr_wo;         // [L] weight of the older sample
    double* pr_wd;         // [L] trapezoid width (0 = lag skipped)
    double* pr_head;       // [L] weight of THIS step's velocity sample (handled by k_finalize), 0 elsewhere
    int* pr_lead;          // [L] 1 for the leading lags whose newer bracket sample is this step's
    int B, Bp, D, L;
    // excitation
    int ngroups;
    const double* tau[kMaxBodies];
    int Le[kMaxBodies];
    int* pe_idx[kMaxBodies];
    double* pe_w1[kMaxBodies];
    double* pe_w2[kMaxBodies];
    const double* eta_t;
    int n_eta;
    double eta_dt;
};

struct FinalizeGroups {
    int dof0[kMaxBodies], nd[kMaxBodies], chunk0[kMaxBodies], nchunk[kMaxBodies];
};

size_t radiation_smem_bytes(int D, int chunk);
size_t radiation_mma_smem_bytes(int chunk);
size_t excitation_smem_bytes(int nd, int chunk);
cudaError_t launch_prestep(const PrestepArgs& a, int mode, cudaStream_t st);
int radiation_ctas_per_sm(int D, int chunk);
int excitation_ctas_per_sm(int nd, int chunk);
// Compact graph of a small ensemble: the convolution kernels plan their own lags / taps and the radiation kernel
// appends the step's sample, so the step has no k_prestep level.  What k_finalize needs of the radiation plan (the
// leading lags) is written to these arrays by the radiation kernel.
struct InlinePlan { double* pr_wd; double* pr_head; int* pr_lead; int B; };
bool radiation_plans_inline(const RadiationArgs& a);
cudaError_t launch_radiation(const RadiationArgs& a, const int* pr_new, const int* pr_old, const double* pr_wn,
                             const double* pr_wo, const double* pr_wd, cudaStream_t st, const InlinePlan* ip = nullptr);
cudaError_t launch_excitation(const ExcitationArgs& a, const ExcGroup& g, const int* idx, const double* w1,
                              const double* w2, cudaStream_t st, bool plan_inline = false);
cudaError_t launch_finalize(const FinalizeArgs& a, const HydrostaticTables& hs, const FinalizeGroups& eg,
                            cudaStream_t st);
cudaError_t launch_eta(const EtaArgs& a, cudaStream_t st);
cudaError_t launch_wave_kinematics(const KinArgs& a, int sm_count, cudaStream_t st);
// ---- excitation look-ahead: the wave force of T consecutive (predicted) step times in one pass over eta ----
// Which finalize kernel serves an ensemble (depends only on its size and chunking, never on the step):
constexpr int kFinalizeWarpMaxB = 8;          // up to this many instances: k_finalize_warp (a warp per (dof, instance))
constexpr int kFinalizeSplitMinParts = 96;    // beyond that, with at least this many partials per item: k_finalize_split;
                                              // otherwise k_finalize (a thread per item: large ensembles, few long chunks)
constexpr int kLaT = 8;        // block length = warps per CTA of k_exc_block
constexpr int kLaRows = 32;    // eta rows per shared-memory stage
struct LookaheadPlanArgs {
    const double* times;      // [T] block times
    const double* tau;        // [Le]
    const double* fw;         // [Le][nd]
    const double* eta_t;      // [n_eta]
    int* idx;                 // [T][Le]  largest i with eta_t[i] <= t - tau_j
    double* w1;               // [T][Le]
    double* w2;               // [T][Le]
    double* taps;             // [nchunk][T][kLaRows][nd]
    double eta_dt;
    int n_eta, Le, nd, T, row0, nrows;   // rows row0 .. row0 + nrows - 1 of eta carry taps
    int frag_order;           // 1: taps in DMMA A-fragment order [chunk][k-step][M-tile][lane] (k_exc_block_mma)
};
struct LookaheadArgs {
    const double* eta;        // [n_eta][Bp]
    const double* taps;       // [nchunk][T][kLaRows][nd]
    double* cache;            // [S][T][D][Bp]: one partial block per segment of eta rows
    int n_eta, Bp, D, dof0, nd, row0, nchunk;
    int use_mma;              // 1: FP64 tensor-core kernel (taps in fragment order)
    int S;                    // segments the stages are split into (1 for k_exc_block)
    int seg0, nseg;           // k_exc_block_mma: this launch evaluates segments [seg0, seg0 + nseg) (grid.y = nseg)
};
// ---- radiation look-ahead: the share of the resident history rows in the next kRbT steps' convolutions, one pass ----
constexpr int kRbT = 8;            // steps per M-tile (rows of one DMMA tile); a block covers kRbT * m steps
constexpr int kRbMaxM = 8;         // largest supported ratio m = RIRF lag spacing / step size
// doubles per lag of the padded kernel table: [row][col padded to a multiple of 4], lag stride = 4 (mod 16) so that
// the 8 lags x 4 columns of one DMMA A fragment fall into 32 different 8-byte banks
__host__ __device__ constexpr int rb_dp(int D) { return 4 * ((D + 3) / 4); }
__host__ __device__ constexpr int rb_stride(int D) { return D * rb_dp(D) + (4 - (D * rb_dp(D)) % 16 + 16) % 16; }
static_assert(rb_stride(12) == 148 && rb_stride(6) == 52 && rb_stride(18) % 16 == 4, "bank-conflict-free lag stride");
constexpr int kRbTileInst = 64;    // instances per CTA of k_rad_block
struct RadBlockArgs {
    const double* hist;       // [cap][D][Bp]
    const double* Kpad;       // [lags + pad][rb_stride(D)]  (K w)[lag][row][col], zero beyond the last lag
    double* partial;          // [kRbT * m][nchunk][D][Bp]
    int D;
    const int* smax;          // [kRbT * m] per block step: largest lag with a bracket
    int head0;                // ring slot of the block's first step (resident row r lives in slot head0 - 1 - r)
    int cap, n_res, Bp, R, nchunk;
    int m;                    // history rows per RIRF lag (lag s of a step = history row m s)
    int g0;                   // 0: the block starts at the snapshot; kRbT: it starts kRbT * m steps after it
    int nchunk_used;          // chunks that hold rows; work items = (instance tile, chunk, residue class), tile fastest
    int item0;                // first work item of this launch (a pass can be cut into slices of consecutive items)
};
struct RadStepArgs {
    double* hist;
    double* times;
    const double* K;          // [L][col][row]
    const double* partial[2]; // [kRbT * m][nchunk][D][Bp], double-buffered
    int D, B, Bp, nchunk, L, m;
};
size_t rad_block_smem_bytes(int D, int R);
cudaError_t launch_rad_block(const RadBlockArgs& a, int nitems, cudaStream_t st);
inline int rad_block_items(const RadBlockArgs& a) { return ((a.Bp + kRbTileInst - 1) / kRbTileInst) * a.nchunk_used * a.m; }
cudaError_t launch_step(const RadStepArgs& a, const FinalizeArgs& fa, const HydrostaticTables& hs, const FinalizeGroups& eg,
                        const StepHeader& hdr, cudaStream_t st);
cudaError_t measure_dfma_peak(double seconds_budget, double* tflops);
cudaError_t measure_dmma_peak(double seconds_budget, double* tflops);
cudaError_t launch_lookahead_plan(const LookaheadPlanArgs& a, cudaStream_t st);
cudaError_t launch_lookahead(const LookaheadArgs& a, cudaStream_t st);

cudaError_t launch_added_mass_mv(const double* M, int n_sys, int D, double c, const double* w, double* R, int B,
                                 cudaStream_t st);

// ---- device-side stepping of free / ground-locked rigid bodies (hc_ensemble_simulate, k_body_step) ----
// The force path evaluates the "evaluation state" (Euler: the state itself; HHT: the predictor); k_body_step reads it and
// the step's hydro force and writes the next evaluation state into the other half of a ping-pong pair.
enum BodyStepMode {
    kBodyInit = 0,       // orientation from the caller's Cardan angles; evaluation state (+ HHT state, spring rest pose)
    kBodyEuler = 1,      // linearised Euler step (ChSystem::StepEnd)
    kBodyHHTStart = 2,   // HHT: initial accelerations from the force at t0, then the first predictor (StepHHTBegin)
    kBodyHHTStep = 3     // HHT: corrector (StepHHTEnd), then the next predictor
};
constexpr int kBodyThreads = 64;
struct BodyStepArgs {
    const double* force;      // [B][D] hydro force of this step's evaluation (unused by kBodyInit)
    const double* pose_in;    // [B][D] evaluation state (kBodyInit: the caller's initial state)
    const double* vel_in;
    double* pose_out;         // [B][D] next evaluation state
    double* vel_out;
    double* q;                // [B][N][4] orientation of the state
    double* qe;               // [B][N][4] HHT: orientation of the predictor
    double* sx;               // [B][D] HHT: state (positions, Cardan angles), updated in place
    double* sv;               // [B][D] HHT: state velocities
    double* Fn;               // [B][D] HHT: generalised force at t_n
    double* an;               // [B][D] HHT: accelerations at t_n
    double* x0;               // [B][D] spring rest pose (kBodyInit writes it when non-null)
    const double* Minv;       // [D][D] inverse of the free-DoF mass matrix, zero rows / columns at locked DoFs
    const double* pto_c;      // [B][D] or null
    const double* pto_k;      // [B][D] or null
    double* energy;           // [B][D] or null: += c v v dt with the evaluation velocity
    double* rec_pose;         // [B][D] or null: state after this step
    double* rec_vel;
    double g[3];
    double mass[kMaxBodies];
    double dt;
    unsigned long long free_mask;   // bit i: DoF i is free
    int B, N, D;
    int keep_q;               // kBodyInit: keep q of an instance whose Cardan angles equal the given ones bit for bit
};
cudaError_t launch_body_step(const BodyStepArgs& a, int mode, cudaStream_t st);

// ---- device-side stepping with prismatic joints and translational spring-dampers (k_body_step_linked) ----
// The same modes, slots and ping-pong pairs as k_body_step (the BodyStepArgs fields keep their meaning; Minv is unused).
// Per instance and step: generalised force (hydro, gravity, per-DoF PTO, spring-dampers), T and the bias from the
// evaluation state, (T^T M T) qdd = T^T (rhs - M bias) by partial-pivot elimination, a = bias + T qdd, the scheme's
// update and the projection of every child onto its joint.
constexpr int kMaxLinkTsda = 16;          // HC_SIM_MAX_TSDA
constexpr int kLinkAsmJoint = 10;         // per joint: offset in the parent frame [3], relative rotation [4], axis in the parent frame [3]
constexpr int kLinkAsmTsda = 7;           // per spring-damper: body-frame points [3] + [3], rest length
struct LinkStepArgs {
    BodyStepArgs s;
    const double* M;          // [D][D] diag(m, I) + A_inf over every DoF
    double* asm_data;         // [B][n_pr kLinkAsmJoint + n_tsda kLinkAsmTsda] assembly data (kBodyInit derives it)
    const double* end_pose;   // [B][D] kBodyInit with keep_asm: the pose the previous linked call ended in
    const double* tsda_c;     // [B][n_tsda] or null
    const double* tsda_k;     // [B][n_tsda] or null
    double* tsda_energy;      // [B][n_tsda] or null: += c ldot ldot dt with the evaluation state's ldot
    int n_pr, n_tsda, nq;
    int keep_asm;             // kBodyInit: keep the assembly data of an instance whose pose equals end_pose bit for bit
    int parent_of[kMaxBodies];        // -2: root body, -1: child of ground, else the parent's index
    int joint_of[kMaxBodies];         // index of the joint whose child the body is, or -1
    int pr_child[kMaxBodies], pr_parent[kMaxBodies];
    double pr_axis[kMaxBodies][3];    // unit axis, world frame at assembly
    int ts_b1[kMaxLinkTsda], ts_b2[kMaxLinkTsda];
    double ts_p1[kMaxLinkTsda][3], ts_p2[kMaxLinkTsda][3], ts_rest[kMaxLinkTsda];
    signed char col_body[6 * kMaxBodies], col_dof[6 * kMaxBodies];   // column c of T: a root DoF (body, 0..5) or a slide (child, 6)
};
// Dynamic shared memory of one CTA of `threads` instances: M plus the per-instance scratch.
size_t link_step_smem(int D, int nq, int threads);
int link_step_threads(int D, int nq);
cudaError_t launch_body_step_linked(const LinkStepArgs& a, int mode, cudaStream_t st);

}  // namespace hc
