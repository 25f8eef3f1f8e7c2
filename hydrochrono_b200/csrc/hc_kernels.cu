// CUDA kernels of the per-step hydrodynamic force path (sm_100a, FP64).
//
//   k_prestep     appends the step's velocities to the device-resident history ring and builds the
//                 instance-independent interpolation plans (bracket + weights per lag) for the radiation
//                 and excitation convolutions            src/hydro_forces.cpp:559-577,601-610,343-381
//                                                        src/wave_types.cpp:796-829
//   k_radiation   batched radiation-damping convolution over the velocity history
//                                                        src/hydro_forces.cpp:586-647
//   k_excitation  batched excitation-IRF convolution over the precomputed free-surface elevation
//                                                        src/wave_types.cpp:552-570,776-844
//   k_rad_block<D> / k_step<D>      radiation look-ahead: the resident history rows' share of the next 8 m steps in
//                 one pass on the FP64 tensor cores (DMMA m8n8k4), and the per-step kernel that completes a step
//                 served that way (append, partial sums, rows appended since the snapshot, finalize)
//   k_la_brackets / k_la_taps / k_exc_block(_mma)<ND>   excitation look-ahead: the wave force of the next 8 predicted
//                 step times in one pass over eta (state-independent, wave_types.cpp:776-844)
//   k_finalize    reduces the lag-chunk partials in fixed order, adds hydrostatics and regular-wave
//                 excitation, forms total = hydrostatic - radiation + waves
//                                                        src/hydro_forces.cpp:263-322,758-760; src/wave_types.cpp:315-327
//   k_radiation<D, true> / k_excitation<ND, true> / k_finalize_warp   the same three for a small ensemble's one-graph
//                 step (the drop-in B = 1 TestHydro): convolution CTAs plan their own lags / taps and append the sample
//                 (no k_prestep level); a warp, not a thread, per (dof, instance) in the finalize
//   k_eta         free-surface elevation synthesis for every realisation
//                                                        src/wave_types.cpp:14-59,717-769
//   k_wave_kinematics  elevation, particle velocity and acceleration at given points for every instance (off the step
//                 path)                                  src/wave_types.cpp:14-160,301-313,515-550
//   k_added_mass_mv  R += c * M * w, batched             src/chloadaddedmass.cpp:55-71
//
// Layout: lanes <-> instances.  History ring hist[slot][dof][instance] and eta[sample][instance] are
// instance-innermost, so a warp reads one contiguous 512-byte segment per (row, dof).  Convolution kernels
// (K / f*w tiles) are staged per CTA in shared memory with a TMA bulk copy and broadcast to all lanes.
#include "hc_kernels.cuh"
#include <cstdlib>

namespace hc {

// ------------------------------------------------------------------------------------------
// small PTX helpers: mbarrier + 1-D TMA bulk copy (global -> shared)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// ------------------------------------------------------------------------------------------
// k_prestep
// ------------------------------------------------------------------------------------------

// Bracket + weights of radiation lag s at the step described by h (hydro_forces.cpp:601-610,343-381).  History index
// i (0 = newest) lives in ring slot (head - i) mod cap; entry 0 is this step (time h.t: its slot may still be on its way
// into the ring, so it is taken from the header).
struct RadLagPlan { int slot_new, slot_old, lead; double wn, wo, wd, head_w; };
__device__ __forceinline__ RadLagPlan plan_radiation_lag(const StepHeader& h, const double* __restrict__ times,
                                                         const double* __restrict__ rirf_t,
                                                         const double* __restrict__ rirf_w, const int s) {
    auto hist_time = [&](int i) -> double {
        if (i == 0) return h.t;
        int sl = h.head - i;
        if (sl < 0) sl += h.cap;
        return times[sl];
    };
    RadLagPlan r{0, 0, 0, 0.0, 0.0, 0.0, 0.0};
    if (h.len <= 1) return r;
    const double q = h.t - rirf_t[s];                            // rirf_query_time, :601
    // AdvanceToBracket (:374-381): smallest i with time(i+1) <= q, i+1 < len
    const double t_oldest = hist_time(h.len - 1);
    if (!(t_oldest <= q)) return r;
    // The answer is unique for monotone times, so any search finds the same index.  Near-uniform steps: guess it
    // from the mean step and walk a few entries (2 dependent loads instead of 13); otherwise bisect.
    int lo = 0, hi = h.len - 2;                                  // answer in [lo, hi]
    bool found = false;
    const double dt_mean = (h.t - t_oldest) / (double)(h.len - 1);
    if (dt_mean > 0.0) {
        int i = (int)ceil((h.t - q) / dt_mean) - 1;
        i = max(0, min(i, h.len - 2));
        int probes = 0;
        while (i > 0 && probes < 4 && hist_time(i) <= q) { --i; ++probes; }
        while (i < h.len - 2 && probes < 8 && hist_time(i + 1) > q) { ++i; ++probes; }
        if (hist_time(i + 1) <= q && (i == 0 || hist_time(i) > q)) { lo = i; found = true; }
    }
    if (!found) {
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (hist_time(mid + 1) <= q) hi = mid; else lo = mid + 1;
        }
    }
    const double newer = hist_time(lo), older = hist_time(lo + 1);
    // InterpolateVelocity6D (:343-371)
    double wn = 0.0, wo = 0.0;
    if (q == older) { wo = 1.0; wn = 0.0; }
    else if (q == newer) { wn = 1.0; wo = 0.0; }
    else if (q > older && q < newer) {
        const double delta = newer - older;
        wo = (delta != 0.0) ? ((newer - q) / delta) : 0.0;
        wn = 1.0 - wo;
        if (h.snap > 0.0) {                                      // optional near-exact-hit snapping
            if (wo <= h.snap) { wo = 0.0; wn = 1.0; }
            else if (wn <= h.snap) { wn = 0.0; wo = 1.0; }
        }
    } else return r;                                             // cannot happen for monotone times
    r.wd = rirf_w[s];                                            // step_width == 0 -> skipped (:622-625)
    r.slot_new = h.head - lo; if (r.slot_new < 0) r.slot_new += h.cap;
    r.slot_old = h.head - lo - 1; if (r.slot_old < 0) r.slot_old += h.cap;
    r.wn = wn; r.wo = wo;
    if (lo == 0) {
        // The newer bracket sample is THIS step's velocity, which may still be on its way to the device: its share
        // (K w)[s] * (wn * v_now)  is added by k_finalize, the convolution kernel only sees the older sample.
        // (lags with lo == 0 are the leading lags)
        r.lead = 1;
        r.head_w = wn;
        r.wn = 0.0;
    }
    return r;
}

// Bracket of excitation tap j (wave_types.cpp:796-829): largest i with eta_t[i] <= t - tau_j; exact hit or lerp.
struct ExcTapPlan { int idx; double w1, w2; };
__device__ __forceinline__ ExcTapPlan plan_excitation_tap(const double t, const double* __restrict__ tau,
                                                          const double* __restrict__ eta_t, const int n_eta,
                                                          const double eta_dt, const int j) {
    const double tt = t - tau[j];
    int i = (int)floor((tt - eta_t[0]) / eta_dt);
    i = max(0, min(i, n_eta - 1));
    while (i > 0 && eta_t[i] > tt) --i;
    while (i + 1 < n_eta && eta_t[i + 1] <= tt) ++i;
    ExcTapPlan r{i, 1.0, 0.0};
    const double t1 = eta_t[i];
    if (tt != t1 && i + 1 < n_eta) {
        const double t2 = eta_t[i + 1];
        r.w1 = (t2 - tt) / (t2 - t1);
        r.w2 = 1.0 - r.w1;
    }
    return r;
}

// mode bit 0: history append (needs the step's velocities); bit 1: interpolation plans (need the header only).
__global__ void __launch_bounds__(256) k_prestep(const PrestepArgs a, const int mode) {
    const StepHeader h = *a.hdr;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;

    // (1) history append: hist[head][c][b] = vel[b][c]   (hydro_forces.cpp:560-574)
    if (mode & 1) {
        double* row = a.hist + (size_t)h.head * a.D * a.Bp;
        const int n = a.D * a.Bp;
        for (int i = tid; i < n; i += nth) {
            const int c = i / a.Bp, b = i - c * a.Bp;
            row[i] = (b < a.B) ? h.vel[(size_t)b * a.D + c] : 0.0;
        }
        if (tid == 0) a.times[h.head] = h.t;
    }
    if (!(mode & 2)) return;

    // (2) radiation plan
    for (int s = tid; s < a.L; s += nth) {
        const RadLagPlan r = plan_radiation_lag(h, a.times, a.rirf_t, a.rirf_w, s);
        a.pr_new[s] = r.slot_new; a.pr_old[s] = r.slot_old;
        a.pr_wn[s] = r.wn; a.pr_wo[s] = r.wo; a.pr_wd[s] = r.wd;
        a.pr_head[s] = r.head_w;
        a.pr_lead[s] = r.lead;
    }

    // (3) excitation plan
    for (int g = 0; g < a.ngroups; ++g) {
        for (int j = tid; j < a.Le[g]; j += nth) {
            const ExcTapPlan r = plan_excitation_tap(h.t, a.tau[g], a.eta_t, a.n_eta, a.eta_dt, j);
            a.pe_idx[g][j] = r.idx; a.pe_w1[g][j] = r.w1; a.pe_w2[g][j] = r.w2;
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_radiation<D>: one CTA = kTileInst instances x one lag chunk.  acc[ipt][row] over all D columns.
// ------------------------------------------------------------------------------------------
struct RadPlanPtrs {
    const int* nw; const int* od; const double* wn; const double* wo; const double* wd;
    // INLINE only: what k_finalize needs of the plan (leading lags), and the real instance count for the append
    double* out_wd; double* out_head; int* out_lead; int B;
};

// INLINE (the compact graph of a small ensemble, where every kernel level costs as much as the kernel): each CTA plans
// the lags of its own chunk instead of reading k_prestep's arrays, and the CTAs of chunk 0 append the step's sample to
// the history (no kernel of the step reads that row) -- the step then has no k_prestep level at all.
template <int D, bool INLINE = false>
__global__ void __launch_bounds__(kThreads, (D <= 12) ? 2 : 1) k_radiation(const RadiationArgs a, const RadPlanPtrs p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int s0 = blockIdx.y * a.chunk;
    const int ns = min(a.chunk, a.L - s0);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);               // 16 bytes reserved
    double* Ks = reinterpret_cast<double*>(smem_raw + 16);               // [chunk][D(col)][D(row)]
    double* s_wn = Ks + (size_t)a.chunk * D * D;
    double* s_wo = s_wn + a.chunk;
    double* s_wd = s_wo + a.chunk;
    int* s_new = reinterpret_cast<int*>(s_wd + a.chunk);
    int* s_old = s_new + a.chunk;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)ns * D * D * sizeof(double);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(Ks, a.K + (size_t)s0 * D * D, bytes, bar);
    }
    if constexpr (INLINE) {
        const StepHeader h = *a.hdr;
        for (int i = threadIdx.x; i < ns; i += blockDim.x) {
            const RadLagPlan r = plan_radiation_lag(h, a.times, a.rirf_t, a.rirf_w, s0 + i);
            s_wn[i] = r.wn; s_wo[i] = r.wo; s_wd[i] = r.wd; s_new[i] = r.slot_new; s_old[i] = r.slot_old;
            if (blockIdx.x == 0) { p.out_wd[s0 + i] = r.wd; p.out_head[s0 + i] = r.head_w; p.out_lead[s0 + i] = r.lead; }
        }
        if (blockIdx.y == 0) {                                   // append (hydro_forces.cpp:560-574)
            double* row = const_cast<double*>(a.hist) + (size_t)h.head * D * a.Bp;
            const int bt = blockIdx.x * kTileInst;
            for (int i = threadIdx.x; i < D * kTileInst; i += blockDim.x) {
                const int c = i / kTileInst, b = bt + (i - c * kTileInst);
                if (b < a.Bp) row[(size_t)c * a.Bp + b] = (b < p.B) ? h.vel[(size_t)b * D + c] : 0.0;
            }
            if (blockIdx.x == 0 && threadIdx.x == 0) const_cast<double*>(a.times)[h.head] = h.t;
        }
    } else {
        for (int i = threadIdx.x; i < ns; i += blockDim.x) {
            s_wn[i] = p.wn[s0 + i]; s_wo[i] = p.wo[s0 + i]; s_wd[i] = p.wd[s0 + i];
            s_new[i] = p.nw[s0 + i]; s_old[i] = p.od[s0 + i];
        }
    }
    __syncthreads();
    mbar_wait(bar, 0);

    const int b0 = (blockIdx.x * kThreads + threadIdx.x) * kIPT;
    double acc0[D], acc1[D];
#pragma unroll
    for (int r = 0; r < D; ++r) { acc0[r] = 0.0; acc1[r] = 0.0; }
    const size_t row_stride = (size_t)D * a.Bp;

    if (b0 < a.Bp) {
        for (int s = 0; s < ns; ++s) {
            const double wd = s_wd[s];
            if (wd == 0.0) continue;
            const double wn = s_wn[s], wo = s_wo[s];
            if (wn == 0.0 && wo == 0.0) continue;          // exact hit on this step's own sample: k_finalize's share
            const double* rn = a.hist + (size_t)s_new[s] * row_stride + b0;
            const double* ro = a.hist + (size_t)s_old[s] * row_stride + b0;
            double2 v[D];
            if (wo == 0.0 && wn == 1.0) {                  // exact hit on the newer sample
#pragma unroll
                for (int c = 0; c < D; ++c) v[c] = __ldg(reinterpret_cast<const double2*>(rn + (size_t)c * a.Bp));
            } else if (wn == 0.0 && wo == 1.0) {           // exact hit on the older sample
#pragma unroll
                for (int c = 0; c < D; ++c) v[c] = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
            } else if (wn == 0.0) {                        // lerp whose newer sample is this step's: older share only
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    v[c] = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
                    v[c].x = __dmul_rn(wo, v[c].x); v[c].y = __dmul_rn(wo, v[c].y);
                }
            } else {
                double2 u[D];
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    u[c] = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
                    v[c] = __ldg(reinterpret_cast<const double2*>(rn + (size_t)c * a.Bp));
                }
#pragma unroll
                for (int c = 0; c < D; ++c) {   // weight_older*older + weight_newer*newer, unfused as on the host
                    v[c].x = __dadd_rn(__dmul_rn(wo, u[c].x), __dmul_rn(wn, v[c].x));
                    v[c].y = __dadd_rn(__dmul_rn(wo, u[c].y), __dmul_rn(wn, v[c].y));
                }
            }
            const double* kk = Ks + (size_t)s * D * D;
#pragma unroll
            for (int c = 0; c < D; ++c) {
                // the trapezoid width w[s] is folded into the staged kernel (K * w, see hc_ensemble_create):
                // K * (v * w) becomes (K * w) * v -- one rounding moved, 24 FP64 multiplies per lag saved
                const double sx = v[c].x, sy = v[c].y;
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    const double k = kk[c * D + r];
                    acc0[r] = fma(k, sx, acc0[r]);
                    acc1[r] = fma(k, sy, acc1[r]);
                }
            }
        }
        double* out = a.partial + (size_t)blockIdx.y * row_stride + b0;
#pragma unroll
        for (int r = 0; r < D; ++r)
            *reinterpret_cast<double2*>(out + (size_t)r * a.Bp) = make_double2(acc0[r], acc1[r]);
    }
}

// ------------------------------------------------------------------------------------------
// k_radiation_mma12: the same convolution for D = 12 on the FP64 tensor cores (DMMA, mma.sync m8n8k4.f64).
// Per lag the update  F[r][b] += sum_c (K w)[r][c] v[c][b]  is a (16 x 12) x (12 x 64) product per warp: A = the
// kernel block padded to 16 rows (2 M-tiles x 3 k-steps, stored in shared memory in fragment order so that every
// lane reads its element with one conflict-free LDS.64), B = the bracketing history row(s) (4 DoF x 8 instances per
// fragment; one 16-byte load per lane feeds two N-tiles: even / odd instances), C = 2 x 8 accumulator tiles.
// On B200 the DMMA path delivers the FP64 peak at ~45 % less dynamic power than the DFMA pipe
// (profiles/microbench/fp64_pipes.cu), which matters because the step runs at the board's power cap.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, const double a, const double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

constexpr int kMmaFragDoubles = 2 * 3 * 32;     // per lag: 2 M-tiles x 3 k-steps x 32 lanes

__global__ void __launch_bounds__(kThreads, 2) k_radiation_mma12(const RadiationArgs a, const RadPlanPtrs p) {
    constexpr int D = 12;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int s0 = blockIdx.y * a.chunk;
    const int ns = min(a.chunk, a.L - s0);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    double* Kf = reinterpret_cast<double*>(smem_raw + 16);               // [chunk][2][3][32]
    double* s_wn = Kf + (size_t)a.chunk * kMmaFragDoubles;
    double* s_wo = s_wn + a.chunk;
    double* s_wd = s_wo + a.chunk;
    int* s_new = reinterpret_cast<int*>(s_wd + a.chunk);
    int* s_old = s_new + a.chunk;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)ns * kMmaFragDoubles * sizeof(double);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(Kf, a.Kfrag + (size_t)s0 * kMmaFragDoubles, bytes, bar);
    }
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
        s_wn[i] = p.wn[s0 + i]; s_wo[i] = p.wo[s0 + i]; s_wd[i] = p.wd[s0 + i];
        s_new[i] = p.nw[s0 + i]; s_old[i] = p.od[s0 + i];
    }
    __syncthreads();
    mbar_wait(bar, 0);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int b0w = (blockIdx.x * (kThreads / 32) + warp) * 64;          // 64 instances per warp
    if (b0w >= a.Bp) return;
    const size_t row_stride = (size_t)D * a.Bp;
    // lane's element of a B fragment: DoF (k-step * 4 + q), instances b0w + ig * 16 + 2 g + {0, 1}
    const size_t lane_off = (size_t)q * a.Bp + b0w + 2 * g;

    double C[2][4][2][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int ig = 0; ig < 4; ++ig) { C[mt][ig][0][0] = C[mt][ig][0][1] = C[mt][ig][1][0] = C[mt][ig][1][1] = 0.0; }

    for (int s = 0; s < ns; ++s) {
        if (s_wd[s] == 0.0) continue;
        const double wn = s_wn[s], wo = s_wo[s];
        if (wn == 0.0 && wo == 0.0) continue;              // exact hit on this step's own sample: k_finalize's share
        const double* rn = a.hist + (size_t)s_new[s] * row_stride + lane_off;
        const double* ro = a.hist + (size_t)s_old[s] * row_stride + lane_off;
        double2 v[3][4];
        if (wo == 0.0 && wn == 1.0) {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                for (int ig = 0; ig < 4; ++ig)
                    v[ks][ig] = __ldg(reinterpret_cast<const double2*>(rn + (size_t)(ks * 4) * a.Bp + ig * 16));
        } else if (wn == 0.0) {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                for (int ig = 0; ig < 4; ++ig)
                    v[ks][ig] = __ldg(reinterpret_cast<const double2*>(ro + (size_t)(ks * 4) * a.Bp + ig * 16));
            if (wo != 1.0) {                               // lerp whose newer sample is this step's: older share only
#pragma unroll
                for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                    for (int ig = 0; ig < 4; ++ig) {
                        v[ks][ig].x = __dmul_rn(wo, v[ks][ig].x); v[ks][ig].y = __dmul_rn(wo, v[ks][ig].y);
                    }
            }
        } else {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks) {
#pragma unroll
                for (int ig = 0; ig < 4; ++ig) {
                    const double2 u = __ldg(reinterpret_cast<const double2*>(ro + (size_t)(ks * 4) * a.Bp + ig * 16));
                    const double2 w = __ldg(reinterpret_cast<const double2*>(rn + (size_t)(ks * 4) * a.Bp + ig * 16));
                    // weight_older*older + weight_newer*newer, unfused as on the host
                    v[ks][ig].x = __dadd_rn(__dmul_rn(wo, u.x), __dmul_rn(wn, w.x));
                    v[ks][ig].y = __dadd_rn(__dmul_rn(wo, u.y), __dmul_rn(wn, w.y));
                }
            }
        }
        const double* kf = Kf + (size_t)s * kMmaFragDoubles + lane;
#pragma unroll
        for (int ks = 0; ks < 3; ++ks) {
            const double a0 = kf[(0 * 3 + ks) * 32], a1 = kf[(1 * 3 + ks) * 32];
#pragma unroll
            for (int ig = 0; ig < 4; ++ig) {
                dmma8x8x4(C[0][ig][0][0], C[0][ig][0][1], a0, v[ks][ig].x);
                dmma8x8x4(C[0][ig][1][0], C[0][ig][1][1], a0, v[ks][ig].y);
                dmma8x8x4(C[1][ig][0][0], C[1][ig][0][1], a1, v[ks][ig].x);
                dmma8x8x4(C[1][ig][1][0], C[1][ig][1][1], a1, v[ks][ig].y);
            }
        }
    }
    // C[mt][ig][par][i]: row mt*8 + g, instance b0w + ig*16 + 2*(2q + i) + par  ->  4 consecutive instances per lane
    double* out = a.partial + (size_t)blockIdx.y * row_stride + b0w + 4 * q;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int r = mt * 8 + g;
        if (r < D) {
#pragma unroll
            for (int ig = 0; ig < 4; ++ig) {
                double* o = out + (size_t)r * a.Bp + ig * 16;
                *reinterpret_cast<double2*>(o) = make_double2(C[mt][ig][0][0], C[mt][ig][1][0]);
                *reinterpret_cast<double2*>(o + 2) = make_double2(C[mt][ig][0][1], C[mt][ig][1][1]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_radiation_hybrid12: D = 12 on BOTH FP64 engines at once.  Rows 0..7 of F form one full DMMA M-tile (no padding):
// 24 DMMA per warp and lag on the tensor cores; rows 8..11 would waste half a tile, so they run on the FMA pipe from
// the same B-fragment registers: every lane holds 3 of the 12 velocity DoF (k-step * 4 + q) for 8 instances, forms
// its partial dot products (96 DFMA per lag) and the four lanes of a quad are summed once per CTA with shuffles.
// Per warp and lag: 384 tensor-pipe cycles || 192 FMA-pipe cycles per SM sub-partition instead of 576 FMA-pipe cycles,
// at a third of the DFMA count (the step runs at the board's power cap).
// Shared memory per lag (144 doubles, as the FMA-pipe kernel): [3][32] A fragments of rows 0..7, then
// [q 0..3][k-step 0..2][row 8..11] for the FMA part.
// ------------------------------------------------------------------------------------------
constexpr int kHybThreads = 128;
__global__ void __launch_bounds__(kHybThreads, 3) k_radiation_hybrid12(const RadiationArgs a, const RadPlanPtrs p) {
    constexpr int D = 12, kLag = 144;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int s0 = blockIdx.y * a.chunk;
    const int ns = min(a.chunk, a.L - s0);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    double* Kh = reinterpret_cast<double*>(smem_raw + 16);               // [chunk][144]
    double* s_wn = Kh + (size_t)a.chunk * kLag;
    double* s_wo = s_wn + a.chunk;
    double* s_wd = s_wo + a.chunk;
    int* s_new = reinterpret_cast<int*>(s_wd + a.chunk);
    int* s_old = s_new + a.chunk;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)ns * kLag * sizeof(double);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(Kh, a.Khyb + (size_t)s0 * kLag, bytes, bar);
    }
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
        s_wn[i] = p.wn[s0 + i]; s_wo[i] = p.wo[s0 + i]; s_wd[i] = p.wd[s0 + i];
        s_new[i] = p.nw[s0 + i]; s_old[i] = p.od[s0 + i];
    }
    __syncthreads();
    mbar_wait(bar, 0);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int b0w = (blockIdx.x * (kHybThreads / 32) + warp) * 64;       // 64 instances per warp
    if (b0w >= a.Bp) return;
    const size_t row_stride = (size_t)D * a.Bp;
    const size_t lane_off = (size_t)q * a.Bp + b0w + 2 * g;

    double C0[4][2][2];        // tensor part: rows 0..7
    double acc[4][4][2];       // FMA part: [row 8 + r][instance group][parity], partial over this lane's 3 DoF
#pragma unroll
    for (int ig = 0; ig < 4; ++ig) {
        C0[ig][0][0] = C0[ig][0][1] = C0[ig][1][0] = C0[ig][1][1] = 0.0;
#pragma unroll
        for (int r = 0; r < 4; ++r) { acc[r][ig][0] = 0.0; acc[r][ig][1] = 0.0; }
    }

    for (int s = 0; s < ns; ++s) {
        if (s_wd[s] == 0.0) continue;
        const double wn = s_wn[s], wo = s_wo[s];
        if (wn == 0.0 && wo == 0.0) continue;
        const double* rn = a.hist + (size_t)s_new[s] * row_stride + lane_off;
        const double* ro = a.hist + (size_t)s_old[s] * row_stride + lane_off;
        double2 v[3][4];
        if (wo == 0.0 && wn == 1.0) {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                for (int ig = 0; ig < 4; ++ig)
                    v[ks][ig] = __ldg(reinterpret_cast<const double2*>(rn + (size_t)(ks * 4) * a.Bp + ig * 16));
        } else if (wn == 0.0) {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                for (int ig = 0; ig < 4; ++ig)
                    v[ks][ig] = __ldg(reinterpret_cast<const double2*>(ro + (size_t)(ks * 4) * a.Bp + ig * 16));
            if (wo != 1.0) {
#pragma unroll
                for (int ks = 0; ks < 3; ++ks)
#pragma unroll
                    for (int ig = 0; ig < 4; ++ig) {
                        v[ks][ig].x = __dmul_rn(wo, v[ks][ig].x); v[ks][ig].y = __dmul_rn(wo, v[ks][ig].y);
                    }
            }
        } else {
#pragma unroll
            for (int ks = 0; ks < 3; ++ks) {
#pragma unroll
                for (int ig = 0; ig < 4; ++ig) {
                    const double2 u = __ldg(reinterpret_cast<const double2*>(ro + (size_t)(ks * 4) * a.Bp + ig * 16));
                    const double2 w = __ldg(reinterpret_cast<const double2*>(rn + (size_t)(ks * 4) * a.Bp + ig * 16));
                    v[ks][ig].x = __dadd_rn(__dmul_rn(wo, u.x), __dmul_rn(wn, w.x));
                    v[ks][ig].y = __dadd_rn(__dmul_rn(wo, u.y), __dmul_rn(wn, w.y));
                }
            }
        }
        const double* kl = Kh + (size_t)s * kLag;
        const double2* kq = reinterpret_cast<const double2*>(kl + 96 + q * 12);     // [k-step][row 8..11]
#pragma unroll
        for (int ks = 0; ks < 3; ++ks) {
            const double a0 = kl[ks * 32 + lane];
            const double2 k01 = kq[ks * 2], k23 = kq[ks * 2 + 1];
#pragma unroll
            for (int ig = 0; ig < 4; ++ig) {
                dmma8x8x4(C0[ig][0][0], C0[ig][0][1], a0, v[ks][ig].x);
                dmma8x8x4(C0[ig][1][0], C0[ig][1][1], a0, v[ks][ig].y);
                acc[0][ig][0] = fma(k01.x, v[ks][ig].x, acc[0][ig][0]); acc[0][ig][1] = fma(k01.x, v[ks][ig].y, acc[0][ig][1]);
                acc[1][ig][0] = fma(k01.y, v[ks][ig].x, acc[1][ig][0]); acc[1][ig][1] = fma(k01.y, v[ks][ig].y, acc[1][ig][1]);
                acc[2][ig][0] = fma(k23.x, v[ks][ig].x, acc[2][ig][0]); acc[2][ig][1] = fma(k23.x, v[ks][ig].y, acc[2][ig][1]);
                acc[3][ig][0] = fma(k23.y, v[ks][ig].x, acc[3][ig][0]); acc[3][ig][1] = fma(k23.y, v[ks][ig].y, acc[3][ig][1]);
            }
        }
    }
    double* base = a.partial + (size_t)blockIdx.y * row_stride + b0w;
    // rows 0..7 from the accumulator tiles: row g, 4 consecutive instances per lane
#pragma unroll
    for (int ig = 0; ig < 4; ++ig) {
        double* o = base + (size_t)g * a.Bp + ig * 16 + 4 * q;
        *reinterpret_cast<double2*>(o) = make_double2(C0[ig][0][0], C0[ig][1][0]);
        *reinterpret_cast<double2*>(o + 2) = make_double2(C0[ig][0][1], C0[ig][1][1]);
    }
    // rows 8..11: sum the quad's partial dot products, lane q of the quad stores row 8 + q
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int ig = 0; ig < 4; ++ig)
#pragma unroll
            for (int par = 0; par < 2; ++par) {
                double x = acc[r][ig][par];
                x += __shfl_xor_sync(0xffffffffu, x, 1);
                x += __shfl_xor_sync(0xffffffffu, x, 2);
                acc[r][ig][par] = x;
            }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (q == r) {
#pragma unroll
            for (int ig = 0; ig < 4; ++ig)
                *reinterpret_cast<double2*>(base + (size_t)(8 + r) * a.Bp + ig * 16 + 2 * g) =
                    make_double2(acc[r][ig][0], acc[r][ig][1]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Radiation look-ahead (D = 6, 12, 18).  When the step times are predictable (t, t + dt, ...) and every lag of every
// step lands exactly on one history row -- lag s on row m s, m = RIRF lag spacing / dt an integer; the host verifies
// this per step with the same bracket arithmetic as k_prestep, see hc_ensemble::rb_step_plan -- the steps j = rho + m g
// (g = 0..7) of a block of 8 m steps all read the resident rows r = m u + (m - 1 - rho), and
//     F_j = sum_{u >= 0} (K w)[u + g + 1] v_res[m u + m - 1 - rho]     (rows resident at the snapshot, r = 0 newest)
//         + sum_{l <= j / m} (K w)[l] v_young[j - m l]                  (rows appended since the snapshot)
// (j counts steps from the snapshot of the history the block works on; a block evaluated one block ahead has
// j = 8 m + its own step index, i.e. g runs over 8..15: RadBlockArgs::g0)
// k_rad_block<D> evaluates the first sum for all 8 m steps in ONE pass over the history (work item = instance tile x
// row chunk x residue class rho; a pass can be launched in slices of consecutive items): per row and warp a
// (8 D x D) x (D x 16) product on the FP64 tensor cores.  M-tile d = the 8 steps of force row d:
// A[g][c] = (K w)[u + g + 1][d][c], read from a shared-memory tile of R + 7 lags with one conflict-free LDS.64 per
// fragment (lag stride = 4 mod 16 doubles, columns padded to a multiple of 4 with zeros); B = the history row, one
// 16-byte load per lane and k-step feeding two N-tiles.  HBM traffic per step falls to 1/8 of the per-step kernel's;
// the kernel is bound by the FP64 tensor pipe.
// k_step<D> (phase 2 of every step served by a block) appends the step's velocities, sums the row-chunk partials in
// fixed order, adds the second sum (at most 16 rows) and finishes the step like k_finalize.
// ------------------------------------------------------------------------------------------
// (D = 6: one lag of slack -- the pair loop's predicated-off read of the second row's A in an odd last iteration may be
//  issued speculatively one lag past the R + 7 the bulk copy fills)
size_t rad_block_smem_bytes(int D, int R) {
    return 16 + size_t(R + kRbT - 1 + (D == 6 ? 1 : 0)) * rb_stride(D) * sizeof(double);
}

template <int D>
__global__ void __launch_bounds__(128, (D <= 12) ? 3 : 2) k_rad_block(const RadBlockArgs a) {
    constexpr int KS = (D + 3) / 4, DP = 4 * KS, STRIDE = rb_stride(D);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    const double* Ks = reinterpret_cast<const double*>(smem_raw + 16);
    const int tiles = (a.Bp + kRbTileInst - 1) / kRbTileInst;
    const int item = a.item0 + blockIdx.x;
    const int tile = item % tiles, rest = item / tiles;
    const int chunk = rest % a.nchunk_used, rho = rest / a.nchunk_used;
    const int off = a.m - 1 - rho;                            // first resident row of this residue class
    const int nu = a.n_res > off ? (a.n_res - off + a.m - 1) / a.m : 0;
    const int r0 = chunk * a.R;                               // first u of this chunk
    const int nr = min(a.R, nu - r0);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)(a.R + kRbT - 1) * STRIDE * sizeof(double);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(const_cast<double*>(Ks), a.Kpad + (size_t)(r0 + 1 + a.g0) * STRIDE, bytes, bar);
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int b0 = tile * kRbTileInst + warp * 16;
    const bool active = b0 < a.Bp;
    // row u feeds step rho + m g iff its lag u + g + 1 has a bracket at that step
    const int rmax_g = __ldg(a.smax + rho + a.m * g) - (g + a.g0) - 1;
    int rmax_min = rmax_g;
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) rmax_min = min(rmax_min, __shfl_xor_sync(0xffffffffu, rmax_min, o));

    double C[D][2][2];
#pragma unroll
    for (int d = 0; d < D; ++d) { C[d][0][0] = C[d][0][1] = C[d][1][0] = C[d][1][1] = 0.0; }

    const size_t row_stride = (size_t)D * a.Bp;
    const double* hl = a.hist + (active ? b0 + 2 * g : 0);
    auto load_row = [&](int u, double2* dst) {
        int slot = (a.head0 - 1 - off - a.m * u) % a.cap;
        if (slot < 0) slot += a.cap;
        const double* p = hl + (size_t)slot * row_stride;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            const int c = min(ks * 4 + q, D - 1);            // padded columns: any finite value (their A is zero)
            dst[ks] = __ldg(reinterpret_cast<const double2*>(p + (size_t)c * a.Bp));
        }
    };
    if constexpr (D == 6) {
        // Single body: 6 columns would pad to 2 k-steps of 4 (a quarter of the DMMAs multiplying zeros).  Two consecutive
        // rows are 12 columns = 3 exact k-steps: k-step 0 = row u, columns 0-3; k-step 1 = columns 4-5 of rows u and
        // u + 1; k-step 2 = row u + 1, columns 0-3 (any split of the K dimension is a valid product; A keeps its tile
        // layout -- in k-step 1 lanes (g, e = 1) and (g + 1, e = 0) read the same word, the rest distinct banks but for
        // one 2-way overlap per half warp).  An odd last row runs with the second row's A zeroed.
        auto slot_of = [&](int u) {
            int slot = (a.head0 - 1 - off - a.m * u) % a.cap;
            return slot < 0 ? slot + a.cap : slot;
        };
        const int e1 = q >> 1;                                   // k-step 1: which row of the pair this lane's column is in
        auto load_pair = [&](int u, bool two, double2* dst) {
            const double* p0 = hl + (size_t)slot_of(u) * row_stride;
            const double* p1 = two ? hl + (size_t)slot_of(u + 1) * row_stride : p0;
            dst[0] = __ldg(reinterpret_cast<const double2*>(p0 + (size_t)q * a.Bp));
            dst[1] = __ldg(reinterpret_cast<const double2*>((e1 ? p1 : p0) + (size_t)(4 + (q & 1)) * a.Bp));
            dst[2] = __ldg(reinterpret_cast<const double2*>(p1 + (size_t)q * a.Bp));
        };
        double2 cur[3], nxt[3];
        if (active && nr > 0) load_pair(r0, nr > 1, cur);
        mbar_wait(bar, 0);
        if (active) {
            const double* kl = Ks + (size_t)g * STRIDE;
            for (int i = 0; i < nr; i += 2) {
                const int r = r0 + i;
                const bool two = i + 1 < nr;
                if (i + 2 < nr) load_pair(r + 2, i + 3 < nr, nxt);
                const double* kr = kl + (size_t)i * STRIDE;      // lag (r + g0 + g + 1) = tile lag i + g
                const bool on0 = r <= rmax_g, on1 = two && (r + 1 <= rmax_g);
                const bool onm = e1 ? on1 : on0;
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const double a0 = on0 ? kr[d * DP + q] : 0.0;
                    const double a1 = onm ? kr[(size_t)e1 * STRIDE + d * DP + 4 + (q & 1)] : 0.0;
                    const double a2 = on1 ? kr[STRIDE + d * DP + q] : 0.0;
                    dmma8x8x4(C[d][0][0], C[d][0][1], a0, cur[0].x);
                    dmma8x8x4(C[d][1][0], C[d][1][1], a0, cur[0].y);
                    dmma8x8x4(C[d][0][0], C[d][0][1], a1, cur[1].x);
                    dmma8x8x4(C[d][1][0], C[d][1][1], a1, cur[1].y);
                    dmma8x8x4(C[d][0][0], C[d][0][1], a2, cur[2].x);
                    dmma8x8x4(C[d][1][0], C[d][1][1], a2, cur[2].y);
                }
#pragma unroll
                for (int ks = 0; ks < 3; ++ks) cur[ks] = nxt[ks];
            }
#pragma unroll
            for (int d = 0; d < D; ++d) {
                double* o = a.partial + (((size_t)(rho + a.m * g) * a.nchunk + chunk) * D + d) * a.Bp + b0 + 4 * q;
                *reinterpret_cast<double2*>(o) = make_double2(C[d][0][0], C[d][1][0]);
                *reinterpret_cast<double2*>(o + 2) = make_double2(C[d][0][1], C[d][1][1]);
            }
        }
        return;
    }
    double2 cur[KS], nxt[KS];
    if (active && nr > 0) load_row(r0, cur);
    mbar_wait(bar, 0);
    if (active) {
        const double* kl = Ks + (size_t)g * STRIDE + q;
        for (int i = 0; i < nr; ++i) {
            const int r = r0 + i;
            if (i + 1 < nr) load_row(r + 1, nxt);
            const double* kr = kl + (size_t)i * STRIDE;          // lag (r + g0 + g + 1) = tile lag i + g
            if (r <= rmax_min) {
#pragma unroll
                for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                    for (int d = 0; d < D; ++d) {
                        const double av = kr[d * DP + ks * 4];
                        dmma8x8x4(C[d][0][0], C[d][0][1], av, cur[ks].x);
                        dmma8x8x4(C[d][1][0], C[d][1][1], av, cur[ks].y);
                    }
            } else {
                const bool on = r <= rmax_g;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                    for (int d = 0; d < D; ++d) {
                        const double av = on ? kr[d * DP + ks * 4] : 0.0;
                        dmma8x8x4(C[d][0][0], C[d][0][1], av, cur[ks].x);
                        dmma8x8x4(C[d][1][0], C[d][1][1], av, cur[ks].y);
                    }
            }
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) cur[ks] = nxt[ks];
        }
        // C[d][par][e]: step j = rho + m g, force row d, instance b0 + 2 (2 q + e) + par
#pragma unroll
        for (int d = 0; d < D; ++d) {
            double* o = a.partial + (((size_t)(rho + a.m * g) * a.nchunk + chunk) * D + d) * a.Bp + b0 + 4 * q;
            *reinterpret_cast<double2*>(o) = make_double2(C[d][0][0], C[d][1][0]);
            *reinterpret_cast<double2*>(o + 2) = make_double2(C[d][0][1], C[d][1][1]);
        }
    }
}

// k_step<D>: phase 2 of a step served by the radiation look-ahead in ONE kernel (append, block partials + young rows,
// then hydrostatics, waves and the total as k_finalize).  One CTA = 32 instances x D DoF; thread (b, d).
constexpr int kRsInst = 32;
struct FinalizeArgs;
__device__ __forceinline__ double finalize_one(const FinalizeArgs& a, const HydrostaticTables& hs, const FinalizeGroups& eg,
                                               const StepHeader& h, const int d, const int b, const bool have_fr,
                                               const double fr_block, const double* pose6,
                                               const double* fr_part_pre = nullptr, const double* fw_pre = nullptr,
                                               const bool write = true);

template <int D>
__global__ void __launch_bounds__(kRsInst * D, (D == 12) ? 4 : 1) k_step(const RadStepArgs a, const __grid_constant__ FinalizeArgs fa,
                                                      const __grid_constant__ HydrostaticTables hs,
                                                      const __grid_constant__ FinalizeGroups eg,
                                                      const __grid_constant__ StepHeader h) {
    constexpr int LAGS = (D <= 12) ? 8 : 4;          // young lags staged per pass
    __shared__ double s_K[LAGS * D * D];             // (K w)[lag][col][row]
    __shared__ double s_v[LAGS][D][kRsInst];         // young rows, [lag][col][instance]
    __shared__ double s_io[kRsInst][D];              // the CTA's tile of pose (in), then of the totals (out)
    const int j = h.rb_j;
    const int nl = min(min(h.rb_jj / a.m, h.rb_smax), a.L - 1) + 1;   // young lags 0 .. nl - 1
    const int tid = threadIdx.x;
    const int bl = tid % kRsInst, d = tid / kRsInst;
    const int b0 = blockIdx.x * kRsInst;
    const int b = b0 + bl;
    const size_t row_stride = (size_t)D * a.Bp;
    // the CTA's [32][D] tile of pose is contiguous: one coalesced read, every value fetched once (finalize_one reads the
    // 6 pose values of its body from shared memory instead of 6 x from global for each of the body's 6 DoF threads)
    {
        const int lb = tid / D, c = tid - lb * D;
        s_io[lb][c] = (b0 + lb < a.B) ? h.pose[(size_t)(b0 + lb) * D + c] : 0.0;
    }
    // Everything this thread will read later (row-chunk partials, look-ahead wave-force segments)
    // is requested from DRAM now, so that the dependent sums below find it in L2: one DRAM round trip instead of ~10.
    {
        const double* p = a.partial[h.rb_buf] + ((size_t)j * a.nchunk * D + d) * a.Bp + b;
        for (int ch = 0; ch < h.rb_nchunk; ++ch) prefetch_l2(p + (size_t)ch * row_stride);
        if (fa.wave_mode == 2 && h.exc_src == 1) {
            const int buf = h.exc_slot / kLaT, pos = h.exc_slot - buf * kLaT;
            const double* e = fa.exc_cache + (((size_t)buf * fa.exc_S * kLaT + pos) * D + d) * a.Bp + b;
            for (int sg = 0; sg < fa.exc_S; ++sg) prefetch_l2(e + (size_t)sg * kLaT * D * a.Bp);
        }
        // ... and the rows appended since the block's snapshot (lags 1 .. nl - 1; lag 0 is this step's own sample)
        for (int l = 1; l < nl; ++l) {
            int slot = (h.head - a.m * l) % h.cap;
            if (slot < 0) slot += h.cap;
            prefetch_l2(a.hist + (size_t)slot * row_stride + (size_t)d * a.Bp + b);
        }
    }
    // fixed-order sum of the row-chunk partials of block step j
    double fr = 0.0;
    {
        const double* p = a.partial[h.rb_buf] + ((size_t)j * a.nchunk * D + d) * a.Bp + b;
        int ch = 0;
        for (; ch + 8 <= h.rb_nchunk; ch += 8) {              // 8 independent loads in flight, summed in order
            double v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldg(p + (size_t)(ch + i) * row_stride);
#pragma unroll
            for (int i = 0; i < 8; ++i) fr = __dadd_rn(fr, v[i]);
        }
        for (; ch + 4 <= h.rb_nchunk; ch += 4) {
            const double p0 = p[(size_t)ch * row_stride], p1 = p[(size_t)(ch + 1) * row_stride];
            const double p2 = p[(size_t)(ch + 2) * row_stride], p3 = p[(size_t)(ch + 3) * row_stride];
            fr = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(fr, p0), p1), p2), p3);
        }
        for (; ch < h.rb_nchunk; ++ch) fr = __dadd_rn(fr, p[(size_t)ch * row_stride]);
    }
    for (int l0 = ((nl - 1) / LAGS) * LAGS; l0 >= 0; l0 -= LAGS) {     // oldest lag group first
        const int n = min(LAGS, nl - l0);
        __syncthreads();
        for (int i = tid; i < n * D * D; i += blockDim.x) s_K[i] = a.K[(size_t)l0 * D * D + i];
        for (int l = 0; l < n; ++l) {
            if (l0 + l == 0) {
                // this step's sample: the CTA's [32][D] tile of vel is contiguous
                const int lb = tid / D, c = tid - lb * D;
                s_v[0][c][lb] = (b0 + lb < a.B) ? h.vel[(size_t)(b0 + lb) * D + c] : 0.0;
            } else {                                               // lag l: the row appended m l steps ago
                int slot = (h.head - a.m * (l0 + l)) % h.cap;
                if (slot < 0) slot += h.cap;
                s_v[l][d][bl] = a.hist[(size_t)slot * row_stride + (size_t)d * a.Bp + b];
            }
        }
        __syncthreads();
        if (l0 == 0) {
            a.hist[(size_t)h.head * row_stride + (size_t)d * a.Bp + b] = s_v[0][d][bl];
            if (blockIdx.x == 0 && tid == 0) a.times[h.head] = h.t;
        }
        for (int l = n - 1; l >= 0; --l) {
            double acc = 0.0;
#pragma unroll
            for (int c = 0; c < D; ++c) acc = fma(s_K[(l * D + c) * D + d], s_v[l][c][bl], acc);
            fr = __dadd_rn(fr, acc);
        }
    }
    // (the loop above ran at least once, so s_io is visible to every thread)
    const double total = (b < a.B) ? finalize_one(fa, hs, eg, h, d, b, true, fr, &s_io[bl][6 * (d / 6)]) : 0.0;
    if (h.force2) {      // second copy of the totals (the caller's buffer): coalesced tile
        __syncthreads();
        s_io[bl][d] = total;
        __syncthreads();
        const int lb = tid / D, c = tid - lb * D;
        if (b0 + lb < a.B) h.force2[(size_t)(b0 + lb) * D + c] = s_io[lb][c];
    }
}

// k_step2<D>: the same step kernel with a fatter thread -- a CTA of 256 threads serves 64 instances x D DoF, every
// thread 3 (instance, DoF) items (D = 12).  k_step is bound by a chain of dependent memory round trips, not by work, so
// its cost to the step is the CTA slots it holds while waiting (slots the look-ahead passes' tensor CTAs would use):
// three items per thread put three times the loads in flight per slot, and the CTA (256 x <= 80 registers, 64 KB of
// shared memory) fits the slot one retiring k_rad_block CTA frees.  Arithmetic and summation order per item are k_step's.
constexpr int kRs2Inst = 64, kRs2Threads = 256;
template <int D>
__global__ void __launch_bounds__(kRs2Threads, 3) k_step2(const RadStepArgs a, const __grid_constant__ FinalizeArgs fa,
                                                          const __grid_constant__ HydrostaticTables hs,
                                                          const __grid_constant__ FinalizeGroups eg,
                                                          const __grid_constant__ StepHeader h) {
    constexpr int LAGS = 8;
    constexpr int IPT = kRs2Inst * D / kRs2Threads;  // items per thread
    static_assert(kRs2Inst * D % kRs2Threads == 0, "items must divide evenly");
    extern __shared__ __align__(16) unsigned char smem2_raw[];      // 63 KB: dynamic (above the 48 KB static limit)
    double* const s_K = reinterpret_cast<double*>(smem2_raw);                                     // (K w)[lag][col][row]
    double (*s_v)[D][kRs2Inst] = reinterpret_cast<double (*)[D][kRs2Inst]>(s_K + LAGS * D * D);    // young rows [lag][col][inst]
    double (*s_io)[D] = reinterpret_cast<double (*)[D]>(s_K + LAGS * D * D + LAGS * D * kRs2Inst); // pose tile in, totals out
    const int j = h.rb_j;
    const int nl = min(min(h.rb_jj / a.m, h.rb_smax), a.L - 1) + 1;   // young lags 0 .. nl - 1
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * kRs2Inst;
    const size_t row_stride = (size_t)D * a.Bp;
    int bl[IPT], dd[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) { const int it = tid + k * kRs2Threads; bl[k] = it % kRs2Inst; dd[k] = it / kRs2Inst; }
    // pose tile [64][D], contiguous
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const int it = tid + k * kRs2Threads, lb = it / D, c = it - lb * D;
        s_io[lb][c] = (b0 + lb < a.B) ? h.pose[(size_t)(b0 + lb) * D + c] : 0.0;
    }
    // request everything the sums below will read
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const int b = b0 + bl[k], d = dd[k];
        const double* p = a.partial[h.rb_buf] + ((size_t)j * a.nchunk * D + d) * a.Bp + b;
        for (int ch = 0; ch < h.rb_nchunk; ++ch) prefetch_l2(p + (size_t)ch * row_stride);
        if (fa.wave_mode == 2 && h.exc_src == 1) {
            const int buf = h.exc_slot / kLaT, pos = h.exc_slot - buf * kLaT;
            const double* e = fa.exc_cache + (((size_t)buf * fa.exc_S * kLaT + pos) * D + d) * a.Bp + b;
            for (int sg = 0; sg < fa.exc_S; ++sg) prefetch_l2(e + (size_t)sg * kLaT * D * a.Bp);
        }
        for (int l = 1; l < nl; ++l) {
            int slot = (h.head - a.m * l) % h.cap;
            if (slot < 0) slot += h.cap;
            prefetch_l2(a.hist + (size_t)slot * row_stride + (size_t)d * a.Bp + b);
        }
    }
    // fixed-order sum of the row-chunk partials of block step j, the IPT items interleaved
    double fr[IPT];
    const double* pp[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        fr[k] = 0.0;
        pp[k] = a.partial[h.rb_buf] + ((size_t)j * a.nchunk * D + dd[k]) * a.Bp + b0 + bl[k];
    }
    {
        int ch = 0;
        for (; ch + 4 <= h.rb_nchunk; ch += 4) {
            double v[IPT][4];
#pragma unroll
            for (int k = 0; k < IPT; ++k)
#pragma unroll
                for (int i = 0; i < 4; ++i) v[k][i] = __ldg(pp[k] + (size_t)(ch + i) * row_stride);
#pragma unroll
            for (int k = 0; k < IPT; ++k)
#pragma unroll
                for (int i = 0; i < 4; ++i) fr[k] = __dadd_rn(fr[k], v[k][i]);
        }
        for (; ch < h.rb_nchunk; ++ch)
#pragma unroll
            for (int k = 0; k < IPT; ++k) fr[k] = __dadd_rn(fr[k], __ldg(pp[k] + (size_t)ch * row_stride));
    }
    for (int l0 = ((nl - 1) / LAGS) * LAGS; l0 >= 0; l0 -= LAGS) {     // oldest lag group first
        const int n = min(LAGS, nl - l0);
        __syncthreads();
        for (int i = tid; i < n * D * D; i += kRs2Threads) s_K[i] = a.K[(size_t)l0 * D * D + i];
        for (int l = 0; l < n; ++l) {
            if (l0 + l == 0) {
#pragma unroll
                for (int k = 0; k < IPT; ++k) {     // this step's sample: the CTA's [64][D] tile of vel is contiguous
                    const int it = tid + k * kRs2Threads, lb = it / D, c = it - lb * D;
                    s_v[0][c][lb] = (b0 + lb < a.B) ? h.vel[(size_t)(b0 + lb) * D + c] : 0.0;
                }
            } else {                                               // lag l: the row appended m l steps ago
                int slot = (h.head - a.m * (l0 + l)) % h.cap;
                if (slot < 0) slot += h.cap;
#pragma unroll
                for (int k = 0; k < IPT; ++k)
                    s_v[l][dd[k]][bl[k]] = a.hist[(size_t)slot * row_stride + (size_t)dd[k] * a.Bp + b0 + bl[k]];
            }
        }
        __syncthreads();
        if (l0 == 0) {
#pragma unroll
            for (int k = 0; k < IPT; ++k)
                a.hist[(size_t)h.head * row_stride + (size_t)dd[k] * a.Bp + b0 + bl[k]] = s_v[0][dd[k]][bl[k]];
            if (blockIdx.x == 0 && tid == 0) a.times[h.head] = h.t;
        }
        for (int l = n - 1; l >= 0; --l) {
#pragma unroll
            for (int k = 0; k < IPT; ++k) {
                double acc = 0.0;
#pragma unroll
                for (int c = 0; c < D; ++c) acc = fma(s_K[(l * D + c) * D + dd[k]], s_v[l][c][bl[k]], acc);
                fr[k] = __dadd_rn(fr[k], acc);
            }
        }
    }
    double total[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const int b = b0 + bl[k];
        total[k] = (b < a.B) ? finalize_one(fa, hs, eg, h, dd[k], b, true, fr[k], &s_io[bl[k]][6 * (dd[k] / 6)]) : 0.0;
    }
    if (h.force2) {      // second copy of the totals (the caller's buffer): coalesced tile
        __syncthreads();
#pragma unroll
        for (int k = 0; k < IPT; ++k) s_io[bl[k]][dd[k]] = total[k];
        __syncthreads();
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int it = tid + k * kRs2Threads, lb = it / D, c = it - lb * D;
            if (b0 + lb < a.B) h.force2[(size_t)(b0 + lb) * D + c] = s_io[lb][c];
        }
    }
}

template <int D>
static cudaError_t launch_rad_block_t(const RadBlockArgs& a, int nitems, cudaStream_t st) {
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(k_rad_block<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    if (nitems <= 0) return cudaSuccess;
    k_rad_block<D><<<nitems, 128, rad_block_smem_bytes(D, a.R), st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_rad_block(const RadBlockArgs& a, int nitems, cudaStream_t st) {
    switch (a.D) {
        case 6: return launch_rad_block_t<6>(a, nitems, st);
        case 12: return launch_rad_block_t<12>(a, nitems, st);
        case 18: return launch_rad_block_t<18>(a, nitems, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_step(const RadStepArgs& a, const FinalizeArgs& fa, const HydrostaticTables& hs, const FinalizeGroups& eg,
                        const StepHeader& hdr, cudaStream_t st) {
    // 34 KB of static shared memory per CTA: ask for the large carve-out so that 4 CTAs of k_step<12> fit per SM and
    // the 512 CTAs of a 16384-instance ensemble run as a single wave
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaFuncSetAttribute(k_step<6>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(k_step<12>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(k_step<18>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        attr_set[dev & 63] = true;
    }
    static int use2 = -1;
    if (use2 < 0) { const char* v = std::getenv("HC_KSTEP2"); use2 = (v && std::atoi(v) == 0) ? 0 : 1; }   // default on
    // k_step2 pays where the step is throughput-bound (its CTAs compete with tensor CTAs for slots); a small ensemble's
    // step is k_step's own latency chain, which three sequential items per thread only lengthen (8 x 2048 instances:
    // 0.046 vs 0.041 ms per step)
    if (use2 && a.D == 12 && a.Bp % kRs2Inst == 0 && a.Bp / kRs2Inst >= 148) {
        constexpr size_t smem2 = sizeof(double) * (8 * 12 * 12 + 8 * 12 * kRs2Inst + kRs2Inst * 12);
        static bool attr2[64] = {};
        if (!attr2[dev & 63]) {
            cudaFuncSetAttribute(k_step2<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
            cudaFuncSetAttribute(k_step2<12>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            attr2[dev & 63] = true;
        }
        k_step2<12><<<a.Bp / kRs2Inst, kRs2Threads, smem2, st>>>(a, fa, hs, eg, hdr);
        return cudaGetLastError();
    }
    switch (a.D) {
        case 6: k_step<6><<<a.Bp / kRsInst, kRsInst * 6, 0, st>>>(a, fa, hs, eg, hdr); break;
        case 12: k_step<12><<<a.Bp / kRsInst, kRsInst * 12, 0, st>>>(a, fa, hs, eg, hdr); break;
        case 18: k_step<18><<<a.Bp / kRsInst, kRsInst * 18, 0, st>>>(a, fa, hs, eg, hdr); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// Generic fallback for large body counts: D at run time, 6 rows (one body) per z-slice, K read from global/L2.
__global__ void __launch_bounds__(kThreads) k_radiation_generic(const RadiationArgs a, const RadPlanPtrs p) {
    const int s0 = blockIdx.y * a.chunk;
    const int ns = min(a.chunk, a.L - s0);
    const int r0 = blockIdx.z * 6;
    const int D = a.D;
    const int b0 = (blockIdx.x * kThreads + threadIdx.x) * kIPT;
    if (b0 >= a.Bp) return;
    double acc0[6] = {0, 0, 0, 0, 0, 0}, acc1[6] = {0, 0, 0, 0, 0, 0};
    const size_t row_stride = (size_t)D * a.Bp;
    for (int s = 0; s < ns; ++s) {
        const double wd = p.wd[s0 + s];
        if (wd == 0.0) continue;
        const double wn = p.wn[s0 + s], wo = p.wo[s0 + s];
        if (wn == 0.0 && wo == 0.0) continue;
        const double* rn = a.hist + (size_t)p.nw[s0 + s] * row_stride + b0;
        const double* ro = a.hist + (size_t)p.od[s0 + s] * row_stride + b0;
        const double* kk = a.K + (size_t)(s0 + s) * D * D;
        for (int c = 0; c < D; ++c) {
            double2 v;
            if (wo == 0.0 && wn == 1.0) v = __ldg(reinterpret_cast<const double2*>(rn + (size_t)c * a.Bp));
            else if (wn == 0.0 && wo == 1.0) v = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
            else if (wn == 0.0) {
                v = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
                v.x = __dmul_rn(wo, v.x); v.y = __dmul_rn(wo, v.y);
            } else {
                const double2 u = __ldg(reinterpret_cast<const double2*>(ro + (size_t)c * a.Bp));
                v = __ldg(reinterpret_cast<const double2*>(rn + (size_t)c * a.Bp));
                v.x = __dadd_rn(__dmul_rn(wo, u.x), __dmul_rn(wn, v.x));
                v.y = __dadd_rn(__dmul_rn(wo, u.y), __dmul_rn(wn, v.y));
            }
            const double sx = v.x, sy = v.y;   // width folded into the staged kernel
#pragma unroll
            for (int r = 0; r < 6; ++r) {
                const double k = __ldg(kk + c * D + r0 + r);
                acc0[r] = fma(k, sx, acc0[r]);
                acc1[r] = fma(k, sy, acc1[r]);
            }
        }
    }
    double* out = a.partial + (size_t)blockIdx.y * row_stride + b0;
#pragma unroll
    for (int r = 0; r < 6; ++r)
        *reinterpret_cast<double2*>(out + (size_t)(r0 + r) * a.Bp) = make_double2(acc0[r], acc1[r]);
}

// ------------------------------------------------------------------------------------------
// k_excitation<ND>: one CTA = kTileInst instances x one lag chunk of one IRF group.
// ------------------------------------------------------------------------------------------
struct ExcPlanPtrs { const int* idx; const double* w1; const double* w2; };

template <int ND, bool INLINE = false>     // INLINE: the CTA plans its own taps (compact graph, see k_radiation)
__global__ void __launch_bounds__(kThreads, 2) k_excitation(const ExcitationArgs a, const ExcGroup g, const ExcPlanPtrs p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int j0 = blockIdx.y * a.chunk;
    const int nj = min(a.chunk, g.Le - j0);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);               // 16 bytes reserved
    double* Fs = reinterpret_cast<double*>(smem_raw + 16);               // [chunk][ND]
    double* s_w1 = Fs + (size_t)a.chunk * ND;
    double* s_w2 = s_w1 + a.chunk;
    int* s_idx = reinterpret_cast<int*>(s_w2 + a.chunk);

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)nj * ND * sizeof(double);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(Fs, g.fw + (size_t)j0 * ND, bytes, bar);
    }
    if constexpr (INLINE) {
        const double t = a.hdr->t;
        for (int i = threadIdx.x; i < nj; i += blockDim.x) {
            const ExcTapPlan r = plan_excitation_tap(t, g.tau, a.eta_t, a.n_eta, a.eta_dt, j0 + i);
            s_w1[i] = r.w1; s_w2[i] = r.w2; s_idx[i] = r.idx;
        }
    } else {
        for (int i = threadIdx.x; i < nj; i += blockDim.x) {
            s_w1[i] = p.w1[j0 + i]; s_w2[i] = p.w2[j0 + i]; s_idx[i] = p.idx[j0 + i];
        }
    }
    __syncthreads();
    mbar_wait(bar, 0);

    const int b0 = (blockIdx.x * kThreads + threadIdx.x) * kIPT;
    if (b0 >= a.Bp) return;
    double acc0[ND], acc1[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) { acc0[d] = 0.0; acc1[d] = 0.0; }

    int prev_idx = -2;
    double2 prev_e = make_double2(0.0, 0.0);
    const double* eta_b = a.eta + b0;
    // One lag = one eta row (16 B per thread).  kExcUnroll independent row loads are issued before the first
    // dependent FMA so that every warp keeps several 512-byte requests in flight (the kernel is latency-bound
    // otherwise: one request per warp at a time).
    constexpr int U = 8;
    int j = 0;
    for (; j + U <= nj; j += U) {
        int idx[U];
        double2 e1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            idx[u] = s_idx[j + u];
            e1[u] = __ldg(reinterpret_cast<const double2*>(eta_b + (size_t)idx[u] * a.Bp));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double w1 = s_w1[j + u], w2 = s_w2[j + u];
            double2 ev = e1[u];
            if (w2 != 0.0) {
                // eta row idx+1 is the row the previous lag interpolated from in the common case
                const double2 e2 = (idx[u] + 1 == prev_idx)
                                       ? prev_e
                                       : __ldg(reinterpret_cast<const double2*>(eta_b + (size_t)(idx[u] + 1) * a.Bp));
                ev.x = __dadd_rn(__dmul_rn(w1, e1[u].x), __dmul_rn(w2, e2.x));   // w1*eta1 + w2*eta2 (:821-824)
                ev.y = __dadd_rn(__dmul_rn(w1, e1[u].y), __dmul_rn(w2, e2.y));
            }
            prev_idx = idx[u]; prev_e = e1[u];
            const double* ff = Fs + (size_t)(j + u) * ND;
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                const double f = ff[d];
                acc0[d] = fma(f, ev.x, acc0[d]);
                acc1[d] = fma(f, ev.y, acc1[d]);
            }
        }
    }
    for (; j < nj; ++j) {
        const int idx = s_idx[j];
        const double w1 = s_w1[j], w2 = s_w2[j];
        const double2 e1 = __ldg(reinterpret_cast<const double2*>(eta_b + (size_t)idx * a.Bp));
        double2 ev = e1;
        if (w2 != 0.0) {
            const double2 e2 = (idx + 1 == prev_idx)
                                   ? prev_e
                                   : __ldg(reinterpret_cast<const double2*>(eta_b + (size_t)(idx + 1) * a.Bp));
            ev.x = __dadd_rn(__dmul_rn(w1, e1.x), __dmul_rn(w2, e2.x));
            ev.y = __dadd_rn(__dmul_rn(w1, e1.y), __dmul_rn(w2, e2.y));
        }
        prev_idx = idx; prev_e = e1;
        const double* ff = Fs + (size_t)j * ND;
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            const double f = ff[d];
            acc0[d] = fma(f, ev.x, acc0[d]);
            acc1[d] = fma(f, ev.y, acc1[d]);
        }
    }
    double* out = a.partial + ((size_t)(g.chunk0 + blockIdx.y) * a.ndmax) * a.Bp + b0;
#pragma unroll
    for (int d = 0; d < ND; ++d) *reinterpret_cast<double2*>(out + (size_t)d * a.Bp) = make_double2(acc0[d], acc1[d]);
}

// ------------------------------------------------------------------------------------------
// Excitation look-ahead.  The wave force does not depend on the body state, so it may be evaluated ahead of
// time for the (predicted) times of the next kLaT steps: one pass over the eta window then serves kLaT steps and
// the eta traffic per step drops by kLaT.  Per block time i and lag j the bracket (idx, w1, w2) is exactly the
// per-step plan; the lerp is folded into per-row taps
//     F_i[d] = sum_j fw[j][d] (w1 eta[idx] + w2 eta[idx+1]) = sum_rows G_i[row][d] eta[row],
//     G_i[row][d] = sum_{j: idx_ij = row} fw[j][d] w1_ij + sum_{j: idx_ij = row-1} fw[j][d] w2_ij   (ascending j).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_la_brackets(const LookaheadPlanArgs a) {
    const int n = a.T * a.Le;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const int i = q / a.Le, j = q - i * a.Le;
        const double tt = a.times[i] - a.tau[j];
        int r = (int)floor((tt - a.eta_t[0]) / a.eta_dt);
        r = max(0, min(r, a.n_eta - 1));
        while (r > 0 && a.eta_t[r] > tt) --r;
        while (r + 1 < a.n_eta && a.eta_t[r + 1] <= tt) ++r;
        double w1 = 1.0, w2 = 0.0;
        const double t1 = a.eta_t[r];
        if (tt != t1 && r + 1 < a.n_eta) {
            const double t2 = a.eta_t[r + 1];
            w1 = (t2 - tt) / (t2 - t1);
            w2 = 1.0 - w1;
        }
        a.idx[q] = r; a.w1[q] = w1; a.w2[q] = w2;
    }
}

__global__ void __launch_bounds__(256) k_la_taps(const LookaheadPlanArgs a) {
    // one thread per (block time i, eta row m); idx[i][.] is non-increasing in j
    const int nchunk = (a.nrows + kLaRows - 1) / kLaRows;
    const int n = a.T * nchunk * kLaRows;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const int i = q / (nchunk * kLaRows), mr = q - i * nchunk * kLaRows;
        const int row = a.row0 + mr;
        const int* idx = a.idx + (size_t)i * a.Le;
        // first j with idx[j] <= row, first j with idx[j] <= row - 1, first j with idx[j] <= row - 2
        auto first_le = [&](int v) {
            int lo = 0, hi = a.Le;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (idx[mid] <= v) hi = mid; else lo = mid + 1; }
            return lo;
        };
        const int j0 = first_le(row), j1 = first_le(row - 1), j2 = first_le(row - 2);
        const int chunk = mr / kLaRows, rr = mr - chunk * kLaRows;
        double* out = a.taps + (((size_t)chunk * a.T + i) * kLaRows + rr) * a.nd;
        for (int d = 0; d < a.nd; ++d) {
            if (a.frag_order) {
                // DMMA A-fragment order: [chunk][k-step = rr/4][M-tile][lane]; A row m = (block time i, dof d),
                // A column = eta row within the k-step; lane = (m % 8) * 4 + rr % 4
                const int m = i * a.nd + d, mtiles = a.T * a.nd / 8;
                out = a.taps + ((((size_t)chunk * (kLaRows / 4) + rr / 4) * mtiles + m / 8) * 32 + (m % 8) * 4 + (rr & 3)) - d;
            }
            double g = 0.0;
            if (mr < a.nrows) {
                for (int j = j0; j < j1; ++j)        // idx == row: weight of the lower bracket sample
                    g = __dadd_rn(g, __dmul_rn(a.fw[(size_t)j * a.nd + d], a.w1[(size_t)i * a.Le + j]));
                for (int j = j1; j < j2; ++j)        // idx == row - 1: weight of the upper bracket sample
                    g = __dadd_rn(g, __dmul_rn(a.fw[(size_t)j * a.nd + d], a.w2[(size_t)i * a.Le + j]));
            }
            out[d] = g;
        }
    }
}

template <int ND>
__global__ void __launch_bounds__(kLaT * 32, 2) k_exc_block(const LookaheadArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);                 // 2 mbarriers (16 bytes)
    constexpr int kStageDoubles = kLaT * kLaRows * ND;
    double* const stage0 = reinterpret_cast<double*>(smem_raw + 16);        // two stages, back to back
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b0 = (blockIdx.x * 32 + lane) * kIPT;
    constexpr uint32_t kStageBytes = kStageDoubles * sizeof(double);

    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_expect_tx(&bars[0], kStageBytes);
        bulk_g2s(stage0, a.taps, kStageBytes, &bars[0]);
    }
    __syncthreads();

    double acc0[ND], acc1[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) { acc0[d] = 0.0; acc1[d] = 0.0; }
    const double* eta_b = a.eta + b0;

    for (int c = 0; c < a.nchunk; ++c) {
        const int st = c & 1;
        if (threadIdx.x == 0 && c + 1 < a.nchunk) {      // prefetch the next stage (its readers left it at the
            mbar_expect_tx(&bars[st ^ 1], kStageBytes);  // __syncthreads closing iteration c - 1)
            bulk_g2s(stage0 + (st ^ 1) * kStageDoubles, a.taps + (size_t)(c + 1) * kStageDoubles, kStageBytes,
                     &bars[st ^ 1]);
        }
        mbar_wait(&bars[st], (c >> 1) & 1);
        // (pointer arithmetic on the extern shared array keeps the loads in the shared address space: LDS.128)
        const double2* tp = reinterpret_cast<const double2*>(smem_raw + 16) +
                            ((size_t)st * kStageDoubles + (size_t)warp * kLaRows * ND) / 2;
        const int rbase = a.row0 + c * kLaRows;
        if (b0 < a.Bp) {
            constexpr int U = 8;
#pragma unroll
            for (int r0 = 0; r0 < kLaRows; r0 += U) {
                double2 e[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int row = min(rbase + r0 + u, a.n_eta - 1);       // rows past the window carry zero taps
                    e[u] = __ldg(reinterpret_cast<const double2*>(eta_b + (size_t)row * a.Bp));
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const double2* g = tp + (r0 + u) * (ND / 2);
#pragma unroll
                    for (int d = 0; d < ND; d += 2) {
                        const double2 gd = g[d / 2];
                        acc0[d] = fma(gd.x, e[u].x, acc0[d]);
                        acc1[d] = fma(gd.x, e[u].y, acc1[d]);
                        acc0[d + 1] = fma(gd.y, e[u].x, acc0[d + 1]);
                        acc1[d + 1] = fma(gd.y, e[u].y, acc1[d + 1]);
                    }
                }
            }
        }
        __syncthreads();
    }
    if (b0 < a.Bp) {
        double* out = a.cache + ((size_t)warp * a.D + a.dof0) * a.Bp + b0;
#pragma unroll
        for (int d = 0; d < ND; ++d) *reinterpret_cast<double2*>(out + (size_t)d * a.Bp) = make_double2(acc0[d], acc1[d]);
    }
}

// k_exc_block_mma<ND>: the look-ahead block on the FP64 tensor cores.  M = (block time, dof) = 8 * ND rows = ND
// M-tiles with no padding, N = instances, K = eta rows: per k-step (4 eta rows) a warp issues ND * 2 DMMAs for its 16
// instances from ONE 16-byte eta load per lane and ND conflict-free LDS.64 of taps; eta is read exactly once.
template <int ND>
__global__ void __launch_bounds__(128, 3) k_exc_block_mma(const LookaheadArgs a) {
    constexpr int MT = ND;                                   // kLaT * ND / 8 with kLaT == 8
    constexpr int KS = kLaRows / 4;                          // k-steps per stage
    constexpr int kStageDoubles = KS * MT * 32;
    constexpr uint32_t kStageBytes = kStageDoubles * sizeof(double);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
    double* const stage0 = reinterpret_cast<double*>(smem_raw + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int b0 = (blockIdx.x * 4 + warp) * 16;             // 16 instances per warp
    const bool active = b0 < a.Bp;
    // this CTA's segment of the stages (eta rows): [c0, c1)
    const int seg = a.seg0 + blockIdx.y;
    const int cps = (a.nchunk + a.S - 1) / a.S;
    const int c0 = seg * cps, c1 = min(a.nchunk, c0 + cps);

    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        if (c0 < c1) {
            mbar_expect_tx(&bars[0], kStageBytes);
            bulk_g2s(stage0, a.taps + (size_t)c0 * kStageDoubles, kStageBytes, &bars[0]);
        }
    }
    __syncthreads();

    double C[MT][2][2];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) { C[mt][0][0] = C[mt][0][1] = C[mt][1][0] = C[mt][1][1] = 0.0; }

    // lane's B element: eta row (k-step * 4 + q), instances b0 + 2 g + {0, 1}.  eta is prefetched half a stage
    // (KH k-steps) ahead: 2 x KH registers pairs instead of 2 x KS leave the compiler room to hoist the tap loads.
    constexpr int KH = KS / 2;
    const double* eta_l = a.eta + (active ? b0 + 2 * g : 0);
    auto load_half = [&](int c, int h, double2* dst) {
#pragma unroll
        for (int k = 0; k < KH; ++k) {
            const int row = min(a.row0 + c * kLaRows + (h * KH + k) * 4 + q, a.n_eta - 1);   // past the window: zero taps
            dst[k] = __ldg(reinterpret_cast<const double2*>(eta_l + (size_t)row * a.Bp));
        }
    };
    auto mma_half = [&](const double* tp, int h, const double2* v) {
#pragma unroll
        for (int k = 0; k < KH; ++k) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const double av = tp[((h * KH + k) * MT + mt) * 32];
                dmma8x8x4(C[mt][0][0], C[mt][0][1], av, v[k].x);
                dmma8x8x4(C[mt][1][0], C[mt][1][1], av, v[k].y);
            }
        }
    };
    double2 cur[KH], nxt[KH];
    if (active && c0 < c1) load_half(c0, 0, cur);

    for (int c = c0; c < c1; ++c) {
        const int st = (c - c0) & 1;
        if (threadIdx.x == 0 && c + 1 < c1) {
            mbar_expect_tx(&bars[st ^ 1], kStageBytes);
            bulk_g2s(stage0 + (st ^ 1) * kStageDoubles, a.taps + (size_t)(c + 1) * kStageDoubles, kStageBytes,
                     &bars[st ^ 1]);
        }
        if (active) load_half(c, 1, nxt);                                 // second half of this stage in flight
        mbar_wait(&bars[st], ((c - c0) >> 1) & 1);
        if (active) {
            const double* tp = reinterpret_cast<const double*>(smem_raw + 16) + (size_t)st * kStageDoubles + lane;
            mma_half(tp, 0, cur);
#pragma unroll
            for (int k = 0; k < KH; ++k) cur[k] = nxt[k];
            if (c + 1 < c1) load_half(c + 1, 0, nxt);                     // first half of the next stage in flight
            mma_half(tp, 1, cur);
#pragma unroll
            for (int k = 0; k < KH; ++k) cur[k] = nxt[k];
        }
        __syncthreads();
    }
    if (active) {
        // C[mt][par][e]: A row m = mt*8 + g -> (block time m / ND, dof m % ND); instance b0 + 2*(2q + e) + par
        double* cache = a.cache + (size_t)seg * kLaT * a.D * a.Bp;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            const int m = mt * 8 + g, i = m / ND, d = m - i * ND;
            double* o = cache + ((size_t)i * a.D + a.dof0 + d) * a.Bp + b0 + 4 * q;
            *reinterpret_cast<double2*>(o) = make_double2(C[mt][0][0], C[mt][1][0]);
            *reinterpret_cast<double2*>(o + 2) = make_double2(C[mt][0][1], C[mt][1][1]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_finalize: one thread per instance.
// ------------------------------------------------------------------------------------------

// Force of (dof d, instance b).  fr_block: the radiation force when the caller already holds it (k_step).
// Returns the total; writes it to h.force (and the components to a.comp).  pose6: the 6 pose values of (b, body).
// fr_part_pre / fw_pre: the sum of the radiation lag-chunk partials / the wave force when the caller has already
// reduced them (k_finalize_warp); write: whether this thread stores the results.
__device__ __forceinline__ double finalize_one(const FinalizeArgs& a, const HydrostaticTables& hs, const FinalizeGroups& eg,
                                               const StepHeader& h, const int d, const int b, const bool have_fr,
                                               const double fr_block, const double* pose6, const double* fr_part_pre,
                                               const double* fw_pre, const bool write) {
    const int D = a.D;
    const int body = d / 6, i = d - 6 * body;
    const double gx = h.g[0], gy = h.g[1], gz = h.g[2];
    // ---- hydrostatics (hydro_forces.cpp:263-322), arithmetic order kept, no FMA contraction ----
    // ChVector3::Length(): sqrt(x*x + y*y + z*z)
    const double glen = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(gx, gx), __dmul_rn(gy, gy)), __dmul_rn(gz, gz)));
    const double rho_g = __dmul_rn(hs.rho, glen);
    double fh = 0.0;
    if (!a.waves_only) {
    const double* pose = pose6;
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j)
        s = __dadd_rn(s, __dmul_rn(hs.Kh[body][i * 6 + j], __dsub_rn(pose[j], hs.equilibrium[body][j])));
    fh = __dmul_rn(-rho_g, s);
    const double V = hs.disp_vol[body];
    const double bx = __dmul_rn(__dmul_rn(hs.rho, -gx), V);
    const double by = __dmul_rn(__dmul_rn(hs.rho, -gy), V);
    const double bz = __dmul_rn(__dmul_rn(hs.rho, -gz), V);
    const double rx = hs.cb_minus_cg[body][0], ry = hs.cb_minus_cg[body][1], rz = hs.cb_minus_cg[body][2];
    double add;
    switch (i) {
        case 0: add = bx; break;
        case 1: add = by; break;
        case 2: add = bz; break;
        case 3: add = __dsub_rn(__dmul_rn(ry, bz), __dmul_rn(rz, by)); break;
        case 4: add = __dsub_rn(__dmul_rn(rz, bx), __dmul_rn(rx, bz)); break;
        default: add = __dsub_rn(__dmul_rn(rx, by), __dmul_rn(ry, bx)); break;
    }
    fh = __dadd_rn(fh, add);
    }
    // ---- radiation: fixed-order sum of lag-chunk partials ----
    double fr = 0.0;
    if (!a.waves_only && have_fr) {
        fr = fr_block;                                                   // k_rad_block + this kernel (k_step)
    } else if (!a.waves_only) {
        if (fr_part_pre) {
            fr = *fr_part_pre;
        } else {
            const double* p = a.rad_partial + (size_t)d * a.Bp + b;
            const size_t stride = (size_t)D * a.Bp;
            int ch = 0;
            for (; ch + 4 <= a.rad_nchunk; ch += 4) {
                const double p0 = p[(size_t)ch * stride], p1 = p[(size_t)(ch + 1) * stride];
                const double p2 = p[(size_t)(ch + 2) * stride], p3 = p[(size_t)(ch + 3) * stride];
                fr = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(fr, p0), p1), p2), p3);
            }
            for (; ch < a.rad_nchunk; ++ch) fr = __dadd_rn(fr, p[(size_t)ch * stride]);
        }
        // share of this step's own velocity sample (leading lags whose newer bracket sample is "now")
        const double* vel = h.vel + (size_t)b * D;
        for (int s = 0; s < a.L && a.pr_lead[s]; ++s) {   // leading lags: contiguous from lag 0
            const double hw = a.pr_head[s];
            if (hw == 0.0 || a.pr_wd[s] == 0.0) continue;
            const double* kk = a.K + (size_t)s * D * D + d;            // (K w)[s][c][row d]
            double acc = 0.0;
            for (int c = 0; c < D; ++c) acc = fma(kk[(size_t)c * D], __dmul_rn(hw, vel[c]), acc);
            fr = __dadd_rn(fr, acc);
        }
    }
    // ---- waves ----
    double fw = 0.0;
    if (a.wave_mode == 1) {
        // mag * A * cos(omega t + phase[rowEx])  (wave_types.cpp:322-323; phase of body 0, reference quirk)
        const double arg = __dadd_rn(__dmul_rn(a.reg_omega[b], h.t), a.reg_phase[(size_t)i * a.Bp + b]);
        fw = __dmul_rn(__dmul_rn(a.reg_mag[(size_t)d * a.Bp + b], a.reg_amp[b]), cos(arg));
    } else if (a.wave_mode == 2 && fw_pre) {
        fw = *fw_pre;
    } else if (a.wave_mode == 2 && h.exc_src == 1) {
        // precomputed by k_exc_block(_mma): slot = buffer * T + block step; S row-segment partials in fixed order
        const int buf = h.exc_slot / kLaT, pos = h.exc_slot - buf * kLaT;
        const double* p = a.exc_cache + (((size_t)buf * a.exc_S * kLaT + pos) * D + d) * a.Bp + b;
        const size_t sstride = (size_t)kLaT * D * a.Bp;
        int sg = 0;
        for (; sg + 4 <= a.exc_S; sg += 4) {                     // 4 independent loads in flight, summed in order
            const double p0 = __ldg(p + (size_t)sg * sstride), p1 = __ldg(p + (size_t)(sg + 1) * sstride);
            const double p2 = __ldg(p + (size_t)(sg + 2) * sstride), p3 = __ldg(p + (size_t)(sg + 3) * sstride);
            fw = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(fw, p0), p1), p2), p3);
        }
        for (; sg < a.exc_S; ++sg) fw = __dadd_rn(fw, p[(size_t)sg * sstride]);
    } else if (a.wave_mode == 2) {
        for (int g = 0; g < a.exc_ngroups; ++g) {
            if (d < eg.dof0[g] || d >= eg.dof0[g] + eg.nd[g]) continue;
            const int dl = d - eg.dof0[g];
            const double* p = a.exc_partial + ((size_t)eg.chunk0[g] * a.exc_ndmax + dl) * a.Bp + b;
            const size_t stride = (size_t)a.exc_ndmax * a.Bp;
            int ch = 0;
            for (; ch + 4 <= eg.nchunk[g]; ch += 4) {
                const double p0 = p[(size_t)ch * stride], p1 = p[(size_t)(ch + 1) * stride];
                const double p2 = p[(size_t)(ch + 2) * stride], p3 = p[(size_t)(ch + 3) * stride];
                fw = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(fw, p0), p1), p2), p3);
            }
            for (; ch < eg.nchunk[g]; ++ch) fw = __dadd_rn(fw, p[(size_t)ch * stride]);
        }
    }
    const size_t o = (size_t)b * D + d;
    if (a.waves_only) { if (write) h.force[o] = fw; return fw; }
    const double total = __dadd_rn(__dsub_rn(fh, fr), fw);           // hs - rad + waves (:758-760)
    if (!write) return total;
    h.force[o] = total;
    if (a.comp) {
        const size_t BD = (size_t)a.B * D;
        a.comp[o] = fh;
        a.comp[BD + o] = fr;
        a.comp[2 * BD + o] = fw;
    }
    return total;
}

__global__ void __launch_bounds__(256) k_finalize(const FinalizeArgs a, const __grid_constant__ HydrostaticTables hs,
                                                  const __grid_constant__ FinalizeGroups eg) {
    // one thread per (dof, instance); instances fastest so the partial reads are coalesced
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int d = tid / a.Bp;
    const int b = tid - d * a.Bp;
    if (d >= a.D || b >= a.B) return;
    const StepHeader h = *a.hdr;
    const double total = finalize_one(a, hs, eg, h, d, b, false, 0.0,
                                      a.waves_only ? nullptr : h.pose + (size_t)b * a.D + 6 * (d / 6));
    if (h.force2 && !a.waves_only) h.force2[(size_t)b * a.D + d] = total;
}

// k_finalize_warp<G>: the same for SMALL ensembles (the drop-in B = 1 TestHydro): there the lag / tap chunks are short so
// that the convolution kernels have CTAs to spread over, which leaves hundreds of partials per (dof, instance) -- 251 +
// 286 for the RM3 shape -- and k_finalize's one thread per item sums them as one dependent chain (63 us cold, most of a
// B = 1 step).  Here G lanes share an item: lane-group member `sub` sums partials sub, sub + G, ... in ascending order
// (8 loads in flight), a butterfly of shuffles over the group (symmetric, so every member holds the same bits) adds the
// G sums, then the item is finished as above.  G = 32 (one item per warp) is what is launched.  Deterministic; the
// association differs from k_finalize's, so the results agree to rounding (1e-16 relative), not bitwise -- which kernel
// serves an ensemble depends only on its size.
template <int G>
__device__ __forceinline__ double group_sum_fixed(double v) {
#pragma unroll
    for (int off = 16; off >= 32 / G; off >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

// member's share of n strided partials: entries sub, sub + G, ... in ascending order, eight loads in flight at a time
template <int G>
__device__ __forceinline__ double member_sum_strided(const double* p, const size_t stride, const int n, const int sub,
                                                     const bool live) {
    double s = 0.0;
    if (!live) return s;
    for (int ch = sub; ch < n; ch += 8 * G) {
        double v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = (ch + G * i < n) ? p[(size_t)(ch + G * i) * stride] : 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (ch + G * i < n) s = __dadd_rn(s, v[i]);
    }
    return s;
}

template <int G>
__global__ void __launch_bounds__(256) k_finalize_warp(const FinalizeArgs a, const __grid_constant__ HydrostaticTables hs,
                                                       const __grid_constant__ FinalizeGroups eg) {
    constexpr int IPW = 32 / G;                        // items (consecutive instances of one dof) per warp
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int bi = lane % IPW, sub = lane / IPW;
    const int wpd = (a.B + IPW - 1) / IPW;             // warps per dof
    const int d = w / wpd, b = (w - d * wpd) * IPW + bi;
    if (d >= a.D) return;                              // (uniform per warp)
    const bool live = b < a.B;
    const StepHeader h = *a.hdr;
    const int D = a.D;
    double fr = 0.0, fw = 0.0;
    if (!a.waves_only)
        fr = group_sum_fixed<G>(member_sum_strided<G>(a.rad_partial + (size_t)d * a.Bp + b, (size_t)D * a.Bp, a.rad_nchunk, sub, live));
    if (a.wave_mode == 2 && h.exc_src == 1) {
        const int buf = h.exc_slot / kLaT, pos = h.exc_slot - buf * kLaT;
        const double* p = a.exc_cache + (((size_t)buf * a.exc_S * kLaT + pos) * D + d) * a.Bp + b;
        fw = group_sum_fixed<G>(member_sum_strided<G>(p, (size_t)kLaT * D * a.Bp, a.exc_S, sub, live));
    } else if (a.wave_mode == 2) {
        for (int g = 0; g < a.exc_ngroups; ++g) {
            if (d < eg.dof0[g] || d >= eg.dof0[g] + eg.nd[g]) continue;
            const double* p = a.exc_partial + ((size_t)eg.chunk0[g] * a.exc_ndmax + (d - eg.dof0[g])) * a.Bp + b;
            fw = __dadd_rn(fw, group_sum_fixed<G>(member_sum_strided<G>(p, (size_t)a.exc_ndmax * a.Bp, eg.nchunk[g], sub, live)));
        }
    }
    if (!live) return;
    const double total = finalize_one(a, hs, eg, h, d, b, false, 0.0,
                                      a.waves_only ? nullptr : h.pose + (size_t)b * a.D + 6 * (d / 6), &fr, &fw, sub == 0);
    if (sub == 0 && h.force2 && !a.waves_only) h.force2[(size_t)b * a.D + d] = total;
}

// k_finalize_split<G>: the same for MID-SIZE ensembles on the per-step path (hundreds to a few thousand instances): still
// hundreds of partials per item (143 + 147 at 1024 instances of the RM3 shape: k_finalize 41 us, the longest kernel of
// the step), but enough instances for coalesced rows.  One CTA = 32 consecutive instances of one dof x G warps; warp g
// sums partials g, g + G, ... (8 loads in flight, lanes = instances: whole 256-byte rows), shared memory holds the G
// sums per instance, warp 0 adds them in ascending g and finishes the items.  Deterministic.
template <int G>
__global__ void __launch_bounds__(32 * G) k_finalize_split(const FinalizeArgs a, const __grid_constant__ HydrostaticTables hs,
                                                           const __grid_constant__ FinalizeGroups eg) {
    __shared__ double s_fr[G][32], s_fw[G][32];
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int tiles = (a.B + 31) / 32;
    const int d = blockIdx.x / tiles, b = (blockIdx.x - d * tiles) * 32 + lane;
    const bool live = b < a.B;
    const StepHeader h = *a.hdr;
    const int D = a.D;
    double fr = 0.0, fw = 0.0;
    if (!a.waves_only)
        fr = member_sum_strided<G>(a.rad_partial + (size_t)d * a.Bp + b, (size_t)D * a.Bp, a.rad_nchunk, grp, live);
    if (a.wave_mode == 2 && h.exc_src == 1) {
        const int buf = h.exc_slot / kLaT, pos = h.exc_slot - buf * kLaT;
        const double* p = a.exc_cache + (((size_t)buf * a.exc_S * kLaT + pos) * D + d) * a.Bp + b;
        fw = member_sum_strided<G>(p, (size_t)kLaT * D * a.Bp, a.exc_S, grp, live);
    } else if (a.wave_mode == 2) {
        for (int g = 0; g < a.exc_ngroups; ++g) {
            if (d < eg.dof0[g] || d >= eg.dof0[g] + eg.nd[g]) continue;
            const double* p = a.exc_partial + ((size_t)eg.chunk0[g] * a.exc_ndmax + (d - eg.dof0[g])) * a.Bp + b;
            fw = __dadd_rn(fw, member_sum_strided<G>(p, (size_t)a.exc_ndmax * a.Bp, eg.nchunk[g], grp, live));
        }
    }
    s_fr[grp][lane] = fr; s_fw[grp][lane] = fw;
    __syncthreads();
    if (grp != 0 || !live) return;
    fr = 0.0; fw = 0.0;
#pragma unroll
    for (int g = 0; g < G; ++g) { fr = __dadd_rn(fr, s_fr[g][lane]); fw = __dadd_rn(fw, s_fw[g][lane]); }
    const double total = finalize_one(a, hs, eg, h, d, b, false, 0.0,
                                      a.waves_only ? nullptr : h.pose + (size_t)b * a.D + 6 * (d / 6), &fr, &fw, true);
    if (h.force2 && !a.waves_only) h.force2[(size_t)b * a.D + d] = total;
}

// ------------------------------------------------------------------------------------------
// k_eta: eta[k][b] = sum_i amp_i cos(k_i*0 - omega_i t_k + phase_{b,i}), ramped.  One thread = one instance
// x KT consecutive samples; the sum runs over i in ascending order like the reference's loop.
// ------------------------------------------------------------------------------------------
constexpr int kEtaKT = 4;
__global__ void __launch_bounds__(128) k_eta(const EtaArgs a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int k0 = blockIdx.y * kEtaKT;
    if (b >= a.Bp) return;
    double tk[kEtaKT], acc[kEtaKT];
#pragma unroll
    for (int q = 0; q < kEtaKT; ++q) {
        tk[q] = a.eta_t[min(k0 + q, a.n_eta - 1)];
        acc[q] = 0.0;
    }
    for (int i = 0; i < a.nf; ++i) {
        const double om = a.omega[i];
        const double am = a.amp_per_instance ? a.amp[(size_t)i * a.Bp + b] : a.amp[i];
        const double ph = a.phase[(size_t)i * a.Bp + b];
#pragma unroll
        for (int q = 0; q < kEtaKT; ++q) {
            // wavenumber*x - omega*time + phase with x = 0  ->  (0 - omega*t) + phase, unfused
            const double arg = __dadd_rn(__dsub_rn(0.0, __dmul_rn(om, tk[q])), ph);
            acc[q] = __dadd_rn(acc[q], __dmul_rn(am, cos(arg)));
        }
    }
#pragma unroll
    for (int q = 0; q < kEtaKT; ++q) {
        if (k0 + q >= a.n_eta) break;
        double e = acc[q];
        if (a.ramp > 0.0 && tk[q] < a.ramp) {                            // wave_types.cpp:759-769
            if (tk[q] <= 0.0) e = __dmul_rn(e, 0.0);
            else e = __dmul_rn(e, __ddiv_rn(tk[q], a.ramp));
        }
        a.eta[(size_t)(k0 + q) * a.Bp + b] = e;
    }
}

// ------------------------------------------------------------------------------------------
// k_wave_kinematics: WaveBase::GetElevation / GetVelocity / GetAcceleration (wave_types.cpp:14-160,301-313,515-550)
// for every instance at its own points.  One thread = one instance x PPT points of it (blockIdx.y strides over point
// groups), so every phase it loads serves all of them.  Per-component fields are staged in shared memory, per-instance
// phases / amplitudes are [nf][Bp] as in k_eta (one coalesced load per warp and component).  The reference's
// expressions with their left-to-right products, every operation rounded on its own (no contraction):
//   arg = (k x - omega t) + phi,  eta += A cos(arg) in ascending i  (at x = 0: bit for bit k_eta's sum)
//   deep water:  v = (omega A) e^{kz} (cos, sin),  a = ((omega omega) A) e^{kz} sin, ((-omega omega) A) e^{kz} cos
//   finite:      e^{kz} -> cosh(k (z + depth)) / sinh(k depth) in x,  sinh(k (z + depth)) / sinh(k depth) in z
// sincos returns bit for bit the cos of k_eta (same reduction and polynomial), so the single pass shares its eta.
// ------------------------------------------------------------------------------------------
struct KinAcc { double eta, vx, vz, ax, az; };

__device__ __forceinline__ double kin_arg(double om, double k, double ph, double t, double x) {
    return __dadd_rn(__dsub_rn(__dmul_rn(k, x), __dmul_rn(om, t)), ph);
}

// one component's share at one point; z = position.z - mwl (stretched for Wheeler)
__device__ __forceinline__ void kin_add(KinAcc& r, double om, double k, bool deep, double shkd, double A, double ph,
                                        double t, double depth, double x, double z, bool with_eta) {
    double s, c;
    sincos(kin_arg(om, k, ph, t, x), &s, &c);
    if (with_eta) r.eta = __dadd_rn(r.eta, __dmul_rn(A, c));
    const double oa = __dmul_rn(om, A);
    const double ooa = __dmul_rn(__dmul_rn(om, om), A);
    const double nooa = __dmul_rn(__dmul_rn(-om, om), A);
    double vx, vz, ax, az;
    if (deep) {                                                         // wave_types.cpp:71-76, :103-108
        const double e = exp(__dmul_rn(k, z));
        vx = __dmul_rn(oa, e); vz = vx;
        ax = __dmul_rn(ooa, e); az = __dmul_rn(nooa, e);
    } else {                                                            // :77-83, :109-115
        const double kz = __dmul_rn(k, __dadd_rn(z, depth));
        const double ch = cosh(kz), sh = sinh(kz);
        vx = __ddiv_rn(__dmul_rn(oa, ch), shkd); vz = __ddiv_rn(__dmul_rn(oa, sh), shkd);
        ax = __ddiv_rn(__dmul_rn(ooa, ch), shkd); az = __ddiv_rn(__dmul_rn(nooa, sh), shkd);
    }
    r.vx = __dadd_rn(r.vx, __dmul_rn(vx, c));
    r.vz = __dadd_rn(r.vz, __dmul_rn(vz, s));
    r.ax = __dadd_rn(r.ax, __dmul_rn(ax, s));
    r.az = __dadd_rn(r.az, __dmul_rn(az, c));
}

// one pass over the irregular components: ETA_ONLY = GetEtaIrregular (Wheeler's first pass), else the kinematics
template <int PPT, bool ETA_ONLY>
__device__ __forceinline__ void kin_irregular_pass(const KinArgs& a, double (*s_c)[kKinChunk], int b, int np,
                                                   const double* x, const double* z, KinAcc* r, bool with_eta) {
    for (int i0 = 0; i0 < a.nf; i0 += kKinChunk) {
        const int n = min(kKinChunk, a.nf - i0);
        __syncthreads();
        for (int q = threadIdx.x; q < n; q += blockDim.x)
#pragma unroll
            for (int f = 0; f < kKinPhase; ++f) s_c[f][q] = a.comp[(size_t)f * a.nf + i0 + q];
        __syncthreads();
        if (np == 0) continue;
        for (int q = 0; q < n; ++q) {
            const size_t ib = (size_t)(i0 + q) * a.Bp + b;
            const double A = a.amp ? a.amp[ib] : s_c[kKinAmp][q];
            const double ph = a.phase[ib];
            const double om = s_c[kKinOmega][q], k = s_c[kKinK][q];
#pragma unroll
            for (int j = 0; j < PPT; ++j) {
                if (j >= np) break;
                if (ETA_ONLY) r[j].eta = __dadd_rn(r[j].eta, __dmul_rn(A, cos(kin_arg(om, k, ph, a.t, x[j]))));
                else kin_add(r[j], om, k, s_c[kKinDeep][q] != 0.0, s_c[kKinSinhKd][q], A, ph, a.t, a.depth, x[j], z[j],
                             with_eta);
            }
        }
    }
}

template <int PPT, bool REGULAR>
__global__ void __launch_bounds__(128) k_wave_kinematics(const KinArgs a) {
    __shared__ double s_c[kKinPhase][kKinChunk];
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int groups = (a.P + PPT - 1) / PPT;
    for (int g = blockIdx.y; g < groups; g += gridDim.y) {             // uniform per CTA (syncthreads inside)
        const int p0 = g * PPT;
        const int np = b < a.B ? min(PPT, a.P - p0) : 0;
        double x[PPT], z[PPT];
        KinAcc r[PPT];
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            x[j] = 0.0; z[j] = 0.0;
            r[j] = KinAcc{0.0, 0.0, 0.0, 0.0, 0.0};
            if (j < np) {
                const double* p = a.points + ((size_t)b * a.P + p0 + j) * 3;
                x[j] = p[0];
                z[j] = __dsub_rn(p[2], a.mwl);                          // z_pos = position.z - mwl
            }
        }
        if (REGULAR) {                                                  // RegularWave: one component, never stretched
            if (np > 0) {
                const double* c = a.comp + b;
                const size_t s = a.Bp;
                const double om = c[kKinOmega * s], k = c[kKinK * s], shkd = c[kKinSinhKd * s];
                const double A = c[kKinAmp * s], ph = c[kKinPhase * s];
                const bool deep = c[kKinDeep * s] != 0.0;
#pragma unroll
                for (int j = 0; j < PPT; ++j)
                    if (j < np) kin_add(r[j], om, k, deep, shkd, A, ph, a.t, a.depth, x[j], z[j], true);
            }
        } else {
            if (a.wheeler) {                                            // wave_types.cpp:530-533
                kin_irregular_pass<PPT, true>(a, s_c, b, np, x, z, r, true);
#pragma unroll
                for (int j = 0; j < PPT; ++j) {
                    const double e = r[j].eta;
                    // position_stretched.z = depth (z_pos - eta) / (depth + eta); GetWaterVelocity subtracts mwl again
                    z[j] = __dsub_rn(__ddiv_rn(__dmul_rn(a.depth, __dsub_rn(z[j], e)), __dadd_rn(a.depth, e)), a.mwl);
                }
            }
            kin_irregular_pass<PPT, false>(a, s_c, b, np, x, z, r, !a.wheeler);
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (j >= np) break;
            const size_t o = (size_t)b * a.P + p0 + j;
            if (a.eta) a.eta[o] = r[j].eta;
            if (a.vel) { a.vel[3 * o] = r[j].vx; a.vel[3 * o + 1] = 0.0; a.vel[3 * o + 2] = r[j].vz; }
            if (a.acc) { a.acc[3 * o] = r[j].ax; a.acc[3 * o + 1] = 0.0; a.acc[3 * o + 2] = r[j].az; }
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_added_mass_mv: R[b][i] += sum_j (c*M[i][j]) * w[b][j];  M is the padded n_sys x n_sys matrix.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_added_mass_mv(const double* __restrict__ M, int n_sys, int D, double c,
                                                       const double* __restrict__ w, double* __restrict__ R, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* wb = w + (size_t)b * n_sys;
    double* Rb = R + (size_t)b * n_sys;
    // rows/cols >= D of M_sys are zero (chloadaddedmass.cpp:35-44): adding c*0*w changes nothing
    for (int i = 0; i < D; ++i) {
        double s = 0.0;
        for (int j = 0; j < D; ++j) s = __dadd_rn(s, __dmul_rn(__dmul_rn(c, M[(size_t)i * D + j]), wb[j]));
        Rb[i] = __dadd_rn(Rb[i], s);
    }
}

// ------------------------------------------------------------------------------------------
// launch wrappers (host)
// ------------------------------------------------------------------------------------------
size_t radiation_smem_bytes(int D, int chunk) {
    return 16 + (size_t)chunk * D * D * 8 + (size_t)chunk * 3 * 8 + (size_t)chunk * 2 * 4 + 16;
}
size_t radiation_mma_smem_bytes(int chunk) {
    return 16 + (size_t)chunk * kMmaFragDoubles * 8 + (size_t)chunk * 3 * 8 + (size_t)chunk * 2 * 4 + 16;
}
size_t excitation_smem_bytes(int nd, int chunk) {
    return 16 + (size_t)chunk * nd * 8 + (size_t)chunk * 2 * 8 + (size_t)chunk * 4 + 16;
}

template <int D, bool INLINE>
static cudaError_t launch_rad_t(const RadiationArgs& a, const RadPlanPtrs& p, dim3 grid, size_t smem, cudaStream_t st) {
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(k_radiation<D, INLINE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    k_radiation<D, INLINE><<<grid, kThreads, smem, st>>>(a, p);
    return cudaGetLastError();
}

bool radiation_plans_inline(const RadiationArgs& a) {      // which launch_radiation dispatches take an InlinePlan
    return (a.D == 6 || a.D == 12) && a.Khyb == nullptr && a.Kfrag == nullptr;
}

cudaError_t launch_radiation(const RadiationArgs& a, const int* pr_new, const int* pr_old, const double* pr_wn,
                             const double* pr_wo, const double* pr_wd, cudaStream_t st, const InlinePlan* ip) {
    RadPlanPtrs p{pr_new, pr_old, pr_wn, pr_wo, pr_wd, nullptr, nullptr, nullptr, 0};
    if (ip) {
        if (!radiation_plans_inline(a)) return cudaErrorInvalidValue;
        p.out_wd = ip->pr_wd; p.out_head = ip->pr_head; p.out_lead = ip->pr_lead; p.B = ip->B;
        dim3 gridi((a.Bp + kTileInst - 1) / kTileInst, a.nchunk, 1);
        const size_t smemi = radiation_smem_bytes(a.D, a.chunk);
        return a.D == 6 ? launch_rad_t<6, true>(a, p, gridi, smemi, st) : launch_rad_t<12, true>(a, p, gridi, smemi, st);
    }
    dim3 grid((a.Bp + kTileInst - 1) / kTileInst, a.nchunk, 1);
    const size_t smem = radiation_smem_bytes(a.D, a.chunk);
    if (a.D == 12 && a.Khyb != nullptr) {
        static bool attr_set[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_set[dev & 63]) {
            cudaError_t e = cudaFuncSetAttribute(k_radiation_hybrid12, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return e;
            attr_set[dev & 63] = true;
        }
        const int tile = (kHybThreads / 32) * 64;
        dim3 gridh((a.Bp + tile - 1) / tile, a.nchunk, 1);
        k_radiation_hybrid12<<<gridh, kHybThreads, radiation_smem_bytes(12, a.chunk), st>>>(a, p);
        return cudaGetLastError();
    }
    if (a.D == 12 && a.Kfrag != nullptr) {
        static bool attr_set[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_set[dev & 63]) {
            cudaError_t e = cudaFuncSetAttribute(k_radiation_mma12, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return e;
            attr_set[dev & 63] = true;
        }
        k_radiation_mma12<<<grid, kThreads, radiation_mma_smem_bytes(a.chunk), st>>>(a, p);
        return cudaGetLastError();
    }
    switch (a.D) {
        case 6: return launch_rad_t<6, false>(a, p, grid, smem, st);
        case 12: return launch_rad_t<12, false>(a, p, grid, smem, st);
        default:
            grid.z = a.D / 6;
            k_radiation_generic<<<grid, kThreads, 0, st>>>(a, p);
            return cudaGetLastError();
    }
}

template <int ND, bool INLINE>
static cudaError_t launch_exc_t(const ExcitationArgs& a, const ExcGroup& g, const ExcPlanPtrs& p, dim3 grid, size_t smem,
                                cudaStream_t st) {
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(k_excitation<ND, INLINE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    k_excitation<ND, INLINE><<<grid, kThreads, smem, st>>>(a, g, p);
    return cudaGetLastError();
}

cudaError_t launch_excitation(const ExcitationArgs& a, const ExcGroup& g, const int* idx, const double* w1,
                              const double* w2, cudaStream_t st, bool plan_inline) {
    ExcPlanPtrs p{idx, w1, w2};
    dim3 grid((a.Bp + kTileInst - 1) / kTileInst, g.nchunk, 1);
    const size_t smem = excitation_smem_bytes(g.nd, a.chunk);
    if (plan_inline) {
        if (g.nd == 6) return launch_exc_t<6, true>(a, g, p, grid, smem, st);
        if (g.nd == 12) return launch_exc_t<12, true>(a, g, p, grid, smem, st);
        return cudaErrorInvalidValue;
    }
    switch (g.nd) {
        case 6: return launch_exc_t<6, false>(a, g, p, grid, smem, st);
        case 12: return launch_exc_t<12, false>(a, g, p, grid, smem, st);
        default: return cudaErrorInvalidValue;   // groups are formed with nd in {6, 12} only
    }
}

int radiation_ctas_per_sm(int D, int chunk) {
    int n = 0;
    const size_t smem = radiation_smem_bytes(D, chunk);
    cudaError_t e = cudaErrorInvalidValue;
    if (D == 6) {
        cudaFuncSetAttribute(k_radiation<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_radiation<6>, kThreads, smem);
    } else if (D == 12) {
        cudaFuncSetAttribute(k_radiation<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_radiation<12>, kThreads, smem);
    } else {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_radiation_generic, kThreads, 0);
    }
    if (e != cudaSuccess) { cudaGetLastError(); return 1; }
    return n > 0 ? n : 1;
}
int excitation_ctas_per_sm(int nd, int chunk) {
    int n = 0;
    const size_t smem = excitation_smem_bytes(nd, chunk);
    cudaError_t e;
    if (nd == 6) {
        cudaFuncSetAttribute(k_excitation<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_excitation<6>, kThreads, smem);
    } else {
        cudaFuncSetAttribute(k_excitation<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_excitation<12>, kThreads, smem);
    }
    if (e != cudaSuccess) { cudaGetLastError(); return 1; }
    return n > 0 ? n : 1;
}

cudaError_t launch_prestep(const PrestepArgs& a, int mode, cudaStream_t st) {
    int work = 1;
    if (mode & 1) work = max(work, a.D * a.Bp);
    if (mode & 2) {
        work = max(work, a.L);
        for (int g = 0; g < a.ngroups; ++g) work = max(work, a.Le[g]);
    }
    int blocks = (work + 255) / 256;
    blocks = max(1, min(blocks, 148 * 8));
    k_prestep<<<blocks, 256, 0, st>>>(a, mode);
    return cudaGetLastError();
}

cudaError_t launch_finalize(const FinalizeArgs& a, const HydrostaticTables& hs, const FinalizeGroups& eg,
                            cudaStream_t st) {
    static int mode = -1;                                           // 0 auto, 1 thread per item, 2 warp per item, 3 split
    if (mode < 0) {
        const char* m = std::getenv("HC_FINALIZE_MODE");            // diagnostic override
        mode = m ? std::atoi(m) : 0;
    }
    int nparts = a.rad_nchunk;
    if (a.wave_mode == 2) for (int g = 0; g < a.exc_ngroups; ++g) nparts = std::max(nparts, a.rad_nchunk + eg.nchunk[g]);
    int pick = mode;
    // measured (RM3 shape, per-step path, us per step, warp / split / thread): B = 16: 42.8 / 41.1 / -, 256: 71.1 / 68.5 / -,
    // 512: 102 / 92 / -, 1024: 136 / 121 / 136, 2048: - / 182 / 181, 4096: - / 295 / 285  (profiles/r02w5_finalize_modes.txt)
    if (pick == 0) pick = (a.B <= kFinalizeWarpMaxB) ? 2 : (nparts >= kFinalizeSplitMinParts ? 3 : 1);
    if (pick == 3) {
        k_finalize_split<16><<<a.D * ((a.B + 31) / 32), 32 * 16, 0, st>>>(a, hs, eg);
        return cudaGetLastError();
    }
    if (pick == 2) {     // small ensemble: a lane group per (dof, instance)
        // (G = 8 -- four consecutive instances per warp, sector-efficient rows -- measured slower at every size: 53 vs
        //  40 us at B = 16, 78 vs 67 us at B = 256: the dependent load rounds per lane count, not the sectors)
        k_finalize_warp<32><<<(a.D * a.B * 32 + 255) / 256, 256, 0, st>>>(a, hs, eg);
    }
    else
        k_finalize<<<(a.D * a.Bp + 255) / 256, 256, 0, st>>>(a, hs, eg);
    return cudaGetLastError();
}

cudaError_t launch_eta(const EtaArgs& a, cudaStream_t st) {
    dim3 grid((a.Bp + 127) / 128, (a.n_eta + kEtaKT - 1) / kEtaKT);
    k_eta<<<grid, 128, 0, st>>>(a);
    return cudaGetLastError();
}

// Points per thread: as many as keep at least two CTAs per SM (more phase reuse per thread while the grid still fills
// the GPU), one when even that leaves SMs short.
cudaError_t launch_wave_kinematics(const KinArgs& a, int sm_count, cudaStream_t st) {
    const int xb = (a.B + 127) / 128;
    auto groups = [&](int ppt) { return (a.P + ppt - 1) / ppt; };
    const int ppt = (long long)xb * groups(kKinPts) >= 2LL * sm_count ? kKinPts
                  : (long long)xb * groups(2) >= 2LL * sm_count ? 2 : 1;
    const dim3 grid(xb, std::min(groups(ppt), 65535));
    if (a.regular) k_wave_kinematics<1, true><<<dim3(xb, std::min(groups(1), 65535)), 128, 0, st>>>(a);
    else if (ppt == kKinPts) k_wave_kinematics<kKinPts, false><<<grid, 128, 0, st>>>(a);
    else if (ppt == 2) k_wave_kinematics<2, false><<<grid, 128, 0, st>>>(a);
    else k_wave_kinematics<1, false><<<grid, 128, 0, st>>>(a);
    return cudaGetLastError();
}

// FP64 FMA peak microbenchmark (the FP64 roofline denominator: MEASURED_PEAKS.json has no FP64 figure).
__global__ void __launch_bounds__(256) k_dfma_peak(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}
cudaError_t measure_dfma_peak(double seconds_budget, double* tflops) {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 8, threads = 256, iters = 1 << 14;
    double* buf = nullptr;
    cudaError_t e = cudaMalloc(&buf, size_t(blocks) * threads * sizeof(double));
    if (e != cudaSuccess) return e;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0.0, spent = 0.0;
    for (int rep = 0; rep < 50 && spent < seconds_budget; ++rep) {
        cudaEventRecord(a);
        k_dfma_peak<<<blocks, threads>>>(buf, iters, 0.999999, 1e-9);
        cudaEventRecord(b);
        e = cudaEventSynchronize(b);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        spent += ms * 1e-3;
        const double tf = 2.0 * 8.0 * double(iters) * blocks * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(buf);
    *tflops = best;
    return e;
}

// FP64 tensor-core (DMMA m8n8k4) peak: 8 independent accumulator tiles per warp.
__global__ void __launch_bounds__(256) k_dmma_peak(double* out, int iters, double a, double b) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) { c[i][0] = threadIdx.x + i; c[i][1] = threadIdx.x - i; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma8x8x4(c[i][0], c[i][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
cudaError_t measure_dmma_peak(double seconds_budget, double* tflops) {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 4, threads = 256, iters = 1 << 12;
    double* buf = nullptr;
    cudaError_t e = cudaMalloc(&buf, size_t(blocks) * threads * sizeof(double));
    if (e != cudaSuccess) return e;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0.0, spent = 0.0;
    for (int rep = 0; rep < 50 && spent < seconds_budget; ++rep) {
        cudaEventRecord(a);
        k_dmma_peak<<<blocks, threads>>>(buf, iters, 1e-3, 1e-3);
        cudaEventRecord(b);
        e = cudaEventSynchronize(b);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        spent += ms * 1e-3;
        // one m8n8k4 DMMA = 8 * 8 * 4 FMA = 512 flop per warp
        const double tf = 512.0 * 8.0 * double(iters) * blocks * (threads / 32) / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(buf);
    *tflops = best;
    return e;
}

cudaError_t launch_lookahead_plan(const LookaheadPlanArgs& a, cudaStream_t st) {
    const int n1 = a.T * a.Le;
    k_la_brackets<<<min((n1 + 255) / 256, 148 * 8), 256, 0, st>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int nchunk = (a.nrows + kLaRows - 1) / kLaRows;
    const int n2 = a.T * nchunk * kLaRows;
    k_la_taps<<<min((n2 + 255) / 256, 148 * 8), 256, 0, st>>>(a);
    return cudaGetLastError();
}

template <int ND>
static cudaError_t launch_la_t(const LookaheadArgs& a, cudaStream_t st) {
    const size_t smem = 16 + size_t(2) * kLaT * kLaRows * ND * sizeof(double);
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(k_exc_block<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    const int tiles = (a.Bp + 32 * kIPT - 1) / (32 * kIPT);
    k_exc_block<ND><<<tiles, kLaT * 32, smem, st>>>(a);
    return cudaGetLastError();
}

template <int ND>
static cudaError_t launch_la_mma_t(const LookaheadArgs& a, cudaStream_t st) {
    const size_t smem = 16 + size_t(2) * (kLaRows / 4) * ND * 32 * sizeof(double);
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(k_exc_block_mma<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    const int tiles = (a.Bp + 63) / 64;                      // 4 warps x 16 instances per CTA
    k_exc_block_mma<ND><<<dim3(tiles, a.nseg, 1), 128, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_lookahead(const LookaheadArgs& a, cudaStream_t st) {
    if (a.use_mma) {
        switch (a.nd) {
            case 6: return launch_la_mma_t<6>(a, st);
            case 12: return launch_la_mma_t<12>(a, st);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (a.nd) {
        case 6: return launch_la_t<6>(a, st);
        case 12: return launch_la_t<12>(a, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_added_mass_mv(const double* M, int n_sys, int D, double c, const double* w, double* R, int B,
                                 cudaStream_t st) {
    k_added_mass_mv<<<(B + 127) / 128, 128, 0, st>>>(M, n_sys, D, c, w, R, B);
    return cudaGetLastError();
}

}  // namespace hc
