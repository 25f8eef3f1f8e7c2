// Multi-device ensemble: the instances of one ensemble partitioned over several GPUs of one node (SURVEY.md 8e).
//
// Ensemble members are independent (own eta realisation, own velocity history, own state) and the hydro tables are small
// and read-only, so the B instances are cut into contiguous blocks, one hc_ensemble per device with the tables
// replicated, and there is NO exchange between devices on the step path.  Each device is driven by its own host thread
// (the C ABI's rule: one host thread per ensemble handle); hc_multi_step hands every worker its slice of the caller's
// [B][6N] pose / velocity arrays and its slice of the force array -- instance-major host arrays partition without a
// copy, and the "final result gather" of the north star is each device's D2H into its slice.  The per-step contract is
// the reference's: one evaluation per time value (src/hydro_forces.cpp:742-767), here for every shard at once.
//
// Workers spin for new work for a short while (a step is tens of microseconds; a condition-variable wake-up would
// cost as much) and then block.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>

#include "hc_internal.h"

#if defined(__x86_64__) || defined(__i386__)
#include <immintrin.h>
#define HC_CPU_RELAX() _mm_pause()
#else
#define HC_CPU_RELAX() std::this_thread::yield()
#endif

namespace hc {

struct Worker {
    int device = 0, first = 0, count = 0;            // CUDA device, first global instance, instances of this shard
    hc_ensemble* ens = nullptr;
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::atomic<uint64_t> posted{0}, done{0};
    std::function<hc_status()> job;                   // runs on the worker thread; returns the C ABI's status
    bool quit = false;
    hc_status status = HC_OK;
    std::string message;

    void loop() {
        uint64_t seen = 0;
        for (;;) {
            int spins = 0;
            while (posted.load(std::memory_order_acquire) == seen) {
                if (++spins < 40000) { HC_CPU_RELAX(); continue; }
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return posted.load(std::memory_order_acquire) != seen; });
            }
            seen = posted.load(std::memory_order_acquire);
            if (quit) break;
            status = job();
            message = status == HC_OK ? std::string() : std::string(hc_last_error());
            done.store(seen, std::memory_order_release);
        }
    }
    void post(std::function<hc_status()> f) {
        job = std::move(f);
        posted.fetch_add(1, std::memory_order_release);
        { std::lock_guard<std::mutex> lk(m); }
        cv.notify_one();
    }
    void wait() const {
        const uint64_t want = posted.load(std::memory_order_acquire);
        int spins = 0;
        while (done.load(std::memory_order_acquire) != want)
            if (++spins < 40000) HC_CPU_RELAX(); else std::this_thread::yield();
    }
};

}  // namespace hc

struct hc_multi_ensemble {
    int B = 0, D = 0;
    std::vector<std::unique_ptr<hc::Worker>> w;

    // runs f(worker) on every worker thread at once; first failure wins
    hc_status run(const std::function<hc_status(hc::Worker&)>& f) {
        for (auto& k : w) { hc::Worker* p = k.get(); p->post([p, &f] { return f(*p); }); }
        hc_status st = HC_OK;
        for (auto& k : w) {
            k->wait();
            if (st == HC_OK && k->status != HC_OK) {
                st = k->status;
                hc::set_last_error("device " + std::to_string(k->device) + " (instances " + std::to_string(k->first) + ".." +
                                   std::to_string(k->first + k->count - 1) + "): " + k->message);
            }
        }
        return st;
    }
    ~hc_multi_ensemble() {
        run([](hc::Worker& k) { if (k.ens) hc_ensemble_destroy(k.ens); k.ens = nullptr; return HC_OK; });
        for (auto& k : w) {
            k->quit = true;
            k->post([] { return HC_OK; });
            if (k->th.joinable()) k->th.join();
        }
    }
};

extern "C" {

void hc_multi_shard_range(int total, int shards, int index, int* first, int* count) {
    const int base = total / shards, rem = total % shards;
    const int lo = index * base + (index < rem ? index : rem);
    if (first) *first = lo;
    if (count) *count = base + (index < rem ? 1 : 0);
}

hc_status hc_multi_ensemble_create(const hc_tables* t, const hc_ensemble_opts* opts, const int* devices, int n_devices,
                                   hc_multi_ensemble** out) {
    try {
        if (!t || !opts || !out || n_devices < 1) hc::fail(HC_ERR_INVALID, "null argument / no devices");
        if (opts->batch < n_devices) hc::fail(HC_ERR_INVALID, "fewer instances than devices");
        if (opts->stream) hc::fail(HC_ERR_INVALID, "a multi-device ensemble creates its own streams (opts.stream must be NULL)");
        const int ndev = hc_device_count();
        if (ndev == 0) hc::fail(HC_ERR_CUDA, "no CUDA device available: hydrochrono_b200 has no CPU fallback");
        std::unique_ptr<hc_multi_ensemble> m(new hc_multi_ensemble());
        m->B = opts->batch; m->D = t->D;
        for (int i = 0; i < n_devices; ++i) {
            const int dev = devices ? devices[i] : i;
            if (dev < 0 || dev >= ndev) hc::fail(HC_ERR_INVALID, "bad device ordinal " + std::to_string(dev));
            auto k = std::make_unique<hc::Worker>();
            k->device = dev;
            hc_multi_shard_range(m->B, n_devices, i, &k->first, &k->count);
            hc::Worker* p = k.get();
            k->th = std::thread([p] { p->loop(); });
            m->w.push_back(std::move(k));
        }
        const hc_ensemble_opts base = *opts;
        const hc_status st = m->run([&](hc::Worker& k) {
            hc_ensemble_opts o = base;
            o.device = k.device; o.batch = k.count;
            return hc_ensemble_create(t, &o, &k.ens);
        });
        if (st != HC_OK) return st;                       // (~hc_multi_ensemble destroys what was created)
        *out = m.release();
        return HC_OK;
    } catch (const hc::StatusError& e) { hc::set_last_error(e.msg); return e.code; }
      catch (const std::exception& e) { hc::set_last_error(e.what()); return HC_ERR_INVALID; }
}

void hc_multi_ensemble_destroy(hc_multi_ensemble* m) { delete m; }
int hc_multi_ensemble_num_shards(const hc_multi_ensemble* m) { return int(m->w.size()); }
int hc_multi_ensemble_batch(const hc_multi_ensemble* m) { return m->B; }

hc_status hc_multi_ensemble_shard(const hc_multi_ensemble* m, int index, int* device, int* first, int* count,
                                  hc_ensemble** ens) {
    if (index < 0 || index >= int(m->w.size())) { hc::set_last_error("shard index out of range"); return HC_ERR_OUT_OF_RANGE; }
    const hc::Worker& k = *m->w[index];
    if (device) *device = k.device;
    if (first) *first = k.first;
    if (count) *count = k.count;
    if (ens) *ens = k.ens;
    return HC_OK;
}

hc_status hc_multi_waves_none(hc_multi_ensemble* m) {
    return m->run([](hc::Worker& k) { return hc_waves_none(k.ens); });
}

hc_status hc_multi_waves_regular(hc_multi_ensemble* m, int count, const double* amplitude, const double* omega,
                                 const double* phase) {
    if (!(count == 1 || count == m->B)) { hc::set_last_error("count must be 1 or the total batch size"); return HC_ERR_INVALID; }
    return m->run([=](hc::Worker& k) {
        const int off = count == 1 ? 0 : k.first;
        return hc_waves_regular(k.ens, count == 1 ? 1 : k.count, amplitude + off, omega + off, phase ? phase + off : nullptr);
    });
}

hc_status hc_multi_waves_irregular(hc_multi_ensemble* m, const hc_irregular_params* p, const int* seeds, const double* Hs,
                                   const double* Tp) {
    return m->run([=](hc::Worker& k) {
        return hc_waves_irregular(k.ens, p, seeds ? seeds + k.first : nullptr, Hs ? Hs + k.first : nullptr,
                                  Tp ? Tp + k.first : nullptr);
    });
}

hc_status hc_multi_waves_irregular_series(hc_multi_ensemble* m, double simulation_dt, int n, const double* time,
                                          const double* eta, int per_instance) {
    if (!time || !eta) { hc::set_last_error("null argument"); return HC_ERR_INVALID; }
    return m->run([=](hc::Worker& k) {
        return hc_waves_irregular_series(k.ens, simulation_dt, n, time, per_instance ? eta + size_t(k.first) * n : eta,
                                         per_instance);
    });
}

hc_status hc_multi_step(hc_multi_ensemble* m, double t, const double* pose, const double* vel, const double g[3],
                        double* force, int* recomputed) {
    if (!pose || !vel || !g || !force) { hc::set_last_error("null argument"); return HC_ERR_INVALID; }
    const int D = m->D;
    const double gv[3] = {g[0], g[1], g[2]};
    std::atomic<int> re{0};
    const hc_status st = m->run([&, t](hc::Worker& k) {
        const size_t off = size_t(k.first) * D;
        int r = 0;
        const hc_status s = hc_step(k.ens, t, pose + off, vel + off, gv, force + off, &r);
        if (r) re.store(1);
        return s;
    });
    if (recomputed) *recomputed = re.load();
    return st;
}

hc_status hc_multi_step_device(hc_multi_ensemble* m, double t, const double* const* d_pose, const double* const* d_vel,
                               const double g[3], double* const* d_force) {
    if (!d_pose || !d_vel || !g || !d_force) { hc::set_last_error("null argument"); return HC_ERR_INVALID; }
    const double gv[3] = {g[0], g[1], g[2]};
    std::vector<hc::Worker*> idx;
    for (auto& k : m->w) idx.push_back(k.get());
    return m->run([&, t](hc::Worker& k) {
        size_t i = 0;
        while (idx[i] != &k) ++i;
        return hc_step_device(k.ens, t, d_pose[i], d_vel[i], gv, d_force[i], nullptr);
    });
}

hc_status hc_multi_waves_kinematics_at_time(hc_multi_ensemble* m, double t, int n_points, const double* points, double mwl,
                                            int wheeler_stretching, double* eta, double* velocity, double* acceleration) {
    if (n_points < 1 || !points) { hc::set_last_error("n_points must be positive and points non-null"); return HC_ERR_INVALID; }
    return m->run([=](hc::Worker& k) {
        const size_t off = size_t(k.first) * n_points;
        return hc_waves_kinematics_at_time(k.ens, t, n_points, points + 3 * off, mwl, wheeler_stretching,
                                           eta ? eta + off : nullptr, velocity ? velocity + 3 * off : nullptr,
                                           acceleration ? acceleration + 3 * off : nullptr);
    });
}

hc_status hc_multi_ensemble_simulate(hc_multi_ensemble* m, const hc_sim_params* p, double* pose, double* vel, double* rec_t,
                                     double* rec_pose, double* rec_vel, double* pto_energy, int* steps_done) {
    if (steps_done) *steps_done = 0;
    if (!p || !pose || !vel) { hc::set_last_error("null params, pose or vel"); return HC_ERR_INVALID; }
    const size_t D = size_t(m->D), stride = size_t(m->B) * D;
    std::atomic<int> fewest{p->n_steps};
    const hc_status st = m->run([&](hc::Worker& k) {
        const size_t off = size_t(k.first) * D;
        hc_sim_params q = *p;
        if (p->pto_damping) q.pto_damping = p->pto_damping + off;
        if (p->pto_stiffness) q.pto_stiffness = p->pto_stiffness + off;
        hc_sim_links l{};
        if (p->links) {            // per-instance spring-damper coefficients and energies: the shard's rows
            l = *p->links;
            const size_t toff = size_t(k.first) * size_t(l.n_tsda > 0 ? l.n_tsda : 0);
            if (l.tsda_damping) l.tsda_damping += toff;
            if (l.tsda_stiffness) l.tsda_stiffness += toff;
            if (l.tsda_energy) l.tsda_energy += toff;
            q.links = &l;
        }
        int done = 0;
        // only the first shard writes the (shared) record times
        const hc_status s = hc_ensemble_simulate_strided(k.ens, &q, pose + off, vel + off, k.first == 0 ? rec_t : nullptr,
                                                         rec_pose ? rec_pose + off : nullptr, rec_vel ? rec_vel + off : nullptr,
                                                         stride, pto_energy ? pto_energy + off : nullptr, &done);
        int cur = fewest.load();
        while (done < cur && !fewest.compare_exchange_weak(cur, done)) {}
        return s;
    });
    if (steps_done) *steps_done = fewest.load();
    return st;
}

hc_status hc_multi_get_components(hc_multi_ensemble* m, double* hs, double* rad, double* waves) {
    const int D = m->D;
    return m->run([=](hc::Worker& k) {
        const size_t off = size_t(k.first) * D;
        return hc_get_components(k.ens, hs ? hs + off : nullptr, rad ? rad + off : nullptr, waves ? waves + off : nullptr);
    });
}

hc_status hc_multi_sync(hc_multi_ensemble* m) {
    return m->run([](hc::Worker& k) { return hc_sync(k.ens); });
}

hc_status hc_multi_reset(hc_multi_ensemble* m) {
    return m->run([](hc::Worker& k) { return hc_ensemble_reset(k.ens); });
}

}  // extern "C"
