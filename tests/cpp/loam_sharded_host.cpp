// TEST-ONLY: locreg_align_loam_batch_sharded driven from a plain C++ host: one host thread per GPU, one surf / edge
// handle pair each, NCCL inside liblocreg.so (no Python, no torch).
//   make -f tests/cpp/loam_sharded_host.mk [OUT=dir]; then
//   loam_sharded_host [world]      world = number of GPUs to use (default: all visible, at most 8)
// The batch has 3 * world + 1 scans (ragged blocks: S % world != 0 from two ranks on); each scan is cut into a surf half
// (its even points) and an edge half (its odd points), one scan has no edge half and one no surf half, and eps > 0 lets
// scans stop early.  Every rank passes only its block and must get back the poses and results of ALL scans, bit for bit
// what one surf / edge pair on GPU 0 returns from locreg_align_loam_batch for the whole batch.
// Exit code 0: ok; 3: no CUDA device; 4: NCCL not available; anything else: failure.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include <dlfcn.h>

#include "../../include/locreg.h"
#include "../../include/locreg_synth.h"

#define CHECK(expr)                                                                                    \
    do {                                                                                               \
        const int rc_ = (expr);                                                                        \
        if (rc_ != LOCREG_OK) {                                                                        \
            std::fprintf(stderr, "%s:%d %s -> %d (%s)\n", __FILE__, __LINE__, #expr, rc_, locreg_last_error()); \
            std::exit(rc_ == LOCREG_E_UNSUPPORTED ? 4 : 1);                                            \
        }                                                                                              \
    } while (0)

static const int kMaxIteration = 10;
static const double kEps = 1e-2;

static int device_count() {
    void* cu = dlopen("libcuda.so.1", RTLD_NOW);
    if (!cu) return 0;
    auto init = reinterpret_cast<int (*)(unsigned)>(dlsym(cu, "cuInit"));
    auto count = reinterpret_cast<int (*)(int*)>(dlsym(cu, "cuDeviceGetCount"));
    int n = 0;
    if (!init || !count || init(0) != 0 || count(&n) != 0) return 0;
    return n;
}

struct Job {
    std::vector<float> map;                  // float4
    std::vector<float> surf, edge;           // float4, S halves concatenated
    std::vector<int64_t> surf_off, edge_off; // S + 1 each
    std::vector<double> init;                // S * 7
    size_t n_map = 0, S = 0;
};

static Job make_job(size_t S) {
    Job j;
    synth_world* w = synth_world_create(80.0, 0x5EED0001ull);
    j.map.resize(4 * 120000);
    j.n_map = synth_world_sample_map(w, 120000, 0.2, 0.01, 0x5EED0001ull, j.map.data());
    std::vector<double> gt(S * 7);
    synth_world_poses(w, S, 0x5EED0003ull, gt.data());
    j.S = S;
    j.surf_off.assign(1, 0);
    j.edge_off.assign(1, 0);
    j.init.resize(S * 7);
    std::vector<float> one(4 * 16 * 500);
    for (size_t s = 0; s < S; ++s) {
        const size_t n = synth_world_scan(w, gt.data() + 7 * s, 16, 500, 0x5EED0002ull + s, one.data());
        for (size_t i = 0; i < n; ++i) {
            const bool to_edge = i % 2 == 1;
            if ((to_edge && s == 1) || (!to_edge && s == 2)) continue;  // scan 1 has no edge half, scan 2 no surf half
            std::vector<float>& half = to_edge ? j.edge : j.surf;
            half.insert(half.end(), one.begin() + 4 * i, one.begin() + 4 * i + 4);
        }
        j.surf_off.push_back(static_cast<int64_t>(j.surf.size() / 4));
        j.edge_off.push_back(static_cast<int64_t>(j.edge.size() / 4));
        synth_perturb_pose(gt.data() + 7 * s, 0x5EED0003ull + 31 * s, 0.3, 0.035, j.init.data() + 7 * s);
    }
    synth_world_destroy(w);
    return j;
}

struct Pair {
    locreg_handle* surf = nullptr;
    locreg_handle* edge = nullptr;
};

static Pair make_pair(const Job& j, int device) {
    Pair p;
    locreg_options o;
    CHECK(locreg_default_options(&o, LOCREG_ICP_P2PLANE));
    CHECK(locreg_create(&o, device, &p.surf));
    CHECK(locreg_default_options(&o, LOCREG_ICP_P2LINE));
    CHECK(locreg_create(&o, device, &p.edge));
    CHECK(locreg_set_target(p.surf, j.map.data(), j.n_map, 16));
    CHECK(locreg_set_target(p.edge, j.map.data(), j.n_map, 16));
    return p;
}

static void destroy_pair(Pair& p) {
    CHECK(locreg_destroy(p.surf));
    CHECK(locreg_destroy(p.edge));
}

static bool same_result(const locreg_result& a, const locreg_result& b) {
    return a.iters == b.iters && a.updates == b.updates && a.converged == b.converged && a.degenerate == b.degenerate &&
           a.n_effective == b.n_effective && a.n_inlier == b.n_inlier &&
           std::memcmp(&a.sum_sq_res, &b.sum_sq_res, sizeof(double)) == 0 && a.pose_written == b.pose_written;
}

struct RankOut {
    std::vector<double> poses;
    std::vector<locreg_result> results;
};

int main(int argc, char** argv) {
    const int n_dev = device_count();
    if (n_dev == 0) { std::printf("no CUDA device\n"); return 3; }
    const int world = argc > 1 ? std::atoi(argv[1]) : (n_dev < 8 ? n_dev : 8);
    if (world < 1 || world > n_dev) { std::printf("world %d does not fit %d device(s)\n", world, n_dev); return 2; }
    const Job job = make_job(3 * static_cast<size_t>(world) + 1);

    // ---- the reference: one surf / edge pair, the whole batch
    Pair p0 = make_pair(job, 0);
    RankOut ref;
    ref.poses.resize(job.S * 7);
    ref.results.resize(2 * job.S);
    CHECK(locreg_align_loam_batch(p0.surf, p0.edge, job.surf.data(), job.surf_off.data(), job.edge.data(), job.edge_off.data(), 16,
                                  job.init.data(), job.S, kMaxIteration, kEps, ref.poses.data(), ref.results.data()));
    destroy_pair(p0);

    // ---- one thread per GPU
    unsigned char id[LOCREG_UNIQUE_ID_BYTES];
    CHECK(locreg_comm_unique_id(id));
    std::vector<RankOut> out(world);
    std::vector<std::thread> th;
    for (int r = 0; r < world; ++r) {
        th.emplace_back([&, r]() {
            Pair p = make_pair(job, r);
            CHECK(locreg_comm_init(p.surf, id, r, world));  // the surf handle's communicator carries the exchange
            size_t lo = 0, hi = 0;
            CHECK(locreg_shard_range(job.S, r, world, &lo, &hi));
            // this rank passes only its block: each half's points, offsets relative to the block's first point, poses
            std::vector<int64_t> so(hi - lo + 1), eo(hi - lo + 1);
            for (size_t s = lo; s <= hi; ++s) {
                so[s - lo] = job.surf_off[s] - job.surf_off[lo];
                eo[s - lo] = job.edge_off[s] - job.edge_off[lo];
            }
            RankOut& o = out[r];
            o.poses.resize(job.S * 7);
            o.results.resize(2 * job.S);
            CHECK(locreg_align_loam_batch_sharded(p.surf, p.edge, job.surf.data() + 4 * job.surf_off[lo], so.data(),
                                                  job.edge.data() + 4 * job.edge_off[lo], eo.data(), 16, job.init.data() + 7 * lo,
                                                  hi - lo, job.S, kMaxIteration, kEps, o.poses.data(), o.results.data()));
            CHECK(locreg_comm_destroy(p.surf));
            destroy_pair(p);
        });
    }
    for (auto& t : th) t.join();

    int bad = 0;
    for (int r = 0; r < world; ++r) {
        const RankOut& o = out[r];
        if (std::memcmp(o.poses.data(), ref.poses.data(), job.S * 7 * sizeof(double)) != 0) {
            std::fprintf(stderr, "rank %d: poses differ from the single-GPU batch\n", r);
            ++bad;
        }
        for (size_t i = 0; i < 2 * job.S; ++i)
            if (!same_result(o.results[i], ref.results[i])) {
                std::fprintf(stderr, "rank %d: result %zu (scan %zu, %s half) differs\n", r, i, i / 2, i % 2 ? "edge" : "surf");
                ++bad;
                break;
            }
    }
    int min_iters = kMaxIteration, max_iters = 0;
    for (size_t s = 0; s < job.S; ++s) {
        min_iters = ref.results[2 * s].iters < min_iters ? ref.results[2 * s].iters : min_iters;
        max_iters = ref.results[2 * s].iters > max_iters ? ref.results[2 * s].iters : max_iters;
    }
    std::printf("loam_sharded_host: world %d, %zu scans (%zu surf + %zu edge points), trips %d..%d: %s\n", world, job.S,
                job.surf.size() / 4, job.edge.size() / 4, min_iters, max_iters, bad ? "MISMATCH" : "ok");
    return bad ? 1 : 0;
}
