// C ABI of the registration hot path (include/locreg.h): handle management, host<->device staging,
// kernel launches.  No CPU fallback: without a CUDA device every computing entry point fails.
#include "../../include/locreg.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <deque>
#include <vector>

#include "align_kernels.cuh"
#include "device_map.cuh"
#include "device_inc_ndt.cuh"
#include "device_ndt.cuh"
#include "filters.cuh"
#include "icp_fused.cuh"
#include "icp_staged.cuh"
#include "icp_persist.cuh"
#include "reloc_select.cuh"
#include "nccl_dyn.h"

#include <nvtx3/nvToolsExt.h>

using namespace locreg;

namespace {

thread_local std::string g_last_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 4 + 256;
        LR_CUDA(cudaMalloc(&p, want));
        cap = want;
    }
    ~DevBuf() { if (p) cudaFree(p); }
    template <class T> T* as() const { return static_cast<T*>(p); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 4 + 256;
        LR_CUDA(cudaMallocHost(&p, want));
        cap = want;
    }
    ~PinBuf() { if (p) cudaFreeHost(p); }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

// NVTX range per phase of an entry point (SURVEY.md section 5): visible in Nsight Systems / `ncu --nvtx`, free otherwise.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

bool is_pinned_or_device(const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

}  // namespace

struct locreg_handle {
    locreg_options opt{};
    int device = 0;
    int num_sms = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaStream_t copy_stream = nullptr;        // host->device copies of later chunks overlap the compute of earlier ones
    std::vector<cudaEvent_t> chunk_events;     // locreg_align_batch
    std::vector<cudaStream_t> chunk_streams;   // compute streams of the chunks after the first (they run concurrently)
    std::vector<cudaEvent_t> chunk_done;       // ... and the events that join them into `stream`
    cudaEvent_t loam_ev[2] = {nullptr, nullptr}; // locreg_align_loam (surf handle): [0] state ready / solved, [1] edge half evaluated
    DeviceVoxelMap icp_map;     // level 0: cells of knn_cell_size, neighbourhood lists
    DeviceVoxelMap icp_coarse[kCoarseLevels];  // cells 4x, 16x larger, block tables only (far queries)
    DeviceVoxelMap icp_mid;     // cells 2x larger, neighbourhood lists: stage 2 of the search (LOCREG_MID=0: off)
    CoarseLevels coarse_views(int mid_shells = -1, int coarse_shells = -1) const {  // -1: the defaults of the build
        CoarseLevels c{};
        c.mid_shells_p1 = mid_shells + 1;
        c.coarse_shells_p1 = coarse_shells + 1;
        for (int l = 0; l < kCoarseLevels; ++l) c.lv[l] = icp_coarse[l].view();
        c.mid = icp_mid.view();
        c.pyr = icp_map.pyramid();  // levels == 0 unless LOCREG_PYR_KERNEL=1 asked for it (build_icp_maps)
        c.pyr_mode = 0;             // the thread-per-query stage 2 uses the shells; k_icp_nn_pyr walks the pyramid
        return c;
    }
    DeviceNdtMap ndt_map;
    DeviceIncNdtMap inc_ndt_map;  // LOCREG_NDT_INCREMENTAL
    bool has_target = false;
    // multi-GPU: the communicator of this handle's rank (locreg_comm_init); nullptr = world of one
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    DevBuf d_gather_pose, d_gather_res, d_bcast;
    DevBuf d_raw, d_src4, d_out, d_partials, d_state, d_acc, d_gate, d_nn, d_offsets, d_poses_in, d_poses_out, d_results,
        d_scores, d_misc, d_target, d_nnpos, d_tile_begin, d_tiles, d_states, d_ringq, d_ringc, d_sortq, d_sortb, d_sorth, d_rescanq, d_rescanc, d_loam, d_lmap_new, d_global, d_local, d_same, d_plane, d_pstat, d_track;
    // locreg_relocalise_staged: the cut's keys, flags / slots, the two index maps of the rounds, the caller-order
    // outputs, and the select state + histogram + best
    DevBuf d_stage_keys, d_stage_slot, d_stage_idx, d_stage_poses, d_stage_scores, d_stage_rounds, d_stage_sel;
    // ... and across ranks (locreg_relocalise_staged_sharded): every round's full pose array, which each rank deals its
    // share from, and the all-gather buffer of the round's results
    DevBuf d_stage_full, d_stage_gather;
    size_t n_global = 0, global_stride = 0;  // Loc's global map kept on the device (locreg_set_global_map)
    // Lio's sliding local map (locreg_local_map_add_keyframe): transformed key frames + the filtered local map
    struct KeyFrame { void* p = nullptr; size_t n = 0; };
    std::deque<KeyFrame> keyframes;
    DevBuf d_lmap, d_lmap_tmp;
    size_t n_lmap = 0, lmap_stride = 0;
    void clear_keyframes() {
        for (KeyFrame& k : keyframes) if (k.p) cudaFree(k.p);
        keyframes.clear();
        n_lmap = 0; lmap_stride = 0;
    }
    PinBuf h_in, h_out, h_small;
    double last_ms = 0;
    long long last_launches = 0;
    // optional per-kernel-class timing (locreg_profile): events around every search / fit / solve launch
    bool profile = false;
    std::vector<cudaEvent_t> prof_events;  // pairs
    std::vector<int> prof_class;
    double prof_ms[4] = {0, 0, 0, 0};
    long long prof_launches[4] = {0, 0, 0, 0};
    std::vector<float> prof_trace;  // per launch: class, ms (LOCREG_PROFILE_TRACE=1 prints it)

    IcpParams icp_params() const {
        IcpParams p;
        p.max_nn_distance = opt.max_nn_distance;
        p.max_plane_distance = opt.max_plane_distance;
        p.max_line_distance = opt.max_line_distance;
        p.plane_fit_eps = 1e-2;
        p.eps = opt.eps;
        p.max_iteration = opt.max_iteration;
        p.min_effective_pts = opt.min_effective_pts;
        return p;
    }
    NdtParams ndt_params() const {
        NdtParams p;
        p.res_outlier_th = opt.res_outlier_th;
        p.eps = opt.eps;
        p.max_iteration = opt.max_iteration;
        p.min_effective_pts = opt.min_effective_pts;
        p.min_pts_in_voxel = opt.min_pts_in_voxel;
        p.n_nearby = opt.nearby_type == LOCREG_NEARBY6 ? 7 : 1;
        return p;
    }
    void begin_timing() {
        g_launch_count = 0;
        LR_CUDA(cudaEventRecord(ev0, stream));
    }
    void end_timing() {
        LR_CUDA(cudaEventRecord(ev1, stream));
        LR_CUDA(cudaEventSynchronize(ev1));
        float ms = 0;
        LR_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
        last_ms = ms;
        last_launches = g_launch_count;
    }
};
namespace { void prof_collect(locreg_handle* h); }

namespace {

// Copies a host (or device) cloud into h->d_raw as-is and produces the float4 view kernels read.
// Returns the float4 device pointer.
const float4* stage_cloud(locreg_handle* h, const float* src, size_t n, size_t stride, bool src_on_device) {
    const size_t bytes = n * stride;
    if (n == 0) return nullptr;
    h->d_raw.reserve(bytes);
    if (src_on_device) {
        LR_CUDA(cudaMemcpyAsync(h->d_raw.p, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
    } else if (is_pinned_or_device(src)) {
        LR_CUDA(cudaMemcpyAsync(h->d_raw.p, src, bytes, cudaMemcpyDefault, h->stream));
    } else {
        h->h_in.reserve(bytes);
        std::memcpy(h->h_in.p, src, bytes);
        LR_CUDA(cudaMemcpyAsync(h->d_raw.p, h->h_in.p, bytes, cudaMemcpyHostToDevice, h->stream));
    }
    if (stride == 16) return h->d_raw.as<float4>();
    h->d_src4.reserve(n * sizeof(float4));
    const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((n + 255) / 256, 4096));
    LR_LAUNCH(k_pack_float4, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>(), n, stride, h->d_src4.as<float4>());
    return h->d_src4.as<float4>();
}

// align = true: the pose starts an Align* loop, which honours zero_initial_translation (see locreg.h)
void init_state(locreg_handle* h, const double* pose7, bool align = false) {
    h->d_state.reserve(sizeof(AlignState));
    h->h_small.reserve(4096);
    AlignState* s = h->h_small.as<AlignState>();
    std::memset(s, 0, sizeof(AlignState));
    std::memcpy(s->pose, pose7, 7 * sizeof(double));
    if (align && h->opt.zero_initial_translation && h->opt.method != LOCREG_NDT_INCREMENTAL) s->pose[4] = s->pose[5] = s->pose[6] = 0.0;
    s->res.pose_written = 1;
    s->stop = 0;
    LR_CUDA(cudaMemcpyAsync(h->d_state.p, s, sizeof(AlignState), cudaMemcpyHostToDevice, h->stream));
}

// ---- NDT: fused kernels -------------------------------------------------------------------------------------
// Launch shape of a whole-GPU evaluation of one scan: as many warps as can be co-resident, each taking
// chunks of `ppw` consecutive points (ppw = 32 when the scan is large enough to keep every warp busy).
template <class PB>
int ndt_persist_grid(const locreg_handle* h, unsigned int n, unsigned int* ppw) {
    int per_sm = 0;
    LR_CUDA(cudaFuncSetAttribute(k_align_persist<PB>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kAccSmemBytes)));
    LR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_align_persist<PB>, 256, kAccSmemBytes));
    if (per_sm < 1) throw std::runtime_error("persistent kernel does not fit on an SM");
    const long long max_blocks = static_cast<long long>(per_sm) * h->num_sms;
    const long long max_warps = max_blocks * 8;
    long long p = (static_cast<long long>(n) + max_warps - 1) / max_warps;
    p = std::max<long long>(1, std::min<long long>(32, p));
    *ppw = static_cast<unsigned int>(p);
    const long long chunks = (static_cast<long long>(n) + p - 1) / p;
    return static_cast<int>(std::max<long long>(1, std::min(max_blocks, (chunks + 7) / 8)));
}
template <class PB>
unsigned int ndt_eval_grid(const locreg_handle* h, unsigned int n, unsigned int* ppw) {
    const long long max_warps = 16ll * h->num_sms * 8;
    long long p = (static_cast<long long>(n) + max_warps - 1) / max_warps;
    p = std::max<long long>(1, std::min<long long>(32, p));
    *ppw = static_cast<unsigned int>(p);
    const long long chunks = (static_cast<long long>(n) + p - 1) / p;
    LR_CUDA(cudaFuncSetAttribute(k_eval<PB>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kAccSmemBytes)));
    return static_cast<unsigned int>(std::max<long long>(1, std::min<long long>((chunks + 7) / 8, 16ll * h->num_sms)));
}

// Whole AlignNdt / AlignIncNdt loop on the device, result left in h->d_state.
template <class PB>
void ndt_run_align(locreg_handle* h, PB pb, const float4* src, unsigned int n) {
    AlignState* st = h->d_state.as<AlignState>();
    if (h->opt.loop_mode == LOCREG_LOOP_PERSISTENT) {
        unsigned int ppw = 0;
        const int grid = ndt_persist_grid<PB>(h, n, &ppw);
        h->d_partials.reserve(static_cast<size_t>(2) * grid * kPartialDoubles * sizeof(double));
        double* partials = h->d_partials.as<double>();
        int final_eval = 0;
        void* args[] = {&pb, &src, &n, &ppw, &st, &partials, &final_eval};
        LR_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_align_persist<PB>), dim3(grid), dim3(256), args, kAccSmemBytes, h->stream));
        ++g_launch_count;
    } else {
        unsigned int ppw = 0;
        const unsigned int grid = ndt_eval_grid<PB>(h, n, &ppw);
        h->d_partials.reserve(static_cast<size_t>(grid) * kPartialDoubles * sizeof(double));
        double* partials = h->d_partials.as<double>();
        for (int it = 0; it < h->opt.max_iteration; ++it) {
            LR_LAUNCH(k_eval<PB>, grid, 256, kAccSmemBytes, h->stream, pb, src, n, ppw, st, partials, nullptr, nullptr);
            LR_LAUNCH(k_finalize<PB>, 1, 256, 0, h->stream, pb, partials, grid, st, 1, nullptr);
        }
    }
}
template <class PB>
void ndt_run_eval(locreg_handle* h, PB pb, const float4* src, unsigned int n, unsigned char* gate) {
    AlignState* st = h->d_state.as<AlignState>();
    unsigned int ppw = 0;
    const unsigned int grid = ndt_eval_grid<PB>(h, n, &ppw);
    h->d_partials.reserve(static_cast<size_t>(grid) * kPartialDoubles * sizeof(double));
    h->d_acc.reserve(32 * sizeof(double));
    LR_LAUNCH(k_eval<PB>, grid, 256, kAccSmemBytes, h->stream, pb, src, n, ppw, st, h->d_partials.as<double>(), gate, nullptr);
    LR_LAUNCH(k_finalize<PB>, 1, 256, 0, h->stream, pb, h->d_partials.as<double>(), grid, st, 0, h->d_acc.as<double>());
}
// offsets == nullptr: every item registers the same scan src[0, n_single) (relocalisation)
template <class PB>
void ndt_run_batch(locreg_handle* h, PB pb, const float4* src, const long long* offsets, const double* poses_in, double* poses_out,
                   DevResult* results, unsigned int S, unsigned int n_single = 0u, int final_eval = 0) {
    int per_sm = 0;
    LR_CUDA(cudaFuncSetAttribute(k_align_batch<PB>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kAccSmemBytes)));
    LR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_align_batch<PB>, 256, kAccSmemBytes));
    if (per_sm < 1) per_sm = 1;
    const unsigned int grid = static_cast<unsigned int>(std::max<long long>(1, std::min<long long>(S, static_cast<long long>(per_sm) * h->num_sms)));
    h->d_misc.reserve(64);
    LR_CUDA(cudaMemsetAsync(h->d_misc.p, 0, 64, h->stream));
    const int zero_t = h->opt.zero_initial_translation && h->opt.method != LOCREG_NDT_INCREMENTAL;
    LR_LAUNCH(k_align_batch<PB>, grid, 256, kAccSmemBytes, h->stream, pb, src, offsets, n_single, poses_in, poses_out, results, S,
              h->d_misc.as<unsigned int>(), final_eval, zero_t);
}
// direct or incremental NDT problem of this handle -> f(problem)
#define NDT_DISPATCH(h, CALL)                                                                   \
    if ((h)->opt.method == LOCREG_NDT_INCREMENTAL) {                                            \
        const IncNdtProblem PB{(h)->inc_ndt_map.view(), (h)->ndt_params()};                     \
        CALL;                                                                                   \
    } else {                                                                                    \
        const NdtProblem PB{(h)->ndt_map.view(), (h)->ndt_params()};                            \
        CALL;                                                                                   \
    }

// Event pair around one launch of kernel class cls (0 search stage 1, 1 fit+reduce, 2 solve, 3 search stage 2) when
// profiling is on.
void prof_mark(locreg_handle* h, int cls, bool begin) {
    if (!h->profile) return;
    cudaEvent_t e;
    LR_CUDA(cudaEventCreate(&e));
    LR_CUDA(cudaEventRecord(e, h->stream));
    h->prof_events.push_back(e);
    if (begin) h->prof_class.push_back(cls);
}
void prof_collect(locreg_handle* h) {
    if (!h->profile) return;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i + 1 < h->prof_events.size(); i += 2) {
        float ms = 0;
        LR_CUDA(cudaEventElapsedTime(&ms, h->prof_events[i], h->prof_events[i + 1]));
        const int c = h->prof_class[i / 2];
        h->prof_ms[c] += ms;
        h->prof_launches[c] += 1;
        if (getenv("LOCREG_PROFILE_TRACE")) fprintf(stderr, "locreg-trace class %d %.4f ms\n", c, ms);
    }
    for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
    h->prof_events.clear();
    h->prof_class.clear();
}

// ---- ICP: three-kernel pipeline (icp_pipeline.cuh) -------------------------------------------------------------
struct IcpJob {
    BatchView bv{};
    AlignState* states = nullptr;
    unsigned int n_tiles = 0;       // grid of the per-point kernels (an upper bound is fine: surplus tiles exit)
    size_t n_scratch_points = 0;    // rows of the per-point scratch arrays
    // Chunks of one batch that run CONCURRENTLY on their own streams (align_batch_resident) each own a slice of the
    // handle's per-job scratch: partial rows (doubles into d_partials), queue counters (uints into d_ringc), queue
    // entries (into d_ringq).  The per-point arrays are indexed by absolute point number and need no slicing.
    size_t partials_off = 0, ringc_off = 0, ringq_off = 0;
};

// nn_mode: kNnSeeds when the per-point neighbour scratch still holds THIS job's previous iteration, kNnTwoPass for the
// first iterations (see k_icp_nn)
// Returns the second partial-row array when the evaluation produced one (the fused tracked path of icp_fused.cuh), else
// nullptr; icp_launch_solve takes it.
template <int METHOD>
const double* icp_launch_eval(locreg_handle* h, const IcpJob& job, int ignore_stop, int nn_mode, unsigned char* gate, int* nn_idx) {
    constexpr int K = METHOD == kIcpP2P ? 1 : 5;
    const VoxelMapView map = h->icp_map.view();
    h->d_nnpos.reserve(job.n_scratch_points * K * sizeof(unsigned int));
    h->d_ringq.reserve(job.n_scratch_points * sizeof(uint2));
    h->d_track.reserve(job.n_scratch_points * sizeof(KnnTrack));
    // P2Plane: per-point plane (k_icp_fit) and the flag that says it still belongs to the point's current neighbours
    const bool small = job.n_tiles <= 2u * static_cast<unsigned int>(h->num_sms);
    const bool cache = METHOD == kIcpP2Plane;
    if (cache) {
        h->d_same.reserve(job.n_scratch_points);
        h->d_plane.reserve(job.n_scratch_points * 4 * sizeof(double));
        h->d_pstat.reserve(job.n_scratch_points);
    }
    // k_icp_post re-zeroes the counters after every use; the first evaluation of a job starts from a known state
    h->d_partials.reserve((job.partials_off + 2 * static_cast<size_t>(job.n_tiles) * kPartialDoubles) * sizeof(double));
    h->d_ringc.reserve((job.ringc_off + 2) * sizeof(unsigned int));
    unsigned int* const ringc = h->d_ringc.as<unsigned int>() + job.ringc_off;
    double* const partials_a = h->d_partials.as<double>() + job.partials_off;
    if (!(nn_mode & kNnSeeds)) LR_CUDA(cudaMemsetAsync(ringc, 0, 2 * sizeof(unsigned int), h->stream));
    if (job.n_tiles == 0) return nullptr;
    const RingQueue queue{ringc, h->d_ringq.as<uint2>() + job.ringq_off};
    // P2Plane, tracked iterations: search + residual + normal equations in one pass (icp_fused.cuh)
    static const int fused_on = getenv("LOCREG_FUSED") ? atoi(getenv("LOCREG_FUSED")) : 0;
    const bool fused = METHOD == kIcpP2Plane && (nn_mode & kNnFused) && !gate && !nn_idx && fused_on;
    double* partials_b = partials_a + static_cast<size_t>(job.n_tiles) * kPartialDoubles;
    // searches that look at every point of the tile: candidate lists staged in shared memory (icp_staged.cuh)
    // LOCREG_STAGED: bit 0 = the unseeded first iteration (measured 1.51 ms against 1.75 ms per 14.1 M points), bit 1 =
    // seeded searches, bit 2 = the first tracked one (both measured slower than k_icp_nn, 1.8 against 1.5-1.7 ms: with
    // good seeds the thread-per-query scan rejects nearly every candidate with one comparison, the branch-free selection
    // pays its compare-exchange chain for all of them)
    static const int staged_on = getenv("LOCREG_STAGED") ? atoi(getenv("LOCREG_STAGED")) : 1;
    int staged_mode = -1;
    if (map.nbr_slots != nullptr) {
        if (nn_mode == kNnTwoPass && (staged_on & 1)) staged_mode = 0;
        else if (nn_mode == kNnSeeds && (staged_on & 2)) staged_mode = 1;
        else if ((nn_mode & kNnTrack) && (nn_mode & kNnFirstTrack) && (staged_on & 4)) staged_mode = 2;
    }
    // Queries stage 1 cannot finish: a small job (one scan) gives each of them a warp (lowest latency, the GPU is idle
    // anyway); a large job keeps one query per thread (most requests in flight).
    prof_mark(h, 0, true);
    if (fused)
    {
        h->d_rescanq.reserve(job.n_scratch_points * sizeof(uint2));
        h->d_rescanc.reserve(2 * sizeof(unsigned int));
        const RingQueue rescan{h->d_rescanc.as<unsigned int>(), h->d_rescanq.as<uint2>()};
        LR_CUDA(cudaMemsetAsync(h->d_rescanc.p, 0, 2 * sizeof(unsigned int), h->stream));
        LR_LAUNCH(k_icp_track_p2plane, job.n_tiles, kTile, 0, h->stream, map, h->icp_params(), job.bv, job.states, ignore_stop,
                  h->d_track.as<KnnTrack>(), rescan, h->d_plane.as<double>(), h->d_pstat.as<unsigned char>(), partials_a);
        const unsigned int g = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + 127) / 128, static_cast<size_t>(h->num_sms) * 8));
        LR_LAUNCH(k_icp_rescan, g, 128, 0, h->stream, map, job.bv, job.states, h->d_nnpos.as<unsigned int>(), h->d_same.as<unsigned char>(),
                  h->d_track.as<KnnTrack>(), queue, rescan);
    }
    else if (staged_mode >= 0) {
        unsigned char* pv = cache ? h->d_same.as<unsigned char>() : nullptr;
        if (staged_mode == 0)
            LR_LAUNCH((k_icp_nn_staged<K, 0>), job.n_tiles, kTile, 0, h->stream, map, job.bv, job.states, ignore_stop, h->d_nnpos.as<unsigned int>(), pv, h->d_track.as<KnnTrack>(), queue);
        else if (staged_mode == 1)
            LR_LAUNCH((k_icp_nn_staged<K, 1>), job.n_tiles, kTile, 0, h->stream, map, job.bv, job.states, ignore_stop, h->d_nnpos.as<unsigned int>(), pv, h->d_track.as<KnnTrack>(), queue);
        else
            LR_LAUNCH((k_icp_nn_staged<K, 2>), job.n_tiles, kTile, 0, h->stream, map, job.bv, job.states, ignore_stop, h->d_nnpos.as<unsigned int>(), pv, h->d_track.as<KnnTrack>(), queue);
    } else if (nn_mode & kNnTrack)
        LR_LAUNCH((k_icp_nn<K, true>), job.n_tiles, kTile, 0, h->stream, map, job.bv, job.states, ignore_stop, nn_mode, h->d_nnpos.as<unsigned int>(),
                  cache ? h->d_same.as<unsigned char>() : nullptr, h->d_track.as<KnnTrack>(), queue);
    else
        LR_LAUNCH((k_icp_nn<K, false>), job.n_tiles, kTile, 0, h->stream, map, job.bv, job.states, ignore_stop, nn_mode, h->d_nnpos.as<unsigned int>(),
                  cache ? h->d_same.as<unsigned char>() : nullptr, h->d_track.as<KnnTrack>(), queue);
    prof_mark(h, 0, false);
    prof_mark(h, 3, true);
    // The queue length is only known on the device, so both forms are launched and each one looks at the count:
    // below kWarpFinishMax entries the warp-per-query kernel takes the queue (what matters is the latency of the
    // slowest query), from there on the thread-per-query kernel (throughput).  A small job never gets there.
    constexpr unsigned int kWarpFinishMax = 16384;
    // stage 2 leaves margins behind only while the loop tracks (LOCREG_TRACK=0: every query searches every time)
    static const int track_env = getenv("LOCREG_TRACK") ? atoi(getenv("LOCREG_TRACK")) : 1;
    KnnTrack* stage2_track = track_env ? h->d_track.as<KnnTrack>() : nullptr;
    // Relocalisation (hypotheses of one scan; LOCREG_SORT_BATCH=1: batches too): queues of LOCREG_SORT_FRAC x the job's
    // points or more are put in spatial order first (k_queue_bin_count / scan / k_queue_bin_scatter).
    static const int sort_on = getenv("LOCREG_SORT") ? atoi(getenv("LOCREG_SORT")) : 1;
    static const int sort_batch = getenv("LOCREG_SORT_BATCH") ? atoi(getenv("LOCREG_SORT_BATCH")) : 0;
    static const double sort_frac = getenv("LOCREG_SORT_FRAC") ? atof(getenv("LOCREG_SORT_FRAC")) : 0.1;
    static const double sort_bin = getenv("LOCREG_SORT_BIN") ? atof(getenv("LOCREG_SORT_BIN")) : 1.0;  // metres
    static const int sort_bits = getenv("LOCREG_SORT_BITS") ? atoi(getenv("LOCREG_SORT_BITS")) : 24;
    static const int sort_sub = getenv("LOCREG_SORT_SUB") ? std::min(5, std::max(0, atoi(getenv("LOCREG_SORT_SUB")))) : 3;  // Morton-ordered bins per hashed group: 2^sub per axis
    // LOCREG_PYR_KERNEL: which kernel serves the long (sorted) queues - 0 (default) the shells (k_icp_nn_finish), 1 the
    // block-pyramid walks with lane refill (k_icp_nn_pyr: 4x fewer candidates, measured slower - DESIGN section 8)
    static const int pyr_kernel = getenv("LOCREG_PYR_KERNEL") ? atoi(getenv("LOCREG_PYR_KERNEL")) : 0;
    // LOCREG_SORT_MIN: shortest queue that is sorted (tools/sanitize_reloc.py lowers it so that a tiny job runs the path)
    static const unsigned int sort_min = getenv("LOCREG_SORT_MIN") ? static_cast<unsigned int>(std::max(1, atoi(getenv("LOCREG_SORT_MIN")))) : kWarpFinishMax;
    const bool sortable = !small && sort_on && (job.bv.offsets == nullptr || sort_batch) && job.n_scratch_points < 0xFFFFFFFFull;
    unsigned int long_min = 0xFFFFFFFFu;  // queues from this length on take the long-queue path (spatial order)
    if (sortable)
        long_min = static_cast<unsigned int>(std::max<double>(sort_min, std::min<double>(4.0e9, sort_frac * static_cast<double>(job.n_scratch_points))));
    {
        const unsigned int g = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + 3) / 4, static_cast<size_t>(h->num_sms) * 8));
        LR_LAUNCH(k_icp_nn_rings<K>, g, 128, 0, h->stream, map, h->coarse_views(), job.bv, job.states, h->d_nnpos.as<unsigned int>(), stage2_track, queue,
                  small ? 0xFFFFFFFFu : std::min(kWarpFinishMax, long_min));
    }
    if (!small) {
        const PyrView pyr = h->icp_map.pyramid();
        RingQueue long_queue = queue;
        if (sortable) {
            const unsigned int buckets = 1u << sort_bits;
            h->d_sortq.reserve(job.n_scratch_points * sizeof(uint2));
            h->d_sortb.reserve(job.n_scratch_points * sizeof(unsigned int));
            h->d_sorth.reserve(static_cast<size_t>(buckets) * sizeof(unsigned int));
            LR_CUDA(cudaMemsetAsync(h->d_sorth.p, 0, static_cast<size_t>(buckets) * sizeof(unsigned int), h->stream));
            const unsigned int gs = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + 255) / 256, static_cast<size_t>(h->num_sms) * 8));
            LR_LAUNCH(k_queue_bin_count, gs, 256, 0, h->stream, job.bv, job.states, queue, long_min, static_cast<float>(1.0 / sort_bin), buckets - 1, sort_sub,
                      h->d_sortb.as<unsigned int>(), h->d_sorth.as<unsigned int>());
            exclusive_scan_u32(h->d_sorth.as<unsigned int>(), h->d_sorth.as<unsigned int>(), buckets, nullptr, h->stream);
            LR_LAUNCH(k_queue_bin_scatter, gs, 256, 0, h->stream, queue, long_min, h->d_sortb.as<unsigned int>(), h->d_sorth.as<unsigned int>(),
                      h->d_sortq.as<uint2>());
            long_queue = RingQueue{queue.count, h->d_sortq.as<uint2>()};
        }
        const unsigned int g = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + 127) / 128, static_cast<size_t>(h->num_sms) * LR_FINISH_MIN_BLOCKS));
        LR_LAUNCH(k_icp_nn_finish<K>, g, 128, 0, h->stream, map, h->coarse_views(), job.bv, job.states, h->d_nnpos.as<unsigned int>(), stage2_track, queue,
                  std::min(kWarpFinishMax, long_min), long_min);
        if (long_min != 0xFFFFFFFFu) {
            if (pyr_kernel == 1 && pyr.levels != 0) {
                const unsigned int gp = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + 127) / 128, static_cast<size_t>(h->num_sms) * LR_PYR_MIN_BLOCKS));
                LR_LAUNCH(k_icp_nn_pyr<K>, gp, 128, 0, h->stream, map, pyr, job.bv, job.states, h->d_nnpos.as<unsigned int>(), stage2_track, long_queue, long_min);
            } else {
                // far-off hypotheses leave the mid level after two shells (LOCREG_RELOC_MID_SHELLS; measured -4 % against the
                // batches' four, which in turn lose 25 % at two)
                static const int reloc_mid_shells = getenv("LOCREG_RELOC_MID_SHELLS") ? std::max(0, atoi(getenv("LOCREG_RELOC_MID_SHELLS"))) : 1;
                static const int reloc_coarse_shells = getenv("LOCREG_RELOC_COARSE_SHELLS") ? std::max(1, atoi(getenv("LOCREG_RELOC_COARSE_SHELLS"))) : -1;
                LR_LAUNCH(k_icp_nn_finish<K>, g, 128, 0, h->stream, map,
                          h->coarse_views(job.bv.offsets == nullptr ? reloc_mid_shells : -1, job.bv.offsets == nullptr ? reloc_coarse_shells : -1), job.bv, job.states,
                          h->d_nnpos.as<unsigned int>(), stage2_track, long_queue, long_min, 0xFFFFFFFFu);
            }
        }
    }
    prof_mark(h, 3, false);
    prof_mark(h, 1, true);
    if (fused) {
        const unsigned int group = small ? 1u : static_cast<unsigned int>(kPendGroup);
        const RingQueue rescan{h->d_rescanc.as<unsigned int>(), h->d_rescanq.as<uint2>()};
        const unsigned int gf = static_cast<unsigned int>(std::min<size_t>((job.n_scratch_points + kFitChunk - 1) / kFitChunk, static_cast<size_t>(h->num_sms) * 4));
        LR_LAUNCH(k_icp_fit_queue, gf, 128, 0, h->stream, map, h->icp_params(), h->d_nnpos.as<unsigned int>(), h->d_same.as<unsigned char>(),
                  h->d_plane.as<double>(), h->d_pstat.as<unsigned char>(), rescan);
        LR_LAUNCH(k_icp_pending, (job.n_tiles + group - 1) / group, kTile, 0, h->stream, h->icp_params(), job.bv, job.states, ignore_stop,
                  h->d_same.as<unsigned char>(), h->d_plane.as<double>(), h->d_pstat.as<unsigned char>(), group, partials_b,
                  ringc);
        prof_mark(h, 1, false);
        return partials_b;
    }
    if (cache) {
        // a single scan spreads its tiles over the SMs (latency); a batch compacts over 16 tiles per block (throughput).
        // The same kernel either way: batch results equal those of single ScanMatch calls bit for bit.
        const unsigned int group = small ? 1u : static_cast<unsigned int>(kFitGroup);
        LR_LAUNCH(k_icp_fit, (job.n_tiles + group - 1) / group, kTile, 0, h->stream, map, h->icp_params(), job.bv, job.states, ignore_stop,
                  h->d_nnpos.as<unsigned int>(), h->d_same.as<unsigned char>(), h->d_plane.as<double>(), h->d_pstat.as<unsigned char>(), group);
    }
    LR_LAUNCH(k_icp_post<METHOD>, job.n_tiles, kTile, 0, h->stream, map, h->icp_params(), job.bv, job.states, ignore_stop,
              h->d_nnpos.as<unsigned int>(), partials_a, gate, nn_idx, ringc,
              cache ? h->d_plane.as<double>() : nullptr, cache ? h->d_pstat.as<unsigned char>() : nullptr);
    prof_mark(h, 1, false);
    return nullptr;
}
template <int METHOD>
void icp_launch_solve(locreg_handle* h, const IcpJob& job, int mode, double* acc_out, const double* partials_b = nullptr) {
    prof_mark(h, 2, true);
    LR_LAUNCH(k_icp_solve<METHOD>, (job.bv.S + 3) / 4, 128, 0, h->stream, h->icp_params(), job.bv, job.states,
              h->d_partials.as<double>() + job.partials_off, partials_b, mode, acc_out);
    prof_mark(h, 2, false);
}
// Search mode of Gauss-Newton trip `it` of a job whose per-point scratch holds its own previous trips.
int icp_loop_nn_mode(int it) {
    static const int tp_iters = getenv("LOCREG_TWOPASS_ITERS") ? atoi(getenv("LOCREG_TWOPASS_ITERS")) : 1;  // iterations whose scan uses the threshold pre-pass (the unseeded one; 1 measured best: 11.2 ms vs 11.5 at 2, 12.0 at 3)
    static const int track = getenv("LOCREG_TRACK") ? atoi(getenv("LOCREG_TRACK")) : 1;  // 0: every query scans its list every time
    static const int track_from = getenv("LOCREG_TRACK_FROM") ? atoi(getenv("LOCREG_TRACK_FROM")) : 3;  // measured: 2 and 3 alike, 4 +1 % on batches; single scans converge sooner
    // the first tracked iteration searches every point (no margins yet): the three-kernel pipeline; from then on the
    // streaming pass of icp_fused.cuh (P2Plane)
    const int seeded = track && it >= track_from ? (kNnSeeds | kNnTrack | (it > track_from ? kNnFused : kNnFirstTrack)) : kNnSeeds;
    return it == 0 ? kNnTwoPass : (it < tp_iters ? (kNnSeeds | kNnTwoPass) : seeded);
}
// The whole Gauss-Newton loop, queued on the stream without a host round-trip; stopped scans make their tiles exit.
template <int METHOD>
void icp_run_loop(locreg_handle* h, const IcpJob& job, int final_eval) {
    for (int it = 0; it < h->opt.max_iteration; ++it) {
        const double* pb = icp_launch_eval<METHOD>(h, job, 0, icp_loop_nn_mode(it), nullptr, nullptr);
        icp_launch_solve<METHOD>(h, job, 1, nullptr, pb);
    }
    if (final_eval) {
        const double* pb = icp_launch_eval<METHOD>(h, job, 1, h->opt.max_iteration > 0 ? kNnSeeds : kNnTwoPass, nullptr, nullptr);
        icp_launch_solve<METHOD>(h, job, 0, nullptr, pb);
    }
}
// LoamRegistration::ScanMatch's loop (SURVEY.md 3.3) for the S scans of js / je, all trips queued with no host round
// trip.  Each trip evaluates the surf halves (P2Plane) on surf's stream and scratch and the edge halves (P2Line) on
// edge's, each scan's two halves at the one pose in the state both jobs point at, so the two evaluations run side by
// side; k_loam_solve then joins their partial rows on surf's stream, one warp per scan.  loam_ev[0] (surf stream: states
// initialised / trip solved) holds the edge half back until the poses it reads are final and the edge partial rows it
// overwrites have been read; loam_ev[1] (edge stream: edge half evaluated) holds the solve back.  With both handles on
// one stream the same calls run serially.  An empty half launches nothing and its zero tiles sum to zeros; stopped
// scans make their tiles and their solve warp exit.  final_eval: after the trips, both halves are evaluated once more at
// every scan's final pose, stopped or not, and an evaluation-only k_loam_solve (mode 0) records the summed sums in the
// states (LOAM relocalisation's score pass, as icp_run_loop's).
void loam_run_loop(locreg_handle* surf, locreg_handle* edge, const IcpJob& js, const IcpJob& je, int max_iteration,
                   double eps, DevResult* d_half, int final_eval = 0) {
    const auto trip = [&](int ignore_stop, int nn_mode, int mode) {
        LR_CUDA(cudaStreamWaitEvent(edge->stream, surf->loam_ev[0], 0));
        const double* eb = icp_launch_eval<kIcpP2Line>(edge, je, ignore_stop, nn_mode, nullptr, nullptr);
        LR_CUDA(cudaEventRecord(surf->loam_ev[1], edge->stream));
        const double* sb = icp_launch_eval<kIcpP2Plane>(surf, js, ignore_stop, nn_mode, nullptr, nullptr);
        LR_CUDA(cudaStreamWaitEvent(surf->stream, surf->loam_ev[1], 0));
        prof_mark(surf, 2, true);
        LR_LAUNCH(k_loam_solve, (js.bv.S + 3) / 4, 128, 0, surf->stream, js.bv, surf->d_partials.as<double>(), sb,
                  surf->opt.min_effective_pts, je.bv, edge->d_partials.as<double>(), eb, edge->opt.min_effective_pts, js.states,
                  eps, max_iteration, mode, d_half);
        prof_mark(surf, 2, false);
        LR_CUDA(cudaEventRecord(surf->loam_ev[0], surf->stream));
    };
    LR_CUDA(cudaEventRecord(surf->loam_ev[0], surf->stream));
    for (int it = 0; it < max_iteration; ++it) trip(0, icp_loop_nn_mode(it), 1);
    if (final_eval) trip(1, max_iteration > 0 ? kNnSeeds : kNnTwoPass, 0);
    // join: whatever the edge stream still has (its cloud copy when no trip ran) is done before surf's stream goes on
    LR_CUDA(cudaEventRecord(surf->loam_ev[1], edge->stream));
    LR_CUDA(cudaStreamWaitEvent(surf->stream, surf->loam_ev[1], 0));
}
// One scan, whole loop in ONE cooperative launch (icp_persist.cuh).  Returns false when the job does not suit it (then
// the per-iteration pipeline runs): the persistent grid holds one block per SM, a scan of more tiles than 8x that would
// serialise what the pipeline spreads over the whole GPU.
template <int METHOD>
bool icp_run_persistent(locreg_handle* h, const IcpJob& job) {
    constexpr int K = METHOD == kIcpP2P ? 1 : 5;
    static const int persist_on = getenv("LOCREG_ICP_PERSIST") ? atoi(getenv("LOCREG_ICP_PERSIST")) : 1;
    if (!persist_on || h->profile || job.bv.S != 1 || job.n_tiles == 0 || h->opt.max_iteration <= 0) return false;
    int per_sm = 0;
    LR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_icp_persist<METHOD>, kTile, 0));
    if (per_sm < 1) return false;
    const unsigned int capacity = static_cast<unsigned int>(per_sm) * static_cast<unsigned int>(h->num_sms);
    if (job.n_tiles > 8u * capacity) return false;
    const VoxelMapView map = h->icp_map.view();
    const bool cache = METHOD == kIcpP2Plane;
    h->d_nnpos.reserve(job.n_scratch_points * K * sizeof(unsigned int));
    h->d_partials.reserve(2 * static_cast<size_t>(job.n_tiles) * kPartialDoubles * sizeof(double));
    h->d_ringq.reserve(job.n_scratch_points * sizeof(uint2));
    h->d_track.reserve(job.n_scratch_points * sizeof(KnnTrack));
    h->d_same.reserve(job.n_scratch_points);
    h->d_plane.reserve(job.n_scratch_points * 4 * sizeof(double));
    h->d_pstat.reserve(job.n_scratch_points);
    h->d_ringc.reserve(6 * sizeof(unsigned int));  // three (count, cursor) pairs used in rotation (icp_persist.cuh)
    LR_CUDA(cudaMemsetAsync(h->d_ringc.p, 0, 6 * sizeof(unsigned int), h->stream));
    (void)cache;
    // every block of the grid lends its warps to the stage-2 queue, so the grid is the full co-resident capacity even
    // when the scan has fewer tiles
    unsigned int grid = capacity;
    CoarseLevels coarse = h->coarse_views();
    IcpParams prm = h->icp_params();
    BatchView bv = job.bv;
    AlignState* st = job.states;
    unsigned int n_tiles = job.n_tiles;
    unsigned int* nn_pos = h->d_nnpos.as<unsigned int>();
    unsigned char* pv = h->d_same.as<unsigned char>();
    KnnTrack* track = h->d_track.as<KnnTrack>();
    RingQueue queue{h->d_ringc.as<unsigned int>(), h->d_ringq.as<uint2>()};
    double* plane = h->d_plane.as<double>();
    unsigned char* pstat = h->d_pstat.as<unsigned char>();
    double* partials = h->d_partials.as<double>();
    static const int track_on = getenv("LOCREG_TRACK") ? atoi(getenv("LOCREG_TRACK")) : 1;
    static const int track_from_env = getenv("LOCREG_TRACK_FROM") ? atoi(getenv("LOCREG_TRACK_FROM")) : 3;
    int track_from = track_on ? track_from_env : 0x7fffffff;
    VoxelMapView mapv = map;
    // LOCREG_PERSIST_STAMPS=1 (tools): phase time stamps of block 0, printed after the launch
    static const bool stamps = getenv("LOCREG_PERSIST_STAMPS") != nullptr;
    unsigned long long* dbg = nullptr;
    if (stamps) {
        h->d_misc.reserve(64 + 6 * 64 * sizeof(unsigned long long));
        dbg = reinterpret_cast<unsigned long long*>(h->d_misc.as<unsigned char>() + 64);
        LR_CUDA(cudaMemsetAsync(dbg, 0, 6 * 64 * sizeof(unsigned long long), h->stream));
    }
    void* args[] = {&mapv, &coarse, &prm, &bv, &st, &n_tiles, &nn_pos, &pv, &track, &queue, &plane, &pstat, &partials, &track_from, &dbg};
    LR_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_icp_persist<METHOD>), dim3(grid), dim3(kTile), args, 0, h->stream));
    ++g_launch_count;
    if (stamps) {
        unsigned long long t[6 * 64];
        LR_CUDA(cudaMemcpyAsync(t, dbg, sizeof(t), cudaMemcpyDeviceToHost, h->stream));
        LR_CUDA(cudaStreamSynchronize(h->stream));
        for (int it = 0; it < std::min(h->opt.max_iteration, 64) && t[it * 6]; ++it)
            fprintf(stderr, "persist it %2d: search %6.1f us  barrier %5.1f  stage2 %6.1f  fit+post %6.1f  barrier %5.1f  | iteration %6.1f us\n", it,
                    (t[it * 6 + 1] - t[it * 6]) * 1e-3, (t[it * 6 + 2] - t[it * 6 + 1]) * 1e-3, (t[it * 6 + 3] - t[it * 6 + 2]) * 1e-3,
                    (t[it * 6 + 4] - t[it * 6 + 3]) * 1e-3, (t[it * 6 + 5] - t[it * 6 + 4]) * 1e-3,
                    ((it + 1 < h->opt.max_iteration && t[(it + 1) * 6] ? t[(it + 1) * 6] : t[it * 6 + 5]) - t[it * 6]) * 1e-3);
    }
    return true;
}
#define ICP_DISPATCH(h, CALL)                                              \
    switch ((h)->opt.method) {                                             \
        case LOCREG_ICP_P2P: { constexpr int M = kIcpP2P; CALL; } break;   \
        case LOCREG_ICP_P2LINE: { constexpr int M = kIcpP2Line; CALL; } break; \
        case LOCREG_ICP_P2PLANE: { constexpr int M = kIcpP2Plane; CALL; } break; \
        default: throw std::invalid_argument("unsupported method");        \
    }

IcpJob icp_single_job(locreg_handle* h, const float4* src, unsigned int n) {
    IcpJob job;
    job.bv.src = src; job.bv.offsets = nullptr; job.bv.tile_begin = nullptr; job.bv.tiles = nullptr;
    job.bv.n_single = n; job.bv.tiles_per_item = std::max(1u, (n + kTile - 1) / kTile); job.bv.S = 1;
    job.states = h->d_state.as<AlignState>();
    job.n_tiles = (n + kTile - 1) / kTile;
    job.n_scratch_points = n;
    return job;
}
// offsets on the device; total = number of points covered by the offsets
// tile_off / tb_off: this job's slice of d_tiles / d_tile_begin (chunks of a batch that run concurrently)
IcpJob icp_batch_job(locreg_handle* h, const float4* src, const long long* d_offsets, unsigned int S, size_t total, size_t tile_off = 0,
                     size_t tb_off = 0) {
    IcpJob job;
    h->d_tile_begin.reserve((tb_off + static_cast<size_t>(S) + 1) * sizeof(unsigned int));
    h->d_states.reserve(static_cast<size_t>(S) * sizeof(AlignState));
    unsigned int* const tile_begin = h->d_tile_begin.as<unsigned int>() + tb_off;
    LR_LAUNCH(k_tile_begin, 1, 1024, 0, h->stream, d_offsets, S, tile_begin);
    job.bv.src = src; job.bv.offsets = d_offsets; job.bv.tile_begin = tile_begin;
    job.bv.n_single = 0; job.bv.tiles_per_item = 0; job.bv.S = S;
    job.states = h->d_states.as<AlignState>();
    job.n_tiles = static_cast<unsigned int>(std::min<size_t>(total / kTile + S, 0x7fffffffu));
    job.n_scratch_points = total;
    job.bv.tiles = nullptr;
    if (job.n_tiles) {
        h->d_tiles.reserve((tile_off + static_cast<size_t>(job.n_tiles)) * sizeof(TileRec));
        LR_LAUNCH(k_tile_table, (job.n_tiles + 255) / 256, 256, 0, h->stream, job.bv, job.n_tiles, h->d_tiles.as<TileRec>() + tile_off);
        job.bv.tiles = h->d_tiles.as<TileRec>() + tile_off;
        job.bv.n_table_tiles = job.n_tiles;
    }
    return job;
}

bool is_ndt(const locreg_handle* h) { return h->opt.method == LOCREG_NDT_DIRECT || h->opt.method == LOCREG_NDT_INCREMENTAL; }

int check_cloud_args(const float* p, size_t n, size_t stride) {
    if ((n > 0 && p == nullptr) || stride < 12 || (stride % 4) != 0) {
        g_last_error = "invalid cloud arguments (null pointer, stride < 12 or stride not a multiple of 4)";
        return LOCREG_E_ARG;
    }
    if (n >= (1ull << 31)) { g_last_error = "cloud too large"; return LOCREG_E_ARG; }
    return LOCREG_OK;
}

void fill_result(locreg_result* out, const DevResult& r) {
    if (!out) return;
    static_assert(sizeof(locreg_result) == sizeof(DevResult), "result layout");
    std::memcpy(out, &r, sizeof(DevResult));
}

template <class F>
int guarded(locreg_handle* h, F&& f) {
    if (!h) { g_last_error = "null handle"; return LOCREG_E_ARG; }
    try {
        if (cudaSetDevice(h->device) != cudaSuccess) { g_last_error = "cudaSetDevice failed"; cudaGetLastError(); return LOCREG_E_CUDA; }
        return f();
    } catch (const CudaError& e) {
        g_last_error = e.what();
        cudaGetLastError();
        return LOCREG_E_CUDA;
    } catch (const NcclError& e) {
        g_last_error = e.what();
        return LOCREG_E_CUDA;
    } catch (const std::invalid_argument& e) {
        g_last_error = e.what();
        return LOCREG_E_ARG;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return LOCREG_E_CUDA;
    }
}

}  // namespace

extern "C" {

const char* locreg_last_error(void) { return g_last_error.c_str(); }
const char* locreg_version(void) { return "locreg-b200 0.1 (sm_100a)"; }

int locreg_default_options(locreg_options* o, int32_t method) {
    if (!o) return LOCREG_E_ARG;
    std::memset(o, 0, sizeof(*o));
    o->method = method;
    o->max_iteration = 20;
    o->min_effective_pts = 10;
    o->use_ann = 0;
    o->eps = 1e-2;
    o->max_nn_distance = 1.0;
    o->max_plane_distance = 0.1;
    o->max_line_distance = 0.5;
    o->voxel_size = 1.0;
    o->res_outlier_th = 20.0;
    o->min_pts_in_voxel = 3;
    o->nearby_type = LOCREG_NEARBY6;
    o->knn_cell_size = 0.5;
    o->knn_lists = 1;
    o->loop_mode = LOCREG_LOOP_PERSISTENT;
    o->ndt_capacity = 100000;
    return LOCREG_OK;
}

int locreg_create(const locreg_options* opt, int32_t device, locreg_handle** out) {
    if (!opt || !out) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    if (opt->method != LOCREG_ICP_P2P && opt->method != LOCREG_ICP_P2LINE && opt->method != LOCREG_ICP_P2PLANE &&
        opt->method != LOCREG_NDT_DIRECT && opt->method != LOCREG_NDT_INCREMENTAL) {
        g_last_error = "unknown method";
        return LOCREG_E_ARG;
    }
    if ((opt->method == LOCREG_NDT_DIRECT || opt->method == LOCREG_NDT_INCREMENTAL) && !(opt->voxel_size > 0)) {
        g_last_error = "voxel_size must be > 0";
        return LOCREG_E_ARG;
    }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        g_last_error = "no CUDA device: locreg has no CPU fallback";
        return LOCREG_E_CUDA;
    }
    if (device < 0 || device >= count) { g_last_error = "device index out of range"; return LOCREG_E_ARG; }
    auto* h = new locreg_handle;
    h->opt = *opt;
    if (!(h->opt.knn_cell_size > 0)) h->opt.knn_cell_size = 0.5;
    h->device = device;
    const int rc = guarded(h, [&]() {
        cudaDeviceProp prop{};
        LR_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) throw std::runtime_error("locreg kernels are built for sm_100a only; found sm_" + std::to_string(prop.major * 10 + prop.minor));
        h->num_sms = prop.multiProcessorCount;
        // stream-ordered scratch (map builds, filters) comes from the device's default pool: keep what it has handed
        // out instead of returning it to the driver at every synchronisation point (the default threshold is 0)
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
        LR_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
        h->stream = h->own_stream;
        LR_CUDA(cudaEventCreate(&h->ev0));
        LR_CUDA(cudaEventCreate(&h->ev1));
        if (h->opt.method == LOCREG_NDT_INCREMENTAL)
            h->inc_ndt_map.configure(h->opt.voxel_size, h->opt.ndt_capacity > 0 ? static_cast<size_t>(h->opt.ndt_capacity) : 100000);
        return LOCREG_OK;
    });
    if (rc != LOCREG_OK) { delete h; return rc; }
    *out = h;
    return LOCREG_OK;
}

int locreg_destroy(locreg_handle* h) {
    if (!h) return LOCREG_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    for (cudaEvent_t e : h->chunk_events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->chunk_done) cudaEventDestroy(e);
    for (cudaEvent_t e : h->loam_ev) if (e) cudaEventDestroy(e);
    for (cudaStream_t st : h->chunk_streams) cudaStreamDestroy(st);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->comm && nccl_api().ok()) nccl_api().CommDestroy(h->comm);
    h->clear_keyframes();
    cudaStream_t s = h->own_stream;
    delete h;
    if (s) cudaStreamDestroy(s);
    return LOCREG_OK;
}

int locreg_set_stream(locreg_handle* h, void* cuda_stream) {
    return guarded(h, [&]() {
        LR_CUDA(cudaStreamSynchronize(h->stream));
        h->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : h->own_stream;
        return LOCREG_OK;
    });
}

static int set_target_impl(locreg_handle* h, const float* xyz, size_t n, size_t stride, bool on_device) {
    const int rc = check_cloud_args(xyz, n, stride);
    if (rc) return rc;
    return guarded(h, [&]() {
        const void* d_xyz = xyz;
        if (!on_device && n) {
            h->d_target.reserve(n * stride);
            if (is_pinned_or_device(xyz)) {
                LR_CUDA(cudaMemcpyAsync(h->d_target.p, xyz, n * stride, cudaMemcpyHostToDevice, h->stream));
            } else {
                LR_CUDA(cudaMemcpy(h->d_target.p, xyz, n * stride, cudaMemcpyHostToDevice));
            }
            d_xyz = h->d_target.p;
        }
        h->begin_timing();
        if (h->opt.method == LOCREG_NDT_DIRECT) {
            h->ndt_map.build(d_xyz, n, stride, h->opt.voxel_size, h->opt.min_pts_in_voxel, h->stream);
        } else if (h->opt.method == LOCREG_NDT_INCREMENTAL) {
            // SetIncNdtTargetCloud ADDS the cloud to the voxel cache: LRU order, evictions and statistics all on the device
            h->inc_ndt_map.add_cloud(d_xyz, n, stride, h->stream);
        } else {
            static const bool use_mid = !(getenv("LOCREG_MID") && atoi(getenv("LOCREG_MID")) == 0);
            if (!use_mid) h->icp_mid.clear();
            build_icp_maps(h->icp_map, h->icp_coarse, use_mid ? &h->icp_mid : nullptr, d_xyz, n, stride, static_cast<float>(h->opt.knn_cell_size), h->opt.knn_lists != 0, h->stream);
        }
        h->end_timing();
        h->has_target = true;
        return LOCREG_OK;
    });
}
int locreg_set_target(locreg_handle* h, const float* xyz, size_t n, size_t stride) { return set_target_impl(h, xyz, n, stride, false); }
int locreg_set_target_device(locreg_handle* h, const float* d_xyz, size_t n, size_t stride) { return set_target_impl(h, d_xyz, n, stride, true); }

int locreg_align(locreg_handle* h, const float* src, size_t n, size_t stride, const double* pose_in, double* pose_out,
                 float* out_xyz, locreg_result* res) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!pose_in || !pose_out) { g_last_error = "null pose"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        const float4* src4 = stage_cloud(h, src, n, stride, false);
        init_state(h, pose_in, true);
        h->begin_timing();
        if (is_ndt(h)) {
            NDT_DISPATCH(h, ndt_run_align(h, PB, src4, static_cast<unsigned int>(n)));
        } else {
            const IcpJob job = icp_single_job(h, src4, static_cast<unsigned int>(n));
            bool ran = false;
            // (P2P / P2Line stage three residual rows per point: their tile bodies together exceed the static shared memory
            // of one kernel, so they keep the per-iteration pipeline)
            if (h->opt.loop_mode == LOCREG_LOOP_PERSISTENT && h->opt.method == LOCREG_ICP_P2PLANE) ran = icp_run_persistent<kIcpP2Plane>(h, job);
            if (!ran) ICP_DISPATCH(h, icp_run_loop<M>(h, job, 0));
        }
        AlignState* st = h->d_state.as<AlignState>();
        const size_t bytes = n * stride;
        if (out_xyz && n) {
            h->d_out.reserve(bytes);
            const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((n + 255) / 256, 4096));
            LR_LAUNCH(k_transform, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>(), h->d_out.as<unsigned char>(), n, stride, st->pose);
        }
        h->h_small.reserve(4096);
        AlignState* hs = h->h_small.as<AlignState>() + 1;
        LR_CUDA(cudaMemcpyAsync(hs, st, sizeof(AlignState), cudaMemcpyDeviceToHost, h->stream));
        const bool direct_out = out_xyz && n && is_pinned_or_device(out_xyz);
        if (out_xyz && n) {
            if (direct_out) {
                LR_CUDA(cudaMemcpyAsync(out_xyz, h->d_out.p, bytes, cudaMemcpyDeviceToHost, h->stream));
            } else {
                h->h_out.reserve(bytes);
                LR_CUDA(cudaMemcpyAsync(h->h_out.p, h->d_out.p, bytes, cudaMemcpyDeviceToHost, h->stream));
            }
        }
        h->end_timing();  // synchronises the stream
        if (hs->res.pose_written) {
            std::memcpy(pose_out, hs->pose, 7 * sizeof(double));
        } else if (out_xyz && n) {
            // direct NDT's early return: result_pose keeps the caller's value and the cloud is transformed with it
            double* dpose = h->d_acc.as<double>();
            h->d_acc.reserve(32 * sizeof(double));
            dpose = h->d_acc.as<double>();
            LR_CUDA(cudaMemcpyAsync(dpose, pose_out, 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((n + 255) / 256, 4096));
            LR_LAUNCH(k_transform, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>(), h->d_out.as<unsigned char>(), n, stride, dpose);
            LR_CUDA(cudaMemcpyAsync(direct_out ? static_cast<void*>(out_xyz) : h->h_out.p, h->d_out.p, bytes, cudaMemcpyDeviceToHost, h->stream));
            LR_CUDA(cudaStreamSynchronize(h->stream));
        }
        if (out_xyz && n && !direct_out) std::memcpy(out_xyz, h->h_out.p, bytes);
        fill_result(res, hs->res);
        return LOCREG_OK;
    });
}

int locreg_compute_hb(locreg_handle* h, const float* src, size_t n, size_t stride, const double* pose, double* H36,
                      double* B6, locreg_result* res) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!pose || !H36 || !B6) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        const float4* src4 = stage_cloud(h, src, n, stride, false);
        init_state(h, pose);
        h->begin_timing();
        h->d_acc.reserve(32 * sizeof(double));
        if (is_ndt(h)) {
            NDT_DISPATCH(h, ndt_run_eval(h, PB, src4, static_cast<unsigned int>(n), nullptr));
        } else {
            const IcpJob job = icp_single_job(h, src4, static_cast<unsigned int>(n));
            ICP_DISPATCH(h, (icp_launch_eval<M>(h, job, 1, kNnTwoPass, nullptr, nullptr), icp_launch_solve<M>(h, job, 0, h->d_acc.as<double>())));
        }
        h->h_small.reserve(4096);
        double* acc = h->h_small.as<double>() + 64;
        LR_CUDA(cudaMemcpyAsync(acc, h->d_acc.p, 30 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        h->end_timing();
        for (int r = 0; r < 6; ++r)
            for (int c = r; c < 6; ++c) { H36[c * 6 + r] = acc[hidx(r, c)]; H36[r * 6 + c] = acc[hidx(r, c)]; }
        for (int i = 0; i < 6; ++i) B6[i] = acc[21 + i];
        DevResult r{};
        r.n_effective = static_cast<long long>(acc[28]);
        r.n_inlier = static_cast<long long>(acc[29]);
        r.sum_sq_res = acc[27];
        r.pose_written = 1;
        double dx[6];
        const bool solvable = gn_solve6(acc, acc + 21, dx);
        const bool few = r.n_effective < h->opt.min_effective_pts;
        r.degenerate = (!solvable || (few && h->opt.method != LOCREG_NDT_DIRECT)) ? 1 : 0;  // direct NDT only looks at det(H) here
        fill_result(res, r);
        return LOCREG_OK;
    });
}

static int loam_check_handles(const locreg_handle* surf, const locreg_handle* edge) {
    if (!surf || !edge) { g_last_error = "null handle"; return LOCREG_E_ARG; }
    if (surf == edge) { g_last_error = "locreg_align_loam needs two distinct handles (surf and edge)"; return LOCREG_E_ARG; }
    if (surf->device != edge->device) { g_last_error = "surf and edge handles are on different devices"; return LOCREG_E_ARG; }
    if (surf->opt.method != LOCREG_ICP_P2PLANE || edge->opt.method != LOCREG_ICP_P2LINE) {
        g_last_error = "locreg_align_loam needs a LOCREG_ICP_P2PLANE surf handle and a LOCREG_ICP_P2LINE edge handle";
        return LOCREG_E_ARG;
    }
    return LOCREG_OK;
}

// One half of a LOAM call: offsets (S + 1, host, relative to xyz) of the batch, or nullptr for one scan of n points.
struct LoamHalf {
    const float* xyz;
    const int64_t* offsets;
    size_t n;
};

// Offsets of one half of locreg_align_loam_batch: non-negative and non-decreasing, the cloud they cover valid.
static int loam_check_half(const LoamHalf& c, size_t stride, size_t S, const char* name) {
    if (!c.offsets) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    for (size_t s = 0; s < S; ++s)
        if (c.offsets[s] < 0 || c.offsets[s + 1] < c.offsets[s]) {
            g_last_error = std::string(name) + " offsets must be non-negative and non-decreasing";
            return LOCREG_E_ARG;
        }
    return check_cloud_args(c.xyz, static_cast<size_t>(c.offsets[S] - c.offsets[0]), stride);
}

// Stages one half's cloud with one copy on its handle's stream; a batch's offsets go to the device relative to it.
static const float4* loam_stage_half(locreg_handle* h, const LoamHalf& c, size_t stride, size_t S) {
    if (!c.offsets) return stage_cloud(h, c.xyz, c.n, stride, false);
    const size_t base = static_cast<size_t>(c.offsets[0]), n_pts = static_cast<size_t>(c.offsets[S]) - base;
    h->h_small.reserve((S + 1) * sizeof(long long));
    long long* rel = h->h_small.as<long long>();
    for (size_t s = 0; s <= S; ++s) rel[s] = c.offsets[s] - static_cast<long long>(base);
    h->d_offsets.reserve((S + 1) * sizeof(long long));
    LR_CUDA(cudaMemcpyAsync(h->d_offsets.p, rel, (S + 1) * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    return stage_cloud(h, reinterpret_cast<const float*>(reinterpret_cast<const char*>(c.xyz) + base * stride), n_pts, stride, false);
}

// One half's job over the S scans (one scan: offsets == nullptr).
static IcpJob loam_half_job(locreg_handle* h, const LoamHalf& c, const float4* src4, size_t S) {
    if (!c.offsets) {
        h->d_state.reserve(sizeof(AlignState));
        return icp_single_job(h, src4, static_cast<unsigned int>(c.n));
    }
    const size_t n_pts = static_cast<size_t>(c.offsets[S] - c.offsets[0]);
    IcpJob job = icp_batch_job(h, src4, h->d_offsets.as<long long>(), static_cast<unsigned int>(S), n_pts);
    if (n_pts == 0) job.n_tiles = 0;  // no point in the whole half: its evaluation launches nothing (its tiles would all exit)
    return job;
}

// locreg_align_loam (S = 1, no offsets) and locreg_align_loam_batch: S independent LOAM loops in one.  The states live
// with the surf job (the edge job points at them); surf->d_loam holds the poses, the loop results and the halves'
// records, copied back in one piece through surf->h_out.
static int loam_prepare(locreg_handle* surf, const locreg_handle* edge) {
    if (!surf->has_target || !edge->has_target) {
        g_last_error = surf->has_target ? "SetInputTarget has not been called on the edge handle"
                                        : "SetInputTarget has not been called on the surf handle";
        return LOCREG_E_STATE;
    }
    for (cudaEvent_t& e : surf->loam_ev)
        if (!e) LR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return LOCREG_OK;
}

static int loam_align(locreg_handle* surf, locreg_handle* edge, const LoamHalf& cs, const LoamHalf& ce, size_t stride,
                      const double* poses_in, size_t S, int32_t max_iteration, double eps, double* poses_out, locreg_result* results) {
    const int rc = loam_prepare(surf, edge);
    if (rc) return rc;
    const unsigned int Su = static_cast<unsigned int>(S);
    // d_loam / h_out: [S x 7 poses][S loop results][2S halves]
    const size_t res_off = S * 7 * sizeof(double), half_off = res_off + S * sizeof(DevResult), bytes = half_off + 2 * S * sizeof(DevResult);
    surf->d_loam.reserve(bytes);
    surf->h_out.reserve(bytes);
    unsigned char* const d = surf->d_loam.as<unsigned char>();
    unsigned char* const hb = surf->h_out.as<unsigned char>();
    double* const d_poses = reinterpret_cast<double*>(d);
    DevResult* const d_res = reinterpret_cast<DevResult*>(d + res_off);
    DevResult* const d_half = reinterpret_cast<DevResult*>(d + half_off);
    const float4* src_s = loam_stage_half(surf, cs, stride, S);
    const float4* src_e = loam_stage_half(edge, ce, stride, S);
    std::memcpy(hb, poses_in, S * 7 * sizeof(double));
    LR_CUDA(cudaMemcpyAsync(d_poses, hb, S * 7 * sizeof(double), cudaMemcpyHostToDevice, surf->stream));
    LR_CUDA(cudaMemsetAsync(d_half, 0, 2 * S * sizeof(DevResult), surf->stream));
    surf->begin_timing();
    IcpJob js = loam_half_job(surf, cs, src_s, S);
    IcpJob je = loam_half_job(edge, ce, src_e, S);
    je.states = js.states;  // one state, one pose per scan: both halves evaluate at it
    // CaculateMatrixHAndB ignores zero_initial_translation: so does the LOAM loop
    LR_LAUNCH(k_states_init, (Su + 255) / 256, 256, 0, surf->stream, d_poses, Su, max_iteration, 0, js.states);
    loam_run_loop(surf, edge, js, je, max_iteration, eps, d_half);
    LR_LAUNCH(k_states_export, (Su + 255) / 256, 256, 0, surf->stream, js.states, Su, d_poses, d_res);
    LR_CUDA(cudaMemcpyAsync(hb, d, bytes, cudaMemcpyDeviceToHost, surf->stream));
    surf->end_timing();  // synchronises surf's stream, which has joined edge's
    std::memcpy(poses_out, hb, S * 7 * sizeof(double));
    const DevResult* hr = reinterpret_cast<const DevResult*>(hb + res_off);
    const DevResult* hh = reinterpret_cast<const DevResult*>(hb + half_off);
    for (size_t i = 0; results && i < 2 * S; ++i) {  // the loop's bookkeeping, the half's last evaluation
        DevResult r = hh[i];
        const DevResult& loop = hr[i / 2];
        r.iters = loop.iters;
        r.updates = loop.updates;
        r.converged = loop.converged;
        r.pose_written = loop.pose_written;
        fill_result(results + i, r);
    }
    return LOCREG_OK;
}

int locreg_align_loam(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf, const float* edge_xyz,
                      size_t n_edge, size_t stride, const double* pose_in, int32_t max_iteration, double eps, double* pose_out,
                      locreg_result* res2) {
    int rc = loam_check_handles(surf, edge);
    if (rc) return rc;
    rc = check_cloud_args(surf_xyz, n_surf, stride);
    if (rc) return rc;
    rc = check_cloud_args(edge_xyz, n_edge, stride);
    if (rc) return rc;
    if (!pose_in || !pose_out) { g_last_error = "null pose"; return LOCREG_E_ARG; }
    return guarded(surf, [&]() {
        return loam_align(surf, edge, LoamHalf{surf_xyz, nullptr, n_surf}, LoamHalf{edge_xyz, nullptr, n_edge}, stride, pose_in, 1,
                          max_iteration, eps, pose_out, res2);
    });
}

int locreg_align_loam_batch(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, const int64_t* surf_offsets,
                            const float* edge_xyz, const int64_t* edge_offsets, size_t stride, const double* poses_in, size_t S,
                            int32_t max_iteration, double eps, double* poses_out, locreg_result* results) {
    int rc = loam_check_handles(surf, edge);
    if (rc) return rc;
    if (S >= (1ull << 31)) { g_last_error = "too many scans"; return LOCREG_E_ARG; }
    if (S == 0) return LOCREG_OK;
    const LoamHalf cs{surf_xyz, surf_offsets, 0}, ce{edge_xyz, edge_offsets, 0};
    rc = loam_check_half(cs, stride, S, "surf");
    if (rc) return rc;
    rc = loam_check_half(ce, stride, S, "edge");
    if (rc) return rc;
    if (!poses_in || !poses_out) { g_last_error = "null pose"; return LOCREG_E_ARG; }
    return guarded(surf, [&]() { return loam_align(surf, edge, cs, ce, stride, poses_in, S, max_iteration, eps, poses_out, results); });
}

int locreg_knn(locreg_handle* h, const float* queries, size_t nq, size_t stride, int32_t k, int32_t* idx) {
    const int rc = check_cloud_args(queries, nq, stride);
    if (rc) return rc;
    if ((k != 1 && k != 5) || !idx) { g_last_error = "k must be 1 or 5"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (h->opt.method == LOCREG_NDT_DIRECT) { g_last_error = "k-NN probe needs an ICP handle"; return LOCREG_E_STATE; }
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        if (nq == 0) return LOCREG_OK;
        const float4* q4 = stage_cloud(h, queries, nq, stride, false);
        h->d_nn.reserve(nq * k * sizeof(int));
        h->d_nnpos.reserve(nq * k * sizeof(unsigned int));
        h->d_ringq.reserve(nq * sizeof(uint2));
        h->d_ringc.reserve(sizeof(unsigned int));
        LR_CUDA(cudaMemsetAsync(h->d_ringc.p, 0, sizeof(unsigned int), h->stream));
        const RingQueue queue{h->d_ringc.as<unsigned int>(), h->d_ringq.as<uint2>()};
        h->begin_timing();
        // the production search: stage 1 per thread, then the queued rest per warp (small: what a single scan runs) or
        // per thread (large: what batches run) - the probe switches at the same job size as icp_launch_eval
        const unsigned int n32 = static_cast<unsigned int>(nq);
        const unsigned int g1 = (n32 + kTile - 1) / kTile;
        const bool small = g1 <= 2u * static_cast<unsigned int>(h->num_sms);
        const unsigned int g2 = static_cast<unsigned int>(std::min<size_t>(small ? (nq + 3) / 4 : (nq + 127) / 128, static_cast<size_t>(h->num_sms) * 8));
        const unsigned int g3 = static_cast<unsigned int>((nq * k + 255) / 256);
        if (k == 1) {
            LR_LAUNCH(k_knn_stage1<1>, g1, kTile, 0, h->stream, h->icp_map.view(), q4, n32, h->d_nnpos.as<unsigned int>(), queue);
            if (small) LR_LAUNCH(k_knn_rings<1>, g2, 128, 0, h->stream, h->icp_map.view(), h->coarse_views(), q4, h->d_nnpos.as<unsigned int>(), queue);
            else LR_LAUNCH(k_knn_finish<1>, g2, 128, 0, h->stream, h->icp_map.view(), h->coarse_views(), q4, h->d_nnpos.as<unsigned int>(), queue);
        } else {
            LR_LAUNCH(k_knn_stage1<5>, g1, kTile, 0, h->stream, h->icp_map.view(), q4, n32, h->d_nnpos.as<unsigned int>(), queue);
            if (small) LR_LAUNCH(k_knn_rings<5>, g2, 128, 0, h->stream, h->icp_map.view(), h->coarse_views(), q4, h->d_nnpos.as<unsigned int>(), queue);
            else LR_LAUNCH(k_knn_finish<5>, g2, 128, 0, h->stream, h->icp_map.view(), h->coarse_views(), q4, h->d_nnpos.as<unsigned int>(), queue);
        }
        LR_LAUNCH(k_knn_export, g3, 256, 0, h->stream, h->icp_map.view(), h->d_nnpos.as<unsigned int>(), nq * k, h->d_nn.as<int>());
        LR_CUDA(cudaMemsetAsync(h->d_ringc.p, 0, sizeof(unsigned int), h->stream));
        h->end_timing();
        LR_CUDA(cudaMemcpy(idx, h->d_nn.p, nq * k * sizeof(int), cudaMemcpyDeviceToHost));
        return LOCREG_OK;
    });
}

int locreg_debug_points(locreg_handle* h, const float* src, size_t n, size_t stride, const double* pose, uint8_t* gate,
                        int32_t* nn) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!pose || !gate) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        if (n == 0) return LOCREG_OK;
        const float4* src4 = stage_cloud(h, src, n, stride, false);
        init_state(h, pose);
        const int k = h->opt.method == LOCREG_ICP_P2P ? 1 : (h->opt.method == LOCREG_NDT_DIRECT ? 0 : 5);
        h->d_gate.reserve(n);
        int* d_nn = nullptr;
        if (nn && k) { h->d_nn.reserve(n * k * sizeof(int)); d_nn = h->d_nn.as<int>(); }
        h->begin_timing();
        if (is_ndt(h)) {
            NDT_DISPATCH(h, ndt_run_eval(h, PB, src4, static_cast<unsigned int>(n), h->d_gate.as<unsigned char>()));
        } else {
            const IcpJob job = icp_single_job(h, src4, static_cast<unsigned int>(n));
            ICP_DISPATCH(h, icp_launch_eval<M>(h, job, 1, kNnTwoPass, h->d_gate.as<unsigned char>(), d_nn));
        }
        h->end_timing();
        LR_CUDA(cudaMemcpy(gate, h->d_gate.p, n, cudaMemcpyDeviceToHost));
        if (d_nn) LR_CUDA(cudaMemcpy(nn, d_nn, n * k * sizeof(int), cudaMemcpyDeviceToHost));
        return LOCREG_OK;
    });
}

int locreg_align_batch_device(locreg_handle* h, const float* d_srcs, const int64_t* d_offsets, const double* d_poses_in,
                              size_t S, size_t total_points, double* d_poses_out, locreg_result* d_results) {
    if (!d_srcs || !d_offsets || !d_poses_in || !d_poses_out) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    if (S >= (1ull << 31)) { g_last_error = "too many scans"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        if (S == 0) return LOCREG_OK;
        h->begin_timing();
        const float4* src4 = reinterpret_cast<const float4*>(d_srcs);
        const long long* offs = reinterpret_cast<const long long*>(d_offsets);
        DevResult* results = reinterpret_cast<DevResult*>(d_results);
        const unsigned int Su = static_cast<unsigned int>(S);
        if (is_ndt(h)) {
            NDT_DISPATCH(h, ndt_run_batch(h, PB, src4, offs, d_poses_in, d_poses_out, results, Su));
        } else {
            const IcpJob job = icp_batch_job(h, src4, offs, Su, total_points);
            LR_LAUNCH(k_states_init, (Su + 255) / 256, 256, 0, h->stream, d_poses_in, Su, h->opt.max_iteration, h->opt.zero_initial_translation, job.states);
            ICP_DISPATCH(h, icp_run_loop<M>(h, job, 0));
            LR_LAUNCH(k_states_export, (Su + 255) / 256, 256, 0, h->stream, job.states, Su, d_poses_out, results);
        }
        h->end_timing();
        return LOCREG_OK;
    });
}

// S ScanMatch calls of a host batch; the poses and results stay in h->d_poses_out / h->d_results (S entries, device).
// offsets[0..S] are relative to srcs; poses_out_init = the IN values of the IN/OUT poses_out.
static void align_batch_resident(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride, const double* poses_in,
                                 size_t S, const double* poses_out_init) {
    NvtxRange nvtx_r("locreg:align_batch");
    const size_t total = static_cast<size_t>(offsets[S]);
    const float* first = reinterpret_cast<const float*>(reinterpret_cast<const char*>(srcs) + static_cast<size_t>(offsets[0]) * stride);
    const double* poses_out = poses_out_init;
    const size_t base = static_cast<size_t>(offsets[0]);
    const size_t n_pts = total - base;
    // Large ICP batches from pinned (or device-visible) memory are cut into chunks of whole scans: the copy of
    // chunk c + 1 runs on a second stream while chunk c is being registered (scans are independent).
    const bool pipelined = !is_ndt(h) && S >= 16 && n_pts >= (1u << 20) && is_pinned_or_device(first);
    const float4* src4 = pipelined ? nullptr : stage_cloud(h, first, n_pts, stride, false);
    h->d_offsets.reserve((S + 1) * sizeof(long long));
    h->d_poses_in.reserve(S * 7 * sizeof(double));
    h->d_poses_out.reserve(S * 7 * sizeof(double));
    h->d_results.reserve(S * sizeof(DevResult));
    std::vector<long long> rel(S + 1);
    for (size_t s = 0; s <= S; ++s) rel[s] = offsets[s] - static_cast<long long>(base);
    LR_CUDA(cudaMemcpyAsync(h->d_offsets.p, rel.data(), (S + 1) * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(h->d_poses_in.p, poses_in, S * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(h->d_poses_out.p, poses_out, S * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaStreamSynchronize(h->stream));  // rel[] is pageable
    const unsigned int Su = static_cast<unsigned int>(S);
    if (pipelined) {
        // LOCREG_CHUNK_STREAMS (default 1): every chunk runs its Gauss-Newton loop on its own stream as soon as its copy has
        // landed, concurrently with the chunks before it.  A chunk's loop is ~70 dependent kernels, each ending in a tail
        // in which the GPU drains (measured: +1.1 to 1.8 ms per additional chunk when the chunks run one after the other);
        // the blocks of another chunk's kernels fill those tails.  Each chunk owns a slice of the per-job scratch (IcpJob).
        static const int streams_env = getenv("LOCREG_CHUNK_STREAMS") ? atoi(getenv("LOCREG_CHUNK_STREAMS")) : 1;
        static const bool fused_env = getenv("LOCREG_FUSED") && atoi(getenv("LOCREG_FUSED")) != 0;
        static const bool sort_batch_env = getenv("LOCREG_SORT_BATCH") && atoi(getenv("LOCREG_SORT_BATCH")) != 0;
        const bool may_run_concurrently = streams_env && !h->profile && !fused_env && !sort_batch_env;
        // Chunk weights (relative point counts): LOCREG_CHUNK_WEIGHTS="w0,w1,...", else LOCREG_CHUNKS chunks growing by
        // LOCREG_CHUNK_RATIO, else the measured optimum.  Only the first chunk's copy is exposed, and a chunk's copy hides
        // behind the compute of the chunks before it (compute takes ~4x as long as the copy of the same points).
        // Measured on B200 (512 scans, 226 MB, profiles/r2_chunk_streams.txt), M points/s end to end:
        //   concurrent chunks: 1:2:3:3 782, 1:3:3:3 780, 1:4:4 777, 1:1:1:1 772, 1:4 726, 1:8 707   (resident: 827)
        //   one after the other: 1:8 707, 1:4:4 669, 1:3:4:4 616, equal halves 674
        static const std::vector<double> kEnvWeights = []() {
            std::vector<double> w;
            if (const char* e = getenv("LOCREG_CHUNK_WEIGHTS")) {
                for (const char* p = e; *p;) {
                    char* end = nullptr;
                    const double v = strtod(p, &end);
                    if (end == p) break;
                    if (v > 0.0) w.push_back(v);
                    if (*end != ',') break;
                    p = end + 1;
                }
                if (w.size() > 16) w.resize(16);
            } else if (getenv("LOCREG_CHUNKS") || getenv("LOCREG_CHUNK_RATIO")) {
                const size_t n = getenv("LOCREG_CHUNKS") ? std::max(1, std::min(16, atoi(getenv("LOCREG_CHUNKS")))) : 2;
                const double ratio = getenv("LOCREG_CHUNK_RATIO") ? std::min(16.0, std::max(1.0, atof(getenv("LOCREG_CHUNK_RATIO")))) : 8.0;
                double v = 1.0;
                for (size_t c = 0; c < n; ++c, v *= ratio) w.push_back(v);
            }
            return w;
        }();
        static const std::vector<double> kConcurrentWeights{1.0, 2.0, 3.0, 3.0}, kSerialWeights{1.0, 8.0}, kHugeWeights{1.0, 3.0, 9.0, 27.0, 41.0};
        // (four chunks only where every one of them still fills the GPU: from 4 M points on.  What is exposed is the FIRST
        // chunk's copy, and ~25 MB is as small as it usefully gets: a 4096-scan batch (113 M points, 1.8 GB) measured 875 M
        // points/s end to end at 1:3:9:27:41 against 824 M at 1:2:3:3 and 936 M resident - profiles/r2_chunk_streams.txt)
        const std::vector<double>& kWeights = !kEnvWeights.empty() ? kEnvWeights
                                              : !may_run_concurrently || n_pts < (4u << 20) ? kSerialWeights
                                              : n_pts < (32u << 20) ? kConcurrentWeights : kHugeWeights;
        const size_t kChunks = kWeights.size();
        if (!h->copy_stream) LR_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        while (h->chunk_events.size() < kChunks) {
            cudaEvent_t e;
            LR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->chunk_events.push_back(e);
        }
        h->d_raw.reserve(n_pts * stride);
        if (stride != 16) h->d_src4.reserve(n_pts * sizeof(float4));
        h->d_states.reserve(S * sizeof(AlignState));
        // chunk boundaries: whole scans, about equal point counts
        std::vector<size_t> cut{0};
        double total_w = 0.0, acc_w = 0.0;
        for (size_t c = 0; c < kChunks; ++c) total_w += kWeights[c];
        for (size_t c = 1; c < kChunks; ++c) {
            acc_w += kWeights[c - 1];
            const long long want = static_cast<long long>(static_cast<double>(n_pts) * acc_w / total_w);
            size_t s = std::lower_bound(rel.begin(), rel.end(), want) - rel.begin();
            s = std::min(std::max(s, cut.back()), S);
            cut.push_back(s);
        }
        cut.push_back(S);
        for (size_t c = 0; c < kChunks; ++c) {
            const size_t p0 = static_cast<size_t>(rel[cut[c]]), p1 = static_cast<size_t>(rel[cut[c + 1]]);
            if (p1 > p0)
                LR_CUDA(cudaMemcpyAsync(h->d_raw.as<unsigned char>() + p0 * stride, reinterpret_cast<const char*>(first) + p0 * stride,
                                        (p1 - p0) * stride, cudaMemcpyHostToDevice, h->copy_stream));
            LR_CUDA(cudaEventRecord(h->chunk_events[c], h->copy_stream));
        }
        const bool concurrent = may_run_concurrently && kChunks > 1;
        std::vector<size_t> tile_off(kChunks + 1, 0);
        for (size_t c = 0; c < kChunks; ++c) {
            const size_t pts = static_cast<size_t>(rel[cut[c + 1]] - rel[cut[c]]);
            tile_off[c + 1] = tile_off[c] + pts / kTile + (cut[c + 1] - cut[c]);  // icp_batch_job's n_tiles
        }
        if (concurrent) {
            // everything the chunks share is allocated before the first launch: a later reserve() must never move a buffer
            const size_t K5 = h->opt.method == LOCREG_ICP_P2P ? 1 : 5;
            h->d_partials.reserve(2 * tile_off[kChunks] * kPartialDoubles * sizeof(double));
            h->d_tiles.reserve(tile_off[kChunks] * sizeof(TileRec));
            h->d_tile_begin.reserve((S + kChunks) * sizeof(unsigned int));
            h->d_ringc.reserve(2 * kChunks * sizeof(unsigned int));
            h->d_nnpos.reserve(n_pts * K5 * sizeof(unsigned int));
            h->d_ringq.reserve(n_pts * sizeof(uint2));
            h->d_track.reserve(n_pts * sizeof(KnnTrack));
            if (h->opt.method == LOCREG_ICP_P2PLANE) {
                h->d_same.reserve(n_pts);
                h->d_plane.reserve(n_pts * 4 * sizeof(double));
                h->d_pstat.reserve(n_pts);
            }
            while (h->chunk_streams.size() + 1 < kChunks) {
                cudaStream_t st;
                LR_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                h->chunk_streams.push_back(st);
                cudaEvent_t e;
                LR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                h->chunk_done.push_back(e);
            }
        }
        h->begin_timing();
        cudaStream_t const main_stream = h->stream;
        for (size_t c = 0; c < kChunks; ++c) {
            const size_t s0 = cut[c], s1 = cut[c + 1];
            // (the launch helpers below issue on h->stream: it is the chunk's stream while the chunk is being queued)
            if (concurrent && c > 0) h->stream = h->chunk_streams[c - 1];
            struct Restore { locreg_handle* h; cudaStream_t s; ~Restore() { h->stream = s; } } restore{h, main_stream};
            LR_CUDA(cudaStreamWaitEvent(h->stream, h->chunk_events[c], 0));
            if (s1 > s0) {
                const size_t p0 = static_cast<size_t>(rel[s0]), p1 = static_cast<size_t>(rel[s1]);
                const unsigned int Sc = static_cast<unsigned int>(s1 - s0);
                if (stride != 16 && p1 > p0) {
                    const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((p1 - p0 + 255) / 256, 4096));
                    LR_LAUNCH(k_pack_float4, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>() + p0 * stride, p1 - p0, stride,
                              h->d_src4.as<float4>() + p0);
                }
                const float4* all4 = stride == 16 ? h->d_raw.as<float4>() : h->d_src4.as<float4>();
                // offsets stay absolute (into the whole batch); only the scan range of the job moves
                IcpJob job = icp_batch_job(h, all4, h->d_offsets.as<long long>() + s0, Sc, p1 - p0, concurrent ? tile_off[c] : 0,
                                           concurrent ? s0 + c : 0);
                job.states = h->d_states.as<AlignState>() + s0;
                job.n_scratch_points = n_pts;  // scratch rows are indexed by absolute point number
                if (concurrent) {
                    job.partials_off = 2 * tile_off[c] * kPartialDoubles;
                    job.ringc_off = 2 * c;
                    job.ringq_off = p0;
                }
                LR_LAUNCH(k_states_init, (Sc + 255) / 256, 256, 0, h->stream, h->d_poses_in.as<double>() + s0 * 7, Sc, h->opt.max_iteration, h->opt.zero_initial_translation, job.states);
                ICP_DISPATCH(h, icp_run_loop<M>(h, job, 0));
                LR_LAUNCH(k_states_export, (Sc + 255) / 256, 256, 0, h->stream, job.states, Sc, h->d_poses_out.as<double>() + s0 * 7,
                          h->d_results.as<DevResult>() + s0);
            }
            if (concurrent && c > 0) {  // the handle's stream ends after every chunk has
                LR_CUDA(cudaEventRecord(h->chunk_done[c - 1], h->stream));
                LR_CUDA(cudaStreamWaitEvent(main_stream, h->chunk_done[c - 1], 0));
            }
        }
        h->end_timing();
    } else {
        h->begin_timing();
        if (is_ndt(h)) {
            NDT_DISPATCH(h, ndt_run_batch(h, PB, src4, h->d_offsets.as<long long>(), h->d_poses_in.as<double>(),
                                          h->d_poses_out.as<double>(), h->d_results.as<DevResult>(), Su));
        } else {
            const IcpJob job = icp_batch_job(h, src4, h->d_offsets.as<long long>(), Su, n_pts);
            LR_LAUNCH(k_states_init, (Su + 255) / 256, 256, 0, h->stream, h->d_poses_in.as<double>(), Su, h->opt.max_iteration, h->opt.zero_initial_translation, job.states);
            ICP_DISPATCH(h, icp_run_loop<M>(h, job, 0));
            LR_LAUNCH(k_states_export, (Su + 255) / 256, 256, 0, h->stream, job.states, Su, h->d_poses_out.as<double>(), h->d_results.as<DevResult>());
        }
        h->end_timing();
    }
}

static int align_batch_check(const float* srcs, const int64_t* offsets, size_t stride, const double* poses_in, size_t S, double* poses_out) {
    if (!offsets || !poses_in || !poses_out) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    if (S >= (1ull << 31)) { g_last_error = "too many scans"; return LOCREG_E_ARG; }
    for (size_t s = 0; s < S; ++s)
        if (offsets[s + 1] < offsets[s] || offsets[s] < 0) { g_last_error = "offsets must be non-decreasing"; return LOCREG_E_ARG; }
    const size_t total = static_cast<size_t>(offsets[S]);
    const float* first = reinterpret_cast<const float*>(reinterpret_cast<const char*>(srcs) + static_cast<size_t>(offsets[0]) * stride);
    return check_cloud_args(first, total - static_cast<size_t>(offsets[0]), stride);
}

int locreg_align_batch(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride, const double* poses_in,
                       size_t S, double* poses_out, locreg_result* results) {
    if (S == 0) return LOCREG_OK;
    const int rc = align_batch_check(srcs, offsets, stride, poses_in, S, poses_out);
    if (rc) return rc;
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        align_batch_resident(h, srcs, offsets, stride, poses_in, S, poses_out);
        LR_CUDA(cudaMemcpy(poses_out, h->d_poses_out.p, S * 7 * sizeof(double), cudaMemcpyDeviceToHost));
        if (results) LR_CUDA(cudaMemcpy(results, h->d_results.p, S * sizeof(DevResult), cudaMemcpyDeviceToHost));
        return LOCREG_OK;
    });
}

int locreg_align_batch_sharded(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride, const double* poses_in,
                               size_t S_local, size_t S_global, double* poses_out, locreg_result* results) {
    if (!h) { g_last_error = "null handle"; return LOCREG_E_ARG; }
    if (!poses_out || S_global >= (1ull << 31)) { g_last_error = "invalid arguments"; return LOCREG_E_ARG; }
    size_t lo = 0, hi = 0;
    locreg_shard_range(S_global, h->comm_rank, h->comm_world, &lo, &hi);
    if (S_local != hi - lo) { g_last_error = "S_local must be this rank's block of locreg_shard_range(S_global, rank, world)"; return LOCREG_E_ARG; }
    if (S_local) {
        const int rc = align_batch_check(srcs, offsets, stride, poses_in, S_local, poses_out);
        if (rc) return rc;
    }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        if (S_global == 0) return LOCREG_OK;
        if (S_local) align_batch_resident(h, srcs, offsets, stride, poses_in, S_local, poses_out + lo * 7);
        // exchange: every rank's block into the global arrays, on the handle's stream (ragged all-gather = one grouped
        // broadcast per rank)
        h->d_gather_pose.reserve(S_global * 7 * sizeof(double));
        h->d_gather_res.reserve(S_global * sizeof(DevResult));
        const NcclApi& nc = nccl_api();
        if (h->comm) {
            NvtxRange r("locreg:align_batch:allgather");
            LR_NCCL(nc.GroupStart());
            for (int r = 0; r < h->comm_world; ++r) {
                size_t rlo = 0, rhi = 0;
                locreg_shard_range(S_global, r, h->comm_world, &rlo, &rhi);
                if (rhi == rlo) continue;
                const bool me = r == h->comm_rank;
                LR_NCCL(nc.Broadcast(me ? h->d_poses_out.p : nullptr, h->d_gather_pose.as<double>() + rlo * 7, (rhi - rlo) * 7, ncclDouble, r, h->comm, h->stream));
                LR_NCCL(nc.Broadcast(me ? h->d_results.p : nullptr, h->d_gather_res.as<DevResult>() + rlo, (rhi - rlo) * sizeof(DevResult), ncclUint8, r, h->comm, h->stream));
            }
            LR_NCCL(nc.GroupEnd());
        } else if (S_local) {
            LR_CUDA(cudaMemcpyAsync(h->d_gather_pose.p, h->d_poses_out.p, S_local * 7 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
            LR_CUDA(cudaMemcpyAsync(h->d_gather_res.p, h->d_results.p, S_local * sizeof(DevResult), cudaMemcpyDeviceToDevice, h->stream));
        }
        LR_CUDA(cudaMemcpyAsync(poses_out, h->d_gather_pose.p, S_global * 7 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (results) LR_CUDA(cudaMemcpyAsync(results, h->d_gather_res.p, S_global * sizeof(DevResult), cudaMemcpyDeviceToHost, h->stream));
        LR_CUDA(cudaStreamSynchronize(h->stream));
        return LOCREG_OK;
    });
}

uint64_t locreg_pack_score(double score, uint32_t index) {
    float f = static_cast<float>(score);
    if (!(f == f) || f < 0) f = INFINITY;
    uint32_t bits;
    std::memcpy(&bits, &f, 4);
    return (static_cast<uint64_t>(bits) << 32) | index;
}

// Hypotheses per wave of a relocalisation of n_hyp hypotheses.  Hypotheses run in waves so that the per-point neighbour
// scratch (K rows per point) stays bounded; the rest of the per-point scratch - planes, margins, queues - scales with it
// (~4.5 GiB in all for P2Plane at 1 GiB of neighbours).  n_mem: points registered per hypothesis, over every job of the
// wave (sizes the memory); n_rows: points of the largest one job (its scratch rows are 32-bit).
static size_t reloc_wave_size(size_t n_hyp, size_t n_mem, size_t n_rows, int K) {
    const size_t per_hyp = std::max<size_t>(n_mem, 1) * K * sizeof(unsigned int);
    // LOCREG_RELOC_WAVE_GIB: neighbour scratch per wave in GiB.  Default 4 (7857 hypotheses of a 27 k-point scan, ~20 GB
    // of scratch in all; measured on 8192 hypotheses: 1.82 s at 1 GiB, 1.75 s at 2, 1.69 s at 4 - larger waves fill the
    // bins of the spatially ordered stage-2 queue better), never more than a third of the free device memory
    static const double wave_gib = getenv("LOCREG_RELOC_WAVE_GIB") ? std::min(16.0, std::max(1e-5, atof(getenv("LOCREG_RELOC_WAVE_GIB")))) : 4.0;
    size_t free_b = 0, total_b = 0;
    LR_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t per_hyp_all = std::max<size_t>(n_mem, 1) * (K * sizeof(unsigned int) + 80);  // + planes, margins, queues, flags
    size_t wave = std::max<size_t>(1, std::min<size_t>(n_hyp, static_cast<size_t>(wave_gib * static_cast<double>(size_t(1) << 30)) / per_hyp));
    wave = std::max<size_t>(1, std::min<size_t>(wave, free_b / 3 / per_hyp_all));
    wave = std::min<size_t>(wave, (size_t(1) << 32) / std::max<size_t>(n_rows, 1) - 1);  // scratch rows are 32-bit
    return wave;
}

// W hypotheses of ONE cloud of n points as one job: BatchView.offsets == nullptr, every item registers the whole cloud
// and owns tiles [i * tiles_per_item, ...).  An empty cloud launches nothing (its items sum zero tiles).
static IcpJob hypothesis_job(const float4* src4, size_t n, unsigned int W, AlignState* states) {
    IcpJob job;
    job.bv.src = src4; job.bv.offsets = nullptr; job.bv.tile_begin = nullptr; job.bv.tiles = nullptr;
    job.bv.n_single = static_cast<unsigned int>(n);
    job.bv.tiles_per_item = std::max<unsigned int>(1u, (static_cast<unsigned int>(n) + kTile - 1) / kTile);
    job.bv.S = W;
    job.states = states;
    job.n_tiles = static_cast<unsigned int>(n ? static_cast<size_t>(job.bv.tiles_per_item) * W : 0);
    job.n_scratch_points = static_cast<size_t>(n) * W;
    return job;
}

// n_local hypotheses (host, 7 doubles each) of ONE scan -> h->d_poses_out / d_results / d_scores and the packed best key
// in device memory (returned pointer); the index in the key is index_base + i * index_stride.  Everything is queued on
// the handle's stream; nothing is synchronised.  poses_in == nullptr: h->d_poses_in already holds the poses (a round of
// locreg_relocalise_staged).  begin_timing: the handle's timing starts here, after the poses' upload; a staged call
// starts it once before its first round instead.  The loop reads max_iteration and zero_initial_translation from h->opt.
static unsigned long long* relocalise_core(locreg_handle* h, const float4* src4, size_t n, const double* poses_in, size_t n_local,
                                           unsigned int index_base, unsigned int index_stride, bool begin_timing) {
    NvtxRange r("locreg:relocalise");
    h->d_poses_in.reserve(std::max<size_t>(n_local, 1) * 7 * sizeof(double));
    h->d_poses_out.reserve(std::max<size_t>(n_local, 1) * 7 * sizeof(double));
    h->d_results.reserve(std::max<size_t>(n_local, 1) * sizeof(DevResult));
    h->d_scores.reserve(std::max<size_t>(n_local, 1) * sizeof(double));
    h->d_misc.reserve(64);
    unsigned long long* d_key = reinterpret_cast<unsigned long long*>(h->d_misc.as<unsigned char>() + 32);
    if (n_local) {
        if (poses_in) LR_CUDA(cudaMemcpyAsync(h->d_poses_in.p, poses_in, n_local * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        LR_CUDA(cudaMemcpyAsync(h->d_poses_out.p, h->d_poses_in.p, n_local * 7 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (begin_timing) h->begin_timing();
    if (n_local && is_ndt(h)) {
        // one CTA per hypothesis: Gauss-Newton loop + one evaluation at the final pose (the score), all inside the CTA
        NDT_DISPATCH(h, ndt_run_batch(h, PB, src4, nullptr, h->d_poses_in.as<double>(), h->d_poses_out.as<double>(),
                                      h->d_results.as<DevResult>(), static_cast<unsigned int>(n_local), static_cast<unsigned int>(n), 1));
    } else if (n_local) {
        const int K = h->opt.method == LOCREG_ICP_P2P ? 1 : 5;
        const size_t wave = reloc_wave_size(n_local, n, n, K);
        h->d_states.reserve(wave * sizeof(AlignState));
        for (size_t w0 = 0; w0 < n_local; w0 += wave) {
            const unsigned int W = static_cast<unsigned int>(std::min(wave, n_local - w0));
            const IcpJob job = hypothesis_job(src4, n, W, h->d_states.as<AlignState>());
            LR_LAUNCH(k_states_init, (W + 255) / 256, 256, 0, h->stream, h->d_poses_in.as<double>() + w0 * 7, W, h->opt.max_iteration, h->opt.zero_initial_translation, job.states);
            ICP_DISPATCH(h, icp_run_loop<M>(h, job, 1));
            LR_LAUNCH(k_states_export, (W + 255) / 256, 256, 0, h->stream, job.states, W, h->d_poses_out.as<double>() + w0 * 7,
                      h->d_results.as<DevResult>() + w0);
        }
    }
    LR_CUDA(cudaMemsetAsync(d_key, 0xFF, sizeof(unsigned long long), h->stream));
    if (n_local)
        LR_LAUNCH(k_score_argmin, static_cast<unsigned int>((n_local + 255) / 256), 256, 0, h->stream, h->d_results.as<DevResult>(),
                  static_cast<unsigned int>(n_local), index_base, index_stride, h->d_scores.as<double>(), d_key);
    return d_key;
}

int locreg_relocalise(locreg_handle* h, const float* src, size_t n, size_t stride, const double* poses_in, size_t n_hyp,
                      double* best_pose, int64_t* best_idx, double* best_score, double* scores, double* poses_out) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!poses_in || n_hyp == 0 || n_hyp >= (1ull << 31)) { g_last_error = "invalid hypotheses"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        const float4* src4 = stage_cloud(h, src, n, stride, false);
        unsigned long long* d_key = relocalise_core(h, src4, n, poses_in, n_hyp, 0u, 1u, true);
        h->end_timing();
        unsigned long long key = 0;
        LR_CUDA(cudaMemcpy(&key, d_key, sizeof(key), cudaMemcpyDeviceToHost));
        const uint32_t bi = static_cast<uint32_t>(key & 0xFFFFFFFFull);
        if (best_idx) *best_idx = bi;
        if (best_score) LR_CUDA(cudaMemcpy(best_score, h->d_scores.as<double>() + bi, sizeof(double), cudaMemcpyDeviceToHost));
        if (best_pose) LR_CUDA(cudaMemcpy(best_pose, h->d_poses_out.as<double>() + static_cast<size_t>(bi) * 7, 7 * sizeof(double), cudaMemcpyDeviceToHost));
        if (scores) LR_CUDA(cudaMemcpy(scores, h->d_scores.p, n_hyp * sizeof(double), cudaMemcpyDeviceToHost));
        if (poses_out) LR_CUDA(cudaMemcpy(poses_out, h->d_poses_out.p, n_hyp * 7 * sizeof(double), cudaMemcpyDeviceToHost));
        return LOCREG_OK;
    });
}

}  // extern "C"

// The handle's loop options as they were, restored when the scope ends (also on an exception): the rounds of a staged
// relocalisation set their own trip count and zero_initial_translation, and every later call must see the caller's.
struct ScopedLoopOptions {
    locreg_handle* h;
    int32_t max_iteration, zero_initial_translation;
    explicit ScopedLoopOptions(locreg_handle* hh)
        : h(hh), max_iteration(hh->opt.max_iteration), zero_initial_translation(hh->opt.zero_initial_translation) {}
    ~ScopedLoopOptions() {
        h->opt.max_iteration = max_iteration;
        h->opt.zero_initial_translation = zero_initial_translation;
    }
    ScopedLoopOptions(const ScopedLoopOptions&) = delete;
    ScopedLoopOptions& operator=(const ScopedLoopOptions&) = delete;
};

// The schedule checks of every staged relocalisation (ICP and LOAM), before any device work.
static int schedule_check(const int32_t* trips, const int64_t* keep, int32_t n_rounds) {
    if (n_rounds < 1 || n_rounds > 32) { g_last_error = "n_rounds must be in [1, 32]"; return LOCREG_E_ARG; }
    if (!trips) { g_last_error = "invalid trips (null)"; return LOCREG_E_ARG; }
    for (int32_t r = 0; r < n_rounds; ++r)
        if (trips[r] < 0) { g_last_error = "invalid trips (negative)"; return LOCREG_E_ARG; }
    if (n_rounds > 1 && !keep) { g_last_error = "invalid keep (null with more than one round)"; return LOCREG_E_ARG; }
    for (int32_t r = 0; r + 1 < n_rounds; ++r)
        if (keep[r] < 1) { g_last_error = "invalid keep (< 1)"; return LOCREG_E_ARG; }
    return LOCREG_OK;
}

// Argument checks of locreg_relocalise_staged[_sharded], before any device work.
static int staged_check(const float* src, size_t n, size_t stride, const double* poses_in, size_t n_hyp, const int32_t* trips,
                        const int64_t* keep, int32_t n_rounds) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!poses_in || n_hyp == 0 || n_hyp >= (1ull << 31)) { g_last_error = "invalid hypotheses"; return LOCREG_E_ARG; }
    return schedule_check(trips, keep, n_rounds);
}

// The positions rank `rank` of `world` runs in a round of m alive hypotheses: rank, rank + world, ...
static unsigned int dealt(unsigned int m, unsigned int rank, unsigned int world) {
    return m > rank ? (m - rank + world - 1) / world : 0u;
}

// Staged relocalisation (include/locreg.h) over `world` ranks of comm (world 1: comm unused), on h's stream, with the
// caller's cloud(s) already staged: run(r, m_q) queues round r on the m_q hypotheses whose poses are in h->d_poses_in
// and leaves their poses and scores in h->d_poses_out / d_scores (relocalise_core for ICP / NDT, loam_relocalise_core
// for LOAM).  Between rounds the survivors are cut on the device (reloc_select.cuh) and their poses gathered into the
// next round's full pose array, so all rounds are queued back to back and the call synchronises once.  Round r's
// positions map to original indices through d_stage_idx half (r & 1) (round 0: the identity, no map).  The winner is the
// same select with k = 1 over the last round, so the cuts and the winner rank by one key, locreg_pack_score's.
// world 1: the full pose array is d_poses_in itself and run() gets all m alive hypotheses.  world > 1: it is
// d_stage_full; rank q deals itself positions q, q + world, ... into d_poses_in and runs those, and the round's results
// come back to every rank through one ncclAllGather (k_reloc_pack / k_reloc_unpack) into d_poses_out / d_scores at all m
// positions, as one GPU leaves them.  The cut and the winner then run redundantly on every rank over identical keys.
template <class Round>
static int relocalise_staged_rounds(locreg_handle* h, const double* poses_in, size_t n_hyp, const int32_t* trips,
                                    const int64_t* keep, int32_t n_rounds, double* best_pose, int64_t* best_idx,
                                    double* best_score, double* scores, double* poses_out, int32_t* rounds_out,
                                    unsigned int rank, unsigned int world, ncclComm_t comm, Round&& run) {
    NvtxRange nr("locreg:relocalise_staged");
    std::vector<size_t> alive(n_rounds);  // hypotheses in round r, known before anything runs
    alive[0] = n_hyp;
    for (int32_t r = 1; r < n_rounds; ++r) alive[r] = std::min<size_t>(static_cast<size_t>(keep[r - 1]), alive[r - 1]);
    // every per-hypothesis buffer at its full size before the first launch (the round's own reserves are then no-ops)
    h->d_poses_in.reserve(n_hyp * 7 * sizeof(double));
    h->d_poses_out.reserve(n_hyp * 7 * sizeof(double));
    h->d_results.reserve(n_hyp * sizeof(DevResult));
    h->d_scores.reserve(n_hyp * sizeof(double));
    h->d_misc.reserve(64);
    h->d_stage_keys.reserve(n_hyp * sizeof(unsigned long long));
    h->d_stage_slot.reserve(n_hyp * sizeof(unsigned int));
    h->d_stage_idx.reserve(2 * n_hyp * sizeof(unsigned int));
    h->d_stage_poses.reserve(n_hyp * 7 * sizeof(double));
    h->d_stage_scores.reserve(n_hyp * sizeof(double));
    h->d_stage_rounds.reserve(n_hyp * sizeof(int32_t));
    if (world > 1) {
        h->d_stage_full.reserve(n_hyp * 7 * sizeof(double));
        h->d_stage_gather.reserve(world * ((n_hyp + world - 1) / world) * 8 * sizeof(double));
    }
    // select state | histogram | best pose + score | best index
    constexpr size_t kHistOff = 64, kBestOff = kHistOff + kSelectBins * sizeof(unsigned int), kBestIdxOff = kBestOff + 8 * sizeof(double);
    h->d_stage_sel.reserve(kBestIdxOff + sizeof(long long));
    unsigned char* sel = h->d_stage_sel.as<unsigned char>();
    SelectState* st = reinterpret_cast<SelectState*>(sel);
    unsigned int* hist = reinterpret_cast<unsigned int*>(sel + kHistOff);
    double* d_best = reinterpret_cast<double*>(sel + kBestOff);
    long long* d_best_idx = reinterpret_cast<long long*>(sel + kBestIdxOff);
    unsigned int* idx[2] = {h->d_stage_idx.as<unsigned int>(), h->d_stage_idx.as<unsigned int>() + n_hyp};
    double* full = world > 1 ? h->d_stage_full.as<double>() : h->d_poses_in.as<double>();  // the round's alive poses
    LR_CUDA(cudaMemcpyAsync(full, poses_in, n_hyp * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemsetAsync(hist, 0, kSelectBins * sizeof(unsigned int), h->stream));  // k_select_digit re-zeroes it
    h->begin_timing();
    {
        unsigned long long* keys = h->d_stage_keys.as<unsigned long long>();
        // st->prefix = the k-th smallest key of the round's m scores (in h->d_scores)
        const auto select_kth = [&](unsigned int m, unsigned int k) {
            const unsigned int g = (m + 255) / 256;
            LR_LAUNCH(k_reloc_keys, g, 256, 0, h->stream, h->d_scores.as<double>(), m, keys);
            const unsigned int gh = std::min<unsigned int>(g, 2u * static_cast<unsigned int>(h->num_sms));
            for (int d = 0; d < 8; ++d) {
                LR_LAUNCH(k_select_hist, gh, 256, 0, h->stream, keys, m, st, d, hist);
                LR_LAUNCH(k_select_digit, 1, kSelectBins, 0, h->stream, st, hist, d, k);
            }
        };
        for (int32_t r = 0; r < n_rounds; ++r) {
            const unsigned int m = static_cast<unsigned int>(alive[r]);
            const unsigned int g = (m + 255) / 256;
            const unsigned int* idx_r = r == 0 ? nullptr : idx[r & 1];
            if (world == 1) {
                run(r, m);
            } else {
                const unsigned int m_q = dealt(m, rank, world), c = (m + world - 1) / world;
                double* gather = h->d_stage_gather.as<double>();
                double* slab = gather + static_cast<size_t>(rank) * c * 8;
                const auto blocks = [](size_t words) { return static_cast<unsigned int>((words + 255) / 256); };  // a thread per double
                if (m_q) LR_LAUNCH(k_reloc_deal, blocks(static_cast<size_t>(m_q) * 7), 256, 0, h->stream, full, m_q, rank, world,
                                   h->d_poses_in.as<double>());
                run(r, m_q);
                if (m_q) LR_LAUNCH(k_reloc_pack, blocks(static_cast<size_t>(m_q) * 8), 256, 0, h->stream, h->d_poses_out.as<double>(),
                                   h->d_scores.as<double>(), m_q, slab);
                {
                    NvtxRange ar("locreg:relocalise_staged:allgather");
                    LR_NCCL(nccl_api().AllGather(slab, gather, static_cast<size_t>(c) * 8, ncclDouble, comm, h->stream));
                }
                LR_LAUNCH(k_reloc_unpack, blocks(static_cast<size_t>(m) * 8), 256, 0, h->stream, gather, m, c, world,
                          h->d_poses_out.as<double>(), h->d_scores.as<double>());
            }
            LR_LAUNCH(k_reloc_scatter, g, 256, 0, h->stream, m, idx_r, h->d_poses_out.as<double>(), h->d_scores.as<double>(), r,
                      h->d_stage_poses.as<double>(), h->d_stage_scores.as<double>(), h->d_stage_rounds.as<int>());
            if (r + 1 == n_rounds) {
                select_kth(m, 1u);
                break;
            }
            select_kth(m, static_cast<unsigned int>(alive[r + 1]));
            unsigned int* slot = h->d_stage_slot.as<unsigned int>();
            LR_LAUNCH(k_select_flags, g, 256, 0, h->stream, keys, m, st, slot);
            exclusive_scan_u32(slot, slot, m, nullptr, h->stream);
            LR_LAUNCH(k_reloc_compact, g, 256, 0, h->stream, keys, m, st, slot, h->d_poses_out.as<double>(), idx_r, full,
                      idx[(r + 1) & 1]);
        }
        LR_LAUNCH(k_reloc_best, 1, 32, 0, h->stream, st, n_rounds > 1 ? idx[(n_rounds - 1) & 1] : nullptr,
                  h->d_stage_poses.as<double>(), h->d_stage_scores.as<double>(), d_best, d_best_idx);
    }
    h->end_timing();
    double b[8];
    long long bi = 0;
    LR_CUDA(cudaMemcpy(b, d_best, sizeof(b), cudaMemcpyDeviceToHost));
    LR_CUDA(cudaMemcpy(&bi, d_best_idx, sizeof(bi), cudaMemcpyDeviceToHost));
    if (best_idx) *best_idx = bi;
    if (best_pose) std::memcpy(best_pose, b, 7 * sizeof(double));
    if (best_score) *best_score = b[7];
    if (scores) LR_CUDA(cudaMemcpy(scores, h->d_stage_scores.p, n_hyp * sizeof(double), cudaMemcpyDeviceToHost));
    if (poses_out) LR_CUDA(cudaMemcpy(poses_out, h->d_stage_poses.p, n_hyp * 7 * sizeof(double), cudaMemcpyDeviceToHost));
    if (rounds_out) LR_CUDA(cudaMemcpy(rounds_out, h->d_stage_rounds.p, n_hyp * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return LOCREG_OK;
}

// The rounds of locreg_relocalise_staged[_sharded]: relocalise_core with the round's trip count set on the handle, and
// zero_initial_translation cleared after round 0 (later rounds start from the pose as the last one left it).
static int relocalise_staged_icp(locreg_handle* h, const float* src, size_t n, size_t stride, const double* poses_in,
                                 size_t n_hyp, const int32_t* trips, const int64_t* keep, int32_t n_rounds, double* best_pose,
                                 int64_t* best_idx, double* best_score, double* scores, double* poses_out,
                                 int32_t* rounds_out, unsigned int rank, unsigned int world, ncclComm_t comm) {
    if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
    const float4* src4 = stage_cloud(h, src, n, stride, false);
    ScopedLoopOptions saved(h);
    return relocalise_staged_rounds(h, poses_in, n_hyp, trips, keep, n_rounds, best_pose, best_idx, best_score, scores,
                                    poses_out, rounds_out, rank, world, comm, [&](int32_t r, unsigned int m_q) {
                                        h->opt.max_iteration = trips[r];
                                        if (r > 0) h->opt.zero_initial_translation = 0;
                                        relocalise_core(h, src4, n, nullptr, m_q, 0u, 1u, false);
                                    });
}

extern "C" {

int locreg_relocalise_staged(locreg_handle* h, const float* src, size_t n, size_t stride, const double* poses_in, size_t n_hyp,
                             const int32_t* trips, const int64_t* keep, int32_t n_rounds, double* best_pose, int64_t* best_idx,
                             double* best_score, double* scores, double* poses_out, int32_t* rounds_out) {
    const int rc = staged_check(src, n, stride, poses_in, n_hyp, trips, keep, n_rounds);
    if (rc) return rc;
    return guarded(h, [&]() {
        return relocalise_staged_icp(h, src, n, stride, poses_in, n_hyp, trips, keep, n_rounds, best_pose, best_idx,
                                     best_score, scores, poses_out, rounds_out, 0u, 1u, nullptr);
    });
}

// locreg_relocalise_staged over the handle's communicator (include/locreg.h); a one-rank communicator or none is the
// single-GPU call itself.
int locreg_relocalise_staged_sharded(locreg_handle* h, const float* src, size_t n, size_t stride, const double* poses_in,
                                     size_t n_hyp, const int32_t* trips, const int64_t* keep, int32_t n_rounds,
                                     double* best_pose, int64_t* best_idx, double* best_score, double* scores,
                                     double* poses_out, int32_t* rounds_out) {
    const int rc = staged_check(src, n, stride, poses_in, n_hyp, trips, keep, n_rounds);
    if (rc) return rc;
    return guarded(h, [&]() {
        const bool shard = h->comm && h->comm_world > 1;
        return relocalise_staged_icp(h, src, n, stride, poses_in, n_hyp, trips, keep, n_rounds, best_pose, best_idx,
                                     best_score, scores, poses_out, rounds_out,
                                     shard ? static_cast<unsigned int>(h->comm_rank) : 0u,
                                     shard ? static_cast<unsigned int>(h->comm_world) : 1u, shard ? h->comm : nullptr);
    });
}

// ---- multi-GPU: NCCL inside the library (SURVEY.md 8e) ---------------------------------------------------------------
int locreg_shard_range(size_t n, int32_t rank, int32_t world, size_t* lo, size_t* hi) {
    if (world < 1 || rank < 0 || rank >= world || !lo || !hi) { g_last_error = "invalid rank / world"; return LOCREG_E_ARG; }
    const size_t base = n / static_cast<size_t>(world), rem = n % static_cast<size_t>(world), r = static_cast<size_t>(rank);
    *lo = r * base + std::min(r, rem);
    *hi = *lo + base + (r < rem ? 1 : 0);
    return LOCREG_OK;
}

int locreg_comm_unique_id(unsigned char* id128) {
    if (!id128) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    const NcclApi& nc = nccl_api();
    if (!nc.ok()) { g_last_error = nc.why; return LOCREG_E_UNSUPPORTED; }
    static_assert(sizeof(ncclUniqueId) == LOCREG_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    const ncclResult_t r = nc.GetUniqueId(&id);
    if (r != ncclSuccess) { g_last_error = std::string("ncclGetUniqueId: ") + nc.GetErrorString(r); return LOCREG_E_CUDA; }
    std::memcpy(id128, &id, sizeof(id));
    return LOCREG_OK;
}

int locreg_comm_init(locreg_handle* h, const unsigned char* id128, int32_t rank, int32_t world) {
    if (!id128 || world < 1 || rank < 0 || rank >= world) { g_last_error = "invalid rank / world / id"; return LOCREG_E_ARG; }
    const NcclApi& nc = nccl_api();
    if (!nc.ok()) { g_last_error = nc.why; return LOCREG_E_UNSUPPORTED; }
    return guarded(h, [&]() {
        if (h->comm) { g_last_error = "the handle already has a communicator"; return LOCREG_E_STATE; }
        ncclUniqueId id;
        std::memcpy(&id, id128, sizeof(id));
        LR_NCCL(nc.CommInitRank(&h->comm, world, id, rank));
        h->comm_rank = rank;
        h->comm_world = world;
        return LOCREG_OK;
    });
}

int locreg_comm_destroy(locreg_handle* h) {
    return guarded(h, [&]() {
        if (h->comm) {
            LR_CUDA(cudaStreamSynchronize(h->stream));
            nccl_api().CommDestroy(h->comm);
            h->comm = nullptr;
        }
        h->comm_rank = 0;
        h->comm_world = 1;
        return LOCREG_OK;
    });
}

int locreg_comm_info(locreg_handle* h, int32_t* rank, int32_t* world, int32_t* nccl_version) {
    if (!h) { g_last_error = "null handle"; return LOCREG_E_ARG; }
    if (rank) *rank = h->comm_rank;
    if (world) *world = h->comm_world;
    if (nccl_version) {
        int v = 0;
        if (nccl_api().ok()) nccl_api().GetVersion(&v);
        *nccl_version = v;
    }
    return LOCREG_OK;
}

}  // extern "C"

// The sharded relocalisations' deal and exchange, on h's stream and communicator (none: a world of one).  Every rank holds
// all n_hyp hypotheses and registers its share of the strided deal, hypotheses rank, rank + world, ...:
// run(mine, n_local, rank, world) queues that (mine: host) and returns the device key of its best, with the poses and
// scores in h->d_poses_out / d_scores.  Then one MIN all-reduce over the packed (score, global index) keys and the
// winner's owner broadcasts pose + score; best_* come back identical on every rank.  The caller's clouds are staged
// before: the deal reuses h->h_in once h's stream has drained.
template <class Run>
static void relocalise_exchange(locreg_handle* h, const double* poses_in, size_t n_hyp, double* best_pose, int64_t* best_idx,
                                double* best_score, Run&& run) {
    const unsigned int rank = static_cast<unsigned int>(h->comm_rank), world = static_cast<unsigned int>(h->comm_world);
    const size_t n_local = n_hyp > rank ? (n_hyp - rank + world - 1) / world : 0;
    LR_CUDA(cudaStreamSynchronize(h->stream));  // stage_cloud's copy out of h_in has finished: the buffer can be reused
    h->h_in.reserve(std::max<size_t>(n_local, 1) * 7 * sizeof(double));
    double* mine = h->h_in.as<double>();
    for (size_t i = 0; i < n_local; ++i) std::memcpy(mine + i * 7, poses_in + (rank + i * world) * 7, 7 * sizeof(double));
    unsigned long long* d_key = run(static_cast<const double*>(mine), n_local, rank, world);
    // the one exchange step, on the same stream: MIN over the packed (score, global index) keys, then the winner's
    // owner broadcasts pose + score
    h->d_bcast.reserve(16 * sizeof(double));
    double* d_b = h->d_bcast.as<double>();
    unsigned long long* d_gkey = reinterpret_cast<unsigned long long*>(d_b + 8);
    const NcclApi& nc = nccl_api();
    {
        NvtxRange r("locreg:relocalise:allreduce_min");
        if (h->comm) LR_NCCL(nc.AllReduce(d_key, d_gkey, 1, ncclUint64, ncclMin, h->comm, h->stream));
        else LR_CUDA(cudaMemcpyAsync(d_gkey, d_key, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, h->stream));
    }
    h->h_small.reserve(4096);
    unsigned long long* h_key = reinterpret_cast<unsigned long long*>(h->h_small.as<unsigned char>() + 2048);
    LR_CUDA(cudaMemcpyAsync(h_key, d_gkey, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    LR_CUDA(cudaStreamSynchronize(h->stream));  // the owner of the winner is a host decision (the root of the broadcast)
    const uint32_t gi = static_cast<uint32_t>(*h_key & 0xFFFFFFFFull);
    const bool none = gi == 0xFFFFFFFFu;  // no rank had a hypothesis
    const unsigned int owner = none ? 0u : gi % world;
    if (owner == rank && !none) {
        const size_t li = (gi - rank) / world;
        LR_CUDA(cudaMemcpyAsync(d_b, h->d_poses_out.as<double>() + li * 7, 7 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        LR_CUDA(cudaMemcpyAsync(d_b + 7, h->d_scores.as<double>() + li, sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (h->comm) {
        NvtxRange r("locreg:relocalise:broadcast_pose");
        LR_NCCL(nc.Broadcast(d_b, d_b, 8, ncclDouble, static_cast<int>(owner), h->comm, h->stream));
    }
    double* h_b = h->h_small.as<double>() + 128;
    LR_CUDA(cudaMemcpyAsync(h_b, d_b, 8 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    h->end_timing();  // synchronises the stream: kernels + both collectives
    if (best_idx) *best_idx = none ? -1 : static_cast<int64_t>(gi);
    if (best_pose && !none) std::memcpy(best_pose, h_b, 7 * sizeof(double));
    if (best_score) *best_score = none ? INFINITY : h_b[7];
}

extern "C" {

int locreg_relocalise_sharded(locreg_handle* h, const float* src, size_t n, size_t stride, const double* poses_in, size_t n_hyp,
                              double* best_pose, int64_t* best_idx, double* best_score) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!poses_in || n_hyp == 0 || n_hyp >= (1ull << 31)) { g_last_error = "invalid hypotheses"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (!h->has_target) { g_last_error = "SetInputTarget has not been called"; return LOCREG_E_STATE; }
        const float4* src4 = stage_cloud(h, src, n, stride, false);
        relocalise_exchange(h, poses_in, n_hyp, best_pose, best_idx, best_score,
                            [&](const double* mine, size_t n_local, unsigned int rank, unsigned int world) {
                                return relocalise_core(h, src4, n, mine, n_local, rank, world, true);
                            });
        return LOCREG_OK;
    });
}

// The wave size of a LOAM relocalisation of n_local hypotheses, with the scratch both halves share reserved for it: the
// states (one per hypothesis, both jobs point at them) and the halves' records, which k_loam_solve writes.  One wave
// size serves both halves: its memory is sized by n_s + n_e points per hypothesis, its 32-bit scratch rows by the
// larger half.
static size_t loam_reloc_reserve(locreg_handle* surf, size_t n_local, size_t n_s, size_t n_e) {
    const size_t wave = reloc_wave_size(n_local, n_s + n_e, std::max(n_s, n_e), 5);
    surf->d_states.reserve(wave * sizeof(AlignState));
    surf->d_loam.reserve(2 * wave * sizeof(DevResult));
    return wave;
}

// LOAM relocalisation: n_local hypotheses (host, 7 doubles each) of ONE surf / edge scan.  Each runs the LOAM loop of
// locreg_align_loam from its pose; then the score pass evaluates both halves once more at the final pose and an
// evaluation-only k_loam_solve leaves the summed counts in the loop's result, from which k_score_argmin takes
// (sum_sq_surf + sum_sq_edge) / (n_inlier_surf + n_inlier_edge), +inf for a singular summed H or no inlier.  Poses,
// results and scores land in surf's d_poses_out / d_results / d_scores; returns the device key of the best (index
// index_base + i * index_stride).  Queued on surf's stream, which joins edge's; nothing is synchronised.
// poses_in == nullptr: surf->d_poses_in already holds the poses (a round of locreg_relocalise_loam_staged).
// begin_timing: surf's timing starts here, after the poses' upload; a staged call starts it once before its first round.
static unsigned long long* loam_relocalise_core(locreg_handle* surf, locreg_handle* edge, const float4* src_s, size_t n_s,
                                                const float4* src_e, size_t n_e, const double* poses_in, size_t n_local,
                                                int32_t max_iteration, double eps, unsigned int index_base, unsigned int index_stride,
                                                bool begin_timing) {
    NvtxRange r("locreg:relocalise_loam");
    const size_t cap = std::max<size_t>(n_local, 1);
    surf->d_poses_in.reserve(cap * 7 * sizeof(double));
    surf->d_poses_out.reserve(cap * 7 * sizeof(double));
    surf->d_results.reserve(cap * sizeof(DevResult));
    surf->d_scores.reserve(cap * sizeof(double));
    surf->d_misc.reserve(64);
    unsigned long long* d_key = reinterpret_cast<unsigned long long*>(surf->d_misc.as<unsigned char>() + 32);
    if (n_local && poses_in)
        LR_CUDA(cudaMemcpyAsync(surf->d_poses_in.p, poses_in, n_local * 7 * sizeof(double), cudaMemcpyHostToDevice, surf->stream));
    if (begin_timing) surf->begin_timing();
    if (n_local) {
        const size_t wave = loam_reloc_reserve(surf, n_local, n_s, n_e);
        for (size_t w0 = 0; w0 < n_local; w0 += wave) {
            const unsigned int W = static_cast<unsigned int>(std::min(wave, n_local - w0));
            const IcpJob js = hypothesis_job(src_s, n_s, W, surf->d_states.as<AlignState>());
            const IcpJob je = hypothesis_job(src_e, n_e, W, js.states);  // one state, one pose per hypothesis
            // the pose as given: the LOAM loop ignores zero_initial_translation
            LR_LAUNCH(k_states_init, (W + 255) / 256, 256, 0, surf->stream, surf->d_poses_in.as<double>() + w0 * 7, W, max_iteration, 0, js.states);
            loam_run_loop(surf, edge, js, je, max_iteration, eps, surf->d_loam.as<DevResult>(), 1);
            LR_LAUNCH(k_states_export, (W + 255) / 256, 256, 0, surf->stream, js.states, W, surf->d_poses_out.as<double>() + w0 * 7,
                      surf->d_results.as<DevResult>() + w0);
        }
    } else {  // no hypothesis on this rank: edge's cloud copy still joins surf's stream
        LR_CUDA(cudaEventRecord(surf->loam_ev[1], edge->stream));
        LR_CUDA(cudaStreamWaitEvent(surf->stream, surf->loam_ev[1], 0));
    }
    LR_CUDA(cudaMemsetAsync(d_key, 0xFF, sizeof(unsigned long long), surf->stream));
    if (n_local)
        LR_LAUNCH(k_score_argmin, static_cast<unsigned int>((n_local + 255) / 256), 256, 0, surf->stream, surf->d_results.as<DevResult>(),
                  static_cast<unsigned int>(n_local), index_base, index_stride, surf->d_scores.as<double>(), d_key);
    return d_key;
}

static int loam_relocalise_check(const locreg_handle* surf, const locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                 const float* edge_xyz, size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp) {
    int rc = loam_check_handles(surf, edge);
    if (rc) return rc;
    rc = check_cloud_args(surf_xyz, n_surf, stride);
    if (rc) return rc;
    rc = check_cloud_args(edge_xyz, n_edge, stride);
    if (rc) return rc;
    if (!poses_in || n_hyp == 0 || n_hyp >= (1ull << 31)) { g_last_error = "invalid hypotheses"; return LOCREG_E_ARG; }
    return LOCREG_OK;
}

int locreg_relocalise_loam(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf, const float* edge_xyz,
                           size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp, int32_t max_iteration, double eps,
                           double* best_pose, int64_t* best_idx, double* best_score, double* scores, double* poses_out) {
    const int rc = loam_relocalise_check(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp);
    if (rc) return rc;
    return guarded(surf, [&]() {
        const int st = loam_prepare(surf, edge);
        if (st) return st;
        const float4* src_s = stage_cloud(surf, surf_xyz, n_surf, stride, false);
        const float4* src_e = stage_cloud(edge, edge_xyz, n_edge, stride, false);
        unsigned long long* d_key = loam_relocalise_core(surf, edge, src_s, n_surf, src_e, n_edge, poses_in, n_hyp, max_iteration, eps, 0u, 1u, true);
        surf->end_timing();
        cudaStream_t const s = surf->stream;
        surf->h_small.reserve(4096);
        unsigned long long* h_key = reinterpret_cast<unsigned long long*>(surf->h_small.as<unsigned char>() + 2048);
        LR_CUDA(cudaMemcpyAsync(h_key, d_key, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        LR_CUDA(cudaStreamSynchronize(s));
        const uint32_t bi = static_cast<uint32_t>(*h_key & 0xFFFFFFFFull);
        if (best_idx) *best_idx = bi;
        if (best_score) LR_CUDA(cudaMemcpyAsync(best_score, surf->d_scores.as<double>() + bi, sizeof(double), cudaMemcpyDeviceToHost, s));
        if (best_pose) LR_CUDA(cudaMemcpyAsync(best_pose, surf->d_poses_out.as<double>() + static_cast<size_t>(bi) * 7, 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (scores) LR_CUDA(cudaMemcpyAsync(scores, surf->d_scores.p, n_hyp * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (poses_out) LR_CUDA(cudaMemcpyAsync(poses_out, surf->d_poses_out.p, n_hyp * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
        LR_CUDA(cudaStreamSynchronize(s));
        return LOCREG_OK;
    });
}

int locreg_relocalise_loam_sharded(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf, const float* edge_xyz,
                                   size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp, int32_t max_iteration, double eps,
                                   double* best_pose, int64_t* best_idx, double* best_score) {
    const int rc = loam_relocalise_check(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp);
    if (rc) return rc;
    return guarded(surf, [&]() {
        const int st = loam_prepare(surf, edge);
        if (st) return st;
        const float4* src_s = stage_cloud(surf, surf_xyz, n_surf, stride, false);
        const float4* src_e = stage_cloud(edge, edge_xyz, n_edge, stride, false);
        // surf's communicator (and stream) carry the exchange; edge's communicator is not used
        relocalise_exchange(surf, poses_in, n_hyp, best_pose, best_idx, best_score,
                            [&](const double* mine, size_t n_local, unsigned int rank, unsigned int world) {
                                return loam_relocalise_core(surf, edge, src_s, n_surf, src_e, n_edge, mine, n_local, max_iteration, eps,
                                                            rank, world, true);
                            });
        return LOCREG_OK;
    });
}

// Argument checks of locreg_relocalise_loam_staged[_sharded]: locreg_relocalise_loam's, then the schedule's.
static int loam_staged_check(const locreg_handle* surf, const locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                             const float* edge_xyz, size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp,
                             const int32_t* trips, const int64_t* keep, int32_t n_rounds) {
    const int rc = loam_relocalise_check(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp);
    if (rc) return rc;
    return schedule_check(trips, keep, n_rounds);
}

// The rounds of locreg_relocalise_loam_staged[_sharded]: loam_relocalise_core with trips[r] trips and the caller's eps,
// on surf's stream and surf's staged buffers.  The handles' options are not touched.
static int relocalise_loam_staged(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                  const float* edge_xyz, size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp,
                                  const int32_t* trips, const int64_t* keep, int32_t n_rounds, double eps, double* best_pose,
                                  int64_t* best_idx, double* best_score, double* scores, double* poses_out,
                                  int32_t* rounds_out, unsigned int rank, unsigned int world, ncclComm_t comm) {
    const int st = loam_prepare(surf, edge);
    if (st) return st;
    const float4* src_s = stage_cloud(surf, surf_xyz, n_surf, stride, false);
    const float4* src_e = stage_cloud(edge, edge_xyz, n_edge, stride, false);
    // round 0 has the most hypotheses: the scratch the halves share is sized for its wave before the first launch, so
    // that round 0's own reserve does not grow (free and reallocate) a buffer once the rounds are being queued
    if (const unsigned int m_q0 = dealt(static_cast<unsigned int>(n_hyp), rank, world)) loam_reloc_reserve(surf, m_q0, n_surf, n_edge);
    return relocalise_staged_rounds(surf, poses_in, n_hyp, trips, keep, n_rounds, best_pose, best_idx, best_score, scores,
                                    poses_out, rounds_out, rank, world, comm, [&](int32_t r, unsigned int m_q) {
                                        loam_relocalise_core(surf, edge, src_s, n_surf, src_e, n_edge, nullptr, m_q, trips[r],
                                                             eps, 0u, 1u, false);
                                    });
}

int locreg_relocalise_loam_staged(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                  const float* edge_xyz, size_t n_edge, size_t stride, const double* poses_in, size_t n_hyp,
                                  const int32_t* trips, const int64_t* keep, int32_t n_rounds, double eps, double* best_pose,
                                  int64_t* best_idx, double* best_score, double* scores, double* poses_out,
                                  int32_t* rounds_out) {
    const int rc = loam_staged_check(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp, trips, keep, n_rounds);
    if (rc) return rc;
    return guarded(surf, [&]() {
        return relocalise_loam_staged(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp, trips, keep,
                                      n_rounds, eps, best_pose, best_idx, best_score, scores, poses_out, rounds_out, 0u, 1u,
                                      nullptr);
    });
}

// locreg_relocalise_loam_staged over the surf handle's communicator (include/locreg.h); a one-rank communicator or none
// is the single-GPU call itself.  The edge handle's communicator is not used.
int locreg_relocalise_loam_staged_sharded(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                          const float* edge_xyz, size_t n_edge, size_t stride, const double* poses_in,
                                          size_t n_hyp, const int32_t* trips, const int64_t* keep, int32_t n_rounds,
                                          double eps, double* best_pose, int64_t* best_idx, double* best_score,
                                          double* scores, double* poses_out, int32_t* rounds_out) {
    const int rc = loam_staged_check(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp, trips, keep, n_rounds);
    if (rc) return rc;
    return guarded(surf, [&]() {
        const bool shard = surf->comm && surf->comm_world > 1;
        return relocalise_loam_staged(surf, edge, surf_xyz, n_surf, edge_xyz, n_edge, stride, poses_in, n_hyp, trips, keep,
                                      n_rounds, eps, best_pose, best_idx, best_score, scores, poses_out, rounds_out,
                                      shard ? static_cast<unsigned int>(surf->comm_rank) : 0u,
                                      shard ? static_cast<unsigned int>(surf->comm_world) : 1u, shard ? surf->comm : nullptr);
    });
}

int locreg_transform_cloud(locreg_handle* h, const float* src, size_t n, size_t stride, const double* pose, float* out_xyz) {
    const int rc = check_cloud_args(src, n, stride);
    if (rc) return rc;
    if (!pose || !out_xyz) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (n == 0) return LOCREG_OK;
        stage_cloud(h, src, n, stride, false);
        h->d_out.reserve(n * stride);
        h->d_acc.reserve(32 * sizeof(double));
        LR_CUDA(cudaMemcpyAsync(h->d_acc.p, pose, 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        LR_CUDA(cudaStreamSynchronize(h->stream));
        h->begin_timing();
        const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((n + 255) / 256, 4096));
        LR_LAUNCH(k_transform, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>(), h->d_out.as<unsigned char>(), n, stride, h->d_acc.as<double>());
        h->end_timing();
        LR_CUDA(cudaMemcpy(out_xyz, h->d_out.p, n * stride, cudaMemcpyDeviceToHost));
        return LOCREG_OK;
    });
}

// Loc::InitGlobalMap (loc.cpp:268-283): the global map goes to the device once and stays there.
int locreg_set_global_map(locreg_handle* h, const float* xyz, size_t n, size_t stride) {
    const int rc = check_cloud_args(xyz, n, stride);
    if (rc) return rc;
    return guarded(h, [&]() {
        h->d_global.reserve(std::max<size_t>(n * stride, 1));
        if (n) LR_CUDA(cudaMemcpyAsync(h->d_global.p, xyz, n * stride, cudaMemcpyHostToDevice, h->stream));
        LR_CUDA(cudaStreamSynchronize(h->stream));
        h->n_global = n;
        h->global_stride = stride;
        return LOCREG_OK;
    });
}
// Loc::ResetLocalMap (loc.cpp:187-206): BoxFilter::SetOrigin + Filter (pcl::CropBox, box_filter.cpp:24-32,46-60) of the
// global map, then SetInputTarget of the cropped cloud - without the cloud leaving the device.
int locreg_reset_local_map(locreg_handle* h, const float* origin3, const float* half_size3, size_t* n_local) {
    if (!origin3 || !half_size3) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        if (h->global_stride == 0) { g_last_error = "locreg_set_global_map has not been called"; return LOCREG_E_STATE; }
        float lo[3], hi[3];
        for (int a = 0; a < 3; ++a) {  // edge = size + origin in float (BoxFilter::CalculateEdge)
            lo[a] = -half_size3[a] + origin3[a];
            hi[a] = half_size3[a] + origin3[a];
        }
        h->d_local.reserve(std::max<size_t>(h->n_global * h->global_stride, 1));
        size_t kept = 0;
        if (h->n_global)
            kept = filter_crop_box(h->d_global.as<unsigned char>(), h->n_global, h->global_stride, lo, hi, h->d_local.as<unsigned char>(), h->stream);
        if (n_local) *n_local = kept;
        return set_target_impl(h, h->d_local.as<float>(), kept, h->global_stride, true);
    });
}

// Lio::AddCloud's local-map bookkeeping (lio.cpp:238-307), on the device.
int locreg_local_map_add_keyframe(locreg_handle* h, const float* scan_xyz, size_t n, size_t stride, const double* pose7,
                                  int32_t max_keyframes, float leaf, size_t* n_local) {
    const int rc = check_cloud_args(scan_xyz, n, stride);
    if (rc) return rc;
    if (!pose7 || max_keyframes < 1) { g_last_error = "null pose or max_keyframes < 1"; return LOCREG_E_ARG; }
    if (h && h->lmap_stride && h->lmap_stride != stride) { g_last_error = "key frames of one local map must share a point stride"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        // key_frame_scan = transformPointCloud(scan, pose) - the Scalar = double instantiation (pose.matrix() is a Matrix4d)
        // The call is transactional: the window, the local map and its size change only after every step that can fail
        // (allocations, the voxel grid's extent check) has succeeded.
        locreg_handle::KeyFrame kf;
        kf.n = n;
        struct KfGuard {  // frees the new key frame's buffer unless the window has taken it over
            void* p = nullptr;
            ~KfGuard() { if (p) cudaFree(p); }
        } guard;
        if (n) {
            stage_cloud(h, scan_xyz, n, stride, false);
            LR_CUDA(cudaMalloc(&kf.p, n * stride));
            guard.p = kf.p;
            h->d_acc.reserve(32 * sizeof(double));
            LR_CUDA(cudaMemcpyAsync(h->d_acc.p, pose7, 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            const unsigned int grid = static_cast<unsigned int>(std::min<size_t>((n + 255) / 256, 4096));
            LR_LAUNCH(k_transform_d, grid, 256, 0, h->stream, h->d_raw.as<unsigned char>(), static_cast<unsigned char*>(kf.p), n, stride,
                      h->d_acc.as<double>());
        }
        // the unfiltered local map: all scans of the window after a pop (:283-292), else the old map + the key frame (:296)
        const bool pop = h->keyframes.size() + 1 > static_cast<size_t>(max_keyframes);
        size_t total = 0;
        if (pop) {
            bool first = true;
            for (const auto& k : h->keyframes) { if (!first) total += k.n; first = false; }
            total += n;
            h->d_lmap_tmp.reserve(std::max<size_t>(total * stride, 1));
            size_t at = 0;
            first = true;
            for (const auto& k : h->keyframes) {
                if (!first && k.n) LR_CUDA(cudaMemcpyAsync(h->d_lmap_tmp.as<unsigned char>() + at * stride, k.p, k.n * stride, cudaMemcpyDeviceToDevice, h->stream));
                if (!first) at += k.n;
                first = false;
            }
            if (n) LR_CUDA(cudaMemcpyAsync(h->d_lmap_tmp.as<unsigned char>() + at * stride, kf.p, n * stride, cudaMemcpyDeviceToDevice, h->stream));
        } else {
            total = h->n_lmap + n;
            h->d_lmap_tmp.reserve(std::max<size_t>(total * stride, 1));
            if (h->n_lmap) LR_CUDA(cudaMemcpyAsync(h->d_lmap_tmp.p, h->d_lmap.p, h->n_lmap * stride, cudaMemcpyDeviceToDevice, h->stream));
            if (n) LR_CUDA(cudaMemcpyAsync(h->d_lmap_tmp.as<unsigned char>() + h->n_lmap * stride, kf.p, n * stride, cudaMemcpyDeviceToDevice, h->stream));
        }
        // local_map_filter_ptr_->Filter(local_map_, local_map_): into a second buffer that replaces d_lmap only on success
        h->d_lmap_new.reserve(std::max<size_t>(total * stride, 1));
        size_t n_new = total;
        if (leaf > 0.0f && total) {
            n_new = filter_voxel_grid(h->d_lmap_tmp.as<unsigned char>(), total, stride, leaf, h->d_lmap_new.as<unsigned char>(), h->stream);
        } else if (total) {
            LR_CUDA(cudaMemcpyAsync(h->d_lmap_new.p, h->d_lmap_tmp.p, total * stride, cudaMemcpyDeviceToDevice, h->stream));
        }
        // ---- commit
        if (pop) {
            LR_CUDA(cudaStreamSynchronize(h->stream));
            if (h->keyframes.front().p) cudaFree(h->keyframes.front().p);
            h->keyframes.pop_front();
        }
        h->keyframes.push_back(kf);
        guard.p = nullptr;
        h->lmap_stride = stride;
        std::swap(h->d_lmap.p, h->d_lmap_new.p);
        std::swap(h->d_lmap.cap, h->d_lmap_new.cap);
        h->n_lmap = n_new;
        if (n_local) *n_local = h->n_lmap;
        if (h->opt.method == LOCREG_NDT_INCREMENTAL) return set_target_impl(h, static_cast<const float*>(kf.p), kf.n, stride, true);
        return set_target_impl(h, h->d_lmap.as<float>(), h->n_lmap, stride, true);
    });
}
int locreg_local_map_get(locreg_handle* h, float* out_xyz, size_t capacity_points, size_t* n_local, size_t* stride_bytes) {
    if (!n_local) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        *n_local = h->n_lmap;
        if (stride_bytes) *stride_bytes = h->lmap_stride;
        if (out_xyz && h->n_lmap) {
            if (capacity_points < h->n_lmap) { g_last_error = "output buffer too small for the local map"; return LOCREG_E_ARG; }
            LR_CUDA(cudaStreamSynchronize(h->stream));
            LR_CUDA(cudaMemcpy(out_xyz, h->d_lmap.p, h->n_lmap * h->lmap_stride, cudaMemcpyDeviceToHost));
        }
        return LOCREG_OK;
    });
}
int locreg_local_map_clear(locreg_handle* h) {
    return guarded(h, [&]() {
        LR_CUDA(cudaStreamSynchronize(h->stream));
        h->clear_keyframes();
        return LOCREG_OK;
    });
}

// kind: 0 remove NaN, 1 crop box (a = min3, b = max3), 2 voxel grid (a[0] = leaf)
static int filter_impl(locreg_handle* h, int kind, const float* xyz, size_t n, size_t stride, const float* a, const float* b,
                       float* out_xyz, size_t* n_out) {
    const int rc = check_cloud_args(xyz, n, stride);
    if (rc) return rc;
    if (!n_out || (n && !out_xyz)) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    if (kind == 2 && !(a[0] > 0)) { g_last_error = "leaf size must be > 0"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        *n_out = 0;
        if (n == 0) return LOCREG_OK;
        stage_cloud(h, xyz, n, stride, false);  // raw copy in d_raw (the float4 view is not needed)
        h->d_out.reserve(n * stride);
        h->begin_timing();
        size_t kept = 0;
        const unsigned char* in = h->d_raw.as<unsigned char>();
        unsigned char* out = h->d_out.as<unsigned char>();
        if (kind == 0) kept = filter_remove_nan(in, n, stride, out, h->stream);
        else if (kind == 1) kept = filter_crop_box(in, n, stride, a, b, out, h->stream);
        else kept = filter_voxel_grid(in, n, stride, a[0], out, h->stream);
        h->end_timing();
        if (kept) LR_CUDA(cudaMemcpy(out_xyz, out, kept * stride, cudaMemcpyDeviceToHost));
        *n_out = kept;
        return LOCREG_OK;
    });
}
int locreg_filter_remove_nan(locreg_handle* h, const float* xyz, size_t n, size_t stride, float* out_xyz, size_t* n_out) {
    return filter_impl(h, 0, xyz, n, stride, nullptr, nullptr, out_xyz, n_out);
}
int locreg_filter_crop_box(locreg_handle* h, const float* xyz, size_t n, size_t stride, const float* min3, const float* max3,
                           float* out_xyz, size_t* n_out) {
    if (!min3 || !max3) { g_last_error = "null argument"; return LOCREG_E_ARG; }
    return filter_impl(h, 1, xyz, n, stride, min3, max3, out_xyz, n_out);
}
int locreg_filter_voxel_grid(locreg_handle* h, const float* xyz, size_t n, size_t stride, float leaf_size, float* out_xyz, size_t* n_out) {
    return filter_impl(h, 2, xyz, n, stride, &leaf_size, nullptr, out_xyz, n_out);
}

int locreg_ndt_num_voxels(locreg_handle* h, size_t* nv) {
    if (!h || !nv) return LOCREG_E_ARG;
    *nv = h->opt.method == LOCREG_NDT_INCREMENTAL ? h->inc_ndt_map.size(h->stream) : h->ndt_map.view().n_voxels;
    return LOCREG_OK;
}
int locreg_ndt_get_voxels(locreg_handle* h, int32_t* keys, double* mu, double* info, int32_t* npts) {
    return guarded(h, [&]() {
        std::vector<int> k, c;
        std::vector<double> m, f;
        if (h->opt.method == LOCREG_NDT_INCREMENTAL) h->inc_ndt_map.download(k, m, f, c, h->stream);
        else h->ndt_map.download(k, m, f, c, h->stream);
        if (keys) std::memcpy(keys, k.data(), k.size() * sizeof(int));
        if (mu) std::memcpy(mu, m.data(), m.size() * sizeof(double));
        if (info) std::memcpy(info, f.data(), f.size() * sizeof(double));
        if (npts) std::memcpy(npts, c.data(), c.size() * sizeof(int));
        return LOCREG_OK;
    });
}

int locreg_profile(locreg_handle* h, int32_t enable, double* ms4, int64_t* launches4) {
    return guarded(h, [&]() {
        prof_collect(h);
        if (ms4) for (int i = 0; i < 4; ++i) ms4[i] = h->prof_ms[i];
        if (launches4) for (int i = 0; i < 4; ++i) launches4[i] = h->prof_launches[i];
        for (int i = 0; i < 4; ++i) { h->prof_ms[i] = 0; h->prof_launches[i] = 0; }
        h->profile = enable != 0;
        return LOCREG_OK;
    });
}

int locreg_index_info(locreg_handle* h, size_t* bytes, size_t* points, size_t* lists_or_voxels) {
    if (!h) { g_last_error = "null handle"; return LOCREG_E_ARG; }
    return guarded(h, [&]() {
        size_t b = 0, p = 0, l = 0;
        if (h->opt.method == LOCREG_NDT_DIRECT) {
            b = h->ndt_map.bytes(); l = h->ndt_map.view().n_voxels;
        } else if (h->opt.method == LOCREG_NDT_INCREMENTAL) {
            l = h->inc_ndt_map.size(h->stream);
        } else {
            b = h->icp_map.bytes() + h->icp_mid.bytes();
            for (int i = 0; i < kCoarseLevels; ++i) b += h->icp_coarse[i].bytes();
            p = h->icp_map.view().n_pts;
            l = h->icp_map.n_lists();
        }
        if (bytes) *bytes = b;
        if (points) *points = p;
        if (lists_or_voxels) *lists_or_voxels = l;
        return LOCREG_OK;
    });
}
int locreg_last_timing(locreg_handle* h, double* kernel_ms, int64_t* launches) {
    if (!h) return LOCREG_E_ARG;
    if (kernel_ms) *kernel_ms = h->last_ms;
    if (launches) *launches = h->last_launches;
    return LOCREG_OK;
}

}  // extern "C"
