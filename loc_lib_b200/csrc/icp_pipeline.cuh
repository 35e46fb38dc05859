// ICP as a three-kernel pipeline per Gauss-Newton iteration (kernels K2/K3/K4 of SURVEY.md §2.3), for one
// scan, a batch of scans (BASELINE config 4) or many pose hypotheses of one scan (config 5):
//
//   k_icp_nn     one thread per source point: transform with the scan's current pose, exact k-NN in the
//                voxel-hash map, write the k neighbour positions (4 B each).  Light on registers (<= 64) so that
//                2048 threads per SM hide the L2 latency of the hash / cell / point loads.
//   k_icp_post   one thread per source point: gather the neighbours, plane fit, gates, Jacobian row, and a
//                fixed-order block reduction of the 28+2 Gauss-Newton sums -> one 256 B partial row per tile.
//   k_icp_solve  one warp per scan: sums the scan's partial rows in tile order, solves the 6x6 system, updates
//                the pose and the convergence flags kept in device memory (AlignState).
//
// Nothing returns to the host between iterations: converged / aborted scans carry a stop flag that makes
// their tiles exit at once.  A tile is 256 consecutive points of one scan; tile t of scan s is block
// tile_begin[s] + t (relocalisation: s * tiles_per_item + t).
#pragma once
#include "device_utils.cuh"
#include "icp_point.cuh"
#include "knn_warp.cuh"

namespace locreg {

// Mirrors locreg_result (include/locreg.h) field for field.
struct DevResult {
    int iters, updates, converged, degenerate;
    long long n_effective, n_inlier;
    double sum_sq_res;
    int pose_written, pad_;
};
static_assert(sizeof(DevResult) == 48, "DevResult must match locreg_result");

struct AlignState {  // one per scan / hypothesis, device resident for the whole Gauss-Newton loop
    double pose[7];
    DevResult res;
    int stop;
    int pad;
};

constexpr int kTile = 256;
constexpr unsigned int kNoNeighbour = kNoPos;

struct BatchView {
    const float4* src;              // all scans' points
    const long long* offsets;       // S+1 point offsets into src, or nullptr: every item is src[0..n_single)
    const unsigned int* tile_begin; // S+1 tile offsets, or nullptr: item s owns tiles [s*tiles_per_item, ...)
    const struct TileRec* tiles;    // with tile_begin: the per-tile table k_tile_table derived from it (one load, no search)
    unsigned int n_table_tiles;     // entries of tiles[]
    unsigned int n_single;
    unsigned int tiles_per_item;
    unsigned int S;
};

// One tile of a ragged batch, precomputed once per job: a block finds its work with one broadcast load instead of a
// binary search of dependent loads in front of every kernel of every iteration.
struct alignas(16) TileRec {
    unsigned int scan, first, count, valid;
    long long base, pad;
};

struct TileCoord {
    unsigned int scan;      // item index
    unsigned int first;     // index of the tile's first point within its scan
    unsigned int count;     // points in this tile (<= kTile)
    long long src_base;     // index of the scan's first point in src
    long long out_base;     // index of the scan's first point in per-point scratch arrays (nn, gate)
    bool valid;
};

__device__ __forceinline__ TileCoord locate_tile_thread(const BatchView& b, unsigned int tile) {
    TileCoord c{};
    c.valid = false;
    unsigned int s, t;
    if (b.tiles) {
        if (tile >= b.n_table_tiles) return c;
        const uint4 a = reinterpret_cast<const uint4*>(b.tiles + tile)[0];
        c.scan = a.x; c.first = a.y; c.count = a.z; c.valid = a.w != 0u;
        c.src_base = c.out_base = b.tiles[tile].base;
        return c;
    }
    if (b.tile_begin) {
        if (tile >= b.tile_begin[b.S]) return c;
        unsigned int lo = 0, hi = b.S - 1;  // last s with tile_begin[s] <= tile
        while (lo < hi) {
            const unsigned int mid = (lo + hi + 1) >> 1;
            if (b.tile_begin[mid] <= tile) lo = mid; else hi = mid - 1;
        }
        s = lo;
        t = tile - b.tile_begin[s];
    } else {
        s = tile / b.tiles_per_item;
        t = tile - s * b.tiles_per_item;
        if (s >= b.S) return c;
    }
    const long long beg = b.offsets ? b.offsets[s] : 0;
    const unsigned int n = b.offsets ? static_cast<unsigned int>(b.offsets[s + 1] - beg) : b.n_single;
    c.scan = s;
    c.first = t * kTile;
    if (c.first >= n) return c;
    c.count = n - c.first < kTile ? n - c.first : kTile;
    c.src_base = beg;
    c.out_base = b.offsets ? beg : static_cast<long long>(s) * b.n_single;
    c.valid = true;
    return c;
}

// Block-wide flavour: thread 0 does the (binary) search, everybody reads the answer from shared memory.
__device__ __forceinline__ TileCoord locate_tile(const BatchView& b, unsigned int tile) {
    if (b.tiles || !b.tile_begin) return locate_tile_thread(b, tile);  // a broadcast load / pure arithmetic: no hand-over needed
    __shared__ TileCoord tc_shared;
    if (threadIdx.x == 0) tc_shared = locate_tile_thread(b, tile);
    __syncthreads();
    return tc_shared;
}

// tile_begin[s] = sum_{r<s} ceil(n_r / kTile); single block, S is at most a few 1e4.
__global__ void k_tile_begin(const long long* __restrict__ offsets, unsigned int S, unsigned int* tile_begin) {
    __shared__ unsigned int carry;
    __shared__ unsigned int warp_sums[33];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (unsigned int base = 0; base < S; base += blockDim.x) {
        const unsigned int s = base + threadIdx.x;
        unsigned int v = 0;
        if (s < S) v = static_cast<unsigned int>((offsets[s + 1] - offsets[s] + kTile - 1) / kTile);
        // block exclusive scan
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        unsigned int inc = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, inc, off);
            if (lane >= off) inc += t;
        }
        if (lane == 31) warp_sums[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            unsigned int w = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0u, winc = w;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const unsigned int t = __shfl_up_sync(0xffffffffu, winc, off);
                if (lane >= off) winc += t;
            }
            warp_sums[lane] = winc - w;
            if (lane == 31) warp_sums[32] = winc;
        }
        __syncthreads();
        if (s < S) tile_begin[s] = carry + warp_sums[warp] + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += warp_sums[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_begin[S] = carry;
}

// tiles[t] for every tile of the grid (surplus tiles: valid = 0), from tile_begin.
__global__ void k_tile_table(BatchView bv, unsigned int n_tiles, TileRec* tiles) {
    const unsigned int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    bv.tiles = nullptr;
    const TileCoord c = locate_tile_thread(bv, t);
    TileRec r;
    r.scan = c.scan; r.first = c.first; r.count = c.valid ? c.count : 0u; r.valid = c.valid ? 1u : 0u;
    r.base = c.src_base; r.pad = 0;
    tiles[t] = r;
}

// ---- K_A: neighbour search ---------------------------------------------------------------------------------
#ifndef LR_NN_MIN_BLOCKS
#define LR_NN_MIN_BLOCKS 6  // 40 registers: 75 % occupancy measured best on B200 (4: +6 % time, 8: +35 %)
#endif
// Stage 1 (k_icp_nn): one thread per source point: transform, seeds + one-list fast path (knn_query_fast).  The few
// queries whose k-th neighbour may lie outside the visited box - 13 % at a 0.3 m / 2 deg initial error, 0.1 % once the
// pose has settled - are NOT finished here, where each of them would hold 31 idle lanes hostage for the length of a
// shell search: they are appended to a queue and finished by k_icp_nn_rings, one queued query per thread.
// mode bit 0 (kNnSeeds):   nn_pos still holds this job's neighbours of the previous Gauss-Newton iteration; they
//                          start each query's k-best set, so that almost no candidate passes the acceptance test.
// mode bit 1 (kNnTwoPass): threshold pre-pass of knn_scan_list (first iterations: no or poor seeds).
constexpr int kNnSeeds = 1, kNnTwoPass = 2;
struct RingQueue {
    unsigned int* count;   // entries appended so far (reset by k_icp_post); count[1] = the consumers' work cursor
    uint2* entries;        // (scratch row of the point, scan index)
};

// Block-aggregated queue append without a block barrier (see k_icp_nn).  pending/done/staged live in shared memory
// and must have been zeroed before a __syncthreads() that every thread of the block has passed.
// local_rows / local_n (optional, shared memory of the caller, *local_n zero on entry): the rows stay in the block - the
// caller serves them itself after a barrier (the single-scan kernel from its second iteration on) - and the global queue
// only counts them.
__device__ __forceinline__ void tile_queue_append(bool mine, unsigned int row, unsigned int scan, unsigned int* pending,
                                                  unsigned int* done, unsigned int* staged, const RingQueue& queue,
                                                  unsigned int* local_rows = nullptr, unsigned int* local_n = nullptr) {
    const unsigned int lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
#if defined(LR_APPEND_BARRIER)
    // Checking build (compute-sanitizer racecheck does not model the fence + arrival-counter hand-over below and reports
    // it as a hazard): the same append behind a block barrier.  profiles/ holds the racecheck logs of both builds.
    if (mine) staged[atomicAdd(pending, 1u)] = row;
    __syncthreads();
    if (threadIdx.x >= 32) return;
    (void)done; (void)n_warps;
    {
        const unsigned int n = *pending;
        if (n == 0u) return;
        if (local_rows != nullptr) {
            for (unsigned int i = lane; i < n; i += 32) local_rows[i] = staged[i];
            if (lane == 0) { *local_n = n; atomicAdd(queue.count, n); }
            return;
        }
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(queue.count, n);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (unsigned int i = lane; i < n; i += 32) queue.entries[base + i] = make_uint2(staged[i], scan);
        return;
    }
#endif
    if (mine) staged[atomicAdd(pending, 1u)] = row;
    __syncwarp();
    unsigned int last = 0;
    if (lane == 0) {
        __threadfence_block();  // this warp's staged rows before its arrival
        last = atomicAdd(done, 1u) == n_warps - 1 ? 1u : 0u;
        __threadfence_block();  // the other warps' staged rows after having seen their arrivals
    }
    if (!__shfl_sync(0xffffffffu, last, 0)) return;
    __syncwarp();  // lane 0's acquire fence orders the other lanes' reads below as well
    const unsigned int n = *reinterpret_cast<volatile unsigned int*>(pending);
    if (n == 0u) return;
    if (local_rows != nullptr) {
        for (unsigned int i = lane; i < n; i += 32) local_rows[i] = reinterpret_cast<volatile unsigned int*>(staged)[i];
        if (lane == 0) { *local_n = n; atomicAdd(queue.count, n); }
        return;
    }
    unsigned int base = 0;
    if (lane == 0) base = atomicAdd(queue.count, n);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (unsigned int i = lane; i < n; i += 32)
        queue.entries[base + i] = make_uint2(reinterpret_cast<volatile unsigned int*>(staged)[i], scan);
}

// mode bit 2 (kNnTrack):   with seeds, no pre-pass: a query that has moved less than its margin since its last full search
//                          (KnnTrack, voxel_map.cuh) only re-sorts its K neighbours.  The queries that do need the list
//                          are compacted over the tile first - by the eighth iteration they are 3 % of the points, and
//                          left in place they would still keep a lane of nearly every warp busy for a whole scan.
constexpr int kNnTrack = 4;
constexpr int kNnFirstTrack = 16;  // host-side only: nothing can take the margin shortcut yet (every point is searched)
constexpr int kNnFused = 8;  // host-side only: run the evaluation through icp_fused.cuh (tracked P2Plane iterations after the first)
#ifndef LR_NN_TRACK_MIN_BLOCKS
#define LR_NN_TRACK_MIN_BLOCKS LR_NN_MIN_BLOCKS
#endif
// The work of one block on one tile: the body of k_icp_nn, also called tile after tile by the persistent single-scan
// kernel (icp_persist.cuh), which separates the calls by block barriers.
template <int K, bool TRACKED>
__device__ __forceinline__ void icp_nn_tile(unsigned int tile, const VoxelMapView& map, const BatchView& bv,
                                            const AlignState* __restrict__ states, int ignore_stop, int mode,
                                            unsigned int* __restrict__ nn_pos, unsigned char* __restrict__ plane_valid, KnnTrack* track,
                                            const RingQueue& queue, unsigned int* local_rows = nullptr, unsigned int* local_n = nullptr) {
    __shared__ Pose T;
    const TileCoord tc = locate_tile(bv, tile);
    if (!tc.valid) return;
    const AlignState* st = states + tc.scan;
    if (st->stop && !ignore_stop) return;
    if (threadIdx.x == 0) pose_load(T, st->pose);
    // Unfinished queries are staged in shared memory; the LAST warp of the tile to finish appends them to the global
    // queue with one atomic.  No barrier after the search: a warp retires as soon as its own queries are done.
    __shared__ unsigned int blk_pending, blk_done, blk_scan;
    __shared__ unsigned int staged[kTile];
    __shared__ unsigned char scan_list[kTile];
    if (threadIdx.x == 0) { blk_pending = 0u; blk_done = 0u; blk_scan = 0u; }
    constexpr bool tracked = TRACKED;  // = (mode & kNnTrack) != 0
    unsigned int slot = threadIdx.x;  // the point of the tile this thread searches
    if (tracked) {
        // phase A: every point tries the cheap way (its data is requested before the barrier thread 0's pose needs)
        // A query inside its margin keeps its K neighbours as a SET (KnnTrack, voxel_map.cuh): nothing is gathered, sorted
        // or stored for it - nn_pos keeps the order of the last full search, and what k_icp_fit derived from the set
        // (a plane / a line does not depend on the order of its five points beyond rounding) stays valid.
        bool need_scan = false;
        const bool mine = threadIdx.x < tc.count;
        const unsigned int p = tc.first + (mine ? threadIdx.x : 0u);
        const size_t row = static_cast<size_t>(tc.out_base + p);
        float4 sp = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        KnnTrack t;
        t.qx = t.qy = t.qz = 0.0f; t.margin = -1.0f;
        if (mine) {
            sp = bv.src[tc.src_base + p];
            t = track[row];
        }
        __syncthreads();
        if (mine) {
            if (finite3(sp.x, sp.y, sp.z) && map.n_pts != 0) {
                double wx, wy, wz;
                pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
                need_scan = !knn_track_holds(t, static_cast<float>(wx), static_cast<float>(wy), static_cast<float>(wz));
            }
        }
        const unsigned int lane = threadIdx.x & 31;
        const unsigned int mask = __ballot_sync(0xffffffffu, need_scan);
        unsigned int base = 0;
        if (lane == 0 && mask != 0u) base = atomicAdd(&blk_scan, static_cast<unsigned int>(__popc(mask)));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (need_scan) scan_list[base + __popc(mask & ((1u << lane) - 1u))] = static_cast<unsigned char>(threadIdx.x);
        __syncthreads();
        // phase B: the first blk_scan threads search the points that need it
        slot = threadIdx.x < blk_scan ? scan_list[threadIdx.x] : kTile;
    }
    const bool in_tile = slot < tc.count;
    const unsigned int p = tc.first + (in_tile ? slot : 0u);
    const float4 sp = bv.src[tc.src_base + p];
    const size_t row = static_cast<size_t>(tc.out_base + p);
    unsigned int* out = nn_pos + row * K;
    // (loaded before sp is looked at, and - in the untracked kernel - before the barrier the pose needs)
    unsigned int seeds[K];
#pragma unroll
    for (int j = 0; j < K; ++j) seeds[j] = (mode & kNnSeeds) && in_tile ? out[j] : kNoPos;
    if (!tracked) __syncthreads();
    // non-finite source points are skipped: P2P as the reference (pcl::isFinite, icp_registration.cpp:64),
    // P2Plane as deviation D1 (the reference would poison H with NaN)
    const bool valid = in_tile && finite3(sp.x, sp.y, sp.z) && map.n_pts != 0;
    bool done = true, same = false;
    KnnResult<K> nn;
    knn_init(nn);
    KnnTrack tr;
    tr.qx = tr.qy = tr.qz = 0.0f; tr.margin = -1.0f;
    if (valid) {
        double wx, wy, wz;
        pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
        const float qx = static_cast<float>(wx), qy = static_cast<float>(wy), qz = static_cast<float>(wz);
        if (tracked) done = knn_query_fast_track<K>(map, qx, qy, qz, nn, seeds, tr);
        else done = knn_query_fast<K>(map, qx, qy, qz, nn, seeds, (mode & kNnTwoPass) != 0);
        // the same neighbours (as a set) as in the previous iteration: what k_icp_fit derived from them still holds
        same = done && (mode & kNnSeeds) != 0;
        same = same && knn_same_set<K>(seeds, nn.pos);
    }
    if (in_tile) {
#pragma unroll
        for (int j = 0; j < K; ++j) out[j] = nn.pos[j];
        if (plane_valid && !same) plane_valid[row] = 0;  // k_icp_fit sets it again
        if (track) track[row] = tr;  // margin -1 unless this was a tracked search that ended here
    }
    tile_queue_append(!done, static_cast<unsigned int>(row), tc.scan, &blk_pending, &blk_done, staged, queue, local_rows, local_n);
}
template <int K, bool TRACKED>
__global__ void __launch_bounds__(kTile, TRACKED ? LR_NN_TRACK_MIN_BLOCKS : LR_NN_MIN_BLOCKS) k_icp_nn(VoxelMapView map, BatchView bv,
                                                                    const AlignState* __restrict__ states, int ignore_stop,
                                                                    int mode, unsigned int* __restrict__ nn_pos,
                                                                    unsigned char* __restrict__ plane_valid, KnnTrack* track,
                                                                    RingQueue queue) {
    icp_nn_tile<K, TRACKED>(blockIdx.x, map, bv, states, ignore_stop, mode, nn_pos, plane_valid, track, queue);
}

// Stage 2 of LARGE jobs (batches, relocalisation), one queued query per thread (knn_query_finish: corner lists, fine
// shells, coarse levels).  With tens of thousands of queued queries the 32-queries-per-warp form keeps far more
// memory requests in flight than a warp per query can, and wins on throughput despite its divergence.  Persistent
// grid-stride launch (the queue length lives on the device).
#ifndef LR_FINISH_MIN_BLOCKS
#define LR_FINISH_MIN_BLOCKS 8  // 64 registers: relocalisation stage 2 1.5x faster than at 80
#endif
template <int K>
__global__ void __launch_bounds__(128, LR_FINISH_MIN_BLOCKS) k_icp_nn_finish(VoxelMapView map, CoarseLevels coarse, BatchView bv,
                                                       const AlignState* __restrict__ states, unsigned int* __restrict__ nn_pos,
                                                       KnnTrack* track, RingQueue queue, unsigned int min_count, unsigned int max_count) {
    const unsigned int n = *queue.count;
    if (n < min_count || n >= max_count) return;  // short queues are k_icp_nn_rings', very long ones k_icp_nn_pyr's
    // Queries differ several-fold in cost, so warps do not own a fixed share of the queue: each one takes the next
    // 32 entries from a shared cursor whenever it has finished its last batch.
    const unsigned int lane = threadIdx.x & 31;
    while (true) {
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(queue.count + 1, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n) break;
        const unsigned int e = base + lane;
        if (e >= n) continue;
        const uint2 q = queue.entries[e];
        const size_t src_idx = bv.offsets ? static_cast<size_t>(q.x) : static_cast<size_t>(q.x) - static_cast<size_t>(q.y) * bv.n_single;
        const float4 sp = bv.src[src_idx];
        Pose T;
        pose_load(T, states[q.y].pose);
        double wx, wy, wz;
        pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
        const float qx = static_cast<float>(wx), qy = static_cast<float>(wy), qz = static_cast<float>(wz);
        unsigned int* out = nn_pos + static_cast<size_t>(q.x) * K;
        KnnResult<K> nn;
        knn_init(nn);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const unsigned int sp_j = out[j];
            if (sp_j < map.n_pts) {
                const float4 c = map.pts[sp_j];
                knn_offer(map.pts, nn, dis2_f32(qx, qy, qz, c.x, c.y, c.z), sp_j);
            }
        }
        // a search that ends with the mid level's list leaves a margin behind, like a tracked stage-1 search: the far
        // points of a scan (sparse parts of the map) take the shortcut in the next iterations instead of queueing again
        float margin = -1.0f;
        knn_query_finish<K>(map, coarse, qx, qy, qz, nn, track ? &margin : nullptr);
#pragma unroll
        for (int j = 0; j < K; ++j) out[j] = nn.pos[j];
        if (track) {
            KnnTrack tr;
            tr.qx = qx; tr.qy = qy; tr.qz = qz; tr.margin = margin;
            track[q.x] = tr;
        }
    }
}

// ---- stage-2 queue in SPATIAL order --------------------------------------------------------------------------------------
// The queue's order is the arrival order of tiles and, inside a tile, of atomics: the 32 queries of a warp lie metres
// apart, walk different cells for different lengths, and 9 lanes of 32 are busy on average.  For the long queues of a
// global relocalisation (thousands of hypotheses of ONE scan: the queued queries of a wave fill the space around the
// map many times over) a counting sort by the query's bin (a cube of `bin` metres, hashed into a table of buckets) puts
// queries that walk the SAME cells into neighbouring lanes: same branches, same addresses (broadcast loads).
// Three kernels behind the device-side queue length: count (also remembers each entry's bucket), scan (exclusive_scan_u32),
// scatter.  Which entry a lane serves never changes a result.
__device__ __forceinline__ void queue_entry_query(const uint2 q, const BatchView& bv, const AlignState* __restrict__ states,
                                                  float& qx, float& qy, float& qz) {
    const size_t src_idx = bv.offsets ? static_cast<size_t>(q.x) : static_cast<size_t>(q.x) - static_cast<size_t>(q.y) * bv.n_single;
    const float4 sp = bv.src[src_idx];
    Pose T;
    pose_load(T, states[q.y].pose);
    double wx, wy, wz;
    pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
    qx = static_cast<float>(wx); qy = static_cast<float>(wy); qz = static_cast<float>(wz);
}
__global__ void __launch_bounds__(256) k_queue_bin_count(BatchView bv, const AlignState* __restrict__ states, RingQueue queue,
                                                         unsigned int min_count, float inv_bin, unsigned int bucket_mask, int sub_bits,
                                                         unsigned int* __restrict__ bucket_of, unsigned int* hist) {
    const unsigned int n = *queue.count;
    if (n < min_count) return;
    for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        float qx, qy, qz;
        queue_entry_query(queue.entries[e], bv, states, qx, qy, qz);
        // bucket = hash of the group of 2^sub_bits bins per axis the query's bin belongs to, then the bin's Morton code
        // inside the group: neighbouring buckets of a group are neighbouring bins
        const int bx = cell_of(cell_coord_f(qx, inv_bin)), by = cell_of(cell_coord_f(qy, inv_bin)), bz = cell_of(cell_coord_f(qz, inv_bin));
        const unsigned long long key = pack_cell(bx >> sub_bits, by >> sub_bits, bz >> sub_bits);
        unsigned int mort = 0u;
        for (int j = 0; j < sub_bits; ++j)
            mort |= (((static_cast<unsigned int>(bx) >> j) & 1u) << (3 * j)) | (((static_cast<unsigned int>(by) >> j) & 1u) << (3 * j + 1)) |
                    (((static_cast<unsigned int>(bz) >> j) & 1u) << (3 * j + 2));
        const unsigned int b = ((hash_block(key) << (3 * sub_bits)) | mort) & bucket_mask;
        bucket_of[e] = b;
        atomicAdd(&hist[b], 1u);
    }
}
__global__ void __launch_bounds__(256) k_queue_bin_scatter(RingQueue queue, unsigned int min_count, const unsigned int* __restrict__ bucket_of,
                                                           unsigned int* cursor, uint2* __restrict__ sorted) {
    const unsigned int n = *queue.count;
    if (n < min_count) return;
    for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x)
        sorted[atomicAdd(&cursor[bucket_of[e]], 1u)] = queue.entries[e];
}

// Stage 2 of VERY LONG queues (global relocalisation: half the points of a wrong hypothesis hang metres away from every
// surface; the unseeded first iteration of a batch): ball queries through the block pyramid (PyrWalk, voxel_map.cuh),
// one walk per LANE, every lane of a warp in the same step loop, and a lane whose walk has ended takes the next queued
// query as soon as kPyrRefill lanes are free - no lane waits for the longest walk of its warp.
#ifndef LR_PYR_MIN_BLOCKS
#define LR_PYR_MIN_BLOCKS 8
#endif
#ifndef LR_PYR_REFILL
#define LR_PYR_REFILL 8
#endif
template <int K>
__global__ void __launch_bounds__(128, LR_PYR_MIN_BLOCKS) k_icp_nn_pyr(VoxelMapView map, const __grid_constant__ PyrView py, BatchView bv,
                                                    const AlignState* __restrict__ states, unsigned int* __restrict__ nn_pos,
                                                    KnnTrack* track, RingQueue queue, unsigned int min_count) {
    const unsigned int n = *queue.count;
    if (n < min_count) return;
    const unsigned int lane = threadIdx.x & 31;
    PyrWalk<K> w;
    unsigned long long todo[kPyrStack];
    constexpr int kFree = 4, kDead = 5;
    int st = kFree, bit = 0;
    bool exhausted = false;  // warp-uniform: the queue's cursor has passed its end
    unsigned int row = 0;
    while (true) {
        // two kinds of step - a point of an opened cell, or the next child of the node on top of the stack (test, open) -
        // and the warp runs the kind more lanes are due for; the other lanes wait for their turn.  Free lanes are handed
        // the next queued queries once LR_PYR_REFILL of them have gathered (or nothing else is left to do).
        const unsigned int b_node = __ballot_sync(0xffffffffu, st == kPyrNode), b_point = __ballot_sync(0xffffffffu, st == kPyrPoint),
                           b_free = __ballot_sync(0xffffffffu, st == kFree);
        const int n_node = __popc(b_node), n_point = __popc(b_point), n_free = __popc(b_free);
        if ((b_node | b_point | b_free) == 0u) break;
        if (n_free >= LR_PYR_REFILL || (b_node | b_point) == 0u) {  // hand out queued queries
            unsigned int base = 0;
            if (lane == 0) base = atomicAdd(queue.count + 1, static_cast<unsigned int>(n_free));
            base = __shfl_sync(0xffffffffu, base, 0);
            exhausted = base + static_cast<unsigned int>(n_free) >= n;
            if (st == kFree) {
                const unsigned int e = base + static_cast<unsigned int>(__popc(b_free & ((1u << lane) - 1u)));
                st = kDead;
                if (e < n) {
                    const uint2 q = queue.entries[e];
                    const size_t src_idx = bv.offsets ? static_cast<size_t>(q.x) : static_cast<size_t>(q.x) - static_cast<size_t>(q.y) * bv.n_single;
                    const float4 sp = bv.src[src_idx];
                    Pose T;
                    pose_load(T, states[q.y].pose);
                    double wx, wy, wz;
                    pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
                    const float qx = static_cast<float>(wx), qy = static_cast<float>(wy), qz = static_cast<float>(wz);
                    row = q.x;
                    const unsigned int* out = nn_pos + static_cast<size_t>(row) * K;
                    knn_init(w.res);
#pragma unroll
                    for (int j = 0; j < K; ++j) {
                        const unsigned int sp_j = out[j];
                        if (sp_j < map.n_pts) {
                            const float4 c = map.pts[sp_j];
                            knn_offer(map.pts, w.res, dis2_f32(qx, qy, qz, c.x, c.y, c.z), sp_j);
                        }
                    }
                    w.start(map, py, qx, qy, qz);
                    st = kPyrNode;
                }
            }
        } else if (n_point >= n_node) {
            if (st == kPyrPoint) st = w.point_step(map);
        } else if (st == kPyrNode) {
            st = w.node_step(map, py, todo, bit);
            if (st == kPyrDone) {
                unsigned int* out = nn_pos + static_cast<size_t>(row) * K;
#pragma unroll
                for (int j = 0; j < K; ++j) out[j] = w.res.pos[j];
                if (track) {
                    KnnTrack tr;
                    tr.qx = w.qx; tr.qy = w.qy; tr.qz = w.qz; tr.margin = -1.0f;
                    track[row] = tr;
                }
                st = exhausted ? kDead : kFree;
            }
        }
    }
}

// One queued query, by one warp: everything after stage 1 (warp_query_finish), seeded with what stage 1 found.
template <int K>
__device__ __forceinline__ void icp_rings_query(const uint2 q, const VoxelMapView& map, const CoarseLevels& coarse, const BatchView& bv,
                                                const AlignState* __restrict__ states, unsigned int* __restrict__ nn_pos, KnnTrack* track) {
    const unsigned int lane = threadIdx.x & 31;
    // scratch rows and source points coincide for a batch; hypotheses of one scan share its points
    const size_t src_idx = bv.offsets ? static_cast<size_t>(q.x) : static_cast<size_t>(q.x) - static_cast<size_t>(q.y) * bv.n_single;
    const float4 sp = bv.src[src_idx];
    Pose T;
    pose_load(T, states[q.y].pose);
    double wx, wy, wz;
    pose_apply(T, static_cast<double>(sp.x), static_cast<double>(sp.y), static_cast<double>(sp.z), wx, wy, wz);
    const float qx = static_cast<float>(wx), qy = static_cast<float>(wy), qz = static_cast<float>(wz);
    unsigned int* out = nn_pos + static_cast<size_t>(q.x) * K;
    KnnResult<K> nn;  // replicated: every lane holds the same set
    knn_init(nn);
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const unsigned int sp_j = out[j];
        if (sp_j < map.n_pts) {
            const float4 c = map.pts[sp_j];
            knn_offer(map.pts, nn, dis2_f32(qx, qy, qz, c.x, c.y, c.z), sp_j);
        }
    }
    float margin = -1.0f;
    warp_query_finish<K>(map, coarse, qx, qy, qz, nn, track ? &margin : nullptr);
    __syncwarp();
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < K; ++j) out[j] = nn.pos[j];
        if (track) {  // (see k_icp_nn_finish)
            KnnTrack tr;
            tr.qx = qx; tr.qy = qy; tr.qz = qz; tr.margin = margin;
            track[q.x] = tr;
        }
    }
}
// Stage 2 of SMALL jobs (one scan): ONE QUERY PER WARP (knn_warp.cuh), seeded with what stage 1 found.  The GPU is
// mostly idle, so what counts is the latency of the slowest query, and 32 lanes cut that ~10x.
// Persistent warp-stride launch: the queue length is only known on the device.
template <int K>
__device__ __forceinline__ void icp_rings_warps(unsigned int n, unsigned int warp, unsigned int n_warps, const VoxelMapView& map,
                                                const CoarseLevels& coarse, const BatchView& bv, const AlignState* __restrict__ states,
                                                unsigned int* __restrict__ nn_pos, KnnTrack* track, const RingQueue& queue) {
    const unsigned int lane = threadIdx.x & 31;
    // Queries differ many-fold in cost (a list scan, or shells up the coarse levels for a point far from everything), and
    // the phase ends with the slowest warp: warps take the next query from a shared cursor (queue.count[1], zero at the
    // start of every evaluation) instead of owning a fixed stride of the queue.
    (void)warp; (void)n_warps;
    while (true) {
        unsigned int e = 0;
        if (lane == 0) e = atomicAdd(queue.count + 1, 1u);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        icp_rings_query<K>(queue.entries[e], map, coarse, bv, states, nn_pos, track);
    }
}
template <int K>
__global__ void __launch_bounds__(128) k_icp_nn_rings(VoxelMapView map, CoarseLevels coarse, BatchView bv,
                                                      const AlignState* __restrict__ states, unsigned int* __restrict__ nn_pos,
                                                      KnnTrack* track, RingQueue queue, unsigned int max_count) {
    const unsigned int n = *queue.count;
    if (n >= max_count) return;  // long queues are k_icp_nn_finish's
    icp_rings_warps<K>(n, (blockIdx.x * blockDim.x + threadIdx.x) >> 5, (gridDim.x * blockDim.x) >> 5, map, coarse, bv, states, nn_pos, track, queue);
}

// ---- the search on its own (locreg_knn parity probe): the same two stages on raw queries ---------------------------
// Stage 1 for queries that are already in map coordinates: no pose, no seeds; unfinished queries are queued with
// (row, 0), and k_knn_rings / k_knn_export complete the probe.
template <int K>
__global__ void __launch_bounds__(kTile, LR_NN_MIN_BLOCKS) k_knn_stage1(VoxelMapView map, const float4* __restrict__ q, unsigned int nq,
                                                                        unsigned int* __restrict__ nn_pos, RingQueue queue) {
    __shared__ unsigned int blk_pending, blk_done;
    __shared__ unsigned int staged[kTile];
    if (threadIdx.x == 0) { blk_pending = 0u; blk_done = 0u; }
    __syncthreads();
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool done = true;
    if (i < nq) {
        const float4 p = q[i];
        KnnResult<K> nn;
        knn_init(nn);
        if (finite3(p.x, p.y, p.z) && map.n_pts != 0) done = knn_query_fast<K>(map, p.x, p.y, p.z, nn, nullptr, true);
#pragma unroll
        for (int j = 0; j < K; ++j) nn_pos[static_cast<size_t>(i) * K + j] = nn.pos[j];
    }
    tile_queue_append(!done, i, 0u, &blk_pending, &blk_done, staged, queue);
}
template <int K>
__global__ void __launch_bounds__(128) k_knn_rings(VoxelMapView map, CoarseLevels coarse, const float4* __restrict__ q,
                                                   unsigned int* __restrict__ nn_pos, RingQueue queue) {
    const unsigned int n = *queue.count;
    const unsigned int lane = threadIdx.x & 31;
    const unsigned int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (unsigned int e = warp; e < n; e += n_warps) {
        const unsigned int i = queue.entries[e].x;
        const float4 p = q[i];
        unsigned int* out = nn_pos + static_cast<size_t>(i) * K;
        KnnResult<K> nn;
        knn_init(nn);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const unsigned int sp_j = out[j];
            if (sp_j < map.n_pts) {
                const float4 c = map.pts[sp_j];
                knn_offer(map.pts, nn, dis2_f32(p.x, p.y, p.z, c.x, c.y, c.z), sp_j);
            }
        }
        warp_query_finish<K>(map, coarse, p.x, p.y, p.z, nn);
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < K; ++j) out[j] = nn.pos[j];
        }
    }
}
template <int K>
__global__ void __launch_bounds__(128) k_knn_finish(VoxelMapView map, CoarseLevels coarse, const float4* __restrict__ q,
                                                    unsigned int* __restrict__ nn_pos, RingQueue queue) {
    const unsigned int n = *queue.count;
    for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const unsigned int i = queue.entries[e].x;
        const float4 p = q[i];
        unsigned int* out = nn_pos + static_cast<size_t>(i) * K;
        KnnResult<K> nn;
        knn_init(nn);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const unsigned int sp_j = out[j];
            if (sp_j < map.n_pts) {
                const float4 c = map.pts[sp_j];
                knn_offer(map.pts, nn, dis2_f32(p.x, p.y, p.z, c.x, c.y, c.z), sp_j);
            }
        }
        knn_query_finish<K>(map, coarse, p.x, p.y, p.z, nn);
#pragma unroll
        for (int j = 0; j < K; ++j) out[j] = nn.pos[j];
    }
}
// canonical positions -> the caller's original indices (-1 = none)
__global__ void k_knn_export(VoxelMapView map, const unsigned int* __restrict__ nn_pos, size_t n, int* __restrict__ idx) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = nn_pos[i] != kNoPos ? knn_index_of(map.pts, nn_pos[i]) : -1;
}

// ---- K_B: fit + gates + accumulate ----------------------------------------------------------------------------
// A thread handles ONE point, so there is nothing to accumulate per thread: it stages its residual row(s)
// (J[0..5], r) in shared memory, and each warp then forms the 28 sums of products over its own 32 points with lane l
// owning one entry of (H upper triangle | B | sum_sq) - 2 LDS + 1 DFMA per point and entry, instead of 28 products
// per thread followed by 30 five-step shuffle trees.  The sums run in point order inside a warp, then over the 8
// warps in order: reproducible for a fixed launch shape.
constexpr int kRowStride = 7;  // J[6] + r

// ---- K_B1: plane fit (P2Plane) ----------------------------------------------------------------------------------
// The plane of a point depends on its five neighbours (and their order) only.  Stage 1 clears plane_valid[row] where
// they changed - every point in the first iteration, 1 % by the tenth - and leaves it alone otherwise: the cached
// coefficients are then the ones a new fit would reproduce bit for bit.  A fit is ~500 dependent fp64 instructions, so
// the rows that need one are compacted first: a block gathers them over `group` consecutive tiles and only then fits,
// every lane busy, instead of one divergent lane holding a warp (and a barrier its whole tile) for the length of a fit.
#ifndef LR_FIT_GROUP
#define LR_FIT_GROUP 16
#endif
constexpr int kFitGroup = LR_FIT_GROUP;
#ifndef LR_FIT_MIN_BLOCKS
#define LR_FIT_MIN_BLOCKS 4  // 64 registers: measured 2..6 on B200 (3: +2 % step time, 2: +4 %, 5-6: +0.5 %)
#endif
// MAXG: the largest `group` the caller passes (sizes the shared-memory list)
template <int MAXG>
__device__ __forceinline__ void icp_fit_group(unsigned int block_index, const VoxelMapView& map, const IcpParams& prm, const BatchView& bv,
                                              const AlignState* __restrict__ states, int ignore_stop, const unsigned int* __restrict__ nn_pos,
                                              unsigned char* plane_valid, double* plane_cache, unsigned char* plane_stat, unsigned int group) {
    __shared__ TileCoord tcs[MAXG];
    __shared__ unsigned int list[MAXG * kTile];
    __shared__ unsigned int list_n;
    if (threadIdx.x < group) {
        TileCoord c = locate_tile_thread(bv, block_index * group + threadIdx.x);
        if (c.valid && states[c.scan].stop && !ignore_stop) c.valid = false;
        tcs[threadIdx.x] = c;
    }
    if (threadIdx.x == 0) list_n = 0u;
    __syncthreads();
    const unsigned int lane = threadIdx.x & 31;
    // all of the thread's flags first (independent loads: one round trip instead of `group` of them), then the appends
    unsigned int need_bits = 0u;
#pragma unroll
    for (unsigned int g = 0; g < static_cast<unsigned int>(MAXG); ++g) {
        if (g < group && tcs[g].valid && threadIdx.x < tcs[g].count) {
            const size_t row = static_cast<size_t>(tcs[g].out_base + tcs[g].first + threadIdx.x);
            need_bits |= (plane_valid[row] == 0 ? 1u : 0u) << g;
        }
    }
    for (unsigned int g = 0; g < group; ++g) {
        const bool need = (need_bits >> g) & 1u;
        const unsigned int mask = __ballot_sync(0xffffffffu, need);
        if (mask == 0u) continue;
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(&list_n, static_cast<unsigned int>(__popc(mask)));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (need) list[base + __popc(mask & ((1u << lane) - 1u))] = static_cast<unsigned int>(tcs[g].out_base + tcs[g].first + threadIdx.x);
    }
    __syncthreads();
    const unsigned int n = list_n;
    for (unsigned int i = threadIdx.x; i < n; i += kTile) {
        const size_t row = list[i];
        KnnResult<5> nn;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            nn.pos[j] = nn_pos[row * 5 + j];
            nn.d2[j] = 0.0f;  // not needed by the fit
        }
        double pl[4] = {0, 0, 0, 0};
        plane_stat[row] = icp_fit_plane(map, prm, nn, pl);
        reinterpret_cast<double4*>(plane_cache)[row] = make_double4(pl[0], pl[1], pl[2], pl[3]);
        plane_valid[row] = 1;
    }
}
__global__ void __launch_bounds__(kTile, LR_FIT_MIN_BLOCKS)
k_icp_fit(VoxelMapView map, IcpParams prm, BatchView bv, const AlignState* __restrict__ states, int ignore_stop,
          const unsigned int* __restrict__ nn_pos, unsigned char* plane_valid, double* plane_cache, unsigned char* plane_stat,
          unsigned int group) {
    icp_fit_group<kFitGroup>(blockIdx.x, map, prm, bv, states, ignore_stop, nn_pos, plane_valid, plane_cache, plane_stat, group);
}

// Upper-triangle entry e = 0..20 of a 6x6 matrix -> its row (col = false) or column (col = true), 3 bits per entry.
constexpr unsigned long long tri_table(bool col) {
    unsigned long long t = 0;
    int e = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b, ++e) t |= static_cast<unsigned long long>(col ? b : a) << (3 * e);
    return t;
}
template <int ROWS>
struct RowSink {
    double* rows;  // this thread's ROWS staged rows
    int n_rows;
    bool eff, inl;
    __device__ __forceinline__ void row(const double (&J)[6], double r) {
        double* o = rows + n_rows * kRowStride;
#pragma unroll
        for (int i = 0; i < 6; ++i) o[i] = J[i];
        o[6] = r;
        ++n_rows;
    }
    __device__ __forceinline__ void inc_eff() { eff = true; }
    __device__ __forceinline__ void inc_inl() { inl = true; }
};

#ifndef LR_POST_MIN_BLOCKS
#define LR_POST_MIN_BLOCKS 6  // 40 registers; the fit lives in k_icp_fit, what is left is latency-bound
#endif
template <int METHOD>
__device__ __forceinline__ void icp_post_tile(unsigned int tile, const VoxelMapView& map, const IcpParams& prm, const BatchView& bv,
                                              const AlignState* __restrict__ states, int ignore_stop, const unsigned int* __restrict__ nn_pos,
                                              double* __restrict__ partials, unsigned char* gate, int* nn_idx,
                                              const double* __restrict__ plane_cache, const unsigned char* __restrict__ plane_stat) {
    constexpr int K = METHOD == kIcpP2P ? 1 : 5;
    constexpr int ROWS = METHOD == kIcpP2Plane ? 1 : 3;  // residual rows per inlier (P2P, P2Line: 3-vector residuals)
    __shared__ Pose T;
    __shared__ double rows[kTile * ROWS * kRowStride + 1];  // + 1: the pad column of the last row (see the Gram step)
    __shared__ double gram[kTile / 32][64];
    __shared__ int counts[kTile / 32][2];
    const TileCoord tc = locate_tile(bv, tile);
    if (!tc.valid) return;
    const AlignState* st = states + tc.scan;
    if (st->stop && !ignore_stop) return;
    if (threadIdx.x == 0) pose_load(T, st->pose);
    // the point's own data is requested before the barrier: its round trip overlaps thread 0's pose load
    const bool in_tile = threadIdx.x < tc.count;
    const unsigned int p = tc.first + (in_tile ? threadIdx.x : 0u);
    float4 sp = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    KnnResult<K> nn;
    double4 pl = make_double4(0, 0, 0, 0);
    unsigned char pst = kPlaneNone;
    if (in_tile) {
        sp = bv.src[tc.src_base + p];
        const unsigned int* in = nn_pos + (tc.out_base + p) * K;
        const bool want_nn = METHOD != kIcpP2Plane || nn_idx != nullptr;  // P2Plane works from k_icp_fit's plane
#pragma unroll
        for (int j = 0; j < K; ++j) {
            nn.pos[j] = want_nn ? in[j] : kNoPos;
            nn.d2[j] = 0.0f;  // not needed downstream
        }
        if (METHOD == kIcpP2Plane) {  // the plane comes from k_icp_fit; fetched together with the point
            pl = reinterpret_cast<const double4*>(plane_cache)[tc.out_base + p];
            pst = plane_stat[tc.out_base + p];
        }
    }
    RowSink<ROWS> sink{rows + threadIdx.x * ROWS * kRowStride, 0, false, false};
    __syncthreads();
    if (in_tile) {
        unsigned char g = kGateSkipped;
        if (finite3(sp.x, sp.y, sp.z)) {
            const double qx = sp.x, qy = sp.y, qz = sp.z;
            double wx, wy, wz;
            pose_apply(T, qx, qy, qz, wx, wy, wz);
            if (METHOD == kIcpP2P) g = icp_p2p_post(map, prm, T, qx, qy, qz, wx, wy, wz, reinterpret_cast<const KnnResult<1>&>(nn), sink);
            else if (METHOD == kIcpP2Line) g = icp_p2line_post(map, prm, T, qx, qy, qz, wx, wy, wz, reinterpret_cast<const KnnResult<5>&>(nn), sink);
            else {
                const double n[4] = {pl.x, pl.y, pl.z, pl.w};
                g = icp_p2plane_residual(prm, T, qx, qy, qz, wx, wy, wz, pst, n, sink);
            }
        }
        if (gate) gate[tc.out_base + p] = g;
        if (nn_idx) {
#pragma unroll
            for (int j = 0; j < K; ++j)
                nn_idx[(tc.out_base + p) * K + j] = nn.pos[j] != kNoNeighbour ? __float_as_int(map.pts[nn.pos[j]].w) : -1;
        }
    }
    // points without a residual contribute zero rows (written here, once, rather than zeroing every row up front)
    for (int i = sink.n_rows * kRowStride; i < ROWS * kRowStride; ++i) sink.rows[i] = 0.0;
    // Per-warp Gram matrix G = R^T R of the warp's 32 * ROWS staged rows R = [J | r] on the fp64 tensor cores:
    // mma.m8n8k4 takes A (8 x 4, A[m][k] = R[4 ks + k][m]) and B (4 x 8, B[k][n] = R[4 ks + k][n]); a lane's A and B
    // fragments are the same element R[4 ks + (lane & 3)][lane >> 2], so one 8 B shared-memory load per lane feeds four
    // rows - where one lane per matrix entry needed two loads and an FMA per row.  Column 7 does not exist: the lanes that
    // would load it pass zeros, which only reach row / column 7 of G (nobody reads them).
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned int eff_mask = __ballot_sync(0xffffffffu, sink.eff);
    __syncwarp();  // the warp's row stores are visible to its loads below
    const unsigned int inl_mask = __ballot_sync(0xffffffffu, sink.inl);
    const double* wrows = rows + warp * 32 * ROWS * kRowStride + (lane & 3) * kRowStride + (lane >> 2);
    double g0 = 0.0, g1 = 0.0;  // G[lane >> 2][2 * (lane & 3) + {0, 1}]
#pragma unroll
    for (int ks = 0; ks < 8 * ROWS; ++ks) {
        // (lanes 28..31 would read column 7 = the next row's first element, for the warp's last row another warp's
        // data: they feed row / column 7 of G, which nobody reads, with zeros instead)
        const double a = lane < 28 ? wrows[4 * ks * kRowStride] : 0.0;
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                     : "+d"(g0), "+d"(g1)
                     : "d"(a), "d"(a));
    }
    gram[warp][(lane >> 2) * 8 + 2 * (lane & 3)] = g0;
    gram[warp][(lane >> 2) * 8 + 2 * (lane & 3) + 1] = g1;
    if (lane == 0) {
        counts[warp][0] = __popc(eff_mask);
        counts[warp][1] = __popc(inl_mask);
    }
    __syncthreads();
    // thread -> entry: 0..20 = H(a, b) upper triangle, 21..26 = B[a] = -sum J[a] r, 27 = sum r r, 28 / 29 = counts
    // (3 bits per entry, packed: rows 0 0 0 0 0 0 1 1 1 1 1 2 2 2 2 3 3 3 4 4 5, columns 0..5 1..5 2..5 3..5 4 5 5)
    if (threadIdx.x < 30) {
        constexpr unsigned long long kTriRow = tri_table(false), kTriCol = tri_table(true);
        const int e = threadIdx.x;
        double t = 0;
        if (e < 28) {
            int ea = 6, eb = 6;
            if (e < 21) {
                ea = static_cast<int>(kTriRow >> (3 * e)) & 7;
                eb = static_cast<int>(kTriCol >> (3 * e)) & 7;
            } else if (e < 27) {
                ea = e - 21;
            }
#pragma unroll
            for (int w = 0; w < kTile / 32; ++w) t += gram[w][ea * 8 + eb];
            if (e >= 21 && e < 27) t = -t;
        } else {
            int c = 0;
#pragma unroll
            for (int w = 0; w < kTile / 32; ++w) c += counts[w][e - 28];
            t = static_cast<double>(c);
        }
        partials[static_cast<size_t>(tile) * kPartialDoubles + threadIdx.x] = t;
    }
}
template <int METHOD>
__global__ void __launch_bounds__(kTile, METHOD == kIcpP2Plane ? LR_POST_MIN_BLOCKS : 2)
k_icp_post(VoxelMapView map, IcpParams prm, BatchView bv, const AlignState* __restrict__ states, int ignore_stop,
           const unsigned int* __restrict__ nn_pos, double* __restrict__ partials, unsigned char* gate, int* nn_idx,
           unsigned int* ring_count, const double* __restrict__ plane_cache, const unsigned char* __restrict__ plane_stat) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { ring_count[0] = 0u; ring_count[1] = 0u; }  // both search stages of this evaluation are done
    icp_post_tile<METHOD>(blockIdx.x, map, prm, bv, states, ignore_stop, nn_pos, partials, gate, nn_idx, plane_cache, plane_stat);
}

// ---- K_C: per-scan reduction + Gauss-Newton update ------------------------------------------------------------
__device__ __forceinline__ void result_from_acc(DevResult& r, const double* acc30) {
    r.n_effective = static_cast<long long>(acc30[28]);
    r.n_inlier = static_cast<long long>(acc30[29]);
    r.sum_sq_res = acc30[27];
}
// Applies one update outcome (0 failed, 1 updated, 2 converged, 3 abort without writing the pose, 4 abort with the
// pose written) to the bookkeeping; returns true if the loop must stop.
__device__ __forceinline__ bool apply_outcome(int outcome, DevResult& r) {
    r.degenerate = (outcome == 0 || outcome == 3 || outcome == 4) ? 1 : 0;
    if (outcome == 1 || outcome == 2) r.updates += 1;
    if (outcome == 2) r.converged = 1;
    if (outcome == 3) r.pose_written = 0;
    return outcome == 2 || outcome == 3 || outcome == 4;
}

// Sum over tiles [t0, t1) of partial-row entry `lane` (< 30; other lanes get 0), in a fixed order: four interleaved
// running sums keep four loads in flight (the loop is pure latency).  partials_b (optional): a second partial row per
// tile (k_icp_pending, icp_fused.cuh), added after the first ones.
__device__ __forceinline__ double icp_sum_tiles(const double* __restrict__ partials, const double* __restrict__ partials_b,
                                                unsigned int t0, unsigned int t1, unsigned int lane) {
    double v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    if (lane < 30) {
        const double* col = partials + lane;
        unsigned int t = t0;
        for (; t + 4 <= t1; t += 4) {
            v0 += col[static_cast<size_t>(t) * kPartialDoubles];
            v1 += col[static_cast<size_t>(t + 1) * kPartialDoubles];
            v2 += col[static_cast<size_t>(t + 2) * kPartialDoubles];
            v3 += col[static_cast<size_t>(t + 3) * kPartialDoubles];
        }
        for (; t < t1; ++t) v0 += col[static_cast<size_t>(t) * kPartialDoubles];
        if (partials_b) {
            double w0 = 0, w1 = 0, w2 = 0, w3 = 0;
            const double* colb = partials_b + lane;
            for (t = t0; t + 4 <= t1; t += 4) {
                w0 += colb[static_cast<size_t>(t) * kPartialDoubles];
                w1 += colb[static_cast<size_t>(t + 1) * kPartialDoubles];
                w2 += colb[static_cast<size_t>(t + 2) * kPartialDoubles];
                w3 += colb[static_cast<size_t>(t + 3) * kPartialDoubles];
            }
            for (; t < t1; ++t) w0 += colb[static_cast<size_t>(t) * kPartialDoubles];
            v0 = ((v0 + v1) + (v2 + v3)) + ((w0 + w1) + (w2 + w3));
            v1 = v2 = v3 = 0;
        }
    }
    return (v0 + v1) + (v2 + v3);
}

// Tiles [t0, t1) of item s: from tile_begin (a batch), else tiles_per_item / n_single (one scan, or hypotheses of one).
__device__ __forceinline__ void item_tiles(const BatchView& bv, unsigned int s, unsigned int& t0, unsigned int& t1) {
    if (bv.tile_begin) { t0 = bv.tile_begin[s]; t1 = bv.tile_begin[s + 1]; }
    else {
        t0 = s * bv.tiles_per_item;
        t1 = t0 + (bv.n_single + kTile - 1) / kTile;
    }
}

// One warp per scan.  mode 1: Gauss-Newton iteration (update the pose; stop on convergence or after
// max_iteration trips); mode 0: evaluation only (compute_hb, relocalisation's final score pass): record the sums,
// leave the pose.  acc_out (optional, 32 doubles per scan) receives the raw sums.
// partials_b (optional): a second partial row per tile (k_icp_pending, icp_fused.cuh), added after the first ones.
template <int METHOD>
__global__ void __launch_bounds__(128) k_icp_solve(IcpParams prm, BatchView bv, AlignState* states,
                                                   const double* __restrict__ partials, const double* __restrict__ partials_b,
                                                   int mode, double* acc_out) {
    __shared__ double sums[4][32];
    const unsigned int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned int s = blockIdx.x * 4 + warp;
    if (s >= bv.S) return;
    AlignState* st = states + s;
    if (mode == 1 && st->stop) return;
    unsigned int t0, t1;
    item_tiles(bv, s, t0, t1);
    sums[warp][lane] = icp_sum_tiles(partials, partials_b, t0, t1, lane);
    __syncwarp();
    if (lane == 0) {
        const double* acc30 = sums[warp];
        result_from_acc(st->res, acc30);
        if (acc_out)
            for (int i = 0; i < 30; ++i) acc_out[static_cast<size_t>(s) * 32 + i] = acc30[i];
        if (mode == 1) {
            Pose T;
            pose_load(T, st->pose);
            st->res.iters += 1;
            const int outcome = icp_gn_update<METHOD>(acc30, static_cast<unsigned int>(acc30[28]), prm, T);
            if (apply_outcome(outcome, st->res) || st->res.iters >= prm.max_iteration) st->stop = 1;
            pose_store(T, st->pose);
        }
    }
}

// One Gauss-Newton trip of LoamRegistration::ScanMatch (SURVEY.md 3.3), one warp per scan: the P2Plane (surf) half's and
// the P2Line (edge) half's partial rows are summed separately, in k_icp_solve's order, then added; H dx = B is solved and
// the pose updated as in the ICP loop, but with neither icp_gn_update's min_effective_pts gate (the halves' own flags do
// not gate the sum) nor P2P's /16.  A singular sum makes no update (outcome 0).  bs / be: the two halves' views of the
// same S scans (each half's tiles of scan s from its own view); states[s] is scan s's one pose, both halves evaluate at
// it.  half[2s] / half[2s + 1] receive scan s's surf / edge counts and degenerate flag as locreg_compute_hb reports them
// at the trip's pose.  mode 1: the trip; a stopped scan's warp exits.  mode 0: evaluation only (LOAM relocalisation's
// score pass), for every scan: st->res receives the summed counts and sum of squares and degenerate = singular sum; the
// pose, iters, updates and converged stay as they are.
__global__ void __launch_bounds__(128) k_loam_solve(BatchView bs, const double* __restrict__ surf, const double* __restrict__ surf_b,
                                                    int min_eff_surf, BatchView be, const double* __restrict__ edge,
                                                    const double* __restrict__ edge_b, int min_eff_edge, AlignState* states,
                                                    double eps, int max_iteration, int mode, DevResult* half) {
    __shared__ double sums[4][3][32];
    const unsigned int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned int s = blockIdx.x * 4 + warp;
    if (s >= bs.S) return;
    AlignState* st = states + s;
    if (mode == 1 && st->stop) return;
    unsigned int t0, t1;
    item_tiles(bs, s, t0, t1);
    const double a = icp_sum_tiles(surf, surf_b, t0, t1, lane);
    item_tiles(be, s, t0, t1);
    const double e = icp_sum_tiles(edge, edge_b, t0, t1, lane);
    sums[warp][0][lane] = a;
    sums[warp][1][lane] = e;
    sums[warp][2][lane] = a + e;
    __syncwarp();
    if (lane < 3) {  // lanes 0 / 1: the halves' own records (their degenerate flags need det of their own H); lane 2: the update
        const double* acc = sums[warp][lane];
        double dx[6];
        const bool solvable = gn_solve6(acc, acc + 21, dx);
        if (lane < 2) {
            DevResult& r = half[2 * static_cast<size_t>(s) + lane];
            result_from_acc(r, acc);
            r.degenerate = (!solvable || r.n_effective < (lane == 0 ? min_eff_surf : min_eff_edge)) ? 1 : 0;
        } else if (mode == 0) {
            result_from_acc(st->res, acc);
            st->res.degenerate = solvable ? 0 : 1;
        } else {
            result_from_acc(st->res, acc);
            Pose T;
            pose_load(T, st->pose);
            st->res.iters += 1;
            int outcome = 0;
            if (solvable) {
                pose_update(T, dx);
                double nrm = 0;
#pragma unroll
                for (int i = 0; i < 6; ++i) nrm += dx[i] * dx[i];
                outcome = sqrt(nrm) < eps ? 2 : 1;
            }
            if (apply_outcome(outcome, st->res) || st->res.iters >= max_iteration) st->stop = 1;
            pose_store(T, st->pose);
        }
    }
}

// poses_in -> fresh states (stop is raised at once when max_iteration <= 0: the reference's loop body never runs)
// zero_t: the Align* loops start from a zero translation (locreg_options::zero_initial_translation)
__global__ void k_states_init(const double* __restrict__ poses_in, unsigned int S, int max_iteration, int zero_t, AlignState* states) {
    const unsigned int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    AlignState st;
    for (int i = 0; i < 7; ++i) st.pose[i] = (zero_t && i >= 4) ? 0.0 : poses_in[static_cast<size_t>(s) * 7 + i];
    st.res = DevResult{0, 0, 0, 0, 0, 0, 0.0, 1, 0};
    st.stop = max_iteration <= 0 ? 1 : 0;
    st.pad = 0;
    states[s] = st;
}
// states -> poses_out (only where the reference would have written result_pose) and results
__global__ void k_states_export(const AlignState* __restrict__ states, unsigned int S, double* poses_out, DevResult* results) {
    const unsigned int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const AlignState st = states[s];
    if (poses_out && st.res.pose_written)
        for (int i = 0; i < 7; ++i) poses_out[static_cast<size_t>(s) * 7 + i] = st.pose[i];
    if (results) results[s] = st.res;
}

}  // namespace locreg
