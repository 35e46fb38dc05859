// Device versions of the cloud pre-filters that sit directly in front of every SetInputTarget / ScanMatch call in the
// reference (SURVEY.md 8f-3): pcl::removeNaNFromPointCloud (point_cloud_utils.h:13-20), pcl::CropBox (BoxFilter,
// box_filter.cpp:24-32) and pcl::VoxelGrid (VoxelFilter, voxel_filter.cpp:20-26; scan 1.0 m / map 0.5 m leaves at
// lio.cpp:236,248, loc.cpp:218).  PCL itself is not under /root/reference: these restate its published algorithms
// (PCL 1.8 filters/voxel_grid.hpp, crop_box.hpp, filter.hpp) - parity is against oracle/filters of this repo.
//   * keep-filters (NaN removal, crop box): flag -> exclusive scan -> scatter, order preserved;
//   * voxel grid: voxel index exactly as PCL computes it (float floor of p * inverse_leaf minus min_b), counting sort
//     over the dense index space, one thread per occupied voxel averaging ALL float words of its points in float32,
//     in point-index order (PCL sorts with an unstable std::sort, so its own summation order is unspecified), output
//     in ascending voxel index like PCL.
// NaN removal and the voxel grid run over a BATCH of scans (offsets[S + 1]) in one pass; a single cloud is the batch
// of one scan.  Segment s of the output is what the filter returns for scan s alone: every per-scan quantity (bounding
// box, grid, overflow rule, voxel ranks, output place) is computed per scan, and scans are kept in order.
#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "device_utils.cuh"
#include "filters.cuh"

namespace locreg {

__global__ void k_flag_finite(const unsigned char* __restrict__ raw, size_t n, size_t stride, unsigned int* flag) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    flag[i] = finite3(p[0], p[1], p[2]) ? 1u : 0u;
}
// pcl::CropBox with the identity transform, negative = false: a point is kept iff min <= p <= max on every axis
// (crop_box.hpp: "if (pt.x < min[0] || ... || pt.x > max[0] ...) -> outside"); non-finite points are dropped.
__global__ void k_flag_box(const unsigned char* __restrict__ raw, size_t n, size_t stride, float3 lo, float3 hi, unsigned int* flag) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    const bool out = !finite3(p[0], p[1], p[2]) || p[0] < lo.x || p[1] < lo.y || p[2] < lo.z || p[0] > hi.x || p[1] > hi.y || p[2] > hi.z;
    flag[i] = out ? 0u : 1u;
}
__global__ void k_compact(const unsigned char* __restrict__ raw, size_t n, size_t stride, const unsigned int* __restrict__ flag,
                          const unsigned int* __restrict__ pos, unsigned char* out) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const unsigned int* s = reinterpret_cast<const unsigned int*>(raw + i * stride);
    unsigned int* d = reinterpret_cast<unsigned int*>(out + static_cast<size_t>(pos[i]) * stride);
    for (size_t w = 0; w < stride / 4; ++w) d[w] = s[w];
}
// out_off[s] = kept points before scan s (s = 0 .. S): the exclusive scan of the flags read at the scan boundaries
__global__ void k_keep_offsets(const long long* __restrict__ offs, unsigned int S, size_t n, const unsigned int* __restrict__ pos,
                               const unsigned int* __restrict__ total, unsigned int* out_off) {
    const unsigned int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > S) return;
    const size_t o = static_cast<size_t>(offs[s]);
    out_off[s] = o < n ? pos[o] : *total;
}

// Scan of point p: the s in [lo, hi) with offs[s] <= p < offs[s + 1] (offs non-decreasing, offs[lo] <= p < offs[hi]).
__device__ __forceinline__ unsigned int scan_of(const long long* __restrict__ offs, unsigned int lo, unsigned int hi, long long p) {
    while (hi - lo > 1) {
        const unsigned int mid = (lo + hi) >> 1;
        if (offs[mid] <= p) lo = mid;
        else hi = mid;
    }
    return lo;
}

// order-preserving float <-> uint map for atomicMin / atomicMax on floats
__device__ __forceinline__ unsigned int f2ord(float f) {
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
static float ord2f(unsigned int o) {
    const unsigned int u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
    float f;
    memcpy(&f, &u, 4);
    return f;
}
// Per-scan bounding box of the finite points: mm[6 s + 0..2] min, [6 s + 3..5] max.  A warp whose points all belong to
// one scan (the common case: scans are thousands of points long) reduces in registers and issues one atomic per axis;
// a warp that straddles a scan boundary falls back to per-lane atomics.
__global__ void k_minmax(const unsigned char* __restrict__ raw, size_t n, size_t stride, const long long* __restrict__ offs,
                         unsigned int S, unsigned int* mm) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    unsigned int lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
    int s = -1;
    bool fin = false;
    if (i < n) {
        s = static_cast<int>(scan_of(offs, 0, S, static_cast<long long>(i)));
        const float* p = reinterpret_cast<const float*>(raw + i * stride);
        fin = finite3(p[0], p[1], p[2]);
        if (fin)
            for (int a = 0; a < 3; ++a) { lo[a] = f2ord(p[a]); hi[a] = lo[a]; }
    }
    const int s0 = __shfl_sync(0xffffffffu, s, 0);  // lane 0 holds a point whenever any lane does
    if (__all_sync(0xffffffffu, s == s0 || s < 0)) {
        for (int a = 0; a < 3; ++a) {
            const unsigned int l = __reduce_min_sync(0xffffffffu, lo[a]), h = __reduce_max_sync(0xffffffffu, hi[a]);
            if ((threadIdx.x & 31) == 0 && s0 >= 0) { atomicMin(&mm[6 * s0 + a], l); atomicMax(&mm[6 * s0 + 3 + a], h); }
        }
    } else if (fin) {
        for (int a = 0; a < 3; ++a) { atomicMin(&mm[6 * s + a], lo[a]); atomicMax(&mm[6 * s + 3 + a], hi[a]); }
    }
}
struct GridSpec {
    float inv_leaf;
    int min_b[3];
    int div_mul[3];
};
// int ijk = static_cast<int>(floor(p * inverse_leaf) - static_cast<float>(min_b))   (voxel_grid.hpp)
__device__ __forceinline__ unsigned int voxel_index(const GridSpec& g, const float* p) {
    const int i0 = static_cast<int>(floorf(__fmul_rn(p[0], g.inv_leaf)) - static_cast<float>(g.min_b[0]));
    const int i1 = static_cast<int>(floorf(__fmul_rn(p[1], g.inv_leaf)) - static_cast<float>(g.min_b[1]));
    const int i2 = static_cast<int>(floorf(__fmul_rn(p[2], g.inv_leaf)) - static_cast<float>(g.min_b[2]));
    return static_cast<unsigned int>(i0 * g.div_mul[0] + i1 * g.div_mul[1] + i2 * g.div_mul[2]);
}
enum : unsigned int { kScanNoPoint = 0, kScanOverflow = 1, kScanGrid = 2 };
// What the voxel grid does with one scan, from its bounding box (6 ordered uints as k_minmax leaves them).
// kScanGrid: *g and *cells (voxels of the index space) are set.
static unsigned int grid_spec(const unsigned int* mm6, float leaf, GridSpec* g, size_t* cells) {
    if (mm6[0] == 0xFFFFFFFFu) return kScanNoPoint;
    g->inv_leaf = 1.0f / leaf;
    long long div[3];
    for (int a = 0; a < 3; ++a) {
        const float lo = ord2f(mm6[a]), hi = ord2f(mm6[3 + a]);
        g->min_b[a] = static_cast<int>(floorf(lo * g->inv_leaf));
        div[a] = static_cast<long long>(static_cast<int>(floorf(hi * g->inv_leaf))) - g->min_b[a] + 1;
    }
    // PCL gives up when the voxel index would overflow an int ("Leaf size is too small for the input dataset. Integer
    // indices would overflow.") and returns the cloud UNFILTERED (voxel_grid.hpp: output = *input): one far outlier in a
    // key frame must not stop Lio
    if (div[0] * div[1] * div[2] > 0x7fffffffll) return kScanOverflow;
    g->div_mul[0] = 1; g->div_mul[1] = static_cast<int>(div[0]); g->div_mul[2] = static_cast<int>(div[0] * div[1]);
    *cells = static_cast<size_t>(div[0] * div[1] * div[2]);
    return kScanGrid;
}
// One scan of a voxel-grid batch.  slot: the scan's first entry in its wave's slot array - a grid scan owns
// ceil(cells / 32) bitmap words there, an overflow scan one entry that holds its point count, a scan without a finite
// point none (its slot is the next scan's).
struct ScanSpec {
    GridSpec g;
    unsigned int mode;
    unsigned int slot;
};

// Voxel grid through a BITMAP of the index space (1 bit per voxel: 256 MB at PCL's own limit of 2^31 voxels, where dense
// per-voxel arrays would take tens of GB): occupied voxels are marked, a voxel's place in the output - PCL emits the
// voxels in ascending index - is the number of set bits below it (prefix sum over the bitmap's words + popcount), and
// everything else is sized by the number of points.  The scans of a wave own consecutive word ranges of one bitmap, so
// one prefix sum over the wave ranks every voxel of every scan at once, in scan order and ascending index within a
// scan.  Kernel arguments are wave-relative: raw / point i = point p0 + i of the batch.
__global__ void k_vg_mark(const unsigned char* __restrict__ raw, size_t p0, size_t n, size_t stride, const long long* __restrict__ offs,
                          unsigned int s0, unsigned int s1, const ScanSpec* __restrict__ specs, unsigned long long* pt_bit,
                          unsigned int* bitmap) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ScanSpec& sp = specs[scan_of(offs, s0, s1, static_cast<long long>(p0 + i))];
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    if (sp.mode != kScanGrid || !finite3(p[0], p[1], p[2])) { pt_bit[i] = ~0ull; return; }
    const unsigned long long bit = 32ull * sp.slot + voxel_index(sp.g, p);
    pt_bit[i] = bit;
    atomicOr(&bitmap[bit >> 5], 1u << (bit & 31u));
}
__global__ void k_vg_popc(const unsigned int* __restrict__ bitmap, size_t words, unsigned int* wcount) {
    const size_t w = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w < words) wcount[w] = static_cast<unsigned int>(__popc(bitmap[w]));
}
// an overflow scan's slot counts its points: they go to the output as they are, in its place in scan order
__global__ void k_vg_slots(const long long* __restrict__ offs, unsigned int s0, unsigned int s1, const ScanSpec* __restrict__ specs,
                           unsigned int* wcount) {
    const unsigned int s = s0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= s1 || specs[s].mode != kScanOverflow) return;
    wcount[specs[s].slot] = static_cast<unsigned int>(offs[s + 1] - offs[s]);
}
// pt_rank[i] = the rank of the point's voxel among the wave's output slots; vcount[rank]++
__global__ void k_vg_rank(size_t n, const unsigned long long* __restrict__ pt_bit, const unsigned int* __restrict__ bitmap,
                          const unsigned int* __restrict__ wprefix, unsigned int* pt_rank, unsigned int* vcount) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long bit = pt_bit[i];
    if (bit == ~0ull) { pt_rank[i] = 0xFFFFFFFFu; return; }
    const size_t w = static_cast<size_t>(bit >> 5);
    const unsigned int r = wprefix[w] + static_cast<unsigned int>(__popc(bitmap[w] & ((1u << (bit & 31u)) - 1u)));
    pt_rank[i] = r;
    atomicAdd(&vcount[r], 1u);
}
__global__ void k_vg_scatter(size_t n, const unsigned int* __restrict__ pt_rank, const unsigned int* __restrict__ start,
                             unsigned int* cursor, unsigned int* members) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n || pt_rank[i] == 0xFFFFFFFFu) return;
    members[start[pt_rank[i]] + atomicAdd(&cursor[pt_rank[i]], 1u)] = static_cast<unsigned int>(i);
}
// one thread per occupied voxel (rank r < *n_out): float32 mean of every float word over its points in point order,
// written to output point *base + r (ranks of an overflow scan's slot have no member: k_vg_copy fills them)
__global__ void k_vg_centroid(const unsigned char* __restrict__ raw, size_t stride, const unsigned int* __restrict__ n_out,
                              const unsigned int* __restrict__ start, unsigned int* members, const unsigned int* __restrict__ base,
                              unsigned char* out) {
    const size_t r = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= *n_out) return;
    const unsigned int beg = start[r], cnt = start[r + 1] - beg;
    if (cnt == 0) return;
    unsigned int* idx = members + beg;
    for (unsigned int a = 1; a < cnt; ++a) {  // point-index order: the atomics above arrive in any order
        const unsigned int v = idx[a];
        unsigned int b = a;
        while (b > 0 && idx[b - 1] > v) { idx[b] = idx[b - 1]; --b; }
        idx[b] = v;
    }
    const size_t words = stride / 4 < 8 ? stride / 4 : 8;
    float sum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (unsigned int j = 0; j < cnt; ++j) {
        const float* p = reinterpret_cast<const float*>(raw + static_cast<size_t>(idx[j]) * stride);
        for (size_t w = 0; w < words; ++w) sum[w] = __fadd_rn(sum[w], p[w]);
    }
    float* o = reinterpret_cast<float*>(out + (*base + r) * stride);
    const float fn = static_cast<float>(cnt);
    for (size_t w = 0; w < words; ++w) o[w] = __fdiv_rn(sum[w], fn);
    for (size_t w = words; w < stride / 4; ++w) o[w] = 0.0f;
}
// the points of an overflow scan, unfiltered, into the output slots its slot entry reserved
__global__ void k_vg_copy(const unsigned char* __restrict__ raw, size_t p0, size_t n, size_t stride, const long long* __restrict__ offs,
                          unsigned int s0, unsigned int s1, const ScanSpec* __restrict__ specs, const unsigned int* __restrict__ wprefix,
                          const unsigned int* __restrict__ base, unsigned char* out) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long p = static_cast<long long>(p0 + i);
    const unsigned int s = scan_of(offs, s0, s1, p);
    if (specs[s].mode != kScanOverflow) return;
    const unsigned int* src = reinterpret_cast<const unsigned int*>(raw + i * stride);
    unsigned int* d = reinterpret_cast<unsigned int*>(out + (*base + wprefix[specs[s].slot] + static_cast<size_t>(p - offs[s])) * stride);
    for (size_t w = 0; w < stride / 4; ++w) d[w] = src[w];
}
// out_off[s] for the wave's scans s0 .. s1 (inclusive: the wave's end), and base[1] = where the next wave starts
__global__ void k_vg_offsets(unsigned int s0, unsigned int s1, const ScanSpec* __restrict__ specs, size_t slots,
                             const unsigned int* __restrict__ wprefix, unsigned int* base, unsigned int* out_off) {
    const unsigned int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > s1 - s0) return;
    const unsigned int o = base[0] + wprefix[t < s1 - s0 ? specs[s0 + t].slot : slots];
    out_off[s0 + t] = o;
    if (t == s1 - s0) base[1] = o;
}

namespace {
struct Tmp {  // stream-ordered scratch
    cudaStream_t s;
    std::vector<void*> ptrs;
    explicit Tmp(cudaStream_t st) : s(st) {}
    template <class T> T* get(size_t count) {
        void* p = nullptr;
        LR_CUDA(cudaMallocAsync(&p, std::max<size_t>(count, 1) * sizeof(T), s));
        ptrs.push_back(p);
        return static_cast<T*>(p);
    }
    ~Tmp() { for (void* p : ptrs) cudaFreeAsync(p, s); }
};
unsigned int blocks(size_t n) { return static_cast<unsigned int>((n + 255) / 256); }
// device copy of the batch's offsets (offs[0] == 0)
long long* upload_offsets(const long long* offs, size_t S, cudaStream_t stream, Tmp& tmp) {
    long long* d = tmp.get<long long>(S + 1);
    LR_CUDA(cudaMemcpyAsync(d, offs, (S + 1) * sizeof(long long), cudaMemcpyHostToDevice, stream));
    return d;
}
// flags (n) -> order-kept compaction into d_out, per-scan output offsets to the host
void run_keep(const unsigned char* d_raw, size_t n, size_t stride, const long long* d_offs, size_t S, unsigned int* flag,
              unsigned char* d_out, long long* out_offs, cudaStream_t stream, Tmp& tmp) {
    unsigned int* pos = tmp.get<unsigned int>(n);
    unsigned int* total = tmp.get<unsigned int>(1);
    unsigned int* d_out_off = tmp.get<unsigned int>(S + 1);
    exclusive_scan_u32(flag, pos, n, total, stream);
    LR_LAUNCH(k_compact, blocks(n), 256, 0, stream, d_raw, n, stride, flag, pos, d_out);
    LR_LAUNCH(k_keep_offsets, blocks(S + 1), 256, 0, stream, d_offs, static_cast<unsigned int>(S), n, pos, total, d_out_off);
    std::vector<unsigned int> h(S + 1);
    LR_CUDA(cudaMemcpyAsync(h.data(), d_out_off, (S + 1) * sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
    LR_CUDA(cudaStreamSynchronize(stream));
    for (size_t s = 0; s <= S; ++s) out_offs[s] = h[s];
}
// LOCREG_FILTER_WAVE_MIB: bitmap memory of one voxel-grid wave in MiB (default: 1 GiB, or a quarter of the free
// device memory when that is less).  Consecutive scans share a wave until their bitmaps would exceed it; a scan whose
// own bitmap is larger runs alone.  The cut never changes a result.
size_t wave_words(size_t total_words) {
    static const double env_mib = getenv("LOCREG_FILTER_WAVE_MIB") ? std::min(4096.0, std::max(1e-3, atof(getenv("LOCREG_FILTER_WAVE_MIB")))) : 0.0;
    if (env_mib > 0.0) return std::max<size_t>(1, static_cast<size_t>(env_mib * (1 << 20) / 4));
    size_t words = (size_t{1} << 30) / 4;
    if (total_words > words / 4) {  // only a batch that might not fit asks the driver
        size_t free_b = 0, total_b = 0;
        LR_CUDA(cudaMemGetInfo(&free_b, &total_b));
        words = std::min(words, std::max<size_t>(1, free_b / 4 / 8));  // bitmap + prefix: 8 B per word
    }
    return words;
}
}  // namespace

void filter_remove_nan_batch(const unsigned char* d_raw, const long long* offs, size_t S, size_t stride, unsigned char* d_out,
                             long long* out_offs, cudaStream_t stream) {
    const size_t n = static_cast<size_t>(offs[S]);
    if (n == 0) { std::fill(out_offs, out_offs + S + 1, 0ll); return; }
    Tmp tmp(stream);
    const long long* d_offs = upload_offsets(offs, S, stream, tmp);
    unsigned int* flag = tmp.get<unsigned int>(n);
    LR_LAUNCH(k_flag_finite, blocks(n), 256, 0, stream, d_raw, n, stride, flag);
    run_keep(d_raw, n, stride, d_offs, S, flag, d_out, out_offs, stream, tmp);
}
size_t filter_remove_nan(const unsigned char* d_raw, size_t n, size_t stride, unsigned char* d_out, cudaStream_t stream) {
    const long long offs[2] = {0, static_cast<long long>(n)};
    long long out[2];
    filter_remove_nan_batch(d_raw, offs, 1, stride, d_out, out, stream);
    return static_cast<size_t>(out[1]);
}
size_t filter_crop_box(const unsigned char* d_raw, size_t n, size_t stride, const float* min3, const float* max3, unsigned char* d_out,
                       cudaStream_t stream) {
    if (n == 0) return 0;
    Tmp tmp(stream);
    const long long offs[2] = {0, static_cast<long long>(n)};
    long long out[2];
    const long long* d_offs = upload_offsets(offs, 1, stream, tmp);
    unsigned int* flag = tmp.get<unsigned int>(n);
    LR_LAUNCH(k_flag_box, blocks(n), 256, 0, stream, d_raw, n, stride,
              make_float3(min3[0], min3[1], min3[2]), make_float3(max3[0], max3[1], max3[2]), flag);
    run_keep(d_raw, n, stride, d_offs, 1, flag, d_out, out, stream, tmp);
    return static_cast<size_t>(out[1]);
}

// Two synchronisations per call: after the bounding boxes (the grids are sized on the host) and at the end.
void filter_voxel_grid_batch(const unsigned char* d_raw, const long long* offs, size_t S, size_t stride, float leaf,
                             unsigned char* d_out, long long* out_offs, cudaStream_t stream) {
    const size_t n = static_cast<size_t>(offs[S]);
    if (n == 0) { std::fill(out_offs, out_offs + S + 1, 0ll); return; }
    Tmp tmp(stream);
    const unsigned int Su = static_cast<unsigned int>(S);
    // offsets and the bounding boxes' initial values in one copy
    std::vector<unsigned char> head((S + 1) * sizeof(long long) + 6 * S * sizeof(unsigned int));
    std::memcpy(head.data(), offs, (S + 1) * sizeof(long long));
    std::vector<unsigned int> mm(6 * S);
    for (size_t s = 0; s < S; ++s)
        for (int a = 0; a < 3; ++a) { mm[6 * s + a] = 0xFFFFFFFFu; mm[6 * s + 3 + a] = 0u; }
    std::memcpy(head.data() + (S + 1) * sizeof(long long), mm.data(), 6 * S * sizeof(unsigned int));
    unsigned char* d_head = tmp.get<unsigned char>(head.size());
    LR_CUDA(cudaMemcpyAsync(d_head, head.data(), head.size(), cudaMemcpyHostToDevice, stream));
    const long long* d_offs = reinterpret_cast<const long long*>(d_head);
    unsigned int* d_mm = reinterpret_cast<unsigned int*>(d_head + (S + 1) * sizeof(long long));
    LR_LAUNCH(k_minmax, blocks(n), 256, 0, stream, d_raw, n, stride, d_offs, Su, d_mm);
    LR_CUDA(cudaMemcpyAsync(mm.data(), d_mm, 6 * S * sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
    LR_CUDA(cudaStreamSynchronize(stream));

    // per-scan grids, slots, and the waves
    struct Wave { unsigned int s0, s1; size_t slots; bool overflow; };
    std::vector<ScanSpec> specs(S);
    std::vector<size_t> slots_of(S);
    size_t total_slots = 0;
    for (size_t s = 0; s < S; ++s) {
        size_t cells = 0;
        specs[s] = ScanSpec{};
        specs[s].mode = grid_spec(&mm[6 * s], leaf, &specs[s].g, &cells);
        slots_of[s] = specs[s].mode == kScanGrid ? (cells + 31) / 32 : specs[s].mode == kScanOverflow ? 1 : 0;
        total_slots += slots_of[s];
    }
    if (total_slots == 0) { std::fill(out_offs, out_offs + S + 1, 0ll); return; }  // no finite point anywhere
    const size_t budget = wave_words(total_slots);
    std::vector<Wave> waves;
    Wave cur{0, 0, 0, false};
    for (size_t s = 0; s < S; ++s) {
        if (slots_of[s] > 0 && cur.slots > 0 && cur.slots + slots_of[s] > budget) {  // every wave has points and slots
            cur.s1 = static_cast<unsigned int>(s);
            waves.push_back(cur);
            cur = Wave{static_cast<unsigned int>(s), 0, 0, false};
        }
        specs[s].slot = static_cast<unsigned int>(cur.slots);
        cur.slots += slots_of[s];
        cur.overflow |= specs[s].mode == kScanOverflow;
    }
    cur.s1 = Su;
    waves.push_back(cur);
    size_t max_pts = 0, max_slots = 0;
    for (const Wave& w : waves) {
        max_pts = std::max(max_pts, static_cast<size_t>(offs[w.s1] - offs[w.s0]));
        max_slots = std::max(max_slots, w.slots);
    }
    // the scan table and the output base of every wave (base[0] = 0) in one copy
    std::vector<unsigned char> table(S * sizeof(ScanSpec) + (waves.size() + 1) * sizeof(unsigned int), 0);
    std::memcpy(table.data(), specs.data(), S * sizeof(ScanSpec));
    unsigned char* d_table = tmp.get<unsigned char>(table.size());
    LR_CUDA(cudaMemcpyAsync(d_table, table.data(), table.size(), cudaMemcpyHostToDevice, stream));
    const ScanSpec* d_specs = reinterpret_cast<const ScanSpec*>(d_table);
    unsigned int* d_base = reinterpret_cast<unsigned int*>(d_table + S * sizeof(ScanSpec));

    unsigned long long* pt_bit = tmp.get<unsigned long long>(max_pts);
    unsigned int* pt_rank = tmp.get<unsigned int>(max_pts);
    unsigned int* bitmap = tmp.get<unsigned int>(max_slots + 1);
    unsigned int* wprefix = tmp.get<unsigned int>(max_slots + 1);
    unsigned int* vstart = tmp.get<unsigned int>(max_pts + 1);  // output slots of a wave <= its points
    unsigned int* cursor = tmp.get<unsigned int>(max_pts);
    unsigned int* members = tmp.get<unsigned int>(max_pts);
    unsigned int* total = tmp.get<unsigned int>(1);
    unsigned int* d_out_off = tmp.get<unsigned int>(S + 1);
    for (size_t wi = 0; wi < waves.size(); ++wi) {
        const Wave& w = waves[wi];
        const size_t p0 = static_cast<size_t>(offs[w.s0]), np = static_cast<size_t>(offs[w.s1]) - p0;
        const unsigned char* raw = d_raw + p0 * stride;
        unsigned int* base = d_base + wi;
        LR_CUDA(cudaMemsetAsync(bitmap, 0, (w.slots + 1) * sizeof(unsigned int), stream));
        LR_CUDA(cudaMemsetAsync(vstart, 0, (np + 1) * sizeof(unsigned int), stream));
        LR_CUDA(cudaMemsetAsync(cursor, 0, np * sizeof(unsigned int), stream));
        LR_LAUNCH(k_vg_mark, blocks(np), 256, 0, stream, raw, p0, np, stride, d_offs, w.s0, w.s1, d_specs, pt_bit, bitmap);
        LR_LAUNCH(k_vg_popc, blocks(w.slots + 1), 256, 0, stream, bitmap, w.slots + 1, wprefix);
        if (w.overflow) LR_LAUNCH(k_vg_slots, blocks(w.s1 - w.s0), 256, 0, stream, d_offs, w.s0, w.s1, d_specs, wprefix);
        exclusive_scan_u32(wprefix, wprefix, w.slots + 1, total, stream);
        LR_LAUNCH(k_vg_rank, blocks(np), 256, 0, stream, np, pt_bit, bitmap, wprefix, pt_rank, vstart);
        exclusive_scan_u32(vstart, vstart, np + 1, nullptr, stream);
        LR_LAUNCH(k_vg_scatter, blocks(np), 256, 0, stream, np, pt_rank, vstart, cursor, members);
        LR_LAUNCH(k_vg_centroid, blocks(np), 256, 0, stream, raw, stride, total, vstart, members, base, d_out);
        if (w.overflow) LR_LAUNCH(k_vg_copy, blocks(np), 256, 0, stream, raw, p0, np, stride, d_offs, w.s0, w.s1, d_specs, wprefix, base, d_out);
        LR_LAUNCH(k_vg_offsets, blocks(w.s1 - w.s0 + 1), 256, 0, stream, w.s0, w.s1, d_specs, w.slots, wprefix, base, d_out_off);
    }
    std::vector<unsigned int> h(S + 1);
    LR_CUDA(cudaMemcpyAsync(h.data(), d_out_off, (S + 1) * sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
    LR_CUDA(cudaStreamSynchronize(stream));
    for (size_t s = 0; s <= S; ++s) out_offs[s] = h[s];
}
size_t filter_voxel_grid(const unsigned char* d_raw, size_t n, size_t stride, float leaf, unsigned char* d_out, cudaStream_t stream) {
    const long long offs[2] = {0, static_cast<long long>(n)};
    long long out[2];
    filter_voxel_grid_batch(d_raw, offs, 1, stride, leaf, d_out, out, stream);
    return static_cast<size_t>(out[1]);
}

}  // namespace locreg
