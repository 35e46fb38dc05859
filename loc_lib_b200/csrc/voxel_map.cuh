// GPU voxel-hash map for exact k-NN (kernels K1/K2 of SURVEY.md §2.3).
//
// Replaces the reference's pointer kd-tree (KdTree::BuildTree / GetClosestPoint, kdtree.cpp:10-31,
// 147-236) with a structure that suits a B200: all map points live in ONE float4 array sorted by
// voxel (w carries the caller's original index), grouped into 4x4x4-cell blocks.  A block is one
// 32-byte open-addressing hash slot {key, 64-bit cell-occupancy mask, first cell id}, so a query
// touches one 32 B sector per block, skips empty cells with bit tricks instead of probes, and reads
// candidate points as contiguous 16 B vectors.  On top of that every cell whose 3x3x3 neighbourhood holds a
// point owns a NEIGHBOURHOOD LIST: all points of those 27 cells copied contiguously (each map point is stored
// 27 times).  The common query is then ONE 16 B probe of a cell-keyed table plus ONE contiguous float4 scan
// (~25 candidates) with no per-cell work and little divergence; the block structure remains the exact fallback
// for queries whose k-th neighbour lies beyond the guaranteed radius (far-off points of the first iteration).
// Layout in HBM (1 M-point map, cell 0.5 m; sized for 180 GB, not for the L2):
//   slots       32 B x capacity (power of two, load <= 0.5)      ~ 2 MB     block table (fallback search)
//   cell_start  4 B x (occupied cells + 1)                        ~ 1.6 MB
//   pts         16 B x N                                           16 MB     sorted by cell; positions [0, N)
//   nbr_slots   16 B x capacity                                   ~ 64 MB    cell -> (start, count) of its list
//   lists       16 B x 27 N                                        432 MB    positions [N, 28 N) of the same array
//
// NN contract (SURVEY.md §8 Q1/Q2): the k nearest points in float32
//   dis2 = dx*dx + (dy*dy + dz*dz)   (Eigen 3.3 association, no FMA; kdtree.h:94)
// under the total order (dis2, original index) ascending, over the de-duplicated point set
// (quirk Q3: of exactly coincident points only the lowest index survives, kdtree.cpp:76-81).
// The search visits cells in Chebyshev shells around the query's cell and stops once the k-th best
// dis2 is strictly below a conservative lower bound of dis2 for every unvisited point, so the
// result is exact, not approximate (see DESIGN.md "Termination proof").
#pragma once
#include "common.cuh"

// test-only instrumentation of the search stages (tests/hostsim built with -DLR_STATS); nothing in the product build
#if defined(LR_STATS) && !defined(__CUDA_ARCH__)
extern unsigned long long g_knn_stats[16];
#define LR_STAT(i, v) (g_knn_stats[i] += (v))
#else
#define LR_STAT(i, v) ((void)0)
#endif

#ifndef LR_BLOCK_PRUNE
#define LR_BLOCK_PRUNE 1
#endif

namespace locreg {

struct __attribute__((aligned(32))) VoxelSlot {
    unsigned long long key;   // packed block coordinate, kEmptyKey if unused
    unsigned long long mask;  // bit (z&3)<<4 | (y&3)<<2 | (x&3) set iff that cell holds points
    unsigned int cell_base;   // id of the block's first occupied cell in cell_start[]
    unsigned int pad0, pad1, pad2;
};
static_assert(sizeof(VoxelSlot) == 32, "slot must be one 32 B sector");

constexpr unsigned long long kEmptyKey = ~0ull;
constexpr int kCoordBias = 1 << 20;        // block coords are biased into 21 bits
constexpr float kCellClamp = 1048000.0f;   // |fine cell index| clamp (fits 21 bits, exact in float)
constexpr int kBruteForceShell = 24;       // beyond this Chebyshev radius fall back to a linear scan

struct __attribute__((aligned(16))) NbrSlot {
    unsigned long long key;  // packed fine-cell coordinate, kEmptyKey if unused
    unsigned int start;      // first entry of the cell's neighbourhood list, as a position in pts[]
    unsigned int count;
};
static_assert(sizeof(NbrSlot) == 16, "neighbourhood slot must be 16 B");

struct VoxelMapView {
    const VoxelSlot* slots;
    const unsigned int* cell_start;
    const float4* pts;        // [0, n_pts): points sorted by cell; [n_pts, ...): neighbourhood lists
    const float4* canon;      // array that canonical positions index (= pts on level 0, level 0's pts on a coarse level)
    int w_is_pos;             // 0: pts[i].w = original index, position = i (level 0); 1: pts[i].w = canonical position
    const NbrSlot* nbr_slots; // nullptr: no neighbourhood lists (fallback search only)
    unsigned int nbr_mask;
    unsigned int slot_mask;  // capacity - 1
    unsigned int n_pts;      // points stored (non-finite inputs are dropped)
    unsigned int n_unique;   // points that survive de-duplication (= KdTree::size())
    float inv_cell;
    float cell;
    int cmin[3], cmax[3];    // inclusive bounds of occupied fine-cell coordinates
};

LR_HD unsigned long long pack_block(int bx, int by, int bz) {
    return (static_cast<unsigned long long>(static_cast<unsigned int>(bx + kCoordBias)) << 42) |
           (static_cast<unsigned long long>(static_cast<unsigned int>(by + kCoordBias)) << 21) |
           static_cast<unsigned long long>(static_cast<unsigned int>(bz + kCoordBias));
}
LR_HD unsigned long long pack_cell(int cx, int cy, int cz) {  // |c| <= kCellClamp < 2^20
    return (static_cast<unsigned long long>(static_cast<unsigned int>(cx + kCoordBias)) << 42) |
           (static_cast<unsigned long long>(static_cast<unsigned int>(cy + kCoordBias)) << 21) |
           static_cast<unsigned long long>(static_cast<unsigned int>(cz + kCoordBias));
}
LR_HD unsigned int hash_block(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return static_cast<unsigned int>(k);
}
// cell coordinate of a float coordinate; monotone non-decreasing in x (needed by the bound proof)
LR_HD float cell_coord_f(float x, float inv_cell) {
    float u = LR_FMUL(x, inv_cell);
    u = fminf(fmaxf(u, -kCellClamp), kCellClamp);
    return u;
}
LR_HD int cell_of(float u) { return static_cast<int>(floorf(u)); }

LR_HD const VoxelSlot* find_block(const VoxelMapView& m, int bx, int by, int bz) {
    const unsigned long long key = pack_block(bx, by, bz);
    unsigned int h = hash_block(key) & m.slot_mask;
    while (true) {
        const VoxelSlot* s = m.slots + h;
        const unsigned long long k = s->key;
        if (k == key) return s;
        if (k == kEmptyKey) return nullptr;
        h = (h + 1) & m.slot_mask;
    }
}

// 4-bit per-axis masks -> 64-bit cell masks (bit = z<<4 | y<<2 | x)
LR_HD unsigned long long spread_x(unsigned int mx) { return 0x1111111111111111ull * mx; }
LR_HD unsigned long long spread_y(unsigned int my) {
    const unsigned int t = ((my & 1u) * 0xFu) | ((my & 2u) * (0xF0u >> 1)) | ((my & 4u) * (0xF00u >> 2)) |
                           ((my & 8u) * (0xF000u >> 3));
    return 0x0001000100010001ull * t;
}
LR_HD unsigned long long spread_z(unsigned int mz) {
    return ((mz & 1u) ? 0x000000000000FFFFull : 0ull) | ((mz & 2u) ? 0x00000000FFFF0000ull : 0ull) |
           ((mz & 4u) ? 0x0000FFFF00000000ull : 0ull) | ((mz & 8u) ? 0xFFFF000000000000ull : 0ull);
}
// bits of a block (origin o = 4*b) whose cell coordinate lies in [lo, hi]
LR_HD unsigned int axis_range_mask(int o, int lo, int hi) {
    int a = lo - o, b = hi - o;
    a = a < 0 ? 0 : a;
    b = b > 3 ? 3 : b;
    if (a > b) return 0u;
    return ((1u << (b + 1)) - 1u) & ~((1u << a) - 1u);
}
// bits of a block whose cell coordinate equals lo or hi
LR_HD unsigned int axis_edge_mask(int o, int lo, int hi) {
    unsigned int m = 0;
    if (lo - o >= 0 && lo - o <= 3) m |= 1u << (lo - o);
    if (hi - o >= 0 && hi - o <= 3) m |= 1u << (hi - o);
    return m;
}

constexpr unsigned int kNoPos = 0xFFFFFFFFu;  // empty result slot / "no neighbour"

// Running k-best set of one query, sorted ascending by (dis2, original index).  Only the position of a point in
// the cell-sorted array pts[0, n_pts) is kept: its original index sits in pts[pos].w and is fetched on the rare
// exact distance ties only, which keeps the state at 2K registers and the insertion at ~5 instructions per slot.
template <int K>
struct KnnResult {
    float d2[K];
    unsigned int pos[K];  // canonical position in pts[0, n_pts), kNoPos = empty
};

template <int K>
LR_HD void knn_init(KnnResult<K>& r) {
#pragma unroll
    for (int j = 0; j < K; ++j) { r.d2[j] = INFINITY; r.pos[j] = kNoPos; }
}
template <int K>
LR_HD int knn_count(const KnnResult<K>& r) {
    int c = 0;
#pragma unroll
    for (int j = 0; j < K; ++j) c += (r.pos[j] != kNoPos) ? 1 : 0;
    return c;
}
// original (caller's) index of the point at canonical position pos; an empty slot sorts after every point
LR_HD int knn_index_of(const float4* pts, unsigned int pos) {
    return pos == kNoPos ? 0x7fffffff : float_as_int(pts[pos].w);
}
// strict total order (dis2, original index)
LR_HD bool knn_less(const float4* pts, float d2a, unsigned int pa, float d2b, unsigned int pb) {
    if (d2a < d2b) return true;
    if (d2a == d2b) return knn_index_of(pts, pa) < knn_index_of(pts, pb);
    return false;
}
// Does candidate (d2, pos) belong into the set?  Not if it is no better than the current k-th, and not if it is
// already a member (seeds from the previous Gauss-Newton iteration are met again in the lists; a point can also
// sit in several lists).  NaN distances (masked duplicates, quirk Q3) are rejected by the first comparison.
template <int K>
LR_HD bool knn_accepts(const float4* pts, const KnnResult<K>& r, float d2, unsigned int pos) {
    if (!(d2 <= r.d2[K - 1])) return false;
    bool member = false;
#pragma unroll
    for (int j = 0; j < K; ++j) member = member || (r.pos[j] == pos);
    if (member) return false;
    if (d2 == r.d2[K - 1]) return knn_index_of(pts, pos) < knn_index_of(pts, r.pos[K - 1]);
    return true;
}
// Sorted insertion of an accepted candidate (precondition: it precedes r[K-1]); straight-line selects.  Exact distance
// ties between distinct points are rare, so the comparisons are made on dis2 alone: where the candidate's dis2 differs
// from a slot's, `d2 < r.d2[j]` IS the (dis2, original index) order.  Only a candidate whose dis2 equals that of one of
// the slots it is compared with looks the indices up, and only for those slots.
template <int K>
LR_HD void knn_insert(const float4* pts, KnnResult<K>& r, float d2, unsigned int pos) {
    unsigned int before = 0u;  // bit j: the candidate precedes slot j
    bool tie = false;
#pragma unroll
    for (int j = 0; j + 1 < K; ++j) {
        before |= (d2 < r.d2[j] ? 1u : 0u) << j;
        tie = tie || d2 == r.d2[j];
    }
    if (tie) {
#pragma unroll
        for (int j = 0; j + 1 < K; ++j)
            if (d2 == r.d2[j] && knn_index_of(pts, pos) < knn_index_of(pts, r.pos[j])) before |= 1u << j;
    }
    bool before_old = true;  // candidate precedes the element that sat in slot j before this insertion
#pragma unroll
    for (int j = K - 1; j >= 1; --j) {
        const bool before_prev = (before >> (j - 1)) & 1u;
        const float nd = before_prev ? r.d2[j - 1] : (before_old ? d2 : r.d2[j]);
        const unsigned int np = before_prev ? r.pos[j - 1] : (before_old ? pos : r.pos[j]);
        r.d2[j] = nd;
        r.pos[j] = np;
        before_old = before_prev;
    }
    if (before_old) { r.d2[0] = d2; r.pos[0] = pos; }
}
template <int K>
LR_HD void knn_offer(const float4* pts, KnnResult<K>& r, float d2, unsigned int pos) {
    if (knn_accepts(pts, r, d2, pos)) knn_insert(pts, r, d2, pos);
}

// knn_offer that also keeps d6 = the smallest dis2 of any candidate that is NOT in the set afterwards (rejected, or
// evicted by this insertion): the search's lower bound for "the best point outside the result" (knn_track_margin).
template <int K>
LR_HD void knn_offer_track(const float4* pts, KnnResult<K>& r, float d2, unsigned int pos, float& d6) {
    if (!(d2 <= r.d2[K - 1])) { d6 = fminf(d6, d2); return; }  // fminf drops the NaN of a masked duplicate
    bool member = false;
#pragma unroll
    for (int j = 0; j < K; ++j) member = member || (r.pos[j] == pos);
    if (member) return;
    if (d2 == r.d2[K - 1] && !(knn_index_of(pts, pos) < knn_index_of(pts, r.pos[K - 1]))) { d6 = fminf(d6, d2); return; }
    d6 = fminf(d6, r.d2[K - 1]);  // the evicted k-th (INFINITY while the set is not full)
    knn_insert(pts, r, d2, pos);
}

LR_HD float dis2_f32(float qx, float qy, float qz, float px, float py, float pz) {
    const float dx = LR_FSUB(qx, px), dy = LR_FSUB(qy, py), dz = LR_FSUB(qz, pz);
    return LR_FADD(LR_FMUL(dx, dx), LR_FADD(LR_FMUL(dy, dy), LR_FMUL(dz, dz)));
}

// Conservative (never over-estimating) distance in metres for a gap of `g` cell units when the
// coordinates involved are about `mag` cell units from the origin: absorbs the rounding of
// x*inv_cell on both the map point and the query, and of the float dis2 itself.
LR_HD float safe_gap(float g, float mag, float cell) {
    const float e = g - 4.8e-7f * (mag + 4.0f);
    return e > 0.0f ? e * cell * 0.99999f : 0.0f;
}

// Scan of one contiguous neighbourhood list pts[beg, beg + cnt) (entries carry the canonical position in w).
// The search is latency bound (one query per thread, every candidate a dependent L1/L2 access), so the device loop
// fetches kScanBatch candidates with independent 16 B loads before it looks at any of them; a short last batch
// re-reads the list's final entry, which the membership test of knn_accepts turns into a no-op.
// two_pass (device only; same result): when the set starts empty or from poor seeds - the first Gauss-Newton
// iterations - a third of the candidates would pass the acceptance test at 32 different moments per warp and the
// (long, divergent) sorted insertion dominates.  A branch-free first pass therefore finds the K-th smallest dis2 of
// the list with a min/max network on the distances alone, and the second pass offers only the <= K (+ ties)
// candidates at or below that threshold.
constexpr int kScanBatch = 4;
// `pts` is the array the list lives in, `canon` the array canonical positions index (the same on level 0).
template <int K>
LR_HD void knn_scan_list(const float4* __restrict__ pts, const float4* __restrict__ canon, KnnResult<K>& res, float qx, float qy,
                         float qz, unsigned int beg, unsigned int cnt, bool two_pass, float* d6 = nullptr) {
    if (d6 != nullptr) {  // seeded scan that also reports the best candidate left outside the set (never with two_pass)
#if defined(__CUDA_ARCH__)
        if (cnt == 0) return;
        const unsigned int last = beg + cnt - 1;
        float best_out = *d6;
        for (unsigned int i = beg; i <= last; i += kScanBatch) {
            float4 p[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) p[u] = pts[min(i + u, last)];
            float d2[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) d2[u] = dis2_f32(qx, qy, qz, p[u].x, p[u].y, p[u].z);
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u)  // a re-read final entry is a member by then, or was counted already
                knn_offer_track(canon, res, d2[u], static_cast<unsigned int>(float_as_int(p[u].w)), best_out);
        }
        *d6 = best_out;
#else
        for (unsigned int i = beg; i < beg + cnt; ++i) {
            const float4 p = pts[i];
            knn_offer_track(canon, res, dis2_f32(qx, qy, qz, p.x, p.y, p.z), static_cast<unsigned int>(float_as_int(p.w)), *d6);
        }
#endif
        return;
    }
#if defined(__CUDA_ARCH__)
    if (cnt == 0) return;
    const unsigned int last = beg + cnt - 1;
    float thr = INFINITY;
    if (two_pass) {
        float t[K];
#pragma unroll
        for (int j = 0; j < K; ++j) t[j] = INFINITY;
        for (unsigned int i = beg; i <= last; i += kScanBatch) {
            float4 p[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) p[u] = pts[min(i + u, last)];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) {
                // a re-read final entry must not enter twice: the network counts multiplicity
                float v = (i + u <= last) ? dis2_f32(qx, qy, qz, p[u].x, p[u].y, p[u].z) : INFINITY;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const float lo = fminf(t[j], v);
                    v = fmaxf(t[j], v);
                    t[j] = lo;
                }
            }
        }
        thr = t[K - 1];
    }
    if (!two_pass) {
        // seeded scan: what passes the bound is almost always a seed met again in the list (rejected by the membership
        // test), now and then a closer point; handled in place
        for (unsigned int i = beg; i <= last; i += kScanBatch) {
            float4 p[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) p[u] = pts[min(i + u, last)];
            float d2[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) d2[u] = dis2_f32(qx, qy, qz, p[u].x, p[u].y, p[u].z);
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) knn_offer(canon, res, d2[u], static_cast<unsigned int>(float_as_int(p[u].w)));
        }
        return;
    }
    // Second pass of the unseeded scan: the <= K (+ ties) candidates at or below the threshold are only MARKED while
    // the list streams through again (branch-free: a bit per entry, 64 entries per chunk), then inserted in a loop all
    // lanes walk together - every lane has about K of them, at different places of its list.
    for (unsigned int chunk = beg; chunk <= last; chunk += 64) {
        const unsigned int cend = min(chunk + 63u, last);
        const float bound = fminf(thr, res.d2[K - 1]);
        unsigned long long marks = 0ull;
        for (unsigned int i = chunk; i <= cend; i += kScanBatch) {
            float4 p[kScanBatch];
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) p[u] = pts[min(i + u, cend)];
            unsigned int m = 0u;
#pragma unroll
            for (int u = 0; u < kScanBatch; ++u) {
                const float d2 = dis2_f32(qx, qy, qz, p[u].x, p[u].y, p[u].z);
                m |= (d2 <= bound && i + u <= cend) ? (1u << u) : 0u;
            }
            marks |= static_cast<unsigned long long>(m) << (i - chunk);
        }
        while (marks) {
            const int bit = ffs64(marks) - 1;
            marks &= marks - 1;
            const float4 p = pts[chunk + bit];
            knn_offer(canon, res, dis2_f32(qx, qy, qz, p.x, p.y, p.z), static_cast<unsigned int>(float_as_int(p.w)));
        }
    }
#else
    (void)two_pass;
    for (unsigned int i = beg; i < beg + cnt; ++i) {
        const float4 p = pts[i];
        knn_offer(canon, res, dis2_f32(qx, qy, qz, p.x, p.y, p.z), static_cast<unsigned int>(float_as_int(p.w)));
    }
#endif
}

// Geometry of a query relative to the cell grid (shared by the two stages of the search).
struct KnnCellFrame {
    int fx, fy, fz;        // the query's cell
    float frx, fry, frz;   // position inside the cell, in cell units
    float mag;             // largest |coordinate| in cell units (rounding allowance of the bounds)
    int R0;                // smallest Chebyshev radius whose box touches the occupied bounds (>= 1)
};
LR_HD KnnCellFrame knn_frame(const VoxelMapView& m, float qx, float qy, float qz) {
    KnnCellFrame c;
    const float ux = cell_coord_f(qx, m.inv_cell), uy = cell_coord_f(qy, m.inv_cell), uz = cell_coord_f(qz, m.inv_cell);
    c.fx = cell_of(ux); c.fy = cell_of(uy); c.fz = cell_of(uz);
    c.frx = ux - static_cast<float>(c.fx); c.fry = uy - static_cast<float>(c.fy); c.frz = uz - static_cast<float>(c.fz);
    c.mag = fmaxf(fmaxf(fabsf(ux), fabsf(uy)), fabsf(uz));
    const int ex = c.fx < m.cmin[0] ? m.cmin[0] - c.fx : (c.fx > m.cmax[0] ? c.fx - m.cmax[0] : 0);
    const int ey = c.fy < m.cmin[1] ? m.cmin[1] - c.fy : (c.fy > m.cmax[1] ? c.fy - m.cmax[1] : 0);
    const int ez = c.fz < m.cmin[2] ? m.cmin[2] - c.fz : (c.fz > m.cmax[2] ? c.fz - m.cmax[2] : 0);
    const int e = ex > ey ? (ex > ez ? ex : ez) : (ey > ez ? ey : ez);
    c.R0 = e > 1 ? e : 1;
    return c;
}
// true when the list scan applies to this query: lists exist and the 3x3x3 box around its cell touches the map
LR_HD bool knn_uses_list(const VoxelMapView& m, const KnnCellFrame& c) { return m.nbr_slots != nullptr && c.R0 == 1; }

// (start, count) of the neighbourhood list of cell (cx, cy, cz); count 0 if the cell has none
LR_HD void knn_find_list(const VoxelMapView& m, int cx, int cy, int cz, unsigned int& beg, unsigned int& cnt) {
    const unsigned long long key = pack_cell(cx, cy, cz);
    unsigned int h = hash_block(key) & m.nbr_mask;
    beg = 0; cnt = 0;
    while (true) {
        const NbrSlot s = m.nbr_slots[h];
        if (s.key == key) { beg = s.start; cnt = s.count; return; }
        if (s.key == kEmptyKey) return;
        h = (h + 1) & m.nbr_mask;
    }
}
// Starts the k-best set from K seed positions.  The common case - all K present, as after any complete search - loads
// the K points with independent accesses and orders them with a sorting network (9 compare-exchanges for K = 5)
// instead of K dependent insertions; seeds are distinct points, so no membership test is needed.
template <int K>
LR_HD void knn_seed(const VoxelMapView& m, float qx, float qy, float qz, const unsigned int* seeds, KnnResult<K>& res) {
    bool all = true;
#pragma unroll
    for (int j = 0; j < K; ++j) all = all && seeds[j] < m.n_pts;
    if (!all) {
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const unsigned int sp = seeds[j];
            if (sp < m.n_pts) {
                const float4 p = m.pts[sp];
                knn_offer(m.pts, res, dis2_f32(qx, qy, qz, p.x, p.y, p.z), sp);
            }
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const float4 p = m.pts[seeds[j]];
        res.d2[j] = dis2_f32(qx, qy, qz, p.x, p.y, p.z);
        res.pos[j] = seeds[j];
    }
    if (K == 5) {
        // on dis2 alone first (as knn_insert); if a comparator met two equal distances the (dis2, original index) order
        // decides: the exact network sorts any permutation of the K distinct seeds into that one order, so it runs over
        // what the first pass left
        constexpr int net[9][2] = {{0, 1}, {3, 4}, {2, 4}, {2, 3}, {1, 4}, {0, 3}, {0, 2}, {1, 3}, {1, 2}};
        bool tie = false;
#pragma unroll
        for (int c = 0; c < 9; ++c) {
            const int a = net[c][0], b = net[c][1];
            tie = tie || res.d2[b] == res.d2[a];
            const bool sw = res.d2[b] < res.d2[a];
            const float da = sw ? res.d2[b] : res.d2[a], db = sw ? res.d2[a] : res.d2[b];
            const unsigned int pa = sw ? res.pos[b] : res.pos[a], pb = sw ? res.pos[a] : res.pos[b];
            res.d2[a] = da; res.d2[b] = db; res.pos[a] = pa; res.pos[b] = pb;
        }
        if (tie) {
#pragma unroll
            for (int c = 0; c < 9; ++c) {
                const int a = net[c][0], b = net[c][1];
                if (knn_less(m.pts, res.d2[b], res.pos[b], res.d2[a], res.pos[a])) {
                    const float td = res.d2[a]; res.d2[a] = res.d2[b]; res.d2[b] = td;
                    const unsigned int tp = res.pos[a]; res.pos[a] = res.pos[b]; res.pos[b] = tp;
                }
            }
        }
    }
    // a NaN distance (a seed that is a masked duplicate cannot occur: results never contain one) would break the order;
    // K == 1 needs no ordering
}

// Do the K (distinct, real) positions of `a` and the K positions of `b` form the same SET?  What k_icp_fit derives from
// a point's neighbours - a plane through five points - does not depend on their order beyond rounding, and early
// Gauss-Newton iterations often only swap neighbours of nearly equal distance.
template <int K>
LR_HD bool knn_same_set(const unsigned int* a, const unsigned int* b) {
    bool same = true;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        bool found = false;
#pragma unroll
        for (int k = 0; k < K; ++k) found = found || a[j] == b[k];
        same = same && found && a[j] != kNoPos;
    }
    return same;
}

// After the list of the query's own cell on level `m` (the box [f-1, f+1]^3) has been scanned: is `res` final?
template <int K>
LR_HD bool knn_list_final(const VoxelMapView& m, const KnnCellFrame& c, const KnnResult<K>& res) {
    if (res.pos[K - 1] != kNoPos) {
        float mf = fminf(c.frx, 1.0f - c.frx);
        mf = fminf(mf, fminf(c.fry, 1.0f - c.fry));
        mf = fminf(mf, fminf(c.frz, 1.0f - c.frz));
        const float g = safe_gap(1.0f + mf, c.mag + 1.0f, m.cell);
        if (res.d2[K - 1] < g * g * 0.99999f) return true;
    }
    return c.fx - 1 <= m.cmin[0] && c.fx + 1 >= m.cmax[0] && c.fy - 1 <= m.cmin[1] && c.fy + 1 >= m.cmax[1] &&
           c.fz - 1 <= m.cmin[2] && c.fz + 1 >= m.cmax[2];
}

// Stage 1 of the exact k-NN of a FINITE query against a NON-EMPTY map: seeds, then the one-list fast path.
//   seeds    optional K canonical positions (kNoPos = none) that start the k-best set - the neighbours found in the
//            previous Gauss-Newton iteration.  Any real, distinct points are valid seeds: they only tighten the
//            acceptance threshold early; the result is still the exact k-NN.
// Returns true when `res` is final; false when the k-th neighbour may lie outside the visited box and stage 2
// (knn_query_rings, seeded with `res`) has to continue.
template <int K>
LR_HD bool knn_query_fast(const VoxelMapView& m, float qx, float qy, float qz, KnnResult<K>& res,
                          const unsigned int* seeds, bool two_pass) {
    knn_init(res);
    const KnnCellFrame c = knn_frame(m, qx, qy, qz);
    if (seeds != nullptr) knn_seed<K>(m, qx, qy, qz, seeds, res);
    if (!knn_uses_list(m, c)) return false;
    // the whole box [f-1, f+1]^3 is one contiguous list
    unsigned int beg = 0, cnt = 0;
    knn_find_list(m, c.fx, c.fy, c.fz, beg, cnt);
    LR_STAT(0, 1); LR_STAT(1, cnt);  // fast-path queries, candidates
    knn_scan_list<K>(m.pts, m.pts, res, qx, qy, qz, beg, cnt, two_pass);  // stage 1 runs on level 0: canon == pts
    return knn_list_final<K>(m, c, res);
}

// ---- skipping the list scan when the query has hardly moved --------------------------------------------------------
// A full stage-1 search at q0 knows more than the K neighbours: every other point is at least r6 away, r6 = the best
// candidate it rejected inside the box, or the distance to the faces of the box for the points outside.  When the query
// of the next Gauss-Newton iteration has moved by delta, every member is at most r5 + delta away and every non-member
// at least r6 - delta: while 2 delta < r6 - r5 (less the rounding of the float distances) the K nearest points are the
// SAME SET, and recomputing and sorting their K distances (knn_seed) reproduces the exact search bit for bit - order
// and ties included - without touching the list.  Late iterations move a query by a millimetre; r6 - r5 is
// centimetres.
struct __attribute__((aligned(16))) KnnTrack {
    float qx, qy, qz;  // the query of the last full search
    float margin;      // how far the query may move from there, metres; <= 0: always search
};
template <int K>
LR_HD float knn_track_margin(const VoxelMapView& m, const KnnCellFrame& c, const KnnResult<K>& res, float d6, float qx, float qy,
                             float qz) {
    if (res.pos[K - 1] == kNoPos) return -1.0f;
    float mf = fminf(c.frx, 1.0f - c.frx);
    mf = fminf(mf, fminf(c.fry, 1.0f - c.fry));
    mf = fminf(mf, fminf(c.frz, 1.0f - c.frz));
    const float g = safe_gap(1.0f + mf, c.mag + 1.0f, m.cell);  // points outside the scanned box
    const float r6 = fminf(sqrtf(d6) * 0.99999f, g);
    const float r5 = sqrtf(res.d2[K - 1]) * 1.00001f;
    // float coordinates this far from the origin carry half an ulp each, in the stored and in the moved query
    const float mag = fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
    return 0.5f * (r6 - r5) - (4e-7f * mag + 1e-6f);
}
LR_HD bool knn_track_holds(const KnnTrack& t, float qx, float qy, float qz) {
    if (!(t.margin > 0.0f)) return false;
    const float dx = qx - t.qx, dy = qy - t.qy, dz = qz - t.qz;
    return sqrtf(dx * dx + dy * dy + dz * dz) * 1.00001f < t.margin;  // NaN anywhere: false
}
// Stage 1 with the bookkeeping above: `track` receives the query and its margin (-1 when the result is not final).
template <int K>
LR_HD bool knn_query_fast_track(const VoxelMapView& m, float qx, float qy, float qz, KnnResult<K>& res, const unsigned int* seeds,
                                KnnTrack& track) {
    knn_init(res);
    track.qx = qx; track.qy = qy; track.qz = qz; track.margin = -1.0f;
    const KnnCellFrame c = knn_frame(m, qx, qy, qz);
    knn_seed<K>(m, qx, qy, qz, seeds, res);
    if (!knn_uses_list(m, c)) return false;
    unsigned int beg = 0, cnt = 0;
    knn_find_list(m, c.fx, c.fy, c.fz, beg, cnt);
    LR_STAT(0, 1); LR_STAT(1, cnt);  // fast-path queries, candidates
    float d6 = INFINITY;
    knn_scan_list<K>(m.pts, m.pts, res, qx, qy, qz, beg, cnt, false, &d6);
    const bool done = knn_list_final<K>(m, c, res);
    // (a query whose box covers the whole map is final too, with the box faces still the bound for "outside": fine)
    if (done) track.margin = knn_track_margin<K>(m, c, res, d6, qx, qy, qz);
    return done;
}
// The cheap attempt: K gathers and a sort.  True: `res` is the exact result for (qx, qy, qz).
template <int K>
LR_HD bool knn_track_try(const VoxelMapView& m, float qx, float qy, float qz, const unsigned int* seeds, const KnnTrack& track,
                         KnnResult<K>& res) {
    if (!knn_track_holds(track, qx, qy, qz)) return false;
    knn_init(res);
    knn_seed<K>(m, qx, qy, qz, seeds, res);
    LR_STAT(9, 1);  // searches skipped
    return res.pos[K - 1] != kNoPos;
}

// Stage 2a: the 5x5x5 box through neighbourhood lists.  The list of the cell f + (sx, sy, sz), s = +-1, covers the
// cells f + [s-1, s+1] per axis, so the eight "corner" lists together cover [f-2, f+2]^3.  Only the cells the ball of
// the current k-th distance touches matter (every other unvisited point is farther than that distance and cannot
// belong to the result), and they are found face by face: where the ball crosses an outer face of the visited
// 3x3x3 box, its cap has radius rho = sqrt(w^2 - depth^2) and reaches the cell offsets floor(fr -+ rho) on the two
// other axes, which fixes the corner signs that are needed there - typically one or two lists instead of a walk
// over up to 98 shell cells.  All quantities are in cell units and inflated by the rounding allowance of the cell
// assignment.  Needs a full set (a finite k-th distance) from stage 1.
// Returns true when `res` is final, false when shells R >= 3 must follow (knn_query_rings with boxes_done = 2).
// Which of the eight corner lists the ball of squared radius worst_d2 needs: bit (sx > 0) | (sy > 0) << 1 | (sz > 0) << 2
LR_HD unsigned int knn_corner_mask(const VoxelMapView& m, const KnnCellFrame& c, float worst_d2) {
    const float slack = 1e-6f * (c.mag + 4.0f);
    const float wc = sqrtf(worst_d2) * m.inv_cell * 1.0001f + slack;  // k-th distance, cell units, rounded up
    const float fr[3] = {c.frx, c.fry, c.frz};
    unsigned int need = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int b1 = (a + 1) % 3, b2 = (a + 2) % 3;
#pragma unroll
        for (int dir = 0; dir < 2; ++dir) {
            const float depth = dir ? 2.0f - fr[a] : 1.0f + fr[a];  // to the outer face of the visited box
            if (wc < depth - slack) continue;
            const float rho = sqrtf(fmaxf(wc * wc - depth * depth, 0.0f)) + 2.0f * slack + 1e-5f;
            bool p1 = floorf(fr[b1] + rho) >= 1.0f, m1 = floorf(fr[b1] - rho) <= -1.0f;
            bool p2 = floorf(fr[b2] + rho) >= 1.0f, m2 = floorf(fr[b2] - rho) <= -1.0f;
            if (!p1 && !m1) m1 = true;
            if (!p2 && !m2) m2 = true;
#pragma unroll
            for (int s1 = 0; s1 < 2; ++s1) {
                if (!(s1 ? p1 : m1)) continue;
#pragma unroll
                for (int s2 = 0; s2 < 2; ++s2) {
                    if (!(s2 ? p2 : m2)) continue;
                    need |= 1u << ((dir << a) | (s1 << b1) | (s2 << b2));
                }
            }
        }
    }
    return need;
}
// After stage 2a: every unvisited point is outside [f-2, f+2]^3 or farther than the k-th distance the mask used
template <int K>
LR_HD bool knn_corners_final(const VoxelMapView& m, const KnnCellFrame& c, const KnnResult<K>& res) {
    float mf = fminf(c.frx, 1.0f - c.frx);
    mf = fminf(mf, fminf(c.fry, 1.0f - c.fry));
    mf = fminf(mf, fminf(c.frz, 1.0f - c.frz));
    const float g = safe_gap(2.0f + mf, c.mag + 2.0f, m.cell);
    if (res.d2[K - 1] < g * g * 0.99999f) return true;
    return c.fx - 2 <= m.cmin[0] && c.fx + 2 >= m.cmax[0] && c.fy - 2 <= m.cmin[1] && c.fy + 2 >= m.cmax[1] &&
           c.fz - 2 <= m.cmin[2] && c.fz + 2 >= m.cmax[2];
}
template <int K>
LR_HD bool knn_query_corners(const VoxelMapView& m, float qx, float qy, float qz, KnnResult<K>& res) {
    const KnnCellFrame c = knn_frame(m, qx, qy, qz);
    LR_STAT(2, 1);  // queries entering stage 2a
    const unsigned int need = knn_corner_mask(m, c, res.d2[K - 1]);
    for (int o = 0; o < 8; ++o) {
        if (!((need >> o) & 1u)) continue;
        unsigned int beg = 0, cnt = 0;
        knn_find_list(m, c.fx + ((o & 1) ? 1 : -1), c.fy + ((o & 2) ? 1 : -1), c.fz + ((o & 4) ? 1 : -1), beg, cnt);
        LR_STAT(3, 1); LR_STAT(4, cnt);  // corner lists scanned, candidates
        knn_scan_list<K>(m.pts, m.canon, res, qx, qy, qz, beg, cnt, false);
    }
    return knn_corners_final<K>(m, c, res);
}

// Geometry of one Chebyshev shell (radius R around the query's cell) clipped to the occupied bounds.
struct KnnShell {
    int lox, hix, loy, hiy, loz, hiz;  // the box [f - R, f + R]
    int clx, chx, cly, chy, clz, chz;  // clipped to the occupied bounds
    int nbx, nby, nbz;                 // blocks spanned by the clipped box per axis (0: the box misses the bounds)
    int R;
    bool first;                        // nothing inside the box has been visited: take the full box, not just the shell
};
LR_HD KnnShell knn_shell(const VoxelMapView& m, const KnnCellFrame& c, int R, bool first) {
    KnnShell s;
    s.R = R; s.first = first;
    s.lox = c.fx - R; s.hix = c.fx + R; s.loy = c.fy - R; s.hiy = c.fy + R; s.loz = c.fz - R; s.hiz = c.fz + R;
    s.clx = s.lox > m.cmin[0] ? s.lox : m.cmin[0]; s.chx = s.hix < m.cmax[0] ? s.hix : m.cmax[0];
    s.cly = s.loy > m.cmin[1] ? s.loy : m.cmin[1]; s.chy = s.hiy < m.cmax[1] ? s.hiy : m.cmax[1];
    s.clz = s.loz > m.cmin[2] ? s.loz : m.cmin[2]; s.chz = s.hiz < m.cmax[2] ? s.hiz : m.cmax[2];
    s.nbx = s.chx >= s.clx ? (s.chx >> 2) - (s.clx >> 2) + 1 : 0;
    s.nby = s.chy >= s.cly ? (s.chy >> 2) - (s.cly >> 2) + 1 : 0;
    s.nbz = s.chz >= s.clz ? (s.chz >> 2) - (s.clz >> 2) + 1 : 0;
    return s;
}
// Conservative (never over-estimated) squared distance from the query to cell (cx, cy, cz)
LR_HD float knn_cell_min_d2(const VoxelMapView& m, const KnnCellFrame& c, int cx, int cy, int cz, float magR) {
    const float gx = cx > c.fx ? static_cast<float>(cx - c.fx) - c.frx : (cx < c.fx ? static_cast<float>(c.fx - cx - 1) + c.frx : 0.0f);
    const float gy = cy > c.fy ? static_cast<float>(cy - c.fy) - c.fry : (cy < c.fy ? static_cast<float>(c.fy - cy - 1) + c.fry : 0.0f);
    const float gz = cz > c.fz ? static_cast<float>(cz - c.fz) - c.frz : (cz < c.fz ? static_cast<float>(c.fz - cz - 1) + c.frz : 0.0f);
    const float sx = safe_gap(gx, magR, m.cell), sy = safe_gap(gy, magR, m.cell), sz = safe_gap(gz, magR, m.cell);
    return (sx * sx + sy * sy + sz * sz) * 0.99999f;
}
// Occupied cells of block (bx, by, bz) that belong to the shell (bit = z << 4 | y << 2 | x), with the block's
// occupancy mask and first cell id; 0 if the block is interior, absent or empty there.
LR_HD unsigned long long knn_shell_block_cells(const VoxelMapView& m, const KnnShell& sh, int bx, int by, int bz,
                                               unsigned long long& occ, unsigned int& base) {
    const int ox = bx << 2, oy = by << 2, oz = bz << 2;
    const unsigned int rx = axis_range_mask(ox, sh.clx, sh.chx), ry = axis_range_mask(oy, sh.cly, sh.chy),
                       rz = axis_range_mask(oz, sh.clz, sh.chz);
    const unsigned int ix = sh.first ? 0u : (rx & ~axis_edge_mask(ox, sh.lox, sh.hix));
    const unsigned int iy = sh.first ? 0u : (ry & ~axis_edge_mask(oy, sh.loy, sh.hiy));
    const unsigned int iz = sh.first ? 0u : (rz & ~axis_edge_mask(oz, sh.loz, sh.hiz));
    // cells of this block inside the box but not strictly interior (= the new shell)
    if (!sh.first && ix == rx && iy == ry && iz == rz) return 0ull;  // block entirely interior
    LR_STAT(6, 1);  // block probes
    const VoxelSlot* s = find_block(m, bx, by, bz);
    if (s == nullptr) return 0ull;
    unsigned long long want = spread_x(rx) & spread_y(ry) & spread_z(rz);
    if (!sh.first) want &= ~(spread_x(ix) & spread_y(iy) & spread_z(iz));
    occ = s->mask;
    base = s->cell_base;
    return occ & want;
}
// Cells of block (bx, by, bz) that belong to the shell: their points are offered to `res`.  bound (<= INFINITY) is an
// additional acceptance / pruning bound on dis2 that does not come from `res` itself (the warp-cooperative search
// passes the replicated global k-th distance while `res` is a lane's private set).
// Conservative squared distance from the query to the 4x4x4 cells of block (bx, by, bz) (as knn_cell_min_d2)
LR_HD float knn_block_min_d2(const VoxelMapView& m, const KnnCellFrame& c, int bx, int by, int bz, float magR) {
    const int ox = bx << 2, oy = by << 2, oz = bz << 2;
    const float gx = ox > c.fx ? static_cast<float>(ox - c.fx) - c.frx : (ox + 3 < c.fx ? static_cast<float>(c.fx - ox - 4) + c.frx : 0.0f);
    const float gy = oy > c.fy ? static_cast<float>(oy - c.fy) - c.fry : (oy + 3 < c.fy ? static_cast<float>(c.fy - oy - 4) + c.fry : 0.0f);
    const float gz = oz > c.fz ? static_cast<float>(oz - c.fz) - c.frz : (oz + 3 < c.fz ? static_cast<float>(c.fz - oz - 4) + c.frz : 0.0f);
    const float sx = safe_gap(gx, magR, m.cell), sy = safe_gap(gy, magR, m.cell), sz = safe_gap(gz, magR, m.cell);
    return (sx * sx + sy * sy + sz * sz) * 0.99999f;
}
template <int K>
LR_HD void knn_shell_block(const VoxelMapView& m, const KnnCellFrame& c, const KnnShell& sh, int bx, int by, int bz,
                           float qx, float qy, float qz, float bound, KnnResult<K>& res) {
    unsigned long long occ = 0ull;
    unsigned int base = 0;
#if LR_BLOCK_PRUNE
    {   // a block the ball of the current K-th distance cannot reach is not even looked up
        const float worst0 = fminf(bound, res.d2[K - 1]);
        if (worst0 < INFINITY && knn_block_min_d2(m, c, bx, by, bz, c.mag + static_cast<float>(sh.R)) > worst0) { LR_STAT(15, 1); return; }
    }
#endif
    unsigned long long todo = knn_shell_block_cells(m, sh, bx, by, bz, occ, base);
    const int ox = bx << 2, oy = by << 2, oz = bz << 2;
    const float magR = c.mag + static_cast<float>(sh.R);
    while (todo) {
        const int bit = ffs64(todo) - 1;
        todo &= todo - 1;
        const float worst = fminf(bound, res.d2[K - 1]);
        if (worst < INFINITY && knn_cell_min_d2(m, c, ox + (bit & 3), oy + ((bit >> 2) & 3), oz + (bit >> 4), magR) > worst) continue;
        const unsigned int cid = base + popc64(occ & ((1ull << bit) - 1ull));
        const unsigned int beg = m.cell_start[cid], end = m.cell_start[cid + 1];
        LR_STAT(7, end - beg);  // shell candidates
        // (kScanBatch independent loads in flight, as in the list scans, measured SLOWER here: relocalisation stage 2
        // 18.3 -> 25.8 ms, a batch's 0.27 -> 0.31 ms - 36 more spilled bytes at 64 registers)
        for (unsigned int i = beg; i < end; ++i) {
            const float4 p = m.pts[i];
            const float d2 = dis2_f32(qx, qy, qz, p.x, p.y, p.z);
            if (d2 <= bound) knn_offer(m.canon, res, d2, m.w_is_pos ? static_cast<unsigned int>(float_as_int(p.w)) : i);
        }
    }
}
// After the box [f - R, f + R]^3 has been dealt with: is `res` final?  Every unvisited point lies outside the box,
// at least R + min(frac, 1 - frac) cell units away along some axis - or the box covers the whole map.
template <int K>
LR_HD bool knn_shell_final(const VoxelMapView& m, const KnnCellFrame& c, const KnnShell& sh, const KnnResult<K>& res) {
    if (res.pos[K - 1] != kNoPos) {
        float mf = fminf(c.frx, 1.0f - c.frx);
        mf = fminf(mf, fminf(c.fry, 1.0f - c.fry));
        mf = fminf(mf, fminf(c.frz, 1.0f - c.frz));
        const float g = safe_gap(static_cast<float>(sh.R) + mf, c.mag + static_cast<float>(sh.R), m.cell);
        if (res.d2[K - 1] < g * g * 0.99999f) return true;
    }
    return sh.lox <= m.cmin[0] && sh.hix >= m.cmax[0] && sh.loy <= m.cmin[1] && sh.hiy >= m.cmax[1] &&
           sh.loz <= m.cmin[2] && sh.hiz >= m.cmax[2];
}

// Stage 2b: Chebyshev shells of cells through the block table of ONE resolution level until the k-th best is
// provably final (returns true) or the shell radius exceeds max_R (returns false: the caller escalates to a coarser
// level).  `res` holds what the earlier stages found (it may be partly or wholly empty); boxes_done = Chebyshev
// radius of the box of THIS level they have dealt with (0: nothing, 1: stage 1's list, 2: stage 2a).
template <int K>
LR_HD bool knn_query_rings(const VoxelMapView& m, float qx, float qy, float qz, KnnResult<K>& res, int boxes_done, int max_R) {
    const KnnCellFrame c = knn_frame(m, qx, qy, qz);
    LR_STAT(5, 1);  // queries entering stage 2b
    bool first = boxes_done == 0;  // nothing visited yet: the first shell is the full box
    for (int R = first ? c.R0 : boxes_done + 1;; ++R) {
        if (R > max_R) return false;
        const KnnShell sh = knn_shell(m, c, R, first);
        for (int jz = 0; jz < sh.nbz; ++jz)
            for (int jy = 0; jy < sh.nby; ++jy)
                for (int jx = 0; jx < sh.nbx; ++jx)
                    knn_shell_block<K>(m, c, sh, (sh.clx >> 2) + jx, (sh.cly >> 2) + jy, (sh.clz >> 2) + jz, qx, qy, qz, INFINITY, res);
        first = false;
        if (knn_shell_final<K>(m, c, sh, res)) return true;
    }
}

// Everything after stage 1 for one query (the body of k_icp_nn_rings).  Escalation: corner lists (5x5x5 fine
// cells), fine shells up to kFineShells, then the COARSE level (cells kCoarseFactor times larger, same points, no
// lists) from scratch - its shells reach kBruteForceShell * kCoarseFactor fine cells, which is what keeps far-off
// queries (global relocalisation hypotheses, points outside the map) from degenerating into a linear scan - and
// only beyond that the linear scan.  Restarting on another level is sound because the set only ever holds real,
// distinct points: what a level re-visits is rejected by the membership / threshold tests.
constexpr int kFineShells = 4;
constexpr int kCoarseFactor = 4;   // cell edge ratio between consecutive levels
constexpr int kCoarseLevels = 2;   // 4x and 16x the fine cell: shells reach 24 * 16 fine cells (192 m at 0.5 m)
#ifndef LR_COARSE_SHELLS
#define LR_COARSE_SHELLS 8  // measured 3..12: 8 (relocalisation stage 2 -10 % against 6, 3 is +65 %)
#endif
constexpr int kCoarseShells = LR_COARSE_SHELLS;   // shells on a level that has a coarser one behind it
#ifndef LR_MID_FACTOR
#define LR_MID_FACTOR 2.0f
#endif
constexpr float kMidFactor = LR_MID_FACTOR;  // the mid level's cell edge / the fine level's
#ifndef LR_MID_SHELLS
#define LR_MID_SHELLS 4  // measured 1..8: 4 (batch stage 2 -25 % against 2; relocalisation indifferent)
#endif
constexpr int kMidShells = LR_MID_SHELLS;  // shells on the mid level when a coarse level can take over
// ---- the block pyramid: a 64-ary tree over the fine level's blocks --------------------------------------------------------
// Level l of the pyramid holds one 16 B record {key, 64-bit child mask} per node of 4^(l+1) fine blocks per axis
// (coordinates = block coordinates >> 2(l+1), pure integer arithmetic on the fine grid, so the levels nest for every
// cell size); a child of a level-0 node is a fine block of m.slots, a child of a block a cell.  It turns stage 2 of the
// search into a depth-first BALL QUERY: from the top, only children whose box can hold a point at or below the current
// K-th distance are opened, nearest child first, so a far-off query (a wrong relocalisation hypothesis: its points hang
// metres away from every surface) costs a dozen 16-32 B records and the points of the few fine cells its ball touches,
// where Chebyshev shells had to look at every cell of a (2R + 1)^2 patch of the nearest surface before they could prune.
struct __attribute__((aligned(16))) PyrSlot {
    unsigned long long key;   // pack_block(node coordinate), kEmptyKey if unused
    unsigned long long mask;  // bit (z&3)<<4 | (y&3)<<2 | (x&3) set iff that child exists
};
constexpr int kPyrMaxLevels = 8;   // 4^(8+1) blocks per axis at the top: more than the 21-bit coordinates can hold
struct PyrView {
    const PyrSlot* slots[kPyrMaxLevels];
    unsigned int mask[kPyrMaxLevels];  // capacity - 1 per level
    int levels;                        // 0: no pyramid; the top level spans the occupied bounds with <= 2 nodes per axis
};
struct CoarseLevels {
    VoxelMapView lv[kCoarseLevels];  // n_pts == 0: level absent
    VoxelMapView mid;                // cells kMidFactor times the fine ones WITH neighbourhood lists; n_pts == 0: absent
    PyrView pyr;                     // block pyramid over the FINE level (levels == 0: absent)
    int pyr_mode;                    // 0: shells only; 1: pyramid after the mid level's list; 2: pyramid instead of the mid level
    int mid_shells_p1;               // 1 + shells on the mid level before a coarse level takes over; 0: kMidShells (batches)
    int coarse_shells_p1;            // 1 + shells on a coarse level that has a coarser one behind it; 0: kCoarseShells
};
LR_HD const PyrSlot* find_pyr(const PyrView& py, int l, int nx, int ny, int nz) {
    const unsigned long long key = pack_block(nx, ny, nz);
    unsigned int h = hash_block(key) & py.mask[l];
    while (true) {
        const PyrSlot* s = py.slots[l] + h;
        const unsigned long long k = s->key;
        if (k == key) return s;
        if (k == kEmptyKey) return nullptr;
        h = (h + 1) & py.mask[l];
    }
}
// bit i of the result = bit (i ^ a) of m: children in the order of i ^ a start with child a
LR_HD unsigned long long xor_permute64(unsigned long long m, unsigned int a) {
    if (a & 1u) m = ((m & 0x5555555555555555ull) << 1) | ((m >> 1) & 0x5555555555555555ull);
    if (a & 2u) m = ((m & 0x3333333333333333ull) << 2) | ((m >> 2) & 0x3333333333333333ull);
    if (a & 4u) m = ((m & 0x0F0F0F0F0F0F0F0Full) << 4) | ((m >> 4) & 0x0F0F0F0F0F0F0F0Full);
    if (a & 8u) m = ((m & 0x00FF00FF00FF00FFull) << 8) | ((m >> 8) & 0x00FF00FF00FF00FFull);
    if (a & 16u) m = ((m & 0x0000FFFF0000FFFFull) << 16) | ((m >> 16) & 0x0000FFFF0000FFFFull);
    if (a & 32u) m = (m << 32) | (m >> 32);
    return m;
}
// children (4 per axis, each 2^shift cells wide) of the node at coordinate n whose cells meet [lo, hi]; 4-bit mask
LR_HD unsigned int axis_child_mask(int n, int shift, int lo, int hi) {
    const int o = n << 2;
    int a = (lo >> shift) - o, b = (hi >> shift) - o;
    a = a < 0 ? 0 : a;
    b = b > 3 ? 3 : b;
    if (a > b) return 0u;
    return ((1u << (b + 1)) - 1u) & ~((1u << a) - 1u);
}
// index (0..3) of the child of node n nearest to cell f along one axis
LR_HD unsigned int axis_near_child(int n, int shift, int f) {
    const int a = (f >> shift) - (n << 2);
    return static_cast<unsigned int>(a < 0 ? 0 : (a > 3 ? 3 : a));
}
// The ball query as a STATE MACHINE: one call of step() looks at one point, opens one child or pops one node, so that
// a kernel can run 32 walks in the lanes of a warp, every lane in the same loop whatever the depth of its walk, and
// hand a lane the next query the moment its walk ends (k_icp_nn_pyr) - the shells' 9 active lanes of 32 came from
// queries of very different length sharing a warp from start to end.
// Soundness: a subtree is skipped only when the conservative distance to its box exceeds the current K-th distance, or
// when it lies outside the cell range that the points at or below that distance can occupy given the box's gaps along
// the other two axes; every point of an opened cell at or below the K-th distance is offered; candidates already in
// the set are rejected by the membership test, ties are decided by the original index as everywhere else.  The set
// may start from any real, distinct points (seeds) or empty.
// todo[] (children still to visit per depth, XOR-permuted: nearest child first) is the caller's array: the one
// dynamically indexed piece of state stays in local memory on its own and everything in the struct in registers.
constexpr int kPyrStack = kPyrMaxLevels + 1;
constexpr int kPyrDone = 0, kPyrNode = 1, kPyrPoint = 2, kPyrPush = 3;
template <int K>
struct PyrWalk {
    KnnResult<K> res;
    float qx, qy, qz;        // the query
    float ux, uy, uz;        // ... in cell units
    int fx, fy, fz;          // its cell
    float eps;               // rounding allowance of a gap, in cell units (safe_gap)
    unsigned long long near_pack;                // 6 bits per depth: the XOR order's first child
    unsigned long long occ;                      // occupancy of the fine block on top of the stack
    unsigned int base;                           // its first cell id
    unsigned int pi, pend;                       // points of the opened cell still to look at
    int nx, ny, nz;                              // coordinate of the node on top of the stack
    int d;                                       // its depth (level P - 1 - d; P: a fine block); -1: at the root
    unsigned int root_todo, root_near;           // the <= 2x2x2 top nodes, same ordering trick
    int rlx, rhx, rly, rhy, rlz, rhz;            // cells a point at or below the K-th distance can lie in (reach box)

    // conservative (never over-estimated) gaps in metres between the query and the box of 2^shift cells per axis at
    // coordinate (cx, cy, cz) (in units of 2^shift cells)
    LR_HD void box_gaps(const VoxelMapView& m, int cx, int cy, int cz, int shift, float& sx, float& sy, float& sz) const {
        const float wdt = static_cast<float>(1 << shift), cs = m.cell * 0.99999f;
        const float lx = static_cast<float>(cx << shift), ly = static_cast<float>(cy << shift), lz = static_cast<float>(cz << shift);
        sx = fmaxf(fmaxf(lx - ux, ux - (lx + wdt)) - eps, 0.0f) * cs;
        sy = fmaxf(fmaxf(ly - uy, uy - (ly + wdt)) - eps, 0.0f) * cs;
        sz = fmaxf(fmaxf(lz - uz, uz - (lz + wdt)) - eps, 0.0f) * cs;
    }
    // The reach box: the cells per axis that a point at or below the current K-th distance can lie in.  Kept in
    // registers and refreshed whenever the K-th distance changes (an insertion into a full set), so that opening a
    // node costs three range masks and no square root.
    LR_HD void refresh_reach(const VoxelMapView& m) {
        const float worst = res.d2[K - 1];
        if (!(worst < INFINITY)) {
            rlx = rly = rlz = -0x40000000; rhx = rhy = rhz = 0x40000000;
            return;
        }
        const float dc = fminf(sqrtf(worst * 1.000001f) * m.inv_cell * 1.0001f + 4.0f * eps + 1e-3f, 4.0e6f);
        rlx = static_cast<int>(floorf(ux - dc)); rhx = static_cast<int>(floorf(ux + dc));
        rly = static_cast<int>(floorf(uy - dc)); rhy = static_cast<int>(floorf(uy + dc));
        rlz = static_cast<int>(floorf(uz - dc)); rhz = static_cast<int>(floorf(uz + dc));
    }
    LR_HD void start(const VoxelMapView& m, const PyrView& py, float x, float y, float z) {
        qx = x; qy = y; qz = z;
        ux = cell_coord_f(x, m.inv_cell); uy = cell_coord_f(y, m.inv_cell); uz = cell_coord_f(z, m.inv_cell);
        fx = cell_of(ux); fy = cell_of(uy); fz = cell_of(uz);
        float mag = fmaxf(fmaxf(fabsf(ux), fabsf(uy)), fabsf(uz));
#pragma unroll
        for (int a = 0; a < 3; ++a)
            mag = fmaxf(mag, fmaxf(fabsf(static_cast<float>(m.cmin[a])), fabsf(static_cast<float>(m.cmax[a]))));
        eps = 4.8e-7f * (mag + 8.0f);
        pi = pend = 0u;
        d = -1;
        near_pack = 0ull;
        occ = 0ull; base = 0u;
        nx = ny = nz = 0;
        const int ts = 2 * py.levels + 2;
        const int t0x = m.cmin[0] >> ts, t0y = m.cmin[1] >> ts, t0z = m.cmin[2] >> ts;
        const int wx = (m.cmax[0] >> ts) - t0x, wy = (m.cmax[1] >> ts) - t0y, wz = (m.cmax[2] >> ts) - t0z;  // 0 or 1
        root_todo = 1u | (wx ? 2u : 0u);
        root_todo |= wy ? root_todo << 2 : 0u;
        root_todo |= wz ? root_todo << 4 : 0u;
        const int ax = (fx >> ts) - t0x, ay = (fy >> ts) - t0y, az = (fz >> ts) - t0z;
        root_near = (ax > 0 && wx ? 1u : 0u) | (ay > 0 && wy ? 2u : 0u) | (az > 0 && wz ? 4u : 0u);
        root_todo = static_cast<unsigned int>(xor_permute64(root_todo, root_near));
        refresh_reach(m);
        LR_STAT(10, 1);  // pyramid queries
    }
    // pushes node (cx, cy, cz) at depth nd with child mask cm
    LR_HD void push(const VoxelMapView& m, const PyrView& py, unsigned long long* todo, int nd, int cx, int cy, int cz, unsigned long long cm) {
        const int gs = 2 * (py.levels - nd);  // cells per child of the new node = 2^gs
        unsigned int na = 0u;
        if (res.d2[K - 1] < INFINITY) {  // children outside the reach box are dropped at once; the order hardly matters any more
            cm &= spread_x(axis_child_mask(cx, gs, rlx, rhx)) & spread_y(axis_child_mask(cy, gs, rly, rhy)) & spread_z(axis_child_mask(cz, gs, rlz, rhz));
            if (cm == 0ull) return;
        } else {  // nothing to prune with yet: nearest child first
            na = axis_near_child(cx, gs, fx) | (axis_near_child(cy, gs, fy) << 2) | (axis_near_child(cz, gs, fz) << 4);
            cm = xor_permute64(cm, na);
        }
        d = nd;
        nx = cx; ny = cy; nz = cz;
        near_pack = (near_pack << 6) | na;
        todo[nd] = cm;
    }
    // The walk is cut into three kinds of step so that a warp can run ONE kind at a time for all the lanes that are
    // due for it (k_icp_nn_pyr): node_step (take the next child of the node on top of the stack and test its box, or
    // pop), push_step (open the interior child that passed: hash probe, reach masks, ordering - the long one) and
    // point_step (one point of the opened cell).  Each returns the kind of step the walk needs next.
    // node_step: kPyrNode again, kPyrPoint (a cell was opened), kPyrPush (child `bit` passed and waits to be opened:
    // a top node when d < 0), or kPyrDone (res is final).
    LR_HD int node_step(const VoxelMapView& m, const PyrView& py, unsigned long long* todo, int& bit_out) {
        const int P = py.levels;
        if (d < 0) {  // the next top node
            if (root_todo == 0u) return kPyrDone;
            const unsigned int i = static_cast<unsigned int>(ffs64(root_todo) - 1) ^ root_near;
            root_todo &= root_todo - 1u;
            const int ts = 2 * P + 2;
            float sx, sy, sz;
            box_gaps(m, (m.cmin[0] >> ts) + static_cast<int>(i & 1u), (m.cmin[1] >> ts) + static_cast<int>((i >> 1) & 1u),
                     (m.cmin[2] >> ts) + static_cast<int>(i >> 2), ts, sx, sy, sz);
            LR_STAT(13, 1);  // box tests
            if ((sx * sx + sy * sy + sz * sz) * 0.99999f > res.d2[K - 1]) return kPyrNode;
            (void)bit_out;
            push_step(m, py, todo, static_cast<int>(i));
            return kPyrNode;
        }
        const unsigned long long t = todo[d];
        if (t == 0ull) {  // node exhausted
            --d;
            nx >>= 2; ny >>= 2; nz >>= 2;
            near_pack >>= 6;
            return kPyrNode;
        }
        const int bit = (ffs64(t) - 1) ^ static_cast<int>(near_pack & 63ull);
        todo[d] = t & (t - 1ull);
        const int cx = (nx << 2) + (bit & 3), cy = (ny << 2) + ((bit >> 2) & 3), cz = (nz << 2) + (bit >> 4);
        float sx, sy, sz;
        box_gaps(m, cx, cy, cz, 2 * (P - d), sx, sy, sz);
        LR_STAT(13, 1);
        if ((sx * sx + sy * sy + sz * sz) * 0.99999f > res.d2[K - 1]) return kPyrNode;
        if (d == P) {  // a cell of the fine block on top of the stack
            const unsigned int cid = base + popc64(occ & ((1ull << bit) - 1ull));
            pi = m.cell_start[cid];
            pend = m.cell_start[cid + 1];
            LR_STAT(12, pend - pi); LR_STAT(14, 1);  // candidates, cells opened
            return pi < pend ? kPyrPoint : kPyrNode;
        }
        push_step(m, py, todo, bit);
        return kPyrNode;
    }
    LR_HD void push_step(const VoxelMapView& m, const PyrView& py, unsigned long long* todo, int bit) {
        const int P = py.levels;
        LR_STAT(11, 1);  // node probes
        if (d < 0) {
            const int ts = 2 * P + 2;
            const int tx = (m.cmin[0] >> ts) + (bit & 1), ty = (m.cmin[1] >> ts) + ((bit >> 1) & 1), tz = (m.cmin[2] >> ts) + (bit >> 2);
            const PyrSlot* s = find_pyr(py, P - 1, tx, ty, tz);
            if (s != nullptr) push(m, py, todo, 0, tx, ty, tz, s->mask);
            return;
        }
        const int cx = (nx << 2) + (bit & 3), cy = (ny << 2) + ((bit >> 2) & 3), cz = (nz << 2) + (bit >> 4);
        if (d == P - 1) {  // the child is a fine block
            const VoxelSlot* s = find_block(m, cx, cy, cz);
            if (s == nullptr) return;
            const unsigned long long cm = s->mask;
            const unsigned int cb = s->cell_base;
            const int d_was = d;
            push(m, py, todo, d + 1, cx, cy, cz, cm);
            if (d != d_was) { occ = cm; base = cb; }
        } else {
            const PyrSlot* s = find_pyr(py, P - 2 - d, cx, cy, cz);
            if (s != nullptr) push(m, py, todo, d + 1, cx, cy, cz, s->mask);
        }
    }
    LR_HD int point_step(const VoxelMapView& m) {
        const float4 p = m.pts[pi];
        const float d2 = dis2_f32(qx, qy, qz, p.x, p.y, p.z);
        const unsigned int pos = m.w_is_pos ? static_cast<unsigned int>(float_as_int(p.w)) : pi;
        if (knn_accepts(m.canon, res, d2, pos)) {
            knn_insert(m.canon, res, d2, pos);
            refresh_reach(m);
        }
        ++pi;
        return pi < pend ? kPyrPoint : kPyrNode;
    }
};
template <int K>
LR_HD void knn_query_pyr(const VoxelMapView& m, const PyrView& py, float qx, float qy, float qz, KnnResult<K>& res) {
    PyrWalk<K> w;
    unsigned long long todo[kPyrStack];
    w.res = res;
    w.start(m, py, qx, qy, qz);
    int st = kPyrNode, bit = 0;
    while (st != kPyrDone) {
        if (st == kPyrNode) st = w.node_step(m, py, todo, bit);
        else if (st == kPyrPoint) st = w.point_step(m);
        else { w.push_step(m, py, todo, bit); st = kPyrNode; }
    }
    res = w.res;
}

// Stage 2 through the mid level: one list of the mid level covers a box three mid cells wide around the query - what
// the corner lists and the first fine shells would have to collect from up to eight lists and dozens of hash-probed
// blocks is one probe and one contiguous scan here.  Returns true when `res` is final; false: coarse levels next.
// margin (optional): the KnnTrack margin when the search ends with the list (which holds every point of the mid box, so
// a seeded scan knows d6 as in knn_query_fast_track), else -1.
template <int K>
LR_HD bool knn_query_mid(const VoxelMapView& md, bool have_coarse, float qx, float qy, float qz, KnnResult<K>& res,
                         float* margin = nullptr, bool list_only = false, int mid_shells = kMidShells) {
    const KnnCellFrame c = knn_frame(md, qx, qy, qz);
    int boxes_done = 0;
    if (margin) *margin = -1.0f;
    if (knn_uses_list(md, c)) {
        unsigned int beg = 0, cnt = 0;
        knn_find_list(md, c.fx, c.fy, c.fz, beg, cnt);
        LR_STAT(3, 1); LR_STAT(4, cnt);  // mid lists scanned, candidates
        if (margin && res.pos[K - 1] != kNoPos) {
            float d6 = INFINITY;
            knn_scan_list<K>(md.pts, md.canon, res, qx, qy, qz, beg, cnt, false, &d6);
            if (knn_list_final<K>(md, c, res)) {
                *margin = knn_track_margin<K>(md, c, res, d6, qx, qy, qz);
                return true;
            }
        } else {
            knn_scan_list<K>(md.pts, md.canon, res, qx, qy, qz, beg, cnt, res.pos[K - 1] == kNoPos);
            if (knn_list_final<K>(md, c, res)) return true;
        }
        boxes_done = 1;
    }
    if (list_only) return false;  // the caller continues with the block pyramid
    if (have_coarse && c.R0 > mid_shells) return false;
    return knn_query_rings<K>(md, qx, qy, qz, res, boxes_done, have_coarse ? mid_shells : kBruteForceShell);
}
template <int K>
LR_HD void knn_query_finish(const VoxelMapView& m, const CoarseLevels& coarse, float qx, float qy, float qz, KnnResult<K>& res,
                            float* margin = nullptr) {
    const bool have_coarse = coarse.lv[0].n_pts != 0;
    if (margin) *margin = -1.0f;
    // (pyr_mode is honoured on the host - tests/hostsim, which checks PyrWalk against brute force - and in device builds
    // with -DLR_FINISH_PYR; the product's thread-per-query kernels stay free of the walk's stack and registers: on the
    // device the pyramid is walked by k_icp_nn_pyr only)
#if !defined(__CUDA_ARCH__) || defined(LR_FINISH_PYR)
    const bool pyr = coarse.pyr.levels != 0 && coarse.pyr_mode != 0;
#else
    const bool pyr = false;
#endif
    if (pyr && (coarse.pyr_mode == 2 || coarse.mid.n_pts == 0)) {  // the ball query does all of stage 2
        knn_query_pyr<K>(m, coarse.pyr, qx, qy, qz, res);
        return;
    }
    if (coarse.mid.n_pts != 0) {
        LR_STAT(2, 1);  // queries entering stage 2a
        if (knn_query_mid<K>(coarse.mid, have_coarse || pyr, qx, qy, qz, res, margin, pyr, coarse.mid_shells_p1 > 0 ? coarse.mid_shells_p1 - 1 : kMidShells)) return;
        if (margin) *margin = -1.0f;
        if (pyr) {  // what the mid level's list could not settle: ball query instead of shells
            knn_query_pyr<K>(m, coarse.pyr, qx, qy, qz, res);
            return;
        }
    } else {
        const KnnCellFrame c = knn_frame(m, qx, qy, qz);
        int boxes_done = knn_uses_list(m, c) ? 1 : 0;
        if (boxes_done == 1 && res.pos[K - 1] != kNoPos) {
            if (knn_query_corners<K>(m, qx, qy, qz, res)) return;
            boxes_done = 2;
        }
        // a query outside the occupied bounds by more than the fine reach goes straight to the coarse levels
        if (!(have_coarse && c.R0 > kFineShells) &&
            knn_query_rings<K>(m, qx, qy, qz, res, boxes_done, have_coarse ? kFineShells : kBruteForceShell))
            return;
    }
    for (int l = 0; l < kCoarseLevels; ++l) {
        const VoxelMapView& cl = coarse.lv[l];
        if (cl.n_pts == 0) break;
        const bool last = l + 1 == kCoarseLevels || coarse.lv[l + 1].n_pts == 0;
        // leave a level early (6 shells) when a coarser one can take over, so that far queries climb quickly
        const int shells = coarse.coarse_shells_p1 > 0 ? coarse.coarse_shells_p1 - 1 : kCoarseShells;
        if (!last && knn_frame(cl, qx, qy, qz).R0 > shells) continue;
        if (knn_query_rings<K>(cl, qx, qy, qz, res, 0, last ? kBruteForceShell : shells)) return;
    }
    LR_STAT(8, 1);  // linear scans
    knn_init(res);
    for (unsigned int i = 0; i < m.n_pts; ++i) {
        const float4 p = m.pts[i];
        knn_offer(m.pts, res, dis2_f32(qx, qy, qz, p.x, p.y, p.z), i);
    }
}

// Exact k-NN of (qx,qy,qz) in one call (parity probe, tests/hostsim).  valid = false: no query, empty result.
template <int K>
LR_HD void knn_query(const VoxelMapView& m, const CoarseLevels& coarse, bool valid, float qx, float qy, float qz,
                     KnnResult<K>& res, const unsigned int* seeds = nullptr, bool two_pass = false) {
    if (!valid || m.n_pts == 0) { knn_init(res); return; }
    if (!knn_query_fast<K>(m, qx, qy, qz, res, seeds, two_pass)) knn_query_finish<K>(m, coarse, qx, qy, qz, res);
}

}  // namespace locreg
