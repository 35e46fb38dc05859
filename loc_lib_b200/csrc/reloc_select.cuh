// Staged relocalisation (locreg_relocalise_staged[_sharded]): the cut between two rounds, the caller-order outputs, and
// the deal and exchange of a round across ranks.
// A round's m hypotheses sit at positions 0 .. m-1 in ascending original index.  Position p's key is
// locreg_pack_score(score[p], p), so unsigned key order is (float32 score, original index) order, and the keys are
// distinct.  The k survivors are the keys <= the k-th smallest key, which an MSB-first radix select finds 8 bits per
// pass (k_select_hist, then k_select_digit fixes the digit and the rank left inside it); k_reloc_compact then packs
// the survivors in position order (flags + exclusive_scan_u32 + scatter), so the next round is in ascending original
// index again.
#pragma once
#include "device_utils.cuh"

namespace locreg {

// the radix select's running result: the digits fixed so far (higher bits of the k-th key) and its 1-based rank
// among the keys that share them
struct SelectState {
    unsigned long long prefix;
    unsigned int rank;
    unsigned int pad;
};
constexpr int kSelectBins = 256;

// keys[p] = locreg_pack_score(scores[p], p): NaN and negative scores rank as +inf
__global__ void k_reloc_keys(const double* __restrict__ scores, unsigned int m, unsigned long long* keys) {
    const unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    float f = static_cast<float>(scores[p]);
    if (!(f == f) || f < 0.0f) f = INFINITY;
    keys[p] = (static_cast<unsigned long long>(__float_as_uint(f)) << 32) | p;
}

// digit d (bits 56 - 8d .. 63 - 8d) of the keys whose higher digits equal st->prefix, counted into hist[256]
// (zero on entry): one shared-memory histogram per block, added to hist once per bin
__global__ void k_select_hist(const unsigned long long* __restrict__ keys, unsigned int m, const SelectState* __restrict__ st,
                              int digit, unsigned int* hist) {
    __shared__ unsigned int sh[kSelectBins];
    for (int b = threadIdx.x; b < kSelectBins; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    const int shift = 56 - 8 * digit;
    const unsigned long long mask = digit == 0 ? 0ull : ~0ull << (shift + 8);
    const unsigned long long prefix = digit == 0 ? 0ull : st->prefix;
    for (unsigned int p = blockIdx.x * blockDim.x + threadIdx.x; p < m; p += gridDim.x * blockDim.x) {
        const unsigned long long key = keys[p];
        if ((key & mask) == prefix) atomicAdd(&sh[(key >> shift) & 0xFF], 1u);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kSelectBins; b += blockDim.x)
        if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// One block of kSelectBins threads: the bin of digit d that holds the rank-th key (rank = k at d = 0) becomes that
// digit of st->prefix, and rank drops by the keys in the bins below.  hist is left zeroed for the next pass.
__global__ void k_select_digit(SelectState* st, unsigned int* hist, int digit, unsigned int k) {
    __shared__ unsigned int incl[kSelectBins];
    const unsigned int b = threadIdx.x;
    const unsigned int c = hist[b];
    const unsigned int rank = digit == 0 ? k : st->rank;
    const unsigned long long prefix = digit == 0 ? 0ull : st->prefix;
    hist[b] = 0;
    incl[b] = c;
    __syncthreads();
    for (unsigned int off = 1; off < kSelectBins; off <<= 1) {
        const unsigned int v = b >= off ? incl[b - off] : 0u;
        __syncthreads();
        incl[b] += v;
        __syncthreads();
    }
    const unsigned int hi = incl[b], lo = hi - c;
    if (lo < rank && rank <= hi) {  // exactly one bin: rank <= the keys counted, which are >= k >= 1
        st->prefix = prefix | (static_cast<unsigned long long>(b) << (56 - 8 * digit));
        st->rank = rank - lo;
    }
}

// flag[p] = 1 for the survivors (key <= the k-th key)
__global__ void k_select_flags(const unsigned long long* __restrict__ keys, unsigned int m, const SelectState* __restrict__ st,
                               unsigned int* flags) {
    const unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) flags[p] = keys[p] <= st->prefix ? 1u : 0u;
}

// survivor p -> slot[p] (exclusive scan of the flags): its pose into poses_next and its original index (idx_in[p];
// idx_in == nullptr: p, the first round) into idx_next
__global__ void k_reloc_compact(const unsigned long long* __restrict__ keys, unsigned int m, const SelectState* __restrict__ st,
                                const unsigned int* __restrict__ slot, const double* __restrict__ poses,
                                const unsigned int* __restrict__ idx_in, double* poses_next, unsigned int* idx_next) {
    const unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m || keys[p] > st->prefix) return;
    const unsigned int j = slot[p];
    for (int i = 0; i < 7; ++i) poses_next[static_cast<size_t>(j) * 7 + i] = poses[static_cast<size_t>(p) * 7 + i];
    idx_next[j] = idx_in ? idx_in[p] : p;
}

// a round's poses / scores / round number (1-based) -> the caller-order arrays at the original indices
__global__ void k_reloc_scatter(unsigned int m, const unsigned int* __restrict__ idx, const double* __restrict__ poses,
                                const double* __restrict__ scores, int round, double* all_poses, double* all_scores, int* all_rounds) {
    const unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const size_t o = idx ? idx[p] : p;
    for (int i = 0; i < 7; ++i) all_poses[o * 7 + i] = poses[static_cast<size_t>(p) * 7 + i];
    all_scores[o] = scores[p];
    all_rounds[o] = round + 1;
}

// the last round's smallest key (the select with k = 1) -> out[0..6] pose, out[7] score, *out_idx original index
__global__ void k_reloc_best(const SelectState* __restrict__ st, const unsigned int* __restrict__ idx,
                             const double* __restrict__ all_poses, const double* __restrict__ all_scores, double* out,
                             long long* out_idx) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned int p = static_cast<unsigned int>(st->prefix & 0xFFFFFFFFull);
    const size_t o = idx ? idx[p] : p;
    for (int i = 0; i < 7; ++i) out[i] = all_poses[o * 7 + i];
    out[7] = all_scores[o];
    *out_idx = static_cast<long long>(o);
}

// ---- locreg_relocalise_staged_sharded: a round over `world` ranks ----------------------------------------------------
// Rank q runs the round's positions q, q + world, q + 2 world, ... (m_q of them); its results travel as records of
// 8 doubles (7 pose + score) in slab q of c = ceil(m / world) records, one ncclAllGather fills all world slabs on every
// rank, and slab q record i is position q + i * world again.  Every rank then holds the whole round, as one GPU would.

// One thread per double in all three (consecutive threads touch consecutive words): launch over m_q * 7, m_q * 8 and
// m * 8 threads.

// rank's share of the round's full pose array -> out (m_q poses)
__global__ void k_reloc_deal(const double* __restrict__ poses, unsigned int m_q, unsigned int rank, unsigned int world,
                             double* out) {
    const size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= static_cast<size_t>(m_q) * 7) return;
    const size_t i = t / 7, k = t % 7;
    out[t] = poses[(rank + i * world) * 7 + k];
}

// the rank's m_q poses + scores -> its slab of records
__global__ void k_reloc_pack(const double* __restrict__ poses, const double* __restrict__ scores, unsigned int m_q,
                             double* slab) {
    const size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= static_cast<size_t>(m_q) * 8) return;
    const size_t i = t / 8, k = t % 8;
    slab[t] = k < 7 ? poses[i * 7 + k] : scores[i];
}

// the gathered slabs (world * c records) -> the round's poses and scores at positions 0 .. m-1
__global__ void k_reloc_unpack(const double* __restrict__ gather, unsigned int m, unsigned int c, unsigned int world,
                               double* poses, double* scores) {
    const size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= static_cast<size_t>(m) * 8) return;
    const size_t p = t / 8, k = t % 8;
    const double v = gather[((p % world) * c + p / world) * 8 + k];
    if (k < 7) poses[p * 7 + k] = v;
    else scores[p] = v;
}

}  // namespace locreg
