// Device cloud pre-filters (filters.cu): raw strided clouds in, compacted / downsampled raw clouds out (same stride).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace locreg {
// each returns the number of points written to d_out (capacity: n points)
size_t filter_remove_nan(const unsigned char* d_raw, size_t n, size_t stride, unsigned char* d_out, cudaStream_t stream);
size_t filter_crop_box(const unsigned char* d_raw, size_t n, size_t stride, const float* min3, const float* max3, unsigned char* d_out,
                       cudaStream_t stream);
size_t filter_voxel_grid(const unsigned char* d_raw, size_t n, size_t stride, float leaf, unsigned char* d_out, cudaStream_t stream);
// Batches: scan s is points [offs[s], offs[s + 1]) of d_raw (host offsets, offs[0] == 0, non-decreasing, S >= 1).
// out_offs (host, S + 1) receives the offsets of the filtered batch in d_out (capacity: offs[S] points); segment s is
// the single-cloud filter's result for scan s alone.  The single-cloud functions above are the batch of one scan.
void filter_remove_nan_batch(const unsigned char* d_raw, const long long* offs, size_t S, size_t stride, unsigned char* d_out,
                             long long* out_offs, cudaStream_t stream);
void filter_voxel_grid_batch(const unsigned char* d_raw, const long long* offs, size_t S, size_t stride, float leaf,
                             unsigned char* d_out, long long* out_offs, cudaStream_t stream);
}  // namespace locreg
