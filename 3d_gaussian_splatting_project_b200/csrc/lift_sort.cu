// Sort step of the spatial ordering (lift_order.cu): (24-bit Morton cell, row index) pairs by
// cell.  The sort is a preprocessing utility, not part of the vote arithmetic, and uses CUB's
// device radix sort (three 8-bit passes) from the CUDA toolkit; its scratch comes out of the
// caller's workspace like everything else.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "lift_internal.cuh"

namespace gsl {

// Upper bound on CUB's scratch for N pairs: its alternate key and value buffers (8 bytes per
// pair) plus histograms and per-tile look-back state.  sort_cells() checks the real requirement
// against it.
size_t sort_temp_capacity(int64_t N)
{
    return (size_t)(N > 0 ? N : 0) * 9 + ((size_t)4 << 20);
}

int sort_cells(const uint32_t *keys_in, uint32_t *keys_out, const int32_t *idx_in, int32_t *idx_out,
               int64_t N, void *temp, size_t temp_bytes, cudaStream_t st)
{
    if (N > 0x7fffffffLL) return fail(GSL_EINVAL, "ordering: more than 2^31 - 1 Gaussians in one call");
    size_t need = 0;
    // The order only has to make tiles compact, it need not be total.  Up to 2 M Gaussians a 65536-cell grid
    // (the top 16 key bits, two 8-bit passes) already holds ~30 per cell, and the third pass costs more than the
    // slightly looser tiles (measured at 750 K: pass 0.576 -> 0.560 ms; at 6 M the gather loses what the sort
    // gains, so the full 24-bit order stays).
    const int low = N <= (2 << 20) ? 8 : 0;
    GSL_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, keys_in, keys_out, idx_in, idx_out, (int)N, low, 24, st));
    if (need > temp_bytes) return fail(GSL_EWORKSPACE, "ordering: sort scratch %zu > reserved %zu", need, temp_bytes);
    GSL_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, need, keys_in, keys_out, idx_in, idx_out, (int)N, low, 24, st));
    return GSL_OK;
}

}  // namespace gsl
