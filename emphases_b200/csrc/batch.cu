// On-device collate of a training batch from a resident corpus
// (emphases/data/collate.py:11-77 for the features and targets): item b of the
// batch is corpus item items[b]; its frame rows are copied from the packed
// frame-major rows into channel-major (B, C, Tmax) and its word targets into
// (B, 1, Wmax), zero past each item's own length.  One launch writes every
// output element, so no memset precedes it.
//
// Grid: (time tiles, channel tiles + 1, B).  A CTA of the channel tiles moves a
// 32-frame x 32-channel tile through shared memory: loads run along channels
// (one frame row = C contiguous floats), stores along time.  The extra slice
// (blockIdx.y == channel tiles) writes the targets of its item.
#include "common.cuh"

namespace emph {

constexpr int kGatherTile = 32;
constexpr int kGatherRows = 8;        // threads per tile column: 32 x 8 = 256

__global__ void __launch_bounds__(kGatherTile * kGatherRows)
gather_batch_kernel(
    const float* __restrict__ rows, int channels,
    const int32_t* __restrict__ row_start, const int32_t* __restrict__ n_rows,
    const float* __restrict__ word_targets, const int32_t* __restrict__ word_start,
    const int32_t* __restrict__ n_words, int n_items, const int32_t* __restrict__ items,
    int tmax, int wmax, float* __restrict__ features, float* __restrict__ targets) {
    const int b = blockIdx.z;
    // an index outside the corpus yields an all-zero item (the host validates
    // indices; this keeps a bad one from reading out of bounds)
    const int item = items[b];
    const bool valid = item >= 0 && item < n_items;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int channel_tiles = (channels + kGatherTile - 1) / kGatherTile;
    if ((int)blockIdx.y == channel_tiles) {
        const int count = valid ? n_words[item] : 0;
        const float* source = word_targets + (valid ? word_start[item] : 0);
        float* destination = targets + (size_t)b * wmax;
        const int threads = kGatherTile * kGatherRows;
        for (int w = blockIdx.x * threads + ty * kGatherTile + tx; w < wmax;
             w += gridDim.x * threads)
            destination[w] = w < count ? source[w] : 0.f;
        return;
    }
    __shared__ float tile[kGatherTile][kGatherTile + 1];
    const int t0 = blockIdx.x * kGatherTile, c0 = blockIdx.y * kGatherTile;
    const int frames = valid ? n_rows[item] : 0;
    const float* source = rows + (valid ? (size_t)row_start[item] * channels : 0);
#pragma unroll
    for (int i = ty; i < kGatherTile; i += kGatherRows) {
        const int t = t0 + i, c = c0 + tx;
        tile[i][tx] = (t < frames && c < channels)
            ? source[(size_t)t * channels + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = ty; i < kGatherTile; i += kGatherRows) {
        const int c = c0 + i, t = t0 + tx;
        if (c < channels && t < tmax)
            features[((size_t)b * channels + c) * tmax + t] = tile[tx][i];
    }
}

}  // namespace emph

extern "C" int emph_gather_batch(
    const float* rows, int32_t channels,
    const int32_t* row_start, const int32_t* n_rows,
    const float* word_targets, const int32_t* word_start, const int32_t* n_words,
    int32_t n_items, const int32_t* items, int32_t batch, int32_t tmax, int32_t wmax,
    float* features, float* targets, void* stream) {
    using namespace emph;
    EMPH_REQUIRE(n_items >= 0, "emph_gather_batch: negative corpus size");
    EMPH_REQUIRE(channels > 0, "emph_gather_batch: channels %d must be positive", channels);
    EMPH_REQUIRE(batch > 0 && batch <= 65535,
                 "emph_gather_batch: batch %d is not in 1 .. 65535", batch);
    EMPH_REQUIRE(tmax > 0 && wmax > 0,
                 "emph_gather_batch: Tmax %d and Wmax %d must be positive", tmax, wmax);
    EMPH_REQUIRE(rows && row_start && n_rows && word_targets && word_start && n_words &&
                 items && features && targets,
                 "emph_gather_batch: NULL buffer");
    const int time_tiles = (tmax + kGatherTile - 1) / kGatherTile;
    const int channel_tiles = (channels + kGatherTile - 1) / kGatherTile;
    dim3 grid(time_tiles, channel_tiles + 1, batch);
    dim3 block(kGatherTile, kGatherRows);
    gather_batch_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
        rows, channels, row_start, n_rows, word_targets, word_start, n_words, n_items, items,
        tmax, wmax, features, targets);
    EMPH_CHECK_LAUNCH("emph_gather_batch");
    return EMPH_OK;
}
