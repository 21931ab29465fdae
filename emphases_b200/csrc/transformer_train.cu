// Training kernels of the Transformer variant that are not attention or
// LayerNorm (those live in attention.cu), fp32, sm_100a:
//   emph_dropout_keep          the keep mask of any index range of a site, through
//                              the device function every dropping kernel uses
//   emph_dropout_rows          y = x * keep / (1 - p) over packed rows: the
//                              positional-encoding and feed-forward sites, and
//                              (same mask, same call) their backward
//   emph_linear_rows           y_m = act(x W_m^T + b_m) for the stacked blocks
//                              W_m of a Linear weight (in_proj: q, k, v)
//   emph_linear_rows_backward  dx = addend + sum_m dy_m W_m
// The weight gradients of the linear maps are emph_conv_weight_grad with
// kernel_size 1 (train.cu).
#include "common.cuh"
#include "dropout.cuh"

namespace emph {

__global__ void dropout_keep_kernel(
    Dropout drop, unsigned long long first, long long count, uint8_t* __restrict__ keep) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
         i += (long long)gridDim.x * blockDim.x)
        keep[i] = dropout_keep(drop, drop.site, first + (unsigned long long)i) ? 1 : 0;
}

// one thread per group of four elements: one Philox call
__global__ void dropout_rows_kernel(
    const float4* __restrict__ x, long long groups, Dropout drop, float4* __restrict__ y) {
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
         g += (long long)gridDim.x * blockDim.x) {
        float4 value = x[g];
        if (drop.threshold != 0ull) {
            const uint4 draws = philox_draws(drop.seed, drop.site, (unsigned long long)g);
            const unsigned long long at = 4ull * (unsigned long long)g;
            value.x *= dropout_factor(drop, draws, at);
            value.y *= dropout_factor(drop, draws, at + 1);
            value.z *= dropout_factor(drop, draws, at + 2);
            value.w *= dropout_factor(drop, draws, at + 3);
        }
        y[g] = value;
    }
}

// 32 rows per CTA, thread (n, ty) owns output column n of rows ty, ty + 4, ...
// The weight block sits in shared memory as ws[contraction][output]: W_m^T
// for the forward, W_m itself for the input gradient.
constexpr int kLinC = 80;
constexpr int kLinRows = 32;
constexpr int kLinY = 4;

template <bool ADJOINT>
__global__ void __launch_bounds__(kLinC * kLinY)
linear_rows_kernel(
    const float* __restrict__ in, const float* __restrict__ weight, const float* __restrict__ bias,
    const float* __restrict__ addend, int parts, int act, const int32_t* __restrict__ row_seq,
    int total_rows, float* __restrict__ out) {
    __shared__ float ws[kLinC][kLinC + 1];
    __shared__ float xs[kLinRows][kLinC];
    const int n = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * kLinC + n;
    const int r0 = blockIdx.x * kLinRows;
    const size_t plane = (size_t)total_rows * kLinC;
    float acc[kLinRows / kLinY];
#pragma unroll
    for (int i = 0; i < kLinRows / kLinY; ++i) {
        const int r = r0 + ty + kLinY * i;
        acc[i] = ADJOINT && addend != nullptr && r < total_rows ? addend[(size_t)r * kLinC + n] : 0.f;
    }
    for (int m = 0; m < parts; ++m) {
        __syncthreads();
        for (int e = tid; e < kLinC * kLinC; e += kLinC * kLinY) {
            const int o = e / kLinC, i = e % kLinC;
            const float w = weight[((size_t)m * kLinC + o) * kLinC + i];
            if (ADJOINT) ws[o][i] = w;
            else ws[i][o] = w;
        }
        if (ADJOINT || m == 0) {
            const float* source = in + (ADJOINT ? m * plane : 0);
            for (int e = tid; e < kLinRows * kLinC; e += kLinC * kLinY) {
                const int r = e / kLinC, c = e % kLinC;
                xs[r][c] = r0 + r < total_rows ? source[(size_t)(r0 + r) * kLinC + c] : 0.f;
            }
        }
        __syncthreads();
        if (!ADJOINT) {
#pragma unroll
            for (int i = 0; i < kLinRows / kLinY; ++i) acc[i] = bias[m * kLinC + n];
        }
#pragma unroll 4
        for (int c = 0; c < kLinC; ++c) {
            const float w = ws[c][n];
#pragma unroll
            for (int i = 0; i < kLinRows / kLinY; ++i) acc[i] = fmaf(xs[ty + kLinY * i][c], w, acc[i]);
        }
        if (!ADJOINT) {
#pragma unroll
            for (int i = 0; i < kLinRows / kLinY; ++i) {
                const int r = r0 + ty + kLinY * i;
                if (r < total_rows)
                    out[m * plane + (size_t)r * kLinC + n] =
                        row_seq[r] >= 0 ? apply_activation(acc[i], act) : 0.f;
            }
        }
    }
    if (ADJOINT) {
#pragma unroll
        for (int i = 0; i < kLinRows / kLinY; ++i) {
            const int r = r0 + ty + kLinY * i;
            if (r < total_rows) out[(size_t)r * kLinC + n] = row_seq[r] >= 0 ? acc[i] : 0.f;
        }
    }
}

}  // namespace emph

extern "C" {

int emph_dropout_keep(
    uint64_t seed, uint32_t site, uint64_t first, int64_t count, float p, uint8_t* keep,
    void* stream) {
    EMPH_REQUIRE(count >= 0 && p >= 0.f && p <= 1.f, "emph_dropout_keep: count %lld, p %f",
                 (long long)count, p);
    if (count == 0) return EMPH_OK;
    long long blocks = (count + 255) / 256;
    if (blocks > emph::sm_count() * 8) blocks = emph::sm_count() * 8;
    emph::dropout_keep_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
        emph::make_dropout(seed, site, p), first, count, keep);
    EMPH_CHECK_LAUNCH("emph_dropout_keep");
    return EMPH_OK;
}

int emph_dropout_rows(
    const float* x, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site, float p,
    float* y, void* stream) {
    EMPH_REQUIRE(total_rows >= 0 && channels > 0 && channels % 4 == 0 && p >= 0.f && p <= 1.f,
                 "emph_dropout_rows: rows %d, channels %d, p %f", total_rows, channels, p);
    const long long groups = (long long)total_rows * channels / 4;
    if (groups == 0) return EMPH_OK;
    long long blocks = (groups + 255) / 256;
    if (blocks > emph::sm_count() * 8) blocks = emph::sm_count() * 8;
    emph::dropout_rows_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(x), groups, emph::make_dropout(seed, site, p),
        reinterpret_cast<float4*>(y));
    EMPH_CHECK_LAUNCH("emph_dropout_rows");
    return EMPH_OK;
}

int emph_linear_rows(
    const float* x, int32_t total_rows, int32_t channels, const float* weight, const float* bias,
    int32_t parts, int32_t act, const int32_t* row_seq, float* y, void* stream) {
    EMPH_REQUIRE(channels == emph::kLinC, "emph_linear_rows: channels %d not compiled in", channels);
    EMPH_REQUIRE(parts >= 1 && act >= EMPH_ACT_NONE && act <= EMPH_ACT_SILU,
                 "emph_linear_rows: parts %d, act %d", parts, act);
    if (total_rows == 0) return EMPH_OK;
    emph::linear_rows_kernel<false>
        <<<(total_rows + emph::kLinRows - 1) / emph::kLinRows, dim3(emph::kLinC, emph::kLinY), 0,
           (cudaStream_t)stream>>>(x, weight, bias, nullptr, parts, act, row_seq, total_rows, y);
    EMPH_CHECK_LAUNCH("emph_linear_rows");
    return EMPH_OK;
}

int emph_linear_rows_backward(
    const float* dy, int32_t total_rows, int32_t channels, const float* weight, int32_t parts,
    const float* addend, const int32_t* row_seq, float* dx, void* stream) {
    EMPH_REQUIRE(channels == emph::kLinC, "emph_linear_rows_backward: channels %d not compiled in",
                 channels);
    EMPH_REQUIRE(parts >= 1, "emph_linear_rows_backward: parts %d", parts);
    if (total_rows == 0) return EMPH_OK;
    emph::linear_rows_kernel<true>
        <<<(total_rows + emph::kLinRows - 1) / emph::kLinRows, dim3(emph::kLinC, emph::kLinY), 0,
           (cudaStream_t)stream>>>(dy, weight, nullptr, addend, parts, EMPH_ACT_NONE, row_seq,
                                   total_rows, dx);
    EMPH_CHECK_LAUNCH("emph_linear_rows_backward");
    return EMPH_OK;
}

}  // extern "C"
