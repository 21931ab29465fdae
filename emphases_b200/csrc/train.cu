// Backward kernels of the conv model for the data-parallel training step
// (BASELINE config 5; reference single-device step: emphases/train/core.py:
// 86-142, loss: emphases/train/core.py:315-353), fp32, sm_100a.
//
// Forward in training keeps every layer's activations (one emph_conv_stack
// launch per layer); backward per Conv1d(C -> C, k, 'same') + activation:
//   dpre = dY * act'(Y)                       emph_activation_backward
//   dX   = conv(dpre, W flipped/transposed)   emph_conv_stack (existing kernel)
//   dW[tap][ci][co] = sum_r X[r + tap - half][ci] dpre[r][co],  db = sum_r dpre
//                                             emph_conv_weight_grad
// plus the backward of word pooling, of the output projection and the masked
// BCE / MSE loss with its gradient, and the dropout after a layer's activation
// (emph_conv_dropout_forward / emph_activation_dropout_backward).
#include <math_constants.h>

#include <cuda_bf16.h>

#include "common.cuh"
#include "dropout.cuh"

namespace emph {

// g * act'(.) at `v`: the layer's OUTPUT for ReLU / LeakyReLU / identity (the
// sign of the output decides) and the PRE-activation for GELU / SiLU (their
// derivative is not a function of the output; the training forward keeps it,
// emph_activation_forward)
__device__ __forceinline__ float activation_grad(float g, float v, int act) {
    if (act == EMPH_ACT_RELU) {
        g = v > 0.f ? g : 0.f;
    } else if (act == EMPH_ACT_LEAKY_RELU) {
        g = v > 0.f ? g : 0.01f * g;
    } else if (act == EMPH_ACT_GELU) {
        // d/dx [x Phi(x)] = Phi(x) + x phi(x)
        const float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752f));
        const float pdf = 0.3989422804014327f * expf(-0.5f * v * v);
        g *= cdf + v * pdf;
    } else if (act == EMPH_ACT_SILU) {
        const float sig = 1.f / (1.f + expf(-v));
        g *= sig * (1.f + v * (1.f - sig));
    }
    return g;
}

// dpre = dy * act'(.), separator rows zeroed
__global__ void activation_backward_kernel(
    const float* __restrict__ dy, const float* __restrict__ y,
    const int32_t* __restrict__ row_seq, int total_rows, int channels, int act,
    float* __restrict__ dpre) {
    const size_t n = (size_t)total_rows * channels;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / channels);
        const float g = activation_grad(dy[i], y[i], act);
        dpre[i] = row_seq[r] >= 0 ? g : 0.f;
    }
}

// y = act(pre), separator rows zeroed (training forward of GELU / SiLU layers,
// whose pre-activation is kept for the backward pass)
__global__ void activation_forward_kernel(
    const float* __restrict__ pre, const int32_t* __restrict__ row_seq, int total_rows,
    int channels, int act, float* __restrict__ y) {
    const size_t n = (size_t)total_rows * channels;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / channels);
        y[i] = row_seq[r] >= 0 ? apply_activation(pre[i], act) : 0.f;
    }
}

// Dropout after a conv layer's activation (emphases/model/layers/
// convolution.py:25-30: Conv1d -> activation -> Dropout).  The element index of
// the mask is the element's position in the reference's padded (N, width, C)
// tensor, channel fastest:  ((n * width + w) * C + c) with n = row_seq[r] and
// w = r - row_start[n], so the mask does not depend on how rows are packed.
// One thread per float4 (four channels of one row: one Philox call, C % 4 == 0).

// y = act(x) * keep / (1 - p), separator rows zeroed.  x may be y (in place).
__global__ void conv_dropout_forward_kernel(
    const float4* x, const int32_t* __restrict__ row_seq,
    const int32_t* __restrict__ row_start, int total_rows, int quads, int width, int act,
    Dropout drop, float4* y) {
    const long long n = (long long)total_rows * quads;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / quads), q = (int)(i % quads);
        const int u = row_seq[r];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (u >= 0) {
            v = x[i];
            v.x = apply_activation(v.x, act);
            v.y = apply_activation(v.y, act);
            v.z = apply_activation(v.z, act);
            v.w = apply_activation(v.w, act);
            if (drop.threshold != 0ull) {
                const unsigned long long group =
                    ((unsigned long long)u * width + (r - row_start[u])) * quads + q;
                const uint4 draws = philox_draws(drop.seed, drop.site, group);
                v.x *= dropout_factor(drop, draws, 4 * group);
                v.y *= dropout_factor(drop, draws, 4 * group + 1);
                v.z *= dropout_factor(drop, draws, 4 * group + 2);
                v.w *= dropout_factor(drop, draws, 4 * group + 3);
            }
        }
        y[i] = v;
    }
}

// dpre = dy * keep / (1 - p) * act'(.), the mask regenerated from the seed;
// `y` as for activation_grad.  For ReLU / LeakyReLU the kept output is the
// dropped one: where the mask keeps an element its sign is the activation's,
// and where it drops one the factor is 0.
__global__ void activation_dropout_backward_kernel(
    const float4* __restrict__ dy, const float4* __restrict__ y,
    const int32_t* __restrict__ row_seq, const int32_t* __restrict__ row_start, int total_rows,
    int quads, int width, int act, Dropout drop, float4* __restrict__ dpre) {
    const long long n = (long long)total_rows * quads;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / quads), q = (int)(i % quads);
        const int u = row_seq[r];
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (u >= 0) {
            g = dy[i];
            const float4 v = y[i];
            if (drop.threshold != 0ull) {
                const unsigned long long group =
                    ((unsigned long long)u * width + (r - row_start[u])) * quads + q;
                const uint4 draws = philox_draws(drop.seed, drop.site, group);
                g.x *= dropout_factor(drop, draws, 4 * group);
                g.y *= dropout_factor(drop, draws, 4 * group + 1);
                g.z *= dropout_factor(drop, draws, 4 * group + 2);
                g.w *= dropout_factor(drop, draws, 4 * group + 3);
            }
            g.x = activation_grad(g.x, v.x, act);
            g.y = activation_grad(g.y, v.y, act);
            g.z = activation_grad(g.z, v.z, act);
            g.w = activation_grad(g.w, v.w, act);
        }
        dpre[i] = g;
    }
}

// Weight / bias gradient of one conv layer.  256 threads: thread (gi, go) owns
// a 5 x 5 block of (ci, co) for all taps (C = 80: 16 x 16 blocks).
// CONV1D: dw is addressed as the Conv1d parameter (out, in, k) instead of the
// packed [k][in][out]
template <int C, int KS, bool CONV1D>
__global__ void __launch_bounds__(256)
conv_weight_grad_kernel(
    const float* __restrict__ x, const float* __restrict__ dpre, int total_rows,
    float* __restrict__ dw, float* __restrict__ db) {
    constexpr int R = 64;                  // rows per smem tile
    constexpr int HALF = (KS - 1) / 2;
    constexpr int B = C / 16;              // block edge (5 for C = 80)
    __shared__ float xs[R + 2 * HALF][C + 1];
    __shared__ float ds[R][C + 1];
    const int tid = threadIdx.x;
    const int gi = tid >> 4, go = tid & 15;
    float acc[KS][B][B];
    float bias_acc[B];
#pragma unroll
    for (int t = 0; t < KS; ++t)
#pragma unroll
        for (int i = 0; i < B; ++i)
#pragma unroll
            for (int o = 0; o < B; ++o) acc[t][i][o] = 0.f;
#pragma unroll
    for (int o = 0; o < B; ++o) bias_acc[o] = 0.f;

    for (int r0 = blockIdx.x * R; r0 < total_rows; r0 += gridDim.x * R) {
        __syncthreads();
        for (int i = tid; i < (R + 2 * HALF) * C; i += 256) {
            const int r = i / C, c = i % C;
            const int g = r0 + r - HALF;
            xs[r][c] = (g >= 0 && g < total_rows) ? x[(size_t)g * C + c] : 0.f;
        }
        for (int i = tid; i < R * C; i += 256) {
            const int r = i / C, c = i % C;
            const int g = r0 + r;
            ds[r][c] = g < total_rows ? dpre[(size_t)g * C + c] : 0.f;
        }
        __syncthreads();
#pragma unroll 2
        for (int r = 0; r < R; ++r) {
            float d[B];
#pragma unroll
            for (int o = 0; o < B; ++o) d[o] = ds[r][go * B + o];
            if (gi == 0) {
#pragma unroll
                for (int o = 0; o < B; ++o) bias_acc[o] += d[o];
            }
#pragma unroll
            for (int t = 0; t < KS; ++t) {
#pragma unroll
                for (int i = 0; i < B; ++i) {
                    const float xv = xs[r + t][gi * B + i];
#pragma unroll
                    for (int o = 0; o < B; ++o) acc[t][i][o] = fmaf(xv, d[o], acc[t][i][o]);
                }
            }
        }
    }
#pragma unroll
    for (int t = 0; t < KS; ++t)
#pragma unroll
        for (int i = 0; i < B; ++i)
#pragma unroll
            for (int o = 0; o < B; ++o)
                atomicAdd(
                    dw + (CONV1D ? ((size_t)(go * B + o) * C + gi * B + i) * KS + t
                                 : ((size_t)t * C + gi * B + i) * C + go * B + o),
                    acc[t][i][o]);
    if (gi == 0) {
#pragma unroll
        for (int o = 0; o < B; ++o) atomicAdd(db + go * B + o, bias_acc[o]);
    }
}

// ---------------------------------------------------------------------------
// Weight gradient on the warp-level tensor path (mma.sync m16n8k16, bf16
// operands split hi + lo, fp32 accumulate): per tap
//     dW_tap[in][out] = sum_r X[r + tap - (KS - 1) / 2][in] * dPre[r][out]
// is a GEMM with the ROW axis as K.  Both operands sit in shared memory as they
// sit in HBM, [row][channel], converted to a bf16 hi and a bf16 lo plane while
// they are staged (x = hi + lo to 16 bits; hi*hi + lo*hi + hi*lo keeps the
// products to ~1.5e-5), and ldmatrix.trans hands out the K-major fragments.
// A tile stages X rows r0 - (KS - 1) / 2 .. r0 + R - 1 + (KS - 1) / 2 (the
// halo of every tap) and dPre rows r0 .. r0 + R - 1.
//
// Work split.  The result is KS x C/16 (tap, m-tile) strips of C/8 m16n8
// tiles each (4 floats per lane per tile).  A CTA keeps PER_WARP strips per
// warp in registers while it walks a contiguous range of 64-row tiles, and
// adds them to the gradient once at the end (split-K over CTAs, one float
// atomic per element and CTA).  When the strips do not fit in one CTA they
// are spread over gridDim.y (SLICES), each slice staging the same tiles:
//   C = 80:  2 strips per warp (80 accumulators), ceil(5 KS / 16) slices:
//            k = 3 one slice (15 strips), k = 5 two, k = 7 three;
//   C = 128: 1 strip per warp (16 n-tiles: 64 accumulators, plus 64
//            registers of dPre fragments per k-step), so one tap per slice.
// Only slice 0 sums the bias.  Every slice gets sm_count / SLICES CTAs, so the
// grid fills the SMs once; <80, 3> keeps its one-slice launch of one CTA per
// SM.  Rows are padded to LD bf16 = C + 8 (176 B at 80, 272 B at 128: odd
// multiples of 16 B, so the 8 row addresses of an ldmatrix hit distinct banks).
// This replaces the FFMA kernel above in the native training step: ~15 instead
// of ~110 us per frame layer at 80 channels, kernel size 3.
// ---------------------------------------------------------------------------
namespace wgrad {
constexpr int R = 64;                       // rows per tile (K of the GEMM)

template <int C, int KS>
struct Shape {
    static constexpr int LD = C + 8;        // bf16 per smem row
    static constexpr int XROWS = R + KS - 1;
    static constexpr int HALF = (KS - 1) / 2;
    static constexpr int MT = C / 16;       // m-tiles per tap
    static constexpr int NT = C / 8;        // n-tiles
    static constexpr int ROWSETS = KS * MT; // (tap, m-tile) strips
    static constexpr int PER_WARP = C <= 80 ? 2 : 1;
    static constexpr int SLICE = 8 * PER_WARP;                  // strips per CTA
    static constexpr int SLICES = (ROWSETS + SLICE - 1) / SLICE;
    static constexpr int C4 = C / 4;        // float4 columns
    static constexpr int ROW_GROUPS = 256 / C4;                 // staging threads per column
};

template <int C, int KS>
struct Smem {
    __nv_bfloat16 x[2][Shape<C, KS>::XROWS][Shape<C, KS>::LD];  // [hi / lo][row][channel]
    __nv_bfloat16 d[2][R][Shape<C, KS>::LD];
    float bias[C];
};

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split_store(__nv_bfloat16* hi, __nv_bfloat16* lo, float4 v) {
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    const float2 b0 = __bfloat1622float2(h0), b1 = __bfloat1622float2(h1);
    const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - b0.x, v.y - b0.y);
    const __nv_bfloat162 l1 = __floats2bfloat162_rn(v.z - b1.x, v.w - b1.y);
    *reinterpret_cast<uint2*>(hi) =
        make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
    *reinterpret_cast<uint2*>(lo) =
        make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
}

template <int C, int KS, bool CONV1D>
__global__ void __launch_bounds__(256)
conv_weight_grad_mma_kernel(
    const float* __restrict__ x, const float* __restrict__ dpre, int total_rows, int tiles_per_cta,
    float* __restrict__ dw, float* __restrict__ db) {
    using S = Shape<C, KS>;
    constexpr int NT = S::NT, MT = S::MT, PER_WARP = S::PER_WARP, C4 = S::C4;
    constexpr int GROUPS = S::ROW_GROUPS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem<C, KS>& sm = *reinterpret_cast<Smem<C, KS>*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float acc[PER_WARP][NT][4];
#pragma unroll
    for (int s = 0; s < PER_WARP; ++s)
#pragma unroll
        for (int n = 0; n < NT; ++n)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[s][n][j] = 0.f;
    // bias gradient: thread (c4 = tid % C4) sums its 4 channels over rows
    // tid / C4, + GROUPS, ...
    float4 bias_acc = make_float4(0.f, 0.f, 0.f, 0.f);

    const int n_tiles = (total_rows + R - 1) / R;
    const int first = blockIdx.x * tiles_per_cta;
    const int last = min(first + tiles_per_cta, n_tiles);
    // strips of this warp: (tap, m-tile) = strip / MT, strip % MT; strips
    // >= ROWSETS do not exist (<80, 3>: strip 15).  Slice 0 sums the bias.
    const int slice = S::SLICES == 1 ? 0 : blockIdx.y;
    const bool bias_slice = slice == 0;
    int strip[PER_WARP];
#pragma unroll
    for (int s = 0; s < PER_WARP; ++s) strip[s] = slice * S::SLICE + warp + 8 * s;

    for (int tile = first; tile < last; ++tile) {
        const int r0 = tile * R;
        __syncthreads();
        // ---- stage X rows r0 - HALF .. r0 + R - 1 + HALF and dPre rows
        // r0 .. r0 + R - 1, split hi / lo; thread = (row % GROUPS, float4
        // column): a fixed column per thread, so the bias gradient (column
        // sums of dPre) accumulates in registers ----
        if (tid < GROUPS * C4) {
            const int c4 = tid % C4;
            for (int r = tid / C4; r < S::XROWS; r += GROUPS) {
                const int g = r0 + r - S::HALF;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g >= 0 && g < total_rows)
                    v = *reinterpret_cast<const float4*>(x + (size_t)g * C + 4 * c4);
                split_store(&sm.x[0][r][4 * c4], &sm.x[1][r][4 * c4], v);
            }
            for (int r = tid / C4; r < R; r += GROUPS) {
                const int g = r0 + r;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g < total_rows)
                    v = *reinterpret_cast<const float4*>(dpre + (size_t)g * C + 4 * c4);
                if (bias_slice) {
                    bias_acc.x += v.x; bias_acc.y += v.y; bias_acc.z += v.z; bias_acc.w += v.w;
                }
                split_store(&sm.d[0][r][4 * c4], &sm.d[1][r][4 * c4], v);
            }
        }
        __syncthreads();
        // ---- 4 k-steps of 16 rows ----
#pragma unroll 1
        for (int k0 = 0; k0 < R; k0 += 16) {
            // B fragments of all NT n-tiles, hi and lo: x4.trans covers two n-tiles
            // (matrices: [k0..7][n0..7], [k0+8..15][n0..7], [k0..7][n0+8..15], [k0+8..15][n0+8..15])
            uint32_t bh[NT][2], bl[NT][2];
#pragma unroll
            for (int n2 = 0; n2 < NT / 2; ++n2) {
                const int row = k0 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int col = 16 * n2 + (lane >> 4) * 8;
                uint32_t t[4];
                ldmatrix_x4_trans(t, &sm.d[0][row][col]);
                bh[2 * n2][0] = t[0]; bh[2 * n2][1] = t[1]; bh[2 * n2 + 1][0] = t[2]; bh[2 * n2 + 1][1] = t[3];
                ldmatrix_x4_trans(t, &sm.d[1][row][col]);
                bl[2 * n2][0] = t[0]; bl[2 * n2][1] = t[1]; bl[2 * n2 + 1][0] = t[2]; bl[2 * n2 + 1][1] = t[3];
            }
#pragma unroll
            for (int s = 0; s < PER_WARP; ++s) {
                if (strip[s] >= S::ROWSETS) continue;              // warp-uniform
                const int tap = strip[s] / MT, m0 = (strip[s] % MT) * 16;
                // A fragment = X^T: matrices [k0..7][m0..7], [k0..7][m0+8..15],
                // [k0+8..15][m0..7], [k0+8..15][m0+8..15]; tap t reads buffer row k + t
                const int row = k0 + tap + (lane & 7) + (lane >> 4) * 8;
                const int col = m0 + ((lane >> 3) & 1) * 8;
                uint32_t ah[4], al[4];
                ldmatrix_x4_trans(ah, &sm.x[0][row][col]);
                ldmatrix_x4_trans(al, &sm.x[1][row][col]);
#pragma unroll
                for (int n = 0; n < NT; ++n) {
                    mma_bf16(acc[s][n], al, bh[n][0], bh[n][1]);      // smallest terms first
                    mma_bf16(acc[s][n], ah, bl[n][0], bl[n][1]);
                    mma_bf16(acc[s][n], ah, bh[n][0], bh[n][1]);
                }
            }
        }
    }
    // ---- add this CTA's partial result to the gradient ----
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int s = 0; s < PER_WARP; ++s) {
        if (strip[s] >= S::ROWSETS) continue;
        const int tap = strip[s] / MT, m0 = (strip[s] % MT) * 16;
#pragma unroll
        for (int n = 0; n < NT; ++n) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int in = m0 + g + (j >> 1) * 8, out = 8 * n + 2 * t + (j & 1);
                atomicAdd(
                    dw + (CONV1D ? ((size_t)out * C + in) * KS + tap : ((size_t)tap * C + in) * C + out),
                    acc[s][n][j]);
            }
        }
    }
    // bias: the GROUPS row-groups' column sums -> shared -> the gradient
    if (!bias_slice) return;                                    // CTA-uniform
    __syncthreads();
    for (int i = tid; i < C; i += 256) sm.bias[i] = 0.f;
    __syncthreads();
    if (tid < GROUPS * C4) {
        const int c4 = tid % C4;
        atomicAdd(&sm.bias[4 * c4 + 0], bias_acc.x);
        atomicAdd(&sm.bias[4 * c4 + 1], bias_acc.y);
        atomicAdd(&sm.bias[4 * c4 + 2], bias_acc.z);
        atomicAdd(&sm.bias[4 * c4 + 3], bias_acc.w);
    }
    __syncthreads();
    for (int i = tid; i < C; i += 256) atomicAdd(db + i, sm.bias[i]);
}

// Adds the gradient of `total_rows` rows to dw / db (zeroed by the caller):
// contiguous ranges of 64-row tiles, sm_count / SLICES CTAs per slice
template <int C, int KS, bool CONV1D>
int launch(const float* x, const float* dpre, int total_rows, float* dw, float* db,
           cudaStream_t st) {
    using S = Shape<C, KS>;
    static bool configured = false;         // one attribute call per instantiation
    if (!configured) {
        int s = check_cuda(
            cudaFuncSetAttribute(conv_weight_grad_mma_kernel<C, KS, CONV1D>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)sizeof(Smem<C, KS>)),
            "weight gradient smem attribute");
        if (s != EMPH_OK) return s;
        configured = true;
    }
    const int n_tiles = (total_rows + R - 1) / R;
    const int per_slice = sm_count() / S::SLICES > 0 ? sm_count() / S::SLICES : 1;
    const int ctas = n_tiles < per_slice ? n_tiles : per_slice;
    const int tiles_per_cta = (n_tiles + ctas - 1) / ctas;
    const int grid = (n_tiles + tiles_per_cta - 1) / tiles_per_cta;
    conv_weight_grad_mma_kernel<C, KS, CONV1D>
        <<<dim3(grid, S::SLICES), 256, sizeof(Smem<C, KS>), st>>>(
            x, dpre, total_rows, tiles_per_cta, dw, db);
    return EMPH_OK;
}
}  // namespace wgrad

// Backward of emph_pool_words: one warp per word row, adds into dx (pre-zeroed)
__global__ void __launch_bounds__(256)
pool_backward_kernel(
    const float* __restrict__ dy, const float* __restrict__ x, int channels,
    const int32_t* __restrict__ row_start, const int32_t* __restrict__ n_rows,
    const int32_t* __restrict__ word_seq, const int32_t* __restrict__ word_lo,
    const int32_t* __restrict__ word_hi, int total_word_rows, int method,
    float* __restrict__ dx) {
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= total_word_rows) return;
    const int u = word_seq[w];
    if (u < 0) return;
    const int lo = word_lo[w], hi = word_hi[w];
    const bool padded_slot = lo == -1 && hi == -1;
    // masked slots never reach the input; padded slots only through `center`,
    // which gathers frame 0 for them (emphases/core.py:458-466)
    if (lo < 0 && !(padded_slot && method == EMPH_POOL_CENTER)) return;
    const int n = n_rows[u];
    const size_t base = (size_t)row_start[u] * channels;
    const float* g = dy + (size_t)w * channels;
    if (method == EMPH_POOL_CENTER) {
        const int idx = padded_slot ? 0 : (lo + hi) >> 1;
        if (idx < n)
            for (int c = lane; c < channels; c += 32)
                atomicAdd(dx + base + (size_t)idx * channels + c, g[c]);
        return;
    }
    const int s = min(max(lo, 0), n), e = min(max(hi, 0), n);
    if (e <= s) return;
    for (int c = lane; c < channels; c += 32) {
        if (method == EMPH_POOL_MAX) {
            int arg = s;
            float best = x[base + (size_t)s * channels + c];
            for (int f = s + 1; f < e; ++f) {
                const float v = x[base + (size_t)f * channels + c];
                if (v > best) { best = v; arg = f; }
            }
            atomicAdd(dx + base + (size_t)arg * channels + c, g[c]);
        } else {
            const float value = method == EMPH_POOL_AVERAGE ? g[c] / (float)(e - s) : g[c];
            for (int f = s; f < e; ++f)
                atomicAdd(dx + base + (size_t)f * channels + c, value);
        }
    }
}

// Backward of emph_output_head (logits only): single CTA, rows are few
__global__ void __launch_bounds__(256)
head_backward_kernel(
    const float* __restrict__ x, const float* __restrict__ dz,
    const int32_t* __restrict__ row_seq, int total_rows, int channels, int kernel_size,
    const float* __restrict__ weight, float* __restrict__ dx, float* __restrict__ dw,
    float* __restrict__ db) {
    const int half = (kernel_size - 1) / 2;
    // dx[r][c] = sum_tap w[tap][c] dz[r + half - tap]
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
         i < (size_t)total_rows * channels; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / channels), c = (int)(i % channels);
        float acc = 0.f;
        for (int tap = 0; tap < kernel_size; ++tap) {
            const int g = r + half - tap;
            if (g >= 0 && g < total_rows && row_seq[g] >= 0) acc = fmaf(weight[tap * channels + c], dz[g], acc);
        }
        dx[i] = row_seq[r] >= 0 ? acc : 0.f;
    }
}

// dw[tap][c] = sum_r x[r + tap - half][c] dz[r];  db = sum_r dz[r] over the rows
// of real sequences: a CTA per chunk of rows, one thread per (tap, c), partial
// sums added to the (zeroed) outputs
constexpr int kHeadGradRows = 64;
__global__ void __launch_bounds__(256)
head_weight_grad_kernel(
    const float* __restrict__ x, const float* __restrict__ dz,
    const int32_t* __restrict__ row_seq, int total_rows, int channels, int kernel_size,
    float* __restrict__ dw, float* __restrict__ db) {
    const int half = (kernel_size - 1) / 2;
    const int r0 = blockIdx.x * kHeadGradRows;
    const int r1 = min(r0 + kHeadGradRows, total_rows);
    for (int i = threadIdx.x; i < kernel_size * channels; i += blockDim.x) {
        const int tap = i / channels, c = i % channels;
        float acc = 0.f;
        for (int r = r0; r < r1; ++r) {
            const int g = r + tap - half;
            if (row_seq[r] >= 0 && g >= 0 && g < total_rows)
                acc = fmaf(x[(size_t)g * channels + c], dz[r], acc);
        }
        if (acc != 0.f) atomicAdd(dw + i, acc);
    }
    if (threadIdx.x == 0) {
        float acc = 0.f;
        for (int r = r0; r < r1; ++r)
            if (row_seq[r] >= 0) acc += dz[r];
        if (acc != 0.f) atomicAdd(db, acc);
    }
}

// Masked loss over packed word rows (emphases/train/core.py:340-353):
// mean over rows with valid[r] != 0 of BCE-with-logits (mode 0) or squared
// error (mode 1); writes the scalar loss and d loss / d logits.  Single CTA.
__global__ void __launch_bounds__(256)
masked_loss_kernel(
    const float* __restrict__ logits, const float* __restrict__ targets,
    const uint8_t* __restrict__ valid, int total_rows, int mode,
    float* __restrict__ loss, float* __restrict__ dlogits) {
    __shared__ float partial[256];
    __shared__ int counts[256];
    float sum = 0.f;
    int count = 0;
    for (int r = threadIdx.x; r < total_rows; r += 256) {
        if (!valid[r]) continue;
        const float z = logits[r], t = targets[r];
        if (mode == 0) sum += fmaxf(z, 0.f) - z * t + log1pf(expf(-fabsf(z)));
        else sum += (z - t) * (z - t);
        ++count;
    }
    partial[threadIdx.x] = sum;
    counts[threadIdx.x] = count;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            partial[threadIdx.x] += partial[threadIdx.x + o];
            counts[threadIdx.x] += counts[threadIdx.x + o];
        }
        __syncthreads();
    }
    const float n = (float)counts[0];
    if (threadIdx.x == 0) loss[0] = partial[0] / n;
    for (int r = threadIdx.x; r < total_rows; r += 256) {
        float g = 0.f;
        if (valid[r]) {
            const float z = logits[r], t = targets[r];
            g = mode == 0 ? (1.f / (1.f + expf(-z)) - t) / n : 2.f * (z - t) / n;
        }
        dlogits[r] = g;
    }
}

}  // namespace emph

extern "C" {

int emph_activation_backward(
    const float* dy, const float* y, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, int32_t act, float* dpre, void* stream) {
    EMPH_REQUIRE(act >= EMPH_ACT_NONE && act <= EMPH_ACT_SILU,
                 "emph_activation_backward: unknown activation %d", act);
    if (total_rows == 0) return EMPH_OK;
    emph::activation_backward_kernel<<<emph::sm_count() * 4, 256, 0, (cudaStream_t)stream>>>(
        dy, y, row_seq, total_rows, channels, act, dpre);
    EMPH_CHECK_LAUNCH("emph_activation_backward");
    return EMPH_OK;
}

int emph_activation_forward(
    const float* pre, const int32_t* row_seq, int32_t total_rows, int32_t channels,
    int32_t act, float* y, void* stream) {
    EMPH_REQUIRE(act >= EMPH_ACT_NONE && act <= EMPH_ACT_SILU,
                 "emph_activation_forward: unknown activation %d", act);
    if (total_rows == 0) return EMPH_OK;
    emph::activation_forward_kernel<<<emph::sm_count() * 4, 256, 0, (cudaStream_t)stream>>>(
        pre, row_seq, total_rows, channels, act, y);
    EMPH_CHECK_LAUNCH("emph_activation_forward");
    return EMPH_OK;
}

static int conv_dropout_grid(int total_rows, int quads) {
    long long blocks = ((long long)total_rows * quads + 255) / 256;
    if (blocks > emph::sm_count() * 8) blocks = emph::sm_count() * 8;
    return (int)blocks;
}

int emph_conv_dropout_forward(
    const float* x, const int32_t* row_seq, const int32_t* row_start, int32_t total_rows,
    int32_t channels, int32_t width, int32_t act, uint64_t seed, uint32_t site, float p,
    float* y, void* stream) {
    EMPH_REQUIRE(act >= EMPH_ACT_NONE && act <= EMPH_ACT_SILU,
                 "emph_conv_dropout_forward: unknown activation %d", act);
    EMPH_REQUIRE(total_rows >= 0 && channels > 0 && channels % 4 == 0 && width > 0 &&
                     p >= 0.f && p <= 1.f,
                 "emph_conv_dropout_forward: rows %d, channels %d, width %d, p %f",
                 total_rows, channels, width, p);
    if (total_rows == 0) return EMPH_OK;
    const int quads = channels / 4;
    emph::conv_dropout_forward_kernel<<<conv_dropout_grid(total_rows, quads), 256, 0,
                                        (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(x), row_seq, row_start, total_rows, quads, width, act,
        emph::make_dropout(seed, site, p), reinterpret_cast<float4*>(y));
    EMPH_CHECK_LAUNCH("emph_conv_dropout_forward");
    return EMPH_OK;
}

int emph_activation_dropout_backward(
    const float* dy, const float* y, const int32_t* row_seq, const int32_t* row_start,
    int32_t total_rows, int32_t channels, int32_t width, int32_t act, uint64_t seed,
    uint32_t site, float p, float* dpre, void* stream) {
    EMPH_REQUIRE(act >= EMPH_ACT_NONE && act <= EMPH_ACT_SILU,
                 "emph_activation_dropout_backward: unknown activation %d", act);
    EMPH_REQUIRE(total_rows >= 0 && channels > 0 && channels % 4 == 0 && width > 0 &&
                     p >= 0.f && p <= 1.f,
                 "emph_activation_dropout_backward: rows %d, channels %d, width %d, p %f",
                 total_rows, channels, width, p);
    if (total_rows == 0) return EMPH_OK;
    const int quads = channels / 4;
    emph::activation_dropout_backward_kernel<<<conv_dropout_grid(total_rows, quads), 256, 0,
                                               (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(dy), reinterpret_cast<const float4*>(y), row_seq,
        row_start, total_rows, quads, width, act, emph::make_dropout(seed, site, p),
        reinterpret_cast<float4*>(dpre));
    EMPH_CHECK_LAUNCH("emph_activation_dropout_backward");
    return EMPH_OK;
}

int emph_conv_weight_grad(
    const float* x, const float* dpre, int32_t total_rows, int32_t channels,
    int32_t kernel_size, float* dw, float* db, void* stream) {
    // 80 channels, kernel size 1 / 3: the FFMA kernel (the per-kernel path's
    // fp32 step and the Linear maps of the Transformer variant); 80 / 5, 7
    // and 128 / 1, 3, 5, 7: the split-bf16 mma.sync kernel
    const bool ffma = channels == 80 && (kernel_size == 1 || kernel_size == 3);
    const bool mma = (channels == 80 && (kernel_size == 5 || kernel_size == 7)) ||
                     (channels == 128 && (kernel_size == 1 || kernel_size == 3 ||
                                          kernel_size == 5 || kernel_size == 7));
    if (!(ffma || mma)) {
        emph::set_error("emph_conv_weight_grad: channels=%d kernel_size=%d not compiled in",
                        channels, kernel_size);
        return EMPH_ENOSYS;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int s = emph::check_cuda(
        cudaMemsetAsync(dw, 0, sizeof(float) * kernel_size * channels * channels, st), "memset dw");
    if (s != EMPH_OK) return s;
    s = emph::check_cuda(cudaMemsetAsync(db, 0, sizeof(float) * channels, st), "memset db");
    if (s != EMPH_OK) return s;
    if (total_rows == 0) return EMPH_OK;
    if (ffma) {
        int grid = (total_rows + 63) / 64;
        if (grid > emph::sm_count() * 2) grid = emph::sm_count() * 2;
        if (kernel_size == 3)
            emph::conv_weight_grad_kernel<80, 3, false><<<grid, 256, 0, st>>>(
                x, dpre, total_rows, dw, db);
        else        // the Linear maps of the Transformer variant
            emph::conv_weight_grad_kernel<80, 1, false><<<grid, 256, 0, st>>>(
                x, dpre, total_rows, dw, db);
    } else {
        namespace w = emph::wgrad;
        if (channels == 80)
            s = kernel_size == 5 ? w::launch<80, 5, false>(x, dpre, total_rows, dw, db, st)
                                 : w::launch<80, 7, false>(x, dpre, total_rows, dw, db, st);
        else if (kernel_size == 1)
            s = w::launch<128, 1, false>(x, dpre, total_rows, dw, db, st);
        else if (kernel_size == 3)
            s = w::launch<128, 3, false>(x, dpre, total_rows, dw, db, st);
        else if (kernel_size == 5)
            s = w::launch<128, 5, false>(x, dpre, total_rows, dw, db, st);
        else
            s = w::launch<128, 7, false>(x, dpre, total_rows, dw, db, st);
        if (s != EMPH_OK) return s;
    }
    EMPH_CHECK_LAUNCH("emph_conv_weight_grad");
    return EMPH_OK;
}
}  // extern "C"

// The same sums written (accumulate = 0: after zeroing) or added straight into
// the gradient of the Conv1d parameter, (out, in, k) and (out): no layout pass
namespace emph {
int conv1d_weight_grad(
    const float* x, const float* dpre, int total_rows, int channels, int kernel_size,
    float* grad_weight, float* grad_bias, int accumulate, cudaStream_t st) {
    if (!(channels == 80 && kernel_size == 3)) {
        set_error("conv1d_weight_grad: channels=%d kernel_size=%d not compiled in",
                  channels, kernel_size);
        return EMPH_ENOSYS;
    }
    if (!accumulate) {
        int s = check_cuda(
            cudaMemsetAsync(grad_weight, 0, sizeof(float) * kernel_size * channels * channels, st),
            "memset dw");
        if (s != EMPH_OK) return s;
        s = check_cuda(cudaMemsetAsync(grad_bias, 0, sizeof(float) * channels, st), "memset db");
        if (s != EMPH_OK) return s;
    }
    if (total_rows == 0) return EMPH_OK;
    // one CTA per SM: every CTA ends with 19,280 atomics on the same addresses,
    // and halving their number beats the second CTA's latency hiding (measured:
    // 2.015 / 2.049 / 2.20 / 2.36 ms per training step at 1 / 2 / 3 / 4 CTAs per SM)
    // tensor-core kernel: contiguous ranges of 64-row tiles, one CTA per SM
    const int s = wgrad::launch<80, 3, true>(x, dpre, total_rows, grad_weight, grad_bias, st);
    if (s != EMPH_OK) return s;
    EMPH_CHECK_LAUNCH("conv1d_weight_grad");
    return EMPH_OK;
}
}  // namespace emph

extern "C" {

int emph_pool_words_backward(
    const float* dy, const float* x, int32_t channels,
    const int32_t* row_start, const int32_t* n_rows,
    const int32_t* word_seq, const int32_t* word_lo, const int32_t* word_hi,
    int32_t total_word_rows, int32_t method, int32_t total_rows, float* dx, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int s = emph::check_cuda(
        cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)total_rows * channels, st), "memset dx");
    if (s != EMPH_OK) return s;
    if (total_word_rows == 0) return EMPH_OK;
    emph::pool_backward_kernel<<<(total_word_rows + 7) / 8, 256, 0, st>>>(
        dy, x, channels, row_start, n_rows, word_seq, word_lo, word_hi, total_word_rows,
        method, dx);
    EMPH_CHECK_LAUNCH("emph_pool_words_backward");
    return EMPH_OK;
}

int emph_output_head_backward(
    const float* x, const float* dz, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, int32_t kernel_size, const float* weight,
    float* dx, float* dw, float* db, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int s = emph::check_cuda(
        cudaMemsetAsync(dw, 0, sizeof(float) * kernel_size * channels, st), "memset head dw");
    if (s != EMPH_OK) return s;
    s = emph::check_cuda(cudaMemsetAsync(db, 0, sizeof(float), st), "memset head db");
    if (s != EMPH_OK) return s;
    if (total_rows == 0) return EMPH_OK;
    int grid = (int)(((size_t)total_rows * channels + 255) / 256);
    if (grid > emph::sm_count() * 4) grid = emph::sm_count() * 4;
    emph::head_backward_kernel<<<grid, 256, 0, st>>>(
        x, dz, row_seq, total_rows, channels, kernel_size, weight, dx, dw, db);
    emph::head_weight_grad_kernel<<<
        (total_rows + emph::kHeadGradRows - 1) / emph::kHeadGradRows, 256, 0, st>>>(
        x, dz, row_seq, total_rows, channels, kernel_size, dw, db);
    EMPH_CHECK_LAUNCH("emph_output_head_backward");
    return EMPH_OK;
}

int emph_masked_loss(
    const float* logits, const float* targets, const uint8_t* valid, int32_t total_rows,
    int32_t mode, float* loss, float* dlogits, void* stream) {
    EMPH_REQUIRE(mode == 0 || mode == 1, "emph_masked_loss: mode must be 0 (bce) or 1 (mse)");
    emph::masked_loss_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(
        logits, targets, valid, total_rows, mode, loss, dlogits);
    EMPH_CHECK_LAUNCH("emph_masked_loss");
    return EMPH_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// Word -> frame interpolation (emphases.upsample, emphases/core.py:472-544),
// used by the frame-resolution training loss of the 'inference' location.
// Operates on the reference's (B, C, W) / (B, C, T) layouts.  Faithful to two
// quirks: the 'linear' branch interpolates CHANNEL 0 for every channel
// (line_idx is all zeros, core.py:516-521) and a single-word item broadcasts
// x[0] (core.py:497-498).
namespace emph {

__global__ void upsample_words_kernel(
    const float* __restrict__ xs, const int64_t* __restrict__ bounds,
    const int64_t* __restrict__ word_lengths, const int64_t* __restrict__ frame_lengths,
    int batch, int channels, int wmax, int tmax, int linear, float* __restrict__ out) {
    const long long n = (long long)batch * channels * tmax;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % tmax);
        const int c = (int)((i / tmax) % channels);
        const int b = (int)(i / ((long long)tmax * channels));
        float value = 0.f;
        const int words = (int)word_lengths[b];
        if (t < (int)frame_lengths[b] && words > 0) {
            const float* x = xs + (size_t)b * channels * wmax;
            const int64_t* lo = bounds + (size_t)b * 2 * wmax;
            const int64_t* hi = lo + wmax;
            if (words == 1) {
                value = x[0];
            } else {
                const float ft = 0.5f + (float)t;
                int count = 0;
                for (int j = 0; j < words; ++j) {
                    const float wt = (float)lo[j] + (float)(hi[j] - lo[j]) / 2.f;
                    count += ft >= wt;
                }
                if (linear) {
                    const int idx = min(max(count - 1, 0), words - 2);
                    const float w0 = (float)lo[idx] + (float)(hi[idx] - lo[idx]) / 2.f;
                    const float w1 = (float)lo[idx + 1] + (float)(hi[idx + 1] - lo[idx + 1]) / 2.f;
                    const float slope = __fdiv_rn(x[idx + 1] - x[idx], w1 - w0);
                    const float intercept = __fsub_rn(x[idx], __fmul_rn(slope, w0));
                    value = __fadd_rn(__fmul_rn(slope, ft), intercept);
                } else {
                    const int idx = min(max(count - 1, 0), words - 1);
                    value = x[(size_t)c * wmax + idx];
                }
            }
        }
        out[i] = value;
    }
}

}  // namespace emph

extern "C" int emph_upsample_words(
    const float* xs, const int64_t* bounds, const int64_t* word_lengths,
    const int64_t* frame_lengths, int32_t batch, int32_t channels, int32_t wmax,
    int32_t tmax, int32_t linear, float* out, void* stream) {
    EMPH_REQUIRE(batch >= 0 && channels > 0 && wmax > 0 && tmax >= 0, "emph_upsample_words: bad shape");
    const long long n = (long long)batch * channels * tmax;
    if (n == 0) return EMPH_OK;
    long long blocks = (n + 255) / 256;
    if (blocks > emph::sm_count() * 8) blocks = emph::sm_count() * 8;
    emph::upsample_words_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        xs, bounds, word_lengths, frame_lengths, batch, channels, wmax, tmax, linear, out);
    EMPH_CHECK_LAUNCH("emph_upsample_words");
    return EMPH_OK;
}
