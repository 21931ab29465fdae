// Transformer-variant kernels over packed rows, fp32, sm_100a.
//
// Replace the pieces of emphases/model/layers/transformer.py:13-52
// (nn.TransformerEncoder of post-norm layers, d_model 80, 2 heads,
// dim_feedforward 80, key-padding mask from the sequence lengths) that are
// not plain per-row linear maps (those run through emph_conv_stack with
// kernel_size 1):
//   emph_add_positional   x + PE[:T]                      transformer.py:50-52
//   emph_attention_rows   softmax(Q K^T / sqrt(d) + key mask) V, per head
//   emph_add_layernorm    LayerNorm(x + residual), eps 1e-5
// and their training forms: emph_attention_rows_train (dropout on the
// probabilities, log-sum-exp kept), emph_attention_rows_backward,
// emph_add_layernorm_train (dropout on the residual branch, statistics kept),
// emph_add_layernorm_backward.
// In the packed layout the key-padding mask is "keys of the same sequence
// with index < n_keys[u]" -- block-diagonal attention with no padded FLOPs.
#include <math_constants.h>

#include "common.cuh"
#include "dropout.cuh"

namespace emph {

constexpr int kAttnThreads = 128;

// 2^x, x <= 0 here (ex2.approx: relative error 2^-22; exp2(-inf) = 0)
__device__ __forceinline__ float exp2_fast(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// 128 queries per CTA (the host cuts query blocks of that size): a lane PAIR owns two queries
constexpr int kAttnK = 64;     // keys per shared-memory tile

// Block-diagonal attention with online softmax, fp32.  Two lanes share two
// queries: lane h of the pair holds dims [h D/2, (h+1) D/2) of both queries'
// q and o vectors, so every 16-byte K / V shared-memory load (a broadcast: the
// 16 pairs of a warp read two addresses) feeds 8 FMAs instead of 4 and the
// partial dot products meet through one shuffle per query and key.  (One
// query per thread, the first version, was bound by the shared-memory pipe at
// 75 % with the FP32 pipe at 45 %, profiles/r01z_attention.md.)
// TRAIN: the training forward.  The probabilities are dropped after the
// normalisation is taken (dropout(softmax(S)) V, as torch), and the per-(row,
// head) log-sum-exp of the log2-domain scores, lse[row * heads + head] =
// max + log2(sum), is written for emph_attention_rows_backward.
template <int D, bool TRAIN>
__global__ void __launch_bounds__(kAttnThreads)
attention_rows_kernel(
    const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
    int channels, const int32_t* __restrict__ row_start, const int32_t* __restrict__ n_queries,
    const int32_t* __restrict__ n_keys,
    const int32_t* __restrict__ block_seq, const int32_t* __restrict__ block_q0,
    float scale, float* __restrict__ out, Dropout drop, float* __restrict__ lse) {
    constexpr int H = D / 2;                   // dims per lane
    static_assert(H % 4 == 0, "head dim must be a multiple of 8");
    __shared__ __align__(16) float ks[kAttnK][D];
    __shared__ __align__(16) float vs[kAttnK][D];
    const int u = block_seq[blockIdx.x];
    const int q0 = block_q0[blockIdx.x];
    const int head = blockIdx.y;
    const int base = row_start[u];
    const int nk = n_keys[u];
    const int nq = n_queries[u];
    const int half = threadIdx.x & 1;
    const int qa = q0 + 2 * (threadIdx.x >> 1), qb = qa + 1;
    const bool active_a = qa < nq, active_b = qb < nq;
    const size_t column = (size_t)head * D + half * H;

    // scores are kept in the log2 domain (log2 e folded into the query scale):
    // every exponential is then one MUFU.EX2
    scale *= 1.4426950408889634f;
    float qra[H], qrb[H], oa[H], ob[H];
#pragma unroll
    for (int d = 0; d < H; ++d) {
        qra[d] = active_a ? q[(size_t)(base + qa) * channels + column + d] * scale : 0.f;
        qrb[d] = active_b ? q[(size_t)(base + qb) * channels + column + d] * scale : 0.f;
        oa[d] = 0.f;
        ob[d] = 0.f;
    }
    float ma = -CUDART_INF_F, la = 0.f, mb = -CUDART_INF_F, lb = 0.f;
    const uint32_t site = drop.site | (uint32_t)head;
    const bool dropping = TRAIN && drop.threshold != 0ull;
    const unsigned long long index_a = (unsigned long long)(base + qa) << 16;
    const unsigned long long index_b = (unsigned long long)(base + qb) << 16;
    uint4 draws_a = make_uint4(0u, 0u, 0u, 0u), draws_b = draws_a;

    for (int kt = 0; kt < nk; kt += kAttnK) {
        const int count = min(kAttnK, nk - kt);
        __syncthreads();
        for (int i = threadIdx.x; i < count * (D / 4); i += kAttnThreads) {
            const int j = i / (D / 4), d4 = i % (D / 4);
            const size_t src = (size_t)(base + kt + j) * channels + (size_t)head * D + 4 * d4;
            *reinterpret_cast<float4*>(&ks[j][4 * d4]) = *reinterpret_cast<const float4*>(k + src);
            *reinterpret_cast<float4*>(&vs[j][4 * d4]) = *reinterpret_cast<const float4*>(v + src);
        }
        __syncthreads();
        // (inactive pairs run along: the shuffles below need every lane)
        for (int j = 0; j < count; ++j) {
            float sa = 0.f, sb = 0.f;
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 kk = *reinterpret_cast<const float4*>(&ks[j][half * H + 4 * d4]);
                sa = fmaf(qra[4 * d4], kk.x, sa);
                sa = fmaf(qra[4 * d4 + 1], kk.y, sa);
                sa = fmaf(qra[4 * d4 + 2], kk.z, sa);
                sa = fmaf(qra[4 * d4 + 3], kk.w, sa);
                sb = fmaf(qrb[4 * d4], kk.x, sb);
                sb = fmaf(qrb[4 * d4 + 1], kk.y, sb);
                sb = fmaf(qrb[4 * d4 + 2], kk.z, sb);
                sb = fmaf(qrb[4 * d4 + 3], kk.w, sb);
            }
            sa += __shfl_xor_sync(0xffffffffu, sa, 1);
            sb += __shfl_xor_sync(0xffffffffu, sb, 1);
            if (sa > ma) {                     // new running maximum: rescale
                const float correction = exp2_fast(ma - sa);
                la *= correction;
#pragma unroll
                for (int d = 0; d < H; ++d) oa[d] *= correction;
                ma = sa;
            }
            if (sb > mb) {
                const float correction = exp2_fast(mb - sb);
                lb *= correction;
#pragma unroll
                for (int d = 0; d < H; ++d) ob[d] *= correction;
                mb = sb;
            }
            float pa = exp2_fast(sa - ma), pb = exp2_fast(sb - mb);
            la += pa;
            lb += pb;
            if (dropping) {
                // keys kt + j; kt is a multiple of 4, so j & 3 starts a draw group
                const unsigned long long key = (unsigned long long)(kt + j);
                if ((j & 3) == 0) {
                    draws_a = philox_draws(drop.seed, site, (index_a | key) >> 2);
                    draws_b = philox_draws(drop.seed, site, (index_b | key) >> 2);
                }
                pa *= dropout_factor(drop, draws_a, key);
                pb *= dropout_factor(drop, draws_b, key);
            }
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 vv = *reinterpret_cast<const float4*>(&vs[j][half * H + 4 * d4]);
                oa[4 * d4] = fmaf(pa, vv.x, oa[4 * d4]);
                oa[4 * d4 + 1] = fmaf(pa, vv.y, oa[4 * d4 + 1]);
                oa[4 * d4 + 2] = fmaf(pa, vv.z, oa[4 * d4 + 2]);
                oa[4 * d4 + 3] = fmaf(pa, vv.w, oa[4 * d4 + 3]);
                ob[4 * d4] = fmaf(pb, vv.x, ob[4 * d4]);
                ob[4 * d4 + 1] = fmaf(pb, vv.y, ob[4 * d4 + 1]);
                ob[4 * d4 + 2] = fmaf(pb, vv.z, ob[4 * d4 + 2]);
                ob[4 * d4 + 3] = fmaf(pb, vv.w, ob[4 * d4 + 3]);
            }
        }
    }
    if (active_a) {
        const float inv = 1.f / la;
        float* dst = out + (size_t)(base + qa) * channels + column;
#pragma unroll
        for (int d = 0; d < H; ++d) dst[d] = oa[d] * inv;
        if (TRAIN && half == 0) lse[(size_t)(base + qa) * gridDim.y + head] = ma + log2f(la);
    }
    if (active_b) {
        const float inv = 1.f / lb;
        float* dst = out + (size_t)(base + qb) * channels + column;
#pragma unroll
        for (int d = 0; d < H; ++d) dst[d] = ob[d] * inv;
        if (TRAIN && half == 0) lse[(size_t)(base + qb) * gridDim.y + head] = mb + log2f(lb);
    }
}

// separator rows are zero
__global__ void attention_clear_kernel(
    const int32_t* __restrict__ row_seq, int total_rows, int channels, float* __restrict__ out) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= total_rows) return;
    if (row_seq[r] >= 0) return;
    for (int c = threadIdx.x & 31; c < channels; c += 32) out[(size_t)r * channels + c] = 0.f;
}

__global__ void add_positional_kernel(
    const float* __restrict__ x, const int32_t* __restrict__ row_start,
    const int32_t* __restrict__ row_seq, int total_rows, int channels,
    const float* __restrict__ table, int table_rows, float* __restrict__ y) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= total_rows) return;
    const int u = row_seq[r];
    for (int c = threadIdx.x & 31; c < channels; c += 32) {
        float value = 0.f;
        if (u >= 0) {
            const int t = r - row_start[u];
            value = x[(size_t)r * channels + c] +
                    (t < table_rows ? table[(size_t)t * channels + c] : 0.f);
        }
        y[(size_t)r * channels + c] = value;
    }
}

// y = LayerNorm(x + residual) * gamma + beta, one warp per row.
// TRAIN: y = LayerNorm(x + dropout(residual)), and the pre-norm sum s = x +
// dropout(residual) and (mean, rstd) per row are kept for the backward
template <bool TRAIN>
__global__ void add_layernorm_kernel(
    const float* __restrict__ x, const float* __restrict__ residual,
    const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
    const int32_t* __restrict__ row_seq, int total_rows, int channels, float* __restrict__ y,
    Dropout drop, float* __restrict__ sum_out, float* __restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= total_rows) return;
    if (row_seq[r] < 0) {
        for (int c = lane; c < channels; c += 32) {
            y[(size_t)r * channels + c] = 0.f;
            if (TRAIN) sum_out[(size_t)r * channels + c] = 0.f;
        }
        if (TRAIN && lane < 2) stats[2 * (size_t)r + lane] = 0.f;
        return;
    }
    float values[4];                                // channels <= 128
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = lane + 32 * i;
        float branch = c < channels ? residual[(size_t)r * channels + c] : 0.f;
        if (TRAIN && c < channels)
            branch *= dropout_keep(drop, drop.site, (unsigned long long)r * channels + c)
                ? drop.scale : 0.f;
        values[i] = c < channels ? x[(size_t)r * channels + c] + branch : 0.f;
        if (TRAIN && c < channels) sum_out[(size_t)r * channels + c] = values[i];
        sum += values[i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / (float)channels;
    float square = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = lane + 32 * i;
        const float d = c < channels ? values[i] - mean : 0.f;
        square = fmaf(d, d, square);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) square += __shfl_xor_sync(0xffffffffu, square, o);
    const float inv = rsqrtf(square / (float)channels + eps);
    if (TRAIN && lane < 2) stats[2 * (size_t)r + lane] = lane == 0 ? mean : inv;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = lane + 32 * i;
        if (c < channels)
            y[(size_t)r * channels + c] = (values[i] - mean) * inv * gamma[c] + beta[c];
    }
}

// ---------------------------------------------------------------------------
// Training backward (FlashAttention-2 form, fp32 CUDA cores).  S and P are
// recomputed per tile from q, k and the forward's log-sum-exp, the dropout
// mask is regenerated from the seed, and no T x T tensor reaches HBM:
//   P = exp2(S2 - lse),  Pd = P * keep / (1 - p),  D_i = sum_d dO_i O_i
//   dV_j = sum_i Pd_ij dO_i,  dS_ij = P_ij (keep_ij / (1 - p) dO_i . v_j - D_i)
//   dK_j = scale sum_i dS_ij q_i,  dQ_i = scale sum_j dS_ij k_j
// Two passes, each writing its rows once (no float atomics, deterministic):
// one over 64-key blocks for dK / dV, one over 64-query blocks for dQ.  A lane
// pair owns one key (one query) and half of its head dims.
// ---------------------------------------------------------------------------
constexpr int kBwdRows = 64;        // keys / queries per CTA and per tile

template <int D>
__global__ void __launch_bounds__(kAttnThreads)
attention_backward_kv_kernel(
    const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
    const float* __restrict__ o, const float* __restrict__ d_o, const float* __restrict__ lse,
    int channels, const int32_t* __restrict__ row_start, const int32_t* __restrict__ n_queries,
    const int32_t* __restrict__ n_keys, const int32_t* __restrict__ block_seq,
    const int32_t* __restrict__ block_k0, float scale, Dropout drop,
    float* __restrict__ dk, float* __restrict__ dv) {
    constexpr int H = D / 2;
    __shared__ __align__(16) float qs[kBwdRows][D];
    __shared__ __align__(16) float dos[kBwdRows][D];
    __shared__ float lses[kBwdRows], deltas[kBwdRows];
    const int u = block_seq[blockIdx.x];
    const int head = blockIdx.y, heads = gridDim.y;
    const int base = row_start[u];
    const int nk = n_keys[u], nq = n_queries[u];
    const int half = threadIdx.x & 1;
    const int j = block_k0[blockIdx.x] + (threadIdx.x >> 1);
    const bool active = j < nk;
    const size_t column = (size_t)head * D + half * H;
    const uint32_t site = drop.site | (uint32_t)head;
    const float scale2 = scale * 1.4426950408889634f;     // log2-domain scores

    float kr[H], vr[H], dkr[H], dvr[H];
#pragma unroll
    for (int d = 0; d < H; ++d) {
        kr[d] = active ? k[(size_t)(base + j) * channels + column + d] * scale2 : 0.f;
        vr[d] = active ? v[(size_t)(base + j) * channels + column + d] : 0.f;
        dkr[d] = 0.f;
        dvr[d] = 0.f;
    }
    for (int i0 = 0; i0 < nq; i0 += kBwdRows) {
        const int count = min(kBwdRows, nq - i0);
        __syncthreads();
        for (int e = threadIdx.x; e < count * (D / 4); e += kAttnThreads) {
            const int i = e / (D / 4), d4 = e % (D / 4);
            const size_t src = (size_t)(base + i0 + i) * channels + (size_t)head * D + 4 * d4;
            *reinterpret_cast<float4*>(&qs[i][4 * d4]) = *reinterpret_cast<const float4*>(q + src);
            *reinterpret_cast<float4*>(&dos[i][4 * d4]) = *reinterpret_cast<const float4*>(d_o + src);
        }
        // D_i = dO_i . O_i over the head: one warp per query
        for (int i = threadIdx.x >> 5; i < count; i += kAttnThreads / 32) {
            const size_t row = (size_t)(base + i0 + i) * channels + (size_t)head * D;
            float acc = 0.f;
            for (int d = threadIdx.x & 31; d < D; d += 32) acc = fmaf(d_o[row + d], o[row + d], acc);
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
            if ((threadIdx.x & 31) == 0) {
                deltas[i] = acc;
                lses[i] = lse[(size_t)(base + i0 + i) * heads + head];
            }
        }
        __syncthreads();
        for (int i = 0; i < count; ++i) {
            float s = 0.f, dp = 0.f;
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 qq = *reinterpret_cast<const float4*>(&qs[i][half * H + 4 * d4]);
                const float4 gg = *reinterpret_cast<const float4*>(&dos[i][half * H + 4 * d4]);
                s = fmaf(qq.x, kr[4 * d4], s);
                s = fmaf(qq.y, kr[4 * d4 + 1], s);
                s = fmaf(qq.z, kr[4 * d4 + 2], s);
                s = fmaf(qq.w, kr[4 * d4 + 3], s);
                dp = fmaf(gg.x, vr[4 * d4], dp);
                dp = fmaf(gg.y, vr[4 * d4 + 1], dp);
                dp = fmaf(gg.z, vr[4 * d4 + 2], dp);
                dp = fmaf(gg.w, vr[4 * d4 + 3], dp);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            dp += __shfl_xor_sync(0xffffffffu, dp, 1);
            const float p = exp2_fast(s - lses[i]);
            float factor = 1.f;
            if (drop.threshold != 0ull)
                factor = dropout_keep(
                    drop, site, ((unsigned long long)(base + i0 + i) << 16) | (unsigned)j)
                    ? drop.scale : 0.f;
            const float pd = p * factor;
            const float ds = p * fmaf(dp, factor, -deltas[i]);
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 qq = *reinterpret_cast<const float4*>(&qs[i][half * H + 4 * d4]);
                const float4 gg = *reinterpret_cast<const float4*>(&dos[i][half * H + 4 * d4]);
                dvr[4 * d4] = fmaf(pd, gg.x, dvr[4 * d4]);
                dvr[4 * d4 + 1] = fmaf(pd, gg.y, dvr[4 * d4 + 1]);
                dvr[4 * d4 + 2] = fmaf(pd, gg.z, dvr[4 * d4 + 2]);
                dvr[4 * d4 + 3] = fmaf(pd, gg.w, dvr[4 * d4 + 3]);
                dkr[4 * d4] = fmaf(ds, qq.x, dkr[4 * d4]);
                dkr[4 * d4 + 1] = fmaf(ds, qq.y, dkr[4 * d4 + 1]);
                dkr[4 * d4 + 2] = fmaf(ds, qq.z, dkr[4 * d4 + 2]);
                dkr[4 * d4 + 3] = fmaf(ds, qq.w, dkr[4 * d4 + 3]);
            }
        }
    }
    if (active) {
        const size_t row = (size_t)(base + j) * channels + column;
#pragma unroll
        for (int d = 0; d < H; ++d) {
            dk[row + d] = dkr[d] * scale;
            dv[row + d] = dvr[d];
        }
    }
}

template <int D>
__global__ void __launch_bounds__(kAttnThreads)
attention_backward_q_kernel(
    const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
    const float* __restrict__ o, const float* __restrict__ d_o, const float* __restrict__ lse,
    int channels, const int32_t* __restrict__ row_start, const int32_t* __restrict__ n_queries,
    const int32_t* __restrict__ n_keys, const int32_t* __restrict__ block_seq,
    const int32_t* __restrict__ block_q0, float scale, Dropout drop,
    float* __restrict__ dq, float* __restrict__ dk, float* __restrict__ dv) {
    constexpr int H = D / 2;
    __shared__ __align__(16) float ks[kBwdRows][D];
    __shared__ __align__(16) float vs[kBwdRows][D];
    const int u = block_seq[blockIdx.x];
    const int head = blockIdx.y, heads = gridDim.y;
    const int base = row_start[u];
    const int nk = n_keys[u], nq = n_queries[u];
    const int half = threadIdx.x & 1;
    const int i = block_q0[blockIdx.x] + (threadIdx.x >> 1);
    const bool active = i < nq;
    const size_t column = (size_t)head * D + half * H;
    const size_t row = (size_t)(base + i) * channels + column;
    const uint32_t site = drop.site | (uint32_t)head;
    const float scale2 = scale * 1.4426950408889634f;

    float qr[H], gr[H], dqr[H];
    float delta = 0.f;
#pragma unroll
    for (int d = 0; d < H; ++d) {
        qr[d] = active ? q[row + d] * scale2 : 0.f;
        gr[d] = active ? d_o[row + d] : 0.f;
        delta = fmaf(gr[d], active ? o[row + d] : 0.f, delta);
        dqr[d] = 0.f;
    }
    delta += __shfl_xor_sync(0xffffffffu, delta, 1);
    const float lse_i = active ? lse[(size_t)(base + i) * heads + head] : 0.f;
    const unsigned long long index = (unsigned long long)(base + i) << 16;
    uint4 draws = make_uint4(0u, 0u, 0u, 0u);

    for (int kt = 0; kt < nk; kt += kBwdRows) {
        const int count = min(kBwdRows, nk - kt);
        __syncthreads();
        for (int e = threadIdx.x; e < count * (D / 4); e += kAttnThreads) {
            const int jj = e / (D / 4), d4 = e % (D / 4);
            const size_t src = (size_t)(base + kt + jj) * channels + (size_t)head * D + 4 * d4;
            *reinterpret_cast<float4*>(&ks[jj][4 * d4]) = *reinterpret_cast<const float4*>(k + src);
            *reinterpret_cast<float4*>(&vs[jj][4 * d4]) = *reinterpret_cast<const float4*>(v + src);
        }
        __syncthreads();
        for (int jj = 0; jj < count; ++jj) {
            float s = 0.f, dp = 0.f;
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 kk = *reinterpret_cast<const float4*>(&ks[jj][half * H + 4 * d4]);
                const float4 vv = *reinterpret_cast<const float4*>(&vs[jj][half * H + 4 * d4]);
                s = fmaf(qr[4 * d4], kk.x, s);
                s = fmaf(qr[4 * d4 + 1], kk.y, s);
                s = fmaf(qr[4 * d4 + 2], kk.z, s);
                s = fmaf(qr[4 * d4 + 3], kk.w, s);
                dp = fmaf(gr[4 * d4], vv.x, dp);
                dp = fmaf(gr[4 * d4 + 1], vv.y, dp);
                dp = fmaf(gr[4 * d4 + 2], vv.z, dp);
                dp = fmaf(gr[4 * d4 + 3], vv.w, dp);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            dp += __shfl_xor_sync(0xffffffffu, dp, 1);
            const float p = exp2_fast(s - lse_i);
            float factor = 1.f;
            if (drop.threshold != 0ull) {
                const unsigned long long key = (unsigned long long)(kt + jj);
                if ((jj & 3) == 0) draws = philox_draws(drop.seed, site, (index | key) >> 2);
                factor = dropout_factor(drop, draws, key);
            }
            const float ds = p * fmaf(dp, factor, -delta);
#pragma unroll
            for (int d4 = 0; d4 < H / 4; ++d4) {
                const float4 kk = *reinterpret_cast<const float4*>(&ks[jj][half * H + 4 * d4]);
                dqr[4 * d4] = fmaf(ds, kk.x, dqr[4 * d4]);
                dqr[4 * d4 + 1] = fmaf(ds, kk.y, dqr[4 * d4 + 1]);
                dqr[4 * d4 + 2] = fmaf(ds, kk.z, dqr[4 * d4 + 2]);
                dqr[4 * d4 + 3] = fmaf(ds, kk.w, dqr[4 * d4 + 3]);
            }
        }
    }
    if (active) {
        if (nk == 0) {
            // no valid key: the forward's softmax is NaN, and so is every
            // gradient through it (as torch's masked softmax backward)
#pragma unroll
            for (int d = 0; d < H; ++d) {
                dq[row + d] = CUDART_NAN_F;
                dk[row + d] = CUDART_NAN_F;
                dv[row + d] = CUDART_NAN_F;
            }
        } else {
#pragma unroll
            for (int d = 0; d < H; ++d) dq[row + d] = dqr[d] * scale;
        }
    }
}

// LayerNorm(x + dropout(b)) backward, one warp per row (grid-stride): ds =
// rstd (g - mean(g) - xhat mean(g xhat)), g = dy gamma, written as dx (the
// residual input's gradient) and d_branch = ds * keep / (1 - p).  Each CTA
// adds its rows' dy xhat and dy into a partial row of `partials`
// [gridDim.x][2 C]; layernorm_reduce_kernel sums the partials in CTA order.
__global__ void __launch_bounds__(256)
layernorm_backward_kernel(
    const float* __restrict__ dy, const float* __restrict__ sums, const float* __restrict__ stats,
    const float* __restrict__ gamma, const int32_t* __restrict__ row_seq, int total_rows,
    int channels, Dropout drop, float* __restrict__ dx, float* __restrict__ d_branch,
    float* __restrict__ partials) {
    __shared__ float warp_sums[8][2][128];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float dgamma[4] = {0.f, 0.f, 0.f, 0.f}, dbeta[4] = {0.f, 0.f, 0.f, 0.f};
    for (int r = blockIdx.x * 8 + warp; r < total_rows; r += gridDim.x * 8) {
        const size_t at = (size_t)r * channels;
        if (row_seq[r] < 0) {
            for (int c = lane; c < channels; c += 32) {
                dx[at + c] = 0.f;
                d_branch[at + c] = 0.f;
            }
            continue;
        }
        const float mean = stats[2 * (size_t)r], rstd = stats[2 * (size_t)r + 1];
        float xhat[4], g[4], sum_g = 0.f, sum_gx = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = lane + 32 * i;
            xhat[i] = c < channels ? (sums[at + c] - mean) * rstd : 0.f;
            const float grad = c < channels ? dy[at + c] : 0.f;
            g[i] = c < channels ? grad * gamma[c] : 0.f;
            dgamma[i] = fmaf(grad, xhat[i], dgamma[i]);
            dbeta[i] += grad;
            sum_g += g[i];
            sum_gx = fmaf(g[i], xhat[i], sum_gx);
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) {
            sum_g += __shfl_xor_sync(0xffffffffu, sum_g, m);
            sum_gx += __shfl_xor_sync(0xffffffffu, sum_gx, m);
        }
        const float mean_g = sum_g / (float)channels, mean_gx = sum_gx / (float)channels;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = lane + 32 * i;
            if (c >= channels) continue;
            const float ds = rstd * (g[i] - mean_g - xhat[i] * mean_gx);
            dx[at + c] = ds;
            d_branch[at + c] =
                dropout_keep(drop, drop.site, (unsigned long long)at + c) ? ds * drop.scale : 0.f;
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        warp_sums[warp][0][lane + 32 * i] = dgamma[i];
        warp_sums[warp][1][lane + 32 * i] = dbeta[i];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 2 * channels; e += 256) {
        const int which = e / channels, c = e % channels;
        float total = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) total += warp_sums[w][which][c];
        partials[(size_t)blockIdx.x * 2 * channels + e] = total;
    }
}

// dgamma, dbeta = the column sums of `partials` [blocks][2 C], in block order
__global__ void layernorm_reduce_kernel(
    const float* __restrict__ partials, int blocks, int channels, float* __restrict__ dgamma,
    float* __restrict__ dbeta) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 2 * channels) return;
    float total = 0.f;
    for (int b = 0; b < blocks; ++b) total += partials[(size_t)b * 2 * channels + e];
    if (e < channels) dgamma[e] = total;
    else dbeta[e - channels] = total;
}

}  // namespace emph

extern "C" {

int emph_add_positional(
    const float* x, const int32_t* row_start, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, const float* table, int32_t table_rows, float* y, void* stream) {
    EMPH_REQUIRE(total_rows >= 0 && channels > 0, "emph_add_positional: bad size");
    if (total_rows == 0) return EMPH_OK;
    emph::add_positional_kernel<<<(total_rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(
        x, row_start, row_seq, total_rows, channels, table, table_rows, y);
    EMPH_CHECK_LAUNCH("emph_add_positional");
    return EMPH_OK;
}

int emph_attention_rows(
    const float* q, const float* k, const float* v, int32_t channels, int32_t heads,
    const int32_t* row_start, const int32_t* n_queries, const int32_t* n_keys,
    const int32_t* row_seq, int32_t total_rows,
    const int32_t* block_seq, const int32_t* block_q0, int32_t n_blocks,
    float scale, float* out, void* stream) {
    EMPH_REQUIRE(heads > 0 && channels % heads == 0, "emph_attention_rows: bad head count");
    const int head_dim = channels / heads;
    if (total_rows == 0) return EMPH_OK;
    cudaStream_t st = (cudaStream_t)stream;
    emph::attention_clear_kernel<<<(total_rows + 7) / 8, 256, 0, st>>>(
        row_seq, total_rows, channels, out);
    EMPH_CHECK_LAUNCH("emph_attention_rows(clear)");
    if (n_blocks == 0) return EMPH_OK;
    dim3 grid(n_blocks, heads);
    if (head_dim == 40) {
        emph::attention_rows_kernel<40, false><<<grid, emph::kAttnThreads, 0, st>>>(
            q, k, v, channels, row_start, n_queries, n_keys, block_seq, block_q0, scale, out,
            emph::Dropout{}, nullptr);
    } else if (head_dim == 32) {
        emph::attention_rows_kernel<32, false><<<grid, emph::kAttnThreads, 0, st>>>(
            q, k, v, channels, row_start, n_queries, n_keys, block_seq, block_q0, scale, out,
            emph::Dropout{}, nullptr);
    } else if (head_dim == 64) {
        emph::attention_rows_kernel<64, false><<<grid, emph::kAttnThreads, 0, st>>>(
            q, k, v, channels, row_start, n_queries, n_keys, block_seq, block_q0, scale, out,
            emph::Dropout{}, nullptr);
    } else {
        emph::set_error("emph_attention_rows: head_dim %d not compiled in", head_dim);
        return EMPH_ENOSYS;
    }
    EMPH_CHECK_LAUNCH("emph_attention_rows");
    return EMPH_OK;
}

int emph_add_layernorm(
    const float* x, const float* residual, const float* gamma, const float* beta, float eps,
    const int32_t* row_seq, int32_t total_rows, int32_t channels, float* y, void* stream) {
    EMPH_REQUIRE(channels > 0 && channels <= 128, "emph_add_layernorm: channels %d > 128", channels);
    if (total_rows == 0) return EMPH_OK;
    emph::add_layernorm_kernel<false><<<(total_rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(
        x, residual, gamma, beta, eps, row_seq, total_rows, channels, y, emph::Dropout{},
        nullptr, nullptr);
    EMPH_CHECK_LAUNCH("emph_add_layernorm");
    return EMPH_OK;
}

int emph_attention_rows_train(
    const float* q, const float* k, const float* v, int32_t channels, int32_t heads,
    const int32_t* row_start, const int32_t* n_queries, const int32_t* n_keys,
    const int32_t* row_seq, int32_t total_rows,
    const int32_t* block_seq, const int32_t* block_q0, int32_t n_blocks,
    float scale, uint64_t seed, uint32_t site, float p, float* out, float* lse, void* stream) {
    EMPH_REQUIRE(heads > 0 && channels == 40 * heads,
                 "emph_attention_rows_train: built for 40-dim heads (channels %d, heads %d)",
                 channels, heads);
    EMPH_REQUIRE(p >= 0.f && p <= 1.f, "emph_attention_rows_train: p = %f", p);
    if (total_rows == 0) return EMPH_OK;
    cudaStream_t st = (cudaStream_t)stream;
    emph::attention_clear_kernel<<<(total_rows + 7) / 8, 256, 0, st>>>(
        row_seq, total_rows, channels, out);
    EMPH_CHECK_LAUNCH("emph_attention_rows_train(clear)");
    int s = emph::check_cuda(
        cudaMemsetAsync(lse, 0, sizeof(float) * (size_t)total_rows * heads, st), "memset lse");
    if (s != EMPH_OK) return s;
    if (n_blocks == 0) return EMPH_OK;
    emph::attention_rows_kernel<40, true><<<dim3(n_blocks, heads), emph::kAttnThreads, 0, st>>>(
        q, k, v, channels, row_start, n_queries, n_keys, block_seq, block_q0, scale, out,
        emph::make_dropout(seed, site, p), lse);
    EMPH_CHECK_LAUNCH("emph_attention_rows_train");
    return EMPH_OK;
}

int emph_attention_rows_backward(
    const float* q, const float* k, const float* v, const float* o, const float* d_o,
    const float* lse, int32_t channels, int32_t heads, const int32_t* row_start,
    const int32_t* n_queries, const int32_t* n_keys, int32_t total_rows,
    const int32_t* key_block_seq, const int32_t* key_block_k0, int32_t n_key_blocks,
    const int32_t* query_block_seq, const int32_t* query_block_q0, int32_t n_query_blocks,
    float scale, uint64_t seed, uint32_t site, float p, float* dq, float* dk, float* dv,
    void* stream) {
    EMPH_REQUIRE(heads > 0 && channels == 40 * heads,
                 "emph_attention_rows_backward: built for 40-dim heads (channels %d, heads %d)",
                 channels, heads);
    EMPH_REQUIRE(p >= 0.f && p <= 1.f, "emph_attention_rows_backward: p = %f", p);
    if (total_rows == 0) return EMPH_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = sizeof(float) * (size_t)total_rows * channels;
    // rows that are no query / no key (separators, padded keys) keep a zero gradient
    int s = emph::check_cuda(cudaMemsetAsync(dq, 0, bytes, st), "memset dq");
    if (s == EMPH_OK) s = emph::check_cuda(cudaMemsetAsync(dk, 0, bytes, st), "memset dk");
    if (s == EMPH_OK) s = emph::check_cuda(cudaMemsetAsync(dv, 0, bytes, st), "memset dv");
    if (s != EMPH_OK) return s;
    const emph::Dropout drop = emph::make_dropout(seed, site, p);
    if (n_key_blocks > 0) {
        emph::attention_backward_kv_kernel<40>
            <<<dim3(n_key_blocks, heads), emph::kAttnThreads, 0, st>>>(
            q, k, v, o, d_o, lse, channels, row_start, n_queries, n_keys, key_block_seq,
            key_block_k0, scale, drop, dk, dv);
        EMPH_CHECK_LAUNCH("emph_attention_rows_backward(dk, dv)");
    }
    if (n_query_blocks > 0) {
        emph::attention_backward_q_kernel<40>
            <<<dim3(n_query_blocks, heads), emph::kAttnThreads, 0, st>>>(
            q, k, v, o, d_o, lse, channels, row_start, n_queries, n_keys, query_block_seq,
            query_block_q0, scale, drop, dq, dk, dv);
        EMPH_CHECK_LAUNCH("emph_attention_rows_backward(dq)");
    }
    return EMPH_OK;
}

int emph_add_layernorm_train(
    const float* x, const float* residual, const float* gamma, const float* beta, float eps,
    const int32_t* row_seq, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site,
    float p, float* y, float* sums, float* stats, void* stream) {
    EMPH_REQUIRE(channels > 0 && channels <= 128,
                 "emph_add_layernorm_train: channels %d > 128", channels);
    EMPH_REQUIRE(p >= 0.f && p <= 1.f, "emph_add_layernorm_train: p = %f", p);
    if (total_rows == 0) return EMPH_OK;
    emph::add_layernorm_kernel<true><<<(total_rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(
        x, residual, gamma, beta, eps, row_seq, total_rows, channels, y,
        emph::make_dropout(seed, site, p), sums, stats);
    EMPH_CHECK_LAUNCH("emph_add_layernorm_train");
    return EMPH_OK;
}

int emph_layernorm_backward_blocks(int32_t total_rows) {
    const int blocks = (total_rows + 7) / 8;
    const int cap = emph::sm_count() * 4;
    return blocks < 1 ? 1 : (blocks > cap ? cap : blocks);
}

int emph_add_layernorm_backward(
    const float* dy, const float* sums, const float* stats, const float* gamma,
    const int32_t* row_seq, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site,
    float p, float* dx, float* d_branch, float* dgamma, float* dbeta, float* partials,
    void* stream) {
    EMPH_REQUIRE(channels > 0 && channels <= 128,
                 "emph_add_layernorm_backward: channels %d > 128", channels);
    EMPH_REQUIRE(p >= 0.f && p <= 1.f, "emph_add_layernorm_backward: p = %f", p);
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = emph_layernorm_backward_blocks(total_rows);
    emph::layernorm_backward_kernel<<<blocks, 256, 0, st>>>(
        dy, sums, stats, gamma, row_seq, total_rows, channels,
        emph::make_dropout(seed, site, p), dx, d_branch, partials);
    EMPH_CHECK_LAUNCH("emph_add_layernorm_backward");
    emph::layernorm_reduce_kernel<<<(2 * channels + 127) / 128, 128, 0, st>>>(
        partials, blocks, channels, dgamma, dbeta);
    EMPH_CHECK_LAUNCH("emph_add_layernorm_backward(reduce)");
    return EMPH_OK;
}

}  // extern "C"
