// Training-mode forward and backward of the convolution model, each as ONE
// native call (BASELINE config 5; emphases/train/core.py:86-142 runs
// model(...) / loss / backward under autograd).  The layer loops, the weight
// re-packing (the parameters change every step) and every intermediate buffer
// live here: the host issues two C-ABI calls per step instead of ~100, all
// activations sit in one caller-provided workspace, and the parameter
// gradients are written in the Conv1d (out, in, k) layout straight into a flat
// buffer the data-parallel all-reduce runs on in place.
//
// The convolutions run through emph_conv_stack one layer at a time (so every
// layer's output is kept for the backward pass) in `precision`: the fp32 FFMA
// kernel, or the split-bf16 tensor-core kernel (bf16x3 / bf16x6, fp32-grade)
// for the forward and the input-gradient passes.  Weight gradients run on the
// split-bf16 mma.sync kernel in every mode (16-bit operands, fp32 accumulate).
//
// Dropout (the reference's Conv1d -> activation -> Dropout blocks): a layer
// with p > 0 runs emph_conv_dropout_forward after its convolution, in place on
// the activated output (ReLU / LeakyReLU / identity) or in place of
// emph_activation_forward (GELU / SiLU, whose pre-activation stays kept).  Its
// output buffer then holds the dropped values that pooling and the next layer
// read, and the backward uses emph_activation_dropout_backward, which
// regenerates the mask from the seed: nothing else is stored, and the
// backward launches no extra kernel.
#include <vector>

#include "common.cuh"

namespace emph {

int pack_conv1d_weights_tc(
    const float* conv_weight, const float* bias, int kernel_size, int precision, int adjoint,
    void* packed, cudaStream_t stream);
size_t conv1d_blob_bytes(int kernel_size, int precision);
int pack_conv1d_weights_tc_batch(
    const float* const* conv_weights, const float* const* biases, int n, int kernel_size,
    int precision, int adjoint, void* packed, size_t stride, cudaStream_t stream);
int conv1d_weight_grad(
    const float* x, const float* dpre, int total_rows, int channels, int kernel_size,
    float* grad_weight, float* grad_bias, int accumulate, cudaStream_t st);

constexpr int kTrainChannels = 80;
constexpr int kTrainKernel = 3;

__global__ void scatter_rows_kernel(
    const float* __restrict__ src, const int32_t* __restrict__ index, int count,
    float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[index[i]] = src[i];
}
__global__ void gather_rows_kernel(
    const float* __restrict__ src, const int32_t* __restrict__ index, int count,
    float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = src[index[i]];
}
__global__ void vector_store_kernel(
    const float* __restrict__ src, int count, int accumulate, float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = accumulate ? dst[i] + src[i] : src[i];
}
// head dw [k][c] -> Conv1d (1, c, k)
__global__ void head_grad_layout_kernel(
    const float* __restrict__ dw, int channels, int kernel, int accumulate,
    float* __restrict__ grad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < channels * kernel) {
        const int k = i % kernel, c = i / kernel;
        const float v = dw[k * channels + c];
        grad[i] = accumulate ? grad[i] + v : v;
    }
}
// logit = head(x) with the bias read from device memory (a parameter)
__global__ void add_bias_kernel(
    float* __restrict__ logits, const int32_t* __restrict__ row_seq, int rows,
    const float* __restrict__ bias) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rows && row_seq[i] >= 0) logits[i] += bias[0];
}

static size_t up(size_t bytes) { return (bytes + 255) / 256 * 256; }

// Everything the two calls share: where each buffer sits in the workspace
struct TrainLayout {
    int batch, frames, wmax, total, total_words, n_frame, n_word;
    // int32 index arrays (one host-built blob)
    size_t blob, blob_words;
    size_t row_start, n_rows, word_row_start, n_words, word_seq, word_lo, word_hi, index;
    size_t row_seq, word_row_seq;
    // activations
    size_t rows;                       // packed features
    std::vector<size_t> frame_out, frame_pre, word_out, word_pre;
    size_t pooled, logits_rows;
    // per-call scratch
    size_t packed_w, adjoint_w, tc_w, tc_stride, dw, db, dz, grad_a, grad_b, head_w, head_dw, head_db;
    size_t total_bytes;
};

static bool keeps_pre(int act) { return act == EMPH_ACT_GELU || act == EMPH_ACT_SILU; }

// p of the dropout after layer `index` (0: none; the input layer has none)
static float dropout_p(const emph_train_model& m, int index) {
    return m.dropout && index > 0 ? m.dropout[index] : 0.f;
}

// dropout site of layer `index`: frame encoder block index - 1, word decoder
// block index - n_frame_layers
static uint32_t dropout_site(const emph_train_model& m, int index) {
    const bool word = index >= m.n_frame_layers;
    return EMPH_DROPOUT_SITE(word ? 1 : 0, word ? index - m.n_frame_layers : index - 1,
                             EMPH_DROPOUT_CONV, 0);
}

// Rows kept per item.  The reference convolves all `frames` padded columns of
// every item (emphases/model/layers/convolution.py:36-37 ignores the lengths),
// and the value of the last frame layer at row t depends on layer-i rows up to
// t + (layers - 1 - i): with `lengths` at least one past the last frame any
// word reads (the caller's duty: a word may end past the audio), rows beyond
// length + n_frame_layers * (k - 1) / 2 cannot reach the loss or any
// gradient, so they are not computed (the rows words read are bit-identical).
static int kept_rows(const emph_train_model& m, int frames, const int64_t* lengths, int b) {
    if (!lengths) return frames;
    const long long reach = lengths[b] + (long long)m.n_frame_layers * ((kTrainKernel - 1) / 2);
    return (int)(reach < frames ? (reach < 1 ? 1 : reach) : frames);
}

// Separator rows between the word rows of two items: the output projection
// (kernel up to 7) reads (head_kernel - 1) / 2 rows on each side of a word, and
// must see zeros there, not the next item's words (a word decoder layer, k = 3,
// needs one)
static int word_gap(const emph_train_model& m) {
    const int half = (m.head_kernel - 1) / 2;
    return half > 1 ? half : 1;
}

static TrainLayout make_layout(
    const emph_train_model& m, int batch, int frames, int wmax, const int64_t* lengths) {
    TrainLayout l;
    l.batch = batch; l.frames = frames; l.wmax = wmax;
    l.total = 1;
    for (int b = 0; b < batch; ++b) l.total += kept_rows(m, frames, lengths, b) + 1;
    l.total_words = batch * (wmax + word_gap(m)) + word_gap(m);
    l.n_frame = m.n_frame_layers; l.n_word = m.n_word_layers;
    size_t cursor = 0;
    auto take = [&](size_t bytes) { size_t at = cursor; cursor += up(bytes); return at; };
    l.blob_words = 4 * (size_t)batch + 3 * (size_t)l.total_words + (size_t)batch * wmax;
    l.blob = take(4 * l.blob_words);
    size_t w = l.blob;
    l.row_start = w; w += 4 * (size_t)batch;
    l.n_rows = w; w += 4 * (size_t)batch;
    l.word_row_start = w; w += 4 * (size_t)batch;
    l.n_words = w; w += 4 * (size_t)batch;
    l.word_seq = w; w += 4 * (size_t)l.total_words;
    l.word_lo = w; w += 4 * (size_t)l.total_words;
    l.word_hi = w; w += 4 * (size_t)l.total_words;
    l.index = w;
    l.row_seq = take(4 * (size_t)l.total);
    l.word_row_seq = take(4 * (size_t)l.total_words);
    const size_t frame_bytes = sizeof(float) * (size_t)l.total * kTrainChannels;
    const size_t word_bytes = sizeof(float) * (size_t)l.total_words * kTrainChannels;
    l.rows = take(frame_bytes);
    for (int i = 0; i < l.n_frame; ++i) {
        l.frame_out.push_back(take(frame_bytes));
        l.frame_pre.push_back(keeps_pre(m.acts[i]) ? take(frame_bytes) : l.frame_out.back());
    }
    l.pooled = take(word_bytes);
    for (int i = 0; i < l.n_word; ++i) {
        l.word_out.push_back(take(word_bytes));
        l.word_pre.push_back(
            keeps_pre(m.acts[l.n_frame + i]) ? take(word_bytes) : l.word_out.back());
    }
    l.logits_rows = take(sizeof(float) * (size_t)l.total_words);
    const size_t weight_bytes = sizeof(float) * kTrainKernel * kTrainChannels * kTrainChannels;
    l.packed_w = take(weight_bytes);
    l.adjoint_w = take(weight_bytes);
    // one operand blob per layer: a whole direction is packed by one launch
    l.tc_stride = up(3 * (kTrainKernel * kTrainChannels * kTrainChannels * 2 + 2 * kTrainChannels * 16) + 1024);
    l.tc_w = take(l.tc_stride * (size_t)(l.n_frame + l.n_word));
    l.dw = take(weight_bytes);
    l.db = take(sizeof(float) * kTrainChannels);
    l.dz = take(sizeof(float) * (size_t)l.total_words);
    l.grad_a = take(frame_bytes);
    l.grad_b = take(frame_bytes);
    l.head_w = take(sizeof(float) * 7 * kTrainChannels);
    l.head_dw = take(sizeof(float) * 7 * kTrainChannels);
    l.head_db = take(256);
    l.total_bytes = cursor;
    return l;
}

static int check_model(const emph_train_model& m) {
    EMPH_REQUIRE(m.channels == kTrainChannels && m.kernel_size == kTrainKernel &&
                     m.head_kernel >= 1 && m.head_kernel <= 7 && (m.head_kernel & 1),
                 "emph_train_*: built for 80 channels, kernel size 3 (got %d, %d, head %d)",
                 m.channels, m.kernel_size, m.head_kernel);
    EMPH_REQUIRE(m.n_frame_layers >= 1 && m.n_word_layers >= 0 &&
                     m.n_frame_layers + m.n_word_layers <= 32,
                 "emph_train_*: layer counts out of range");
    for (int precision : {m.precision, m.forward_precision})
        EMPH_REQUIRE(precision == EMPH_PREC_FP32 || precision == EMPH_PREC_BF16X3_TC ||
                         precision == EMPH_PREC_BF16X6_TC,
                     "emph_train_*: precision %d (fp32, bf16x3 or bf16x6)", precision);
    for (int i = 1; m.dropout && i < m.n_frame_layers + m.n_word_layers; ++i)
        EMPH_REQUIRE(m.dropout[i] >= 0.f && m.dropout[i] < 1.f,
                     "emph_train_*: dropout p %f after layer %d", m.dropout[i], i);
    return EMPH_OK;
}

// one conv layer y = act(conv(x, W) + b) with W in the Conv1d (out, in, k) layout
// (tensor-core modes: layer `index`'s blob was packed by pack_direction)
static int conv_layer(
    const emph_train_model& m, const TrainLayout& l, uint8_t* base, const float* x,
    const int32_t* row_seq, int rows, int index, const float* bias, int act,
    bool adjoint, float* y, void* stream) {
    const float* weight = m.weights[index];
    const int32_t acts[1] = {act};
    const int precision = adjoint ? m.precision : m.forward_precision;
    if (precision == EMPH_PREC_FP32) {
        float* packed = reinterpret_cast<float*>(base + (adjoint ? l.adjoint_w : l.packed_w));
        int s = adjoint
            ? emph_pack_conv_weights_adjoint(weight, kTrainChannels, kTrainChannels, kTrainKernel, packed, stream)
            : emph_pack_conv_weights(weight, kTrainChannels, kTrainChannels, kTrainKernel, packed, stream);
        if (s != EMPH_OK) return s;
        return emph_conv_stack(x, row_seq, rows, packed, bias, acts, 1, kTrainChannels,
                               kTrainKernel, EMPH_PREC_FP32, y, stream);
    }
    const void* blob = base + l.tc_w + l.tc_stride * (size_t)index;
    return emph_conv_stack(x, row_seq, rows, static_cast<const float*>(blob), bias, acts, 1,
                           kTrainChannels, kTrainKernel, precision, y, stream);
}

// tensor-core modes: the Conv1d weights of all layers go straight into their
// operand blobs (forward: with the biases; adjoint: transposed, taps flipped,
// zero bias) in ONE launch
static int pack_direction(
    const emph_train_model& m, const TrainLayout& l, uint8_t* base, bool adjoint, void* stream) {
    const int precision = adjoint ? m.precision : m.forward_precision;
    if (precision == EMPH_PREC_FP32) return EMPH_OK;
    const int n = l.n_frame + l.n_word;
    const float* biases[32];
    for (int i = 0; i < n; ++i) biases[i] = adjoint ? m.zero_bias : m.biases[i];
    return pack_conv1d_weights_tc_batch(
        m.weights, biases, n, kTrainKernel, precision, adjoint, base + l.tc_w, l.tc_stride,
        (cudaStream_t)stream);
}

}  // namespace emph

extern "C" long long emph_train_workspace(
    const emph_train_model* model, int32_t batch, int32_t frames, int32_t wmax) {
    if (!model || batch <= 0 || frames <= 0 || wmax <= 0) return -1;
    if (emph::check_model(*model) != EMPH_OK) return -1;
    return (long long)emph::make_layout(*model, batch, frames, wmax, nullptr).total_bytes;
}

extern "C" int emph_train_forward(
    const emph_train_model* model, const float* features, int32_t batch, int32_t frames,
    const int64_t* frame_lengths_host,
    const int64_t* word_bounds_host, const int64_t* word_lengths_host, int32_t wmax,
    void* workspace, long long workspace_bytes, float* logits, void* stream) {
    using namespace emph;
    EMPH_REQUIRE(model && features && word_bounds_host && word_lengths_host && workspace && logits,
                 "emph_train_forward: null argument");
    int s = check_model(*model);
    if (s != EMPH_OK) return s;
    const emph_train_model& m = *model;
    const TrainLayout l = make_layout(m, batch, frames, wmax, frame_lengths_host);
    EMPH_REQUIRE((long long)l.total_bytes <= workspace_bytes, "emph_train_forward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* base = static_cast<uint8_t*>(workspace);
    auto ints = [&](size_t at) { return reinterpret_cast<int32_t*>(base + at); };
    auto floats = [&](size_t at) { return reinterpret_cast<float*>(base + at); };

    // ---- index arrays (model.word_rows / engine.packed_starts), one copy ----
    std::vector<int32_t> blob(l.blob_words, 0);
    int32_t* h = blob.data();
    int32_t* row_start = h, *n_rows = h + batch, *word_row_start = h + 2 * batch,
            *n_words = h + 3 * batch, *word_seq = h + 4 * batch, *word_lo = word_seq + l.total_words,
            *word_hi = word_lo + l.total_words, *index = word_hi + l.total_words;
    for (int w = 0; w < l.total_words; ++w) word_seq[w] = -1;
    int next_row = 1;
    for (int b = 0; b < batch; ++b) {
        row_start[b] = next_row;
        n_rows[b] = kept_rows(m, frames, frame_lengths_host, b);
        next_row += n_rows[b] + 1;
        word_row_start[b] = word_gap(m) + b * (wmax + word_gap(m));
        n_words[b] = wmax;
        const int64_t count = word_lengths_host[b];
        for (int j = 0; j < wmax; ++j) {
            const int w = word_row_start[b] + j;
            word_seq[w] = b;
            const bool real = j < count;
            // slots past the item's words are marked (-1, -1): padded
            word_lo[w] = real ? (int32_t)word_bounds_host[((size_t)b * 2 + 0) * wmax + j] : -1;
            word_hi[w] = real ? (int32_t)word_bounds_host[((size_t)b * 2 + 1) * wmax + j] : -1;
            index[b * wmax + j] = w;
        }
    }
    if ((s = staged_upload(base + l.blob, h, 4 * l.blob_words, st)) != EMPH_OK) return s;
    if ((s = emph_row_index(ints(l.row_start), ints(l.n_rows), batch, ints(l.row_seq), l.total, stream))) return s;
    if ((s = emph_row_index(ints(l.word_row_start), ints(l.n_words), batch, ints(l.word_row_seq),
                            l.total_words, stream))) return s;
    if ((s = emph_pack_rows(features, batch, kTrainChannels, frames, ints(l.row_start), ints(l.n_rows),
                            ints(l.row_seq), l.total, floats(l.rows), stream))) return s;

    // ---- layers, every output kept ----
    if ((s = pack_direction(m, l, base, false, stream))) return s;
    // `starts` / `width`: the sequences' first rows and the reference's padded
    // width, which place a row in the dropout masks
    auto run_stack = [&](int first, int count, const float* input, const int32_t* seq, int rows,
                         const int32_t* starts, int width,
                         const std::vector<size_t>& out, const std::vector<size_t>& pre) -> int {
        const float* x = input;
        for (int i = 0; i < count; ++i) {
            const int act = m.acts[first + i];
            const float p = dropout_p(m, first + i);
            int status;
            if (keeps_pre(act)) {
                status = conv_layer(m, l, base, x, seq, rows, first + i, m.biases[first + i],
                                    EMPH_ACT_NONE, false, floats(pre[i]), stream);
                if (status == EMPH_OK && p > 0.f)
                    status = emph_conv_dropout_forward(
                        floats(pre[i]), seq, starts, rows, kTrainChannels, width, act, m.seed,
                        dropout_site(m, first + i), p, floats(out[i]), stream);
                else if (status == EMPH_OK)
                    status = emph_activation_forward(floats(pre[i]), seq, rows, kTrainChannels, act,
                                                     floats(out[i]), stream);
            } else {
                status = conv_layer(m, l, base, x, seq, rows, first + i, m.biases[first + i],
                                    act, false, floats(out[i]), stream);
                if (status == EMPH_OK && p > 0.f)
                    status = emph_conv_dropout_forward(
                        floats(out[i]), seq, starts, rows, kTrainChannels, width, EMPH_ACT_NONE,
                        m.seed, dropout_site(m, first + i), p, floats(out[i]), stream);
            }
            if (status != EMPH_OK) return status;
            x = floats(out[i]);
        }
        return EMPH_OK;
    };
    if ((s = run_stack(0, l.n_frame, floats(l.rows), ints(l.row_seq), l.total, ints(l.row_start),
                       frames, l.frame_out, l.frame_pre))) return s;
    if ((s = emph_pool_words(floats(l.frame_out.back()), kTrainChannels, ints(l.row_start), ints(l.n_rows),
                             ints(l.word_seq), ints(l.word_lo), ints(l.word_hi), l.total_words,
                             m.pool_method, floats(l.pooled), stream))) return s;
    if ((s = run_stack(l.n_frame, l.n_word, floats(l.pooled), ints(l.word_row_seq), l.total_words,
                       ints(l.word_row_start), wmax, l.word_out, l.word_pre))) return s;
    const float* head_in = l.n_word ? floats(l.word_out.back()) : floats(l.pooled);
    // output layer: Conv1d (1, C, k) weight -> [k][C], bias from device memory
    float* head_w = floats(l.head_w);
    if ((s = emph_pack_conv_weights(m.weights[l.n_frame + l.n_word], 1, kTrainChannels, m.head_kernel,
                                    head_w, stream))) return s;
    if ((s = emph_output_head(head_in, ints(l.word_row_seq), l.total_words, kTrainChannels, m.head_kernel,
                              head_w, 0.f, EMPH_HEAD_LOGITS, floats(l.logits_rows), nullptr, stream))) return s;
    add_bias_kernel<<<(l.total_words + 255) / 256, 256, 0, st>>>(
        floats(l.logits_rows), ints(l.word_row_seq), l.total_words, m.biases[l.n_frame + l.n_word]);
    EMPH_CHECK_LAUNCH("emph_train_forward(bias)");
    gather_rows_kernel<<<(batch * wmax + 255) / 256, 256, 0, st>>>(
        floats(l.logits_rows), ints(l.index), batch * wmax, logits);
    EMPH_CHECK_LAUNCH("emph_train_forward(gather)");
    return EMPH_OK;
}

extern "C" int emph_train_backward(
    const emph_train_model* model, const float* grad_logits, int32_t batch, int32_t frames,
    const int64_t* frame_lengths_host,
    int32_t wmax, void* workspace, long long workspace_bytes, float* const* grads,
    int32_t accumulate, void* stream) {
    using namespace emph;
    EMPH_REQUIRE(model && grad_logits && workspace && grads, "emph_train_backward: null argument");
    int s = check_model(*model);
    if (s != EMPH_OK) return s;
    const emph_train_model& m = *model;
    const TrainLayout l = make_layout(m, batch, frames, wmax, frame_lengths_host);
    EMPH_REQUIRE((long long)l.total_bytes <= workspace_bytes, "emph_train_backward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* base = static_cast<uint8_t*>(workspace);
    auto ints = [&](size_t at) { return reinterpret_cast<int32_t*>(base + at); };
    auto floats = [&](size_t at) { return reinterpret_cast<float*>(base + at); };
    const int n_layers = l.n_frame + l.n_word;

    // d loss / d logits of the (B, 1, Wmax) tensor -> packed word rows
    s = check_cuda(cudaMemsetAsync(base + l.dz, 0, sizeof(float) * (size_t)l.total_words, st),
                   "emph_train_backward: memset");
    if (s != EMPH_OK) return s;
    scatter_rows_kernel<<<(batch * wmax + 255) / 256, 256, 0, st>>>(
        grad_logits, ints(l.index), batch * wmax, floats(l.dz));
    EMPH_CHECK_LAUNCH("emph_train_backward(scatter)");

    // output projection
    const float* head_in = l.n_word ? floats(l.word_out.back()) : floats(l.pooled);
    float* head_w = floats(l.head_w);        // packed by the forward call
    float* dx = floats(l.grad_a);
    float* other = floats(l.grad_b);
    if ((s = emph_output_head_backward(head_in, floats(l.dz), ints(l.word_row_seq), l.total_words,
                                       kTrainChannels, m.head_kernel, head_w, dx, floats(l.head_dw),
                                       floats(l.head_db), stream))) return s;
    head_grad_layout_kernel<<<(kTrainChannels * m.head_kernel + 255) / 256, 256, 0, st>>>(
        floats(l.head_dw), kTrainChannels, m.head_kernel, accumulate, grads[2 * n_layers]);
    vector_store_kernel<<<1, 32, 0, st>>>(floats(l.head_db), 1, accumulate, grads[2 * n_layers + 1]);
    EMPH_CHECK_LAUNCH("emph_train_backward(head)");

    // conv stacks, last layer first; dy in `dx`, result back in `dx`
    if ((s = pack_direction(m, l, base, true, stream))) return s;
    auto stack_backward = [&](int first, int count, const float* input, const int32_t* seq, int rows,
                              const int32_t* starts, int width,
                              const std::vector<size_t>& out, const std::vector<size_t>& pre) -> int {
        for (int i = count - 1; i >= 0; --i) {
            const int act = m.acts[first + i];
            const float p = dropout_p(m, first + i);
            const float* x_in = i ? floats(out[i - 1]) : input;       // dropped, as the forward read it
            int status = p > 0.f
                ? emph_activation_dropout_backward(dx, floats(pre[i]), seq, starts, rows,
                                                   kTrainChannels, width, act, m.seed,
                                                   dropout_site(m, first + i), p, other, stream)
                : emph_activation_backward(dx, floats(pre[i]), seq, rows, kTrainChannels, act,
                                           other, stream);                          // dpre
            if (status != EMPH_OK) return status;
            // straight into the parameters' gradients, (out, in, k) and (out)
            status = conv1d_weight_grad(x_in, other, rows, kTrainChannels, kTrainKernel,
                                        grads[2 * (first + i)], grads[2 * (first + i) + 1],
                                        accumulate, st);
            if (status != EMPH_OK) return status;
            if (first + i == 0) break;          // the features need no gradient
            // dx = conv(dpre, W flipped and transposed), zero bias, no activation
            status = conv_layer(m, l, base, other, seq, rows, first + i, m.zero_bias,
                                EMPH_ACT_NONE, true, dx, stream);
            if (status != EMPH_OK) return status;
        }
        return EMPH_OK;
    };
    if (l.n_word) {
        if ((s = stack_backward(l.n_frame, l.n_word, floats(l.pooled), ints(l.word_row_seq),
                                l.total_words, ints(l.word_row_start), wmax, l.word_out,
                                l.word_pre))) return s;
    }
    // pooling adjoint: d pooled (in dx) -> d frames (in other), then swap roles
    if ((s = emph_pool_words_backward(dx, floats(l.frame_out.back()), kTrainChannels, ints(l.row_start),
                                      ints(l.n_rows), ints(l.word_seq), ints(l.word_lo), ints(l.word_hi),
                                      l.total_words, m.pool_method, l.total, other, stream))) return s;
    std::swap(dx, other);
    return stack_backward(0, l.n_frame, floats(l.rows), ints(l.row_seq), l.total, ints(l.row_start),
                          frames, l.frame_out, l.frame_pre);
}
