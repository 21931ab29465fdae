// One utterance through the whole path in ONE native call (BASELINE config 1:
// emphases.from_alignment_and_audio on a single utterance,
// emphases/core.py:223-287).  The batched engine plans with numpy and launches
// through seven ctypes calls: ~0.45 ms of host work around 0.13 ms of GPU time.
// Here the plan of the common case -- batch_size=None, the utterance is one
// chunk -- is made in C++ with the same float64 operations as
// engine.chunk_words, the index arrays travel in one copy, and the seven
// kernels are launched back to back on the caller's stream.  Anything unusual
// (a second chunk, a dropped chunk, bounds the reference raises on) returns
// EMPH_ENOSYS and the caller takes the general path.
#include <math.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace emph {

constexpr int kSampleRate = 16000;
constexpr int kHopsize = 160;
constexpr int kPadding = 432;

// Python's float // float (floatobject.c float_floor_div) == numpy's
// npy_divmod: the quotient emphases/convert.py:19-31 and the chunker use
static double floor_divide(double a, double b) {
    double mod = fmod(a, b);
    double div = (a - mod) / b;
    if (mod != 0.0) {
        if ((b < 0) != (mod < 0)) div -= 1.0;
    }
    if (div != 0.0) {
        double floordiv = floor(div);
        if (div - floordiv > 0.5) floordiv += 1.0;
        return floordiv;
    }
    return copysign(0.0, a / b);
}

static size_t align_up(size_t value, size_t to) { return (value + to - 1) / to * to; }

struct UtterancePlan {
    int32_t chunk_start, chunk_len, n_rows, total_rows, total_word_rows;
    std::vector<int32_t> word_lo, word_hi;
};

// engine.chunk_words + engine._assemble_plan for one utterance that is one
// chunk; false = not that case
static bool plan_single_chunk(
    const double* times, int n_words, long long n_samples, int method, UtterancePlan& plan) {
    if (n_words <= 0 || n_samples <= 0) return false;
    const long long padded = n_samples + 2 * kPadding;
    const long long total_frames = (long long)((double)padded / (double)kHopsize);
    // frames accumulated over words 0 .. W-2 must not exceed the chunk limit
    double running = 0.0;
    for (int w = 0; w < n_words; ++w) {
        const double frames = floor_divide((times[2 * w + 1] - times[2 * w]) * kSampleRate, kHopsize);
        if (!(frames >= 0.0)) return false;
        if (w + 1 < n_words) {
            running += frames;
            if ((long long)running > total_frames) return false;
        }
    }
    const double origin = times[0];
    const long long start_sample = kHopsize * (long long)floor_divide(times[0] * kSampleRate, kHopsize);
    const long long end_sample =
        kHopsize * (long long)floor_divide(times[2 * (n_words - 1) + 1] * kSampleRate, kHopsize);
    const long long lo = std::min(std::max(start_sample, 0LL), padded);
    const long long hi = std::min(std::max(end_sample, 0LL), padded);
    const long long length = std::max(hi - lo, 0LL);
    if (length <= kPadding) return false;
    const long long n_rows = length / kHopsize;
    if (n_rows + 2 >= (1LL << 31)) return false;
    plan.chunk_start = (int32_t)lo;
    plan.chunk_len = (int32_t)length;
    plan.n_rows = (int32_t)n_rows;
    // one separator row each side: enough at kernel sizes 5 and 7 too, since
    // both conv kernels read rows before 0 and from total_rows on as zeros
    plan.total_rows = (int32_t)n_rows + 2;
    plan.total_word_rows = n_words + 2;
    plan.word_lo.assign(plan.total_word_rows, 0);
    plan.word_hi.assign(plan.total_word_rows, 0);
    for (int w = 0; w < n_words; ++w) {
        // pypar slice re-based to its first word, then int(t * sr / hop)
        const long long b0 = (long long)((times[2 * w] - origin) * kSampleRate / kHopsize);
        const long long b1 = (long long)((times[2 * w + 1] - origin) * kSampleRate / kHopsize);
        if (b0 < INT32_MIN || b0 > INT32_MAX || b1 < INT32_MIN || b1 > INT32_MAX) return false;
        // engine.validate_bounds: where the reference raises, the general path does
        const long long s = std::min(std::max(b0, 0LL), n_rows), e = std::min(std::max(b1, 0LL), n_rows);
        if (method == EMPH_POOL_MAX && e <= s) return false;
        if (method == EMPH_POOL_CENTER && floor_divide((double)(b0 + b1), 2.0) >= (double)n_rows)
            return false;
        plan.word_lo[w + 1] = (int32_t)b0;
        plan.word_hi[w + 1] = (int32_t)b1;
    }
    return true;
}

// device workspace: [index blob][audio][features][frames][pooled][words][logits][scores]
struct Layout {
    size_t blob, audio, features, frames, pooled, words, logits, scores, total;
};
static Layout layout_for(long long n_samples, int n_words, int channels, int n_mels, int audio_bytes) {
    const long long rows = (n_samples + 2 * kPadding) / kHopsize + 3;
    const long long word_rows = n_words + 2;
    Layout l;
    size_t cursor = 0;
    auto take = [&](size_t bytes) { size_t at = cursor; cursor = align_up(cursor + bytes, 256); return at; };
    l.blob = take(sizeof(int32_t) * (size_t)(16 + rows + 4 * word_rows) + 64);
    l.audio = take((size_t)audio_bytes * (size_t)(n_samples + 16));
    l.features = take(sizeof(float) * (size_t)rows * (size_t)std::max(n_mels, channels));
    l.frames = take(sizeof(float) * (size_t)rows * channels);
    l.pooled = take(sizeof(float) * (size_t)word_rows * channels);
    l.words = take(sizeof(float) * (size_t)word_rows * channels);
    l.logits = take(sizeof(float) * (size_t)word_rows);
    l.scores = take(sizeof(float) * (size_t)word_rows);
    l.total = cursor;
    return l;
}

}  // namespace emph

extern "C" long long emph_infer_utterance_workspace(
    long long n_samples, int32_t n_words, int32_t channels, int32_t n_mels) {
    if (n_samples < 0 || n_words < 0 || channels <= 0) return -1;
    return (long long)emph::layout_for(n_samples, n_words, channels, n_mels, 4).total;
}

extern "C" int emph_infer_utterance(
    const emph_utterance_model* model, const double* times, int32_t n_words,
    const void* audio, int32_t audio_is_int16, long long n_samples,
    void* workspace, long long workspace_bytes,
    float** logits_out, float** scores_out, void* stream) {
    using namespace emph;
    EMPH_REQUIRE(model && times && audio && workspace, "emph_infer_utterance: null argument");
    UtterancePlan plan;
    if (!plan_single_chunk(times, n_words, n_samples, model->pool_method, plan)) {
        set_error("emph_infer_utterance: not a single-chunk utterance (general path)");
        return EMPH_ENOSYS;
    }
    const int channels = model->frame.channels;
    const int audio_bytes = audio_is_int16 ? 2 : 4;
    const Layout l = layout_for(n_samples, n_words, channels, model->n_mels, audio_bytes);
    EMPH_REQUIRE((long long)l.total <= workspace_bytes, "emph_infer_utterance: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* base = static_cast<uint8_t*>(workspace);

    // ---- index arrays: one blob, one copy through the pinned staging ring ----
    const int rows = plan.total_rows, word_rows = plan.total_word_rows;
    // [audio_off (int64: 2 words)][audio_len][chunk_start][chunk_len][row_start][n_rows]
    // [word_row_start][n_words][word_seq w][word_lo w][word_hi w]
    const size_t blob_words = 16 + 3 * (size_t)word_rows;
    std::vector<int32_t> host_blob(blob_words, 0);
    int32_t* host = host_blob.data();
    host[2] = (int32_t)n_samples;       // audio_len
    host[3] = plan.chunk_start;
    host[4] = plan.chunk_len;
    host[5] = 1;                        // row_start
    host[6] = plan.n_rows;
    host[7] = 1;                        // word_row_start
    host[8] = n_words;
    int32_t* word_seq = host + 16;
    int32_t* word_lo = word_seq + word_rows;
    int32_t* word_hi = word_lo + word_rows;
    for (int w = 0; w < word_rows; ++w) word_seq[w] = (w >= 1 && w <= n_words) ? 0 : -1;
    memcpy(word_lo, plan.word_lo.data(), sizeof(int32_t) * word_rows);
    memcpy(word_hi, plan.word_hi.data(), sizeof(int32_t) * word_rows);
    int32_t* dev = reinterpret_cast<int32_t*>(base + l.blob);
    int s = staged_upload(dev, host, blob_words * 4, st);
    if (s != EMPH_OK) return s;
    const int64_t* audio_off = reinterpret_cast<const int64_t*>(dev);
    const int32_t *audio_len = dev + 2, *chunk_start = dev + 3, *chunk_len = dev + 4,
                  *row_start = dev + 5, *n_rows = dev + 6, *word_row_start = dev + 7,
                  *n_words_dev = dev + 8, *d_word_seq = dev + 16,
                  *d_word_lo = d_word_seq + word_rows, *d_word_hi = d_word_lo + word_rows;
    int32_t* row_seq = dev + 16 + 3 * word_rows;          // [rows]
    int32_t* word_row_seq = row_seq + rows;               // [word_rows]

    // ---- audio (a device pointer is used in place) ----
    cudaPointerAttributes attributes;
    const void* device_audio = audio;
    const bool on_device =
        cudaPointerGetAttributes(&attributes, audio) == cudaSuccess &&
        attributes.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    if (!on_device || (reinterpret_cast<uintptr_t>(audio) & 15) != 0) {
        s = check_cuda(
            cudaMemcpyAsync(base + l.audio, audio, (size_t)audio_bytes * (size_t)n_samples,
                            on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st),
            "emph_infer_utterance: audio copy");
        if (s != EMPH_OK) return s;
        device_audio = base + l.audio;
    }

    float* features = reinterpret_cast<float*>(base + l.features);
    float* frames = reinterpret_cast<float*>(base + l.frames);
    float* pooled = reinterpret_cast<float*>(base + l.pooled);
    float* words = reinterpret_cast<float*>(base + l.words);
    float* logits = reinterpret_cast<float*>(base + l.logits);
    float* scores = reinterpret_cast<float*>(base + l.scores);

    // ---- the seven kernels ----
    if ((s = emph_row_index(row_start, n_rows, 1, row_seq, rows, stream)) != EMPH_OK) return s;
    if ((s = emph_row_index(word_row_start, n_words_dev, 1, word_row_seq, word_rows, stream)) != EMPH_OK)
        return s;
    s = audio_is_int16
        ? emph_logmel_i16(static_cast<const int16_t*>(device_audio), audio_off, audio_len, chunk_start,
                          chunk_len, row_start, 1, row_seq, rows, model->mel_ptr, model->mel_col,
                          model->mel_val, model->n_mels, model->normalize, features, stream)
        : emph_logmel_f32(static_cast<const float*>(device_audio), audio_off, audio_len, chunk_start,
                          chunk_len, row_start, 1, row_seq, rows, model->mel_ptr, model->mel_col,
                          model->mel_val, model->n_mels, model->normalize, features, stream);
    if (s != EMPH_OK) return s;
    const emph_utterance_stack& f = model->frame;
    s = emph_conv_stack(features, row_seq, rows, static_cast<const float*>(f.weights), f.bias,
                        f.acts_host, f.n_layers, f.channels, f.kernel_size, f.precision, frames, stream);
    if (s != EMPH_OK) return s;
    s = emph_pool_words(frames, channels, row_start, n_rows, d_word_seq, d_word_lo, d_word_hi,
                        word_rows, model->pool_method, pooled, stream);
    if (s != EMPH_OK) return s;
    const float* head_input = pooled;
    if (model->has_word_stack) {
        const emph_utterance_stack& w = model->word;
        s = emph_conv_stack(pooled, word_row_seq, word_rows, static_cast<const float*>(w.weights),
                            w.bias, w.acts_host, w.n_layers, w.channels, w.kernel_size, w.precision,
                            words, stream);
        if (s != EMPH_OK) return s;
        head_input = words;
    }
    s = emph_output_head(head_input, word_row_seq, word_rows, channels, model->head_kernel,
                         model->head_weight, model->head_bias, model->head_mode, logits, scores,
                         stream);
    if (s != EMPH_OK) return s;
    // word w of the utterance is row 1 + w
    if (logits_out) *logits_out = logits + 1;
    if (scores_out) *scores_out = scores + 1;
    return EMPH_OK;
}
