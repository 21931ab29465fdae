/*
 * emphases_b200 -- C ABI of the B200-native (sm_100a) inference hot path of
 * interactiveaudiolab/emphases:
 *
 *   waveform + word alignment -> log-mel -> framewise Conv1d/ReLU stack ->
 *   word-bound segment pooling -> word decoder -> Conv1d(->1) -> sigmoid
 *
 * The reference has no FFI of its own (it is pure Python/PyTorch); every entry
 * point below replaces one Python/PyTorch call site of the reference, cited as
 * file:line relative to the reference root.  The host mirror of the reference's
 * Python API (emphases_b200/) binds these with ctypes; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all work is asynchronous on it;
 *   - every function returns 0 on success, a negative EMPH_E* code on failure,
 *     never throws; emph_last_error() returns a thread-local message;
 *   - nothing allocates: the caller owns all buffers;
 *   - index arrays are int32 (int64 for sample offsets).
 *
 * Packed ("ragged, no padding FLOPs") layout
 *   A launch processes n_seq sequences (utterance chunks).  All frame-resolution
 *   tensors are [total_rows][channels] fp32, row-major (channel contiguous).
 *   Sequence u owns rows [row_start[u], row_start[u] + n_rows[u]); between two
 *   sequences, before the first and after the last there is at least ONE
 *   separator row, whose content is forced to zero at every layer -- that
 *   reproduces Conv1d(padding='same') zero padding per utterance
 *   (emphases/model/layers/convolution.py:17-20) without per-utterance launches.
 *   `row_seq[r]` = owning sequence of row r, or -1 for a separator.
 *   The word-resolution tensors use the same layout over "word rows".
 */
#ifndef EMPHASES_B200_H
#define EMPHASES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMPH_OK 0
#define EMPH_EINVAL (-22)   /* bad argument */
#define EMPH_ECUDA (-5)     /* CUDA runtime error, see emph_last_error() */
#define EMPH_ENOSYS (-38)   /* configuration not compiled in */

/* activation codes (emphases/config/defaults.py:181 ACTIVATION_FUNCTION and the
 * config/hparam-search activations) */
#define EMPH_ACT_NONE 0
#define EMPH_ACT_RELU 1
#define EMPH_ACT_GELU 2
#define EMPH_ACT_LEAKY_RELU 3
#define EMPH_ACT_SILU 4

/* pooling methods (emphases/core.py:426-469 DOWNSAMPLE_METHOD) */
#define EMPH_POOL_AVERAGE 0
#define EMPH_POOL_MAX 1
#define EMPH_POOL_SUM 2
#define EMPH_POOL_CENTER 3

/* head modes (emphases/core.py:335-342 postprocess) */
#define EMPH_HEAD_LOGITS 0
#define EMPH_HEAD_SIGMOID 1   /* LOSS == 'bce' */
#define EMPH_HEAD_CLAMP 2     /* LOSS == 'mse' */

/* precision modes of the conv stack */
#define EMPH_PREC_FP32 0      /* CUDA-core FFMA, max-abs 1e-5 on scores */
#define EMPH_PREC_BF16_TC 1   /* tcgen05 bf16 MMA, fp32 accumulate, 2e-3 */
#define EMPH_PREC_BF16X3_TC 2 /* tcgen05, hi/lo split of both operands (3 MMAs per
                                product, 16 mantissa bits per operand): 1e-4 */
#define EMPH_PREC_BF16X6_TC 3 /* tcgen05, hi/mid/lo split of both operands (6 MMAs per
                                product, 24 mantissa bits per operand): fp32-grade,
                                1e-5 on scores like EMPH_PREC_FP32 */

int emph_version(void);
const char* emph_last_error(void);

/* Number of SMs of the current device (for callers that size work lists). */
int emph_device_sm_count(void);

/*
 * row_seq[r] = u if row_start[u] <= r < row_start[u] + n_rows[u] else -1.
 * row_start must be strictly increasing.  Replaces the implicit batch
 * dimension of the reference's padded tensors (emphases/data/collate.py:11-78).
 */
int emph_row_index(
    const int32_t* row_start, const int32_t* n_rows, int32_t n_seq,
    int32_t* row_seq, int32_t total_rows, void* stream);

/*
 * Log-mel features of every chunk, fused: zero pad (emphases/core.py:357-358),
 * chunk slice (core.py:395-401), reflect pad (emphases/data/preprocess/
 * mels.py:32-36), Hann window + 1024-point real FFT with hop 160
 * (mels.py:39-48), sqrt(re^2+im^2+1e-6) (mels.py:51), mel projection and
 * log(clamp(.,1e-5)) (mels.py:94-109), optional (x+10)/10 (mels.py:57-58).
 *
 *   audio          packed fp32 samples (channel 0 of each utterance)
 *   audio_off[u]   first sample of the utterance chunk u is cut from
 *                  (must be a multiple of 4: frames are read with 4-sample
 *                  vector loads; when it is a multiple of 4 (fp32) / 8
 *                  (int16) samples, i.e. 16 bytes, tiles of 16 interior
 *                  frames are staged into shared memory with one
 *                  cp.async.bulk instead of per-frame loads)
 *   audio_len[u]   T, that utterance's length in samples
 *   chunk_start[u] first sample of the chunk in ZERO-PADDED coordinates
 *                  (432 zeros before the utterance), = 160 * first frame
 *   chunk_len[u]   L, chunk length in samples (> 432); frames = L / 160
 *   row_start[u]   first packed row of the chunk; n_rows = L / 160
 *   mel_ptr/col/val  CSR of the (n_mels x 513) mel basis (an input, as in
 *                  the reference where librosa supplies it, mels.py:97-100)
 *   out            [total_rows][n_mels] fp32; separator rows are zeroed
 */
int emph_logmel_f32(
    const float* audio,
    const int64_t* audio_off, const int32_t* audio_len,
    const int32_t* chunk_start, const int32_t* chunk_len,
    const int32_t* row_start, int32_t n_seq,
    const int32_t* row_seq, int32_t total_rows,
    const int32_t* mel_ptr, const int16_t* mel_col, const float* mel_val,
    int32_t n_mels, int32_t normalize,
    float* out, void* stream);

/* Same, int16 PCM input scaled by 1/32768 (what torchaudio.load returns for
 * 16-bit wav files, emphases/load.py:11-17). */
int emph_logmel_i16(
    const int16_t* audio,
    const int64_t* audio_off, const int32_t* audio_len,
    const int32_t* chunk_start, const int32_t* chunk_len,
    const int32_t* row_start, int32_t n_seq,
    const int32_t* row_seq, int32_t total_rows,
    const int32_t* mel_ptr, const int16_t* mel_col, const float* mel_val,
    int32_t n_mels, int32_t normalize,
    float* out, void* stream);

/*
 * emph_logmel_* with the sample-rate conversion of emphases.resample
 * (emphases/core.py:613-619 -> torchaudio.transforms.Resample) fused into the
 * front end: `audio` is packed at the SOURCE rate (audio_off / source_len in
 * source samples per sequence) while audio_len, chunk_start and chunk_len stay
 * in model-rate (16 kHz) samples, audio_len[u] = ceil(new * source_len / orig).
 * Every model-rate sample the frames need is the polyphase windowed-sinc sum
 * of csrc/resample.cu (emph_resample_*: same filter bank, same order, so the
 * features equal those of resampling first, bit for bit) -- computed tile by
 * tile in shared memory, never written to HBM.
 *
 *   filter      [new_freq][2 * width + orig_freq] fp32 (rates divided by their
 *               gcd), tap_lo / tap_hi [new_freq]: the range of taps of each
 *               phase that are not exactly zero
 */
int emph_logmel_resampled_f32(
    const float* audio, const int64_t* audio_off, const int32_t* source_len,
    const int32_t* audio_len, const int32_t* chunk_start, const int32_t* chunk_len,
    const int32_t* row_start, int32_t n_seq, const int32_t* row_seq, int32_t total_rows,
    const int32_t* mel_ptr, const int16_t* mel_col, const float* mel_val,
    int32_t n_mels, int32_t normalize,
    const float* filter, const int32_t* tap_lo, const int32_t* tap_hi,
    int32_t orig_freq, int32_t new_freq, int32_t width, float* out, void* stream);
int emph_logmel_resampled_i16(
    const int16_t* audio, const int64_t* audio_off, const int32_t* source_len,
    const int32_t* audio_len, const int32_t* chunk_start, const int32_t* chunk_len,
    const int32_t* row_start, int32_t n_seq, const int32_t* row_seq, int32_t total_rows,
    const int32_t* mel_ptr, const int16_t* mel_col, const float* mel_val,
    int32_t n_mels, int32_t normalize,
    const float* filter, const int32_t* tap_lo, const int32_t* tap_hi,
    int32_t orig_freq, int32_t new_freq, int32_t width, float* out, void* stream);

/*
 * A stack of n_layers Conv1d(channels -> channels, kernel_size,
 * padding='same') layers, each followed by its activation, over the packed row
 * axis (emphases/model/core.py:17-20 input_layer + emphases/model/layers/
 * convolution.py:13-37; also the word decoder, model/core.py:105-107).
 *
 *   x, y       [total_rows][channels] fp32; must NOT alias (CTAs read halo
 *              rows of x that neighbouring CTAs own in y)
 *   weights    EMPH_PREC_FP32: [n_layers][kernel_size][channels(in)]
 *              [channels(out)] fp32, produced by emph_pack_conv_weights from
 *              Conv1d (out, in, k); EMPH_PREC_BF16_TC / _BF16X3_TC: the blob
 *              produced by emph_pack_conv_weights_tc for that precision
 *   bias       [n_layers][channels]
 *   acts       [n_layers] EMPH_ACT_* codes (host pointer)
 *   precision  EMPH_PREC_*
 */
int emph_conv_stack(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const float* bias, const int32_t* acts_host,
    int32_t n_layers, int32_t channels, int32_t kernel_size,
    int32_t precision, float* y, void* stream);

/*
 * Weights for precision == EMPH_PREC_BF16_TC / _BF16X3_TC / _BF16X6_TC (the
 * split modes pack 2 / 3 bf16 blobs per layer: hi, (mid,) lo): fp32 weights
 * [n_layers][k][in][out] (the layout above) and bias [n_layers][out] -> per
 * layer a bf16 blob in the UMMA shared-memory operand layout, split in two
 * halves of the output channels, [2][k][in / 8][out / 2][8] (one half per CTA
 * of the kernel's CTA pairs), followed by a bias chunk (the bias as three bf16 parts, rebuilt exactly to
 * fp32 and added by the kernel's epilogue).  emph_conv_weights_tc_bytes gives the blob size (0 if
 * the configuration is not compiled in).  Pass the blob as `weights` of
 * emph_conv_stack; `bias` is then unused.
 */
int emph_conv_weights_tc_bytes(
    int32_t n_layers, int32_t channels, int32_t kernel_size, int32_t precision);
int emph_pack_conv_weights_tc(
    const float* weights, const float* bias, int32_t n_layers, int32_t channels,
    int32_t kernel_size, int32_t precision, void* packed, void* stream);

/*
 * emph_conv_stack (tensor-core precisions, channels 80, kernel size 3) with
 * the frame -> word pooling of emph_pool_words fused into the last layer's
 * epilogue: emphases/model/core.py:92-101 (frame_encoder followed by
 * downsample at the 'intermediate' location) in one pass, the frame rows never
 * travelling to HBM unless `y` is given.
 *
 * Requirements (else EMPH_ENOSYS and nothing is written: call emph_conv_stack
 * + emph_pool_words instead): the words of a sequence do not overlap (each
 * frame row belongs to at most one word), the last activation is ReLU (or
 * none, except for `max`).
 *
 *   row_word    scratch [total_rows] int32, word_count scratch
 *               [total_word_rows] int32, fixed scratch [total_word_rows]
 *               [channels] int64 (sum / average only; may be null otherwise)
 *   pooled      [total_word_rows][channels] fp32, as emph_pool_words writes it
 *               (word rows without frames: 0 for sum / max / center -- the
 *               host raises before launching for those -- NaN for average)
 *   y           [total_rows][channels] fp32 frame rows, or NULL
 *
 * Sums are formed in 64-bit fixed point (2^-28 units, values clamped to
 * +-2^19), so the result is independent of how tiles cut a word and of the
 * order the atomics land: bit-identical for every packing of the corpus.
 */
int emph_conv_stack_pool(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const int32_t* acts_host, int32_t n_layers, int32_t channels,
    int32_t kernel_size, int32_t precision,
    const int32_t* row_start, const int32_t* n_rows,
    const int32_t* word_seq, const int32_t* word_lo, const int32_t* word_hi,
    int32_t total_word_rows, int32_t method,
    int32_t* row_word, int32_t* word_count, long long* fixed,
    float* pooled, float* y, void* stream);

/* (out, in, k) Conv1d weight -> [k][in][out] (device to device). */
int emph_pack_conv_weights(
    const float* conv_weight, int32_t out_channels, int32_t in_channels,
    int32_t kernel_size, float* packed, void* stream);
/* (out, in, k) Conv1d weight -> the adjoint convolution in the same packed
 * layout, [k][out][in] with the taps flipped: the input gradient of a layer is
 * emph_conv_stack(dY, adjoint weights, zero bias, no activation). */
int emph_pack_conv_weights_adjoint(
    const float* conv_weight, int32_t out_channels, int32_t in_channels,
    int32_t kernel_size, float* packed, void* stream);

/*
 * Frame -> word segment pooling (emphases/core.py:426-469 `downsample`).
 * One warp per word row, driven by integer offset arrays, no host round trip.
 *
 *   x              [total_rows][channels] fp32 frame-resolution activations
 *   row_start[u], n_rows[u]  frame rows of sequence u
 *   word_seq[w]    owning sequence of word row w, -1 for separator word rows
 *   word_lo/hi[w]  word bounds [lo, hi) in frames relative to the sequence
 *                  start, exactly the int64 bounds of core.py:384-392;
 *                  hi is clipped to n_rows[u] like a torch slice.  lo = hi =
 *                  -1 marks a padded word slot (j >= word_lengths[i]): zeros
 *                  for average/max/sum, frame 0 for center (core.py:458-466).
 *                  lo = hi = -2 forces zeros for every method (the word mask
 *                  of the 'input' location, emphases/model/core.py:77-82).
 *   y              [total_word_rows][channels]; separator rows zeroed
 * Empty segments: sum -> 0, average -> NaN (as torch.mean of an empty slice),
 * max -> -inf (the reference raises IndexError; the host mirror raises it
 * before launching).
 */
int emph_pool_words(
    const float* x, int32_t channels,
    const int32_t* row_start, const int32_t* n_rows,
    const int32_t* word_seq, const int32_t* word_lo, const int32_t* word_hi,
    int32_t total_word_rows, int32_t method, float* y, void* stream);

/*
 * One utterance through the whole path in one call: BASELINE config 1,
 * emphases.from_alignment_and_audio on a single utterance with batch_size =
 * None (emphases/core.py:223-287: preprocess -> infer -> postprocess).  The
 * chunk plan (emphases/core.py:361-401 for an utterance that is ONE chunk) is
 * made on the host with the same float64 operations as the batched planner,
 * the index arrays travel in one copy, and the seven kernels
 * (2 row maps, log-mel, frame stack, pooling, word stack, head) are launched
 * back to back on `stream`.
 *
 * Returns EMPH_ENOSYS -- nothing launched -- when the utterance is not a single
 * chunk or its bounds are ones the reference raises on: take the general path.
 *
 *   model       stacks as emph_conv_stack takes them (weights = the blob that
 *               matches `precision`), head as emph_output_head, the mel basis
 *               as emph_logmel_*; has_word_stack = 0 for the locations without
 *               a word decoder
 *   times       host [n_words][2] float64 word (start, end) seconds
 *   audio       n_samples fp32 (or int16 PCM) samples, host or device memory
 *   workspace   device scratch of emph_infer_utterance_workspace(...) bytes
 *   logits_out, scores_out  receive device pointers INTO the workspace:
 *               n_words values each, valid until the workspace is reused
 */
typedef struct {
    const void* weights;
    const float* bias;
    const int32_t* acts_host;
    int32_t n_layers, channels, kernel_size, precision;
} emph_utterance_stack;

typedef struct {
    emph_utterance_stack frame, word;
    int32_t has_word_stack;
    const float* head_weight;
    float head_bias;
    int32_t head_kernel, head_mode;
    const int32_t* mel_ptr;
    const int16_t* mel_col;
    const float* mel_val;
    int32_t n_mels, normalize, pool_method;
} emph_utterance_model;

long long emph_infer_utterance_workspace(
    long long n_samples, int32_t n_words, int32_t channels, int32_t n_mels);
int emph_infer_utterance(
    const emph_utterance_model* model, const double* times, int32_t n_words,
    const void* audio, int32_t audio_is_int16, long long n_samples,
    void* workspace, long long workspace_bytes,
    float** logits_out, float** scores_out, void* stream);

/*
 * Output projection Conv1d(channels -> 1, kernel_size, 'same') over packed rows
 * (emphases/model/core.py:33-37,138) + postprocess (core.py:335-342).
 *   weight [kernel_size][channels], bias_host scalar.
 *   logits/scores [total_rows] (either may be NULL); separator rows get 0.
 */
int emph_output_head(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, int32_t kernel_size, const float* weight, float bias_host,
    int32_t mode, float* logits, float* scores, void* stream);

/* (B, C, T) channel-major tensor (the reference's layout, model/core.py:39)
 * <-> packed rows.  Sequence b occupies rows [row_start[b], +n_rows[b]) and
 * columns [0, n_rows[b]) of its (C, T) plane with plane stride C * T. */
int emph_pack_rows(
    const float* bct, int32_t batch, int32_t channels, int32_t frames,
    const int32_t* row_start, const int32_t* n_rows,
    const int32_t* row_seq, int32_t total_rows, float* rows, void* stream);
int emph_unpack_rows(
    const float* rows, const int32_t* row_start, const int32_t* n_rows,
    int32_t batch, int32_t channels, int32_t frames, float* bct, void* stream);

/*
 * Zero-extend packed rows [rows][channels_in] to [rows][channels_out] (both
 * multiples of 4): the 80 log-mel features entering a model whose CHANNELS is
 * larger (128 in the reference's config/hparam-search), emphases/model/
 * core.py:17-20 input_layer being Conv1d(NUM_FEATURES -> CHANNELS).
 */
int emph_widen_rows(
    const float* x, int32_t rows, int32_t channels_in, int32_t channels_out, float* y,
    void* stream);

/*
 * Word segmentation for the 'input' downsample location (emphases/core.py:
 * 552-586 `segment`): segment q copies count[q] rows of x starting at absolute
 * row src_row[q] into its own sequence of seg_len rows (zero-filled tail),
 * dst rows [dst_row_start[q], +seg_len).  dst_row_seq maps dst rows to q / -1.
 */
int emph_segment_rows(
    const float* x, int32_t channels,
    const int32_t* src_row, const int32_t* count, const int32_t* dst_row_start,
    int32_t n_seg, const int32_t* dst_row_seq, int32_t total_dst_rows,
    float* y, void* stream);

/*
 * Transformer variant (emphases/model/layers/transformer.py:13-52), fp32.
 * Per-row linear maps (in_proj, out_proj, linear1/2) run through
 * emph_conv_stack with kernel_size 1; these cover the rest.
 *
 * emph_add_positional: y = x + table[t] with t the row's index inside its
 *   sequence (transformer.py:50-52; `table` is the module's (max_len, channels)
 *   `position.encoding` buffer).
 * emph_attention_rows: out = softmax(q k^T * scale + key mask) v per head over
 *   the rows of each sequence; keys with index >= n_keys[u] are the padded
 *   positions of the reference's src_key_padding_mask (transformer.py:26-29).
 *   All n_queries[u] rows are computed as queries, padded ones included, as
 *   nn.TransformerEncoder does (their values reach valid words through the
 *   k=3 output conv).  The caller supplies the query blocks (block_seq[b],
 *   block_q0[b]): 128 queries each, never crossing a sequence.
 * emph_attention_rows_tc: the same attention on the tensor cores (mma.sync
 *   m16n8k16, fp32 accumulation and softmax; csrc/attention_tc.cu).  `mode`:
 *   0 = one fp16 per operand (the reference itself runs attention in half
 *   precision under torch.autocast, core.py:606), 1 = every operand a bf16
 *   (hi, lo) pair, three MMAs per product (fp32 grade: scores within 1e-5 of
 *   the fp32 path).  K and V are first converted into `workspace`
 *   (emph_attention_tc_workspace bytes, 256-byte aligned; -1 = unsupported
 *   head dim), which a later call may reuse.
 * emph_add_layernorm: y = LayerNorm(x + residual; gamma, beta, eps).
 */
int emph_add_positional(
    const float* x, const int32_t* row_start, const int32_t* row_seq,
    int32_t total_rows, int32_t channels, const float* table,
    int32_t table_rows, float* y, void* stream);
int emph_attention_rows(
    const float* q, const float* k, const float* v, int32_t channels,
    int32_t heads, const int32_t* row_start, const int32_t* n_queries,
    const int32_t* n_keys, const int32_t* row_seq, int32_t total_rows,
    const int32_t* block_seq,
    const int32_t* block_q0, int32_t n_blocks, float scale, float* out,
    void* stream);
int emph_attention_rows_tc(
    const float* q, const float* k, const float* v, int32_t channels,
    int32_t heads, const int32_t* row_start, const int32_t* n_queries,
    const int32_t* n_keys, const int32_t* row_seq, int32_t total_rows,
    const int32_t* block_seq,
    const int32_t* block_q0, int32_t n_blocks, float scale, int32_t mode,
    void* workspace, int64_t workspace_bytes, float* out, void* stream);
int64_t emph_attention_tc_workspace(
    int32_t total_rows, int32_t channels, int32_t heads, int32_t mode);

/*
 * One Transformer encoder layer (transformer.py:18-23: post-norm
 * nn.TransformerEncoderLayer, ReLU, dim_feedforward = channels = 80) as three
 * fused per-row passes around the attention kernel (csrc/transformer_tc.cu),
 * on mma.sync: activations and weights split into `parts` bf16 parts (2: three
 * products, 3: six products: fp32 grade) or, parts = 1, rounded to one fp16
 * value (the 2e-3 mode).  Weight blobs are 16-bit [matrix][part][out][in + 8]
 * (part p = bf16 of what parts < p left over; parts = 1: fp16).
 *
 * emph_transformer_qkv: q = x Wq^T + bq as fp32 rows; k and v are written
 *   directly as the 16-bit records emph_attention_rows_staged reads
 *   (`attention_mode` as in emph_attention_rows_tc; the buffer has
 *   emph_attention_tc_workspace bytes = heads x (total_rows + 64) records,
 *   head-major; the caller zeroes the 64 records behind each head's rows).
 *   weights: 3 matrices (rows 0..79 / 80..159 / 160..239 of in_proj_weight).
 * emph_attention_rows_staged: emph_attention_rows_tc without the staging pass.
 * emph_transformer_proj_norm: y = LayerNorm(residual + x W^T + b).
 * emph_transformer_ffn_norm: y = LayerNorm(x + relu(x W1^T + b1) W2^T + b2)
 *   (weights: 2 matrices, bias: b1 then b2).  Separator rows of y are zero.
 */
int emph_transformer_qkv(
    const float* x, int32_t total_rows, int32_t channels, const void* weights,
    const float* bias, int32_t parts, int32_t attention_mode, float* q,
    void* staged, int64_t staged_bytes, void* stream);
int emph_attention_rows_staged(
    const float* q, const void* staged, int64_t staged_bytes, int32_t channels,
    int32_t heads, const int32_t* row_start, const int32_t* n_queries,
    const int32_t* n_keys, int32_t total_rows, const int32_t* block_seq,
    const int32_t* block_q0, int32_t n_blocks, float scale, int32_t mode,
    float* out, void* stream);
int emph_transformer_proj_norm(
    const float* x, const float* residual, int32_t total_rows, int32_t channels,
    const void* weights, const float* bias, int32_t parts, const float* gamma,
    const float* beta, float eps, const int32_t* row_seq, float* y,
    void* stream);
int emph_transformer_ffn_norm(
    const float* x, int32_t total_rows, int32_t channels, const void* weights,
    const float* bias, int32_t parts, const float* gamma, const float* beta,
    float eps, const int32_t* row_seq, float* y, void* stream);
/* Both of the above in one pass (weights: out-projection, linear1, linear2;
 * bias: bo, b1, b2): the LayerNorm1 output never leaves registers. */
int emph_transformer_layer_tail(
    const float* x, const float* residual, int32_t total_rows, int32_t channels,
    const void* weights, const float* bias, int32_t parts, const float* gamma1,
    const float* beta1, const float* gamma2, const float* beta2, float eps,
    const int32_t* row_seq, float* y, void* stream);
int emph_add_layernorm(
    const float* x, const float* residual, const float* gamma,
    const float* beta, float eps, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, float* y, void* stream);

/*
 * Training step (BASELINE config 5; the reference's single-device step is
 * emphases/train/core.py:86-142, its loss :315-353), fp32.  Forward keeps each
 * layer's output (one emph_conv_stack launch per layer); per layer backward:
 *   emph_activation_backward  dpre = dy * act'(.), separators zeroed; `y` is the
 *                             layer output for ReLU / LeakyReLU / identity and
 *                             the pre-activation for GELU / SiLU, which the
 *                             forward keeps by running the conv with
 *                             EMPH_ACT_NONE and emph_activation_forward after it
 *   emph_conv_stack           dx = conv(dpre, W flipped and transposed)
 *   emph_conv_weight_grad     dw [k][in][out], db [out] (zeroed, then summed);
 *                             channels 80 at kernel sizes 1 / 3: fp32 FFMA
 *                             kernel; channels 80 at 5 / 7 and 128 at 1 / 3 /
 *                             5 / 7: split-bf16 mma.sync kernel (hi*hi +
 *                             lo*hi + hi*lo, fp32 accumulation, ~1e-6 of
 *                             |X|^T |dPre|); any other shape: EMPH_ENOSYS,
 *                             nothing launched.  A model narrower than 80 or
 *                             between 80 and 128 channels trains zero-padded
 *                             to the next of these widths.
 * emph_pool_words_backward / emph_output_head_backward are the adjoints of
 * emph_pool_words / emph_output_head (logits).  emph_masked_loss: mean BCE-with-
 * logits (mode 0) or squared error (mode 1) over word rows with valid != 0, and
 * its gradient with respect to the logits.
 */
int emph_activation_backward(
    const float* dy, const float* y, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, int32_t act, float* dpre, void* stream);
int emph_activation_forward(
    const float* pre, const int32_t* row_seq, int32_t total_rows, int32_t channels,
    int32_t act, float* y, void* stream);
int emph_conv_weight_grad(
    const float* x, const float* dpre, int32_t total_rows, int32_t channels,
    int32_t kernel_size, float* dw, float* db, void* stream);
int emph_pool_words_backward(
    const float* dy, const float* x, int32_t channels,
    const int32_t* row_start, const int32_t* n_rows,
    const int32_t* word_seq, const int32_t* word_lo, const int32_t* word_hi,
    int32_t total_word_rows, int32_t method, int32_t total_rows, float* dx,
    void* stream);
int emph_output_head_backward(
    const float* x, const float* dz, const int32_t* row_seq, int32_t total_rows,
    int32_t channels, int32_t kernel_size, const float* weight,
    float* dx, float* dw, float* db, void* stream);
int emph_masked_loss(
    const float* logits, const float* targets, const uint8_t* valid,
    int32_t total_rows, int32_t mode, float* loss, float* dlogits, void* stream);
/*
 * Dropout of the convolution model (emphases/model/layers/convolution.py:
 * 25-30: Conv1d -> activation -> Dropout(p) in every block of frame_encoder and
 * word_decoder), with the masks of EMPH_DROPOUT_CONV sites (see the dropout
 * comment below).  Rows are packed sequences: sequence n = row_seq[r] (-1 on
 * separator rows) starts at row_start[n] and stands for item (or segment) n of
 * the reference's padded tensor of `width` columns (T, max_length at the
 * 'input' location, or Wmax); channels % 4 == 0.
 *   emph_conv_dropout_forward        y = act(x) * keep / (1 - p), separators
 *                                    zero; with EMPH_ACT_NONE in place on a conv
 *                                    output whose activation is applied, with
 *                                    GELU / SiLU on the kept pre-activation
 *   emph_activation_dropout_backward dpre = dy * keep / (1 - p) * act'(.), the
 *                                    mask regenerated; `y` as for
 *                                    emph_activation_backward, where the output
 *                                    of ReLU / LeakyReLU / identity layers is
 *                                    the dropped output
 */
int emph_conv_dropout_forward(
    const float* x, const int32_t* row_seq, const int32_t* row_start, int32_t total_rows,
    int32_t channels, int32_t width, int32_t act, uint64_t seed, uint32_t site, float p,
    float* y, void* stream);
int emph_activation_dropout_backward(
    const float* dy, const float* y, const int32_t* row_seq, const int32_t* row_start,
    int32_t total_rows, int32_t channels, int32_t width, int32_t act, uint64_t seed,
    uint32_t site, float p, float* dpre, void* stream);

/*
 * Training of the Transformer variant (emphases/model/layers/transformer.py:
 * 13-52 in training mode: dropout after the positional encoding, on the
 * attention probabilities, on the attention output, inside the feed-forward
 * block and on its output), fp32, channels 80, 40-dim heads.
 *
 * Dropout: Philox4x32-10 keyed by a 64-bit `seed` (one per training forward);
 * element i of a site keeps its value iff its 32-bit draw >= round(p 2^32),
 * kept values are scaled by 1 / (1 - p); p = 0 keeps everything, scale 1.
 * The draw is a function of (seed, site, element index) only, so the
 * backward regenerates the forward's masks, and emph_dropout_keep writes
 * keep[i] (1 / 0) for element indices first .. first + count - 1 of any site.
 *   site  EMPH_DROPOUT_SITE(stack, layer, kind, head): stack 0 frame encoder,
 *         1 word decoder; the attention kernels add the head themselves.  The
 *         convolution model's blocks use EMPH_DROPOUT_CONV with `layer` the
 *         block index in its stack and head 0 (no dropout on input_layer or
 *         output_layer)
 *   index row-wise sites: packed_row * channels + channel;
 *         attention: packed_query_row << 16 | key index within the sequence;
 *         conv blocks: (n * width + w) * channels + channel, the element's
 *         position in the reference's padded (N, C, width) tensor taken
 *         channel fastest (n the item or segment, w its column), so any
 *         packing of the rows draws the same mask, and emph_dropout_keep over
 *         0 .. N * width * channels - 1 returns it in (N, width, C) order
 *
 *   emph_dropout_rows            y = x * keep / (1 - p), element index = flat
 *                                index of x (packed rows); its own backward
 *   emph_linear_rows             y_m = act(x W_m^T + b_m), m < parts: W is the
 *                                (parts * 80, 80) Linear weight, y is
 *                                [parts][rows][80]; separator rows zero
 *   emph_linear_rows_backward    dx = addend + sum_m dy_m W_m (addend may be
 *                                NULL), dy [parts][rows][80]
 *   emph_conv_weight_grad        with kernel_size 1: dW^T [in][out] of a Linear
 *   emph_attention_rows_train    emph_attention_rows with dropout(softmax) V and
 *                                lse[row * heads + head] = log2-domain
 *                                log-sum-exp (max + log2 sum) of the scores
 *                                S * scale * log2(e)
 *   emph_attention_rows_backward dq, dk, dv from q, k, v, out, d_out, lse (one
 *                                pass over 64-key blocks, key_block_*, one over
 *                                64-query blocks, query_block_*: no atomics);
 *                                rows that are no key get dk = dv = 0, and every
 *                                row of a sequence without keys NaN (its
 *                                softmax is NaN)
 *   emph_add_layernorm_train     emph_add_layernorm with dropout on `residual`;
 *                                keeps sums = x + dropout(residual) and stats
 *                                [rows][2] = (mean, rstd)
 *   emph_add_layernorm_backward  dx = d sums, d_branch = dx * keep / (1 - p),
 *                                dgamma / dbeta over the non-separator rows via
 *                                `partials` [emph_layernorm_backward_blocks(rows)]
 *                                [2 * channels] (per-CTA sums, then one ordered
 *                                reduction: deterministic)
 */
#define EMPH_DROPOUT_SITE(stack, layer, kind, head) \
    (((uint32_t)(stack) << 24) | ((uint32_t)(layer) << 16) | ((uint32_t)(kind) << 8) | (uint32_t)(head))
enum {
    EMPH_DROPOUT_POSITIONAL = 0,   /* position.dropout */
    EMPH_DROPOUT_ATTENTION = 1,    /* self_attn.dropout, on the probabilities */
    EMPH_DROPOUT_RESIDUAL1 = 2,    /* dropout1, attention output */
    EMPH_DROPOUT_FEEDFORWARD = 3,  /* dropout, between linear1 and linear2 */
    EMPH_DROPOUT_RESIDUAL2 = 4,    /* dropout2, feed-forward output */
    EMPH_DROPOUT_CONV = 5          /* convolution model: after each block's activation */
};
int emph_dropout_keep(
    uint64_t seed, uint32_t site, uint64_t first, int64_t count, float p, uint8_t* keep,
    void* stream);
int emph_dropout_rows(
    const float* x, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site, float p,
    float* y, void* stream);
int emph_linear_rows(
    const float* x, int32_t total_rows, int32_t channels, const float* weight, const float* bias,
    int32_t parts, int32_t act, const int32_t* row_seq, float* y, void* stream);
int emph_linear_rows_backward(
    const float* dy, int32_t total_rows, int32_t channels, const float* weight, int32_t parts,
    const float* addend, const int32_t* row_seq, float* dx, void* stream);
int emph_attention_rows_train(
    const float* q, const float* k, const float* v, int32_t channels, int32_t heads,
    const int32_t* row_start, const int32_t* n_queries, const int32_t* n_keys,
    const int32_t* row_seq, int32_t total_rows,
    const int32_t* block_seq, const int32_t* block_q0, int32_t n_blocks,
    float scale, uint64_t seed, uint32_t site, float p, float* out, float* lse, void* stream);
int emph_attention_rows_backward(
    const float* q, const float* k, const float* v, const float* out, const float* d_out,
    const float* lse, int32_t channels, int32_t heads, const int32_t* row_start,
    const int32_t* n_queries, const int32_t* n_keys, int32_t total_rows,
    const int32_t* key_block_seq, const int32_t* key_block_k0, int32_t n_key_blocks,
    const int32_t* query_block_seq, const int32_t* query_block_q0, int32_t n_query_blocks,
    float scale, uint64_t seed, uint32_t site, float p, float* dq, float* dk, float* dv,
    void* stream);
int emph_add_layernorm_train(
    const float* x, const float* residual, const float* gamma, const float* beta, float eps,
    const int32_t* row_seq, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site,
    float p, float* y, float* sums, float* stats, void* stream);
int emph_layernorm_backward_blocks(int32_t total_rows);
int emph_add_layernorm_backward(
    const float* dy, const float* sums, const float* stats, const float* gamma,
    const int32_t* row_seq, int32_t total_rows, int32_t channels, uint64_t seed, uint32_t site,
    float p, float* dx, float* d_branch, float* dgamma, float* dbeta, float* partials,
    void* stream);
/*
 * Training-mode forward and backward of the convolution model, ONE call each
 * (emphases/train/core.py:111-142: model(...) and backward() of one step).
 * Built for channels = NUM_MELS = 80, kernel size 3 and the word-resolution
 * locations ('intermediate': with word decoder, 'loss': without); other
 * configurations use the per-kernel entry points above.
 *
 *   model     layers in order: input layer, frame encoder layers, word decoder
 *             layers (n_word_layers may be 0), then the output projection.
 *             weights[i] / biases[i] are the Conv1d parameters themselves
 *             ((out, in, k) fp32 on the device; they change every step, so
 *             both calls re-pack what they need); acts[i] the EMPH_ACT_* code
 *             after layer i.  forward_precision / precision: EMPH_PREC_FP32,
 *             EMPH_PREC_BF16X3_TC or _BF16X6_TC for the forward / the
 *             input-gradient convolutions.  The weight gradients run on
 *             mma.sync in every mode: bf16 hi + lo operands (16 bits each),
 *             hi*hi + lo*hi + hi*lo with fp32 accumulation, ~2^-16 relative
 *             per product.
 *   features  (B, 80, T) fp32 device; word_bounds (B, 2, Wmax) / word_lengths
 *             (B) int64 HOST arrays (emphases/data/collate.py:72-78).
 *             frame_lengths (B) int64 host, or NULL: the reference convolves
 *             all T padded columns of every item.  With lengths given, rows
 *             further than one row per frame layer beyond frame_lengths[b] are
 *             skipped, which keeps the last frame layer exact up to row
 *             frame_lengths[b] only: same logits and gradients as long as no
 *             word of item b reads a frame at or past frame_lengths[b].  A word
 *             may end past the audio, so pass per item max(length, 1 + the
 *             last frame any word reads: hi - 1, or (lo + hi) / 2 for
 *             `center`), and the same array to both calls.
 *   workspace device scratch of emph_train_workspace(...) bytes: it carries the
 *             kept activations from emph_train_forward to emph_train_backward
 *   logits    (B, 1, Wmax) fp32 device out (padded slots included, as
 *             emphases/model/core.py:138 returns them)
 *   grads     host array of device pointers, two per layer (weight then bias)
 *             in the order above plus the output projection's: gradients in
 *             the parameters' own layouts, written (accumulate = 0) or added
 *   dropout   host array, p after layer i's activation (one per frame and
 *             word layer; the input layer's is ignored), or NULL: layer i of
 *             the frame stack (i >= 1) draws its mask from site
 *             EMPH_DROPOUT_SITE(0, i - 1, EMPH_DROPOUT_CONV, 0), word layer j
 *             from (1, j, EMPH_DROPOUT_CONV, 0), keyed by `seed`.  The forward
 *             keeps the dropped outputs and the backward regenerates the
 *             masks, so both calls need the same seed.  p = 0 everywhere (or
 *             NULL) launches no dropout kernel.
 */
typedef struct {
    int32_t n_frame_layers, n_word_layers, channels, kernel_size, head_kernel;
    int32_t pool_method;
    int32_t forward_precision;      /* the forward convolutions */
    int32_t precision;              /* the input-gradient convolutions */
    const int32_t* acts;
    const float* const* weights;
    const float* const* biases;
    const float* zero_bias;         /* device [channels] zeros */
    const float* dropout;           /* host [n_frame_layers + n_word_layers] or NULL */
    uint64_t seed;                  /* dropout key of this step */
} emph_train_model;

long long emph_train_workspace(
    const emph_train_model* model, int32_t batch, int32_t frames, int32_t wmax);
int emph_train_forward(
    const emph_train_model* model, const float* features, int32_t batch, int32_t frames,
    const int64_t* frame_lengths_host,
    const int64_t* word_bounds_host, const int64_t* word_lengths_host, int32_t wmax,
    void* workspace, long long workspace_bytes, float* logits, void* stream);
int emph_train_backward(
    const emph_train_model* model, const float* grad_logits, int32_t batch, int32_t frames,
    const int64_t* frame_lengths_host,
    int32_t wmax, void* workspace, long long workspace_bytes, float* const* grads,
    int32_t accumulate, void* stream);

/*
 * Word -> frame interpolation (emphases/core.py:472-544 `upsample`) on the
 * reference's layouts: xs (B, C, Wmax) fp32, bounds (B, 2, Wmax) int64,
 * lengths int64 -> out (B, C, Tmax), zero past frame_lengths[b].  linear != 0:
 * UPSAMPLE_METHOD 'linear' (interpolates channel 0 for every channel, as the
 * reference does), else 'nearest'.
 */
int emph_upsample_words(
    const float* xs, const int64_t* bounds, const int64_t* word_lengths,
    const int64_t* frame_lengths, int32_t batch, int32_t channels, int32_t wmax,
    int32_t tmax, int32_t linear, float* out, void* stream);

/*
 * Evaluation caller (emphases/evaluate/core.py:27-110 with the metric classes of
 * emphases/evaluate/metrics.py:13-111): fp64 per-file sums over packed word rows
 * (file u owns rows word_row_start[u] .. + n_words[u]).  p = sigmoid(logit)
 * (loss_mode 0, LOSS 'bce') or clamp(logit, 0, 1) (loss_mode 1, LOSS 'mse').
 *   pass 0: sums[u][0..1] = sum p, sum t            (dataset mean / std pass)
 *   pass 1: sums[u][0..4] = sum (p-mean_p)^2, sum (t-mean_t)^2,
 *           sum (p-mean_p)(t-mean_t), sum bce(logit, t), sum (p-t)^2
 * sums is (n_seq, 5) fp64 on the device.
 */
int emph_word_metric_sums(
    const float* logits, const float* targets,
    const int32_t* word_row_start, const int32_t* n_words, int32_t n_seq,
    int32_t loss_mode, int32_t pass, double mean_p, double mean_t,
    double* sums, void* stream);

/*
 * Polyphase windowed-sinc resampling (emphases/core.py:613-619 `resample`, which
 * is torchaudio.transforms.Resample): y[q * new + p] = sum_k kernel[p][k] *
 * xpad[q * orig + k], xpad = zeros(width) ++ x ++ zeros(width + orig).
 * `kernel` is the (new_freq, 2 * width + orig_freq) filter bank (rates already
 * divided by their gcd), built on the host like torchaudio builds it.
 */
int emph_resample_f32(
    const float* x, int64_t length, const float* kernel, int32_t orig_freq,
    int32_t new_freq, int32_t width, float* y, int64_t target_length, void* stream);

/*
 * The same resampler over a packed int16 PCM corpus (samples are x / 32768,
 * what torchaudio.load returns, emphases/load.py:11-17) in one launch:
 * utterance u reads x[in_off[u] .. + in_len[u]) and writes
 * y[out_off[u] .. + out_len[u]), out_len = ceil(new * in_len / orig); out_off
 * ascending; y positions outside every utterance (alignment gaps) are zeroed.
 * This is the non-16 kHz branch of from_files_to_files (core.py:169-179 calls
 * emphases.resample per file).
 */
int emph_resample_packed_i16(
    const int16_t* x, const int64_t* in_off, const int64_t* in_len,
    const int64_t* out_off, const int64_t* out_len, int32_t n_utterances,
    const float* kernel, int32_t orig_freq, int32_t new_freq, int32_t width,
    float* y, int64_t total_out, void* stream);
/* The same for packed fp32 samples (a caller's list of tensors at another rate). */
int emph_resample_packed_f32(
    const float* x, const int64_t* in_off, const int64_t* in_len,
    const int64_t* out_off, const int64_t* out_len, int32_t n_utterances,
    const float* kernel, int32_t orig_freq, int32_t new_freq, int32_t width,
    float* y, int64_t total_out, void* stream);

/*
 * Host-side corpus ingest / egress for from_files_to_files (HOST pointers, no
 * CUDA): reads n_files (TextGrid, 16-bit PCM wav) pairs on a thread pool,
 * replacing per file emphases.load.audio (emphases/load.py:11-17),
 * pypar.Alignment(file) (emphases/core.py:49) and alignment.save
 * (emphases/core.py:111).  emph_corpus_open parses headers and alignments;
 * emph_corpus_info reports per file: status (0 = ok, otherwise the Python path
 * must handle the file), sample rate, channels, samples per channel, words
 * (gaps filled with silences); emph_corpus_fill writes channel 0 as int16 at
 * audio_dst + sample_offsets[i] (e.g. a pinned buffer) and (start, end) word
 * times as float64 pairs at times_dst + 2 * word_offsets[i];
 * emph_corpus_write_textgrids re-serialises the parsed alignments.
 */
typedef struct emph_corpus emph_corpus;
emph_corpus* emph_corpus_open(
    const char* const* text_paths, const char* const* audio_paths,
    int32_t n_files, int32_t n_threads);
int emph_corpus_info(
    const emph_corpus* corpus, int32_t* status, int32_t* sample_rate,
    int32_t* channels, int64_t* n_samples, int32_t* n_words);
const char* emph_corpus_error(const emph_corpus* corpus, int32_t index);
int emph_corpus_fill(
    emph_corpus* corpus, int16_t* audio_dst, const int64_t* sample_offsets,
    double* times_dst, const int64_t* word_offsets, int32_t n_threads);
/* The same for the listed files only (offset arrays still indexed by file), so
 * a corpus can be decoded group by group while earlier groups upload. */
int emph_corpus_fill_files(
    emph_corpus* corpus, const int32_t* file_indices, int32_t n_indices,
    int16_t* audio_dst, const int64_t* sample_offsets,
    double* times_dst, const int64_t* word_offsets, int32_t n_threads);
int emph_corpus_write_textgrids(
    const emph_corpus* corpus, const char* const* output_paths, int32_t n_threads);
void emph_corpus_close(emph_corpus* corpus);

/*
 * Pack a list of utterances (channel 0, fp32 HOST pointers) into one staging
 * buffer on the native thread pool: utterance i goes to dst[offsets[i] ..
 * + lengths[i]).  When dst_i16 and narrowed are given and EVERY sample is
 * k / 32768 with integer k in [-32768, 32767] -- audio decoded from 16-bit PCM,
 * which is what emphases.load.audio returns (emphases/load.py:11-17) -- the
 * samples are written to dst_i16 instead (same values, half the upload) and
 * *narrowed is set to 1; otherwise dst_f32 is filled and *narrowed is 0.
 * The caller's per-utterance tensors of from_alignment_and_audio
 * (emphases/core.py:223-230), batched.
 */
int emph_pack_audio_f32(
    const float* const* sources, const int64_t* lengths, const int64_t* offsets,
    int32_t n_utterances, float* dst_f32, int16_t* dst_i16, int32_t* narrowed,
    int32_t n_threads);

/*
 * torch.save(scores, f'{prefix}.pt') for a whole file list (emphases/core.py:
 * 112,177) on the native thread pool: file i receives scores[offsets[i] ..
 * + counts[i]) as a (1, counts[i]) float32 tensor in the zip-archive layout
 * torch.load reads (data.pkl, byteorder, data/0, version; stored, CRC-32).
 * HOST pointers; a NULL / empty path skips the file.
 */
int emph_write_score_files(
    const char* const* paths, const float* scores, const int64_t* offsets,
    const int32_t* counts, int32_t n_files, int32_t n_threads);
/* The same with one HOST pointer per file (rows[i] holds counts[i] floats).
 * n_threads < 0: -n_threads threads of the call's own instead of the shared
 * worker pool (a writer that runs beside a decode occupying the pool). */
int emph_write_score_rows(
    const char* const* paths, const float* const* rows, const int32_t* counts,
    int32_t n_files, int32_t n_threads);

/* The same three entry points with the paths as ONE buffer of NUL-terminated
 * strings, back to back (a char*[] of tens of thousands of strings costs the
 * Python binding more than parsing the files does).  write_textgrids_blob:
 * only the paths of the files with mask[i] != 0, in file order;
 * write_score_rows_blob: file i holds counts[i] values from base[starts[i]]. */
emph_corpus* emph_corpus_open_blob(
    const char* text_blob, const char* audio_blob, int32_t n_files, int32_t n_threads);
int emph_corpus_write_textgrids_blob(
    const emph_corpus* corpus, const char* path_blob, const uint8_t* mask, int32_t n_threads);
int emph_write_score_rows_blob(
    const char* path_blob, const float* base, const int64_t* starts, const int32_t* counts,
    int32_t n_files, int32_t n_threads);
/* sizes[i] = bytes of file i of a NUL-separated path buffer, -1 if it cannot
 * be stat'ed: the cost proxy of the length-balanced sharding of a file list
 * (emphases/core.py:169-179 walks the files in order on one device). */
int emph_file_sizes(const char* path_blob, int32_t n_files, int32_t n_threads, int64_t* sizes);

#ifdef __cplusplus
}
#endif
#endif /* EMPHASES_B200_H */
