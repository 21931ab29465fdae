"""Packed-batch execution engine: host planning + kernel launches.

Everything that computes runs in libemphases_b200.so (hand-written sm_100a
kernels, include/emphases_b200.h).  PyTorch is used for device memory, streams
and host<->device copies only.
"""
import dataclasses
from typing import Optional, Sequence

import ctypes
import os

import numpy as np
import torch

from . import _lib

SAMPLE_RATE = 16000
HOPSIZE = 160
NUM_FFT = 1024
WINDOW_SIZE = 1024
PADDING = int((WINDOW_SIZE - HOPSIZE) / 2)   # 432, emphases/core.py:357
KERNEL_CHANNELS = 80      # channel width of the tensor-core kernels and of the default model
WIDE_CHANNELS = 128       # fp32 tap-streamed conv kernel: CHANNELS=128 of the reference's sweep

ACTIVATIONS = {
    'ReLU': _lib.ACT_RELU,
    'GELU': _lib.ACT_GELU,
    'LeakyReLU': _lib.ACT_LEAKY_RELU,
    'SiLU': _lib.ACT_SILU,
    'Identity': _lib.ACT_NONE,
}


###############################################################################
# Mel basis (librosa.filters.mel restatement; reference call site
# emphases/data/preprocess/mels.py:97-100)
###############################################################################


def _hz_to_mel(frequencies):
    frequencies = np.atleast_1d(np.asarray(frequencies, dtype=np.float64))
    f_sp = 200.0 / 3
    mels = frequencies / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    log_t = frequencies >= min_log_hz
    mels[log_t] = min_log_mel + np.log(frequencies[log_t] / min_log_hz) / logstep
    return mels


def _mel_to_hz(mels):
    mels = np.atleast_1d(np.asarray(mels, dtype=np.float64))
    f_sp = 200.0 / 3
    freqs = f_sp * mels
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    log_t = mels >= min_log_mel
    freqs[log_t] = min_log_hz * np.exp(logstep * (mels[log_t] - min_log_mel))
    return freqs


def mel_basis(sample_rate=SAMPLE_RATE, n_fft=NUM_FFT, n_mels=80):
    """Slaney-scale, Slaney-normalised triangular filterbank (n_mels, 513)"""
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sample_rate)
    edges = _mel_to_hz(np.linspace(
        _hz_to_mel(0.0)[0], _hz_to_mel(sample_rate / 2.0)[0], n_mels + 2))
    widths = np.diff(edges)
    ramps = edges[:, None] - fftfreqs[None, :]
    basis = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float32)
    for i in range(n_mels):
        basis[i] = np.maximum(
            0, np.minimum(-ramps[i] / widths[i], ramps[i + 2] / widths[i + 1]))
    basis *= (2.0 / (edges[2:] - edges[:-2]))[:, None]
    return basis


def basis_to_csr(basis):
    """Dense (n_mels, 513) fp32 basis -> CSR arrays for emph_logmel_*"""
    basis = np.asarray(basis, dtype=np.float32)
    ptr = [0]
    cols, vals = [], []
    for row in basis:
        nz = np.nonzero(row)[0]
        cols.append(nz.astype(np.int16))
        vals.append(row[nz])
        ptr.append(ptr[-1] + len(nz))
    return (
        np.asarray(ptr, dtype=np.int32),
        np.concatenate(cols).astype(np.int16),
        np.concatenate(vals).astype(np.float32))


###############################################################################
# Host planning: chunker + packed layout (bit-exact integer logic)
###############################################################################


# Utterances start at multiples of 8 samples in a packed audio buffer: 16 bytes
# for int16 PCM, 32 for fp32 -- the alignment the log-mel kernel's bulk
# (cp.async.bulk) staging and vector loads need
AUDIO_ALIGN = 8


def align_samples(samples):
    """Round a sample count (int or array) up to AUDIO_ALIGN"""
    return (samples + AUDIO_ALIGN - 1) // AUDIO_ALIGN * AUDIO_ALIGN


def seconds_to_frames(seconds):
    """emphases/convert.py:19-31: float floor division"""
    return (seconds * SAMPLE_RATE) // HOPSIZE


def chunk_words(times: np.ndarray, num_samples: int, batch_size=None):
    """Word-aligned chunking of emphases.preprocess (emphases/core.py:361-401)

    times: (W, 2) float64 word (start, end) seconds.
    Returns a list of (word_start, word_end, start_sample, length, bounds)
    with bounds an (Wc, 2) int64 array relative to the chunk start; samples
    are in zero-padded coordinates.  Chunks of <= 432 samples are dropped as
    the reference silently does (core.py:413-415).
    """
    num_words = len(times)
    padded = num_samples + 2 * PADDING
    total_frames = int(padded / HOPSIZE)
    batch_size = total_frames if batch_size is None else batch_size
    durations = times[:, 1] - times[:, 0]
    word_frames = (durations * SAMPLE_RATE) // HOPSIZE     # float, floor-div
    chunks = []
    start = 0
    while start < num_words:
        end = num_words
        if start + 1 < num_words:
            # frames accumulated after adding words start .. e-1, e = start+1..W-1
            running = np.cumsum(word_frames[start:num_words - 1])
            over = np.nonzero(running.astype(np.int64) > batch_size)[0]
            if len(over):
                end = start + int(over[0]) + 1
        origin = times[start, 0]
        chunk = times[start:end]
        # pypar slice re-based to its first word, then int(t * sr / hop)
        bounds = np.stack([
            ((chunk[:, 0] - origin) * SAMPLE_RATE / HOPSIZE).astype(np.int64),
            ((chunk[:, 1] - origin) * SAMPLE_RATE / HOPSIZE).astype(np.int64)],
            axis=1)
        start_sample = HOPSIZE * int(seconds_to_frames(float(times[start, 0])))
        end_sample = HOPSIZE * int(seconds_to_frames(float(times[end - 1, 1])))
        lo = min(max(start_sample, 0), padded)       # torch slice clipping
        hi = min(max(end_sample, 0), padded)
        length = max(hi - lo, 0)
        if length > PADDING:
            chunks.append((start, end, lo, length, bounds))
        start = end
    return chunks


@dataclasses.dataclass
class Plan:
    """Host-side description of one packed launch"""
    n_seq: int
    total_rows: int
    total_word_rows: int
    utterance: np.ndarray        # (n_seq,) owning utterance of each chunk
    word_first: np.ndarray       # (n_seq,) first word (in the utterance)
    audio_off: np.ndarray        # int64 (n_seq,)
    audio_len: np.ndarray        # int32 ...
    chunk_start: np.ndarray
    chunk_len: np.ndarray
    row_start: np.ndarray
    n_rows: np.ndarray
    word_row_start: np.ndarray
    n_words: np.ndarray
    word_seq: np.ndarray         # (total_word_rows,)
    word_lo: np.ndarray
    word_hi: np.ndarray
    audio_samples: int           # packed audio length (samples)
    audio_offsets: np.ndarray    # int64 (n_utterances,) offset of each utterance

    def words_disjoint(self):
        """True when every frame row belongs to at most one word and no word is
        empty: the words of a sequence are in order and their clipped [lo, hi)
        do not overlap (what an alignment produces).  The fused conv + pooling
        kernel needs it; anything else takes the separate pooling kernel."""
        cached = getattr(self, '_words_disjoint', None)
        if cached is None:
            keep = self.word_seq >= 0
            seq = self.word_seq[keep]
            frames = self.n_rows[seq].astype(np.int64)
            lo = np.clip(self.word_lo[keep].astype(np.int64), 0, frames)
            hi = np.clip(self.word_hi[keep].astype(np.int64), 0, frames)
            same = seq[1:] == seq[:-1]
            cached = bool(
                np.all(hi > lo) and np.all(self.word_lo[keep] >= 0) and
                np.all(~same | (lo[1:] >= hi[:-1])))
            self._words_disjoint = cached
        return cached

    def int32_blob(self):
        parts = [
            self.audio_len, self.chunk_start, self.chunk_len, self.row_start,
            self.n_rows, self.word_row_start, self.n_words, self.word_seq,
            self.word_lo, self.word_hi]
        return np.concatenate([p.astype(np.int32, copy=False) for p in parts])


def separator_rows():
    """Separator rows needed between packed sequences: a Conv1d with kernel k
    reaches (k - 1) / 2 rows across a boundary, so that many zero rows
    reproduce its per-utterance 'same' padding (1 for the default k = 3)."""
    import emphases_b200 as emphases
    kernel = max(emphases.ENCODER_KERNEL_SIZE, emphases.DECODER_KERNEL_SIZE)
    return max(1, (int(kernel) - 1) // 2)


def packed_starts(lengths, gap=None):
    """Row layout with `gap` separator rows before, between and after
    sequences (default: what the configured kernel sizes need)"""
    if gap is None:
        gap = separator_rows()
    lengths = np.asarray(lengths, dtype=np.int64)
    starts = gap + np.concatenate([[0], np.cumsum(lengths[:-1] + gap)]) \
        if len(lengths) else np.zeros(0, dtype=np.int64)
    total = int(starts[-1] + lengths[-1] + gap) if len(lengths) else gap
    return starts, total


def make_plan(
    utterances: Sequence,
    batch_size: Optional[int] = None,
    validate_method: Optional[str] = None
) -> Plan:
    """utterances: sequence of (times (W, 2) float64, num_samples).

    With batch_size=None every utterance is normally ONE chunk; that case is
    planned for the whole corpus with vectorised numpy (same float64
    operations, element-wise, as the scalar chunker).  Anything else goes
    through `chunk_words` utterance by utterance."""
    if batch_size is None and len(utterances) > 1:
        plan = _make_plan_single_chunk(utterances, validate_method)
        if plan is not None:
            return plan
    utterance, word_first = [], []
    audio_off, audio_len, chunk_start, chunk_len = [], [], [], []
    bounds_list = []
    offsets = np.zeros(len(utterances), dtype=np.int64)
    cursor = 0
    for index, (times, num_samples) in enumerate(utterances):
        offsets[index] = cursor
        for (w0, w1, start, length, bounds) in chunk_words(
            np.asarray(times, dtype=np.float64).reshape(-1, 2),
            int(num_samples),
            batch_size
        ):
            utterance.append(index)
            word_first.append(w0)
            audio_off.append(cursor)
            audio_len.append(num_samples)
            chunk_start.append(start)
            chunk_len.append(length)
            bounds_list.append(bounds)
        cursor += align_samples(int(num_samples))
    all_bounds = np.concatenate(bounds_list, axis=0) if bounds_list \
        else np.zeros((0, 2), dtype=np.int64)
    return _assemble_plan(
        np.asarray(utterance, dtype=np.int64),
        np.asarray(word_first, dtype=np.int64),
        np.asarray(audio_off, dtype=np.int64),
        np.asarray(audio_len, dtype=np.int64),
        np.asarray(chunk_start, dtype=np.int64),
        np.asarray(chunk_len, dtype=np.int64),
        np.asarray([len(b) for b in bounds_list], dtype=np.int64),
        all_bounds, offsets, cursor, validate_method)


def _make_plan_single_chunk(utterances, validate_method):
    """Whole-corpus plan when every utterance is exactly one chunk
    (emphases/core.py:361-401 with batch_size = total_frames); returns None
    when any utterance needs the general chunker."""
    counts = np.fromiter(
        (len(times) for times, _ in utterances), dtype=np.int64,
        count=len(utterances))
    if np.any(counts == 0):
        return None
    samples = np.fromiter(
        (int(n) for _, n in utterances), dtype=np.int64, count=len(utterances))
    times = np.concatenate([
        np.asarray(t, dtype=np.float64).reshape(-1, 2) for t, _ in utterances])
    first = np.concatenate([[0], np.cumsum(counts[:-1])])
    last = first + counts - 1
    padded = samples + 2 * PADDING
    total_frames = (padded / HOPSIZE).astype(np.int64)        # int(len / hop)
    word_frames = ((times[:, 1] - times[:, 0]) * SAMPLE_RATE) // HOPSIZE
    if np.any(word_frames < 0):
        return None
    # the chunk loop accumulates the frames of words 0 .. W-2 (integer-valued
    # floats: any summation order is exact) and breaks when int(sum) > limit
    running = np.add.reduceat(word_frames, first) - word_frames[last]
    if np.any(running.astype(np.int64) > total_frames):
        return None
    origin = np.repeat(times[first, 0], counts)
    bounds = np.stack([
        ((times[:, 0] - origin) * SAMPLE_RATE / HOPSIZE).astype(np.int64),
        ((times[:, 1] - origin) * SAMPLE_RATE / HOPSIZE).astype(np.int64)],
        axis=1)
    start_sample = HOPSIZE * (
        (times[first, 0] * SAMPLE_RATE) // HOPSIZE).astype(np.int64)
    end_sample = HOPSIZE * (
        (times[last, 1] * SAMPLE_RATE) // HOPSIZE).astype(np.int64)
    lo = np.minimum(np.maximum(start_sample, 0), padded)
    hi = np.minimum(np.maximum(end_sample, 0), padded)
    length = np.maximum(hi - lo, 0)
    if np.any(length <= PADDING):
        return None                       # dropped chunks: general path
    aligned = align_samples(samples)
    offsets = np.concatenate([[0], np.cumsum(aligned[:-1])])
    return _assemble_plan(
        np.arange(len(utterances), dtype=np.int64),
        np.zeros(len(utterances), dtype=np.int64),
        offsets, samples, lo, length, counts, bounds, offsets,
        int(aligned.sum()), validate_method)


def _assemble_plan(
    utterance, word_first, audio_off, audio_len, chunk_start, chunk_len,
    n_words, all_bounds, offsets, cursor, validate_method
):
    n_seq = len(utterance)
    n_rows = chunk_len // HOPSIZE
    row_start, total_rows = packed_starts(n_rows)
    word_row_start, total_word_rows = packed_starts(n_words)
    if total_rows >= 2 ** 31 or cursor >= 2 ** 40:
        raise ValueError('batch too large for one launch; split it')
    word_seq = np.full(total_word_rows, -1, dtype=np.int32)
    word_lo = np.zeros(total_word_rows, dtype=np.int32)
    word_hi = np.zeros(total_word_rows, dtype=np.int32)
    if n_seq:
        # word rows of sequence u: word_row_start[u] + (0 .. n_words[u])
        sequence = np.repeat(np.arange(n_seq, dtype=np.int64), n_words)
        within = np.arange(len(sequence), dtype=np.int64) - np.repeat(
            np.concatenate([[0], np.cumsum(n_words[:-1])]), n_words)
        index = word_row_start[sequence] + within
        word_seq[index] = sequence
        word_lo[index] = all_bounds[:, 0]
        word_hi[index] = all_bounds[:, 1]
        if validate_method is not None:
            validate_bounds(all_bounds, n_rows[sequence], validate_method)
    return Plan(
        n_seq=n_seq,
        total_rows=total_rows,
        total_word_rows=total_word_rows,
        utterance=utterance,
        word_first=word_first,
        audio_off=audio_off.astype(np.int64),
        audio_len=audio_len.astype(np.int32),
        chunk_start=chunk_start.astype(np.int32),
        chunk_len=chunk_len.astype(np.int32),
        row_start=row_start.astype(np.int32),
        n_rows=n_rows.astype(np.int32),
        word_row_start=word_row_start.astype(np.int32),
        n_words=n_words.astype(np.int32),
        word_seq=word_seq,
        word_lo=word_lo,
        word_hi=word_hi,
        audio_samples=max(int(cursor), AUDIO_ALIGN),
        audio_offsets=np.asarray(offsets, dtype=np.int64))


def validate_bounds(bounds, frames, method):
    """Raise where the reference raises (SURVEY.md A.4, torch indexing)"""
    lo = np.minimum(np.maximum(bounds[:, 0], 0), frames)
    hi = np.minimum(np.maximum(bounds[:, 1], 0), frames)
    if method == 'max' and np.any(hi <= lo):
        raise IndexError(
            'max(): Expected reduction dim 1 to have non-zero size '
            '(a word spans zero frames)')
    if method == 'center' and np.any((bounds[:, 0] + bounds[:, 1]) // 2 >= frames):
        raise IndexError('center frame index out of range for a word')


###############################################################################
# Weights
###############################################################################


@dataclasses.dataclass
class ConvStack:
    weights: torch.Tensor        # [L][K][C][C] fp32 device
    bias: torch.Tensor           # [L][C]
    acts: np.ndarray             # int32 host
    kernel_size: int
    channels: int
    weights_tc: Optional[dict] = None            # precision -> UMMA-layout blob

    def tensor_core_weights(self, precision):
        """bf16 (or bf16 hi + lo) operand-layout copy for the tcgen05 path,
        packed on demand"""
        if self.weights_tc is None:
            self.weights_tc = {}
        if precision not in self.weights_tc:
            size = _lib.load().emph_conv_weights_tc_bytes(
                self.n_layers, self.channels, self.kernel_size, precision)
            if size <= 0:
                raise _lib.EmphasesB200Error(
                    f'the tensor-core conv stack is not compiled for '
                    f'channels={self.channels} kernel_size={self.kernel_size}; '
                    "use PRECISION='fp32'")
            blob = torch.empty(
                size, dtype=torch.uint8, device=self.weights.device)
            _lib.call(
                'emph_pack_conv_weights_tc', _lib.ptr(self.weights),
                _lib.ptr(self.bias), self.n_layers, self.channels,
                self.kernel_size, precision, _lib.ptr(blob), _lib.stream_ptr())
            self.weights_tc[precision] = blob
        return self.weights_tc[precision]

    @property
    def n_layers(self):
        return len(self.acts)


@dataclasses.dataclass
class ModelWeights:
    frame: ConvStack
    word: Optional[ConvStack]
    head_weight: torch.Tensor    # [K][C]
    head_bias: float
    head_kernel: int
    channels: int


def _pack_conv(weight, device):
    """Conv1d (out, in, k) -> [k][in][out] on device via the C ABI"""
    weight = weight.detach().to(device=device, dtype=torch.float32).contiguous()
    out_channels, in_channels, kernel = weight.shape
    packed = torch.empty(
        (kernel, in_channels, out_channels), dtype=torch.float32, device=device)
    _lib.call(
        'emph_pack_conv_weights', _lib.ptr(weight), out_channels, in_channels,
        kernel, _lib.ptr(packed), _lib.stream_ptr())
    return packed


def kernel_width(largest):
    """Channel count the kernels run a model at whose widest conv has
    `largest` channels: 80, or 128 for wider models"""
    return KERNEL_CHANNELS if largest <= KERNEL_CHANNELS else WIDE_CHANNELS


def pad(tensor, shape):
    """Zero-pad a weight/bias to the kernels' channel count.  Padded
    output channels compute act(0) = 0 for every supported activation and
    padded input channels multiply zeros, so the embedding is exact."""
    tensor = tensor.detach().to(torch.float32)
    if tuple(tensor.shape) == tuple(shape):
        return tensor
    padded = torch.zeros(shape, dtype=torch.float32, device=tensor.device)
    padded[tuple(slice(0, n) for n in tensor.shape)] = tensor
    return padded


def pack_weights(state, device, layers, activation, dropout, has_decoder):
    """Reference state_dict (SURVEY.md A.8) -> packed device buffers

    `state` keys: input_layer, frame_encoder.{i}, word_decoder.{i},
    output_layer; Sequential indices step by 2, or 3 with dropout
    (emphases/model/layers/convolution.py:25-30).
    """
    step = 3 if dropout is not None else 2
    act = ACTIVATIONS[activation]
    width = kernel_width(max(
        max(value.shape[0], value.shape[1]) for key, value in state.items()
        if key.endswith('.weight') and value.dim() == 3))

    def stack(first, prefix):
        convs = list(first)
        convs += [
            (state[f'{prefix}.{i * step}.weight'],
             state[f'{prefix}.{i * step}.bias']) for i in range(layers)]
        kernel = convs[-1][0].shape[2]
        if (kernel - 1) // 2 > separator_rows():
            raise ValueError(
                f'kernel size {kernel} needs {(kernel - 1) // 2} separator rows; '
                'set ENCODER_KERNEL_SIZE / DECODER_KERNEL_SIZE with '
                'emphases_b200.configure before running this model')
        for weight, _ in convs:
            if max(weight.shape[0], weight.shape[1]) > width or weight.shape[2] != kernel:
                raise NotImplementedError(
                    f'conv stack shape {tuple(weight.shape)} is not built: the '
                    f'kernels cover up to {width} channels (smaller models are '
                    'zero-padded) with one kernel size per stack')
        weights = torch.stack([
            _pack_conv(pad(w, (width, width, kernel)), device) for w, _ in convs])
        bias = torch.stack([pad(b, (width,)).to(device) for _, b in convs])
        acts = np.asarray(
            [_lib.ACT_NONE] * len(first) + [act] * layers, dtype=np.int32)
        return ConvStack(weights.contiguous(), bias.contiguous(), acts, kernel, width)

    frame = stack(
        [(state['input_layer.weight'], state['input_layer.bias'])],
        'frame_encoder')
    word = stack([], 'word_decoder') if has_decoder else None
    head = state['output_layer.weight']                  # (1, C, K)
    head = pad(head, (1, width, head.shape[2])).to(device)
    head_weight = head[0].t().contiguous()               # [K][C]
    return ModelWeights(
        frame=frame,
        word=word,
        head_weight=head_weight,
        head_bias=float(state['output_layer.bias'].detach().float().cpu()[0]),
        head_kernel=head.shape[2],
        channels=frame.channels)


###############################################################################
# Engine
###############################################################################


# Frame stack + word pooling as ONE kernel at the 'intermediate' location (the
# frame embeddings never travel to HBM).  Measured on a B200 (3.31 M frames):
# in the plain bf16 mode (4 tile slots) the fused stage takes 1.42 ms against
# 1.25 + 0.25 ms for conv stack + pooling kernel; in the split modes (2 slots:
# the longer last-layer epilogue sits in series with the slot's next tile) it
# loses, 9.88 against 9.53 ms per step in bf16x6
# (profiles/r02i_fused_pooling.md).  Default: fused in the bf16 mode only;
# EMPHASES_B200_FUSE_POOLING=1 / 0 forces it on (where applicable) / off.
FUSE_POOLING = os.environ.get('EMPHASES_B200_FUSE_POOLING', 'auto')


def fuse_pooling(precision):
    if FUSE_POOLING in ('0', '1'):
        return FUSE_POOLING == '1'
    return precision == _lib.PREC_BF16_TC


def tensor_core_shape(stack):
    """Conv stacks the tcgen05 kernel is compiled for: 80 channels, kernel
    size 1, 3, 5 or 7 (128 channels run on the FFMA kernel)"""
    return stack.channels == KERNEL_CHANNELS and stack.kernel_size in (1, 3, 5, 7)


def linear_precision(stack):
    """Per-row linear maps of the Transformer variant (kernel-size-1 stacks) run
    at fp32 grade on the tensor cores whenever a tensor-core PRECISION is
    selected: split-bf16 `bf16x6` in the 1e-5 mode, `bf16x3` in the 'bf16x3'
    and 'bf16' modes (scores of bench.py's corpus within 9e-6 of the fp32 mode
    with x3 maps and split-bf16 attention, 2.8e-4 with fp16 attention); else
    the FFMA kernel.  LayerNorm and the residual path stay fp32."""
    precision = emphases_precision()
    if precision != _lib.PREC_FP32 and tensor_core_shape(stack):
        return _lib.PREC_BF16X6_TC if precision == _lib.PREC_BF16X6_TC else _lib.PREC_BF16X3_TC
    return _lib.PREC_FP32


def emphases_precision():
    import emphases_b200
    return emphases_b200.precision_code()


def frame_precision(precision, stack):
    """Tensor-core modes apply to shapes the tcgen05 kernel is compiled for;
    any other conv shape runs on the (stricter) fp32 FFMA kernel"""
    if precision != _lib.PREC_FP32 and not tensor_core_shape(stack):
        return _lib.PREC_FP32
    return precision


def word_precision(precision, stack):
    """The word decoder always runs at fp32 grade (bf16 there costs 1.5e-3 of
    the 2e-3 budget, SURVEY.md section 7): on the tensor cores as bf16x3 when
    a tensor-core mode is selected and the shape is compiled in, else FFMA"""
    if precision == _lib.PREC_BF16X6_TC and tensor_core_shape(stack):
        return _lib.PREC_BF16X6_TC
    if precision != _lib.PREC_FP32 and tensor_core_shape(stack):
        return _lib.PREC_BF16X3_TC
    return _lib.PREC_FP32


class Workspace:
    """Grow-only device buffers reused across launches.  Launch sizes vary, so
    fresh torch allocations make the caching allocator fragment and fall back
    to cudaMalloc (50-200 ms stalls); a workspace per stream slot makes the
    steady state allocation-free.  Buffers are handed out as views, valid
    until the next launch that uses the same workspace."""

    def __init__(self, device):
        self.device = device
        self.buffers = {}

    def get(self, name, shape, dtype):
        numel = 1
        for extent in shape:
            numel *= int(extent)
        buffer = self.buffers.get(name)
        if buffer is None or buffer.numel() < numel or buffer.dtype != dtype:
            # 10 % headroom: launches of one corpus have similar sizes
            buffer = torch.empty(
                max(int(numel * 1.1) + 16, 16), dtype=dtype, device=self.device)
            self.buffers[name] = buffer
        return buffer[:numel].view(*shape)


def _empty(ws, name, shape, dtype, device):
    if ws is None:
        return torch.empty(shape, dtype=dtype, device=device)
    return ws.get(name, shape, dtype)



class Engine:
    """Owns device-side constants and launches the kernels of one GPU"""

    def __init__(self, device, n_mels=80):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.EmphasesB200Error(
                'emphases_b200 runs on CUDA devices only (no CPU fallback)')
        _lib.load()
        self.n_mels = n_mels
        with torch.cuda.device(self.device):
            ptr, col, val = basis_to_csr(mel_basis(n_mels=n_mels))
            self.mel_ptr = torch.from_numpy(ptr).to(self.device)
            self.mel_col = torch.from_numpy(col).to(self.device)
            self.mel_val = torch.from_numpy(val).to(self.device)
        self._pinned = {}
        self._workspaces = {}

    def workspace(self, slot):
        if slot not in self._workspaces:
            self._workspaces[slot] = Workspace(self.device)
        return self._workspaces[slot]

    # -- host staging ------------------------------------------------------

    def pinned(self, key, numel, dtype):
        """Grow-only pinned staging buffer"""
        buffer = self._pinned.get(key)
        if buffer is None or buffer.numel() < numel or buffer.dtype != dtype:
            buffer = torch.empty(
                max(numel, 1), dtype=dtype, pin_memory=True)
            self._pinned[key] = buffer
        return buffer[:numel]

    def upload_plan(self, plan: Plan, slot=0, ws=None):
        """One H2D copy for all int32 index arrays (+ one for int64 offsets).
        `slot` selects the pinned staging buffer: launches whose copies may
        still be in flight must not share one."""
        blob = plan.int32_blob()
        staging = self.pinned(('plan32', slot), len(blob), torch.int32)
        staging.numpy()[:] = blob
        device_blob = _empty(ws, 'plan32', (len(blob),), torch.int32, self.device)
        device_blob.copy_(staging, non_blocking=True)
        off_staging = self.pinned(
            ('plan64', slot), max(plan.n_seq, 1), torch.int64)
        off_staging.numpy()[:plan.n_seq] = plan.audio_off
        audio_off = _empty(
            ws, 'plan64', (off_staging.numel(),), torch.int64, self.device)
        audio_off.copy_(off_staging, non_blocking=True)
        n, w = plan.n_seq, plan.total_word_rows
        sizes = [n, n, n, n, n, n, n, w, w, w]
        names = [
            'audio_len', 'chunk_start', 'chunk_len', 'row_start', 'n_rows',
            'word_row_start', 'n_words', 'word_seq', 'word_lo', 'word_hi']
        views, cursor = {}, 0
        for name, size in zip(names, sizes):
            views[name] = device_blob[cursor:cursor + size]
            cursor += size
        views['audio_off'] = audio_off
        return views

    # -- kernels -----------------------------------------------------------

    def row_index(self, row_start, n_rows, n_seq, total_rows, ws=None, name='row_seq'):
        row_seq = _empty(ws, name, (total_rows,), torch.int32, self.device)
        _lib.call(
            'emph_row_index', _lib.ptr(row_start), _lib.ptr(n_rows), n_seq,
            _lib.ptr(row_seq), total_rows, _lib.stream_ptr())
        return row_seq

    def logmel(self, audio, views, plan, row_seq, normalize=False, ws=None,
               resample=None):
        """resample: None, or the fused sample-rate conversion -- `audio` is then
        packed at the source rate and `resample` holds the device filter bank
        (resampling.device_bank) plus per-sequence `source_off` (int64) and
        `source_len` (int32) in source samples; the plan stays in 16 kHz samples"""
        out = _empty(
            ws, 'features', (plan.total_rows, self.n_mels), torch.float32,
            self.device)
        if resample is not None:
            name = {torch.float32: 'emph_logmel_resampled_f32',
                    torch.int16: 'emph_logmel_resampled_i16'}[audio.dtype]
            bank = resample['bank']
            _lib.call(
                name, _lib.ptr(audio), _lib.ptr(resample['source_off']),
                _lib.ptr(resample['source_len']), _lib.ptr(views['audio_len']),
                _lib.ptr(views['chunk_start']), _lib.ptr(views['chunk_len']),
                _lib.ptr(views['row_start']), plan.n_seq, _lib.ptr(row_seq),
                plan.total_rows, _lib.ptr(self.mel_ptr), _lib.ptr(self.mel_col),
                _lib.ptr(self.mel_val), self.n_mels, int(bool(normalize)),
                _lib.ptr(bank['filter']), _lib.ptr(bank['tap_lo']),
                _lib.ptr(bank['tap_hi']), bank['orig'], bank['new'], bank['width'],
                _lib.ptr(out), _lib.stream_ptr())
            return out
        name = {torch.float32: 'emph_logmel_f32', torch.int16: 'emph_logmel_i16'}[
            audio.dtype]
        _lib.call(
            name, _lib.ptr(audio), _lib.ptr(views['audio_off']),
            _lib.ptr(views['audio_len']), _lib.ptr(views['chunk_start']),
            _lib.ptr(views['chunk_len']), _lib.ptr(views['row_start']),
            plan.n_seq, _lib.ptr(row_seq), plan.total_rows,
            _lib.ptr(self.mel_ptr), _lib.ptr(self.mel_col),
            _lib.ptr(self.mel_val), self.n_mels, int(bool(normalize)),
            _lib.ptr(out), _lib.stream_ptr())
        return out

    def widen(self, x, channels, ws=None, name='widened'):
        """Zero-extend packed rows to `channels` columns"""
        y = _empty(ws, name, (x.shape[0], channels), torch.float32, self.device)
        _lib.call(
            'emph_widen_rows', _lib.ptr(x), x.shape[0], x.shape[1], channels,
            _lib.ptr(y), _lib.stream_ptr())
        return y

    def conv_stack(self, x, row_seq, stack: ConvStack, precision, ws=None,
                   name='conv'):
        if x.shape[1] < stack.channels:
            # the 80 log-mel features entering a wider model
            x = self.widen(x, stack.channels, ws, name + '_in')
        y = _empty(ws, name, tuple(x.shape), torch.float32, self.device)
        acts = stack.acts.astype(np.int32)
        weights = stack.weights if precision == _lib.PREC_FP32 \
            else stack.tensor_core_weights(precision)
        _lib.call(
            'emph_conv_stack', _lib.ptr(x), _lib.ptr(row_seq), x.shape[0],
            _lib.ptr(weights), _lib.ptr(stack.bias),
            acts.ctypes.data_as(ctypes.c_void_p), stack.n_layers,
            stack.channels, stack.kernel_size, precision, _lib.ptr(y),
            _lib.stream_ptr())
        return y

    def conv_stack_pool(self, x, row_seq, stack: ConvStack, precision, views,
                        total_word_rows, method, ws=None, keep_frames=False):
        """conv_stack followed by pool in ONE kernel (emph_conv_stack_pool):
        returns (pooled, frames or None); None when the configuration is not
        fused (the caller then runs the two kernels)"""
        last = int(stack.acts[-1])
        if (
            precision == _lib.PREC_FP32 or not tensor_core_shape(stack) or
            stack.kernel_size == 1 or x.shape[1] != stack.channels or
            not (last == _lib.ACT_RELU or (last == _lib.ACT_NONE and method != 'max'))
        ):
            return None
        rows, channels = x.shape[0], stack.channels
        pooled = _empty(
            ws, 'pooled', (total_word_rows, channels), torch.float32, self.device)
        frames = _empty(ws, 'frames', (rows, channels), torch.float32, self.device) \
            if keep_frames else None
        row_word = _empty(ws, 'row_word', (rows,), torch.int32, self.device)
        word_count = _empty(ws, 'word_count', (total_word_rows,), torch.int32, self.device)
        fixed = _empty(
            ws, 'pooled_fixed', (total_word_rows, channels), torch.int64, self.device) \
            if method in ('sum', 'average') else None
        acts = stack.acts.astype(np.int32)
        _lib.call(
            'emph_conv_stack_pool', _lib.ptr(x), _lib.ptr(row_seq), rows,
            _lib.ptr(stack.tensor_core_weights(precision)),
            acts.ctypes.data_as(ctypes.c_void_p), stack.n_layers, channels,
            stack.kernel_size, precision, _lib.ptr(views['row_start']),
            _lib.ptr(views['n_rows']), _lib.ptr(views['word_seq']),
            _lib.ptr(views['word_lo']), _lib.ptr(views['word_hi']), total_word_rows,
            _lib.POOL[method], _lib.ptr(row_word), _lib.ptr(word_count),
            _lib.ptr(fixed) if fixed is not None else None, _lib.ptr(pooled),
            _lib.ptr(frames) if frames is not None else None, _lib.stream_ptr())
        return pooled, frames

    def pool(self, x, row_start, n_rows, word_seq, word_lo, word_hi, method,
             ws=None):
        total_word_rows = word_seq.shape[0]
        y = _empty(
            ws, 'pooled', (total_word_rows, x.shape[1]), torch.float32,
            self.device)
        _lib.call(
            'emph_pool_words', _lib.ptr(x), x.shape[1], _lib.ptr(row_start),
            _lib.ptr(n_rows), _lib.ptr(word_seq), _lib.ptr(word_lo),
            _lib.ptr(word_hi), total_word_rows, _lib.POOL[method], _lib.ptr(y),
            _lib.stream_ptr())
        return y

    def head(self, x, row_seq, weights: ModelWeights, mode, want_logits=True,
             want_scores=True, ws=None):
        rows = x.shape[0]
        logits = _empty(ws, 'logits', (rows,), torch.float32, self.device) \
            if want_logits else None
        scores = _empty(ws, 'scores', (rows,), torch.float32, self.device) \
            if want_scores else None
        _lib.call(
            'emph_output_head', _lib.ptr(x), _lib.ptr(row_seq), rows,
            weights.channels, weights.head_kernel, _lib.ptr(weights.head_weight),
            weights.head_bias, mode, _lib.ptr(logits), _lib.ptr(scores),
            _lib.stream_ptr())
        return logits, scores

    # -- whole path --------------------------------------------------------

    def prepare_weights(self, weights, precision):
        """Pack (and cache) the tensor-core operand blobs the packed path will
        use at `precision`, on the current stream"""
        if hasattr(weights, 'input_layer'):      # transformer variant: packed by its own code
            return
        with _lib.same_stream():
            chosen = frame_precision(precision, weights.frame)
            if chosen != _lib.PREC_FP32:
                weights.frame.tensor_core_weights(chosen)
            if weights.word is not None:
                chosen = word_precision(precision, weights.word)
                if chosen != _lib.PREC_FP32:
                    weights.word.tensor_core_weights(chosen)

    def forward_packed(
        self,
        audio,
        plan: Plan,
        weights: ModelWeights,
        method='sum',
        location='intermediate',
        precision=_lib.PREC_FP32,
        head_mode=_lib.HEAD_SIGMOID,
        normalize=False,
        views=None,
        keep=False,
        timers=None,
        ws=None,
        resample=None
    ):
        """audio: packed device tensor (fp32 or int16).  Returns dict with
        `scores` and `logits` per packed word row (device tensors).
        resample: see Engine.logmel."""
        if location not in ('intermediate', 'loss', 'inference'):
            raise ValueError(
                f'Downsample location {location} not handled by the packed path')
        with _lib.same_stream():
            return self._forward_packed(
                audio, plan, weights, method, location, precision, head_mode,
                normalize, views, keep, timers, ws, resample)

    def _forward_packed(
        self, audio, plan, weights, method, location, precision, head_mode,
        normalize, views, keep, timers, ws, resample=None
    ):
        if views is None:
            views = self.upload_plan(plan)

        def timed(name, launch, kernels=1):
            # CUDA events on the launch stream around one stage (bench.py);
            # `kernels` = kernel launches of ours the stage issues
            if timers is None:
                return launch()
            start = torch.cuda.Event(enable_timing=True)
            end = torch.cuda.Event(enable_timing=True)
            start.record()
            output = launch()
            end.record()
            timers[name] = (start, end, kernels)
            return output

        row_seq = timed('row_index_frames', lambda: self.row_index(
            views['row_start'], views['n_rows'], plan.n_seq, plan.total_rows,
            ws))
        word_row_seq = timed('row_index_words', lambda: self.row_index(
            views['word_row_start'], views['n_words'], plan.n_seq,
            plan.total_word_rows, ws, 'word_row_seq'))
        features = timed('logmel', lambda: self.logmel(
            audio, views, plan, row_seq, normalize, ws, resample))
        transformer_variant = hasattr(weights, 'input_layer')
        pooled = None
        if transformer_variant:
            from . import transformer
            embedded = self.conv_stack(
                features, row_seq, weights.input_layer,
                linear_precision(weights.input_layer))
            frames = timed('conv_frames', lambda: transformer.run_stack(
                self, weights.frame, embedded, views['row_start'], plan.n_rows,
                plan.n_rows, row_seq, self.device, ws, 'frame_'))
        else:
            fused = None
            if location == 'intermediate' and plan.words_disjoint() and fuse_pooling(
                    frame_precision(precision, weights.frame)):
                # frame stack + word pooling in one kernel: the frame embeddings
                # never travel to HBM (kept only on request)
                # (word-of-row map, conv + pooling, fixed point -> fp32 for sums)
                fused = timed('conv_frames', lambda: self.conv_stack_pool(
                    features, row_seq, weights.frame,
                    frame_precision(precision, weights.frame), views,
                    plan.total_word_rows, method, ws, keep_frames=keep),
                    kernels=3 if method in ('sum', 'average') else 2)
            if fused is not None:
                pooled, frames = fused
            else:
                frames = timed('conv_frames', lambda: self.conv_stack(
                    features, row_seq, weights.frame,
                    frame_precision(precision, weights.frame), ws, 'frames'))
        if pooled is None:
            pooled = timed('pool', lambda: self.pool(
                frames, views['row_start'], views['n_rows'], views['word_seq'],
                views['word_lo'], views['word_hi'], method, ws))
        if location == 'intermediate' and transformer_variant:
            from . import transformer
            words = timed('conv_words', lambda: transformer.run_stack(
                self, weights.word, pooled, views['word_row_start'],
                plan.n_words, plan.n_words, word_row_seq, self.device, ws, 'word_'))
        elif location == 'intermediate':
            words = timed('conv_words', lambda: self.conv_stack(
                pooled, word_row_seq, weights.word,
                word_precision(precision, weights.word), ws, 'words'))
        else:
            words = pooled
        logits, scores = timed('head', lambda: self.head(
            words, word_row_seq, weights, head_mode, ws=ws))
        result = {'scores': scores, 'logits': logits}
        if keep:
            result.update(
                features=features, frames=frames, pooled=pooled,
                row_seq=row_seq, word_row_seq=word_row_seq, views=views)
        return result
