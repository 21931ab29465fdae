"""`emphases.Model` mirror (emphases/model/core.py:13-138).

The module holds exactly the reference's parameters (same `state_dict` keys,
SURVEY.md A.8) so reference checkpoints load unchanged; `forward` has the
reference's signature and return shape but runs the sm_100a kernels of
libemphases_b200.so on packed rows.  There is no PyTorch compute fallback.
"""
import functools

import numpy as np
import torch

import emphases_b200 as emphases
from . import _lib, engine


class Convolution(torch.nn.Sequential):
    """Parameter container mirroring emphases/model/layers/convolution.py"""

    def __init__(self, kernel_size):
        conv_fn = functools.partial(
            torch.nn.Conv1d, kernel_size=kernel_size, padding='same')
        layers = []
        channels = emphases.CHANNELS
        for _ in range(emphases.LAYERS):
            layers.extend((
                conv_fn(channels, channels),
                emphases.ACTIVATION_FUNCTION()))
            if emphases.DROPOUT is not None:
                layers.append(torch.nn.Dropout(emphases.DROPOUT))
        super().__init__(*layers)

    def forward(self, x, _):
        raise _lib.EmphasesB200Error(
            'submodules are parameter containers; call Model.forward')


def Layers(**kwargs):
    """emphases/model/layers/__init__.py:7-14"""
    if emphases.ARCHITECTURE == 'convolution':
        return Convolution(**kwargs)
    if emphases.ARCHITECTURE == 'transformer':
        from .transformer import Transformer
        return Transformer()
    raise ValueError(
        f'Network layer {emphases.ARCHITECTURE} is not defined')


def mask_from_lengths(lengths):
    """emphases/model/core.py:146-149"""
    x = torch.arange(
        lengths.max(), dtype=lengths.dtype, device=lengths.device)
    return (x.unsqueeze(0) < lengths.unsqueeze(1)).unsqueeze(1)


class Model(torch.nn.Module):

    def __init__(self):
        super().__init__()
        # Configuration is captured at construction, like the reference
        # module structure is
        self.architecture = emphases.ARCHITECTURE
        self.location = emphases.DOWNSAMPLE_LOCATION
        self.layers = emphases.LAYERS
        self.dropout = emphases.DROPOUT
        self.activation = emphases.ACTIVATION_FUNCTION.__name__
        if self.location not in ('input', 'intermediate', 'inference', 'loss'):
            raise ValueError(
                f'Downsample location {self.location} not recognized')
        self.input_layer = torch.nn.Conv1d(
            emphases.NUM_FEATURES,
            emphases.CHANNELS,
            kernel_size=emphases.ENCODER_KERNEL_SIZE,
            padding='same')
        self.frame_encoder = Layers(kernel_size=emphases.ENCODER_KERNEL_SIZE)
        if self.location in ['input', 'intermediate']:
            self.word_decoder = Layers(
                kernel_size=emphases.DECODER_KERNEL_SIZE)
        self.output_layer = torch.nn.Conv1d(
            emphases.CHANNELS,
            1,
            kernel_size=emphases.DECODER_KERNEL_SIZE,
            padding='same')
        self._packed = None
        self._packed_key = None

    # -- weights -----------------------------------------------------------

    def packed_weights(self):
        """Kernel-layout weights, re-packed only when parameters change"""
        # (walking the module tree costs more than a small launch: the
        # Parameter objects are stable, only their storage / version change)
        parameters = getattr(self, '_parameter_list', None)
        if parameters is None:
            parameters = list(self.parameters())
            object.__setattr__(self, '_parameter_list', parameters)
        device = parameters[0].device
        key = (device, tuple((p.data_ptr(), p._version) for p in parameters))
        if self._packed_key != key:
            if self.architecture == 'transformer':
                from . import transformer
                self._packed = transformer.pack_weights(self, device)
            else:
                self._packed = engine.pack_weights(
                    self.state_dict(), device, self.layers, self.activation,
                    self.dropout, hasattr(self, 'word_decoder'))
            self._packed_key = key
        return self._packed

    # -- forward -----------------------------------------------------------

    def forward(self, features, frame_lengths, word_bounds, word_lengths):
        """features (B, F, T) fp32 CUDA; word_bounds (B, 2, Wmax) int64;
        returns logits (B, 1, Wmax) fp32 (or (B, 1, T) for the 'inference'
        location in training mode), as emphases/model/core.py:39-138."""
        if features.device.type != 'cuda':
            raise _lib.EmphasesB200Error(
                'emphases_b200.Model runs on CUDA tensors only '
                '(there is no CPU fallback)')
        if self.input_layer.in_channels != emphases.NUM_MELS:
            emphases.require_mel_features_only()
        if torch.is_grad_enabled() and any(
            p.requires_grad for p in self.parameters()
        ) and self.training:
            from . import training
            return training.forward_with_grad(
                self, features, frame_lengths, word_bounds, word_lengths)
        if self.training and self.dropout is not None:
            # the reference applies torch.nn.Dropout after every activation in
            # training mode (emphases/model/layers/convolution.py:29-30); the
            # training step (autograd on) applies it, the inference kernels do not
            raise NotImplementedError(
                'dropout is not implemented in a training-mode forward without '
                'autograd: enable gradients, set DROPOUT=None or call model.eval()')
        with torch.cuda.device(features.device):
            return run_forward(
                self, features, frame_lengths, word_bounds, word_lengths)


def pack_batch(eng, xs):
    """Packed rows of a padded (B, C, T) batch: every item is a sequence of
    all T columns, padding included.  One H2D copy of (row_start, n_rows),
    then emph_row_index and emph_pack_rows.  Returns (rows, row_seq, device
    row_start, device n_rows, host starts, total rows)."""
    batch, channels, frames = xs.shape
    device = eng.device
    starts, total = engine.packed_starts([frames] * batch)
    meta = torch.from_numpy(np.concatenate([
        starts.astype(np.int32), np.full(batch, frames, dtype=np.int32)])
    ).to(device)
    row_start, n_rows = meta[:batch], meta[batch:]
    row_seq = eng.row_index(row_start, n_rows, batch, total)
    rows = torch.empty((total, channels), dtype=torch.float32, device=device)
    xs = xs.detach().to(device, torch.float32).contiguous()
    _lib.call(
        'emph_pack_rows', _lib.ptr(xs), batch, channels, frames,
        _lib.ptr(row_start), _lib.ptr(n_rows), _lib.ptr(row_seq), total,
        _lib.ptr(rows), _lib.stream_ptr())
    return rows, row_seq, row_start, n_rows, starts, total


def slot_index(starts, width, device):
    """(B, width) int64 device index of the packed rows of every item's
    `width` slots: row starts[b] + j"""
    return torch.from_numpy(
        (starts[:, None] + np.arange(width)[None]).astype(np.int64)).to(device)


def check_word_bounds(bounds, lengths, frames, method):
    """Raise where the reference's downsample raises, for the slots j <
    lengths[b] of host bounds (B, 2, W) over a padded batch of `frames`
    columns"""
    valid = np.arange(bounds.shape[2])[None] < lengths[:, None]
    engine.validate_bounds(
        np.stack([bounds[:, 0][valid], bounds[:, 1][valid]], axis=1),
        frames, method)


def slot_views(word_seq, word_lo, word_hi, device):
    """Device word-row arrays of a padded batch from (B, W) host arrays: every
    item gets W slots, separator rows read (-1, 0, 0).  One H2D copy.
    Returns (views, host word starts, total word rows)."""
    batch, width = word_seq.shape
    starts, total = engine.packed_starts([width] * batch)
    rows = np.zeros((3, total), dtype=np.int32)
    rows[0] = -1
    for b, s in enumerate(starts):
        rows[:, s:s + width] = word_seq[b], word_lo[b], word_hi[b]
    blob = torch.from_numpy(np.concatenate([
        starts.astype(np.int32), np.full(batch, width, dtype=np.int32),
        rows.reshape(-1)])).to(device)
    views = {
        'word_row_start': blob[:batch],
        'n_words': blob[batch:2 * batch],
        'word_seq': blob[2 * batch:2 * batch + total],
        'word_lo': blob[2 * batch + total:2 * batch + 2 * total],
        'word_hi': blob[2 * batch + 2 * total:]}
    return views, starts, total


def word_rows(word_bounds, word_lengths, device):
    """Packed word-row arrays for padded (B, 2, Wmax) bounds: every item gets
    Wmax slots; slots j >= word_lengths[i] are marked (-1, -1)"""
    batch, _, wmax = word_bounds.shape
    bounds = word_bounds.detach().to('cpu', torch.int64).numpy()
    lengths = word_lengths.detach().to('cpu', torch.int64).numpy()
    masked = np.arange(wmax)[None] >= lengths[:, None]
    views, starts, total = slot_views(
        np.repeat(np.arange(batch)[:, None], wmax, axis=1),
        np.where(masked, -1, bounds[:, 0]), np.where(masked, -1, bounds[:, 1]),
        device)
    return views, starts, total, bounds, lengths


def conv_encoders(eng, weights, precision):
    """(encode, decode) of the convolution architecture: the frame and word
    conv stacks.  Every packed row is a query and a key alike
    (convolution.py:36-37 ignores the lengths), so the counts go unread."""

    def encode(rows, row_seq, row_start, n_queries, n_keys):
        return eng.conv_stack(
            rows, row_seq, weights.frame,
            engine.frame_precision(precision, weights.frame))

    def decode(pooled, word_row_seq, word_start, n_queries, n_keys):
        return eng.conv_stack(
            pooled, word_row_seq, weights.word,
            engine.word_precision(precision, weights.word))

    return encode, decode


def run_forward(model, features, frame_lengths, word_bounds, word_lengths):
    """Model.forward on packed rows, for both architectures.  The encoder pair
    takes (rows, row_seq, device row_start, host n_queries, n_keys): every
    sequence has n_queries rows, of which the first n_keys are valid keys."""
    eng = emphases.get_engine(features.device)
    weights = model.packed_weights()
    method = emphases.DOWNSAMPLE_METHOD
    if method not in _lib.POOL:
        raise ValueError(f'Interpolation method {method} is not defined')
    precision = emphases.precision_code()
    if model.architecture == 'transformer':
        from . import transformer
        encode, decode = transformer.encoders(eng, weights)
    else:
        encode, decode = conv_encoders(eng, weights, precision)
    device = features.device
    batch, _, frames = features.shape
    wmax = word_bounds.shape[2]
    if model.location == 'input':
        from . import segments
        words, word_row_seq, word_starts = segments.run_forward_input(
            eng, features, word_bounds, word_lengths, method, encode, decode)
    else:
        rows, row_seq, row_start, n_rows, starts, _ = pack_batch(eng, features)
        # frame_lengths goes in as given: only the Transformer reads it on the
        # host (a device tensor costs a sync)
        frame_rows = encode(
            rows, row_seq, row_start, np.full(batch, frames), frame_lengths)
        if model.location == 'inference' and model.training:
            # frame-resolution logits (model/core.py:119-122)
            logits, _ = eng.head(
                frame_rows, row_seq, weights, _lib.HEAD_LOGITS,
                want_scores=False)
            return logits[slot_index(starts, frames, device)][:, None, :]
        views, word_starts, total_words, bounds, lengths = word_rows(
            word_bounds, word_lengths, device)
        check_word_bounds(bounds, lengths, frames, method)
        words = eng.pool(
            frame_rows, row_start, n_rows, views['word_seq'], views['word_lo'],
            views['word_hi'], method)
        word_row_seq = eng.row_index(
            views['word_row_start'], views['n_words'], batch, total_words)
        if model.location == 'intermediate':
            words = decode(
                words, word_row_seq, views['word_row_start'],
                np.full(batch, wmax), lengths)
    logits, _ = eng.head(
        words, word_row_seq, weights, _lib.HEAD_LOGITS, want_scores=False)
    return logits[slot_index(word_starts, wmax, device)][:, None, :]
