"""Training step on device: forward with saved activations, hand-written
backward kernels (csrc/train.cu for the conv model, csrc/attention.cu and
csrc/transformer_train.cu for the Transformer variant), masked loss, and a
flat-bucket gradient all-reduce for data parallelism.

The reference trains on one device (emphases/train/core.py:86-142) with
torch autograd; it has no data-parallel code.  Here `Model.forward` in
training mode goes through `forward_with_grad`: a torch.autograd.Function
whose backward fills the `.grad` of the Model's own torch parameters, so any
torch optimizer (the reference uses Adam, train/core.py:69-75) can step.
"""
import ctypes
import os

import numpy as np
import torch

import emphases_b200 as emphases
from . import _lib, engine


def _layer_list(model):
    """[(weight, bias, act)] per conv layer, frame side then word side"""
    step = 3 if model.dropout is not None else 2
    act = engine.ACTIVATIONS[model.activation]
    frame = [(model.input_layer.weight, model.input_layer.bias, _lib.ACT_NONE)]
    frame += [
        (model.frame_encoder[i * step].weight,
         model.frame_encoder[i * step].bias, act)
        for i in range(model.layers)]
    word = []
    if hasattr(model, 'word_decoder'):
        word = [
            (model.word_decoder[i * step].weight,
             model.word_decoder[i * step].bias, act)
            for i in range(model.layers)]
    return frame, word


def _dropout_rates(model):
    """p of the Dropout after each layer of _layer_list, read from the modules
    (a model whose modules are set to p = 0 trains without dropout); the input
    layer has none (emphases/model/layers/convolution.py:25-30)"""
    if model.dropout is None:
        frame, word = _layer_list(model)
        return [0.] * len(frame), [0.] * len(word)
    frame = [0.] + [float(model.frame_encoder[3 * i + 2].p) for i in range(model.layers)]
    word = []
    if hasattr(model, 'word_decoder'):
        word = [float(model.word_decoder[3 * i + 2].p) for i in range(model.layers)]
    return frame, word


def _draw_seed(model):
    """One dropout seed per training forward from torch's default CPU
    generator (no device sync; torch.manual_seed makes a step reproducible);
    None, and no draw, for a model without dropout modules"""
    if model.architecture == 'convolution' and model.dropout is None:
        return None
    return int(torch.randint(0, 2 ** 62, ()))


def _kernel_width(model):
    """Channel count the conv model trains at, by inference's rule
    (engine.pack_weights): 80, or 128 when its widest conv is wider.  Its
    weights and biases are zero-padded to it: a padded channel stays zero
    through every layer, as act(0) = 0 and dropout keeps a zero a zero."""
    frame, word = _layer_list(model)
    largest = max(max(w.shape[0], w.shape[1]) for w, _, _ in frame + word)
    if largest > engine.WIDE_CHANNELS:
        raise NotImplementedError(
            f'the training kernels are built for up to {engine.WIDE_CHANNELS} '
            f'channels (this model has {largest})')
    return engine.kernel_width(largest)


def _stack(weight, bias, act, device, width, backward=False):
    """One-layer ConvStack at `width` channels (the weight zero-padded to
    (width, width, k)); backward=True packs the adjoint (taps flipped, channel
    matrix transposed) with zero bias and no activation"""
    kernel = weight.shape[2]
    padded = engine.pad(weight, (width, width, kernel))
    if backward:
        source = padded.to(device).contiguous()
        packed = torch.empty((kernel, width, width), dtype=torch.float32, device=device)
        _lib.call(
            'emph_pack_conv_weights_adjoint', _lib.ptr(source), width, width, kernel,
            _lib.ptr(packed), _lib.stream_ptr())
        bias = _zero_bias(width, device)
        act = _lib.ACT_NONE
    else:
        packed = engine._pack_conv(padded, device)      # [k][in][out]
        bias = engine.pad(bias, (width,)).to(device)
    return engine.ConvStack(
        packed[None], bias[None], np.asarray([act], dtype=np.int32), kernel, width)


_zero_biases = {}


def _zero_bias(channels, device):
    key = (channels, device)
    if key not in _zero_biases:
        _zero_biases[key] = torch.zeros(channels, dtype=torch.float32, device=device)
    return _zero_biases[key]


def _conv_dropout(x, seq, act, drop, y):
    """y = act(x) * keep / (1 - p) (emph_conv_dropout_forward); `drop` is
    (seed, site, p, device row_start, width)"""
    seed, site, p, row_start, width = drop
    _lib.call(
        'emph_conv_dropout_forward', _lib.ptr(x), _lib.ptr(seq), _lib.ptr(row_start),
        x.shape[0], x.shape[1], width, act, seed, site, p, _lib.ptr(y), _lib.stream_ptr())


def _layer_forward(eng, x, seq, weight, bias, act, device, drop=None):
    """One conv layer of the training forward on rows `x` of the kernel
    width, with the dropout `drop` of _conv_dropout after it (None: none):
    (output, what emph_activation_backward needs): GELU / SiLU keep the
    pre-activation, the others their (dropped) output"""
    width = x.shape[1]
    if act in (_lib.ACT_GELU, _lib.ACT_SILU):
        pre = eng.conv_stack(
            x, seq, _stack(weight, bias, _lib.ACT_NONE, device, width), _lib.PREC_FP32)
        y = torch.empty_like(pre)
        if drop is not None:
            _conv_dropout(pre, seq, act, drop, y)
        else:
            _lib.call(
                'emph_activation_forward', _lib.ptr(pre), _lib.ptr(seq),
                pre.shape[0], pre.shape[1], act, _lib.ptr(y), _lib.stream_ptr())
        return y, pre
    y = eng.conv_stack(x, seq, _stack(weight, bias, act, device, width), _lib.PREC_FP32)
    if drop is not None:
        _conv_dropout(y, seq, _lib.ACT_NONE, drop, y)
    return y, y


def _conv_backward(eng, layers, acts, keys, row_seq, dy, grads, drops=None,
                   input_grad=True):
    """Adjoint of conv layers run by _layer_forward (`drops`: their dropout,
    the masks regenerated): weight and bias gradients into `grads`, sliced
    from the kernel width to each parameter's shape; returns the gradient of
    the first layer's input (None without input_grad)"""
    device = dy.device
    channels = dy.shape[1]
    for position in range(len(layers) - 1, -1, -1):
        weight, bias, act = layers[position]
        x_in, y_out = acts[position], keys[position]
        dpre = torch.empty_like(dy)
        drop = drops[position] if drops else None
        if drop is not None:
            seed, site, p, row_start, width = drop
            _lib.call(
                'emph_activation_dropout_backward', _lib.ptr(dy), _lib.ptr(y_out),
                _lib.ptr(row_seq), _lib.ptr(row_start), dy.shape[0], channels, width, act,
                seed, site, p, _lib.ptr(dpre), _lib.stream_ptr())
        else:
            _lib.call(
                'emph_activation_backward', _lib.ptr(dy), _lib.ptr(y_out),
                _lib.ptr(row_seq), dy.shape[0], channels, act,
                _lib.ptr(dpre), _lib.stream_ptr())
        kernel = weight.shape[2]
        dw = torch.empty(
            (kernel, channels, channels), dtype=torch.float32,
            device=device)
        db = torch.empty(channels, dtype=torch.float32, device=device)
        _lib.call(
            'emph_conv_weight_grad', _lib.ptr(x_in), _lib.ptr(dpre),
            dy.shape[0], channels, kernel, _lib.ptr(dw), _lib.ptr(db),
            _lib.stream_ptr())
        out_channels, in_channels, _ = weight.shape
        grads[weight] = dw.permute(2, 1, 0)[:out_channels, :in_channels].contiguous()
        grads[bias] = db[:out_channels]
        if position == 0 and not input_grad:
            return None
        dy = eng.conv_stack(
            dpre, row_seq,
            _stack(weight, bias, act, device, channels, backward=True),
            _lib.PREC_FP32)
    return dy


def _conv_encoders(eng, model, device, seed=None):
    """(encode, decode, encode_backward, decode_backward) of the conv model
    for _model_forward / _model_backward: the frame layers (input layer
    included) and the word layers, with dropout drawn from `seed`.  The conv
    layers read every packed row, so the key counts go unread; every sequence
    has n_queries[0] rows, the padded width that places a row in the dropout
    masks (T, max_length at 'input', or Wmax).  Every layer runs at the
    kernel width (_kernel_width): the 80 input features enter a wider model
    widened, and the masks are drawn over the padded channels.  The frame
    stack's input gradient is not computed: the features carry none."""
    frame_layers, word_layers = _layer_list(model)
    frame_rates, word_rates = _dropout_rates(model)
    kernel_width = _kernel_width(model)

    def run(layers, rates, stack):
        # frame stack: layer 0 is the input layer, block i - 1 of frame_encoder
        first_block = -1 if stack == 0 else 0

        def forward(x, row_seq, row_start, n_queries, n_keys):
            width = max(int(n_queries[0]), 1) if len(n_queries) else 1
            if x.shape[1] < kernel_width:
                x = eng.widen(x, kernel_width)
            acts, keys, drops = [x], [], []
            for i, ((weight, bias, act), p) in enumerate(zip(layers, rates)):
                drop = None
                if p > 0:
                    site = _lib.dropout_site(stack, first_block + i, _lib.DROPOUT_CONV)
                    drop = (seed, site, p, row_start, width)
                y, key = _layer_forward(
                    eng, acts[-1], row_seq, weight, bias, act, device, drop)
                acts.append(y)
                keys.append(key)
                drops.append(drop)
            return acts[-1], (acts, keys, row_seq, drops)

        def backward(saved, dy, grads):
            acts, keys, row_seq, drops = saved
            return _conv_backward(
                eng, layers, acts, keys, row_seq, dy, grads, drops, input_grad=stack != 0)
        return forward, backward

    encode, encode_backward = run(frame_layers, frame_rates, 0)
    decode, decode_backward = run(word_layers, word_rates, 1)
    return encode, decode, encode_backward, decode_backward


def _transformer_encoders(eng, model, device, seed):
    """The same four functions for the Transformer variant: the input layer and
    the frame encoder, and the word decoder (transformer.stack_forward_train /
    stack_backward), dropout drawn from `seed`"""
    from . import transformer
    tables = model.packed_weights()
    input_layer = [(model.input_layer.weight, model.input_layer.bias, _lib.ACT_NONE)]

    def encode(rows, row_seq, row_start, n_queries, n_keys):
        embedded, key = _layer_forward(eng, rows, row_seq, *input_layer[0], device)
        out, saved = transformer.stack_forward_train(
            model.frame_encoder, tables.frame.table, embedded, row_start, n_queries,
            n_keys, row_seq, seed, 0)
        return out, ([rows, embedded], [key], row_seq, saved)

    def encode_backward(saved, dy, grads):
        acts, keys, row_seq, stack = saved
        d_embedded, stack_grads = transformer.stack_backward(stack, dy)
        grads.update(stack_grads)
        return _conv_backward(eng, input_layer, acts, keys, row_seq, d_embedded, grads)

    def decode(pooled, word_row_seq, word_start, n_queries, n_keys):
        if not hasattr(model, 'word_decoder'):
            return pooled, None
        return transformer.stack_forward_train(
            model.word_decoder, tables.word.table, pooled, word_start, n_queries,
            n_keys, word_row_seq, seed, 1)

    def decode_backward(saved, dy, grads):
        if saved is None:
            return dy
        d_pooled, stack_grads = transformer.stack_backward(saved, dy)
        grads.update(stack_grads)
        return d_pooled

    return encode, decode, encode_backward, decode_backward


def _model_forward(ctx, model, features, frame_lengths, word_bounds, word_lengths, encoders):
    """Training forward on packed rows for both architectures, with the encoder
    functions of _conv_encoders / _transformer_encoders; keeps in ctx.saved
    what _model_backward reads"""
    from . import model as model_module
    device = features.device
    eng = emphases.get_engine(device)
    method = emphases.DOWNSAMPLE_METHOD
    if method not in _lib.POOL:
        raise ValueError(f'Interpolation method {method} is not defined')
    if model.architecture == 'convolution':
        _kernel_width(model)                # raises above 128 channels
    elif model.input_layer.out_channels != engine.KERNEL_CHANNELS:
        raise NotImplementedError(
            f'the Transformer variant trains at {engine.KERNEL_CHANNELS} channels '
            f'(this model has {model.input_layer.out_channels})')
    batch, _, frames = features.shape
    wmax = word_bounds.shape[2]
    with torch.cuda.device(device), _lib.same_stream():
        encode, decode, _, _ = encoders(eng, model, device)
        input_location = model.location == 'input'
        if input_location:
            # every word segment is a packed sequence of max_length rows
            # (emphases/model/core.py:41-87) that attends over its own
            # frames; the features carry no gradient, so the gather needs
            # no adjoint
            from . import segments
            _, word_counts, max_length, lo, count = segments._segment_plan(
                word_bounds, word_lengths, frames)
            rows, row_seq, row_start, n_rows, _, total = segments._gather(
                eng, features, lo, count, max_length)
            n_queries, n_keys = np.full(lo.size, max_length), count.reshape(-1)
        else:
            rows, row_seq, row_start, n_rows, starts, total = \
                model_module.pack_batch(eng, features)
            n_queries = np.full(batch, frames)
            n_keys = None if frame_lengths is None else \
                frame_lengths.detach().to('cpu', torch.int64).numpy()
        frame_rows, frame_saved = encode(rows, row_seq, row_start, n_queries, n_keys)
        weights = model.packed_weights()
        if model.location == 'inference':
            # frame-resolution logits (model/core.py:119-122)
            logits, _ = eng.head(
                frame_rows, row_seq, weights, _lib.HEAD_LOGITS,
                want_scores=False)
            index = model_module.slot_index(starts, frames, device)
            ctx.model = model
            ctx.saved = dict(
                frame_saved=frame_saved, frame_rows=frame_rows,
                row_seq=row_seq, index=index,
                total=total, head_weight=weights.head_weight,
                head_kernel=weights.head_kernel, frame_level=True)
            return logits[index][:, None, :]
        if input_location:
            views, word_starts, total_words = segments.input_word_rows(
                batch, wmax, word_counts, count, max_length, method, device)
        else:
            views, word_starts, total_words, bounds, word_counts = \
                model_module.word_rows(word_bounds, word_lengths, device)
        pooled = eng.pool(
            frame_rows, row_start, n_rows, views['word_seq'],
            views['word_lo'], views['word_hi'], method)
        word_row_seq = eng.row_index(
            views['word_row_start'], views['n_words'], batch, total_words)
        word_rows, word_saved = decode(
            pooled, word_row_seq, views['word_row_start'], np.full(batch, wmax),
            word_counts)
        logits, _ = eng.head(
            word_rows, word_row_seq, weights, _lib.HEAD_LOGITS,
            want_scores=False)
        index = model_module.slot_index(word_starts, wmax, device)
    ctx.model = model
    ctx.saved = dict(
        frame_saved=frame_saved, word_saved=word_saved, frame_rows=frame_rows,
        word_rows=word_rows, row_seq=row_seq,
        word_row_seq=word_row_seq, row_start=row_start, n_rows=n_rows,
        views=views, index=index, total=total, total_words=total_words,
        method=method, head_weight=weights.head_weight,
        head_kernel=weights.head_kernel, frame_level=False)
    return logits[index][:, None, :]


def _model_backward(ctx, grad_logits, encoders):
    """Gradients of every parameter, in model.parameters() order"""
    model, s = ctx.model, ctx.saved
    device = grad_logits.device
    eng = emphases.get_engine(device)
    channels = s['frame_rows'].shape[1]
    frame_level = s['frame_level']
    with torch.cuda.device(device), _lib.same_stream():
        _, _, encode_backward, decode_backward = encoders(eng, model, device)
        rows = s['total'] if frame_level else s['total_words']
        head_seq = s['row_seq'] if frame_level else s['word_row_seq']
        dz = torch.zeros(rows, dtype=torch.float32, device=device)
        dz[s['index'].reshape(-1)] = grad_logits.reshape(-1).to(torch.float32)
        grads = {}

        # output projection
        x = s['frame_rows'] if frame_level else s['word_rows']
        dx = torch.empty_like(x)
        dw = torch.empty_like(s['head_weight'])
        db = torch.empty(1, dtype=torch.float32, device=device)
        _lib.call(
            'emph_output_head_backward', _lib.ptr(x), _lib.ptr(dz),
            _lib.ptr(head_seq), rows, channels,
            s['head_kernel'], _lib.ptr(s['head_weight']), _lib.ptr(dx),
            _lib.ptr(dw), _lib.ptr(db), _lib.stream_ptr())
        grads[model.output_layer.weight] = \
            dw.t()[None, :model.output_layer.in_channels].contiguous()
        grads[model.output_layer.bias] = db

        if frame_level:
            encode_backward(s['frame_saved'], dx, grads)
        else:
            d_pooled = decode_backward(s['word_saved'], dx, grads)
            d_frames = torch.empty_like(s['frame_rows'])
            views = s['views']
            _lib.call(
                'emph_pool_words_backward', _lib.ptr(d_pooled),
                _lib.ptr(s['frame_rows']), channels, _lib.ptr(s['row_start']),
                _lib.ptr(s['n_rows']), _lib.ptr(views['word_seq']),
                _lib.ptr(views['word_lo']), _lib.ptr(views['word_hi']),
                s['total_words'], _lib.POOL[s['method']], s['total'],
                _lib.ptr(d_frames), _lib.stream_ptr())
            encode_backward(s['frame_saved'], d_frames, grads)
    return [
        grads[p].to(p.dtype) if p in grads else None
        for p in model.parameters()]


class _ConvModelFunction(torch.autograd.Function):
    """Per-kernel training step of the conv model; a model with dropout
    modules draws one seed per forward (_draw_seed), from which the backward
    regenerates the masks"""

    @staticmethod
    def forward(ctx, model, features, word_bounds, word_lengths, *parameters):
        if model.architecture != 'convolution':
            raise NotImplementedError(
                'the training step is built for the convolution architecture')
        seed = ctx.seed = _draw_seed(model)
        return _model_forward(
            ctx, model, features, None, word_bounds, word_lengths,
            lambda eng, model, device: _conv_encoders(eng, model, device, seed))

    @staticmethod
    def backward(ctx, grad_logits):
        seed = ctx.seed
        return (None, None, None, None, *_model_backward(
            ctx, grad_logits,
            lambda eng, model, device: _conv_encoders(eng, model, device, seed)))


class _TransformerModelFunction(torch.autograd.Function):
    """Training forward and backward of the Transformer variant, with the
    reference's dropout: one seed per forward, drawn from torch's default CPU
    generator (no device sync; torch.manual_seed makes a step reproducible),
    from which the backward regenerates every mask"""

    @staticmethod
    def forward(ctx, model, features, frame_lengths, word_bounds, word_lengths, *parameters):
        seed = ctx.seed = _draw_seed(model)
        return _model_forward(
            ctx, model, features, frame_lengths, word_bounds, word_lengths,
            lambda eng, model, device: _transformer_encoders(eng, model, device, seed))

    @staticmethod
    def backward(ctx, grad_logits):
        seed = ctx.seed
        return (None, None, None, None, None, *_model_backward(
            ctx, grad_logits,
            lambda eng, model, device: _transformer_encoders(eng, model, device, seed)))


###############################################################################
# Native step: one C-ABI call for the forward, one for the backward
###############################################################################

# Precision of the convolutions of the native step, forward+backward:
# 'bf16x6' (default): tensor cores with hi/mid/lo-split operands, fp32 grade --
# every parameter gradient within 2e-4 of autograd, like the fp32 kernels.
# 'bf16x3' (hi/lo split, 1e-5 class logits) leaves 2e-3 on the gradient of the
# first layer, and so does 'bf16x3+bf16x6' (x3 forward, x6 input gradients:
# the forward's 1e-5 is what the deep gradients amplify); 2.01 instead of
# 2.10 ms per step.  'fp32': the FFMA kernels, 4.1 ms.  In every mode the
# weight gradients run on mma.sync with split bf16 operands (hi*hi + lo*hi +
# hi*lo: 16-bit operands, fp32 accumulation), ~2^-16 relative per product.
TRAIN_PRECISION = os.environ.get('EMPHASES_B200_TRAIN_PRECISION', 'bf16x6')
_TRAIN_PRECISIONS = {
    'fp32': (_lib.PREC_FP32, _lib.PREC_FP32),
    'bf16x3': (_lib.PREC_BF16X3_TC, _lib.PREC_BF16X3_TC),
    'bf16x6': (_lib.PREC_BF16X6_TC, _lib.PREC_BF16X6_TC),
    'bf16x3+bf16x6': (_lib.PREC_BF16X3_TC, _lib.PREC_BF16X6_TC)}


class _NativeState:
    """Per-model launch descriptor, flat gradient buffer and workspace of
    csrc/train_step.cu"""

    def __init__(self, model, device):
        self.device = device
        frame, word = _layer_list(model)
        self.layers = frame + word
        self.n_frame, self.n_word = len(frame), len(word)
        # parameters in descriptor order: (weight, bias) per layer, then the head
        self.ordered = []
        for weight, bias, _ in self.layers:
            self.ordered += [weight, bias]
        self.ordered += [model.output_layer.weight, model.output_layer.bias]
        sizes = [p.numel() for p in self.ordered]
        self.offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self.flat = torch.zeros(int(self.offsets[-1]), dtype=torch.float32, device=device)
        self.zero_bias = torch.zeros(engine.KERNEL_CHANNELS, dtype=torch.float32, device=device)
        self.acts = np.ascontiguousarray(
            np.asarray([act for _, _, act in self.layers], dtype=np.int32))
        self.dropout = np.zeros(len(self.layers), dtype=np.float32)
        count = len(self.layers) + 1
        self.weight_pointers = (ctypes.c_void_p * count)()
        self.bias_pointers = (ctypes.c_void_p * count)()
        self.grad_pointers = (ctypes.c_void_p * (2 * count))()
        self.descriptor = _lib.TrainModel()
        self.workspace = None
        self.generation = 0           # forward calls so far: the workspace holds the last one
        self.pointer_key = None
        self.lib = _lib.load()

    def refresh(self, model):
        """Parameter storage is stable across optimizer steps; re-read the
        pointers only when it moved (model.to(...), load_state_dict)"""
        key = tuple(p.data_ptr() for p in self.ordered)
        if key == self.pointer_key:
            return
        self.pointer_key = key
        weights = [w for w, _, _ in self.layers] + [model.output_layer.weight]
        biases = [b for _, b, _ in self.layers] + [model.output_layer.bias]
        for i, (w, b) in enumerate(zip(weights, biases)):
            self.weight_pointers[i] = w.data_ptr()
            self.bias_pointers[i] = b.data_ptr()
        d = self.descriptor
        d.n_frame_layers, d.n_word_layers = self.n_frame, self.n_word
        d.channels = engine.KERNEL_CHANNELS
        d.kernel_size = int(model.input_layer.weight.shape[2])
        d.head_kernel = int(model.output_layer.weight.shape[2])
        d.acts = self.acts.ctypes.data
        d.weights = ctypes.cast(self.weight_pointers, ctypes.c_void_p)
        d.biases = ctypes.cast(self.bias_pointers, ctypes.c_void_p)
        d.zero_bias = self.zero_bias.data_ptr()

    def views(self, flat=None):
        flat = self.flat if flat is None else flat
        return [
            flat[int(a):int(b)].view(p.shape)
            for a, b, p in zip(self.offsets[:-1], self.offsets[1:], self.ordered)]

    def aliases_flat(self, parameter, index):
        grad = parameter.grad
        return (
            grad is not None and grad.dtype == torch.float32 and grad.is_contiguous() and
            grad.data_ptr() == self.flat.data_ptr() + 4 * int(self.offsets[index]))


def _native_state(model, device):
    state = getattr(model, '_native_train_state', None)
    if state is None or state.device != device:
        state = _NativeState(model, device)
        object.__setattr__(model, '_native_train_state', state)
    state.refresh(model)
    return state


def native_step_supported(model, features):
    """The configurations csrc/train_step.cu is built for"""
    return (
        os.environ.get('EMPHASES_B200_TRAIN_NATIVE', '1') != '0' and
        model.architecture == 'convolution' and
        model.location in ('intermediate', 'loss') and
        emphases.CHANNELS == engine.KERNEL_CHANNELS == emphases.NUM_FEATURES and
        int(model.input_layer.weight.shape[2]) == 3 and
        all(int(w.shape[2]) == 3 for w, _, _ in sum(_layer_list(model), [])) and
        emphases.DOWNSAMPLE_METHOD in _lib.POOL and
        features.dtype == torch.float32 and features.is_cuda and
        TRAIN_PRECISION in _TRAIN_PRECISIONS)


class _NativeConvFunction(torch.autograd.Function):

    @staticmethod
    def forward(ctx, model, features, frame_lengths, word_bounds, word_lengths, *parameters):
        device = features.device
        state = _native_state(model, device)
        features = features.detach().contiguous()
        batch, _, frames = features.shape
        wmax = int(word_bounds.shape[2])
        bounds = word_bounds.detach().to('cpu', torch.int64).contiguous()
        lengths = word_lengths.detach().to('cpu', torch.int64).contiguous()
        # Rows kept per item (see csrc/train_step.cu, kept_rows): a word may end
        # past its item's length (an alignment running past the audio), and the
        # rows it pools must be computed over all padded columns as the
        # reference does, so an item reaches to the last frame any word reads
        # (hi - 1, or the center (lo + hi) // 2)
        lo, hi = bounds[:, 0].numpy(), bounds[:, 1].numpy()
        real = np.arange(wmax)[None] < lengths.numpy()[:, None]
        reach = np.where(real, np.maximum(hi, (lo + hi) // 2 + 1), 0).max(axis=1)
        frame_lengths = torch.from_numpy(np.maximum(
            frame_lengths.detach().to('cpu', torch.int64).numpy(), reach))
        descriptor = state.descriptor
        ctx.seed = _draw_seed(model)
        if ctx.seed is None:
            descriptor.dropout, descriptor.seed = None, 0
        else:
            frame_rates, word_rates = _dropout_rates(model)
            state.dropout[:] = frame_rates + word_rates
            ctx.dropout = state.dropout.copy()
            descriptor.dropout, descriptor.seed = state.dropout.ctypes.data, ctx.seed
        descriptor.pool_method = _lib.POOL[emphases.DOWNSAMPLE_METHOD]
        descriptor.forward_precision, descriptor.precision = _TRAIN_PRECISIONS[TRAIN_PRECISION]
        need = state.lib.emph_train_workspace(ctypes.byref(descriptor), batch, frames, wmax)
        if need < 0:
            raise _lib.EmphasesB200Error(
                'emph_train_workspace: ' + state.lib.emph_last_error().decode())
        if state.workspace is None or state.workspace.numel() < need:
            state.workspace = None
            state.workspace = torch.empty(
                int(need * 1.1) + 4096, dtype=torch.uint8, device=device)
        logits = torch.empty((batch, 1, wmax), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            stream = torch._C._cuda_getCurrentRawStream(device.index)
            status = state.lib.emph_train_forward(
                ctypes.byref(descriptor), features.data_ptr(), batch, frames,
                frame_lengths.data_ptr(), bounds.data_ptr(), lengths.data_ptr(), wmax,
                state.workspace.data_ptr(), state.workspace.numel(),
                logits.data_ptr(), stream)
        if status != 0:
            raise _lib.EmphasesB200Error(
                f'emph_train_forward failed ({status}): ' +
                state.lib.emph_last_error().decode('utf-8', 'replace'))
        state.generation += 1
        ctx.model, ctx.state = model, state
        ctx.generation = state.generation
        ctx.shape = (batch, frames, wmax)
        ctx.frame_lengths = frame_lengths
        return logits

    @staticmethod
    def backward(ctx, grad_logits):
        model, state = ctx.model, ctx.state
        if ctx.generation != state.generation:
            raise RuntimeError(
                'the native training step keeps ONE forward pass of a model alive (its '
                'activations live in a per-model workspace): call backward() before the '
                "next training-mode forward, or set EMPHASES_B200_TRAIN_NATIVE=0 for the "
                'per-kernel path')
        batch, frames, wmax = ctx.shape
        device = grad_logits.device
        grad_logits = grad_logits.detach().to(torch.float32).contiguous()
        # Gradients land in the flat buffer, in the parameters' own layouts.
        # Parameters whose .grad already IS their slice of the flat buffer are
        # accumulated into in place (nothing is returned for them); otherwise
        # fresh views of the buffer are handed to autograd, which adopts them as
        # .grad -- so the data-parallel all-reduce runs on the buffer itself.
        aliased = [state.aliases_flat(p, i) for i, p in enumerate(state.ordered)]
        in_place = all(aliased)
        target = state.flat if (in_place or not any(aliased)) else torch.empty_like(state.flat)
        views = state.views(target)
        for i, view in enumerate(views):
            state.grad_pointers[i] = view.data_ptr()
        if ctx.seed is not None:
            # the descriptor is shared: the masks are this forward's
            state.dropout[:] = ctx.dropout
            state.descriptor.dropout = state.dropout.ctypes.data
            state.descriptor.seed = ctx.seed
        with torch.cuda.device(device):
            stream = torch._C._cuda_getCurrentRawStream(device.index)
            status = state.lib.emph_train_backward(
                ctypes.byref(state.descriptor), grad_logits.data_ptr(), batch, frames,
                ctx.frame_lengths.data_ptr(), wmax,
                state.workspace.data_ptr(), state.workspace.numel(),
                ctypes.cast(state.grad_pointers, ctypes.c_void_p), int(in_place), stream)
        if status != 0:
            raise _lib.EmphasesB200Error(
                f'emph_train_backward failed ({status}): ' +
                state.lib.emph_last_error().decode('utf-8', 'replace'))
        by_parameter = {id(p): v for p, v in zip(state.ordered, views)}
        del views
        ordered = [
            None if in_place else by_parameter.get(id(p)) for p in model.parameters()]
        del by_parameter
        return (None, None, None, None, None, *ordered)


def forward_with_grad(model, features, frame_lengths, word_bounds, word_lengths):
    """Model.forward in training mode (gradients flow to model.parameters())"""
    method = emphases.DOWNSAMPLE_METHOD
    if model.location in ('intermediate', 'loss') and method in ('max', 'center'):
        # raise where the reference's downsample raises; it slices the padded
        # (B, C, T) tensor, so a word may reach any of the T columns
        from . import model as model_module
        model_module.check_word_bounds(
            word_bounds.detach().to('cpu', torch.int64).numpy(),
            word_lengths.detach().to('cpu', torch.int64).numpy(),
            features.shape[2], method)
    if model.architecture == 'transformer':
        return _TransformerModelFunction.apply(
            model, features, frame_lengths, word_bounds, word_lengths,
            *model.parameters())
    if native_step_supported(model, features):
        return _NativeConvFunction.apply(
            model, features, frame_lengths, word_bounds, word_lengths,
            *model.parameters())
    return _ConvModelFunction.apply(
        model, features, word_bounds, word_lengths, *model.parameters())


class _MaskedLoss(torch.autograd.Function):

    @staticmethod
    def forward(ctx, scores, targets, mask, mode):
        device = scores.device
        flat = scores.detach().reshape(-1).to(torch.float32).contiguous()
        target = targets.detach().reshape(-1).to(device, torch.float32).contiguous()
        valid = mask.reshape(-1).to(device, torch.uint8).contiguous()
        loss = torch.empty(1, dtype=torch.float32, device=device)
        grad = torch.empty_like(flat)
        with torch.cuda.device(device), _lib.same_stream():
            _lib.call(
                'emph_masked_loss', _lib.ptr(flat), _lib.ptr(target),
                _lib.ptr(valid), flat.numel(), mode, _lib.ptr(loss),
                _lib.ptr(grad), _lib.stream_ptr())
        ctx.save_for_backward(grad)
        ctx.shape = scores.shape
        return loss[0]

    @staticmethod
    def backward(ctx, grad_output):
        (grad,) = ctx.saved_tensors
        return (grad.reshape(ctx.shape) * grad_output, None, None, None)


def _device_mask(lengths, device):
    """mask_from_lengths on `device` without a device -> host round trip:
    lengths that live on the host (what the collate produces) are turned into
    the mask there and uploaded asynchronously (torch.arange(lengths.max()) on
    device lengths synchronises the stream: a bubble in every training step)"""
    from . import model as model_module
    if lengths.device.type == 'cuda':
        return model_module.mask_from_lengths(lengths)
    mask = model_module.mask_from_lengths(lengths)
    if torch.cuda.is_available():
        mask = mask.pin_memory()
    return mask.to(device, non_blocking=True)


def loss(
    scores, targets, frame_lengths, word_bounds, word_lengths, training=False,
    loss_fn=None
):
    """Masked loss, mirroring emphases.loss (emphases/train/core.py:315-353)
    for the word-resolution branch"""
    from . import model as model_module
    if loss_fn is None:
        loss_fn = emphases.LOSS
    if loss_fn not in ('bce', 'mse'):
        raise ValueError(f'Loss {loss_fn} is not recognized')
    if training and emphases.DOWNSAMPLE_LOCATION == 'inference':
        # scores are frame resolution: upsample the word targets
        # (train/core.py:324-338)
        targets = emphases.upsample(
            targets.to(scores.device), word_bounds, word_lengths, frame_lengths)
        if emphases.UPSAMPLE_METHOD == 'linear':
            targets = torch.clamp(targets, min=0., max=1.)
        mask = _device_mask(frame_lengths, scores.device)
    else:
        mask = _device_mask(word_lengths, scores.device)
    return _MaskedLoss.apply(scores, targets, mask, 0 if loss_fn == 'bce' else 1)


###############################################################################
# Data parallelism
###############################################################################


def allreduce_gradients(model, average=True):
    """One all-reduce over a flat fp32 bucket holding every gradient
    (250,881 floats ~ 1 MB for the default model: latency bound, so a single
    NCCL call beats per-tensor calls).  No-op without a process group."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return
    world = dist.get_world_size()
    if world == 1:
        return
    state = getattr(model, '_native_train_state', None)
    if state is not None and all(
        state.aliases_flat(p, i) for i, p in enumerate(state.ordered)
    ) and len(state.ordered) == sum(1 for _ in model.parameters()):
        # the native step wrote every gradient into one flat buffer that the
        # .grad tensors alias: reduce it in place, no packing or copy-back
        if average and dist.get_backend() == 'nccl':
            dist.all_reduce(state.flat, op=dist.ReduceOp.AVG)     # no separate scaling launch
            return
        dist.all_reduce(state.flat, op=dist.ReduceOp.SUM)
        if average:
            state.flat.div_(world)
        return
    parameters = [p for p in model.parameters() if p.grad is not None]
    flat = torch.cat([p.grad.reshape(-1).to(torch.float32) for p in parameters])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    if average:
        flat.div_(world)
    cursor = 0
    for p in parameters:
        count = p.grad.numel()
        p.grad.copy_(flat[cursor:cursor + count].reshape(p.grad.shape))
        cursor += count


def train_step(model, optimizer, batch):
    """One data-parallel step: forward, masked loss, backward, gradient
    all-reduce (mean over ranks), optimizer step.  `batch` follows the
    reference collate order (emphases/data/collate.py:72-78):
    (features, frame_lengths, word_bounds, word_lengths, targets)."""
    features, frame_lengths, word_bounds, word_lengths, targets = batch[:5]
    model.train()
    optimizer.zero_grad(set_to_none=True)
    scores = model(features, frame_lengths, word_bounds, word_lengths)
    value = loss(
        scores, targets, frame_lengths, word_bounds, word_lengths, training=True)
    value.backward()
    allreduce_gradients(model)
    optimizer.step()
    return value.detach()
