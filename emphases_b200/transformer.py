"""Transformer variant (`ARCHITECTURE = 'transformer'`), mirroring
emphases/model/layers/transformer.py:13-52 on packed rows.

The modules below are parameter containers with the reference's state_dict
keys (`position.encoding`, `model.layers.{i}.self_attn.in_proj_weight`, ...,
SURVEY.md A.7); the math runs in libemphases_b200.so: per-row linear maps
through the fused fp32 conv stack with kernel size 1 (the feed-forward block
is ONE fused two-layer launch), attention / LayerNorm / positional add through
csrc/attention.cu.
"""
import dataclasses
import math
from typing import List

import numpy as np
import torch

import emphases_b200 as emphases
from . import _lib, engine

HEADS = 2                      # transformer.py:20
MAX_LENGTH = 5000              # transformer.py:38


class PositionalEncoding(torch.nn.Module):
    """transformer.py:36-52 (buffer only; dropout is identity in eval)"""

    def __init__(self, channels, dropout=.1, max_len=MAX_LENGTH):
        super().__init__()
        self.dropout = torch.nn.Dropout(p=dropout)
        index = torch.arange(max_len).unsqueeze(1)
        frequency = torch.exp(
            torch.arange(0, channels, 2) * (-math.log(10000.0) / channels))
        encoding = torch.zeros(max_len, 1, channels)
        encoding[:, 0, 0::2] = torch.sin(index * frequency)
        encoding[:, 0, 1::2] = torch.cos(index * frequency)
        self.register_buffer('encoding', encoding)


class Transformer(torch.nn.Module):
    """transformer.py:13-30"""

    def __init__(self):
        super().__init__()
        channels = emphases.CHANNELS
        self.position = PositionalEncoding(channels, .1)
        self.model = torch.nn.TransformerEncoder(
            torch.nn.TransformerEncoderLayer(
                channels, HEADS, dim_feedforward=emphases.CHANNELS),
            emphases.LAYERS,
            enable_nested_tensor=False)

    def forward(self, x, lengths):
        raise _lib.EmphasesB200Error(
            'submodules are parameter containers; call Model.forward')


###############################################################################
# Packed weights
###############################################################################


@dataclasses.dataclass
class FusedLayer:
    """Operands of csrc/transformer_tc.cu: bf16 weight parts
    [matrix][part][out][in + 8] and fp32 biases"""
    qkv_weight: torch.Tensor
    qkv_bias: torch.Tensor
    out_weight: torch.Tensor
    out_bias: torch.Tensor
    ffn_weight: torch.Tensor
    ffn_bias: torch.Tensor
    tail_weight: torch.Tensor        # out-projection, linear1, linear2 in one blob
    tail_bias: torch.Tensor


def split_parts(matrices, parts, device):
    """[(out, in) fp32] -> bf16 (matrices, parts, out, in + 8): part p is the
    bf16 rounding of what parts < p left over (round to nearest even, like
    cvt.rn.bf16x2.f32 on the activation side)"""
    dtype = torch.float16 if parts == 1 else torch.bfloat16      # one fp16 value, or bf16 parts
    blob = torch.zeros(
        (len(matrices), parts) + (matrices[0].shape[0], matrices[0].shape[1] + 8),
        dtype=dtype, device=device)
    for index, matrix in enumerate(matrices):
        rest = matrix.detach().to(device, torch.float32).clone()
        for part in range(parts):
            rounded = rest.to(dtype)
            blob[index, part, :, :matrix.shape[1]] = rounded
            rest -= rounded.float()
    return blob.contiguous()


@dataclasses.dataclass
class EncoderLayer:
    qkv: List[engine.ConvStack]          # three 1-layer, kernel-1 stacks
    out_proj: engine.ConvStack
    feedforward: engine.ConvStack        # linear1 + ReLU + linear2, fused
    norm1: tuple
    norm2: tuple
    raw: dict = None                     # the module's fp32 tensors (fused path)
    packs: dict = dataclasses.field(default_factory=dict)

    def fused(self, parts, device) -> FusedLayer:
        if parts not in self.packs:
            raw, channels = self.raw, self.norm1[0].shape[0]
            in_proj = raw['in_proj_weight']

            def vector(*names):
                return torch.cat([
                    raw[name].detach().to(device, torch.float32).reshape(-1)
                    for name in names]).contiguous()
            self.packs[parts] = FusedLayer(
                split_parts(
                    [in_proj[i * channels:(i + 1) * channels] for i in range(3)],
                    parts, device),
                vector('in_proj_bias'),
                split_parts([raw['out_proj.weight']], parts, device),
                vector('out_proj.bias'),
                split_parts([raw['linear1.weight'], raw['linear2.weight']], parts, device),
                vector('linear1.bias', 'linear2.bias'),
                split_parts(
                    [raw['out_proj.weight'], raw['linear1.weight'], raw['linear2.weight']],
                    parts, device),
                vector('out_proj.bias', 'linear1.bias', 'linear2.bias'))
        return self.packs[parts]


@dataclasses.dataclass
class TransformerStack:
    table: torch.Tensor                  # (max_len, channels) positional table
    layers: List[EncoderLayer]
    channels: int


def _linear_stack(pairs, acts, device):
    """[(weight (out, in), bias)] -> ConvStack with kernel size 1"""
    weights = torch.stack([
        engine._pack_conv(weight[:, :, None], device) for weight, _ in pairs])
    bias = torch.stack([
        b.detach().to(device=device, dtype=torch.float32) for _, b in pairs])
    return engine.ConvStack(
        weights.contiguous(), bias.contiguous(),
        np.asarray(acts, dtype=np.int32), 1, pairs[0][0].shape[0])


def pack_stack(state, prefix, layers, channels, device):
    encoder_layers = []
    for index in range(layers):
        p = f'{prefix}.model.layers.{index}'
        w = state[f'{p}.self_attn.in_proj_weight']
        b = state[f'{p}.self_attn.in_proj_bias']
        qkv = [
            _linear_stack(
                [(w[i * channels:(i + 1) * channels],
                  b[i * channels:(i + 1) * channels])],
                [_lib.ACT_NONE], device)
            for i in range(3)]
        out_proj = _linear_stack(
            [(state[f'{p}.self_attn.out_proj.weight'],
              state[f'{p}.self_attn.out_proj.bias'])], [_lib.ACT_NONE], device)
        if state[f'{p}.linear1.weight'].shape != (channels, channels):
            raise NotImplementedError('dim_feedforward must equal CHANNELS')
        feedforward = _linear_stack(
            [(state[f'{p}.linear1.weight'], state[f'{p}.linear1.bias']),
             (state[f'{p}.linear2.weight'], state[f'{p}.linear2.bias'])],
            [_lib.ACT_RELU, _lib.ACT_NONE], device)

        def norm(name):
            return (
                state[f'{p}.{name}.weight'].detach().to(device, torch.float32).contiguous(),
                state[f'{p}.{name}.bias'].detach().to(device, torch.float32).contiguous())
        raw = {
            'in_proj_weight': w, 'in_proj_bias': b,
            'out_proj.weight': state[f'{p}.self_attn.out_proj.weight'],
            'out_proj.bias': state[f'{p}.self_attn.out_proj.bias'],
            'linear1.weight': state[f'{p}.linear1.weight'],
            'linear1.bias': state[f'{p}.linear1.bias'],
            'linear2.weight': state[f'{p}.linear2.weight'],
            'linear2.bias': state[f'{p}.linear2.bias']}
        encoder_layers.append(EncoderLayer(
            qkv, out_proj, feedforward, norm('norm1'), norm('norm2'), raw))
    table = state[f'{prefix}.position.encoding'].detach().to(
        device, torch.float32)[:, 0, :].contiguous()
    return TransformerStack(table, encoder_layers, channels)


@dataclasses.dataclass
class TransformerWeights:
    input_layer: engine.ConvStack
    frame: TransformerStack
    word: TransformerStack
    head_weight: torch.Tensor
    head_bias: float
    head_kernel: int
    channels: int


def pack_weights(model, device):
    state = model.state_dict()
    channels = state['input_layer.weight'].shape[0]
    if state['input_layer.weight'].shape[1] != channels:
        raise NotImplementedError('input layer needs equal in/out channels')
    kernel = state['input_layer.weight'].shape[2]
    input_layer = engine.ConvStack(
        engine._pack_conv(state['input_layer.weight'], device)[None].contiguous(),
        state['input_layer.bias'].detach().to(device, torch.float32)[None].contiguous(),
        np.asarray([_lib.ACT_NONE], dtype=np.int32), kernel, channels)
    head = state['output_layer.weight'].detach().to(device, torch.float32)
    return TransformerWeights(
        input_layer=input_layer,
        frame=pack_stack(state, 'frame_encoder', model.layers, channels, device),
        word=pack_stack(state, 'word_decoder', model.layers, channels, device)
        if hasattr(model, 'word_decoder') else None,
        head_weight=head[0].t().contiguous(),
        head_bias=float(state['output_layer.bias'].detach().float().cpu()[0]),
        head_kernel=head.shape[2],
        channels=channels)


###############################################################################
# Execution on packed rows
###############################################################################


ATTENTION_MODES = {'fp16': 0, 'bf16x3': 1}     # operand modes of csrc/attention_tc.cu


def attention_mode():
    """How attention runs for the configured PRECISION: None = the fp32
    CUDA-core kernel (emph_attention_rows), else the operand mode of the
    tensor-core kernel (emph_attention_rows_tc): fp16 operands in the 2e-3
    'bf16' mode (3e-4 on the scores of bench.py's corpus), split bf16 in the
    fp32-grade modes (3e-6).  EMPHASES_B200_ATTENTION = fp32 | fp16 | bf16x3
    overrides."""
    import os
    choice = os.environ.get('EMPHASES_B200_ATTENTION') or {
        'fp32': 'fp32', 'bf16': 'fp16', 'bf16x3': 'bf16x3', 'bf16x6': 'bf16x3',
    }[emphases.PRECISION]
    if choice != 'fp32' and choice not in ATTENTION_MODES:
        raise ValueError(f'EMPHASES_B200_ATTENTION={choice} is not defined')
    return ATTENTION_MODES.get(choice)


def attention_workspace(total_rows, channels, mode, device, zero=False, ws=None, tag=''):
    """Device buffer for the 16-bit K / V records of one attention call: heads x
    (total_rows + 64) records, head-major.  `zero`: the 64 records of slack
    behind each head's rows are cleared (the fused q / k / v pass writes the
    records of the rows only; emph_attention_rows_tc's staging pass writes all)"""
    size = _lib.load().emph_attention_tc_workspace(total_rows, channels, HEADS, mode)
    if size < 0:
        raise NotImplementedError(
            f'tensor-core attention is not compiled for {channels // HEADS}-dim heads')
    records = engine._empty(ws, f'{tag}records', (max(size, 1),), torch.uint8, device)
    if zero and size:
        per_head = size // HEADS
        record = per_head // (total_rows + 64)
        for head in range(HEADS):
            records[head * per_head + total_rows * record:(head + 1) * per_head].zero_()
    return records


FUSED_CHANNELS = 80                # csrc/transformer_tc.cu is compiled for d_model 80
# out-projection + LayerNorm + feed-forward + LayerNorm as ONE pass
# (emph_transformer_layer_tail) instead of two
import os as _os
FUSED_TAIL = _os.environ.get('EMPHASES_B200_FUSED_TAIL', '1') != '0'


def fused_layers(channels, mode):
    """The fused per-row passes (emph_transformer_qkv / _proj_norm / _ffn_norm)
    serve the default width whenever attention runs on the tensor cores;
    EMPHASES_B200_FUSED_LAYERS=0 keeps the per-op launches"""
    import os
    return (
        mode is not None and channels == FUSED_CHANNELS
        and os.environ.get('EMPHASES_B200_FUSED_LAYERS', '1') != '0')


def fused_parts():
    """Operand parts of the fused per-row passes: 3 bf16 parts in 'bf16x6', 2 in
    'bf16x3' and 'bf16'.  EMPHASES_B200_LINEAR_PARTS=1 selects one fp16 value
    per operand: on bench.py's corpus 48.3 instead of 52.7 ms per pass in the
    'bf16' mode at 1.1e-3 instead of 3.0e-4 on the scores -- inside the 2e-3
    bar, but with half the margin, so it is not the default"""
    import os
    override = os.environ.get('EMPHASES_B200_LINEAR_PARTS')
    if override:
        return int(override)
    return 3 if emphases.PRECISION == 'bf16x6' else 2


def run_fused_layers(
    stack, h, mode, row_start, n_queries, n_keys, row_seq, d_block_seq, d_block_q0,
    n_blocks, scale, device, ws=None, tag='frame_'
):
    """Every encoder layer as qkv -> attention -> out_proj + LayerNorm ->
    feed-forward + LayerNorm: four launches, five row buffers for the stack.
    With a launch workspace `ws` all buffers are grow-only views of it (fresh
    gigabyte allocations per call make the caching allocator fall back to
    cudaMalloc / cudaFree: 30-40 ms stalls)"""
    total_rows, channels = h.shape
    parts = fused_parts()
    records = attention_workspace(
        total_rows, channels, mode, device, zero=True, ws=ws, tag=tag)
    q, context, normed, spare = (
        engine._empty(ws, f'{tag}{name}', tuple(h.shape), torch.float32, device)
        for name in ('q', 'context', 'normed', 'spare'))
    stream = _lib.stream_ptr()
    for layer in stack.layers:
        pack = layer.fused(parts, device)
        _lib.call(
            'emph_transformer_qkv', _lib.ptr(h), total_rows, channels,
            _lib.ptr(pack.qkv_weight), _lib.ptr(pack.qkv_bias), parts, mode, _lib.ptr(q),
            _lib.ptr(records), records.numel(), stream)
        _lib.call(
            'emph_attention_rows_staged', _lib.ptr(q), _lib.ptr(records), records.numel(),
            channels, HEADS, _lib.ptr(row_start), _lib.ptr(n_queries), _lib.ptr(n_keys),
            total_rows, _lib.ptr(d_block_seq), _lib.ptr(d_block_q0), n_blocks, scale, mode,
            _lib.ptr(context), stream)
        if FUSED_TAIL and parts <= 2:
            # (with three parts the pass is bound by its 18 products per
            # element, not by the row traffic it saves: no gain measured)
            _lib.call(
                'emph_transformer_layer_tail', _lib.ptr(context), _lib.ptr(h), total_rows,
                channels, _lib.ptr(pack.tail_weight), _lib.ptr(pack.tail_bias), parts,
                _lib.ptr(layer.norm1[0]), _lib.ptr(layer.norm1[1]),
                _lib.ptr(layer.norm2[0]), _lib.ptr(layer.norm2[1]), 1e-5, _lib.ptr(row_seq),
                _lib.ptr(spare), stream)
            h, spare = spare, h
            continue
        _lib.call(
            'emph_transformer_proj_norm', _lib.ptr(context), _lib.ptr(h), total_rows, channels,
            _lib.ptr(pack.out_weight), _lib.ptr(pack.out_bias), parts,
            _lib.ptr(layer.norm1[0]), _lib.ptr(layer.norm1[1]), 1e-5, _lib.ptr(row_seq),
            _lib.ptr(normed), stream)
        _lib.call(
            'emph_transformer_ffn_norm', _lib.ptr(normed), total_rows, channels,
            _lib.ptr(pack.ffn_weight), _lib.ptr(pack.ffn_bias), parts,
            _lib.ptr(layer.norm2[0]), _lib.ptr(layer.norm2[1]), 1e-5, _lib.ptr(row_seq),
            _lib.ptr(spare), stream)
        h, spare = spare, h
    return h


def query_blocks(n_keys, block=128):
    """(block_seq, block_q0): 128-query blocks (kAttnQ of csrc/attention.cu)
    that never cross a sequence"""
    n_keys = np.asarray(n_keys, dtype=np.int64)
    counts = (n_keys + block - 1) // block
    sequence = np.repeat(np.arange(len(n_keys)), counts)
    first = np.concatenate([[0], np.cumsum(counts[:-1])]) if len(counts) else counts
    within = np.arange(int(counts.sum())) - np.repeat(first, counts)
    return sequence.astype(np.int32), (within * block).astype(np.int32)


def run_stack(
    eng, stack, x, row_start, n_rows_host, n_keys_host, row_seq, device, ws=None,
    tag='frame_'
):
    """x: packed rows (total_rows, C); sequence u has n_rows[u] rows (all are
    queries) of which the first n_keys[u] are valid keys.  `ws`: the launch's
    grow-only engine workspace (buffers named with `tag`; the result then lives
    there until the next stack with the same tag runs on it)"""
    if int(np.max(n_rows_host, initial=0)) > stack.table.shape[0]:
        raise RuntimeError(
            f'The size of tensor a ({int(np.max(n_rows_host))}) must match the '
            f'size of tensor b ({stack.table.shape[0]}) at non-singleton '
            'dimension 0 (positional encoding table, transformer.py:52)')
    total_rows, channels = x.shape
    block_seq, block_q0 = query_blocks(n_rows_host)
    meta = torch.from_numpy(np.concatenate([
        np.asarray(n_rows_host, dtype=np.int32),
        np.asarray(n_keys_host, dtype=np.int32), block_seq, block_q0])).to(device)
    n_seq = len(n_keys_host)
    n_queries, n_keys = meta[:n_seq], meta[n_seq:2 * n_seq]
    d_block_seq = meta[2 * n_seq:2 * n_seq + len(block_seq)]
    d_block_q0 = meta[2 * n_seq + len(block_seq):]
    scale = 1.0 / math.sqrt(channels // HEADS)
    mode = attention_mode()
    fused = fused_layers(channels, mode)
    workspace = None if mode is None or fused else attention_workspace(
        total_rows, channels, mode, device)

    h = engine._empty(ws, f'{tag}positional', tuple(x.shape), torch.float32, device)
    _lib.call(
        'emph_add_positional', _lib.ptr(x), _lib.ptr(row_start),
        _lib.ptr(row_seq), total_rows, channels, _lib.ptr(stack.table),
        stack.table.shape[0], _lib.ptr(h), _lib.stream_ptr())
    if fused:
        return run_fused_layers(
            stack, h, mode, row_start, n_queries, n_keys, row_seq, d_block_seq,
            d_block_q0, len(block_seq), scale, device, ws, tag)
    for layer in stack.layers:
        q, k, v = (
            eng.conv_stack(h, row_seq, part, engine.linear_precision(part))
            for part in layer.qkv)
        context = torch.empty_like(h)
        if mode is None:
            _lib.call(
                'emph_attention_rows', _lib.ptr(q), _lib.ptr(k), _lib.ptr(v),
                channels, HEADS, _lib.ptr(row_start), _lib.ptr(n_queries),
                _lib.ptr(n_keys), _lib.ptr(row_seq), total_rows, _lib.ptr(d_block_seq),
                _lib.ptr(d_block_q0), len(block_seq), scale, _lib.ptr(context),
                _lib.stream_ptr())
        else:
            _lib.call(
                'emph_attention_rows_tc', _lib.ptr(q), _lib.ptr(k), _lib.ptr(v),
                channels, HEADS, _lib.ptr(row_start), _lib.ptr(n_queries),
                _lib.ptr(n_keys), _lib.ptr(row_seq), total_rows, _lib.ptr(d_block_seq),
                _lib.ptr(d_block_q0), len(block_seq), scale, mode, _lib.ptr(workspace),
                workspace.numel(), _lib.ptr(context), _lib.stream_ptr())
        attended = eng.conv_stack(
            context, row_seq, layer.out_proj, engine.linear_precision(layer.out_proj))
        normed = torch.empty_like(h)
        _lib.call(
            'emph_add_layernorm', _lib.ptr(h), _lib.ptr(attended),
            _lib.ptr(layer.norm1[0]), _lib.ptr(layer.norm1[1]), 1e-5,
            _lib.ptr(row_seq), total_rows, channels, _lib.ptr(normed),
            _lib.stream_ptr())
        forward = eng.conv_stack(
            normed, row_seq, layer.feedforward,
            engine.linear_precision(layer.feedforward))
        h = torch.empty_like(normed)
        _lib.call(
            'emph_add_layernorm', _lib.ptr(normed), _lib.ptr(forward),
            _lib.ptr(layer.norm2[0]), _lib.ptr(layer.norm2[1]), 1e-5,
            _lib.ptr(row_seq), total_rows, channels, _lib.ptr(h),
            _lib.stream_ptr())
    return h


def encoders(eng, weights):
    """(encode, decode) of the Transformer architecture for model.run_forward:
    input_layer and the frame stack, and the word stack.  A sequence of
    n_queries[u] rows attends over its first n_keys[u] rows."""

    def encode(rows, row_seq, row_start, n_queries, n_keys):
        # input_layer is a Conv1d over ALL T columns, padding included
        embedded = eng.conv_stack(
            rows, row_seq, weights.input_layer,
            engine.linear_precision(weights.input_layer))
        if torch.is_tensor(n_keys):          # frame_lengths, maybe on the device
            n_keys = n_keys.detach().to('cpu', torch.int64).numpy()
        return run_stack(
            eng, weights.frame, embedded, row_start, n_queries, n_keys, row_seq,
            eng.device)

    def decode(pooled, word_row_seq, word_start, n_queries, n_keys):
        return run_stack(
            eng, weights.word, pooled, word_start, n_queries, n_keys,
            word_row_seq, eng.device, tag='word_')

    return encode, decode


###############################################################################
# Training: forward with saved activations, and its backward
###############################################################################

TRAIN_CHANNELS = 80              # the training kernels are built for 40-dim heads
KEY_BLOCK = 64                   # kBwdRows of csrc/attention.cu


def _f32(tensor):
    return tensor.detach().to(torch.float32).contiguous()


def dropout_rates(module):
    """p of the five dropout sites of one TransformerEncoderLayer container,
    read from its modules (a model set to p = 0 trains without dropout)"""
    return [
        [layer.self_attn.dropout, layer.dropout1.p, layer.dropout.p, layer.dropout2.p]
        for layer in module.model.layers]


def stack_forward_train(
    module, table, x, row_start, n_queries, n_keys, row_seq, seed, stack
):
    """Training forward of one Transformer container (`frame_encoder` or
    `word_decoder`, stack 0 / 1 of the dropout sites) on packed rows x: the
    positional encoding, then per layer post-norm self-attention and
    feed-forward with the reference's five dropout sites.  Sequence u has
    n_queries[u] rows (host), of which the first n_keys[u] are keys.
    Returns (rows, saved): saved keeps per layer only what stack_backward
    reads (layer input, q / k / v, attention output and log-sum-exp, the
    LayerNorm sums and statistics, the feed-forward activation); the dropout
    masks are regenerated from `seed`."""
    total_rows, channels = x.shape
    if channels != TRAIN_CHANNELS:
        raise NotImplementedError(
            f'the Transformer training kernels are built for {TRAIN_CHANNELS} channels')
    if int(np.max(n_queries, initial=0)) > table.shape[0]:
        raise RuntimeError(
            f'The size of tensor a ({int(np.max(n_queries))}) must match the '
            f'size of tensor b ({table.shape[0]}) at non-singleton '
            'dimension 0 (positional encoding table, transformer.py:52)')
    device = x.device
    n_seq = len(n_queries)
    blocks = [query_blocks(n_queries), query_blocks(n_keys, KEY_BLOCK),
              query_blocks(n_queries, KEY_BLOCK)]
    parts = [np.asarray(n_queries, dtype=np.int32), np.asarray(n_keys, dtype=np.int32)]
    for sequence, first in blocks:
        parts += [sequence, first]
    meta = torch.from_numpy(np.concatenate(parts)).to(device)
    cursor, views = 0, []
    for part in parts:
        views.append(meta[cursor:cursor + len(part)])
        cursor += len(part)
    geometry = dict(
        row_start=row_start, row_seq=row_seq, n_queries=views[0], n_keys=views[1],
        forward_blocks=(views[2], views[3], len(blocks[0][0])),
        key_blocks=(views[4], views[5], len(blocks[1][0])),
        query_blocks=(views[6], views[7], len(blocks[2][0])),
        scale=1.0 / math.sqrt(channels // HEADS), seq=n_seq)
    rates = dropout_rates(module)
    p_position = float(module.position.dropout.p)
    stream = _lib.stream_ptr()

    def site(layer, kind):
        return _lib.dropout_site(stack, layer, kind)

    def empty(*shape):
        return torch.empty(shape, dtype=torch.float32, device=device)

    h = empty(total_rows, channels)
    _lib.call(
        'emph_add_positional', _lib.ptr(x), _lib.ptr(row_start), _lib.ptr(row_seq),
        total_rows, channels, _lib.ptr(table), table.shape[0], _lib.ptr(h), stream)
    _lib.call(
        'emph_dropout_rows', _lib.ptr(h), total_rows, channels, seed,
        site(0, _lib.DROPOUT_POSITIONAL), p_position, _lib.ptr(h), stream)
    saved = []
    for index, layer in enumerate(module.model.layers):
        p_attention, p_1, p_feedforward, p_2 = rates[index]
        qkv = empty(3, total_rows, channels)
        _lib.call(
            'emph_linear_rows', _lib.ptr(h), total_rows, channels,
            _lib.ptr(_f32(layer.self_attn.in_proj_weight)),
            _lib.ptr(_f32(layer.self_attn.in_proj_bias)), 3, _lib.ACT_NONE,
            _lib.ptr(row_seq), _lib.ptr(qkv), stream)
        context = empty(total_rows, channels)
        lse = empty(total_rows, HEADS)
        block_seq, block_q0, n_blocks = geometry['forward_blocks']
        _lib.call(
            'emph_attention_rows_train', _lib.ptr(qkv[0]), _lib.ptr(qkv[1]),
            _lib.ptr(qkv[2]), channels, HEADS, _lib.ptr(row_start),
            _lib.ptr(geometry['n_queries']), _lib.ptr(geometry['n_keys']),
            _lib.ptr(row_seq), total_rows, _lib.ptr(block_seq), _lib.ptr(block_q0),
            n_blocks, geometry['scale'], seed, site(index, _lib.DROPOUT_ATTENTION),
            p_attention, _lib.ptr(context), _lib.ptr(lse), stream)
        attended = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows', _lib.ptr(context), total_rows, channels,
            _lib.ptr(_f32(layer.self_attn.out_proj.weight)),
            _lib.ptr(_f32(layer.self_attn.out_proj.bias)), 1, _lib.ACT_NONE,
            _lib.ptr(row_seq), _lib.ptr(attended), stream)
        normed, sums1, stats1 = empty(total_rows, channels), empty(total_rows, channels), \
            empty(total_rows, 2)
        _lib.call(
            'emph_add_layernorm_train', _lib.ptr(h), _lib.ptr(attended),
            _lib.ptr(_f32(layer.norm1.weight)), _lib.ptr(_f32(layer.norm1.bias)),
            layer.norm1.eps, _lib.ptr(row_seq), total_rows, channels, seed,
            site(index, _lib.DROPOUT_RESIDUAL1), p_1, _lib.ptr(normed), _lib.ptr(sums1),
            _lib.ptr(stats1), stream)
        hidden = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows', _lib.ptr(normed), total_rows, channels,
            _lib.ptr(_f32(layer.linear1.weight)), _lib.ptr(_f32(layer.linear1.bias)), 1,
            _lib.ACT_RELU, _lib.ptr(row_seq), _lib.ptr(hidden), stream)
        dropped = empty(total_rows, channels)
        _lib.call(
            'emph_dropout_rows', _lib.ptr(hidden), total_rows, channels, seed,
            site(index, _lib.DROPOUT_FEEDFORWARD), p_feedforward, _lib.ptr(dropped), stream)
        forward = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows', _lib.ptr(dropped), total_rows, channels,
            _lib.ptr(_f32(layer.linear2.weight)), _lib.ptr(_f32(layer.linear2.bias)), 1,
            _lib.ACT_NONE, _lib.ptr(row_seq), _lib.ptr(forward), stream)
        out, sums2, stats2 = empty(total_rows, channels), empty(total_rows, channels), \
            empty(total_rows, 2)
        _lib.call(
            'emph_add_layernorm_train', _lib.ptr(normed), _lib.ptr(forward),
            _lib.ptr(_f32(layer.norm2.weight)), _lib.ptr(_f32(layer.norm2.bias)),
            layer.norm2.eps, _lib.ptr(row_seq), total_rows, channels, seed,
            site(index, _lib.DROPOUT_RESIDUAL2), p_2, _lib.ptr(out), _lib.ptr(sums2),
            _lib.ptr(stats2), stream)
        saved.append(dict(
            x=h, qkv=qkv, context=context, lse=lse, normed=normed, sums1=sums1,
            stats1=stats1, hidden=hidden, sums2=sums2, stats2=stats2))
        h = out
    return h, dict(
        module=module, layers=saved, geometry=geometry, seed=seed, stack=stack,
        rates=rates, p_position=p_position)


def stack_backward(saved, d_rows):
    """Adjoint of stack_forward_train: (gradient of its input rows, {parameter:
    gradient}) from the gradient of its output rows"""
    module, g = saved['module'], saved['geometry']
    seed, stack = saved['seed'], saved['stack']
    total_rows, channels = d_rows.shape
    device = d_rows.device
    row_seq = g['row_seq']
    stream = _lib.stream_ptr()
    grads = {}

    def site(layer, kind):
        return _lib.dropout_site(stack, layer, kind)

    def empty(*shape):
        return torch.empty(shape, dtype=torch.float32, device=device)

    partials = empty(_lib.load().emph_layernorm_backward_blocks(total_rows), 2 * channels)

    def weight_grad(x, dy, dw, db):
        """dw [in][out] (the Linear gradient transposed), db [out]"""
        _lib.call(
            'emph_conv_weight_grad', _lib.ptr(x), _lib.ptr(dy), total_rows, channels, 1,
            _lib.ptr(dw), _lib.ptr(db), stream)

    def norm_backward(dy, sums, stats, norm, kind, p, index):
        dx, d_branch = empty(total_rows, channels), empty(total_rows, channels)
        dgamma, dbeta = empty(channels), empty(channels)
        _lib.call(
            'emph_add_layernorm_backward', _lib.ptr(dy), _lib.ptr(sums), _lib.ptr(stats),
            _lib.ptr(_f32(norm.weight)), _lib.ptr(row_seq), total_rows, channels, seed,
            site(index, kind), p, _lib.ptr(dx), _lib.ptr(d_branch), _lib.ptr(dgamma),
            _lib.ptr(dbeta), _lib.ptr(partials), stream)
        grads[norm.weight], grads[norm.bias] = dgamma, dbeta
        return dx, d_branch

    def linear_backward(x, dy, linear):
        """weight / bias gradient of one Linear, and dy W"""
        dw, db = empty(channels, channels), empty(channels)
        weight_grad(x, dy, dw, db)
        grads[linear.weight], grads[linear.bias] = dw.t().contiguous(), db
        dx = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows_backward', _lib.ptr(dy), total_rows, channels,
            _lib.ptr(_f32(linear.weight)), 1, None, _lib.ptr(row_seq), _lib.ptr(dx), stream)
        return dx

    d = d_rows.contiguous()
    for index in range(len(saved['layers']) - 1, -1, -1):
        layer, s = module.model.layers[index], saved['layers'][index]
        p_attention, p_1, p_feedforward, p_2 = saved['rates'][index]
        # h2 = LayerNorm2(h1 + dropout2(linear2(dropout(relu(linear1(h1))))))
        d_normed, d_forward = norm_backward(
            d, s['sums2'], s['stats2'], layer.norm2, _lib.DROPOUT_RESIDUAL2, p_2, index)
        dropped = empty(total_rows, channels)
        _lib.call(
            'emph_dropout_rows', _lib.ptr(s['hidden']), total_rows, channels, seed,
            site(index, _lib.DROPOUT_FEEDFORWARD), p_feedforward, _lib.ptr(dropped), stream)
        d_dropped = linear_backward(dropped, d_forward, layer.linear2)
        _lib.call(
            'emph_dropout_rows', _lib.ptr(d_dropped), total_rows, channels, seed,
            site(index, _lib.DROPOUT_FEEDFORWARD), p_feedforward, _lib.ptr(d_dropped), stream)
        d_pre = empty(total_rows, channels)
        _lib.call(
            'emph_activation_backward', _lib.ptr(d_dropped), _lib.ptr(s['hidden']),
            _lib.ptr(row_seq), total_rows, channels, _lib.ACT_RELU, _lib.ptr(d_pre), stream)
        dw, db = empty(channels, channels), empty(channels)
        weight_grad(s['normed'], d_pre, dw, db)
        grads[layer.linear1.weight], grads[layer.linear1.bias] = dw.t().contiguous(), db
        d_h1 = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows_backward', _lib.ptr(d_pre), total_rows, channels,
            _lib.ptr(_f32(layer.linear1.weight)), 1, _lib.ptr(d_normed), _lib.ptr(row_seq),
            _lib.ptr(d_h1), stream)
        # h1 = LayerNorm1(h + dropout1(out_proj(attention(h))))
        d_h, d_attended = norm_backward(
            d_h1, s['sums1'], s['stats1'], layer.norm1, _lib.DROPOUT_RESIDUAL1, p_1, index)
        d_context = linear_backward(s['context'], d_attended, layer.self_attn.out_proj)
        qkv, d_qkv = s['qkv'], empty(3, total_rows, channels)
        key_seq, key_k0, n_key_blocks = g['key_blocks']
        query_seq, query_q0, n_query_blocks = g['query_blocks']
        _lib.call(
            'emph_attention_rows_backward', _lib.ptr(qkv[0]), _lib.ptr(qkv[1]),
            _lib.ptr(qkv[2]), _lib.ptr(s['context']), _lib.ptr(d_context), _lib.ptr(s['lse']),
            channels, HEADS, _lib.ptr(g['row_start']), _lib.ptr(g['n_queries']),
            _lib.ptr(g['n_keys']), total_rows, _lib.ptr(key_seq), _lib.ptr(key_k0),
            n_key_blocks, _lib.ptr(query_seq), _lib.ptr(query_q0), n_query_blocks,
            g['scale'], seed, site(index, _lib.DROPOUT_ATTENTION), p_attention,
            _lib.ptr(d_qkv[0]), _lib.ptr(d_qkv[1]), _lib.ptr(d_qkv[2]), stream)
        dw, db = empty(3, channels, channels), empty(3 * channels)
        for part in range(3):
            weight_grad(s['x'], d_qkv[part], dw[part], db[part * channels:])
        grads[layer.self_attn.in_proj_weight] = \
            dw.transpose(1, 2).reshape(3 * channels, channels).contiguous()
        grads[layer.self_attn.in_proj_bias] = db
        d = empty(total_rows, channels)
        _lib.call(
            'emph_linear_rows_backward', _lib.ptr(d_qkv), total_rows, channels,
            _lib.ptr(_f32(layer.self_attn.in_proj_weight)), 3, _lib.ptr(d_h),
            _lib.ptr(row_seq), _lib.ptr(d), stream)
    # x + PE[:T] under dropout: the positional table is a buffer
    _lib.call(
        'emph_dropout_rows', _lib.ptr(d), total_rows, channels, seed,
        site(0, _lib.DROPOUT_POSITIONAL), saved['p_position'], _lib.ptr(d), stream)
    return d, grads
