"""80-channel conv stacks of kernel size 5 and 7 on the tcgen05 kernel in
bf16, bf16x3 and bf16x6: the kernel against fp64 with ragged rows whose
sequence and tile edges fall at every offset of the halo, every layer count up
to the deepest stack that still leaves a tile, every activation; fused word
pooling; the whole model of the reference's sweep against the oracle; path
selection; and the single-utterance native call."""
import numpy as np
import pytest
import torch

from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

MODES = ['bf16', 'bf16x3', 'bf16x6']
KERNELS = [5, 7]
ACTIVATIONS = ['relu', 'gelu', 'leaky_relu', 'silu']


@pytest.fixture(scope='module')
def eng():
    from emphases_b200 import engine
    return engine.Engine('cuda:0')


@pytest.fixture
def emphases():
    import emphases_b200
    emphases_b200.reset_configuration()
    yield emphases_b200
    emphases_b200.reset_configuration()


def _precision(mode):
    from emphases_b200 import _lib
    return {'fp32': _lib.PREC_FP32, 'bf16': _lib.PREC_BF16_TC,
            'bf16x3': _lib.PREC_BF16X3_TC, 'bf16x6': _lib.PREC_BF16X6_TC}[mode]


def _act_code(name):
    from emphases_b200 import _lib
    return {'none': _lib.ACT_NONE, 'relu': _lib.ACT_RELU, 'gelu': _lib.ACT_GELU,
            'leaky_relu': _lib.ACT_LEAKY_RELU, 'silu': _lib.ACT_SILU}[name]


def _deepest(kernel):
    """most layers whose halo leaves 32 rows of a 128-row tile (the kernel
    takes at most 16)"""
    return min(16, (128 - 32) // (kernel - 1))


def _random_stack(kernel, n_layers, activation, seed):
    """input layer (no activation) + n_layers - 1 activated layers, weights
    scaled so that activations stay O(1) through the deepest stack"""
    from emphases_b200 import engine
    generator = torch.Generator().manual_seed(seed)
    gain = 1.0 if activation == 'none' else 1.5
    weights = torch.randn(n_layers, kernel, 80, 80, generator=generator) * (
        gain / np.sqrt(80 * kernel))
    bias = torch.randn(n_layers, 80, generator=generator) * 0.1
    acts = np.asarray(
        [_act_code('none')] + [_act_code(activation)] * (n_layers - 1), dtype=np.int32)
    return engine.ConvStack(weights.cuda(), bias.cuda(), acts, kernel, 80)


def _layer(stack, layer):
    """layer `layer` of a stack as a one-layer stack"""
    from emphases_b200 import engine
    return engine.ConvStack(
        stack.weights[layer:layer + 1].contiguous(), stack.bias[layer:layer + 1].contiguous(),
        stack.acts[layer:layer + 1].copy(), stack.kernel_size, stack.channels)


def _lengths(kernel, n_layers, seed):
    """short sequences, lengths at and around multiples of the tile's useful
    rows, and random ones"""
    tile = 128 - 2 * n_layers * ((kernel - 1) // 2)
    rng = np.random.default_rng(seed)
    lengths = [1, 2, 3, tile - 1, tile, tile + 1, 2 * tile - 1, 2 * tile, 2 * tile + 1, 1, 3]
    lengths += [int(n) for n in rng.integers(1, 400, 12)]
    lengths += [3 * tile + 2, 2, 1]
    return lengths


def _rows(eng, kernel, lengths, seed):
    from emphases_b200 import engine
    starts, total = engine.packed_starts(lengths, gap=(kernel - 1) // 2)
    row_seq = eng.row_index(
        torch.tensor(starts, dtype=torch.int32, device='cuda:0'),
        torch.tensor(lengths, dtype=torch.int32, device='cuda:0'), len(lengths), total)
    generator = torch.Generator().manual_seed(seed)
    x = torch.randn(total, 80, generator=generator)
    x[(row_seq < 0).cpu()] = 0
    return row_seq, x


def _activate(h, code):
    from emphases_b200 import _lib
    if code == _lib.ACT_RELU:
        return torch.relu(h)
    if code == _lib.ACT_GELU:
        return torch.nn.functional.gelu(h)
    if code == _lib.ACT_LEAKY_RELU:
        return torch.nn.functional.leaky_relu(h, 0.01)
    if code == _lib.ACT_SILU:
        return torch.nn.functional.silu(h)
    return h


def _reference(stack, x, row_seq, quantize=False):
    """fp64 stack over the whole packed buffer, separator rows zeroed after
    every layer (= each sequence convolved on its own with zero padding:
    there are (k - 1) / 2 separator rows); `quantize` rounds every operand to
    bf16 like the one-part kernel"""
    keep = (row_seq >= 0).cpu().double()[None, :, None]
    h = x.double()[None]
    for layer in range(stack.n_layers):
        weight = stack.weights[layer].cpu().double()          # [K][in][out]
        bias = stack.bias[layer].cpu().double()
        if quantize:
            h = h.to(torch.bfloat16).double()
            weight = weight.to(torch.bfloat16).double()
        conv = torch.nn.functional.conv1d(
            h.transpose(1, 2), weight.permute(2, 1, 0), bias,
            padding=(stack.kernel_size - 1) // 2)
        h = _activate(conv.transpose(1, 2), int(stack.acts[layer])) * keep
        if quantize:
            h = h.float().double()     # the kernel's epilogue works in fp32
    return h[0]


###############################################################################
# A. The kernel
###############################################################################


@pytest.mark.parametrize('activation', ACTIVATIONS)
@pytest.mark.parametrize('kernel', KERNELS)
@pytest.mark.parametrize('mode', MODES)
def test_conv_stack_tc_kernel_sizes(eng, mode, kernel, activation):
    """emph_conv_stack at k = 5 / 7 against fp64 at 1, 7, 8 and the deepest
    layer count: bf16x6 within the FFMA kernel's 2e-6 bar at one layer (2e-5
    deeper), bf16x3 within 5e-5, bf16 within 3e-2 of fp32 and, layer by
    layer, 2e-3 of a bf16-emulating reference; the stack equal to its
    one-layer launches; separator rows exactly zero; bf16 really differs from
    the FFMA result; two launches bit-identical"""
    precision = _precision(mode)
    for n_layers in (1, 7, 8, _deepest(kernel)):
        seed = 1000 * kernel + n_layers
        stack = _random_stack(kernel, n_layers, activation, seed)
        row_seq, x = _rows(eng, kernel, _lengths(kernel, n_layers, seed), seed)
        y = eng.conv_stack(x.cuda(), row_seq, stack, precision).cpu()
        expected = _reference(stack, x, row_seq)
        scale = max(expected.abs().max().item(), 1.0)
        error = (y.double() - expected).abs().max().item()
        bar = {'bf16': 3e-2, 'bf16x3': 5e-5, 'bf16x6': 2e-6}[mode]
        if mode == 'bf16x6' and n_layers > 1:
            # the tensor core truncates every MMA's sum into its class
            # accumulator, k * 5 times per class and layer: through 7 to 16
            # layers of kernel size 5 / 7 that gathers 3e-6 .. 5.2e-6 of the
            # scale (measured on a B200), where one layer stays within the
            # FFMA kernel's 2e-6; the bar leaves room for the deepest stacks
            bar = 2e-5
        assert error < bar * scale, (n_layers, error, scale)
        assert y[(row_seq < 0).cpu()].abs().max().item() == 0
        # The stack equals its layers launched one at a time, bit for bit: a
        # layer's fp32 output is rounded to the operand format at the same
        # point either way, and every row's sums run in the same order
        # wherever the row sits in a tile.  In bf16 each layer is also held
        # to a bf16-emulating reference given the same input (through a deep
        # stack the rounding flips of fp32 against fp64 sums add up, so the
        # whole stack is held to the fp64 bar above).
        h = x
        for layer in range(n_layers):
            one = _layer(stack, layer)
            out = eng.conv_stack(h.cuda(), row_seq, one, precision).cpu()
            if mode == 'bf16':
                emulated = _reference(one, h, row_seq, quantize=True)
                tight = (out.double() - emulated).abs().max().item()
                layer_scale = max(emulated.abs().max().item(), 1.0)
                assert tight < 2e-3 * layer_scale, (n_layers, layer, tight, layer_scale)
            h = out
        assert torch.equal(h, y), n_layers
        if mode == 'bf16':
            exact = eng.conv_stack(x.cuda(), row_seq, stack, _precision('fp32')).cpu()
            assert not torch.equal(exact, y)
        again = eng.conv_stack(x.cuda(), row_seq, stack, precision).cpu()
        assert torch.equal(again, y)


@pytest.mark.parametrize('kernel', KERNELS)
@pytest.mark.parametrize('mode', MODES)
def test_conv_stack_tc_too_deep_is_an_error(eng, mode, kernel):
    """One layer past the deepest stack is refused, not launched"""
    from emphases_b200 import _lib
    n_layers = _deepest(kernel) + 1
    stack = _random_stack(kernel, n_layers, 'relu', 5)
    row_seq, x = _rows(eng, kernel, [100, 3, 250], 5)
    with pytest.raises(_lib.EmphasesB200Error):
        eng.conv_stack(x.cuda(), row_seq, stack, _precision(mode))
    torch.cuda.synchronize()


###############################################################################
# B. Pooling, the API and the single-utterance call
###############################################################################


def _corpus(eng, emphases, kernel, seeds):
    """packed plan of synthetic utterances with (k - 1) / 2 separator rows"""
    from emphases_b200 import engine
    emphases.configure(ENCODER_KERNEL_SIZE=kernel)
    assert engine.separator_rows() == (kernel - 1) // 2
    utterances = []
    for seed in seeds:
        times, audio = oracle.synthetic_utterance(seed)
        utterances.append((np.asarray(times), audio.shape[-1]))
    plan = engine.make_plan(utterances)
    views = eng.upload_plan(plan)
    row_seq = eng.row_index(views['row_start'], views['n_rows'], plan.n_seq, plan.total_rows)
    return utterances, plan, views, row_seq


@pytest.mark.parametrize('method', ['sum', 'average', 'max', 'center'])
@pytest.mark.parametrize('kernel', KERNELS)
@pytest.mark.parametrize('mode', MODES)
def test_fused_pooling_kernel_sizes(eng, emphases, mode, kernel, method):
    """emph_conv_stack_pool == emph_conv_stack followed by emph_pool_words:
    max / center bit for bit, sum / average within 2e-6 of the largest value"""
    precision = _precision(mode)
    stack = _random_stack(kernel, 7, 'relu', 30 + kernel)
    _, plan, views, row_seq = _corpus(eng, emphases, kernel, range(300, 309))
    assert plan.words_disjoint()
    generator = torch.Generator().manual_seed(3)
    x = torch.randn(plan.total_rows, 80, generator=generator).cuda()
    x[row_seq < 0] = 0
    frames = eng.conv_stack(x, row_seq, stack, precision)
    separate = eng.pool(
        frames, views['row_start'], views['n_rows'], views['word_seq'],
        views['word_lo'], views['word_hi'], method)
    fused, kept = eng.conv_stack_pool(
        x, row_seq, stack, precision, views, plan.total_word_rows, method,
        keep_frames=True)
    assert torch.equal(kept, frames)
    keep = torch.from_numpy(plan.word_seq >= 0).cuda()
    assert (fused[~keep] == 0).all()
    if method in ('max', 'center'):
        assert torch.equal(fused[keep], separate[keep])
    else:
        scale = separate[keep].abs().max().item()
        assert (fused[keep] - separate[keep]).abs().max().item() < 2e-6 * scale
    alone, none = eng.conv_stack_pool(
        x, row_seq, stack, precision, views, plan.total_word_rows, method)
    assert none is None and torch.equal(alone, fused)


@pytest.mark.parametrize('kernel', KERNELS)
def test_fused_pooling_segment_assignment_kernel_sizes(eng, emphases, kernel):
    """A one-layer identity stack (centre tap = I) in bf16x6 passes frame
    indicators and indices through unchanged, so the fused sums recover every
    word's [lo, hi) exactly"""
    from emphases_b200 import _lib, engine
    utterances, plan, views, row_seq = _corpus(eng, emphases, kernel, range(200, 206))
    weights = torch.zeros(1, kernel, 80, 80)
    weights[0, (kernel - 1) // 2] = torch.eye(80)
    stack = engine.ConvStack(
        weights.cuda(), torch.zeros(1, 80).cuda(),
        np.asarray([_lib.ACT_NONE], dtype=np.int32), kernel, 80)
    x = torch.zeros(plan.total_rows, 80)
    for u in range(plan.n_seq):
        s, n = int(plan.row_start[u]), int(plan.n_rows[u])
        x[s:s + n, 0] = 1
        x[s:s + n, 1] = torch.arange(n, dtype=torch.float32)
    pooled, _ = eng.conv_stack_pool(
        x.cuda(), row_seq, stack, _lib.PREC_BF16X6_TC, views, plan.total_word_rows, 'sum')
    pooled = pooled.cpu()
    center, _ = eng.conv_stack_pool(
        x.cuda(), row_seq, stack, _lib.PREC_BF16X6_TC, views, plan.total_word_rows, 'center')
    center = center.cpu()
    for u in range(plan.n_seq):
        expected = oracle.word_bounds([tuple(t) for t in utterances[u][0].tolist()])
        s = int(plan.word_row_start[u])
        for j, (lo, hi) in enumerate(expected):
            hi = min(hi, int(plan.n_rows[u]))
            assert pooled[s + j, 0].item() == hi - lo
            assert pooled[s + j, 1].item() == (lo + hi - 1) * (hi - lo) // 2
            assert center[s + j, 1].item() == (lo + hi) // 2


SWEEP_SHAPES = [
    dict(ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=7),
    dict(ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=1),
]


@pytest.mark.parametrize('method', ['sum', 'max'])
@pytest.mark.parametrize('location', ['input', 'intermediate', 'inference', 'loss'])
@pytest.mark.parametrize('shape', SWEEP_SHAPES, ids=lambda d: '-'.join(map(str, d.values())))
@pytest.mark.parametrize('mode', MODES)
def test_sweep_shapes_on_tensor_cores(emphases, mode, shape, location, method):
    """The sweep's kernel sizes end to end through from_alignments_and_audio,
    random init with x1.5 weights, against the oracle: 1e-5 (bf16x6), 2e-5
    (bf16x3), 2e-3 (bf16; 1e-2 where frame logits are summed per word)"""
    emphases.configure(
        PRECISION=mode, DOWNSAMPLE_LOCATION=location, DOWNSAMPLE_METHOD=method, **shape)
    torch.manual_seed(3)
    model = emphases.Model()
    for parameter in model.parameters():
        if parameter.dim() > 1:
            parameter.data.mul_(1.5)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().eval()
    config = dict(DOWNSAMPLE_LOCATION=location, DOWNSAMPLE_METHOD=method, **shape)
    alignments, audios, expected = [], [], []
    for seed in range(3):
        times, audio = oracle.synthetic_utterance(1200 + seed, duration=2.5 + seed)
        alignments.append(emphases.Alignment.from_times(times))
        audios.append(audio)
        expected.append(oracle.from_alignment_and_audio(times, audio, state, config))
    scores = emphases.from_alignments_and_audio(
        alignments, audios, 16000, model=model, gpu=0)
    bar = {'bf16': 2e-3, 'bf16x3': 2e-5, 'bf16x6': 1e-5}[mode]
    if mode == 'bf16' and method == 'sum' and location in ('inference', 'loss'):
        # the score is a sigmoid of the SUM of the word's ~25 frame logits,
        # each with bf16's error: 5.7e-3 / 6.8e-3 measured (B200)
        bar = 1e-2
    for got, want in zip(scores, expected):
        assert got.shape == want.shape
        assert (got - want).abs().max() < bar


def test_path_selection(eng):
    """80-channel stacks of kernel size 5 and 7 take the tensor-core modes;
    128 channels stays on the FFMA kernel"""
    from emphases_b200 import _lib, engine
    lib = _lib.load()
    for kernel in KERNELS:
        stack = engine.ConvStack(None, None, np.zeros(7, dtype=np.int32), kernel, 80)
        wide = engine.ConvStack(None, None, np.zeros(7, dtype=np.int32), kernel, 128)
        for mode in MODES:
            precision = _precision(mode)
            assert engine.frame_precision(precision, stack) == precision
            assert engine.frame_precision(precision, wide) == _lib.PREC_FP32
            assert engine.word_precision(precision, wide) == _lib.PREC_FP32
            assert lib.emph_conv_weights_tc_bytes(7, 80, kernel, precision) > 0
            assert lib.emph_conv_weights_tc_bytes(7, 128, kernel, precision) == 0
        assert engine.word_precision(_precision('bf16'), stack) == _lib.PREC_BF16X3_TC
        assert engine.word_precision(_precision('bf16x3'), stack) == _lib.PREC_BF16X3_TC
        assert engine.word_precision(_precision('bf16x6'), stack) == _lib.PREC_BF16X6_TC
        assert engine.frame_precision(_lib.PREC_FP32, stack) == _lib.PREC_FP32


@pytest.mark.parametrize('kernel', KERNELS)
@pytest.mark.parametrize('mode', MODES)
def test_single_utterance_native_call_kernel_sizes(emphases, mode, kernel):
    """emph_infer_utterance (one separator row each side) gives bit for bit
    what the batched path gives with (k - 1) / 2 separator rows"""
    from emphases_b200 import single
    emphases.configure(
        PRECISION=mode, DOWNSAMPLE_METHOD='max', ENCODER_KERNEL_SIZE=kernel,
        DECODER_KERNEL_SIZE=kernel)
    device = torch.device('cuda', 0)
    torch.manual_seed(4)
    model = emphases.Model().to(device).eval()
    for seed in range(3):
        times, audio = oracle.synthetic_utterance(700 + seed, duration=0.8 + 1.7 * seed)
        alignment = emphases.Alignment.from_times(times)
        fast = single.from_alignment_and_audio(model, alignment, audio, 16000, device)
        assert fast is not None
        slow = emphases.from_alignments_and_audio(
            [alignment], [audio], 16000, model=model, gpu=0, to_cpu=False)[0]
        assert fast.shape == slow.shape == (1, len(times))
        assert torch.equal(fast, slow), seed
