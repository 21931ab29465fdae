"""Training of the convolution model with dropout (DROPOUT = p: Conv1d ->
activation -> Dropout in every block of frame_encoder and word_decoder,
emphases/model/layers/convolution.py:25-30).

A. emph_conv_dropout_forward / emph_activation_dropout_backward on a ragged
   packed layout with separator rows, against the masks replayed through
   emph_dropout_keep and fp64 torch autograd.
B. The native step and the per-kernel path draw the same masks although they
   pack rows differently, and the same torch seed gives the same step.
C. The whole model at p = 0.1 against an fp64 reference built from the
   oracle's pieces with the replayed masks: each block's output times the mask
   of emph_dropout_keep over the reference's padded (N, C, width) tensor.
D. p = 0 changes nothing, eval mode ignores dropout, Adam steps lower the loss,
   and a training-mode forward without autograd still raises.

The whole-model tolerances are those of tests/test_training_gpu.py and
tests/test_training_backward_gpu.py; the kernel bounds were measured on a B200
at a 1000 W power limit, with the value beside them.  Every error is printed.
"""
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from golden_util import state_from_golden
from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C = 80
P = 0.1
METHODS = ['sum', 'average', 'max', 'center']
LOCATIONS = ['intermediate', 'input', 'loss', 'inference']


@pytest.fixture
def emphases():
    import emphases_b200
    emphases_b200.reset_configuration()
    yield emphases_b200
    emphases_b200.reset_configuration()


@pytest.fixture(scope='module')
def lib():
    from emphases_b200 import _lib
    _lib.load()
    return _lib


def _within(what, error, bound):
    print(f'measured {what}: {error:.3e} (bound {bound:.1e})')
    assert np.isfinite(error) and error <= bound, (what, error, bound)


def _keep(lib, seed, site, first, count, p):
    keep = torch.empty(count, dtype=torch.uint8, device='cuda')
    lib.call('emph_dropout_keep', seed, site, first, count, p, lib.ptr(keep), lib.stream_ptr())
    return keep.cpu().bool()


def _seed_of(torch_seed):
    """the dropout seed a training forward draws after torch.manual_seed"""
    torch.manual_seed(torch_seed)
    return int(torch.randint(0, 2 ** 62, ()))


###############################################################################
# A. Kernels
###############################################################################


def _ragged(width, kept, gap):
    """row_start, row_seq, total: sequence n keeps kept[n] <= width rows, with
    `gap` separator rows before each"""
    starts, row = [], gap
    for n in kept:
        starts.append(row)
        row += n + gap
    row_seq = np.full(row, -1, dtype=np.int32)
    for u, (s, n) in enumerate(zip(starts, kept)):
        row_seq[s:s + n] = u
    return np.asarray(starts, dtype=np.int32), row_seq, row


ACTS = {0: lambda x: x, 1: torch.relu, 2: torch.nn.functional.gelu,
        3: torch.nn.functional.leaky_relu, 4: torch.nn.functional.silu}


@pytest.mark.parametrize('act', [0, 1, 2, 3, 4])
@pytest.mark.parametrize('p', [0.0, P])
def test_kernels_against_replayed_masks(lib, act, p):
    width, kept, gap = 70, [70, 1, 33, 70, 2, 69], 2
    starts, row_seq, total = _ragged(width, kept, gap)
    generator = torch.Generator().manual_seed(act)
    x = torch.randn(total, C, generator=generator, dtype=torch.float64) * 3
    dy = torch.randn(total, C, generator=generator, dtype=torch.float64)  # separators too
    x, dy = x.float().double(), dy.float().double()
    seed, site = 987654321987, lib.dropout_site(1, 4, lib.DROPOUT_CONV)
    d_x, d_dy = x.float().cuda(), dy.float().cuda()
    d_seq, d_start = torch.from_numpy(row_seq).cuda(), torch.from_numpy(starts).cuda()
    stream = lib.stream_ptr()

    def forward(source, a, out):
        lib.call('emph_conv_dropout_forward', lib.ptr(source), lib.ptr(d_seq), lib.ptr(d_start),
                 total, C, width, a, seed, site, p, lib.ptr(out), stream)

    y = torch.full_like(d_x, 7.)
    forward(d_x, act, y)
    activated = torch.empty_like(d_x)
    lib.call('emph_activation_forward', lib.ptr(d_x), lib.ptr(d_seq), total, C, act,
             lib.ptr(activated), stream)
    in_place = activated.clone()
    forward(in_place, lib.ACT_NONE, in_place)
    torch.cuda.synchronize()

    # the mask of element (n, w, c) is emph_dropout_keep's, in (N, width, C) order
    valid = torch.from_numpy(row_seq) >= 0
    keep = _keep(lib, seed, site, 0, len(kept) * width * C, p).reshape(len(kept), width, C)
    mask = torch.zeros(total, C, dtype=torch.bool)
    for n, (s, count) in enumerate(zip(starts, kept)):
        mask[s:s + count] = keep[n, :count]
    factor = mask.double() / (1 - p)
    xr = x.clone().requires_grad_(True)
    expected = ACTS[act](xr) * factor
    (expected[valid] * dy[valid]).sum().backward()

    assert torch.all(y.cpu()[~valid] == 0) and torch.all(in_place.cpu()[~valid] == 0)
    dropped = valid[:, None] & ~mask
    assert torch.all(y.cpu()[dropped] == 0)
    if p == 0:
        assert bool(mask[valid].all())
        assert torch.equal(y, activated)                      # emph_activation_forward
        assert torch.equal(in_place, activated)               # identity
    elif act in (0, 1, 3):
        # the activation commutes with a positive scale: in place on the
        # activated output is the same arithmetic
        assert torch.equal(y, in_place)
    scale = float(expected.detach().abs().max())
    error = float((y.cpu().double() - expected.detach())[valid].abs().max()) / scale
    # measured on a B200 (1000 W): <= 1.4e-7 (SiLU)
    _within(f'forward act {act} p {p}', error, 1e-6)

    key = d_x if act in (2, 4) else y          # GELU / SiLU: pre-activation, else the output
    dpre = torch.full_like(d_x, 7.)
    lib.call('emph_activation_dropout_backward', lib.ptr(d_dy), lib.ptr(key), lib.ptr(d_seq),
             lib.ptr(d_start), total, C, width, act, seed, site, p, lib.ptr(dpre), stream)
    torch.cuda.synchronize()
    assert torch.all(dpre.cpu()[~valid] == 0)
    assert torch.all(dpre.cpu()[dropped] == 0)
    want = xr.grad[valid]
    error = float((dpre.cpu().double()[valid] - want).abs().max()) / float(want.abs().max())
    # measured on a B200 (1000 W): <= 3.1e-7 (SiLU)
    _within(f'backward act {act} p {p}', error, 2e-6)


def test_drop_rate_is_p(lib):
    """the fraction of dropped elements of one layer is within 5 sigma of p"""
    width, kept = 2000, [2000, 1500, 1999, 7, 2000] * 8
    starts, row_seq, total = _ragged(width, kept, 1)
    ones = torch.ones(total, C, device='cuda')
    d_seq, d_start = torch.from_numpy(row_seq).cuda(), torch.from_numpy(starts).cuda()
    lib.call('emph_conv_dropout_forward', lib.ptr(ones), lib.ptr(d_seq), lib.ptr(d_start),
             total, C, width, lib.ACT_RELU, 5, lib.dropout_site(0, 2, lib.DROPOUT_CONV), P,
             lib.ptr(ones), lib.stream_ptr())
    values = ones.cpu()[torch.from_numpy(row_seq) >= 0]
    n = values.numel()
    rate = float((values == 0).double().mean())
    sigma = math.sqrt(P * (1 - P) / n)
    print(f'drop rate {rate:.6f} over {n} elements, sigma {sigma:.1e}')
    assert abs(rate - P) < 5 * sigma
    assert torch.all((values == 0) | (values == torch.tensor(1 / 0.9, dtype=torch.float32)))


###############################################################################
# Whole model
###############################################################################


def padded_batch(seed=0, items=3, past_length=False):
    """tests/test_training_gpu.py's batch; past_length: item 1's last word ends
    27 frames past its length (the reference pools the padded columns)"""
    generator = torch.Generator().manual_seed(seed)
    lengths = [260, 143, 201][:items]
    words = [9, 4, 6][:items]
    tmax, wmax = max(lengths), max(words)
    features = torch.zeros(items, 80, tmax)
    bounds = torch.zeros(items, 2, wmax, dtype=torch.long)
    for i, (t, w) in enumerate(zip(lengths, words)):
        features[i, :, :t] = torch.randn(80, t, generator=generator)
        cuts = torch.sort(torch.randperm(t - 2, generator=generator)[:w - 1] + 1).values
        edges = torch.cat([torch.tensor([0]), cuts, torch.tensor([t])])
        bounds[i, 0, :w] = edges[:-1]
        bounds[i, 1, :w] = edges[1:]
    if past_length:
        bounds[1, 1, 3] = 170
    targets = torch.rand(items, 1, wmax, generator=generator)
    return (features, torch.tensor(lengths), bounds, torch.tensor(words), targets)


def _bench_batch():
    """synthetic_batch() of tools/train_bench.py, the batch it times"""
    spec = importlib.util.spec_from_file_location(
        'train_bench', os.path.join(ROOT, 'tools', 'train_bench.py'))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module.synthetic_batch(100)


def _with_dropout_keys(state):
    """a DROPOUT=None state dict (Sequential stride 2) -> stride 3"""
    out = {}
    for key, value in state.items():
        parts = key.split('.')
        if parts[0] in ('frame_encoder', 'word_decoder'):
            parts[1] = str(int(parts[1]) // 2 * 3)
        out['.'.join(parts)] = value
    return out


def _model(emphases, golden, p=P, **config):
    """golden 'sweep' weights in a model configured with DROPOUT = p"""
    emphases.configure(DROPOUT=p, **config)
    model = emphases.Model()
    state = state_from_golden(golden('sweep'))
    if p is not None:
        state = _with_dropout_keys(state)
    own = model.state_dict()
    state = {k: v for k, v in state.items() if k in own}
    model.load_state_dict(state)
    return model.cuda().train(), state


def _step(emphases, model, batch, torch_seed=None, per_kernel=False):
    """(loss, logits, {name: grad}) of one training step on the device"""
    from emphases_b200 import training
    features, frame_lengths, bounds, word_lengths, targets = batch
    model.zero_grad(set_to_none=True)
    if torch_seed is not None:
        torch.manual_seed(torch_seed)
    if per_kernel:
        logits = training._ConvModelFunction.apply(
            model, features.cuda(), bounds, word_lengths, *model.parameters())
    else:
        logits = model(features.cuda(), frame_lengths, bounds, word_lengths)
    value = emphases.loss(
        logits, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()
    return (value.detach().double().cpu(), logits.detach().double().cpu(),
            {n: p.grad.detach().double().cpu().clone() for n, p in model.named_parameters()})


def _reference(lib, state, batch, config, seed, p):
    """fp64 autograd of the reference's training forward, every block's output
    times its replayed mask / (1 - p): (loss, logits, {name: grad})"""
    from emphases_b200 import _lib
    config = dict(oracle.default_config(), **config)
    location, method = config['DOWNSAMPLE_LOCATION'], config['DOWNSAMPLE_METHOD']
    activation = oracle._ACTIVATIONS[config['ACTIVATION']]
    features, frame_lengths, bounds, word_lengths, targets = batch
    params = {k: v.double().clone().requires_grad_(True) for k, v in state.items()}
    channels = params['input_layer.weight'].shape[0]
    conv = oracle._conv

    def stack(prefix, x, stack_id):
        for i in range(config['LAYERS']):
            x = activation(conv(x, params[f'{prefix}.{3 * i}.weight'],
                                params[f'{prefix}.{3 * i}.bias']))
            n, _, width = x.shape
            site = _lib.dropout_site(stack_id, i, _lib.DROPOUT_CONV)
            keep = _keep(lib, seed, site, 0, n * width * channels, p)
            x = x * keep.reshape(n, width, channels).permute(0, 2, 1).double() / (1 - p)
        return x

    def input_layer(x):
        return conv(x, params['input_layer.weight'], params['input_layer.bias'])

    def output_layer(x):
        return conv(x, params['output_layer.weight'], params['output_layer.bias'])

    features = features.double()
    if location == 'input':                       # oracle.model_forward, model/core.py:41-87
        segments, seg_bounds, seg_lengths = oracle.segment(features, bounds, word_lengths)
        frames = stack('frame_encoder', input_layer(segments), 0)
        if method == 'average':
            words = frames.mean(dim=2, keepdim=True)
        elif method == 'max':
            words = frames.max(dim=2, keepdim=True).values
        elif method == 'sum':
            words = frames.sum(dim=2, keepdim=True)
        else:
            words = oracle.downsample(
                frames, seg_bounds, torch.ones((len(seg_lengths),), dtype=torch.long), 'center')
        words = words.squeeze(2).transpose(0, 1).reshape(
            words.shape[1], bounds.shape[0], bounds.shape[2]).permute(1, 0, 2)
        words = stack('word_decoder', words * oracle.mask_from_lengths(word_lengths), 1)
        logits = output_layer(words)
    else:
        frames = stack('frame_encoder', input_layer(features), 0)
        if location == 'inference':
            logits = output_layer(frames)
        else:
            words = oracle.downsample(frames, bounds, word_lengths, method)
            assert words.shape[2] == bounds.shape[2]     # width Wmax
            if location == 'intermediate':
                words = stack('word_decoder', words, 1)
            logits = output_layer(words)
    if location == 'inference':
        value = oracle.loss(logits, targets.double(), word_lengths, 'bce', frame_lengths, bounds,
                            'linear')
    else:
        value = oracle.loss(logits, targets.double(), word_lengths, config['LOSS'])
    value.backward()
    return (value.detach(), logits.detach(),
            {k: v.grad for k, v in params.items() if v.grad is not None})


def _compare(what, got, want, grad_bound=2e-4):
    """tests/test_training_gpu.py's bars: loss 1e-5, logits rtol 1e-5 + atol
    2e-5, every gradient 2e-4 x its largest element"""
    (value, logits, grads), (ref_value, ref_logits, ref_grads) = got, want
    _within(f'{what} loss', abs(float(value) - float(ref_value)) / max(1., abs(float(ref_value))),
            1e-5)
    torch.testing.assert_close(logits, ref_logits, rtol=1e-5, atol=2e-5)
    assert set(grads) == set(ref_grads)
    worst = max(
        (float((grads[n] - ref_grads[n]).abs().max()) /
         (float(ref_grads[n].abs().max()) + 1e-12), n) for n in grads)
    _within(f'{what} worst gradient ({worst[1]})', worst[0], grad_bound)


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('location', LOCATIONS)
def test_per_kernel_path_matches_fp64(emphases, golden, lib, monkeypatch, location, method):
    from emphases_b200 import training
    monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    config = {'DOWNSAMPLE_LOCATION': location, 'DOWNSAMPLE_METHOD': method}
    model, state = _model(emphases, golden, **config)
    batch = padded_batch()
    assert not training.native_step_supported(model, batch[0].cuda())
    got = _step(emphases, model, batch, 31)
    want = _reference(lib, state, batch, config, _seed_of(31), P)
    _compare(f'per-kernel {location}/{method}', got, want)


@pytest.mark.parametrize('path', ['native', 'kernels'])
@pytest.mark.parametrize('location,method', [
    ('intermediate', 'sum'), ('intermediate', 'max'), ('intermediate', 'center'),
    ('loss', 'average'), ('loss', 'max')])
def test_native_and_past_length_match_fp64(emphases, golden, lib, monkeypatch, path, location,
                                           method):
    """the native step at the locations it covers, and a word ending past its
    item's length on both paths"""
    from emphases_b200 import training
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    config = {'DOWNSAMPLE_LOCATION': location, 'DOWNSAMPLE_METHOD': method}
    model, state = _model(emphases, golden, **config)
    for past_length in (False, True):
        batch = padded_batch(seed=2, past_length=past_length)
        assert training.native_step_supported(model, batch[0].cuda()) == (path == 'native')
        got = _step(emphases, model, batch, 8)
        want = _reference(lib, state, batch, config, _seed_of(8), P)
        _compare(f'{path} {location}/{method} past_length={past_length}', got, want)


@pytest.mark.parametrize('path', ['native', 'kernels'])
@pytest.mark.parametrize('activation', ['GELU', 'SiLU'])
def test_gelu_silu_match_fp64(emphases, golden, lib, monkeypatch, path, activation):
    """dropout in place of emph_activation_forward, the pre-activation kept"""
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    model, state = _model(emphases, golden, ACTIVATION_FUNCTION=getattr(torch.nn, activation))
    batch = padded_batch(seed=3)
    got = _step(emphases, model, batch, 12)
    want = _reference(lib, state, batch, {'ACTIVATION': activation.lower()}, _seed_of(12), P)
    _compare(f'{path} {activation}', got, want)


def test_native_step_at_benchmark_shape(emphases, lib):
    """tools/train_bench.py's batch (37 items, <= 75,000 padded frames) on the
    native bf16x6 step, with tests/test_training_backward_gpu.py's bounds at
    that shape: (loss 1e-6, logits 5e-6, per-parameter Frobenius 3e-3 and max
    5e-3 relative), the first frame layers being ill-conditioned in fp32"""
    from emphases_b200 import training
    assert training.TRAIN_PRECISION == 'bf16x6'
    emphases.configure(DROPOUT=P)
    torch.manual_seed(0)
    model = emphases.Model()
    for parameter in model.parameters():
        if parameter.dim() > 1:
            parameter.data.mul_(1.4)          # as the existing test: no dead ReLUs
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().train()
    batch = _bench_batch()
    assert training.native_step_supported(model, batch[0].cuda())
    value, logits, grads = _step(emphases, model, batch, 21)
    ref_value, ref_logits, ref_grads = _reference(lib, state, batch, {}, _seed_of(21), P)
    _within('bench loss', abs(float(value - ref_value)) / abs(float(ref_value)), 1e-6)
    _within('bench logits', float((logits - ref_logits).abs().max() / ref_logits.abs().max()),
            5e-6)
    for name, want in ref_grads.items():
        got = grads[name]
        _within(f'bench {name} frobenius', float((got - want).norm() / want.norm()), 3e-3)
        _within(f'bench {name} max', float((got - want).abs().max() / want.abs().max()), 5e-3)


###############################################################################
# B. Packing independence and reproducibility
###############################################################################


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3', 'bf16x6', 'bf16x3+bf16x6'])
def test_native_step_matches_per_kernel_path(emphases, golden, monkeypatch, precision):
    """The native step keeps fewer frame rows per item and other word gaps
    than the per-kernel path, yet draws the same masks from the same torch
    seed: tests/test_training_gpu.py's comparison of the two at p = 0.1, with
    the flat gradient buffer and the accumulation of a second backward"""
    from emphases_b200 import training
    batch = padded_batch(seed=5)
    results = {}
    for name in ('native', 'kernels'):
        model, _ = _model(emphases, golden)
        if name == 'native':
            monkeypatch.setattr(training, 'TRAIN_PRECISION', precision)
            assert training.native_step_supported(model, batch[0].cuda())
            native = model
        results[name] = _step(emphases, model, batch, 44, per_kernel=name == 'kernels')
    tolerance = {'fp32': 1e-6, 'bf16x3': 3e-5, 'bf16x6': 3e-6, 'bf16x3+bf16x6': 3e-5}[precision]
    gradient_tolerance = {
        'fp32': 2e-5, 'bf16x3': 5e-2, 'bf16x6': 1e-4, 'bf16x3+bf16x6': 5e-2}[precision]
    assert (results['native'][1] - results['kernels'][1]).abs().max() < tolerance
    for name, want in results['kernels'][2].items():
        got = results['native'][2][name]
        scale = want.abs().max().item() + 1e-12
        assert (got - want).abs().max().item() < gradient_tolerance * scale + 1e-8, name
    flat_state = native._native_train_state
    assert all(flat_state.aliases_flat(p, i) for i, p in enumerate(flat_state.ordered))
    # a second step from the same torch seed accumulates the same gradients
    features, frame_lengths, bounds, word_lengths, targets = batch
    torch.manual_seed(44)
    scores = native(features.cuda(), frame_lengths, bounds, word_lengths)
    emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True).backward()
    for name, parameter in native.named_parameters():
        want = 2 * results['native'][2][name]
        scale = want.abs().max().item() + 1e-12
        assert (parameter.grad.double().cpu() - want).abs().max().item() < 1e-5 * scale + 1e-9, \
            name


@pytest.mark.parametrize('path', ['native', 'kernels'])
def test_same_seed_same_step_other_seed_other_masks(emphases, golden, monkeypatch, path):
    """the same torch seed gives bitwise-equal loss and logits (the weight
    gradients sum CTA partials with float atomics: equal to rounding); another
    seed other logits; train-mode logits differ from eval-mode logits"""
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    model, _ = _model(emphases, golden)
    batch = padded_batch(seed=6)
    runs = [_step(emphases, model, batch, seed) for seed in (5, 5, 6)]
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for name, want in runs[0][2].items():
        scale = want.abs().max().item() + 1e-12
        assert (runs[1][2][name] - want).abs().max().item() < 1e-5 * scale + 1e-9, name
    assert not torch.equal(runs[0][1], runs[2][1])
    features, frame_lengths, bounds, word_lengths, _ = batch
    model.eval()
    with torch.no_grad():
        evaluated = model(features.cuda(), frame_lengths, bounds, word_lengths).double().cpu()
    assert not torch.allclose(evaluated, runs[0][1], rtol=1e-3, atol=1e-3)


###############################################################################
# D. p = 0, eval mode, training, no autograd
###############################################################################


def _kernel_names(step):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize('path', ['native', 'kernels'])
def test_p0_is_no_dropout(emphases, golden, monkeypatch, path):
    """DROPOUT=0.0 gives the logits of DROPOUT=None bit for bit and the same
    gradients (to float-atomic rounding) and launches the same kernels.  A
    DROPOUT=None step draws no torch random number, a model with Dropout
    modules one (its seed)"""
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    batch = padded_batch(seed=7)
    steps, kernels = {}, {}
    for p in (None, 0.0, P):
        emphases.reset_configuration()
        model, _ = _model(emphases, golden, p=p)
        torch.manual_seed(9)
        steps[p] = _step(emphases, model, batch)
        after = torch.rand(4)
        torch.manual_seed(9)
        fresh = torch.rand(4) if p is None else (torch.randint(0, 2 ** 62, ()), torch.rand(4))[1]
        assert torch.equal(after, fresh), p          # None: no draw; with modules: one
        kernels[p] = _kernel_names(lambda: _step(emphases, model, batch))
    assert torch.equal(steps[None][0], steps[0.0][0])
    assert torch.equal(steps[None][1], steps[0.0][1])
    for name, want in steps[None][2].items():
        name3 = _with_dropout_keys({name: 0}).popitem()[0]
        scale = want.abs().max().item() + 1e-12
        assert (steps[0.0][2][name3] - want).abs().max().item() < 1e-5 * scale + 1e-9, name
    assert kernels[None] == kernels[0.0]
    assert not any('dropout' in k for k in kernels[None])
    assert any('conv_dropout_forward' in k for k in kernels[P])
    assert any('activation_dropout_backward' in k for k in kernels[P])
    assert not torch.equal(steps[None][1], steps[P][1])


def test_modules_set_to_p0_train_without_dropout(emphases, golden):
    """p is read from the Dropout modules, not from DROPOUT"""
    batch = padded_batch(seed=7)
    model, _ = _model(emphases, golden, p=P)
    for module in model.modules():
        if isinstance(module, torch.nn.Dropout):
            module.p = 0.
    zero = _step(emphases, model, batch, 1)
    emphases.reset_configuration()
    reference, _ = _model(emphases, golden, p=None)
    none = _step(emphases, reference, batch, 1)
    assert torch.equal(zero[1], none[1])


def test_adam_steps_lower_the_loss(emphases, golden):
    model, _ = _model(emphases, golden)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    batch = padded_batch(1)
    batch = (batch[0].cuda(),) + batch[1:4] + ((batch[4] > 0.5).float().cuda(),)
    torch.manual_seed(0)
    losses = [float(emphases.training.train_step(model, optimizer, batch)) for _ in range(30)]
    print('losses', losses[0], losses[-1])
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < np.mean(losses[:5])


def test_training_forward_without_autograd_still_raises(emphases, golden):
    model, _ = _model(emphases, golden)
    features, frame_lengths, bounds, word_lengths, _ = padded_batch()
    with torch.no_grad(), pytest.raises(NotImplementedError, match='without autograd'):
        model(features.cuda(), frame_lengths, bounds, word_lengths)
