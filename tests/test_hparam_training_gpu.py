"""Training of every convolution model of the reference's hyper-parameter
sweep (config/hparam-search): CHANNELS 64 and 128, kernel sizes 5 and 7.

A model trains at the kernel width inference uses (80, or 128 when a conv is
wider), its parameters zero-padded; the weight gradients of 80 channels at
kernel sizes 5 / 7 and of 128 channels run on the split-bf16 mma.sync kernel.

A. emph_conv_weight_grad at every new (channels, kernel size) against fp64, at
   row counts around its 64-row tiles and the benchmarked batch's 75,000 rows,
   with the tests/test_training_backward_gpu.py bars of that kernel.
B. The whole per-kernel step against fp64 autograd on a 3-item padded batch
   at every location, with GELU and with dropout (masks replayed through
   emph_dropout_keep on the padded layout), and on tools/train_bench.py's batch.
C. Gradient shapes, Adam, and the shapes that still raise.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOCATIONS = ['intermediate', 'input', 'loss', 'inference']
P = 0.1


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
    """error <= bound (error may be an array: its worst element)"""
    worst = float(np.max(np.asarray(error))) if np.size(error) else 0.
    print(f'measured {what}: {worst:.3e} (bound {bound:.1e})')
    assert np.isfinite(worst) and worst <= bound, (what, worst, bound)


def _ratio(error, bound):
    """worst elementwise error / bound (bound > 0 where it matters)"""
    error, bound = error.double(), bound.double()
    return float(torch.where(error > 0, error / bound.clamp_min(1e-300), 0.).max())


###############################################################################
# A. The weight-gradient kernel
###############################################################################

# (channels, kernel size) served by the mma.sync kernel
NEW_SHAPES = [(80, 5), (80, 7), (128, 1), (128, 3), (128, 5), (128, 7)]


def _ragged_row_seq(total, rng, gap=1, first=0):
    """Sequence id per packed row, -1 on the `gap` separator rows between
    sequences: ragged lengths, one- and two-row sequences included"""
    seq = np.full(total, -1, dtype=np.int32)
    lengths = [1, 2, 1, 64, 3, 1]
    row, u = first, 0
    while row < total:
        n = lengths[u] if u < len(lengths) else int(rng.integers(1, 700))
        seq[row:row + n] = u
        row, u = row + n + gap, u + 1
    return seq


def _shifted(x, offset):
    """rows r + offset of x (zero outside), the operand of tap offset + half"""
    out = torch.zeros_like(x)
    n = x.shape[0]
    if abs(offset) >= n:
        return out
    if offset >= 0:
        out[:n - offset] = x[offset:]
    else:
        out[-offset:] = x[:n + offset]
    return out


@pytest.mark.parametrize('total', [1, 63, 64, 65, 9473, 75000])
@pytest.mark.parametrize('channels,kernel', NEW_SHAPES)
def test_weight_grad_against_fp64(lib, channels, kernel, total):
    """dW per tap and db against fp64 on ragged packed rows with (k - 1) / 2
    zero separator rows; dw and db start at 7 to show they are zeroed"""
    half = (kernel - 1) // 2
    rng = np.random.default_rng(total * 10 + kernel)
    seq = torch.from_numpy(_ragged_row_seq(total, rng, gap=max(1, half)))
    generator = torch.Generator().manual_seed(total + channels)
    x = torch.randn(total, channels, generator=generator)
    d = torch.randn(total, channels, generator=generator)
    x[seq < 0] = 0.
    d[seq < 0] = 0.
    x_dev, d_dev = x.cuda(), d.cuda()
    dw = torch.full((kernel, channels, channels), 7., device='cuda')
    db = torch.full((channels,), 7., device='cuda')
    lib.call('emph_conv_weight_grad', lib.ptr(x_dev), lib.ptr(d_dev), total, channels, kernel,
             lib.ptr(dw), lib.ptr(db), lib.stream_ptr())
    X, D = x_dev.double(), d_dev.double()
    got = dw.double()
    worst = 0.
    for tap in range(kernel):
        shifted = _shifted(X, tap - half)
        want = shifted.T @ D
        bound = shifted.abs().T @ D.abs()
        worst = max(worst, _ratio((got[tap] - want).abs(), bound))
    # split bf16 (16-bit operands): the bound is a weighted mean of the
    # products' relative errors, measured 1.2e-6 over many rows
    # (tests/test_training_backward_gpu.py).  With one row every element is
    # one product, whose error (a missing lo*lo term and the rounding of lo,
    # ~3 x 2^-16 at worst) does not average down: measured 2.2e-5 on a B200
    # (1000 W power limit)
    _within(f'{channels}/k{kernel} rows {total} dW / (|X|^T|dPre|)', worst,
            5e-5 if total == 1 else 1e-5)
    _within(f'{channels}/k{kernel} rows {total} db / sum|dPre|', _ratio(
        (db.double() - D.sum(0)).abs(), D.abs().sum(0)), 1e-6)


@pytest.mark.parametrize('channels,kernel', [(96, 3), (80, 9), (64, 3), (128, 9)])
def test_weight_grad_uncompiled_shape_fails(lib, channels, kernel):
    """a shape no kernel is built for returns EMPH_ENOSYS and writes nothing"""
    x = torch.ones(100, channels, device='cuda')
    dw = torch.full((kernel, channels, channels), 7., device='cuda')
    db = torch.full((channels,), 7., device='cuda')
    status = lib.load().emph_conv_weight_grad(
        lib.ptr(x), lib.ptr(x), 100, channels, kernel, lib.ptr(dw), lib.ptr(db),
        lib.stream_ptr())
    assert status == lib.ENOSYS
    assert b'not compiled in' in lib.load().emph_last_error()
    torch.cuda.synchronize()
    assert bool((dw == 7).all()) and bool((db == 7).all())


###############################################################################
# B. The whole step against fp64
###############################################################################


def padded_batch(seed=0):
    """tests/test_conv_dropout_training_gpu.py's 3-item batch"""
    generator = torch.Generator().manual_seed(seed)
    lengths, words = [260, 143, 201], [9, 4, 6]
    tmax, wmax = max(lengths), max(words)
    features = torch.zeros(3, 80, tmax)
    bounds = torch.zeros(3, 2, wmax, dtype=torch.long)
    for i, (t, w) in enumerate(zip(lengths, words)):
        features[i, :, :t] = torch.randn(80, t, generator=generator)
        cuts = torch.sort(torch.randperm(t - 2, generator=generator)[:w - 1] + 1).values
        edges = torch.cat([torch.tensor([0]), cuts, torch.tensor([t])])
        bounds[i, 0, :w] = edges[:-1]
        bounds[i, 1, :w] = edges[1:]
    targets = torch.rand(3, 1, wmax, generator=generator)
    return (features, torch.tensor(lengths), bounds, torch.tensor(words), targets)


def _bench_batch():
    """synthetic_batch() of tools/train_bench.py, the batch it times"""
    spec = importlib.util.spec_from_file_location(
        'train_bench', os.path.join(ROOT, 'tools', 'train_bench.py'))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module.synthetic_batch(100)


def _model(emphases, scale=1.5, seed=3, **config):
    """A configured model with random init, weights scaled as in
    tests/test_api_gpu.py::test_hyperparameter_shapes: (model, state)"""
    emphases.configure(**config)
    torch.manual_seed(seed)
    model = emphases.Model()
    for parameter in model.parameters():
        if parameter.dim() > 1:
            parameter.data.mul_(scale)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return model.cuda().train(), state


def _oracle_config(emphases):
    return dict(
        oracle.default_config(), CHANNELS=emphases.CHANNELS, LAYERS=emphases.LAYERS,
        ENCODER_KERNEL_SIZE=emphases.ENCODER_KERNEL_SIZE,
        DECODER_KERNEL_SIZE=emphases.DECODER_KERNEL_SIZE, DROPOUT=emphases.DROPOUT,
        DOWNSAMPLE_LOCATION=emphases.DOWNSAMPLE_LOCATION,
        DOWNSAMPLE_METHOD=emphases.DOWNSAMPLE_METHOD, LOSS=emphases.LOSS,
        ACTIVATION={'ReLU': 'relu', 'GELU': 'gelu', 'LeakyReLU': 'leaky_relu',
                    'SiLU': 'silu'}[emphases.ACTIVATION_FUNCTION.__name__])


def _keep(lib, seed, site, count, p):
    keep = torch.empty(count, dtype=torch.uint8, device='cuda')
    lib.call('emph_dropout_keep', seed, site, 0, count, p, lib.ptr(keep), lib.stream_ptr())
    return keep.cpu().bool()


def _reference(lib, state, batch, config, seed=None, width=None, dtype=torch.float64):
    """fp64 autograd of the reference's training forward: (loss, logits,
    {name: grad}).  With DROPOUT, every block's output is multiplied by its
    mask / (1 - p), replayed with emph_dropout_keep over the padded
    (N, width, `width` channels) layout the kernels run at, of which the
    model's own channels are the first"""
    from emphases_b200 import _lib
    location, method = config['DOWNSAMPLE_LOCATION'], config['DOWNSAMPLE_METHOD']
    p = config['DROPOUT']
    features, frame_lengths, bounds, word_lengths, targets = batch
    params = {k: v.to(dtype).clone().requires_grad_(True) for k, v in state.items()}
    if p is None:
        logits = oracle.model_forward(
            params, features.to(dtype), frame_lengths, bounds, word_lengths, config,
            training=True)
    else:
        activation = oracle._ACTIVATIONS[config['ACTIVATION']]
        channels, conv = config['CHANNELS'], oracle._conv

        def stack(prefix, x, stack_id):
            for i in range(config['LAYERS']):
                x = activation(conv(x, params[f'{prefix}.{3 * i}.weight'],
                                    params[f'{prefix}.{3 * i}.bias']))
                n, _, columns = x.shape
                site = _lib.dropout_site(stack_id, i, _lib.DROPOUT_CONV)
                keep = _keep(lib, seed, site, n * columns * width, p)
                keep = keep.reshape(n, columns, width)[:, :, :channels]
                x = x * keep.permute(0, 2, 1).to(dtype) / (1 - p)
            return x

        def input_layer(x):
            return conv(x, params['input_layer.weight'], params['input_layer.bias'])

        def output_layer(x):
            return conv(x, params['output_layer.weight'], params['output_layer.bias'])

        x = features.to(dtype)
        if location == 'input':                       # oracle.model_forward, model/core.py:41-87
            segments, seg_bounds, seg_lengths = oracle.segment(x, bounds, word_lengths)
            frames = stack('frame_encoder', input_layer(segments), 0)
            if method == 'average':
                words = frames.mean(dim=2, keepdim=True)
            elif method == 'max':
                words = frames.max(dim=2, keepdim=True).values
            elif method == 'sum':
                words = frames.sum(dim=2, keepdim=True)
            else:
                words = oracle.downsample(
                    frames, seg_bounds, torch.ones((len(seg_lengths),), dtype=torch.long),
                    'center')
            words = words.squeeze(2).transpose(0, 1).reshape(
                words.shape[1], bounds.shape[0], bounds.shape[2]).permute(1, 0, 2)
            words = stack('word_decoder', words * oracle.mask_from_lengths(word_lengths), 1)
            logits = output_layer(words)
        else:
            frames = stack('frame_encoder', input_layer(x), 0)
            if location == 'inference':
                logits = output_layer(frames)
            else:
                words = oracle.downsample(frames, bounds, word_lengths, method)
                if location == 'intermediate':
                    words = stack('word_decoder', words, 1)
                logits = output_layer(words)
    if location == 'inference':
        value = oracle.loss(logits, targets.to(dtype), word_lengths, 'bce', frame_lengths, bounds,
                            'linear')
    else:
        value = oracle.loss(logits, targets.to(dtype), word_lengths, config['LOSS'])
    value.backward()
    return (value.detach().double(), logits.detach().double(),
            {k: v.grad.double() for k, v in params.items() if v.grad is not None})


def _step(emphases, model, batch, torch_seed=None):
    """(loss, logits, {name: grad}) of one training step on the device"""
    features, frame_lengths, bounds, word_lengths, targets = batch
    model.zero_grad(set_to_none=True)
    if torch_seed is not None:
        torch.manual_seed(torch_seed)
    logits = model(features.cuda(), frame_lengths, bounds, word_lengths)
    value = emphases.loss(
        logits, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()
    for name, parameter in model.named_parameters():
        assert parameter.grad.shape == parameter.shape, name
    return (value.detach().double().cpu(), logits.detach().double().cpu(),
            {n: p.grad.detach().double().cpu().clone() for n, p in model.named_parameters()})


def _compare(what, got, want, fp32_grads=None, grad_bound=2e-4):
    """tests/test_training_gpu.py's bars: loss 1e-5, logits rtol 1e-5 + atol
    2e-5, every gradient 2e-4 x its largest element.  Where the reference
    computed in fp32 (`fp32_grads`) is itself further than that from fp64, a
    gradient is ill-conditioned in fp32 and its bar is 4x that distance."""
    (value, logits, grads), (ref_value, ref_logits, ref_grads) = got, want
    _within(f'{what} loss', abs(float(value) - float(ref_value)) / max(1., abs(float(ref_value))),
            1e-5)
    torch.testing.assert_close(logits, ref_logits.cpu(), rtol=1e-5, atol=2e-5)
    assert set(grads) == set(ref_grads)
    def error(grad, n):
        return float((grad - ref_grads[n]).abs().max()) / (float(ref_grads[n].abs().max()) + 1e-12)
    bounds = {n: grad_bound if fp32_grads is None else max(grad_bound, 4 * error(fp32_grads[n], n))
              for n in grads}
    worst = max((error(grads[n], n) / bounds[n], n) for n in grads)
    name = worst[1]
    _within(f'{what} worst gradient ({name})', error(grads[name], name), bounds[name])


SWEEP = [
    dict(CHANNELS=64),
    dict(CHANNELS=128),
    dict(ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=7),
    dict(ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=1),
    dict(CHANNELS=128, ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=1)]
WIDE = [
    dict(CHANNELS=channels, **extra, DOWNSAMPLE_LOCATION=location)
    for channels in (64, 128)
    for extra, locations in (
        (dict(ACTIVATION_FUNCTION=torch.nn.GELU), ['intermediate']),
        (dict(DROPOUT=P), LOCATIONS))
    for location in locations]


def _name(config):
    return '-'.join(
        f'{k}={getattr(v, "__name__", v)}' for k, v in config.items())


@pytest.mark.parametrize(
    'config', [dict(shape, DOWNSAMPLE_LOCATION=location)
               for shape in SWEEP for location in LOCATIONS] + WIDE, ids=_name)
def test_step_matches_fp64(emphases, lib, config):
    from emphases_b200 import training
    model, state = _model(emphases, **config)
    batch = padded_batch()
    assert not training.native_step_supported(model, batch[0].cuda())
    got = _step(emphases, model, batch, 31)
    torch.manual_seed(31)
    seed = int(torch.randint(0, 2 ** 62, ()))      # the one draw of a forward with dropout
    width = training._kernel_width(model)
    reference = _oracle_config(emphases)
    want = _reference(lib, state, batch, reference, seed, width)
    # CHANNELS=128, kernel size 5 at 'input': the fp32 reference is 4.4e-3
    # from fp64 on frame_encoder.0.weight (the step measured 4.4e-3 on a B200)
    fp32 = _reference(lib, state, batch, reference, seed, width, torch.float32)[2]
    _compare(_name(config), got, want, fp32)


@pytest.mark.parametrize('config', [
    dict(CHANNELS=128), dict(ENCODER_KERNEL_SIZE=7)], ids=_name)
def test_step_at_benchmark_shape(emphases, lib, config):
    """tools/train_bench.py's batch (37 items, <= 75,000 padded frames), with
    tests/test_training_backward_gpu.py's per-kernel bounds at that shape
    (loss 1e-6, logits 5e-6, per-parameter Frobenius 3e-3 and max 5e-3
    relative: the first frame layers' gradients are ill-conditioned in fp32)"""
    model, state = _model(emphases, scale=1.4, seed=0, **config)
    batch = _bench_batch()
    value, logits, grads = _step(emphases, model, batch)
    ref_value, ref_logits, ref_grads = _reference(lib, state, batch, _oracle_config(emphases))
    _within('bench loss', abs(float(value - ref_value)) / abs(float(ref_value)), 1e-6)
    _within('bench logits', float((logits - ref_logits).abs().max() / ref_logits.abs().max()),
            5e-6)
    for name, want in ref_grads.items():
        got = grads[name]
        _within(f'bench {name} frobenius', float((got - want).norm() / want.norm()), 3e-3)
        _within(f'bench {name} max', float((got - want).abs().max() / want.abs().max()), 5e-3)


###############################################################################
# C. Shapes, Adam, rejections
###############################################################################


def test_adam_steps_lower_the_loss_wide_long_kernel_dropout(emphases):
    """CHANNELS=128, kernel size 7, DROPOUT=0.1: every .grad has its
    parameter's shape (the padded channels are sliced off) and twenty Adam
    steps lower the loss"""
    model, _ = _model(emphases, CHANNELS=128, ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=7,
                      DROPOUT=P)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    batch = padded_batch(1)
    batch = (batch[0].cuda(),) + batch[1:4] + ((batch[4] > 0.5).float().cuda(),)
    torch.manual_seed(0)
    losses = []
    for _ in range(20):
        losses.append(float(emphases.training.train_step(model, optimizer, batch)))
        for name, parameter in model.named_parameters():
            assert parameter.grad.shape == parameter.shape, name
    print('losses', losses[0], losses[-1])
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < np.mean(losses[:5])


def test_native_step_only_for_the_default_shape(emphases):
    from emphases_b200 import training
    features = padded_batch()[0].cuda()
    for config in SWEEP:
        emphases.reset_configuration()
        model, _ = _model(emphases, **config)
        assert not training.native_step_supported(model, features), config
    emphases.reset_configuration()
    model, _ = _model(emphases)
    assert training.native_step_supported(model, features)


@pytest.mark.parametrize('config', [
    dict(CHANNELS=256), dict(ARCHITECTURE='transformer', CHANNELS=64)], ids=_name)
def test_unsupported_widths_raise(emphases, config):
    model, _ = _model(emphases, **config)
    features, frame_lengths, bounds, word_lengths, _ = padded_batch()
    with pytest.raises(NotImplementedError):
        model(features.cuda(), frame_lengths, bounds, word_lengths)
