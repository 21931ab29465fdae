"""Training-step parity: loss and every parameter gradient of the conv model
vs torch autograd through the CPU oracle (fp32)."""
import numpy as np
import pytest
import torch

from golden_util import state_from_golden
from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu


@pytest.fixture
def emphases():
    import emphases_b200
    emphases_b200.reset_configuration()
    yield emphases_b200
    emphases_b200.reset_configuration()


def padded_batch(seed=0, items=3):
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
    targets = torch.rand(items, 1, wmax, generator=generator)
    return (features, torch.tensor(lengths), bounds, torch.tensor(words), targets)


@pytest.mark.parametrize('method', ['sum', 'average', 'max', 'center'])
@pytest.mark.parametrize('loss_fn', ['bce', 'mse'])
def test_gradients_match_autograd(emphases, golden, method, loss_fn):
    emphases.configure(DOWNSAMPLE_METHOD=method, LOSS=loss_fn)
    data = golden('sweep')
    state = state_from_golden(data)
    model = emphases.Model()
    model.load_state_dict({k: v for k, v in state.items() if k in model.state_dict()})
    model = model.cuda().train()
    features, frame_lengths, bounds, word_lengths, targets = padded_batch()

    scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
    assert scores.requires_grad
    value = emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()

    reference = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    expected_scores = oracle.model_forward(
        reference, features, frame_lengths, bounds, word_lengths,
        {'DOWNSAMPLE_METHOD': method})
    expected = oracle.loss(expected_scores, targets, word_lengths, loss_fn)
    expected.backward()

    assert abs(value.item() - expected.item()) < 1e-5 * max(1, abs(expected.item()))
    np.testing.assert_allclose(
        scores.detach().cpu().numpy(), expected_scores.detach().numpy(),
        rtol=1e-5, atol=2e-5)
    for name, parameter in model.named_parameters():
        want = reference[name].grad
        got = parameter.grad.cpu()
        scale = want.abs().max().item() + 1e-12
        error = (got - want).abs().max().item()
        assert error < 2e-4 * scale + 1e-7, (name, error, scale)


@pytest.mark.parametrize('activation', ['GELU', 'LeakyReLU', 'SiLU'])
def test_gradients_other_activations(emphases, golden, activation):
    """The activations of the reference's hyper-parameter sweep in training:
    loss and every parameter gradient vs torch autograd through the oracle"""
    emphases.configure(ACTIVATION_FUNCTION=getattr(torch.nn, activation))
    data = golden('sweep')
    state = state_from_golden(data)
    model = emphases.Model()
    model.load_state_dict({k: v for k, v in state.items() if k in model.state_dict()})
    model = model.cuda().train()
    features, frame_lengths, bounds, word_lengths, targets = padded_batch()
    scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
    value = emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()

    reference = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    config = {'ACTIVATION': {
        'GELU': 'gelu', 'LeakyReLU': 'leaky_relu', 'SiLU': 'silu'}[activation]}
    expected_scores = oracle.model_forward(
        reference, features, frame_lengths, bounds, word_lengths, config)
    expected = oracle.loss(expected_scores, targets, word_lengths, 'bce')
    expected.backward()
    assert abs(value.item() - expected.item()) < 1e-5 * max(1, abs(expected.item()))
    for name, parameter in model.named_parameters():
        want = reference[name].grad
        got = parameter.grad.cpu()
        scale = want.abs().max().item() + 1e-12
        error = (got - want).abs().max().item()
        assert error < 2e-4 * scale + 1e-7, (name, error, scale)


@pytest.mark.parametrize('method', ['sum', 'average', 'max', 'center'])
def test_gradients_input_location(emphases, golden, method):
    """Training at DOWNSAMPLE_LOCATION='input' (every word segment is encoded
    on its own, reduction over the padded segment, model/core.py:41-87): loss
    and every parameter gradient vs torch autograd through the oracle"""
    emphases.configure(DOWNSAMPLE_LOCATION='input', DOWNSAMPLE_METHOD=method)
    data = golden('sweep')
    state = state_from_golden(data)
    model = emphases.Model()
    model.load_state_dict({k: v for k, v in state.items() if k in model.state_dict()})
    model = model.cuda().train()
    features, frame_lengths, bounds, word_lengths, targets = padded_batch()
    scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
    assert scores.requires_grad
    value = emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()

    reference = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    expected_scores = oracle.model_forward(
        reference, features, frame_lengths, bounds, word_lengths,
        {'DOWNSAMPLE_METHOD': method, 'DOWNSAMPLE_LOCATION': 'input'})
    expected = oracle.loss(expected_scores, targets, word_lengths, 'bce')
    expected.backward()
    assert abs(value.item() - expected.item()) < 1e-5 * max(1, abs(expected.item()))
    for name, parameter in model.named_parameters():
        want = reference[name].grad
        got = parameter.grad.cpu()
        scale = want.abs().max().item() + 1e-12
        error = (got - want).abs().max().item()
        assert error < 2e-4 * scale + 1e-7, (name, error, scale)


def test_train_step_reduces_loss(emphases, golden):
    data = golden('sweep')
    state = state_from_golden(data)
    model = emphases.Model()
    model.load_state_dict({k: v for k, v in state.items() if k in model.state_dict()})
    model = model.cuda()
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    batch = padded_batch(1)
    batch = (batch[0].cuda(),) + batch[1:4] + (batch[4].cuda(),)
    losses = [emphases.training.train_step(model, optimizer, batch).item()
              for _ in range(8)]
    assert losses[-1] < losses[0]


@pytest.mark.parametrize('method', ['linear', 'nearest'])
def test_upsample_and_frame_loss_golden(emphases, golden, method):
    """emphases.upsample and the frame-resolution loss vs the reference"""
    data = golden('upsample')
    emphases.configure(UPSAMPLE_METHOD=method, DOWNSAMPLE_LOCATION='inference')
    bounds = torch.from_numpy(data['bounds'])
    word_lengths = torch.from_numpy(data['word_lengths'])
    frame_lengths = torch.from_numpy(data['frame_lengths'])
    for name in ('xs', 'wide'):
        result = emphases.upsample(
            torch.from_numpy(data[name]).cuda(), bounds, word_lengths, frame_lengths)
        np.testing.assert_allclose(
            result.cpu().numpy(), data[f'{method}.{name}'], rtol=1e-6, atol=1e-6)
    for loss_fn in ('bce', 'mse'):
        value = emphases.loss(
            torch.from_numpy(data['scores']).cuda(), torch.from_numpy(data['xs']).cuda(),
            frame_lengths, bounds, word_lengths, training=True, loss_fn=loss_fn)
        np.testing.assert_allclose(
            value.item(), float(data[f'{method}.loss.{loss_fn}']), rtol=2e-6)


@pytest.mark.parametrize('location', ['loss', 'inference'])
def test_gradients_other_locations(emphases, golden, location):
    """Training step at the 'loss' (pool -> head) and 'inference' (frame-level
    head + upsampled targets) locations vs torch autograd through the oracle"""
    emphases.configure(DOWNSAMPLE_LOCATION=location)
    data = golden('sweep')
    state = state_from_golden(data)
    model = emphases.Model()
    own = model.state_dict()
    model.load_state_dict({k: v for k, v in state.items() if k in own})
    model = model.cuda().train()
    features, frame_lengths, bounds, word_lengths, targets = padded_batch(2)
    scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
    value = emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()
    reference = {
        k: v.clone().requires_grad_(True) for k, v in state.items() if k in own}
    config = {'DOWNSAMPLE_LOCATION': location}
    expected_scores = oracle.model_forward(
        reference, features, frame_lengths, bounds, word_lengths, config,
        training=True)
    if location == 'inference':
        expected = oracle.loss(
            expected_scores, targets, word_lengths, 'bce', frame_lengths, bounds,
            'linear')
    else:
        expected = oracle.loss(expected_scores, targets, word_lengths, 'bce')
    expected.backward()
    assert scores.shape == expected_scores.shape
    assert abs(value.item() - expected.item()) < 1e-5
    for name, parameter in model.named_parameters():
        want = reference[name].grad
        got = parameter.grad.cpu()
        scale = want.abs().max().item() + 1e-12
        assert (got - want).abs().max().item() < 2e-4 * scale + 1e-7, name


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3', 'bf16x6', 'bf16x3+bf16x6'])
def test_native_step_matches_per_kernel_path(emphases, golden, precision):
    """csrc/train_step.cu (one call per forward / backward) against the
    per-kernel Python orchestration it replaces: same logits and gradients
    (fp32: the same kernels in the same order; the tensor-core modes within
    their forward tolerance), gradients land in ONE flat buffer the .grad
    tensors alias, and a second backward without zero_grad accumulates"""
    from emphases_b200 import training
    state = state_from_golden(golden('sweep'))
    batch = padded_batch(seed=5)
    features, frame_lengths, bounds, word_lengths, targets = batch
    results = {}
    for name in ('native', 'kernels'):
        model = emphases.Model()
        model.load_state_dict({k: v for k, v in state.items() if k in model.state_dict()})
        model = model.cuda().train()
        if name == 'native':
            training.TRAIN_PRECISION = precision
            assert training.native_step_supported(model, features.cuda())
            scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
        else:
            scores = training._ConvModelFunction.apply(
                model, features.cuda(), bounds, word_lengths, *model.parameters())
        value = emphases.loss(
            scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
        value.backward()
        results[name] = (scores.detach(), {n: p.grad.clone() for n, p in model.named_parameters()})
        if name == 'native':
            native = model
    tolerance = {'fp32': 1e-6, 'bf16x3': 3e-5, 'bf16x6': 3e-6, 'bf16x3+bf16x6': 3e-5}[precision]
    # (bf16x3's 16-bit operands: 1e-5 class logits, but up to 2 % on the gradient
    # of the first layers after thirteen input-gradient convolutions -- which is
    # why the default is bf16x6)
    gradient_tolerance = {
        'fp32': 2e-5, 'bf16x3': 5e-2, 'bf16x6': 1e-4, 'bf16x3+bf16x6': 5e-2}[precision]
    assert (results['native'][0] - results['kernels'][0]).abs().max() < tolerance
    for name, want in results['kernels'][1].items():
        got = results['native'][1][name]
        scale = want.abs().max().item() + 1e-12
        assert (got - want).abs().max().item() < gradient_tolerance * scale + 1e-8, name
    # every .grad is a slice of the flat buffer ...
    flat_state = native._native_train_state
    assert all(flat_state.aliases_flat(p, i) for i, p in enumerate(flat_state.ordered))
    assert len(flat_state.ordered) == len(list(native.parameters()))
    # ... and a second backward accumulates into it
    scores = native(features.cuda(), frame_lengths, bounds, word_lengths)
    emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True).backward()
    training.TRAIN_PRECISION = 'bf16x6'
    for name, parameter in native.named_parameters():
        want = 2 * results['native'][1][name]
        scale = want.abs().max().item() + 1e-12
        # (float atomics in the weight-gradient kernel: sums agree to rounding)
        assert (parameter.grad - want).abs().max().item() < 1e-5 * scale + 1e-9, name
