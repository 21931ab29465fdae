"""Training gradients against fp64.

A. Each backward kernel of csrc/train.cu, called through the C ABI, against
   fp64 torch autograd of the same operation, at the shapes and values where
   such kernels go wrong: row counts around the tile and grid sizes of the
   weight-gradient kernels, adversarial word bounds, separators, head taps that
   reach them, saturated logits.
B. The whole training step at the shape tools/train_bench.py times (about 37
   items, 75,000 frames) against fp64 autograd through the oracle.
C. A small batch of edge cases (one-frame items, zero-length words, words that
   end past their item's length) through the native step and the per-kernel
   path, and the IndexError the reference raises.

The reference is the oracle run in float64.  Every tolerance is a value
measured on a B200 (1000 W power limit), with 4-10x headroom, and the
measured value is written beside it.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C = 80
METHODS = ['sum', 'average', 'max', 'center']


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
    error, bound = np.asarray(error, np.float64), np.asarray(bound, np.float64)
    return np.max(np.where(error > 0, error / np.maximum(bound, 1e-300), 0.))


def _cuda(array, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(array)).to(dtype).cuda()


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


###############################################################################
# The reference is sound
###############################################################################


def _edge_batch(empty_words=True, tmax=40):
    """8 items: lengths 1, 2, 7, 8 around the 7 frame layers and one of Tmax; a
    single-word item, a late first word, padded word slots, a zero-length word
    (empty_words; else a one-frame word), and words ending 1, 2 and 10 frames
    past their item's length"""
    lengths = [1, 2, 7, 8, tmax, 20, 15, 12]
    middle = [(5, 5), (5, 12)] if empty_words else [(5, 6), (6, 12)]
    words = [
        [(0, 1)],
        [(0, 1), (1, 2)],
        [(3, 5), (5, 7)],
        [(0, 3), (3, 8)],
        [(0, 5)] + middle + [(12, tmax)],
        [(0, 10), (10, 15), (15, 21)],
        [(0, 6), (6, 10), (10, 17)],
        [(0, 4), (4, 8), (8, 22)]]
    generator = torch.Generator().manual_seed(7)
    wmax = max(len(w) for w in words)
    features = torch.zeros(len(lengths), C, tmax)
    bounds = torch.zeros(len(lengths), 2, wmax, dtype=torch.long)
    for i, (t, item) in enumerate(zip(lengths, words)):
        features[i, :, :t] = torch.randn(C, t, generator=generator)
        bounds[i, :, :len(item)] = torch.tensor(item).T
    targets = torch.rand(len(lengths), 1, wmax, generator=generator)
    return (features, torch.tensor(lengths), bounds,
            torch.tensor([len(w) for w in words]), targets)


def _scaled_state(emphases, seed):
    """A fresh model's parameters, weights x1.4 so the ReLUs are not dead"""
    torch.manual_seed(seed)
    model = emphases.Model()
    for parameter in model.parameters():
        if parameter.dim() > 1:
            parameter.data.mul_(1.4)
    return model, {k: v.detach().clone() for k, v in model.state_dict().items()}


def _oracle_step(state, batch, config, dtype=torch.float64):
    """(loss, logits, {name: grad}) of fp64 (or `dtype`) autograd through the oracle"""
    features, frame_lengths, bounds, word_lengths, targets = batch
    params = {k: v.to(dtype).clone().requires_grad_(True) for k, v in state.items()}
    logits = oracle.model_forward(
        params, features.to(dtype), frame_lengths, bounds, word_lengths, config,
        training=True)
    if config.get('DOWNSAMPLE_LOCATION') == 'inference':
        value = oracle.loss(
            logits, targets.to(dtype), word_lengths, 'bce', frame_lengths, bounds, 'linear')
    else:
        value = oracle.loss(logits, targets.to(dtype), word_lengths, 'bce')
    value.backward()
    return (value.detach().double(), logits.detach().double(),
            {k: p.grad.double() for k, p in params.items()})


def test_fp32_oracle_agrees_with_fp64_oracle(emphases):
    """The fp64 reference is the same computation as the fp32 oracle the other
    training tests use: on a small batch they agree to rounding"""
    _, state = _scaled_state(emphases, 3)
    batch = _edge_batch()
    loss32, logits32, grads32 = _oracle_step(state, batch, {}, torch.float32)
    loss64, logits64, grads64 = _oracle_step(state, batch, {})
    assert abs(loss32 - loss64) <= 1e-6 * abs(loss64)
    # measured: 1.3e-8
    _within('fp32 oracle logits', (logits32 - logits64).abs().max().item(), 1e-7)
    for name, want in grads64.items():
        error = (grads32[name] - want).abs().max().item() / want.abs().max().item()
        # measured: 9.0e-7 worst over the parameters (the oracle runs on the CPU)
        _within(f'fp32 oracle grad {name}', error, 5e-6)


###############################################################################
# A. Backward kernels against fp64 autograd of the same operation
###############################################################################

SPECIAL = [0., 1e-3, -1e-3, 3., -3., 20., -20., 100., -100.]
_ACTIVATIONS64 = {
    0: lambda x: x,
    1: torch.relu,
    2: lambda x: F.gelu(x),                       # exact erf GELU
    3: lambda x: F.leaky_relu(x, 0.01),
    4: F.silu}


@pytest.mark.parametrize('act', [0, 1, 2, 3, 4])
def test_activation_forward_backward(lib, act):
    rng = np.random.default_rng(act)
    total = 997
    seq = _ragged_row_seq(total, rng, first=1)
    pre = rng.standard_normal((total, C)) * 5.
    pre[:, :len(SPECIAL)] = SPECIAL
    pre = pre.astype(np.float32)
    real = seq >= 0
    pre_dev, seq_dev = _cuda(pre), _cuda(seq, torch.int32)
    y = torch.full_like(pre_dev, 7.)
    lib.call('emph_activation_forward', lib.ptr(pre_dev), lib.ptr(seq_dev), total, C, act,
             lib.ptr(y), lib.stream_ptr())
    pre64 = torch.from_numpy(pre).double().requires_grad_(True)
    want = _ACTIVATIONS64[act](pre64)
    y_host = y.cpu().double()
    assert (y_host[~real] == 0).all()
    scale = 1. + pre64.detach().abs()
    # measured: 0 (none, relu), 7.4e-10 (leaky), 9.1e-8 (gelu), 1.05e-7 (silu) x (1 + |x|)
    _within(f'activation {act} forward', _ratio(
        (y_host - want.detach())[real].abs(), scale[real] * 1e-6), 1.)

    dy = rng.standard_normal((total, C)).astype(np.float32)
    dy_dev = _cuda(dy)
    # GELU / SiLU take the pre-activation, the others the layer output
    key = pre_dev if act in (lib.ACT_GELU, lib.ACT_SILU) else y
    dpre = torch.full_like(pre_dev, 7.)
    lib.call('emph_activation_backward', lib.ptr(dy_dev), lib.ptr(key), lib.ptr(seq_dev),
             total, C, act, lib.ptr(dpre), lib.stream_ptr())
    (want_grad,) = torch.autograd.grad(want, pre64, torch.from_numpy(dy).double())
    dpre_host = dpre.cpu().double()
    assert (dpre_host[~real] == 0).all()
    # measured: 0 (none, relu), 8.0e-10 (leaky), 8.6e-8 (gelu), 1.04e-7 (silu) x |dy| (1 + |x|)
    bound = torch.from_numpy(np.abs(dy)).double() * scale * 1e-6
    _within(f'activation {act} backward', _ratio(
        (dpre_host - want_grad)[real].abs(), bound[real]), 1.)


def _shifted(x, tap):
    """rows r + tap - 1 of x (zero outside), the operand of tap `tap`"""
    out = torch.zeros_like(x)
    if tap == 0:
        out[1:] = x[:-1]
    elif tap == 1:
        out[:] = x
    else:
        out[:-1] = x[1:]
    return out


@pytest.mark.parametrize('total', [1, 63, 64, 65, 9473, 40000])
def test_conv_weight_grad_ffma(lib, total):
    """emph_conv_weight_grad (the per-kernel path's fp32 FFMA kernel): 40,000
    rows make the grid of 296 CTAs x 64 rows loop"""
    rng = np.random.default_rng(total)
    seq = _ragged_row_seq(total, rng)
    x = rng.standard_normal((total, C)).astype(np.float32)
    d = rng.standard_normal((total, C)).astype(np.float32)
    x[seq < 0] = 0.
    d[seq < 0] = 0.
    dw = torch.full((3, C, C), 7., device='cuda')
    db = torch.full((C,), 7., device='cuda')
    x_dev, d_dev = _cuda(x), _cuda(d)
    lib.call('emph_conv_weight_grad', lib.ptr(x_dev), lib.ptr(d_dev), total, C, 3,
             lib.ptr(dw), lib.ptr(db), lib.stream_ptr())
    X, D = torch.from_numpy(x).double(), torch.from_numpy(d).double()
    got = dw.cpu().double()
    for tap in range(3):
        shifted = _shifted(X, tap)
        want = shifted.T @ D
        bound = shifted.abs().T @ D.abs()
        # measured: 2.6e-7 x (|X|^T |dPre|), worst over the taps and row counts
        _within(f'ffma dW tap {tap} / (|X|^T|dPre|)', _ratio((got[tap] - want).abs(), bound), 2e-6)
    # measured: 7.7e-8 x sum |dPre|
    _within('ffma db / sum|dPre|', _ratio(
        (db.cpu().double() - D.sum(0)).abs(), D.abs().sum(0)), 5e-7)


def _tiled_bounds(lengths, words, rng):
    """Word bounds that tile [0, length) of every item"""
    bounds = torch.zeros(len(lengths), 2, max(words), dtype=torch.long)
    for i, (t, w) in enumerate(zip(lengths, words)):
        cuts = np.sort(rng.choice(np.arange(1, t), size=w - 1, replace=False))
        edges = np.concatenate([[0], cuts, [t]])
        bounds[i, 0, :w] = torch.from_numpy(edges[:-1])
        bounds[i, 1, :w] = torch.from_numpy(edges[1:])
    return bounds


@pytest.mark.parametrize('items,frames', [(2, 300), (4, 2384), (37, 2026)])
def test_tensor_core_weight_grad(emphases, items, frames):
    """The split-bf16 mma.sync weight gradient of the native step, through a
    one-layer model (input layer, no activation) at the 'loss' location, where
    dW = sum feat x dPre.  Packed rows 1 + items * (frames + 1): 603 (one tile
    per CTA), 9,541 (150 tiles, the last one ragged: two tiles per CTA) and
    75,000 (the benchmarked batch: eight tiles per CTA)."""
    from emphases_b200 import training
    emphases.configure(LAYERS=0, DOWNSAMPLE_LOCATION='loss', DOWNSAMPLE_METHOD='sum')
    config = {'LAYERS': 0, 'DOWNSAMPLE_LOCATION': 'loss', 'DOWNSAMPLE_METHOD': 'sum'}
    rng = np.random.default_rng(items)
    torch.manual_seed(items)
    model = emphases.Model()
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().train()
    lengths = torch.full((items,), frames, dtype=torch.long)
    words = [int(rng.integers(frames // 60, frames // 30)) for _ in range(items)]
    words[0] = max(words)
    bounds = _tiled_bounds([frames] * items, words, rng)
    features = torch.randn(items, C, frames)
    assert training.native_step_supported(model, features.cuda())
    scores = model(features.cuda(), lengths, bounds, torch.tensor(words))
    grad = torch.randn(scores.shape)
    scores.backward(grad.cuda())

    params = {k: v.double().requires_grad_(True) for k, v in state.items()}
    features64 = features.double()
    logits, inter = oracle.model_forward(
        params, features64, lengths, bounds, torch.tensor(words), config,
        return_intermediates=True)
    pre = inter['frame_embeddings']             # the input layer's output
    pre.retain_grad()
    logits.backward(grad.double())
    weight = params['input_layer.weight']
    bound = torch.nn.grad.conv1d_weight(
        features64.abs(), weight.shape, pre.grad.abs(), padding=1)
    got = model.input_layer.weight.grad.cpu().double()
    # split bf16 (16-bit operands): measured 1.2e-6 x (|X|^T |dPre|); a lost
    # lo*hi or hi*lo term is 2^-8 class
    _within('tensor-core dW / (|X|^T|dPre|)', _ratio((got - weight.grad).abs(), bound), 1e-5)
    # measured: 1.4e-7 x sum |dPre|
    got_bias = model.input_layer.bias.grad.cpu().double()
    _within('tensor-core db / sum|dPre|', _ratio(
        (got_bias - params['input_layer.bias'].grad).abs(), pre.grad.abs().sum((0, 2))), 1e-6)


def _pool_case(data, method):
    """Packed rows of the golden pool inputs; every item's words are followed
    by its padded (-1, -1) slots and one masked (-2, -2) slot"""
    from emphases_b200 import engine
    xs = data['xs']                                          # (2, 80, 50)
    bounds, lengths = data['bounds'], data['lengths']
    batch, _, frames = xs.shape
    wmax = bounds.shape[2]
    slots = wmax + 1
    row_start, total = engine.packed_starts([frames] * batch, 1)
    word_start, total_words = engine.packed_starts([slots] * batch, 1)
    rows = np.zeros((total, C), dtype=np.float32)
    word_seq = np.full(total_words, -1, dtype=np.int32)
    word_lo = np.zeros(total_words, dtype=np.int32)
    word_hi = np.zeros(total_words, dtype=np.int32)
    for b in range(batch):
        rows[row_start[b]:row_start[b] + frames] = xs[b].T
        s = word_start[b]
        word_seq[s:s + slots] = b
        word_lo[s:s + wmax], word_hi[s:s + wmax] = bounds[b, 0], bounds[b, 1]
        word_lo[s + lengths[b]:s + wmax] = -1                # padded slots
        word_hi[s + lengths[b]:s + wmax] = -1
        word_lo[s + wmax] = word_hi[s + wmax] = -2           # masked slot
    return (xs, bounds, lengths, rows, row_start.astype(np.int32),
            np.full(batch, frames, dtype=np.int32), word_start, word_seq, word_lo,
            word_hi, total)


def _pool_backward(lib, rows, row_start, n_rows, word_seq, word_lo, word_hi, dy, method):
    dx = torch.full((rows.shape[0], C), 7., device='cuda')
    tensors = [_cuda(rows), _cuda(row_start, torch.int32), _cuda(n_rows, torch.int32),
               _cuda(word_seq, torch.int32), _cuda(word_lo, torch.int32),
               _cuda(word_hi, torch.int32), _cuda(dy)]
    x_dev, start_dev, n_dev, seq_dev, lo_dev, hi_dev, dy_dev = tensors
    lib.call('emph_pool_words_backward', lib.ptr(dy_dev), lib.ptr(x_dev), C,
             lib.ptr(start_dev), lib.ptr(n_dev), lib.ptr(seq_dev), lib.ptr(lo_dev),
             lib.ptr(hi_dev), len(word_seq), lib.POOL[method], rows.shape[0], lib.ptr(dx),
             lib.stream_ptr())
    return dx.cpu().double().numpy()


@pytest.mark.parametrize('method', METHODS)
def test_pool_words_backward(lib, golden, method):
    """Adjoint of word pooling on the adversarial bounds of the pool golden set
    (zero-length and one-frame words, bounds past T, a late first word) plus
    padded and masked slots, against fp64 autograd of oracle.downsample.  The
    words the reference rejects (NaN for `average`, IndexError for `max` and
    `center`) take no part; the kernel must leave them out as well."""
    data = golden('pool')
    (xs, bounds, lengths, rows, row_start, n_rows, word_start, word_seq, word_lo,
     word_hi, total) = _pool_case(data, method)
    batch, _, frames = xs.shape
    wmax = bounds.shape[2]
    rng = np.random.default_rng(1)
    dy = rng.standard_normal((len(word_seq), C)).astype(np.float32)
    dx = _pool_backward(lib, rows, row_start, n_rows, word_seq, word_lo, word_hi, dy, method)

    reference_bounds = torch.from_numpy(bounds.copy())
    dy_words = torch.zeros(batch, C, wmax, dtype=torch.float64)
    for b in range(batch):
        for j in range(wmax):
            lo, hi = int(bounds[b, 0, j]), int(bounds[b, 1, j])
            if j >= lengths[b]:
                reference_bounds[b, :, j] = 0        # padded: `center` reads frame 0
            elif method in ('average', 'max') and min(hi, frames) <= min(lo, frames):
                reference_bounds[b, :, j] = torch.tensor([0, 1])
                continue                             # rejected by the reference
            elif method == 'center' and (lo + hi) // 2 >= frames:
                reference_bounds[b, :, j] = 0
                continue
            dy_words[b, :, j] = torch.from_numpy(dy[word_start[b] + j]).double()
    x64 = torch.from_numpy(xs).double().requires_grad_(True)
    pooled = oracle.downsample(x64, reference_bounds, torch.from_numpy(lengths), method)
    (want,) = torch.autograd.grad(pooled, x64, dy_words[:, :, :pooled.shape[2]])
    got = np.stack([dx[row_start[b]:row_start[b] + frames].T for b in range(batch)])
    separators = np.ones(total, dtype=bool)
    for b in range(batch):
        separators[row_start[b]:row_start[b] + frames] = False
    assert (dx[separators] == 0).all()
    want = want.numpy()
    # rows no word reads (and, for max, every frame but the argmax) get exactly 0
    assert (got[want == 0] == 0).all()
    # measured: 1.6e-7 x max|dy| (a few fp32 adds per frame)
    _within(f'pool backward {method}', np.abs(got - want).max() / np.abs(dy).max(), 1e-6)


def test_pool_max_backward_ties_go_to_the_first_frame(lib):
    """Equal values in a word: `max` routes the whole gradient to its first
    frame, the index torch.max reports"""
    frames, lo, hi = 12, 3, 9
    rows = np.zeros((frames + 2, C), dtype=np.float32)
    rows[1:frames + 1] = 1.
    rows[1 + 5, :C // 2] = 2.                  # a unique maximum in half the channels
    rows[1 + 7, :C // 2] = 2.                  # ... tied with a later frame
    word_seq = np.array([-1, 0, -1], dtype=np.int32)
    word_lo = np.array([0, lo, 0], dtype=np.int32)
    word_hi = np.array([0, hi, 0], dtype=np.int32)
    dy = np.zeros((3, C), dtype=np.float32)
    dy[1] = np.arange(1, C + 1)
    dx = _pool_backward(
        lib, rows, np.array([1], np.int32), np.array([frames], np.int32), word_seq,
        word_lo, word_hi, dy, 'max')
    want = np.zeros_like(dx)
    want[1 + 5, :C // 2] = dy[1, :C // 2]
    want[1 + lo, C // 2:] = dy[1, C // 2:]
    np.testing.assert_array_equal(dx, want)
    x = torch.from_numpy(rows[1:frames + 1, :].T.copy())
    assert (x[:, lo:hi].max(dim=1).indices == torch.tensor(
        [5 - lo] * (C // 2) + [0] * (C // 2))).all()


@pytest.mark.parametrize('kernel', [1, 3, 5, 7])
def test_output_head_backward(lib, kernel):
    """dx, dw, db of the output projection (Conv1d C -> 1, asymmetric taps)
    against fp64 autograd per sequence; one- and two-row sequences make the
    taps reach the (kernel - 1) / 2 separator rows on both sides"""
    from emphases_b200 import engine
    half = (kernel - 1) // 2
    lengths = [1, 2, 5, 1, 37, 2, 300, 1]
    starts, total = engine.packed_starts(lengths, max(1, half))
    rng = np.random.default_rng(kernel)
    seq = np.full(total, -1, dtype=np.int32)
    for u, (s, n) in enumerate(zip(starts, lengths)):
        seq[s:s + n] = u
    x = rng.standard_normal((total, C)).astype(np.float32)
    x[seq < 0] = 0.                              # activations are zero on separators
    dz = rng.standard_normal(total).astype(np.float32)   # separators: ignored
    weight = (rng.standard_normal((1, C, kernel)) *
              np.arange(1, kernel + 1)).astype(np.float32)    # taps differ
    packed = _cuda(weight[0].T)                  # [k][C]
    dx = torch.full((total, C), 7., device='cuda')
    dw = torch.full((kernel, C), 7., device='cuda')
    db = torch.full((1,), 7., device='cuda')
    x_dev, dz_dev, seq_dev = _cuda(x), _cuda(dz), _cuda(seq, torch.int32)
    lib.call('emph_output_head_backward', lib.ptr(x_dev), lib.ptr(dz_dev), lib.ptr(seq_dev),
             total, C, kernel, lib.ptr(packed), lib.ptr(dx), lib.ptr(dw), lib.ptr(db),
             lib.stream_ptr())

    def reference(x, weight, dz):
        """fp64 autograd per sequence: (dx rows, dW (1, C, k), db)"""
        w64 = torch.from_numpy(weight).double().requires_grad_(True)
        b64 = torch.zeros(1, dtype=torch.float64, requires_grad=True)
        dx64 = np.zeros((total, C))
        for s, n in zip(starts, lengths):
            xs = torch.from_numpy(x[s:s + n].T.copy()).double()[None].requires_grad_(True)
            z = F.conv1d(xs, w64, b64, padding=half)
            gx, = torch.autograd.grad(z, xs, torch.from_numpy(dz[s:s + n]).double()[None, None],
                                      retain_graph=True)
            z.backward(torch.from_numpy(dz[s:s + n]).double()[None, None])
            dx64[s:s + n] = gx[0].T.numpy()
        return dx64, w64.grad.numpy(), b64.grad.numpy()

    want_dx, want_dw, want_db = reference(x, weight, dz)
    bound_dx, bound_dw, bound_db = reference(np.abs(x), np.abs(weight), np.abs(dz))
    got_dx = dx.cpu().double().numpy()
    assert (got_dx[seq < 0] == 0).all()
    # measured: 1.5e-7 (dx), 5.0e-8 (dw), 1.6e-8 (db), relative to the sums of |terms|
    _within(f'head {kernel} dx', _ratio(np.abs(got_dx - want_dx), bound_dx), 1e-6)
    got_dw = dw.cpu().double().numpy().T[None]   # [k][C] -> (1, C, k)
    _within(f'head {kernel} dw', _ratio(np.abs(got_dw - want_dw), bound_dw), 5e-7)
    _within(f'head {kernel} db', _ratio(np.abs(db.cpu().double().numpy() - want_db), bound_db), 1e-7)


LOGITS = [-100., -30., -17., 0., 17., 30., 100.]
TARGETS = [0., 0.3, 1.]


@pytest.mark.parametrize('case', ['grid', 'single', 'frames'])
@pytest.mark.parametrize('mode', [0, 1])
def test_masked_loss(lib, mode, case):
    """Mean BCE-with-logits / squared error over the valid rows and its
    gradient: saturated logits, a mask with one valid row, and 75,000 rows
    (the frame loss of the 'inference' location at the benchmarked batch)"""
    rng = np.random.default_rng(mode)
    grid = np.array([(z, t) for z in LOGITS for t in TARGETS])
    if case == 'frames':
        rows = 75000
        logits = rng.standard_normal(rows) * 4.
        targets = rng.random(rows)
        logits[:len(grid)], targets[:len(grid)] = grid[:, 0], grid[:, 1]
        valid = rng.random(rows) < 0.9
        valid[:len(grid)] = True
    else:
        logits = np.concatenate([grid[:, 0], [3., -2.]])
        targets = np.concatenate([grid[:, 1], [0.5, 0.5]])
        valid = np.ones(len(logits), dtype=bool)
        valid[-2:] = False
        if case == 'single':
            valid[:] = False
            valid[LOGITS.index(100.) * len(TARGETS)] = True    # z = 100, t = 0
    logits, targets = logits.astype(np.float32), targets.astype(np.float32)
    z_dev, t_dev = _cuda(logits), _cuda(targets)
    valid_dev = _cuda(valid, torch.uint8)
    loss = torch.full((1,), 7., device='cuda')
    grad = torch.full_like(z_dev, 7.)
    lib.call('emph_masked_loss', lib.ptr(z_dev), lib.ptr(t_dev), lib.ptr(valid_dev), len(logits),
             mode, lib.ptr(loss), lib.ptr(grad), lib.stream_ptr())
    z64 = torch.from_numpy(logits).double().requires_grad_(True)
    t64 = torch.from_numpy(targets).double()
    mask = torch.from_numpy(valid)
    if mode == 0:
        want = F.binary_cross_entropy_with_logits(z64[mask], t64[mask])
    else:
        want = F.mse_loss(z64[mask], t64[mask])
    want.backward()
    got_loss, got_grad = loss.item(), grad.cpu().double()
    assert np.isfinite(got_loss) and torch.isfinite(got_grad).all()
    # measured: 8.2e-8 relative
    _within(f'loss mode {mode} {case}', abs(got_loss - want.item()) / abs(want.item()), 5e-7)
    count = int(valid.sum())
    # BCE: sigmoid(z) - t to fp32 rounding of 1 / count; MSE: 2 (z - t) / count,
    # relative.  measured: 1.4e-7
    bound = 1. / count if mode == 0 else z64.grad.abs().numpy()
    _within(f'loss grad mode {mode} {case}', _ratio(
        (got_grad - z64.grad).abs().numpy(), bound), 1e-6)
    assert (got_grad[~mask] == 0).all()


###############################################################################
# B. The whole step at the benchmarked shape
###############################################################################


def _bench_batch():
    """synthetic_batch() of tools/train_bench.py, the batch it times"""
    spec = importlib.util.spec_from_file_location(
        'train_bench', os.path.join(ROOT, 'tools', 'train_bench.py'))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module.synthetic_batch(100)


_reference = {}     # (batch, config) -> fp64 (loss, logits, grads), shared by the paths


def _step_errors(emphases, name, batch, state, config):
    """Run one training step on the device; its errors against fp64 (the
    reference of batch `name` is computed once per configuration)"""
    features, frame_lengths, bounds, word_lengths, targets = batch
    model = emphases.Model()
    model.load_state_dict(state)
    model = model.cuda().train()
    scores = model(features.cuda(), frame_lengths, bounds, word_lengths)
    value = emphases.loss(
        scores, targets.cuda(), frame_lengths, bounds, word_lengths, training=True)
    value.backward()
    key = (name, tuple(sorted(config.items())))
    if key not in _reference:
        _reference[key] = _oracle_step(state, batch, config)
    loss64, logits64, grads64 = _reference[key]
    errors = {
        'loss': abs(value.item() - loss64.item()) / abs(loss64.item()),
        'logits': (scores.detach().cpu().double() - logits64).abs().max().item() /
        logits64.abs().max().item()}
    for name, parameter in model.named_parameters():
        got, want = parameter.grad.cpu().double(), grads64[name]
        errors[f'{name} frobenius'] = ((got - want).norm() / want.norm()).item()
        errors[f'{name} max'] = ((got - want).abs().max() / want.abs().max()).item()
    return errors


def _check(errors, loss, logits, frobenius, worst, what):
    for name, error in errors.items():
        bound = {'loss': loss, 'logits': logits}.get(
            name, frobenius if name.endswith('frobenius') else worst)
        _within(f'{what} {name}', error, bound)


# (loss, logits, per-parameter Frobenius and max relative errors) at the
# benchmarked shape.  The gradients of the first frame layers there are
# ill-conditioned in fp32 (long sums with cancellation over 75,000 frames):
# the fp32 oracle itself, on the CPU, is 7.0e-4 (Frobenius) and 8.5e-4 (max)
# away from fp64 on input_layer.weight with `sum` pooling, so the bounds are
# fp32's reach there, not the 2e-4 of a 600-frame batch.
STEP_TOLERANCE = {
    # measured: 1.9e-7, 9.9e-7, 6.2e-4 (`average`, frame_encoder.0), 9.9e-4
    'bf16x6': (1e-6, 5e-6, 3e-3, 5e-3),
    # measured: 7.8e-8, 5.1e-7, 3.7e-4, 4.2e-4
    'fp32': (1e-6, 5e-6, 2e-3, 3e-3),
    # 16-bit operands in the forward: measured 7.8e-8, 1.2e-5, 5.0e-3, 6.5e-3
    'bf16x3+bf16x6': (1e-6, 1e-4, 3e-2, 5e-2),
    # the per-kernel path, fp32 FFMA throughout: measured 7.8e-8, 5.1e-7,
    # 6.8e-4, 9.0e-4 (the frame loss of the 'inference' location)
    'kernels': (1e-6, 5e-6, 3e-3, 5e-3)}
# the same on the 8-item edge batch, where nothing is ill-conditioned
EDGE_TOLERANCE = {
    # measured: 1.1e-7, 4.1e-7, 1.3e-5, 2.3e-5
    'native': (1e-6, 3e-6, 1e-4, 2e-4),
    # measured: 1.1e-7, 4.3e-7, 1.2e-6, 1.3e-6
    'kernels': (1e-6, 3e-6, 1e-5, 1e-5)}


@pytest.mark.parametrize('method,location,precision', [
    ('sum', 'intermediate', 'bf16x6'),
    ('average', 'intermediate', 'bf16x6'),
    ('max', 'intermediate', 'bf16x6'),
    ('center', 'intermediate', 'bf16x6'),
    ('sum', 'intermediate', 'fp32'),
    ('sum', 'intermediate', 'bf16x3+bf16x6'),
    ('sum', 'loss', 'bf16x6')])
def test_native_step_at_benchmark_shape(emphases, monkeypatch, method, location, precision):
    from emphases_b200 import training
    monkeypatch.setattr(training, 'TRAIN_PRECISION', precision)
    emphases.configure(DOWNSAMPLE_METHOD=method, DOWNSAMPLE_LOCATION=location)
    model, state = _scaled_state(emphases, 0)
    batch = _bench_batch()
    assert training.native_step_supported(model.cuda(), batch[0].cuda())
    config = {'DOWNSAMPLE_METHOD': method, 'DOWNSAMPLE_LOCATION': location}
    errors = _step_errors(emphases, 'bench', batch, state, config)
    _check(errors, *STEP_TOLERANCE[precision], f'native {precision} {method} {location}')


@pytest.mark.parametrize('location', ['intermediate', 'inference'])
def test_per_kernel_step_at_benchmark_shape(emphases, monkeypatch, location):
    """EMPHASES_B200_TRAIN_NATIVE=0 (and the 'inference' location, which the
    native step does not cover): the FFMA emph_conv_weight_grad over 75,000
    rows, and at 'inference' the frame-level loss over every frame"""
    from emphases_b200 import training
    monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    emphases.configure(DOWNSAMPLE_LOCATION=location)
    model, state = _scaled_state(emphases, 0)
    batch = _bench_batch()
    assert not training.native_step_supported(model.cuda(), batch[0].cuda())
    config = {'DOWNSAMPLE_LOCATION': location}
    errors = _step_errors(emphases, 'bench', batch, state, config)
    _check(errors, *STEP_TOLERANCE['kernels'], f'per-kernel {location}')


###############################################################################
# C. Edge cases through both paths
###############################################################################


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('path', ['native', 'kernels'])
@pytest.mark.parametrize('location,head_kernel', [('intermediate', 3), ('loss', 7)])
def test_edge_batch(emphases, monkeypatch, method, path, location, head_kernel):
    """One-frame items, a late first word, padded slots, zero-length words
    (`sum`, `center`) and words ending 1, 2 and 10 frames past their item's
    length, which the reference pools over the padded columns.  At 'loss' a
    head of kernel 7 reaches three word rows beyond each item's last word."""
    from emphases_b200 import training
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    emphases.configure(
        DOWNSAMPLE_METHOD=method, DOWNSAMPLE_LOCATION=location,
        DECODER_KERNEL_SIZE=head_kernel)
    model, state = _scaled_state(emphases, 4)
    batch = _edge_batch(empty_words=method in ('sum', 'center'))
    assert training.native_step_supported(model.cuda(), batch[0].cuda()) == (path == 'native')
    config = {'DOWNSAMPLE_METHOD': method, 'DOWNSAMPLE_LOCATION': location,
              'DECODER_KERNEL_SIZE': head_kernel}
    errors = _step_errors(emphases, f'edge {method}', batch, state, config)
    _check(errors, *EDGE_TOLERANCE[path],
           f'edge {path} {method} {location}')


@pytest.mark.parametrize('path', ['native', 'kernels'])
@pytest.mark.parametrize('method', ['max', 'center'])
def test_training_forward_raises_where_reference_raises(emphases, monkeypatch, path, method):
    """`max` over a zero-length word, a `center` index >= T"""
    if path == 'kernels':
        monkeypatch.setenv('EMPHASES_B200_TRAIN_NATIVE', '0')
    emphases.configure(DOWNSAMPLE_METHOD=method)
    model, state = _scaled_state(emphases, 5)
    features, frame_lengths, bounds, word_lengths, targets = _edge_batch(
        empty_words=method == 'max')
    if method == 'center':
        bounds[4, :, 3] = torch.tensor([30, 50])     # center 40 == T
    with pytest.raises(IndexError):
        oracle.model_forward(
            state, features, frame_lengths, bounds, word_lengths,
            {'DOWNSAMPLE_METHOD': method}, training=True)
    model = model.cuda().train()
    with pytest.raises(IndexError):
        model(features.cuda(), frame_lengths, bounds, word_lengths)
