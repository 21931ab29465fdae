"""The tensor-core conv stack runs on CTA pairs: pair tile p is tiles 2p and
2p + 1, and a persistent grid of pairs walks the tiles in rounds of
2 x clusters x slots.  These tests put the tile count at the edges of that
walk -- one tile (a pair with an empty second half), two, three, one below and
one above a full round, several rounds with an odd last pair -- with rows that
end inside the last tile, in every precision, at kernel sizes 3 and 1, and
with every fused pooling mode."""
import numpy as np
import pytest
import torch

from golden_util import state_from_golden
from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

SLOTS = {'bf16': 4, 'bf16x3': 2, 'bf16x6': 2}


@pytest.fixture(scope='module')
def eng():
    from emphases_b200 import engine
    return engine.Engine('cuda:0')


def _precision(mode):
    from emphases_b200 import _lib
    return {'bf16': _lib.PREC_BF16_TC, 'bf16x3': _lib.PREC_BF16X3_TC,
            'bf16x6': _lib.PREC_BF16X6_TC}[mode]


def _tiles_per_round(mode):
    # one CTA per SM, two SMs per pair, each CTA one tile per slot
    return torch.cuda.get_device_properties(0).multi_processor_count * SLOTS[mode]


def _tile_counts(mode):
    per_round = _tiles_per_round(mode)
    return [1, 2, 3, per_round - 1, per_round + 1, 3 * per_round + 1]


def _lengths(total, seed):
    """ragged sequence lengths whose packed layout is exactly `total` rows"""
    from emphases_b200 import engine
    gap = engine.separator_rows()
    rng = np.random.default_rng(seed)
    lengths, used = [], gap
    while total - used > 700 + gap:
        n = int(rng.integers(1, 700))
        lengths.append(n)
        used += n + gap
    lengths.append(total - used - gap)
    assert lengths[-1] >= 1
    assert engine.packed_starts(lengths)[1] == total
    return lengths


def _rows(eng, lengths, seed):
    from emphases_b200 import engine
    starts, total = engine.packed_starts(lengths)
    row_seq = eng.row_index(
        torch.tensor(starts, dtype=torch.int32, device='cuda:0'),
        torch.tensor(lengths, dtype=torch.int32, device='cuda:0'), len(lengths), total)
    generator = torch.Generator().manual_seed(seed)
    x = torch.randn(total, 80, generator=generator)
    x[(row_seq < 0).cpu()] = 0
    return row_seq, x


def _reference(stack, x, row_seq, quantize):
    """fp64 stack over the whole packed buffer, separator rows zeroed after
    every layer (= each sequence convolved on its own with zero padding);
    `quantize` rounds every operand to bf16 like the one-part kernel"""
    keep = (row_seq >= 0).cpu().double()[None, :, None]
    kernel = stack.kernel_size
    h = x.double()[None]
    for layer in range(stack.n_layers):
        weight = stack.weights[layer].cpu().double()          # [K][in][out]
        bias = stack.bias[layer].cpu().double()
        if quantize:
            h = h.to(torch.bfloat16).double()
            weight = weight.to(torch.bfloat16).double()
        conv = torch.nn.functional.conv1d(
            h.transpose(1, 2), weight.permute(2, 1, 0), bias, padding=(kernel - 1) // 2)
        h = conv.transpose(1, 2)
        if int(stack.acts[layer]) == 1:
            h = torch.relu(h)
        h = (h * keep).float().double()
    return h[0].float()


def _frame_stack(golden):
    from emphases_b200 import engine
    state = state_from_golden(golden('c1'))
    return engine.pack_weights(
        state, torch.device('cuda:0'), layers=6, activation='ReLU',
        dropout=None, has_decoder=True).frame


def _linear_stack():
    """a k = 1 stack (the per-row maps of the Transformer variant's path)"""
    from emphases_b200 import _lib, engine
    generator = torch.Generator().manual_seed(11)
    weights = torch.randn(3, 1, 80, 80, generator=generator) / 9
    bias = torch.randn(3, 80, generator=generator) / 10
    acts = np.asarray([_lib.ACT_RELU, _lib.ACT_RELU, _lib.ACT_NONE], dtype=np.int32)
    return engine.ConvStack(weights.cuda(), bias.cuda(), acts, 1, 80)


def _check(y, expected, row_seq, mode):
    scale = max(expected.abs().max().item(), 1.0)
    error = (y - expected).abs().max().item()
    # bf16: against the bf16-emulating reference (one rounding flip of an
    # intermediate ~3e-4); the split modes: against fp64 with the bars of the
    # single-launch tests
    bar = {'bf16': 2e-3, 'bf16x3': 5e-5, 'bf16x6': 2e-6}[mode]
    assert error < bar * scale, (error, scale)
    assert y[(row_seq < 0).cpu()].abs().max().item() == 0


@pytest.mark.parametrize('mode', ['bf16', 'bf16x3', 'bf16x6'])
def test_pair_tile_counts_k3(eng, golden, mode):
    """The 7-layer frame stack (114-row tiles) at every edge tile count"""
    stack = _frame_stack(golden)
    tile_rows = 128 - 2 * stack.n_layers
    for index, n_tiles in enumerate(_tile_counts(mode)):
        total = (n_tiles - 1) * tile_rows + 37           # rows end inside the last tile
        row_seq, x = _rows(eng, _lengths(total, index), index)
        y = eng.conv_stack(x.cuda(), row_seq, stack, _precision(mode)).cpu()
        _check(y, _reference(stack, x, row_seq, mode == 'bf16'), row_seq, mode)
        if n_tiles > 3:
            again = eng.conv_stack(x.cuda(), row_seq, stack, _precision(mode)).cpu()
            assert torch.equal(again, y)


@pytest.mark.parametrize('mode', ['bf16', 'bf16x3', 'bf16x6'])
def test_pair_tile_counts_k1(eng, mode):
    """A kernel-size-1 stack (128-row tiles, no halo) at every edge tile count"""
    stack = _linear_stack()
    for index, n_tiles in enumerate(_tile_counts(mode)):
        total = (n_tiles - 1) * 128 + 91
        row_seq, x = _rows(eng, _lengths(total, 100 + index), 100 + index)
        y = eng.conv_stack(x.cuda(), row_seq, stack, _precision(mode)).cpu()
        _check(y, _reference(stack, x, row_seq, mode == 'bf16'), row_seq, mode)


def _corpus(eng, seeds, durations=None):
    from emphases_b200 import engine
    utterances = []
    for index, seed in enumerate(seeds):
        duration = None if durations is None else durations[index]
        times, audio = oracle.synthetic_utterance(seed, duration)
        utterances.append((np.asarray(times), audio.shape[-1]))
    plan = engine.make_plan(utterances)
    views = eng.upload_plan(plan)
    row_seq = eng.row_index(views['row_start'], views['n_rows'], plan.n_seq, plan.total_rows)
    generator = torch.Generator().manual_seed(len(seeds))
    x = torch.randn(plan.total_rows, 80, generator=generator).cuda()
    x[row_seq < 0] = 0
    return plan, views, row_seq, x


@pytest.mark.parametrize('mode', ['bf16', 'bf16x3', 'bf16x6'])
@pytest.mark.parametrize('method', ['sum', 'average', 'max', 'center'])
def test_pair_fused_pooling(eng, golden, mode, method):
    """Fused pooling on one tile, on three, and over several rounds: equal to
    the conv stack followed by the pooling kernel (max / center bit for bit,
    sums to fp32 rounding), and bit-identical run to run"""
    stack = _frame_stack(golden)
    corpora = [
        ([500], [0.9]),                          # one tile
        ([501, 502], [1.5, 1.4]),                # three tiles
        (list(range(600, 760)), None),           # ~1500 tiles: several rounds
    ]
    for seeds, durations in corpora:
        plan, views, row_seq, x = _corpus(eng, seeds, durations)
        frames = eng.conv_stack(x, row_seq, stack, _precision(mode))
        separate = eng.pool(
            frames, views['row_start'], views['n_rows'], views['word_seq'],
            views['word_lo'], views['word_hi'], method)
        fused, kept = eng.conv_stack_pool(
            x, row_seq, stack, _precision(mode), views, plan.total_word_rows, method,
            keep_frames=True)
        assert torch.equal(kept, frames)
        keep = torch.from_numpy(plan.word_seq >= 0).cuda()
        assert (fused[~keep] == 0).all()
        if method in ('max', 'center'):
            assert torch.equal(fused[keep], separate[keep])
        else:
            scale = separate[keep].abs().max().item()
            assert (fused[keep] - separate[keep]).abs().max().item() < 2e-6 * scale
        again, _ = eng.conv_stack_pool(
            x, row_seq, stack, _precision(mode), views, plan.total_word_rows, method)
        assert torch.equal(again, fused)
