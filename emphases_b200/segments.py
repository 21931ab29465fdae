"""Word segmentation (`emphases.segment`, emphases/core.py:552-586) and the
'input' downsample location of Model.forward (emphases/model/core.py:41-87).

Each word slot becomes its own packed sequence of `max_length` rows: the
word's frames followed by zeros.  The frame encoder runs over ALL of those
rows and the reduction covers the padded tail too, exactly like the
reference's `frame_embeddings.mean(dim=2)` over the padded segment tensor
(SURVEY.md A.5 quirk 3).
"""
import numpy as np
import torch

import emphases_b200 as emphases
from . import _lib, engine
from .model import slot_views


def _segment_plan(word_bounds, word_lengths, frames):
    """Host integer plan shared by `segment` and the input-location forward"""
    bounds = word_bounds.detach().to('cpu', torch.int64).numpy()
    lengths = word_lengths.detach().to('cpu', torch.int64).numpy()
    batch, _, wmax = bounds.shape
    max_length = int((bounds[:, 1] - bounds[:, 0]).max())
    slot = np.minimum(
        np.arange(wmax)[None], lengths[:, None] - 1)          # core.py:574
    lo = np.take_along_axis(bounds[:, 0], slot, axis=1)
    hi = np.take_along_axis(bounds[:, 1], slot, axis=1)
    count = hi - lo
    if np.any(hi > frames) or np.any(lo < 0) or np.any(count < 0):
        raise RuntimeError(
            'segment(): word bounds outside the frame range (the reference '
            'fails with a shape mismatch here, emphases/core.py:583)')
    return bounds, lengths, max_length, lo, count


def _gather(eng, xs, lo, count, max_length):
    """(B, C, T) -> packed segment rows [(B*Wmax) sequences of max_length]"""
    device = xs.device
    batch, channels, frames = xs.shape
    n_seg = lo.size
    src_starts, src_total = engine.packed_starts([frames] * batch)
    seg_starts, seg_total = engine.packed_starts([max_length] * n_seg)
    src_row = (src_starts[:, None] + lo).reshape(-1)
    meta = torch.from_numpy(np.concatenate([
        src_starts, np.full(batch, frames),
        src_row, count.reshape(-1), seg_starts, np.full(n_seg, max_length)]
    ).astype(np.int32)).to(device)
    row_start, n_rows = meta[:batch], meta[batch:2 * batch]
    cursor = 2 * batch
    d_src_row = meta[cursor:cursor + n_seg]
    d_count = meta[cursor + n_seg:cursor + 2 * n_seg]
    d_seg_start = meta[cursor + 2 * n_seg:cursor + 3 * n_seg]
    d_seg_rows = meta[cursor + 3 * n_seg:]
    row_seq = eng.row_index(row_start, n_rows, batch, src_total)
    rows = torch.empty((src_total, channels), dtype=torch.float32, device=device)
    xs32 = xs.detach().to(torch.float32).contiguous()
    _lib.call(
        'emph_pack_rows', _lib.ptr(xs32), batch, channels, frames,
        _lib.ptr(row_start), _lib.ptr(n_rows), _lib.ptr(row_seq), src_total,
        _lib.ptr(rows), _lib.stream_ptr())
    seg_row_seq = eng.row_index(d_seg_start, d_seg_rows, n_seg, seg_total)
    segments = torch.empty(
        (seg_total, channels), dtype=torch.float32, device=device)
    _lib.call(
        'emph_segment_rows', _lib.ptr(rows), channels, _lib.ptr(d_src_row),
        _lib.ptr(d_count), _lib.ptr(d_seg_start), n_seg,
        _lib.ptr(seg_row_seq), seg_total, _lib.ptr(segments),
        _lib.stream_ptr())
    return segments, seg_row_seq, d_seg_start, d_seg_rows, seg_starts, seg_total


def segment(xs, word_bounds, word_lengths):
    """emphases.segment: returns (segments (B*Wmax, C, max_length),
    bounds (B*Wmax, 2, 1), lengths (B*Wmax,))"""
    device = emphases.resolve_device(None, xs)
    eng = emphases.get_engine(device)
    xs = xs.to(device)
    with torch.cuda.device(device):
        _, _, max_length, lo, count = _segment_plan(
            word_bounds, word_lengths, xs.shape[2])
        n_seg = lo.size
        segments, _, d_seg_start, d_seg_rows, _, _ = _gather(
            eng, xs, lo, count, max_length)
        result = torch.empty(
            (n_seg, xs.shape[1], max(max_length, 1)), dtype=torch.float32,
            device=device)
        if max_length > 0:
            _lib.call(
                'emph_unpack_rows', _lib.ptr(segments), _lib.ptr(d_seg_start),
                _lib.ptr(d_seg_rows), n_seg, xs.shape[1], max_length,
                _lib.ptr(result), _lib.stream_ptr())
        result = result[:, :, :max_length].to(xs.dtype)
        lengths = torch.from_numpy(count.reshape(-1)).to(device)
        result_bounds = torch.zeros(
            (n_seg, 2, 1), dtype=torch.long, device=device)
        result_bounds[:, 1, 0] = lengths
        return result, result_bounds, lengths


def input_word_rows(batch, wmax, lengths, count, max_length, method, device):
    """Packed word rows of the 'input' location: one word row per segment, laid
    out as B sequences of Wmax word slots; row w pools segment word_seq[w] over
    its padded length (model/core.py:55-63), masked slots are (-2, -2).
    Returns (device views, host word_starts, total_words)."""
    if method == 'max' and max_length == 0:
        raise IndexError('max(): Expected reduction dim 2 to have non-zero size')
    masked = np.arange(wmax)[None] >= lengths[:, None]          # word mask (:77-82)
    if method == 'center':
        if np.any((count // 2)[~masked] >= max(max_length, 1)):
            raise IndexError('center frame index out of range for a word')
        # downsample(frame_embeddings, [0, frames], ones): (0 + frames) // 2
        hi = count
    else:
        # reduction over the whole padded segment (model/core.py:55-63)
        hi = np.full_like(count, max_length)
    return slot_views(
        np.arange(batch * wmax).reshape(batch, wmax), np.where(masked, -2, 0),
        np.where(masked, -2, hi), device)


def run_forward_input(eng, features, word_bounds, word_lengths, method, encode, decode):
    """Model.forward for DOWNSAMPLE_LOCATION == 'input' up to the output head,
    with model.run_forward's encoder pair: every word segment is a sequence of
    max_length queries whose keys are the segment's own frames (the Transformer
    attends within each segment).  Returns (decoded word rows, word_row_seq,
    host word starts)."""
    batch, _, frames = features.shape
    wmax = word_bounds.shape[2]
    _, lengths, max_length, lo, count = _segment_plan(
        word_bounds, word_lengths, frames)
    segments, seg_row_seq, d_seg_start, d_seg_rows, _, _ = _gather(
        eng, features, lo, count, max_length)
    frame_rows = encode(
        segments, seg_row_seq, d_seg_start, np.full(lo.size, max_length),
        count.reshape(-1))
    views, word_starts, total_words = input_word_rows(
        batch, wmax, lengths, count, max_length, method, eng.device)
    pooled = eng.pool(
        frame_rows, d_seg_start, d_seg_rows, views['word_seq'], views['word_lo'],
        views['word_hi'], method)
    word_row_seq = eng.row_index(
        views['word_row_start'], views['n_words'], batch, total_words)
    words = decode(
        pooled, word_row_seq, views['word_row_start'], np.full(batch, wmax), lengths)
    return words, word_row_seq, word_starts
