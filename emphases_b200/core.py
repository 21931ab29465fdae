"""Public inference API, mirroring emphases/core.py (same names, arguments,
defaults, return shapes and error behaviour), executed by sm_100a kernels.

Differences from the reference, all documented in DESIGN.md:
  * `gpu=None` means the current CUDA device (no CPU path);
  * scores are returned in fp32 (the reference returns bf16 / fp16 from its
    autocast context, core.py:606);
  * `from_files_to_files` batches all files into packed launches instead of
    looping over files (core.py:174-179), and accepts a list of GPU indices.
"""
import contextlib
import os
import threading
from pathlib import Path

import numpy as np
import torch

import emphases_b200 as emphases
from . import _lib, engine, resampling
from .alignment import Alignment, as_times

__all__ = [
    'from_file', 'from_file_to_file', 'from_files_to_files',
    'from_text_and_audio', 'from_alignment_and_audio',
    'from_alignments_and_audio', 'infer', 'infer_with_model', 'postprocess', 'preprocess',
    'downsample', 'upsample', 'segment', 'inference_context', 'resample',
    'load_model']


###############################################################################
# Emphasis annotation API (emphases/core.py:23-287)
###############################################################################


def from_file(text_file, audio_file, checkpoint=None, batch_size=None, gpu=None):
    """Produce emphasis scores for each word for files on disk
    (emphases/core.py:23-73).  `.TextGrid` -> scores (1, W)."""
    audio = emphases.load.audio(audio_file)
    if str(text_file).endswith('.TextGrid'):
        alignment = Alignment(text_file)
        return from_alignment_and_audio(
            alignment, audio, emphases.SAMPLE_RATE, checkpoint, batch_size, gpu)
    with open(text_file, encoding='utf-8') as file:
        text = file.read()
    return from_text_and_audio(
        text, audio, emphases.SAMPLE_RATE, checkpoint, batch_size, gpu)


def from_file_to_file(
    text_file,
    audio_file,
    output_prefix=None,
    checkpoint=None,
    batch_size=None,
    gpu=None
):
    """emphases/core.py:76-112: writes {prefix}.TextGrid and {prefix}.pt"""
    text_file = Path(text_file)
    if output_prefix is None:
        output_prefix = text_file.stem
    results = from_file(text_file, audio_file, checkpoint, batch_size, gpu)
    if text_file.name.endswith('.txt'):
        alignment, results = results
    else:
        alignment = Alignment(text_file)
    alignment.save(f'{output_prefix}.TextGrid')
    torch.save(results.cpu(), f'{output_prefix}.pt')


# from_files_to_files: write a launch's .pt files while later launches run
# (EMPHASES_B200_OVERLAP_SCORE_WRITES=0: all of them after the last launch)
OVERLAP_SCORE_WRITES = os.environ.get('EMPHASES_B200_OVERLAP_SCORE_WRITES', '1') != '0'
SCORE_WRITER_THREADS = 8


def from_files_to_files(
    text_files,
    audio_files,
    output_prefixes=None,
    checkpoint=None,
    batch_size=None,
    gpu=None
):
    """emphases/core.py:115-179.  All files are decoded by a thread pool,
    packed into length-balanced launches (one shard per GPU when `gpu` is a
    list of indices) and written back as {prefix}.TextGrid / {prefix}.pt."""
    if output_prefixes is None:
        output_prefixes = [Path(file).stem for file in text_files]
    text_files = [os.fspath(file) for file in text_files]
    audio_files = [os.fspath(file) for file in audio_files]
    output_prefixes = [os.fspath(prefix) for prefix in output_prefixes]
    if any(file.endswith('.txt') for file in text_files):
        raise NotImplementedError(
            'Transcript (.txt) inputs need forced alignment with pyfoal/HTK '
            '(emphases/core.py:138-166), which is outside this build; pass '
            '.TextGrid alignments')

    from . import corpus
    # host threads of this process: the ranks of one box (torchrun) share its cores
    local_world = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))
    workers = max(2, min(32, (os.cpu_count() or 1) // local_world))
    with corpus.Corpus(text_files, audio_files, workers) as parsed:
        # Fast path: 16-bit PCM wav + a parsable TextGrid go through the native
        # reader into pinned int16 / float64 buffers; files at the model rate
        # first, then one packed GPU resampling pass per other sample rate
        # (the reference resamples file by file, core.py:613-619)
        parsable = parsed.usable(None)
        rates = sorted(
            {int(rate) for rate in parsed.sample_rate[parsable]},
            key=lambda rate: rate != emphases.SAMPLE_RATE)
        scores = [None] * len(text_files)
        failure = []
        single_device = not (isinstance(gpu, (list, tuple)) and len(gpu) > 1)
        flat_results = []       # (file indices, flat host scores, words per file)

        def write_alignments():
            try:
                parsed.write_textgrids_to_prefixes(output_prefixes, parsable)
            except Exception as error:      # re-raised on the caller's thread
                failure.append(error)

        # the alignments do not depend on the scores: they are written while
        # the GPU works
        writer = threading.Thread(target=write_alignments)
        if parsable.any():
            writer.start()
        try:
            for rate in rates:
                indices, times, packed = parsed.load(
                    parsable & (parsed.sample_rate == rate))
                if rate != emphases.SAMPLE_RATE and single_device:
                    # converted inside the log-mel kernel, launch by launch
                    from . import scheduler
                    packed = scheduler.ResampledSource(packed, rate)
                elif rate != emphases.SAMPLE_RATE:
                    device = emphases.resolve_device(
                        gpu[0] if isinstance(gpu, (list, tuple)) and gpu else gpu)
                    packed = resampling.resample_packed(
                        packed, rate, emphases.SAMPLE_RATE, device)
                if single_device:
                    # per launch: the words of its files in one flat host tensor
                    # (no 24,000-way split: the native writer takes pointers),
                    # written as {prefix}.pt -- the archives torch.save would
                    # write -- on a background thread while later launches are
                    # decoded and run; on its own few threads (negative count),
                    # beside the decode that owns the worker pool
                    def write_launch(members, flat_scores, counts, indices=indices):
                        files = indices[np.asarray(members, dtype=np.int64)]
                        corpus.write_score_rows(
                            [output_prefixes[i] for i in files.tolist()], flat_scores,
                            counts, -SCORE_WRITER_THREADS, suffix='.pt')
                        for index in files:
                            scores[int(index)] = True

                    if OVERLAP_SCORE_WRITES:
                        from_alignments_and_audio(
                            times, packed, emphases.SAMPLE_RATE, checkpoint, batch_size,
                            gpu, flat=True, sink=write_launch)
                        continue
                    for members, flat_scores, counts in from_alignments_and_audio(
                        times, packed, emphases.SAMPLE_RATE, checkpoint, batch_size,
                        gpu, flat=True
                    ):
                        files = indices[np.asarray(members, dtype=np.int64)]
                        flat_results.append((files, flat_scores, counts))
                        for index in files:
                            scores[int(index)] = True
                    continue
                results = from_alignments_and_audio(
                    times, packed, emphases.SAMPLE_RATE, checkpoint, batch_size, gpu)
                for index, result in zip(indices, results):
                    scores[index] = result
        finally:
            if parsable.any():
                writer.join()
        if failure:
            raise failure[0]
        indices = np.nonzero(parsable)[0]

    # {prefix}.pt: same archives torch.save would write, from the native pool
    for files, flat_scores, counts in flat_results:
        corpus.write_score_rows(
            [output_prefixes[i] for i in files.tolist()], flat_scores, counts, workers,
            suffix='.pt')
    done = [int(i) for i in indices if scores[int(i)] is not True]
    if done:
        corpus.write_scores(
            [f'{output_prefixes[i]}.pt' for i in done], [scores[i] for i in done],
            workers)

    # Everything else (other encodings / sample rates) goes file by file
    first_gpu = gpu[0] if isinstance(gpu, (list, tuple)) and gpu else gpu
    for index in range(len(text_files)):
        if scores[index] is None:
            from_file_to_file(
                text_files[index], audio_files[index], output_prefixes[index],
                checkpoint, batch_size, first_gpu)


def from_text_and_audio(
    text, audio, sample_rate, checkpoint=None, batch_size=None, gpu=None
):
    """emphases/core.py:182-220.  Needs the pyfoal P2FA forced aligner (HTK);
    used when installed, otherwise a clear error."""
    try:
        import pyfoal
    except ImportError as error:
        raise NotImplementedError(
            'from_text_and_audio needs pyfoal (P2FA/HTK forced alignment, '
            'emphases/core.py:205-209), which is not installed; pass an '
            'alignment to from_alignment_and_audio instead') from error
    alignment = pyfoal.from_text_and_audio(
        text, audio, sample_rate, aligner='p2fa')
    scores = from_alignment_and_audio(
        alignment, audio, sample_rate, checkpoint, batch_size, gpu)
    return alignment, scores


def from_alignment_and_audio(
    alignment, audio, sample_rate, checkpoint=None, batch_size=None, gpu=None
):
    """Produce emphasis scores for each word (emphases/core.py:223-287)

    Returns scores (1, W) fp32 on the CUDA device.  All chunks of the
    utterance run in ONE packed launch sequence (no per-chunk forward, no
    per-word host sync)."""
    if emphases.METHOD != 'neural':
        if emphases.METHOD in (
            'prominence', 'pitch-variance', 'duration-variance'
        ):
            raise NotImplementedError(
                f'The {emphases.METHOD} baseline is a CPU numpy method of the '
                'reference (emphases/baselines) and is out of scope here')
        raise ValueError(
            f'Emphasis annotation method {emphases.METHOD} is not defined')
    if batch_size is None and not isinstance(gpu, (list, tuple)):
        # one utterance, one chunk: a single native call plans and launches
        # the whole path (csrc/utterance.cu); None = not that case
        from . import single
        device = emphases.resolve_device(gpu)
        with torch.cuda.device(device):
            scores = single.from_alignment_and_audio(
                load_model(checkpoint, device), alignment, audio, sample_rate, device)
        if scores is not None:
            return scores
    return from_alignments_and_audio(
        [alignment], [audio], sample_rate, checkpoint, batch_size, gpu,
        to_cpu=False)[0]


def from_alignments_and_audio(
    alignments,
    audios,
    sample_rate,
    checkpoint=None,
    batch_size=None,
    gpu=None,
    to_cpu=True,
    model=None,
    flat=False,
    sink=None
):
    """Batched form of from_alignment_and_audio (extension): lists in, list
    of (1, W_i) score tensors out.  `gpu` may be a list of device indices:
    utterances are split with the length-balanced scheduler and each shard
    runs on its own device; results are gathered on the host.  flat=True
    (one device): scheduler.run_on_device's unsplit per-launch results, handed
    to `sink` launch by launch on a background thread when one is given."""
    from . import scheduler
    if isinstance(gpu, (list, tuple)) and len(gpu) > 1:
        if flat:
            raise ValueError('flat results are a single-device form')
        return scheduler.run_sharded(
            alignments, audios, sample_rate, checkpoint, batch_size, list(gpu))
    if isinstance(gpu, (list, tuple)):
        gpu = gpu[0] if gpu else None
    device = emphases.resolve_device(gpu)
    if model is None:
        model = load_model(checkpoint, device)
    with torch.cuda.device(device):
        return scheduler.run_on_device(
            model, alignments, audios, sample_rate, batch_size, device, to_cpu,
            flat=flat, sink=sink)


###############################################################################
# Inference steps (emphases/core.py:295-418)
###############################################################################


def resolve_checkpoint(checkpoint):
    """checkpoint=None is the published model (emphases/core.py:307-310)"""
    if checkpoint is not None:
        return checkpoint
    try:
        import huggingface_hub
        return huggingface_hub.hf_hub_download('maxrmorrison/emphases', 'model.pt')
    except Exception as error:
        raise RuntimeError(
            'checkpoint=None downloads maxrmorrison/emphases from the '
            'HuggingFace hub (emphases/core.py:307-310), which needs '
            'network access; pass a checkpoint path') from error


_models = {}                       # device -> (key, model): one entry per device
_models_lock = threading.Lock()


def load_model(checkpoint, device):
    """Model cache of emphases.infer (core.py:298-315), keyed on
    (checkpoint, device) and on the configuration the Model captured.  One
    model is kept per device (the multi-GPU workers of from_files_to_files
    share this loader), replaced when the key changes."""
    device = torch.device(device)
    if device.type == 'cuda' and device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    key = (
        None if checkpoint is None else str(checkpoint),
        emphases.ARCHITECTURE, emphases.DOWNSAMPLE_LOCATION, emphases.LAYERS,
        emphases.CHANNELS, emphases.DROPOUT,
        emphases.ACTIVATION_FUNCTION.__name__, emphases.ENCODER_KERNEL_SIZE,
        emphases.DECODER_KERNEL_SIZE)
    with _models_lock:
        cached = _models.get(device)
        if cached is None or cached[0] != key:
            model = emphases.Model()
            state = torch.load(
                resolve_checkpoint(checkpoint), map_location='cpu',
                weights_only=False)
            model.load_state_dict(state['model'] if 'model' in state else state)
            cached = (key, model.to(device).eval())
            _models[device] = cached
        return cached[1]


def infer(features, word_bounds, checkpoint=None):
    """Model inference for one chunk (emphases/core.py:295-332):
    features (1, F, T), word_bounds (1, 2, W) -> logits (1, 1, W)"""
    device = emphases.resolve_device(None, features)
    return infer_with_model(load_model(checkpoint, device), features, word_bounds)


def infer_with_model(model, features, word_bounds):
    """`infer` with an explicit, already loaded model"""
    device = next(model.parameters()).device
    features = features.to(device)
    frame_lengths = torch.tensor(
        [features.shape[-1]], dtype=torch.long, device=device)
    word_lengths = torch.tensor(
        [word_bounds.shape[-1]], dtype=torch.long, device=device)
    with inference_context(model):
        return model(features, frame_lengths, word_bounds, word_lengths)


def postprocess(logits):
    """emphases/core.py:335-342"""
    if emphases.METHOD == 'neural':
        if emphases.LOSS == 'bce':
            return torch.sigmoid(logits)
        elif emphases.LOSS == 'mse':
            return torch.clamp(logits, 0., 1.)
    return logits


def preprocess(
    alignment, audio, sample_rate=None, batch_size=None, gpu=None
):
    """Convert audio to model input (emphases/core.py:345-418): yields
    (features (1, F, Tc) CUDA fp32, word_bounds (1, 2, Wc) int64) per
    word-aligned chunk.  All chunks' features come from one kernel launch."""
    if sample_rate is None:
        sample_rate = emphases.SAMPLE_RATE
    if sample_rate != emphases.SAMPLE_RATE:
        audio = resample(audio, sample_rate)
    device = emphases.resolve_device(gpu, audio)
    eng = emphases.get_engine(device)
    times = as_times(alignment)
    plan = engine.make_plan([(times, audio.shape[-1])], batch_size)
    if plan.n_seq == 0:
        return
    with torch.cuda.device(device):
        samples = audio[0].detach().to(device, torch.float32).contiguous()
        views = eng.upload_plan(plan)
        row_seq = eng.row_index(
            views['row_start'], views['n_rows'], plan.n_seq, plan.total_rows)
        rows = eng.logmel(samples, views, plan, row_seq, emphases.NORMALIZE)
    for u in range(plan.n_seq):
        start, frames = int(plan.row_start[u]), int(plan.n_rows[u])
        ws, words = int(plan.word_row_start[u]), int(plan.n_words[u])
        bounds = torch.from_numpy(np.stack([
            plan.word_lo[ws:ws + words],
            plan.word_hi[ws:ws + words]]).astype(np.int64))[None]
        yield rows[start:start + frames].t().contiguous()[None], bounds


###############################################################################
# Word and frame resolution resampling (emphases/core.py:426-469, 552-586)
###############################################################################


def downsample(xs, word_bounds, word_lengths):
    """Interpolate from frame to word resolution (emphases/core.py:426-469):
    xs (B, C, T) CUDA fp32, word_bounds (B, 2, Wmax), word_lengths (B,)
    -> (B, C, Wmax)"""
    from . import model as model_module
    method = emphases.DOWNSAMPLE_METHOD
    if method not in _lib.POOL:
        raise ValueError(f'Interpolation method {method} is not defined')
    device = emphases.resolve_device(None, xs)
    eng = emphases.get_engine(device)
    batch, _, frames = xs.shape
    with torch.cuda.device(device):
        rows, _, row_start, n_rows, _, _ = model_module.pack_batch(eng, xs)
        views, word_starts, _, bounds, lengths = \
            model_module.word_rows(word_bounds, word_lengths, device)
        if method == 'center':
            # center gathers every slot, padded ones included (core.py:458-466)
            views['word_lo'].clamp_(min=0)
            views['word_hi'].clamp_(min=0)
            lengths = np.full(batch, word_bounds.shape[2])
        model_module.check_word_bounds(bounds, lengths, frames, method)
        pooled = eng.pool(
            rows, row_start, n_rows, views['word_seq'], views['word_lo'],
            views['word_hi'], method)
        index = model_module.slot_index(word_starts, int(lengths.max()), device)
        return pooled[index].transpose(1, 2).contiguous().to(xs.dtype)


def upsample(xs, word_bounds, word_lengths, frame_lengths):
    """Interpolate from word to frame resolution (emphases/core.py:472-544):
    xs (B, C, Wmax) -> (B, C, max(frame_lengths)), UPSAMPLE_METHOD 'linear' or
    'nearest'"""
    method = emphases.UPSAMPLE_METHOD
    if method not in ('linear', 'nearest'):
        raise ValueError(f'Interpolation method {method} is not defined')
    device = emphases.resolve_device(None, xs)
    batch, channels, wmax = xs.shape
    tmax = int(frame_lengths.max())
    with torch.cuda.device(device):
        values = xs.detach().to(device, torch.float32).contiguous()
        bounds = word_bounds.detach().to(device, torch.int64).contiguous()
        words = word_lengths.detach().to(device, torch.int64).contiguous()
        frames = frame_lengths.detach().to(device, torch.int64).contiguous()
        out = torch.empty(
            (batch, channels, tmax), dtype=torch.float32, device=device)
        _lib.call(
            'emph_upsample_words', _lib.ptr(values), _lib.ptr(bounds),
            _lib.ptr(words), _lib.ptr(frames), batch, channels, wmax, tmax,
            int(method == 'linear'), _lib.ptr(out), _lib.stream_ptr())
    return out.to(xs.dtype)


def segment(xs, word_bounds, word_lengths):
    """Convert acoustic features to word segments (emphases/core.py:552-586)"""
    from . import segments
    return segments.segment(xs, word_bounds, word_lengths)


###############################################################################
# Utilities (emphases/core.py:594-619)
###############################################################################


@contextlib.contextmanager
def inference_context(model):
    """eval + no_grad (emphases/core.py:594-610).  The reference also enters
    torch.autocast; precision here is chosen by emphases_b200.PRECISION."""
    was_training = model.training
    model.eval()
    with torch.no_grad():
        yield
    if was_training:
        model.train()


def resample(audio, sample_rate, target_rate=None):
    """emphases/core.py:613-619: windowed-sinc resampling with torchaudio's
    default filter, computed by csrc/resample.cu.  The result lives on the
    device of `audio` like in the reference (a CPU tensor makes a round trip
    through the current CUDA device)."""
    if target_rate is None:
        target_rate = emphases.SAMPLE_RATE
    if sample_rate == target_rate:
        return audio
    from . import resampling
    device = emphases.resolve_device(None, audio)
    result = resampling.resample(audio, sample_rate, target_rate, device)
    return result if audio.device.type == 'cuda' else result.cpu()
