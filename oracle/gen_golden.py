"""Generate golden vectors from the UNMODIFIED reference (test infrastructure).

Run in the build container only (needs /root/reference):

    python -m oracle.gen_golden

Writes tests/golden/*.npz.  Every array is an input to, or an output of, the
reference's own code (`emphases.preprocess`, `emphases.Model.forward`,
`emphases.downsample`, `emphases.segment`, `emphases.loss`,
`emphases.from_alignment_and_audio`) imported through `oracle/ref_stubs.py`.
The GPU box has no /root/reference; tests there replay these files.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from golden_util import save_golden  # noqa: E402
from oracle import ref_stubs  # noqa: E402
from oracle import emphases_oracle as oracle  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
CHECKPOINT = os.path.join(
    ref_stubs.REFERENCE_ROOT,
    'emphases', 'assets', 'checkpoints', 'checkpoint.pt')

METHODS = ['average', 'max', 'sum', 'center']
LOCATIONS = ['input', 'intermediate', 'inference', 'loss']


def to_numpy(state):
    return {k: v.detach().cpu().float().numpy() for k, v in state.items()}


def c1_inputs():
    """SURVEY.md section 8c known-answer inputs"""
    torch.manual_seed(0)
    audio = (0.1 * torch.randn(1, 160000)).clamp(-1, 1)
    generator = torch.Generator().manual_seed(1)
    cuts = torch.sort(torch.rand(24, generator=generator) * 10).values
    edges = [0.0] + [float(c) for c in cuts] + [10.0]
    times = list(zip(edges[:-1], edges[1:]))
    return times, audio


def scaled_random_state(emphases, gain, seed=0):
    """Random-init reference Model with conv weights scaled by `gain`
    (random init alone is dominated by the bias chain, SURVEY section 4)"""
    torch.manual_seed(seed)
    model = emphases.Model()
    state = model.state_dict()
    for key, value in state.items():
        if key.endswith('weight') and value.dim() >= 2 and 'norm' not in key:
            value.mul_(gain)
    return {k: v.clone() for k, v in state.items()}


def padded_batch(items):
    """collate-style padding (emphases/data/collate.py:11-78)"""
    B = len(items)
    tmax = max(f.shape[-1] for f, _ in items)
    wmax = max(b.shape[-1] for _, b in items)
    features = torch.zeros(B, items[0][0].shape[1], tmax)
    bounds = torch.zeros(B, 2, wmax, dtype=torch.long)
    frame_lengths = torch.zeros(B, dtype=torch.long)
    word_lengths = torch.zeros(B, dtype=torch.long)
    for i, (f, b) in enumerate(items):
        features[i, :, :f.shape[-1]] = f[0]
        bounds[i, :, :b.shape[-1]] = b[0]
        frame_lengths[i] = f.shape[-1]
        word_lengths[i] = b.shape[-1]
    return features, frame_lengths, bounds, word_lengths


def gen_c1():
    times, audio = c1_inputs()
    out = {'audio': audio.numpy(), 'times': np.array(times, dtype=np.float64)}
    with ref_stubs.reference() as emphases:
        assert emphases.DOWNSAMPLE_METHOD == 'sum'
        alignment = ref_stubs.Alignment.from_times(times)
        model = emphases.Model()
        state = torch.load(
            CHECKPOINT, map_location='cpu', weights_only=False)['model']
        model.load_state_dict(state)
        model.eval()
        for key, value in to_numpy(state).items():
            out[f'state.{key}'] = value
        out['mel_basis'] = oracle.mel_basis()
        for batch_size in (None, 300, 100):
            tag = 'full' if batch_size is None else f'bs{batch_size}'
            chunks = list(emphases.preprocess(
                alignment, audio, 16000, batch_size, None))
            out[f'{tag}.num_chunks'] = np.array(len(chunks))
            scores = []
            for i, (features, bounds) in enumerate(chunks):
                out[f'{tag}.{i}.bounds'] = bounds.numpy()
                out[f'{tag}.{i}.frames'] = np.array(features.shape[-1])
                if batch_size in (None, 300):
                    out[f'{tag}.{i}.features'] = features.numpy()
                with torch.no_grad():
                    logits = model(
                        features,
                        torch.tensor([features.shape[-1]]),
                        bounds,
                        torch.tensor([bounds.shape[-1]]))
                scores.append(emphases.postprocess(logits[0]))
            out[f'{tag}.scores'] = torch.cat(scores, 1).numpy()
        # Intermediates for the unchunked case
        features, bounds = next(iter(
            emphases.preprocess(alignment, audio, 16000, None, None)))
        with torch.no_grad():
            frame_embeddings = model.frame_encoder(
                model.input_layer(features), None)
            word_embeddings = emphases.downsample(
                frame_embeddings, bounds, torch.tensor([bounds.shape[-1]]))
        out['full.frame_embeddings'] = frame_embeddings.numpy()
        out['full.word_embeddings'] = word_embeddings.numpy()
        # The reference's own public call (bf16 autocast on CPU)
        import tempfile
        with tempfile.TemporaryDirectory() as directory:
            path = os.path.join(directory, 'ckpt.pt')
            torch.save({'model': state}, path)
            result = emphases.from_alignment_and_audio(
                alignment, audio, 16000, checkpoint=path)
        out['full.scores_autocast'] = result.float().numpy()
        out['full.scores_autocast_dtype'] = np.array(str(result.dtype))
    save_golden('c1', out)
    print('c1', {k: v.shape for k, v in out.items() if 'state' not in k})


def gen_sweep():
    """method x location sweep, B=1 and padded B=2, gain-scaled random init"""
    out = {}
    t1, a1 = oracle.synthetic_utterance(11, duration=3.0, words=8)
    t2, a2 = oracle.synthetic_utterance(12, duration=2.0, words=5)
    out['audio1'], out['times1'] = a1.numpy(), np.array(t1)
    out['audio2'], out['times2'] = a2.numpy(), np.array(t2)
    base_state = None
    for location in LOCATIONS:
        for method in METHODS:
            overrides = {
                'DOWNSAMPLE_LOCATION': location,
                'DOWNSAMPLE_METHOD': method}
            with ref_stubs.reference(overrides) as emphases:
                if base_state is None:
                    assert location == 'input'
                    base_state = scaled_random_state(emphases, 1.6)
                    for key, value in to_numpy(base_state).items():
                        out[f'state.{key}'] = value
                model = emphases.Model()
                model.load_state_dict(
                    {k: v for k, v in base_state.items()
                     if k in model.state_dict()})
                model.eval()
                items = []
                for times, audio in ((t1, a1), (t2, a2)):
                    alignment = ref_stubs.Alignment.from_times(times)
                    items.append(next(iter(emphases.preprocess(
                        alignment, audio, 16000, None, None))))
                tag = f'{location}.{method}'
                with torch.no_grad():
                    features, bounds = items[0]
                    logits = model(
                        features,
                        torch.tensor([features.shape[-1]]),
                        bounds,
                        torch.tensor([bounds.shape[-1]]))
                    out[f'{tag}.b1.logits'] = logits.numpy()
                    batch = padded_batch(items)
                    out[f'{tag}.b2.logits'] = model(*batch).numpy()
                    if location == 'inference':
                        model.train()
                        out[f'{tag}.b2.frame_logits'] = model(*batch).numpy()
                        model.eval()
                if tag == 'input.average':
                    out['b1.features'] = items[0][0].numpy()
                    out['b1.bounds'] = items[0][1].numpy()
                    for name, value in zip(
                        ('features', 'frame_lengths', 'bounds', 'word_lengths'),
                        batch
                    ):
                        out[f'b2.{name}'] = value.numpy()
    save_golden('sweep', out)
    print('sweep', len(out))


def gen_pool():
    """emphases.downsample / emphases.segment on adversarial bounds"""
    out = {}
    generator = torch.Generator().manual_seed(5)
    xs = torch.randn(2, 80, 50, generator=generator)
    # item 0: zero-length word, single-frame word, overshoot by 1 and far
    # past T, first word starting after 0.  item 1: one word, rest padding.
    bounds = torch.tensor([
        [[3, 10, 10, 11, 30, 49, 60], [10, 10, 11, 30, 49, 51, 70]],
        [[0, 0, 0, 0, 0, 0, 0], [50, 0, 0, 0, 0, 0, 0]]], dtype=torch.long)
    lengths = torch.tensor([7, 1])
    out['xs'], out['bounds'], out['lengths'] = (
        xs.numpy(), bounds.numpy(), lengths.numpy())
    # a clean case every method accepts
    clean_bounds = torch.tensor([
        [[0, 7, 8, 20, 33], [7, 8, 20, 33, 50]],
        [[2, 25, 0, 0, 0], [25, 48, 0, 0, 0]]], dtype=torch.long)
    clean_lengths = torch.tensor([5, 2])
    out['clean_bounds'] = clean_bounds.numpy()
    out['clean_lengths'] = clean_lengths.numpy()
    for method in METHODS:
        with ref_stubs.reference({'DOWNSAMPLE_METHOD': method}) as emphases:
            out[f'clean.{method}'] = emphases.downsample(
                xs, clean_bounds, clean_lengths).numpy()
            try:
                out[f'adversarial.{method}'] = emphases.downsample(
                    xs, bounds, lengths).numpy()
                out[f'adversarial.{method}.error'] = np.array('')
            except Exception as error:
                out[f'adversarial.{method}.error'] = np.array(
                    type(error).__name__)
            if method == 'sum':
                segments, seg_bounds, seg_lengths = emphases.segment(
                    xs, clean_bounds, clean_lengths)
                out['segment.segments'] = segments.numpy()
                out['segment.bounds'] = seg_bounds.numpy()
                out['segment.lengths'] = seg_lengths.numpy()
    save_golden('pool', out)
    print('pool', {k: (v.shape if v.ndim else str(v)) for k, v in out.items()})


def gen_transformer():
    out = {}
    t1, a1 = oracle.synthetic_utterance(21, duration=3.0, words=8)
    t2, a2 = oracle.synthetic_utterance(22, duration=2.0, words=5)
    overrides = {'ARCHITECTURE': 'transformer'}
    with ref_stubs.reference(overrides) as emphases:
        assert emphases.DOWNSAMPLE_LOCATION == 'intermediate'
        state = scaled_random_state(emphases, 1.0, seed=3)
        model = emphases.Model()
        model.load_state_dict(state)
        model.eval()
        for key, value in to_numpy(state).items():
            if key.endswith('position.encoding'):
                continue  # deterministic table, rebuilt by the consumer
            out[f'state.{key}'] = value
        items = []
        for times, audio in ((t1, a1), (t2, a2)):
            alignment = ref_stubs.Alignment.from_times(times)
            items.append(next(iter(emphases.preprocess(
                alignment, audio, 16000, None, None))))
        with torch.no_grad():
            features, bounds = items[0]
            out['b1.features'] = features.numpy()
            out['b1.bounds'] = bounds.numpy()
            out['b1.logits'] = model(
                features,
                torch.tensor([features.shape[-1]]),
                bounds,
                torch.tensor([bounds.shape[-1]])).numpy()
            out['b1.frame_embeddings'] = model.frame_encoder(
                model.input_layer(features),
                torch.tensor([features.shape[-1]])).numpy()
            batch = padded_batch(items)
            for name, value in zip(
                ('features', 'frame_lengths', 'bounds', 'word_lengths'), batch
            ):
                out[f'b2.{name}'] = value.numpy()
            out['b2.logits'] = model(*batch).numpy()
    save_golden('transformer', out)
    print('transformer', len(out))


def gen_transformer_input():
    """Transformer variant at DOWNSAMPLE_LOCATION='input' (word segments are
    the sequences the encoder attends over, emphases/model/core.py:41-87),
    B=1 and a padded B=2 batch"""
    out = {}
    t1, a1 = oracle.synthetic_utterance(41, duration=1.6, words=6)
    t2, a2 = oracle.synthetic_utterance(42, duration=1.1, words=4)
    overrides = {'ARCHITECTURE': 'transformer', 'DOWNSAMPLE_LOCATION': 'input'}
    with ref_stubs.reference(overrides) as emphases:
        assert emphases.DOWNSAMPLE_LOCATION == 'input'
        state = scaled_random_state(emphases, 1.0, seed=5)
        model = emphases.Model()
        model.load_state_dict(state)
        model.eval()
        for key, value in to_numpy(state).items():
            if key.endswith('position.encoding'):
                continue
            out[f'state.{key}'] = value
        items = []
        for times, audio in ((t1, a1), (t2, a2)):
            alignment = ref_stubs.Alignment.from_times(times)
            items.append(next(iter(emphases.preprocess(
                alignment, audio, 16000, None, None))))
        with torch.no_grad():
            features, bounds = items[0]
            out['b1.features'] = features.numpy()
            out['b1.bounds'] = bounds.numpy()
            out['b1.logits'] = model(
                features,
                torch.tensor([features.shape[-1]]),
                bounds,
                torch.tensor([bounds.shape[-1]])).numpy()
            batch = padded_batch(items)
            for name, value in zip(
                ('features', 'frame_lengths', 'bounds', 'word_lengths'), batch
            ):
                out[f'b2.{name}'] = value.numpy()
            out['b2.logits'] = model(*batch).numpy()
    save_golden('transformer_input', out)
    print('transformer_input', len(out))


def gen_loss():
    out = {}
    generator = torch.Generator().manual_seed(9)
    scores = torch.randn(3, 1, 12, generator=generator)
    targets = torch.rand(3, 1, 12, generator=generator)
    word_lengths = torch.tensor([12, 7, 1])
    out['scores'], out['targets'], out['word_lengths'] = (
        scores.numpy(), targets.numpy(), word_lengths.numpy())
    with ref_stubs.reference() as emphases:
        for loss_fn in ('bce', 'mse'):
            out[loss_fn] = emphases.loss(
                scores, targets, None, None, word_lengths,
                loss_fn=loss_fn).numpy()
    save_golden('loss', out)
    print('loss', out['bce'], out['mse'])


def gen_upsample():
    """emphases.upsample and the frame-resolution loss (inference location)"""
    out = {}
    generator = torch.Generator().manual_seed(13)
    xs = torch.rand(3, 1, 9, generator=generator)
    bounds = torch.tensor([
        [[0, 7, 8, 20, 33, 40, 41, 60, 77], [7, 8, 20, 33, 40, 41, 60, 77, 90]],
        [[2, 25, 30, 31, 0, 0, 0, 0, 0], [25, 30, 31, 48, 0, 0, 0, 0, 0]],
        [[0, 0, 0, 0, 0, 0, 0, 0, 0], [55, 0, 0, 0, 0, 0, 0, 0, 0]]],
        dtype=torch.long)
    word_lengths = torch.tensor([9, 4, 1])
    frame_lengths = torch.tensor([90, 50, 55])
    wide = torch.rand(3, 4, 9, generator=generator)
    scores = torch.randn(3, 1, 90, generator=generator)
    for name, value in (
        ('xs', xs), ('wide', wide), ('bounds', bounds), ('scores', scores),
        ('word_lengths', word_lengths), ('frame_lengths', frame_lengths)
    ):
        out[name] = value.numpy()
    for method in ('linear', 'nearest'):
        overrides = {
            'UPSAMPLE_METHOD': method, 'DOWNSAMPLE_LOCATION': 'inference'}
        with ref_stubs.reference(overrides) as emphases:
            out[f'{method}.xs'] = emphases.upsample(
                xs, bounds, word_lengths, frame_lengths).numpy()
            out[f'{method}.wide'] = emphases.upsample(
                wide, bounds, word_lengths, frame_lengths).numpy()
            for loss_fn in ('bce', 'mse'):
                out[f'{method}.loss.{loss_fn}'] = emphases.loss(
                    scores, xs, frame_lengths, bounds, word_lengths,
                    training=True, loss_fn=loss_fn).numpy()
    save_golden('upsample', out)
    print('upsample', {k: v.shape for k, v in out.items()})


def gen_sampler():
    """Sampler.batch / Dataset.buckets / collate of the unmodified reference"""
    out = {}
    rng = np.random.default_rng(17)
    with ref_stubs.reference() as emphases:
        for name, size, max_frames in (
            ('a', 101, 20000), ('b', 64, 75000), ('c', 7, 3000)
        ):
            lengths = rng.integers(200, 2001, size=size)

            class Fake:
                def __len__(self):
                    return len(lengths)
            fake = Fake()
            fake.lengths = lengths.tolist()
            fake.buckets = lambda fake=fake: emphases.data.Dataset.buckets(fake)
            # (`emphases.data.sampler` is shadowed by the function of that name)
            sampler = sys.modules['emphases.data.sampler'].Sampler(
                fake, max_frames)
            out[f'{name}/lengths'] = lengths
            out[f'{name}/max_frames'] = np.int64(max_frames)
            for epoch in (0, 3):
                sampler.set_epoch(epoch)
                batches = sampler.batch()
                out[f'{name}/epoch{epoch}/flat'] = np.array(
                    [i for batch in batches for i in batch], dtype=np.int64)
                out[f'{name}/epoch{epoch}/sizes'] = np.array(
                    [len(batch) for batch in batches], dtype=np.int64)

        # collate (emphases/data/collate.py:11-77)
        generator = torch.Generator().manual_seed(19)
        items = []
        for index, (frames, words) in enumerate(((50, 6), (80, 3), (64, 9))):
            features = torch.randn(80, frames, generator=generator)
            scores = torch.rand(1, words, generator=generator)
            cuts = torch.sort(torch.randperm(
                frames - 1, generator=generator)[:words - 1] + 1).values
            edges = torch.cat([
                torch.zeros(1, dtype=torch.long), cuts,
                torch.full((1,), frames)])
            bounds = torch.stack([edges[:-1], edges[1:]])
            audio = torch.randn(1, frames * 160 + 37 * index, generator=generator)
            items.append((features, scores, bounds, None, audio, f'stem{index}'))
            out[f'collate/item{index}/features'] = features.numpy()
            out[f'collate/item{index}/scores'] = scores.numpy()
            out[f'collate/item{index}/bounds'] = bounds.numpy()
            out[f'collate/item{index}/audio'] = audio.numpy()
        batch = emphases.data.collate(items)
        for key, value in zip(
            ('features', 'frame_lengths', 'word_bounds', 'word_lengths',
             'scores', None, 'audio', None), batch
        ):
            if key is not None:
                out[f'collate/{key}'] = value.numpy()
    save_golden('sampler', out)
    print('sampler.npz', len(out))


def gen_evaluate():
    """The loop body of emphases.evaluate.datasets (evaluate/core.py:27-110)
    with the reference's own Statistics / Metrics classes, on synthetic logits
    and targets for six 'files' (torchutil restated, see ref_stubs)"""
    out = {}
    generator = torch.Generator().manual_seed(23)
    sizes = (12, 5, 31, 2, 18, 9)
    logits = [2 * torch.randn(1, 1, n, generator=generator) for n in sizes]
    targets = [torch.rand(1, 1, n, generator=generator) for n in sizes]
    for index, (x, t) in enumerate(zip(logits, targets)):
        # correlate predictions and targets a little
        logits[index] = x + 3 * (t - .5)
        out[f'logits{index}'] = logits[index].numpy()
        out[f'targets{index}'] = t.numpy()
    for loss_fn in ('bce', 'mse'):
        with ref_stubs.reference({'LOSS': loss_fn}) as emphases:
            metrics = emphases.evaluate.metrics
            target_stats = metrics.Statistics()
            predicted_stats = metrics.Statistics()
            for x, t in zip(logits, targets):
                lengths = torch.tensor([x.shape[-1]])
                scores = emphases.postprocess(x[0])           # (1, W)
                target_stats.update(t, lengths)
                predicted_stats.update(scores[None], lengths)
            file_metrics = emphases.evaluate.Metrics(predicted_stats, target_stats)
            dataset_metrics = emphases.evaluate.Metrics(predicted_stats, target_stats)
            granular = []
            for x, t in zip(logits, targets):
                lengths = torch.tensor([x.shape[-1]])
                file_metrics.reset()
                file_metrics.update(x, t, lengths)
                dataset_metrics.update(x, t, lengths)
                granular.append(file_metrics())
            overall = dataset_metrics()
            keys = ('pearson_correlation', 'bce', 'mse')
            out[f'{loss_fn}/overall'] = np.array(
                [overall[k] for k in keys], dtype=np.float64)
            out[f'{loss_fn}/granular'] = np.array(
                [[g[k] for k in keys] for g in granular], dtype=np.float64)
            out[f'{loss_fn}/stats'] = np.array(
                [*predicted_stats(), *target_stats()], dtype=np.float64)
    save_golden('evaluate', out)
    print('evaluate.npz', len(out))


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(1)
    if len(sys.argv) > 1:            # e.g. `python oracle/gen_golden.py transformer_input`
        for name in sys.argv[1:]:
            globals()[f'gen_{name}']()
        return
    gen_c1()
    gen_sweep()
    gen_pool()
    gen_transformer()
    gen_transformer_input()
    gen_loss()
    gen_upsample()
    gen_sampler()
    gen_evaluate()


if __name__ == '__main__':
    main()
