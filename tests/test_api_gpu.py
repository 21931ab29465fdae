"""GPU parity tests of the reference-facing Python API (emphases_b200.*),
against goldens from the unmodified reference."""
import os

import numpy as np
import pytest
import torch

from golden_util import state_from_golden, times_list
from oracle import emphases_oracle as oracle

pytestmark = pytest.mark.gpu

METHODS = ['average', 'max', 'sum', 'center']
LOCATIONS = ['input', 'intermediate', 'inference', 'loss']


@pytest.fixture
def emphases():
    import emphases_b200
    emphases_b200.reset_configuration()
    yield emphases_b200
    emphases_b200.reset_configuration()


@pytest.fixture(scope='module')
def c1_checkpoint(tmp_path_factory, golden):
    path = tmp_path_factory.mktemp('ckpt') / 'checkpoint.pt'
    torch.save({'model': state_from_golden(golden('c1'))}, path)
    return path


def build_model(emphases, state):
    model = emphases.Model()
    own = model.state_dict()
    model.load_state_dict({k: v for k, v in state.items() if k in own})
    return model.cuda().eval()


@pytest.mark.parametrize('location', LOCATIONS)
@pytest.mark.parametrize('method', METHODS)
def test_model_forward_sweep(emphases, golden, location, method):
    """Model.forward, B=1 and padded B=2, every method x location"""
    data = golden('sweep')
    emphases.configure(
        DOWNSAMPLE_LOCATION=location, DOWNSAMPLE_METHOD=method)
    model = build_model(emphases, state_from_golden(data))
    tag = f'{location}.{method}'
    with torch.no_grad():
        features = torch.from_numpy(data['b1.features']).cuda()
        bounds = torch.from_numpy(data['b1.bounds'])
        logits = model(
            features, torch.tensor([features.shape[-1]]), bounds,
            torch.tensor([bounds.shape[-1]]))
        expected = data[f'{tag}.b1.logits']
        assert logits.shape == expected.shape
        np.testing.assert_allclose(
            logits.cpu().numpy(), expected, rtol=1e-5, atol=2e-5)
        batch = [torch.from_numpy(data[f'b2.{name}']) for name in (
            'features', 'frame_lengths', 'bounds', 'word_lengths')]
        batch[0] = batch[0].cuda()
        logits = model(*batch)
        expected = data[f'{tag}.b2.logits']
        assert logits.shape == expected.shape
        np.testing.assert_allclose(
            logits.cpu().numpy(), expected, rtol=1e-5, atol=2e-5)
        if location == 'inference':
            model.train()
            frame_logits = model(*batch)
            np.testing.assert_allclose(
                frame_logits.cpu().numpy(), data[f'{tag}.b2.frame_logits'],
                rtol=1e-5, atol=2e-5)


@pytest.mark.parametrize('batch_size', [None, 300, 100])
def test_from_alignment_and_audio(emphases, golden, c1_checkpoint, batch_size):
    data = golden('c1')
    alignment = emphases.Alignment.from_times(times_list(data['times']))
    audio = torch.from_numpy(data['audio'])
    scores = emphases.from_alignment_and_audio(
        alignment, audio, 16000, checkpoint=c1_checkpoint,
        batch_size=batch_size, gpu=0)
    tag = 'full' if batch_size is None else f'bs{batch_size}'
    assert scores.shape == data[f'{tag}.scores'].shape
    assert scores.dtype == torch.float32 and scores.device.type == 'cuda'
    error = np.abs(scores.cpu().numpy() - data[f'{tag}.scores']).max()
    assert error < 1e-5, error
    # and against the reference's own public (bf16 autocast) answer
    if batch_size is None:
        np.testing.assert_allclose(
            scores.cpu().numpy(), data['full.scores_autocast'], atol=4e-3)


def test_preprocess_infer_postprocess_seams(emphases, golden, c1_checkpoint):
    """The inner seams other reference code calls (evaluate/core.py:85-95)"""
    data = golden('c1')
    alignment = emphases.Alignment.from_times(times_list(data['times']))
    audio = torch.from_numpy(data['audio'])
    chunks = list(emphases.preprocess(alignment, audio, 16000, 300, 0))
    assert len(chunks) == 3
    scores = []
    for i, (features, bounds) in enumerate(chunks):
        np.testing.assert_array_equal(bounds.numpy(), data[f'bs300.{i}.bounds'])
        np.testing.assert_allclose(
            features.cpu().numpy(), data[f'bs300.{i}.features'], atol=2e-5)
        logits = emphases.infer(features, bounds, c1_checkpoint)
        assert logits.shape == (1, 1, bounds.shape[-1])
        scores.append(emphases.postprocess(logits[0]))
    scores = torch.cat(scores, 1).cpu().numpy()
    assert np.abs(scores - data['bs300.scores']).max() < 1e-5
    features = emphases.data.preprocess.from_audio(audio[:, :48000], 0)
    expected = oracle.logmel(audio[:, :48000], data['mel_basis'])
    assert features.shape == (1, 80, 300)
    assert (features[0].cpu() - expected).abs().max() < 2e-5
    with pytest.raises(RuntimeError):
        emphases.data.preprocess.from_audio(audio[:, :400], 0)


@pytest.mark.parametrize('method', METHODS)
def test_downsample_api(emphases, golden, method):
    data = golden('pool')
    emphases.configure(DOWNSAMPLE_METHOD=method)
    xs = torch.from_numpy(data['xs']).cuda()
    result = emphases.downsample(
        xs, torch.from_numpy(data['clean_bounds']),
        torch.from_numpy(data['clean_lengths']))
    np.testing.assert_allclose(
        result.cpu().numpy(), data[f'clean.{method}'], rtol=1e-6, atol=1e-6)
    error = str(data[f'adversarial.{method}.error'])
    bounds = torch.from_numpy(data['bounds'])
    lengths = torch.from_numpy(data['lengths'])
    if error:
        with pytest.raises(IndexError):
            emphases.downsample(xs, bounds, lengths)
    else:
        result = emphases.downsample(xs, bounds, lengths).cpu().numpy()
        expected = data[f'adversarial.{method}']
        np.testing.assert_array_equal(np.isnan(result), np.isnan(expected))
        np.testing.assert_allclose(
            np.nan_to_num(result), np.nan_to_num(expected), rtol=1e-6, atol=1e-6)


def test_downsample_unknown_method(emphases):
    emphases.configure(DOWNSAMPLE_METHOD='median')
    with pytest.raises(ValueError):
        emphases.downsample(
            torch.zeros(1, 80, 10).cuda(), torch.zeros(1, 2, 1).long(),
            torch.ones(1).long())


def test_segment_api(emphases, golden):
    data = golden('pool')
    segments, bounds, lengths = emphases.segment(
        torch.from_numpy(data['xs']).cuda(),
        torch.from_numpy(data['clean_bounds']),
        torch.from_numpy(data['clean_lengths']))
    np.testing.assert_array_equal(
        segments.cpu().numpy(), data['segment.segments'])
    np.testing.assert_array_equal(bounds.cpu().numpy(), data['segment.bounds'])
    np.testing.assert_array_equal(lengths.cpu().numpy(), data['segment.lengths'])


def test_files_roundtrip(emphases, golden, c1_checkpoint, tmp_path):
    """from_file / from_file_to_file / from_files_to_files on wav + TextGrid"""
    data = golden('c1')
    state = state_from_golden(data)
    os.chdir(tmp_path)
    text_files, audio_files, expected = [], [], []
    for seed in range(5):
        times, audio = oracle.synthetic_utterance(700 + seed)
        # 16-bit PCM on disk: the oracle sees the same quantised samples
        wav = tmp_path / f'utt{seed}.wav'
        emphases.load.save_wav(wav, audio)
        loaded = emphases.load.audio(wav)
        grid = tmp_path / f'utt{seed}.TextGrid'
        emphases.Alignment.from_times(times).save(grid)
        reread = emphases.Alignment(grid)
        assert np.array_equal(reread.times(), np.asarray(times))
        text_files.append(grid)
        audio_files.append(wav)
        expected.append(oracle.from_alignment_and_audio(times, loaded, state))
    scores = emphases.from_file(
        text_files[0], audio_files[0], checkpoint=c1_checkpoint, gpu=0)
    assert (scores.cpu() - expected[0]).abs().max() < 1e-5
    prefixes = [tmp_path / 'out' / f'utt{seed}' for seed in range(5)]
    (tmp_path / 'out').mkdir()
    emphases.from_files_to_files(
        text_files, audio_files, prefixes, checkpoint=c1_checkpoint, gpu=0)
    for prefix, want in zip(prefixes, expected):
        got = torch.load(f'{prefix}.pt')
        assert got.shape == want.shape
        assert (got - want).abs().max() < 1e-5
        assert os.path.exists(f'{prefix}.TextGrid')
    emphases.from_file_to_file(
        text_files[1], audio_files[1], tmp_path / 'single',
        checkpoint=c1_checkpoint, gpu=0)
    got = torch.load(tmp_path / 'single.pt')
    assert (got - expected[1]).abs().max() < 1e-5


def test_multiple_launches_match_single(emphases, golden, c1_checkpoint):
    """Launch bucketing must not change results"""
    alignments, audios = [], []
    for seed in range(9):
        times, audio = oracle.synthetic_utterance(800 + seed)
        alignments.append(emphases.Alignment.from_times(times))
        audios.append(audio)
    single = emphases.from_alignments_and_audio(
        alignments, audios, 16000, c1_checkpoint, gpu=0)
    emphases.configure(MAX_ROWS_PER_LAUNCH=2500)
    split = emphases.from_alignments_and_audio(
        alignments, audios, 16000, c1_checkpoint, gpu=0)
    for a, b in zip(single, split):
        assert torch.equal(a, b)


def test_errors(emphases, golden, c1_checkpoint):
    data = golden('c1')
    alignment = emphases.Alignment.from_times(times_list(data['times']))
    audio = torch.from_numpy(data['audio'])
    emphases.configure(METHOD='bogus')
    with pytest.raises(ValueError):
        emphases.from_alignment_and_audio(alignment, audio, 16000, c1_checkpoint)
    emphases.reset_configuration()
    emphases.configure(DOWNSAMPLE_LOCATION='nowhere')
    with pytest.raises(ValueError):
        emphases.Model()
    emphases.reset_configuration()
    emphases.configure(ARCHITECTURE='lstm')
    with pytest.raises(ValueError):
        emphases.Model()


def test_files_at_other_sample_rates_take_the_packed_path(
    emphases, golden, c1_checkpoint, tmp_path
):
    """from_files_to_files on a corpus mixing 16 kHz, 24 kHz and 22.05 kHz
    wavs: every rate goes through the native reader and ONE packed GPU
    resampling launch; results equal the per-file API (which resamples like
    torchaudio, test_resample_matches_torchaudio) and the oracle"""
    import torchaudio
    data = golden('c1')
    state = state_from_golden(data)
    text_files, audio_files, expected, rates = [], [], [], []
    for seed, rate in enumerate([24000, 16000, 22050, 24000, 16000, 24000]):
        times, audio = oracle.synthetic_utterance(760 + seed, duration=1.5 + seed / 3)
        generator = torch.Generator().manual_seed(seed)
        native = 0.1 * torch.randn(
            1, int(audio.shape[-1] * rate / 16000), generator=generator)
        wav = tmp_path / f'utt{seed}.wav'
        emphases.load.save_wav(wav, native, rate)
        loaded, loaded_rate = emphases.load.wav(wav)
        assert loaded_rate == rate
        resampled = loaded if rate == 16000 else \
            torchaudio.transforms.Resample(rate, 16000)(loaded)
        grid = tmp_path / f'utt{seed}.TextGrid'
        emphases.Alignment.from_times(times).save(grid)
        text_files.append(grid)
        audio_files.append(wav)
        expected.append(oracle.from_alignment_and_audio(times, resampled, state))
        rates.append(rate)
    prefixes = [tmp_path / 'out' / f'utt{seed}' for seed in range(len(rates))]
    (tmp_path / 'out').mkdir()
    # no per-file fallback may be needed
    calls = []
    original = emphases.core.from_file_to_file
    emphases.core.from_file_to_file = lambda *a, **k: calls.append(a)
    try:
        emphases.from_files_to_files(
            text_files, audio_files, prefixes, checkpoint=c1_checkpoint, gpu=0)
    finally:
        emphases.core.from_file_to_file = original
    assert not calls
    for index, (prefix, want) in enumerate(zip(prefixes, expected)):
        got = torch.load(f'{prefix}.pt')
        assert got.shape == want.shape
        assert (got - want).abs().max() < 2e-5, rates[index]
        single = emphases.from_file(
            text_files[index], audio_files[index], checkpoint=c1_checkpoint, gpu=0)
        assert (got - single.cpu()).abs().max() < 2e-6
        assert os.path.exists(f'{prefix}.TextGrid')


def test_list_api_streams_and_narrows_losslessly(emphases, golden, c1_checkpoint):
    """from_alignments_and_audio on a list of CPU tensors: packed launch by
    launch in the background; 16-bit-PCM-valued audio travels as int16 and
    gives bit-identical scores to the fp32 upload"""
    from emphases_b200 import scheduler
    data = golden('c1')
    state = state_from_golden(data)
    alignments, audios, expected = [], [], []
    for seed in range(6):
        times, audio = oracle.synthetic_utterance(820 + seed, duration=1.5 + seed / 2)
        audio = (audio * 32768.).round().clamp(-32768, 32767) / 32768.   # PCM values
        alignments.append(emphases.Alignment.from_times(times))
        audios.append(audio)
        expected.append(oracle.from_alignment_and_audio(times, audio, state))
    emphases.configure(MAX_ROWS_PER_LAUNCH=600)          # several launches
    seen = []
    original = scheduler.StreamedPack.launch_source

    def spy(self, number, first, last):
        source = original(self, number, first, last)
        seen.append(source.dtype)
        return source

    scheduler.StreamedPack.launch_source = spy
    try:
        narrow = emphases.from_alignments_and_audio(
            alignments, audios, 16000, checkpoint=c1_checkpoint, gpu=0)
        assert len(seen) > 1 and all(dtype == torch.int16 for dtype in seen)
        seen.clear()
        noisy = [audio.clone() for audio in audios]
        noisy[3][0, 5000] += 1e-5                        # one launch cannot narrow
        mixed = emphases.from_alignments_and_audio(
            alignments, noisy, 16000, checkpoint=c1_checkpoint, gpu=0)
        assert torch.float32 in seen and torch.int16 in seen
    finally:
        scheduler.StreamedPack.launch_source = original
    packed = scheduler.pack_audio(audios)
    plain = emphases.from_alignments_and_audio(
        alignments, packed, 16000, checkpoint=c1_checkpoint, gpu=0)
    for got, same, other, want in zip(narrow, plain, mixed, expected):
        assert torch.equal(got, same)
        assert (got - want).abs().max() < 1e-5
        assert (other - want).abs().max() < 1e-4


def test_batched_api_edge_cases(emphases, golden, c1_checkpoint):
    """Empty list, an utterance too short to yield a chunk (dropped like
    emphases/core.py:413-415), stereo (channel 0 is used, mels.py:48),
    float64 and CUDA inputs, a zero-length word under `sum`, chunked and
    resampled inputs -- all through the list API in one call each"""
    data = golden('c1')
    state = state_from_golden(data)
    make = emphases.Alignment.from_times
    generator = torch.Generator().manual_seed(4)
    run = lambda alignments, audios, rate=16000, **kw: emphases.from_alignments_and_audio(
        alignments, audios, rate, checkpoint=c1_checkpoint, gpu=0, **kw)
    assert run([], []) == []
    times = [(0., .4), (.4, .4), (.4, 1.1), (1.1, 2.)]          # one empty word
    audio = 0.1 * torch.randn(1, 32000, generator=generator)
    want = oracle.from_alignment_and_audio(times, audio, state)
    short = 0.1 * torch.randn(1, 400, generator=generator)
    got = run([make([(0., .02)]), make(times)], [short, audio])
    assert got[0].shape == (1, 0)
    assert (got[1] - want).abs().max() < 1e-5
    stereo = torch.cat([audio, -audio])
    for variant in (stereo, audio.double(), audio.cuda()):
        both = run([make(times)] * 2, [variant] * 2)
        assert all((b - want).abs().max() < 1e-5 for b in both)
    chunked = run([make(times)] * 2, [audio] * 2, batch_size=60)
    want_chunked = oracle.from_alignment_and_audio(times, audio, state, batch_size=60)
    assert all((c - want_chunked).abs().max() < 1e-5 for c in chunked)
    native = 0.1 * torch.randn(1, 48000, generator=generator)
    import torchaudio
    want_24k = oracle.from_alignment_and_audio(
        times, torchaudio.transforms.Resample(24000, 16000)(native), state)
    assert all((r - want_24k).abs().max() < 2e-5
               for r in run([make(times)] * 2, [native] * 2, 24000))


def test_transformer_variant(emphases, golden):
    """ARCHITECTURE='transformer' Model.forward vs the reference (B=1 and a
    padded B=2 batch whose key-padding mask matters)"""
    data = golden('transformer')
    emphases.configure(ARCHITECTURE='transformer')
    model = emphases.Model()
    state = state_from_golden(data)
    missing = model.load_state_dict(state, strict=False)
    assert all('position.encoding' in key for key in missing.missing_keys)
    assert not missing.unexpected_keys
    model = model.cuda().eval()
    with torch.no_grad():
        features = torch.from_numpy(data['b1.features']).cuda()
        bounds = torch.from_numpy(data['b1.bounds'])
        logits = model(
            features, torch.tensor([features.shape[-1]]), bounds,
            torch.tensor([bounds.shape[-1]]))
        np.testing.assert_allclose(
            logits.cpu().numpy(), data['b1.logits'], rtol=0, atol=3e-5)
        batch = [torch.from_numpy(data[f'b2.{name}']) for name in (
            'features', 'frame_lengths', 'bounds', 'word_lengths')]
        batch[0] = batch[0].cuda()
        logits = model(*batch).cpu().numpy()
        for i, words in enumerate(batch[3].tolist()):
            np.testing.assert_allclose(
                logits[i, :, :words], data['b2.logits'][i, :, :words],
                rtol=0, atol=3e-5)


@pytest.mark.parametrize('location', ['loss', 'inference'])
def test_transformer_variant_without_word_decoder(emphases, golden, location):
    """Transformer variant at the locations that have no word decoder, vs the
    oracle in fp64 on the golden weights (B=1 and the padded B=2 batch), and
    at 'inference' the training-mode frame logits over the valid frames"""
    data = golden('transformer')
    emphases.configure(ARCHITECTURE='transformer', DOWNSAMPLE_LOCATION=location)
    model = emphases.Model()
    own = model.state_dict()
    missing = model.load_state_dict(
        {k: v for k, v in state_from_golden(data).items() if k in own},
        strict=False)
    assert all('position.encoding' in key for key in missing.missing_keys)
    model = model.cuda().eval()
    # the golden state has no position.encoding; the model's buffer supplies it
    reference = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    config = {'ARCHITECTURE': 'transformer', 'DOWNSAMPLE_LOCATION': location}
    features = torch.from_numpy(data['b1.features'])
    bounds = torch.from_numpy(data['b1.bounds'])
    b1 = [features, torch.tensor([features.shape[-1]]), bounds,
          torch.tensor([bounds.shape[-1]])]
    b2 = [torch.from_numpy(data[f'b2.{name}']) for name in (
        'features', 'frame_lengths', 'bounds', 'word_lengths')]
    cases = [(b1, False), (b2, False)] + [(b2, True)] * (location == 'inference')
    for batch, training in cases:
        model.train(training)
        with torch.no_grad():
            logits = model(batch[0].cuda(), *batch[1:]).cpu().numpy()
        expected = oracle.model_forward(
            reference, batch[0].double(), *batch[1:], config=config,
            training=training).numpy()
        assert logits.shape == expected.shape
        # The 'sum'-pooled word logits reach |52| on this batch; fp32
        # summation order alone moves them by 5.5e-5 from fp64 (1e-6
        # relative, B200).  Hence the rtol of test_model_forward_sweep.
        valid = batch[1] if training else batch[3]
        for i, count in enumerate(valid.tolist()):
            np.testing.assert_allclose(
                logits[i, :, :count], expected[i, :, :count], rtol=1e-5, atol=3e-5)


def test_transformer_variant_input_location(emphases, golden):
    """Transformer variant at DOWNSAMPLE_LOCATION='input' vs the reference
    (B=1 and a padded B=2 batch): attention runs inside each word segment"""
    data = golden('transformer_input')
    emphases.configure(ARCHITECTURE='transformer', DOWNSAMPLE_LOCATION='input')
    model = emphases.Model()
    state = state_from_golden(data)
    missing = model.load_state_dict(state, strict=False)
    assert all('position.encoding' in key for key in missing.missing_keys)
    assert not missing.unexpected_keys
    model = model.cuda().eval()
    with torch.no_grad():
        features = torch.from_numpy(data['b1.features']).cuda()
        bounds = torch.from_numpy(data['b1.bounds'])
        logits = model(
            features, torch.tensor([features.shape[-1]]), bounds,
            torch.tensor([bounds.shape[-1]]))
        np.testing.assert_allclose(
            logits.cpu().numpy(), data['b1.logits'], rtol=0, atol=3e-5)
        batch = [torch.from_numpy(data[f'b2.{name}']) for name in (
            'features', 'frame_lengths', 'bounds', 'word_lengths')]
        batch[0] = batch[0].cuda()
        logits = model(*batch).cpu().numpy()
        for i, words in enumerate(batch[3].tolist()):
            np.testing.assert_allclose(
                logits[i, :, :words], data['b2.logits'][i, :, :words],
                rtol=0, atol=3e-5)


def test_transformer_variant_linear_maps_on_tensor_cores(emphases, golden):
    """With a tensor-core PRECISION the Transformer variant's per-row linear
    maps (kernel-size-1 stacks: QKV, output projection, feed-forward) run in
    the fp32-grade bf16x6 tcgen05 mode and attention in the split-bf16
    tensor-core form.  Same parity bar as the all-fp32 path."""
    data = golden('transformer')
    emphases.configure(ARCHITECTURE='transformer', PRECISION='bf16x6')
    model = emphases.Model()
    model.load_state_dict(state_from_golden(data), strict=False)
    model = model.cuda().eval()
    with torch.no_grad():
        batch = [torch.from_numpy(data[f'b2.{name}']) for name in (
            'features', 'frame_lengths', 'bounds', 'word_lengths')]
        batch[0] = batch[0].cuda()
        logits = model(*batch).cpu().numpy()
        for i, words in enumerate(batch[3].tolist()):
            np.testing.assert_allclose(
                logits[i, :, :words], data['b2.logits'][i, :, :words],
                rtol=0, atol=3e-5)


# logits; the 'bf16' bar is the 2e-3 score tolerance (sigmoid slope <= 1/4)
TRANSFORMER_TC_TOLERANCE = {'bf16': 8e-3, 'bf16x3': 1e-4}


@pytest.mark.parametrize('precision', ['bf16', 'bf16x3'])
@pytest.mark.parametrize('location', ['intermediate', 'input'])
def test_transformer_variant_tensor_core_attention(emphases, golden, precision, location):
    """PRECISION 'bf16' / 'bf16x3': attention itself runs on the tensor cores
    (fp16 / split-bf16 operands, csrc/attention_tc.cu), vs the reference logits"""
    from emphases_b200 import transformer
    data = golden('transformer' if location == 'intermediate' else 'transformer_input')
    emphases.configure(
        ARCHITECTURE='transformer', PRECISION=precision, DOWNSAMPLE_LOCATION=location)
    expected_mode = {'bf16': 'fp16', 'bf16x3': 'bf16x3'}[precision]
    assert transformer.attention_mode() == transformer.ATTENTION_MODES[expected_mode]
    model = emphases.Model()
    model.load_state_dict(state_from_golden(data), strict=False)
    model = model.cuda().eval()
    with torch.no_grad():
        batch = [torch.from_numpy(data[f'b2.{name}']) for name in (
            'features', 'frame_lengths', 'bounds', 'word_lengths')]
        batch[0] = batch[0].cuda()
        logits = model(*batch).cpu().numpy()
        for i, words in enumerate(batch[3].tolist()):
            error = np.abs(logits[i, :, :words] - data['b2.logits'][i, :, :words]).max()
            print(f'{precision} {location} utterance {i}: max |logit error| {error:.3e}')
            assert error < TRANSFORMER_TC_TOLERANCE[precision]


def test_transformer_end_to_end(emphases, golden, tmp_path):
    """from_alignment_and_audio with the transformer variant vs the oracle"""
    data = golden('transformer')
    emphases.configure(ARCHITECTURE='transformer')
    state = state_from_golden(data)
    encoding = oracle.positional_encoding(80)
    state['frame_encoder.position.encoding'] = encoding
    state['word_decoder.position.encoding'] = encoding
    path = tmp_path / 'transformer.pt'
    torch.save({'model': state}, path)
    times, audio = oracle.synthetic_utterance(31, duration=4.0, words=9)
    scores = emphases.from_alignment_and_audio(
        emphases.Alignment.from_times(times), audio, 16000, checkpoint=path,
        gpu=0)
    expected = oracle.from_alignment_and_audio(
        times, audio, state, config={'ARCHITECTURE': 'transformer'})
    assert scores.shape == expected.shape
    assert (scores.cpu() - expected).abs().max() < 2e-5


def test_transformer_packed_corpus(emphases, golden, tmp_path):
    """Several ragged utterances through the packed transformer path"""
    data = golden('transformer')
    emphases.configure(ARCHITECTURE='transformer')
    state = state_from_golden(data)
    encoding = oracle.positional_encoding(80)
    state['frame_encoder.position.encoding'] = encoding
    state['word_decoder.position.encoding'] = encoding
    path = tmp_path / 'transformer.pt'
    torch.save({'model': state}, path)
    alignments, audios, expected = [], [], []
    for seed in range(4):
        times, audio = oracle.synthetic_utterance(900 + seed, duration=2.0 + seed)
        alignments.append(emphases.Alignment.from_times(times))
        audios.append(audio)
        expected.append(oracle.from_alignment_and_audio(
            times, audio, state, config={'ARCHITECTURE': 'transformer'}))
    scores = emphases.from_alignments_and_audio(
        alignments, audios, 16000, checkpoint=path, gpu=0)
    for got, want in zip(scores, expected):
        assert got.shape == want.shape
        assert (got - want).abs().max() < 2e-5


HPARAMS = [
    # the reference's config/hparam-search space (SURVEY.md A.1)
    dict(CHANNELS=64),
    dict(CHANNELS=128),
    dict(CHANNELS=128, ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=1),
    dict(LAYERS=5),
    dict(LAYERS=7),
    dict(ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=7),
    dict(ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=1),
    dict(ACTIVATION_FUNCTION=torch.nn.GELU),
    dict(ACTIVATION_FUNCTION=torch.nn.LeakyReLU),
    dict(ACTIVATION_FUNCTION=torch.nn.SiLU),
    dict(DROPOUT=.1),
    dict(LOSS='mse'),
]


@pytest.mark.parametrize('overrides', HPARAMS, ids=lambda d: '-'.join(map(str, d)))
def test_hyperparameter_shapes(emphases, overrides):
    """Model shapes of the reference's hyper-parameter sweep, random init,
    against the oracle (fp32 mode, end to end from audio)"""
    emphases.configure(**overrides)
    torch.manual_seed(3)
    model = emphases.Model()
    for parameter in model.parameters():
        if parameter.dim() > 1:
            parameter.data.mul_(1.5)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().eval()
    activation = emphases.ACTIVATION_FUNCTION.__name__
    config = dict(
        CHANNELS=emphases.CHANNELS, LAYERS=emphases.LAYERS,
        DROPOUT=emphases.DROPOUT, LOSS=emphases.LOSS,
        ACTIVATION={'ReLU': 'relu', 'GELU': 'gelu', 'LeakyReLU': 'leaky_relu',
                    'SiLU': 'silu'}[activation])
    alignments, audios, expected = [], [], []
    for seed in range(3):
        times, audio = oracle.synthetic_utterance(1200 + seed, duration=2.5 + seed)
        alignments.append(emphases.Alignment.from_times(times))
        audios.append(audio)
        expected.append(oracle.from_alignment_and_audio(times, audio, state, config))
    scores = emphases.from_alignments_and_audio(
        alignments, audios, 16000, model=model, gpu=0)
    for got, want in zip(scores, expected):
        assert got.shape == want.shape
        assert (got - want).abs().max() < 1e-5


@pytest.mark.parametrize('channels', [64, 128])
def test_transformer_other_widths_fail_loudly(emphases, channels):
    """The Transformer variant is built for the default width (its LayerNorm
    and head split cannot be zero-padded the way the conv stacks are); another
    CHANNELS raises instead of computing something else"""
    emphases.configure(ARCHITECTURE='transformer', CHANNELS=channels)
    model = emphases.Model().cuda().eval()
    with pytest.raises(NotImplementedError):
        model.packed_weights()


def test_wide_model_is_rejected_loudly(emphases):
    emphases.configure(CHANNELS=256)
    model = emphases.Model().cuda().eval()
    with pytest.raises(NotImplementedError):
        model.packed_weights()


@pytest.mark.parametrize('rate', [24000, 44100, 8000])
def test_resample_matches_torchaudio(emphases, rate):
    """emphases.resample vs torchaudio.transforms.Resample on CPU"""
    import torchaudio
    generator = torch.Generator().manual_seed(rate)
    audio = 0.3 * torch.randn(2, rate + 37, generator=generator)
    expected = torchaudio.transforms.Resample(rate, 16000)(audio)
    got = emphases.resample(audio.cuda(), rate)
    assert got.shape == expected.shape and got.device.type == 'cuda'
    assert (got.cpu() - expected).abs().max() < 2e-6
    assert emphases.resample(audio, rate).device.type == 'cpu'
    assert emphases.resample(audio, 16000) is audio


def test_non_16k_audio_end_to_end(emphases, golden, c1_checkpoint):
    """from_alignment_and_audio resamples like the reference (core.py:353-354)"""
    import torchaudio
    data = golden('c1')
    state = state_from_golden(data)
    generator = torch.Generator().manual_seed(4)
    audio = 0.1 * torch.randn(1, 72000, generator=generator)          # 3 s at 24 kHz
    times = oracle.synthetic_alignment(3.0, 8, generator)
    expected = oracle.from_alignment_and_audio(
        times, torchaudio.transforms.Resample(24000, 16000)(audio), state)
    scores = emphases.from_alignment_and_audio(
        emphases.Alignment.from_times(times), audio, 24000,
        checkpoint=c1_checkpoint, gpu=0)
    assert (scores.cpu() - expected).abs().max() < 1e-5


@pytest.mark.parametrize('method,location', [
    ('sum', 'intermediate'), ('average', 'intermediate'), ('max', 'loss'),
    ('center', 'inference')])
def test_single_utterance_native_call_matches_batched_path(
    emphases, golden, c1_checkpoint, method, location
):
    """emph_infer_utterance (one native call: C++ chunk plan + seven launches)
    must give bit for bit what the batched scheduler gives, for host and
    device audio; what it declines falls back to the general path"""
    from emphases_b200 import single
    emphases.configure(DOWNSAMPLE_METHOD=method, DOWNSAMPLE_LOCATION=location)
    device = torch.device('cuda', 0)
    torch.manual_seed(3)
    model = emphases.Model().to(device).eval()
    for seed in range(5):
        times, audio = oracle.synthetic_utterance(900 + seed, duration=0.8 + 1.7 * seed)
        alignment = emphases.Alignment.from_times(times)
        forms = {'host': audio, 'device': audio.to(device), 'flat': audio[0].clone()}
        for name, form in forms.items():
            fast = single.from_alignment_and_audio(model, alignment, form, 16000, device)
            assert fast is not None, name
            slow = emphases.from_alignments_and_audio(
                [alignment], [form.reshape(1, -1)], 16000, model=model, gpu=0,
                to_cpu=False)[0]
            assert fast.shape == slow.shape == (1, len(times))
            assert torch.equal(fast, slow), (method, location, seed, name)
    # the public entry point takes the native call ...
    times, audio = oracle.synthetic_utterance(950)
    alignment = emphases.Alignment.from_times(times)
    expected = oracle.from_alignment_and_audio(
        times, audio, {k: v.detach().cpu() for k, v in model.state_dict().items()},
        {'DOWNSAMPLE_METHOD': method, 'DOWNSAMPLE_LOCATION': location})
    checkpoint = c1_checkpoint.parent / f'single_{method}_{location}.pt'
    torch.save({'model': model.state_dict()}, checkpoint)
    got = emphases.from_alignment_and_audio(alignment, audio, 16000, checkpoint, gpu=0)
    assert (got.cpu() - expected).abs().max() < 1e-5
    # ... and what the native planner declines (other sample rates, chunked
    # calls, stereo) still goes through the general path
    assert single.from_alignment_and_audio(model, alignment, audio, 22050, device) is None
    assert single.from_alignment_and_audio(
        model, alignment, torch.cat([audio, audio]), 16000, device) is None
    chunked = emphases.from_alignment_and_audio(
        alignment, audio, 16000, checkpoint, batch_size=120, gpu=0)
    assert chunked.shape == got.shape
