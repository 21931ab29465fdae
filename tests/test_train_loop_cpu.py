"""CPU tests of the training loop's host side: dataset reading from the cache
layout, the per-rank epoch schedule, checkpoint selection and the gather
kernel's build."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from synthetic_cache import write_cache

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def emphases():
    import emphases_b200
    emphases_b200.reset_configuration()
    yield emphases_b200
    emphases_b200.reset_configuration()


@pytest.fixture
def cache(emphases, tmp_path):
    partitions = write_cache(
        tmp_path, 'synthetic', {'train': 6, 'valid': 2, 'test': 1}, seconds=(1., 3.))
    emphases.configure(
        CACHE_DIR=tmp_path / 'cache', PARTITION_DIR=tmp_path / 'partitions')
    return tmp_path, partitions


def test_dataset_reads_partition_bounds_lengths_and_buckets(emphases, cache):
    root, partitions = cache
    dataset = emphases.data.Dataset('synthetic', 'train')
    assert dataset.stems == partitions['train']
    assert len(dataset) == 6
    for i, stem in enumerate(dataset.stems):
        alignment = emphases.Alignment(
            root / 'cache' / 'synthetic' / 'alignment' / f'{stem}.TextGrid')
        want = alignment.word_bounds(
            emphases.SAMPLE_RATE, emphases.HOPSIZE, silences=True)
        start, count = int(dataset.word_start[i]), int(dataset.n_words[i])
        assert [tuple(b) for b in dataset.bounds[start:start + count].tolist()] == want
        audio, rate = emphases.load.wav(
            root / 'cache' / 'synthetic' / 'audio' / f'{stem}.wav')
        assert rate == emphases.SAMPLE_RATE
        assert dataset.lengths[i] == audio.shape[-1] // emphases.HOPSIZE
        scores = torch.load(root / 'cache' / 'synthetic' / 'scores' / f'{stem}.pt')
        assert torch.equal(dataset.targets[start:start + count], scores)
    got = dataset.buckets()
    want = emphases.data.buckets(dataset.lengths)
    assert len(got) == len(want) == emphases.BUCKETS
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)
    # several datasets concatenate in order
    both = emphases.data.Dataset(['synthetic', 'synthetic'], 'valid')
    assert both.stems == partitions['valid'] * 2
    # a later read leaves the audio of an earlier dataset as it was
    for i, stem in enumerate(dataset.stems):
        audio, _ = emphases.load.wav(
            root / 'cache' / 'synthetic' / 'audio' / f'{stem}.wav', normalize=False)
        offset, samples = int(dataset.audio_offsets[i]), int(dataset.samples[i])
        assert torch.equal(dataset.audio[offset:offset + samples], audio[0])


def test_dataset_errors_name_the_file(emphases, cache):
    root, partitions = cache
    with pytest.raises(KeyError, match='synthetic.json'):
        emphases.data.Dataset('synthetic', 'evaluation')

    stem = partitions['train'][1]
    scores = root / 'cache' / 'synthetic' / 'scores' / f'{stem}.pt'
    saved = torch.load(scores)
    torch.save(saved[:-1], scores)
    with pytest.raises(ValueError, match=stem):
        emphases.data.Dataset('synthetic', 'train')
    torch.save(saved, scores)

    stem = partitions['valid'][0]
    audio = root / 'cache' / 'synthetic' / 'audio' / f'{stem}.wav'
    samples, _ = emphases.load.wav(audio)
    emphases.load.save_wav(audio, samples, 22050)
    with pytest.raises(ValueError, match=f'{stem}.wav'):
        emphases.data.Dataset('synthetic', 'valid')


def test_short_file_raises_naming_the_stem(emphases):
    with pytest.raises(RuntimeError, match='stem-b: Padding size'):
        emphases.engine.feature_plan([1000, 432, 500], ['stem-a', 'stem-b', 'stem-c'])
    with pytest.raises(RuntimeError, match='^Padding size'):
        emphases.engine.feature_plan([432])


def test_feature_plan_layout(emphases):
    lengths = np.array([16000, 433, 4001])
    plan = emphases.engine.feature_plan(lengths)
    np.testing.assert_array_equal(plan.n_rows, lengths // 160)
    np.testing.assert_array_equal(plan.chunk_start, [432] * 3)
    np.testing.assert_array_equal(plan.chunk_len, lengths)
    np.testing.assert_array_equal(plan.audio_len, lengths)
    np.testing.assert_array_equal(plan.row_start, [1, 102, 105])
    assert plan.total_rows == 105 + 25 + 1
    offsets, _ = emphases.scheduler.PackedAudio.layout(lengths)
    np.testing.assert_array_equal(plan.audio_off, offsets)
    assert np.all(plan.audio_off % emphases.engine.AUDIO_ALIGN == 0)


@pytest.mark.parametrize('world', range(1, 9))
def test_rank_schedule_equal_disjoint_ordered(emphases, golden, world):
    from emphases_b200.train import rank_batches
    data = golden('sampler')
    for name in ('a', 'b', 'c'):
        lengths = data[f'{name}/lengths']
        sampler = emphases.data.Sampler(
            emphases.data.LengthDataset(lengths), int(data[f'{name}/max_frames']))
        for epoch in (0, 1, 3):
            sampler.set_epoch(epoch)
            batches = [list(map(int, b)) for b in sampler.batch()]
            shares = [rank_batches(batches, rank, world) for rank in range(world)]
            assert len({len(share) for share in shares}) == 1
            assert len(shares[0]) == len(batches) // world
            seen = [tuple(b) for share in shares for b in share]
            assert len(seen) == len(set(seen)) == len(shares[0]) * world
            for share in shares:
                positions = [batches.index(b) for b in share]
                assert positions == sorted(positions)


def test_checkpoint_keys_and_resume_selection(emphases, tmp_path, monkeypatch):
    from emphases_b200.train import checkpoints, latest_checkpoint
    assert latest_checkpoint(tmp_path) is None
    for step in (100, 2000, 300):
        torch.save({'step': step}, tmp_path / f'{step:08d}.pt')
    torch.save({'step': -1}, tmp_path / 'best.pt')
    assert [p.name for p in checkpoints(tmp_path)] == [
        '00000100.pt', '00000300.pt', '00002000.pt']
    assert latest_checkpoint(tmp_path).name == '00002000.pt'

    # the loop's checkpoint is the released checkpoint's keys + rng, and
    # load_model's reading of it ('model') takes it as it is
    from emphases_b200.train import checkpoint_state
    model = emphases.Model()
    optimizer = torch.optim.Adam(model.parameters(), lr=emphases.LEARNING_RATE)
    cuda_state = torch.zeros(16, dtype=torch.uint8)
    monkeypatch.setattr(torch.cuda, 'get_rng_state', lambda device: cuda_state)
    state = checkpoint_state(model, optimizer, 2, 300, 0.25, 0.5, 'cuda:0')
    assert set(state) == {'model', 'optimizer', 'epoch', 'step', 'score', 'best', 'rng'}
    assert (state['epoch'], state['step'], state['score'], state['best']) == (2, 300, .25, .5)
    assert torch.equal(state['rng']['cpu'], torch.get_rng_state())
    assert state['rng']['cuda'] is cuda_state
    file = tmp_path / 'best.pt'
    torch.save(state, file)
    loaded = emphases.Model()
    state = torch.load(file, weights_only=False)
    loaded.load_state_dict(state['model'])
    for a, b in zip(model.state_dict().values(), loaded.state_dict().values()):
        assert torch.equal(a, b)


def test_training_configuration_defaults(emphases):
    assert emphases.NUM_STEPS == 6000
    assert emphases.EVALUATION_INTERVAL == 100
    assert emphases.LEARNING_RATE == 1e-3


def test_cli_help():
    result = subprocess.run(
        [os.sys.executable, '-m', 'emphases_b200.train', '--help'],
        cwd=ROOT, capture_output=True, text=True)
    assert result.returncode == 0, result.stderr
    for flag in ('--config', '--datasets', '--directory', '--gpu'):
        assert flag in result.stdout


def test_gather_kernel_has_no_spills(tmp_path):
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    if not os.path.exists(nvcc):
        pytest.skip('nvcc is not installed')
    result = subprocess.run(
        [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17',
         '-Xptxas=-v', '-c', os.path.join(ROOT, 'emphases_b200', 'csrc', 'batch.cu'),
         '-o', str(tmp_path / 'batch.o')],
        capture_output=True, text=True)
    assert result.returncode == 0, result.stderr
    report = result.stdout + result.stderr
    assert 'gather_batch_kernel' in report
    spills = re.findall(r'(\d+) bytes spill stores, (\d+) bytes spill loads', report)
    assert spills and all(int(a) == 0 and int(b) == 0 for a, b in spills)
