"""The training loop on the GPU: resident features, the on-device collate
(emph_gather_batch), loop steps against a hand-written loop of train_step,
resume, validation metrics, checkpoints, the command line and two-GPU data
parallelism."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import emphases_oracle as oracle
from synthetic_cache import write_cache

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNTS = {'train': 32, 'valid': 8, 'test': 2}


@pytest.fixture(scope='module')
def cache_root(tmp_path_factory):
    root = tmp_path_factory.mktemp('cache')
    write_cache(root, 'synthetic', COUNTS, seed=3, seconds=(1., 3.5))
    return root


@pytest.fixture
def emphases(cache_root):
    import emphases_b200
    emphases_b200.reset_configuration()
    emphases_b200.configure(
        CACHE_DIR=cache_root / 'cache', PARTITION_DIR=cache_root / 'partitions')
    yield emphases_b200
    emphases_b200.reset_configuration()


@pytest.fixture
def recorder(emphases, monkeypatch):
    """Every train_step call's CPU generator state (dropout seeds are drawn
    from it) and batch, on the host"""
    calls = []
    original = emphases.training.train_step

    def record(model, optimizer, batch):
        calls.append((torch.get_rng_state(), [t.cpu() for t in batch[:5]]))
        return original(model, optimizer, batch)
    monkeypatch.setattr(emphases.training, 'train_step', record)
    return calls


def assert_same_calls(a, b):
    assert len(a) == len(b)
    for (state_a, batch_a), (state_b, batch_b) in zip(a, b):
        assert torch.equal(state_a, state_b)
        for x, y in zip(batch_a, batch_b):
            assert x.dtype == y.dtype and torch.equal(x, y)


def spread_bound(states, key=lambda state: state):
    """Four times the largest difference between runs that should agree: the
    weight-gradient kernels accumulate with atomics, so identical runs may
    differ and Adam lets the differences grow"""
    return 4 * max(
        largest_difference(key(a), key(b))
        for i, a in enumerate(states) for b in states[i + 1:])


def state_of(directory, step):
    return torch.load(directory / f'{step:08d}.pt', map_location='cpu', weights_only=False)


def assert_same_state(a, b):
    assert a.keys() == b.keys()
    for key in a:
        assert torch.equal(a[key], b[key]), key


def largest_difference(a, b):
    return max((a[key].cpu() - b[key].cpu()).abs().max().item() for key in a)


def hand_loop(emphases, steps):
    """train_step on collate batches in the sampler's order, on a model built
    as the loop builds it"""
    dataset = emphases.data.Dataset('synthetic', 'train')
    torch.manual_seed(emphases.RANDOM_SEED)
    model = emphases.Model().cuda()
    optimizer = torch.optim.Adam(model.parameters(), lr=emphases.LEARNING_RATE)
    sampler = emphases.data.Sampler(dataset)
    step, epoch = 0, 0
    while step < steps:
        sampler.set_epoch(epoch)
        for indices in sampler.batch():
            batch = emphases.data.collate([dataset[i] for i in indices])[:5]
            batch = (batch[0].cuda(),) + batch[1:4] + (batch[4].cuda(),)
            emphases.training.train_step(model, optimizer, batch)
            step += 1
            if step == steps:
                break
        epoch += 1
    return model, optimizer


def test_resident_features_equal_from_audio_and_oracle(emphases):
    dataset = emphases.data.Dataset('synthetic', 'train')
    for i in range(len(dataset)):
        audio = dataset[i][4]
        resident = dataset.features(i)
        single = emphases.data.preprocess.mels.from_audio(audio.cuda())
        assert resident.shape == single.shape == (80, audio.shape[-1] // 160)
        assert torch.equal(resident, single), dataset.stems[i]
        expected = oracle.logmel(audio)
        assert (resident.cpu() - expected).abs().max().item() < 2e-5
    rows = dataset.resident()['rows']
    for start in dataset.plan.row_start:
        assert rows[start - 1].abs().max().item() == 0       # separator rows


def test_batch_equals_collate_with_every_element_written(emphases):
    dataset = emphases.data.Dataset('synthetic', 'train')
    frames, words = dataset.lengths, dataset.n_words
    longest = int(np.argmax(frames))
    wordiest = int(np.argmax(np.where(np.arange(len(frames)) == longest, -1, words)))
    assert frames[longest] % 32 != 0
    other = [i for i in range(len(dataset)) if i not in (longest, wordiest)]
    cases = [
        [longest],                                  # B = 1
        [wordiest, other[0], longest],              # Wmax and Tmax from different items
        [other[3], other[1]],
        other[:12]]
    for indices in cases:
        batch = dataset.batch(indices)
        torch.cuda.synchronize()
        workspace = dataset.resident()['workspace']
        for name in ('batch_features', 'batch_targets'):
            workspace.buffers[name].fill_(float('nan'))
        batch = dataset.batch(indices)
        want = emphases.data.collate([dataset[i] for i in indices])[:5]
        assert batch[0].is_cuda and batch[4].is_cuda
        assert not batch[1].is_cuda and batch[2].dtype == torch.int64
        for got, expected in zip(batch, want):
            assert got.shape == expected.shape and got.dtype == expected.dtype
            assert torch.equal(got.cpu(), expected)
        # padding is exactly zero (and the NaN fill is gone everywhere)
        assert not torch.isnan(batch[0]).any() and not torch.isnan(batch[4]).any()
        for b, i in enumerate(indices):
            assert batch[0][b, :, int(frames[i]):].abs().sum().item() == 0
            assert batch[4][b, :, int(words[i]):].abs().sum().item() == 0


def test_loop_equals_hand_loop_and_loss_falls(emphases, tmp_path, recorder):
    emphases.configure(NUM_STEPS=50, EVALUATION_INTERVAL=10)
    model = emphases.train(['synthetic'], tmp_path)
    final = state_of(tmp_path, 50)
    assert_same_state(final['model'], {k: v.cpu() for k, v in model.state_dict().items()})
    loop_calls = recorder[:]
    # a hand-written loop of train_step on collate batches in the sampler's
    # order takes exactly the loop's batches, bit for bit
    hands = []
    for _ in range(3):
        del recorder[:]
        hands.append(hand_loop(emphases, 50)[0].state_dict())
        assert_same_calls(loop_calls, recorder)
    # and reaches the same weights: bit for bit where the hand loops agree bit
    # for bit, else within their spread
    assert largest_difference(final['model'], hands[0]) <= spread_bound(hands)
    log = [json.loads(line) for line in open(tmp_path / 'log.jsonl')]
    assert [line['step'] for line in log] == [10, 20, 30, 40, 50]
    assert log[-1]['train_loss'] < log[0]['train_loss']
    assert all(line['ms_per_step'] > 0 for line in log)

    # the logged metrics are evaluate.metrics over the valid batches
    valid = emphases.data.Dataset('synthetic', 'valid')
    for line in (log[0], log[-1]):
        state = state_of(tmp_path, line['step'])
        check = emphases.Model().cuda()
        check.load_state_dict(state['model'])
        check.eval()
        outputs = []
        predicted = emphases.evaluate.metrics.Statistics()
        target = emphases.evaluate.metrics.Statistics()
        with torch.no_grad():
            for indices in emphases.data.sampler(valid, 'valid'):
                features, frame_lengths, bounds, lengths, targets = \
                    emphases.data.collate([valid[i] for i in indices])[:5]
                logits = check(features.cuda(), frame_lengths, bounds, lengths)
                outputs.append((logits, targets, lengths))
                predicted.update(torch.sigmoid(logits), lengths)
                target.update(targets, lengths)
        metrics = emphases.evaluate.metrics.Metrics(predicted, target)
        for logits, targets, lengths in outputs:
            metrics.update(logits, targets, lengths)
        result = metrics()
        assert line['valid_loss'] == pytest.approx(result['bce'], rel=1e-9)
        assert line['pearson_correlation'] == pytest.approx(
            result['pearson_correlation'], rel=1e-9)
        assert state['score'] == line['pearson_correlation']
    best = torch.load(tmp_path / 'best.pt', weights_only=False)
    top = max(log, key=lambda line: line['pearson_correlation'])
    assert best['step'] == top['step']
    assert best['best'] == top['pearson_correlation'] == final['best']

    # inference from best.pt equals a model loaded from the saved state dict
    cache = emphases.CACHE_DIR / 'synthetic'
    stems = json.load(open(emphases.PARTITION_DIR / 'synthetic.json'))['test']
    text = [cache / 'alignment' / f'{s}.TextGrid' for s in stems]
    audio = [cache / 'audio' / f'{s}.wav' for s in stems]
    torch.save(best['model'], tmp_path / 'state_dict.pt')
    outputs = []
    for checkpoint in ('best.pt', 'state_dict.pt'):
        prefixes = [tmp_path / f'{checkpoint}-{s}' for s in stems]
        emphases.from_files_to_files(text, audio, prefixes, checkpoint=tmp_path / checkpoint)
        outputs.append([torch.load(f'{p}.pt') for p in prefixes])
    for a, b in zip(*outputs):
        assert torch.equal(a, b)


@pytest.mark.parametrize('dropout', [None, 0.1])
def test_resume_equals_uninterrupted(emphases, tmp_path, recorder, dropout):
    emphases.configure(DROPOUT=dropout, NUM_STEPS=40, EVALUATION_INTERVAL=10)
    runs = []
    for name in ('straight', 'again', 'third'):
        del recorder[:]
        emphases.train(['synthetic'], tmp_path / name)
        runs.append(recorder[:])
    del recorder[:]
    emphases.configure(NUM_STEPS=20)
    emphases.train(['synthetic'], tmp_path / 'resumed')
    assert not (tmp_path / 'resumed' / '00000030.pt').exists()
    emphases.configure(NUM_STEPS=40)
    emphases.train(['synthetic'], tmp_path / 'resumed')
    # the resumed run takes the same batches with the same generator state
    # (the same dropout seeds) at every step
    assert_same_calls(runs[0], recorder)
    uninterrupted = [
        state_of(tmp_path / name, 40) for name in ('straight', 'again', 'third')]
    resumed = state_of(tmp_path / 'resumed', 40)
    straight = uninterrupted[0]
    assert straight['epoch'] == resumed['epoch'] and straight['step'] == resumed['step']
    assert straight['optimizer']['param_groups'] == resumed['optimizer']['param_groups']
    for part in (model_tensors, optimizer_tensors):
        difference = largest_difference(part(straight), part(resumed))
        assert difference <= spread_bound(uninterrupted, part), part.__name__


def model_tensors(state):
    return state['model']


def optimizer_tensors(state):
    return {
        f'{index}.{key}': value.float()
        for index, values in state['optimizer']['state'].items()
        for key, value in values.items()}


def test_command_line(emphases, cache_root, tmp_path):
    config = tmp_path / 'config.py'
    config.write_text(
        f"CACHE_DIR = {str(cache_root / 'cache')!r}\n"
        f"PARTITION_DIR = {str(cache_root / 'partitions')!r}\n"
        "NUM_STEPS = 6\nEVALUATION_INTERVAL = 3\n")
    result = subprocess.run(
        [sys.executable, '-m', 'emphases_b200.train', '--config', str(config),
         '--datasets', 'synthetic', '--directory', str(tmp_path / 'run'), '--gpu', '0'],
        cwd=ROOT, capture_output=True, text=True)
    assert result.returncode == 0, result.stderr[-3000:]
    assert (tmp_path / 'run' / '00000003.pt').exists()
    assert (tmp_path / 'run' / '00000006.pt').exists()
    assert (tmp_path / 'run' / 'best.pt').exists()
    log = [json.loads(line) for line in open(tmp_path / 'run' / 'log.jsonl')]
    assert [line['step'] for line in log] == [3, 6]


@pytest.mark.parametrize('config', [
    {'ARCHITECTURE': 'transformer'},
    {'CHANNELS': 128, 'ENCODER_KERNEL_SIZE': 7, 'DECODER_KERNEL_SIZE': 7}])
def test_other_architectures_run_loop_steps(emphases, tmp_path, config):
    emphases.configure(NUM_STEPS=4, EVALUATION_INTERVAL=2, **config)
    model = emphases.train(['synthetic'], tmp_path)
    log = [json.loads(line) for line in open(tmp_path / 'log.jsonl')]
    assert [line['step'] for line in log] == [2, 4]
    assert all(np.isfinite(line['valid_loss']) for line in log)
    assert all(torch.isfinite(p).all() for p in model.parameters())


def _worker(rank, world, port, root, directory, max_frames):
    os.environ.update(
        MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
        WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    try:
        import emphases_b200 as emphases
        emphases.configure(
            CACHE_DIR=os.path.join(root, 'cache'),
            PARTITION_DIR=os.path.join(root, 'partitions'),
            MAX_TRAINING_FRAMES=max_frames, NUM_STEPS=6, EVALUATION_INTERVAL=3)
        model = emphases.train(['synthetic'], directory, rank)
        flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        copies = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(copies, flat)
        assert torch.equal(copies[0], copies[1])
        optimizer_steps = torch.load(
            os.path.join(directory, '00000006.pt'), weights_only=False)['step']
        assert optimizer_steps == 6
        with open(os.path.join(directory, f'ok{rank}'), 'w') as stream:
            stream.write('ok')
    finally:
        dist.destroy_process_group()


def test_two_gpu_loop_with_an_odd_batch_count(emphases, cache_root, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    dataset = emphases.data.Dataset('synthetic', 'train')
    for max_frames in range(1500, 6000, 100):
        if len(emphases.data.Sampler(dataset, max_frames).batch()) % 2 == 1:
            break
    else:
        pytest.fail('no frame budget gives an odd batch count')
    port = 33500 + os.getpid() % 2000
    mp.spawn(
        _worker, args=(2, port, str(cache_root), str(tmp_path), max_frames),
        nprocs=2, join=True)
    assert all((tmp_path / f'ok{r}').exists() for r in range(2))
    log = [json.loads(line) for line in open(tmp_path / 'log.jsonl')]
    assert [line['step'] for line in log] == [3, 6]
