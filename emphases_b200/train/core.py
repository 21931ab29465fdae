"""Training loop (emphases/train/core.py): step-based Adam training of
`Model` over a dataset cache, periodic validation, checkpoints and resume.

Every step is `training.train_step` on a batch that `data.Dataset.batch`
assembles on the device from the resident corpus.  Under torch.distributed
every rank runs the loop on its own GPU; `train_step` all-reduces gradients.
"""
import json
import math
import time
from pathlib import Path

import torch

import emphases_b200 as emphases
from .. import data, distributed, training
from ..evaluate import metrics


def rank_batches(batches, rank, world):
    """Rank `rank`'s batches of one epoch: batches r, r + world, ... of the
    epoch's list, trimmed to a multiple of `world`.  The trim gives every rank
    the same number of steps: an epoch whose batch count is not a multiple of
    `world` would otherwise leave the ranks without an extra batch waiting in
    the gradient all-reduce of the others' extra step."""
    return batches[:len(batches) // world * world][rank::world]


def checkpoints(directory):
    """Step checkpoints `<step:08d>.pt` of `directory`, in step order"""
    found = [
        (int(path.stem), path) for path in Path(directory).glob('*.pt')
        if path.stem.isdigit()]
    return [path for _, path in sorted(found)]


def latest_checkpoint(directory):
    """The checkpoint of the highest step in `directory`, or None"""
    found = checkpoints(directory)
    return found[-1] if found else None


def checkpoint_state(model, optimizer, epoch, step, score, best, device):
    """The released checkpoint's keys (model, optimizer, epoch, step, score,
    best) and 'rng', the torch CPU and CUDA generator states: dropout seeds
    are drawn from them, so a resumed run continues as it would have"""
    return {
        'model': model.state_dict(), 'optimizer': optimizer.state_dict(),
        'epoch': epoch, 'step': step, 'score': score, 'best': best,
        'rng': {'cpu': torch.get_rng_state(), 'cuda': torch.cuda.get_rng_state(device)}}


def evaluate(model, loader):
    """(loss, Pearson correlation) of `model` in eval mode over `loader`'s
    batches, with the evaluation metric classes: dataset statistics of the
    postprocessed scores and the targets, then the metrics.  The loss is the
    metric named by LOSS ('bce' or 'mse')."""
    model.eval()
    outputs = []
    predicted, target = metrics.Statistics(), metrics.Statistics()
    with torch.no_grad():
        for features, frame_lengths, word_bounds, word_lengths, targets in loader:
            logits = model(features, frame_lengths, word_bounds, word_lengths)
            targets = targets.clone()   # the loader reuses its buffers
            outputs.append((logits, targets, word_lengths))
            predicted.update(emphases.postprocess(logits), word_lengths)
            target.update(targets, word_lengths)
    result = metrics.Metrics(predicted, target)
    for logits, targets, word_lengths in outputs:
        result.update(logits, targets, word_lengths)
    values = result()
    return values['bce' if emphases.LOSS == 'bce' else 'mse'], values['pearson_correlation']


def train(datasets, directory, gpu=None):
    """Train `Model()` with Adam(LEARNING_RATE) for NUM_STEPS steps on the
    'train' partition of `datasets`, validating on 'valid' every
    EVALUATION_INTERVAL steps and at the end.

    Each validation appends one JSON line to `directory/log.jsonl` (step,
    train loss since the last validation, valid loss, Pearson correlation,
    milliseconds per training step) and saves `directory/<step:08d>.pt` with
    the keys of the released checkpoint ('model', 'optimizer', 'epoch',
    'step', 'score', 'best') plus 'rng', the torch CPU and CUDA generator
    states, so dropout continues on resume as it would have; `best.pt` is
    also written when the Pearson correlation improves.  A directory that
    holds checkpoints resumes from the highest step.

    Under torch.distributed, rank r takes batches r, r + world, ... of each
    epoch (`rank_batches`), and rank 0 alone validates and writes files
    while the others wait at a barrier.  Returns the trained model."""
    import torch.distributed as dist
    directory = Path(directory)
    rank, world = distributed.rank_and_world()
    device = emphases.resolve_device(gpu)
    torch.cuda.set_device(device)
    if rank == 0:
        directory.mkdir(parents=True, exist_ok=True)

    train_data = data.Dataset(datasets, 'train', device.index)
    valid_data = data.Dataset(datasets, 'valid', device.index) if rank == 0 else None

    torch.manual_seed(emphases.RANDOM_SEED)      # identical replicas on every rank
    model = emphases.Model().to(device)
    optimizer = torch.optim.Adam(model.parameters(), lr=emphases.LEARNING_RATE)
    step, epoch, best = 0, 0, -math.inf
    latest = latest_checkpoint(directory)
    if latest is not None:
        state = torch.load(latest, map_location='cpu', weights_only=False)
        model.load_state_dict(state['model'])
        optimizer.load_state_dict(state['optimizer'])
        step, epoch, best = int(state['step']), int(state['epoch']), float(state['best'])
        torch.set_rng_state(state['rng']['cpu'])
        torch.cuda.set_rng_state(state['rng']['cuda'], device)

    sampler = data.Sampler(train_data)

    def epoch_batches(number):
        sampler.set_epoch(number)
        batches = rank_batches(sampler.batch(), rank, world)
        if not batches:
            raise ValueError(
                f'{len(sampler.batch())} batches per epoch cannot feed {world} ranks')
        return batches

    # steps of the epochs before `epoch`: where in its epoch a resumed run is
    offset = step - sum(len(epoch_batches(e)) for e in range(epoch))
    losses, count = torch.zeros((), device=device), 0
    start = time.perf_counter()

    def validate():
        nonlocal best, losses, count, start
        torch.cuda.synchronize(device)
        milliseconds = 1000. * (time.perf_counter() - start) / max(count, 1)
        if rank == 0:
            valid_loss, pearson = evaluate(model, data.loader(valid_data, 'valid'))
            improved = pearson > best
            best = max(best, pearson)
            checkpoint = checkpoint_state(
                model, optimizer, epoch, step, pearson, best, device)
            torch.save(checkpoint, directory / f'{step:08d}.pt')
            if improved:
                torch.save(checkpoint, directory / 'best.pt')
            line = {
                'step': step,
                'train_loss': losses.item() / max(count, 1),
                'valid_loss': valid_loss,
                'pearson_correlation': pearson,
                'ms_per_step': milliseconds}
            with open(directory / 'log.jsonl', 'a') as stream:
                stream.write(json.dumps(line) + '\n')
        if world > 1 and dist.is_initialized():
            dist.barrier()
        losses.zero_()
        count = 0
        start = time.perf_counter()

    while step < emphases.NUM_STEPS:
        for indices in epoch_batches(epoch)[offset:]:
            losses += training.train_step(model, optimizer, train_data.batch(indices))
            count += 1
            step += 1
            if step % emphases.EVALUATION_INTERVAL == 0 or step == emphases.NUM_STEPS:
                validate()
            if step >= emphases.NUM_STEPS:
                break
        else:
            epoch, offset = epoch + 1, 0
    return model
