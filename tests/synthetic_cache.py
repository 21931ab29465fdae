"""A synthetic dataset in the reference's cache layout: 16-bit wav, TextGrid
and per-word scores under `<root>/cache/<name>/{audio,alignment,scores}` and
the partition file `<root>/partitions/<name>.json`.  Every word of a file is
noise at its own gain and its score is that gain, so a model can learn it."""
import json
from pathlib import Path

import numpy as np
import torch

SAMPLE_RATE = 16000
HOPSIZE = 160


def layout(count, seed, seconds=(2., 20.), words_per_second=2.5):
    """bench.py's corpus layout: durations U(lo, hi) s on the hop grid,
    max(2, floor(2.5 dur)) words tiling each file, at least 2 frames a word"""
    rng = np.random.default_rng(seed)
    samples = (rng.uniform(*seconds, count) * SAMPLE_RATE).astype(np.int64)
    samples = samples // HOPSIZE * HOPSIZE
    times = []
    for n in samples:
        duration = n / SAMPLE_RATE
        frames = n // HOPSIZE
        words = min(max(2, int(words_per_second * duration)), frames // 2 - 1)
        cuts = np.sort(rng.choice(
            np.arange(1, frames // 2), size=words - 1, replace=False)) * 2
        cuts = (cuts + rng.uniform(0.05, 0.95, words - 1)) * HOPSIZE / SAMPLE_RATE
        edges = np.concatenate([[0.], cuts, [duration]])
        times.append(np.stack([edges[:-1], edges[1:]], axis=1))
    return samples, times


def write_cache(root, name, counts, seed=0, seconds=(2., 20.), sample_rate=SAMPLE_RATE):
    """`counts` = {partition: number of files}.  Returns {partition: stems}"""
    import emphases_b200 as emphases
    root = Path(root)
    cache = root / 'cache' / name
    for sub in ('audio', 'alignment', 'scores'):
        (cache / sub).mkdir(parents=True, exist_ok=True)
    total = sum(counts.values())
    samples, times = layout(total, seed, seconds)
    rng = np.random.default_rng(seed + 1)
    generator = torch.Generator().manual_seed(seed)
    stems = [f'{name}-{i:05d}' for i in range(total)]
    for stem, n, t in zip(stems, samples, times):
        gains = rng.uniform(0.05, 1., len(t))
        edges = np.minimum((t[:, 1] * SAMPLE_RATE).astype(np.int64), n)
        edges[-1] = n
        envelope = np.repeat(gains, np.diff(np.concatenate([[0], edges])))
        audio = 0.3 * torch.randn(1, int(n), generator=generator) * \
            torch.from_numpy(envelope).float()[None]
        emphases.load.save_wav(
            cache / 'audio' / f'{stem}.wav', audio.clamp(-1, 1), sample_rate)
        emphases.Alignment.from_times(
            [tuple(x) for x in t.tolist()]).save(cache / 'alignment' / f'{stem}.TextGrid')
        torch.save(torch.from_numpy(gains).float(), cache / 'scores' / f'{stem}.pt')
    partitions, cursor = {}, 0
    for partition, count in counts.items():
        partitions[partition] = stems[cursor:cursor + count]
        cursor += count
    (root / 'partitions').mkdir(parents=True, exist_ok=True)
    with open(root / 'partitions' / f'{name}.json', 'w') as stream:
        json.dump(partitions, stream)
    return partitions
