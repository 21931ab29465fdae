"""Training corpus from the reference's cache layout
(emphases/data/dataset.py), resident on the GPU.

The reference loads one cached `mels/<stem>.pt` per item in DataLoader
workers and copies every padded batch to the device.  Here a partition is read
once (TextGrid + 16-bit wav through the native corpus reader, scores through
torch.load), its log-mel features are computed once by the log-mel kernel in
the training framing (`engine.feature_plan`) and stay on the device with the
word targets, and each padded batch is assembled there by one
`emph_gather_batch` launch: no host I/O per step.
"""
import json
from pathlib import Path

import numpy as np
import torch

import emphases_b200 as emphases
from .. import corpus, engine
from .sampler import buckets, sampler


class Dataset:
    """Items of partition `partition` of the datasets `names`
    (`CACHE_DIR/<name>/{alignment,audio,scores}/<stem>.*`, stems from
    `PARTITION_DIR/<name>.json[partition]`).

    `__getitem__` returns the reference's item tuple; `batch(indices)` returns
    what `training.train_step` takes, features and targets on the device.
    Host metadata is read at construction; the device copy (features and
    targets) is built on first use on GPU `gpu` (None: the current device)."""

    def __init__(self, names, partition, gpu=None):
        if isinstance(names, str):
            names = [names]
        self.partition = partition
        self.gpu = gpu
        self.stems, self.text_files, self.audio_files, score_files = [], [], [], []
        for name in names:
            file = Path(emphases.PARTITION_DIR) / f'{name}.json'
            with open(file) as stream:
                partitions = json.load(stream)
            if partition not in partitions:
                raise KeyError(f'{file} has no partition {partition!r}')
            cache = Path(emphases.CACHE_DIR) / name
            for stem in partitions[partition]:
                self.stems.append(stem)
                self.text_files.append(str(cache / 'alignment' / f'{stem}.TextGrid'))
                self.audio_files.append(str(cache / 'audio' / f'{stem}.wav'))
                score_files.append(cache / 'scores' / f'{stem}.pt')

        with corpus.Corpus(self.text_files, self.audio_files) as reader:
            for i in range(len(self.stems)):
                if reader.status[i] != 0:
                    raise ValueError(
                        f'{self.audio_files[i]}: {reader.error(i)} (training reads '
                        '16-bit PCM wav files and TextGrid alignments)')
                if reader.sample_rate[i] != emphases.SAMPLE_RATE:
                    raise ValueError(
                        f'{self.audio_files[i]}: sample rate {reader.sample_rate[i]} Hz, '
                        f'the training cache holds {emphases.SAMPLE_RATE} Hz audio')
                if reader.n_words[i] == 0:
                    raise ValueError(f'{self.text_files[i]}: no words')
            self.samples = reader.n_samples.copy()
            # raises for a file the reference's reflect pad cannot take
            self.plan = engine.feature_plan(self.samples, self.stems)
            _, times, packed = reader.load(
                np.ones(len(self.stems), dtype=bool), pin=torch.cuda.is_available())
            if len(self.stems):
                packed.ready(len(self.stems) - 1)
        # channel 0 as int16, host: a copy of its own, since the reader's
        # staging buffer is reused by the next corpus read of this thread
        self.audio = torch.empty(
            packed.buffer.shape, dtype=torch.int16, pin_memory=torch.cuda.is_available())
        self.audio.copy_(packed.buffer)
        self.audio_offsets = packed.offsets

        # dataset.py:41-50: alignment.word_bounds(SAMPLE_RATE, HOPSIZE,
        # silences=True), i.e. int(t * sample_rate / hopsize) per word edge
        bounds = [
            (t * emphases.SAMPLE_RATE / emphases.HOPSIZE).astype(np.int64)
            for t in times]
        targets = []
        for stem, file, bound in zip(self.stems, score_files, bounds):
            scores = torch.load(file, map_location='cpu', weights_only=False)
            scores = scores.detach().reshape(-1).to(torch.float32)
            if scores.numel() != len(bound):
                raise ValueError(
                    f'{stem}: {scores.numel()} scores for {len(bound)} words ({file})')
            targets.append(scores)
        self.n_words = np.array([len(b) for b in bounds], dtype=np.int32)
        self.word_start = np.concatenate(
            [[0], np.cumsum(self.n_words[:-1], dtype=np.int64)]).astype(np.int32) \
            if len(bounds) else np.zeros(0, dtype=np.int32)
        self.bounds = np.concatenate(bounds) if bounds else np.zeros((0, 2), np.int64)
        self.targets = torch.cat(targets) if targets else torch.zeros(0)
        self.lengths = self.plan.n_rows.astype(np.int64)
        self._device = None

    def __len__(self):
        return len(self.stems)

    def buckets(self):
        """dataset.py:97-117"""
        return buckets(self.lengths)

    # -- device residency ----------------------------------------------------

    def resident(self):
        """The device copy: frame rows (packed, one separator row between
        files), word targets and the per-item index arrays"""
        if self._device is not None:
            return self._device
        device = emphases.resolve_device(self.gpu)
        eng = emphases.get_engine(device)
        plan = self.plan
        with torch.cuda.device(device):
            audio = self.audio.to(device, non_blocking=True)
            views = eng.upload_plan(plan)
            row_seq = eng.row_index(
                views['row_start'], views['n_rows'], plan.n_seq, plan.total_rows)
            rows = eng.logmel(audio, views, plan, row_seq, emphases.NORMALIZE)
            index = torch.from_numpy(np.concatenate([
                plan.row_start, plan.n_rows, self.word_start, self.n_words
            ]).astype(np.int32)).to(device)
            n = len(self)
            self._device = {
                'engine': eng, 'rows': rows,
                'row_start': index[:n], 'n_rows': index[n:2 * n],
                'word_start': index[2 * n:3 * n], 'n_words': index[3 * n:],
                'targets': self.targets.to(device),
                'workspace': eng.workspace('batch')}
            # the staging buffers of the upload are shared: finish before return
            torch.cuda.current_stream().synchronize()
        return self._device

    def features(self, index):
        """(NUM_MELS, T) device features of item `index` (a view)"""
        resident = self.resident()
        start, frames = int(self.plan.row_start[index]), int(self.plan.n_rows[index])
        return resident['rows'][start:start + frames].t()

    # -- access --------------------------------------------------------------

    def __getitem__(self, index):
        """dataset.py:27-62: (features (80, T), scores (1, W), word_bounds
        (2, W) int64, alignment, audio (1, S), stem), on the host"""
        start, count = int(self.word_start[index]), int(self.n_words[index])
        offset, samples = int(self.audio_offsets[index]), int(self.samples[index])
        audio = self.audio[offset:offset + samples].to(torch.float32) / 32768.
        return (
            self.features(index).cpu(),
            self.targets[start:start + count].clone()[None],
            torch.from_numpy(self.bounds[start:start + count].T.copy()),
            emphases.Alignment(self.text_files[index]),
            audio[None],
            self.stems[index])

    def batch(self, indices):
        """(features (B, NUM_MELS, Tmax), frame_lengths (B,), word_bounds
        (B, 2, Wmax) int64, word_lengths (B,), targets (B, 1, Wmax)) of items
        `indices`, equal to data.collate([self[i] for i in indices])[:5].
        Features and targets are device tensors built by one kernel launch;
        they are views of a grow-only buffer, valid until the next `batch`
        call on this device.  Lengths and bounds are host tensors."""
        indices = np.asarray(indices, dtype=np.int64).reshape(-1)
        if len(indices) == 0:
            raise ValueError('an empty batch')
        if indices.min() < 0 or indices.max() >= len(self):
            raise IndexError(f'batch index out of range for {len(self)} items')
        resident = self.resident()
        frames = self.lengths[indices]
        words = self.n_words[indices].astype(np.int64)
        tmax, wmax = int(frames.max()), int(words.max())
        within = np.arange(wmax)[None]
        real = within < words[:, None]
        source = np.where(real, self.word_start[indices][:, None] + within, 0)
        word_bounds = np.where(
            real[:, None], self.bounds[source].transpose(0, 2, 1), 0)
        items = torch.from_numpy(indices.astype(np.int32))
        ws = resident['workspace']
        device_items = ws.get('batch_items', (len(indices),), torch.int32)
        with torch.cuda.device(device_items.device):
            if torch.cuda.is_available():
                items = items.pin_memory()   # the caching host allocator keeps
            device_items.copy_(items, non_blocking=True)   # it until the copy ends
            features, targets = resident['engine'].gather_batch(
                resident['rows'], resident['row_start'], resident['n_rows'],
                resident['targets'], resident['word_start'], resident['n_words'],
                device_items, tmax, wmax, ws)
        return (
            features, torch.from_numpy(frames.copy()), torch.from_numpy(word_bounds),
            torch.from_numpy(words), targets)


class Loader:
    """Device batches of `dataset` in the order of `batch_sampler`"""

    def __init__(self, dataset, batch_sampler):
        self.dataset = dataset
        self.batch_sampler = batch_sampler

    def __iter__(self):
        for indices in self.batch_sampler:
            yield self.dataset.batch(indices)

    def __len__(self):
        return len(self.batch_sampler)


def loader(dataset, partition):
    """emphases/data/loader.py: batches in the order of
    `data.sampler(dataset, partition)`, assembled on the device"""
    return Loader(dataset, sampler(dataset, partition))
