"""The training loop's data path on one GPU: a synthetic dataset in the
reference's cache layout (16-bit wav + TextGrid + scores, bench.py's corpus:
U(2, 20) s files, 2.5 words/s), read into a resident corpus and fed to
`training.train_step` through `emph_gather_batch`.

    python tools/train_loop_bench.py [--files 3000] [--output FILE]

Prints one JSON line:
- `load_s`: reading the files (`read_s`), then the upload and the log-mel
  kernel over the partition (`features_s`), host clock around a synchronise;
- `gather`: `emph_gather_batch` over the epoch's batches, CUDA events around
  `--passes` passes; bytes per batch from shapes (the real rows read, the
  padded features and targets written) and the rate over that time.  The
  resident rows (about 1.1 GB) exceed the 126 MB L2, so reads come from HBM;
- `loop_ms` against `bare_ms`: host clock per step around a synchronise,
  `train_step` on `Dataset.batch` batches against `train_step` on the same
  batches built beforehand (device copies), the two arms alternated `--rounds`
  times in this process over the first `--steps` batches of the epoch, and
  `batch_host_ms`, the host time of one `Dataset.batch` call (enqueue only);
- the card's name and power limit, read in the same run.
The synthetic dataset goes to a temporary directory that is removed at exit.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def card():
    index = torch.cuda.current_device()
    try:
        limit = subprocess.run(
            ['nvidia-smi', f'--id={index}', '--query-gpu=power.limit',
             '--format=csv,noheader'], capture_output=True, text=True,
            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = ''
    return torch.cuda.get_device_name(), limit or 'unknown'


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--files', type=int, default=3000)
    parser.add_argument('--passes', type=int, default=20)
    parser.add_argument('--steps', type=int, default=40)
    parser.add_argument('--rounds', type=int, default=5)
    parser.add_argument('--output')
    args = parser.parse_args()

    import emphases_b200 as emphases
    from synthetic_cache import write_cache
    device = torch.device('cuda', 0)
    torch.cuda.set_device(device)
    base = '/dev/shm' if os.path.isdir('/dev/shm') else None
    root = tempfile.mkdtemp(prefix='emphases_b200_train_loop_', dir=base)
    try:
        write_cache(root, 'bench', {'train': args.files}, seed=4321)
        emphases.configure(
            CACHE_DIR=os.path.join(root, 'cache'),
            PARTITION_DIR=os.path.join(root, 'partitions'))
        torch.zeros(1, device=device)
        emphases.get_engine(device)

        start = time.perf_counter()
        dataset = emphases.data.Dataset('bench', 'train', 0)
        read = time.perf_counter() - start
        dataset.resident()
        torch.cuda.synchronize()
        load = time.perf_counter() - start
        resident = dataset.resident()
        frames_total = int(dataset.lengths.sum())

        # gather: every batch of epoch 0, items uploaded beforehand
        sampler = emphases.data.Sampler(dataset)
        batches = sampler.batch()
        items = [torch.tensor(b, dtype=torch.int32, device=device) for b in batches]
        shapes = [
            (len(b), int(dataset.lengths[b].max()), int(dataset.n_words[b].max()))
            for b in batches]
        channels = resident['rows'].shape[1]
        moved = sum(
            4 * (channels * int(dataset.lengths[b].sum()) + int(dataset.n_words[b].sum()) +
                 n * channels * tmax + n * wmax)
            for b, (n, tmax, wmax) in zip(batches, shapes))
        eng, ws = resident['engine'], resident['workspace']

        def gather_pass():
            for index, (n, tmax, wmax) in zip(items, shapes):
                eng.gather_batch(
                    resident['rows'], resident['row_start'], resident['n_rows'],
                    resident['targets'], resident['word_start'], resident['n_words'],
                    index, tmax, wmax, ws)
        gather_pass()
        torch.cuda.synchronize()
        begin, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        begin.record()
        for _ in range(args.passes):
            gather_pass()
        end.record()
        end.synchronize()
        gather_ms = begin.elapsed_time(end) / (args.passes * len(batches))
        gather_bytes = moved / len(batches)

        # loop step against the bare step on the same batches
        torch.manual_seed(0)
        model = emphases.Model().to(device)
        optimizer = torch.optim.Adam(model.parameters(), lr=emphases.LEARNING_RATE)
        chosen = batches[:args.steps]
        prebuilt = []
        for indices in chosen:
            batch = dataset.batch(indices)
            prebuilt.append((batch[0].clone(),) + batch[1:4] + (batch[4].clone(),))

        def loop():
            for indices in chosen:
                emphases.training.train_step(model, optimizer, dataset.batch(indices))

        def bare():
            for batch in prebuilt:
                emphases.training.train_step(model, optimizer, batch)

        loop()
        bare()
        # host time of Dataset.batch alone (bounds assembly, index upload, the
        # gather launch), enqueue only
        torch.cuda.synchronize()
        start = time.perf_counter()
        for indices in chosen:
            dataset.batch(indices)
        batch_host_ms = 1000. * (time.perf_counter() - start) / len(chosen)
        torch.cuda.synchronize()
        times = {'loop': [], 'bare': []}
        for _ in range(args.rounds):
            for name, run in (('loop', loop), ('bare', bare)):
                torch.cuda.synchronize()
                start = time.perf_counter()
                run()
                torch.cuda.synchronize()
                times[name].append(1000. * (time.perf_counter() - start) / len(chosen))
        name, power_limit = card()
        loop_ms, bare_ms = float(np.median(times['loop'])), float(np.median(times['bare']))
        result = {
            'tool': 'train_loop_bench',
            'files': args.files,
            'frames': frames_total,
            'audio_hours': frames_total * emphases.HOPSIZE / emphases.SAMPLE_RATE / 3600,
            'load_s': load, 'read_s': read, 'features_s': load - read,
            'gather': {
                'batches': len(batches),
                'mean_batch': float(np.mean([n for n, _, _ in shapes])),
                'ms_per_batch': gather_ms,
                'mb_per_batch': gather_bytes / 1e6,
                'gb_per_s': gather_bytes / (gather_ms * 1e-3) / 1e9,
                'share_of_7.7_tb_per_s': gather_bytes / (gather_ms * 1e-3) / 7.7e12},
            'steps': len(chosen), 'rounds': args.rounds,
            'loop_ms': loop_ms, 'bare_ms': bare_ms,
            'loop_over_bare': loop_ms / bare_ms - 1.,
            'batch_host_ms': batch_host_ms,
            'loop_ms_rounds': times['loop'], 'bare_ms_rounds': times['bare'],
            'gpu': name, 'power_limit': power_limit,
            'train_precision': emphases.training.TRAIN_PRECISION}
        line = json.dumps(result)
        print(line)
        if args.output:
            os.makedirs(os.path.dirname(os.path.abspath(args.output)), exist_ok=True)
            with open(args.output, 'w') as stream:
                stream.write(line + '\n')
    finally:
        shutil.rmtree(root, ignore_errors=True)


if __name__ == '__main__':
    main()
