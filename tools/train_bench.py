"""BASELINE config 5: one data-parallel training step (forward + backward, BCE
on word scores, NCCL gradient all-reduce, Adam) on a synthetic padded batch
shaped like the reference's collate (B * Tmax <= MAX_TRAINING_FRAMES = 75,000
frames per GPU, emphases/config/defaults.py:230; utterances U(2, 20) s).

    python tools/train_bench.py                                  # 1 GPU
    python tools/train_bench.py --architecture transformer       # Transformer variant
    python tools/train_bench.py --dropout 0.1                    # conv model, DROPOUT=0.1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N \\
        --master-addr 127.0.0.1 --master-port 29533 tools/train_bench.py

Prints one JSON line: ms per step (CUDA events, max over ranks), frames/s and
audio-s/s over all ranks (weak scaling: every rank has its own batch), and the
share of the step spent in the gradient all-reduce, with the card's name and
power limit read in the same run.
"""
import argparse
import json
import subprocess
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def synthetic_batch(seed, max_frames=75000):
    generator = np.random.default_rng(seed)
    lengths = []
    while True:
        frames = int(generator.uniform(2., 20.) * 100)
        if (len(lengths) + 1) * max(lengths + [frames]) > max_frames:
            break
        lengths.append(frames)
    words = [max(2, int(2.5 * t / 100)) for t in lengths]
    tmax, wmax = max(lengths), max(words)
    torch_generator = torch.Generator().manual_seed(seed)
    features = torch.zeros(len(lengths), 80, tmax)
    bounds = torch.zeros(len(lengths), 2, wmax, dtype=torch.long)
    for i, (t, w) in enumerate(zip(lengths, words)):
        features[i, :, :t] = torch.randn(80, t, generator=torch_generator)
        cuts = np.sort(generator.choice(np.arange(1, t - 1), size=w - 1, replace=False))
        edges = np.concatenate([[0], cuts, [t]])
        bounds[i, 0, :w] = torch.from_numpy(edges[:-1])
        bounds[i, 1, :w] = torch.from_numpy(edges[1:])
    targets = torch.rand(len(lengths), 1, wmax, generator=torch_generator)
    return (features, torch.tensor(lengths), bounds, torch.tensor(words), targets)


def card():
    """(name, power limit) of the current GPU"""
    try:
        index = torch.cuda.current_device()
        limit = subprocess.run(
            ['nvidia-smi', f'--id={index}', '--query-gpu=power.limit',
             '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = 'unknown'
    return torch.cuda.get_device_name(), limit or 'unknown'


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument(
        '--architecture', choices=['convolution', 'transformer'], default='convolution',
        help='ARCHITECTURE of the trained model (the transformer step trains with the '
             "reference's dropout, p = 0.1)")
    parser.add_argument(
        '--dropout', type=float, default=None,
        help='DROPOUT of the convolution model (the reference sweeps 0.05 and 0.1); '
             'default None: no dropout modules')
    args = parser.parse_args()
    if args.dropout is not None and args.architecture != 'convolution':
        parser.error('--dropout sets DROPOUT, which only the convolution model reads')
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)
    import emphases_b200 as emphases
    emphases.reset_configuration()
    emphases.configure(ARCHITECTURE=args.architecture)
    if args.dropout is not None:
        emphases.configure(DROPOUT=args.dropout)
    torch.manual_seed(0)
    model = emphases.Model().to(device)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)
    batch = synthetic_batch(100 + rank)
    batch = (batch[0].to(device),) + batch[1:4] + (batch[4].to(device),)
    frames = int(batch[1].sum())
    steps, warmup = 20, 3

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(device)

    for _ in range(warmup):
        emphases.training.train_step(model, optimizer, batch)
    barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        value = emphases.training.train_step(model, optimizer, batch)
    end.record()
    barrier()
    ms = start.elapsed_time(end) / steps

    # the all-reduce alone (same flat bucket)
    reduce_ms = 0.
    if world > 1:
        for p in model.parameters():
            p.grad = torch.zeros_like(p)
        barrier()
        start.record()
        for _ in range(steps):
            emphases.training.allreduce_gradients(model)
        end.record()
        barrier()
        reduce_ms = start.elapsed_time(end) / steps

    stats = torch.tensor([ms, reduce_ms, frames], dtype=torch.float64, device=device)
    if world > 1:
        worst = stats.clone()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        total = stats.clone()
        dist.all_reduce(total, op=dist.ReduceOp.SUM)
        ms, reduce_ms, frames_total = worst[0].item(), worst[1].item(), total[2].item()
    else:
        frames_total = frames
    if rank == 0:
        name, power_limit = card()
        print(json.dumps({
            'architecture': args.architecture, 'dropout': args.dropout,
            'gpu': name, 'power_limit': power_limit,
            'metric': 'training step (config 5)', 'n_gpus': world,
            'ms_per_step': ms, 'allreduce_ms': reduce_ms,
            'frames_per_s': frames_total / (ms * 1e-3),
            'audio_s_per_s': frames_total / 100. / (ms * 1e-3),
            'batch': {'utterances': int(batch[0].shape[0]), 'tmax': int(batch[0].shape[2]),
                      'frames': frames, 'padded_frames': int(batch[0].shape[0] * batch[0].shape[2])},
            'loss': float(value), 'precision': 'fp32 forward/backward kernels',
            'scaling': 'weak'}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
