"""BASELINE config 5: one data-parallel training step (forward + backward, BCE
on word scores, NCCL gradient all-reduce, Adam) on a synthetic padded batch
shaped like the reference's collate (B * Tmax <= MAX_TRAINING_FRAMES = 75,000
frames per GPU, emphases/config/defaults.py:230; utterances U(2, 20) s).

    python tools/train_bench.py                                  # 1 GPU
    python tools/train_bench.py --architecture transformer       # Transformer variant
    python tools/train_bench.py --dropout 0.1                    # conv model, DROPOUT=0.1
    python tools/train_bench.py --channels 128 --encoder-kernel 7  # a hyper-parameter sweep shape
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N \\
        --master-addr 127.0.0.1 --master-port 29533 tools/train_bench.py

Prints one JSON line: ms per step (CUDA events, max over ranks), frames/s and
audio-s/s over all ranks (weak scaling: every rank has its own batch), and the
share of the step spent in the gradient all-reduce, with the card's name and
power limit read in the same run.  A convolution model of another shape than
the default also gets `weight_grad`: the time per layer of emph_conv_weight_grad
at its kernel width and each kernel size, from CUDA events over 50 launches on
the batch's packed frame rows, and its useful rate 2 k C^2 rows / time; beside
it the native step's <80, 3> weight gradient, timed with torch.profiler on the
same batch (a LAYERS=0 model at 'loss', whose one weight gradient is the input
layer's over the native step's kept frame rows).
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


def time_weight_grad(emphases, width, kernel, rows, launches=50):
    """(us per launch, rows) of emph_conv_weight_grad on random (rows, width)
    operands, CUDA events over `launches` launches after a warm-up"""
    from emphases_b200 import _lib
    generator = torch.Generator(device='cuda').manual_seed(kernel)
    x = torch.randn(rows, width, device='cuda', generator=generator)
    dpre = torch.randn(rows, width, device='cuda', generator=generator)
    dw = torch.empty(kernel, width, width, device='cuda')
    db = torch.empty(width, device='cuda')

    def launch():
        _lib.call('emph_conv_weight_grad', _lib.ptr(x), _lib.ptr(dpre), rows, width, kernel,
                  _lib.ptr(dw), _lib.ptr(db), _lib.stream_ptr())
    for _ in range(5):
        launch()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        launch()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / launches


def native_weight_grad(emphases, batch, steps=20):
    """us per launch of the native step's <80, 3> weight gradient and its rows:
    a LAYERS=0 model at 'loss' runs it once per step, on the input layer"""
    from torch.profiler import ProfilerActivity, profile
    emphases.reset_configuration()
    emphases.configure(LAYERS=0, DOWNSAMPLE_LOCATION='loss')
    model = emphases.Model().cuda().train()
    features, frame_lengths, bounds, word_lengths, targets = batch
    assert emphases.training.native_step_supported(model, features)

    def step():
        model.zero_grad(set_to_none=True)
        model(features, frame_lengths, bounds, word_lengths).sum().backward()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    times = [e.device_time for e in prof.events()
             if e.device_type == torch.autograd.DeviceType.CUDA and
             'conv_weight_grad_mma_kernel' in e.name]
    assert len(times) == steps, len(times)
    # the native step keeps length + 1 rows per item (one frame layer, k = 3)
    # and one separator row before and after each (csrc/train_step.cu, kept_rows)
    frames = features.shape[2]
    rows = 1 + sum(min(frames, int(t) + 1) + 1 for t in frame_lengths)
    return sum(times) / steps, rows


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
    parser.add_argument('--channels', type=int, default=None, help='CHANNELS (64, 80, 128)')
    parser.add_argument('--layers', type=int, default=None, help='LAYERS')
    parser.add_argument('--encoder-kernel', type=int, default=None, help='ENCODER_KERNEL_SIZE')
    parser.add_argument('--decoder-kernel', type=int, default=None, help='DECODER_KERNEL_SIZE')
    args = parser.parse_args()
    shape = {key: value for key, value in (
        ('CHANNELS', args.channels), ('LAYERS', args.layers),
        ('ENCODER_KERNEL_SIZE', args.encoder_kernel),
        ('DECODER_KERNEL_SIZE', args.decoder_kernel)) if value is not None}
    if args.architecture != 'convolution' and (args.dropout is not None or shape):
        parser.error('--dropout and the shape options configure the convolution model')
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
    emphases.configure(ARCHITECTURE=args.architecture, **shape)
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
    weight_grad = None
    if rank == 0 and shape:
        from emphases_b200 import engine
        width = engine.kernel_width(emphases.CHANNELS)
        starts, rows = engine.packed_starts([int(batch[0].shape[2])] * int(batch[0].shape[0]))
        weight_grad = {}
        for kernel in sorted({emphases.ENCODER_KERNEL_SIZE, emphases.DECODER_KERNEL_SIZE}):
            us = time_weight_grad(emphases, width, kernel, rows)
            weight_grad[f'{width}/k{kernel}'] = {
                'us_per_layer': us, 'rows': rows,
                'useful_tflops': 2 * kernel * width ** 2 * rows / (us * 1e-6) / 1e12}
        us, native_rows = native_weight_grad(emphases, batch)
        weight_grad['80/k3 native'] = {
            'us_per_layer': us, 'rows': native_rows,
            'useful_tflops': 2 * 3 * 80 ** 2 * native_rows / (us * 1e-6) / 1e12}
    if rank == 0:
        name, power_limit = card()
        print(json.dumps({
            'architecture': args.architecture, 'dropout': args.dropout, 'shape': shape,
            'weight_grad': weight_grad,
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
