"""Conv models of kernel size 5 and 7 (the reference's hyper-parameter sweep)
on bench.py's corpus, in every PRECISION: the FFMA kernel (`fp32`) against the
tcgen05 stacks (`bf16`, `bf16x3`, `bf16x6`).

    python tools/conv_kernel_size_bench.py [--utterances 3000] [--steps 5]
                                           [--repeats 3] [--out FILE]

Shapes (random init, seeded): ENCODER / DECODER kernel sizes 5 / 7, 7 / 1,
and 7 / 7 with LAYERS = 7 (the largest halo the sweep builds).  The modes of a
shape run alternated, `--repeats` rounds of `--steps` passes each, in one
process.  Per (shape, mode) one JSON line with
  ms_per_pass        engine.forward_packed over the whole corpus (CUDA events;
                     the corpus' audio and features are far larger than L2),
                     median over the rounds
  frame_stack_ms     events around the frame stack alone (conv_stack, or
                     conv_stack_pool with the word pooling fused in)
  *_tflops           useful rate: 2 k C^2 rows layers over that time (frame
                     stack; the pass counts the word decoder too)
  max_score_diff_vs_fp32  over every word of the corpus
  speedup_vs_fp32, within_bar (the mode's score bar against the fp32 pass)
and the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [
    dict(ENCODER_KERNEL_SIZE=5, DECODER_KERNEL_SIZE=7),
    dict(ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=1),
    dict(ENCODER_KERNEL_SIZE=7, DECODER_KERNEL_SIZE=7, LAYERS=7),
]
MODES = ['fp32', 'bf16', 'bf16x3', 'bf16x6']
# scores against the fp32 pass (the tests' bars against the reference)
BARS = {'bf16': 2e-3, 'bf16x3': 2e-5, 'bf16x6': 1e-5}
CHANNELS = 80


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


def parse_args():
    parser = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    parser.add_argument('--utterances', type=int, default=3000)
    parser.add_argument('--steps', type=int, default=5)
    parser.add_argument('--repeats', type=int, default=3)
    parser.add_argument('--out', default=os.path.join(
        ROOT, 'profiles', 'r07_conv_kernel_sizes.jsonl'))
    return parser.parse_args()


def run_shape(emphases, engine, shape, lengths, times, device_audio, args, gpu):
    emphases.reset_configuration()
    emphases.configure(**shape)
    torch.manual_seed(7)
    model = emphases.Model().cuda().eval()
    weights = model.packed_weights()
    eng = emphases.get_engine(torch.device('cuda', 0))
    plan = engine.make_plan([(t, int(n)) for t, n in zip(times, lengths)], None, 'sum')
    views = eng.upload_plan(plan)
    words = torch.from_numpy(plan.word_seq >= 0).cuda()
    frames = int(plan.n_rows.sum())
    n_words = int(words.sum().item())
    layers = emphases.LAYERS
    k_frame, k_word = shape['ENCODER_KERNEL_SIZE'], shape['DECODER_KERNEL_SIZE']
    frame_flop = 2 * k_frame * CHANNELS ** 2 * frames * (layers + 1)
    word_flop = 2 * k_word * CHANNELS ** 2 * n_words * layers
    codes = {}
    for mode in MODES:
        emphases.configure(PRECISION=mode)
        codes[mode] = emphases.precision_code()
        eng.prepare_weights(weights, codes[mode])

    def step(mode, timers=None):
        return eng.forward_packed(
            device_audio, plan, weights, method='sum', location='intermediate',
            precision=codes[mode], views=views, timers=timers)

    scores, kernels = {}, {}
    for mode in MODES:                        # warm-up, and the scores
        step(mode)
        scores[mode] = step(mode)['scores'][words].clone()
        mode_code = codes[mode]
        kernels[mode] = {
            'frame': engine.frame_precision(mode_code, weights.frame),
            'word': engine.word_precision(mode_code, weights.word)}
    torch.cuda.synchronize()
    passes = {mode: [] for mode in MODES}
    stacks = {mode: [] for mode in MODES}
    for _ in range(args.repeats):
        for mode in MODES:                    # alternated within every round
            timers = [{} for _ in range(args.steps)]
            start = torch.cuda.Event(enable_timing=True)
            end = torch.cuda.Event(enable_timing=True)
            start.record()
            for timed in timers:
                step(mode, timed)
            end.record()
            torch.cuda.synchronize()
            passes[mode].append(start.elapsed_time(end) / args.steps)
            stacks[mode].append(statistics.mean(
                t['conv_frames'][0].elapsed_time(t['conv_frames'][1]) for t in timers))
    name, power_limit = gpu
    lines = []
    base_pass = statistics.median(passes['fp32'])
    base_stack = statistics.median(stacks['fp32'])
    for mode in MODES:
        ms = statistics.median(passes[mode])
        stack_ms = statistics.median(stacks[mode])
        diff = (scores[mode] - scores['fp32']).abs().max().item()
        line = {
            'shape': shape, 'mode': mode,
            'kernels': {k: {0: 'fp32 ffma', 1: 'bf16 tc', 2: 'bf16x3 tc', 3: 'bf16x6 tc'}[v]
                        for k, v in kernels[mode].items()},
            'ms_per_pass': round(ms, 3),
            'ms_per_pass_rounds': [round(v, 3) for v in passes[mode]],
            'frame_stack_ms': round(stack_ms, 3),
            'frame_stack_ms_rounds': [round(v, 3) for v in stacks[mode]],
            'frame_stack_tflops': round(frame_flop / (stack_ms * 1e-3) / 1e12, 2),
            'pass_conv_tflops': round((frame_flop + word_flop) / (ms * 1e-3) / 1e12, 2),
            'max_score_diff_vs_fp32': diff,
            'frames': frames, 'words': n_words, 'utterances': args.utterances,
            'steps': args.steps, 'repeats': args.repeats,
            'gpu': name, 'power_limit': power_limit}
        if mode != 'fp32':
            line['speedup_vs_fp32'] = round(base_pass / ms, 2)
            line['frame_stack_speedup_vs_fp32'] = round(base_stack / stack_ms, 2)
            line['bar'] = BARS[mode]
            line['within_bar'] = diff < BARS[mode]
        lines.append(line)
    return lines


def main():
    args = parse_args()
    import bench
    import emphases_b200 as emphases
    from emphases_b200 import engine

    if not torch.cuda.is_available():
        raise SystemExit('conv_kernel_size_bench: no CUDA device')
    torch.cuda.set_device(0)
    gpu = card()
    lengths, times = bench.corpus_layout(args.utterances, seed=1234)
    device_audio, _ = bench.make_audio(lengths, seed=99, device=torch.device('cuda', 0))
    lines = []
    for shape in SHAPES:
        for line in run_shape(emphases, engine, shape, lengths, times, device_audio, args, gpu):
            print(json.dumps(line), flush=True)
            lines.append(line)
    emphases.reset_configuration()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as file:
        for line in lines:
            file.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
