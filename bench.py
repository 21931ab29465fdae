"""Benchmark of the emphases batched-inference hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--precision fp32|bf16|bf16x3|bf16x6] [--utterances U]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): the default framewise conv model
(80 mels, 6 layers, sum pooling at the intermediate location, random init)
over a synthetic corpus of U = 3000 utterances of 2-20 s of 16 kHz audio with
2.5 words/s synthetic alignments (about 9.2 h of audio, ragged, packed).
A "step" is one pass of the whole path over the whole corpus:
    log-mel -> 7 frame convs -> word pooling -> 6 word convs -> head+sigmoid.

`value`  : audio-seconds per wall-second, inputs resident in HBM (kernel-only);
           with N > 1 (torchrun) every rank runs its own corpus of the same
           size (weak scaling, no data-path collective), max time over ranks.
`e2e`    : the same metric through the API BASELINE.json names for this
           config, emphases_b200.from_files_to_files, on ONE on-disk corpus of
           wav + TextGrid files shared by all N ranks (strong scaling, 8 x the
           kernel corpus so that 8 GPUs have work): file reads, int16 H2D,
           kernels, D2H and the .pt / .TextGrid outputs inside the timing.
           Sub-keys keep the packed-pinned-host-buffer figures of the same
           kernels (`pinned_packed`, `int16_pcm_upload`, `list_of_tensors`).
`roofline`: the dominant kernel (log-mel: framing + FFT + mel + log) from CUDA
           events recorded on the launch stream inside the timed region; DRAM
           traffic and pipe utilisation come from the committed ncu summary
           profiles/kernel_metrics.json (keyed by kernel, with its commit).
`cpu_baseline`: the CPU oracle port of the reference path (its own bf16
           autocast numerics) on a bounded sample, all host threads.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLE_RATE = 16000
HOPSIZE = 160
# Algorithmic work (SURVEY.md section 8d, DESIGN.md)
CONV_FLOP_PER_FRAME = 7 * 2 * 80 * 80 * 3          # 268,800
LOGMEL_BYTES_PER_FRAME = 640 + 320
# fp32 operations the log-mel kernel issues per frame (packed FADD2 / FMUL2 = 2,
# FFMA2 = 4, FFMA = 2 per lane, 32 lanes; FFT + unpack 24.6 k, mel 2.0 k)
LOGMEL_FLOP_PER_FRAME = 26600
POOL_BYTES_PER_FRAME = 320


def kernel_metrics():
    """ncu measurements per kernel (dram bytes per frame, pipe utilisation)
    with the capture they come from: profiles/kernel_metrics.json"""
    path = os.path.join(ROOT, 'profiles', 'kernel_metrics.json')
    try:
        with open(path) as file:
            return json.load(file)['kernels']
    except (OSError, KeyError, ValueError):
        return {}


def parse_args():
    parser = argparse.ArgumentParser()
    parser.add_argument('--gpus', type=int, default=1)
    parser.add_argument(
        '--steps', type=int, default=20,
        help='timed steps of the headline kernel-only loop (the value, ms_per_step and '
             '--dump-outputs); the pinned-host end-to-end legs run max(3, min(K, 10)), '
             'the other legs their own fixed or --transformer-steps counts')
    parser.add_argument('--warmup', type=int, default=3)
    parser.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    parser.add_argument(
        '--precision', default=None, choices=['fp32', 'bf16', 'bf16x3', 'bf16x6'])
    parser.add_argument('--utterances', type=int, default=3000)
    parser.add_argument(
        '--architecture', default='convolution',
        choices=['convolution', 'transformer'],
        help='transformer = BASELINE config 3 (informational, fp32 kernels)')
    parser.add_argument('--cpu-seconds', type=float, default=15.)
    parser.add_argument(
        '--transformer-steps', type=int, default=2,
        help='timed passes of the config-3 (Transformer variant) leg; 0 skips it')
    parser.add_argument('--file-utterances', type=int, default=3000)
    parser.add_argument(
        '--corpus-copies', type=int, default=8,
        help='the shared on-disk corpus of the e2e leg holds this many hard-linked '
             'copies of the --file-utterances base files')
    parser.add_argument(
        '--no-list-api', dest='list_api', action='store_false',
        help='skip the list-of-tensors end-to-end leg')
    parser.add_argument(
        '--dump-outputs', metavar='DIR',
        help='after the timed steps, write the word scores and logits of the last '
             'timed step as DIR/scores.npy and DIR/logits.npy (float32, one value '
             'per word in corpus order; rank r of N > 1 writes scores.rank<r>.npy)')
    args = parser.parse_args()
    if args.steps < 1:
        parser.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        parser.error('--dump-outputs writes the GPU path\'s outputs; not with --impl reference')
    return args


###############################################################################
# Synthetic corpus
###############################################################################


def corpus_layout(utterances, seed):
    """Durations U(2, 20) s (multiple of a hop), W = max(2, floor(2.5 dur))
    words tiling the utterance, every word >= 2 frames"""
    rng = np.random.default_rng(seed)
    samples = (rng.uniform(2., 20., utterances) * SAMPLE_RATE).astype(np.int64)
    samples = samples // HOPSIZE * HOPSIZE
    times = []
    for count in samples:
        duration = count / SAMPLE_RATE
        words = max(2, int(2.5 * duration))
        frames = count // HOPSIZE
        # cut points on a frame grid with >= 2 frames per word, jittered
        # inside the frame so word times are not frame aligned
        cuts = np.sort(rng.choice(
            np.arange(1, frames // 2), size=words - 1, replace=False)) * 2
        cuts = (cuts + rng.uniform(0.05, 0.95, words - 1)) * HOPSIZE / SAMPLE_RATE
        edges = np.concatenate([[0.], cuts, [duration]])
        times.append(np.stack([edges[:-1], edges[1:]], axis=1))
    return samples, times


def make_audio(lengths, seed, device=None, pin=False):
    """0.1 * randn audio packed with aligned utterance offsets"""
    from emphases_b200 import scheduler
    offsets, total = scheduler.PackedAudio.layout(lengths)
    if device is not None:
        generator = torch.Generator(device=device).manual_seed(seed)
        buffer = 0.1 * torch.randn(
            total, generator=generator, device=device, dtype=torch.float32)
        buffer.clamp_(-1, 1)
        return buffer, offsets
    generator = torch.Generator().manual_seed(seed)
    buffer = torch.empty(total, dtype=torch.float32, pin_memory=pin)
    torch.randn(total, generator=generator, out=buffer)
    buffer.mul_(0.1).clamp_(-1, 1)
    return buffer, offsets


def random_state(seed=0, architecture='convolution'):
    """Random-init weights of the default architecture"""
    import emphases_b200 as emphases
    emphases.reset_configuration()
    emphases.configure(ARCHITECTURE=architecture)
    torch.manual_seed(seed)
    return {k: v.detach().clone() for k, v in emphases.Model().state_dict().items()}


###############################################################################
# Clocks
###############################################################################


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML
    polled every ~5 ms from a thread (nvidia-smi -lms as a fallback)"""

    REASONS = {
        'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'sw_thermal_slowdown': 0x20,
        'hw_thermal_slowdown': 0x40}
    QUERY = (
        'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
        'clocks_event_reasons.hw_thermal_slowdown,'
        'clocks_event_reasons.sw_thermal_slowdown,'
        'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.sm, self.sm_max, self.reasons = [], [], set()
        self.stop_flag = threading.Event()
        self.thread = None
        self.process = None
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            physical = self.index
            if visible:
                entries = [v.strip() for v in visible.split(',') if v.strip()]
                if self.index < len(entries) and entries[self.index].isdigit():
                    physical = int(entries[self.index])
            handle = pynvml.nvmlDeviceGetHandleByIndex(physical)
            maximum = pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM)

            def poll():
                while not self.stop_flag.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(
                            handle, pynvml.NVML_CLOCK_SM)))
                        self.sm_max.append(float(maximum))
                        mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                        for name, bit in self.REASONS.items():
                            if mask & bit:
                                self.reasons.add(name)
                    except pynvml.NVMLError:
                        pass
                    time.sleep(0.005)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            self.source = 'nvml'
            return
        except Exception:
            self.source = None
        try:
            self.process = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.QUERY}', f'--id={self.index}',
                 '--format=csv,noheader,nounits', '-lms', '50'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.lines = []
            self.thread = threading.Thread(
                target=lambda: self.lines.extend(self.process.stdout), daemon=True)
            self.thread.start()
            self.source = 'nvidia-smi'
        except OSError:
            self.process = None

    def stop(self):
        self.stop_flag.set()
        if self.process is not None:
            self.process.terminate()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if self.source == 'nvidia-smi':
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                     'sw_power_cap']
            for line in self.lines:
                fields = [f.strip() for f in line.split(',')]
                if len(fields) < 7:
                    continue
                try:
                    self.sm.append(float(fields[0]))
                    self.sm_max.append(float(fields[1]))
                except ValueError:
                    continue
                for name, value in zip(names, fields[3:7]):
                    if value.lower().startswith('active'):
                        self.reasons.add(name)
        if not self.sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        return {
            'sm_mhz': statistics.median(self.sm),
            'sm_max_mhz': max(self.sm_max),
            'samples': len(self.sm),
            'source': self.source,
            'reasons': sorted(self.reasons)}


###############################################################################
# CPU baseline (oracle port of the reference path)
###############################################################################


def cpu_reference_pass(
    state, lengths, times, seed, budget_seconds, max_items, packed=None,
    architecture='convolution'
):
    """Time oracle.from_alignment_and_audio (reference numerics: bf16 autocast,
    per-utterance serial loop, emphases/core.py:169-179) over the first
    utterances of the corpus until `budget_seconds` of CPU work."""
    from oracle import emphases_oracle as oracle
    torch.set_num_threads(os.cpu_count() or 1)
    basis = oracle.mel_basis()
    generator = torch.Generator().manual_seed(seed)
    audios = []
    for index, count in enumerate(lengths[:max_items]):
        if packed is not None:
            audios.append(packed[index].clone())
        else:
            audios.append((0.1 * torch.randn(
                1, int(count), generator=generator)).clamp(-1, 1))
    config = {'ARCHITECTURE': architecture}
    if architecture == 'transformer':
        state = dict(state)
        for prefix in ('frame_encoder', 'word_decoder'):
            state.setdefault(
                f'{prefix}.position.encoding', oracle.positional_encoding(80))
    oracle.from_alignment_and_audio(                       # warm up
        [tuple(t) for t in times[0].tolist()], audios[0], state, config,
        basis=basis, autocast=True)
    seconds = words = 0.
    items = 0
    start = time.perf_counter()
    for audio, word_times in zip(audios, times):
        oracle.from_alignment_and_audio(
            [tuple(t) for t in word_times.tolist()], audio, state, config,
            basis=basis, autocast=True)
        seconds += audio.shape[-1] / SAMPLE_RATE
        words += len(word_times)
        items += 1
        if time.perf_counter() - start > budget_seconds:
            break
    elapsed = time.perf_counter() - start
    return seconds, words, items, elapsed


###############################################################################
# Main
###############################################################################


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (the
    oracle port; the Python reference cannot travel to the GPU box), all host
    threads, each step a bounded sample of the workload.  Rank 0 only."""
    if rank != 0:
        return
    lengths, times = corpus_layout(args.utterances, seed=1234)
    state = random_state(architecture=args.architecture)
    per_step = min(300, args.utterances)
    for _ in range(args.warmup):
        cpu_reference_pass(
            state, lengths, times, 99, 1e9, per_step,
            architecture=args.architecture)
    seconds = words = elapsed = 0.
    for _ in range(args.steps):
        s, w, _, e = cpu_reference_pass(
            state, lengths, times, 99, 1e9, per_step,
            architecture=args.architecture)
        seconds += s
        words += w
        elapsed += e
    value = seconds / elapsed
    cores = torch.get_num_threads()
    sample = (f'first {per_step} utterances of the corpus per step '
              f'({seconds / args.steps:.0f} audio-s), serial per-utterance '
              'loop, bf16 autocast')
    print(json.dumps({
        'impl': 'reference',
        'metric': 'audio-sec/sec',
        'value': value,
        'unit': 'audio-s/s',
        'words_per_s': words / elapsed,
        'n_gpus': args.gpus,
        'steps': args.steps,
        'warmup': args.warmup,
        'ms_per_step': 1e3 * elapsed / args.steps,
        'higher_is_better': True,
        'scaling': 'weak',
        'vs_baseline': None,
        'dtype': 'bf16-autocast(cpu)',
        'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {
            'value': value, 'unit': 'audio-s/s', 'cores': cores,
            'kind': 'port', 'sample': sample},
        'e2e': {
            'value': value, 'unit': 'audio-s/s', 'h2d_bytes_per_step': 0,
            'd2h_bytes_per_step': 0}}))


def corpus_root():
    """tmpfs when present (the files leg measures the path, not a disk)"""
    import tempfile
    base = '/dev/shm' if os.path.isdir('/dev/shm') else tempfile.gettempdir()
    token = os.environ.get('MASTER_PORT', 'single')
    return os.path.join(base, f'emphases_b200_bench_{os.getuid()}_{token}')


def build_corpus(emphases, root, count, copies, state):
    """`count` base utterances (16-bit wav + TextGrid) written once and
    hard-linked `copies` times: one corpus of count * copies files.  Returns
    (text_files, audio_files, prefixes, checkpoint, audio_seconds, words)."""
    import shutil
    from pathlib import Path
    root = Path(root)
    shutil.rmtree(root, ignore_errors=True)
    (root / 'out').mkdir(parents=True)
    lengths, times = corpus_layout(count, seed=4321)
    need = int(lengths.sum()) * 2 * 1.1 + count * copies * 16384
    stats = os.statvfs(root)
    if stats.f_bavail * stats.f_frsize < need:
        raise OSError(f'{root}: {need / 1e9:.1f} GB needed')
    generator = torch.Generator().manual_seed(5)
    for i, (n, t) in enumerate(zip(lengths, times)):
        audio = (0.1 * torch.randn(1, int(n), generator=generator)).clamp(-1, 1)
        emphases.load.save_wav(root / f'u0_{i}.wav', audio)
        emphases.Alignment.from_times(
            [tuple(x) for x in t.tolist()]).save(root / f'u0_{i}.TextGrid')
        for c in range(1, copies):
            os.link(root / f'u0_{i}.wav', root / f'u{c}_{i}.wav')
            os.link(root / f'u0_{i}.TextGrid', root / f'u{c}_{i}.TextGrid')
    torch.save({'model': state}, root / 'checkpoint.pt')
    return corpus_files(root, count, copies)


def corpus_files(root, count, copies):
    from pathlib import Path
    root = Path(root)
    lengths, times = corpus_layout(count, seed=4321)
    names = [f'u{c}_{i}' for c in range(copies) for i in range(count)]
    return (
        [root / f'{name}.TextGrid' for name in names],
        [root / f'{name}.wav' for name in names],
        [root / 'out' / name for name in names],
        root / 'checkpoint.pt',
        float(lengths.sum()) / SAMPLE_RATE * copies,
        int(sum(len(t) for t in times)) * copies,
        int(lengths.sum()) * copies)


def time_files_path(emphases, args, state, rank, world, local_rank, device, barrier):
    """The end-to-end leg: emphases_b200.from_files_to_files (through
    emphases_b200.distributed: every rank takes its LPT shard of the SAME file
    list and writes its own outputs) on one on-disk corpus.  Wall clock
    between barriers, max over ranks by construction."""
    import shutil
    from emphases_b200 import distributed
    root = corpus_root()
    count, copies = args.file_utterances, max(1, args.corpus_copies)
    failure = None
    if rank == 0:
        try:
            build_corpus(emphases, root, count, copies, state)
        except OSError as error:      # e.g. no room: the leg is reported as unavailable
            failure = f'{type(error).__name__}: {error}'
    if world > 1:
        import torch.distributed as dist
        box = [failure]
        dist.broadcast_object_list(box, src=0)
        failure = box[0]
    if failure is not None:
        return {'unavailable': failure}
    try:
        text, audio, prefixes, checkpoint, seconds, words, samples = corpus_files(
            root, count, copies)

        def run():
            distributed.from_files_to_files(
                text, audio, prefixes, checkpoint=checkpoint, gpu=local_rank)
            torch.cuda.synchronize(device)

        run()                               # warm-up: model load, workspaces, page cache
        barrier()
        repeats = 3
        start = time.perf_counter()
        for _ in range(repeats):
            run()
            barrier()
        elapsed = (time.perf_counter() - start) / repeats
        written = len(os.listdir(os.path.join(root, 'out'))) if rank == 0 else None
        barrier()
        # the host side of the same call on its own: everything but the kernels
        # (file reads, parsing, planning, uploads, score download, both writers)
        from emphases_b200 import scheduler as scheduler_module
        scheduler_module.HOST_PATH_PROBE = True
        try:
            run()
            barrier()
            start = time.perf_counter()
            for _ in range(2):
                run()
                barrier()
            host_path = (time.perf_counter() - start) / 2
        finally:
            scheduler_module.HOST_PATH_PROBE = False
        run()                               # the outputs left behind are real scores
        barrier()
        # ceiling of the reader alone: the native reader decoding this
        # rank's shard into pinned memory, all ranks at once, no GPU work
        from emphases_b200 import corpus as corpus_module
        mine = distributed.shard(distributed.audio_costs(audio), rank, world)
        local_world = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))
        threads = max(2, min(32, (os.cpu_count() or 1) // local_world))
        with corpus_module.Corpus(
                [os.fspath(text[i]) for i in mine], [os.fspath(audio[i]) for i in mine],
                threads) as parsed:
            barrier()
            t0 = time.perf_counter()
            indices, _, packed = parsed.load(parsed.usable(None))
            packed.ready(len(indices) - 1)
            barrier()
            ingest = time.perf_counter() - t0
        return {
            'value': seconds / elapsed, 'unit': 'audio-s/s',
            'words_per_s': words / elapsed,
            'ms_per_step': 1e3 * elapsed,
            'files': count * copies, 'ms_per_file': 1e3 * elapsed / (count * copies),
            'audio_hours': seconds / 3600.,
            'h2d_bytes_per_step': int(samples * 2),
            'd2h_bytes_per_step': int(words * 4),
            'h2d_gbs_aggregate': samples * 2 / elapsed / 1e9,
            'host_ingest_gbs_probe': samples * 2 / ingest / 1e9,
            'host_ingest_ms_probe': 1e3 * ingest,
            'host_path_ms_probe': 1e3 * host_path,
            'host_bound_fraction': host_path / elapsed,
            'outputs_written': written,
            'scaling': 'strong',
            'api': 'emphases_b200.distributed.from_files_to_files (one rank per GPU, '
                   'LPT shard of one file list per rank)',
            'note': 'wav + TextGrid read, int16 H2D, inference, D2H, .pt + .TextGrid '
                    'written; wall clock between barriers.  Host-bound: '
                    'host_path_ms_probe is the same call with the kernels skipped '
                    '(reads, parsing, planning, copies, writers), '
                    'host_ingest_*_probe is the native wav reader alone (headers '
                    'already parsed) filling pinned memory on the same cores'}
    finally:
        barrier()
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)


def time_transformer_variant(
    emphases, engine, eng, device, device_audio, plan, views, audio_seconds, steps
):
    """configs[2]: the Transformer-layer variant (padding-masked attention over
    frames, emphases/model/layers/transformer.py:13-52) with random-init
    weights over the SAME packed corpus, inputs resident in HBM"""
    emphases.configure(ARCHITECTURE='transformer')
    torch.manual_seed(0)
    model = emphases.Model().to(device).eval()
    weights = model.packed_weights()
    code = emphases.precision_code()

    def step():
        # (the launch workspace the product path uses, scheduler.run_on_device:
        # no gigabyte allocations per pass)
        return eng.forward_packed(
            device_audio, plan, weights, method='sum', location='intermediate',
            precision=code, views=views, ws=eng.workspace('bench_transformer'))

    step()
    torch.cuda.synchronize(device)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        result = step()
    end.record()
    torch.cuda.synchronize(device)
    ms = start.elapsed_time(end) / steps
    assert torch.isfinite(result['scores']).all()
    del model, weights, result
    return {
        'value': audio_seconds / (ms * 1e-3), 'unit': 'audio-s/s', 'ms_per_step': ms,
        'steps': steps, 'utterances': int(plan.n_seq),
        'workload': 'configs[2]: Transformer-layer variant, same corpus, kernel-only',
        'note': ('per layer: fused q/k/v, out-projection + LayerNorm and feed-forward + '
                 'LayerNorm passes (csrc/transformer_tc.cu, split-bf16 mma.sync) around '
                 'tensor-core attention (csrc/attention_tc.cu: fp16 operands in the bf16 mode, '
                 'split bf16 in the fp32-grade modes)')}


def synthetic_training_batch(seed, max_frames=75000):
    """A padded batch shaped like the reference's collate (B * Tmax <=
    MAX_TRAINING_FRAMES = 75,000 frames, emphases/config/defaults.py;
    utterances U(2, 20) s, 2.5 words/s)"""
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


def time_train_step(emphases, rank, world, device, barrier, steps=20, warmup=5):
    """configs[4]: forward + backward (BCE on word scores) + NCCL gradient
    all-reduce + Adam on one synthetic collate-shaped batch per rank (weak
    scaling); CUDA events, max over ranks"""
    from emphases_b200 import training
    saved = {key: getattr(emphases, key) for key in ('PRECISION',)}
    torch.manual_seed(0)
    model = emphases.Model().to(device)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)
    batch = synthetic_training_batch(100 + rank)
    batch = (batch[0].to(device),) + batch[1:4] + (batch[4].to(device),)
    frames = int(batch[1].sum())
    for _ in range(warmup):
        value = training.train_step(model, optimizer, batch)
    barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        value = training.train_step(model, optimizer, batch)
    end.record()
    barrier()
    ms = start.elapsed_time(end) / steps
    stats = torch.tensor([ms, frames], dtype=torch.float64, device=device)
    if world > 1:
        import torch.distributed as dist
        worst, total = stats.clone(), stats.clone()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        dist.all_reduce(total, op=dist.ReduceOp.SUM)
        ms, frames_total = worst[0].item(), total[1].item()
    else:
        frames_total = frames
    emphases.configure(**saved)
    return {
        'ms_per_step': ms, 'frames_per_s': frames_total / (ms * 1e-3),
        'value': frames_total / 100. / (ms * 1e-3), 'unit': 'audio-s/s',
        'scaling': 'weak', 'n_gpus': world,
        'batch': {'utterances': int(batch[0].shape[0]), 'tmax': int(batch[0].shape[2]),
                  'frames': frames,
                  'padded_frames': int(batch[0].shape[0] * batch[0].shape[2])},
        'loss': float(value),
        'precision': (f'{training.TRAIN_PRECISION} forward / input gradients, fp32 weight '
                      'gradients, Adam'),
        'workload': ('configs[4]: forward + backward + BCE on word scores + NCCL gradient '
                     'all-reduce (flat buffer, in place) + optimizer step, one '
                     'collate-shaped batch per rank')}


def time_single_utterance(emphases, model, gpu, calls=200):
    """configs[0] on the GPU: emphases_b200.from_alignment_and_audio on one
    10 s utterance with a 25-word alignment (the native single-utterance call,
    csrc/utterance.cu), pageable host audio in, scores read back to the host:
    median wall time per call"""
    import tempfile
    generator = torch.Generator().manual_seed(11)
    audio = (0.1 * torch.randn(1, 10 * SAMPLE_RATE, generator=generator)).clamp(-1, 1)
    cuts = torch.sort(torch.rand(24, generator=generator) * 10).values.tolist()
    edges = [0.] + cuts + [10.]
    alignment = emphases.Alignment.from_times(list(zip(edges[:-1], edges[1:])))
    with tempfile.TemporaryDirectory() as directory:
        checkpoint = os.path.join(directory, 'checkpoint.pt')
        torch.save({'model': model.state_dict()}, checkpoint)
        samples = []
        for index in range(calls + 20):
            torch.cuda.synchronize()
            start = time.perf_counter()
            emphases.from_alignment_and_audio(
                alignment, audio, SAMPLE_RATE, checkpoint=checkpoint, gpu=gpu).cpu()
            if index >= 20:
                samples.append(time.perf_counter() - start)
    median = statistics.median(samples)
    return {
        'ms_per_call': 1e3 * median, 'value': 10. / median, 'unit': 'audio-s/s',
        'calls': calls, 'workload': 'configs[0]: one 10 s utterance, 25 words',
        'api': 'emphases_b200.from_alignment_and_audio (host audio in, scores on the host out)'}


def dump_outputs(directory, result, plan, rank, world):
    """The word rows of a forward_packed result (separator rows dropped) as
    float32 .npy files, so that two builds can be compared output for output"""
    os.makedirs(directory, exist_ok=True)
    rows = torch.from_numpy(np.flatnonzero(plan.word_seq >= 0)).to(result['scores'].device)
    suffix = '' if world == 1 else f'.rank{rank}'
    for name in ('scores', 'logits'):
        values = result[name].reshape(-1).index_select(0, rows).float().cpu().numpy()
        np.save(os.path.join(directory, f'{name}{suffix}.npy'), values)


def workload_config(args):
    return {
        'workload': (
            ('config2: default framewise conv model'
             if args.architecture == 'convolution' else
             'config3: Transformer-layer variant') +
            f' (80 mel, 6 layers, sum '
            f'pooling @ intermediate, random init) over {args.utterances} '
            'synthetic utterances U(2,20) s @16 kHz, 2.5 words/s, ragged, '
            'one packed batch per GPU'),
        'utterances_per_gpu': args.utterances,
        'l2': 'inputs (packed audio + activations, >2 GB) exceed the 126 MB L2',
        'parallelism': f'utterance-sharded x{args.gpus}, no collective'}


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import emphases_b200 as emphases
    from emphases_b200 import engine, scheduler

    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    numa_cpus = scheduler.bind_to_gpu_numa_node(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)

    precision = args.precision or default_precision()
    state = random_state(architecture=args.architecture)   # resets the configuration
    emphases.configure(PRECISION=precision)

    # ---- corpus: each rank owns its own shard of the same size (weak) ----
    lengths, times = corpus_layout(args.utterances, seed=1234 + rank)
    audio_seconds = float(lengths.sum()) / SAMPLE_RATE
    n_words = int(sum(len(t) for t in times))
    host_audio, offsets = make_audio(lengths, seed=99 + rank, pin=True)
    packed = scheduler.PackedAudio(host_audio, offsets, lengths)
    alignments = times                      # (W, 2) arrays are accepted as-is

    model = emphases.Model()
    model.load_state_dict(state)
    model = model.to(device).eval()
    weights = model.packed_weights()
    eng = emphases.get_engine(device)

    # ---- kernel-only leg: everything resident in HBM ----
    plan = engine.make_plan(
        [(t, int(n)) for t, n in zip(times, lengths)], None, 'sum')
    device_audio = host_audio.to(device)
    views = eng.upload_plan(plan)
    frames = int(plan.n_rows.sum())
    prec_code = emphases.precision_code()

    def step(timed=None):
        return eng.forward_packed(
            device_audio, plan, weights, method='sum',
            location='intermediate', precision=prec_code, views=views,
            timers=timed)

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(max(args.warmup, 3)):
        result = step()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    timers = []
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for _ in range(args.steps):
        timers.append({})
        result = step(timers[-1])
    end.record()
    barrier()
    elapsed_ms = start.elapsed_time(end)
    clock_summary = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result, plan, rank, world)
    del result
    launches_per_step = sum(entry[2] for entry in timers[0].values())
    kernel_ms = {
        name: statistics.mean(t[name][0].elapsed_time(t[name][1]) for t in timers)
        for name in timers[0]}

    # ---- when the pooling runs inside the conv stack's epilogue: the two
    # kernels on their own, for the conv stack's stand-alone tensor fraction ----
    unfused_ms = None
    if rank == 0 and 'pool' not in kernel_ms:
        saved = engine.FUSE_POOLING
        engine.FUSE_POOLING = '0'
        try:
            step()
            samples = [{} for _ in range(3)]
            for sample in samples:
                step(sample)
            torch.cuda.synchronize(device)
            unfused_ms = {
                name: statistics.mean(t[name][0].elapsed_time(t[name][1]) for t in samples)
                for name in ('conv_frames', 'pool')}
        finally:
            engine.FUSE_POOLING = saved

    # ---- the same step in the product's default precision (bf16x6: fp32-grade on
    # the tensor cores); the headline stays the reference's own bf16 class ----
    default_leg = None
    product_default = emphases.config.PRECISION if hasattr(emphases, 'config') else 'bf16x6'
    if rank == 0 and precision != product_default:
        emphases.configure(PRECISION=product_default)
        code = emphases.precision_code()

        def default_step():
            return eng.forward_packed(
                device_audio, plan, weights, method='sum', location='intermediate',
                precision=code, views=views)

        default_step()
        torch.cuda.synchronize(device)
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(3):
            default_step()
        d1.record()
        torch.cuda.synchronize(device)
        default_ms = d0.elapsed_time(d1) / 3
        default_leg = {
            'precision': product_default, 'ms_per_step': default_ms,
            'value': audio_seconds / (default_ms * 1e-3), 'unit': 'audio-s/s',
            'note': ('kernel-only step in the package default PRECISION (scores within 1e-5 '
                     'of the reference fp32 forward); the headline uses the reference\'s own '
                     'inference precision class (bf16 autocast, emphases/core.py:594-610)')}
        emphases.configure(PRECISION=precision)

    # ---- end-to-end leg: host (pinned) audio through the public API ----
    def e2e_step():
        return emphases.from_alignments_and_audio(
            alignments, packed, SAMPLE_RATE, model=model, gpu=local_rank)

    for _ in range(2):
        e2e_step()
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        results = e2e_step()
    torch.cuda.synchronize(device)
    e2e_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    e2e_ms_rank0 = e2e_ms
    assert sum(r.shape[-1] for r in results) == n_words
    # raw pinned host->device bandwidth of this box right now (context for e2e)
    probe = host_audio[:min(host_audio.numel(), 1 << 28)]
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(3):
        probe.to(device, non_blocking=True)
    torch.cuda.synchronize(device)
    pcie_gbs = 3 * probe.numel() * 4 / (time.perf_counter() - t0) / 1e9

    # the same with 16-bit PCM on the host (what wav files hold): half the bytes
    pcm = scheduler.PackedAudio(
        (host_audio * 32768.).round_().clamp_(-32768, 32767).to(torch.int16).pin_memory(),
        offsets, lengths)
    for _ in range(2):
        emphases.from_alignments_and_audio(
            alignments, pcm, SAMPLE_RATE, model=model, gpu=local_rank)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        emphases.from_alignments_and_audio(
            alignments, pcm, SAMPLE_RATE, model=model, gpu=local_rank)
    torch.cuda.synchronize(device)
    e2e_pcm_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    del pcm

    # the reference's calling convention, batched: a LIST of per-utterance
    # (1, T) fp32 CPU tensors in pageable memory (rank 0 only); packing into
    # pinned staging is inside the timed region (native pool, launch by launch,
    # overlapped with the uploads)
    list_ms = None
    if rank == 0 and args.list_api:
        audios = [
            host_audio[o:o + n][None].clone()
            for o, n in zip(offsets.tolist(), lengths.tolist())]
        for _ in range(2):
            emphases.from_alignments_and_audio(
                alignments, audios, SAMPLE_RATE, model=model, gpu=local_rank)
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            emphases.from_alignments_and_audio(
                alignments, audios, SAMPLE_RATE, model=model, gpu=local_rank)
        torch.cuda.synchronize(device)
        list_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
        del audios
    h2d_bytes = host_audio.numel() * 4 + plan.int32_blob().nbytes + plan.n_seq * 8
    d2h_bytes = plan.total_word_rows * 4

    # ---- BASELINE config 1 as a latency: one 10 s utterance, 25 words, host audio
    # in, scores on the host out, through emphases_b200.from_alignment_and_audio ----
    single = None
    if rank == 0:
        single = time_single_utterance(emphases, model, local_rank)

    # ---- BASELINE config 3: the Transformer-layer variant over the same corpus,
    # kernel-only, rank 0 (informational: the conv model is the headline) ----
    transformer_leg = None
    if rank == 0 and args.architecture == 'convolution' and args.transformer_steps > 0:
        transformer_leg = time_transformer_variant(
            emphases, engine, eng, device, device_audio, plan, views, audio_seconds,
            args.transformer_steps)
        emphases.configure(ARCHITECTURE='convolution', PRECISION=precision)

    # ---- BASELINE config 5: the data-parallel training step (every rank) ----
    train_leg = time_train_step(emphases, rank, world, device, barrier)

    # ---- the API BASELINE.json names: from_files_to_files on one shared corpus ----
    files_leg = None
    if args.file_utterances > 0:
        files_leg = time_files_path(
            emphases, args, state, rank, world, local_rank, device, barrier)

    # ---- reduce over ranks: max time, summed units ----
    stats = torch.tensor(
        [elapsed_ms, e2e_ms, audio_seconds, n_words, frames], dtype=torch.float64,
        device=device)
    if world > 1:
        worst = stats.clone()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        total = stats.clone()
        dist.all_reduce(total, op=dist.ReduceOp.SUM)
        elapsed_ms, e2e_ms = worst[0].item(), worst[1].item()
        audio_total, words_total, frames_total = (
            total[2].item(), total[3].item(), total[4].item())
    else:
        audio_total, words_total, frames_total = audio_seconds, n_words, frames

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = elapsed_ms / args.steps
    value = audio_total / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (rank 0's events) ----
    peaks = {}
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peaks = json.load(open(peaks_path))
    tensor_peak = peaks.get('bf16_tflops_sustained', 1400.0)
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    source = ('MEASURED_PEAKS.json (hbm_gbs; bf16_tflops_sustained: kernels '
              'timed inside a long step)' if peaks else 'fallback')
    conv_tflops = frames * CONV_FLOP_PER_FRAME / (kernel_ms['conv_frames'] * 1e-3) / 1e12
    logmel_gbs = frames * LOGMEL_BYTES_PER_FRAME / (kernel_ms['logmel'] * 1e-3) / 1e9
    # (absent when the pooling runs inside the conv stack's last-layer epilogue)
    pool_gbs = (frames * POOL_BYTES_PER_FRAME + n_words * 328) / (
        kernel_ms['pool'] * 1e-3) / 1e9 if 'pool' in kernel_ms else None
    conv_bound = 'tensor (fp32 FFMA mode)' if precision == 'fp32' else 'tensor'
    measured = kernel_metrics()

    def traffic(name, when=True):
        entry = measured.get(name)
        if not when or not entry or 'dram_bytes_per_frame' not in entry:
            return None
        return entry['dram_bytes_per_frame'] * frames

    def ncu_source(name):
        entry = measured.get(name) or {}
        return {k: entry[k] for k in ('capture', 'commit') if k in entry}

    sm_clock_hz = 1e6 * (clock_summary.get('sm_mhz') or peaks.get('sm_max_mhz', 1965.0))
    fp32_peak = 148 * 128 * 2 * sm_clock_hz / 1e12          # TFLOP/s at the clock seen
    logmel_tflops = frames * LOGMEL_FLOP_PER_FRAME / (kernel_ms['logmel'] * 1e-3) / 1e12
    candidates = {
        'logmel': {
            'kernel': 'logmel_kernel (framing + 1024-pt rFFT + mel + log)',
            'bound': 'hbm',
            'achieved': logmel_gbs, 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': logmel_gbs / hbm_peak,
            'traffic': traffic('logmel'),
            # HBM is not what binds this kernel: the FP32 and shared-memory pipes do
            'fp32_frac': logmel_tflops / fp32_peak,
            'fp32_tflops': logmel_tflops, 'fp32_peak_tflops': fp32_peak,
            'pipes_ncu': (measured.get('logmel') or {}).get('pipes'),
            'ncu': ncu_source('logmel'),
            'note': ('packed-fp32 FFT: bound by the shared-memory pipe and the FP32 '
                     'pipe, not by HBM (960 algorithmic B/frame vs ~27 kFLOP/frame), '
                     'DESIGN.md 4.1')},
        'conv_frames': {
            'kernel': ('conv_stack (7 fused frame layers)' if 'pool' in kernel_ms else
                       'conv_stack + word pooling (7 fused frame layers, pooling in '
                       'the last epilogue: frame embeddings never reach HBM)'),
            'bound': conv_bound,
            'achieved': conv_tflops, 'peak': tensor_peak, 'unit': 'TFLOP/s',
            'frac': conv_tflops / tensor_peak,
            'traffic': traffic(
                'conv_frames' if 'pool' in kernel_ms else 'conv_frames_fused',
                precision == 'bf16'),
            'ncu': ncu_source('conv_frames' if 'pool' in kernel_ms else 'conv_frames_fused')}}
    if pool_gbs is not None:
        candidates['pool'] = {
            'kernel': 'pool_words_kernel',
            'bound': 'hbm',
            'achieved': pool_gbs, 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': pool_gbs / hbm_peak, 'traffic': traffic('pool'),
            'ncu': ncu_source('pool')}
    if unfused_ms is not None:
        alone = frames * CONV_FLOP_PER_FRAME / (unfused_ms['conv_frames'] * 1e-3) / 1e12
        candidates['conv_frames']['separate_kernels'] = {
            'conv_frames_ms': unfused_ms['conv_frames'], 'pool_ms': unfused_ms['pool'],
            'conv_tflops': alone, 'conv_frac': alone / tensor_peak,
            'note': ('the same stage as conv stack + pooling kernel '
                     '(EMPHASES_B200_FUSE_POOLING=0), 3 launches outside the timed region')}
    for name, entry in candidates.items():
        entry['ms'] = kernel_ms[name]
        entry['share_of_step'] = kernel_ms[name] / ms_per_step
    dominant = max(candidates, key=lambda name: kernel_ms[name])
    roofline = dict(candidates[dominant])
    roofline['peak_source'] = source
    roofline['others'] = {
        name: entry for name, entry in candidates.items() if name != dominant}
    roofline['kernel_ms'] = kernel_ms

    # ---- CPU baseline on the host cores (rank 0, N = 1 only) ----
    cpu = None
    if world == 1 and args.cpu_seconds > 0:
        seconds, words, items, elapsed = cpu_reference_pass(
            state, lengths, times, 99, args.cpu_seconds, len(lengths), packed,
            architecture=args.architecture)
        cpu = {
            'value': seconds / elapsed,
            'unit': 'audio-s/s',
            'words_per_s': words / elapsed,
            'cores': torch.get_num_threads(),
            'kind': 'port',
            'sample': (
                f'first {items} utterances of the same corpus '
                f'({seconds:.0f} audio-s, {elapsed:.1f} s of CPU work), oracle '
                'port of the reference path with its bf16 autocast, serial '
                'per-utterance loop like emphases/core.py:169-179')}

    pinned = {
        'value': audio_total / (e2e_ms * 1e-3),
        'unit': 'audio-s/s',
        'words_per_s': words_total / (e2e_ms * 1e-3),
        'ms_per_step': e2e_ms,
        'h2d_bytes_per_step': int(h2d_bytes),
        'd2h_bytes_per_step': int(d2h_bytes),
        'h2d_gbs_effective': h2d_bytes / (e2e_ms_rank0 * 1e-3) / 1e9,
        'pinned_h2d_gbs_probe': pcie_gbs,
        'gpu_local_cpus': numa_cpus,
        'scaling': 'weak',
        'api': ('emphases_b200.from_alignments_and_audio(alignments, PackedAudio, '
                'model=...) -- a pre-packed pinned fp32 host buffer per rank'),
        'note': ('PCIe-bound: one pinned H2D of the fp32 audio per '
                 'launch, kernels overlap the next launch copy')}
    extras = {
        'pinned_packed': pinned,
        'int16_pcm_upload': {
            'value': audio_seconds / (e2e_pcm_ms * 1e-3), 'unit': 'audio-s/s',
            'ms_per_step': e2e_pcm_ms, 'note': 'rank 0, same call, int16 host audio'},
        'list_of_tensors': None if list_ms is None else {
            'value': audio_seconds / (list_ms * 1e-3), 'unit': 'audio-s/s',
            'ms_per_step': list_ms,
            'note': ('rank 0, same call with a list of pageable per-utterance '
                     'fp32 tensors: packing to pinned staging included')}}
    if files_leg is not None and 'value' in files_leg:
        # the headline: the API BASELINE.json names for this config
        e2e = dict(files_leg)
        e2e.update(extras)
    else:
        e2e = dict(pinned)
        e2e.update({k: v for k, v in extras.items() if k != 'pinned_packed'})

    print(json.dumps({
        'metric': 'audio-sec/sec',
        'value': value,
        'unit': 'audio-s/s',
        'words_per_s': words_total / (ms_per_step * 1e-3),
        'n_gpus': world,
        'steps': args.steps,
        'warmup': max(args.warmup, 3),
        'ms_per_step': ms_per_step,
        'higher_is_better': True,
        'scaling': 'weak',
        'vs_baseline': None,
        'dtype': {
            'fp32': 'f32',
            'bf16': 'bf16 (tcgen05, f32 accumulate)',
            'bf16x3': 'bf16x3 (tcgen05, hi/lo split operands, f32 accumulate)',
            'bf16x6': 'bf16x6 (tcgen05, hi/mid/lo split operands, f32 accumulate: fp32-grade)'}[precision],
        'data': 'synthetic',
        'config': workload_config(args),
        'clocks': clock_summary,
        'e2e': e2e,
        'files_e2e': files_leg,
        'default_precision': default_leg,
        'single_utterance': single,
        'train_step': train_leg,
        'transformer_variant': transformer_leg,
        'gpu_launches': launches_per_step * args.steps,
        'roofline': roofline,
        'cpu_baseline': cpu}))
    if world > 1:
        dist.destroy_process_group()


def default_precision():
    return os.environ.get('EMPHASES_B200_PRECISION', 'bf16')


if __name__ == '__main__':
    main()
