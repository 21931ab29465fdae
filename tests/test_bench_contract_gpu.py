"""bench.py's JSON line on a small workload: every key the driver and the
judge read is present and consistent."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_contract():
    result = subprocess.run(
        [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3', '--warmup', '3',
         '--utterances', '150', '--cpu-seconds', '1', '--file-utterances', '20'],
        cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert result.returncode == 0, result.stderr[-2000:]
    lines = [line for line in result.stdout.splitlines() if line.startswith('{')]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step',
                'higher_is_better', 'scaling', 'vs_baseline', 'dtype', 'data', 'config',
                'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert key in line, key
    assert line['metric'] == 'audio-sec/sec' and line['n_gpus'] == 1 and line['steps'] == 3
    assert line['vs_baseline'] is None and line['scaling'] == 'weak'
    # kernels per pass: 2 row maps, log-mel, frame stack (+ word-of-row map and
    # fixed-point finish when the pooling is fused, else the pooling kernel),
    # word stack, head
    assert line['gpu_launches'] in (7 * 3, 8 * 3)
    roofline = line['roofline']
    for key in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert key in roofline, key
    assert roofline['bound'] in ('hbm', 'tensor')
    assert abs(roofline['frac'] - roofline['achieved'] / roofline['peak']) < 1e-9
    assert 'conv_frames' in roofline['others'] or 'conv_frames' in roofline['kernel']
    e2e = line['e2e']
    assert e2e['value'] > 0 and e2e['h2d_bytes_per_step'] > 0 and e2e['d2h_bytes_per_step'] > 0
    assert e2e['value'] < line['value']           # copies inside the timed region
    cpu = line['cpu_baseline']
    assert cpu['kind'] == 'port' and cpu['cores'] >= 1 and cpu['value'] > 0 and cpu['sample']
    assert 'sm_mhz' in line['clocks'] and 'reasons' in line['clocks']
    assert 'workload' in line['config']


def test_bench_dump_outputs_match_oracle(tmp_path):
    """--dump-outputs: one score and one logit per word, in corpus order,
    equal to the CPU oracle on the bench's own inputs (fp32-grade bf16x6, so
    that the word-to-word spread of the random-init scores exceeds the
    tolerance and a dropped, extra or misplaced row shows)"""
    import numpy as np
    import torch
    import bench
    from oracle import emphases_oracle as oracle
    result = subprocess.run(
        [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '1',
         '--utterances', '150', '--precision', 'bf16x6', '--cpu-seconds', '0',
         '--transformer-steps', '0', '--file-utterances', '0', '--no-list-api',
         '--dump-outputs', str(tmp_path)],
        cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert result.returncode == 0, result.stderr[-2000:]
    scores = np.load(tmp_path / 'scores.npy')
    logits = np.load(tmp_path / 'logits.npy')
    lengths, times = bench.corpus_layout(150, seed=1234)
    words = np.array([len(t) for t in times])
    assert scores.dtype == np.float32 and scores.shape == (words.sum(),)
    assert logits.dtype == np.float32 and logits.shape == scores.shape
    np.testing.assert_allclose(scores, 1 / (1 + np.exp(-logits)), atol=1e-5)
    audio, offsets = bench.make_audio(lengths, seed=99)
    state = bench.random_state()
    first = np.concatenate([[0], np.cumsum(words)])
    for u in (0, 75, len(lengths) - 1):
        expected = oracle.from_alignment_and_audio(
            [tuple(t) for t in times[u].tolist()],
            audio[offsets[u]:offsets[u] + lengths[u]][None], state)
        got = torch.from_numpy(scores[first[u]:first[u + 1]])
        assert (got - expected.reshape(-1)).abs().max() < 1e-5, u
