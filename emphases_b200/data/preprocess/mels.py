"""Mirror of emphases/data/preprocess/mels.py:16-59 (`from_audio`)"""
import torch

import emphases_b200 as emphases
from emphases_b200 import engine


def from_audio(audio, gpu=None):
    """Log-mel spectrogram of one chunk: audio (C, L) -> (NUM_MELS, L // 160)

    Channel 0 only (mels.py:48).  Raises RuntimeError when L <= 432, where
    the reference's reflect pad raises (emphases/core.py:413-415 relies on it).
    """
    length = audio.shape[-1]
    plan = engine.feature_plan([length])
    device = emphases.resolve_device(gpu, audio)
    eng = emphases.get_engine(device)
    with torch.cuda.device(device):
        frames = length // emphases.HOPSIZE
        samples = audio[0].detach().to(device, torch.float32).contiguous()
        views = eng.upload_plan(plan)
        row_seq = eng.row_index(
            views['row_start'], views['n_rows'], 1, plan.total_rows)
        rows = eng.logmel(samples, views, plan, row_seq, emphases.NORMALIZE)
        return rows[1:1 + frames].t().contiguous()
