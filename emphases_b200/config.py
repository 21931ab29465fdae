"""Configuration constants of the hot path, same names and defaults as the
reference (emphases/config/defaults.py, emphases/config/static.py).

Like the reference, code reads them at call time as `emphases_b200.NAME`, so
`emphases_b200.configure(...)` (the stand-in for yapecs' `--config file.py`
override, emphases/__init__.py:10-11) takes effect immediately.
"""
from pathlib import Path

import torch

# Metadata (defaults.py:14)
CONFIG = 'emphases'

# Directories (defaults.py:22-41), only read by evaluate.datasets
ASSETS_DIR = Path(__file__).parent / 'assets'
CACHE_DIR = Path(__file__).parent.parent / 'data' / 'cache'
EVAL_DIR = Path(__file__).parent.parent / 'eval'
PARTITION_DIR = ASSETS_DIR / 'partitions'

# Audio parameters (defaults.py:53-74)
HOPSIZE = 160
NUM_FFT = 1024
NUM_MELS = 80
SAMPLE_RATE = 16000
WINDOW_SIZE = 1024

# Data parameters (defaults.py:89-116)
MEL_FEATURE = True
LOUDNESS_FEATURE = False
PITCH_FEATURE = False
PERIODICITY_FEATURE = False
NORMALIZE = False
RANDOM_SEED = 0

# Model parameters (defaults.py:181-215)
ACTIVATION_FUNCTION = torch.nn.ReLU
ARCHITECTURE = 'convolution'
CHANNELS = 80
DECODER_KERNEL_SIZE = 3
DROPOUT = None
DOWNSAMPLE_LOCATION = 'intermediate'
DOWNSAMPLE_METHOD = 'sum'
ENCODER_KERNEL_SIZE = 3
LAYERS = 6
METHOD = 'neural'
UPSAMPLE_METHOD = 'linear'

# Training parameters (defaults.py:224-230)
BUCKETS = 2
LOSS = 'bce'
MAX_TRAINING_FRAMES = 75000
# Training loop (emphases_b200.train).  The reference's emphases/train/core.py
# is not in this repository; these are the values SURVEY.md section 2, row 8
# records for it
NUM_STEPS = 6000
EVALUATION_INTERVAL = 100
LEARNING_RATE = 1e-3

# emphases_b200 extensions (not in the reference)
# 'bf16x6' (default): tcgen05 tensor-core conv stacks with hi/mid/lo-split bf16
# operands (6 MMAs per product, all 24 mantissa bits of both operands):
# fp32-grade, scores within 1e-5 of the reference's fp32 forward (measured
# 8.6e-7).  'bf16x3': hi/lo split (3 MMAs per product, 16 mantissa bits per
# operand): within 2e-5 (measured 5.7e-6).  'bf16': plain bf16 operands, the
# reference's own autocast precision class, within 2e-3, fastest (the word
# decoder then runs as bf16x3).  'fp32': CUDA-core FFMA conv stacks, within
# 1e-5, 6x slower than 'bf16x6'.  Conv shapes the tensor-core kernel is not
# compiled for (channels other than 80, kernel sizes other than 1 and 3)
# always run on the FFMA kernel, whatever the mode.
PRECISION = 'bf16x6'
# Upper bound on packed frame rows per launch (~1 KB of HBM per row).  A corpus
# larger than this runs as several launches on two alternating streams so the
# host->device copy of launch i+1 overlaps the kernels of launch i.
MAX_ROWS_PER_LAUNCH = 1 << 19


def static(namespace):
    """Derived values (emphases/config/static.py:29-46)"""
    namespace['HOPSIZE_SECONDS'] = namespace['HOPSIZE'] / namespace['SAMPLE_RATE']
    namespace['NUM_FEATURES'] = (
        namespace['MEL_FEATURE'] * namespace['NUM_MELS'] +
        int(namespace['PITCH_FEATURE']) +
        int(namespace['PERIODICITY_FEATURE']) +
        int(namespace['LOUDNESS_FEATURE']))
