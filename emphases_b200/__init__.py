"""emphases_b200 -- B200-native (sm_100a) drop-in for the batched inference hot
path of interactiveaudiolab/emphases.

    import emphases_b200 as emphases
    scores = emphases.from_alignment_and_audio(alignment, audio, 16000,
                                               checkpoint=path, gpu=0)

Same public functions, argument names and semantics as emphases/core.py; the
compute runs in hand-written CUDA kernels behind the C ABI declared in
include/emphases_b200.h.  There is no CPU path: `gpu=None` means the current
CUDA device.
"""
from . import config as _config
from .config import *  # noqa: F401,F403

_config.static(globals())

from . import _lib  # noqa: E402
from ._lib import EmphasesB200Error  # noqa: E402,F401

_engines = {}


def configure(source=None, **overrides):
    """Override configuration constants (the stand-in for yapecs'
    `--config file.py`, emphases/__init__.py:10-11).  `source` may be a path
    to a python file of UPPER_CASE assignments or a dict."""
    values = {}
    if isinstance(source, dict):
        values.update(source)
    elif source is not None:
        namespace = {}
        with open(source) as stream:
            exec(compile(stream.read(), str(source), 'exec'), namespace)
        values.update(
            {k: v for k, v in namespace.items() if k.isupper()})
    values.update(overrides)
    globals().update(values)
    _config.static(globals())


def reset_configuration():
    """Restore the reference defaults"""
    globals().update(
        {k: v for k, v in vars(_config).items() if k.isupper()})
    _config.static(globals())


def resolve_device(gpu=None, tensor=None):
    """`gpu` index -> torch.device.  None = the tensor's CUDA device or the
    current CUDA device (the reference maps None to the CPU; this build has
    no CPU path -- the one documented deviation, SURVEY.md section 8b)."""
    import torch
    if gpu is not None:
        return torch.device('cuda', int(gpu))
    if tensor is not None and tensor.device.type == 'cuda':
        return tensor.device
    if not torch.cuda.is_available():
        raise EmphasesB200Error(
            'emphases_b200 needs a CUDA device (B200, sm_100a); there is no '
            'CPU fallback')
    return torch.device('cuda', torch.cuda.current_device())


def get_engine(device):
    """One Engine (device constants, staging buffers) per device"""
    import torch
    from . import engine
    device = torch.device(device)
    if device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    if device not in _engines:
        _engines[device] = engine.Engine(device, NUM_MELS)
    return _engines[device]


def require_mel_features_only():
    """Only the mel feature exists here: pitch / periodicity / loudness are
    disabled by default in the reference (emphases/config/defaults.py) and
    need the `penn` network.  Every entry point that builds or consumes
    features checks this, so that an 81-wide input layer is never fed zeros."""
    if PITCH_FEATURE or PERIODICITY_FEATURE or LOUDNESS_FEATURE or not MEL_FEATURE:
        raise NotImplementedError(
            'pitch / periodicity / loudness features are out of scope: '
            'emphases_b200 computes the mel feature only')


def precision_code():
    if PRECISION == 'fp32':
        return _lib.PREC_FP32
    if PRECISION == 'bf16':
        return _lib.PREC_BF16_TC
    if PRECISION == 'bf16x3':
        return _lib.PREC_BF16X3_TC
    if PRECISION == 'bf16x6':
        return _lib.PREC_BF16X6_TC
    raise ValueError(f'Precision {PRECISION} is not defined')


from .alignment import Alignment, Word, SILENCE  # noqa: E402,F401
from .core import *  # noqa: E402,F401,F403
from .model import Model  # noqa: E402,F401
from . import convert  # noqa: E402,F401
from . import data  # noqa: E402,F401
from . import evaluate  # noqa: E402,F401
from . import load  # noqa: E402,F401
from . import model  # noqa: E402,F401
from . import training  # noqa: E402,F401
from .scheduler import PackedAudio, pack_audio  # noqa: E402,F401
from .training import loss  # noqa: E402,F401
# the training loop; `emphases_b200.train` is the function, as in the reference
from .train import train  # noqa: E402,F401
