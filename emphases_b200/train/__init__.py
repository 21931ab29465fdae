"""emphases.train: the training loop and its command line
(`python -m emphases_b200.train`)"""
from .core import checkpoint_state, checkpoints, evaluate, latest_checkpoint, rank_batches, train
