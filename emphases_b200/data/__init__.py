from . import preprocess
from .collate import collate
from .dataset import Dataset, Loader, loader
from .sampler import LengthDataset, Sampler, buckets, sampler
