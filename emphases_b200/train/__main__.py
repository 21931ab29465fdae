"""python -m emphases_b200.train --datasets NAME [NAME ...] --directory DIR
[--config FILE] [--gpu N]   (emphases/train/__main__.py)

Under torchrun (WORLD_SIZE > 1) every rank joins an NCCL process group and
trains on its LOCAL_RANK GPU; --gpu is then ignored."""
import argparse
import os
from pathlib import Path

import torch

import emphases_b200 as emphases


def parse_args():
    parser = argparse.ArgumentParser(description='Train a model')
    parser.add_argument(
        '--config', type=Path,
        help='Python file of configuration overrides (UPPER_CASE assignments)')
    parser.add_argument(
        '--datasets', nargs='+', required=True,
        help='Datasets of CACHE_DIR / PARTITION_DIR to train on')
    parser.add_argument(
        '--directory', type=Path, required=True,
        help='Directory of the checkpoints and the log; a run resumes from it')
    parser.add_argument('--gpu', type=int, help='GPU index (default: the current device)')
    return parser.parse_args()


def main():
    args = parse_args()
    if args.config is not None:
        emphases.configure(args.config)
    gpu = args.gpu
    distributed = int(os.environ.get('WORLD_SIZE', 1)) > 1
    if distributed:
        import torch.distributed as dist
        gpu = int(os.environ['LOCAL_RANK'])
        torch.cuda.set_device(gpu)
        dist.init_process_group('nccl', device_id=torch.device('cuda', gpu))
    try:
        emphases.train(args.datasets, args.directory, gpu)
    finally:
        if distributed:
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
