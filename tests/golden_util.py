"""Helpers shared by the test modules (golden loading and writing).

A golden set `<name>` is kept small (no file above 1 MB):
- `<name>.npz` holds its arrays, except the large inputs of PARTS, which go to
  `<name>.<part>.npz`: the model weights (`state.*`) to `<name>.state.npz`, an
  input recording (`audio`) to `<name>.audio.npz`;
- an array equal to one stored before it in the same file is stored once,
  `_aliases` lists the (key, stored key) pairs (a freshly built Transformer's
  layers, for one, are copies of each other).
"""
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

PARTS = {
    'state': lambda key: key.startswith('state.'),
    'audio': lambda key: key == 'audio'}


def _read(path):
    with np.load(path) as stored:
        arrays = dict(stored)
    for key, target in arrays.pop('_aliases', ()):
        arrays[str(key)] = arrays[str(target)].copy()
    return arrays


def _write(path, arrays):
    stored, aliases, seen = {}, [], {}
    for key, value in arrays.items():
        value = np.asarray(value)
        fingerprint = (value.dtype.str, value.shape, value.tobytes())
        if fingerprint in seen:
            aliases.append((key, seen[fingerprint]))
        else:
            seen[fingerprint] = key
            stored[key] = value
    if aliases:
        stored['_aliases'] = np.array(aliases)
    np.savez_compressed(path, **stored)


def load_golden(name):
    data = _read(os.path.join(GOLDEN, f'{name}.npz'))
    for part in PARTS:
        path = os.path.join(GOLDEN, f'{name}.{part}.npz')
        if os.path.exists(path):
            data.update(_read(path))
    return data


def save_golden(name, arrays):
    """Write `arrays` as the golden set `name` in the layout load_golden reads"""
    files = {None: {}, **{part: {} for part in PARTS}}
    for key, value in arrays.items():
        part = next((p for p, owns in PARTS.items() if owns(key)), None)
        files[part][key] = value
    for part, members in files.items():
        path = os.path.join(GOLDEN, f'{name}.npz' if part is None else f'{name}.{part}.npz')
        if members or part is None:
            _write(path, members)
        elif os.path.exists(path):
            os.remove(path)


def state_from_golden(data, prefix='state.'):
    return {
        key[len(prefix):]: torch.from_numpy(value)
        for key, value in data.items() if key.startswith(prefix)}


def times_list(array):
    return [(float(a), float(b)) for a, b in array]
