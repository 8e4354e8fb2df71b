"""Golden arrays stored as one or more .npz files of at most PART_BYTES of array data each.

`save(stem, arrays)` writes tests/golden/<stem>.npz when everything fits, else <stem>-1.npz, <stem>-2.npz, ...;
`load(stem)` returns the merged {name: array} of whichever form is present.  An array larger than PART_BYTES is
stored as consecutive row blocks named <name>@0, <name>@1, ... and concatenated again on loading."""
from __future__ import annotations

import glob
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PART_BYTES = 900_000          # uncompressed; every stored file stays under 1 MB


def _parts(stem, directory):
    whole = os.path.join(directory, stem + ".npz")
    if os.path.exists(whole):
        return [whole]
    return sorted(glob.glob(os.path.join(directory, glob.escape(stem) + "-[0-9]*.npz")),
                  key=lambda p: int(p[:-4].rsplit("-", 1)[1]))


def exists(stem, directory=GOLD) -> bool:
    return bool(_parts(stem, directory))


def load(stem, directory=GOLD) -> dict:
    parts = _parts(stem, directory)
    assert parts, f"no golden file {stem}.npz or {stem}-N.npz in {directory}"
    out, blocks = {}, {}
    for p in parts:
        with np.load(p) as z:
            for k in z.files:
                if "@" in k:
                    name, i = k.rsplit("@", 1)
                    blocks.setdefault(name, {})[int(i)] = z[k]
                    out.setdefault(name, None)
                else:
                    out[k] = z[k]
    for name, b in blocks.items():
        out[name] = np.concatenate([b[i] for i in range(len(b))])
    return out


def save(stem, arrays: dict, directory=GOLD) -> list:
    for old in _parts(stem, directory):
        os.remove(old)
    flat = {}
    for k, v in arrays.items():
        v = np.asarray(v)
        if v.nbytes > PART_BYTES and v.ndim and v.shape[0] > 1:
            rows = max(1, PART_BYTES // 2 // max(1, v.nbytes // v.shape[0]))
            for i, a in enumerate(range(0, v.shape[0], rows)):
                flat[f"{k}@{i}"] = v[a:a + rows]
        else:
            flat[k] = v
    arrays = flat
    groups, size = [[]], 0
    for k, v in arrays.items():
        n = v.nbytes
        if groups[-1] and size + n > PART_BYTES:
            groups.append([])
            size = 0
        groups[-1].append(k)
        size += n
    names = [stem + ".npz"] if len(groups) == 1 else [f"{stem}-{i + 1}.npz" for i in range(len(groups))]
    paths = []
    for name, keys in zip(names, groups):
        path = os.path.join(directory, name)
        np.savez_compressed(path, **{k: arrays[k] for k in keys})
        assert os.path.getsize(path) < 1_000_000, (path, os.path.getsize(path))
        paths.append(path)
    return paths
