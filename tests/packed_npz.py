"""Golden files with thousands of small arrays, stored compactly.

``np.savez_compressed`` spends a zip entry and a .npy header on every array;
for files of many tiny per-case arrays (tests/golden/helpers.npz,
tr_subproblem.npz) that overhead is most of the file.  ``save`` concatenates
the arrays of each dtype into one buffer and records (buffer, offset, shape)
per key; ``Packed`` gives back every array with its dtype, shape and bytes.
"""
import json

import numpy as np

_INDEX = "index"


def save(path, arrays):
    groups, index = {}, {}
    for key, a in arrays.items():
        a = np.asarray(a)
        parts = groups.setdefault(a.dtype.str, [])
        off = sum(p.size for p in parts)
        parts.append(a.ravel())
        index[key] = [a.dtype.str, off, list(a.shape)]
    names = {dt: f"b{i}" for i, dt in enumerate(groups)}
    for v in index.values():
        v[0] = names[v[0]]
    bufs = {names[dt]: np.concatenate(parts) for dt, parts in groups.items()}
    np.savez_compressed(path, **bufs, **{_INDEX: np.array(json.dumps(index))})


class Packed:
    """Read-only mapping over a file written by ``save``.  Like an NpzFile,
    every lookup returns a fresh array, so a caller may modify it in place."""

    def __init__(self, path):
        with np.load(path, allow_pickle=False) as z:
            self._index = json.loads(str(z[_INDEX]))
            self._bufs = {k: z[k] for k in z.files if k != _INDEX}

    def __getitem__(self, key):
        name, off, shape = self._index[key]
        size = int(np.prod(shape, dtype=np.int64))
        return self._bufs[name][off:off + size].reshape(shape).copy()
