"""Golden fixtures under tests/golden/ (written by oracle/make_golden.py, read by tests/).

One logical fixture set `name.npz` may be stored as several parts -- `name.npz`, `name.part2.npz`, ... -- so that no
committed file passes 1 MB; `load()` merges them back into one mapping with the `np.load` interface the tests use
(`G[key]`, `G.files`)."""
from __future__ import annotations

import glob
import os
import re

import numpy as np

PART_BYTES = 900_000          # raw array bytes per part; random float64 barely compresses, so this bounds the file size


class GoldenSet(dict):
    @property
    def files(self):
        return list(self)


def _parts(path):
    base = path[:-len(".npz")]
    num = lambda p: int(re.search(r"\.part(\d+)\.npz$", p).group(1))
    return sorted(glob.glob(glob.escape(base) + ".part*.npz"), key=num)


def save(path, arrays):
    """Write `arrays` (insertion order kept) as path plus as many .partN.npz files as needed; stale parts are removed."""
    parts, cur, size = [], {}, 0
    for k, a in arrays.items():
        a = np.asarray(a)
        if cur and size + a.nbytes > PART_BYTES:
            parts.append(cur)
            cur, size = {}, 0
        cur[k] = a
        size += a.nbytes
    parts.append(cur)
    for p in _parts(path):
        os.remove(p)
    for i, p in enumerate(parts):
        np.savez_compressed(path if i == 0 else f"{path[:-len('.npz')]}.part{i + 1}.npz", **p)


def load(path):
    out = GoldenSet()
    for p in [path] + _parts(path):
        with np.load(p) as z:
            out.update((k, z[k]) for k in z.files)
    return out
