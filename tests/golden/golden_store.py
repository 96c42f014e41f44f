"""The committed golden vectors as split .npz archives, and the OpenBLAS thread count they were produced with.

An archive `<name>` is stored as `<name>.00.npz`, `<name>.01.npz`, ... so that no single file exceeds
MAX_PART_BYTES; `load(name)` reads the parts back as one read-only mapping with the interface the tests use
from `np.load` of a single .npz (`archive[key]`, `archive.files`).
"""
import glob
import io
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# OpenBLAS threads of make_golden.py; the oracle replays its long runs bit for bit only with the same count
# (test_oracle_pinned.golden_blas_threads)
BLAS_THREADS = 8
MAX_PART_BYTES = 1_000_000
_PACK_BYTES = 900_000          # packing target per part: the size estimate leaves out the zip headers


class Archive:
    def __init__(self, parts):
        self._owner = {}
        for part in parts:
            for key in part.files:
                if key in self._owner:
                    raise ValueError(f"{key} is stored in more than one part")
                self._owner[key] = part
        self.files = list(self._owner)

    def __getitem__(self, key):
        return self._owner[key][key]


def part_paths(name, directory=HERE):
    return sorted(glob.glob(os.path.join(directory, f"{name}.[0-9][0-9].npz")))


def load(name, directory=HERE):
    paths = part_paths(name, directory)
    if not paths:
        raise FileNotFoundError(f"no parts of the golden archive {name!r} in {directory}")
    return Archive([np.load(p) for p in paths])


def _compressed_size(a):
    buf = io.BytesIO()
    np.lib.format.write_array(buf, np.asarray(a), allow_pickle=False)
    return len(zlib.compress(buf.getvalue()))


def save(name, arrays, directory=HERE):
    """Writes `arrays` (key -> array, in order) as the parts of archive `name`, replacing any earlier parts."""
    parts, cur, size = [], {}, 0
    for key, a in arrays.items():
        n = _compressed_size(a)
        if cur and size + n > _PACK_BYTES:
            parts.append(cur)
            cur, size = {}, 0
        cur[key] = np.asarray(a)
        size += n
    if cur:
        parts.append(cur)
    for p in part_paths(name, directory):
        os.remove(p)
    paths = []
    for i, part in enumerate(parts):
        path = os.path.join(directory, f"{name}.{i:02d}.npz")
        np.savez_compressed(path, **part)
        if os.path.getsize(path) > MAX_PART_BYTES:
            raise ValueError(f"{path}: {os.path.getsize(path)} bytes > {MAX_PART_BYTES} (an array too large for one part?)")
        paths.append(path)
    return paths
