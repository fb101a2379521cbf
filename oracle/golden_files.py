"""Golden fixtures kept in files of at most 1 MB: ``<stem>.npz`` and, when the arrays do not fit one, ``<stem>.1.npz``,
``<stem>.2.npz`` ... Written by make_golden.py, read by the tests; each array lies whole in exactly one part."""
import glob
import io
import os
import zlib

import numpy as np

MAX_FILE_BYTES = 1 << 20
PART_PAYLOAD = 900_000  # deflated bytes per part: leaves room for the zip headers under MAX_FILE_BYTES


def _paths(directory, stem):
    parts = glob.glob(os.path.join(directory, f"{stem}.[0-9]*.npz"))
    first = os.path.join(directory, f"{stem}.npz")
    return [first] + sorted(parts, key=lambda p: int(p[len(first) - 3:-4]))


def save(directory, stem, arrays):
    """Write ``arrays`` (name -> array) as ``<stem>.npz`` plus as many numbered parts as needed; returns the paths."""
    parts, size = [{}], 0
    for key in sorted(arrays):
        buf = io.BytesIO()
        np.save(buf, np.asarray(arrays[key]))
        n = len(zlib.compress(buf.getvalue()))
        if parts[-1] and size + n > PART_PAYLOAD:
            parts.append({})
            size = 0
        parts[-1][key] = arrays[key]
        size += n
    for old in _paths(directory, stem)[1:]:
        os.remove(old)
    paths = [os.path.join(directory, f"{stem}.npz" if i == 0 else f"{stem}.{i}.npz") for i in range(len(parts))]
    for path, part in zip(paths, parts):
        np.savez_compressed(path, **part)
        if os.path.getsize(path) > MAX_FILE_BYTES:
            raise ValueError(f"{path} is {os.path.getsize(path)} bytes: an array of it alone exceeds {MAX_FILE_BYTES}")
    return paths


def load(directory, stem):
    """name -> array over every part of ``<stem>``."""
    out = {}
    for path in _paths(directory, stem):
        with np.load(path) as f:
            for key in f.files:
                assert key not in out, f"{key} is stored twice"
                out[key] = f[key]
    return out
