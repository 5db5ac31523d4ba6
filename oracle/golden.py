"""Reading and writing the fixtures under tests/golden/ so that no file exceeds 1 MB.

A fixture `name.npz` is stored as `name.npz`, `name.1.npz`, `name.2.npz`, ... each holding at most PART_BYTES of
compressed data.  An array too large for one part is cut along its first axis into pieces stored as `key#0`, `key#1`,
...; load() merges the parts and joins the pieces back into one dict.  TEST INFRASTRUCTURE ONLY.
"""
import os
import zlib

import numpy as np

PART_BYTES = 900_000


def _parts(path):
    stem = path[:-len(".npz")]
    return [path] + [f"{stem}.{i}.npz" for i in range(1, 100)]


def _pieces(arrays):
    for k, v in arrays.items():
        v = np.asarray(v)
        n = len(zlib.compress(v.tobytes(), 6))
        if n <= PART_BYTES:
            yield k, v, n
            continue
        for i, piece in enumerate(np.array_split(v, -(-n // PART_BYTES) + 1)):
            yield f"{k}#{i}", piece, len(zlib.compress(piece.tobytes(), 6))


def save(path, arrays):
    parts, size = [{}], 0
    for k, v, n in _pieces(arrays):
        if parts[-1] and size + n > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += n
    for p in _parts(path):
        if os.path.exists(p):
            os.remove(p)
    for p, part in zip(_parts(path), parts):
        np.savez_compressed(p, **part)
        assert os.path.getsize(p) < 1_000_000, p


def load(path):
    """The fixture as a dict of arrays, all parts merged and split arrays joined."""
    out, pieces = {}, {}
    for p in _parts(path):
        if not os.path.exists(p):
            break
        with np.load(p) as z:
            for k in z.files:
                if "#" in k:
                    key, i = k.rsplit("#", 1)
                    pieces.setdefault(key, {})[int(i)] = z[k]
                else:
                    out[k] = z[k]
    for key, ps in pieces.items():
        out[key] = np.concatenate([ps[i] for i in range(len(ps))])
    return out
