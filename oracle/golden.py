"""Golden-vector archives under tests/golden/ (TEST INFRASTRUCTURE).

An archive whose arrays do not fit in MAX_BYTES is stored in parts: <stem>.npz, <stem>.1.npz, <stem>.2.npz, ...,
each a plain .npz below MAX_BYTES holding some of the arrays.  save() writes that layout (oracle/gen_golden.py) and
load() joins it again (the tests), so a test sees every array of the archive under its own name."""
from __future__ import annotations

import io
import os

import numpy as np

MAX_BYTES = 1_000_000           # no file of the repository is larger


def _part_path(path, k):
    return path if k == 0 else path[:-len(".npz")] + f".{k}.npz"


def _serialise(arrays, compressed):
    buf = io.BytesIO()
    (np.savez_compressed if compressed else np.savez)(buf, **arrays)
    return buf.getvalue()


def save(path, compressed=False, **arrays):
    """np.savez / np.savez_compressed of `arrays` into path, continued in numbered parts when it would exceed MAX_BYTES
    (arrays in the order given, each whole in one part)."""
    parts, cur = [], {}
    for name, a in arrays.items():
        cur[name] = np.asarray(a)
        if len(cur) > 1 and len(_serialise(cur, compressed)) > MAX_BYTES:
            del cur[name]
            parts.append(cur)
            cur = {name: np.asarray(a)}
    parts.append(cur)
    for k, part in enumerate(parts):
        data = _serialise(part, compressed)
        if len(data) > MAX_BYTES:
            raise ValueError(f"{_part_path(path, k)}: the array {next(iter(part))} alone exceeds {MAX_BYTES} bytes")
        with open(_part_path(path, k), "wb") as f:
            f.write(data)
    k = len(parts)
    while os.path.exists(_part_path(path, k)):          # parts of an earlier, larger version of the archive
        os.remove(_part_path(path, k))
        k += 1


def load(path):
    """{name: array} of path and all its numbered parts."""
    out, k = {}, 0
    while k == 0 or os.path.exists(_part_path(path, k)):
        with np.load(_part_path(path, k)) as z:
            out.update({name: z[name] for name in z.files})
        k += 1
    return out
