"""Storage of the golden fixtures under ``tests/golden/`` -- TEST INFRASTRUCTURE ONLY.

A fixture is a (nested) dict saved with ``torch.save``.  One that would exceed ``MAX_BYTES`` on disk is
stored as ``NAME.0.pt``, ``NAME.1.pt``, ... instead of ``NAME.pt``: every part holds a list of
``(key path, value)`` entries, dicts too large for one part being split by key, and ``load`` merges the
parts back into the original dict (same keys, same order, same values).
"""
import glob
import io
import os

import torch

MAX_BYTES = 1_000_000


def _nbytes(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.tell()


def _entries(obj, path=()):
    if isinstance(obj, dict) and obj and _nbytes(obj) > MAX_BYTES // 2:
        for k, v in obj.items():
            yield from _entries(v, path + (k,))
    else:
        yield path, obj


def _parts(path):
    stem = path[:-len(".pt")]
    return sorted(glob.glob(glob.escape(stem) + ".[0-9]*.pt"), key=lambda p: int(p[len(stem) + 1:-3]))


def save(obj, path):
    """``torch.save(obj, path)``, or the parts of ``obj`` when one file would exceed ``MAX_BYTES``."""
    for p in _parts(path) + ([path] if os.path.exists(path) else []):
        os.remove(p)
    if _nbytes(obj) <= MAX_BYTES:
        torch.save(obj, path)
        return [path]
    parts, cur = [], []
    for e in _entries(obj):
        if cur and _nbytes(cur + [e]) > MAX_BYTES:
            parts.append(cur)
            cur = []
        if _nbytes([e]) > MAX_BYTES:
            raise ValueError("golden entry %r alone exceeds %d bytes" % (e[0], MAX_BYTES))
        cur.append(e)
    parts.append(cur)
    names = []
    for i, part in enumerate(parts):
        names.append(path[:-len(".pt")] + ".%d.pt" % i)
        torch.save(part, names[-1])
    return names


def load(path):
    """The fixture ``save`` stored under ``path`` (one file or its parts)."""
    if os.path.exists(path):
        return torch.load(path, weights_only=False)
    parts = _parts(path)
    if not parts:
        raise FileNotFoundError(path)
    obj = {}
    for p in parts:
        for keys, value in torch.load(p, weights_only=False):
            d = obj
            for k in keys[:-1]:
                d = d.setdefault(k, {})
            d[keys[-1]] = value
    return obj
