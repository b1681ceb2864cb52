"""Golden vectors produced by running the reference (see make_golden.py)."""
import glob
import gzip
import io
import lzma
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))


def _read(path: str):
    opener = lzma.open if path.endswith(".xz") else gzip.open
    with opener(path, "rb") as f:
        return torch.load(io.BytesIO(f.read()), weights_only=True)


def load(name: str):
    """load tests/golden/<name>.pt.gz or <name>.pt.xz (plain tensors / python scalars only); a list of cases too large for one file
    is stored in parts <name>.<i>.pt.xz, returned concatenated"""
    for ext in (".pt.gz", ".pt.xz"):
        if os.path.exists(os.path.join(_HERE, name + ext)):
            return _read(os.path.join(_HERE, name + ext))
    parts = sorted(glob.glob(os.path.join(_HERE, glob.escape(name) + ".*.pt.xz")), key=lambda p: int(p.split(".")[-3]))
    if not parts:
        raise FileNotFoundError(f"no golden vectors named {name!r} in {_HERE}")
    return [case for p in parts for case in _read(p)]
