"""
The reference's side of the differential fuzz scripts (fuzz_*.py), stored as digests so that the comparison runs without the reference.

Each script draws its cases from fixed seeds, so the cases are the same on every run.  Run with `--record` (where the reference can be
imported, see tests/golden/make_golden.py), a script evaluates the reference on every case and stores one digest per outcome in
tests/golden/reference_fuzz/<script>.json: for a value, a hash of its tensors' dtypes, shapes and bits (or of its plain-Python form);
for an exception, its type name.  Run without it, the script compares this package's outcome on the same case with the stored digest.
Where the reference's result feeds a later step of a case, the scripts use this package's own result there, which is bit-identical to
the reference's whenever its digest matched.
"""
import hashlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
FP8 = torch.float8_e4m3fn


def _canon(v):
    """plain-Python form of a value: tensors by dtype, shape and bits; containers recursively"""
    if isinstance(v, torch.Tensor):
        t = v.detach().cpu().contiguous()
        if t.dtype == FP8:
            t = t.view(torch.uint8)
        elif t.is_floating_point():
            t = t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])
        return ["tensor", str(v.dtype), list(v.shape), hashlib.sha256(t.numpy().tobytes()).hexdigest()]
    if isinstance(v, dict):
        return ["dict", sorted([str(k), _canon(x)] for k, x in v.items())]
    if isinstance(v, (list, tuple)):
        return [_canon(x) for x in v]
    if isinstance(v, torch.dtype):
        return str(v)
    return repr(v)


def digest(v) -> str:
    return hashlib.sha256(json.dumps(_canon(v)).encode()).hexdigest()[:16]


def values_of(t: torch.Tensor):
    """a float tensor up to value equality (-0 == +0), NaN standing for itself: compares like torch.equal on nan_to_num(nan=7)"""
    if t.is_floating_point():
        return str(t.dtype), torch.nan_to_num(t.double(), nan=7.0) + 0.0
    return str(t.dtype), t


class Outcome:
    """`error` is the exception's type name, or None; `key` identifies the value"""

    def __init__(self, error=None, key=None):
        self.error, self.key = error, key

    @property
    def ok(self):
        return self.error is None

    def __eq__(self, other):
        return (self.error, self.key if self.error is None else None) == (other.error, other.key if other.error is None else None)

    def __repr__(self):
        return f"error {self.error}" if self.error else f"value {self.key}"


def evaluate(fn, canon=lambda v: v) -> Outcome:
    """this package's outcome of fn()"""
    try:
        return Outcome(key=digest(canon(fn())))
    except Exception as e:  # noqa: BLE001
        return Outcome(error=type(e).__name__)


class Reference:
    """`recording`: evaluate the reference and store the digests; else replay them in the same order"""

    def __init__(self, script: str):
        self.path = os.path.join(ROOT, "tests", "golden", "reference_fuzz", script + ".json")
        self.recording = "--record" in sys.argv
        if self.recording:
            sys.argv.remove("--record")
            self.parts = {}
        else:
            with open(self.path) as f:
                self.parts = json.load(f)
        self.pos = {}

    def __call__(self, part: str, fn, canon=lambda v: v) -> Outcome:
        """the reference's outcome of fn() (called only when recording)"""
        if self.recording:
            o = evaluate(fn, canon)
            self.parts.setdefault(part, []).append(o.key if o.ok else "!" + o.error)
            return o
        i = self.pos.get(part, 0)
        self.pos[part] = i + 1
        entries = self.parts.get(part, [])
        if i >= len(entries):
            return Outcome(error="<no recorded outcome>")
        e = entries[i]
        return Outcome(error=e[1:]) if e.startswith("!") else Outcome(key=e)

    def finish(self) -> int:
        """store the recording, or count the recorded outcomes the replay did not reach (a sign the cases drifted from the recording)"""
        if self.recording:
            os.makedirs(os.path.dirname(self.path), exist_ok=True)
            with open(self.path, "w") as f:
                json.dump(self.parts, f, indent=0, sort_keys=True)
                f.write("\n")
            return 0
        left = sum(len(v) - self.pos.get(k, 0) for k, v in self.parts.items())
        if left:
            print(f"{left} recorded outcomes were not replayed")
        return left
