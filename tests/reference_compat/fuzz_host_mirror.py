"""
Differential fuzz of the host mirror against the reference itself (TEST INFRASTRUCTURE), on seeded cases, against the reference's
outcomes recorded in tests/golden/reference_fuzz/fuzz_host_mirror.json (recorded.py; `--record` re-records them, importing the
reference through tests/golden/make_golden.py).

    python tests/reference_compat/fuzz_host_mirror.py [iterations] [--record]

Three parts, each compares outcome AND exception type:
  args     random QuantizationArgs keyword sets (valid and invalid)            -> model_dump()
  schemes  every preset, random QuantizationScheme(weights / input / output)   -> model_dump()
  qparams  calculate_qparams, compute_dynamic_scales_and_zp, generate_gparam   -> bit-equal tensors, INT / FP8 / NVFP4 / MXFP4 / MXFP8 args
Prints one line per part ("<part>: N checked, 0 mismatches") and exits non-zero on any mismatch.
"""
import os
import random
import sys
import warnings

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [HERE, os.path.join(ROOT, "tests", "golden"), ROOT]
from loguru import logger  # noqa: E402

logger.remove()
import torch  # noqa: E402

from recorded import Reference, evaluate, values_of  # noqa: E402

REF = Reference("fuzz_host_mirror")
if REF.recording:
    import make_golden as mg  # noqa: E402,F401  (imports the reference as `compressed_tensors` from a temp copy)
    import compressed_tensors.quantization as R  # noqa: E402
    import compressed_tensors.quantization.quant_scheme as RS  # noqa: E402
    from compressed_tensors.quantization.utils import calculate_qparams as rq, compute_dynamic_scales_and_zp as rd, generate_gparam as rg  # noqa: E402

import compressed_tensors_b200.quantization as M  # noqa: E402
import compressed_tensors_b200.quantization.quant_scheme as MS  # noqa: E402
from compressed_tensors_b200.quantization.utils import calculate_qparams as mq, compute_dynamic_scales_and_zp as md, generate_gparam as mgp  # noqa: E402

FP8 = torch.float8_e4m3fn


def norm(v):
    if isinstance(v, dict):
        return {k: norm(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [norm(x) for x in v]
    v = getattr(v, "value", v)
    return str(v) if isinstance(v, torch.dtype) else v


def fuzz_args(n):
    rnd = random.Random(0)
    space = dict(
        num_bits=[1, 2, 4, 8, 16, 0, 3], type=["int", "float", "INT", "bad"], symmetric=[True, False],
        strategy=[None, "tensor", "channel", "group", "block", "token", "tensor_group", "attn_head", "bad"],
        group_size=[None, -1, 0, 16, 32, 128], block_structure=[None, [128, 128], "128x128", [1], "bad"], dynamic=[False, True, "local"],
        actorder=[None, "group", "weight", "static", "dynamic", True, False], scale_dtype=[None, FP8, torch.bfloat16, "float16", torch.uint8],
        zp_dtype=[None, torch.int8, torch.uint8, FP8], observer=[None, "minmax", "memoryless_minmax", "mse"])
    bad = 0
    for _ in range(n):
        kw = {k: rnd.choice(v) for k, v in space.items() if rnd.random() < 0.6}
        r = REF("args", lambda: (lambda a: (norm(a.model_dump()), str(a.pytorch_dtype())))(R.QuantizationArgs(**kw)))
        m = evaluate(lambda: (lambda a: (norm(a.model_dump()), str(a.pytorch_dtype())))(M.QuantizationArgs(**kw)))
        if r != m:
            bad += 1
            if bad <= 5:
                print("ARGS", kw, "\n  reference", r, "\n  mirror   ", m)
    return n, bad


def fuzz_schemes(n):
    bad = 0
    checked = 0
    if REF("presets", lambda: sorted(RS.PRESET_SCHEMES)) != evaluate(lambda: sorted(MS.PRESET_SCHEMES)):
        bad += 1
        print("PRESET NAMES differ")
    for name in sorted(MS.PRESET_SCHEMES):
        checked += 1
        if REF("presets", lambda: norm(R.preset_name_to_scheme(name, ["Linear"]).model_dump())) != evaluate(lambda: norm(M.preset_name_to_scheme(name, ["Linear"]).model_dump())):
            bad += 1
            print("PRESET", name)
    rnd = random.Random(1)

    def rand_args():
        kw = dict(num_bits=rnd.choice([4, 8]), type=rnd.choice(["int", "float"]), symmetric=rnd.choice([True, False]),
                  strategy=rnd.choice(["tensor", "channel", "group", "block", "token", "tensor_group", "attn_head"]), dynamic=rnd.choice([False, True, "local"]),
                  actorder=rnd.choice([None, "group", "weight"]))
        if kw["strategy"] in ("group", "tensor_group"):
            kw["group_size"] = rnd.choice([16, 32, 128])
        if kw["strategy"] == "block":
            kw["block_structure"] = [128, 128]
        return kw

    for _ in range(n):
        parts = {k: (rand_args() if rnd.random() < 0.7 else None) for k in ("weights", "input_activations", "output_activations")}
        fmt = rnd.choice([None, "pack-quantized", "int-quantized", "float-quantized", "nvfp4-pack-quantized", "dense", "bogus"])

        def run(Q):
            return norm(Q.QuantizationScheme(targets=["Linear"], format=fmt, **{k: (Q.QuantizationArgs(**v) if v else None) for k, v in parts.items()}).model_dump())

        checked += 1
        r, m = REF("schemes", lambda: run(R)), evaluate(lambda: run(M))
        if r != m:
            bad += 1
            if bad <= 5:
                print("SCHEME", parts, fmt, "\n  reference", r, "\n  mirror   ", m)
    return checked, bad


def same_values(pair):
    """qparams compare like torch.equal, NaN standing for itself (fp8 by bits)"""
    return [values_of(t.view(torch.uint8)) if t.dtype == FP8 else values_of(t) for t in pair]


def fuzz_qparams(n):
    rnd = random.Random(3)
    g = torch.Generator().manual_seed(3)
    cfgs = [dict(num_bits=4, type="int", symmetric=True), dict(num_bits=4, type="int", symmetric=False), dict(num_bits=8, type="int", symmetric=True),
            dict(num_bits=8, type="int", symmetric=False), dict(num_bits=8, type="float", symmetric=True),
            dict(num_bits=4, type="float", symmetric=True, strategy="tensor_group", group_size=16, scale_dtype=FP8, zp_dtype=FP8),
            dict(num_bits=4, type="float", symmetric=True, strategy="group", group_size=32, scale_dtype=torch.uint8, zp_dtype=torch.uint8),
            dict(num_bits=8, type="float", symmetric=True, strategy="group", group_size=32, scale_dtype=torch.uint8, zp_dtype=torch.uint8)]
    bad = checked = 0

    for _ in range(n):
        kw = dict(rnd.choice(cfgs))
        kw.setdefault("strategy", rnd.choice(["tensor", "channel", "group", "token"]))
        if kw["strategy"] == "group":
            kw.setdefault("group_size", 32)
        dt = rnd.choice([torch.bfloat16, torch.float16, torch.float32])
        shape = rnd.choice([(1,), (7, 1), (5, 4), ()])
        mag = 10 ** rnd.uniform(-4, 3)
        lo, hi = (-torch.rand(shape, generator=g) * mag).to(dt), (torch.rand(shape, generator=g) * mag).to(dt)
        if rnd.random() < 0.1:
            lo = torch.zeros_like(lo)
        if rnd.random() < 0.1:
            hi = torch.zeros_like(hi)
        gs = None
        if kw["strategy"] == "tensor_group":
            gs = mgp(lo.min(), hi.max())       # once it matches, bit-identical to the reference's
            checked += 1
            if REF("qparams", lambda: same_values([rg(lo.min(), hi.max())])) != evaluate(lambda: same_values([gs])):
                bad += 1
                print("GPARAM", lo.min(), hi.max(), gs)
        extra = dict(global_scale=gs) if gs is not None else {}
        r = REF("qparams", lambda: same_values(rq(lo, hi, R.QuantizationArgs(**kw), **extra)))
        m = evaluate(lambda: same_values(mq(lo, hi, M.QuantizationArgs(**kw), **extra)))
        checked += 1
        if r != m:
            bad += 1
            if bad <= 5:
                print("QPARAMS", kw, dt, shape, r, m)
        x = (torch.randn(rnd.choice([(2, 3, 64), (4, 64), (64,)]), generator=g) * mag).to(dt)
        kd = dict(kw, dynamic=True)
        r = REF("qparams", lambda: same_values(rd(value=x, args=R.QuantizationArgs(**kd), module=torch.nn.Identity(), **extra)))
        m = evaluate(lambda: same_values(md(value=x, args=M.QuantizationArgs(**kd), module=torch.nn.Identity(), **extra)))
        checked += 1
        if r != m:
            bad += 1
            if bad <= 5:
                print("DYNAMIC", kd, dt, tuple(x.shape), r, m)
    return checked, bad


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
    total_bad = 0
    for name, fn, k in (("args", fuzz_args, 4 * n), ("schemes", fuzz_schemes, 2 * n), ("qparams", fuzz_qparams, n)):
        checked, bad = fn(k)
        total_bad += bad
        print(f"{name}: {checked} checked, {bad} mismatches", flush=True)
    total_bad += REF.finish()
    sys.exit(1 if total_bad else 0)


if __name__ == "__main__":
    main()
