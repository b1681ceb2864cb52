"""
Differential fuzz of `ModelCompressor` against the reference's (TEST INFRASTRUCTURE): the same seeded random small model and
quantization config go through apply_quantization_config -> (identical qparams) -> ModelCompressor.from_pretrained_model ->
compress_model -> update_config -> decompress_model in this package (its tensor-level front end rebound to the CPU oracle), against
the reference's outcomes recorded in tests/golden/reference_fuzz/fuzz_model_compressor.json (recorded.py; `--record` re-records them,
importing the reference as `compressed_tensors` through tests/golden/make_golden.py).  Compared: every module's state dict after
initialisation, after compress (keys, dtypes, shapes, bits), the `quantization_config` written to config.json, and every module's state
dict after decompress.

    python tests/reference_compat/fuzz_model_compressor.py [models] [--record]
"""
import copy
import json
import os
import random
import sys
import tempfile
import warnings

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [HERE, os.path.join(ROOT, "tests", "golden"), ROOT]
from loguru import logger  # noqa: E402

logger.remove()
import torch  # noqa: E402

from recorded import Reference, evaluate  # noqa: E402

REF = Reference("fuzz_model_compressor")
if REF.recording:
    import make_golden as mg  # noqa: E402,F401
    import compressed_tensors as R  # noqa: E402
    import compressed_tensors.quantization as RQ  # noqa: E402
    from compressed_tensors.utils import get_direct_state_dict as r_state  # noqa: E402

import oracle_patch  # noqa: E402

oracle_patch.apply("compressed_tensors_b200")
import compressed_tensors_b200 as M  # noqa: E402
import compressed_tensors_b200.quantization as MQ  # noqa: E402
from compressed_tensors_b200.quantization.utils import calculate_qparams as m_qparams, generate_gparam as m_gparam  # noqa: E402
from compressed_tensors_b200.utils import get_direct_state_dict as m_state  # noqa: E402

PRESETS = ["W4A16", "W4A16_ASYM", "W8A16", "W8A8", "W4A8", "FP8", "FP8_DYNAMIC", "FP8_BLOCK", "NVFP4A16", "NVFP4", "MXFP4A16", "MXFP4"]


def build(rnd, seed):
    torch.manual_seed(seed)
    model = torch.nn.Sequential()
    n = rnd.randint(1, 5)
    for i in range(n):
        model.add_module(f"proj{i}", torch.nn.Linear(128 * rnd.choice([1, 2, 3]), 128 * rnd.choice([1, 2]), bias=rnd.random() < 0.3).to(torch.bfloat16))
    model.add_module("norm", torch.nn.LayerNorm(128).to(torch.bfloat16))
    model.add_module("lm_head", torch.nn.Linear(128, 64, bias=False).to(torch.bfloat16))
    return model


def calibrate(model):
    """memoryless min-max weights observer with the reference's rule (this package's calculate_qparams / generate_gparam, compared with
    the reference's by fuzz_host_mirror.py); returns {module name: {param: tensor}} to load into both models"""
    out = {}
    for name, m in model.named_modules():
        scheme = getattr(m, "quantization_scheme", None)
        if scheme is None or scheme.weights is None:
            continue
        a, w = scheme.weights, m.weight.data
        s = a.strategy
        gs = None
        if s == "tensor":
            lo, hi = w.amin().reshape(1), w.amax().reshape(1)
        elif s == "channel":
            lo, hi = w.amin(-1, keepdim=True), w.amax(-1, keepdim=True)
        elif s in ("group", "tensor_group"):
            grp = w.unflatten(-1, (-1, a.group_size))
            lo, hi = grp.amin(-1), grp.amax(-1)
        else:
            bh, bw = a.block_structure
            blk = w.reshape(w.shape[0] // bh, bh, w.shape[1] // bw, bw)
            lo, hi = blk.amin((1, 3)), blk.amax((1, 3))
        q = {}
        if s == "tensor_group":
            gs = m_gparam(w.amin(), w.amax())
            q["weight_global_scale"] = gs
        sc, zp = m_qparams(lo, hi, a, global_scale=gs) if gs is not None else m_qparams(lo, hi, a)
        q["weight_scale"], q["weight_zero_point"] = sc, zp
        for base in ("input", "output"):        # static activation qparams are allocated uninitialised
            for suffix, val in (("scale", 0.5), ("zero_point", 0), ("global_scale", 2.0)):
                if hasattr(m, f"{base}_{suffix}"):
                    q[f"{base}_{suffix}"] = torch.full_like(getattr(m, f"{base}_{suffix}").data, val)
        out[name] = q
    return out


def load_qparams(model, q):
    for name, m in model.named_modules():
        for k, v in q.get(name, {}).items():
            if hasattr(m, k):
                getattr(m, k).data = v.clone().to(getattr(m, k).dtype).reshape(getattr(m, k).shape)


def states(model, fn):
    return {n: {k: v for k, v in fn(m).items()} for n, m in model.named_modules()}


def quantization_config(compressor):
    with tempfile.TemporaryDirectory() as d:
        compressor.update_config(d)
        c = json.load(open(os.path.join(d, "config.json")))["quantization_config"]
    c.pop("version", None)
    return c


def try_decompress(compressor, model, state):
    try:
        compressor.decompress_model(model)
    except Exception:  # noqa: BLE001  (e.g. FP8_BLOCK with an [N, 1] scale grid: dequantize infers CHANNEL and the broadcast fails)
        return "raised"       # both raising, whatever the exception, counts as agreement
    return states(model, state)


STAGES = ("initialized", "compressed", "config.json", "decompressed")


def pipeline(pkg, model, q, state):
    """the four stages of one case: module states after loading the qparams and after compress, the quantization_config, and the
    outcome of decompress"""
    load_qparams(model, q)
    yield states(model, state)
    compressor = pkg.ModelCompressor.from_pretrained_model(model)
    compressor.compress_model(model)
    yield states(model, state)
    yield quantization_config(compressor)
    yield try_decompress(compressor, model, state)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    rnd = random.Random(31)
    checked = bad = 0
    for case in range(n):
        preset = rnd.choice(PRESETS)
        seed = rnd.randint(0, 10 ** 6)
        st = rnd.getstate()
        my_model = build(rnd, seed)
        cfg = dict(config_groups={preset: ["Linear"]}, ignore=["lm_head"])
        MQ.apply_quantization_config(my_model, MQ.QuantizationConfig(**cfg))
        q = calibrate(my_model)
        mine = pipeline(M, my_model, q, m_state)
        if REF.recording:
            rnd.setstate(st)
            ref_model = build(rnd, seed)
            RQ.apply_quantization_config(ref_model, RQ.QuantizationConfig(**cfg))
            ref_stages = pipeline(R, ref_model, q, r_state)
        err = None
        for stage in STAGES:
            r = REF(stage, lambda: next(ref_stages))
            m = evaluate(lambda: next(mine))
            if err is None and r != m:
                err = f"{stage}: reference {r}, mirror {m}"
        checked += 1
        if err:
            bad += 1
            if bad <= 8:
                print(f"model {case} {preset}: {err}")
    print(f"model_compressor: {checked} models checked, {bad} mismatches", flush=True)
    left = REF.finish()
    sys.exit(1 if (bad or left) else 0)


if __name__ == "__main__":
    main()
