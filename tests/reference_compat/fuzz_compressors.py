"""
Differential fuzz of the compressor plugins (the `compress(state_dict, scheme)` / `decompress(...)` classmethods of the registry) against
the reference's on seeded random weights and schemes (TEST INFRASTRUCTURE), against the reference's outcomes recorded in
tests/golden/reference_fuzz/fuzz_compressors.json (recorded.py; `--record` re-records them, importing the reference as
`compressed_tensors` through tests/golden/make_golden.py).  This package is imported under its own name with its tensor-level front end
rebound to the CPU oracle (oracle_patch.apply), so the comparison covers the host mirror (keys, dtypes, shapes, what is dropped or packed,
block padding, zero-point handling) and the oracle arithmetic together.

    python tests/reference_compat/fuzz_compressors.py [cases] [--record]
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

from recorded import Reference, evaluate  # noqa: E402

REF = Reference("fuzz_compressors")
if REF.recording:
    import make_golden as mg  # noqa: E402,F401  (imports the reference as `compressed_tensors` from a temp copy)
    import compressed_tensors.compressors as RC  # noqa: E402
    import compressed_tensors.quantization as RQ  # noqa: E402
    from compressed_tensors.quantization.utils import calculate_qparams as r_qparams, generate_gparam as r_gparam  # noqa: E402

import oracle_patch  # noqa: E402

oracle_patch.apply("compressed_tensors_b200")
import compressed_tensors_b200.compressors as MC  # noqa: E402
import compressed_tensors_b200.quantization as MQ  # noqa: E402
from compressed_tensors_b200.quantization.utils import calculate_qparams as m_qparams, generate_gparam as m_gparam  # noqa: E402

FP8 = torch.float8_e4m3fn


FORMATS = {
    "pack-quantized": [dict(num_bits=4, type="int"), dict(num_bits=8, type="int"), dict(num_bits=3, type="int")],
    "int-quantized": [dict(num_bits=8, type="int"), dict(num_bits=4, type="int")],
    "float-quantized": [dict(num_bits=8, type="float")],
    "naive-quantized": [dict(num_bits=8, type="int"), dict(num_bits=8, type="float")],
    "nvfp4-pack-quantized": [dict(num_bits=4, type="float", strategy="tensor_group", group_size=16, scale_dtype=FP8, zp_dtype=FP8)],
    "mxfp4-pack-quantized": [dict(num_bits=4, type="float", strategy="group", group_size=32, scale_dtype=torch.uint8, zp_dtype=torch.uint8)],
    "mxfp8-quantized": [dict(num_bits=8, type="float", strategy="group", group_size=32, scale_dtype=torch.uint8, zp_dtype=torch.uint8)],
}


def fuzz_converters(n):
    """AutoAWQConverter.process and FP8BlockDequantizer._create_dequantized_weight (entrypoints/convert/converters/autoawq.py:109-262,
    fp8block_dequantizer.py:111-158) on random checkpoints tensors"""
    if REF.recording:
        from compressed_tensors.entrypoints.convert import AutoAWQConverter as RAwq, FP8BlockDequantizer as RFp8
    from compressed_tensors_b200.entrypoints.convert import AutoAWQConverter as MAwq, FP8BlockDequantizer as MFp8

    rnd = random.Random(22)
    g = torch.Generator().manual_seed(22)
    checked = bad = 0
    for case in range(n):
        gsz = rnd.choice([8, 32, 128])
        k, nn, zp = gsz * rnd.choice([1, 2, 5]), 8 * rnd.choice([1, 3, 8, 65]), rnd.random() < 0.7
        t = {"m.q_proj.qweight": torch.randint(-2 ** 31, 2 ** 31 - 1, (k, nn // 8), generator=g, dtype=torch.int64).to(torch.int32),
             "m.q_proj.scales": (torch.rand(k // gsz, nn, generator=g) * 0.02).to(torch.float16)}
        if zp:
            t["m.q_proj.qzeros"] = torch.randint(-2 ** 31, 2 ** 31 - 1, (k // gsz, nn // 8), generator=g, dtype=torch.int64).to(torch.int32)
        want = REF("converters", lambda: dict(RAwq(group_size=gsz, zero_point=zp).process({a: b.clone() for a, b in t.items()})))
        got = evaluate(lambda: dict(MAwq(group_size=gsz, zero_point=zp).process({a: b.clone() for a, b in t.items()})))
        checked += 1
        if got != want:
            bad += 1
            print(f"converter case {case} k={k} n={nn} g={gsz} zp={zp}: autoawq differs")
        r, c = rnd.choice([8, 130, 256]), rnd.choice([8, 136, 300])
        bs = rnd.choice([(128, 128), (32, 64)])
        dt = rnd.choice([torch.bfloat16, torch.float16])
        w = (torch.randn(r, c, generator=g) * 3).to(FP8)
        si = torch.randn(-(-r // bs[0]), -(-c // bs[1]), generator=g).abs() * 0.01 + 1e-4
        want = REF("converters", lambda: RFp8(weight_block_size=bs, dtype=dt)._create_dequantized_weight(w, si))
        got = evaluate(lambda: MFp8(weight_block_size=bs, dtype=dt)._create_dequantized_weight(w, si))
        checked += 1
        if got != want:
            bad += 1
            print(f"converter case {case} fp8 block {r}x{c} {bs} {dt}: differs")
    return checked, bad


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    c_checked, c_bad = fuzz_converters(max(20, n // 4))
    print(f"converters: {c_checked} checked, {c_bad} mismatches", flush=True)
    rnd = random.Random(21)
    g = torch.Generator().manual_seed(21)
    checked = bad = skipped = 0
    for case in range(n):
        fmt = rnd.choice(list(FORMATS))
        kw = dict(rnd.choice(FORMATS[fmt]))
        if "strategy" not in kw:
            kw["strategy"] = rnd.choice(["tensor", "channel", "group", "block"])
            kw["symmetric"] = rnd.random() < 0.6 or kw["type"] == "float"
            if kw["strategy"] == "group":
                kw["group_size"] = rnd.choice([32, 128])
            if kw["strategy"] == "block":
                kw["block_structure"] = rnd.choice([[128, 128], [16, 32]])
        else:
            kw["symmetric"] = True
        gsz = kw.get("group_size") or 32
        rows, cols = rnd.choice([8, 48, 130, 256]), gsz * rnd.choice([1, 2, 4])
        dt = torch.bfloat16 if fmt.startswith(("nvfp4", "mxfp")) else rnd.choice([torch.bfloat16, torch.float16, torch.float32])
        w = (torch.randn(rows, cols, generator=g) * 10 ** rnd.uniform(-2.5, 0.5)).to(dt)
        r_schema = {}

        def r_make():
            r_schema["args"] = RQ.QuantizationArgs(**kw)
            r_schema["scheme"] = RQ.QuantizationScheme(targets=["Linear"], weights=r_schema["args"], format=fmt)

        try:
            r_ok = REF("schema", r_make).ok
            m_args = MQ.QuantizationArgs(**kw)
            m_scheme = MQ.QuantizationScheme(targets=["Linear"], weights=m_args, format=fmt)
        except Exception:  # noqa: BLE001  (combinations the schema rejects; the schema itself is fuzzed in fuzz_host_mirror.py)
            r_ok = False
        if not r_ok:
            skipped += 1
            continue
        # qparams from the reference's observer rule on the strategy's reduction
        s = kw["strategy"]
        if s == "tensor":
            lo, hi = w.amin().reshape(1), w.amax().reshape(1)
        elif s == "channel":
            lo, hi = w.amin(-1, keepdim=True), w.amax(-1, keepdim=True)
        elif s in ("group", "tensor_group"):
            grp = w.unflatten(-1, (-1, gsz))
            lo, hi = grp.amin(-1), grp.amax(-1)
        else:
            bh, bw = kw["block_structure"]
            pr, pc = (-rows) % bh, (-cols) % bw
            wp = torch.nn.functional.pad(w, (0, pc, 0, pr))
            blk = wp.reshape(wp.shape[0] // bh, bh, wp.shape[1] // bw, bw)
            lo, hi = blk.amin((1, 3)), blk.amax((1, 3))
        state = {"weight": w}
        gs = None
        # qparams by the reference's observer rule; this package's, once they match the reference's bit for bit
        if s == "tensor_group":
            gs = m_gparam(w.amin(), w.amax())
            checked += 1
            if REF("qparams", lambda: r_gparam(w.amin(), w.amax())) != evaluate(lambda: gs):
                bad += 1
                print(f"case {case} {fmt} {kw}: generate_gparam differs")
            state["weight_global_scale"] = gs
        qkw = dict(global_scale=gs) if gs is not None else {}
        scale, zp = m_qparams(lo, hi, m_args, **qkw)
        checked += 1
        if REF("qparams", lambda: r_qparams(lo, hi, r_schema["args"], **qkw)) != evaluate(lambda: (scale, zp)):
            bad += 1
            print(f"case {case} {fmt} {kw}: calculate_qparams differs")
        state["weight_scale"], state["weight_zero_point"] = scale, zp
        if kw["strategy"] == "group" and fmt == "pack-quantized" and rnd.random() < 0.3:
            state["weight_g_idx"] = (torch.arange(cols) // gsz)[torch.randperm(cols, generator=g)].to(torch.int32)
        m_cls = MC.BaseCompressor.get_value_from_registry(fmt)
        r_out = REF("compress", lambda: RC.BaseCompressor.get_value_from_registry(fmt).compress({k: v.clone() for k, v in state.items()}, r_schema["scheme"]))
        m_out = evaluate(lambda: m_cls.compress({k: v.clone() for k, v in state.items()}, m_scheme))
        checked += 1
        if not r_out.ok:
            # the reference rejects the combination: check that the mirror does too
            err = None if m_out.error == r_out.error else f"reference raised {r_out.error}, mirror {m_out}"
        else:
            err = None if m_out == r_out else f"compress: reference {r_out}, mirror {m_out}"
        if err is None and r_out.ok:
            m_compressed = m_cls.compress({k: v.clone() for k, v in state.items()}, m_scheme)     # bit-identical to the reference's

            def back(cls, scheme):
                return cls.decompress({k: (v.clone() if v is not None else None) for k, v in m_compressed.items()}, scheme)

            r_back = REF("decompress", lambda: back(RC.BaseCompressor.get_value_from_registry(fmt), r_schema["scheme"]))
            m_back = evaluate(lambda: back(m_cls, m_scheme))
            checked += 1
            if not r_back.ok or not m_back.ok:
                # both reject (e.g. the reference's shape inference on ragged block grids: the reference with the RuntimeError of a failed
                # broadcast, the mirror with its ValueError up front) = agreement
                err = None if (not r_back.ok and not m_back.ok) else f"decompress: reference {r_back}, mirror {m_back}"
            elif m_back != r_back:
                err = f"decompress: reference {r_back}, mirror {m_back}"
        if err:
            bad += 1
            if bad <= 10:
                print(f"case {case} {fmt} {dt} {rows}x{cols} {kw}: {err}")
    print(f"compressors: {checked} checked, {bad} mismatches ({skipped} schema-rejected cases skipped)", flush=True)
    left = REF.finish()
    sys.exit(1 if (bad or c_bad or left) else 0)


if __name__ == "__main__":
    main()
