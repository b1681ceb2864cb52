"""
Differential fuzz of the CPU oracle against the reference itself (TEST INFRASTRUCTURE).  The committed goldens pin the oracle on fixed
vectors; this runs the same comparison on seeded random cases, against the reference's outcomes recorded in
tests/golden/reference_fuzz/fuzz_oracle.json (recorded.py; `--record` re-records them, importing the reference through
tests/golden/make_golden.py):

    python tests/reference_compat/fuzz_oracle.py [cases] [--record]

  quant   quantize / dequantize / fake_quantize: tensor, channel, group (with and without g_idx), block, token (3-D), tensor_group with a
          global scale, attn_head (4-D); int 2..8 bits symmetric / asymmetric, fp8, fp4; bf16 / fp16 / fp32 inputs, scale dtype equal or not
          (and once more with the scale addressing computed by the PRODUCT's front end, ops._resolve, feeding the oracle's C arithmetic)
  pack    pack_to_int32 / unpack_from_int32 for 1..8 bits on both dims, ragged widths; fp4 nibble pack / unpack; MX scale codes
Prints "<part>: N checked, M mismatches" and exits non-zero on any mismatch.
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

REF = Reference("fuzz_oracle")
if REF.recording:
    import make_golden as mg  # noqa: E402,F401  (imports the reference as `compressed_tensors` from a temp copy)
    from compressed_tensors.compressors.mx_utils import compress_mx_scale, decompress_mx_scale  # noqa: E402
    from compressed_tensors.compressors.nvfp4.helpers import pack_fp4_to_uint8, unpack_fp4_from_uint8  # noqa: E402
    from compressed_tensors.compressors.pack_quantized.helpers import pack_to_int32, unpack_from_int32  # noqa: E402
    from compressed_tensors.quantization import QuantizationArgs as RefArgs  # noqa: E402
    from compressed_tensors.quantization.lifecycle.forward import dequantize, fake_quantize, quantize  # noqa: E402
    from compressed_tensors.utils.helpers import pack_bitmasks, unpack_bitmasks  # noqa: E402
from compressed_tensors_b200.quantization import QuantizationArgs  # noqa: E402

import oracle  # noqa: E402

FP8 = torch.float8_e4m3fn


def product_addressing_quantize(x, scale, zp, args, g_idx, out_dtype):
    import ctypes

    from compressed_tensors_b200 import ops

    p = ops._resolve(x, scale, zp, args, g_idx)
    cd = torch.result_type(x, scale)
    x2 = x.reshape(p.rows, p.cols).contiguous()
    out = torch.empty(p.rows, p.cols, dtype=out_dtype)
    sc = p.scale.contiguous()
    z = p.zp.contiguous() if p.zp is not None else None
    gi = p.g_idx.to(torch.int32).contiguous() if p.g_idx is not None else None
    qt = getattr(args.type, "value", args.type)
    rc = oracle.lib().orc_quantize(oracle._p(x2), oracle.DT[x2.dtype], oracle._p(sc), oracle.DT[sc.dtype], oracle._p(z),
                                   oracle.DT[z.dtype] if z is not None else -1, oracle._p(gi), oracle._p(out), oracle.DT[out.dtype],
                                   ctypes.c_int64(p.rows), ctypes.c_int64(p.cols), ctypes.c_int64(p.rdiv), ctypes.c_int64(p.cdiv),
                                   ctypes.c_int64(p.srs), oracle.DT[cd], 0 if qt == "int" else 1, args.num_bits)
    assert rc == 0
    return out.reshape(x.shape)


def fuzz_quant(n):
    rnd = random.Random(11)
    g = torch.Generator().manual_seed(11)
    bad = checked = 0
    made = {}

    def qargs(**kw):
        made["kw"] = kw
        return QuantizationArgs(**kw)

    def reference(x, s, zp, qdt, g_idx, gs):
        args = RefArgs(**made["kw"])
        q = quantize(x, s, zp, args, dtype=qdt, g_idx=g_idx, global_scale=gs)
        return q, fake_quantize(x, s, zp, args, g_idx=g_idx, global_scale=gs), dequantize(q, s, zp, args=args, g_idx=g_idx, global_scale=gs)

    for case in range(n):
        dt = rnd.choice([torch.bfloat16, torch.float16, torch.float32])
        sdt = dt if rnd.random() < 0.7 else rnd.choice([torch.bfloat16, torch.float16, torch.float32])
        strat = rnd.choice(["tensor", "channel", "group", "group_gidx", "block", "token", "tensor_group", "attn_head"])
        if strat == "tensor_group":
            qtype, nbits, sym = "float", 4, True
        else:
            qtype, nbits = rnd.choice([("int", 4), ("int", 8), ("int", rnd.randint(2, 8)), ("float", 8)])
            sym = rnd.random() < 0.6 or qtype == "float"
        gsz = rnd.choice([16, 32, 128])
        rows = rnd.choice([1, 3, 8, 33])
        cols = gsz * rnd.choice([1, 2, 5]) if strat.startswith(("group", "tensor_group")) else rnd.choice([8, 24, 100, 256])
        shape, g_idx, gs = (rows, cols), None, None
        kw = dict(num_bits=nbits, type=qtype, symmetric=sym)
        if strat == "tensor":
            args, sshape = qargs(strategy="tensor", **kw), (1,)
        elif strat == "channel":
            args, sshape = qargs(strategy="channel", **kw), (rows, 1)
        elif strat in ("group", "group_gidx"):
            args, sshape = qargs(strategy="group", group_size=gsz, **kw), (rows, cols // gsz)
            if strat == "group_gidx":
                g_idx = (torch.arange(cols) // gsz)[torch.randperm(cols, generator=g)].to(torch.int32)
        elif strat == "block":
            bh, bw = rnd.choice([(4, 8), (16, 16), (128, 128), (8, 24)])
            args, sshape = qargs(strategy="block", block_structure=[bh, bw], **kw), (-(-rows // bh), -(-cols // bw))
        elif strat == "token":
            shape = (2, rows, cols)
            args, sshape = qargs(strategy="token", dynamic=True, **kw), (2, rows, 1)
        elif strat == "tensor_group":
            args, sshape = qargs(strategy="tensor_group", group_size=16, scale_dtype=FP8, **kw), (rows, cols // 16)
            gs = torch.tensor([rnd.uniform(0.5, 3000.0)], dtype=torch.float32)
        else:
            shape = (2, 4, rows, cols)
            args, sshape = qargs(strategy="attn_head", **kw), (4, 1, 1)
        x = (torch.randn(shape, generator=g) * 10 ** rnd.uniform(-3, 1)).to(dt)
        qmax = {"int": 2 ** (nbits - 1) - 0.5, "float": 448.0 if nbits == 8 else 6.0}[qtype]
        s = ((torch.rand(sshape, generator=g) + 0.25) * float(x.float().abs().max().clamp_min(1e-6)) / qmax)
        if gs is not None:
            s = (s * gs).clamp(2 ** -9, 448).to(FP8).float()       # an fp8-representable local scale, as the NVFP4 observer produces
        s = s.to(sdt)
        zp = None if sym else torch.randint(-(2 ** (nbits - 1)), 2 ** (nbits - 1), sshape, generator=g).to(torch.int8)
        qdt = torch.int8 if qtype == "int" else (FP8 if nbits == 8 else None)
        okw = dict(strategy=args.strategy, group_size=args.group_size, block_structure=args.block_structure, num_bits=nbits, qtype=qtype,
                   g_idx=g_idx, global_scale=gs)
        wants = [REF("quant", lambda: reference(x, s, zp, qdt, g_idx, gs)[i]) for i in range(3)]
        if not wants[0].ok:       # a combination the reference itself rejects is not a case
            continue
        got_q = oracle.quantize(x, s, zp, dtype=qdt, **okw)
        got = [got_q, oracle.fake_quantize(x, s, zp, **okw),
               oracle.dequantize(got_q, s, zp, strategy=args.strategy, group_size=args.group_size, block_structure=args.block_structure, g_idx=g_idx, global_scale=gs)]
        if gs is None:
            # the PRODUCT's front end (ops._resolve: strategy -> scale addressing, broadcasting, g_idx handling; pure Python) driving the
            # oracle's C arithmetic must land on the reference's result as well
            got.append(product_addressing_quantize(x, s, zp, args, g_idx, got_q.dtype))
            names = ("quantize", "fake_quantize", "dequantize", "quantize via the product's addressing")
            wants.append(wants[0])
        else:
            names = ("quantize", "fake_quantize", "dequantize")
        for name, a, b in zip(names, got, wants):
            checked += 1
            if evaluate(lambda: a) != b:
                bad += 1
                if bad <= 8:
                    print(f"QUANT case {case} {name}: {strat} {dt} scale {sdt} {qtype}{nbits} sym={sym} {tuple(shape)}: {a.dtype}{tuple(a.shape)}, reference {b}")
    return checked, bad


def fuzz_pack(n):
    rnd = random.Random(12)
    g = torch.Generator().manual_seed(12)
    bad = checked = 0

    def check(part, got, want):
        """one comparison; returns `got` (bit-identical to the reference's value when it matched) for the steps that follow"""
        nonlocal bad, checked
        checked += 1
        bad += evaluate(lambda: got) != want
        return got

    for _ in range(n):
        nb = rnd.randint(1, 8)
        shape = (rnd.choice([1, 2, 7, 33]), rnd.choice([1, 8, 31, 32, 100, 257]))
        if rnd.random() < 0.2:
            shape = (3,) + shape
        codes = torch.randint(-(2 ** (nb - 1)), 2 ** (nb - 1), shape, generator=g).to(torch.int8)
        dim = rnd.choice([0, 1]) if len(shape) == 2 else 1
        packed = check("pack", oracle.pack_to_int32(codes, nb, dim), REF("pack", lambda: pack_to_int32(codes, nb, packed_dim=dim)))
        check("pack", oracle.unpack_from_int32(packed, nb, torch.Size(shape), dim),
              REF("pack", lambda: unpack_from_int32(pack_to_int32(codes, nb, packed_dim=dim), nb, torch.Size(shape), packed_dim=dim)))
    e2m1 = torch.tensor([0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0])
    for _ in range(n // 2):
        m, k = rnd.choice([1, 4, 9]), 2 * rnd.choice([1, 8, 33])
        dt = rnd.choice([torch.bfloat16, torch.float16, torch.float32])
        v = (e2m1[torch.randint(0, 8, (m, k), generator=g)] * (torch.randint(0, 2, (m, k), generator=g) * 2 - 1)).to(dt)
        nib = check("fp4", oracle.pack_fp4_to_uint8(v), REF("fp4", lambda: pack_fp4_to_uint8(v)))
        check("fp4", oracle.unpack_fp4_from_uint8(nib, m, k, dt), REF("fp4", lambda: unpack_fp4_from_uint8(pack_fp4_to_uint8(v), m, k, dtype=dt)))
        sc = (2.0 ** torch.randint(-20, 10, (m, k // 2), generator=g).float()).to(rnd.choice([torch.bfloat16, torch.float32]))
        code = check("mx", oracle.compress_mx_scale(sc, torch.uint8), REF("mx", lambda: compress_mx_scale(sc, torch.uint8)))
        check("mx", oracle.decompress_mx_scale(code), REF("mx", lambda: decompress_mx_scale(compress_mx_scale(sc, torch.uint8))))
    for _ in range(n // 2):                       # bitmask bit order (utils/helpers.py:306-343), ragged widths
        shape = (rnd.choice([1, 5, 64]), rnd.choice([1, 7, 8, 9, 63, 64, 200]))
        mask = torch.rand(shape, generator=g) < rnd.random()
        packed = check("bitmask", oracle.pack_bitmasks(mask), REF("bitmask", lambda: pack_bitmasks(mask)))
        check("bitmask", oracle.unpack_bitmasks(packed, list(shape)), REF("bitmask", lambda: unpack_bitmasks(pack_bitmasks(mask), list(shape))))
    return checked, bad


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 400
    total = 0
    for name, fn in (("quant", fuzz_quant), ("pack", fuzz_pack)):
        checked, bad = fn(n)
        total += bad
        print(f"{name}: {checked} checked, {bad} mismatches", flush=True)
    total += REF.finish()
    sys.exit(1 if total else 0)


if __name__ == "__main__":
    main()
