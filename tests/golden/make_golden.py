#!/usr/bin/env python
"""
Generate the golden input/output vectors in tests/golden/*.pt by IMPORTING THE
REFERENCE (vllm-project/compressed-tensors mounted at /root/reference) and
running its own CPU code path on seeded inputs.

Run (in the build container only; /root/reference does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference package does `from .version import *` and version.py is
generated at build time, so the source tree is copied to a temp dir and a
two-line version.py shim is added (SURVEY.md 8(c)).  No reference source is
copied into this repository; only tensors produced by running it are stored.

Everything stored is a plain dict of tensors / python scalars, loadable with
torch.load(weights_only=True).
"""
import glob
import os
import shutil
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = "/root/reference/src/compressed_tensors"


def import_reference():
    tmp = tempfile.mkdtemp(prefix="ct_ref_")
    shutil.copytree(REF_SRC, os.path.join(tmp, "compressed_tensors"))
    with open(os.path.join(tmp, "compressed_tensors", "version.py"), "w") as f:
        f.write('__version__ = version = "0.0.0+ref"\n__all__=["__version__","version"]\n')
    sys.path.insert(0, tmp)
    import compressed_tensors  # noqa

    assert compressed_tensors.__file__.startswith(tmp)
    return tmp


import_reference()

from compressed_tensors.compressors import BaseCompressor  # noqa: E402
from compressed_tensors.compressors.pack_quantized.helpers import (  # noqa: E402
    pack_to_int32,
    unpack_from_int32,
)
from compressed_tensors.quantization import (  # noqa: E402
    QuantizationArgs,
    QuantizationScheme,
    preset_name_to_scheme,
)
from compressed_tensors.quantization.lifecycle.forward import (  # noqa: E402
    dequantize,
    fake_quantize,
    quantize,
)
from compressed_tensors.quantization.utils import calculate_qparams  # noqa: E402
from compressed_tensors.utils.helpers import pack_bitmasks, unpack_bitmasks  # noqa: E402
from compressed_tensors.utils import semi_structured_conversions as ssc  # noqa: E402
from compressed_tensors.utils.permutations_24 import get_permutations_24  # noqa: E402


MAX_FILE_BYTES = 1 << 20


def save(name, obj):
    """xz-compressed torch.save (load with tests/golden/__init__.py:load); a list of cases that would pass MAX_FILE_BYTES is written in
    parts <stem>.<i>.pt.xz of consecutive cases"""
    import io
    import lzma

    def encode(o):
        buf = io.BytesIO()
        torch.save(o, buf)
        return lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME)

    stem = name[: -len(".pt")]
    data = encode(obj)
    chunks = [(stem + ".pt.xz", data)]
    k = 1
    while max(len(d) for _, d in chunks) > MAX_FILE_BYTES:
        if not isinstance(obj, list) or k >= len(obj):
            raise ValueError(f"{name}: {len(data)} bytes compressed, more than {MAX_FILE_BYTES}")
        k += 1
        step = -(-len(obj) // k)
        chunks = [(f"{stem}.{i}.pt.xz", encode(obj[j:j + step])) for i, j in enumerate(range(0, len(obj), step))]
    for old in [stem + ".pt.gz", stem + ".pt.xz"] + [os.path.basename(p) for p in glob.glob(os.path.join(HERE, stem + ".*.pt.xz"))]:
        if os.path.exists(os.path.join(HERE, old)):
            os.remove(os.path.join(HERE, old))
    for fname, d in chunks:
        with open(os.path.join(HERE, fname), "wb") as f:
            f.write(d)
        print(f"{fname}: {len(d) / 1024:.0f} KiB")


# --------------------------------------------------------------------------- #
# A. pack / unpack
# --------------------------------------------------------------------------- #
def gen_pack():
    g = torch.Generator().manual_seed(1234)
    cases = []
    shapes1 = [(1, 32), (2, 33), (3, 100), (2, 700), (4, 1024), (8, 64), (5, 1), (1, 7)]
    shapes0 = [(9, 2), (33, 5), (100, 3), (64, 16), (7, 1)]
    for bits in range(1, 9):
        lo, hi = -(1 << (bits - 1)), (1 << (bits - 1))
        for shape in shapes1:
            v = torch.randint(lo, hi, shape, dtype=torch.int8, generator=g)
            p = pack_to_int32(v, bits)
            u = unpack_from_int32(p, bits, v.shape)
            assert torch.equal(u, v)
            cases.append(dict(bits=bits, packed_dim=1, value=v, packed=p.contiguous()))
        for shape in shapes0:
            v = torch.randint(lo, hi, shape, dtype=torch.int8, generator=g)
            p = pack_to_int32(v, bits, packed_dim=0)
            u = unpack_from_int32(p, bits, v.shape, packed_dim=0)
            assert torch.equal(u, v)
            cases.append(dict(bits=bits, packed_dim=0, value=v, packed=p.contiguous(), view_shape=list(p.shape),
                              view_contiguous=p.is_contiguous()))
        v = torch.randint(lo, hi, (2, 3, 40), dtype=torch.int8, generator=g)
        p = pack_to_int32(v, bits)
        cases.append(dict(bits=bits, packed_dim=1, value=v, packed=p.contiguous()))
    # out-of-range inputs: pins the scatter_add (sum, not or) semantics
    for bits in (3, 4, 5):
        v = torch.randint(-128, 128, (3, 64), dtype=torch.int8, generator=g)
        cases.append(dict(bits=bits, packed_dim=1, value=v, packed=pack_to_int32(v, bits).contiguous(), out_of_range=True))
    # the literal vectors of tests/test_compressors/test_pack_quant.py:103-131
    for lit, bits in [([[1, 2], [3, 4]], 4), ([[1, 2, 3, 4, 5, 6, 7, 0], [-1, -2, -3, -4, -5, -6, -7, -8]], 4),
                      ([[30, 40], [50, 60]], 8)]:
        v = torch.tensor(lit, dtype=torch.int8)
        cases.append(dict(bits=bits, packed_dim=1, value=v, packed=pack_to_int32(v, bits).contiguous()))
    save("pack.pt", cases)


# --------------------------------------------------------------------------- #
# B. quantize / dequantize / fake_quantize
# --------------------------------------------------------------------------- #
def observer_qparams(x, args):
    """min/max 'observer' exactly like tests/conftest.py:21-102 of the reference"""
    st = args.strategy
    if st == "tensor":
        mn, mx = x.aminmax()
        return calculate_qparams(mn.reshape(1), mx.reshape(1), args)
    if st == "channel":
        mn = x.amin(dim=-1, keepdim=True)
        mx = x.amax(dim=-1, keepdim=True)
        return calculate_qparams(mn, mx, args)
    if st == "token":
        mn = x.amin(dim=-1, keepdim=True)
        mx = x.amax(dim=-1, keepdim=True)
        return calculate_qparams(mn, mx, args)
    if st == "group":
        xr = x.unflatten(-1, (-1, args.group_size))
        return calculate_qparams(xr.amin(-1), xr.amax(-1), args)
    if st == "block":
        bh, bw = args.block_structure
        R, C = x.shape
        nr, nc = -(-R // bh), -(-C // bw)
        xp = torch.zeros(nr * bh, nc * bw, dtype=x.dtype)
        xp[:R, :C] = x
        xb = xp.reshape(nr, bh, nc, bw).transpose(1, 2).reshape(nr, nc, -1)
        return calculate_qparams(xb.amin(-1), xb.amax(-1), args)
    raise ValueError(st)


def gen_quant():
    torch.manual_seed(4321)
    R, C = 12, 256
    base = torch.randn(R, C) * 0.02
    base[0, :8] = torch.tensor([0.0, -0.0, 1e-30, -1e-30, 0.5, -0.5, 1e4, -1e4])
    xs = {"bf16": base.bfloat16(), "fp16": base.half(), "fp32": base.clone()}
    tdt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}
    cases = []

    def add(xname, args, sdt=None, zdt=None, g_idx=None, zero_dim_scale=False, x=None, tag=""):
        x = xs[xname] if x is None else x
        scale, zp = observer_qparams(x.float() if x.dtype != torch.float32 else x, args)
        scale = scale.to(sdt if sdt is not None else x.dtype)
        if zero_dim_scale:
            scale = scale.reshape(())
            zp = zp.reshape(())
        if zdt is not None:
            zp = zp.to(zdt)
        zp_arg = None if args.symmetric and tag != "symzp" else zp
        if args.symmetric and tag == "symzp":
            zp_arg = zp  # zeros, but still goes through the add
        qdtype = args.pytorch_dtype()
        q = quantize(x, scale, zp_arg, args, dtype=qdtype, g_idx=g_idx)
        qf = quantize(x, scale, zp_arg, args, dtype=None, g_idx=g_idx)
        dq = dequantize(q, scale, zp_arg, args=args, g_idx=g_idx)
        dq_inferred = None
        if x.ndim == 2:
            try:
                dq_inferred = dequantize(q, scale, zp_arg, g_idx=g_idx)
            except Exception:
                dq_inferred = None
        fq = fake_quantize(x, scale, zp_arg, args, g_idx=g_idx)
        cases.append(dict(
            x=xname if x is xs[xname] else x, tag=tag,
            args=args.model_dump(mode="json"), scale=scale, zp=zp_arg, g_idx=g_idx,
            q=q, qf=qf, dq=dq, dq_inferred=dq_inferred, fq=fq,
        ))

    strategies = [
        dict(strategy="tensor"),
        dict(strategy="channel"),
        dict(strategy="group", group_size=32),
        dict(strategy="group", group_size=128),
        dict(strategy="block", block_structure=[32, 128]),
        dict(strategy="block", block_structure=[16, 64]),
    ]
    types = [dict(num_bits=4, type="int"), dict(num_bits=8, type="int"), dict(num_bits=8, type="float")]
    for xname in ("bf16", "fp16", "fp32"):
        for st in strategies:
            for ty in types:
                for sym in (True, False):
                    if ty["type"] == "float" and not sym:
                        continue
                    args = QuantizationArgs(symmetric=sym, **st, **ty)
                    add(xname, args)
    # odd bit widths
    for bits in (1, 2, 3, 5, 6, 7):
        for sym in (True, False):
            add("bf16", QuantizationArgs(num_bits=bits, symmetric=sym, strategy="group", group_size=64))
            add("fp32", QuantizationArgs(num_bits=bits, symmetric=sym, strategy="channel"))
    # promotion corner cases of SURVEY Appendix B1
    a4g = QuantizationArgs(num_bits=4, strategy="channel")
    add("bf16", a4g, sdt=torch.float32, tag="scale_fp32_dim")
    add("fp16", a4g, sdt=torch.float32, tag="scale_fp32_dim")
    a4t = QuantizationArgs(num_bits=4, strategy="tensor")
    add("bf16", a4t, sdt=torch.float32, zero_dim_scale=True, tag="scale_fp32_0dim")
    add("fp16", a4t, sdt=torch.float32, zero_dim_scale=True, tag="scale_fp32_0dim")
    add("fp32", a4t, sdt=torch.float32, zero_dim_scale=True, tag="scale_fp32_0dim")
    add("fp16", a4t, sdt=torch.bfloat16, tag="scale_bf16_x_fp16")
    add("fp32", QuantizationArgs(num_bits=8, strategy="channel"), sdt=torch.bfloat16, tag="scale_bf16_x_fp32")
    add("fp32", QuantizationArgs(num_bits=8, type="float", strategy="tensor"), sdt=torch.bfloat16, tag="scale_bf16_x_fp32")
    # zero-point dtypes seen in the reference tests: int32 (test_int_quant.py:48), fp32 (test_fp8_quant.py:49)
    add("fp32", QuantizationArgs(num_bits=8, symmetric=False, strategy="channel"), zdt=torch.int32, tag="zp_int32")
    add("bf16", QuantizationArgs(num_bits=8, symmetric=False, strategy="group", group_size=128), zdt=torch.int32, tag="zp_int32")
    add("fp32", QuantizationArgs(num_bits=8, type="float", strategy="tensor"), zdt=torch.float32, tag="symzp")
    add("bf16", QuantizationArgs(num_bits=8, type="float", strategy="channel"), zdt=torch.bfloat16, tag="symzp")
    add("bf16", QuantizationArgs(num_bits=8, type="float", symmetric=False, strategy="tensor"), tag="fp8_asym")
    add("fp32", QuantizationArgs(num_bits=8, type="float", symmetric=False, strategy="channel"), tag="fp8_asym")
    # activation ordering (g_idx)
    g = torch.Generator().manual_seed(7)
    for gs in (32, 128):
        gi = (torch.arange(C) // gs)[torch.randperm(C, generator=g)].to(torch.int32)
        for sym in (True, False):
            add("bf16", QuantizationArgs(num_bits=4, symmetric=sym, strategy="group", group_size=gs, actorder="group"), g_idx=gi, tag="g_idx")
        add("fp32", QuantizationArgs(num_bits=8, symmetric=False, strategy="group", group_size=gs, actorder="group"), g_idx=gi, tag="g_idx")
    # 3-D activations, token strategy (dynamic path computes qparams like this)
    act = (torch.randn(2, 5, 64) * 3).bfloat16()
    add("bf16", QuantizationArgs(num_bits=8, strategy="token", dynamic=True), x=act, tag="token3d")
    add("bf16", QuantizationArgs(num_bits=8, type="float", strategy="token", dynamic=True), x=act, tag="token3d")
    add("bf16", QuantizationArgs(num_bits=8, type="float", strategy="tensor"), x=act, tag="tensor3d")
    add("bf16", QuantizationArgs(num_bits=4, strategy="group", group_size=32), x=act, tag="group3d")
    # group with a single-row scale [1, C/G] (forward.py:109-117 example 1)
    xg = xs["bf16"]
    a = QuantizationArgs(num_bits=4, strategy="group", group_size=64)
    xr = xg.float().unflatten(-1, (-1, 64))
    sc, zp = calculate_qparams(xr.amin((0, 2)).reshape(1, -1), xr.amax((0, 2)).reshape(1, -1), a)
    sc = sc.bfloat16()
    q = quantize(xg, sc, None, a, dtype=torch.int8)
    cases.append(dict(x="bf16", tag="group_row1", args=a.model_dump(mode="json"), scale=sc, zp=None, g_idx=None,
                      q=q, qf=quantize(xg, sc, None, a), dq=dequantize(q, sc, None, args=a),
                      dq_inferred=dequantize(q, sc, None), fq=fake_quantize(xg, sc, None, a)))
    save("quant.pt", dict(x=xs, cases=cases))


# --------------------------------------------------------------------------- #
# C. exhaustive bit-pattern sweeps (outputs only; inputs are arange patterns)
# --------------------------------------------------------------------------- #
def gen_sweep():
    out = {}
    pat = torch.arange(65536, dtype=torch.int32).to(torch.uint16)
    for name, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16)):
        x = pat.view(dt).reshape(256, 256).clone()
        x[x.isnan()] = 0  # NaN excluded from the bit-exact set (SURVEY B2)
        for sval in (2.0 ** -7, 0.01, 1.0, 37.5):
            s = torch.tensor([sval]).to(dt)
            key = f"{name}/s{sval}"
            a4 = QuantizationArgs(num_bits=4, strategy="tensor")
            out[key + "/int4"] = quantize(x, s, None, a4, dtype=torch.int8)
            a8 = QuantizationArgs(num_bits=8, symmetric=False, strategy="tensor")
            zp = torch.tensor([3], dtype=torch.int8)
            out[key + "/int8zp3"] = quantize(x, s, zp, a8, dtype=torch.int8)
            af = QuantizationArgs(num_bits=8, type="float", strategy="tensor")
            out[key + "/fp8"] = quantize(x, s, None, af, dtype=torch.float8_e4m3fn).view(torch.uint8)
            out[key + "/fq_int4"] = fake_quantize(x, s, None, a4).view(torch.int16)
            out[key + "/fq_fp8"] = fake_quantize(x, s, None, af).view(torch.int16)
    # dequantize: every int8 code / every fp8 code against a few scales
    codes = torch.arange(-128, 128, dtype=torch.int8).reshape(1, 256)
    f8 = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(torch.float8_e4m3fn).reshape(1, 256)
    for name, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16), ("fp32", torch.float32)):
        for sval in (0.00731, 0.02, 1.0, 1.7):
            s = torch.tensor([sval]).to(dt)
            zp = torch.tensor([-5], dtype=torch.int8)
            out[f"dq/{name}/s{sval}/int8"] = dequantize(codes, s, None)
            out[f"dq/{name}/s{sval}/int8zp"] = dequantize(codes, s, zp)
            d = dequantize(f8, s, None)
            d[d.isnan()] = 0
            out[f"dq/{name}/s{sval}/fp8"] = d
    save("sweep.pt", out)


# --------------------------------------------------------------------------- #
# D. compressor level (state-dict in / state-dict out)
# --------------------------------------------------------------------------- #
def gen_compressors():
    torch.manual_seed(99)
    R, C = 64, 512
    w = (torch.randn(R, C) * 0.02).bfloat16()
    cases = []

    def run(fmt, scheme, weight, g_idx=None, tag=""):
        args = scheme.weights
        scale, zp = observer_qparams(weight.float(), args)
        scale = scale.to(weight.dtype)
        sd = {"weight": weight, "weight_scale": scale, "weight_zero_point": zp}
        if g_idx is not None:
            sd["weight_g_idx"] = g_idx
        comp = BaseCompressor.get_value_from_registry(fmt)
        csd = comp.compress(sd, scheme)
        dsd = comp.decompress(csd, scheme)
        fq = fake_quantize(weight, scale, None if args.symmetric else zp, args, g_idx=g_idx)
        if "pad" not in tag:  # strategy inference from a padded block scale differs (forward.py:118-126)
            assert torch.equal(dsd["weight"], fq.to(dsd["weight"].dtype)), (fmt, tag)
        cases.append(dict(format=fmt, tag=tag, scheme=scheme.model_dump(mode="json"),
                          state_dict=sd, compressed=csd, decompressed=dsd,
                          param_names=list(comp.compression_param_names(scheme))))

    for preset in ("W4A16", "W4A16_ASYM", "W8A16"):
        run("pack-quantized", preset_name_to_scheme(preset, ["Linear"]), w, tag=preset)
    for bits in (2, 3, 5, 8):
        for sym in (True, False):
            sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=bits, symmetric=sym, strategy="group", group_size=64))
            run("pack-quantized", sch, w, tag=f"g64_b{bits}_{'sym' if sym else 'asym'}")
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=4, symmetric=False, strategy="tensor"))
    run("pack-quantized", sch, w, tag="tensor_asym")
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=4, symmetric=False, strategy="channel"))
    run("pack-quantized", sch, w[:50], tag="channel_asym_r50")
    g = torch.Generator().manual_seed(5)
    gi = (torch.arange(C) // 128)[torch.randperm(C, generator=g)].to(torch.int32)
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=4, symmetric=False, strategy="group", group_size=128, actorder="group"))
    run("pack-quantized", sch, w, g_idx=gi, tag="actorder")
    # ragged columns (not a multiple of 32 elements per row)
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=4, symmetric=True, strategy="channel"))
    run("pack-quantized", sch, w[:, :100].contiguous(), tag="ragged_c100")
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=3, symmetric=True, strategy="channel"))
    run("pack-quantized", sch, w[:, :100].contiguous(), tag="ragged_c100_b3")
    # naive / int / float
    for preset, fmt in (("FP8", "float-quantized"), ("W8A8", "int-quantized"), ("FP8_DYNAMIC", "float-quantized"), ("FP8_BLOCK", "float-quantized")):
        run(fmt, preset_name_to_scheme(preset, ["Linear"]), w, tag=preset)
    # block quant with padding (test_fp8_quant.py:134-175)
    sch = preset_name_to_scheme("FP8_BLOCK", ["Linear"])
    run("float-quantized", sch, (torch.randn(200, 300) * 0.02).bfloat16(), tag="FP8_BLOCK_pad")
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=8, symmetric=False, strategy="group", group_size=128))
    run("naive-quantized", sch, w, tag="int8_g128_asym")
    sch = QuantizationScheme(targets=["Linear"], weights=QuantizationArgs(num_bits=8, type="float", strategy="channel"))
    run("naive-quantized", sch, w.float(), tag="fp8_channel_fp32")
    save("compressors.pt", cases)


# --------------------------------------------------------------------------- #
# E. bitmasks + 2:4 semi-structured conversions / marlin-24 permutations
# --------------------------------------------------------------------------- #
def gen_sparse():
    g = torch.Generator().manual_seed(77)
    out = {"bitmask": [], "semi": [], "mask_creator": []}
    for shape in [(3, 8), (5, 13), (4, 100), (2, 3, 24), (1, 1), (64, 512)]:
        m = torch.rand(shape, generator=g) > 0.5
        p = pack_bitmasks(m)
        assert torch.equal(unpack_bitmasks(p, list(shape)), m)
        out["bitmask"].append(dict(mask=m, packed=p))
    for dt, (m, k) in [(torch.int8, (64, 64)), (torch.half, (64, 64)), (torch.bfloat16, (128, 128)), (torch.float, (64, 32))]:
        dense = torch.randn(m, k, generator=g)
        if dt == torch.int8:
            dense = (dense * 20).round().clamp(-127, 127)
        dense = dense.to(dt)
        mask = ssc.mask_creator(dense.float()).bool()
        out["mask_creator"].append(dict(x=dense, mask=mask))
        pruned = dense * mask.to(dt)
        sparse, meta = ssc.sparse_semi_structured_from_dense_cutlass(pruned)
        back = ssc.sparse_semi_structured_to_dense_cutlass(sparse, meta)
        if dt != torch.float:  # fp32 is the 1:2 layout; a 2:4 mask does not round-trip there
            assert torch.equal(back, pruned)
        out["semi"].append(dict(dense=pruned, sparse=sparse, meta=meta, back=back))
    perm = {}
    for bits in (4, 8):
        p, sp, sps = get_permutations_24(bits)
        perm[bits] = dict(perm=p, scale_perm=torch.tensor(sp), scale_perm_single=torch.tensor(sps))
    out["perm24"] = perm
    save("sparse.pt", out)


if __name__ == "__main__":
    gen_pack()
    gen_quant()
    gen_sweep()
    gen_compressors()
    gen_sparse()
