#!/usr/bin/env python
"""
bench.py -- headline benchmark of the compress/decompress hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--layers L] [--dump-outputs DIR]

Workload (configs[1] of BASELINE.json): W4A16 group_size=128 quantize + pack_to_int32 over every
Linear weight of a Llama-3-8B-shaped model (32 layers x {q,k,v,o,gate,up,down} = 224 bf16 tensors,
6.98 G elements, 13.96 GB), synthetic N(0, 0.02^2) weights, scales from the min/max observer rule.
One "step" = one pass of the hot path over all 224 tensors (a single multi-tensor launch).
`value` = weight bytes processed per second with tensors resident in HBM; `e2e` = the same pass
through the compressor plugin API on HOST (pinned) state dicts, H2D and D2H inside the timed region.
The inputs (14 GB) are far larger than the 126 MB L2, so every step streams from HBM.

Under torchrun (N > 1) every rank owns its own full-size tensor set (weak scaling, no data-path
collective); timing = max over ranks.

--impl reference times the CPU restatement of the reference path (oracle/, plain C + OpenMP on all
host threads; the reference itself is Python and cannot travel to the GPU box) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the 70B-sharded leg fills most of the 180 GB: keep the caching allocator from fragmenting (must be set before CUDA initialises)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "weight_GBps_w4a16_g128_quantize_pack_llama3_8b"
UNIT = "GB/s"
LAYER_SHAPES = [(4096, 4096), (1024, 4096), (1024, 4096), (4096, 4096), (14336, 4096), (14336, 4096), (4096, 14336)]
GROUP = 128
BITS = 4
ALG_BYTES_PER_ELEM = 2 + BITS / 8 + 2 / GROUP          # bf16 in + packed out + bf16 scale (SURVEY 8d) = 2.515625
FALLBACK_HBM_GBS = 6650.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def profile_traffic(kernel: str):
    """per-launch DRAM bytes of the dominant kernel from the committed ncu capture, if any"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def traffic_per_launch(kernel: str, n_elems: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the committed `ncu --set full` capture
    (profiles/ncu_ops_r1.md, taken on 4 layers), scaled by element count to this launch's size"""
    t = profile_traffic(kernel)
    if not t:
        return None
    return int(t["dram_bytes_per_launch"] / t["elements_per_launch"] * n_elems)


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML every few ms during the timed region
    (nvidia-smi itself takes ~100 ms per query, too coarse for a sub-second region)"""

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self._h = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v for v in vis.split(",") if v.strip() != ""]
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.002)

    def __enter__(self):
        if self._h is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def make_weights(device, layers: int, seed0: int):
    """bf16 weights + observer scales, generated on the device"""
    ws, scs = [], []
    for li in range(layers):
        for ti, (r, c) in enumerate(LAYER_SHAPES):
            g = torch.Generator(device=device).manual_seed(seed0 + li * len(LAYER_SHAPES) + ti)
            w = torch.empty(r, c, dtype=torch.bfloat16, device=device)
            step = 2048
            for r0 in range(0, r, step):  # bounded fp32 temporaries
                w[r0:r0 + step] = (torch.randn(min(step, r - r0), c, device=device, generator=g) * 0.02).bfloat16()
            # calculate_qparams, symmetric int4: scale = max|w| / 7.5 in the weight dtype (utils/helpers.py:79-87)
            sc = (w.unflatten(-1, (-1, GROUP)).abs().amax(-1).float() / 7.5).bfloat16()
            ws.append(w)
            scs.append(sc)
    return ws, scs


def args_w4():
    from types import SimpleNamespace
    return SimpleNamespace(strategy="group", group_size=GROUP, block_structure=None, num_bits=BITS, type="int", symmetric=True)


def time_steps(fn, steps: int, warmup: int, dist_on: bool, sampler=None):
    """W untimed steps, then exactly K steps bracketed by barrier + synchronize; CUDA events on the launching stream"""
    import torch.distributed as dist

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler is not None:
        sampler.__enter__()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.__exit__()
    if dist_on:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def run_b200(a):
    import torch.distributed as dist

    from compressed_tensors_b200 import _native as N
    from compressed_tensors_b200 import ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1 or (a.cfg5 and "RANK" in os.environ)     # a 1-rank torchrun launch with --cfg5 exercises the NCCL path on one GPU
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU path")
    # CPU legs first: a fresh pinned subprocess while this process holds neither a CUDA context nor pinned host memory
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        try:
            cpu = cpu_arm(seconds=a.cpu_seconds)
        except Exception as e:  # noqa: BLE001
            print(f"[bench] cpu baseline leg failed: {e}", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if dist_on:
        dist.init_process_group("nccl", device_id=dev)
    if a.gpus != world:
        print(f"[bench] note: --gpus {a.gpus} but WORLD_SIZE={world}", file=sys.stderr)

    layers = a.layers
    ws, scs = make_weights(dev, layers, 1000 + rank * 100000)
    n_elems = sum(w.numel() for w in ws)
    n_tensors = len(ws)
    weight_bytes = n_elems * 2
    alg_bytes = n_elems * ALG_BYTES_PER_ELEM
    qargs = args_w4()

    # device-resident problem table for the multi-tensor launch
    outs = [torch.empty(w.shape[0], w.shape[1] * BITS // 32, dtype=torch.int32, device=dev) for w in ws]
    probs = []
    for w, sc, o in zip(ws, scs, outs):
        p = ops._resolve(w, sc, None, qargs, None)
        d = ops._desc(p, w.dtype, sc.dtype, None, torch.bfloat16, torch.int8, None, N.Q_INT, BITS)
        probs.append((d, w, sc, None, o))

    plan = ops.BatchedPlan(N.OP_QUANTIZE_PACK, probs, local)   # descriptors validated against their tensors once, pointer tables built once

    def step():
        plan.run()                                               # one ct_batched call = one multi-tensor launch

    l0 = N.launch_count()
    cs = ClockSampler(local)
    ms = time_steps(step, a.steps, a.warmup, dist_on, sampler=cs)
    launches = (N.launch_count() - l0) - a.warmup  # one launch per step
    verified, verified_idx = (verify_timed_outputs(ws, scs, outs) if rank == 0 else (None, None))
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, outs)
    clocks = cs.summary()
    ms_per_step = ms / a.steps
    value = world * weight_bytes / (ms_per_step * 1e-3) / 1e9
    peak, peak_src = peaks()
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9

    # secondary ops of the metric (same tensors), device-resident, reported beside the headline
    extra = {}
    if not a.no_extra:
        def rate(fn, bytes_alg, nelem_bytes):
            # secondary ops: one CUDA-event pair per launch, median over the launches (a host hiccup between two
            # sub-millisecond launches would otherwise dominate a short timed region); the headline keeps the contract's
            # single bracket around exactly K steps
            k = max(5, a.steps)
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
            for e0, e1 in ev:
                e0.record()
                fn()
                e1.record()
            torch.cuda.synchronize()
            ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
            t = ms[len(ms) // 2]
            return {"weight_GBps": round(nelem_bytes / (t * 1e-3) / 1e9, 1), "hbm_GBps": round(bytes_alg / (t * 1e-3) / 1e9, 1),
                    "frac_of_peak": round(bytes_alg / (t * 1e-3) / 1e9 / peak, 3), "ms": round(t, 3), "ms_worst": round(ms[-1], 3), "launches": k}

        # decompress: unpack + dequantize
        dq = [torch.empty_like(w) for w in ws]
        dprobs = []
        for w, sc, o, dst in zip(ws, scs, outs, dq):
            p = ops._resolve(torch.empty(w.shape, dtype=torch.int8, device="meta"), sc, None, qargs, None)
            d = ops._desc(p, None, sc.dtype, None, None, torch.int8, torch.bfloat16, N.Q_INT, BITS)
            dprobs.append((d, o, sc, None, dst))
        extra["w4a16_unpack_dequantize"] = rate(ops.BatchedPlan(N.OP_UNPACK_DEQUANTIZE, dprobs, local).run, alg_bytes, weight_bytes)
        del dq, dprobs
        # FP8 per-tensor quantize / dequantize (configs[2])
        from types import SimpleNamespace
        f8 = SimpleNamespace(strategy="tensor", group_size=None, block_structure=None, num_bits=8, type="float", symmetric=True)
        s8 = [(w.abs().max().float() / 448).bfloat16().reshape(1) for w in ws]
        q8 = [torch.empty(w.shape, dtype=torch.float8_e4m3fn, device=dev) for w in ws]
        qprobs, dqprobs = [], []
        back = [torch.empty_like(w) for w in ws]
        for w, sc, q, b in zip(ws, s8, q8, back):
            p = ops._resolve(w, sc, None, f8, None)
            qprobs.append((ops._desc(p, w.dtype, sc.dtype, None, torch.bfloat16, torch.float8_e4m3fn, None, N.Q_FLOAT, 8), w, sc, None, q))
            dqprobs.append((ops._desc(p, None, sc.dtype, None, None, torch.float8_e4m3fn, torch.bfloat16, N.Q_INT, 8), q, sc, None, b))
        extra["fp8_quantize"] = rate(ops.BatchedPlan(N.OP_QUANTIZE, qprobs, local).run, n_elems * 3.0, weight_bytes)
        extra["fp8_dequantize"] = rate(ops.BatchedPlan(N.OP_DEQUANTIZE, dqprobs, local).run, n_elems * 3.0, weight_bytes)
        del q8, back, qprobs, dqprobs
        # standalone int4 pack / unpack on int8 codes (one big tensor set: largest shape x 8)
        codes = [torch.randint(-8, 8, (14336, 4096), dtype=torch.int8, device=dev) for _ in range(32)]  # 1.88 G codes: 2.8 GB of traffic per launch
        nel = sum(c.numel() for c in codes)
        pk = [torch.empty(c.shape[0], c.shape[1] // 8, dtype=torch.int32, device=dev) for c in codes]
        pdesc = []
        for c in codes:
            d = N.QuantDesc()
            d.rows, d.cols, d.num_bits = c.shape[0], c.shape[1], 4
            pdesc.append(d)
        pack_probs = [(d, c, None, None, o) for d, c, o in zip(pdesc, codes, pk)]
        unpack_probs = [(d, o, None, None, c) for d, c, o in zip(pdesc, codes, pk)]
        extra["int4_pack"] = rate(ops.BatchedPlan(N.OP_PACK_INT32, pack_probs, local).run, nel * 1.5, nel)
        extra["int4_unpack"] = rate(ops.BatchedPlan(N.OP_UNPACK_INT32, unpack_probs, local).run, nel * 1.5, nel)
        del codes, pk
        # NVFP4 (SURVEY 8(f) rank 2): fp4 e2m1, groups of 16, bf16 group scales (fp8-representable, as after calibration) and a
        # float32 global scale per tensor; decompress reads the scales as stored (float8_e4m3fn)
        nv = SimpleNamespace(strategy="tensor_group", group_size=16, block_structure=None, num_bits=4, type="float", symmetric=True)
        gss = [(448.0 * 6.0 / w.abs().max().float()).reshape(1) for w in ws]
        s8s = [(w.unflatten(-1, (-1, 16)).abs().amax(-1).float() / 6.0 * g).clamp(2.0 ** -9, 448.0).to(torch.float8_e4m3fn) for w, g in zip(ws, gss)]
        sbs = [s.to(torch.bfloat16) for s in s8s]
        nib = [torch.empty(w.shape[0], w.shape[1] // 2, dtype=torch.uint8, device=dev) for w in ws]
        nback = [torch.empty_like(w) for w in ws]
        cprobs, uprobs = [], []
        for w, sb, s8_, g, o, b in zip(ws, sbs, s8s, gss, nib, nback):
            p = ops._resolve(w, sb, None, nv, None)
            d = ops._desc(p, w.dtype, sb.dtype, None, torch.float32, w.dtype, None, N.Q_FP4, 4, torch.float32)
            d.global_scale = g.data_ptr()
            cprobs.append((d, w, sb, None, o))
            d2 = ops._desc(p, None, torch.float32, None, None, None, torch.bfloat16, N.Q_FP4, 4, torch.float32)
            d2.scale_dtype = N.DT[torch.float8_e4m3fn]
            d2.global_scale = g.data_ptr()
            uprobs.append((d2, o, s8_, None, b))
        extra["nvfp4_quantize_pack"] = rate(ops.BatchedPlan(N.OP_QUANTIZE_PACK_FP4, cprobs, local).run, n_elems * (2 + 2 / 16 + 0.5), weight_bytes)
        extra["nvfp4_unpack_dequantize"] = rate(ops.BatchedPlan(N.OP_UNPACK_DEQUANTIZE_FP4, uprobs, local).run, n_elems * (0.5 + 1 / 16 + 2), weight_bytes)
        del nib, nback, cprobs, uprobs, sbs, s8s
        # BASELINE config 4: Sparse24BitMask + int4 on 2:4-pruned weights, w * mask_creator(w) (reference utils/semi_structured_conversions.py:301-330),
        # g128 scales of the pruned weights; fused 2:4 select + quantize + pack and its inverse, one multi-tensor launch per direction.
        # Algorithmic traffic per dense element: 2 (bf16) + 0.25 (kept nibbles) + 0.125 (mask) + 2/128 (scale) = 2.39 B (SURVEY 8(d)).  Parity unpinned.
        from compressed_tensors_b200.utils.semi_structured_conversions import mask_creator
        w24 = [w * mask_creator(w).to(w.dtype) for w in ws]
        s24 = [(w.unflatten(-1, (-1, GROUP)).abs().amax(-1).float() / 7.5).bfloat16() for w in w24]
        pk24 = [torch.empty(w.shape[0], w.shape[1] // 16, dtype=torch.int32, device=dev) for w in w24]
        bm24 = [torch.empty(w.shape[0], w.shape[1] // 8, dtype=torch.uint8, device=dev) for w in w24]
        bk24 = [torch.empty_like(w) for w in w24]
        c24, d24 = [], []
        for w, sc, pk, bm, bk in zip(w24, s24, pk24, bm24, bk24):
            p = ops._resolve(w, sc, None, qargs, None)
            d = ops._desc(p, w.dtype, sc.dtype, None, torch.bfloat16, torch.int8, None, N.Q_INT, BITS)
            d.aux = bm.data_ptr()
            d2 = ops._desc(p, None, sc.dtype, None, None, torch.int8, torch.bfloat16, N.Q_INT, BITS)
            d2.aux = bm.data_ptr()
            c24.append((d, w, sc, None, pk))
            d24.append((d2, pk, sc, None, bk))
        b24 = n_elems * (2 + 0.25 + 0.125 + 2 / GROUP)
        extra["cfg4_sparse24_int4_compress"] = rate(ops.BatchedPlan(N.OP_SPARSE24_QUANTIZE_PACK, c24, local).run, b24, weight_bytes)
        extra["cfg4_sparse24_int4_decompress"] = rate(ops.BatchedPlan(N.OP_SPARSE24_UNPACK_DEQUANTIZE, d24, local).run, b24, weight_bytes)
        # what the timed launches wrote: decompress(compress(w24)) == fake_quantize(w24) on the kept columns, 0 elsewhere, for three tensors
        ok24 = True
        for i in (0, 4, len(w24) - 1):
            fq = ops.fake_quantize(w24[i], s24[i], None, qargs)
            ok24 &= bool(torch.equal(bk24[i], torch.where(w24[i] != 0, fq, torch.zeros_like(fq))))
        extra["cfg4_sparse24_int4_compress"]["round_trip_equals_masked_fake_quantize"] = ok24
        extra["cfg4_sparse24_int4_compress"]["parity"] = "unpinned composite (compressor pair absent from the reference); pieces pinned, see tests/test_gpu_sparse24q.py"
        del w24, s24, pk24, bm24, bk24, c24, d24

    # end to end through the plugin API on host (pinned) state dicts
    e2e = None
    if not a.no_e2e:
        e2e = run_e2e(ws, scs, a, dist_on, world, outs)


    cfg5 = None
    if dist_on and not a.no_cfg5 and (world > 1 or a.cfg5):
        ws = scs = outs = probs = plan = None      # the 8B replica set makes room
        torch.cuda.empty_cache()
        cfg5 = run_cfg5_70b_sharded(a, rank, world, dev)

    if dist_on:
        dist.barrier()
    if rank == 0:
        tn = N.lib()
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"W4A16 g128 symmetric quantize+pack_to_int32, Llama-3-8B-shaped Linear weights, {layers} layers x 7 = {n_tensors} bf16 tensors per GPU, {n_elems/1e9:.3f} G elements",
                       "l2": "inputs (%.1f GB per step) >> 126 MB L2, no flush needed" % (weight_bytes / 1e9),
                       "launch": "one multi-tensor persistent launch per step", "pipe": os.environ.get("CT_B200_PIPE", "tma")},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                         "traffic": traffic_per_launch("quantize_pack", n_elems), "peak_source": peak_src,
                         "traffic_source": "NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full capture of "
                                           "this kernel (" + str((profile_traffic("quantize_pack") or {}).get("source")) + "), scaled by element count",
                         "algorithmic_bytes_per_launch": alg_bytes, "frac_of_8TBps_nominal": round(achieved / 8000.0, 4)},
            "gpu_launches": int(launches), "clocks": clocks,
            "verified": verified, "verified_against": f"oracle (CPU) on every packed word of tensors {verified_idx} written by the timed launches",
        }
        if e2e is not None:
            line["e2e"] = e2e
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if cfg5 is not None:
            extra["cfg5_70b_sharded"] = cfg5
        if extra:
            line["ops"] = extra
        print(json.dumps(line))
    if dist_on:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# BASELINE config 5: ModelCompressor.compress_model on a Llama-3-70B-shaped model sharded tensor-per-GPU (N >= 2)
# ------------------------------------------------------------------------------------------------
SHAPES_70B = [(8192, 8192), (1024, 8192), (1024, 8192), (8192, 8192), (28672, 8192), (28672, 8192), (8192, 28672)]


def gen_weight_70b(i: int, dev):
    """tensor i of the 70B set, bit-identical on whichever rank generates it (seed 1000 + i, SURVEY 8(d) cfg5)"""
    r, c = SHAPES_70B[i % len(SHAPES_70B)]
    g = torch.Generator(device=dev).manual_seed(1000 + i)
    w = torch.empty(r, c, dtype=torch.bfloat16, device=dev)
    step = 2048
    for r0 in range(0, r, step):
        w[r0:r0 + step] = (torch.randn(min(step, r - r0), c, device=dev, generator=g) * 0.02).bfloat16()
    sc = torch.empty(r, c // GROUP, dtype=torch.bfloat16, device=dev)
    for r0 in range(0, r, step):
        sc[r0:r0 + step] = (w[r0:r0 + step].unflatten(-1, (-1, GROUP)).abs().amax(-1).float() / 7.5).bfloat16()
    return w, sc


def run_cfg5_70b_sharded(a, rank: int, world: int, dev):
    """560 bf16 tensors with Llama-3-70B shapes, each generated on its OWNER rank only (greedy_bin_packing on bytes, reference
    distributed/assign.py:12-42); every other rank holds the module on meta.  Timed: ModelCompressor.compress_model(distributed=True)
    -> replace_module_parallel (reference distributed/module_parallel.py:23-90, model_compressor.py:138-172): `compress` = the
    owners' kernels, `recouple` = the NCCL broadcast of the packed tensors, reported separately (max over ranks).  Then
    decompress_model(distributed=True) (the flow the reference leaves as a TODO, model_compressor.py:196).  Parity: a sample of
    tensors is recomputed on EVERY rank through the single-tensor plugin path and compared bit for bit with what the rank holds
    after the recouple; checksums of all 560 packed tensors must agree across ranks; one tensor is checked against the CPU oracle."""
    import torch.distributed as dist

    from compressed_tensors_b200.compressors import ModelCompressor, PackedQuantizationCompressor
    from compressed_tensors_b200.distributed import greedy_bin_packing, module_size
    from compressed_tensors_b200.quantization import QuantizationConfig, QuantizationStatus, apply_quantization_config
    from compressed_tensors_b200.utils import get_direct_state_dict, replace_direct_state_dict

    layers = a.cfg5_layers
    n = layers * len(SHAPES_70B)
    model = torch.nn.Module()
    mods = []
    for i in range(n):
        r, c = SHAPES_70B[i % len(SHAPES_70B)]
        lin = torch.nn.Linear(c, r, bias=False, device="meta", dtype=torch.bfloat16)
        model.add_module(f"linear_{i}", lin)
        mods.append(lin)
    apply_quantization_config(model, QuantizationConfig(config_groups={"W4A16": ["Linear"]}))
    index = {id(m): i for i, m in enumerate(mods)}
    _, bins, owner = greedy_bin_packing(list(mods), world, module_size)     # the deal replace_module_parallel will make
    loads = [sum(m.weight.numel() * 2 for m in b) for b in bins]
    dense_total = sum(loads)
    mine = [m for m in mods if owner[m] == rank]
    scheme = mods[0].quantization_scheme

    t0 = time.perf_counter()
    originals = {}
    for m in mine:
        w, sc = gen_weight_70b(index[id(m)], dev)
        originals[id(m)] = (w, sc, torch.zeros(sc.shape, dtype=torch.int8, device=dev))
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0

    def reset():
        for m in mods:
            if owner[m] == rank:
                w, sc, zp = originals[id(m)]
                replace_direct_state_dict(m, {"weight": w, "weight_scale": sc, "weight_zero_point": zp})
            else:
                r, c = m.out_features, m.in_features
                replace_direct_state_dict(m, {"weight": torch.empty(r, c, dtype=torch.bfloat16, device="meta"),
                                              "weight_scale": torch.empty(r, c // GROUP, dtype=torch.bfloat16, device="meta"),
                                              "weight_zero_point": torch.empty(r, c // GROUP, dtype=torch.int8, device="meta")})
            m.quantization_status = QuantizationStatus.FROZEN

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    mc = ModelCompressor.from_pretrained_model(model)
    runs = []
    for k in range(1 + a.cfg5_reps):          # first pass untimed (NCCL communicator, kernel images)
        reset()
        mc.remove_decompression_hook(model)
        torch.cuda.synchronize()
        dist.barrier()
        st = {}
        t0 = time.perf_counter()
        mc.compress_model(model, distributed=True, stats=st)
        torch.cuda.synchronize()
        total = time.perf_counter() - t0
        recouple_how = st.get("recouple_how")
        if k > 0:
            runs.append(reduce_max([st["apply_s"], st["recouple_s"], total, st["device_ms"] or 0.0, st["mirror_host_s"]]) + [st["recouple_bytes"]])
    best = min(runs, key=lambda r: r[2])

    # ---- parity ----
    sums = torch.stack([m.weight_packed.sum(dtype=torch.int64) + m.weight_scale.view(torch.int16).sum(dtype=torch.int64) for m in mods])
    hi, lo = sums.clone(), sums.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    ranks_agree = bool(torch.equal(hi, lo))
    sample = sorted({0, 1, 4, 6, n - 1, n // 2})
    sample_ok = True
    for i in sample:
        w, sc = gen_weight_70b(i, dev)
        want = PackedQuantizationCompressor.compress({"weight": w, "weight_scale": sc, "weight_zero_point": torch.zeros(sc.shape, dtype=torch.int8, device=dev)}, scheme)
        got = get_direct_state_dict(mods[i])
        sample_ok &= bool(torch.equal(got["weight_packed"], want["weight_packed"]) and torch.equal(got["weight_scale"], want["weight_scale"])
                          and got["weight_shape"].tolist() == list(w.shape) and got["weight_packed"].device == dev)
        del w, sc, want, got            # `got` holds views of a gathered recouple buffer: a survivor would keep that buffer alive
    oracle_ok = None
    if rank == 0:
        import oracle   # checker only

        w, sc = gen_weight_70b(1, dev)
        q = oracle.quantize(w.cpu(), sc.cpu(), None, strategy="group", group_size=GROUP, num_bits=BITS, dtype=torch.int8)
        oracle_ok = bool(torch.equal(mods[1].weight_packed.cpu(), oracle.pack_to_int32(q, BITS)))
        del w, sc, q
    ok = torch.tensor([int(sample_ok)], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    sample_ok = bool(ok.item())

    # ---- the way back: distributed decompress (every rank ends with the complete dense model, 2 bytes x 68.45 G elements) ----
    originals.clear()
    torch.cuda.empty_cache()
    free_b, _ = torch.cuda.mem_get_info()
    packed_here = sum(m.weight_packed.numel() * 4 for m in mods)
    dec = None
    fits = torch.tensor([int(free_b + packed_here > dense_total + (12 << 30))], device=dev)
    dist.all_reduce(fits, op=dist.ReduceOp.MIN)          # one decision for all ranks: the leg is full of collectives
    if bool(fits.item()):
        from compressed_tensors_b200 import ops

        d_runs = []
        for k in range(2):        # the first pass grows the allocator to 137 GB of dense output (cuMemMap, ~1 s); the second one is timed
            if k > 0:
                mc.compress_model(model, distributed=True)              # back to the compressed state
                mc.remove_decompression_hook(model)
            torch.cuda.synchronize()
            dist.barrier()
            st = {}
            t0 = time.perf_counter()
            mc.decompress_model(model, distributed=True, stats=st)
            torch.cuda.synchronize()
            total = time.perf_counter() - t0
            d_runs.append(reduce_max([st["apply_s"], st["recouple_s"], total, st["device_ms"] or 0.0]) + [st["recouple_bytes"]])
            d_how = st.get("recouple_how")
        d_apply, d_rec, d_total, d_dev, d_bytes = d_runs[-1]
        dsums = torch.stack([m.weight.view(torch.int16).sum(dtype=torch.int64) for m in mods])
        hi, lo = dsums.clone(), dsums.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        d_ok = True
        for i in sample[:3]:
            w, sc = gen_weight_70b(i, dev)
            fq = ops.fake_quantize(w, sc, None, scheme.weights)
            d_ok &= bool(torch.equal(mods[i].weight, fq))      # torch.equal, the reference's own assertion: -0.0 == +0.0 (a code 0 dequantizes to +0)
            del w, sc, fq
        okd = torch.tensor([int(d_ok)], device=dev)
        dist.all_reduce(okd, op=dist.ReduceOp.MIN)
        dec = {"decompress_ms": round(d_apply * 1e3, 2), "decompress_device_ms": round(d_dev, 2), "recouple_ms": round(d_rec * 1e3, 2),
               "total_ms": round(d_total * 1e3, 2), "weight_GBps_decompress_only": round(dense_total / d_apply / 1e9, 1),
               "weight_GBps_decompress_device_time": round(dense_total / (d_dev * 1e-3) / 1e9, 1) if d_dev else None,
               "recouple_GBps_per_rank": round(d_bytes / d_rec / 1e9, 1), "recouple_how": d_how, "first_pass_total_ms": round(d_runs[0][2] * 1e3, 1),
               "ranks_agree": bool(torch.equal(hi, lo)), "sample_equals_fake_quantize": bool(okd.item())}
    else:
        dec = {"skipped": f"{free_b / 2**30:.0f} GiB free, the recoupled dense model needs {dense_total / 2**30:.0f} GiB"}
    for m in mods:                         # release before the process exits its NCCL group
        replace_direct_state_dict(m, {})
    torch.cuda.empty_cache()

    apply_s, rec_s, total_s, dev_ms, mirror_s, rec_bytes = best
    return {
        "workload": f"ModelCompressor.compress_model(distributed=True), W4A16 g128, {n} Llama-3-70B-shaped bf16 tensors ({dense_total / 1e9:.1f} GB), each generated on its owner rank only",
        "world_size": world, "tensors": n, "dense_bytes": int(dense_total),
        "per_rank_dense_GB": [round(b / 1e9, 2) for b in loads], "imbalance_max_over_mean": round(max(loads) / (sum(loads) / world), 4),
        "compress_ms": round(apply_s * 1e3, 2), "compress_device_ms": round(dev_ms, 3), "meta_mirror_host_ms": round(mirror_s * 1e3, 2),
        "recouple_ms": round(rec_s * 1e3, 2), "total_ms": round(total_s * 1e3, 2),
        "weight_GBps_compress_only": round(dense_total / apply_s / 1e9, 1), "weight_GBps_with_recouple": round(dense_total / total_s / 1e9, 1),
        "weight_GBps_compress_device_time": round(dense_total / (dev_ms * 1e-3) / 1e9, 1) if dev_ms else None,
        "note": "compress_ms = host clock of the owners' launches + the meta mirror of the other ranks' modules (Python, per module), device-synchronised; "
                "compress_device_ms = CUDA events around the slowest rank's kernels alone",
        "recouple_bytes_per_rank": int(rec_bytes), "recouple_GBps_per_rank": round(rec_bytes / rec_s / 1e9, 1), "recouple_how": recouple_how,
        "reps": len(runs), "timing": "host clock around the call with device synchronisation on both sides, max over ranks (the call includes the Python module loop)",
        "generate_s": round(gen_s, 2),
        "parity": {"ranks_agree_on_all_checksums": ranks_agree, "sample_equals_single_rank": sample_ok, "sample": sample, "oracle_tensor_1": oracle_ok},
        "decompress": dec,
    }


def _physical_gpu_index(device_index: int) -> int:
    """NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list"""
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        ids = [v for v in vis.split(",") if v.strip() != ""]
        if device_index < len(ids) and ids[device_index].strip().isdigit():
            return int(ids[device_index])
    return device_index


def _bind_to_gpu_numa(device_index: int):
    """Run this rank on the CPUs NVML names as local to its GPU and prefer that socket's memory, BEFORE the pinned host buffers of the
    e2e leg are allocated: at 8 ranks the leg moves 8 x 17.5 GB per step through host memory, and buffers that sit on the other
    socket cross the inter-socket link on every copy (round 1: 0.64 scaling efficiency at N = 8 with NUMA-blind buffers).
    On by default; CT_BENCH_NUMA=0 turns it off (for the A/B).  Returns (previous affinity, info dict) or (None, None)."""
    if os.environ.get("CT_BENCH_NUMA", "1") != "1" or not hasattr(os, "sched_setaffinity"):
        return None, None
    try:
        import pynvml

        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(_physical_gpu_index(device_index))
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        before = os.sched_getaffinity(0)
        cpus &= before
        if not cpus:
            return None, None
        os.sched_setaffinity(0, cpus)
        node = None
        try:
            entries = os.listdir(f"/sys/devices/system/cpu/cpu{min(cpus)}")
            node = next((int(e[4:]) for e in entries if e.startswith("node") and e[4:].isdigit()), None)
        except OSError:
            pass
        preferred = node is not None and set_mempolicy(1, [node])          # MPOL_PREFERRED: this socket first, never fail
        return before, {"gpu_local_cpus": len(cpus), "numa_node": node, "mempolicy_preferred": bool(preferred)}
    except Exception:  # noqa: BLE001  (no NVML, no permission: keep the launcher's affinity)
        return None, None


def verify_timed_outputs(ws, scs, outs):
    """what the TIMED launches wrote, against the CPU oracle (checker only): the largest, the smallest and the last tensor of the
    set, every packed word"""
    import oracle

    by_size = sorted(range(len(ws)), key=lambda i: ws[i].numel())
    picks = sorted({by_size[-1], by_size[0], len(ws) - 1})
    ok = True
    for i in picks:
        q = oracle.quantize(ws[i].cpu(), scs[i].cpu(), None, strategy="group", group_size=GROUP, num_bits=BITS, dtype=torch.int8)
        ok &= bool(torch.equal(outs[i].cpu(), oracle.pack_to_int32(q, BITS)))
    return ok, picks


DUMP_WORDS_PER_TENSOR = 8192
DUMP_SEED = 0


def dump_outputs(directory: str, outs):
    """What the last timed step wrote, for comparing two builds output for output: the packed int32 words at the same seeded
    positions of every tensor (all 3.5 GB would not fit a 64 MB dump).  Written as float64, which holds every int32 exactly:
      weight_packed_sample.npy        [tensors, DUMP_WORDS_PER_TENSOR]  the sampled words
      weight_packed_sample_index.npy  [tensors, DUMP_WORDS_PER_TENSOR]  their flat positions in each [rows, cols / 8] output"""
    import numpy as np

    g = torch.Generator().manual_seed(DUMP_SEED)
    words, index = [], []
    for o in outs:
        n = min(DUMP_WORDS_PER_TENSOR, o.numel())
        idx = torch.randint(0, o.numel(), (n,), generator=g).sort().values
        words.append(o.reshape(-1)[idx.to(o.device)].cpu().double())
        index.append(idx.double())
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "weight_packed_sample.npy"), torch.stack(words).numpy())
    np.save(os.path.join(directory, "weight_packed_sample_index.npy"), torch.stack(index).numpy())


def run_e2e(ws, scs, a, dist_on, world, outs=None):
    """The same pass end to end through the public API: ModelCompressor.compress_model() on a HOST-resident
    model (pinned weights and scales), i.e. the call llm-compressor makes before save_pretrained.  Every step
    uploads all weights + scales (H2D), runs the kernels and brings the packed words back (D2H); the timed
    region is the compress_model call itself.  Modules are reset to their uncompressed state between steps
    (pointer swaps, untimed)."""
    from compressed_tensors_b200.compressors import ModelCompressor
    from compressed_tensors_b200.quantization import QuantizationConfig, QuantizationStatus, apply_quantization_config
    from compressed_tensors_b200.utils import replace_direct_state_dict

    layers = min(a.e2e_layers, len(ws) // len(LAYER_SHAPES))
    n = layers * len(LAYER_SHAPES)
    previous_affinity, numa = _bind_to_gpu_numa(ws[0].device.index or 0)
    hw = [w.cpu().pin_memory() for w in ws[:n]]
    hs = [s.cpu().pin_memory() for s in scs[:n]]
    wbytes = sum(t.numel() * 2 for t in hw)
    h2d = wbytes + sum(t.numel() * 2 for t in hs)
    d2h = sum(t.numel() // 8 * 4 for t in hw)

    model = torch.nn.Module()
    mods = []
    for i, w in enumerate(hw):
        lin = torch.nn.Linear(w.shape[1], w.shape[0], bias=False, device="meta", dtype=torch.bfloat16)
        lin.weight = torch.nn.Parameter(w, requires_grad=False)
        model.add_module(f"linear_{i}", lin)
        mods.append(lin)
    apply_quantization_config(model, QuantizationConfig(config_groups={"W4A16": ["Linear"]}))
    mc = ModelCompressor.from_pretrained_model(model)

    def reset():
        for lin, w, sc in zip(mods, hw, hs):
            replace_direct_state_dict(lin, {"weight": w, "weight_scale": sc})
            lin.quantization_status = QuantizationStatus.FROZEN
        mc.remove_decompression_hook(model)

    steps = max(2, min(a.steps, 5))
    times = []
    for k in range(2 + steps):
        reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mc.compress_model(model, distributed=False)   # every rank holds its own shard of the job (weak scaling), no exchange
        torch.cuda.synchronize()
        if k >= 2:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    if dist_on:
        import torch.distributed as dist
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    packed = mods[0].weight_packed
    assert packed.dtype == torch.int32 and not packed.is_cuda and mods[-1].quantization_status == QuantizationStatus.COMPRESSED
    # the host result of the last timed step == the device-resident result of the headline launch (itself checked against the oracle)
    e2e_ok = all(bool(torch.equal(mods[i].weight_packed, outs[i].cpu())) for i in sorted({0, 1, n // 2, n - 1})) if outs is not None else None
    out = {"value": round(world * wbytes / dt / 1e9, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "api": "ModelCompressor.compress_model(model) on a host-resident (pinned) model", "tensors_per_step": n, "steps": steps,
           "ms_per_step": round(dt * 1e3, 2), "verified_equal_to_device_result": e2e_ok}
    out["numa"] = numa if numa is not None else "off"
    if previous_affinity is not None:
        os.sched_setaffinity(0, previous_affinity)
        set_mempolicy(0, [])                             # MPOL_DEFAULT
    return out


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm.  Two implementations of the same path are timed on the host cores, on the same bounded sample
# (one of the 32 layers: 7 tensors, 436 MB of bf16), in a FRESH subprocess whose OpenMP / ATen threads are pinned one per
# physical core and whose memory is interleaved over the NUMA nodes:
#   "reference": the UNMODIFIED reference from baseline/_ref (tools/install_reference.py) through its own public API,
#                PackedQuantizationCompressor.compress (reference compressors/pack_quantized/base.py:96-104) -- torch eager on ATen CPU kernels
#   "port"     : oracle/ct_oracle.c, the C + OpenMP restatement of that path (test infrastructure; timed here as the checker's speed)
# The arm's `value` is the reference when baseline/_ref travelled with the snapshot, else the port.  Median of >= 5 repetitions.
# ------------------------------------------------------------------------------------------------
def cpu_topology():
    """(one hardware thread per physical core inside the affinity mask, all allowed cpus, NUMA node ids, CPU model string)"""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    seen, phys = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            phys.append(c)
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
    except OSError:
        nodes = [0]
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return phys, allowed, nodes or [0], model


def set_mempolicy(mode: int, nodes) -> bool:
    """set_mempolicy(2) through libc's syscall(): 1 = MPOL_PREFERRED, 3 = MPOL_INTERLEAVE (no numactl / libnuma in the image)"""
    import ctypes

    try:
        mask = 0
        for n in nodes:
            mask |= 1 << n
        buf = (ctypes.c_ulong * 16)(*[(mask >> (64 * i)) & (2 ** 64 - 1) for i in range(16)])
        libc = ctypes.CDLL(None, use_errno=True)
        return libc.syscall(238, ctypes.c_int(mode), buf, ctypes.c_ulong(16 * 64 + 1)) == 0      # x86_64: __NR_set_mempolicy = 238
    except Exception:  # noqa: BLE001
        return False


def oracle_compress_layer(ws, scs, tmp):
    """quantize(int8) -> pack_to_int32 for each tensor of the sample, through the C oracle"""
    import ctypes

    import oracle

    L = oracle.lib()
    for w, sc, (q8, out) in zip(ws, scs, tmp):
        r, c = w.shape
        L.orc_quantize_pack(oracle._p(w), 2, oracle._p(sc), 2, ctypes.c_void_p(0), -1, ctypes.c_void_p(0), oracle._p(out), oracle._p(q8),
                            ctypes.c_int64(r), ctypes.c_int64(c), ctypes.c_int64(1), ctypes.c_int64(GROUP), ctypes.c_int64(c // GROUP), 2, BITS)


def cpu_sample():
    """one layer of the workload (7 tensors, 218 M elements, 436 MB of bf16)"""
    ws, scs, tmp = [], [], []
    for ti, (r, c) in enumerate(LAYER_SHAPES):
        g = torch.Generator().manual_seed(1000 + ti)
        w = (torch.randn(r, c, generator=g) * 0.02).bfloat16()
        sc = (w.unflatten(-1, (-1, GROUP)).abs().amax(-1).float() / 7.5).bfloat16()
        ws.append(w)
        scs.append(sc)
        tmp.append((torch.empty(r, c, dtype=torch.int8), torch.empty(r, c // 8, dtype=torch.int32)))
    return ws, scs, tmp


def _median_time(fn, budget_s: float, min_reps: int, max_reps: int, warmup: int = 1):
    """median of the timed repetitions.  min_reps == max_reps = the exact count the reference arm was asked for (--steps K), which the
    time budget may only cut short after 5 repetitions"""
    for _ in range(max(warmup, 1)):
        fn()                                # warm-up
    times = []
    t_start = time.perf_counter()
    exact = min_reps == max_reps
    while len(times) < max_reps and (len(times) < (5 if exact else min_reps) or time.perf_counter() - t_start < budget_s):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    times.sort()
    return times[len(times) // 2], times


def run_cpu_worker(a):
    """the subprocess body of both CPU legs; prints one JSON object"""
    # the parent computed the topology: in here OMP_PROC_BIND has already bound the initial thread to its place (one CPU), so the
    # affinity mask no longer shows what this process may use.  OMP_PLACES (set by the parent) lists one hardware thread per
    # physical core -- SMT siblings stay idle -- and both OpenMP runtimes (the oracle's and ATen's) put thread i on place i.
    _, _, nodes, model = cpu_topology()
    phys = [int(c) for c in a.cpu_list.split(",")] if a.cpu_list else sorted(os.sched_getaffinity(0))
    allowed = list(range(a.nproc or len(phys)))
    interleaved = len(nodes) > 1 and set_mempolicy(3, nodes)     # inherited by the OpenMP threads (created at the first parallel region)
    torch.set_num_threads(len(phys))
    import oracle

    oracle.set_num_threads(len(phys))
    ws, scs, tmp = cpu_sample()
    wbytes = sum(w.numel() * 2 for w in ws)
    budget = float(a.cpu_seconds)
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    have_ref = os.path.exists(os.path.join(ref_dir, "compressed_tensors", "version.py"))
    # --impl reference --steps K --warmup W: the MAIN leg (the reference when it is installed, else the port) does W warm-ups and
    # exactly K timed repetitions, cut short only by a 300 s budget; the other leg stays a short time-bounded sample
    k, wup = int(a.cpu_steps), max(int(a.cpu_warmup), 1)
    if k > 0:
        k = max(k, 5)                       # a median needs at least 5 repetitions (VERDICT r1 item 3); --steps below that is raised
    if k > 0 and not have_ref:
        med, times = _median_time(lambda: oracle_compress_layer(ws, scs, tmp), 300.0, k, k, wup)
    else:
        med, times = _median_time(lambda: oracle_compress_layer(ws, scs, tmp), (8.0 if k > 0 else budget * 0.4), 5, 40)
    out = {"nproc": len(allowed), "threads": len(phys), "cpu_model": model, "numa_nodes": len(nodes), "memory_interleaved": bool(interleaved),
           "sample_bytes": wbytes,
           "port": {"GBps": round(wbytes / med / 1e9, 3), "ms_median": round(med * 1e3, 1), "ms_min": round(times[0] * 1e3, 1),
                    "ms_max": round(times[-1] * 1e3, 1), "reps": len(times), "threads": oracle.num_threads()},
           "reference": None}
    if have_ref:
        try:
            sys.path.insert(0, ref_dir)
            import compressed_tensors                                   # the reference itself, not site-packages' older release
            from compressed_tensors.compressors import PackedQuantizationCompressor
            from compressed_tensors.quantization import preset_name_to_scheme

            assert os.path.realpath(compressed_tensors.__file__).startswith(os.path.realpath(ref_dir)), compressed_tensors.__file__
            scheme = preset_name_to_scheme("W4A16", ["Linear"])
            sds = [{"weight": w, "weight_scale": sc, "weight_zero_point": torch.zeros(sc.shape, dtype=torch.int8)} for w, sc in zip(ws, scs)]
            got = []

            def ref_layer():
                got.clear()
                with torch.no_grad():
                    for sd in sds:
                        got.append(PackedQuantizationCompressor.compress(sd, scheme)["weight_packed"])

            rmed, rtimes = _median_time(ref_layer, 300.0, k, k, wup) if k > 0 else _median_time(ref_layer, budget * 0.6, 5, 20)
            same = all(torch.equal(g, t[1]) for g, t in zip(got, tmp))     # the oracle port reproduces the reference's words on the sample
            out["reference"] = {"GBps": round(wbytes / rmed / 1e9, 3), "ms_median": round(rmed * 1e3, 1), "ms_min": round(rtimes[0] * 1e3, 1),
                                "ms_max": round(rtimes[-1] * 1e3, 1), "reps": len(rtimes), "threads": torch.get_num_threads(),
                                "api": "PackedQuantizationCompressor.compress (baseline/_ref, unmodified reference, torch eager CPU)",
                                "equals_port_bit_for_bit": bool(same)}
        except Exception as e:  # noqa: BLE001
            out["reference"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    print("CPUWORKER " + json.dumps(out))


def cpu_arm(seconds: float, steps: int = 0, warmup: int = 1):
    """run the CPU legs in a fresh, pinned subprocess and shape the `cpu_baseline` object (steps > 0: the main leg runs exactly that
    many timed repetitions after `warmup` warm-ups -- the reference arm's --steps / --warmup)"""
    phys, allowed, nodes, model = cpu_topology()
    env = {k: v for k, v in os.environ.items() if not k.startswith(("OMP_", "MKL_", "GOMP_", "KMP_")) and k not in
           ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID")}
    env.update(OMP_NUM_THREADS=str(len(phys)), MKL_NUM_THREADS=str(len(phys)), OMP_PROC_BIND="close",
               OMP_PLACES=",".join("{%d}" % c for c in phys), CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-worker", "--cpu-seconds", str(seconds),
                        "--cpu-list", ",".join(str(c) for c in phys), "--nproc", str(len(allowed)),
                        "--cpu-steps", str(steps), "--cpu-warmup", str(warmup)],
                       capture_output=True, text=True, env=env, timeout=900)
    line = next((ln for ln in r.stdout.splitlines() if ln.startswith("CPUWORKER ")), None)
    if r.returncode != 0 or line is None:
        raise RuntimeError(f"cpu worker failed (rc {r.returncode}): {r.stderr[-1500:]}")
    w = json.loads(line[len("CPUWORKER "):])
    ref = w["reference"] if (w["reference"] and "GBps" in w["reference"]) else None
    kind = "reference" if ref else "port"
    main = ref or w["port"]
    sample = (f"1 of 32 Llama-3-8B layers (7 tensors, {w['sample_bytes'] / 1e6:.0f} MB bf16), W4A16 g128 quantize + pack_to_int32; "
              + ("the unmodified reference's PackedQuantizationCompressor.compress (torch eager, ATen CPU kernels) from baseline/_ref" if ref
                 else "oracle/ct_oracle.c (C + OpenMP restatement of the reference path)")
              + f"; median of {main['reps']} reps ({main['ms_min']}-{main['ms_max']} ms), {w['threads']} threads pinned one per physical core of "
                f"{w['nproc']} logical CPUs ({w['cpu_model']}), {w['numa_nodes']} NUMA node(s), memory {'interleaved' if w['memory_interleaved'] else 'default policy'}, fresh subprocess")
    out = {"value": main["GBps"], "unit": UNIT, "cores": w["threads"], "kind": kind, "sample": sample, "nproc": w["nproc"], "cpu_model": w["cpu_model"],
           "numa_nodes": w["numa_nodes"], "reps": main["reps"], "ms_median": main["ms_median"],
           "port": w["port"], "reference": w["reference"]}
    return out


def run_reference(a):
    """reference arm: the reference's own CPU implementation of the path (or, without baseline/_ref, its C restatement) on the host cores"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_arm(seconds=20.0, steps=a.steps, warmup=a.warmup)          # exactly --steps timed repetitions after --warmup warm-ups
    v = cb["value"]
    if cb["reps"] != a.steps:
        cb["sample"] += (f"; {a.steps} steps were asked for, {cb['reps']} were timed "
                         + ("(a median needs 5)" if a.steps < 5 else "(300 s budget)"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": cb["reps"], "warmup": max(a.warmup, 1),
        "ms_per_step": cb["ms_median"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "W4A16 g128 symmetric quantize+pack_to_int32, Llama-3-8B-shaped Linear weights (bounded sample: 1 layer per step)"},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "cpu-worker"])
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="time budget of the CPU legs (bounded sample)")
    ap.add_argument("--cpu-list", default="", help=argparse.SUPPRESS)   # cpu-worker only: one hardware thread per physical core
    ap.add_argument("--cpu-steps", type=int, default=0, help=argparse.SUPPRESS)    # cpu-worker only: exact repetition count of the main leg
    ap.add_argument("--cpu-warmup", type=int, default=1, help=argparse.SUPPRESS)
    ap.add_argument("--nproc", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--layers", type=int, default=32, help="Llama-3-8B layers per GPU (32 = the full model)")
    ap.add_argument("--e2e-layers", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the 70B-sharded ModelCompressor leg (runs whenever N >= 2)")
    ap.add_argument("--cfg5", action="store_true", help="run the sharded leg even with one rank (under a 1-rank torchrun; pick --cfg5-layers <= 40)")
    ap.add_argument("--cfg5-layers", type=int, default=80, help="Llama-3-70B layers of the sharded leg (80 = the full model, 560 tensors)")
    ap.add_argument("--cfg5-reps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of the last step's packed words to DIR/*.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == "cpu-worker":
        run_cpu_worker(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
