"""
The host mirror, the CPU oracle and the compressor / ModelCompressor layers against the reference, on the seeded cases of the
differential fuzz scripts under tests/reference_compat/, compared with the reference's outcomes recorded in
tests/golden/reference_fuzz/ (tests/reference_compat/recorded.py).  The tensor-level ops are backed by the CPU oracle
(tests/reference_compat/oracle_patch.py); the CUDA kernels are covered by the `-m gpu` tests, which re-express the reference's own
hot-path test files (tests/test_gpu_reference_suite.py, test_gpu_fp4.py, test_gpu_convert.py).
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_mirror_matches_the_reference_under_fuzz():
    """random QuantizationArgs / QuantizationScheme constructions and qparam computations give the same values -- or the same
    exception type -- in the mirror as in the reference (tests/reference_compat/fuzz_host_mirror.py, ~2500 comparisons)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reference_compat", "fuzz_host_mirror.py"), "300"],
                       capture_output=True, text=True, cwd="/tmp", timeout=600)
    lines = [line for line in r.stdout.splitlines() if "checked" in line]
    assert r.returncode == 0 and len(lines) == 3 and all(line.endswith(" 0 mismatches") for line in lines), r.stdout[-2000:] + r.stderr[-1000:]


def test_oracle_matches_the_reference_under_fuzz():
    """seeded random cases, beyond the committed goldens: the CPU oracle against the reference's own quantize / dequantize / fake_quantize
    (every strategy, int 2..8 / fp8 / fp4, three dtypes) and pack / unpack functions (tests/reference_compat/fuzz_oracle.py)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reference_compat", "fuzz_oracle.py"), "200"],
                       capture_output=True, text=True, cwd="/tmp", timeout=600)
    lines = [line for line in r.stdout.splitlines() if "checked" in line]
    assert r.returncode == 0 and len(lines) == 2 and all(line.endswith(" 0 mismatches") for line in lines), r.stdout[-2000:] + r.stderr[-1000:]


def test_compressor_plugins_match_the_reference_under_fuzz():
    """compress() / decompress() of every registered quantization format on random weights, schemes and strategies: same keys, dtypes,
    shapes and bits as the reference's classes (tests/reference_compat/fuzz_compressors.py; oracle-backed ops, CPU)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reference_compat", "fuzz_compressors.py"), "150"],
                       capture_output=True, text=True, cwd="/tmp", timeout=600)
    lines = [line for line in r.stdout.splitlines() if "checked" in line]
    assert r.returncode == 0 and len(lines) == 2 and all(" 0 mismatches" in line for line in lines), r.stdout[-2000:] + r.stderr[-1000:]


def test_model_compressor_matches_the_reference_under_fuzz():
    """ModelCompressor end to end on random small models and presets, next to the reference's: module state dicts after
    apply_quantization_config, after compress_model and after decompress_model, and the quantization_config written to config.json
    (tests/reference_compat/fuzz_model_compressor.py; oracle-backed ops, CPU)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reference_compat", "fuzz_model_compressor.py"), "30"],
                       capture_output=True, text=True, cwd="/tmp", timeout=600)
    lines = [line for line in r.stdout.splitlines() if "checked" in line]
    assert r.returncode == 0 and len(lines) == 1 and lines[0].endswith(" 0 mismatches"), r.stdout[-2000:] + r.stderr[-600:]
