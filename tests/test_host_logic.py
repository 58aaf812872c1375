"""CPU-only checks of the product's host side: the C-ABI library loads and exports every declared symbol, the file
reader / quantizer / error layer behave like the reference's, and the device code's bit twiddling is right (compiled
for the host). No kernel is launched here."""
import ctypes
import hashlib
import json
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, QUANT_FORMATS, ROOT, VERSIONS, has_gpu, model_path
import ggml_file as gf
import rwkv_oracle as ro

# what the compiled reference exports and writes (tests/golden/make_ref_library_golden.py)
REF_LIBRARY = json.load(open(os.path.join(GOLDEN, "ref_library.json")))

ERR = dict(ARGS=1 << 8, FILE=2 << 8, MODEL=3 << 8, MODEL_PARAMS=4 << 8, GRAPH=5 << 8, CTX=6 << 8, ALLOC=1, FILE_OPEN=2, FILE_STAT=3,
           FILE_READ=4, FILE_WRITE=5, FILE_MAGIC=6, FILE_VERSION=7, DATA_TYPE=8, UNSUPPORTED=9, SHAPE=10, DIMENSION=11, KEY=12,
           DATA=13, PARAM_MISSING=14)


def test_exports_every_declared_symbol(lib):
    declared = set()
    for header in ("rwkv.h", "rwkv_b200.h"):
        text = open(os.path.join(ROOT, "include", header)).read()
        declared |= set(re.findall(r"RWKV_API[^;(]*?\b(rwkv_[a-z0-9_]+)\s*\(", text))
    assert len(declared) >= 29
    out = subprocess.run(["nm", "-D", "--defined-only", lib.path], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (rwkv_[a-z0-9_]+)", out))
    assert declared <= exported, declared - exported
    for name in declared:
        getattr(lib.library, name)
    # nothing from the oracle or torch leaks into the product library
    deps = subprocess.run(["ldd", lib.path], capture_output=True, text=True).stdout
    assert "torch" not in deps and "rwkv_ref" not in deps


def test_reference_abi_signatures_match():
    """Same exported names as the reference library (SURVEY.md 8b), as listed in tests/golden/ref_library.json."""
    ref_syms = set(REF_LIBRARY["exported_symbols"])
    assert len(ref_syms) >= 19
    import __graft_entry__
    ours = set(re.findall(r" T (rwkv_[a-z0-9_]+)", subprocess.run(["nm", "-D", "--defined-only", __graft_entry__.load_package().library_path()],
                                                                 capture_output=True, text=True).stdout))
    assert ref_syms <= ours, ref_syms - ours


@pytest.mark.parametrize("ver", VERSIONS)
def test_inspect_file_matches_oracle(lib, ver):
    for fmt in ("FP32", "Q5_1"):
        info = lib.rwkv_b200_inspect_file(model_path(ver, fmt))
        m = ro.OracleModel(model_path(ver, fmt))
        assert (info.n_vocab, info.n_embed, info.n_layer) == (m.n_vocab, m.n_embed, m.n_layer)
        assert (info.arch_major, info.arch_minor) == (m.major, m.minor)
        assert (info.head_count, info.head_size) == (m.head_count, m.head_size)
        assert info.state_len == m.state_len
        assert info.n_tensors == len(m.file.tensors)
        assert info.bytes_per_token == ro.bytes_per_token(model_path(ver, fmt))


def test_file_errors(lib, tmp_path):
    from rwkv_cpp_b200.shared_library import FileInfo
    lib.rwkv_set_print_errors(None, False)

    def inspect(path):   # raw C call: returns (ok, flags)
        ok = lib.library.rwkv_b200_inspect_file(str(path).encode(), ctypes.byref(FileInfo()))
        return ok, lib.rwkv_get_last_error(None)

    assert inspect("/nonexistent/model.bin") == (False, ERR["FILE"] | ERR["FILE_OPEN"])   # rwkv_model_loading.inc:295
    assert lib.rwkv_get_last_error(None) == 0                                              # reading clears (rwkv.cpp:229-234)
    assert inspect(model_path("4v0-660K", "FP32")) == (True, 0)
    good = open(model_path("4v0-660K", "FP32"), "rb").read()
    cases = {
        "magic": (struct.pack("<I", 0x12345678) + good[4:], ERR["FILE"] | ERR["FILE_MAGIC"]),        # rwkv_file_format.inc:117
        "version": (good[:4] + struct.pack("<I", 99) + good[8:], ERR["FILE"] | ERR["FILE_VERSION"]),  # :118
        "dtype": (good[:20] + struct.pack("<I", 4) + good[24:], ERR["FILE"] | ERR["DATA_TYPE"]),     # Q4_1_O removed format, :123-130
        "short": (good[:10], ERR["FILE"] | ERR["FILE_READ"]),                                         # :116
    }
    for name, (blob, want) in cases.items():
        p = tmp_path / f"{name}.bin"
        p.write_bytes(blob)
        assert inspect(p) == (False, want), name
    p = tmp_path / "truncated.bin"
    p.write_bytes(good[:len(good) // 2])
    ok, flags = inspect(p)
    assert not ok and flags & ERR["MODEL_PARAMS"]
    # quantised payload in a version-100 file is rejected (rwkv_file_format.inc:132-139)
    q = open(model_path("4v0-660K", "Q5_1"), "rb").read()
    p = tmp_path / "oldq.bin"
    p.write_bytes(q[:4] + struct.pack("<I", 100) + q[8:])
    assert inspect(p) == (False, ERR["FILE"] | ERR["DATA_TYPE"])
    with pytest.raises(ValueError):
        lib.rwkv_b200_inspect_file(str(p))
    # K-quants / Q8_1: ids 10..16 are in the reference's table (rwkv_file_format.inc:28-47) and ggml can run them; this engine has
    # kernels for FP32, FP16, Q4_0, Q4_1, Q5_0, Q5_1, Q8_0 only (rwkv.h documents exactly those as quantisation targets) and says so
    # with MODEL_PARAMS | UNSUPPORTED instead of loading something it cannot evaluate (documented in include/rwkv.h, INTEGRATION.md)
    first = 24                                   # first tensor header: dim_count, key_length, data_type
    for dt in (10, 11, 12, 13, 14, 15, 16):
        p = tmp_path / f"kquant{dt}.bin"
        p.write_bytes(q[:first + 8] + struct.pack("<i", dt) + q[first + 12:])
        assert inspect(p) == (False, ERR["MODEL_PARAMS"] | ERR["UNSUPPORTED"]), dt


def test_print_errors_flag(lib):
    assert lib.rwkv_get_print_errors(None) is False
    lib.rwkv_set_print_errors(None, True)
    assert lib.rwkv_get_print_errors(None) is True
    lib.rwkv_set_print_errors(None, False)


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(lib):
    """Without a CUDA device the product must fail loudly -- there is no host execution path to fall back to."""
    with pytest.raises(ValueError):
        lib.rwkv_init_from_file(model_path("6v0-3m", "FP32"), 1, 0)
    lib.rwkv_init_from_file  # noqa
    ptr = lib.library.rwkv_init_from_file(model_path("6v0-3m", "FP32").encode(), 1, 0)
    assert not ptr
    assert lib.rwkv_get_last_error(None) == ERR["CTX"] | ERR["UNSUPPORTED"]
    y = np.zeros(4, np.float32)
    ok = lib.library.rwkv_b200_matvec(0, 4, 4, 1, np.eye(4, dtype=np.float32).ctypes.data, y.ctypes.data_as(ctypes.POINTER(ctypes.c_float)),
                                      y.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), 0)
    assert not ok


@pytest.mark.parametrize("fmt", QUANT_FORMATS)
def test_quantizer_bit_exact_vs_oracle(lib, fmt, tmp_path):
    """rwkv_quantize_model_file (rwkv_quantize.inc:16-171) vs the numpy restatement of quantize_row_*_ref, tensor by tensor."""
    for ver, src in (("6v0-3m", "FP32"), ("7v0-834K", "FP16"), ("5v1-730K", "FP32")):
        out = tmp_path / f"{ver}-{src}-{fmt}.bin"
        lib.rwkv_quantize_model_file(model_path(ver, src), str(out), fmt)
        a, b = gf.read_model_file(model_path(ver, src)), gf.read_model_file(str(out))
        assert b.version == 101 and b.data_type == gf.TYPE_IDS[fmt] and list(a.tensors) == list(b.tensors)
        n_quant = 0
        for name, ta in a.tensors.items():
            tb = b.tensors[name]
            assert ta.ne == tb.ne
            skip = name in ("emb.weight", "head.weight") or any(s in name for s in ("att.v1", "att.v2", "att.g1", "att.g2", "att.a1", "att.a2", "att.w1", "att.w2", "att.r_k"))
            if len(ta.ne) == 2 and not skip:
                n_quant += 1
                assert tb.dtype == gf.TYPE_IDS[fmt], name
                x = ro.dequantize(ta.dtype, ta.raw, int(np.prod(ta.ne)))
                assert np.array_equal(ro.quantize_row_ref(tb.dtype, x), tb.raw), name
            else:
                assert tb.dtype == ta.dtype and np.array_equal(ta.raw, tb.raw), name
        assert n_quant > 0


def test_quantizer_matches_compiled_reference(lib, tmp_path):
    """The files the compiled reference's rwkv_quantize_model_file writes, byte for byte (size and SHA-256 in tests/golden/ref_library.json)."""
    for ver in ("4v0-660K", "6v0-3m"):
        for fmt in QUANT_FORMATS:
            a = tmp_path / "a.bin"
            lib.rwkv_quantize_model_file(model_path(ver, "FP16"), str(a), fmt)
            data = a.read_bytes()
            want = REF_LIBRARY["quantized_from_fp16"][f"{ver}/{fmt}"]
            assert (len(data), hashlib.sha256(data).hexdigest()) == (want["bytes"], want["sha256"]), (ver, fmt)


def test_quantizer_errors(lib, tmp_path):
    with pytest.raises(ValueError):
        lib.rwkv_quantize_model_file(model_path("4v0-660K", "FP32"), str(tmp_path / "x.bin"), "Q3_K")
    assert not lib.library.rwkv_quantize_model_file(model_path("4v0-660K", "FP32").encode(), str(tmp_path / "x.bin").encode(), b"FP16")
    assert lib.rwkv_get_last_error(None) == ERR["ARGS"] | ERR["DATA_TYPE"]          # rwkv_quantize.inc:20-25
    assert not lib.library.rwkv_quantize_model_file(model_path("4v0-660K", "Q5_1").encode(), str(tmp_path / "x.bin").encode(), b"Q4_0")
    assert lib.rwkv_get_last_error(None) == ERR["FILE"]                              # input must be FP32/FP16 (rwkv_quantize.inc:45-50)


def test_device_bit_twiddling_on_host(tmp_path):
    """Compiles the __host__ __device__ quant decoding of the GEMV kernel for the CPU and checks it against a scalar decode."""
    exe = tmp_path / "host_kernels_check"
    cmd = ["/usr/local/cuda/bin/nvcc", "-std=c++17", "-O1", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-ffp-contract=off,-Wno-unknown-pragmas",
           "-o", str(exe), os.path.join(ROOT, "tests", "host_kernels_check.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout


def test_synthetic_model_loads_in_oracle(tmp_path):
    import synthetic_model as sm
    p = tmp_path / "syn.bin"
    sm.write_direct(str(p), "rwkv6-small", "Q5_1", seed=3)
    m = ro.OracleModel(str(p))
    logits, state = m.eval_sequence(sm.synthetic_tokens(4, m.n_vocab))
    assert np.isfinite(logits).all() and 0.3 < logits.std() < 3.0


def test_quantize_cli_matches_library_call(lib, tmp_path):
    """rwkv.cpp_b200/quantize.py (the reference's python/quantize.py CLI) writes the file the library call writes."""
    src = model_path("5v2-730K", "FP16")
    a, b = tmp_path / "cli.bin", tmp_path / "lib.bin"
    r = subprocess.run([os.sys.executable, os.path.join(ROOT, "rwkv.cpp_b200", "quantize.py"), src, str(a), "Q4_1"], capture_output=True, text=True)
    assert r.returncode == 0 and "Done" in r.stdout, r.stderr[-500:]
    lib.rwkv_quantize_model_file(src, str(b), "Q4_1")
    assert a.read_bytes() == b.read_bytes()
    r = subprocess.run([os.sys.executable, os.path.join(ROOT, "rwkv.cpp_b200", "quantize.py"), src, str(a), "Q9_9"], capture_output=True, text=True)
    assert r.returncode != 0


def test_no_kernel_spills_its_parameters(lib):
    """Round 2, GPU call 10: a `const LnTail &` taken INTO the kernel parameter made nvcc copy the 1.6 KB GemvBatch into every
    thread's local memory at kernel entry (a 1624-byte stack frame): every GEMV launch 2-4x slower, found only on the GPU. This reads
    the resource usage of the built library on the CPU: no kernel of the eval path may have a stack frame above 256 bytes
    (the sampling kernel, one launch per sampled token, keeps its sorted candidate list in local memory on purpose)."""
    r = subprocess.run(["cuobjdump", "--dump-resource-usage", lib.path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump not available")
    names = re.findall(r"Function ([^:\s]+):\s*\n\s*REG:(\d+) STACK:(\d+)", r.stdout)
    assert len(names) > 20, "no kernels found in %s" % lib.path
    fat = [(n, int(st)) for n, _, st in names if int(st) > 256 and "sample_kernel" not in n]
    assert not fat, fat


def test_bench_reference_arm_line(tmp_path):
    """`bench.py --impl reference` (the driver's reference arm) on a tiny synthetic workload, on the CPU: ONE JSON line on stdout with
    the keys the contract names, timed through the UNMODIFIED reference library (oracle/_ref) -- no CUDA needed for this arm."""
    import json
    import ref_lib
    import sys
    if ref_lib.reference_library_path() is None:
        pytest.skip("oracle/_ref not built")
    env = dict(os.environ, RWKV_B200_BENCH_DIR=str(tmp_path))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "rwkv6-small:Q5_1", "--steps", "4", "--warmup", "1",
                        "--cpu-budget-s", "5"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "decode_tokens_per_sec" and line["unit"] == "tokens/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert "workload" in line["config"] and "model" not in line["config"]


def test_decode_gemv_instantiations_stay_small(lib):
    """Round 2: the single-token GEMV launches of a model whose matrices share one weight format run an instantiation compiled for that
    format (and, for every launch but the head, without the LayerNorm prologue): ~2 600 instructions where the one-kernel-for-everything
    build had 15 500, of which ncu charged a third of the stall cycles to instruction fetch (2.81 -> 2.41 ms per 7B token). This reads
    the SASS of the built library: the per-format instantiations must exist for all seven formats and stay compact."""
    r = subprocess.run(["cuobjdump", "-sass", lib.path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump not available")
    sizes, name, count = {}, None, 0
    for ln in r.stdout.splitlines():
        if "Function :" in ln:
            if name:
                sizes[name] = count
            name, count = ln.split("Function :")[1].strip(), 0
        elif "/*" in ln and name and re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln):
            count += 1
    if name:
        sizes[name] = count
    per_type = {n: c for n, c in sizes.items() if "gemv_tma_kernelILi1ELb1ELi" in n and "ELin1E" not in n}
    no_ln = [c for n, c in per_type.items() if n.endswith("ELb0EEEvNS_9GemvBatchE")]
    with_ln = [c for n, c in per_type.items() if n.endswith("ELb1EEEvNS_9GemvBatchE")]
    assert len(no_ln) == 7 and len(with_ln) == 7, sorted(per_type)
    assert max(no_ln) < 3500 and max(with_ln) < 5500, (no_ln, with_ln)
    generic = [c for n, c in sizes.items() if "gemv_tma_kernelILi1ELb1ELin1E" in n]
    assert generic and max(no_ln) * 3 < generic[0], (generic, no_ln)
