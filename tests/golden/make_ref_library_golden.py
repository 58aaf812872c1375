"""Generates tests/golden/ref_library.json from the UNMODIFIED reference library (oracle/_ref, built by oracle/Makefile from
the original rwkv.cpp sources, so run this where those exist): the rwkv_* symbols it exports, and the size and SHA-256 of the
files its rwkv_quantize_model_file writes from the FP16 fixtures. tests/test_host_logic.py checks our library against both."""
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_lib  # noqa: E402

QUANT_FORMATS = ["Q4_0", "Q4_1", "Q5_0", "Q5_1", "Q8_0"]


def main():
    path = ref_lib.reference_library_path()
    ref = ref_lib.load_reference_library()
    ref.rwkv_set_print_errors(None, False)
    nm = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    out = {"exported_symbols": sorted(set(re.findall(r" T (rwkv_[a-z0-9_]+)", nm))), "quantized_from_fp16": {}}
    with tempfile.TemporaryDirectory() as d:
        for ver in ("4v0-660K", "6v0-3m"):
            for fmt in QUANT_FORMATS:
                q = os.path.join(d, f"{ver}-{fmt}.bin")
                src = os.path.join(ROOT, "tests", "golden", "models", f"tiny-rwkv-{ver}-FP16.bin")
                assert ref.rwkv_quantize_model_file(src.encode(), q.encode(), fmt.encode()), (ver, fmt)
                data = open(q, "rb").read()
                out["quantized_from_fp16"][f"{ver}/{fmt}"] = {"sha256": hashlib.sha256(data).hexdigest(), "bytes": len(data)}
    json.dump(out, open(os.path.join(ROOT, "tests", "golden", "ref_library.json"), "w"), indent=1, sort_keys=True)
    print("wrote", len(out["exported_symbols"]), "symbols,", len(out["quantized_from_fp16"]), "hashes; library:", path)


if __name__ == "__main__":
    main()
