"""Writes tests/golden/funasrruntime_client_symbols.txt: the C++ runtime entry points (FunOffline*, FunASR*, FunWfst*,
CompileHotwordEmbedding, as mangled names) that examples/offline_runtime_client.cpp needs when it is compiled against the REFERENCE's
own runtime/onnxruntime/include/funasrruntime.h.  tests/test_abi_host.py checks that libfunasr_b200.so defines every one of them,
which is what makes a client built against that header link.  TEST INFRASTRUCTURE ONLY; needs the reference tree, g++ and nm.
Usage: python oracle/make_runtime_symbols_golden.py"""
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)

import ref_shim  # noqa: E402

SYMBOLS = os.path.join(ROOT, "tests", "golden", "funasrruntime_client_symbols.txt")


def reference_header_dir():
    return os.path.join(ref_shim.REFERENCE_ROOT, "runtime", "onnxruntime", "include")


def client_runtime_symbols(header, include_dir):
    """Compile the example client (-c) with FUNASR_RUNTIME_HEADER=header found in include_dir -> sorted undefined symbols that are
    free functions at global scope (mangled _Z<length><name>...), i.e. the runtime API; libstdc++ / libc symbols are left out."""
    with tempfile.TemporaryDirectory() as d:
        obj = os.path.join(d, "client.o")
        subprocess.run(["g++", "-std=c++17", "-c", "-DFUNASR_RUNTIME_HEADER=" + header, "-I" + include_dir, "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "offline_runtime_client.cpp"), "-o", obj], check=True, capture_output=True, text=True)
        out = subprocess.run(["nm", "-u", obj], check=True, capture_output=True, text=True).stdout
    return sorted(s for s in (ln.split()[-1] for ln in out.splitlines() if ln.strip()) if re.match(r"_Z\d+", s))


if __name__ == "__main__":
    assert os.path.exists(os.path.join(reference_header_dir(), "funasrruntime.h")), "needs the reference tree"
    syms = client_runtime_symbols('"funasrruntime.h"', reference_header_dir())
    with open(SYMBOLS, "w") as f:
        f.write("\n".join(syms) + "\n")
    print("wrote", SYMBOLS, len(syms), "symbols")
