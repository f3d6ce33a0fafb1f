"""TEST ONLY: builds adapter/_build/libsva_adapter_test.so = adapter/sva_functions.cpp (+ test glue) compiled against oracle/cvshim
and the reference's headers, linked to stereovisionarray_b200/libsva_b200.so.  The headers are the reference's own
($SVA_REFERENCE_DIR/include) where that tree is given, otherwise the stand-ins in adapter/refshim."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("SVA_REFERENCE_DIR", "")
OUT = os.path.join(HERE, "_build", "libsva_adapter_test.so")


def reference_include():
    inc = os.path.join(REF, "include") if REF else ""
    return inc if inc and os.path.exists(os.path.join(inc, "functions.h")) else os.path.join(HERE, "refshim")


def build():
    inc = reference_include()
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    srcs = [os.path.join(HERE, "sva_functions.cpp"), os.path.join(HERE, "adapter_test_glue.cpp")]
    deps = srcs + [os.path.join(inc, h) for h in ("Camera.h", "functions.h", "dlibFaceSelect.h")]
    lib = os.path.join(ROOT, "stereovisionarray_b200", "libsva_b200.so")
    if os.path.exists(OUT) and all(os.path.getmtime(OUT) > os.path.getmtime(s) for s in deps + [lib]):
        return OUT
    cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-I" + os.path.join(ROOT, "oracle", "cvshim"), "-I" + inc,
           "-I" + os.path.join(ROOT, "include")] + srcs + ["-o", OUT, lib, "-Wl,-rpath,$ORIGIN/../../stereovisionarray_b200", "-Wl,--no-undefined"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("adapter test build failed")
    return OUT


if __name__ == "__main__":
    print(build())
