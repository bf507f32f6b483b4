"""The drop-in boundary: the C-ABI library builds, loads, exports exactly what
include/hypergen_b200.h declares, and refuses to run without a GPU (no CPU fallback)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "hypergen_b200.h")).read()
    return sorted(set(re.findall(r"HG_API\s+[\w\s\*]+?\b(hg_\w+)\s*\(", src)))


def test_header_symbols_all_exported(hg):
    lib = hg.ffi.load()
    names = _declared()
    assert len(names) >= 17
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(hg.ffi.EXPORTS) == names


def test_library_is_sm100a_native(hg):
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", hg.ffi.lib_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback_without_device(hg):
    # in a child process that sees no device, so that the check also runs where a GPU is present
    import subprocess
    import sys
    code = ("import hypergen_b200 as hg\n"
            "try:\n"
            "    hg.Context(0)\n"
            "except hg.HyperGenError as e:\n"
            "    assert e.code == hg.ffi.HG_E_CUDA and 'no CPU fallback' in str(e), e\n"
            "else:\n"
            "    raise SystemExit('hg_init succeeded without a visible device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "hyper-gen_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import oracle|from oracle)", txt, re.M), f
                assert "libhg_oracle" not in txt and "libhgref" not in txt, f
                assert not re.search(r"#include\s*[<\"].*oracle", txt), f


def test_struct_layouts(hg):
    assert ctypes.sizeof(hg.ffi.SketchParams) == 24
    assert hg.ffi.HIT_DTYPE.itemsize == 16
