"""The C-ABI boundary: libggb200.so loads without a GPU, exports every symbol include/ggb200.h and
include/gg_synth.h declare, and refuses loudly to run without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

from greengage_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gg_[a-z0-9_]+)\s*\(", txt)))


def _exported(lib):
    out = subprocess.check_output(["nm", "-D", "--defined-only", lib]).decode()
    return {ln.split()[-1] for ln in out.splitlines() if " T " in ln}


def test_device_library_exports_every_declared_symbol():
    decl = _declared("ggb200.h")
    assert len(decl) > 25
    exp = _exported(os.path.join(ROOT, "greengage_b200", "libggb200.so"))
    missing = [s for s in decl if s not in exp]
    assert missing == [], missing


def test_host_library_exports_every_declared_symbol():
    decl = _declared("gg_synth.h")
    exp = _exported(os.path.join(ROOT, "greengage_b200", "libgghost.so"))
    assert [s for s in decl if s not in exp] == []


def test_struct_layouts_match_header():
    # sizes the C side is compiled with (gg_plan.h)
    assert C.sizeof(capi.gg_attr) == 16 and C.sizeof(capi.gg_expr) == 48 and C.sizeof(capi.gg_aggval) == 40
    assert C.sizeof(capi.gg_tupdesc) == 8 + 16 * 32
    assert C.sizeof(capi.gg_aggrow) == 8 * 4 + 4 * 4 + 4 * 4 + 40 * 16
    assert C.sizeof(capi.gg_agg) == 4 + 4 + 16 + 4 + 4 + 8 * 16 + 8


def test_no_gpu_means_no_engine():
    """in a process that sees no CUDA device, which on a GPU machine takes an empty CUDA_VISIBLE_DEVICES"""
    code = ("import ctypes as C\n"
            "from greengage_b200 import capi\n"
            "h = C.c_void_p()\n"
            "rc = capi.dev_lib().gg_engine_create(0, C.byref(h))\n"
            "assert rc != 0 and not h\n"
            "assert b'no CPU fallback' in capi.dev_lib().gg_last_error()\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
