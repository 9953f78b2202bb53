"""The C-ABI library loads on a CPU-only box and exports exactly what
include/b200pt.h declares; the ctypes mirror matches the compiled structs."""
import ctypes as C
import os
import re
import subprocess
import sys

from conftest import ROOT


def test_library_loads_and_exports_every_symbol(built):
    from mitsuba3_b200 import abi
    lib = abi.load()
    header = open(os.path.join(ROOT, "include", "b200pt.h")).read()
    declared = sorted(set(re.findall(r"^B200PT_API [^;(]*?\b(b200pt_[a-z_0-9]+)\s*\(", header, re.M)))
    assert declared == sorted(abi.SYMBOLS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.b200pt_abi_version() == abi.ABI_VERSION


def test_struct_sizes_match(built):
    from mitsuba3_b200 import abi
    lib = abi.load()
    for i, st in enumerate([abi.Texture, abi.Bsdf, abi.Shape, abi.Emitter, abi.Sensor, abi.SceneDesc, abi.RenderParams, abi.Stats]):
        assert lib.b200pt_abi_sizeof(i) == C.sizeof(st), st.__name__


def test_fails_loudly_without_gpu(built):
    """No CPU fallback: without a device the product raises, it never routes elsewhere. The render runs in a
    subprocess that sees no device (empty CUDA_VISIBLE_DEVICES), so the check also runs on a machine with a GPU."""
    code = ("import mitsuba3_b200 as mb\n"
            "from mitsuba3_b200 import abi\n"
            "assert abi.load().b200pt_device_count() == 0\n"
            "sc = mb.load_dict(mb.cornell_box())\n"
            "try:\n"
            "    mb.render(sc, spp=1)\n"
            "except abi.B200PTError as e:\n"
            "    assert 'no CPU fallback' in str(e), e\n"
            "    print('RAISED')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join([ROOT, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "RAISED" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure; nothing under mitsuba3_b200/ may reference it."""
    pkg = os.path.join(ROOT, "mitsuba3_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.lower(), os.path.join(dp, f)
