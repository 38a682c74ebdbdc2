"""The C-ABI library loads on a CPU-only box and exports every symbol include/dark_bwt.h declares
(no compute calls here: there is no GPU and no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def declared_functions():
    src = open(os.path.join(ROOT, "include", "dark_bwt.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dark_bwt_[a-z_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(lib):
    from dark_b200 import _ffi
    names = declared_functions()
    assert len(names) >= 14
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/dark_bwt.h but not exported"
    assert sorted(_ffi.SYMBOLS) == names


def test_abi_version_and_strerror(lib):
    assert lib.dark_bwt_abi_version() == 2
    msgs = {lib.dark_bwt_strerror(c).decode() for c in range(0, 7)}
    assert len(msgs) == 7 and "ok" in msgs


def test_stats_struct_layout_matches_header():
    """ctypes mirror vs the C struct: compile a tiny C program that prints sizeof/offsetof."""
    import subprocess
    import tempfile
    from dark_b200 import _ffi
    fields = [f for f, _ in _ffi.Stats._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "dark_bwt.h"\nint main(){printf("%zu", sizeof(dark_bwt_stats));\n'
    for f in fields:
        prog += f'printf(" %zu", offsetof(dark_bwt_stats, {f}));\n'
    prog += "return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(prog)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        vals = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert vals[0] == ctypes.sizeof(_ffi.Stats)
    assert vals[1:] == [getattr(_ffi.Stats, f).offset for f in fields]


def test_dc_info_struct_layout_matches_header():
    import subprocess
    import tempfile
    from dark_b200 import _ffi
    fields = [f for f, _ in _ffi.DcInfo._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "dark_bwt.h"\nint main(){printf("%zu", sizeof(dark_bwt_dc_info));\n'
    for f in fields:
        prog += f'printf(" %zu", offsetof(dark_bwt_dc_info, {f}));\n'
    prog += "return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(prog)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        vals = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert vals[0] == ctypes.sizeof(_ffi.DcInfo)
    assert vals[1:] == [getattr(_ffi.DcInfo, f).offset for f in fields]


def test_null_arguments_are_rejected_before_any_device_work(lib):
    """Argument checks of the entry points run before anything touches CUDA: DARK_BWT_E_INVALID_ARG (2), no crash."""
    from dark_b200 import _ffi
    o = ctypes.c_uint64(0)
    assert lib.dark_bwt_forward(None, None, 10, None, ctypes.byref(o), None, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_device(None, None, 10, None, ctypes.byref(o), None, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_batch(None, None, None, None, None, None, 3, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_many(None, None, None, None, None, 3, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_many_device(None, None, None, 3, None, None, None, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_capacity(None) == 0
    lib.dark_bwt_destroy(None)


def test_no_cpu_fallback_create_fails_without_gpu(lib):
    """Where no CUDA device is visible the product path must fail loudly.  The check runs in a fresh process that sees
    no device, so that it also runs on a machine that has one."""
    import subprocess
    import sys
    code = ("from dark_b200 import saca, DarkBwtError\n"
            "try:\n"
            "    saca.Constructor(1024)\n"
            "except DarkBwtError:\n"
            "    print('raised')\n")
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=ROOT,
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "raised", (out.stdout, out.stderr[-2000:])


def test_product_never_touches_the_oracle():
    """dark_b200/ (the product) must not import, link or mention oracle/."""
    pkg = os.path.join(ROOT, "dark_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in text and "liboracle" not in text and "oracle/" not in text.replace(
                    "oracle/gen.c; tests", ""), f


def test_cpp_mirror_compiles_and_links(lib, tmp_path):
    """The C++ host-side mirror of saca::Constructor (dark_b200/csrc/saca.hpp) builds against the C ABI."""
    import subprocess
    from dark_b200 import _ffi
    exe = tmp_path / "saca_cpp_demo"
    libdir = os.path.dirname(_ffi.lib_path())
    subprocess.check_call(["g++", "-std=c++17", "-I", ROOT, os.path.join(ROOT, "examples", "saca_cpp_demo.cpp"), "-L", libdir,
                           "-ldark_bwt", f"-Wl,-rpath,{libdir}", "-o", str(exe)])
    assert exe.exists()
