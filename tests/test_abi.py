"""CPU tests of the drop-in boundary: the C-ABI library builds, loads and exports exactly the
symbols include/bfgpu.h declares; without a GPU every compute entry point fails loudly (no CPU
fallback)."""
import os
import re
import subprocess

import pytest

import zkvm_brainfuck_b200 as bf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "bfgpu.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(bfgpu_[a-z0-9_]+)\s*\(", txt)))


def test_header_and_binding_table_agree():
    assert header_symbols() == sorted(bf.ABI)


def test_library_exports_every_declared_symbol():
    out = subprocess.check_output(["nm", "-D", "--defined-only", bf.SO_PATH], text=True)
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    missing = [s for s in header_symbols() if s not in exported]
    assert not missing, missing
    lib = bf.lib()
    for s in header_symbols():
        assert getattr(lib, s)


def test_library_is_sm100a_native():
    # the toolkit that built the library (build.py's nvcc), which need not be on PATH
    cuobjdump = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
    out = subprocess.run([cuobjdump if os.path.exists(cuobjdump) else "cuobjdump", "-lelf", bf.SO_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(bf.BfGpuError, match="no CPU fallback"):
        bf.Context()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "zkvm-brainfuck_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("no oracle", ""), os.path.join(dirpath, f)


def test_rust_sys_crate_declares_every_symbol():
    """integration/bf-gpu-sys/src/lib.rs is generated from include/bfgpu.h (scripts/gen_rust_sys.py): the committed file must be what
    the generator emits today, and it must declare every symbol the library exports."""
    import importlib.util
    import re
    spec = importlib.util.spec_from_file_location("gen_rust_sys", os.path.join(ROOT, "scripts", "gen_rust_sys.py"))
    g = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(g)
    src, names = g.render()
    assert open(g.OUT).read() == src, "run `python scripts/gen_rust_sys.py`"
    declared = set(re.findall(r"pub fn (bfgpu_[a-z_0-9]+)\(", src))
    assert declared == set(bf.ABI), (declared ^ set(bf.ABI))


def test_header_is_plain_c():
    """The boundary is a C ABI: include/bfgpu.h must compile as C99 (what cgo / bindgen / a C caller sees), warning-free, and as C++."""
    import subprocess
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bfgpu.h")
    for cmd in (["gcc", "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", hdr],
                ["g++", "-fsyntax-only", "-x", "c++", "-std=c++17", "-Wall", "-Wextra", "-Werror", hdr]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
