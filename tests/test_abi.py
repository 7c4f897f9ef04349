"""The C-ABI library on a machine without a GPU: it builds (nvcc cross-compiles sm_100a), loads, exports
every function include/multimm_b200.h declares, and refuses to work rather than falling back."""
import ctypes
import os
import re
import subprocess

import pytest

from multimm_b200 import _lib
from multimm_b200.build import cuda_tool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "multimm_b200.h")


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mmm_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_list_agree():
    assert declared_functions() == sorted(_lib.EXPORTS)


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    missing = [name for name in declared_functions() if not hasattr(lib, name)]
    assert not missing, missing
    assert lib.mmm_abi_version() == 1


def test_library_is_sm100a_only_and_has_no_undefined_nccl_dependency(built_lib):
    out = subprocess.run([cuda_tool("cuobjdump"), "--list-elf", built_lib], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs
    # NCCL is opened with dlopen (single-GPU users and this CPU box need no libnccl at load time)
    needed = subprocess.run(["readelf", "-d", built_lib], capture_output=True, text=True).stdout
    assert "libnccl" not in needed


def test_every_entry_point_cites_the_reference():
    """Each block of the header names the reference lines it replaces."""
    text = open(HEADER).read()
    assert text.count("model.py:") >= 30 and "initial_structure_tools.py:157-166" in text and "plots.py" in text


def test_no_cpu_fallback_without_a_device(built_lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from multimm_b200.engine import Engine, Error

    with pytest.raises(Error, match="CUDA error"):
        Engine(100)


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under multimm_b200/ may import or load it."""
    pkg = os.path.join(ROOT, "multimm_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in src and "import oracle" not in src and "from oracle" not in src, f


def test_pair_kernel_resources_allow_two_ctas_per_sm(built_lib):
    """The Newton-3 kernel is designed for two resident 256-thread CTAs per SM (DESIGN.md 4.1):
    <= 128 registers per thread, static shared memory within the 48 KB that needs no opt-in, and the
    hot variant on packed f32x2 arithmetic.  A change that silently breaks one of these costs ~2x."""
    out = subprocess.run([cuda_tool("cuobjdump"), "--dump-resource-usage", built_lib], capture_output=True, text=True).stdout
    rows = re.findall(r"Function (\S*k_pair_n3\S*):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+)", out)
    assert len(rows) >= 16, len(rows)
    for name, reg, stack, shared in rows:
        assert int(reg) <= 128, (name, reg)
        assert int(shared) <= 48 * 1024, (name, shared)
        if "k_pair_n3ILin1E" in name:  # the generic variant (EVP = -1): FP64 body, i-beads indexed at run time
            assert int(stack) <= 512, (name, stack)  # (local memory by design: the slow path)
            continue
        assert int(stack) <= 192, (name, stack)  # spilled words live in the rare variants' prologues, never in a pair loop
    gw = [n for n, *_ in rows if "k_pair_n3ILi6ELi1ELb1" in n]
    assert len(gw) == 1
    sass = subprocess.run([cuda_tool("cuobjdump"), "-sass", "-fun", gw[0], built_lib], capture_output=True, text=True).stdout
    assert sass.count("FFMA2") >= 100 and "FMUL2" in sass and "FADD2" in sass
    assert "REDG.E.ADD.64" in sass  # the 64-bit fixed-point force accumulation
    # no pair loop (a backward branch around >= 100 packed FMAs) touches local memory: spills stay outside
    ins = re.findall(r"/\*([0-9a-f]{4,})\*/\s+(.*?);", sass)
    addr = {int(a, 16): k for k, (a, _) in enumerate(ins)}
    loops = 0
    for k, (a, op) in enumerate(ins):
        m = re.search(r"BRA\s+(?:\w+,\s*)?0x([0-9a-f]+)", op)
        if m and int(m.group(1), 16) < int(a, 16) and int(m.group(1), 16) in addr:
            body = [o for _, o in ins[addr[int(m.group(1), 16)]:k + 1]]
            if sum("FFMA2" in o for o in body) >= 100 and len(body) < 1200:
                loops += 1
                assert not any(o.startswith(("LDL", "STL")) for o in body), "spill inside a pair loop"
    assert loops >= 2  # the hot variant and at least one of the rarer ones
