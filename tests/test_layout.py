"""Repo-layout contract (CPU): the C-ABI library exports every symbol include/avb200.h declares and
the ctypes table types each of them; the product package never touches oracle/ or a CPU fallback."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "avb200.h")).read()
    return sorted(set(re.findall(r"AVB_API\s+[\w\s\*]+?\b(avb_\w+)\s*\(", src)))


def test_header_symbols_exported_and_typed():
    from animal_vision_b200 import _abi
    names = _declared()
    assert len(names) >= 10
    lib = _abi.load()                      # builds with nvcc if needed; no GPU required to load
    for n in names:
        assert hasattr(lib, n), f"libavb200.so does not export {n}"
        assert n in _abi.SIGNATURES, f"_abi.SIGNATURES does not type {n}"
    assert sorted(_abi.SIGNATURES) == names, "ctypes table and header disagree"
    assert lib.avb_version() == _abi.AVB_VERSION
    raw = ctypes.CDLL(_abi.lib_path())
    assert raw.avb_version() == _abi.AVB_VERSION


def test_product_never_imports_oracle_or_reference():
    pkg = os.path.join(ROOT, "animal_vision_b200")
    bad = []
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(d, f), errors="replace").read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M) or "/root/reference" in txt:
                    bad.append(os.path.join(d, f))
    assert not bad, f"product code must not import the oracle or read the reference: {bad}"


def test_compute_fails_loudly_without_gpu():
    import numpy as np
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from animal_vision_b200._abi import AvbError
    from animal_vision_b200.animals import Dog
    with pytest.raises(AvbError):
        Dog().visualize(np.zeros((4, 4, 3), np.uint8))


def test_kernel_sources_have_no_variant_switches():
    """Kernel variants are chosen from the input alone: no source under csrc/ reads an AVB_* environment variable, and
    the retired #ifdef experiments stay gone."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "animal_vision_b200", "csrc", "*.cu")) +
                   glob.glob(os.path.join(ROOT, "animal_vision_b200", "csrc", "*.cuh")))
    assert files
    for f in files:
        src = open(f).read()
        name = os.path.basename(f)
        assert not re.search(r'getenv\s*\(\s*"AVB_', src), f"{name} reads an AVB_* environment variable"
        assert not re.search(r"#\s*ifdef\s+(AVB_ENC_NO_THRESHOLD|UV_SQRT_RN)\b", src), f"{name} keeps a retired experiment"
