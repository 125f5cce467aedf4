"""CPU: the C-ABI library loads and exports every symbol include/auvrrt.h declares; without a GPU
every compute entry fails loudly (no CPU fallback)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def auvrrt():
    from auvrrt import build
    build.build()
    import auvrrt
    return auvrrt


def test_every_declared_symbol_is_exported(auvrrt):
    with open(os.path.join(ROOT, "include", "auvrrt.h")) as f:
        hdr = f.read()
    declared = set(re.findall(r"\b(auvrrt_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    L = auvrrt.lib()
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert declared == set(auvrrt._lib.EXPORTS)


def test_struct_layouts_match_header(auvrrt):
    import ctypes as C
    assert C.sizeof(auvrrt._lib.PlanRecord) == 96
    assert C.sizeof(auvrrt._lib.PlanParams) == 2 * 4 + 10 * 8 + 4 * 4 + 8 + 3 * 8 + 2 * 4
    assert auvrrt.api.RECORD_DTYPE.itemsize == 96


def test_no_cpu_fallback(auvrrt):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert auvrrt.api.device_count() == 0
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        auvrrt.Env([[0, 0, 1]], [[0, 0], [1, 0], [0, 1]])
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        auvrrt.api.nn([[0, 0]], [[1, 1]])
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        auvrrt.api.steer_arc([[0, 0, 0, 0, 0]], [0.5] * 4, [0, 4], [2.0, 0.5, 30.0, 0.5, 2.0])
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        auvrrt.api.steer_dubins([[0, 0, 0]], [[5, 5, 1]], W=4)
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        auvrrt.api.calibrate_fp32()
    from auvrrt import device
    with pytest.raises(auvrrt.AuvrrtError, match="no CUDA device"):
        device.SharkOccupancy([[[0, 0], [1, 0], [1, 1], [0, 1]]], [0, 0, 4, 4], 1.0, 5.0, 2.0, 2, 1, 16)


def test_product_never_imports_oracle():
    """only comments may mention the oracle; no import / load / include of anything under oracle/"""
    pkg = os.path.join(ROOT, "auv-sim_b200")
    bad = re.compile(r"(^\s*(from|import)\s+oracle)|liborc|orc\.|#include\s+\"[^\"]*oracle", re.M)
    for d, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                with open(os.path.join(d, fn)) as f:
                    assert not bad.search(f.read()), (d, fn)
