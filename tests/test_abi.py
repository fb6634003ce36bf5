"""CPU: the C-ABI library loads and exports every symbol include/step_b200.h declares; the product
never imports the oracle; no compute calls are made here (no GPU in this tier)."""
import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "step_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(step_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from step_b200 import _lib
    lib = _lib.lib()
    declared = header_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), "libstep_b200.so does not export %s" % name
    assert lib.step_version() == 100
    # python binding covers the whole header (plus the debug hook)
    bound = set(_lib.exported_symbols())
    assert set(declared) <= bound, sorted(set(declared) - bound)


def test_library_is_sm100a_native():
    from step_b200 import build
    # the toolkit that built the library, also when its bin/ is not on PATH
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(build.NVCC), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", os.path.join(ROOT, "step_b200", "libstep_b200.so")],
                         capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_product_never_touches_the_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "step_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M) or "oracle/" in txt or "/root/reference" in txt:
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_ops_raise_without_cuda_tensor():
    import pytest
    import torch
    from step_b200 import roi_layers
    x = torch.zeros(1, 8, 4, 4)
    with pytest.raises(RuntimeError):
        roi_layers.roi_align(x, torch.zeros(1, 5), (7, 7), 1 / 16., 0)
    assert roi_layers.nms(torch.zeros(0, 4), torch.zeros(0), 0.4).numel() == 0  # empty in -> empty out, nms.h:41


def test_argument_errors_are_reported_before_any_device_work():
    """The entry points validate their arguments first (STEP_E_ARG + step_last_error text), the role AT_ASSERTM plays in
    the reference's ops: checked here without a GPU on the fused bottleneck exit, which exists for the reference's head
    widths only (two_branch.py:190-192)."""
    import ctypes
    from step_b200 import _lib
    lib = _lib.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    rc = lib.step_bottleneck_exit_f16(p, 128, p, p, 1024, p, None, 1, None, 0, p, 256, 64, 128, 1024, 256, None)
    assert rc == 10001                                        # STEP_E_ARG
    lib.step_last_error.restype = ctypes.c_char_p
    assert b"planes 256" in lib.step_last_error()
    rc = lib.step_bottleneck_exit_f16(None, 256, p, p, 1024, p, None, 1, None, 0, p, 256, 64, 256, 1024, 256, None)
    assert rc == 10001 and b"null pointer" in lib.step_last_error()
