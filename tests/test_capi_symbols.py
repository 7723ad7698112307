"""CPU: the C-ABI library builds/loads and exports every symbol include/mmbidaf_b200.h declares."""
import os
import re
import subprocess
import sys

from conftest import ROOT


def _declared():
    text = open(os.path.join(ROOT, "include", "mmbidaf_b200.h")).read()
    return sorted(set(re.findall(r"MMB_API\s+[\w\s\*]+?\b(mmb_\w+)\s*\(", text)))


def test_header_declares_entry_points():
    names = _declared()
    assert "mmb_bidaf_fwd" in names and "mmb_version" in names


def test_library_exports_every_declared_symbol():
    from mmbidaf_b200 import _lib, build
    build.build()
    handle = _lib.load()
    for name in _declared():
        assert hasattr(handle, name), name
        assert name in _lib.SIGNATURES, f"{name} missing from the ctypes signature table"
    assert set(_lib.SIGNATURES) == set(_declared())
    assert handle.mmb_version() >= 100


def test_no_cpu_fallback_without_device():
    """In a process that sees no CUDA device (none installed, or hidden from it), every op refuses to run."""
    code = ("import pytest\nfrom mmbidaf_b200 import _lib\n"
            "with pytest.raises(RuntimeError, match='no CPU path'):\n    _lib.lib()\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
