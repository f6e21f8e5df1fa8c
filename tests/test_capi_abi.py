"""The C-ABI shared library builds for sm_100a without a GPU, loads, exports every symbol that
include/frcnn_b200.h declares with the argument count the ctypes binding uses, and fails loudly (error
code, no crash, no fallback) when no CUDA device is present.  No compute calls here."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "frcnn_b200.h")


@pytest.fixture(scope="module")
def lib():
    from faster_rcnn_b200 import _build, _lib
    _build.build()
    return _lib.load()


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    decls = {}
    for m in re.finditer(r"FRCNN_API\s+[\w\s\*]+?\b(frcnn_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        decls[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    return decls


def test_every_declared_symbol_is_exported_and_bound(lib):
    from faster_rcnn_b200 import _lib
    decls = _declared()
    assert len(decls) >= 20
    assert set(decls) == set(_lib.SIGNATURES), "ctypes table and header disagree"
    for name, n_args in decls.items():
        assert getattr(lib, name) is not None
        assert len(_lib.SIGNATURES[name][1]) == n_args, name
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\b(frcnn_\w+)\b", out))
    assert exported == set(decls), "the .so must export exactly the header's symbols"


def test_library_carries_sm100a_code_only(lib):
    from faster_rcnn_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_sources_read_no_environment_variables():
    """Launch configurations follow from the source, the problem shape and the device alone."""
    csrc = os.path.join(ROOT, "faster_rcnn_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, name)) as f:
            assert "getenv" not in f.read(), name


def test_abi_version_and_loud_failure_without_gpu(lib):
    import torch
    assert lib.frcnn_abi_version() == 1
    assert lib.frcnn_last_error(None) == b"null handle"
    assert lib.frcnn_launch_count(None) == 0
    if not torch.cuda.is_available():
        h = C.c_void_p()
        assert lib.frcnn_create(C.byref(h), 0) < 0 and not h.value
        from faster_rcnn_b200 import runtime
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            runtime.get_context()
        import numpy as np
        from faster_rcnn_b200 import det_util
        with pytest.raises(RuntimeError):
            det_util.nms(np.zeros((3, 4), np.int16), np.ones(3, np.float32))
