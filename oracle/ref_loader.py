"""Loads the UNMODIFIED reference modules for oracle validation and golden generation.

Test infrastructure only.  Works only where a checkout of the reference
(Kelicious/faster_rcnn) is present: at oracle/_ref/ (git-ignored), or wherever
FRCNN_REFERENCE_DIR names its `faster_rcnn` module folder.  Nothing under
`-m gpu`, smoke() or bench.py may call this.  The reference is a flat script
directory (modules import each other by bare name), so its folder is pushed on
sys.path; `@profile` (custom_decorators.py:8-33) prints a call tree on every
call, which `quiet()` swallows.
"""
import contextlib
import io
import os
import sys

REF_DIR = os.environ.get("FRCNN_REFERENCE_DIR",
                         os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "faster_rcnn"))
# the VOC2007 annotations the reference ships next to its module folder
VOC_DIR = os.path.join(os.path.dirname(os.path.abspath(REF_DIR)), "test_data", "VOC_test")


def available():
    return os.path.isfile(os.path.join(REF_DIR, "det_util.py"))


def load():
    """Returns a namespace with the numpy-only reference modules."""
    if not available():
        raise RuntimeError("reference not present: check it out at oracle/_ref/ or set FRCNN_REFERENCE_DIR "
                           "to its faster_rcnn folder")
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import types
    import util, shapes, shared_constants, rpn_util, det_util      # noqa: E401
    from data import voc_data_helpers
    return types.SimpleNamespace(util=util, shapes=shapes, shared_constants=shared_constants,
                                 rpn_util=rpn_util, det_util=det_util, voc=voc_data_helpers)


def quiet():
    return contextlib.redirect_stdout(io.StringIO())
