"""Import the ORIGINAL PROJECT's package (OpenPPL/ppq, unmodified) -- test infrastructure, used only to record the golden results under
tests/golden/ that the tests compare against (tests/refrecord.py).

Where it comes from: the checkout named by $PPQ_REFERENCE_ROOT, else baseline/_ref (`pip install --no-deps --target baseline/_ref`,
git-ignored; DESIGN.md §10).

Two shims are needed (SURVEY.md §0 fact 6): the stale caffe protobuf module needs the pure-python protobuf implementation, and every
exporter imports `onnx` (absent) at package import time.  Neither touches the path under test.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CANDIDATES = [os.environ.get('PPQ_REFERENCE_ROOT'), os.path.join(ROOT, 'baseline', '_ref')]


def root():
    for c in _CANDIDATES:
        if c and os.path.isdir(os.path.join(c, 'ppq', 'core')):
            return c
    return None


def available() -> bool:
    return root() is not None


def load():
    """Returns the imported `ppq` package (the unmodified reference) or None when it is not on this machine."""
    r = root()
    if r is None:
        return None
    os.environ['PROTOCOL_BUFFERS_PYTHON_IMPLEMENTATION'] = 'python'
    from unittest.mock import MagicMock
    for m in ['onnx', 'onnx.helper', 'onnx.numpy_helper', 'onnx.mapping', 'onnx.checker', 'onnx.shape_inference']:
        sys.modules.setdefault(m, MagicMock())
    if r not in sys.path:
        sys.path.insert(0, r)
    import ppq
    return ppq


class use_extension:
    """Context: the real ppq.core.ffi serves `module` (ours or the reference's own build) and never tries to JIT."""

    def __init__(self, module):
        self.module = module

    def __enter__(self):
        import ppq.core.ffi as ffi
        h = ffi.CUDA_COMPLIER
        self._saved = (getattr(h, '__CUDA_EXTENTION__', None), type(h).complie)
        h.__CUDA_EXTENTION__ = self.module
        type(h).complie = lambda self_: None
        return self.module

    def __exit__(self, *exc):
        import ppq.core.ffi as ffi
        h = ffi.CUDA_COMPLIER
        h.__CUDA_EXTENTION__, type(h).complie = self._saved
        return False
