"""Results of the original project (OpenPPL/ppq: its own CUDA kernels compiled for sm_100a, its Python package), stored under
tests/golden/ so that the tests compare against them on any machine, without the original installed.

A test computes its own result and hands it over together with a zero-argument callable that computes the original's:

    rec.bits(key, ours, lambda: ref.QuantizeTensor_LT(...))            bit-exact: sha256 of the bytes, 128 bits kept (dtype and shape included)
    rec.values(key, ours, lambda: ..., rtol=..., atol=...)            float tolerance: the original's values are stored

Check mode (the default): the callable is never called; `ours` is compared with the stored record tests/golden/<name>.json.
Record mode (PPQ_RECORD_GOLDEN=<dir>, with the original available): the callable runs, `ours` is compared with it live, and
<dir>/<name>.json is written when the test module finishes -- commit it under tests/golden/.  Inputs must come from seeded
generators so that both modes see the same tensors.
"""
import hashlib
import importlib.util
import json
import os

import numpy as np

TESTS = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(TESTS, 'golden')
REF_SO = os.path.join(os.path.dirname(TESTS), 'oracle', '_ref', 'PPQ_Cuda_Impls_ref.so')


def record_dir():
    return os.environ.get('PPQ_RECORD_GOLDEN') or None


def reference_extension():
    """The original's own CUDA extension (oracle/build_ref.py), loaded only to record; None in check mode."""
    if record_dir() is None:
        return None
    assert os.path.exists(REF_SO), f'recording needs {REF_SO} (python oracle/build_ref.py)'
    spec = importlib.util.spec_from_file_location('PPQ_Cuda_Impls_ref', REF_SO)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def plus_zero(t):
    """-0.0 as +0.0: for comparisons that, like torch.equal, do not tell the two apart."""
    return t.where(t != 0, t.new_zeros(()))


def _np(a):
    if hasattr(a, 'detach'):
        a = a.detach().contiguous().cpu().numpy()
    return np.ascontiguousarray(a)


def digest(a) -> str:
    a = _np(a)
    return f'{a.dtype.str}{list(a.shape)}:' + hashlib.sha256(a.tobytes()).hexdigest()[:32]


class Record:
    def __init__(self, name: str, recording: bool):
        self.name, self.recording = name, recording
        if recording:
            os.makedirs(record_dir(), exist_ok=True)
            self.data = {}
        else:
            with open(os.path.join(GOLDEN, name + '.json')) as f:
                self.data = json.load(f)

    def _want(self, key, make):
        if self.recording:
            assert key not in self.data, f'duplicate record key {key!r}'
            self.data[key] = make()
        assert key in self.data, f'{self.name}: no stored result for {key!r}'
        return self.data[key]

    def stored(self, key, original):
        """The original's JSON-able result itself (computed and stored when recording), for checks that need its values."""
        return self._want(key, original)

    def bits(self, key, ours, original):
        assert digest(ours) == self._want(key, lambda: digest(original())), (self.name, key)

    def values(self, key, ours, original, rtol, atol=0.0):
        want = self._want(key, lambda: _np(original()).astype(np.float64).reshape(-1).tolist())
        got = _np(ours).astype(np.float64).reshape(-1)
        np.testing.assert_allclose(got, np.asarray(want, np.float64), rtol=rtol, atol=atol, err_msg=f'{self.name}: {key}')

    def save(self):
        if self.recording:
            with open(os.path.join(record_dir(), self.name + '.json'), 'w') as f:
                json.dump(self.data, f, indent=0, sort_keys=True)
