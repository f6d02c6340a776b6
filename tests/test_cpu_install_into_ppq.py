"""Drop-in check of ppq_b200.install against the ORIGINAL PROJECT's package, from what was recorded of it in tests/golden/ref_install.json
(tests/refrecord.py: recorded with PPQ_RECORD_GOLDEN set and the original importable, tests/refppq.py):
  * `calls`: which extension function each of its ppq.core.ffi.CUDA wrappers calls, with which arguments in which order (it re-orders some
    between Python and C++) -- logged by serving its ffi from a stand-in extension;
  * `observers`: the classes its observer table holds by key, and the module attributes its calibration passes compare `type(observer)` with.
install() / uninstall() then run against a stand-in `ppq` module tree of that shape (ffi served by a ComplieHelper), and every recorded call
must reach ppq_b200/_C.so through ppq_b200.ffi.CUDA -- no GPU here, so each must fail with OUR loud CPU-tensor error."""
import contextlib
import sys
import types

import pytest
import torch

import refppq
import refrecord

X, S, O = torch.zeros(2, 3, 4, 4), torch.ones(3), torch.zeros(3)
CALLS = [                                                  # (wrapper of ffi.CUDA, its arguments)
    ('LinearQuantize_T', (X, S[:1], O[:1], -128, 127, 0)),
    ('LinearQuantize_C', (X, S, O, 1, -128, 127, 0)),
    ('LinearQuantize_T_B', (X, S[:1], O[:1], X, -128, 127, 0)),
    ('LinearQuantize_C_B', (X, S, O, X, -128, 127, 1, 0)),
    ('Histogram_T', (X, torch.zeros(8, dtype=torch.int32), 0.1)),
    ('Histogram_Asymmetric_T', (-1.0, 1.0, X, torch.zeros(8, dtype=torch.int32))),
    ('Histogram_C', (X, 1, torch.zeros(3, 8, dtype=torch.int32), 0.1)),
    ('Quantile', (X, 0.9999)),
    ('TensorClip_T', (X, X, S[:1])),
    ('TensorClip_C', (X, X, S, 1)),
    ('RoundingLoss_LT', (X, S[:1], O[:1], -128, 127, 0)),
    ('RoundingLoss_LT_B', (X, S[:1], S[:1], O[:1], -128, 127, 0)),
    ('RoundingLoss_LC', (X, S, O, 1, -128, 127, 0)),
    ('RoundingLoss_LC_B', (X, S[:1], S, O, 1, -128, 127, 0)),
    ('FloatingQuantize_T', (X, S[:1], O[:1], 4, 3, -448.0, 448.0, 0)),
    ('FloatingQuantize_C', (X, S, O, 1, 4, 3, -448.0, 448.0, 0)),
    ('FloatingQuantize_T_B', (X, S[:1], O[:1], X, 4, 3, -448.0, 448.0, 0)),
    ('FloatingQuantize_C_B', (X, S, O, X, 4, 3, -448.0, 448.0, 1, 0)),
    ('compute_mse_loss', ([1, 2, 3, 4], 0, 1, 2)),
]
INPUTS = {'X': X, 'S': S, 'O': O}


def describe(v):
    """An argument as JSON: tensors by shape and dtype (and by name when they are one of this module's inputs or a view of one)."""
    if isinstance(v, torch.Tensor):
        name = next((k for k, t in INPUTS.items() if v.data_ptr() == t.data_ptr()), None)
        return {'tensor': list(v.shape), 'dtype': str(v.dtype), 'input': name}
    if isinstance(v, (list, tuple)):
        return [describe(a) for a in v]
    return v


def rebuild(d):
    if isinstance(d, dict):
        t = INPUTS[d['input']] if d['input'] else torch.zeros(d['tensor'], dtype=getattr(torch, d['dtype'].split('.')[-1]))
        return t[:d['tensor'][0]] if d['input'] and list(t.shape) != d['tensor'] else t
    if isinstance(d, list):
        return [rebuild(a) for a in d]
    return d


class CallLog:
    """Stand-in extension: logs [function, described arguments] of every call, returns 0.0."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append([name, describe(list(args))])
            return 0.0
        return fn


def calls_of(cuda, serve):
    """The extension calls the wrappers of `cuda` make, one list per entry of CALLS; `serve(log)` makes `log` the extension they reach."""
    out = []
    for wrapper, args in CALLS:
        log = CallLog()
        with serve(log):
            getattr(cuda, wrapper)(*args)
        out.append(log.calls)
    return out


OBSERVER_MODULES = ('ppq.quantization.optim.calibration', 'ppq.quantization.optim.ssd')
OBSERVER_ATTRS = ('TorchHistObserver', 'TorchMSEObserver', 'TorchMinMaxObserver')


def original_shape():
    """Recorded facts about the original package (computed from it when recording)."""
    def calls():
        assert refppq.load() is not None, 'recording needs the original package (tests/refppq.py)'
        import ppq.core.ffi as ffi
        return calls_of(ffi.CUDA, refppq.use_extension)

    def observers():
        import importlib
        assert refppq.load() is not None, 'recording needs the original package (tests/refppq.py)'
        import ppq.quantization.observer as obs
        sites = {m: {a: getattr(importlib.import_module(m), a).__name__ for a in OBSERVER_ATTRS if hasattr(importlib.import_module(m), a)}
                 for m in OBSERVER_MODULES}
        return {'table': {k: v.__name__ for k, v in obs.OBSERVER_TABLE.items()}, 'sites': sites}

    rec = refrecord.Record('ref_install', recording=refrecord.record_dir() is not None)
    shape = {'calls': rec.stored('calls', calls), 'observers': rec.stored('observers', observers)}
    rec.save()
    return shape


@pytest.fixture
def ppq():
    """A stand-in `ppq` module tree with the recorded shape, in sys.modules for the duration of one test."""
    import ppq_b200.ffi as ours
    shape = original_shape()
    classes = {}

    def cls(name):
        return classes.setdefault(name, type(name, (), {'__init__': lambda self, **kw: None}))
    mods = {n: types.ModuleType(n) for n in ('ppq', 'ppq.core', 'ppq.core.ffi', 'ppq.quantization', 'ppq.quantization.observer',
                                              'ppq.quantization.optim') + OBSERVER_MODULES}
    mods['ppq.core.ffi'].CUDA_COMPLIER = type('ComplieHelper', (ours.ComplieHelper,), {})()
    mods['ppq.quantization.observer'].OBSERVER_TABLE = {k: cls(v) for k, v in shape['observers']['table'].items()}
    for m, attrs in shape['observers']['sites'].items():
        for a, name in attrs.items(): setattr(mods[m], a, cls(name))
    for n, m in mods.items():
        if '.' in n: setattr(mods[n.rsplit('.', 1)[0]], n.rsplit('.', 1)[1], m)
    saved = {n: sys.modules.get(n) for n in mods}
    sys.modules.update(mods)
    try:
        yield types.SimpleNamespace(modules=mods, shape=shape)
    finally:
        for n, m in saved.items():
            if m is None: sys.modules.pop(n, None)
            else: sys.modules[n] = m


@contextlib.contextmanager
def serve_ours(log):
    import ppq_b200.ffi as ours
    saved = ours.CUDA_COMPLIER.__CUDA_EXTENTION__
    ours.CUDA_COMPLIER.__CUDA_EXTENTION__ = log
    try: yield
    finally: ours.CUDA_COMPLIER.__CUDA_EXTENTION__ = saved


def test_install_routes_every_ffi_call_to_our_extension(ppq):
    import ppq_b200.install
    from ppq_b200.ffi import CUDA
    ffi = ppq.modules['ppq.core.ffi']
    helper_type = type(ffi.CUDA_COMPLIER)
    original_complie = helper_type.complie
    ext = ppq_b200.install.install(replace_observers=False)
    try:
        assert ffi.CUDA_COMPLIER.CUDA_EXTENSION is ext
        assert ffi.CUDA_COMPLIER.complie() is None and ffi.CUDA_COMPLIER.CUDA_EXTENSION is ext     # complie() no longer builds or loads
    finally:
        ppq_b200.install.uninstall()
    assert helper_type.complie is original_complie and ffi.CUDA_COMPLIER.__CUDA_EXTENTION__ is not ext
    want = ppq.shape['calls']
    assert calls_of(CUDA, serve_ours) == want                                   # our wrappers make the original's extension calls
    for (wrapper, _), calls in zip(CALLS, want):
        assert len(calls) == 1, wrapper
        name, args = calls[0]
        if name == 'compute_mse_loss':
            assert isinstance(getattr(ext, name)(*rebuild(args)), float)
            continue
        with pytest.raises(RuntimeError, match='not on a CUDA device'):       # argument counts / types bind (no TypeError), then our device check fires
            getattr(ext, name)(*rebuild(args))


def test_observer_table_replaced(ppq):
    import ppq_b200.install
    import ppq_b200.observer as ours
    ref_obs, ref_cal, ref_ssd = (ppq.modules[n] for n in ('ppq.quantization.observer',) + OBSERVER_MODULES)
    before = dict(ref_obs.OBSERVER_TABLE)
    ref_hist, ref_mse = ref_cal.TorchHistObserver, ref_cal.TorchMSEObserver
    ppq_b200.install.install(replace_observers=True)
    try:
        for k in ('minmax', 'kl', 'mse', 'percentile'):
            assert ref_obs.OBSERVER_TABLE[k] is ours.OBSERVER_TABLE[k]
        # the original keeps an observer for calibration phase 2 only if `type(observer) in {TorchHistObserver, TorchMSEObserver}` as
        # imported by optim/calibration.py:10-13 (:195) and optim/ssd.py:14 (:445): the replaced classes must satisfy that test
        cfg = ppq_b200.LinearQuantizationConfig(calibration='kl')
        assert type(ref_obs.OBSERVER_TABLE['kl'](watch_on=None, quant_cfg=cfg)) in {ref_cal.TorchHistObserver, ref_cal.TorchMSEObserver}
        assert type(ref_obs.OBSERVER_TABLE['mse'](watch_on=None, quant_cfg=cfg)) in {ref_cal.TorchHistObserver, ref_cal.TorchMSEObserver}
        assert type(ref_obs.OBSERVER_TABLE['kl'](watch_on=None, quant_cfg=cfg)) in {ref_ssd.TorchHistObserver}
        assert type(ref_obs.OBSERVER_TABLE['minmax'](watch_on=None, quant_cfg=cfg)) not in {ref_cal.TorchHistObserver, ref_cal.TorchMSEObserver}
    finally:
        ppq_b200.install.uninstall()
    assert ref_obs.OBSERVER_TABLE == before
    assert ref_cal.TorchHistObserver is ref_hist and ref_cal.TorchMSEObserver is ref_mse and ref_ssd.TorchHistObserver is ref_hist
