"""Generate the golden fixtures in tests/golden/ by IMPORTING THE REAL REFERENCE (OpenPPL/ppq at
/root/reference, CPU / torch path, USING_CUDA_KERNEL = False) in the build container.

The reference is a Python package and cannot travel to the GPU box, so its outputs are committed
here as small fixtures; this script is the recipe that made them (SURVEY.md §8c, appendix C).

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz / *.json

Inputs are produced by numpy's legacy RandomState (bit-stable across numpy versions) so that large
cases (BASELINE config 1, 1x512x28x28) can be stored as seed + expected output instead of as data.
"""
import hashlib
import json
import os
import sys

os.environ['PROTOCOL_BUFFERS_PYTHON_IMPLEMENTATION'] = 'python'
from unittest.mock import MagicMock

for m in ['onnx', 'onnx.helper', 'onnx.numpy_helper', 'onnx.mapping', 'onnx.checker', 'onnx.shape_inference']:
    sys.modules.setdefault(m, MagicMock())
sys.path.insert(0, os.environ.get('PPQ_REFERENCE_ROOT', '/root/reference'))

import numpy as np
import torch

import ppq  # noqa: F401  (the real reference)
from ppq.core import PPQ_CONFIG, QuantizationStates, RoundingPolicy
from ppq.lib import LinearQuantizationConfig, Observer
from ppq.quantization.measure import torch_KL_divergence
from ppq.quantization.observer.range import TorchMSEObserver, minmax_to_scale_offset
from ppq.quantization.qfunction.linear import PPQLinearQuant_toInt, PPQLinearQuantFunction
from ppq.utils.round import ppq_numerical_round, ppq_round_to_power_of_2

assert PPQ_CONFIG.USING_CUDA_KERNEL is False
torch.set_num_threads(1)   # deterministic reductions
HERE = os.path.dirname(os.path.abspath(__file__))


def rs(seed):
    return np.random.RandomState(seed)


def activate(cfg, scale, offset):
    cfg.scale = torch.as_tensor(scale, dtype=torch.float32)
    cfg.offset = torch.as_tensor(offset, dtype=torch.float32)
    cfg.state = QuantizationStates.ACTIVATED
    return cfg


# ------------------------------------------------------------------------------------------------
# 1. per-tensor INT fake-quant: the reference test's distribution (tests/test_cuda_kernel.py:17-37)
#    x = rand*32, s = rand, o = 0 | randint(0,255), clip 0..255, plus INT8-sym / INT4 / randn cases.
# ------------------------------------------------------------------------------------------------
def gen_linear_t():
    out = {}
    cases = []
    shapes = [[1, 1, 1, 1], [5, 12, 13, 4], [1, 7, 15, 41], [12, 4, 15, 3], [50, 7, 13, 1], [3, 1, 10, 4]]
    k = 0
    for shape in shapes:
        for sym in (True, False):
            r = rs(1000 + k)
            x = (r.rand(*shape) * 32).astype(np.float32)
            s = np.float32(r.rand())
            o = np.float32(0.0 if sym else r.randint(0, 255))
            cfg = LinearQuantizationConfig(symmetrical=False, quant_min=0, quant_max=255)
            activate(cfg, s, o)
            y = PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()
            q = PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy()
            out[f'x{k}'], out[f'y{k}'], out[f'q{k}'] = x, y, q.astype(np.int32)
            cases.append(dict(k=k, scale=float(s), offset=float(o), qmin=0, qmax=255, mode=0))
            k += 1
    # signed INT8 / INT4, gaussian data, negative values, all torch-path rounding modes
    for (qmin, qmax) in ((-128, 127), (-8, 7)):
        for mode in (RoundingPolicy.ROUND_HALF_EVEN, RoundingPolicy.ROUND_HALF_UP, RoundingPolicy.ROUND_HALF_DOWN,
                     RoundingPolicy.ROUND_HALF_TOWARDS_ZERO, RoundingPolicy.ROUND_HALF_FAR_FORM_ZERO,
                     RoundingPolicy.ROUND_UP):
            r = rs(2000 + k)
            x = (r.standard_normal(size=(3, 5, 7, 11)) * 3).astype(np.float32)
            # sprinkle exact .5 ties (in units of the scale) so every rounding mode is exercised
            s = np.float32(0.125)
            x.reshape(-1)[::7] = (np.arange(x.size)[::7] % 41 - 20 + 0.5).astype(np.float32) * s
            cfg = LinearQuantizationConfig(symmetrical=True, quant_min=qmin, quant_max=qmax, rounding=mode)
            activate(cfg, s, 0.0)
            y = PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()
            q = PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy()
            out[f'x{k}'], out[f'y{k}'], out[f'q{k}'] = x, y, q.astype(np.int32)
            cases.append(dict(k=k, scale=float(s), offset=0.0, qmin=qmin, qmax=qmax, mode=mode.value))
            k += 1
    out['cases'] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'linear_t.npz'), **out)
    return len(cases)


# ------------------------------------------------------------------------------------------------
# 2. BASELINE config 1: LinearQuant_T INT8 per-tensor, 1x512x28x28, CPU path.  Stored as seed +
#    int8 quantised values + sha256 of the dequantised floats.
# ------------------------------------------------------------------------------------------------
def gen_config1():
    r = rs(20260922)
    x = r.standard_normal(size=(1, 512, 28, 28)).astype(np.float32)
    res = {}
    # (a) symmetric, scale from the reference's own minmax observer
    cfg = LinearQuantizationConfig(symmetrical=True, quant_min=-128, quant_max=127, calibration='minmax')
    ob = Observer(cfg)
    ob.observe(torch.from_numpy(x))
    ob.render_quantization_config()
    y = PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()
    q = PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy()
    res['sym_scale'] = np.float32(cfg.scale.item()); res['sym_offset'] = np.float32(cfg.offset.item())
    res['sym_q'] = q.astype(np.int8); res['sym_y_sha256'] = np.frombuffer(hashlib.sha256(y.tobytes()).digest(), np.uint8)
    # (b) asymmetric 0..255
    cfg = LinearQuantizationConfig(symmetrical=False, quant_min=0, quant_max=255, calibration='minmax')
    ob = Observer(cfg)
    ob.observe(torch.from_numpy(x))
    ob.render_quantization_config()
    y = PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()
    q = PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy()
    res['asym_scale'] = np.float32(cfg.scale.item()); res['asym_offset'] = np.float32(cfg.offset.item())
    res['asym_q'] = q.astype(np.uint8); res['asym_y_sha256'] = np.frombuffer(hashlib.sha256(y.tobytes()).digest(), np.uint8)
    res['seed'] = np.int64(20260922)
    np.savez_compressed(os.path.join(HERE, 'config1_lt_1x512x28x28.npz'), **res)


# ------------------------------------------------------------------------------------------------
# 3. per-channel INT fake-quant (tests/test_cuda_kernel.py:40-63; axes 1, 0, 3; epc 9 depth-wise)
# ------------------------------------------------------------------------------------------------
def gen_linear_c():
    out, cases, k = {}, [], 0
    specs = [([1, 1, 1, 1], 1), ([5, 12, 13, 4], 1), ([1, 7, 15, 41], 1), ([12, 4, 15, 3], 1),
             ([51, 7, 7, 1], 0), ([37, 1, 10, 4], 0), ([10, 10, 12, 47], 3), ([19, 4, 15, 3], 3),
             ([32, 1, 3, 3], 0), ([24, 96, 1, 1], 0), ([16], 0), ([7, 5], 1)]
    for shape, axis in specs:
        for sym in (True, False):
            r = rs(3000 + k)
            C = shape[axis]
            x = (r.rand(*shape) * 32).astype(np.float32)
            s = r.rand(C).astype(np.float32) + np.float32(1e-3)
            o = np.zeros(C, np.float32) if sym else r.randint(0, 255, size=C).astype(np.float32)
            cfg = LinearQuantizationConfig(symmetrical=False, quant_min=0, quant_max=255, channel_axis=axis)
            activate(cfg, s, o)
            y = PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()
            q = PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy()
            out[f'y{k}'], out[f'q{k}'], out[f's{k}'], out[f'o{k}'] = y, q.astype(np.int32), s, o      # x: regenerated from seed + shape
            cases.append(dict(k=k, axis=axis, qmin=0, qmax=255, mode=0, seed=3000 + k, shape=list(shape)))
            k += 1
    # signed weights, scales from the reference's per-channel minmax observer (BASELINE config 3 style)
    for shape in ([32, 3, 3, 3], [32, 1, 3, 3], [16, 32, 1, 1], [96, 1, 3, 3], [10, 64]):
        r = rs(3000 + k)
        w = (r.standard_normal(size=shape) * 0.1).astype(np.float32)
        cfg = LinearQuantizationConfig(symmetrical=True, quant_min=-128, quant_max=127, channel_axis=0, calibration='minmax')
        ob = Observer(cfg)
        ob.observe(torch.from_numpy(w))
        ob.render_quantization_config()
        y = PPQLinearQuantFunction(torch.from_numpy(w), cfg).numpy()
        q = PPQLinearQuant_toInt(torch.from_numpy(w), cfg).numpy()
        out[f'x{k}'], out[f'y{k}'], out[f'q{k}'] = w, y, q.astype(np.int32)
        out[f's{k}'], out[f'o{k}'] = cfg.scale.numpy().copy(), cfg.offset.numpy().copy()
        cases.append(dict(k=k, axis=0, qmin=-128, qmax=127, mode=0, observed=True))
        k += 1
    out['cases'] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'linear_c.npz'), **out)
    return len(cases)


# ------------------------------------------------------------------------------------------------
# 4. host scalar rounding + scale/offset KATs (tests/test_rounding.py; observer/range.py:22-75)
# ------------------------------------------------------------------------------------------------
def gen_scalar_kats():
    kat = {'numerical_round': [], 'pow2': [], 'minmax_to_scale_offset': []}
    vals = [1.5, 2.5, 0.5, -0.5, 1.1, 1.2, 1.3, -1.1, -1.2, -1.3, -1.5, -2.5, 3.5, 1e-9, -7.49999, 254.5, 255.5, 0.0]
    for p in RoundingPolicy:
        for v in vals:
            kat['numerical_round'].append([p.value, v, int(ppq_numerical_round(float(v), policy=p))])
    for v in [1.0, 1.2, 3.2, 0.26, 0.24, 0.5, 0.0078125, 1e-8, 17.0, 4.0, 0.75, 1.5, 3.0]:
        for p in (RoundingPolicy.ROUND_UP, RoundingPolicy.ROUND_HALF_UP, RoundingPolicy.ROUND_HALF_EVEN):
            kat['pow2'].append([p.value, v, ppq_round_to_power_of_2(float(v), policy=p)])
    r = rs(4000)
    for i in range(64):
        lo, hi = sorted((float(np.float32(r.standard_normal() * 4)), float(np.float32(r.standard_normal() * 4))))
        if i % 9 == 0: lo = 0.0
        if i % 13 == 0: hi = lo  # degenerate range
        if i % 11 == 0: lo, hi = float(np.float32(abs(lo) + 0.1)), float(np.float32(abs(lo) + abs(hi) + 0.2))   # strictly positive range (fp32-representable: the observers hand fp32 min/max to this function)
        for sym in (True, False):
            for pow2 in (False, True):
                for (qmin, qmax) in ((-128, 127), (0, 255), (-8, 7)):
                    cfg = LinearQuantizationConfig(symmetrical=sym, power_of_2=pow2, quant_min=qmin, quant_max=qmax)
                    s, o = minmax_to_scale_offset(lo, hi, cfg)
                    kat['minmax_to_scale_offset'].append([lo, hi, int(sym), int(pow2), qmin, qmax, float(s), float(o)])
    with open(os.path.join(HERE, 'scalar_kats.json'), 'w') as f:
        json.dump(kat, f)


# ------------------------------------------------------------------------------------------------
# 5. observers end-to-end on the CPU path (range.py): minmax (T, C), kl, mse, percentile
#    Data by seed; fixture = scales/offsets (+ histogram for kl/mse for bin-level diagnosis).
# ------------------------------------------------------------------------------------------------
def batches(seed, n, shape, relu):
    r = rs(seed)
    out = []
    for _ in range(n):
        x = r.standard_normal(size=shape).astype(np.float32)
        if relu: x = np.maximum(x, 0)
        out.append(x)
    return out


def gen_observers():
    res, cases = {}, []
    k = 0
    for algo in ('minmax', 'kl', 'mse', 'percentile'):
        for sym in (True, False):
            if algo == 'kl' and not sym: continue          # KL is symmetric-only upstream (range.py:219-220)
            for relu in (False, True):
                seed, n, shape = 5000 + k, 4, (2, 8, 14, 14)
                data = batches(seed, n, shape, relu)
                cfg = LinearQuantizationConfig(symmetrical=sym, quant_min=-128 if sym else 0,
                                               quant_max=127 if sym else 255, calibration=algo)
                ob = Observer(cfg)
                for x in data: ob.observe(torch.from_numpy(x))
                ob.render_quantization_config()
                if algo in ('kl', 'mse'):
                    for x in data: ob.observe(torch.from_numpy(x))
                    res[f'hist{k}'] = ob._hist.numpy().copy()
                    res[f'hist_scale{k}'] = np.float64(ob._hist_scale)
                    res[f'minmax{k}'] = np.array([ob._min, ob._max], np.float64)
                    ob.render_quantization_config()
                assert cfg.state == QuantizationStates.ACTIVATED
                res[f'scale{k}'] = cfg.scale.numpy().copy(); res[f'offset{k}'] = cfg.offset.numpy().copy()
                cases.append(dict(k=k, algo=algo, sym=sym, relu=relu, seed=seed, n=n, shape=shape))
                k += 1
    # per-channel symmetric minmax on a weight (ParameterQuantizePass path, parameters.py:172-215)
    for shape, axis in (((32, 3, 3, 3), 0), ((8, 24, 1, 1), 1)):
        seed = 5000 + k
        w = batches(seed, 1, shape, False)[0]
        cfg = LinearQuantizationConfig(symmetrical=True, channel_axis=axis, calibration='minmax')
        ob = Observer(cfg); ob.observe(torch.from_numpy(w)); ob.render_quantization_config()
        res[f'scale{k}'] = cfg.scale.numpy().copy(); res[f'offset{k}'] = cfg.offset.numpy().copy()
        cases.append(dict(k=k, algo='minmax', sym=True, relu=False, seed=seed, n=1, shape=shape, axis=axis))
        k += 1
    res['cases'] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'observers.npz'), **res)
    return k


# ------------------------------------------------------------------------------------------------
# 6. KL search + KL divergence + MSE search on synthetic histograms (range.py:190-282, 406-520)
# ------------------------------------------------------------------------------------------------
def gen_hist_search():
    res, cases, k = {}, [], 0
    for bits in (8, 4):
        for kind in ('gauss', 'relu', 'laplace', 'uniform', 'spike'):
            r = rs(6000 + k)
            n = 200000
            if kind == 'gauss': v = np.abs(r.standard_normal(n))
            elif kind == 'relu': v = np.maximum(r.standard_normal(n), 0)
            elif kind == 'laplace': v = np.abs(r.laplace(size=n))
            elif kind == 'uniform': v = r.rand(n)
            else: v = np.concatenate([np.abs(r.standard_normal(n - 10)) * 0.1, np.full(10, 50.0)])
            v = v.astype(np.float32)
            hist_scale = float(v.max()) / 4096
            hist = torch.histc(torch.from_numpy(v), 4096, min=0, max=hist_scale * 4096).int()
            cfg = LinearQuantizationConfig(symmetrical=True, quant_min=-(2 ** (bits - 1)), quant_max=2 ** (bits - 1) - 1,
                                           num_of_bits=bits, calibration='kl')
            ob = Observer(cfg)
            ob._hist_bins = 4096
            s, o = ob.hist_to_scale_offset(histogram=hist.clone(), hist_bins=4096, hist_scale=hist_scale, config=cfg)
            res[f'hist{k}'] = hist.numpy().copy()
            cases.append(dict(k=k, bits=bits, kind=kind, hist_scale=hist_scale, scale=float(s), offset=float(o)))
            k += 1
    # torch_KL_divergence KATs
    r = rs(6100)
    p = r.rand(6, 128).astype(np.float32); q = r.rand(6, 128).astype(np.float32)
    p /= p.sum(1, keepdims=True); q /= q.sum(1, keepdims=True)
    res['kl_p'], res['kl_q'] = p, q
    res['kl_val'] = np.array([torch_KL_divergence(torch.from_numpy(a), torch.from_numpy(b)) for a, b in zip(p, q)], np.float64)
    # MSE observer search (sym + asym) on 2048-bin histograms, python-twin loss (range.py:431-454)
    mse_cases = []
    for j, sym in enumerate((True, False, True, False)):
        r = rs(6200 + j)
        v = (r.standard_normal(50000) * (1 + j)).astype(np.float32)
        if j >= 2: v = np.maximum(v, 0)
        cfg = LinearQuantizationConfig(symmetrical=sym, quant_min=-128 if sym else 0, quant_max=127 if sym else 255,
                                       calibration='mse')
        ob = Observer(cfg)
        assert isinstance(ob, TorchMSEObserver)
        ob.observe(torch.from_numpy(v)); ob.render_quantization_config()
        ob.observe(torch.from_numpy(v))
        res[f'mse_hist{j}'] = ob._hist.numpy().copy()
        ob.render_quantization_config()
        mse_cases.append(dict(j=j, sym=sym, hist_scale=float(ob._hist_scale), vmin=float(ob._min), vmax=float(ob._max),
                              scale=float(cfg.scale.item()), offset=float(cfg.offset.item())))
    res['cases'] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    res['mse_cases'] = np.frombuffer(json.dumps(mse_cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, 'hist_search.npz'), **res)


# ------------------------------------------------------------------------------------------------
# 7. compute_mse_loss from the reference's own C++ (oracle/_ref/hist_mse_ref.so, compiled in place)
# ------------------------------------------------------------------------------------------------
def gen_mse_loss():
    import ctypes
    so = os.path.join(HERE, '..', '..', 'oracle', '_ref', 'hist_mse_ref.so')
    lib = ctypes.CDLL(so)
    lib.ref_compute_mse_loss.restype = ctypes.c_float
    lib.ref_compute_mse_loss.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    r = rs(7000)
    hists, args, vals = [], [], []
    for i in range(48):
        nb = [2048, 2048, 256, 64][i % 4]
        h = (r.gamma(0.7, 200.0, size=nb) * (r.rand(nb) > 0.2)).astype(np.int64)
        step = int(r.randint(1, max(2, nb // 256 + 2)))
        start = int(r.randint(0, 64)) if i % 3 else 0
        end = start + 256 * step if nb >= 256 else start + 16 * step
        hp = np.zeros(2048, np.int64); hp[:nb] = h
        hists.append(hp); args.append([nb, start, step, end])
        vals.append(lib.ref_compute_mse_loss(h.ctypes.data, nb, start, step, end))
    np.savez_compressed(os.path.join(HERE, 'mse_loss.npz'), hists=np.stack(hists), args=np.array(args, np.int64),
                        vals=np.array(vals, np.float32))


if __name__ == '__main__':
    print('linear_t cases', gen_linear_t())
    gen_config1()
    print('linear_c cases', gen_linear_c())
    gen_scalar_kats()
    print('observer cases', gen_observers())
    gen_hist_search()
    gen_mse_loss()
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))
