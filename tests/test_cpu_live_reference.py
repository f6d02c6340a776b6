"""Pinning of the CPU oracle against the ORIGINAL PROJECT's own CPU / torch path (USING_CUDA_KERNEL = False) on inputs drawn at run time
from a fixed seed (unlike the fixtures of test_oracle_pinning.py, which store their inputs).  What the original returned for them is stored
in tests/golden/ref_cpu_live.json (tests/refrecord.py): recorded with PPQ_RECORD_GOLDEN set and the original package importable
(tests/refppq.py) -- PPQ_FUZZ_SEED then draws other inputs (a number, or `random`), which check the oracle live against the original.
CPU only."""
import os
import time

import numpy as np
import pytest
import torch

import refppq
import refrecord

DEFAULT_SEED = 20260923


@pytest.fixture(scope='module')
def ref():
    """The original package when recording, else None."""
    if refrecord.record_dir() is None:
        return None
    ppq = refppq.load()
    assert ppq is not None, 'recording needs the original package (tests/refppq.py)'
    from ppq.core import PPQ_CONFIG
    assert PPQ_CONFIG.USING_CUDA_KERNEL is False
    torch.set_num_threads(1)
    return ppq


@pytest.fixture(scope='module')
def seed(ref):
    env = os.environ.get('PPQ_FUZZ_SEED', str(DEFAULT_SEED)) if ref is not None else str(DEFAULT_SEED)
    s = time.time_ns() % (2 ** 31) if env == 'random' else int(env)
    print(f'PPQ_FUZZ_SEED={s}')
    return s


@pytest.fixture(scope='module')
def rec(ref, seed):
    r = refrecord.Record('ref_cpu_live', recording=ref is not None)
    yield r
    if seed == DEFAULT_SEED: r.save()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def activated(cfg, scale, offset):
    from ppq.core import QuantizationStates
    cfg.scale, cfg.offset, cfg.state = torch.as_tensor(scale, dtype=torch.float32), torch.as_tensor(offset, dtype=torch.float32), QuantizationStates.ACTIVATED
    return cfg


def linear_config(mode, **kw):
    """The original's LinearQuantizationConfig with rounding policy `mode` (a ppq_b200.RoundingPolicy, same names and values)."""
    from ppq.core import RoundingPolicy
    from ppq.lib import LinearQuantizationConfig
    return LinearQuantizationConfig(rounding=RoundingPolicy[mode.name], **kw)


def original_fake_quant(x, cfg):
    from ppq.quantization.qfunction.linear import PPQLinearQuantFunction
    return PPQLinearQuantFunction(torch.from_numpy(x), cfg).numpy()


def original_to_int(x, cfg):
    from ppq.quantization.qfunction.linear import PPQLinearQuant_toInt
    return PPQLinearQuant_toInt(torch.from_numpy(x), cfg).numpy().astype(np.int32)


def test_linear_fake_quant_per_tensor_and_per_channel(ref, rec, oracle, seed):
    from ppq_b200 import RoundingPolicy
    r = np.random.RandomState(seed)
    modes = [RoundingPolicy.ROUND_HALF_EVEN, RoundingPolicy.ROUND_HALF_UP, RoundingPolicy.ROUND_HALF_DOWN,
             RoundingPolicy.ROUND_HALF_TOWARDS_ZERO, RoundingPolicy.ROUND_HALF_FAR_FORM_ZERO]
    for it in range(24):
        shape = tuple(int(v) for v in r.randint(1, 9, size=r.randint(1, 5)))
        x = (r.standard_normal(shape) * 10 ** r.uniform(-2, 2)).astype(np.float32)
        x.reshape(-1)[:: 7] = np.round(x.reshape(-1)[:: 7] * 2) / 2                     # ties
        sym = bool(r.randint(2)); bits_ = int(r.choice([4, 8]))
        qmin, qmax = (-(1 << (bits_ - 1)), (1 << (bits_ - 1)) - 1) if sym else (0, (1 << bits_) - 1)
        mode = modes[it % len(modes)]
        # per tensor
        s = np.float32(10 ** r.uniform(-3, 0)); o = np.float32(0 if sym else r.randint(qmin, qmax + 1))
        cfg = lambda: activated(linear_config(mode, symmetrical=sym, quant_min=qmin, quant_max=qmax), s, o)   # noqa: E731
        got = oracle.linear_quant_t_torchpath(x, s, o, qmin, qmax, mode.value)
        rec.bits(f'{it} LT {shape} {mode.name}', bits(got), lambda: bits(original_fake_quant(x, cfg())))
        if mode == RoundingPolicy.ROUND_HALF_EVEN:
            got_dev, q_dev = oracle.linear_quant_t(x, s, o, qmin, qmax, 0, return_int=True)  # device semantics agree for integral offsets
            rec.bits(f'{it} LT device semantics', bits(got_dev), lambda: bits(original_fake_quant(x, cfg())))
            rec.bits(f'{it} toInt', q_dev, lambda: original_to_int(x, cfg()))
        # per channel
        if len(shape) >= 2:
            axis = int(r.randint(len(shape))); C = shape[axis]
            sc = (10 ** r.uniform(-3, 0, size=C)).astype(np.float32)
            oc = np.zeros(C, np.float32) if sym else r.randint(qmin, qmax + 1, size=C).astype(np.float32)
            cfgc = lambda: activated(linear_config(mode, symmetrical=sym, quant_min=qmin, quant_max=qmax, channel_axis=axis), sc, oc)   # noqa: E731
            gotc = oracle.linear_quant_c_torchpath(x, sc, oc, axis, qmin, qmax, mode.value)
            rec.bits(f'{it} LC {shape} axis {axis} {mode.name}', bits(gotc), lambda: bits(original_fake_quant(x, cfgc())))


def test_scalar_rounding_and_scale_offset(ref, rec, oracle, seed):
    from ppq_b200 import RoundingPolicy

    def original_round(values, mode):
        from ppq.core import RoundingPolicy as P
        from ppq.utils.round import ppq_numerical_round
        return [ppq_numerical_round(float(v), P[mode.name]) for v in values]

    def original_pow2(values, mode):
        from ppq.core import RoundingPolicy as P
        from ppq.utils.round import ppq_round_to_power_of_2
        return [ppq_round_to_power_of_2(float(v), P[mode.name]) for v in values]

    r = np.random.RandomState(seed + 1)
    for mode in (RoundingPolicy.ROUND_HALF_EVEN, RoundingPolicy.ROUND_HALF_UP, RoundingPolicy.ROUND_HALF_DOWN, RoundingPolicy.ROUND_HALF_TOWARDS_ZERO,
                 RoundingPolicy.ROUND_HALF_FAR_FORM_ZERO, RoundingPolicy.ROUND_TO_NEAR_INT, RoundingPolicy.ROUND_UP):
        vals = list(r.uniform(-50, 50, size=40)) + [k + 0.5 for k in range(-6, 6)] + [0.0, -0.0, 1e-9, -1e-9]
        rec.values(f'numerical_round {mode.name}', np.float64([oracle.numerical_round(float(v), mode.value) for v in vals]),
                   lambda: np.float64(original_round(vals, mode)), rtol=0)
    for mode in (RoundingPolicy.ROUND_HALF_UP, RoundingPolicy.ROUND_UP):
        vals = list(10 ** r.uniform(-8, 4, size=60)) + [1.0, 2.0, 0.5, 3.0, 0.75, 1.5]
        rec.values(f'round_to_power_of_2 {mode.name}', np.float64([oracle.round_to_power_of_2(float(v), mode.value) for v in vals]),
                   lambda: np.float64(original_pow2(vals, mode)), rtol=0)
    for it in range(200):
        lo = float(np.float32(r.uniform(-20, 5) * 10 ** r.uniform(-3, 1))); hi = float(np.float32(lo + abs(r.uniform(0, 30)) * 10 ** r.uniform(-3, 1)))
        if it % 17 == 0: lo, hi = 0.0, 0.0                                                # degenerate range -> min scale
        sym = bool(r.randint(2)); pow2 = bool(r.randint(2)); bits_ = int(r.choice([4, 8]))
        qmin, qmax = (-(1 << (bits_ - 1)), (1 << (bits_ - 1)) - 1) if sym else (0, (1 << bits_) - 1)

        def original():
            from ppq.lib import LinearQuantizationConfig
            from ppq.quantization.observer.range import minmax_to_scale_offset
            want = minmax_to_scale_offset(lo, hi, LinearQuantizationConfig(symmetrical=sym, quant_min=qmin, quant_max=qmax, power_of_2=pow2))
            return np.float64([float(want[0]), float(want[1])])
        got = oracle.minmax_to_scale_offset(lo, hi, qmin, qmax, sym, pow2)
        rec.values(f'minmax_to_scale_offset {it}', np.float64([float(got[0]), float(got[1])]), original, rtol=0)


def test_kl_and_mse_search_on_random_histograms(ref, rec, oracle, seed):
    r = np.random.RandomState(seed + 2)
    for it in range(6):
        bins = 4096
        kind = it % 3
        if kind == 0: hist = r.poisson(np.linspace(400, 0.01, bins) ** 1.2).astype(np.int64)
        elif kind == 1: hist = (r.poisson(3.0, size=bins) * (r.rand(bins) < 0.3)).astype(np.int64)       # sparse
        else:
            hist = np.zeros(bins, np.int64); hist[: 64] = r.randint(0, 10 ** 6, size=64); hist[r.randint(64, bins, 20)] = r.randint(1, 50, size=20)
        hs = float(10 ** r.uniform(-5, -1))
        for nbits in (8, 4):
            def original():
                from ppq.lib import LinearQuantizationConfig
                from ppq.quantization.observer.range import TorchHistObserver
                cfg = LinearQuantizationConfig(symmetrical=True, num_of_bits=nbits, quant_min=-(1 << (nbits - 1)), quant_max=(1 << (nbits - 1)) - 1, calibration='kl')
                ob = TorchHistObserver(watch_on=None, quant_cfg=cfg)
                want = ob.hist_to_scale_offset(histogram=torch.tensor(hist.astype(np.int32)), hist_bins=bins, hist_scale=hs, config=cfg)
                return np.float64([float(want[0]), float(want[1])])
            got = oracle.kl_search(hist, hs, nbits)
            rec.values(f'kl_search {it} bits {nbits}', np.float64([float(got[0]), float(got[1])]), original, rtol=0)
    for it in range(4):
        bins = 2048
        hist = r.poisson(np.linspace(200, 0.05, bins)).astype(np.int64)
        if it % 2: hist = hist[::-1].copy()
        for sym in (True, False):
            qmin, qmax = (-128, 127) if sym else (0, 255)
            vmin, vmax = -3.0, 5.0
            hs = (max(abs(vmin), abs(vmax)) if sym else (vmax - vmin)) / bins

            def original():
                from ppq.lib import LinearQuantizationConfig
                from ppq.quantization.observer.range import TorchMSEObserver
                cfg = LinearQuantizationConfig(symmetrical=sym, quant_min=qmin, quant_max=qmax, calibration='mse')
                ob = TorchMSEObserver(watch_on=None, quant_cfg=cfg)
                ob._min, ob._max = vmin, vmax
                want = ob.hist_to_scale_offset(histogram=torch.tensor(hist.astype(np.int32)), hist_bins=bins, hist_scale=hs, config=cfg)
                return np.float64([np.float32(want[0]), float(want[1])])
            got = oracle.mse_search(hist, hs, vmin, qmin, qmax, sym, loss_fn=oracle.mse_loss_python_twin)
            rec.values(f'mse_search {it} sym {sym}', np.float64([np.float32(got[0]), float(got[1])]), original, rtol=0)


def test_observers_end_to_end(ref, rec, oracle, seed):
    """ppq.lib.Observer (CPU path) on fresh data: min/max per tensor and per channel, percentile (kthvalue indices of the CPU branch), and the
    two-phase KL / MSE observers, whose histogram (torch.histc on the CPU branch) is fed to the oracle's search."""
    r = np.random.RandomState(seed + 3)
    for it, algo in enumerate(('minmax', 'percentile', 'kl', 'mse', 'minmax', 'mse')):
        sym = (it % 2 == 0) or algo == 'kl'
        relu = bool(r.randint(2))
        shape = (int(r.randint(1, 4)), int(r.randint(2, 9)), int(r.randint(5, 15)), int(r.randint(5, 15)))
        data = [(np.maximum(x, 0) if relu else x) for x in ((r.standard_normal(shape) * 10 ** r.uniform(-1, 1)).astype(np.float32) for _ in range(3))]
        qmin, qmax = (-128, 127) if sym else (0, 255)

        def original():
            """The observer's statistics and the config it renders: {min, max, hist, hist_scale} of phase 2 (KL / MSE), scale, offset."""
            from ppq.lib import LinearQuantizationConfig, Observer
            cfg = LinearQuantizationConfig(symmetrical=sym, quant_min=qmin, quant_max=qmax, calibration=algo)
            ob = Observer(cfg)
            for x in data: ob.observe(torch.from_numpy(x))
            ob.render_quantization_config()
            out = {}
            if algo in ('kl', 'mse'):
                for x in data: ob.observe(torch.from_numpy(x))
                out = {'min': float(ob._min), 'max': float(ob._max), 'hist': ob._hist.numpy().tolist(), 'hist_scale': float(ob._hist_scale)}
                ob.render_quantization_config()
            return dict(out, scale=float(cfg.scale.item()), offset=float(cfg.offset.item()))
        want = rec.stored(f'observer {it} {algo}', original)
        lo = min(float(oracle.minmax_t(x)[0]) for x in data); hi = max(float(oracle.minmax_t(x)[1]) for x in data)
        if algo in ('kl', 'mse'):
            hist, hs = np.asarray(want['hist']), want['hist_scale']
            assert (want['min'], want['max']) == (lo, hi), (seed, it)
            s, o = oracle.kl_search(hist, hs, 8) if algo == 'kl' else oracle.mse_search(hist, hs, lo, qmin, qmax, sym, loss_fn=oracle.mse_loss_python_twin)
        elif algo == 'percentile':
            pairs = []
            for x in data:
                v = np.sort(x.reshape(-1)); n = v.size
                pairs.append([v[min(int(n * 0.9999), n - 1)], v[max(0, int(n * (1 - 0.9999)))]])
            m = torch.tensor(np.array(pairs, np.float32)).mean(dim=0)
            s, o = oracle.minmax_to_scale_offset(m[1].item(), m[0].item(), qmin, qmax, sym)
        else:
            s, o = oracle.minmax_to_scale_offset(lo, hi, qmin, qmax, sym)
        assert (np.float32(s), np.float32(o)) == (np.float32(want['scale']), np.float32(want['offset'])), (seed, it, algo, sym, relu, shape)
    # per-channel symmetric min/max on a weight (ParameterQuantizePass path)
    for axis in (0, 1):
        w = (r.standard_normal((int(r.randint(2, 20)), int(r.randint(2, 20)), 3, 3)) * 0.1).astype(np.float32)

        def original():
            from ppq.lib import LinearQuantizationConfig, Observer
            cfg = LinearQuantizationConfig(symmetrical=True, channel_axis=axis, calibration='minmax')
            ob = Observer(cfg); ob.observe(torch.from_numpy(w)); ob.render_quantization_config()
            return np.concatenate([cfg.scale.numpy().reshape(-1), cfg.offset.numpy().reshape(-1)])
        lo, hi = oracle.minmax_c(w, axis)
        so = [oracle.minmax_to_scale_offset(float(a), float(b), -128, 127, True) for a, b in zip(lo, hi)]
        rec.bits(f'per-channel minmax axis {axis}', np.float32([s for s, _ in so] + [o for _, o in so]), original)
