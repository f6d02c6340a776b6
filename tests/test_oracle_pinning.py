"""Pin the CPU oracle (oracle/) against the golden vectors produced by the REAL reference
(tests/golden/make_golden.py, CPU / torch path) and against the reference's own compiled hist_mse.cc.

CPU-only.  If these fail the oracle is wrong and no GPU parity claim means anything.
"""
import hashlib
import json
import os

import numpy as np

import refrecord
from conftest import GOLDEN, cases_of, golden_input, load_golden, seeded_batches


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_linear_t_matches_reference_cpu_path(oracle):
    g = load_golden('linear_t.npz')
    for c in cases_of(g):
        k = c['k']
        x, y_ref, q_ref = g[f'x{k}'], g[f'y{k}'], g[f'q{k}']
        # torch-path restatement: valid for every rounding mode the torch path implements
        y, q = oracle.linear_quant_t_torchpath(x, c['scale'], c['offset'], c['qmin'], c['qmax'], c['mode'], return_int=True)
        assert np.array_equal(bits(y), bits(y_ref)), c
        assert np.array_equal(q.astype(np.int32), q_ref), c
        # device-semantics restatement: must agree too (integral offsets, |x/s| small; the fp64 "+.5" modes
        # differ from the fp32 torch path only within 1 ulp of a tie -- not present in these vectors)
        y2, q2 = oracle.linear_quant_t(x, c['scale'], c['offset'], c['qmin'], c['qmax'], c['mode'], return_int=True)
        assert np.array_equal(q2, q_ref), c
        assert np.array_equal(bits(y2), bits(y_ref)), c


def test_config1_int8_bit_exact(oracle):
    """BASELINE config 1: LinearQuant_T INT8 per-tensor on 1x512x28x28, CPU path, bit-exact."""
    g = load_golden('config1_lt_1x512x28x28.npz')
    x = np.random.RandomState(int(g['seed'])).standard_normal(size=(1, 512, 28, 28)).astype(np.float32)
    for tag, lo, hi, dt in (('sym', -128, 127, np.int8), ('asym', 0, 255, np.uint8)):
        y, q = oracle.linear_quant_t(x, g[f'{tag}_scale'], g[f'{tag}_offset'], lo, hi, 0, return_int=True)
        assert np.array_equal(q.astype(dt), g[f'{tag}_q'])
        assert hashlib.sha256(y.tobytes()).digest() == bytes(g[f'{tag}_y_sha256'])


def test_linear_c_matches_reference_cpu_path(oracle):
    g = load_golden('linear_c.npz')
    for c in cases_of(g):
        k = c['k']
        x, y_ref, q_ref, s, o = golden_input(g, c), g[f'y{k}'], g[f'q{k}'], g[f's{k}'], g[f'o{k}']
        y, q = oracle.linear_quant_c(x, s, o, c['axis'], c['qmin'], c['qmax'], c['mode'], return_int=True)
        assert np.array_equal(q, q_ref), c
        assert np.array_equal(bits(y), bits(y_ref)), c
        y2 = oracle.linear_quant_c_torchpath(x, s, o, c['axis'], c['qmin'], c['qmax'], c['mode'])
        assert np.array_equal(bits(y2), bits(y_ref)), c


def test_scalar_rounding_and_scale_offset_kats(oracle):
    kat = json.load(open(os.path.join(GOLDEN, 'scalar_kats.json')))
    for mode, v, want in kat['numerical_round']:
        assert oracle.numerical_round(v, mode) == want, (mode, v)
    for mode, v, want in kat['pow2']:
        assert oracle.round_to_power_of_2(v, mode) == want, (mode, v)
    for lo, hi, sym, pow2, qmin, qmax, s, o in kat['minmax_to_scale_offset']:
        got = oracle.minmax_to_scale_offset(lo, hi, qmin, qmax, bool(sym), bool(pow2))
        assert got[0] == s and got[1] == o, (lo, hi, sym, pow2, qmin, qmax)


def test_reference_rounding_known_answers(oracle):
    """tests/test_rounding.py:5-36 of the reference, verbatim expectations."""
    r = oracle.numerical_round
    assert [r(v, 0) for v in (1.5, 2.5, 0.5, -0.5, 1.1, -1.3)] == [2, 2, 0, 0, 1, -1]
    assert [r(v, 1) for v in (1.5, 2.5, 0.5, -0.5)] == [2, 3, 1, 0]
    assert [r(v, 2) for v in (1.5, 2.5, 0.5, -0.5)] == [1, 2, 0, -1]
    assert [r(v, 3) for v in (1.5, 2.5, 0.5)] == [1, 2, 0]
    p = oracle.round_to_power_of_2
    assert (p(1.0), p(1.2), p(3.2), p(0.26), p(0.24)) == (1, 2, 4, 0.5, 0.25)


def test_device_round2int_modes(oracle):
    r = oracle.round2int
    assert [r(v, 0) for v in (0.5, 1.5, 2.5, -0.5, -1.5, 3e9, -3e9, float('nan'))] == [0, 2, 2, 0, -2, 2**31 - 1, -2**31, 0]
    assert [r(v, 1) for v in (0.5, 1.5, -0.5, -1.5)] == [1, 2, 0, -1]
    assert [r(v, 2) for v in (0.5, 1.5, -0.5, -1.5)] == [0, 1, -1, -2]
    assert [r(v, 3) for v in (0.5, 1.5, -0.5, -1.5)] == [0, 1, 0, -1]
    assert [r(v, 4) for v in (0.5, 1.5, -0.5, -1.5)] == [1, 2, -1, -2]
    assert [r(v, 5) for v in (0.5, 1.5, -0.5, -1.5, 2.4)] == [1, 2, -1, -2, 2]
    assert [r(v, 6) for v in (0.1, -0.1, 1.0)] == [1, 0, 1]
    assert [r(v, 7) for v in (0.9, -0.1, 1.0)] == [0, -1, 1]
    # the "+ .5" is done in fp64 on the device: 0.49999997f + .5 < 1 there (fp32 would give 1.0)
    assert r(np.float32(0.49999997), 1) == 0


def test_observers_match_reference(oracle):
    g = load_golden('observers.npz')
    for c in cases_of(g):
        k, algo, sym = c['k'], c['algo'], c['sym']
        data = seeded_batches(c['seed'], c['n'], tuple(c['shape']), c['relu'])
        qmin, qmax = (-128, 127) if sym else (0, 255)
        want_s, want_o = g[f'scale{k}'], g[f'offset{k}']
        if 'axis' in c:
            lo, hi = oracle.minmax_c(data[0], c['axis'])
            so = [oracle.minmax_to_scale_offset(float(a), float(b), qmin, qmax, True) for a, b in zip(lo, hi)]
            assert np.array_equal(np.float32([s for s, _ in so]), want_s)
            assert np.array_equal(np.float32([o for _, o in so]), want_o)
            continue
        mm = [oracle.minmax_t(x) for x in data]
        lo, hi = min(m[0] for m in mm), max(m[1] for m in mm)
        if algo == 'minmax':
            s, o = oracle.minmax_to_scale_offset(float(lo), float(hi), qmin, qmax, sym)
        elif algo == 'percentile':
            # CPU branch upstream uses kthvalue with int() truncation (range.py:341-346): restated inline
            pairs = []
            for x in data:
                v = np.sort(x.reshape(-1)); n = v.size
                lo_i = max(0, int(n * (1 - 0.9999))); hi_i = min(int(n * 0.9999), n - 1)
                pairs.append([v[hi_i], v[lo_i]])
            import torch
            m = torch.tensor(np.array(pairs, np.float32)).mean(dim=0)
            s, o = oracle.minmax_to_scale_offset(m[1].item(), m[0].item(), qmin, qmax, sym)
        else:
            # two-phase hist observers.  The reference CPU branch collects with torch.histc, so feed the search
            # with the fixture's histogram (the search is what is pinned here); the device-semantics histogram
            # is compared to it separately below.
            hist = g[f'hist{k}']; hs = float(g[f'hist_scale{k}']); vmin, vmax = g[f'minmax{k}']
            assert float(lo) == vmin and float(hi) == vmax
            want_hs = (max(abs(vmin), abs(vmax)) if sym else (vmax - vmin)) / (4096 if algo == 'kl' else 2048)
            assert hs == want_hs
            if algo == 'kl':
                s, o = oracle.kl_search(hist, hs, 8)
            else:
                s, o = oracle.mse_search(hist, hs, vmin, qmin, qmax, sym, loss_fn=oracle.mse_loss_python_twin)
        assert np.float32(s) == want_s and np.float32(o) == want_o, c


def test_device_histogram_close_to_histc(oracle):
    """Same bar as the reference's own test (tests/test_cuda_kernel.py:197-208): |device hist - histc| < 100."""
    g = load_golden('observers.npz')
    for c in cases_of(g):
        if c['algo'] not in ('kl', 'mse') or 'axis' in c: continue
        k = c['k']
        data = seeded_batches(c['seed'], c['n'], tuple(c['shape']), c['relu'])
        ref = g[f'hist{k}']; hs = np.float32(g[f'hist_scale{k}']); vmin, vmax = g[f'minmax{k}']
        h = np.zeros_like(ref)
        for x in data:
            if c['sym']: oracle.histogram_t(x, hs, hist=h)
            else: oracle.histogram_asym_t(x, vmin, vmax, hist=h)
        assert np.abs(h.astype(np.int64) - ref).max() < 100
        assert abs(int(h.sum()) - int(ref.sum())) <= 8     # only the x == max samples are dropped


def test_kl_search_and_divergence(oracle):
    g = load_golden('hist_search.npz')
    for c in cases_of(g):
        s, o = oracle.kl_search(g[f"hist{c['k']}"], c['hist_scale'], c['bits'])
        assert s == c['scale'] and o == c['offset'], c
    for p, q, want in zip(g['kl_p'], g['kl_q'], g['kl_val']):
        assert oracle.kl_divergence(p, q) == want


def test_mse_search(oracle):
    g = load_golden('hist_search.npz')
    for c in cases_of(g, 'mse_cases'):
        sym = c['sym']
        qmin, qmax = (-128, 127) if sym else (0, 255)
        s, o = oracle.mse_search(g[f"mse_hist{c['j']}"], c['hist_scale'], c['vmin'], qmin, qmax, sym,
                                 loss_fn=oracle.mse_loss_python_twin)
        assert np.float32(s) == np.float32(c['scale']) and float(o) == c['offset'], c


def test_compute_mse_loss_vs_reference_cpp(oracle):
    g = load_golden('mse_loss.npz')
    for h, (nb, start, step, end), want in zip(g['hists'], g['args'], g['vals']):
        got = oracle.compute_mse_loss(h[:nb], start, step, end)
        assert np.float32(got) == want, (nb, start, step, end)


def test_compute_mse_loss_vs_live_reference_build(oracle):
    """200 seeded cases against the reference's hist_mse.cc compiled in place (oracle/_ref/hist_mse_ref.so); its results are stored in
    tests/golden/ref_hist_mse.json (tests/refrecord.py: recorded with PPQ_RECORD_GOLDEN set and oracle/_ref built)."""
    import ctypes
    recording = refrecord.record_dir() is not None
    if recording:
        lib = ctypes.CDLL(os.path.join(os.path.dirname(GOLDEN), '..', 'oracle', '_ref', 'hist_mse_ref.so'))
        lib.ref_compute_mse_loss.restype = ctypes.c_float
        lib.ref_compute_mse_loss.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    rec = refrecord.Record('ref_hist_mse', recording=recording)
    r = np.random.RandomState(99)
    for i in range(200):
        nb = int(r.choice([16, 100, 2048]))
        h = r.randint(0, 5000, size=nb).astype(np.int64)
        step = int(r.randint(1, 9)); start = int(r.randint(0, nb // 2)); end = start + int(r.randint(1, 300)) * step
        rec.values(f'{i} bins {nb} start {start} step {step} end {end}', np.float32(oracle.compute_mse_loss(h, start, step, end)),
                   lambda: np.float32(lib.ref_compute_mse_loss(h.ctypes.data, nb, start, step, end)), rtol=0)
    rec.save()


def test_fp8_restatement_sanity(oracle):
    """FP8 has no CPU path upstream (parity is pinned on the GPU box against the reference's CUDA kernel).
    Here: the documented known answers from SURVEY.md appendix A (tie rule, saturation, subnormal grid) and
    agreement with torch.float8_e4m3fn away from ties."""
    import torch
    f = oracle.float_quant_scalar
    assert [f(v) for v in (1.1875, 1.4375, 2.375, 19.0, -1.1875)] == [1.125, 1.375, 2.25, 18.0, -1.125]   # ties toward zero
    assert f(464.0) == 448.0 and f(-1e9) == -448.0 and f(float('inf')) == 448.0
    assert f(1.5 * 2**-9) == 2 * 2**-9 and f(2.5 * 2**-9) == 2 * 2**-9 and f(2**-10) == 0.0
    # the subnormal branch goes through an int (round2int(...) * min_subnormal): the sign of zero is lost
    assert not np.signbit(np.float32(f(-0.0))) and not np.signbit(np.float32(f(-2**-11)))
    x = (np.random.RandomState(3).standard_normal(200000) * 10).astype(np.float32)
    y = oracle.float_quant_t(x, 1.0)
    t = torch.from_numpy(x).to(torch.float8_e4m3fn).float().numpy()
    assert np.array_equal(y, t)
    # E5M2 grid: 57344 max, clip given explicitly
    assert f(70000.0, 1.0, 5, 2, -57344.0, 57344.0) == 57344.0
    assert f(1.3, 1.0, 5, 2, -57344.0, 57344.0) == 1.25


def test_quantile_indices(oracle):
    x = np.arange(10000, dtype=np.float32)[::-1].copy()
    out = oracle.quantile_t(x, 0.9999)
    assert out[0] == 9999.0 and out[1] == 1.0
    assert np.array_equal(oracle.quantile_t(np.float32([3.0]), 0.9999), np.float32([3.0, 3.0]))


def test_fp8_and_histogram_vs_reference_cuda_kernels(oracle):
    """Vectors produced ON THE B200 BY THE REFERENCE'S OWN CUDA KERNELS (oracle/_ref/PPQ_Cuda_Impls_ref.so; written by
    tests/test_gpu_vs_reference_cuda.py, committed under tests/golden/ref_cuda_*.npz): this pins the C restatement of the paths that have
    no CPU implementation upstream -- QuantizeTensor_FT (all tie / subnormal / saturation / special-value cases, two rounding modes,
    four formats) and Histogram_T."""
    import re
    g = load_golden('ref_cuda_fp8.npz')
    x = g['x']
    n = 0
    for key in g.files:
        m = re.fullmatch(r'y_E(\d)M(\d)_c(\d+)_s([\d.]+)_o([\d.]+)_m(\d)', key)
        if not m: continue
        E, M, c, s, o, mode = int(m[1]), int(m[2]), float(m[3]), float(m[4]), float(m[5]), int(m[6])
        y = oracle.float_quant_t(x, s, o, E, M, -c, c, mode)
        assert np.array_equal(y.view(np.uint32), g[key].view(np.uint32)), key
        n += 1
    assert n >= 8
    h = load_golden('ref_cuda_hist.npz')
    got = oracle.histogram_t(h['x'], h['hist_scale'], 4096, True)
    assert np.array_equal(got, h['hist'])
