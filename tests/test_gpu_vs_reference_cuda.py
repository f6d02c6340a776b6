"""GPU parity against the ORIGINAL PROJECT'S OWN CUDA KERNELS (ppq/csrc compiled unmodified for sm_100a by oracle/build_ref.py into
oracle/_ref/PPQ_Cuda_Impls_ref.so).  This is what pins the paths that have no CPU implementation and no test upstream: FP8
(QuantizeTensor_FT/_FC), Histogram_T / _Asymmetric_T / _C, non-default rounding modes on the device.  Bit-exact everywhere.
The original's outputs for these seeded inputs are stored in tests/golden/ref_cuda_kernels.json (tests/refrecord.py: recorded on a
B200 with PPQ_RECORD_GOLDEN set and oracle/_ref built; checked against that record otherwise).  Recording also writes the original
kernels' FP8 and histogram vectors that pin the CPU oracle (tests/golden/ref_cuda_fp8.npz, ref_cuda_hist.npz).
"""
import os

import numpy as np
import pytest
import torch

import refrecord

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ref():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return refrecord.reference_extension()


@pytest.fixture(scope='module')
def rec(ref):
    r = refrecord.Record('ref_cuda_kernels', recording=ref is not None)
    yield r
    r.save()


@pytest.fixture(scope='module')
def ext():
    from ppq_b200.ffi import extension
    return extension()


def t1(v):
    return torch.tensor([v], dtype=torch.float32, device='cuda')


def fp_inputs(n, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.randn(n, device='cuda', generator=g) * 10
    x[::3] = x[::3].half().float()
    x[1::11] = torch.randn(x[1::11].numel(), device='cuda', generator=g) * 2 ** -8
    x[2::13] = torch.randn(x[2::13].numel(), device='cuda', generator=g) * 300
    sp = torch.tensor([0.0, -0.0, float('inf'), float('-inf'), 1e-45, 464.0, 480.0, 448.0, 1.1875, 1.4375, 2.375, 19.0, -1.1875,
                       1.5 * 2 ** -9, 2.5 * 2 ** -9, 2 ** -10, -2 ** -11, 2 ** -6, 3e38, -3e38], device='cuda')
    x[:sp.numel()] = sp
    return x


def test_linear_t_c_vs_reference_kernels(ref, ext, rec):
    g = torch.Generator(device='cuda').manual_seed(1)
    for shape, axis in (([1, 1, 1, 1], 1), ([5, 12, 13, 4], 1), ([50, 120, 130, 4], 1), ([12, 74, 15, 411], 1), ([5011, 7, 7, 1], 0),
                        ([10, 10, 124, 47], 3), ([32, 1, 3, 3], 0), ([2048, 512, 3, 3], 0), ([1, 512, 28, 28], 1)):
        x = torch.rand(shape, device='cuda', generator=g) * 32 - 8
        s, o = torch.rand(1, device='cuda', generator=g) + 1e-3, torch.randint(0, 255, (1,), device='cuda', generator=g).float()
        for mode in range(8):
            for lo, hi in ((0, 255), (-128, 127), (-8, 7)):
                rec.bits(f'LT {shape} mode {mode} [{lo}, {hi}]', ext.QuantizeTensor_LT(x, s, o, lo, hi, mode),
                         lambda: ref.QuantizeTensor_LT(x, s, o, lo, hi, mode))
        C = shape[axis]
        sc, oc = torch.rand(C, device='cuda', generator=g) + 1e-3, torch.randint(0, 255, (C,), device='cuda', generator=g).float()
        for mode in (0, 2, 5):
            rec.bits(f'LC {shape} axis {axis} mode {mode}', ext.QuantizeTensor_LC(x, sc, oc, 0, 255, axis, mode),
                     lambda: ref.QuantizeTensor_LC(x, sc, oc, 0, 255, axis, mode))


def test_fp8_vs_reference_kernels_and_emit_golden(ref, ext, rec):
    """The FP8 pin: ours == the reference's QuantizeTensor_FT/_FC, bit for bit, including exact ties, the subnormal grid,
    saturation, signed zeros and infinities."""
    x = fp_inputs(1 << 20, 7)
    for (E, M, cmin, cmax) in ((4, 3, -448.0, 448.0), (5, 2, -57344.0, 57344.0), (4, 3, -240.0, 240.0), (3, 4, -30.0, 30.0)):
        for s, o in ((1.0, 0.0), (0.125, 0.0), (4.0, 0.0), (0.0078125, 0.0), (0.3, 2.5)):
            for mode in (0, 1, 2, 3, 4, 5, 6, 7):
                rec.bits(f'FT E{E}M{M} [{cmin}, {cmax}] s {s} o {o} mode {mode}', ext.QuantizeTensor_FT(x, t1(s), t1(o), E, M, cmin, cmax, mode),
                         lambda: ref.QuantizeTensor_FT(x, t1(s), t1(o), E, M, cmin, cmax, mode))
    if rec.recording:
        n = 16384                                                        # the first n elements: specials, ties, subnormals and bulk
        out = {'x': x[:n].cpu().numpy()}
        for (E, M, cmin, cmax) in ((4, 3, -448.0, 448.0), (5, 2, -57344.0, 57344.0), (4, 3, -240.0, 240.0), (3, 4, -30.0, 30.0)):
            for s, o in ((1.0, 0.0), (0.3, 2.5)):
                for mode in (0, 1):
                    out[f'y_E{E}M{M}_c{int(cmax)}_s{s}_o{o}_m{mode}'] = ref.QuantizeTensor_FT(x, t1(s), t1(o), E, M, cmin, cmax, mode)[:n].cpu().numpy()
        np.savez_compressed(os.path.join(refrecord.record_dir(), 'ref_cuda_fp8.npz'), **out)
    xs = x[:64 * 27 * 16].view(64, 27, 16)
    g = torch.Generator(device='cuda').manual_seed(8)
    for axis in (0, 1, 2):
        C = xs.shape[axis]
        sc = 2.0 ** torch.randint(-7, 6, (C,), device='cuda', generator=g).float()
        oc = torch.zeros(C, device='cuda')
        rec.bits(f'FC axis {axis}', ext.QuantizeTensor_FC(xs, sc, oc, 4, 3, -448.0, 448.0, axis, 0),
                 lambda: ref.QuantizeTensor_FC(xs, sc, oc, 4, 3, -448.0, 448.0, axis, 0))


def test_histograms_vs_reference_kernels(ref, ext, rec):
    g = torch.Generator(device='cuda').manual_seed(3)

    def hist_of(fn, bins):
        h = torch.zeros(bins, dtype=torch.int32, device='cuda')
        fn(h)
        return h

    for n, relu in ((31, False), (401408, True), (1 << 21, False)):
        x = torch.randn(n, device='cuda', generator=g) * 2
        if relu: x = torch.relu(x)
        for bins in (4096, 2048, 50):
            hs = float(x.abs().max().item()) / bins
            mn, mx = float(x.min().item()), float(x.max().item())
            for clip in (True, False):
                rec.bits(f'Histogram_T n {n} bins {bins} clip {clip}', hist_of(lambda h: ext.Histogram_T(x, hs, clip, h), bins),
                         lambda: hist_of(lambda h: ref.Histogram_T(x, hs, clip, h), bins))
                rec.bits(f'Histogram_Asymmetric_T n {n} bins {bins} clip {clip}', hist_of(lambda h: ext.Histogram_Asymmetric_T(mn, mx, x, clip, h), bins),
                         lambda: hist_of(lambda h: ref.Histogram_Asymmetric_T(mn, mx, x, clip, h), bins))
        if n == 401408 and rec.recording:
            xh = x[:65536].contiguous(); hs = float(xh.abs().max().item()) / 4096
            np.savez_compressed(os.path.join(refrecord.record_dir(), 'ref_cuda_hist.npz'), x=xh.cpu().numpy(), hist_scale=np.float32(hs),
                                hist=hist_of(lambda h: ref.Histogram_T(xh, hs, True, h), 4096).cpu().numpy())
    x = torch.randn(4, 8, 1000, device='cuda', generator=g)
    for axis in (0, 1):
        C = x.shape[axis]
        a = torch.zeros(C, 128, dtype=torch.int32, device='cuda'); b = torch.zeros_like(a)
        ext.Histogram_C(x, axis, 0.03, True, a)
        rec.bits(f'Histogram_C axis {axis}', a, lambda: (ref.Histogram_C(x, axis, 0.03, True, b), b)[1])


def test_compute_mse_loss_vs_reference(ref, ext, rec):
    r = np.random.RandomState(5)
    for i in range(50):
        h = r.randint(0, 9000, size=2048).tolist()
        step = int(r.randint(1, 9)); start = int(r.randint(0, 512)); end = start + 256 * step
        rec.values(f'compute_mse_loss {i}', np.float64(ext.compute_mse_loss(h, start, step, end)),
                   lambda: np.float64(ref.compute_mse_loss(h, start, step, end)), rtol=0)
