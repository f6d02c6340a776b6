"""GPU parity: the sm_100a kernels (through the torch binding AND through the raw C ABI) against the CPU oracle and the
golden vectors of the real reference.  Bit-exact for every integer / fake-quant output (the reference's own bar:
tests/test_cuda_kernel.py:35-37 `diff.abs().max() != 0 -> fail`).

Run on the B200 box:  python -m pytest tests -m gpu -x -q
"""
import ctypes
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, cases_of, golden_input, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ext():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from ppq_b200.ffi import extension
    return extension()


@pytest.fixture(scope='module')
def cabi():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    lib = ctypes.CDLL(os.path.join(ROOT, 'ppq_b200', '_lib', 'libppq_b200.so'))
    return lib


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits(a):
    if isinstance(a, torch.Tensor): a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bits_equal(got, want, msg=''):
    g, w = bits(got), bits(want)
    if not np.array_equal(g, w):
        bad = np.flatnonzero(g.reshape(-1) != w.reshape(-1))
        raise AssertionError(f'{msg}: {bad.size} of {g.size} elements differ, first at {bad[0]}: '
                             f'{g.reshape(-1)[bad[0]]:#x} vs {w.reshape(-1)[bad[0]]:#x}')


def t1(v):
    return torch.tensor([v], dtype=torch.float32, device='cuda')


# ------------------------------------------------------------------------------------------------ INT, per tensor
def test_lt_golden_reference_vectors(ext):
    g = load_golden('linear_t.npz')
    for c in cases_of(g):
        k = c['k']
        y = ext.QuantizeTensor_LT(dev(g[f'x{k}']), t1(c['scale']), t1(c['offset']), c['qmin'], c['qmax'], c['mode'])
        assert_bits_equal(y, g[f'y{k}'], f'LT golden case {c}')
        q = ext.QuantizeTensor_toInt(dev(g[f'x{k}']), t1(c['scale']), t1(c['offset']), c['qmin'], c['qmax'], -1000, c['mode'], 32)
        assert np.array_equal(q.cpu().numpy(), g[f'q{k}']), c


def test_lt_config1_bit_exact(ext):
    """BASELINE config 1 (1x512x28x28 INT8 per-tensor): int8 values and dequantised floats identical to the reference CPU path."""
    g = load_golden('config1_lt_1x512x28x28.npz')
    x = np.random.RandomState(int(g['seed'])).standard_normal(size=(1, 512, 28, 28)).astype(np.float32)
    for tag, lo, hi in (('sym', -128, 127), ('asym', 0, 255)):
        s, o = t1(float(g[f'{tag}_scale'])), t1(float(g[f'{tag}_offset']))
        y = ext.QuantizeTensor_LT(dev(x), s, o, lo, hi, 0)
        assert hashlib.sha256(y.cpu().numpy().tobytes()).digest() == bytes(g[f'{tag}_y_sha256'])
        q = ext.QuantizeTensor_toInt(dev(x), s, o, lo, hi, -1000, 0, 8)
        assert q.dtype == (torch.int8 if tag == 'sym' else torch.uint8)
        assert np.array_equal(q.cpu().numpy(), g[f'{tag}_q'])


REF_SHAPES = [[1, 1, 1, 1], [5, 12, 13, 4], [1, 7, 15, 41], [50, 120, 130, 4], [12, 74, 15, 411], [50, 7, 130, 1],
              [12, 4, 15, 3], [5011, 7, 7, 1], [122552, 1, 10, 4], [10, 10, 124, 47], [19, 42, 150, 3]]


@pytest.mark.parametrize('shape', REF_SHAPES)
def test_lt_reference_test_shapes(ext, oracle, shape):
    """The shapes / distributions of the reference's own kernel test (tests/test_cuda_kernel.py:17-37, 145-156), seeded."""
    r = np.random.RandomState(sum(shape))
    for sym in (True, False):
        x = (r.rand(*shape) * 32).astype(np.float32)
        s = np.float32(r.rand() + 1e-3)
        o = np.float32(0 if sym else r.randint(0, 255))
        y = ext.QuantizeTensor_LT(dev(x), t1(s), t1(o), 0, 255, 0)
        assert_bits_equal(y, oracle.linear_quant_t(x, s, o, 0, 255, 0), f'LT {shape} sym={sym}')
        assert y.shape == tuple(shape) and y.data_ptr() != 0


@pytest.mark.parametrize('mode', range(8))
def test_lt_all_rounding_modes_and_ranges(ext, oracle, mode):
    r = np.random.RandomState(100 + mode)
    x = (r.standard_normal(70001) * 40).astype(np.float32)
    s = np.float32(0.25)
    x[::5] = ((np.arange(x.size)[::5] % 201) - 100 + 0.5).astype(np.float32) * s          # exact ties
    x[1::97] = np.float32(0.49999997) * s
    for (lo, hi, o) in ((-128, 127, 0), (0, 255, 131), (-8, 7, 0), (0, 15, 7), (-2 ** 31 + 1, 2 ** 31 - 1, 0)):
        y = ext.QuantizeTensor_LT(dev(x), t1(s), t1(o), lo, hi, mode)
        assert_bits_equal(y, oracle.linear_quant_t(x, s, o, lo, hi, mode), f'mode {mode} range {lo}..{hi}')


@pytest.mark.parametrize('mode', range(8))
def test_rounding_modes_fp32_formulation_matches_double(ext, oracle, mode):
    """The device evaluates the "+ .5" modes in fp32 (floor/ceil + fraction test), the reference in double: same integers on the inputs
    where the two could differ -- neighbours of every half-way point, fractions that round when subtracted, 2^23..2^31, specials."""
    h = np.arange(-300, 300, dtype=np.float32) + np.float32(0.5)
    near = np.concatenate([h, np.nextafter(h, np.float32(np.inf)), np.nextafter(h, np.float32(-np.inf))])
    tiny = np.float32([-1e-30, 1e-30, -1e-45, 1e-45, -0.49999997, 0.49999997, -0.50000006, 0.50000006, -0.5, 0.5, -0.0, 0.0,
                       -0.25 - 2.0 ** -26, -(0.5 - 2.0 ** -25), 0.5 - 2.0 ** -25, -0.99999994, 0.99999994, -1.0000001, 1.0000001])
    big = np.float32([2 ** 23 - 0.5, 2 ** 23 + 1, 2 ** 22 + 0.5, -(2 ** 22 + 0.5), -(2 ** 23 - 0.5), 2 ** 24 + 2, 2147483520.0, -2147483520.0,
                      2 ** 31, -2 ** 31, -2147483904.0, 3e38, -3e38, np.inf, -np.inf, np.nan, 4194303.5, -4194303.5, 8388607.5, -8388607.5])
    r = np.random.RandomState(mode)
    rnd = (r.standard_normal(50000) * np.exp(r.uniform(-20, 20, 50000))).astype(np.float32)
    x = np.concatenate([near, tiny, big, rnd, -rnd])
    for (lo, hi) in ((-2 ** 31 + 1, 2 ** 31 - 1), (-128, 127)):
        y = ext.QuantizeTensor_LT(dev(x), t1(1.0), t1(0), lo, hi, mode)
        assert_bits_equal(y, oracle.linear_quant_t(x, np.float32(1.0), 0, lo, hi, mode), f'mode {mode} {lo}..{hi}')
        q = ext.QuantizeTensor_toInt(dev(x), t1(1.0), t1(0), lo, hi, -1000, mode, 32)
        assert np.array_equal(q.cpu().numpy(), oracle.linear_quant_t(x, np.float32(1.0), 0, lo, hi, mode, return_int=True)[1]), mode
    c = ext.QuantizeTensor_LC(dev(x[:x.size // 4 * 4]).view(4, -1), dev(np.ones(4, np.float32)), dev(np.zeros(4, np.float32)), -2 ** 31 + 1, 2 ** 31 - 1, 0, mode)
    assert_bits_equal(c.view(-1), oracle.linear_quant_t(x[:x.size // 4 * 4], np.float32(1.0), 0, -2 ** 31 + 1, 2 ** 31 - 1, mode), f'LC mode {mode}')


def test_lt_special_values_and_scales(ext, oracle):
    sp = np.float32([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1e-38, 3e38, -3e38, 1e20, -1e20, 2 ** 31, -2 ** 31,
                     2147483520.0, 16777217.0, 0.5, 1.5, 2.5, -0.5, 1e-30, 123456.789])
    x = np.tile(sp, 300)[:6001]
    for s in (1.0, 0.1, 1e-8, 1e-20, 1e20, 3e-39, 2 ** -60, 2 ** 60, 7.5e-10, -0.25, 1.17549435e-38):
        for (lo, hi, o) in ((-128, 127, 0), (0, 255, 128), (-2 ** 31 + 1, 2 ** 31 - 1, 0)):
            y = ext.QuantizeTensor_LT(dev(x), t1(s), t1(o), lo, hi, 0)
            assert_bits_equal(y, oracle.linear_quant_t(x, np.float32(s), o, lo, hi, 0), f'special s={s} {lo}..{hi}')


def test_lt_exact_division_stress(ext, oracle):
    """x / s must be the IEEE quotient: x chosen so that x/s sits within an ulp of k + 0.5 for random s."""
    r = np.random.RandomState(7)
    for _ in range(20):
        s = np.float32(10.0 ** r.uniform(-6, 3))
        k = r.randint(-120, 120, size=200000).astype(np.float32) + np.float32(0.5)
        x = (k * s).astype(np.float32)
        x = np.concatenate([x, np.nextafter(x, np.float32(np.inf)), np.nextafter(x, np.float32(-np.inf))])
        y = ext.QuantizeTensor_LT(dev(x), t1(s), t1(0), -128, 127, 0)
        assert_bits_equal(y, oracle.linear_quant_t(x, s, 0, -128, 127, 0), f'division stress s={s}')


def test_lt_unaligned_and_noncontiguous(ext, oracle):
    r = np.random.RandomState(5)
    base = dev((r.rand(4099) * 32).astype(np.float32))
    for off in (1, 2, 3):
        v = base[off:]                                   # data_ptr not 16-byte aligned -> scalar kernel
        y = ext.QuantizeTensor_LT(v, t1(0.37), t1(3), 0, 255, 0)
        assert_bits_equal(y, oracle.linear_quant_t(v.cpu().numpy(), 0.37, 3, 0, 255, 0), f'offset {off}')
    m = dev((r.rand(64, 48) * 32).astype(np.float32)).t()   # non-contiguous: output is a fresh contiguous tensor
    y = ext.QuantizeTensor_LT(m, t1(0.37), t1(0), 0, 255, 0)
    assert y.is_contiguous()
    assert_bits_equal(y, oracle.linear_quant_t(m.contiguous().cpu().numpy(), 0.37, 0, 0, 255, 0), 'transposed')
    assert y.data_ptr() != m.data_ptr()                  # never in place


def test_lt_tma_variant_bit_identical(ext, oracle):
    r = np.random.RandomState(11)
    for n in (4096, 8192 + 4, 1 << 20, (1 << 20) + 7, 3 * 2048 * 1184 + 1028):
        x = (r.standard_normal(n) * 5).astype(np.float32)
        xd = dev(x)
        y0 = ext.QuantizeTensor_LT(xd, t1(0.05), t1(0), -128, 127, 0)
        ext.set_variant('linear_quant_t', 1)
        try:
            y1 = ext.QuantizeTensor_LT(xd, t1(0.05), t1(0), -128, 127, 0)
        finally:
            ext.set_variant('linear_quant_t', 0)
        assert torch.equal(y0, y1), n
        if n <= (1 << 20) + 7:
            assert_bits_equal(y1, oracle.linear_quant_t(x, 0.05, 0, -128, 127, 0), f'tma n={n}')


def test_lt_errors(ext):
    with pytest.raises(RuntimeError, match='Invalid dtype of Input tensor: Value'):
        ext.QuantizeTensor_LT(torch.zeros(4, device='cuda', dtype=torch.float16), t1(1), t1(0), 0, 255, 0)
    with pytest.raises(RuntimeError, match='Tensor is empty: Value'):
        ext.QuantizeTensor_LT(torch.zeros(0, device='cuda'), t1(1), t1(0), 0, 255, 0)
    with pytest.raises(RuntimeError, match='Invalid dtype of Input tensor: Scale'):
        ext.QuantizeTensor_LT(torch.zeros(4, device='cuda'), t1(1).double(), t1(0), 0, 255, 0)
    with pytest.raises(RuntimeError, match='not on a CUDA device'):
        ext.QuantizeTensor_LT(torch.zeros(4), t1(1), t1(0), 0, 255, 0)


# ------------------------------------------------------------------------------------------------ INT, per channel
def test_lc_golden_reference_vectors(ext):
    g = load_golden('linear_c.npz')
    for c in cases_of(g):
        k = c['k']
        x, s, o = dev(golden_input(g, c)), dev(g[f's{k}']), dev(g[f'o{k}'])
        y = ext.QuantizeTensor_LC(x, s, o, c['qmin'], c['qmax'], c['axis'], c['mode'])
        assert_bits_equal(y, g[f'y{k}'], f'LC golden case {c}')
        q = ext.QuantizeTensor_toInt(x, s, o, c['qmin'], c['qmax'], c['axis'], c['mode'], 32)
        assert np.array_equal(q.cpu().numpy(), g[f'q{k}']), c


LC_SPECS = [([1, 1, 1, 1], 1), ([5, 12, 13, 4], 1), ([1, 7, 15, 41], 1), ([50, 120, 130, 4], 1), ([12, 74, 15, 411], 1),
            ([50, 7, 130, 1], 1), ([12, 4, 15, 3], 1), ([5011, 7, 7, 1], 0), ([122552, 1, 10, 4], 0), ([10, 10, 124, 47], 3),
            ([19, 42, 150, 3], 3), ([32, 1, 3, 3], 0), ([1280, 320, 1, 1], 0), ([1000, 1280], 0), ([2048, 512, 3, 3], 0),
            ([64], 0), ([4, 64, 56, 56], 1), ([8, 197, 768], 2), ([3, 5, 7], -1), ([6, 16, 10], -2)]


@pytest.mark.parametrize('shape,axis', LC_SPECS)
def test_lc_shapes_axes(ext, oracle, shape, axis):
    r = np.random.RandomState(sum(shape) + axis)
    C = shape[axis]
    for sym in (True, False):
        x = (r.rand(*shape) * 32).astype(np.float32)
        s = (r.rand(C) + 1e-3).astype(np.float32)
        o = np.zeros(C, np.float32) if sym else r.randint(0, 255, size=C).astype(np.float32)
        view = [1 if a != (axis % len(shape)) else -1 for a in range(len(shape))]
        # the reference test passes scale / offset pre-viewed as [1, C, 1, 1] (tests/test_cuda_kernel.py:50-58)
        y = ext.QuantizeTensor_LC(dev(x), dev(s).view(view), dev(o).view(view), 0, 255, axis, 0)
        assert_bits_equal(y, oracle.linear_quant_c(x, s, o, axis, 0, 255, 0), f'LC {shape} axis {axis} sym={sym}')


def test_lc_fc_channel_last(ext, oracle):
    """Channel-last layouts (epc == 1): the dedicated kernel (C % 4 == 0, aligned), its fall-backs (C % 4 != 0, unaligned view, fewer
    threads than channel groups), every output type, all rounding modes, badly scaled channels (IEEE slow path) and FP8."""
    r = np.random.RandomState(77)
    for rows, C in ((197 * 8, 768), (3, 4), (1, 8), (4097, 12), (2, 400000), (1000, 47), (33, 1024)):
        x = (r.standard_normal((rows, C)) * 6).astype(np.float32)
        x.reshape(-1)[:: 97] *= 1e6
        s = (r.rand(C) * 0.1 + 1e-3).astype(np.float32); s[1] = 1e-25; s[C - 2] = 1e25
        o = r.randint(-5, 5, size=C).astype(np.float32)
        for mode in ((0, 1, 2, 3, 4, 5, 6, 7) if C == 768 else (0, 4)):
            y = ext.QuantizeTensor_LC(dev(x), dev(s), dev(o), -128, 127, 1, mode)
            assert_bits_equal(y, oracle.linear_quant_c(x, s, o, 1, -128, 127, mode), f'LC last [{rows},{C}] mode {mode}')
        want_q = oracle.linear_quant_c(x, s, o, 1, -128, 127, 0, return_int=True)[1]
        for bits in (32, 8):
            q = ext.QuantizeTensor_toInt(dev(x), dev(s), dev(o), -128, 127, 1, 0, bits)
            assert np.array_equal(q.cpu().numpy().astype(np.int64), want_q.astype(np.int64)), (rows, C, bits)
        xf = fp_inputs(r, max(rows * C, 32))[:rows * C].reshape(rows, C)
        sf = np.exp2(r.randint(-4, 4, size=C)).astype(np.float32) * (1 + r.rand(C).astype(np.float32)); sf[0] = 1e-25
        of = np.zeros(C, np.float32)
        for mode in (0, 1):
            y = ext.QuantizeTensor_FC(dev(xf), dev(sf), dev(of), 4, 3, -448.0, 448.0, 1, mode)
            assert_bits_equal(y, oracle.float_quant_c(xf, sf, of, 1, 4, 3, -448.0, 448.0, mode), f'FC last [{rows},{C}] mode {mode}')
    base = dev((r.standard_normal(1 + 64 * 256) * 4).astype(np.float32))
    v = base[1:].view(64, 256)                                          # not 16-byte aligned -> generic kernel
    s = (r.rand(256) * 0.1 + 1e-3).astype(np.float32); o = np.zeros(256, np.float32)
    assert_bits_equal(ext.QuantizeTensor_LC(v, dev(s), dev(o), -128, 127, 1, 0), oracle.linear_quant_c(v.cpu().numpy(), s, o, 1, -128, 127, 0), 'unaligned')


def test_lc_unaligned_modes_and_special(ext, oracle):
    r = np.random.RandomState(9)
    base = dev((r.standard_normal(3 + 96 * 64) * 4).astype(np.float32))
    s = (r.rand(96) * 0.1 + 1e-3).astype(np.float32); s[5] = 1e-25; s[6] = 1e25
    o = r.randint(-5, 5, size=96).astype(np.float32)
    for off in (0, 1, 3):
        v = base[off:off + 96 * 64].view(96, 64)
        for mode in (0, 1, 4, 7):
            y = ext.QuantizeTensor_LC(v, dev(s), dev(o), -128, 127, 0, mode)
            assert_bits_equal(y, oracle.linear_quant_c(v.cpu().numpy(), s, o, 0, -128, 127, mode), f'off {off} mode {mode}')


def test_multi_tensor_lc_matches_single_launches(ext, oracle):
    """One launch over a table of weights (MobileNetV2-like shapes incl. depth-wise epc = 9, bias-like epc = 1, unaligned views)."""
    from ppq_b200.calibration import MultiWeightQuantizer
    r = np.random.RandomState(77)
    shapes = [(32, 3, 3, 3), (32, 1, 3, 3), (16, 32, 1, 1), (96, 16, 1, 1), (96, 1, 3, 3), (1280, 320, 1, 1), (1000, 1280), (64,), (7, 5, 3), (512, 512, 3, 3), (3, 1000), (5, 132), (1, 4), (2, 1, 1, 1)]
    ws = [dev((r.standard_normal(s) * 0.1).astype(np.float32)) for s in shapes]
    ws[4] = dev(np.concatenate([np.zeros(1, np.float32), ws[4].cpu().numpy().reshape(-1)]))[1:].view(96, 1, 3, 3)     # not 16-byte aligned
    scales = [(w.abs().amax(dim=tuple(range(1, w.dim()))) / 127).clamp_min(1e-8) if w.dim() > 1 else (w.abs() / 127).clamp_min(1e-8) for w in ws]
    offsets = [torch.zeros_like(s) for s in scales]
    mq = MultiWeightQuantizer(ws, scales, offsets, channel_axis=0)
    outs = mq()
    for w, s, o, y in zip(ws, scales, offsets, outs):
        assert torch.equal(y, ext.QuantizeTensor_LC(w, s, o, -128, 127, 0, 0)), tuple(w.shape)
        assert_bits_equal(y, oracle.linear_quant_c(w.cpu().numpy(), s.cpu().numpy(), o.cpu().numpy(), 0, -128, 127, 0), str(tuple(w.shape)))
    offsets = [torch.full_like(s, 3.0) for s in scales]
    outs = MultiWeightQuantizer(ws, scales, offsets, channel_axis=0, quant_min=-8, quant_max=7, rounding=4)()
    for w, s, o, y in zip(ws, scales, offsets, outs):
        assert_bits_equal(y, oracle.linear_quant_c(w.cpu().numpy(), s.cpu().numpy(), o.cpu().numpy(), 0, -8, 7, 4), 'int4 mode 4 ' + str(tuple(w.shape)))


def test_multi_tensor_lt_matches_single_launches(ext, oracle):
    """Multi_QuantizeTensor_LT: the per-tensor activation configs of a graph in one launch, each tensor with its OWN scale and offset (ragged
    sizes, a tensor of 1 element, a tail of 1..3 elements after the last vector, an unaligned view), all rounding modes."""
    from ppq_b200.calibration import MultiWeightQuantizer
    r = np.random.RandomState(78)
    sizes = [401408, 150528, 1, 3, 4099, 1000, 513, 512, 7, 25088 * 3 + 2]
    xs = [dev((r.standard_normal(n) * (1 + i)).astype(np.float32)) for i, n in enumerate(sizes)]
    xs[4] = dev(np.concatenate([np.zeros(1, np.float32), xs[4].cpu().numpy()]))[1:]                        # not 16-byte aligned
    scales = [dev(np.float32([0.01 * (i + 1)])) for i in range(len(xs))]
    offsets = [dev(np.float32([float(i % 5)])) for i in range(len(xs))]
    for mode in range(8):
        outs = MultiWeightQuantizer(xs, scales, offsets, channel_axis=None, quant_min=-100, quant_max=120, rounding=mode)()
        for x, s_, o_, y in zip(xs, scales, offsets, outs):
            assert torch.equal(y, ext.QuantizeTensor_LT(x, s_, o_, -100, 120, mode)), (mode, x.numel())
            assert_bits_equal(y, oracle.linear_quant_t(x.cpu().numpy(), float(s_.item()), float(o_.item()), -100, 120, mode), f'mode {mode} n {x.numel()}')


# ------------------------------------------------------------------------------------------------ FP8 & friends
FP_FORMATS = [(4, 3, -448.0, 448.0), (5, 2, -57344.0, 57344.0), (4, 3, -240.0, 240.0), (5, 10, -65504.0, 65504.0), (3, 4, -30.0, 30.0),
              (2, 1, -6.0, 6.0)]


def fp_inputs(r, n):
    x = (r.standard_normal(n) * 10).astype(np.float32)
    x[::3] = x[::3].astype(np.float16).astype(np.float32)                    # tie-rich: exactly representable in few bits
    x[1::11] = (r.standard_normal(x[1::11].size) * 2 ** -8).astype(np.float32)   # subnormal range of E4M3
    x[2::13] = (r.standard_normal(x[2::13].size) * 300).astype(np.float32)      # saturation
    sp = np.float32([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, 464.0, 480.0, 448.0, 1.1875, 1.4375, 2.375, 19.0, -1.1875,
                     1.5 * 2 ** -9, 2.5 * 2 ** -9, 2 ** -10, -2 ** -11, 2 ** -6, 2 ** -6 * (1 - 2 ** -24), 3e38])
    x[:sp.size] = sp
    return x


@pytest.mark.parametrize('E,M,cmin,cmax', FP_FORMATS)
def test_ft_vs_oracle(ext, oracle, E, M, cmin, cmax):
    r = np.random.RandomState(E * 10 + M)
    x = fp_inputs(r, 200003)
    for s, o in ((1.0, 0.0), (0.125, 0.0), (4.0, 0.0), (0.0078125, 0.0), (0.3, 2.5), (1e-22, 0.0)):
        for mode in (0, 1, 3, 6):
            y = ext.QuantizeTensor_FT(dev(x), t1(s), t1(o), E, M, cmin, cmax, mode)
            assert_bits_equal(y, oracle.float_quant_t(x, s, o, E, M, cmin, cmax, mode), f'FT E{E}M{M} s={s} o={o} mode={mode}')


def test_fc_vs_oracle(ext, oracle):
    r = np.random.RandomState(3)
    for shape, axis in (([64, 3, 3, 3], 0), ([16, 32, 1, 1], 0), ([8, 24, 9], 1), ([4, 12, 64], 2), ([7, 5, 3], 1)):
        x = fp_inputs(r, int(np.prod(shape))).reshape(shape)
        C = shape[axis]
        s = np.float32(2.0) ** r.randint(-7, 6, size=C).astype(np.float32)
        o = np.zeros(C, np.float32)
        y = ext.QuantizeTensor_FC(dev(x), dev(s), dev(o), 4, 3, -448.0, 448.0, axis, 0)
        assert_bits_equal(y, oracle.float_quant_c(x, s, o, axis, 4, 3, -448.0, 448.0, 0), f'FC {shape} axis {axis}')


def test_ft_matches_hardware_fp8_away_from_ties(ext):
    x = (torch.randn(1 << 20, device='cuda', generator=torch.Generator(device='cuda').manual_seed(325)) * 10)
    y = ext.QuantizeTensor_FT(x, t1(1.0), t1(0.0), 4, 3, -448.0, 448.0, 0)
    hw = x.to(torch.float8_e4m3fn).float()
    # differences are confined to exact ties (reference rule: ties toward zero; ~1e-6 of fp32 values are exact E4M3 ties)
    diff = y != hw
    assert diff.sum().item() <= 16 and bool(((x[diff].view(torch.int32) & 0xFFFFF) == 0x80000).all())


# ------------------------------------------------------------------------------------------------ collectors
def test_minmax_t_and_c(ext, oracle):
    r = np.random.RandomState(21)
    for n in (1, 3, 1000, 65537, 1 << 20):
        x = (r.standard_normal(n) * 3).astype(np.float32)
        for off in (0, 1):
            xd = dev(np.concatenate([np.zeros(off, np.float32), x]))[off:]
            mm = torch.empty(2, device='cuda'); ext.MinMax_Init(mm[0:1], mm[1:2])
            ext.MinMax_T(xd, mm)
            assert mm.tolist() == [float(x.min()), float(x.max())]
    # accumulation across calls == global min/max (the observer never keeps per-batch lists)
    mm = torch.empty(2, device='cuda'); ext.MinMax_Init(mm[0:1], mm[1:2])
    xs = [(r.standard_normal(5000) * (i + 1)).astype(np.float32) for i in range(4)]
    for x in xs: ext.MinMax_T(dev(x), mm)
    assert mm.tolist() == [float(min(x.min() for x in xs)), float(max(x.max() for x in xs))]
    # all-negative / all-positive / signed zeros / NaN poisoning (torch.min / torch.max propagate NaN)
    for arr in ([-3.0, -1.0, -2.0], [3.0, 1.0, 2.0], [0.0, -0.0], [1.0, float('nan'), -5.0]):
        mm = torch.empty(2, device='cuda'); ext.MinMax_Init(mm[0:1], mm[1:2])
        t = torch.tensor(arr, device='cuda'); ext.MinMax_T(t, mm)
        want = [t.min().item(), t.max().item()]
        got = mm.tolist()
        assert all((g == w) or (g != g and w != w) for g, w in zip(got, want)), (arr, got, want)
    for shape, axis in (([64, 3, 3, 3], 0), ([32, 1, 3, 3], 0), ([8, 24, 14, 14], 1), ([5, 7, 9], 2), ([2048, 4608], 0), ([3, 10000], 0)):
        x = (r.standard_normal(shape) * 2).astype(np.float32)
        C = shape[axis]
        lo = torch.empty(C, device='cuda'); hi = torch.empty(C, device='cuda'); ext.MinMax_Init(lo, hi)
        ext.MinMax_C(dev(x), axis, lo, hi)
        wlo, whi = oracle.minmax_c(x, axis)
        assert np.array_equal(lo.cpu().numpy(), wlo) and np.array_equal(hi.cpu().numpy(), whi), (shape, axis)


@pytest.mark.parametrize('variant', [0, 1, 2, 3, 4, 7, 8])
def test_histograms_exact_vs_oracle(ext, oracle, variant):
    r = np.random.RandomState(31 + variant)
    ext.set_variant('histogram', variant)
    try:
        for n, relu in ((1, False), (31, True), (4099, False), (401408, True), (1 << 21, False)):
            x = (r.standard_normal(n) * 2).astype(np.float32)
            if relu: x = np.maximum(x, 0)
            x[:min(n, 4)] = np.float32([np.nan, np.inf, -0.0, 1e-40])[:min(n, 4)]
            for bins in (4096, 2048, 50):
                hs = np.float32(np.abs(x[np.isfinite(x)]).max() / bins) if np.isfinite(x).any() and np.abs(x[np.isfinite(x)]).max() > 0 else np.float32(0.01)
                for clip in (True, False):
                    h = torch.zeros(bins, dtype=torch.int32, device='cuda')
                    ext.Histogram_T(dev(x), float(hs), clip, h)
                    ext.Histogram_T(dev(x), float(hs), clip, h)                                 # accumulates in place
                    want = oracle.histogram_t(x, hs, bins, clip); want = oracle.histogram_t(x, hs, clip_outliers=clip, hist=want)
                    assert np.array_equal(h.cpu().numpy(), want), (n, bins, clip, variant)
            fin = x[np.isfinite(x)]
            if fin.size:
                vmin, vmax = float(fin.min()), float(fin.max() + 1e-3)
                for clip in (True, False):
                    h = torch.zeros(2048, dtype=torch.int32, device='cuda')
                    ext.Histogram_Asymmetric_T(vmin, vmax, dev(x), clip, h)
                    assert np.array_equal(h.cpu().numpy(), oracle.histogram_asym_t(x, vmin, vmax, 2048, clip)), (n, clip, variant)
    finally:
        ext.set_variant('histogram', 0)


def test_histogram_c_and_reference_histc_bar(ext, oracle):
    r = np.random.RandomState(41)
    for shape, axis in (([16, 3, 3, 3], 0), ([4, 8, 100], 1), ([2, 5, 70000], 1)):
        x = (r.standard_normal(shape)).astype(np.float32)
        C = shape[axis]
        h = torch.zeros(C, 256, dtype=torch.int32, device='cuda')
        ext.Histogram_C(dev(x), axis, 0.02, True, h)
        assert np.array_equal(h.cpu().numpy(), oracle.histogram_c(x, axis, np.float32(0.02), 256, True)), shape
    # the reference's own check (tests/test_cuda_kernel.py:197-208): |kernel - torch.histc| < 100 on rand(128,3,224,224), 50 bins
    t = torch.rand(16, 3, 224, 224, device='cuda', generator=torch.Generator(device='cuda').manual_seed(401))
    h = torch.zeros(50, dtype=torch.int32, device='cuda')
    ext.Histogram_T(t, 0.01, True, h)
    ref = torch.histc(torch.abs(t), bins=50, min=0, max=0.5)
    assert torch.abs(ref - h).max().item() < 100


def test_histogram_device_scale_and_multi_tensor(ext, oracle):
    r = np.random.RandomState(51)
    tensors = [np.maximum(r.standard_normal(n) * (i + 1), 0).astype(np.float32) for i, n in enumerate((1000, 401408, 70001, 5, 200000))]
    T, bins = len(tensors), 4096
    devs = [dev(x) for x in tensors]
    arena_mm = torch.empty(T, 2, device='cuda'); arena_mm[:, 0] = float('inf'); arena_mm[:, 1] = float('-inf')
    descs = torch.tensor([[d.data_ptr(), d.numel(), i] for i, d in enumerate(devs)], dtype=torch.int64, device='cuda')
    ext.Multi_MinMax_T(descs, max(d.numel() for d in devs), arena_mm)
    for i, x in enumerate(tensors):
        assert arena_mm[i].tolist() == [float(x.min()), float(x.max())]
    hs = ext.Hist_Scale_From_MinMax(arena_mm, True, bins)
    for i, x in enumerate(tensors):
        assert hs[i].item() == np.float32(max(abs(float(x.min())), abs(float(x.max()))) / bins)
    hist = torch.zeros(T, bins, dtype=torch.int32, device='cuda')
    ext.Multi_Histogram_T(descs, max(d.numel() for d in devs), hs, True, hist, bins)
    one = torch.zeros(bins, dtype=torch.int32, device='cuda')
    for i, x in enumerate(tensors):
        want = oracle.histogram_t(x, hs[i].item(), bins, True)
        assert np.array_equal(hist[i].cpu().numpy(), want), i
        one.zero_(); ext.Histogram_T_DeviceScale(devs[i], hs[i:i + 1], True, one)
        assert np.array_equal(one.cpu().numpy(), want), i


# ------------------------------------------------------------------------------------------------ scale search on the device
def test_minmax_to_scale_offset_kernel_vs_reference_kats(ext):
    import json
    from conftest import GOLDEN
    kat = json.load(open(os.path.join(GOLDEN, 'scalar_kats.json')))['minmax_to_scale_offset']
    groups = {}
    for lo, hi, sym, pow2, qmin, qmax, s, o in kat:
        groups.setdefault((sym, pow2, qmin, qmax), []).append((lo, hi, s, o))
    for (sym, pow2, qmin, qmax), rows in groups.items():
        lo = torch.tensor([r[0] for r in rows], dtype=torch.float32, device='cuda')
        hi = torch.tensor([r[1] for r in rows], dtype=torch.float32, device='cuda')
        s, o = ext.MinMax_To_Scale_Offset(lo, hi, 1, qmin, qmax, bool(sym), bool(pow2), 1e-8)
        assert np.array_equal(s.cpu().numpy(), np.float32([r[2] for r in rows])), (sym, pow2, qmin, qmax)
        assert np.array_equal(o.cpu().numpy(), np.float32([r[3] for r in rows])), (sym, pow2, qmin, qmax)


@pytest.mark.parametrize('variant', [0, 1])
def test_kl_search_kernel_vs_reference(ext, variant):
    g = load_golden('hist_search.npz')
    cs = cases_of(g)
    ext.set_variant('kl_search', variant)            # 0: one warp per candidate (default), 1: the serial-candidate kernel
    for bits_ in (8, 4):
        sel = [c for c in cs if c['bits'] == bits_]
        hist = torch.tensor(np.stack([g[f"hist{c['k']}"] for c in sel]), dtype=torch.int32, device='cuda')
        hs = torch.tensor([c['hist_scale'] for c in sel], dtype=torch.float32, device='cuda')
        scale, best = ext.KL_Search(hist, 4096, hs, None, bits_, False, 1e-8)
        for i, c in enumerate(sel):
            qb = 2 ** (bits_ - 1)
            want_best = round(c['scale'] / c['hist_scale'] * qb)
            assert best[i].item() == want_best, (c, best[i].item())
            assert scale[i].item() == np.float32((want_best / 4096) * float(np.float32(c['hist_scale'])) * (4096 / qb)), c
    ext.set_variant('kl_search', 0)


def test_kl_search_small_histograms_and_oracle_fuzz(ext, oracle):
    """OBSERVER_KL_HIST_BINS_MANUL_OVERRIDE values below the CTA width (256, 512 bins: ADVICE r1) and random histograms of several shapes: both
    device kernels pick the oracle's bin range (the oracle's KL search is itself pinned on the reference's, tests/test_oracle_pinning.py)."""
    r = np.random.RandomState(91)
    for bins, bits_ in ((256, 8), (512, 8), (1024, 8), (4096, 8), (4096, 4), (2048, 6), (8192, 8)):
        hs_ = []
        for kind in range(6):
            base = r.gamma(0.6 + 0.4 * kind, 40.0, size=bins) * np.exp(-np.arange(bins) / (bins / (1.5 + kind)))
            if kind == 4: base[bins // 3:] = 0                                  # empty tail
            if kind == 5: base[r.rand(bins) < 0.7] = 0                          # sparse
            hs_.append(np.floor(base).astype(np.int32))
        hist = torch.tensor(np.stack(hs_), dtype=torch.int32, device='cuda')
        hscale = torch.full((len(hs_),), 0.01, dtype=torch.float32, device='cuda')
        want = [oracle.kl_search(h_, float(np.float32(0.01)), bits_, return_losses=True) for h_ in hs_]
        for variant in (0, 1):
            ext.set_variant('kl_search', variant)
            try:
                scale, best = ext.KL_Search(hist, bins, hscale, None, bits_, False, 1e-8)
            finally:
                ext.set_variant('kl_search', 0)
            for i, wres in enumerate(want):
                losses = np.asarray(wres[3], dtype=np.float64)
                wb = wres[2]
                got = best[i].item()
                if got != wb:                                                   # only a numerical tie may move the argmin
                    qb = 2 ** (bits_ - 1)
                    assert abs(losses[got // qb - 1] - losses[wb // qb - 1]) <= 1e-12 * max(1.0, abs(losses[wb // qb - 1])), (bins, bits_, variant, i, got, wb)
                else:
                    assert scale[i].item() == np.float32(wres[0]), (bins, bits_, variant, i)


def test_mse_search_kernel_vs_host_search(ext, oracle):
    """Device MSE grid search == the host search over the native compute_mse_loss (the reference's USING_CUDA_KERNEL=True flow), sym and asym,
    on the reference-generated histograms and on random ones; ties resolved to the first candidate like python's stable sort."""
    from ppq_b200.search import mse_search_host
    g = load_golden('hist_search.npz')
    hists, mms, want = [], [], []
    for c in cases_of(g, 'mse_cases'):
        hists.append(g[f"mse_hist{c['j']}"]); mms.append((np.float32(c['vmin']), np.float32(c['vmax']))); want.append(c)
    r = np.random.RandomState(8)
    for j in range(6):
        h = (r.gamma(0.6, 300.0, size=2048) * (r.rand(2048) > 0.3)).astype(np.int32)
        if j == 5: h[:] = 7                                   # flat histogram: many tied candidates
        lo, hi = np.float32(-r.rand() * 3 - 0.1), np.float32(r.rand() * 5 + 0.1)
        hists.append(h); mms.append((lo, hi)); want.append(None)
    H = torch.tensor(np.stack(hists), dtype=torch.int32, device='cuda')
    MM = torch.tensor(np.array(mms, np.float32), device='cuda')
    for sym in (True, False):
        qmin, qmax = (-128, 127) if sym else (0, 255)
        s, o = ext.MSE_Search(H, 2048, MM, qmin, qmax, sym, False, 1e-8, 8)
        for i, (h, (lo, hi)) in enumerate(zip(hists, mms)):
            hs = (max(abs(float(lo)), abs(float(hi))) if sym else (float(hi) - float(lo))) / 2048
            ws, wo = mse_search_host(h.tolist(), hs, float(lo), qmin, qmax, sym, False, 1e-8)
            assert s[i].item() == np.float32(ws) and o[i].item() == np.float32(wo), (sym, i, s[i].item(), ws)
            os_, oo = oracle.mse_search(h, hs, float(lo), qmin, qmax, sym)
            assert np.float32(os_) == np.float32(ws) and float(oo) == float(wo)


def test_observers_end_to_end_vs_reference(ext, oracle):
    """Same data (seeded) through ppq_b200 observers on the GPU.
    minmax (per tensor / per channel): scales and offsets must equal the reference CPU pipeline's (tests/golden/observers.npz).
    kl / mse: the reference's CPU branch collects with torch.histc while its CUDA branch (and ours, bit-exact with its kernel:
    test_gpu_vs_reference_cuda.py) floors |x|/hist_scale and drops x == max, so the expected scale is the oracle chain
    device-histogram -> reference search; the CPU-path golden scale must still be within one search candidate."""
    from conftest import seeded_batches
    from ppq_b200 import LinearQuantizationConfig, QuantizationStates
    from ppq_b200.observer import Observer
    g = load_golden('observers.npz')
    for c in cases_of(g):
        if c['algo'] == 'percentile': continue          # Quantile_T path: covered in test_gpu_next_rows.py
        k, sym = c['k'], c['sym']
        host = seeded_batches(c['seed'], c['n'], tuple(c['shape']), c['relu'])
        data = [dev(x) for x in host]
        qmin, qmax = (-128, 127) if sym else (0, 255)
        cfg = LinearQuantizationConfig(symmetrical=sym, quant_min=qmin, quant_max=qmax, calibration=c['algo'], channel_axis=c.get('axis'))
        ob = Observer(cfg)
        for x in data: ob.observe(x)
        ob.render_quantization_config()
        if c['algo'] in ('kl', 'mse'):
            for x in data: ob.observe(x)
            ob.render_quantization_config()
        assert cfg.state == QuantizationStates.ACTIVATED
        got_s, got_o = cfg.scale.cpu().numpy().reshape(-1), cfg.offset.cpu().numpy().reshape(-1)
        if c['algo'] == 'minmax':
            assert np.array_equal(got_s, g[f'scale{k}'].reshape(-1)), c
            assert np.array_equal(got_o, g[f'offset{k}'].reshape(-1)), c
            continue
        vmin, vmax = (float(v) for v in g[f'minmax{k}'])
        bins = 4096 if c['algo'] == 'kl' else 2048
        hs = (max(abs(vmin), abs(vmax)) if sym else (vmax - vmin)) / bins
        hist = np.zeros(bins, np.int32)
        for x in host:
            if sym: oracle.histogram_t(x, np.float32(hs), hist=hist)
            else: oracle.histogram_asym_t(x, vmin, vmax, hist=hist)
        assert np.array_equal(ob._hist.cpu().numpy(), hist), c
        if c['algo'] == 'kl': want_s, want_o = oracle.kl_search(hist, hs, 8)
        else: want_s, want_o = oracle.mse_search(hist, hs, vmin, qmin, qmax, sym)
        assert got_s[0] == np.float32(want_s) and got_o[0] == np.float32(want_o), (c, got_s, want_s)
        ref_s = float(g[f'scale{k}'].reshape(-1)[0])
        assert 0.8 <= got_s[0] / ref_s <= 1.25, (c, got_s, ref_s)            # CPU-path (histc) scale: a neighbouring search candidate at most


# ------------------------------------------------------------------------------------------------ raw C ABI + full-size properties
def test_c_abi_direct_call(cabi, oracle):
    x = torch.rand(1000003, device='cuda', generator=torch.Generator(device='cuda').manual_seed(535)) * 32
    y = torch.empty_like(x)
    s, o = t1(0.11), t1(17)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = cabi.ppq_b200_linear_quant_t(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), ctypes.c_int64(x.numel()),
                                      ctypes.c_void_p(s.data_ptr()), ctypes.c_void_p(o.data_ptr()), 0, 255, 0, st)
    assert rc == 0
    assert_bits_equal(y, oracle.linear_quant_t(x.cpu().numpy(), 0.11, 17, 0, 255, 0), 'C ABI LT')
    assert cabi.ppq_b200_linear_quant_t(None, None, ctypes.c_int64(0), None, None, 0, 255, 0, st) == 1     # cudaErrorInvalidValue
    assert cabi.ppq_b200_float_quant_t(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), ctypes.c_int64(8),
                                       ctypes.c_void_p(s.data_ptr()), ctypes.c_void_p(o.data_ptr()), 9, 3,
                                       ctypes.c_float(-1), ctypes.c_float(1), 0, st) == 1


def test_full_size_properties(ext):
    """BASELINE-size tensors (1x2048x64x64 and BERT [32,512,768]): size-independent properties instead of a CPU oracle."""
    g = torch.Generator(device='cuda').manual_seed(20260922)
    for shape in ((1, 2048, 64, 64), (32, 512, 768)):
        x = torch.randn(shape, device='cuda', generator=g) * 3
        s, o = t1(0.05), t1(0)
        y = ext.QuantizeTensor_LT(x, s, o, -128, 127, 0)
        assert torch.equal(ext.QuantizeTensor_LT(y, s, o, -128, 127, 0), y)                 # idempotent
        q = ext.QuantizeTensor_toInt(x, s, o, -128, 127, -1000, 0, 8)
        assert torch.equal(q.float() * 0.05, y)                                            # dequantised ints == fake-quant
        # error bound: half a step inside the range, distance to the clamp outside it (+ fp32 rounding of the subtraction itself)
        assert (y - x).abs().max().item() <= max(0.025, x.abs().max().item() - 127 * 0.05) + 1e-5
        assert torch.equal(ext.QuantizeTensor_LT(-x, s, o, -127, 127, 0), -ext.QuantizeTensor_LT(x, s, o, -127, 127, 0))  # odd symmetry
        # per-channel with equal scales == per-tensor
        C = shape[1]
        yc = ext.QuantizeTensor_LC(x, torch.full((C,), 0.05, device='cuda'), torch.zeros(C, device='cuda'), -128, 127, 1, 0)
        assert torch.equal(yc, y)
        # FP8: idempotent, matches the hardware conversion away from ties
        f = ext.QuantizeTensor_FT(x, t1(1.0), t1(0.0), 4, 3, -448.0, 448.0, 0)
        assert torch.equal(ext.QuantizeTensor_FT(f, t1(1.0), t1(0.0), 4, 3, -448.0, 448.0, 0), f)
        hw = x.to(torch.float8_e4m3fn).float()
        diff = f != hw
        # exact ties (low 20 mantissa bits == 0x80000: ~1e-6 of fp32 values) follow the reference rule (toward zero), hardware is ties-to-even
        assert diff.sum().item() <= x.numel() * 4e-6 and bool(((x[diff].view(torch.int32) & 0xFFFFF) == 0x80000).all())
        # collectors: min/max equal torch's, histogram mass == number of in-range samples
        mm = torch.empty(2, device='cuda'); ext.MinMax_Init(mm[0:1], mm[1:2]); ext.MinMax_T(x, mm)
        assert mm[0].item() == x.min().item() and mm[1].item() == x.max().item()
        hs = float(x.abs().max().item()) / 4096
        h = torch.zeros(4096, dtype=torch.int32, device='cuda'); ext.Histogram_T(x, hs, True, h)
        inrange = (torch.floor(x.abs() / torch.tensor(hs, device='cuda', dtype=torch.float32)) <= 4095).sum().item()
        assert h.sum().item() == inrange and x.numel() - inrange <= 4


# ------------------------------------------------------------------------------------------------ limits
def test_maximum_size_and_too_many_elements(ext):
    """The reference accepts numel <= 2^31 - 1 and throws beyond (linear.cu:108-109).  2^31 - 1 fp32 elements = 8.6 GB in + 8.6 GB out."""
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9: pytest.skip('needs ~26 GB of free HBM')
    n = 2 ** 31 - 1
    x = torch.empty(n, device='cuda').uniform_(-4, 4)
    s, o = t1(0.031), t1(0)
    y = ext.QuantizeTensor_LT(x, s, o, -128, 127, 0)
    for sl in (slice(0, 1 << 20), slice(n - (1 << 20) - 3, n), slice(n // 2 - 5, n // 2 + (1 << 20))):      # head, ragged tail, middle
        assert torch.equal(y[sl], ext.QuantizeTensor_LT(x[sl].clone(), s, o, -128, 127, 0))
    mm = torch.empty(2, device='cuda'); ext.MinMax_Init(mm[0:1], mm[1:2]); ext.MinMax_T(x, mm)
    assert mm[0].item() == x.min().item() and mm[1].item() == x.max().item()
    h = torch.zeros(4096, dtype=torch.int32, device='cuda'); ext.Histogram_T(x, 4.0 / 4096, True, h)
    assert h.sum().item() == n - int((torch.floor(x.abs() / torch.tensor(4.0 / 4096, device='cuda')) > 4095).sum().item())
    del y
    big = torch.empty(2 ** 31, device='cuda')
    with pytest.raises(RuntimeError, match='too many element'):
        ext.QuantizeTensor_LT(big, s, o, -128, 127, 0)
    with pytest.raises(RuntimeError, match='too many element'):
        ext.QuantizeTensor_LC(big.view(2, -1), torch.ones(2, device='cuda'), torch.zeros(2, device='cuda'), -128, 127, 0, 0)


def test_histogram_many_bins_and_tiny_inputs(ext, oracle):
    r = np.random.RandomState(61)
    x = (r.standard_normal(300000) * 3).astype(np.float32)
    for bins in (12287, 12288, 65536, 1):                       # shared-memory limit, global-atomic fallback, degenerate
        hs = np.float32(12.0 / bins)
        h = torch.zeros(bins, dtype=torch.int32, device='cuda')
        ext.Histogram_T(dev(x), float(hs), True, h)
        assert np.array_equal(h.cpu().numpy(), oracle.histogram_t(x, hs, bins, True)), bins
    for n in (1, 2, 3, 4, 5, 31, 32, 33):                       # ragged tails around the vector / warp widths
        xs = x[:n].copy()
        h = torch.zeros(64, dtype=torch.int32, device='cuda'); ext.Histogram_T(dev(xs), 0.2, False, h)
        assert np.array_equal(h.cpu().numpy(), oracle.histogram_t(xs, np.float32(0.2), 64, False)), n
        y = ext.QuantizeTensor_LT(dev(xs), t1(0.1), t1(1), -8, 7, 0)
        assert_bits_equal(y, oracle.linear_quant_t(xs, 0.1, 1, -8, 7, 0), f'tiny n={n}')
