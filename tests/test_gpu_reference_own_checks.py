"""The original project's own checks of its CUDA surface, run on ppq_b200's mirror of that surface (ppq_b200.ffi.CUDA with the original's
argument orders, ppq_b200.qfunction.PPQLinearQuantFunction / PPQFloatingQuantFunction, ppq_b200.observer.Observer), on CUDA tensors:

  * the way the original's tests/test_cuda_kernel.py checks its kernels (re-stated here: same shapes, symmetric / asymmetric offsets, same pass
    criteria: fake-quant and grad_x bit-equal to the torch formulation, grad_s within its SNR bar, 50-bin histogram within 100 counts of histc),
  * against what the original's own functions return for the same call -- its torch path (`USING_CUDA_KERNEL = False`) and its own CUDA
    extension -- stored in tests/golden/ref_python_surface.json (tests/refrecord.py; recording runs the original package with its
    extension installed, see tests/refppq.py).
"""
from math import sqrt

import pytest
import torch

import refppq
import refrecord

pytestmark = pytest.mark.gpu
Q_MIN, Q_MAX = 0, 255


@pytest.fixture(scope='module')
def original():
    """(the original `ppq` package, its own CUDA extension) when recording, else None."""
    if not torch.cuda.is_available(): pytest.skip('no CUDA device')
    ref = refrecord.reference_extension()
    if ref is None: return None
    pkg = refppq.load()
    assert pkg is not None, 'recording needs the original package (tests/refppq.py)'
    return pkg, ref


@pytest.fixture(scope='module')
def rec(original):
    r = refrecord.Record('ref_python_surface', recording=original is not None)
    yield r
    r.save()


def tensor_round(t):
    """ppq_tensor_round with ROUND_HALF_EVEN (utils/round.py)."""
    return torch.round(t)


def snr_error(y_pred, y_real):
    """torch_snr_error (quantization/measure/norm.py): mean over rows of ||y_pred - y_real||^2 / ||y_real||^2."""
    noise = torch.pow(y_pred - y_real, 2).sum(dim=-1)
    signal = torch.pow(y_real, 2).sum(dim=-1)
    return (noise / signal).mean()


SHAPES_T = [([1, 1, 1, 1], True), ([1, 1, 1, 1], False), ([5, 12, 13, 4], True), ([1, 7, 15, 41], False), ([50, 120, 130, 4], True),
            ([12, 74, 15, 411], False), ([50, 7, 130, 1], True), ([12, 4, 15, 3], False), ([5011, 7, 7, 1], True), ([122552, 1, 10, 4], False),
            ([10, 10, 124, 47], True), ([19, 42, 150, 3], False)]
SHAPES_C = [(s, sym, 1) for s, sym in SHAPES_T[:8]] + [([5011, 7, 7, 1], True, 0), ([122552, 1, 10, 4], False, 0), ([10, 10, 124, 47], True, 3),
                                                       ([19, 42, 150, 3], False, 3)]


def offsets(sym, n):
    return torch.zeros(n).cuda() if sym else torch.randint(low=0, high=255, size=[n]).float().cuda()


def test_linear_quantize_t_and_c_the_way_the_reference_tests_them():
    """tests/test_cuda_kernel.py:17-63 re-stated: CUDA.LinearQuantize_T / _C == round(t / s) + o, clip, dequantise in torch, bit for bit."""
    from ppq_b200 import RoundingPolicy
    from ppq_b200.ffi import CUDA
    torch.manual_seed(0)
    policy = RoundingPolicy.ROUND_HALF_EVEN
    for size, sym in SHAPES_T:
        for _ in range(3):
            t = torch.rand(size=size).cuda() * 32
            s, o = torch.rand(size=[1]).cuda(), offsets(sym, 1)
            want = ((tensor_round(t / s) + o).clip(Q_MIN, Q_MAX) - o) * s
            got = CUDA.LinearQuantize_T(t, s, o, Q_MIN, Q_MAX, policy.value)
            assert (want - got).abs().max() == 0, (size, sym)
    for size, sym, c in SHAPES_C:
        for _ in range(3):
            t = torch.rand(size=size).cuda() * 32
            s, o = torch.rand(size=[t.shape[c]]).cuda(), offsets(sym, t.shape[c])
            shape = [1 if axis != c else -1 for axis in range(t.ndim)]
            want = ((tensor_round(t / s.view(shape)) + o.view(shape)).clip(Q_MIN, Q_MAX) - o.view(shape)) * s.view(shape)
            got = CUDA.LinearQuantize_C(t, s, o, c, Q_MIN, Q_MAX, policy.value)
            assert (want - got).abs().max() == 0, (size, sym, c)


def test_linear_quantize_backward_the_way_the_reference_tests_it():
    """tests/test_cuda_kernel.py:66-138 re-stated: grad_x bit-equal, grad_s within the reference's SNR bar (1e-5 unless the gradient is tiny)."""
    from ppq_b200 import RoundingPolicy
    from ppq_b200.ffi import CUDA
    torch.manual_seed(1)
    policy = RoundingPolicy.ROUND_HALF_EVEN

    def grads(value, dy, scale, offset, axis):
        """Straight-through gradient of fake-quant w.r.t. the input and LSQ-style gradient w.r.t. the scale, normalised by sqrt(numel * levels)."""
        q = tensor_round(value / scale) + offset
        below, above = q < Q_MIN, q > Q_MAX
        inside = ~(below | above)
        dx = dy * inside
        per_elem = inside * (((q - offset) * scale - value) / scale) + above * (Q_MAX - offset) + below * (Q_MIN - offset)
        ds = per_elem * dy
        ds = ds.sum() if axis is None else ds.movedim(axis, 0).flatten(1).sum(dim=1)
        return dx, ds / sqrt(value.numel() * (Q_MAX - Q_MIN))               # the whole tensor's element count, per channel too (test_cuda_kernel.py:118)

    def check_scale_grad(got, want, tag):
        snr = snr_error(got.reshape([1, -1]), want.reshape([1, -1])).item()
        assert snr <= 1e-5 or got.abs().max().item() <= 1, tag + (snr,)

    for size, sym in [([1, 1, 1, 1], True), ([5, 12, 13, 4], True), ([1, 7, 15, 41], False), ([5, 12, 2130, 4], True), ([12, 74, 315, 41], False),
                      ([501, 7, 73, 1], True), ([1222, 12, 10, 4], False), ([19, 42, 120, 3], False)]:
        t = torch.rand(size=size).cuda() * 50
        s, o, dy = torch.rand(size=[1]).cuda(), offsets(sym, 1), torch.rand(size=size).cuda()
        gx, gs = CUDA.LinearQuantize_T_B(t, s, o, dy, Q_MIN, Q_MAX, policy.value)
        rx, rs = grads(t, dy, s, o, None)
        assert (rx.flatten() - gx.flatten()).abs().max() == 0, size
        check_scale_grad(gs, rs, (size, 'T'))
    for size, sym, c in [([1, 1, 1, 1], True, 1), ([5, 12, 14, 12], True, 1), ([1, 7, 15, 41], False, 1), ([12, 74, 15, 41], False, 1),
                         ([501, 7, 7, 1], True, 0), ([1222, 1, 10, 4], False, 0), ([10, 10, 14, 47], True, 3), ([19, 42, 10, 3], False, 3)]:
        t = torch.rand(size=size).cuda() * 50
        s, o, dy = torch.rand(size=[t.shape[c]]).cuda(), offsets(sym, t.shape[c]), torch.rand(size=size).cuda()
        shape = [1 if axis != c else -1 for axis in range(t.ndim)]
        gx, gs = CUDA.LinearQuantize_C_B(t, s, o, dy, Q_MIN, Q_MAX, c, policy.value)
        rx, rs = grads(t, dy, s.view(shape), o.view(shape), c)
        assert (rx.flatten() - gx.flatten()).abs().max() == 0, (size, c)
        check_scale_grad(gs, rs, (size, c))


def test_histogram_the_way_the_reference_tests_it():
    """tests/test_cuda_kernel.py:198-208 re-stated: 50-bin Histogram_T of |t| at scale 0.01 within 100 counts of torch.histc per bin."""
    from ppq_b200.ffi import CUDA
    torch.manual_seed(2)
    for _ in range(3):
        t = torch.rand(size=[128, 3, 224, 224]).cuda()
        hist = torch.histc(torch.abs(t), bins=50, min=0, max=0.5)
        got = CUDA.Histogram_T(t, torch.zeros(size=[50]).cuda().int(), 0.01)
        assert torch.abs(hist - got).max().item() < 100


def run_original(original, fn):
    """fn() inside the original package with its own CUDA extension serving ppq.core.ffi."""
    _, ref = original
    from ppq.core import PPQ_CONFIG
    with refppq.use_extension(ref):
        PPQ_CONFIG.USING_CUDA_KERNEL = True
        try: return fn()
        finally: PPQ_CONFIG.USING_CUDA_KERNEL = False


@pytest.mark.parametrize('per_channel', [False, True])
def test_reference_linear_quant_function_cuda_path_equals_its_torch_path(original, rec, per_channel):
    """PPQLinearQuantFunction (qfunction/linear.py:200-215) on CUDA tensors, forward and backward, all 8 rounding policies: ours == the original
    function with its own CUDA extension, and, for ROUND_HALF_EVEN (the policy its own test compares; its torch path spells the others as fp32
    floor / ceil formulas, NEAR_INT not at all), == the original's torch formulation (USING_CUDA_KERNEL False).  Equality as torch.equal:
    -0.0 reads as +0.0."""
    import ppq_b200
    from ppq_b200.qfunction import PPQLinearQuantFunction
    torch.manual_seed(3)
    x = (torch.randn(6, 16, 17, 9).cuda() * 3).requires_grad_(True)
    dy = torch.randn_like(x)
    for rounding in ppq_b200.RoundingPolicy:
        n = 16 if per_channel else 1
        scale = (torch.rand(n).cuda() * 0.1 + 0.01)
        offset = torch.zeros(n).cuda() if not per_channel else torch.randint(0, 255, [n]).float().cuda()

        def forward_backward(fn, config, policies, states):
            cfg = config(symmetrical=not per_channel, channel_axis=1 if per_channel else None, quant_min=-128 if not per_channel else 0,
                         quant_max=127 if not per_channel else 255, rounding=getattr(policies, rounding.name))
            cfg.scale, cfg.offset, cfg.state = scale, offset, states.ACTIVATED
            y = fn(x, cfg)
            (g,) = torch.autograd.grad(y, x, dy)
            return refrecord.plus_zero(torch.stack([y.detach(), g]))

        ours = forward_backward(PPQLinearQuantFunction, ppq_b200.LinearQuantizationConfig, ppq_b200.RoundingPolicy, ppq_b200.QuantizationStates)

        def original_fn():
            import ppq.lib as PFL
            from ppq import QuantizationStates, RoundingPolicy
            from ppq.quantization.qfunction.linear import PPQLinearQuantFunction as F
            return forward_backward(F, PFL.LinearQuantizationConfig, RoundingPolicy, QuantizationStates)

        key = f'LinearQuantFunction per_channel {per_channel} {rounding.name}'
        rec.bits(key + ' cuda', ours, lambda: run_original(original, original_fn))
        if rounding == ppq_b200.RoundingPolicy.ROUND_HALF_EVEN:
            rec.bits(key + ' torch', ours, original_fn)


def test_reference_floating_quant_function_with_our_kernels(original, rec):
    """PPQFloatingQuantFunction (qfunction/floating.py:95-125) has no torch path: ours vs the original function with its own CUDA extension,
    per tensor and per channel (forward: the original's backward returns one gradient too many for autograd, floating.py:48-49)."""
    import ppq_b200
    from ppq_b200.qfunction import PPQFloatingQuantFunction
    torch.manual_seed(4)
    x = torch.randn(4, 24, 33).cuda() * 40
    for axis in (None, 1):
        n = 1 if axis is None else 24
        scale, offset = torch.rand(n).cuda() + 0.5, torch.zeros(n).cuda()

        def config(ctor, states):
            cfg = ctor(channel_axis=axis)
            cfg.scale, cfg.offset, cfg.state = scale, offset, states.ACTIVATED
            if axis is not None: cfg.channel_axis = axis
            return cfg

        cfg = config(ppq_b200.FloatingQuantizationConfig, ppq_b200.QuantizationStates)

        def original_fn():
            import ppq.lib as PFL
            from ppq import QuantizationStates
            from ppq.quantization.qfunction.floating import PPQFloatingQuantFunction as F
            return run_original(original, lambda: F(x, config(PFL.FloatingQuantizationConfig, QuantizationStates)))

        rec.bits(f'FloatingQuantFunction axis {axis}', PPQFloatingQuantFunction(x, cfg), original_fn)
    with pytest.raises(PermissionError):
        PPQFloatingQuantFunction(x.cpu(), cfg)                              # no CPU floating quantisation, as in the original


@pytest.mark.parametrize('algo', ['minmax', 'percentile', 'kl', 'mse'])
def test_reference_observers_through_ppq_lib_with_our_kernels(original, rec, algo):
    """ppq.lib.Observer (lib/quant.py:47-56): observe() + render over the same batches, ours (ppq_b200.observer.Observer) vs the original's own
    observer classes on its own CUDA extension (Quantile / Histogram_T / compute_mse_loss): the same scale and offset, bit for bit."""
    import ppq_b200
    from ppq_b200.observer import Observer
    torch.manual_seed(5)
    batches = [torch.relu(torch.randn(8, 32, 28, 28).cuda()) * (1 + 0.1 * k) for k in range(4)]

    def run(config, observer):
        cfg = config(symmetrical=True, calibration=algo)
        ob = observer(quant_config=cfg)
        phases = 2 if algo in ('kl', 'mse') else 1
        for _ in range(phases):
            for b in batches: ob.observe(b)
            ob.render_quantization_config()
        return torch.cat([cfg.scale.reshape(-1).float().cpu(), cfg.offset.reshape(-1).float().cpu()])

    def original_fn():
        import ppq.lib as PFL
        return run_original(original, lambda: run(PFL.LinearQuantizationConfig, PFL.Observer))

    rec.bits(f'Observer {algo}', run(ppq_b200.LinearQuantizationConfig, Observer), original_fn)
