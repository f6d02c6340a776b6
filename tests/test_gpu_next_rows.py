"""GPU parity of the "next" rows (SURVEY.md §8f): Quantile_T / Isotone_T by radix select, LSQ backward, float backward,
TensorClip, RoundingLoss -- against the original project's own CUDA kernels (their outputs for these seeded inputs are stored in
tests/golden/ref_cuda_next_rows.json, see tests/refrecord.py), and against the oracle / the torch formulas of the original's test
(tests/test_cuda_kernel.py:66-143).
Element-wise outputs must be bit-identical; scalar fp32 reductions (grad_s, loss) to 1e-4 relative (the reference's own bar is SNR 1e-3)."""
from math import sqrt

import numpy as np
import pytest
import torch

import refrecord

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ext():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from ppq_b200.ffi import extension
    return extension()


@pytest.fixture(scope='module')
def ref():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return refrecord.reference_extension()


@pytest.fixture(scope='module')
def rec(ref):
    r = refrecord.Record('ref_cuda_next_rows', recording=ref is not None)
    yield r
    r.save()


def close(a, b, rtol=1e-4, atol=1e-6):
    return torch.allclose(a.double(), b.double(), rtol=rtol, atol=atol)


def test_quantile_vs_sort_oracle_and_reference(ext, ref, rec, oracle):
    g = torch.Generator(device='cuda').manual_seed(0)
    for n in (1, 2, 3, 17, 1000, 4099, 401408, (1 << 21) + 5):
        for kind in ('randn', 'relu', 'negrelu', 'const', 'ints', 'close'):
            x = torch.randn(n, device='cuda', generator=g) * 3
            if kind == 'relu': x = torch.relu(x)
            if kind == 'negrelu': x = -torch.relu(x)                              # half of the elements are -0.0: the bucket of +0 must take them
            if kind == 'const': x = torch.full((n,), -1.25, device='cuda')
            if kind == 'ints': x = torch.randint(-5, 5, (n,), device='cuda', generator=g).float()
            if kind == 'close':                                                   # three values that share the top 11 / top 22 key bits: a bucket too
                vals = torch.tensor([1.0, 1.0 + 2.0 ** -23, 1.0 + 2.0 ** -12], device='cuda')   # big to compact (n = 2 M) must be refined by passes 1 and 2
                x = vals[torch.randint(0, 3, (n,), device='cuda', generator=g)]
            if n > 8: x[3] = -0.0; x[5] = 0.0
            for q in (0.9999, 0.999, 0.5, 1.0, 0.0):
                got = ext.Quantile_T(x, q)
                srt = torch.sort(x)[0]
                fa = np.float32(n) * np.float32(q); fb = np.float32(n) * (np.float32(1) - np.float32(q))
                ia = int(min(max(np.rint(fa), 0), n - 1)); ib = int(min(max(np.rint(fb), 0), n - 1))
                want = torch.stack([srt[ia], srt[ib]])
                assert torch.equal(got, want), (n, kind, q, got, want)          # value equality (-0.0 == +0.0)
                if n <= 4099:
                    assert np.array_equal(got.cpu().numpy(), oracle.quantile_t(x.cpu().numpy(), q)), (n, kind, q)
                if n > 1:                                                         # bits with -0.0 read as +0.0
                    rec.bits(f'Quantile_T n {n} {kind} q {q}', refrecord.plus_zero(got), lambda: refrecord.plus_zero(ref.Quantile_T(x, q)))
    # unaligned view + non-contiguous input
    base = torch.randn(10007, device='cuda', generator=g)
    v = base[1:]
    assert torch.equal(ext.Quantile_T(v, 0.99), torch.stack([torch.sort(v)[0][int(np.rint(np.float32(v.numel()) * np.float32(0.99)))],
                                                             torch.sort(v)[0][int(np.rint(np.float32(v.numel()) * (np.float32(1) - np.float32(0.99))))]]))


def test_multi_tensor_quantile_matches_single_launches(ext):
    """Multi_Quantile_T: one launch per pass over a table of tensors (ragged sizes, tiny tensors, post-ReLU tensors) must select the very same
    elements as one Quantile_T per tensor -- with a workspace big enough to compact the selected buckets, and with a tiny one that forces the
    refine-by-histogram fallback on every level."""
    g = torch.Generator(device='cuda').manual_seed(5)
    sizes = [1, 3, 1000, 4099, 401408, 150528, 7, (1 << 20) + 3, 25088, 2]
    xs = []
    for i, n in enumerate(sizes):
        x = torch.randn(n, device='cuda', generator=g) * (i + 1)
        if i % 3 == 1: x = torch.relu(x)
        if i == 5: x = torch.randint(-3, 3, (n,), device='cuda', generator=g).float()
        xs.append(x)
    slots = list(range(len(xs)))[::-1]                                           # results land in the slot the descriptor names
    descs = torch.tensor([[x.data_ptr(), x.numel(), s] for x, s in zip(xs, slots)], dtype=torch.int64, device='cuda')
    for q in (0.9999, 0.99, 0.5):
        want = torch.stack([ext.Quantile_T(x, q) for x in xs])
        for cap in (1 << 16, 64):
            ws = torch.empty(ext.Multi_Quantile_Workspace_Bytes(len(xs), cap), dtype=torch.uint8, device='cuda')
            out = torch.full((len(xs), 3), -7.0, device='cuda')                  # out_stride 3: the third column must stay untouched
            ext.Multi_Quantile_T(descs, max(sizes), q, out, 3, ws, cap, None)
            assert torch.equal(out[slots, :2], want), (q, cap, out, want)
            assert bool((out[:, 2] == -7.0).all())
    with pytest.raises(RuntimeError, match='workspace is too small'):
        ext.Multi_Quantile_T(descs, max(sizes), 0.5, torch.zeros(len(xs), 2, device='cuda'), 2, torch.empty(16, dtype=torch.uint8, device='cuda'), 64, None)


def test_cold_quantile_with_thresholds_from_a_sample(ext, ref, rec):
    """Tensors of >= 8 M elements: a cold Quantile_T draws 16384 samples in its init CTA and speculates on thresholds derived from them (select.cu,
    "self-speculation").  Whatever the sample says, the result must be the exact order statistics: well-behaved data, post-ReLU zeros and clipped
    maxima (the threshold key itself is massively repeated), a constant, few outliers the sample cannot see, structure with the sampling period,
    and -- with the sample positions reproduced here -- values planted exactly where the sampler looks, which makes its thresholds useless."""
    g = torch.Generator(device='cuda').manual_seed(21)
    n = (1 << 23) + 4099
    m, stride = 16384, ((1 << 23) + 4099) // 16384
    i = torch.arange(m, dtype=torch.int64)
    pos = (i * stride + ((i * 0x9E3779B1) % (1 << 32)) % stride).cuda()     # the sampler's positions: one per stride window at a hashed offset

    def check(x, q, tag):
        got = ext.Quantile_T(x, q)
        srt = torch.sort(x)[0]
        ia = int(min(max(np.rint(np.float32(n) * np.float32(q)), 0), n - 1)); ib = int(min(max(np.rint(np.float32(n) * (np.float32(1) - np.float32(q))), 0), n - 1))
        assert torch.equal(got, torch.stack([srt[ia], srt[ib]])), (tag, q, got, srt[ia], srt[ib])
        rec.bits(f'cold Quantile_T {tag} q {q}', refrecord.plus_zero(got), lambda: refrecord.plus_zero(ref.Quantile_T(x, q)))
        ext.set_variant('select', 64)                                        # the same call without the sample: the regular two-pass route
        try: assert torch.equal(ext.Quantile_T(x, q), got), (tag, q)
        finally: ext.set_variant('select', 0)

    base = torch.randn(n, device='cuda', generator=g) * 2
    cases = {'randn': base, 'relu': torch.relu(base), 'relu6-like': torch.clamp(base, 0.0, 1.5), 'const': torch.full((n,), 0.75, device='cuda')}
    x = torch.zeros(n, device='cuda'); x[:700] = 5.0 + torch.rand(700, device='cuda', generator=g); x[-300:] = -3.0
    cases['outliers the sample cannot see'] = x
    cases['period of the stride'] = (torch.arange(n, device='cuda') % stride).float()
    x = base.clone(); x[pos[:64]] = 1e6; x[pos[64:128]] = -1e6                 # the sampler sees 64 huge values: its thresholds keep ~64 candidates, far fewer than needed
    cases['planted at the sample positions'] = x
    x = torch.relu(base); x[pos] = 3.0                                         # every sample is the same mid-range value: both thresholds equal 3.0
    cases['all samples equal'] = x
    for tag, x in cases.items():
        for q in (0.9999, 0.99999, 0.999, 0.99):
            check(x, q, tag)
    # the first call with a guess buffer samples too, later calls use the remembered thresholds
    guess = ext.Quantile_Guess_Init(1, torch.zeros(1, device='cuda'))
    for step in range(3):
        x = torch.relu(torch.randn(n, device='cuda', generator=g)) * (1 + 0.05 * step)
        srt = torch.sort(x)[0]
        ia = int(np.rint(np.float32(n) * np.float32(0.9999))); ib = int(np.rint(np.float32(n) * (np.float32(1) - np.float32(0.9999))))
        assert torch.equal(ext.Quantile_T_Guess(x, 0.9999, guess), torch.stack([srt[ia], srt[ib]])), step


def test_speculative_quantile_over_consecutive_batches(ext):
    """With a `guess` buffer the select compacts, during its first pass, the keys beyond the thresholds remembered from the previous call of the
    same slot -- consecutive calibration batches of one activation then need ONE pass over the tensor.  Whatever the guess is worth (first call,
    a distribution that drifts, jumps, collapses to a constant, a tiny workspace that overflows), the results must be the exact order statistics."""
    g = torch.Generator(device='cuda').manual_seed(9)
    sizes = [401408, 150528, 5, 1 << 20, 25088, 3000]
    slots = [2, 0, 5, 1, 4, 3]
    q = 0.9999

    def batch(step):
        xs = []
        for i, n in enumerate(sizes):
            scale = (1 + i) * (1.0 + 0.02 * step)                                # slow drift
            if step == 6: scale *= 3.0                                          # jump up: too few candidates -> regular second pass
            if step == 8: scale *= 0.2                                          # jump down: too many candidates
            x = torch.randn(n, device='cuda', generator=g) * scale
            if i % 2 == 1: x = torch.relu(x)                                    # lower quantile = an exact 0 among ~n/2 zeros
            if step == 10 and i == 0: x = torch.full((n,), 2.5, device='cuda')  # constant tensor
            if step == 11 and i == 3: x = torch.randint(-2, 3, (n,), device='cuda', generator=g).float()
            xs.append(x)
        return xs

    for cap in (1 << 16, 256):
        guess = ext.Quantile_Guess_Init(len(sizes), torch.zeros(1, device='cuda'))
        ws = torch.empty(ext.Multi_Quantile_Workspace_Bytes(len(sizes), cap), dtype=torch.uint8, device='cuda')
        for step in range(13):
            xs = batch(step)
            descs = torch.tensor([[x.data_ptr(), x.numel(), s] for x, s in zip(xs, slots)], dtype=torch.int64, device='cuda')
            out = torch.zeros(len(sizes), 2, device='cuda')
            ext.Multi_Quantile_T(descs, max(sizes), q, out, 2, ws, cap, guess)
            for x, s in zip(xs, slots):
                srt = torch.sort(x)[0]; n = x.numel()
                ia = int(min(max(np.rint(np.float32(n) * np.float32(q)), 0), n - 1)); ib = int(min(max(np.rint(np.float32(n) * (np.float32(1) - np.float32(q))), 0), n - 1))
                assert torch.equal(out[s], torch.stack([srt[ia], srt[ib]])), (cap, step, n, out[s], srt[ia], srt[ib])
        gk = guess.view(len(sizes), 2, 4)
        assert bool((gk[:, :, 3] == 0).all())                                   # layout: {threshold, last key, margin, 0} per side


def test_isotone_top2_bottom2(ext, ref, rec):
    g = torch.Generator(device='cuda').manual_seed(1)
    for n in (1, 2, 5, 1000, 100003):
        x = torch.randn(n, device='cuda', generator=g)
        got = ext.Isotone_T(x)
        s = torch.sort(x)[0]
        want = torch.stack([s[-1], s[-2], s[0], s[1]]) if n > 1 else torch.stack([s[0]] * 4)
        assert torch.equal(got, want), n
        if n > 1:
            rec.bits(f'Isotone_T n {n}', got, lambda: ref.Isotone_T(x))


def test_percentile_observer_end_to_end(ext):
    from ppq_b200 import LinearQuantizationConfig, QuantizationStates
    from ppq_b200.observer import Observer
    g = torch.Generator(device='cuda').manual_seed(2)
    data = [torch.randn(4, 16, 28, 28, device='cuda', generator=g) for _ in range(4)]
    cfg = LinearQuantizationConfig(symmetrical=True, calibration='percentile')
    ob = Observer(cfg)
    for x in data: ob.observe(x)
    ob.render_quantization_config()
    assert cfg.state == QuantizationStates.ACTIVATED
    pairs = []
    for x in data:
        s = torch.sort(x.flatten())[0]; n = s.numel()
        pairs.append(torch.stack([s[int(np.rint(np.float32(n) * np.float32(0.9999)))], s[int(np.rint(np.float32(n) * (np.float32(1) - np.float32(0.9999))))]]))
    m = torch.stack(pairs).float().mean(dim=0).cpu()
    want = 2 * max(abs(m[0].item()), abs(m[1].item())) / 255
    assert cfg.scale.item() == np.float32(want) and cfg.offset.item() == 0


def lsq_reference(value, dy, scale, offset, qmin, qmax, c=None):
    """tests/test_cuda_kernel.py:67-79 / 99-114 (the reference's own torch formula)."""
    if c is not None:
        shape = [1 if a != c else -1 for a in range(value.ndim)]
        scale, offset = scale.view(shape), offset.view(shape)
    qt = torch.round(value / scale) + offset
    cl = qt.clip(qmin, qmax)
    dx = torch.where(cl != qt, torch.zeros_like(dy), dy)
    ds = torch.where(cl == qt, (((qt - offset) * scale) - value) * dy / scale, torch.zeros_like(dy))
    ds = ds + torch.where(qt > qmax, (qmax - offset) * dy, torch.zeros_like(dy))
    ds = ds + torch.where(qt < qmin, (qmin - offset) * dy, torch.zeros_like(dy))
    return dx, ds


def test_lsq_backward_t_and_c(ext, ref, rec):
    g = torch.Generator(device='cuda').manual_seed(3)
    for shape, c in (([1, 1, 1, 1], 1), ([5, 12, 13, 4], 1), ([12, 74, 15, 41], 1), ([501, 7, 73, 1], 0), ([10, 10, 14, 47], 3), ([8192 * 3], 0)):
        for sym in (True, False):
            t = torch.rand(shape, device='cuda', generator=g) * 50
            dy = torch.rand(shape, device='cuda', generator=g)
            s = torch.rand(1, device='cuda', generator=g) + 0.01
            o = torch.zeros(1, device='cuda') if sym else torch.randint(0, 255, (1,), device='cuda', generator=g).float()
            gx, gs = ext.QuantizeTensor_LT_B(t, s, o, dy, 0, 255, 0)
            dx, ds = lsq_reference(t, dy, s, o, 0, 255)
            assert torch.equal(gx, dx), (shape, sym)
            assert close(gs, (ds.double().sum() / sqrt(t.numel() * 255)).float().view(1), rtol=1e-3), (shape, sym)
            key = f'LT_B {shape} sym {sym}'
            rec.bits(key + ' grad_x', gx, lambda: ref.QuantizeTensor_LT_B(t, s, o, dy, 0, 255, 0)[0])
            # the reference kernel block-reduces inside `if (index < N)` with __syncthreads (linear.cu:252-281): its grad_s is only
            # well defined when N is a multiple of the 1024-thread block
            if t.numel() % 1024 == 0: rec.values(key + ' grad_s', gs, lambda: ref.QuantizeTensor_LT_B(t, s, o, dy, 0, 255, 0)[1], rtol=1e-3, atol=1e-6)
            if len(shape) > 1:
                C = shape[c]
                sc = torch.rand(C, device='cuda', generator=g) + 0.01
                oc = torch.zeros(C, device='cuda') if sym else torch.randint(0, 255, (C,), device='cuda', generator=g).float()
                gx, gs = ext.QuantizeTensor_LC_B(t, sc, oc, dy, 0, 255, 0, c)
                dx, ds = lsq_reference(t, dy, sc, oc, 0, 255, c)
                assert torch.equal(gx, dx), (shape, sym, 'C')
                want = ds.double().transpose(0, c).flatten(1).sum(dim=-1) / sqrt(t.numel() * 255)      # the kernel's factor is rsqrt(N * qmax) (linear.cu:402)
                assert close(gs, want.float(), rtol=1e-3, atol=1e-5), (shape, sym, 'C')
                key = f'LC_B {shape} axis {c} sym {sym}'
                rec.bits(key + ' grad_x', gx, lambda: ref.QuantizeTensor_LC_B(t, sc, oc, dy, 0, 255, 0, c)[0])
                rec.values(key + ' grad_s', gs, lambda: ref.QuantizeTensor_LC_B(t, sc, oc, dy, 0, 255, 0, c)[1], rtol=1e-3, atol=1e-5)


def test_float_backward(ext, ref, rec):
    g = torch.Generator(device='cuda').manual_seed(4)
    x = torch.randn(1024 * 64, device='cuda', generator=g) * 200          # sizes on which the reference kernel's block-wide syncs are safe
    dy = torch.rand(x.shape, device='cuda', generator=g)
    s, o = torch.tensor([0.5], device='cuda'), torch.tensor([0.0], device='cuda')
    gx, gs = ext.QuantizeTensor_FT_B(x, s, o, dy, 4, 3, -448.0, 448.0, 0)
    u = x / s
    sat = (u > 449) | (u < -449)          # the backward kernel quantises with the clip range widened by one (floating.cu:157-158)
    assert torch.equal(gx, torch.where(sat, torch.zeros_like(dy), dy))
    rec.bits('FT_B grad_x', gx, lambda: ref.QuantizeTensor_FT_B(x, s, o, dy, 4, 3, -448.0, 448.0, 0)[0])
    rec.values('FT_B grad_s', gs, lambda: ref.QuantizeTensor_FT_B(x, s, o, dy, 4, 3, -448.0, 448.0, 0)[1], rtol=2e-3, atol=1e-6)
    xc = x.view(8, 8, 1024)
    sc = 2.0 ** torch.randint(-3, 3, (8,), device='cuda', generator=g).float(); oc = torch.zeros(8, device='cuda')
    gx, gs = ext.QuantizeTensor_FC_B(xc, sc, oc, dy.view(8, 8, 1024), 4, 3, -448.0, 448.0, 0, 1)
    rec.bits('FC_B grad_x', gx, lambda: ref.QuantizeTensor_FC_B(xc, sc, oc, dy.view(8, 8, 1024), 4, 3, -448.0, 448.0, 0, 1)[0])
    rec.values('FC_B grad_s', gs, lambda: ref.QuantizeTensor_FC_B(xc, sc, oc, dy.view(8, 8, 1024), 4, 3, -448.0, 448.0, 0, 1)[1], rtol=2e-3, atol=1e-5)


def test_tensor_clip_and_rounding_loss(ext, ref, rec):
    g = torch.Generator(device='cuda').manual_seed(5)
    for shape, c in (([7], 0), ([5, 12, 13, 4], 1), ([64, 32, 3, 3], 0), ([3, 1000], 1)):
        v = torch.randn(shape, device='cuda', generator=g)
        r = torch.randn(shape, device='cuda', generator=g)
        lim = torch.rand(1, device='cuda', generator=g)
        want = torch.minimum(torch.maximum(v, r - lim), r + lim)
        assert torch.equal(ext.TensorClip_T(v, r, lim), want), shape
        C = shape[c]
        limc = torch.rand(C, device='cuda', generator=g)
        view = [1 if a != c else -1 for a in range(len(shape))]
        wantc = torch.minimum(torch.maximum(v, r - limc.view(view)), r + limc.view(view))
        assert torch.equal(ext.TensorClip_C(v, r, limc, c), wantc), shape
        s = torch.rand(1, device='cuda', generator=g) * 0.1 + 0.01; o = torch.tensor([3.0], device='cuda')
        sc = torch.rand(C, device='cuda', generator=g) * 0.1 + 0.01; oc = torch.randint(-3, 3, (C,), device='cuda', generator=g).float()
        dyy = torch.tensor([0.7], device='cuda')
        loss_t, loss_c = ext.RoundingLoss_LT(v, s, o, -128, 127, 0), ext.RoundingLoss_LC(v, sc, oc, -128, 127, c, 0)
        gt, gc = ext.RoundingLoss_LT_B(v, dyy, s, o, -128, 127, 0), ext.RoundingLoss_LC_B(v, dyy, sc, oc, -128, 127, c, 0)
        # torch restatement of train.cu:125-141
        q = torch.clamp(torch.round(v / s) + o, -128, 127); deq = (q - o) * s
        clipped = (v > s * (127 - o)) | (v < s * (-128 - o))
        assert close(loss_t, (torch.where(clipped, torch.zeros_like(v), (deq - v).abs()).double().sum() / sqrt(v.numel())).float().view(1), rtol=1e-4)
        assert torch.equal(gt, torch.where(clipped, torch.zeros_like(v), torch.where(v > deq, 1.0, -1.0) * dyy) / torch.sqrt(torch.tensor(float(v.numel()), device='cuda')))
        key = f'{shape} axis {c}'
        rec.bits('TensorClip_T ' + key, ext.TensorClip_T(v, r, lim), lambda: ref.TensorClip_T(v, r, lim))
        rec.bits('TensorClip_C ' + key, ext.TensorClip_C(v, r, limc, c), lambda: ref.TensorClip_C(v, r, limc, c))
        rec.values('RoundingLoss_LT ' + key, loss_t, lambda: ref.RoundingLoss_LT(v, s, o, -128, 127, 0), rtol=1e-4, atol=1e-6)
        rec.values('RoundingLoss_LC ' + key, loss_c, lambda: ref.RoundingLoss_LC(v, sc, oc, -128, 127, c, 0), rtol=1e-4, atol=1e-6)
        rec.bits('RoundingLoss_LT_B ' + key, gt, lambda: ref.RoundingLoss_LT_B(v, dyy, s, o, -128, 127, 0))
        rec.bits('RoundingLoss_LC_B ' + key, gc, lambda: ref.RoundingLoss_LC_B(v, dyy, sc, oc, -128, 127, c, 0))


def test_culsq_autograd_functions(ext):
    """CuLSQ_LT / _LC (algorithm/training.py:17-90) through autograd: grad wrt the tensor is the clip-masked STE, grad wrt the scale is the LSQ term."""
    from ppq_b200.core import RoundingPolicy
    from ppq_b200.qfunction import CuLSQ_LC, CuLSQ_LT
    g = torch.Generator(device='cuda').manual_seed(9)
    x = (torch.rand(6, 8, 16, 16, device='cuda', generator=g) * 40).requires_grad_()
    s = torch.tensor([0.11], device='cuda', requires_grad=True); o = torch.tensor([3.0], device='cuda')
    y = CuLSQ_LT.apply(x, s, o, 0, 255, RoundingPolicy.ROUND_HALF_EVEN)
    w = torch.rand(y.shape, device='cuda', generator=g)
    (y * w).sum().backward()
    dx, ds = lsq_reference(x.detach(), w, s.detach(), o, 0, 255)
    assert torch.equal(x.grad, dx) and close(s.grad, (ds.double().sum() / sqrt(x.numel() * 255)).float().view(1), rtol=1e-3)
    x2 = x.detach().clone().requires_grad_()
    sc = (torch.rand(8, device='cuda', generator=g) * 0.2 + 0.05).requires_grad_(); oc = torch.zeros(8, device='cuda')
    y = CuLSQ_LC.apply(x2, sc, oc, 1, -128, 127, RoundingPolicy.ROUND_HALF_EVEN)
    (y * w).sum().backward()
    dx, ds = lsq_reference(x2.detach(), w, sc.detach(), oc, -128, 127, 1)
    assert torch.equal(x2.grad, dx)
    assert close(sc.grad, (ds.double().transpose(0, 1).flatten(1).sum(dim=-1) / sqrt(x2.numel() * 127)).float(), rtol=1e-3, atol=1e-5)
