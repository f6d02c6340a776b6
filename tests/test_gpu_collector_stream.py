"""The multi-tensor collectors (Multi_MinMax_T, Multi_Histogram_T) against the single-tensor kernels, the CPU oracle and the kernels they
replaced (variant 1 of the "minmax" / "multi_histogram" keys), bit for bit, on ragged tables: bench's own activation sets, unaligned bases,
odd lengths, one huge tensor among tiny ones, shared statistics slots and special values."""
import numpy as np
import pytest
import torch

from bench import WORKLOADS, numel

pytestmark = pytest.mark.gpu
BINS = 4096


@pytest.fixture(scope='module')
def ext():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from ppq_b200.ffi import extension
    return extension()


def assert_same_floats(got, want, msg):
    g, w = np.asarray(got, np.float32).reshape(-1), np.asarray(want, np.float32).reshape(-1)
    same = (g.view(np.uint32) == w.view(np.uint32)) | (np.isnan(g) & np.isnan(w))
    assert same.all(), f'{msg}: {g[~same][:4]} vs {w[~same][:4]}'


def descs_of(tensors, slots):
    return torch.tensor([[t.data_ptr(), t.numel(), s] for t, s in zip(tensors, slots)], dtype=torch.int64, device='cuda')


def multi(ext, tensors, slots, nslots, hs=None, clip=True, bins=BINS):
    """Both multi-tensor launches over one table: min/max arena, hist_scale (derived unless given), histogram arena."""
    d = descs_of(tensors, slots)
    max_n = max(t.numel() for t in tensors)
    mm = torch.empty(nslots, 2, device='cuda'); mm[:, 0] = float('inf'); mm[:, 1] = float('-inf')
    ext.Multi_MinMax_T(d, max_n, mm)
    if hs is None: hs = ext.Hist_Scale_From_MinMax(mm, True, bins)
    hist = torch.zeros(nslots, bins, dtype=torch.int32, device='cuda')
    ext.Multi_Histogram_T(d, max_n, hs, clip, hist, bins)
    torch.cuda.synchronize()
    return mm, hs, hist


def single(ext, tensors, slots, nslots, hs, clip=True, bins=BINS):
    """The same statistics from one single-tensor launch per tensor."""
    mm = torch.empty(nslots, 2, device='cuda'); mm[:, 0] = float('inf'); mm[:, 1] = float('-inf')
    hist = torch.zeros(nslots, bins, dtype=torch.int32, device='cuda')
    for t, s in zip(tensors, slots):
        ext.MinMax_T(t, mm[s])
        ext.Histogram_T_DeviceScale(t, hs[s:s + 1], clip, hist[s])
    torch.cuda.synchronize()
    return mm, hist


def replaced(ext, *args, **kw):
    ext.set_variant('minmax', 1); ext.set_variant('multi_histogram', 1)
    try:
        return multi(ext, *args, **kw)
    finally:
        ext.set_variant('minmax', 0); ext.set_variant('multi_histogram', 0)


def check(ext, oracle, tensors, slots=None, hs=None, clip=True, bins=BINS, with_oracle=True):
    slots = list(range(len(tensors))) if slots is None else slots
    nslots = max(slots) + 1
    mm, hs, hist = multi(ext, tensors, slots, nslots, hs, clip, bins)
    mm1, hist1 = single(ext, tensors, slots, nslots, hs, clip, bins)
    assert_same_floats(mm.cpu().numpy(), mm1.cpu().numpy(), 'min/max vs single-tensor kernel')
    assert torch.equal(hist, hist1), 'histogram vs single-tensor kernel'
    mm0, hs0, hist0 = replaced(ext, tensors, slots, nslots, hs, clip, bins)
    assert_same_floats(mm.cpu().numpy(), mm0.cpu().numpy(), 'min/max vs the replaced kernel')
    assert torch.equal(hist, hist0), 'histogram vs the replaced kernel'
    if with_oracle:
        for s in range(nslots):
            xs = [t.cpu().numpy().reshape(-1) for t, k in zip(tensors, slots) if k == s]
            if not xs: continue
            x = np.concatenate(xs)
            lo, hi = oracle.minmax_t(x)
            got = mm[s].cpu().numpy()                                       # by value, as test_gpu_parity does: the oracle's zero may differ in sign
            assert all(g == w or (g != g and w != w) for g, w in zip(got, (lo, hi))), f'min/max of slot {s} vs oracle: {got} vs {(lo, hi)}'
            want = oracle.histogram_t(x, hs[s].item(), bins, clip)
            assert np.array_equal(hist[s].cpu().numpy(), want), f'histogram of slot {s} vs oracle'
    return mm, hist


@pytest.mark.parametrize('workload', ['resnet50', 'yolov5s'])
def test_bench_tables_batch2(ext, oracle, workload):
    acts, _ = WORKLOADS[workload]['table']()
    g = torch.Generator(device='cuda').manual_seed(7)
    ts = []
    for i, shp in enumerate(acts):
        t = torch.randn((2,) + tuple(shp), device='cuda', generator=g)
        if i % 2 == 1: t.relu_()
        ts.append(t)
    assert sum(t.numel() for t in ts) == 2 * sum(numel(s) for s in acts)
    check(ext, oracle, ts)


def test_unaligned_bases_and_odd_lengths(ext, oracle):
    r = np.random.RandomState(3)
    lengths = [1, 3, 5, 7, 9, 13, 31, 33, 255, 1001, 4099, 65537, 100003, 1 << 20, (1 << 20) + 5]
    buf = torch.from_numpy((r.standard_normal(sum(lengths) + 4 * len(lengths)) * 3).astype(np.float32)).cuda()
    ts, pos = [], 0
    for i, n in enumerate(lengths):
        off = (i % 3) + 1                                                   # bases 4, 8 and 12 bytes past a 16-byte boundary
        ts.append(buf[pos + off: pos + off + n]); pos += off + n
    for clip in (True, False):
        check(ext, oracle, ts, clip=clip)
    check(ext, oracle, ts[::-1], bins=50)


def test_one_huge_tensor_among_tiny_ones(ext, oracle):
    r = np.random.RandomState(5)
    tiny = [torch.from_numpy(r.standard_normal(n).astype(np.float32)).cuda() for n in (1, 2, 3, 4, 5, 6, 7, 8, 17, 100) * 5]
    huge = torch.randn(1 << 25, device='cuda', generator=torch.Generator(device='cuda').manual_seed(5)).relu_()
    check(ext, oracle, tiny[:25] + [huge] + tiny[25:])


def test_shared_slots(ext, oracle):
    r = np.random.RandomState(9)
    ts = [torch.from_numpy((r.standard_normal(n) * (i + 1)).astype(np.float32)).cuda() for i, n in enumerate((70001, 5, 401408, 3, 200000))]
    check(ext, oracle, ts, slots=[0, 1, 0, 2, 1])


def test_special_values(ext, oracle):
    r = np.random.RandomState(11)
    x = (r.standard_normal(300007) * 2).astype(np.float32)
    nan = x.copy(); nan[123456] = np.nan
    inf = x.copy(); inf[7] = np.inf; inf[300000] = -np.inf
    zeros = np.zeros(200003, np.float32)
    negz = np.full(50001, -0.0, np.float32)
    mixz = np.where(r.rand(40000) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
    relu = np.maximum(x, 0)
    ts = [torch.from_numpy(a).cuda() for a in (nan, inf, zeros, negz, mixz, relu, x)]
    hs = torch.full((len(ts),), 5.0 / BINS, device='cuda')                   # finite scales: NaN / inf tensors still bin
    for clip in (True, False):
        check(ext, oracle, ts, hs=hs, clip=clip)
    mm, _ = check(ext, oracle, ts)                                           # derived scales (NaN / inf / 0 for some slots)
    assert np.isnan(mm[0].cpu().numpy()).all(), 'a NaN poisons both slots'


def test_multi_weight_table_ragged_epc(ext, oracle):
    from ppq_b200.calibration import MultiWeightQuantizer
    r = np.random.RandomState(13)
    shapes = [(64, 3, 7, 7), (64, 64, 1, 1), (64, 64, 3, 3), (256, 64, 1, 1), (1000, 2048), (5, 3, 7, 7), (3, 147)]
    ws = [torch.from_numpy((r.standard_normal(s) * 0.05).astype(np.float32)).cuda() for s in shapes]
    scales = [(w.abs().amax(dim=tuple(range(1, w.dim()))) / 127).clamp_min(1e-8) for w in ws]
    offsets = [torch.zeros_like(s) for s in scales]
    outs = MultiWeightQuantizer(ws, scales, offsets, channel_axis=0)()
    for w, s, o, y in zip(ws, scales, offsets, outs):
        assert torch.equal(y, ext.QuantizeTensor_LC(w, s, o, -128, 127, 0, 0)), tuple(w.shape)
        want = oracle.linear_quant_c(w.cpu().numpy(), s.cpu().numpy(), o.cpu().numpy(), 0, -128, 127, 0)
        assert np.array_equal(y.cpu().numpy().view(np.uint32), want.view(np.uint32)), tuple(w.shape)
