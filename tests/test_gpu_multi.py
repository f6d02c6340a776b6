"""Multi-GPU / multi-device tests (need >= 2 visible GPUs: `gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`; skipped on a 1-GPU box).

  * BASELINE config 5's flow over REAL NCCL: two ranks, one per GPU, each calibrating its sample shard of a YOLOv5s-like activation set
    through ArenaCalibrator (multi-tensor launches, the two all-reduces of SURVEY 8e) -- all four observer algorithms -- must reproduce the
    single-process statistics and scales bit for bit;
  * one process driving TWO devices: the kernels that opt in to > 48 KB of dynamic shared memory (KL search at 4096 bins, the TMA-staged
    fake-quant variant) and every persistent grid (sm_count()) must work on the second device too (VERDICT r1: per-device function attributes).
"""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(3, 160, 160), (32, 80, 80), (64, 40, 40), (128, 20, 20), (256, 10, 10), (255, 20, 20), (255, 10, 10)]
METHODS = ('kl', 'minmax', 'mse', 'percentile')


def _free_port():
    s = socket.socket(); s.bind(('127.0.0.1', 0)); p = s.getsockname()[1]; s.close(); return p


def _samples(device, n=12):
    g = torch.Generator(device=device).manual_seed(5)
    return [[(torch.randn((2,) + s, device=device, generator=g) * (1 + i % 3)).relu_() if k % 2 else torch.randn((2,) + s, device=device, generator=g)
             for k, s in enumerate(SHAPES)] for i in range(n)]


def _calibrate(cal, samples):
    while True:
        for smp in samples:
            cal.begin_batch()
            cal.observe(smp)
        if cal.end_phase(): break
    return cal


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from ppq_b200.calibration import ArenaCalibrator, shard_indices
    os.environ['MASTER_ADDR'] = '127.0.0.1'; os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    dev = torch.device('cuda', rank)
    samples = _samples(dev)                                              # the same global sample list on every rank (same seed); each keeps its shard
    mine = [samples[i] for i in shard_indices(len(samples), rank, world)]
    out = {}
    for method in METHODS:
        cal = _calibrate(ArenaCalibrator(len(SHAPES), dev, method=method), mine)
        out[method] = {'scale': cal.scale.cpu(), 'offset': cal.offset.cpu(), 'minmax': cal.minmax.cpu(), 'hist': cal.hist.cpu()}
    torch.save(out, os.path.join(out_dir, f'nccl{rank}.pt'))
    dist.barrier()
    dist.destroy_process_group()


def test_config5_two_ranks_over_nccl_equal_the_single_process_calibration(tmp_path):
    if torch.cuda.device_count() < 2: pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    from ppq_b200.calibration import ArenaCalibrator
    world, port = 2, _free_port()
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    got = [torch.load(tmp_path / f'nccl{r}.pt') for r in range(world)]
    dev = torch.device('cuda', 0)
    samples = _samples(dev)
    for method in METHODS:
        full = _calibrate(ArenaCalibrator(len(SHAPES), dev, method=method), samples)
        for r in range(world):
            g = got[r][method]
            assert torch.equal(g['scale'], full.scale.cpu()) and torch.equal(g['offset'], full.offset.cpu()), (method, r, g['scale'], full.scale)
            if method != 'percentile': assert torch.equal(g['minmax'], full.minmax.cpu()), (method, r)
            if method in ('kl', 'mse'): assert torch.equal(g['hist'], full.hist.cpu()), (method, r)


def test_one_process_two_devices():
    if torch.cuda.device_count() < 2: pytest.skip('needs 2 GPUs')
    from ppq_b200.ffi import extension
    ext = extension()
    res = []
    for d in (0, 1):
        dev = torch.device('cuda', d)
        g = torch.Generator(device=dev).manual_seed(3)
        x = torch.randn(4, 64, 56, 56, device=dev, generator=g)
        mm = torch.empty(2, device=dev); ext.MinMax_Init(mm[0:1], mm[1:2]); ext.MinMax_T(x, mm)
        hs = ext.Hist_Scale_From_MinMax(mm.view(1, 2), True, 4096)
        hist = torch.zeros(4096, dtype=torch.int32, device=dev)
        ext.Histogram_T_DeviceScale(x, hs, True, hist)
        scale, best = ext.KL_Search(hist.view(1, -1), 4096, hs, mm.view(1, 2), 8, False, 1e-8)       # > 48 KB of dynamic shared memory
        s, o = torch.tensor([0.05], device=dev), torch.tensor([0.0], device=dev)
        y0 = ext.QuantizeTensor_LT(x, s, o, -128, 127, 0)
        ext.set_variant('linear_quant_t', 1)                                                          # TMA-staged variant: opt-in smem as well
        try: y1 = ext.QuantizeTensor_LT(x, s, o, -128, 127, 0)
        finally: ext.set_variant('linear_quant_t', 0)
        torch.cuda.synchronize(dev)
        assert torch.equal(y0, y1)
        q = ext.Quantile_T(x, 0.9999)
        res.append((scale.cpu(), best.cpu(), hist.cpu(), y0.cpu(), q.cpu()))
    for a, b in zip(res[0], res[1]): assert torch.equal(a, b)                                         # same seed, same results on both devices
