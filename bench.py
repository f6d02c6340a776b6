#!/usr/bin/env python
"""bench.py -- calibration / fake-quant throughput of the PPQ quantization-simulation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload resnet50|yolov5s] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): ResNet-50 RuntimeCalibrationPass, minmax + KL-histogram, 512 synthetic 3x224x224 samples per GPU,
calibration batch B = 32 (the reference's ImageNet calibration batch: ppq/samples/QuantZoo/QuantZoo_Imagenet.py:21).
One "step" = ONE WHOLE CALIBRATION of the GPU's 512-sample share through the hot path:
    phase 1   16 batches x { per-channel INT8 fake-quant of the 54 Conv/Gemm weights (the executor re-quantises weights every forward:
              executor/torch.py:516-518) + fused min/max over the observed activation tensors of the forward }
    exchange  all-reduce(MAX) of {-min, max}; hist_scale on the device
    phase 2   16 batches x { the same weight fake-quant + 4096-bin histogram over the same activation tensors }
    exchange  all-reduce(SUM) of the histogram arena; on-device KL scale search
so both exchange steps and the search are inside every timed step.  Conv/Gemm forward execution itself is outside the path (SURVEY.md
§8: stays in torch/cuDNN), so `value` replays the activation tensor set of the network (shapes traced from torchvision resnet50 after BN
fusion; synthetic randn / relu(randn) values) resident in HBM; `e2e` runs the real thing -- images from pinned host memory, torch forward
of the network with our hooks, scales read back -- through ppq_b200's public API.

`--workload yolov5s` (BASELINE.json configs[4]) replays the activation set of the public YOLOv5s architecture at 3x640x640 (batch 16,
512 samples per GPU = 4096 samples on 8 GPUs); its e2e arm runs the architecture itself (bench_models.YOLOv5s, random init).

Prints ONE JSON line (see the task contract): metric/value (imgs/s, whole job), roofline of the dominant kernel, cpu_baseline (the
reference's USING_CUDA_KERNEL=False CPU path restated in oracle/ with torch CPU ops, timed on this host), clocks, e2e, gpu_launches,
per-rank timing table, plus `fakequant` (LinearQuant elems/s and HBM fraction over 1x3x224x224 ... 1x2048x64x64).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'calibration_imgs_per_s'
UNIT = 'imgs/s'
BINS = 4096
SAMPLES_PER_GPU = 512
VENDOR_HBM_GBS = 8000.0          # NVIDIA's B200 HBM3e figure (BASELINE.md §3 asks for both denominators)


# ------------------------------------------------------------------------------------------------ workload definition
def resnet50_tensor_table():
    """Per-image shapes of the observed activations (model input + output of every Conv / ReLU call site / pool / fc, BatchNorm
    folded into the convs as PPQ does at load: core/common.py:41) and the shapes of the Conv/Gemm weights.  Traced on the meta
    device; falls back to the recorded table if torchvision is unavailable."""
    try:
        import torchvision
        m = torchvision.models.resnet50(weights=None).eval().to('meta')
        acts, weights = [(3, 224, 224)], []
        hooks = []
        for mod in m.modules():
            if isinstance(mod, (torch.nn.Conv2d, torch.nn.ReLU, torch.nn.MaxPool2d, torch.nn.AdaptiveAvgPool2d, torch.nn.Linear)):
                hooks.append(mod.register_forward_hook(lambda _m, _i, o: acts.append(tuple(o.shape[1:]))))
            if isinstance(mod, (torch.nn.Conv2d, torch.nn.Linear)):
                weights.append(tuple(mod.weight.shape))
        with torch.no_grad():
            m(torch.empty(1, 3, 224, 224, device='meta'))
        for h in hooks: h.remove()
        return acts, weights
    except Exception:
        acts = [(3, 224, 224), (64, 112, 112), (64, 112, 112), (64, 56, 56)]
        weights = [(64, 3, 7, 7)]
        cfg = [(64, 256, 56, 3), (128, 512, 28, 4), (256, 1024, 14, 6), (512, 2048, 7, 3)]
        cin = 64
        for mid, out, hw, blocks in cfg:
            for b in range(blocks):
                first = b == 0
                hw_in = hw * 2 if (first and mid != 64) else hw
                acts += [(mid, hw_in, hw_in), (mid, hw_in, hw_in), (mid, hw, hw), (mid, hw, hw), (out, hw, hw)]
                weights += [(mid, cin, 1, 1), (mid, mid, 3, 3), (out, mid, 1, 1)]
                if first:
                    acts.append((out, hw, hw)); weights.append((out, cin, 1, 1))
                acts.append((out, hw, hw))
                cin = out
        acts += [(2048, 1, 1), (1000,)]
        weights.append((1000, 2048))
        return acts, weights


def yolov5s_tensor_table(size=640):
    """Activation / weight shapes of the public YOLOv5s (v6.0, width 0.5, depth 0.33) at size x size, as the reference would observe them
    (ppq/samples/Yolo/yolo_5.py:10-13 convention: 3x640x640 inputs): the output of every Conv+SiLU (the reference fuses Conv-Sigmoid-Mul,
    optim/refine.py:210-239), of every shortcut Add, Concat and Upsample, and the three detection convolutions.  From general knowledge of
    the architecture -- the model file is not part of the reference (SURVEY.md §8d config 5)."""
    acts, weights = [(3, size, size)], []

    def conv(cin, cout, k, hw):
        weights.append((cout, cin, k, k)); acts.append((cout, hw, hw)); return cout

    def c3(cin, cout, n, hw, shortcut=True):
        h = cout // 2
        conv(cin, h, 1, hw); conv(cin, h, 1, hw)
        for _ in range(n):
            conv(h, h, 1, hw); conv(h, h, 3, hw)
            if shortcut: acts.append((h, hw, hw))                     # Add
        acts.append((2 * h, hw, hw))                                  # Concat
        return conv(2 * h, cout, 1, hw)
    s = size
    c = conv(3, 32, 6, s // 2); c = conv(c, 64, 3, s // 4); c = c3(c, 64, 1, s // 4)
    c = conv(c, 128, 3, s // 8); p3 = c3(c, 128, 2, s // 8)
    c = conv(p3, 256, 3, s // 16); p4 = c3(c, 256, 3, s // 16)
    c = conv(p4, 512, 3, s // 32); c = c3(c, 512, 1, s // 32)
    conv(c, 256, 1, s // 32); acts.append((1024, s // 32, s // 32)); c = conv(1024, 512, 1, s // 32)          # SPPF (max-pools are passive)
    h10 = conv(c, 256, 1, s // 32); acts.append((256, s // 16, s // 16)); acts.append((512, s // 16, s // 16))  # upsample, concat with p4
    c3(512, 256, 1, s // 16, shortcut=False)
    h14 = conv(256, 128, 1, s // 16); acts.append((128, s // 8, s // 8)); acts.append((256, s // 8, s // 8))    # upsample, concat with p3
    o3 = c3(256, 128, 1, s // 8, shortcut=False)
    conv(o3, 128, 3, s // 16); acts.append((256, s // 16, s // 16)); o4 = c3(256, 256, 1, s // 16, shortcut=False)
    conv(o4, 256, 3, s // 32); acts.append((512, s // 32, s // 32)); o5 = c3(512, 512, 1, s // 32, shortcut=False)
    for ch, hw in ((o3, s // 8), (o4, s // 16), (o5, s // 32)): conv(ch, 255, 1, hw)                           # Detect
    del h10, h14
    return acts, weights


WORKLOADS = {
    'resnet50': dict(table=resnet50_tensor_table, batch=32, image=(3, 224, 224),
                     name='ResNet-50 RuntimeCalibrationPass (minmax + KL 4096-bin histogram), 512 synthetic 3x224x224 samples per GPU'),
    'yolov5s': dict(table=yolov5s_tensor_table, batch=16, image=(3, 640, 640),
                    name='YOLOv5s RuntimeCalibrationPass (minmax + KL 4096-bin histogram), 512 synthetic 3x640x640 samples per GPU'),
}


def numel(shape):
    n = 1
    for d in shape: n *= d
    return n


class Workload:
    """R rotating sets of synthetic activation tensors for one calibration batch + the network's weights, resident in HBM."""

    def __init__(self, device, kind, batch, rotate, seed=0):
        self.kind = kind
        self.acts, self.weights = WORKLOADS[kind]['table']()
        self.batch, self.device = batch, device
        g = torch.Generator(device=device).manual_seed(seed)
        self.sets = []
        for r in range(rotate):
            ts = []
            for i, shp in enumerate(self.acts):
                t = torch.randn((batch,) + shp, device=device, generator=g)
                if i % 2 == 1: t.relu_()                                  # post-ReLU tensors: half of the mass in bin 0
                ts.append(t)
            self.sets.append(ts)
        self.w = [torch.randn(shp, device=device, generator=g) * 0.05 for shp in self.weights]
        self.w_scale = [(w.abs().amax(dim=tuple(range(1, w.dim()))) / 127).clamp_min(1e-8).contiguous() for w in self.w]
        self.w_offset = [torch.zeros_like(s) for s in self.w_scale]
        self.act_elems = sum(numel(s) for s in self.acts) * batch
        self.w_elems = sum(numel(s) for s in self.weights)

    def bytes_per_batch(self):
        # algorithmic HBM bytes of one calibration batch: 4 B/elem per collector pass (2 passes) + 8 B/elem per weight fake-quant (2 forwards)
        return 2 * 4 * self.act_elems + 2 * 8 * self.w_elems


def workload_config(args, wl_acts, wl_weights, batches_per_step):
    """The `config` object: identical in the GPU arm and in the reference arm (same workload, same batch)."""
    return {'workload': WORKLOADS[args.workload]['name'], 'batch': args.batch, 'samples_per_gpu_per_step': batches_per_step * args.batch,
            'step': 'one whole two-phase calibration of the per-GPU sample share (both exchange steps + scale search inside)',
            'observed_tensors': len(wl_acts), 'observed_elems_per_image': sum(numel(s) for s in wl_acts),
            'weight_tensors': len(wl_weights), 'weight_elems': sum(numel(s) for s in wl_weights)}


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled DURING the timed region through NVML at 20 Hz (a 1 kHz poll from every rank contended for the
    driver lock with the launch loop: round-1 N=8 straggler), rank 0 only."""

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.err, self.period = index, [], False, None, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                                            # noqa: BLE001
            self.nv, self.err = None, f'{type(e).__name__}: {e}'

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            parts = [p for p in vis.split(',') if p.strip()]
            if i < len(parts) and parts[i].strip().isdigit(): return int(parts[i])
        return i

    def sample(self):
        nv = self.nv
        self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                             nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons')
                             else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))

    def run(self):
        if self.nv is None: return
        while not self.stop_flag:
            try:
                self.sample()
            except Exception as e:                                        # noqa: BLE001
                self.err = f'{type(e).__name__}: {e}'
                break
            time.sleep(self.period)

    def summary(self):
        if not self.samples: return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable: ' + str(self.err)]}
        sm = sorted(s[0] for s in self.samples)
        bits = 0
        for s in self.samples: bits |= int(s[1])
        names = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap', 0x80: 'hw_power_brake_slowdown'}
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': self.max_sm, 'reasons': sorted(n for b, n in names.items() if bits & b),
                'samples': len(self.samples), 'period_s': self.period}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs: device-to-device copy, read + write)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def stats(v):
    v = sorted(v)
    return {'min': round(v[0], 4), 'median': round(v[len(v) // 2], 4), 'max': round(v[-1], 4)}


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, rank, world, local_rank):
    from ppq_b200.calibration import ArenaCalibrator, MultiWeightQuantizer
    from ppq_b200.ffi import extension
    ext = extension()
    device = torch.device('cuda', local_rank)
    torch.cuda.set_device(device)
    wl = Workload(device, args.workload, args.batch, args.rotate, seed=1234 + rank)
    T = len(wl.acts)
    nb = max(1, SAMPLES_PER_GPU // args.batch)                    # calibration batches per step (= per whole calibration)
    cal = ArenaCalibrator(T, device, bins=BINS, num_of_bits=8, method='kl')
    stream = torch.cuda.current_stream()
    hist_events, mm_events, launches, last_weights = [], [], [0], [None]
    wq = MultiWeightQuantizer(wl.w, wl.w_scale, wl.w_offset, channel_axis=0)

    def weights_pass():
        if args.per_tensor_weight_launches:
            out = [ext.QuantizeTensor_LC(w, s, o, -128, 127, 0, 0) for w, s, o in zip(wl.w, wl.w_scale, wl.w_offset)]
            launches[0] += len(wl.w)
            return out
        launches[0] += 1
        return wq()                                               # all weights, one launch

    def calibrate(timed):
        """One step: a whole two-phase calibration of this GPU's 512-sample share."""
        cal.reset()
        for k in range(nb):                                     # phase 1
            weights_pass()
            if timed: e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(stream)
            cal.observe(wl.sets[k % args.rotate])
            if timed: e1.record(stream); mm_events.append((e0, e1))
        cal.end_phase()
        for k in range(nb):                                     # phase 2
            wq_out = weights_pass()
            if timed: e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(stream)
            cal.observe(wl.sets[k % args.rotate])
            if timed: e1.record(stream); hist_events.append((e0, e1))
        cal.end_phase()
        last_weights[0] = wq_out
        return cal.scale

    def barrier():
        if world > 1: dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)): calibrate(False)        # W untimed warm-up steps (whole calibrations, both exchange steps included)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler is not None: sampler.start()
    cal.launches = 0; launches[0] = 0
    cal.exchange_events = {}                                    # CUDA events around the two exchange steps (SURVEY 8e scaling report)
    step_events = []
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push('timed')
    t0.record(stream)
    for _ in range(args.steps):
        a = torch.cuda.Event(enable_timing=True); a.record(stream)
        scales = calibrate(True)
        b = torch.cuda.Event(enable_timing=True); b.record(stream)
        step_events.append((a, b))
    t1.record(stream)
    torch.cuda.synchronize()
    torch.cuda.nvtx.range_pop()
    barrier()
    if sampler is not None:
        sampler.stop_flag = True
        if not sampler.samples and sampler.nv is not None:
            try: sampler.sample()
            except Exception: pass
    ms_local = t0.elapsed_time(t1)
    ms = ms_local
    h_list = [a.elapsed_time(b) for a, b in hist_events]
    m_list = [a.elapsed_time(b) for a, b in mm_events]
    s_list = [a.elapsed_time(b) for a, b in step_events]
    mine = torch.tensor([ms_local, sum(h_list) / len(h_list), sum(m_list) / len(m_list), min(h_list), max(h_list), min(m_list), max(m_list),
                         min(s_list), sorted(s_list)[len(s_list) // 2], max(s_list)], device=device)
    per_rank = [mine]
    if world > 1:
        t = torch.tensor([ms], device=device); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = t.item()
        per_rank = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(per_rank, mine)
    assert torch.isfinite(scales).all() and (scales > 0).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cal, last_weights[0])

    # ---- roofline of the dominant kernel (multi-tensor histogram; 4 B/element) from the events of the timed region
    peak, peak_src = measured_peaks()
    h_ms = sum(h_list) / len(h_list)
    m_ms = sum(m_list) / len(m_list)
    hist_gbs = 4.0 * wl.act_elems / (h_ms * 1e-3) / 1e9
    mm_gbs = 4.0 * wl.act_elems / (m_ms * 1e-3) / 1e9
    traffic = None
    try:                                                                    # dram__bytes_read + dram__bytes_write of one launch, from the committed ncu capture
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))
        if tj.get('batch') == args.batch and args.workload == 'resnet50': traffic = tj['traffic_bytes_per_launch']
    except Exception:
        pass
    roofline = {'bound': 'hbm', 'kernel': 'multi_histogram_t_kernel', 'achieved': round(hist_gbs, 1), 'peak': peak, 'unit': 'GB/s',
                'frac': round(hist_gbs / peak, 4), 'traffic': traffic, 'peak_source': peak_src,
                'peak_vendor': VENDOR_HBM_GBS, 'frac_of_vendor_peak': round(hist_gbs / VENDOR_HBM_GBS, 4), 'ms_per_launch': round(h_ms, 4),
                'algorithmic_bytes_per_launch': 4 * wl.act_elems,
                'other_kernels': {'multi_minmax_t_kernel': {'achieved': round(mm_gbs, 1), 'frac': round(mm_gbs / peak, 4),
                                                            'frac_of_vendor_peak': round(mm_gbs / VENDOR_HBM_GBS, 4), 'ms_per_launch': round(m_ms, 4)}}}
    cfg = workload_config(args, wl.acts, wl.weights, nb)
    cfg.update({'parallelism': f'dp{world} (sample-sharded, 2 all-reduces per calibration)',
                'l2_policy': f'inputs larger than L2: {args.rotate} rotating activation sets of {4 * wl.act_elems / 1e9:.2f} GB each'})
    result = {
        'metric': METRIC, 'value': round(world * args.steps * nb * args.batch / (ms * 1e-3), 1), 'unit': UNIT, 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms / args.steps, 4), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': cfg,
        'roofline': roofline,
        'gpu_launches': cal.launches + launches[0],
        'clocks': sampler.summary() if sampler is not None else None,
        'timed_region_s': round(ms * 1e-3, 4),
        'algorithmic_gbs': round(nb * wl.bytes_per_batch() / (ms / args.steps * 1e-3) / 1e9, 1),
        # the two exchange steps per calibration (this rank's view, device time incl. waiting for the slowest rank)
        'exchange_ms_per_step': {k: round(sum(a.elapsed_time(b) for a, b in v) / args.steps, 4) for k, v in cal.exchange_events.items()},
        # per-rank view of the timed region (ms): total, mean / min / max per launch of both collectors, per-step min / median / max
        'per_rank': [{'rank': r, 'total_ms': round(float(v[0]), 3), 'hist_ms': {'mean': round(float(v[1]), 4), 'min': round(float(v[3]), 4), 'max': round(float(v[4]), 4)},
                      'minmax_ms': {'mean': round(float(v[2]), 4), 'min': round(float(v[5]), 4), 'max': round(float(v[6]), 4)},
                      'step_ms': {'min': round(float(v[7]), 3), 'median': round(float(v[8]), 3), 'max': round(float(v[9]), 3)}}
                     for r, v in enumerate(per_rank)],
    }
    cal.exchange_events = None
    have_model = True
    if rank == 0:
        result['fakequant'] = fakequant_sweep(ext, device, peak) if not args.no_sweep else None
    if not args.no_e2e and have_model:
        e2e = run_e2e(args, device, world, rank)
        if rank == 0: result['e2e'] = e2e
    elif rank == 0:
        result['e2e'] = None if args.no_e2e else {'value': None, 'unit': UNIT, 'unavailable': 'activation-set replay only: the network is not in this image'}
    if rank == 0:
        result['cpu_baseline'] = cpu_baseline(args) if not args.no_cpu_baseline else None
    return result


DUMP_WEIGHT_SAMPLE = 1 << 20


def dump_outputs(out_dir, cal, weights):
    """What the last timed step handed its caller, as .npy (float32, or float64 for the int32 histogram counts): the calibrated scales and
    offsets with the statistics they came from (min/max, histogram scale, histogram arena), and a fixed sample (seed 0) of
    DUMP_WEIGHT_SAMPLE elements of the fake-quantised weights, whose ~100 MB in full would not fit the 64 MB the dump may take."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    flat = torch.cat([w.reshape(-1) for w in weights])
    idx = np.sort(np.random.RandomState(0).choice(flat.numel(), size=min(DUMP_WEIGHT_SAMPLE, flat.numel()), replace=False))
    arrays = {'scale': cal.scale.float(), 'offset': cal.offset.float(), 'minmax': cal.minmax, 'hist_scale': cal.hist_scale,
              'histogram': cal.hist.double(), 'weights_fakequant_sample': flat[torch.from_numpy(idx).to(flat.device)],
              'weights_fakequant_sample_index': torch.from_numpy(idx.astype(np.float64))}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().cpu().numpy())


def fakequant_sweep(ext, device, peak):
    """LinearQuant_T INT8 over the north-star shape range (1x3x224x224 ... 1x2048x64x64, plus BERT-sized tensors).  Per shape:
      us_per_call        the public op, eager (python -> binding -> at::empty_like -> kernel), what ppq.executor pays per fake-quant;
      kernel_us / gbs    the kernel alone: the C-ABI launch captured in a CUDA graph over rotating input AND output buffers (> L2 in total
                         for the large shapes), replayed back to back -- no host launch overhead, no allocator.
    The small shapes are L2-resident and launch-latency bound by nature: their HBM fraction is reported but means latency."""
    import ctypes
    lib = ctypes.CDLL(os.path.join(ROOT, 'ppq_b200', '_lib', 'libppq_b200.so'))
    out = []
    s, o = torch.tensor([0.05], device=device), torch.tensor([0.0], device=device)
    for shape in ((1, 3, 224, 224), (1, 512, 28, 28), (1, 256, 56, 56), (1, 1024, 14, 14), (1, 2048, 64, 64), (32, 512, 768), (32, 12, 512, 512)):
        n = numel(shape)
        nbuf = max(2, min(64, int(1.5e9 // (8 * n)) + 1))
        xs = [torch.randn(shape, device=device) for _ in range(nbuf)]
        ys = [torch.empty_like(x) for x in xs]
        outs = [None] * nbuf
        for i in range(nbuf): outs[i] = ext.QuantizeTensor_LT(xs[i], s, o, -128, 127, 0)
        reps = max(nbuf, 40)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); a.record()
        for i in range(reps): outs[i % nbuf] = ext.QuantizeTensor_LT(xs[i % nbuf], s, o, -128, 127, 0)
        b.record(); torch.cuda.synchronize()
        op_us = a.elapsed_time(b) * 1e3 / reps
        del outs
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                st = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
                for i in range(nbuf):
                    lib.ppq_b200_linear_quant_t(ctypes.c_void_p(xs[i].data_ptr()), ctypes.c_void_p(ys[i].data_ptr()), ctypes.c_int64(n),
                                                ctypes.c_void_p(s.data_ptr()), ctypes.c_void_p(o.data_ptr()), -128, 127, 0, st)
        torch.cuda.current_stream(device).wait_stream(side)
        g.replay(); torch.cuda.synchronize()
        rounds = max(1, 64 // nbuf)
        a.record()
        for _ in range(rounds): g.replay()
        b.record(); torch.cuda.synchronize()
        k_us = a.elapsed_time(b) * 1e3 / (rounds * nbuf)
        gbs = 8.0 * n / (k_us * 1e-6) / 1e9
        out.append({'shape': 'x'.join(map(str, shape)), 'elems': n, 'us_per_call': round(op_us, 2), 'kernel_us': round(k_us, 2),
                    'gelems_per_s': round(n / k_us / 1e3, 1), 'gbs': round(gbs, 1), 'frac_of_hbm_peak': round(gbs / peak, 4),
                    'frac_of_vendor_peak': round(gbs / VENDOR_HBM_GBS, 4), 'distinct_buffers': nbuf})
        del xs, ys, g
    # the executor's many small tensors, batched: 64 tensors of 1x512x28x28 (BASELINE config 1 shape) in ONE multi-tensor launch
    from ppq_b200.calibration import MultiWeightQuantizer
    xs = [torch.randn(1, 512, 28, 28, device=device) for _ in range(64 * 8)]
    qs = [MultiWeightQuantizer(xs[i * 64:(i + 1) * 64], [s] * 64, [o] * 64, channel_axis=None) for i in range(8)]     # 8 x 103 MB: rotates past L2
    for q in qs: q()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for r in range(40): qs[r % 8]()
    b.record(); torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1e3 / 40
    n = 64 * 512 * 28 * 28
    out.append({'shape': '64 x (1x512x28x28) in one multi-tensor launch', 'elems': n, 'us_per_call': round(us, 2), 'kernel_us': round(us, 2),
                'us_per_tensor_amortised': round(us / 64, 3),
                'gelems_per_s': round(n / us / 1e3, 1), 'gbs': round(8.0 * n / (us * 1e-6) / 1e9, 1),
                'frac_of_hbm_peak': round(8.0 * n / (us * 1e-6) / 1e9 / peak, 4), 'distinct_buffers': 8})
    return out


def run_e2e(args, device, world, rank):
    try:
        from ppq_b200.executor import e2e_calibration_benchmark
    except Exception as e:                                               # executor lands after the kernels; never silently fake a number
        return {'value': None, 'unit': UNIT, 'unavailable': f'{type(e).__name__}: {e}'}
    import bench_models
    return e2e_calibration_benchmark(batch=args.batch, batches=max(1, SAMPLES_PER_GPU // args.batch), steps=args.e2e_steps,
                                     warmup=args.warmup, device=device, world=world, seed=rank, channels_last=not args.e2e_nchw,
                                     model=bench_models.build(args.workload), image=WORKLOADS[args.workload]['image'],
                                     distinct_host_batches=16 if args.workload == 'resnet50' else 4)


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port of the reference CPU path)
class CpuReplay:
    """The reference's USING_CUDA_KERNEL=False path over the replayed activation set on the host cores, restated in oracle/ with torch CPU
    ops (qfunction/linear.py:73-81, observer/range.py:91-92, :183, :190-282): per batch, both phases; the KL search separately."""

    def __init__(self, workload, batch, seed=0):
        import oracle as ora
        self.ora = ora
        torch.set_num_threads(ora.host_threads())
        acts, weights = WORKLOADS[workload]['table']()
        g = torch.Generator().manual_seed(seed)
        self.ts = []
        for i, shp in enumerate(acts):
            t = torch.randn((batch,) + shp, generator=g)
            if i % 2 == 1: t.relu_()
            self.ts.append(t)
        self.ws = [torch.randn(shp, generator=g) * 0.05 for shp in weights]
        self.wscale = [(w.abs().amax(dim=tuple(range(1, w.dim()))) / 127).clamp_min(1e-8) for w in self.ws]
        self.woff = [torch.zeros_like(s) for s in self.wscale]
        self.mins = [float('inf')] * len(self.ts); self.maxs = [float('-inf')] * len(self.ts)
        self.hists = None

    def batch_both_phases(self):
        """Seconds for one calibration batch: phase-1 work + phase-2 work (the histogram range comes from this batch's own min/max)."""
        ora = self.ora
        t0 = time.perf_counter()
        for w, s, o in zip(self.ws, self.wscale, self.woff): ora.torch_cpu_linear_quant_c(w, s, o, 0, -128, 127)
        for i, t in enumerate(self.ts):
            lo, hi = ora.torch_cpu_minmax(t)
            self.mins[i] = min(self.mins[i], lo.item()); self.maxs[i] = max(self.maxs[i], hi.item())
        self.hs = [max(abs(a), abs(b)) / BINS for a, b in zip(self.mins, self.maxs)]
        if self.hists is None: self.hists = [torch.zeros(BINS, dtype=torch.int32) for _ in self.ts]
        for w, s, o in zip(self.ws, self.wscale, self.woff): ora.torch_cpu_linear_quant_c(w, s, o, 0, -128, 127)
        for i, t in enumerate(self.ts): self.hists[i] += ora.torch_cpu_hist_sym(t, self.hs[i], BINS)
        return time.perf_counter() - t0

    def search(self):
        t0 = time.perf_counter()
        for h, s in zip(self.hists, self.hs): self.ora.kl_search(h, s, 8)
        return time.perf_counter() - t0


def cpu_replay_rate(args, budget_s, max_batches):
    """imgs/s of the CPU replay for the GPU arm's workload: (batches_per_step x mean batch time + one KL search) per 512 samples, measured on a
    bounded sample of whole batches of the GPU arm's batch size."""
    import oracle as ora
    rep = CpuReplay(args.workload, args.batch)
    rep.batch_both_phases()                                             # warm-up (allocator, thread pool), discarded
    times = []
    while len(times) < max_batches and (sum(times) < budget_s or len(times) < 2): times.append(rep.batch_both_phases())
    t_search = rep.search()
    nb = max(1, SAMPLES_PER_GPU // args.batch)
    t_batch = sum(times) / len(times)
    rate = nb * args.batch / (nb * t_batch + t_search)
    return rate, {'timed_batches': len(times), 'batch_s': stats(times), 'kl_search_s': round(t_search, 3), 'threads': ora.host_threads(),
                  'cpus_reported': os.cpu_count(), 'seconds': round(sum(times) + t_search, 1)}


def cpu_baseline(args):
    import oracle as ora
    rate, info = cpu_replay_rate(args, budget_s=12.0, max_batches=16)
    return {'value': round(rate, 2), 'unit': UNIT, 'cores': ora.host_threads(), 'kind': 'port',
            'sample': f"{info['timed_batches']} calibration batch(es) of {args.batch} images (the GPU arm's batch), both phases each: per-forward weight fake-quant, "
                      f"min/max + histc over the replayed activation tensors; + one KL search over all tensors ({info['kl_search_s']} s), combined as "
                      f"{max(1, SAMPLES_PER_GPU // args.batch)} batches + 1 search per {SAMPLES_PER_GPU} samples; torch CPU ops (oracle/ restatement of the reference "
                      f"USING_CUDA_KERNEL=False path) on {info['threads']} threads (host reports {info['cpus_reported']} CPUs); {info['seconds']} s",
            'detail': info}


def run_reference(args, rank, world):
    """The reference arm: the reference's own CPU implementation of the path (USING_CUDA_KERNEL=False) on the host cores, on the GPU arm's config
    (same workload, same calibration batch), each step a bounded sample = ONE calibration batch of `--batch` images through both phases:
      value   the activation-set replay (what the GPU arm's `value` measures): oracle port of the CPU collectors, 106 tensors
      e2e     the whole pipeline (what the GPU arm's `e2e` measures): images in host memory, torch CPU forward of ResNet-50 with per-forward
              weight fake-quant, min/max + histc observers (oracle/cpu_pipeline.py: pinned bit for bit against the unmodified reference
              pipeline, tests/test_cpu_graph_parity.py)
    both with the KL search of a whole calibration amortised over its 16 batches.  The timed steps are capped by wall-clock, never the batch."""
    if rank != 0: return None
    import oracle as ora
    torch.set_num_threads(ora.host_threads())
    nb = max(1, SAMPLES_PER_GPU // args.batch)
    budget = float(args.ref_budget)
    rate, info = cpu_replay_rate(args, budget_s=budget * 0.4, max_batches=args.steps)
    acts, weights = WORKLOADS[args.workload]['table']()
    e2e, e2e_info = None, None
    if True:
        import bench_models
        from oracle.cpu_pipeline import CpuPipeline
        torch.manual_seed(0)
        image = WORKLOADS[args.workload]['image']
        pipe = CpuPipeline(bench_models.build(args.workload), torch.zeros((1,) + image))
        pipe.quantize_parameters()
        g = torch.Generator().manual_seed(1)
        x = torch.rand((args.batch,) + image, generator=g)
        times, t_search = [], None
        t_begin = time.perf_counter()
        for k in range(args.steps + 1):
            t0 = time.perf_counter()
            t_search = pipe.calibrate([x], 'kl', return_search_seconds=True)
            dt = time.perf_counter() - t0 - t_search
            if k > 0: times.append(dt)                                   # the first call is the warm-up
            for _, c in pipe.observed_all(): c.state = 'INITIAL'         # next step calibrates again
            if time.perf_counter() - t_begin > budget * 0.6 and len(times) >= 2: break
        t_batch = sum(times) / len(times)
        e2e = nb * args.batch / (nb * t_batch + t_search)
        e2e_info = {'timed_batches': len(times), 'batch_s': stats(times), 'kl_search_s': round(t_search, 3), 'observed_tensors': len(pipe.observed_all())}
    v = round(rate, 2)
    cfg = workload_config(args, acts, weights, nb)
    cfg.update({'parallelism': f'dp{world} (sample-sharded, 2 all-reduces per calibration)',
                'l2_policy': f'inputs larger than L2: {args.rotate} rotating activation sets of {4 * sum(numel(s) for s in acts) * args.batch / 1e9:.2f} GB each'})
    return {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': round(1e3 * nb * args.batch / rate, 2), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': cfg,
            'arm': {'host_threads': torch.get_num_threads(), 'cpus_reported': os.cpu_count(), 'replay': info, 'pipeline': e2e_info},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
                             'sample': f"each step = one calibration batch of {args.batch} images through both phases (replay port of the CPU collectors over the "
                                       f"{len(acts)} activation tensors); {info['timed_batches']} step(s) timed + one KL search ({info['kl_search_s']} s) amortised over "
                                       f"{nb} batches; {info['seconds']} s on {info['threads']} threads"},
            'e2e': {'value': None if e2e is None else round(e2e, 2), 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                    'what': 'CPU end-to-end pipeline incl. the torch CPU forward (oracle/cpu_pipeline.py), same network and batch as the GPU arm'}}


def host_cpu_quota():
    """CPUs this process may actually use (cgroup quota / affinity), not the CPUs the host reports: the B200 boxes report 128 and grant 16, and
    one OpenMP thread per *reported* CPU makes torch's host-side ops crawl (spinning threads under a CFS quota)."""
    n = os.cpu_count() or 1
    try: n = min(n, len(os.sched_getaffinity(0)))
    except Exception: pass
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max': n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read()); p_ = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0: n = min(n, max(1, q // p_))
        except Exception: pass
    return max(1, n)


def main():
    import faulthandler
    faulthandler.enable()
    faulthandler.dump_traceback_later(240, repeat=True, file=sys.stderr)          # a stuck run leaves its stacks in stderr instead of nothing
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed steps; one step = one whole calibration of 512 samples per GPU')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=None, help='calibration batch (default: 32 for resnet50, 16 for yolov5s)')
    ap.add_argument('--workload', default='resnet50', choices=sorted(WORKLOADS))
    ap.add_argument('--rotate', type=int, default=4, help='distinct activation sets cycled through (each > L2)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--e2e-steps', type=int, default=5, help='timed end-to-end calibrations of 512 samples (each ~0.12 s)')
    ap.add_argument('--e2e-nchw', action='store_true', help='run the torch network of the e2e arm in NCHW; default is NHWC (channels_last: cuDNN\'s native layout -- '
                    'measured 3.09 vs 3.83-4.24 ms per 32-image forward; the hot path reads dense tensors in storage order either way)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-sweep', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='profiling runs only')
    ap.add_argument('--ref-budget', type=float, default=100.0, help='wall-clock budget (s) of the CPU reference arm')
    ap.add_argument('--per-tensor-weight-launches', action='store_true', help='one QuantizeTensor_LC launch per weight (the reference flow) instead of the multi-tensor launch')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed to DIR/<name>.npy (same arguments, same inputs: comparable across builds)')
    args = ap.parse_args()
    if args.batch is None: args.batch = WORKLOADS[args.workload]['batch']
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1)); local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        res = run_reference(args, rank, world)
        if res is not None: print(json.dumps(res), flush=True)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the hot path has no CPU fallback); use --impl reference for the CPU arm')
    if 'OMP_NUM_THREADS' not in os.environ: torch.set_num_threads(host_cpu_quota())   # torchrun sets it to 1 per rank; a bare `python bench.py` must not take 128
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    res = run_ours(args, rank, world, local_rank)
    if rank == 0: print(json.dumps(res), flush=True)
    if world > 1: dist.destroy_process_group()


if __name__ == '__main__':
    main()
