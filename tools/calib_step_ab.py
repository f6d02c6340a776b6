#!/usr/bin/env python
"""A/B of the multi-tensor collectors inside bench.py's exact calibration step (variant keys "minmax" and "multi_histogram", variants.h).

    python tools/calib_step_ab.py [--workload resnet50|yolov5s] [--rounds 5] [--steps 3] [--arms old,new]

Replays bench.py's step -- same Workload, same ArenaCalibrator, same MultiWeightQuantizer, same rotation -- once per arm and round, the
arms alternating inside one process.  Prints per-arm median / min / max of the step and of the two collector launches (CUDA events), and
checks that every arm computes bit-identical min/max, hist_scale, histogram arena, scales and fake-quantised weights.
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import BINS, SAMPLES_PER_GPU, WORKLOADS, Workload  # noqa: E402
from ppq_b200.calibration import ArenaCalibrator, MultiWeightQuantizer  # noqa: E402
from ppq_b200.ffi import extension  # noqa: E402

# arm name -> (variant of "minmax", variant of "multi_histogram"); 1 selects the replaced kernels
ARMS = {'old': (1, 1), 'new': (0, 0), 'minmax_only': (0, 1), 'hist_only': (1, 0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workload', default='resnet50', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=None)
    ap.add_argument('--rotate', type=int, default=4)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=3, help='timed steps per arm and round')
    ap.add_argument('--arms', default='old,new')
    args = ap.parse_args()
    batch = args.batch or WORKLOADS[args.workload]['batch']
    arms = args.arms.split(',')
    ext = extension()
    device = torch.device('cuda', 0)
    torch.cuda.set_device(device)
    wl = Workload(device, args.workload, batch, args.rotate, seed=1234)
    nb = max(1, SAMPLES_PER_GPU // batch)
    cal = ArenaCalibrator(len(wl.acts), device, bins=BINS, num_of_bits=8, method='kl')
    wq = MultiWeightQuantizer(wl.w, wl.w_scale, wl.w_offset, channel_axis=0)
    stream = torch.cuda.current_stream()

    def ev():
        e = torch.cuda.Event(enable_timing=True); e.record(stream); return e

    def calibrate(times):
        cal.reset()
        for phase in (1, 2):
            for k in range(nb):
                wq()
                a = ev(); cal.observe(wl.sets[k % args.rotate]); b = ev()
                times['minmax' if phase == 1 else 'hist'].append((a, b))
            cal.end_phase()

    def set_arm(name):
        mm, h = ARMS[name]
        ext.set_variant('minmax', mm); ext.set_variant('multi_histogram', h)

    outputs = {}
    for name in arms:                                          # warm-up + the outputs every arm must reproduce
        set_arm(name)
        for _ in range(2): calibrate({'minmax': [], 'hist': []})
        torch.cuda.synchronize()
        outputs[name] = [cal.minmax.clone(), cal.hist_scale.clone(), cal.hist.clone(), cal.scale.clone()] + [y.clone() for y in wq.outputs]
    same = {n: all(torch.equal(a, b) for a, b in zip(outputs[arms[0]], outputs[n])) for n in arms}

    res = {n: {'step': [], 'minmax': [], 'hist': []} for n in arms}
    for r in range(args.rounds):
        for name in (arms if r % 2 == 0 else arms[::-1]):
            set_arm(name)
            times = {'minmax': [], 'hist': []}
            steps = []
            for _ in range(args.steps):
                a = ev(); calibrate(times); b = ev(); steps.append((a, b))
            torch.cuda.synchronize()
            res[name]['step'].append(sorted(a.elapsed_time(b) for a, b in steps)[len(steps) // 2])
            for k in ('minmax', 'hist'):
                res[name][k].append(sum(a.elapsed_time(b) for a, b in times[k]) / len(times[k]))
    set_arm('new')

    gb = 4.0 * wl.act_elems / 1e9
    print(f'{args.workload} batch {batch}: {len(wl.acts)} activation tensors, {gb:.3f} GB per collector launch, {nb} batches per phase, '
          f'{args.rounds} rounds x {args.steps} steps per arm on {torch.cuda.get_device_name(0)}')
    med = {}
    for name in arms:
        line = [f'{name:>4} {str(ARMS[name]):>7}']
        for k in ('step', 'minmax', 'hist'):
            v = sorted(res[name][k]); m = v[len(v) // 2]
            med[(name, k)] = m
            extra = f' {gb / (m * 1e-3):6.0f} GB/s' if k != 'step' else ''
            line.append(f'{k} median {m:8.4f} ms [{v[0]:.4f} .. {v[-1]:.4f}]{extra}')
        line.append(f'outputs identical to {arms[0]}: {same[name]}')
        print('   '.join(line), flush=True)
    if 'old' in arms:
        for name in arms:
            if name != 'old':
                print(f'{name} vs old: step {100 * (med[("old", "step")] / med[(name, "step")] - 1):+.1f} % faster, '
                      f'minmax {med[("old", "minmax")] / med[(name, "minmax")]:.3f}x, hist {med[("old", "hist")] / med[(name, "hist")]:.3f}x')
    if not all(same.values()):
        sys.exit('outputs differ between arms')


if __name__ == '__main__':
    main()
