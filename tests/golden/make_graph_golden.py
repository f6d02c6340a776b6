"""Graph-level golden fixture: the UNMODIFIED reference pipeline (TRT_INT8 quantizer -> QuantizeFusionPass -> QuantizeSimplifyPass ->
ParameterQuantizePass -> RuntimeCalibrationPass -> QuantAlignmentPass -> PassiveParameterQuantizePass -> ParameterBakingPass; CPU /
torch path, USING_CUDA_KERNEL = False) run on a programmatically built BaseGraph (SURVEY.md appendix C2).

    PPQ_REFERENCE_ROOT=<checkout> python tests/golden/make_graph_golden.py          # rewrites tests/golden/graph_pipeline.npz

Stored: for every activation algorithm (kl, minmax, percentile, mse) every TensorQuantizationConfig's state / dominator / scale /
offset right after RuntimeCalibrationPass and after the last pass, the quantised graph's output on the first batch, and the baked
weights.  Weights and calibration data are regenerated from seeds by tests/netspec.py.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import numpy as np
import torch

import netspec
import refppq

NETS = {'tinyres': ('kl', 'minmax', 'percentile', 'mse'), 'tinycat': ('kl', 'percentile')}
PARAM_SEED, DATA_SEED, STEPS, BATCH = 7, 11, 8, 4


def generate(ppq, net, methods):
    spec = netspec.SPECS[net]
    params = netspec.make_params(spec, PARAM_SEED)
    data = netspec.make_data(net, DATA_SEED, STEPS, BATCH)
    arrays, meta = {}, dict(net=net, param_seed=PARAM_SEED, data_seed=DATA_SEED, steps=STEPS, batch=BATCH, methods={})
    for method in methods:
        res = netspec.run_reference_pipeline(ppq, spec, params, data, method)
        entry = {'passes': res['passes']}
        for stage in ('calibrated', 'final'):
            rows = []
            for i, row in enumerate(res[stage]):
                r = {k: row[k] for k in ('op', 'var', 'state', 'algo', 'dominator')}
                for k in ('scale', 'offset'):
                    if row[k] is not None:
                        key = f'{method}.{stage}.{i}.{k}'
                        arrays[key] = row[k].astype(np.float32)
                        r[k] = key
                rows.append(r)
            entry[stage] = rows
        arrays[f'{method}.output'] = res['output']
        for k, v in res['baked'].items(): arrays[f'{method}.baked.{k}'] = v
        meta['methods'][method] = entry
    arrays['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    out = os.path.join(HERE, 'graph_pipeline.npz' if net == 'tinyres' else f'graph_pipeline_{net}.npz')
    np.savez_compressed(out, **arrays)
    print(out, os.path.getsize(out), 'bytes;', {m: sum(r['state'] == 'ACTIVATED' for r in meta['methods'][m]['calibrated']) for m in methods})


def main():
    ppq = refppq.load()
    assert ppq is not None and refppq.root() == os.environ.get('PPQ_REFERENCE_ROOT'), 'generate fixtures from a checkout named by $PPQ_REFERENCE_ROOT'
    from ppq.core import PPQ_CONFIG
    assert PPQ_CONFIG.USING_CUDA_KERNEL is False
    torch.set_num_threads(1)                                   # deterministic reductions
    for net, methods in NETS.items(): generate(ppq, net, methods)


if __name__ == '__main__':
    main()
