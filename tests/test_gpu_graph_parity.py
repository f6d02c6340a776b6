"""Graph-level parity ON THE B200 against the ORIGINAL PROJECT's pipeline (OpenPPL/ppq, unmodified: TRT_INT8 quantizer's own pass list,
TorchExecutor(device='cuda') inside `with ENABLE_CUDA_KERNEL():`, served by its own CUDA extension compiled for sm_100a).  What that pipeline
produced -- every config's state / dominator / scale / offset after calibration and at the end, the baked weights, the quantised network
output, the graphwise SNR of its own evaluation loop -- is stored in tests/golden/graph_pipeline_gpu.npz and graph_pipeline_tinycat_gpu.npz
(recorded with PPQ_RECORD_GOLDEN set, the original package and oracle/_ref present: tests/refrecord.py, tests/refppq.py).  Checked here:

  C. ppq_b200's own executor + RuntimeCalibrationPass / calibrate_arena on the equivalent torch module reproduce those results bit for bit;
  D. they agree with the committed CPU-path fixture (tests/golden/graph_pipeline.npz) to float tolerance (cuDNN vs CPU convs), weights and
     the network input bit for bit.
"""
import json
import os

import numpy as np
import pytest
import torch

import netspec
import refppq
import refrecord
from conftest import load_golden

pytestmark = pytest.mark.gpu
METHODS = ['kl', 'minmax', 'percentile', 'mse']


def make_env(fixture):
    if not torch.cuda.is_available(): pytest.skip('no CUDA device')
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    z = load_golden(fixture)
    meta = json.loads(bytes(z['meta']).decode())
    spec = netspec.SPECS[meta['net']]
    params = netspec.make_params(spec, meta['param_seed'])
    data = netspec.make_data(meta['net'], meta['data_seed'], meta['steps'], meta['batch'])
    recorded = fixture.replace('.npz', '_gpu.npz')
    env = dict(z=z, meta=meta, spec=spec, params=params, data=data, recorded=recorded, cache={})
    if refrecord.record_dir() is not None:
        env['ppq'], env['ref'] = refppq.load(), refrecord.reference_extension()
        assert env['ppq'] is not None, 'recording needs the original package (tests/refppq.py)'
    else:
        env['stored'] = load_golden(recorded)
    return env


def save_records(env):
    if refrecord.record_dir() is None: return
    arrays, meta = {}, {}
    for key, res in env['cache'].items():
        meta[key] = pack(key, res, arrays)
    arrays['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    os.makedirs(refrecord.record_dir(), exist_ok=True)
    np.savez_compressed(os.path.join(refrecord.record_dir(), env['recorded']), **arrays)


@pytest.fixture(scope='module')
def env():
    e = make_env('graph_pipeline.npz')
    yield e
    save_records(e)


@pytest.fixture(scope='module')
def env_cat():
    """The second graph: Concat ('Align to Output'), conv -> Sigmoid fusion, AveragePool, a max-pool whose producer has two consumers."""
    e = make_env('graph_pipeline_tinycat.npz')
    yield e
    save_records(e)


def pack(key, res, arrays):
    """One pipeline result -> JSON-able metadata; its arrays go into `arrays` under names derived from `key`."""
    meta = {'passes': res['passes'], 'graphwise': None if 'graphwise' not in res else {k: float(v) for k, v in res['graphwise'].items()}}
    for stage in ('calibrated', 'final'):
        rows = []
        for i, r in enumerate(res[stage]):
            row = {k: r[k] for k in ('op', 'var', 'state', 'dominator')}
            for k in ('scale', 'offset'):
                row[k] = None if r[k] is None else f'{key}.{stage}.{i}.{k}'
                if r[k] is not None: arrays[row[k]] = np.asarray(r[k], np.float32)
            rows.append(row)
        meta[stage] = rows
    meta['baked'] = {}
    for k, v in res['baked'].items():
        meta['baked'][k] = f'{key}.baked.{k}'
        arrays[meta['baked'][k]] = v
    arrays[f'{key}.output'] = res['output']
    return meta


def unpack(key, z):
    meta = json.loads(bytes(z['meta']).decode())[key]
    res = {'passes': meta['passes'], 'output': z[f'{key}.output'], 'baked': {k: z[v] for k, v in meta['baked'].items()}}
    if meta['graphwise'] is not None: res['graphwise'] = meta['graphwise']
    for stage in ('calibrated', 'final'):
        res[stage] = [dict(r, scale=None if r['scale'] is None else z[r['scale']], offset=None if r['offset'] is None else z[r['offset']])
                      for r in meta[stage]]
    return res


def bits(a):
    return np.asarray(a, dtype=np.float32).reshape(-1).view(np.uint32)


def reference_run(env, method, analyse=False):
    """The original pipeline on cuda with its own CUDA extension: run when recording, else read from the stored record."""
    key = method + ('-analyse' if analyse else '')
    if key in env['cache']: return env['cache'][key]
    if refrecord.record_dir() is None:
        res = unpack(key, env['stored'])
    else:
        with refppq.use_extension(env['ref']):
            res = netspec.run_reference_pipeline(env['ppq'], env['spec'], env['params'], env['data'], method, device='cuda', cuda_kernel=True,
                                                 analyse=analyse)
    env['cache'][key] = res
    return res


def our_executor(env):
    from ppq_b200.executor import TorchExecutor
    model = netspec.SpecNet(env['spec'], env['params']).cuda()
    batches = [torch.from_numpy(x).cuda() for x in env['data']]
    ex = TorchExecutor(model, batches[0], fuse_bn=False)
    ex.quantize_parameters()
    return ex, batches


def rows_of(ex, spec):
    """our configs keyed like the fixture rows: (op, var) -> config."""
    out = {}
    ops = dict(ex.quantable_operations())
    for o in spec:
        op = ops[o['name'] + '#0']
        for i, v in enumerate(o['inputs']): out[(o['name'], v)] = op.input_cfgs[i]
        out[(o['name'], o['out'])] = op.output_cfg
        if op.weight_cfg is not None: out[(o['name'], o['name'] + '.w')] = op.weight_cfg
    return out


def check_against(ex, env, want_rows, tag):
    ours = rows_of(ex, env['spec'])
    for r in want_rows:
        if r['state'] == 'FP32': continue
        c = ours[(r['op'], r['var'])]
        assert c.state.name == r['state'], (tag, r['op'], r['var'], c.state, r['state'])
        if r['dominator'] is not None:
            dop, dvar = r['dominator'].split('|')
            assert c.dominated_by is ours[(dop, dvar)], (tag, r['op'], r['var'])
        assert np.array_equal(bits(c.scale.cpu().numpy()), bits(r['scale'])), (tag, r['op'], r['var'], c.scale, r['scale'])
        assert np.array_equal(bits(c.offset.cpu().numpy()), bits(r['offset'])), (tag, r['op'], r['var'])


@pytest.mark.parametrize('flow,method', [('hooks', m) for m in METHODS] + [('arena', m) for m in METHODS] + [('arena-deferred', 'kl')])
def test_our_executor_reproduces_the_reference_pipeline(env, flow, method):
    """C: ppq_b200.executor (+ RuntimeCalibrationPass with the device-resident observers, or the arena calibrator: one multi-tensor launch
    per forward) on the equivalent torch module vs the real pipeline on the same GPU: same observed set, bit-identical scales, then the
    same aligned / baked / quantised forward."""
    from ppq_b200.calibration import RuntimeCalibrationPass
    from ppq_b200.executor import calibrate_arena
    want = reference_run(env, method)
    ex, batches = our_executor(env)
    if flow == 'hooks':
        RuntimeCalibrationPass(method=method).optimize(ex, batches, ex, calib_steps=len(batches))
    else:
        calibrate_arena(ex, batches, method=method, deferred=(True if flow == 'arena-deferred' else 'auto'))
    check_against(ex, env, want['calibrated'], f'{flow}/{method}/calibrated')
    ex.align_quantization()
    ex.bake_parameters()
    check_against(ex, env, want['final'], f'{flow}/{method}/final')
    for o in env['spec']:
        if o['op'] in ('Conv', 'Gemm'):
            assert np.array_equal(bits(getattr(ex.model, o['name']).weight.data.cpu().numpy()), bits(want['baked'][o['name'] + '.w'])), o['name']
    out = ex.forward(batches[0]).cpu().numpy()
    assert np.array_equal(bits(out), bits(want['output'])), np.abs(out - want['output']).max()


@pytest.mark.parametrize('method', ['minmax', 'percentile'])
def test_gpu_pipeline_agrees_with_the_cpu_path_fixture(env, method):
    """D: CPU-path fixture vs the same reference pipeline on the GPU with our kernels.  Weights: bit-equal.  Activations differ by conv
    rounding (cuDNN vs CPU) only: scales within 1e-4 relative; the percentile observer additionally selects a neighbouring order statistic
    on the CPU path (int() truncation vs round-to-nearest index, SURVEY appendix B)."""
    z, entry = env['z'], env['meta']['methods'][method]
    got = reference_run(env, method)
    for r, g in zip(entry['calibrated'], got['calibrated']):
        assert (r['op'], r['var'], r['state'], r['dominator']) == (g['op'], g['var'], g['state'], g['dominator'])
        if r['state'] == 'FP32': continue
        if r['var'].endswith('.w') or (r['var'] == 'x' and method == 'minmax'):
            assert np.array_equal(bits(z[r['scale']]), bits(g['scale'])), (r['op'], r['var'])
        else:
            np.testing.assert_allclose(g['scale'], z[r['scale']], rtol=0.15 if method == 'percentile' else 1e-4)   # percentile: the next order statistic of a tail
    np.testing.assert_allclose(got['output'], z[f'{method}.output'], atol=0.08 if method == 'minmax' else 0.5)   # a few quantisation steps of the last layer


def test_parameter_baking_states_values_and_no_requantisation(env):
    """ParameterBakingPass semantics (ppq/IR/quantize.py:98-111, optim/baking.py:34-47): ACTIVATED -> BAKED, PASSIVE -> PASSIVE_BAKED, the
    baked value IS the fake-quantised value, and later forwards use it as is (no weight fake-quant launch, the parameter is not touched)."""
    from ppq_b200.core import QuantizationStates as S
    from ppq_b200.qfunction import PPQuantFunction
    ex, batches = our_executor(env)
    ops = dict(ex.quantable_operations())
    ops['conv3#0'].weight_cfg.master_by = ops['conv2#0'].weight_cfg        # a passive parameter config: shares conv2's per-channel scales (16 channels each)
    assert ops['conv3#0'].weight_cfg.state == S.PASSIVE and ops['conv3#0'].weight_cfg.scale is ops['conv2#0'].weight_cfg.scale
    weighted = {n: op for n, op in ops.items() if op.weight_cfg is not None}
    fp32 = {n: op.module.weight.data.clone() for n, op in weighted.items()}
    want = {n: PPQuantFunction(op.module.weight.data, op.weight_cfg).clone() for n, op in weighted.items()}
    assert len(ex._quantize_all_weights()) == len(weighted)                # before baking: every ACTIVATED / PASSIVE weight is re-quantised per forward (one launch)
    ex._restore_weights()
    ex.bake_parameters()
    for n, op in weighted.items():
        assert op.weight_cfg.state == (S.PASSIVE_BAKED if n == 'conv3#0' else S.BAKED), (n, op.weight_cfg.state)
        assert np.array_equal(bits(op.module.weight.data.cpu().numpy()), bits(want[n].cpu().numpy())), n
    assert ex._quantize_all_weights() == {}                                # nothing left to quantise per forward
    ptrs = {n: op.module.weight.data_ptr() for n, op in weighted.items()}
    ex.forward(batches[0])
    for n, op in weighted.items():
        assert op.module.weight.data_ptr() == ptrs[n] and np.array_equal(bits(op.module.weight.data.cpu().numpy()), bits(want[n].cpu().numpy())), n
    ex.bake_parameters()                                                   # idempotent: BAKED configs are skipped
    for n, op in weighted.items():
        assert np.array_equal(bits(op.module.weight.data.cpu().numpy()), bits(want[n].cpu().numpy())), n
    # dequantize() / restore_quantize_state() (IR/quantize.py:118-160): the fp32 weights come back from `stored_value`, every config reads FP32
    ex.dequantize()
    for n, op in weighted.items():
        assert op.weight_cfg.state == S.FP32 and op.output_cfg.state == S.FP32
        assert np.array_equal(bits(op.module.weight.data.cpu().numpy()), bits(fp32[n].cpu().numpy())), n
    ex.restore_quantize_state()
    for n, op in weighted.items():
        assert op.weight_cfg.state == (S.PASSIVE_BAKED if n == 'conv3#0' else S.BAKED)
        assert np.array_equal(bits(op.module.weight.data.cpu().numpy()), bits(want[n].cpu().numpy())), n


def test_graphwise_error_analyse_equals_the_reference_function(env):
    """The evaluation loop (SURVEY 8f-3): the original's own graphwise_error_analyse on its quantised graph vs ours on the equivalent module with
    bit-identical configs -- same operations, same seeded sample of 4096 elements per image, same SNR."""
    from ppq_b200.executor import calibrate_arena, graphwise_error_analyse
    want = reference_run(env, 'kl', analyse=True)
    ex, batches = our_executor(env)
    calibrate_arena(ex, batches, method='kl')
    ex.align_quantization(); ex.bake_parameters()
    check_against(ex, env, want['final'], 'analyse/final')
    got = graphwise_error_analyse(ex, batches, fetchs=4096)
    assert sorted(got) == sorted(k + '#0' for k in want['graphwise']), (sorted(got), sorted(want['graphwise']))
    for k, v in want['graphwise'].items():
        assert abs(got[k + '#0'] - v) <= 1e-6 + 2e-4 * abs(v), (k, got[k + '#0'], v)
    full = graphwise_error_analyse(ex, batches)                            # whole tensors, every operation: same order of magnitude, all below the 0.1 bar
    assert len(full) == len(ex.quantable_operations()) and all(0 <= e < 0.1 for e in full.values())


@pytest.mark.parametrize('method', ['kl', 'percentile'])
def test_second_graph_concat_alignment_and_sigmoid_fusion(env_cat, method):
    """C on the Concat graph: our executor (arena flow, then Concat 'Align to Output' + baking) reproduces the original pipeline's configs, baked
    weights and quantised output bit for bit."""
    from ppq_b200.executor import calibrate_arena
    env = env_cat
    want = reference_run(env, method)
    ex, batches = our_executor(env)
    calibrate_arena(ex, batches, method=method)
    check_against(ex, env, want['calibrated'], f'tinycat/{method}/calibrated')
    ex.align_quantization(); ex.bake_parameters()
    check_against(ex, env, want['final'], f'tinycat/{method}/final')
    out = ex.forward(batches[0]).cpu().numpy()
    assert np.array_equal(bits(out), bits(want['output'])), np.abs(out - want['output']).max()
