"""Graph-level parity on the CPU (VERDICT r1 item 1): the fixture tests/golden/graph_pipeline.npz was produced by the UNMODIFIED reference
pipeline (TRT_INT8 quantizer's own pass list on a programmatically built BaseGraph, tests/golden/make_graph_golden.py).  Checked here:
  * oracle/cpu_pipeline.py (the CPU arm of bench.py) reproduces it bit for bit: observed set, dominators, states, scales / offsets of all
    four observers, aligned Add inputs, baked weights and the quantised network output -- so the CPU arm is a pinned port;
  * ppq_b200.executor's topology passes (fusion + simplify, which need no GPU) give the same states / dominators / observed set.
The GPU twin (tests/test_gpu_graph_parity.py) checks ppq_b200's executor against the same pipeline run on the B200.
"""
import json

import numpy as np
import pytest
import torch

import netspec
from conftest import load_golden


FIXTURES = {'tinyres': 'graph_pipeline.npz', 'tinycat': 'graph_pipeline_tinycat.npz'}


def load_fixture(net):
    z = load_golden(FIXTURES[net])
    return z, json.loads(bytes(z['meta']).decode())


@pytest.fixture(scope='module')
def fx():
    return load_fixture('tinyres')


def labels(spec):
    """fixture (op, var) -> label used by oracle.cpu_pipeline / key used for ppq_b200.executor configs."""
    m = {}
    for o in spec:
        for i, v in enumerate(o['inputs']): m[(o['name'], v)] = (f"{o['name']}#0", f'in{i}')
        m[(o['name'], o['out'])] = (f"{o['name']}#0", 'out')
        if o['op'] in ('Conv', 'Gemm'): m[(o['name'], o['name'] + '.w')] = (f"{o['name']}#0", 'w')
    return m


def net_and_data(meta):
    spec = netspec.SPECS[meta['net']]
    params = netspec.make_params(spec, meta['param_seed'])
    data = [torch.from_numpy(x) for x in netspec.make_data(meta['net'], meta['data_seed'], meta['steps'], meta['batch'])]
    return spec, params, data


def bits(a):
    return np.asarray(a, dtype=np.float32).reshape(-1).view(np.uint32)


@pytest.mark.parametrize('net,method', [('tinyres', m) for m in ('kl', 'minmax', 'percentile', 'mse')] + [('tinycat', 'kl'), ('tinycat', 'percentile')])
def test_cpu_pipeline_port_reproduces_the_reference_pipeline(net, method):
    from oracle.cpu_pipeline import CpuPipeline
    z, meta = load_fixture(net)
    torch.set_num_threads(1)
    spec, params, data = net_and_data(meta)
    lab = labels(spec)
    pipe = CpuPipeline(netspec.SpecNet(spec, params), data[0], fuse_bn=False)
    port = {}
    for op in pipe.ops:
        for i, c in enumerate(op.ins): port[(op.name, f'in{i}')] = c
        port[(op.name, 'out')] = op.out
        if op.w is not None: port[(op.name, 'w')] = op.w
    entry = meta['methods'][method]
    # the observed set = the activation configs the reference calibrated, in execution order
    want = [lab[(r['op'], r['var'])] for r in entry['calibrated'] if r['state'] == 'ACTIVATED' and not r['var'].endswith('.w')]
    got = [tuple(label.split('|')) for label, _ in pipe.observed()]
    assert got == want
    pipe.quantize_parameters()
    pipe.calibrate(data, method)

    def check(stage):
        for r in entry[stage]:
            if r['state'] == 'FP32': continue                                  # bias
            c = port[lab[(r['op'], r['var'])]]
            assert c.state == r['state'], (stage, r['op'], r['var'], c.state, r['state'])
            if r['dominator'] is not None:
                dop, dvar = r['dominator'].split('|')
                assert c.root is port[lab[(dop, dvar)]], (stage, r['op'], r['var'])
            assert np.array_equal(bits(c.scale), bits(z[r['scale']])), (stage, r['op'], r['var'], c.scale, z[r['scale']])
            assert np.array_equal(bits(c.offset), bits(z[r['offset']]))
    check('calibrated')
    pipe.align(); pipe.bake()
    check('final')
    for o in spec:
        if o['op'] in ('Conv', 'Gemm'):
            assert np.array_equal(bits(getattr(pipe.model, o['name']).weight.data.numpy()), bits(z[f"{method}.baked.{o['name']}.w"])), o['name']
    out = pipe.forward(data[0]).numpy()
    assert np.array_equal(bits(out), bits(z[f'{method}.output'])), np.abs(out - z[f'{method}.output']).max()


@pytest.mark.parametrize('net', ['tinyres', 'tinycat'])
def test_executor_topology_matches_the_reference_passes(net):
    """QuantizeFusionPass + QuantizeSimplifyPass as mirrored by ppq_b200.executor: same OVERLAPPED configs, same group roots, same observed
    tensors in the same order as the reference graph (no GPU needed: tracing runs the fp32 modules on the CPU)."""
    from ppq_b200.executor import TorchExecutor
    _, meta = load_fixture(net)
    spec, params, data = net_and_data(meta)
    lab = labels(spec)
    ex = TorchExecutor(netspec.SpecNet(spec, params), data[0], fuse_bn=False)
    ours = {}
    for name, op in ex.quantable_operations():
        for i, c in enumerate(op.input_cfgs): ours[(name, f'in{i}')] = c
        ours[(name, 'out')] = op.output_cfg
        if op.weight_cfg is not None: ours[(name, 'w')] = op.weight_cfg
    rows = meta['methods']['kl']['calibrated']
    assert len([r for r in rows if r['state'] != 'FP32']) == len(ours)
    for r in rows:
        if r['state'] == 'FP32': continue
        c = ours[lab[(r['op'], r['var'])]]
        want = 'OVERLAPPED' if r['state'] == 'OVERLAPPED' else 'INITIAL'          # ACTIVATED after calibration == INITIAL before it
        assert c.state.name == want, (r['op'], r['var'], c.state, r['state'])
        if r['dominator'] is not None:
            dop, dvar = r['dominator'].split('|')
            assert c.dominated_by is ours[lab[(dop, dvar)]], (r['op'], r['var'])
        else:
            assert c.dominated_by is c
    want = [ours[lab[(r['op'], r['var'])]] for r in rows if r['state'] == 'ACTIVATED' and not r['var'].endswith('.w')]
    got = ex.observed_configs()
    assert len(got) == len(want) and all(a is b for a, b in zip(got, want))


def test_executor_topology_on_torchvision_resnet():
    """Functional residual adds (`out += identity`) and torch.flatten are invisible to module hooks; the observed set must still be the one
    the reference graph has: input, every ReLU output, the conv outputs that feed an Add (conv3 / downsample), global pool, fc --
    NOT the max-pool output (passive op: shares its input's config) and NOT the fc input (a view of the pooled tensor)."""
    torchvision = pytest.importorskip('torchvision')
    from ppq_b200.executor import TorchExecutor
    ex = TorchExecutor(torchvision.models.resnet18(weights=None), torch.zeros(1, 3, 64, 64))
    ops = dict(ex.quantable_operations())
    assert ops['maxpool#0'].output_cfg.state.name == 'OVERLAPPED' and ops['maxpool#0'].output_cfg.dominated_by is ops['relu#0'].output_cfg
    assert ops['conv1#0'].output_cfg.state.name == 'OVERLAPPED'                              # conv -> relu fusion
    assert ops['layer1.0.conv2#0'].output_cfg.state.name == 'INITIAL'                        # feeds the (invisible) Add: observed
    assert ops['layer1.0.relu#1'].input_cfgs[0].dominated_by is ops['layer1.0.relu#1'].output_cfg   # Add -> Relu fusion
    assert ops['fc#0'].input_cfgs[0].dominated_by is ops['avgpool#0'].output_cfg             # flatten is a view: passive
    n_relu = sum(1 for n, o in ops.items() if o.kind == 'Relu')
    n_to_add = sum(1 for n in ops if n.endswith('conv2#0') or 'downsample.0' in n)
    assert len(ex.observed_configs()) == 1 + n_relu + n_to_add + 2                           # input + relus + add operands + avgpool + fc


def test_executor_dequantize_and_restore_swap_states_and_stored_weights(fx):
    """IR/quantize.py:118-160 as mirrored by the executor: dequantize() stores every config's state, sets FP32 and swaps baked parameters with their
    stored fp32 values; restore_quantize_state() undoes both (host logic only: no kernel involved)."""
    from ppq_b200.core import QuantizationStates as S
    from ppq_b200.executor import TorchExecutor
    _, meta = fx
    spec, params, data = net_and_data(meta)
    ex = TorchExecutor(netspec.SpecNet(spec, params), data[0], fuse_bn=False)
    ops = dict(ex.quantable_operations())
    conv = ops['conv1#0']
    fp32 = conv.module.weight.data.clone()
    baked = fp32 * 0.5                                                     # stand-in for the fake-quantised value
    conv.stored_weight, conv.module.weight.data, conv.weight_cfg.state = conv.module.weight.data, baked, S.BAKED
    before = {(n, i): c.state for n, op in ops.items() for i, c in enumerate(op.input_cfgs + [op.output_cfg])}
    ex.dequantize()
    assert all(c.state == S.FP32 for op in ops.values() for c in op.input_cfgs + [op.output_cfg]) and conv.weight_cfg.state == S.FP32
    assert torch.equal(conv.module.weight.data, fp32) and torch.equal(conv.stored_weight, baked)
    ex.dequantize()                                                        # idempotent
    assert torch.equal(conv.module.weight.data, fp32)
    ex.restore_quantize_state()
    assert {(n, i): c.state for n, op in ops.items() for i, c in enumerate(op.input_cfgs + [op.output_cfg])} == before
    assert conv.weight_cfg.state == S.BAKED and torch.equal(conv.module.weight.data, baked) and torch.equal(conv.stored_weight, fp32)
