"""Mint the golden fixtures from the UNMODIFIED reference (run in the build container only).

    python tests/golden/make_golden.py          # writes the fixtures that do not exist yet (new cases)
    python tests/golden/make_golden.py --all    # re-mints every fixture

For every case of ``tests/cases.build_cases()`` this runs the real ``ding.rl_utils`` functions (loaded read-only
from /root/reference by ``oracle/ref_loader.py``) on CPU fp32 and stores inputs, scalar parameters, forward
outputs and input-gradients in ``tests/golden/<case>.npz``.  The reference holds no golden vectors of its own for
this path (SURVEY.md section 8c) so these files are the pins that travel to the GPU box.

It also (re)writes ``tests/golden/reference/``: what the tests that compare with the reference itself compare against,
so that they run without it --
  api.json            signatures, namedtuple fields and module layout of the hot-path functions (test_host_logic.py)
  hpc_dispatch.json   what its ENABLE_DI_HPC wrapper hands to hpc_rll on a fixed sequence of calls (test_host_logic.py)
  bench_shapes.npz    outputs at the medium BASELINE shapes, a fixed sample of the large ones (test_oracle.py)
  policy_gae.npz      gae at the shapes of the policy-level restatement test (test_oracle.py)
  suite_records.npz   every value the ported reference unit tests record, run on the reference, as float32 with a JSON
                      index of (test body and arguments::name, offset, shape) (test_reference_suite.py)
"""
import inspect
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_DIR = os.path.join(HERE, 'reference')
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from tests import cases  # noqa: E402

SAMPLE = 512  # outputs larger than this are stored as a fixed sample plus their float64 sum and absolute sum


def bench_shape_cases():
    """medium shapes of the five BASELINE configs (kept to a few seconds on the host)"""
    return {
        'gae_D': cases.gae_case(100, 128, 512, p_done=0.01),
        'ppo_D': cases.ppo_case(101, 128 * 64, 6, clip_ratio=0.2),
        'qntd_B': cases.qntd_case(102, 512, 6, 3, value_gamma='tensor', gamma=0.99, done='bern'),
        'dntd_C': cases.dntd_case(103, 512, 6, 51, 3, gamma=0.99, value_gamma='tensor'),
        'vtrace_E': cases.vtrace_case(104, 64, 256, 6, gamma=0.99, lambda_=0.95),
    }


def policy_gae_inputs():
    """the inputs of test_oracle.py::test_policy_level_restatements_match_the_reference_lines, in its draw order"""
    g = torch.Generator().manual_seed(77)
    out = []
    for shape, std in (((400, ), None), ((400, ), 1.7320508), ((33, 5), 0.6)):
        value = torch.randn(*shape, generator=g)
        next_value = torch.randn(*shape, generator=g)
        reward = torch.randn(*shape, generator=g)
        done = (torch.rand(*shape, generator=g) < 0.05).float()
        traj = done.clone()
        traj[-1] = 1.0
        out.append((value, next_value, reward, done, traj, std))
    return out, g


def _default(v):
    if v is inspect.Parameter.empty:
        return {'empty': True}
    if callable(v):
        return {'type': type(v).__name__, 'name': getattr(v, '__name__', None)}
    return {'value': v}


def _mint_api(ref):
    import di_engine_b200 as b2
    fns, layout = {}, {}
    for name in b2.rl_utils.HOT_PATH_FUNCTIONS:
        fn = getattr(ref, name)
        fns[name] = {'module': fn.__module__,
                     'params': [[k, _default(p.default)] for k, p in inspect.signature(fn).parameters.items()]}
    for mod_name, mod in sorted(sys.modules.items()):
        if mod_name.startswith('ding.rl_utils.'):
            held = [n for n in b2.rl_utils.HOT_PATH_FUNCTIONS if getattr(mod, n, None) is getattr(ref, n)]
            if held:
                layout[mod_name] = held
    types_ = {name: list(getattr(ref, name)._fields) for name in b2.rl_utils.HOT_PATH_TYPES}
    with open(os.path.join(REF_DIR, 'api.json'), 'w') as f:
        json.dump({'functions': fns, 'types': types_, 'modules': layout}, f, indent=1, sort_keys=True)
        f.write('\n')


def sample_index(size):
    """the evenly spaced elements of a flattened output that bench_shapes.npz keeps when it is larger than SAMPLE"""
    return np.linspace(0, size - 1, SAMPLE).astype(np.int64)


def _mint_bench_shapes(ref):
    blob = {}
    for case, (op, tensors, params) in bench_shape_cases().items():
        for k, v in cases.run_api(ref, op, tensors, params).items():
            v = np.asarray(v)
            if v.size <= SAMPLE:
                blob[case + '/' + k] = v
                continue
            flat = v.reshape(-1)
            blob[case + '/' + k + '/sample'] = flat[sample_index(v.size)]
            blob[case + '/' + k + '/sums'] = np.array([flat.astype(np.float64).sum(), np.abs(flat.astype(np.float64)).sum()])
            blob[case + '/' + k + '/shape'] = np.array(v.shape, dtype=np.int64)
    np.savez_compressed(os.path.join(REF_DIR, 'bench_shapes.npz'), **blob)


def _mint_policy_gae(ref):
    blob = {}
    for i, (value, next_value, reward, done, traj, std) in enumerate(policy_gae_inputs()[0]):
        v, nv = value.clone(), next_value.clone()
        if std is not None:
            v *= std
            nv *= std
        blob['adv_%d' % i] = ref.gae(ref.gae_data(v, nv, reward, done, traj), 0.99, 0.95).numpy()
    np.savez_compressed(os.path.join(REF_DIR, 'policy_gae.npz'), **blob)


def _mint_suite_records():
    """runs the ported reference unit tests on the reference (their 'reference' parameter) and keeps every recorded value"""
    import pytest
    from tests import test_reference_suite as suite
    records = {}
    run = suite._run

    def recording_run(body, impl, *args):
        rec = suite.Rec()
        body(impl[0], impl[1], rec, *args)
        if impl[2] == 'reference':
            for k, v in rec.items():
                records[suite.record_key(body, args) + '::' + k] = v
        return rec

    suite._run = recording_run
    try:
        rc = pytest.main([suite.__file__, '-q', '-m', 'not gpu', '-k', 'not b200_dry', '-p', 'no:cacheprovider'])
    finally:
        suite._run = run
    assert rc == 0 and records, rc
    index, values, at = [], [], 0
    for k in sorted(records):
        v = records[k]
        index.append([k, at, list(v.shape)])
        values.append(v.astype(np.float32).reshape(-1))
        at += v.size
    np.savez_compressed(os.path.join(REF_DIR, 'suite_records.npz'), values=np.concatenate(values),
                        index=np.frombuffer(json.dumps(index).encode(), dtype=np.uint8))


def _mint_hpc_dispatch(ref):
    """what the reference's ENABLE_DI_HPC wrapper hands to hpc_rll for each call of test_host_logic.hpc_wrapper_calls"""
    import ding
    import ding.hpc_rl.wrapper as hw
    import di_engine_b200 as b2
    from di_engine_b200 import installer
    from tests import test_host_logic
    log, current = [], []

    def enc(x):
        for i, f in enumerate(current[-1]):
            if f is not None and x is f:
                return {'field': i}
        if x is None:
            return {'none': True}
        assert isinstance(x, (bool, int, float)), type(x)
        return {'value': x}

    class Recorder:

        def __init__(self, module, cls, *shape):
            self.entry = {'module': module, 'cls': cls, 'shape': list(shape)}

        def cuda(self):
            return self

        def __call__(self, *args, **kwargs):
            log.append(dict(self.entry, args=[enc(a) for a in args], kwargs={k: enc(v) for k, v in kwargs.items()}))

    b2.install_hpc_rll(force=True)
    for mod_name, classes in installer._HPC_LAYOUT.items():
        for cls in classes:
            setattr(sys.modules[mod_name], cls, lambda *shape, m=mod_name, c=cls: Recorder(m, c, *shape))
    hw.hpc_fns.clear()
    ding.enable_hpc_rl = True
    try:
        for fn, data, args, kwargs in test_host_logic.hpc_wrapper_calls(ref):
            current.append(data)
            getattr(ref, fn)(data, *args, **kwargs)
            log[-1]['fn'] = fn
    finally:
        ding.enable_hpc_rl = False
        hw.hpc_fns.clear()
        for k in list(sys.modules):
            if k == 'hpc_rll' or k.startswith('hpc_rll.'):
                del sys.modules[k]
    with open(os.path.join(REF_DIR, 'hpc_dispatch.json'), 'w') as f:
        json.dump(log, f, indent=1, sort_keys=True)
        f.write('\n')


def mint_reference_checks(ref):
    os.makedirs(REF_DIR, exist_ok=True)
    _mint_api(ref)
    _mint_hpc_dispatch(ref)
    _mint_bench_shapes(ref)
    _mint_policy_gae(ref)
    _mint_suite_records()
    print('wrote the reference checks to %s' % REF_DIR)


def _encode_params(params):
    out = {}
    for k, v in params.items():
        if isinstance(v, list):  # NGU list-gamma: list of 0-dim tensors
            out[k] = {'__tensor_list__': [float(x) for x in v]}
        else:
            out[k] = v
    return out


def main():
    torch.set_num_threads(1)
    ref = ref_loader.load()
    n = 0
    for name, (op, tensors, params) in cases.build_cases().items():
        if '--all' not in sys.argv and os.path.isfile(os.path.join(HERE, name + '.npz')):
            continue
        res = cases.run_api(ref, op, tensors, params)
        blob = {}
        meta = {'op': op, 'params': _encode_params(params), 'none_inputs': [], 'bool_inputs': [],
                'torch': torch.__version__}
        for k, v in tensors.items():
            if v is None:
                meta['none_inputs'].append(k)
            else:
                if v.dtype == torch.bool:
                    meta['bool_inputs'].append(k)
                blob['in_' + k] = v.numpy()
        blob.update(res)
        blob['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **blob)
        n += 1
    print('wrote %d fixtures to %s' % (n, HERE))
    mint_reference_checks(ref)


if __name__ == '__main__':
    main()
