"""CPU suite (-m "not gpu"): host-side logic of the product package, with NO compute.

* the C-ABI library loads and exports every symbol ``include/b200rl.h`` declares, and the ctypes prototypes agree
  with the header's parameter lists;
* the Python mirror of the reference interface: namedtuple fields, signatures/defaults, ``shape_fn_*`` return values
  (ding/rl_utils/tests/test_td.py:509-588, test_ppo.py:17-21), error behaviour (ppo.py:129, :54; td.py:257, :284, :854);
* every public operator marshals its arguments into the C entry points without error -- checked against a recording
  stand-in for the library (no kernel runs: there is no GPU here);
* ``install()`` / ``uninstall()`` rebinding and the ``hpc_rll`` shim layout (ding/hpc_rl/wrapper.py:62-73);
* the product refuses to run without CUDA (no CPU fallback) and never imports the oracle.
"""
import collections
import contextlib
import ctypes
import inspect
import json
import os
import re
import sys
import types

import pytest
import torch
import torch.nn as nn

import di_engine_b200 as b2
from di_engine_b200 import _lib, ops
from tests import cases, golden_io

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_decls():
    text = open(os.path.join(ROOT, 'include', 'b200rl.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    decls = {}
    for m in re.finditer(r'B200RL_API\s+(\w+)\s+(b200rl_\w+)\s*\((.*?)\)\s*;', text, flags=re.S):
        params = [p.strip() for p in m.group(3).split(',')]
        if params == ['void']:
            params = []
        decls[m.group(2)] = (m.group(1), params)
    return decls


def test_library_exports_every_declared_symbol():
    decls = _header_decls()
    assert len(decls) >= 19
    lib = _lib.load()
    for name in decls:
        assert hasattr(lib, name), name
    assert set(decls) == set(_lib.PROTOTYPES), set(decls) ^ set(_lib.PROTOTYPES)
    assert lib.b200rl_version() >= 100
    assert lib.b200rl_built_for_sm() == 100
    assert lib.b200rl_workspace_bytes() >= 1 << 20


def test_ctypes_prototypes_match_header():
    ctype_of = {'double': ctypes.c_double, 'int': ctypes.c_int, 'long long': ctypes.c_longlong,
                'size_t': ctypes.c_size_t}
    for name, (ret, params) in _header_decls().items():
        want = []
        for p in params:
            if '*' in p:
                want.append(ctypes.c_void_p)
            else:
                ty = re.sub(r'\s+\w+$', '', p.replace('const ', '')).strip()
                want.append(ctype_of[ty])
        assert _lib.PROTOTYPES[name] == want, name


def test_namedtuple_fields_match_reference():
    r = b2.rl_utils
    assert r.gae_data._fields == ('value', 'next_value', 'reward', 'done', 'traj_flag')  # gae.py:5
    assert r.ppo_data._fields == ('logit_new', 'logit_old', 'action', 'value_new', 'value_old', 'adv', 'return_',
                                  'weight', 'logit_pretrained')  # ppo.py:8-11
    assert r.ppo_loss._fields == ('policy_loss', 'value_loss', 'entropy_loss', 'kl_div')
    assert r.ppo_info._fields == ('approx_kl', 'clipfrac')
    assert r.q_nstep_td_data._fields == ('q', 'next_n_q', 'action', 'next_n_action', 'reward', 'done', 'weight')
    assert r.dist_nstep_td_data._fields == ('dist', 'next_n_dist', 'act', 'next_n_act', 'reward', 'done', 'weight')
    assert r.dist_nstep_td_data.__name__ == 'dist_1step_td_data'  # td.py:386
    assert r.td_lambda_data._fields == ('value', 'reward', 'weight')
    assert r.vtrace_data._fields == ('target_output', 'behaviour_output', 'action', 'value', 'reward', 'weight')
    assert r.vtrace_loss._fields == ('policy_loss', 'value_loss', 'entropy_loss')
    assert r.ppo_policy_data._fields == ('logit_new', 'logit_old', 'action', 'adv', 'weight', 'logit_pretrained')  # ppo.py:12-14
    assert r.ppo_policy_loss._fields == ('policy_loss', 'entropy_loss', 'kl_div')
    assert r.ppo_value_data._fields == ('value_new', 'value_old', 'return_', 'weight')
    assert r.q_1step_td_data._fields == ('q', 'next_q', 'act', 'next_act', 'reward', 'done', 'weight')  # td.py:14
    assert r.v_1step_td_data._fields == ('v', 'next_v', 'reward', 'done', 'weight')  # td.py:526
    assert r.v_nstep_td_data._fields == ('v', 'next_n_v', 'reward', 'done', 'weight', 'value_gamma')  # td.py:576


def test_signatures_match_reference_defaults():
    def sig(fn):
        return [(k, v.default) for k, v in inspect.signature(fn).parameters.items()]

    E = inspect.Parameter.empty
    r = b2.rl_utils
    assert sig(r.gae) == [('data', E), ('gamma', 0.99), ('lambda_', 0.97)]
    assert sig(r.ppo_error) == [('data', E), ('clip_ratio', 0.2), ('use_value_clip', True), ('dual_clip', None),
                                ('kl_type', 'k1')]
    assert sig(r.ppo_policy_error) == [('data', E), ('clip_ratio', 0.2), ('dual_clip', None), ('entropy_bonus', True),
                                       ('kl_type', 'k1')]  # ppo.py:143-149
    assert sig(r.ppo_value_error) == [('data', E), ('clip_ratio', 0.2), ('use_value_clip', True)]  # ppo.py:233-237
    assert [k for k, _ in sig(r.q_1step_td_error)] == ['data', 'gamma', 'criterion']  # td.py:26-30
    assert [k for k, _ in sig(r.v_1step_td_error)] == ['data', 'gamma', 'criterion']  # td.py:529-533
    assert [(k, d) for k, d in sig(r.v_nstep_td_error)][:3] == [('data', E), ('gamma', E), ('nstep', 1)]  # td.py:579-584
    s = sig(r.q_nstep_td_error)
    assert [k for k, _ in s] == ['data', 'gamma', 'nstep', 'cum_reward', 'value_gamma', 'criterion']
    assert s[2][1] == 1 and s[3][1] is False and s[4][1] is None and isinstance(s[5][1], nn.MSELoss)
    s = sig(r.q_nstep_td_error_with_rescale)
    assert [k for k, _ in s] == ['data', 'gamma', 'nstep', 'value_gamma', 'criterion', 'trans_fn', 'inv_trans_fn']
    assert s[5][1] is r.value_transform and s[6][1] is r.value_inv_transform
    assert sig(r.dist_nstep_td_error) == [('data', E), ('gamma', E), ('v_min', E), ('v_max', E), ('n_atom', E),
                                          ('nstep', 1), ('value_gamma', None)]
    assert sig(r.td_lambda_error) == [('data', E), ('gamma', 0.9), ('lambda_', 0.8)]
    assert sig(r.generalized_lambda_returns) == [('bootstrap_values', E), ('rewards', E), ('gammas', E),
                                                 ('lambda_', E), ('done', None)]
    assert sig(r.vtrace_error_discrete_action) == [('data', E), ('gamma', 0.99), ('lambda_', 0.95),
                                                   ('rho_clip_ratio', 1.0), ('c_clip_ratio', 1.0),
                                                   ('rho_pg_clip_ratio', 1.0)]
    assert sig(r.upgo_loss) == [('target_output', E), ('rhos', E), ('action', E), ('rewards', E),
                                ('bootstrap_values', E), ('mask', None)]


def _reference_api():
    with open(os.path.join(golden_io.GOLDEN_DIR, 'reference', 'api.json')) as f:
        return json.load(f)


def test_every_hot_path_signature_matches_the_live_reference():
    """every rebound function, against the unmodified reference (its signatures recorded in tests/golden/reference/api.json):
    same parameter names in the same order, same defaults (callables / modules by type or by name)"""
    ref = _reference_api()
    for name in b2.rl_utils.HOT_PATH_FUNCTIONS:
        ours, theirs = getattr(b2.rl_utils, name), ref['functions'].get(name)
        assert theirs is not None, name
        po, pt = inspect.signature(ours).parameters, dict(theirs['params'])
        assert list(po) == [k for k, _ in theirs['params']], (name, list(po), list(pt))
        for k in po:
            a, b = po[k].default, pt[k]
            if a is inspect.Parameter.empty or 'empty' in b:
                assert a is inspect.Parameter.empty and 'empty' in b, (name, k)
            elif callable(a) or 'type' in b:
                assert type(a).__name__ == b.get('type') or getattr(a, '__name__', None) == b.get('name'), (name, k)
            else:
                assert json.loads(json.dumps(a)) == b['value'], (name, k, a, b)
    for name in b2.rl_utils.HOT_PATH_TYPES:
        assert list(getattr(b2.rl_utils, name)._fields) == ref['types'][name], name


def test_shape_fns():
    r = b2.rl_utils
    d = r.gae_data(None, None, torch.zeros(5, 3), None, None)
    assert tuple(r.shape_fn_gae([d], {})) == (5, 3) and tuple(r.shape_fn_gae([], {'data': d})) == (5, 3)
    d = r.ppo_data(torch.zeros(7, 4), *[None] * 8)
    assert tuple(r.shape_fn_ppo([d], {})) == (7, 4) and tuple(r.shape_fn_ppo([], {'data': d})) == (7, 4)
    d = r.q_nstep_td_data(torch.zeros(4, 3), None, None, None, torch.zeros(5, 4), None, None)
    for fn in (r.shape_fn_qntd, r.shape_fn_qntd_rescale):
        assert fn([d], {}) == [5, 4, 3] and fn([], {'data': d}) == [5, 4, 3]
    d = r.dist_nstep_td_data(torch.zeros(4, 3, 51), None, None, None, torch.zeros(5, 4), None, None)
    assert r.shape_fn_dntd([d], {}) == [5, 4, 3, 51] and r.shape_fn_dntd([], {'data': d}) == [5, 4, 3, 51]
    d = r.td_lambda_data(None, torch.zeros(8, 4), None)
    assert tuple(r.shape_fn_td_lambda([d], {})) == (8, 4)
    assert r.shape_fn_td_lambda([], {'data': d}) == 8  # keyword form returns T only, td.py:1526-1527
    d = r.vtrace_data(torch.zeros(4, 8, 16), None, None, None, None, None)
    assert tuple(r.shape_fn_vtrace_discrete_action([d], {})) == (4, 8, 16)


def test_no_cpu_fallback_and_no_oracle_import(monkeypatch):
    """without a CUDA device every operator raises (simulated, so that the check also runs on a machine with a GPU)"""
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)
    t = torch.zeros(4, 3)
    with pytest.raises(_lib.B200RLError):
        b2.gae(b2.gae_data(t, t.clone(), t, None, None))
    with pytest.raises(_lib.B200RLError):
        b2.install()
    pkg_dir = os.path.join(ROOT, 'di-engine_b200')
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, flags=re.M), f
                assert 'rl_oracle' not in src and 'ref_loader' not in src, f


# ----------------------------------------------------------------------------------------------------------------
# marshalling dry run against a recording stand-in for the library (no kernels, no GPU)
# ----------------------------------------------------------------------------------------------------------------
class _RecordingLib:

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        proto = _lib.PROTOTYPES[name]

        def fn(*args):
            assert len(args) == len(proto), (name, len(args), len(proto))
            for a, ty in zip(args, proto):
                ty.from_param(a)  # raises on a type ctypes could not marshal
            self.calls.append(name)
            return 1 if name in ('b200rl_ppo_fused_supported', 'b200rl_vtrace_fused_supported') else 0

        if name == 'b200rl_workspace_bytes':
            return lambda: 1 << 20
        return fn


@pytest.fixture
def dry(monkeypatch):
    rec = _RecordingLib()
    monkeypatch.setattr(ops, 'lib', lambda: rec)
    monkeypatch.setattr(ops, 'require_cuda', lambda: None)
    monkeypatch.setattr(ops, 'compute_device', lambda *t: torch.device('cpu'))
    monkeypatch.setattr(ops, 'stream_ptr', lambda: 0)
    monkeypatch.setattr(torch.cuda, 'device', lambda d: contextlib.nullcontext())
    monkeypatch.setattr(b2.rl_utils.td, 'CHECK_DIST_POSITIVE', False)
    ops._WS.clear()
    yield rec
    ops._WS.clear()
    ops._CONST.clear()
    b2.rl_utils.td._SUPPORT_CACHE.clear()


EXPECTED_CALLS = {
    'gae': ['b200rl_gae'],
    'ppo': ['b200rl_ppo_fused_supported', 'b200rl_ppo_fwd_grad', 'b200rl_ppo_bwd'],
    'ppo_policy': ['b200rl_ppo_fused_supported', 'b200rl_ppo_fwd_grad', 'b200rl_ppo_bwd'],
    'ppo_value': ['b200rl_ppo_value_fwd', 'b200rl_scale'],
    'ppoc': ['b200rl_ppo_continuous_fwd_grad', 'b200rl_ppo_continuous_fwd_grad'],
    'a2c': ['b200rl_a2c_fwd_grad', 'b200rl_a2c_fwd_grad'],
    'vtc': ['b200rl_vtrace_continuous_fwd', 'b200rl_vtrace_continuous_bwd'],
    'qntd': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'qntd_rescale': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'q1td': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'v1td': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'vntd': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'dntd': ['b200rl_dntd_fwd', 'b200rl_dntd_bwd'],
    'bdq': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'qseq': ['b200rl_qntd_fwd', 'b200rl_qntd_bwd'],
    'd1td': ['b200rl_dntd_fwd', 'b200rl_dntd_bwd'],
    'td_lambda': ['b200rl_td_lambda_fwd', 'b200rl_scale'],
    'upgo': ['b200rl_lambda_returns', 'b200rl_upgo_head_fwd', 'b200rl_upgo_head_bwd'],
    'vtrace': ['b200rl_vtrace_fused_supported', 'b200rl_vtrace_fwd_grad', 'b200rl_vtrace_fwd_grad'],
    'qrdqn': ['b200rl_quantile_td_fwd', 'b200rl_quantile_td_bwd'],
    'iqn': ['b200rl_quantile_td_fwd', 'b200rl_quantile_td_bwd'],
    'fqf': ['b200rl_quantile_td_fwd', 'b200rl_quantile_td_bwd'],
    'retrace': ['b200rl_q_retraces'],
    'ppg': ['b200rl_ppo_value_fwd', 'b200rl_ppg_bc_fwd', 'b200rl_scale', 'b200rl_scale'],
    'happoc': ['b200rl_ppo_continuous_fwd_grad', 'b200rl_ppo_continuous_fwd_grad'],
    'acer': ['b200rl_acer_policy_fwd', 'b200rl_acer_value_fwd', 'b200rl_acer_policy_bwd', 'b200rl_acer_value_bwd',
             'b200rl_acer_trust_region'],
    'happo': ['b200rl_ppo_fused_supported', 'b200rl_ppo_fwd_grad', 'b200rl_ppo_bwd'],
}


@pytest.mark.parametrize('name', sorted(cases.build_cases().keys()))
def test_marshalling_dry_run(dry, name):
    op, tensors, params = cases.build_cases()[name]
    res = cases.run_api(b2.rl_utils, op, tensors, params)
    want = EXPECTED_CALLS[op]
    if op == 'gae' and tensors['value'].dim() == 1:
        want = ['b200rl_gae_returns']  # ONE sequence: the segment-parallel single-CTA kernel (csrc/policy.cu)
    assert dry.calls == want, dry.calls
    assert any(k.startswith('out_') for k in res)
    for k in cases.GRAD_INPUTS[op]:
        assert 'grad_' + k in res and res['grad_' + k].shape == tuple(tensors[k].shape)


def test_gae_ppo_error_dry_run_forward_and_backward(dry):
    """the one-launch step through the public API: every ctypes call (forward, verification) marshals to its prototype"""
    T, B, N = 8, 16, 6
    _, g, _ = cases.gae_case(50, T, B)
    _, t, _ = cases.ppo_case(51, T * B, N)
    tt = cases.prepare('ppo', t)
    gd = b2.gae_data(g['value'], g['next_value'], g['reward'], g['done'], g['traj_flag'])
    pd = b2.ppo_data(tt['logit_new'], tt['logit_old'], tt['action'], tt['value_new'], tt['value_old'], None, tt['return_'], None,
                     None)
    adv, loss, info = b2.gae_ppo_error(gd, pd, 0.99, 0.95, 0.2, True, None)
    (loss.policy_loss + 0.5 * loss.value_loss - 0.01 * loss.entropy_loss).backward()
    assert tt['logit_new'].grad is not None and tt['value_new'].grad is not None
    assert dry.calls[-1] == 'b200rl_ppo_bwd', dry.calls


def test_optional_index_range_check(dry, monkeypatch):
    """B200RL_CHECK_INDICES / ops.CHECK_INDICES: out-of-range actions raise IndexError before any pointer reaches a kernel
    (off by default: the check costs a device synchronisation)"""
    op, t, p = cases.ppo_case(3, 12, 5)
    bad = dict(t)
    bad['action'] = t['action'].clone()
    bad['action'][3] = 5
    data = b2.ppo_data(*bad.values())
    b2.ppo_error(data)  # unchecked by default
    monkeypatch.setattr(ops, 'CHECK_INDICES', True)
    dry.calls.clear()
    with pytest.raises(IndexError, match='out of range for 5 classes'):
        b2.ppo_error(data)
    assert dry.calls == []
    op, t, p = cases.qntd_case(4, 8, 4, 3)
    t = dict(t)
    t['next_n_action'] = t['next_n_action'].clone()
    t['next_n_action'][0] = -1
    with pytest.raises(IndexError, match='next_n_action'):
        b2.q_nstep_td_error(b2.q_nstep_td_data(*[t[k] for k in ('q', 'next_n_q', 'action', 'next_n_action', 'reward', 'done',
                                                                  'weight')]), 0.9, nstep=3)
    op, t, p = cases.vtrace_case(5, 6, 4, 3)
    b2.vtrace_error_discrete_action(b2.vtrace_data(*t.values()))  # in range: passes with the check on


def test_custom_criterion_and_transforms_dry_run(dry):
    op, t, p = cases.qntd_case(1, 8, 4, 3, weight='tensor')
    t = cases.prepare(op, t)
    data = b2.q_nstep_td_data(*[t[k] for k in ('q', 'next_n_q', 'action', 'next_n_action', 'reward', 'done', 'weight')])

    class Quartic(nn.Module):
        reduction = 'none'

        def forward(self, a, b):
            return (a - b) ** 4

    loss, per = b2.q_nstep_td_error(data, 0.9, nstep=3, criterion=Quartic())
    assert dry.calls == ['b200rl_qntd_fwd'] and per.shape == (8, )
    loss.backward()
    assert t['q'].grad is not None
    for crit in (nn.SmoothL1Loss(reduction='none'), nn.HuberLoss(reduction='none', delta=0.5),
                 nn.L1Loss(reduction='none')):
        dry.calls.clear()
        b2.q_nstep_td_error(data, 0.9, nstep=3, criterion=crit)
        assert dry.calls == ['b200rl_qntd_fwd']
    dry.calls.clear()
    loss, per = b2.q_nstep_td_error_with_rescale(data, 0.9, nstep=3, trans_fn=lambda x: x * 2,
                                                  inv_trans_fn=lambda x: x / 2)
    assert dry.calls == ['b200rl_qntd_fwd'] and per.shape == (8, )


def test_error_behaviour_matches_reference(dry):
    op, t, p = cases.ppo_case(1, 8, 4)
    data = b2.ppo_data(*t.values())
    with pytest.raises(AssertionError, match='dual_clip value must be greater than 1.0'):  # ppo.py:129
        b2.ppo_error(data, dual_clip=0.5)
    op, t, p = cases.ppo_case(1, 8, 4, pretrained=True)
    with pytest.raises(ValueError, match='Unknown kl_type'):  # ppo.py:54
        b2.ppo_error(b2.ppo_data(*t.values()), kl_type='k9')
    op, t, p = cases.qntd_case(1, 8, 4, 3)
    data = b2.q_nstep_td_data(*[t[k] for k in ('q', 'next_n_q', 'action', 'next_n_action', 'reward', 'done', 'weight')])
    with pytest.raises(TypeError, match='gamma should be float or list'):  # td.py:284
        b2.q_nstep_td_error(data, 1, nstep=3)
    with pytest.raises(AssertionError):  # td.py:257
        b2.q_nstep_td_error(data, 0.9, nstep=2)
    bad = data._replace(action=torch.zeros(8, 2, dtype=torch.long))
    with pytest.raises(AssertionError):  # td.py:854
        b2.q_nstep_td_error_with_rescale(bad, 0.9, nstep=3)
    with pytest.raises(TypeError, match='float32'):
        v = torch.zeros(4, 3, dtype=torch.float64)
        b2.gae(b2.gae_data(v, v.clone(), v, None, None))


def test_install_rebinds_and_uninstall_restores(dry, monkeypatch):
    def ref_gae(data, gamma=0.99, lambda_=0.97):
        return 'reference'

    def ref_ppo(data):
        return 'reference'

    fake = {}
    for name in ('ding', 'ding.rl_utils', 'ding.rl_utils.gae', 'ding.rl_utils.ppo', 'ding.policy', 'ding.policy.ppo',
                 'dizoo', 'dizoo.common', 'dizoo.common.policy', 'dizoo.common.policy.md_ppo', 'ding.rl_utils.adder'):
        fake[name] = types.ModuleType(name)
        monkeypatch.setitem(sys.modules, name, fake[name])
    for m in ('ding.rl_utils', 'ding.rl_utils.gae', 'ding.policy.ppo', 'dizoo.common.policy.md_ppo',
              'ding.rl_utils.adder'):
        fake[m].gae = ref_gae
    fake['ding.rl_utils'].ppo_error = ref_ppo
    fake['ding.rl_utils.ppo'].ppo_error = ref_ppo
    fake['ding.policy.ppo'].ppo_error = ref_ppo
    fake['ding.policy.ppo'].unrelated = ref_ppo
    done = b2.install(skip_modules=('ding.rl_utils.adder', ))
    assert ('ding.policy.ppo', 'gae') in done and ('ding.policy.ppo', 'ppo_error') in done
    assert fake['ding.policy.ppo'].gae is b2.rl_utils.gae
    assert fake['dizoo.common.policy.md_ppo'].gae is b2.rl_utils.gae
    assert fake['ding.rl_utils'].ppo_error is b2.rl_utils.ppo_error
    assert fake['ding.rl_utils.adder'].gae is ref_gae  # skipped
    assert fake['ding.policy.ppo'].unrelated is ref_ppo
    b2.uninstall()
    assert fake['ding.policy.ppo'].gae is ref_gae and fake['ding.rl_utils'].ppo_error is ref_ppo


def test_install_on_the_live_reference_rebinds_every_hot_path_function(dry, monkeypatch):
    """the module layout of the real ding.rl_utils (recorded in tests/golden/reference/api.json: which submodule defines each
    function, which submodules hold it): install() replaces every function of HOT_PATH_FUNCTIONS in the package namespace
    and in the submodule that defines it; a policy-like module that imported the names keeps working through the
    rebinding; uninstall() restores the originals"""
    api = _reference_api()
    pkg = types.ModuleType('ding.rl_utils')
    mods = {'ding': types.ModuleType('ding'), 'ding.rl_utils': pkg}
    for m in api['modules']:
        mods[m] = types.ModuleType(m)
    for name, mod in mods.items():
        monkeypatch.setitem(sys.modules, name, mod)

    def stand_in(name, module):
        def fn(*a, **k):
            return 'reference'
        fn.__name__, fn.__module__ = name, module
        return fn

    originals = {n: stand_in(n, api['functions'][n]['module']) for n in b2.rl_utils.HOT_PATH_FUNCTIONS}
    for n, fn in originals.items():
        setattr(pkg, n, fn)
    for m, held in api['modules'].items():
        for n in held:
            setattr(mods[m], n, originals[n])
    for n, fields in api['types'].items():
        setattr(pkg, n, collections.namedtuple(n, fields))
    ref = pkg
    policy = types.ModuleType('ding.policy.fake_for_install_test')
    for n, fn in originals.items():
        setattr(policy, n, fn)  # `from ding.rl_utils import ...` at import time
    sys.modules[policy.__name__] = policy
    try:
        done = b2.install()
        names = {n for _, n in done}
        assert names == set(b2.rl_utils.HOT_PATH_FUNCTIONS), set(b2.rl_utils.HOT_PATH_FUNCTIONS) - names
        for n in b2.rl_utils.HOT_PATH_FUNCTIONS:
            ours = getattr(b2.rl_utils, n)
            assert getattr(ref, n) is ours, n
            assert getattr(policy, n) is ours, n
            defining = sys.modules[originals[n].__module__]
            assert getattr(defining, n) is ours, (n, defining.__name__)
        # a rebound operator is callable through the reference's own namedtuple (positional unpacking)
        op, t, p = cases.gae_case(1, 6, 4)
        adv = policy.gae(ref.gae_data(t['value'], t['next_value'], t['reward'], t['done'], t['traj_flag']), 0.9, 0.8)
        assert adv.shape == (6, 4) and dry.calls[-1] == 'b200rl_gae'
    finally:
        b2.uninstall()
        del sys.modules[policy.__name__]
    for n, fn in originals.items():
        assert getattr(ref, n) is fn, n


def test_hpc_rll_shim_layout(monkeypatch):
    for k in list(sys.modules):
        if k == 'hpc_rll' or k.startswith('hpc_rll.'):
            monkeypatch.delitem(sys.modules, k)
    b2.install_hpc_rll()
    import importlib
    mapping = {  # ding/hpc_rl/wrapper.py:62-73 (the eight operators on this path)
        'gae': ['hpc_rll.rl_utils.gae', 'GAE'],
        'dist_nstep_td_error': ['hpc_rll.rl_utils.td', 'DistNStepTD'],
        'ppo_error': ['hpc_rll.rl_utils.ppo', 'PPO'],
        'q_nstep_td_error': ['hpc_rll.rl_utils.td', 'QNStepTD'],
        'q_nstep_td_error_with_rescale': ['hpc_rll.rl_utils.td', 'QNStepTDRescale'],
        'td_lambda_error': ['hpc_rll.rl_utils.td', 'TDLambda'],
        'upgo_loss': ['hpc_rll.rl_utils.upgo', 'UPGO'],
        'vtrace_error_discrete_action': ['hpc_rll.rl_utils.vtrace', 'VTrace'],
    }
    for fn, (mod, cls) in mapping.items():
        op = getattr(importlib.import_module(mod), cls)(4, 3).cuda()
        assert callable(op)
    for k in list(sys.modules):
        if k == 'hpc_rll' or k.startswith('hpc_rll.'):
            del sys.modules[k]


def test_packed_batch_layout():
    """PackedBatch (data.py): 256-byte aligned back-to-back layout, dtype / shape preserving views, None passthrough."""
    like = {'a': torch.arange(7, dtype=torch.float32), 'act': torch.arange(5, dtype=torch.int64).reshape(5, 1), 'none': None,
            'm': torch.ones(3, 4, 2)}
    pb = b2.PackedBatch(like, 'cpu')
    offs = [spec[0] for spec in pb.layout.values() if spec is not None]
    assert all(o % 256 == 0 for o in offs) and offs == sorted(offs)
    assert pb.payload_bytes() == 7 * 4 + 5 * 8 + 24 * 4
    d, ev = pb.upload()
    assert ev is None and d['none'] is None
    for k in ('a', 'act', 'm'):
        assert d[k].dtype == like[k].dtype and d[k].shape == like[k].shape and torch.equal(d[k], like[k])
    pb.host['a'].add_(1.0)
    assert torch.equal(pb.upload()[0]['a'], like['a'] + 1.0)


@pytest.mark.skipif(not __import__('oracle.ref_loader', fromlist=['x']).available(), reason='reference not importable here')
def test_live_hpc_wrapper_dispatches_into_the_shim(dry, monkeypatch):
    """The boundary end to end on the CPU box: the LIVE reference decorator (ding/hpc_rl/wrapper.py:86-133, the unmodified
    ding.rl_utils functions it wraps) with ``ding.enable_hpc_rl = True`` resolves ``hpc_rll.rl_utils.*`` to the classes
    ``install_hpc_rll()`` registers, constructs them as ``Class(*shape).cuda()``, caches them per shape (:74-83) and calls
    them with the whitelisted arguments -- which must reach the C ABI (here: the recording stand-in for the library)."""
    from oracle import ref_loader
    ref = ref_loader.load()  # puts the reference (tree or byte-compiled archive) on sys.path
    import ding
    import ding.hpc_rl.wrapper as hw
    for k in list(sys.modules):
        if k == 'hpc_rll' or k.startswith('hpc_rll.'):
            monkeypatch.delitem(sys.modules, k)
    b2.install_hpc_rll(force=True)
    monkeypatch.setattr(ding, 'enable_hpc_rl', True)
    hw.hpc_fns.clear()
    g = torch.Generator().manual_seed(5)
    try:
        # gae: include_args [0,1,2] -> hpc_fn(*data, gamma, lambda_)
        T, B = 16, 8
        d = ref.gae_data(torch.randn(T, B, generator=g), torch.randn(T, B, generator=g), torch.randn(T, B, generator=g),
                         torch.zeros(T, B), None)
        adv = ref.gae(d, 0.99, 0.95)
        assert dry.calls == ['b200rl_gae'] and adv.shape == (T, B)
        assert list(hw.hpc_fns['gae'].keys()) == ['gae_%d_%d' % (T, B)]  # runtime_name = fn name + shape_fn(...) (:97)
        ref.gae(d, gamma=0.9, lambda_=0.8)  # keyword form: 'lambda_' is renamed 'lambda' by the wrapper (:113-114)
        assert dry.calls == ['b200rl_gae'] * 2 and len(hw.hpc_fns['gae']) == 1  # cached instance reused
        # ppo_error: hpc_fn(*data (9 fields), clip_ratio, use_value_clip, dual_clip)
        dry.calls.clear()
        op, t, p = cases.ppo_case(3, 12, 5, weight='tensor')
        tt = cases.prepare(op, t)
        data = ref.ppo_data(*[tt[k] for k in ('logit_new', 'logit_old', 'action', 'value_new', 'value_old', 'adv', 'return_',
                                              'weight', 'logit_pretrained')])
        loss, info = ref.ppo_error(data, 0.2, True, None)
        assert dry.calls[:2] == ['b200rl_ppo_fused_supported', 'b200rl_ppo_fwd_grad'] and len(loss) == 4
        # q_nstep_td_error: only (data, gamma) are forwarded (:648); nstep is re-derived from the reward tensor by the shim
        dry.calls.clear()
        op, t, p = cases.qntd_case(4, 8, 4, 3)
        data = ref.q_nstep_td_data(*[t[k] for k in ('q', 'next_n_q', 'action', 'next_n_action', 'reward', 'done', 'weight')])
        loss, per = ref.q_nstep_td_error(data, 0.95, nstep=3)
        assert dry.calls == ['b200rl_qntd_fwd'] and per.shape == (8, )
        # dist_nstep_td_error: (data, gamma, v_min, v_max) forwarded, n_atom / nstep dropped with a warning (:407-412)
        dry.calls.clear()
        op, t, p = cases.dntd_case(5, 6, 3, 51, 2)
        data = ref.dist_nstep_td_data(*[t[k] for k in ('dist', 'next_n_dist', 'act', 'next_n_act', 'reward', 'done', 'weight')])
        loss, per = ref.dist_nstep_td_error(data, 0.95, -10., 10., 51, 2)
        assert dry.calls == ['b200rl_dntd_fwd'] and per.shape == (6, )
        # td_lambda_error and vtrace_error_discrete_action
        dry.calls.clear()
        op, t, p = cases.td_lambda_case(6, 8, 4)
        ref.td_lambda_error(ref.td_lambda_data(t['value'], t['reward'], t['weight']), 0.9, 0.8)
        assert dry.calls == ['b200rl_td_lambda_fwd']
        dry.calls.clear()
        op, t, p = cases.vtrace_case(7, 4, 8, 6)
        ref.vtrace_error_discrete_action(ref.vtrace_data(*[t[k] for k in ('target_output', 'behaviour_output', 'action',
                                                                          'value', 'reward', 'weight')]), 0.99, 0.95)
        assert dry.calls[:2] == ['b200rl_vtrace_fused_supported', 'b200rl_vtrace_fwd_grad']
        # per_fn_limit = 3 shapes per function, FIFO eviction (:80-81)
        for Tn in (3, 4, 5, 6):
            dn = ref.gae_data(torch.zeros(Tn, 2), torch.zeros(Tn, 2), torch.zeros(Tn, 2), None, None)
            ref.gae(dn)
        assert len(hw.hpc_fns['gae']) == 3 and 'gae_%d_%d' % (T, B) not in hw.hpc_fns['gae']
    finally:
        hw.hpc_fns.clear()
        for k in list(sys.modules):
            if k == 'hpc_rll' or k.startswith('hpc_rll.'):
                del sys.modules[k]


def hpc_wrapper_calls(api):
    """(operator, data, positional, keyword arguments): the calls of the test above, through ``api``'s namedtuples"""
    g = torch.Generator().manual_seed(5)
    T, B = 16, 8
    d = api.gae_data(torch.randn(T, B, generator=g), torch.randn(T, B, generator=g), torch.randn(T, B, generator=g),
                     torch.zeros(T, B), None)
    yield 'gae', d, (0.99, 0.95), {}
    yield 'gae', d, (), {'gamma': 0.9, 'lambda_': 0.8}
    op, t, p = cases.ppo_case(3, 12, 5, weight='tensor')
    tt = cases.prepare(op, t)
    yield 'ppo_error', api.ppo_data(*[tt[k] for k in ('logit_new', 'logit_old', 'action', 'value_new', 'value_old', 'adv',
                                                      'return_', 'weight', 'logit_pretrained')]), (0.2, True, None), {}
    op, t, p = cases.qntd_case(4, 8, 4, 3)
    yield 'q_nstep_td_error', api.q_nstep_td_data(*[t[k] for k in ('q', 'next_n_q', 'action', 'next_n_action', 'reward',
                                                                   'done', 'weight')]), (0.95, ), {'nstep': 3}
    op, t, p = cases.dntd_case(5, 6, 3, 51, 2)
    yield 'dist_nstep_td_error', api.dist_nstep_td_data(*[t[k] for k in ('dist', 'next_n_dist', 'act', 'next_n_act', 'reward',
                                                                         'done', 'weight')]), (0.95, -10., 10., 51, 2), {}
    op, t, p = cases.td_lambda_case(6, 8, 4)
    yield 'td_lambda_error', api.td_lambda_data(t['value'], t['reward'], t['weight']), (0.9, 0.8), {}
    op, t, p = cases.vtrace_case(7, 4, 8, 6)
    yield 'vtrace_error_discrete_action', api.vtrace_data(*[t[k] for k in ('target_output', 'behaviour_output', 'action',
                                                                           'value', 'reward', 'weight')]), (0.99, 0.95), {}
    for Tn in (3, 4, 5, 6):
        yield 'gae', api.gae_data(torch.zeros(Tn, 2), torch.zeros(Tn, 2), torch.zeros(Tn, 2), None, None), (), {}


HPC_SHAPE_FN = {'gae': 'shape_fn_gae', 'ppo_error': 'shape_fn_ppo', 'q_nstep_td_error': 'shape_fn_qntd',
                'dist_nstep_td_error': 'shape_fn_dntd', 'td_lambda_error': 'shape_fn_td_lambda',
                'vtrace_error_discrete_action': 'shape_fn_vtrace_discrete_action'}
HPC_FIRST_CALLS = {'gae': ['b200rl_gae'], 'ppo_error': ['b200rl_ppo_fused_supported', 'b200rl_ppo_fwd_grad'],
                   'q_nstep_td_error': ['b200rl_qntd_fwd'], 'dist_nstep_td_error': ['b200rl_dntd_fwd'],
                   'td_lambda_error': ['b200rl_td_lambda_fwd'],
                   'vtrace_error_discrete_action': ['b200rl_vtrace_fused_supported', 'b200rl_vtrace_fwd_grad']}


def test_recorded_hpc_wrapper_dispatch_reaches_the_c_abi(dry, monkeypatch):
    """What the reference's decorator (ding/hpc_rl/wrapper.py:86-133) with ``ding.enable_hpc_rl = True`` hands to
    ``hpc_rll`` for each call of ``hpc_wrapper_calls``, recorded from the live reference in
    tests/golden/reference/hpc_dispatch.json: the module and class it imports, the shape it constructs them with (which
    this package's ``shape_fn_*`` must reproduce) and the arguments it keeps.  Replayed against the classes
    ``install_hpc_rll()`` registers, every call must reach the C ABI (here: the recording stand-in for the library)."""
    import importlib
    with open(os.path.join(golden_io.GOLDEN_DIR, 'reference', 'hpc_dispatch.json')) as f:
        recorded = json.load(f)
    for k in list(sys.modules):
        if k == 'hpc_rll' or k.startswith('hpc_rll.'):
            monkeypatch.delitem(sys.modules, k)
    b2.install_hpc_rll(force=True)
    calls = list(hpc_wrapper_calls(b2.rl_utils))
    assert len(calls) == len(recorded)
    try:
        for (fn, data, args, kwargs), r in zip(calls, recorded):
            assert r['fn'] == fn
            assert list(getattr(b2.rl_utils, HPC_SHAPE_FN[fn])((data, ) + tuple(args), kwargs)) == r['shape'], fn

            def arg(x):
                return data[x['field']] if 'field' in x else x.get('value')

            dry.calls.clear()
            op = getattr(importlib.import_module(r['module']), r['cls'])(*r['shape']).cuda()
            op(*[arg(x) for x in r['args']], **{k: arg(v) for k, v in r['kwargs'].items()})
            assert dry.calls[:len(HPC_FIRST_CALLS[fn])] == HPC_FIRST_CALLS[fn], (fn, dry.calls)
    finally:
        for k in list(sys.modules):
            if k == 'hpc_rll' or k.startswith('hpc_rll.'):
                del sys.modules[k]
