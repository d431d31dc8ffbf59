"""The reference's OWN hot-path unit tests, ported and run against three implementations of the same API:

  reference   the unmodified ``ding.rl_utils`` (oracle/ref_loader.py: the tree in the build container, the byte-compiled
              archive oracle/_ref/ding_hotpath.zip elsewhere) on CPU tensors -- proves the port is a faithful harness;
  b200_dry    ``di_engine_b200.rl_utils`` on CPU with a recording stand-in for the CUDA library: shapes, autograd wiring,
              error behaviour and the host-side shape algebra, no GPU needed (values are uninitialised memory);
  b200        ``di_engine_b200.rl_utils`` on the GPU (``-m gpu``): every assertion of the reference's test AND value parity
              of every output and gradient against what the reference recorded on the same inputs (1e-5).

What the reference records is stored in ``tests/golden/reference/suite_records.npz`` (tests/golden/make_golden.py), so
the parity check needs no reference next to the GPU; the ``reference`` run checks those records against the reference.

Ported from ding/rl_utils/tests/test_gae.py, test_ppo.py (discrete, continuous, shape_fn), test_a2c.py (discrete), test_td.py (the operators on this
path: q_nstep, q_nstep_ngu, bdq_nstep, q_1step_compatible, dist_1step, dist_1step_compatible, dist_1step multi agent,
dist_nstep, dist_nstep multi agent, rescale, rescale_ngu, qrdqn_nstep, iqn_nstep, fqf_nstep, td_lambda, v_1step, v_1step multi agent, v_nstep, the four shape_fn
tests), test_vtrace.py (discrete), test_happo.py (discrete), test_retrace.py, test_upgo.py and test_value_rescale.py.  The reference draws unseeded random inputs; the
ports seed them (so the three implementations see identical bits) and keep every assertion.
"""
import contextlib
import functools
import json
import os

import numpy as np
import pytest
import torch

import di_engine_b200 as b2
from di_engine_b200 import _lib, ops
from oracle import ref_loader
from tests import golden_io

HAVE_REF = ref_loader.available()
RECORDS = os.path.join(golden_io.GOLDEN_DIR, 'reference', 'suite_records.npz')
IMPLS = [
    pytest.param('reference', marks=pytest.mark.skipif(not HAVE_REF, reason='reference not importable here')),
    pytest.param('b200_dry'),
    pytest.param('b200', marks=pytest.mark.gpu),
]


class _RecordingLib:
    """Stand-in for libb200rl.so: checks that every argument marshals to the declared ctypes prototype, computes nothing."""

    def __getattr__(self, name):
        proto = _lib.PROTOTYPES[name]

        def fn(*args):
            assert len(args) == len(proto), (name, len(args), len(proto))
            for a, ty in zip(args, proto):
                ty.from_param(a)
            return 1 if name.endswith('_supported') else 0

        if name == 'b200rl_workspace_bytes':
            return lambda: 1 << 20
        return fn


@pytest.fixture
def impl(request, monkeypatch):
    """-> (api namespace, device, kind)"""
    kind = request.param
    if kind == 'reference':
        torch.set_num_threads(1)
        return ref_loader.load(), 'cpu', kind
    if kind == 'b200_dry':
        rec = _RecordingLib()
        monkeypatch.setattr(ops, 'lib', lambda: rec)
        monkeypatch.setattr(ops, 'require_cuda', lambda: None)
        monkeypatch.setattr(ops, 'compute_device', lambda *t: torch.device('cpu'))
        monkeypatch.setattr(ops, 'stream_ptr', lambda: 0)
        monkeypatch.setattr(torch.cuda, 'device', lambda d: contextlib.nullcontext())
        monkeypatch.setattr(b2.rl_utils.td, 'CHECK_DIST_POSITIVE', False)
        monkeypatch.setattr(b2.rl_utils.ppo, 'LAZY_INFO', False)
        ops._WS.clear()
        return b2.rl_utils, 'cpu', kind
    return b2.rl_utils, 'cuda', kind


def pytest_generate_tests(metafunc):
    if 'impl' in metafunc.fixturenames:
        metafunc.parametrize('impl', IMPLS, indirect=True)


class Rec(dict):
    """named results of one ported test, for the cross-implementation value check"""

    def put(self, name, x):
        if isinstance(x, torch.Tensor):
            x = x.detach().cpu().numpy().copy()
        self[name] = np.asarray(x, dtype=np.float64)


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def record_key(body, args):
    """name of one run of a ported test body in the stored reference records"""
    return body.__qualname__ + repr(tuple(args))


@functools.lru_cache(maxsize=None)
def _reference_records():
    with np.load(RECORDS) as z:
        values, index = z['values'], json.loads(bytes(z['index']).decode())
    out = {}
    for name, at, shape in index:
        key, k = name.rsplit('::', 1)
        out.setdefault(key, {})[k] = values[at:at + int(np.prod(shape))].astype(np.float64).reshape(shape)
    return out


def _run(body, impl, *args):
    """Run a ported test body on ``impl``; on the GPU and on the reference compare every recorded value with what the
    reference recorded on the same inputs."""
    api, dev, kind = impl
    rec = Rec()
    body(api, dev, rec, *args)
    if kind in ('b200', 'reference'):
        want = _reference_records()[record_key(body, args)]
        assert set(rec) == set(want)
        for k in want:
            a, b = rec[k], want[k]
            assert a.shape == b.shape, (k, a.shape, b.shape)
            scale = max(1.0, float(np.max(np.abs(b)))) if k.startswith('grad') and b.size else 1.0
            assert np.allclose(a, b, rtol=1e-5, atol=1e-5 * scale, equal_nan=True), (k, float(np.max(np.abs(a - b))))
    return rec


# =================================================================================================================
# ding/rl_utils/tests/test_gae.py
# =================================================================================================================
def _gae_body(api, dev, rec):
    g = _gen(1)
    T, B = 32, 4  # batch trajectory case (test_gae.py:9-16)
    value, next_value, reward = (torch.randn(T, B, generator=g).to(dev) for _ in range(3))
    done = torch.zeros((T, B)).to(dev)
    adv = api.gae(api.gae_data(value, next_value, reward, done, None))
    assert adv.shape == (T, B)
    rec.put('adv_tb', adv)
    T = 24  # single trajectory / concat trajectory case (test_gae.py:17-25)
    value, next_value, reward = (torch.randn(T, generator=g).to(dev) for _ in range(3))
    done = torch.zeros((T)).to(dev)
    adv = api.gae(api.gae_data(value, next_value, reward, done, None))
    assert adv.shape == (T, )
    rec.put('adv_t', adv)


def test_gae(impl):
    _run(_gae_body, impl)


def _gae_marl_body(api, dev, rec):
    g = _gen(2)
    T, B, A = 32, 4, 8  # test_gae.py:28-36
    value = torch.randn(T, B, A, generator=g).to(dev)
    next_value = torch.randn(T, B, A, generator=g).to(dev)
    reward = torch.randn(T, B, generator=g).to(dev)
    done = torch.zeros(T, B).to(dev)
    adv = api.gae(api.gae_data(value, next_value, reward, done, None))
    assert adv.shape == (T, B, A)
    rec.put('adv', adv)


def test_gae_multi_agent(impl):
    _run(_gae_marl_body, impl)


# =================================================================================================================
# ding/rl_utils/tests/test_ppo.py
# =================================================================================================================
def test_shape_fn_ppo(impl):
    api = impl[0]
    data = api.ppo_data(torch.randn(3, 5, 8), None, None, None, None, None, None, None, None)
    shape1 = api.shape_fn_ppo([data], {})
    shape2 = api.shape_fn_ppo([], {'data': data})
    assert shape1 == shape2 == (3, 5, 8)


def _ppo_body(api, dev, rec, use_value_clip, dual_clip, weighted):
    g = _gen(3)
    B, N = 4, 32  # test_ppo.py:27-46
    weight = (torch.rand(4, generator=g) + 1).to(dev) if weighted else None
    logit_new = torch.randn(B, N, generator=g).to(dev).requires_grad_(True)
    logit_old = logit_new.detach() + torch.rand(B, N, generator=g).to(dev) * 0.1
    action = torch.randint(0, N, size=(B, ), generator=g).to(dev)
    value_new = torch.randn(B, generator=g).to(dev).requires_grad_(True)
    value_old = value_new.detach() + torch.rand(B, generator=g).to(dev) * 0.1
    adv = torch.rand(B, generator=g).to(dev)
    return_ = (torch.randn(B, generator=g) * 2).to(dev)
    data = api.ppo_data(logit_new, logit_old, action, value_new, value_old, adv, return_, weight, None)
    loss, info = api.ppo_error(data, use_value_clip=use_value_clip, dual_clip=dual_clip)
    assert all([l.shape == tuple() for l in loss])
    assert all([np.isscalar(i) for i in info])
    assert logit_new.grad is None
    assert value_new.grad is None
    total_loss = sum(loss)
    total_loss.backward()
    assert isinstance(logit_new.grad, torch.Tensor)
    assert isinstance(value_new.grad, torch.Tensor)
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    rec.put('approx_kl', info.approx_kl)
    rec.put('clipfrac', info.clipfrac)
    rec.put('grad_logit', logit_new.grad)
    rec.put('grad_value', value_new.grad)


@pytest.mark.parametrize('use_value_clip', [True, False])
@pytest.mark.parametrize('dual_clip', [None, 5.0])
@pytest.mark.parametrize('weighted', [False, True])
def test_ppo(impl, use_value_clip, dual_clip, weighted):
    _run(_ppo_body, impl, use_value_clip, dual_clip, weighted)


def _happo_body(api, dev, rec, use_value_clip, dual_clip, weighted):
    g = _gen(33)
    B, N = 4, 32  # tests/test_happo.py:27-45
    weight = (torch.rand(4, generator=g) + 1).to(dev) if weighted else None
    factor = torch.rand(4, 1, generator=g).to(dev)
    logit_new = torch.randn(B, N, generator=g).to(dev).requires_grad_(True)
    logit_old = logit_new.detach() + torch.rand(B, N, generator=g).to(dev) * 0.1
    action = torch.randint(0, N, size=(B, ), generator=g).to(dev)
    value_new = torch.randn(B, generator=g).to(dev).requires_grad_(True)
    value_old = value_new.detach() + torch.rand(B, generator=g).to(dev) * 0.1
    adv = torch.rand(B, generator=g).to(dev)
    return_ = (torch.randn(B, generator=g) * 2).to(dev)
    data = api.happo_data(logit_new, logit_old, action, value_new, value_old, adv, return_, weight, factor)
    loss, info = api.happo_error(data, use_value_clip=use_value_clip, dual_clip=dual_clip)
    assert all([l.shape == tuple() for l in loss])
    assert all([np.isscalar(i) for i in info])
    assert logit_new.grad is None
    assert value_new.grad is None
    total_loss = sum(loss)
    total_loss.backward()
    assert isinstance(logit_new.grad, torch.Tensor)
    assert isinstance(value_new.grad, torch.Tensor)
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    rec.put('approx_kl', info.approx_kl)
    rec.put('clipfrac', info.clipfrac)
    rec.put('grad_logit', logit_new.grad)
    rec.put('grad_value', value_new.grad)
    # the two halves, as HAPPOPolicy could call them (happo.py:81,150)
    ln2 = logit_new.detach().clone().requires_grad_(True)
    pl, pinfo = api.happo_policy_error(api.happo_policy_data(ln2, logit_old, action, adv, weight, factor), dual_clip=dual_clip)
    vl = api.happo_value_error(api.happo_value_data(value_new.detach(), value_old, return_, weight),
                               use_value_clip=use_value_clip)
    rec.put('half_policy', pl.policy_loss)
    rec.put('half_entropy', pl.entropy_loss)
    rec.put('half_value', vl)


@pytest.mark.parametrize('use_value_clip', [True, False])
@pytest.mark.parametrize('dual_clip', [None, 5.0])
@pytest.mark.parametrize('weighted', [False, True])
def test_happo(impl, use_value_clip, dual_clip, weighted):
    _run(_happo_body, impl, use_value_clip, dual_clip, weighted)


def _mappo_body(api, dev, rec):
    g = _gen(4)
    B, A, N = 4, 8, 32  # test_ppo.py:49-68
    logit_new = torch.randn(B, A, N, generator=g).to(dev).requires_grad_(True)
    logit_old = logit_new.detach() + torch.rand(B, A, N, generator=g).to(dev) * 0.1
    action = torch.randint(0, N, size=(B, A), generator=g).to(dev)
    value_new = torch.randn(B, A, generator=g).to(dev).requires_grad_(True)
    value_old = value_new.detach() + torch.rand(B, A, generator=g).to(dev) * 0.1
    adv = torch.rand(B, A, generator=g).to(dev)
    return_ = (torch.randn(B, A, generator=g) * 2).to(dev)
    data = api.ppo_data(logit_new, logit_old, action, value_new, value_old, adv, return_, None, None)
    loss, info = api.ppo_error(data)
    assert all([l.shape == tuple() for l in loss])
    assert all([np.isscalar(i) for i in info])
    assert logit_new.grad is None
    assert value_new.grad is None
    total_loss = sum(loss)
    total_loss.backward()
    assert isinstance(logit_new.grad, torch.Tensor)
    assert isinstance(value_new.grad, torch.Tensor)
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    rec.put('grad_logit', logit_new.grad)
    rec.put('grad_value', value_new.grad)


def test_mappo(impl):
    _run(_mappo_body, impl)


def _ppo_continuous_body(api, dev, rec, use_value_clip, dual_clip, weighted):
    g = _gen(30)
    B, N = 4, 6  # test_ppo.py:71-92
    weight = (torch.rand(4, generator=g) + 1).to(dev) if weighted else None
    mu_sigma_new = {'mu': torch.rand(B, N, generator=g).to(dev).requires_grad_(True),
                    'sigma': (torch.rand(B, N, generator=g) + 0.1).to(dev).requires_grad_(True)}
    mu_sigma_old = {
        'mu': mu_sigma_new['mu'].detach() + torch.rand(B, N, generator=g).to(dev) * 0.1,
        'sigma': mu_sigma_new['sigma'].detach() + torch.rand(B, N, generator=g).to(dev) * 0.1
    }
    action = torch.rand(B, N, generator=g).to(dev)
    value_new = torch.randn(B, generator=g).to(dev).requires_grad_(True)
    value_old = value_new.detach() + torch.rand(B, generator=g).to(dev) * 0.1
    adv = torch.rand(B, generator=g).to(dev)
    return_ = (torch.randn(B, generator=g) * 2).to(dev)
    data = api.ppo_data(mu_sigma_new, mu_sigma_old, action, value_new, value_old, adv, return_, weight, None)
    loss, info = api.ppo_error_continuous(data, use_value_clip=use_value_clip, dual_clip=dual_clip)
    assert all([l.shape == tuple() for l in loss])
    assert all([np.isscalar(i) for i in info])
    assert mu_sigma_new['mu'].grad is None
    assert value_new.grad is None
    total_loss = sum(loss)
    total_loss.backward()
    assert isinstance(mu_sigma_new['mu'].grad, torch.Tensor)
    assert isinstance(value_new.grad, torch.Tensor)
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    rec.put('approx_kl', info.approx_kl)
    rec.put('grad_mu', mu_sigma_new['mu'].grad)
    rec.put('grad_sigma', mu_sigma_new['sigma'].grad)
    rec.put('grad_value', value_new.grad)


@pytest.mark.parametrize('use_value_clip', [True, False])
@pytest.mark.parametrize('dual_clip', [None, 5.0])
@pytest.mark.parametrize('weighted', [False, True])
def test_ppo_error_continous(impl, use_value_clip, dual_clip, weighted):
    _run(_ppo_continuous_body, impl, use_value_clip, dual_clip, weighted)


# =================================================================================================================
# ding/rl_utils/tests/test_a2c.py (discrete)
# =================================================================================================================
def _a2c_body(api, dev, rec, weighted):
    g = _gen(31)
    B, N = 4, 32  # test_a2c.py:12-27
    weight = (torch.rand(4, generator=g) + 1).to(dev) if weighted else None
    logit = torch.randn(B, N, generator=g).to(dev).requires_grad_(True)
    action = torch.randint(0, N, size=(B, ), generator=g).to(dev)
    value = torch.randn(B, generator=g).to(dev).requires_grad_(True)
    adv = torch.rand(B, generator=g).to(dev)
    return_ = (torch.randn(B, generator=g) * 2).to(dev)
    data = api.a2c_data(logit, action, value, adv, return_, weight)
    loss = api.a2c_error(data)
    assert all([l.shape == tuple() for l in loss])
    assert logit.grad is None
    assert value.grad is None
    total_loss = sum(loss)
    total_loss.backward()
    assert isinstance(logit.grad, torch.Tensor)
    assert isinstance(value.grad, torch.Tensor)
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    rec.put('grad_logit', logit.grad)
    rec.put('grad_value', value.grad)


@pytest.mark.parametrize('weighted', [False, True])
def test_a2c(impl, weighted):
    _run(_a2c_body, impl, weighted)


# =================================================================================================================
# ding/rl_utils/tests/test_td.py
# =================================================================================================================
def _qntd_inputs(g, dev, batch_size=4, action_dim=3):
    next_q = torch.randn(batch_size, action_dim, generator=g).to(dev)
    done = torch.randn(batch_size, generator=g).to(dev)
    action = torch.randint(0, action_dim, size=(batch_size, ), generator=g).to(dev)
    next_action = torch.randint(0, action_dim, size=(batch_size, ), generator=g).to(dev)
    return next_q, done, action, next_action


def _q_nstep_td_body(api, dev, rec):
    g = _gen(5)
    batch_size, action_dim = 4, 3  # test_td.py:13-37
    next_q, done, action, next_action = _qntd_inputs(g, dev)
    for nstep in range(1, 10):
        q = torch.randn(batch_size, action_dim, generator=g).to(dev).requires_grad_(True)
        reward = torch.rand(nstep, batch_size, generator=g).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.q_nstep_td_error(data, 0.95, nstep=nstep)
        assert td_error_per_sample.shape == (batch_size, )
        assert loss.shape == ()
        assert q.grad is None
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('loss_%d' % nstep, loss)
        rec.put('td_%d' % nstep, td_error_per_sample)
        rec.put('grad_%d' % nstep, q.grad)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.q_nstep_td_error(data, 0.95, nstep=nstep, cum_reward=True)
        rec.put('cum_loss_%d' % nstep, loss)
        rec.put('cum_td_%d' % nstep, td_error_per_sample)  # (nstep, B): the (nstep, B) reward broadcasts
        value_gamma = torch.tensor(0.9).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.q_nstep_td_error(data, 0.95, nstep=nstep, cum_reward=True,
                                                         value_gamma=value_gamma)
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('cumvg_loss_%d' % nstep, loss)
        rec.put('cumvg_td_%d' % nstep, td_error_per_sample)
        rec.put('cumvg_grad_%d' % nstep, q.grad)  # accumulated over the two backward passes


def test_q_nstep_td(impl):
    _run(_q_nstep_td_body, impl)


def _bdq_nstep_td_body(api, dev, rec):
    g = _gen(6)
    batch_size, branch_num, action_per_branch = 8, 6, 3  # test_td.py:40-68
    next_q = torch.randn(batch_size, branch_num, action_per_branch, generator=g).to(dev)
    done = torch.randn(batch_size, generator=g).to(dev)
    action = torch.randint(0, action_per_branch, size=(batch_size, branch_num), generator=g).to(dev)
    next_action = torch.randint(0, action_per_branch, size=(batch_size, branch_num), generator=g).to(dev)
    for nstep in range(1, 10):
        q = torch.randn(batch_size, branch_num, action_per_branch, generator=g).to(dev).requires_grad_(True)
        reward = torch.rand(nstep, batch_size, generator=g).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.bdq_nstep_td_error(data, 0.95, nstep=nstep)
        assert td_error_per_sample.shape == (batch_size, )
        assert loss.shape == ()
        assert q.grad is None
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('loss_%d' % nstep, loss)
        rec.put('td_%d' % nstep, td_error_per_sample)
        rec.put('grad_%d' % nstep, q.grad)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.bdq_nstep_td_error(data, 0.95, nstep=nstep, cum_reward=True)
        rec.put('cum_loss_%d' % nstep, loss)
        rec.put('cum_td_%d' % nstep, td_error_per_sample)
        value_gamma = torch.tensor(0.9).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.bdq_nstep_td_error(data, 0.95, nstep=nstep, cum_reward=True,
                                                           value_gamma=value_gamma)
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('cumvg_loss_%d' % nstep, loss)
        rec.put('cumvg_grad_%d' % nstep, q.grad)


def test_bdq_nstep_td(impl):
    _run(_bdq_nstep_td_body, impl)


def _quantile_body(kind):
    """test_td.py:249-268 (qrdqn), :461-481 (iqn), :485-505 (fqf)"""

    def body(api, dev, rec):
        g = _gen({'qrdqn': 21, 'iqn': 22, 'fqf': 23}[kind])
        batch_size, action_dim, tau = 4, 3, 3
        shape = {'qrdqn': (batch_size, action_dim, tau), 'iqn': (tau, batch_size, action_dim),
                 'fqf': (batch_size, tau, action_dim)}[kind]
        next_q = torch.randn(*shape, generator=g).to(dev)
        done = torch.randn(batch_size, generator=g).to(dev)
        action = torch.randint(0, action_dim, size=(batch_size, ), generator=g).to(dev)
        next_action = torch.randint(0, action_dim, size=(batch_size, ), generator=g).to(dev)
        data_t = getattr(api, kind + '_nstep_td_data')
        fn = getattr(api, kind + '_nstep_td_error')
        for nstep in range(1, 10):
            q = torch.randn(*shape, generator=g).to(dev).requires_grad_(True)
            if kind == 'qrdqn':
                extra = tau  # a python int, as in the reference's test
            elif kind == 'iqn':
                extra = torch.randn([tau, batch_size, 1], generator=g).to(dev)
            else:
                extra = torch.randn([batch_size, tau], generator=g).to(dev)
            reward = torch.rand(nstep, batch_size, generator=g).to(dev)
            data = data_t(q, next_q, action, next_action, reward, done, extra, None)
            loss, td_error_per_sample = fn(data, 0.95, nstep=nstep)
            assert td_error_per_sample.shape == (batch_size, )
            assert loss.shape == ()
            assert q.grad is None
            loss.backward()
            assert isinstance(q.grad, torch.Tensor)
            rec.put('loss_%d' % nstep, loss)
            rec.put('td_%d' % nstep, td_error_per_sample)
            rec.put('grad_%d' % nstep, q.grad)
            loss, td_error_per_sample = fn(data, 0.95, nstep=nstep, value_gamma=torch.tensor(0.9).to(dev))
            assert td_error_per_sample.shape == (batch_size, )
            rec.put('vg_loss_%d' % nstep, loss)

    body.__qualname__ = '_quantile_body(%r)' % kind
    return body


@pytest.mark.parametrize('kind', ['qrdqn', 'iqn', 'fqf'])
def test_quantile_nstep_td(impl, kind):
    _run(_quantile_body(kind), impl)


def _q_retraces_body(api, dev, rec):
    g = _gen(31)
    T, B, N = 64, 32, 6  # tests/test_retrace.py:8-18
    q_values = torch.randn(T + 1, B, N, generator=g).to(dev)
    v_pred = torch.randn(T + 1, B, 1, generator=g).to(dev)
    rewards = torch.randn(T, B, generator=g).to(dev)
    ratio = (torch.rand(T, B, N, generator=g) * 0.4 + 0.8).to(dev)
    assert ratio.max() <= 1.2 and ratio.min() >= 0.8
    weights = torch.rand(T, B, generator=g).to(dev)
    actions = torch.randint(0, N, size=(T, B), generator=g).to(dev)
    with torch.no_grad():
        q_retraces = api.compute_q_retraces(q_values, v_pred, rewards, actions, weights, ratio, gamma=0.99)
    assert q_retraces.shape == (T + 1, B, 1)
    rec.put('q_retraces', q_retraces)


def test_compute_q_retraces(impl):
    _run(_q_retraces_body, impl)


def _q_nstep_td_ngu_body(api, dev, rec):
    g = _gen(7)
    batch_size, action_dim = 4, 3  # test_td.py:71-90
    next_q, done, action, next_action = _qntd_inputs(g, dev)
    gamma = [torch.tensor(0.95).to(dev) for i in range(batch_size)]
    for nstep in range(1, 10):
        q = torch.randn(batch_size, action_dim, generator=g).to(dev).requires_grad_(True)
        reward = torch.rand(nstep, batch_size, generator=g).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, td_error_per_sample = api.q_nstep_td_error(data, gamma, nstep=nstep)
        assert td_error_per_sample.shape == (batch_size, )
        assert loss.shape == ()
        assert q.grad is None
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('loss_%d' % nstep, loss)
        rec.put('td_%d' % nstep, td_error_per_sample)
        rec.put('grad_%d' % nstep, q.grad)


def test_q_nstep_td_ngu(impl):
    _run(_q_nstep_td_ngu_body, impl)


def _dist_inputs(g, dev, lead, action_dim=3, n_atom=51):
    dist = torch.randn(*lead, action_dim, n_atom, generator=g).abs().to(dev).requires_grad_(True)
    next_dist = torch.randn(*lead, action_dim, n_atom, generator=g).abs().to(dev)
    action = torch.randint(0, action_dim, size=lead, generator=g).to(dev)
    next_action = torch.randint(0, action_dim, size=lead, generator=g).to(dev)
    return dist, next_dist, action, next_action


def _dist_1step_td_body(api, dev, rec):
    g = _gen(8)
    batch_size, n_atom, v_min, v_max = 4, 51, -10.0, 10.0  # test_td.py:93-110
    dist, next_dist, action, next_action = _dist_inputs(g, dev, (batch_size, ))
    done = torch.randn(batch_size, generator=g).to(dev)
    reward = torch.randn(batch_size, generator=g).to(dev)
    data = api.dist_1step_td_data(dist, next_dist, action, next_action, reward, done, None)
    loss = api.dist_1step_td_error(data, 0.95, v_min, v_max, n_atom)
    assert loss.shape == ()
    assert dist.grad is None
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('grad', dist.grad)


def test_dist_1step_td(impl):
    _run(_dist_1step_td_body, impl)


def test_q_1step_compatible(impl):
    api, dev, kind = impl
    g = _gen(9)
    batch_size, action_dim = 4, 3  # test_td.py:113-126
    next_q, done, action, next_action = _qntd_inputs(g, dev)
    q = torch.randn(batch_size, action_dim, generator=g).to(dev).requires_grad_(True)
    reward = torch.rand(batch_size, generator=g).to(dev)
    nstep_data = api.q_nstep_td_data(q, next_q, action, next_action, reward.unsqueeze(0), done, None)
    onestep_data = api.q_1step_td_data(q, next_q, action, next_action, reward, done, None)
    nstep_loss, _ = api.q_nstep_td_error(nstep_data, 0.99, nstep=1)
    onestep_loss = api.q_1step_td_error(onestep_data, 0.99)
    if kind != 'b200_dry':
        assert pytest.approx(nstep_loss.item()) == onestep_loss.item()


def _dist_nstep_td_body(api, dev, rec):
    g = _gen(10)
    batch_size, n_atom, v_min, v_max, nstep = 4, 51, -10.0, 10.0, 5  # test_td.py:129-155
    dist, next_n_dist, action, next_action = _dist_inputs(g, dev, (batch_size, ))
    done = torch.randn(batch_size, generator=g).to(dev)
    reward = torch.randn(nstep, batch_size, generator=g).to(dev)
    data = api.dist_nstep_td_data(dist, next_n_dist, action, next_action, reward, done, None)
    loss, per = api.dist_nstep_td_error(data, 0.95, v_min, v_max, n_atom, nstep)
    assert loss.shape == ()
    assert dist.grad is None
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('td', per)
    rec.put('grad', dist.grad)
    weight = torch.tensor([0.9]).to(dev)
    value_gamma = torch.tensor(0.9).to(dev)
    data = api.dist_nstep_td_data(dist, next_n_dist, action, next_action, reward, done, weight)
    loss, per = api.dist_nstep_td_error(data, 0.95, v_min, v_max, n_atom, nstep, value_gamma)
    assert loss.shape == ()
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss_w', loss)
    rec.put('td_w', per)
    rec.put('grad_w', dist.grad)


def test_dist_nstep_td(impl):
    _run(_dist_nstep_td_body, impl)


def _dist_nstep_marl_body(api, dev, rec, dry):
    g = _gen(11)
    batch_size, agent_num, n_atom, v_min, v_max, nstep = 4, 2, 51, -10.0, 10.0, 5  # test_td.py:158-204
    dist, next_n_dist, action, next_action = _dist_inputs(g, dev, (batch_size, agent_num))
    done = torch.randint(0, 2, (batch_size, ), generator=g).to(dev)
    reward = torch.randn(nstep, batch_size, generator=g).to(dev)
    data = api.dist_nstep_td_data(dist, next_n_dist, action, next_action, reward, done, None)
    loss, _ = api.dist_nstep_td_error(data, 0.95, v_min, v_max, n_atom, nstep)
    assert loss.shape == ()
    assert dist.grad is None
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('grad', dist.grad)
    weight = 0.9
    value_gamma = 0.9
    data = api.dist_nstep_td_data(dist, next_n_dist, action, next_action, reward, done, weight)
    loss, _ = api.dist_nstep_td_error(data, 0.95, v_min, v_max, n_atom, nstep, value_gamma)
    assert loss.shape == ()
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss_w', loss)
    agent_total_loss = 0
    for i in range(agent_num):
        data = api.dist_nstep_td_data(dist[:, i, ], next_n_dist[:, i, ], action[:, i, ], next_action[:, i, ], reward,
                                      done, weight)
        agent_loss, _ = api.dist_nstep_td_error(data, 0.95, v_min, v_max, n_atom, nstep, value_gamma)
        agent_total_loss = agent_total_loss + agent_loss
    agent_average_loss = agent_total_loss / agent_num
    if not dry:
        assert abs(agent_average_loss.item() - loss.item()) < 1e-5


def test_dist_nstep_multi_agent_td(impl):
    _run(_dist_nstep_marl_body, impl, impl[2] == 'b200_dry')


def _rescale_body(api, dev, rec, ngu):
    g = _gen(12)
    batch_size, action_dim = 4, 3  # test_td.py:207-243
    next_q, done, action, next_action = _qntd_inputs(g, dev)
    gamma = [torch.tensor(0.95).to(dev) for i in range(batch_size)] if ngu else 0.95
    for nstep in range(1, 10):
        q = torch.randn(batch_size, action_dim, generator=g).to(dev).requires_grad_(True)
        reward = torch.rand(nstep, batch_size, generator=g).to(dev)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        loss, _ = api.q_nstep_td_error_with_rescale(data, gamma, nstep=nstep)
        assert loss.shape == ()
        assert q.grad is None
        loss.backward()
        assert isinstance(q.grad, torch.Tensor)
        rec.put('loss_%d' % nstep, loss)
        rec.put('grad_%d' % nstep, q.grad)


@pytest.mark.parametrize('ngu', [False, True])
def test_q_nstep_td_with_rescale(impl, ngu):
    _run(_rescale_body, impl, ngu)


def test_dist_1step_compatible(impl):
    api, dev, kind = impl
    g = _gen(13)
    batch_size, n_atom, v_min, v_max = 4, 51, -10.0, 10.0  # test_td.py:272-289
    dist, next_dist, action, next_action = _dist_inputs(g, dev, (batch_size, ))
    done = torch.randn(batch_size, generator=g).to(dev)
    reward = torch.randn(batch_size, generator=g).to(dev)
    onestep_data = api.dist_1step_td_data(dist, next_dist, action, next_action, reward, done, None)
    nstep_data = api.dist_nstep_td_data(dist, next_dist, action, next_action, reward.unsqueeze(0), done, None)
    onestep_loss = api.dist_1step_td_error(onestep_data, 0.95, v_min, v_max, n_atom)
    nstep_loss, _ = api.dist_nstep_td_error(nstep_data, 0.95, v_min, v_max, n_atom, nstep=1)
    if kind != 'b200_dry':
        assert pytest.approx(nstep_loss.item()) == onestep_loss.item()


def _dist_1step_marl_body(api, dev, rec, dry):
    g = _gen(14)
    batch_size, agent_num, n_atom, v_min, v_max = 4, 2, 51, -10.0, 10.0  # test_td.py:292-332
    dist, next_dist, action, next_action = _dist_inputs(g, dev, (batch_size, agent_num))
    done = torch.randint(0, 2, (batch_size, ), generator=g).to(dev)
    reward = torch.randn(batch_size, generator=g).to(dev)
    data = api.dist_1step_td_data(dist, next_dist, action, next_action, reward, done, None)
    loss = api.dist_1step_td_error(data, 0.95, v_min, v_max, n_atom)
    assert loss.shape == ()
    assert dist.grad is None
    loss.backward()
    assert isinstance(dist.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('grad', dist.grad)
    agent_total_loss = 0
    for i in range(agent_num):
        data = api.dist_1step_td_data(dist[:, i, ], next_dist[:, i, ], action[:, i, ], next_action[:, i, ], reward, done,
                                      None)
        agent_loss = api.dist_1step_td_error(data, 0.95, v_min, v_max, n_atom)
        agent_total_loss = agent_total_loss + agent_loss
    agent_average_loss = agent_total_loss / agent_num
    if not dry:
        assert abs(agent_average_loss.item() - loss.item()) < 1e-5


def test_dist_1step_multi_agent_td(impl):
    _run(_dist_1step_marl_body, impl, impl[2] == 'b200_dry')


def _td_lambda_body(api, dev, rec):
    g = _gen(15)
    T, B = 8, 4  # test_td.py:335-343
    value = torch.randn(T + 1, B, generator=g).to(dev).requires_grad_(True)
    reward = torch.rand(T, B, generator=g).to(dev)
    loss = api.td_lambda_error(api.td_lambda_data(value, reward, None))
    assert loss.shape == ()
    assert value.grad is None
    loss.backward()
    assert isinstance(value.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('grad', value.grad)


def test_td_lambda(impl):
    _run(_td_lambda_body, impl)


def _v_1step_body(api, dev, rec, agent_num):
    g = _gen(16)
    batch_size = 5  # test_td.py:346-380
    shape = (batch_size, ) if agent_num is None else (batch_size, agent_num)
    v = torch.randn(*shape, generator=g).to(dev).requires_grad_(True)
    next_v = torch.randn(*shape, generator=g).to(dev)
    reward = torch.rand(batch_size, generator=g).to(dev)
    done = torch.zeros(batch_size).to(dev)
    data = api.v_1step_td_data(v, next_v, reward, done, None)
    loss, td_error_per_sample = api.v_1step_td_error(data, 0.99)
    assert loss.shape == ()
    assert v.grad is None
    loss.backward()
    assert isinstance(v.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('td', td_error_per_sample)
    rec.put('grad', v.grad)
    data = api.v_1step_td_data(v, next_v, reward, None, None)
    loss, td_error_per_sample = api.v_1step_td_error(data, 0.99)
    loss.backward()
    assert isinstance(v.grad, torch.Tensor)
    rec.put('loss_nodone', loss)
    rec.put('grad_nodone', v.grad)


@pytest.mark.parametrize('agent_num', [None, 2])
def test_v_1step_td(impl, agent_num):
    _run(_v_1step_body, impl, agent_num)


def _v_nstep_body(api, dev, rec):
    g = _gen(17)
    batch_size = 5  # test_td.py:383-398
    v = torch.randn(batch_size, generator=g).to(dev).requires_grad_(True)
    next_v = torch.randn(batch_size, generator=g).to(dev)
    reward = torch.rand(5, batch_size, generator=g).to(dev)
    done = torch.zeros(batch_size).to(dev)
    data = api.v_nstep_td_data(v, next_v, reward, done, 0.9, 0.99)
    loss, td_error_per_sample = api.v_nstep_td_error(data, 0.99, 5)
    assert loss.shape == ()
    assert v.grad is None
    loss.backward()
    assert isinstance(v.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('td', td_error_per_sample)
    rec.put('grad', v.grad)
    data = api.v_nstep_td_data(v, next_v, reward, done, None, 0.99)
    loss, td_error_per_sample = api.v_nstep_td_error(data, 0.99, 5)
    loss.backward()
    assert isinstance(v.grad, torch.Tensor)
    rec.put('loss_now', loss)
    rec.put('grad_now', v.grad)


def test_v_nstep_td(impl):
    _run(_v_nstep_body, impl)


@pytest.mark.parametrize('fn', ['shape_fn_qntd', 'shape_fn_qntd_rescale'])
def test_shape_fn_qntd(impl, fn):
    api = impl[0]
    shape_fn = getattr(api, fn)
    g = _gen(18)
    batch_size, action_dim = 4, 3  # test_td.py:509-528, :557-576
    next_q, done, action, next_action = _qntd_inputs(g, 'cpu')
    for nstep in range(1, 10):
        q = torch.randn(batch_size, action_dim).requires_grad_(True)
        reward = torch.rand(nstep, batch_size)
        data = api.q_nstep_td_data(q, next_q, action, next_action, reward, done, None)
        for tmp in (shape_fn([data, 0.95, 1], {}), shape_fn([], {'gamma': 0.95, 'nstep': 1, 'data': data})):
            assert tmp[0] == reward.shape[0]
            assert tmp[1] == q.shape[0]
            assert tmp[2] == q.shape[1]


def test_shape_fn_dntd(impl):
    api = impl[0]
    g = _gen(19)
    batch_size, n_atom, v_min, v_max, nstep = 4, 51, -10.0, 10.0, 5  # test_td.py:531-554
    dist, next_n_dist, action, next_action = _dist_inputs(g, 'cpu', (batch_size, ))
    done = torch.randn(batch_size)
    reward = torch.randn(nstep, batch_size)
    data = api.dist_nstep_td_data(dist, next_n_dist, action, next_action, reward, done, None)
    for tmp in (api.shape_fn_dntd([data, 0.9, v_min, v_max, n_atom, nstep], {}),
                api.shape_fn_dntd([], {'data': data, 'gamma': 0.9, 'v_min': v_min, 'v_max': v_max, 'n_atom': n_atom,
                                       'nstep': 5})):
        assert tmp[0] == reward.shape[0]
        assert tmp[1] == dist.shape[0]
        assert tmp[2] == dist.shape[1]
        assert tmp[3] == n_atom


def test_fn_td_lambda(impl):
    api = impl[0]
    T, B = 8, 4  # test_td.py:579-588
    value = torch.randn(T + 1, B).requires_grad_(True)
    reward = torch.rand(T, B)
    data = api.td_lambda_data(value, reward, None)
    tmp = api.shape_fn_td_lambda([], {'data': data})
    assert tmp == reward.shape[0]
    tmp = api.shape_fn_td_lambda([data], {})
    assert tmp == reward.shape


# =================================================================================================================
# ding/rl_utils/tests/test_vtrace.py (discrete action)
# =================================================================================================================
def _vtrace_body(api, dev, rec):
    g = _gen(20)
    T, B, N = 4, 8, 16  # test_vtrace.py:7-22
    value = torch.randn(T + 1, B, generator=g).to(dev).requires_grad_(True)
    reward = torch.rand(T, B, generator=g).to(dev)
    target_output = torch.randn(T, B, N, generator=g).to(dev).requires_grad_(True)
    behaviour_output = torch.randn(T, B, N, generator=g).to(dev)
    action = torch.randint(0, N, size=(T, B), generator=g).to(dev)
    data = api.vtrace_data(target_output, behaviour_output, action, value, reward, None)
    loss = api.vtrace_error_discrete_action(data, rho_clip_ratio=1.1)
    assert all([l.shape == tuple() for l in loss])
    assert target_output.grad is None
    assert value.grad is None
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    loss = sum(loss)
    loss.backward()
    assert isinstance(target_output, torch.Tensor)
    assert isinstance(value, torch.Tensor)
    rec.put('grad_logit', target_output.grad)
    rec.put('grad_value', value.grad)


def test_vtrace_discrete_action(impl):
    _run(_vtrace_body, impl)


def _vtrace_continuous_body(api, dev, rec):
    g = _gen(32)
    T, B, N = 4, 8, 16  # test_vtrace.py:25-47
    value = torch.randn(T + 1, B, generator=g).to(dev).requires_grad_(True)
    reward = torch.rand(T, B, generator=g).to(dev)
    target_output = {}
    target_output['mu'] = torch.randn(T, B, N, generator=g).to(dev).requires_grad_(True)
    target_output['sigma'] = torch.exp(torch.randn(T, B, N, generator=g)).to(dev).requires_grad_(True)
    behaviour_output = {}
    behaviour_output['mu'] = torch.randn(T, B, N, generator=g).to(dev)
    behaviour_output['sigma'] = torch.exp(torch.randn(T, B, N, generator=g)).to(dev)
    action = torch.randn((T, B, N), generator=g).to(dev)
    data = api.vtrace_data(target_output, behaviour_output, action, value, reward, None)
    loss = api.vtrace_error_continuous_action(data, rho_clip_ratio=1.1)
    assert all([l.shape == tuple() for l in loss])
    assert target_output['mu'].grad is None
    assert target_output['sigma'].grad is None
    assert value.grad is None
    for k, v in zip(loss._fields, loss):
        rec.put(k, v)
    loss = sum(loss)
    loss.backward()
    assert isinstance(target_output['mu'], torch.Tensor)
    assert isinstance(target_output['sigma'], torch.Tensor)
    assert isinstance(value, torch.Tensor)
    rec.put('grad_mu', target_output['mu'].grad)
    rec.put('grad_sigma', target_output['sigma'].grad)
    rec.put('grad_value', value.grad)


def test_vtrace_continuous_action(impl):
    _run(_vtrace_continuous_body, impl)


# =================================================================================================================
# ding/rl_utils/tests/test_upgo.py
# =================================================================================================================
def _upgo_body(api, dev, rec):
    g = _gen(21)
    T, B, N, N2 = 4, 8, 5, 7  # test_upgo.py:7-43
    # tb_cross_entropy: 3 tests
    logit = torch.randn(T, B, N, N2, generator=g).softmax(-1).to(dev).requires_grad_(True)
    action = logit.argmax(-1).detach()
    ce = api.tb_cross_entropy(logit, action)
    assert ce.shape == (T, B)
    rec.put('ce_4d', ce)
    ce.sum().backward()
    rec.put('grad_ce_4d', logit.grad)

    logit = torch.randn(T, B, N, N2, 2, generator=g).softmax(-1).to(dev).requires_grad_(True)
    action = logit.argmax(-1).detach()
    with pytest.raises(AssertionError):
        ce = api.tb_cross_entropy(logit, action)

    logit = torch.randn(T, B, N, generator=g).softmax(-1).to(dev).requires_grad_(True)
    action = logit.argmax(-1).detach()
    ce = api.tb_cross_entropy(logit, action)
    assert ce.shape == (T, B)
    rec.put('ce_3d', ce)

    # upgo_returns
    rewards = torch.randn(T, B, generator=g).to(dev)
    bootstrap_values = torch.randn(T + 1, B, generator=g).to(dev).requires_grad_(True)
    returns = api.upgo_returns(rewards, bootstrap_values)
    assert returns.shape == (T, B)
    rec.put('returns', returns)

    # upgo loss
    rhos = torch.randn(T, B, generator=g).to(dev)
    loss = api.upgo_loss(logit, rhos, action, rewards, bootstrap_values)
    assert logit.requires_grad
    assert bootstrap_values.requires_grad
    for t in [logit, bootstrap_values]:
        assert t.grad is None
    loss.backward()
    for t in [logit]:
        assert isinstance(t.grad, torch.Tensor)
    rec.put('loss', loss)
    rec.put('grad_logit', logit.grad)
    # beyond the reference's test: upgo_returns is differentiable w.r.t. bootstrap_values there, and so here
    returns.sum().backward()
    assert isinstance(bootstrap_values.grad, torch.Tensor)
    rec.put('grad_bootstrap', bootstrap_values.grad)


def test_upgo(impl):
    _run(_upgo_body, impl)


# =================================================================================================================
# ding/rl_utils/tests/test_value_rescale.py
# =================================================================================================================
def test_value_rescale(impl):
    api, dev, kind = impl
    g = _gen(22)
    for _ in range(10):
        t = torch.rand((2, 3), generator=g).to(dev)
        assert isinstance(api.value_transform(t), torch.Tensor)
        assert api.value_transform(t).shape == t.shape
        assert isinstance(api.value_inv_transform(t), torch.Tensor)
        assert api.value_inv_transform(t).shape == t.shape
    for _ in range(10):
        t = torch.rand((4, 16), generator=g).to(dev)
        diff = api.value_inv_transform(api.value_transform(t)) - t
        assert pytest.approx(diff.abs().max().item(), abs=2e-5) == 0


# =================================================================================================================
# differentiability the reference has by construction (plain torch arithmetic) and its callers rely on
# =================================================================================================================
def _lambda_returns_grad_body(api, dev, rec):
    """generalized_lambda_returns back-propagates into bootstrap_values and rewards (MBSAC's actor loss,
    ding/policy/mbpolicy/mbsac.py:137,153; Dreamer's (H, B, 1) call, mbpolicy/utils.py:75) and into tensor gammas / lambdas."""
    g = _gen(23)
    T, B = 9, 5
    v = torch.randn(T + 1, B, generator=g).to(dev).requires_grad_(True)
    r = torch.randn(T, B, generator=g).to(dev).requires_grad_(True)
    done = (torch.rand(T, B, generator=g) < 0.2).float().to(dev)
    ret = api.generalized_lambda_returns(v, r, 0.99, 0.95, done)
    assert ret.shape == (T, B) and ret.requires_grad
    w = torch.randn(T, B, generator=g).to(dev)
    (ret * w).sum().backward()
    rec.put('ret', ret)
    rec.put('grad_v', v.grad)
    rec.put('grad_r', r.grad)
    gam = torch.rand(T, B, generator=g).to(dev)  # (the reference's in-place loop cannot differentiate w.r.t. these two;
    lam = torch.rand(T, B, generator=g).to(dev)  # tests/test_gpu_parity.py covers that superset of the product)
    v2 = v.detach().clone().requires_grad_(True)
    ret = api.generalized_lambda_returns(v2, r.detach(), gam, lam)
    (ret * w).sum().backward()
    rec.put('ret_t', ret)
    rec.put('grad_v_t', v2.grad)
    # Dreamer's layout: trailing singleton dim
    v3 = torch.randn(T + 1, B, 1, generator=g).to(dev).requires_grad_(True)
    r3 = torch.randn(T, B, 1, generator=g).to(dev)
    d3 = torch.rand(T, B, 1, generator=g).to(dev)
    ret = api.generalized_lambda_returns(v3, r3, d3, 0.95)
    assert ret.shape == (T, B, 1)
    ret.mean().backward()
    rec.put('ret_3d', ret)
    rec.put('grad_v_3d', v3.grad)


def test_generalized_lambda_returns_is_differentiable(impl):
    _run(_lambda_returns_grad_body, impl)


def _td_attached_body(api, dev, rec):
    """td_error_per_sample carries gradient in the reference (td.py:718-719): a loss built from it reaches q."""
    g = _gen(24)
    B, N, nstep = 6, 4, 3
    next_q, done, action, next_action = _qntd_inputs(g, dev, B, N)
    q = torch.randn(B, N, generator=g).to(dev).requires_grad_(True)
    reward = torch.rand(nstep, B, generator=g).to(dev)
    w = torch.rand(B, generator=g).to(dev)
    loss, per = api.q_nstep_td_error(api.q_nstep_td_data(q, next_q, action, next_action, reward, done, w), 0.97,
                                     nstep=nstep)
    assert per.requires_grad
    (0.3 * loss + (per * torch.arange(B, device=dev).float()).sum()).backward()
    rec.put('loss', loss)
    rec.put('td', per)
    rec.put('grad', q.grad)


def test_td_error_per_sample_is_attached(impl):
    _run(_td_attached_body, impl)


def _marl_qntd_body(api, dev, rec):
    """The reference's multi-agent branch (td.py:700-705): action (B, A, 1) against q (B, A, N)."""
    g = _gen(25)
    B, A, N, nstep = 5, 3, 4, 2
    q = torch.randn(B, A, N, generator=g).to(dev).requires_grad_(True)
    next_q = torch.randn(B, A, N, generator=g).to(dev)
    action = torch.randint(0, N, size=(B, A, 1), generator=g).to(dev)
    next_action = torch.randint(0, N, size=(B, A), generator=g).to(dev)
    reward = torch.rand(nstep, B, generator=g).to(dev)
    done = (torch.rand(B, generator=g) < 0.3).float().to(dev)
    weight = torch.rand(B, generator=g).to(dev)
    vg = torch.rand(B, generator=g).to(dev)
    loss, per = api.q_nstep_td_error(api.q_nstep_td_data(q, next_q, action, next_action, reward, done, weight), 0.9,
                                     nstep=nstep, value_gamma=vg)
    assert per.shape == (B, A)
    loss.backward()
    rec.put('loss', loss)
    rec.put('td', per)
    rec.put('grad', q.grad)


def test_q_nstep_td_multi_agent_branch(impl):
    _run(_marl_qntd_body, impl)


def test_q_nstep_td_inconsistent_multi_agent_shapes_raise_like_the_reference(impl):
    """q (B, A, N) with action (B, A) takes the reference's FIRST branch (td.py:695-699) whose n-step return then fails to
    broadcast (B,) against (B, A): a RuntimeError there, the same here (never a silent wrong answer)."""
    api, dev, kind = impl
    g = _gen(26)
    B, A, N = 5, 3, 4
    q = torch.randn(B, A, N, generator=g).to(dev)
    action = torch.randint(0, N, size=(B, A), generator=g).to(dev)
    reward = torch.rand(2, B, generator=g).to(dev)
    done = torch.zeros(B).to(dev)
    with pytest.raises(RuntimeError):
        api.q_nstep_td_error(api.q_nstep_td_data(q, q.clone(), action, action, reward, done, None), 0.9, nstep=2)
