"""CPU suite (-m "not gpu"): pins the oracle restatement.

1. against the committed golden fixtures (outputs of the unmodified reference, see tests/golden/make_golden.py);
2. against what the unmodified reference computed, bit-exact, since the oracle uses the same torch primitives in the
   same order (the fixtures, and ``tests/golden/reference/`` for the medium shapes and the policy-level lines);
3. relational identities the reference's own tests hold (tests/test_td.py:113-126, :196-204,
   tests/test_value_rescale.py:21-26).
"""
import os

import numpy as np
import pytest
import torch

from oracle import rl_oracle
from tests import cases, golden_io
from tests.golden import make_golden

CASES = cases.build_cases()
REF_DIR = os.path.join(golden_io.GOLDEN_DIR, 'reference')


def test_fixture_set_matches_case_registry():
    assert sorted(CASES.keys()) == golden_io.names()


@pytest.mark.parametrize('name', golden_io.names())
def test_oracle_matches_golden(name):
    op, tensors, params, expected = golden_io.load(name)
    res = cases.run_oracle(rl_oracle, op, tensors, params)
    # same torch build; another host CPU may vectorise exp/log differently -> 1-2 ulp. gae is pure mul/add: exact.
    if op in ('gae', 'retrace'):
        cases.compare(res, expected, exact=True)
    else:
        cases.compare(res, expected, rtol=2e-6, atol=2e-6)


@pytest.mark.parametrize('name', golden_io.names())
def test_case_builders_reproduce_fixture_inputs(name):
    """The seeded builders regenerate exactly the inputs stored in the fixtures (so big-size GPU tests can rely on
    the builders while small-size tests rely on the fixtures)."""
    op, tensors, params, _ = golden_io.load(name)
    op2, tensors2, params2 = CASES[name]
    assert op == op2
    for k, v in tensors2.items():
        if v is None:
            assert tensors.get(k) is None
        else:
            assert torch.equal(v, tensors[k]), k


@pytest.mark.parametrize('name', sorted(CASES.keys()))
def test_oracle_bit_exact_vs_live_reference(name):
    """bit for bit against the reference's outputs stored in the fixture (single-threaded on both sides)"""
    op, tensors, params = CASES[name]
    torch.set_num_threads(1)
    want = golden_io.load(name)[3]
    got = cases.run_oracle(rl_oracle, op, tensors, params)
    cases.compare(got, want, exact=True)


def test_oracle_vs_live_reference_bench_shapes():
    """Medium shapes of the five BASELINE configs (kept to a few seconds), against the reference's outputs stored in
    tests/golden/reference/bench_shapes.npz: small outputs whole, large ones as a fixed sample plus their sums."""
    with np.load(os.path.join(REF_DIR, 'bench_shapes.npz')) as z:
        want = {k: z[k] for k in z.files}
    for name, (op, tensors, params) in make_golden.bench_shape_cases().items():
        got = cases.run_oracle(rl_oracle, op, tensors, params)
        keys = {k.split('/')[1] for k in want if k.startswith(name + '/')}
        assert keys == set(got), (name, keys, set(got))
        for k in sorted(keys):
            a, w = np.asarray(got[k]), name + '/' + k
            if w in want:
                assert np.allclose(a, want[w], rtol=1e-6, atol=1e-6), (w, float(np.max(np.abs(a - want[w]))))
                continue
            assert a.shape == tuple(want[w + '/shape']), w
            flat = a.reshape(-1)
            sample = flat[make_golden.sample_index(flat.size)]
            assert np.allclose(sample, want[w + '/sample'], rtol=1e-6, atol=1e-6), (w, float(np.max(np.abs(sample - want[w + '/sample']))))
            total, abs_total = want[w + '/sums']
            assert abs(flat.astype(np.float64).sum() - total) <= 1e-6 * abs_total + 1e-6, w


def test_nstep1_equals_one_step_form():
    """tests/test_td.py:113-126: n-step(1) == r + gamma*(1-done)*q' one-step TD."""
    g = torch.Generator().manual_seed(0)
    B, N = 16, 5
    q = torch.randn(B, N, generator=g)
    nq = torch.randn(B, N, generator=g)
    a = torch.randint(0, N, (B, ), generator=g)
    na = torch.randint(0, N, (B, ), generator=g)
    r = torch.rand(B, generator=g)
    d = (torch.rand(B, generator=g) < 0.3).float()
    loss, per = rl_oracle.q_nstep_td_error(q, nq, a, na, r.unsqueeze(0), d, None, gamma=0.99, nstep=1)
    tgt = r + 0.99 * (1 - d) * nq[torch.arange(B), na]
    want = (q[torch.arange(B), a] - tgt) ** 2
    assert torch.allclose(per, want, atol=1e-6)
    assert abs(loss.item() - want.mean().item()) < 1e-6


def test_dist_nstep_multi_agent_equals_mean_of_agents():
    """tests/test_td.py:159-204: joint multi-agent loss == mean of the per-agent losses (<1e-5)."""
    op, t, p = cases.dntd_case(7, 4, 3, 51, 5, marl_A=2)
    joint, _ = rl_oracle.dist_nstep_td_error(**t, **p)
    parts = []
    for a in range(2):
        la, _ = rl_oracle.dist_nstep_td_error(
            t['dist'][:, a], t['next_n_dist'][:, a], t['act'][:, a], t['next_n_act'][:, a], t['reward'], t['done'],
            None, **p
        )
        parts.append(la)
    assert abs(joint.item() - torch.stack(parts).mean().item()) < 1e-5


def test_value_rescale_round_trip():
    """tests/test_value_rescale.py:21-26."""
    x = torch.randn(64) * 20
    assert (rl_oracle.value_inv_transform(rl_oracle.value_transform(x)) - x).abs().max() < 2e-5 * 20


def test_projection_conserves_mass():
    """C51 projection property: every projected row still sums to the mass of the source row."""
    op, t, p = cases.dntd_case(9, 32, 4, 51, 3, integer_bins=True, gamma=1.0)
    # td_per_sample = -sum_j log p_j m_j ; with dist == uniform, log p is constant -> td = -log(1/n) * sum m
    t = dict(t)
    t['dist'] = torch.full_like(t['dist'], 1.0 / 51)
    _, per = rl_oracle.dist_nstep_td_error(**t, **p)
    assert torch.allclose(per, torch.full_like(per, float(np.log(51.0))), atol=1e-5)


def test_policy_level_restatements_match_the_reference_lines():
    """ding/policy/ppo.py cannot be imported (it pulls the whole framework), so its lines :276-292 and :304-306 are executed
    here literally around the reference gae (its outputs on these inputs are stored in tests/golden/reference/policy_gae.npz)
    and compared with the oracle's restatement, bit for bit."""
    inputs, g = make_golden.policy_gae_inputs()
    with np.load(os.path.join(REF_DIR, 'policy_gae.npz')) as z:
        ref_adv = [torch.from_numpy(z['adv_%d' % i]) for i in range(len(inputs))]
    for (value, next_value, reward, done, traj, std), adv in zip(inputs, ref_adv):
        got = rl_oracle.ppo_policy_gae_returns(value, next_value, reward, done, traj, 0.99, 0.95, std)
        v = value.clone()
        if std is not None:
            v *= std
        unnormalized_returns = v + adv
        if std is not None:
            val, ret = v / std, unnormalized_returns / std
        else:
            val, ret = v, unnormalized_returns
        for a, b in zip(got[:4], (adv, val, ret, unnormalized_returns)):
            assert torch.equal(a, b)
        x = unnormalized_returns.numpy().reshape(-1)
        assert got[4] == (float(np.mean(x)), float(np.var(x)), float(x.shape[0]))
    adv = torch.randn(320, generator=g) * 3 + 1
    assert torch.equal(rl_oracle.normalize_advantage(adv), (adv - adv.mean()) / (adv.std() + 1e-8))
    # IMPALAPolicy._reshape_data, policy/impala.py:316-322, executed literally
    values = torch.randn(9, 4, generator=g)
    rewards = torch.rand(8, 4, generator=g)
    done = (torch.rand(8, 4, generator=g) < 0.3)
    got = rl_oracle.impala_reshape_data(values, rewards, done)
    v = values.clone()
    weights_ = 1 - done.float()
    weights = torch.ones_like(rewards)
    v[1:] = v[1:] * weights_
    weights[1:] = weights_[:-1]
    r = rewards * weights
    assert torch.equal(got[0], v) and torch.equal(got[1], r) and torch.equal(got[2], weights)
