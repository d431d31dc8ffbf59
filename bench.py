#!/usr/bin/env python
"""Benchmark of the learner hot path (BASELINE.json): trajectory return/advantage + policy-loss operators, forward AND
backward, on synthetic batches of the reference's shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-cuda]
                    [--config D|B|C|E] [--scaling weak|strong] [--dump-outputs DIR]

Configs (BASELINE.json `configs`, SURVEY.md section 8d):
  D (default, the metric of record)  Atari PPO: gae -> ppo_error, T=128, B=4096, N=6 per GPU (`--scaling strong`: B=4096 in
                                     total, sharded), gamma 0.99, lambda 0.95, clip 0.2, value clip on
  B                                  Pong DQN: q_nstep_td_error, B=512, N=6, nstep=3, value_gamma tensor
  C                                  Atari C51: dist_nstep_td_error, B=512, N=6, 51 atoms, nstep=3
  E                                  IMPALA: vtrace_error_discrete_action, T=64, B=8192, N=6 per GPU
One step = one pass of the config's operators, forward and backward, over one batch.

  value     inputs resident in HBM; the step's launches replayed as ONE CUDA graph that holds exactly K steps between two
            timing events (event-record nodes inside the graph: device time of exactly K steps, bracketed by barrier +
            synchronize); buffer sets are rotated so that consecutive steps never find their data in the 126 MB L2; max over
            ranks.  `ms_per_step_host_bracketed` is the same replay timed with events around the graph launch.
  e2e       the same step through the public API starting from PINNED HOST buffers: per step the H2D copy of every input
            (one packed copy, di_engine_b200.PackedBatch), the kernels, a D2H read of the loss.
  roofline  CUDA-event timing of the dominant kernel against MEASURED_PEAKS.json (HBM copy bandwidth).
  cpu_baseline / --impl reference
            the reference's own functions on the host cores: the unmodified ding.rl_utils byte-compiled into
            oracle/_ref/ding_hotpath.zip by oracle/make_ref.py (kind "reference"); the oracle port only if that archive is
            absent (kind "port").  --impl reference-cuda: the same functions on CUDA tensors on the B200.

Multi-GPU (torchrun, one rank per GPU): the batch shards along B with no data-path exchange.  Config D: the six loss scalars
are exchanged by the step's own loss-finalisation launch (NVLink peer-memory mailboxes; mean of the rank means, as DI-engine's
DDP does, ding/utils/pytorch_ddp_dist_helper.py:38-47) -- no collective launch; `--collective nccl|p2p-kernel` select the
older separate exchanges.  `param_allreduce` reports the step with the parameter-gradient bucket all-reduce of the Atari VAC
network (ding/policy/base_policy.py:431-450) appended.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_LEN, B_COLS, N_ACT = 128, 4096, 6
GAMMA, LAMBDA, CLIP = 0.99, 0.95, 0.2
W_VALUE, W_ENTROPY = 0.5, -0.01
NSETS = 4
# Atari VAC of pong_ppo_config.py:21-28 (obs [4,84,84], encoder [64,64,128] k8s4/k4s2/k3s1, fc 6272->128, actor 128->128->6,
# critic 128->128->1): 16448 + 65600 + 73856 + 802944 + 17286 + 16641 parameters
VAC_PARAMS = 992775
DUMP_LIMIT = 64 << 20  # --dump-outputs: bytes written at most (the largest config, P, writes 22 MiB)


# ----------------------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------------------
def make_batch(seed, T=T_LEN, B=B_COLS, N=N_ACT):
    """config D (SURVEY.md section 8d): seeded CPU tensors, so that every arm sees identical bits"""
    g = torch.Generator().manual_seed(seed)
    value = torch.randn(T, B, generator=g)
    done = (torch.rand(T, B, generator=g) < 0.01).float()
    next_value = torch.cat([value[1:], torch.randn(1, B, generator=g)], 0)
    next_value = torch.where(done.bool(), torch.randn(T, B, generator=g), next_value).contiguous()
    reward = torch.randn(T, B, generator=g)
    traj = done.clone()
    traj[-1] = 1.0
    logit_new = torch.randn(T * B, N, generator=g)
    logit_old = logit_new + 0.1 * torch.rand(T * B, N, generator=g)
    action = torch.randint(0, N, (T * B, ), generator=g)
    value_new = torch.randn(T * B, generator=g)
    value_old = value_new + 0.1 * torch.rand(T * B, generator=g)
    return_ = torch.randn(T * B, generator=g)
    return dict(value=value, next_value=next_value, reward=reward, done=done, traj_flag=traj, logit_new=logit_new,
                logit_old=logit_old, action=action, value_new=value_new, value_old=value_old, return_=return_)


def batch_bytes(b):
    return sum(v.numel() * v.element_size() for v in b.values() if isinstance(v, torch.Tensor))


def _p(o, t):
    return o.ptr(t)


class WorkloadD:
    """gae -> ppo_error forward + backward(policy + 0.5 value - 0.01 entropy): 128 B / transition (24 + 104)."""
    key = 'D'
    unit = 'transitions'
    alg_bytes = {'gae_ppo_fwd_grad': 128, 'gae': 24, 'ppo_fwd': 76, 'ppo_bwd': 100, 'ppo_fwd_grad': 104, 'ppo_bwd_check': 0}
    step_bytes_per_unit = 128

    def __init__(self, B=B_COLS, T=T_LEN, N=N_ACT, mode='onepass'):
        self.T, self.B, self.N, self.mode = T, B, N, mode
        self.units = T * B
        self.metric = 'learner transitions/sec (GAE+ppo_error fwd+bwd, T=128 x B=4096 per GPU)'
        self.workload = ('configs[3] Atari PPO gae+ppo_error fwd+bwd, T=%d x B=%d x N=%d per GPU, fp32, gamma 0.99 lambda 0.95 '
                         'clip 0.2 value-clip on, loss mix [1, 0.5, -0.01]' % (T, B, N))

    def make_batch(self, seed):
        return make_batch(seed, self.T, self.B, self.N)

    def cpu_step(self, api, b, device=None):
        """the reference API (ding.rl_utils names): gae, ppo_error, backward"""
        nv = b['next_value'].clone()
        adv = api.gae(api.gae_data(b['value'], nv, b['reward'], b['done'], b['traj_flag']), GAMMA, LAMBDA)
        ln = b['logit_new'].detach().requires_grad_(True)
        vn = b['value_new'].detach().requires_grad_(True)
        loss, info = api.ppo_error(api.ppo_data(ln, b['logit_old'], b['action'], vn, b['value_old'], adv.reshape(-1),
                                                b['return_'], None, None), CLIP, True, None)
        (loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss).backward()
        return loss.policy_loss.detach()

    def device_step(self, host_batch, dev, exchange=None):
        return DeviceStepD(self, host_batch, dev, exchange)

    def e2e_compute(self, b2, d, three):
        ln = d['logit_new'].requires_grad_(True)
        vn = d['value_new'].requires_grad_(True)
        gd = b2.gae_data(d['value'], d['next_value'], d['reward'], d['done'], d['traj_flag'])
        if not three:
            adv, loss, info = b2.gae_ppo_error(
                gd, b2.ppo_data(ln, d['logit_old'], d['action'], vn, d['value_old'], None, d['return_'], None, None),
                GAMMA, LAMBDA, CLIP, True, None)
        else:
            adv = b2.gae(gd, GAMMA, LAMBDA)
            loss, info = b2.ppo_error(
                b2.ppo_data(ln, d['logit_old'], d['action'], vn, d['value_old'], adv.view(-1), d['return_'], None,
                            None), CLIP, True, None)
        total = loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss
        total.backward()
        return total


class DeviceStepD:
    """One config-D learner step on device-resident buffers through the C ABI (the layer under the public API)."""

    def __init__(self, wl, host_batch, dev, exchange=None):
        from di_engine_b200 import ops
        self.ops, self.wl, self.exchange = ops, wl, exchange
        self.hint = torch.tensor([1.0, W_VALUE, W_ENTROPY, 0.0], device=dev)
        self.g_used = torch.zeros(4, device=dev)
        self.b = {k: v.to(dev) for k, v in host_batch.items()}
        self.nv0 = self.b['next_value'].clone()
        self.S = wl.T * wl.B
        self.g_p = torch.tensor(1.0, device=dev)
        self.g_v = torch.tensor(W_VALUE, device=dev)
        self.g_e = torch.tensor(W_ENTROPY, device=dev)
        self.adv = torch.empty_like(self.b['value'])
        self.out = torch.zeros(8, device=dev)
        self.grad_logit = torch.empty_like(self.b['logit_new'])
        self.grad_value = torch.empty_like(self.b['value_new'])
        self.ws = ops.workspace(torch.device(dev))

    def _ppo_in(self):
        b, o = self.b, self.ops
        return (_p(o, b['logit_new']), _p(o, b['logit_old']), None, _p(o, b['action']), _p(o, b['value_new']),
                _p(o, b['value_old']), _p(o, self.adv), _p(o, b['return_']), None, self.S, 1, self.wl.N, CLIP, 1, 0.0, 1, None, None)

    def gae(self):
        b, o = self.b, self.ops
        rc = o.lib().b200rl_gae(_p(o, b['value']), _p(o, b['next_value']), _p(o, b['reward']), _p(o, b['done']),
                                _p(o, b['traj_flag']), _p(o, self.adv), self.wl.T, self.wl.B, 1, GAMMA, LAMBDA, 1,
                                o.stream_ptr())
        assert rc == 0, rc

    def ppo_fwd(self):
        o = self.ops
        rc = o.lib().b200rl_ppo_fwd(*self._ppo_in(), _p(o, self.out), _p(o, self.ws), self.ws.numel() * 4, o.stream_ptr())
        assert rc == 0, rc

    def ppo_bwd(self):
        o = self.ops
        rc = o.lib().b200rl_ppo_bwd(*self._ppo_in(), _p(o, self.g_p), _p(o, self.g_v), _p(o, self.g_e), None, None, None,
                                    _p(o, self.grad_logit), _p(o, self.grad_value), o.stream_ptr())
        assert rc == 0, rc

    def ppo_fwd_grad(self):
        o = self.ops
        rc = o.lib().b200rl_ppo_fwd_grad(*self._ppo_in(), _p(o, self.hint), _p(o, self.g_used), _p(o, self.out),
                                         _p(o, self.grad_logit), _p(o, self.grad_value), _p(o, self.ws),
                                         self.ws.numel() * 4, o.stream_ptr())
        assert rc == 0, rc

    def ppo_bwd_check(self):
        o = self.ops
        rc = o.lib().b200rl_ppo_bwd(*self._ppo_in(), _p(o, self.g_p), _p(o, self.g_v), _p(o, self.g_e), None,
                                    _p(o, self.g_used), _p(o, self.hint), _p(o, self.grad_logit),
                                    _p(o, self.grad_value), o.stream_ptr())
        assert rc == 0, rc

    def gae_ppo_fwd_grad(self):
        b, o = self.b, self.ops
        head = (_p(o, b['value']), _p(o, b['next_value']), _p(o, b['reward']), _p(o, b['done']), _p(o, b['traj_flag']),
                self.wl.T, self.wl.B, GAMMA, LAMBDA, 1, _p(o, b['logit_new']), _p(o, b['logit_old']), None,
                _p(o, b['action']), _p(o, b['value_new']), _p(o, b['value_old']), _p(o, b['return_']), None, self.wl.N,
                CLIP, 1, 0.0, 1, _p(o, self.hint), _p(o, self.g_used), _p(o, self.adv), _p(o, self.out),
                _p(o, self.grad_logit), _p(o, self.grad_value))
        tail = (_p(o, self.ws), self.ws.numel() * 4, o.stream_ptr())
        if self.exchange is not None:  # the loss scalars travel in the step's finalize launch (NVLink mailboxes)
            rc = o.lib().b200rl_gae_ppo_fwd_grad_dp(*head, *self.exchange.args(), *tail)
        else:
            rc = o.lib().b200rl_gae_ppo_fwd_grad(*head, *tail)
        assert rc == 0, rc

    def kernels(self):
        if self.wl.mode == 'onepass':
            return [('gae_ppo_fwd_grad', self.gae_ppo_fwd_grad), ('ppo_bwd_check', self.ppo_bwd_check)]
        if self.wl.mode == 'three':
            return [('gae', self.gae), ('ppo_fwd_grad', self.ppo_fwd_grad), ('ppo_bwd_check', self.ppo_bwd_check)]
        return [('gae', self.gae), ('ppo_fwd', self.ppo_fwd), ('ppo_bwd', self.ppo_bwd)]

    def launches_per_step(self):
        return {'onepass': 3, 'three': 5, 'unfused': 4}[self.wl.mode]

    def loss_vector(self):
        return self.out

    def outputs(self):
        """what a caller of gae_ppo_error receives from this step: the advantage, ppo_loss, ppo_info and the gradients"""
        names = ('policy_loss', 'value_loss', 'entropy_loss', 'kl_div', 'approx_kl', 'clipfrac')
        return dict(adv=self.adv, **{n: self.out[i] for i, n in enumerate(names)}, grad_logit_new=self.grad_logit,
                    grad_value_new=self.grad_value)

    def __call__(self):
        for _, k in self.kernels():
            k()

    def check(self, host_batch):
        """correctness guard against the CPU oracle (outside every timed region)"""
        from oracle import rl_oracle
        self()
        torch.cuda.synchronize()
        hb = host_batch
        adv_ref = rl_oracle.gae(hb['value'], hb['next_value'].clone(), hb['reward'], hb['done'], hb['traj_flag'], GAMMA,
                                LAMBDA)
        assert torch.equal(self.adv.cpu(), adv_ref), 'gae parity broken'
        self.b['next_value'].copy_(self.nv0)


class WorkloadP(WorkloadD):
    """Config D as PPOPolicy._forward_learn really composes it (ding/policy/ppo.py:274-306): value-norm scale -> gae ->
    unnormalized return / stored value / return_ + running statistics -> (adv - mean) / (std + 1e-8) -> ppo_error, backward.
    gae_returns 36 B (20 in + 16 out; the advantage statistics come out of the same pass) + ppo forward-with-gradient 104 B per
    transition."""
    key = 'P'
    alg_bytes = {'gae_returns': 36, 'ppo_fwd_grad': 104, 'ppo_bwd_check': 0}
    step_bytes_per_unit = 140
    STD = 1.7320508

    def __init__(self, B=B_COLS, T=T_LEN, N=N_ACT):
        super().__init__(B=B, T=T, N=N, mode='policy')
        self.metric = 'learner transitions/sec (PPOPolicy advantage recompute + ppo_error fwd+bwd, T=128 x B=4096 per GPU)'
        self.workload = ('configs[3] as PPOPolicy._forward_learn composes it (policy/ppo.py:274-306): value_norm scale, gae, '
                         'returns + running stats, advantage normalisation, ppo_error fwd+bwd; T=%d x B=%d x N=%d per GPU, '
                         'fp32' % (T, B, N))

    def make_batch(self, seed):
        b = make_batch(seed, self.T, self.B, self.N)
        del b['return_'], b['value_old']  # both come out of the advantage recompute (policy/ppo.py:283-292)
        return b

    def cpu_step(self, api, b, device=None):
        """policy/ppo.py:274-306 executed literally around the reference API (RunningMeanStd.update's numpy reduction included)"""
        std = self.STD
        with torch.no_grad():
            value, next_value = b['value'] * std, b['next_value'] * std
            adv = api.gae(api.gae_data(value, next_value, b['reward'], b['done'], b['traj_flag']), GAMMA, LAMBDA)
            unnormalized_returns = value + adv
            value, return_ = value / std, unnormalized_returns / std
            x = unnormalized_returns.cpu().numpy()
            x.mean(), x.var()
            adv = adv.reshape(-1)
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        ln = b['logit_new'].detach().requires_grad_(True)
        vn = b['value_new'].detach().requires_grad_(True)
        loss, info = api.ppo_error(api.ppo_data(ln, b['logit_old'], b['action'], vn, value.reshape(-1), adv,
                                                return_.reshape(-1), None, None), CLIP, True, None)
        (loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss).backward()
        return loss.policy_loss.detach()

    def device_step(self, host_batch, dev, exchange=None):
        return DeviceStepP(self, host_batch, dev)

    def e2e_compute(self, b2, d, three):
        ln = d['logit_new'].requires_grad_(True)
        vn = d['value_new'].requires_grad_(True)
        g = b2.gae_returns(b2.gae_data(d['value'], d['next_value'], d['reward'], d['done'], d['traj_flag']), GAMMA, LAMBDA,
                           self.STD)
        loss, info = b2.ppo_error_adv_norm(
            b2.ppo_data(ln, d['logit_old'], d['action'], vn, g.value.view(-1), g.adv.view(-1), g.return_.view(-1), None, None),
            CLIP, True, None, adv_stats=g.adv_stats)
        total = loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss
        total.backward()
        return total


class DeviceStepP(DeviceStepD):

    def __init__(self, wl, host_batch, dev):
        super().__init__(wl, host_batch, dev)
        self.unnorm, self.vout, self.rout = (torch.empty_like(self.adv) for _ in range(3))
        self.ret_stats = torch.zeros(3, device=dev)
        self.adv_stats = torch.zeros(2, device=dev)

    def _ppo_in(self):
        b, o = self.b, self.ops
        return (_p(o, b['logit_new']), _p(o, b['logit_old']), None, _p(o, b['action']), _p(o, b['value_new']),
                _p(o, self.vout), _p(o, self.adv), _p(o, self.rout), None, self.S, 1, self.wl.N, CLIP, 1, 0.0, 1,
                _p(o, self.adv_stats), None)

    def gae_returns(self):
        b, o = self.b, self.ops
        rc = o.lib().b200rl_gae_returns(
            _p(o, b['value']), _p(o, b['next_value']), _p(o, b['reward']), _p(o, b['done']), _p(o, b['traj_flag']), self.wl.T,
            self.wl.B, 1, GAMMA, LAMBDA, 0, self.wl.STD, _p(o, self.adv), _p(o, self.unnorm), _p(o, self.vout), _p(o, self.rout),
            _p(o, self.ret_stats), _p(o, self.adv_stats), _p(o, self.ws), self.ws.numel() * 4, o.stream_ptr())
        assert rc == 0, rc

    def kernels(self):
        return [('gae_returns', self.gae_returns), ('ppo_fwd_grad', self.ppo_fwd_grad), ('ppo_bwd_check', self.ppo_bwd_check)]

    def launches_per_step(self):
        return 5  # gae scan, returns + both statistics, ppo forward-with-gradient, finalize_sums, backward check

    def outputs(self):
        return dict(super().outputs(), value=self.vout, return_=self.rout, unnormalized_return=self.unnorm)

    def check(self, host_batch):
        from oracle import rl_oracle
        self()
        torch.cuda.synchronize()
        hb = host_batch
        want = rl_oracle.ppo_policy_gae_returns(hb['value'], hb['next_value'], hb['reward'], hb['done'], hb['traj_flag'], GAMMA,
                                                LAMBDA, self.wl.STD)
        for got, w, name in zip((self.adv, self.vout, self.rout, self.unnorm), want[:4], ('adv', 'value', 'return', 'unnorm')):
            assert torch.equal(got.cpu(), w), 'gae_returns parity broken: ' + name


def DeviceStep(host_batch, dev, fused='onepass'):
    """entry point of the round-1 experiment tools (tools/exp_*.py, trace_*.py, sweep_col.py): one config-D buffer set with
    the launch decomposition they name ('onepass' | True = three launches | False = unfused)"""
    mode = {'onepass': 'onepass', True: 'three', False: 'unfused'}[fused]
    T, B = host_batch['value'].shape
    return DeviceStepD(WorkloadD(B=B, T=T, N=host_batch['logit_new'].shape[-1], mode=mode), host_batch, dev)


class WorkloadB:
    """q_nstep_td_error forward + backward: one launch + its verification; 120 B / sample at N=6, n=3 with value_gamma."""
    key = 'B'
    unit = 'samples'

    def __init__(self, B=512, N=6, nstep=3):
        self.B, self.N, self.nstep = B, N, nstep
        self.units = B
        self.metric = 'learner samples/sec (q_nstep_td_error fwd+bwd, B=512 N=6 nstep=3)'
        self.workload = 'configs[1] Pong DQN q_nstep_td_error fwd+bwd, B=%d N=%d nstep=%d, gamma 0.99, value_gamma tensor, fp32' % (
            B, N, nstep)
        per = 8 * N + 16 + 4 * nstep + 12 + 4 + 4 + 4 * N  # SURVEY.md section 8d (+4: value_gamma)
        self.alg_bytes = {'qntd_fwd_grad': per, 'qntd_bwd_check': 0}
        self.step_bytes_per_unit = per

    def make_batch(self, seed):
        g = torch.Generator().manual_seed(seed)
        B, N, n = self.B, self.N, self.nstep
        return dict(q=torch.randn(B, N, generator=g), next_n_q=torch.randn(B, N, generator=g),
                    action=torch.randint(0, N, (B, ), generator=g), next_n_action=torch.randint(0, N, (B, ), generator=g),
                    reward=torch.rand(n, B, generator=g), done=(torch.rand(B, generator=g) < 0.05).float(),
                    value_gamma=torch.full((B, ), GAMMA ** n))

    def cpu_step(self, api, b, device=None):
        q = b['q'].detach().requires_grad_(True)
        data = api.q_nstep_td_data(q, b['next_n_q'], b['action'], b['next_n_action'], b['reward'], b['done'], None)
        loss, per = api.q_nstep_td_error(data, GAMMA, nstep=self.nstep, value_gamma=b['value_gamma'])
        loss.backward()
        return loss.detach()

    def device_step(self, host_batch, dev, exchange=None):
        return DeviceStepTD(self, host_batch, dev)

    def e2e_compute(self, b2, d, three):
        q = d['q'].requires_grad_(True)
        data = b2.q_nstep_td_data(q, d['next_n_q'], d['action'], d['next_n_action'], d['reward'], d['done'], None)
        loss, per = b2.q_nstep_td_error(data, GAMMA, nstep=self.nstep, value_gamma=d['value_gamma'])
        loss.backward()
        return loss


class WorkloadC(WorkloadB):
    """dist_nstep_td_error (C51) forward + backward; 1672 B / sample (SURVEY.md section 8d: selected rows in, dense grad out)."""
    key = 'C'

    def __init__(self, B=512, N=6, n_atom=51, nstep=3):
        self.B, self.N, self.n_atom, self.nstep = B, N, n_atom, nstep
        self.units = B
        self.metric = 'learner samples/sec (dist_nstep_td_error fwd+bwd, B=512 N=6 n_atom=51 nstep=3)'
        self.workload = ('configs[2] Atari C51 dist_nstep_td_error fwd+bwd, B=%d N=%d n_atom=%d nstep=%d, gamma 0.99, '
                         'v in [-10, 10], fp32' % (B, N, n_atom, nstep))
        per = 2 * 4 * n_atom + 16 + 4 * nstep + 8 + 4 * N * n_atom + 4
        self.alg_bytes = {'dntd_fwd_grad': per, 'dntd_bwd_check': 0}
        self.step_bytes_per_unit = per

    def make_batch(self, seed):
        g = torch.Generator().manual_seed(seed)
        B, N, n, A = self.B, self.N, self.nstep, self.n_atom
        return dict(dist=torch.softmax(torch.randn(B, N, A, generator=g), -1),
                    next_n_dist=torch.softmax(torch.randn(B, N, A, generator=g), -1),
                    act=torch.randint(0, N, (B, ), generator=g), next_n_act=torch.randint(0, N, (B, ), generator=g),
                    reward=torch.rand(n, B, generator=g), done=(torch.rand(B, generator=g) < 0.05).float())

    def cpu_step(self, api, b, device=None):
        dist = b['dist'].detach().requires_grad_(True)
        data = api.dist_nstep_td_data(dist, b['next_n_dist'], b['act'], b['next_n_act'], b['reward'], b['done'], None)
        loss, per = api.dist_nstep_td_error(data, GAMMA, -10., 10., self.n_atom, self.nstep)
        loss.backward()
        return loss.detach()

    def e2e_compute(self, b2, d, three):
        dist = d['dist'].requires_grad_(True)
        data = b2.dist_nstep_td_data(dist, d['next_n_dist'], d['act'], d['next_n_act'], d['reward'], d['done'], None)
        loss, per = b2.dist_nstep_td_error(data, GAMMA, -10., 10., self.n_atom, self.nstep)
        loss.backward()
        return loss


class DeviceStepTD:
    """configs B / C on device-resident buffers through the C ABI: the one-launch forward+gradient and its verification."""

    def __init__(self, wl, host_batch, dev):
        from di_engine_b200 import ops
        from di_engine_b200.rl_utils import td as tdmod
        self.ops, self.wl = ops, wl
        self.b = {k: v.to(dev) for k, v in host_batch.items()}
        self.one = torch.tensor(1.0, device=dev)
        B, N = wl.B, wl.N
        self.loss = torch.zeros((), device=dev)
        self.td = torch.empty(B, device=dev)
        self.ws = ops.workspace(torch.device(dev))
        if wl.key == 'B':
            self.dcrit = torch.empty(B, device=dev)
            self.target = torch.empty(B, device=dev)
            self.grad = torch.empty(B, N, device=dev)
        else:
            self.proj = torch.empty(B, wl.n_atom, device=dev)
            self.grad = torch.empty(B, N, wl.n_atom, device=dev)
            self.support = tdmod._support(-10., 10., wl.n_atom, torch.device(dev))
            self.bad = torch.zeros(1, dtype=torch.int32, device=dev)

    def fwd_grad(self):
        b, o, wl = self.b, self.ops, self.wl
        if wl.key == 'B':
            rc = o.lib().b200rl_qntd_fwd(
                _p(o, b['q']), _p(o, b['next_n_q']), _p(o, b['action']), _p(o, b['next_n_action']), _p(o, b['reward']),
                _p(o, b['done']), None, _p(o, b['value_gamma']), 1, None, wl.B, 1, wl.N, wl.nstep, GAMMA, 0, 0, 1e-2, 0,
                0.0, 0, 0, 0.0, _p(o, self.loss), _p(o, self.td), _p(o, self.dcrit), _p(o, self.target), _p(o, self.grad),
                None, _p(o, self.ws), self.ws.numel() * 4, o.stream_ptr())
        else:
            rc = o.lib().b200rl_dntd_fwd(
                _p(o, b['dist']), _p(o, b['next_n_dist']), _p(o, b['act']), _p(o, b['next_n_act']), _p(o, b['reward']),
                _p(o, b['done']), None, 0, None, 0, _p(o, self.support), wl.B, 1, wl.N, wl.n_atom, wl.nstep, GAMMA, -10.,
                10., _p(o, self.loss), _p(o, self.td), _p(o, self.proj), _p(o, self.bad), _p(o, self.grad), _p(o, self.ws),
                self.ws.numel() * 4, o.stream_ptr())
        assert rc == 0, rc

    def bwd_check(self):
        b, o, wl = self.b, self.ops, self.wl
        if wl.key == 'B':
            rc = o.lib().b200rl_qntd_bwd(_p(o, self.dcrit), None, _p(o, b['action']), _p(o, self.one), None, wl.B, 1, wl.N,
                                         0, 0, 1, _p(o, self.grad), o.stream_ptr())
        else:
            rc = o.lib().b200rl_dntd_bwd(_p(o, b['dist']), _p(o, b['act']), _p(o, self.proj), None, 0, _p(o, self.one),
                                         None, wl.B, wl.N, wl.n_atom, 1, _p(o, self.grad), o.stream_ptr())
        assert rc == 0, rc

    def kernels(self):
        pre = 'qntd' if self.wl.key == 'B' else 'dntd'
        return [(pre + '_fwd_grad', self.fwd_grad), (pre + '_bwd_check', self.bwd_check)]

    def launches_per_step(self):
        return 2

    def loss_vector(self):
        return self.loss

    def outputs(self):
        grad = 'grad_q' if self.wl.key == 'B' else 'grad_dist'
        return {'loss': self.loss, 'td_error_per_sample': self.td, grad: self.grad}

    def __call__(self):
        for _, k in self.kernels():
            k()

    def check(self, host_batch):
        self()
        torch.cuda.synchronize()
        api = _cpu_api()[0]
        want = self.wl.cpu_step(api, host_batch)
        assert abs(float(self.loss) - float(want)) <= 1e-5 + 1e-5 * abs(float(want)), (float(self.loss), float(want))


class WorkloadE:
    """vtrace_error_discrete_action forward + backward in one launch + verification: 96 B / transition (68 in + 28 out)."""
    key = 'E'
    unit = 'transitions'
    alg_bytes = {'vtrace_fwd_grad': 96, 'vtrace_bwd_check': 0}
    step_bytes_per_unit = 96

    def __init__(self, T=64, B=8192, N=6):
        self.T, self.B, self.N = T, B, N
        self.units = T * B
        self.metric = 'learner transitions/sec (vtrace_error_discrete_action fwd+bwd, T=64 x B=8192 per GPU)'
        self.workload = ('configs[4] IMPALA vtrace_error_discrete_action fwd+bwd, T=%d x B=%d x N=%d per GPU, fp32, gamma 0.99 '
                         'lambda 0.95 clips 1.0, loss mix [1, 0.5, -0.01]' % (T, B, N))

    def make_batch(self, seed):
        g = torch.Generator().manual_seed(seed)
        T, B, N = self.T, self.B, self.N
        tgt = torch.randn(T, B, N, generator=g)
        return dict(target_output=tgt, behaviour_output=tgt + 0.5 * torch.randn(T, B, N, generator=g),
                    action=torch.randint(0, N, (T, B), generator=g), value=torch.randn(T + 1, B, generator=g),
                    reward=torch.rand(T, B, generator=g), weight=torch.ones(T, B))

    def cpu_step(self, api, b, device=None):
        tgt = b['target_output'].detach().requires_grad_(True)
        val = b['value'].detach().requires_grad_(True)
        loss = api.vtrace_error_discrete_action(
            api.vtrace_data(tgt, b['behaviour_output'], b['action'], val, b['reward'], b['weight']), GAMMA, LAMBDA)
        (loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss).backward()
        return loss.policy_loss.detach()

    def device_step(self, host_batch, dev, exchange=None):
        return DeviceStepE(self, host_batch, dev)

    def e2e_compute(self, b2, d, three):
        tgt = d['target_output'].requires_grad_(True)
        val = d['value'].requires_grad_(True)
        loss = b2.vtrace_error_discrete_action(
            b2.vtrace_data(tgt, d['behaviour_output'], d['action'], val, d['reward'], d['weight']), GAMMA, LAMBDA)
        total = loss.policy_loss + W_VALUE * loss.value_loss + W_ENTROPY * loss.entropy_loss
        total.backward()
        return total


class DeviceStepE:

    def __init__(self, wl, host_batch, dev):
        from di_engine_b200 import ops
        self.ops, self.wl = ops, wl
        self.b = {k: v.to(dev) for k, v in host_batch.items()}
        self.hint = torch.tensor([1.0, W_VALUE, W_ENTROPY], device=dev)
        self.g_used = torch.zeros(3, device=dev)
        self.g = [torch.tensor(x, device=dev) for x in (1.0, W_VALUE, W_ENTROPY)]
        self.out = torch.zeros(4, device=dev)
        self.grad_logit = torch.empty_like(self.b['target_output'])
        self.grad_value = torch.empty_like(self.b['value'])
        self.ws = ops.workspace(torch.device(dev))

    def _call(self, verify):
        b, o, wl = self.b, self.ops, self.wl
        rc = o.lib().b200rl_vtrace_fwd_grad(
            _p(o, b['target_output']), _p(o, b['behaviour_output']), _p(o, b['action']), _p(o, b['value']),
            _p(o, b['reward']), _p(o, b['weight']), wl.T, wl.B, wl.N, GAMMA, LAMBDA, 1.0, 1.0, 1.0,
            None if verify else _p(o, self.hint), 1 if verify else 0, _p(o, self.g[0]) if verify else None,
            _p(o, self.g[1]) if verify else None, _p(o, self.g[2]) if verify else None, _p(o, self.g_used),
            _p(o, self.hint) if verify else None, None if verify else _p(o, self.out), _p(o, self.grad_logit),
            _p(o, self.grad_value), _p(o, self.ws), self.ws.numel() * 4, o.stream_ptr())
        assert rc == 0, rc

    def kernels(self):
        return [('vtrace_fwd_grad', lambda: self._call(False)), ('vtrace_bwd_check', lambda: self._call(True))]

    def launches_per_step(self):
        return 3

    def loss_vector(self):
        return self.out

    def outputs(self):
        return dict(policy_loss=self.out[0], value_loss=self.out[1], entropy_loss=self.out[2],
                    grad_target_output=self.grad_logit, grad_value=self.grad_value)

    def __call__(self):
        for _, k in self.kernels():
            k()

    def check(self, host_batch):
        self()
        torch.cuda.synchronize()
        assert torch.isfinite(self.out[:3]).all()


WORKLOADS = {'D': WorkloadD, 'P': WorkloadP, 'B': WorkloadB, 'C': WorkloadC, 'E': WorkloadE}


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own functions on the host cores
# ----------------------------------------------------------------------------------------------------------------
def _cpu_api():
    """(api namespace, kind): the unmodified reference (tree or byte-compiled archive) when present, else the oracle port"""
    from oracle import ref_loader
    if ref_loader.available():
        return ref_loader.load(), 'reference'
    from oracle import port_api
    return port_api, 'port'


def usable_cores():
    """Host cores this process may actually use: affinity mask, clipped by the cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def pick_threads(wl, api, b):
    """All the host threads the reference can USE: the fastest of {usable, 64, 32, 16, 8, 4} torch intra-op threads, best of
    three timed steps per candidate (over-subscribing a throttled container makes torch slower, not faster)."""
    usable = usable_cores()
    best, best_t = None, None
    for n in sorted({usable, 64, 32, 16, 8, 4}):
        if n > usable:
            continue
        torch.set_num_threads(n)
        wl.cpu_step(api, b)
        dt = None
        for _ in range(3):
            t0 = time.perf_counter()
            wl.cpu_step(api, b)
            d = time.perf_counter() - t0
            dt = d if dt is None else min(dt, d)
        if best_t is None or dt < best_t:
            best, best_t = n, dt
        if dt > 4 * best_t:
            break
    return best


def run_cpu(wl, steps, warmup):
    api, kind = _cpu_api()
    b = wl.make_batch(0)
    cores = pick_threads(wl, api, b)
    torch.set_num_threads(cores)
    for _ in range(warmup):
        wl.cpu_step(api, b)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        wl.cpu_step(api, b)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return dict(value=wl.units / med, ms_per_step=med * 1e3, total_s=sum(times), cores=cores, kind=kind,
                threads=torch.get_num_threads())


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except OSError:
        pass
    return 'unknown'


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.samples = []
        self.proc = None
        self.idx = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            f = [x.strip() for x in s.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except (KeyError, ValueError):
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def kernel_source_sha(files):
    """sha256 over the CUDA sources that define a kernel: ties a committed ncu capture to the code that is being timed"""
    h = hashlib.sha256()
    for f in files:
        with open(os.path.join(ROOT, 'di-engine_b200', 'csrc', f), 'rb') as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json) -- only if that capture
    was taken from the sources the loaded library was built from; otherwise (None, why)."""
    try:
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json'))).get(kernel)
    except (OSError, ValueError):
        return None, 'profiles/ncu_traffic.json missing'
    if not tr:
        return None, 'no ncu capture recorded for %s' % kernel
    want = tr.get('source_sha16')
    have = kernel_source_sha(tr.get('sources', [])) if tr.get('sources') else None
    if not want or want != have:
        return None, 'ncu capture is of other sources (%s != %s)' % (want, have)
    return tr['dram_read'] + tr['dram_write'], 'profiles/%s' % tr.get('capture', 'ncu_traffic.json')


def set_rank_affinity(local_rank):
    """Bind this rank's host threads (and with them its pinned staging buffers, first-touch) to the CPUs NVML reports as
    local to its GPU: the e2e loader of 8 ranks otherwise crosses the socket interconnect for half of them."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def dbg(*a):
    if os.environ.get('BENCH_DEBUG'):
        print('[bench %s]' % os.environ.get('RANK', '0'), *a, file=sys.stderr, flush=True)


def run_gpu(args):
    import torch.distributed as dist
    import di_engine_b200 as b2

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        raise SystemExit('launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)' % (args.gpus, world))
    affinity = set_rank_affinity(local)
    torch.cuda.set_device(local)
    dev = 'cuda:%d' % local
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, max(args.warmup, 3)
    strong = args.scaling == 'strong'
    if args.config == 'D':
        Bl = B_COLS // world if strong else B_COLS
        if strong and B_COLS % world:
            raise SystemExit('strong scaling needs world | %d' % B_COLS)
        wl = WorkloadD(B=Bl, mode='unfused' if args.unfused else ('three' if args.three else 'onepass'))
    elif args.config == 'E':
        wl = WorkloadE(B=(8192 // world) if strong else 8192)
    elif args.config == 'P':
        wl = WorkloadP(B=(B_COLS // world) if strong else B_COLS)
    else:
        wl = WORKLOADS[args.config]()
        if world > 1:
            raise SystemExit('configs B / C are single-GPU, launch-bound cases (SURVEY.md section 8d)')

    main = torch.cuda.Stream()
    side = torch.cuda.Stream()
    from di_engine_b200.parallel import FusedLossExchange, LossAllReduce, P2PLossAllReduce
    exchange, fused_x, reducers = 'none', None, None
    if world > 1:
        mode = args.collective
        if mode == 'auto':
            mode = 'fused' if (wl.key == 'D' and wl.mode == 'onepass') else 'p2p-kernel'
        if mode == 'fused':
            try:
                fused_x = FusedLossExchange(dev)
                exchange = 'fused'
            except Exception as e:
                if rank == 0:
                    print('bench: peer-memory mailboxes unavailable (%s); using NCCL' % e, file=sys.stderr)
                mode = 'nccl'
        if mode == 'p2p-kernel':
            try:
                reducers = [P2PLossAllReduce(6, dev) for _ in range(NSETS)]
                exchange = 'p2p-kernel'
            except Exception as e:
                if rank == 0:
                    print('bench: peer-memory all-reduce unavailable (%s); using NCCL' % e, file=sys.stderr)
                mode = 'nccl'
        if mode == 'nccl':
            reducers = [LossAllReduce(6, dev) for _ in range(NSETS)]
            exchange = 'nccl'

    dbg('setup done')
    hosts = [wl.make_batch(1000 * rank + i) for i in range(NSETS)]
    sets = [wl.device_step(hosts[i], dev, fused_x) for i in range(NSETS)]
    names = [n for n, _ in sets[0].kernels()]
    step_bytes = wl.step_bytes_per_unit * wl.units

    def exchange_losses(j):
        """separate exchange kernels (older modes): mean over ranks of set j's loss scalars, on the current stream"""
        if exchange == 'p2p-kernel':
            reducers[j].reduce(sets[j].loss_vector())
        elif exchange == 'nccl':
            reducers[j].buf.copy_(sets[j].loss_vector().reshape(-1)[:6], non_blocking=True)
            reducers[j].reduce()

    # ---- correctness guard on rank 0 (outside every timed region) ---------------------------------------------------
    if rank == 0:
        chk = wl.make_batch(0)
        wl.device_step(chk, dev).check(chk)
    barrier()

    dbg('check done')
    bucket = torch.zeros(VAC_PARAMS, device=dev) if world > 1 else None

    def record_steps(n):
        """n steps over the rotated buffer sets on the current (capturing) stream"""
        for i in range(n):
            j = i % NSETS
            if exchange in ('p2p-kernel', 'nccl') and i > 0:  # software-pipelined on a forked branch, as in round 1
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    exchange_losses((j - 1) % NSETS)
            sets[j]()
            if exchange in ('p2p-kernel', 'nccl') and i > 0:
                main.wait_stream(side)
        if exchange in ('p2p-kernel', 'nccl'):
            exchange_losses((n - 1) % NSETS)
        elif exchange == 'fused':
            fused_x.drain()

    def timed_graph(n, lead=0):
        """ONE graph: [rank alignment] [lead untimed steps] e0 | n steps | e1 -- the two events are nodes of the graph (external
        events), so their difference is the device time of exactly n steps, free of the host's launch latency"""
        e0 = torch.cuda.Event(enable_timing=True, external=True)
        e1 = torch.cuda.Event(enable_timing=True, external=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=main):
            if world > 1 and align is not None:
                align.reduce(align_src)  # device-side rank alignment: every rank leaves within one NVLink flag round
            if lead:
                record_steps(lead)
            e0.record(main)
            record_steps(n)
            e1.record(main)
        return g, e0, e1

    align, align_src = None, None
    with torch.cuda.stream(main):
        for s in sets:
            s()
            s()
        if exchange == 'fused':
            fused_x.drain()
        elif world > 1:
            for j in range(NSETS):
                exchange_losses(j)
        if world > 1:
            try:
                align = P2PLossAllReduce(1, dev)
                align_src = torch.ones(8, device=dev)
                align.reduce(align_src)
            except Exception:
                align = None
        main.synchronize()
        barrier()
        dbg('eager warm done')
        graph_warm, _w0, _w1 = timed_graph(250)  # (the event-record nodes need their events alive)
        graph_k, e0, e1 = timed_graph(K, lead=int(os.environ.get('BENCH_LEAD_STEPS', '0')))
        main.synchronize()
        barrier()

        # pre-heat: ~0.25 s of the same steps (untimed) so SM/memory clocks are in steady state -- one step is far shorter
        # than the clock governor's reaction time.  FIXED counts: with an exchange in the graph every rank must launch exactly
        # the same number of steps.
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()  # spawned before the pre-heat so that the process start-up does not leave the GPU idle later
        for _ in range(60):
            graph_warm.replay()
        main.synchronize()
        dbg('preheat done')
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        # the W warm-up steps run IMMEDIATELY before the K timed steps (enqueued back to back, no idle gap: a GPU that has sat
        # idle for a barrier runs its first tens of microseconds slower); the timed region is delimited by the two event
        # nodes inside graph_k
        for _ in range(max(1, (W + 249) // 250)):
            graph_warm.replay()
        h0.record(main)
        graph_k.replay()
        h1.record(main)
        barrier()
        dbg('timed replay done')
        # device-side copy of the last timed step's outputs before later replays reuse its buffer set
        last_outputs = {k: v.clone() for k, v in sets[(K - 1) % NSETS].outputs().items()} if args.dump_outputs else None
        dev_ms = e0.elapsed_time(e1)
        host_ms = h0.elapsed_time(h1)
        # keep the GPU under the same load while nvidia-smi samples (a 20-step region lasts 0.3 ms)
        for _ in range(40):
            graph_warm.replay()
        main.synchronize()
        clocks = sampler.stop() if rank == 0 else None

        # ---- the step with the parameter-gradient bucket all-reduce of the Atari VAC net appended (SURVEY section 8e) -----
        par = None
        if world > 1:
            try:
                for _ in range(3):
                    dist.all_reduce(bucket)
                main.synchronize()
                barrier()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(main)
                for _ in range(50):
                    dist.all_reduce(bucket)
                a1.record(main)
                main.synchronize()
                ar_us = a0.elapsed_time(a1) * 1e3 / 50
                # eager launches (no NCCL inside a CUDA graph: an eager collective after a captured one has been seen to hang)
                n_par = max(20, min(K, 200))
                barrier()
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record(main)
                for i in range(n_par):
                    sets[i % NSETS]()
                    dist.all_reduce(bucket)
                if exchange == 'fused':
                    fused_x.drain()
                p1.record(main)
                main.synchronize()
                barrier()
                par = dict(bytes=VAC_PARAMS * 4, nccl_allreduce_us_alone=ar_us, ms_per_step_with=p0.elapsed_time(p1) / n_par,
                           steps=n_par, launch='eager')
            except Exception as e:  # never let the secondary figure break the benchmark
                if rank == 0:
                    print('bench: param all-reduce leg skipped (%s)' % e, file=sys.stderr)
                torch.cuda.synchronize()

        # ---- the same step launched eagerly (one ctypes call per launch, no graph): host-bound --------------------------
        dbg('param leg done')
        eager_ms = None
        if world == 1:
            n_eager = 200
            for i in range(8):
                sets[i % NSETS]()
            main.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(main)
            for i in range(n_eager):
                sets[i % NSETS]()
            g1.record(main)
            main.synchronize()
            eager_ms = g0.elapsed_time(g1) / n_eager

        # ---- per-kernel timing: each API call alone, back to back over the rotated sets, in a graph --------------------
        dbg('eager done')
        per = {}
        reps = max(100, min(K, 2000) // NSETS)
        if fused_x is None:
            for ki, name in enumerate(names):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=main):
                    for s in sets:
                        s.kernels()[ki][1]()
                for _ in range(3):
                    g.replay()
                k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                main.synchronize()
                k0.record(main)
                for _ in range(reps):
                    g.replay()
                k1.record(main)
                main.synchronize()
                per[name] = k0.elapsed_time(k1) / (reps * NSETS)

    # ---- end-to-end through the public API from pinned host buffers ------------------------------------------------
    dbg('per-kernel done')
    packed = not args.e2e_separate_copies
    if packed:  # one pinned buffer + one device buffer per slot: the H2D transfer of a step is a single copy
        narrow = None
        if args.e2e_compact:  # one-byte actions and flags on the wire, widened on the device after the copy (exact)
            narrow = {k: torch.uint8 for k in ('action', 'done', 'traj_flag', 'next_n_action', 'act', 'next_n_act')}
        slots = [b2.PackedBatch(wl.make_batch(2000 * rank + i), dev, narrow=narrow) for i in range(2)]
        host = slots
        h2d = slots[0].payload_bytes()
    else:
        host = [{k: v.pin_memory() for k, v in wl.make_batch(2000 * rank + i).items()} for i in range(2)]
        h2d = batch_bytes(host[0])

    # two-deep prefetching loader (what DI-engine's CudaFetcher, ding/torch_utils/data_helper.py:543, does for the learner):
    # the H2D copy of step i+1 is enqueued on a copy stream before step i's result is read back.  Every byte of every step is
    # still copied inside the timed region.
    copy_stream = torch.cuda.Stream()

    def upload(hb):
        if packed:
            return hb.upload(copy_stream)
        with torch.cuda.stream(copy_stream):
            d = {k: v.to(dev, non_blocking=True) for k, v in hb.items()}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return d, ev

    def e2e_loop(n):
        nxt = upload(host[0])
        last = None
        for i in range(n):
            d, ev = nxt
            if i + 1 < n:
                nxt = upload(host[(i + 1) % 2])
            torch.cuda.current_stream().wait_event(ev)
            if not packed:
                for v in d.values():
                    v.record_stream(torch.cuda.current_stream())
            total = wl.e2e_compute(b2, d, args.three or args.unfused)
            last = total.item()  # D2H read of the step's result
        return last

    e2e_steps = max(5, min(K, 20)) if wl.key in ('D', 'E', 'P') else max(20, min(K, 200))
    e2e_loop(3)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_loop(e2e_steps)
    f1.record()
    barrier()
    e2e_ms = f0.elapsed_time(f1)

    # ---- max over ranks --------------------------------------------------------------------------------------------
    dbg('e2e done')
    vals = [dev_ms, e2e_ms, host_ms, par['ms_per_step_with'] if par else 0.0]
    t = torch.tensor(vals, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, host_ms, par_ms = t.tolist()

    if rank == 0:
        peak, peak_src = load_peaks()
        units_per_step = wl.units * world
        ms_step = dev_ms / K
        value = units_per_step / (ms_step * 1e-3)
        step_achieved = step_bytes / (ms_step * 1e-3) / 1e9
        roof = {'bound': 'hbm', 'peak': peak, 'unit': 'GB/s', 'peak_source': peak_src,
                'step': {'alg_bytes': step_bytes, 'achieved': step_achieved, 'frac': step_achieved / peak}}
        if per:
            dom = max(per, key=per.get)
            dom_bytes = wl.alg_bytes[dom] * wl.units
            achieved = dom_bytes / (per[dom] * 1e-3) / 1e9
            traffic, traffic_src = ncu_traffic(dom)
            roof.update({'kernel': dom, 'achieved': achieved, 'frac': achieved / peak, 'traffic': traffic,
                         'traffic_source': traffic_src, 'alg_bytes_per_launch': dom_bytes, 'kernel_ms': per})
        else:  # the exchange rides inside the kernel: per-kernel timing alone would deadlock on the peers
            roof.update({'kernel': names[0], 'achieved': step_achieved, 'frac': step_achieved / peak, 'traffic': None,
                         'traffic_source': 'per-kernel timing is a single-GPU leg', 'alg_bytes_per_launch': step_bytes})
        cpu = run_cpu(wl, steps=8 if wl.key in ('D', 'E', 'P') else 40, warmup=2) if world == 1 else None
        e2e_value = units_per_step / (e2e_ms / e2e_steps * 1e-3)
        coll = 'none'
        if world > 1:
            coll = {'fused': 'the 6 loss scalars ride on the step\'s own launches: finalize_sums stages {tag, value} locally, the first '
                             'CTA of the NEXT step\'s kernel consumes the peers\' words of two steps ago and publishes the staged ones '
                             '(one 8-byte st.relaxed.sys per peer into NVLink peer-memory mailboxes) while it waits for its first '
                             'chunk; mean of rank means; one drain kernel after the last step; no collective launch, no forked branch',
                    'p2p-kernel': 'one small NVLink peer-memory kernel per step (b200rl_p2p_allreduce_mean) on a forked '
                                  'graph branch',
                    'nccl': 'one NCCL all-reduce of the 6 loss scalars per step on a forked graph branch'}[exchange]
        line = {
            'metric': wl.metric, 'value': value, 'unit': wl.unit + '/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {
                'workload': wl.workload,
                'units_per_step_per_gpu': wl.units, 'parallelism': 'dp%d' % world,
                'sharding': 'B sharded across GPUs, no data-path exchange' if world > 1 else 'single GPU',
                'l2_policy': 'inputs rotated over %d buffer sets (%.0f MB in total, > 126 MB L2 for configs D/E; configs '
                             'B/C are launch-bound and L2-resident by nature) between consecutive steps' %
                             (NSETS, NSETS * step_bytes / 1e6),
                'launch': 'ONE CUDA graph holding exactly %d steps between two in-graph timing events; %d launches per '
                          'step (%s)' % (K, sets[0].launches_per_step(), ', '.join(names)),
                'collective': coll,
                'cpu_affinity': affinity,
            },
            'ms_per_step_host_bracketed': host_ms / K,  # events around the graph launch: + the host's launch latency / K
            'roofline': roof,
            'cpu_baseline': None if cpu is None else {
                'value': cpu['value'], 'unit': wl.unit + '/s', 'cores': cpu['cores'], 'kind': cpu['kind'],
                'sample': 'full batch of the workload, median of %d steps after 2 warm-up (%.1f s CPU), %s' %
                          (8 if wl.key in ('D', 'E', 'P') else 40, cpu['total_s'], cpu_model()),
                'ms_per_step': cpu['ms_per_step'],
            },
            'e2e': {'value': e2e_value, 'unit': wl.unit + '/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4 + (8 if wl.key == 'D' else 0),
                    'ms_per_step': e2e_ms / e2e_steps, 'steps': e2e_steps},
            'eager_ms_per_step': eager_ms,  # same launches without the CUDA graph (host-bound; `value` is the graph replay)
            'gpu_launches': sets[0].launches_per_step() * K,
            'clocks': clocks,
        }
        if par:
            line['param_allreduce'] = dict(par, ms_per_step_with=par_ms,
                                           note='the step followed by an NCCL all-reduce of a %d-float dummy gradient '
                                                'bucket (Atari VAC net) on the same stream, eager launches' % VAC_PARAMS)
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, last_outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        # graphs that captured NCCL work must be gone before the communicator is torn down; then leave without waiting on
        # NCCL's own teardown (a destroy_process_group after captured collectives has been seen to hang)
        del graph_warm, graph_k
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def dump_outputs(out_dir, tensors):
    """DIR/<name>.npy in float32 for every output of the last timed step (rank 0's shard under data parallelism)"""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit('--dump-outputs: %d bytes of outputs exceed %d' % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cfg = getattr(args, 'config', 'D')
    wl = WORKLOADS[cfg]()
    steps = min(args.steps, 400 if cfg in ('D', 'E', 'P') else 2000)
    r = run_cpu(wl, steps=steps, warmup=max(args.warmup, 1))
    line = {
        'impl': 'reference', 'metric': wl.metric, 'value': r['value'], 'unit': wl.unit + '/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': max(args.warmup, 1), 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
        'scaling': getattr(args, 'scaling', 'weak'), 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl.workload, 'parallelism': 'cpu',
                   'implementation': 'unmodified ding.rl_utils (oracle/_ref/ding_hotpath.zip)' if r['kind'] == 'reference'
                   else 'oracle port (oracle/rl_oracle.py)'},
        'cpu_baseline': {'value': r['value'], 'unit': wl.unit + '/s', 'cores': r['cores'], 'kind': r['kind'],
                         'sample': 'one full batch of the workload per step, %d torch threads (best of the candidates, '
                                   'best-of-3 each), %s' % (r['threads'], cpu_model())},
        'e2e': {'value': r['value'], 'unit': wl.unit + '/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


def run_reference_cuda(args):
    """--impl reference-cuda: the reference's torch functions on CUDA tensors on the B200 -- the same-hardware baseline
    (BASELINE.md section 3).  Eager torch, CUDA events, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.config]()
    api, kind = _cpu_api()
    dev = 'cuda:0'
    bs = [{k: v.to(dev) for k, v in wl.make_batch(i).items()} for i in range(NSETS)]
    for i in range(max(args.warmup, 3)):
        wl.cpu_step(api, bs[i % NSETS])
    torch.cuda.synchronize()
    steps = min(args.steps, 200)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        wl.cpu_step(api, bs[i % NSETS])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak, peak_src = load_peaks()
    ach = wl.step_bytes_per_unit * wl.units / (ms * 1e-3) / 1e9
    line = {
        'impl': 'reference-cuda', 'metric': wl.metric, 'value': wl.units / (ms * 1e-3), 'unit': wl.unit + '/s',
        'n_gpus': 1, 'steps': steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl.workload, 'parallelism': 'dp1',
                   'implementation': ('unmodified ding.rl_utils' if kind == 'reference' else 'oracle port') +
                   ' torch functions on CUDA tensors, eager launches'},
        'roofline': {'bound': 'hbm', 'peak': peak, 'unit': 'GB/s', 'peak_source': peak_src,
                     'step': {'alg_bytes': wl.step_bytes_per_unit * wl.units, 'achieved': ach, 'frac': ach / peak}},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-cuda'])
    ap.add_argument('--config', default='D', choices=['D', 'P', 'B', 'C', 'E'],
                    help='BASELINE.json configs: D (default) gae+ppo_error, B q_nstep_td_error, C dist_nstep_td_error, E vtrace')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='N>1: weak = a full batch per GPU (default); strong = the config-D/E batch sharded over the GPUs')
    ap.add_argument('--collective', default='auto', choices=['auto', 'fused', 'p2p-kernel', 'nccl'],
                    help='N>1: exchange of the loss scalars (auto = fused into the step kernel for config D)')
    ap.add_argument('--unfused', action='store_true', help='config D: separate gae / ppo forward / ppo backward kernels')
    ap.add_argument('--three', action='store_true',
                    help='config D: gae, fused ppo forward+grad, verification as three calls (default: the one-launch step)')
    ap.add_argument('--e2e-wide', dest='e2e_compact', action='store_false',
                    help='e2e: int64 actions / fp32 flags on the wire (default: one byte each, widened on the device)')
    ap.add_argument('--e2e-separate-copies', action='store_true',
                    help='e2e: one pinned tensor and one H2D copy per input (default: di_engine_b200.PackedBatch, one copy)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps write the outputs of the last one (losses, advantages, gradients) as '
                         'DIR/<name>.npy, float32; the inputs are seeded, so two builds can be compared output for output')
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
    elif args.impl == 'reference-cuda':
        run_reference_cuda(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
