"""Central value (asymmetric critic) on the GPU (rl_games_b200/agent_cv.py, csrc/critic.cu); first green on a B200 in round 2.
The host logic and the kernel's row arithmetic are also checked on CPU (tests/test_agent_cv_host_cpu.py, tests/test_critic_rows_cpu.py)."""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

pytestmark = [pytest.mark.gpu]
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
RUNS = tempfile.TemporaryDirectory(prefix='b200_test_runs_')      # the agents' train_dir: private to this process, removed at exit


@pytest.mark.parametrize('masked', [False, True])
def test_value_loss_kernel_vs_autograd(masked):
    from rl_games_b200 import ops
    g = torch.Generator().manual_seed(2)
    H, N, epm = 4, 96, 32
    M = H * epm
    e0 = 32
    v = torch.randn(M, 1, generator=g).requires_grad_(True)
    old_v, ret = torch.randn(H, N, generator=g), torch.randn(H, N, generator=g)
    mask = (torch.rand(H, N, generator=g) < 0.7).float() if masked else None
    sl = lambda t: torch.cat([t[h, e0:e0 + epm] for h in range(H)])   # noqa: E731  minibatch rows in kernel order (chunk-major)
    c = O.critic_loss(sl(old_v).unsqueeze(1), v, 0.2, sl(ret).unsqueeze(1), True).squeeze(1)
    w = torch.full((M,), 1.0 / M) if mask is None else sl(mask) / sl(mask).sum()
    loss = (c * w).sum()
    loss.backward()
    d = lambda t: None if t is None else t.to(DEV)   # noqa: E731
    dv = torch.zeros(M, 1, device=DEV)
    part = torch.zeros((M + 255) // 256, 8, dtype=torch.float64, device=DEV)
    inv = None if mask is None else torch.tensor([1.0 / float(sl(mask).sum())], device=DEV)
    ov, rt, mk = d(old_v), d(ret), d(mask)
    nb = ops.value_loss(d(v.detach()), 1, ov[0, e0:], rt[0, e0:], None if mk is None else mk[0, e0:], epm, N, M, 0.2, True, inv, dv, 1, part)
    torch.cuda.synchronize()
    assert float(part[:nb, 0].sum()) == pytest.approx(float(loss), rel=1e-5)
    torch.testing.assert_close(dv.cpu(), v.grad, rtol=1e-5, atol=1e-9)


class _Env:
    def __init__(self, g):
        self.g = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in g.items()}
        self.i = 0

    def _o(self, j):
        return {'obs': self.g['obs_tape'][j].clone(), 'states': self.g['state_tape'][j].clone()}

    def reset(self):
        self.i = 0
        return self._o(0)

    def step(self, actions):
        g = self.g
        rew = -(actions * actions).sum(-1) * 0.1
        self.i += 1
        j = self.i % g['obs_tape'].shape[0]
        return self._o(j), rew, g['done_tape'][j].clone(), {'time_outs': g['timeout_tape'][j].clone()}

    def get_env_info(self):
        from rl_games_b200.common import Box
        info = {'observation_space': Box(-np.inf, np.inf, (self.g['D'],)), 'action_space': Box(-1.0, 1.0, (self.g['A'],)),
                'state_space': Box(-np.inf, np.inf, (self.g['S'],))}
        if self.g['autoreset'] != 'same_step':
            info['autoreset_mode'] = self.g['autoreset']
        return info

    def get_env_state(self):
        return None

    def set_env_state(self, s):
        pass


@pytest.mark.parametrize('graph', [False, True])
def test_central_value_agent_matches_reference_golden(graph):
    from rl_games_b200.runner import Runner
    g = torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False)
    cfgk = g['config']
    env = _Env(g)
    cv_cfg = dict(g['cv_config'])
    cv_cfg['network'] = {'name': 'actor_critic', 'central_value': True,
                         'mlp': {'units': g['cv_units'], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    config = {k: v for k, v in cfgk.items() if k not in ('device', 'torch_compile')}
    config.update({'device': DEV, 'env_info': env.get_env_info(), 'vec_env': env, 'reward_shaper': {'scale_value': 1.0},
                   'mixed_precision': False, 'b200_cuda_graph': graph, 'train_dir': RUNS.name,
                   'lr_schedule': cfgk.get('lr_schedule', None), 'central_value_config': cv_cfg})
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': g['units'], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    r = Runner()
    r.load({'params': {'seed': 7, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network,
                       'config': config}})
    r.params['config']['vec_env'] = env
    agent = r.algo_factory.create(r.algo_name, base_name='parity', params=r.params)
    agent.model.load_state_dict({k: v.to(DEV) for k, v in g['init_state'].items()}, strict=False)
    cv = agent.central_value_net
    cv.load_state_dict({k: v.to(DEV) for k, v in g['cv_init_state'].items()})
    agent.init_tensors()
    agent._repack()
    agent.obs = agent.env_reset()
    flat_noise = g['noise'].reshape(-1, g['N'], g['A']).to(DEV)
    for ep, ref in enumerate(g['epochs_out']):
        agent.epoch_num += 1
        agent.train_epoch(noise=flat_noise[ep * g['H']:(ep + 1) * g['H']])
        torch.testing.assert_close(agent.values.cpu().unsqueeze(2), ref['mb_values'], rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(agent.rewards.cpu().unsqueeze(2), ref['mb_rewards'], rtol=1e-5, atol=1e-6)
        assert agent.last_lr == pytest.approx(ref['last_lr'], rel=1e-12) and cv.lr == pytest.approx(ref['cv_lr'], rel=1e-12)
        sd = agent.model.state_dict()
        for k in O.param_names(len(g['units'])):
            torch.testing.assert_close(sd[k].cpu(), ref['state'][k], rtol=1e-3, atol=2e-5, msg=lambda m: k + ': ' + m)
        csd = cv.state_dict()
        for k in g['cv_param_order']:
            torch.testing.assert_close(csd[k].cpu(), ref['cv_state'][k], rtol=1e-3, atol=2e-5, msg=lambda m: 'cv ' + k + ': ' + m)
        assert int(csd['value_mean_std.count']) == int(ref['cv_state']['value_mean_std.count'])
