"""SURVEY 8f rank 4 on the GPU: a manager-based TENSOR env (mjlab's ManagerBasedRlEnv API: observation groups, bool terminated /
truncated tensors on the simulation device, a reused extras dict with per-burst episode metrics) behind `ManagerBasedEnvAdapter`, with the
device-resident `IsaacAlgoObserver` in the training loop, through the CUDA kernels of the C ABI.

The env replays the tapes of the reference's own golden runs, so the adapter route has the SAME answer as the plain-IVecEnv route the golden
tests use: `agent_masked.pt` (next_step autoreset, masked rows, time-outs) and `agent_cv.pt` ('critic' group -> central-value `states`).
What is specific to this route and only runs here: bool dones / time-outs ingested by the post-step kernel without a cast launch, the
per-step infos reaching the observer without done indices (no per-step host sync), episode metrics accumulated on the device.
(File name: sorts after the other GPU test files -- the newest test of the suite runs last.)"""
import os
import types

import pytest
import torch

from oracle import ppo_oracle as O
from tests.test_agent_gpu import DEV, GOLDEN, RUNS, _check_epoch, make_agent

pytestmark = pytest.mark.gpu


class _TapeManagerEnvGPU:
    """the golden tapes, resident on the GPU, behind mjlab's manager-based API"""

    def __init__(self, g, critic=False):
        self.g = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in g.items()}
        self.i, self.critic = 0, critic
        self.action_space = types.SimpleNamespace(shape=(g['N'], g['A']))
        self.extras = {}                                                 # reused across steps, like the real env's
        self.metric = torch.zeros(g['N'], device=DEV)                    # the tensor the env reports its burst metrics in, reused too
        self.n_resets = 0

    def _groups(self, j):
        o = {'actor': self.g['obs_tape'][j].clone()}
        if self.critic:
            o['critic'] = self.g['state_tape'][j].clone()
        return o

    def reset(self):
        self.i = 0
        self.n_resets += 1
        return self._groups(0), self.extras

    def step(self, actions):
        g = self.g
        assert actions.dtype == torch.float32 and actions.shape == (g['N'], g['A'])
        self.i += 1
        j = self.i % g['obs_tape'].shape[0]
        done, trunc = g['done_tape'][j] > 0, g['timeout_tape'][j] > 0                   # bool tensors on the device
        # per-burst episode metric: env index of every finished episode, written into the REUSED tensor; empty log between bursts.
        # (whether a burst happened is known from the host copy of the tape: no device sync in the loop)
        n_done = self.host_done_counts[j]
        if n_done:
            self.metric[:n_done] = done.nonzero().reshape(-1).float()
            self.extras['log'] = {'ep_len': self.metric[:n_done], 'plain': 2.0}
        else:
            self.extras['log'] = {}
        return self._groups(j), -(actions * actions).sum(-1) * 0.1, done & ~trunc, trunc, self.extras

    def close(self):
        pass


def _adapter(g, critic=False):
    from rl_games_b200.env_adapters import ManagerBasedEnvAdapter
    backend = _TapeManagerEnvGPU(g, critic=critic)
    backend.host_done_counts = [int((g['done_tape'][j] > 0).sum()) for j in range(g['done_tape'].shape[0])]
    env = ManagerBasedEnvAdapter(backend, device=DEV)
    if g['autoreset'] != 'same_step':           # the tapes were recorded from a next_step-autoreset env; a manager env reports that in its info
        env.get_env_info = lambda base=env.get_env_info: {**base(), 'autoreset_mode': g['autoreset']}
    return env, backend


def _golden_over(g, graph):
    cfgk = g['config']
    over = {k: cfgk[k] for k in ('clip_value', 'use_smooth_clamp', 'bound_loss_type', 'bounds_loss_coef', 'entropy_coef', 'truncate_grads',
                                 'value_bootstrap', 'mini_epochs', 'lr_schedule', 'weight_decay', 'critic_coef', 'learning_rate', 'kl_threshold',
                                 'max_epochs', 'normalize_input', 'normalize_value', 'normalize_advantage', 'e_clip', 'tau', 'gamma') if k in cfgk}
    over.setdefault('lr_schedule', None)
    over['b200_cuda_graph'] = graph
    return over


@pytest.mark.parametrize('graph', [False, True])
def test_manager_based_adapter_and_isaac_observer_reproduce_the_reference_golden_run(graph):
    g = torch.load(os.path.join(GOLDEN, 'agent_masked.pt'), weights_only=False)
    assert int(((g['timeout_tape'] > 0) & ~(g['done_tape'] > 0)).sum()) == 0       # truncated implies done in this API: same tapes
    env, backend = _adapter(g)
    info = env.get_env_info()
    assert info['observation_space'].shape == (g['D'],) and info['action_space'].shape == (g['A'],) and 'state_space' not in info
    over = _golden_over(g, graph)
    over['algo_observer'] = 'isaac'
    agent = make_agent(over, g['N'], g['H'], g['D'], g['A'], g['units'], g['mb'], env, g['init_state'])
    from rl_games_b200.common import IsaacAlgoObserver
    assert isinstance(agent.algo_observer, IsaacAlgoObserver)
    assert not agent._whole_epoch_graph_ok()            # the observer reads every step's infos: the env step stays outside the rollout graph
    rows = []
    agent.algo_observer.writer = type('W', (), {'add_scalar': lambda self, *r: rows.append(r)})()
    n_tape = g['obs_tape'].shape[0]
    for ep, ref in enumerate(g['epochs_out']):
        agent.epoch_num += 1
        agent.train_epoch(noise=g['noise'][ep].to(DEV))
        assert torch.equal(agent.dones_buf.cpu(), ref['mb_dones'])
        torch.testing.assert_close(agent.rewards.cpu().unsqueeze(2), ref['mb_rewards'], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(agent.values.cpu().unsqueeze(2), ref['mb_values'], rtol=1e-4, atol=1e-5)
        _check_epoch(agent, ref['state'], ref['dataset'], {'a': ref['a_losses'], 'c': ref['c_losses'], 'e': ref['entropies']},
                     ref['last_lr'], g['units'])
        torch.testing.assert_close(agent.game_rewards.mean, ref['game_rewards_mean'].reshape(-1), rtol=1e-4, atol=1e-5)
        assert agent.game_rewards.current_size == ref['game_rewards_size']
        torch.testing.assert_close(agent.game_lengths.mean, ref['game_lengths_mean'].reshape(-1), rtol=1e-5, atol=1e-5)
        # the observer's episode metric = mean over every burst of the epoch (reference: concatenate the bursts' tensors, then mean,
        # algo_observer.py:131-147); the env's reused metric tensor must have been copied at every step
        steps = range(ep * g['H'] + 1, (ep + 1) * g['H'] + 1)
        want = torch.cat([(g['done_tape'][j % n_tape] > 0).nonzero().reshape(-1).float() for j in steps])
        rows.clear()
        agent.algo_observer.after_print_stats(123, agent.epoch_num, 0.5)
        got = dict((r[0], r[1]) for r in rows)
        assert got['Episode/ep_len'] == pytest.approx(want.mean().item(), rel=1e-6)
        assert got['Episode/plain'] == pytest.approx(2.0)
    assert backend.n_resets == 2                        # the constructor's probing reset + env_reset(), like the reference wrapper


@pytest.mark.parametrize('graph', [False, True])
def test_critic_group_feeds_the_central_value_net_like_the_reference_golden_run(graph):
    """'critic' observation group -> `states` + use_global_observations (mjlab_vecenv.py:76-98, 134-150) -> A2CAgentCV on the GPU"""
    from rl_games_b200.runner import Runner
    g = torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False)
    assert int(((g['timeout_tape'] > 0) & ~(g['done_tape'] > 0)).sum()) == 0
    env, _ = _adapter(g, critic=True)
    info = env.get_env_info()
    assert info['state_space'].shape == (g['S'],) and info['use_global_observations'] is True
    cfgk = g['config']
    cv_cfg = dict(g['cv_config'])
    cv_cfg['network'] = {'name': 'actor_critic', 'central_value': True,
                         'mlp': {'units': g['cv_units'], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    config = {k: v for k, v in cfgk.items() if k not in ('device', 'torch_compile')}
    config.update({'device': DEV, 'env_info': info, 'vec_env': env, 'reward_shaper': {'scale_value': 1.0}, 'mixed_precision': False,
                   'b200_cuda_graph': graph, 'train_dir': RUNS.name, 'lr_schedule': cfgk.get('lr_schedule', None),
                   'central_value_config': cv_cfg, 'algo_observer': 'isaac'})
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': g['units'], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    r = Runner()
    r.load({'params': {'seed': 7, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network,
                       'config': config}})
    r.params['config']['vec_env'] = env
    agent = r.algo_factory.create(r.algo_name, base_name='parity', params=r.params)
    assert agent.has_central_value
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


@pytest.mark.parametrize('graph', [False, True])
def test_separate_actor_critic_trunks_match_the_reference_golden_run(graph):
    """separate: True for a CONTINUOUS policy (network_builder.py:494-512; configs/ppo_continuous.yaml, ppo_lunar.yaml, ppo_reacher.yaml ...):
    the two trunks run as one block-structured MLP of twice the width through the same fp32 kernels (rl_games_b200/model.py); the gradient
    entries of the structural zeros are masked before the optimiser.  Against the reference's own run (`agent_separate.pt`: masked rows,
    global-norm clip over both trunks, weight decay, entropy bonus, bound loss); the structural zeros are still exactly zero afterwards."""
    from tests.test_agent_gpu import _golden_run
    agent = _golden_run('agent_separate.pt', graph)
    m = agent.model
    assert m.separate and m.units == [2 * u for u in m.trunk_units]
    structural = m.grad_mask == 0
    for arena in (m.flat, m.grad, m.exp_avg, m.exp_avg_sq):
        assert float(arena[structural].abs().max()) == 0.0
